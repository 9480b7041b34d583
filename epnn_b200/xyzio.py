"""Reader for the reference's xyz dialect (``charge_gn.py:309-330``; SURVEY.md section 5.6).

line 1: atom count (ignored: atoms = every line after line 2)
line 2: first token = net charge Q (float32); remaining tokens ignored
line 3+: ``Elem x y z [ignored columns]``; coordinates are rounded to float32 like the reference.
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np


@dataclass
class System:
    name: str
    symbols: List[str]
    xyz: np.ndarray            # (n, 3) float32
    Q: np.float32
    labels: Optional[np.ndarray] = None   # (n,) float32 MBIS labels if <stem>.npy exists

    @property
    def n(self) -> int:
        return len(self.symbols)


def parse_xyz_text(text: str, name: str = "") -> System:
    lines = text.splitlines()
    if len(lines) < 3:
        raise ValueError(f"{name}: xyz file needs at least one atom line")
    Q = np.float32(lines[1].strip().split()[0])
    symbols, coords = [], []
    for line in lines[2:]:
        data = line.split()
        if not data:            # the reference would IndexError on a blank line; tolerate a trailing one
            continue
        symbols.append(data[0])
        coords.append([data[1], data[2], data[3]])
    xyz = np.array(coords, dtype=np.float32)
    if not (np.isfinite(xyz).all() and np.isfinite(Q)):      # same rule as the native parser: nan / inf is an input error
        raise ValueError(f"{name}: non-finite coordinate or charge")
    return System(name=name, symbols=symbols, xyz=xyz, Q=Q)


def read_xyz(path: str) -> System:
    with open(path, "r") as f:
        s = parse_xyz_text(f.read(), os.path.basename(path)[:-4])
    lab = path[:-4] + ".npy"
    if os.path.exists(lab):
        s.labels = np.array(np.load(lab), dtype=np.float32).reshape(-1)
    return s


def read_directory(path: str, sort: bool = False) -> List[System]:
    """All ``*.xyz`` of a directory in ``os.listdir`` order (reference ``charge_gn.py:301``)."""
    names = os.listdir(path)
    if sort:
        names = sorted(names)
    return [read_xyz(os.path.join(path, n)) for n in names if n.endswith(".xyz")]


def pack(systems: Sequence[System], n_x: int):
    """Concatenate systems into the SoA arrays the C-ABI takes: offsets, xyz, species, Q."""
    from .elements import species_index
    offsets = np.zeros(len(systems) + 1, dtype=np.int32)
    for i, s in enumerate(systems):
        offsets[i + 1] = offsets[i] + s.n
    xyz = np.concatenate([s.xyz for s in systems], axis=0).astype(np.float32) if systems else np.zeros((0, 3), np.float32)
    species = np.concatenate([species_index(s.symbols, n_x) for s in systems]) if systems else np.zeros(0, np.int32)
    Q = np.array([s.Q for s in systems], dtype=np.float32)
    return offsets, np.ascontiguousarray(xyz), np.ascontiguousarray(species, dtype=np.int32), Q


def read_splits(path: str, stems: Sequence[str]) -> np.ndarray:
    """For each stem, the index where the second monomer starts, read from ``<path>/<stem>splits.npy`` (the SSI dimers of
    the reference's data set carry one; ``charge_gn.py:305-308`` loads it), or -1.  A missing file gives -1 silently; a
    file that does not hold one integer index inside [1, n - 1] of its system gives -1 with a warning (n is read from
    the atom lines of ``<stem>.xyz``)."""
    import warnings
    out = np.full(len(stems), -1, np.int64)
    for k, stem in enumerate(stems):
        f = os.path.join(path, stem + "splits.npy")
        if not os.path.exists(f):
            continue
        try:
            a = np.load(f, allow_pickle=False)
            n = read_xyz(os.path.join(path, stem + ".xyz")).n
        except Exception as e:      # noqa: BLE001 -- an unreadable split file is reported, not fatal
            warnings.warn(f"{f}: cannot be read ({e}); no split")
            continue
        v = a.reshape(-1)[0] if a.size == 1 else None
        if v is None or not (a.dtype.kind in "iu" or (a.dtype.kind == "f" and np.isfinite(v) and float(v).is_integer())):
            warnings.warn(f"{f}: expected one integer index, got shape {a.shape} dtype {a.dtype}; no split")
            continue
        v = int(v)
        if not 1 <= v <= n - 1:
            warnings.warn(f"{f}: split {v} is outside [1, {n - 1}] for {n} atoms; no split")
            continue
        out[k] = v
    return out


def fragments_from_splits(offsets, splits) -> np.ndarray:
    """int32 fragment label per atom for ``Engine.electrostatics``: 0 before the split of its system, 1 from it on; every
    atom of a system whose split is -1 gets 0 (no pair of that system then counts: its fragment energy is 0)."""
    offsets = np.asarray(offsets, np.int64)
    splits = np.asarray(splits, np.int64)
    sys_of = np.repeat(np.arange(len(splits)), np.diff(offsets))
    local = np.arange(int(offsets[-1])) - offsets[:-1][sys_of]
    return ((splits[sys_of] >= 0) & (local >= splits[sys_of])).astype(np.int32)


# ------------------------------------------------------------------------------------------------ native ingest
def _collect(lib, handle):
    import ctypes as C
    try:
        kind, idx = C.c_int(0), C.c_int(-1)
        lib.epnn_xyz_error(handle, C.byref(kind), C.byref(idx))
        if kind.value:
            msg = lib.epnn_xyz_error_message(handle).decode()
            if kind.value == 3:
                raise KeyError(msg.split("'")[1] if "'" in msg else msg)      # the reference's dict lookup raises KeyError
            if kind.value == 1:
                raise FileNotFoundError(msg)
            raise ValueError(msg)
        n_sys, n_at = lib.epnn_xyz_n_systems(handle), lib.epnn_xyz_n_atoms(handle)

        def arr(ptr, ctype, n, dtype):
            if n == 0:
                return np.zeros(0, dtype)
            return np.ctypeslib.as_array((ctype * n).from_address(ptr)).astype(dtype, copy=True)

        offsets = arr(lib.epnn_xyz_offsets(handle), C.c_int32, n_sys + 1, np.int32)
        xyz = arr(lib.epnn_xyz_coords(handle), C.c_float, 3 * n_at, np.float32).reshape(n_at, 3)
        species = arr(lib.epnn_xyz_species(handle), C.c_int32, n_at, np.int32)
        Q = arr(lib.epnn_xyz_charges(handle), C.c_float, n_sys, np.float32)
        return offsets, xyz, species, Q
    finally:
        lib.epnn_xyz_free(handle)


def load_packed(paths: Sequence[str], n_x: int, threads: int = 0):
    """Parse xyz files with the library's multi-threaded reader (epnn_xyz_load) straight into the packed arrays
    ``(offsets, xyz, species, Q)`` of the C-ABI.  Same dialect and rounding as :func:`parse_xyz_text`; file order = the
    order of ``paths``.  Unknown element -> KeyError, malformed file -> ValueError (like the Python path)."""
    import ctypes as C
    from . import _capi
    lib = _capi.load()
    enc = [os.fsencode(p) for p in paths]
    arr = (C.c_char_p * len(enc))(*enc)
    h = C.c_void_p()
    rc = lib.epnn_xyz_load(arr, len(enc), n_x, threads, C.byref(h))
    if not h:
        raise _capi.EpnnError(rc, "epnn_xyz_load failed")
    return _collect(lib, h)


def parse_packed(text: str, n_x: int):
    import ctypes as C
    from . import _capi
    lib = _capi.load()
    raw = text.encode()
    h = C.c_void_p()
    rc = lib.epnn_xyz_parse_text(raw, len(raw), n_x, C.byref(h))
    if not h:
        raise _capi.EpnnError(rc, "epnn_xyz_parse_text failed")
    return _collect(lib, h)


def read_directory_packed(path: str, n_x: int, sort: bool = False, threads: int = 0):
    """``(names, offsets, xyz, species, Q)`` for every ``*.xyz`` of a directory in ``os.listdir`` order
    (reference ``charge_gn.py:301``), parsed natively."""
    names = os.listdir(path)
    if sort:
        names = sorted(names)
    names = [n for n in names if n.endswith(".xyz")]
    offsets, xyz, species, Q = load_packed([os.path.join(path, n) for n in names], n_x, threads)
    return [n[:-4] for n in names], offsets, xyz, species, Q
