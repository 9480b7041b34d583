"""CPU warp emulation of the electrostatics kernels (epnn_elst.cu), and the dimer splits that label the fragments.

The kernel source is compiled for the host with -DEPNN_CPU_EMU (tools/emu/cuda_emu.h).  tools/emu/emu_elst.cpp builds the
same work plan as the library (epnn_elst.cuh) and runs the small-system, pair and reduction kernels on the adversarial batch
of tests/elst_ref.py: 1 ... 49 atoms around the 32 lanes and the 48-atom bound, the pair kernel's tile and source-split
edges up to 1 000 atoms, charges of both signs with Q != 0, coincident atoms, and every fragment labelling the issue of
dimer energies needs.  The SM count is a parameter of the plan, so the emulation reaches source splits a B200 only makes
at ten thousand atoms and more."""
import ctypes as C
import os
import shutil
import subprocess
import warnings

import numpy as np
import pytest

from elst_ref import adversarial_batch, batch_ref, check, fragment_variants, kernel_constants, system_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "build", "libemu_elst.so")
GOLDEN_XYZ = os.path.join(ROOT, "tests", "golden", "xyz")
K = kernel_constants()
# pair CTAs the plan aims at (ELST_CTAS_PER_SM x SM count): 1 never splits, 20 splits some systems by the CTA count (odd
# part counts included), 10**6 splits every system as far as ELST_MIN_PART allows
TARGETS = (1, 20, 10 ** 6)


@pytest.fixture(scope="module")
def emu():
    os.makedirs(os.path.join(ROOT, "build"), exist_ok=True)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-pthread", "-DEPNN_CPU_EMU",
                           "-Wno-unknown-pragmas", "-o", LIB, os.path.join(ROOT, "tools", "emu", "emu_elst.cpp")])
    lib = C.CDLL(LIB)
    lib.emu_elst_parts.argtypes = [C.c_int, C.c_longlong]
    lib.emu_elst.argtypes = [C.c_int] + [C.c_void_p] * 4 + [C.c_longlong] + [C.c_void_p] * 3
    return lib


@pytest.fixture(scope="module")
def batch():
    offs, xyz, q, labels = adversarial_batch()
    return dict(offs=offs, xyz=xyz, q=q, labels=labels, refs={None: batch_ref(offs, xyz, q)})


def run(emu, offs, xyz, q, frag=None, target=10 ** 6):
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    n_sys, n = len(offs) - 1, int(offs[-1])
    out = {"energy": np.full(n_sys, np.nan), "dipole": np.full((n_sys, 3), np.nan), "phi": np.full(n, np.nan)}
    emu.emu_elst(n_sys, p(offs), p(xyz), p(q), p(frag), target, p(out["energy"]), p(out["dipole"]), p(out["phi"]))
    return out


def test_the_batch_reaches_the_kernel_edges(emu, batch):
    n = np.diff(batch["offs"])
    T, MP, SM = K["ELST_TILE"], K["ELST_MIN_PART"], K["ELST_SMALL_MAX"]
    assert {1, 31, 32, 33, SM, SM + 1, T - 1, T, T + 1, MP, MP + 1} <= set(n.tolist())
    parts = {t: [emu.emu_elst_parts(int(m), t) for m in n if m > SM] for t in TARGETS}
    assert set(parts[1]) == {1}
    assert {1, 2, 3} <= set(parts[20]) and any(p < -(-m // MP) for p, m in zip(parts[20], n[n > SM]))   # CTA-count bound
    assert parts[10 ** 6] == [-(-int(m) // MP) for m in n if m > SM] and max(parts[10 ** 6]) == 4     # ELST_MIN_PART bound


@pytest.mark.parametrize("target", TARGETS)
def test_emulated_kernels_match_the_definition(emu, batch, target):
    got = run(emu, batch["offs"], batch["xyz"], batch["q"], target=target)
    check(batch["offs"], got, batch["refs"][None])
    assert got["energy"][0] == 0.0 and np.array_equal(got["dipole"][0], np.zeros(3))      # one atom: nothing to add up


@pytest.mark.parametrize("kind", ["split1", "split_last", "own", "interleaved"])
def test_emulated_kernels_with_fragments(emu, batch, kind):
    offs, xyz, q = batch["offs"], batch["xyz"], batch["q"]
    frag = fragment_variants(offs)[kind]
    got = run(emu, offs, xyz, q, frag, target=20)
    check(offs, got, batch_ref(offs, xyz, q, frag))
    plain = run(emu, offs, xyz, q, None, target=20)
    assert np.array_equal(got["dipole"], plain["dipole"])                 # fragments do not change mu
    if kind == "own":                                                     # every pair included: the same bits as NULL
        assert np.array_equal(got["energy"], plain["energy"]) and np.array_equal(got["phi"], plain["phi"])


def test_a_system_alone_gives_the_bits_it_gives_in_the_batch(emu, batch):
    offs, xyz, q = batch["offs"], batch["xyz"], batch["q"]
    full = run(emu, offs, xyz, q, target=20)
    for s in (5, 8, len(offs) - 2):
        a0, a1 = int(offs[s]), int(offs[s + 1])
        one = run(emu, np.array([0, a1 - a0], np.int32), xyz[a0:a1], q[a0:a1], target=20)
        assert one["energy"][0] == full["energy"][s] and np.array_equal(one["dipole"][0], full["dipole"][s])
        assert np.array_equal(one["phi"], full["phi"][a0:a1])


def test_null_outputs_are_skipped(emu, batch):
    offs, xyz, q = batch["offs"], batch["xyz"], batch["q"]
    e = np.full(len(offs) - 1, np.nan)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    emu.emu_elst(len(offs) - 1, p(offs), p(xyz), p(q), None, 20, p(e), None, None)
    assert np.array_equal(e, run(emu, offs, xyz, q, target=20)["energy"])


def test_reference_agrees_with_the_pair_loop():
    """The dense reference against the definition written as a loop over i < j."""
    offs, xyz, q, _ = adversarial_batch()
    a0, a1 = int(offs[5]), int(offs[6])
    x, c = xyz[a0:a1].astype(np.float64), q[a0:a1]
    f = np.arange(a1 - a0) % 3
    E = sum(c[i] * c[j] / np.linalg.norm(x[i] - x[j]) for i in range(len(c)) for j in range(i + 1, len(c))
            if np.linalg.norm(x[i] - x[j]) > 0 and f[i] != f[j])
    assert abs(system_ref(x, c, f)["energy"] - E) < 1e-13


# ------------------------------------------------------------------------------------------------ dimer splits
def test_read_splits_on_the_golden_directory():
    from epnn_b200 import xyzio
    stems = sorted(n[:-4] for n in os.listdir(GOLDEN_XYZ) if n.endswith(".xyz"))
    with warnings.catch_warnings():
        warnings.simplefilter("error")                                 # the golden files are well formed
        sp = xyzio.read_splits(GOLDEN_XYZ, stems)
    want = {"SSI-081ILE-085ARG-1-dimer": 6, "SSI-001ASN-030MET-1-dimer": 8}
    assert sp.tolist() == [want.get(s, -1) for s in stems]


def test_read_splits_rejects_malformed_files(tmp_path):
    from epnn_b200 import xyzio
    src = os.path.join(GOLDEN_XYZ, "SSI-081ILE-085ARG-1-dimer.xyz")        # 24 atoms
    bad = {"vec": np.array([6, 7]), "zero": np.int64(0), "n": np.int64(24), "neg": np.int64(-3), "frac": np.float64(6.5),
           "nan": np.float64(np.nan), "text": np.array("6"), "ok_float": np.float64(6.0), "ok_last": np.array([23])}
    for stem, v in bad.items():
        shutil.copy(src, tmp_path / f"{stem}.xyz")
        np.save(tmp_path / f"{stem}splits.npy", v)
    shutil.copy(src, tmp_path / "garbage.xyz")
    (tmp_path / "garbagesplits.npy").write_bytes(b"not an npy file")
    shutil.copy(src, tmp_path / "nosplit.xyz")
    stems = list(bad) + ["garbage", "nosplit"]
    with pytest.warns(UserWarning) as rec:
        sp = xyzio.read_splits(str(tmp_path), stems)
    assert sp.tolist() == [-1] * 7 + [6, 23] + [-1, -1]
    assert len(rec) == 8                                                  # every malformed file warns; a missing one does not


def test_fragments_from_splits():
    from epnn_b200 import xyzio
    f = xyzio.fragments_from_splits(np.array([0, 3, 5, 9], np.int32), np.array([1, -1, 2]))
    assert f.dtype == np.int32 and f.tolist() == [0, 1, 1, 0, 0, 0, 0, 1, 1]
