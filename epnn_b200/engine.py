"""Engine: one libepnn_b200 context on one GPU (host-side mirror of the model object the reference
builds with ``charge_gn.make_model(...)`` + ``load_weights`` -- reference charge_gn.py:369-391, infer.py:56-57)."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _capi
from .checkpoint import Weights

# Unit conversions of the electrostatics outputs (the C-ABI works in e and Angstrom)
COULOMB_KCAL = 332.0637133       # e^2/A -> kcal/mol: e^2 / (4 pi eps0 A) in kcal/mol, CODATA 2018
DEBYE_PER_E_ANGSTROM = 4.80320471   # e*A -> Debye, CODATA 2018
BOHR_ANGSTROM = 0.529177210903     # Bohr radius in A, CODATA 2018: phi [e/A] * BOHR_ANGSTROM = phi [e/bohr]


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _as(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


class Engine:
    def __init__(self, weights: Weights, device: int = 0, precision: int = 32):
        self.lib = _capi.load()
        self.weights = weights
        self.T, self.n_x = weights.T, weights.n_x
        packed = weights.packed()
        h = C.c_void_p()
        rc = self.lib.epnn_create(device, weights.T, weights.n_x, _ptr(packed), packed.size, C.byref(h))
        if rc != 0:
            raise _capi.EpnnError(rc, self.lib.epnn_last_error(None).decode())
        self._h = h
        self.device = device
        self.last_stats = None
        if precision != 32:
            self.set_option("precision", precision)

    # ------------------------------------------------------------------ plumbing
    def _check(self, rc):
        if rc != 0:
            raise _capi.EpnnError(rc, self.lib.epnn_last_error(self._h).decode())

    def set_option(self, key: str, value: float):
        self._check(self.lib.epnn_set_option(self._h, key.encode(), float(value)))

    def close(self):
        if getattr(self, "_h", None):
            self.lib.epnn_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream(self) -> int:
        """The ctx's cudaStream_t as an integer handle (for torch.cuda.ExternalStream / caller-side events)."""
        p = C.c_void_p()
        self._check(self.lib.epnn_get_stream(self._h, C.byref(p)))
        return p.value or 0

    def set_stream(self, handle: int = 0):
        """Enqueue on the caller's CUDA stream (integer cudaStream_t, e.g. ``torch.cuda.current_stream().cuda_stream``);
        0 restores the ctx's own stream (epnn_set_stream)."""
        self._check(self.lib.epnn_set_stream(self._h, C.c_void_p(handle or None)))

    def set_shard(self, rank: int, world: int, group=None):
        """Shard the large systems of every following call over ``world`` ranks (epnn_shard_init; collective).  The NCCL
        unique id is made on rank 0 and broadcast through ``torch.distributed`` (any backend); the data-path exchanges
        are ncclAllGather calls inside the library, on this ctx's stream.  ``world == 1`` switches sharding off."""
        if world > 1:
            from .shard import broadcast_unique_id
            uid = broadcast_unique_id(self.lib, rank, group, self.device)
            self._check(self.lib.epnn_shard_init(self._h, rank, world, uid))
        else:
            self._check(self.lib.epnn_shard_init(self._h, 0, 1, None))

    @property
    def shard_state(self):
        """{"calls", "bytes"}: all-gathers issued and bytes received by this rank since ``set_shard``."""
        calls, nbytes = C.c_int64(0), C.c_int64(0)
        self._check(self.lib.epnn_shard_stats(self._h, C.byref(calls), C.byref(nbytes)))
        return {"calls": calls.value, "bytes": nbytes.value}

    def measure_fp32_peak(self, repeats: int = 5) -> float:
        """Measured FP32 FMA peak of this GPU in TFLOP/s (epnn_measure_fp32_peak)."""
        out = C.c_double(0.0)
        self._check(self.lib.epnn_measure_fp32_peak(self._h, repeats, C.byref(out)))
        return out.value

    def pinned_empty(self, shape, dtype):
        """numpy array backed by page-locked host memory (epnn_host_alloc); freed by ``free_pinned``."""
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        p = C.c_void_p()
        rc = self.lib.epnn_host_alloc(C.byref(p), max(n, 1))
        if rc != 0:
            raise _capi.EpnnError(rc, "epnn_host_alloc failed")
        buf = (C.c_char * max(n, 1)).from_address(p.value)
        a = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
        self._pinned = getattr(self, "_pinned", [])
        self._pinned.append(p)
        return a

    def free_pinned(self):
        """Frees every buffer handed out by ``pinned_empty``.  The numpy views of those buffers must not be used afterwards
        (they are plain views of the page-locked memory, not owners)."""
        for p in getattr(self, "_pinned", []):
            self.lib.epnn_host_free(p)
        self._pinned = []

    # ------------------------------------------------------------------ hot path
    def infer_batch(self, offsets, xyz, species, Q, npad=None, want_f64: bool = False, out=None):
        """Charges for a packed batch (see epnn_infer_batch in include/epnn_b200.h).  Host numpy arrays."""
        offsets = _as(offsets, np.int32)
        xyz = _as(xyz, np.float32)
        species = _as(species, np.int32)
        Q = _as(Q, np.float32)
        n_sys = offsets.shape[0] - 1
        n_atoms = int(offsets[-1]) if n_sys >= 0 and offsets.size else 0
        if xyz.size != 3 * n_atoms or species.size != n_atoms or Q.size != n_sys:
            raise ValueError("array sizes are inconsistent with atom_offsets")
        npad_a = None if npad is None else _as(np.broadcast_to(npad, (n_sys,)), np.int32)
        if out is not None and (not isinstance(out, np.ndarray) or out.dtype != np.float32 or out.size != n_atoms
                                or not out.flags.c_contiguous or not out.flags.writeable):
            raise ValueError("out must be a writeable C-contiguous float32 array with one entry per atom")
        q32 = out if out is not None else np.empty(n_atoms, np.float32)
        q64 = np.empty(n_atoms, np.float64) if want_f64 else None
        st = _capi.Stats()
        self._check(self.lib.epnn_infer_batch(self._h, n_sys, _ptr(offsets), _ptr(xyz), _ptr(species), _ptr(Q),
                                              _ptr(npad_a), _ptr(q32), _ptr(q64), C.byref(st)))
        self.last_stats = st.as_dict()
        return (q32, q64) if want_f64 else q32

    def infer_batch_dev(self, offsets_host, xyz_dev: int, species_dev: int, Q_dev: int, npad_host, q_out_dev: int,
                        q_out64_dev: int = 0):
        """Device-pointer variant: the ``*_dev`` arguments are raw CUDA device addresses (ints)."""
        offsets_host = _as(offsets_host, np.int32)
        n_sys = offsets_host.shape[0] - 1
        npad_a = None if npad_host is None else _as(np.broadcast_to(npad_host, (n_sys,)), np.int32)
        st = _capi.Stats()
        self._check(self.lib.epnn_infer_batch_dev(self._h, n_sys, _ptr(offsets_host), C.c_void_p(xyz_dev),
                                                  C.c_void_p(species_dev), C.c_void_p(Q_dev), _ptr(npad_a),
                                                  C.c_void_p(q_out_dev), C.c_void_p(q_out64_dev or None), C.byref(st)))
        self.last_stats = st.as_dict()

    def electrostatics(self, offsets, xyz, q, fragment=None, potential: bool = False):
        """Coulomb energy (e^2/A), dipole (e*A, about the unweighted centroid) and, with ``potential``, the potential at
        every atom (e/A) of each system of a packed batch, in FP64 on the GPU (epnn_electrostatics in
        include/epnn_b200.h).  ``q`` is one charge per atom (float32 charges are widened to float64); ``fragment`` is an
        optional int label per atom: only pairs with different labels count in the energy and the potential, so a
        dimer labelled by its split gives the inter-monomer energy.  Returns ``{"energy": (S,), "dipole": (S, 3)
        [, "phi": (n_atoms,)]}`` float64 arrays."""
        offsets = _as(offsets, np.int32)
        xyz = _as(xyz, np.float32)
        q = _as(q, np.float64)
        n_sys = offsets.shape[0] - 1
        n_atoms = int(offsets[-1]) if n_sys >= 0 and offsets.size else 0
        frag = None if fragment is None else _as(fragment, np.int32)
        if xyz.size != 3 * n_atoms or q.size != n_atoms or (frag is not None and frag.size != n_atoms):
            raise ValueError("array sizes are inconsistent with atom_offsets")
        out = {"energy": np.empty(n_sys, np.float64), "dipole": np.empty((n_sys, 3), np.float64)}
        if potential:
            out["phi"] = np.empty(n_atoms, np.float64)
        self._check(self.lib.epnn_electrostatics(self._h, n_sys, _ptr(offsets), _ptr(xyz), _ptr(q), _ptr(frag),
                                                 _ptr(out["energy"]), _ptr(out["dipole"]), _ptr(out.get("phi"))))
        return out

    def electrostatics_dev(self, offsets_host, xyz_dev: int, q_dev: int, fragment_dev: int = 0, energy_dev: int = 0,
                           dipole_dev: int = 0, phi_dev: int = 0):
        """Device-pointer variant of :meth:`electrostatics`: the ``*_dev`` arguments are raw CUDA device addresses (ints,
        0 = NULL); ``q_dev`` holds float64 charges, e.g. the ``q_out64_dev`` of :meth:`infer_batch_dev`."""
        offsets_host = _as(offsets_host, np.int32)
        n_sys = offsets_host.shape[0] - 1
        self._check(self.lib.epnn_electrostatics_dev(self._h, n_sys, _ptr(offsets_host), C.c_void_p(xyz_dev),
                                                     C.c_void_p(q_dev), C.c_void_p(fragment_dev or None),
                                                     C.c_void_p(energy_dev or None), C.c_void_p(dipole_dev or None),
                                                     C.c_void_p(phi_dev or None)))

    def potential_points(self, offsets, xyz, q, point_offsets, points, field: bool = False):
        """Potential phi(p) = sum_j q_j / r_pj (e/A) and, with ``field``, E(p) = sum_j q_j (p - x_j) / r_pj^3 (e/A^2) of
        the charges of each system at its own points, in FP64 on the GPU (epnn_potential_points in include/epnn_b200.h).
        System s owns the points ``points[point_offsets[s]:point_offsets[s + 1]]`` (a system may have none); atoms at
        r = 0 from a point are skipped.  Returns ``{"phi": (P,) [, "field": (P, 3)]}`` float64 arrays."""
        offsets = _as(offsets, np.int32)
        xyz = _as(xyz, np.float32)
        q = _as(q, np.float64)
        poff = _as(point_offsets, np.int64)
        pts = _as(points, np.float64)
        n_sys = offsets.shape[0] - 1
        n_atoms = int(offsets[-1]) if n_sys >= 0 and offsets.size else 0
        if poff.shape[0] != offsets.shape[0]:
            raise ValueError("point_offsets must have one entry per system plus one, like atom_offsets")
        n_pts = int(poff[-1]) if poff.size else 0
        if xyz.size != 3 * n_atoms or q.size != n_atoms or pts.size != 3 * n_pts:
            raise ValueError("array sizes are inconsistent with atom_offsets / point_offsets")
        out = {"phi": np.empty(n_pts, np.float64)}
        if field:
            out["field"] = np.empty((n_pts, 3), np.float64)
        self._check(self.lib.epnn_potential_points(self._h, n_sys, _ptr(offsets), _ptr(xyz), _ptr(q), _ptr(poff),
                                                   _ptr(pts), _ptr(out["phi"]), _ptr(out.get("field"))))
        return out

    def potential_points_dev(self, offsets_host, xyz_dev: int, q_dev: int, point_offsets_host, points_dev: int,
                             phi_dev: int = 0, field_dev: int = 0):
        """Device-pointer variant of :meth:`potential_points`: the ``*_dev`` arguments are raw CUDA device addresses (ints,
        0 = NULL); both offset arrays stay on the host.  ``q_dev`` holds float64 charges, e.g. the ``q_out64_dev`` of
        :meth:`infer_batch_dev`."""
        offsets_host = _as(offsets_host, np.int32)
        poff = _as(point_offsets_host, np.int64)
        n_sys = offsets_host.shape[0] - 1
        if poff.shape[0] != offsets_host.shape[0]:
            raise ValueError("point_offsets must have one entry per system plus one, like atom_offsets")
        self._check(self.lib.epnn_potential_points_dev(self._h, n_sys, _ptr(offsets_host), C.c_void_p(xyz_dev),
                                                       C.c_void_p(q_dev), _ptr(poff), C.c_void_p(points_dev or None),
                                                       C.c_void_p(phi_dev or None), C.c_void_p(field_dev or None)))

    def neighbors(self, offsets, xyz, which: int = 0):
        """(rowptr, col) CSR of the is_near set (which=0) or the e != 0 set (which=1); global atom indices."""
        offsets = _as(offsets, np.int32)
        xyz = _as(xyz, np.float32)
        n_sys = offsets.shape[0] - 1
        n_atoms = int(offsets[-1])
        rowptr = np.zeros(n_atoms + 1, np.int32)
        cap = max(64, 24 * n_atoms)
        while True:
            col = np.empty(cap, np.int32)
            nnz = C.c_int64(0)
            rc = self.lib.epnn_neighbors(self._h, n_sys, _ptr(offsets), _ptr(xyz), which, _ptr(rowptr), _ptr(col), cap,
                                         C.byref(nnz))
            if rc == -4:
                cap = int(nnz.value)
                continue
            self._check(rc)
            return rowptr, col[:nnz.value].copy()

    def init_edges(self, xyz):
        xyz = _as(xyz, np.float32)
        n = xyz.shape[0]
        e = np.empty((n, n, 48), np.float32)
        self._check(self.lib.epnn_init_edges(self._h, n, _ptr(xyz), _ptr(e)))
        return e

    def hidden(self, n_atoms: int):
        h = np.empty((n_atoms, 48), np.float32)
        self._check(self.lib.epnn_get_hidden(self._h, _ptr(h), h.size))
        return h

    def infer_dense(self, h, e, x, q, mask):
        """Keras-shaped compat path (epnn_infer_dense): arrays (B,N,N,.) as gen_padded_init_state makes them."""
        h = _as(h, np.float32); e = _as(e, np.float32); x = _as(x, np.float32); q = _as(q, np.float32)
        mask = _as(mask, np.float32)
        B, N = e.shape[0], e.shape[1]
        out = np.empty((B, N), np.float32)
        self._check(self.lib.epnn_infer_dense(self._h, B, N, _ptr(h), _ptr(e), _ptr(x), _ptr(q), _ptr(mask), _ptr(out)))
        return out.reshape(B, N, 1)
