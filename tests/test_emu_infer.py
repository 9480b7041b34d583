"""A WHOLE charge inference on the CPU through the product's own code: weights packed and folded by epnn_pack.h (what
epnn_create runs), then every kernel of the FP32 path -- neighbour list, descriptors, far lists, bundle kernels, row-group
kernels, per-atom kernel -- executed by the warp emulation (tools/emu/emu_infer.cpp) in run_chunk's launch order.
Compared with the float64 oracle and with the reference's own shipped predictions.  Variants ("variant" argument of
emu_infer): 0 the round-1 warp-tile kernels ("pair_const" 0), 1 the pair-per-thread kernels everywhere (epnn_bundle_const.cu,
epnn_atom_const.cu, epnn_gnn_far_const.cu; "pair_const" 1), 2 variant 0 with the mma.sync electron-passing kernel
(epnn_bundle_mma.cu, "pair_tensor" 1; its fragment layout is emulated lane by lane), 3 the shipped FP32 set ("pair_const" 2):
the row-run GNN bundle kernel (epnn_bundle_run.cu), the pair-per-thread electron-passing bundle kernel and far_const
for large systems, with the SIMT per-atom kernel (the tensor per-atom kernel has its own emulation test).
This is test infrastructure, not a fallback: nothing in epnn_b200/ can reach it."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import epnn_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "build", "libemu_infer.so")
TOL_FP32 = {"decay_model_weights": 1e-5, "model2_weights": 5e-5, "model_weights": 1e-3}      # tests/test_gpu_parity.py


@pytest.fixture(scope="module")
def emu():
    os.makedirs(os.path.join(ROOT, "build"), exist_ok=True)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-pthread", "-DEPNN_CPU_EMU",
                           "-Wno-unknown-pragmas", "-o", LIB, os.path.join(ROOT, "tools", "emu", "emu_infer.cpp")])
    lib = C.CDLL(LIB)
    lib.emu_infer.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_int] + [C.c_void_p] * 5 + [C.c_int, C.c_int] + [C.c_void_p] * 4
    return lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _infer(emu, w, offs, xyz, sp, Q, npad, pair_const=0, dedup=1):
    n = int(offs[-1])
    packed = w.packed()
    q32 = np.full(n, np.nan, np.float32); q64 = np.full(n, np.nan); h = np.full((n, 48), np.nan, np.float32)
    rows = np.zeros(1, np.int64)
    offs = np.ascontiguousarray(offs, np.int32); xyz = np.ascontiguousarray(xyz, np.float32)
    sp = np.ascontiguousarray(sp, np.int32); Q = np.ascontiguousarray(Q, np.float32)
    npad_a = None if npad is None else np.ascontiguousarray(np.broadcast_to(npad, (len(Q),)), np.int32)
    rc = emu.emu_infer(w.T, w.n_x, _p(packed), packed.size, len(Q), _p(offs), _p(xyz), _p(sp), _p(Q), _p(npad_a), pair_const, dedup,
                       _p(q32), _p(q64), _p(h), _p(rows))
    assert rc == 0
    return q32, q64, h, int(rows[0])


@pytest.mark.parametrize("pair_const", [0, 1, 2, 3])      # the emulated kernel set ("variant", see the module docstring)
def test_emulated_inference_reproduces_shipped_predictions(emu, weights, mixed, val871, pair_const):
    """decay_model_weights, pad 41: the reference's own predictions (models/model_systems/test_pred_charges.npy)."""
    w = weights["decay_model_weights"]
    pick = [0, 200, 400, 600, 800, 870]
    idx = [mixed.index[val871["names"][k]] for k in pick]
    offs, xyz, sp, Q = mixed.batch(idx, 9)
    q32, q64, _, _ = _infer(emu, w, offs, xyz, sp, Q, 41, pair_const=pair_const)
    for j, k in enumerate(pick):
        n = offs[j + 1] - offs[j]
        assert np.abs(q32[offs[j]:offs[j + 1]] - val871["pred"][k][:n]).max() < 1e-5, (k, pair_const)
    assert np.abs(np.add.reduceat(q64, offs[:-1]) - Q).max() < 1e-6
    ref = O.predict_batch(w, offs, xyz, sp, Q, np.full(len(Q), 41))
    assert np.abs(q64 - ref).max() < 1e-5


@pytest.mark.parametrize("name", ["model2_weights", "model_weights"])
@pytest.mark.parametrize("pair_const", [0, 1, 2, 3])
def test_emulated_inference_live_checkpoints(emu, weights, mixed, name, pair_const):
    """Checkpoints whose hidden state is live: charges AND the GNN-layer output against the oracle (only step 0 collapses)."""
    w = weights[name]
    idx = mixed.usable(w.n_x)[[3, 1400, 2900, 4100]].tolist()
    offs, xyz, sp, Q = mixed.batch(idx, w.n_x)
    npad = np.array([41, int(offs[2] - offs[1]), 41, 41])               # one system without padding
    q32, q64, h, _ = _infer(emu, w, offs, xyz, sp, Q, npad, pair_const=pair_const)
    ref = O.predict_batch(w, offs, xyz, sp, Q, npad)
    assert np.abs(q64 - ref).max() < TOL_FP32[name], (name, np.abs(q64 - ref).max())
    assert np.abs(np.add.reduceat(q64, offs[:-1]) - Q).max() < 1e-6
    for k in range(len(idx)):
        tr = {}
        O.forward_factorised(w, xyz[offs[k]:offs[k + 1]], sp[offs[k]:offs[k + 1]], Q[k], int(npad[k]), trace=tr)
        assert tr["h"].std(axis=0).max() > 1e-3
        assert np.abs(h[offs[k]:offs[k + 1]] - tr["h"]).max() < 2e-4 * np.abs(tr["h"]).max(), (name, k)


@pytest.mark.parametrize("pair_const,dedup", [(0, 1), (0, 0), (1, 1), (3, 1), (3, 0)])
def test_emulated_inference_with_a_large_system(emu, weights, mixed, protein, pair_const, dedup):
    """A 90-atom protein cut (row-group kernels, three partial-sum planes, species tables) between two small molecules."""
    w = weights["decay_model_weights"]
    offs, xyz, sp, Q = mixed.batch(mixed.usable(9)[[10, 2000]].tolist(), 9)
    n0 = int(offs[1])
    cut = slice(300, 390)
    offs = np.array([0, n0, n0 + 90, n0 + 90 + int(offs[2] - offs[1])], np.int32)
    xyz = np.concatenate([xyz[:n0], protein["xyz"][cut], xyz[n0:]]).astype(np.float32)
    sp = np.concatenate([sp[:n0], O.species_from_Z(protein["Z"][cut], 9), sp[n0:]]).astype(np.int32)
    Q = np.array([Q[0], 1.0, Q[1]], np.float32)
    npad = np.array([41, 96, 29], np.int32)
    q32, q64, _, rows = _infer(emu, w, offs, xyz, sp, Q, npad, pair_const=pair_const, dedup=dedup)
    ref = O.predict_batch(w, offs, xyz, sp, Q, npad)
    assert np.abs(q64 - ref).max() < 1e-5, np.abs(q64 - ref).max()
    assert np.abs(np.add.reduceat(q64, offs[:-1]) - Q).max() < 1e-6
    assert rows == (3 * 90 if dedup else 0)                              # 3 of the 5 steps collapse for this checkpoint (DESIGN.md)


@pytest.mark.parametrize("seed,pair_const", [(1, 0), (2, 0), (3, 1), (4, 3)])
def test_emulated_inference_random_systems(emu, weights, seed, pair_const):
    """Randomly sized synthetic systems (1 .. 48 atoms and a few larger ones, jittered-lattice geometries, random species
    and net charges, padded and unpadded) -- tile and bundle boundaries fall wherever they fall."""
    w = weights["model2_weights"]                     # T = 3, live hidden state
    rng = np.random.default_rng(seed)
    sizes = list(rng.integers(1, 49, size=7)) + [int(rng.integers(49, 80))] + list(rng.integers(1, 30, size=3))
    rng.shuffle(sizes)
    offs, xyz, sp = [0], [], []
    for n in sizes:
        side = int(np.ceil(n ** (1 / 3))) + 1
        grid = np.stack(np.meshgrid(*[np.arange(side)] * 3, indexing="ij"), -1).reshape(-1, 3)
        pts = grid[rng.permutation(len(grid))[:n]] * 1.3 + rng.normal(scale=0.12, size=(n, 3))
        xyz.append(pts); sp.append(rng.integers(0, 8, size=n)); offs.append(offs[-1] + n)
    offs = np.array(offs, np.int32)
    xyz = np.concatenate(xyz).astype(np.float32)
    sp = np.concatenate(sp).astype(np.int32)
    Q = rng.integers(-2, 3, size=len(sizes)).astype(np.float32)
    npad = np.array([n if k % 2 else n + int(rng.integers(1, 12)) for k, n in enumerate(sizes)], np.int32)
    q32, q64, _, _ = _infer(emu, w, offs, xyz, sp, Q, npad, pair_const=pair_const)
    ref = O.predict_batch(w, offs, xyz, sp, Q, npad)
    scale = max(1.0, np.abs(ref).max())
    assert np.abs(q64 - ref).max() < 5e-5 * scale, (seed, np.abs(q64 - ref).max(), scale)
    assert np.abs(np.add.reduceat(q64, offs[:-1]) - Q).max() < 1e-6 * scale
