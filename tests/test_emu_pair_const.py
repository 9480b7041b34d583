"""CPU warp emulation of the pair-per-thread bundle kernels, epnn_b200/csrc/epnn_bundle_const.cu ("pair_const" 1; its
electron-passing variant is also part of the FP32 default set, "pair_const" 2).

The kernel source is compiled for the host with -DEPNN_CPU_EMU (tools/emu/cuda_emu.h: every lane is a host thread,
shuffles / votes / __syncwarp through a per-warp barrier, shared memory a host buffer) and run on index lists built here
from the reference's own molecules exactly the way the CUDA prep kernels build them (pair lists sorted by i, per-bundle
far lists, species-compressed far lists, representatives).  Its outputs -- the message sums S of a message-passing step
and the per-pair transfers delta of an electron-passing pass -- are compared with a direct float64 evaluation of the
reference formulas (charge_gn.py:62-70, :101-116).  This checks the kernel's indexing, control flow, shared-memory
layout and summation logic without a GPU; it says nothing about performance."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from emu_common import build_lists as _build_lists, build_lists_raw as _build_lists_raw, epn_reference, gnn_reference as _gnn_reference, \
    relu as _relu, weights as _weights

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "build", "libemu_bundle_const.so")


@pytest.fixture(scope="module")
def emu():
    os.makedirs(os.path.join(ROOT, "build"), exist_ok=True)
    src = os.path.join(ROOT, "tools", "emu", "emu_bundle_const.cpp")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-pthread", "-DEPNN_CPU_EMU", "-Wno-unknown-pragmas",
                           "-o", LIB, src])
    return C.CDLL(LIB)


def _run(emu, L, W, epn, dedup, n_warps):
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    S = np.full((L["n"], 32), np.nan, np.float32)
    delta = np.full(L["P"], np.nan, np.float32)
    counter = np.zeros(1, np.int32)
    weights = np.concatenate([W["Cw"].ravel(), W["W2"].ravel(), W["b2"], W["x32"]]).astype(np.float32)
    emu.emu_bundle_const.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 13 + [C.c_int] + [C.c_void_p] * 7
    rc = emu.emu_bundle_const(int(epn), n_warps, p(weights), len(L["bundles"]), p(L["bundles"]), p(counter),
                              p(L["ustart"]), p(L["pair_i"]), p(L["pair_j"]), p(L["near"]), p(L["coef"]),
                              p(L["far_off"]), p(L["far_list"]), p(L["far0_off"]), p(L["far0_list"]), p(L["far0_w"]), p(L["rep"]), int(dedup),
                              p(L["atom_sys"]), p(L["offs"]), p(L["npad"]), p(L["u"]), p(L["v"]), p(S), p(delta))
    assert rc == 0
    return S, delta


@pytest.mark.parametrize("dedup", [0, 1])
def test_emulated_gnn_bundle_kernel_matches_the_definition(emu, mixed, dedup):
    rng = np.random.default_rng(7)
    idx = mixed.usable(9)[[5, 40, 300, 1500, 1501, 2500, 3000, 3600, 4000]].tolist()
    sizes = np.array([mixed.offsets[i + 1] - mixed.offsets[i] for i in idx])
    npad = np.where(np.arange(len(idx)) % 3 == 1, sizes, 41)            # every third system without padding
    L = _build_lists(mixed, idx, 9, npad, rng, equal_v_systems=[0, 1, 2, 3, 6])
    assert len(L["bundles"]) >= 3
    W = _weights(rng)
    S, _ = _run(emu, L, W, epn=False, dedup=dedup, n_warps=3)
    Cw, W2, b2, b1 = (W[k].astype(np.float64) for k in ("Cw", "W2", "b2", "x32"))
    u, v = L["u"].astype(np.float64), L["v"].astype(np.float64)
    ce = {}
    for p in range(L["P"]):
        c = L["coef"][p].astype(np.float64) @ Cw
        ce[(L["pair_i"][p], L["pair_j"][p])] = c
        ce[(L["pair_j"][p], L["pair_i"][p])] = c
    ref = np.zeros((L["n"], 32))
    for i in range(L["n"]):
        s = L["atom_sys"][i]
        for j in range(L["offs"][s], L["offs"][s + 1]):                 # ALL columns of the system, the self pair included
            ref[i] += _relu(_relu(ce.get((i, j), 0.0) + u[i] + v[j]) @ W2 + b2)
        n_s = L["offs"][s + 1] - L["offs"][s]
        ref[i] += (npad[s] - n_s) * _relu(_relu(u[i] + b1) @ W2 + b2)   # padded atoms: a_j = 0, e = 0 -> v = b1
    assert np.isfinite(S).all()
    assert np.abs(S - ref).max() < 2e-5 * np.abs(ref).max(), np.abs(S - ref).max()


def test_emulated_epn_bundle_kernel_matches_the_definition(emu, mixed):
    rng = np.random.default_rng(8)
    idx = mixed.usable(9)[[7, 41, 301, 1600, 2501, 3001, 4100]].tolist()
    L = _build_lists(mixed, idx, 9, np.full(len(idx), 41), rng, equal_v_systems=[])
    L["near"][::7] = 0          # pairs with e != 0 that fail is_near are rare (2.994 A <= D < 3 A): plant some, the kernel only reads the flag
    W = _weights(rng)
    _, delta = _run(emu, L, W, epn=True, dedup=1, n_warps=2)
    Cw, W2, b2, w3 = (W[k].astype(np.float64) for k in ("Cw", "W2", "b2", "x32"))
    u, v = L["u"].astype(np.float64), L["v"].astype(np.float64)
    ref = np.zeros(L["P"])
    for p in range(L["P"]):
        i, j = L["pair_i"][p], L["pair_j"][p]
        c = L["coef"][p].astype(np.float64) @ Cw
        f_ij = _relu(_relu(c + u[i] + v[j]) @ W2 + b2) @ w3
        f_ji = _relu(_relu(c + u[j] + v[i]) @ W2 + b2) @ w3
        ref[p] = 0.5 * (f_ij - f_ji) * L["near"][p]                     # charge_gn.py:116
    assert L["near"].min() == 0 and L["near"].max() == 1               # both kinds of pair are present
    assert np.isfinite(delta).all()
    assert np.abs(delta - ref).max() < 2e-5 * max(1.0, np.abs(ref).max()), np.abs(delta - ref).max()


@pytest.mark.parametrize("dedup", [0, 1])
def test_emulated_gnn_edge_cases(emu, mixed, dedup):
    """A single atom, two atoms beyond the cutoff (no e != 0 pair at all), a bundle filled to exactly 48 atoms (last
    staged row next to the pad row), a bundle without any padded system, more warps than bundles."""
    rng = np.random.default_rng(11)
    ok = mixed.usable(9)
    sizes = np.diff(mixed.offsets)[ok]
    i29 = int(ok[np.nonzero(sizes == 29)[0][0]])
    i19 = int(ok[np.nonzero(sizes == 19)[0][0]])
    o2, x2, s2, _ = mixed.batch([i29, i19], 9)
    o3, x3, s3, _ = mixed.batch([int(ok[3])], 9)
    offs = np.concatenate([o2, [49, 51], 51 + o3[1:]]).astype(np.int32)                 # 29 | 19 | 1 | 2 | n
    xyz = np.concatenate([x2, [[0.0, 0.0, 0.0]], [[0.0, 0.0, 0.0], [5.0, 0.0, 0.0]], x3]).astype(np.float32)
    sp = np.concatenate([s2, [1], [0, 3], s3]).astype(np.int32)
    npad = np.array([29, 19, 1, 7, 41], np.int32)                      # systems 0, 1, 2 unpadded: the first bundle has no pad slot
    L = _build_lists_raw(offs, xyz, sp, npad, rng, equal_v_systems=[0, 1, 2, 3])
    assert int(L["bundles"][0][1]) == 48 and len(L["bundles"]) == 2
    W = _weights(rng)
    S, _ = _run(emu, L, W, epn=False, dedup=dedup, n_warps=8)
    ref = _gnn_reference(L, W, npad)
    assert np.isfinite(S).all()
    assert np.abs(S - ref).max() < 2e-5 * np.abs(ref).max(), np.abs(S - ref).max()
