"""CPU warp emulation of the row-run GNN bundle kernel (epnn_bundle_run.cu, the FP32 default for small systems).

The kernel source is compiled for the host with -DEPNN_CPU_EMU (tools/emu/cuda_emu.h) and run on the lists built by
tests/emu_common.py from the adversarial small systems of tests/small_cases.py: maximal and empty near lists, lists of
31 ... 66 slots around the 32-lane cut, rows spread over several lanes, bundles whose systems have different pad weights,
and bundles where only some systems have species-equal v rows (the far-column collapse ``use0`` is then exact for some
rows of the bundle and wrong for others, so the whole bundle must take the plain far list).  Its message sums S are
compared with a float64 evaluation of the reference formula (charge_gn.py:62-70)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from emu_common import build_lists_raw, csr, gnn_reference, large_system_tables, weights as random_weights
from small_cases import edge_counts, small_batch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "build", "libemu_bundle_run.so")
RTOL = 2e-5                       # as the other bundle emulations (tests/test_emu_pair_const.py), but row by row: the pad
                                  # weights (up to 952 here) make some rows a thousand times larger than others


def row_err(S, ref):
    return float((np.abs(S - ref).max(1) / np.abs(ref).max(1)).max())


@pytest.fixture(scope="module")
def emu():
    os.makedirs(os.path.join(ROOT, "build"), exist_ok=True)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-pthread", "-DEPNN_CPU_EMU",
                           "-Wno-unknown-pragmas", "-o", LIB, os.path.join(ROOT, "tools", "emu", "emu_bundle_run.cpp")])
    lib = C.CDLL(LIB)
    lib.emu_bundle_run.argtypes = [C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 14 + [C.c_int] + [C.c_void_p] * 7
    return lib


@pytest.fixture(scope="module")
def case():
    """The small-system batch (n_x = 9), its lists, random weights and the float64 reference of S."""
    rng = np.random.default_rng(5)
    offs, xyz, sp, _, npad, _ = small_batch(9)
    # species-equal v rows in every third system: bundles with several systems mix equal and unequal ones
    L = build_lists_raw(offs, xyz, sp, npad, rng, equal_v_systems=list(range(0, len(npad), 3)))
    rowptr, col = csr(L)
    pid = large_system_tables(L)[3]
    b0_of = np.zeros(L["n"], np.int64)
    for b0, bn in L["bundles"]:
        b0_of[b0:b0 + bn] = b0
    rows_of = np.repeat(np.arange(L["n"]), np.diff(rowptr))
    rowl = np.concatenate([(rows_of - b0_of[rows_of]).astype(np.uint8), np.zeros(16, np.uint8)])
    W = random_weights(rng)
    return dict(L=L, rowptr=rowptr, col=col, pid=pid, rowl=rowl, W=W, ref=gnn_reference(L, W, npad))


def _run(emu, c, dedup, n_warps):
    L, W = c["L"], c["W"]
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    S = np.full((L["n"], 32), np.nan, np.float32)
    counter = np.zeros(1, np.int32)
    slots = np.zeros(2, np.uint64)
    weights = np.concatenate([W["Cw"].ravel(), W["W2"].ravel(), W["b2"], W["x32"]]).astype(np.float32)
    bundles = np.ascontiguousarray(L["bundles"], np.int32)
    rc = emu.emu_bundle_run(n_warps, p(weights), len(bundles), p(bundles), p(counter),
                            p(c["rowptr"]), p(c["col"]), p(c["pid"]), p(c["rowl"]), p(L["coef"]), p(L["ustart"]),
                            p(L["far_off"]), p(L["far_list"]), p(L["far0_off"]), p(L["far0_list"]), p(L["far0_w"]), p(L["rep"]), int(dedup),
                            p(L["atom_sys"]), p(L["offs"]), p(L["npad"]), p(L["u"]), p(L["v"]), p(S), p(slots))
    assert rc == 0
    return S, slots


@pytest.mark.parametrize("n_x", [9, 10])
def test_the_batch_reaches_the_edges_it_names(n_x):
    """Counted on the oracle's own neighbour sets: the edges tests/small_cases.py names occur in the batch that the GPU
    comparison (n_x 9 and 10) and this emulation (n_x 9) run."""
    offs, xyz, sp, _, npad, labels = small_batch(n_x)
    counts, coincident, far_not_near = edge_counts(offs, xyz, npad)
    by = dict(zip(labels, counts))
    assert by["ball48"]["near"] == 48 * 47 and by["ball48"]["maxdeg"] == 47
    assert by["lattice48"]["near"] == 0 and by["lattice48"]["far"] == 48 * 48 + 48
    for k in (30, 32, 34, 64, 66):
        assert by[f"near{k}"]["near"] == k
    for k in (31, 32, 33, 64, 65):
        assert by[f"far{k}"]["far"] == k and by[f"far{k}"]["nbr"] == 0
    for lab in ("cluster3", "cluster4_pad", "cluster5", "cluster6_pad"):
        n = int(lab[7])
        assert by[lab]["near"] == n * (n - 1) < 32                     # J = 1, each row over n - 1 lanes
    assert coincident >= 1 and far_not_near >= 3
    n = np.diff(offs)
    assert {0, 1, 1000 - 48, 255 - 6, 41 - 12} <= set((npad - n).tolist())
    assert (n == 1).sum() >= 48 and set(range(n_x - 1)) <= set(sp.tolist())     # every species, the highest n_x - 2 included


@pytest.mark.parametrize("dedup", [0, 1])
def test_emulated_run_kernel_matches_the_definition(emu, case, dedup):
    S, slots = _run(emu, case, dedup, n_warps=8)
    assert np.isfinite(S).all()                                        # S starts as NaN: every row of every bundle is written
    err = row_err(S, case["ref"])
    assert err < RTOL, err
    L = case["L"]
    assert int(slots[0]) == int(case["rowptr"][-1])                     # every CSR entry is one near slot
    if not dedup:
        assert int(slots[1]) == len(L["far_list"])
    else:                                                               # some bundles collapse their far columns, some cannot
        assert len(L["far0_list"]) < int(slots[1]) < len(L["far_list"])


def test_use0_is_decided_for_the_whole_bundle(emu, case):
    """A bundle that mixes systems with and without species-equal v rows must take the plain far list: the collapsed
    list is exact only when every row of the bundle has its representative's v."""
    L = case["L"]
    mixed_bundles = 0
    for b0, bn in L["bundles"]:
        eq = [np.array_equal(L["v"][i], L["v"][L["rep"][i]]) for i in range(b0, b0 + bn)]
        mixed_bundles += any(eq) and not all(eq) and any(L["rep"][i] != i for i in range(b0, b0 + bn) if eq[i - b0])
    assert mixed_bundles >= 3
    S, _ = _run(emu, case, 1, n_warps=3)
    assert row_err(S, case["ref"]) < RTOL


def test_run_kernel_is_bitwise_independent_of_the_warp_count(emu, case):
    """Every addition has a fixed position: which warp runs a bundle does not change a bit of S."""
    for dedup in (0, 1):
        a, _ = _run(emu, case, dedup, n_warps=1)
        b, _ = _run(emu, case, dedup, n_warps=8)
        assert np.array_equal(a, b), dedup
