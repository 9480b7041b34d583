"""Host-side planning of the inference path (epnn_b200/csrc/epnn_plan.h) through tools/emu/emu_plan.cpp: chunk bounds,
bundle packing, the row slices and unit ranges of sharded calls, the far kernel and its partial-sum planes, and the kernel
choice of every combination of options and precision."""
import ctypes as C
import itertools
import os
import subprocess

import numpy as np
import pytest

from epnn_b200 import _capi
from small_cases import pack_bundles

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "build", "libemu_plan.so")
SMALL_MAX = 48
GNN_TILE, GNN_CONST, GNN_RUN = 0, 1, 2
EPN_TILE, EPN_CONST, EPN_MMA = 0, 1, 2
ATOM_SIMT, ATOM_MMA, ATOM_CONST = 0, 1, 2
FAR_SIMT, FAR_TC, FAR_TC2, FAR_CONST = 0, 1, 2, 3
FIELDS = ["ok", "n_bundles", "has_large", "max_n", "n_rg_large", "sharded", "row_lo", "row_hi", "rg_begin", "rg_end", "n_rowblk",
          "blk_begin", "blk_end", "far", "nsplit", "n_large", "n_cells"]


@pytest.fixture(scope="module")
def emu():
    os.makedirs(os.path.join(ROOT, "build"), exist_ok=True)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-pthread", "-DEPNN_CPU_EMU", "-o", LIB,
                           os.path.join(ROOT, "tools", "emu", "emu_plan.cpp")])
    lib = C.CDLL(LIB)
    lib.emu_plan_chunks.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]
    lib.emu_resolve_kernels.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.emu_plan_chunk.argtypes = [C.c_void_p] + [C.c_int] * 6 + [C.c_void_p] * 3
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _opts(pair_const=2, pair_tensor=0, far_tensor=2, far_tensor_min=16384, far_tensor_impl=1):
    return np.array([pair_const, pair_tensor, far_tensor, far_tensor_min, far_tensor_impl], np.int32)


def plan(emu, offs, sm_count=148, rank=0, world=1, precision=32, atom_tensor=1, **opts):
    offs = np.ascontiguousarray(offs, np.int32)
    n_sys = len(offs) - 1
    bundles = np.zeros(2 * max(n_sys, 1), np.int32)
    out = np.zeros(len(FIELDS), np.int64)
    emu.emu_plan_chunk(_p(offs), n_sys, sm_count, rank, world, precision, atom_tensor, _p(_opts(**opts)), _p(bundles), _p(out))
    p = dict(zip(FIELDS, out.tolist()))
    p["bundles"] = [tuple(b) for b in bundles[:2 * p["n_bundles"]].reshape(-1, 2).tolist()]
    return p


def random_offs(rng, n_sys, large=True):
    pool = [1, 2, 5, 17, 30, 47, 48, 48, 49] + ([49, 60, 97, 130, 600] if large else [])
    return np.concatenate([[0], np.cumsum(rng.choice(pool, size=n_sys))]).astype(np.int32)


def units(offs, size):
    """First rows of the `size`-row units (4-row groups, 32-row blocks) of the systems above SMALL_MAX atoms, in order."""
    return [int(offs[s]) + i for s in range(len(offs) - 1) if offs[s + 1] - offs[s] > SMALL_MAX
            for i in range(0, int(offs[s + 1] - offs[s]), size)]


def reference_bundles(offs):
    """pack_bundles over every run of consecutive systems of at most SMALL_MAX atoms: a larger system ends a bundle."""
    out, s0, n_sys = [], 0, len(offs) - 1
    for s in range(n_sys + 1):
        if s == n_sys or offs[s + 1] - offs[s] > SMALL_MAX:
            if s > s0:
                out += pack_bundles(offs[s0:s + 1])
            s0 = s + 1
    return out


@pytest.mark.parametrize("seed", range(6))
def test_bundles_match_the_reference_packing(emu, seed):
    rng = np.random.default_rng(seed)
    offs = random_offs(rng, 300, large=seed % 2 == 1)
    assert plan(emu, offs)["bundles"] == reference_bundles(offs)
    k = 37                                                  # a chunk that starts inside the batch: chunk-local first atoms
    assert plan(emu, offs[k:])["bundles"] == reference_bundles(offs[k:] - offs[k])


def test_chunk_bounds_are_maximal(emu):
    rng = np.random.default_rng(7)
    for chunk_atoms in (64, 200, 1000):
        offs = random_offs(rng, 400)
        bounds = np.zeros(len(offs), np.int64)
        nb = emu.emu_plan_chunks(_p(offs), len(offs) - 1, chunk_atoms, _p(bounds))
        b = bounds[:nb].tolist()
        assert b[0] == 0 and b[-1] == len(offs) - 1 and all(x < y for x, y in zip(b, b[1:]))
        for s, e in zip(b, b[1:]):
            if e - s > 1:
                assert offs[e] - offs[s] <= chunk_atoms
            else:
                assert offs[e] - offs[s] <= chunk_atoms or offs[s + 1] - offs[s] > chunk_atoms      # a larger system: a chunk of its own
            if e < len(offs) - 1:
                assert offs[e + 1] - offs[s] > chunk_atoms                                         # the next system did not fit


@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("pair_const", [0, 2])
def test_sharded_slices_and_unit_ranges(emu, world, pair_const):
    lib = _capi.load()
    rng = np.random.default_rng(world)
    offs = random_offs(rng, 60)
    offs = np.concatenate([offs, offs[-1] + np.array([1500, 1503])]).astype(np.int32)     # systems of 1 500 and 3 atoms at the end
    n = int(offs[-1])
    groups, blocks = units(offs, 4), units(offs, 32)
    covered_g, covered_b = set(), set()
    for rank in range(world):
        p = plan(emu, offs, rank=rank, world=world, pair_const=pair_const)
        assert p["sharded"] == 1
        lo, hi = C.c_int64(), C.c_int64()
        assert lib.epnn_shard_slice(n, rank, world, C.byref(lo), C.byref(hi)) == 0
        assert (p["row_lo"], p["row_hi"]) == (lo.value, hi.value)
        # a unit belongs to the range when its nominal rows [first, first + size) meet the rank's rows
        want_g = [g for g, a in enumerate(groups) if a + 3 >= lo.value and a < hi.value]
        want_b = [k for k, a in enumerate(blocks) if a + 31 >= lo.value and a < hi.value]
        assert list(range(p["rg_begin"], p["rg_end"])) == want_g, rank
        assert list(range(p["blk_begin"], p["blk_end"])) == want_b, rank
        covered_g |= set(want_g); covered_b |= set(want_b)
    assert covered_g == set(range(len(groups))) and covered_b == set(range(len(blocks)))
    assert p["n_rg_large"] == len(groups) and p["n_rowblk"] == len(blocks)
    # unsharded (world 1), or a chunk without a large system: every row, every unit
    p = plan(emu, offs, rank=0, world=1)
    assert (p["sharded"], p["row_lo"], p["row_hi"], p["rg_begin"], p["rg_end"], p["blk_begin"], p["blk_end"]) == \
        (0, 0, n, 0, len(groups), 0, len(blocks))
    small = np.arange(0, 41, 5, dtype=np.int32)
    p = plan(emu, small, rank=1, world=world)
    assert (p["sharded"], p["has_large"], p["row_lo"], p["row_hi"], p["n_rg_large"], p["far"], p["nsplit"]) == (0, 0, 0, 40, 0, FAR_SIMT, 1)


@pytest.mark.parametrize("sm_count", [1, 2, 8, 148, 1000])
def test_far_kernel_and_planes(emu, sm_count):
    rng = np.random.default_rng(sm_count)
    for trial in range(4):
        offs = random_offs(rng, 20 * (trial + 1))
        offs = np.concatenate([offs, offs[-1] + np.array([200 + 400 * trial])]).astype(np.int32)
        n_rg, n_blk = len(units(offs, 4)), len(units(offs, 32))
        for far_tensor, impl, pair_const in itertools.product([0, 1], [1, 2], [0, 1, 2]):
            for precision in (32, 48, 64):
                p = plan(emu, offs, sm_count=sm_count, precision=precision, pair_const=pair_const, far_tensor=far_tensor,
                         far_tensor_impl=impl)
                assert p["n_rg_large"] == n_rg and p["max_n"] == int(np.diff(offs).max())
                if far_tensor and precision != 64:
                    assert p["far"] == (FAR_TC2 if impl == 2 else FAR_TC)
                    assert p["nsplit"] == min(max(-(-8 * sm_count // n_rg), 1), 15) + 1
                elif pair_const and precision != 64:
                    assert p["far"] == FAR_CONST
                    assert p["nsplit"] == min(max(-(-32 * sm_count // n_blk), 1), 15) + 1
                else:
                    assert p["far"] == FAR_SIMT
                    assert p["nsplit"] == min(max(-(-64 * sm_count // n_rg), 1), 32)
                assert (2 <= p["nsplit"] <= 16) if p["far"] != FAR_SIMT else (1 <= p["nsplit"] <= 32)


def test_far_tensor_auto_threshold(emu):
    """gnn_far_tensor 2: the tensor-core far kernel once the largest system of the chunk has at least gnn_far_tensor_min atoms."""
    for max_n, pair_const in itertools.product([99, 100, 101], [0, 1, 2]):
        offs = np.array([0, 20, 20 + max_n, 40 + max_n], np.int32)
        p = plan(emu, offs, pair_const=pair_const, far_tensor=2, far_tensor_min=100)
        assert p["far"] == (FAR_TC if max_n >= 100 else FAR_CONST if pair_const else FAR_SIMT), (max_n, pair_const)


def test_cell_budget(emu):
    offs = np.cumsum([0, 10, 512, 513, 12, 2000]).astype(np.int32)           # 513 and 2 000 atoms take a cell list, 512 does not
    p = plan(emu, offs)
    assert (p["ok"], p["n_large"], p["n_cells"]) == (1, 2, 4 * 513 + 64 + 4 * 2000 + 64)
    big = np.array([0, 600_000_000], np.int32)                               # 4 n + 64 cells reach 2^31
    assert plan(emu, big)["ok"] == 0


def expected_choice(precision, atom_tensor, pair_const, pair_tensor, far_tensor, far_tensor_impl):
    """The kernel selection of the FP32 paths (precision 32 and 48; precision 64 runs the warp-tile FP64 kernels)."""
    fp32 = precision != 64
    pc = pair_const if fp32 else 0
    gnn = {0: GNN_TILE, 1: GNN_CONST, 2: GNN_RUN}[pc]
    epn = EPN_MMA if fp32 and pair_tensor else EPN_CONST if pc else EPN_TILE
    scoped = ATOM_MMA if precision == 32 and atom_tensor else ATOM_SIMT
    atom = ATOM_CONST if precision == 32 and pc == 1 else scoped
    far = FAR_CONST if pc else FAR_SIMT
    far_tc = (FAR_TC2 if far_tensor_impl == 2 else FAR_TC) if fp32 and far_tensor else far
    far_tc_min = (0 if far_tensor == 1 else 16384) if fp32 and far_tensor else 2**31 - 1
    return [gnn, epn, atom, scoped, far, far_tc, far_tc_min, int(gnn == GNN_RUN), int(gnn != GNN_RUN)]


def test_kernel_choice_table(emu):
    out = np.zeros(9, np.int32)
    for precision, atom_tensor, pair_const, pair_tensor, far_tensor, impl in itertools.product(
            [32, 48, 64], [0, 1], [0, 1, 2], [0, 1], [0, 1, 2], [1, 2]):
        emu.emu_resolve_kernels(precision, atom_tensor, _p(_opts(pair_const, pair_tensor, far_tensor, 16384, impl)), _p(out))
        want = expected_choice(precision, atom_tensor, pair_const, pair_tensor, far_tensor, impl)
        assert out.tolist() == want, (precision, atom_tensor, pair_const, pair_tensor, far_tensor, impl)
