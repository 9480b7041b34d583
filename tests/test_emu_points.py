"""CPU warp emulation of the point kernels of epnn_elst.cu (epnn_potential_points).

The kernel source is compiled for the host with -DEPNN_CPU_EMU (tools/emu/cuda_emu.h).  tools/emu/emu_points.cpp builds
the same chunks and work plan as the library (epnn_elst.cuh) and runs the point and reduction kernels.  The atoms are the
adversarial batch of tests/elst_ref.py plus systems at the part length edges; the points hit the tile edges, sit exactly
on atoms (the coincident pair included) and 1 000 A away, and some systems have none.  The chunk budget and atom bound are
parameters of the emulation, so small calls reach chunk boundaries inside a system."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from points_ref import batch_ref, check, edge_points, kernel_constants, part_edge_batch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "build", "libemu_points.so")
K = kernel_constants()
BIG = 1 << 40                                                            # no atom bound


@pytest.fixture(scope="module")
def emu():
    os.makedirs(os.path.join(ROOT, "build"), exist_ok=True)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-pthread", "-DEPNN_CPU_EMU",
                           "-Wno-unknown-pragmas", "-o", LIB, os.path.join(ROOT, "tools", "emu", "emu_points.cpp")])
    lib = C.CDLL(LIB)
    lib.emu_points_parts.argtypes = [C.c_int]
    lib.emu_points_chunks.argtypes = [C.c_longlong, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_void_p, C.c_int]
    lib.emu_points.argtypes = [C.c_longlong] + [C.c_void_p] * 5 + [C.c_longlong, C.c_longlong, C.c_void_p, C.c_void_p]
    lib.emu_points.restype = C.c_longlong
    return lib


@pytest.fixture(scope="module")
def batch():
    offs, xyz, q = part_edge_batch()
    poff, pts = edge_points(offs, xyz)
    return dict(offs=offs, xyz=xyz, q=q, poff=poff, pts=pts, ref=batch_ref(offs, xyz, q, poff, pts))


def p_(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def run(emu, offs, xyz, q, poff, pts, outputs=("phi", "field"), max_atoms=BIG, budget=K["ELST_PT_CHUNK"]):
    n = int(poff[-1])
    out = {k: np.full(n if k == "phi" else (n, 3), np.nan) for k in outputs}
    emu.emu_points(len(offs) - 1, p_(offs), p_(xyz), p_(q), p_(poff), p_(pts), max_atoms, budget, p_(out.get("phi")),
                   p_(out.get("field")))
    return out


def chunks(emu, offs, poff, max_atoms=BIG, budget=K["ELST_PT_CHUNK"]):
    buf = np.zeros(4 * 4096, np.int64)
    m = emu.emu_points_chunks(len(offs) - 1, p_(offs), p_(poff), max_atoms, budget, p_(buf), 4096)
    return buf[:4 * m].reshape(m, 4)


def test_the_batch_reaches_the_edges(emu, batch):
    offs, poff = batch["offs"], batch["poff"]
    n, m = np.diff(offs), np.diff(poff)
    T, P = K["ELST_PT_TILE"], K["ELST_PT_PART"]
    assert {1, T - 1, T, T + 1, 2 * T + 1} <= set(m.tolist())
    zero = np.nonzero(m == 0)[0]
    assert len(zero) and all(m[:s].sum() > 0 and m[s + 1:].sum() > 0 for s in zero)    # 0 points between systems with points
    with_pts = n[m > 0]
    assert {P - 1, P, P + 1, 2 * P + 1} <= set(with_pts.tolist())
    assert [emu.emu_points_parts(int(k)) for k in (1, P - 1, P, P + 1, 2 * P + 1)] == [1, 1, 1, 2, 3]
    # points exactly on an atom that another atom of the system coincides with
    on_pair = [s for s in range(len(n)) if m[s] and n[s] >= 3 and np.array_equal(batch["pts"][poff[s]], batch["xyz"][offs[s] + n[s] // 2])]
    assert on_pair
    far = [np.linalg.norm(batch["pts"][poff[s]:poff[s + 1]] - batch["xyz"][offs[s]:offs[s + 1]].mean(0), axis=1).max()
           for s in range(len(n)) if m[s] >= 3]
    assert min(far) > 999.0                                              # a point 1 000 A away in every system of 3+ points


@pytest.mark.parametrize("outputs", [("phi",), ("field",), ("phi", "field")])
def test_emulated_kernels_match_the_definition(emu, batch, outputs):
    got = run(emu, batch["offs"], batch["xyz"], batch["q"], batch["poff"], batch["pts"], outputs)
    for k in outputs:
        assert np.isfinite(got[k]).all(), k                             # every output written over the NaN start
    check(got, batch["ref"])


def test_points_on_atoms_skip_the_atom(emu, batch):
    """A point on atom 0 of a system (where atom n // 2 sits too) gets the sum over the other atoms only."""
    offs, xyz, q, poff = batch["offs"], batch["xyz"], batch["q"], batch["poff"]
    got = run(emu, offs, xyz, q, poff, batch["pts"], ("phi",))
    for s in range(len(offs) - 1):
        a0, a1, p0 = int(offs[s]), int(offs[s + 1]), int(poff[s])
        if poff[s + 1] == p0 or a1 - a0 < 3:
            continue
        x = xyz[a0:a1].astype(np.float64)
        r = np.linalg.norm(x - x[0], axis=1)
        keep = r > 0
        assert keep.sum() == a1 - a0 - 2
        want = float(q[a0:a1][keep] @ (1.0 / r[keep]))
        assert abs(got["phi"][p0] - want) <= 1e-11 * float(np.abs(q[a0:a1][keep]) @ (1.0 / r[keep]))


def test_chunks_cut_inside_a_system_and_change_no_bit(emu, batch):
    offs, xyz, q, poff, pts = batch["offs"], batch["xyz"], batch["q"], batch["poff"], batch["pts"]
    whole = run(emu, offs, xyz, q, poff, pts)
    assert len(chunks(emu, offs, poff)) == 1
    budget = 3 * 37                                                      # at least the largest part count (3)
    ch = chunks(emu, offs, poff, max_atoms=2000, budget=budget)
    assert len(ch) > 10
    assert ch[0][2] == 0 and ch[-1][3] == poff[-1] and (ch[1:, 2] == ch[:-1, 3]).all()      # the points, once each
    sys_of_p0 = np.searchsorted(poff, ch[1:, 2], side="right") - 1
    assert (ch[1:, 2] > poff[sys_of_p0]).any()                           # some chunk starts inside a system's points
    assert (ch[:, 1] - ch[:, 0] > 1).any()                               # and some hold several systems
    cut = run(emu, offs, xyz, q, poff, pts, max_atoms=2000, budget=budget)
    for k in whole:
        assert np.array_equal(cut[k], whole[k]), k


def test_a_point_depends_only_on_its_system(emu, batch):
    """Every 7th point alone, a system alone, and the systems in reverse order give the bits of the full call."""
    offs, xyz, q, poff, pts = batch["offs"], batch["xyz"], batch["q"], batch["poff"], batch["pts"]
    whole = run(emu, offs, xyz, q, poff, pts)
    S = len(offs) - 1
    # every 7th point of every system
    sel = np.arange(0, int(poff[-1]), 7)
    sys_of = np.searchsorted(poff, sel, side="right") - 1
    poff7 = np.searchsorted(sys_of, np.arange(S + 1)).astype(np.int64)
    sub = run(emu, offs, xyz, q, poff7, np.ascontiguousarray(pts[sel]))
    for k in whole:
        assert np.array_equal(sub[k], whole[k][sel]), k
    # systems in reverse order
    order = np.arange(S)[::-1]
    n, m = np.diff(offs), np.diff(poff)
    roffs = np.concatenate([[0], np.cumsum(n[order])]).astype(np.int32)
    rpoff = np.concatenate([[0], np.cumsum(m[order])]).astype(np.int64)
    cat = lambda a, o: np.ascontiguousarray(np.concatenate([a[o[s]:o[s + 1]] for s in order]))
    rev = run(emu, roffs, cat(xyz, offs), cat(q, offs), rpoff, cat(pts, poff))
    for k in whole:
        assert np.array_equal(rev[k], cat(whole[k], poff)), k
    # one split system alone
    s = S - 1
    a0, a1, p0, p1 = int(offs[s]), int(offs[s + 1]), int(poff[s]), int(poff[s + 1])
    one = run(emu, np.array([0, a1 - a0], np.int32), xyz[a0:a1], q[a0:a1], np.array([0, p1 - p0], np.int64), pts[p0:p1])
    for k in whole:
        assert np.array_equal(one[k], whole[k][p0:p1]), k


def test_phi_with_and_without_the_field_agree(emu, batch):
    args = (batch["offs"], batch["xyz"], batch["q"], batch["poff"], batch["pts"])
    a, b = run(emu, *args, outputs=("phi",)), run(emu, *args)
    check({"phi": a["phi"]}, batch["ref"])
    assert np.abs(a["phi"] - b["phi"]).max() <= 1e-11 * batch["ref"]["phi_scale"].max()


def test_reference_agrees_with_a_loop():
    """The blocked reference against the definition written as a loop over atoms."""
    from points_ref import system_ref
    rng = np.random.default_rng(2)
    x = rng.uniform(-3, 3, size=(17, 3))
    q = rng.normal(size=17)
    pts = np.concatenate([x[:2], rng.uniform(-5, 5, size=(5, 3))])
    r = system_ref(x, q, pts, block=3)
    for i, p in enumerate(pts):
        phi, E = 0.0, np.zeros(3)
        for j in range(17):
            d = p - x[j]
            rr = np.linalg.norm(d)
            if rr > 0:
                phi += q[j] / rr
                E += q[j] * d / rr ** 3
        assert abs(r["phi"][i] - phi) < 1e-12 and np.abs(r["field"][i] - E).max() < 1e-12
