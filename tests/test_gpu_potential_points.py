"""epnn_potential_points on the GPU against the float64 reference of tests/points_ref.py.

Covers the edge batch of the emulation test, real molecules with the engine's charges on grids, Galectin-3C and a
100 000-atom system, the identity with the atom potentials of epnn_electrostatics, the multipole limit far away, the
field as the gradient of phi, bitwise independence of a point from the rest of the call (other points, other systems,
chunks) and from repetition, host / device / chained calls on a caller stream, argument checks and the CLI's --cube."""
import ctypes as C
import os

import numpy as np
import pytest

from elst_ref import adversarial_batch, tol
from points_ref import batch_ref, check, edge_points, kernel_constants, part_edge_batch, system_ref, system_ref_torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
K = kernel_constants()


@pytest.fixture(scope="module")
def eng(engines):
    return engines("decay_model_weights")


def charges(eng, offs, xyz, sp, Q, npad=None):
    return eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)[1]


def grids(offs, xyz, spacing, margin):
    """Point offsets and points of a grid_around each system."""
    from epnn_b200 import cube
    poff, pts = [0], []
    for s in range(len(offs) - 1):
        o, d = cube.grid_around(xyz[offs[s]:offs[s + 1]], spacing, margin)
        ix, iy, iz = np.meshgrid(*(np.arange(k) for k in d), indexing="ij")
        pts.append(np.stack([ix.ravel(), iy.ravel(), iz.ravel()], 1) * spacing + o)
        poff.append(poff[-1] + len(pts[-1]))
    return np.array(poff, np.int64), np.concatenate(pts)


def test_edge_batch(eng):
    offs, xyz, q = part_edge_batch()
    poff, pts = edge_points(offs, xyz)
    ref = batch_ref(offs, xyz, q, poff, pts)
    both = eng.potential_points(offs, xyz, q, poff, pts, field=True)
    check(both, ref)
    phi = eng.potential_points(offs, xyz, q, poff, pts)
    assert set(phi) == {"phi"}
    check(phi, ref)
    # field only, through the C-ABI, over a NaN start
    fld = np.full((len(pts), 3), np.nan)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert eng.lib.epnn_potential_points(eng._h, len(offs) - 1, p(offs), p(xyz), p(q), p(poff), p(pts), None, p(fld)) == 0
    check({"field": fld}, ref)


def test_real_molecules_with_engine_charges(eng, mixed):
    names = mixed.names
    qm9 = [i for i, n in enumerate(names) if n.startswith("dsgdb9nsd")][:40]
    ssi = [i for i, n in enumerate(names) if n.startswith("SSI")][:40]
    idx = [i for i in qm9 + ssi if i in set(mixed.usable(9).tolist())]
    offs, xyz, sp, Q = mixed.batch(idx, 9)
    q = charges(eng, offs, xyz, sp, Q, np.full(len(idx), 41, np.int32))
    poff, pts = grids(offs, xyz, 0.7, 3.0)
    got = eng.potential_points(offs, xyz, q, poff, pts, field=True)
    check(got, batch_ref(offs, xyz, q, poff, pts))


def test_galectin_on_a_coarse_grid(eng, protein):
    from oracle.epnn_oracle import species_from_Z
    xyz = protein["xyz"].astype(np.float32)
    offs = np.array([0, len(xyz)], np.int32)
    q = charges(eng, offs, xyz, species_from_Z(protein["Z"], 9), np.array([protein["Q"]], np.float32))
    poff, pts = grids(offs, xyz, 1.5, 4.0)
    got = eng.potential_points(offs, xyz, q, poff, pts, field=True)
    ref = system_ref_torch(xyz, q, pts)
    ref["n"] = np.full(len(pts), len(xyz))
    check(got, ref)


def test_100k_atoms(eng):
    from epnn_b200 import synth
    offs, xyz, sp, Q = synth.protein_like(100_000, 9, seed=1)
    q = charges(eng, offs, xyz, sp, Q)
    rng = np.random.default_rng(3)
    lo, hi = xyz.min(0) - 3.0, xyz.max(0) + 3.0
    pts = np.concatenate([xyz[:500].astype(np.float64), rng.uniform(lo, hi, size=(3000, 3))])
    poff = np.array([0, len(pts)], np.int64)
    got = eng.potential_points(offs, xyz, q, poff, pts, field=True)
    ref = system_ref_torch(xyz, q, pts)
    ref["n"] = np.full(len(pts), len(xyz))
    check(got, ref)


def test_identity_with_the_atom_potentials(eng):
    offs, xyz, q, _ = adversarial_batch()
    poff = offs.astype(np.int64)
    got = eng.potential_points(offs, xyz, q, poff, xyz.astype(np.float64), field=True)
    phi = eng.electrostatics(offs, xyz, q, potential=True)["phi"]
    ref = batch_ref(offs, xyz, q, poff, xyz.astype(np.float64))
    check(got, ref)
    t = np.where(ref["n"] <= 48, tol(48), tol(49))
    assert (np.abs(got["phi"] - phi) <= t * ref["phi_scale"]).all()


def test_multipole_limit(eng, mixed):
    idx = mixed.usable(9)[:200:7].tolist()
    offs, xyz, sp, Q = mixed.batch(idx, 9)
    q = np.random.default_rng(5).normal(scale=0.3, size=int(offs[-1]))
    mu = eng.electrostatics(offs, xyz, q)["dipole"]
    R = 1000.0
    rng = np.random.default_rng(6)
    poff, pts, want, bound = [0], [], [], []
    for s in range(len(idx)):
        a0, a1 = int(offs[s]), int(offs[s + 1])
        x = xyz[a0:a1].astype(np.float64)
        c = x.mean(0)
        u = rng.normal(size=(16, 3))
        u /= np.linalg.norm(u, axis=1, keepdims=True)
        pts.append(c + R * u)
        poff.append(poff[-1] + 16)
        d = np.linalg.norm(x - c, axis=1)
        want.append(q[a0:a1].sum() / R + (u @ mu[s]) / R ** 2)
        bound.append(np.full(16, np.abs(q[a0:a1]) @ d ** 2 / (R ** 2 * (R - d.max())) + tol(a1 - a0) * np.abs(q[a0:a1]).sum() / (R - d.max())))
    got = eng.potential_points(offs, xyz, q, np.array(poff, np.int64), np.concatenate(pts))["phi"]
    assert (np.abs(got - np.concatenate(want)) <= np.concatenate(bound)).all()


def test_field_is_the_gradient_of_phi(eng, mixed):
    idx = mixed.usable(9)[:300:10].tolist()
    offs, xyz, sp, Q = mixed.batch(idx, 9)
    q = charges(eng, offs, xyz, sp, Q, np.full(len(idx), 41, np.int32))
    rng = np.random.default_rng(8)
    h = 1e-3
    poff, pts = [0], []
    for s in range(len(idx)):
        x = xyz[offs[s]:offs[s + 1]].astype(np.float64)
        cand = rng.uniform(x.min(0) - 3.0, x.max(0) + 3.0, size=(200, 3))
        d = np.linalg.norm(cand[:, None] - x[None], axis=2).min(1)
        cand = cand[d >= 1.0][:20]
        pts.append(cand)
        poff.append(poff[-1] + len(cand))
    pts = np.concatenate(pts)
    poff = np.array(poff, np.int64)
    got = eng.potential_points(offs, xyz, q, poff, pts, field=True)
    ref = batch_ref(offs, xyz, q, poff, pts)
    sys_of = np.searchsorted(poff, np.arange(len(pts)), side="right") - 1
    for c in range(3):
        e = np.zeros(3)
        e[c] = h
        plus = eng.potential_points(offs, xyz, q, poff, pts + e)["phi"]
        minus = eng.potential_points(offs, xyz, q, poff, pts - e)["phi"]
        fd = -(plus - minus) / (2 * h)
        for i in range(len(pts)):
            s = sys_of[i]
            x = xyz[offs[s]:offs[s + 1]].astype(np.float64)
            r = np.linalg.norm(pts[i] - x, axis=1) - h
            trunc = h * h * float(np.abs(q[offs[s]:offs[s + 1]]) @ (1.0 / r ** 4))   # h^2/6 * max|phi'''|, |d^3(1/r)| <= 6/r^4
            rnd = tol(len(x)) * 2 * ref["phi_scale"][i] / h
            assert abs(got["field"][i, c] - fd[i]) <= trunc + rnd, (i, c)


def test_a_point_depends_only_on_its_system(eng, mixed, protein):
    idx = mixed.usable(9)[:60:3].tolist()
    offs_s, xyz_s, _, _ = mixed.batch(idx, 9)
    xp = protein["xyz"].astype(np.float32)
    offs = np.concatenate([offs_s[:-1], [offs_s[-1], offs_s[-1] + len(xp)]]).astype(np.int32)
    xyz = np.concatenate([xyz_s, xp])
    q = np.random.default_rng(1).normal(scale=0.3, size=int(offs[-1]))
    poff, pts = grids(offs, xyz, 1.0, 3.0)
    S = len(offs) - 1
    full = eng.potential_points(offs, xyz, q, poff, pts, field=True)
    again = eng.potential_points(offs, xyz, q, poff, pts, field=True)
    for k in full:
        assert np.array_equal(full[k], again[k]), k
    # every 7th point alone
    sel = np.arange(0, len(pts), 7)
    sys_of = np.searchsorted(poff, sel, side="right") - 1
    poff7 = np.searchsorted(sys_of, np.arange(S + 1)).astype(np.int64)
    sub = eng.potential_points(offs, xyz, q, poff7, pts[sel], field=True)
    for k in full:
        assert np.array_equal(sub[k], full[k][sel]), k
    # systems reordered, and the protein alone
    order = np.random.default_rng(2).permutation(S)
    n, m = np.diff(offs), np.diff(poff)
    cat = lambda a, o: np.concatenate([a[o[s]:o[s + 1]] for s in order])
    rev = eng.potential_points(np.concatenate([[0], np.cumsum(n[order])]).astype(np.int32), cat(xyz, offs), cat(q, offs),
                               np.concatenate([[0], np.cumsum(m[order])]).astype(np.int64), cat(pts, poff), field=True)
    for k in full:
        assert np.array_equal(rev[k], cat(full[k], poff)), k
    a0, p0 = int(offs[-2]), int(poff[-2])
    one = eng.potential_points(np.array([0, len(xp)], np.int32), xp, q[a0:], np.array([0, len(pts) - p0], np.int64), pts[p0:], field=True)
    for k in full:
        assert np.array_equal(one[k], full[k][p0:]), k


def test_chunk_boundaries_change_no_bit(eng):
    """A call whose points span several chunks (ELST_PT_CHUNK cost units; a point of a split system costs its part
    count) equals the same points in pieces cut elsewhere."""
    from epnn_b200 import synth
    offs, xyz, _, _ = synth.protein_like(100_000, 9, seed=1)
    q = np.random.default_rng(4).normal(scale=0.3, size=100_000)
    parts = -(-100_000 // K["ELST_PT_PART"])
    n_pts = 2 * K["ELST_PT_CHUNK"] // parts + 1000                      # three chunks
    rng = np.random.default_rng(9)
    pts = rng.uniform(xyz.min(0), xyz.max(0), size=(n_pts, 3))
    full = eng.potential_points(offs, xyz, q, np.array([0, n_pts], np.int64), pts)
    cuts = [0, 777, n_pts // 2 + 3, n_pts]
    for a, b in zip(cuts[:-1], cuts[1:]):
        piece = eng.potential_points(offs, xyz, q, np.array([0, b - a], np.int64), pts[a:b])
        assert np.array_equal(piece["phi"], full["phi"][a:b]), (a, b)
    ref = system_ref_torch(xyz, q, pts[::997])
    ref["n"] = np.full(len(ref["phi"]), 100_000)
    check({"phi": full["phi"][::997]}, ref)


def test_host_device_and_chained_on_a_caller_stream(eng, mixed):
    import torch
    idx = mixed.usable(9)[:300:3].tolist()
    offs, xyz, sp, Q = mixed.batch(idx, 9)
    npad = np.full(len(idx), 41, np.int32)
    n = int(offs[-1])
    q64 = charges(eng, offs, xyz, sp, Q, npad)
    poff, pts = grids(offs, xyz, 0.8, 2.0)
    P = len(pts)
    ref = eng.potential_points(offs, xyz, q64, poff, pts, field=True)
    # device pointers on the ctx stream
    d_xyz, d_q, d_pts = (torch.from_numpy(a).cuda() for a in (xyz, q64, pts))
    phi, fld = torch.empty(P, dtype=torch.float64, device="cuda"), torch.empty(3 * P, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    eng.potential_points_dev(offs, d_xyz.data_ptr(), d_q.data_ptr(), poff, d_pts.data_ptr(), phi.data_ptr(), fld.data_ptr())
    assert np.array_equal(phi.cpu().numpy(), ref["phi"]) and np.array_equal(fld.cpu().numpy().reshape(-1, 3), ref["field"])
    # chained after infer_batch_dev on a caller stream whose inputs come after a ~100 ms sleep
    src = [torch.from_numpy(a).cuda() for a in (xyz, sp, Q, pts)]
    dst = [torch.zeros_like(a) for a in src]
    q32_d, q64_d = torch.empty(n, dtype=torch.float32, device="cuda"), torch.empty(n, dtype=torch.float64, device="cuda")
    phi2, fld2 = torch.full((P,), float("nan"), dtype=torch.float64, device="cuda"), torch.full((3 * P,), float("nan"), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    st = torch.cuda.Stream()
    eng.set_stream(st.cuda_stream)
    try:
        with torch.cuda.stream(st):
            torch.cuda._sleep(200_000_000)
            for d_, s_ in zip(dst, src):
                d_.copy_(s_)
            eng.infer_batch_dev(offs, dst[0].data_ptr(), dst[1].data_ptr(), dst[2].data_ptr(), npad, q32_d.data_ptr(), q64_d.data_ptr())
            eng.potential_points_dev(offs, dst[0].data_ptr(), q64_d.data_ptr(), poff, dst[3].data_ptr(), phi2.data_ptr(), fld2.data_ptr())
        st.synchronize()
    finally:
        eng.set_stream(0)
    assert np.array_equal(q64_d.cpu().numpy(), q64)
    assert np.array_equal(phi2.cpu().numpy(), ref["phi"]) and np.array_equal(fld2.cpu().numpy().reshape(-1, 3), ref["field"])


def test_argument_checks(eng):
    from epnn_b200 import _capi
    lib, h = eng.lib, eng._h
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    offs = np.array([0, 2, 5], np.int32)
    xyz = np.zeros((5, 3), np.float32)
    xyz[:, 0] = np.arange(5)
    q = np.ones(5)
    poff = np.array([0, 1, 3], np.int64)
    pts = np.full((3, 3), 7.0)
    phi, fld = np.full(3, np.nan), np.full(9, np.nan)
    INVALID = -1
    for fn in (lib.epnn_potential_points, lib.epnn_potential_points_dev):
        assert fn(h, 2, p(offs), None, p(q), p(poff), p(pts), p(phi), None) == INVALID
        assert b"NULL input" in lib.epnn_last_error(h)
        assert fn(h, 2, p(offs), p(xyz), None, p(poff), p(pts), p(phi), None) == INVALID
        assert fn(h, 2, p(offs), p(xyz), p(q), p(poff), p(pts), None, None) == INVALID
        assert b"every output pointer is NULL" in lib.epnn_last_error(h)
        assert fn(h, 2, p(offs), p(xyz), p(q), None, p(pts), p(phi), None) == INVALID
        assert fn(h, 2, p(offs), p(xyz), p(q), p(np.array([1, 1, 3], np.int64)), p(pts), p(phi), None) == INVALID
        assert fn(h, 2, p(offs), p(xyz), p(q), p(np.array([0, 2, 1], np.int64)), p(pts), p(phi), None) == INVALID
        assert b"point_offsets decrease" in lib.epnn_last_error(h)
        assert fn(h, 2, p(offs), p(xyz), p(q), p(poff), None, p(phi), None) == INVALID
        assert b"points is NULL" in lib.epnn_last_error(h)
        assert fn(h, 2, None, p(xyz), p(q), p(poff), p(pts), p(phi), None) == INVALID
        assert fn(h, -1, p(offs), p(xyz), p(q), p(poff), p(pts), p(phi), None) == INVALID
        assert fn(h, 2, p(np.array([0, 2, 2], np.int32)), p(xyz), p(q), p(poff), p(pts), p(phi), None) == INVALID
        assert fn(h, 2, p(np.array([1, 2, 5], np.int32)), p(xyz), p(q), p(poff), p(pts), p(phi), None) == INVALID
        assert fn(None, 2, p(offs), p(xyz), p(q), p(poff), p(pts), p(phi), None) == INVALID
        assert fn(h, 0, p(np.array([0], np.int32)), None, None, p(np.array([0], np.int64)), None, None, None) == _capi.EPNN_OK
    assert np.isnan(phi).all() and np.isnan(fld).all()                 # nothing ran
    # no points at all: points may be NULL
    assert lib.epnn_potential_points(h, 2, p(offs), p(xyz), p(q), p(np.zeros(3, np.int64)), None, p(phi), None) == _capi.EPNN_OK
    with pytest.raises(ValueError):
        eng.potential_points(offs, xyz, q, poff, pts[:2])
    with pytest.raises(ValueError):
        eng.potential_points(offs, xyz, q, poff[:2], pts)
    out = eng.potential_points(offs, xyz, q.astype(np.float32), poff, pts, field=True)   # float32 charges are widened
    assert out["phi"].dtype == np.float64 and out["field"].shape == (3, 3)
    r = system_ref(xyz[2:], q[2:], pts[1:])
    assert np.allclose(out["phi"][1:], r["phi"], rtol=1e-13, atol=0)


def test_cli_cube(tmp_path, monkeypatch):
    from epnn_b200 import cube, elements, infer, xyzio
    from epnn_b200.checkpoint import load_weights
    from epnn_b200.engine import BOHR_ANGSTROM, Engine
    from test_cube import parse_cube
    d = os.path.join(GOLDEN, "xyz")
    ck = os.path.join(GOLDEN, "checkpoints", "decay_model_weights")
    monkeypatch.chdir(tmp_path)
    out = tmp_path / "cubes"
    with pytest.raises(SystemExit):
        infer.main(["--path", d, "--weights", ck, "--dense", "--cube", str(out)])
    infer.main(["--path", d, "--weights", ck, "--cube", str(out), "--cube-spacing", "0.6", "--cube-margin", "3"])
    stems, offs, xyz, sp, Q = xyzio.read_directory_packed(d, 9)
    assert sorted(os.listdir(out)) == sorted(s + ".cube" for s in stems)
    eng = Engine(load_weights(ck))
    try:
        q64 = eng.infer_batch(offs, xyz, sp, Q, int(np.diff(offs).max()), want_f64=True)[1]
        Z = elements.z_table(9)[sp]
        for i, s in enumerate(stems):
            a0, a1 = int(offs[i]), int(offs[i + 1])
            c = parse_cube(out / (s + ".cube"))
            o, dims = cube.grid_around(xyz[a0:a1], 0.6, 3.0)
            assert c["dims"] == dims.tolist() and [int(a[0]) for a in c["atoms"]] == Z[a0:a1].astype(int).tolist()
            ix, iy, iz = np.meshgrid(*(np.arange(k) for k in dims), indexing="ij")
            pts = np.stack([ix.ravel(), iy.ravel(), iz.ravel()], 1) * 0.6 + o
            want = eng.potential_points(np.array([0, a1 - a0], np.int32), xyz[a0:a1], q64[a0:a1],
                                        np.array([0, len(pts)], np.int64), pts)["phi"] * BOHR_ANGSTROM
            got = np.array([float(v) for line in c["body"] for v in line.split()])
            assert np.array_equal(got, np.array([float("%13.5E" % v) for v in want])), s
    finally:
        eng.close()
