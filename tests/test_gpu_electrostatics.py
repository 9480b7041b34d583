"""epnn_electrostatics on the GPU against the float64 reference of tests/elst_ref.py.

Covers the adversarial batch of the emulation test (with the B200's own SM count, so the source splits are the ones a
user gets), real molecules with the engine's FP64 charges, large systems up to 100 000 atoms, the dimer identity
E_full = E_A + E_B + E_AB, bitwise repeatability and independence from the rest of the batch, host / device / chained
calls on a caller stream, argument checks and the CLI's --elst output."""
import ctypes as C
import os

import numpy as np
import pytest

from elst_ref import adversarial_batch, batch_ref, check, fragment_variants, system_ref, system_ref_torch, tol

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def eng(engines):
    return engines("decay_model_weights")


def charges(eng, offs, xyz, sp, Q, npad=None):
    return eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)[1]


def test_adversarial_batch(eng):
    offs, xyz, q, _ = adversarial_batch()
    got = eng.electrostatics(offs, xyz, q, potential=True)
    check(offs, got, batch_ref(offs, xyz, q))
    for kind, frag in fragment_variants(offs).items():
        g = eng.electrostatics(offs, xyz, q, fragment=frag, potential=True)
        check(offs, g, batch_ref(offs, xyz, q, frag))
        assert np.array_equal(g["dipole"], got["dipole"]), kind
        if kind == "own":
            assert np.array_equal(g["energy"], got["energy"]) and np.array_equal(g["phi"], got["phi"])


def test_real_molecules_with_engine_charges(eng, mixed):
    names = mixed.names
    qm9 = [i for i, n in enumerate(names) if n.startswith("dsgdb9nsd")][:400]
    ssi = [i for i, n in enumerate(names) if n.startswith("SSI")][:400]
    idx = [i for i in qm9 + ssi if i in set(mixed.usable(9).tolist())]
    offs, xyz, sp, Q = mixed.batch(idx, 9)
    q = charges(eng, offs, xyz, sp, Q, np.full(len(idx), 41, np.int32))
    got = eng.electrostatics(offs, xyz, q, potential=True)
    check(offs, got, batch_ref(offs, xyz, q))
    assert np.diff(offs).max() > 32                                   # targets on both halves of the warp


@pytest.mark.parametrize("n_atoms", [2220, 16384, 100_000])
def test_large_systems(eng, n_atoms, protein):
    from epnn_b200 import synth
    from oracle.epnn_oracle import species_from_Z
    if n_atoms == 2220:
        xyz = protein["xyz"].astype(np.float32)
        offs, sp, Q = np.array([0, n_atoms], np.int32), species_from_Z(protein["Z"], 9), np.array([protein["Q"]], np.float32)
    else:
        offs, xyz, sp, Q = synth.protein_like(n_atoms, 9, seed=1)
    q = charges(eng, offs, xyz, sp, Q)
    frag = (np.arange(n_atoms) >= n_atoms // 3).astype(np.int32)
    for f in (None, frag):
        got = eng.electrostatics(offs, xyz, q, fragment=f, potential=True)
        check(offs, got, [system_ref_torch(xyz, q, f)])


def test_dimer_identity(eng):
    """E(dimer) = E(A alone) + E(B alone) + E_AB(fragments), for the two SSI dimers and a protein cut in two (large path),
    within the scaled bound."""
    from epnn_b200 import xyzio
    d = os.path.join(GOLDEN, "xyz")
    stems = ["SSI-081ILE-085ARG-1-dimer", "SSI-001ASN-030MET-1-dimer"]
    offs, xyz, _, _ = xyzio.load_packed([os.path.join(d, s + ".xyz") for s in stems], 10)
    splits = xyzio.read_splits(d, stems)
    pr = np.load(os.path.join(GOLDEN, "protein.npz"))
    offs = np.concatenate([offs, [offs[-1] + len(pr["Z"])]]).astype(np.int32)
    xyz = np.concatenate([xyz, pr["xyz"].astype(np.float32)])
    splits = np.concatenate([splits, [900]])
    q = np.random.default_rng(0).normal(scale=0.3, size=int(offs[-1]))
    full = eng.electrostatics(offs, xyz, q)
    ab = eng.electrostatics(offs, xyz, q, fragment=xyzio.fragments_from_splits(offs, splits))
    for s in range(len(splits)):
        a0, a1, k = int(offs[s]), int(offs[s + 1]), int(splits[s])
        parts = [eng.electrostatics(np.array([0, m1 - m0], np.int32), xyz[m0:m1], q[m0:m1])["energy"][0]
                 for m0, m1 in ((a0, a0 + k), (a0 + k, a1))]
        scale = system_ref(xyz[a0:a1], q[a0:a1])["e_scale"]
        assert abs(full["energy"][s] - (parts[0] + parts[1] + ab["energy"][s])) <= tol(a1 - a0) * scale, s


def test_bitwise_repeatable_and_independent_of_the_batch(eng, mixed):
    from epnn_b200 import synth
    offs_l, xyz_l, sp_l, Q_l = synth.protein_like(16384, 9, seed=2)
    idx = mixed.usable(9)[:3000:3].tolist()
    offs_s, xyz_s, sp_s, Q_s = mixed.batch(idx, 9)
    # a large mixed batch: small molecules, the 16 384-atom system, more small molecules
    cut = len(idx) // 2
    offs = np.concatenate([offs_s[:cut + 1], offs_s[cut] + offs_l[1:], offs_s[cut + 1:] + offs_l[-1]]).astype(np.int32)
    xyz = np.concatenate([xyz_s[:offs_s[cut]], xyz_l, xyz_s[offs_s[cut]:]])
    rng = np.random.default_rng(1)
    q = rng.normal(scale=0.3, size=int(offs[-1]))
    a = eng.electrostatics(offs, xyz, q, potential=True)
    b = eng.electrostatics(offs, xyz, q, potential=True)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    for s in (0, cut - 1, cut, cut + 1, len(offs) - 2):
        a0, a1 = int(offs[s]), int(offs[s + 1])
        one = eng.electrostatics(np.array([0, a1 - a0], np.int32), xyz[a0:a1], q[a0:a1], potential=True)
        assert one["energy"][0] == a["energy"][s] and np.array_equal(one["dipole"][0], a["dipole"][s]), s
        assert np.array_equal(one["phi"], a["phi"][a0:a1]), s
    # the device variant gives the host variant's bits
    import torch
    d = [torch.from_numpy(x).cuda() for x in (xyz, q)]
    e, mu, phi = (torch.empty(n, dtype=torch.float64, device="cuda") for n in (len(offs) - 1, 3 * (len(offs) - 1), int(offs[-1])))
    eng.electrostatics_dev(offs, d[0].data_ptr(), d[1].data_ptr(), 0, e.data_ptr(), mu.data_ptr(), phi.data_ptr())
    assert np.array_equal(e.cpu().numpy(), a["energy"]) and np.array_equal(mu.cpu().numpy().reshape(-1, 3), a["dipole"])
    assert np.array_equal(phi.cpu().numpy(), a["phi"])


def test_chained_on_a_caller_stream(eng, mixed):
    """infer_batch_dev -> electrostatics_dev on a caller stream whose inputs are produced after a ~100 ms sleep: both calls
    are ordered after the producer, and the result equals the host path."""
    import torch
    idx = mixed.usable(9)[:600:3].tolist() + [0]
    offs, xyz, sp, Q = mixed.batch(idx, 9)
    npad = np.full(len(idx), 41, np.int32)
    frag = (np.arange(int(offs[-1])) % 3 == 0).astype(np.int32)
    n, S = int(offs[-1]), len(idx)
    q64 = charges(eng, offs, xyz, sp, Q, npad)
    ref = eng.electrostatics(offs, xyz, q64, fragment=frag, potential=True)
    src = [torch.from_numpy(a).cuda() for a in (xyz, sp, Q, frag)]
    dst = [torch.zeros_like(a) for a in src]
    q32_d, q64_d = torch.empty(n, dtype=torch.float32, device="cuda"), torch.empty(n, dtype=torch.float64, device="cuda")
    e, mu, phi = (torch.empty(m, dtype=torch.float64, device="cuda") for m in (S, 3 * S, n))
    torch.cuda.synchronize()
    st = torch.cuda.Stream()
    eng.set_stream(st.cuda_stream)
    try:
        with torch.cuda.stream(st):
            torch.cuda._sleep(200_000_000)                             # about 100 ms at B200 clocks
            for d_, s_ in zip(dst, src):
                d_.copy_(s_)
            eng.infer_batch_dev(offs, dst[0].data_ptr(), dst[1].data_ptr(), dst[2].data_ptr(), npad, q32_d.data_ptr(), q64_d.data_ptr())
            eng.electrostatics_dev(offs, dst[0].data_ptr(), q64_d.data_ptr(), dst[3].data_ptr(), e.data_ptr(), mu.data_ptr(), phi.data_ptr())
        st.synchronize()
    finally:
        eng.set_stream(0)
    assert np.array_equal(q64_d.cpu().numpy(), q64)
    assert np.array_equal(e.cpu().numpy(), ref["energy"]) and np.array_equal(mu.cpu().numpy().reshape(-1, 3), ref["dipole"])
    assert np.array_equal(phi.cpu().numpy(), ref["phi"])


def test_argument_checks(eng):
    from epnn_b200 import _capi
    lib, h = eng.lib, eng._h
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    offs = np.array([0, 2, 5], np.int32)
    xyz = np.zeros((5, 3), np.float32)
    q = np.zeros(5)
    e, mu = np.zeros(2), np.zeros(6)
    INVALID = -1
    for fn in (lib.epnn_electrostatics, lib.epnn_electrostatics_dev):
        assert fn(h, 2, p(offs), None, p(q), None, p(e), None, None) == INVALID
        assert b"NULL input" in lib.epnn_last_error(h)
        assert fn(h, 2, p(offs), p(xyz), None, None, p(e), None, None) == INVALID
        assert fn(h, 2, p(offs), p(xyz), p(q), None, None, None, None) == INVALID
        assert b"every output pointer is NULL" in lib.epnn_last_error(h)
        assert fn(h, 2, None, p(xyz), p(q), None, p(e), None, None) == INVALID
        assert fn(h, -1, p(offs), p(xyz), p(q), None, p(e), None, None) == INVALID
        assert fn(h, 2, p(np.array([0, 2, 2], np.int32)), p(xyz), p(q), None, p(e), None, None) == INVALID
        assert fn(h, 2, p(np.array([1, 2, 5], np.int32)), p(xyz), p(q), None, p(e), None, None) == INVALID
        assert fn(h, 0, p(np.array([0], np.int32)), None, None, None, None, None, None) == _capi.EPNN_OK
        assert fn(None, 2, p(offs), p(xyz), p(q), None, p(e), None, None) == INVALID
    with pytest.raises(ValueError):
        eng.electrostatics(offs, xyz[:4], q)
    with pytest.raises(ValueError):
        eng.electrostatics(offs, xyz, q, fragment=np.zeros(4, np.int32))
    out = eng.electrostatics(offs, xyz, q.astype(np.float32))              # float32 charges are widened
    assert out["energy"].dtype == np.float64 and out["dipole"].shape == (2, 3) and "phi" not in out


def test_cli_elst(tmp_path, monkeypatch):
    from epnn_b200 import infer, xyzio
    from epnn_b200.engine import COULOMB_KCAL, DEBYE_PER_E_ANGSTROM, Engine
    from epnn_b200.checkpoint import load_weights
    d = os.path.join(GOLDEN, "xyz")
    ck = os.path.join(GOLDEN, "checkpoints", "decay_model_weights")
    monkeypatch.chdir(tmp_path)                                        # the CLI writes test_names.npy to the working directory
    out = str(tmp_path / "elst.npz")
    with pytest.raises(SystemExit):
        infer.main(["--path", d, "--weights", ck, "--dense", "--elst", out])
    infer.main(["--path", d, "--weights", ck, "--elst", out])
    r = np.load(out)
    stems, offs, xyz, sp, Q = xyzio.read_directory_packed(d, 9)
    assert r["names"].tolist() == stems
    eng = Engine(load_weights(ck))
    try:
        q64 = eng.infer_batch(offs, xyz, sp, Q, int(np.diff(offs).max()), want_f64=True)[1]
    finally:
        eng.close()
    want = {"SSI-081ILE-085ARG-1-dimer": 6, "SSI-001ASN-030MET-1-dimer": 8}
    assert r["split"].tolist() == [want.get(s, -1) for s in stems]
    for i, s in enumerate(stems):
        a0, a1 = int(offs[i]), int(offs[i + 1])
        full = system_ref(xyz[a0:a1], q64[a0:a1])
        assert abs(r["energy_kcal"][i] - full["energy"] * COULOMB_KCAL) <= 1e-12 * full["e_scale"] * COULOMB_KCAL
        assert np.abs(r["dipole_debye"][i] - full["dipole"] * DEBYE_PER_E_ANGSTROM).max() <= 1e-12 * full["mu_scale"] * DEBYE_PER_E_ANGSTROM
        if s in want:
            k = want[s]
            ref = system_ref(xyz[a0:a1], q64[a0:a1], (np.arange(a1 - a0) >= k).astype(np.int32))
            assert abs(r["inter_kcal"][i] - ref["energy"] * COULOMB_KCAL) <= 1e-12 * ref["e_scale"] * COULOMB_KCAL
            assert abs(r["q_first_fragment"][i] - q64[a0:a0 + k].sum()) < 1e-12
        else:
            assert np.isnan(r["inter_kcal"][i]) and np.isnan(r["q_first_fragment"][i])
