"""Parity of the CUDA path (through the C-ABI) against the oracle and the reference's golden vectors.

Tolerances (BASELINE.json north_star): neighbour lists bit-exact; per-atom charges max|dq| <= 1e-5 e;
sum of charges within 1e-6 e of the net charge.

Measured distance to the float64 oracle on the B200 (tools/measure_noise_floor.py, 400 systems of data/mixed per
checkpoint, pad 41 and pad n; profiles/r02/call15_noise_floor.log):

    checkpoint            FP32 (32)   mixed (48)   FP64 (64)   "precision" 0 (auto) picks
    decay_model_weights   7.8e-7      7.9e-7       2.7e-15     32
    model2_weights        3.9e-6      1.3e-6       2.2e-14     32
    model_weights         1.0e-4      9.0e-5       3.5e-10     64

FP32 meets the reference's 1e-5 for decay_model_weights and model2_weights.  It cannot for model_weights against ANY
float64 implementation (|h| reaches 150: numpy float32 of the same formulas is 1.8e-4 off; SURVEY.md trap 7) -- there the
FP32 tolerance below is the measured floor with a factor 2, and the north_star bound is met by the FP64 kernels, which
"precision" 0 selects by itself from a probe of the caller's own systems (test_auto_precision_meets_the_reference_tolerance).
"""
import numpy as np
import pytest

from oracle import epnn_oracle as O

pytestmark = pytest.mark.gpu

TOL = 1e-5
TOL_FP32 = {"decay_model_weights": 2e-6, "model2_weights": 1e-5, "model_weights": 2e-4}     # measured 7.8e-7 / 5.4e-6 / 1.1e-4 (tensor per-atom kernel; SIMT: 3.9e-6 / 1.0e-4)
TOL_MIXED = {"decay_model_weights": 2e-6, "model2_weights": 4e-6, "model_weights": 2e-4}    # measured 7.9e-7 / 1.3e-6 / 9.0e-5
TOL_FP64 = 1e-9                                                                              # measured <= 3.5e-10


def _oracle_batch(w, offs, xyz, sp, Q, npad):
    return O.predict_batch(w, offs, xyz, sp, Q, np.broadcast_to(npad, (len(Q),)))


# ------------------------------------------------------------------------------------------------ neighbour list
def test_neighbor_list_bit_exact_all_mixed(engines, mixed):
    """is_near CSR of all 4379 systems of data/mixed == oracle mask, entry for entry."""
    eng = engines("decay_model_weights")
    rowptr, col = eng.neighbors(mixed.offsets, mixed.xyz, which=0)
    exp_rp = np.zeros(int(mixed.offsets[-1]) + 1, np.int64)
    exp_col = []
    pos = 0
    for i in range(len(mixed.names)):
        xyz, _, _ = mixed.system(i)
        rp, c = O.neighbor_csr(xyz)
        a0 = int(mixed.offsets[i])
        exp_rp[a0 + 1:a0 + len(rp)] = pos + rp[1:]
        pos += int(rp[-1])
        exp_col.append(c + a0)
    exp_col = np.concatenate(exp_col)
    assert np.array_equal(rowptr, exp_rp.astype(np.int32))
    assert np.array_equal(col, exp_col.astype(np.int32))


def test_neighbor_list_protein_and_e_set(engines, protein):
    eng = engines("decay_model_weights")
    offs = np.array([0, len(protein["Z"])], np.int32)
    rowptr, col = eng.neighbors(offs, protein["xyz"], which=0)
    rp, c = O.neighbor_csr(protein["xyz"])
    assert np.array_equal(rowptr, rp) and np.array_equal(col, c)
    assert rowptr[-1] == 25530                                   # SURVEY 8a: ordered near pairs of Galectin-3C
    rowptr1, col1 = eng.neighbors(offs, protein["xyz"], which=1)
    D = O.distance_matrix(protein["xyz"])
    m = (D < 3.0) & ~np.eye(len(D), dtype=bool)
    assert np.array_equal(col1, np.nonzero(m)[1].astype(np.int32))
    assert np.array_equal(rowptr1[1:], np.cumsum(m.sum(1)).astype(np.int32))


def test_init_edges_matches_reference_descriptor(engines, mixed):
    eng = engines("decay_model_weights")
    for i in (0, 777, 2500, 4378):
        xyz, _, _ = mixed.system(i)
        e = eng.init_edges(xyz)
        ref, _ = O.get_init_edges(xyz)
        assert e.shape == ref.shape
        # float64 evaluation on both sides, rounded to float32 once: equal except (rarely) where the two
        # libm implementations differ in the last float64 bit right at a float32 rounding boundary
        diff = np.abs(e.astype(np.float64) - ref.astype(np.float64))
        assert np.all(diff <= np.spacing(np.abs(ref)).astype(np.float64))
        assert (e != ref).mean() < 1e-5
        assert np.array_equal(O.is_near_from_e(e), O.is_near_from_e(ref))


def test_neighbor_synthetic_shell_pairs(engines):
    """10^6 pairs drawn right around the decision boundary D* ~ 2.99396 of is_near and the 3.0 cutoff (the hardest cases: the
    flag rests on CUDA's float64 exp / cos agreeing with the host libm at float32 rounding boundaries, VERDICT r01 weak 10)."""
    rng = np.random.default_rng(5)
    n_sys = 1_000_000
    D = np.concatenate([rng.uniform(2.9935, 2.9945, n_sys // 4), rng.uniform(2.99390, 2.99402, n_sys // 4),
                        rng.uniform(2.9995, 3.0005, n_sys // 4), rng.uniform(2.99998, 3.00002, n_sys // 4)])
    u = rng.normal(size=(n_sys, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    a = rng.uniform(-5, 5, size=(n_sys, 3))
    xyz = np.empty((n_sys, 2, 3), np.float32)
    xyz[:, 0] = a
    xyz[:, 1] = a + u * D[:, None]
    xyz = xyz.reshape(-1, 3)
    offs = np.arange(0, 2 * n_sys + 1, 2, dtype=np.int32)
    eng = engines("decay_model_weights")
    for which in (0, 1):
        rowptr, col = eng.neighbors(offs, xyz, which=which)
        x64 = xyz.astype(np.float64).reshape(n_sys, 2, 3)
        d = np.abs(x64[:, 1] - x64[:, 0])
        sq = d * d
        Dm = np.sqrt((sq[:, 0] + sq[:, 1]) + sq[:, 2])
        if which == 1:
            exp = Dm < 3.0
        else:
            C = (np.cos(np.pi * Dm / 3.0) + 1.0) / 2.0
            C[Dm >= 3.0] = 0
            e = (C[:, None] * np.exp(-2.0 * (Dm[:, None] - np.linspace(0.1, 3.0, 48)[None]) ** 2)).astype(np.float32)
            exp = e.max(1) > np.float32(1e-5)
        got = (rowptr[1:] - rowptr[:-1]).reshape(n_sys, 2)
        assert np.array_equal(got[:, 0] == 1, exp) and np.array_equal(got[:, 1] == 1, exp)
        assert 0.2 < exp.mean() < 0.8


# ------------------------------------------------------------------------------------------------ charges
def test_golden_871_decay(engines, weights, mixed, val871):
    """All 871 shipped validation predictions (decay_model_weights, pad 41) in one batched call."""
    w = weights["decay_model_weights"]
    idx = [mixed.index[n] for n in val871["names"]]
    offs, xyz, sp, Q = mixed.batch(idx, 9)
    eng = engines("decay_model_weights")
    q, q64 = eng.infer_batch(offs, xyz, sp, Q, 41, want_f64=True)
    worst = 0.0
    for k in range(871):
        a0, a1 = offs[k], offs[k + 1]
        worst = max(worst, np.abs(q[a0:a1] - val871["pred"][k, :a1 - a0]).max())
        assert abs(q64[a0:a1].sum() - float(Q[k])) < 1e-6
    assert worst < TOL, worst
    ref = _oracle_batch(w, offs, xyz, sp, Q, 41)
    assert np.abs(q - ref).max() < TOL
    st = eng.last_stats
    assert st["n_systems"] == 871 and st["n_atoms"] == offs[-1] and st["n_launches"] > 20


@pytest.mark.parametrize("name", ["decay_model_weights", "model2_weights", "model_weights"])
@pytest.mark.parametrize("precision", [32, 48, 64])
def test_charges_vs_oracle(engines, weights, mixed, name, precision):
    """QM9 + SSI + charged systems for every checkpoint, FP32, mixed and all-FP64 kernels, pad 41 and pad n."""
    w = weights[name]
    rng = np.random.default_rng(11)
    idx = sorted(rng.choice(mixed.usable(w.n_x), 160, replace=False).tolist())
    offs, xyz, sp, Q = mixed.batch(idx, w.n_x)
    eng = engines(name, precision)
    for npad in (41, None):
        q, q64 = eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)
        npads = np.full(len(idx), 41) if npad else np.diff(offs)
        ref = O.predict_batch(w, offs, xyz, sp, Q, npads)
        tol = {64: TOL_FP64, 48: TOL_MIXED[name], 32: TOL_FP32[name]}[precision]
        err = np.abs(q64 - ref).max()
        assert err < tol, (name, precision, npad, err)
        sums = np.add.reduceat(q64, offs[:-1])
        assert np.abs(sums - Q.astype(np.float64)).max() < 1e-6


@pytest.mark.parametrize("name", ["decay_model_weights", "model2_weights", "model_weights"])
def test_auto_precision_meets_the_reference_tolerance(weights, mixed, name):
    """"precision" 0: the engine probes a prefix of the first call with the FP32 (tensor per-atom kernel, then SIMT), mixed and FP64 kernels and keeps the cheapest one
    within auto_tol of FP64 -- the shipped checkpoints then all meet max|dq| <= 1e-5 e without the caller knowing which of
    them is ill-conditioned (infer.py:57 loads whatever prefix it is given)."""
    from epnn_b200.engine import Engine
    w = weights[name]
    rng = np.random.default_rng(23)
    idx = sorted(rng.choice(mixed.usable(w.n_x), 300, replace=False).tolist())
    offs, xyz, sp, Q = mixed.batch(idx, w.n_x)
    eng = Engine(w, device=0, precision=0)
    try:
        q, q64 = eng.infer_batch(offs, xyz, sp, Q, 41, want_f64=True)
        st = eng.last_stats
        again = eng.infer_batch(offs, xyz, sp, Q, 41, want_f64=True)[1]
        assert eng.last_stats["precision_used"] == st["precision_used"]          # sticky: no second probe, same kernels
        assert np.array_equal(q64, again)
    finally:
        eng.close()
    ref = O.predict_batch(w, offs, xyz, sp, Q, np.full(len(idx), 41))
    assert np.abs(q64 - ref).max() < TOL, (name, st["precision_used"], np.abs(q64 - ref).max())
    assert st["precision_used"] == {"decay_model_weights": 32, "model2_weights": 32, "model_weights": 64}[name]
    assert st["probe_err32"] >= 0 and (st["precision_used"] == 32 or st["probe_err48"] >= 0)    # candidates are probed cheapest first
    assert st["atom_tensor_used"] in (0, 1) and (st["precision_used"] == 32 or st["atom_tensor_used"] == 0)
    assert np.abs(np.add.reduceat(q64, offs[:-1]) - Q).max() < 1e-6


@pytest.mark.parametrize("name", ["model_weights", "model2_weights"])
def test_hidden_state_vs_oracle(engines, weights, mixed, name):
    """GNN-layer output h (live for these checkpoints; the default checkpoint's h is a dead constant)."""
    w = weights[name]
    idx = [3, 1400, 2900, 4100]
    offs, xyz, sp, Q = mixed.batch(idx, w.n_x)
    for precision, rtol in ((32, 2e-4), (48, 1e-4), (64, 3e-7)):      # hidden() returns float32
        eng = engines(name, precision)
        eng.infer_batch(offs, xyz, sp, Q, 41)
        h = eng.hidden(int(offs[-1]))
        for k, i in enumerate(idx):
            tr = {}
            O.forward_factorised(w, xyz[offs[k]:offs[k + 1]], sp[offs[k]:offs[k + 1]], Q[k], 41, trace=tr)
            ref = tr["h"]
            assert ref.std(axis=0).max() > 1e-3          # the GNN really is live here
            scale = np.abs(ref).max()
            assert np.abs(h[offs[k]:offs[k + 1]] - ref).max() < rtol * scale, (name, precision)


def test_protein_golden_and_conservation(engines, weights, protein):
    """Galectin-3C, 2220 atoms, Q=+2, decay_model_weights, pad n: the LARGE-system kernels."""
    w = weights["decay_model_weights"]
    n = len(protein["Z"])
    offs = np.array([0, n], np.int32)
    sp = O.species_from_Z(protein["Z"], 9)
    Q = np.array([protein["Q"]], np.float32)
    eng = engines("decay_model_weights")
    q, q64 = eng.infer_batch(offs, protein["xyz"], sp, Q, None, want_f64=True)
    assert np.abs(q - protein["preds"]).max() < TOL
    assert abs(q64.sum() - 2.0) < 1e-6              # the reference itself only reaches 1.5e-5 here
    ref = O.forward_factorised(w, protein["xyz"], sp, Q[0], None)
    assert np.abs(q64 - ref).max() < TOL


@pytest.mark.parametrize("name,precision,rtol", [("model_weights", 64, 1e-8), ("model2_weights", 64, 1e-8),
                                                 ("model2_weights", 32, 2e-4), ("model_weights", 32, 2e-2)])
def test_large_system_live_gnn(engines, weights, protein, name, precision, rtol):
    """A 600-atom cut of the protein with checkpoints whose GNN is live: exercises the tiled all-pairs
    GNN kernel, the masked e != 0 members, the j-range split and (npad > n) the weighted pad pair.
    These checkpoints were never trained on such systems and blow up (|q| ~ 300 e), so the comparison is
    relative to max|q|; FP64 kernels must agree to 1e-8, FP32 only to its (ill-conditioned) noise."""
    w = weights[name]
    n = 600
    xyz = protein["xyz"][:n]
    Zs = protein["Z"][:n]
    sp = O.species_from_Z(Zs, w.n_x)
    offs = np.array([0, n], np.int32)
    Q = np.array([1.0], np.float32)
    eng = engines(name, precision)
    for npad in (None, 640):
        q, q64 = eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)
        ref = O.forward_factorised(w, xyz, sp, Q[0], npad)
        err = np.abs(q64 - ref).max() / np.abs(ref).max()
        assert err < rtol, (name, precision, npad, err)


def test_mixed_small_and_large_systems_one_batch(engines, weights, mixed, protein):
    w = weights["model2_weights"]
    offs, xyz, sp, Q = mixed.batch([0, 1, 2], 9)
    n = 150
    pz = O.species_from_Z(protein["Z"][:n], 9)
    offs2 = np.concatenate([offs, [offs[-1] + n, offs[-1] + n + 65, offs[-1] + n + 65 + 64]]).astype(np.int32)
    xyz2 = np.concatenate([xyz, protein["xyz"][:n], protein["xyz"][200:265], protein["xyz"][300:364]])
    sp2 = np.concatenate([sp, pz, O.species_from_Z(protein["Z"][200:265], 9), O.species_from_Z(protein["Z"][300:364], 9)])
    Q2 = np.concatenate([Q, [0.0, -1.0, 2.0]]).astype(np.float32)
    npad = np.array([41, 41, 29, 150, 70, 64], np.int32)
    eng = engines("model2_weights", 64)
    q, q64 = eng.infer_batch(offs2, xyz2, sp2, Q2, npad, want_f64=True)
    ref = O.predict_batch(w, offs2, xyz2, sp2, Q2, npad)
    assert np.abs(q64 - ref).max() < TOL


# ------------------------------------------------------------------------------------------------ properties
def test_permutation_equivariance_and_determinism(engines, weights, mixed):
    w = weights["model_weights"]
    offs, xyz, sp, Q = mixed.batch([42], 10)
    eng = engines("model_weights", 64)
    q1 = eng.infer_batch(offs, xyz, sp, Q, 41, want_f64=True)[1]
    q1b = eng.infer_batch(offs, xyz, sp, Q, 41, want_f64=True)[1]
    assert np.array_equal(q1, q1b)                       # bitwise reproducible (no float atomics)
    perm = np.random.default_rng(0).permutation(len(sp))
    q2 = eng.infer_batch(offs, xyz[perm], sp[perm], Q, 41, want_f64=True)[1]
    assert np.abs(q2 - q1[perm]).max() < 1e-9


def test_chunking_is_invisible(engines, weights, mixed):
    w = weights["decay_model_weights"]
    idx = mixed.usable(9)[0:600:3].tolist()
    offs, xyz, sp, Q = mixed.batch(idx, 9)
    eng = engines("decay_model_weights")
    a = eng.infer_batch(offs, xyz, sp, Q, 41).copy()
    eng.set_option("chunk_atoms", 500)
    try:
        b = eng.infer_batch(offs, xyz, sp, Q, 41).copy()
        assert eng.last_stats["n_chunks"] > 5
        eng.set_option("chunk_streams", 2)               # two chunks in flight on two streams, each with its own workspaces
        c2 = eng.infer_batch(offs, xyz, sp, Q, 41).copy()
        assert eng.last_stats["n_chunks"] > 5
    finally:
        eng.set_option("chunk_atoms", 4 * 1024 * 1024)
        eng.set_option("chunk_streams", 1)
    assert np.array_equal(a, b) and np.array_equal(a, c2)


def test_fused_list_building_equals_the_general_path(weights, mixed):
    """Chunks of small systems build their lists with the warp-per-bundle kernels (epnn_bundle_prep.cu); "fused_prep" 0 sends
    them through the general thread-per-atom kernels: identical neighbour lists (both sets) and bit-identical charges."""
    from epnn_b200.engine import Engine
    w = weights["model2_weights"]
    idx = mixed.usable(w.n_x)[0:1500:2].tolist()
    offs, xyz, sp, Q = mixed.batch(idx, w.n_x)
    out = []
    for fused in (1, 0):
        eng = Engine(w, device=0)
        try:
            eng.set_option("fused_prep", fused)
            q64 = eng.infer_batch(offs, xyz, sp, Q, 41, want_f64=True)[1].copy()
            out.append((q64, eng.neighbors(offs, xyz, which=0), eng.neighbors(offs, xyz, which=1), eng.last_stats["n_launches"]))
        finally:
            eng.close()
    assert np.array_equal(out[0][0], out[1][0])
    for k in (1, 2):
        assert np.array_equal(out[0][k][0], out[1][k][0]) and np.array_equal(out[0][k][1], out[1][k][1])


def test_tensor_per_atom_kernel_against_simt(weights, mixed):
    """FP32 calls run the per-atom GEMMs (update MLP, projections) on the warp-level tensor path (3xTF32, epnn_atom_mma.cu);
    "atom_tensor" 0 is the FP32 SIMT kernel.  Same formulas: the charges differ by FP32 round-off only, and both stay inside
    the checkpoint's FP32 tolerance against the float64 oracle."""
    from epnn_b200.engine import Engine
    w = weights["model2_weights"]
    idx = mixed.usable(w.n_x)[5:1205:3].tolist()
    offs, xyz, sp, Q = mixed.batch(idx, w.n_x)
    ref = O.predict_batch(w, offs, xyz, sp, Q, np.full(len(idx), 41))
    q = {}
    for tensor in (1, 0):
        eng = Engine(w, device=0)
        try:
            eng.set_option("atom_tensor", tensor)
            q[tensor] = eng.infer_batch(offs, xyz, sp, Q, 41, want_f64=True)[1].copy()
            assert eng.last_stats["atom_tensor_used"] == tensor
        finally:
            eng.close()
    assert not np.array_equal(q[0], q[1])                         # two different kernels really ran
    assert np.abs(q[1] - q[0]).max() < TOL_FP32["model2_weights"]
    for tensor in (1, 0):
        assert np.abs(q[tensor] - ref).max() < TOL_FP32["model2_weights"]


def test_caller_stream_and_device_pointers(weights, mixed):
    """epnn_set_stream + epnn_infer_batch_dev: the library runs on the caller's stream, ordered after the kernels that
    produce its inputs there, and leaves its outputs in HBM -- same charges as the host-buffer call."""
    import torch
    from epnn_b200.engine import Engine
    w = weights["decay_model_weights"]
    idx = mixed.usable(w.n_x)[:600:3].tolist()
    offs, xyz, sp, Q = mixed.batch(idx, w.n_x)
    eng = Engine(w, device=0)
    try:
        ref = eng.infer_batch(offs, xyz, sp, Q, 41)
        own = eng.stream
        st = torch.cuda.Stream()
        eng.set_stream(st.cuda_stream)
        assert eng.stream == st.cuda_stream
        with torch.cuda.stream(st):
            d_xyz = (torch.from_numpy(xyz).cuda() * 2.0) * 0.5          # produced on the caller's stream, not synchronised
            d_sp, d_Q = torch.from_numpy(sp).cuda(), torch.from_numpy(Q).cuda()
            d_out = torch.empty(int(offs[-1]), dtype=torch.float32, device="cuda")
            eng.infer_batch_dev(offs, d_xyz.data_ptr(), d_sp.data_ptr(), d_Q.data_ptr(), np.full(len(idx), 41, np.int32), d_out.data_ptr())
        assert np.array_equal(d_out.cpu().numpy(), ref)
        eng.set_stream(0)
        assert eng.stream == own
        assert np.array_equal(eng.infer_batch(offs, xyz, sp, Q, 41), ref)
    finally:
        eng.close()


def test_caller_stream_precision_probe_reads_the_callers_inputs(weights, mixed):
    """"precision" 0 with device pointers on a caller stream: the precision probe reads its prefix of the inputs on that
    stream, after the kernels that write them.  The input buffers hold zeros until a copy that the caller stream runs
    after a ~100 ms sleep, without a host sync: a probe ordered on any other stream would choose from the zeros (and
    the choice is sticky).  Same precision, same probe error and the same charges as a host-buffer call."""
    import torch
    from epnn_b200.engine import Engine
    w = weights["model_weights"]
    idx = mixed.usable(w.n_x)[:600:3].tolist()
    offs, xyz, sp, Q = mixed.batch(idx, w.n_x)
    npad = np.full(len(idx), 41, np.int32)
    n = int(offs[-1])
    host = Engine(w, device=0, precision=0)
    try:
        ref32, ref64 = host.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)
        ref_st = host.last_stats
    finally:
        host.close()
    eng = Engine(w, device=0, precision=0)
    try:
        src = [torch.from_numpy(a).cuda() for a in (xyz, sp, Q)]
        dst = [torch.zeros_like(a) for a in src]
        d_out, d_out64 = torch.empty(n, dtype=torch.float32, device="cuda"), torch.empty(n, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        st = torch.cuda.Stream()
        eng.set_stream(st.cuda_stream)
        with torch.cuda.stream(st):
            torch.cuda._sleep(200_000_000)                             # about 100 ms at B200 clocks
            for d, s in zip(dst, src):
                d.copy_(s)
            eng.infer_batch_dev(offs, dst[0].data_ptr(), dst[1].data_ptr(), dst[2].data_ptr(), npad, d_out.data_ptr(), d_out64.data_ptr())
        got = eng.last_stats
        st.synchronize()
        eng.set_stream(0)
    finally:
        eng.close()
    assert got["precision_used"] == ref_st["precision_used"] == 64
    assert got["probe_err32"] == ref_st["probe_err32"] and got["probe_err48"] == ref_st["probe_err48"]
    assert np.array_equal(d_out.cpu().numpy(), ref32) and np.array_equal(d_out64.cpu().numpy(), ref64)


def test_edge_cases(engines, weights):
    w = weights["decay_model_weights"]
    eng = engines("decay_model_weights", 64)
    # single atom; two coincident atoms (D = 0 -> C = 1, charge_gn.py:151); isolated far atoms; n = 5 (n % 4 != 0)
    cases = [
        (np.zeros((1, 3), np.float32), [3], -1.0),
        (np.array([[0, 0, 0], [0, 0, 0]], np.float32), [0, 3], 0.0),
        (np.array([[0, 0, 0], [10, 0, 0], [0, 10, 0]], np.float32), [1, 0, 0], 1.0),
        (np.array([[0, 0, 0], [1, 0, 0], [0, 1.1, 0], [0, 0, 1.2], [2.5, 2.5, 0]], np.float32), [1, 0, 0, 2, 3], 0.0),
    ]
    for xyz, sp, Qv in cases:
        sp = np.array(sp, np.int32)
        offs = np.array([0, len(sp)], np.int32)
        for npad in (None, 41):
            q64 = eng.infer_batch(offs, xyz, sp, np.array([Qv], np.float32), npad, want_f64=True)[1]
            ref = O.forward_literal(w, xyz, sp, np.float32(Qv), npad)
            assert np.abs(q64 - ref).max() < 1e-9, (len(sp), npad)
    # empty batch
    out = eng.infer_batch(np.array([0], np.int32), np.zeros((0, 3), np.float32), np.zeros(0, np.int32), np.zeros(0, np.float32))
    assert out.shape == (0,)


def test_error_behaviour(engines, mixed):
    from epnn_b200._capi import EpnnError
    eng = engines("decay_model_weights")
    offs, xyz, sp, Q = mixed.batch([0], 9)
    with pytest.raises(EpnnError):
        eng.infer_batch(offs, xyz, sp, Q, 2)                       # npad < n
    bad = sp.copy()
    bad[0] = 8                                                     # 9-wide table has 8 species
    with pytest.raises(EpnnError):
        eng.infer_batch(offs, xyz, bad, Q, 41)
    with pytest.raises(EpnnError):
        eng.infer_batch(np.array([0, 0], np.int32), np.zeros((0, 3), np.float32), np.zeros(0, np.int32), np.zeros(1, np.float32))
    q = eng.infer_batch(offs, xyz, sp, Q, 41)                      # ctx still usable after errors
    assert np.isfinite(q).all()


# ------------------------------------------------------------------------------------------------ big systems (cell list)
def test_cell_list_neighbors_big_system(engines):
    """~30k-atom protein-like system (Galectin-3C tiled): the cell-list build must give the same sorted CSR as an
    exact float64 evaluation of the reference predicate on the candidate pairs found by a KD-tree."""
    from scipy.spatial import cKDTree
    from epnn_b200 import synth
    offs, xyz, sp, Q = synth.protein_like(30000, 9, seed=3)
    eng = engines("decay_model_weights")
    x64 = xyz.astype(np.float64)
    cand = cKDTree(x64).query_pairs(3.05, output_type="ndarray")
    d = np.abs(x64[cand[:, 1]] - x64[cand[:, 0]])
    sq = d * d
    D = np.sqrt((sq[:, 0] + sq[:, 1]) + sq[:, 2])
    C = (np.cos(np.pi * D / 3.0) + 1.0) / 2.0
    C[D >= 3.0] = 0
    C[D <= 0.0] = 1.0
    mu = np.linspace(0.1, 3.0, 48)
    near = np.zeros(len(D), bool)
    for k0 in range(0, len(D), 200000):
        sl = slice(k0, k0 + 200000)
        e = (C[sl, None] * np.exp(-2.0 * (D[sl, None] - mu[None]) ** 2)).astype(np.float32)
        near[sl] = e.max(1) > np.float32(1e-5)
    for which, sel in ((1, D < 3.0), (0, near)):
        ij = cand[sel]
        rows = np.concatenate([ij[:, 0], ij[:, 1]])
        cols = np.concatenate([ij[:, 1], ij[:, 0]])
        order = np.lexsort((cols, rows))
        exp_col = cols[order].astype(np.int32)
        exp_rp = np.zeros(len(xyz) + 1, np.int64)
        np.add.at(exp_rp, rows + 1, 1)
        exp_rp = np.cumsum(exp_rp).astype(np.int32)
        rowptr, col = eng.neighbors(offs, xyz, which=which)
        assert np.array_equal(rowptr, exp_rp) and np.array_equal(col, exp_col), which
    assert exp_rp[-1] / len(xyz) > 8                       # a protein-like density (about 11 near neighbours per atom)


def test_big_system_charges_and_chunk_of_mixed_sizes(engines, weights, protein, mixed):
    """One call holding a cell-list system (2220 atoms), a brute-force large system and small bundles."""
    w = weights["decay_model_weights"]
    eng = engines("decay_model_weights", 64)
    offs, xyz, sp, Q = mixed.batch([5, 6, 7], 9)
    pz = O.species_from_Z(protein["Z"], 9)
    n, m = len(pz), 300
    offs2 = np.concatenate([offs, [offs[-1] + n, offs[-1] + n + m]]).astype(np.int32)
    xyz2 = np.concatenate([xyz, protein["xyz"], protein["xyz"][500:500 + m]]).astype(np.float32)
    sp2 = np.concatenate([sp, pz, pz[500:500 + m]]).astype(np.int32)
    Q2 = np.concatenate([Q, [2.0, -1.0]]).astype(np.float32)
    npad = np.array([41, 41, 41, n, m + 7], np.int32)
    q, q64 = eng.infer_batch(offs2, xyz2, sp2, Q2, npad, want_f64=True)
    ref = O.predict_batch(w, offs2, xyz2, sp2, Q2, npad)
    assert np.abs(q64 - ref).max() < 1e-8
    assert np.abs(q[offs[-1]:offs[-1] + n] - protein["preds"]).max() < TOL


def boundary_batch(protein):
    """Cuts of the protein at sizes around the bundle capacity (48) and the small/large routing threshold."""
    sizes = [1, 1, 1, 47, 1, 48, 49, 50, 24, 24, 24, 25, 23, 1, 48, 2, 46, 3]
    pz = O.species_from_Z(protein["Z"], 9)
    offs = [0]
    xyz, sp, Q, npad = [], [], [], []
    start = 0
    for k, n in enumerate(sizes):
        xyz.append(protein["xyz"][start:start + n])
        sp.append(pz[start:start + n])
        start += n + 5
        offs.append(offs[-1] + n)
        Q.append([0.0, 1.0, -1.0][k % 3])
        npad.append(n if k % 2 else n + (k % 5) * 9)
    offs = np.array(offs, np.int32)
    xyz = np.concatenate(xyz).astype(np.float32)
    sp = np.concatenate(sp).astype(np.int32)
    Q = np.array(Q, np.float32)
    npad = np.array(npad, np.int32)
    return offs, xyz, sp, Q, npad


def test_bundle_boundaries_and_routing(engines, weights, protein):
    """Sizes around the bundle capacity (48) and the small/large routing threshold, many 1-atom systems, systems
    that exactly fill a bundle, pad sizes equal to / far above n -- all in one batch, FP64 kernels vs the oracle."""
    w = weights["model2_weights"]
    eng = engines("model2_weights", 64)
    offs, xyz, sp, Q, npad = boundary_batch(protein)
    q, q64 = eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)
    ref = O.predict_batch(w, offs, xyz, sp, Q, npad)
    assert np.abs(q64 - ref).max() < 1e-8 * max(1.0, np.abs(ref).max())
    assert eng.last_stats["n_row_groups"] > 0
    # the FP32 default path on the same batch: measured 7.6e-7 on a B200 (1 000 W; tools/measure_small_floor.py), bound 3x
    q32 = engines("model2_weights").infer_batch(offs, xyz, sp, Q, npad, want_f64=True)[1]
    assert np.abs(q32 - ref).max() < 2.3e-6 * max(1.0, np.abs(ref).max())


def test_synthetic_qm9_stream_properties(engines, weights):
    """The bench workload (BASELINE config 4) at a size the oracle cannot cover in full: 20 000 QM9-shaped molecules
    in several chunks.  Size-independent properties: charge conservation per molecule, a random sample against the
    oracle, and independence of a molecule's charges from where it sits in the batch (bundles, tiles and chunks differ)."""
    from epnn_b200 import synth
    w = weights["model2_weights"]                      # live GNN: exercises every kernel
    n_mol = 20000
    offs, xyz, sp, Q = synth.qm9_shaped(n_mol, 9, seed=7)
    Q = Q.copy()
    Q[::3] = 1.0
    Q[1::3] = -1.0
    npad = np.full(n_mol, 29, np.int32)
    eng = engines("model2_weights")
    eng.set_option("chunk_atoms", 100000)
    try:
        q, q64 = eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)
        assert eng.last_stats["n_chunks"] >= 3
        sums = np.add.reduceat(q64, offs[:-1])
        assert np.abs(sums - Q.astype(np.float64)).max() < 1e-6
        rng = np.random.default_rng(0)
        pick = rng.choice(n_mol, 40, replace=False)
        for k in pick:
            a0, a1 = offs[k], offs[k + 1]
            ref = O.forward_factorised(w, xyz[a0:a1], sp[a0:a1], Q[k], 29)
            assert np.abs(q64[a0:a1] - ref).max() < 5e-5, k
        # the same molecules in reverse order: other bundles, other tiles, other chunks
        order = np.arange(n_mol)[::-1]
        sizes = np.diff(offs)
        offs_r = np.concatenate([[0], np.cumsum(sizes[order])]).astype(np.int32)
        idx = np.concatenate([np.arange(offs[k], offs[k + 1]) for k in order])
        q_r = eng.infer_batch(offs_r, xyz[idx], sp[idx], Q[order], npad, want_f64=True)[1]
        back = np.empty_like(q_r)
        back[idx] = q_r
        assert np.abs(back - q64).max() < 2e-5
    finally:
        eng.set_option("chunk_atoms", 4 * 1024 * 1024)


@pytest.mark.parametrize("name", ["decay_model_weights", "model2_weights", "model_weights"])
def test_far_dedup_is_exact(engines, weights, mixed, name):
    """Collapsing species-equivalent far columns (dedup_far, default on) reuses bit-identical messages: it must change
    nothing beyond the order of a few additions -- FP64 kernels agree to 1e-12, FP32 to FP32 round-off -- whether the
    hidden state is live (model2 / model_weights: only step 0 collapses) or species-wise constant (decay: every step)."""
    w = weights[name]
    rng = np.random.default_rng(21)
    idx = sorted(rng.choice(mixed.usable(w.n_x), 120, replace=False).tolist())
    offs, xyz, sp, Q = mixed.batch(idx, w.n_x)
    for precision, tol in ((64, 1e-12), (32, 3e-6 if name != "model_weights" else 3e-4)):
        eng = engines(name, precision)
        on = eng.infer_batch(offs, xyz, sp, Q, 41, want_f64=True)[1].copy()
        eng.set_option("dedup_far", 0)
        try:
            off = eng.infer_batch(offs, xyz, sp, Q, 41, want_f64=True)[1].copy()
        finally:
            eng.set_option("dedup_far", 1)
        assert np.abs(on - off).max() < tol * max(1.0, np.abs(off).max()), (name, precision, np.abs(on - off).max())
