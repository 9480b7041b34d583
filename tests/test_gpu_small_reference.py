"""Every small-system kernel set against the float64 oracle on adversarial systems (tests/small_cases.py).

Systems of 48 atoms or fewer run on the bundle kernels.  The default FP32 set ("pair_const" 2) is the row-run GNN kernel
(epnn_bundle_run.cu), the pair-per-thread electron-passing kernel (epnn_bundle_const.cu), the tensor per-atom kernel
(epnn_atom_mma.cu) and the fused list building (epnn_bundle_prep.cu).  The batch of small_cases.py puts these kernels at
their edges: maximal and empty near lists, lists of 30 ... 66 slots around the 32-lane cut, rows over several lanes,
full bundles, pad weights that differ inside a bundle, coincident atoms, pairs just inside the cutoff that are not near,
one species only, every species, the highest species index.  Starting from the default, one option at a time is
changed; every configuration runs the same batch with the two checkpoints whose GNN is live (model2_weights, T = 3, and
model_weights, T = 5), and with decay_model_weights (whose GNN output is a constant) for the electron-passing and
per-atom kernels.

Observables: q64 against O.predict_batch, the hidden state h after the GNN layer (keep_hidden, single-chunk runs)
against O.forward_factorised(..., trace)["h"] system by system, charge conservation, bitwise repeatability, and
bitwise equality of the fused and the general list building (charges and both neighbour sets).

Error = max over systems of max|x - ref| / max(1, max|ref|) within the system: on these unphysical geometries the
checkpoints blow up (a 48-atom ball with npad 1 000 reaches |q| = 4e5 with model2_weights, 1e6 with model_weights).
FP64 runs: q64 within 1e-9, h within 1e-6 (hidden() returns float32).  FP32 and mixed runs: 3x the floor measured on a B200 (148 SMs, 1 000 W
power limit), per checkpoint and configuration (FLOOR below, q64 / h):

    configuration     model2_weights      model_weights       decay_model_weights
    default           6.9e-6 / 2.9e-6     9.5e-4 / 7.8e-7     7.3e-6 / 4.4e-7
    pair_const 1      9.3e-6 / 4.9e-6     8.9e-4 / 3.6e-7     7.3e-6 / 2.2e-7
    pair_const 0      6.4e-6 / 2.5e-6     1.0e-3 / 7.2e-7
    pair_tensor 1     7.2e-6 / 2.9e-6     1.7e-3 / 7.8e-7     5.3e-5 / 4.4e-7
    atom_tensor 0     4.8e-6 / 3.9e-6     1.3e-3 / 3.6e-7     7.3e-6 / 2.0e-7
    fused_prep 0      6.9e-6 / 2.9e-6     9.5e-4 / 7.8e-7
    dedup_far 0       6.9e-6 / 2.9e-6     1.7e-3 / 7.8e-7
    precision 48      2.5e-6 / 1.3e-6     9.0e-4 / 2.3e-7
    precision 64      2.1e-14 / 5.4e-8    5.5e-12 / 5.5e-8    2.2e-14 / 1.0e-8
    chunk_atoms 400   6.9e-6 / -          9.5e-4 / -           (4 chunks, chunk_streams 1 and 2 alike)

model_weights in FP32 is already 1e-4 from the oracle on QM9 (test_gpu_parity.py); on this batch every FP32 and mixed
configuration lands near 1e-3.  Re-measure with tools/measure_small_floor.py.

The FP32 bound of test_gpu_parity.py::test_bundle_boundaries_and_routing comes from the same measurement (7.6e-7).
"""
import numpy as np
import pytest

from oracle import epnn_oracle as O
from small_cases import pack_bundles, small_batch

pytestmark = pytest.mark.gpu

CONFIGS = {
    "default": {},
    "pair_const1": {"pair_const": 1},
    "pair_const0": {"pair_const": 0},
    "pair_tensor1": {"pair_tensor": 1},
    "atom_tensor0": {"atom_tensor": 0},
    "fused_prep0": {"fused_prep": 0},
    "dedup_far0": {"dedup_far": 0},
    "precision48": {"precision": 48},
    "precision64": {"precision": 64},
    "chunks": {"chunk_atoms": 400, "chunk_streams": 1},
    "chunks_2streams": {"chunk_atoms": 400, "chunk_streams": 2},
}
LIVE = ("model2_weights", "model_weights")
DECAY_CONFIGS = ("default", "pair_const1", "pair_tensor1", "atom_tensor0", "precision64")
CASES = [(n, c) for n in LIVE for c in CONFIGS] + [("decay_model_weights", c) for c in DECAY_CONFIGS]
RTOL64_Q, RTOL64_H = 1e-9, 1e-6
# measured floors (q64, h) on a B200, rounded up to two digits; the bound is 3x
FLOOR = {
    ("model2_weights", "default"): (6.9e-06, 3e-06),
    ("model2_weights", "pair_const1"): (9.4e-06, 5e-06),
    ("model2_weights", "pair_const0"): (6.5e-06, 2.6e-06),
    ("model2_weights", "pair_tensor1"): (7.2e-06, 3e-06),
    ("model2_weights", "atom_tensor0"): (4.9e-06, 3.9e-06),
    ("model2_weights", "fused_prep0"): (6.9e-06, 3e-06),
    ("model2_weights", "dedup_far0"): (6.9e-06, 3e-06),
    ("model2_weights", "precision48"): (2.5e-06, 1.3e-06),
    ("model2_weights", "chunks"): (6.9e-06, None),
    ("model2_weights", "chunks_2streams"): (6.9e-06, None),
    ("model_weights", "default"): (0.00096, 7.8e-07),
    ("model_weights", "pair_const1"): (0.0009, 3.7e-07),
    ("model_weights", "pair_const0"): (0.001, 7.2e-07),
    ("model_weights", "pair_tensor1"): (0.0017, 7.8e-07),
    ("model_weights", "atom_tensor0"): (0.0014, 3.6e-07),
    ("model_weights", "fused_prep0"): (0.00096, 7.8e-07),
    ("model_weights", "dedup_far0"): (0.0018, 7.8e-07),
    ("model_weights", "precision48"): (0.0009, 2.4e-07),
    ("model_weights", "chunks"): (0.00096, None),
    ("model_weights", "chunks_2streams"): (0.00096, None),
    ("decay_model_weights", "default"): (7.3e-06, 4.5e-07),
    ("decay_model_weights", "pair_const1"): (7.3e-06, 2.2e-07),
    ("decay_model_weights", "pair_tensor1"): (5.3e-05, 4.5e-07),
    ("decay_model_weights", "atom_tensor0"): (7.3e-06, 2.1e-07),
}


def _tol(name, config):
    if CONFIGS[config].get("precision") == 64:
        return RTOL64_Q, RTOL64_H
    q, h = FLOOR[(name, config)]
    return 3 * q, None if h is None else 3 * h


_REF = {}


def reference(weights, name):
    """(batch, q64, [h per system]) of the float64 oracle for the small-case batch of this checkpoint's element table."""
    if name not in _REF:
        w = weights[name]
        offs, xyz, sp, Q, npad, _ = small_batch(w.n_x)
        q = O.predict_batch(w, offs, xyz, sp, Q, npad)
        hs = []
        for k in range(len(Q)):
            tr = {}
            O.forward_factorised(w, xyz[offs[k]:offs[k + 1]], sp[offs[k]:offs[k + 1]], Q[k], int(npad[k]), trace=tr)
            hs.append(tr["h"])
        _REF[name] = ((offs, xyz, sp, Q, npad), q, hs)
    return _REF[name]


def rel_err(x, ref_parts, offs):
    """max over systems of max|x - ref| / max(1, max|ref|)"""
    return max(float(np.abs(x[offs[k]:offs[k + 1]] - r).max() / max(1.0, np.abs(r).max())) for k, r in enumerate(ref_parts))


def run_config(weights, name, config):
    """Runs one configuration twice on the batch; returns (observables, errors)."""
    from epnn_b200.engine import Engine
    (offs, xyz, sp, Q, npad), ref, ref_h = reference(weights, name)
    opts = dict(CONFIGS[config])
    eng = Engine(weights[name], device=0, precision=opts.pop("precision", 32))
    try:
        for k, v in opts.items():
            eng.set_option(k, v)
        chunked = "chunk_atoms" in opts
        if not chunked:
            eng.set_option("keep_hidden", 1)
        q32, q64 = (a.copy() for a in eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True))
        st = eng.last_stats
        h = None if chunked else eng.hidden(int(offs[-1]))
        q32b, q64b = eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)
        nbr = [eng.neighbors(offs, xyz, which=k) for k in (0, 1)]
    finally:
        eng.close()
    ref_q = [ref[offs[k]:offs[k + 1]] for k in range(len(Q))]
    out = dict(q32=q32, q64=q64, h=h, stats=st, nbr=nbr, repeat_equal=bool(np.array_equal(q64, q64b) and np.array_equal(q32, q32b)),
               sum_err=float(np.abs(np.add.reduceat(q64, offs[:-1]) - Q).max()))
    err = dict(q=rel_err(q64, ref_q, offs), h=None if h is None else rel_err(h, ref_h, offs))
    return out, err


_RUNS = {}


def cached_run(weights, name, config):
    if (name, config) not in _RUNS:
        _RUNS[(name, config)] = run_config(weights, name, config)
    return _RUNS[(name, config)]


@pytest.mark.parametrize("name,config", CASES)
def test_small_systems_against_the_oracle(weights, name, config):
    out, err = cached_run(weights, name, config)
    offs = reference(weights, name)[0][0]
    tol_q, tol_h = _tol(name, config)
    assert err["q"] < tol_q, (name, config, err)
    if err["h"] is not None:
        assert err["h"] < tol_h, (name, config, err)
    assert out["sum_err"] < 1e-6, (name, config, out["sum_err"])
    assert out["repeat_equal"], (name, config)
    st = out["stats"]
    if "chunk_atoms" in CONFIGS[config]:
        assert st["n_chunks"] >= 3
    else:
        assert st["n_chunks"] == 1
        assert st["n_row_groups"] == len(pack_bundles(offs)) and st["n_systems"] == len(offs) - 1
    if config == "atom_tensor0":
        assert st["atom_tensor_used"] == 0
    if config == "default":
        assert st["atom_tensor_used"] == 1


@pytest.mark.parametrize("name", LIVE)
def test_fused_list_building_is_bitwise_the_general_path(weights, name):
    """"fused_prep" 0 builds the lists of the same batch with the general thread-per-atom kernels: bitwise equal charges
    and neighbour lists (both sets), here on full bundles, empty and maximal masks and the cutoff shell."""
    a, _ = cached_run(weights, name, "default")
    b, _ = cached_run(weights, name, "fused_prep0")
    assert np.array_equal(a["q64"], b["q64"]) and np.array_equal(a["q32"], b["q32"])
    for k in (0, 1):
        assert np.array_equal(a["nbr"][k][0], b["nbr"][k][0]) and np.array_equal(a["nbr"][k][1], b["nbr"][k][1]), k


def test_neighbour_sets_are_the_oracles(weights):
    """Both neighbour sets of the engine on the small-case batch equal the oracle's: is_near (electron passing) and
    e != 0 (message passing); the pairs at 2.994 A < D < 3 A are in the second only."""
    (offs, xyz, sp, Q, npad), _, _ = reference(weights, "model2_weights")
    a, _ = cached_run(weights, "model2_weights", "default")
    n_only_gnn = 0
    for which in (0, 1):
        rowptr, col = a["nbr"][which]
        for s in range(len(offs) - 1):
            x = xyz[offs[s]:offs[s + 1]]
            n = len(x)
            e, _ = O.get_init_edges(x)
            D = O.distance_matrix(x)
            off_diag = ~np.eye(n, dtype=bool)
            want = ((e.max(-1) > np.float32(1e-5)) if which == 0 else (D < 3.0)) & off_diag
            if which == 1:
                n_only_gnn += int((want & ~(e.max(-1) > np.float32(1e-5))).sum())
            for i in range(n):
                r = offs[s] + i
                assert np.array_equal(col[rowptr[r]:rowptr[r + 1]], offs[s] + np.nonzero(want[i])[0]), (which, s, i)
    assert n_only_gnn >= 6                                             # three pairs, both directions
