"""The scalable float64 oracle (oracle/epnn_oracle_sparse.py, torch on the CPU here) against the dense one.

The sparse oracle is the reference of the large-system GPU tests (tests/test_gpu_large_reference.py), at sizes the dense
oracle cannot reach; these tests pin it to ``forward_factorised`` wherever both run."""
import numpy as np
import pytest

from oracle import epnn_oracle as O
from oracle import epnn_oracle_sparse as OS

RTOL = 1e-12


def _close(w, xyz, sp, Q, npad, rtol_q=RTOL):
    tr_d, tr_s = {}, {}
    ref = O.forward_factorised(w, xyz, sp, Q, npad, trace=tr_d)
    got = OS.forward_sparse(w, xyz, sp, Q, npad, trace=tr_s)
    assert np.abs(got - ref).max() <= rtol_q * max(np.abs(ref).max(), 1e-300), (xyz.shape[0], npad)
    assert np.abs(tr_s["h"] - tr_d["h"]).max() <= RTOL * max(np.abs(tr_d["h"]).max(), 1e-300)
    assert len(tr_s["messages"]) == len(tr_d["messages"]) == w.T
    for ms, md in zip(tr_s["messages"], tr_d["messages"]):
        assert np.abs(ms - md).max() <= RTOL * max(np.abs(md).max(), 1e-300)


@pytest.mark.parametrize("name", ["decay_model_weights", "model_weights", "model2_weights"])
def test_sparse_equals_factorised_mixed(weights, mixed, name):
    w = weights[name]
    usable = mixed.usable(w.n_x)
    sizes = np.diff(mixed.offsets)[usable]
    # every 400th usable system plus the largest one (the SSI dimers reach the size where most pairs are far)
    pick = sorted(set(usable[::400].tolist()) | {int(usable[np.argmax(sizes)])})
    for i in pick:
        xyz, Z, Q = mixed.system(i)
        sp = O.species_from_Z(Z, w.n_x)
        for npad in (41 if len(Z) <= 41 else None, len(Z)):
            _close(w, xyz, sp, Q, npad)


# model_weights on the protein cut: charges reach |q| ~ 400 e, and its five electron-passing passes amplify a relative
# change of 1e-15 in h (float64 round-off of a different summation order) to 5e-12 in q; h and M still agree to 1e-12
@pytest.mark.parametrize("name,npad,rtol_q", [("model2_weights", None, RTOL), ("model2_weights", 640, RTOL),
                                              ("model_weights", None, 2e-11), ("model_weights", 640, 2e-11)])
def test_sparse_equals_factorised_protein_cut(weights, protein, name, npad, rtol_q):
    w = weights[name]
    n = 600
    _close(w, protein["xyz"][:n], O.species_from_Z(protein["Z"][:n], w.n_x), protein["Q"], npad, rtol_q)


@pytest.mark.parametrize("name", ["model_weights", "model2_weights"])
def test_sparse_coincident_and_single_atom(weights, mixed, name):
    w = weights[name]
    xyz, Z, Q = mixed.system(int(mixed.usable(w.n_x)[0]))
    sp = O.species_from_Z(Z, w.n_x)
    # two coincident atoms: D = 0 gives C = 1 (charge_gn.py:151), a nonzero descriptor on an off-diagonal pair
    xyz2 = np.concatenate([xyz, xyz[:1]]).astype(np.float32)
    sp2 = np.concatenate([sp, sp[:1]])
    pi, pj, e = OS.sparse_edges(xyz2)
    dup = (pi == 0) & (pj == len(Z))
    assert dup.sum() == 1 and e[dup].max() > 0
    _close(w, xyz2, sp2, Q, None)
    _close(w, xyz2, sp2, Q, 41)
    _close(w, xyz[:1], sp[:1], Q, None)
    _close(w, xyz[:1], sp[:1], Q, 7)


def test_sparse_near_set_equals_neighbor_csr(protein):
    xyz = protein["xyz"]
    rowptr, col = O.neighbor_csr(xyz)
    pi, pj, e = OS.sparse_edges(xyz)
    near = OS.is_near(e)
    n = xyz.shape[0]
    rp = np.zeros(n + 1, np.int64)
    rp[1:] = np.cumsum(np.bincount(pi[near], minlength=n))
    assert np.array_equal(rp, rowptr)
    assert np.array_equal(pj[near], col)
    # the e != 0 set is the dense oracle's too
    e_dense, _ = O.get_init_edges(xyz[:700])
    di, dj = np.nonzero((e_dense != 0).any(axis=-1))
    si, sj, se = OS.sparse_edges(xyz[:700])
    assert np.array_equal(si, di) and np.array_equal(sj, dj)
    assert np.array_equal(se, e_dense[di, dj])
