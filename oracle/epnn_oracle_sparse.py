"""Float64 oracle that scales past the dense one: torch, sparse pair set, one block of rows at a time.

THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE (same rules as ``epnn_oracle``; it never imports ``epnn_b200``).

``forward_factorised`` builds dense (n, n, 48) descriptors, which stops it a little past the 2220-atom protein.  The
mathematics below is the same, line for line, with two changes of data structure only:

  * the pair set comes from a k-d tree (every pair within 3 A + 1e-3), and the oracle's own predicate is applied to it:
    D = sqrt((dx^2 + dy^2) + dz^2) in float64 of the float32 coordinates, C as in ``get_init_edges`` (C = 1 at D = 0),
    e rounded once to float32; the GNN keeps the pairs with any e != 0, the EPN the ``is_near`` pairs;
  * the all-pairs message sum is evaluated per block of rows: z = u[blk, None] + v[None] of shape (R, n, 32), the
    block's sparse c_e added at its (i, j) entries, then relu(relu(z) @ W2 + b2).sum(1) -- every column j of the row
    is evaluated explicitly (no "full sum minus near terms").

On a GPU (``device="cuda"``) a 50 k-atom system takes seconds; on the CPU it is meant for systems of a few thousand atoms.
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np
import torch

from .epnn_oracle import CUTOFF, E_DIM, ETA, NEAR_TOL, features, initial_charge

Z_BLOCK_BYTES = 2 * 1024 ** 3        # one (R, n, 32) float64 tensor of the message sum stays under this


def sparse_edges(xyz):
    """Pairs (i, j), i != j, both orientations, with e_ij != 0, and their float32 descriptors e (P, 48).

    The values are those of ``epnn_oracle.get_init_edges`` bit for bit: the same float64 expressions on the same float32
    coordinates, in numpy."""
    from scipy.spatial import cKDTree
    x = np.asarray(xyz, dtype=np.float32).astype(np.float64)
    n = x.shape[0]
    if n < 2:
        return np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros((0, E_DIM), np.float32)
    pu = cKDTree(x).query_pairs(CUTOFF + 1e-3, output_type="ndarray").astype(np.int64)
    pi = np.concatenate([pu[:, 0], pu[:, 1]])
    pj = np.concatenate([pu[:, 1], pu[:, 0]])
    d = np.abs(x[pj] - x[pi])
    sq = d * d
    D = np.sqrt((sq[:, 0] + sq[:, 1]) + sq[:, 2])
    mu = np.linspace(0.1, CUTOFF, num=E_DIM)
    C = (np.cos(np.pi * (D - 0.0) / CUTOFF) + 1.0) / 2.0
    C[D >= CUTOFF] = 0.0
    C[D <= 0.0] = 1.0
    e = np.array(C[:, None] * np.exp(-ETA * (D[:, None] - mu[None, :]) ** 2), dtype=np.float32)
    keep = (e != 0).any(axis=1)
    order = np.lexsort((pj[keep], pi[keep]))                # row-major, like np.nonzero of the dense mask
    return pi[keep][order], pj[keep][order], e[keep][order]


def is_near(e):
    """The ``is_near`` mask (max_k e_ijk > float32(1e-5), ``epnn_oracle.is_near_from_e``) of ``sparse_edges`` descriptors."""
    return e.max(axis=1) > NEAR_TOL


def _mlp(mlp, x):
    n = len(mlp.W)
    for i, (W, b) in enumerate(zip(mlp.W, mlp.b)):
        x = x @ torch.as_tensor(W, dtype=torch.float64, device=x.device) + torch.as_tensor(b, dtype=torch.float64, device=x.device)
        if i < n - 1:
            x = torch.relu(x)
    return x


def forward_sparse(w, xyz, species, Q, npad=None, device="cpu", trace: Optional[Dict] = None):
    """``epnn_oracle.forward_factorised`` for one system (float64); returns q (numpy, n real atoms).

    ``trace`` (a dict) receives "messages" (M of every message-passing step), "h_steps" and "h" as numpy arrays, like the
    dense oracle's trace."""
    dev = torch.device(device)
    f64 = dict(dtype=torch.float64, device=dev)
    xyz = np.asarray(xyz, dtype=np.float32)
    n = xyz.shape[0]
    N = n if npad is None else int(npad)
    if N < n:
        raise ValueError("npad must be >= number of atoms")
    F = w.F
    T = lambda a: torch.as_tensor(np.asarray(a), **f64)     # noqa: E731
    x = T(features(species, w.n_x))
    h = torch.zeros((n, w.h_dim), **f64)
    q = torch.full((n, 1), float(initial_charge(Q, n)), **f64)
    pi_np, pj_np, e_np = sparse_edges(xyz)
    pi = torch.as_tensor(pi_np, device=dev)
    pj = torch.as_tensor(pj_np, device=dev)
    e_nz = T(e_np)
    row_start = np.searchsorted(pi_np, np.arange(n + 1))   # pairs are sorted by row
    R = max(1, min(n, Z_BLOCK_BYTES // max(1, n * 32 * 8)))
    for t in range(w.T):
        W1, b1 = T(w.msg[t].W[0]), T(w.msg[t].b[0])
        W2, b2 = T(w.msg[t].W[1]), T(w.msg[t].b[1])
        W3, b3 = T(w.msg[t].W[2]), T(w.msg[t].b[2])
        a = torch.cat([x, h, q], dim=1)
        u = a @ W1[:F]
        v = a @ W1[F:2 * F] + b1
        ce = e_nz @ W1[2 * F:]
        S = torch.zeros((n, 32), **f64)
        for r0 in range(0, n, R):
            r1 = min(n, r0 + R)
            z = u[r0:r1, None, :] + v[None, :, :]
            p0, p1 = int(row_start[r0]), int(row_start[r1])
            z.index_put_((pi[p0:p1] - r0, pj[p0:p1]), ce[p0:p1], accumulate=True)
            z.relu_()
            m = torch.matmul(z, W2)
            del z
            m.add_(b2).relu_()
            S[r0:r1] = m.sum(dim=1)
            del m
        S += (N - n) * torch.relu(torch.relu(u + b1) @ W2 + b2)
        M = S @ W3 + N * b3
        h = _mlp(w.upd, torch.cat([h, M], dim=1))
        if trace is not None:
            trace.setdefault("messages", []).append(M.cpu().numpy())
            trace.setdefault("h_steps", []).append(h.cpu().numpy())
    if trace is not None:
        trace["h"] = h.cpu().numpy()
    near = is_near(e_np) & (pi_np < pj_np)
    qi = torch.as_tensor(pi_np[near], device=dev)
    qj = torch.as_tensor(pj_np[near], device=dev)
    ep = T(e_np[near])
    for t in range(w.T):
        W1, b1 = T(w.pas[t].W[0]), T(w.pas[t].b[0])
        W2, b2 = T(w.pas[t].W[1]), T(w.pas[t].b[1])
        W3 = T(w.pas[t].W[2])
        a = torch.cat([x, h, q], dim=1)
        u = a @ W1[:F]
        v = a @ W1[F:2 * F] + b1
        ce = ep @ W1[2 * F:]
        f_ij = torch.relu(torch.relu(u[qi] + v[qj] + ce) @ W2 + b2) @ W3
        f_ji = torch.relu(torch.relu(u[qj] + v[qi] + ce) @ W2 + b2) @ W3
        d = 0.5 * (f_ij - f_ji)[:, 0]
        dq = torch.zeros(n, **f64)
        dq.index_add_(0, qi, d)
        dq.index_add_(0, qj, -d)
        q = q + dq[:, None]
        if trace is not None:
            trace.setdefault("q_steps", []).append(q[:, 0].cpu().numpy())
    return q[:, 0].cpu().numpy()


def predict_batch_sparse(w, offsets, xyz, species, Q, npad=None, device="cpu", traces=None):
    """``forward_sparse`` over a packed batch (the argument layout of ``epnn_infer_batch``; ``npad`` None = no padding).

    ``traces``: optional list that receives one trace dict per system."""
    out = np.zeros(int(offsets[-1]), dtype=np.float64)
    for s in range(len(offsets) - 1):
        a0, a1 = int(offsets[s]), int(offsets[s + 1])
        tr = {} if traces is not None else None
        out[a0:a1] = forward_sparse(w, xyz[a0:a1], species[a0:a1], Q[s], None if npad is None else int(npad[s]), device, tr)
        if traces is not None:
            traces.append(tr)
    return out
