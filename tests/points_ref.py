"""Float64 reference of epnn_potential_points (include/epnn_b200.h), its error bounds, and the point sets its tests use.

Errors are bounded against the absolute-value scale of each sum, per point p of a system of n atoms:
    |phi - phi_ref|   <= tol(n) * sum_j |q_j| / r_pj
    |E_c - E_c,ref|   <= tol(n) * sum_j |q_j| / r_pj^2      (each component c)
with tol from tests/elst_ref.py (1e-12 for n <= 48, 1e-11 above).  Atoms at r = 0 are left out of every sum."""
import os
import re

import numpy as np

from elst_ref import adversarial_batch, tol

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def kernel_constants():
    """The ELST_PT_* constants of epnn_b200/csrc/epnn_elst.cuh (point tile, part length, chunk budget)."""
    src = open(os.path.join(ROOT, "epnn_b200", "csrc", "epnn_elst.cuh")).read()
    return {k: int(v) for k, v in re.findall(r"#define (ELST_PT_\w+) (\d+)", src)}


def _block(X, Q, P):
    """phi, field, phi_scale, field_scale of the atoms X (n, 3) with charges Q at the points P (m, 3), numpy float64."""
    d = P[:, None, :] - X[None, :, :]
    r = np.sqrt((d * d).sum(-1))
    inc = r > 0
    rinv = np.where(inc, 1.0 / np.where(inc, r, 1.0), 0.0)
    r3 = rinv ** 3
    return rinv @ Q, np.einsum("pj,pjc->pc", r3 * Q[None, :], d), rinv @ np.abs(Q), (rinv * rinv) @ np.abs(Q)


def system_ref(x, q, pts, block=2048):
    """One system in float64 numpy, a block of points at a time."""
    X, Q, P = (np.asarray(a, np.float64) for a in (x, q, pts))
    P = P.reshape(-1, 3)
    parts = [_block(X, Q, P[b:b + block]) for b in range(0, len(P), block)] or [_block(X, Q, P)]
    phi, field, ps, fs = (np.concatenate([p[k] for p in parts]) for k in range(4))
    return dict(phi=phi, field=field.reshape(-1, 3), phi_scale=ps, field_scale=fs)


def system_ref_torch(x, q, pts, block=4096, device="cuda"):
    """One large system in float64 torch, a block of points at a time."""
    import torch
    X = torch.from_numpy(np.asarray(x, np.float64)).to(device)
    Q = torch.from_numpy(np.asarray(q, np.float64)).to(device)
    P = torch.from_numpy(np.asarray(pts, np.float64).reshape(-1, 3)).to(device)
    out = {k: [] for k in ("phi", "field", "phi_scale", "field_scale")}
    for b0 in range(0, P.shape[0], block):
        d = P[b0:b0 + block, None, :] - X[None, :, :]
        r = d.square().sum(-1).sqrt()
        inc = r > 0
        rinv = torch.where(inc, 1.0 / torch.where(inc, r, torch.ones_like(r)), torch.zeros_like(r))
        out["phi"].append(rinv @ Q)
        out["field"].append(torch.einsum("pj,pjc->pc", rinv ** 3 * Q[None, :], d))
        out["phi_scale"].append(rinv @ Q.abs())
        out["field_scale"].append(rinv.square() @ Q.abs())
        del d, r, inc, rinv
    return {k: torch.cat(v).cpu().numpy() for k, v in out.items()}


def batch_ref(offs, xyz, q, poff, pts, large=None):
    """Concatenated references of a packed call; systems above `large` atoms (if given) use the torch reference."""
    out = {"phi": [], "field": [], "phi_scale": [], "field_scale": [], "n": []}
    for s in range(len(offs) - 1):
        a0, a1, p0, p1 = int(offs[s]), int(offs[s + 1]), int(poff[s]), int(poff[s + 1])
        if p1 == p0:
            continue
        fn = system_ref_torch if large is not None and a1 - a0 > large else system_ref
        r = fn(xyz[a0:a1], q[a0:a1], pts[p0:p1])
        for k in ("phi", "field", "phi_scale", "field_scale"):
            out[k].append(r[k])
        out["n"].append(np.full(p1 - p0, a1 - a0))
    if not out["n"]:
        return {"phi": np.zeros(0), "field": np.zeros((0, 3)), "phi_scale": np.zeros(0), "field_scale": np.zeros(0),
                "n": np.zeros(0, np.int64)}
    return {k: np.concatenate(v) for k, v in out.items()}


def check(got, ref):
    """Asserts the scaled bounds at every point for the outputs present in `got`; returns the largest error over scale."""
    t = np.where(ref["n"] <= 48, tol(48), tol(49))                   # tol(n) is a step at 48 atoms
    worst = 0.0
    if "phi" in got:
        d = np.abs(got["phi"] - ref["phi"])
        bad = ~(d <= t * ref["phi_scale"])                               # NaN fails
        assert not bad.any(), (np.nonzero(bad)[0][:5], d[bad][:5])
        worst = max(worst, float((d / np.maximum(ref["phi_scale"], 1e-300)).max(initial=0.0)))
    if "field" in got:
        d = np.abs(np.asarray(got["field"]).reshape(-1, 3) - ref["field"])
        bad = ~(d <= (t * ref["field_scale"])[:, None])
        assert not bad.any(), (np.nonzero(bad.any(1))[0][:5], d[bad][:5])
        worst = max(worst, float((d / np.maximum(ref["field_scale"], 1e-300)[:, None]).max(initial=0.0)))
    return worst


def points_for(x, m, rng):
    """m points for the atoms x (n, 3): atom 0 (which adversarial systems of n >= 3 atoms share with atom n // 2), the
    last atom, a point 1 000 A from the centroid, then points in the atoms' box grown by 2 A."""
    x = np.asarray(x, np.float64)
    u = rng.normal(size=3)
    special = [x[0], x[-1], x.mean(0) + 1000.0 * u / np.linalg.norm(u)]
    lo, hi = x.min(0) - 2.0, x.max(0) + 2.0
    rest = rng.uniform(lo, hi, size=(max(0, m - 3), 3))
    return np.concatenate([np.array(special[:m]).reshape(-1, 3), rest])


def part_edge_batch(seed=5):
    """adversarial_batch (the electrostatics edges: 1 ... 49 atoms, tile and split edges, coincident atoms, net charge,
    a system 1 000 A from the origin) followed by systems at the point kernel's part length PART: PART - 1, PART, PART + 1
    and 2 PART + 1 atoms, made the same way."""
    offs, xyz, q, _ = adversarial_batch()
    P = kernel_constants()["ELST_PT_PART"]
    rng = np.random.default_rng(seed)
    offs, xyz, q = list(offs), [xyz], [q]
    for n in (P - 1, P, P + 1, 2 * P + 1):
        x = rng.uniform(-1.0, 1.0, size=(n, 3)) * (1.9 * n ** (1 / 3))
        x[n // 2] = x[0]
        xyz.append(x.astype(np.float32))
        q.append(rng.normal(scale=0.4, size=n) + rng.uniform(-1.0, 1.0) / n)
        offs.append(offs[-1] + n)
    return np.array(offs, np.int32), np.concatenate(xyz), np.concatenate(q)


def edge_points(offs, xyz, seed=11):
    """Point offsets (int64) and points for a batch: per system a count from 1, 0, TILE - 1, TILE, TILE + 1, 2 TILE + 1,
    3, 5 in turn (every 0 sits between systems with points), each set from points_for."""
    T = kernel_constants()["ELST_PT_TILE"]
    counts = [1, 0, T - 1, T, T + 1, 2 * T + 1, 3, 5]
    rng = np.random.default_rng(seed)
    poff, pts = [0], []
    for s in range(len(offs) - 1):
        m = counts[s % len(counts)]
        pts.append(points_for(xyz[offs[s]:offs[s + 1]], m, rng))
        poff.append(poff[-1] + m)
    return np.array(poff, np.int64), np.concatenate(pts)
