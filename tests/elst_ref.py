"""Float64 reference of epnn_electrostatics (include/epnn_b200.h), the error bounds its tests use, and the adversarial
batch they run.

Error is measured against the absolute-value scale of each sum, because E is a cancelling sum:
    |E - E_ref|   <= tol * sum_{i<j included} |q_i q_j| / r_ij
    |phi_i - ref| <= tol * sum_{j included} |q_j| / r_ij
    |mu - ref|    <= tol * sum_i |q_i| |x_i - c|
with tol = 1e-12 for systems of at most 48 atoms and 1e-11 above."""
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def kernel_constants():
    """The ELST_* constants of epnn_b200/csrc/epnn_elst.cuh (tile size, source-split bounds)."""
    src = open(os.path.join(ROOT, "epnn_b200", "csrc", "epnn_elst.cuh")).read()
    return {k: int(v) for k, v in re.findall(r"#define (ELST_\w+) (\d+)", src)}


def tol(n):
    return 1e-12 if n <= 48 else 1e-11


def _finish(x, q, phi, phis):
    c = x.mean(0)
    return dict(energy=0.5 * float(q @ phi), phi=phi, dipole=q @ (x - c),
                e_scale=0.5 * float(np.abs(q) @ phis), phi_scale=phis, mu_scale=float(np.abs(q) @ np.linalg.norm(x - c, axis=1)))


def system_ref(x, q, f=None):
    """One system in float64 numpy (dense n x n)."""
    x = np.asarray(x, np.float64)
    q = np.asarray(q, np.float64)
    d = x[:, None, :] - x[None, :, :]
    r = np.sqrt((d * d).sum(-1))
    inc = r > 0
    if f is not None:
        f = np.asarray(f)
        inc &= f[:, None] != f[None, :]
    rinv = np.where(inc, 1.0 / np.where(inc, r, 1.0), 0.0)
    return _finish(x, q, rinv @ q, rinv @ np.abs(q))


def system_ref_torch(x, q, f=None, block=1024, device="cuda"):
    """One large system in float64 torch, one block of target rows at a time (as oracle/epnn_oracle_sparse.py)."""
    import torch
    X = torch.from_numpy(np.asarray(x, np.float64)).to(device)
    Qv = torch.from_numpy(np.asarray(q, np.float64)).to(device)
    F = None if f is None else torch.from_numpy(np.asarray(f, np.int64)).to(device)
    n = X.shape[0]
    phi = torch.empty(n, dtype=torch.float64, device=device)
    phis = torch.empty_like(phi)
    for b0 in range(0, n, block):
        b1 = min(n, b0 + block)
        r = (X[b0:b1, None, :] - X[None, :, :]).square().sum(-1).sqrt()
        inc = r > 0
        if F is not None:
            inc &= F[b0:b1, None] != F[None, :]
        rinv = torch.where(inc, 1.0 / torch.where(inc, r, torch.ones_like(r)), torch.zeros_like(r))
        phi[b0:b1] = rinv @ Qv
        phis[b0:b1] = rinv @ Qv.abs()
        del r, inc, rinv
    return _finish(np.asarray(x, np.float64), np.asarray(q, np.float64), phi.cpu().numpy(), phis.cpu().numpy())


def batch_ref(offs, xyz, q, frag=None, large=None):
    """Per-system references of a packed batch; systems above `large` atoms (if given) use the torch reference."""
    out = []
    for s in range(len(offs) - 1):
        a0, a1 = int(offs[s]), int(offs[s + 1])
        f = None if frag is None else frag[a0:a1]
        fn = system_ref_torch if large is not None and a1 - a0 > large else system_ref
        out.append(fn(xyz[a0:a1], q[a0:a1], f))
    return out


def check(offs, got, refs, phi=True):
    """Asserts the scaled bounds system by system; returns the largest error over scale seen (for reporting)."""
    worst = 0.0
    for s, r in enumerate(refs):
        a0, a1 = int(offs[s]), int(offs[s + 1])
        t = tol(a1 - a0)
        de = abs(got["energy"][s] - r["energy"])
        assert de <= t * r["e_scale"], (s, a1 - a0, de, r["e_scale"])
        dm = np.abs(got["dipole"][s] - r["dipole"]).max()
        assert dm <= t * r["mu_scale"], (s, a1 - a0, dm, r["mu_scale"])
        worst = max(worst, de / max(r["e_scale"], 1e-300), dm / max(r["mu_scale"], 1e-300))
        if phi:
            dp = np.abs(got["phi"][a0:a1] - r["phi"])
            assert (dp <= t * r["phi_scale"]).all(), (s, a1 - a0, dp.max())
            worst = max(worst, float((dp / np.maximum(r["phi_scale"], 1e-300)).max()))
    return worst


def adversarial_batch(seed=3):
    """(offsets, xyz float32, q float64, labels): systems at the small-kernel edges (1 ... 49 atoms, around the 32 lanes and
    the 48-atom bound) and at the large kernel's tile and source-split edges up to about 1 000 atoms; charges of both signs,
    systems with Q != 0, coincident atoms, and one system 1 000 A from the origin."""
    k = kernel_constants()
    T, P = k["ELST_TILE"], k["ELST_MIN_PART"]
    sizes = [1, 2, 3, 31, 32, 33, 47, 48, 49, T - 1, T, T + 1, 2 * T + 1, P, P + 1, 3 * T, 2 * P + 1, 3 * P + 1, 1000]
    rng = np.random.default_rng(seed)
    offs, xyz, q, labels = [0], [], [], []
    for s, n in enumerate(sizes):
        x = rng.uniform(-1.0, 1.0, size=(n, 3)) * (1.9 * n ** (1 / 3))    # about one atom per 7 A^3, like a molecule
        if n >= 3:
            x[n // 2] = x[0]                                          # coincident atoms: the pair is skipped
        if s == len(sizes) - 2:
            x += 1000.0                                               # far from the origin: the dipole needs the centroid
        c = rng.normal(scale=0.4, size=n)
        c += (s % 3 - 1) * rng.uniform(0.2, 1.0) / n                  # net charge -1 .. +1 on two systems in three
        offs.append(offs[-1] + n)
        xyz.append(x.astype(np.float32))
        q.append(c)
        labels.append(f"n{n}")
    return np.array(offs, np.int32), np.concatenate(xyz), np.concatenate(q), labels


def fragment_variants(offs):
    """Fragment labelings of a batch: a split after the first atom, before the last, every atom its own label (must
    equal NULL), and interleaved A B A B ...  Labels are offset per system: only equality within a system matters."""
    sizes = np.diff(offs)
    sys_of = np.repeat(np.arange(len(sizes)), sizes)
    local = np.arange(int(offs[-1])) - offs[:-1][sys_of]
    return {
        "split1": ((local >= 1) + 5 * sys_of).astype(np.int32),
        "split_last": ((local >= sizes[sys_of] - 1) - 3 * sys_of).astype(np.int32),
        "own": np.arange(int(offs[-1]), dtype=np.int32),
        "interleaved": (local % 2 + 2 * (sys_of % 4)).astype(np.int32),
    }
