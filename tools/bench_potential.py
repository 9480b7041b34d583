"""Potential (and field) of charges at arbitrary points on one GPU: epnn_potential_points_dev.

Workloads (synth.protein_like(100 000) is bench.py's large-system shape; Galectin-3C is the protein it tiles):
  split      64 random points in the box of the 100 000-atom system: few points, many atoms (the source-split path)
  grid_phi   a 100^3 grid (10^6 points) over the 100 000-atom system, phi only
  grid_field the same grid, phi and field
  galectin   a 0.3 A grid, 4 A margin, around Galectin-3C (2 220 atoms), phi only
  qm9        synth.qm9_shaped(10 000) molecules, each with its own 0.3 A / 4 A grid (the --cube defaults), phi only
  atoms_phi  epnn_electrostatics_dev, phi only, of the 100 000-atom system: the atom pair kernel on the same card
Charges are seeded normal(0, 0.3) per atom (the kernels' cost does not depend on their values).  Every call is timed with
CUDA events on the engine's stream after warm-up, in two windows, and a sample of points is checked against float64
numpy.  Pairs are point-atom pairs (ordered atom pairs for atoms_phi); bytes are the points read and the outputs written.
Prints one JSON line (and writes it to --out).

    python tools/bench_potential.py --out profiles/r04/potential_b200.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    """Card name and power limit, read-only."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, limit = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit": limit}
    except Exception as e:      # noqa: BLE001
        return {"name": None, "power_limit": None, "error": str(e)}


def timed(torch, stream, fn, warmup, calls):
    """Milliseconds per call: CUDA events on the engine's stream around `calls` calls, after `warmup` calls."""
    for _ in range(warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(calls):
        fn()
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1) / calls


def grid_points(torch, origins, dims, spacing):
    """Device points of one grid per system (x slowest, z fastest) and their int64 host offsets."""
    cnt = dims.prod(1)
    poff = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    P = int(poff[-1])
    idx = torch.arange(P, device="cuda")
    m = torch.searchsorted(dev(poff[1:]), idx, right=True)
    loc = idx - dev(poff)[m]
    nz, nyz = dev(dims[:, 2])[m], dev(dims[:, 1] * dims[:, 2])[m]
    ix = loc // nyz
    r = loc - ix * nyz
    iy = r // nz
    ijk = torch.stack([ix, iy, r - iy * nz], 1).double()
    del idx, loc, nz, nyz, ix, r, iy
    return (dev(origins)[m] + spacing * ijk).contiguous(), poff


def check_sample(xyz, q, offs, poff, pts_dev, phi_dev, fld_dev, rng, k=256):
    """Largest |error| / scale over k sampled points (phi and, if given, field)."""
    sel = np.sort(rng.choice(int(poff[-1]), size=min(k, int(poff[-1])), replace=False))
    P = pts_dev[sel].cpu().numpy()
    phi = phi_dev[sel].cpu().numpy()
    fld = None if fld_dev is None else fld_dev.view(-1, 3)[sel].cpu().numpy()
    sys_of = np.searchsorted(poff, sel, side="right") - 1
    worst = {"phi": 0.0, "field": 0.0 if fld is not None else None}
    for i, s in enumerate(sys_of):
        x = xyz[offs[s]:offs[s + 1]].astype(np.float64)
        c = q[offs[s]:offs[s + 1]]
        d = P[i] - x
        r = np.sqrt((d * d).sum(1))
        rinv = np.where(r > 0, 1.0 / np.where(r > 0, r, 1.0), 0.0)
        worst["phi"] = max(worst["phi"], abs(phi[i] - c @ rinv) / max(np.abs(c) @ rinv, 1e-300))
        if fld is not None:
            E = (c * rinv ** 3) @ d
            worst["field"] = max(worst["field"], float(np.abs(fld[i] - E).max() / max(np.abs(c) @ rinv ** 2, 1e-300)))
    return worst


def run(args):
    import torch
    from epnn_b200 import cube, synth
    from epnn_b200.checkpoint import load_weights
    from epnn_b200.engine import Engine
    w = load_weights(os.path.join(ROOT, "tests", "golden", "checkpoints", "decay_model_weights"))
    eng = Engine(w, device=0)
    stream = torch.cuda.ExternalStream(eng.stream)
    rng = np.random.default_rng(7)
    result = {"gpu": gpu_info(), "workloads": []}
    big = synth.protein_like(args.atoms, w.n_x, seed=1)
    for name in args.workloads:
        field = name == "grid_field"
        if name in ("split", "grid_phi", "grid_field", "atoms_phi"):
            offs, xyz = big[0], big[1]
            if name == "split":
                lo, hi = xyz.min(0), xyz.max(0)
                pts = torch.from_numpy(rng.uniform(lo, hi, size=(64, 3))).cuda()
                poff = np.array([0, 64], np.int64)
                desc = f"64 random points, synth.protein_like({args.atoms})"
            elif name != "atoms_phi":
                lo, hi = xyz.min(0).astype(np.float64), xyz.max(0).astype(np.float64)
                sp = float((hi - lo).max()) / 99
                pts, poff = grid_points(torch, lo[None], np.array([[100, 100, 100]]), sp)
                desc = f"100^3 grid ({sp:.3f} A) over synth.protein_like({args.atoms})" + (", phi + field" if field else ", phi")
            else:
                desc = f"electrostatics_dev, phi only, synth.protein_like({args.atoms})"
        elif name == "galectin":
            xyz, _, _ = synth.protein()
            offs = np.array([0, len(xyz)], np.int32)
            o, d = cube.grid_around(xyz, 0.3, 4.0)
            pts, poff = grid_points(torch, o[None], d[None], 0.3)
            desc = f"Galectin-3C ({len(xyz)} atoms), 0.3 A grid, 4 A margin: {'x'.join(map(str, d.tolist()))}"
        else:
            offs, xyz, _, _ = synth.qm9_shaped(args.molecules, w.n_x, seed=0)
            S = len(offs) - 1
            lo = np.minimum.reduceat(xyz.astype(np.float64), offs[:-1], axis=0) - 4.0
            hi = np.maximum.reduceat(xyz.astype(np.float64), offs[:-1], axis=0) + 4.0
            dims = np.ceil((hi - lo) / 0.3 - 1e-9).astype(np.int64) + 1                 # cube.grid_around, vectorised
            assert S and np.array_equal(cube.grid_around(xyz[offs[0]:offs[1]], 0.3, 4.0)[1], dims[0])
            pts, poff = grid_points(torch, lo, dims, 0.3)
            desc = f"synth.qm9_shaped({args.molecules}), one 0.3 A / 4 A grid each"
        n_sys, n = len(offs) - 1, int(offs[-1])
        q = np.random.default_rng(3).normal(scale=0.3, size=n)
        d_xyz, d_q = torch.from_numpy(xyz).cuda(), torch.from_numpy(q).cuda()
        if name == "atoms_phi":
            phi = torch.empty(n, dtype=torch.float64, device="cuda")
            fn = lambda: eng.electrostatics_dev(offs, d_xyz.data_ptr(), d_q.data_ptr(), 0, 0, 0, phi.data_ptr())
            pairs, nbytes, P, fld = n * (n - 1), None, n, None
        else:
            P = int(poff[-1])
            phi = torch.empty(P, dtype=torch.float64, device="cuda")
            fld = torch.empty(3 * P, dtype=torch.float64, device="cuda") if field else None
            fn = lambda: eng.potential_points_dev(offs, d_xyz.data_ptr(), d_q.data_ptr(), poff, pts.data_ptr(), phi.data_ptr(),
                                                  fld.data_ptr() if field else 0)
            sizes = np.diff(offs).astype(np.int64)
            pairs = int((np.diff(poff) * sizes).sum())
            nbytes = P * (24 + (32 if field else 8))
        torch.cuda.synchronize()
        calls = args.calls if pairs > 1e9 else 10 * args.calls
        ms = timed(torch, stream, fn, args.warmup, calls)
        ms2 = timed(torch, stream, fn, 0, calls)
        if name == "atoms_phi":
            worst = None
        else:
            worst = check_sample(xyz, q, offs, poff, pts, phi, fld, rng)
        row = {"workload": name, "desc": desc, "systems": n_sys, "atoms": n, "points": P, "pairs": pairs, "calls": calls,
               "ms": round(ms, 4), "ms_repeat": round(ms2, 4), "gpairs_per_s": round(pairs / (ms * 1e-3) / 1e9, 1),
               "checked_max_err_over_scale": worst}
        if nbytes:
            row["bytes"] = nbytes
            row["gbytes_per_s"] = round(nbytes / (ms * 1e-3) / 1e9, 1)
        print(f"{name}: {ms:.4f} / {ms2:.4f} ms, {row['gpairs_per_s']} G pairs/s"
              + (f", {row['gbytes_per_s']} GB/s" if nbytes else "") + f", errors {worst}", flush=True)
        result["workloads"].append(row)
        del d_xyz, d_q, phi, fld
        if name not in ("atoms_phi",):
            del pts
        torch.cuda.empty_cache()
    eng.close()
    return result


def main():
    names = ["split", "grid_phi", "grid_field", "galectin", "qm9", "atoms_phi"]
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workloads", nargs="+", default=names, choices=names)
    ap.add_argument("--atoms", type=int, default=100_000)
    ap.add_argument("--molecules", type=int, default=10_000)
    ap.add_argument("--calls", type=int, default=10, help="timed calls per window (10x for calls under 10^9 pairs)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()
    res = run(args)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
