"""Electrostatics of the predicted charges against the inference that produced them, on one GPU.

Workloads (the two headline shapes of bench.py):
  qm9      synth.qm9_shaped(1 000 000) molecules, pad N = 29, decay_model_weights (bench.py's default workload)
  protein  synth.protein_like(100 000), one system
For each: the inference call (infer_batch_dev) and the electrostatics of its device-resident FP64 charges
(electrostatics_dev: energy, dipole and potential) are timed with CUDA events on the engine's stream after warm-up, and a
sample of the outputs is checked against a float64 numpy evaluation.  Prints one JSON line (and writes it to --out).

    python tools/bench_electrostatics.py --out profiles/r03/electrostatics_b200.json
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


def run(args):
    import torch
    from epnn_b200 import synth
    from epnn_b200.checkpoint import load_weights
    from epnn_b200.engine import Engine
    w = load_weights(os.path.join(ROOT, "tests", "golden", "checkpoints", "decay_model_weights"))
    eng = Engine(w, device=0)
    stream = torch.cuda.ExternalStream(eng.stream)
    result = {"gpu": gpu_info(), "workloads": []}
    for name in args.workloads:
        if name == "qm9":
            offs, xyz, sp, Q = synth.qm9_shaped(args.molecules, w.n_x, seed=0)
            npad = np.full(len(offs) - 1, 29, np.int32)
            desc = f"synth.qm9_shaped({args.molecules}), pad N = 29, decay_model_weights"
        else:
            offs, xyz, sp, Q = synth.protein_like(args.atoms, w.n_x, seed=1)
            npad = None
            desc = f"synth.protein_like({args.atoms}), decay_model_weights"
        S, n = len(offs) - 1, int(offs[-1])
        d_xyz, d_sp, d_Q = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (xyz, sp, Q))
        q32, q64 = torch.empty(n, dtype=torch.float32, device="cuda"), torch.empty(n, dtype=torch.float64, device="cuda")
        e, mu, phi = (torch.empty(m, dtype=torch.float64, device="cuda") for m in (S, 3 * S, n))
        torch.cuda.synchronize()
        infer = lambda: eng.infer_batch_dev(offs, d_xyz.data_ptr(), d_sp.data_ptr(), d_Q.data_ptr(), npad, q32.data_ptr(), q64.data_ptr())
        elst = lambda: eng.electrostatics_dev(offs, d_xyz.data_ptr(), q64.data_ptr(), 0, e.data_ptr(), mu.data_ptr(), phi.data_ptr())
        ms_infer = timed(torch, stream, infer, args.warmup, args.infer_calls)
        ms_elst = timed(torch, stream, elst, args.warmup, args.calls)
        ms_elst_again = timed(torch, stream, elst, 0, args.calls)          # a second window: the spread of the number
        # check a sample against float64 numpy
        qh, eh, muh, phih = q64.cpu().numpy(), e.cpu().numpy(), mu.cpu().numpy().reshape(-1, 3), phi.cpu().numpy()
        rng = np.random.default_rng(7)
        worst = {"energy": None, "dipole": 0.0, "phi": 0.0}          # energy: only systems whose every row is sampled
        pairs = 0
        for s in (rng.choice(S, size=min(S, 2000), replace=False) if S > 1 else [0]):      # 512 sampled rows above 4 096 atoms
            a0, a1 = int(offs[s]), int(offs[s + 1])
            x = xyz[a0:a1].astype(np.float64)
            c = x.mean(0)
            ref_mu = qh[a0:a1] @ (x - c)
            mu_scale = np.abs(qh[a0:a1]) @ np.linalg.norm(x - c, axis=1)
            worst["dipole"] = max(worst["dipole"], float(np.abs(muh[s] - ref_mu).max() / max(mu_scale, 1e-300)))
            idx = np.arange(a1 - a0) if a1 - a0 <= 4096 else np.sort(rng.choice(a1 - a0, size=512, replace=False))
            rinv_rows = []
            for b0 in range(0, len(idx), 128):
                d = x[idx[b0:b0 + 128]][:, None, :] - x[None, :, :]
                r = np.sqrt((d * d).sum(-1))
                rinv_rows.append(np.where(r > 0, 1.0 / np.where(r > 0, r, 1.0), 0.0))
            rinv = np.concatenate(rinv_rows)
            pairs += rinv.size
            ref_phi, phi_scale = rinv @ qh[a0:a1], rinv @ np.abs(qh[a0:a1])
            worst["phi"] = max(worst["phi"], float((np.abs(phih[a0 + idx] - ref_phi) / np.maximum(phi_scale, 1e-300)).max()))
            if len(idx) == a1 - a0:
                ref_e, e_scale = 0.5 * qh[a0:a1] @ ref_phi, 0.5 * np.abs(qh[a0:a1]) @ phi_scale
                worst["energy"] = max(worst["energy"] or 0.0, float(abs(eh[s] - ref_e) / max(e_scale, 1e-300)))
        sizes = np.diff(offs).astype(np.int64)
        ordered_pairs = int((sizes * (sizes - 1)).sum())
        row = {"workload": name, "desc": desc, "systems": S, "atoms": n, "ordered_pairs": ordered_pairs,
               "ms_infer": round(ms_infer, 3), "ms_electrostatics": round(ms_elst, 4), "ms_electrostatics_repeat": round(ms_elst_again, 4),
               "electrostatics_over_infer": round(ms_elst / ms_infer, 5),
               "gpairs_per_s": round(ordered_pairs / (ms_elst * 1e-3) / 1e9, 1),
               "checked": {"max_err_over_scale": worst, "sampled_pairs": pairs, "bound": "1e-12 (n <= 48) / 1e-11 (n > 48)"}}
        print(f"{name}: infer {ms_infer:.3f} ms, electrostatics {ms_elst:.4f} / {ms_elst_again:.4f} ms "
              f"({100 * ms_elst / ms_infer:.2f} % of inference), {row['gpairs_per_s']} G ordered pairs/s, errors {worst}", flush=True)
        result["workloads"].append(row)
        del d_xyz, d_sp, d_Q, q32, q64, e, mu, phi
        torch.cuda.empty_cache()
    eng.close()
    return result


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workloads", nargs="+", default=["qm9", "protein"], choices=["qm9", "protein"])
    ap.add_argument("--molecules", type=int, default=1_000_000)
    ap.add_argument("--atoms", type=int, default=100_000)
    ap.add_argument("--calls", type=int, default=20, help="timed electrostatics calls per window")
    ap.add_argument("--infer-calls", type=int, default=5, help="timed inference calls")
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
