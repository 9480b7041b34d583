"""Measures the distance to the float64 oracle of every configuration of tests/test_gpu_small_reference.py (q64 and h,
relative per system) and the FP32 error of tests/test_gpu_parity.py::test_bundle_boundaries_and_routing; prints one JSON
object.  The bounds of those tests are 3x these floors.  Needs a GPU:  python tools/measure_small_floor.py [out.json]"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from epnn_b200.checkpoint import load_weights  # noqa: E402
from oracle import epnn_oracle as O  # noqa: E402
import test_gpu_small_reference as T  # noqa: E402


def main():
    G = os.path.join(ROOT, "tests", "golden")
    weights = {n: load_weights(os.path.join(G, "checkpoints", n)) for n in ("decay_model_weights", "model2_weights", "model_weights")}
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    out = {"gpu": gpu, "small": {}}
    runs = {}
    for name, config in T.CASES:
        t0 = time.time()
        res, err = runs[(name, config)] = T.run_config(weights, name, config)
        out["small"][f"{name}/{config}"] = dict(err, sum=res["sum_err"], repeat=res["repeat_equal"], s=round(time.time() - t0, 1),
                                                max_ref_q=float(np.abs(T.reference(weights, name)[1]).max()))
        print(name, config, out["small"][f"{name}/{config}"], flush=True)
    for name in T.LIVE:
        a, b = runs[(name, "default")][0], runs[(name, "fused_prep0")][0]
        out[f"fused_equal/{name}"] = bool(np.array_equal(a["q64"], b["q64"]) and all(
            np.array_equal(a["nbr"][k][i], b["nbr"][k][i]) for k in (0, 1) for i in (0, 1)))
    import test_gpu_parity as P
    from epnn_b200.engine import Engine
    d = np.load(os.path.join(G, "protein.npz"))
    offs, xyz, sp, Q, npad = P.boundary_batch({"xyz": d["xyz"], "Z": d["Z"]})
    ref = O.predict_batch(weights["model2_weights"], offs, xyz, sp, Q, npad)
    eng = Engine(weights["model2_weights"], device=0)
    q32 = eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)[1]
    eng.close()
    out["boundaries_fp32"] = float(np.abs(q32 - ref).max() / max(1.0, np.abs(ref).max()))
    s = json.dumps(out, indent=1)
    print(s)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
