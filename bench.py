#!/usr/bin/env python
"""bench.py -- atoms/s of EPNN charge inference (BASELINE.json metric) on N B200s of one node.

A "step" is one pass of the hot path (neighbour list + descriptors -> T message-passing steps -> T
electron-passing passes -> charges) over one batch of synthetic input:

  workload "qm9"     (default; BASELINE.json configs[3]) : --molecules QM9-shaped molecules PER GPU, drawn from
                     the 1338 QM9 molecules of data/mixed, randomly rotated + jittered (epnn_b200/synth.py),
                     Q = 0, pad N = 29, decay_model_weights.  Molecules are independent, so N GPUs hold N
                     disjoint shards of the same stream (molecule k depends only on (seed, k)) and there is
                     no data-path collective: "scaling": "weak".
  workload "qm9_test" / "ssi" (BASELINE.json configs[0]/[1]): the reference's own data -- the 1338 QM9 molecules of
                     data/mixed with model_weights, the 2979 SSI dimers (net charge 0, +-1, +-2) with model2_weights --
                     from the packed fixture tests/golden/mixed.npz, pad N = 41 (the pad of the reference's mixed set).
                     Small batches (24 k / 66 k atoms): these lines are latency-bound and secondary; parity on the
                     same systems is tests/test_gpu_parity.py.  Every rank runs the whole set (replicas only).
  workload "protein" (BASELINE.json configs[2]/[4])      : one protein-like system of --atoms atoms (Galectin-3C
                     tiled), exact all-pairs GNN.  With --gpus N the SAME system is sharded over the N ranks
                     (epnn_set_shard: pair kernels split by ranges, one NCCL all-reduce per step / pass): "scaling":
                     "strong".  --gnn-far-tensor 1 moves the O(n^2) far part to the tcgen05 tensor cores (3xTF32).

Printed JSON (rank 0, one line): the driver contract + "roofline" (dominant kernel, FP32-SIMT bound, against
the FMA peak measured in the same run; the HBM-side kernels against MEASURED_PEAKS.json) + "cpu_baseline"
(the numpy oracle's reference formulation on the box's host cores, bounded sample).

`--impl reference` times that CPU formulation as its own arm (rank 0 only).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"        # NCCL's version banner goes to stdout; stdout carries exactly one JSON line
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

METRIC = "atoms/sec EPNN charge inference"
UNIT = "atoms/s"
FLOP_PAIR = 2 * 32 * 32 + 3 * 32           # per ordered (i,j) pair per GNN step (SURVEY.md 8d): 2144
FLOP_PAIR_E = 2 * 48 * 32                  # extra for pairs with e != 0: 3072
FLOP_EPN_PAIR = 2 * (48 * 32 + 2 * (32 * 32 + 32)) + 2 * 64   # per unordered near pair per pass: 7424
DUMP_MAX_ATOMS = 4_000_000                 # --dump-outputs: 12 B per atom (float32 + float64 charge), at most 48 MB


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="qm9", choices=["qm9", "protein", "qm9_test", "ssi"])
    ap.add_argument("--molecules", type=int, default=1_000_000, help="QM9-shaped molecules per GPU per step")
    ap.add_argument("--atoms", type=int, default=2220, help="atoms of the protein-like system (workload protein)")
    ap.add_argument("--npad", type=int, default=29, help="pad size N of the reference's dense model (qm9 workload)")
    ap.add_argument("--checkpoint", default=None, help="default: decay_model_weights (qm9, protein), model_weights (qm9_test), model2_weights (ssi)")
    ap.add_argument("--precision", type=int, default=32, choices=[0, 32, 48, 64], help="0 auto (probe), 32 FP32, 48 mixed (FP64 per-atom kernel), 64 all FP64")
    ap.add_argument("--chunk-atoms", type=int, default=0, help="override the library's internal batch size")
    ap.add_argument("--ref-molecules", type=int, default=2048, help="molecules per step of the CPU reference arm")
    ap.add_argument("--gnn-far-tensor", type=int, default=2, choices=[0, 1, 2],
                    help="big systems: far part of the message sum on tcgen05 tensor cores (3xTF32) instead of FP32 SIMT; 2 = auto (>= 16384 atoms)")
    ap.add_argument("--pair-tensor", type=int, default=0, choices=[0, 1],
                    help="small systems: electron-passing pair MLP on mma.sync 3xTF32 instead of FP32 SIMT (opt-in)")
    ap.add_argument("--atom-tensor", type=int, default=1, choices=[0, 1],
                    help="FP32 per-atom kernel (update MLP, projections: GEMMs over all atoms) on mma.sync 3xTF32 (default) instead of FP32 SIMT")
    ap.add_argument("--pair-const", type=int, default=2, choices=[0, 1, 2],
                    help="FP32 kernel set: 2 default (row-run GNN bundle kernel + pair-per-thread EPN kernel), 1 pair-per-thread everywhere, 0 round-1 warp-tile kernels")
    ap.add_argument("--dedup-far", type=int, default=1, choices=[0, 1], help="collapse species-equivalent far columns (exact; 0 = ablation)")
    ap.add_argument("--secondary", type=int, default=1, choices=[0, 1], help="append the secondary blocks (strong scaling, live-GNN checkpoints, the reference's own configs) to the JSON line")
    ap.add_argument("--strong-atoms", type=int, default=100_000, help="atoms of the large system of the strong-scaling block")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write rank 0's charges of the last timed step to DIR/charges.npy (float32) and "
                         f"DIR/charges_f64.npy (float64); above {DUMP_MAX_ATOMS} atoms both hold the same fixed, seeded sample of atoms")
    args = ap.parse_args()
    if args.checkpoint is None:
        args.checkpoint = {"qm9_test": "model_weights", "ssi": "model2_weights"}.get(args.workload, "decay_model_weights")
    if args.workload in ("qm9_test", "ssi") and args.npad == 29:
        args.npad = 41
    return args


# ------------------------------------------------------------------------------------------------ workloads
_QM9_CACHE = {}


def qm9_stream(n_mol, n_x, seed, first):
    """synth.qm9_shaped, memoised: the secondary blocks reuse the headline stream (generation is host work, outside every timed region)."""
    from epnn_b200 import synth
    key = (n_mol, seed, first)
    if key not in _QM9_CACHE:
        _QM9_CACHE.clear()
        offs, xyz, sp9, Q = synth.qm9_shaped(n_mol, 9, seed=seed, first=first)
        _QM9_CACHE[key] = (offs, np.ascontiguousarray(xyz, np.float32), sp9, Q)
    offs, xyz, sp9, Q = _QM9_CACHE[key]
    sp = sp9 if n_x == 9 else np.where(sp9 >= 5, sp9 + 1, sp9).astype(np.int32)      # the 10-wide table inserts P at index 5
    return offs, xyz, sp, Q


def make_workload(args, w, rank):
    from epnn_b200 import synth
    if args.workload == "qm9":
        offs, xyz, sp, Q = qm9_stream(args.molecules, w.n_x, args.seed, rank * args.molecules)
        npad = np.full(args.molecules, args.npad, np.int32)
        desc = {"workload": f"synthetic QM9-shaped molecules (<=29 atoms), {args.molecules} per GPU per step, pad N={args.npad}",
                "molecules_per_gpu": args.molecules}
    elif args.workload in ("qm9_test", "ssi"):
        offs, xyz, sp, Q, n_sel = real_set(args.workload, w.n_x, limit=getattr(args, "limit_systems", 0))
        npad = np.full(n_sel, args.npad, np.int32)
        desc = {"workload": f"{'QM9 molecules' if args.workload == 'qm9_test' else 'SSI dimers'} of the reference's data/mixed "
                            f"({n_sel} systems, {int(offs[-1])} atoms per step), pad N={args.npad}", "systems_per_gpu": n_sel}
    else:
        offs, xyz, sp, Q = synth.protein_like(args.atoms, w.n_x, seed=1)      # the SAME system on every rank (sharded)
        npad = np.array([args.atoms], np.int32)
        desc = {"workload": f"protein-like single system, {args.atoms} atoms (Galectin-3C tiled), pad N=n, exact all-pairs GNN",
                "atoms": args.atoms}
    return offs, np.ascontiguousarray(xyz, np.float32), sp, Q, npad, desc


def data_kind(args):
    return "synthetic" if args.workload in ("qm9", "protein") else "reference data/mixed (tests/golden/mixed.npz)"


def real_set(which, n_x, limit=0):
    """Packed arrays of the reference's own QM9 molecules / SSI dimers (tests/golden/mixed.npz, made by
    tests/golden/make_fixtures.py from data/mixed.tar.gz), in fixture order."""
    from epnn_b200 import synth
    d = np.load(os.path.join(GOLDEN, "mixed.npz"))
    names = [str(x) for x in d["names"]]
    prefix = "dsgdb9nsd_" if which == "qm9_test" else "SSI-"
    sel = [i for i, nm in enumerate(names) if nm.startswith(prefix)]
    if limit:
        sel = sel[:limit]
    o = d["offsets"]
    idx = np.concatenate([np.arange(o[i], o[i + 1]) for i in sel])
    sizes = np.array([o[i + 1] - o[i] for i in sel])
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    return (offs, np.ascontiguousarray(d["xyz"][idx], np.float32), synth.species_from_Z(d["Z"][idx], n_x).astype(np.int32),
            np.ascontiguousarray(d["Q"][sel], np.float32), len(sel))


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.lines = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smax.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ CPU reference arm
_W = None


def _ref_init(ckpt):
    global _W
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:
        pass
    from epnn_b200.checkpoint import load_weights
    _W = load_weights(os.path.join(GOLDEN, "checkpoints", ckpt))


def _ref_work(job):
    """The reference formulation (dense padded (N*N,K) pair inputs, three Dense layers per MLP, float32 like
    Keras) for a slice of systems, including get_init_edges: oracle.forward_literal."""
    from oracle import epnn_oracle as O
    xyz, sp, Q, offs, npad = job
    out = []
    for s in range(len(Q)):
        a0, a1 = offs[s], offs[s + 1]
        out.append(O.forward_literal(_W, xyz[a0:a1], sp[a0:a1], Q[s], int(npad[s]), np.float32))
    return np.concatenate(out) if out else np.zeros(0)


def run_reference(args):
    """`--impl reference`: rank 0 times the CPU port of the reference path on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    from epnn_b200.checkpoint import load_weights
    w = load_weights(os.path.join(GOLDEN, "checkpoints", args.checkpoint))
    cores = os.cpu_count() or 1
    sub = argparse.Namespace(**vars(args))
    if args.workload == "qm9":
        sub.molecules = args.ref_molecules
        sample = f"{args.ref_molecules} molecules of the same synthetic stream per step (of {args.molecules} per GPU)"
    elif args.workload in ("qm9_test", "ssi"):
        sub.limit_systems = min(args.ref_molecules, 512)
        sample = f"the first {sub.limit_systems} systems of the set per step"
    else:
        sub.atoms = min(args.atoms, 2220)
        sample = f"one {sub.atoms}-atom system per step"
    offs, xyz, sp, Q, npad, desc = make_workload(sub, w, 0)
    n_sys = len(Q)
    # one job per core (contiguous slices); a single big system cannot be split -> 1 process using BLAS threads
    if n_sys >= cores:
        bounds = np.linspace(0, n_sys, cores + 1).astype(int)
        jobs = []
        for c in range(cores):
            s0, s1 = bounds[c], bounds[c + 1]
            a0, a1 = offs[s0], offs[s1]
            jobs.append((xyz[a0:a1], sp[a0:a1], Q[s0:s1], offs[s0:s1 + 1] - a0, npad[s0:s1]))
        pool = mp.get_context("fork").Pool(cores, initializer=_ref_init, initargs=(args.checkpoint,))
        step = lambda: pool.map(_ref_work, jobs)
        used = cores
    else:
        pool = None
        global _W
        _W = w
        jobs = [(xyz, sp, Q, offs, npad)]
        step = lambda: [_ref_work(jobs[0])]
        used = cores      # OpenBLAS default: all cores
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    if pool is not None:
        pool.close()
    atoms = int(offs[-1]) * args.steps
    value = atoms / dt
    _, _, _, _, _, full_desc = make_workload_desc_only(args)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": data_kind(args), "config": full_desc,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": "port", "sample": sample,
                             "what": "numpy float32 restatement of the reference formulation (oracle.forward_literal: "
                                     "get_init_edges + dense padded pair tensors + 3 Dense layers per MLP); TensorFlow is "
                                     "not installable in this image"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def make_workload_desc_only(args):
    if args.workload == "qm9":
        desc = {"workload": f"synthetic QM9-shaped molecules (<=29 atoms), {args.molecules} per GPU per step, pad N={args.npad}",
                "molecules_per_gpu": args.molecules}
    elif args.workload in ("qm9_test", "ssi"):
        desc = {"workload": f"{'QM9 molecules' if args.workload == 'qm9_test' else 'SSI dimers'} of the reference's data/mixed, pad N={args.npad}"}
    else:
        desc = {"workload": f"protein-like single system, {args.atoms} atoms (Galectin-3C tiled), pad N=n, exact all-pairs GNN",
                "atoms_per_gpu": args.atoms}
    desc.update({"checkpoint": args.checkpoint, "parallelism": f"molecule-shards x{args.gpus}, no collective"})
    return None, None, None, None, None, desc


def cpu_baseline_subprocess(args):
    """Run the reference arm in a fresh interpreter (no CUDA context to fork) and return its cpu_baseline."""
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "1",
           "--workload", args.workload, "--molecules", str(args.molecules), "--atoms", str(min(args.atoms, 2220)),
           "--npad", str(args.npad), "--checkpoint", args.checkpoint, "--ref-molecules", str(args.ref_molecules),
           "--seed", str(args.seed)]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE")}
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
        for ln in reversed(out.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)["cpu_baseline"]
        return {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": "failed: " + out.stderr[-300:]}
    except Exception as ex:      # noqa: BLE001
        return {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex}"}


# ------------------------------------------------------------------------------------------------ B200 arm
class Box:
    """torch / torch.distributed plumbing of one rank (device memory, streams, barriers) -- not the product."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: epnn_b200 has no CPU fallback (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, x):
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([x], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, xs):
        if self.world == 1:
            return [float(x) for x in xs]
        t = self.torch.tensor(list(xs), device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t)
        return [float(x) for x in t.tolist()]


def make_engine(box, args, ckpt, precision=None, timing=True):
    from epnn_b200.checkpoint import load_weights
    from epnn_b200.engine import Engine
    w = load_weights(os.path.join(GOLDEN, "checkpoints", ckpt))
    eng = Engine(w, device=box.local, precision=args.precision if precision is None else precision)
    if timing:
        eng.set_option("timing", 1)
    if args.chunk_atoms:
        eng.set_option("chunk_atoms", args.chunk_atoms)
    eng.set_option("gnn_far_tensor", args.gnn_far_tensor)
    if not args.dedup_far:
        eng.set_option("dedup_far", 0)
    if args.pair_tensor:
        eng.set_option("pair_tensor", 1)
    eng.set_option("pair_const", args.pair_const)
    eng.set_option("atom_tensor", args.atom_tensor)
    return w, eng


def time_case(box, eng, offs, xyz, sp, Q, npad, steps, warmup, host_too=True, clocks=False):
    """W warm-up + K timed steps of one workload on this rank's engine.  Device-resident arm (inputs already in HBM, CUDA
    events on the ctx stream, max over ranks) and, if asked, the end-to-end arm through the host API (pinned host buffers,
    H2D + D2H inside the timed region).  Returns a dict; q64 = the FP64 copy of the charges of the device arm."""
    torch = box.torch
    n_atoms = int(offs[-1])
    stream = torch.cuda.ExternalStream(eng.stream, device=box.dev)

    def timed(step_fn):
        for _ in range(warmup):
            step_fn()
        box.barrier()
        clk = ClockSampler(box.local)
        if clocks and box.rank == 0:
            clk.start()
            time.sleep(0.25)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        acc = {}
        box.barrier()
        e0.record(stream)
        for _ in range(steps):
            step_fn()
            for k, v in eng.last_stats.items():
                acc[k] = acc.get(k, 0) + v
        e1.record(stream)
        e1.synchronize()
        box.barrier()
        ms = box.max_over_ranks(e0.elapsed_time(e1))
        return ms, acc, (clk.stop() if clocks and box.rank == 0 else None)

    d_xyz = torch.from_numpy(xyz).to(box.dev)
    d_sp = torch.from_numpy(sp).to(box.dev)
    d_Q = torch.from_numpy(Q).to(box.dev)
    d_out = torch.empty(n_atoms, dtype=torch.float32, device=box.dev)
    d_out64 = torch.empty(n_atoms, dtype=torch.float64, device=box.dev)
    torch.cuda.synchronize(box.dev)

    def step_dev():
        eng.infer_batch_dev(offs, d_xyz.data_ptr(), d_sp.data_ptr(), d_Q.data_ptr(), npad, d_out.data_ptr(), d_out64.data_ptr())

    ms_dev, acc, clk = timed(step_dev)
    res = {"ms_dev": ms_dev, "acc": acc, "clocks": clk, "q32": d_out.cpu().numpy(), "q64": d_out64.cpu().numpy(), "n_atoms": n_atoms,
           "e2e_ms": None}
    del d_xyz, d_sp, d_Q, d_out, d_out64
    if host_too:
        h_xyz = eng.pinned_empty(xyz.shape, np.float32); h_xyz[...] = xyz
        h_sp = eng.pinned_empty(sp.shape, np.int32); h_sp[...] = sp
        h_Q = eng.pinned_empty(Q.shape, np.float32); h_Q[...] = Q
        h_out = eng.pinned_empty((n_atoms,), np.float32)

        def step_host():
            eng.infer_batch(offs, h_xyz, h_sp, h_Q, npad, out=h_out)

        ms_e2e, _, _ = timed(step_host)
        if not np.array_equal(h_out, res["q32"]):
            raise SystemExit("host-API and device-API results differ")
        res["e2e_ms"] = ms_e2e
        res["h2d"] = int(xyz.nbytes + sp.nbytes + Q.nbytes + offs.nbytes + npad.nbytes)
        res["d2h"] = int(h_out.nbytes)
        eng.free_pinned()
    return res


def conservation(q64, offs, Q):
    """max |sum_i q_i - Q| per system from the FP64 charges, next to the floor the reference's own initial state imposes:
    q0 = fl32(fl32(Q)/n) on every atom (charge_gn.py:337-338) already misses Q by up to n * ulp(Q/n)/2."""
    n = np.diff(offs).astype(np.float64)
    sums = np.add.reduceat(q64, offs[:-1])
    q0 = (Q.astype(np.float32) / n.astype(np.float32)).astype(np.float32).astype(np.float64)
    return {"max_abs_sum_q_minus_Q": float(np.abs(sums - Q.astype(np.float64)).max()),
            "q0_floor_max_abs_n_q0_minus_Q": float(np.abs(q0 * n - Q.astype(np.float64)).max()),
            "from": "FP64 copy of the charges (q_out_f64); the float32 output rounds each charge by up to 6e-8 |q| on top"}


def dump_outputs(out_dir, q32, q64):
    """--dump-outputs: the charges the device arm's caller holds after the last timed step (q_out float32, q_out64 float64).
    Above DUMP_MAX_ATOMS atoms both files hold the same atoms, drawn with a fixed seed and kept in atom order, so two builds
    run with the same arguments can be compared entry for entry."""
    os.makedirs(out_dir, exist_ok=True)
    if len(q32) > DUMP_MAX_ATOMS:
        idx = np.sort(np.random.default_rng(0).choice(len(q32), DUMP_MAX_ATOMS, replace=False))
        q32, q64 = q32[idx], q64[idx]
    np.save(os.path.join(out_dir, "charges.npy"), np.ascontiguousarray(q32, np.float32))
    np.save(os.path.join(out_dir, "charges_f64.npy"), np.ascontiguousarray(q64, np.float64))


def secondary_blocks(box, args, main_res, main_value):
    """Driver-visible evidence beyond the headline line (VERDICT r01 items 3 and 8): strong scaling of both multi-GPU configs,
    a live-GNN checkpoint on the headline workload, and the reference's own three configurations.  Short runs (3 steps)."""
    from epnn_b200 import synth
    out = {}
    world, rank = box.world, box.rank
    K, W = 3, 3
    # ---- strong scaling, many small molecules: --molecules in TOTAL, a contiguous 1/N of the stream per rank, no collective
    if world > 1:
        w, eng = make_engine(box, args, "decay_model_weights")
        per = args.molecules // world
        offs, xyz, sp, Q = synth.qm9_shaped(per, w.n_x, seed=args.seed, first=rank * per)      # another slice of the stream: not cached
        r = time_case(box, eng, offs, np.ascontiguousarray(xyz, np.float32), sp, Q, np.full(per, args.npad, np.int32), K, W, host_too=False)
        tot = box.sum_over_ranks([r["n_atoms"]])[0]
        out["strong_qm9"] = {"workload": f"{per * world} QM9-shaped molecules in total, {per} per GPU, no collective", "scaling": "strong",
                             "value": tot * K / (r["ms_dev"] * 1e-3), "unit": UNIT, "ms_per_step": r["ms_dev"] / K, "steps": K, "warmup": W,
                             "limiter": "per-chunk fixed cost (one host sync after the neighbour count, ~60 launches) over 1/N of the atoms"}
        eng.close()
    else:
        out["strong_qm9"] = {"workload": f"{args.molecules} QM9-shaped molecules in total on 1 GPU (= the headline line)", "scaling": "strong",
                             "value": main_value, "unit": UNIT, "ms_per_step": main_res["ms_dev"] / args.steps, "steps": args.steps, "warmup": args.warmup}
    # ---- strong scaling, one large system sharded over the ranks (BASELINE config 5 at a size that steps in about a second)
    w, eng = make_engine(box, args, "decay_model_weights")
    offs, xyz, sp, Q = synth.protein_like(args.strong_atoms, w.n_x, seed=1)
    xyz = np.ascontiguousarray(xyz, np.float32)
    npad = np.array([args.strong_atoms], np.int32)
    ident = None
    if world > 1:
        single = None
        if rank == 0:                                        # rank 0's single-GPU result: the sharded run must reproduce it bit for bit
            single = eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)[1].copy()
        eng.set_shard(rank, world)
    r = time_case(box, eng, offs, xyz, sp, Q, npad, K, 1, host_too=False)
    if world > 1 and rank == 0:
        ident = bool(np.array_equal(single, r["q64"]))
    ph = {k: r["acc"][k] / K for k in r["acc"] if k.startswith("ms_")}
    out["strong_protein"] = {"workload": f"protein-like single system, {args.strong_atoms} atoms, exact all-pairs GNN, sharded over {world} GPU(s)",
                             "scaling": "strong", "value": args.strong_atoms * K / (r["ms_dev"] * 1e-3), "unit": UNIT,
                             "ms_per_step": r["ms_dev"] / K, "steps": K, "warmup": 1, "phases_ms_per_step": ph,
                             "bit_identical_to_single_gpu": ident, "exchange": getattr(eng, "shard_state", None) and
                             {k: v for k, v in eng.shard_state.items() if k in ("calls", "bytes")},
                             "checks": conservation(r["q64"], offs, Q)}
    eng.set_shard(0, 1)
    eng.close()
    # ---- the headline workload with a checkpoint whose GNN is live at every step but the first (the default checkpoint's update
    #      MLP is dead at 3 of 5 steps, which the exact far-column de-duplication exploits)
    for ck in ("model2_weights", "model_weights"):
        w, eng = make_engine(box, args, ck, precision=32)
        n_mol = args.molecules
        offs, xyz, sp, Q = qm9_stream(n_mol, w.n_x, args.seed, rank * n_mol)
        r = time_case(box, eng, offs, np.ascontiguousarray(xyz, np.float32), sp, Q, np.full(n_mol, args.npad, np.int32), K, W, host_too=False)
        tot = box.sum_over_ranks([r["n_atoms"]])[0]
        out["live_gnn_" + ck] = {"workload": f"{n_mol} QM9-shaped molecules per GPU, {ck} (T={w.T}), FP32 kernels", "scaling": "weak",
                                 "value": tot * K / (r["ms_dev"] * 1e-3), "unit": UNIT, "ms_per_step": r["ms_dev"] / K, "steps": K, "warmup": W,
                                 "fp32_distance_to_oracle": {"model2_weights": "<= 3.9e-6 e", "model_weights": "<= 1.0e-4 e (needs the FP64 kernels for 1e-5)"}[ck] +
                                                            " on data/mixed (profiles/r02/call15_noise_floor.log)"}
        eng.close()
    # ---- the reference's own configurations (BASELINE.json configs[0..2]), rank 0 only: replicas, no sharding
    if rank == 0:
        for wl, ck in (("qm9_test", "model_weights"), ("ssi", "model2_weights")):
            w, eng = make_engine(box, args, ck, precision=0)          # auto: the probe picks the precision that holds 1e-5
            offs, xyz, sp, Q, n_sel = real_set(wl, w.n_x)
            sub = Box.__new__(Box); sub.__dict__.update(box.__dict__); sub.world = 1
            r = time_case(sub, eng, offs, xyz, sp, Q, np.full(n_sel, 41, np.int32), 10, W, host_too=True)
            st = eng.last_stats
            out["config_" + wl] = {"workload": f"{n_sel} {'QM9 molecules' if wl == 'qm9_test' else 'SSI dimers'} of data/mixed, {ck}, pad N=41",
                                   "value": r["n_atoms"] * 10 / (r["ms_dev"] * 1e-3), "unit": UNIT, "ms_per_step": r["ms_dev"] / 10,
                                   "e2e": r["n_atoms"] * 10 / (r["e2e_ms"] * 1e-3), "precision_used": st["precision_used"], "atom_tensor_used": st["atom_tensor_used"],
                                   "probe_max_abs_dq_fp32_vs_fp64_kernels": st["probe_err32"], "probe_max_abs_dq_mixed_vs_fp64_kernels": st["probe_err48"],
                                   "note": "precision 0 (auto): cheapest candidate (FP32 with the tensor per-atom kernel, FP32 SIMT, mixed, FP64; -1 = not needed) whose probe charges are within 2.5e-6 e of the FP64 kernels "
                                           "(which agree with the float64 oracle to 1e-9, tests/test_gpu_parity.py)",
                                   "checks": conservation(r["q64"], offs, Q)}
            eng.close()
        w, eng = make_engine(box, args, "decay_model_weights", precision=32)
        d = np.load(os.path.join(GOLDEN, "protein.npz"))
        n = len(d["Z"])
        offs = np.array([0, n], np.int32)
        xyz = np.ascontiguousarray(d["xyz"], np.float32)
        sp = synth.species_from_Z(d["Z"], 9).astype(np.int32)
        Q = np.array([d["Q"]], np.float32)
        sub = Box.__new__(Box); sub.__dict__.update(box.__dict__); sub.world = 1
        r = time_case(sub, eng, offs, xyz, sp, Q, np.array([n], np.int32), 20, 5, host_too=True)
        out["config_galectin3c"] = {"workload": "Galectin-3C, 2220 atoms, Q=+2, decay_model_weights, pad N=n", "value": n * 20 / (r["ms_dev"] * 1e-3),
                                    "unit": UNIT, "ms_per_step": r["ms_dev"] / 20, "e2e": n * 20 / (r["e2e_ms"] * 1e-3),
                                    "max_abs_dq_vs_reference_preds_npy": float(np.abs(r["q32"] - d["preds"].reshape(-1)).max()),
                                    "checks": conservation(r["q64"], offs, Q)}
        eng.close()
    box.barrier()
    return out


def run_b200(args):
    box = Box(args)
    torch, dist = box.torch, box.dist
    rank, world, local, dev = box.rank, box.world, box.local, box.dev

    # CPU baseline first (rank 0, N = 1 only), before this process owns a CUDA context
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_baseline_subprocess(args)

    w, eng = make_engine(box, args, args.checkpoint)
    offs, xyz, sp, Q, npad, desc = make_workload(args, w, rank)
    n_atoms = int(offs[-1])
    sharded_system = args.workload == "protein" and world > 1
    if sharded_system:                       # one big system: sharded over the ranks
        eng.set_shard(rank, world)
    res = time_case(box, eng, offs, xyz, sp, Q, npad, args.steps, args.warmup, host_too=not args.no_e2e, clocks=True)
    ms_dev, acc, clocks = res["ms_dev"], res["acc"], res["clocks"]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res["q32"], res["q64"])
    e2e = None
    if res["e2e_ms"] is not None:
        e2e = {"value": (1 if sharded_system else world) * n_atoms * args.steps / (res["e2e_ms"] * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": res["h2d"], "d2h_bytes_per_step": res["d2h"], "ms_per_step": res["e2e_ms"] / args.steps}
    checks = conservation(res["q64"], offs, Q)

    # ---- totals over ranks
    tot_atoms, launches = box.sum_over_ranks([n_atoms, acc["n_launches"]])
    tot_atoms, launches = int(tot_atoms), int(launches)
    if sharded_system:
        tot_atoms = n_atoms              # every rank worked on the same atoms (strong scaling)
    value = tot_atoms * args.steps / (ms_dev * 1e-3)

    line = None
    if rank == 0:
        # roofline of the dominant kernel (message-passing pair MLP): FLOPs / CUDA-event time of its launches
        n_sys_sizes = np.diff(offs).astype(np.float64)
        ordered_pairs = float((n_sys_sizes ** 2).sum() + (n_sys_sizes * (npad > np.diff(offs))).sum())
        nnz = 2.0 * acc["n_pairs_e"] / args.steps
        gnn_flops_step = w.T * (FLOP_PAIR * ordered_pairs + FLOP_PAIR_E * nnz)
        epn_flops_step = w.T * FLOP_EPN_PAIR * acc["n_pairs_near"] / args.steps
        ms_gnn = acc["ms_gnn_pair"] / args.steps
        ms_epn = acc["ms_epn_pair"] / args.steps
        fp32_peak = eng.measure_fp32_peak(5)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        phases = {k: acc[k] / args.steps for k in acc if k.startswith("ms_")}
        dominant = max(("ms_gnn_pair", "ms_epn_pair", "ms_neighbor", "ms_gnn_atom", "ms_epn_atom"), key=lambda k: phases[k])
        n_chunks = acc["n_chunks"] / args.steps
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
                if tj.get("workload") == args.workload and not sharded_system:
                    # ncu --set full capture of one launch (profiles/), scaled per atom to this run's launch size
                    traffic = tj["gnn_pair_dram_bytes_per_atom_per_launch"] * n_atoms / n_chunks
            except Exception:   # noqa: BLE001
                traffic = None
        algorithmic = gnn_flops_step / (ms_gnn * 1e-3) * 1e-12 / (world if sharded_system else 1)
        # what the small-system kernel really evaluated (device counters): every slot = one 32x32 second-layer product + glue,
        # every near slot additionally the rank-16 descriptor product -- the exact de-duplication of species-equivalent far columns
        # and the rank-16 basis make this smaller than the algorithmic count
        slots_near = acc.get("n_gnn_near_slots", 0) / args.steps
        slots_far = acc.get("n_gnn_far_slots", 0) / args.steps
        executed = None
        if slots_near + slots_far > 0 and args.workload != "protein":
            executed = (FLOP_PAIR * (slots_near + slots_far) + 2 * 16 * 32 * slots_near) / (ms_gnn * 1e-3) * 1e-12
        headline = executed if executed is not None else algorithmic
        roofline = {
            "kernel": "bundle_run_kernel (message-passing pair MLP of the small systems, FP32 SIMT, FFMA2 with uniform weight operands)"
                      if args.workload != "protein" else "gnn_pair_kernel + gnn_far_const_kernel (message-passing pair MLP of large systems, FP32 SIMT)",
            "bound": "fp32", "achieved": headline, "peak": fp32_peak, "unit": "TFLOP/s", "frac": headline / fp32_peak if fp32_peak else None,
            "achieved_is": "EXECUTED FLOPs (slots the kernel evaluated, device counters) / CUDA-event time" if executed is not None
                           else "ALGORITHMIC FLOPs (SURVEY 8d) / CUDA-event time",
            "algorithmic": {"achieved": algorithmic, "frac": algorithmic / fp32_peak if fp32_peak else None,
                            "note": "SURVEY 8d count of the reference's unmasked n^2 sum: 2144 FLOP per ordered pair + 3072 per e != 0 pair, per step; "
                                    "not a utilisation figure -- the exact far-column de-duplication and the rank-16 descriptor basis skip part of it"},
            "peak_source": "FP32 FMA micro-benchmark measured in this run (epnn_measure_fp32_peak); MEASURED_PEAKS.json "
                           "holds no SIMT peak. north_star: pair MLP defaults to FP32 SIMT, tensor pipe unused",
            "traffic": traffic,
            "launches_per_step": w.T * n_chunks, "avg_launch_ms": ms_gnn / (w.T * n_chunks),
            "algorithmic_flops_per_launch": gnn_flops_step / (w.T * n_chunks),
            "share_of_step": ms_gnn / phases["ms_total"],
            "dominant_phase": dominant,
            "epn_pair": {"achieved": epn_flops_step / (ms_epn * 1e-3) * 1e-12, "unit": "TFLOP/s",
                         "frac": epn_flops_step / (ms_epn * 1e-3) * 1e-12 / fp32_peak if fp32_peak else None},
            "hbm_side": {
                "bound": "hbm", "peak": hbm_peak, "unit": "GB/s",
                "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 (B200_PROFILING.md)",
                "neighbor_build": {"achieved": (20.0 * n_atoms + 4.0 * nnz) / (phases["ms_neighbor"] * 1e-3) * 1e-9},
                "charge_reduction": {"achieved": w.T * (4.0 * nnz + 8.0 * n_atoms) / (phases["ms_epn_atom"] * 1e-3) * 1e-9},
                # the per-atom kernels (update MLP + projections on the tensor path, charge reduction): bytes they have to move per
                # launch (DESIGN.md 4.3: l2 / S rows in, l2 / u / v rows out at 128 B each; q 16 B; 12 B per CSR entry and pass)
                # over the CUDA-event time of their phases
                "per_atom_gnn_phase": {"achieved": n_atoms * (256.0 + 512.0 + max(w.T - 2, 0) * 640.0) / (phases["ms_gnn_atom"] * 1e-3) * 1e-9},
                "per_atom_epn_phase": {"achieved": (n_atoms * (832.0 + (w.T - 1) * 400.0 + 20.0) + w.T * 12.0 * nnz) / (phases["ms_epn_atom"] * 1e-3) * 1e-9},
            },
        }
        if args.workload == "protein":
            # what the message-passing kernels actually executed: far columns of a row collapse to one slot per species (+ the
            # pad slot) at the steps where the device-side check finds the v rows species-wise equal (dedup_far, exact)
            row_steps = float(n_atoms) * w.T
            dd_rows = acc.get("n_far_dedup_rows", 0) / args.steps
            n_slots = len(np.unique(sp)) + (1 if int(npad[0]) > n_atoms else 0)
            far_exec = dd_rows * n_slots + (row_steps - dd_rows) * max(n_atoms - nnz / n_atoms, 0.0)
            exec_flops = FLOP_PAIR * (w.T * nnz + far_exec) + 2 * (16 if args.precision != 64 else 48) * 32 * w.T * nnz
            executed = exec_flops / (ms_gnn * 1e-3) * 1e-12 / (world if sharded_system else 1)
            roofline["far_dedup"] = {"row_steps_collapsed": dd_rows, "row_steps": row_steps, "slots_per_collapsed_row": n_slots}
            if dd_rows > 0:          # the algorithmic count is meaningless once rows collapse: quote what really ran
                roofline.update({"achieved": executed, "frac": executed / fp32_peak if fp32_peak else None,
                                 "achieved_is": "EXECUTED FLOPs (near pairs + species slots + column-by-column far rows) / CUDA-event time"})
        if (args.gnn_far_tensor == 1 or (args.gnn_far_tensor == 2 and n_atoms >= 16384)) and args.precision != 64 and args.workload == "protein":
            # the O(n^2) far part runs on tcgen05 (3xTF32): executed tensor FLOPs = 3 x (2*32*32) per far ordered pair per step
            far_pair_steps = (row_steps - dd_rows) * max(n_atoms - nnz / n_atoms, 0.0)
            tf32_exec = 3.0 * 2 * 32 * 32 * far_pair_steps / (ms_gnn * 1e-3) * 1e-12 / (world if sharded_system else 1)
            tf32_peak = peaks.get("bf16_tflops", 1590.0) / 2.0
            roofline["tensor_far"] = {
                "kernel": "gnn_far_tc_kernel (tcgen05.mma kind::tf32, M128 N32 K8, A in tensor memory, 3xTF32 split)",
                "bound": "tensor", "achieved": tf32_exec, "peak": tf32_peak, "unit": "TFLOP/s", "frac": tf32_exec / tf32_peak,
                "peak_source": "half of MEASURED_PEAKS.json bf16_tflops (TF32 dense = half the bf16 rate)" if "bf16_tflops" in peaks
                               else "half of the fallback 1590 (B200_PROFILING.md)"}
            if far_pair_steps > 0:       # the O(n^2) rows that did not collapse went through the tcgen05 kernel: it is the dominant kernel
                roofline["fp32_view"] = {k: roofline[k] for k in ("kernel", "bound", "achieved", "peak", "unit", "frac", "achieved_is")}
                for k in ("kernel", "bound", "achieved", "peak", "unit", "frac", "peak_source"):
                    roofline[k] = roofline["tensor_far"][k]
                roofline["achieved_is"] = "EXECUTED tensor FLOPs (three TF32 MMAs of the 3xTF32 split per far pair) / CUDA-event time of the message-passing phase"
        for k in ("neighbor_build", "charge_reduction", "per_atom_gnn_phase", "per_atom_epn_phase"):
            roofline["hbm_side"][k]["frac"] = roofline["hbm_side"][k]["achieved"] / hbm_peak
        par = (f"one system sharded x{world}" if sharded_system else f"molecule-shards x{world}, no collective")
        desc.update({"checkpoint": args.checkpoint, "parallelism": par,
                     "l2": "inputs larger than L2 (no flush needed)" if n_atoms * 16 > 126e6 else "inputs smaller than L2",
                     "atoms_per_gpu_per_step": n_atoms, "T": w.T, "precision": args.precision, "precision_used": int(acc["precision_used"] / args.steps),
                     "gnn_far_tensor": args.gnn_far_tensor, "dedup_far": args.dedup_far, "pair_tensor": args.pair_tensor, "pair_const": args.pair_const, "atom_tensor": args.atom_tensor})
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
                "scaling": "strong" if sharded_system else "weak", "vs_baseline": None,
                "dtype": "f64" if int(acc["precision_used"] / args.steps) == 64 else "f32", "data": data_kind(args), "config": desc, "clocks": clocks,
                "e2e": e2e, "gpu_launches": launches, "roofline": roofline,
                "cpu_baseline": cpu_base, "phases_ms_per_step": phases, "checks": checks}
    eng.close()
    if args.secondary and args.workload == "qm9":
        sec = secondary_blocks(box, args, res, value)
        if rank == 0:
            line["secondary"] = sec
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        import socket
        s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    run_b200(args)


if __name__ == "__main__":
    main()
