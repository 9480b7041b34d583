"""Two real GPUs (skipped on a 1-GPU box): the sharded large-system path (epnn_shard_init: rows owned per rank,
ncclAllGather of v / l2 / q inside the library) must reproduce the single-GPU charges BIT FOR BIT on every rank,
including a batch that mixes small systems in, a system cut in the middle of a row block, and the hidden state."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _inputs():
    from epnn_b200 import synth
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    d = np.load(os.path.join(root, "tests", "golden", "protein.npz"))
    sp = synth.species_from_Z(d["Z"], 9)
    offs_s, xyz_s, sp_s, Q_s = synth.qm9_shaped(5, 9, seed=2)
    n = len(sp)
    offs = np.concatenate([offs_s, [offs_s[-1] + n, offs_s[-1] + n + 700]]).astype(np.int32)
    xyz = np.concatenate([xyz_s, d["xyz"], d["xyz"][100:800]]).astype(np.float32)
    spc = np.concatenate([sp_s, sp, sp[100:800]]).astype(np.int32)
    Q = np.concatenate([Q_s, [2.0, -1.0]]).astype(np.float32)
    npad = np.concatenate([np.full(5, 29), [n, 720]]).astype(np.int32)
    return offs, xyz, spc, Q, npad


def _worker(rank, world, port, tmp):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from epnn_b200.checkpoint import load_weights
        from epnn_b200.engine import Engine
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        offs, xyz, sp, Q, npad = _inputs()
        for name in ("decay_model_weights", "model2_weights"):
            w = load_weights(os.path.join(root, "tests", "golden", "checkpoints", name))
            eng = Engine(w, device=rank)
            single = eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)[1].copy()
            eng.set_option("keep_hidden", 1)
            eng.infer_batch(offs, xyz, sp, Q, npad)
            h1 = eng.hidden(int(offs[-1])).copy()
            eng.set_shard(rank, world)
            sharded = eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)[1].copy()
            h2 = eng.hidden(int(offs[-1])).copy()
            st = eng.shard_state
            assert st["calls"] == (w.T - 1) + 2 + w.T + 1 and st["bytes"] > 0      # v per step but the last, l2 + h, q per pass, full degrees
            assert np.array_equal(single, sharded), (name, np.abs(single - sharded).max())
            assert np.array_equal(h1, h2)
            eng.set_shard(0, 1)
            again = eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)[1]
            assert np.array_equal(single, again)
            # the optional tensor-core far kernel shards the same way and stays bit-identical to its own 1-GPU run
            eng.set_option("gnn_far_tensor", 1)
            tc1 = eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)[1].copy()
            eng.set_shard(rank, world)
            tc2 = eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)[1].copy()
            assert np.array_equal(tc1, tc2), (name, "tensor", np.abs(tc1 - tc2).max())
            eng.close()
        # the all-FP64 kernels and the mixed precision shard the same way; several chunks per call (the staging pipeline) too
        w = load_weights(os.path.join(root, "tests", "golden", "checkpoints", "model2_weights"))
        for precision in (64, 48):
            eng = Engine(w, device=rank, precision=precision)
            eng.set_option("chunk_atoms", 3000)              # 3 chunks: small systems | protein | 700-atom system
            single = eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)[1].copy()
            eng.set_shard(rank, world)
            sharded = eng.infer_batch(offs, xyz, sp, Q, npad, want_f64=True)[1].copy()
            assert np.array_equal(single, sharded), (precision, np.abs(single - sharded).max())
            eng.close()
        open(os.path.join(tmp, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_large_system_is_bit_identical(tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert os.path.exists(tmp_path / "ok0") and os.path.exists(tmp_path / "ok1")
