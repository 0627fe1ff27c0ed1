"""Spawn helpers for multi-process tests (gloo on CPU, NCCL on GPU)."""
import os
import traceback

import torch
import torch.multiprocessing as mp


def _entry(rank, world, port, fn, args, errq):
    try:
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(port)
        os.environ["RANK"] = str(rank)
        os.environ["WORLD_SIZE"] = str(world)
        os.environ["LOCAL_RANK"] = str(rank)
        torch.set_num_threads(1)
        import tree_attention_b200 as ta

        ta.setup(rank, world, master_addr="127.0.0.1", master_port=port)
        try:
            fn(rank, world, *args)
        finally:
            ta.cleanup()
    except Exception:
        errq.put((rank, traceback.format_exc()))
        raise


def run_distributed(fn, world, port, args=(), cuda=False):
    """Run ``fn(rank, world, *args)`` on ``world`` spawned ranks.  ``cuda=False``: the ranks see no CUDA device, so they run
    on CPU over gloo on every machine (with CUDA visible, setup() picks NCCL, which refuses two ranks on one GPU).
    ``cuda=True``: one GPU per rank, NCCL."""
    ctx = mp.get_context("spawn")
    errq = ctx.SimpleQueue()
    visible = os.environ.get("CUDA_VISIBLE_DEVICES")
    if not cuda:
        os.environ["CUDA_VISIBLE_DEVICES"] = ""        # inherited by the spawned ranks before they load CUDA
    try:
        mp.spawn(_entry, args=(world, port, fn, args, errq), nprocs=world, join=True)
    except Exception as e:
        msgs = []
        while not errq.empty():
            msgs.append("rank %d:\n%s" % errq.get())
        raise AssertionError("distributed test failed:\n" + "\n".join(msgs) + f"\n{e}")
    finally:
        if visible is None:
            os.environ.pop("CUDA_VISIBLE_DEVICES", None)
        else:
            os.environ["CUDA_VISIBLE_DEVICES"] = visible
