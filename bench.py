"""Headline benchmark (driver contract): ``python bench.py --gpus N --steps K --warmup W [--impl reference]``.

Metric (BASELINE.json): attention forward tokens/sec, whole box, device-timed, max over ranks, at
seq = 128K, 32 heads, d = 128, bf16, synthetic Q/K/V.  The step is the reference's only mode -- ONE
tree-decode attention forward (Sq = 1) over the full 128K-token KV sequence, which is sharded across the
N GPUs (strong scaling: the sequence is fixed, S/N keys per rank).  ``value`` = B * S_global / latency
(sequence tokens attended per second); ``decode_tokens_per_s`` = B / latency is reported alongside.

Own arm: one fused sm_100a kernel per rank per step (local split-KV attention + in-kernel cross-GPU
combine over symmetric memory, no NCCL on the path).
Reference arm (``--impl reference``): the UNMODIFIED ``baseline/_ref/model.py`` ``tree_decode`` through its
own public API on BHSD tensors.  For N > 1 it raises at model.py:111 (SURVEY.md D3) and the arm reports
``unavailable``.

Timing rules implemented here: W >= 3 warm-ups; CUDA events on the launching stream bracketed by barrier +
synchronize; max over ranks; the KV working set cycled per step is > 4x the 126 MB L2 (several KV buffers
are rotated like layers of a model) so no step is served from L2; SM clocks / throttle reasons are sampled
with nvidia-smi DURING the timed region.  Multi-GPU: after the host barrier every rank enqueues TWO untimed steps
before the start event -- each step ends with an all-to-all, so the ranks leave it together and the host-side
start skew of the barrier (hundreds of microseconds, i.e. several steps) is absorbed on the device instead of
being charged to a K = 20 timed region.  Both arms, and the NCCL-structured comparator, use the same loop.

Extra blocks of the JSON line (they explain the headline; the driver reads value / e2e):
``vs_minfix`` (N > 1): the runnable "reference's own NCCL build" -- baseline/nccl_minfix.py, the reference's structure
with its four documented defects fixed -- same steps / warm-up / KV rotation, with clocks, and own / minfix.
``baseline_configs`` (N = 8, or --heavy on): the other BASELINE.json configs -- full-Sq 128K forward, 256K block-scaled
fp8 decode on tcgen05, 1M GQA forward+backward -- each with latency, roofline fraction and clocks.
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

L2_BYTES = 126 << 20


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=4000)
    p.add_argument("--warmup", type=int, default=50)
    p.add_argument("--impl", default="own", choices=["own", "reference"])
    p.add_argument("--seq", type=int, default=131072, help="GLOBAL KV sequence length")
    p.add_argument("--heads", type=int, default=32)
    p.add_argument("--kv-heads", type=int, default=None)
    p.add_argument("--head-dim", type=int, default=128)
    p.add_argument("--batch", type=int, default=1)
    p.add_argument("--dtype", default="bf16")
    p.add_argument("--backend", default="fused")
    p.add_argument("--no-extras", action="store_true", help="skip the NCCL-comparator / full-forward extras")
    p.add_argument("--graph", action=argparse.BooleanOptionalAction, default=True,
                   help="replay the step from a CUDA graph (launch-bound at 8 GPUs)")
    p.add_argument("--pdl", action=argparse.BooleanOptionalAction, default=True,
                   help="device-timed loop: prepared launches chained by programmatic dependent launch (the e2e loop, which "
                        "synchronises every step, replays the CUDA graph)")
    p.add_argument("--heavy", default="auto", choices=["auto", "on", "off"],
                   help="also measure the other BASELINE.json configs (full-Sq 128K forward, 256K fp8, 1M GQA fwd+bwd); "
                        "auto = only on 8 GPUs")
    p.add_argument("--host-io", default="copy", choices=["zero_copy", "copy"],
                   help="e2e step: the kernel reads q / writes the result in pinned host memory itself (zero_copy), or a CUDA graph "
                        "[H2D memcpy | attention | D2H memcpy] (copy); the other variant is reported in e2e.other_transfer unless --no-extras")
    p.add_argument("--align", type=int, default=2, help="untimed steps enqueued between the host barrier and the start event")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write the result of the last timed step as DIR/<name>.npy (float32, at most "
                        "64 MiB in all: a larger result is replaced by a fixed, seeded sample of its elements)")
    return p.parse_args()


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi sampler (the profiling recipe's clocks line) running while the timed region executes."""

    FIELDS = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int, period_ms: int = 50):
        self.gpu_index = gpu_index
        self.rows = []
        self.proc = None
        self.t_start = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-i", str(gpu_index),
                 "-lms", str(period_ms)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0: float, t1: float) -> dict:
        sm, mx, reasons, power = [], [], set(), []
        for ts, line in self.rows:
            if ts < t0 or ts > t1 + 0.06:
                continue
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 10:
                continue
            try:
                sm.append(float(parts[2])); mx.append(float(parts[3])); power.append(float(parts[4]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[6:10]):
                if val.lower() == "active":
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power)}


# ------------------------------------------------------------------------------------------------
def emit(d: dict):
    print(json.dumps(d), flush=True)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict):
    """Write each tensor of ``arrays`` as float32 ``out_dir/<name>.npy``.  Inputs are seeded, so two builds run with the
    same arguments can be compared output for output.  Past 64 MiB in all, every array is flattened and replaced by the
    same share of its elements, drawn with a fixed seed (sorted indices, so the sample is identical from run to run)."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    total = sum(t.numel() for t in arrays.values())
    limit = DUMP_LIMIT_BYTES // 4
    for name, t in arrays.items():
        t = t.detach().float()
        if total > limit:
            keep = max(1, t.numel() * limit // total)
            idx = torch.randint(0, t.numel(), (keep,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.cpu().numpy())


def reexec_with_torchrun(args):
    port = 29500 + (os.getpid() % 2000)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
    os.execv(sys.executable, cmd)


def timed_loop(torch, dist, step_fn, steps, warmup, align, world, dev, barrier, sampler=None):
    """warm-up -> host barrier -> `align` untimed steps (device-side alignment of the ranks) -> [event | K steps | event]
    -> max over ranks.  Returns (ms total, (wall t0, wall t1))."""
    for i in range(warmup):
        step_fn(i)
    barrier()
    t0w = time.time()
    for i in range(align):
        step_fn(warmup + i)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step_fn(warmup + align + i)
    e1.record()
    torch.cuda.synchronize()
    t1w = time.time()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), (t0w, t1w)


def sampled_clocks(torch, dist, sampler, window, step_fn, ms_per_step, steps, world, dev, barrier):
    """Clock record of a timed region; when it was too short for nvidia-smi (50 ms period), an identical loop is run for
    ~1.5 s right after it and sampled instead (and the record says so)."""
    source = "nvidia-smi during the timed region"
    clocks = sampler.summary(*window) if sampler is not None else None
    need = torch.tensor([1 if (clocks is not None and clocks["samples"] < 3) else 0], device=dev)
    if world > 1:
        dist.broadcast(need, 0)
    if int(need.item()):
        reps = max(steps, int(1.5e3 / max(ms_per_step, 1e-3)))
        barrier()
        p0 = time.time()
        for i in range(reps):
            step_fn(i)
        torch.cuda.synchronize()
        p1 = time.time()
        if sampler is not None:
            clocks = sampler.summary(p0, p1)
            source = f"nvidia-smi during an identical {reps}-step loop run right after the timed region (too short to sample)"
    if clocks is not None:
        clocks["source"] = source
    return clocks


def main():
    args = parse_args()
    n = args.gpus
    if n > 1 and "RANK" not in os.environ:
        reexec_with_torchrun(args)
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", str(rank)))
    if not torch.cuda.is_available():
        if rank == 0:
            emit({"impl": args.impl, "unavailable": "no CUDA device visible"} if args.impl == "reference" else
                 {"metric": "attention fwd tokens/sec", "value": None, "error": "no CUDA device visible"})
        return 0
    if world != n:
        n = world
    dtype = {"bf16": torch.bfloat16, "fp16": torch.float16}[args.dtype]
    steps, warmup = max(1, args.steps), max(3, args.warmup)

    import tree_attention_b200 as ta
    from tree_attention_b200.ops import reference as ref

    ta.setup(rank, world, local_rank=local_rank)
    dev = torch.device("cuda", torch.cuda.current_device())
    B, Hq, D, S = args.batch, args.heads, args.head_dim, args.seq
    Hkv = args.kv_heads or Hq
    assert S % world == 0
    s_local = S // world
    scale = D ** -0.5
    kv_bytes_rank = 2 * B * Hkv * s_local * D * 2
    nbuf = max(1, -(-4 * L2_BYTES // kv_bytes_rank))  # working set > 4 x L2
    nbuf = min(nbuf, 8)
    gq = torch.Generator(device=dev).manual_seed(1234)
    q = torch.randn(B, Hq, 1, D, device=dev, generator=gq).to(dtype)  # same seed on every rank: replicated Q
    kvs = []
    for i in range(nbuf):
        _, k, v = ta.make_data((B, Hq, s_local, D), rank, dev, dtype=dtype, num_kv_heads=Hkv, seed=100 + i, log=False)
        kvs.append((k, v))
    config = {
        "model": "tree-attention decode forward (Sq=1), KV sharded over GPUs", "global_batch": B, "seq_len": S,
        "heads": Hq, "kv_heads": Hkv, "head_dim": D, "kv_tokens_per_rank": s_local,
        "parallelism": f"sp{world}" if world > 1 else "single",
        "l2": f"inputs larger than L2: {nbuf} KV buffer(s) x {kv_bytes_rank / 2**20:.0f} MiB/rank rotated per step "
              f"(> 4 x 126 MiB L2), no flush",
    }
    metric = "attention fwd tokens/sec (decode step Sq=1: KV tokens attended per second, whole box, device-timed, max over ranks) at seq=128K"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # --------------------------------------------------------------------------------------------
    if args.impl == "reference":
        ref_path = os.path.join(ROOT, "baseline", "_ref", "model.py")
        if not os.path.exists(ref_path):
            if rank == 0:
                emit({"impl": "reference", "unavailable": "baseline/_ref/model.py missing (run baseline/install_ref.sh)"})
            ta.cleanup()
            return 0
        spec = importlib.util.spec_from_file_location("ref_model", ref_path)
        rm = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(rm)
        try:
            rm.logger.remove()  # keep its per-call log lines off the terminal; the calls themselves still run
        except Exception:
            pass
        # The reference's own public API: tree_decode(q, k, v, rank, world_size, device) on the layout its
        # flash_res_lse documents (B, nh, 1, C) / (B, nh, T, C) (model.py:65-67).  Stock code path, default
        # softmax_scale=1.0 (model.py:60,100).
        last = {}

        def ref_step(i):
            k, v = kvs[i % nbuf]
            last["out"] = rm.tree_decode(q, k, v, rank, world, dev)
            return last["out"]
        try:
            for i in range(warmup):
                ref_step(i)
            torch.cuda.synchronize()
        except Exception as e:  # world_size > 1: RuntimeError at model.py:111, always (SURVEY.md D3)
            msg = f"unmodified reference tree_decode raises at world_size={world}: {type(e).__name__}: {str(e)[:160]}"
            if rank == 0:
                emit({"impl": "reference", "unavailable": msg, "n_gpus": world})
            ta.cleanup()
            return 0
        sampler = ClockSampler(local_rank) if rank == 0 else None
        ms, window = timed_loop(torch, dist, ref_step, steps, 0, args.align, world, dev, barrier)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, last)
        # e2e: pinned q -> device, step, result -> pinned host, every step
        qh = q.cpu().pin_memory()
        oh = torch.empty((B, Hq, 1, D), dtype=dtype).pin_memory()
        qd = torch.empty_like(q)
        barrier()
        te0 = time.perf_counter()
        for i in range(steps):
            qd.copy_(qh, non_blocking=True)
            k, v = kvs[i % nbuf]
            o = rm.tree_decode(qd, k, v, rank, world, dev)
            oh.copy_(o, non_blocking=True)
            torch.cuda.synchronize()
        te1 = time.perf_counter()
        e2e_ms = (te1 - te0) * 1e3
        clocks = sampled_clocks(torch, dist, sampler, window, ref_step, ms / steps, steps, world, dev, barrier)
        if sampler is not None:
            sampler.stop()
        if rank == 0:
            lat = ms / steps
            emit({"impl": "reference", "metric": metric, "value": B * S / (lat * 1e-3), "unit": "tokens/s",
                  "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": lat, "higher_is_better": True,
                  "scaling": "strong", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
                  "config": config, "clocks": clocks, "decode_tokens_per_s": B / (lat * 1e-3),
                  "e2e": {"value": B * S / (e2e_ms / steps * 1e-3), "unit": "tokens/s",
                          "h2d_bytes_per_step": qh.numel() * qh.element_size(),
                          "d2h_bytes_per_step": oh.numel() * oh.element_size()},
                  "gpu_launches": 0,
                  "note": "unmodified /root/reference model.py tree_decode (local branch; stock torch ops; softmax_scale=1.0)"})
        ta.cleanup()
        return 0

    # --------------------------------------------------------------------------------------------
    # own arm
    from tree_attention_b200 import _build

    C = _build.load()
    from tree_attention_b200.models.decoder import TreeDecodeSession

    sess = TreeDecodeSession(kvs, softmax_scale=scale, backend=args.backend, use_graph=args.graph, pdl=args.pdl,
                             host_io=args.host_io)

    # correctness gate before timing (never time a wrong kernel)
    out = sess.step_device(q, 0)
    launches_per_step = sess.launches_per_step
    o_p, l_p = ref.attention_partial_ref(q, kvs[0][0], kvs[0][1], scale, False, 0, 0, torch.float32, block=16384)
    if world > 1:
        packed = torch.cat([o_p, l_p[..., None]], -1).contiguous()
        bufs = [torch.empty_like(packed) for _ in range(world)]
        dist.all_gather(bufs, packed)
        o_ref, _ = ref.merge_many([b[..., :-1] for b in bufs], [b[..., -1] for b in bufs])
    else:
        o_ref = o_p
    err = float((out.float() - o_ref).abs().max())
    if not err < 2e-2:
        if rank == 0:
            emit({"metric": metric, "value": None, "error": f"output mismatch vs oracle: {err}"})
        ta.cleanup()
        return 1

    sess.q_static.copy_(q)
    # this box's copy bandwidth, measured like MEASURED_PEAKS.json (b.copy_(a), read + write bytes, best of 10): boxes of the
    # pool differ by several percent, so every roofline fraction below is also given against THIS box
    box_copy_gbs = None
    try:
        ca = torch.empty(1 << 29, dtype=torch.bfloat16, device=dev)
        cb = torch.empty_like(ca)
        best = 1e9
        for _ in range(10):
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record(); cb.copy_(ca); c1.record()
            torch.cuda.synchronize()
            best = min(best, c0.elapsed_time(c1))
        box_copy_gbs = 2 * ca.numel() * 2 / (best * 1e-3) / 1e9
        del ca, cb
        torch.cuda.empty_cache()
    except Exception:
        pass
    sampler = ClockSampler(local_rank) if rank == 0 else None
    own_step = lambda i: sess.step_device(None, i)
    ms, window = timed_loop(torch, dist, own_step, steps, warmup, args.align, world, dev, barrier)
    if args.dump_outputs and rank == 0:
        # the last timed step ran KV buffer (warmup + align + steps - 1) % nbuf; its result stays in the session's output
        # buffer for that buffer until the end-to-end loop below runs it again.  The combined output is the same on every rank.
        dump_outputs(args.dump_outputs, {"out": sess.out_static[(warmup + args.align + steps - 1) % nbuf]})

    # end-to-end through the public API: pinned host q -> device, step, result -> pinned host, every step.  Measured right
    # after the device-timed region and BEFORE the seconds-long clock-sampling loop below, i.e. in the same thermal / power
    # state as the device-timed number (the reference arm uses the same order)
    def run_e2e(session):
        r = session.run_e2e(q, steps, barrier)
        t = torch.tensor([r["ms"]], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        # what the host receives from that path, against the fp32 oracle (never report a wrong step's time)
        r["err"] = None
        if session.q_host is not None and session.out_host[0] is not None:
            session.out_host[0].zero_()
            session.step(session.q_host, session.out_host[0], 0)      # one more (untimed) step on buffer 0, checked
            r["err"] = float((session.out_host[0].float().to(dev) - o_ref0).abs().max())
        return r, float(t.item()) / steps

    o_ref0 = o_ref
    e2e, e2e_lat = run_e2e(sess)
    clocks = sampled_clocks(torch, dist, sampler, window, own_step, ms / steps, steps, world, dev, barrier)

    # ---- the contract line is complete at this point; everything below only ADDS explanatory keys to it.  A watchdog
    # guarantees the line: if an extra (second e2e variant, NCCL comparator, the heavy BASELINE configs at 8 GPUs) wedges
    # or overruns its budget, rank 0 prints the line with what has been collected so far and every rank exits.
    lat = ms / steps
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = peaks.get("hbm_gbs", 6650.0)
    gbs = kv_bytes_rank / (lat * 1e-3) / 1e9
    extras = {}
    e2e_blk = {"value": B * S / (e2e_lat * 1e-3), "unit": "tokens/s", "ms_per_step": e2e_lat,
               "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": e2e["d2h"], "transfer": e2e["transfer"],
               "max_abs_err_vs_oracle": e2e["err"], "other_transfer": None,
               "per_step_ms_rank0": {"median": e2e["median_ms"], "min": e2e["min_ms"], "max": e2e["max_ms"]}}

    def main_line():
        return {
            "metric": metric, "value": B * S / (lat * 1e-3), "unit": "tokens/s", "n_gpus": world, "steps": steps,
            "warmup": warmup, "ms_per_step": lat, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": args.dtype, "data": "synthetic", "config": config, "clocks": clocks,
            "timing": f"CUDA events around {steps} steps after {warmup} warm-ups; {args.align} untimed step(s) between the host barrier "
                      "and the start event align the ranks on the device (every step ends with an all-to-all); max over ranks",
            "e2e": e2e_blk,
            "gpu_launches": launches_per_step * steps,
            "decode_tokens_per_s": B / (lat * 1e-3),
            "hbm_gbs_per_gpu": gbs, "hbm_frac_of_measured": gbs / hbm,
            "box_copy_gbs_rank0": box_copy_gbs, "hbm_frac_of_this_box_copy": (gbs / box_copy_gbs) if box_copy_gbs else None,
            "max_abs_err_vs_oracle": err, "backend": args.backend, "cuda_graph": bool(sess.graphs), "pdl": bool(args.pdl),
            "launch_path": "prepared C++ launch (_C.DecodeStep), one cudaLaunchKernelEx per step" if getattr(sess, "_steps", None) else "python",
            **extras,
        }

    import threading

    emitted = threading.Lock()
    extras_budget_s = float(os.environ.get("TREE_ATTN_BENCH_EXTRAS_BUDGET_S", "240"))

    def watchdog_fire():
        if not emitted.acquire(blocking=False):
            return
        if rank == 0:
            line = main_line()
            line["extras_watchdog"] = f"extras exceeded {extras_budget_s:.0f} s and were cut off; the contract keys were complete before them"
            emit(line)
        os._exit(0)

    watchdog = threading.Timer(extras_budget_s, watchdog_fire)
    watchdog.daemon = True
    if not args.no_extras:
        watchdog.start()

    if not args.no_extras:
        # the other host-I/O variant of the same end-to-end step, same loop, for the record
        try:
            other = "copy" if args.host_io == "zero_copy" else "zero_copy"
            sess2 = TreeDecodeSession(kvs, softmax_scale=scale, backend=args.backend, use_graph=args.graph, pdl=args.pdl, host_io=other)
            sess2.step_device(q, 0)
            r2, lat2 = run_e2e(sess2)
            e2e_blk["other_transfer"] = {"transfer": r2["transfer"], "ms_per_step": lat2, "value": B * S / (lat2 * 1e-3),
                                         "per_step_ms_rank0": {"median": r2["median_ms"], "min": r2["min_ms"], "max": r2["max_ms"]},
                                         "note": "measured after the primary variant (second-measured runs ~5 us faster either way round)"}
            sess2.close()
        except Exception as e:
            e2e_blk["other_transfer"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    if world > 1 and not args.no_extras:
        # the runnable "reference's own NCCL build" on the same box, same loop, with its own clock record
        try:
            sys.path.insert(0, os.path.join(ROOT, "baseline"))
            import nccl_minfix

            mf_step = lambda i: nccl_minfix.tree_decode_minfix(q, kvs[i % nbuf][0], kvs[i % nbuf][1], scale)
            mf_ms, mf_window = timed_loop(torch, dist, mf_step, steps, warmup, args.align, world, dev, barrier)
            mf_clocks = sampled_clocks(torch, dist, sampler, mf_window, mf_step, mf_ms / steps, steps, world, dev, barrier)
            mf_lat = mf_ms / steps
            extras["vs_minfix"] = {
                "impl": "baseline/nccl_minfix.py: the reference's structure (stock torch matmul/softmax + all_reduce MAX, SUM, SUM "
                        "on NCCL) with its four documented defects fixed; the verbatim reference raises at model.py:111 for N > 1",
                "ms_per_step": mf_lat, "value": B * S / (mf_lat * 1e-3), "unit": "tokens/s", "steps": steps, "warmup": warmup,
                "own_ms_per_step": ms / steps, "ratio_own_over_minfix": mf_lat / (ms / steps), "clocks": mf_clocks,
            }
        except Exception as e:
            extras["vs_minfix"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    if sampler is not None:
        sampler.stop()
    if not args.no_extras:
        extras.update(run_extras(args, ta, sess, q, kvs, scale, world, rank, dev, barrier))
        heavy = args.heavy == "on" or (args.heavy == "auto" and world == 8)
        if heavy:
            try:
                from bench_tools import configs as heavy_configs

                extras["baseline_configs"] = heavy_configs.run_all(ta, world, rank, dev, barrier, ROOT)
            except Exception as e:
                extras["baseline_configs"] = {"error": f"{type(e).__name__}: {e}"[:200]}

    watchdog.cancel()
    if not emitted.acquire(blocking=False):     # the watchdog is printing / has printed the line
        time.sleep(3600)
    if rank == 0:
        emit(main_line())
    # teardown must not be able to take the (already printed) line down with it: if an extra failed, a peer or the CUDA context
    # may be in a bad state and the collective barrier inside cleanup() could raise or wait forever -- leave without it
    def _has_error(v, depth=0):
        return isinstance(v, dict) and ("error" in v or (depth < 2 and any(_has_error(x, depth + 1) for x in v.values())))

    failed = [k for k, v in extras.items() if _has_error(v)]
    if failed:
        print(f"[bench] extras {failed} failed; skipping the collective teardown", file=sys.stderr)
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    bail = threading.Timer(45.0, lambda: os._exit(0))     # a peer that already left would make the teardown barrier wait forever
    bail.daemon = True
    bail.start()
    ta.cleanup()
    bail.cancel()
    return 0


def run_extras(args, ta, sess, q, kvs, scale, world, rank, dev, barrier):
    """Numbers that explain the headline: un-graphed launch path, NCCL-structured comparator."""
    import torch
    import torch.distributed as dist

    out = {}
    nb = len(kvs)

    def timeit(fn, steps=50, warmup=5):
        for i in range(warmup):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1) / steps], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    try:
        if sess.graphs:
            out["graph_replay_ms_per_step"] = timeit(lambda i: sess.graphs[i % nb].replay(), steps=200)
        out["python_api_launch_ms_per_step"] = timeit(
            lambda i: ta.tree_attention(q, kvs[i % nb][0], kvs[i % nb][1], softmax_scale=scale, backend=args.backend))
        if world > 1:
            out["own_kernel_plus_nccl_allreduce3_ms_per_step"] = timeit(
                lambda i: ta.tree_attention(q, kvs[i % nb][0], kvs[i % nb][1], softmax_scale=scale, backend="nccl",
                                            schedule="allreduce3"))
        # block-scaled fp8 (MX) KV cache: same decode step on e4m3 + UE8M0 KV (BASELINE.json fp8 config)
        from tree_attention_b200.ops.quant import MXFP8Tensor

        kq, vq = MXFP8Tensor.from_float(kvs[0][0]), MXFP8Tensor.from_float(kvs[0][1])
        o8 = ta.tree_attention(q, kq, vq, softmax_scale=scale, backend=args.backend)
        o16 = ta.tree_attention(q, kvs[0][0], kvs[0][1], softmax_scale=scale, backend=args.backend)
        out["mxfp8_kv_max_abs_diff_vs_bf16"] = float((o8.float() - o16.float()).abs().max())
        out["mxfp8_kv_eager_ms_per_step"] = timeit(
            lambda i: ta.tree_attention(q, kq, vq, softmax_scale=scale, backend=args.backend), steps=200)
        if q.shape[-1] == 128 and (q.shape[1] // kvs[0][0].shape[1]) * q.shape[2] <= 16:
            # the same MX cache with V blocked along the keys: both GEMMs on tcgen05.mma.kind::mxf8f6f4.block_scale
            from tree_attention_b200.ops.quant import FP8ChannelTensor, MXFP8SeqTensor

            vs = MXFP8SeqTensor.from_float(kvs[0][1])
            o8t = ta.tree_attention(q, kq, vs, softmax_scale=scale, backend=args.backend)
            out["mxfp8_block_scaled_tcgen05_max_abs_diff_vs_bf16"] = float((o8t.float() - o16.float()).abs().max())
            out["mxfp8_block_scaled_tcgen05_eager_ms_per_step"] = timeit(
                lambda i: ta.tree_attention(q, kq, vs, softmax_scale=scale, backend=args.backend), steps=200)
            kc, vc = FP8ChannelTensor.from_float(kvs[0][0]), FP8ChannelTensor.from_float(kvs[0][1])
            out["fp8_per_channel_tcgen05_eager_ms_per_step"] = timeit(
                lambda i: ta.tree_attention(q, kc, vc, softmax_scale=scale, backend=args.backend), steps=200)
            del vs, kc, vc
        del kq, vq
        reg = getattr(sess, "region", None)
        if world > 1 and reg is not None:
            reg.combine_stamps(reset=True)
            for i in range(200):
                sess.step_device(None, i)
            torch.cuda.synchronize()
            st = reg.combine_stamps(reset=True)
            B_, Hq_, D_ = q.shape[0], q.shape[1], q.shape[3]
            recv = (world - 1) * B_ * Hq_ * (D_ + 1) * 8
            out["combine_step"] = {
                **st, "bytes_received_per_rank": recv,
                "nvlink_gbs_per_combine_step": recv / max(st["combine_step_ns"], 1),
                "note": "in-kernel globaltimer stamps, max over CTAs and 200 steps: publish -> merged output written; "
                        "payload = (W-1) x heads x (D+1) tagged 8-byte words per rank",
            }
    except Exception as e:  # extras must never take the headline down
        out["extras_error"] = f"{type(e).__name__}: {e}"[:200]
    return out


if __name__ == "__main__":
    sys.exit(main())
