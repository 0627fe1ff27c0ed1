"""Multi-GPU: fused in-kernel tree combine over symmetric memory vs the NCCL path vs the oracle.
Needs >= 2 GPUs (skipped otherwise)."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

from _dist_utils import run_distributed

NGPU = torch.cuda.device_count() if torch.cuda.is_available() else 0
need2 = pytest.mark.skipif(NGPU < 2, reason="needs >= 2 GPUs")
WORLDS = [w for w in (2, 4, 8) if w <= NGPU]
if os.environ.get("TREE_ATTN_TEST_WORLDS"):
    WORLDS = [int(w) for w in os.environ["TREE_ATTN_TEST_WORLDS"].split(",") if int(w) <= NGPU]


def _oracle(q, k, v, world, scale, causal):
    import torch.distributed as dist
    from tree_attention_b200.ops import reference as ref

    ks = [torch.empty_like(k) for _ in range(world)]
    vs = [torch.empty_like(v) for _ in range(world)]
    dist.all_gather(ks, k.contiguous())
    dist.all_gather(vs, v.contiguous())
    return ref.attention_partial_ref(q, torch.cat(ks, 2), torch.cat(vs, 2), scale, causal,
                                     world * k.shape[2] - q.shape[2], 0, torch.float32, block=16384)


def _worker_fused(rank, world):
    import torch.distributed as dist
    import tree_attention_b200 as ta

    dev = torch.device("cuda", rank)
    for (b, hq, hkv, sq, s, d, dtype, causal) in [
        (1, 32, 32, 1, 4096, 128, torch.bfloat16, False),
        (2, 8, 2, 1, 1500, 128, torch.bfloat16, True),
        (1, 16, 16, 1, 64000 // 8, 128, torch.float16, False),
        (1, 8, 4, 3, 999, 64, torch.bfloat16, True),
    ]:
        q, k, v = ta.make_data((b, hq, s, d), rank, dev, dtype=dtype, sq=sq, num_kv_heads=hkv, log=False)
        scale = d ** -0.5
        o_ref, l_ref = _oracle(q, k, v, world, scale, causal)
        results = {}
        for backend, sched in [("fused", "oneshot"), ("symm", "oneshot"), ("symm", "butterfly"),
                               ("nccl", "allreduce3"), ("nccl", "allgather"), ("nccl", "butterfly")]:
            out, lse = ta.tree_attention(q, k, v, causal=causal, return_lse=True, backend=backend, schedule=sched)
            torch.cuda.synchronize()
            err = (out.float() - o_ref).abs().max().item()
            assert err < 2e-2, (backend, sched, err)
            assert (lse - l_ref).abs().max().item() < 3e-3, (backend, sched)
            results[(backend, sched)] = out
            if backend in ("fused", "symm"):
                outs = [torch.empty_like(out) for _ in range(world)]
                dist.all_gather(outs, out.contiguous())
                for o in outs:
                    assert torch.equal(o, outs[0]), f"{backend}/{sched}: ranks disagree bitwise"
    # per-channel fp8 KV cache through the fused tcgen05 decode kernels (swap-AB for <= 16 rows, packed rows above)
    from tree_attention_b200.ops.quant import FP8ChannelTensor

    for (b, hq, hkv, sq, s) in [(1, 8, 8, 1, 2048), (2, 8, 2, 2, 1111), (1, 32, 1, 1, 777)]:
        q, k, v = ta.make_data((b, hq, s, 128), rank, dev, dtype=torch.bfloat16, sq=sq, num_kv_heads=hkv, log=False)
        k8, v8 = FP8ChannelTensor.from_float(k), FP8ChannelTensor.from_float(v)
        o_ref, l_ref = _oracle(q, k8.dequantize(torch.bfloat16), v8.dequantize(torch.bfloat16), world, 128 ** -0.5, False)
        out, lse = ta.tree_attention(q, k8, v8, return_lse=True)
        torch.cuda.synchronize()
        assert (out.float() - o_ref).abs().max().item() < 6e-2, (hq, hkv, sq)
        assert (lse - l_ref).abs().max().item() < 6e-2, (hq, hkv, sq)
        outs = [torch.empty_like(out) for _ in range(world)]
        dist.all_gather(outs, out.contiguous())
        for o in outs:
            assert torch.equal(o, outs[0]), "fp8 fused decode: ranks disagree bitwise"
    # block-scaled (MX) fp8 KV on the tensor cores, fused combine
    from tree_attention_b200.ops.quant import MXFP8SeqTensor, MXFP8Tensor

    for (b, hq, hkv, sq, s) in [(1, 8, 8, 1, 2048), (2, 8, 2, 2, 1111)]:
        q, k, v = ta.make_data((b, hq, s, 128), rank, dev, dtype=torch.bfloat16, sq=sq, num_kv_heads=hkv, log=False)
        kq, vq = MXFP8Tensor.from_float(k), MXFP8SeqTensor.from_float(v)
        o_ref, l_ref = _oracle(q, kq.dequantize(torch.bfloat16), vq.dequantize(torch.bfloat16), world, 128 ** -0.5, False)
        out, lse = ta.tree_attention(q, kq, vq, return_lse=True)
        torch.cuda.synchronize()
        assert (out.float() - o_ref).abs().max().item() < 6e-2, (hq, hkv, sq)
        assert (lse - l_ref).abs().max().item() < 6e-2, (hq, hkv, sq)
        outs = [torch.empty_like(out) for _ in range(world)]
        dist.all_gather(outs, out.contiguous())
        for o in outs:
            assert torch.equal(o, outs[0]), "mx fused decode: ranks disagree bitwise"


@need2
@pytest.mark.parametrize("world", WORLDS)
def test_fused_tree_attention(world, port):
    run_distributed(_worker_fused, world, port, cuda=True)


def _worker_prefill(rank, world):
    """tcgen05 forward with the fused in-kernel combine (compute + merge CTAs in one launch)."""
    import torch.distributed as dist
    import tree_attention_b200 as ta

    dev = torch.device("cuda", rank)
    for (b, hq, hkv, sq, s, d, dtype, causal) in [
        (1, 4, 4, 256, 512, 128, torch.bfloat16, False),
        (2, 8, 2, 300, 777, 128, torch.bfloat16, True),      # ragged, GQA, some (tile, rank) pairs fully masked
        (1, 4, 4, 1024, 1024, 64, torch.float16, True),
        (1, 32, 8, 2048, 2048, 128, torch.bfloat16, True),   # many more items than SMs: merge CTAs interleave
    ]:
        q, k, v = ta.make_data((b, hq, s, d), rank, dev, dtype=dtype, sq=sq, num_kv_heads=hkv, log=False)
        scale = d ** -0.5
        o_ref, l_ref = _oracle(q, k, v, world, scale, causal)
        for backend in ("fused", "symm", "nccl"):
            out, lse = ta.tree_attention(q, k, v, causal=causal, return_lse=True, backend=backend,
                                         schedule="allgather" if backend == "nccl" else "oneshot")
            torch.cuda.synchronize()
            err = (out.float() - o_ref).abs().max().item()
            assert err < 3e-2, (backend, err)
            dead = torch.isinf(l_ref)
            assert (lse[~dead] - l_ref[~dead]).abs().max().item() < 5e-3, backend
            if backend == "fused":
                outs = [torch.empty_like(out) for _ in range(world)]
                dist.all_gather(outs, out.contiguous())
                for o in outs:
                    assert torch.equal(o, outs[0]), "fused prefill: ranks disagree bitwise"
                # Sq-sharded output: the reduce-scatter half only -- this rank's rows, bitwise the replicated result
                o_sh, l_sh = ta.tree_attention(q, k, v, causal=causal, return_lse=True, backend="fused", output="sharded")
                torch.cuda.synchronize()
                n = ((sq + 127) // 128 + world - 1) // world * 128
                assert o_sh.shape == (b, hq, n, d) and l_sh.shape == (b, hq, n)
                lo, hi = min(rank * n, sq), min((rank + 1) * n, sq)
                assert torch.equal(o_sh[:, :, : hi - lo], out[:, :, lo:hi]), "sharded rows differ from the replicated result"
                assert torch.equal(l_sh[:, :, : hi - lo], lse[:, :, lo:hi])
    # repeated launches: slot / epoch reuse of both modes, interleaved
    for it in range(50):
        out = ta.tree_attention(q, k, v, causal=True, backend="fused")
        if it % 5 == 0:
            o_sh = ta.tree_attention(q, k, v, causal=True, backend="fused", output="sharded")
    torch.cuda.synchronize()
    assert (out.float() - o_ref).abs().max().item() < 3e-2
    assert torch.equal(o_sh[:, :, : hi - lo], out[:, :, lo:hi])
    # a long query block in chunks (symmetric buffer capped): same result
    import os
    os.environ["TREE_ATTN_FWD_SYMM_CAP_GB"] = "0.004"
    out_c = ta.tree_attention(q, k, v, causal=True, backend="fused")
    torch.cuda.synchronize()
    del os.environ["TREE_ATTN_FWD_SYMM_CAP_GB"]
    assert torch.equal(out_c, out), "chunked fused prefill differs"


@need2
@pytest.mark.parametrize("world", WORLDS)
def test_fused_prefill_tcgen05(world, port):
    run_distributed(_worker_prefill, world, port, cuda=True)


def _worker_zigzag(rank, world):
    """kv_layout="zigzag" on GPUs: every rank owns chunks r and 2W-1-r of a causal sequence.  The fused backend runs ONE
    tcgen05 launch over the two-segment shard (combine included); symm / nccl merge per-rank partials; all equal plain
    causal attention over the whole sequence, forward and backward."""
    import torch.distributed as dist
    import tree_attention_b200 as ta
    from tree_attention_b200.ops import reference as ref
    from tree_attention_b200.ops.autograd import tree_attention_func

    dev = torch.device("cuda", rank)
    for (hq, hkv, S, d, dtype) in [(4, 4, 256 * 2 * world, 128, torch.bfloat16), (8, 2, 128 * 2 * world, 64, torch.float16),
                                   (4, 2, 200 * 2 * world, 128, torch.bfloat16)]:   # last: chunks not tile-aligned -> two partials
        g = torch.Generator(device=dev).manual_seed(5)
        q = torch.randn(1, hq, S, d, device=dev, generator=g).to(dtype)
        k_full = torch.randn(1, hkv, S, d, device=dev, generator=g).to(dtype)
        v_full = torch.randn(1, hkv, S, d, device=dev, generator=g).to(dtype)
        k, v = ta.zigzag_shard(k_full, rank, world).contiguous(), ta.zigzag_shard(v_full, rank, world).contiguous()
        o_ref, l_ref = ref.attention_partial_ref(q, k_full, v_full, d ** -0.5, True, 0, 0, torch.float32)
        for backend in ("fused", "symm", "nccl"):
            out, lse = ta.tree_attention(q, k, v, causal=True, return_lse=True, backend=backend, kv_layout="zigzag",
                                         schedule="allgather" if backend == "nccl" else "oneshot")
            torch.cuda.synchronize()
            err = (out.float() - o_ref).abs().max().item()
            assert err < 3e-2, (backend, S, err)
            assert (lse - l_ref).abs().max().item() < 5e-3, backend
        out = ta.tree_attention(q, k, v, causal=True, backend="fused", kv_layout="zigzag")
        o_sh = ta.tree_attention(q, k, v, causal=True, backend="fused", kv_layout="zigzag", output="sharded")
        torch.cuda.synchronize()
        n = o_sh.shape[2]
        lo, hi = min(rank * n, S), min((rank + 1) * n, S)
        assert (o_sh[:, :, : hi - lo].float() - out[:, :, lo:hi].float()).abs().max().item() < 1e-2
        # the contiguous interpretation of the same shards is a different (wrong) sequence order
        o_c = ta.tree_attention(q, k, v, causal=True, backend="fused")
        assert (o_c.float() - o_ref).abs().max().item() > 1e-2
    # backward through the zigzag layout (tcgen05 backward per segment, dQ reduced over symmetric memory)
    qg = q.clone().requires_grad_(True)
    kg, vg = k.clone().requires_grad_(True), v.clone().requires_grad_(True)
    do = torch.randn(q.shape, device=dev, generator=g).to(dtype)
    tree_attention_func(qg, kg, vg, causal=True, kv_layout="zigzag").backward(do)
    qo, ko, vo = (t.float().clone().requires_grad_(True) for t in (q, k_full, v_full))
    ref.attention_partial_ref(qo, ko, vo, d ** -0.5, True, 0, 0, torch.float32)[0].backward(do.float())
    torch.cuda.synchronize()
    for got, exp, name in ((qg.grad, qo.grad, "dq"), (kg.grad, ta.zigzag_shard(ko.grad, rank, world), "dk"),
                           (vg.grad, ta.zigzag_shard(vo.grad, rank, world), "dv")):
        rel = (got.float() - exp).abs().max().item() / max(exp.abs().max().item(), 1e-6)
        assert rel < 3e-2, (name, rel)


@need2
@pytest.mark.parametrize("world", WORLDS)
def test_zigzag_causal_prefill(world, port):
    run_distributed(_worker_zigzag, world, port, cuda=True)


def _worker_stress(rank, world):
    """>= 1000 back-to-back fused steps: epoch/parity reuse must never serve stale partials."""
    import tree_attention_b200 as ta
    from tree_attention_b200.parallel import symm

    dev = torch.device("cuda", rank)
    q, k, v = ta.make_data((1, 8, 2048, 128), rank, dev, dtype=torch.bfloat16, log=False)
    o_ref, _ = _oracle(q, k, v, world, 0.088, False)
    import torch.distributed as dist

    qs = [torch.randn_like(q) for _ in range(4)]
    for t in qs:  # Q is replicated: every rank must attend with the same query
        dist.broadcast(t, 0)
    refs = [_oracle(qq, k, v, world, 0.088, False)[0] for qq in qs]
    for it in range(1200):
        out = ta.tree_attention(qs[it % 4], k, v, softmax_scale=0.088, backend="fused")
        if it % 97 == 0 or it > 1190:
            assert (out.float() - refs[it % 4]).abs().max().item() < 2e-2, it
    torch.cuda.synchronize()
    reg = symm.regions()[("decode", 0)]
    reg.check()
    assert reg.epoch() >= 1200


@need2
def test_epoch_reuse_stress(port):
    run_distributed(_worker_stress, 2, port, cuda=True)


def _worker_graph(rank, world):
    import tree_attention_b200 as ta

    dev = torch.device("cuda", rank)
    q, k, v = ta.make_data((1, 8, 4096, 128), rank, dev, dtype=torch.bfloat16, log=False)
    ta.tree_attention(q, k, v, backend="fused")  # allocate workspaces + symmetric region
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g):
            out = ta.tree_attention(q, k, v, backend="fused")
    for i in range(5):
        q.copy_(torch.randn_like(q))
        import torch.distributed as dist
        dist.broadcast(q, 0)
        g.replay()
        torch.cuda.synchronize()
        o_ref, _ = _oracle(q, k, v, world, 128 ** -0.5, False)
        assert (out.float() - o_ref).abs().max().item() < 2e-2, i


@need2
def test_fused_cuda_graph_replay(port):
    run_distributed(_worker_graph, 2, port, cuda=True)


def _worker_fault(rank, world):
    """Fault injection: rank 1 never publishes -> rank 0's bounded spin reports it instead of hanging."""
    import tree_attention_b200 as ta
    from tree_attention_b200.parallel import symm

    dev = torch.device("cuda", rank)
    q, k, v = ta.make_data((1, 4, 1024, 128), rank, dev, dtype=torch.bfloat16, log=False)
    ta.tree_attention(q, k, v, backend="fused")
    torch.cuda.synchronize()
    reg = symm.regions()[("decode", 0)]
    reg.comm.timeout_s = 0.2
    if rank == 1:
        reg.comm.skip_publish = 1
    out = ta.tree_attention(q, k, v, backend="fused")
    torch.cuda.synchronize()
    with pytest.raises(RuntimeError, match="never arrived"):
        reg.check()
    assert torch.isnan(out.float()).any()  # a failed combine can never be consumed silently
    code, item, src, ep = reg.status()
    assert src == 1


@need2
def test_failure_detection_bounded_spin(port):
    run_distributed(_worker_fault, 2, port, cuda=True)


def _worker_reduce_and_bwd(rank, world):
    """Symmetric-memory all-reduce (the backward's dQ tree reduce) and the distributed fwd+bwd."""
    import torch.distributed as dist
    import tree_attention_b200 as ta
    from tree_attention_b200.ops import reference as ref
    from tree_attention_b200.ops.autograd import tree_attention_func
    from tree_attention_b200.parallel.tree import allreduce_sum

    dev = torch.device("cuda", rank)
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    for n in (4096, 4 * 1000, 3 * 4096 + 512, 1 << 22):
        x = torch.randn(n, device=dev, generator=g)
        y = allreduce_sum(x)
        exp = x.clone()
        dist.all_reduce(exp)
        assert torch.allclose(y, exp, atol=1e-4), n
        ys = [torch.empty_like(y) for _ in range(world)]
        dist.all_gather(ys, y)
        for t in ys:
            assert torch.equal(t, ys[0]), "all-reduce result differs across ranks"
    for _ in range(20):  # epoch / parity reuse
        y = allreduce_sum(x)
    assert torch.allclose(y, exp, atol=1e-4)

    # distributed forward + backward: dK/dV local, dQ summed over ranks by the symmetric-memory kernel
    b, hq, hkv, sq, s_local, d = 1, 8, 4, 256, 384, 128
    q, k, v = ta.make_data((b, hq, s_local, d), rank, dev, dtype=torch.bfloat16, sq=sq, num_kv_heads=hkv, log=False)
    do = torch.randn(b, hq, sq, d, device=dev, generator=torch.Generator(device=dev).manual_seed(7)).bfloat16()
    ks = [torch.empty_like(k) for _ in range(world)]
    vs = [torch.empty_like(v) for _ in range(world)]
    dist.all_gather(ks, k)
    dist.all_gather(vs, v)
    qf = q.float().requires_grad_(True)
    kf = torch.cat(ks, 2).float().requires_grad_(True)
    vf = torch.cat(vs, 2).float().requires_grad_(True)
    o_ref, _ = ref.attention_partial_ref(qf, kf, vf, None, True, world * s_local - sq, 0)
    o_ref.backward(do.float())
    ql, kl, vl = (t.clone().requires_grad_(True) for t in (q, k, v))
    o = tree_attention_func(ql, kl, vl, causal=True)
    o.backward(do)
    torch.cuda.synchronize()
    assert (o.float() - o_ref).abs().max().item() < 3e-2
    sl = slice(rank * s_local, (rank + 1) * s_local)
    for name, got, exp in (("dq", ql.grad, qf.grad), ("dk", kl.grad, kf.grad[:, :, sl]), ("dv", vl.grad, vf.grad[:, :, sl])):
        err = (got.float() - exp).abs().max().item() / (exp.abs().max().item() + 1e-6)
        assert err < 4e-2, (name, err)


@need2
def test_symm_allreduce_and_distributed_backward(port):
    run_distributed(_worker_reduce_and_bwd, min(NGPU, 4) if NGPU >= 4 else 2, port, cuda=True)


def _worker_fill_levels(rank, world):
    """Ragged, device-resident fill levels across ranks (one rank EMPTY), fused decode kernels + TreeDecodeSession on the
    native fast path: every rank must still publish (the identity for an empty shard) and the result must equal
    attention over the filled rows only; an append on one rank is picked up by the captured graphs."""
    import torch.distributed as dist
    import tree_attention_b200 as ta
    from tree_attention_b200.models.decoder import TreeDecodeSession
    from tree_attention_b200.ops import reference as ref

    dev = torch.device("cuda", rank)
    cap = 4096
    lens = [cap, 1000, 0, 77, 129, 4095, 1, 2048][:world]
    if world == 2:
        lens = [1000, 0]
    for hq, hkv in [(16, 16), (16, 4)]:        # CUDA-core streaming kernel / tcgen05 swap-AB kernel
        q, k, v = ta.make_data((1, hq, cap, 128), rank, dev, dtype=torch.bfloat16, num_kv_heads=hkv, log=False)
        n = lens[rank]
        k[:, :, n:] = 0
        v[:, :, n:] = 0
        sess = TreeDecodeSession([(k, v)], softmax_scale=0.088, q_shape=(1, hq, 1, 128), kv_lens=[n], backend="fused",
                                 host_io="zero_copy")

        def oracle():
            cur = torch.tensor([sess.kv_len_host[0]], device=dev)
            all_lens = [torch.empty_like(cur) for _ in range(world)]
            dist.all_gather(all_lens, cur)
            ks = [torch.empty_like(k) for _ in range(world)]
            vs = [torch.empty_like(v) for _ in range(world)]
            dist.all_gather(ks, k)
            dist.all_gather(vs, v)
            kf = torch.cat([ks[r][:, :, : int(all_lens[r])] for r in range(world)], 2)
            vf = torch.cat([vs[r][:, :, : int(all_lens[r])] for r in range(world)], 2)
            return ref.attention_partial_ref(q, kf, vf, 0.088, False, 0, 0, torch.float32)[0]

        out = sess.step_device(q, 0).clone()
        torch.cuda.synchronize()
        assert (out.float() - oracle()).abs().max().item() < 2e-2, (hq, hkv, "initial")
        g = torch.Generator(device=dev).manual_seed(100 + rank)
        for it in range(3):
            owner = (it + 1) % world
            if rank == owner and sess.kv_len_host[0] + 5 <= cap:
                k_new = torch.randn(1, hkv, 5, 128, device=dev, generator=g).bfloat16()
                v_new = torch.randn(1, hkv, 5, 128, device=dev, generator=g).bfloat16()
                sess.append_kv(0, k_new, v_new)
            out = sess.step_device(q, 0).clone()
            torch.cuda.synchronize()
            assert (out.float() - oracle()).abs().max().item() < 2e-2, (hq, hkv, it)
            outs = [torch.empty_like(out) for _ in range(world)]
            dist.all_gather(outs, out.contiguous())
            for o in outs:
                assert torch.equal(o, outs[0]), "fill levels: ranks disagree bitwise"
        # latency path: the fused kernel reads q from pinned host memory and posts the combined result into pinned host
        # memory (zero-copy twin of the prepared step: same workspace, region and launch-tag counters)
        qh = q.cpu().pin_memory()
        oh = torch.zeros(1, hq, 1, 128, dtype=torch.bfloat16).pin_memory()
        got = sess.step(qh, oh, 0).clone()
        assert sess._steps_zc, "the native session should take the zero-copy latency path"
        assert torch.equal(got.to(dev), outs[0]), (hq, hkv, "zero-copy step differs from the device-resident step")
        sess.region.check()
        sess.close()


@need2
@pytest.mark.parametrize("world", WORLDS)
def test_fused_decode_ragged_fill_levels(world, port):
    run_distributed(_worker_fill_levels, world, port, cuda=True)
