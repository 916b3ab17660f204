"""GPU tests (B200) of the two-kernel backward one ring hop per launch (``memory="ring"``).

On one device the W ranks are emulated (``ops.fused.emulate_ring_backward(fused=False, hopwise=True)``): the per-hop
launches must match the fp32 oracle, reproduce the one-launch (gather) backward bit for bit where the summation order
is the same (dQ always, dK / dV without grouped heads), and be deterministic.  With >= 2 GPUs a real ring runs both
memory modes on the same inputs."""
import pytest
import torch

pytestmark = pytest.mark.gpu

CASES = {
    "w2_plain_causal_d64_ragged": dict(world=2, n=300, h=2, d=64, causal=True),
    "w2_plain_kmask_gqa_d128_fp16": dict(world=2, n=777, h=4, hk=1, d=128, kmask=True, dtype="fp16", b=2),
    "w3_zigzag_causal_d64": dict(world=3, n=300, h=2, d=64, layout="zigzag", causal=True),
    "w3_plain_kmask_gqa_d64_ragged": dict(world=3, n=777, h=4, hk=2, d=64, kmask=True),
    "w4_striped_causal_gqa_d64": dict(world=4, n=300, h=4, hk=2, d=64, layout="striped", causal=True),
    "w4_zigzag_causal_d128": dict(world=4, n=384, h=2, d=128, layout="zigzag", causal=True),
    "w4_plain_window_d64": dict(world=4, n=256, h=2, d=64, causal=True, window=300),
    "w4_zigzag_softclamp_fp16_d64": dict(world=4, n=384, h=2, d=64, layout="zigzag", causal=True, softclamp=20.0,
                                         dtype="fp16"),
    "w4_striped_kmask_d128": dict(world=4, n=300, h=2, d=128, layout="striped", kmask=True, b=2),
    "w8_plain_causal_d64": dict(world=8, n=256, h=2, d=64, causal=True),
    "w8_striped_causal_gqa_d128": dict(world=8, n=256, h=4, hk=2, d=128, layout="striped", causal=True),
    "w8_plain_window_sparse_gqa_d64": dict(world=8, n=256, h=4, hk=2, d=64, causal=True, window=300),
}


def _oracle_grads(qs, ks, vs, dos, layout, causal, window, softclamp, kms):
    from ring_attention_pytorch_b200.ops.oracle import attention_with_positions
    from ring_attention_pytorch_b200.parallel.layout import make_position_map

    world, n = len(qs), qs[0].shape[1]
    pm = make_position_map(layout, world, n)
    qf = [q.float().requires_grad_() for q in qs]
    kf = [k.float().requires_grad_() for k in ks]
    vf = [v.float().requires_grad_() for v in vs]
    k_all, v_all = torch.cat(kf, 1), torch.cat(vf, 1)
    k_pos = torch.cat([pm.positions(r, "cuda") for r in range(world)])
    km = None if kms is None else torch.cat(kms, 1)
    loss = 0.0
    for r in range(world):
        o = attention_with_positions(qf[r], k_all, v_all, pm.positions(r, "cuda"), k_pos, causal=causal, window=window,
                                     key_mask=km, softclamp_value=softclamp)
        loss = loss + (o * dos[r].float()).sum()
    loss.backward()
    return [(qf[r].grad, kf[r].grad, vf[r].grad) for r in range(world)]


@pytest.mark.parametrize("name", list(CASES))
def test_two_kernel_hopwise_backward(name):
    from ring_attention_pytorch_b200.ops.fused import emulate_ring_backward, emulate_ring_forward

    c = dict(b=1, hk=None, layout="plain", causal=False, window=None, softclamp=0.0, kmask=False, dtype="bf16")
    c.update(CASES[name])
    world, b, n, h, d = c["world"], c["b"], c["n"], c["h"], c["d"]
    hk = c["hk"] or h
    dt = torch.bfloat16 if c["dtype"] == "bf16" else torch.float16
    torch.manual_seed(0)
    qs = [torch.randn(b, n, h, d, device="cuda", dtype=dt) for _ in range(world)]
    ks = [torch.randn(b, n, hk, d, device="cuda", dtype=dt) for _ in range(world)]
    vs = [torch.randn(b, n, hk, d, device="cuda", dtype=dt) for _ in range(world)]
    dos = [torch.randn(b, n, h, d, device="cuda", dtype=dt) for _ in range(world)]
    kms = [torch.rand(b, n, device="cuda") > 0.3 for _ in range(world)] if c["kmask"] else None
    kw = dict(layout=c["layout"], causal=c["causal"], window=c["window"], softclamp=c["softclamp"], key_masks=kms)
    outs, lses = emulate_ring_forward(qs, ks, vs, **kw)
    gather = emulate_ring_backward(qs, ks, vs, outs, lses, dos, fused=False, hopwise=False, **kw)
    hop = emulate_ring_backward(qs, ks, vs, outs, lses, dos, fused=False, hopwise=True, **kw)
    again = emulate_ring_backward(qs, ks, vs, outs, lses, dos, fused=False, hopwise=True, **kw)
    torch.cuda.synchronize()

    for r in range(world):
        for i, what in enumerate(("dq", "dk", "dv")):
            assert torch.equal(hop[r][i], again[r][i]), (r, what, "not deterministic")
            if what == "dq" or hk == h:
                assert torch.equal(hop[r][i], gather[r][i]), (r, what, "differs from the one-launch backward")
    ref = _oracle_grads(qs, ks, vs, dos, c["layout"], c["causal"], c["window"], c["softclamp"], kms)
    for i, what in enumerate(("dq", "dk", "dv")):
        err = max((hop[r][i].float() - ref[r][i]).abs().max().item() for r in range(world))
        scale = max(ref[r][i].abs().max().item() for r in range(world))
        assert err / max(scale, 1e-6) < 3e-2, (what, err, scale)
        assert not any(torch.isnan(hop[r][i].float()).any().item() for r in range(world)), what


# ------------------------------------------------------------------------------------------------
# real ring, head dim 64, memory="ring" against memory="gather" on the same inputs – needs >= 2 devices
# ------------------------------------------------------------------------------------------------
def _hop_ring_worker(rank, world, layout, hk, kmask):
    import torch.distributed as dist

    from ring_attention_pytorch_b200.ops import ring_cuda
    from ring_attention_pytorch_b200.ops.fused import pad64
    from ring_attention_pytorch_b200.ops.ring_cuda import ring_flash_attn_cuda
    from ring_attention_pytorch_b200.parallel.symm import get_workspace
    from ring_attention_pytorch_b200.utils.check import sampled_check

    n, h, d = 8192, 8, 64
    torch.manual_seed(100 + rank)
    dev = torch.device("cuda", rank)
    q = torch.randn(1, n, h, d, device=dev, dtype=torch.bfloat16, requires_grad=True)
    k = torch.randn(1, n, hk, d, device=dev, dtype=torch.bfloat16, requires_grad=True)
    v = torch.randn(1, n, hk, d, device=dev, dtype=torch.bfloat16, requires_grad=True)
    g = torch.randn(1, n, h, d, device=dev, dtype=torch.bfloat16)
    causal = layout != "plain"
    mask = None
    if kmask:
        gen = torch.Generator(device=dev).manual_seed(7 + rank)
        mask = torch.rand(1, n, device=dev, generator=gen) > 0.3

    def run(memory):
        ring_cuda.CONFIG["memory"] = memory
        out = ring_flash_attn_cuda(q, k, v, mask, causal, 1024, True, layout == "striped", None, world, False, 50.0,
                                   layout)
        torch.cuda.synchronize(dev)
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        grads = torch.autograd.grad(out, (q, k, v), g)
        torch.cuda.synchronize(dev)
        return out.detach(), grads, torch.cuda.max_memory_allocated(dev) - base

    out, (dq, dk, dv), hop_peak = run("ring")
    kv_slot = 2 * n * hk * d * 2
    qdo_slot = 2 * n * h * d * 2 + 2 * h * pad64(n) * 4  # Q/dO + statistics
    regions = get_workspace(world, dev).regions
    # the workspace is O(n / W): own slots (double buffered), never a W-slot gather
    assert "kv_gather" not in regions, list(regions)
    assert regions["kv_own"].nbytes <= 2 * kv_slot + 1024 and regions["qdo"].nbytes <= 2 * qdo_slot + 1024, \
        {name: r.nbytes for name, r in regions.items()}
    # and so is the backward's own allocation: two 2-slot windows, the fp32 carries and the 16-bit gradients
    carries = n * h * d * 4 + 2 * n * hk * d * 4
    grads16 = (n * h * d + 2 * n * hk * d) * 2
    assert hop_peak <= 2 * qdo_slot + 2 * kv_slot + carries + grads16 + (16 << 20), hop_peak

    if not kmask:  # the sampled oracle has no key mask: the masked case is held to the gather mode, bit for bit
        res = sampled_check(q.detach(), k.detach(), v.detach(), g, out, dq, dk, dv, causal=causal, layout=layout,
                            world=world, rank=rank, head_index=h - 1, samples=48, chunk=1024)
        assert res["ok"], res
    assert all(torch.isfinite(t.float()).all() for t in (dq, dk, dv))

    out_g, (dq_g, dk_g, dv_g), gather_peak = run("gather")
    assert torch.equal(out, out_g)
    assert torch.equal(dq, dq_g)
    if hk == h:
        assert torch.equal(dk, dk_g) and torch.equal(dv, dv_g)
    if world >= 4:
        # gather mode holds W Q/dO + statistics slots in the allocator (its K/V gather is symmetric memory); hop mode
        # holds two of them plus what it adds: the carries and the K/V window
        assert gather_peak - hop_peak >= (world - 2) * qdo_slot - carries - 2 * kv_slot, (gather_peak, hop_peak)
    torch.cuda.synchronize()
    dist.barrier()


@pytest.mark.parametrize("layout,hk,kmask", [("striped", 2, False), ("zigzag", 8, False), ("plain", 8, True)])
def test_real_ring_two_kernel_hop_mode_d64(layout, hk, kmask):
    """Head dim 64 under ``memory="ring"`` on every visible GPU (2, 4 or 8): sampled rows against the fp32 oracle,
    bitwise equal to ``memory="gather"`` (dQ; dK / dV without grouped heads), and O(n / W) memory."""
    world = torch.cuda.device_count()
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    from dist_utils import run_distributed

    world = 8 if world >= 8 else (4 if world >= 4 else 2)
    run_distributed(_hop_ring_worker, world, layout, hk, kmask, backend="nccl", timeout=600.0)
