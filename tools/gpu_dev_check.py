"""GPU bring-up checks, each case in its own subprocess with a timeout so a trap or hang in one kernel
cannot take the rest of the (expensive) gpurun call down.

    python tools/gpu_dev_check.py [--only probe,fwd,ring,perf] [--timeout 120]

Writes gpurun_out/dev_check.log and prints a summary.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


# ----------------------------------------------------------------------------------------------
# individual cases (run in a child process: `python tools/gpu_dev_check.py --case NAME`)
# ----------------------------------------------------------------------------------------------
def _idesc(M, N, a_mn, b_mn, bf16=1):
    return (1 << 4) | (bf16 << 7) | (bf16 << 10) | (a_mn << 15) | (b_mn << 16) | ((N >> 3) << 17) | ((M >> 4) << 24)


def case_probe(mode: int, variant: str = "base"):
    import torch
    from ring_attention_pytorch_b200.ops import _ext

    ops = _ext.ops()
    torch.manual_seed(0)
    n, k = 128, 128
    if variant == "n64":
        n = 64
    if variant == "k64":
        k = 64
    a = torch.randn(128, k, device="cuda", dtype=torch.bfloat16)
    if mode == 0:
        b = torch.randn(n, k, device="cuda", dtype=torch.bfloat16)
        ref = a.float() @ b.float().t()
        idesc = _idesc(128, n, 0, 0)
        out = ops.umma_probe(a, b, 0, n, k, idesc, 16, 1024, 16, 1024, 0)
    else:
        b = torch.randn(k, n, device="cuda", dtype=torch.bfloat16)
        ref = a.float() @ b.float()
        idesc = _idesc(128, n, 0, 1)
        lbo, sbo, kstep = 16384, 1024, 2048
        if variant == "swap":
            lbo, sbo = 1024, 16384
        out = ops.umma_probe(a, b, mode, n, k, idesc, 16, 1024, lbo, sbo, kstep)
    torch.cuda.synchronize()
    err = (out - ref).abs().max().item()
    rel = err / ref.abs().max().item()
    return {"max_abs_err": err, "rel": rel, "ok": rel < 2e-2}


def case_probe_mn_a(k: int = 128):
    """MN-major A from shared memory plus a B tile written by the threads with a hand-applied 128B swizzle — the two
    operand flavours the one-kernel (5-GEMM) backward needs for dQ^T = K^T dS^T."""
    import torch
    from ring_attention_pytorch_b200.ops import _ext

    ops = _ext.ops()
    torch.manual_seed(0)
    at = torch.randn(k, 128, device="cuda", dtype=torch.bfloat16)   # A^T: [K][M]
    b = torch.randn(k, 64, device="cuda", dtype=torch.bfloat16)     # B:   [K][N]
    ref = at.float().t() @ b.float()
    idesc = _idesc(128, 64, 1, 1)
    out = ops.umma_probe(at, b, 3, 64, k, idesc, 16384, 1024, 16384, 1024, 2048)
    torch.cuda.synchronize()
    err = (out - ref).abs().max().item()
    rel = err / ref.abs().max().item()
    return {"max_abs_err": err, "rel": rel, "ok": rel < 2e-2}


def _ref_ring(qs, ks, vs, layout, causal, window, softclamp, key_masks):
    import torch
    from ring_attention_pytorch_b200.ops.oracle import attention_with_positions
    from ring_attention_pytorch_b200.parallel.layout import make_position_map

    world = len(qs)
    n = qs[0].shape[1]
    pm = make_position_map(layout, world, n)
    k_all = torch.cat([k.float() for k in ks], 1)
    v_all = torch.cat([v.float() for v in vs], 1)
    k_pos = torch.cat([pm.positions(r, qs[0].device) for r in range(world)])
    km = None if key_masks is None else torch.cat(list(key_masks), 1)
    outs, lses = [], []
    for r in range(world):
        o, lse = attention_with_positions(qs[r].float(), k_all, v_all, pm.positions(r, qs[0].device), k_pos,
                                          causal=causal, window=window, key_mask=km, softclamp_value=softclamp,
                                          return_lse=True)
        outs.append(o)
        lses.append(lse)
    return outs, lses


def case_fwd(world=1, b=1, n=256, h=2, hk=None, d=128, layout="plain", causal=False, window=None, softclamp=0.0,
             kmask=False, dtype="bf16", seed=0, hopwise=False):
    import torch
    from ring_attention_pytorch_b200.ops.fused import emulate_ring_forward

    hk = hk or h
    torch.manual_seed(seed)
    dt = torch.bfloat16 if dtype == "bf16" else torch.float16
    qs = [torch.randn(b, n, h, d, device="cuda", dtype=dt) for _ in range(world)]
    ks = [torch.randn(b, n, hk, d, device="cuda", dtype=dt) for _ in range(world)]
    vs = [torch.randn(b, n, hk, d, device="cuda", dtype=dt) for _ in range(world)]
    kms = None
    if kmask:
        kms = [torch.rand(b, n, device="cuda") > 0.3 for _ in range(world)]
    outs, lses = emulate_ring_forward(qs, ks, vs, layout=layout, causal=causal, window=window, softclamp=softclamp,
                                      key_masks=kms, hopwise=hopwise)
    torch.cuda.synchronize()
    routs, rlses = _ref_ring(qs, ks, vs, layout, causal, window, softclamp, kms)
    err = max((o.float() - r).abs().max().item() for o, r in zip(outs, routs))
    fin = [torch.isfinite(r) for r in rlses]
    lerr = max(((l - r)[f]).abs().max().item() if f.any() else 0.0 for l, r, f in zip(lses, rlses, fin))
    nan = any(torch.isnan(o.float()).any().item() for o in outs)
    return {"max_abs_err": err, "lse_err": lerr, "nan": nan, "ok": (err < 3e-2) and (lerr < 2e-2) and not nan}


def case_bwd(world=1, b=1, n=256, h=2, hk=None, d=128, layout="plain", causal=False, window=None, softclamp=0.0,
             kmask=False, dtype="bf16", seed=0, fused=None, hopwise=False):
    import torch
    from ring_attention_pytorch_b200.ops.fused import emulate_ring_backward, emulate_ring_forward
    from ring_attention_pytorch_b200.ops.oracle import attention_with_positions
    from ring_attention_pytorch_b200.parallel.layout import make_position_map

    hk = hk or h
    torch.manual_seed(seed)
    dt = torch.bfloat16 if dtype == "bf16" else torch.float16
    qs = [torch.randn(b, n, h, d, device="cuda", dtype=dt) for _ in range(world)]
    ks = [torch.randn(b, n, hk, d, device="cuda", dtype=dt) for _ in range(world)]
    vs = [torch.randn(b, n, hk, d, device="cuda", dtype=dt) for _ in range(world)]
    dos = [torch.randn(b, n, h, d, device="cuda", dtype=dt) for _ in range(world)]
    kms = None
    if kmask:
        kms = [torch.rand(b, n, device="cuda") > 0.3 for _ in range(world)]
    outs, lses = emulate_ring_forward(qs, ks, vs, layout=layout, causal=causal, window=window, softclamp=softclamp,
                                      key_masks=kms, hopwise=hopwise)
    grads = emulate_ring_backward(qs, ks, vs, outs, lses, dos, layout=layout, causal=causal, window=window,
                                  softclamp=softclamp, key_masks=kms, fused=fused, hopwise=hopwise)
    torch.cuda.synchronize()
    # fp32 oracle through autograd
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
    errs = {"dq": 0.0, "dk": 0.0, "dv": 0.0}
    scale_ref = {"dq": 0.0, "dk": 0.0, "dv": 0.0}
    nan = False
    for r in range(world):
        for name, got, ref in (("dq", grads[r][0], qf[r].grad), ("dk", grads[r][1], kf[r].grad),
                               ("dv", grads[r][2], vf[r].grad)):
            errs[name] = max(errs[name], (got.float() - ref).abs().max().item())
            scale_ref[name] = max(scale_ref[name], ref.abs().max().item())
            nan = nan or bool(torch.isnan(got.float()).any().item())
    rel = {k2: errs[k2] / max(scale_ref[k2], 1e-6) for k2 in errs}
    ok = all(v < 3e-2 for v in rel.values()) and not nan
    res = {"abs": errs, "rel": rel, "nan": nan, "ok": ok}
    if not ok:
        # localise: per rank / tensor / head / 128-row tile error (nan -> 999)
        detail = {}
        for r in range(world):
            for name, got, ref in (("dq", grads[r][0], qf[r].grad), ("dk", grads[r][1], kf[r].grad),
                                   ("dv", grads[r][2], vf[r].grad)):
                e = torch.nan_to_num((got.float() - ref).abs(), nan=999.0)
                nt = (n + 127) // 128
                pad = nt * 128 - n
                e = torch.nn.functional.pad(e, (0, 0, 0, 0, 0, pad))
                tile = e.view(b, nt, 128, e.shape[2], d).amax(dim=(2, 4))  # [b, tile, head]
                detail[f"r{r}_{name}"] = [[round(x, 3) for x in row] for row in tile[0].tolist()]
        res["detail_b0_tile_by_head"] = detail
    return res


def case_perf_bwd_fused(n=16384, h=16, causal=True, iters=5, b=1, hk=None):
    """The one-kernel backward (prep + kernel + dQ convert), timed like case_perf_bwd."""
    import torch
    from ring_attention_pytorch_b200.ops import _ext
    from ring_attention_pytorch_b200.ops.fused import (AttnProblem, alloc_kv_buffer, alloc_qdo_buffer,
                                                       alloc_stat_buffer, fused_attn_bwd_ring, fused_attn_fwd)
    from ring_attention_pytorch_b200.parallel.layout import make_position_map

    ops = _ext.ops()
    hk = hk or h
    d = 128
    dt = torch.bfloat16
    q = torch.randn(b, n, h, d, device="cuda", dtype=dt)
    k = torch.randn(b, n, hk, d, device="cuda", dtype=dt)
    v = torch.randn(b, n, hk, d, device="cuda", dtype=dt)
    do = torch.randn(b, n, h, d, device="cuda", dtype=dt)
    pm = make_position_map("plain", 1, n)
    kv = alloc_kv_buffer(1, b, hk, n, d, dt, "cuda")
    qdo = alloc_qdo_buffer(1, b, h, n, d, dt, "cuda")
    stat = alloc_stat_buffer(1, b, h, n, "cuda")
    ops.pack_kv(k, v, kv[0])
    ready = torch.zeros(1, dtype=torch.int32, device="cuda")
    prob = AttnProblem(b, h, hk, 0, pm, causal, None, d ** -0.5)
    o, lse = fused_attn_fwd(prob, q, kv, [0], ready)
    dq = torch.empty_like(q)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]

    def run(timed=False):
        if timed:
            ev[0].record()
        ops.bwd_prep(q, o, do, lse, qdo, stat, 0)
        if timed:
            ev[1].record()
        acc = torch.zeros(b * h, stat.shape[-1], d, dtype=torch.float32, device="cuda")
        if timed:
            ev[2].record()
        _, dk, dv = fused_attn_bwd_ring(prob, qdo[0], stat[0], kv, dq_acc=acc)
        if timed:
            ev[3].record()
        ops.acc_convert(acc, dq, d ** -0.5)
        if timed:
            ev[4].record()
        return dq, dk, dv

    for _ in range(2):
        run()
    torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    ms = sorted(times)[len(times) // 2]
    flops = 2.5 * 4.0 * b * h * n * n * d * (0.5 if causal else 1.0)
    run(timed=True)
    torch.cuda.synchronize()
    return {"ms": ms, "tflops_5gemm": flops / ms / 1e9, "ms_prep": ev[0].elapsed_time(ev[1]),
            "ms_zero": ev[1].elapsed_time(ev[2]), "ms_kernel": ev[2].elapsed_time(ev[3]),
            "ms_convert": ev[3].elapsed_time(ev[4]), "tflops_kernel_only": flops / ev[2].elapsed_time(ev[3]) / 1e9,
            "ok": True}


def case_perf_bwd(n=16384, h=16, d=128, causal=True, iters=5, b=1, hk=None):
    import torch
    from ring_attention_pytorch_b200.ops import _ext
    from ring_attention_pytorch_b200.ops.fused import (AttnProblem, alloc_kv_buffer, alloc_qdo_buffer,
                                                       alloc_stat_buffer, fused_attn_bwd, fused_attn_fwd)
    from ring_attention_pytorch_b200.parallel.layout import make_position_map

    ops = _ext.ops()
    hk = hk or h
    dt = torch.bfloat16
    q = torch.randn(b, n, h, d, device="cuda", dtype=dt)
    k = torch.randn(b, n, hk, d, device="cuda", dtype=dt)
    v = torch.randn(b, n, hk, d, device="cuda", dtype=dt)
    do = torch.randn(b, n, h, d, device="cuda", dtype=dt)
    pm = make_position_map("plain", 1, n)
    kv = alloc_kv_buffer(1, b, hk, n, d, dt, "cuda")
    qdo = alloc_qdo_buffer(1, b, h, n, d, dt, "cuda")
    stat = alloc_stat_buffer(1, b, h, n, "cuda")
    ops.pack_kv(k, v, kv[0])
    ready = torch.zeros(1, dtype=torch.int32, device="cuda")
    prob = AttnProblem(b, h, hk, 0, pm, causal, None, d ** -0.5)
    o, lse = fused_attn_fwd(prob, q, kv, [0], ready)

    def run():
        ops.bwd_prep(q, o, do, lse, qdo, stat, 0)
        return fused_attn_bwd(prob, qdo, kv, stat)

    for _ in range(2):
        run()
    torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    ms = sorted(times)[len(times) // 2]
    flops = 2.5 * 4.0 * b * h * n * n * d * (0.5 if causal else 1.0)
    res = {"ms": ms, "tflops_5gemm_equiv": flops / ms / 1e9, "tflops_executed_7gemm": flops * 1.4 / ms / 1e9}
    # per-kernel split
    e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    e[0].record()
    ops.bwd_prep(q, o, do, lse, qdo, stat, 0)
    e[1].record()
    ops.attn_bwd_dq(qdo, kv, stat, None, 0, *prob.tail([0]))
    e[2].record()
    ops.attn_bwd_dkdv(qdo, kv, stat, None, 0, *prob.tail([0]))
    e[3].record()
    torch.cuda.synchronize()
    res["ms_prep"], res["ms_dq"], res["ms_dkdv"] = e[0].elapsed_time(e[1]), e[1].elapsed_time(e[2]), e[2].elapsed_time(e[3])
    try:
        from flash_attn import flash_attn_func

        qq, kk, vv = (t.clone().requires_grad_() for t in (q, k, v))
        out = flash_attn_func(qq, kk, vv, causal=causal)
        out.backward(do, retain_graph=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            out.backward(do, retain_graph=True)
        e1.record()
        torch.cuda.synchronize()
        res["flash_attn2_bwd_tflops"] = flops / (e0.elapsed_time(e1) / 3) / 1e9
    except Exception as ex:  # noqa: BLE001
        res["flash_attn2_bwd_tflops"] = f"n/a: {type(ex).__name__}"
    res["ok"] = True
    return res


def case_perf_decode(batch=256, h=32, hk=8, n=8192, d=128, fp8=False, iters=20, tensor_core="auto"):
    import torch
    from ring_attention_pytorch_b200.ops import tree_decode_cuda as tdc
    from ring_attention_pytorch_b200.ops.tree_decode_cuda import tree_decode_cuda

    tdc.CONFIG["tensor_core"] = tensor_core

    q = torch.randn(batch, h, 1, d, device="cuda", dtype=torch.bfloat16)
    k = torch.randn(batch, hk, n, d, device="cuda", dtype=torch.bfloat16)
    v = torch.randn(batch, hk, n, d, device="cuda", dtype=torch.bfloat16)
    ks = vs = None
    if fp8:
        k, v = k.to(torch.float8_e4m3fn), v.to(torch.float8_e4m3fn)
        ks = torch.ones(batch * hk, device="cuda")
        vs = torch.ones(batch * hk, device="cuda")
    for _ in range(3):
        out = tree_decode_cuda(q, k, v, dim_v=d, k_scale=ks, v_scale=vs)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        out = tree_decode_cuda(q, k, v, dim_v=d, k_scale=ks, v_scale=vs)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    kv_bytes = 2 * k.numel() * k.element_size()
    # correctness spot check on a slice
    kx = k[:2].float().repeat(1, h // hk, 1, 1)
    vx = v[:2].float().repeat(1, h // hk, 1, 1)
    sim = torch.einsum("bhid,bhjd->bhij", q[:2].float(), kx) * d ** -0.5
    ref = torch.einsum("bhij,bhjd->bhid", sim.softmax(-1), vx)
    err = (out[:2].float() - ref).abs().max().item()
    return {"ms": ms, "kv_gb_per_s": kv_bytes / ms / 1e6, "hbm_frac_of_6585": kv_bytes / ms / 1e6 / 6585.0, "err": err,
            "tensor_core": tensor_core, "launches_per_step": 1, "ok": err < 3e-2}


def case_perf_hop(world=4, n=16384, h=8, hk=None, d=128, layout="striped", causal=True, iters=3):
    """Cost of the hop-at-a-time schedule (memory="ring") against the single-launch schedule for one emulated rank:
    same K/V slots (already local: no transfer in either arm), forward and one-kernel backward."""
    import torch
    from ring_attention_pytorch_b200.ops import _ext
    from ring_attention_pytorch_b200.ops.fused import (AttnProblem, alloc_kv_buffer, alloc_qdo_buffer,
                                                       alloc_stat_buffer, backward_hops, forward_hops,
                                                       fused_attn_bwd_ring, fused_attn_fwd, pad128)
    from ring_attention_pytorch_b200.parallel.layout import make_position_map

    ops = _ext.ops()
    hk = hk or h
    dt = torch.bfloat16
    b, rank = 1, world - 1
    q = torch.randn(b, n, h, d, device="cuda", dtype=dt)
    do = torch.randn(b, n, h, d, device="cuda", dtype=dt)
    buf = alloc_kv_buffer(world, b, hk, n, d, dt, "cuda")
    for o_ in range(world):
        ops.pack_kv(torch.randn(b, n, hk, d, device="cuda", dtype=dt), torch.randn(b, n, hk, d, device="cuda", dtype=dt),
                    buf[o_])
    pm = make_position_map(layout, world, n)
    prob = AttnProblem(b, h, hk, rank, pm, causal, None, d ** -0.5)
    hops = prob.kv_owners()
    ready = torch.zeros(world, dtype=torch.int32, device="cuda")
    accs = [torch.zeros(2, b * hk, pad128(n), d, dtype=torch.float32, device="cuda") for _ in range(world)]
    ptrs = [a.data_ptr() for a in accs]
    state = {}

    def fwd_single():
        state["o"], state["lse"] = fused_attn_fwd(prob, q, buf, [buf[o_].data_ptr() if o_ != rank else 0
                                                                 for o_ in range(world)], ready)

    def fwd_hop():
        state["o"], state["lse"] = forward_hops(ops, prob, q, hops, lambda s: buf[hops[s]])

    def prep():
        qdo = alloc_qdo_buffer(1, b, h, n, d, dt, "cuda")
        stat = alloc_stat_buffer(1, b, h, n, "cuda")
        ops.bwd_prep(q, state["o"], do, state["lse"], qdo, stat, 0)
        return qdo, stat

    def bwd_single():
        fused_attn_bwd_ring(prob, state["qdo"][0], state["stat"][0], buf, dq_acc=state["dq"], dkv_acc_ptrs=ptrs,
                            nk_pad=pad128(n))

    def bwd_hop():
        backward_hops(ops, prob, state["qdo"][0], state["stat"][0], state["dq"], hops, lambda s: buf[hops[s]],
                      dkv_acc_ptrs=ptrs, nk_pad=pad128(n))

    def timeit(fn):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(iters):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return sorted(ts)[len(ts) // 2]

    res = {"hops": len(hops)}
    res["fwd_single_ms"] = timeit(fwd_single)
    o_ref = state["o"].clone()
    res["fwd_hop_ms"] = timeit(fwd_hop)
    res["fwd_max_diff"] = (state["o"].float() - o_ref.float()).abs().max().item()
    state["qdo"], state["stat"] = prep()
    state["dq"] = torch.zeros(b * h, state["stat"].shape[-1], d, dtype=torch.float32, device="cuda")
    res["bwd_single_ms"] = timeit(bwd_single)
    res["bwd_hop_ms"] = timeit(bwd_hop)
    flops = 4.0 * b * h * n * (n * world) * d * (0.5 if causal else 1.0)
    res["fwd_single_tflops"] = flops / res["fwd_single_ms"] / 1e9
    res["fwd_hop_tflops"] = flops / res["fwd_hop_ms"] / 1e9
    res["bwd_single_tflops"] = 2.5 * flops / res["bwd_single_ms"] / 1e9
    res["bwd_hop_tflops"] = 2.5 * flops / res["bwd_hop_ms"] / 1e9
    res["ok"] = res["fwd_max_diff"] < 2e-2
    return res


def case_perf(n=16384, h=16, d=128, causal=True, iters=5, b=1, hk=None):
    import torch
    from ring_attention_pytorch_b200.ops import _ext
    from ring_attention_pytorch_b200.ops.fused import AttnProblem, alloc_kv_buffer, fused_attn_fwd
    from ring_attention_pytorch_b200.parallel.layout import make_position_map

    ops = _ext.ops()
    hk = hk or h
    dt = torch.bfloat16
    q = torch.randn(b, n, h, d, device="cuda", dtype=dt)
    k = torch.randn(b, n, hk, d, device="cuda", dtype=dt)
    v = torch.randn(b, n, hk, d, device="cuda", dtype=dt)
    pm = make_position_map("plain", 1, n)
    buf = alloc_kv_buffer(1, b, hk, n, d, dt, "cuda")
    ops.pack_kv(k, v, buf[0])
    ready = torch.zeros(1, dtype=torch.int32, device="cuda")

    prob = AttnProblem(b, h, hk, 0, pm, causal, None, d ** -0.5)

    def run():
        return fused_attn_fwd(prob, q, buf, [0], ready)

    for _ in range(2):
        run()
    torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    ms = sorted(times)[len(times) // 2]
    flops = 4.0 * b * h * n * n * d * (0.5 if causal else 1.0)
    res = {"ms": ms, "tflops": flops / ms / 1e9}
    try:
        from flash_attn import flash_attn_func

        for _ in range(2):
            flash_attn_func(q, k, v, causal=causal)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            flash_attn_func(q, k, v, causal=causal)
        e1.record()
        torch.cuda.synchronize()
        res["flash_attn2_tflops"] = flops / (e0.elapsed_time(e1) / 3) / 1e9
    except Exception as e:  # noqa: BLE001
        res["flash_attn2_tflops"] = f"n/a: {type(e).__name__}"
    res["ok"] = True
    return res


CASES = {
    # descriptor probes
    "probe_ss_kmajor": lambda: case_probe(0),
    "probe_ss_kmajor_k64": lambda: case_probe(0, "k64"),
    "probe_ss_mnmajor": lambda: case_probe(1),
    "probe_ss_mnmajor_n64": lambda: case_probe(1, "n64"),
    "probe_ss_mnmajor_swap": lambda: case_probe(1, "swap"),
    "probe_ts_mnmajor": lambda: case_probe(2),
    "probe_ts_mnmajor_n64": lambda: case_probe(2, "n64"),
    # single-rank forward
    "fwd_d128_n256": lambda: case_fwd(),
    "fwd_d128_n128_h1": lambda: case_fwd(n=128, h=1),
    "fwd_d128_causal_n512": lambda: case_fwd(n=512, causal=True),
    "fwd_d128_n300_tail": lambda: case_fwd(n=300, b=2),
    "fwd_d128_causal_n1000": lambda: case_fwd(n=1000, causal=True, h=4),
    "fwd_d64_n512": lambda: case_fwd(n=512, d=64, h=4),
    "fwd_d64_causal_n777": lambda: case_fwd(n=777, d=64, h=4, causal=True),
    "fwd_gqa_causal": lambda: case_fwd(n=512, h=8, hk=2, causal=True),
    "fwd_kmask": lambda: case_fwd(n=384, h=2, kmask=True, b=2),
    "fwd_softclamp": lambda: case_fwd(n=384, h=2, softclamp=20.0),
    "fwd_window": lambda: case_fwd(n=1024, h=2, causal=True, window=200),
    "fwd_fp16": lambda: case_fwd(n=512, h=2, causal=True, dtype="fp16"),
    "fwd_many_items": lambda: case_fwd(n=2048, h=16, b=2, causal=True),
    # emulated rings (W ranks on one GPU)
    "ring2_plain": lambda: case_fwd(world=2, n=256, h=2),
    "ring2_plain_causal": lambda: case_fwd(world=2, n=256, h=2, causal=True),
    "ring4_striped_causal": lambda: case_fwd(world=4, n=384, h=4, hk=2, layout="striped", causal=True),
    "ring4_zigzag_causal": lambda: case_fwd(world=4, n=512, h=2, layout="zigzag", causal=True),
    "ring4_plain_window": lambda: case_fwd(world=4, n=256, h=2, causal=True, window=300),
    "ring3_kmask": lambda: case_fwd(world=3, n=200, h=2, kmask=True),
    "ring8_striped_causal_big": lambda: case_fwd(world=8, n=1024, h=8, hk=2, layout="striped", causal=True),
    # backward, single rank
    "probe_mn_a": lambda: case_probe_mn_a(),
    "probe_mn_a_k64": lambda: case_probe_mn_a(64),
    "bwd_d128_n256": lambda: case_bwd(),
    "bwd_d128_n128_h1": lambda: case_bwd(n=128, h=1),
    "bwd_d128_n64_h1": lambda: case_bwd(n=64, h=1),
    "bwd_d128_causal_n512": lambda: case_bwd(n=512, causal=True),
    "bwd_d128_n300_tail": lambda: case_bwd(n=300, b=2),
    "bwd_d128_causal_n1000": lambda: case_bwd(n=1000, causal=True, h=4),
    "bwd_d64_n512": lambda: case_bwd(n=512, d=64, h=4),
    "bwd_d64_causal_n777": lambda: case_bwd(n=777, d=64, h=4, causal=True),
    "bwd_gqa_causal": lambda: case_bwd(n=512, h=8, hk=2, causal=True),
    "bwd_kmask": lambda: case_bwd(n=384, h=2, kmask=True, b=2),
    "bwd_softclamp": lambda: case_bwd(n=384, h=2, softclamp=20.0),
    "bwd_window": lambda: case_bwd(n=1024, h=2, causal=True, window=200),
    "bwd_fp16": lambda: case_bwd(n=512, h=2, causal=True, dtype="fp16"),
    "bwd_many_items": lambda: case_bwd(n=2048, h=16, b=2, causal=True),
    # backward, emulated rings
    "rbwd2_plain_h1": lambda: case_bwd(world=2, n=128, h=1),
    "rbwd3_plain": lambda: case_bwd(world=3, n=128, h=1),
    "rbwd3_plain_causal": lambda: case_bwd(world=3, n=128, h=1, causal=True),
    "rbwd4_plain_causal": lambda: case_bwd(world=4, n=256, h=2, causal=True),
    "rbwd2_plain": lambda: case_bwd(world=2, n=256, h=2),
    "rbwd2_plain_causal": lambda: case_bwd(world=2, n=256, h=2, causal=True),
    "rbwd4_striped_causal": lambda: case_bwd(world=4, n=384, h=4, hk=2, layout="striped", causal=True),
    "rbwd4_zigzag_causal": lambda: case_bwd(world=4, n=512, h=2, layout="zigzag", causal=True),
    "rbwd4_plain_window": lambda: case_bwd(world=4, n=256, h=2, causal=True, window=300),
    "rbwd3_kmask": lambda: case_bwd(world=3, n=200, h=2, kmask=True),
    # the two-kernel backward at head dim 128 (the default there is the one-kernel backward)
    "bwd2k_d128_causal_n1000": lambda: case_bwd(n=1000, causal=True, h=4, fused=False),
    "bwd2k_gqa_causal": lambda: case_bwd(n=512, h=8, hk=2, causal=True, fused=False),
    "bwd2k_ring4_striped_causal": lambda: case_bwd(world=4, n=384, h=4, hk=2, layout="striped", causal=True, fused=False),
    # performance
    "perffz_causal_16k": lambda: case_perf_bwd_fused(),
    "perffz_full_8k": lambda: case_perf_bwd_fused(n=8192, causal=False),
    "perffz_causal_64k_h8": lambda: case_perf_bwd_fused(n=65536, h=8, iters=3),
    "perffz_gqa_causal_32k": lambda: case_perf_bwd_fused(n=32768, h=16, hk=4, iters=3),
    "perfbwd_causal_16k": lambda: case_perf_bwd(),
    "perfbwd_full_8k": lambda: case_perf_bwd(n=8192, causal=False),
    "perfbwd_causal_64k_h8": lambda: case_perf_bwd(n=65536, h=8, iters=3),
    "dec_small_tc": lambda: case_perf_decode(batch=2, h=8, hk=2, n=512, iters=1),
    "dec_small_tc_fp8": lambda: case_perf_decode(batch=2, h=8, hk=2, n=512, iters=1, fp8=True),
    "dec_small_cudacore": lambda: case_perf_decode(batch=2, h=8, hk=2, n=512, iters=1, tensor_core=False),
    "perfdec_bf16": lambda: case_perf_decode(),
    "perfdec_fp8": lambda: case_perf_decode(fp8=True),
    "perfdec_mha_b32": lambda: case_perf_decode(batch=32, h=32, hk=32, n=8192),
    "perfdec_cudacore_bf16": lambda: case_perf_decode(tensor_core=False),
    "perfdec_cudacore_fp8": lambda: case_perf_decode(fp8=True, tensor_core=False),
    "perfdec_g16_bf16": lambda: case_perf_decode(batch=64, h=64, hk=4, n=16384),
    "perfhop_w4_striped_16k": lambda: case_perf_hop(),
    "perfhop_w8_striped_8k_h16": lambda: case_perf_hop(world=8, n=8192, h=16),
    "perf_causal_16k": lambda: case_perf(),
    "perf_full_8k": lambda: case_perf(n=8192, causal=False),
    "perf_causal_64k_h8": lambda: case_perf(n=65536, h=8, iters=3),
    "perf_d64_causal_16k": lambda: case_perf(d=64, h=32),
}

GROUPS = {
    "probe": [c for c in CASES if c.startswith("probe")],
    "fwd": [c for c in CASES if c.startswith("fwd")],
    "ring": [c for c in CASES if c.startswith("ring")],
    "bwd": [c for c in CASES if c.startswith("bwd")],
    "rbwd": [c for c in CASES if c.startswith("rbwd")],
    "bwd2k": [c for c in CASES if c.startswith("bwd2k")],
    "perffz": [c for c in CASES if c.startswith("perffz")],
    "perfbwd": [c for c in CASES if c.startswith("perfbwd")],
    "perfdec": [c for c in CASES if c.startswith("perfdec")],
    "perf": [c for c in CASES if c.startswith("perf_")],
    "perfhop": [c for c in CASES if c.startswith("perfhop")],
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--case")
    ap.add_argument("--only", default="probe,fwd,ring,perf")
    ap.add_argument("--timeout", type=int, default=150)
    ap.add_argument("--log", default=os.path.join(ROOT, "gpurun_out", "dev_check.log"))
    ap.add_argument("--max-fail", type=int, default=0, help="stop after this many failed cases (0: never)")
    args = ap.parse_args()

    if args.case:
        res = CASES[args.case]()
        print("RESULT " + json.dumps(res))
        return

    os.makedirs(os.path.dirname(args.log), exist_ok=True)
    names = []
    for g in args.only.split(","):
        names += GROUPS.get(g, [g] if g in CASES else [])
    summary = []
    nfail = 0
    with open(args.log, "a") as log:
        log.write(f"\n==== dev check {time.strftime('%F %T')} only={args.only}\n")
        for name in names:
            t0 = time.time()
            try:
                proc = subprocess.run([sys.executable, os.path.abspath(__file__), "--case", name], capture_output=True,
                                      text=True, timeout=args.timeout)
                out = proc.stdout + proc.stderr
                line = [l for l in proc.stdout.splitlines() if l.startswith("RESULT ")]
                status = line[-1][7:] if line else f"FAILED rc={proc.returncode}"
            except subprocess.TimeoutExpired as e:
                out = (e.stdout or b"").decode() if isinstance(e.stdout, bytes) else (e.stdout or "")
                out += (e.stderr or b"").decode() if isinstance(e.stderr, bytes) else (e.stderr or "")
                status = "TIMEOUT"
            dt = time.time() - t0
            msg = f"{name:32s} {dt:6.1f}s  {status}"
            print(msg, flush=True)
            summary.append(msg)
            log.write(msg + "\n")
            if not status.startswith("{") or '"ok": false' in status:
                log.write("---- output tail\n" + out[-3000:] + "\n----\n")
                nfail += 1
            log.flush()
            if args.max_fail and nfail >= args.max_fail:
                print(f"stopping after {nfail} failed cases", flush=True)
                break


if __name__ == "__main__":
    main()
