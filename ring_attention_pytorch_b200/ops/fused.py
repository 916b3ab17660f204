"""Thin Python wrappers over the sm_100a kernels (``torch.ops.rab.*``).

These are the building blocks the autograd ops in :mod:`ring_attention_pytorch_b200.ops.ring_cuda`
compose; they are also what the GPU unit tests drive directly.  ``emulate_ring_forward`` runs a whole
W-rank ring on ONE device by giving every emulated rank its own K/V gather buffer and pointing the
"peer" addresses at the other ranks' buffers – the kernel cannot tell the difference, which lets the
multi-hop fetch/ready-flag protocol be tested on a single GPU.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, List, Optional, Sequence, Tuple

import torch

from ring_attention_pytorch_b200.ops import _ext
from ring_attention_pytorch_b200.parallel.layout import (PositionMap, make_position_map, ring_hop_owners,
                                                          ring_query_owners)


def pack_key_mask_bits(mask: torch.Tensor) -> torch.Tensor:
    """[world, b, n] bool (True = keep) -> [world, b, words] int32 bit-packed, words % 4 == 0."""
    world, b, n = mask.shape
    words = ((n + 127) // 128) * 4
    padded = torch.zeros(world, b, words * 32, dtype=torch.bool, device=mask.device)
    padded[..., :n] = mask
    bits = padded.view(world, b, words, 32).to(torch.int64)
    weights = (1 << torch.arange(32, device=mask.device, dtype=torch.int64))
    packed = (bits * weights).sum(-1)
    packed = torch.where(packed >= 2 ** 31, packed - 2 ** 32, packed)
    return packed.to(torch.int32).contiguous()


def alloc_kv_buffer(world: int, batch: int, kv_heads: int, n_k: int, d: int, dtype, device) -> torch.Tensor:
    return torch.empty(world, 2, batch * kv_heads, n_k, d, dtype=dtype, device=device)


@dataclass(frozen=True)
class AttnProblem:
    """The attention problem one ring rank's kernel launches share: shapes, ring position, masking and scaling.

    :meth:`tail` gives the arguments every ``torch.ops.rab.attn_*`` op ends with, in schema order."""
    batch: int
    heads: int
    kv_heads: int
    rank: int
    pm: PositionMap
    causal: bool
    window: Optional[int]
    scale: float
    softclamp: float = 0.0
    q_pos_offset: int = 0

    def kv_owners(self) -> List[int]:
        """K/V owners this rank visits, itself first."""
        return ring_hop_owners(self.pm, self.rank, self.causal, self.window)

    def q_owners(self) -> List[int]:
        """Ranks whose queries see this rank's keys, itself first."""
        return ring_query_owners(self.pm, self.rank, self.causal, self.window)

    def tail(self, hop_owner: Sequence[int], kmask_bits: Optional[torch.Tensor] = None) -> tuple:
        pm = self.pm
        return (kmask_bits, self.batch, self.heads, self.kv_heads, self.rank, bool(self.causal), int(self.window or 0),
                float(self.scale), float(self.softclamp), pm.stride, pm.seg_len, pm.base0, pm.base1,
                int(self.q_pos_offset), list(hop_owner))


def fused_attn_fwd(prob: AttnProblem, q: torch.Tensor, kv_buf: torch.Tensor, peer_ptrs: Sequence[int],
                   ready: torch.Tensor, kmask_bits: Optional[torch.Tensor] = None):
    """The whole ring in one launch: ``kv_buf`` ``[world, 2, b*hk, n_k, d]`` holds this rank's slot, the kernel's
    fetchers pull owner o's slot from ``peer_ptrs[o]`` (0: already in ``kv_buf``).  Returns (o, lse)."""
    return _ext.ops().attn_fwd(q, kv_buf, list(peer_ptrs), ready, *prob.tail(prob.kv_owners(), kmask_bits))


def alloc_fwd_carry(q: torch.Tensor):
    b, n_q, h, d = q.shape
    return (torch.empty(b, n_q, h, d, dtype=torch.float32, device=q.device),
            torch.empty(2, b * h, n_q, dtype=torch.float32, device=q.device))


def _no_hook(s: int) -> None:
    pass


def forward_hops(ops, prob: AttnProblem, q: torch.Tensor, hops: Sequence[int], slot: Callable[[int], torch.Tensor],
                 kmask_bits: Optional[torch.Tensor] = None, launched: Callable[[int], None] = _no_hook):
    """The forward one ring hop per launch (``memory="ring"``): hop ``s`` runs ``q`` against ``slot(s)``, owner
    ``hops[s]``'s K/V ``[2, b*hk, n_k, d]``; ``launched(s)`` follows each launch.

    The online-softmax state travels between the launches in fp32 carry buffers (un-normalised O, running maximum /
    sum); the last launch returns the final (o, lse).  The reference carries (o, m, lse) between its per-hop Triton
    launches the same way (ring_flash_attention_cuda.py:143-173)."""
    carry_o, carry_ml = alloc_fwd_carry(q)
    for s, owner in enumerate(hops):
        o, lse = ops.attn_fwd_hop(q, slot(s)[None], carry_o, carry_ml, s > 0, s + 1 < len(hops),
                                  *prob.tail([owner], kmask_bits))
        launched(s)
    return o, lse


def emulate_ring_forward(
    qs: Sequence[torch.Tensor],
    ks: Sequence[torch.Tensor],
    vs: Sequence[torch.Tensor],
    *,
    layout: str = "plain",
    causal: bool = False,
    window: Optional[int] = None,
    softclamp: float = 0.0,
    key_masks: Optional[Sequence[torch.Tensor]] = None,
    scale: Optional[float] = None,
    hopwise: bool = False,
):
    """Run the fused forward for every rank of a W-rank ring on the current device.

    qs/ks/vs: per-rank shards ``[b, n, h, d]`` / ``[b, n, hk, d]``.  Returns (outs, lses) lists.
    ``hopwise``: one launch per hop with carried softmax state (the ``memory="ring"`` schedule).
    """
    ops = _ext.ops()
    world = len(qs)
    b, n, h, d = qs[0].shape
    hk = ks[0].shape[2]
    dev, dt = qs[0].device, qs[0].dtype
    pm = make_position_map(layout, world, n)
    scale = d ** -0.5 if scale is None else scale
    bufs = [alloc_kv_buffer(world, b, hk, n, d, dt, dev) for _ in range(world)]
    for r in range(world):
        bufs[r].zero_()
        ops.pack_kv(ks[r], vs[r], bufs[r][r])
    kbits = None
    if key_masks is not None:
        kbits = pack_key_mask_bits(torch.stack(list(key_masks), 0))
    outs, lses = [], []
    for r in range(world):
        prob = AttnProblem(b, h, hk, r, pm, causal, window, scale, softclamp)
        q = qs[r].contiguous()
        if hopwise:
            hops = prob.kv_owners()
            o, lse = forward_hops(ops, prob, q, hops, lambda s: bufs[hops[s]][hops[s]], kbits)
        else:
            ready = torch.zeros(world, dtype=torch.int32, device=dev)
            peers = [bufs[o][o].data_ptr() for o in range(world)]  # owner o's own slot
            o, lse = fused_attn_fwd(prob, q, bufs[r], peers, ready, kbits)
        outs.append(o)
        lses.append(lse)
    return outs, lses


def pad64(n: int) -> int:
    return (n + 63) // 64 * 64


def alloc_qdo_buffer(world: int, batch: int, heads: int, n_q: int, d: int, dtype, device) -> torch.Tensor:
    return torch.empty(world, 2, batch * heads, n_q, d, dtype=dtype, device=device)


def alloc_stat_buffer(world: int, batch: int, heads: int, n_q: int, device) -> torch.Tensor:
    return torch.zeros(world, 2, batch * heads, pad64(n_q), dtype=torch.float32, device=device)


def fused_attn_bwd(prob: AttnProblem, qdo_buf: torch.Tensor, kv_buf: torch.Tensor, stat_buf: torch.Tensor,
                   kmask_bits: Optional[torch.Tensor] = None):
    """Run both backward kernels on already gathered buffers; returns (dq, dk, dv)."""
    ops = _ext.ops()
    dq = ops.attn_bwd_dq(qdo_buf, kv_buf, stat_buf, None, 0, *prob.tail(prob.kv_owners(), kmask_bits))
    dk, dv = ops.attn_bwd_dkdv(qdo_buf, kv_buf, stat_buf, None, 0, *prob.tail(prob.q_owners(), kmask_bits))
    return dq, dk, dv


def pad128(n: int) -> int:
    return (n + 127) // 128 * 128


def fused_attn_bwd_ring(
    prob: AttnProblem,
    qdo: torch.Tensor,
    stat: torch.Tensor,
    kv_buf: torch.Tensor,
    kmask_bits: Optional[torch.Tensor] = None,
    *,
    dq_acc: Optional[torch.Tensor] = None,
    dkv_acc_ptrs: Sequence[int] = (),
    nk_pad: int = 0,
    ready: Optional[torch.Tensor] = None,
    ready_target: int = 0,
):
    """The one-kernel (5-GEMM) backward over every owner's K/V, head dim 128 (``csrc/attn_bwd_fused_sm100.cu``).

    ``qdo`` [2, b*h, n_q, d] / ``stat`` [2, b*h, n_pad] are this rank's ``bwd_prep`` output, ``kv_buf`` the K/V gather
    (slot o usable once ``ready[o] >= ready_target``; no flags: all usable).
    dQ (unscaled) is added into ``dq_acc`` (fp32 [b*h, n_pad, d], allocated zeroed when not given).  Without
    ``dkv_acc_ptrs`` dK / dV come back as 16-bit tensors; with them (one fp32 [2, b*hk, nk_pad, d] accumulator address
    per ring rank) the kernel adds its tiles into the owners' accumulators and returns empty tensors.
    Returns (dq_acc, dk, dv)."""
    if dq_acc is None:
        dq_acc = torch.zeros(prob.batch * prob.heads, stat.shape[-1], kv_buf.shape[-1], dtype=torch.float32,
                             device=kv_buf.device)
    dk, dv = _ext.ops().attn_bwd_ring(qdo, kv_buf, stat, dq_acc, ready, int(ready_target), list(dkv_acc_ptrs),
                                      int(nk_pad), *prob.tail(prob.kv_owners(), kmask_bits))
    return dq_acc, dk, dv


def backward_hops(ops, prob: AttnProblem, qdo: torch.Tensor, stat: torch.Tensor, dq_acc: torch.Tensor,
                  hops: Sequence[int], slot: Callable[[int], torch.Tensor], *, dkv_acc_ptrs: Sequence[int],
                  nk_pad: int, kmask_bits: Optional[torch.Tensor] = None, launched: Callable[[int], None] = _no_hook):
    """The one-kernel backward one ring hop per launch (``memory="ring"``): hop ``s`` runs against ``slot(s)``, owner
    ``hops[s]``'s K/V ``[2, b*hk, n_k, d]``; ``launched(s)`` follows each launch.  dQ adds up in ``dq_acc``, dK / dV
    in the owners' accumulators ``dkv_acc_ptrs``, across the launches."""
    for s, owner in enumerate(hops):
        ops.attn_bwd_ring(qdo, slot(s)[None], stat, dq_acc, None, 0, list(dkv_acc_ptrs), int(nk_pad),
                          *prob.tail([owner], kmask_bits))
        launched(s)


def two_kernel_backward_hops(ops, prob: AttnProblem, qdo_own: torch.Tensor, stat_own: torch.Tensor,
                             kv_slot: Callable[[int], torch.Tensor],
                             qdo_slot: Callable[[int], Tuple[torch.Tensor, torch.Tensor]],
                             kmask_bits: Optional[torch.Tensor] = None, launched: Callable[[int], None] = _no_hook):
    """The two-kernel backward one ring hop per launch (``memory="ring"``).  Returns (dq, dk, dv).

    Step ``s`` launches dQ hop ``s``: this rank's ``qdo_own`` [2, b*h, n_q, d] / ``stat_own`` [2, b*h, n_pad] against
    ``kv_slot(s)``, the K/V [2, b*hk, n_k, d] of ``prob.kv_owners()[s]``; then dK/dV hop ``s``: this rank's K/V
    (``kv_slot(0)``) against ``qdo_slot(s)``, the (Q/dO, stat) pair of ``prob.q_owners()[s]``.  A step past the end of
    one list launches only the other kernel.  ``launched(s)`` follows the launches of step ``s``.

    The fp32 accumulators travel between the launches in carry buffers, and each launch reloads them into TMEM before
    its first MMA: the launches add the same products in the same order as one launch over every hop, so dQ (and dK /
    dV without grouped heads) come out bitwise equal to the gather mode."""
    kv_hops, q_hops = prob.kv_owners(), prob.q_owners()
    b, h, hk = prob.batch, prob.heads, prob.kv_heads
    kv_own = kv_slot(0)
    n_q, d = qdo_own.shape[2], qdo_own.shape[3]
    n_k = kv_own.shape[2]
    dev = qdo_own.device
    none = torch.empty(0, dtype=torch.float32, device=dev)  # a single launch carries nothing
    dq_carry = torch.empty(b, n_q, h, d, dtype=torch.float32, device=dev) if len(kv_hops) > 1 else none
    dkv_carry = torch.empty(2, b, n_k, hk, d, dtype=torch.float32, device=dev) if len(q_hops) > 1 else none
    for s in range(max(len(kv_hops), len(q_hops))):
        if s < len(kv_hops):
            kv = kv_own if s == 0 else kv_slot(s)
            dq = ops.attn_bwd_dq_hop(qdo_own[None], kv[None], stat_own[None], dq_carry, s > 0, s + 1 < len(kv_hops),
                                     *prob.tail([kv_hops[s]], kmask_bits))
        if s < len(q_hops):
            qdo, stat = qdo_slot(s)
            dk, dv = ops.attn_bwd_dkdv_hop(qdo[None], kv_own[None], stat[None], dkv_carry, s > 0, s + 1 < len(q_hops),
                                           *prob.tail([q_hops[s]], kmask_bits))
        launched(s)
    return dq, dk, dv


def emulate_ring_backward(
    qs, ks, vs, outs, lses, douts, *,
    layout: str = "plain",
    causal: bool = False,
    window: Optional[int] = None,
    softclamp: float = 0.0,
    key_masks=None,
    scale: Optional[float] = None,
    fused: Optional[bool] = None,
    hopwise: bool = False,
):
    """Backward of :func:`emulate_ring_forward` for every emulated rank on the current device.
    ``hopwise``: one launch per hop (and per kernel of the two-kernel pair) against one-slot views of the gathered
    buffers (the ``memory="ring"`` schedule).

    ``fused`` (default: head dim 128) selects the one-kernel backward: every emulated rank adds its dK / dV tiles into
    the owners' fp32 accumulators, exactly what the ranks of a real ring do over NVLink."""
    ops = _ext.ops()
    world = len(qs)
    b, n, h, d = qs[0].shape
    hk = ks[0].shape[2]
    dev, dt = qs[0].device, qs[0].dtype
    pm = make_position_map(layout, world, n)
    scale = d ** -0.5 if scale is None else scale
    kv_all = alloc_kv_buffer(world, b, hk, n, d, dt, dev)
    qdo_all = alloc_qdo_buffer(world, b, h, n, d, dt, dev)
    stat_all = alloc_stat_buffer(world, b, h, n, dev)
    for r in range(world):
        ops.pack_kv(ks[r], vs[r], kv_all[r])
        ops.bwd_prep(qs[r].contiguous(), outs[r].contiguous(), douts[r].contiguous(), lses[r].contiguous(), qdo_all,
                     stat_all, r)
    kbits = None
    if key_masks is not None:
        kbits = pack_key_mask_bits(torch.stack(list(key_masks), 0))
    if fused is None:
        fused = d == 128
    res = []
    if fused:
        nk_pad = pad128(n)
        ring = world > 1
        accs = [torch.zeros(2, b * hk, nk_pad, d, dtype=torch.float32, device=dev) for _ in range(world)] if ring else []
        ptrs = [a.data_ptr() for a in accs]
        dqs, direct = [], []
        for r in range(world):
            prob = AttnProblem(b, h, hk, r, pm, causal, window, scale, softclamp)
            if hopwise and ring:
                hops = prob.kv_owners()
                dq_acc = torch.zeros(b * h, stat_all.shape[-1], d, dtype=torch.float32, device=dev)
                backward_hops(ops, prob, qdo_all[r], stat_all[r], dq_acc, hops, lambda s: kv_all[hops[s]],
                              dkv_acc_ptrs=ptrs, nk_pad=nk_pad, kmask_bits=kbits)
                dk = dv = None
            else:
                dq_acc, dk, dv = fused_attn_bwd_ring(prob, qdo_all[r], stat_all[r], kv_all, kbits, dkv_acc_ptrs=ptrs,
                                                     nk_pad=nk_pad)
            dqs.append(dq_acc)
            direct.append((dk, dv))
        for r in range(world):
            dq = torch.empty(b, n, h, d, dtype=dt, device=dev)
            ops.acc_convert(dqs[r], dq, scale)
            if ring:
                dk = torch.empty(b, n, hk, d, dtype=dt, device=dev)
                dv = torch.empty_like(dk)
                ops.acc_convert(accs[r][0], dk, 1.0)
                ops.acc_convert(accs[r][1], dv, 1.0)
            else:
                dk, dv = direct[r]
            res.append((dq, dk, dv))
        return res
    for r in range(world):
        prob = AttnProblem(b, h, hk, r, pm, causal, window, scale, softclamp)
        if hopwise:
            kv_hops, q_hops = prob.kv_owners(), prob.q_owners()
            res.append(two_kernel_backward_hops(ops, prob, qdo_all[r], stat_all[r], lambda s: kv_all[kv_hops[s]],
                                                lambda s: (qdo_all[q_hops[s]], stat_all[q_hops[s]]), kbits))
        else:
            # every emulated rank sees the same fully gathered buffers (what the NVLink gather produces)
            res.append(fused_attn_bwd(prob, qdo_all, kv_all, stat_all, kbits))
    return res
