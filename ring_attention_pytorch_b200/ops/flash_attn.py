"""Single-hop flash-attention building blocks with carried state.

Counterpart of the reference's Triton host wrappers ``flash_attn_forward`` / ``flash_attn_backward``
(reference triton_flash_attn.py:304-430, 988-1128): the same positional signatures, the same carried
``(o, m, lse)`` contract between hops, the same "gradients are written into the buffers you pass" contract
for the backward.  They exist for users who drive their own hop loop (the reference's ring op does,
ring_flash_attention_cuda.py:136-186 / 271-337); the ring ops of this package do *not* use them — they run
every hop inside one kernel and never spill the accumulator.

On a B200 with 16-bit inputs and no bias (or a key-padding bias, the only kind the reference ring op ever
builds, ring_flash_attention_cuda.py:147-148) one hop is one launch of the sm_100a forward kernel
(``torch.ops.rab.attn_fwd``) or of the two backward kernels; the merge of the hop into the carried state is
the max-rescale identity in fp32.  Everything else (CPU tensors, fp32, arbitrary additive bias matrices)
takes a dense fp32 PyTorch path with identical semantics, which is also the oracle of the unit tests.

Carried-state contract (identical to the reference): ``o`` is the un-normalised accumulator relative to the
running reference ``m``; ``lse`` is the running log-sum-exp; ``o * exp(m - lse)`` is the attention output.
Unlike the reference, ``o`` may be an fp32 buffer — pass one to avoid its 16-bit round trip between hops
(SURVEY D11).  Differences kept on purpose: grouped-query K/V (``hk`` dividing ``h``) are accepted, fully
masked rows give 0 instead of NaN, and dK/dV of a hop are exact.
"""
from __future__ import annotations

from math import ceil
from typing import Optional, Tuple

import torch
import torch.nn.functional as F
from torch import Tensor

from ring_attention_pytorch_b200.ops.oracle import expand_kv_heads, softclamp
from ring_attention_pytorch_b200.parallel.layout import make_position_map

NEG_MAX = -torch.finfo(torch.float32).max
_MASKED_BELOW = -1e30  # bias / lse values below this mean "masked" / "nothing accumulated yet"


def _rounded(n: int) -> int:
    return ceil(n / 128) * 128


def _key_keep_from_bias(bias: Optional[Tensor], batch: int, seqlen_k: int) -> Tuple[Optional[Tensor], bool]:
    """Return (keep [b, j] bool | None, is_pure_key_padding)."""
    if bias is None:
        return None, True
    vec = None
    if bias.ndim == 2 and bias.shape == (batch, seqlen_k):
        vec = bias
    elif bias.ndim == 4 and bias.shape[1:3] == (1, 1) and bias.shape[-1] == seqlen_k:
        vec = bias[:, 0, 0].expand(batch, seqlen_k)
    if vec is None:
        return None, False
    keep = vec > _MASKED_BELOW
    pure = bool(((vec == 0) | ~keep).all().item())
    return keep, pure


def _visible(seqlen_q: int, seqlen_k: int, causal: bool, strict: bool, device) -> Optional[Tensor]:
    if not causal:
        return None
    i = torch.arange(seqlen_q, device=device)[:, None]
    j = torch.arange(seqlen_k, device=device)[None, :]
    return (i > j) if strict else (i >= j)  # top-left aligned, triton_flash_attn.py:216-221


def _dense_logits(q, k, bias, causal, strict, scale, clamp):
    b, n_q, h, _ = q.shape
    n_k = k.shape[1]
    sim = torch.einsum("bihd,bjhd->bhij", q.float(), expand_kv_heads(k, h).float()) * scale
    if clamp > 0:
        sim = softclamp(sim, clamp)
    vis = torch.ones(b, 1, n_q, n_k, dtype=torch.bool, device=q.device)
    if bias is not None:
        bias4 = bias[:, None, None, :] if bias.ndim == 2 else bias
        bias4 = bias4.float()
        vis = vis & (bias4 > _MASKED_BELOW)
        sim = sim + bias4.clamp(min=_MASKED_BELOW)
    cm = _visible(n_q, n_k, causal, strict, q.device)
    if cm is not None:
        vis = vis & cm[None, None]
    return sim, vis.expand_as(sim)


def _dense_hop_forward(q, k, v, bias, causal, strict, scale, clamp):
    """-> (o normalised fp32 [b, n, h, d], lse fp32 [b, h, n] with NEG_MAX for rows that saw no key)."""
    sim, vis = _dense_logits(q, k, bias, causal, strict, scale, clamp)
    sim = sim.masked_fill(~vis, NEG_MAX)
    any_vis = vis.any(-1)
    m = sim.amax(-1, keepdim=True)
    p = (sim - m).exp().masked_fill(~vis, 0.0)
    l = p.sum(-1, keepdim=True)
    attn = p / l.clamp(min=torch.finfo(torch.float32).tiny)
    o = torch.einsum("bhij,bjhd->bihd", attn, expand_kv_heads(v, q.shape[2]).float())
    lse = torch.where(any_vis, (m + l.clamp(min=torch.finfo(torch.float32).tiny).log()).squeeze(-1),
                      torch.full_like(m.squeeze(-1), NEG_MAX))
    return o, lse


def _use_kernel(q: Tensor, pure_key_padding: bool) -> bool:
    return q.is_cuda and q.dtype in (torch.bfloat16, torch.float16) and pure_key_padding and q.shape[-1] <= 128


def _pad_d(t: Tensor, d_pad: int) -> Tensor:
    return t if t.shape[-1] == d_pad else F.pad(t, (0, d_pad - t.shape[-1]))


def _kernel_hop_forward(q, k, v, keep, causal, strict, scale, clamp):
    from ring_attention_pytorch_b200.ops import _ext
    from ring_attention_pytorch_b200.ops.fused import AttnProblem, alloc_kv_buffer, fused_attn_fwd, pack_key_mask_bits

    ops = _ext.ops()
    b, n_q, h, d = q.shape
    n_k, hk = k.shape[1], k.shape[2]
    d_pad = 64 if d <= 64 else 128
    qp, kp, vp = (_pad_d(t, d_pad).contiguous() for t in (q, k, v))
    kv = alloc_kv_buffer(1, b, hk, n_k, d_pad, q.dtype, q.device)
    ops.pack_kv(kp, vp, kv[0])
    ready = torch.zeros(1, dtype=torch.int32, device=q.device)
    kbits = pack_key_mask_bits(keep[None]) if keep is not None else None
    pm = make_position_map("plain", 1, n_k)
    # strict causal (diagonal masked) == causal with every query position shifted down by one
    prob = AttnProblem(b, h, hk, 0, pm, causal, None, scale, clamp, q_pos_offset=-1 if (causal and strict) else 0)
    o, lse = fused_attn_fwd(prob, qp, kv, [0], ready, kbits)
    lse = torch.where(torch.isinf(lse), torch.full_like(lse, NEG_MAX), lse)
    return o[..., :d].float(), lse


def flash_attn_forward(
    q: Tensor,
    k: Tensor,
    v: Tensor,
    bias: Optional[Tensor] = None,
    causal: bool = False,
    o: Optional[Tensor] = None,
    m: Optional[Tensor] = None,
    lse: Optional[Tensor] = None,
    softmax_scale: Optional[float] = None,
    causal_mask_diagonal: bool = False,
    return_normalized_output: bool = False,
    load_accumulated: bool = True,
    softclamp_qk_sim: bool = False,
    softclamp_value: float = 50.0,
    head_first_dim: bool = False,
    remove_padding: bool = False,
):
    """One hop of flash attention merged into the carried ``(o, m, lse)``; returns ``(o, m, lse)``.

    q ``[b, n, h, d]``, k / v ``[b, j, hk, d]`` (``[b, h, n, d]`` when ``head_first_dim``); ``bias`` is an additive
    bias ``[b, j]`` (key padding: 0 keep / very negative drop), ``[b, 1, 1, j]`` or ``[b, h, n, j]``;
    ``causal_mask_diagonal`` masks the diagonal as well (striped ring hops from a later rank,
    reference ring_flash_attention_cuda.py:157-160).  ``m`` / ``lse`` are ``[b, h, ceil(n / 128) * 128]`` fp32
    (sliced to ``n`` with ``remove_padding``).  Buffers that are passed in are updated in place.
    """
    if head_first_dim:
        q, k, v = (t.transpose(1, 2) for t in (q, k, v))
        if o is not None:
            o = o.transpose(1, 2)
    b, n_q, h, d = q.shape
    n_k = k.shape[1]
    assert k.shape[0] == b and v.shape == k.shape and h % k.shape[2] == 0 and k.shape[-1] == d
    scale = d ** -0.5 if softmax_scale is None else float(softmax_scale)
    clamp = float(softclamp_value) if softclamp_qk_sim else 0.0
    nr = _rounded(n_q)

    keep, pure = _key_keep_from_bias(bias, b, n_k)
    if _use_kernel(q, pure):
        o_hop, lse_hop = _kernel_hop_forward(q, k, v, keep, causal, causal_mask_diagonal, scale, clamp)
    else:
        o_hop, lse_hop = _dense_hop_forward(q, k, v, bias, causal, causal_mask_diagonal, scale, clamp)

    def stat(buf):
        if buf is None or not load_accumulated:
            fresh = torch.full((b, h, nr), NEG_MAX, device=q.device, dtype=torch.float32)
            if buf is not None:
                buf.copy_(fresh[..., :buf.shape[-1]])
                return buf
            return fresh
        return buf

    m, lse = stat(m), stat(lse)
    if o is None:
        o = torch.zeros_like(q)
    elif not load_accumulated:
        o.zero_()

    m_old, lse_old = m[..., :n_q], lse[..., :n_q]
    m_new = torch.maximum(m_old, lse_hop)
    lse_new = torch.logaddexp(lse_old, lse_hop)
    w_old = (m_old - m_new).exp().transpose(1, 2).unsqueeze(-1)   # [b, n, h, 1]
    w_hop = (lse_hop - m_new).exp().transpose(1, 2).unsqueeze(-1)
    acc = o.float() * w_old + o_hop * w_hop
    if return_normalized_output:
        acc = acc * (m_new - lse_new).exp().transpose(1, 2).unsqueeze(-1)
    o.copy_(acc)
    m[..., :n_q] = m_new
    lse[..., :n_q] = lse_new

    if head_first_dim:
        o = o.transpose(1, 2)
    if remove_padding:
        m, lse = m[..., :n_q], lse[..., :n_q]
    return o, m, lse


def _dense_hop_backward(do, q, k, v, o, lse, bias, causal, strict, scale, clamp):
    h, hk = q.shape[2], k.shape[2]
    sim, vis = _dense_logits(q, k, bias, causal, strict, scale, clamp)
    lse_q = torch.where(lse <= _MASKED_BELOW, torch.full_like(lse, float("inf")), lse)
    p = (sim - lse_q.unsqueeze(-1)).exp().masked_fill(~vis, 0.0)
    dof = do.float()
    delta = (o.float() * dof).sum(-1).transpose(1, 2)              # [b, h, n]
    vx, kx = expand_kv_heads(v, h).float(), expand_kv_heads(k, h).float()
    dv = torch.einsum("bhij,bihd->bjhd", p, dof)
    dp = torch.einsum("bihd,bjhd->bhij", dof, vx)
    ds = p * (dp - delta.unsqueeze(-1))
    if clamp > 0:
        raw = torch.einsum("bihd,bjhd->bhij", q.float(), kx) * scale
        ds = ds * (1.0 - (raw / clamp).tanh() ** 2)
    ds = ds * scale
    dq = torch.einsum("bhij,bjhd->bihd", ds, kx)
    dk = torch.einsum("bhij,bihd->bjhd", ds, q.float())
    if hk != h:  # query head j reads kv head j % hk
        b, n_k, _, d = dk.shape
        dk = dk.view(b, n_k, h // hk, hk, d).sum(2)
        dv = dv.view(b, n_k, h // hk, hk, d).sum(2)
    return dq, dk, dv, delta


def _kernel_hop_backward(do, q, k, v, o, lse, keep, causal, strict, scale, clamp):
    from ring_attention_pytorch_b200.ops import _ext
    from ring_attention_pytorch_b200.ops.fused import (AttnProblem, alloc_kv_buffer, alloc_qdo_buffer,
                                                       alloc_stat_buffer, fused_attn_bwd, pack_key_mask_bits)

    ops = _ext.ops()
    b, n_q, h, d = q.shape
    n_k, hk = k.shape[1], k.shape[2]
    d_pad = 64 if d <= 64 else 128
    dt = q.dtype
    qp, kp, vp, op, dop = (_pad_d(t.to(dt), d_pad).contiguous() for t in (q, k, v, o, do))
    kv = alloc_kv_buffer(1, b, hk, n_k, d_pad, dt, q.device)
    ops.pack_kv(kp, vp, kv[0])
    qdo = alloc_qdo_buffer(1, b, h, n_q, d_pad, dt, q.device)
    stat = alloc_stat_buffer(1, b, h, n_q, q.device)
    lse_k = torch.where(lse <= _MASKED_BELOW, torch.full_like(lse, float("inf")), lse).contiguous()
    ops.bwd_prep(qp, op, dop, lse_k, qdo, stat, 0)
    kbits = pack_key_mask_bits(keep[None]) if keep is not None else None
    pm = make_position_map("plain", 1, n_k)
    prob = AttnProblem(b, h, hk, 0, pm, causal, None, scale, clamp, q_pos_offset=-1 if (causal and strict) else 0)
    dq, dk, dv = fused_attn_bwd(prob, qdo, kv, stat, kbits)
    delta = stat[0, 1].view(b, h, -1)[..., :n_q]
    return dq[..., :d], dk[..., :d], dv[..., :d], delta


def flash_attn_backward(
    do: Tensor,
    q: Tensor,
    k: Tensor,
    v: Tensor,
    o: Tensor,
    lse: Tensor,
    dq: Tensor,
    dk: Tensor,
    dv: Tensor,
    delta: Optional[Tensor] = None,
    bias: Optional[Tensor] = None,
    causal: bool = False,
    causal_mask_diagonal: bool = False,
    softmax_scale: Optional[float] = None,
    softclamp_qk_sim: bool = False,
    softclamp_value: float = 50.0,
) -> Tensor:
    """Gradients of one hop: ``o`` and ``lse`` are the FINAL normalised output and log-sum-exp of the whole ring,
    ``k`` / ``v`` the hop's keys and values.  Overwrites ``dq``, ``dk``, ``dv`` with this hop's contributions (the
    caller accumulates across hops, as the reference does at ring_flash_attention_cuda.py:335-337) and returns
    ``delta = rowsum(o * do)`` as ``[b, h, ceil(n / 128) * 128]`` fp32.  ``delta`` may be passed for signature
    parity; it is recomputed (it is fused into the backward's prep kernel here)."""
    b, n_q, h, d = q.shape
    n_k = k.shape[1]
    scale = d ** -0.5 if softmax_scale is None else float(softmax_scale)
    clamp = float(softclamp_value) if softclamp_qk_sim else 0.0
    lse_n = lse[..., :n_q]
    keep, pure = _key_keep_from_bias(bias, b, n_k)
    if _use_kernel(q, pure):
        g = _kernel_hop_backward(do, q, k, v, o, lse_n, keep, causal, causal_mask_diagonal, scale, clamp)
    else:
        g = _dense_hop_backward(do, q, k, v, o, lse_n, bias, causal, causal_mask_diagonal, scale, clamp)
    dq.copy_(g[0])
    dk.copy_(g[1])
    dv.copy_(g[2])
    out = torch.zeros(b, h, _rounded(n_q), device=q.device, dtype=torch.float32)
    out[..., :n_q] = g[3]
    return out
