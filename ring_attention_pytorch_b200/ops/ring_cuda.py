"""Ring flash attention on the sm_100a kernels (autograd Function + reference-compatible wrapper).

Public surface mirrors reference ring_flash_attention_cuda.py:353-371 (``ring_flash_attn_cuda`` /
``ring_flash_attn_cuda_``) plus a ``layout`` argument ('plain' | 'striped' | 'zigzag').

Forward, per rank (no host synchronisation, no NCCL on the hot path), ``CONFIG["memory"]``:

``"ring"`` (what the default ``"auto"`` picks for K/V slots >= 256 MiB per rank) — O(n / W) workspace, like the reference's send/recv ring (ring_flash_attention_cuda.py:128-178):

    pack_kv (K,V -> head-major) into this rank's own SYMMETRIC slot -> device barrier -> one tcgen05 flash-attention
    launch per ring hop; hop 0 reads the own slot in place, hop s reads a 2-slot window that the COPY ENGINES fill up
    to two hops ahead over NVLink (side stream, events); the un-normalised O / running max / running sum travel between
    the launches in fp32 buffers (in TMEM inside a launch)

``"gather"`` (``"auto"`` for short shards) — one launch per rank for the whole ring:

    pack_kv straight into this rank's slot of a W-slot symmetric gather workspace -> device barrier -> ONE fused
    kernel: flash attention over every hop while its fetcher warps pull the other ranks' K/V slots over NVLink
    (bulk TMA) into the local gather buffer; O / max / sum never leave TMEM and registers

Measured at the headline config (S=262144, h=32, fwd+bwd): same box, back to back, 2 GPUs: 1656 ("ring") vs 1646
("gather") TFLOP/s, i.e. on par; 8 GPUs: 6369 ("ring") against 6174 ("gather", measured earlier in the round on another
box, so inside box-to-box variation).  What "ring" buys is memory: S = 4 194 304 on 8 GPUs runs (96 GB per GPU) where the
W-slot gather alone would need 137 GB.  At short shards the extra launches cost (see ``CONFIG`` below).

Only q, k, v, o and the log-sum-exp are saved for the backward (O(n / W) activation memory per layer; the reference
saves the same, ring_flash_attention_cuda.py:188-198).  The workspaces are transient and shared by all layers.

Backward, head dim 128 (``CONFIG["backward"] = "fused"``):

    bwd_prep (delta, lse -> log2, Q/dO head-major) -> pack_kv into the own slot, zero the fp32 accumulators
    -> device barrier -> the one-kernel backward (5 GEMMs per tile pair, dQ added into a local fp32 accumulator by TMA
    reduction, dK/dV tiles added into their OWNER's fp32 accumulators over NVLink from the kernel's epilogue), launched
    once per hop against the 2-slot window ("ring") or once over the gathered slots, which the copy engines re-pull
    behind per-owner flags ("gather") -> device barrier -> fp32 -> 16 bit

Head dim 64 (or ``CONFIG["backward"] = "two_kernel"``): dQ kernel + dK/dV kernel (7 GEMMs, no atomics, deterministic).

    "ring": bwd_prep writes Q / dO / statistics straight into this rank's own symmetric slot, pack_kv re-packs the own
    K/V slot -> device barrier -> per ring hop one dQ launch (local queries against the K/V of the hop's owner) and one
    dK/dV launch (local keys against the Q / dO / statistics of the hop's query owner), each against a 2-slot window
    that the copy engines fill ahead; the fp32 dQ and dK / dV accumulators travel between the launches in carry buffers
    and are reloaded into TMEM, so the result is bitwise that of the one-launch backward (dK / dV with grouped heads:
    same sums, another order)
    "gather": the peers' K/V and Q / dO / statistics gathered into W-slot buffers by the copy engines while the dQ
    kernel runs
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.distributed as dist
import torch.nn.functional as F
from torch import Tensor
from torch.autograd import Function

from ring_attention_pytorch_b200.ops import _ext
from ring_attention_pytorch_b200.ops.fused import (
    AttnProblem,
    alloc_kv_buffer,
    alloc_qdo_buffer,
    alloc_stat_buffer,
    backward_hops,
    forward_hops,
    fused_attn_bwd_ring,
    fused_attn_fwd,
    pack_key_mask_bits,
    pad64,
    pad128,
    two_kernel_backward_hops,
)
from ring_attention_pytorch_b200.parallel.distributed import default, exists, get_rank, get_world_size, is_distributed
from ring_attention_pytorch_b200.parallel.layout import make_position_map
from ring_attention_pytorch_b200.parallel.symm import get_workspace
from ring_attention_pytorch_b200.utils.timing import nvtx_range
from ring_attention_pytorch_b200.utils.validate import check_attention_inputs, typecheck

# counts launches of our own kernels (bench.py reports it as gpu_launches)
LAUNCHES = {"count": 0}

# backward="fused"     : head dim 128 runs the whole backward in ONE KV-stationary kernel (5 GEMMs; dQ through fp32 TMA
#                        reductions, dK/dV added into the owner's accumulators over NVLink).
# backward="two_kernel": the dQ + dK/dV kernel pair (7 GEMMs, no atomics, deterministic); head dim 64 always uses it.
# memory="ring"        : one launch per ring hop against a 2-slot window that the copy engines fill ahead of the
#                        kernels; the online-softmax state (forward) and the fp32 accumulators (both backwards, every
#                        head dim) carry over between the launches.  Workspace O(n / W) per rank; on par with "gather"
#                        at the headline size (see the module docstring).
# memory="gather"      : one forward launch per rank; its fetcher warps pull all W-1 peer slots into a W-slot gather
#                        buffer (transient, shared by all layers); workspace O(n) per rank.  Fewer launches: better for
#                        short shards, where the one-kernel backward's per-launch ramp shows (8 hops x 8192 keys, h=16:
#                        726 vs 826 TFLOP/s).
# memory="auto"        : "ring" when one rank's K/V slot is at least AUTO_RING_SLOT_BYTES, else "gather".  Measured on 2
#                        GPUs: 128 MiB slots (S=16384, h=32) ring 1441 vs gather 1546 TFLOP/s — ~90 us of ramp per extra
#                        launch against 5 ms steps; 2 GiB slots (S=262144) 1656 vs 1646 (same box, back to back).
AUTO_RING_SLOT_BYTES = 256 << 20
CONFIG = {"backward": "fused", "memory": "auto"}


def _use_hop_window(slot_bytes: int) -> bool:
    mode = CONFIG["memory"]
    assert mode in ("auto", "ring", "gather"), mode
    return mode == "ring" or (mode == "auto" and slot_bytes >= AUTO_RING_SLOT_BYTES)


def _count(n: int = 1) -> None:
    LAUNCHES["count"] += n


def _pad_head_dim(t: Tensor, d_pad: int) -> Tensor:
    d = t.shape[-1]
    return t if d == d_pad else F.pad(t, (0, d_pad - d))


def _gather_ring_masks(mask: Tensor, ring_size: int) -> Tensor:
    """[b, n] bool on every rank -> [ring, b, n] for this rank's ring set (cold path, NCCL)."""
    world = get_world_size()
    gathered = [torch.empty_like(mask, dtype=torch.uint8) for _ in range(world)]
    dist.all_gather(gathered, mask.to(torch.uint8).contiguous())
    ring_set = get_rank() // ring_size
    return torch.stack(gathered[ring_set * ring_size:(ring_set + 1) * ring_size]).bool()


def _slot_bytes(b, hk, n_k, d_pad) -> int:
    """Bytes of one owner's K/V slot ``[2, b*hk, n_k, d]`` (16 bit)."""
    return 2 * b * hk * n_k * d_pad * 2


def _ring_gather_workspace(ws, ring_size, b, hk, n_k, d_pad, dt):
    """This call's K/V gather buffer ``[W, 2, b*hk, n_k, d]`` inside the symmetric workspace (double buffered across
    calls) and, per ring rank, the address of THAT rank's own slot in ITS buffer (what the fetchers pull from)."""
    slot_bytes = _slot_bytes(b, hk, n_k, d_pad)
    local, bases = ws.staging("kv_gather", ring_size * slot_bytes)
    gather = local[:ring_size * slot_bytes].view(dt).view(ring_size, 2, b * hk, n_k, d_pad)
    own_slot_ptrs = [bases[o] + o * slot_bytes for o in range(ring_size)]
    return gather, own_slot_ptrs, slot_bytes


def _own_slot_workspace(ws, b, hk, n_k, d_pad, dt):
    """``memory="ring"``: this rank's own K/V slot ``[2, b*hk, n_k, d]`` in symmetric memory (double buffered across
    calls) and every ring rank's address of ITS slot."""
    slot_bytes = _slot_bytes(b, hk, n_k, d_pad)
    local, bases = ws.staging("kv_own", slot_bytes)
    return local[:slot_bytes].view(dt).view(2, b * hk, n_k, d_pad), bases, slot_bytes


def _place_kv(ws, hop_mode: bool, rank: int, ring_size: int, b, hk, n_k, d_pad, dt, dev):
    """Where this rank packs its K/V and what the kernels read it through: ``(target, kv_buf, own_ptrs, slot_bytes)``.

    ``target`` is the ``[2, b*hk, n_k, d]`` slot to pack into; ``own_ptrs[o]`` is ring rank o's address of ITS own
    slot, what the peers pull from.
      hop mode (``memory="ring"``): this rank's own symmetric slot; ``kv_buf`` is None (the kernels read a _HopWindow)
      gather: slot ``rank`` of the W-slot symmetric gather buffer ``kv_buf``
      single rank (``ws`` is None): slot 0 of a local 1-slot ``kv_buf``; no ``own_ptrs``"""
    if ws is None:
        kv = alloc_kv_buffer(1, b, hk, n_k, d_pad, dt, dev)
        return kv[0], kv, None, _slot_bytes(b, hk, n_k, d_pad)
    if hop_mode:
        own, own_ptrs, slot_bytes = _own_slot_workspace(ws, b, hk, n_k, d_pad, dt)
        return own, None, own_ptrs, slot_bytes
    gather, own_ptrs, slot_bytes = _ring_gather_workspace(ws, ring_size, b, hk, n_k, d_pad, dt)
    return gather[rank], gather, own_ptrs, slot_bytes


class _HopWindow:
    """Two local K/V slots that the copy engines fill up to two hops ahead of the kernel that reads them.

    Hop 0 reads this rank's own slot in place; hop s >= 1 reads ``win[(s - 1) % 2]``, pulled from its owner's symmetric slot
    on the side stream.  Everything is stream ordered (events), nothing blocks the host.  Create it after the device
    barrier that publishes the peers' slots."""

    def __init__(self, ops, ws, own: Tensor, own_ptrs, slot_bytes: int, hops):
        dev = own.device
        self.ops, self.own, self.own_ptrs, self.slot_bytes, self.hops = ops, own, own_ptrs, slot_bytes, list(hops)
        self.main, self.side = torch.cuda.current_stream(dev), ws.side_stream
        self.win = torch.empty((min(2, max(len(self.hops) - 1, 0)),) + tuple(own.shape), dtype=own.dtype, device=dev)
        self.copied = {}
        start = torch.cuda.Event()
        start.record(self.main)
        self._prefetch(1, start)
        self._prefetch(2, start)

    def _prefetch(self, s: int, after) -> None:
        if s >= len(self.hops):
            return
        with torch.cuda.stream(self.side):
            self.side.wait_event(after)
            self.ops.peer_copy(self.win[(s - 1) % 2], self.own_ptrs[self.hops[s]], self.slot_bytes)
            ev = torch.cuda.Event()
            ev.record(self.side)
        self.copied[s] = ev

    def slot(self, s: int) -> Tensor:
        if s == 0:
            return self.own
        self.main.wait_event(self.copied.pop(s))
        return self.win[(s - 1) % 2]

    def launched(self, s: int) -> None:
        """The kernel of hop ``s`` is enqueued: once it finishes its slot is free for hop s + 2."""
        if s >= 1 and s + 2 < len(self.hops):
            done = torch.cuda.Event()
            done.record(self.main)
            self._prefetch(s + 2, done)


def _pack_slot(ops, k: Tensor, v: Tensor, slot: Tensor, angles: Optional[Tensor]) -> None:
    """K, V [b, n, hk, d] -> head-major slot [2, b*hk, n, d]; with ``angles`` K is rotated on the way in."""
    if angles is None:
        ops.pack_kv(k, v, slot, 3)
    else:
        ops.rotary(k, angles, slot[0], True, 1.0)
        ops.pack_kv(k, v, slot, 2)  # V half only


class RingFlashAttentionCUDAFunction(Function):
    @staticmethod
    def forward(
        ctx,
        q: Tensor,
        k: Tensor,
        v: Tensor,
        mask: Optional[Tensor],
        causal: bool,
        bucket_size: int,
        ring_reduce_col: bool,
        striped_ring_attn: bool,
        max_lookback_seq_len: Optional[int],
        ring_size: Optional[int],
        softclamp_qk_sim: bool = False,
        softclamp_value: float = 50.0,
        layout: Optional[str] = None,
        rotary_freqs: Optional[Tensor] = None,
    ):
        assert q.is_cuda and k.is_cuda and v.is_cuda, "ring_flash_attn_cuda needs CUDA tensors"
        ops = _ext.ops()
        orig_dtype = q.dtype
        if q.dtype not in (torch.bfloat16, torch.float16):
            q, k, v = (t.to(torch.bfloat16) for t in (q, k, v))  # reference casts fp32 to fp16 (_cuda.py:72-79)
        dt = q.dtype
        k, v = k.to(dt), v.to(dt)

        ring_size = default(ring_size, get_world_size())
        cross_attn = q.shape[1] != k.shape[1]
        use_ring = bool(ring_reduce_col) and is_distributed() and not cross_attn and ring_size > 1
        layout = default(layout, "striped" if (striped_ring_attn and use_ring) else "plain")
        if not use_ring:
            layout, ring_size = "plain", 1
        assert not (exists(max_lookback_seq_len) and not causal), "look-back windows need causal attention"
        if causal:
            mask = None  # reference _cuda.py:105-106

        b, n_q, h, d = q.shape
        n_k, hk = k.shape[1], k.shape[2]
        assert h % hk == 0 and v.shape == k.shape
        assert d <= 128, "head dimension up to 128 is supported"
        d_pad = 64 if d <= 64 else 128
        scale = d ** -0.5
        # Rotary embedding (rotate-half pairs, reference ring_attention.py:160-172) is applied by the op's own pack
        # kernels: Q into its padded contiguous copy, K straight into the gather slot; the backward rotates dQ / dK back.
        ang = None
        fused_k_rotary = False
        if exists(rotary_freqs):
            assert not cross_attn and d % 16 == 0, "in-kernel rotary needs self-attention and head dim % 16 == 0"
            ang = rotary_freqs.detach().to(device=q.device, dtype=torch.float32).contiguous()
            assert ang.dim() == 2 and ang.shape[0] == n_q and ang.shape[1] >= d // 2
            q_rot = (torch.zeros if d_pad != d else torch.empty)(b, n_q, h, d_pad, dtype=dt, device=q.device)
            ops.rotary(q, ang, q_rot, False, 1.0)
            _count()
            qp = q_rot
            fused_k_rotary = d_pad == d
            if not fused_k_rotary:
                k_rot = torch.empty(b, n_k, hk, d, dtype=dt, device=q.device)
                ops.rotary(k, ang, k_rot, False, 1.0)
                _count()
                kp, vp = (_pad_head_dim(t, d_pad).contiguous() for t in (k_rot, v))
            else:
                kp, vp = k, v  # unit stride on d is all the pack kernels need
        else:
            qp, kp, vp = (_pad_head_dim(t, d_pad).contiguous() for t in (q, k, v))

        rank = get_rank() % ring_size if use_ring else 0
        pm = make_position_map(layout, ring_size, n_k)
        q_off = (n_k - n_q) if (cross_attn and causal) else 0
        softclamp = float(softclamp_value) if softclamp_qk_sim else 0.0
        prob = AttnProblem(b, h, hk, rank, pm, causal, max_lookback_seq_len, scale, softclamp, q_off)
        dev = q.device

        hop_mode = use_ring and _use_hop_window(_slot_bytes(b, hk, n_k, d_pad))
        ws = get_workspace(ring_size, dev) if use_ring else None
        with nvtx_range("rab.fwd.pack+barrier"):
            own, kv_gather, own_ptrs, slot_bytes = _place_kv(ws, hop_mode, rank, ring_size, b, hk, n_k, d_pad, dt, dev)
            _pack_slot(ops, kp, vp, own, ang if fused_k_rotary else None)
            _count()
            kbits = None
            if use_ring:
                ws.barrier()  # every peer's own slot is complete
                _count()
                if exists(mask):
                    kbits = pack_key_mask_bits(_gather_ring_masks(mask, ring_size))
            elif exists(mask):
                kbits = pack_key_mask_bits(mask[None])

        with nvtx_range("rab.fwd.kernel"):
            if hop_mode:
                hops = prob.kv_owners()
                window_slots = _HopWindow(ops, ws, own, own_ptrs, slot_bytes, hops)
                o, lse = forward_hops(ops, prob, qp, hops, window_slots.slot, kbits, window_slots.launched)
                _count(len(hops))
            else:
                ready = torch.zeros(ring_size, dtype=torch.int32, device=dev)
                peers = [0 if o_ == rank else own_ptrs[o_] for o_ in range(ring_size)] if use_ring else [0]
                o, lse = fused_attn_fwd(prob, qp, kv_gather, peers, ready, kbits)
                _count()

        ctx.prob = prob
        ctx.cfg = (ring_size, rank, use_ring, d, d_pad, orig_dtype, fused_k_rotary)
        # single rank: the packed K/V is exactly what the backward needs; ring: keep the (small) inputs, re-pack later
        none = torch.empty(0, device=dev)
        ctx.save_for_backward(qp, kp if use_ring else none, vp if use_ring else none, o, lse,
                              none if use_ring else kv_gather, kbits if kbits is not None else none,
                              ang if ang is not None else none)
        out = o[..., :d]
        return out.to(orig_dtype) if orig_dtype != dt else out

    @staticmethod
    def backward(ctx, do: Tensor):
        ops = _ext.ops()
        prob = ctx.prob
        ring_size, rank, use_ring, d, d_pad, orig_dtype, fused_k_rotary = ctx.cfg
        qp, kp, vp, o, lse, kv_saved, kbits, ang = ctx.saved_tensors
        kbits = kbits if kbits.numel() > 0 else None
        ang = ang if ang.numel() > 0 else None
        dt = qp.dtype
        b, n_q, h, _ = qp.shape
        hk = prob.kv_heads
        dev = qp.device
        dop = _pad_head_dim(do.to(dt), d_pad).contiguous()
        n_k = kp.shape[1] if use_ring else kv_saved.shape[3]
        hop_owner = prob.kv_owners()

        ws, kv_own_ptrs, kv_bytes = None, None, 0
        hop_mode = use_ring and _use_hop_window(_slot_bytes(b, hk, n_k, d_pad))
        if use_ring:  # re-pack this rank's own slot (the forward's buffers are long reused)
            ws = get_workspace(ring_size, dev)
            own, kv_gather, kv_own_ptrs, kv_bytes = _place_kv(ws, hop_mode, rank, ring_size, b, hk, n_k, d_pad, dt, dev)
            _pack_slot(ops, kp, vp, own, ang if fused_k_rotary else None)
            _count()
        else:
            kv_gather = kv_saved

        def pull_kv_slots():
            """Side stream: copy engines pull the peers' K/V slots and publish one stream-ordered flag per owner, so the
            backward kernel's hop 0 (local K/V) overlaps with the transfer.  Call after the device barrier."""
            ready = torch.zeros(ring_size, dtype=torch.int32, device=dev)
            main = torch.cuda.current_stream(dev)
            start = torch.cuda.Event()
            start.record(main)
            with torch.cuda.stream(ws.side_stream):
                ws.side_stream.wait_event(start)
                for o_rank in hop_owner[1:]:
                    ops.peer_copy(kv_gather[o_rank], kv_own_ptrs[o_rank], kv_bytes)
                    ops.stream_write_u32(ready, o_rank, 1)  # stream memory op: needs no SM (the kernel owns them all)
                done = torch.cuda.Event()
                done.record(ws.side_stream)
            ready.record_stream(ws.side_stream)
            return ready, done

        if d_pad == 128 and CONFIG["backward"] == "fused":
            # ---------------- one-kernel backward (csrc/attn_bwd_fused_sm100.cu) ----------------
            with nvtx_range("rab.bwd.prep"):
                qdo = alloc_qdo_buffer(1, b, h, n_q, d_pad, dt, dev)
                stat = alloc_stat_buffer(1, b, h, n_q, dev)
                ops.bwd_prep(qp, o, dop, lse, qdo, stat, 0)
                dq_acc = torch.zeros(b * h, stat.shape[-1], d_pad, dtype=torch.float32, device=dev)
                _count(2)
            ready, ready_target, side_done, acc, acc_ptrs, nk_pad = None, 0, None, None, (), 0
            if use_ring:
                with nvtx_range("rab.bwd.zero+barrier"):
                    nk_pad = pad128(n_k)
                    acc_bytes = 2 * b * hk * nk_pad * d_pad * 4
                    region = ws.region("dkv_acc", acc_bytes)
                    acc = region.local[:acc_bytes].view(torch.float32).view(2, b * hk, nk_pad, d_pad)
                    acc.zero_()
                    acc_ptrs = region.peer_ptrs
                    ws.barrier()  # every peer's accumulators are zero and its own K/V slot is complete
                    _count(2)
                    if not hop_mode:
                        ready, side_done = pull_kv_slots()
                        ready_target = 1
            with nvtx_range("rab.bwd.kernel"):
                if hop_mode:  # one launch per hop against the 2-slot window; dq_acc / the owners' dK, dV accumulate
                    window_slots = _HopWindow(ops, ws, own, kv_own_ptrs, kv_bytes, hop_owner)
                    backward_hops(ops, prob, qdo[0], stat[0], dq_acc, hop_owner, window_slots.slot,
                                  dkv_acc_ptrs=acc_ptrs, nk_pad=nk_pad, kmask_bits=kbits,
                                  launched=window_slots.launched)
                    _count(len(hop_owner))
                else:
                    _, dk, dv = fused_attn_bwd_ring(prob, qdo[0], stat[0], kv_gather, kbits, dq_acc=dq_acc,
                                                    dkv_acc_ptrs=acc_ptrs, nk_pad=nk_pad, ready=ready,
                                                    ready_target=ready_target)
                    _count()
                dq = torch.empty(b, n_q, h, d_pad, dtype=dt, device=dev)
                ops.acc_convert(dq_acc, dq, prob.scale)
                _count()
            if use_ring:
                with nvtx_range("rab.bwd.barrier+convert"):
                    if side_done is not None:
                        torch.cuda.current_stream(dev).wait_event(side_done)
                    ws.barrier()  # every rank's kernel has finished adding into this rank's accumulators
                    dk = torch.empty(b, n_k, hk, d_pad, dtype=dt, device=dev)
                    dv = torch.empty_like(dk)
                    ops.acc_convert(acc[0], dk, 1.0)
                    ops.acc_convert(acc[1], dv, 1.0)
                    _count(3)
        elif hop_mode:
            # ---------------- two-kernel backward, one launch per hop and kernel ----------------
            # bwd_prep writes this rank's Q/dO + statistics straight into its one symmetric slot; after the barrier the
            # copy engines fill two 2-slot windows: the peers' K/V (for dQ) and their Q/dO + statistics (for dK/dV)
            n_pad = pad64(n_q)
            qdo_bytes = 2 * b * h * n_q * d_pad * qp.element_size()
            qdo_stat_bytes = qdo_bytes + 2 * b * h * n_pad * 4
            stage, qdo_ptrs = ws.staging("qdo", qdo_stat_bytes)
            qdo_flat = stage[:qdo_stat_bytes]

            def qdo_stat(flat: Tensor):
                return (flat[:qdo_bytes].view(dt).view(2, b * h, n_q, d_pad),
                        flat[qdo_bytes:].view(torch.float32).view(2, b * h, n_pad))

            qdo_own, stat_own = qdo_stat(qdo_flat)
            with nvtx_range("rab.bwd.prep+barrier"):
                if n_pad > n_q:  # the dK/dV kernel reads the padding rows (and masks them): keep them finite
                    stat_own[..., n_q:].zero_()
                    _count()
                ops.bwd_prep(qp, o, dop, lse, qdo_own[None], stat_own[None], 0)
                ws.barrier()  # every peer's own K/V and Q/dO + statistics slots are complete
                _count(2)
            with nvtx_range("rab.bwd.kernel"):
                q_hops = prob.q_owners()
                kv_window = _HopWindow(ops, ws, own, kv_own_ptrs, kv_bytes, hop_owner)
                qdo_window = _HopWindow(ops, ws, qdo_flat, qdo_ptrs, qdo_stat_bytes, q_hops)

                def launched(s: int) -> None:
                    kv_window.launched(s)
                    qdo_window.launched(s)

                dq, dk, dv = two_kernel_backward_hops(ops, prob, qdo_own, stat_own, kv_window.slot,
                                                      lambda s: qdo_stat(qdo_window.slot(s)), kbits, launched)
                _count(len(hop_owner) + len(q_hops))
        else:
            # ---------------- two-kernel backward (csrc/attn_bwd_sm100.cu) ----------------
            qdo_gather = alloc_qdo_buffer(ring_size, b, h, n_q, d_pad, dt, dev)
            stat_gather = alloc_stat_buffer(ring_size, b, h, n_q, dev)
            ops.bwd_prep(qp, o, dop, lse, qdo_gather, stat_gather, rank)
            _count()
            ready_kv, gather_done = None, None
            if use_ring:
                qdo_bytes = qdo_gather[rank].numel() * qdo_gather.element_size()
                stat_bytes = stat_gather[rank].numel() * 4
                stage, peer_ptrs = ws.staging("qdo", qdo_bytes + stat_bytes)
                stage[:qdo_bytes].copy_(qdo_gather[rank].view(torch.uint8).reshape(-1))
                stage[qdo_bytes:qdo_bytes + stat_bytes].copy_(stat_gather[rank].view(torch.uint8).reshape(-1))
                ws.barrier()
                _count(3)
                ready_kv, _ = pull_kv_slots()  # K/V first: the dQ kernel consumes it hop by hop
                with torch.cuda.stream(ws.side_stream):
                    for o_rank in prob.q_owners()[1:]:
                        ops.peer_copy(qdo_gather[o_rank], peer_ptrs[o_rank], qdo_bytes)
                        ops.peer_copy(stat_gather[o_rank], peer_ptrs[o_rank] + qdo_bytes, stat_bytes)
                    gather_done = torch.cuda.Event()
                    gather_done.record(ws.side_stream)
                qdo_gather.record_stream(ws.side_stream)
                stat_gather.record_stream(ws.side_stream)
            # dQ only needs the K/V slots (flag per owner): it overlaps with the Q/dO gather
            dq = ops.attn_bwd_dq(qdo_gather, kv_gather, stat_gather, ready_kv, 1 if ready_kv is not None else 0,
                                 *prob.tail(hop_owner, kbits))
            if gather_done is not None:
                torch.cuda.current_stream(dev).wait_event(gather_done)
            dk, dv = ops.attn_bwd_dkdv(qdo_gather, kv_gather, stat_gather, None, 0, *prob.tail(prob.q_owners(), kbits))
            _count(2)

        dq, dk, dv = dq[..., :d], dk[..., :d], dv[..., :d]
        if ang is not None:  # gradients w.r.t. the un-rotated q / k: rotate back (the rotation is orthogonal)
            dq_in, dk_in = torch.empty(b, n_q, h, d, dtype=dt, device=dev), torch.empty(b, n_k, hk, d, dtype=dt, device=dev)
            ops.rotary(dq, ang, dq_in, False, -1.0)
            ops.rotary(dk, ang, dk_in, False, -1.0)
            _count(2)
            dq, dk = dq_in, dk_in
        if orig_dtype != dt:
            dq, dk, dv = dq.to(orig_dtype), dk.to(orig_dtype), dv.to(orig_dtype)
        return dq, dk, dv, None, None, None, None, None, None, None, None, None, None, None


ring_flash_attn_cuda_ = RingFlashAttentionCUDAFunction.apply


@torch.autocast("cuda", enabled=False)
@typecheck
def ring_flash_attn_cuda(
    q: Tensor,
    k: Tensor,
    v: Tensor,
    mask: Optional[Tensor] = None,
    causal: bool = False,
    bucket_size: int = 1024,
    ring_reduce_col: bool = False,
    striped_ring_attn: bool = False,
    max_lookback_seq_len: Optional[int] = None,
    ring_size: Optional[int] = None,
    softclamp_qk_sim: bool = False,
    softclamp_value: float = 50.0,
    layout: Optional[str] = None,
    rotary_freqs: Optional[Tensor] = None,
) -> Tensor:
    """q [b, n, h, d]; k, v [b, n, hk, d] (this rank's shard when ``ring_reduce_col``).  ``bucket_size`` is
    accepted for signature parity; tiling is fixed by the kernel (128 x 128).  ``rotary_freqs`` ([n, d] or [n, d/2]
    fp32 angles, e.g. the output of ``RingRotaryEmbedding``): rotary embedding of q and k applied inside the op's pack
    kernels instead of by eager PyTorch passes."""
    check_attention_inputs(q, k, v, mask, name="ring_flash_attn_cuda", max_head_dim=128)
    return ring_flash_attn_cuda_(q, k, v, mask, causal, bucket_size, ring_reduce_col, striped_ring_attn,
                                 max_lookback_seq_len, ring_size, softclamp_qk_sim, softclamp_value, layout,
                                 rotary_freqs)
