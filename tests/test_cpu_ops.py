"""Single-process checks of the portable ops against the dense oracle (runs on CPU)."""
import pytest
import torch

from ring_attention_pytorch_b200 import default_attention, ring_flash_attn
from ring_attention_pytorch_b200.ops.oracle import attention_with_positions
from ring_attention_pytorch_b200.parallel.layout import (from_layout, make_position_map, ring_hop_owners,
                                                         ring_query_owners, to_layout)


@pytest.mark.parametrize("causal", [False, True])
@pytest.mark.parametrize("kmask", [False, True])
@pytest.mark.parametrize("softclamp", [False, True])
def test_naive_flash_matches_dense(causal, kmask, softclamp):
    torch.manual_seed(0)
    q = torch.randn(2, 62, 4, 16, requires_grad=True)
    k = torch.randn(2, 62, 2, 16, requires_grad=True)
    v = torch.randn(2, 62, 2, 16, requires_grad=True)
    mask = (torch.rand(2, 62) > 0.3) if kmask else None
    out = ring_flash_attn(q, k, v, mask, causal, 4, False, False, None, None, softclamp, 30.0)
    ref = default_attention(q, k, v, mask, causal, softclamp, 30.0)
    g = torch.randn_like(out)
    got = torch.autograd.grad(out, (q, k, v), g)
    want = torch.autograd.grad(ref, (q, k, v), g)
    assert torch.allclose(out, ref, atol=2e-6)
    for a, b in zip(got, want):
        assert torch.allclose(a, b, atol=5e-6)


def test_cross_attention_causal_alignment():
    torch.manual_seed(0)
    q, k, v = torch.randn(1, 5, 2, 8), torch.randn(1, 12, 2, 8), torch.randn(1, 12, 2, 8)
    out = ring_flash_attn(q, k, v, None, True, 4)
    ref = default_attention(q, k, v, causal=True)
    assert torch.allclose(out, ref, atol=2e-6)


def test_fully_masked_rows_are_zero_not_nan():
    q, k, v = torch.randn(1, 4, 1, 8), torch.randn(1, 4, 1, 8), torch.randn(1, 4, 1, 8)
    mask = torch.zeros(1, 4, dtype=torch.bool)
    out = ring_flash_attn(q, k, v, mask)
    assert torch.equal(out, torch.zeros_like(out))
    out2, lse = attention_with_positions(q, k, v, key_mask=mask, return_lse=True)
    assert torch.equal(out2, torch.zeros_like(out2)) and torch.isinf(lse).all()


@pytest.mark.parametrize("layout", ["plain", "striped", "zigzag"])
def test_layout_roundtrip_and_positions(layout):
    world, n = 4, 8
    x = torch.arange(world * n).float()[None, :, None]
    y = to_layout(x, layout, world)
    assert torch.equal(from_layout(y, layout, world), x)
    pm = make_position_map(layout, world, n)
    allpos = torch.cat([pm.positions(r) for r in range(world)])
    assert sorted(allpos.tolist()) == list(range(world * n))
    assert torch.equal(y.flatten(), allpos.float())


def test_hop_and_query_owner_schedules():
    pm = make_position_map("plain", 4, 8)
    assert ring_hop_owners(pm, 2, True, None) == [2, 1, 0]
    assert ring_hop_owners(pm, 2, False, None) == [2, 1, 0, 3]
    assert ring_hop_owners(pm, 3, True, 8) == [3, 2]          # look-back of 8 tokens reaches one rank back
    assert ring_query_owners(pm, 1, True, None) == [1, 2, 3]
    pm = make_position_map("striped", 4, 8)
    assert ring_hop_owners(pm, 0, True, None) == [0, 3, 2, 1]
    assert ring_query_owners(pm, 0, True, None) == [0, 1, 2, 3]


def test_lookback_window_matches_oracle():
    torch.manual_seed(1)
    q, k, v = (torch.randn(1, 40, 2, 8) for _ in range(3))
    out = ring_flash_attn(q, k, v, None, True, 8, False, False, 7)
    pos = torch.arange(40)
    ref = attention_with_positions(q, k, v, pos, pos, causal=True, window=7)
    assert torch.allclose(out, ref, atol=2e-6)


# ---- single-hop building blocks (reference triton_flash_attn.py flash_attn_forward / flash_attn_backward) ----

def _hop_inputs(b=2, n=37, h=4, hk=2, d=16, hops=3, seed=0):
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(b, n, h, d, generator=g)
    ks = [torch.randn(b, n, hk, d, generator=g) for _ in range(hops)]
    vs = [torch.randn(b, n, hk, d, generator=g) for _ in range(hops)]
    return q, ks, vs


@pytest.mark.parametrize("fp32_acc", [False, True])
def test_hop_forward_carried_state_matches_dense(fp32_acc):
    from ring_attention_pytorch_b200.ops.flash_attn import flash_attn_forward

    q, ks, vs = _hop_inputs()
    o = torch.zeros_like(q, dtype=torch.float32) if fp32_acc else None
    m = lse = None
    for hop, (k, v) in enumerate(zip(ks, vs)):
        o, m, lse = flash_attn_forward(q, k, v, o=o, m=m, lse=lse, load_accumulated=hop > 0,
                                       return_normalized_output=hop == len(ks) - 1)
    ref, ref_lse = attention_with_positions(q, torch.cat(ks, 1), torch.cat(vs, 1), return_lse=True)
    assert m.shape == (2, 4, 128) and lse.shape == (2, 4, 128)
    assert torch.allclose(o, ref, atol=1e-5)
    assert torch.allclose(lse[..., :37], ref_lse, atol=1e-5)


def test_hop_forward_striped_diagonal_rule_and_bias():
    """Two striped ranks emulated by hand: hop from the later rank masks the diagonal (reference
    ring_flash_attention_cuda.py:157-160), key padding rides as an additive bias."""
    from ring_attention_pytorch_b200.ops.flash_attn import flash_attn_forward

    q, ks, vs = _hop_inputs(hops=2, seed=1)
    n = q.shape[1]
    # rank 0 of a 2-rank striped ring: own keys at positions 2j, peer keys at 2j + 1
    o, m, lse = flash_attn_forward(q, ks[0], vs[0], causal=True, load_accumulated=False)
    o, m, lse = flash_attn_forward(q, ks[1], vs[1], causal=True, causal_mask_diagonal=True, o=o, m=m, lse=lse,
                                   return_normalized_output=True, remove_padding=True)
    pos = torch.arange(n)
    ref = attention_with_positions(q, torch.cat(ks, 1), torch.cat(vs, 1), 2 * pos, torch.cat([2 * pos, 2 * pos + 1]),
                                   causal=True)
    assert lse.shape[-1] == n
    assert torch.allclose(o, ref, atol=1e-5)

    keep = torch.rand(2, n, generator=torch.Generator().manual_seed(3)) > 0.4
    keep[0] = False  # a batch row with every key dropped must give zeros, not NaN
    bias = torch.where(keep, 0.0, -torch.finfo(torch.float32).max)
    o2, _, _ = flash_attn_forward(q, ks[0], vs[0], bias=bias, load_accumulated=False, return_normalized_output=True)
    ref2 = default_attention(q, ks[0], vs[0], keep)
    assert torch.isfinite(o2).all() and torch.allclose(o2, ref2, atol=1e-5)
    assert o2[0].abs().max() == 0


@pytest.mark.parametrize("softclamp", [False, True])
def test_hop_backward_accumulates_to_autograd(softclamp):
    from ring_attention_pytorch_b200.ops.flash_attn import flash_attn_backward, flash_attn_forward

    q, ks, vs = _hop_inputs(seed=2)
    o = m = lse = None
    for hop, (k, v) in enumerate(zip(ks, vs)):
        o, m, lse = flash_attn_forward(q, k, v, causal=hop == 0, o=o, m=m, lse=lse, load_accumulated=hop > 0,
                                       return_normalized_output=hop == len(ks) - 1, softclamp_qk_sim=softclamp,
                                       softclamp_value=3.0)
    do = torch.randn_like(o)
    dq = torch.zeros_like(q)
    dks, dvs = [], []
    for hop, (k, v) in enumerate(zip(ks, vs)):
        hq, hk_, hv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
        delta = flash_attn_backward(do, q, k, v, o, lse, hq, hk_, hv, causal=hop == 0, softclamp_qk_sim=softclamp,
                                    softclamp_value=3.0)
        dq += hq
        dks.append(hk_)
        dvs.append(hv)
    assert torch.allclose(delta[..., :q.shape[1]], (o * do).sum(-1).transpose(1, 2), atol=1e-5)

    # oracle: hop 0 is causal on its own block, later hops are fully visible
    n = q.shape[1]
    qr = q.clone().requires_grad_()
    kr = [k.clone().requires_grad_() for k in ks]
    vr = [v.clone().requires_grad_() for v in vs]
    h = q.shape[2]
    from ring_attention_pytorch_b200.ops.oracle import expand_kv_heads, softclamp as clamp_fn
    sim = torch.einsum("bihd,bjhd->bhij", qr, expand_kv_heads(torch.cat(kr, 1), h)) * q.shape[-1] ** -0.5
    if softclamp:
        sim = clamp_fn(sim, 3.0)
    vis = torch.ones(n, 3 * n, dtype=torch.bool)
    vis[:, :n] = torch.tril(torch.ones(n, n, dtype=torch.bool))
    ref = torch.einsum("bhij,bjhd->bihd", sim.masked_fill(~vis, float("-inf")).softmax(-1),
                       expand_kv_heads(torch.cat(vr, 1), h))
    assert torch.allclose(o, ref, atol=1e-5)
    ref.backward(do)
    assert torch.allclose(dq, qr.grad, atol=2e-5)
    for a, b_ in zip(dks + dvs, kr + vr):
        assert torch.allclose(a, b_.grad, atol=2e-5)


def test_blockwise_feedforward_matches_plain_and_shares_state_dict():
    from ring_attention_pytorch_b200 import RingTransformer

    torch.manual_seed(0)
    kw = dict(num_tokens=64, dim=32, depth=2, causal=True, dim_head=8, heads=4, bucket_size=8, use_cuda_kernel=False)
    plain, block = RingTransformer(**kw), RingTransformer(ff_chunk_size=5, **kw)
    block.load_state_dict(plain.state_dict())          # identical parameter names
    x = torch.randint(0, 64, (2, 23))
    la, lb = plain(x, return_loss=True), block(x, return_loss=True)
    la.backward()
    lb.backward()
    assert torch.allclose(la, lb, atol=1e-6)
    for (na, pa), (nb, pb) in zip(plain.named_parameters(), block.named_parameters()):
        assert na == nb and torch.allclose(pa.grad, pb.grad, atol=1e-5), na


def test_poly_exp2_reference():
    """Host emulation (fp32 op by op) of ``poly_exp2x2`` in csrc/ptx.cuh, the FMA-pipe exponential the forward kernel
    runs for a quarter of its softmax (POLYQ in csrc/attn_fwd_sm100.cu): relative error < 1.5e-4, masked logits give exactly 0."""
    import numpy as np

    c = np.array([1.0, 0.6932103037834167, 0.24221116304397583, 0.05536489188671112], dtype=np.float32)

    def poly_exp2(x):
        x = np.maximum(x.astype(np.float32), np.float32(-127.0))
        magic = np.float32(12582912.0)
        t = (x + magic).astype(np.float32)
        nf = (t - magic).astype(np.float32)
        fr = (x - nf).astype(np.float32)
        p = (c[3] * fr + c[2]).astype(np.float32)
        p = (p * fr + c[1]).astype(np.float32)
        p = (p * fr + c[0]).astype(np.float32)
        eb = (t.view(np.uint32) << np.uint32(23)).astype(np.uint32)
        return (p.view(np.uint32) + eb).astype(np.uint32).view(np.float32)

    x = np.linspace(-40, 8, 400001).astype(np.float32)
    got, ref = poly_exp2(x), np.exp2(x.astype(np.float64))
    assert np.max(np.abs(got - ref) / ref) < 1.5e-4
    special = poly_exp2(np.array([-np.inf, -1000.0, 0.0], dtype=np.float32))
    assert special[0] == 0.0 and special[1] == 0.0 and special[2] == 1.0


def test_transformer_loss_ignores_padded_targets():
    """Derived labels are x[:, 1:], so their validity is mask[:, 1:] (reference ring_attention.py:614): the first pad token of
    a right-padded sequence must not be trained as a target."""
    import torch.nn.functional as F

    from ring_attention_pytorch_b200 import RingTransformer

    torch.manual_seed(0)
    model = RingTransformer(num_tokens=64, dim=32, depth=1, causal=True, dim_head=8, heads=4, bucket_size=8, ring_attn=False,
                            use_cuda_kernel=False)
    x = torch.randint(0, 64, (3, 17))
    lengths = torch.tensor([17, 9, 4])
    mask = torch.arange(17)[None, :] < lengths[:, None]
    loss = model(x, mask=mask, return_loss=True)
    logits = model(x[:, :-1], mask=mask[:, :-1])
    labels = x[:, 1:].masked_fill(~mask[:, 1:], model.ignore_index)
    want = F.cross_entropy(logits.transpose(1, 2), labels, ignore_index=model.ignore_index)
    assert torch.allclose(loss, want, atol=1e-6), (loss, want)
    # the shifted-by-one mask (what round 1 used) gives a different number on this batch
    wrong = F.cross_entropy(logits.transpose(1, 2), x[:, 1:].masked_fill(~mask[:, :-1], model.ignore_index),
                            ignore_index=model.ignore_index)
    assert not torch.allclose(want, wrong, atol=1e-4)


def test_argument_validation_names_the_offending_argument():
    from ring_attention_pytorch_b200.utils.validate import check_attention_inputs

    q = torch.randn(2, 8, 4, 16)
    k = torch.randn(2, 8, 3, 16)
    with pytest.raises(ValueError, match="multiple of key/value heads"):
        check_attention_inputs(q, k, k)
    k = torch.randn(2, 8, 2, 16)
    with pytest.raises(ValueError, match="mask must be bool"):
        check_attention_inputs(q, k, k, torch.ones(2, 7, dtype=torch.bool))
    check_attention_inputs(q, k, k, torch.ones(2, 8, dtype=torch.bool))


def test_memory_mode_selection():
    """CONFIG["memory"]: "auto" switches to the hop window at AUTO_RING_SLOT_BYTES; forward and backward decide from
    the same slot size, so they always agree."""
    from ring_attention_pytorch_b200.ops import ring_cuda

    old = ring_cuda.CONFIG["memory"]
    try:
        ring_cuda.CONFIG["memory"] = "auto"
        assert not ring_cuda._use_hop_window(ring_cuda.AUTO_RING_SLOT_BYTES - 1)
        assert ring_cuda._use_hop_window(ring_cuda.AUTO_RING_SLOT_BYTES)
        # headline config: S=262144, h=32, d=128 on 8 GPUs -> 512 MiB slots -> hop window
        assert ring_cuda._use_hop_window(2 * (262144 // 8) * 32 * 128 * 2)
        ring_cuda.CONFIG["memory"] = "ring"
        assert ring_cuda._use_hop_window(1)
        ring_cuda.CONFIG["memory"] = "gather"
        assert not ring_cuda._use_hop_window(1 << 40)
        ring_cuda.CONFIG["memory"] = "bogus"
        with pytest.raises(AssertionError):
            ring_cuda._use_hop_window(1)
    finally:
        ring_cuda.CONFIG["memory"] = old


def test_decode_cache_prefix_detection():
    """Which K/V layouts the tensor-core decode kernel may read in place (tensor-map plane stride) instead of copying."""
    from ring_attention_pytorch_b200.ops.tree_decode_cuda import _is_cache_prefix

    cache = torch.zeros(3, 2, 1000, 128, dtype=torch.bfloat16)
    assert _is_cache_prefix(cache)                       # dense
    assert _is_cache_prefix(cache[:, :, :300])           # filled prefix of a growing cache
    assert _is_cache_prefix(cache[:, :, 200:500])        # a sequence chunk (tree_attn_decode(shard_kv_seq=True))
    assert not _is_cache_prefix(cache[:, :, ::2])        # rows not dense
    assert not _is_cache_prefix(cache[..., :64])         # head dim sliced
    assert not _is_cache_prefix(cache.transpose(0, 1)[:, :, :300])  # planes not uniformly strided
    assert not _is_cache_prefix(torch.zeros(3, 1000, 2, 128).transpose(1, 2))  # [b, n, h, d] storage
    odd = torch.zeros(3, 2, 1001, 4, dtype=torch.float8_e4m3fn)  # plane stride 4004 B: not 16-byte aligned
    assert not _is_cache_prefix(odd[:, :, :300])
