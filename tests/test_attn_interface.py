"""The attention ops' launch interface: one problem-argument tail shared by every op, and the per-hop protocol of the
shared forward / backward hop loops (``memory="ring"``)."""
import os
import shutil

import pytest
import torch

from ring_attention_pytorch_b200.ops.fused import AttnProblem, backward_hops, forward_hops
from ring_attention_pytorch_b200.parallel.layout import make_position_map

ATTN_OPS = ("attn_fwd", "attn_fwd_hop", "attn_bwd_dq", "attn_bwd_dkdv", "attn_bwd_ring")


def _problem(world=4):
    return AttnProblem(batch=2, heads=8, kv_heads=4, rank=3, pm=make_position_map("zigzag", world, 64), causal=True,
                       window=96, scale=0.125, softclamp=30.0, q_pos_offset=-1)


def _nvcc():
    return shutil.which("nvcc") or os.path.exists(os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"),
                                                              "bin", "nvcc"))


@pytest.mark.skipif(not _nvcc(), reason="building the extension needs nvcc")
def test_attention_ops_share_one_problem_tail():
    from ring_attention_pytorch_b200.ops import _ext

    assert _ext.load()
    ops = torch.ops.rab
    prob = _problem()
    kbits = torch.zeros(4, 2, 4, dtype=torch.int32)
    tail = prob.tail([3, 2], kbits)
    schemas = [getattr(ops, name).default._schema.arguments for name in ATTN_OPS]
    tails = [[(a.name, str(a.type)) for a in args[-len(tail):]] for args in schemas]
    assert all(t == tails[0] for t in tails[1:]), tails
    # nothing problem-shaped sits outside the tail
    for args in schemas:
        assert not {a.name for a in args[:-len(tail)]} & {name for name, _ in tails[0]}

    pm = prob.pm
    expected = {"kmask_bits": kbits, "batch": 2, "heads": 8, "kv_heads": 4, "rank": 3, "causal": True, "window": 96,
                "scale": 0.125, "softclamp": 30.0, "pos_stride": pm.stride, "seg_len": pm.seg_len,
                "base0": pm.base0, "base1": pm.base1, "q_pos_offset": -1, "hop_owner": [3, 2]}
    assert [name for name, _ in tails[0]] == list(expected)
    for (name, _), value in zip(tails[0], tail):
        assert value is expected[name] if name == "kmask_bits" else value == expected[name], name
        assert type(value) is type(expected[name]), name
    assert prob.tail([0])[0] is None and prob.tail([0])[5] is True
    assert AttnProblem(1, 1, 1, 0, pm, False, None, 1.0).tail([0])[6] == 0  # no window -> 0


class _FakeOps:
    def __init__(self):
        self.calls = []

    def attn_fwd_hop(self, q, kv_slot, carry_o, carry_ml, carry_in, carry_out, *tail):
        self.calls.append(("fwd", kv_slot, carry_o, carry_ml, carry_in, carry_out, tail))
        return ("o", len(self.calls)), ("lse", len(self.calls))

    def attn_bwd_ring(self, qdo, kv_slot, stat, dq_acc, ready, ready_target, dkv_acc_ptrs, nk_pad, *tail):
        self.calls.append(("bwd", kv_slot, dq_acc, ready, ready_target, dkv_acc_ptrs, nk_pad, tail))
        return torch.empty(0), torch.empty(0)


@pytest.mark.parametrize("n_hops", [1, 2, 8])
def test_forward_hop_loop_protocol(n_hops):
    prob = _problem(world=8)
    hops = [(prob.rank - s) % 8 for s in range(n_hops)]
    slots = {s: torch.full((2, 1, 1, 1), float(s)) for s in range(n_hops)}
    launched, ops = [], _FakeOps()
    kbits = torch.zeros(8, 2, 4, dtype=torch.int32)
    o, lse = forward_hops(ops, prob, torch.zeros(2, 16, 8, 64), hops, slots.__getitem__, kbits, launched.append)
    assert launched == list(range(n_hops))
    assert [c[4:6] for c in ops.calls] == [(s > 0, s + 1 < n_hops) for s in range(n_hops)]
    for s, c in enumerate(ops.calls):
        assert c[1].shape == (1, 2, 1, 1, 1) and c[1][0] is not None and float(c[1][0, 0, 0, 0, 0]) == s
        assert c[6] == prob.tail([hops[s]], kbits)
        assert c[2] is ops.calls[0][2] and c[3] is ops.calls[0][3]  # one carry travels through every hop
    assert ops.calls[0][2].shape == (2, 16, 8, 64) and ops.calls[0][3].shape == (2, 2 * 8, 16)
    assert (o, lse) == (("o", n_hops), ("lse", n_hops))  # the last launch's result


@pytest.mark.parametrize("n_hops", [1, 2, 8])
def test_backward_hop_loop_protocol(n_hops):
    prob = _problem(world=8)
    hops = [(prob.rank - s) % 8 for s in range(n_hops)]
    slots = {s: torch.full((2, 1, 1, 1), float(s)) for s in range(n_hops)}
    launched, ops = [], _FakeOps()
    dq_acc = torch.zeros(16, 64, 128)
    backward_hops(ops, prob, torch.zeros(2, 16, 64, 128), torch.zeros(2, 16, 64), dq_acc, hops, slots.__getitem__,
                  dkv_acc_ptrs=range(8), nk_pad=128, launched=launched.append)
    assert launched == list(range(n_hops))
    assert len(ops.calls) == n_hops
    for s, c in enumerate(ops.calls):
        assert c[1].shape == (1, 2, 1, 1, 1) and float(c[1][0, 0, 0, 0, 0]) == s
        assert c[2] is dq_acc and c[3] is None and c[4] == 0 and c[5] == list(range(8)) and c[6] == 128
        assert c[7] == prob.tail([hops[s]])
