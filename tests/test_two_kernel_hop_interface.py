"""The two-kernel backward one ring hop per launch (``memory="ring"``): the hop ops share the attention ops' problem tail,
and the hop loop launches dQ and dK/dV hops in order with the right slots, carry flags and hooks."""
import os
import shutil
from dataclasses import dataclass

import pytest
import torch

from ring_attention_pytorch_b200.ops.fused import AttnProblem, two_kernel_backward_hops
from ring_attention_pytorch_b200.parallel.layout import make_position_map

HOP_OPS = ("attn_fwd", "attn_bwd_dq_hop", "attn_bwd_dkdv_hop")


def _nvcc():
    return shutil.which("nvcc") or os.path.exists(os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"),
                                                              "bin", "nvcc"))


@pytest.mark.skipif(not _nvcc(), reason="building the extension needs nvcc")
def test_two_kernel_hop_ops_share_the_problem_tail():
    from ring_attention_pytorch_b200.ops import _ext

    assert _ext.load()
    prob = AttnProblem(batch=2, heads=8, kv_heads=4, rank=3, pm=make_position_map("zigzag", 4, 64), causal=True,
                       window=96, scale=0.125, softclamp=30.0, q_pos_offset=-1)
    tail = prob.tail([3, 2], torch.zeros(4, 2, 4, dtype=torch.int32))
    schemas = {name: getattr(torch.ops.rab, name).default._schema for name in HOP_OPS}
    tails = {name: [(a.name, str(a.type)) for a in s.arguments[-len(tail):]] for name, s in schemas.items()}
    assert tails["attn_bwd_dq_hop"] == tails["attn_fwd"] and tails["attn_bwd_dkdv_hop"] == tails["attn_fwd"], tails
    heads = {name: [(a.name, str(a.type)) for a in s.arguments[:-len(tail)]] for name, s in schemas.items()}
    assert heads["attn_bwd_dq_hop"] == [("qdo_own", "Tensor"), ("kv_slot", "Tensor"), ("stat_own", "Tensor"),
                                        ("carry", "Tensor"), ("carry_in", "bool"), ("carry_out", "bool")]
    assert heads["attn_bwd_dkdv_hop"] == [("qdo_slot", "Tensor"), ("kv_own", "Tensor"), ("stat_slot", "Tensor"),
                                          ("carry", "Tensor"), ("carry_in", "bool"), ("carry_out", "bool")]
    for name in ("attn_bwd_dq_hop", "attn_bwd_dkdv_hop"):
        carry = schemas[name].arguments[3]
        assert carry.alias_info is not None and carry.alias_info.is_write, name  # the carry is written in place
    assert len(schemas["attn_bwd_dq_hop"].returns) == 1 and len(schemas["attn_bwd_dkdv_hop"].returns) == 2


class _FakeOps:
    def __init__(self):
        self.calls = []

    def attn_bwd_dq_hop(self, qdo_own, kv_slot, stat_own, carry, carry_in, carry_out, *tail):
        self.calls.append(("dq", qdo_own, kv_slot, stat_own, carry, carry_in, carry_out, tail))
        return ("dq", len(self.calls))

    def attn_bwd_dkdv_hop(self, qdo_slot, kv_own, stat_slot, carry, carry_in, carry_out, *tail):
        self.calls.append(("dkdv", qdo_slot, kv_own, stat_slot, carry, carry_in, carry_out, tail))
        return ("dk", len(self.calls)), ("dv", len(self.calls))


@dataclass(frozen=True)
class _Problem(AttnProblem):
    """A problem with given owner lists (a causal plain ring gives rank 0 one K/V hop and W query hops)."""
    kv_hops: tuple = ()
    q_hops: tuple = ()

    def kv_owners(self):
        return list(self.kv_hops)

    def q_owners(self):
        return list(self.q_hops)


def _slot(tag, s):
    return torch.full((2, 1, 1, 1), float(100 * tag + s))


def _run(kv_hops, q_hops):
    prob = _Problem(batch=2, heads=4, kv_heads=2, rank=kv_hops[0], pm=make_position_map("plain", 8, 64), causal=True,
                    window=None, scale=0.125, kv_hops=tuple(kv_hops), q_hops=tuple(q_hops))
    b, h, hk, n_q, n_k, d = 2, 4, 2, 16, 24, 64
    qdo_own, stat_own = torch.zeros(2, b * h, n_q, d), torch.zeros(2, b * h, 64)
    kv_slots = {s: torch.full((2, b * hk, n_k, d), float(s)) for s in range(len(kv_hops))}
    qdo_slots = {s: (_slot(1, s), _slot(2, s)) for s in range(len(q_hops))}
    asked, launched, ops = [], [], _FakeOps()
    kbits = torch.zeros(8, 2, 4, dtype=torch.int32)

    def kv_slot(s):
        asked.append(("kv", s))
        return kv_slots[s]

    def qdo_slot(s):
        asked.append(("qdo", s))
        return qdo_slots[s]

    def hook(s):
        launched.append(s)
        asked.append(("launched", s))

    dq, dk, dv = two_kernel_backward_hops(ops, prob, qdo_own, stat_own, kv_slot, qdo_slot, kbits, hook)
    return prob, ops, asked, launched, (dq, dk, dv), (qdo_own, stat_own, kv_slots, qdo_slots, kbits, (b, h, hk, n_q, n_k, d))


@pytest.mark.parametrize("n_kv,n_q", [(1, 1), (2, 2), (8, 8), (1, 8), (8, 1), (3, 5)])
def test_two_kernel_hop_loop_protocol(n_kv, n_q):
    kv_hops = [(5 - s) % 8 for s in range(n_kv)]
    q_hops = [(5 + s) % 8 for s in range(n_q)]
    prob, ops, asked, launched, (dq, dk, dv), (qdo_own, stat_own, kv_slots, qdo_slots, kbits, shape) = \
        _run(kv_hops, q_hops)
    b, h, hk, n_q_rows, n_k, d = shape
    steps = max(n_kv, n_q)

    # launch order: dQ hop s, then dK/dV hop s, step by step; a step past one list launches the other kernel only
    kinds = [c[0] for c in ops.calls]
    expected = [k for s in range(steps) for k, n in (("dq", n_kv), ("dkdv", n_q)) if s < n]
    assert kinds == expected
    assert launched == list(range(steps))
    # each slot is asked for once, before the launch that reads it; the hook follows the step's launches
    want = [("kv", 0)]
    for s in range(steps):
        if 0 < s < n_kv:
            want.append(("kv", s))
        if s < n_q:
            want.append(("qdo", s))
        want.append(("launched", s))
    assert asked == want

    dq_calls = [c for c in ops.calls if c[0] == "dq"]
    dkdv_calls = [c for c in ops.calls if c[0] == "dkdv"]
    for s, c in enumerate(dq_calls):
        _, q, kv, st, carry, cin, cout, tail = c
        assert (cin, cout) == (s > 0, s + 1 < n_kv)
        assert q.shape == (1,) + tuple(qdo_own.shape) and q.data_ptr() == qdo_own.data_ptr()
        assert st.shape == (1,) + tuple(stat_own.shape) and st.data_ptr() == stat_own.data_ptr()
        assert kv.shape == (1,) + tuple(kv_slots[s].shape) and kv.data_ptr() == kv_slots[s].data_ptr()
        assert tail == prob.tail([kv_hops[s]], kbits)
        assert carry is dq_calls[0][4]  # one carry travels through every hop
        assert carry.dtype == torch.float32
        assert carry.shape == ((b, n_q_rows, h, d) if n_kv > 1 else (0,))
    for s, c in enumerate(dkdv_calls):
        _, q, kv, st, carry, cin, cout, tail = c
        assert (cin, cout) == (s > 0, s + 1 < n_q)
        assert q.shape[0] == 1 and q.data_ptr() == qdo_slots[s][0].data_ptr()
        assert st.shape[0] == 1 and st.data_ptr() == qdo_slots[s][1].data_ptr()
        assert kv.data_ptr() == kv_slots[0].data_ptr()  # dK/dV always runs against this rank's own K/V
        assert tail == prob.tail([q_hops[s]], kbits)
        assert carry is dkdv_calls[0][4]
        assert carry.shape == ((2, b, n_k, hk, d) if n_q > 1 else (0,))
    # the results are the last launch of each kernel
    last_dq = max(i for i, c in enumerate(ops.calls) if c[0] == "dq") + 1
    last_dkdv = max(i for i, c in enumerate(ops.calls) if c[0] == "dkdv") + 1
    assert dq == ("dq", last_dq) and (dk, dv) == (("dk", last_dkdv), ("dv", last_dkdv))


def test_two_kernel_hop_loop_follows_the_problem_owner_lists():
    """With a real problem the loop walks ``kv_owners()`` for dQ and ``q_owners()`` for dK/dV."""
    for layout, causal in (("plain", True), ("striped", True), ("zigzag", True), ("plain", False)):
        for rank in range(4):
            prob = AttnProblem(1, 2, 1, rank, make_position_map(layout, 4, 128), causal, None, 0.125)
            ops = _FakeOps()
            two_kernel_backward_hops(ops, prob, torch.zeros(2, 2, 128, 64), torch.zeros(2, 2, 128),
                                     lambda s: torch.zeros(2, 1, 128, 64),
                                     lambda s: (torch.zeros(2, 2, 128, 64), torch.zeros(2, 2, 128)))
            assert [c[7][-1] for c in ops.calls if c[0] == "dq"] == [[o] for o in prob.kv_owners()]
            assert [c[7][-1] for c in ops.calls if c[0] == "dkdv"] == [[o] for o in prob.q_owners()]
