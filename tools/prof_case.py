"""One launch of every hot kernel on a mid-sized problem, for ncu captures:

    ncu --set full --clock-control none --import-source on -k regex:"attn_|tree_decode" -o gpurun_out/prof_r2 \
        python tools/prof_case.py

Kernels launched (in order): pack_kv, attn_fwd_kernel, bwd_prep_kernel, attn_bwd_fused_kernel (one-kernel 5-GEMM backward),
acc_convert_kernel, attn_bwd_dq_kernel + attn_bwd_dkdv_kernel (two-kernel pair), tree_decode_tc_kernel (bf16 and fp8 KV).
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ring_attention_pytorch_b200.ops import _ext  # noqa: E402
from ring_attention_pytorch_b200.ops.fused import (AttnProblem, alloc_kv_buffer, alloc_qdo_buffer,  # noqa: E402
                                                   alloc_stat_buffer, fused_attn_bwd, fused_attn_bwd_ring,
                                                   fused_attn_fwd)
from ring_attention_pytorch_b200.ops.tree_decode_cuda import tree_decode_cuda  # noqa: E402
from ring_attention_pytorch_b200.parallel.layout import make_position_map  # noqa: E402

n = int(os.environ.get("PROF_N", 16384))
h = int(os.environ.get("PROF_H", 16))
d = int(os.environ.get("PROF_D", 128))
causal = os.environ.get("PROF_CAUSAL", "1") == "1"
ops = _ext.ops()
dt = torch.bfloat16
q, k, v, do = (torch.randn(1, n, h, d, device="cuda", dtype=dt) for _ in range(4))
pm = make_position_map("plain", 1, n)
prob = AttnProblem(1, h, h, 0, pm, causal, None, d ** -0.5)
kv = alloc_kv_buffer(1, 1, h, n, d, dt, "cuda")
qdo = alloc_qdo_buffer(1, 1, h, n, d, dt, "cuda")
stat = alloc_stat_buffer(1, 1, h, n, "cuda")
ready = torch.zeros(1, dtype=torch.int32, device="cuda")
ops.pack_kv(k, v, kv[0])
o, lse = fused_attn_fwd(prob, q, kv, [0], ready)
ops.bwd_prep(q, o, do, lse, qdo, stat, 0)
if d == 128:
    dq_acc, dk, dv = fused_attn_bwd_ring(prob, qdo[0], stat[0], kv)
    dq = torch.empty_like(q)
    ops.acc_convert(dq_acc, dq, d ** -0.5)
fused_attn_bwd(prob, qdo, kv, stat)
# decode: 8192 keys, batch 64, 32 / 8 heads
qd = torch.randn(64, 32, 1, 128, device="cuda", dtype=dt)
kd = torch.randn(64, 8, 8192, 128, device="cuda", dtype=dt)
vd = torch.randn(64, 8, 8192, 128, device="cuda", dtype=dt)
tree_decode_cuda(qd, kd, vd, dim_v=128)
one = torch.ones(64 * 8, device="cuda")
tree_decode_cuda(qd, kd.to(torch.float8_e4m3fn), vd.to(torch.float8_e4m3fn), dim_v=128, k_scale=one, v_scale=one)
torch.cuda.synchronize()
print("done")
