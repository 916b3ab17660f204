"""Peer K/V fetch micro-benchmark: what do the forward kernel's in-kernel fetchers sustain over NVLink?

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 \
        tools/bench_fetch.py --slot-mb 512 --out profiles/peer_fetch_n2.json

The fused forward is launched with a NEGLIGIBLE attention problem (128 queries, one head) against large K/V slots, so
the kernel's duration is the transfer: every one of the 148 CTAs' fetcher warps moves its 1/148 share of every remote
slot (peer global -> shared memory -> local global, two 16 KB bulk-TMA copies in flight per SM).  Reported per rank:

* ``gbps_window``  bytes pulled / the window between the first fetcher starting and the last one finishing
                   (``%globaltimer``, recorded by the kernel itself)
* ``gbps_kernel``  bytes pulled / CUDA-event duration of the whole launch

against the measured peer-copy rate (770 GB/s per direction) and the nominal 900 GB/s of NVLink 5.  Also times a
``cudaMemcpyAsync`` peer pull of the same bytes (the copy-engine path the backward uses) for comparison.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--slot-mb", type=int, default=512, help="bytes of ONE rank's K+V slot")
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world > 1, "run under torchrun with >= 2 ranks"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    from ring_attention_pytorch_b200.ops import _ext
    from ring_attention_pytorch_b200.ops.fused import AttnProblem, fused_attn_fwd
    from ring_attention_pytorch_b200.ops.ring_cuda import _ring_gather_workspace
    from ring_attention_pytorch_b200.parallel.layout import make_position_map
    from ring_attention_pytorch_b200.parallel.symm import get_workspace

    ops = _ext.ops()
    d, hk, b = 128, 1, 1
    n_k = args.slot_mb * (1 << 20) // (2 * hk * d * 2)  # K + V, 16 bit
    n_k = n_k // 128 * 128
    dt = torch.bfloat16
    ws = get_workspace(world, dev)
    pm = make_position_map("plain", world, n_k)
    prob = AttnProblem(b, 1, hk, rank, pm, False, None, d ** -0.5)
    q = torch.randn(b, 128, 1, d, device=dev, dtype=dt)
    k = torch.randn(b, n_k, hk, d, device=dev, dtype=dt)
    v = torch.randn(b, n_k, hk, d, device=dev, dtype=dt)
    times = torch.zeros(256, 2, dtype=torch.int64, device=dev)
    res_w, res_k = [], []
    pulled = None
    for it in range(args.iters + 2):
        gather, own_ptrs, slot_bytes = _ring_gather_workspace(ws, world, b, hk, n_k, d, dt)
        ops.pack_kv(k, v, gather[rank])
        ws.barrier()
        peers = [0 if o == rank else own_ptrs[o] for o in range(world)]
        ready = torch.zeros(world, dtype=torch.int32, device=dev)
        times.zero_()
        ops.set_fetch_timing(times)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        # non-causal: every owner is visited, 128 queries x n_k keys of one head per owner: microseconds of MMA work
        fused_attn_fwd(prob, q, gather, peers, ready)
        e1.record()
        torch.cuda.synchronize()
        ops.set_fetch_timing(None)
        ft = times[times[:, 1] > 0]
        pulled = (world - 1) * slot_bytes
        if it >= 2 and ft.numel() > 0:
            res_w.append(pulled / float((ft[:, 1].max() - ft[:, 0].min()).item()))
            res_k.append(pulled / (e0.elapsed_time(e1) * 1e6))
    # the copy-engine path for the same bytes
    gather, own_ptrs, slot_bytes = _ring_gather_workspace(ws, world, b, hk, n_k, d, dt)
    ws.barrier()
    torch.cuda.synchronize()
    ce = []
    for it in range(args.iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s_ in range(1, world):  # staggered like the backward's pull (r-1, r-2, ...): no two ranks hit one source at once
            o = (rank - s_) % world
            ops.peer_copy(gather[o], own_ptrs[o], slot_bytes)
        e1.record()
        torch.cuda.synchronize()
        ce.append(pulled / (e0.elapsed_time(e1) * 1e6))
    mine = {"rank": rank, "gbps_window": sorted(res_w)[len(res_w) // 2], "gbps_kernel": sorted(res_k)[len(res_k) // 2],
            "gbps_copy_engine": sorted(ce)[len(ce) // 2]}
    allr = [None] * world
    dist.all_gather_object(allr, mine)
    if rank == 0:
        res = {"n_gpus": world, "slot_mb": args.slot_mb, "bytes_pulled_per_rank": pulled, "per_rank": allr,
               "min_gbps_window": min(a["gbps_window"] for a in allr),
               "of_measured_770": min(a["gbps_window"] for a in allr) / 770.0,
               "of_nominal_900": min(a["gbps_window"] for a in allr) / 900.0,
               "how": "fused forward with negligible attention work; in-kernel globaltimer window of the 148 fetchers"}
        print(json.dumps(res))
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                json.dump(res, f, indent=1)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
