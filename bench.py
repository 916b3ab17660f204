#!/usr/bin/env python
"""Headline benchmark: causal striped ring flash attention, forward + backward.

Config (BASELINE.json config 1): total sequence 262144, 32 heads, head dim 128, bf16, batch 1, causal,
striped layout, sequence sharded over the N GPUs of one box (STRONG scaling: total work is fixed).
A "step" is one forward + one backward of the ring attention op on synthetic q/k/v (random-init).

    python bench.py                      # N=1
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference     # the unmodified reference from baseline/_ref (Triton + NCCL P2P)
    python bench.py --dump-outputs DIR   # also write what the last timed step returned, to compare two builds

Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.  The
q/k/v shards (>= 268 MB each) are larger than the 126 MB L2, so no explicit flush is needed.

Besides the contract fields the JSON line carries: ``roofline_frac`` (value over N x the measured sustained cuBLAS bf16
rate of MEASURED_PEAKS.json; the NVLink term of the roofline is reported next to it), ``ring_kv_gbps`` (K/V bytes a
rank pulls in the forward over the time its in-kernel fetchers are active, N > 1), ``check`` (sampled rows of out / dQ /
dK / dV of one head against a chunked fp32 oracle at the benchmark's own scale) and ``rows`` with the 1 048 576-token
configuration the metric sentence of BASELINE.json names (fewer steps, same timing rules).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DUMP_BYTES = 32 * 2 ** 20  # --dump-outputs: float32 bytes over all arrays and ranks


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--seq-len", type=int, default=262144, help="TOTAL sequence length (all GPUs)")
    ap.add_argument("--heads", type=int, default=32)
    ap.add_argument("--kv-heads", type=int, default=None)
    ap.add_argument("--dim-head", type=int, default=128)
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--check", default="on", choices=["on", "off", "strict"],
                    help="after timing, verify sampled rows of out/dQ/dK/dV of one head against a chunked fp32 oracle "
                         "(strict: exit 1 on mismatch)")
    ap.add_argument("--no-1m", action="store_true", help="skip the extra 1 048 576-token row")
    ap.add_argument("--ref-budget-s", type=float, default=150.0,
                    help="reference arm only: cap the timed steps so that one timed loop stays inside this budget")
    ap.add_argument("--probe-device", type=int, default=None, help=argparse.SUPPRESS)
    ap.add_argument("--fwd-only", action="store_true", help="diagnostic only (not a valid headline number)")
    ap.add_argument("--memory", default="auto", choices=["auto", "gather", "ring"],
                    help="ring_cuda.CONFIG['memory']: 'ring' = per-hop launches against a 2-slot K/V window (O(n/W) "
                         "workspace); 'auto' picks it for K/V slots >= 256 MiB per rank (the headline config at any N)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (out, dq, dk, dv of this rank's "
                         "shard) as float32 DIR/<name>.npy (DIR/<name>_rank<r>.npy for N > 1): the same seeded sample "
                         f"of token rows on every run, {DUMP_BYTES // 2 ** 20} MiB at most over all ranks")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(out_dir: str, arrays: dict, rank: int, world: int) -> dict:
    """Write float32 samples of ``arrays`` ([batch, tokens, heads, dim] each): the same token rows of every array, drawn
    from a fixed seed, as many as fit ``DUMP_BYTES`` over all ranks (all rows when the shard is small enough)."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    n = next(iter(arrays.values())).shape[1]
    row_bytes = sum(t[:, :1].numel() * 4 for t in arrays.values())
    n_rows = max(1, min(n, DUMP_BYTES // (world * row_bytes)))
    rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:n_rows].sort().values
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, t in arrays.items():
        sample = t.detach().index_select(1, rows.to(t.device)).float().cpu().numpy()
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), sample)
    return {"dir": out_dir, "arrays": sorted(arrays), "token_rows": n_rows, "of": n}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:  # noqa: BLE001
            self.proc = None
            return

        def reader():
            for line in self.proc.stdout:
                self.rows.append(line.strip())

        self.thread = threading.Thread(target=reader, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for row in self.rows:
            parts = [p.strip() for p in row.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {
            "sm_mhz": statistics.median(sm) if sm else None,
            "sm_max_mhz": max(smax) if smax else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


def load_peaks() -> dict:
    """Roofline denominators: the driver's measurement of this pool's B200s, else the profiling recipe's fallback."""
    peaks = {"bf16_tflops_sustained": 1400.0, "bf16_tflops": 1590.0, "hbm_gbs": 6650.0, "source": "fallback"}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            m = json.load(f)
        peaks.update({k_: m[k_] for k_ in ("bf16_tflops_sustained", "bf16_tflops", "hbm_gbs") if k_ in m})
        peaks["source"] = "MEASURED_PEAKS.json"
    except Exception:  # noqa: BLE001
        pass
    peaks["nvlink_gbs"] = 770.0  # measured peer-copy rate per direction (B200_PROFILING.md)
    return peaks


def install_reference_shims():
    """The reference refuses to import unless a distribution literally named ``triton-nightly`` exists
    (reference triton_flash_attn.py:31-37).  Provide that *metadata only* next to the installed reference;
    the reference's code is untouched."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref, "ring_attention_pytorch")):
        raise RuntimeError("reference is not installed in baseline/_ref (see DESIGN.md)")
    import triton

    ver = triton.__version__.split("+")[0]
    shim = os.path.join(ref, f"triton_nightly-{ver}.dist-info")
    os.makedirs(shim, exist_ok=True)
    meta = os.path.join(shim, "METADATA")
    if not os.path.exists(meta):
        with open(meta, "w") as f:
            f.write(f"Metadata-Version: 2.1\nName: triton-nightly\nVersion: {ver}\n")
    sys.path.insert(0, ref)


def probe_reference_backward(local_rank: int) -> dict:
    """Does the reference's stock backward launch on this GPU?  Asked in a SUBPROCESS (tiny problem, one device) so that a
    kernel that compiles but cannot be loaded does not stay in this process's Triton cache.

    On sm_100, Triton 3.6 lowers the reference's 128x128 ``_bwd_kernel`` to tcgen05 with 704 TMEM columns (512 exist) and
    the launch raises OutOfResources.  Triton has its own switch for that, ``DISABLE_MMA_V5`` (emit mma.sync); when the
    probe reports exactly that failure the reference arm sets it AFTER its forward kernels were compiled (they keep
    tcgen05) and BEFORE its first backward.  The reference's code and call path are untouched, and the switch is reported
    in the JSON line.  Any other outcome leaves the environment alone."""
    if "DISABLE_MMA_V5" in os.environ:
        return {}
    try:
        env = {k_: v_ for k_, v_ in os.environ.items()
               if k_ not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "LOCAL_WORLD_SIZE", "GROUP_RANK", "ROLE_RANK")}
        proc = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--probe-device",
                               str(local_rank)], capture_output=True, text=True, timeout=600, env=env)
        lines = [ln for ln in proc.stdout.splitlines() if ln.startswith("{")]
        res = json.loads(lines[-1]) if lines else {}
    except Exception as e:  # noqa: BLE001
        print(f"[bench] reference probe did not run: {type(e).__name__}: {e}", file=sys.stderr)
        return {}
    err = res.get("probe_error", "")
    if "tensor memory" in err:
        return {"DISABLE_MMA_V5": "1 (set between the first forward and the first backward)", "because": err[:200]}
    return {}


def run_reference_probe(device_index: int) -> None:
    """Body of the probe subprocess: one tiny forward + backward of the reference on one GPU, stock environment."""
    import torch

    res = {}
    try:
        torch.cuda.set_device(device_index)
        install_reference_shims()
        from ring_attention_pytorch.ring_flash_attention_cuda import ring_flash_attn_cuda as ref_attn

        q, k, v = (torch.randn(1, 1024, 2, 128, device="cuda", dtype=torch.bfloat16, requires_grad=True) for _ in range(3))
        out = ref_attn(q, k, v, None, True, 1024, False, False, None, 1)
        out.backward(torch.randn_like(out))
        torch.cuda.synchronize()
        res["probe_ok"] = True
    except BaseException as e:  # noqa: BLE001
        res["probe_error"] = f"{type(e).__name__}: {e}".replace("\n", " ")[:400]
    print(json.dumps(res))


def main():
    args = parse_args()
    if args.probe_device is not None:
        run_reference_probe(args.probe_device)
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch multi-GPU runs with torch.distributed.run (see module docstring)")
        args.gpus = world

    def unavailable(why: str):
        if rank == 0:
            print(json.dumps({"impl": args.impl, "unavailable": why.replace("\n", " ")[:300]}))
        sys.exit(0)

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        if args.impl == "reference":
            unavailable("no CUDA device")
        raise SystemExit("bench.py needs a CUDA device")

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    S, H, D, B = args.seq_len, args.heads, args.dim_head, args.batch
    HK = args.kv_heads or H
    assert S % world == 0
    n = S // world
    ring = world > 1

    if args.impl == "reference":
        try:
            install_reference_shims()
            from ring_attention_pytorch.ring_flash_attention_cuda import ring_flash_attn_cuda as ref_attn
        except BaseException as e:  # noqa: BLE001  (the reference calls exit() on import problems)
            unavailable(f"reference import failed: {type(e).__name__}: {e}")

        def attn(q, k, v, bucket):
            return ref_attn(q, k, v, None, True, bucket, ring, ring, None, world)

        launches = {"count": 0}
        ref_env = probe_reference_backward(local_rank)
    else:
        from ring_attention_pytorch_b200.ops import ring_cuda

        ring_cuda.CONFIG["memory"] = args.memory

        def attn(q, k, v, bucket):
            return ring_cuda.ring_flash_attn_cuda(q, k, v, None, True, bucket, ring, ring, None, world)

        launches = ring_cuda.LAUNCHES
        ref_env = {}

    peaks = load_peaks()
    dt = torch.bfloat16

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def flops_of(S_: int) -> float:
        fwd = 4.0 * B * H * float(S_) * float(S_) * D * 0.5
        return fwd * (1.0 if args.fwd_only else 3.5)

    def measure(S_: int, steps: int, warmup: int, with_e2e: bool, with_check: bool, sample_clocks: bool,
                dump_dir: str | None = None):
        """One configuration: device-timed loop (+ e2e loop, + sampled-row check).  Returns a dict (rank 0 prints)."""
        n_ = S_ // world
        torch.cuda.reset_peak_memory_stats(dev)
        torch.manual_seed(1234 + rank)
        q = torch.randn(B, n_, H, D, device=dev, dtype=dt, requires_grad=True)
        k = torch.randn(B, n_, HK, D, device=dev, dtype=dt, requires_grad=True)
        v = torch.randn(B, n_, HK, D, device=dev, dtype=dt, requires_grad=True)
        w = torch.randn(B, n_, H, D, device=dev, dtype=dt)  # fixed projection used as upstream gradient
        bucket = min(n_, 1024)

        def call(q_, k_, v_):
            return attn(q_, k_, v_, bucket)

        def step():
            """One timed step; returns what a caller receives (the output and, with the backward, dQ / dK / dV)."""
            out = call(q, k, v)
            if args.fwd_only:
                return {"out": out}
            if ref_env:
                os.environ["DISABLE_MMA_V5"] = "1"  # forward kernels are compiled by now and keep tcgen05
            out.backward(w)
            res = {"out": out, "dq": q.grad, "dk": k.grad, "dv": v.grad}
            q.grad = k.grad = v.grad = None
            return res

        for _ in range(warmup):
            step()
        sync()

        # the reference at N=1 needs ~8 s per step: keep its timed loops inside a budget instead of timing out
        if args.impl == "reference":
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            step()
            t1.record()
            sync()
            per = max_over_ranks(t0.elapsed_time(t1)) * 1e-3
            steps = max(2, min(steps, int(args.ref_budget_s / max(per, 1e-6))))

        fetch_times = None
        hop_window = args.impl == "ours" and world > 1 and ring_cuda._use_hop_window(2 * B * n_ * HK * D * 2)
        if args.impl == "ours" and world > 1 and not hop_window:
            fetch_times = torch.zeros(256, 2, dtype=torch.int64, device=dev)
            torch.ops.rab.set_fetch_timing(fetch_times)
            step()
            sync()
            torch.ops.rab.set_fetch_timing(None)

        sampler = ClockSampler(local_rank)
        if rank == 0 and sample_clocks:
            sampler.start()
        launches_before = launches["count"]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync()
        e0.record()
        for _ in range(steps - 1):  # no step's results are held while the next one runs
            step()
        last = step()
        e1.record()
        sync()
        ms = max_over_ranks(e0.elapsed_time(e1))
        clocks = sampler.stop() if (rank == 0 and sample_clocks) else None
        n_launch = launches["count"] - launches_before
        dumped = dump_outputs(dump_dir, last, rank, world) if dump_dir else None
        del last

        flops_per_step = flops_of(S_)
        row = {
            "seq_len": S_,
            "steps": steps,
            "warmup": warmup,
            "value": flops_per_step * steps / (ms * 1e-3) / 1e12,
            "unit": "TFLOP/s",
            "ms_per_step": ms / steps,
            "tokens_per_s": B * S_ * steps / (ms * 1e-3),
            "gpu_launches": n_launch if args.impl == "ours" else 0,
            "clocks": clocks,
        }
        row["hop_window"] = bool(hop_window)
        if dumped:
            row["dumped_outputs"] = dumped
        if args.impl == "ours":
            # device memory: caching-allocator peak + the symmetric (cudaMalloc / IPC) workspace of the ring
            symm = 0
            if world > 1:
                from ring_attention_pytorch_b200.parallel.symm import get_workspace

                symm = sum(r.nbytes for r in get_workspace(world, dev).regions.values())
            row["memory_gb"] = {"allocator_peak": torch.cuda.max_memory_allocated(dev) / 2 ** 30,
                                "symmetric_workspace": symm / 2 ** 30,
                                "inputs_q_k_v_w": (2 * B * n_ * H * D + 2 * B * n_ * HK * D) * 2 / 2 ** 30}
        # roofline: the slower of FLOPs at the measured sustained GEMM rate and the bytes that must cross NVLink
        kv_bytes_fwd = (world - 1) * 2 * B * n_ * HK * D * 2  # K/V slots a rank pulls in the forward
        link_bytes = kv_bytes_fwd * (1 if args.fwd_only else 2) + (0 if args.fwd_only else (world - 1) * 2 * B * n_ * HK * D * 4)
        t_flops = flops_per_step / world / (peaks["bf16_tflops_sustained"] * 1e12)
        t_link = link_bytes / (peaks["nvlink_gbs"] * 1e9)
        row["roofline"] = {
            "frac": (max(t_flops, t_link) * 1e3) / (ms / steps),
            "t_flops_ms": t_flops * 1e3,
            "t_nvlink_ms": t_link * 1e3,
            "nvlink_bytes_per_rank": link_bytes,
            "peaks": peaks,
        }
        if fetch_times is not None:
            ft = fetch_times[fetch_times[:, 1] > 0]
            if ft.numel() > 0:
                window_ns = float((ft[:, 1].max() - ft[:, 0].min()).item())
                gbps = kv_bytes_fwd / max(window_ns, 1.0)
                t = torch.tensor([gbps], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MIN)
                row["ring_kv_gbps"] = {"value": float(t.item()), "of_nvlink_770": float(t.item()) / peaks["nvlink_gbs"],
                                       "bytes_per_rank": kv_bytes_fwd,
                                       "how": "forward K/V bytes pulled per rank / window in which its 148 in-kernel "
                                              "fetchers were active (globaltimer), min over ranks"}

        if hop_window:
            # the 2-slot window is filled by the copy engines: time a standalone pull of the forward's K/V bytes
            from ring_attention_pytorch_b200.ops.ring_cuda import _own_slot_workspace
            from ring_attention_pytorch_b200.parallel.symm import get_workspace

            ws = get_workspace(world, dev)
            own, own_ptrs, slot_bytes = _own_slot_workspace(ws, B, HK, n_, D, dt)
            dst = torch.empty_like(own)
            ws.barrier()
            sync()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for s_ in range(1, world):  # ring order: no two ranks read one source at the same time
                torch.ops.rab.peer_copy(dst, own_ptrs[(rank - s_) % world], slot_bytes)
            c1.record()
            sync()
            t = torch.tensor([kv_bytes_fwd / (c0.elapsed_time(c1) * 1e6)], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            row["ring_kv_gbps"] = {"value": float(t.item()), "of_nvlink_770": float(t.item()) / peaks["nvlink_gbs"],
                                   "bytes_per_rank": kv_bytes_fwd,
                                   "how": "copy-engine pull of the forward's K/V slots from every peer (what fills the "
                                          "2-slot window one hop ahead), standalone after the timed loop, min over ranks"}
            del dst

        # ---------------- end-to-end: pinned host inputs -> device every step, loss read back ------------
        if with_e2e and not args.fwd_only:
            hq = torch.randn(B, n_, H, D, dtype=dt).pin_memory()
            hk = torch.randn(B, n_, HK, D, dtype=dt).pin_memory()
            hv = torch.randn(B, n_, HK, D, dtype=dt).pin_memory()
            host = (hq, hk, hv)

            def run_e2e(prefetch: bool, nsteps: int) -> float:
                """nsteps end-to-end steps; returns elapsed ms on the device.  Every step's inputs are copied from
                pinned host memory inside the timed region and its loss is read back.  With ``prefetch`` the copy of
                step i+1 runs on a copy stream into the other device buffer while step i computes (what a prefetching
                data loader does); without it the copy is serial on the compute stream."""
                main_s = torch.cuda.current_stream(dev)
                nbuf = 2 if prefetch else 1
                bufs = [tuple(torch.empty_like(t_, device=dev) for t_ in host) for _ in range(nbuf)]
                copy_stream = torch.cuda.Stream(device=dev) if prefetch else main_s
                ready = [torch.cuda.Event() for _ in range(nbuf)]
                free = [torch.cuda.Event() for _ in range(nbuf)]

                def issue_copy(i):
                    bi = i % nbuf
                    with torch.cuda.stream(copy_stream):
                        if prefetch:
                            copy_stream.wait_event(free[bi])  # the step that last read this buffer is done
                        for d_, h_ in zip(bufs[bi], host):
                            d_.copy_(h_, non_blocking=True)
                        if prefetch:
                            ready[bi].record(copy_stream)

                def compute(i):
                    bi = i % nbuf
                    if prefetch:
                        main_s.wait_event(ready[bi])
                    qq, kk, vv = (t_.detach().requires_grad_() for t_ in bufs[bi])
                    out = call(qq, kk, vv)
                    loss = (out * w).sum(dtype=torch.float32)
                    loss.backward()
                    if prefetch:
                        free[bi].record(main_s)
                    return float(loss.item())  # device -> host read of the step's result

                sync()
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record()
                issue_copy(0)
                for i in range(nsteps):
                    if prefetch and i + 1 < nsteps:
                        issue_copy(i + 1)
                    compute(i)
                    if not prefetch and i + 1 < nsteps:
                        issue_copy(i + 1)
                s1.record()
                sync()
                return s0.elapsed_time(s1)

            pipeline, ems = "double-buffered H2D prefetch on a copy stream", None
            try:
                run_e2e(True, 1)  # untimed warm-up of the e2e path
                ems = run_e2e(True, steps)
            except Exception as e:  # noqa: BLE001 - fall back to the serial loop rather than lose the number
                print(f"[bench] prefetching e2e loop failed ({type(e).__name__}: {e}); using the serial loop",
                      file=sys.stderr)
            if ems is None:  # outside the except block so the failed attempt's buffers are released first
                pipeline = "serial H2D on the compute stream"
                torch.cuda.empty_cache()
                run_e2e(False, 1)
                ems = run_e2e(False, steps)
            ems = max_over_ranks(ems)
            h2d = (hq.numel() + hk.numel() + hv.numel()) * 2 * world
            row["e2e"] = {
                "value": flops_per_step * steps / (ems * 1e-3) / 1e12,
                "unit": "TFLOP/s",
                "ms_per_step": ems / steps,
                "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 4 * world,
                "pipeline": pipeline,
            }
            del hq, hk, hv, host

        # ---------------- sampled-row verification at this very scale --------------------------------------
        if with_check and not args.fwd_only:
            try:
                from ring_attention_pytorch_b200.utils.check import sampled_check

                out = call(q, k, v)
                out.backward(w)
                res = sampled_check(q.detach(), k.detach(), v.detach(), w, out.detach(), q.grad, k.grad, v.grad,
                                    causal=True, layout="striped" if ring else "plain", world=world, rank=rank,
                                    head_index=H // 2 + 1 if H > 2 else 0, samples=64)
                q.grad = k.grad = v.grad = None
                row["check"] = res
            except Exception as e:  # noqa: BLE001 - a broken checker must not lose the measurement
                row["check"] = {"ok": None, "error": f"{type(e).__name__}: {e}"[:300]}
        return row

    try:
        main_row = measure(S, args.steps, args.warmup, with_e2e=not args.no_e2e,
                           with_check=(args.check != "off" and args.impl == "ours"), sample_clocks=True,
                           dump_dir=args.dump_outputs)
    except BaseException as e:  # noqa: BLE001
        if args.impl == "reference":
            unavailable(f"reference failed to run: {type(e).__name__}: {e}")
        raise

    # the 1 048 576-token row of the metric sentence: a couple of steps, skipped when it would not fit the time budget
    rows = []
    S1M = 1048576
    if not args.no_1m and S != S1M and not args.fwd_only and S1M % world == 0:
        est = main_row["ms_per_step"] * 1e-3 * (S1M / S) ** 2
        if est * 4 <= 240.0:
            torch.cuda.empty_cache()
            try:
                r1m = measure(S1M, 2, 1, with_e2e=False, with_check=False, sample_clocks=False)
                r1m["note"] = "1 warm-up + 2 timed steps (the row is sized to stay inside the driver's time budget)"
                rows.append(r1m)
            except BaseException as e:  # noqa: BLE001
                rows.append({"seq_len": S1M, "skipped": f"{type(e).__name__}: {e}"[:200]})
        else:
            rows.append({"seq_len": S1M, "skipped": f"estimated {est:.0f} s per step does not fit the time budget"})

    if rank == 0:
        line = {
            "metric": "attention TFLOP/s (fwd+bwd, whole box, device-timed, max over ranks), causal striped ring",
            "value": main_row["value"],
            "unit": "TFLOP/s",
            "tokens_per_s": main_row["tokens_per_s"],
            "n_gpus": world,
            "steps": main_row["steps"],
            "warmup": main_row["warmup"],
            "ms_per_step": main_row["ms_per_step"],
            "higher_is_better": True,
            "scaling": "strong",
            "vs_baseline": None,
            "dtype": "bf16",
            "data": "synthetic q/k/v (random normal), random upstream gradient",
            "impl": args.impl,
            "config": {
                "model": "causal striped ring flash-attn (BASELINE.json config 1)",
                "global_batch": B,
                "seq_len": S,
                "heads": H,
                "kv_heads": HK,
                "dim_head": D,
                "parallelism": f"cp{world}" + (" (striped ring)" if ring else ""),
                "flops": "fwd 4*b*h*S^2*d*0.5, bwd 2.5x fwd (algorithmic 5-GEMM count)",
                "l2": "inputs larger than L2 (no flush needed)",
                "fwd_only": bool(args.fwd_only),
                "memory": args.memory + (" (hop window)" if main_row.get("hop_window") else ""),
                **({"reference_env": ref_env} if ref_env else {}),
                **({"steps_requested": args.steps} if main_row["steps"] != args.steps else {}),
            },
            "clocks": main_row["clocks"],
            "e2e": main_row.get("e2e"),
            "gpu_launches": main_row["gpu_launches"],
            "roofline_frac": main_row["roofline"]["frac"],
            "roofline": main_row["roofline"],
            **({"ring_kv_gbps": main_row["ring_kv_gbps"]} if "ring_kv_gbps" in main_row else {}),
            **({"check": main_row["check"]} if "check" in main_row else {}),
            **({"memory_gb": main_row["memory_gb"]} if "memory_gb" in main_row else {}),
            **({"dumped_outputs": main_row["dumped_outputs"]} if "dumped_outputs" in main_row else {}),
            "rows": rows,
        }
        print(json.dumps(line))

    failed = args.check == "strict" and main_row.get("check", {}).get("ok") is False
    if world > 1:
        dist.destroy_process_group()
    if failed:
        sys.exit(1)


if __name__ == "__main__":
    main()
