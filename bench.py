#!/usr/bin/env python
"""bench.py -- Gaussian messages/sec on the batched LGSSM smoothing sweep (BASELINE.json metric).

Workload (BASELINE.json configs[1], SURVEY.md 8d config 2): notebook model lifted to d = m = 4,
T = 1000, batch = 65 536 chains PER GPU (weak scaling), shared (A, B, P, Q, prior), fp32 I/O.
One "step" = one forward+backward sum-product sweep over the whole batch through the C ABI
(`rxg_lgssm_smooth_f32`): gain-table kernels + the fused sweep kernel; messages = 6 * T * batch.

  value     device-resident inputs/outputs, CUDA events on the launching stream, max over ranks
  e2e       same call with HOST (pinned) buffers: H2D of y and D2H of posteriors inside the timed region
  roofline  dominant kernel (lgssm_shared_kernel): algorithmic 96 B per (chain, step) / its own
            event-timed duration, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  fp64 C port of the reference's message schedule (oracle/c) on the host cores

`--impl reference` times that CPU port alone (the reference itself is Julia and cannot run here).
`--dump-outputs DIR` writes what the timed path returned in its last step as DIR/<name>.npy (see dump_outputs), so that
two builds can be compared output for output: the inputs are seeded and the same from run to run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

D, M, T, BATCH = 4, 4, 1000, 65536
MSG_PER_STEP = 6                      # rule invocations per (chain, time step), SURVEY.md 8a
ALGO_BYTES_PER_STEP = 4 * (M + D + D * D)   # 96 B: read y_t, write mu_t and full Sigma_t (SURVEY.md 8d)
METRIC = "gaussian_messages_per_sec_batched_lgssm_d4_T1000"
DUMP_BYTES = 64 * 10**6               # --dump-outputs: all files together stay below this


def dump_outputs(path, slabs, seed=0):
    """Writes device outputs as <path>/<name>.npy in their own dtype (float32).  ``slabs`` maps each name to a tensor
    [G, ..., b] of G * b chains in rank-major slabs (G = 1 on one GPU); the files are [..., chains].  When every chain does
    not fit in DUMP_BYTES, all arrays keep the same seeded sample of chains, in ascending chain order."""
    import torch
    os.makedirs(path, exist_ok=True)
    first = next(iter(slabs.values()))
    G, b = first.shape[0], first.shape[-1]
    per_chain = sum(t[0, ..., 0].numel() * t.element_size() for t in slabs.values())
    k = min(G * b, max(1, (DUMP_BYTES - 4096) // per_chain))           # 4 KB for the .npy headers
    idx = torch.as_tensor(np.sort(np.random.default_rng(seed).choice(G * b, k, replace=False)), device=first.device)
    for name, t in slabs.items():
        np.save(os.path.join(path, name + ".npy"), t[idx // b, ..., idx % b].movedim(0, -1).cpu().numpy())


def notebook_model_f32():
    def rot(th):
        return np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
    A = np.zeros((4, 4)); A[:2, :2] = rot(np.pi / 15); A[2:, 2:] = rot(np.pi / 35)
    mod = dict(A=A, B=np.diag([1.3, 0.7, 1.3, 0.7]), P=0.05 * np.eye(4), Q=10.0 * np.eye(4),
               m0=np.zeros(4), S0=100.0 * np.eye(4))
    return {k: v.astype(np.float32) for k, v in mod.items()}


def notebook_model_d2_f32():
    """The notebook's own d = 2 parameters (benchmarks/...ipynb:158-162): rotation pi/15, B = diag(1.3, 0.7)."""
    th = np.pi / 15
    mod = dict(A=np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]]), B=np.diag([1.3, 0.7]),
               P=0.05 * np.eye(2), Q=10.0 * np.eye(2), m0=np.zeros(2), S0=100.0 * np.eye(2))
    return {k: v.astype(np.float32) for k, v in mod.items()}


def dense_model_f32(d, seed=64):
    """BASELINE configs[2] family (SURVEY.md 8d config 3): A = 0.99 * Orth (Q factor of a seeded Gaussian), B = I,
    P = 0.05 I, Q = 10 I, prior N(0, 100 I)."""
    rng = np.random.default_rng(seed)
    Qf, _ = np.linalg.qr(rng.standard_normal((d, d)))
    mod = dict(A=0.99 * Qf, B=np.eye(d), P=0.05 * np.eye(d), Q=10.0 * np.eye(d), m0=np.zeros(d), S0=100.0 * np.eye(d))
    return {k: v.astype(np.float32) for k, v in mod.items()}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def host_cores():
    """Host threads this process can actually use: min(affinity, cgroup CPU quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per))))
    except Exception:
        pass
    return n


def cpu_baseline(seconds_target=12.0, chunk=2048, parity_sample=None):
    """fp64 C port of the reference schedule on all host cores, bounded sample of the same workload.
    `parity_sample` (chains of the GPU arm's timed buffers): recomputed here by the port and compared -- the parity
    gate of the timed workload itself (mean relative L2 < 1e-5, covariance relative Frobenius < 1e-4)."""
    from oracle import c_twin
    mod = {k: v.astype(np.float64) for k, v in notebook_model_f32().items()}
    parity = None
    if parity_sample is not None:
        ref = c_twin.smooth(parity_sample["y"], **mod, nthreads=1)
        parity = {"chains": parity_sample["chains"],
                  "mean_rel_l2": float(np.linalg.norm(parity_sample["mean"] - ref["mean"]) / np.linalg.norm(ref["mean"])),
                  "cov_rel_fro": float(np.linalg.norm(parity_sample["cov"] - ref["cov"]) / np.linalg.norm(ref["cov"])),
                  "tolerance": {"mean": 1e-5, "cov": 1e-4}, "checker": "fp64 C port (oracle/c/rxg_oracle.c), inside the cpu_baseline leg"}
        assert parity["mean_rel_l2"] < 1e-5 and parity["cov_rel_fro"] < 1e-4, parity
    cores = host_cores()
    rng = np.random.default_rng(0)
    y = (rng.standard_normal((T, M, chunk)) * 3.0).astype(np.float32)
    c_twin.smooth(y[:, :, :64].copy(), **mod, nthreads=cores)         # warm-up
    done, t0 = 0, time.perf_counter()
    while True:
        c_twin.smooth(y, **mod, nthreads=cores)
        done += chunk
        el = time.perf_counter() - t0
        if el >= seconds_target or done >= BATCH:
            break
    # BASELINE configs[0]: ONE chain (d = 4, T = 1000) on one core -- the reference's own CPU-runnable case; its
    # published time for one d = 2 chain is 77.231 ms (benchmarks/...ipynb:799), this allocation-free port needs ~1 ms
    y1 = y[:, :, :1].copy()
    c_twin.smooth(y1, **mod, nthreads=1)
    t1 = time.perf_counter()
    for _ in range(50):
        c_twin.smooth(y1, **mod, nthreads=1)
    one_ms = (time.perf_counter() - t1) / 50 * 1e3
    return {"parity": parity, "value": MSG_PER_STEP * T * done / el, "unit": "messages/s", "cores": cores, "kind": "port",
            "sample": f"{done} chains x T={T} (d=4) of the same workload, fp64 C port of the reference schedule "
                      f"(oracle/c/rxg_oracle.c), OpenMP over chains, {el:.1f} s",
            "single_chain_ms": one_ms, "single_chain_note": "configs[0]: one chain d=4 T=1000 on one core; the reference "
            "publishes 77.231 ms for one d=2 chain (ipynb:799): the C port is an optimistic stand-in"}


def run_reference_arm(args, rank, world, emit=lambda o: print(json.dumps(o))):
    """--impl reference: the reference's CPU path = the fp64 C port (the Julia reference cannot be
    installed: no julia, no registry packages; see DESIGN.md).  Rank 0 only."""
    if rank != 0:
        return
    from oracle import c_twin
    mod = {k: v.astype(np.float64) for k, v in notebook_model_f32().items()}
    cores = host_cores()
    chunk = 4096                                     # bounded sample per step
    rng = np.random.default_rng(0)
    y = (rng.standard_normal((T, M, chunk)) * 3.0).astype(np.float32)
    for _ in range(max(args.warmup, 1)):
        c_twin.smooth(y[:, :, :512].copy(), **mod, nthreads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        c_twin.smooth(y, **mod, nthreads=cores)
    el = time.perf_counter() - t0
    val = MSG_PER_STEP * T * chunk * args.steps / el
    sample = f"{chunk} chains x T={T} per step (1/{BATCH // chunk} of the GPU arm's per-GPU batch), fp64, OpenMP x{cores}"
    emit(({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "messages/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "batched LGSSM smoothing d=4 m=4 T=1000, notebook model, shared parameters",
                   "sample": sample},
        "cpu_baseline": {"value": val, "unit": "messages/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "messages/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def bench_other_config(args, ctx, dev, emit):
    """BASELINE configs[2] (d = 64, T = 1000, batch = 4096, contract output: per-chain covariances) and configs[3]
    (HGF, T = 1000, batch = 32 768, 20 VMP iterations): same timing protocol and JSON keys as the headline line."""
    import torch
    sampler = ClockSampler(dev.index or 0)
    g = torch.Generator(device=dev).manual_seed(7)
    peak, peak_src = peaks()

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launches
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps, ctx.launches - l0, sampler.stop()

    if args.config == 2:
        d, batch = 64, 4096
        md = dense_model_f32(d)
        y = torch.randn(T, d, batch, device=dev, generator=g) * 3.3
        mean = torch.empty(T, d, batch, device=dev)
        cov = torch.empty(T, d, d, batch, device=dev)            # 67 GB: the contract output
        ctx.set_profiling(True)
        parts = []
        def step():
            ctx.lgssm(y, **md, smooth=True, out_mean=mean, out_cov=cov, asynchronous=True)
        ms, launches, clocks = timed(step)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"mean": mean[None], "cov": cov[None]})
        for _ in range(3):
            step(); parts.append(ctx.profile_last_ms())
        sweep_ms, gain_ms = float(np.mean([p[0] for p in parts])), float(np.mean([p[1] for p in parts]))
        bcast_ms = ms - gain_ms - sweep_ms        # the covariance broadcast follows the sweep on the same stream
        algo = 4 * (d + d + d * d) * T * batch
        cov_bytes = 4 * d * d * T * batch
        out = {"metric": "gaussian_messages_per_sec_batched_lgssm_d64_T1000", "value": MSG_PER_STEP * T * batch / (ms * 1e-3),
               "unit": "messages/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (tensor pipe: 3xTF32 split, fp32 accumulate; gain tables fp64)",
               "data": "synthetic",
               "config": {"workload": "BASELINE configs[2]: LGSSM d=64 m=64 T=1000 batch=4096, dense A = 0.99 Orth, shared model; "
                                      "contract output = per-chain covariances [T][64][64][4096] (67 GB)",
                          "l2_policy": "outputs (68 GB) larger than L2", "data_note": "y = randn * 3.3"},
               "roofline": {"bound": "hbm", "kernel": "broadcast_cov_kernel (per-chain covariance materialisation)",
                            "achieved": cov_bytes / (bcast_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                            "frac": cov_bytes / (bcast_ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                            "kernel_ms": bcast_ms, "algorithmic_bytes_per_launch": cov_bytes,
                            "whole_step_frac": algo / (ms * 1e-3) / 1e9 / peak,
                            "breakdown_ms": {"gain_tables_fp64": gain_ms, "mean_sweep_tcgen05": sweep_ms, "covariance_broadcast": bcast_ms},
                            "mean_sweep_TFLOPs": 8 * d * d * T * batch / (sweep_ms * 1e-3) / 1e12},
               "e2e": None, "e2e_note": "not measured for this config: the contract output alone is 67 GB of pinned host memory",
               "gpu_launches": int(launches), "clocks": clocks}
        emit(out)
        return
    # config 3: HGF
    batch, iters = 32768, 20
    yh = (torch.randn(T, batch, device=dev, generator=g).cumsum(0) * 0.5).contiguous()
    outb = torch.empty(T, 4, batch, device=dev)
    ms, launches, clocks = timed(lambda: ctx.hgf_filter(yh, iters=iters, out=outb))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"out": outb[None]})
    msgs = 6 * iters * T * batch
    # end to end: host observations in, host posteriors out through the same entry point
    yhh = torch.empty(T, batch).pin_memory(); yhh.copy_(yh)
    outh = torch.empty(T, 4, batch).pin_memory()
    ydev = torch.empty_like(yh)
    def e2e_step():
        ydev.copy_(yhh, non_blocking=True)
        ctx.hgf_filter(ydev, iters=iters, out=outb)
        outh.copy_(outb, non_blocking=True)
    e2e_step(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        e2e_step()
    e1.record(); torch.cuda.synchronize()
    e_ms = e0.elapsed_time(e1) / 3
    io = 20 * T * batch
    out = {"metric": "gaussian_messages_per_sec_hgf_T1000_20its", "value": msgs / (ms * 1e-3), "unit": "messages/s", "n_gpus": 1,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "BASELINE configs[3]: Hierarchical Gaussian Filter (GCV node, GH-31), T=1000 batch=32768, 20 VMP iterations per datum",
                      "vmp_iterations_per_s": iters * T * batch / (ms * 1e-3), "exp_per_s": (31 + 1 + iters * 32) * T * batch / (ms * 1e-3),
                      "messages_per_chain_step_iteration": 6},
           "roofline": {"bound": "hbm", "kernel": "hgf_filter_kernel", "achieved": io / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": io / (ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src, "kernel_ms": ms,
                        "algorithmic_bytes_per_launch": io,
                        "note": "SFU / FP32-issue bound (652 ex2 + ~5 k FMA per 20 B of I/O): the HBM fraction is not the meaningful "
                                "ceiling here (SURVEY.md 8d); see profiles/ for the pipe utilisation"},
           "e2e": {"value": msgs / (e_ms * 1e-3), "unit": "messages/s", "ms_per_step": e_ms, "h2d_bytes_per_step": int(yhh.numel() * 4),
                   "d2h_bytes_per_step": int(outh.numel() * 4)},
           "gpu_launches": int(launches), "clocks": clocks}
    emit(out)


def main():
    # keep stdout clean for the ONE JSON line: libraries (NCCL's version banner, torchrun notes) print to
    # fd 1 as well, so everything else is routed to stderr and the result goes to the saved descriptor
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH, help="chains per GPU (default = BASELINE config)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--per-chain-path", action="store_true", help="time the per-chain covariance recursion instead")
    ap.add_argument("--config", type=int, default=1, choices=[1, 2, 3],
                    help="BASELINE.json configs[] index: 1 = headline (d=4, batch 65536), 2 = d=64 batch 4096 (tensor-core family), "
                         "3 = HGF T=1000 batch 32768, 20 VMP iterations")
    ap.add_argument("--sweep-variant", type=int, default=0, help="RXG_OPT_SWEEP_VARIANT (0 auto, 1 stash, 2 checkpoint, 3/4 time-segmented)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy "
                    f"(float32; a fixed seeded sample of the chains when all of them exceed {DUMP_BYTES // 10**6} MB)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the CUDA path's outputs (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world, emit)
        return

    import torch
    import torch.distributed as dist
    import rxinfer_jl_b200 as rx

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    ctx = rx.Context(local)
    if args.sweep_variant:
        ctx.set_option("sweep_variant", args.sweep_variant)
    if args.config != 1:
        if world > 1:
            raise SystemExit("bench.py --config 2/3 are single-GPU configurations")
        return bench_other_config(args, ctx, dev, emit)
    mod = notebook_model_f32()
    batch = args.batch
    kw = dict(A=mod["A"], B=mod["B"], P=mod["P"], Q=mod["Q"], m0=mod["m0"], S0=mod["S0"])

    # synthetic observations of the model's own scale (state O(1), obs noise sd sqrt(10)); generated on device
    g = torch.Generator(device=dev).manual_seed(42 + rank)
    y = torch.randn(T, M, batch, device=dev, generator=g) * 3.3
    if world == 1:
        mean = torch.empty(T, D, batch, device=dev)
        cov = torch.empty(T, D, D, batch, device=dev)

    # N > 1: the north_star all-gather of posterior marginals is PART of the step.  Every rank maps its peers'
    # gathered buffers (CUDA IPC over NVLink) and the sweep kernel stores the posteriors into all of them while it
    # runs (rxg_lgssm_smooth_gather_f32); `value` is the literal full gather (means AND per-chain covariances cross
    # NVLink), the RXG_COV_REPLICATE variant (bit-identical buffers, covariances replicated locally) is reported as
    # `gather.replicated_cov`, the sweep without any gather as `gather.sweep_only`.
    grp = None
    if world > 1:
        from rxinfer_jl_b200.sharding import PeerGroup
        grp = PeerGroup(ctx, T, D, batch)                     # 8 GPUs: 42 GB of gathered posteriors per GPU
        mean, cov = grp.mean[rank], grp.cov[rank]             # the plain sweep writes this rank's slab

    def step():
        return ctx.lgssm(y, **kw, smooth=True, out_mean=mean, out_cov=cov, asynchronous=True,
                         force_per_chain_path=args.per_chain_path)

    def step_gather(replicate):
        return grp.smooth_gather(y, mod, replicate_cov=replicate, asynchronous=True,
                                 force_per_chain_path=args.per_chain_path)

    def timed(fn, steps):
        """K steps between two events on the launching stream, barrier + synchronize on both sides, max over ranks."""
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0_ = ctx.launches
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t_ = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t_, op=dist.ReduceOp.MAX)
        return float(t_.item()) / steps, ctx.launches - l0_

    ctx.set_profiling(True)
    for _ in range(args.warmup):
        step()
        if world > 1:
            step_gather(False); step_gather(True)
    ctx.sync()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    msgs = MSG_PER_STEP * T * batch * world
    gather = None
    if world == 1:
        ms_per_step, launches = timed(step, args.steps)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"mean": mean[None], "cov": cov[None]})
    else:
        ms_per_step, launches = timed(lambda: step_gather(False), args.steps)          # contract: full gather in the step
        if args.dump_outputs and rank == 0:                   # the peers wait at the next timed() barrier
            dump_outputs(args.dump_outputs, {"mean": grp.mean, "cov": grp.cov})
        ms_rep, l_rep = timed(lambda: step_gather(True), args.steps)
        ms_sweep, _ = timed(step, args.steps)
        slab = (mean.numel() + cov.numel()) * 4
        # correctness of what was just timed: every slab of this rank's buffers equals an independent sweep of that shard
        step_gather(False); ctx.sync(); dist.barrier()
        own_mean, own_cov = mean.clone(), cov[:8].clone()
        chk = [grp.mean[r][::97].clone() for r in range(world)]
        chk_c = [grp.cov[r][:4].clone() for r in range(world)]
        grp.mean.zero_(); grp.cov.zero_(); torch.cuda.synchronize(); dist.barrier()
        step_gather(True); ctx.sync(); dist.barrier()
        assert torch.equal(grp.mean[rank], own_mean) and torch.equal(grp.cov[rank][:8], own_cov)
        assert all(torch.equal(grp.mean[r][::97], chk[r]) and torch.equal(grp.cov[r][:4], chk_c[r]) for r in range(world)), \
            "RXG_COV_REPLICATE buffers differ from the full gather"
        assert bool((grp.mean[(rank + 1) % world].abs().sum() > 0).item())
        del own_mean, own_cov, chk, chk_c
        gather = {
            "in_value": "full gather: (G-1) x (means + per-chain covariances) stored over NVLink by the sweep kernel itself",
            "ms_per_step_full": ms_per_step, "nvlink_bytes_out_per_gpu_full": (world - 1) * slab,
            "nvlink_GBs_out_per_gpu_full": (world - 1) * slab / ms_per_step / 1e6,
            "replicated_cov": {"ms_per_step": ms_rep, "value": msgs / (ms_rep * 1e-3), "gpu_launches": int(l_rep),
                               "nvlink_bytes_out_per_gpu": (world - 1) * mean.numel() * 4,
                               "nvlink_GBs_out_per_gpu": (world - 1) * mean.numel() * 4 / ms_rep / 1e6,
                               "note": "RXG_COV_REPLICATE: shared model => covariances chain independent; means over NVLink, "
                                       "covariance slabs replicated locally during the sweep; buffers bit-identical (asserted)"},
            "sweep_only": {"ms_per_step": ms_sweep, "value": msgs / (ms_sweep * 1e-3),
                           "note": "no gather (round-1 headline); NOT the contract at N > 1"},
            "nvlink_floor_ms": {"full": (world - 1) * slab / 770e9 * 1e3, "replicated_cov": (world - 1) * mean.numel() * 4 / 770e9 * 1e3,
                                "note": "bytes that must arrive per GPU / 770 GB/s measured peer bandwidth (B200_PROFILING.md)"},
        }
        # the round-1 design for comparison: sweep, then ncclAllGather of the finished posteriors (into the same buffers)
        try:
            rx.sharding.init_comm(ctx)
            ctx.allgather_posteriors(mean, cov, world, out_mean=grp.mean, out_cov=grp.cov)
            def nccl_step():
                step()
                ctx.allgather_posteriors(mean, cov, world, out_mean=grp.mean, out_cov=grp.cov)
            ms_nccl, _ = timed(nccl_step, max(2, min(args.steps, 3)))
            gather["nccl_after_sweep"] = {"ms_per_step": ms_nccl, "value": msgs / (ms_nccl * 1e-3),
                                          "note": "round-1 design: plain ncclAllGather issued after the sweep (in place, same buffers)"}
        except Exception as ex:       # noqa: BLE001 -- a comparison leg only
            gather["nccl_after_sweep"] = {"error": str(ex)[:200]}
    value = msgs / (ms_per_step * 1e-3)
    # per-kernel timing of the dominant kernel: separate pass so the event syncs do not sit in the timed loop
    main_ms, gain_ms = [], []
    for _ in range(args.steps):
        step()
        a, b = ctx.profile_last_ms()
        main_ms.append(a); gain_ms.append(b)
    # parity of the timed workload itself: sampled chains of the buffers the timed loop wrote go to the CPU leg below,
    # where the fp64 port recomputes them (the oracle is only ever executed inside cpu_baseline())
    parity_sample = None
    if rank == 0 and not args.no_cpu:
        idx = [0, 1, batch // 2 + 1, batch - 1]
        step(); ctx.sync()
        parity_sample = {"chains": idx, "y": y[:, :, idx].cpu().numpy(), "mean": mean[:, :, idx].cpu().numpy(),
                         "cov": cov[:, :, :, idx].cpu().numpy()}

    # ---- e2e through the C ABI with host buffers (rank-local; all ranks run it concurrently)
    e2e = None
    if not args.no_e2e:
        try:
            # host buffers from the library's own allocator (pinned; NUMA-interleaved on multi-socket hosts), as a C /
            # Julia host of the ABI would obtain them
            from rxinfer_jl_b200.context import host_empty
            yh = host_empty(T, M, batch)
            yh.copy_(y)
            mh = host_empty(T, D, batch)
            ch = host_empty(T, D, D, batch)
        except (RuntimeError, rx.RxGaussError) as ex:       # pinned host memory exhausted (8 ranks x 6.3 GB): report, do not die
            yh = None
            e2e = {"value": None, "unit": "messages/s", "error": f"pinned host allocation failed: {ex}"[:200]}
        if yh is not None:
            e_steps = max(2, min(args.steps, 5))
            ctx.lgssm(yh, **kw, smooth=True, out_mean=mh, out_cov=ch)           # warm-up (staging alloc)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(e_steps):
                ctx.lgssm(yh, **kw, smooth=True, out_mean=mh, out_cov=ch, asynchronous=True)
            e1.record(); torch.cuda.synchronize()
            te = torch.tensor([e0.elapsed_time(e1) / e_steps], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            bcast = ctx.get_option("host_cov_d2h") == 0 and ctx.host_fill_threads() >= 4
            e2e = {"value": msgs / (float(te.item()) * 1e-3), "unit": "messages/s", "ms_per_step": float(te.item()),
                   "h2d_bytes_per_step": int(yh.numel() * 4),
                   "d2h_bytes_per_step": int((mh.numel() + (T * D * D if bcast else ch.numel())) * 4),
                   "host_bytes_written_per_step": int((mh.numel() + ch.numel()) * 4),
                   "api": "rxg_lgssm_smooth_f32 with host pointers (rxg_host_alloc: pinned, NUMA-interleaved), sliced 3-stream pipeline; " +
                          ("per-chain covariances (chain independent for the shared model) fetched once as a [T][d][d] table "
                           "and broadcast into the caller's buffer by %d host threads" % ctx.host_fill_threads() if bcast else
                           "full device->host copy of the per-chain covariances")}
            # the same call with the covariance broadcast disabled: every byte of the per-chain covariances over PCIe
            if bcast:
                ctx.set_option("host_cov_d2h", 1)
                ctx.lgssm(yh, **kw, smooth=True, out_mean=mh, out_cov=ch)
                torch.cuda.synchronize()
                if world > 1:
                    dist.barrier()
                e0.record()
                for _ in range(e_steps):
                    ctx.lgssm(yh, **kw, smooth=True, out_mean=mh, out_cov=ch, asynchronous=True)
                e1.record(); torch.cuda.synchronize()
                ctx.set_option("host_cov_d2h", 0)
                tf_ = torch.tensor([e0.elapsed_time(e1) / e_steps], device=dev, dtype=torch.float64)
                if world > 1:
                    dist.all_reduce(tf_, op=dist.ReduceOp.MAX)
                e2e["full_d2h"] = {"value": msgs / (float(tf_.item()) * 1e-3), "ms_per_step": float(tf_.item()),
                                   "d2h_bytes_per_step": int((mh.numel() + ch.numel()) * 4)}
            # same call with RXG_COV_SHARED_OUT: the chain-independent covariances come back once ([T][d][d])
            # instead of per chain -- what a host binding that aliases one matrix per time step would request
            del ch
            cs = host_empty(T, D, D)
            ctx.lgssm(yh, **kw, smooth=True, out_mean=mh, out_cov=cs, cov_shared_out=True)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            e0.record()
            for _ in range(e_steps):
                ctx.lgssm(yh, **kw, smooth=True, out_mean=mh, out_cov=cs, cov_shared_out=True, asynchronous=True)
            e1.record(); torch.cuda.synchronize()
            ts = torch.tensor([e0.elapsed_time(e1) / e_steps], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(ts, op=dist.ReduceOp.MAX)
            e2e["shared_cov_out"] = {"value": msgs / (float(ts.item()) * 1e-3), "ms_per_step": float(ts.item()),
                                     "d2h_bytes_per_step": int((mh.numel() + cs.numel()) * 4),
                                     "note": "RXG_COV_SHARED_OUT: posterior covariances de-duplicated over chains (not the contract output)"}
            del yh, mh, cs
        elif world > 1:
            dist.barrier()
    if grp is not None:
        grp.close()

    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        peak, peak_src = peaks()
        k_ms = float(np.mean(main_ms))
        algo = ALGO_BYTES_PER_STEP * T * batch
        achieved = algo / (k_ms * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic_bytes.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("per_chain_path" if args.per_chain_path else "shared_path")
        out = {
            "metric": METRIC, "value": value, "unit": "messages/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "batched LGSSM smoothing (BASELINE configs[1]): d=4 m=4 T=1000 batch=%d per GPU, "
                                   "notebook model lifted to d=4, shared (A,B,P,Q,prior)" % batch,
                       "global_batch": batch * world,
                       "parallelism": (f"batch-sharded x{world}; all-gather of posterior marginals INSIDE the timed step "
                                       "(peer-mapped NVLink stores fused into the sweep kernel, device-side barrier)") if world > 1
                                      else "single GPU (no gather needed: the posteriors are already where they end up)",
                       "data_note": "y = randn * 3.3 per chain (the model's observation scale), not sampled from the model: the "
                                    "sweep is linear in y, timing is value independent; parity of the timed buffers is checked "
                                    "against the fp64 oracle on sampled chains (`parity`)",
                       "path": "per-chain covariance recursion" if args.per_chain_path else "gain tables + mean sweeps",
                       "sweep_variant": ctx.get_option("sweep_variant"),
                       "messages_per_chain_step": MSG_PER_STEP, "l2_policy": "inputs+outputs (6.3 GB) larger than L2"},
            "roofline": {"bound": "hbm", "kernel": "lgssm_chain_kernel" if args.per_chain_path else "lgssm_shared_kernel",
                         "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "kernel_ms": k_ms, "gain_kernels_ms": float(np.mean(gain_ms)),
                         "algorithmic_bytes_per_launch": algo},
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        }
        if gather:
            out["gather"] = gather
        if not args.no_cpu:
            out["cpu_baseline"] = cpu_baseline(parity_sample=parity_sample)
            out["parity"] = out["cpu_baseline"].pop("parity", None)
        emit(out)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
