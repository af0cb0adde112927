#!/usr/bin/env python
"""bench.py -- images/s of the TaskPrompter ViT-L PASCAL-Context forward (BASELINE.json configs[3],
512x512, 5 tasks, bs 4 per GPU) on N B200s of one node, one process per GPU.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps K --warmup W      # CPU arm (oracle port of the reference)
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # also write the last timed step's outputs

A "step" is one forward pass over one synthetic batch (the hot path named by BASELINE.json's
north_star; the reference publishes no throughput, so vs_baseline is null). Rank 0 prints ONE JSON
line. `value` = whole-job images/s with inputs resident in HBM; `e2e` = the same through the public
nn.Module call with pinned-host inputs (H2D) and a D2H read of every task's logits inside the timed
region. The forward shards over the batch with no collective (weak scaling): NCCL is used only for
the start/stop barrier and the max-over-ranks time.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

_OUT = sys.stdout  # main() replaces it with a duplicate of the original stdout
GFLOP_PER_IMAGE = {"tp_cfg4": 993.2, "tp_cfg2": 1163.5, "tp_cfg5": 12842.7, "ip_cfg3": 1344.8,
                   "tps_swinB": 3678.8}  # SURVEY.md 8(d); tps_swinB: FlopCounterMode over the oracle forward (bs 1)
WORKLOAD = {
    "tp_cfg4": "TaskPrompter ViT-L PASCAL-Context (5 tasks) 512x512 forward",
    "tp_cfg2": "TaskPrompter ViT-B NYUD-v2 (4 tasks) 448x576 forward",
    "tp_cfg5": "TaskPrompter ViT-L Cityscapes-3D shape (seg + depth + 18-channel 3ddet ConvHead stand-in) 1024x2048 forward",
    "ip_cfg3": "InvPT ViT-L PASCAL-Context (5 tasks) 512x512 forward",
    "tps_swinB": "TaskPrompter Swin-B Cityscapes-3D shape (seg + depth, DEConvHead) 1024x2048 forward",
}
DEFAULT_BATCH = {"tp_cfg4": 4, "tp_cfg2": 4, "tp_cfg5": 1, "ip_cfg3": 4, "tps_swinB": 1}


def family(cfg_name):
    """(config dict, product module, oracle module) for a named configuration."""
    from mtt_b200 import configs
    if cfg_name.startswith("ip_"):
        from mtt_b200 import invpt as M
        return configs.invpt(cfg_name), M, "oracle.invpt_ref"
    if cfg_name.startswith("tps_"):
        from mtt_b200 import taskprompter_swin as M
        return configs.taskprompter_swin(cfg_name), M, "oracle.taskprompter_swin_ref"
    from mtt_b200 import taskprompter as M
    return configs.taskprompter(cfg_name), M, "oracle.taskprompter_ref"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def dump_outputs(path, outs, limit=64 * 10**6):
    """Writes every output tensor as <path>/<name>.npy in float32 (rank 0's last timed step). When they exceed `limit`
    bytes in all, each is cut to the same fraction of its elements, at flat indices drawn (sorted) from a generator with
    a fixed seed, so two runs of the same command write the same positions."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    host = {k: v.detach().float().cpu() for k, v in outs.items()}
    keep = min(1.0, (limit - 4096 * len(host)) / (4 * sum(v.numel() for v in host.values())))
    for k, v in host.items():
        if keep < 1.0:
            idx = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(0))[:int(v.numel() * keep)]
            v = v.reshape(-1)[idx.sort().values]
        np.save(os.path.join(path, f"{k}.npy"), v.numpy())


# ------------------------------------------------------------------------------------------------
def pick_cpu_threads():
    """Eager PyTorch on a many-core host collapses when over-subscribed (measured on the 128-thread GPU
    box: 16 threads 0.61 s, 64 threads 1.4 s, 128 threads 56 s for the same 4-block slice), so the CPU arm
    uses the thread count that is actually fastest for this workload, found on a short slice."""
    from mtt_b200 import configs
    from oracle import taskprompter_ref as TPR

    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu})
    if len(cands) == 1:
        return cands[0]
    cfg = configs.taskprompter("tp_cfg4_d4")
    cfg["depth"], cfg["select"] = 3, [1, 2, 3]
    sd = TPR.init_state_dict(cfg, seed=0)
    x = torch.randn(1, 3, *cfg["img_size"], generator=torch.Generator().manual_seed(1))
    best, best_t = cands[0], float("inf")
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            TPR.forward(sd, cfg, x)
            t0 = time.perf_counter()
            TPR.forward(sd, cfg, x)
            dt = time.perf_counter() - t0
            if dt < best_t:
                best, best_t = c, dt
            if dt > 4 * best_t:
                break
    return best


def reference_forward(cfg_name, device="cpu"):
    """A callable x -> outputs running the reference algorithm in eager PyTorch on `device`, and its kind:
    "reference" = the UNMODIFIED reference model imported through oracle/shim (only where /root/reference or
    $MTT_REFERENCE or baseline/_ref exists -- not on the GPU box), "port" = the oracle restatement."""
    import importlib

    from oracle import ref_loader
    cfg, _, oracle_name = family(cfg_name)
    R = importlib.import_module(oracle_name)
    sd = R.init_state_dict(cfg, seed=0)
    if ref_loader.available():
        build = (ref_loader.build_invpt if cfg_name.startswith("ip_") else
                 ref_loader.build_taskprompter_swin if cfg_name.startswith("tps_") else ref_loader.build_taskprompter)
        model = build(cfg).eval()
        model.load_state_dict(sd, strict=not cfg_name.startswith("tps_"))   # Swin: index / mask buffers are derived
        model = model.to(device)
        return (lambda x: model(x)), "reference", cfg
    sd = {k: v.to(device) for k, v in sd.items()}
    return (lambda x: R.forward(sd, cfg, x)), "port", cfg


def cpu_oracle_rate(cfg_name, steps, warmup, threads, batch=1):
    """images/s of the reference's eager fp32 CPU forward (the unmodified reference where importable, else its
    port oracle/*_ref.py) on a bounded sample: `batch` images of the same workload per step."""
    torch.set_num_threads(threads)
    fwd, kind, cfg = reference_forward(cfg_name, "cpu")
    x = torch.randn(batch, 3, *cfg["img_size"], generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        for _ in range(warmup):
            fwd(x)
        t0 = time.perf_counter()
        for _ in range(steps):
            fwd(x)
        dt = time.perf_counter() - t0
    return batch * steps / dt, dt / steps, kind


def gpu_eager_baseline(cfg_name, batch, dev, steps=5, warmup=2):
    """The library-call baseline SURVEY.md 2.2 / 8(d) sets: the reference algorithm in eager PyTorch (cuBLAS / cuDNN)
    on the SAME B200, same batch, CUDA-event timed: fp32 with TF32 off (the reference's arithmetic), TF32 on, and
    bf16 autocast. A baseline leg like cpu_baseline -- nothing here is on the product path."""
    fwd, kind, cfg = reference_forward(cfg_name, dev)
    x = torch.randn(batch, 3, *cfg["img_size"], device=dev)
    res = {"kind": kind, "batch": batch, "steps": steps, "warmup": warmup, "unit": "images/s",
           "what": "eager PyTorch forward of the reference algorithm on this GPU (cuBLAS / cuDNN kernels)"}
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)

    def timed(ctx):
        with torch.no_grad(), ctx:
            for _ in range(warmup):
                fwd(x)
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(steps):
                fwd(x)
            e.record()
            torch.cuda.synchronize()
        return batch * steps / (s.elapsed_time(e) * 1e-3)

    import contextlib
    try:
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        res["fp32"] = timed(contextlib.nullcontext())
        torch.backends.cuda.matmul.allow_tf32 = True
        torch.backends.cudnn.allow_tf32 = True
        res["tf32"] = timed(contextlib.nullcontext())
        res["bf16_autocast"] = timed(torch.autocast("cuda", dtype=torch.bfloat16))
    except Exception as ex:  # e.g. out of memory at cfg5: report what ran
        res["error"] = f"{type(ex).__name__}: {ex}"[:200]
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    return res


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = pick_cpu_threads()
    B = args.batch
    rate, sec, kind = cpu_oracle_rate(args.config, args.steps, args.warmup, threads, batch=B)
    what = "the unmodified reference model" if kind == "reference" else "CPU port of the reference forward (oracle/)"
    sample = (f"batch {B} of {args.config} per step (fp32 eager CPU, eval, {what}), {args.warmup} warm-up + "
              f"{args.steps} timed steps, {threads} of {os.cpu_count()} host threads (fastest setting, see pick_cpu_threads)")
    line = {
        "impl": "reference", "metric": "images/sec", "value": rate, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{WORKLOAD[args.config]}, {args.config}, bs {B}/GPU, random-init weights, eval",
                   "global_batch": B, "parallelism": "one CPU process (rank 0), host threads as stated",
                   "precision_mode": "fp32 eager CPU"},
        "cpu_baseline": {"value": rate, "unit": "images/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": rate, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=_OUT, flush=True)


# ------------------------------------------------------------------------------------------------
def gemm_roofline(model, plan, x_dev, peaks, peak_src):
    """Average duration and algorithmic FLOPs of the dominant kernel family (the tcgen05 GEMM / implicit-GEMM
    conv kernels: every mtt_gemm launch of one forward, including those inside the composite block operators),
    measured live with CUDA events recorded by the library around each launch on the launching stream
    (mtt_profile_begin / mtt_profile_end).

    The forward is enqueued eagerly on ONE stream behind a device-side blocker, so the whole launch queue is
    resident before the first kernel runs and the events bracket device time only (without the blocker an
    eager pass measures the host's per-launch latency instead: 102 us / launch against 44 us real)."""
    from mtt_b200 import ops

    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    plan.serial = True
    try:
        plan._launch(x_dev)   # warm
        torch.cuda.synchronize()
        torch.cuda._sleep(int(60e6))   # ~30 ms of device time: the host enqueues the whole forward meanwhile
        ops.profile_begin()
        f0.record()
        plan._launch(x_dev)
        f1.record()
        prof = ops.profile_end()
    finally:
        plan.serial = False

    class _R:      # (ms, flops, backbone?) records in the shape the summary below expects
        def __init__(self, ms):
            self.ms = ms

        def elapsed_time(self, other):
            return self.ms

    recs = [(_R(ms), None, fl, min(N, K) >= 1024) for kind, M, N, K, ms, fl in prof if kind == 0]
    arecs = [(_R(ms), None, fl) for kind, M, N, K, ms, fl in prof if kind == 1]
    fwd_ms = f0.elapsed_time(f1)
    tot_ms = sum(s.elapsed_time(e) for s, e, _, _ in recs)
    tot_fl = sum(f for _, _, f, _ in recs)
    bb_ms = sum(s.elapsed_time(e) for s, e, _, bb in recs if bb)
    bb_fl = sum(f for _, _, f, bb in recs if bb)
    achieved = tot_fl / (tot_ms * 1e-3) / 1e12
    peak = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
    mma_factor = 3 if model.nsplit == 2 else 1
    # DRAM bytes per launch of the same kernel family, from the committed ncu capture of one forward of this workload
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if (os.path.exists(tpath) and model.nsplit == 2 and tuple(x_dev.shape) == (4, 3, 512, 512)
            and type(model).__name__ == "TaskPrompterWrapper"):
        with open(tpath) as f:
            tj = json.load(f)
        traffic = tj["gemm_family"]["bytes_per_launch"]
        traffic_src = ("dram__bytes_read.sum + dram__bytes_write.sum averaged over the %d GEMM / conv launches of one "
                       "tp_cfg4 bs 4 forward (profiles/dram_traffic.json <- %s)" % (tj["gemm_family"]["launches"],
                                                                                    tj.get("source", "").rsplit(", ", 1)[-1]))
    bb = bb_fl / (bb_ms * 1e-3) / 1e12 if bb_ms > 0 else None
    at_ms = sum(s.elapsed_time(e) for s, e, _ in arecs)
    at = sum(f for _, _, f in arecs) / (at_ms * 1e-3) / 1e12 if at_ms > 0 else None
    return {
        "bound": "tensor",
        "kernel": "gemm_tc_kernel + gemm2_tc_kernel (every GEMM / implicit-GEMM conv launch of one forward)",
        "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
        "peak_source": f"bf16 dense sustained, {peak_src}", "traffic": traffic, "traffic_unit": "bytes per launch",
        "traffic_source": traffic_src,
        "launches": len(recs), "avg_launch_us": tot_ms * 1e3 / len(recs),
        "share_of_forward": tot_ms / fwd_ms, "serial_forward_ms": fwd_ms,
        "issued_mma_tflops": achieved * mma_factor, "issued_mma_frac": achieved * mma_factor / peak,
        "backbone_gemms": None if bb is None else {
            "launches": sum(1 for r in recs if r[3]), "achieved": bb, "issued_mma_tflops": bb * mma_factor,
            "issued_mma_frac": bb * mma_factor / peak, "avg_launch_us": bb_ms * 1e3 / sum(1 for r in recs if r[3])},
        "attention": None if at is None else {
            "kernel": "attention5_kernel (fused QK^T / softmax / PV, one launch per transformer block)", "launches": len(arecs),
            "avg_launch_us": at_ms * 1e3 / len(arecs), "achieved": at, "issued_mma_tflops": at * mma_factor,
            "issued_mma_frac": at * mma_factor / peak, "share_of_forward": at_ms / fwd_ms,
            "flops": "4*B*H*N*N*64 per launch (QK^T + PV)"},
        "note": ("achieved counts the reference's ALGORITHMIC fp32 FLOPs (2*M*N*K*taps per launch, DESIGN.md); the "
                 f"parity mode issues {mma_factor} bf16 tcgen05.mma per product (issued_mma_*); one eager forward on a "
                 "single stream behind a device-side blocker, CUDA events around every launch; backbone_gemms = the "
                 "qkv / proj / fc1 / fc2 launches alone"),
    }


def run_ours(args):
    import mtt_b200  # noqa: F401
    from mtt_b200 import dist as D
    from mtt_b200 import ops

    rank, world, local = D.setup("nccl")
    barrier, max_over_ranks = D.barrier, D.max_over_ranks
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    cfg, M, _ = family(args.config)
    nsplit = 2 if args.mode == "parity" else 1
    torch.manual_seed(0)
    with torch.device(dev):
        model = M.build_from_config(cfg, nsplit=nsplit, use_graph=True).eval()
    B = args.batch
    H, W = cfg["img_size"]
    n_rot = 4
    g = torch.Generator().manual_seed(1 + rank)
    host_in = [torch.randn(B, 3, H, W, generator=g).pin_memory() for _ in range(n_rot)]
    dev_in = [h.to(dev) for h in host_in]
    plan = model.plan(B, dev)
    with torch.no_grad():
        out = model(dev_in[0])
    torch.cuda.synchronize()
    launches_per_fwd = plan.launches_per_forward()
    torch.cuda.synchronize()

    def flat(o):      # InvPT returns {'task': ..., 'inter_preds': {'task': ...}}: every tensor is read back
        r = {}
        for k, v in o.items():
            if isinstance(v, dict):
                r.update({f"{k}.{k2}": v2 for k2, v2 in v.items()})
            else:
                r[k] = v
        return r

    # ---------------- device-resident throughput ("value")
    with torch.no_grad():
        for i in range(args.warmup):
            model(dev_in[i % n_rot])
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # `repeats` timed regions of EXACTLY `steps` steps each (barrier + synchronize on both sides, max over ranks);
    # the reported region is the median one, so a single power-cap excursion does not move the headline
    regions = []
    for _ in range(max(1, args.repeats)):
        barrier(world)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        with torch.no_grad():
            for i in range(args.steps):
                last = model(dev_in[i % n_rot])
        e.record()
        torch.cuda.synchronize()
        barrier(world)
        regions.append(max_over_ranks(s.elapsed_time(e), world, dev))
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, flat(last))   # before the next call reuses the output buffers
    del last
    ms_total = sorted(regions)[len(regions) // 2]
    value = world * B * args.steps / (ms_total * 1e-3)

    # ---------------- end to end through the public call, host buffers, H2D + D2H inside the timed region
    out = flat(out)
    out_bytes = sum(v.numel() * v.element_size() for v in out.values())
    in_bytes = host_in[0].numel() * 4
    host_out = [{k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in out.items()} for _ in range(2)]
    stage = [{k: torch.empty_like(v) for k, v in out.items()} for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    d2h_done = [torch.cuda.Event(), torch.cuda.Event()]
    staged = [torch.cuda.Event(), torch.cuda.Event()]

    def e2e_steps(n):
        main = torch.cuda.current_stream()
        for i in range(n):
            j = i & 1
            x = host_in[i % n_rot].to(dev, non_blocking=True)        # H2D from pinned memory
            with torch.no_grad():
                o = flat(model(x))                                   # public nn.Module call
            main.wait_event(d2h_done[j])                             # staging buffer j is free again
            for k in o:
                stage[j][k].copy_(o[k], non_blocking=True)
            staged[j].record(main)
            with torch.cuda.stream(copy_stream):                     # D2H overlaps the next step
                copy_stream.wait_event(staged[j])
                for k in o:
                    host_out[j][k].copy_(stage[j][k], non_blocking=True)
                d2h_done[j].record(copy_stream)
        copy_stream.synchronize()

    e2e_steps(max(2, args.warmup))
    torch.cuda.synchronize()
    barrier(world)
    t0 = time.perf_counter()
    s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s2.record()
    e2e_steps(args.steps)
    torch.cuda.current_stream().wait_stream(copy_stream)
    e2.record()
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3
    barrier(world)
    e2e_ms = max_over_ranks(max(s2.elapsed_time(e2), 0.0), world, dev)
    e2e_value = world * B * args.steps / (e2e_ms * 1e-3)

    want_train = (not args.no_train_leg and family(args.config)[2] == "oracle.taskprompter_ref"
                  and not args.config.startswith("tp_cfg5"))
    line = None
    if rank == 0:
        peaks, peak_src = load_peaks()
        roof = gemm_roofline(model, plan, dev_in[0], peaks, peak_src)
        gflop_img = GFLOP_PER_IMAGE.get(args.config)
        tot_gflop = gflop_img * B if gflop_img else None
        line = {
            "metric": "images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16x3 (split-bf16 operands, fp32 accumulate)" if nsplit == 2 else "bf16",
            "data": "synthetic",
            "config": {
                "workload": f"{WORKLOAD[args.config]}, {args.config}, bs {B}/GPU, random-init weights, eval",
                "global_batch": world * B, "parallelism": f"dp{world} (batch-sharded forward, no collective)",
                "precision_mode": args.mode,
                "l2": "no explicit flush: each step streams 1.6 GB of packed weights plus ~1 GB of activations "
                      "(>> 126 MB L2) and the input rotates over 4 buffers",
            },
            "clocks": clocks,
            "repeats": {"n": len(regions), "steps_each": args.steps, "reported": "median region",
                        "images_per_s": [world * B * args.steps / (r * 1e-3) for r in regions]},
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": in_bytes,
                    "d2h_bytes_per_step": out_bytes, "ms_per_step": e2e_ms / args.steps, "wall_ms_per_step": wall_ms / args.steps,
                    "note": "pinned-host input -> H2D -> model(x) -> all task logits D2H (overlapped with the next step)"},
            "gpu_launches": int(launches_per_fwd * args.steps),
            "launches_per_step": int(launches_per_fwd),
            "roofline": roof,
        }
        if gflop_img:
            line["model_tflops_algorithmic"] = value * gflop_img / 1e3 / world
            peak = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
            line["whole_step"] = {"gflop_per_step_algorithmic": tot_gflop, "tflops_algorithmic": value * gflop_img / 1e3 / world,
                                  "frac_of_sustained_bf16_peak": value * gflop_img / 1e3 / world / peak,
                                  "note": "every FLOP of the reference forward (SURVEY.md 8d) over the whole step time"}
    del model, plan, out, stage, dev_in
    torch.cuda.empty_cache()
    if rank == 0 and world == 1 and not args.no_gpu_eager:
        ge = gpu_eager_baseline(args.config, B, dev)
        for k in ("fp32", "tf32", "bf16_autocast"):
            if k in ge:
                ge[f"ours_over_{k}"] = value / ge[k]
        line["gpu_eager_baseline"] = ge
        torch.cuda.empty_cache()
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = pick_cpu_threads()
        n_fwd = 1 if args.config in ("tp_cfg5", "tps_swinB") else 3
        rate, sec, kind = cpu_oracle_rate(args.config, n_fwd, 1, threads)
        line["cpu_baseline"] = {"value": rate, "unit": "images/s", "cores": threads, "kind": kind,
                                "sample": f"{n_fwd} forward(s) of batch 1 of {args.config} (fp32 eager, eval, "
                                          f"{threads} of {os.cpu_count()} host threads = fastest setting)"}

    # ---------------- the training step on the same ranks (`train_step`): the part of the job with a real collective.
    # The inference line above is complete before this starts and is printed whatever happens here: a watchdog prints it
    # (rank 0) and ends the process if the leg does not come back, an exception is recorded in the block.
    def emit():
        if rank == 0:
            print(json.dumps(line), file=_OUT, flush=True)

    if want_train:
        def give_up():
            if rank == 0:
                line["train_step"] = {"error": f"no result within {args.train_leg_timeout} s (watchdog)"}
                emit()
            os._exit(0)
        dog = threading.Timer(args.train_leg_timeout, give_up)
        dog.daemon = True
        dog.start()
        try:
            block = train_leg(args, rank, world, dev)
        except Exception as ex:  # noqa: BLE001 -- the inference line must survive a failure of the extra leg
            block = {"error": f"{type(ex).__name__}: {ex}"[:300]}
        dog.cancel()
        if rank == 0:
            line["train_step"] = block
    emit()
    if world > 1:                    # a process group that has been captured into CUDA graphs can block in its destructor:
        w = threading.Timer(30.0, lambda: os._exit(0))   # the line is out, so do not let the tear-down hang the job
        w.daemon = True
        w.start()
    D.teardown(world)


# ------------------------------------------------------------------------------------------------
# --train: the training step (SURVEY.md 8f N1; TaskPrompter/utils/train_utils.py:34-51). A separate line from the
# contract's inference metric: same JSON shape, metric "train images/sec".
def _train_criterion(cfg):
    from mtt_b200 import losses
    w = {"semseg": 1.0, "human_parts": 2.0, "sal": 5.0, "edge": 50.0, "normals": 10.0, "depth": 1.0}   # the ymls
    p = dict(TASKS=dict(NAMES=list(cfg["tasks"])), edge_w=0.95, ignore_index=255, ignore_invalid_area_depth=True,
             loss_kwargs=dict(loss_weights={t: w[t] for t in cfg["tasks"]}))
    return losses.get_criterion(p), w


def _train_labels(cfg, B, g):
    """Synthetic labels of the shapes the reference's datasets produce (ignore regions included)."""
    H, W = cfg["img_size"]
    lab = {}
    hole = lambda frac: torch.rand(B, 1, H, W, generator=g) < frac
    for t in cfg["tasks"]:
        if t in ("semseg", "human_parts"):
            y = torch.randint(0, cfg["num_output"][t], (B, 1, H, W), generator=g).float()
            y[hole(0.1)] = 255.0
        elif t in ("sal", "edge"):
            y = (torch.rand(B, 1, H, W, generator=g) < (0.3 if t == "sal" else 0.1)).float()
            y[hole(0.05)] = 255.0
        elif t == "normals":
            y = torch.nn.functional.normalize(torch.randn(B, 3, H, W, generator=g), dim=1)
            y = torch.where(hole(0.1).expand(-1, 3, -1, -1), torch.full_like(y, 255.0), y)
        else:
            y = torch.rand(B, 1, H, W, generator=g) * 9 + 0.5
            y[hole(0.15)] = -1.0
        lab[t] = y
    return lab


def train_eager_baseline(cfg_name, batch, dev, labels, steps=3, warmup=1):
    """The training step of the reference algorithm in eager PyTorch on the same GPU: train-mode restatement (oracle,
    pinned to the reference by tests/test_train.py) -> criterion restatement -> autograd -> clip_grad_norm_ -> Adam."""
    import contextlib

    from oracle import loss_ref
    from oracle import taskprompter_ref as TPR
    cfg, _, _ = family(cfg_name)
    sd = {k: v.to(dev) for k, v in TPR.init_state_dict(cfg, seed=0).items()}
    params = [v.requires_grad_(True) for k, v in sd.items() if v.is_floating_point() and "running_" not in k]
    opt = torch.optim.Adam(params, lr=2e-5, weight_decay=1e-6)
    x = torch.randn(batch, 3, *cfg["img_size"], device=dev)
    w = _train_criterion(cfg)[1]
    res = {"kind": "port", "batch": batch, "steps": steps, "warmup": warmup, "unit": "images/s",
           "what": "eager PyTorch training step of the reference algorithm on this GPU (cuBLAS / cuDNN + autograd + Adam)"}
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)

    def one(ctx):
        with ctx, TPR.train_mode(0.15):
            out = TPR.forward(sd, cfg, x)
        loss = loss_ref.multi_task_loss({t: o.float() for t, o in out.items()}, labels, cfg["tasks"], w)
        opt.zero_grad()
        loss["total"].backward()
        torch.nn.utils.clip_grad_norm_(params, 10.0)
        opt.step()

    def timed(ctx):
        for _ in range(warmup):
            one(ctx)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            one(ctx)
        e.record()
        torch.cuda.synchronize()
        return batch * steps / (s.elapsed_time(e) * 1e-3)

    try:
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        res["fp32"] = timed(contextlib.nullcontext())
        torch.backends.cuda.matmul.allow_tf32 = True
        torch.backends.cudnn.allow_tf32 = True
        res["tf32"] = timed(contextlib.nullcontext())
        res["bf16_autocast"] = timed(torch.autocast("cuda", dtype=torch.bfloat16))
    except Exception as ex:
        res["error"] = f"{type(ex).__name__}: {ex}"[:200]
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    return res


def train_leg(args, rank, world, dev, warmup=3, repeats=3):
    """The TRAINING step of the same workload on the same ranks, appended to the inference line as `train_step`: the
    forward shards over the batch without any exchange, so the scaling run would otherwise never exercise a collective.
    Here every step all-reduces the SyncBatchNorm statistics and the whole gradient arena over NCCL (captured with the
    step in one CUDA graph). Same step and timing rules as `bench.py --train` (barrier + synchronize around each timed
    region, max over ranks, median region); every rank takes part, rank 0 gets the numbers back."""
    from mtt_b200 import dist as D
    from mtt_b200.train import TrainStep

    steps = args.steps
    cfg, M, _ = family(args.config)
    nsplit = 2 if args.mode == "parity" else 1
    torch.manual_seed(0)
    with torch.device(dev):
        model = M.build_from_config(cfg, nsplit=nsplit, use_graph=False)
    pg = torch.distributed.group.WORLD if world > 1 else None
    ts = TrainStep(model, nsplit=nsplit, process_group=pg, use_graph=True)
    crit, _ = _train_criterion(cfg)
    B = args.batch
    g = torch.Generator().manual_seed(11 + rank)
    n_rot = 2
    host_x = [torch.randn(B, 3, *cfg["img_size"], generator=g).pin_memory() for _ in range(n_rot)]
    host_y = [{t: v.pin_memory() for t, v in _train_labels(cfg, B, g).items()} for _ in range(n_rot)]
    in_bytes = host_x[0].numel() * 4 + sum(v.numel() * 4 for v in host_y[0].values())
    last = None
    with torch.no_grad():
        for i in range(warmup):                       # the first call warms the allocator and captures the step
            ts.step(host_x[i % n_rot], host_y[i % n_rot], crit)
        torch.cuda.synchronize()
        regions = []
        for _ in range(repeats):
            D.barrier(world)
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for i in range(steps):
                loss = ts.step(host_x[i % n_rot], host_y[i % n_rot], crit)
                last = float(loss["total"])           # the step's result is read back (D2H) every step
            e.record()
            torch.cuda.synchronize()
            D.barrier(world)
            regions.append(D.max_over_ranks(s.elapsed_time(e), world, dev))
    ms_total = sorted(regions)[len(regions) // 2]
    grad_bytes = ts.grads.flat.numel() * 4
    ts._graph = None                                  # the captured step (and the NCCL work in it) goes before the group does
    del ts, model
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return {
        "metric": "train images/sec", "value": world * B * steps / (ms_total * 1e-3), "unit": "images/s",
        "ms_per_step": ms_total / steps, "steps": steps, "warmup": warmup, "global_batch": world * B,
        "repeats": [world * B * steps / (r * 1e-3) for r in regions], "last_loss": last,
        "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": 4,
        "what": ("pinned-host images + labels -> H2D -> train-mode forward (DropPath 0.15, batch-statistics BatchNorm) -> "
                 "criterion -> reverse pass -> clip_grad_norm_ 10 -> Adam -> loss scalar D2H, one CUDA-graph replay per step; "
                 "the line `python bench.py --train` prints, measured here on the ranks of this run"),
        "parallelism": (f"dp{world}: SyncBatchNorm statistics + bucketed NCCL all-reduce of the {grad_bytes / 1e6:.0f} MB fp32 "
                        "gradient arena on a communication stream behind the reverse pass") if world > 1 else "dp1 (no collective)",
        "allreduce_bytes_per_step": grad_bytes if world > 1 else 0,
    }


def run_train(args):
    import mtt_b200  # noqa: F401
    from mtt_b200 import dist as D
    from mtt_b200 import ops
    from mtt_b200.train import TrainStep

    rank, world, local = D.setup("nccl")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    cfg, M, _ = family(args.config)
    nsplit = 2 if args.mode == "parity" else 1
    torch.manual_seed(0)
    with torch.device(dev):
        model = M.build_from_config(cfg, nsplit=nsplit, use_graph=False)
    pg = torch.distributed.group.WORLD if world > 1 else None
    ts = TrainStep(model, nsplit=nsplit, process_group=pg, use_graph=not args.no_graph)
    crit, _ = _train_criterion(cfg)
    B = args.batch
    g = torch.Generator().manual_seed(1 + rank)
    n_rot = 2
    host_x = [torch.randn(B, 3, *cfg["img_size"], generator=g).pin_memory() for _ in range(n_rot)]
    host_y = [{t: v.pin_memory() for t, v in _train_labels(cfg, B, g).items()} for _ in range(n_rot)]
    in_bytes = host_x[0].numel() * 4 + sum(v.numel() * 4 for v in host_y[0].values())

    def step(i):
        if ts.use_graph:                                   # the step copies pinned host buffers straight into the graph's inputs
            x, y = host_x[i % n_rot], host_y[i % n_rot]
        else:
            x = host_x[i % n_rot].to(dev, non_blocking=True)
            y = {t: v.to(dev, non_blocking=True) for t, v in host_y[i % n_rot].items()}
        with torch.no_grad():
            return ts.step(x, y, crit)

    for i in range(args.warmup):
        loss = step(i)
    torch.cuda.synchronize()
    ops.launch_count(reset=True)
    with torch.no_grad():
        ts._fwd_bwd(host_x[0].to(dev), {t: v.to(dev) for t, v in host_y[0].items()}, crit, None)   # eager: counts the launches
    torch.cuda.synchronize()
    launches = ops.launch_count() + 2
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    regions, last = [], None
    for _ in range(max(1, args.repeats)):
        D.barrier(world)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(args.steps):
            loss = step(i)
            last = float(loss["total"])                   # the step's result is read back (D2H) every step
        e.record()
        torch.cuda.synchronize()
        D.barrier(world)
        regions.append(D.max_over_ranks(s.elapsed_time(e), world, dev))
    clocks = sampler.stop() if rank == 0 else None
    ms_total = sorted(regions)[len(regions) // 2]
    value = world * B * args.steps / (ms_total * 1e-3)
    # phases of one step (events) and the tensor-core share (library profiling hook)
    x = host_x[0].to(dev)
    y = {t: v.to(dev) for t, v in host_y[0].items()}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    with torch.no_grad():
        ts.zero_grad()
        ev[0].record()
        out = ts.forward(x)
        ev[1].record()
        leaves = {t: o.requires_grad_(True) for t, o in out.items()}
        with torch.enable_grad():
            ls = crit(leaves, y, tasks=cfg["tasks"])
            gr = torch.autograd.grad(ls["total"], [leaves[t] for t in cfg["tasks"]])
        ev[2].record()
        ts.backward(dict(zip(cfg["tasks"], gr)))
        ev[3].record()
        ts.optimizer_step()
        ev[4].record()
    torch.cuda.synchronize()
    phases = {k: ev[i].elapsed_time(ev[i + 1]) for i, k in enumerate(("forward_ms", "loss_ms", "backward_ms", "optimizer_ms"))}
    ops.profile_begin()
    with torch.no_grad():
        ts._fwd_bwd(x, y, crit, None)                      # eager pass: the profiling hook brackets every tensor-core launch
    recs = ops.profile_end(max_recs=16384)
    tc_ms = sum(r[4] for r in recs)
    tc_flops = sum(r[5] for r in recs)
    ts._graph = None                 # the captured step (and the NCCL work inside it) goes before the process group does
    torch.cuda.synchronize()
    D.barrier(world)
    if world > 1:                    # a process group that has been captured into CUDA graphs can block in its destructor:
        import threading             # the result is already measured, so do not let the tear-down hang the job
        w = threading.Timer(30.0, lambda: os._exit(0))
        w.daemon = True
        w.start()
    shapes = {}
    for kind, M_, N_, K_, ms, fl in recs:
        a = shapes.setdefault((kind, M_, N_, K_), [0, 0.0, 0.0])
        a[0] += 1
        a[1] += ms
        a[2] += fl
    top = [{"kind": "attention" if k[0] == 1 else "gemm", "M": k[1], "N": k[2], "K": k[3], "launches": v[0], "ms": v[1],
            "tflops": v[2] / (v[1] * 1e-3) / 1e12 if v[1] else None}
           for k, v in sorted(shapes.items(), key=lambda kv: -kv[1][1])[:24]]
    if rank != 0:
        D.teardown(world)
        return
    peaks, peak_src = load_peaks()
    peak = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
    line = {
        "metric": "train images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16x3 (split-bf16 operands, fp32 accumulate)" if nsplit == 2 else "bf16",
        "data": "synthetic",
        "config": {"workload": f"{WORKLOAD[args.config]}, {args.config}, TRAINING step (train-mode forward, criterion, "
                               f"backward, gradient all-reduce, clip_grad_norm_ 10, Adam), bs {B}/GPU, DropPath 0.15",
                   "global_batch": world * B,
                   "parallelism": f"dp{world}: SyncBatchNorm statistics + bucketed NCCL all-reduce of the gradient arena "
                                  "overlapped with the reverse pass" if world > 1 else "dp1",
                   "precision_mode": args.mode, "l2": "activations and weights of a step are >> 126 MB L2"},
        "clocks": clocks, "last_loss": last,
        "repeats": {"n": len(regions), "steps_each": args.steps, "reported": "median region",
                    "images_per_s": [world * B * args.steps / (r * 1e-3) for r in regions]},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": 4,
                "note": "the timed step IS end to end: pinned-host images + labels -> H2D -> TrainStep.step -> loss scalar D2H"},
        "gpu_launches": int(launches * args.steps), "launches_per_step": int(launches),
        "phases": phases, "top_tensor_shapes": top,
        "roofline": {"bound": "tensor", "achieved": tc_flops / (tc_ms * 1e-3) / 1e12 if tc_ms else None, "peak": peak,
                     "unit": "TFLOP/s", "frac": (tc_flops / (tc_ms * 1e-3) / 1e12 / peak) if tc_ms else None, "traffic": None,
                     "peak_source": peak_src, "kernel": "mtt_gemm / mtt_gemm_grouped / mtt_attention launches of one step",
                     "launches": len(recs), "tensor_ms_per_step": tc_ms, "algorithmic_gflop_per_step": tc_flops / 1e9,
                     "share_of_step": tc_ms / (ms_total / args.steps)},
    }
    if world == 1 and not args.no_gpu_eager:
        del ts, model
        torch.cuda.empty_cache()
        ge = train_eager_baseline(args.config, B, dev, y)
        for k in ("fp32", "tf32", "bf16_autocast"):
            if k in ge:
                ge[f"ours_over_{k}"] = value / ge[k]
        line["gpu_eager_baseline"] = ge
    print(json.dumps(line), file=_OUT, flush=True)
    D.teardown(world)


def run_reference_train(args):
    """--impl reference --train: the reference's training step on the host cores (rank 0 only): the unmodified reference
    model + criterion where importable, else the train-mode restatement; autograd, clip_grad_norm_, Adam."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import loss_ref, ref_loader
    from oracle import taskprompter_ref as TPR
    threads = pick_cpu_threads()
    torch.set_num_threads(threads)
    cfg, _, _ = family(args.config)
    B = args.batch
    g = torch.Generator().manual_seed(1)
    x = torch.randn(B, 3, *cfg["img_size"], generator=g)
    y = _train_labels(cfg, B, g)
    w = {"semseg": 1.0, "human_parts": 2.0, "sal": 5.0, "edge": 50.0, "normals": 10.0, "depth": 1.0}
    sd = TPR.init_state_dict(cfg, seed=0)
    if ref_loader.available():
        kind = "reference"
        model = ref_loader.build_taskprompter(cfg).train()
        model.load_state_dict(sd, strict=True)
        params = list(model.parameters())
        fwd = lambda: model(x)
    else:
        kind = "port"
        params = [v.requires_grad_(True) for k, v in sd.items() if v.is_floating_point() and "running_" not in k]

        def fwd():
            with TPR.train_mode(0.15):
                return TPR.forward(sd, cfg, x)
    opt = torch.optim.Adam(params, lr=2e-5, weight_decay=1e-6)

    def one():
        loss = loss_ref.multi_task_loss(fwd(), y, cfg["tasks"], w)
        opt.zero_grad()
        loss["total"].backward()
        torch.nn.utils.clip_grad_norm_(params, 10.0)
        opt.step()
    for _ in range(args.warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one()
    sec = (time.perf_counter() - t0) / max(args.steps, 1)
    rate = B / sec
    sample = (f"training step on batch {B} of {args.config} (fp32 eager CPU, "
              f"{'the unmodified reference model' if kind == 'reference' else 'train-mode restatement (oracle/)'}, criterion "
              f"restatement, autograd, clip, Adam), {args.warmup} warm-up + {args.steps} timed steps, {threads} host threads")
    line = {"impl": "reference", "metric": "train images/sec", "value": rate, "unit": "images/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{WORKLOAD[args.config]}, {args.config}, TRAINING step, bs {B}", "global_batch": B,
                       "parallelism": "one CPU process (rank 0)", "precision_mode": "fp32 eager CPU"},
            "cpu_baseline": {"value": rate, "unit": "images/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": rate, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), file=_OUT, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps per timed region")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="parity", choices=["parity", "speed"])
    ap.add_argument("--config", default="tp_cfg4")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (default: the config's)")
    ap.add_argument("--repeats", type=int, default=5, help="timed regions of --steps steps; the median is reported")
    ap.add_argument("--no-graph", action="store_true", help="--train: launch the step eagerly instead of replaying its CUDA graph")
    ap.add_argument("--train", action="store_true", help="time the TRAINING step (TaskPrompter ViT configs) instead of the forward")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true")
    ap.add_argument("--no-train-leg", action="store_true",
                    help="skip the `train_step` block (the training step timed on the same ranks after the forward)")
    ap.add_argument("--train-leg-timeout", type=float, default=150.0,
                    help="seconds after which the watchdog prints the finished inference line without the train_step block")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="forward benchmark: write the outputs of the last timed step as DIR/<name>.npy (float32, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.train or args.impl != "ours"):
        ap.error("--dump-outputs covers the forward benchmark (--impl ours without --train)")
    if args.config not in WORKLOAD:       # any named configuration of mtt_b200/configs.py (tiny ones: contract tests)
        try:
            family(args.config)
        except KeyError:
            ap.error(f"--config: unknown configuration {args.config!r}")
        WORKLOAD[args.config] = f"{args.config} (test configuration)"
    if args.batch <= 0:
        args.batch = DEFAULT_BATCH.get(args.config, 2)
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    # stdout carries exactly ONE JSON line: whatever a library prints to file descriptor 1 (NCCL's "NCCL version ..."
    # banner at init, for one) is sent to stderr; the JSON line goes to the saved descriptor.
    global _OUT
    sys.stdout.flush()
    _OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.train and family(args.config)[2] != "oracle.taskprompter_ref":
        ap.error("--train covers the ViT TaskPrompter configurations (tp_*)")
    if args.impl == "reference":
        (run_reference_train if args.train else run_reference)(args)
    elif args.train:
        run_train(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
