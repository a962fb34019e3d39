#!/usr/bin/env python
"""Benchmark of the camera->BEV lift (BASELINE.json metric: lift frames/sec, 6-cam 224x480 -> 200x200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg3_baseline] [--dump-outputs DIR]

One "step" = one pass of the hot path {head tensor, intrinsics, extrinsics} -> BEV (B', C, X, Y) over one batch of
synthetic frames (SURVEY.md section 8d).  Prints ONE JSON line (rank 0).

  value      whole-job frames/s, inputs resident in HBM, through the public Python API (LiftSplat.capture -> C ABI): one step =
             tile kernels (geometry evaluated inside) + layout passes of the whole batch (nothing is cached between steps)
  e2e        same metric with HOST (pinned) inputs and a host copy of the BEV inside the timed region
  roofline   the PATH against the measured HBM copy bandwidth (MEASURED_PEAKS.json): algorithmic bytes of the step / step time;
             `kernels` lists every kernel of the step with its OWN algorithmic bytes, the duration of the launches the step really
             runs (event pairs on their streams, fiery_lift_forward_timed) and the ncu DRAM bytes of the committed capture
  roofline_bwd  the same for the backward (grad of the head tensor)
  cpu_baseline  the oracle's torch-CPU restatement of the reference op chain on this box's host cores, bounded sample

`--impl reference` times that CPU restatement itself (the reference is pure PyTorch; /root/reference is not on the GPU
box, oracle/lift_oracle.py restates it op for op and is pinned to it by oracle/gen_golden.py).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

from fiery_b200.synthetic import CONFIGS, LiftConfig, make_calibration, make_grad_bev, make_head  # noqa: F401

METRIC = "camera->BEV lift frames/sec (6-cam 224x480 -> 200x200)"
L2_FLUSH_BYTES = 256 << 20
DUMP_BYTES = 60 << 20           # --dump-outputs: array data of all files together; with the .npy headers it stays under 64 MB


def dump_outputs(out_dir: str, arrays: dict):
    """Writes each array as ``out_dir/<name>.npy`` in float32 (float64 stays float64), flattened in logical (C) order when sampled.
    An array larger than its equal share of DUMP_BYTES is replaced by a sample of its elements at indices drawn from a fixed seed,
    so two runs with the same arguments store the same elements and two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        a = np.ascontiguousarray(a if a.dtype in (np.float32, np.float64) else a.astype(np.float32))
        if a.nbytes > share:
            pick = np.sort(np.random.default_rng(0).choice(a.size, size=share // a.itemsize, replace=False))
            a = a.reshape(-1)[pick]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def load_traffic(workload: str):
    """ncu DRAM bytes (read + write) per step of every kernel of this workload, from the committed captures
    (profiles/traffic.json: {workload: {kernel: bytes per step}}); {} when there is no capture."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(path) as fh:
            v = json.load(fh).get(workload)
        return {k: int(b) for k, b in v.items()} if isinstance(v, dict) else {}
    except (OSError, ValueError):
        return {}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clocks and throttle reasons with nvidia-smi while the timed region runs."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_lift_once(oracle, head, K, E, gout=None):
    if gout is None:
        with torch.no_grad():
            return oracle.lift(head, K, E)
    h = head.clone().requires_grad_(True)                     # forward + autograd backward to the head tensor
    oracle.lift(h, K, E).backward(gout)
    return h.grad


def _best_thread_count(oracle, head, K, E, candidates):
    """The reference's op chain is many small ATen ops; on a many-core host the default (all cores) can be far slower
    than a moderate thread count.  One quick rep per candidate, keep the fastest -- the baseline gets its best setting."""
    best, best_t = None, float("inf")
    for t in candidates:
        torch.set_num_threads(t)
        with torch.no_grad():
            oracle.lift(head, K, E)
            t0 = time.perf_counter()
            oracle.lift(head, K, E)
            dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = t, dt
    return best


def time_cpu_reference(cfg: LiftConfig, frames: int, reps: int, warmup: int = 1, backward: bool = False):
    """Times the oracle's torch-CPU restatement of the reference op chain (fiery.py:193-273, encoder.py:99-100,
    geometry.py:283-314) on the host cores, at the thread count that is fastest on this box.
    Returns (frames_per_s, seconds_per_call, threads, output of the last timed call)."""
    from oracle import lift_oracle as O
    cores = os.cpu_count() or 1
    sub = LiftConfig(**{**cfg.__dict__, "frames": frames})
    K, E = make_calibration(sub, seed=0)
    K, E = torch.from_numpy(K), torch.from_numpy(E)
    head = torch.from_numpy(make_head(sub, seed=0))
    oracle = O.LiftOracle.from_config(sub)
    one = LiftConfig(**{**cfg.__dict__, "frames": 1})
    K1, E1 = make_calibration(one, seed=0)
    cands = sorted({t for t in (4, 8, 16, 32, 64, cores) if t <= cores})
    threads = _best_thread_count(O.LiftOracle.from_config(one), torch.from_numpy(make_head(one, seed=0)),
                                 torch.from_numpy(K1), torch.from_numpy(E1), cands)
    torch.set_num_threads(threads)
    gout = torch.from_numpy(make_grad_bev(sub, seed=0)) if backward else None
    for _ in range(warmup):
        cpu_lift_once(oracle, head, K, E, gout)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = cpu_lift_once(oracle, head, K, E, gout)
        ts.append(time.perf_counter() - t0)
    sec = float(np.median(ts))
    return frames / sec, sec, threads, out


def config_dict(cfg: LiftConfig, args, world: int):
    """`config` of the JSON line: identical for both arms (the reference arm runs the same frames per step)."""
    X, Y = cfg.bev_hw
    return {"workload": cfg.name, "frames_per_step_per_gpu": cfg.frames, "n_cameras": cfg.n_cameras,
            "final_dim": list(cfg.final_dim), "feat_hw": list(cfg.feat_hw), "depth_bins": cfg.depth_bins,
            "channels": cfg.out_channels, "bev": [X, Y], "direction": args.direction, "output_layout": args.layout,
            "head_dtype": args.head_dtype}


def run_reference(args, cfg: LiftConfig, rank: int):
    if rank != 0:
        return
    frames = cfg.frames                       # the same batch the GPU arm lifts per step
    steps = args.steps
    backward = args.direction == "fwd_bwd"
    fps, sec, threads, out = time_cpu_reference(cfg, frames, reps=steps, warmup=max(1, min(args.warmup, 2)), backward=backward)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"grad_head" if backward else "bev": out})
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(cfg, args, 1),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                         "sample": f"{steps} reps of {frames} frame(s) of {cfg.name}, torch-CPU op chain of the reference "
                                   f"(oracle/lift_oracle.py), best of thread counts up to {os.cpu_count()}: {threads} threads"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# (batch, sequence) of the reference configs the workloads stand for: frames per step = batch x time receptive field
BATCH_SEQ = {"cfg1_tiny": (1, 1), "cfg2_static_lss": (1, 1), "cfg2_static_lss_b8": (8, 1), "cfg3_baseline": (3, 3), "cfg4_pon": (4, 3),
             "cfg6_res_0p4_0p3": (2, 1)}


def run_train(args, cfg: LiftConfig, rank: int, local_rank: int, world: int):
    """--direction fwd_bwd: one data-parallel training step per timed step (fiery_b200.train.LiftTrainer), weak scaling: every rank
    trains on its own (batch x seq) samples of the global batch, ONE NCCL all-reduce of the flat gradient per step."""
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device: fiery_b200 has no CPU path")
    import torch.distributed as dist
    from fiery_b200 import _lib, hostmem
    from fiery_b200.train import LiftTrainer, synthetic_batch
    _lib.load()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = hostmem.bind_to_gpu_numa(local_rank, local_rank, 1)
    distributed = world > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    b, s = BATCH_SEQ[cfg.name]
    frames = b * s
    precision = 16 if args.head_dtype == "f16" else 32
    trainer = LiftTrainer(cfg, dev, precision=precision, feature_input=True, seed=0)
    batch = synthetic_batch(cfg, b, s, dev, seed=1000, feature_input=True, first_sample=rank * b)
    host = {k: v.cpu().pin_memory() for k, v in batch.items()}
    flush = torch.empty(L2_FLUSH_BYTES // 4, dtype=torch.float32, device=dev)
    W, S = max(args.warmup, 3), args.steps

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn):
        pairs = []
        for _ in range(S):
            flush.fill_(1.0)
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); e.record()
            pairs.append((a, e))
        torch.cuda.synchronize()
        return float(np.mean([a.elapsed_time(e) for a, e in pairs]))

    last = {}

    def step_dev():
        last["loss"] = trainer.step(batch)

    def step_e2e():                                   # the step's inputs come from pinned host memory, its loss goes back to the host
        dev_batch = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        return float(trainer.step(dev_batch))

    sampler = ClockSampler(local_rank)
    if rank == 0:                                     # before the warm-up: see main()
        sampler.start()
        time.sleep(1.0)
    barrier()
    for _ in range(W):
        step_dev()
    barrier()
    ms_dev = timed(step_dev)
    if args.dump_outputs and rank == 0:               # the last timed step's loss and the weights its optimizer step left
        dump_outputs(args.dump_outputs, {"loss": last["loss"],
                                         "params": torch.cat([p.detach().flatten() for p in trainer.bucket.params])})
    barrier()
    for _ in range(2):
        step_e2e()
    barrier()
    ms_e2e = timed(step_e2e)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    # the lift's share of the step: forward + backward through the autograd function alone, same tensors
    head = trainer.model.encoder.depth_layer(batch["image"].reshape(frames * cfg.n_cameras, *batch["image"].shape[3:])).detach()
    K_p, E_p = batch["intrinsics"].reshape(frames, cfg.n_cameras, 3, 3), batch["extrinsics"].reshape(frames, cfg.n_cameras, 4, 4)
    X, Y = cfg.bev_hw
    g_cl = torch.randn(frames, X, Y, cfg.out_channels, device=dev).permute(0, 3, 1, 2)
    hg = head.clone().requires_grad_(True)

    def lift_only():
        hg.grad = None
        trainer.model.lift(hg, K_p, E_p).backward(g_cl)
    for _ in range(3):
        lift_only()
    ms_lift = timed(lift_only)

    def reduce_max(x):
        if not distributed:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    ms_dev, ms_e2e, ms_lift = reduce_max(ms_dev), reduce_max(ms_e2e), reduce_max(ms_lift)
    if rank == 0:
        peak, peak_src = load_peaks()
        total = frames * world
        alg = (cfg.fwd_bytes_per_frame(4) + cfg.bwd_bytes_per_frame(4)) * frames
        h2d = int(sum(v.numel() * v.element_size() for v in host.values()))
        line = {
            "metric": METRIC, "value": total / (ms_dev * 1e-3), "unit": "frames/s", "n_gpus": world, "steps": S, "warmup": W,
            "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": config_dict(cfg, args, world),          # identical in both arms
            "details": {"batch_per_gpu": b, "time_receptive_field": s,
                       "precision": precision, "step": "depth_layer (tcgen05 GEMM: half features -> fp32 head; backward: cuDNN) -> fused lift forward (channels-last BEV) -> BEV head "
                       "+ uncertainty-weighted losses -> fused lift backward (shared geometry plan) -> ONE all-reduce of the flat fp32 "
                       "gradient -> clip 5 -> Adam(3e-4, wd 1e-7); image backbone excluded (feature maps are the input)",
                       "parallelism": f"dp{world}: batch sharded over {world} GPU(s), single NCCL all-reduce of {trainer.bucket.nbytes} gradient bytes per step",
                       "l2": "flushed before every timed step (256 MiB write)",
                       "host": {"numa_node": numa[0], "cores_bound": numa[1], "note": numa[2]},
                       "timing": "CUDA events around the step, mean over steps, max over ranks"},
            "e2e": {"value": total / (ms_e2e * 1e-3), "unit": "frames/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": 4},
            "gpu_launches": 3 * S,          # per step: lift_plan_kernel, lift_forward_cols_kernel, lift_backward_kernel
            "lift_fwd_bwd": {"ms_per_step": ms_lift, "frames_per_s": total / (ms_lift * 1e-3),
                             "what": "plan + lift forward + lift backward alone (autograd function, channels-last BEV and gradient)"},
            "roofline": {"bound": "hbm", "kernel": "lift_plan_kernel + lift_forward_cols_kernel + lift_backward_kernel",
                         "achieved": alg / (ms_lift * 1e-3) / 1e9, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                         "frac": alg / (ms_lift * 1e-3) / 1e9 / peak, "traffic": None, "algorithmic_bytes_per_step": alg,
                         "how": "algorithmic bytes of lift forward + backward (SURVEY.md 8d) / time of the lift's autograd forward+backward"},
            "clocks": clocks,
        }
        if not args.no_cpu_baseline:
            fps, sec, threads, _ = time_cpu_reference(cfg, min(frames, args.cpu_frames), reps=max(2, args.cpu_reps // 2), backward=True)
            line["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                                    "sample": f"forward+backward of the lift (oracle/lift_oracle.py through torch autograd) on "
                                              f"{min(frames, args.cpu_frames)} frame(s) of {cfg.name}, {threads} threads"}
        print(json.dumps(line), flush=True)
    if distributed:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    # default = BASELINE.json configs[1] (literature/static_lss_setting.yml, 6-cam 224x480 -> 200x200) at its own BATCHSIZE 8
    # (single_timeframe.yml:8), the configuration the metric is quoted on; cfg3_baseline (9 frames) etc. via --workload
    ap.add_argument("--workload", default="cfg2_static_lss_b8", choices=sorted(CONFIGS))
    ap.add_argument("--layout", default="contiguous", choices=["contiguous", "channels_last"])
    ap.add_argument("--direction", default="forward", choices=["forward", "fwd_bwd"],
                    help="forward: the lift (the metric's definition).  fwd_bwd: the data-parallel TRAINING step around it "
                         "(fiery_b200.train: depth_layer -> lift forward -> BEV head + losses -> lift backward -> ONE gradient "
                         "all-reduce -> clip -> Adam), BASELINE.json configs[4] with --workload cfg3_baseline --head-dtype f16 --gpus 8")
    ap.add_argument("--head-dtype", default="f32", choices=["f32", "f16"],
                    help="dtype of the head tensor: f32 (the metric's definition) or f16 (AMP heads, baseline.yml PRECISION 16: the "
                         "forward tile kernel reads the half-precision tensor itself; all arithmetic stays fp32)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the VoxelsSumming / warp / reference-ops-on-GPU side measurements")
    ap.add_argument("--e2e-chunk", default="1,2", help="frames per upload/lift/download pipeline stage in the e2e run: one number, or the "
                                                      "sizes of the first stages (the last repeats)")
    ap.add_argument("--cpu-frames", type=int, default=3)
    ap.add_argument("--cpu-reps", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path returned in its last step as DIR/<name>.npy (rank 0; "
                         "float32, at most 64 MB in all: a larger output is replaced by a fixed seeded sample of its elements). "
                         "forward: bev; fwd_bwd: loss and the updated params; --impl reference: bev, or grad_head with fwd_bwd")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = CONFIGS[args.workload]

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, cfg, rank)
        return
    if args.direction == "fwd_bwd":
        run_train(args, cfg, rank, local_rank, world)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device: fiery_b200 has no CPU path")
    import ctypes
    import torch.distributed as dist
    from fiery_b200 import _lib, hostmem
    from fiery_b200.geometry import _stream_ptr
    from fiery_b200.lift import LiftSplat
    lib = _lib.load()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # one process per GPU, bound to the cores of its GPU's NUMA node before any pinned buffer exists (e2e: 118 MB cross PCIe per step)
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    n_gpu_node = max(1, sum(1 for i in range(torch.cuda.device_count()) if hostmem.gpu_numa_node(i) == hostmem.gpu_numa_node(local_rank)))
    numa = hostmem.bind_to_gpu_numa(local_rank, local_rank, min(local_world, n_gpu_node))
    distributed = world > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    # ---- per-rank shard: weak scaling, every rank lifts its own B' frames (SURVEY.md section 8e) ------------------------
    frames = cfg.frames
    K, E = make_calibration(cfg, seed=100 + rank)
    head_np = make_head(cfg, seed=100 + rank)
    lift = LiftSplat.from_config(cfg, output_layout=args.layout).to(dev)
    K_d, E_d = torch.from_numpy(K).to(dev), torch.from_numpy(E).to(dev)
    head_d = torch.from_numpy(head_np).to(dev)
    head_dtype = torch.float16 if args.head_dtype == "f16" else torch.float32
    if head_dtype != torch.float32:
        head_d = head_d.to(head_dtype)
    flush = torch.empty(L2_FLUSH_BYTES // 4, dtype=torch.float32, device=dev)
    W, S = max(args.warmup, 3), args.steps
    X, Y = cfg.bev_hw

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_steps(step_fn, n_steps, do_flush=True):
        """Per-step CUDA events on the current stream; L2 flushed (256 MiB write) before each step, outside the events.  All steps
        are enqueued before the host waits, so a step's interval is device time: a descheduled host thread between the start event
        and the launch would otherwise show up as a multi-millisecond "step" (seen at N = 8, profiles/r02_notes.md)."""
        pairs = []
        for _ in range(n_steps):
            if do_flush:
                flush.fill_(1.0)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step_fn()
            b.record()
            pairs.append((a, b))
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in pairs]

    # ---- value: device-resident inputs through the public API ----------------------------------------------------------
    # LiftSplat.capture() records the forward lift (TMA descriptors + the tile-kernel / layout-pass chains of every frame group, forked
    # over internal streams) into a CUDA graph once; a step is one replay and recomputes EVERYTHING of the path, the geometry included
    # (the tile kernels evaluate it).  value_static_rig: the same with the geometry plan cached (capture(static_calibration=True), the
    # inference case of a fixed camera rig) -- reported next to the value, never as the value.
    def step_eager():
        with torch.no_grad():
            return lift(head_d, K_d, E_d)

    graphed = lift.capture(head_d, K_d, E_d)
    graphed_static = lift.capture(head_d, K_d, E_d, static_calibration=True)

    # the clock sampler (an nvidia-smi process) starts BEFORE the warm-up: its NVML start-up touches every GPU of the box and showed
    # up as multi-millisecond outliers in the first timed steps of every rank at N = 8 (profiles/r02_notes.md)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(1.0)
    barrier()
    for _ in range(W):
        graphed()
        graphed_static()
        step_eager()
    barrier()
    t_dev = timed_steps(graphed, S)
    if args.dump_outputs and rank == 0:               # the BEV of the last timed replay, before anything replays the graph again
        dump_outputs(args.dump_outputs, {"bev": graphed.output})
    barrier()
    t_dev_noflush = timed_steps(graphed, S, do_flush=False)
    t_static = timed_steps(graphed_static, S)
    t_eager = timed_steps(step_eager, S)
    barrier()

    # ---- forward + backward through autograd (the training-step view of the same path) -----------------------------------
    gout_d = torch.from_numpy(make_grad_bev(cfg, seed=100 + rank)).to(dev)
    gout_cl = gout_d.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)        # the same gradient, channels-last strides
    head_g = head_d.clone().requires_grad_(True)

    def step_fwd_bwd(g=gout_d):
        head_g.grad = None
        lift(head_g, K_d, E_d).backward(g)

    plan_d = lift.plan(K_d, E_d)
    head_f32 = head_d.float()

    def step_bwd_only(g):
        return lift._launch_backward(head_f32, K_d, E_d, g, plan=plan_d)

    # the lift's training path as device time: plan -> forward (planned) -> backward, through the C ABI with static buffers, captured in
    # a CUDA graph (the eager autograd step above is host-bound: ~30 launches and 4 large allocations from Python per step)
    c0 = lift._constants(dev)
    d_tr = lift._desc(c0, frames, cfg.n_cameras, torch.float32, _lib.CALIB_RAW, _lib.BEV_NCHW)
    tr_plan = torch.empty(int(lib.fiery_lift_plan_bytes(d_tr)), dtype=torch.uint8, device=dev)
    tr_scratch = torch.zeros(max(1, int(lib.fiery_lift_scratch_bytes(d_tr)) // 4), dtype=torch.float32, device=dev)
    tr_ws = torch.empty(max(1, int(lib.fiery_lift_workspace_bytes(d_tr)) // 4), dtype=torch.float32, device=dev)
    tr_out = torch.empty((frames, cfg.out_channels, X, Y), dtype=torch.float32, device=dev)
    tr_grad = torch.empty_like(head_f32)

    def train_path(sp):
        args6 = (K_d.data_ptr(), E_d.data_ptr(), c0["u"].data_ptr(), c0["v"].data_ptr(), c0["d"].data_ptr())
        _lib.check(lib.fiery_lift_plan(d_tr, *args6, tr_plan.data_ptr(), sp), "plan")
        _lib.check(lib.fiery_lift_forward(d_tr, head_f32.data_ptr(), *args6, tr_out.data_ptr(), tr_scratch.data_ptr(), tr_plan.data_ptr(), sp), "fwd")
        _lib.check(lib.fiery_lift_backward(d_tr, head_f32.data_ptr(), *args6, gout_d.data_ptr(), tr_grad.data_ptr(), tr_ws.data_ptr(),
                                           tr_plan.data_ptr(), sp), "bwd")
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for _ in range(2):
            train_path(side.cuda_stream)
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    g_train = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g_train):
        train_path(torch.cuda.current_stream(dev).cuda_stream)

    for _ in range(3):
        step_fwd_bwd()
        step_bwd_only(gout_d)
        step_bwd_only(gout_cl)
        g_train.replay()
    barrier()
    t_fb_graph = timed_steps(g_train.replay, S)
    t_fb = timed_steps(step_fwd_bwd, S)
    t_bwd = timed_steps(lambda: step_bwd_only(gout_d), S)
    t_bwd_cl = timed_steps(lambda: step_bwd_only(gout_cl), S)
    barrier()

    # ---- e2e: pinned host inputs, host copy of the result, all inside the timed region ---------------------------------
    head_h = torch.from_numpy(head_np).to(head_dtype).pin_memory()
    K_h, E_h = torch.from_numpy(K).pin_memory(), torch.from_numpy(E).pin_memory()
    out_h = torch.empty((frames, cfg.out_channels, X, Y), dtype=torch.float32).pin_memory()

    e2e_chunks = [int(x) for x in str(args.e2e_chunk).split(",")]

    def step_e2e():
        # public host-buffer entry point: chunked upload / lift / download on three streams; returns after the BEV is on the host
        lift.lift_from_host(head_h, K_h, E_h, out=out_h, device=dev, chunk_frames=e2e_chunks)

    for _ in range(3):
        step_e2e()
    barrier()
    t_e2e = timed_steps(step_e2e, S)
    barrier()
    clocks = sampler.stop() if rank == 0 else None

    # ---- per-kernel durations of the launches the step really runs (event pairs on the chains' own streams) ----------------------
    c = lift._constants(dev)
    stream = _stream_ptr(dev)
    layout_code = _lib.BEV_NHWC if args.layout == "channels_last" else _lib.BEV_NCHW
    desc = lift._desc(c, frames, cfg.n_cameras, head_dtype, _lib.CALIB_RAW, layout_code)
    launches_per_step = int(lib.fiery_lift_forward_launches(desc))
    scratch = torch.zeros(max(1, int(lib.fiery_lift_scratch_bytes(desc)) // 4), dtype=torch.float32, device=dev)
    out_buf = (torch.zeros((frames, X, Y, cfg.out_channels), dtype=torch.float32, device=dev) if layout_code == _lib.BEV_NHWC
               else torch.empty((frames, cfg.out_channels, X, Y), dtype=torch.float32, device=dev))
    KIND = {1: "lift_forward_cols_kernel", 2: "finalize_tma_kernel"}
    per_kind = {k: [] for k in KIND}
    cap = 64
    ms_arr, kind_arr, n_arr = (ctypes.c_float * cap)(), (ctypes.c_int32 * cap)(), ctypes.c_int32(0)
    for it in range(3 + S):
        flush.fill_(1.0)
        _lib.check(lib.fiery_lift_forward_timed(desc, head_d.data_ptr(), K_d.data_ptr(), E_d.data_ptr(), c["u"].data_ptr(),
                                                c["v"].data_ptr(), c["d"].data_ptr(), out_buf.data_ptr(), scratch.data_ptr(), None,
                                                stream, cap, ms_arr, kind_arr, ctypes.byref(n_arr)), "fiery_lift_forward_timed")
        if it >= 3:
            for i in range(n_arr.value):
                per_kind[int(kind_arr[i])].append(float(ms_arr[i]))
    barrier()

    # ---- the literal drop-in at fiery.py:261: VoxelsSumming on one frame's rank-sorted point features ------------------------
    vs_extra = None
    if rank == 0 and not args.no_cpu_baseline and not args.no_extras:
        try:
            from fiery_b200.geometry import VoxelsSumming
            with torch.no_grad():
                idx1, valid1, pillar1 = lift.point_indices(K_d[:1], E_d[:1])
                keep1 = valid1[0]
                ranks1 = pillar1[0][keep1].long()
                order1 = ranks1.argsort()
                ranks1 = ranks1[order1]
                geo1 = idx1[0][keep1][order1]
                feats1 = torch.randn(ranks1.numel(), cfg.out_channels, device=dev)
                for _ in range(2):
                    VoxelsSumming.apply(feats1, geo1, ranks1)
                t_vs = timed_steps(lambda: VoxelsSumming.apply(feats1, geo1, ranks1), 10)
                t_cs = timed_steps(lambda: feats1.cumsum(0), 3)
            vs_extra = {"rows": int(ranks1.numel()), "ms": float(np.mean(t_vs)), "torch_cumsum_ms": float(np.mean(t_cs)),
                        "what": "fiery_b200.geometry.VoxelsSumming.apply (plan + segmented sum, incl. its host sync) on one frame's "
                                "sorted (Nm, 64) features vs the torch.cumsum(0) alone that the reference's VoxelsSumming starts with"}
        except Exception as exc:               # an extra must never take the bench line down
            vs_extra = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    # ---- next row of the path (SURVEY.md section 8f): cumulative_warp_features on the lifted BEV (b=3 samples x s=3 steps) ---------
    warp_extra = None
    if rank == 0 and not args.no_extras:
        try:
            from fiery_b200.warp import cumulative_warp_features, _device_theta
            from fiery_b200.synthetic import make_egomotion
            wb, ws = 3, 3
            xw = torch.randn(wb, ws, cfg.out_channels, X, Y, device=dev)
            fl = torch.from_numpy(make_egomotion(wb, ws, seed=7)).to(dev)
            ext = (float(cfg.x_bound[1]), float(cfg.y_bound[1]))
            with torch.no_grad():
                for _ in range(3):
                    cumulative_warp_features(xw, fl, mode="bilinear", spatial_extent=ext)
                t_w = timed_steps(lambda: cumulative_warp_features(xw, fl, mode="bilinear", spatial_extent=ext), S)
            w_bytes = 2 * xw.numel() * 4                                    # read every frame once + write every frame once
            w_ms = float(np.mean(t_w))
            th_w, mask_w = _device_theta(fl, ext, cumulative=True)
            out_w = torch.empty_like(xw)
            chw = cfg.out_channels * X * Y

            def warp_kernel_only():
                _lib.check(lib.fiery_warp_features_forward(wb * ws, cfg.out_channels, X, Y, xw.data_ptr(), chw, th_w.data_ptr(),
                                                           mask_w.data_ptr(), out_w.data_ptr(), chw, 0, stream), "warp")
            for _ in range(3):
                warp_kernel_only()
            wk_ms = float(np.mean(timed_steps(warp_kernel_only, S)))
            gx_w = torch.empty_like(xw)

            def warp_backward_only():                                       # gather adjoint (+ the scatter launch that exits at once)
                _lib.check(lib.fiery_warp_features_backward(wb * ws, cfg.out_channels, X, Y, out_w.data_ptr(), chw, th_w.data_ptr(),
                                                            mask_w.data_ptr(), gx_w.data_ptr(), chw, 0, stream), "warp backward")
            for _ in range(3):
                warp_backward_only()
            wkb_ms = float(np.mean(timed_steps(warp_backward_only, S)))
            warp_extra = {"frames": wb * ws, "ms_per_call": w_ms, "frames_per_s": wb * ws / (w_ms * 1e-3),
                          "algorithmic_bytes": w_bytes, "kernel_ms": wk_ms, "achieved_gbs": w_bytes / (wk_ms * 1e-3) / 1e9,
                          "backward_ms": wkb_ms, "backward_achieved_gbs": w_bytes / (wkb_ms * 1e-3) / 1e9,
                          "what": "fiery_b200.warp.cumulative_warp_features, (3, 3, 64, X, Y) fp32: ms_per_call = the eager "
                                  "public call (pose-algebra kernel + sampling kernel + output allocation), kernel_ms / "
                                  "achieved_gbs = warp_forward_kernel alone via fiery_warp_features_forward; L2 flushed "
                                  "before every timed call"}
            if not args.no_cpu_baseline:
                from oracle import warp_oracle as WO
                with torch.no_grad():
                    for _ in range(2):
                        WO.cumulative_warp_features(xw.clone(), fl, mode="bilinear", spatial_extent=ext)
                    t_wr = timed_steps(lambda: WO.cumulative_warp_features(xw.clone(), fl, mode="bilinear", spatial_extent=ext), 5)
                warp_extra["reference_ops_on_gpu_ms"] = float(np.mean(t_wr))
            del out_w, gx_w
            # lift + warp as one chain (fiery_lift_forward_warped) against the two public calls, on this run's own frames
            seq = 3 if frames % 3 == 0 else (2 if frames % 2 == 0 else 0)
            if seq and args.layout != "channels_last":
                fb_ = frames // seq
                fl2 = torch.from_numpy(make_egomotion(fb_, seq, seed=11)).to(dev)
                head32 = head_d.float()
                with torch.no_grad():
                    def unfused():
                        return cumulative_warp_features(lift._launch_forward(head32, K_d, E_d).unflatten(0, (fb_, seq)), fl2,
                                                        mode="bilinear", spatial_extent=ext)

                    def fused():
                        return lift.forward_warped(head32, K_d, E_d, fl2, ext)
                    for _ in range(3):
                        unfused(); fused()
                    u_ms = float(np.mean(timed_steps(unfused, S)))
                    f_ms = float(np.mean(timed_steps(fused, S)))
                    # the same two call sequences captured in CUDA graphs: device time without the host's launch gaps
                    torch.cuda.synchronize()
                    g_u, g_f = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g_u):
                        keep_u = unfused()
                    with torch.cuda.graph(g_f):
                        keep_f = fused()
                    for _ in range(3):
                        g_u.replay(); g_f.replay()
                    ug_ms = float(np.mean(timed_steps(g_u.replay, S)))
                    fg_ms = float(np.mean(timed_steps(g_f.replay, S)))
                    del keep_u, keep_f, g_u, g_f
                warp_extra["lift_plus_warp"] = {"frames": frames, "sequence": seq, "unfused_ms": ug_ms, "fused_ms": fg_ms,
                                                "unfused_eager_ms": u_ms, "fused_eager_ms": f_ms,
                                                "what": "this run's head tensor: lift (NCHW) + cumulative_warp_features (pose kernel + "
                                                        "sampling kernel: two passes over the BEV) vs LiftSplat.forward_warped (the warp is "
                                                        "the lift's layout pass); graph replay of the public calls, and the eager calls "
                                                        "(host-paced); L2 flushed before every call"}
                del head32
        except Exception as exc:               # an extra must never take the bench line down
            warp_extra = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    # ---- next row (SURVEY.md section 8f, next-2): Decoder.first_conv 7x7 s2 64->64 on tcgen05, fed by the channel-last lift output ------
    conv_extra = None
    if rank == 0 and not args.no_extras:
        try:
            from fiery_b200.bev_conv import first_conv_forward, pack_weight
            xb = torch.randn(frames, X, Y, cfg.out_channels, device=dev).permute(0, 3, 1, 2)       # channels-last, like LiftSplat(channels_last)
            wc = torch.randn(64, 64, 7, 7, device=dev) * 0.02
            wp = pack_weight(wc)
            with torch.no_grad():
                for _ in range(3):
                    first_conv_forward(xb, wp)
                c_ms = float(np.mean(timed_steps(lambda: first_conv_forward(xb, wp), S)))
                old_tf32 = torch.backends.cudnn.allow_tf32
                torch.backends.cudnn.allow_tf32 = True
                for _ in range(3):
                    torch.nn.functional.conv2d(xb, wc, stride=2, padding=3)
                l_ms = float(np.mean(timed_steps(lambda: torch.nn.functional.conv2d(xb, wc, stride=2, padding=3), S)))
                torch.backends.cudnn.allow_tf32 = old_tf32
            Ho, Wo = (X - 1) // 2 + 1, (Y - 1) // 2 + 1
            flops = 2.0 * frames * Ho * Wo * 64 * 64 * 49
            try:
                with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                    bf16_peak = float(json.load(fh)["bf16_tflops"])
            except (OSError, ValueError, KeyError):
                bf16_peak = 1590.0
            conv_extra = {"frames": frames, "ms_per_call": c_ms, "tflops": flops / (c_ms * 1e-3) / 1e12, "flops": flops,
                          "library_cudnn_tf32_ms": l_ms, "tf32_peak_tflops": bf16_peak / 2,
                          "frac_of_tf32_peak": flops / (c_ms * 1e-3) / 1e12 / (bf16_peak / 2),
                          "what": "fiery_b200.bev_conv.first_conv_forward (tcgen05 kind::tf32 implicit GEMM, TMA stride-2 im2col) on a "
                                  "channel-last (B', 200, 200, 64) fp32 BEV; peak = measured cuBLAS bf16 burst / 2 (TF32 runs at half the "
                                  "bf16 rate); library line: torch conv2d, cuDNN with allow_tf32, same tensors; L2 flushed before every call"}
        except Exception as exc:               # an extra must never take the bench line down
            conv_extra = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    depth_extra = None
    if rank == 0 and not args.no_extras:
        try:
            from fiery_b200.depth_layer import depth_layer_forward, pack_weight as pack_depth_weight
            n_out = cfg.head_channels
            fh, fw = cfg.feat_hw
            feat16 = torch.randn(frames * cfg.n_cameras, 128, fh, fw, device=dev).half()          # the backbone's output under AMP
            wd = torch.randn(n_out, 128, 1, 1, device=dev) * 0.05
            bd = torch.randn(n_out, device=dev)
            wdp, wd16, bd16 = pack_depth_weight(wd, torch.float16), wd.half(), bd.half()
            with torch.no_grad():
                for _ in range(3):
                    depth_layer_forward(feat16, wd, bd, wdp)
                    torch.nn.functional.conv2d(feat16, wd16, bd16).float()
                d_ms = float(np.mean(timed_steps(lambda: depth_layer_forward(feat16, wd, bd, wdp), S)))
                dl_ms = float(np.mean(timed_steps(lambda: torch.nn.functional.conv2d(feat16, wd16, bd16), S)))
                dlw_ms = float(np.mean(timed_steps(lambda: torch.nn.functional.conv2d(feat16, wd16, bd16).float(), S)))
            d_bytes = feat16.numel() * 2 + feat16.shape[0] * n_out * fh * fw * 4 + 128 * 128 * 2
            depth_extra = {"frames": frames, "ms_per_call": d_ms, "bytes": d_bytes, "achieved_gbs": d_bytes / (d_ms * 1e-3) / 1e9,
                           "library_cudnn_fp16_ms": dl_ms, "library_cudnn_fp16_plus_widening_ms": dlw_ms,
                           "what": "fiery_b200.depth_layer.depth_layer_forward (Encoder.depth_layer, encoder.py:36,96: persistent tcgen05 "
                                   "kind::f16 GEMM, fp16 NCHW features in, fp32 NCHW head tensor out, TMA both ways); bytes = features "
                                   "read once + head written once + weights; library lines: torch conv2d (cuDNN, fp16 out) alone and "
                                   "followed by the .float() an AMP step needs before the fp32 lift; L2 flushed before every call"}
            del feat16
        except Exception as exc:               # an extra must never take the bench line down
            depth_extra = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    def reduce_max(x):
        if not distributed:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ms_dev = reduce_max(float(np.mean(t_dev)))
    ms_dev_noflush = reduce_max(float(np.mean(t_dev_noflush)))
    ms_static = reduce_max(float(np.mean(t_static)))
    ms_eager = reduce_max(float(np.mean(t_eager)))
    ms_fb = reduce_max(float(np.mean(t_fb)))
    ms_fb_graph = reduce_max(float(np.mean(t_fb_graph)))
    ms_bwd = reduce_max(float(np.mean(t_bwd)))
    ms_bwd_cl = reduce_max(float(np.mean(t_bwd_cl)))
    ms_e2e = reduce_max(float(np.mean(t_e2e)))
    total_frames = frames * world

    if rank == 0:
        peak, peak_src = load_peaks()
        gbs = lambda nbytes, ms: nbytes / (ms * 1e-3) / 1e9                     # noqa: E731
        es = head_d.element_size()
        alg_bytes = cfg.fwd_bytes_per_frame(head_itemsize=es) * frames
        head_bytes = head_d.numel() * es
        bev_bytes = frames * cfg.out_channels * X * Y * 4
        # counts of the plan: runs / stream entries written by the plan kernel, pillars that receive a point (accumulator rows the tile
        # kernels reduce into and the layout pass gathers)
        ps = lift.plan_summary(plan_d, frames, cfg.n_cameras)
        touched_rows = ps["touched_pillars"]
        row_bytes = cfg.out_channels * 4
        own = {"lift_forward_cols_kernel": head_bytes + touched_rows * row_bytes,             # read head once, each touched row written once
               "finalize_tma_kernel": 2 * touched_rows * row_bytes + bev_bytes}               # gather + re-zero touched rows, write the BEV
        traffic = load_traffic(cfg.name) if args.head_dtype == "f32" else {}
        kernels = []
        for k, name in KIND.items():
            if not per_kind[k]:
                continue
            n_launch = len(per_kind[k]) // S
            mean_ms = float(np.mean(per_kind[k]))
            kernels.append({"kernel": name, "launches_per_step": n_launch, "ms_per_launch": mean_ms,
                            "algorithmic_bytes_per_launch": own[name] // max(1, n_launch),
                            "achieved": gbs(own[name] / max(1, n_launch), mean_ms), "unit": "GB/s",
                            "frac": gbs(own[name] / max(1, n_launch), mean_ms) / peak,
                            "traffic_per_step": traffic.get(name)})
        bwd_alg = cfg.bwd_bytes_per_frame(head_itemsize=4) * frames
        line = {
            "metric": METRIC, "value": total_frames / (ms_dev * 1e-3), "unit": "frames/s", "n_gpus": world, "steps": S,
            "warmup": W, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "ms_per_step_median_rank0": float(np.median(t_dev)), "ms_per_step_max_rank0": float(np.max(t_dev)),
            "value_no_l2_flush": total_frames / (ms_dev_noflush * 1e-3), "ms_per_step_no_l2_flush": ms_dev_noflush,
            "value_static_rig": total_frames / (ms_static * 1e-3), "ms_per_step_static_rig": ms_static,
            "value_eager": total_frames / (ms_eager * 1e-3), "ms_per_step_eager": ms_eager,
            "fwd_bwd": {"value": total_frames / (ms_fb_graph * 1e-3), "unit": "frames/s", "ms_per_step": ms_fb_graph,
                        "frac_of_hbm_peak": (cfg.fwd_bytes_per_frame(4) + cfg.bwd_bytes_per_frame(4)) * frames / (ms_fb_graph * 1e-3) / 1e9 / load_peaks()[0],
                        "ms_per_step_eager_autograd": ms_fb,
                        "what": "the lift's training path: geometry plan + forward (planned) + backward to the head tensor, NCHW BEV and "
                                "gradient, C ABI with static buffers, CUDA-graph replay (device time); ms_per_step_eager_autograd = "
                                "LiftSplat.forward + autograd backward from Python (host-bound)"},
            "config": config_dict(cfg, args, world),          # identical in both arms
            "details": {"parallelism": f"frames sharded over {world} GPU(s), no data-path collective",
                        "l2": "flushed before every timed step (256 MiB write); step time = CUDA events around the step",
                        "api": "value: LiftSplat.capture() CUDA-graph replay (tile kernels incl. geometry + layout passes every step); "
                               "value_static_rig: capture(static_calibration=True); value_eager: LiftSplat.forward; "
                               "e2e: LiftSplat.lift_from_host (pinned host in/out, 3-stream chunk pipeline)",
                        "host": {"numa_node": numa[0], "cores_bound": numa[1], "note": numa[2]},
                        "timing": "mean over steps, max over ranks"},
            "e2e": {"value": total_frames / (ms_e2e * 1e-3), "unit": "frames/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": int(head_h.numel() * head_h.element_size() + K_h.numel() * 4 + E_h.numel() * 4),
                    "d2h_bytes_per_step": int(out_h.numel() * 4)},
            # kernels of the timed `value` region: per step and frame group one tile kernel (+ one layout pass)
            "gpu_launches": launches_per_step * S,
            "roofline": {"bound": "hbm", "kernel": "path: " + " + ".join(k["kernel"] for k in kernels),
                         "achieved": gbs(alg_bytes, ms_dev), "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                         "frac": gbs(alg_bytes, ms_dev) / peak,
                         "traffic": (sum(v for v in traffic.values()) if traffic else None),
                         "algorithmic_bytes_per_step": alg_bytes, "step_ms": ms_dev,
                         "frac_no_l2_flush": gbs(alg_bytes, ms_dev_noflush) / peak,
                         "frac_static_rig": gbs(alg_bytes, ms_static) / peak,
                         "touched_pillars": touched_rows, "kernels": kernels,
                         "how": "frac = algorithmic bytes of the step (head read once + BEV written once, SURVEY.md 8d) / graph-replay "
                                "step time / measured copy bandwidth; kernels[]: own algorithmic bytes (DESIGN.md section 4) / mean "
                                "duration of the launches the step runs (chains overlap, so durations include contention)"},
            "roofline_bwd": {"bound": "hbm", "kernel": "nchw_to_nhwc_kernel + lift_backward_kernel",
                             "achieved": gbs(bwd_alg, ms_bwd), "peak": peak, "unit": "GB/s", "frac": gbs(bwd_alg, ms_bwd) / peak,
                             "algorithmic_bytes_per_step": bwd_alg, "step_ms": ms_bwd,
                             "channels_last_grad": {"kernel": "lift_backward_kernel", "step_ms": ms_bwd_cl,
                                                    "achieved": gbs(bwd_alg, ms_bwd_cl), "frac": gbs(bwd_alg, ms_bwd_cl) / peak},
                             "traffic": (sum(load_traffic(cfg.name + "__bwd").values()) or None),
                             "how": "fiery_lift_backward with the forward's plan, eager C-ABI call, L2 flushed before every step; "
                                    "algorithmic bytes = read grad BEV + read head + write grad head (SURVEY.md 8d)"},
            "clocks": clocks,
        }
        if vs_extra is not None:
            line["voxels_summing_dropin"] = vs_extra
        if conv_extra is not None:
            line["next_row_first_bev_conv"] = conv_extra
        if depth_extra is not None:
            if "achieved_gbs" in depth_extra:
                depth_extra["frac_of_hbm_peak"] = depth_extra["achieved_gbs"] / peak
            line["next_row_depth_layer"] = depth_extra
        if warp_extra is not None:
            if "achieved_gbs" in warp_extra:
                warp_extra["frac_of_hbm_peak"] = warp_extra["achieved_gbs"] / peak
            line["next_row_cumulative_warp"] = warp_extra
        if not args.no_cpu_baseline:
            if not args.no_extras:
                # the reference's own op chain (torch library kernels: softmax, inverse, argsort, cumsum, index_put ...) on this
                # GPU -- the GPU-vs-GPU comparison SURVEY.md section 8d asks for next to the CPU number; baseline only
                from oracle import lift_oracle as O
                o_gpu = O.LiftOracle.from_config(cfg).to(dev)
                head_ref = head_d.float()                     # the reference's chain is timed on fp32 values
                with torch.no_grad():
                    for _ in range(2):
                        o_gpu.lift(head_ref, K_d, E_d)
                    t_ref_gpu = timed_steps(lambda: o_gpu.lift(head_ref, K_d, E_d), 5)
                line["reference_ops_on_gpu"] = {"value": frames / (float(np.mean(t_ref_gpu)) * 1e-3), "unit": "frames/s",
                                                "ms_per_step": float(np.mean(t_ref_gpu)),
                                                "what": "oracle/lift_oracle.py (the reference's PyTorch op chain) on CUDA tensors, "
                                                        "torch library kernels, same inputs, 5 steps"}
            fps, sec, threads, _ = time_cpu_reference(cfg, min(frames, args.cpu_frames), reps=args.cpu_reps)
            line["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                                    "sample": f"{args.cpu_reps} reps of {min(frames, args.cpu_frames)} frame(s) of {cfg.name}: "
                                              f"torch-CPU op chain of the reference (oracle/lift_oracle.py), median, "
                                              f"{threads} threads (fastest of the thread counts tried, {os.cpu_count()} cores)"}
        print(json.dumps(line), flush=True)
    if distributed:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
