#!/usr/bin/env python
"""Headline benchmark: driver frames/sec/GPU @512x512 through the volumetric-avatar hot path (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # B200 arm (this framework)
    python bench.py --impl reference --gpus N --steps K ...   # reference arm: the reference's CPU path (oracle port)

One "step" = one driver frame (batch 1) through head-pose regressor -> expression embedder -> predict_embed ->
uv warp generator -> 2 x grid_sample_3d -> decoder, against a cached source identity (the throughput path,
notebooks/infer.py:511-644).  N > 1: rank 0 runs the source pass, broadcasts the identity state over NCCL, every rank
then processes its own K frames (weak scaling, no data-path collective).

--dump-outputs DIR writes, after the timed steps, what the timed path returned in its last step as DIR/<name>.npy (float32):
the driver frame's image, or stage 2's (resized, add, ffhq).  The inputs are seeded, so two builds run with the same arguments
can be compared output for output.  Nothing is written into the source tree (bytecode caches included).
"""
from __future__ import annotations

import argparse
import json
import os
import pathlib
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the tree may be read-only; importing the package must not add __pycache__ to it

SIZE = 512
DUMP_BYTES = 64 * 10 ** 6  # --dump-outputs: at most this much in all, .npy headers included
METRIC = "driver frames/sec/GPU @512^2 (shipped model: 96ch x 16 x 64 x 64 volume); grid_sample_3d HBM GB/s vs peak"


def frame(size, seed):
    a = (np.random.RandomState(seed).rand(size, size, 3) * 255).astype(np.uint8)
    return torch.from_numpy(a).permute(2, 0, 1)[None].float().div(255).contiguous()


def dump_outputs(out_dir, arrays):
    """Write name -> tensor as out_dir/<name>.npy, float32.  If the arrays hold more than DUMP_BYTES in all, each is replaced by
    the same fraction of its flattened elements, drawn without replacement by a fixed seed (sorted flat indices), so that two
    runs with the same arguments write the same positions."""
    out = pathlib.Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total, budget = sum(a.nbytes for a in arrays.values()), DUMP_BYTES - 4096 * len(arrays)
    for name, a in arrays.items():
        if total > budget:
            a = a.reshape(-1)
            keep = a.size * budget // total
            a = a[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(out / f"{name}.npy", np.ascontiguousarray(a, dtype=np.float32))


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.nv = None

    def start(self):
        # NVML polled every 5 ms from a thread (the timed region lasts ~0.15 s; nvidia-smi -lms 100 would see it once or twice)
        try:
            import threading
            import pynvml as N
            N.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.idx]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else self.idx
            h = N.nvmlDeviceGetHandleByIndex(phys)
            self.nv = {"sm": [], "reasons": set(), "stop": False, "max": float(N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM))}
            bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

            def poll():
                while not self.nv["stop"]:
                    try:
                        self.nv["sm"].append(float(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)))
                        r = N.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        for k, b in bits.items():
                            if r & b:
                                self.nv["reasons"].add(k)
                    except Exception:
                        pass
                    time.sleep(0.005)

            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if getattr(self, "nv", None):
            self.nv["stop"] = True
            self.thread.join(timeout=1)
            sm = self.nv["sm"]
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.nv["max"], "reasons": sorted(self.nv["reasons"]),
                    "samples": len(sm), "how": "NVML polled every 5 ms during the timed region"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_port_fps(steps, warmup, threads=None):
    """The reference's own path on the host cores: the oracle port (oracle/restatement.py — the reference is Python and
    cannot travel to the GPU box).  Timed on a bounded sample: `steps` driver frames at 512^2."""
    from emoportraits_b200.checkpoint import synthetic_head_pose_state_dict, synthetic_state_dict
    from emoportraits_b200.config import shipped_config
    from oracle import restatement as R

    if threads is None:
        # "all the host threads it can use": pick the thread count that is fastest for a representative conv
        # (oversubscribed or quota-limited boxes get slower past a point)
        avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        x, w = torch.randn(1, 128, 256, 256), torch.randn(128, 128, 3, 3)
        best = (1e9, 1)
        for t in sorted({min(avail, c) for c in (8, 16, 32, 64, avail)}):
            torch.set_num_threads(t)
            torch.nn.functional.conv2d(x, w, padding=1)
            t0 = time.perf_counter()
            for _ in range(3):
                torch.nn.functional.conv2d(x, w, padding=1)
            dt = time.perf_counter() - t0
            if dt < best[0]:
                best = (dt, t)
        threads = best[1]
    torch.set_num_threads(threads)
    cfg = shipped_config(SIZE)
    sd, hsd = synthetic_state_dict(cfg, 0), synthetic_head_pose_state_dict(0)
    ocfg = R.config_from_state_dict(sd, SIZE)
    with torch.no_grad():
        # source state: the driver loop only needs the cached identity; build a cheap synthetic one of the right shape
        st = {"idt_embed": torch.randn(1, 512, 4, 4) * 0.5,
              "source_theta": R.get_transform_matrix(torch.tensor([[1., 1., 1.]]), torch.tensor([[.15, -.1, .05]]), torch.tensor([[.03, -.02, .01]])),
              "target_latent_volume": torch.randn(1, cfg.C, cfg.D, cfg.S, cfg.S)}
        drv = [frame(SIZE, 100 + i) for i in range(max(steps, 1))]
        for i in range(warmup):
            R.driver_pass(sd, hsd, st, drv[i % len(drv)], ocfg)
        t0 = time.perf_counter()
        for i in range(steps):
            R.driver_pass(sd, hsd, st, drv[i % len(drv)], ocfg)
        dt = time.perf_counter() - t0
    return steps / dt, dt, threads


def wrapper_fps(sd, hsd, K):
    """frames/s through emoportraits_b200.infer.InferenceWrapper.forward with PIL images in and PIL images out (uint8 H2D,
    on-device ToTensor, captured driver frame, on-device clamp + uint8, D2H, PIL.Image.fromarray), wall clock."""
    from PIL import Image

    from emoportraits_b200.infer import InferenceWrapper

    args_txt = ROOT / "tests" / "golden" / f"args_{SIZE}.txt"
    w = InferenceWrapper(experiment_name="bench", model_file_name="", project_dir=str(ROOT), args_path=args_txt, state_dict=sd,
                         head_pose_state_dict=hsd, print_params=False)
    pil = [Image.fromarray((np.random.RandomState(2000 + i).rand(SIZE, SIZE, 3) * 255).astype(np.uint8)) for i in range(8)]
    kw = dict(crop=False, mix=True, mix_old=False)
    w.forward(pil[0], pil[1], **kw)
    for i in range(3):
        w.forward(None, pil[i], **kw)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(K):
        out, img = w.forward(None, pil[i % 8], **kw)
    torch.cuda.synchronize()
    per_call = K / (time.perf_counter() - t0)
    LIST = 32  # frames per call of the list form (a caller with a long clip hands it over in chunks: one call converts, copies
    batch = [pil[i % 8] for i in range(LIST)]  # back and wraps ALL of its frames after the last one is computed)
    w.forward(None, batch[:4], **kw)
    torch.cuda.synchronize()
    calls = max(1, K // LIST)
    t0 = time.perf_counter()
    for _ in range(calls):
        out, img = w.forward(None, batch, **kw)
    torch.cuda.synchronize()
    listed = calls * LIST / (time.perf_counter() - t0)
    assert len(out) == LIST and out[0].size == (SIZE, SIZE)
    return {"one_frame_per_call": per_call, "list_of_frames_per_call": listed, "frames_per_list_call": LIST, "unit": "frames/s",
            "what": "InferenceWrapper.forward(None, PIL...) -> (list[PIL], tensor): uint8 H2D 0.79 MB + D2H 0.79 MB per frame, wall clock"}


def graph_time_conv(shape_key: str, reps: int = 10):
    """Device time per launch of one conv shape of the frame, free of host launch cost: CUDA-graph replays of `reps` back-to-back
    launches (with and without a same-resolution residual: the ResBlock's two convs), CUDA events on the replaying stream.
    shape_key as ops.ConvProfiler names it: 'NxDxHxWxCin->Cout kDHW sS pP[ up2-subpixel]'."""
    import math
    import re

    from emoportraits_b200 import ops

    m = re.match(r"(\d+)x(\d+)x(\d+)x(\d+)x(\d+)->(\d+) k(\d)(\d)(\d) s(\d) p(\w+)( up2-subpixel)?", shape_key)
    if not m:
        return None
    N, D, H, W, Ci, Co, kd, kh, kw, st_, pl, up = m.groups()
    N, D, H, W, Ci, Co, kd, kh, kw, st_ = map(int, (N, D, H, W, Ci, Co, kd, kh, kw, st_))
    planes = "h2" if pl == "h2" else int(pl)
    dev = "cuda"
    x = torch.randn((N, D, H, W, Ci), device=dev)
    w = torch.randn((Co, Ci, kd, kh, kw) if kd > 1 else (Co, Ci, kh, kw), device="cpu") / math.sqrt(Ci * kd * kh * kw)
    a = ops.split_bf16(x, planes)
    pw = ops.pack_upconv_weight(w) if up else ops.pack_conv_weight(w, planes=planes)
    stride = (1, st_, st_)
    pad = (kd // 2, 1, 1) if kh == 4 else None            # the folded `conv -> avgpool` is a 4x4 stride-2 pad-1 convolution
    Ho, Wo = (2 * H, 2 * W) if up else ((H + 2 * (1 if kh == 4 else kh // 2) - kh) // st_ + 1, (W + 2 * (1 if kw == 4 else kw // 2) - kw) // st_ + 1)
    oshape = (N, D, Ho, Wo, Co)
    out = torch.empty(oshape, device=dev)
    bias = torch.zeros(Co, device=dev)
    res_full = torch.randn(oshape, device=dev) if Co % 4 == 0 else None
    times = {}
    for label, res in (("no_residual", None), ("residual", res_full)):
        ops.begin_pass(dev)
        stt = ops.new_stats(N, 32, dev) if Co % 32 == 0 else None
        run = lambda: ops.conv_igemm(a, pw, stride=stride, pad=pad, out=out, bias=bias, residual=res, stats=stt, upconv=bool(up))
        for _ in range(2):
            run()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(reps):
                run()
        g.replay(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            g.replay()
        e1.record(); torch.cuda.synchronize()
        times[label] = e0.elapsed_time(e1) / (5 * reps) * 1000.0
    return times


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = args.steps, args.warmup
    fps, dt, threads = cpu_port_fps(steps, warm)
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": 1000.0 / fps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": f"driver frame @{SIZE}^2, C96 D16 S64, batch 1 (configs[1])", "host_threads": threads},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                         "sample": f"{steps} driver frames @512^2 after {warm} warm-up, oracle/restatement.py (torch CPU fp32)"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def grid_sample_roofline(peaks, reps=20):
    """config 3 microbench (SURVEY §8d): 96ch volume, D=64 (BASELINE's "64^3") and D=16 (model-true), channels-last,
    L2 flushed between reps (256 MB written and read back; the write-only flush is reported beside it).  Variants: `jitter` = identity lattice + 0.1*randn grid tensor (the spec'd
    workload: sigma = 3.2 voxels, i.e. an L2-resident random gather), `affine` = fused theta lattice (30 deg rotation +
    0.2 translation; no grid tensor; the hot path's rotation warp), batch 1, 8 and 32 (BASELINE configs[2]: "batch 1-32")."""
    import math

    from emoportraits_b200 import ops

    out = {}
    dev = "cuda"
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    a = math.radians(30)
    theta1 = torch.tensor([[[math.cos(a), -math.sin(a), 0, 0.2], [math.sin(a), math.cos(a), 0, 0.2], [0, 0, 1.0, 0.2]]])

    def timeit(fn, clean=True):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(reps):
            ops.l2_flush(flush, clean=clean)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return float(np.median(ts))

    def entry(fn, alg):
        # headline: L2 flushed and left CLEAN (256 MB written, then read back); `*_dirty_flush`: after the write pass only, when
        # the kernel under test also pays for the write-back of the flush's own 126 MB of dirty lines (8 us at 64^3, measured)
        ms, ms_d = timeit(fn, True), timeit(fn, False)
        return {"ms": ms, "algorithmic_bytes": alg, "achieved_gbs": alg / ms / 1e6, "frac": alg / ms / 1e6 / peaks["hbm_gbs"],
                "ms_dirty_flush": ms_d, "frac_dirty_flush": alg / ms_d / 1e6 / peaks["hbm_gbs"]}

    for name, D, B in (("d64", 64, 1), ("d16", 16, 1), ("d64_b8", 64, 8), ("d64_b32", 64, 32)):
        try:
            C, S = 96, 64
            zs, ys = torch.linspace(-1, 1, D), torch.linspace(-1, 1, S)
            w, v, u = torch.meshgrid(zs, ys, ys, indexing="ij")
            if B <= 8:
                g = torch.Generator(device="cpu").manual_seed(0)
                vol = torch.randn(B, D, S, S, C, generator=g).to(dev)
                grid = (torch.stack([u, v, w], -1)[None] + 0.1 * torch.randn(B, D, S, S, 3, generator=g)).contiguous().to(dev)
            else:  # BASELINE configs[2] upper end (25.8 GB in, 25.8 GB out): generate on the device
                g = torch.Generator(device=dev).manual_seed(0)
                vol = torch.randn(B, D, S, S, C, generator=g, device=dev)
                grid = (torch.stack([u, v, w], -1)[None].to(dev) + 0.1 * torch.randn(B, D, S, S, 3, generator=g, device=dev)).contiguous()
            theta = theta1.repeat(B, 1, 1).contiguous().to(dev)
            out[name] = entry(lambda: ops.grid_sample3d(vol, grid=grid, in_layout="cl"), (2 * C * D * S * S + 3 * D * S * S) * 4 * B)
            out[name + "_affine"] = entry(lambda: ops.grid_sample3d(vol, theta=theta, out_size=(D, S, S), in_layout="cl"),
                                          (2 * C * D * S * S) * 4 * B)
            del vol, grid
        except RuntimeError as e:  # e.g. out of memory on a shared device: report, do not lose the whole bench line
            out[name] = {"error": str(e)[:200]}
        torch.cuda.empty_cache()
    return out


def run_ours(args):
    import torch.distributed as dist

    from emoportraits_b200 import lib as L
    from emoportraits_b200 import ops
    from emoportraits_b200.checkpoint import synthetic_head_pose_state_dict, synthetic_state_dict
    from emoportraits_b200.config import shipped_config
    from emoportraits_b200.infer import Model

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (B200 arm) needs a GPU; use --impl reference for the CPU arm"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    cfg = shipped_config(SIZE)
    sd, hsd = synthetic_state_dict(cfg, 0), synthetic_head_pose_state_dict(0)
    model = Model(cfg, sd, hsd, dev)
    peaks = measured_peaks()

    # ---- source pass on rank 0, identity state broadcast over NCCL (SURVEY §8e) ----
    from emoportraits_b200.dist import broadcast_source_state

    st = model.source_pass(frame(SIZE, 0).to(dev)) if rank == 0 else None
    broadcast_ms = None
    if world > 1:
        # the one exchange step of the path (SURVEY 8e): 25.2 MB identity state from the rank that ran the source pass.
        # First call = NCCL communicator warm-up; the second is timed with CUDA events, max over ranks.
        st0 = st
        st = broadcast_source_state(st0, cfg, dev, src=0)
        torch.cuda.synchronize()
        dist.barrier()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record()
        st = broadcast_source_state(st0 if rank == 0 else st, cfg, dev, src=0)
        b1.record()
        torch.cuda.synchronize()
        tb = torch.tensor([b0.elapsed_time(b1)], device=dev)
        dist.all_reduce(tb, op=dist.ReduceOp.MAX)
        broadcast_ms = tb.item()
    torch.cuda.synchronize()

    K, W = args.steps, max(args.warmup, 3)
    frames_host = [frame(SIZE, 1000 + rank * 131 + i).pin_memory() for i in range(8)]
    frames_dev = [f.to(dev) for f in frames_host]

    from emoportraits_b200.infer import DriverPipeline

    depth = 1 if args.eager else max(1, args.inflight)
    pipe = DriverPipeline(model, st, depth=depth, mix=True) if not args.eager else None
    runner = pipe.slots[0].run if pipe is not None else None

    def step_dev(i):
        if pipe is not None:
            return pipe.submit(frames_dev[i % len(frames_dev)])
        return model.driver_pass(st, frames_dev[i % len(frames_dev)], mix=True)[0]

    ring = 2 * depth  # frames the host may run ahead: two per stream, so that neither stream ever drains
    out_hosts = [torch.empty((1, 3, SIZE, SIZE), dtype=torch.float32).pin_memory() for _ in range(ring)]
    tickets = [None] * ring

    def step_e2e(i):
        # the call a user makes per video frame: pinned host frame in, host image out.  The host blocks on frame i - ring
        # (its image is then in out_hosts[i % ring] and the buffer may be reused) before it queues frame i.
        if pipe is not None:
            t = tickets[i % ring]
            if t is not None:
                t.done.synchronize()
            tickets[i % ring] = pipe.submit(frames_host[i % len(frames_host)], host_out=out_hosts[i % ring])
            return
        x = frames_host[i % len(frames_host)].to(dev, non_blocking=True)
        img = model.driver_pass(st, x, mix=True)[0]
        out_hosts[0].copy_(img, non_blocking=True)
        torch.cuda.synchronize()

    def drain():
        if pipe is not None:
            pipe.drain()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ----
    for i in range(W):
        step_dev(i)
    drain()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = L.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last = None
    for i in range(K):
        last = step_dev(i)
    drain()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    # what the caller received in the last timed step (frame K - 1's image), copied out before the e2e loop reuses the slots
    outputs = None
    if args.dump_outputs and rank == 0 and last is not None:
        outputs = {"image": (last.slot.run.static_out if pipe is not None else last).cpu()}
    launches_eager = L.launch_count - l0
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = t.item()

    # ---- end-to-end: pinned host frame in, host image out, every step ----
    for i in range(2 * ring):
        step_e2e(i)
    drain()
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        step_e2e(i)
    drain()
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = t.item()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    frame_ms = ms_max / K
    # ---- latency of ONE frame alone (what an interactive caller sees): one captured frame at a time, device-resident ----
    lat_pipe = DriverPipeline(model, st, depth=1, mix=True) if not args.eager else None
    latency_ms = None
    if lat_pipe is not None:
        for i in range(3):
            lat_pipe.submit(frames_dev[i % len(frames_dev)])
        lat_pipe.drain(); torch.cuda.synchronize()
        l0e, l1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0e.record()
        for i in range(K):
            lat_pipe.submit(frames_dev[i % len(frames_dev)])
        lat_pipe.drain()
        l1e.record(); torch.cuda.synchronize()
        latency_ms = l0e.elapsed_time(l1e) / K
        del lat_pipe
    # ---- the drop-in call itself: InferenceWrapper.forward(None, PIL) -> (list[PIL], tensor), one frame per call and a
    #      list of frames per call (notebooks/infer.py:355-357; E_emo_infer_video.ipynb calls it per frame) ----
    e2e_wrapper = None
    if not args.quick:
        e2e_wrapper = wrapper_fps(sd, hsd, K)
    # ---- per-kernel evidence (rank 0, eager, CUDA events around every tensor-core conv launch) ----
    prof = ops.ConvProfiler()
    ops.set_conv_profiler(prof)
    l0 = L.launch_count
    for i in range(3):
        model.driver_pass(st, frames_dev[i % len(frames_dev)], mix=True)
    torch.cuda.synchronize()
    launches_per_step = (L.launch_count - l0) // 3
    ops.set_conv_profiler(None)
    conv_ms, conv_flops, n_conv = prof.summary()
    if args.layer_csv:
        with open(args.layer_csv, "w") as f:
            f.write("shape,launches(3 frames),ms_total,algorithmic_TFLOPs,mma_TFLOPs\n")
            for r in prof.table():
                f.write(f"{r[0]},{r[1]},{r[2]:.4f},{r[3]:.1f},{r[4]:.1f}\n")
    conv_tflops = conv_flops / conv_ms / 1e9 if conv_ms > 0 else 0.0
    # the dominant kernel instance: the conv shape with the largest total time in the frame
    top = prof.table()[0]
    top_shape, top_n, top_ms, top_alg_tf, top_mma_tf = top
    top_ms_per_launch = top_ms / top_n
    # the dominant shape once more WITHOUT host launch cost (the eager table above carries it): graph-timed
    top_graph = graph_time_conv(top_shape)
    if top_graph:
        top_us = 0.5 * (top_graph["no_residual"] + top_graph["residual"])
        top_flops = top_alg_tf * 1e12 * (top_ms_per_launch * 1e-3)          # algorithmic flops of one launch
        top_alg_tf_graph = top_flops / (top_us * 1e-6) / 1e12
    else:
        top_us, top_alg_tf_graph = top_ms_per_launch * 1000.0, top_alg_tf
    # every conv shape of the frame the same way: sum of graph-timed launch durations vs the frame's algorithmic conv flops
    conv_us_graph, conv_flops_graph = 0.0, 0.0
    for name, n_l, ms_l, alg_tf_l, _ in prof.table():
        gt = graph_time_conv(name) if not args.quick else None
        if gt is None:
            conv_us_graph = None
            break
        us_l = 0.5 * (gt["no_residual"] + gt["residual"])
        conv_us_graph += us_l * (n_l / 3.0)
        conv_flops_graph += alg_tf_l * 1e12 * (ms_l * 1e-3) / 3.0
    traffic = None
    tf = ROOT / "profiles" / "traffic.json"
    if tf.exists():
        traffic = json.loads(tf.read_text()).get(top_shape)
    gs = grid_sample_roofline(peaks) if not args.quick else {"d64_affine": {"achieved_gbs": 0.0, "frac": 0.0}, "skipped": "--quick"}

    cpu = None
    if world == 1 and not args.no_cpu_baseline and not args.quick:
        fps_cpu, dt, threads = cpu_port_fps(4, 1)
        cpu = {"value": fps_cpu, "unit": "frames/s", "cores": threads, "kind": "port",
               "sample": f"4 driver frames @512^2 after 1 warm-up ({dt:.1f} s), oracle/restatement.py torch-CPU fp32"}

    fps = world * K / (ms_max / 1000.0)
    line = {
        "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": frame_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "two 16-bit operand planes per fp32 operand, 3 tcgen05 MMAs per product (bf16 x2 in the decoder, fp16 x2 elsewhere), fp32 accumulate / fp32 elsewhere",
        "data": "synthetic",
        "config": {"workload": f"driver frame @{SIZE}^2, shipped model C96 D16 S64, batch 1 (BASELINE configs[1]); "
                               "BASELINE's '64^3' volume is the grid_sample microbench shape, reported in roofline_grid_sample3d",
                   "parallelism": f"frame-parallel x{world}, NCCL broadcast of the identity state",
                   "l2": "per-step working set (~3 GB of activations + 0.3 GB of weights) exceeds the 126 MB L2; microbench flushes L2",
                   "cuda_graph": runner is not None,
                   "frames_in_flight": depth,
                   "e2e_host_run_ahead": ring,
                   "frames_in_flight_note": "consecutive driver frames replay on alternating streams (infer.DriverPipeline); "
                                            "each frame still runs alone through the same kernels, batch 1"},
        "e2e": {"value": world * K / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": 3 * SIZE * SIZE * 4,
                "d2h_bytes_per_step": 3 * SIZE * SIZE * 4},
        "gpu_launches": launches_per_step * K,
        "gpu_launches_per_step": launches_per_step,
        "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": f"conv_igemm_kernel, layer {top_shape} (largest share of the frame; {top_n // 3} launches/frame)",
                     "achieved": top_alg_tf_graph, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                     "frac": top_alg_tf_graph / peaks["bf16_tflops_sustained"], "traffic": traffic,
                     "launch_us": top_us,
                     "launch_us_how": "CUDA-graph replays of 10 back-to-back launches of this shape, CUDA events on the replaying stream, mean of the "
                                      "ResBlock's two forms (with / without residual)" if top_graph else "eager",
                     "launch_us_detail": top_graph, "launch_us_eager_incl_host": top_ms_per_launch * 1000.0,
                     "tensor_pipe_frac_est_graph": 3.0 * top_alg_tf_graph / peaks["bf16_tflops_sustained"],
                     "peak_source": peaks["source"] + ", sustained bf16 (kernel timed inside a long step)",
                     "mma_passes": "3 MMAs per algorithmic product (two-plane split operands)",
                     "tensor_pipe_frac_est": top_mma_tf / peaks["bf16_tflops_sustained"],
                     "all_convs": {"achieved": conv_tflops, "frac": conv_tflops / peaks["bf16_tflops_sustained"],
                                   "tensor_pipe_frac_est": (prof.mma_flops / conv_ms / 1e9) / peaks["bf16_tflops_sustained"],
                                   "algorithmic_flops_per_step": conv_flops / 3, "kernel_ms_per_step": conv_ms / 3,
                                   "launches_per_step": n_conv // 3, "share_of_step_eager": (conv_ms / 3) / frame_ms,
                                   "note": "CUDA events around every conv launch of 3 eager frames (host launch cost and tensor-map encoding inside)",
                                   "graph_timed": None if not conv_us_graph else {
                                       "kernel_ms_per_step": conv_us_graph / 1000.0, "achieved": conv_flops_graph / (conv_us_graph * 1e-6) / 1e12,
                                       "frac": conv_flops_graph / (conv_us_graph * 1e-6) / 1e12 / peaks["bf16_tflops_sustained"],
                                       "share_of_step": (conv_us_graph / 1000.0) / latency_ms if latency_ms else None,
                                       "how": "every conv shape of the frame as CUDA-graph replays of 10 back-to-back launches (split-K layers with their "
                                              "finalize), launches-per-frame weighted; share = of the one-frame-alone latency"}}},
        "roofline_grid_sample3d": {"bound": "hbm", "unit": "GB/s", "peak": peaks["hbm_gbs"], "peak_source": peaks["source"],
                                   "achieved": gs.get("d64", gs["d64_affine"]).get("achieved_gbs", 0.0), "frac": gs.get("d64", gs["d64_affine"]).get("frac", 0.0),
                                   "headline": "d64 = BASELINE configs[2] at batch 1: 96ch x 64^3 volume sampled through a 64^3 x 3 warp-field "
                                               "tensor (identity + 0.1 randn); *_affine = fused affine lattice (no grid tensor), d16 = model-true depth",
                                   "flush": "every rep runs on a flushed L2: 256 MB written and read back (L2 left full of clean foreign lines); "
                                            "ms_dirty_flush / frac_dirty_flush = after the write pass only (the kernel then also pays for the "
                                            "write-back of the flush's own dirty lines)", **gs},
    }
    if cpu:
        line["cpu_baseline"] = cpu
    if latency_ms is not None:
        line["latency_ms_one_frame_alone"] = latency_ms
    if e2e_wrapper is not None:
        line["e2e_wrapper"] = e2e_wrapper
    if broadcast_ms is not None:
        line["broadcast_ms"] = {"value": broadcast_ms, "bytes": 4 * (cfg.D * cfg.S * cfg.S * cfg.C + cfg.idt_channels * cfg.embed_size ** 2 + 16),
                                "what": "identity state rank 0 -> all ranks (second call, CUDA events, max over ranks); outside the timed region, once per identity"}
    if world == 1 and not args.quick:
        del pipe, model
        torch.cuda.empty_cache()
        try:
            line["stage2"] = stage2_numbers(5, 3)
        except RuntimeError as e:
            line["stage2"] = {"error": str(e)[:200]}
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def stage2_numbers(K, W, outputs=None):
    """BASELINE config 5: stage-2 refinement encoder+decoder @1024^2, batch 4 (secondary workload).  `outputs` (a dict): receives
    the (resized, add, ffhq) of the last timed step on the host."""
    from emoportraits_b200 import lib as L
    from emoportraits_b200 import ops
    from emoportraits_b200.stage2 import Stage2Config, Stage2Model, synthetic_state_dict_s2

    cfg = Stage2Config(output_size=1024)
    model = Stage2Model(cfg, synthetic_state_dict_s2(cfg, 0), "cuda")
    B = 4
    img = torch.rand(B, 3, 512, 512, generator=torch.Generator().manual_seed(0)).cuda()
    for _ in range(W):
        model.forward(img)
    torch.cuda.synchronize()
    prof = ops.ConvProfiler()
    l0 = L.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = None
    for _ in range(K):
        out = model.forward(img)
    e1.record()
    torch.cuda.synchronize()
    if outputs is not None and out is not None:
        outputs.update({name: t.cpu() for name, t in zip(("resized", "add", "ffhq"), out)})
    ms = e0.elapsed_time(e1) / K
    launches = (L.launch_count - l0) // K
    ops.set_conv_profiler(prof)
    model.forward(img)
    ops.set_conv_profiler(None)
    conv_ms, conv_flops, n_conv = prof.summary()
    peaks = measured_peaks()
    return {"metric": "stage-2 refinement images/s @1024^2, batch 4 (BASELINE configs[4])", "value": B * 1000.0 / ms, "unit": "images/s",
            "ms_per_step": ms, "steps": K, "warmup": W, "gpu_launches_per_step": launches,
            "config": {"workload": "stage-2 LocalEncoderOld + Decoder_stage2, output_size_s2 1024, batch 4, default stage-2 args"},
            "roofline": {"bound": "tensor", "kernel": "conv_igemm_kernel (all conv layers of one step)", "achieved": conv_flops / conv_ms / 1e9,
                         "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": conv_flops / conv_ms / 1e9 / peaks["bf16_tflops_sustained"],
                         "traffic": None, "tensor_pipe_frac_est": prof.mma_flops / conv_ms / 1e9 / peaks["bf16_tflops_sustained"]}}


def run_stage2(args):
    """`--workload stage2`: the secondary workload alone, as its own JSON line (the default run carries it under "stage2")."""
    torch.cuda.set_device(0)
    K, W = args.steps, max(args.warmup, 3)
    outputs = {} if args.dump_outputs else None
    d = stage2_numbers(K, W, outputs)
    if outputs:
        dump_outputs(args.dump_outputs, outputs)
    line = {"metric": d["metric"], "value": d["value"], "unit": d["unit"], "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": d["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16x2-split operands, fp32 accumulate",
            "data": "synthetic", "config": d["config"], "gpu_launches": d["gpu_launches_per_step"] * K, "roofline": d["roofline"]}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)  # 0.65 s of device time at ~300 frames/s: ~130 NVML clock samples in the timed region
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--eager", action="store_true", help="do not capture the driver frame in a CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="A/B runs: skip the grid_sample microbench and the CPU baseline (not a bench record)")
    ap.add_argument("--inflight", type=int, default=4, help="driver frames in flight per GPU (1 = strictly one after the other; measured "
                    "round 2, final tree: 239 / 291 / 304 / 312 frames/s with 1 / 2 / 3 / 4)")
    ap.add_argument("--workload", default="driver", choices=["driver", "stage2"],
                    help="driver = the headline metric (default); stage2 = BASELINE config 5, secondary")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step returned as "
                    "DIR/<name>.npy (float32; at most 64 MB in all, a fixed seeded sample of each array beyond that)")
    ap.add_argument("--layer-csv", metavar="FILE", help="write the per-conv-shape table of the eager profile to FILE")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the B200 arm (--impl ours)")
    # stdout carries exactly ONE JSON line: libraries that print to fd 1 (NCCL's version banner at the first collective)
    # are sent to stderr for the duration of the run, and print() is bound to the saved descriptor.
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(saved, "w", buffering=1)
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "stage2":
        run_stage2(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
