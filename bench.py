#!/usr/bin/env python
"""bench.py — throughput of the render hot path on B200 (BASELINE.json metric: Mrays/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c1|c2|c3|c4|c5] [--fast-math] [--dump-outputs DIR]
    python bench.py --impl reference ...          # the reference's CPU algorithm (oracle port)

A "step" is one full frame of the workload (one pass of the per-pixel render loop,
common.rs:320-361, over every pixel and sample).  A "ray" is one ray segment = one World::hit
call (common.rs:268), counted by the kernel itself.

  N = 1 : BASELINE config 2 — default scene, 1920x1080, 64 spp, depth 8 — one persistent
          render-kernel launch per step.
  N > 1 : BASELINE config 4 — default scene, 3840x2160, 1,024 spp as 16 progressive passes of
          64 spp (fused into one persistent launch per GPU), the frame sharded by 16-row tiles across
          the ranks (stripes of N tiles dealt alternately forwards and backwards, rt_shard_tile; the
          tail of the frame is stolen across GPUs over NVLink), the finished RGBA8 tiles stored by the
          render kernels into rank 0's frame over NVLink (the only exchange).
          Strong scaling: the frame is fixed, N GPUs split it.  The line carries, measured in the same
          run, the 1-GPU time of the same frame (`strong_scaling`) and `parity` (sha256 of the gathered
          frame == sha256 of the single-GPU frame, ray counts equal); a mismatch makes the run fail.

`value`  : rays/s with everything resident in HBM, timed with CUDA events on the launching
           stream, L2 flushed (256 MiB write) between steps outside the events, max over ranks.
`e2e`    : the same frame through the reference-facing C-ABI call with a PAGEABLE host framebuffer
           (render_with_options; what the reference's callers pass), the frame's way to the host inside
           the timed region; `e2e_pinned` is the same with an rt_alloc_pixels buffer.
`workloads` (N = 1 default line): C3, C5 and C4-on-one-GPU timed the same way, each with its roofline.
`roofline`: FP32 CUDA-core roofline (no tensor-core work exists on this path): algorithmic
           flops (DESIGN.md / SURVEY.md §8d) / kernel time / FFMA peak measured in this run.
The default kernel is the bit-exact one (IEEE arithmetic in the reference's association order,
no FMA contraction); --fast-math selects the relaxed kernel, which is not bit-exact.

--dump-outputs DIR writes the frame of the last timed step (rank 0; N > 1: the gathered frame) for
comparing two builds output for output: DIR/frame.npy, [H, W, 4] float32 RGBA values 0-255; a frame
over DUMP_BYTES (C4's 3840x2160) is written as a fixed seeded sample of its pixels instead,
DIR/frame_sample.npy [n, 4] float32 with DIR/frame_sample_index.npy [n] float64 (row-major pixel
index).  Scenes and render seeds are fixed, so the same arguments render the same frame.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOADS = {
    # key: (description, scene, W, H, spp, depth, passes)
    "c1": ("C1: default scene (world.txt, 8 spheres), 400x224, 50 spp, depth 8", "default", 400, 224, 50, 8, 1),
    "c2": ("C2: default scene (world.txt, 8 spheres), 1920x1080, 64 spp, depth 8", "default", 1920, 1080, 64, 8, 1),
    "c3": ("C3: synthetic 1,000 spheres, 1920x1080, 256 spp, depth 8", "c3", 1920, 1080, 256, 8, 1),
    "c4": ("C4: default scene, 3840x2160, 1,024 spp (16 progressive passes x 64), depth 8, 16-row tiles",
           "default", 3840, 2160, 1024, 8, 16),
    "c5": ("C5: synthetic 8,000 spheres + 2,000 triangles, 1280x720, 16 spp, depth 16", "c5", 1280, 720, 16, 16, 1),
}


# dram__bytes_read.sum + dram__bytes_write.sum of one render-kernel launch, from the committed
# `ncu --set full` captures (profiles/r02_bench.md); None where no capture of that exact launch exists.
NCU_TRAFFIC_BYTES = {("c2", False): 36352}      # 36.4 KB read, 0 B written: the 8.3 MB frame stays in the 126 MB L2
# Counters of the same captures, quoted (not measured in this run) so that the line explains its own
# `frac`: on the 8-sphere scene the counted-flops model covers less than half of the instructions a
# segment needs (IEEE divide/sqrt sequences, integer RNG, predicates), and the kernel is issue-bound.
NCU_CONTEXT = {
    ("c2", False): {"issue_slots_busy": 0.852, "ipc": 3.40, "fp32_pipe_active": 0.483, "alu_pipe_active": 0.502,
                    "active_lanes_per_warp": 20.1, "source": "profiles/r02_c2_exact_details.txt (16-spp capture)"},
    ("c3", False): {"issue_slots_busy": 0.654, "ipc": 2.61, "fp32_pipe_active": 0.614, "active_lanes_per_warp": 29.8,
                    "source": "profiles/r02_c3_exact_details.txt (8-spp capture; FFMA2 filter: two FMAs per issued instruction)"},
    ("c5", False): {"issue_slots_busy": 0.640, "ipc": 2.37, "fp32_pipe_active": 0.475, "active_lanes_per_warp": 21.3,
                    "source": "profiles/r02_c5_exact_details.txt (2-spp capture)"},
}


def scene_text(scenes, key):
    return {"default": scenes.default_world, "c3": scenes.c3_world, "c5": scenes.c5_world}[key]()


DUMP_BYTES = 64_000_000
DUMP_SAMPLE_PIXELS = 1 << 21          # 16 B of RGBA + 8 B of index each: 50.3 MB
DUMP_SAMPLE_SEED = 0


def dump_outputs(out_dir, rgba8):
    """--dump-outputs: rgba8 is the [H, W, 4] uint8 frame of the last timed step."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    if rgba8.size * 4 <= DUMP_BYTES:
        np.save(os.path.join(out_dir, "frame.npy"), rgba8.astype(np.float32))
        return
    px = rgba8.reshape(-1, 4)
    idx = np.sort(np.random.default_rng(DUMP_SAMPLE_SEED).choice(len(px), DUMP_SAMPLE_PIXELS, replace=False))
    np.save(os.path.join(out_dir, "frame_sample.npy"), px[idx].astype(np.float32))
    np.save(os.path.join(out_dir, "frame_sample_index.npy"), idx.astype(np.float64))


def algorithmic_flops(rays, samples, pixels, n_sph, n_tri):
    """SURVEY.md §8d: N_seg*(17*S + 12*T + 60) + N_s*34 + W*H*11, FMA counted as 2."""
    return rays * (17 * n_sph + 12 * n_tri + 60) + samples * 34 + pixels * 11


class ClockSampler:
    """Samples SM clock and clock-event reasons with NVML while the timed region runs."""

    def __init__(self, index: int, period: float = 0.05):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:       # noqa: BLE001
            self.nv, self.err = None, repr(e)
        self.period = period

    def _run(self):
        nv = self.nv
        names = {nv.nvmlClocksEventReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksEventReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksEventReasonHwPowerBrakeSlowdown: "hw_power_brake",
                 nv.nvmlClocksEventReasonApplicationsClocksSetting: "applications_clocks_setting"}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:        # noqa: BLE001
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        if self.nv:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread:
            self._thread.join()

    def summary(self):
        if not self.nv:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "error": self.err}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ---------------------------------------------------------------------------------- CPU legs

def cpu_baseline_serial(scenes, wl, budget_s=15.0):
    """The reference's algorithm (oracle port, serial RNG stream, 1 thread) on a bounded sample of
    the workload: the full frame at reduced spp (cost is exactly linear in spp)."""
    sys.path.insert(0, str(ROOT / "oracle"))
    import oracle_binding as ob
    desc, key, W, H, spp, depth, _ = wl
    cam, world = ob.parse_input(scene_text(scenes, key))
    # size the sample from a short probe
    probe_h = max(2, H // 16)
    t = time.perf_counter()
    _, r0, _ = ob.ray_trace(world, cam, W, probe_h, 1, depth, rng_mode=ob.RNG_SERIAL, threads=1)
    per_spp = (time.perf_counter() - t) * (H / probe_h)
    s = int(max(1, min(spp, budget_s / max(per_spp, 1e-6))))
    t = time.perf_counter()
    _, rays, _ = ob.ray_trace(world, cam, W, H, s, depth, rng_mode=ob.RNG_SERIAL, threads=1)
    dt = time.perf_counter() - t
    ncores = os.cpu_count() or 1
    t = time.perf_counter()
    _, rays_mt, _ = ob.ray_trace(world, cam, W, H, s, depth, rng_mode=ob.RNG_PER_SAMPLE, threads=ncores)
    dt_mt = time.perf_counter() - t
    return {"value": rays / dt / 1e6, "unit": "Mrays/s", "cores": 1, "kind": "port",
            "sample": f"{W}x{H} full frame at {s} of {spp} spp, depth {depth}; oracle/rt_oracle.c serial-RNG mode "
                      f"(the reference's one xorshift32 stream, common.rs:321), {dt:.1f} s; extrapolated frame time "
                      f"{dt * spp / s:.0f} s",
            "ms_per_frame_extrapolated": dt * spp / s * 1e3,
            "all_cores": {"value": rays_mt / dt_mt / 1e6, "cores": ncores,
                          "note": "oracle per-sample-RNG mode, OpenMP over rows (not something the reference can do)"}}


def run_reference(args, scenes):
    """--impl reference: the reference's CPU implementation of the path.  The Rust crate cannot be
    built in this image (no rustc/cargo), so this is the oracle port in the reference's own
    serial-RNG mode on 1 thread — the reference's render loop is single-threaded by construction
    (one &mut Random shared by every pixel, common.rs:321-340)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    sys.path.insert(0, str(ROOT / "oracle"))
    import oracle_binding as ob
    wl = WORKLOADS[args.workload]
    desc, key, W, H, spp, depth, _ = wl
    cam, world = ob.parse_input(scene_text(scenes, key))
    # one step = the full frame at `s` spp, sized so that (K + W) steps take <= ~60 s
    probe_h = max(2, H // 16)
    t = time.perf_counter()
    ob.ray_trace(world, cam, W, probe_h, 1, depth, rng_mode=ob.RNG_SERIAL, threads=1)
    per_spp = (time.perf_counter() - t) * (H / probe_h)
    s = int(max(1, min(spp, 60.0 / max(per_spp * (args.steps + args.warmup), 1e-6))))
    for _ in range(args.warmup):
        ob.ray_trace(world, cam, W, H, s, depth, rng_mode=ob.RNG_SERIAL, threads=1)
    rays_total, t0 = 0, time.perf_counter()
    for _ in range(args.steps):
        _, rays, _ = ob.ray_trace(world, cam, W, H, s, depth, rng_mode=ob.RNG_SERIAL, threads=1)
        rays_total += rays
    dt = time.perf_counter() - t0
    value = rays_total / dt / 1e6
    ncores = os.cpu_count() or 1
    t = time.perf_counter()
    _, rays_mt, _ = ob.ray_trace(world, cam, W, H, s, depth, rng_mode=ob.RNG_PER_SAMPLE, threads=ncores)
    dt_mt = time.perf_counter() - t
    sample = (f"each step = {W}x{H} full frame at {s} of {spp} spp, depth {depth}, oracle/rt_oracle.c in the "
              f"reference's serial-RNG mode, 1 thread (the reference is single-threaded)")
    line = {"impl": "reference", "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": desc, "sample": f"each step renders {s} of the workload's {spp} spp (full frame, full depth)",
                       "note": "rays/s is independent of spp; frame time scales linearly in spp"},
            "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": 1, "kind": "port", "sample": sample,
                             "all_cores": {"value": rays_mt / dt_mt / 1e6, "cores": ncores,
                                           "note": "oracle per-sample-RNG mode with OpenMP over rows"}},
            "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------- GPU arm

def _events(torch, n):
    return [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]


def time_workload_1gpu(torch, rt, multi, scenes, key, dev, flush, steps, warmup, fast=False, cull=False, fp32_peak=0.0):
    """Device-timed rays/s of one workload on ONE GPU (this rank's), same method as the headline: CUDA events
    on the launching stream around every step, L2 flushed in between.  Used for the `workloads` record of the
    N = 1 line and for the in-run single-GPU base of the N > 1 lines."""
    desc, skey, W, H, spp, depth, passes = WORKLOADS[key]
    handle = rt.load_world(scene_text(scenes, skey))
    r = multi.ShardedRenderer(rt, handle, W, H, 0, 1, tile_rows=16, device=dev)
    st = rt.RenderStats()
    frame, rays = r.render(spp, depth, passes, fast_math=fast, count_rays=True, group_cull=cull, stats=st)
    for _ in range(max(warmup - 1, 0)):
        flush.zero_()
        r.render(spp, depth, passes, fast_math=fast, group_cull=cull)
    torch.cuda.synchronize()
    ev = _events(torch, steps)
    for a, b in ev:
        flush.zero_()
        a.record()
        frame, _ = r.render(spp, depth, passes, fast_math=fast, group_cull=cull)
        b.record()
    torch.cuda.synchronize()
    ms = sum(a.elapsed_time(b) for a, b in ev) / steps
    sha = __import__("hashlib").sha256(frame.cpu().numpy().tobytes()).hexdigest()
    S, T = handle.n_spheres, handle.n_triangles
    flops = algorithmic_flops(rays, W * H * spp, W * H, S, T)
    achieved = flops / (ms * 1e-3) / 1e12
    rec = {"workload": desc, "ms_per_step": ms, "value": rays / (ms * 1e-3) / 1e6, "unit": "Mrays/s", "steps": steps,
           "rays_per_step": int(rays), "launches_per_step": int(st.launches), "passes_fused": int(st.passes_fused),
           "sample_items": int(st.sample_items), "kernel": "fast-math" if fast else "exact",
           "roofline": {"bound": "fp32", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s",
                        "frac": achieved / fp32_peak if fp32_peak else None, "flops_per_step": flops}}
    r.close()
    return rec, sha, int(rays)


def ppm_record(rt, torch, dev):
    """SURVEY.md 8f-3: the step right after the path in the CLI and the example (image.rs:59-81) — writing
    a 3840x2160 frame as ASCII P3 (the reference's format) and as binary P6, to tmpfs when there is one."""
    import tempfile
    W, H = 3840, 2160
    fb = rt.Framebuffer(W, H)
    fb.pixels[...] = (torch.arange(W * H * 4, dtype=torch.int64) * 2654435761 >> 13).to(torch.uint8).numpy().reshape(H, W, 4)
    d = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    out = {}
    for name, binary in (("p3", False), ("p6", True)):
        path = os.path.join(d, f"rt_bench_{os.getpid()}_{name}.ppm")
        best = 1e9
        for _ in range(3):
            t0 = time.perf_counter()
            rt.write_image(fb, path, binary=binary)
            best = min(best, time.perf_counter() - t0)
        size = os.path.getsize(path)
        os.unlink(path)
        out[name] = {"ms": best * 1e3, "bytes": size, "MB_per_s": size / best / 1e6, "Mpixels_per_s": W * H / best / 1e6}
    out["frame"] = f"{W}x{H}"
    out["dir"] = d
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--fast-math", action="store_true", help="relaxed-arithmetic kernel (not bit-exact)")
    ap.add_argument("--spp", type=int, default=None, help="override the workload's spp (profiling only: "
                    "the line then says so in config.workload)")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="N > 1: 'peer' = render kernels store their tiles into rank 0's frame over NVLink "
                         "(CUDA IPC mapping); 'nccl' = compact buffers + one dist.gather")
    ap.add_argument("--no-steal", action="store_true", help="N > 1: static tile deal only (no cross-GPU work stealing)")
    ap.add_argument("--no-row-gather", action="store_true",
                    help="N > 1: every finished pixel is stored straight into rank 0's frame (one 4-byte store over NVLink) "
                         "instead of being rendered into a local frame and copied across as 16-byte vectors by a second kernel")
    ap.add_argument("--devices", type=int, default=0,
                    help="N = 1 launch only: also time render_with_options(n_devices=D), ONE process driving D GPUs "
                         "(the shape the C-ABI callers have); reported under e2e_one_process")
    ap.add_argument("--cull", action="store_true",
                    help="opt-in acceleration mode (RT_OPT_GROUP_CULL): same frame, fewer sphere tests — a separately "
                         "reported mode, NOT the brute-force path the BASELINE metric is defined on")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the extra records (N = 1: workloads c3/c5/c4, ppm; N > 1: single-GPU base + parity, "
                         "one-process C-ABI e2e)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame of the last timed step to DIR as .npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm sizes its spp from a timing probe, so its frame is not reproducible")
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    default_line = args.workload is None and not args.spp and not args.fast_math and not args.cull
    if args.workload is None:
        args.workload = "c2" if max(args.gpus, world_size) == 1 else "c4"
    heavy = args.workload in ("c3", "c4")
    if args.steps is None:
        args.steps = 5 if heavy else 50
    if args.warmup is None:
        args.warmup = 3 if heavy else 5

    if args.impl != "reference":
        args.warmup = max(args.warmup, 3)            # timing rule: at least 3 untimed warm-up steps

    scenes = importlib.import_module("rust-swift-raytracer_b200.scenes")
    if args.impl == "reference":
        return run_reference(args, scenes)

    import hashlib
    import numpy as np
    import torch
    import torch.distributed as dist
    build = importlib.import_module("rust-swift-raytracer_b200.build")
    rt = importlib.import_module("rust-swift-raytracer_b200")
    if not rt.LIB_PATH.exists():
        build.build()
    multi = importlib.import_module("rust-swift-raytracer_b200.multi")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available() or rt.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: the render path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world_size > 1:
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank),
                                timeout=datetime.timedelta(seconds=300))    # a failed rank must not stall the run for long
        # a CPU-side group: while rank 0 measures something alone, the others wait on the HOST — an NCCL barrier
        # would keep a spinning kernel on their GPUs, which rank 0's one-process leg needs for itself
        host_group = dist.new_group(backend="gloo", timeout=datetime.timedelta(seconds=300))
    n_gpus = world_size
    if args.gpus != n_gpus and rank == 0:
        print(f"# note: --gpus {args.gpus} but WORLD_SIZE={world_size}; using {n_gpus}", file=sys.stderr)

    wl = WORKLOADS[args.workload]
    desc, key, W, H, spp, depth, passes = wl
    if args.spp:
        spp, passes = args.spp, 1
        desc += f" [REDUCED to {spp} spp for profiling — not a bench line]"
    handle = rt.load_world(scene_text(scenes, key))
    S, T = handle.n_spheres, handle.n_triangles
    dev = torch.device("cuda", local_rank)
    renderer = multi.ShardedRenderer(rt, handle, W, H, rank, n_gpus, tile_rows=16, device=dev, gather=args.gather,
                                     steal=not args.no_steal, row_gather=not args.no_row_gather)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def barrier():
        if n_gpus > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def host_barrier():
        torch.cuda.synchronize()
        if n_gpus > 1:
            dist.barrier(group=host_group)

    def allreduce(x, op):
        if n_gpus == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    fast = args.fast_math
    # FP32 peak of this box, measured before the timed region (FFMA-chain microbenchmark)
    fp32_peak = rt.measure_fp32_peak(local_rank) if rank == 0 else 0.0

    # ---- warm-up (first step also counts the rays of one frame; the frame is deterministic) ----
    st0 = rt.RenderStats()
    _, rays_local = renderer.render(spp, depth, passes, fast_math=fast, count_rays=True, group_cull=args.cull, stats=st0)
    rays_frame = allreduce(float(rays_local), dist.ReduceOp.SUM if n_gpus > 1 else None)
    stolen_first = allreduce(float(st0.stolen_slots), dist.ReduceOp.SUM if n_gpus > 1 else None)
    launches_all = allreduce(float(st0.launches), dist.ReduceOp.SUM if n_gpus > 1 else None)   # kernels per step, all ranks
    for _ in range(max(args.warmup - 1, 0)):
        flush.zero_()
        renderer.render(spp, depth, passes, fast_math=fast, group_cull=args.cull)
    barrier()

    # ---- timed region: K steps, CUDA events on the launching stream around every step ----
    ev = _events(torch, args.steps)
    with ClockSampler(local_rank) as clocks:
        barrier()
        t_wall = time.perf_counter()
        for a, b in ev:
            flush.zero_()                       # L2 flush, outside the events
            a.record()
            frame_dev, _ = renderer.render(spp, depth, passes, fast_math=fast, group_cull=args.cull)
            b.record()
        barrier()
        t_wall = time.perf_counter() - t_wall
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    dev_ms = allreduce(dev_ms, dist.ReduceOp.MAX if n_gpus > 1 else None)
    ms_per_step = dev_ms / args.steps
    value = rays_frame / (ms_per_step * 1e-3) / 1e6

    # sha256 of the frame of the last timed step (rank 0; N > 1: the gathered frame in rank 0's memory)
    frame_sha = None
    if rank == 0:
        if renderer.gather == "peer" and n_gpus > 1:
            host = torch.empty((H, W), dtype=torch.int32).pin_memory()
            rt.copy_to_host(host.data_ptr(), frame_dev, W * H * 4, torch.cuda.current_stream(dev).cuda_stream)
            torch.cuda.synchronize()
            frame_host = host.numpy()
        else:
            frame_host = frame_dev.cpu().numpy()
        frame_sha = hashlib.sha256(frame_host.tobytes()).hexdigest()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, frame_host.view(np.uint8).reshape(H, W, 4))
    barrier()

    # ---- e2e: HOST framebuffer through the public API, host<->device traffic inside the timed region ----
    def time_calls(fn, steps):
        fn()
        barrier()
        tot = 0.0
        for _ in range(steps):
            flush.zero_()
            barrier()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            tot += allreduce(time.perf_counter() - t0, dist.ReduceOp.MAX if n_gpus > 1 else None)
        return tot / steps

    e2e = e2e_pinned = None
    h2d = 360 + 112                               # RtFrameParams + RtSceneView travel as kernel arguments; the scene
    # blob is uploaded once by load_world (the reference's API has the same split: load_world, then render)
    if not args.no_e2e:
        if n_gpus == 1:
            opts = rt.Options(spp, depth, fast_math=fast, group_cull=args.cull, passes=passes)
            fb_page = rt.Framebuffer(W, H, pinned=False)       # plain malloc'ed pixels: what the reference's callers
            fb_pin = rt.Framebuffer(W, H, pinned=True)         # pass (GameView.swift:125-129, c_raytracer.rs:53)
            t = time_calls(lambda: rt.render_with_options(fb_page, handle, opts), args.steps)
            e2e = {"value": rays_frame / t / 1e6, "unit": "Mrays/s", "ms_per_frame": t * 1e3,
                   "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": W * H * 4,
                   "api": "render_with_options (C ABI), PAGEABLE host framebuffer (np.zeros / malloc): the kernel stores "
                          "its pixels into the library's pinned staging frame over PCIe and flags every finished 16-row tile; "
                          "the calling thread copies flagged tiles into the caller's buffer while the kernel renders the rest"}
            t = time_calls(lambda: rt.render_with_options(fb_pin, handle, opts), args.steps)
            e2e_pinned = {"value": rays_frame / t / 1e6, "unit": "Mrays/s", "ms_per_frame": t * 1e3,
                          "api": "render_with_options (C ABI), pinned framebuffer from rt_alloc_pixels: pixels stored straight "
                                 "into the caller's buffer, no copy at all"}
            assert np.array_equal(fb_page.pixels, fb_pin.pixels)
        else:
            t = time_calls(lambda: renderer.render(spp, depth, passes, fast_math=fast, to_host=True, group_cull=args.cull),
                           args.steps)
            e2e = {"value": rays_frame / t / 1e6, "unit": "Mrays/s", "ms_per_frame": t * 1e3,
                   "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": W * H * 4,
                   "api": f"multi.ShardedRenderer.render(to_host=True): one process per GPU, tile shards -> {renderer.gather} "
                          "gather -> one D2H on rank 0 into pinned host memory"}

    # ---- extras (outside the headline timing) ----
    extras = {}
    if not args.no_extras and default_line:
        if n_gpus == 1:
            wls = {}
            for k, steps_k in (("c3", 3), ("c5", 5), ("c4", 3)):
                rec, _, _ = time_workload_1gpu(torch, rt, multi, scenes, k, dev, flush, steps_k, 3, fp32_peak=fp32_peak)
                wls[k if k != "c4" else "c4_1gpu"] = rec
            extras["workloads"] = wls
            try:
                extras["ppm"] = ppm_record(rt, torch, dev)
            except Exception as e:      # noqa: BLE001
                extras["ppm"] = {"error": repr(e)}
        else:
            # the SAME frame on one GPU, in this run: the base of the strong-scaling figure and the parity check
            host_barrier()
            base = None
            if rank == 0:
                rec, sha1, rays1 = time_workload_1gpu(torch, rt, multi, scenes, args.workload, dev, flush, 2, 3,
                                                      fp32_peak=fp32_peak)
                base = (rec, sha1, rays1)
            host_barrier()
            if rank == 0:
                rec, sha1, rays1 = base
                extras["strong_scaling"] = {"base_ms_1gpu": rec["ms_per_step"], "base_value_1gpu": rec["value"],
                                            "speedup": rec["ms_per_step"] / ms_per_step,
                                            "note": "1-GPU base = the same frame rendered by rank 0 alone in this run "
                                                    "(2 timed steps after 3 warm-ups, same timing method)"}
                extras["parity"] = {"frame_sha256": frame_sha, "single_gpu_sha256": sha1,
                                    "equals_single_gpu": frame_sha == sha1,
                                    "rays": int(rays_frame), "single_gpu_rays": rays1, "rays_equal": int(rays_frame) == rays1}
            # one process driving all N GPUs through the C ABI (what a caller of render_with_options gets)
            if rank == 0:
                try:
                    fbm = rt.Framebuffer(W, H, pinned=False)
                    om = rt.Options(spp, depth, fast_math=fast, n_devices=n_gpus, passes=passes)
                    stm = rt.RenderStats()
                    rt.render_with_options(fbm, handle, om, stm)
                    tot = 0.0
                    for _ in range(3):
                        t0 = time.perf_counter()
                        rt.render_with_options(fbm, handle, om)
                        tot += time.perf_counter() - t0
                    sham = hashlib.sha256(np.ascontiguousarray(fbm.pixels).tobytes()).hexdigest()
                    extras["e2e_one_process"] = {
                        "devices": int(stm.devices), "peer_gather": int(stm.peer_gather), "stolen_slots": int(stm.stolen_slots),
                        "passes_fused": int(stm.passes_fused), "value": rays_frame / (tot / 3) / 1e6, "unit": "Mrays/s",
                        "ms_per_frame": tot / 3 * 1e3, "d2h_bytes_per_step": W * H * 4,
                        "equals_multi_process_frame": sham == frame_sha,
                        "api": "render_with_options(n_devices=N, passes) — C ABI, ONE process drives the N GPUs (peer access), "
                               "pageable host framebuffer"}
                except Exception as e:      # noqa: BLE001
                    extras["e2e_one_process"] = {"error": repr(e)}
            host_barrier()

    one_process = None
    if args.devices > 1 and n_gpus == 1:
        fbm = rt.Framebuffer(W, H, pinned=False)
        om = rt.Options(spp, depth, fast_math=fast, n_devices=args.devices, group_cull=args.cull, passes=passes)
        stm = rt.RenderStats()
        rt.render_with_options(fbm, handle, om, stm)
        tot = 0.0
        for _ in range(args.steps):
            t0 = time.perf_counter()
            rt.render_with_options(fbm, handle, om)
            tot += time.perf_counter() - t0
        one_process = {"devices": int(stm.devices), "peer_gather": int(stm.peer_gather), "stolen_slots": int(stm.stolen_slots),
                       "value": rays_frame / (tot / args.steps) / 1e6, "unit": "Mrays/s",
                       "ms_per_frame": tot / args.steps * 1e3, "d2h_bytes_per_step": W * H * 4,
                       "frame_sha256": hashlib.sha256(np.ascontiguousarray(fbm.pixels).tobytes()).hexdigest(),
                       "api": "render_with_options(n_devices=D): one process, tiles stored into device 0's frame "
                              "over NVLink peer mappings, one D2H"}
    steal_on = bool(renderer.steal)
    row_gather_on = bool(renderer.row_gather) and renderer.gather == "peer"
    gather = renderer.gather
    renderer.close()
    if rank != 0:
        if n_gpus > 1:
            dist.destroy_process_group()
        return 0

    samples = W * H * spp
    flops = algorithmic_flops(rays_frame, samples, W * H, S, T)
    achieved = flops / (ms_per_step * 1e-3) / 1e12
    line = {
        "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": n_gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong" if n_gpus > 1 else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "spheres": S, "triangles": T, "rays_per_step": int(rays_frame),
                   "samples_per_step": samples, "kernel": "fast-math" if fast else "exact (bit-identical to the oracle)",
                   "passes": (f"{passes} progressive passes of {spp // passes} spp fused into one persistent launch "
                              "(float4 sums through HBM between passes)") if passes > 1 else "1",
                   "sphere_walk": ("group-cull (opt-in acceleration: the roofline fraction below still counts the brute-force "
                                   "algorithmic flops, so it is a speed-up measure, not a pipe utilisation)") if args.cull
                                  else "brute force over the list (filtered for >= 64 spheres)",
                   "parallelism": (f"row-tile shards x{n_gpus} (static boustrophedon deal"
                                   + (" + cross-GPU work stealing of the tail over NVLink atomics" if steal_on else "")
                                   + f"), {gather} gather to rank 0 "
                                   + (("(ranks != 0 render into a local frame; a copy kernel on the same stream moves their pixels into rank 0's "
                                       "frame over NVLink as 16-byte vectors, CUDA IPC)") if row_gather_on else
                                      "(fused into the render kernels: every finished pixel is stored into rank 0's frame over NVLink, CUDA IPC)"
                                      if gather == "peer" else "(compact buffers + dist.gather)"))
                   if n_gpus > 1 else "1 GPU",
                   "launch": {"block": int(st0.block), "grid": int(st0.grid), "smem_bytes": int(st0.smem_bytes),
                              "sample_items": bool(st0.sample_items), "paths_per_lane": int(st0.paths_per_lane)},
                   "stolen_slots_first_step": int(stolen_first) if n_gpus > 1 else 0,
                   "l2": "flushed between steps (256 MiB write, outside the CUDA events)",
                   "wall_ms_per_step_incl_flush": t_wall / args.steps * 1e3,
                   "frame_sha256": frame_sha,
                   },
        "e2e": e2e,
        "gpu_launches": args.steps * int(launches_all),     # render kernels (+ the row-gather copy kernel on ranks != 0)
        "roofline": {"bound": "fp32", "achieved": achieved, "peak": fp32_peak * n_gpus, "unit": "TFLOP/s",
                     "frac": achieved / (fp32_peak * n_gpus) if fp32_peak else None,
                     "traffic": NCU_TRAFFIC_BYTES.get((args.workload, fast)) if (n_gpus == 1 and not args.spp) else None,
                     "peak_source": "FFMA-chain microbenchmark run on this GPU before the timed region "
                                    "(MEASURED_PEAKS.json has no FP32 CUDA-core figure; nominal 2*128*148*1.965 GHz = 74.4)",
                     "flops_per_step": flops,
                     "flops_model": "rays*(17*S + 12*T + 60) + samples*34 + pixels*11, FMA = 2 (SURVEY.md 8d)",
                     "hbm_bytes_per_step": W * H * 4 + (passes - 1) * 2 * W * H * 16,
                     "ncu_context": NCU_CONTEXT.get((args.workload, fast)) if n_gpus == 1 else None},
        "clocks": clocks.summary(),
    }
    if e2e_pinned:
        line["e2e_pinned"] = e2e_pinned
    line.update(extras)
    if one_process:
        line["e2e_one_process"] = one_process
    if not args.no_cpu_baseline and n_gpus == 1:
        line["cpu_baseline"] = cpu_baseline_serial(scenes, wl)
    print(json.dumps(line), flush=True)
    if n_gpus > 1:
        dist.destroy_process_group()
    parity = extras.get("parity")
    if parity and not (parity["equals_single_gpu"] and parity["rays_equal"]):
        print("bench.py: PARITY FAILURE — the multi-GPU frame differs from the single-GPU frame", file=sys.stderr)
        return 3
    return 0


if __name__ == "__main__":
    sys.exit(main())
