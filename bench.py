#!/usr/bin/env python
"""bench.py -- RAFT correlation hot path: build + 12-iteration lookup, frame pairs/s at 1920x1088.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--volume-dtype fp32|bf16]
                    [--dump-outputs DIR]

One "step" = one synthetic frame pair (BASELINE.json configs[1]): correlation volume + 4-level
pyramid from two (1, 256, 136, 240) feature maps, then 12 radius-4 lookups with drifting
coordinates.  Prints ONE JSON line (rank 0).  See DESIGN.md section "Measurement".

  value        pairs/s, inputs resident in HBM, CUDA events on the launching stream, max over ranks
  e2e          pairs/s through the C-ABI host entry points rdvc_corr_pair_host_submit / _wait (two pairs in
               flight): pinned HOST feature maps + coords in, all 12 lookup tensors of every pair back to HOST,
               copies inside the timed region
  e2e_f16_out  the same with fp16 results (rdvc_corr_pair_host_submit_ex): half the bytes back over PCIe -- what the
               reference's default consumer casts the features to anyway (autocast, R:codec_processing.py:1436)
  roofline     the build kernel alone: algorithmic bytes / its CUDA-event duration vs measured HBM peak
  cpu_baseline the reference's implementation (torchvision CorrBlock, CPU fp32) on this box's cores, one FULL pair
  gpu_library_baseline   stock torchvision CorrBlock on the SAME B200 (fp32 and fp16 autocast): the library-call bar
  gop_sharded  BASELINE.json configs 3 / 4 at this N: P-frames/s of the 600-frame synthetic 1080p sequence (GOP 10)
               through the motion branch's RAFT call, sharded over the ranks (bench_gop.run_sharded), + at N = 1 the
               CPU comparator (stock RAFT.forward on the host cores for one P-frame)

--impl reference times the reference's own CPU implementation as its own arm (rank 0 only): every step is one FULL
1920x1088 pair through torchvision's CorrBlock.build_pyramid + 12 x index_pyramid, warm-up included.
No number here is taken under a profiler.

--dump-outputs DIR (ours, rank 0) writes what the timed loop computed in its last step, as float32 .npy files, so that
two builds can be compared output for output (the inputs are seeded, identical from run to run):
  lookup.npy            the last of the step's 12 lookups, (1, 324, 136, 240), in full
  pyramid_level<l>.npy  the pyramid rows of DUMP_ROWS query pixels drawn with a fixed seed, (DUMP_ROWS, 1, h_l, w_l)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "raft_corr_build_plus_12iter_lookup_frame_pairs_per_s_1080p"
UNIT = "pairs/s"
B, D, H8, W8 = 1, 256, 136, 240          # 1920x1088 frames -> 1/8-resolution feature maps
LEVELS, RADIUS, ITERS = 4, 4, 12
N = H8 * W8
RING = 4                                   # distinct input sets rotated through (268 MB > 126 MB L2)
WORKLOAD = ("1 frame pair 1920x1088 per step per GPU: corr volume + 4-level pyramid + 12 radius-4 lookups "
            "(BASELINE.json configs[1])")
DUMP_ROWS = 64                             # --dump-outputs: 42.3 MB of lookup + 11.1 MB of pyramid rows


# ----------------------------------------------------------------------------- workload maths
def algorithmic_bytes(vol_bytes: int):
    """SURVEY.md 8(d): bytes one frame pair must move."""
    pyr_elems = sum((H8 >> l) * (W8 >> l) for l in range(LEVELS)) * N * B
    build = 2 * B * N * D * 2 + vol_bytes * pyr_elems
    side = 2 * RADIUS + 2
    lookup = B * N * (LEVELS * side * side * vol_bytes + 2 * 4 + LEVELS * (2 * RADIUS + 1) ** 2 * 4)
    return build, lookup


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(vol: str):
    """dram bytes read+write of the build kernel from the committed ncu capture (or None)."""
    for name in ("r02_build_kernel_ncu.json", "r01_build_kernel_ncu.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                d = json.load(f)
            v = d.get(vol, {}).get("dram_bytes_read_plus_write")
            if v is not None:
                return v
        except Exception:
            continue
    return None


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    NAMES = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) == 6:
                self.samples.append(parts)

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        sm = [int(s[0]) for s in self.samples if s[0].isdigit()]
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        reasons = sorted({n for s in self.samples for n, v in zip(self.NAMES, s[2:]) if v == "Active"})
        return {"sm_mhz": (statistics.median(sm) if sm else None), "sm_max_mhz": (max(mx) if mx else None),
                "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------- reference arm
def reference_inputs():
    """The synthetic pair of BASELINE.json configs[1] on the host: seed-0 randn feature maps, 12 drifting coordinate fields."""
    import torch
    from oracle import corr_numpy as cn
    g = torch.Generator().manual_seed(0)
    f1 = torch.randn(B, D, H8, W8, generator=g)
    f2 = torch.randn(B, D, H8, W8, generator=g)
    base = torch.from_numpy(cn.make_coords_grid(B, H8, W8))
    g1 = torch.Generator().manual_seed(1)
    coords = []
    c = base.clone()
    for _ in range(ITERS):
        c = c + 0.5 * torch.randn(c.shape, generator=g1)
        coords.append(c.clone())
    return f1, f2, coords


REFERENCE_SAMPLE = (f"1 full frame pair 1920x1088 per step through the stock torchvision CorrBlock "
                    f"(build_pyramid + {ITERS} x index_pyramid), CPU fp32, all host threads")


def reference_pair_seconds(steps: int, warmup: int):
    """torchvision CorrBlock (what RDVC's encoder executes, R:codec_processing.py:1442) on the host cores, fp32:
    EVERY step -- warm-up steps included -- is one full 1920x1088 pair through the stock class, nothing sliced,
    restated or extrapolated.  Returns (mean seconds per pair over the timed steps, sample description, threads)."""
    import torch
    from oracle import tv_corr as tv
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    f1, f2, coords = reference_inputs()
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        with torch.no_grad():
            tv.build_and_lookup(f1, f2, coords, LEVELS, RADIUS)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return sum(times) / len(times), REFERENCE_SAMPLE, cores


def gpu_library_pair_ms(dev, reps: int = 3):
    """Stock torchvision CorrBlock on the SAME GPU (SURVEY.md 8d, BASELINE.md 4: the "library-call" comparator and
    what RDVC executes today, R:codec_processing.py:1442): build_pyramid + 12 x index_pyramid on one 1920x1088 pair,
    fp32 and under fp16 autocast (the reference's GPU default, R:codec_processing.py:1436).  Median of `reps`
    after one warm-up, CUDA events."""
    import torch
    from oracle import tv_corr as tv
    f1, f2, coords = (x.to(dev) if hasattr(x, "to") else [c.to(dev) for c in x] for x in reference_inputs())
    out = {}
    for name, amp in (("fp32", False), ("autocast_fp16", True)):
        ms = []
        for i in range(reps + 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            e0.record()
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=amp):
                a, b_ = (f1.half(), f2.half()) if amp else (f1, f2)      # the feature encoder emits fp16 under autocast
                tv.build_and_lookup(a, b_, coords, LEVELS, RADIUS)
            e1.record()
            torch.cuda.synchronize(dev)
            if i > 0:
                ms.append(e0.elapsed_time(e1))
        out[name] = {"ms_per_pair": statistics.median(ms), "value": 1e3 / statistics.median(ms), "unit": UNIT}
        torch.cuda.empty_cache()
    out["note"] = "stock torchvision CorrBlock.build_pyramid + 12 x index_pyramid on this GPU, median of %d after 1 warm-up" % reps
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    sec, sample, cores = reference_pair_seconds(args.steps, args.warmup)
    v = 1.0 / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "fmap": [B, D, H8, W8], "iters": ITERS, "volume_dtype": "fp32",
                   "host": "cpu: stock torchvision CorrBlock, every step one full pair"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


# ----------------------------------------------------------------------------- our arm
def dump_outputs(out_dir: str, pyr, lookup):
    """Write the last step's lookup and a fixed sample of its pyramid (see --dump-outputs) as float32 .npy."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    rows = torch.randperm(B * N, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    arrays = {"lookup": lookup}
    for l in range(LEVELS):
        arrays[f"pyramid_level{l}"] = pyr.level(l, rows.to(lookup.device))
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def run_ours(args):
    import numpy as np
    import torch
    import rdvc_corr_b200 as rc

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert world == args.gpus or world == 1, f"WORLD_SIZE={world} but --gpus {args.gpus}"
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    lib = rc._cabi.load()  # raises if the CUDA library is missing: no fallback
    vol_dtype = torch.float32 if args.volume_dtype == "fp32" else torch.bfloat16
    vol_bytes = 4 if vol_dtype == torch.float32 else 2
    dev = torch.device("cuda", local_rank)

    # synthetic inputs: RING distinct feature-map pairs, 12 drifting coordinate fields per pair
    g = torch.Generator(device=dev).manual_seed(1000 * rank)
    fmaps = [(torch.randn(B, D, H8, W8, device=dev, generator=g), torch.randn(B, D, H8, W8, device=dev, generator=g))
             for _ in range(RING)]
    ys, xs = torch.meshgrid(torch.arange(H8, device=dev), torch.arange(W8, device=dev), indexing="ij")
    base = torch.stack([xs, ys], dim=0).float()[None].repeat(B, 1, 1, 1)   # TV:_utils.py:22-26
    g1 = torch.Generator(device=dev).manual_seed(1)
    coords = []
    c = base.clone()
    for _ in range(ITERS):
        c = c + 0.5 * torch.randn(c.shape, device=dev, generator=g1)
        coords.append(c.clone())

    blk = rc.TVCorrBlock(num_levels=LEVELS, radius=RADIUS, volume_dtype=vol_dtype)
    out = torch.empty((B, LEVELS * (2 * RADIUS + 1) ** 2, H8, W8), dtype=torch.float32, device=dev)

    def step(i, ev=None):
        f1, f2 = fmaps[i % RING]
        if ev is not None:
            lib.rdvc_corr_set_profile_events(ev[0].cuda_event, ev[1].cuda_event)
        blk.build_pyramid(f1, f2)
        for k in range(ITERS):
            rc.index_pyramid(blk._pyr, coords[k], RADIUS, out=out)
        if ev is not None:
            ev[2].record()          # end of the 12 lookups (same stream)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    # kernel-level events for the roofline: one pair per timed step around the build kernel
    kev = [tuple(torch.cuda.Event(enable_timing=True) for _ in range(3)) for _ in range(args.steps)]
    for evs in kev:   # force creation of the underlying cudaEvent_t handles
        for e_ in evs:
            e_.record()
    barrier()

    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = lib.rdvc_corr_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        step(args.warmup + i, kev[i])
    e1.record()
    barrier()
    lib.rdvc_corr_set_profile_events(None, None)
    ms_total = e0.elapsed_time(e1)
    launches = lib.rdvc_corr_launch_count() - launches0
    build_ms = [a.elapsed_time(b_) for a, b_, _ in kev]
    lookup_ms = [b_.elapsed_time(c_) for _, b_, c_ in kev]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, blk._pyr, out)

    # ---- the same timed loop with the other pyramid storage type (reported beside the headline: the
    # reference's own GPU default is an fp16 volume under autocast, R:codec_processing.py:1436)
    alt = None
    if not args.no_alt:
        alt_dtype = torch.bfloat16 if vol_dtype == torch.float32 else torch.float32
        blk.release()
        torch.cuda.empty_cache()
        blk_alt = rc.TVCorrBlock(num_levels=LEVELS, radius=RADIUS, volume_dtype=alt_dtype)

        def step_alt(i):
            f1, f2 = fmaps[i % RING]
            blk_alt.build_pyramid(f1, f2)
            for k in range(ITERS):
                rc.index_pyramid(blk_alt._pyr, coords[k], RADIUS, out=out)

        for i in range(args.warmup):
            step_alt(i)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a0.record()
        for i in range(args.steps):
            step_alt(args.warmup + i)
        a1.record()
        barrier()
        alt = (alt_dtype, a0.elapsed_time(a1))
        blk_alt.release()

    # ---- end to end through the C ABI with host buffers (pinned), copies inside the timed region.
    # Two slots of rdvc_corr_pair_host_submit / _wait: pair i+1's host->device copies and kernels run while
    # pair i's 508 MB of results are still crossing PCIe (every pair is copied in and out in full).
    h_f = [(f1.cpu().pin_memory(), f2.cpu().pin_memory()) for f1, f2 in fmaps[:2]]
    h_co = torch.stack([c_.cpu() for c_ in coords]).contiguous().pin_memory()
    h_out = [torch.empty((ITERS, B, LEVELS * (2 * RADIUS + 1) ** 2, H8, W8), dtype=torch.float32).pin_memory()
             for _ in range(2)]
    blk.release()
    torch.cuda.empty_cache()
    vd = rc.RDVC_DT_F32 if vol_dtype == torch.float32 else rc.RDVC_DT_BF16

    def e2e_submit(i):
        f1, f2 = h_f[i % 2]
        rc_ = lib.rdvc_corr_pair_host_submit(f1.data_ptr(), f2.data_ptr(), h_co.data_ptr(), h_out[i % 2].data_ptr(),
                                             B, D, H8, W8, LEVELS, RADIUS, ITERS, vd, i % 2)
        rc._cabi.check(rc_, "rdvc_corr_pair_host_submit")

    def e2e_wait(i):
        rc._cabi.check(lib.rdvc_corr_pair_host_wait(i % 2), "rdvc_corr_pair_host_wait")

    def e2e_run(n):
        e2e_submit(0)
        for i in range(1, n):
            e2e_submit(i)          # next pair in flight ...
            e2e_wait(i - 1)        # ... while the previous one's results land
        e2e_wait(n - 1)

    e2e_run(max(2, min(args.warmup, 3)))
    barrier()
    t0 = time.perf_counter()
    e2e_run(args.steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    # the same with fp16 results: half the bytes back (the reference's consumer runs under autocast)
    del h_out
    h_out16 = [torch.empty((ITERS, B, LEVELS * (2 * RADIUS + 1) ** 2, H8, W8), dtype=torch.float16).pin_memory()
               for _ in range(2)]

    def e2e16_submit(i):
        f1, f2 = h_f[i % 2]
        rc_ = lib.rdvc_corr_pair_host_submit_ex(f1.data_ptr(), f2.data_ptr(), h_co.data_ptr(), h_out16[i % 2].data_ptr(),
                                                B, D, H8, W8, LEVELS, RADIUS, ITERS, vd, rc.RDVC_DT_F16, i % 2)
        rc._cabi.check(rc_, "rdvc_corr_pair_host_submit_ex")

    def e2e16_run(n):
        e2e16_submit(0)
        for i in range(1, n):
            e2e16_submit(i)
            e2e_wait(i - 1)
        e2e_wait(n - 1)

    e2e16_run(2)
    barrier()
    t0 = time.perf_counter()
    e2e16_run(args.steps)
    barrier()
    e2e16_s = time.perf_counter() - t0
    clocks = sampler.stop()
    del h_out16
    h2d = 2 * B * D * N * 4 + ITERS * B * 2 * N * 4
    d2h = ITERS * B * LEVELS * (2 * RADIUS + 1) ** 2 * N * 4

    # ---- max over ranks
    alt_ms = alt[1] if alt is not None else 0.0
    if dist is not None:
        t = torch.tensor([ms_total, e2e_s, alt_ms, e2e16_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, e2e_s, alt_ms, e2e16_s = t[0].item(), t[1].item(), t[2].item(), t[3].item()
    value = world * args.steps / (ms_total / 1e3)
    e2e_value = world * args.steps / e2e_s
    lib.rdvc_corr_release()
    torch.cuda.empty_cache()

    # ---- BASELINE.json configs 3 / 4 at this N: the 600-frame GOP-sharded motion branch (every rank takes part)
    gop_line = None
    if not args.no_gop:
        import bench_gop
        # fp16 autocast like the reference's GPU default (R:codec_processing.py:1436, "AMP on" in R:jockey.txt:9)
        gop_line = bench_gop.run_sharded(bench_gop.sharded_args(frames=args.gop_frames, amp=not args.gop_fp32),
                                         own_process_group=False)
        torch.cuda.empty_cache()

    line = None
    if rank == 0:
        bytes_build, bytes_lookup = algorithmic_bytes(vol_bytes)
        peak, peak_src = measured_peaks()
        kms = statistics.mean(build_ms)
        achieved = bytes_build / (kms * 1e-3) / 1e9
        roof_pair_s = (bytes_build + ITERS * bytes_lookup) / (peak * 1e9)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {
                "workload": WORKLOAD,
                "fmap": [B, D, H8, W8], "volume_dtype": args.volume_dtype, "operands": "bf16, fp32 accumulate",
                "iters": ITERS, "sharding": "independent frame pairs per GPU, no collective",
                "l2": f"inputs rotate over {RING} fmap sets (268 MB) and the 5.7 GB pyramid is rewritten every step: working set >> 126 MB L2",
            },
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "rdvc_corr_pair_host_submit / _wait, 2 slots (C ABI, pinned host buffers, all 12 fp32 lookup tensors "
                           "of every pair copied back; consecutive pairs overlap)",
                    "bound": "PCIe device->host: %.0f MB of results per pair" % (d2h / 1e6),
                    "d2h_gb_per_s": e2e_value / world * d2h / 1e9},
            "e2e_f16_out": {"value": world * args.steps / e2e16_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
                            "d2h_bytes_per_step": d2h // 2,
                            "api": "rdvc_corr_pair_host_submit_ex(out_dtype = F16) / _wait: the same call with fp16 results "
                                   "(what the reference's autocast consumer casts the features to); not the headline"},
            "gpu_launches": int(launches) * world,
            "roofline": {
                "bound": "hbm", "kernel": "corr_build_kernel (MODE_LINEAR)", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic(args.volume_dtype),
                "algorithmic_bytes_per_launch": bytes_build, "kernel_ms": kms, "peak_source": peak_src,
                "whole_step_frac_of_roofline": (roof_pair_s * 1e3) / (ms_total / args.steps),
                "secondary": {
                    "kernel": "corr_lookup_tiled_kernel x %d" % ITERS, "us_per_launch": 1e3 * statistics.mean(lookup_ms) / ITERS,
                    "algorithmic_bytes_per_launch": bytes_lookup,
                    "achieved": bytes_lookup / (statistics.mean(lookup_ms) / ITERS * 1e-3) / 1e9,
                    "frac": bytes_lookup / (statistics.mean(lookup_ms) / ITERS * 1e-3) / 1e9 / peak,
                    "note": "steady-state DRAM traffic per launch is ~145 MB (64-byte atoms + the 42 MB result), see DESIGN.md 3.3",
                },
            },
        }
        if alt is not None:
            ab = 2 if alt[0] == torch.bfloat16 else 4
            bb, bl = algorithmic_bytes(ab)
            line["alt_volume_dtype"] = {
                "volume_dtype": "bf16" if ab == 2 else "fp32", "value": world * args.steps / (alt_ms / 1e3), "unit": UNIT,
                "ms_per_step": alt_ms / args.steps,
                "whole_step_frac_of_roofline": ((bb + ITERS * bl) / (peak * 1e9) * 1e3) / (alt_ms / args.steps),
                "note": "same timed loop, other pyramid storage type; not the headline",
            }
        if gop_line is not None:
            line["gop_sharded"] = {k: gop_line[k] for k in ("metric", "value", "unit", "n_gpus", "scaling", "p_frames",
                                                             "seconds_total_max_over_ranks", "seconds_encode_max_over_ranks",
                                                             "rank0_p_frames_per_s", "epe_vs_stock_px",
                                                             "stream_bytes", "total_pframe_payload_bytes", "config")}
        if world == 1 and not args.no_gpu_baseline:
            line["gpu_library_baseline"] = gpu_library_pair_ms(dev)
        if world == 1 and not args.no_cpu_baseline:
            sec, sample, cores = reference_pair_seconds(steps=1, warmup=1)
            line["cpu_baseline"] = {"value": 1.0 / sec, "unit": UNIT, "cores": cores, "kind": "reference",
                                    "sample": sample + " (1 warm-up pair, 1 timed pair)"}
            if gop_line is not None:
                import bench_gop
                sec_p, cores_p = bench_gop.cpu_raft_pframe_seconds(1088, 1920, 1)
                line["gop_sharded"]["cpu_baseline"] = {
                    "value": 1.0 / sec_p, "unit": "P-frames/s", "cores": cores_p, "kind": "reference",
                    "sample": "1 P-frame 1920x1088: stock torchvision raft_large forward (its own CorrBlock), 12 updates, "
                              "fp32, all host threads"}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--volume-dtype", choices=["fp32", "bf16"], default="fp32")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-alt", action="store_true", help="skip the extra timed loop with the other volume dtype")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the stock-torchvision-on-this-GPU comparator")
    ap.add_argument("--no-gop", action="store_true", help="skip the GOP-sharded motion-branch run (configs 3 / 4)")
    ap.add_argument("--gop-frames", type=int, default=600, help="frames of the GOP-sharded run (config 4: 600)")
    ap.add_argument("--gop-fp32", action="store_true", help="run the GOP-sharded RAFT in fp32 / TF32 instead of fp16 autocast")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's lookup and a fixed sample of its pyramid to DIR as .npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the CUDA path: use it with --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3   # timing rule: at least 3 warm-up steps
    return run_reference(args) if args.impl == "reference" else run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
