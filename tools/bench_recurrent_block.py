#!/usr/bin/env python
"""Stock torchvision RecurrentBlock vs rc.RecurrentBlock on what raft_flow runs per refinement iteration at 1080p:
B = 9 P-frames, 136 x 240 pixels at 1/8 resolution, fp16 autocast, channels_last tensors and weights.

    python tools/bench_recurrent_block.py [--out profiles/r03_recurrent_block_bench.json]

Both arms get the inputs raft_flow hands them: hidden state and context fp16 (B, 128, h, w), motion features fp32
(B, 128, h, w) (the cat with the fp32 flow promotes them).  The stock arm concatenates them first, as
``_update_block_fused`` does for the stock block; ours takes the parts.  Timed with CUDA events, the arms alternating,
a 256 MB buffer written between timed passes so that no pass starts from an L2 that holds its inputs or weights.
Also timed: one whole stock update step (``model.update_block``: motion encoder + recurrent block + flow head) on the
same tensors, which gives the stock GRU's measured share of an update step.  FLOP counts come from the shapes.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch

FLOP_PER_PIXEL = 2 * (2 * 1920 * 256 + 2 * 1920 * 128)      # two ConvGRUs: z|r (N = 256) + q (N = 128), K = 5 x 384


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=9)
    ap.add_argument("--height", type=int, default=136)
    ap.add_argument("--width", type=int, default=240)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_recurrent_block_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a B200: no CUDA device")
    import rdvc_corr_b200 as rc
    from torchvision.models.optical_flow import raft_large

    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    model = raft_large(weights=None).eval().to(dev)
    ub = model.update_block.to(memory_format=torch.channels_last)
    stock = ub.recurrent_block
    ours = rc.RecurrentBlock(input_size=256, hidden_size=128)
    ours.load_state_dict(stock.state_dict())
    ours = ours.to(dev).to(memory_format=torch.channels_last)

    B, h, w = args.batch, args.height, args.width
    cl = torch.channels_last
    g = torch.Generator(device=dev).manual_seed(1)
    hid = torch.tanh(torch.randn(B, 128, h, w, device=dev, generator=g)).half().contiguous(memory_format=cl)
    ctx = torch.relu(torch.randn(B, 128, h, w, device=dev, generator=g)).half().contiguous(memory_format=cl)
    mot = torch.relu(torch.randn(B, 128, h, w, device=dev, generator=g)).contiguous(memory_format=cl)
    corr = torch.rand(B, 324, h, w, device=dev, generator=g).contiguous(memory_format=cl)
    flow = torch.randn(B, 2, h, w, device=dev, generator=g).contiguous(memory_format=cl)
    scratch = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def run_stock():
        return stock(hid, torch.cat([ctx, mot], dim=1))

    def run_ours():
        return ours.forward_parts(hid, ctx, mot)

    def run_step():
        return ub(hid, ctx, corr, flow)

    arms = {"stock": run_stock, "ours": run_ours, "stock_update_step": run_step}
    times = {k: [] for k in arms}
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
        for fn in arms.values():                     # warm-up: cuDNN algorithm choice, packing, allocator
            for _ in range(3):
                fn()
        out_s, out_o = run_stock(), run_ours()
        max_diff = (out_s.float() - out_o.float()).abs().max().item()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for _ in range(args.reps):
            for k, fn in arms.items():               # alternating
                scratch.fill_(1)
                ev[0].record()
                fn()
                ev[1].record()
                torch.cuda.synchronize()
                times[k].append(ev[0].elapsed_time(ev[1]))
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    spread = {k: [min(v), max(v)] for k, v in times.items()}
    flop = FLOP_PER_PIXEL * B * h * w
    name = torch.cuda.get_device_name(dev)
    try:
        import subprocess
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True).stdout.strip()
    except OSError:
        power = "unknown"
    iters_per_pframe = 12 / B
    line = {
        "metric": "recurrent_block_ms_per_iteration", "unit": "ms",
        "device": name, "power_limit": power,
        "workload": f"B={B}, {h}x{w} at 1/8 resolution (1080p input), fp16 autocast, channels_last; "
                    "hidden/context fp16, motion features fp32 as raft_flow passes them",
        "timing": f"CUDA events, median of {args.reps} alternating passes per arm, 256 MB written between passes (L2 flushed)",
        "stock_ms": med["stock"], "ours_ms": med["ours"], "speedup": med["stock"] / med["ours"],
        "stock_update_step_ms": med["stock_update_step"],
        "stock_gru_share_of_update_step": med["stock"] / med["stock_update_step"],
        "stock_gru_ms_per_pframe": med["stock"] * iters_per_pframe, "ours_ms_per_pframe": med["ours"] * iters_per_pframe,
        "flop_per_call": flop, "stock_tflops": flop / med["stock"] / 1e9, "ours_tflops": flop / med["ours"] / 1e9,
        "spread_ms_min_max": spread, "max_abs_diff_vs_stock": max_diff,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(line) + "\n")
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
