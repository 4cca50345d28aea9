#!/usr/bin/env python
"""Stock torchvision update block vs this library's drop-ins on what raft_flow runs per refinement iteration at 1080p:
B = 9 P-frames, 136 x 240 pixels at 1/8 resolution, fp16 autocast, channels_last tensors and weights.

    python tools/bench_update_block.py [--out profiles/r03_update_block_bench.json]

Arms, each timed per iteration:
  * motion encoder after convcorr1: stock (convcorr2, convflow1, convflow2, conv and the two cats, as
    ``_update_block_fused`` runs them) vs ``rc.MotionEncoder.forward_fused`` on convcorr1's NHWC 16-bit output;
  * flow head: stock ``FlowHead`` vs ``rc.FlowHead`` on the fp16 channels_last hidden state;
  * the whole update step after the fused lookup + 1x1: stock motion encoder tail + cat + stock GRU + stock flow head
    vs the three drop-ins (motion features handed to ``RecurrentBlock.forward_parts`` in place).
Both arms start from the same fp16 channels_last convcorr1 output, made once outside the timed window (under autocast
the fused lookup + 1x1 returns fp16 either way; the stock arm then pays one transpose per iteration that is not timed
here).  Timed with CUDA
events, the arms alternating, a 256 MB buffer written between timed passes so that no pass starts from an L2 that holds
its inputs or weights.  MAC counts come from the shapes.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch

# multiply-accumulates per pixel at 1/8 resolution (raft_large)
MAC_ME = 9 * 256 * 192 + 49 * 2 * 128 + 9 * 128 * 64 + 9 * 256 * 126      # convcorr2, convflow1, convflow2, conv
MAC_FH = 9 * 128 * 256 + 9 * 256 * 2
MAC_GRU = 2 * (5 * 384 * 256 + 5 * 384 * 128)


def power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True).stdout.strip()
    except OSError:
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=9)
    ap.add_argument("--height", type=int, default=136)
    ap.add_argument("--width", type=int, default=240)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_update_block_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a B200: no CUDA device")
    import rdvc_corr_b200 as rc
    from torchvision.models.optical_flow import raft_large

    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    model = raft_large(weights=None).eval().to(dev)
    ub = model.update_block.to(memory_format=torch.channels_last)
    sme, sfh, srb = ub.motion_encoder, ub.flow_head, ub.recurrent_block
    me = rc.MotionEncoder(in_channels_corr=324)
    me.load_state_dict(sme.state_dict())
    fh = rc.FlowHead(in_channels=128, hidden_size=256)
    fh.load_state_dict(sfh.state_dict())
    rb = rc.RecurrentBlock(input_size=256, hidden_size=128)
    rb.load_state_dict(srb.state_dict())
    me, fh, rb = me.to(dev).eval(), fh.to(dev).eval(), rb.to(dev).eval()

    B, h, w = args.batch, args.height, args.width
    cl = torch.channels_last
    g = torch.Generator(device=dev).manual_seed(1)
    hid = torch.tanh(torch.randn(B, 128, h, w, device=dev, generator=g)).half().contiguous(memory_format=cl)
    ctx = torch.relu(torch.randn(B, 128, h, w, device=dev, generator=g)).half().contiguous(memory_format=cl)
    flow = (4 * torch.randn(B, 2, h, w, device=dev, generator=g)).contiguous(memory_format=cl)
    c1_stock = torch.relu(torch.randn(B, 256, h, w, device=dev, generator=g)).half().contiguous(memory_format=cl)
    c1_ours = c1_stock.clone(memory_format=cl)                    # the NHWC 16-bit output of the fused 1x1
    scratch = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def stock_me():                                               # raft_flow's stock motion encoder after convcorr1
        corr = sme.convcorr2(c1_stock)
        f = sme.convflow2(sme.convflow1(flow))
        return torch.cat([sme.conv(torch.cat([corr, f], dim=1)), flow], dim=1)

    def ours_me():
        return me.forward_fused(flow, c1_ours)

    def stock_fh():
        return sfh(hid)

    def ours_fh():
        return fh(hid)

    def stock_step():
        mf = stock_me()
        hs = srb(hid, torch.cat([ctx, mf], dim=1))
        return hs, sfh(hs)

    def ours_step():
        hs = rb.forward_parts(hid, ctx, ours_me())
        return hs, fh(hs)

    arms = {"stock_me": stock_me, "ours_me": ours_me, "stock_fh": stock_fh, "ours_fh": ours_fh,
            "stock_step": stock_step, "ours_step": ours_step}
    times = {k: [] for k in arms}
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
        for fn in arms.values():                     # warm-up: cuDNN algorithm choice, packing, allocator
            for _ in range(3):
                fn()
        diff = {
            "motion_features": (stock_me().float() - ours_me().float()).abs().max().item(),
            "delta_flow": (stock_fh().float() - ours_fh().float()).abs().max().item(),
            "step_delta_flow": (stock_step()[1].float() - ours_step()[1].float()).abs().max().item(),
        }
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
    px = B * h * w
    line = {
        "metric": "update_block_ms_per_iteration", "unit": "ms",
        "device": torch.cuda.get_device_name(dev), "power_limit": power_limit(),
        "workload": f"B={B}, {h}x{w} at 1/8 resolution (1080p input), fp16 autocast, channels_last; the step starts "
                    "from convcorr1's output, fp16 channels_last, for both arms",
        "timing": f"CUDA events, median of {args.reps} alternating passes per arm, 256 MB written between passes (L2 flushed)",
        "ms": med, "spread_ms_min_max": spread,
        "speedup": {"motion_encoder": med["stock_me"] / med["ours_me"], "flow_head": med["stock_fh"] / med["ours_fh"],
                    "update_step": med["stock_step"] / med["ours_step"]},
        "ms_per_pframe_12_iters": {k: v * 12 / B for k, v in med.items()},
        "tflops": {"stock_me": 2 * MAC_ME * px / med["stock_me"] / 1e9, "ours_me": 2 * MAC_ME * px / med["ours_me"] / 1e9,
                   "stock_fh": 2 * MAC_FH * px / med["stock_fh"] / 1e9, "ours_fh": 2 * MAC_FH * px / med["ours_fh"] / 1e9,
                   "stock_step": 2 * (MAC_ME + MAC_FH + MAC_GRU) * px / med["stock_step"] / 1e9,
                   "ours_step": 2 * (MAC_ME + MAC_FH + MAC_GRU) * px / med["ours_step"] / 1e9},
        "max_abs_diff_vs_stock": diff,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(line) + "\n")
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
