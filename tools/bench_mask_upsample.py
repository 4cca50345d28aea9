#!/usr/bin/env python
"""Stock torchvision mask predictor + upsample_flow vs ``rc.MaskPredictor.upsample_flow`` as raft_flow runs them after
the last refinement iteration: 136 x 240 pixels at 1/8 resolution (1080p input), B = 9 P-frames and B = 1, fp16
autocast, channels_last hidden state and weights.

    python tools/bench_mask_upsample.py [--out profiles/r03_mask_upsample_bench.json]

Arms, per batch size:
  * stock: ``mask_predictor(hidden_state).contiguous()`` then torchvision's ``upsample_flow`` (softmax, unfold, product,
    sum, permute + reshape), exactly the code of ``raft_flow``'s stock path;
  * ours: ``rc.MaskPredictor.upsample_flow(flow, hidden_state)`` -- convrelu on the tcgen05 3x3 kernel, then the 1x1
    GEMM with the softmax, the convex combination and the pixel shuffle in its epilogue.
Timed with CUDA events, the arms alternating, a 256 MB buffer written between timed passes so that no pass starts from
an L2 that holds its inputs or weights.  MACs and algorithmic bytes come from the shapes.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch

MAC_CONVRELU = 9 * 128 * 256          # per pixel at 1/8 resolution
MAC_MASK = 256 * 576


def power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True).stdout.strip()
    except OSError:
        return "unknown"


def algorithmic_bytes(B, h, w):
    """Bytes each arm has to move at least, from the shapes (fp16 activations, fp32 flow and output; weights once)."""
    px = B * h * w
    hidden, inter, flow, out = px * 128 * 2, px * 256 * 2, px * 2 * 4, px * 64 * 2 * 4
    weights = (9 * 128 * 256 + 256 * 576) * 2
    mask16, mask32, prod = px * 576 * 2, px * 576 * 4, px * 2 * 576 * 4
    return {
        # convrelu (read h, write + read the intermediate), then the fused GEMM (read the flow, write the output)
        "ours": hidden + 2 * inter + flow + out + weights,
        # the same, plus: the mask written and read (fp16), softmax writes / reads it in fp32, the (B, 2, 9, 8, 8, h, w)
        # product written and read by the sum, the sum's result written and copied by permute().reshape()
        "stock": hidden + 2 * inter + flow + weights + 2 * mask16 + 2 * mask32 + 2 * prod + 3 * out,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--height", type=int, default=136)
    ap.add_argument("--width", type=int, default=240)
    ap.add_argument("--batches", default="9,1")
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_mask_upsample_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a B200: no CUDA device")
    import rdvc_corr_b200 as rc
    from torchvision.models.optical_flow import raft_large
    from torchvision.models.optical_flow._utils import upsample_flow

    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    model = raft_large(weights=None).eval().to(dev)
    smp = model.mask_predictor.to(memory_format=torch.channels_last)
    mp = rc.MaskPredictor(in_channels=128, hidden_size=256, multiplier=smp.multiplier)
    mp.load_state_dict(smp.state_dict())
    mp = mp.to(dev).eval()
    scratch = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    h, w = args.height, args.width
    results = {}
    for B in (int(b) for b in args.batches.split(",")):
        g = torch.Generator(device=dev).manual_seed(B)
        hid = torch.tanh(torch.randn(B, 128, h, w, device=dev, generator=g)).half().contiguous(
            memory_format=torch.channels_last)
        flow = 4 * torch.randn(B, 2, h, w, device=dev, generator=g)

        def stock():                                   # raft_flow's stock path
            up_mask = smp(hid).contiguous()
            return upsample_flow(flow=flow.contiguous(), up_mask=up_mask)

        def ours():
            return mp.upsample_flow(flow, hid)

        arms = {"stock": stock, "ours": ours}
        times = {k: [] for k in arms}
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            for fn in arms.values():                   # warm-up: cuDNN algorithm choice, packing, allocator
                for _ in range(3):
                    fn()
            F = (8 * flow).abs().max().item()
            diff = (stock().float() - ours()).abs().max().item()
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            for _ in range(args.reps):
                for k, fn in arms.items():             # alternating
                    scratch.fill_(1)
                    ev[0].record()
                    fn()
                    ev[1].record()
                    torch.cuda.synchronize()
                    times[k].append(ev[0].elapsed_time(ev[1]))
        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
        px = B * h * w
        nbytes = algorithmic_bytes(B, h, w)
        results[f"B={B}"] = {
            "ms": med, "spread_ms_min_max": {k: [min(v), max(v)] for k, v in times.items()},
            "speedup": med["stock"] / med["ours"],
            "gmac": {"convrelu": MAC_CONVRELU * px / 1e9, "mask_conv": MAC_MASK * px / 1e9},
            "tflops": {k: 2 * (MAC_CONVRELU + MAC_MASK) * px / v / 1e9 for k, v in med.items()},
            "algorithmic_bytes": nbytes,
            "algorithmic_gb_per_s": {k: nbytes[k] / v / 1e6 for k, v in med.items()},
            "max_abs_diff_vs_stock_over_F": diff / F,
        }
    line = {
        "metric": "mask_predictor_upsample_ms", "unit": "ms",
        "device": torch.cuda.get_device_name(dev), "power_limit": power_limit(),
        "workload": f"{h}x{w} at 1/8 resolution (1080p input), fp16 autocast, channels_last hidden state and weights; "
                    "one mask predictor + upsampling pass (raft_flow runs one per call)",
        "timing": f"CUDA events, median of {args.reps} alternating passes per arm, 256 MB written between passes "
                  "(L2 flushed)",
        "results": results,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(line) + "\n")
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
