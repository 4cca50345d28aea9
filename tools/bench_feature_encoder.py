#!/usr/bin/env python
"""Stock torchvision feature encoder vs ``rc.FeatureEncoder.forward_trunk`` as raft_flow runs them: 1088 x 1920 input,
B = 10 (the n + 1 images of a run of 9 P-frames, raft_flow_sequence) and B = 1, fp16 autocast.

    python tools/bench_feature_encoder.py [--out profiles/r03_feature_encoder_bench.json]

Arms, per batch size:
  * stock: what raft_flow's fused encoder tail runs with the stock module -- NCHW, ``fe.layer3(fe.layer2(fe.layer1(
    fe.convnormrelu(x))))``, replayed as one CUDA graph;
  * ours: ``rc.FeatureEncoder.forward_trunk(x)``, also replayed as one CUDA graph.
Timed with CUDA events, the arms alternating, a 256 MB buffer written between timed passes so that no pass starts from
an L2 that holds its inputs or weights.  MACs and algorithmic bytes per layer come from the shapes.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch


def gpu_facts():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                               "-i", "0"], capture_output=True, text=True).stdout.strip()
    except OSError:
        return "unknown"


def layer_table(B, H, W):
    """Per layer (name, MACs, bytes) of the drop-in from the shapes: 16-bit activations, layer2 at a 128-channel stride,
    GEMM MACs as issued (padded K and N included).  Convolution: input read once, raw output (and the downsample's)
    written once, partials written; apply: raw output (+ residual or downsample) read, activation written."""
    H1, W1 = (H + 1) // 2, (W + 1) // 2
    H2, W2 = (H1 + 1) // 2, (W1 + 1) // 2
    H3, W3 = (H2 + 1) // 2, (W2 + 1) // 2
    p1, p2, p3 = B * H1 * W1, B * H2 * W2, B * H3 * W3
    part = lambda p, nt: p / 128 * nt * 8                               # noqa: E731  (mean, M2) per tile and channel
    rows = [("stem pack", 0, B * H * W * 3 * 2 + p1 * 64 * 2),
            ("convnormrelu conv", p1 * 64 * 256, 2 * p1 * 64 * 2 + part(p1, 64)),
            ("convnormrelu apply", 0, 2 * p1 * 64 * 2)]
    for blk in ("layer1.0", "layer1.1"):
        rows += [(blk + ".convnormrelu1 conv", p1 * 64 * 64 * 9, 2 * p1 * 64 * 2 + part(p1, 64)),
                 (blk + ".convnormrelu1 apply", 0, 2 * p1 * 64 * 2),
                 (blk + ".convnormrelu2 conv", p1 * 64 * 64 * 9, 2 * p1 * 64 * 2 + part(p1, 64)),
                 (blk + ".convnormrelu2 apply+res", 0, 3 * p1 * 64 * 2)]
    for name, pin, cin, pout in (("layer2", p1, 64, p2), ("layer3", p2, 128, p3)):
        rows += [(name + ".0.convnormrelu1+downsample conv", pout * 128 * cin * 10,
                  pin * cin * 2 + 2 * pout * 128 * 2 + part(pout, 256)),
                 (name + ".0.convnormrelu1 apply", 0, 2 * pout * 128 * 2),
                 (name + ".0.convnormrelu2 conv", pout * 128 * 128 * 9, 2 * pout * 128 * 2 + part(pout, 128)),
                 (name + ".0.convnormrelu2 apply+downsample", 0, 3 * pout * 128 * 2)]
        rows += [(name + ".1.convnormrelu1 conv", pout * 128 * 128 * 9, 2 * pout * 128 * 2 + part(pout, 128)),
                 (name + ".1.convnormrelu1 apply", 0, 2 * pout * 128 * 2),
                 (name + ".1.convnormrelu2 conv", pout * 128 * 128 * 9, 2 * pout * 128 * 2 + part(pout, 128)),
                 (name + ".1.convnormrelu2 apply+res", 0, 3 * pout * 128 * 2)]
    return [{"layer": n, "gmac": m / 1e9, "mb": b / 1e6} for n, m, b in rows]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--height", type=int, default=1088)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--batches", default="10,1")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_feature_encoder_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a B200: no CUDA device")
    import rdvc_corr_b200 as rc
    from torchvision.models.optical_flow import raft_large

    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    model = raft_large(weights=None).eval().to(dev)
    stock_fe = model.feature_encoder
    fe = rc.FeatureEncoder()
    fe.load_state_dict(stock_fe.state_dict())
    fe = fe.to(dev)
    scratch = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    H, W = args.height, args.width
    results = {}
    for B in (int(b) for b in args.batches.split(",")):
        g = torch.Generator(device=dev).manual_seed(B)
        img = torch.rand(B, 3, H, W, device=dev, generator=g)

        def stock():                                   # raft_flow's fused encoder tail with the stock module (NCHW)
            return stock_fe.layer3(stock_fe.layer2(stock_fe.layer1(stock_fe.convnormrelu(img))))

        def ours():
            return fe.forward_trunk(img)

        graphs, outs = {}, {}
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            for k, fn in (("stock", stock), ("ours", ours)):
                side = torch.cuda.Stream(device=dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(side):
                    for _ in range(3):                 # cuDNN algorithm choice, packing, allocator
                        fn()
                torch.cuda.current_stream(dev).wait_stream(side)
                torch.cuda.synchronize(dev)
                gr = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gr):
                    outs[k] = fn()
                graphs[k] = gr
        times = {k: [] for k in graphs}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for _ in range(args.reps):
            for k, gr in graphs.items():               # alternating
                scratch.fill_(1)
                ev[0].record()
                gr.replay()
                ev[1].record()
                torch.cuda.synchronize(dev)
                times[k].append(ev[0].elapsed_time(ev[1]))
        diff = (outs["stock"].float() - outs["ours"].float()).abs().max().item()
        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
        table = layer_table(B, H, W)
        mb = sum(r["mb"] for r in table)
        results[f"B={B}"] = {
            "ms": med, "spread_ms_min_max": {k: [min(v), max(v)] for k, v in times.items()},
            "speedup": med["stock"] / med["ours"],
            "ours_gmac_issued": sum(r["gmac"] for r in table),
            "ours_algorithmic_mb": mb,
            "ours_gb_per_s": mb / med["ours"],
            "ours_tflops_issued": 2 * sum(r["gmac"] for r in table) / med["ours"],
            "layers": table,
            "max_abs_diff_vs_stock": diff,
            "max_abs_stock": outs["stock"].float().abs().max().item(),
        }
    line = {
        "metric": "feature_encoder_trunk_ms", "unit": "ms", "gpu": gpu_facts(),
        "workload": f"{H}x{W} input, fp16 autocast; the feature encoder up to layer3 (raft_flow's fused encoder tail "
                    "runs the final 1x1 inside the correlation build); default raft_large weights",
        "timing": f"CUDA graph per arm, CUDA events, median of {args.reps} alternating passes, 256 MB written between "
                  "passes (L2 flushed)",
        "results": results,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(line) + "\n")
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
