"""Time the whole RAFT call through the C ABI (rdvc_corr_raft_flow_sequence) against the Python path with all six drop-ins.

    python tools/bench_raft_cabi.py [--out profiles/r03_raft_cabi_bench.json]

Arms, alternated pass by pass in one process, on a run of --frames consecutive frames (the n - 1 flows of an open-loop
GOP span), fp16 autocast / act F16, fp32 volume, 12 iterations, seeded raft_large weights:
  c_eager   rdvc_corr_raft_flow_sequence called eagerly through ctypes;
  c_graph   the same call captured once into a CUDA graph and replayed;
  py_graph  rc.GraphedRaftFlow(model).sequence(frames) with the six drop-ins swapped in.
The outputs of all three are checked to be bit-identical before timing.  Timing: CUDA events, median of --reps passes.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402


def gpu_facts():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                               "-i", "0"], capture_output=True, text=True).stdout.strip()
    except OSError:
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="368x640,1088x1920")
    ap.add_argument("--frames", type=int, default=10)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_raft_cabi_bench.json"))
    args = ap.parse_args()
    import rdvc_corr_b200 as rc
    import test_raft_cabi as t
    lib = rc._cabi.load()
    F16, F32 = rc._cabi.RDVC_DT_F16, rc._cabi.RDVC_DT_F32
    model, _ = t.dropin_model(F32)
    blob = t.device_blob(lib)
    results = {}
    for size in args.sizes.split(","):
        H, W = (int(v) for v in size.split("x"))
        g = torch.Generator(device="cuda").manual_seed(1)
        frames = torch.rand(args.frames, 3, H, W, device="cuda", generator=g)
        n = args.frames
        need = lib.rdvc_corr_raft_workspace_bytes(n, n - 1, H, W, F16, F32)
        ws = torch.empty(need, dtype=torch.uint8, device="cuda")
        out = torch.empty((n - 1, 2, H, W), dtype=torch.float32, device="cuda")
        strides = (ctypes.c_longlong * 4)(*frames.stride())

        def c_call():
            code = lib.rdvc_corr_raft_flow_sequence(frames.data_ptr(), strides, F32, n, H, W, 12, F16, F32, blob.data_ptr(),
                                                    0.25, ws.data_ptr(), need, out.data_ptr(),
                                                    torch.cuda.current_stream().cuda_stream)
            assert code == 0, rc._cabi.last_error()

        c_call()
        torch.cuda.synchronize()
        eager = out.clone()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            c_call()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, eager)
        runner = rc.GraphedRaftFlow(model, 12, amp_dtype=torch.float16)
        assert torch.equal(runner.sequence(frames), eager)
        arms = {"c_eager": c_call, "c_graph": graph.replay, "py_graph": lambda: runner.sequence(frames)}
        times = {k: [] for k in arms}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for _ in range(args.reps):
            for k, fn in arms.items():
                torch.cuda.synchronize()
                ev[0].record()
                fn()
                ev[1].record()
                ev[1].synchronize()
                times[k].append(ev[0].elapsed_time(ev[1]))
        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
        results[size] = {"ms_per_run": med, "ms_per_flow": {k: v / (n - 1) for k, v in med.items()},
                         "spread_ms_min_max": {k: [min(v), max(v)] for k, v in times.items()},
                         "workspace_gb": need / 1e9}
        runner.release()
        del ws, graph
        torch.cuda.empty_cache()
    line = {"metric": "raft_cabi_sequence_ms", "unit": "ms", "gpu": gpu_facts(),
            "workload": f"runs of {args.frames} frames ({args.frames - 1} flows), 12 iterations, fp16 activations "
                        "(autocast for the Python arm), fp32 volume, seeded raft_large weights, random frames",
            "timing": f"CUDA events around one call, median of {args.reps} passes alternating the three arms; "
                      "outputs bit-identical across arms", "results": results}
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(line) + "\n")
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
