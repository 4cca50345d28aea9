#!/usr/bin/env python
"""bench_gop.py -- BASELINE.json configs 3 and 4 ("next" rows): P-frames/s of the motion branch's RAFT
call on synthetic 1080p GOPs (I-frame every 10 -> 9 P-frames).

    python bench_gop.py                                  # config 3: one GOP, 1 GPU, vs stock torchvision
    torchrun --nproc-per-node N bench_gop.py --frames 600   # config 4: GOP-sharded over N GPUs

Config 4 shards whole GOPs over the ranks (gop_shard.assign_gops), every rank runs RAFT with the B200
correlation block on its own P-frames, and rank 0 gathers the per-GOP frame records into one `.rdvc`
stream on the host -- no collective on the data path.  The codec networks and the entropy coder are
out of scope (SURVEY.md 8f-4): the P payload carries a quantised 1/8-resolution flow as a stand-in for
the motion bitstream, the I payload a small thumbnail, so the container, the frame indices and the
gather are exercised for real while the byte counts mean nothing.

Not the driver's bench (that is bench.py).  Compares, on the same B200 and the same seeded
random-init raft_large (no weights offline):
  stock   torchvision RAFT.forward with its own CorrBlock (what RDVC runs today)
  ours    rc.raft_flow with TVCorrBlock (B200 correlation block, final-only upsampling)
and reports the end-point error between the two.  Frames are a smooth random texture translated
by a known per-frame motion, generated at RAFT's input size 1088x1920, values in [0,1] like
R:codec_processing.py:751-759.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch
import torch.nn.functional as F


def make_gop(n, h, w, device, seed=0):
    g = torch.Generator(device=device).manual_seed(seed)
    base = torch.rand(1, 3, h // 16 + 8, w // 16 + 8, device=device, generator=g)
    big = F.interpolate(base, size=(h + 64, w + 64), mode="bicubic", align_corners=False).clamp(0, 1)
    frames = []
    for t in range(n):
        dx, dy = 3 * t, 2 * t          # known global motion: (3, 2) px per frame
        frames.append(big[:, :, 32 - dy:32 - dy + h, 32 - dx:32 - dx + w].contiguous())
    return frames


def timed(fn, n_warm=1):
    for _ in range(n_warm):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def frame_at(big, t, h, w):
    """Frame t of the synthetic sequence: the texture translated by (3, 2) px per frame, wrapped every 10."""
    k = t % 10
    dx, dy = 3 * k, 2 * k
    return big[:, :, 32 - dy:32 - dy + h, 32 - dx:32 - dx + w].contiguous()


def raft_kw(args):
    """The rc.raft_flow / rc.GraphedRaftFlow switches the command line controls."""
    return dict(fuse_convcorr1=args.fuse_convcorr1, update_block_channels_last=getattr(args, "update_channels_last", True))


def sharded_args(**kw):
    """The argument namespace of run_sharded with its command-line defaults (for callers such as bench.py)."""
    d = dict(frames=600, height=1088, width=1920, gop=10, amp=False, graph=True, volume="fp32", from_uint8=False,
             mcn=False, batch_gop=True, shard="frames", fuse_convcorr1=True, entropy=True, share_features=True, overlap_host=True,
             update_channels_last=True)
    d.update(kw)
    return argparse.Namespace(**d)


def run_sharded(args, own_process_group=True):
    """BASELINE.json config 4: `--frames` frames in GOPs of `--gop`, sharded over the ranks -- by whole GOPs
    (`--shard gops`, the north star's unit: 60 GOPs / 8 ranks caps at 7.5x) or by frame spans (`--shard frames`,
    the default: the encoder is open loop, so every rank takes a contiguous span with the same number of P-frames,
    540 / 8 -> 67 or 68: 7.94x).  Either way the `.rdvc` stream is byte-identical to the 1-rank encode.
    Returns the JSON line (a dict) on rank 0, None elsewhere.  With own_process_group=False the caller has
    already initialised torch.distributed (NCCL) and keeps it."""
    import torch.distributed as dist
    import rdvc_corr_b200 as rc
    from torchvision.models.optical_flow import raft_large
    gs, fmt = rc.gop_shard, rc.rdvc_format
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    host_group = None
    if world > 1:
        if own_process_group:
            dist.init_process_group("nccl", device_id=dev)
        host_group = dist.new_group(backend="gloo")      # byte strings travel over the host
    torch.manual_seed(0)
    vol = torch.float32 if args.volume == "fp32" else torch.bfloat16
    model = raft_large(weights=None, corr_block=rc.TVCorrBlock(volume_dtype=vol)).eval().to(dev)
    if getattr(args, "b200_recurrent_block", False):      # same weights, the SepConvGRU as this library's kernels
        rb = rc.RecurrentBlock(input_size=256, hidden_size=model.update_block.recurrent_block.hidden_size)
        rb.load_state_dict(model.update_block.recurrent_block.state_dict())
        model.update_block.recurrent_block = rb.to(dev)
    if getattr(args, "b200_update_block", False):         # same weights, all three update-block submodules as this library's
        ub = model.update_block
        me, fh = rc.MotionEncoder(in_channels_corr=324), rc.FlowHead(in_channels=128, hidden_size=256)
        me.load_state_dict(ub.motion_encoder.state_dict())
        fh.load_state_dict(ub.flow_head.state_dict())
        rb = rc.RecurrentBlock(input_size=256, hidden_size=ub.recurrent_block.hidden_size)
        rb.load_state_dict(ub.recurrent_block.state_dict())
        ub.motion_encoder, ub.recurrent_block, ub.flow_head = me.to(dev), rb.to(dev), fh.to(dev)
    if getattr(args, "b200_mask_predictor", False):       # same weights, mask + convex upsampling as one fused GEMM
        mp = rc.MaskPredictor(in_channels=128, hidden_size=256, multiplier=model.mask_predictor.multiplier)
        mp.load_state_dict(model.mask_predictor.state_dict())
        model.mask_predictor = mp.to(dev)
    if getattr(args, "b200_context_encoder", False):      # same weights and BatchNorm statistics, folded into tcgen05 convolutions
        ce = rc.ContextEncoder()
        ce.load_state_dict(model.context_encoder.state_dict())
        model.context_encoder = ce.to(dev).eval()
    if getattr(args, "b200_feature_encoder", False):      # same weights, InstanceNorm statistics in tcgen05 epilogues
        fe = rc.FeatureEncoder()
        fe.load_state_dict(model.feature_encoder.state_dict())
        model.feature_encoder = fe.to(dev).eval()
    h, w = args.height, args.width
    g = torch.Generator(device=dev).manual_seed(0)
    base = torch.rand(1, 3, h // 16 + 8, w // 16 + 8, device=dev, generator=g)
    big = F.interpolate(base, size=(h + 64, w + 64), mode="bicubic", align_corners=False).clamp(0, 1)
    host_frames = None
    if args.from_uint8:      # the ten distinct frames of the synthetic sequence as uint8 HWC host arrays, 8 rows shorter
        fh_ = h - 8 if h % 16 == 0 and h > 64 else h
        host_frames = [torch.from_numpy((frame_at(big, t, h, w)[0, :, :fh_].permute(1, 2, 0) * 255).round().to(torch.uint8).cpu().numpy()).pin_memory()
                       for t in range(10)]
    gops = gs.split_gops(args.frames, args.gop)
    mine = gs.assign_gops(gops, world)[rank]
    spans = gs.assign_frames(args.frames, args.gop, world)
    by_frames = (args.shard == "frames")
    share = bool(getattr(args, "share_features", True)) and args.batch_gop     # runs of consecutive frames: each frame's features once
    overlap = bool(getattr(args, "overlap_host", True)) and args.batch_gop and by_frames   # entropy-code batch k while batch k + 1 runs
    ctx = lambda: torch.autocast("cuda", dtype=torch.float16, enabled=args.amp)

    def enc_i(frame):
        thumb = (F.avg_pool2d(frame, 64) * 255).round().to(torch.uint8).cpu().numpy().tobytes()
        return fmt.iframe_payload(thumb, ".raw")

    fh = args.height - 8 if args.height % 16 == 0 and args.height > 64 else args.height   # 1088 -> 1080 codec frame

    runner = (rc.GraphedRaftFlow(model, 12, amp_dtype=torch.float16 if args.amp else None, volume_dtype=vol,
                                 **raft_kw(args)) if args.graph else None)
    coder = rc.entropy_coder.FlowCoder() if args.entropy else None

    mcn_net = None
    if args.mcn:     # step 5b of the reference (R:codec_processing.py:1458); seeded weights, non-trivial BatchNorm statistics
        mcn_net = rc.MotionCompensationNetwork()
        gm = torch.Generator().manual_seed(1)
        for m in mcn_net.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.copy_(torch.randn(m.num_features, generator=gm) * 0.3)
                m.running_var.copy_(torch.rand(m.num_features, generator=gm) * 1.5 + 0.25)
        mcn_net = mcn_net.eval().to(dev)

    def predict(warped, flow, prev_codec, cur_codec):
        """Motion-compensated prediction and the mean |residual| the residual codec would see."""
        if mcn_net is None:
            return None
        with torch.no_grad():
            pred = mcn_net(warped, flow, prev_codec)
        return (cur_codec - pred).abs().mean(dim=(1, 2, 3))

    def enc_p(prev, cur):
        if runner is not None:
            flow = runner(prev, cur)
        else:
            with torch.no_grad(), ctx():
                flow = rc.raft_flow(model, prev, cur, 12, **raft_kw(args))
        # steps 3 + 5a of the reference (R:codec_processing.py:1446,1456): flow to frame resolution and the
        # warped previous frame, one fused launch; the MCN / residual / codecs that consume them are out of scope
        prev_codec = prev[:, :, :fh].contiguous()
        warped, flow = rc.motion_warp(prev_codec, flow, (fh, w))
        res = predict(warped, flow, prev_codec, cur[:, :, :fh])
        small = F.avg_pool2d(flow.float(), 8)
        q = motion_bytes((small * 4).round().clamp(-127, 127).to(torch.int8).cpu().numpy())[0]
        rbytes = b"" if res is None else res.cpu().numpy().astype("<f4").tobytes()
        return fmt.pframe_payload(tuple(small.shape[-2:]), q, (0, 0) if res is None else (1, 1), rbytes)

    def motion_bytes(q_int8):
        """(n, 2, h/8, w/8) int8 quantised flow -> one motion bitstream per frame.  With --entropy (default) through
        the factorised-prior range coder stand-in (rc.entropy_coder; the reference's EntropyBottleneck.compress is
        compressai's, absent here: bitstream parity unpinned) so the byte counts follow the symbol statistics;
        otherwise the raw int8 dump."""
        if coder is None:
            return [q_int8[i].tobytes() for i in range(q_int8.shape[0])]
        return [coder.compress(q_int8[i]) for i in range(q_int8.shape[0])]

    def get_frame(t):
        """Frame t as the encoder loop sees it: a (RAFT input, codec input) pair of device tensors."""
        if host_frames is None:
            f = frame_at(big, t, h, w)
            return f
        u8 = host_frames[t % 10]
        return rc.preprocess_frame_raft(u8, (h, w), dev)      # R:codec_processing.py:1430-1431

    def enc_p_batch(prevs, curs):
        prevs, curs = list(prevs), list(curs)
        if share and all(prevs[i + 1] is curs[i] for i in range(len(curs) - 1)):
            # a run of consecutive frames (gop_shard hands over the same objects on both sides): the feature encoder
            # sees each frame once (rc.raft_flow_sequence)
            frames = torch.cat(prevs + [curs[-1]], 0)
            a, b = frames[:-1], frames[1:]
            if runner is not None:
                flow = runner.sequence(frames)
            else:
                with torch.no_grad(), ctx():
                    flow = rc.raft_flow_sequence(model, frames, 12, **raft_kw(args))
        else:
            a, b = torch.cat(prevs, 0), torch.cat(curs, 0)
            if runner is not None:
                flow = runner(a, b)
            else:
                with torch.no_grad(), ctx():
                    flow = rc.raft_flow(model, a, b, 12, **raft_kw(args))
        a_codec = a[:, :, :fh].contiguous()
        warped, flow = rc.motion_warp(a_codec, flow, (fh, w))
        res = predict(warped, flow, a_codec, b[:, :, :fh])
        small = F.avg_pool2d(flow.float(), 8)
        q_dev = (small * 4).round().clamp(-127, 127).to(torch.int8)
        shape = tuple(small.shape[-2:])
        if not overlap:
            q = motion_bytes(q_dev.cpu().numpy())
            rb = None if res is None else res.cpu().numpy().astype("<f4")
            return [fmt.pframe_payload(shape, q[i], (0, 0) if rb is None else (1, 1),
                                       b"" if rb is None else rb[i].tobytes()) for i in range(len(q))]
        # device -> pinned host copies on the stream, an event behind them; the entropy coding (host C) happens in the
        # returned callable, which gop_shard.encode_span calls AFTER it has submitted the next batch
        q_host = torch.empty(q_dev.shape, dtype=torch.int8, pin_memory=True)
        q_host.copy_(q_dev, non_blocking=True)
        r_host = None
        if res is not None:
            r_host = torch.empty(res.shape, dtype=torch.float32, pin_memory=True)
            r_host.copy_(res.float(), non_blocking=True)
        done = torch.cuda.Event()
        done.record()

        def finish():
            done.synchronize()
            q = motion_bytes(q_host.numpy())
            rb = None if r_host is None else r_host.numpy().astype("<f4")
            return [fmt.pframe_payload(shape, q[i], (0, 0) if rb is None else (1, 1),
                                       b"" if rb is None else rb[i].tobytes()) for i in range(len(q))]
        return finish

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    batch = max(1, min(args.gop, args.frames) - 1)        # P-frames per RAFT batch: a GOP's worth
    if args.batch_gop:                                    # warm-up at the batched shape(s) (and graph capture)
        if by_frames:                                     # the batch sizes this rank's span will produce
            ts_p = [t for t in spans[rank] if not gs.is_iframe(t, args.gop)]
            shapes = {len(c) for c in gs.pframe_batches(ts_p, batch, share)}
        else:
            shapes = {batch}
        for npf in sorted(shapes, reverse=True):
            for _ in range(2):
                fr = [frame_at(big, t, h, w) for t in range(npf + 1)]
                out = enc_p_batch(fr[:-1], fr[1:])
                if callable(out):
                    out()
    if runner is not None:                                # warm-up: capture the graph outside the timed region
        for _ in range(2):
            runner(frame_at(big, 0, h, w), frame_at(big, 1, h, w))
    with torch.no_grad(), ctx():                          # warm-up: cuDNN autotune + allocator
        for _ in range(2):
            rc.raft_flow(model, frame_at(big, 0, h, w), frame_at(big, 1, h, w), 12, **raft_kw(args))
    barrier()
    t0 = time.perf_counter()
    meta_in = {"rdvc_version": "b200-bench", "iframe_interval": args.gop}
    if by_frames:
        data, tail_failed = gs.encode_span(spans[rank], args.gop, get_frame, enc_i, enc_p,
                                           enc_p_batch if args.batch_gop else None, batch=batch,
                                           consecutive_runs=share)
        torch.cuda.synchronize()
        t_local = time.perf_counter() - t0
        stream = gs.gather_spans(data, tail_failed, spans, meta_in, rank, world, host_group,
                                 reencode_iframe=lambda t: enc_i(get_frame(t)), as_parts=True)   # ready for the writer
    else:
        if args.batch_gop:
            local = {gp.index: gs.encode_gop_batched(gp, get_frame, enc_i, enc_p_batch, enc_p) for gp in mine}
        else:
            local = {gp.index: gs.encode_gop(gp, get_frame, enc_i, enc_p) for gp in mine}
        torch.cuda.synchronize()
        t_local = time.perf_counter() - t0
        stream = gs.gather_stream(local, len(gops), meta_in, rank, world, host_group)
    barrier()
    t_all = time.perf_counter() - t0
    times = torch.tensor([t_all, t_local], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    line = None
    if rank == 0:
        if isinstance(stream, fmt.StreamParts):          # what a writer would f.write() piece by piece; joined here only
            stream = stream.tobytes()                    # for the checks below, outside the timed region
        meta, recs = fmt.read_stream(stream)
        n_p = sum(1 for r in recs if r.kind == "P")
        assert [r.index for r in recs] == list(range(args.frames)), "frame records out of order"
        assert n_p == sum(gp.num_pframes for gp in gops)
        assert all(len(fmt.parse_pframe_payload(r.payload)[1]) > 0 for r in recs if r.kind == "P"), "a P-frame failed"
        line = {
            "metric": "gop_sharded_raft_motion_branch_p_frames_per_s_1080p", "value": n_p / times[0].item(),
            "unit": "P-frames/s", "n_gpus": world, "scaling": "strong",
            "config": {"workload": f"{args.frames} synthetic frames {w}x{h}, GOP {args.gop}, 12 RAFT updates, "
                                   "seed-0 random-init raft_large, B200 correlation block, final-only upsampling",
                       "amp_fp16": args.amp, "cuda_graph": args.graph, "batched_gop": args.batch_gop, "volume_dtype": args.volume, "frames_from_host_uint8": args.from_uint8,
                       "motion_compensation_network": args.mcn, "lookup_fused_with_convcorr1": args.fuse_convcorr1,
                       "sharding": ("frame spans (contiguous, P-frames balanced to one)" if by_frames else "whole GOPs (LPT)"),
                       "gops": len(gops), "gops_per_rank_max": max(len(x) for x in gs.assign_gops(gops, world)),
                       "pframes_per_rank_max": (max(sum(1 for t in sp if not gs.is_iframe(t, args.gop)) for sp in spans)
                                                if by_frames else max(sum(g_.num_pframes for g_ in x) for x in gs.assign_gops(gops, world))),
                       "payload": ("motion: 1/8-resolution quantised flow through the factorised-prior range coder stand-in "
                                   "(bitstream parity unpinned: compressai absent); codec networks out of scope" if args.entropy
                                   else "placeholder int8 dump (codec networks out of scope)"),
                       "feature_encoder_tail_fused": True,
                       "feature_maps_shared_by_consecutive_pairs": share,
                       "cudnn_benchmark": bool(torch.backends.cudnn.benchmark),
                       "host_entropy_coding_overlaps_next_batch": overlap,
                       "update_block_channels_last": bool(getattr(args, "update_channels_last", True)) and args.fuse_convcorr1,
                       "collective": "none on the data path; host-side gather of per-rank byte strings into the writer "
                                     "(/dev/shm files on one node, gloo tensors otherwise)"},
            "seconds_total_max_over_ranks": times[0].item(), "seconds_encode_max_over_ranks": times[1].item(),
            "p_frames": n_p, "stream_bytes": len(stream), "total_frames_processed": meta["total_frames_processed"],
            # "one rank's rate": rank 0's own P-frames over its own encode time, inside this run
            "rank0_p_frames_per_s": (sum(1 for t in spans[0] if not gs.is_iframe(t, args.gop)) if by_frames
                                     else sum(g_.num_pframes for g_ in mine)) / max(t_local, 1e-9),
        }
        if getattr(args, "b200_recurrent_block", False):
            line["config"]["b200_recurrent_block"] = True
        if getattr(args, "b200_update_block", False):
            line["config"]["b200_update_block"] = True
        if getattr(args, "b200_mask_predictor", False):
            line["config"]["b200_mask_predictor"] = True
        if getattr(args, "b200_context_encoder", False):
            line["config"]["b200_context_encoder"] = True
        if getattr(args, "b200_feature_encoder", False):
            line["config"]["b200_feature_encoder"] = True
        # flow end-point error of this configuration against STOCK torchvision RAFT (same weights, same autocast
        # setting) on one frame pair of the sequence -- outside the timed region
        a, b = frame_at(big, 3, h, w), frame_at(big, 4, h, w)
        with torch.no_grad(), ctx():
            if share:       # the pair as the middle of a run, the way the timed region computed it
                run = torch.cat([frame_at(big, 2, h, w), a, b, frame_at(big, 5, h, w)], 0)
                ours_flow = rc.raft_flow_sequence(model, run, 12, **raft_kw(args))[1:2]
            else:
                ours_flow = rc.raft_flow(model, a, b, 12, **raft_kw(args))
        model.corr_block.release()
        torch.manual_seed(0)
        stock = raft_large(weights=None).eval().to(dev)
        with torch.no_grad(), ctx():
            stock_flow = stock(a, b, num_flow_updates=12)[-1]
        line["epe_vs_stock_px"] = (ours_flow.float() - stock_flow.float()).pow(2).sum(1).sqrt().mean().item()
        del stock, stock_flow, ours_flow
        line["total_pframe_payload_bytes"] = meta["total_pframe_payload_bytes"]
    if runner is not None:
        runner.release()
    model.corr_block.release()
    if world > 1:
        dist.barrier()
        if own_process_group:
            dist.destroy_process_group()
    return line


def cpu_raft_pframe_seconds(height=1088, width=1920, frames=1):
    """CPU comparator for configs 3 / 4 (SURVEY.md 8d): the reference's motion-branch RAFT call -- stock torchvision
    raft_large (seed 0, its own CorrBlock), 12 updates, fp32 -- on the host cores for `frames` P-frames."""
    from torchvision.models.optical_flow import raft_large
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    model = raft_large(weights=None).eval()
    g = torch.Generator().manual_seed(0)
    base = torch.rand(1, 3, height // 16 + 8, width // 16 + 8, generator=g)
    big = F.interpolate(base, size=(height + 64, width + 64), mode="bicubic", align_corners=False).clamp(0, 1)
    t0 = time.perf_counter()
    with torch.no_grad():
        for t in range(frames):
            model(frame_at(big, t, height, width), frame_at(big, t + 1, height, width), num_flow_updates=12)
    return (time.perf_counter() - t0) / frames, cores


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=0, help="> 0: GOP-sharded run over all ranks (config 4)")
    ap.add_argument("--height", type=int, default=1088)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--gop", type=int, default=10)
    ap.add_argument("--stock-pframes", type=int, default=2, help="stock RAFT is slow at 1080p: time only this many")
    ap.add_argument("--amp", action="store_true", help="fp16 autocast like the reference's GPU default")
    ap.add_argument("--graph", action="store_true", help="replay rc.raft_flow as one CUDA graph (rc.GraphedRaftFlow)")
    ap.add_argument("--volume", choices=["fp32", "bf16"], default="fp32", help="storage type of the correlation pyramid")
    ap.add_argument("--from-uint8", action="store_true",
                    help="config 4: frames start as uint8 HWC host arrays (1080 rows) and go through "
                         "rc.preprocess_frame_raft / _codec, like the reference's loop (R:codec_processing.py:1430-1450)")
    ap.add_argument("--mcn", action="store_true",
                    help="also run the motion-compensation network on every P-frame (rc.MotionCompensationNetwork, "
                         "R:codec_processing.py:1458) with seeded random weights")
    ap.add_argument("--batch-gop", action="store_true",
                    help="run all P-frames of a GOP through RAFT as one batch (the encoder is open loop)")
    ap.add_argument("--shard", choices=["gops", "frames"], default="frames",
                    help="config 4: partition by whole GOPs or by contiguous frame spans (P-frames balanced to one)")
    ap.add_argument("--no-fuse-convcorr1", dest="fuse_convcorr1", action="store_false",
                    help="keep the stock convcorr1 module after an fp32 lookup instead of the fused lookup + 1x1 GEMM")
    ap.add_argument("--no-share-features", dest="share_features", action="store_false",
                    help="run the feature encoder on both frames of every pair (2n images per batch) instead of once per "
                         "frame of a run of consecutive frames (n + 1 images, rc.raft_flow_sequence)")
    ap.add_argument("--no-update-channels-last", dest="update_channels_last", action="store_false",
                    help="feed the stock update block NCHW tensors like RAFT.forward does (cuDNN then transposes around every convolution)")
    ap.add_argument("--no-overlap-host", dest="overlap_host", action="store_false",
                    help="entropy-code a batch's flows right after its device work instead of while the next batch runs")
    ap.add_argument("--cudnn-benchmark", action="store_true",
                    help="torch.backends.cudnn.benchmark = True for the stock convolutions (ours and the stock comparator alike)")
    ap.add_argument("--no-entropy", dest="entropy", action="store_false",
                    help="config 4: raw int8 motion payload instead of the range coder stand-in")
    ap.add_argument("--cpu-baseline", action="store_true", help="also time stock RAFT on the host cores for 1 P-frame")
    ap.add_argument("--b200-recurrent-block", action="store_true",
                    help="config 4: swap rc.RecurrentBlock (the SepConvGRU as fused tcgen05 convolutions) into the model")
    ap.add_argument("--b200-update-block", action="store_true",
                    help="swap rc.MotionEncoder, rc.RecurrentBlock and rc.FlowHead (the whole update block as this "
                         "library's kernels) into the model")
    ap.add_argument("--b200-mask-predictor", action="store_true",
                    help="swap rc.MaskPredictor into the model: the mask, its softmax and the convex 8x upsampling as "
                         "one fused GEMM")
    ap.add_argument("--b200-context-encoder", action="store_true",
                    help="swap rc.ContextEncoder into the model: the context encoder with BatchNorm folded into tcgen05 "
                         "convolutions, RAFT's tanh / relu in its last epilogue")
    ap.add_argument("--b200-feature-encoder", action="store_true",
                    help="swap rc.FeatureEncoder into the model: the feature encoder as tcgen05 convolutions whose "
                         "epilogues write InstanceNorm statistics, one normalising pass per layer")
    args = ap.parse_args()
    if args.cudnn_benchmark:
        torch.backends.cudnn.benchmark = True
    if args.frames > 0:
        line = run_sharded(args)
        if line is not None:
            if args.cpu_baseline:
                sec, cores = cpu_raft_pframe_seconds(args.height, args.width, 1)
                line["cpu_baseline"] = {"value": 1.0 / sec, "unit": "P-frames/s", "cores": cores, "kind": "reference",
                                        "sample": "1 P-frame: stock torchvision raft_large forward, 12 updates, fp32, host cores"}
            print(json.dumps(line), flush=True)
        return
    import rdvc_corr_b200 as rc
    from torchvision.models.optical_flow import raft_large
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    stock = raft_large(weights=None).eval().to(dev)
    torch.manual_seed(0)
    ours = raft_large(weights=None, corr_block=rc.TVCorrBlock()).eval().to(dev)
    frames = make_gop(args.gop, args.height, args.width, dev)
    pairs = [(frames[t - 1], frames[t]) for t in range(1, args.gop)]     # open loop: originals

    ctx = lambda: torch.autocast("cuda", dtype=torch.float16, enabled=args.amp)

    runner = (rc.GraphedRaftFlow(ours, 12, amp_dtype=torch.float16 if args.amp else None,
                                 **raft_kw(args)) if args.graph else None)

    def run_ours():
        if args.batch_gop:
            a_, b_ = torch.cat([p_[0] for p_ in pairs], 0), torch.cat([p_[1] for p_ in pairs], 0)
            if runner is not None:
                return list(runner(a_, b_).split(1, 0))
            with torch.no_grad(), ctx():
                return list(rc.raft_flow(ours, a_, b_, 12, **raft_kw(args)).split(1, 0))
        if runner is not None:
            return [runner(a, b) for a, b in pairs]
        with torch.no_grad(), ctx():
            return [rc.raft_flow(ours, a, b, 12, **raft_kw(args)) for a, b in pairs]

    def run_stock():
        with torch.no_grad(), ctx():
            return [stock(a, b, num_flow_updates=12)[-1] for a, b in pairs[:args.stock_pframes]]

    t_ours, f_ours = timed(run_ours)
    t_stock, f_stock = timed(run_stock, n_warm=1)
    epe = torch.stack([(x.float() - y.float()).pow(2).sum(1).sqrt().mean() for x, y in zip(f_ours, f_stock)])
    line = {
        "metric": "raft_motion_branch_p_frames_per_s_1080p", "unit": "P-frames/s", "n_gpus": 1,
        "config": {"workload": f"synthetic GOP of {args.gop} frames {args.width}x{args.height}, 12 RAFT updates, "
                               "seed-0 random-init raft_large", "amp_fp16": args.amp, "cuda_graph": args.graph, "batched_gop": args.batch_gop,
                   "lookup_fused_with_convcorr1": args.fuse_convcorr1},
        "ours": {"value": len(pairs) / t_ours, "ms_per_pframe": 1e3 * t_ours / len(pairs), "pframes": len(pairs)},
        "stock_torchvision_same_gpu": {"value": args.stock_pframes / t_stock,
                                       "ms_per_pframe": 1e3 * t_stock / args.stock_pframes,
                                       "pframes": args.stock_pframes},
        "speedup": (len(pairs) / t_ours) / (args.stock_pframes / t_stock),
        "epe_vs_stock_px": {"mean": epe.mean().item(), "max_over_frames": epe.max().item()},
    }
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
