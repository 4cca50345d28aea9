"""The motion branch's RAFT call, restated around the B200 correlation block ("next" row f-2).

RDVC calls ``raft_model(img1, img2, num_flow_updates=12)`` and keeps only ``flow_preds[-1]``
(R:codec_processing.py:1442-1444).  ``RAFT.forward`` (TV:raft.py:484-533) nevertheless runs the
mask predictor and the 8x convex upsampling after EVERY update and keeps all 12 full-resolution
flows.  :func:`raft_flow` executes the same modules in the same order but upsamples once, at the
end -- bit-identical final flow, 11 mask-predictor + upsample passes fewer -- and uses the
correlation block's preallocated output so the refinement loop allocates nothing.

With ``fuse_convcorr1=True`` (default) the lookup and the first layer of the motion encoder --
``MotionEncoder.convcorr1`` = 1x1 convolution 324 -> 256 + ReLU, TV:raft.py:185,202 -- run as
``TVCorrBlock.index_pyramid_convcorr1`` ("next" row f-1): the (B, 324, h, w) fp32 lookup tensor is never
written, and the rest of ``MotionEncoder.forward`` / ``UpdateBlock.forward`` (TV:raft.py:200-210, 278-285)
is restated module by module.  The 1x1 convolution then multiplies 16-bit operands with fp32 accumulation
(the stock fp32 path multiplies in TF32 / fp32): flows differ by ~1e-3 px, far inside the 0.05 px budget;
``fuse_convcorr1=False`` keeps the stock modules and is bit-identical to ``RAFT.forward``.

With ``fuse_encoder_tail=True`` (default) the feature encoder's LAST layer -- ``FeatureEncoder.conv`` = 1x1
convolution 128 -> 256, TV:raft.py:139,150 -- is not run by cuDNN either: the 128-channel activations go to
``TVCorrBlock.build_pyramid_from_encoder`` (row f-2, last sub-item), which produces the build's K-major 16-bit operand
rows directly; the (2B, 256, h, w) fp32 feature maps (67 MB at 1080p) are never written or re-read.

:func:`raft_flow_sequence` is the same call for a RUN of n + 1 consecutive frames (the n pairs of an open-loop GOP):
the feature encoder sees each frame once.

All other convolutions stay stock PyTorch/cuDNN; only the correlation block (and those two 1x1s) is this library's --
unless the model's ``update_block.recurrent_block`` has been swapped for :class:`rc.RecurrentBlock`, which the fused
path then hands ``context`` and the motion features as separate parts (no concatenation).  With
:class:`rc.MotionEncoder` swapped in, the fused path has the 1x1 GEMM write convcorr1's output NHWC and the module
reads it in place; :class:`rc.FlowHead` reads the hidden state in place.  With :class:`rc.MaskPredictor` as
``model.mask_predictor`` the mask, its softmax and the convex 8x upsampling run as one GEMM epilogue
(``MaskPredictor.upsample_flow``), in the fused and the unfused path alike.  With :class:`rc.ContextEncoder` as
``model.context_encoder`` the hidden state and context come from ``ContextEncoder.forward_split``: RAFT's tanh and
ReLU run in its last layer's epilogue, and both are channel slices of one NHWC buffer.  With :class:`rc.FeatureEncoder`
as ``model.feature_encoder`` the fused encoder tail reads ``FeatureEncoder.forward_trunk``'s layer3 output, and the
unfused path calls the module itself.

:class:`GraphedRaftFlow` replays the whole call as ONE CUDA graph per input shape.  At the reference's
default RAFT size (368x640, R:codec_processing.py:649-650) a P-frame's ~700 kernel launches cost more
CPU time than their GPU time (9.9 ms per P-frame eager, launch-bound); replayed as a graph the same
kernels run back to back.  Same kernels, same order, same numbers (the test requires bit identity).
"""
from __future__ import annotations

from typing import List, Optional

import torch
import torch.nn.functional as F
from torch import Tensor

from .context_encoder import ContextEncoder
from .corr_block import TVCorrBlock, index_pyramid
from .feature_encoder import FeatureEncoder
from .mask_predictor import MaskPredictor
from .motion_encoder import MotionEncoder
from .recurrent_block import RecurrentBlock


def _coords_grid(batch: int, h: int, w: int, device) -> Tensor:
    """TV:_utils.py:22-26 -- channel 0 = x, channel 1 = y."""
    ys, xs = torch.meshgrid(torch.arange(h, device=device), torch.arange(w, device=device), indexing="ij")
    return torch.stack([xs, ys], dim=0).float()[None].repeat(batch, 1, 1, 1)


@torch.no_grad()
def _update_block_fused(model, blk: TVCorrBlock, hidden_state: Tensor, context: Tensor, coords1: Tensor, flow: Tensor,
                        channels_last: bool = False):
    """``UpdateBlock.forward`` (TV:raft.py:278-285) with ``MotionEncoder.forward`` (TV:raft.py:200-210) inlined and its
    first step -- ``convcorr1(index_pyramid(coords1))`` -- replaced by the fused call.  With ``channels_last`` the
    tensors entering the stock convolutions are NHWC (see ``raft_flow``)."""
    ub = model.update_block
    me = ub.motion_encoder
    conv = me.convcorr1[0]                              # Conv2dNormActivation(324, 256, norm_layer=None, kernel_size=1): [Conv2d, ReLU]
    if isinstance(me, MotionEncoder):       # convcorr1 writes NHWC 16-bit, the rest of the encoder reads it in place
        motion_features = me.forward_fused(flow, blk.index_pyramid_convcorr1(coords1, conv.weight, conv.bias, relu=True,
                                                                             nhwc=True))
    else:
        corr = blk.index_pyramid_convcorr1(coords1, conv.weight, conv.bias, relu=True)
        if channels_last:
            corr = corr.contiguous(memory_format=torch.channels_last)
            flow = flow.contiguous(memory_format=torch.channels_last)
        corr = me.convcorr2(corr)
        flow_orig = flow
        f = me.convflow2(me.convflow1(flow))
        corr_flow = me.conv(torch.cat([corr, f], dim=1))
        motion_features = torch.cat([corr_flow, flow_orig], dim=1)
    if isinstance(ub.recurrent_block, RecurrentBlock):       # reads context and motion features in place
        hidden_state = ub.recurrent_block.forward_parts(hidden_state, context, motion_features)
    else:
        x = torch.cat([context, motion_features], dim=1)
        hidden_state = ub.recurrent_block(hidden_state, x)
    return hidden_state, ub.flow_head(hidden_state)


def _can_fuse_encoder_tail(model) -> bool:
    """The feature encoder must be torchvision's: convnormrelu, layer1..3, then Conv2d(128 -> 256, k = 1)."""
    fe = model.feature_encoder
    conv = getattr(fe, "conv", None)
    return (all(hasattr(fe, n) for n in ("convnormrelu", "layer1", "layer2", "layer3")) and isinstance(conv, torch.nn.Conv2d)
            and conv.kernel_size == (1, 1) and conv.stride == (1, 1) and conv.padding == (0, 0) and conv.groups == 1
            and conv.in_channels == 128 and conv.out_channels == 256)


def _can_fuse_convcorr1(model) -> bool:
    """convcorr1 must be exactly Conv2d(k=1, stride 1, no padding, groups 1) + ReLU with cout a multiple of 32 <= 256."""
    try:
        seq = model.update_block.motion_encoder.convcorr1
        conv, act = seq[0], seq[1]
    except Exception:
        return False
    return (len(seq) == 2 and isinstance(conv, torch.nn.Conv2d) and isinstance(act, torch.nn.ReLU)
            and conv.kernel_size == (1, 1) and conv.stride == (1, 1) and conv.padding == (0, 0) and conv.groups == 1
            and conv.out_channels % 32 == 0 and conv.out_channels <= 256)


@torch.no_grad()
def raft_flow(model, image1: Tensor, image2: Tensor, num_flow_updates: int = 12,
              corr_block: Optional[TVCorrBlock] = None, all_predictions: bool = False,
              fuse_convcorr1: bool = True, fuse_encoder_tail: bool = True, update_block_channels_last: bool = True):
    """Final optical flow (B, 2, H, W) of a torchvision RAFT ``model`` for one frame pair.

    ``corr_block`` defaults to ``model.corr_block``, which must be a :class:`TVCorrBlock`
    (inject it with ``raft_large(corr_block=TVCorrBlock())``).  With ``all_predictions=True`` the
    list of all upsampled flows is returned, exactly like ``RAFT.forward``.
    ``update_block_channels_last`` (with the fused path): the stock update block, mask predictor and context encoder
    get NHWC inputs and have their weights stored NHWC (values unchanged) -- cuDNN then skips its layout transposes.
    """
    if image1.dim() != 4 or image1.shape[-2:] != image2.shape[-2:]:
        raise ValueError(f"input images should have the same shape, instead got {tuple(image1.shape[-2:])} != {tuple(image2.shape[-2:])}")
    batch = image1.shape[0]
    return _raft_flow_impl(model, torch.cat([image1, image2], dim=0), lambda x: (x[:batch], x[batch:]), image1,
                           num_flow_updates, corr_block, all_predictions, fuse_convcorr1, fuse_encoder_tail,
                           update_block_channels_last)


@torch.no_grad()
def raft_flow_sequence(model, frames: Tensor, num_flow_updates: int = 12, corr_block: Optional[TVCorrBlock] = None,
                       all_predictions: bool = False, fuse_convcorr1: bool = True, fuse_encoder_tail: bool = True,
                       update_block_channels_last: bool = True):
    """Flows (n, 2, H, W) of the n CONSECUTIVE pairs (frames[i], frames[i + 1]) of a run of n + 1 frames -- what the
    open-loop encoder asks for inside a GOP (R:codec_processing.py:1498-1499: every P-frame's reference is the previous
    ORIGINAL frame).  Same modules, same order as ``raft_flow(model, frames[:-1], frames[1:])``, but the feature
    encoder sees each frame ONCE (n + 1 images instead of 2n): its normalisation is per sample (InstanceNorm,
    TV:raft.py:790), so a frame's feature map does not depend on which pair it is part of; the context encoder still
    runs on every pair's first frame."""
    if frames.dim() != 4 or frames.shape[0] < 2:
        raise ValueError(f"frames should be (n + 1 >= 2, 3, H, W), got {tuple(frames.shape)}")
    fe_norms = [m for m in model.feature_encoder.modules() if isinstance(m, torch.nn.modules.batchnorm._BatchNorm)]
    if any(m.training or not m.track_running_stats for m in fe_norms):
        raise RuntimeError("raft_flow_sequence needs a feature encoder whose normalisation is per sample (InstanceNorm) or "
                           "frozen (BatchNorm in eval mode); batch statistics would couple the frames")
    return _raft_flow_impl(model, frames, lambda x: (x[:-1], x[1:]), frames[:-1], num_flow_updates, corr_block,
                           all_predictions, fuse_convcorr1, fuse_encoder_tail, update_block_channels_last)


def _to_channels_last(module) -> None:
    """Store the module's convolution weights NHWC (values unchanged; a no-op when they already are).  NOTE: this
    re-allocates the weights once -- CUDA graphs captured before it must be re-captured (GraphedRaftFlow checks)."""
    if not getattr(module, "_rdvc_channels_last", False):
        module.to(memory_format=torch.channels_last)
        module._rdvc_channels_last = True


def _raft_flow_impl(model, enc_in: Tensor, split, image1: Tensor, num_flow_updates, corr_block, all_predictions,
                    fuse_convcorr1, fuse_encoder_tail, update_block_channels_last=True):
    """``enc_in``: every image the feature encoder has to see; ``split``: its output -> (first, second) feature maps of
    the pairs; ``image1``: the pairs' first frames (context encoder input)."""
    from torchvision.models.optical_flow._utils import upsample_flow

    blk = corr_block if corr_block is not None else model.corr_block
    if not isinstance(blk, TVCorrBlock):
        raise TypeError("raft_flow needs a rdvc_corr_b200.TVCorrBlock as the model's corr_block")
    batch, _, h, w = image1.shape
    if not ((h % 8 == 0) and (w % 8 == 0)):
        raise ValueError(f"input image H and W should be divisible by 8, instead got {h} (h) and {w} (w)")

    fe = model.feature_encoder
    if fuse_encoder_tail and _can_fuse_encoder_tail(model):
        if isinstance(fe, FeatureEncoder):      # layer3's output as a view of one NHWC buffer
            x = fe.forward_trunk(enc_in)
        else:
            x = fe.layer3(fe.layer2(fe.layer1(fe.convnormrelu(enc_in))))   # TV:raft.py:145-149
        fmap1, fmap2 = split(x)                                   # 128-channel activations; fe.conv runs inside the block
        if fmap1.shape[-2:] != (h // 8, w // 8):                  # TV:raft.py:494-495
            raise ValueError("The feature encoder should downsample H and W by 8")
        blk.build_pyramid_from_encoder(fmap1, fmap2, fe.conv.weight, fe.conv.bias)
    else:
        fmap1, fmap2 = split(fe(enc_in))
        if fmap1.shape[-2:] != (h // 8, w // 8):            # TV:raft.py:494-495
            raise ValueError("The feature encoder should downsample H and W by 8")
        blk.build_pyramid(fmap1, fmap2)
    fuse = fuse_convcorr1 and blk.layout == 1 and _can_fuse_convcorr1(model)      # 1 = RDVC_LAYOUT_TILED

    # Stock convolutions in NHWC where it pays: the update block's twelve convolutions per iteration and the context
    # encoder's run NHWC inside cuDNN; fed NCHW tensors (as RAFT.forward does) every one of them is wrapped in
    # nchw->nhwc / nhwc->nchw transposes -- 24 % of a P-frame's GPU time at 1080p
    # (profiles/r02raft_launches_summary.csv).  With the fused path their inputs are made channels_last and their
    # weights are stored NHWC: the same convolution kernels without the transposes (update block 10.3 -> 7.8 ms,
    # context encoder 2.6 -> 1.8 ms per P-frame at 1080p, tools/exp_update_block_layout.py, exp_encoder_layout.py).
    # The feature encoder stays NCHW: its InstanceNorm is slower in NHWC (3.1 -> 4.3 ms).
    cl = bool(update_block_channels_last) and fuse
    own_ce = isinstance(model.context_encoder, ContextEncoder)
    if cl:
        if not own_ce:
            _to_channels_last(model.context_encoder)
        _to_channels_last(model.update_block)
        if model.mask_predictor is not None:
            _to_channels_last(model.mask_predictor)
        if not own_ce:
            image1 = image1.contiguous(memory_format=torch.channels_last)
    hidden_size = model.update_block.hidden_state_size
    if own_ce:      # tanh / relu in the last layer's epilogue; both are channel slices of one NHWC buffer
        hidden_state, context = model.context_encoder.forward_split(image1, hidden_size)
    else:
        context_out = model.context_encoder(image1)
        hidden_state, context = torch.split(context_out, [hidden_size, context_out.shape[1] - hidden_size], dim=1)
        hidden_state = torch.tanh(hidden_state)
        context = F.relu(context)
        if cl:      # no-ops when the context encoder already produced NHWC
            hidden_state = hidden_state.contiguous(memory_format=torch.channels_last)
            context = context.contiguous(memory_format=torch.channels_last)

    coords0 = _coords_grid(batch, h // 8, w // 8, fmap1.device)
    coords1 = coords0.clone()
    corr_out = None if fuse else torch.empty((batch, blk.out_channels, h // 8, w // 8), dtype=torch.float32,
                                             device=fmap1.device)
    preds: List[Tensor] = []
    for it in range(num_flow_updates):
        flow = coords1 - coords0
        if fuse:
            hidden_state, delta_flow = _update_block_fused(model, blk, hidden_state, context, coords1, flow, cl)
        else:
            corr_features = index_pyramid(blk._pyr, coords1, blk.radius, out=corr_out)
            hidden_state, delta_flow = model.update_block(hidden_state, context, corr_features, flow)
        coords1 = coords1 + delta_flow
        if all_predictions or it == num_flow_updates - 1:
            if isinstance(model.mask_predictor, MaskPredictor):     # mask, softmax and convex sum in one GEMM epilogue
                preds.append(model.mask_predictor.upsample_flow(coords1 - coords0, hidden_state))
            else:
                up_mask = None if model.mask_predictor is None else model.mask_predictor(hidden_state).contiguous()   # upsample_flow views it
                preds.append(upsample_flow(flow=(coords1 - coords0).contiguous(), up_mask=up_mask))
    return preds if all_predictions else preds[-1]



class GraphedRaftFlow:
    """``raft_flow`` captured into a CUDA graph (one per input shape / dtype / autocast setting).

    ``runner = GraphedRaftFlow(model); flow = runner(image1, image2)`` -- the first call for a shape
    warms up, captures and replays; later calls copy the frames into the graph's static inputs and
    replay.  Every captured shape owns its own :class:`TVCorrBlock` (the graph bakes in the pyramid's
    address), so the model's own block stays free for eager use.  Inference only.
    """

    def __init__(self, model, num_flow_updates: int = 12, amp_dtype: Optional[torch.dtype] = None,
                 volume_dtype: torch.dtype = torch.float32, fuse_convcorr1: bool = True, max_entries: int = 4,
                 fuse_encoder_tail: bool = True, update_block_channels_last: bool = True):
        if not isinstance(model.corr_block, TVCorrBlock):
            raise TypeError("GraphedRaftFlow needs a model built with corr_block=rdvc_corr_b200.TVCorrBlock()")
        if model.training:
            # a graph captured in train mode would update BatchNorm running statistics on every replay
            raise RuntimeError("GraphedRaftFlow is inference only: call model.eval() first")
        self.model = model
        self.num_flow_updates = num_flow_updates
        self.amp_dtype = amp_dtype
        self.volume_dtype = volume_dtype
        self.fuse_convcorr1 = fuse_convcorr1
        self.fuse_encoder_tail = fuse_encoder_tail
        self.update_block_channels_last = update_block_channels_last
        self.max_entries = max_entries        # every captured shape pins a pyramid (5.7 GB at 1080p fp32)
        self._entries = {}                    # insertion-ordered: least recently used first

    def _run(self, blk, a, b):
        with torch.autocast("cuda", dtype=self.amp_dtype or torch.float16, enabled=self.amp_dtype is not None):
            kw = dict(corr_block=blk, fuse_convcorr1=self.fuse_convcorr1, fuse_encoder_tail=self.fuse_encoder_tail,
                      update_block_channels_last=self.update_block_channels_last)
            if b is None:      # a = a run of n + 1 frames
                return raft_flow_sequence(self.model, a, self.num_flow_updates, **kw)
            return raft_flow(self.model, a, b, self.num_flow_updates, **kw)

    def _weights_signature(self):
        """Where the model's parameters live: a captured graph has these addresses baked in, so a model that was
        moved / re-typed / re-laid-out since (``.half()``, ``.to(memory_format=...)``, a new device) must be re-captured."""
        return tuple(p.data_ptr() for p in self.model.parameters())

    def release(self, key=None) -> None:
        """Drop the captured graph(s) and the pyramids they pin (all shapes, or one ``(shape, dtype, device)`` key)."""
        keys = list(self._entries) if key is None else [key]
        for k in keys:
            e = self._entries.pop(k, None)
            if e is not None:
                e["graph"] = None
                e["blk"].release()

    def _capture(self, image1: Tensor, image2: Optional[Tensor]):
        dev = image1.device
        blk = TVCorrBlock(num_levels=self.model.corr_block.num_levels, radius=self.model.corr_block.radius,
                          volume_dtype=self.volume_dtype, layout=self.model.corr_block.layout)
        in1, in2 = image1.clone(), None if image2 is None else image2.clone()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(3):                      # cuDNN algorithm choice, workspaces, the pyramid buffer
                self._run(blk, in1, in2)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        with torch.no_grad(), torch.cuda.graph(graph):
            out = self._run(blk, in1, in2)
        return {"graph": graph, "in1": in1, "in2": in2, "out": out, "blk": blk, "weights": self._weights_signature()}

    @torch.no_grad()
    def __call__(self, image1: Tensor, image2: Tensor) -> Tensor:
        if not image1.is_cuda:
            raise RuntimeError("rdvc_corr_b200 runs on an sm_100 GPU only; got CPU frames.")
        if image1.shape != image2.shape or image1.dtype != image2.dtype:
            raise ValueError(f"input images should have the same shape and dtype, got {image1.shape} / {image2.shape}")
        if self.model.training:
            raise RuntimeError("GraphedRaftFlow is inference only: the model was switched back to train mode")
        return self._replay((tuple(image1.shape), image1.dtype, image1.device), image1, image2)

    @torch.no_grad()
    def sequence(self, frames: Tensor) -> Tensor:
        """``raft_flow_sequence(model, frames)`` -- the n flows of a run of n + 1 consecutive frames, the feature
        encoder seeing each frame once -- as one graph per run length."""
        if not frames.is_cuda:
            raise RuntimeError("rdvc_corr_b200 runs on an sm_100 GPU only; got CPU frames.")
        if frames.dim() != 4 or frames.shape[0] < 2:
            raise ValueError(f"frames should be (n + 1 >= 2, 3, H, W), got {tuple(frames.shape)}")
        if self.model.training:
            raise RuntimeError("GraphedRaftFlow is inference only: the model was switched back to train mode")
        return self._replay(("sequence", tuple(frames.shape), frames.dtype, frames.device), frames, None)

    def _replay(self, key, image1: Tensor, image2: Optional[Tensor]) -> Tensor:
        e = self._entries.pop(key, None)
        if e is not None and e["weights"] != self._weights_signature():
            e["graph"] = None                                       # the parameters moved since the capture
            e["blk"].release()
            e = None
        if e is None:
            while len(self._entries) >= self.max_entries:          # evict the least recently used shape
                self.release(next(iter(self._entries)))
            e = self._capture(image1, image2)
        self._entries[key] = e                                      # most recently used last
        e["in1"].copy_(image1)
        if image2 is not None:
            e["in2"].copy_(image2)
        e["graph"].replay()
        return e["out"].clone()
