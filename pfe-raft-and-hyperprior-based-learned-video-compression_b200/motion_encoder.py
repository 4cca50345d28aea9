"""B200 drop-ins for the rest of RAFT's update block: torchvision's ``MotionEncoder`` (TV:raft.py:171-211) and
``FlowHead`` (TV:raft.py:272-285), as convolutions over NHWC 16-bit activations.

* ``MotionEncoder(in_channels_corr=324)`` with ``forward(flow, corr_features)``      TV:raft.py:177-211
* ``FlowHead(in_channels=128, hidden_size=256)`` with ``forward(x)``                   TV:raft.py:275-285

Both keep the reference's constructor and parameter tree (``convcorr1.0.weight`` ... ``conv.0.bias``; ``conv1.*`` /
``conv2.*``), so state dicts load with ``strict=True`` in both directions, and convcorr1 stays a ``Conv2d`` + ``ReLU``
sequence, which is what ``raft_flow`` fuses with the correlation lookup.  The 3x3 layers run as tcgen05 implicit GEMMs
(``rdvc_corr_update_conv``), convflow1 (7x7, 2 -> 128) as a CUDA-core direct convolution; every ``torch.cat`` of the stock
module is a write into a channel slice.  16-bit operands, fp32 accumulation, bias and ReLU in fp32.  There is no
fallback: CPU tensors, other configurations (raft_small's included) and gradient-carrying calls raise.

Swap all three submodules of a torchvision ``raft_large``::

    ub = model.update_block
    me, fh = rc.MotionEncoder(in_channels_corr=324), rc.FlowHead(in_channels=128, hidden_size=256)
    me.load_state_dict(ub.motion_encoder.state_dict()); fh.load_state_dict(ub.flow_head.state_dict())
    ub.motion_encoder, ub.flow_head = me.to(device), fh.to(device)

One difference from the stock module: under autocast, the stock ``torch.cat([corr_flow, flow])`` promotes the motion
features to fp32 (the flow is fp32); this module returns them in the autocast dtype.  The stock recurrent block rounds
them to that dtype anyway before its first convolution.
"""
from __future__ import annotations

import ctypes
from typing import Dict

import numpy as np
import torch
from torch import Tensor, nn

from . import _cabi
from .corr_block import PackedConv1x1, _param_key, feat_shape
from .recurrent_block import _DT, _need_cuda, _nhwc

_CORR_IN, _CORR_LAYERS, _FLOW_LAYERS, _OUT = 324, (256, 192), (128, 64), 128
_FH_IN, _FH_HIDDEN = 128, 256
_LEVELS, _RADIUS = 4, 4
from ._cabi import (RDVC_UC_CONV as UC_CONV, RDVC_UC_CONVCORR2 as UC_CONVCORR2, RDVC_UC_CONVFLOW1 as UC_CONVFLOW1,  # noqa: E402
                    RDVC_UC_CONVFLOW2 as UC_CONVFLOW2, RDVC_UC_FH_CONV1 as UC_FH_CONV1, RDVC_UC_FH_CONV2 as UC_FH_CONV2)


class PackedUpdateConv:
    """One layer's weight as the kernel's 16-bit GEMM operand (``rdvc_corr_update_conv_pack_weights``, host) + its fp32 bias,
    on the device.  Rebuilt when a parameter changes version, address or device."""

    def __init__(self, conv: nn.Conv2d, layer: int, op_dtype: torch.dtype, device):
        lib = _cabi.load()
        w = np.ascontiguousarray(conv.weight.detach().to(torch.float32).cpu().numpy())
        packed = np.zeros(lib.rdvc_corr_update_conv_packed_weight_bytes(layer) // 2, np.uint16)
        _cabi.check(lib.rdvc_corr_update_conv_pack_weights(layer, w.ctypes.data, _DT[op_dtype], packed.ctypes.data),
                    "rdvc_corr_update_conv_pack_weights")
        self.weight = torch.from_numpy(packed.view(np.int16)).to(device)
        self.bias = conv.bias.detach().to(torch.float32).to(device).contiguous()
        self.key = _param_key(conv.weight, conv.bias, op_dtype, device)


def _dtypes(ref: Tensor):
    """(activation dtype, 16-bit operand dtype): the autocast dtype when autocast is on, else ``ref``'s."""
    act = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else ref.dtype
    if act not in _DT:
        raise ValueError(f"unsupported dtype {act}")
    return act, (torch.float16 if act == torch.float32 else act)


def _stream(dev) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def _ptrs(ctype, values):
    return (ctype * len(values))(*values)


class _Packs:
    """Per-module cache of packed layers, keyed by layer index."""

    def __init__(self):
        self._d: Dict[int, object] = {}

    def get(self, i: int, key, make):
        pk = self._d.get(i)
        if pk is None or pk.key != key:
            pk = self._d[i] = make()
        return pk


class MotionEncoder(nn.Module):
    """TV:raft.py:171-211 for raft_large's configuration.  Same constructor, parameter names and ``forward`` contract.

    ``forward(flow, corr_features)``: the stock contract (``model(img1, img2)`` works with the module swapped in).  The
    (B, 324, h, w) lookup is repacked into the 1x1 GEMM's K-major feature rows with torch ops and convcorr1 runs through
    ``rdvc_conv1x1_ex``, writing NHWC; then :meth:`forward_fused`.
    ``forward_fused(flow, c1)``: from convcorr1's output (B, 256, h, w) -- ideally the channels_last 16-bit tensor of
    ``TVCorrBlock.index_pyramid_convcorr1(..., nhwc=True)``, which is what ``raft_flow`` passes.

    The result is the (B, 128, h, w) motion features [conv | flow], channels_last, in the activation dtype: fp32 in,
    fp32 out (operands rounded to fp16 -- the stock fp32 path multiplies in TF32, the same 10-bit mantissa); autocast
    gives its dtype (operands in it).  Inference only.

    Weights are packed once per parameter version and device.  A CUDA graph captured through this module replays the
    weights that were packed when it was captured: after changing parameters in place, run the module eagerly (it
    re-packs) and re-capture the graph -- the same contract as the library's fused 1x1 convolution weights.  Moving
    the parameters (``.to(...)``, ``load_state_dict`` into a moved module) re-packs on the next call.
    """

    def __init__(self, *, in_channels_corr: int, corr_layers=_CORR_LAYERS, flow_layers=_FLOW_LAYERS,
                 out_channels: int = _OUT):
        from torchvision.ops import Conv2dNormActivation
        super().__init__()
        if (in_channels_corr != _CORR_IN or tuple(corr_layers) != _CORR_LAYERS or tuple(flow_layers) != _FLOW_LAYERS
                or out_channels != _OUT):
            raise ValueError(
                f"the B200 kernels cover raft_large's motion encoder only (in_channels_corr={_CORR_IN}, "
                f"corr_layers={_CORR_LAYERS}, flow_layers={_FLOW_LAYERS}, out_channels={_OUT}); got "
                f"in_channels_corr={in_channels_corr}, corr_layers={corr_layers}, flow_layers={flow_layers}, "
                f"out_channels={out_channels}")
        self.convcorr1 = Conv2dNormActivation(_CORR_IN, _CORR_LAYERS[0], norm_layer=None, kernel_size=1)
        self.convcorr2 = Conv2dNormActivation(_CORR_LAYERS[0], _CORR_LAYERS[1], norm_layer=None, kernel_size=3)
        self.convflow1 = Conv2dNormActivation(2, _FLOW_LAYERS[0], norm_layer=None, kernel_size=7)
        self.convflow2 = Conv2dNormActivation(_FLOW_LAYERS[0], _FLOW_LAYERS[1], norm_layer=None, kernel_size=3)
        self.conv = Conv2dNormActivation(_CORR_LAYERS[-1] + _FLOW_LAYERS[-1], _OUT - 2, norm_layer=None, kernel_size=3)
        self.out_channels = out_channels
        self._packs = _Packs()

    def _layers(self, op, dev):
        seq = ((UC_CONVCORR2, self.convcorr2), (UC_CONVFLOW1, self.convflow1), (UC_CONVFLOW2, self.convflow2),
               (UC_CONV, self.conv))
        return [self._packs.get(i, _param_key(m[0].weight, m[0].bias, op, dev),
                                lambda m=m, i=i: PackedUpdateConv(m[0], i, op, dev)) for i, m in seq]

    def _check(self, flow: Tensor, x: Tensor, name: str, channels: int):
        _cabi.forward_only("MotionEncoder", flow, x)
        if self.training and torch.is_grad_enabled():
            raise RuntimeError("rdvc_corr_b200.MotionEncoder is forward-only: call .eval() or run under torch.no_grad()")
        _need_cuda(flow, x)
        if x.dim() != 4 or x.shape[1] != channels:
            raise ValueError(f"{name} must be (B, {channels}, h, w), got {tuple(x.shape)}")
        if flow.dim() != 4 or flow.shape[1] != 2 or flow.shape[0] != x.shape[0] or flow.shape[2:] != x.shape[2:]:
            raise ValueError(f"flow must be (B, 2, h, w) like {name} {tuple(x.shape)}, got {tuple(flow.shape)}")

    def forward(self, flow: Tensor, corr_features: Tensor) -> Tensor:
        self._check(flow, corr_features, "corr_features", _CORR_IN)
        act, op = _dtypes(corr_features)
        dev = corr_features.device
        B, _, h, w = corr_features.shape
        conv = self.convcorr1[0]
        pk = self._packs.get(-1, _param_key(conv.weight, conv.bias, op, dev),
                             lambda: PackedConv1x1(conv.weight, conv.bias, _LEVELS, _RADIUS, op, dev))
        # the lookup's K-major feature rows (corr_block.index_pyramid_kmajor): feature l * 88 + j * 9 + i is torchvision
        # channel l * 81 + i * 9 + j, features 81..87 of a level are zero; chunk-major (K / 8, rows, 8)
        kc, rows, _ = feat_shape(B, h, w, _LEVELS, _RADIUS)
        S = 2 * _RADIUS + 1
        c = corr_features.detach().to(op).reshape(B, _LEVELS, S, S, h * w).transpose(2, 3).reshape(B, _LEVELS, S * S, h * w)
        c = torch.nn.functional.pad(c, (0, 0, 0, kc * 8 // _LEVELS - S * S))          # (B, L, 88, h*w)
        k = c.reshape(B, kc * 8, h * w).permute(1, 0, 2).reshape(kc * 8, B * h * w)
        feat = torch.zeros(kc, rows, 8, dtype=op, device=dev)
        feat[:, :B * h * w] = k.reshape(kc, 8, B * h * w).transpose(1, 2)
        c1 = torch.empty((B, h, w, _CORR_LAYERS[0]), dtype=op, device=dev)
        with torch.cuda.device(dev):
            _cabi.check(_cabi.load().rdvc_conv1x1_ex(feat.data_ptr(), _DT[op], pk.weight.data_ptr(), pk.bias.data_ptr(), B, h,
                                                     w, _LEVELS, _RADIUS, _CORR_LAYERS[0], _cabi.RDVC_ACT_RELU,
                                                     c1.data_ptr(), _DT[op], _CORR_LAYERS[0], _stream(dev)),
                        "rdvc_conv1x1_ex")
        return self._run(flow, c1.permute(0, 3, 1, 2), act, op)

    def forward_fused(self, flow: Tensor, c1: Tensor) -> Tensor:
        """``forward`` from convcorr1's output ``c1`` = relu(convcorr1(corr_features)), (B, 256, h, w)."""
        self._check(flow, c1, "c1", _CORR_LAYERS[0])
        act, op = _dtypes(flow)
        return self._run(flow, c1, act, op)

    def _run(self, flow: Tensor, c1: Tensor, act, op) -> Tensor:
        dev = c1.device
        B, _, h, w = c1.shape
        x, ps = _nhwc(c1.detach() if c1.dtype == op else c1.detach().to(op))
        f = flow.detach().to(torch.float32)
        packs = self._layers(op, dev)
        lib = _cabi.load()
        ws_bytes = lib.rdvc_corr_motion_encoder_workspace_bytes(B, h, w)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        out = torch.empty((B, h, w, _OUT), dtype=act, device=dev)
        fs = _ptrs(ctypes.c_longlong, list(f.stride()))
        with torch.cuda.device(dev):
            rc = lib.rdvc_corr_motion_encoder(x.data_ptr(), ps, f.data_ptr(), fs, B, h, w, _DT[op],
                                         _ptrs(ctypes.c_void_p, [p.weight.data_ptr() for p in packs]),
                                         _ptrs(ctypes.c_void_p, [p.bias.data_ptr() for p in packs]), ws.data_ptr(),
                                         ws_bytes, out.data_ptr(), _OUT, _DT[act], _stream(dev))
        _cabi.check(rc, "rdvc_corr_motion_encoder")
        return out.permute(0, 3, 1, 2)


class FlowHead(nn.Module):
    """TV:raft.py:272-285 for raft_large's configuration (in_channels=128, hidden_size=256).  Same constructor,
    parameter names and ``forward`` contract.

    ``forward(x)``: the hidden state (B, 128, h, w), NCHW or channels_last (the fast path: read in place, a channel
    slice of a channels_last tensor included) -> the delta flow (B, 2, h, w), contiguous, in the activation dtype (fp32
    in -> fp32 out with fp16 operands; autocast -> its dtype).  Inference only.  Weights are packed once per parameter
    version and device, with the CUDA-graph contract of :class:`MotionEncoder`.
    """

    def __init__(self, *, in_channels: int, hidden_size: int):
        super().__init__()
        if in_channels != _FH_IN or hidden_size != _FH_HIDDEN:
            raise ValueError(f"the B200 kernels cover raft_large's flow head only (in_channels={_FH_IN}, "
                             f"hidden_size={_FH_HIDDEN}); got in_channels={in_channels}, hidden_size={hidden_size}")
        self.conv1 = nn.Conv2d(in_channels, hidden_size, 3, padding=1)
        self.conv2 = nn.Conv2d(hidden_size, 2, 3, padding=1)
        self.relu = nn.ReLU(inplace=True)
        self._packs = _Packs()

    def forward(self, x: Tensor) -> Tensor:
        _cabi.forward_only("FlowHead", x)
        if self.training and torch.is_grad_enabled():
            raise RuntimeError("rdvc_corr_b200.FlowHead is forward-only: call .eval() or run under torch.no_grad()")
        _need_cuda(x)
        if x.dim() != 4 or x.shape[1] != _FH_IN:
            raise ValueError(f"x must be (B, {_FH_IN}, h, w), got {tuple(x.shape)}")
        act, op = _dtypes(x)
        dev = x.device
        B, _, h, w = x.shape
        xh, ps = _nhwc(x.detach() if x.dtype == act else x.detach().to(act))
        packs = [self._packs.get(i, _param_key(c.weight, c.bias, op, dev), lambda c=c, i=i: PackedUpdateConv(c, i, op, dev))
                 for i, c in ((UC_FH_CONV1, self.conv1), (UC_FH_CONV2, self.conv2))]
        lib = _cabi.load()
        ws_bytes = lib.rdvc_corr_flow_head_workspace_bytes(B, h, w, _DT[act])
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        out = torch.empty((B, 2, h, w), dtype=act, device=dev)
        with torch.cuda.device(dev):
            rc = lib.rdvc_corr_flow_head(xh.data_ptr(), ps, _DT[act], B, h, w, _DT[op],
                                    _ptrs(ctypes.c_void_p, [p.weight.data_ptr() for p in packs]),
                                    _ptrs(ctypes.c_void_p, [p.bias.data_ptr() for p in packs]), ws.data_ptr(), ws_bytes,
                                    out.data_ptr(), _stream(dev))
        _cabi.check(rc, "rdvc_corr_flow_head")
        return out
