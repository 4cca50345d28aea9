"""B200 drop-in for RAFT's context encoder: torchvision's ``FeatureEncoder`` with ``norm_layer=BatchNorm2d``
(TV:raft.py:116-168) in eval mode, with every BatchNorm folded into its convolution.

* ``ContextEncoder()`` -- torchvision's constructor; only raft_large's context configuration is accepted
  - ``forward(x)``: the stock contract, (B, 3, H, W) -> (B, 256, ceil(H / 8), ceil(W / 8)), channels_last memory, so
    ``RAFT.forward`` works with the module swapped in;
  - ``forward_split(x, hidden_size=128)``: ``(tanh(out[:, :128]), relu(out[:, 128:]))`` computed in the last layer's
    epilogue, two channel slices of one NHWC buffer.  ``raft_flow`` calls this when the module is swapped in.

The parameter and buffer tree is torchvision's (the constructor adopts the submodules of a ``FeatureEncoder``), so state
dicts load with ``strict=True`` in both directions.  The 16 convolutions run as tcgen05 implicit GEMMs
(``rdvc_corr_context_encoder``): 16-bit operands, fp32 accumulation, fp32 epilogues, every activation rounded once to
the operand dtype.  There is no fallback: CPU tensors, other configurations, gradient-carrying inputs and training
mode raise -- training mode even under ``torch.no_grad()``, because the stock BatchNorm would then normalise with
batch statistics and update its running statistics, which folded weights cannot do.

Swap it into a torchvision ``raft_large``::

    ce = rc.ContextEncoder()
    ce.load_state_dict(model.context_encoder.state_dict())
    model.context_encoder = ce.to(device).eval()
"""
from __future__ import annotations

import ctypes
from typing import Tuple

import numpy as np
import torch
from torch import Tensor, nn

from . import _cabi
from .motion_encoder import _dtypes, _ptrs, _stream
from .recurrent_block import _DT, _need_cuda

_LAYERS, _STRIDES, _OUT = (64, 64, 96, 128, 256), (2, 1, 2, 2), 256


def _convs_and_norms(m: nn.Module):
    """The 16 (conv, BatchNorm or None) pairs in the order of ``include/rdvc_corr.h`` (parameter-tree order)."""
    out = [(m.convnormrelu[0], m.convnormrelu[1])]
    for layer in (m.layer1, m.layer2, m.layer3):
        for blk in layer:
            out.append((blk.convnormrelu1[0], blk.convnormrelu1[1]))
            if isinstance(blk.downsample, nn.Sequential):
                out.append((blk.downsample[0], blk.downsample[1]))
            out.append((blk.convnormrelu2[0], blk.convnormrelu2[1]))
    out.append((m.conv, None))
    return out


def _version(t: Tensor):
    return t.data_ptr(), t._version


class PackedContextEncoder:
    """All 16 layers with BatchNorm folded in fp64 (``rdvc_corr_context_encoder_pack_weights``, host): the 16-bit GEMM
    operand and the fp32 biases, on the device."""

    def __init__(self, layers, op_dtype: torch.dtype, device, key):
        lib = _cabi.load()
        f32 = lambda t: np.ascontiguousarray(t.detach().to(torch.float32).cpu().numpy())   # noqa: E731
        keep = []                                                    # the host arrays must outlive the call

        def arr(ts):
            a = [f32(t) for t in ts]
            keep.extend(a)
            return _ptrs(ctypes.c_void_p, [x.ctypes.data for x in a])

        norms = [bn for _, bn in layers[:-1]]
        conv_w, conv_b = arr([c.weight for c, _ in layers]), arr([c.bias for c, _ in layers])
        bn_w, bn_b = arr([bn.weight for bn in norms]), arr([bn.bias for bn in norms])
        bn_m, bn_v = arr([bn.running_mean for bn in norms]), arr([bn.running_var for bn in norms])
        eps = _ptrs(ctypes.c_double, [float(bn.eps) for bn in norms] + [0.0])
        packed = np.zeros(lib.rdvc_corr_context_encoder_packed_weight_bytes() // 2, np.uint16)
        bias = np.zeros(lib.rdvc_corr_context_encoder_packed_bias_bytes() // 4, np.float32)
        _cabi.check(lib.rdvc_corr_context_encoder_pack_weights(conv_w, conv_b, bn_w, bn_b, bn_m, bn_v, eps, _DT[op_dtype],
                                                               packed.ctypes.data, bias.ctypes.data),
                    "rdvc_corr_context_encoder_pack_weights")
        self.weight = torch.from_numpy(packed.view(np.int16)).to(device)
        self.bias = torch.from_numpy(bias).to(device)
        self.key = key


class ContextEncoder(nn.Module):
    """TV:raft.py:116-168 with ``norm_layer=BatchNorm2d`` for raft_large's context configuration.  Same constructor,
    parameter and buffer names, ``forward`` contract.

    The image is read at its own strides (NCHW or channels_last) in fp32, fp16 or bf16.  fp32 in -> fp16 operands and
    fp32 out; autocast -> its dtype as the operands and the output; fp16 / bf16 in -> that dtype throughout.
    Inference only, in eval mode.

    Weights are folded and packed once per key and device; the key covers every convolution weight and bias, every
    BatchNorm weight, bias, running mean and running variance (address and version) and eps, so a
    ``load_state_dict`` that changes only the running statistics re-packs.  A CUDA graph captured through this module
    replays the weights that were packed when it was captured: after changing parameters or running statistics in
    place, run the module eagerly (it re-packs) and re-capture the graph.
    """

    def __init__(self, *, block=None, layers=_LAYERS, strides=_STRIDES, norm_layer=nn.BatchNorm2d):
        """``block=None`` stands for torchvision's ``ResidualBlock`` (the package does not import torchvision before a
        module is built)."""
        from torchvision.models.optical_flow.raft import ResidualBlock
        block = ResidualBlock if block is None else block
        if block is not ResidualBlock or tuple(layers) != _LAYERS or tuple(strides) != _STRIDES or norm_layer is not nn.BatchNorm2d:
            raise ValueError(
                f"the B200 kernels cover raft_large's context encoder only (block=ResidualBlock, layers={_LAYERS}, "
                f"strides={_STRIDES}, norm_layer=BatchNorm2d); got block={getattr(block, '__name__', block)}, "
                f"layers={tuple(layers)}, strides={tuple(strides)}, norm_layer={getattr(norm_layer, '__name__', norm_layer)}. "
                "InstanceNorm (the feature encoder), norm_layer=None and raft_small's BottleneckBlock are not supported")
        from torchvision.models.optical_flow.raft import FeatureEncoder
        super().__init__()
        fe = FeatureEncoder(block=block, layers=layers, strides=strides, norm_layer=norm_layer)   # its tree and init
        self.convnormrelu, self.layer1, self.layer2, self.layer3, self.conv = (fe.convnormrelu, fe.layer1, fe.layer2,
                                                                               fe.layer3, fe.conv)
        self.output_dim, self.downsample_factor = fe.output_dim, fe.downsample_factor
        self._pack = None

    def _key(self, op, dev):
        key = [op, torch.device(dev)]
        for conv, bn in _convs_and_norms(self):
            key += [_version(conv.weight), _version(conv.bias)]
            if bn is not None:
                key += [_version(bn.weight), _version(bn.bias), _version(bn.running_mean), _version(bn.running_var),
                        float(bn.eps)]
        return tuple(key)

    def _check(self, x: Tensor):
        _cabi.forward_only("ContextEncoder", x)
        norms = [m for m in self.modules() if isinstance(m, nn.modules.batchnorm._BatchNorm)]
        if self.training or any(m.training or not m.track_running_stats for m in norms):
            raise RuntimeError("rdvc_corr_b200.ContextEncoder folds BatchNorm's running statistics into its weights and "
                               "runs in eval mode only (in train mode BatchNorm would use batch statistics): call .eval()")
        _need_cuda(x)
        if x.dim() != 4 or x.shape[1] != 3:
            raise ValueError(f"the image must be (B, 3, H, W), got {tuple(x.shape)}")
        if x.dtype not in _DT:
            raise ValueError(f"unsupported image dtype {x.dtype}")

    def forward(self, x: Tensor) -> Tensor:
        """TV:raft.py:144-152: (B, 256, ceil(H / 8), ceil(W / 8)) in the activation dtype, channels_last memory."""
        self._check(x)
        return self._run(x, _cabi.RDVC_CE_OUT_RAW).permute(0, 3, 1, 2)

    def forward_split(self, x: Tensor, hidden_size: int = 128) -> Tuple[Tensor, Tensor]:
        """RAFT's ``tanh`` / ``relu`` of the split context (TV:raft.py:502-505): ``(hidden_state, context)``, channels
        0-127 and 128-255 of one (B, h, w, 256) NHWC buffer, as (B, C, h, w) views."""
        if hidden_size != 128:
            raise ValueError(f"the fused split covers raft_large's hidden_size=128, got {hidden_size}")
        self._check(x)
        out = self._run(x, _cabi.RDVC_CE_OUT_SPLIT).permute(0, 3, 1, 2)
        return out[:, :hidden_size], out[:, hidden_size:]

    def _run(self, x: Tensor, out_form: int) -> Tensor:
        act, op = _dtypes(x)
        dev = x.device
        B, _, H, W = x.shape
        key = self._key(op, dev)
        if self._pack is None or self._pack.key != key:
            self._pack = PackedContextEncoder(_convs_and_norms(self), op, dev, key)
        pk = self._pack
        lib = _cabi.load()
        ws_bytes = lib.rdvc_corr_context_encoder_workspace_bytes(B, H, W, _DT[act])
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        out = torch.empty((B, (H + 7) // 8, (W + 7) // 8, _OUT), dtype=act, device=dev)
        xs = x.detach()
        with torch.cuda.device(dev):
            rc = lib.rdvc_corr_context_encoder(xs.data_ptr(), _ptrs(ctypes.c_longlong, list(xs.stride())), _DT[xs.dtype],
                                               B, H, W, _DT[op], pk.weight.data_ptr(), pk.bias.data_ptr(), out_form,
                                               ws.data_ptr(), ws_bytes, out.data_ptr(), _OUT, _DT[act], _stream(dev))
        _cabi.check(rc, "rdvc_corr_context_encoder")
        return out
