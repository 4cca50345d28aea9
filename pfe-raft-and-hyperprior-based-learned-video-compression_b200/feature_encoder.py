"""B200 drop-in for RAFT's feature encoder: torchvision's ``FeatureEncoder`` with ``norm_layer=InstanceNorm2d``
(TV:raft.py:116-168), raft_large's feature configuration.

* ``FeatureEncoder()`` -- torchvision's constructor; only raft_large's feature configuration is accepted
  - ``forward(x)``: the stock contract, (B, 3, H, W) -> (B, 256, ceil(H / 8), ceil(W / 8)), channels_last memory, so
    ``RAFT.forward`` works with the module swapped in;
  - ``forward_trunk(x)``: layer3's output (B, 128, ceil(H / 8), ceil(W / 8)), a view of an NHWC buffer in the operand
    dtype -- the input of ``conv``.  ``raft_flow`` hands it to ``TVCorrBlock.build_pyramid_from_encoder``.

The parameter tree is torchvision's (the constructor adopts the submodules of a ``FeatureEncoder``): the 16 convolution
weights and biases, so state dicts load with ``strict=True`` in both directions.  The 16 convolutions run as tcgen05
implicit GEMMs (``rdvc_corr_feature_encoder``) whose epilogues store the raw output and per-tile InstanceNorm
statistics; a finalize and an apply kernel per layer normalise it.  Every activation is rounded once to the operand
dtype.  There is no fallback: CPU tensors, other configurations and gradient-carrying inputs raise.  InstanceNorm
without running statistics computes the same in train and eval mode, so both are accepted.

Swap it into a torchvision ``raft_large``::

    fe = rc.FeatureEncoder()
    fe.load_state_dict(model.feature_encoder.state_dict())
    model.feature_encoder = fe.to(device)
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch
from torch import Tensor, nn

from . import _cabi
from .context_encoder import _convs_and_norms, _version
from .motion_encoder import _dtypes, _ptrs, _stream
from .recurrent_block import _DT, _need_cuda

_LAYERS, _STRIDES, _OUT, _TRUNK = (64, 64, 96, 128, 256), (2, 1, 2, 2), 256, 128


class PackedFeatureEncoder:
    """The 16 convolutions packed by ``rdvc_corr_context_encoder_pack_weights`` with the identity norm (gamma 1, beta 0,
    mean 0, variance 1, eps 0: the scale is exactly 1 in fp64, so each weight is rounded once): the 16-bit GEMM operand
    and the fp32 biases, on the device."""

    def __init__(self, convs, op_dtype: torch.dtype, device, key):
        lib = _cabi.load()
        f32 = lambda t: np.ascontiguousarray(t.detach().to(torch.float32).cpu().numpy())   # noqa: E731
        keep = []                                                    # the host arrays must outlive the call

        def arr(a):
            keep.extend(a)
            return _ptrs(ctypes.c_void_p, [x.ctypes.data for x in a])

        norms = [(np.ones(c.out_channels, np.float32), np.zeros(c.out_channels, np.float32)) for c in convs[:-1]]
        conv_w, conv_b = arr([f32(c.weight) for c in convs]), arr([f32(c.bias) for c in convs])
        ones, zeros = arr([o for o, _ in norms]), arr([z for _, z in norms])
        eps = _ptrs(ctypes.c_double, [0.0] * len(convs))
        packed = np.zeros(lib.rdvc_corr_context_encoder_packed_weight_bytes() // 2, np.uint16)
        bias = np.zeros(lib.rdvc_corr_context_encoder_packed_bias_bytes() // 4, np.float32)
        _cabi.check(lib.rdvc_corr_context_encoder_pack_weights(conv_w, conv_b, ones, zeros, zeros, ones, eps, _DT[op_dtype],
                                                               packed.ctypes.data, bias.ctypes.data),
                    "rdvc_corr_context_encoder_pack_weights")
        self.weight = torch.from_numpy(packed.view(np.int16)).to(device)
        self.bias = torch.from_numpy(bias).to(device)
        self.key = key


class FeatureEncoder(nn.Module):
    """TV:raft.py:116-168 with ``norm_layer=InstanceNorm2d`` for raft_large's feature configuration.  Same constructor,
    parameter names, ``forward`` contract.

    The image is read at its own strides (NCHW or channels_last) in fp32, fp16 or bf16.  fp32 in -> fp16 operands and
    fp32 out; autocast -> its dtype as the operands and the output; fp16 / bf16 in -> that dtype throughout.
    ``forward_trunk`` returns the operand dtype.  Inference only (no gradients), in train or eval mode.

    Weights are packed once per key: every convolution weight and bias (address and version), the device and the
    operand dtype.  Each InstanceNorm's eps is read at every call.  A CUDA graph captured through this module replays
    the weights that were packed when it was captured: after changing parameters in place, run the module eagerly
    (it re-packs) and re-capture the graph.
    """

    def __init__(self, *, block=None, layers=_LAYERS, strides=_STRIDES, norm_layer=nn.InstanceNorm2d):
        """``block=None`` stands for torchvision's ``ResidualBlock`` (the package does not import torchvision before a
        module is built)."""
        from torchvision.models.optical_flow.raft import FeatureEncoder as TVFeatureEncoder, ResidualBlock
        block = ResidualBlock if block is None else block
        ok = block is ResidualBlock and tuple(layers) == _LAYERS and tuple(strides) == _STRIDES and norm_layer is not None
        fe = TVFeatureEncoder(block=block, layers=layers, strides=strides, norm_layer=norm_layer) if ok else None
        norms = [] if fe is None else [n for _, n in _convs_and_norms(fe)[:-1]]
        if not ok or not all(type(n) is nn.InstanceNorm2d and not n.affine and not n.track_running_stats for n in norms):
            raise ValueError(
                f"the B200 kernels cover raft_large's feature encoder only (block=ResidualBlock, layers={_LAYERS}, "
                f"strides={_STRIDES}, norm_layer=InstanceNorm2d without affine parameters or running statistics); got "
                f"block={getattr(block, '__name__', block)}, layers={tuple(layers)}, strides={tuple(strides)}, "
                f"norm_layer={getattr(norm_layer, '__name__', norm_layer)}.  BatchNorm2d is rc.ContextEncoder; "
                "norm_layer=None and raft_small's BottleneckBlock are not supported")
        super().__init__()
        self.convnormrelu, self.layer1, self.layer2, self.layer3, self.conv = (fe.convnormrelu, fe.layer1, fe.layer2,
                                                                               fe.layer3, fe.conv)
        self.output_dim, self.downsample_factor = fe.output_dim, fe.downsample_factor
        self._pack = None

    def _convs(self):
        return [c for c, _ in _convs_and_norms(self)]

    def _eps(self):
        return [float(n.eps) for _, n in _convs_and_norms(self)[:-1]]

    def _key(self, op, dev):
        key = [op, torch.device(dev)]
        for conv in self._convs():
            key += [_version(conv.weight), _version(conv.bias)]
        return tuple(key)

    def _check(self, x: Tensor):
        _cabi.forward_only("FeatureEncoder", x)
        if x.dim() != 4 or x.shape[1] != 3:
            raise ValueError(f"the image must be (B, 3, H, W), got {tuple(x.shape)}")
        if x.dtype not in _DT:
            raise ValueError(f"unsupported image dtype {x.dtype}")
        if (x.shape[2] + 7) // 8 == 1 and (x.shape[3] + 7) // 8 == 1:
            raise ValueError(f"Expected more than 1 spatial element when training, got input size {tuple(x.shape)}: "
                             "layer3's InstanceNorm would normalise a 1 x 1 plane")
        _need_cuda(x)

    def forward(self, x: Tensor) -> Tensor:
        """TV:raft.py:144-152: (B, 256, ceil(H / 8), ceil(W / 8)) in the activation dtype, channels_last memory."""
        self._check(x)
        act, _ = _dtypes(x)
        return self._run(x, _cabi.RDVC_FE_OUT_FEATURES, _OUT, act).permute(0, 3, 1, 2)

    def forward_trunk(self, x: Tensor) -> Tensor:
        """TV:raft.py:145-149: layer3's output (B, 128, ceil(H / 8), ceil(W / 8)) in the operand dtype, a view of an
        NHWC buffer."""
        self._check(x)
        _, op = _dtypes(x)
        return self._run(x, _cabi.RDVC_FE_OUT_TRUNK, _TRUNK, op).permute(0, 3, 1, 2)

    def _run(self, x: Tensor, out_form: int, channels: int, out_dtype: torch.dtype) -> Tensor:
        act, op = _dtypes(x)
        dev = x.device
        B, _, H, W = x.shape
        key = self._key(op, dev)
        if self._pack is None or self._pack.key != key:
            self._pack = PackedFeatureEncoder(self._convs(), op, dev, key)
        pk = self._pack
        lib = _cabi.load()
        ws_bytes = lib.rdvc_corr_feature_encoder_workspace_bytes(B, H, W, _DT[act])
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        out = torch.empty((B, (H + 7) // 8, (W + 7) // 8, channels), dtype=out_dtype, device=dev)
        xs = x.detach()
        with torch.cuda.device(dev):
            rc = lib.rdvc_corr_feature_encoder(xs.data_ptr(), _ptrs(ctypes.c_longlong, list(xs.stride())), _DT[xs.dtype],
                                               B, H, W, _DT[op], pk.weight.data_ptr(), pk.bias.data_ptr(),
                                               _ptrs(ctypes.c_double, self._eps()), out_form, ws.data_ptr(), ws_bytes,
                                               out.data_ptr(), channels, _DT[out_dtype], _stream(dev))
        _cabi.check(rc, "rdvc_corr_feature_encoder")
        return out
