"""B200 drop-in for RAFT's mask predictor: torchvision's ``MaskPredictor`` (TV:raft.py:311-334) and, fused into its
1x1 GEMM, the convex 8x upsampling of ``upsample_flow`` (TV:_utils.py:29-48).

* ``MaskPredictor(in_channels=128, hidden_size=256, multiplier=0.25)``
  - ``forward(x)``: the stock contract, the contiguous (B, 576, h, w) mask, so ``RAFT.forward`` works with the module
    swapped in;
  - ``upsample_flow(flow, hidden_state)``: ``torchvision upsample_flow(flow, self(hidden_state))`` as (B, 2, 8h, 8w)
    fp32, without the mask ever reaching memory.  ``raft_flow`` calls this when the module is swapped in.

The parameter tree is the reference's (``convrelu.0.*``, ``conv.*``), so state dicts load with ``strict=True`` in both
directions.  convrelu (3x3, 128 -> 256 + ReLU) runs on the kernel of ``FlowHead.conv1`` (same shape); the 1x1 is a
tcgen05 GEMM whose epilogue does the softmax over the 9 taps, the convex combination with ``8 * flow`` and the 8x8
pixel shuffle.  16-bit operands, fp32 accumulation, fp32 epilogue.  There is no fallback: CPU tensors, other
configurations (raft_small has no mask predictor) and gradient-carrying calls raise.

Swap it into a torchvision ``raft_large``::

    mp = rc.MaskPredictor(in_channels=128, hidden_size=256, multiplier=model.mask_predictor.multiplier)
    mp.load_state_dict(model.mask_predictor.state_dict())
    model.mask_predictor = mp.to(device)
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch
from torch import Tensor, nn

from . import _cabi
from .corr_block import _param_key
from .motion_encoder import PackedUpdateConv, _dtypes, _Packs, _ptrs, _stream
from .recurrent_block import _DT, _need_cuda, _nhwc

_IN, _HIDDEN, _MASK = 128, 256, 576


class PackedMaskConv:
    """``conv``'s weight as the kernel's 16-bit GEMM operand and its fp32 bias, both in GEMM row order
    (``rdvc_corr_mask_conv_pack_weights``, host), on the device.  Rebuilt when a parameter changes version, address or
    device."""

    def __init__(self, conv: nn.Conv2d, op_dtype: torch.dtype, device):
        lib = _cabi.load()
        w = np.ascontiguousarray(conv.weight.detach().to(torch.float32).cpu().numpy().reshape(_MASK, _HIDDEN))
        b = np.ascontiguousarray(conv.bias.detach().to(torch.float32).cpu().numpy())
        packed = np.zeros(lib.rdvc_corr_mask_conv_packed_weight_bytes() // 2, np.uint16)
        bias = np.zeros(_MASK, np.float32)
        _cabi.check(lib.rdvc_corr_mask_conv_pack_weights(w.ctypes.data, b.ctypes.data, _DT[op_dtype], packed.ctypes.data,
                                                         bias.ctypes.data), "rdvc_corr_mask_conv_pack_weights")
        self.weight = torch.from_numpy(packed.view(np.int16)).to(device)
        self.bias = torch.from_numpy(bias).to(device)
        self.key = _param_key(conv.weight, conv.bias, op_dtype, device)


class MaskPredictor(nn.Module):
    """TV:raft.py:311-334 for raft_large's configuration (in_channels=128, hidden_size=256; any multiplier).  Same
    constructor, parameter names and ``forward`` contract.

    The hidden state is read NCHW or channels_last (the fast path: read in place, a channel slice of a channels_last
    tensor included).  fp32 in -> fp16 operands; autocast -> its dtype as the operands.  Inference only.  Weights are
    packed once per parameter version and device, with the CUDA-graph contract of :class:`MotionEncoder`; the
    multiplier is read at every call (a captured graph keeps the value it was captured with).
    """

    def __init__(self, *, in_channels: int, hidden_size: int, multiplier: float = 0.25):
        from torchvision.ops import Conv2dNormActivation
        super().__init__()
        if in_channels != _IN or hidden_size != _HIDDEN:
            raise ValueError(f"the B200 kernels cover raft_large's mask predictor only (in_channels={_IN}, "
                             f"hidden_size={_HIDDEN}); got in_channels={in_channels}, hidden_size={hidden_size}")
        self.convrelu = Conv2dNormActivation(in_channels, hidden_size, norm_layer=None, kernel_size=3)
        self.conv = nn.Conv2d(hidden_size, 8 * 8 * 9, 1, padding=0)
        self.multiplier = multiplier
        self._packs = _Packs()

    def _check(self, x: Tensor, *more: Tensor):
        _cabi.forward_only("MaskPredictor", x, *more)
        if self.training and torch.is_grad_enabled():
            raise RuntimeError("rdvc_corr_b200.MaskPredictor is forward-only: call .eval() or run under torch.no_grad()")
        _need_cuda(x, *more)
        if x.dim() != 4 or x.shape[1] != _IN:
            raise ValueError(f"the hidden state must be (B, {_IN}, h, w), got {tuple(x.shape)}")

    def forward(self, x: Tensor) -> Tensor:
        """TV:raft.py:331-334: ``multiplier * conv(convrelu(x))``, (B, 576, h, w) contiguous in the activation dtype."""
        self._check(x)
        act, _ = _dtypes(x)
        B, _, h, w = x.shape
        out = torch.empty((B, _MASK, h, w), dtype=act, device=x.device)
        return self._run(x, None, _cabi.RDVC_MASK_OUT_MASK, out)

    def upsample_flow(self, flow: Tensor, hidden_state: Tensor) -> Tensor:
        """TV:_utils.py:29-48 with ``up_mask = self(hidden_state)``: the (B, 2, 8h, 8w) fp32 flow.  ``flow`` is (B, 2,
        h, w), read as fp32 at its own strides."""
        self._check(hidden_state, flow)
        B, _, h, w = hidden_state.shape
        if flow.dim() != 4 or tuple(flow.shape) != (B, 2, h, w):
            raise ValueError(f"flow must be (B, 2, h, w) like the hidden state {tuple(hidden_state.shape)}, "
                             f"got {tuple(flow.shape)}")
        out = torch.empty((B, 2, 8 * h, 8 * w), dtype=torch.float32, device=hidden_state.device)
        return self._run(hidden_state, flow.detach().to(torch.float32), _cabi.RDVC_MASK_OUT_UPSAMPLED, out)

    def _run(self, x: Tensor, flow, out_form: int, out: Tensor) -> Tensor:
        act, op = _dtypes(x)
        dev = x.device
        B, _, h, w = x.shape
        xh, ps = _nhwc(x.detach() if x.dtype == act else x.detach().to(act))
        c1, c2 = self.convrelu[0], self.conv
        packs = [self._packs.get(0, _param_key(c1.weight, c1.bias, op, dev),
                                 lambda: PackedUpdateConv(c1, _cabi.RDVC_UC_FH_CONV1, op, dev)),
                 self._packs.get(1, _param_key(c2.weight, c2.bias, op, dev), lambda: PackedMaskConv(c2, op, dev))]
        lib = _cabi.load()
        ws_bytes = lib.rdvc_corr_mask_predictor_workspace_bytes(B, h, w, _DT[act])
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        fp, fs = (0, None) if flow is None else (flow.data_ptr(), _ptrs(ctypes.c_longlong, list(flow.stride())))
        with torch.cuda.device(dev):
            rc = lib.rdvc_corr_mask_predictor(xh.data_ptr(), ps, _DT[act], B, h, w, _DT[op],
                                              _ptrs(ctypes.c_void_p, [p.weight.data_ptr() for p in packs]),
                                              _ptrs(ctypes.c_void_p, [p.bias.data_ptr() for p in packs]),
                                              float(self.multiplier), fp, fs, out_form, ws.data_ptr(), ws_bytes,
                                              out.data_ptr(), _stream(dev))
        _cabi.check(rc, "rdvc_corr_mask_predictor")
        return out
