"""B200 drop-in for RAFT's recurrent block: torchvision's ``RecurrentBlock`` (TV:raft.py:238-270), the SepConvGRU every
refinement iteration runs, as fused tcgen05 convolutions.

* ``RecurrentBlock(input_size=256, hidden_size=128)`` with ``forward(h, x)``      TV:raft.py:232-270

The module has the reference's constructor and parameter tree (``convgru1.convz.weight`` ... ``convgru2.convq.bias``),
so ``load_state_dict(model.update_block.recurrent_block.state_dict())`` works with ``strict=True``.  Each ConvGRU
(TV:raft.py:214-229) runs as two launches behind ``rdvc_corr_convgru``: conv z|r + bias + sigmoid writing z and r*h, then
conv q + bias + tanh + the blend ``(1 - z) h + z q``; ``x`` is read in place as two 128-channel parts (context, motion
features), nothing is concatenated.  16-bit operands, fp32 accumulation and epilogue.  There is no fallback: CPU
tensors, other configurations (raft_small's 3x3 GRU included) and gradient-carrying calls raise.

Swap it into a torchvision RAFT::

    rb = rc.RecurrentBlock(input_size=256, hidden_size=128)
    rb.load_state_dict(model.update_block.recurrent_block.state_dict())
    model.update_block.recurrent_block = rb.to(device)
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional, Tuple

import numpy as np
import torch
from torch import Tensor, nn

from . import _cabi
from .corr_block import _param_key

_HIDDEN, _INPUT = 128, 256
_KERNELS = ((1, 5), (5, 1))
_PADDING = ((0, 2), (2, 0))
_AXES = (_cabi.RDVC_GRU_HORIZONTAL, _cabi.RDVC_GRU_VERTICAL)
_DT = {torch.float32: _cabi.RDVC_DT_F32, torch.float16: _cabi.RDVC_DT_F16, torch.bfloat16: _cabi.RDVC_DT_BF16}


class _ConvGRU(nn.Module):
    """Parameter container with the key names of torchvision's ConvGRU (TV:raft.py:214-221)."""

    def __init__(self, input_size: int, hidden_size: int, kernel_size, padding):
        super().__init__()
        self.convz = nn.Conv2d(hidden_size + input_size, hidden_size, kernel_size=kernel_size, padding=padding)
        self.convr = nn.Conv2d(hidden_size + input_size, hidden_size, kernel_size=kernel_size, padding=padding)
        self.convq = nn.Conv2d(hidden_size + input_size, hidden_size, kernel_size=kernel_size, padding=padding)


class PackedConvGRU:
    """One ConvGRU's weights as the kernels' 16-bit tap matrices (``rdvc_corr_convgru_pack_weights``, host) + its three fp32
    biases, on the device.  Rebuilt when a parameter changes version, address or device."""

    def __init__(self, gru: _ConvGRU, op_dtype: torch.dtype, device):
        lib = _cabi.load()
        ws = [np.ascontiguousarray(c.weight.detach().to(torch.float32).cpu().numpy()) for c in (gru.convz, gru.convr, gru.convq)]
        packed = np.zeros(lib.rdvc_corr_convgru_packed_weight_bytes() // 2, np.uint16)
        _cabi.check(lib.rdvc_corr_convgru_pack_weights(ws[0].ctypes.data, ws[1].ctypes.data, ws[2].ctypes.data, _DT[op_dtype],
                                                  packed.ctypes.data), "rdvc_corr_convgru_pack_weights")
        self.weight = torch.from_numpy(packed.view(np.int16)).to(device)
        self.bias_z, self.bias_r, self.bias_q = (c.bias.detach().to(torch.float32).to(device).contiguous()
                                                 for c in (gru.convz, gru.convr, gru.convq))
        self.key = _gru_key(gru, op_dtype, device)


def _gru_key(gru: _ConvGRU, op_dtype, device):
    return tuple(_param_key(c.weight, c.bias, op_dtype, device) for c in (gru.convz, gru.convr, gru.convq))


def _need_cuda(*ts: Tensor):
    if any(not t.is_cuda for t in ts):
        raise RuntimeError("rdvc_corr_b200 runs on an sm_100 GPU only; got CPU tensors. There is no CPU fallback.")


def _nhwc(t: Tensor) -> Tuple[Tensor, int]:
    """(B, C, H, W) tensor -> (a tensor whose memory is NHWC with channel stride 1, its pixel stride in elements).
    A channels_last tensor or a channel slice of one is used in place; anything else is copied once."""
    B, C, H, W = t.shape
    sb, sc, sh, sw = t.stride()
    es = t.element_size()
    if (W > 1 and sc == 1 and sw >= C and (sw * es) % 16 == 0 and (H == 1 or sh == W * sw)
            and (B == 1 or sb == H * W * sw) and t.data_ptr() % 16 == 0):
        return t, sw
    return t.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2), C


class RecurrentBlock(nn.Module):
    """TV:raft.py:232-270 for raft_large's configuration.  Same constructor, parameter names and ``forward`` contract.

    ``forward(h, x)``: ``h`` (B, 128, H, W), ``x`` (B, 256, H, W) = [context | motion features], NCHW or channels_last
    (the fast path; channel slices of channels_last tensors are read in place).  The result has ``h``'s memory format
    and dtype: fp32 in, fp32 out (operands rounded to fp16 -- the stock fp32 path multiplies in TF32, the same 10-bit
    mantissa); fp16 / bf16 inputs or autocast give that dtype (operands in it).  Inference only.

    Weights are packed once per parameter version and device.  A CUDA graph captured through this module replays the
    weights that were packed when it was captured: after changing parameters in place, run the module eagerly (it
    re-packs) and re-capture the graph -- the same contract as the library's fused 1x1 convolution weights.  Moving
    the parameters (``.to(...)``, ``load_state_dict`` into a moved module) re-packs on the next call.
    """

    def __init__(self, *, input_size: int, hidden_size: int, kernel_size=_KERNELS, padding=_PADDING):
        super().__init__()
        ks = tuple(tuple(k) if isinstance(k, (tuple, list)) else (k, k) for k in kernel_size)
        pd = tuple(tuple(p) if isinstance(p, (tuple, list)) else (p, p) for p in padding)
        if input_size != _INPUT or hidden_size != _HIDDEN or ks != _KERNELS or pd != _PADDING:
            raise ValueError(
                f"the B200 kernels cover raft_large's recurrent block only (input_size={_INPUT}, hidden_size={_HIDDEN}, "
                f"kernel_size={_KERNELS}, padding={_PADDING}); got input_size={input_size}, hidden_size={hidden_size}, "
                f"kernel_size={kernel_size}, padding={padding}")
        self.convgru1 = _ConvGRU(input_size, hidden_size, _KERNELS[0], _PADDING[0])
        self.convgru2 = _ConvGRU(input_size, hidden_size, _KERNELS[1], _PADDING[1])
        self.hidden_size = hidden_size
        self._packed: Dict[int, PackedConvGRU] = {}

    def _pack(self, i: int, gru: _ConvGRU, op_dtype, device) -> PackedConvGRU:
        pk = self._packed.get(i)
        if pk is None or pk.key != _gru_key(gru, op_dtype, device):
            pk = self._packed[i] = PackedConvGRU(gru, op_dtype, device)
        return pk

    def forward(self, h: Tensor, x: Tensor) -> Tensor:
        if x.dim() != 4 or x.shape[1] != _INPUT:
            raise ValueError(f"x must be (B, {_INPUT}, H, W), got {tuple(x.shape)}")
        return self.forward_parts(h, x[:, :_HIDDEN], x[:, _HIDDEN:])

    def forward_parts(self, h: Tensor, context: Tensor, motion: Tensor) -> Tensor:
        """``forward(h, torch.cat([context, motion], 1))`` without the concatenation: each part is read in place."""
        _cabi.forward_only("RecurrentBlock", h, context, motion)
        if self.training and torch.is_grad_enabled():
            raise RuntimeError("rdvc_corr_b200.RecurrentBlock is forward-only: call .eval() or run under torch.no_grad()")
        _need_cuda(h, context, motion)
        if h.dim() != 4 or h.shape[1] != _HIDDEN:
            raise ValueError(f"h must be (B, {_HIDDEN}, H, W), got {tuple(h.shape)}")
        for t in (context, motion):
            if t.shape != h.shape:
                raise ValueError(f"x parts must be (B, {_HIDDEN}, H, W) like h {tuple(h.shape)}, got {tuple(t.shape)}")
        if torch.is_autocast_enabled("cuda"):
            act = torch.get_autocast_dtype("cuda")
        else:
            act = h.dtype
        if act not in _DT:
            raise ValueError(f"unsupported dtype {act}")
        op = torch.float16 if act == torch.float32 else act
        dev = h.device
        channels_last = not h.is_contiguous()
        parts = [_nhwc(t.detach() if t.dtype == act else t.detach().to(act)) for t in (h, context, motion)]
        (c, cps), (m, mps) = parts[1], parts[2]
        B, _, H, W = h.shape
        lib = _cabi.load()
        ws_bytes = lib.rdvc_corr_convgru_workspace_bytes(B, H, W, _DT[act])
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        cur, cps_h = parts[0]
        with torch.cuda.device(dev):
            st = torch.cuda.current_stream(dev).cuda_stream
            for i, gru in enumerate((self.convgru1, self.convgru2)):
                pk = self._pack(i, gru, op, dev)
                out = torch.empty((B, H, W, _HIDDEN), dtype=act, device=dev)
                rc = lib.rdvc_corr_convgru(cur.data_ptr(), cps_h, c.data_ptr(), cps, m.data_ptr(), mps, _DT[act], _DT[op],
                                      _AXES[i], B, H, W, pk.weight.data_ptr(), pk.bias_z.data_ptr(), pk.bias_r.data_ptr(),
                                      pk.bias_q.data_ptr(), ws.data_ptr(), ws_bytes, out.data_ptr(), st)
                _cabi.check(rc, "rdvc_corr_convgru")
                cur, cps_h = out.permute(0, 3, 1, 2), _HIDDEN
        return cur if channels_last else cur.contiguous()
