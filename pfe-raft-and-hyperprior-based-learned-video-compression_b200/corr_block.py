"""Host-side mirror of the reference's correlation-block interface.

Two surfaces over the same C ABI (``include/rdvc_corr.h``):

* :class:`TVCorrBlock` -- an ``nn.Module`` with torchvision's ``CorrBlock``
  surface (TV:raft.py:337-431): ``build_pyramid(fmap1, fmap2)``,
  ``index_pyramid(centroids_coords)``, ``out_channels``, ``num_levels``,
  ``radius``, ``corr_pyramid``.  Inject it where RDVC builds its RAFT
  (R:codec_processing.py:1289-1291): ``raft_large(weights=..., corr_block=TVCorrBlock())``
  -- ``_raft`` pops the ``corr_block`` kwarg at TV:raft.py:792.
* :class:`CorrBlock` -- the princeton-vl ``core/corr.py`` style façade that the
  reference's ``local`` RAFT backend expects (R:codec_processing.py:64-72):
  ``CorrBlock(fmap1, fmap2, num_levels=4, radius=4)`` builds on construction,
  ``__call__(coords)`` looks up.

PyTorch only provides device memory and the current stream; the arithmetic is
in ``librdvc_corr.so``.  There is no fallback path.
"""
from __future__ import annotations

from typing import List, Optional

import torch
from torch import Tensor, nn

from . import _cabi

_IN_DTYPES = {torch.float32: _cabi.RDVC_DT_F32, torch.bfloat16: _cabi.RDVC_DT_BF16,
              torch.float16: _cabi.RDVC_DT_F16}
_VOL_DTYPES = {torch.float32: _cabi.RDVC_DT_F32, torch.bfloat16: _cabi.RDVC_DT_BF16}


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


ROWMAJOR, TILED = _cabi.RDVC_LAYOUT_ROWMAJOR, _cabi.RDVC_LAYOUT_TILED


def tile_shape(volume_dtype: torch.dtype):
    """(tile_w, tile_h) of the tiled pyramid layout for this storage type (include/rdvc_corr.h)."""
    import ctypes
    tw, th = ctypes.c_int(0), ctypes.c_int(0)
    _cabi.check(_cabi.load().rdvc_corr_tile_shape(_VOL_DTYPES[volume_dtype], ctypes.byref(tw),
                                                  ctypes.byref(th)), "rdvc_corr_tile_shape")
    return tw.value, th.value


class CorrPyramid:
    """Device-resident correlation pyramid: one byte buffer + its geometry and layout
    (``ROWMAJOR`` = torchvision's element order, ``TILED`` = the gather-friendly default)."""

    def __init__(self, B: int, h: int, w: int, num_levels: int, volume_dtype: torch.dtype,
                 buffer: Tensor, layout: int = TILED):
        self.B, self.h, self.w = B, h, w
        self.num_levels = num_levels
        self.volume_dtype = volume_dtype
        self.buffer = buffer  # uint8, 256-byte aligned
        self.layout = layout

    def _tiles(self, l: int):
        hl, wl = self.h >> l, self.w >> l
        if self.layout == ROWMAJOR:
            return hl, wl, 1, 1, hl, wl
        tw, th = tile_shape(self.volume_dtype)
        return hl, wl, tw, th, -(-hl // th) * th, -(-wl // tw) * tw

    def storage(self, l: int) -> Tensor:
        """Level ``l`` as stored: (B*h*w, image_elems) in the pyramid's own layout; for ``TILED`` the
        first padded_h * padded_w elements of a row are the tiles, the rest is padding to 256 bytes."""
        lib = _cabi.load()
        vd = _VOL_DTYPES[self.volume_dtype]
        off = lib.rdvc_corr_level_offset_bytes(self.B, self.h, self.w, l, vd, self.layout)
        img = lib.rdvc_corr_level_image_elems(self.h, self.w, l, vd, self.layout)
        n = self.B * self.h * self.w * img
        es = torch.empty((), dtype=self.volume_dtype).element_size()
        return self.buffer[off: off + n * es].view(self.volume_dtype).view(self.B * self.h * self.w, img)

    def level(self, l: int, rows: Optional[Tensor] = None) -> Tensor:
        """Level ``l`` shaped like torchvision's ``corr_pyramid[l]``: (B*h*w, 1, h >> l, w >> l).
        A view for ``ROWMAJOR``; an un-tiled copy for ``TILED``.  ``rows`` (an index tensor) restricts
        it to those query pixels -- the only way to look at a 4K volume, whose levels do not fit twice."""
        hl, wl, tw, th, hp, wp = self._tiles(l)
        st = self.storage(l)
        if rows is not None:
            st = st[rows]
        if self.layout == ROWMAJOR:
            return st.view(-1, 1, hl, wl)
        img = st[:, : hp * wp].reshape(-1, hp // th, wp // tw, th, tw).permute(0, 1, 3, 2, 4).reshape(-1, hp, wp)
        return img[:, :hl, :wl].unsqueeze(1).contiguous()

    def set_level(self, l: int, value: Tensor) -> None:
        """Store a torchvision-ordered level tensor (B*h*w, [1,] h_l, w_l) in this pyramid's layout."""
        hl, wl, tw, th, hp, wp = self._tiles(l)
        value = value.reshape(-1, hl, wl).to(self.volume_dtype)
        st = self.storage(l)
        if self.layout == ROWMAJOR:
            st.view(-1, hl, wl).copy_(value)
            return
        img = torch.zeros(value.shape[0], hp, wp, dtype=self.volume_dtype, device=st.device)
        img[:, :hl, :wl] = value
        st.zero_()
        st[:, : hp * wp] = img.view(-1, hp // th, th, wp // tw, tw).permute(0, 1, 3, 2, 4).reshape(-1, hp * wp)

    def levels(self) -> List[Tensor]:
        return [self.level(l) for l in range(self.num_levels)]


def _check_fmaps(fmap1: Tensor, fmap2: Tensor, num_levels: int):
    # same checks, same messages as TV:raft.py:368-383
    if fmap1.shape != fmap2.shape:
        raise ValueError(
            f"Input feature maps should have the same shape, instead got {fmap1.shape} (fmap1.shape) != {fmap2.shape} (fmap2.shape)"
        )
    if fmap1.dim() != 4:
        raise ValueError(f"Feature maps should be (B, C, H, W), got {tuple(fmap1.shape)}")
    min_fmap_size = 2 * (2 ** (num_levels - 1))
    if any(fmap_size < min_fmap_size for fmap_size in fmap1.shape[-2:]):
        raise ValueError(
            "Feature maps are too small to be down-sampled by the correlation pyramid. "
            f"H and W of feature maps should be at least {min_fmap_size}; got: {fmap1.shape[-2:]}. "
            "Remember that input images to the model are downsampled by 8, so that means their "
            f"dimensions should be at least 8 * {min_fmap_size} = {8 * min_fmap_size}."
        )
    if not fmap1.is_cuda or not fmap2.is_cuda:
        raise RuntimeError(
            "rdvc_corr_b200 runs on an sm_100 GPU only; got CPU feature maps. There is no CPU fallback."
        )
    if fmap1.dtype != fmap2.dtype or fmap1.dtype not in _IN_DTYPES:
        raise ValueError(f"unsupported feature-map dtypes {fmap1.dtype} / {fmap2.dtype}")
    _cabi.forward_only("build_pyramid", fmap1, fmap2)


def build_pyramid(fmap1: Tensor, fmap2: Tensor, num_levels: int = 4,
                  volume_dtype: torch.dtype = torch.float32,
                  out: Optional[CorrPyramid] = None,
                  workspace: Optional[Tensor] = None, layout: int = TILED) -> CorrPyramid:
    """Correlation volume + pyramid through ``rdvc_corr_build`` on the current stream."""
    _check_fmaps(fmap1, fmap2, num_levels)
    if volume_dtype not in _VOL_DTYPES:
        raise ValueError(f"volume_dtype must be float32 or bfloat16, got {volume_dtype}")
    lib = _cabi.load()
    B, D, h, w = fmap1.shape
    dev = fmap1.device
    f1 = fmap1.contiguous()
    f2 = fmap2.contiguous()
    vd = _VOL_DTYPES[volume_dtype]
    pyr_bytes = lib.rdvc_corr_pyramid_bytes(B, h, w, num_levels, vd, layout)
    ws_bytes = lib.rdvc_corr_workspace_bytes(B, D, h, w)
    with torch.cuda.device(dev):
        if out is not None and out.buffer.numel() >= pyr_bytes and out.buffer.device == dev:
            buf = out.buffer
        else:
            buf = torch.empty(pyr_bytes, dtype=torch.uint8, device=dev)
        if workspace is None or workspace.numel() < ws_bytes or workspace.device != dev:
            workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        rc = lib.rdvc_corr_build(f1.data_ptr(), f2.data_ptr(), B, D, h, w, _IN_DTYPES[f1.dtype],
                                 buf.data_ptr(), vd, layout, num_levels, workspace.data_ptr(),
                                 workspace.numel(), _stream_ptr(dev))
    _cabi.check(rc, "rdvc_corr_build")
    # the workspace is consumed by kernels already enqueued on this stream; torch's
    # caching allocator keeps it stream-ordered when it is dropped here
    pyr = CorrPyramid(B, h, w, num_levels, volume_dtype, buf, layout)
    pyr._workspace = workspace
    return pyr


def _check_coords(pyr: CorrPyramid, coords: Tensor) -> Tensor:
    if coords.dim() != 4 or coords.shape[1] != 2:
        raise ValueError(f"coords should be (B, 2, h, w), got {tuple(coords.shape)}")
    B, _, h, w = coords.shape
    if (B, h, w) != (pyr.B, pyr.h, pyr.w):
        raise ValueError(
            f"coords {tuple(coords.shape)} do not match the pyramid built for (B, h, w) = {(pyr.B, pyr.h, pyr.w)}"
        )
    if not coords.is_cuda:
        raise RuntimeError("rdvc_corr_b200 runs on an sm_100 GPU only; got CPU coords.")
    _cabi.forward_only("index_pyramid", coords)
    return coords.detach().to(torch.float32).contiguous()


def index_pyramid(pyr: CorrPyramid, coords: Tensor, radius: int = 4,
                  out: Optional[Tensor] = None, out_dtype: torch.dtype = torch.float32) -> Tensor:
    """(B, 2, h, w) coords -> (B, L*(2r+1)^2, h, w) through ``rdvc_corr_lookup_ex``: fp32 like torchvision's
    ``index_pyramid``, or fp16 (``out_dtype=torch.float16``: what the consumer casts the features to under the
    reference's default autocast, R:codec_processing.py:1436; tiled pyramids only)."""
    lib = _cabi.load()
    c = _check_coords(pyr, coords)
    B, _, h, w = coords.shape
    dev = coords.device
    if out_dtype not in (torch.float32, torch.float16):
        raise ValueError(f"out_dtype must be float32 or float16, got {out_dtype}")
    S = 2 * radius + 1
    C = pyr.num_levels * S * S
    if out is None:
        out = torch.empty((B, C, h, w), dtype=out_dtype, device=dev)
    elif tuple(out.shape) != (B, C, h, w) or out.dtype != out_dtype or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous {out_dtype} tensor of shape (B, L*(2r+1)^2, h, w)")
    with torch.cuda.device(dev):
        rc = lib.rdvc_corr_lookup_ex(pyr.buffer.data_ptr(), _VOL_DTYPES[pyr.volume_dtype], pyr.layout, c.data_ptr(),
                                     B, h, w, pyr.num_levels, radius, out.data_ptr(), _IN_DTYPES[out_dtype],
                                     _cabi.RDVC_OUT_NCHW, _stream_ptr(dev))
    _cabi.check(rc, "rdvc_corr_lookup_ex")
    return out


_FEAT_DTYPES = {torch.bfloat16: _cabi.RDVC_DT_BF16, torch.float16: _cabi.RDVC_DT_F16}


def feat_pitch(num_levels: int = 4, radius: int = 4) -> int:
    """Elements per K-major feature row (include/rdvc_corr.h: rdvc_corr_feat_pitch)."""
    return int(_cabi.load().rdvc_corr_feat_pitch(num_levels, radius))


def feat_shape(B: int, h: int, w: int, num_levels: int = 4, radius: int = 4):
    """Shape of the K-major feature buffer: (K / 8 chunks, rows = B*h*w rounded up to 8, 8)."""
    lib = _cabi.load()
    return (int(lib.rdvc_corr_feat_pitch(num_levels, radius)) // 8, int(lib.rdvc_corr_feat_rows(B, h, w)), 8)


def index_pyramid_kmajor(pyr: CorrPyramid, coords: Tensor, radius: int = 4, feat_dtype: torch.dtype = torch.bfloat16,
                         out: Optional[Tensor] = None) -> Tensor:
    """The lookup as the K-major 16-bit A operand of the 1x1 convolution (``conv1x1``), chunk-major
    (K/8, rows, 8): ``out[k // 8, m, k % 8]`` is feature k = l*PL + j*S + i (torchvision channel l*S*S + i*S + j,
    PL = S*S rounded up to 8, padding features 0) of query pixel m; rows m >= B*h*w are not written."""
    lib = _cabi.load()
    c = _check_coords(pyr, coords)
    B, _, h, w = coords.shape
    dev = coords.device
    kp = feat_pitch(pyr.num_levels, radius)
    if kp == 0 or feat_dtype not in _FEAT_DTYPES:
        raise ValueError(f"unsupported (levels, radius, feat_dtype) = ({pyr.num_levels}, {radius}, {feat_dtype})")
    shape = feat_shape(B, h, w, pyr.num_levels, radius)
    if out is None:
        out = torch.empty(shape, dtype=feat_dtype, device=dev)
    elif tuple(out.shape) != shape or out.dtype != feat_dtype or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous {feat_dtype} tensor of shape {shape}")
    with torch.cuda.device(dev):
        rc = lib.rdvc_corr_lookup_ex(pyr.buffer.data_ptr(), _VOL_DTYPES[pyr.volume_dtype], pyr.layout, c.data_ptr(),
                                     B, h, w, pyr.num_levels, radius, out.data_ptr(), _FEAT_DTYPES[feat_dtype],
                                     _cabi.RDVC_OUT_KMAJOR, _stream_ptr(dev))
    _cabi.check(rc, "rdvc_corr_lookup_ex")
    return out


class PackedConv1x1:
    """A 1x1 convolution's weight (cout, L*S*S[, 1, 1]) packed for ``rdvc_conv1x1`` (host function
    ``rdvc_conv1x1_pack_weights``: permuted to the lookup's column order, zero padded, 16-bit) + its bias, on the
    device.  Built once per (module, feat_dtype); rebuilt if the parameters change version or device."""

    def __init__(self, weight: Tensor, bias: Optional[Tensor], num_levels: int, radius: int, feat_dtype: torch.dtype,
                 device):
        import ctypes
        import numpy as np
        lib = _cabi.load()
        cout = weight.shape[0]
        w2 = weight.detach().to(torch.float32).reshape(cout, -1).cpu().contiguous().numpy()
        S = 2 * radius + 1
        if w2.shape[1] != num_levels * S * S:
            raise ValueError(f"weight has {w2.shape[1]} input channels, the lookup produces {num_levels * S * S}")
        nbytes = lib.rdvc_conv1x1_packed_weight_bytes(cout, num_levels, radius)
        if nbytes == 0:
            raise ValueError(f"unsupported 1x1 convolution: cout={cout} (multiple of 32, <= 256), levels={num_levels}, radius={radius}")
        packed = np.zeros(nbytes // 2, np.uint16)
        _cabi.check(lib.rdvc_conv1x1_pack_weights(w2.ctypes.data_as(ctypes.c_void_p), cout, num_levels, radius,
                                                  _FEAT_DTYPES[feat_dtype], packed.ctypes.data_as(ctypes.c_void_p)),
                    "rdvc_conv1x1_pack_weights")
        self.cout = cout
        self.feat_dtype = feat_dtype
        self.weight = torch.from_numpy(packed.view(np.int16)).to(device)       # raw 16-bit patterns
        self.bias = None if bias is None else bias.detach().to(torch.float32).to(device).contiguous()
        self.key = _param_key(weight, bias, feat_dtype, device)


class PackedLinear:
    """A 1x1 convolution's weight (cout, cin[, 1, 1]) as plain 16-bit rows on the device (``rdvc_linear_pack_weights``,
    host) + its fp32 bias: the encoder tail's operands.  Rebuilt when the parameters change version or device."""

    def __init__(self, weight: Tensor, bias: Optional[Tensor], op_dtype: torch.dtype, device):
        import ctypes
        import numpy as np
        lib = _cabi.load()
        cout = weight.shape[0]
        w2 = weight.detach().to(torch.float32).reshape(cout, -1).cpu().contiguous().numpy()
        packed = np.zeros(w2.size, np.uint16)
        _cabi.check(lib.rdvc_linear_pack_weights(w2.ctypes.data_as(ctypes.c_void_p), cout, w2.shape[1],
                                                 _FEAT_DTYPES[op_dtype], packed.ctypes.data_as(ctypes.c_void_p)),
                    "rdvc_linear_pack_weights")
        self.cout, self.cin = cout, w2.shape[1]
        self.weight = torch.from_numpy(packed.view(np.int16)).to(device)
        self.bias = None if bias is None else bias.detach().to(torch.float32).to(device).contiguous()
        self.key = _param_key(weight, bias, op_dtype, device)


def _param_key(weight, bias, feat_dtype, device):
    return (weight.data_ptr(), weight._version, None if bias is None else (bias.data_ptr(), bias._version),
            feat_dtype, torch.device(device))


def conv1x1(feat: Tensor, packed: PackedConv1x1, B: int, h: int, w: int, num_levels: int = 4, radius: int = 4,
            relu: bool = True, out_dtype: torch.dtype = torch.float32, out: Optional[Tensor] = None) -> Tensor:
    """(K/8, rows, 8) K-major features (``index_pyramid_kmajor``) -> (B, cout, h, w) = act(W . feat + bias) through
    ``rdvc_conv1x1``."""
    lib = _cabi.load()
    dev = feat.device
    if out is None:
        out = torch.empty((B, packed.cout, h, w), dtype=out_dtype, device=dev)
    with torch.cuda.device(dev):
        rc = lib.rdvc_conv1x1(feat.data_ptr(), _FEAT_DTYPES[feat.dtype], packed.weight.data_ptr(),
                              0 if packed.bias is None else packed.bias.data_ptr(), B, h, w, num_levels, radius,
                              packed.cout, _cabi.RDVC_ACT_RELU if relu else _cabi.RDVC_ACT_NONE, out.data_ptr(),
                              _IN_DTYPES[out.dtype], _stream_ptr(dev))
    _cabi.check(rc, "rdvc_conv1x1")
    return out


class TVCorrBlock(nn.Module):
    """torchvision-surface correlation block backed by librdvc_corr.so.

    Stateful like the original (``self.corr_pyramid``, TV:raft.py:352,389): one
    instance per concurrent RAFT call.
    """

    def __init__(self, *, num_levels: int = 4, radius: int = 4,
                 volume_dtype: torch.dtype = torch.float32, layout: int = TILED):
        super().__init__()
        self.num_levels = num_levels
        self.radius = radius
        self.volume_dtype = volume_dtype
        self.layout = layout
        self.out_channels = num_levels * (2 * radius + 1) ** 2  # TV:raft.py:358
        self._pyr: Optional[CorrPyramid] = None
        self._workspace: Optional[Tensor] = None
        self._levels: Optional[List[Tensor]] = None
        self._packed: Optional[PackedConv1x1] = None     # convcorr1 weights packed for rdvc_conv1x1
        self._packed_tail: Optional[PackedLinear] = None # the feature encoder's final 1x1 convolution, 16-bit rows
        self._workspace_in: Optional[Tensor] = None      # K-major rows of the encoder's 128-channel activations
        self._feat: Optional[Tensor] = None              # K-major feature rows between the two launches

    @property
    def corr_pyramid(self) -> List[Tensor]:
        """torchvision's attribute (TV:raft.py:352,389): the levels as (B*h*w, 1, h_l, w_l) tensors.
        RAFT itself never reads it; with the tiled layout it is materialised on first access."""
        if self._pyr is None:
            return [torch.tensor(0)]
        if self._levels is None:
            self._levels = self._pyr.levels()
        return self._levels

    def build_pyramid(self, fmap1: Tensor, fmap2: Tensor) -> None:
        self._pyr = build_pyramid(fmap1, fmap2, self.num_levels, self.volume_dtype,
                                  out=self._pyr, workspace=self._workspace, layout=self.layout)
        self._workspace = self._pyr._workspace
        self._levels = None

    def index_pyramid(self, centroids_coords: Tensor) -> Tensor:
        if self._pyr is None:
            raise RuntimeError("index_pyramid called before build_pyramid")
        corr_features = index_pyramid(self._pyr, centroids_coords, self.radius)
        batch_size, _, h, w = centroids_coords.shape
        expected_output_shape = (batch_size, self.out_channels, h, w)
        if corr_features.shape != expected_output_shape:  # TV:raft.py:416-420
            raise ValueError(
                f"Output shape of index pyramid is incorrect. Should be {expected_output_shape}, got {corr_features.shape}"
            )
        return corr_features

    def build_pyramid_from_encoder(self, x1: Tensor, x2: Tensor, weight: Tensor, bias: Optional[Tensor] = None) -> None:
        """``build_pyramid(conv(x1), conv(x2))`` for the feature encoder's final 1x1 convolution ``conv`` (TV:raft.py:139,
        150; ``weight``: (256, 128[, 1, 1])) WITHOUT materialising the fp32 feature maps: the 128-channel activations are
        repacked K-major (``rdvc_corr_pack``), a tcgen05 GEMM turns every packed row into the build's 256-channel operand
        row (``rdvc_corr_encoder_tail``; a 1x1 convolution commutes with the transpose and the mean pooling), and the
        build multiplies those rows (``rdvc_corr_build_packed``).  16-bit operands (bf16; fp16 for fp16 activations),
        fp32 accumulation, 16-bit operand rows: feature rows within one 16-bit ulp of the rounded stock feature maps."""
        _check_fmaps(x1, x2, self.num_levels)
        lib = _cabi.load()
        B, Din, h, w = x1.shape
        Dout = weight.shape[0]
        dev = x1.device
        op_dtype = torch.float16 if x1.dtype == torch.float16 else torch.bfloat16
        key = _param_key(weight, bias, op_dtype, dev)
        if self._packed_tail is None or self._packed_tail.key != key:
            self._packed_tail = PackedLinear(weight, bias, op_dtype, dev)
        if self._packed_tail.cin != Din:
            raise ValueError(f"weight expects {self._packed_tail.cin} input channels, the activations have {Din}")
        vd = _VOL_DTYPES[self.volume_dtype]
        pyr_bytes = lib.rdvc_corr_pyramid_bytes(B, h, w, self.num_levels, vd, self.layout)
        ws_in_bytes = lib.rdvc_corr_workspace_bytes(B, Din, h, w)
        ws_out_bytes = lib.rdvc_corr_workspace_bytes(B, Dout, h, w)
        a, b = x1.contiguous(), x2.contiguous()
        with torch.cuda.device(dev):
            if self._pyr is not None and self._pyr.buffer.numel() >= pyr_bytes and self._pyr.buffer.device == dev:
                buf = self._pyr.buffer
            else:
                buf = torch.empty(pyr_bytes, dtype=torch.uint8, device=dev)
            if self._workspace is None or self._workspace.numel() < ws_out_bytes or self._workspace.device != dev:
                self._workspace = torch.empty(ws_out_bytes, dtype=torch.uint8, device=dev)
            if self._workspace_in is None or self._workspace_in.numel() < ws_in_bytes or self._workspace_in.device != dev:
                self._workspace_in = torch.empty(ws_in_bytes, dtype=torch.uint8, device=dev)
            st = _stream_ptr(dev)
            _cabi.check(lib.rdvc_corr_pack(a.data_ptr(), b.data_ptr(), B, Din, h, w, _IN_DTYPES[a.dtype], vd, self.layout,
                                           self.num_levels, self._workspace_in.data_ptr(), self._workspace_in.numel(), st),
                        "rdvc_corr_pack")
            pt = self._packed_tail
            _cabi.check(lib.rdvc_corr_encoder_tail(self._workspace_in.data_ptr(), self._workspace_in.numel(), Din,
                                                   pt.weight.data_ptr(), 0 if pt.bias is None else pt.bias.data_ptr(), Dout,
                                                   B, h, w, _FEAT_DTYPES[op_dtype], vd, self.layout, self.num_levels,
                                                   self._workspace.data_ptr(), self._workspace.numel(), st),
                        "rdvc_corr_encoder_tail")
            _cabi.check(lib.rdvc_corr_build_packed(B, Dout, h, w, _FEAT_DTYPES[op_dtype], buf.data_ptr(), vd, self.layout,
                                                   self.num_levels, self._workspace.data_ptr(), self._workspace.numel(), st),
                        "rdvc_corr_build_packed")
        self._pyr = CorrPyramid(B, h, w, self.num_levels, self.volume_dtype, buf, self.layout)
        self._pyr._workspace = self._workspace
        self._levels = None

    def index_pyramid_convcorr1(self, centroids_coords: Tensor, weight: Tensor, bias: Optional[Tensor] = None,
                                relu: bool = True, out_dtype: Optional[torch.dtype] = None,
                                feat_dtype: Optional[torch.dtype] = None, nhwc: bool = False) -> Tensor:
        """``relu(conv1x1(index_pyramid(coords), weight, bias))`` -- the lookup fused with
        ``MotionEncoder.convcorr1`` (TV:raft.py:185,202) through ``rdvc_corr_lookup_conv1x1``: the (B, 324, h, w)
        fp32 lookup tensor is never written.  ``weight``: (cout, L*S*S[, 1, 1]) in torchvision's channel order.
        16-bit operands, fp32 accumulation: fp16 by default (11-bit mantissa: within 2e-3 of the stock fp32
        convolution, and exactly what the stock path multiplies under the reference's default fp16 autocast; the
        conversion saturates at +-65504, three orders above any correlation value RAFT's features produce),
        ``feat_dtype=torch.bfloat16`` trades mantissa for range (within 1e-2).  The result is fp32, or the autocast
        dtype when autocast is on.

        ``nhwc=True``: the result is a channels_last (B, cout, h, w) tensor in ``feat_dtype``, written by the GEMM's
        epilogue straight from the accumulator (``rdvc_corr_lookup_conv1x1_ex``), bit-identical to the default output
        rounded to that dtype; it is what ``MotionEncoder.forward_fused`` reads in place."""
        if self._pyr is None:
            raise RuntimeError("index_pyramid_convcorr1 called before build_pyramid")
        pyr = self._pyr
        c = _check_coords(pyr, centroids_coords)
        B, _, h, w = centroids_coords.shape
        dev = centroids_coords.device
        amp = torch.is_autocast_enabled("cuda")
        if out_dtype is None:
            out_dtype = torch.get_autocast_dtype("cuda") if amp else torch.float32
        if feat_dtype is None:
            feat_dtype = torch.bfloat16 if (amp and torch.get_autocast_dtype("cuda") == torch.bfloat16) else torch.float16
        key = _param_key(weight, bias, feat_dtype, dev)
        if self._packed is None or self._packed.key != key:
            self._packed = PackedConv1x1(weight, bias, self.num_levels, self.radius, feat_dtype, dev)
        shape = feat_shape(B, h, w, self.num_levels, self.radius)
        if self._feat is None or tuple(self._feat.shape) != shape or self._feat.dtype != feat_dtype or self._feat.device != dev:
            self._feat = torch.zeros(shape, dtype=feat_dtype, device=dev)
        lib = _cabi.load()
        if nhwc:
            out = torch.empty((B, h, w, self._packed.cout), dtype=feat_dtype, device=dev)
            with torch.cuda.device(dev):
                rc = lib.rdvc_corr_lookup_conv1x1_ex(
                    pyr.buffer.data_ptr(), _VOL_DTYPES[pyr.volume_dtype], pyr.layout, c.data_ptr(), B, h, w,
                    self.num_levels, self.radius, self._packed.weight.data_ptr(),
                    0 if self._packed.bias is None else self._packed.bias.data_ptr(), self._packed.cout,
                    _cabi.RDVC_ACT_RELU if relu else _cabi.RDVC_ACT_NONE, _FEAT_DTYPES[feat_dtype], self._feat.data_ptr(),
                    self._feat.numel() * 2, out.data_ptr(), _FEAT_DTYPES[feat_dtype], self._packed.cout, _stream_ptr(dev))
            _cabi.check(rc, "rdvc_corr_lookup_conv1x1_ex")
            return out.permute(0, 3, 1, 2)
        out = torch.empty((B, self._packed.cout, h, w), dtype=out_dtype, device=dev)
        with torch.cuda.device(dev):
            rc = lib.rdvc_corr_lookup_conv1x1(
                pyr.buffer.data_ptr(), _VOL_DTYPES[pyr.volume_dtype], pyr.layout, c.data_ptr(), B, h, w, self.num_levels,
                self.radius, self._packed.weight.data_ptr(), 0 if self._packed.bias is None else self._packed.bias.data_ptr(),
                self._packed.cout, _cabi.RDVC_ACT_RELU if relu else _cabi.RDVC_ACT_NONE, _FEAT_DTYPES[feat_dtype],
                self._feat.data_ptr(), self._feat.numel() * 2, out.data_ptr(), _IN_DTYPES[out_dtype], _stream_ptr(dev))
        _cabi.check(rc, "rdvc_corr_lookup_conv1x1")
        return out

    def release(self) -> None:
        """Drop the pyramid (5.7 GB at 1080p fp32) back to torch's allocator."""
        self._pyr = None
        self._workspace = None
        self._levels = None
        self._feat = None
        self._workspace_in = None


class CorrBlock:
    """princeton-vl style façade: ``CorrBlock(fmap1, fmap2, num_levels, radius)(coords)``.

    ``coords`` is (B, 2, h, w) with channel 0 = x, channel 1 = y, as produced by
    ``coords_grid`` in that code base; the result is (B, L*(2r+1)^2, h, w) fp32.
    """

    def __init__(self, fmap1: Tensor, fmap2: Tensor, num_levels: int = 4, radius: int = 4,
                 volume_dtype: torch.dtype = torch.float32, layout: int = TILED):
        self.num_levels = num_levels
        self.radius = radius
        self.pyramid = build_pyramid(fmap1, fmap2, num_levels, volume_dtype, layout=layout)

    @property
    def corr_pyramid(self) -> List[Tensor]:
        return self.pyramid.levels()

    def __call__(self, coords: Tensor) -> Tensor:
        return index_pyramid(self.pyramid, coords, self.radius)
