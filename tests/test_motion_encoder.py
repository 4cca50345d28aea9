"""RAFT's motion encoder and flow head (torchvision MotionEncoder / FlowHead, TV:raft.py:171-211, 272-285) as NHWC
convolutions, and the 1x1 GEMM's NHWC output.

CPU part (-m "not gpu"): parameter trees and strict state_dict round trips against torchvision's classes, the refused
configurations, each layer's host-packed weights evaluated the way the kernels walk them, the C ABI's argument errors
and size queries, the module refusals (the kernels' SASS and registers: test_tap_conv.py).
GPU part (-m gpu): every layer against an fp64 evaluation with the kernels' rounding points, input forms, whole modules
against the stock ones, the 1x1 NHWC output, the flow channels and untouched channel slices, determinism / streams /
graphs / re-packing, and RAFT end to end.

Rounding points of the kernels (u = unit roundoff of the output type: 2^-11 fp16, 2^-8 bf16, 0 fp32):
  input activations and weights rounded to the 16-bit operand type; fp32 accumulation (K <= 9 x 256 = 2304); bias
  and ReLU in fp32; the result rounded once to the output type.
Tolerances (absolute, per element):
  * one layer vs fp64 with the same operand rounding, result unrounded ... u |ref| + 2e-4
      the final rounding is within u |ref| (one rounding of a value within 2e-4 of ref); fp32 sums of K <= 2304
      products of O(1) terms are within sqrt(K) 2^-24 x O(1) ~ 3e-6 of the exact sum, 2e-4 leaves room for an
      accumulation order that is not the best case.
  * whole module vs the fp64 chain (each layer's result rounded to the operand type before the next) ... twice the
      layer tolerance + 2 u_op max |ref|: an intermediate on a rounding boundary may round the other way in the kernel.
  * vs the stock modules (cuDNN, TF32 off for fp32) ........ 2e-2 (fp32, fp16), 1e-1 (bf16): the stock fp32 path keeps
      fp32 operands, the autocast path rounds every intermediate the same way but sums in another order; an
      intermediate that lands on a rounding boundary moves the next layer by one ulp of its input (2^-8 |x| for bf16).
  * the flow channels 126-127 .............................. exact: flow.to(dtype).
  * RAFT flow vs stock torchvision, mean EPE ................ < 0.05 px
"""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import rdvc_corr_b200 as rc
from rdvc_corr_b200 import _cabi
from rdvc_corr_b200.motion_encoder import PackedUpdateConv

U = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8, torch.float32: 0.0}
TOL_STOCK = {torch.float32: 2e-2, torch.float16: 2e-2, torch.bfloat16: 1e-1}
TOL_EPE = 0.05
SHAPES = [(1, 46, 80), (2, 18, 22), (1, 17, 19), (1, 33, 47), (9, 136, 240)]
DTYPES = [torch.float32, torch.float16, torch.bfloat16]
ADT = {torch.float32: rc.RDVC_DT_F32, torch.float16: rc.RDVC_DT_F16, torch.bfloat16: rc.RDVC_DT_BF16}
# layer -> (cin, cout, kernel, GEMM width N)
LAYERS = {_cabi.RDVC_UC_CONVCORR2: (256, 192, 3, 192), _cabi.RDVC_UC_CONVFLOW1: (2, 128, 7, 128),
          _cabi.RDVC_UC_CONVFLOW2: (128, 64, 3, 64), _cabi.RDVC_UC_CONV: (256, 126, 3, 128),
          _cabi.RDVC_UC_FH_CONV1: (128, 256, 3, 256), _cabi.RDVC_UC_FH_CONV2: (256, 2, 3, 16)}


@pytest.fixture(scope="module")
def lib():
    rc._build.build()
    return rc._cabi.load()


def tv_me():
    from torchvision.models.optical_flow.raft import MotionEncoder
    return MotionEncoder(in_channels_corr=324, corr_layers=(256, 192), flow_layers=(128, 64), out_channels=128)


def tv_fh():
    from torchvision.models.optical_flow.raft import FlowHead
    return FlowHead(in_channels=128, hidden_size=256)


def seeded(seed=0):
    torch.manual_seed(seed)
    return rc.MotionEncoder(in_channels_corr=324), rc.FlowHead(in_channels=128, hidden_size=256)


def conv_of(me, fh, layer):
    return {_cabi.RDVC_UC_CONVCORR2: me.convcorr2[0], _cabi.RDVC_UC_CONVFLOW1: me.convflow1[0],
            _cabi.RDVC_UC_CONVFLOW2: me.convflow2[0], _cabi.RDVC_UC_CONV: me.conv[0], _cabi.RDVC_UC_FH_CONV1: fh.conv1,
            _cabi.RDVC_UC_FH_CONV2: fh.conv2}[layer]


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize("which", ["me", "fh"])
def test_state_dict_matches_torchvision(which):
    ours = seeded()[0 if which == "me" else 1]
    tv, tv2 = (tv_me(), tv_me()) if which == "me" else (tv_fh(), tv_fh())
    assert list(ours.state_dict().keys()) == list(tv.state_dict().keys())
    assert all(ours.state_dict()[k].shape == v.shape for k, v in tv.state_dict().items())
    ours.load_state_dict(tv.state_dict(), strict=True)
    tv2.load_state_dict(ours.state_dict(), strict=True)
    assert all(torch.equal(tv2.state_dict()[k], v) for k, v in tv.state_dict().items())


def test_convcorr1_is_still_fusable():
    from rdvc_corr_b200.raft_flow import _can_fuse_convcorr1

    class M:
        pass
    m = M()
    m.update_block = M()
    m.update_block.motion_encoder = seeded()[0]
    assert _can_fuse_convcorr1(m)


@pytest.mark.parametrize("kw", [
    dict(in_channels_corr=324, corr_layers=(96,), flow_layers=(64, 32), out_channels=82),     # raft_small's
    dict(in_channels_corr=196, corr_layers=(256, 192), flow_layers=(128, 64), out_channels=128),
    dict(in_channels_corr=324, corr_layers=(256, 128), flow_layers=(128, 64), out_channels=128),
    dict(in_channels_corr=324, corr_layers=(256, 192), flow_layers=(128, 64), out_channels=130),
])
def test_unsupported_motion_encoders_raise(kw):
    with pytest.raises(ValueError):
        rc.MotionEncoder(**kw)


@pytest.mark.parametrize("kw", [dict(in_channels=96, hidden_size=128), dict(in_channels=128, hidden_size=128),
                                dict(in_channels=256, hidden_size=256)])
def test_unsupported_flow_heads_raise(kw):
    with pytest.raises(ValueError):
        rc.FlowHead(**kw)


def _packed(lib, layer, weight, op):
    nbytes = lib.rdvc_corr_update_conv_packed_weight_bytes(layer)
    packed = np.zeros(nbytes // 2, np.uint16)
    w = np.ascontiguousarray(weight.detach().numpy().astype(np.float32))
    _cabi.check(lib.rdvc_corr_update_conv_pack_weights(layer, w.ctypes.data, ADT[op], packed.ctypes.data), "pack")
    return torch.from_numpy(packed.view(np.int16)).view(op).double().numpy()


@pytest.mark.parametrize("op", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("layer", sorted(LAYERS))
def test_packed_weights_reproduce_the_convolution(lib, layer, op):
    """The packed operand, walked the way the kernels walk it, is the convolution (fp64, operands rounded)."""
    cin, cout, k, n = LAYERS[layer]
    torch.manual_seed(10 + layer)
    conv = torch.nn.Conv2d(cin, cout, k, padding=k // 2)
    p = _packed(lib, layer, conv.weight, op)
    a = torch.randn(2, cin, 9, 11).to(op).double()
    want = F.conv2d(a, conv.weight.detach().to(op).double(), padding=k // 2).numpy()
    B, _, H, W = a.shape
    ap = np.pad(a.numpy(), ((0, 0), (0, 0), (k // 2, k // 2), (k // 2, k // 2)))
    if layer == _cabi.RDVC_UC_CONVFLOW1:
        assert p.size == 128 * 128
        pm = p.reshape(128, 128)                          # [n][(ky * 7 + kx) * 2 + ci], K = 98 padded to 128
        assert not pm[cout:].any() and not pm[:, 98:].any()
        col = np.zeros((B, H, W, 128))
        for ky in range(7):
            for kx in range(7):
                for ci in range(2):
                    col[..., (ky * 7 + kx) * 2 + ci] = ap[:, ci, ky:ky + H, kx:kx + W]
        got = np.einsum("bhwk,nk->bnhw", col, pm)
    else:
        kb = cin // 64
        assert p.size == kb * 9 * n * 64
        pm = p.reshape(kb, 9, n, 64)                     # [k-block][dy * 3 + dx][N][64]
        assert not pm[:, :, cout:].any()
        got = np.zeros((B, n, H, W))
        for b in range(kb):
            for dy in range(3):
                for dx in range(3):
                    got += np.einsum("bchw,nc->bnhw", ap[:, b * 64:(b + 1) * 64, dy:dy + H, dx:dx + W], pm[b, dy * 3 + dx])
    assert not got[:, cout:].any()
    assert np.abs(got[:, :cout] - want).max() <= 1e-9 * np.abs(want).max()


def test_cabi_argument_errors(lib):
    A = 1 << 20           # a 16-byte aligned fake device address: every call below fails its checks before any access
    fs = (ctypes.c_longlong * 4)(2 * 64, 64, 8, 1)
    for layer, (cin, cout, k, n) in LAYERS.items():
        want = (128 * 128 if layer == _cabi.RDVC_UC_CONVFLOW1 else cin // 64 * 9 * n * 64) * 2
        assert lib.rdvc_corr_update_conv_packed_weight_bytes(layer) == want
    assert lib.rdvc_corr_update_conv_packed_weight_bytes(6) == 0 and lib.rdvc_corr_update_conv_packed_weight_bytes(-1) == 0

    def conv(**kw):
        a = dict(layer=_cabi.RDVC_UC_CONVCORR2, x=A, xps=256, f=A, fs=fs, B=1, H=8, W=8, op=rc.RDVC_DT_F16, w=A, b=A,
                 out=2 * A, ops=256, odt=rc.RDVC_DT_F16)
        a.update(kw)
        return lib.rdvc_corr_update_conv(a["layer"], a["x"], a["xps"], a["f"], a["fs"], a["B"], a["H"], a["W"], a["op"], a["w"],
                                    a["b"], a["out"], a["ops"], a["odt"], None)
    assert conv(layer=6) == -5 and conv(layer=-1) == -5
    assert conv(x=None) == -1 and conv(w=None) == -1 and conv(b=None) == -1 and conv(out=None) == -1
    assert conv(layer=_cabi.RDVC_UC_CONV, f=None) == -1 and conv(layer=_cabi.RDVC_UC_CONVFLOW1, fs=None) == -1
    assert conv(B=0) == -2 and conv(H=-1) == -2
    assert conv(op=rc.RDVC_DT_F32) == -4 and conv(odt=rc.RDVC_DT_F32) == -4 and conv(odt=rc.RDVC_DT_BF16) == -4
    assert conv(xps=128) == -5 and conv(ops=128) == -5
    assert conv(xps=260) == -7 and conv(x=A + 8) == -7 and conv(out=A + 2) == -7 and conv(w=A + 4) == -7
    assert conv(layer=_cabi.RDVC_UC_CONV, odt=rc.RDVC_DT_F32, ops=130) == -7
    assert lib.rdvc_corr_motion_encoder_workspace_bytes(1, 8, 8) >= 64 * (128 + 256) * 2
    assert lib.rdvc_corr_motion_encoder_workspace_bytes(0, 8, 8) == 0
    assert lib.rdvc_corr_flow_head_workspace_bytes(1, 8, 8, rc.RDVC_DT_F32) > lib.rdvc_corr_flow_head_workspace_bytes(1, 8, 8, rc.RDVC_DT_F16) > 0
    assert lib.rdvc_corr_flow_head_workspace_bytes(1, 8, 8, 7) == 0 and lib.rdvc_corr_flow_head_workspace_bytes(1, 0, 8, rc.RDVC_DT_F16) == 0

    ptr4 = (ctypes.c_void_p * 4)(A, A, A, A)
    me_ws = lib.rdvc_corr_motion_encoder_workspace_bytes(1, 8, 8)

    def me(**kw):
        a = dict(c1=A, ps=256, f=A, fs=fs, B=1, H=8, W=8, op=rc.RDVC_DT_F16, w=ptr4, b=ptr4, ws=A, wsb=me_ws, out=2 * A,
                 ops=128, odt=rc.RDVC_DT_F32)
        a.update(kw)
        return lib.rdvc_corr_motion_encoder(a["c1"], a["ps"], a["f"], a["fs"], a["B"], a["H"], a["W"], a["op"], a["w"], a["b"],
                                       a["ws"], a["wsb"], a["out"], a["ops"], a["odt"], None)
    assert me(c1=None) == -1 and me(w=None) == -1 and me(w=(ctypes.c_void_p * 4)(A, A, None, A)) == -1
    assert me(B=0) == -2 and me(wsb=me_ws - 1) == -6 and me(ws=A + 16) == -7

    ptr2 = (ctypes.c_void_p * 2)(A, A)
    fh_ws = lib.rdvc_corr_flow_head_workspace_bytes(1, 8, 8, rc.RDVC_DT_F16)

    def fh(**kw):
        a = dict(h=A, ps=128, act=rc.RDVC_DT_F16, B=1, H=8, W=8, op=rc.RDVC_DT_F16, w=ptr2, b=ptr2, ws=A, wsb=fh_ws,
                 out=2 * A)
        a.update(kw)
        return lib.rdvc_corr_flow_head(a["h"], a["ps"], a["act"], a["B"], a["H"], a["W"], a["op"], a["w"], a["b"], a["ws"],
                                  a["wsb"], a["out"], None)
    assert fh(h=None) == -1 and fh(b=(ctypes.c_void_p * 2)(A, None)) == -1
    assert fh(W=0) == -2 and fh(act=9) == -4 and fh(act=rc.RDVC_DT_BF16) == -4 and fh(op=rc.RDVC_DT_F32) == -4
    assert fh(ps=64) == -5 and fh(ps=132) == -7 and fh(wsb=fh_ws - 1) == -6
    assert fh(act=rc.RDVC_DT_F32, wsb=fh_ws) == -6                      # fp32 h needs the larger workspace
    for rcode in (fh(h=None), me(B=0), conv(layer=9)):
        assert rcode < 0 and _cabi.last_error()
    w = np.zeros(4, np.float32)
    assert lib.rdvc_corr_update_conv_pack_weights(0, None, rc.RDVC_DT_F16, w.ctypes.data) == -1
    assert lib.rdvc_corr_update_conv_pack_weights(0, w.ctypes.data, rc.RDVC_DT_F32, w.ctypes.data) == -4
    assert lib.rdvc_corr_update_conv_pack_weights(7, w.ctypes.data, rc.RDVC_DT_F16, w.ctypes.data) == -5

    def c1x1(**kw):
        a = dict(out=A, odt=rc.RDVC_DT_F16, ps=256)
        a.update(kw)
        return lib.rdvc_conv1x1_ex(A, rc.RDVC_DT_F16, A, A, 1, 8, 8, 4, 4, 256, 1, a["out"], a["odt"], a["ps"], None)
    assert c1x1(odt=rc.RDVC_DT_F32) == -4 and c1x1(ps=128) == -5 and c1x1(ps=-1) == -5
    assert c1x1(ps=260) == -7 and c1x1(out=A + 8) == -7


def test_module_refusals_on_cpu():
    me, fh = (m.eval() for m in seeded())
    flow, corr, h = torch.randn(1, 2, 8, 8), torch.randn(1, 324, 8, 8), torch.randn(1, 128, 8, 8)
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            me(flow, corr)
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            fh(h)
    with pytest.raises(RuntimeError, match="forward-only"):
        me(flow, corr.requires_grad_())
    with pytest.raises(RuntimeError, match="forward-only"):
        fh(h.requires_grad_())
    me.train(), fh.train()
    with pytest.raises(RuntimeError, match="forward-only"):
        me(flow, corr.detach())
    with pytest.raises(RuntimeError, match="forward-only"):
        fh(h.detach())


# ------------------------------------------------------------------ GPU
def _r(t, dt):
    return t.to(dt).double()


def _op(dt):
    return torch.float16 if dt == torch.float32 else dt


def ref_layer(conv, x, op, relu=True):
    """One layer in fp64 with the kernels' operand rounding (to ``op``); the result is left unrounded, so that a kernel
    output is within one rounding (u |ref|) of it."""
    k = conv.kernel_size[0]
    y = F.conv2d(_r(x, op), _r(conv.weight.detach(), op), conv.bias.detach().double(), padding=k // 2)
    return y.clamp_min(0) if relu else y


def _tol(ref, out_dt):
    return U[out_dt] * ref.double().abs() + 2e-4


def _flow(B, H, W, g):
    return (4 * torch.randn(B, 2, H, W, device="cuda", generator=g)).float()


def run_layer(lib, layer, conv, x, flow, op, out_dt):
    """x: (B, cin, H, W) channels_last op-dtype view (or None for convflow1) -> (B, cout, H, W); conv -> all 128
    channels (motion features + flow); flow_head.conv2 -> (B, 2, H, W)."""
    B, H, W = flow.shape[0], flow.shape[2], flow.shape[3]
    cin, cout, k, n = LAYERS[layer]
    pk = PackedUpdateConv(conv, layer, op, "cuda")
    fs = (ctypes.c_longlong * 4)(*flow.stride())
    if layer == _cabi.RDVC_UC_FH_CONV2:
        out = torch.empty(B, 2, H, W, dtype=out_dt, device="cuda")
        ps = 0
    else:
        out = torch.empty(B, H, W, n, dtype=out_dt, device="cuda")
        ps = n
    xp, xps = (0, 0) if x is None else (x.data_ptr(), x.stride(3))
    _cabi.check(lib.rdvc_corr_update_conv(layer, xp, xps, flow.data_ptr(), fs, B, H, W, ADT[op], pk.weight.data_ptr(),
                                     pk.bias.data_ptr(), out.data_ptr(), ps, ADT[out_dt],
                                     torch.cuda.current_stream().cuda_stream), "rdvc_corr_update_conv")
    keep = 128 if layer == _cabi.RDVC_UC_CONV else cout          # conv: 126 channels + the flow in 126-127
    return out if layer == _cabi.RDVC_UC_FH_CONV2 else out.permute(0, 3, 1, 2)[:, :keep]


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("shape", SHAPES)
def test_layers_match_fp64(lib, shape, dt):
    B, H, W = shape
    me, fh = (m.cuda().eval() for m in seeded(1))
    op = _op(dt)
    g = torch.Generator(device="cuda").manual_seed(B * H * W)
    flow = _flow(B, H, W, g)
    cl = torch.channels_last
    for layer, (cin, cout, k, n) in LAYERS.items():
        conv = conv_of(me, fh, layer)
        out_dt = dt if layer in (_cabi.RDVC_UC_CONV, _cabi.RDVC_UC_FH_CONV2) else op
        if layer == _cabi.RDVC_UC_CONVFLOW1:
            x, xin = None, flow
        else:
            xin = torch.rand(B, cin, H, W, device="cuda", generator=g).to(op).contiguous(memory_format=cl)
            x = xin
        got = run_layer(lib, layer, conv, x, flow, op, out_dt)
        ref = ref_layer(conv, xin, op, relu=layer != _cabi.RDVC_UC_FH_CONV2)
        if layer == _cabi.RDVC_UC_CONV:
            assert torch.equal(got[:, 126:], flow.to(out_dt)), "flow channels"
            got = got[:, :126]
        err = (got.double() - ref.double()).abs()
        assert bool((err <= _tol(ref, out_dt)).all()), (layer, err.max().item())


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("shape", SHAPES)
def test_modules_match_fp64_chain_and_stock(lib, shape, dt):
    """Whole modules (fused entry of the motion encoder) against the fp64 chain and against torchvision's modules."""
    B, H, W = shape
    me, fh = (m.cuda().eval() for m in seeded(2))
    op = _op(dt)
    g = torch.Generator(device="cuda").manual_seed(7 + B * H * W)
    flow = _flow(B, H, W, g)
    c1 = torch.rand(B, 256, H, W, device="cuda", generator=g).to(op).contiguous(memory_format=torch.channels_last)
    h = torch.tanh(torch.randn(B, 128, H, W, device="cuda", generator=g)).to(dt).contiguous(memory_format=torch.channels_last)
    with torch.no_grad(), torch.autocast("cuda", dtype=op, enabled=dt != torch.float32):
        mf = me.forward_fused(flow, c1)
        d = fh(h)
    assert mf.dtype == dt and mf.shape == (B, 128, H, W) and mf.is_contiguous(memory_format=torch.channels_last)
    assert d.dtype == dt and d.shape == (B, 2, H, W)
    with torch.no_grad():
        f2 = ref_layer(me.convflow2[0], ref_layer(me.convflow1[0], flow, op), op)
        cf = torch.cat([ref_layer(me.convcorr2[0], c1, op), f2], 1)
        ref_mf = torch.cat([ref_layer(me.conv[0], cf, op), flow.to(dt).double()], 1)
        ref_d = ref_layer(fh.conv2, ref_layer(fh.conv1, h, op), op, relu=False)
    for got, ref in ((mf, ref_mf), (d, ref_d)):
        err = (got.double() - ref.double()).abs()
        assert bool((err <= 2 * _tol(ref, dt) + 2 * U[op] * ref.double().abs().max()).all()), err.max().item()
    # stock torchvision modules (cuDNN; TF32 off for fp32), autocast for 16-bit
    tme, tfh = tv_me().cuda().eval(), tv_fh().cuda().eval()
    tme.load_state_dict(me.state_dict())
    tfh.load_state_dict(fh.state_dict())
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad(), torch.autocast("cuda", dtype=op, enabled=dt != torch.float32):
            c1s = c1.to(dt)
            s_mf = tme.conv(torch.cat([tme.convcorr2(c1s), tme.convflow2(tme.convflow1(flow.to(dt)))], 1))
            s_mf = torch.cat([s_mf, flow], 1)
            s_d = tfh(h)
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    scale = max(1.0, s_mf.abs().max().item())
    assert (mf.float() - s_mf.float()).abs().max().item() <= TOL_STOCK[dt] * scale
    assert (d.float() - s_d.float()).abs().max().item() <= TOL_STOCK[dt] * max(1.0, s_d.abs().max().item())


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES)
def test_stock_contract_forward_matches_torchvision(lib, dt):
    """``forward(flow, corr_features)``: the 324-channel lookup in, against torchvision's MotionEncoder."""
    B, H, W = 2, 18, 22
    me = seeded(3)[0].cuda().eval()
    tme = tv_me().cuda().eval()
    tme.load_state_dict(me.state_dict())
    g = torch.Generator(device="cuda").manual_seed(5)
    flow = _flow(B, H, W, g)
    corr = torch.rand(B, 324, H, W, device="cuda", generator=g)
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad(), torch.autocast("cuda", dtype=_op(dt), enabled=dt != torch.float32):
            got = me(flow, corr)
            ref = tme(flow, corr)
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    assert got.dtype == dt and got.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(got[:, 126:], flow.to(dt))
    assert (got.float() - ref.float()).abs().max().item() <= TOL_STOCK[dt] * max(1.0, ref.abs().max().item())


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("layout", ["nchw", "channels_last", "slice"])
def test_input_forms(lib, dt, layout):
    """NCHW, channels_last and channel slices of channels_last tensors give the same bits."""
    B, H, W = 2, 17, 19
    me, fh = (m.cuda().eval() for m in seeded(4))
    op = _op(dt)
    g = torch.Generator(device="cuda").manual_seed(9)
    flow = _flow(B, H, W, g)
    big = torch.rand(B, 512, H, W, device="cuda", generator=g).to(dt).contiguous(memory_format=torch.channels_last)
    c1, h = big[:, :256].to(op), big[:, 256:384]
    c1_cl, h_cl = c1.contiguous(memory_format=torch.channels_last), h.contiguous(memory_format=torch.channels_last)
    with torch.no_grad(), torch.autocast("cuda", dtype=op, enabled=dt != torch.float32):
        ref_mf, ref_d = me.forward_fused(flow, c1_cl), fh(h_cl)
        if layout == "nchw":
            args = (flow.contiguous(), c1_cl.contiguous(), h_cl.contiguous())
        elif layout == "channels_last":
            args = (flow.contiguous(memory_format=torch.channels_last), c1_cl, h_cl)
        else:
            big16 = big.to(op)
            args = (flow, big16[:, :256], big[:, 256:384])
            assert args[1].stride(1) == 1 and args[1].stride(3) == 512 and args[2].stride(3) == 512
        mf, d = me.forward_fused(args[0], args[1]), fh(args[2])
    assert torch.equal(mf, ref_mf) and torch.equal(d, ref_d)


@pytest.mark.gpu
@pytest.mark.parametrize("feat", [torch.float16, torch.bfloat16])
def test_conv1x1_nhwc_output_is_the_nchw_output_permuted(lib, feat):
    B, D, h, w = 2, 256, 23, 37
    g = torch.Generator(device="cuda").manual_seed(11)
    f1 = torch.randn(B, D, h, w, device="cuda", generator=g)
    f2 = torch.randn(B, D, h, w, device="cuda", generator=g)
    blk = rc.TVCorrBlock()
    blk.build_pyramid(f1, f2)
    ys, xs = torch.meshgrid(torch.arange(h, device="cuda"), torch.arange(w, device="cuda"), indexing="ij")
    coords = torch.stack([xs, ys], 0).float()[None].repeat(B, 1, 1, 1)
    coords = coords + 3 * torch.randn(coords.shape, device="cuda", generator=g)
    conv = torch.nn.Conv2d(324, 256, 1).cuda()
    with torch.no_grad():
        nchw = blk.index_pyramid_convcorr1(coords, conv.weight, conv.bias, out_dtype=feat, feat_dtype=feat)
        nhwc = blk.index_pyramid_convcorr1(coords, conv.weight, conv.bias, feat_dtype=feat, nhwc=True)
    assert nhwc.dtype == feat and nhwc.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(nhwc, nchw)


@pytest.mark.gpu
def test_channels_outside_the_slice_are_untouched(lib):
    """A layer writes its N channels of every pixel and nothing else: sentinel-filled buffers keep their other channels."""
    B, H, W = 2, 17, 19
    me, fh = (m.cuda().eval() for m in seeded(5))
    g = torch.Generator(device="cuda").manual_seed(13)
    flow = _flow(B, H, W, g)
    f1 = torch.rand(B, H, W, 128, device="cuda", generator=g).half()
    st = torch.cuda.current_stream().cuda_stream
    fs = (ctypes.c_longlong * 4)(*flow.stride())
    for layer, src, width, lo, out_dt in ((_cabi.RDVC_UC_CONVFLOW2, f1, 256, 192, torch.float16),
                                          (_cabi.RDVC_UC_CONV, torch.rand(B, H, W, 256, device="cuda", generator=g).half(),
                                           160, 16, torch.float32)):
        n = LAYERS[layer][3]
        pk = PackedUpdateConv(conv_of(me, fh, layer), layer, torch.float16, "cuda")
        buf = torch.full((B, H, W, width), 12345.0, dtype=out_dt, device="cuda")
        _cabi.check(lib.rdvc_corr_update_conv(layer, src.data_ptr(), src.shape[-1], flow.data_ptr(), fs, B, H, W, rc.RDVC_DT_F16,
                                         pk.weight.data_ptr(), pk.bias.data_ptr(), buf[..., lo:].data_ptr(), width,
                                         ADT[out_dt], st), "rdvc_corr_update_conv")
        torch.cuda.synchronize()
        assert bool((buf[..., :lo] == 12345.0).all()) and bool((buf[..., lo + n:] == 12345.0).all()), layer
        assert torch.isfinite(buf).all() and not bool((buf[..., lo:lo + n] == 12345.0).any())


@pytest.mark.gpu
def test_deterministic_streams_graphs_and_repacking(lib):
    me, fh = (m.cuda().eval() for m in seeded(6))
    B, H, W = 2, 46, 80
    g = torch.Generator(device="cuda").manual_seed(3)
    flow = _flow(B, H, W, g)
    corr = torch.rand(B, 324, H, W, device="cuda", generator=g)
    h = torch.tanh(torch.randn(B, 128, H, W, device="cuda", generator=g)).half().contiguous(memory_format=torch.channels_last)

    def run():
        with torch.autocast("cuda", dtype=torch.float16):
            return me(flow, corr), fh(h)
    with torch.no_grad():
        a, b = run(), run()
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            c = run()
        torch.cuda.current_stream().wait_stream(side)
        assert torch.equal(a[0], c[0]) and torch.equal(a[1], c[1])
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            d = run()
        gr.replay()
        torch.cuda.synchronize()
        assert torch.equal(a[0], d[0]) and torch.equal(a[1], d[1])
        me.conv[0].bias.add_(0.5)                      # an in-place change bumps the version: re-packed
        fh.conv2.weight.mul_(2.0)
        e = run()
        assert not torch.equal(a[0], e[0]) and not torch.equal(a[1], e[1])
        other_me, other_fh = (m.cuda().eval() for m in seeded(7))
        me.load_state_dict(other_me.state_dict())
        fh.load_state_dict(other_fh.state_dict())
        with torch.autocast("cuda", dtype=torch.float16):
            assert torch.equal(run()[0], other_me(flow, corr)) and torch.equal(run()[1], other_fh(h))


# ------------------------------------------------------------------ RAFT end to end
def _seeded_raft(swap, corr_block=True):
    from torchvision.models.optical_flow import raft_large
    torch.manual_seed(0)
    model = raft_large(weights=None, **({"corr_block": rc.TVCorrBlock()} if corr_block else {})).eval().cuda()
    ub = model.update_block
    if swap in ("me_fh", "all"):
        me, fh = rc.MotionEncoder(in_channels_corr=324), rc.FlowHead(in_channels=128, hidden_size=256)
        me.load_state_dict(ub.motion_encoder.state_dict())
        fh.load_state_dict(ub.flow_head.state_dict())
        ub.motion_encoder, ub.flow_head = me.cuda(), fh.cuda()
    if swap == "all":
        rb = rc.RecurrentBlock(input_size=256, hidden_size=128)
        rb.load_state_dict(ub.recurrent_block.state_dict())
        ub.recurrent_block = rb.cuda()
    return model


def _frames(golden_dir, size):
    import torchvision.transforms.functional as TF
    g = np.load(os.path.join(golden_dir, "frames_im1_im2.npz"))
    return [TF.resize(TF.to_tensor(g[k]), list(size), antialias=True).unsqueeze(0).cuda() for k in ("im1", "im2")]


def _synthetic_1080p():
    g = torch.Generator(device="cuda").manual_seed(12)
    base = F.interpolate(torch.rand(1, 3, 68, 120, device="cuda", generator=g), size=(1080, 1920), mode="bicubic",
                         align_corners=False).clamp(0, 1)
    return base, torch.roll(base, (3, -5), (2, 3))


def _epe(a, b):
    return (a.float() - b.float()).pow(2).sum(dim=1).sqrt().mean().item()


@pytest.mark.gpu
@pytest.mark.parametrize("amp", [False, True])
@pytest.mark.parametrize("swap", ["me_fh", "all"])
@pytest.mark.parametrize("case", ["368x640", "1080p"])
def test_raft_epe_vs_stock(lib, golden_dir, case, swap, amp):
    a, b = _frames(golden_dir, (368, 640)) if case == "368x640" else _synthetic_1080p()
    model = _seeded_raft(swap)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=amp):
        ref = _seeded_raft(None, corr_block=False)(a, b, num_flow_updates=12)[-1]
        got = rc.raft_flow(model, a, b, 12)
        stock_call = model(a, b, num_flow_updates=12)[-1]             # RAFT.forward with the drop-ins swapped in
    assert isinstance(model.update_block.motion_encoder, rc.MotionEncoder)
    assert isinstance(model.update_block.flow_head, rc.FlowHead)
    assert torch.isfinite(got).all() and torch.isfinite(stock_call).all()
    assert _epe(got, ref) < TOL_EPE, _epe(got, ref)
    assert _epe(stock_call, ref) < TOL_EPE, _epe(stock_call, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("swap", ["me_fh", "all"])
def test_raft_sequence_and_graphs(lib, golden_dir, swap):
    """raft_flow_sequence and GraphedRaftFlow with the drop-ins: the sequence matches the pair-wise calls and stock
    torchvision, the graph replays eager bit for bit."""
    a, b = _frames(golden_dir, (368, 640))
    frames = torch.cat([a, b, torch.roll(a, (3, -5), (2, 3))], 0)
    model = _seeded_raft(swap)
    with torch.no_grad():
        pairs = rc.raft_flow(model, frames[:-1], frames[1:], 12)
        seq = rc.raft_flow_sequence(model, frames, 12)
        ref = _seeded_raft(None, corr_block=False)(frames[:-1], frames[1:], num_flow_updates=12)[-1]
    assert _epe(seq, pairs) < 2e-3
    assert _epe(seq, ref) < TOL_EPE
    for amp in (None, torch.float16):
        runner = rc.GraphedRaftFlow(model, 12, amp_dtype=amp)
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=amp is not None):
            eager = rc.raft_flow(model, a, b, 12)
            eager_seq = rc.raft_flow_sequence(model, frames, 12)
        assert torch.equal(runner(a, b), eager) and torch.equal(runner(a, b), eager)
        assert torch.equal(runner.sequence(frames), eager_seq)
        assert _epe(runner(a, b), ref[:1]) < TOL_EPE
        runner.release()
