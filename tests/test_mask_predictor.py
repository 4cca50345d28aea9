"""RAFT's mask predictor (torchvision MaskPredictor, TV:raft.py:311-334) with the convex 8x upsampling of
upsample_flow (TV:_utils.py:29-48) fused into its 1x1 GEMM.

CPU part (-m "not gpu"): parameter tree and strict state_dict round trips against torchvision's class, the refused
configurations, the host-packed 1x1 operand evaluated the way the kernel walks it, the C ABI's argument errors and
size queries, the module refusals, the kernels' SASS and their spill-free register allocation.
GPU part (-m gpu): both output forms against an fp64 evaluation with the kernels' rounding points and against stock
torchvision, tiny shapes, image borders, the softmax range, input forms, batch invariance, determinism / streams /
graphs / re-packing, strided flows, and RAFT end to end.

Rounding points of the kernels (u = unit roundoff: 2^-11 fp16, 2^-8 bf16, 0 fp32):
  the hidden state and both weights rounded to the 16-bit operand type (fp16 for fp32 activations); convrelu
  accumulated in fp32, bias + ReLU in fp32, rounded to the operand type; the 1x1 accumulated in fp32; then in fp32:
  logit = multiplier * (acc + bias), softmax over the 9 taps with the max subtracted, sum_k p_k * 8 * flow_k with the
  fp32 flow (MASK form: the logit rounded once to the activation dtype).
Tolerances (absolute, per element; F = max |8 flow|):
  * UPSAMPLED vs fp64 with the same rounding points ........ 1e-3 F
      the fp32 logits are within ~1e-5 of the fp64 ones (K = 256 fp32 sums, plus a convrelu result that may round the
      other way on a boundary); the softmax weights move by that relative amount and the output by that times F.
  * MASK vs fp64 of the 1x1 on the kernel's own convrelu output . multiplier (u |ref / multiplier| + 2e-4)
      the per-layer bound of test_motion_encoder.py on conv + bias, scaled by the multiplier.  The 1x1's input is
      taken from the FH_CONV1 launch the module runs convrelu on (that layer has its own bound in
      test_motion_encoder.py): an fp64 convrelu result on a rounding boundary of the operand type may round the other
      way in the kernel, which moves the 1x1's input by a whole ulp -- up to ~2e-4 of a logit for bf16.
  * vs stock torchvision (cuDNN, TF32 off for fp32) ........ 2e-2 F (fp32, fp16), 1e-1 F (bf16); the mask form the same
      relative to max(1, max |mask|): the stock fp32 path keeps fp32 operands, autocast rounds the same intermediates
      but sums in another order.
  * a constant flow inside the image ........................ 8 flow up to fp32 rounding: 1e-6 relative (two fp32
      sums of 9 terms and a reciprocal).
  * RAFT flow vs stock torchvision, mean EPE ................ < 0.05 px
A wrong tap, sub-pixel or channel mapping shows up as an O(1) F error.
"""
import ctypes
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import rdvc_corr_b200 as rc
from rdvc_corr_b200 import _cabi
from rdvc_corr_b200.motion_encoder import PackedUpdateConv

U = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8, torch.float32: 0.0}
TOL_STOCK = {torch.float32: 2e-2, torch.float16: 2e-2, torch.bfloat16: 1e-1}
TOL_FP64 = 1e-3
TOL_EPE = 0.05
SHAPES = [(1, 46, 80), (2, 18, 22), (1, 17, 19), (1, 33, 47), (9, 136, 240), (1, 5, 7)]
DTYPES = [torch.float32, torch.float16, torch.bfloat16]
ADT = {torch.float32: rc.RDVC_DT_F32, torch.float16: rc.RDVC_DT_F16, torch.bfloat16: rc.RDVC_DT_BF16}
PKG = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                   "pfe-raft-and-hyperprior-based-learned-video-compression_b200")


@pytest.fixture(scope="module")
def lib():
    rc._build.build()
    return rc._cabi.load()


def tv_mp(multiplier=0.25):
    from torchvision.models.optical_flow.raft import MaskPredictor
    return MaskPredictor(in_channels=128, hidden_size=256, multiplier=multiplier)


def seeded(seed=0, multiplier=0.25):
    torch.manual_seed(seed)
    return rc.MaskPredictor(in_channels=128, hidden_size=256, multiplier=multiplier)


def stock_upsample(flow, mask):
    from torchvision.models.optical_flow._utils import upsample_flow
    return upsample_flow(flow=flow, up_mask=mask)


# ------------------------------------------------------------------ CPU
def test_state_dict_matches_torchvision():
    ours, tv, tv2 = seeded(), tv_mp(), tv_mp()
    assert list(ours.state_dict().keys()) == list(tv.state_dict().keys())
    assert all(ours.state_dict()[k].shape == v.shape for k, v in tv.state_dict().items())
    ours.load_state_dict(tv.state_dict(), strict=True)
    tv2.load_state_dict(ours.state_dict(), strict=True)
    assert all(torch.equal(tv2.state_dict()[k], v) for k, v in tv.state_dict().items())
    assert seeded(multiplier=1.0).multiplier == 1.0


@pytest.mark.parametrize("kw", [dict(in_channels=96, hidden_size=64), dict(in_channels=128, hidden_size=128),
                                dict(in_channels=256, hidden_size=256)])
def test_unsupported_mask_predictors_raise(kw):
    with pytest.raises(ValueError):
        rc.MaskPredictor(**kw)


def _packed(lib, conv, op):
    w = np.ascontiguousarray(conv.weight.detach().numpy().reshape(576, 256).astype(np.float32))
    b = np.ascontiguousarray(conv.bias.detach().numpy().astype(np.float32))
    packed = np.zeros(lib.rdvc_corr_mask_conv_packed_weight_bytes() // 2, np.uint16)
    bias = np.zeros(576, np.float32)
    _cabi.check(lib.rdvc_corr_mask_conv_pack_weights(w.ctypes.data, b.ctypes.data, ADT[op], packed.ctypes.data,
                                                     bias.ctypes.data), "pack")
    return torch.from_numpy(packed.view(np.int16)).view(op).double().numpy(), bias


@pytest.mark.parametrize("op", [torch.float16, torch.bfloat16])
def test_packed_operand_reproduces_the_convolution(lib, op):
    """The packed operand walked the way the kernel walks it -- chunk c, k-block, GEMM row c * 144 + k * 16 + s, which
    the epilogue reads as tap k of sub-pixel (2c + s // 8, s % 8) -- is the 1x1 convolution in stock channel order."""
    torch.manual_seed(3)
    conv = torch.nn.Conv2d(256, 576, 1)
    p, bias = _packed(lib, conv, op)
    assert p.size == 576 * 256
    pm = p.reshape(4, 4, 144, 64)                         # [c][k-block][144][64]
    a = torch.randn(2, 256, 5, 6).to(op).double()
    want = F.conv2d(a, conv.weight.detach().to(op).double(), conv.bias.detach().double()).numpy()
    an = a.numpy()
    got = np.zeros_like(want)
    for c in range(4):
        acc = sum(np.einsum("bchw,nc->bnhw", an[:, kb * 64:(kb + 1) * 64], pm[c, kb]) for kb in range(4))
        for k in range(9):
            for s in range(16):
                i, j = 2 * c + s // 8, s % 8
                ch = k * 64 + i * 8 + j                   # torchvision's mask channel of tap k, sub-pixel (i, j)
                got[:, ch] = acc[:, k * 16 + s] + bias[c * 144 + k * 16 + s]
    assert np.abs(got - want).max() <= 1e-9 * np.abs(want).max()


def test_cabi_argument_errors(lib):
    A = 1 << 20           # a 16-byte aligned fake device address: every call below fails its checks before any access
    fs = (ctypes.c_longlong * 4)(2 * 64, 64, 8, 1)
    assert lib.rdvc_corr_mask_conv_packed_weight_bytes() == 576 * 256 * 2
    ws16 = lib.rdvc_corr_mask_predictor_workspace_bytes(1, 8, 8, rc.RDVC_DT_F16)
    ws32 = lib.rdvc_corr_mask_predictor_workspace_bytes(1, 8, 8, rc.RDVC_DT_F32)
    assert ws32 > ws16 >= 64 * 256 * 2
    assert lib.rdvc_corr_mask_predictor_workspace_bytes(0, 8, 8, rc.RDVC_DT_F16) == 0
    assert lib.rdvc_corr_mask_predictor_workspace_bytes(1, 8, 8, 7) == 0
    ptr2 = (ctypes.c_void_p * 2)(A, A)

    def mp(**kw):
        a = dict(h=A, ps=128, act=rc.RDVC_DT_F16, B=1, H=8, W=8, op=rc.RDVC_DT_F16, w=ptr2, b=ptr2, mult=0.25, f=A, fs=fs,
                 form=_cabi.RDVC_MASK_OUT_UPSAMPLED, ws=A, wsb=ws16, out=2 * A)
        a.update(kw)
        return lib.rdvc_corr_mask_predictor(a["h"], a["ps"], a["act"], a["B"], a["H"], a["W"], a["op"], a["w"], a["b"],
                                            a["mult"], a["f"], a["fs"], a["form"], a["ws"], a["wsb"], a["out"], None)
    assert mp(h=None) == -1 and mp(w=None) == -1 and mp(b=(ctypes.c_void_p * 2)(A, None)) == -1
    assert mp(out=None) == -1 and mp(ws=None) == -1 and mp(f=None) == -1 and mp(fs=None) == -1
    assert mp(form=2) == -5 and mp(form=-1) == -5
    assert mp(B=0) == -2 and mp(H=-1) == -2 and mp(W=0) == -2
    assert mp(act=9) == -4 and mp(act=rc.RDVC_DT_BF16) == -4 and mp(op=rc.RDVC_DT_F32) == -4
    assert mp(ps=64) == -5 and mp(ps=132) == -7 and mp(h=A + 8) == -7 and mp(out=A + 4) == -7
    assert mp(w=(ctypes.c_void_p * 2)(A, A + 2)) == -7 and mp(ws=A + 16) == -7
    assert mp(wsb=ws16 - 1) == -6 and mp(act=rc.RDVC_DT_F32) == -6          # fp32 h needs the larger workspace
    for rcode in (mp(h=None), mp(form=5)):
        assert rcode < 0 and _cabi.last_error()
    w = np.zeros(4, np.float32)
    assert lib.rdvc_corr_mask_conv_pack_weights(None, w.ctypes.data, rc.RDVC_DT_F16, w.ctypes.data, w.ctypes.data) == -1
    assert lib.rdvc_corr_mask_conv_pack_weights(w.ctypes.data, w.ctypes.data, rc.RDVC_DT_F16, w.ctypes.data, None) == -1
    assert lib.rdvc_corr_mask_conv_pack_weights(w.ctypes.data, w.ctypes.data, rc.RDVC_DT_F32, w.ctypes.data,
                                                w.ctypes.data) == -4


def test_module_refusals_on_cpu():
    mp = seeded().eval()
    h, flow = torch.randn(1, 128, 8, 8), torch.randn(1, 2, 8, 8)
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            mp(h)
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            mp.upsample_flow(flow, h)
    with pytest.raises(RuntimeError, match="forward-only"):
        mp(h.requires_grad_())
    with pytest.raises(RuntimeError, match="forward-only"):
        mp.upsample_flow(flow.requires_grad_(), h.detach())
    mp.train()
    with pytest.raises(RuntimeError, match="forward-only"):
        mp(h.detach())


def test_sass_has_tcgen05_and_tma(lib):
    """Every instantiation of the fused kernel is Blackwell-native: tcgen05.mma (UTCHMMA), TMA loads (UTMALDG) and
    TMEM reads (LDTM)."""
    out = subprocess.run(["cuobjdump", "-sass", rc._cabi.lib_path()], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    funcs = [f for f in out.stdout.split("Function : ") if f.startswith("_ZN4rdvc20mask_upsample_kernel")]
    assert len(funcs) == 6, len(funcs)       # UPSAMPLED x 2 operand dtypes + MASK x (fp32, 16-bit) x 2 operand dtypes
    for f in funcs:
        assert "UTCHMMA" in f and "UTMALDG" in f and "LDTM" in f, f.splitlines()[0]


def test_no_register_spills():
    """-Xptxas -v over every instantiation of the fused kernel: no spill stores or loads."""
    from rdvc_corr_b200 import _build
    src = """
#include "mask_upsample_sm100.cuh"
namespace rdvc {
#define MU(E, O, P) template __global__ void mask_upsample_kernel<E, O, P>(const __grid_constant__ CUtensorMap, const __grid_constant__ CUtensorMap, const MuParams);
MU(0, float, __half) MU(0, float, __nv_bfloat16) MU(1, float, __half) MU(1, float, __nv_bfloat16)
MU(1, __half, __half) MU(1, __nv_bfloat16, __nv_bfloat16)
}
"""
    with tempfile.TemporaryDirectory() as d:
        cu = os.path.join(d, "spills.cu")
        with open(cu, "w") as f:
            f.write(src)
        res = subprocess.run([_build.nvcc_path(), "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                              "-Xptxas", "-v", "-I", os.path.join(PKG, "csrc"), "-c", cu, "-o", os.path.join(d, "s.o")],
                             capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-3000:]
    props = [ln for ln in res.stderr.splitlines() if "spill stores" in ln]
    assert len(props) == 6, res.stderr[-3000:]
    assert all("0 bytes spill stores, 0 bytes spill loads" in ln for ln in props), props


# ------------------------------------------------------------------ GPU
def _op(dt):
    return torch.float16 if dt == torch.float32 else dt


def _r(t, dt):
    return t.to(dt).double()


def ref_logits(mp, h, op, y=None):
    """fp64 with the kernels' rounding points: h and weights rounded to ``op``, convrelu's result rounded to ``op``;
    the logits multiplier * (conv + bias) left unrounded.  ``y``: use this convrelu output instead of the fp64 one."""
    if y is None:
        c1 = mp.convrelu[0]
        y = F.conv2d(_r(h, op), _r(c1.weight.detach(), op), c1.bias.detach().double(), padding=1).clamp_min(0)
    y = _r(y, op)
    return mp.multiplier * F.conv2d(y, _r(mp.conv.weight.detach(), op), mp.conv.bias.detach().double())


def kernel_convrelu(lib, mp, h, op):
    """convrelu through the library's FH_CONV1 launch, the kernel the module runs it on: (B, 256, H, W) in ``op``."""
    B, _, H, W = h.shape
    x = h.to(op).contiguous(memory_format=torch.channels_last)
    pk = PackedUpdateConv(mp.convrelu[0], _cabi.RDVC_UC_FH_CONV1, op, "cuda")
    out = torch.empty(B, H, W, 256, dtype=op, device="cuda")
    _cabi.check(lib.rdvc_corr_update_conv(_cabi.RDVC_UC_FH_CONV1, x.data_ptr(), x.stride(3), None, None, B, H, W, ADT[op],
                                          pk.weight.data_ptr(), pk.bias.data_ptr(), out.data_ptr(), 256, ADT[op],
                                          torch.cuda.current_stream().cuda_stream), "rdvc_corr_update_conv")
    return out.permute(0, 3, 1, 2)


def _flow(B, H, W, g):
    return (4 * torch.randn(B, 2, H, W, device="cuda", generator=g)).float()


def _hidden(B, H, W, dt, g):
    return torch.tanh(torch.randn(B, 128, H, W, device="cuda", generator=g)).to(dt).contiguous(
        memory_format=torch.channels_last)


def _run_both(mp, h, flow, dt):
    with torch.no_grad(), torch.autocast("cuda", dtype=_op(dt), enabled=dt != torch.float32):
        return mp.upsample_flow(flow, h), mp(h)


def _fh_refuses(B, H, W, dt):
    """The error the existing 3x3 launcher (FlowHead) gives at this shape, or None."""
    fh = rc.FlowHead(in_channels=128, hidden_size=256).cuda().eval()
    h = torch.zeros(B, 128, H, W, device="cuda", dtype=dt)
    try:
        with torch.no_grad():
            fh(h)
    except ValueError as e:
        return str(e)
    return None


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("shape", SHAPES)
def test_matches_fp64_and_stock(lib, shape, dt):
    B, H, W = shape
    mp = seeded(1).cuda().eval()
    op = _op(dt)
    g = torch.Generator(device="cuda").manual_seed(B * H * W)
    flow = _flow(B, H, W, g)
    h = _hidden(B, H, W, dt, g)
    refused = _fh_refuses(B, H, W, op) if (H < 8 or W < 16) else None
    if refused is not None:
        with pytest.raises(ValueError) as ei:
            _run_both(mp, h, flow, dt)
        assert str(ei.value).split(": ", 1)[1] == refused.split(": ", 1)[1]
        return
    up, mask = _run_both(mp, h, flow, dt)
    torch.cuda.synchronize()
    assert up.dtype == torch.float32 and up.shape == (B, 2, 8 * H, 8 * W) and up.is_contiguous()
    assert mask.dtype == dt and mask.shape == (B, 576, H, W) and mask.is_contiguous()
    Fmax = (8 * flow).abs().max().item()
    with torch.no_grad():
        logits = ref_logits(mp, h, op)
        ref_up = stock_upsample(flow.double(), logits)
    assert (up.double() - ref_up).abs().max().item() <= TOL_FP64 * Fmax
    # MASK: the per-layer bound of the 1x1 on the kernel's own convrelu output (an fp64 convrelu result that sits on a
    # rounding boundary of the operand type may round the other way in the kernel, a whole ulp of the 1x1's input)
    with torch.no_grad():
        logits_1x1 = ref_logits(mp, h, op, y=kernel_convrelu(lib, mp, h, op))
    tol = U[dt] * logits_1x1.abs() + 2e-4 * mp.multiplier
    err = (mask.double() - logits_1x1).abs()
    assert bool((err <= tol).all()), err.max().item()
    # stock torchvision (cuDNN; TF32 off for fp32), autocast for 16-bit
    tmp = tv_mp().cuda().eval()
    tmp.load_state_dict(mp.state_dict())
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad(), torch.autocast("cuda", dtype=op, enabled=dt != torch.float32):
            s_mask = tmp(h)
            s_up = stock_upsample(flow, s_mask)
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    assert (up - s_up.float()).abs().max().item() <= TOL_STOCK[dt] * Fmax
    assert (mask.float() - s_mask.float()).abs().max().item() <= TOL_STOCK[dt] * max(1.0, s_mask.abs().max().item())


def _biased(mp, tap, logit):
    """Zero weights and a bias that gives tap ``tap`` of every sub-pixel the logit ``logit``, the others 0."""
    with torch.no_grad():
        mp.conv.weight.zero_()
        mp.conv.bias.zero_()
        mp.conv.bias[tap * 64:(tap + 1) * 64] = logit / mp.multiplier
    return mp


@pytest.mark.gpu
@pytest.mark.parametrize("tap", [0, 2, 6, 8])
def test_borders(lib, tap):
    """A constant flow with every sub-pixel's weight pushed towards one out-of-image neighbour (the corner taps reach
    out of the image at two edges each): stock at the edges, where that neighbour is zero but keeps its weight, and
    exactly 8 flow inside."""
    B, H, W = 2, 19, 37
    mp = _biased(seeded(2).cuda().eval(), tap, 5.0)
    flow = torch.empty(B, 2, H, W, device="cuda")
    flow[:, 0], flow[:, 1] = 3.25, -1.5
    h = torch.rand(B, 128, H, W, device="cuda")
    with torch.no_grad():
        up = mp.upsample_flow(flow, h)
        mask = mp(h)
        ref = stock_upsample(flow.double(), mask.double())
    Fmax = 8 * 3.25
    assert (up.double() - ref).abs().max().item() <= 1e-5 * Fmax
    ky, kx = divmod(tap, 3)
    rows = slice(8, 8 * (H - 1)) if ky != 1 else slice(None)
    cols = slice(8, 8 * (W - 1)) if kx != 1 else slice(None)
    inner = up[:, :, rows, cols]
    want = (8 * flow[:, :, :1, :1]).expand_as(inner)
    assert ((inner - want).abs() <= 1e-6 * want.abs()).all()
    edge = up[:, :, :8] if ky == 0 else up[:, :, -8:] if ky == 2 else up[:, :, :, :8] if kx == 0 else up[:, :, :, -8:]
    assert edge.abs().max().item() < 0.1 * Fmax                          # the zero neighbour dominates there


@pytest.mark.gpu
def test_softmax_range(lib):
    """Logits of +-60 after the multiplier: finite, and the fp64 result."""
    B, H, W = 1, 24, 40
    mp = seeded(3).cuda().eval()
    g = torch.Generator(device="cuda").manual_seed(4)
    with torch.no_grad():
        mp.conv.weight.mul_(1e-2)
        mp.conv.bias.copy_(torch.where(torch.rand(576, device="cuda", generator=g) < 0.5, -60.0, 60.0) / mp.multiplier)
    flow = _flow(B, H, W, g)
    h = _hidden(B, H, W, torch.float32, g)
    with torch.no_grad():
        up = mp.upsample_flow(flow, h)
        ref = stock_upsample(flow.double(), ref_logits(mp, h, torch.float16))
    assert torch.isfinite(up).all()
    assert (up.double() - ref).abs().max().item() <= TOL_FP64 * (8 * flow).abs().max().item()


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("layout", ["nchw", "channels_last", "slice"])
def test_input_forms(lib, dt, layout):
    """NCHW, channels_last and a channel slice of a channels_last tensor give the same bits."""
    B, H, W = 2, 17, 19
    mp = seeded(4).cuda().eval()
    g = torch.Generator(device="cuda").manual_seed(9)
    flow = _flow(B, H, W, g)
    big = torch.rand(B, 384, H, W, device="cuda", generator=g).to(dt).contiguous(memory_format=torch.channels_last)
    h_cl = big[:, 128:256].contiguous(memory_format=torch.channels_last)
    ref = _run_both(mp, h_cl, flow, dt)
    x = {"nchw": h_cl.contiguous(), "channels_last": h_cl, "slice": big[:, 128:256]}[layout]
    if layout == "slice":
        assert x.stride(1) == 1 and x.stride(3) == 384
    got = _run_both(mp, x, flow, dt)
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])


@pytest.mark.gpu
def test_batch_invariance_and_strided_flow(lib):
    """The samples of a batch are bit-identical to single-sample runs; a flow at other strides gives the same bits."""
    B, H, W = 2, 33, 47
    mp = seeded(5).cuda().eval()
    g = torch.Generator(device="cuda").manual_seed(6)
    flow = _flow(B, H, W, g)
    h = _hidden(B, H, W, torch.float16, g)
    both = _run_both(mp, h, flow, torch.float16)
    for b in range(B):
        one = _run_both(mp, h[b:b + 1], flow[b:b + 1], torch.float16)
        assert torch.equal(one[0], both[0][b:b + 1]) and torch.equal(one[1], both[1][b:b + 1])
    nhwc = flow.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)          # (B, 2, H, W) with channel stride 1
    wide = torch.zeros(B, 5, H, 2 * W, device="cuda")
    wide[:, 1:3, :, ::2] = flow
    for f in (nhwc, wide[:, 1:3, :, ::2]):
        assert not f.is_contiguous()
        with torch.no_grad():
            assert torch.equal(mp.upsample_flow(f, h), both[0])


@pytest.mark.gpu
def test_deterministic_streams_graphs_and_repacking(lib):
    mp = seeded(6).cuda().eval()
    B, H, W = 2, 46, 80
    g = torch.Generator(device="cuda").manual_seed(3)
    flow = _flow(B, H, W, g)
    h = _hidden(B, H, W, torch.float16, g)

    def run():
        return _run_both(mp, h, flow, torch.float16)
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
        mp.conv.bias.add_(0.5)                        # an in-place change bumps the version: re-packed
        e = run()
        assert not torch.equal(a[0], e[0]) and not torch.equal(a[1], e[1])
        mp.convrelu[0].weight.mul_(2.0)
        f = run()
        assert not torch.equal(e[1], f[1])
        other = seeded(7).cuda().eval()
        mp.load_state_dict(other.state_dict())
        assert torch.equal(run()[0], _run_both(other, h, flow, torch.float16)[0])


# ------------------------------------------------------------------ RAFT end to end
def _seeded_raft(swap, corr_block=True):
    from torchvision.models.optical_flow import raft_large
    torch.manual_seed(0)
    model = raft_large(weights=None, **({"corr_block": rc.TVCorrBlock()} if corr_block else {})).eval().cuda()
    if swap is None:
        return model
    mp = rc.MaskPredictor(in_channels=128, hidden_size=256, multiplier=model.mask_predictor.multiplier)
    mp.load_state_dict(model.mask_predictor.state_dict())
    model.mask_predictor = mp.cuda()
    if swap == "all":
        ub = model.update_block
        me, fh = rc.MotionEncoder(in_channels_corr=324), rc.FlowHead(in_channels=128, hidden_size=256)
        rb = rc.RecurrentBlock(input_size=256, hidden_size=128)
        me.load_state_dict(ub.motion_encoder.state_dict())
        fh.load_state_dict(ub.flow_head.state_dict())
        rb.load_state_dict(ub.recurrent_block.state_dict())
        ub.motion_encoder, ub.flow_head, ub.recurrent_block = me.cuda(), fh.cuda(), rb.cuda()
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
@pytest.mark.parametrize("swap", ["mask", "all"])
@pytest.mark.parametrize("case", ["368x640", "1080p"])
def test_raft_epe_vs_stock(lib, golden_dir, case, swap, amp):
    a, b = _frames(golden_dir, (368, 640)) if case == "368x640" else _synthetic_1080p()
    model = _seeded_raft(swap)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=amp):
        refs = _seeded_raft(None, corr_block=False)(a, b, num_flow_updates=12)
        got = rc.raft_flow(model, a, b, 12)
        stock_call = model(a, b, num_flow_updates=12)[-1]             # RAFT.forward with the drop-ins swapped in
        allp = rc.raft_flow(model, a, b, 12, all_predictions=True) if case == "368x640" else None
    assert isinstance(model.mask_predictor, rc.MaskPredictor)
    assert got.dtype == torch.float32 and got.shape == refs[-1].shape
    assert torch.isfinite(got).all() and torch.isfinite(stock_call).all()
    assert _epe(got, refs[-1]) < TOL_EPE, _epe(got, refs[-1])
    assert _epe(stock_call, refs[-1]) < TOL_EPE, _epe(stock_call, refs[-1])
    if allp is not None:
        assert len(allp) == 12 and torch.equal(allp[-1], got)
        for p, r in zip(allp, refs):
            assert _epe(p, r) < TOL_EPE, _epe(p, r)


@pytest.mark.gpu
@pytest.mark.parametrize("swap", ["mask", "all"])
def test_raft_sequence_and_graphs(lib, golden_dir, swap):
    """raft_flow_sequence and GraphedRaftFlow with the drop-in: the sequence matches the pair-wise calls and stock
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
