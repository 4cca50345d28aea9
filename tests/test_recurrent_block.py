"""RAFT's recurrent block (torchvision RecurrentBlock, TV:raft.py:214-270) as fused tcgen05 convolutions.

CPU part (-m "not gpu"): parameter tree and strict state_dict round trips against torchvision's class, the refused
configurations, the host-packed tap matrices evaluated as a convolution (both tap axes), the C ABI's argument errors,
and the refusals of the module (the kernels' SASS and registers: test_tap_conv.py).
GPU part (-m gpu): passes and whole blocks against an fp64 evaluation with the kernel's rounding points and against
the stock module, guard bands, determinism / streams / graphs, re-packing, and RAFT end to end.

Rounding points of the kernels (u = unit roundoff of the 16-bit type: 2^-11 fp16, 2^-8 bf16; |z| < 1, |h| <= 1):
  operands h, context, motion and weights rounded to the operand type; fp32 accumulation over K = 1920; z and r*h
  rounded to the operand type; q = tanh(.) and (1 - z) h + z q in fp32; the result rounded to h's dtype.
Tolerances (absolute):
  * vs fp64 with the same rounding points, one pass ............. 2 u_op + u_out + 1e-4
      a z or r*h whose fp32 value sits on a rounding boundary may round the other way: one ulp of z moves the
      blend by <= u_op |q - h| <= 2 u_op; the result itself may round either way (u_out; 0 for fp32 out);
      fp32 accumulation order: < 1e-4.  Whole block (two passes, the first one's error carried): twice that.
  * vs the stock module (cuDNN, TF32 off for fp32) ............... 1e-2 (fp32, fp16), 6e-2 (bf16)
      the stock path keeps fp32 operands (fp32) or rounds z, r, r*h, q and the blend to 16 bits (autocast).
  * RAFT flow vs stock torchvision, mean EPE ..................... < 0.05 px
"""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import rdvc_corr_b200 as rc
from rdvc_corr_b200 import _cabi
from rdvc_corr_b200.recurrent_block import PackedConvGRU

U = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8, torch.float32: 0.0}
TOL_STOCK = {torch.float32: 1e-2, torch.float16: 1e-2, torch.bfloat16: 6e-2}
TOL_EPE = 0.05
KS, PAD = ((1, 5), (5, 1)), ((0, 2), (2, 0))
SHAPES = [(1, 46, 80), (2, 18, 22), (1, 17, 19), (1, 33, 47), (9, 136, 240)]


def tol_pass(act):
    op = torch.float16 if act == torch.float32 else act
    return 2 * U[op] + U[act] + 1e-4


@pytest.fixture(scope="module")
def lib():
    rc._build.build()
    return rc._cabi.load()


def tv_block():
    from torchvision.models.optical_flow.raft import RecurrentBlock
    return RecurrentBlock(input_size=256, hidden_size=128)


def seeded_block(seed=0):
    torch.manual_seed(seed)
    rb = rc.RecurrentBlock(input_size=256, hidden_size=128)
    return rb


# ------------------------------------------------------------------ CPU
def test_state_dict_matches_torchvision():
    ours, tv = seeded_block(), tv_block()
    assert list(ours.state_dict().keys()) == list(tv.state_dict().keys())
    assert all(ours.state_dict()[k].shape == v.shape for k, v in tv.state_dict().items())
    ours.load_state_dict(tv.state_dict(), strict=True)
    tv2 = tv_block()
    tv2.load_state_dict(ours.state_dict(), strict=True)
    assert all(torch.equal(tv2.state_dict()[k], v) for k, v in tv.state_dict().items())
    assert ours.hidden_size == 128


@pytest.mark.parametrize("kw", [
    dict(input_size=256, hidden_size=96),
    dict(input_size=128, hidden_size=128),
    dict(input_size=146, hidden_size=96, kernel_size=(3,), padding=(1,)),          # raft_small's single 3x3 GRU
    dict(input_size=256, hidden_size=128, kernel_size=((5, 1), (1, 5)), padding=((2, 0), (0, 2))),
    dict(input_size=256, hidden_size=128, kernel_size=((1, 5), (5, 1)), padding=((0, 1), (1, 0))),
])
def test_unsupported_configurations_raise(kw):
    with pytest.raises(ValueError):
        rc.RecurrentBlock(**kw)


def _conv_from_packed(a, packed, n, axis):
    """What the kernel computes from the packed slabs: a (B, 384, H, W) float64, packed [6][5][n][64] -> (B, n, H, W)."""
    B, _, H, W = a.shape
    pad = ((0, 0), (0, 0), (0, 0), (2, 2)) if axis == 0 else ((0, 0), (0, 0), (2, 2), (0, 0))
    ap = np.pad(a, pad)
    out = np.zeros((B, n, H, W))
    for kb in range(6):
        for t in range(5):
            sh = ap[:, kb * 64:(kb + 1) * 64, :, t:t + W] if axis == 0 else ap[:, kb * 64:(kb + 1) * 64, t:t + H, :]
            out += np.einsum("bchw,nc->bnhw", sh, packed[kb, t])
    return out


@pytest.mark.parametrize("op", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("axis", [0, 1])
def test_packed_weights_reproduce_the_convolution(lib, op, axis):
    torch.manual_seed(3 + axis)
    gru = rc.recurrent_block._ConvGRU(256, 128, KS[axis], PAD[axis])
    ws = [np.ascontiguousarray(c.weight.detach().numpy()) for c in (gru.convz, gru.convr, gru.convq)]
    nbytes = lib.rdvc_corr_convgru_packed_weight_bytes()
    assert nbytes == (6 * 5 * 256 * 64 + 6 * 5 * 128 * 64) * 2
    packed = np.zeros(nbytes // 2, np.uint16)
    dt = rc.RDVC_DT_F16 if op == torch.float16 else rc.RDVC_DT_BF16
    _cabi.check(lib.rdvc_corr_convgru_pack_weights(ws[0].ctypes.data, ws[1].ctypes.data, ws[2].ctypes.data, dt,
                                              packed.ctypes.data), "pack")
    as_float = torch.from_numpy(packed.view(np.int16)).view(op).double().numpy()
    zr = as_float[:6 * 5 * 256 * 64].reshape(6, 5, 256, 64)
    q = as_float[6 * 5 * 256 * 64:].reshape(6, 5, 128, 64)
    a = torch.randn(2, 384, 9, 11).to(op).double()
    got = {"zr": _conv_from_packed(a.numpy(), zr, 256, axis), "q": _conv_from_packed(a.numpy(), q, 128, axis)}
    w16 = {k: c.weight.detach().to(op).double() for k, c in (("z", gru.convz), ("r", gru.convr), ("q", gru.convq))}
    want_zr = torch.cat([F.conv2d(a, w16["z"], padding=PAD[axis]), F.conv2d(a, w16["r"], padding=PAD[axis])], 1).numpy()
    want_q = F.conv2d(a, w16["q"], padding=PAD[axis]).numpy()
    assert np.abs(got["zr"] - want_zr).max() <= 1e-9 * np.abs(want_zr).max()
    assert np.abs(got["q"] - want_q).max() <= 1e-9 * np.abs(want_q).max()


def test_cabi_argument_errors(lib):
    A = 1 << 20           # a 16-byte aligned fake device address: every call below fails its checks before any access
    ws_need = lib.rdvc_corr_convgru_workspace_bytes(1, 8, 8, rc.RDVC_DT_F16)
    assert ws_need > 0 and lib.rdvc_corr_convgru_workspace_bytes(1, 8, 8, rc.RDVC_DT_F32) > ws_need
    assert lib.rdvc_corr_convgru_workspace_bytes(0, 8, 8, rc.RDVC_DT_F16) == 0
    assert lib.rdvc_corr_convgru_workspace_bytes(1, 8, 8, 7) == 0

    def call(**kw):
        a = dict(h=A, hps=128, c=A, cps=256, m=A + 256, mps=256, act=rc.RDVC_DT_F16, op=rc.RDVC_DT_F16, axis=0, B=1, H=8,
                 W=8, w=A, bz=A, br=A, bq=A, ws=A, wsb=ws_need, out=2 * A)
        a.update(kw)
        return lib.rdvc_corr_convgru(a["h"], a["hps"], a["c"], a["cps"], a["m"], a["mps"], a["act"], a["op"], a["axis"], a["B"],
                                a["H"], a["W"], a["w"], a["bz"], a["br"], a["bq"], a["ws"], a["wsb"], a["out"], None)
    assert call(h=None) == -1 and call(bq=None) == -1 and call(ws=None) == -1 and call(out=None) == -1
    assert call(B=0) == -2 and call(H=-1) == -2 and call(W=0) == -2
    assert call(act=9) == -4 and call(op=rc.RDVC_DT_F32) == -4
    assert call(act=rc.RDVC_DT_BF16, op=rc.RDVC_DT_F16) == -4            # 16-bit activations are their own operands
    assert call(axis=2) == -5 and call(cps=64) == -5 and call(out=A) == -5
    assert call(m=A + 8) == -7 and call(hps=132) == -7 and call(w=A + 2) == -7 and call(ws=A + 16) == -7
    assert call(act=rc.RDVC_DT_F32, hps=130) == -7
    assert call(wsb=ws_need - 1) == -6
    assert call(act=rc.RDVC_DT_F32, wsb=ws_need) == -6                  # fp32 activations need the larger workspace
    for rcode in (call(h=None), call(B=0)):
        assert rcode < 0 and _cabi.last_error()
    w = np.zeros(4, np.float32)
    assert lib.rdvc_corr_convgru_pack_weights(None, w.ctypes.data, w.ctypes.data, rc.RDVC_DT_F16, w.ctypes.data) == -1
    assert lib.rdvc_corr_convgru_pack_weights(w.ctypes.data, w.ctypes.data, w.ctypes.data, rc.RDVC_DT_F32, w.ctypes.data) == -4


def test_module_refusals_on_cpu():
    rb = seeded_block().eval()
    h, x = torch.randn(1, 128, 8, 8), torch.randn(1, 256, 8, 8)
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU fallback"):
        rb(h, x)
    with pytest.raises(RuntimeError, match="forward-only"):
        rb(h.requires_grad_(), x)
    rb.train()
    with pytest.raises(RuntimeError, match="forward-only"):
        rb(h.detach(), x)


# ------------------------------------------------------------------ GPU
def _r(t, dt):
    return t.to(dt).double()


def ref_pass(gru, h, ctx, mot, axis, op):
    """One ConvGRU in fp64 with the kernel's rounding points; h / ctx / mot in the activation dtype."""
    hd = h.double()
    w = {k: _r(getattr(gru, "conv" + k).weight.detach(), op) for k in "zrq"}
    b = {k: getattr(gru, "conv" + k).bias.detach().double() for k in "zrq"}
    hx = torch.cat([_r(h, op), _r(ctx, op), _r(mot, op)], 1)
    z = torch.sigmoid(F.conv2d(hx, w["z"], b["z"], padding=PAD[axis]))
    r = torch.sigmoid(F.conv2d(hx, w["r"], b["r"], padding=PAD[axis]))
    z16, rh16 = _r(z, op), _r(r * hd, op)
    q = torch.tanh(F.conv2d(torch.cat([rh16, _r(ctx, op), _r(mot, op)], 1), w["q"], b["q"], padding=PAD[axis]))
    return ((1 - z16) * hd + z16 * q).to(h.dtype)


def inputs(B, H, W, dt, seed, layout="channels_last"):
    g = torch.Generator(device="cuda").manual_seed(seed)
    h = torch.tanh(torch.randn(B, 128, H, W, device="cuda", generator=g))
    x = torch.relu(torch.randn(B, 256, H, W, device="cuda", generator=g))
    x[:, :128] = torch.tanh(x[:, :128])
    h, x = h.to(dt), x.to(dt)
    if layout == "channels_last":
        h, x = h.contiguous(memory_format=torch.channels_last), x.contiguous(memory_format=torch.channels_last)
    return h, x


def stock_out(rb, h, x):
    tv = tv_block().cuda().eval()
    tv.load_state_dict(rb.state_dict())
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad(), torch.autocast("cuda", dtype=h.dtype, enabled=h.dtype != torch.float32):
            return tv(h, x)
    finally:
        torch.backends.cudnn.allow_tf32 = prev


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [torch.float32, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("shape", SHAPES)
def test_block_matches_fp64_and_stock(lib, shape, dt):
    B, H, W = shape
    rb = seeded_block(1).cuda().eval()
    h, x = inputs(B, H, W, dt, seed=H * W + B)
    op = torch.float16 if dt == torch.float32 else dt
    with torch.no_grad():
        got = rb(h, x)
        assert got.dtype == dt and got.shape == h.shape and got.is_contiguous(memory_format=torch.channels_last)
        mid = ref_pass(rb.convgru1, h, x[:, :128], x[:, 128:], 0, op)
        ref = ref_pass(rb.convgru2, mid, x[:, :128], x[:, 128:], 1, op)
        err = (got.double() - ref.double()).abs()
        assert err.max().item() <= 2 * tol_pass(dt), err.max().item()
        assert err.mean().item() <= 0.1 * tol_pass(dt), err.mean().item()
        assert (got.float() - stock_out(rb, h, x).float()).abs().max().item() <= TOL_STOCK[dt]


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [torch.float32, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("layout", ["nchw", "channels_last", "slice"])
def test_layouts_and_channel_slices(lib, dt, layout):
    """NCHW in -> NCHW out, channels_last in -> channels_last out, and x given as channel-slice views (forward_parts on
    x[:, :128] / x[:, 128:] of a channels_last tensor, what raft_flow passes) -- all the same numbers."""
    B, H, W = 2, 18, 22
    rb = seeded_block(2).cuda().eval()
    h, x = inputs(B, H, W, dt, seed=7, layout="nchw" if layout == "nchw" else "channels_last")
    with torch.no_grad():
        ref = rb(h.contiguous(memory_format=torch.channels_last), x.contiguous(memory_format=torch.channels_last))
        if layout == "slice":
            c, m = x[:, :128], x[:, 128:]
            assert c.stride(1) == 1 and c.stride(3) == 256          # views, not copies
            got = rb.forward_parts(h, c, m)
        else:
            got = rb(h, x)
    if layout == "nchw":
        assert got.is_contiguous()
    else:
        assert got.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(got, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [torch.float32, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("axis", [0, 1])
def test_single_pass_through_the_abi(lib, dt, axis):
    """One rdvc_corr_convgru call per tap axis against the fp64 rounding-point evaluation."""
    rb = seeded_block(4).cuda().eval()
    gru = (rb.convgru1, rb.convgru2)[axis]
    op = torch.float16 if dt == torch.float32 else dt
    for (B, H, W) in [(1, 17, 19), (2, 33, 47)]:
        h, x = inputs(B, H, W, dt, seed=11 + axis)
        pk = PackedConvGRU(gru, op, "cuda")
        ws_bytes = lib.rdvc_corr_convgru_workspace_bytes(B, H, W, rc.RDVC_DT_F32 if dt == torch.float32 else
                                                    (rc.RDVC_DT_F16 if dt == torch.float16 else rc.RDVC_DT_BF16))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        out = torch.empty(B, H, W, 128, dtype=dt, device="cuda")
        adt = {torch.float32: rc.RDVC_DT_F32, torch.float16: rc.RDVC_DT_F16, torch.bfloat16: rc.RDVC_DT_BF16}
        _cabi.check(lib.rdvc_corr_convgru(h.data_ptr(), 128, x.data_ptr(), 256, x.data_ptr() + 128 * x.element_size(), 256,
                                     adt[dt], adt[op], axis, B, H, W, pk.weight.data_ptr(), pk.bias_z.data_ptr(),
                                     pk.bias_r.data_ptr(), pk.bias_q.data_ptr(), ws.data_ptr(), ws_bytes, out.data_ptr(),
                                     torch.cuda.current_stream().cuda_stream), "rdvc_corr_convgru")
        ref = ref_pass(gru, h, x[:, :128], x[:, 128:], axis, op)
        err = (out.permute(0, 3, 1, 2).double() - ref.double()).abs().max().item()
        assert err <= tol_pass(dt), (B, H, W, err)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [torch.float32, torch.float16])
def test_no_out_of_bounds_writes(lib, dt):
    """Guard bands before and after the workspace and the output survive, and every output element is written (the
    buffers start as 0xFF bytes: NaN in fp16 and fp32), on odd shapes."""
    GUARD = 4096
    adt = rc.RDVC_DT_F32 if dt == torch.float32 else rc.RDVC_DT_F16
    rb = seeded_block(5).cuda().eval()
    st = torch.cuda.current_stream().cuda_stream
    for (B, H, W) in [(1, 17, 19), (2, 9, 13), (1, 33, 47), (3, 5, 7)]:
        h, x = inputs(B, H, W, dt, seed=B * H * W)
        for axis, gru in enumerate((rb.convgru1, rb.convgru2)):
            pk = PackedConvGRU(gru, torch.float16, "cuda")
            sizes = {"ws": lib.rdvc_corr_convgru_workspace_bytes(B, H, W, adt), "out": B * H * W * 128 * h.element_size()}
            bufs = {k: torch.full((n + 2 * GUARD,), 0xFF, dtype=torch.uint8, device="cuda") for k, n in sizes.items()}
            ptr = {k: v.data_ptr() + GUARD for k, v in bufs.items()}
            _cabi.check(lib.rdvc_corr_convgru(h.data_ptr(), 128, x.data_ptr(), 256, x.data_ptr() + 128 * h.element_size(), 256,
                                         adt, rc.RDVC_DT_F16, axis, B, H, W, pk.weight.data_ptr(), pk.bias_z.data_ptr(),
                                         pk.bias_r.data_ptr(), pk.bias_q.data_ptr(), ptr["ws"], sizes["ws"], ptr["out"], st),
                        "rdvc_corr_convgru")
            torch.cuda.synchronize()
            for k, v in bufs.items():
                assert bool((v[:GUARD] == 0xFF).all()) and bool((v[-GUARD:] == 0xFF).all()), (k, (B, H, W), axis)
            out = bufs["out"][GUARD:-GUARD].view(dt)
            assert torch.isfinite(out).all(), ((B, H, W), axis)


@pytest.mark.gpu
def test_deterministic_on_the_callers_stream(lib):
    """Two calls give the same bits; the work is enqueued on the caller's stream (a graph captured on a side stream
    replays it -- a launch on any other stream would break the capture) and the replay gives the same bits again."""
    rb = seeded_block(6).cuda().eval()
    h, x = inputs(2, 46, 80, torch.float16, seed=3)
    with torch.no_grad():
        a = rb(h, x)
        b = rb(h, x)
        assert torch.equal(a, b)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            c = rb(h, x)
        torch.cuda.current_stream().wait_stream(side)
        assert torch.equal(a, c)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            d = rb(h, x)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(a, d)


@pytest.mark.gpu
def test_new_weights_are_repacked(lib):
    rb = seeded_block(7).cuda().eval()
    h, x = inputs(1, 33, 47, torch.float32, seed=9)
    other = seeded_block(8).cuda().eval()
    with torch.no_grad():
        before = rb(h, x)
        rb.load_state_dict(other.state_dict())
        after = rb(h, x)
        assert not torch.equal(before, after)
        assert torch.equal(after, other(h, x))
        rb.convgru2.convq.bias.add_(0.5)                        # an in-place change bumps the version: re-packed too
        assert not torch.equal(rb(h, x), after)


# ------------------------------------------------------------------ RAFT end to end
def _seeded_raft(swap):
    from torchvision.models.optical_flow import raft_large
    torch.manual_seed(0)
    model = raft_large(weights=None, corr_block=rc.TVCorrBlock()).eval().cuda()
    if swap:
        rb = rc.RecurrentBlock(input_size=256, hidden_size=128)
        rb.load_state_dict(model.update_block.recurrent_block.state_dict())
        model.update_block.recurrent_block = rb.cuda()
    return model


def _stock_raft():
    from torchvision.models.optical_flow import raft_large
    torch.manual_seed(0)
    return raft_large(weights=None).eval().cuda()


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
@pytest.mark.parametrize("case", ["368x640", "1080p"])
def test_raft_epe_vs_stock(lib, golden_dir, case, amp):
    a, b = _frames(golden_dir, (368, 640)) if case == "368x640" else _synthetic_1080p()
    model = _seeded_raft(True)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=amp):
        ref = _stock_raft()(a, b, num_flow_updates=12)[-1]
        got = rc.raft_flow(model, a, b, 12)
        plain = rc.raft_flow(_seeded_raft(False), a, b, 12)
    assert isinstance(model.update_block.recurrent_block, rc.RecurrentBlock)
    assert torch.isfinite(got).all()
    assert _epe(got, ref) < TOL_EPE, _epe(got, ref)
    assert _epe(got, plain) < TOL_EPE


@pytest.mark.gpu
def test_raft_sequence_and_graphs(lib, golden_dir):
    """raft_flow_sequence == the pair-wise calls (the existing sequence test's tolerance), GraphedRaftFlow == eager bit
    for bit, and a graph captured before the channels_last weight move re-captures after it."""
    a, b = _frames(golden_dir, (256, 448))
    frames = torch.cat([a, b, torch.roll(a, (3, -5), (2, 3))], 0)
    model = _seeded_raft(True)
    with torch.no_grad():
        pairs = rc.raft_flow(model, frames[:-1], frames[1:], 12)
        seq = rc.raft_flow_sequence(model, frames, 12)
    assert _epe(seq, pairs) < 2e-3
    runner = rc.GraphedRaftFlow(model, 12)
    with torch.no_grad():
        eager = rc.raft_flow(model, a, b, 12)
    assert torch.equal(runner(a, b), eager) and torch.equal(runner(a, b), eager)
    assert torch.equal(runner.sequence(frames), seq)
    runner.release()

    model = _seeded_raft(True)
    rb = model.update_block.recurrent_block
    runner = rc.GraphedRaftFlow(model, 12, update_block_channels_last=False)
    with torch.no_grad():
        nchw = rc.raft_flow(model, a, b, 12, update_block_channels_last=False)
        assert torch.equal(runner(a, b), nchw)
        ptr0 = rb.convgru1.convz.weight.data_ptr()
        nhwc = rc.raft_flow(model, a, b, 12)                             # moves the update block's weights to NHWC
        assert rb.convgru1.convz.weight.data_ptr() != ptr0
        assert _epe(nhwc, nchw) < 2e-3
        again = runner(a, b)                                             # weights moved -> re-captured, re-packed
        assert len(runner._entries) == 1
        assert _epe(again, nchw) < 2e-3
        assert torch.equal(runner(b, a), rc.raft_flow(model, b, a, 12, update_block_channels_last=False))
    runner.release()
