"""RAFT's context encoder (torchvision FeatureEncoder with norm_layer=BatchNorm2d in eval mode, TV:raft.py:116-168) with
BatchNorm folded into tcgen05 convolutions.

CPU part (-m "not gpu"): parameter tree and strict state_dict round trips against torchvision's class, the refused
configurations, the host fold + pack evaluated the way the kernels walk it (the stem's polyphase unrolling at odd H and
W, the 96-channel padding, the fused downsample's slab and bias layout), the packing key, the C ABI's argument errors
and size queries, the module refusals, the kernels' SASS and their spill-free register allocation.
GPU part (-m gpu): each layer kind against fp64 on the kernel's own inputs (read back from the workspace, which keeps
every intermediate), the whole module against the fp64 chain and against stock torchvision, NaN-filled workspaces,
determinism / streams / graphs / batch composition / input layouts, re-packing, and RAFT end to end.  Every test uses
random BatchNorm statistics and affine parameters: with torchvision's default init the fold is the identity.

Rounding points of the kernels (u = unit roundoff of the operand type: 2^-11 fp16, 2^-8 bf16):
  BatchNorm folded in fp64 and each weight rounded once to the operand type, each bias once to fp32; the image rounded
  to the operand type; every convolution accumulated in fp32 (K <= 9 x 128) with bias, ReLU, residual add and the
  outer ReLU in fp32; every intermediate activation rounded once to the operand type; the last layer rounded once to
  the output dtype (fp32 for fp32 images: no rounding).
Tolerances (absolute, per element):
  * one layer vs fp64 on the kernel's own inputs, result rounded like the kernel ... 2 u |ref| + 2e-4 max(1, |ref|max)
      a value within fp32 accumulation error (~sqrt(K) 2^-24 of O(1) terms) of a rounding boundary may round the
      other way: one ulp, 2 u |ref|.
  * the stem operand ........................................ exact (a permutation of the rounded image and zeros)
  * padded channels 96-127 of layer2's activations ........ exact zeros
  * whole module vs the fp64 chain .......................... 4 u_op max |ref| (fp16) / 8 u_op max |ref| (bf16): the
      chain is 16 layers deep and an intermediate on a rounding boundary moves the next layer by one ulp of its input.
  * vs stock torchvision (cuDNN, TF32 off for fp32; autocast for 16-bit) ... 2e-2 (fp32, fp16), 1e-1 (bf16) of
      max(1, max |stock|): the stock fp32 path keeps fp32 operands; the autocast path rounds BatchNorm's output, not a
      folded weight.
  * RAFT flow vs stock torchvision, mean EPE ................ < 0.05 px
A wrong tap, phase, channel or slab shows up as an O(1) relative error.
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
from rdvc_corr_b200.context_encoder import PackedContextEncoder, _convs_and_norms

U = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8}
CHAIN = {torch.float16: 4, torch.bfloat16: 8}
TOL_STOCK = {torch.float32: 2e-2, torch.float16: 2e-2, torch.bfloat16: 1e-1}
TOL_EPE = 0.05
DTYPES = [torch.float32, torch.float16, torch.bfloat16]
ADT = {torch.float32: rc.RDVC_DT_F32, torch.float16: rc.RDVC_DT_F16, torch.bfloat16: rc.RDVC_DT_BF16}
PKG = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                   "pfe-raft-and-hyperprior-based-learned-video-compression_b200")
SMALL = [(1, 36, 52), (2, 70, 98), (1, 37, 53), (1, 368, 640)]
# (geometry, N, epilogue) of every kernel instantiation, per operand dtype (csrc/context_encoder_sm100.cuh)
INSTANCES = [(2, 64, 0, "P"), (0, 64, 0, "P"), (0, 64, 1, "P"), (0, 128, 0, "P"), (0, 128, 1, "P"), (1, 128, 2, "P"),
             (3, 256, 3, "P"), (3, 256, 3, "float"), (3, 256, 4, "P"), (3, 256, 4, "float")]


@pytest.fixture(scope="module")
def lib():
    rc._build.build()
    return rc._cabi.load()


def tv_fe(**kw):
    from torchvision.models.optical_flow.raft import FeatureEncoder
    return FeatureEncoder(norm_layer=torch.nn.BatchNorm2d, **kw)


def randomize_bn(module, seed):
    """Random running statistics (variance in [0.5, 2]) and affine parameters in every BatchNorm of ``module``."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for m in module.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                c = m.num_features
                m.running_mean.copy_(0.5 * torch.randn(c, generator=g))
                m.running_var.copy_(0.5 + 1.5 * torch.rand(c, generator=g))
                m.weight.copy_(0.5 + torch.rand(c, generator=g))
                m.bias.copy_(0.3 * torch.randn(c, generator=g))
    return module


def seeded(seed=0):
    torch.manual_seed(seed)
    return randomize_bn(rc.ContextEncoder(), seed + 100).eval()


def folded(conv, bn):
    """fp64 w' = w s, b' = beta + (b - mean) s, s = gamma / sqrt(var + eps)."""
    w, b = conv.weight.detach().double().cpu(), conv.bias.detach().double().cpu()
    if bn is None:
        return w, b
    s = bn.weight.detach().double().cpu() / torch.sqrt(bn.running_var.detach().double().cpu() + bn.eps)
    return w * s[:, None, None, None], bn.bias.detach().double().cpu() + (b - bn.running_mean.detach().double().cpu()) * s


def pack(lib, ce, op):
    """(unit weights as fp64 arrays keyed by unit, unit biases) of the library's host packing."""
    pk = PackedContextEncoder(_convs_and_norms(ce), op, "cpu", None)
    w = pk.weight.view(op).double().numpy()
    b = pk.bias.double().numpy()
    units = [("stem", 64, 1, 4, 64), *[("s1", 64, 1, 9, 64)] * 4, ("s2", 128, 1, 10, 256),
             *[("s1", 128, 2, 9, 128)] * 3, ("s2", 128, 2, 10, 256), *[("s1", 128, 2, 9, 128)] * 3,
             ("1x1", 256, 2, 1, 256)]
    out, wo, bo = [], 0, 0
    for kind, n, kb, slabs, nb in units:
        size = kb * slabs * n * 64
        out.append((kind, w[wo:wo + size].reshape(kb, slabs, n, 64), b[bo:bo + nb]))
        wo, bo = wo + size, bo + nb
    assert wo == w.size and bo == b.size
    return out


def stem_operand(img):
    """The stem's GEMM operand (B, H1, W1, 64) from an image (B, 3, H, W): column k < 48 is tx = k // 12,
    py = k % 12 // 6, px = k % 6 // 3, c = k % 3 -> img[c, 2 Y + py, 2 (X + tx - 2) + px]."""
    B, _, H, W = img.shape
    H1, W1 = (H + 1) // 2, (W + 1) // 2
    pad = torch.zeros(B, 3, 2 * H1 + 2, 2 * W1 + 8, dtype=img.dtype, device=img.device)
    pad[:, :, :H, 4:4 + W] = img                           # x offset 4: taps reach 4 pixels left
    out = torch.zeros(B, H1, W1, 64, dtype=img.dtype, device=img.device)
    for k in range(48):
        tx, py, px, c = k // 12, k % 12 // 6, k % 6 // 3, k % 3
        out[..., k] = pad[:, c, py:py + 2 * H1:2, 4 + 2 * (tx - 2) + px::2][:, :, :W1]
    return out


# ------------------------------------------------------------------ CPU
def test_state_dict_matches_torchvision():
    ours, tv, tv2 = seeded(), randomize_bn(tv_fe(), 5), tv_fe()
    assert list(ours.state_dict().keys()) == list(tv.state_dict().keys())
    assert "layer3.1.convnormrelu2.1.num_batches_tracked" in ours.state_dict() and "conv.bias" in ours.state_dict()
    assert all(ours.state_dict()[k].shape == v.shape for k, v in tv.state_dict().items())
    ours.load_state_dict(tv.state_dict(), strict=True)
    tv2.load_state_dict(ours.state_dict(), strict=True)
    assert all(torch.equal(tv2.state_dict()[k], v) for k, v in tv.state_dict().items())


@pytest.mark.parametrize("kw", [dict(norm_layer=torch.nn.InstanceNorm2d), dict(norm_layer=None),
                                dict(layers=(32, 32, 64, 96, 160)), dict(strides=(1, 1, 2, 2)),
                                dict(layers=(64, 64, 96, 128, 128)), "bottleneck"])
def test_unsupported_configurations_raise(kw):
    if kw == "bottleneck":
        from torchvision.models.optical_flow.raft import BottleneckBlock
        kw = dict(block=BottleneckBlock, layers=(32, 32, 64, 96, 160), norm_layer=None)
    with pytest.raises(ValueError, match="raft_large's context encoder"):
        rc.ContextEncoder(**kw)


def _tol_conv(x, layer, stride, pad, u):
    """Bound on the effect of rounding each folded weight once (u * conv(|x|, |w'|)) and each bias to fp32."""
    w, b = folded(*layer)
    return u * F.conv2d(x.abs(), w.abs(), None, stride=stride, padding=pad) + 2.0 ** -24 * b.abs().max().item() + 1e-12


@pytest.mark.parametrize("op", [torch.float16, torch.bfloat16])
def test_packed_operand_reproduces_the_folded_convolutions(lib, op):
    """The host fold + pack walked the way the kernels walk it, against fp64 F.conv2d + eval F.batch_norm: the stem
    as a 4x1 GEMM over the polyphase operand (odd H and W), a stride-2 unit with its fused downsample (96 channels
    padded to 128), a 96-channel 3x3 and the 1x1; every padded row, column and bias is zero."""
    ce = seeded(1)
    units = pack(lib, ce, op)
    layers = _convs_and_norms(ce)
    u = U[op]
    g = torch.Generator().manual_seed(2)

    def stock(i, x, stride, pad):
        conv, bn = layers[i]
        y = F.conv2d(x, conv.weight.double(), conv.bias.double(), stride=stride, padding=pad)
        if bn is None:
            return y
        return F.batch_norm(y, bn.running_mean.double(), bn.running_var.double(), bn.weight.double(), bn.bias.double(),
                            False, 0.0, bn.eps)

    with torch.no_grad():
        # the stem: 4 vertical taps ty at rows Y + ty - 2 of the operand
        img = torch.rand(2, 3, 13, 21, generator=g, dtype=torch.float64)
        S = stem_operand(img)                                                  # (B, H1, W1, 64)
        _, w0, b0 = units[0]
        H1, W1 = S.shape[1:3]
        Sp = F.pad(S, (0, 0, 0, 0, 2, 1))
        got = sum(torch.einsum("byxk,nk->bnyx", Sp[:, ty:ty + H1], torch.from_numpy(w0[0, ty])) for ty in range(4))
        got = got + torch.from_numpy(b0)[None, :, None, None]
        want = stock(0, img, 2, 3)
        assert got.shape == want.shape
        assert ((got - want).abs() <= _tol_conv(img, layers[0], 2, 3, u)).all()
        assert not w0[0, :, :, 48:].any()
        # stride-2 unit 5: layer2.0.convnormrelu1 (taps 0-8) + downsample (slab 9) over 64 channels, N = 128
        x = torch.rand(1, 64, 9, 11, generator=g, dtype=torch.float64)
        _, w5, b5 = units[5]
        xp = F.pad(x, (1, 1, 1, 1))
        Ho, Wo = 5, 6
        acc = torch.zeros(1, 128, Ho, Wo, dtype=torch.float64)
        for t in range(9):
            dy, dx = divmod(t, 3)
            a = xp[:, :, dy:dy + 2 * Ho:2, dx:dx + 2 * Wo:2]
            acc += torch.einsum("bcyx,nc->bnyx", a, torch.from_numpy(w5[0, t]))
        ds = torch.einsum("bcyx,nc->bnyx", x[:, :, ::2, ::2], torch.from_numpy(w5[0, 9]))
        acc += torch.from_numpy(b5[:128])[None, :, None, None]
        ds += torch.from_numpy(b5[128:])[None, :, None, None]
        assert ((acc[:, :96] - stock(5, x, 2, 1)).abs() <= _tol_conv(x, layers[5], 2, 1, u)).all()
        assert ((ds[:, :96] - stock(6, x, 2, 0)).abs() <= _tol_conv(x, layers[6], 2, 0, u)).all()
        assert not w5[:, :, 96:].any() and not b5[96:128].any() and not b5[224:].any()
        # unit 7 (layer2.1.convnormrelu1): 96 input channels in two k-blocks, the second half padding
        x = torch.rand(1, 96, 6, 7, generator=g, dtype=torch.float64)
        _, w7, b7 = units[7]
        xp = F.pad(torch.cat([x, torch.zeros(1, 32, 6, 7, dtype=torch.float64)], 1), (1, 1, 1, 1))
        acc = torch.zeros(1, 128, 6, 7, dtype=torch.float64)
        for kb in range(2):
            for t in range(9):
                dy, dx = divmod(t, 3)
                acc += torch.einsum("bcyx,nc->bnyx", xp[:, kb * 64:(kb + 1) * 64, dy:dy + 6, dx:dx + 7],
                                    torch.from_numpy(w7[kb, t]))
        acc += torch.from_numpy(b7)[None, :, None, None]
        assert ((acc[:, :96] - stock(8, x, 1, 1)).abs() <= _tol_conv(x, layers[8], 1, 1, u)).all()
        assert not w7[1, :, :, 32:].any() and not w7[:, :, 96:].any()
        # the 1x1 (no BatchNorm)
        x = torch.rand(1, 128, 3, 4, generator=g, dtype=torch.float64)
        _, w13, b13 = units[13]
        acc = sum(torch.einsum("bcyx,nc->bnyx", x[:, kb * 64:(kb + 1) * 64], torch.from_numpy(w13[kb, 0])) for kb in range(2))
        acc += torch.from_numpy(b13)[None, :, None, None]
        assert ((acc - stock(15, x, 1, 0)).abs() <= _tol_conv(x, layers[15], 1, 0, u)).all()
        # each weight rounded once from the fp64 fold: within half an ulp
        wf, bf = folded(*layers[1])
        p = torch.from_numpy(units[1][1][0]).permute(1, 2, 0).reshape(64, 64, 3, 3)     # [t][n][c] -> [n][c][ky][kx]
        assert ((p - wf).abs() <= u * wf.abs() * (1 + 1e-12) + 2.0 ** -25).all()     # 2^-25: fp16 subnormals
        assert np.array_equal(units[1][2], bf.float().double().numpy())


def test_packing_key_covers_running_stats():
    """A load_state_dict that changes only running statistics (buffers, not parameters) changes the packing key."""
    ce = seeded(2)
    k0 = ce._key(torch.float16, "cuda")
    sd = ce.state_dict()
    sd["layer2.1.convnormrelu1.1.running_var"] = sd["layer2.1.convnormrelu1.1.running_var"] * 1.5
    ce.load_state_dict(sd)
    assert ce._key(torch.float16, "cuda") != k0
    k1 = ce._key(torch.float16, "cuda")
    ce.layer1[0].convnormrelu1[1].eps = 1e-3
    assert ce._key(torch.float16, "cuda") != k1


def test_cabi_argument_errors(lib):
    A = 1 << 20           # a 16-byte aligned fake device address: every call below fails its checks before any access
    B, H, W = 1, 37, 53
    strides = (ctypes.c_longlong * 4)(3 * H * W, H * W, W, 1)
    assert lib.rdvc_corr_context_encoder_packed_bias_bytes() == 4 * (64 * 5 + 256 + 128 * 3 + 256 + 128 * 3 + 256)
    assert lib.rdvc_corr_context_encoder_packed_weight_bytes() == 2 * 64 * (
        4 * 64 + 4 * 9 * 64 + 10 * 128 + 3 * 2 * 9 * 128 + 2 * 10 * 128 + 3 * 2 * 9 * 128 + 2 * 256)
    ws = lib.rdvc_corr_context_encoder_workspace_bytes(B, H, W, rc.RDVC_DT_F16)
    a256 = lambda x: (x + 255) // 256 * 256                                          # noqa: E731
    assert ws == 6 * a256(19 * 27 * 64 * 2) + 5 * a256(10 * 14 * 128 * 2) + 5 * a256(5 * 7 * 128 * 2)
    assert lib.rdvc_corr_context_encoder_workspace_bytes(B, H, W, rc.RDVC_DT_F32) == ws
    assert lib.rdvc_corr_context_encoder_workspace_bytes(0, H, W, rc.RDVC_DT_F16) == 0
    assert lib.rdvc_corr_context_encoder_workspace_bytes(B, H, W, 7) == 0
    OUT = 1 << 30

    def ce(**kw):
        a = dict(img=A, s=strides, idt=rc.RDVC_DT_F32, B=B, H=H, W=W, op=rc.RDVC_DT_F16, w=A, b=A,
                 form=_cabi.RDVC_CE_OUT_SPLIT, ws=1 << 28, wsb=ws, out=OUT, ps=256, odt=rc.RDVC_DT_F32)
        a.update(kw)
        return lib.rdvc_corr_context_encoder(a["img"], a["s"], a["idt"], a["B"], a["H"], a["W"], a["op"], a["w"], a["b"],
                                             a["form"], a["ws"], a["wsb"], a["out"], a["ps"], a["odt"], None)
    assert ce(img=None) == -1 and ce(s=None) == -1 and ce(w=None) == -1 and ce(b=None) == -1
    assert ce(ws=None) == -1 and ce(out=None) == -1
    assert ce(form=2) == -5 and ce(form=-1) == -5
    assert ce(B=0) == -2 and ce(H=-1) == -2 and ce(W=0) == -2
    assert ce(idt=9) == -4 and ce(op=rc.RDVC_DT_F32) == -4 and ce(odt=rc.RDVC_DT_BF16) == -4
    assert ce(s=(ctypes.c_longlong * 4)(-1, 1, 1, 1)) == -5
    assert ce(H=1 << 24) == -5
    assert ce(img=A + 2) == -7 and ce(w=A + 8) == -7 and ce(b=A + 4) == -7 and ce(out=OUT + 8) == -7
    assert ce(ps=128) == -5 and ce(ps=258) == -7
    assert ce(wsb=ws - 1) == -6 and ce(ws=(1 << 28) + 16) == -7
    assert ce(out=A) == -5                                       # overlaps the image
    assert ce(out=(1 << 28) + 4096) == -5                        # inside the workspace
    for rcode in (ce(img=None), ce(form=5)):
        assert rcode < 0 and _cabi.last_error()
    f = np.zeros(4, np.float32)
    p16 = (ctypes.c_void_p * 16)(*([f.ctypes.data] * 16))
    eps = (ctypes.c_double * 16)(*([1e-5] * 16))
    out = np.zeros(4, np.float32)
    assert lib.rdvc_corr_context_encoder_pack_weights(None, p16, p16, p16, p16, p16, eps, rc.RDVC_DT_F16, out.ctypes.data,
                                                      out.ctypes.data) == -1
    assert lib.rdvc_corr_context_encoder_pack_weights(p16, p16, p16, p16, p16, p16, eps, rc.RDVC_DT_F16, out.ctypes.data,
                                                      None) == -1
    nul = (ctypes.c_void_p * 16)(*([f.ctypes.data] * 3 + [None] + [f.ctypes.data] * 12))
    assert lib.rdvc_corr_context_encoder_pack_weights(p16, p16, nul, p16, p16, p16, eps, rc.RDVC_DT_F16, out.ctypes.data,
                                                      out.ctypes.data) == -1
    assert lib.rdvc_corr_context_encoder_pack_weights(p16, p16, p16, p16, p16, p16, eps, rc.RDVC_DT_F32, out.ctypes.data,
                                                      out.ctypes.data) == -4


def test_module_refusals_on_cpu():
    ce = seeded(3)
    x = torch.rand(1, 3, 16, 16)
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            ce(x)
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            ce.forward_split(x)
    with pytest.raises(RuntimeError, match="forward-only"):
        ce(x.clone().requires_grad_())
    ce.train()
    with torch.no_grad(), pytest.raises(RuntimeError, match="eval mode"):         # train mode, even without grad
        ce(x)
    ce.eval()
    ce.layer2[1].convnormrelu2[1].train()                                         # one BatchNorm in train mode
    with torch.no_grad(), pytest.raises(RuntimeError, match="eval mode"):
        ce.forward_split(x)
    ce.eval()
    ce.layer1[0].convnormrelu1[1].track_running_stats = False
    with torch.no_grad(), pytest.raises(RuntimeError, match="eval mode"):
        ce(x)
    with pytest.raises(ValueError, match="hidden_size=128"):
        seeded(4).forward_split(x, hidden_size=96)


def test_sass_has_tcgen05_and_tma(lib):
    """Every instantiation of the context-encoder kernel is Blackwell-native: tcgen05.mma (UTCHMMA), TMA loads
    (UTMALDG) and TMEM reads (LDTM)."""
    out = subprocess.run(["cuobjdump", "-sass", rc._cabi.lib_path()], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    funcs = [f for f in out.stdout.split("Function : ") if f.startswith("_ZN4rdvc19context_conv_kernel")]
    assert len(funcs) == 2 * len(INSTANCES), len(funcs)
    for f in funcs:
        assert "UTCHMMA" in f and "UTMALDG" in f and "LDTM" in f, f.splitlines()[0]


def test_no_register_spills():
    """-Xptxas -v over every instantiation of the context-encoder kernel and the stem pack: no spills."""
    from rdvc_corr_b200 import _build
    inst = []
    for op in ("__half", "__nv_bfloat16"):
        for g, n, e, o in INSTANCES:
            inst.append(f"template __global__ void context_conv_kernel<{g}, {n}, {e}, {op if o == 'P' else o}, {op}>"
                        "(const __grid_constant__ CUtensorMap, const __grid_constant__ CUtensorMap, const CeParams);")
        for t in ("float", "__half", "__nv_bfloat16"):
            inst.append(f"template __global__ void ce_stem_pack_kernel<{t}, {op}>(const CeStemParams);")
    src = '#include "context_encoder_sm100.cuh"\nnamespace rdvc {\n' + "\n".join(inst) + "\n}\n"
    with tempfile.TemporaryDirectory() as d:
        cu = os.path.join(d, "spills.cu")
        with open(cu, "w") as f:
            f.write(src)
        res = subprocess.run([_build.nvcc_path(), "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                              "-Xptxas", "-v", "-I", os.path.join(PKG, "csrc"), "-c", cu, "-o", os.path.join(d, "s.o")],
                             capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-3000:]
    props = [ln for ln in res.stderr.splitlines() if "spill stores" in ln]
    assert len(props) == len(inst), res.stderr[-3000:]
    assert all("0 bytes spill stores, 0 bytes spill loads" in ln for ln in props), props


# ------------------------------------------------------------------ GPU
def _op(dt):
    return torch.float16 if dt == torch.float32 else dt


def _image(B, H, W, dt, seed, channels_last=False):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = (2 * torch.rand(B, 3, H, W, device="cuda", generator=g) - 1).to(dt)
    return x.contiguous(memory_format=torch.channels_last) if channels_last else x


def _sizes(H, W):
    H1, W1 = (H + 1) // 2, (W + 1) // 2
    H2, W2 = (H1 + 1) // 2, (W1 + 1) // 2
    return H1, W1, H2, W2, (H2 + 1) // 2, (W2 + 1) // 2


def run_abi(lib, ce, x, form, out_dt, op, ws=None):
    """The module's call through the C ABI with a caller-owned workspace; returns (out NHWC, the 16 intermediates as
    (B, C, h, w) fp64 views in the order of include/rdvc_corr.h, workspace)."""
    B, _, H, W = x.shape
    key = ce._key(op, x.device)
    pk = PackedContextEncoder(_convs_and_norms(ce), op, x.device, key)
    wsb = lib.rdvc_corr_context_encoder_workspace_bytes(B, H, W, ADT[out_dt])
    if ws is None:
        ws = torch.zeros(wsb, dtype=torch.uint8, device="cuda")
    H1, W1, H2, W2, H3, W3 = _sizes(H, W)
    out = torch.empty(B, H3, W3, 256, dtype=out_dt, device="cuda")
    strides = (ctypes.c_longlong * 4)(*x.stride())
    _cabi.check(lib.rdvc_corr_context_encoder(x.data_ptr(), strides, ADT[x.dtype], B, H, W, ADT[op], pk.weight.data_ptr(),
                                              pk.bias.data_ptr(), form, ws.data_ptr(), wsb, out.data_ptr(), 256,
                                              ADT[out_dt], torch.cuda.current_stream().cuda_stream), "context_encoder")
    planes, off = [], 0
    for n, (h, w, c) in enumerate([(H1, W1, 64)] * 6 + [(H2, W2, 128)] * 5 + [(H3, W3, 128)] * 5):
        size = B * h * w * c * 2
        planes.append(ws[off:off + size].view(op).view(B, h, w, c).permute(0, 3, 1, 2))
        off += (size + 255) // 256 * 256
    return out, planes, ws


class Chain:
    """fp64 evaluation with the kernels' rounding points."""

    def __init__(self, ce, op):
        self.op = op
        self.wb = []
        for conv, bn in _convs_and_norms(ce):
            w, b = folded(conv, bn)
            self.wb.append((w.to(op).double().cuda(), b.float().double().cuda()))

    def r(self, t):
        return t.to(self.op).double()

    def conv(self, i, x, stride, pad):
        w, b = self.wb[i]
        return F.conv2d(x, w, b, stride=stride, padding=pad)

    def block(self, x, i1, i2, ids=None):
        stride = 1 if ids is None else 2
        t = self.r(self.conv(i1, x, stride, 1).clamp_min(0))
        res = x if ids is None else self.r(self.conv(ids, x, 2, 0))
        return self.r((res + self.conv(i2, t, 1, 1).clamp_min(0)).clamp_min(0))

    def __call__(self, img):
        x = self.r(img)                                                 # the image rounded to the operand type
        x = self.r(self.conv(0, x, 2, 3).clamp_min(0))
        x = self.block(self.block(x, 1, 2), 3, 4)
        x = self.block(self.block(x, 5, 7, 6), 8, 9)
        x = self.block(self.block(x, 10, 12, 11), 13, 14)
        return self.conv(15, x, 1, 0)


def _split(raw):
    return torch.cat([torch.tanh(raw[:, :128]), raw[:, 128:].clamp_min(0)], 1)


def _layer_ok(got, ref, op):
    tol = 2 * U[op] * ref.abs() + 2e-4 * max(1.0, ref.abs().max().item())
    err = (got.double() - ref).abs()
    return bool((err <= tol).all()), err.max().item()


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("shape", SMALL)
def test_layers_vs_fp64_on_kernel_inputs(lib, shape, dt):
    """Each layer kind on the kernel's own inputs: the stem operand, the stem, 3x3 s1 with and without the residual
    epilogue, 3x3 s2 with the fused downsample (layer2 and layer3), the 1x1 RAW and SPLIT; padded channels zero."""
    B, H, W = shape
    op = _op(dt)
    ce = seeded(10).cuda()
    ch = Chain(ce, op)
    x = _image(B, H, W, dt, B * H * W)
    with torch.no_grad():
        raw, P, _ = run_abi(lib, ce, x, _cabi.RDVC_CE_OUT_RAW, dt, op)
        split, P2, _ = run_abi(lib, ce, x, _cabi.RDVC_CE_OUT_SPLIT, dt, op)
        torch.cuda.synchronize()
        assert torch.equal(stem_operand(x.to(op)).permute(0, 3, 1, 2), P[0])
        checks = [
            ("stem", P[1], ch.r(ch.conv(0, ch.r(x), 2, 3).clamp_min(0))),
            ("3x3", P[4], ch.r(ch.conv(3, P[3].double(), 1, 1).clamp_min(0))),
            ("3x3+res", P[5], ch.r((P[3].double() + ch.conv(4, P[4].double(), 1, 1).clamp_min(0)).clamp_min(0))),
            ("s2", P[6][:, :96], ch.r(ch.conv(5, P[5].double(), 2, 1).clamp_min(0))),
            ("s2-ds", P[7][:, :96], ch.r(ch.conv(6, P[5].double(), 2, 0))),
            ("layer2 res", P[8][:, :96], ch.r((P[7][:, :96].double() + ch.conv(7, P[6][:, :96].double(), 1, 1)
                                               .clamp_min(0)).clamp_min(0))),
            ("l3 s2", P[11], ch.r(ch.conv(10, P[10][:, :96].double(), 2, 1).clamp_min(0))),
            ("l3 s2-ds", P[12], ch.r(ch.conv(11, P[10][:, :96].double(), 2, 0))),
            ("l3 res", P[15], ch.r((P[13].double() + ch.conv(14, P[14].double(), 1, 1).clamp_min(0)).clamp_min(0))),
        ]
        fin = ch.conv(15, P[15].double(), 1, 0)
        if dt != torch.float32:
            fin_raw, fin_split = ch.r(fin), ch.r(_split(fin))
        else:
            fin_raw, fin_split = fin, _split(fin)
        checks += [("1x1 raw", raw.permute(0, 3, 1, 2), fin_raw), ("1x1 split", split.permute(0, 3, 1, 2), fin_split)]
        for name, got, ref in checks:
            ok, err = _layer_ok(got, ref, op)
            assert ok, (name, err)
        for i in range(6, 11):
            assert not P[i][:, 96:].any(), i                               # layer2's padded channels are zero
        assert all(torch.equal(a, b) for a, b in zip(P, P2))               # the forms differ only in the last epilogue
        # the residual epilogue is relu(res + relu(acc + b)), not relu(acc + b + res): the two differ here
        alt = ch.r((P[3].double() + ch.conv(4, P[4].double(), 1, 1)).clamp_min(0))
        assert (alt - P[5].double()).abs().max().item() > 0.1


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("shape", SMALL + [(9, 1088, 1920)])
def test_module_vs_fp64_chain_and_stock(lib, shape, dt):
    B, H, W = shape
    op = _op(dt)
    ce = seeded(11).cuda()
    x = _image(B, H, W, dt, 7 + B * H * W)
    amp = dt != torch.float32
    with torch.no_grad(), torch.autocast("cuda", dtype=op, enabled=amp):
        out = ce(x.float() if amp else x)                                  # autocast: fp32 image, 16-bit everything
        hs, cx = ce.forward_split(x.float() if amp else x)
    assert out.shape == (B, 256, (H + 7) // 8, (W + 7) // 8) and out.dtype == dt
    assert out.is_contiguous(memory_format=torch.channels_last)
    assert hs.shape == (B, 128, (H + 7) // 8, (W + 7) // 8) and hs.dtype == dt and cx.dtype == dt
    assert hs.data_ptr() + 128 * hs.element_size() == cx.data_ptr() and hs.stride(1) == 1 and hs.stride(3) == 256
    n = B if B < 9 else 1                                                  # the fp64 chain on sample 0 at 1080p
    with torch.no_grad():
        ref = Chain(ce, op)(x[:n].float() if amp else x[:n])
    scale = ref.abs().max().item()
    assert (out[:n].double() - ref).abs().max().item() <= CHAIN[op] * U[op] * scale
    sref = _split(ref)
    assert (torch.cat([hs[:n], cx[:n]], 1).double() - sref).abs().max().item() <= CHAIN[op] * U[op] * max(1.0, scale)
    tv = tv_fe().cuda().eval()
    tv.load_state_dict(ce.state_dict())
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad(), torch.autocast("cuda", dtype=op, enabled=amp):
            s = tv(x.float() if amp else x)
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    assert (out.float() - s.float()).abs().max().item() <= TOL_STOCK[dt] * max(1.0, s.abs().max().item())
    if B == 9:                                                             # batch composition: bit-identical samples
        with torch.no_grad(), torch.autocast("cuda", dtype=op, enabled=amp):
            for i in (0, 4, 8):
                assert torch.equal(ce(x[i:i + 1].float() if amp else x[i:i + 1]), out[i:i + 1])


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES)
def test_nan_workspace_layouts_streams_graphs_batches(lib, dt):
    """A NaN-filled workspace gives the bits of a zeroed one; repeated runs, a side stream, a CUDA graph replay,
    NCHW vs channels_last input and batch composition (sample i of B = 9 vs B = 1) are bit-identical."""
    B, H, W = 9, 70, 98
    op = _op(dt)
    ce = seeded(12).cuda()
    x = _image(B, H, W, dt, 3)
    with torch.no_grad():
        a, _, ws = run_abi(lib, ce, x, _cabi.RDVC_CE_OUT_SPLIT, dt, op)
        ws.fill_(255)                                                      # 0xFFFF: NaN in fp16 and bf16
        b, _, _ = run_abi(lib, ce, x, _cabi.RDVC_CE_OUT_SPLIT, dt, op, ws=ws)
        assert torch.equal(a, b)
        h0, c0 = ce.forward_split(x)
        assert torch.equal(torch.cat([h0, c0], 1), a.permute(0, 3, 1, 2))
        h1, c1 = ce.forward_split(x.contiguous(memory_format=torch.channels_last))
        assert torch.equal(h0, h1) and torch.equal(c0, c1)
        assert torch.equal(ce(x), ce(x))
        for i in (0, 5, 8):
            hi, ci = ce.forward_split(x[i:i + 1].clone())
            assert torch.equal(hi, h0[i:i + 1]) and torch.equal(ci, c0[i:i + 1])
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            s = ce(x)
        torch.cuda.current_stream().wait_stream(side)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            gout = ce(x)
        gr.replay()
        torch.cuda.synchronize()
        r = ce(x)
        assert torch.equal(s, r) and torch.equal(gout, r)


@pytest.mark.gpu
def test_repacking(lib):
    """Re-packed after a load_state_dict that changes only running statistics and after an in-place weight change."""
    ce = seeded(13).cuda()
    x = _image(1, 3 * 8 + 5, 41, torch.float32, 5)
    with torch.no_grad():
        a = ce(x).clone()
        other = randomize_bn(seeded(13), 999).cuda()                       # same convolutions, other BN statistics
        sd = ce.state_dict()
        for k, v in other.state_dict().items():
            if "running" in k:
                sd[k] = v
        ce.load_state_dict(sd)
        b = ce(x).clone()
        assert not torch.equal(a, b)
        fresh = seeded(13).cuda()
        fresh.load_state_dict(sd)
        assert torch.equal(b, fresh(x))
        ce.layer3[1].convnormrelu2[0].weight.mul_(1.5)
        c = ce(x)
        assert not torch.equal(b, c)
        fresh.layer3[1].convnormrelu2[0].weight.mul_(1.5)
        assert torch.equal(c, fresh(x))


# ------------------------------------------------------------------ RAFT end to end
def _seeded_raft(swap, corr_block=True):
    from torchvision.models.optical_flow import raft_large
    torch.manual_seed(0)
    model = raft_large(weights=None, **({"corr_block": rc.TVCorrBlock()} if corr_block else {}))
    randomize_bn(model.context_encoder, 77)
    model = model.eval().cuda()
    if swap is None:
        return model
    ce = rc.ContextEncoder()
    ce.load_state_dict(model.context_encoder.state_dict())
    model.context_encoder = ce.cuda().eval()
    if swap == "all":
        ub = model.update_block
        me, fh = rc.MotionEncoder(in_channels_corr=324), rc.FlowHead(in_channels=128, hidden_size=256)
        rb = rc.RecurrentBlock(input_size=256, hidden_size=128)
        mp = rc.MaskPredictor(in_channels=128, hidden_size=256, multiplier=model.mask_predictor.multiplier)
        me.load_state_dict(ub.motion_encoder.state_dict())
        fh.load_state_dict(ub.flow_head.state_dict())
        rb.load_state_dict(ub.recurrent_block.state_dict())
        mp.load_state_dict(model.mask_predictor.state_dict())
        ub.motion_encoder, ub.flow_head, ub.recurrent_block = me.cuda(), fh.cuda(), rb.cuda()
        model.mask_predictor = mp.cuda()
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
@pytest.mark.parametrize("swap", ["ce", "all"])
@pytest.mark.parametrize("case", ["368x640", "1080p"])
def test_raft_epe_vs_stock(lib, golden_dir, case, swap, amp):
    a, b = _frames(golden_dir, (368, 640)) if case == "368x640" else _synthetic_1080p()
    model = _seeded_raft(swap)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=amp):
        ref = _seeded_raft(None, corr_block=False)(a, b, num_flow_updates=12)[-1]
        got = rc.raft_flow(model, a, b, 12)
        unfused = rc.raft_flow(model, a, b, 12, fuse_convcorr1=False)
        stock_call = model(a, b, num_flow_updates=12)[-1]             # RAFT.forward with the drop-ins swapped in
    assert isinstance(model.context_encoder, rc.ContextEncoder)
    assert got.dtype == torch.float32 and got.shape == ref.shape
    for f in (got, unfused, stock_call):
        assert torch.isfinite(f).all()
        assert _epe(f, ref) < TOL_EPE, _epe(f, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("swap", ["ce", "all"])
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
