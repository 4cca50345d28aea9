"""RAFT's feature encoder (torchvision FeatureEncoder with norm_layer=InstanceNorm2d, TV:raft.py:116-168) as tcgen05
convolutions whose epilogues write per-tile InstanceNorm statistics, a finalize and an apply pass per layer.

CPU part (-m "not gpu"): parameter tree and strict state_dict round trips against torchvision's class, the refused
configurations, the identity-norm packing, the C ABI's argument errors and workspace arithmetic, SASS and registers of
the new kernels.
GPU part (-m gpu): each stage on its own inputs read back from the workspace (raw convolutions, mean / rstd, the three
apply forms, the padded channels), the dropped bias, the whole module against the fp64 chain and stock torchvision,
odd and smallest sizes, NaN-filled workspaces, determinism / streams / graphs / batch invariance, and RAFT end to end.
Images are 0.85 + 0.1 U(-1, 1): the stem's channels have a mean many times their standard deviation, so the
statistics are computed in the presence of cancellation.  Conv biases are random.

Rounding points of the kernels (u = unit roundoff of the operand type: 2^-11 fp16, 2^-8 bf16):
  each weight rounded once to the operand type (identity-norm packing: the scale is exactly 1); the image rounded to the
  operand type; every convolution accumulated in fp32 WITHOUT its bias (InstanceNorm cancels it) and its raw output y
  rounded once to the operand type; per-tile (mean, M2) of the rounded y in fp32, merged per sample in fp64, mean and
  rstd = 1 / sqrt(var + eps) rounded once to fp32; the apply evaluated in fp32 and rounded once to the operand type;
  the final 1x1 with its bias rounded once to the output dtype (fp32 for fp32 images: no rounding).
Tolerances (absolute, per element):
  * raw convolution vs fp64 on the kernel's input ......... 2 u |ref| + 2e-4 max(1, max |ref|) (as for the context encoder)
  * mean / rstd vs fp64 over the stored raw values ........ 1e-5 relative (mean: of |mean| + std): fp32 tile partials
  * apply vs fp64 on the kernel's y and mean / rstd ........ u |ref| + 1e-6 (|IN(y)| + |other term|) + 2^-24: one
      rounding, after an fp32 evaluation a few fp32 ulps from fp64
  * padded channels 96-127 ................................ exact zeros
  * whole module vs the fp64 chain ......................... 16 u max |ref|: 15 normalised layers, each of whose inputs
      may sit one ulp away from the chain's after a rounding-boundary flip
  * vs stock torchvision (TF32 off for fp32; autocast for 16-bit) ... 2e-2 (fp32, fp16), 1e-1 (bf16) of max(1, |stock|)
  * RAFT flow vs stock torchvision, mean EPE ................ < 0.05 px
A wrong tap, tile, channel, statistic or form shows up as an O(1) error.
"""
import ctypes
import functools
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import rdvc_corr_b200 as rc
from rdvc_corr_b200 import _cabi
from rdvc_corr_b200.context_encoder import _convs_and_norms
from rdvc_corr_b200.feature_encoder import PackedFeatureEncoder

PKG = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                   "pfe-raft-and-hyperprior-based-learned-video-compression_b200")
U = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8}
TOL_STOCK = {torch.float32: 2e-2, torch.float16: 2e-2, torch.bfloat16: 1e-1}
TOL_EPE = 0.05
DTYPES = [torch.float32, torch.float16, torch.bfloat16]
ADT = {torch.float32: rc.RDVC_DT_F32, torch.float16: rc.RDVC_DT_F16, torch.bfloat16: rc.RDVC_DT_BF16}
# odd sizes with tail tiles, the smallest legal size (layer3 plane 1 x 2), odd tile counts, RAFT's size
SMALL = [(1, 37, 53), (2, 70, 98), (1, 8, 9), (3, 24, 40), (1, 368, 640)]
G_S1, G_S2, G_STEM = 0, 1, 2
STATS, DS_STATS = 9, 10
IN_INSTANCES = [(G_STEM, 64, STATS), (G_S1, 64, STATS), (G_S1, 128, STATS), (G_S2, 128, DS_STATS)]
OPS = ("__half", "__nv_bfloat16")
NT = [64] * 5 + [256, 128, 128, 128, 256, 128, 128, 128]         # per normalised unit


@pytest.fixture(scope="module")
def lib():
    rc._build.build()
    return rc._cabi.load()


def tv_fe(**kw):
    from torchvision.models.optical_flow.raft import FeatureEncoder
    return FeatureEncoder(norm_layer=torch.nn.InstanceNorm2d, **kw)


def randomize_bias(module, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for m in module.modules():
            if isinstance(m, torch.nn.Conv2d):
                m.bias.copy_(0.3 * torch.randn(m.out_channels, generator=g))
    return module


def seeded(seed=0):
    torch.manual_seed(seed)
    return randomize_bias(rc.FeatureEncoder(), seed + 100)


def a256(x):
    return (x + 255) // 256 * 256


def _sizes(H, W):
    H1, W1 = (H + 1) // 2, (W + 1) // 2
    H2, W2 = (H1 + 1) // 2, (W1 + 1) // 2
    return H1, W1, H2, W2, (H2 + 1) // 2, (W2 + 1) // 2


def unit_grids(H, W):
    H1, W1, H2, W2, H3, W3 = _sizes(H, W)
    return [(H1, W1)] * 5 + [(H2, W2)] * 4 + [(H3, W3)] * 4


def ws_bytes(B, H, W):
    H1, W1, H2, W2, H3, W3 = _sizes(H, W)
    n = 11 * a256(B * H1 * W1 * 128) + 9 * a256(B * H2 * W2 * 256) + 9 * a256(B * H3 * W3 * 256)
    for (h, w), nt in zip(unit_grids(H, W), NT):
        n += a256(B * -(-w // 16) * -(-h // 8) * nt * 8)
    return n + sum(a256(B * 2 * nt * 4) for nt in NT)


# ------------------------------------------------------------------ CPU
def test_state_dict_matches_torchvision():
    ours, tv, tv2 = seeded(), randomize_bias(tv_fe(), 5), tv_fe()
    assert list(ours.state_dict().keys()) == list(tv.state_dict().keys())
    assert len(ours.state_dict()) == 32 and "layer3.0.downsample.0.bias" in ours.state_dict()
    ours.load_state_dict(tv.state_dict(), strict=True)
    tv2.load_state_dict(ours.state_dict(), strict=True)
    assert all(torch.equal(tv2.state_dict()[k], v) for k, v in tv.state_dict().items())


@pytest.mark.parametrize("kw", [dict(norm_layer=torch.nn.BatchNorm2d), dict(norm_layer=None),
                                dict(norm_layer=functools.partial(torch.nn.InstanceNorm2d, affine=True)),
                                dict(norm_layer=functools.partial(torch.nn.InstanceNorm2d, track_running_stats=True)),
                                dict(layers=(32, 32, 64, 96, 160)), dict(strides=(1, 1, 2, 2)),
                                dict(layers=(64, 64, 96, 128, 128)), "bottleneck"])
def test_unsupported_configurations_raise(kw):
    if kw == "bottleneck":
        from torchvision.models.optical_flow.raft import BottleneckBlock
        kw = dict(block=BottleneckBlock, layers=(32, 32, 64, 96, 160), norm_layer=torch.nn.InstanceNorm2d)
    with pytest.raises(ValueError, match="raft_large's feature encoder"):
        rc.FeatureEncoder(**kw)


@pytest.mark.parametrize("op", [torch.float16, torch.bfloat16])
def test_identity_norm_packing_rounds_each_weight_once(lib, op):
    """The context encoder's packing with the identity norm is each conv weight rounded once and each bias as is."""
    fe = seeded(1)
    convs = [c for c, _ in _convs_and_norms(fe)]
    pk = PackedFeatureEncoder(convs, op, "cpu", None)
    w = pk.weight.view(op)
    b = pk.bias
    # unit 1 (layer1.0.convnormrelu1): [k-block 0][tap t][n][c]; it follows the stem's 4 x 64 x 64
    off = 4 * 64 * 64
    got = w[off:off + 9 * 64 * 64].view(9, 64, 64).permute(1, 2, 0).reshape(64, 64, 3, 3)
    assert torch.equal(got, convs[1].weight.detach().to(op))
    # unit 5 (layer2.0.convnormrelu1 + downsample): slab 9 is the downsample; 96 rows of 128 real
    off += 4 * 9 * 64 * 64
    u5 = w[off:off + 10 * 128 * 64].view(10, 128, 64)
    assert torch.equal(u5[:9, :96].permute(1, 2, 0).reshape(96, 64, 3, 3), convs[5].weight.detach().to(op))
    assert torch.equal(u5[9, :96], convs[6].weight.detach()[:, :, 0, 0].to(op))
    assert not u5[:, 96:].any()
    assert torch.equal(b[:64], convs[0].bias.detach()) and torch.equal(b[-256:], convs[15].bias.detach())
    bo = 64 * 5
    assert torch.equal(b[bo:bo + 96], convs[5].bias.detach()) and torch.equal(b[bo + 128:bo + 224], convs[6].bias.detach())


def test_cabi_argument_errors_and_workspace(lib):
    A = 1 << 20           # a 16-byte aligned fake device address: every call below fails its checks before any access
    B, H, W = 2, 37, 53
    strides = (ctypes.c_longlong * 4)(3 * H * W, H * W, W, 1)
    eps = (ctypes.c_double * 15)(*([1e-5] * 15))
    for shape in ((B, H, W), (1, 8, 9), (3, 1088, 1920), (1, 9, 8)):
        assert lib.rdvc_corr_feature_encoder_workspace_bytes(*shape, rc.RDVC_DT_F16) == ws_bytes(*shape), shape
    ws = lib.rdvc_corr_feature_encoder_workspace_bytes(B, H, W, rc.RDVC_DT_F16)
    assert lib.rdvc_corr_feature_encoder_workspace_bytes(B, H, W, rc.RDVC_DT_F32) == ws
    assert lib.rdvc_corr_feature_encoder_workspace_bytes(0, H, W, rc.RDVC_DT_F16) == 0
    assert lib.rdvc_corr_feature_encoder_workspace_bytes(B, H, W, 7) == 0
    for h, w in ((8, 8), (1, 1), (5, 3)):                          # one-element layer3 plane
        assert lib.rdvc_corr_feature_encoder_workspace_bytes(1, h, w, rc.RDVC_DT_F16) == 0
    OUT = 1 << 30

    def fe(**kw):
        a = dict(img=A, s=strides, idt=rc.RDVC_DT_F32, B=B, H=H, W=W, op=rc.RDVC_DT_F16, w=A, b=A, eps=eps,
                 form=_cabi.RDVC_FE_OUT_FEATURES, ws=1 << 28, wsb=ws, out=OUT, ps=256, odt=rc.RDVC_DT_F32)
        a.update(kw)
        return lib.rdvc_corr_feature_encoder(a["img"], a["s"], a["idt"], a["B"], a["H"], a["W"], a["op"], a["w"], a["b"],
                                             a["eps"], a["form"], a["ws"], a["wsb"], a["out"], a["ps"], a["odt"], None)
    assert fe(img=None) == -1 and fe(s=None) == -1 and fe(w=None) == -1 and fe(b=None) == -1 and fe(eps=None) == -1
    assert fe(ws=None) == -1 and fe(out=None) == -1
    assert fe(form=2) == -5 and fe(form=-1) == -5
    assert fe(B=0) == -2 and fe(H=-1) == -2 and fe(W=0) == -2
    assert fe(H=8, W=8) == -2 and fe(H=1, W=1) == -2                 # InstanceNorm over a one-element plane
    assert "spatial element" in _cabi.last_error()
    assert fe(idt=9) == -4 and fe(op=rc.RDVC_DT_F32) == -4 and fe(odt=rc.RDVC_DT_BF16) == -4
    assert fe(form=_cabi.RDVC_FE_OUT_TRUNK, ps=128) == -4            # the trunk is op_dtype
    for bad in (-1.0, float("nan"), float("inf")):
        e = (ctypes.c_double * 15)(*([1e-5] * 14 + [bad]))
        assert fe(eps=e) == -5
    assert fe(s=(ctypes.c_longlong * 4)(-1, 1, 1, 1)) == -5
    assert fe(H=1 << 24) == -5
    assert fe(img=A + 2) == -7 and fe(w=A + 8) == -7 and fe(b=A + 4) == -7 and fe(out=OUT + 8) == -7
    assert fe(ps=128) == -5 and fe(ps=258) == -7
    assert fe(form=_cabi.RDVC_FE_OUT_TRUNK, odt=rc.RDVC_DT_F16, ps=64) == -5
    assert fe(wsb=ws - 1) == -6 and fe(ws=(1 << 28) + 16) == -7
    assert fe(out=A) == -5                                       # overlaps the image
    assert fe(out=(1 << 28) + 4096) == -5                        # inside the workspace


def test_module_refusals_on_cpu():
    fe = seeded(3)
    x = torch.rand(1, 3, 16, 16)
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            fe(x)
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            fe.forward_trunk(x)
        with pytest.raises(ValueError, match="more than 1 spatial element"):
            fe(torch.rand(1, 3, 8, 8))
    with pytest.raises(RuntimeError, match="forward-only"):
        fe(x.clone().requires_grad_())


def test_sass_of_the_statistics_entry(lib):
    """tap_conv_in_kernel holds exactly the feature encoder's 8 instantiations, each with tcgen05.mma (UTCHMMA), TMA
    loads (UTMALDG) and TMEM reads (LDTM)."""
    out = subprocess.run(["cuobjdump", "-sass", rc._cabi.lib_path()], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    funcs = [f for f in out.stdout.split("Function : ") if f.startswith("_ZN4rdvc18tap_conv_in_kernel")]
    for f in funcs:
        assert "UTCHMMA" in f and "UTMALDG" in f and "LDTM" in f, f.splitlines()[0]
    names = subprocess.run(["cu++filt"], input="\n".join(f.split(None, 1)[0] for f in funcs), capture_output=True,
                           text=True, check=True).stdout.split("\n")[:len(funcs)]
    got = sorted(tuple(re.search(r"tap_conv_in_kernel<([^>]*)>", n).group(1).replace("(int)", "").split(", "))
                 for n in names)
    assert got == sorted((str(g), str(n), str(e), op) for g, n, e in IN_INSTANCES for op in OPS)
    assert len([f for f in out.stdout.split("Function : ") if f.startswith("_ZN4rdvc18in_finalize_kernel")]) == 1
    assert len([f for f in out.stdout.split("Function : ") if f.startswith("_ZN4rdvc15in_apply_kernel")]) == 6


def test_no_register_spills():
    """-Xptxas -v over tap_conv_in_kernel's instantiations, the finalize and the apply kernels: no spills."""
    from rdvc_corr_b200 import _build
    inst = [f"template __global__ void tap_conv_in_kernel<{g}, {n}, {e}, {op}>"
            f"(const __grid_constant__ TapMaps<TapGeom<{g}>::MAPS>, const TapParams);" for g, n, e in IN_INSTANCES
            for op in OPS]
    inst += [f"template __global__ void in_apply_kernel<{f}, {op}>(const InApplyParams);" for f in range(3) for op in OPS]
    src = '#include "instance_norm_sm100.cuh"\nnamespace rdvc {\n' + "\n".join(inst) + "\n}\n"
    with tempfile.TemporaryDirectory() as d:
        cu = os.path.join(d, "spills.cu")
        with open(cu, "w") as f:
            f.write(src)
        res = subprocess.run([_build.nvcc_path(), "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                              "-Xptxas", "-v", "-I", os.path.join(PKG, "csrc"), "-c", cu, "-o", os.path.join(d, "s.o")],
                             capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-3000:]
    props = [ln for ln in res.stderr.splitlines() if "spill stores" in ln]
    assert len(props) == len(inst) + 1, res.stderr[-3000:]                  # + in_finalize_kernel
    assert all("0 bytes spill stores, 0 bytes spill loads" in ln for ln in props), props


# ------------------------------------------------------------------ GPU
def _op(dt):
    return torch.float16 if dt == torch.float32 else dt


def _image(B, H, W, dt, seed, channels_last=False):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = (0.85 + 0.1 * (2 * torch.rand(B, 3, H, W, device="cuda", generator=g) - 1)).to(dt)
    return x.contiguous(memory_format=torch.channels_last) if channels_last else x


def run_abi(lib, fe, x, form, out_dt, op, ws=None):
    """The module's call through the C ABI with a caller-owned workspace; returns (out NHWC, the workspace's stages as a
    dict of (B, C, h, w) views / (B, NT) mean and rstd, workspace)."""
    B, _, H, W = x.shape
    pk = PackedFeatureEncoder(fe._convs(), op, x.device, None)
    wsb = lib.rdvc_corr_feature_encoder_workspace_bytes(B, H, W, ADT[out_dt])
    if ws is None:
        ws = torch.zeros(wsb, dtype=torch.uint8, device="cuda")
    H1, W1, H2, W2, H3, W3 = _sizes(H, W)
    trunk = form == _cabi.RDVC_FE_OUT_TRUNK
    out = torch.empty(B, H3, W3, 128 if trunk else 256, dtype=op if trunk else out_dt, device="cuda")
    strides = (ctypes.c_longlong * 4)(*x.stride())
    eps = (ctypes.c_double * 15)(*fe._eps())
    _cabi.check(lib.rdvc_corr_feature_encoder(x.data_ptr(), strides, ADT[x.dtype], B, H, W, ADT[op], pk.weight.data_ptr(),
                                              pk.bias.data_ptr(), eps, form, ws.data_ptr(), wsb, out.data_ptr(),
                                              out.shape[-1], ADT[out.dtype], torch.cuda.current_stream().cuda_stream),
                "feature_encoder")
    names = (["S"] + [f"{k}{i}" for i in range(5) for k in "YA"] + ["Y5", "D5", "A5", "Y6", "A6", "Y7", "A7", "Y8", "A8"]
             + ["Y9", "D9", "A9", "Y10", "A10", "Y11", "A11", "Y12", "A12"])
    st, off = {}, 0
    for n, (h, w, c) in zip(names, [(H1, W1, 64)] * 11 + [(H2, W2, 128)] * 9 + [(H3, W3, 128)] * 9):
        size = B * h * w * c * 2
        st[n] = ws[off:off + size].view(op).view(B, h, w, c).permute(0, 3, 1, 2)
        off += a256(size)
    for i, ((h, w), nt) in enumerate(zip(unit_grids(H, W), NT)):
        off += a256(B * -(-w // 16) * -(-h // 8) * nt * 8)
    for i, nt in enumerate(NT):
        s = ws[off:off + B * 2 * nt * 4].view(torch.float32).view(B, 2, nt)
        st[f"mean{i}"], st[f"rstd{i}"] = s[:, 0], s[:, 1]
        off += a256(B * 2 * nt * 4)
    assert off == wsb
    return out, st, ws


class Chain:
    """fp64 evaluation with the kernels' rounding points."""

    def __init__(self, fe, op):
        self.op = op
        self.w = [c.weight.detach().to(op).double().cuda() for c in fe._convs()]
        self.b15 = fe.conv.bias.detach().double().cuda()
        self.eps = fe._eps()

    def r(self, t):
        return t.to(self.op).double()

    def conv(self, i, x, stride, pad):                     # normalised layers: no bias
        return F.conv2d(x, self.w[i], None, stride=stride, padding=pad)

    def norm(self, i, y):
        var, mean = torch.var_mean(y, dim=(2, 3), unbiased=False, keepdim=True)
        return (y - mean) / torch.sqrt(var + self.eps[i])

    def block(self, x, i1, i2, ids=None):
        stride = 1 if ids is None else 2
        t = self.r(self.norm(i1, self.r(self.conv(i1, x, stride, 1))).clamp_min(0))
        res = x if ids is None else self.norm(ids, self.r(self.conv(ids, x, 2, 0)))
        return self.r((res + self.norm(i2, self.r(self.conv(i2, t, 1, 1))).clamp_min(0)).clamp_min(0))

    def trunk(self, img):
        x = self.r(img)
        x = self.r(self.norm(0, self.r(self.conv(0, x, 2, 3))).clamp_min(0))
        x = self.block(self.block(x, 1, 2), 3, 4)
        x = self.block(self.block(x, 5, 7, 6), 8, 9)
        return self.block(self.block(x, 10, 12, 11), 13, 14)

    def __call__(self, img):
        return F.conv2d(self.trunk(img), self.w[15], self.b15)


def _raw_ok(got, ref, op):
    tol = 2 * U[op] * ref.abs() + 2e-4 * max(1.0, ref.abs().max().item())
    err = (got.double() - ref).abs()
    return bool((err <= tol).all()), err.max().item()


def _in(y, mean, rstd):
    return (y.double() - mean.double()[:, :, None, None]) * rstd.double()[:, :, None, None]


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("shape", SMALL)
def test_stages_vs_fp64_on_kernel_inputs(lib, shape, dt):
    """Raw convolutions (STATS: stem, 3x3 64 and 128; DS_STATS: layer2 and layer3), mean / rstd over the stored raw
    values, the three apply forms, the padded channels and the final 1x1, each on the kernel's own inputs."""
    B, H, W = shape
    op = _op(dt)
    fe = seeded(10).cuda()
    ch = Chain(fe, op)
    u = U[op]
    x = _image(B, H, W, dt, B * H * W)
    with torch.no_grad():
        out, P, _ = run_abi(lib, fe, x, _cabi.RDVC_FE_OUT_FEATURES, dt, op)
        trunk, P2, _ = run_abi(lib, fe, x, _cabi.RDVC_FE_OUT_TRUNK, dt, op)
        torch.cuda.synchronize()
        d = lambda k: P[k].double()                                        # noqa: E731
        # raw convolutions (no bias), each rounded once
        stem_in = F.conv2d(ch.r(x), ch.w[0], None, stride=2, padding=3)
        raws = [("Y0", stem_in), ("Y1", ch.conv(1, d("A0"), 1, 1)), ("Y4", ch.conv(4, d("A3"), 1, 1)),
                ("Y5", ch.conv(5, d("A4"), 2, 1)), ("D5", ch.conv(6, d("A4"), 2, 0)),
                ("Y7", ch.conv(8, d("A6")[:, :96], 1, 1)), ("Y9", ch.conv(10, d("A8")[:, :96], 2, 1)),
                ("D9", ch.conv(11, d("A8")[:, :96], 2, 0)), ("Y12", ch.conv(14, d("A11"), 1, 1))]
        for name, ref in raws:
            ok, err = _raw_ok(P[name][:, :ref.shape[1]], ref, op)
            assert ok, (name, err)
        # mean / rstd of every normalised unit over its stored raw values
        ys = [("Y0",), ("Y1",), ("Y2",), ("Y3",), ("Y4",), ("Y5", "D5"), ("Y6",), ("Y7",), ("Y8",), ("Y9", "D9"),
              ("Y10",), ("Y11",), ("Y12",)]
        conv_of = [0, 1, 2, 3, 4, (5, 6), 7, 8, 9, (10, 11), 12, 13, 14]
        for i, parts in enumerate(ys):
            y = torch.cat([d(k) for k in parts], 1)
            cs = [c for c in range(y.shape[1]) if c % 128 < (64 if i < 5 else 96 if i < 9 else 128)]
            y = y[:, cs]
            var, mean = torch.var_mean(y, dim=(2, 3), unbiased=False)
            li = conv_of[i] if isinstance(conv_of[i], tuple) else (conv_of[i],)
            eps = torch.tensor([fe._eps()[li[0] if c < 128 or len(li) == 1 else li[1]] for c in cs], dtype=torch.float64,
                               device="cuda")
            m, r = P[f"mean{i}"][:, cs].double(), P[f"rstd{i}"][:, cs].double()
            assert ((m - mean).abs() <= 1e-5 * (mean.abs() + var.sqrt())).all(), (i, (m - mean).abs().max().item())
            rref = 1 / torch.sqrt(var + eps)
            assert ((r - rref).abs() <= 1e-5 * rref).all(), (i, ((r - rref).abs() / rref).max().item())

        def apply_ok(name, got, a, b=None):
            ref = a.clamp_min(0) if b is None else (b + a.clamp_min(0)).clamp_min(0)
            scale = a.abs() + (0 if b is None else b.abs())
            tol = u * ref.abs() + 1e-6 * scale + 2.0 ** -24
            assert ((got.double() - ref).abs() <= tol).all(), (name, (got.double() - ref).abs().max().item())

        n = lambda i, k, lo=0, hi=None: _in(d(k)[:, lo:hi], P[f"mean{i}"][:, lo:hi], P[f"rstd{i}"][:, lo:hi])  # noqa: E731
        apply_ok("relu stem", P["A0"], n(0, "Y0"))
        apply_ok("relu l1", P["A1"], n(1, "Y1"))
        apply_ok("res l1", P["A2"], n(2, "Y2"), d("A0"))
        apply_ok("relu s2", P["A5"][:, :96], n(5, "Y5", 0, 96))
        ds5 = _in(d("D5")[:, :96], P["mean5"][:, 128:224], P["rstd5"][:, 128:224])
        apply_ok("ds l2", P["A6"][:, :96], n(6, "Y6", 0, 96), ds5)
        apply_ok("res l2", P["A8"][:, :96], n(8, "Y8", 0, 96), d("A6")[:, :96])
        ds9 = _in(d("D9"), P["mean9"][:, 128:], P["rstd9"][:, 128:])
        apply_ok("ds l3", P["A10"], n(10, "Y10"), ds9)
        apply_ok("res l3", P["A12"], n(12, "Y12"), d("A10"))
        for k in ("Y5", "D5", "A5", "Y6", "A6", "Y7", "A7", "Y8", "A8"):
            assert not P[k][:, 96:].any(), k                               # exact zeros, not 0 * rsqrt(eps)
        fin = F.conv2d(d("A12"), ch.w[15], ch.b15)
        ok, err = _raw_ok(out.permute(0, 3, 1, 2), fin if dt == torch.float32 else ch.r(fin), op)
        assert ok, ("1x1", err)
        assert torch.equal(trunk.permute(0, 3, 1, 2), P["A12"])            # the trunk is layer3's output
        assert all(torch.equal(P[k], P2[k]) for k in P if k != "A12")      # the forms differ only at the end


@pytest.mark.gpu
def test_normalised_biases_are_dropped(lib):
    """A normalised layer's conv bias cancels in InstanceNorm and is not used: changing it leaves the output bit-
    identical.  The final 1x1's bias is used."""
    fe = seeded(20).cuda()
    x = _image(2, 70, 98, torch.float32, 1)
    with torch.no_grad():
        a = fe(x).clone()
        for c in fe._convs()[:-1]:
            c.bias.add_(torch.randn_like(c.bias))
        assert torch.equal(fe(x), a)
        fe.conv.bias.add_(1.0)
        assert not torch.equal(fe(x), a)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("shape", SMALL + [(10, 1088, 1920)])
def test_module_vs_fp64_chain_and_stock(lib, shape, dt):
    B, H, W = shape
    op = _op(dt)
    fe = seeded(11).cuda()
    x = _image(B, H, W, dt, 7 + B * H * W)
    amp = dt != torch.float32
    xin = x.float() if amp else x
    with torch.no_grad(), torch.autocast("cuda", dtype=op, enabled=amp):
        out = fe(xin)                                                      # autocast: fp32 image, 16-bit everything
        trunk = fe.forward_trunk(xin)
    h, w = (H + 7) // 8, (W + 7) // 8
    assert out.shape == (B, 256, h, w) and out.dtype == dt and out.is_contiguous(memory_format=torch.channels_last)
    assert trunk.shape == (B, 128, h, w) and trunk.dtype == op and trunk.stride(1) == 1
    n = B if B < 10 else 1                                                 # the fp64 chain on sample 0 at 1080p
    ch = Chain(fe, op)
    with torch.no_grad():
        tref = ch.trunk(xin[:n])
        ref = ch(xin[:n])
    assert (trunk[:n].double() - tref).abs().max().item() <= 16 * U[op] * tref.abs().max().item()
    assert (out[:n].double() - ref).abs().max().item() <= 16 * U[op] * ref.abs().max().item()
    if dt == torch.bfloat16 and h * w == 2:
        # layer3's planes have 2 elements: InstanceNorm maps each channel to +-1 by the sign of their difference, which
        # bf16 rounding of stock's y + bias (our y is stored without the bias) can flip -- an O(1) difference that is
        # not an error of either; the fp64 chain above holds.
        return
    tv = tv_fe().cuda().eval()
    tv.load_state_dict(fe.state_dict())
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad(), torch.autocast("cuda", dtype=op, enabled=amp):
            s = tv(xin)
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    assert (out.float() - s.float()).abs().max().item() <= TOL_STOCK[dt] * max(1.0, s.abs().max().item())


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPES)
def test_nan_workspace_determinism_streams_graphs_batches(lib, dt):
    """A NaN-filled workspace gives the bits of a zeroed one; repeated runs, a side stream, a CUDA graph replay, NCHW vs
    channels_last input, train mode, and a frame alone vs at every position of a batch of 3 are bit-identical."""
    B, H, W = 3, 70, 98
    op = _op(dt)
    fe = seeded(12).cuda()
    x = _image(B, H, W, dt, 3)
    with torch.no_grad():
        a, _, ws = run_abi(lib, fe, x, _cabi.RDVC_FE_OUT_TRUNK, dt, op)
        ws.fill_(255)                                                      # 0xFFFF: NaN in fp16 and bf16, fp32 too
        b, _, _ = run_abi(lib, fe, x, _cabi.RDVC_FE_OUT_TRUNK, dt, op, ws=ws)
        assert torch.equal(a, b)
        t0 = fe.forward_trunk(x)
        assert torch.equal(t0, a.permute(0, 3, 1, 2))
        assert torch.equal(fe.forward_trunk(x.contiguous(memory_format=torch.channels_last)), t0)
        assert torch.equal(fe(x), fe(x))
        fe.train()
        assert torch.equal(fe.forward_trunk(x), t0)
        fe.eval()
        for i in range(B):                                                 # batch invariance
            alone = fe.forward_trunk(x[i:i + 1].clone())
            assert torch.equal(alone, t0[i:i + 1])
            others = [j for j in range(B) if j != i]
            for pos in range(3):
                order = others[:pos] + [i] + others[pos:]
                batch = fe.forward_trunk(torch.cat([_image(1, H, W, dt, 50 + j) if j != i else x[i:i + 1]
                                                    for j in order]))
                assert torch.equal(batch[pos:pos + 1], alone), (i, pos)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            s = fe(x)
        torch.cuda.current_stream().wait_stream(side)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            gout = fe(x)
        gr.replay()
        torch.cuda.synchronize()
        r = fe(x)
        assert torch.equal(s, r) and torch.equal(gout, r)


# ------------------------------------------------------------------ RAFT end to end
def _seeded_raft(swap, corr_block=True):
    from torchvision.models.optical_flow import raft_large
    torch.manual_seed(0)
    model = raft_large(weights=None, **({"corr_block": rc.TVCorrBlock()} if corr_block else {}))
    randomize_bias(model.feature_encoder, 55)
    g = torch.Generator().manual_seed(77)
    with torch.no_grad():
        for m in model.context_encoder.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                c = m.num_features
                m.running_mean.copy_(0.5 * torch.randn(c, generator=g))
                m.running_var.copy_(0.5 + 1.5 * torch.rand(c, generator=g))
                m.weight.copy_(0.5 + torch.rand(c, generator=g))
                m.bias.copy_(0.3 * torch.randn(c, generator=g))
    model = model.eval().cuda()
    if swap is None:
        return model
    fe = rc.FeatureEncoder()
    fe.load_state_dict(model.feature_encoder.state_dict())
    model.feature_encoder = fe.cuda()
    if swap == "all":
        ub = model.update_block
        ce = rc.ContextEncoder()
        me, fh = rc.MotionEncoder(in_channels_corr=324), rc.FlowHead(in_channels=128, hidden_size=256)
        rb = rc.RecurrentBlock(input_size=256, hidden_size=128)
        mp = rc.MaskPredictor(in_channels=128, hidden_size=256, multiplier=model.mask_predictor.multiplier)
        ce.load_state_dict(model.context_encoder.state_dict())
        me.load_state_dict(ub.motion_encoder.state_dict())
        fh.load_state_dict(ub.flow_head.state_dict())
        rb.load_state_dict(ub.recurrent_block.state_dict())
        mp.load_state_dict(model.mask_predictor.state_dict())
        model.context_encoder = ce.cuda().eval()
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
@pytest.mark.parametrize("swap", ["fe", "all"])
@pytest.mark.parametrize("case", ["368x640", "1080p"])
def test_raft_epe_vs_stock(lib, golden_dir, case, swap, amp):
    a, b = _frames(golden_dir, (368, 640)) if case == "368x640" else _synthetic_1080p()
    model = _seeded_raft(swap)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=amp):
        ref = _seeded_raft(None, corr_block=False)(a, b, num_flow_updates=12)[-1]
        got = rc.raft_flow(model, a, b, 12)
        unfused = rc.raft_flow(model, a, b, 12, fuse_convcorr1=False, fuse_encoder_tail=False)
        stock_call = model(a, b, num_flow_updates=12)[-1]             # RAFT.forward with the drop-ins swapped in
    assert isinstance(model.feature_encoder, rc.FeatureEncoder)
    assert got.dtype == torch.float32 and got.shape == ref.shape
    for f in (got, unfused, stock_call):
        assert torch.isfinite(f).all()
        assert _epe(f, ref) < TOL_EPE, _epe(f, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("swap", ["fe", "all"])
def test_raft_sequence_bit_identical_and_graphs(lib, golden_dir, swap):
    """With per-sample statistics from per-tile partials a frame's features do not depend on its batch:
    raft_flow_sequence equals the pair-wise call bit for bit, and the graphs replay eager bit for bit."""
    a, b = _frames(golden_dir, (368, 640))
    frames = torch.cat([a, b, torch.roll(a, (3, -5), (2, 3))], 0)
    model = _seeded_raft(swap)
    for amp in (None, torch.float16):
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=amp is not None):
            pairs = rc.raft_flow(model, frames[:-1], frames[1:], 12)
            seq = rc.raft_flow_sequence(model, frames, 12)
            eager = rc.raft_flow(model, a, b, 12)
        assert torch.equal(seq, pairs)
        runner = rc.GraphedRaftFlow(model, 12, amp_dtype=amp)
        assert torch.equal(runner(a, b), eager) and torch.equal(runner(a, b), eager)
        assert torch.equal(runner.sequence(frames), seq)
        runner.release()
