"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI, against the oracles.

Tolerances (BASELINE.json north_star, SURVEY.md 8c), all max-norm relative = max|a-b| / max|ref|:
  * correlation volume / pyramid vs the fp32 reference ......... 2e-2  (bf16 operands, fp32 accumulate)
  * same, vs an fp64 evaluation of the SAME rounded operands .... 1e-4  (fp32 out) / 8e-3 (bf16 out)
    (pooled levels at full size: 5e-4 -- the pooled fmap2 means are rounded to bf16 once, and a mean
     within fp32 summation-order distance of a bf16 rounding boundary may round the other way than the
     test's own avg_pool2d: ~2^-15 of the operand elements differ by one bf16 ulp)
  * lookup vs the oracle's lookup of the SAME pyramid ........... 1e-3  (observed ~1e-6)
  * RAFT flow end-point error vs stock torchvision, 12 updates .. 0.05 px mean
"""
import ctypes
import os

import numpy as np
import pytest
import torch

import rdvc_corr_b200 as rc
from helpers import bf16_round, fp16_round, pyramid_from_levels, ref_pyramid_linear, rel_max
from oracle import corr_c as cc
from oracle import corr_numpy as cn
from oracle import tv_corr as tv

pytestmark = pytest.mark.gpu

TOL_VOLUME = 2e-2
TOL_SAME_OPERANDS_F32 = 1e-4
TOL_SAME_OPERANDS_BF16 = 8e-3
TOL_SAME_OPERANDS_POOLED = 5e-4
TOL_LOOKUP = 1e-3
TOL_EPE = 0.05
SIGMAS = (0.0, 0.3, 4.0, 40.0)
MODES = {"fused": 1, "linear": 2}
ROW, TILED = rc.RDVC_LAYOUT_ROWMAJOR, rc.RDVC_LAYOUT_TILED
LAYOUTS = {"rowmajor": ROW, "tiled": TILED}
# lookup code paths: (pyramid layout, lookup variant option)
LOOKUP_PATHS = {"row_scalar": (ROW, 1), "row_vec": (ROW, 2), "tiled": (TILED, 0)}


@pytest.fixture(scope="module")
def lib():
    assert torch.cuda.is_available(), "GPU tests need a B200"
    L = rc._cabi.load()
    yield L
    for k in list(range(10)) + [12]:
        L.rdvc_corr_set_option(k, {3: 15, 5: 1}.get(k, 0))


def set_opts(lib, **kw):
    keys = {"lookup": 0, "tile": 1, "msplit": 2, "mode": 4, "tma": 5, "epi": 9, "pair": 12}
    for k, v in kw.items():
        assert lib.rdvc_corr_set_option(keys[k], v) == 0


def gpu(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def need_experiments(mode=None):
    """The fused-pooling build mode, the CTA-pair build kernel and the work-skipping knobs are compiled into
    lib/librdvc_corr_exp.so only (-DRDVC_EXPERIMENTS; `RDVC_CORR_LIB=.../librdvc_corr_exp.so pytest -m gpu`)."""
    if mode in (None, "fused") and not rc._cabi.has_experiments():
        pytest.skip("needs the RDVC_EXPERIMENTS build of the library (not the product build)")


# ------------------------------------------------------------------ lookup
@pytest.mark.parametrize("path", list(LOOKUP_PATHS))
@pytest.mark.parametrize("shape", [(2, 8, 18, 22), (1, 8, 46, 80), (1, 4, 16, 16), (1, 4, 17, 19)])
def test_lookup_matches_oracle(lib, shape, path):
    B, C, h, w = shape
    layout, variant = LOOKUP_PATHS[path]
    f1, f2 = cn.synth_fmaps(B, C, h, w, seed=3)
    flat = cc.build_pyramid(f1, f2, 4)
    pyr = pyramid_from_levels(rc, cc.split_levels(flat, B, h, w, 4), B, h, w, layout=layout)
    set_opts(lib, lookup=variant)
    for sigma in SIGMAS:
        co = cn.synth_coords(B, h, w, sigma, seed=1)
        got = rc.index_pyramid(pyr, gpu(co), 4).cpu().numpy()
        assert got.shape == (B, 324, h, w)
        assert rel_max(got, cc.index_pyramid(flat, co, 4, 4)) < TOL_LOOKUP
    set_opts(lib, lookup=0)


@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_lookup_golden_small_odd(lib, golden_dir, layout):
    """Pyramid and lookups from torchvision's CorrBlock, pinned to the fixture (every `stride`-th element)."""
    g = np.load(os.path.join(golden_dir, "corr_small_odd.npz"))
    B, C, h, w = [int(x) for x in g["shape"]]
    st = int(g["stride"])
    f1, f2 = cn.synth_fmaps(B, C, h, w, seed=int(g["seed"]))
    levels = tv.build_pyramid(torch.from_numpy(f1), torch.from_numpy(f2), 4)
    for l in range(4):
        assert rel_max(levels[l][:, 0].numpy().reshape(-1)[::st], g[f"level{l}"]) < 2e-6
    pyr = pyramid_from_levels(rc, [lv[:, 0].numpy() for lv in levels], B, h, w, layout=LAYOUTS[layout])
    for s in SIGMAS:
        co = cn.synth_coords(B, h, w, s, seed=1)
        got = rc.index_pyramid(pyr, gpu(co), 4).cpu().numpy()
        assert rel_max(got.reshape(-1)[::st], g[f"lookup_sigma{s:g}"]) < TOL_LOOKUP
        assert rel_max(got, tv.index_pyramid(levels, torch.from_numpy(co), 4).numpy()) < TOL_LOOKUP


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("vol", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("radius,levels", [(3, 3), (1, 1), (2, 4)])
def test_lookup_other_radius_and_levels(lib, radius, levels, vol, layout):
    B, C, h, w = 2, 8, 18, 22
    f1, f2 = cn.synth_fmaps(B, C, h, w, seed=4)
    flat = cc.build_pyramid(f1, f2, levels)
    if vol == torch.bfloat16:
        flat = bf16_round(flat)
    pyr = pyramid_from_levels(rc, cc.split_levels(flat, B, h, w, levels), B, h, w, vol, layout=LAYOUTS[layout])
    co = cn.synth_coords(B, h, w, 2.5, seed=2)
    got = rc.index_pyramid(pyr, gpu(co), radius).cpu().numpy()
    assert got.shape == (B, levels * (2 * radius + 1) ** 2, h, w)
    assert rel_max(got, cc.index_pyramid(flat, co, levels, radius)) < TOL_LOOKUP


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("shape", [(1, 8, 24, 40), (2, 8, 18, 22), (1, 4, 17, 19)])
def test_lookup_bf16_volume(lib, shape, layout):
    B, C, h, w = shape
    f1, f2 = cn.synth_fmaps(B, C, h, w, seed=6)
    flat = bf16_round(cc.build_pyramid(f1, f2, 4))   # what a bf16 pyramid stores
    pyr = pyramid_from_levels(rc, cc.split_levels(flat, B, h, w, 4), B, h, w, torch.bfloat16,
                              layout=LAYOUTS[layout])
    for sigma in SIGMAS:
        co = cn.synth_coords(B, h, w, sigma, seed=3)
        got = rc.index_pyramid(pyr, gpu(co), 4).cpu().numpy()
        assert rel_max(got, cc.index_pyramid(flat, co, 4, 4)) < TOL_LOOKUP


def test_layouts_give_identical_lookups(lib):
    """The layout is storage only: the same pyramid values in either layout -> bit-identical features."""
    B, C, h, w = 2, 8, 18, 22
    f1, f2 = cn.synth_fmaps(B, C, h, w, seed=14)
    levels = cc.split_levels(cc.build_pyramid(f1, f2, 4), B, h, w, 4)
    co = gpu(cn.synth_coords(B, h, w, 6.0, seed=2))
    for vol in (torch.float32, torch.bfloat16):
        a = rc.index_pyramid(pyramid_from_levels(rc, levels, B, h, w, vol, layout=ROW), co, 4)
        b = rc.index_pyramid(pyramid_from_levels(rc, levels, B, h, w, vol, layout=TILED), co, 4)
        assert torch.equal(a, b)
    # and the tiled storage round-trips through level()/set_level()
    pyr = pyramid_from_levels(rc, levels, B, h, w, layout=TILED)
    for l in range(4):
        assert np.array_equal(pyr.level(l)[:, 0].cpu().numpy(), levels[l])


def test_lookup_integer_coords_are_exact_gathers(lib):
    B, C, h, w = 1, 8, 16, 24
    f1, f2 = cn.synth_fmaps(B, C, h, w, seed=9)
    lv = cc.split_levels(cc.build_pyramid(f1, f2, 1), B, h, w, 1)
    pyr = pyramid_from_levels(rc, lv, B, h, w)
    assert pyr.layout == TILED
    got = rc.index_pyramid(pyr, gpu(cn.make_coords_grid(B, h, w)), 4).cpu().numpy()
    q = 7 * w + 9
    for (i, j) in [(4, 4), (6, 2), (0, 8), (8, 0)]:
        assert got[0, i * 9 + j, 7, 9] == lv[0][q, 7 + j - 4, 9 + i - 4]
    assert np.all(got[0, 0 * 9 + 4, :, 0:4] == 0)  # dx = -4 at the left border: zero padding


# ------------------------------------------------------------------ build
BUILD_SHAPES = [(1, 64, 16, 16), (2, 64, 18, 22), (1, 128, 33, 47), (1, 256, 46, 80), (3, 64, 24, 40),
                (1, 192, 20, 28)]


@pytest.mark.parametrize("mode", ["fused", "linear"])
@pytest.mark.parametrize("shape", BUILD_SHAPES)
def test_build_fp32_volume(lib, shape, mode):
    need_experiments(mode)
    B, D, h, w = shape
    f1, f2 = cn.synth_fmaps(B, D, h, w, seed=5)
    ref32 = cn.build_pyramid(f1, f2, 4)                       # fp64 math on the un-rounded inputs
    same = (cn.build_pyramid(bf16_round(f1), bf16_round(f2), 4) if mode == "fused"
            else ref_pyramid_linear(f1, f2, 4))               # fp64 math on what the kernel multiplies
    # fused mode: both tile shapes, row-major only; linear mode: both layouts
    for tile, layout in (((1, ROW), (2, ROW)) if mode == "fused" else ((0, ROW), (0, TILED))):
        set_opts(lib, mode=MODES[mode], tile=tile)
        pyr = rc.build_pyramid(gpu(f1), gpu(f2), 4, layout=layout)
        for l in range(4):
            got = pyr.level(l)[:, 0].cpu().numpy()
            assert got.shape == ref32[l].shape
            assert rel_max(got, same[l]) < TOL_SAME_OPERANDS_F32, (mode, tile, layout, l)
            assert rel_max(got, ref32[l]) < TOL_VOLUME, (mode, tile, layout, l)
        if layout == TILED:  # padding pixels of the tiled storage are exact zeros
            for l in range(4):
                hl, wl, tw, th, hp, wp = pyr._tiles(l)
                raw = pyr.storage(l)
                st = raw[:, : hp * wp].reshape(-1, hp // th, wp // tw, th, tw).permute(0, 1, 3, 2, 4).reshape(-1, hp, wp)
                assert not st[:, hl:, :].any() and not st[:, :, wl:].any() and not raw[:, hp * wp:].any()
    set_opts(lib, mode=0, tile=0)


@pytest.mark.parametrize("mode", ["fused", "linear"])
def test_build_bf16_volume(lib, mode):
    need_experiments(mode)
    B, D, h, w = 1, 128, 46, 80
    f1, f2 = cn.synth_fmaps(B, D, h, w, seed=5)
    ref32 = cn.build_pyramid(f1, f2, 4)
    set_opts(lib, mode=MODES[mode])
    for layout in ((ROW,) if mode == "fused" else (ROW, TILED)):
        pyr = rc.build_pyramid(gpu(f1), gpu(f2), 4, torch.bfloat16, layout=layout)
        for l in range(4):
            got = pyr.level(l)[:, 0].float().cpu().numpy()
            assert rel_max(got, ref32[l]) < TOL_VOLUME
    set_opts(lib, mode=0)


@pytest.mark.parametrize("epi", [4, 8])
@pytest.mark.parametrize("vol", [torch.float32, torch.bfloat16])
def test_build_epilogue_shapes(lib, epi, vol):
    """Both epilogue shapes of the linear build (4 warps x 3 staging buffers, 8 warps x 1) for both
    storage types, on a shape with partial m-blocks, partial n-tiles and B > 1."""
    B, D, h, w = 2, 64, 18, 22
    f1, f2 = cn.synth_fmaps(B, D, h, w, seed=15)
    ref = ref_pyramid_linear(f1, f2, 4)
    tol = TOL_SAME_OPERANDS_F32 if vol == torch.float32 else TOL_SAME_OPERANDS_BF16
    set_opts(lib, epi=epi)
    for layout in (ROW, TILED):
        pyr = rc.build_pyramid(gpu(f1), gpu(f2), 4, vol, layout=layout)
        for l in range(4):
            assert rel_max(pyr.level(l)[:, 0].float().cpu().numpy(), ref[l]) < tol, (layout, l)
    set_opts(lib, epi=0)


@pytest.mark.parametrize("vol", [torch.float32, torch.bfloat16])
def test_build_cta_pair_kernel_is_bit_identical(lib, vol):
    """The opt-in CTA-pair build (tcgen05 cta_group::2, M = 256 over two SMs; option key 12 = 2) performs the
    same MMAs in the same K order as the single-CTA kernel: the pyramids must be bit-identical, including
    partial 256-row blocks (N = 396: the peer CTA's rows fall off the end), partial tiles and B > 1."""
    need_experiments()
    for (B, D, h, w) in [(2, 64, 18, 22), (1, 128, 33, 47), (1, 256, 46, 80)]:
        f1, f2 = cn.synth_fmaps(B, D, h, w, seed=17)
        set_opts(lib, pair=1)
        a = rc.build_pyramid(gpu(f1), gpu(f2), 4, vol).buffer.clone()
        set_opts(lib, pair=2)
        b = rc.build_pyramid(gpu(f1), gpu(f2), 4, vol).buffer.clone()
        assert torch.equal(a, b), (B, D, h, w)
    set_opts(lib, pair=0)


@pytest.mark.parametrize("vol", [torch.float32, torch.bfloat16])
def test_build_cluster_multicast_is_bit_identical(lib, vol):
    """fmap1 TMA-multicast across CTA pairs (option key 12 = 3): two CTAs holding neighbouring fmap2 tiles share one
    fmap1 stream.  Same MMAs, same K order: the pyramid must be bit-identical to the one-CTA-per-tile build, incl. an
    odd number of tiles (the last cluster's second CTA owns no tile), partial m-blocks, B > 1 and forced m-splits."""
    need_experiments()
    for (B, D, h, w) in [(1, 64, 16, 16), (2, 64, 18, 22), (1, 128, 33, 47), (1, 256, 46, 80), (3, 64, 24, 40)]:
        f1, f2 = cn.synth_fmaps(B, D, h, w, seed=19)
        for msplit in (0, 3):
            set_opts(lib, pair=1, msplit=msplit)
            a = rc.build_pyramid(gpu(f1), gpu(f2), 4, vol).buffer.clone()
            set_opts(lib, pair=3, msplit=msplit)
            b = rc.build_pyramid(gpu(f1), gpu(f2), 4, vol).buffer.clone()
            assert torch.equal(a, b), (B, D, h, w, msplit)
    set_opts(lib, pair=0, msplit=0)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_build_half_inputs(lib, dtype):
    """Under the reference's default AMP the fmaps arrive in half precision (SURVEY.md 0.7).  fp16 inputs are
    multiplied AS fp16 (tcgen05 kind::f16 takes either format): nothing of the input is lost, so the volume is
    within 1e-3 of the fp32 reference instead of the 4e-3 of bf16 operands."""
    B, D, h, w = 1, 64, 24, 40
    f1, f2 = cn.synth_fmaps(B, D, h, w, seed=8)
    ref32 = cn.build_pyramid(f1, f2, 4)
    pyr = rc.build_pyramid(gpu(f1).to(dtype), gpu(f2).to(dtype), 4)
    rnd = fp16_round if dtype == torch.float16 else bf16_round
    same = ref_pyramid_linear(rnd(f1), rnd(f2), 4, round_fn=rnd)     # what the kernel multiplies, in fp64
    for l in range(4):
        got = pyr.level(l)[:, 0].cpu().numpy()
        assert rel_max(got, ref32[l]) < (1e-3 if dtype == torch.float16 else TOL_VOLUME), l
        assert rel_max(got, same[l]) < (TOL_SAME_OPERANDS_F32 if l == 0 else TOL_SAME_OPERANDS_POOLED), l


@pytest.mark.parametrize("levels", [1, 2, 3])
def test_build_fewer_levels(lib, levels):
    B, D, h, w = 1, 64, 18, 22
    f1, f2 = cn.synth_fmaps(B, D, h, w, seed=2)
    ref = ref_pyramid_linear(f1, f2, levels)
    pyr = rc.build_pyramid(gpu(f1), gpu(f2), levels)
    assert len(pyr.levels()) == levels
    for l in range(levels):
        assert rel_max(pyr.level(l)[:, 0].cpu().numpy(), ref[l]) < TOL_SAME_OPERANDS_F32


@pytest.mark.parametrize("tma", [0, 2])
@pytest.mark.parametrize("vol", [torch.float32, torch.bfloat16])
def test_build_other_store_paths(lib, tma, vol):
    """Linear mode without the wide TMA boxes: staged st.global (tma=0, the path odd-sized row-major
    levels take) and 32-row x 128-byte boxes (tma=2, 16-byte-aligned row pitches)."""
    B, D, h, w = 1, 64, 24, 40
    f1, f2 = cn.synth_fmaps(B, D, h, w, seed=12)
    ref = ref_pyramid_linear(f1, f2, 4)
    tol = TOL_SAME_OPERANDS_F32 if vol == torch.float32 else TOL_SAME_OPERANDS_BF16
    set_opts(lib, mode=2, tma=tma)
    for layout in (ROW, TILED):
        pyr = rc.build_pyramid(gpu(f1), gpu(f2), 4, vol, layout=layout)
        for l in range(4):
            assert rel_max(pyr.level(l)[:, 0].float().cpu().numpy(), ref[l]) < tol
    set_opts(lib, mode=0, tma=1)


def test_build_golden_ref_default(lib, golden_dir):
    """D=256, 46x80: RDVC's default RAFT size; sampled entries from torchvision's fp32 CorrBlock."""
    g = np.load(os.path.join(golden_dir, "corr_ref_default.npz"))
    B, D, h, w = [int(x) for x in g["shape"]]
    f1, f2 = cn.synth_fmaps(B, D, h, w, seed=int(g["seed"]))
    blk = rc.TVCorrBlock()
    blk.build_pyramid(gpu(f1), gpu(f2))
    for l in range(4):
        got = blk.corr_pyramid[l].reshape(-1)[torch.from_numpy(g[f"level{l}_idx"]).cuda()].cpu().numpy()
        assert rel_max(got, g[f"level{l}_val"]) < TOL_VOLUME
    own = [blk.corr_pyramid[l][:, 0].cpu().numpy() for l in range(4)]
    flat = np.concatenate([x.reshape(-1) for x in own])
    for s in SIGMAS:
        co = cn.synth_coords(B, h, w, s, seed=1)
        got = blk.index_pyramid(centroids_coords=gpu(co)).cpu().numpy()
        # vs the oracle's lookup of OUR pyramid: isolates the lookup kernel (1e-3) ...
        assert rel_max(got, cc.index_pyramid(flat, co, 4, 4)) < TOL_LOOKUP
        # ... and end to end vs the fixture (bf16 operand error carried through): 2e-2
        assert rel_max(got.reshape(-1)[::33], g[f"lookup_sigma{s:g}_stride33"]) < TOL_VOLUME


def test_build_rejects_unsupported(lib):
    f = torch.zeros(1, 32, 18, 22, device="cuda")
    with pytest.raises(ValueError, match="RDVC_E_UNSUPPORTED"):
        rc.build_pyramid(f, f, 4)
    with pytest.raises(ValueError, match="too small"):
        rc.build_pyramid(torch.zeros(1, 64, 8, 22, device="cuda"), torch.zeros(1, 64, 8, 22, device="cuda"), 4)


def test_build_is_linear_and_deterministic(lib):
    B, D, h, w = 1, 64, 24, 40
    f1, f2 = cn.synth_fmaps(B, D, h, w, seed=13)
    a = rc.build_pyramid(gpu(f1), gpu(f2), 4).buffer.clone()
    b = rc.build_pyramid(gpu(f1), gpu(f2), 4).buffer.clone()
    assert torch.equal(a, b)                                   # bit-identical reruns
    p2 = rc.build_pyramid(gpu(f1), gpu(f2 * 2.0), 4)           # power-of-two scaling is exact in bf16
    p1 = rc.build_pyramid(gpu(f1), gpu(f2), 4)
    for l in range(4):
        assert torch.equal(p2.level(l), p1.level(l) * 2.0)
    # the layout only permutes storage: row-major and tiled builds hold bit-identical values
    pr = rc.build_pyramid(gpu(f1), gpu(f2), 4, layout=ROW)
    for l in range(4):
        assert torch.equal(pr.level(l), p1.level(l))


# ------------------------------------------------------------------ full size: 1920x1088
@pytest.mark.parametrize("vol", [torch.float32, torch.bfloat16], ids=["fp32vol", "bf16vol"])
def test_1080p_properties(lib, vol):
    """BASELINE.json config 2 shape, BOTH pyramid storage types (the bf16 volume takes another build
    instantiation -- 4 epilogue warps, 2 staging buffers, 4-stage ring -- and another lookup instantiation): the
    oracle cannot hold the 5.7 GB pyramid in seconds, so check size-independent properties + sampled rows
    against a torch fp64 matmul of the same rounded operands."""
    B, D, h, w = 1, 256, 136, 240
    N = h * w
    bf = vol == torch.bfloat16
    g = torch.Generator(device="cuda").manual_seed(0)
    f1 = torch.randn(B, D, h, w, device="cuda", generator=g)
    f2 = torch.randn(B, D, h, w, device="cuda", generator=g)
    blk = rc.TVCorrBlock(volume_dtype=vol)
    blk.build_pyramid(f1, f2)
    pyr = blk._pyr
    a = f1.to(torch.bfloat16).float().view(D, N)
    f2p = [f2] + [torch.nn.functional.avg_pool2d(f2, 2 ** l) for l in (1, 2, 3)]
    rows = torch.tensor([0, 1, 127, 128, 4097, 17000, N - 129, N - 1], device="cuda")
    shapes = [(136, 240), (68, 120), (34, 60), (17, 30)]
    for l in range(4):
        b = f2p[l].to(torch.bfloat16).float().view(D, -1)
        ref = (a[:, rows].t().double() @ b.double() / 16.0).float()
        got4 = pyr.level(l, rows)
        assert tuple(got4.shape) == (len(rows), 1) + shapes[l] and got4.dtype == vol
        got = got4[:, 0].reshape(len(rows), -1).float()
        err = (got - ref).abs().max().item() / ref.abs().max().item()
        tol = TOL_SAME_OPERANDS_BF16 if bf else (TOL_SAME_OPERANDS_F32 if l == 0 else TOL_SAME_OPERANDS_POOLED)
        assert err < tol, (l, err)
    # pyramid consistency: level l+1 is the 2x2 mean of level l (to bf16-operand accuracy)
    sl = torch.arange(5000, 5256, device="cuda")
    for l in range(3):
        lo, hi = pyr.level(l, sl).float(), pyr.level(l + 1, sl).float()
        pooled = torch.nn.functional.avg_pool2d(lo, 2)
        err = (pooled - hi).abs().max().item() / hi.abs().max().item()
        assert err < TOL_VOLUME, (l, err)
    # checksum of checksums: sum over fmap2 pixels == fmap1 . sum(fmap2)
    tot = pyr.level(0, rows)[:, 0].double().sum(dim=(1, 2))
    ref = (a[:, rows].t().double() @ f2.to(torch.bfloat16).double().view(D, N).sum(dim=1)) / 16.0
    assert ((tot - ref).abs().max() / ref.abs().max()).item() < (2e-2 if bf else 1e-3)
    # lookup at the identity grid: centre tap of level 0 is the volume diagonal
    co = gpu(cn.make_coords_grid(B, h, w))
    out = blk.index_pyramid(centroids_coords=co)
    assert out.shape == (B, 324, h, w) and out.is_contiguous() and out.dtype == torch.float32
    lv0 = pyr.level(0)                                   # (N, 1, h, w): 4.3 GB fp32 / 2.1 GB bf16
    assert torch.equal(out[0, 4 * 9 + 4].reshape(-1), lv0.view(N, N).diagonal().float())
    del lv0
    # and a drifting lookup against torchvision's own index_pyramid ON OUR PYRAMID (up-cast for the bf16 volume:
    # the kernel reads bf16 and interpolates in fp32, which is what grid_sample does on the up-cast copy)
    co2 = gpu(cn.synth_coords(B, h, w, 3.0, seed=4))
    got = blk.index_pyramid(centroids_coords=co2)
    ref = tv.index_pyramid([pyr.level(l).float() for l in range(4)], co2, 4)
    err = (got - ref).abs().max().item() / ref.abs().max().item()
    assert err < TOL_LOOKUP, err
    blk.release()


# ------------------------------------------------------------------ config 5: the resolution sweep, asserted
def _lookup_rows_reference(levels_rows, coords_rows, radius):
    """torchvision's index_pyramid arithmetic (TV:raft.py:394-422) on a SUBSET of query pixels: levels_rows[l] is
    (R, 1, h_l, w_l) fp32 (the rows' level images), coords_rows (R, 2) their (x, y) centroids -> (R, L*S*S)."""
    from torchvision.models.optical_flow._utils import grid_sample
    S = 2 * radius + 1
    di = torch.linspace(-radius, radius, S, device=coords_rows.device)
    delta = torch.stack(torch.meshgrid(di, di, indexing="ij"), dim=-1).view(1, S, S, 2)
    cc = coords_rows.view(-1, 1, 1, 2)
    out = []
    for lv in levels_rows:
        out.append(grid_sample(lv, cc + delta, align_corners=True, mode="bilinear").view(lv.shape[0], S * S))
        cc = cc / 2
    return torch.cat(out, dim=1)


@pytest.mark.parametrize("frame,vol", [((1280, 720), torch.float32), ((1280, 720), torch.bfloat16),
                                       ((2560, 1440), torch.float32), ((2560, 1440), torch.bfloat16),
                                       ((3840, 2160), torch.bfloat16)],
                         ids=["720p-fp32", "720p-bf16", "1440p-fp32", "1440p-bf16", "4k-bf16"])
def test_resolution_sweep_parity(lib, frame, vol):
    """BASELINE.json config 5 shapes (SURVEY.md 8d): build AND lookup parity on sampled query rows, including the
    last one, at sizes where pix * image_elems crosses 2^32 elements (1440p, 4K).  The volumes do not fit twice
    (4K bf16: 45 GB), so rows are read back with CorrPyramid.level(l, rows) and the lookup reference is
    torchvision's grid_sample arithmetic on just those rows' level images."""
    W, H = frame
    B, D, h, w = 1, 256, H // 8, W // 8
    N = h * w
    bf = vol == torch.bfloat16
    g = torch.Generator(device="cuda").manual_seed(7)
    f1 = torch.randn(B, D, h, w, device="cuda", generator=g)
    f2 = torch.randn(B, D, h, w, device="cuda", generator=g)
    blk = rc.TVCorrBlock(volume_dtype=vol)
    blk.build_pyramid(f1, f2)
    pyr = blk._pyr
    # incl. the first rows whose element offset pix * image_elems passes 2^31 and 2^32 (where they exist)
    rows = torch.tensor([0, 1, w - 1, w, N // 3, N // 2 + 7, min(N - 3, (1 << 31) // N + 1), min(N - 4, (1 << 32) // N + 1),
                         N - w - 1, N - 2, N - 1], device="cuda")
    a = f1.to(torch.bfloat16).float().view(D, N)[:, rows].t().double()
    lv_rows = []
    for l in range(4):
        b = torch.nn.functional.avg_pool2d(f2, 2 ** l) if l else f2
        ref = (a @ b.to(torch.bfloat16).double().view(D, -1) / 16.0).float()
        got = pyr.level(l, rows)
        assert tuple(got.shape) == (len(rows), 1, h >> l, w >> l)
        lv_rows.append(got.float())
        err = ((got[:, 0].reshape(len(rows), -1).float() - ref).abs().max() / ref.abs().max()).item()
        tol = TOL_SAME_OPERANDS_BF16 if bf else (TOL_SAME_OPERANDS_F32 if l == 0 else TOL_SAME_OPERANDS_POOLED)
        assert err < tol, (frame, l, err)
    # lookups of the whole frame; compare the sampled rows (fractional drift + some windows off the border)
    ys, xs = torch.meshgrid(torch.arange(h, device="cuda"), torch.arange(w, device="cuda"), indexing="ij")
    co = torch.stack([xs, ys], 0).float()[None] + 2.5 * torch.randn(1, 2, h, w, device="cuda", generator=g)
    out = blk.index_pyramid(centroids_coords=co)                       # (1, 324, h, w)
    got = out.view(324, N)[:, rows].t()
    ref = _lookup_rows_reference(lv_rows, co.view(2, N)[:, rows].t().contiguous(), 4)
    err = ((got - ref).abs().max() / ref.abs().max()).item()
    assert err < TOL_LOOKUP, (frame, err)
    blk.release()
    torch.cuda.empty_cache()


# ------------------------------------------------------------------ drop-in: torchvision RAFT
def _preprocess(frame_u8, size_hw):
    """R:codec_processing.py:751-759: to_tensor -> resize(antialias) -> [0,1], batch of 1."""
    import torchvision.transforms.functional as TF
    t = TF.resize(TF.to_tensor(frame_u8), list(size_hw), antialias=True)
    return t.unsqueeze(0)


def _seeded_raft(corr_block=None):
    from torchvision.models.optical_flow import raft_large
    torch.manual_seed(0)
    kw = {} if corr_block is None else {"corr_block": corr_block}
    return raft_large(weights=None, **kw).eval().cuda()


@pytest.mark.parametrize("vol_dtype", [torch.float32, torch.bfloat16])
def test_raft_flow_epe_vs_stock_torchvision(lib, golden_dir, vol_dtype):
    """BASELINE.json config 1 shape: R:im1.png / R:im2.png at 368x640, 12 updates, seed-0
    random-init raft_large (no weights offline), [0,1] inputs like the reference."""
    g = np.load(os.path.join(golden_dir, "frames_im1_im2.npz"))
    a = _preprocess(g["im1"], (368, 640)).cuda()
    b = _preprocess(g["im2"], (368, 640)).cuda()
    with torch.no_grad():
        ref = _seeded_raft()(a, b, num_flow_updates=12)[-1]
        blk = rc.TVCorrBlock(volume_dtype=vol_dtype)
        n0 = lib.rdvc_corr_launch_count()
        got = _seeded_raft(blk)(a, b, num_flow_updates=12)[-1]
        launched = lib.rdvc_corr_launch_count() - n0
    assert launched == 2 + 12, launched            # pack, build, 12 lookups
    epe = (got - ref).pow(2).sum(dim=1).sqrt()
    assert torch.isfinite(got).all()
    assert epe.mean().item() < TOL_EPE, epe.mean().item()
    # the CPU fixture (stock torchvision, CPU fp32) is a second, looser anchor
    cpu_ref = torch.from_numpy(g["flow_stride4"]).cuda()
    epe_cpu = (got[0, :, ::4, ::4] - cpu_ref).pow(2).sum(dim=0).sqrt()
    assert epe_cpu.mean().item() < 2 * TOL_EPE, epe_cpu.mean().item()


def test_raft_under_autocast(lib, golden_dir):
    """The reference's default GPU setting wraps RAFT in autocast (R:codec_processing.py:1436)."""
    g = np.load(os.path.join(golden_dir, "frames_im1_im2.npz"))
    a = _preprocess(g["im1"], (256, 448)).cuda()
    b = _preprocess(g["im2"], (256, 448)).cuda()
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
        ref = _seeded_raft()(a, b, num_flow_updates=12)[-1]
        got = _seeded_raft(rc.TVCorrBlock())(a, b, num_flow_updates=12)[-1]
    epe = (got.float() - ref.float()).pow(2).sum(dim=1).sqrt()
    assert epe.mean().item() < TOL_EPE, epe.mean().item()


def test_raft_flow_runner_matches_forward(lib, golden_dir):
    """rc.raft_flow == RAFT.forward(...)[-1] with the same block: same modules, same order, the 11
    unused mask/upsample passes skipped (the caller keeps only flow_preds[-1], R:codec_processing.py:1444)."""
    g = np.load(os.path.join(golden_dir, "frames_im1_im2.npz"))
    a = _preprocess(g["im1"], (256, 448)).cuda()
    b = _preprocess(g["im2"], (256, 448)).cuda()
    model = _seeded_raft(rc.TVCorrBlock())
    with torch.no_grad():
        ref = model(a, b, num_flow_updates=12)
        got = rc.raft_flow(model, a, b, num_flow_updates=12, fuse_convcorr1=False, fuse_encoder_tail=False)
        every = rc.raft_flow(model, a, b, num_flow_updates=12, all_predictions=True, fuse_convcorr1=False,
                             fuse_encoder_tail=False)
    assert torch.allclose(got, ref[-1], rtol=0, atol=1e-5)
    assert len(every) == 12 and all(torch.allclose(x, y, rtol=0, atol=1e-5) for x, y in zip(every, ref))
    fused = rc.raft_flow(model, a, b, num_flow_updates=12)      # default: both 1x1 convolutions fused (16-bit operands)
    assert (fused - ref[-1]).pow(2).sum(dim=1).sqrt().mean().item() < TOL_EPE
    with pytest.raises(TypeError):
        rc.raft_flow(_seeded_raft(), a, b)
    with pytest.raises(ValueError, match="divisible by 8"):
        rc.raft_flow(model, a[..., :250, :], b[..., :250, :])


def test_graphed_raft_flow_is_bit_identical(lib, golden_dir):
    """GraphedRaftFlow replays rc.raft_flow as one CUDA graph: same kernels, same order -> the same bits,
    for the captured pair and for new frames copied into the graph's static inputs."""
    g = np.load(os.path.join(golden_dir, "frames_im1_im2.npz"))
    a = _preprocess(g["im1"], (256, 448)).cuda()
    b = _preprocess(g["im2"], (256, 448)).cuda()
    model = _seeded_raft(rc.TVCorrBlock())
    runner = rc.GraphedRaftFlow(model, 12)
    with torch.no_grad():
        eager_ab = rc.raft_flow(model, a, b, 12)
        eager_ba = rc.raft_flow(model, b, a, 12)
    n0 = lib.rdvc_corr_launch_count()
    got_ab = runner(a, b)                 # warm-up + capture + replay
    captured = lib.rdvc_corr_launch_count() - n0
    got_ba = runner(b, a)                 # replay only: no launch goes through the C ABI again
    assert lib.rdvc_corr_launch_count() - n0 == captured
    assert torch.equal(got_ab, eager_ab) and torch.equal(got_ba, eager_ba)
    assert torch.equal(runner(a, b), eager_ab)
    with pytest.raises(TypeError):
        rc.GraphedRaftFlow(_seeded_raft())
    with pytest.raises(RuntimeError, match="inference only"):
        rc.GraphedRaftFlow(_seeded_raft(rc.TVCorrBlock()).train())
    runner.release()
    assert not runner._entries


def test_raft_flow_sequence_matches_pairs(lib, golden_dir):
    """rc.raft_flow_sequence(frames) == the flows of the consecutive pairs, the feature encoder having seen each frame
    once (n + 1 images instead of 2n): InstanceNorm is per sample, so only cuDNN's batch-size-dependent algorithm choice
    can differ -- and the pairs' flows against STOCK RAFT.forward stay inside the EPE budget."""
    g = np.load(os.path.join(golden_dir, "frames_im1_im2.npz"))
    a = _preprocess(g["im1"], (256, 448)).cuda()
    b = _preprocess(g["im2"], (256, 448)).cuda()
    frames = torch.cat([a, b, torch.roll(a, (3, -5), (2, 3)), torch.roll(b, (-2, 4), (2, 3))], 0)     # a run of 4 frames
    model = _seeded_raft(rc.TVCorrBlock())
    with torch.no_grad():
        for kw in ({}, {"fuse_convcorr1": False, "fuse_encoder_tail": False}):
            pairs = rc.raft_flow(model, frames[:-1], frames[1:], 12, **kw)
            seq = rc.raft_flow_sequence(model, frames, 12, **kw)
            assert seq.shape == pairs.shape == (3, 2, 256, 448)
            epe = (seq - pairs).pow(2).sum(dim=1).sqrt().mean().item()
            assert epe < 2e-3, (kw, epe)
        stock = _seeded_raft()
        ref = torch.cat([stock(frames[i:i + 1], frames[i + 1:i + 2], num_flow_updates=12)[-1] for i in range(3)], 0)
        assert (seq - ref).pow(2).sum(dim=1).sqrt().mean().item() < TOL_EPE
        every = rc.raft_flow_sequence(model, frames, 12, all_predictions=True)
        assert len(every) == 12 and every[-1].shape == (3, 2, 256, 448)
        with pytest.raises(ValueError, match="n \\+ 1"):
            rc.raft_flow_sequence(model, frames[:1], 12)
    # graphed: one graph per run length, bit-identical to the eager call, also for new frames
    runner = rc.GraphedRaftFlow(model, 12)
    with torch.no_grad():
        eager = rc.raft_flow_sequence(model, frames, 12)
        eager_rev = rc.raft_flow_sequence(model, frames.flip(0), 12)
    assert torch.equal(runner.sequence(frames), eager)
    assert torch.equal(runner.sequence(frames.flip(0).contiguous()), eager_rev)
    assert torch.equal(runner(frames[:-1], frames[1:]), rc.raft_flow(model, frames[:-1], frames[1:], 12))   # pair graphs coexist
    assert len(runner._entries) == 2
    runner.release()


def test_update_block_channels_last_and_graph_recapture(lib, golden_dir):
    """The fused path feeds the stock update block NHWC tensors and stores its weights NHWC (cuDNN then runs the same
    kernels without nchw<->nhwc transposes): same flow as with NCHW tensors.  Storing the weights NHWC re-allocates
    them, so a graph captured before must notice and re-capture instead of reading freed memory."""
    g = np.load(os.path.join(golden_dir, "frames_im1_im2.npz"))
    a = _preprocess(g["im1"], (256, 448)).cuda()
    b = _preprocess(g["im2"], (256, 448)).cuda()
    model = _seeded_raft(rc.TVCorrBlock())
    w = model.update_block.flow_head.conv1.weight
    runner = rc.GraphedRaftFlow(model, 12, update_block_channels_last=False)
    with torch.no_grad():
        nchw = rc.raft_flow(model, a, b, 12, update_block_channels_last=False)
        assert torch.equal(runner(a, b), nchw)
        assert model.update_block.flow_head.conv1.weight.is_contiguous()                     # untouched so far
        ptr0 = w.data_ptr()
        nhwc = rc.raft_flow(model, a, b, 12)                                                 # default: channels_last
        w2 = model.update_block.flow_head.conv1.weight
        assert w2.is_contiguous(memory_format=torch.channels_last) and w2.data_ptr() != ptr0
        assert (nhwc - nchw).pow(2).sum(dim=1).sqrt().mean().item() < 2e-3       # fp32 here: cuDNN picks other algorithms for NHWC
        stock = _seeded_raft()(a, b, num_flow_updates=12)[-1]
        assert (nhwc - stock).pow(2).sum(dim=1).sqrt().mean().item() < TOL_EPE
        n_before = len(runner._entries)
        again = runner(a, b)                                                                 # weights moved -> re-captured
        assert n_before == len(runner._entries) == 1
        assert (again - nchw).pow(2).sum(dim=1).sqrt().mean().item() < 2e-3      # NHWC weights now steer cuDNN's choice
        assert torch.equal(runner(b, a), rc.raft_flow(model, b, a, 12, update_block_channels_last=False))
    runner.release()


def test_princeton_facade(lib):
    B, D, h, w = 1, 64, 24, 40
    f1, f2 = cn.synth_fmaps(B, D, h, w, seed=21)
    corr = rc.CorrBlock(gpu(f1), gpu(f2), num_levels=4, radius=4)
    co = cn.synth_coords(B, h, w, 1.5, seed=5)
    got = corr(gpu(co)).cpu().numpy()
    own = np.concatenate([x[:, 0].cpu().numpy().reshape(-1) for x in corr.corr_pyramid])
    assert got.shape == (B, 324, h, w)
    assert rel_max(got, cc.index_pyramid(own, co, 4, 4)) < TOL_LOOKUP


# ------------------------------------------------------------------ other forms of the lookup result
@pytest.mark.parametrize("vol", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("radius,levels", [(4, 4), (3, 4), (4, 3), (2, 2)])
def test_lookup_output_forms(lib, radius, levels, vol):
    """rdvc_corr_lookup_ex: the fp16 NCHW result is the fp32 result rounded once; the K-major feature rows hold the
    same numbers (bf16 / fp16 rounded) at column l*PL + j*S + i for torchvision channel l*S*S + i*S + j, zeros in
    the padding columns."""
    B, C, h, w = 2, 8, 18, 22
    S = 2 * radius + 1
    f1, f2 = cn.synth_fmaps(B, C, h, w, seed=23)
    flat = cc.build_pyramid(f1, f2, levels)
    pyr = pyramid_from_levels(rc, cc.split_levels(flat, B, h, w, levels), B, h, w, vol)
    co = gpu(cn.synth_coords(B, h, w, 3.0, seed=2))
    ref = rc.index_pyramid(pyr, co, radius)                                     # (B, L*S*S, h, w) fp32
    assert torch.equal(rc.index_pyramid(pyr, co, radius, out_dtype=torch.float16), ref.half())
    kp = rc.corr_block.feat_pitch(levels, radius)
    PL = (S * S + 7) // 8 * 8
    assert kp == (levels * PL + 15) // 16 * 16
    # torchvision channel (l, i, j) -> column l*PL + j*S + i
    l_, i_, j_ = torch.meshgrid(torch.arange(levels), torch.arange(S), torch.arange(S), indexing="ij")
    col = (l_ * PL + j_ * S + i_).reshape(-1).cuda()
    M = B * h * w
    shape = rc.corr_block.feat_shape(B, h, w, levels, radius)
    assert shape == (kp // 8, (M + 7) // 8 * 8, 8)
    for fd in (torch.bfloat16, torch.float16):
        km = torch.full(shape, float("nan"), dtype=fd, device="cuda")
        rc.corr_block.index_pyramid_kmajor(pyr, co, radius, fd, out=km)
        want = torch.zeros((M, kp), dtype=fd, device="cuda")
        want[:, col] = ref.permute(0, 2, 3, 1).reshape(M, levels * S * S).to(fd)
        got = km[:, :M].permute(1, 0, 2).reshape(M, kp)                   # (chunk, row, 8) -> (row, K)
        assert torch.equal(got, want), (fd, radius, levels)
        assert torch.isnan(km[:, M:].float()).all()                       # rows past B*h*w are left alone
    with pytest.raises(ValueError, match="RDVC_LAYOUT_TILED"):
        rc.index_pyramid(pyramid_from_levels(rc, cc.split_levels(flat, B, h, w, levels), B, h, w, vol, layout=ROW),
                         co, radius, out_dtype=torch.float16)


TOL_CONV1X1_SAME_OPERANDS = 2e-5     # vs fp64 on the same 16-bit operands: fp32 accumulation over K = 324
TOL_CONV1X1 = 1e-2                   # vs the stock fp32 convolution of the un-rounded features (bf16 operands)


@pytest.mark.parametrize("shape", [(1, 46, 80), (2, 18, 22), (1, 17, 19), (3, 24, 40)])
@pytest.mark.parametrize("cout,fd,od", [(256, torch.bfloat16, torch.float32), (256, torch.float16, torch.float16),
                                        (96, torch.bfloat16, torch.bfloat16), (32, torch.float16, torch.float32)])
def test_conv1x1_matches_fp64(lib, shape, cout, fd, od):
    """rdvc_conv1x1 alone: random K-major feature rows (incl. garbage-free padding) x packed weights + bias, ReLU."""
    B, h, w = shape
    kp = rc.corr_block.feat_pitch(4, 4)
    g = torch.Generator(device="cuda").manual_seed(h * w + cout)
    feats_tv = torch.randn(B * h * w, 324, device="cuda", generator=g) * 3.0     # torchvision channel order
    weight = torch.randn(cout, 324, 1, 1, device="cuda", generator=g) * 0.1
    bias = torch.randn(cout, device="cuda", generator=g)
    l_, i_, j_ = torch.meshgrid(torch.arange(4), torch.arange(9), torch.arange(9), indexing="ij")
    col = (l_ * 88 + j_ * 9 + i_).reshape(-1).cuda()
    M = B * h * w
    rows = torch.zeros(M, kp, dtype=fd, device="cuda")
    rows[:, col] = feats_tv.to(fd)
    km = torch.full(rc.corr_block.feat_shape(B, h, w), float("nan"), dtype=fd, device="cuda")   # garbage rows past M
    km[:, :M] = rows.view(M, kp // 8, 8).permute(1, 0, 2)
    packed = rc.corr_block.PackedConv1x1(weight, bias, 4, 4, fd, "cuda")
    for relu in (True, False):
        got = rc.corr_block.conv1x1(km, packed, B, h, w, relu=relu, out_dtype=od)
        assert got.shape == (B, cout, h, w) and got.dtype == od
        ref = feats_tv.to(fd).double() @ weight.view(cout, 324).to(fd).double().t() + bias.double()
        if relu:
            ref = ref.clamp(min=0)
        ref = ref.view(B, h, w, cout).permute(0, 3, 1, 2)
        tol = TOL_CONV1X1_SAME_OPERANDS if od == torch.float32 else (1e-3 if od == torch.float16 else 8e-3)
        err = ((got.double() - ref).abs().max() / ref.abs().max()).item()
        assert err < tol, (shape, cout, fd, od, relu, err)


@pytest.mark.parametrize("hw,vol", [((46, 80), torch.float32), ((46, 80), torch.bfloat16), ((136, 240), torch.float32)])
def test_lookup_convcorr1_vs_stock_modules(lib, hw, vol):
    """Row f-1: TVCorrBlock.index_pyramid_convcorr1 == MotionEncoder.convcorr1(index_pyramid(coords)) (TV:raft.py:185,
    202) of a seed-0 raft_large, at RDVC's default RAFT size and at 1080p: <= 2e-3 max-norm relative with the default
    fp16 operands, <= 1e-2 with bf16 operands, and <= 5e-3 under fp16 autocast against the stock fp16 convolution."""
    h, w = hw
    B, D = 1, 256
    model = _seeded_raft(rc.TVCorrBlock(volume_dtype=vol))
    conv = model.update_block.motion_encoder.convcorr1
    g = torch.Generator(device="cuda").manual_seed(11)
    f1 = torch.randn(B, D, h, w, device="cuda", generator=g)
    f2 = torch.randn(B, D, h, w, device="cuda", generator=g)
    blk = model.corr_block
    blk.build_pyramid(f1, f2)
    co = gpu(cn.synth_coords(B, h, w, 2.0, seed=3))
    with torch.no_grad():
        torch.backends.cudnn.allow_tf32 = False
        ref = conv(blk.index_pyramid(centroids_coords=co))
        torch.backends.cudnn.allow_tf32 = True
        n0 = lib.rdvc_corr_launch_count()
        got = blk.index_pyramid_convcorr1(co, conv[0].weight, conv[0].bias)       # default: fp16 operands
        assert lib.rdvc_corr_launch_count() - n0 == 2                   # lookup (K-major features) + GEMM
        assert got.shape == ref.shape == (B, 256, h, w) and got.dtype == torch.float32
        err = ((got - ref).abs().max() / ref.abs().max()).item()
        assert err < 2e-3, err
        assert (got >= 0).all()
        got_bf = blk.index_pyramid_convcorr1(co, conv[0].weight, conv[0].bias, feat_dtype=torch.bfloat16)
        err_bf = ((got_bf - ref).abs().max() / ref.abs().max()).item()
        assert err_bf < TOL_CONV1X1, err_bf
        with torch.autocast("cuda", dtype=torch.float16):
            ref16 = conv(blk.index_pyramid(centroids_coords=co))
            got16 = blk.index_pyramid_convcorr1(co, conv[0].weight, conv[0].bias)
        assert got16.dtype == ref16.dtype == torch.float16
        err16 = ((got16.float() - ref16.float()).abs().max() / ref16.float().abs().max()).item()
        assert err16 < 5e-3, err16
    blk.release()


@pytest.mark.parametrize("size", [(368, 640), (1088, 1920)], ids=["368x640", "1080p"])
def test_raft_flow_fused_convcorr1_epe(lib, golden_dir, size):
    """rc.raft_flow with the lookup fused into convcorr1 (its default) vs STOCK torchvision RAFT.forward: mean EPE
    < 0.05 px at RDVC's default RAFT size and at 1920x1088 (BASELINE.json config 3's frame size), 12 updates;
    3 + 2 x 12 launches of this library per pair (pack, encoder tail, build; lookup + 1x1 GEMM per update)."""
    g = np.load(os.path.join(golden_dir, "frames_im1_im2.npz"))
    a = _preprocess(g["im1"], size).cuda()
    b = _preprocess(g["im2"], size).cuda()
    with torch.no_grad():
        ref = _seeded_raft()(a, b, num_flow_updates=12)[-1]
        model = _seeded_raft(rc.TVCorrBlock())
        n0 = lib.rdvc_corr_launch_count()
        got = rc.raft_flow(model, a, b, 12)
        assert lib.rdvc_corr_launch_count() - n0 == 3 + 2 * 12
        unfused = rc.raft_flow(model, a, b, 12, fuse_convcorr1=False, fuse_encoder_tail=False)
        only_tail = rc.raft_flow(model, a, b, 12, fuse_convcorr1=False)
        assert (only_tail - ref).pow(2).sum(dim=1).sqrt().mean().item() < TOL_EPE
    assert torch.isfinite(got).all()
    epe = (got - ref).pow(2).sum(dim=1).sqrt().mean().item()
    epe_u = (unfused - ref).pow(2).sum(dim=1).sqrt().mean().item()
    assert epe < TOL_EPE and epe_u < TOL_EPE, (epe, epe_u)
    model.corr_block.release()


@pytest.mark.parametrize("vol", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", [(1, 46, 80), (2, 18, 22), (1, 17, 19), (1, 33, 47)])
def test_build_from_encoder_tail(lib, shape, vol):
    """Row f-2, last sub-item: TVCorrBlock.build_pyramid_from_encoder(x1, x2, W, b) == build_pyramid(conv(x1), conv(x2))
    for the feature encoder's final 1x1 convolution (TV:raft.py:139,150), without the fp32 feature maps: vs an fp64
    evaluation with the SAME rounding points (pooled activations, weights and operand rows rounded to bf16 once
    each), vs the stock order of work through rdvc_corr_build, and the layout's padding pixels stay exact zeros
    (the bias must not leak into them)."""
    B, h, w = shape
    Din, Dout, L = 128, 256, 4
    g = torch.Generator(device="cuda").manual_seed(h * w + B)
    x1 = torch.randn(B, Din, h, w, device="cuda", generator=g).relu()          # post-ReLU activations like the encoder's
    x2 = torch.randn(B, Din, h, w, device="cuda", generator=g).relu()
    W = torch.randn(Dout, Din, 1, 1, device="cuda", generator=g) * 0.09
    bias = torch.randn(Dout, device="cuda", generator=g) * 0.5
    blk = rc.TVCorrBlock(volume_dtype=vol)
    n0 = lib.rdvc_corr_launch_count()
    blk.build_pyramid_from_encoder(x1, x2, W, bias)
    assert lib.rdvc_corr_launch_count() - n0 == 3                              # pack, encoder tail, build
    bf = lambda t: t.to(torch.bfloat16).double()
    Wd = bf(W.view(Dout, Din))
    rows1 = bf((bf(x1).view(B, Din, h * w).transpose(1, 2) @ Wd.t() + bias.double()).float())      # (B, N, 256)
    tol = TOL_SAME_OPERANDS_BF16 if vol == torch.bfloat16 else TOL_SAME_OPERANDS_POOLED
    # the stock order of work: fp32 convolution, then the library's own build
    torch.backends.cudnn.allow_tf32 = False
    f1 = torch.nn.functional.conv2d(x1, W, bias)
    f2 = torch.nn.functional.conv2d(x2, W, bias)
    torch.backends.cudnn.allow_tf32 = True
    stock = rc.build_pyramid(f1, f2, L, vol)
    for l in range(L):
        xp = torch.nn.functional.avg_pool2d(x2, 2 ** l) if l else x2
        rows2 = bf((bf(xp).flatten(2).transpose(1, 2) @ Wd.t() + bias.double()).float())          # (B, n_l, 256)
        ref = (rows1 @ rows2.transpose(1, 2) / 16.0).reshape(B * h * w, h >> l, w >> l)
        got = blk._pyr.level(l)[:, 0].double()
        err = ((got - ref).abs().max() / ref.abs().max()).item()
        assert err < tol, (shape, l, err)
        err_stock = ((got - stock.level(l)[:, 0].double()).abs().max() / ref.abs().max()).item()
        assert err_stock < TOL_VOLUME, (shape, l, err_stock)
        hl, wl, tw, th, hp, wp = blk._pyr._tiles(l)                            # padding pixels: exact zeros
        raw = blk._pyr.storage(l)
        st = raw[:, : hp * wp].reshape(-1, hp // th, wp // tw, th, tw).permute(0, 1, 3, 2, 4).reshape(-1, hp, wp)
        assert not st[:, hl:, :].any() and not st[:, :, wl:].any() and not raw[:, hp * wp:].any()
    # fp16 activations keep fp16 operands (what the stock path multiplies under the reference's autocast)
    blk.build_pyramid_from_encoder(x1.half(), x2.half(), W, bias)
    err16 = ((blk._pyr.level(0)[:, 0].double() - stock.level(0)[:, 0].double()).abs().max() / stock.level(0).abs().max()).item()
    assert err16 < TOL_VOLUME, err16
    with pytest.raises(ValueError, match="input channels"):
        blk.build_pyramid_from_encoder(x1[:, :64], x2[:, :64], W, bias)
    # the interchange layout (no padding rows): the same numbers, bit for bit
    blk.build_pyramid_from_encoder(x1, x2, W, bias)
    row = rc.TVCorrBlock(volume_dtype=vol, layout=ROW)
    row.build_pyramid_from_encoder(x1, x2, W, bias)
    for l in range(L):
        assert torch.equal(row._pyr.level(l), blk._pyr.level(l)), l
    blk.release()
    row.release()


def test_build_plan_cache(lib):
    """A repeated rdvc_corr_build with the same buffers, shape and options finds its TMA descriptors and work split
    in the per-process cache (SURVEY.md 8b) and writes the same bits; another shape or option misses."""
    B, D, h, w = 1, 64, 24, 40
    f1, f2 = cn.synth_fmaps(B, D, h, w, seed=51)
    blk = rc.TVCorrBlock()
    blk.build_pyramid(gpu(f1), gpu(f2))
    first = blk._pyr.buffer.clone()
    h0 = lib.rdvc_corr_plan_cache_hits()
    blk.build_pyramid(gpu(f1), gpu(f2))                 # same pyramid buffer and workspace are reused by the block
    assert lib.rdvc_corr_plan_cache_hits() == h0 + 1
    assert torch.equal(blk._pyr.buffer, first)
    set_opts(lib, msplit=3)
    blk.build_pyramid(gpu(f1), gpu(f2))                 # an option changed: new plan, same result
    assert lib.rdvc_corr_plan_cache_hits() == h0 + 1
    assert torch.equal(blk._pyr.buffer, first)
    set_opts(lib, msplit=0)


# ------------------------------------------------------------------ ABI details
def test_pair_host_entry_point(lib):
    """rdvc_corr_pair_host: host buffers in, host buffers out, same numbers as the device calls."""
    B, D, h, w, iters = 1, 64, 24, 40, 3
    f1, f2 = cn.synth_fmaps(B, D, h, w, seed=31)
    coords = np.stack([cn.synth_coords(B, h, w, 1.0 + i, seed=i) for i in range(iters)])
    out = np.empty((iters, B, 324, h, w), np.float32)
    fp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    rc_ = lib.rdvc_corr_pair_host(fp(f1), fp(f2), fp(coords), fp(out), B, D, h, w, 4, 4, iters, rc.RDVC_DT_F32)
    rc._cabi.check(rc_, "rdvc_corr_pair_host")
    blk = rc.TVCorrBlock()
    blk.build_pyramid(gpu(f1), gpu(f2))
    for i in range(iters):
        ref = blk.index_pyramid(centroids_coords=gpu(coords[i])).cpu().numpy()
        assert np.array_equal(out[i], ref)
    # the split call: two pairs in flight on the two slots, each result in its own host buffer
    out2 = [np.empty_like(out), np.empty_like(out)]
    f1b, f2b = cn.synth_fmaps(B, D, h, w, seed=32)
    for slot, (x1, x2) in enumerate(((f1, f2), (f1b, f2b))):
        rc._cabi.check(lib.rdvc_corr_pair_host_submit(fp(x1), fp(x2), fp(coords), fp(out2[slot]), B, D, h, w, 4, 4,
                                                      iters, rc.RDVC_DT_F32, slot), "submit")
    assert lib.rdvc_corr_pair_host_submit(fp(f1), fp(f2), fp(coords), fp(out2[0]), B, D, h, w, 4, 4, iters,
                                          rc.RDVC_DT_F32, 0) == -5          # slot 0 is still pending
    for slot in (0, 1):
        rc._cabi.check(lib.rdvc_corr_pair_host_wait(slot), "wait")
    assert np.array_equal(out2[0], out)
    blk.build_pyramid(gpu(f1b), gpu(f2b))
    for i in range(iters):
        assert np.array_equal(out2[1][i], blk.index_pyramid(centroids_coords=gpu(coords[i])).cpu().numpy())
    assert lib.rdvc_corr_pair_host_wait(1) == 0 and lib.rdvc_corr_pair_host_wait(5) == -5
    # fp16 results (half the bytes over PCIe): the fp32 results rounded once
    out16 = np.empty((iters, B, 324, h, w), np.float16)
    rc._cabi.check(lib.rdvc_corr_pair_host_submit_ex(fp(f1), fp(f2), fp(coords), fp(out16), B, D, h, w, 4, 4, iters,
                                                     rc.RDVC_DT_F32, rc.RDVC_DT_F16, 0), "submit_ex")
    rc._cabi.check(lib.rdvc_corr_pair_host_wait(0), "wait")
    assert np.array_equal(out16, out.astype(np.float16))
    assert lib.rdvc_corr_pair_host_submit_ex(fp(f1), fp(f2), fp(coords), fp(out16), B, D, h, w, 4, 4, iters,
                                             7, rc.RDVC_DT_F16, 0) == -4            # bad vol_dtype: RDVC_E_DTYPE
    lib.rdvc_corr_release()


@pytest.mark.parametrize("mode,layout", [("fused", ROW), ("linear", ROW), ("linear", TILED)])
@pytest.mark.parametrize("vol", [torch.float32, torch.bfloat16])
def test_no_out_of_bounds_writes(lib, mode, layout, vol):
    """compute-sanitizer is closed on this pool, so bounds are checked with canaries: every byte
    outside the pyramid levels / lookup output / workspace (guard bands before and after, and the
    256-byte padding between levels) must survive a build + lookups on odd shapes."""
    need_experiments(mode)
    CANARY, GUARD = 0xAB, 4096
    vd = rc.RDVC_DT_F32 if vol == torch.float32 else rc.RDVC_DT_BF16
    es = 4 if vol == torch.float32 else 2
    set_opts(lib, mode=MODES[mode])
    for (B, D, h, w) in [(2, 64, 18, 22), (1, 128, 33, 47), (1, 64, 17, 16)]:
        N = h * w
        f1, f2 = cn.synth_fmaps(B, D, h, w, seed=3)
        a, b = gpu(f1), gpu(f2)
        pb = lib.rdvc_corr_pyramid_bytes(B, h, w, 4, vd, layout)
        wb = lib.rdvc_corr_workspace_bytes(B, D, h, w)
        ob = B * 324 * N * 4
        bufs = {k: torch.full((n + 2 * GUARD,), CANARY, dtype=torch.uint8, device="cuda")
                for k, n in (("pyr", pb), ("ws", wb), ("out", ob))}
        ptr = {k: v.data_ptr() + GUARD for k, v in bufs.items()}
        assert all(p % 256 == 0 for p in ptr.values())
        st = torch.cuda.current_stream().cuda_stream
        rc._cabi.check(lib.rdvc_corr_build(a.data_ptr(), b.data_ptr(), B, D, h, w, rc.RDVC_DT_F32, ptr["pyr"],
                                           vd, layout, 4, ptr["ws"], wb, st), "build")
        co = gpu(cn.synth_coords(B, h, w, 5.0, seed=1))
        for variant in (1, 2):
            set_opts(lib, lookup=variant)
            rc._cabi.check(lib.rdvc_corr_lookup(ptr["pyr"], vd, layout, co.data_ptr(), B, h, w, 4, 4, ptr["out"],
                                                st), "lookup")
        torch.cuda.synchronize()
        for k, v in bufs.items():
            assert bool((v[:GUARD] == CANARY).all()) and bool((v[-GUARD:] == CANARY).all()), (k, "guard band")
        body = bufs["pyr"][GUARD:-GUARD]
        for l in range(4):
            off = lib.rdvc_corr_level_offset_bytes(B, h, w, l, vd, layout)
            end = off + B * N * lib.rdvc_corr_level_image_elems(h, w, l, vd, layout) * es
            nxt = lib.rdvc_corr_level_offset_bytes(B, h, w, l + 1, vd, layout)
            assert bool((body[end:nxt] == CANARY).all()), ("padding after level", l)
            lvl = body[off:end].view(vol).float()
            assert torch.isfinite(lvl).all()          # every element was written (0xABAB.. is finite but
            assert not bool((body[off:end] == CANARY).all())   # ... the level is not all canary)
        assert torch.isfinite(bufs["out"][GUARD:-GUARD].view(torch.float32)).all()
    set_opts(lib, mode=0, lookup=0)


@pytest.mark.parametrize("fdt", [torch.float16, torch.bfloat16])
def test_no_out_of_bounds_writes_round2_entry_points(lib, fdt):
    """The same canary check for the round-2 entry points on odd shapes: K-major lookup (rdvc_corr_lookup_ex), the 1x1
    GEMM (rdvc_conv1x1, vector and scalar store paths), pack -> encoder tail -> packed build.  Guard bands before and
    after every buffer the library writes must survive; feature rows beyond B*h*w are documented as not written."""
    import ctypes
    CANARY, GUARD = 0xAB, 4096
    vd, layout = rc.RDVC_DT_F32, TILED
    fd = rc.RDVC_DT_F16 if fdt == torch.float16 else rc.RDVC_DT_BF16
    st = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device="cuda").manual_seed(5)
    for (B, Din, h, w, cout) in [(2, 128, 18, 22, 256), (1, 128, 33, 47, 96), (1, 128, 17, 16, 32)]:
        N, D = h * w, 256
        x1 = torch.randn(B, Din, h, w, device="cuda", generator=g)
        x2 = torch.randn(B, Din, h, w, device="cuda", generator=g)
        wt = torch.randn(D, Din, generator=torch.Generator().manual_seed(1)) / Din ** 0.5
        wp = np.zeros(D * Din, np.uint16)
        w32 = wt.numpy().copy()
        rc._cabi.check(lib.rdvc_linear_pack_weights(w32.ctypes.data_as(ctypes.c_void_p), D, Din, fd,
                                                    wp.ctypes.data_as(ctypes.c_void_p)), "pack linear")
        wdev = torch.from_numpy(wp.view(np.int16)).cuda()
        kp = lib.rdvc_corr_feat_pitch(4, 4)
        rows = lib.rdvc_corr_feat_rows(B, h, w)
        sizes = {"pyr": lib.rdvc_corr_pyramid_bytes(B, h, w, 4, vd, layout),
                 "ws_in": lib.rdvc_corr_workspace_bytes(B, Din, h, w),
                 "ws": lib.rdvc_corr_workspace_bytes(B, D, h, w),
                 "feat": lib.rdvc_corr_feat_bytes(B, h, w, 4, 4),
                 "out32": B * cout * N * 4, "out16": B * cout * N * 2}
        bufs = {k: torch.full((n + 2 * GUARD,), CANARY, dtype=torch.uint8, device="cuda") for k, n in sizes.items()}
        ptr = {k: v.data_ptr() + GUARD for k, v in bufs.items()}
        assert all(p % 256 == 0 for p in ptr.values())
        rc._cabi.check(lib.rdvc_corr_pack(x1.data_ptr(), x2.data_ptr(), B, Din, h, w, rc.RDVC_DT_F32, vd, layout, 4,
                                          ptr["ws_in"], sizes["ws_in"], st), "pack")
        rc._cabi.check(lib.rdvc_corr_encoder_tail(ptr["ws_in"], sizes["ws_in"], Din, wdev.data_ptr(), 0, D, B, h, w, fd,
                                                  vd, layout, 4, ptr["ws"], sizes["ws"], st), "tail")
        rc._cabi.check(lib.rdvc_corr_build_packed(B, D, h, w, fd, ptr["pyr"], vd, layout, 4, ptr["ws"], sizes["ws"], st),
                       "build_packed")
        co = gpu(cn.synth_coords(B, h, w, 5.0, seed=1))
        rc._cabi.check(lib.rdvc_corr_lookup_ex(ptr["pyr"], vd, layout, co.data_ptr(), B, h, w, 4, 4, ptr["feat"], fd,
                                               rc._cabi.RDVC_OUT_KMAJOR, st), "lookup_ex")
        cw = torch.randn(cout, 324, generator=torch.Generator().manual_seed(2)) / 18
        packed = rc.corr_block.PackedConv1x1(cw, torch.zeros(cout), 4, 4, fdt, "cuda")
        for key, od in (("out32", rc.RDVC_DT_F32), ("out16", rc.RDVC_DT_F16)):
            rc._cabi.check(lib.rdvc_conv1x1(ptr["feat"], fd, packed.weight.data_ptr(), packed.bias.data_ptr(), B, h, w,
                                            4, 4, cout, rc._cabi.RDVC_ACT_RELU, ptr[key], od, st), "conv1x1")
        torch.cuda.synchronize()
        for k, v in bufs.items():
            assert bool((v[:GUARD] == CANARY).all()) and bool((v[-GUARD:] == CANARY).all()), (k, "guard band", (B, h, w))
        feat = bufs["feat"][GUARD:-GUARD].view(kp // 8, rows, 16)
        assert bool((feat[:, B * N:, :] == CANARY).all()), "feature rows beyond B*h*w were written"
        assert not bool((feat[:, :B * N, :] == CANARY).all(dim=-1).any()), "a feature row chunk was not written"
        o32 = bufs["out32"][GUARD:-GUARD].view(torch.float32)
        o16 = bufs["out16"][GUARD:-GUARD].view(torch.float16)
        assert torch.isfinite(o32).all() and bool((o32 >= 0).all())        # every element written (canary = -1.2e-12 < 0)
        assert torch.equal(o32.to(torch.float16), o16)


def test_inputs_requiring_grad_are_refused(lib):
    """Forward-only: with grad mode on, activations that require grad raise (a silent ``detach`` would train nothing)."""
    f1 = torch.randn(1, 64, 16, 16, device="cuda", requires_grad=True)
    f2 = torch.randn(1, 64, 16, 16, device="cuda")
    blk = rc.TVCorrBlock()
    with pytest.raises(RuntimeError, match="forward-only"):
        blk.build_pyramid(f1, f2)
    with torch.no_grad():
        blk.build_pyramid(f1, f2)
    co = torch.zeros(1, 2, 16, 16, device="cuda", requires_grad=True)
    with pytest.raises(RuntimeError, match="forward-only"):
        blk.index_pyramid(co)
    assert blk.index_pyramid(co.detach()).shape == (1, 324, 16, 16)
    x = torch.rand(1, 3, 32, 32, device="cuda", requires_grad=True)
    with pytest.raises(RuntimeError, match="forward-only"):
        rc.WarpingLayer()(x, torch.zeros(1, 2, 32, 32, device="cuda"))
    blk.release()


def test_runs_on_callers_stream(lib):
    B, D, h, w = 1, 64, 24, 40
    f1, f2 = cn.synth_fmaps(B, D, h, w, seed=41)
    a, b = gpu(f1), gpu(f2)
    co = gpu(cn.synth_coords(B, h, w, 2.0, seed=1))
    ref = rc.CorrBlock(a, b)(co)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        got = rc.CorrBlock(a, b)(co)
    s.synchronize()
    assert torch.equal(got, ref)


# ------------------------------------------------------------------ next row: flow resize + warp
TOL_FLOW_RESIZE = 1e-5    # relative to max(1, max|flow|): fp32 bilinear, same association as aten
TOL_WARP = 1e-3           # absolute, images in [0,1]: the reference rounds its sampling grid through
                          # linspace(-1,1,W) + flow/((W-1)/2) in fp32 (~1e-4 px at W = 1920); ours samples
                          # at the absolute coordinate j + dx


def test_motion_warp_matches_reference_fixtures(lib, golden_dir):
    """rdvc_motion_warp vs the outputs of the reference's own resize_flow + WarpingLayer."""
    from oracle import motion_warp as mw
    g = np.load(os.path.join(golden_dir, "motion_warp.npz"))
    names = sorted(k[: -len("_shape")] for k in g.files if k.endswith("_shape"))
    for name in names:
        B, C, H, W, h_in, w_in = [int(v) for v in g[f"{name}_shape"]]
        img, flow = mw.synth_case(B, C, H, W, h_in, w_in, float(g[f"{name}_sigma"]), seed=len(name))
        n0 = lib.rdvc_corr_launch_count()
        warped, f = rc.motion_warp(gpu(img), gpu(flow), (H, W))
        assert lib.rdvc_corr_launch_count() - n0 == 1                  # one launch for both steps
        scale = max(1.0, float(np.abs(g[f"{name}_flow_frame"]).max()))
        assert np.abs(f.cpu().numpy() - g[f"{name}_flow_frame"]).max() / scale < TOL_FLOW_RESIZE, name
        assert np.abs(warped.cpu().numpy() - g[f"{name}_warped"]).max() < TOL_WARP, name
        # the two reference-named entry points give the same numbers as the fused call
        f2 = rc.resize_flow(gpu(flow), (H, W))
        assert torch.equal(f2, f) if (h_in, w_in) != (H, W) else f2.data_ptr() != 0
        assert torch.equal(rc.WarpingLayer()(gpu(img), f), warped)


def test_motion_warp_vs_torch_ops_odd_shapes(lib):
    """Against the same torch ops the reference composes (interpolate + grid_sample), on the GPU, for
    shapes the fixtures do not cover (up- and down-scaling, C = 1..4, B = 3)."""
    import torch.nn.functional as F
    for (B, C, H, W, h_in, w_in) in [(3, 1, 31, 45, 17, 23), (1, 4, 64, 96, 72, 104), (2, 3, 50, 50, 25, 100)]:
        gen = torch.Generator(device="cuda").manual_seed(H * W)
        x = torch.rand(B, C, H, W, device="cuda", generator=gen)
        fl = 3.0 * torch.randn(B, 2, h_in, w_in, device="cuda", generator=gen)
        warped, f = rc.motion_warp(x, fl, (H, W))
        ref_f = F.interpolate(fl, size=(H, W), mode="bilinear", align_corners=False, antialias=False)
        ref_f = ref_f * torch.tensor([W / w_in, H / h_in], device="cuda").view(1, 2, 1, 1)
        assert ((f - ref_f).abs().max() / ref_f.abs().max().clamp(min=1)).item() < TOL_FLOW_RESIZE
        gy, gx = torch.meshgrid(torch.linspace(-1, 1, H, device="cuda"), torch.linspace(-1, 1, W, device="cuda"), indexing="ij")
        grid = torch.stack((gx, gy), 2)[None] + torch.stack((ref_f[:, 0] / ((W - 1) / 2), ref_f[:, 1] / ((H - 1) / 2)), 3)
        ref_w = F.grid_sample(x, grid, mode="bilinear", padding_mode="border", align_corners=True)
        assert (warped - ref_w).abs().max().item() < TOL_WARP


def test_motion_warp_1080p_properties(lib):
    """Frame 1920x1080, RAFT flow at 1920x1088 (R:codec_processing.py:1446): size-independent properties."""
    B, C, H, W, h_in, w_in = 1, 3, 1080, 1920, 1088, 1920
    gen = torch.Generator(device="cuda").manual_seed(7)
    x = torch.rand(B, C, H, W, device="cuda", generator=gen)
    zero = torch.zeros(B, 2, h_in, w_in, device="cuda")
    warped, f = rc.motion_warp(x, zero, (H, W))
    assert torch.equal(warped, x) and not f.any()                       # zero flow: identity, bit exact
    shift = zero.clone(); shift[:, 0] = 5.0; shift[:, 1] = -3.0 * h_in / H   # dy scales by H / h_in -> -3 px
    warped, f = rc.motion_warp(x, shift, (H, W))
    assert torch.allclose(f[:, 0], torch.full_like(f[:, 0], 5.0)) and torch.allclose(f[:, 1], torch.full_like(f[:, 1], -3.0), atol=1e-5)
    assert torch.allclose(warped[:, :, 3:, : W - 5], x[:, :, : H - 3, 5:], atol=2e-5)   # integer shift = copy
    assert torch.allclose(warped[:, :, 3:, W - 5:], x[:, :, : H - 3, W - 1:].expand(-1, -1, -1, 5), atol=2e-5)  # border
    lin = torch.arange(w_in, device="cuda", dtype=torch.float32).view(1, 1, 1, w_in).expand(B, 1, h_in, w_in)
    fl = torch.cat([lin * 0.001, lin * 0.0], 1).contiguous()             # resize is linear: exact on a ramp
    f = rc.resize_flow(fl, (H, W))
    assert torch.allclose(f[:, 0], (lin[:, 0, :H] * 0.001), atol=1e-5) and f.shape == (B, 2, H, W)


# ------------------------------------------------------------------ next row: frame preparation
TOL_PREP = 2e-5           # absolute on [0, 1]: fp32 triangle-filter sums in one pass instead of aten's two
                          # (observed up to 9e-6 at 1080 -> 1088)


def test_preprocess_matches_reference_fixtures(lib, golden_dir):
    """rdvc_preprocess_frame vs the outputs of the reference's own preprocess_frame_raft / _codec."""
    from oracle import preprocess as pp
    g = np.load(os.path.join(golden_dir, "preprocess.npz"))
    for name in sorted(k[: -len("_shape")] for k in g.files if k.endswith("_shape")):
        H, W, C, h, w = [int(v) for v in g[f"{name}_shape"]]
        frame = pp.synth_frame(H, W, C, seed=len(name))
        fr = frame if C > 1 else frame[:, :, 0]
        got = rc.preprocess_frame_raft(fr, (h, w), torch.device("cuda"))
        assert got.shape == (1, C, h, w) and got.dtype == torch.float32
        assert np.abs(got.cpu().numpy() - g[f"{name}_raft"]).max() < TOL_PREP, name
        assert np.abs(rc.preprocess_frame_codec(fr, "cuda").cpu().numpy() - g[f"{name}_codec"]).max() < 1e-7, name


def test_preprocess_1080p_vs_torchvision(lib):
    """Full size against the reference's ops run on the GPU: 1080p -> 1088x1920 (what the 1080p runs need) and
    1080p -> 368x640 (the reference's default RAFT size, 2.9x down with anti-aliasing)."""
    import torchvision.transforms.functional as TF
    from oracle import preprocess as pp
    frame = pp.synth_frame(1080, 1920, 3, seed=3)
    t = torch.from_numpy(frame).cuda().permute(2, 0, 1).float() / 255.0
    for size in ((1088, 1920), (368, 640), (1080, 1920)):
        n0 = lib.rdvc_corr_launch_count()
        got = rc.preprocess_frame_raft(frame, size, "cuda")
        assert lib.rdvc_corr_launch_count() - n0 == 1
        ref = TF.resize(t, list(size), antialias=True).unsqueeze(0)
        assert (got - ref).abs().max().item() < TOL_PREP, size
    assert torch.equal(rc.preprocess_frame_codec(frame, "cuda")[0], (t * 255.0).round() / 255.0) or \
        (rc.preprocess_frame_codec(frame, "cuda")[0] - t).abs().max().item() < 1e-7


# ------------------------------------------------------------------ randomized sweep over the parameter space
def test_random_configurations_against_oracle(lib):
    """24 seeded random configurations (batch, channels, odd sizes, levels, radius, storage type, layout):
    build vs the fp64 statement of what the kernel multiplies, lookup vs the C oracle on the library's pyramid."""
    rng = np.random.default_rng(2026)
    for case in range(24):
        levels = int(rng.integers(1, 5))
        lo = 2 * 2 ** (levels - 1)
        B, D = int(rng.integers(1, 3)), int(rng.choice([64, 128, 192, 256]))
        h, w = int(rng.integers(lo, 41)), int(rng.integers(lo, 49))
        radius = int(rng.integers(1, 5))
        vol = torch.float32 if rng.random() < 0.5 else torch.bfloat16
        layout = ROW if rng.random() < 0.4 else TILED
        sigma = float(rng.choice([0.0, 0.5, 3.0, 30.0]))
        tag = (case, B, D, h, w, levels, radius, str(vol), layout, sigma)
        f1, f2 = cn.synth_fmaps(B, D, h, w, seed=100 + case)
        pyr = rc.build_pyramid(gpu(f1), gpu(f2), levels, vol, layout=layout)
        ref = ref_pyramid_linear(f1, f2, levels)
        own = []
        for l in range(levels):
            got = pyr.level(l)[:, 0].float().cpu().numpy()
            tol = TOL_SAME_OPERANDS_BF16 if vol == torch.bfloat16 else (TOL_SAME_OPERANDS_F32 if l == 0 else TOL_SAME_OPERANDS_POOLED)
            assert rel_max(got, ref[l]) < tol, tag + (l,)
            own.append(got)
        co = cn.synth_coords(B, h, w, sigma, seed=case)
        got = rc.index_pyramid(pyr, gpu(co), radius).cpu().numpy()
        flat = np.concatenate([x.reshape(-1) for x in own])
        assert got.shape == (B, levels * (2 * radius + 1) ** 2, h, w)
        assert rel_max(got, cc.index_pyramid(flat, co, levels, radius)) < TOL_LOOKUP, tag
