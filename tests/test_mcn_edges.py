"""Motion-compensation network (DESIGN 3.6): the tcgen05 convolutions at every tile edge, MMA schedule, persistent-loop
residue, batch and entry point.  test_mcn.py checks a handful of shapes; this file sweeps the places where the two
kernels (mcn_conv_kernel: three boxes per 16-super-pixel tile; mcn_convx_kernel: one box per tile, 14 output columns,
L / R accumulators exchanged with warp shuffles) and the entry points around them can go wrong.

CPU part (-m "not gpu"): the host weight packing for every channel count the ABI accepts, the schedule rdvc_mcn_conv
picks for each packed mask, and the shape generators of the GPU part.
GPU part (-m gpu): rdvc_mcn_conv on every width 1..66 and on tile counts around multiples of the SM count,
schedule pairs that must agree bit for bit, rdvc_mcn_conv_out directly, the module contract (block counts, batch,
dtypes, layouts, streams, CUDA graphs, re-packing), guard bands and NaN-filled workspaces of rdvc_mcn_forward, and
full-size frames.

References are fp64 evaluations of the same fp16-rounded operands: oracle/mcn.py, or torch's fp64 conv2d on the CPU
(pinned to oracle.mcn.conv2d_same by a CPU test), except the full-size check, which uses cuDNN fp32 as test_mcn.py does.
Tolerances (absolute unless stated; frames and refinement maps live in [0, 1]):
  * packed weights evaluated as the kernels walk them vs conv2d_same .. 1e-9 x max|ref|  (fp64 sums in another order)
  * one layer vs the fp16-rounding reference ..... TOL_LAYER_REL = 4e-3 x max|ref| (test_mcn.py)   observed 7.8e-4
  * output layer vs fp64 warped * sigmoid(conv + b) from the fp16 operands ........... 5e-6  observed 6.4e-7
      (fp32 accumulation of <= 800 products and __expf; the first estimate, 2e-5, was 30x the observed error)
  * network vs om.mcn_forward(emulate_fp16=True) .. TOL_NET_SAME_ROUNDING = 1e-3 (test_mcn.py)    observed 1.8e-4
  * full-size network vs cuDNN fp32 with TF32 off ... TOL_NET_FP32 = 3e-3 (test_mcn.py)           observed 5.1e-4
  (observed: largest over every case of this file on one B200)
  * schedule pairs, batch invariance, input forms, streams, graphs, NaN workspaces ........ bit for bit
"""
import ctypes
import functools

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import rdvc_corr_b200 as rc
from oracle import mcn as om
from rdvc_corr_b200 import _cabi
from rdvc_corr_b200 import mcn as hm
from test_mcn import TOL_LAYER_REL, TOL_NET_FP32, TOL_NET_SAME_ROUNDING

TOL_PACK_REL = 1e-9
TOL_OUT = 5e-6
CANARY, GUARD = 0xAB, 4096
OPT_MCN_KERNEL = 14                                       # rdvc_corr_set_option key: 0 auto, 1 three boxes, 2 one box
KERNELS = {"auto": 0, "three_boxes": 1, "one_box": 2}
TILE_COLS = {"three_boxes": 16, "one_box": 14}            # output super-pixels per tile row (MCN_TX, MCNX_TXO)
TILE_ROWS = 8                                             # MCN_TY
B200_SMS = 148

# restated from csrc/mcn_conv_sm100.cuh: the compile-time MMA schedules and the run-time masks they cover
K_FULL, K_3X3, K_C16 = 0, 1, 2


def kstep_on(kpat, dsx_idx, k):
    """mcn_kstep_on: does schedule `kpat` issue k-step `k` (16 columns) of a tap in column offset `dsx_idx` (0..2)?"""
    if kpat == K_FULL:
        return True
    if kpat == K_3X3:
        return k >= 2 if dsx_idx == 0 else (True if dsx_idx == 1 else k < 2)
    return k in (0, 2)


def pattern_mask(kpat, ksize):
    """mcn_pattern_mask: bit 4 t + k, t = dy_idx * 3 + dsx_idx."""
    return sum(1 << (4 * (dy * 3 + dsx) + k) for dy in range(ksize) for dsx in range(3) for k in range(4)
               if kstep_on(kpat, dsx, k))


def schedule_for(kmask, ksize):
    """The schedule rdvc_mcn_conv instantiates for a mask: the reduced one if it covers every set bit, else FULL."""
    reduced = K_3X3 if ksize == 3 else K_C16
    return reduced if kmask & ~pattern_mask(reduced, ksize) == 0 else K_FULL


# ------------------------------------------------------------------ references and shapes
def f16(x):
    """Round to fp16 and back (numpy: one rounding from any float type)."""
    return np.asarray(x).astype(np.float16).astype(np.float64)


def conv64(x, w):
    """oracle.mcn.conv2d_same restated with torch's fp64 conv2d (the numpy version is too slow for the sweeps)."""
    x, w = torch.as_tensor(np.asarray(x, np.float64)), torch.as_tensor(np.asarray(w, np.float64))
    return F.conv2d(x, w, padding=w.shape[-1] // 2).numpy()


def ref_layer(x, w, b, act, res=None):
    """om.conv_layer(x, w, b, act, res, emulate_fp16=True) with conv64."""
    y = conv64(f16(x), f16(w)) + np.asarray(b, np.float64)[None, :, None, None]
    if res is not None:
        y = y + f16(res)
    if act:
        y = np.where(y > 0, y, om.LEAKY_SLOPE * y)
    return f16(y)


def ref_out_layer(x, w, b, warped):
    """What rdvc_mcn_conv_out computes, in fp64: warped * sigmoid(conv5x5(x) + b) with fp16 x and w, fp32 warped."""
    z = conv64(f16(x), f16(w)) + np.asarray(b, np.float64)[None, :, None, None]
    return np.asarray(warped, np.float64) / (1.0 + np.exp(-z))


H_CYCLE = (1, 2, 7, 8, 9, 15, 16, 17)
B3_WIDTHS = (2, 29, 33, 58, 66)     # Wsp = 1, 15, 17, 29, 33: a last tile with one column for both tile widths


def sweep_shapes():
    """Every W in 1..66 (Wsp 1..33: every residue mod 16 and mod 14, both parities of W), H cycling through
    H_CYCLE (a partial last tile row of 1, 2, 7 rows, exact multiples of 8, one row past them), B = 3 on B3_WIDTHS."""
    return [(3 if W in B3_WIDTHS else 1, H_CYCLE[(W - 1) % len(H_CYCLE)], W) for W in range(1, 67)]


def n_tiles(B, H, W, kernel):
    return B * -(-H // TILE_ROWS) * -(-((W + 1) // 2) // TILE_COLS[kernel])


def shape_with_tiles(target, kernel, i):
    """(B, H, W) whose tiling by `kernel` has exactly `target` tiles; the last tile row and column are ragged (the
    amounts vary with i), and the tiles are split over 1..3 images and 1..2 tile columns."""
    tc = TILE_COLS[kernel]
    ntx = 2 if target % 2 == 0 else 1
    m = target // ntx
    B = 3 if m % 3 == 0 else (2 if m % 2 == 0 else 1)
    nty = m // B
    H = TILE_ROWS * (nty - 1) + 1 + (3 * i) % TILE_ROWS
    Wsp = tc * (ntx - 1) + 1 + (5 * i) % tc
    W = 2 * Wsp - (i & 1)
    return B, H, W


def persistent_cases(sms):
    """Tile counts k * SMs + r, r in {0, 1, SMs - 1}: every CTA walks k or k + 1 tiles, so the last tile of a CTA
    ends on every accumulator (tile index mod 4, or mod 2 for the one-box 5x5 32 -> 32) and both epilogue parities,
    and k = 5 wraps the accumulator phase."""
    return [(k, r) for r in (0, 1, sms - 1) for k in (1, 2, 3, 5)]


def rand16(gen, *shape, scale=1.0):
    """fp32 tensor of fp16-representable values."""
    return (torch.randn(*shape, generator=gen) * scale).half().float()


def layer_case(seed, B, H, W, k, cin, with_res):
    g = torch.Generator().manual_seed(seed)
    x = rand16(g, B, cin, H, W)
    w = (torch.randn(32, cin, k, k, generator=g) / np.sqrt(cin * k * k)).float()
    b = (torch.randn(32, generator=g) * 0.3).float()
    res = rand16(g, B, 32, H, W) if with_res else None
    return x, w, b, res


def plane_proper_bytes(B, H, W):
    return B * H * ((W + 1) // 2) * 128


def guarded(nbytes, fill=CANARY):
    """A device buffer of `nbytes` between two GUARD-byte canary bands; the body starts GUARD (256-aligned) in."""
    buf = torch.full((nbytes + 2 * GUARD,), CANARY, dtype=torch.uint8, device="cuda")
    buf[GUARD:GUARD + nbytes] = fill
    return buf


def guards_intact(buf):
    return bool((buf[:GUARD] == CANARY).all()) and bool((buf[-GUARD:] == CANARY).all())


def run_conv(plane, packed_dev, kmask, bias, k, act, B, H, W, residual=None):
    """rdvc_mcn_conv into a canary-guarded output plane; returns the guarded buffer (plane at offset GUARD)."""
    lib = _cabi.load()
    nbytes = lib.rdvc_mcn_plane_bytes(B, H, W)
    out = guarded(nbytes)
    b = np.ascontiguousarray(np.asarray(bias, np.float32))
    _cabi.check(lib.rdvc_mcn_conv(plane.data_ptr(), packed_dev.data_ptr(), kmask, b.ctypes.data, k, act,
                                  None if residual is None else residual.data_ptr(), out.data_ptr() + GUARD, B, H, W,
                                  torch.cuda.current_stream().cuda_stream), "rdvc_mcn_conv")
    return out


def assert_within(got, want, tol, what, rel=False):
    """max|got - want| <= tol (x max|want| if rel); returns the error (relative if rel)."""
    if isinstance(got, torch.Tensor):
        err, scale = float((got - want).abs().max()), float(want.abs().max())
    else:
        err, scale = float(np.abs(got - want).max()), float(np.abs(want).max())
    if rel:
        err /= scale
    assert err <= tol, (what, err, tol)
    return err


def check_layer_out(out, want, B, H, W, what):
    """Values against the reference, the odd-width padding pixel exactly 0, and nothing written outside the plane
    proper (guard bands and the tail up to the plane's 1 KB rounding keep the canary)."""
    torch.cuda.synchronize()
    proper = plane_proper_bytes(B, H, W)
    body = out[GUARD:-GUARD]
    assert_within(hm.plane_to_nchw(body, B, H, W).cpu().numpy(), want, TOL_LAYER_REL, what, rel=True)
    if W % 2:
        full = body[:proper].view(torch.float16).reshape(B, H, W + 1, 32)
        assert float(full[:, :, W].abs().max()) == 0.0, (what, "padding pixel")
    assert guards_intact(out) and bool((body[proper:] == CANARY).all()), (what, "written outside the plane")


@pytest.fixture
def mcn_kernel():
    """Sets option 14 (which MCN convolution kernel runs); option 14 is back at 0 (auto) after the test, pass or fail."""
    lib = _cabi.load()

    def use(name):
        assert lib.rdvc_corr_set_option(OPT_MCN_KERNEL, KERNELS[name]) == 0

    yield use
    lib.rdvc_corr_set_option(OPT_MCN_KERNEL, 0)


# ------------------------------------------------------------------ CPU
@functools.lru_cache(maxsize=None)
def packed_case(cout, cin, k):
    rng = np.random.default_rng(1000 * cout + 10 * cin + k)
    w = (rng.standard_normal((cout, cin, k, k)) * 0.1).astype(np.float32)
    packed_u8, mask = hm.pack_conv_weights(torch.from_numpy(w))
    return w, packed_u8.numpy().view(np.float16), mask


PACK_CASES = [(cout, cin, k) for k in (3, 5) for cout in (1, 2, 3, 4, 5, 6, 7, 8, 32) for cin in range(1, 33)]


@pytest.mark.parametrize("k", [3, 5])
def test_packing_reproduces_the_convolution_for_every_channel_count(k):
    """rdvc_mcn_pack_weights for every cin in 1..32, cout in 1..8 (the 16-row output-layer layout) and 32: the packed
    tap matrices, evaluated the way each kernel walks them, are conv2d_same of the fp16-rounded weights.  Channels of the
    activation at or beyond cin hold noise, so a weight packed into one of their columns shows."""
    rng = np.random.default_rng(k)
    x = rng.standard_normal((1, 32, 6, 10)).astype(np.float16).astype(np.float32)
    for cout, cin, kk in PACK_CASES:
        if kk != k:
            continue
        w, packed, mask = packed_case(cout, cin, k)
        nout = 64 if cout > 8 else 16
        assert packed.size == 3 * k * nout * 64, (cout, cin)
        want = om.conv2d_same(x[:, :cin], f16(w))
        scale = TOL_PACK_REL * max(1.0, np.abs(want).max())
        for walk in (om.superpixel_gemm_conv, om.superpixel_gemm_conv_xhalo):
            got = walk(x, packed, k, nout, mask)
            assert np.abs(got[:, :cout] - want).max() <= scale, (walk.__name__, cout, cin)
            assert not got[:, cout:].any(), (walk.__name__, cout, cin, "rows beyond cout")
        # the mask: exactly the k-steps with a non-zero weight (16-channel groups within cin, |dx| <= R)
        groups = (cin + 15) // 16
        for t in range(3 * k):
            dsx = t % 3 - 1
            expect = 0
            for p in range(2):
                if any(abs(2 * dsx + p - q) <= k // 2 for q in range(2)):
                    expect |= ((1 << groups) - 1) << (2 * p)
            assert (mask >> (4 * t)) & 15 == expect, (cout, cin, t)


def test_schedule_choice_covers_every_nonzero_kstep():
    """Which compile-time schedule rdvc_mcn_conv runs for each packed mask: MCN_K_3X3 for every 3x3 and MCN_K_C16
    exactly when cin <= 16 for 5x5; and every k-step that holds a non-zero weight is one the schedule issues.  (The
    output layer, rdvc_mcn_conv_out, always runs MCN_K_FULL.)  A packing change that moves a layer to FULL, or a mask
    that drops a non-zero step, fails here; the GPU tests below then know which instantiation they run."""
    assert pattern_mask(K_FULL, 3) == (1 << 36) - 1 and pattern_mask(K_FULL, 5) == (1 << 60) - 1
    assert bin(pattern_mask(K_3X3, 3)).count("1") == 24 and bin(pattern_mask(K_C16, 5)).count("1") == 30
    for cout, cin, k in PACK_CASES:
        _, packed, mask = packed_case(cout, cin, k)
        nout = 64 if cout > 8 else 16
        steps = packed.reshape(3 * k, nout, 4, 16).astype(np.float32)
        nonzero = sum(1 << (4 * t + s) for t in range(3 * k) for s in range(4) if steps[t, :, s].any())
        assert mask == nonzero, (cout, cin, k)
        kpat = schedule_for(mask, k)
        assert kpat == (K_3X3 if k == 3 else (K_C16 if cin <= 16 else K_FULL)), (cout, cin, k, kpat)
        assert nonzero & ~pattern_mask(kpat, k) == 0, (cout, cin, k)
        for t in range(3 * k):                                   # the same, step by step through mcn_kstep_on
            for s in range(4):
                if steps[t, :, s].any():
                    assert kstep_on(kpat, t % 3, s), (cout, cin, k, t, s)


def test_torch_reference_restates_the_oracle():
    rng = np.random.default_rng(2)
    for (B, ci, co, H, W, k) in [(2, 32, 32, 5, 7, 3), (1, 8, 32, 9, 4, 5), (3, 32, 3, 1, 1, 5), (1, 32, 32, 2, 17, 3)]:
        x = rng.standard_normal((B, ci, H, W))
        w = rng.standard_normal((co, ci, k, k))
        want = om.conv2d_same(x, w)
        assert np.abs(conv64(x, w) - want).max() <= 1e-12 * np.abs(want).max()
        b = rng.standard_normal(co)
        res = rng.standard_normal((B, co, H, W))
        for act in (False, True):
            assert np.array_equal(ref_layer(x, w, b, act, res), om.conv_layer(x, w, b, act, res, emulate_fp16=True))


def test_sweep_covers_every_tile_residue():
    shapes = sweep_shapes()
    for tc in TILE_COLS.values():
        residues = {(((W + 1) // 2) % tc, W % 2) for _, _, W in shapes}
        assert residues == {(r, p) for r in range(tc) for p in (0, 1)}
        assert any(B == 3 and (W + 1) // 2 % tc == 1 and (W + 1) // 2 > 1 for B, _, W in shapes)
    assert {H % TILE_ROWS for _, H, _ in shapes} == {0, 1, 2, 7}
    assert {(H, W) for _, H, W in shapes} >= {(1, 1), (2, 2)}


@pytest.mark.parametrize("sms", [B200_SMS, 132, 7])
def test_persistent_shapes_hit_their_tile_counts(sms):
    for kernel in TILE_COLS:
        for i, (k, r) in enumerate(persistent_cases(sms)):
            B, H, W = shape_with_tiles(k * sms + r, kernel, i)
            assert n_tiles(B, H, W, kernel) == k * sms + r, (kernel, k, r, (B, H, W))
            assert W >= 1 and H >= 1 and B <= 65535


# ------------------------------------------------------------------ GPU: single layers
LAYERS = {               # name: (k, cin, residual)
    "3x3": (3, 32, False),
    "3x3_residual": (3, 32, True),
    "5x5": (5, 32, False),
    "5x5_c16": (5, 8, False),           # the network's first layer: the MCN_K_C16 schedule
}


@functools.lru_cache(maxsize=None)
def sweep_case(layer, B, H, W):
    k, cin, with_res = LAYERS[layer]
    x, w, b, res = layer_case(W * 131 + k * 7 + cin, B, H, W, k, cin, with_res)
    act = W % 3 != 0                    # every third width without the activation (negative values pass through)
    want = ref_layer(x.numpy(), w.numpy(), b.numpy(), act, None if res is None else res.numpy())
    return x, w, b, res, act, want


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["three_boxes", "one_box"])
@pytest.mark.parametrize("layer", list(LAYERS))
def test_layer_on_every_width(mcn_kernel, layer, kernel):
    """Tile decode of the last partial tile in x (every Wsp residue of both tile widths, a last tile with one column,
    W = 1 and 2) and in y (H in 1, 2, 7, 8, 9, 15, 16, 17), B = 3, the odd-width padding pixel, TMA store clipping."""
    mcn_kernel(kernel)
    k = LAYERS[layer][0]
    for B, H, W in sweep_shapes():
        x, w, b, res, act, want = sweep_case(layer, B, H, W)
        packed, mask = hm.pack_conv_weights(w)
        plane = hm.plane_from_nchw(x.cuda())
        rplane = None if res is None else hm.plane_from_nchw(res.cuda())
        out = run_conv(plane, packed.cuda(), mask, b.numpy(), k, hm.ACT_LEAKY if act else hm.ACT_NONE, B, H, W, rplane)
        check_layer_out(out, want, B, H, W, (layer, kernel, B, H, W))


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,layer", [("three_boxes", "3x3_residual"), ("one_box", "3x3_residual"),
                                          ("three_boxes", "5x5"), ("one_box", "5x5")])
def test_persistent_loop_residues(mcn_kernel, kernel, layer):
    """Tile counts k * SMs + r around the persistent grid: which accumulator (4, or 2 for the one-box 5x5 32 -> 32),
    accumulator phase, epilogue parity and residual-barrier phase end each CTA's walk; half the cases walk the tiles in
    reverse order (RDVC_MCN_REVERSE_ORDER)."""
    mcn_kernel(kernel)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    k, cin, with_res = LAYERS[layer]
    for i, (kk, r) in enumerate(persistent_cases(sms)):
        B, H, W = shape_with_tiles(kk * sms + r, kernel, i)
        x, w, b, res = layer_case(1000 + i, B, H, W, k, cin, with_res)
        want = ref_layer(x.numpy(), w.numpy(), b.numpy(), True, None if res is None else res.numpy())
        packed, mask = hm.pack_conv_weights(w)
        plane = hm.plane_from_nchw(x.cuda())
        rplane = None if res is None else hm.plane_from_nchw(res.cuda())
        act = hm.ACT_LEAKY | (hm.REVERSE_ORDER if i % 2 else 0)
        out = run_conv(plane, packed.cuda(), mask, b.numpy(), k, act, B, H, W, rplane)
        check_layer_out(out, want, B, H, W, (kernel, layer, kk, r, (B, H, W)))


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["three_boxes", "one_box"])
@pytest.mark.parametrize("k,cin", [(3, 32), (5, 8), (5, 16)])
def test_reduced_schedule_equals_full_schedule(mcn_kernel, kernel, k, cin):
    """MCN_K_3X3 (3x3) and MCN_K_C16 (5x5, cin <= 16) against MCN_K_FULL, forced by an all-ones k-step mask, on the
    same weights: the extra k-steps multiply exact zeros into fp32 accumulators, so the planes are equal bit for bit."""
    mcn_kernel(kernel)
    full_mask = (1 << (4 * 3 * k)) - 1
    for (B, H, W) in [(2, 19, 45), (1, 40, 93), (3, 8, 30)]:
        x, w, b, res = layer_case(7 * W + k, B, H, W, k, cin, with_res=(k == 3))
        packed, mask = hm.pack_conv_weights(w)
        assert schedule_for(mask, k) == (K_3X3 if k == 3 else K_C16) and schedule_for(full_mask, k) == K_FULL
        plane = hm.plane_from_nchw(x.cuda())
        rplane = None if res is None else hm.plane_from_nchw(res.cuda())
        outs = [run_conv(plane, packed.cuda(), m, b.numpy(), k, hm.ACT_LEAKY, B, H, W, rplane) for m in (mask, full_mask)]
        want = ref_layer(x.numpy(), w.numpy(), b.numpy(), True, None if res is None else res.numpy())
        check_layer_out(outs[0], want, B, H, W, (kernel, k, cin, "reduced"))
        proper = plane_proper_bytes(B, H, W)
        assert torch.equal(outs[0][GUARD:GUARD + proper], outs[1][GUARD:GUARD + proper]), (kernel, k, cin, (B, H, W))


# ------------------------------------------------------------------ GPU: the output layer
OUT_WIDTHS = (1, 2, 3, 4, 27, 28, 29, 30, 31, 32, 33, 34, 35, 57, 58, 65, 66)


def run_conv_out(plane, packed_dev, kmask, bias, cout, warped, out_ptr, B, H, W):
    """rdvc_mcn_conv_out: (B, cout, H, W) fp32 = warped * sigmoid(conv5x5(plane) + bias)."""
    lib = _cabi.load()
    b = np.ascontiguousarray(np.asarray(bias, np.float32))
    _cabi.check(lib.rdvc_mcn_conv_out(plane.data_ptr(), packed_dev.data_ptr(), kmask, b.ctypes.data, 5, cout,
                                      warped.data_ptr(), out_ptr, B, H, W, torch.cuda.current_stream().cuda_stream),
                "rdvc_mcn_conv_out")


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["auto", "three_boxes", "one_box"])
@pytest.mark.parametrize("cout", [1, 3, 8])
def test_output_layer(mcn_kernel, kernel, cout):
    """rdvc_mcn_conv_out for every cout the ABI's ends and middle (1, 3, 8), the scalar (odd W) and float2 (even W)
    store paths at every tile residue, B = 1 and 3: element by element against fp64; every byte around (B, cout, H, W)
    keeps its canary, every element is written, and for odd W each row's first pixel holds its own value (not the
    previous row's padding pixel)."""
    mcn_kernel(kernel)
    g = torch.Generator().manual_seed(cout)
    w = (torch.randn(cout, 32, 5, 5, generator=g) / np.sqrt(800)).float()
    bias = (torch.randn(cout, generator=g) * 0.5).float()
    packed, mask = hm.pack_conv_weights(w)
    packed = packed.cuda()
    for i, W in enumerate(OUT_WIDTHS):
        B, H = (3 if i % 2 else 1), H_CYCLE[(W - 1) % len(H_CYCLE)]
        x = rand16(g, B, 32, H, W)
        warped = torch.rand(B, cout, H, W, generator=g)
        want = ref_out_layer(x.numpy(), w.numpy(), bias.numpy(), warped.numpy())
        n = B * cout * H * W
        out = guarded(4 * n)
        run_conv_out(hm.plane_from_nchw(x.cuda()), packed, mask, bias.numpy(), cout, warped.cuda(),
                     out.data_ptr() + GUARD, B, H, W)
        torch.cuda.synchronize()
        what = (kernel, cout, (B, H, W))
        assert guards_intact(out), (what, "guard band")
        got = out[GUARD:GUARD + 4 * n].view(torch.float32).reshape(B, cout, H, W).cpu().numpy()
        assert (got >= 0).all(), (what, "an element was not written (the canary is negative)")
        assert_within(got, want, TOL_OUT, what)
        if W % 2:
            assert_within(got[..., 0], want[..., 0], TOL_OUT, (what, "first pixel of a row"))


# ------------------------------------------------------------------ GPU: the module
def seeded_net(num_res_blocks=3, seed=0):
    """A network with seeded weights and non-trivial BatchNorm statistics and affine parameters (as bench_gop.py)."""
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(seed)
        net = rc.MotionCompensationNetwork(num_res_blocks=num_res_blocks)
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.3)
                m.running_var.copy_(torch.rand(m.num_features, generator=g) * 1.5 + 0.25)
                m.weight.copy_(torch.rand(m.num_features, generator=g) + 0.5)
                m.bias.copy_(torch.randn(m.num_features, generator=g) * 0.1)
    return net.eval().cuda()


def frames(B, H, W, seed, device="cuda"):
    g = torch.Generator().manual_seed(seed)
    a, r = torch.rand(B, 3, H, W, generator=g), torch.rand(B, 3, H, W, generator=g)
    f = torch.randn(B, 2, H, W, generator=g) * 4
    return a.to(device), f.to(device), r.to(device)


def oracle(net, a, f, r):
    params = {k: v.detach().cpu().numpy() for k, v in net.state_dict().items()}
    return om.mcn_forward(params, *(t.cpu().numpy() for t in (a, f, r)), num_res_blocks=net.num_res_blocks,
                          emulate_fp16=True)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 2, 5])
def test_other_block_counts(n):
    """num_res_blocks != 3 (the constructor and rdvc_mcn_forward take 0..64): the layer indexing of rdvc_mcn_forward,
    the ping-pong of its workspace planes, and one launch per layer plus the input pack (3 + 2 n)."""
    net = seeded_net(n, seed=n)
    a, f, r = frames(2, 19, 37, seed=n)
    lib = _cabi.load()
    with torch.no_grad():
        net(a, f, r)                                 # packs the weights
        n0 = lib.rdvc_corr_launch_count()
        out = net(a, f, r)
        assert lib.rdvc_corr_launch_count() - n0 == 3 + 2 * n
    torch.cuda.synchronize()
    assert_within(out.cpu().numpy(), oracle(net, a, f, r), TOL_NET_SAME_ROUNDING, n)


@pytest.mark.gpu
def test_batch_invariance(mcn_kernel):
    """Every image of a batch gets the same bits as when it runs alone, under each kernel choice."""
    net = seeded_net()
    a, f, r = frames(3, 21, 45, seed=4)
    with torch.no_grad():
        for kernel in KERNELS:
            mcn_kernel(kernel)
            out = net(a, f, r)
            for i in range(3):
                assert torch.equal(out[i:i + 1], net(a[i:i + 1], f[i:i + 1], r[i:i + 1])), (kernel, i)


@pytest.mark.gpu
def test_input_forms():
    """fp16 / bf16 inputs return that dtype and equal the fp32 run on the same rounded values; channels_last and
    sliced (non-contiguous) inputs equal the contiguous run bit for bit."""
    net = seeded_net()
    a, f, r = frames(2, 23, 41, seed=5)
    with torch.no_grad():
        base = net(a, f, r)
        for dt in (torch.float16, torch.bfloat16):
            args = [t.to(dt) for t in (a, f, r)]
            out = net(*args)
            assert out.dtype == dt
            assert torch.equal(out, net(*(t.float() for t in args)).to(dt)), dt
        cl = [t.contiguous(memory_format=torch.channels_last) for t in (a, f, r)]
        assert not cl[0].is_contiguous()
        assert torch.equal(net(*cl), base)
        big = [torch.zeros(2, t.shape[1] + 1, 23 + 3, 41 + 5, device="cuda") for t in (a, f, r)]
        sl = []
        for t, bg in zip((a, f, r), big):
            bg[:, 1:, 1:24, 2:43] = t
            sl.append(bg[:, 1:, 1:24, 2:43])
        assert not sl[0].is_contiguous()
        assert torch.equal(net(*sl), base)


@pytest.mark.gpu
def test_side_stream_and_cuda_graph():
    """forward on a side stream, captured in a CUDA graph and replayed, and replayed after new inputs are copied into
    the static tensors: all equal to eager runs on the default stream."""
    net = seeded_net()
    a, f, r = frames(2, 27, 53, seed=6)
    a2, f2, r2 = frames(2, 27, 53, seed=7)
    with torch.no_grad():
        base, base2 = net(a, f, r), net(a2, f2, r2)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            side = net(a, f, r)
            for _ in range(2):                       # warm-up on the capture stream
                net(a, f, r)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        assert torch.equal(side, base)
        sa, sf, sr = a.clone(), f.clone(), r.clone()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            sout = net(sa, sf, sr)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(sout, base)
        for static, new in ((sa, a2), (sf, f2), (sr, r2)):
            static.copy_(new)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(sout, base2)


@pytest.mark.gpu
def test_load_state_dict_repacks():
    """The folded, packed weights are rebuilt when a BatchNorm buffer changes: a load_state_dict that changes only
    running_var changes the output, and the new output matches the oracle with the new statistics."""
    net = seeded_net()
    a, f, r = frames(2, 17, 31, seed=8)
    with torch.no_grad():
        before = net(a, f, r)
        sd = net.state_dict()
        g = torch.Generator().manual_seed(9)
        changed = {k: (v.cpu() * (torch.rand(v.shape, generator=g) * 3 + 0.5)) if k.endswith("running_var") else v
                   for k, v in sd.items()}
        net.load_state_dict(changed)
        after = net(a, f, r)
    torch.cuda.synchronize()
    assert_within(after.cpu().numpy(), oracle(net, a, f, r), TOL_NET_SAME_ROUNDING, "new statistics")
    assert float((after - before).abs().max()) > 10 * TOL_NET_SAME_ROUNDING


# ------------------------------------------------------------------ GPU: rdvc_mcn_forward's memory
def packed_network(net):
    """What MotionCompensationNetwork._prepare hands rdvc_mcn_forward, built from the public helpers."""
    dev_w, masks = [], []
    layers = net.folded_layers()
    biases = np.zeros((len(layers), 32), np.float32)
    for i, (w, b) in enumerate(layers):
        packed, mask = hm.pack_conv_weights(w)
        dev_w.append(packed.cuda())
        masks.append(mask)
        biases[i, :b.numel()] = b.numpy()
    return (dev_w, (ctypes.c_void_p * len(dev_w))(*[t.data_ptr() for t in dev_w]),
            (ctypes.c_ulonglong * len(masks))(*masks), biases)


@pytest.mark.gpu
def test_forward_guard_bands_and_nan_workspace(mcn_kernel):
    """rdvc_mcn_forward on odd W, H not a multiple of 8, B = 2 and tiny frames, for each kernel choice: with the
    workspace filled with 0xFF (fp16 NaN) the output equals the run on a zeroed workspace (no layer reads a padding
    pixel or plane tail that nobody wrote); 4 KB canary bands around warped, flow, ref, workspace and out survive; the
    inputs are unchanged bit for bit; every output element is written and matches the oracle."""
    net = seeded_net()
    dev_w, ptrs, masks, biases = packed_network(net)      # dev_w keeps the device weights that ptrs points to alive
    lib = _cabi.load()
    st = torch.cuda.current_stream().cuda_stream
    for (B, H, W) in [(1, 1, 1), (1, 2, 3), (2, 5, 7), (1, 9, 17), (2, 13, 29), (1, 3, 30), (2, 17, 33)]:
        a, f, r = frames(B, H, W, seed=W)
        want = oracle(net, a, f, r)
        ins = {}
        for name, t in (("warped", a), ("flow", f), ("ref", r)):
            buf = guarded(4 * t.numel())
            buf[GUARD:GUARD + 4 * t.numel()] = t.reshape(-1).view(torch.uint8)
            ins[name] = (buf, buf.clone())
        wsb = lib.rdvc_mcn_workspace_bytes(B, H, W)
        for kernel in KERNELS:
            mcn_kernel(kernel)
            outs = []
            for fill in (0x00, 0xFF):
                ws, out = guarded(wsb, fill), guarded(4 * B * 3 * H * W)
                _cabi.check(lib.rdvc_mcn_forward(*(ins[k][0].data_ptr() + GUARD for k in ("warped", "flow", "ref")),
                                                 B, H, W, 3, ptrs, masks, biases.ctypes.data, ws.data_ptr() + GUARD, wsb,
                                                 out.data_ptr() + GUARD, st), "rdvc_mcn_forward")
                torch.cuda.synchronize()
                what = (kernel, (B, H, W), hex(fill))
                assert guards_intact(ws) and guards_intact(out), (what, "guard band")
                for name, (buf, orig) in ins.items():
                    assert torch.equal(buf, orig), (what, name, "input or its guard band changed")
                outs.append(out[GUARD:-GUARD].view(torch.float32).reshape(B, 3, H, W))
            assert torch.equal(outs[0], outs[1]), (kernel, (B, H, W), "NaN workspace")
            got = outs[0].cpu().numpy()
            assert (got >= 0).all(), (kernel, (B, H, W), "an element was not written")
            assert_within(got, want, TOL_NET_SAME_ROUNDING, (kernel, (B, H, W)))


# ------------------------------------------------------------------ GPU: full size
def torch_folded(net, a, f, r):
    """The same folded network through cuDNN in fp32 with TF32 off (as test_mcn.py's full-size test)."""
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        layers = [(w.cuda(), b.cuda()) for w, b in net.folded_layers()]
        x = F.leaky_relu(F.conv2d(torch.cat([a, f, r], 1), *layers[0], padding=2), 0.2)
        for i in range(net.num_res_blocks):
            t = F.leaky_relu(F.conv2d(x, *layers[1 + 2 * i], padding=1), 0.2)
            x = F.leaky_relu(F.conv2d(t, *layers[2 + 2 * i], padding=1) + x, 0.2)
        return a * torch.sigmoid(F.conv2d(x, *layers[-1], padding=2))
    finally:
        torch.backends.cudnn.allow_tf32 = old


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,W", [(2, 1080, 1920), (1, 2160, 3840)])
def test_full_size(mcn_kernel, B, H, W):
    """1080p with B = 2 (each image also equal to its B = 1 run) and 4K with B = 1, under each kernel choice."""
    net = seeded_net()
    g = torch.Generator(device="cuda").manual_seed(B)
    a = torch.rand(B, 3, H, W, device="cuda", generator=g)
    r = torch.rand(B, 3, H, W, device="cuda", generator=g)
    f = torch.randn(B, 2, H, W, device="cuda", generator=g) * 4
    with torch.no_grad():
        want = torch_folded(net, a, f, r)
        for kernel in KERNELS:
            mcn_kernel(kernel)
            got = net(a, f, r)
            assert_within(got, want, TOL_NET_FP32, kernel)
            if B > 1:
                for i in range(B):
                    assert torch.equal(got[i:i + 1], net(a[i:i + 1], f[i:i + 1], r[i:i + 1])), (kernel, i)
