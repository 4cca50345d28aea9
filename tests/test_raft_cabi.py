"""The whole RAFT call through the C ABI: rdvc_corr_raft_pack_weights, rdvc_corr_raft_workspace_bytes, rdvc_corr_raft_flow,
rdvc_corr_raft_flow_sequence (include/rdvc_corr.h), rdvc_corr_pack_nhwc and examples/raft_flow.c.

Without a GPU: the packed blob against the per-module pack functions called directly, key-order independence, the
refused state dicts, workspace arithmetic, every argument refusal, and the example compiling against the header.
On the GPU: bit identity with rc.raft_flow / rc.raft_flow_sequence with all six drop-ins (act fp32 / fp16 autocast,
volume fp32 / bf16, 368x640 golden frames and 1088x1920, B = 1 and 3), EPE against stock RAFT, batch and sequence
identities, CUDA-graph capture, NaN-filled workspaces, canaries, the example's output and the launch count.
"""
import ctypes
import os
import random
import struct
import subprocess

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import rdvc_corr_b200 as rc
from rdvc_corr_b200 import _cabi
from rdvc_corr_b200.context_encoder import PackedContextEncoder, _convs_and_norms
from rdvc_corr_b200.corr_block import PackedConv1x1, PackedLinear
from rdvc_corr_b200.feature_encoder import PackedFeatureEncoder
from rdvc_corr_b200.mask_predictor import PackedMaskConv
from rdvc_corr_b200.motion_encoder import PackedUpdateConv
from rdvc_corr_b200.recurrent_block import PackedConvGRU

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32, F16, BF16 = _cabi.RDVC_DT_F32, _cabi.RDVC_DT_F16, _cabi.RDVC_DT_BF16
E_NULL, E_SHAPE, E_TOO_SMALL, E_DTYPE, E_UNSUPPORTED, E_WORKSPACE, E_ALIGN = -1, -2, -3, -4, -5, -6, -7
TOL_EPE = 0.05
SECTIONS = _cabi.RDVC_RAFT_SECTIONS


@pytest.fixture(scope="module")
def lib():
    rc._build.build()
    return _cabi.load()


def seeded_state(small=False):
    from torchvision.models.optical_flow import raft_large, raft_small
    torch.manual_seed(0)
    model = (raft_small if small else raft_large)(weights=None)
    g = torch.Generator().manual_seed(77)
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.Conv2d) and m.bias is not None:
                m.bias.copy_(0.3 * torch.randn(m.out_channels, generator=g))
            if isinstance(m, torch.nn.BatchNorm2d):
                c = m.num_features
                m.running_mean.copy_(0.5 * torch.randn(c, generator=g))
                m.running_var.copy_(0.5 + 1.5 * torch.rand(c, generator=g))
                m.weight.copy_(0.5 + torch.rand(c, generator=g))
                m.bias.copy_(0.3 * torch.randn(c, generator=g))
    return model.eval()


def pack(lib, sd, op=F16):
    """rdvc_corr_raft_pack_weights on (name, tensor) pairs in the given order -> (rc, blob as uint8 numpy)."""
    items = list(sd.items())
    arrs = [np.ascontiguousarray(v.detach().to(torch.float32).cpu().numpy()) for _, v in items]
    shapes = [(ctypes.c_longlong * max(a.ndim, 1))(*a.shape) for a in arrs]
    n = len(items)
    nbytes = lib.rdvc_corr_raft_packed_weight_bytes(op) or 1
    blob = np.zeros(nbytes, np.uint8)
    code = lib.rdvc_corr_raft_pack_weights((ctypes.c_char_p * n)(*[k.encode() for k, _ in items]),
                                           (ctypes.c_void_p * n)(*[a.ctypes.data for a in arrs]),
                                           (ctypes.c_int * n)(*[a.ndim for a in arrs]),
                                           (ctypes.c_void_p * n)(*[ctypes.addressof(s) for s in shapes]), n, op,
                                           blob.ctypes.data, blob.nbytes)
    return code, blob


def expected_blob(model):
    """The blob rebuilt from the per-module pack functions, called directly, behind the documented header."""
    cpu, h16 = "cpu", torch.float16
    fe, ce, ub, mp = model.feature_encoder, model.context_encoder, model.update_block, model.mask_predictor
    me = ub.motion_encoder
    b32 = lambda t: t.detach().to(torch.float32).numpy().tobytes()                       # noqa: E731
    pfe = PackedFeatureEncoder([c for c, _ in _convs_and_norms(fe)], h16, cpu, None)
    pce = PackedContextEncoder(_convs_and_norms(ce), h16, cpu, None)
    tail = PackedLinear(fe.conv.weight, fe.conv.bias, h16, cpu)
    cc1 = PackedConv1x1(me.convcorr1[0].weight, me.convcorr1[0].bias, 4, 4, h16, cpu)
    mes = [PackedUpdateConv(m[0], i, h16, cpu) for i, m in enumerate((me.convcorr2, me.convflow1, me.convflow2, me.conv))]
    fhs = [PackedUpdateConv(c, 4 + i, h16, cpu) for i, c in enumerate((ub.flow_head.conv1, ub.flow_head.conv2))]
    grus = [PackedConvGRU(g, h16, cpu) for g in (ub.recurrent_block.convgru1, ub.recurrent_block.convgru2)]
    mrelu, mconv = PackedUpdateConv(mp.convrelu[0], 4, h16, cpu), PackedMaskConv(mp.conv, h16, cpu)
    raw = lambda p: p.weight.numpy().tobytes()                                          # noqa: E731
    secs = [raw(pfe), b32(pfe.bias), raw(pce), b32(pce.bias), raw(tail), b32(tail.bias), raw(cc1), b32(cc1.bias)]
    secs += [raw(p) for p in mes] + [b32(p.bias) for p in mes] + [raw(p) for p in fhs] + [b32(p.bias) for p in fhs]
    secs += [raw(p) for p in grus] + [b32(b) for p in grus for b in (p.bias_z, p.bias_r, p.bias_q)]
    secs += [raw(mrelu), raw(mconv), b32(mrelu.bias), b32(mconv.bias)]
    assert len(secs) == SECTIONS
    a256 = lambda x: (x + 255) // 256 * 256                                             # noqa: E731
    offs, o = [], a256(16 + 16 * SECTIONS)
    for s in secs:
        offs.append(o)
        o = a256(o + len(s))
    blob = bytearray(o)
    blob[:16 + 16 * SECTIONS] = struct.pack(f"<IIii{SECTIONS}Q{SECTIONS}Q", 0x54464152, 1, F16, SECTIONS, *offs,
                                            *[len(s) for s in secs])
    for off, s in zip(offs, secs):
        blob[off:off + len(s)] = s
    return np.frombuffer(bytes(blob), np.uint8)


# ------------------------------------------------------------------ packing (no GPU)
def test_pack_is_the_module_packs_concatenated(lib):
    model = seeded_state()
    code, blob = pack(lib, model.state_dict())
    assert code == 0, _cabi.last_error()
    exp = expected_blob(model)
    assert blob.size == exp.size and np.array_equal(blob, exp)


def test_pack_ignores_key_order(lib):
    sd = seeded_state().state_dict()
    items = list(sd.items())
    random.Random(5).shuffle(items)
    a, b = pack(lib, sd), pack(lib, dict(items))
    assert a[0] == 0 and b[0] == 0 and np.array_equal(a[1], b[1])


def test_pack_refusals_name_the_key(lib):
    sd = seeded_state().state_dict()
    missing = dict(sd)
    del missing["update_block.flow_head.conv2.bias"]
    extra = dict(sd, **{"update_block.flow_head.conv3.weight": torch.zeros(2, 2, 3, 3)})
    wrong = dict(sd, **{"mask_predictor.conv.weight": torch.zeros(576, 256, 3, 3)})
    swapped = dict(sd, **{"update_block.recurrent_block.convgru1.convz.weight": torch.zeros(128, 384, 5, 1)})
    for d, code, key in ((missing, E_SHAPE, "update_block.flow_head.conv2.bias"),
                         (extra, E_UNSUPPORTED, "update_block.flow_head.conv3.weight"),
                         (wrong, E_SHAPE, "mask_predictor.conv.weight"),
                         (swapped, E_SHAPE, "update_block.recurrent_block.convgru1.convz.weight")):
        got, _ = pack(lib, d)
        assert got == code and key in _cabi.last_error(), (got, _cabi.last_error())
    got, _ = pack(lib, seeded_state(small=True).state_dict())             # raft_small: bottleneck blocks, no mask
    assert got in (E_SHAPE, E_UNSUPPORTED) and "encoder" in _cabi.last_error(), _cabi.last_error()
    assert lib.rdvc_corr_raft_packed_weight_bytes(BF16) == 0 and pack(lib, sd, BF16)[0] == E_DTYPE


# ------------------------------------------------------------------ sizes and argument errors (no GPU)
def test_workspace_bytes(lib):
    ws = lib.rdvc_corr_raft_workspace_bytes
    for args in ((2, 1, 364, 640, F32, F32), (2, 1, 368, 644, F32, F32), (2, 1, 120, 640, F32, F32),
                 (1, 1, 368, 640, F32, F32), (5, 2, 368, 640, F32, F32), (2, 0, 368, 640, F32, F32),
                 (2, 1, 368, 640, BF16, F32), (2, 1, 368, 640, F32, F16), (2, 1, -8, 640, F32, F32)):
        assert ws(*args) == 0, args
    assert ws(2, 1, 128, 128, F16, BF16) > 0
    for act in (F32, F16):
        for vd in (F32, BF16):
            for B in (1, 3):
                h, w = 1088 // 8, 1920 // 8
                assert ws(2 * B, B, 1088, 1920, act, vd) >= lib.rdvc_corr_pyramid_bytes(B, h, w, 4, vd, rc.RDVC_LAYOUT_TILED)
            sizes = [ws(n + 1, n, 368, 640, act, vd) for n in range(1, 10)] + [ws(2 * n, n, 368, 640, act, vd)
                                                                               for n in range(1, 10)]
            assert all(s > 0 for s in sizes)
            assert all(a <= b for a, b in zip(sizes[:9], sizes[1:9])) and all(a <= b for a, b in zip(sizes[9:], sizes[10:]))
            frames = [(128, 128), (128, 136), (136, 136), (368, 640), (376, 640), (1088, 1920)]
            fs = [ws(4, 3, H, W, act, vd) for H, W in frames]
            assert all(a <= b for a, b in zip(fs, fs[1:])), fs
    assert ws(2, 1, 1088, 1920, F32, F32) > 5.7e9          # the pyramid is the bulk: 5.7 GB per 1080p pair


def test_argument_errors(lib):
    """Every refusal of rdvc_corr_raft_flow / _sequence returns its code before anything touches the device (the pointers
    below are never dereferenced)."""
    H, W, B = 368, 640, 1
    need = lib.rdvc_corr_raft_workspace_bytes(2 * B, B, H, W, F32, F32)
    im1, im2, ws, out, wt = 1 << 40, 2 << 40, 3 << 40, 4 << 40, 5 << 40
    s = (ctypes.c_longlong * 4)(3 * H * W, H * W, W, 1)
    base = dict(image1=im1, image2=im2, strides=s, in_dtype=F32, B=B, H=H, W=W, iters=12, act=F32, vol=F32, w=wt,
                ws=ws, ws_bytes=need, out=out)

    def call(**kw):
        a = dict(base, **kw)
        return lib.rdvc_corr_raft_flow(a["image1"], a["image2"], a["strides"], a["in_dtype"], a["B"], a["H"], a["W"],
                                       a["iters"], a["act"], a["vol"], a["w"], 0.25, a["ws"], a["ws_bytes"], a["out"], None)

    cases = [(dict(image2=None), E_NULL), (dict(w=None), E_NULL), (dict(ws=None), E_NULL), (dict(out=None), E_NULL),
             (dict(H=372), E_SHAPE), (dict(W=644), E_SHAPE), (dict(B=0), E_SHAPE), (dict(iters=0), E_SHAPE),
             (dict(H=120), E_TOO_SMALL), (dict(W=120), E_TOO_SMALL),
             (dict(in_dtype=7), E_DTYPE), (dict(act=BF16), E_DTYPE), (dict(vol=F16), E_DTYPE),
             (dict(ws_bytes=need - 1), E_WORKSPACE),
             (dict(ws=ws + 16), E_ALIGN), (dict(w=wt + 16), E_ALIGN), (dict(out=out + 4), E_ALIGN),
             (dict(image1=im1 + 2), E_ALIGN),
             (dict(strides=(ctypes.c_longlong * 4)(-1, H * W, W, 1)), E_UNSUPPORTED),
             (dict(out=ws + 256), E_UNSUPPORTED), (dict(image2=ws), E_UNSUPPORTED)]
    for kw, code in cases:
        assert call(**kw) == code, (kw, call(**kw), _cabi.last_error())
    fs = lib.rdvc_corr_raft_flow_sequence
    need_s = lib.rdvc_corr_raft_workspace_bytes(3, 2, H, W, F32, F32)
    assert fs(im1, s, F32, 1, H, W, 12, F32, F32, wt, 0.25, ws, need_s, out, None) == E_SHAPE
    assert fs(im1, s, F32, 3, H, W, 0, F32, F32, wt, 0.25, ws, need_s, out, None) == E_SHAPE
    assert fs(im1, s, F32, 3, H, W, 12, F32, F32, wt, 0.25, ws, need_s - 256, out, None) == E_WORKSPACE
    # rdvc_corr_pack_nhwc: 16-bit maps, pixel stride >= D and a multiple of 8, aligned bases
    pk = lib.rdvc_corr_pack_nhwc
    pn = lib.rdvc_corr_workspace_bytes(1, 128, 46, 80)
    assert pk(im1, im2, 128, 1, 128, 46, 80, F32, F32, 1, 4, ws, pn, None) == E_DTYPE
    assert pk(im1, im2, 132, 1, 128, 46, 80, F16, F32, 1, 4, ws, pn, None) == E_ALIGN
    assert pk(im1, im2 + 8, 128, 1, 128, 46, 80, F16, F32, 1, 4, ws, pn, None) == E_ALIGN
    assert pk(im1, im2, 64, 1, 128, 46, 80, F16, F32, 1, 4, ws, pn, None) == E_UNSUPPORTED
    assert pk(im1, im2, 0, 1, 128, 46, 80, F16, F32, 1, 4, ws, pn, None) == E_UNSUPPORTED


def cuda_root():
    return os.path.dirname(os.path.dirname(os.path.realpath(rc._build.nvcc_path())))


def build_example(tmp_path):
    src = os.path.join(ROOT, "examples", "raft_flow.c")
    obj, exe = str(tmp_path / "raft_flow.o"), str(tmp_path / "raft_flow")
    cu = cuda_root()
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-I",
                           os.path.join(cu, "include"), "-c", src, "-o", obj])
    libdir = os.path.dirname(_cabi.lib_path())
    cudalib = next(d for d in (os.path.join(cu, "lib64"), os.path.join(cu, "targets", "x86_64-linux", "lib"))
                   if os.path.isdir(d))
    subprocess.check_call(["gcc", obj, "-o", exe, "-L", libdir, "-lrdvc_corr", "-L", cudalib, "-lcudart", "-lm",
                           "-Wl,-rpath," + libdir, "-Wl,-rpath," + cudalib])
    return exe


def test_example_compiles_against_the_header(lib, tmp_path):
    assert os.path.exists(build_example(tmp_path))


# ------------------------------------------------------------------ on the GPU
_MODELS = {}


def dropin_model(vd):
    """Seeded raft_large with all six drop-ins and a TVCorrBlock of volume dtype vd (cached per vd)."""
    if vd not in _MODELS:
        model = seeded_state()
        vdt = torch.float32 if vd == F32 else torch.bfloat16
        sd = model.state_dict()
        from torchvision.models.optical_flow import raft_large
        torch.manual_seed(0)
        m = raft_large(weights=None, corr_block=rc.TVCorrBlock(volume_dtype=vdt))
        m.load_state_dict(sd)
        m = m.eval().cuda()
        ub = m.update_block
        fe, ce = rc.FeatureEncoder(), rc.ContextEncoder()
        me, fh = rc.MotionEncoder(in_channels_corr=324), rc.FlowHead(in_channels=128, hidden_size=256)
        rb = rc.RecurrentBlock(input_size=256, hidden_size=128)
        mp = rc.MaskPredictor(in_channels=128, hidden_size=256, multiplier=m.mask_predictor.multiplier)
        for new, old in ((fe, m.feature_encoder), (ce, m.context_encoder), (me, ub.motion_encoder), (fh, ub.flow_head),
                         (rb, ub.recurrent_block), (mp, m.mask_predictor)):
            new.load_state_dict(old.state_dict())
        m.feature_encoder, m.context_encoder = fe.cuda(), ce.cuda().eval()
        ub.motion_encoder, ub.flow_head, ub.recurrent_block, m.mask_predictor = me.cuda(), fh.cuda(), rb.cuda(), mp.cuda()
        _MODELS[vd] = (m, sd)
    return _MODELS[vd]


_BLOB = {}


def device_blob(lib):
    if "w" not in _BLOB:
        code, blob = pack(lib, seeded_state().state_dict())
        assert code == 0, _cabi.last_error()
        _BLOB["w"] = torch.from_numpy(blob).cuda()
    return _BLOB["w"]


def frames(golden_dir, size, n):
    """n frames: the golden pair resized (or a synthetic 1080p texture), then shifted copies."""
    if size == (368, 640):
        import torchvision.transforms.functional as TF
        g = np.load(os.path.join(golden_dir, "frames_im1_im2.npz"))
        a, b = [TF.resize(TF.to_tensor(g[k]), list(size), antialias=True).unsqueeze(0).cuda() for k in ("im1", "im2")]
    else:
        gen = torch.Generator(device="cuda").manual_seed(12)
        a = F.interpolate(torch.rand(1, 3, size[0] // 16, size[1] // 16, device="cuda", generator=gen), size=size,
                          mode="bicubic", align_corners=False).clamp(0, 1)
        b = torch.roll(a, (3, -5), (2, 3))
    out = [a, b]
    while len(out) < n:
        out.append(torch.roll(out[-2], (2 * len(out) - 1, -len(out)), (2, 3)))
    return torch.cat(out[:n], 0).contiguous()


def c_flow(lib, a, b, act, vd, iters=12, ws=None, out=None):
    B, _, H, W = a.shape
    need = lib.rdvc_corr_raft_workspace_bytes(2 * B, B, H, W, act, vd)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda") if ws is None else ws
    out = torch.empty((B, 2, H, W), dtype=torch.float32, device="cuda") if out is None else out
    assert a.stride() == b.stride()
    code = lib.rdvc_corr_raft_flow(a.data_ptr(), b.data_ptr(), (ctypes.c_longlong * 4)(*a.stride()), F32, B, H, W, iters,
                                   act, vd, device_blob(lib).data_ptr(), 0.25, ws.data_ptr(), need, out.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream)
    assert code == 0, _cabi.last_error()
    return out


def c_sequence(lib, fr, act, vd, iters=12):
    n, _, H, W = fr.shape
    need = lib.rdvc_corr_raft_workspace_bytes(n, n - 1, H, W, act, vd)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    out = torch.empty((n - 1, 2, H, W), dtype=torch.float32, device="cuda")
    code = lib.rdvc_corr_raft_flow_sequence(fr.data_ptr(), (ctypes.c_longlong * 4)(*fr.stride()), F32, n, H, W, iters, act,
                                            vd, device_blob(lib).data_ptr(), 0.25, ws.data_ptr(), need, out.data_ptr(),
                                            torch.cuda.current_stream().cuda_stream)
    assert code == 0, _cabi.last_error()
    return out


def py_flow(model, a, b, act):
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=act == F16):
        return rc.raft_flow(model, a, b, 12)


@pytest.mark.gpu
@pytest.mark.parametrize("vd", [F32, BF16], ids=["vol_f32", "vol_bf16"])
@pytest.mark.parametrize("act", [F32, F16], ids=["act_f32", "act_f16"])
@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("size", [(368, 640), (1088, 1920)], ids=["368x640", "1088x1920"])
def test_bit_identical_to_python_dropins(lib, golden_dir, size, B, act, vd):
    model, _ = dropin_model(vd)
    fr = frames(golden_dir, size, B + 1)
    a, b = fr[:-1].contiguous(), fr[1:].contiguous()
    ref = py_flow(model, a, b, act)
    model.corr_block.release()
    got = c_flow(lib, a, b, act, vd)
    torch.cuda.synchronize()
    assert torch.isfinite(got).all()
    assert torch.equal(got, ref), (got - ref).abs().max().item()


def _epe(a, b):
    return (a.float() - b.float()).pow(2).sum(dim=1).sqrt().mean().item()


@pytest.mark.gpu
@pytest.mark.parametrize("act", [F32, F16], ids=["act_f32", "act_f16"])
def test_epe_vs_stock_raft(lib, golden_dir, act):
    fr = frames(golden_dir, (368, 640), 2)
    stock = seeded_state().cuda()
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=act == F16):
        ref = stock(fr[:1], fr[1:], num_flow_updates=12)[-1]
    got = c_flow(lib, fr[:1].contiguous(), fr[1:].contiguous(), act, F32)
    assert _epe(got, ref) < TOL_EPE, _epe(got, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("act", [F32, F16], ids=["act_f32", "act_f16"])
def test_sequence_batch_and_pairs(lib, golden_dir, act):
    model, _ = dropin_model(F32)
    fr = frames(golden_dir, (368, 640), 4)
    seq = c_sequence(lib, fr, act, F32)
    pairs = c_flow(lib, fr[:-1].contiguous(), fr[1:].contiguous(), act, F32)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=act == F16):
        py_seq = rc.raft_flow_sequence(model, fr, 12)
    assert torch.equal(seq, pairs) and torch.equal(seq, py_seq)
    for i in range(3):
        alone = c_flow(lib, fr[i:i + 1].contiguous(), fr[i + 1:i + 2].contiguous(), act, F32)
        assert torch.equal(alone[0], pairs[i]), i


@pytest.mark.gpu
@pytest.mark.parametrize("act", [F32, F16], ids=["act_f32", "act_f16"])
def test_graph_capture_replays_eager(lib, golden_dir, act):
    """Captured on the capture stream in torch's global capture mode, which refuses allocations and synchronisations;
    replays on frames copied in afterwards equal eager calls bit for bit."""
    fr = frames(golden_dir, (368, 640), 5)
    a, b = fr[0:2].clone(), fr[1:3].clone()
    B, _, H, W = a.shape
    need = lib.rdvc_corr_raft_workspace_bytes(2 * B, B, H, W, act, F32)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    out = torch.empty((B, 2, H, W), dtype=torch.float32, device="cuda")
    c_flow(lib, a, b, act, F32, ws=ws, out=out)                      # warm-up: kernel attributes, build plan
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        c_flow(lib, a, b, act, F32, ws=ws, out=out)
    for lo in (2, 0):
        a.copy_(fr[lo:lo + 2])
        b.copy_(fr[lo + 1:lo + 3])
        graph.replay()
        replayed = out.clone()
        eager = c_flow(lib, fr[lo:lo + 2].contiguous(), fr[lo + 1:lo + 3].contiguous(), act, F32)
        torch.cuda.synchronize()
        assert torch.equal(replayed, eager), lo


@pytest.mark.gpu
@pytest.mark.parametrize("act", [F32, F16], ids=["act_f32", "act_f16"])
def test_nan_workspace_and_canaries(lib, golden_dir, act):
    fr = frames(golden_dir, (368, 640), 3)
    a, b = fr[:-1].contiguous(), fr[1:].contiguous()
    B, _, H, W = a.shape
    ref = c_flow(lib, a, b, act, F32)
    need = lib.rdvc_corr_raft_workspace_bytes(2 * B, B, H, W, act, F32)
    ws_buf = torch.full((need + 512,), 0xFF, dtype=torch.uint8, device="cuda")        # every float / half is NaN
    ws_buf[:256] = 0xA5
    ws_buf[-256:] = 0x5A
    n_out = B * 2 * H * W
    out_buf = torch.full((n_out + 128,), 12345.5, dtype=torch.float32, device="cuda")
    got = c_flow(lib, a, b, act, F32, ws=ws_buf[256:256 + need], out=out_buf[64:64 + n_out].view(B, 2, H, W))
    torch.cuda.synchronize()
    assert torch.equal(got, ref)
    assert (ws_buf[:256] == 0xA5).all() and (ws_buf[-256:] == 0x5A).all()
    assert (out_buf[:64] == 12345.5).all() and (out_buf[-64:] == 12345.5).all()


@pytest.mark.gpu
@pytest.mark.parametrize("act", [F32, F16], ids=["act_f32", "act_f16"])
def test_launch_count(lib, golden_dir, act):
    """The count documented in include/rdvc_corr.h."""
    fr = frames(golden_dir, (368, 640), 3)
    per_iter, tail = (15, 3) if act == F32 else (12, 2)
    for iters in (1, 12):
        for seq in (False, True):
            n0 = lib.rdvc_corr_launch_count()
            if seq:
                c_sequence(lib, fr, act, F32, iters)
            else:
                c_flow(lib, fr[:-1].contiguous(), fr[1:].contiguous(), act, F32, iters)
            assert lib.rdvc_corr_launch_count() - n0 == 40 * (1 if seq else 2) + 3 + 15 + 1 + iters * per_iter + tail


@pytest.mark.gpu
@pytest.mark.parametrize("layout", [rc.RDVC_LAYOUT_TILED, rc.RDVC_LAYOUT_ROWMAJOR], ids=["tiled", "rowmajor"])
@pytest.mark.parametrize("dt", [F16, BF16], ids=["f16", "bf16"])
def test_nhwc_pack_writes_the_nchw_bytes(lib, dt, layout):
    """rdvc_corr_pack_nhwc on an NHWC buffer (rows of one trunk, and a wider pixel stride) writes the bytes rdvc_corr_pack
    writes for the same values in NCHW, padding included."""
    tdt = torch.float16 if dt == F16 else torch.bfloat16
    g = torch.Generator(device="cuda").manual_seed(3)
    st = torch.cuda.current_stream().cuda_stream
    for B, h, w, ps in ((1, 46, 80, 128), (2, 37, 53, 136), (3, 17, 16, 128)):
        trunk = torch.randn(B + 1, h, w, ps, device="cuda", generator=g).to(tdt)
        x1, x2 = trunk[:-1, ..., :128], trunk[1:, ..., :128]
        for vd in (F32, BF16):
            n = lib.rdvc_corr_workspace_bytes(B, 128, h, w)
            w_nchw = torch.full((n,), 0x3C, dtype=torch.uint8, device="cuda")
            w_nhwc = w_nchw.clone()
            a, b = x1.permute(0, 3, 1, 2).contiguous(), x2.permute(0, 3, 1, 2).contiguous()
            assert lib.rdvc_corr_pack(a.data_ptr(), b.data_ptr(), B, 128, h, w, dt, vd, layout, 4, w_nchw.data_ptr(), n,
                                      st) == 0
            assert lib.rdvc_corr_pack_nhwc(x1.data_ptr(), x2.data_ptr(), ps, B, 128, h, w, dt, vd, layout, 4,
                                           w_nhwc.data_ptr(), n, st) == 0, _cabi.last_error()
            torch.cuda.synchronize()
            assert torch.equal(w_nchw, w_nhwc), (B, h, w, ps, vd)


def example_frames():
    """The frames examples/raft_flow.c generates: a texture moving by (2, 1) pixels per frame."""
    f, c, y, x = np.meshgrid(np.arange(3), np.arange(3), np.arange(368), np.arange(640), indexing="ij")
    u, v = x - 2 * f + 64, y - f + 64
    return ((u * 7 + v * 13 + (u // 16) * (v // 16) * 29 + c * 31) % 256).astype(np.float32) / np.float32(255.0)


@pytest.mark.gpu
def test_example_program_matches_ctypes(lib, tmp_path):
    exe = build_example(tmp_path)
    sd = seeded_state().state_dict()
    with open(tmp_path / "state.bin", "wb") as f:
        f.write(struct.pack("<I", len(sd)))
        for k, v in sd.items():
            a = np.ascontiguousarray(v.detach().to(torch.float32).numpy())
            f.write(struct.pack("<I", len(k)) + k.encode() + struct.pack("<I", a.ndim))
            f.write(struct.pack(f"<{a.ndim}q", *a.shape) + a.tobytes())
    subprocess.check_call([exe, str(tmp_path / "flows.f32"), str(tmp_path / "state.bin")])
    got = np.fromfile(tmp_path / "flows.f32", np.float32).reshape(2, 2, 368, 640)
    ref = c_sequence(lib, torch.from_numpy(example_frames()).cuda(), F16, F32).cpu().numpy()
    assert np.array_equal(got, ref)
