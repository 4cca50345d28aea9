"""The tcgen05 tap-convolution engine (csrc/tap_conv_sm100.cuh) behind the recurrent block, the motion encoder and flow
head, and the context encoder, and the CUDA-core helpers next to it: every instantiation the dispatch tables make is
Blackwell-native (tcgen05.mma, TMA loads, TMEM reads) and allocates its registers without spills.  No GPU needed; the
modules' numerics are tested on the GPU in test_recurrent_block.py, test_motion_encoder.py and test_context_encoder.py.
"""
import os
import re
import subprocess
import tempfile

import pytest

import rdvc_corr_b200 as rc

PKG = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                   "pfe-raft-and-hyperprior-based-learned-video-compression_b200")

G_S1, G_S2, G_STEM, G_1X1, G_GRU5 = range(5)                                          # TAP_G_*
RELU, RES, DS, RAW, SPLIT, RELU_FLOW, FLOW2, GRU_ZR, GRU_Q = range(9)                 # TAP_EPI_*
# (geometry, N, epilogue, output dtype) of every tap_conv_kernel instantiation, per operand dtype P
INSTANCES = [
    # recurrent block (rdvc_corr_convgru): z|r and q passes, fp32 or 16-bit hidden state
    (G_GRU5, 256, GRU_ZR, "float"), (G_GRU5, 256, GRU_ZR, "P"), (G_GRU5, 128, GRU_Q, "float"), (G_GRU5, 128, GRU_Q, "P"),
    # motion encoder and flow head (rdvc_corr_update_conv): convcorr2, convflow2 (= layer1's conv1), flow_head.conv1,
    # conv, flow_head.conv2
    (G_S1, 192, RELU, "P"), (G_S1, 64, RELU, "P"), (G_S1, 256, RELU, "P"), (G_S1, 128, RELU_FLOW, "float"),
    (G_S1, 128, RELU_FLOW, "P"), (G_S1, 16, FLOW2, "float"), (G_S1, 16, FLOW2, "P"),
    # context encoder (rdvc_corr_context_encoder)
    (G_STEM, 64, RELU, "P"), (G_S1, 64, RES, "P"), (G_S1, 128, RELU, "P"), (G_S1, 128, RES, "P"), (G_S2, 128, DS, "P"),
    (G_1X1, 256, RAW, "float"), (G_1X1, 256, RAW, "P"), (G_1X1, 256, SPLIT, "float"), (G_1X1, 256, SPLIT, "P"),
]
OPS = ("__half", "__nv_bfloat16")


def expected():
    return sorted((g, n, e, op if o == "P" else o, op) for op in OPS for g, n, e, o in INSTANCES)


@pytest.fixture(scope="module")
def lib():
    rc._build.build()
    return rc._cabi.load()


def test_sass_has_tcgen05_and_tma(lib):
    """The library holds exactly the listed tap_conv_kernel instantiations, and each of them, the NHWC variant of the
    1x1 GEMM behind the fused lookup, is Blackwell-native: tcgen05.mma (UTCHMMA), TMA loads (UTMALDG) and TMEM reads
    (LDTM)."""
    out = subprocess.run(["cuobjdump", "-sass", rc._cabi.lib_path()], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    funcs = out.stdout.split("Function : ")
    tap = [f for f in funcs if f.startswith("_ZN4rdvc15tap_conv_kernel")]
    nhwc = [f for f in funcs if f.startswith("_ZN4rdvc24corr_conv1x1_nhwc_kernel")]
    assert len(tap) == len(expected()), len(tap)
    assert len(nhwc) == 2, len(nhwc)
    for f in tap + nhwc:
        assert "UTCHMMA" in f and "UTMALDG" in f and "LDTM" in f, f.splitlines()[0]
    assert len([f for f in funcs if f.startswith("_ZN4rdvc16convflow1_kernel")]) == 2
    names = subprocess.run(["cu++filt"], input="\n".join(f.split(None, 1)[0] for f in tap), capture_output=True,
                           text=True, check=True).stdout.split("\n")
    got = []
    for name in names[:len(tap)]:
        g, n, e, out_t, op = re.search(r"tap_conv_kernel<([^>]*)>", name).group(1).split(", ")
        got.append((int(g.replace("(int)", "")), int(n.replace("(int)", "")), int(e.replace("(int)", "")), out_t, op))
    assert sorted(got) == expected()


def test_no_register_spills():
    """-Xptxas -v over every tap_conv_kernel instantiation and the CUDA-core helpers: no spill stores or loads."""
    from rdvc_corr_b200 import _build
    inst = [f"template __global__ void tap_conv_kernel<{g}, {n}, {e}, {o}, {op}>"
            f"(const __grid_constant__ TapMaps<TapGeom<{g}>::MAPS>, const TapParams);" for g, n, e, o, op in expected()]
    for op in OPS:
        inst.append(f"template __global__ void convflow1_kernel<{op}>(const Cf1Params);")
        inst.append(f"template __global__ void corr_conv1x1_nhwc_kernel<{op}>(const __grid_constant__ CUtensorMap, "
                    "const __grid_constant__ CUtensorMap, const Conv1x1Params);")
        for t in ("float", "__half", "__nv_bfloat16"):
            inst.append(f"template __global__ void ce_stem_pack_kernel<{t}, {op}>(const CeStemParams);")
    src = '#include "tap_conv_sm100.cuh"\n#include "corr_conv1x1_sm100.cuh"\nnamespace rdvc {\n' + "\n".join(inst) + "\n}\n"
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
