// tap_conv_sm100.cuh -- the tcgen05 tap-convolution engine behind RAFT's recurrent block (ConvGRU, TV:raft.py:214-270),
// motion encoder and flow head (TV:raft.py:171-211, 272-285), context encoder (FeatureEncoder with frozen BatchNorm,
// TV:raft.py:116-168) and feature encoder (the same with InstanceNorm): implicit GEMMs over NHWC 16-bit activations,
// one pipeline with the tap geometry G and the epilogue EPI as template parameters, entered through tap_conv_kernel or,
// for the InstanceNorm statistics epilogues, tap_conv_in_kernel.  The CUDA-core helpers of those modules (convflow1,
// the fp32 -> 16-bit operand cast, the stem's polyphase pack) are at the end of this file; the feature encoder's
// finalize and apply kernels are in instance_norm_sm100.cuh.
//
// Tile.  16 x 8 pixels of the activation map's x and y (M = 128 GEMM rows, row m = pixel (m % 16, m / 16)).  A map is
// 4-D {C, x, y, B} with the caller's pixel stride, so a channel slice of a channels_last tensor is read in place; one
// box of {64, 16, BOX_Y, 1} lands as 16 * BOX_Y rows of 128 B (SWIZZLE_128B), and the A operand of a tap `row` rows
// further down the box is a descriptor offset of row * 2 KB = two whole 1 KB swizzle atoms, no extra load.  Zero
// padding and every tail tile are TMA's out-of-bounds fill on the load side and a per-pixel mask on the store side.
//
// Geometries (TapGeom<G>: per 64-channel k-block BOXES boxes of BOX_Y rows; box l feeds n_slabs(l) weight slabs, slab i
// at row offset row(l, i)):
//   S1    3x3 stride 1: one box {64, 16, 10} per dx at (x0 + dx - 1, y0 - 1), the 3 dy taps are row offsets.
//   S2    3x3 stride 2: the map has TMA element strides 2 along x and y, so a box {64, 32, 18} lands 16 x 9 pixels of one
//         polyphase component.  Per dx two boxes: rows 2y - 1, 2y + 1, ... (dy = 0 at row offset 0, dy = 2 at offset 1)
//         and rows 2y, 2y + 2, ... (dy = 1).  The centre tap's A operand is exactly the 1x1 stride-2 downsample's input,
//         so with TAP_EPI_DS its tenth slab's MMAs ride on that box into a second accumulator range (columns N..2N).
//   STEM  the 7x7 stride-2 stem over 3 channels as a 4x1 stride-1 convolution over the operand of ce_stem_pack_kernel:
//         one box {64, 16, 11} at (x0, y0 - 2), the 4 vertical taps are row offsets.
//   1X1   one box {64, 16, 8}.
//   GRU5  a 1x5 or 5x1 kernel over [h or r*h | context | motion]: six k-blocks read through three maps (k-block kb from
//         map kb / 2 at channel (kb & 1) * 64), one box {64, 16, 12} at (x0, y0 - 2) per k-block, the 5 taps are row
//         offsets.  The map's y is the tap axis: for the 1x5 pass (p.horiz) the host lists y before x in the map
//         (non-monotonic strides; TMA only multiplies coordinates by strides) and the epilogue swaps the pixel back.
// Weights stream from L2 as (k-block, slab) slabs of N x 64, packed [k-block][slab][N][64], each feeding TAP_P tiles.
//
// Persistent, one CTA per SM, warp-specialised:
//   warp 0     TMA producer: per super-tile (TAP_P tiles), k-block and box the TAP_P boxes (2-stage ring), then that
//              box's weight slabs (TapCfg::W_STAGES-stage ring)
//   warp 1     tcgen05.mma issuer (converged warp; tcgen05 under elect_one): M128 x N x K16, 16-bit operands, fp32
//              accumulators in TMEM (NT columns per tile)
//   warp 2     TMEM allocator
//   warps 4-11 epilogue: warp 4 + e reads TMEM lane quarter e % 4 of tile e / 4; thread = pixel, 16 columns at a time
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>
#include <type_traits>

#include "ptx_sm100.cuh"

namespace rdvc {

constexpr int TAP_TX = 16;                             // tile pixels along the map's x
constexpr int TAP_TY = 8;                              // tile pixels along the map's y
constexpr int TAP_DY_STEP = TAP_TX * 128;              // 2 KB: one box row = two swizzle atoms
constexpr int TAP_P = 2;                               // pixel tiles per weight slab
constexpr int TAP_A_STAGES = 2;
constexpr int TAP_THREADS = 128 + 8 * 32;              // 4 service warps + 8 epilogue warps

constexpr int TAP_G_S1 = 0;
constexpr int TAP_G_S2 = 1;
constexpr int TAP_G_STEM = 2;
constexpr int TAP_G_1X1 = 3;
constexpr int TAP_G_GRU5 = 4;

// epilogues: OutT NHWC at (out, out_ps) unless stated
constexpr int TAP_EPI_RELU = 0;       // relu(acc + bias)
constexpr int TAP_EPI_RES = 1;        // relu(res + relu(acc + bias)); res: OpT NHWC at (res, res_ps)
constexpr int TAP_EPI_DS = 2;         // columns 0..N-1: relu(acc + bias) -> out; N..2N-1: acc + bias -> out2 (OpT, out_ps)
constexpr int TAP_EPI_RAW = 3;        // acc + bias
constexpr int TAP_EPI_SPLIT = 4;      // tanh(acc + bias) on channels 0-127, relu(acc + bias) on the rest
constexpr int TAP_EPI_RELU_FLOW = 5;  // relu(acc + bias); channels N-2, N-1 are the flow (fp32, strided) rounded to OutT
constexpr int TAP_EPI_FLOW2 = 6;      // acc + bias, channels 0-1 -> OutT planes (B, 2, H, W)
constexpr int TAP_EPI_GRU_ZR = 7;     // N = 256: z = sigmoid(acc + bias) -> out, r * h = sigmoid(acc' + bias_r) * h -> out2
constexpr int TAP_EPI_GRU_Q = 8;      // N = 128: h' = (1 - z) h + z tanh(acc + bias) -> out (OutT)
// InstanceNorm statistics epilogues (tap_conv_in_kernel; OutT = OpT).  The conv bias is not added: InstanceNorm
// subtracts each (sample, channel)'s mean, so a per-channel constant cancels exactly, IN(y + b) = IN(y), and without it
// the stored values are smaller and rounded more finely.  Per tile and channel the kernel writes (mean, M2 about that
// mean) of the values AS STORED (rounded to OpT) over the tile's pixels inside the image to part[tile * NT + c]; the
// 4 lane-quarter warps of a tile merge theirs through shared memory (Chan).  No atomics and no per-CTA sums: a tile
// never spans images and its partials do not depend on which CTA ran it, so a sample's statistics do not depend on
// the batch it is in.
constexpr int TAP_EPI_STATS = 9;      // acc -> out (OpT, out_ps)
constexpr int TAP_EPI_DS_STATS = 10;  // columns 0..N-1: acc -> out; N..2N-1 (the fused downsample): acc -> out2 (out_ps)

// ConvGRU: hidden = context = motion channels; z, r*h and h' are dense 128-channel NHWC
constexpr int GRU_C = 128;
constexpr int GRU_KB = 6;                               // 64-channel K-blocks: [h or r*h] 0-1, context 2-3, motion 4-5
constexpr int GRU_TAPS = 5;
constexpr int GRU_ZR_N = 2 * GRU_C, GRU_Q_N = GRU_C;
// packed weights of one ConvGRU: z|r slabs [k-block][tap][256][64], then q slabs [k-block][tap][128][64]
constexpr long long GRU_W_ZR_ELEMS = static_cast<long long>(GRU_KB) * GRU_TAPS * GRU_ZR_N * 64;
constexpr long long GRU_W_Q_ELEMS = static_cast<long long>(GRU_KB) * GRU_TAPS * GRU_Q_N * 64;

struct TapParams {
    int B, H, W;                // output image
    int n_kb;                   // 64-channel k-blocks of the input
    int horiz;                  // GRU5: 1 = taps along x (1x5 kernel, the map lists y before x), 0 = taps along y
    int n_tx, n_ty;             // tiles along the map's x / y
    int n_tiles, n_super;       // B * n_tx * n_ty; ceil(n_tiles / TAP_P)
    const float* bias;          // NT floats (device); RELU_FLOW / FLOW2: cout floats; GRU_ZR: convz's; GRU_Q: convq's
    const float* bias_r;        // GRU_ZR: convr's bias
    int cout;                   // RELU_FLOW / FLOW2: real output channels (channel c reads bias[min(c, cout - 1)])
    void* out;                  // OutT NHWC, pixel stride out_ps; FLOW2: planes (B, 2, H, W); GRU_ZR: z (OpT); GRU_Q: h'
    long long out_ps;
    void* out2;                 // DS: OpT NHWC, pixel stride out_ps; GRU_ZR: r * h (OpT)
    const void* res;            // RES: OpT NHWC; GRU_*: h (OutT); pixel stride res_ps
    long long res_ps;
    const void* z;              // GRU_Q: z (OpT)
    const float* flow;          // RELU_FLOW: fp32 flow at flow[b * fs_b + c * fs_c + y * fs_y + x * fs_x]
    long long fs_b, fs_c, fs_y, fs_x;
    float2* part;               // STATS / DS_STATS: per-tile (mean, M2) partials [n_tiles][NT]
};

template <int G> struct TapGeom;
struct TapGeomOneMap {          // k-block kb is channels kb * 64 of the one map, whose (x, y) are the image's
    static constexpr int MAPS = 1;
    __device__ __forceinline__ static int map(int) { return 0; }
    __device__ __forceinline__ static int chan(int kb) { return kb * 64; }
    __device__ __forceinline__ static void pixel(const TapParams&, int u, int v, int& x, int& y) { x = u; y = v; }
};
template <> struct TapGeom<TAP_G_S1> : TapGeomOneMap {
    static constexpr int BOXES = 3, BOX_Y = TAP_TY + 2, SLABS = 9;
    __device__ __forceinline__ static int n_slabs(int) { return 3; }
    __device__ __forceinline__ static int slab(int l, int i) { return i * 3 + l; }     // dy = i, dx = l
    __device__ __forceinline__ static int row(int, int i) { return i; }
    __device__ __forceinline__ static void box(int l, int x0, int y0, int& x, int& y) { x = x0 + l - 1; y = y0 - 1; }
};
template <> struct TapGeom<TAP_G_S2> : TapGeomOneMap {
    static constexpr int BOXES = 6, BOX_Y = TAP_TY + 1, SLABS = 10;
    __device__ __forceinline__ static int n_slabs(int l) {      // l = 3: dy = 1, dx = 1 and the downsample
        return ((l & 1) == 0 || l == 3) ? 2 : 1;
    }
    __device__ __forceinline__ static int slab(int l, int i) {
        return (l & 1) == 0 ? (i == 0 ? 0 : 6) + (l >> 1) : (i == 0 ? 3 + (l >> 1) : 9);
    }
    __device__ __forceinline__ static int row(int l, int i) { return (l & 1) == 0 ? i : 0; }
    __device__ __forceinline__ static void box(int l, int x0, int y0, int& x, int& y) {
        x = 2 * x0 + (l >> 1) - 1;
        y = 2 * y0 - 1 + (l & 1);
    }
};
template <> struct TapGeom<TAP_G_STEM> : TapGeomOneMap {
    static constexpr int BOXES = 1, BOX_Y = TAP_TY + 3, SLABS = 4;
    __device__ __forceinline__ static int n_slabs(int) { return 4; }
    __device__ __forceinline__ static int slab(int, int i) { return i; }
    __device__ __forceinline__ static int row(int, int i) { return i; }
    __device__ __forceinline__ static void box(int, int x0, int y0, int& x, int& y) { x = x0; y = y0 - 2; }
};
template <> struct TapGeom<TAP_G_1X1> : TapGeomOneMap {
    static constexpr int BOXES = 1, BOX_Y = TAP_TY, SLABS = 1;
    __device__ __forceinline__ static int n_slabs(int) { return 1; }
    __device__ __forceinline__ static int slab(int, int) { return 0; }
    __device__ __forceinline__ static int row(int, int) { return 0; }
    __device__ __forceinline__ static void box(int, int x0, int y0, int& x, int& y) { x = x0; y = y0; }
};
template <> struct TapGeom<TAP_G_GRU5> {
    static constexpr int MAPS = 3, BOXES = 1, BOX_Y = TAP_TY + GRU_TAPS - 1, SLABS = GRU_TAPS;
    __device__ __forceinline__ static int n_slabs(int) { return GRU_TAPS; }
    __device__ __forceinline__ static int slab(int, int i) { return i; }
    __device__ __forceinline__ static int row(int, int i) { return i; }
    __device__ __forceinline__ static void box(int, int x0, int y0, int& x, int& y) { x = x0; y = y0 - GRU_TAPS / 2; }
    __device__ __forceinline__ static int map(int kb) { return kb < 2 ? 0 : kb < 4 ? 1 : 2; }
    __device__ __forceinline__ static int chan(int kb) { return (kb & 1) * 64; }
    __device__ __forceinline__ static void pixel(const TapParams& p, int u, int v, int& x, int& y) {
        x = p.horiz ? v : u;
        y = p.horiz ? u : v;
    }
};

template <int NM> struct TapMaps {
    CUtensorMap a[NM];          // activations {C, x, y, B}
    CUtensorMap w;              // weight slabs {64, N, n_kb * SLABS}, box {64, N, 1}
};

template <int G, int N, int EPI>
struct TapCfg {
    static constexpr bool HAS_DS = EPI == TAP_EPI_DS || EPI == TAP_EPI_DS_STATS;   // fused stride-2 downsample
    static constexpr bool STATS = EPI == TAP_EPI_STATS || EPI == TAP_EPI_DS_STATS;
    static constexpr int NT = HAS_DS ? 2 * N : N;                           // accumulator columns per tile
    static constexpr int W_STAGES = EPI == TAP_EPI_GRU_ZR ? 3 : 4;          // z|r: 3 x 32 KB next to its 48 KB A stages
    static constexpr int BOX_BYTES = TAP_TX * TapGeom<G>::BOX_Y * 128;
    static constexpr int W_BYTES = N * 128;
    static constexpr int A_BYTES = TAP_P * BOX_BYTES;
    static constexpr int SMEM_A = 0;
    static constexpr int SMEM_W = TAP_A_STAGES * A_BYTES;
    static constexpr int SMEM_BAR = SMEM_W + W_STAGES * W_BYTES;
    static constexpr int SMEM_SCR = SMEM_BAR + 256;                         // STATS: per tile [4 warps][NT] (mean, M2)
    static constexpr int SCR_TILE_BYTES = STATS ? 4 * NT * 8 : 0;
    static constexpr int SMEM_TOTAL = SMEM_SCR + TAP_P * SCR_TILE_BYTES;
    static constexpr int SMEM_LAUNCH = SMEM_TOTAL + 1024;                   // slack for 1024-byte alignment
    static constexpr int TMEM_COLS = TAP_P * NT <= 32 ? 32 : TAP_P * NT <= 64 ? 64 : TAP_P * NT <= 128 ? 128
                                   : TAP_P * NT <= 256 ? 256 : 512;
    static_assert(N % 16 == 0 && N >= 16 && N <= 256, "UMMA N");
    static_assert(BOX_BYTES % 1024 == 0, "boxes must start on swizzle atoms");
    static_assert(SMEM_LAUNCH <= 227 * 1024, "shared memory");
    static_assert(TAP_P * NT <= 512, "tensor memory");
    static_assert(!HAS_DS || G == TAP_G_S2, "the fused downsample rides on the stride-2 centre tap");
    static_assert((EPI != TAP_EPI_GRU_ZR && EPI != TAP_EPI_GRU_Q) || G == TAP_G_GRU5, "GRU epilogues");
};

template <typename T> struct GruVec;   // 16 values of T <-> fp32
template <> struct GruVec<float> {
    __device__ static void load(const float* p, float* v) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float4 f = *reinterpret_cast<const float4*>(p + 4 * i);
            v[4 * i] = f.x; v[4 * i + 1] = f.y; v[4 * i + 2] = f.z; v[4 * i + 3] = f.w;
        }
    }
    __device__ static void store(float* p, const float* v) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            *reinterpret_cast<float4*>(p + 4 * i) = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    }
};
template <> struct GruVec<__half> {
    __device__ static void load(const __half* p, float* v) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const uint4 u = *reinterpret_cast<const uint4*>(p + 8 * i);
            const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[j]));
                v[8 * i + 2 * j] = f.x; v[8 * i + 2 * j + 1] = f.y;
            }
        }
    }
    __device__ static void store(__half* p, const float* v) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            uint32_t w[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const __half2 t = __floats2half2_rn(v[8 * i + 2 * j], v[8 * i + 2 * j + 1]);
                w[j] = *reinterpret_cast<const uint32_t*>(&t);
            }
            *reinterpret_cast<uint4*>(p + 8 * i) = make_uint4(w[0], w[1], w[2], w[3]);
        }
    }
};
template <> struct GruVec<__nv_bfloat16> {
    __device__ static void load(const __nv_bfloat16* p, float* v) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const uint4 u = *reinterpret_cast<const uint4*>(p + 8 * i);
            const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[j]));
                v[8 * i + 2 * j] = f.x; v[8 * i + 2 * j + 1] = f.y;
            }
        }
    }
    __device__ static void store(__nv_bfloat16* p, const float* v) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            uint32_t w[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const __nv_bfloat162 t = __floats2bfloat162_rn(v[8 * i + 2 * j], v[8 * i + 2 * j + 1]);
                w[j] = *reinterpret_cast<const uint32_t*>(&t);
            }
            *reinterpret_cast<uint4*>(p + 8 * i) = make_uint4(w[0], w[1], w[2], w[3]);
        }
    }
};

__device__ __forceinline__ float gru_sigmoid(float x) { return 1.f / (1.f + __expf(-x)); }

// tile index -> (batch, first pixel along the map's x, first along its y); tiles run along x first
__device__ __forceinline__ void tap_tile(const TapParams& p, int t, int& b, int& x0, int& y0) {
    const int per_img = p.n_tx * p.n_ty;
    b = t / per_img;
    const int rem = t - b * per_img;
    y0 = (rem / p.n_tx) * TAP_TY;
    x0 = (rem % p.n_tx) * TAP_TX;
}

// One tile's epilogue: this thread's pixel (b, x, y) = NHWC pixel index pix, its TMEM row at taddr; ok = inside the image.
template <int EPI, int N, typename OutT, typename OpT>
__device__ __forceinline__ void tap_epilogue(const TapParams& p, uint32_t taddr, int b, int x, int y, long long pix,
                                             bool ok) {
    if constexpr (EPI == TAP_EPI_FLOW2) {
        float v[16];
        ptx::tmem_ld_x16(taddr, v);
        ptx::tmem_ld_wait();
        if (ok) {
            const long long plane = static_cast<long long>(p.H) * p.W;
            OutT* o = static_cast<OutT*>(p.out) + static_cast<long long>(b) * 2 * plane + (pix - b * plane);
            o[0] = static_cast<OutT>(v[0] + __ldg(p.bias));
            o[plane] = static_cast<OutT>(v[1] + __ldg(p.bias + min(1, p.cout - 1)));
        }
    } else if constexpr (EPI == TAP_EPI_GRU_ZR || EPI == TAP_EPI_GRU_Q) {
        const OutT* hp = static_cast<const OutT*>(p.res) + pix * p.res_ps;
#pragma unroll 1
        for (int c = 0; c < GRU_C; c += 16) {
            float v0[16], hv[16];
            if constexpr (EPI == TAP_EPI_GRU_ZR) {
                float v1[16];
                ptx::tmem_ld_x16(taddr + c, v0);
                ptx::tmem_ld_x16(taddr + GRU_C + c, v1);
                ptx::tmem_ld_wait();
                if (ok) {
                    GruVec<OutT>::load(hp + c, hv);
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        v0[i] = gru_sigmoid(v0[i] + __ldg(p.bias + c + i));              // z
                        v1[i] = gru_sigmoid(v1[i] + __ldg(p.bias_r + c + i)) * hv[i];    // r * h
                    }
                    GruVec<OpT>::store(static_cast<OpT*>(p.out) + pix * GRU_C + c, v0);
                    GruVec<OpT>::store(static_cast<OpT*>(p.out2) + pix * GRU_C + c, v1);
                }
            } else {
                ptx::tmem_ld_x16(taddr + c, v0);
                ptx::tmem_ld_wait();
                if (ok) {
                    float zv[16];
                    GruVec<OutT>::load(hp + c, hv);
                    GruVec<OpT>::load(static_cast<const OpT*>(p.z) + pix * GRU_C + c, zv);
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        const float qv = tanhf(v0[i] + __ldg(p.bias + c + i));
                        v0[i] = (1.f - zv[i]) * hv[i] + zv[i] * qv;
                    }
                    GruVec<OutT>::store(static_cast<OutT*>(p.out) + pix * GRU_C + c, v0);
                }
            }
        }
    } else {
        constexpr int NT = EPI == TAP_EPI_DS ? 2 * N : N;
        OutT* o = static_cast<OutT*>(p.out) + pix * p.out_ps;
#pragma unroll 1
        for (int c = 0; c < NT; c += 16) {
            float v[16];
            ptx::tmem_ld_x16(taddr + c, v);
            ptx::tmem_ld_wait();
            if (ok) {
#pragma unroll
                for (int i = 0; i < 16; ++i)   // RELU_FLOW: bias has N - 2 floats; the flow channels read its last
                    v[i] += __ldg(p.bias + (EPI == TAP_EPI_RELU_FLOW ? min(c + i, p.cout - 1) : c + i));
                if constexpr (EPI == TAP_EPI_RELU || EPI == TAP_EPI_RELU_FLOW) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.f);
                } else if constexpr (EPI == TAP_EPI_RES) {
                    float r[16];
                    GruVec<OpT>::load(static_cast<const OpT*>(p.res) + pix * p.res_ps + c, r);
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] = fmaxf(r[i] + fmaxf(v[i], 0.f), 0.f);
                } else if constexpr (EPI == TAP_EPI_SPLIT) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] = c < 128 ? tanhf(v[i]) : fmaxf(v[i], 0.f);
                }
                if constexpr (EPI == TAP_EPI_RELU_FLOW) {
                    if (c == N - 16) {
                        const float* f = p.flow + b * p.fs_b + y * p.fs_y + x * p.fs_x;
                        v[14] = __ldg(f);
                        v[15] = __ldg(f + p.fs_c);
                    }
                }
                if constexpr (EPI == TAP_EPI_DS) {
                    if (c < N) {
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.f);
                        GruVec<OutT>::store(o + c, v);
                    } else {
                        GruVec<OpT>::store(static_cast<OpT*>(p.out2) + pix * p.out_ps + (c - N), v);
                    }
                } else {
                    GruVec<OutT>::store(o + c, v);
                }
            }
        }
    }
}

template <typename OpT>
__device__ __forceinline__ float tap_round(float v) {
    if constexpr (std::is_same<OpT, __half>::value) return __half2float(__float2half_rn(v));
    else return __bfloat162float(__float2bfloat16_rn(v));
}

// 16 values per lane -> lane l returns the warp's sum of value (l >> 1) & 15.  A halving exchange (16 shuffles instead
// of 80) in a fixed order, so the sums are the same on every run.
__device__ __forceinline__ float warp_sum16(float* v, int lane) {
#pragma unroll
    for (int o = 16, h = 8; o >= 2; o >>= 1, h >>= 1) {
        const bool hi = (lane & o) != 0;
#pragma unroll
        for (int i = 0; i < h; ++i) {
            const float send = hi ? v[i] : v[i + h];
            const float keep = hi ? v[i + h] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
    }
    return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 1);
}

__device__ __forceinline__ void tap_named_sync(int id, int threads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

// STATS / DS_STATS epilogue of one tile (tile < n_tiles) at (x0, y0): store acc rounded to OpT, then per channel the
// tile's (mean, M2) of the stored values over its pixels inside the image.  Each warp reduces its 32 pixels (lane-
// quarter q = tile rows 2q and 2q + 1) about its own mean; the 4 warps merge in order through scr ([4][NT] float2).
template <int N, int NT, typename OpT>
__device__ __forceinline__ void tap_stats_epilogue(const TapParams& p, uint32_t taddr, long long pix, bool ok, int tile,
                                                   int x0, int y0, int q, int lane, int bar_id, float2* scr) {
    const float n_w = static_cast<float>(__popc(__ballot_sync(0xffffffffu, ok)));
#pragma unroll 1
    for (int c = 0; c < NT; c += 16) {
        float v[16], s[16];
        ptx::tmem_ld_x16(taddr + c, v);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            v[i] = ok ? tap_round<OpT>(v[i]) : 0.f;
            s[i] = v[i];
        }
        if (ok) {
            OpT* o = c < N ? static_cast<OpT*>(p.out) + pix * p.out_ps + c
                           : static_cast<OpT*>(p.out2) + pix * p.out_ps + (c - N);
            GruVec<OpT>::store(o, v);
        }
        const float mean = n_w > 0.f ? warp_sum16(s, lane) / n_w : 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i) {      // every lane shuffles (a full-mask shuffle under `ok` would never complete)
            const float m = __shfl_sync(0xffffffffu, mean, 2 * i);
            const float d = ok ? v[i] - m : 0.f;
            s[i] = d * d;
        }
        const float m2 = warp_sum16(s, lane);
        if ((lane & 1) == 0) scr[q * NT + c + (lane >> 1)] = make_float2(mean, m2);
    }
    tap_named_sync(bar_id, 128);
    const float nx = static_cast<float>(min(TAP_TX, p.W - x0));
#pragma unroll 1
    for (int c = q * 32 + lane; c < NT; c += 128) {
        float n = 0.f, mean = 0.f, m2 = 0.f;
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            const float nq = nx * static_cast<float>(max(0, min(2, p.H - y0 - 2 * w)));
            if (nq == 0.f) continue;
            const float2 a = scr[w * NT + c];
            if (n == 0.f) {
                n = nq; mean = a.x; m2 = a.y;
            } else {
                const float nn = n + nq, d = a.x - mean;
                mean += d * (nq / nn);
                m2 += a.y + d * d * (n * nq / nn);
                n = nn;
            }
        }
        p.part[static_cast<long long>(tile) * NT + c] = make_float2(mean, m2);
    }
    tap_named_sync(bar_id, 128);                         // scr is free for the next super-tile
}

// The persistent pipeline shared by tap_conv_kernel and tap_conv_in_kernel.  G: TAP_G_*; N: GEMM width (output
// channels padded to a multiple of 16); EPI: TAP_EPI_*; OutT: output dtype (GRU epilogues: the dtype of h and h');
// OpT: 16-bit operand dtype.  All maps 128-byte swizzled.
template <int G, int N, int EPI, typename OutT, typename OpT>
__device__ __forceinline__ void tap_conv_body(const TapMaps<TapGeom<G>::MAPS>& maps, const TapParams& p) {
    using Geo = TapGeom<G>;
    using Cfg = TapCfg<G, N, EPI>;
    constexpr int NT = Cfg::NT;
    constexpr int WST = Cfg::W_STAGES;
    constexpr bool DS = Cfg::HAS_DS;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    const uint32_t s_a = ptx::smem_u32(smem + Cfg::SMEM_A);
    const uint32_t s_w = ptx::smem_u32(smem + Cfg::SMEM_W);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::SMEM_BAR);
    const uint32_t bar0 = ptx::smem_u32(bars);
    constexpr int A_FULL = 0, A_EMPTY = TAP_A_STAGES, W_FULL = 2 * TAP_A_STAGES, W_EMPTY = W_FULL + WST,
                  T_FULL = W_EMPTY + WST, T_EMPTY = T_FULL + 1;
    auto bar = [&](int i) { return bar0 + 8u * i; };
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(bars + T_EMPTY + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
#pragma unroll
        for (int i = 0; i < Geo::MAPS; ++i) ptx::prefetch_tensormap(&maps.a[i]);
        ptx::prefetch_tensormap(&maps.w);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < TAP_A_STAGES; ++i) {
            ptx::mbar_init(bar(A_FULL + i), 1);
            ptx::mbar_init(bar(A_EMPTY + i), 1);
        }
        for (int i = 0; i < WST; ++i) {
            ptx::mbar_init(bar(W_FULL + i), 1);
            ptx::mbar_init(bar(W_EMPTY + i), 1);
        }
        ptx::mbar_init(bar(T_FULL), 1);
        ptx::mbar_init(bar(T_EMPTY), 8);
        ptx::fence_mbar_init();
    }
    if (warp == 2) {
        ptx::tmem_alloc(ptx::smem_u32(const_cast<uint32_t*>(tmem_slot)), Cfg::TMEM_COLS);
        ptx::tmem_relinquish();
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            uint32_t a_it = 0, w_it = 0;
            for (int s = blockIdx.x; s < p.n_super; s += gridDim.x) {
                int b[TAP_P], x0[TAP_P], y0[TAP_P];
#pragma unroll
                for (int j = 0; j < TAP_P; ++j)      // a missing last tile reloads the one before (its stores are masked)
                    tap_tile(p, min(s * TAP_P + j, p.n_tiles - 1), b[j], x0[j], y0[j]);
                for (int kb = 0; kb < p.n_kb; ++kb) {
                    const CUtensorMap* am = &maps.a[Geo::map(kb)];
                    for (int l = 0; l < Geo::BOXES; ++l, ++a_it) {
                        const uint32_t st = a_it % TAP_A_STAGES, ph = (a_it / TAP_A_STAGES) & 1;
                        ptx::mbar_wait(bar(A_EMPTY + st), ph ^ 1);
                        ptx::mbar_arrive_expect_tx(bar(A_FULL + st), Cfg::A_BYTES);
#pragma unroll
                        for (int j = 0; j < TAP_P; ++j) {
                            int x, y;
                            Geo::box(l, x0[j], y0[j], x, y);
                            ptx::tma_load_4d(s_a + st * Cfg::A_BYTES + j * Cfg::BOX_BYTES, am, bar(A_FULL + st),
                                             Geo::chan(kb), x, y, b[j]);
                        }
                        const int ns = Geo::n_slabs(l);
                        for (int i = 0; i < ns; ++i, ++w_it) {
                            const uint32_t ws = w_it % WST, wph = (w_it / WST) & 1;
                            ptx::mbar_wait(bar(W_EMPTY + ws), wph ^ 1);
                            ptx::mbar_arrive_expect_tx(bar(W_FULL + ws), Cfg::W_BYTES);
                            ptx::tma_load_3d(s_w + ws * Cfg::W_BYTES, &maps.w, bar(W_FULL + ws), 0, 0,
                                             kb * Geo::SLABS + Geo::slab(l, i));
                        }
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================== MMA issuer (converged warp; tcgen05 under elect_one) =====================
        constexpr uint32_t idesc = ptx::umma_idesc(128, N, std::is_same<OpT, __nv_bfloat16>::value ? 1 : 0);
        uint32_t a_it = 0, w_it = 0, t_it = 0;
        for (int s = blockIdx.x; s < p.n_super; s += gridDim.x, ++t_it) {
            ptx::mbar_wait(bar(T_EMPTY), (t_it & 1) ^ 1);
            ptx::tc_fence_after();
            for (int kb = 0; kb < p.n_kb; ++kb) {
                for (int l = 0; l < Geo::BOXES; ++l, ++a_it) {
                    const uint32_t st = a_it % TAP_A_STAGES, ph = (a_it / TAP_A_STAGES) & 1;
                    ptx::mbar_wait(bar(A_FULL + st), ph);
                    ptx::tc_fence_after();
                    const uint64_t a_desc0 = ptx::umma_desc_k_sw128(s_a + st * Cfg::A_BYTES);
                    const int ns = Geo::n_slabs(l);
#pragma unroll 1
                    for (int i = 0; i < ns; ++i, ++w_it) {
                        const uint32_t ws = w_it % WST, wph = (w_it / WST) & 1;
                        ptx::mbar_wait(bar(W_FULL + ws), wph);
                        ptx::tc_fence_after();
                        const uint64_t b_desc0 = ptx::umma_desc_k_sw128(s_w + ws * Cfg::W_BYTES);
                        const bool ds = DS && l == 3 && i == 1;                  // the downsample's slab
                        const uint32_t col = ds ? N : 0;
                        const bool first = ds ? kb == 0 : (kb | l | i) == 0;
                        const int row = Geo::row(l, i);
                        if (ptx::elect_one()) {
#pragma unroll
                            for (int j = 0; j < TAP_P; ++j) {
#pragma unroll
                                for (int k = 0; k < 4; ++k)
                                    ptx::umma_bf16(tmem_base + j * NT + col,
                                                   a_desc0 + ((j * Cfg::BOX_BYTES + row * TAP_DY_STEP + k * 32) >> 4),
                                                   b_desc0 + ((k * 32) >> 4), idesc, (first && k == 0) ? 0u : 1u);
                            }
                            ptx::umma_commit(bar(W_EMPTY + ws));                     // slab free when these MMAs retire
                            if (i == ns - 1) ptx::umma_commit(bar(A_EMPTY + st));
                            if (i == ns - 1 && l == Geo::BOXES - 1 && kb == p.n_kb - 1) ptx::umma_commit(bar(T_FULL));
                        }
                        __syncwarp();
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ===================== epilogue =====================
        const int e = warp - 4;
        const int q = e & 3;                 // TMEM lane quarter (warp % 4)
        const int j = e >> 2;                // tile of the super-tile
        const int m = q * 32 + lane;         // GEMM row = pixel of the tile
        uint32_t t_it = 0;
        for (int s = blockIdx.x; s < p.n_super; s += gridDim.x, ++t_it) {
            const int tile = s * TAP_P + j;
            int b, x0, y0, x, y;
            tap_tile(p, min(tile, p.n_tiles - 1), b, x0, y0);
            Geo::pixel(p, x0 + (m & (TAP_TX - 1)), y0 + m / TAP_TX, x, y);
            const bool ok = (tile < p.n_tiles) && (x < p.W) && (y < p.H);
            const long long pix = (static_cast<long long>(b) * p.H + y) * p.W + x;
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + j * NT;
            ptx::mbar_wait(bar(T_FULL), t_it & 1);
            ptx::tc_fence_after();
            if constexpr (Cfg::STATS) {       // the duplicated last tile of an odd super-tile writes nothing
                if (tile < p.n_tiles)
                    tap_stats_epilogue<N, NT, OpT>(p, taddr, pix, ok, tile, x0, y0, q, lane, 1 + j,
                                                   reinterpret_cast<float2*>(smem + Cfg::SMEM_SCR +
                                                                             j * Cfg::SCR_TILE_BYTES));
            } else {
                tap_epilogue<EPI, N, OutT, OpT>(p, taddr, b, x, y, pix, ok);
            }
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(bar(T_EMPTY));      // accumulators back to the MMA warp
        }
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 2) ptx::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

template <int G, int N, int EPI, typename OutT, typename OpT>
__global__ void __launch_bounds__(TAP_THREADS, 1)
tap_conv_kernel(const __grid_constant__ TapMaps<TapGeom<G>::MAPS> maps, const TapParams p) {
    static_assert(!TapCfg<G, N, EPI>::STATS, "the statistics epilogues run in tap_conv_in_kernel");
    tap_conv_body<G, N, EPI, OutT, OpT>(maps, p);
}

// The InstanceNorm layers' convolutions (EPI = TAP_EPI_STATS or TAP_EPI_DS_STATS): the raw output in OpT and per-tile
// statistics partials, normalised afterwards by in_finalize_kernel and in_apply_kernel.
template <int G, int N, int EPI, typename OpT>
__global__ void __launch_bounds__(TAP_THREADS, 1)
tap_conv_in_kernel(const __grid_constant__ TapMaps<TapGeom<G>::MAPS> maps, const TapParams p) {
    static_assert(TapCfg<G, N, EPI>::STATS, "tap_conv_in_kernel runs the statistics epilogues");
    tap_conv_body<G, N, EPI, OpT, OpT>(maps, p);
}

// ===================== CUDA-core helpers =====================

// fp32 activations -> the 16-bit NHWC operand copies the GEMMs read (h, context, motion: blockIdx.y = source).
// One thread converts 8 channels of one pixel.
struct GruCastParams {
    const float* src[3];
    long long ps[3];            // pixel strides (elements)
    void* dst[3];               // OpT [B*H*W][128]
    long long n_pix;
};

template <typename OpT>
__global__ void __launch_bounds__(256) convgru_cast_kernel(const GruCastParams p) {
    const long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
    const int s = blockIdx.y;
    if (i >= p.n_pix * (GRU_C / 8)) return;
    const long long pix = i / (GRU_C / 8);
    const int c = static_cast<int>(i % (GRU_C / 8)) * 8;
    // (selects instead of p.src[s]: a dynamically indexed parameter array goes through a local-memory copy)
    const float* src = (s == 0 ? p.src[0] + pix * p.ps[0] : s == 1 ? p.src[1] + pix * p.ps[1] : p.src[2] + pix * p.ps[2]) + c;
    void* dst = s == 0 ? p.dst[0] : s == 1 ? p.dst[1] : p.dst[2];
    const float4 a = *reinterpret_cast<const float4*>(src), b = *reinterpret_cast<const float4*>(src + 4);
    const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    uint32_t w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if constexpr (std::is_same<OpT, __half>::value) {
            const __half2 t = __floats2half2_rn(v[2 * j], v[2 * j + 1]);
            w[j] = *reinterpret_cast<const uint32_t*>(&t);
        } else {
            const __nv_bfloat162 t = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
            w[j] = *reinterpret_cast<const uint32_t*>(&t);
        }
    }
    *reinterpret_cast<uint4*>(static_cast<OpT*>(dst) + pix * GRU_C + c) = make_uint4(w[0], w[1], w[2], w[3]);
}

// convflow1: 7x7 convolution 2 -> 128 + bias + ReLU of the fp32 flow, padding 3 -> OpT NHWC at (out, out_ps).
// Weights: the packed GEMM operand [128][128] (row n, column k = (ky * 7 + kx) * 2 + ci, K = 98 padded to 128; see
// rdvc_corr_update_conv_pack_weights), staged once per CTA in shared memory as fp32 [98][128].  Lane = pixel (consecutive x, so
// the flow loads coalesce), warp % 4 = a 32-channel group (its weights are warp-uniform: shared-memory broadcasts).
// Operands are rounded to OpT and summed in fp32 in k order.
constexpr int CF1_K = 98;
constexpr int CF1_KP = 128;
constexpr int CF1_THREADS = 256;
constexpr int CF1_SMEM = CF1_K * 128 * 4;   // 49 KB

struct Cf1Params {
    const float* flow;          // flow[b * fs_b + c * fs_c + y * fs_y + x * fs_x]
    long long fs_b, fs_c, fs_y, fs_x;
    const void* w;              // OpT [128][128]
    const float* bias;          // 128 floats
    void* out;                  // OpT NHWC, pixel stride out_ps
    long long out_ps;
    int B, H, W;
    long long n_pix;
};

template <typename OpT>
__device__ __forceinline__ float cf1_round(float v) {
    if constexpr (std::is_same<OpT, __half>::value) return __half2float(__float2half_rn(v));
    else return __bfloat162float(__float2bfloat16_rn(v));
}

template <typename OpT>
__global__ void __launch_bounds__(CF1_THREADS) convflow1_kernel(const Cf1Params p) {
    extern __shared__ float cf1_w[];                 // [k][n]
    const OpT* wg = static_cast<const OpT*>(p.w);
    for (int i = threadIdx.x; i < CF1_K * 128; i += CF1_THREADS) {
        const int k = i / 128, n = i % 128;
        cf1_w[i] = static_cast<float>(wg[n * CF1_KP + k]);
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int cg = (warp & 3) * 32;
    float bias[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) bias[i] = __ldg(p.bias + cg + i);
    const long long groups = (p.n_pix + 31) / 32;
    for (long long g = static_cast<long long>(blockIdx.x) * 2 + (warp >> 2); g < groups; g += 2LL * gridDim.x) {
        const long long pix = g * 32 + lane;
        const bool ok = pix < p.n_pix;
        const long long pc = ok ? pix : p.n_pix - 1;
        const int x = static_cast<int>(pc % p.W);
        const long long r = pc / p.W;
        const int y = static_cast<int>(r % p.H);
        const int b = static_cast<int>(r / p.H);
        const float* fb = p.flow + b * p.fs_b;
        float acc[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) acc[i] = 0.f;
#pragma unroll 1
        for (int ky = 0; ky < 7; ++ky) {
            const int yy = y + ky - 3;
            const bool oky = (yy >= 0) && (yy < p.H);
#pragma unroll 1
            for (int kx = 0; kx < 7; ++kx) {
                const int xx = x + kx - 3;
                float f0 = 0.f, f1 = 0.f;
                if (oky && xx >= 0 && xx < p.W) {
                    const float* f = fb + yy * p.fs_y + xx * p.fs_x;
                    f0 = cf1_round<OpT>(__ldg(f));
                    f1 = cf1_round<OpT>(__ldg(f + p.fs_c));
                }
                const float4* w0 = reinterpret_cast<const float4*>(cf1_w + ((ky * 7 + kx) * 2) * 128 + cg);
                const float4* w1 = w0 + 32;           // next k: 128 floats further
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float4 a = w0[i], c = w1[i];
                    acc[4 * i] = fmaf(f1, c.x, fmaf(f0, a.x, acc[4 * i]));
                    acc[4 * i + 1] = fmaf(f1, c.y, fmaf(f0, a.y, acc[4 * i + 1]));
                    acc[4 * i + 2] = fmaf(f1, c.z, fmaf(f0, a.z, acc[4 * i + 2]));
                    acc[4 * i + 3] = fmaf(f1, c.w, fmaf(f0, a.w, acc[4 * i + 3]));
                }
            }
        }
        if (ok) {
#pragma unroll
            for (int i = 0; i < 32; ++i) acc[i] = fmaxf(acc[i] + bias[i], 0.f);
            OpT* o = static_cast<OpT*>(p.out) + pix * p.out_ps + cg;
            GruVec<OpT>::store(o, acc);
            GruVec<OpT>::store(o + 16, acc + 16);
        }
    }
}

// The stem's GEMM operand: per half-resolution pixel (X, Y) of image b, 64 OpT values; column k < 48 is
// tx = k / 12, py = k % 12 / 6, px = k % 6 / 3, c = k % 3 -> image[b, c, 2 Y + py, 2 (X + tx - 2) + px] (zero outside the
// image), columns 48-63 are zero.  With vertical taps ty at rows Y + ty - 2 the 4x4 stride-1 GEMM covers the 7x7
// stride-2 stencil: ky = 2 ty + py - 1, kx = 2 tx + px - 1 (the one unused row / column per axis has zero weights).
struct CeStemParams {
    const void* img;                    // InT, element strides sb, sc, sy, sx
    long long sb, sc, sy, sx;
    int H, W, H1, W1;                   // image and half-resolution sizes
    void* out;                          // OpT [B * H1 * W1][64]
    long long n_pix;                    // B * H1 * W1
};

template <typename InT, typename OpT>
__global__ void __launch_bounds__(256) ce_stem_pack_kernel(const CeStemParams p) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;   // (pixel, 8-column group)
    if (i >= p.n_pix * 8) return;
    const long long pix = i >> 3;
    const int g = static_cast<int>(i & 7);
    const int X = static_cast<int>(pix % p.W1);
    const long long r = pix / p.W1;
    const int Y = static_cast<int>(r % p.H1);
    const long long b = r / p.H1;
    const InT* img = static_cast<const InT*>(p.img) + b * p.sb;
    uint32_t w[4];
#pragma unroll
    for (int e = 0; e < 8; e += 2) {
        float v[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int k = g * 8 + e + h;
            v[h] = 0.f;
            if (k < 48) {
                const int tx = k / 12, py = k % 12 / 6, px = k % 6 / 3, c = k % 3;
                const int sy = 2 * Y + py, sx = 2 * (X + tx - 2) + px;
                if (sy < p.H && sx >= 0 && sx < p.W) v[h] = static_cast<float>(img[c * p.sc + sy * p.sy + sx * p.sx]);
            }
        }
        if constexpr (std::is_same<OpT, __half>::value) {
            const __half2 t = __floats2half2_rn(v[0], v[1]);
            w[e / 2] = *reinterpret_cast<const uint32_t*>(&t);
        } else {
            const __nv_bfloat162 t = __floats2bfloat162_rn(v[0], v[1]);
            w[e / 2] = *reinterpret_cast<const uint32_t*>(&t);
        }
    }
    *reinterpret_cast<uint4*>(static_cast<OpT*>(p.out) + pix * 64 + g * 8) = make_uint4(w[0], w[1], w[2], w[3]);
}

}  // namespace rdvc
