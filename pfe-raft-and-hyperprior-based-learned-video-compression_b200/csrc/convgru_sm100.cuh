// convgru_sm100.cuh -- RAFT's recurrent block (torchvision RecurrentBlock / ConvGRU, TV:raft.py:214-270) as tcgen05
// implicit GEMMs over NHWC 16-bit activations.  One ConvGRU pass (TV:raft.py:223-229)
//
//   z = sigmoid(convz([h | x]))   r = sigmoid(convr([h | x]))   q = tanh(convq([r*h | x]))   h' = (1 - z) h + z q
//
// with 1x5 or 5x1 kernels, hidden size 128 and x = [context (128) | motion features (128)] runs as two launches:
//   gru_zr : M = pixels, N = 256 (convz | convr), K = 5 taps x 384 channels; epilogue bias -> sigmoid, writes z and
//            r*h (16-bit, NHWC, 128 channels) to the workspace;
//   gru_q  : the same GEMM shape with N = 128 over [r*h | x]; epilogue bias -> tanh -> h' = (1 - z) h + z q in fp32,
//            stored in h's dtype.
// Nothing is concatenated: the 384 channels are six 64-channel K-blocks read through three tensor maps (h or r*h,
// context, motion), each with its own pixel stride, so a channel slice of a channels_last tensor is read in place.
//
// Tile geometry.  A tile is 16 pixels ACROSS the tap axis x 8 pixels ALONG it (M = 128).  The activation maps are 4-D
// {64-channel half, across, along, batch}: for the 5x1 (vertical) pass `across` is x and `along` is y -- the usual
// NHWC order -- and for the 1x5 (horizontal) pass the map lists y before x (non-monotonic strides; TMA only
// multiplies coordinates by strides).  Either way one box of {64, 16, 8 + 4, 1} = 24 KB lands as 192 rows of 128 B
// (one SWIZZLE_128B row per pixel, row = along * 16 + across), and the A operand of tap t is the box shifted by t
// along-steps = t * 16 rows = two whole 1 KB swizzle atoms: a descriptor offset, no extra load.  The convolution's
// zero padding and every tail tile (odd H / W, H*W not a multiple of 128) are TMA's out-of-bounds fill on the load side
// and a per-pixel mask on the store side.
//
// Weights (983 KB z|r, 492 KB q per pass) cannot stay in shared memory: they stream from L2 in (k-block, tap) slabs
// of N x 64 (32 / 16 KB), and every slab feeds GRU_P = 2 pixel tiles (TMEM: 2 x 256 columns for z|r), halving the
// L2 -> SM weight traffic of a one-tile CTA.
//
// Persistent, one CTA per SM, warp-specialised:
//   warp 0     TMA producer: per super-tile (GRU_P tiles) and k-block, the GRU_P activation boxes (2-stage ring), then
//              the 5 tap slabs of that k-block (3 / 4-stage ring)
//   warp 1     tcgen05.mma issuer: M128 x N x K16, 16-bit operands, fp32 accumulators in TMEM (one per tile)
//   warp 2     TMEM allocator
//   warps 4-11 epilogue: warp 4 + e reads TMEM lane quarter e % 4 of tile e / 4; thread = pixel, 16 channels at a time
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>
#include <type_traits>

#include "ptx_sm100.cuh"

namespace rdvc {

constexpr int GRU_C = 128;                             // hidden = context = motion channels
constexpr int GRU_KB = 6;                               // 64-channel K-blocks: [h or r*h] 0-1, context 2-3, motion 4-5
constexpr int GRU_TAPS = 5;
constexpr int GRU_TA = 16;                              // tile pixels across the tap axis
constexpr int GRU_TL = 8;                               // tile pixels along the tap axis
constexpr int GRU_BOX_L = GRU_TL + GRU_TAPS - 1;        // 12: a box carries the tap halo
constexpr int GRU_BOX_BYTES = GRU_TA * GRU_BOX_L * 128; // 24 KB
constexpr int GRU_TAP_STEP = GRU_TA * 128;              // 2 KB: one along-step = two swizzle atoms
constexpr int GRU_P = 2;                                // pixel tiles per weight slab
constexpr int GRU_A_STAGES = 2;
constexpr int GRU_THREADS = 128 + 8 * 32;               // 4 service warps + 8 epilogue warps
constexpr int GRU_ZR_N = 2 * GRU_C, GRU_Q_N = GRU_C;
// packed weights of one ConvGRU: z|r slabs [k-block][tap][256][64], then q slabs [k-block][tap][128][64]
constexpr long long GRU_W_ZR_ELEMS = static_cast<long long>(GRU_KB) * GRU_TAPS * GRU_ZR_N * 64;
constexpr long long GRU_W_Q_ELEMS = static_cast<long long>(GRU_KB) * GRU_TAPS * GRU_Q_N * 64;

template <int N>
struct GruCfg {
    static constexpr int W_BYTES = N * 128;                       // one (k-block, tap) slab: 32 / 16 KB
    static constexpr int W_STAGES = (N == 256) ? 3 : 4;
    static constexpr int A_BYTES = GRU_P * GRU_BOX_BYTES;         // 48 KB
    static constexpr int SMEM_A = 0;
    static constexpr int SMEM_W = GRU_A_STAGES * A_BYTES;
    static constexpr int SMEM_BAR = SMEM_W + W_STAGES * W_BYTES;
    static constexpr int SMEM_TOTAL = SMEM_BAR + 256;
    static constexpr int SMEM_LAUNCH = SMEM_TOTAL + 1024;          // slack for 1024-byte alignment
    static constexpr int TMEM_COLS = GRU_P * N;                   // 512 / 256
    static_assert(SMEM_LAUNCH <= 227 * 1024, "shared memory");
    static_assert(TMEM_COLS <= 512, "tensor memory");
};

struct GruParams {
    int B, H, W;
    int horiz;                  // 1: taps along x (1x5 kernel), 0: taps along y (5x1)
    int n_across, n_along;      // tiles across / along the tap axis
    int n_tiles, n_super;       // B * n_across * n_along; ceil(n_tiles / GRU_P)
    const void* h;              // ActT, NHWC with pixel stride h_ps elements
    long long h_ps;
    const float* bias0;         // z|r pass: convz bias; q pass: convq bias (device, 128 floats)
    const float* bias1;         // z|r pass: convr bias
    void* z;                    // OpT [B*H*W][128] (workspace)
    void* rh;                   // OpT [B*H*W][128] (workspace): r * h, the q pass's first two K-blocks
    void* out;                  // ActT [B*H*W][128]: h'
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

// tile index -> (batch, first pixel across, first pixel along); tiles run across first
__device__ __forceinline__ void gru_tile(const GruParams& p, int t, int& b, int& a0, int& l0) {
    const int per_img = p.n_across * p.n_along;
    b = t / per_img;
    const int rem = t - b * per_img;
    l0 = (rem / p.n_across) * GRU_TL;
    a0 = (rem % p.n_across) * GRU_TA;
}

// MODE 0: z|r pass (N = 256), MODE 1: q pass (N = 128).  ActT: dtype of h and h'; OpT: 16-bit operand dtype.
// tm_a0: h (MODE 0) or r*h (MODE 1), tm_a1: context, tm_a2: motion -- each {128, across, along, B}, box {64, 16, 12, 1};
// tm_w: the pass's weight slabs {64, N, 30}, box {64, N, 1}.  All 128-byte swizzled.
template <int MODE, typename ActT, typename OpT>
__global__ void __launch_bounds__(GRU_THREADS, 1)
convgru_kernel(const __grid_constant__ CUtensorMap tm_a0, const __grid_constant__ CUtensorMap tm_a1,
               const __grid_constant__ CUtensorMap tm_a2, const __grid_constant__ CUtensorMap tm_w, const GruParams p) {
    constexpr int N = (MODE == 0) ? GRU_ZR_N : GRU_Q_N;
    using Cfg = GruCfg<N>;
    constexpr int WST = Cfg::W_STAGES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    const uint32_t s_a = ptx::smem_u32(smem + Cfg::SMEM_A);
    const uint32_t s_w = ptx::smem_u32(smem + Cfg::SMEM_W);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::SMEM_BAR);
    const uint32_t bar0 = ptx::smem_u32(bars);
    constexpr int A_FULL = 0, A_EMPTY = GRU_A_STAGES, W_FULL = 2 * GRU_A_STAGES, W_EMPTY = W_FULL + WST,
                  T_FULL = W_EMPTY + WST, T_EMPTY = T_FULL + 1;
    auto bar = [&](int i) { return bar0 + 8u * i; };
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(bars + T_EMPTY + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tensormap(&tm_a0);
        ptx::prefetch_tensormap(&tm_a1);
        ptx::prefetch_tensormap(&tm_a2);
        ptx::prefetch_tensormap(&tm_w);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < GRU_A_STAGES; ++i) {
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
                int b[GRU_P], a0[GRU_P], l0[GRU_P];
#pragma unroll
                for (int j = 0; j < GRU_P; ++j)      // a missing last tile reloads the one before (its stores are masked)
                    gru_tile(p, min(s * GRU_P + j, p.n_tiles - 1), b[j], a0[j], l0[j]);
                for (int kb = 0; kb < GRU_KB; ++kb, ++a_it) {
                    const uint32_t st = a_it % GRU_A_STAGES, ph = (a_it / GRU_A_STAGES) & 1;
                    ptx::mbar_wait(bar(A_EMPTY + st), ph ^ 1);
                    ptx::mbar_arrive_expect_tx(bar(A_FULL + st), Cfg::A_BYTES);
                    const CUtensorMap* m = kb < 2 ? &tm_a0 : kb < 4 ? &tm_a1 : &tm_a2;
#pragma unroll
                    for (int j = 0; j < GRU_P; ++j)
                        ptx::tma_load_4d(s_a + st * Cfg::A_BYTES + j * GRU_BOX_BYTES, m, bar(A_FULL + st), (kb & 1) * 64,
                                         a0[j], l0[j] - GRU_TAPS / 2, b[j]);
                    for (int t = 0; t < GRU_TAPS; ++t, ++w_it) {
                        const uint32_t ws = w_it % WST, wph = (w_it / WST) & 1;
                        ptx::mbar_wait(bar(W_EMPTY + ws), wph ^ 1);
                        ptx::mbar_arrive_expect_tx(bar(W_FULL + ws), Cfg::W_BYTES);
                        ptx::tma_load_3d(s_w + ws * Cfg::W_BYTES, &tm_w, bar(W_FULL + ws), 0, 0, kb * GRU_TAPS + t);
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================== MMA issuer (converged warp; tcgen05 under elect_one, see mcn_conv_sm100.cuh) =====================
        constexpr uint32_t idesc = ptx::umma_idesc(128, N, std::is_same<OpT, __nv_bfloat16>::value ? 1 : 0);
        uint32_t a_it = 0, w_it = 0, t_it = 0;
        for (int s = blockIdx.x; s < p.n_super; s += gridDim.x, ++t_it) {
            ptx::mbar_wait(bar(T_EMPTY), (t_it & 1) ^ 1);
            ptx::tc_fence_after();
            for (int kb = 0; kb < GRU_KB; ++kb, ++a_it) {
                const uint32_t st = a_it % GRU_A_STAGES, ph = (a_it / GRU_A_STAGES) & 1;
                ptx::mbar_wait(bar(A_FULL + st), ph);
                ptx::tc_fence_after();
                const uint64_t a_desc0 = ptx::umma_desc_k_sw128(s_a + st * Cfg::A_BYTES);
#pragma unroll 1
                for (int t = 0; t < GRU_TAPS; ++t, ++w_it) {
                    const uint32_t ws = w_it % WST, wph = (w_it / WST) & 1;
                    ptx::mbar_wait(bar(W_FULL + ws), wph);
                    ptx::tc_fence_after();
                    const uint64_t b_desc0 = ptx::umma_desc_k_sw128(s_w + ws * Cfg::W_BYTES);
                    if (ptx::elect_one()) {
#pragma unroll
                        for (int j = 0; j < GRU_P; ++j) {
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                ptx::umma_bf16(tmem_base + j * N,
                                               a_desc0 + ((j * GRU_BOX_BYTES + t * GRU_TAP_STEP + k * 32) >> 4),
                                               b_desc0 + ((k * 32) >> 4), idesc, (kb | t | k) != 0 ? 1u : 0u);
                        }
                        ptx::umma_commit(bar(W_EMPTY + ws));                        // slab free when these MMAs retire
                        if (t == GRU_TAPS - 1) ptx::umma_commit(bar(A_EMPTY + st));
                        if (t == GRU_TAPS - 1 && kb == GRU_KB - 1) ptx::umma_commit(bar(T_FULL));
                    }
                    __syncwarp();
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
            const int tile = s * GRU_P + j;
            int b, a0, l0;
            gru_tile(p, min(tile, p.n_tiles - 1), b, a0, l0);
            const int ai = a0 + (m & (GRU_TA - 1)), li = l0 + m / GRU_TA;
            const int x = p.horiz ? li : ai, y = p.horiz ? ai : li;
            const bool ok = (tile < p.n_tiles) && (x < p.W) && (y < p.H);
            const long long pix = (static_cast<long long>(b) * p.H + y) * p.W + x;
            const ActT* hp = static_cast<const ActT*>(p.h) + pix * p.h_ps;
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + j * N;
            ptx::mbar_wait(bar(T_FULL), t_it & 1);
            ptx::tc_fence_after();
#pragma unroll 1
            for (int c = 0; c < GRU_C; c += 16) {
                float v0[16], hv[16];
                if constexpr (MODE == 0) {
                    float v1[16];
                    ptx::tmem_ld_x16(taddr + c, v0);
                    ptx::tmem_ld_x16(taddr + GRU_C + c, v1);
                    ptx::tmem_ld_wait();
                    if (ok) {
                        GruVec<ActT>::load(hp + c, hv);
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            v0[i] = gru_sigmoid(v0[i] + __ldg(p.bias0 + c + i));           // z
                            v1[i] = gru_sigmoid(v1[i] + __ldg(p.bias1 + c + i)) * hv[i];   // r * h
                        }
                        GruVec<OpT>::store(static_cast<OpT*>(p.z) + pix * GRU_C + c, v0);
                        GruVec<OpT>::store(static_cast<OpT*>(p.rh) + pix * GRU_C + c, v1);
                    }
                } else {
                    ptx::tmem_ld_x16(taddr + c, v0);
                    ptx::tmem_ld_wait();
                    if (ok) {
                        float zv[16];
                        GruVec<ActT>::load(hp + c, hv);
                        GruVec<OpT>::load(static_cast<const OpT*>(p.z) + pix * GRU_C + c, zv);
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const float qv = tanhf(v0[i] + __ldg(p.bias0 + c + i));
                            v0[i] = (1.f - zv[i]) * hv[i] + zv[i] * qv;
                        }
                        GruVec<ActT>::store(static_cast<ActT*>(p.out) + pix * GRU_C + c, v0);
                    }
                }
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

}  // namespace rdvc
