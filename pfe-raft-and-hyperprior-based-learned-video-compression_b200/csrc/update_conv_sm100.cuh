// update_conv_sm100.cuh -- the rest of RAFT's update block (torchvision MotionEncoder, TV:raft.py:171-211, and FlowHead,
// TV:raft.py:272-285) as tcgen05 implicit GEMMs over NHWC 16-bit activations:
//
//   layer            kernel  Cin -> N      epilogue                        out
//   convcorr2        3x3     256 -> 192    bias, ReLU                      channels 0-191 of CF (B, h, w, 256), OpT
//   convflow2        3x3     128 -> 64     bias, ReLU                      channels 192-255 of CF, OpT
//   conv             3x3     256 -> 128    bias, ReLU; channels 126-127    MF (B, h, w, 128), ActT: the motion features
//                                          are the flow (N padded 126->128)  the recurrent block reads in place
//   flow_head.conv1  3x3     128 -> 256    bias, ReLU                      FH (B, h, w, 256), OpT
//   flow_head.conv2  3x3     256 -> 16     bias (2 real channels)          delta flow (B, 2, h, w) planes, ActT
//
// convflow1 (7x7, 2 -> 128) has 12.5 K MAC per pixel, 1 % of the update block's; it is a CUDA-core direct convolution
// at the end of this file (convflow1_kernel) with the same rounding points (16-bit operands, fp32 sums).
//
// Each concatenation of the stock module is a write into a channel slice: the epilogue stores at (pointer, pixel stride),
// and the next layer reads that buffer through a tensor map with the same pixel stride.
//
// Tile geometry.  A tile is 16 pixels along x by 8 rows (M = 128).  The activation map is {Cin, W, H, B} with the
// caller's pixel stride; one box of {64, 16, 8 + 2, 1} = 20 KB lands as 160 rows of 128 B (one SWIZZLE_128B row per
// pixel, row = y * 16 + x).  A 3x3 convolution loads one box per dx (shifted by dx - 1 in x, as mcn_conv does), and
// the A operand of tap (dy, dx) is that box shifted by dy rows = dy * 16 smem rows = two whole 1 KB swizzle atoms: a
// descriptor offset, no extra load.  Zero padding and every tail tile are TMA's out-of-bounds fill on the load side and
// a per-pixel mask on the store side.
//
// Weights stream from L2 in (k-block, tap) slabs of N x 64 (packed [k-block][dy * 3 + dx][N][64], rdvc_corr_update_conv_pack_weights),
// and every slab feeds UC_P = 2 pixel tiles (TMEM: 2 x N columns).
//
// Persistent, one CTA per SM, warp-specialised as convgru_sm100.cuh:
//   warp 0     TMA producer: per super-tile, k-block and dx the UC_P boxes (2-stage ring), then the 3 dy slabs (4 stages)
//   warp 1     tcgen05.mma issuer: M128 x N x K16, 16-bit operands, fp32 accumulators in TMEM (one per tile)
//   warp 2     TMEM allocator
//   warps 4-11 epilogue: warp 4 + e reads TMEM lane quarter e % 4 of tile e / 4; thread = pixel, 16 channels at a time
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>
#include <type_traits>

#include "convgru_sm100.cuh"
#include "ptx_sm100.cuh"

namespace rdvc {

constexpr int UC_TX = 16;                              // tile pixels along x
constexpr int UC_TY = 8;                               // tile rows
constexpr int UC_BOX_Y = UC_TY + 2;                    // 10: a box carries the vertical tap halo
constexpr int UC_BOX_BYTES = UC_TX * UC_BOX_Y * 128;   // 20 KB
constexpr int UC_DY_STEP = UC_TX * 128;                // 2 KB: one row = two swizzle atoms
constexpr int UC_P = 2;                                // pixel tiles per weight slab
constexpr int UC_A_STAGES = 2;
constexpr int UC_W_STAGES = 4;
constexpr int UC_THREADS = 128 + 8 * 32;

// epilogues (one instantiation each, chosen per layer)
constexpr int UC_EPI_RELU = 0;        // bias + ReLU -> OutT NHWC at (out, out_ps)
constexpr int UC_EPI_RELU_FLOW = 1;   // the same; channels N-2, N-1 are the flow (fp32, strided) rounded to OutT
constexpr int UC_EPI_FLOW2 = 2;       // bias only, channels 0-1 -> OutT planes (B, 2, H, W)

template <int N>
struct UcCfg {
    static constexpr int W_BYTES = N * 128;
    static constexpr int A_BYTES = UC_P * UC_BOX_BYTES;           // 40 KB
    static constexpr int SMEM_A = 0;
    static constexpr int SMEM_W = UC_A_STAGES * A_BYTES;
    static constexpr int SMEM_BAR = SMEM_W + UC_W_STAGES * W_BYTES;
    static constexpr int SMEM_TOTAL = SMEM_BAR + 256;
    static constexpr int SMEM_LAUNCH = SMEM_TOTAL + 1024;          // slack for 1024-byte alignment
    static constexpr int TMEM_COLS = UC_P * N <= 32 ? 32 : UC_P * N <= 64 ? 64 : UC_P * N <= 128 ? 128
                                   : UC_P * N <= 256 ? 256 : 512;
    static_assert(N % 16 == 0 && N >= 16 && N <= 256, "UMMA N");
    static_assert(SMEM_LAUNCH <= 227 * 1024, "shared memory");
    static_assert(UC_P * N <= 512, "tensor memory");
};

struct UcParams {
    int B, H, W;
    int n_kb;                   // 64-channel k-blocks of the input
    int n_tx, n_ty;             // tiles along x / y
    int n_tiles, n_super;       // B * n_tx * n_ty; ceil(n_tiles / UC_P)
    const float* bias;          // cout floats (device); channel c reads bias[min(c, cout - 1)]
    int cout;
    void* out;                  // OutT: NHWC with pixel stride out_ps, or (UC_EPI_FLOW2) planes (B, 2, H, W)
    long long out_ps;
    const float* flow;          // UC_EPI_RELU_FLOW: fp32 flow at flow[b * fs_b + c * fs_c + y * fs_y + x * fs_x]
    long long fs_b, fs_c, fs_y, fs_x;
};

__device__ __forceinline__ void uc_tile(const UcParams& p, int t, int& b, int& x0, int& y0) {
    const int per_img = p.n_tx * p.n_ty;
    b = t / per_img;
    const int rem = t - b * per_img;
    y0 = (rem / p.n_tx) * UC_TY;
    x0 = (rem % p.n_tx) * UC_TX;
}

// N: GEMM width (output channels, padded to a multiple of 16); OutT: output dtype; OpT: 16-bit operand dtype.
// tm_a: input {Cin, W, H, B}, box {64, 16, 10, 1}; tm_w: weight slabs {64, N, n_kb * 9}, box {64, N, 1}.  128-byte swizzle.
template <int N, int EPI, typename OutT, typename OpT>
__global__ void __launch_bounds__(UC_THREADS, 1)
update_conv_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_w, const UcParams p) {
    using Cfg = UcCfg<N>;
    constexpr int WST = UC_W_STAGES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    const uint32_t s_a = ptx::smem_u32(smem + Cfg::SMEM_A);
    const uint32_t s_w = ptx::smem_u32(smem + Cfg::SMEM_W);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::SMEM_BAR);
    const uint32_t bar0 = ptx::smem_u32(bars);
    constexpr int A_FULL = 0, A_EMPTY = UC_A_STAGES, W_FULL = 2 * UC_A_STAGES, W_EMPTY = W_FULL + WST,
                  T_FULL = W_EMPTY + WST, T_EMPTY = T_FULL + 1;
    auto bar = [&](int i) { return bar0 + 8u * i; };
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(bars + T_EMPTY + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tensormap(&tm_a);
        ptx::prefetch_tensormap(&tm_w);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < UC_A_STAGES; ++i) {
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
                int b[UC_P], x0[UC_P], y0[UC_P];
#pragma unroll
                for (int j = 0; j < UC_P; ++j)       // a missing last tile reloads the one before (its stores are masked)
                    uc_tile(p, min(s * UC_P + j, p.n_tiles - 1), b[j], x0[j], y0[j]);
                for (int kb = 0; kb < p.n_kb; ++kb) {
                    for (int dx = 0; dx < 3; ++dx, ++a_it) {
                        const uint32_t st = a_it % UC_A_STAGES, ph = (a_it / UC_A_STAGES) & 1;
                        ptx::mbar_wait(bar(A_EMPTY + st), ph ^ 1);
                        ptx::mbar_arrive_expect_tx(bar(A_FULL + st), Cfg::A_BYTES);
#pragma unroll
                        for (int j = 0; j < UC_P; ++j)
                            ptx::tma_load_4d(s_a + st * Cfg::A_BYTES + j * UC_BOX_BYTES, &tm_a, bar(A_FULL + st), kb * 64,
                                             x0[j] + dx - 1, y0[j] - 1, b[j]);
                        for (int dy = 0; dy < 3; ++dy, ++w_it) {
                            const uint32_t ws = w_it % WST, wph = (w_it / WST) & 1;
                            ptx::mbar_wait(bar(W_EMPTY + ws), wph ^ 1);
                            ptx::mbar_arrive_expect_tx(bar(W_FULL + ws), Cfg::W_BYTES);
                            ptx::tma_load_3d(s_w + ws * Cfg::W_BYTES, &tm_w, bar(W_FULL + ws), 0, 0, kb * 9 + dy * 3 + dx);
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
                for (int dx = 0; dx < 3; ++dx, ++a_it) {
                    const uint32_t st = a_it % UC_A_STAGES, ph = (a_it / UC_A_STAGES) & 1;
                    ptx::mbar_wait(bar(A_FULL + st), ph);
                    ptx::tc_fence_after();
                    const uint64_t a_desc0 = ptx::umma_desc_k_sw128(s_a + st * Cfg::A_BYTES);
#pragma unroll 1
                    for (int dy = 0; dy < 3; ++dy, ++w_it) {
                        const uint32_t ws = w_it % WST, wph = (w_it / WST) & 1;
                        ptx::mbar_wait(bar(W_FULL + ws), wph);
                        ptx::tc_fence_after();
                        const uint64_t b_desc0 = ptx::umma_desc_k_sw128(s_w + ws * Cfg::W_BYTES);
                        if (ptx::elect_one()) {
#pragma unroll
                            for (int j = 0; j < UC_P; ++j) {
#pragma unroll
                                for (int k = 0; k < 4; ++k)
                                    ptx::umma_bf16(tmem_base + j * N,
                                                   a_desc0 + ((j * UC_BOX_BYTES + dy * UC_DY_STEP + k * 32) >> 4),
                                                   b_desc0 + ((k * 32) >> 4), idesc, (kb | dx | dy | k) != 0 ? 1u : 0u);
                            }
                            ptx::umma_commit(bar(W_EMPTY + ws));                     // slab free when these MMAs retire
                            if (dy == 2) ptx::umma_commit(bar(A_EMPTY + st));
                            if (dy == 2 && dx == 2 && kb == p.n_kb - 1) ptx::umma_commit(bar(T_FULL));
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
            const int tile = s * UC_P + j;
            int b, x0, y0;
            uc_tile(p, min(tile, p.n_tiles - 1), b, x0, y0);
            const int x = x0 + (m & (UC_TX - 1)), y = y0 + m / UC_TX;
            const bool ok = (tile < p.n_tiles) && (x < p.W) && (y < p.H);
            const long long pix = (static_cast<long long>(b) * p.H + y) * p.W + x;
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + j * N;
            ptx::mbar_wait(bar(T_FULL), t_it & 1);
            ptx::tc_fence_after();
            if constexpr (EPI == UC_EPI_FLOW2) {
                float v[16];
                ptx::tmem_ld_x16(taddr, v);
                ptx::tmem_ld_wait();
                if (ok) {
                    const long long plane = static_cast<long long>(p.H) * p.W;
                    OutT* o = static_cast<OutT*>(p.out) + static_cast<long long>(b) * 2 * plane + (pix - b * plane);
                    o[0] = static_cast<OutT>(v[0] + __ldg(p.bias));
                    o[plane] = static_cast<OutT>(v[1] + __ldg(p.bias + min(1, p.cout - 1)));
                }
            } else {
                OutT* o = static_cast<OutT*>(p.out) + pix * p.out_ps;
#pragma unroll 1
                for (int c = 0; c < N; c += 16) {
                    float v[16];
                    ptx::tmem_ld_x16(taddr + c, v);
                    ptx::tmem_ld_wait();
                    if (ok) {
#pragma unroll
                        for (int i = 0; i < 16; ++i)
                            v[i] = fmaxf(v[i] + __ldg(p.bias + min(c + i, p.cout - 1)), 0.f);
                        if constexpr (EPI == UC_EPI_RELU_FLOW) {
                            if (c == N - 16) {
                                const float* f = p.flow + b * p.fs_b + y * p.fs_y + x * p.fs_x;
                                v[14] = __ldg(f);
                                v[15] = __ldg(f + p.fs_c);
                            }
                        }
                        GruVec<OutT>::store(o + c, v);
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

}  // namespace rdvc
