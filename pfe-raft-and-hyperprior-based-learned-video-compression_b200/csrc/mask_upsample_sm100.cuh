// mask_upsample_sm100.cuh -- the 1x1 convolution of RAFT's mask predictor (torchvision MaskPredictor.conv, 256 -> 576,
// TV:raft.py:311-334) as a persistent tcgen05 GEMM over the NHWC 16-bit output of convrelu (update_conv_kernel's
// flow_head.conv1 instantiation), with torchvision's convex 8x upsampling (TV:_utils.py:29-48) fused into its epilogue.
//
// Channel mapping (torchvision): mask channel k * 64 + i * 8 + j (tap k = ky * 3 + kx) weighs neighbour
// (y + ky - 1, x + kx - 1) for output pixel (8y + i, 8x + j).  N = 576 exceeds both UMMA's N <= 256 and TMEM's 512
// columns, so the host permutes the weight rows (rdvc_corr_mask_conv_pack_weights): GEMM row n = c * 144 + k * 16 + s
// holds stock channel k * 64 + 16c + s, c = 0..3 a chunk of 16 sub-pixels (sub-rows i = 2c and 2c + 1), s = 0..15.
// One chunk is one M128 x N144 accumulator; two chunks double-buffer in TMEM (columns 0 and 256), so the epilogue of
// chunk c overlaps the MMAs of chunk c + 1.  Column k * 16 + 8h + j of chunk c is tap k of sub-pixel (2c + h, j).
//
// Tile geometry.  A tile is 16 pixels along x by 8 rows (M = 128), the A operand four TMA boxes {64, 16, 8, 1} of
// the 256-channel input {C, W, H, B} at the caller's pixel stride (one SWIZZLE_128B row per pixel, row = y * 16 + x):
// 64 KB, double-buffered.  Tails are TMA's out-of-bounds fill on the load side and a per-pixel mask on the store side.
// Weights stream from L2 in (chunk, k-block) slabs of 144 x 64 (packed [c][k-block][144][64], 18 KB) through a
// 4-stage ring; every tile reads all 16 slabs (288 KB).
//
// Persistent, one CTA per SM, warp-specialised as update_conv_sm100.cuh:
//   warp 0     TMA producer: per tile the 4 A boxes, then the 16 weight slabs
//   warp 1     tcgen05.mma issuer (converged warp, tcgen05 under elect_one): M128 x N144 x K16, fp32 accumulators
//   warp 2     TMEM allocator
//   warps 4-11 epilogue: warp 4 + e reads TMEM lane quarter e % 4 and sub-row half h = e / 4 of every chunk: thread =
//              pixel, 9 taps x 8 sub-pixels.
// Epilogues:
//   MU_EPI_UPSAMPLED  logit = multiplier * (acc + bias) in fp32; per sub-pixel a softmax over its 9 logits (max
//                     subtracted); out = sum_k p_k * 8 * flow[y + ky - 1, x + kx - 1] with the fp32 flow, neighbours
//                     outside the image zero but weighted (F.unfold(padding=1)); out (B, 2, 8H, 8W) fp32, two
//                     32-byte runs per thread and sub-row.
//   MU_EPI_MASK       multiplier * (acc + bias) in OutT to a contiguous (B, 576, H, W) in stock channel order.
// No atomics: every output element is written once by one thread, so results are deterministic and independent of
// the batch composition.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>
#include <type_traits>

#include "ptx_sm100.cuh"

namespace rdvc {

constexpr int MU_CIN = 256;
constexpr int MU_COUT = 576;
constexpr int MU_KB = MU_CIN / 64;                        // 4 k-blocks
constexpr int MU_CHUNKS = 4;
constexpr int MU_NC = MU_COUT / MU_CHUNKS;                // 144: GEMM width of one chunk
constexpr int MU_TX = 16;
constexpr int MU_TY = 8;
constexpr int MU_BOX_BYTES = MU_TX * MU_TY * 128;         // 16 KB
constexpr int MU_A_BYTES = MU_KB * MU_BOX_BYTES;          // 64 KB
constexpr int MU_W_BYTES = MU_NC * 128;                   // 18 KB
constexpr int MU_A_STAGES = 2;
constexpr int MU_W_STAGES = 4;
constexpr int MU_SMEM_A = 0;
constexpr int MU_SMEM_W = MU_A_STAGES * MU_A_BYTES;
constexpr int MU_SMEM_BAR = MU_SMEM_W + MU_W_STAGES * MU_W_BYTES;
constexpr int MU_SMEM_LAUNCH = MU_SMEM_BAR + 256 + 1024;  // barriers + slack for 1024-byte alignment
constexpr int MU_TMEM_COLS = 512;
constexpr int MU_TMEM_BUF = 256;                          // column offset of the second chunk buffer
constexpr int MU_THREADS = 128 + 8 * 32;
static_assert(MU_SMEM_LAUNCH <= 227 * 1024, "shared memory");
static_assert(MU_TMEM_BUF + MU_NC <= MU_TMEM_COLS, "tensor memory");
static_assert(MU_W_BYTES % 1024 == 0, "weight slabs must keep the 1 KB swizzle-atom alignment");

constexpr int MU_EPI_UPSAMPLED = 0;
constexpr int MU_EPI_MASK = 1;

struct MuParams {
    int B, H, W;
    int n_tx, n_ty, n_tiles;
    const float* bias;          // 576 floats in GEMM row order (rdvc_corr_mask_conv_pack_weights)
    float multiplier;
    void* out;                  // UPSAMPLED: fp32 (B, 2, 8H, 8W); MASK: OutT (B, 576, H, W)
    const float* flow;          // UPSAMPLED: flow[b * fs_b + c * fs_c + y * fs_y + x * fs_x]
    long long fs_b, fs_c, fs_y, fs_x;
};

__device__ __forceinline__ void mu_tile(const MuParams& p, int t, int& b, int& x0, int& y0) {
    const int per_img = p.n_tx * p.n_ty;
    b = t / per_img;
    const int rem = t - b * per_img;
    y0 = (rem / p.n_tx) * MU_TY;
    x0 = (rem % p.n_tx) * MU_TX;
}

// 32 lanes x 8 consecutive fp32 columns: thread i <- lane (base_lane + i), v[j] <- column j.
__device__ __forceinline__ void mu_tmem_ld_x8(uint32_t taddr, float* v) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

// One thread's share of a chunk: v[k][j] = accumulator of tap k, sub-pixel (i, j) of pixel (b, y, x); bias_n = the GEMM
// row of (k = 0, j = 0).  f0 / f1: 8 * flow of the 3x3 neighbourhood (UPSAMPLED).
template <int EPI, typename OutT>
__device__ __forceinline__ void mu_store(const MuParams& p, float (&v)[9][8], const float (&f0)[9], const float (&f1)[9],
                                         int b, int x, int y, int i, int bias_n) {
    const float* bias = p.bias + bias_n;
#pragma unroll
    for (int k = 0; k < 9; ++k)
#pragma unroll
        for (int j = 0; j < 8; ++j) v[k][j] = (v[k][j] + __ldg(bias + k * 16 + j)) * p.multiplier;
    if constexpr (EPI == MU_EPI_UPSAMPLED) {
        float o0[8], o1[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {                 // TV:_utils.py:40-44: softmax over the taps, then the convex sum
            float mx = v[0][j];
#pragma unroll
            for (int k = 1; k < 9; ++k) mx = fmaxf(mx, v[k][j]);
            float s = 0.f, a0 = 0.f, a1 = 0.f;
#pragma unroll
            for (int k = 0; k < 9; ++k) {
                const float w = __expf(v[k][j] - mx);
                s += w;
                a0 = fmaf(w, f0[k], a0);
                a1 = fmaf(w, f1[k], a1);
            }
            const float inv = 1.f / s;
            o0[j] = a0 * inv;
            o1[j] = a1 * inv;
        }
        // TV:_utils.py:46: out[b, ch, 8y + i, 8x + j]; 8 consecutive floats, 32-byte aligned
        const long long W8 = 8LL * p.W, plane = 64LL * p.H * p.W;
        float* o = static_cast<float*>(p.out) + 2LL * b * plane + (8LL * y + i) * W8 + 8LL * x;
        float4* d0 = reinterpret_cast<float4*>(o);
        float4* d1 = reinterpret_cast<float4*>(o + plane);
        d0[0] = make_float4(o0[0], o0[1], o0[2], o0[3]);
        d0[1] = make_float4(o0[4], o0[5], o0[6], o0[7]);
        d1[0] = make_float4(o1[0], o1[1], o1[2], o1[3]);
        d1[1] = make_float4(o1[4], o1[5], o1[6], o1[7]);
    } else {
        const long long plane = static_cast<long long>(p.H) * p.W;
        OutT* o = static_cast<OutT*>(p.out) + static_cast<long long>(b) * MU_COUT * plane + static_cast<long long>(y) * p.W + x;
#pragma unroll
        for (int k = 0; k < 9; ++k)
#pragma unroll
            for (int j = 0; j < 8; ++j) o[(k * 64 + i * 8 + j) * plane] = static_cast<OutT>(v[k][j]);
    }
}

// EPI: MU_EPI_*; OutT: MASK's output dtype (unused by UPSAMPLED); OpT: 16-bit operand dtype.
// tm_a: input {256, W, H, B}, box {64, 16, 8, 1}; tm_w: weight slabs {64, 144, 16}, box {64, 144, 1}.  128-byte swizzle.
template <int EPI, typename OutT, typename OpT>
__global__ void __launch_bounds__(MU_THREADS, 1)
mask_upsample_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_w, const MuParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    const uint32_t s_a = ptx::smem_u32(smem + MU_SMEM_A);
    const uint32_t s_w = ptx::smem_u32(smem + MU_SMEM_W);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + MU_SMEM_BAR);
    const uint32_t bar0 = ptx::smem_u32(bars);
    constexpr int A_FULL = 0, A_EMPTY = MU_A_STAGES, W_FULL = 2 * MU_A_STAGES, W_EMPTY = W_FULL + MU_W_STAGES,
                  T_FULL = W_EMPTY + MU_W_STAGES, T_EMPTY = T_FULL + 2, N_BARS = T_EMPTY + 2;
    auto bar = [&](int i) { return bar0 + 8u * i; };
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(bars + N_BARS);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tensormap(&tm_a);
        ptx::prefetch_tensormap(&tm_w);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < MU_A_STAGES; ++i) {
            ptx::mbar_init(bar(A_FULL + i), 1);
            ptx::mbar_init(bar(A_EMPTY + i), 1);
        }
        for (int i = 0; i < MU_W_STAGES; ++i) {
            ptx::mbar_init(bar(W_FULL + i), 1);
            ptx::mbar_init(bar(W_EMPTY + i), 1);
        }
        for (int i = 0; i < 2; ++i) {
            ptx::mbar_init(bar(T_FULL + i), 1);
            ptx::mbar_init(bar(T_EMPTY + i), 8);
        }
        ptx::fence_mbar_init();
    }
    if (warp == 2) {
        ptx::tmem_alloc(ptx::smem_u32(const_cast<uint32_t*>(tmem_slot)), MU_TMEM_COLS);
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
            for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x, ++a_it) {
                int b, x0, y0;
                mu_tile(p, t, b, x0, y0);
                const uint32_t st = a_it % MU_A_STAGES, ph = (a_it / MU_A_STAGES) & 1;
                ptx::mbar_wait(bar(A_EMPTY + st), ph ^ 1);
                ptx::mbar_arrive_expect_tx(bar(A_FULL + st), MU_A_BYTES);
#pragma unroll
                for (int kb = 0; kb < MU_KB; ++kb)
                    ptx::tma_load_4d(s_a + st * MU_A_BYTES + kb * MU_BOX_BYTES, &tm_a, bar(A_FULL + st), kb * 64, x0, y0, b);
                for (int slab = 0; slab < MU_CHUNKS * MU_KB; ++slab, ++w_it) {
                    const uint32_t ws = w_it % MU_W_STAGES, wph = (w_it / MU_W_STAGES) & 1;
                    ptx::mbar_wait(bar(W_EMPTY + ws), wph ^ 1);
                    ptx::mbar_arrive_expect_tx(bar(W_FULL + ws), MU_W_BYTES);
                    ptx::tma_load_3d(s_w + ws * MU_W_BYTES, &tm_w, bar(W_FULL + ws), 0, 0, slab);
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================== MMA issuer (converged warp; tcgen05 under elect_one) =====================
        constexpr uint32_t idesc = ptx::umma_idesc(128, MU_NC, std::is_same<OpT, __nv_bfloat16>::value ? 1 : 0);
        uint32_t a_it = 0, w_it = 0, c_it = 0;
        for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x, ++a_it) {
            const uint32_t st = a_it % MU_A_STAGES, ph = (a_it / MU_A_STAGES) & 1;
            ptx::mbar_wait(bar(A_FULL + st), ph);
            ptx::tc_fence_after();
            const uint64_t a_desc0 = ptx::umma_desc_k_sw128(s_a + st * MU_A_BYTES);
#pragma unroll 1
            for (int c = 0; c < MU_CHUNKS; ++c, ++c_it) {
                const uint32_t tb = c_it & 1, tph = (c_it >> 1) & 1;
                ptx::mbar_wait(bar(T_EMPTY + tb), tph ^ 1);
                ptx::tc_fence_after();
#pragma unroll 1
                for (int kb = 0; kb < MU_KB; ++kb, ++w_it) {
                    const uint32_t ws = w_it % MU_W_STAGES, wph = (w_it / MU_W_STAGES) & 1;
                    ptx::mbar_wait(bar(W_FULL + ws), wph);
                    ptx::tc_fence_after();
                    const uint64_t b_desc0 = ptx::umma_desc_k_sw128(s_w + ws * MU_W_BYTES);
                    if (ptx::elect_one()) {
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            ptx::umma_bf16(tmem_base + tb * MU_TMEM_BUF, a_desc0 + ((kb * MU_BOX_BYTES + k * 32) >> 4),
                                           b_desc0 + ((k * 32) >> 4), idesc, (kb | k) != 0 ? 1u : 0u);
                        ptx::umma_commit(bar(W_EMPTY + ws));                       // slab free when these MMAs retire
                        if (kb == MU_KB - 1) {
                            ptx::umma_commit(bar(T_FULL + tb));
                            if (c == MU_CHUNKS - 1) ptx::umma_commit(bar(A_EMPTY + st));
                        }
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
        const int h = e >> 2;                // sub-row half: sub-rows 2c + h
        const int m = q * 32 + lane;         // GEMM row = pixel of the tile
        uint32_t c_it = 0;
        for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x) {
            int b, x0, y0;
            mu_tile(p, t, b, x0, y0);
            const int x = x0 + (m & (MU_TX - 1)), y = y0 + m / MU_TX;
            const bool ok = (x < p.W) && (y < p.H);
            // UPSAMPLED: 8 * flow of the 3x3 neighbourhood, zero outside the image (TV:_utils.py:43 unfold, padding 1)
            float f0[9] = {}, f1[9] = {};
            if constexpr (EPI == MU_EPI_UPSAMPLED) {
                const float* fb = p.flow + b * p.fs_b;
#pragma unroll
                for (int k = 0; k < 9; ++k) {
                    const int yy = y + k / 3 - 1, xx = x + k % 3 - 1;
                    if (ok && yy >= 0 && yy < p.H && xx >= 0 && xx < p.W) {
                        const float* f = fb + yy * p.fs_y + xx * p.fs_x;
                        f0[k] = 8.f * __ldg(f);
                        f1[k] = 8.f * __ldg(f + p.fs_c);
                    }
                }
            }
#pragma unroll 1
            for (int c = 0; c < MU_CHUNKS; ++c, ++c_it) {
                const uint32_t tb = c_it & 1, tph = (c_it >> 1) & 1;
                const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + tb * MU_TMEM_BUF + 8 * h;
                ptx::mbar_wait(bar(T_FULL + tb), tph);
                __syncwarp();
                ptx::tc_fence_after();
                float v[9][8];                                    // [tap][sub-pixel j] of sub-row i = 2c + h
#pragma unroll
                for (int k = 0; k < 9; ++k) mu_tmem_ld_x8(taddr + k * 16, v[k]);
                ptx::tmem_ld_wait();
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(bar(T_EMPTY + tb));     // the buffer is back to the MMA warp
                if (ok) mu_store<EPI, OutT>(p, v, f0, f1, b, x, y, 2 * c + h, c * MU_NC + 8 * h);
            }
        }
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 2) ptx::tmem_dealloc(tmem_base, MU_TMEM_COLS);
}

}  // namespace rdvc
