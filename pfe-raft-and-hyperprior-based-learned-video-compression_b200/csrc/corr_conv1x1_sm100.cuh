// corr_conv1x1_sm100.cuh -- "next" row f-1: the 1x1 convolution + bias + ReLU that consumes the correlation
// features (MotionEncoder.convcorr1, TV:raft.py:185 construction, :202 call), as a tcgen05 GEMM over the K-major
// feature rows the lookup kernel emits (corr_lookup.cuh, LKP_OUT_KM_*):
//
//   out[b, n, y, x] = act( sum_k feat[b*N + y*w + x][k] * Wp[n][k] + bias[n] ),   n < cout <= 256
//
// feat: bf16 / fp16, chunk-major [kp / 8][rows][8] (kp = rdvc_corr_feat_pitch, 352 for 4 levels x radius 4; see
// corr_lookup.cuh), Wp: the convolution's weight permuted to the lookup's feature order and zero-padded
// (rdvc_conv1x1_pack_weights), fp32 accumulation in TMEM, bias + ReLU in the epilogue, result written ONCE as
// the (B, cout, h, w) tensor convcorr2 reads -- the (B, 324, h, w) fp32 lookup tensor (42 MB per iteration at
// 1080p) and its re-read by cuDNN are gone.
//
// Operand layouts in shared memory.  A (features): a TMA box of 8 chunks x 128 rows x 16 bytes lands as
// [chunk][row][16 B], i.e. core matrices of 8 rows x 16 bytes stored contiguously -- the UN-SWIZZLED K-major
// canonical layout of tcgen05 (descriptor layout type 0, stride byte offset = 128 between 8-row groups, leading
// byte offset = 2048 between the two 8-element chunks of a K = 16 step).  B (weights): [cout / 2][64] rows with
// the 128-byte swizzle, as in the build kernel.
//
// Shape of the computation at 1080p: M = 32640 pixels, N = 256, K = 352: 5.9 GFLOP (3.5 us at the bf16 peak),
// 23 MB of features in (L2-resident: the lookup wrote them a moment ago), 33 MB fp32 out (5.1 us at the HBM
// peak).  What has to be avoided is re-streaming the 176 KB weight matrix per 128-pixel tile through L2 -> SM
// (the feed ceiling measured on the MCN layers, ~7 TB/s): so CTA PAIRS (tcgen05 cta_group::2, M = 256): each
// CTA keeps only its HALF of the output channels' weights (6 k-blocks x 16 KB = 96 KB) stationary for the
// whole kernel and streams its own 128 pixel rows through a 4-stage ring.  Every CTA owns a contiguous pixel
// range (total / grid, rounded to 32), so the output bytes per SM are equal.
//
// The epilogue is the critical path (time stamps, tools/exp_conv1x1_timeline.py: both tiles' MMAs are done ~7 us
// into the kernel; the rest is getting 2 x 128 KB of results out of each SM), and it went through four forms:
// one 4-byte store per lane and channel (128-byte requests: ~26 GB/s per SM whatever the warp count), a
// release-ordered remote arrive per tile that compiled to MEMBAR.ALL.GPU (waited for every store in flight),
// quads of lanes transposing 4 x 4 with shuffles (512-byte requests, but ~300 instructions per 32 channels), and
// now a per-warp 4 KB shared-memory transpose: 32 conflict-free st.shared, then every lane reads FOUR consecutive
// pixels of one channel (ld.shared.v4), adds the bias, applies ReLU and writes 16 bytes -- a warp-wide store
// covers four whole 128-byte lines of the (B, cout, h, w) tensor.
//
// Protocol as in corr_build2_sm100.cuh ("leader" = cluster rank 0; barriers at the same offset in both CTAs):
//   W_FULL, A_FULL[s]   leader only; armed by the leader's producer for BOTH CTAs' bytes, completed by each
//                       CTA's TMA loads.
//   A_EMPTY[s], T_FULL[a]  both CTAs, tcgen05.commit multicast from the leader's issuing warp.
//   T_EMPTY[a]          leader only, 16 arrivals (every epilogue warp of both CTAs).
// The issuing warp runs converged; only the tcgen05 instructions sit under elect_one().
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>

#include "ptx_sm100.cuh"

namespace rdvc {

constexpr int C1_BLOCK_M = 128;                 // pixel rows per CTA and tile
constexpr int C1_BLOCK_K = 64;                  // 16-bit elements per 128-byte swizzle row
constexpr int C1_MAX_KB = 6;                    // K <= 384
constexpr int C1_MAX_COUT = 256;
constexpr int C1_A_STAGES = 4;                  // 16 KB each (a tile is 6 k-blocks; the MMAs are far off the critical path)
constexpr int C1_A_STAGE_BYTES = C1_BLOCK_M * C1_BLOCK_K * 2;            // 16 KB
constexpr int C1_W_SLAB_BYTES = (C1_MAX_COUT / 2) * C1_BLOCK_K * 2;      // 16 KB: half the channels x one k-block
constexpr int C1_EPI_WARPS = 16;               // four per TMEM lane quarter, a quarter of the channels each
constexpr int C1_THREADS = 128 + C1_EPI_WARPS * 32;
constexpr int C1_SMEM_W = 0;
constexpr int C1_SMEM_A = C1_SMEM_W + C1_MAX_KB * C1_W_SLAB_BYTES;       // 98304
constexpr int C1_STG_BYTES = 32 * 32 * 4;       // per epilogue warp: 32 channels x 32 pixels fp32, the transpose buffer
constexpr int C1_SMEM_STG = C1_SMEM_A + C1_A_STAGES * C1_A_STAGE_BYTES;  // 163840
constexpr int C1_SMEM_BIAS = C1_SMEM_STG + C1_EPI_WARPS * C1_STG_BYTES;  // 229376
constexpr int C1_SMEM_BAR = C1_SMEM_BIAS + C1_MAX_COUT * 4;
constexpr int C1_SMEM_TOTAL = C1_SMEM_BAR + 256;
constexpr int C1_SMEM_LAUNCH = C1_SMEM_TOTAL + 1024;                     // slack for 1024-byte alignment

struct Conv1x1Params {
    void* out;              // (B, cout, n_pix) OutT
    const float* bias;      // cout floats on the device, or nullptr
    long long m_total;      // B * n_pix feature rows
    int n_pix;              // h * w
    int cout;               // multiple of 32, <= 256
    int kp;                 // feature-row pitch in elements (multiple of 16, <= 384)
    int rows_per_cta;       // pixel rows owned by one CTA (multiple of 32)
    int tiles_per_cta;      // ceil(rows_per_cta / 128)
    int relu;
    int vec4;               // n_pix % 4 == 0 and `out` 16-byte aligned: quads of lanes transpose 4 x 4 and store 4 pixels at once
    int ab_format;          // tcgen05 kind::f16 operand format: 1 = bf16, 0 = fp16
    unsigned long long* dbg_timeline;   // RDVC_EXPERIMENTS builds only: 16 globaltimer stamps per CTA (nullptr = off)
    int dbg_flags;                      // RDVC_EXPERIMENTS builds only: 1 = no output stores, 2 = no TMEM reads (timing)
    long long out_ps;                   // NHWC instantiations: `out` is (B*h*w) pixels of out_ps elements, channel stride 1
};

#ifdef RDVC_EXPERIMENTS
__device__ __forceinline__ void c1_stamp(const Conv1x1Params& p, int slot) {
    if (p.dbg_timeline) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t) :: "memory");
        p.dbg_timeline[blockIdx.x * 16 + slot] = t;
    }
}
#define C1_STAMP(slot) c1_stamp(p, slot)
#define C1_DBG(bit) ((p.dbg_flags & (bit)) != 0)
#else
#define C1_STAMP(slot) ((void)0)
#define C1_DBG(bit) false
#endif

// four consecutive pixels of one channel -> one 16-byte (fp32) / 8-byte (16-bit) store
__device__ __forceinline__ void c1_store4(float* dst, float a, float b, float c, float d) {
    *reinterpret_cast<float4*>(dst) = make_float4(a, b, c, d);
}
__device__ __forceinline__ void c1_store4(__half* dst, float a, float b, float c, float d) {
    const __half2 lo = __floats2half2_rn(a, b), hi = __floats2half2_rn(c, d);
    *reinterpret_cast<uint2*>(dst) = make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
}
__device__ __forceinline__ void c1_store4(__nv_bfloat16* dst, float a, float b, float c, float d) {
    const __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
    *reinterpret_cast<uint2*>(dst) = make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
}

__device__ __forceinline__ void sts_f32(uint32_t addr, float v) {
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ float lds_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}
// Loads of shared memory that is READ-ONLY after the kernel's set-up barrier (the bias): not volatile, no memory clobber,
// so the compiler may hoist and batch them instead of issuing load -> wait -> use one at a time (the encoder tail's
// epilogue spent 2.2 us per tile on 128 such chains).
__device__ __forceinline__ float lds_ro_f32(uint32_t addr) {
    float v;
    asm("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ float4 lds_ro_f32x4(uint32_t addr) {
    float4 v;
    asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ float4 lds_f32x4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
    return v;
}

template <typename OutT> __device__ __forceinline__ OutT c1_cvt(float x);
template <> __device__ __forceinline__ float c1_cvt<float>(float x) { return x; }
template <> __device__ __forceinline__ __half c1_cvt<__half>(float x) { return __float2half_rn(x); }
template <> __device__ __forceinline__ __nv_bfloat16 c1_cvt<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }

// 16 values -> one pixel's 16 consecutive 16-bit channels: two 16-byte stores
template <typename OutT>
__device__ __forceinline__ void c1_store16(OutT* dst, const float* v) {
    static_assert(sizeof(OutT) == 2, "NHWC output is 16-bit");
    uint32_t w[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const OutT lo = c1_cvt<OutT>(v[2 * j]), hi = c1_cvt<OutT>(v[2 * j + 1]);
        w[j] = static_cast<uint32_t>(*reinterpret_cast<const uint16_t*>(&lo)) |
               (static_cast<uint32_t>(*reinterpret_cast<const uint16_t*>(&hi)) << 16);
    }
    reinterpret_cast<uint4*>(dst)[0] = make_uint4(w[0], w[1], w[2], w[3]);
    reinterpret_cast<uint4*>(dst)[1] = make_uint4(w[4], w[5], w[6], w[7]);
}

// grid: an even number of CTAs (clusters of 2); block: C1_THREADS; dynamic smem: C1_SMEM_LAUNCH.
// tm_a: features as a {64 (8 rows x 8 elements), rows / 8, kp / 8} tensor, box {64, 16, 8}, no swizzle;
// tm_w: packed weights {kpw, cout, 1}, box {64, cout / 2, 1}, 128-byte swizzle.
// NHWC: the result goes out as (pixel, channel) rows of p.out_ps 16-bit elements straight from the accumulator (thread =
// pixel, 16-byte stores, no transpose): the layout the 3x3 convolutions that follow read (tap_conv_sm100.cuh).
template <typename OutT, bool NHWC>
__device__ __forceinline__ void corr_conv1x1_body(const CUtensorMap& tm_a, const CUtensorMap& tm_w, const Conv1x1Params p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(
        (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
    const uint32_t s_w = ptx::smem_u32(smem + C1_SMEM_W);
    const uint32_t s_a = ptx::smem_u32(smem + C1_SMEM_A);
    const uint32_t s_stg = ptx::smem_u32(smem + C1_SMEM_STG);
    // the bias is read with explicit ld.shared: through the generic pointer the compiler emitted LD.E (generic loads, a
    // long-scoreboard wait in front of every FADD of the epilogue -- half of its samples in the profile)
    const uint32_t s_bias = ptx::smem_u32(smem + C1_SMEM_BIAS);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C1_SMEM_BAR);
    const uint32_t bar0 = ptx::smem_u32(bars);
    constexpr int A_FULL = 0, A_EMPTY = C1_A_STAGES, W_FULL = 2 * C1_A_STAGES, T_FULL = W_FULL + 1, T_EMPTY = T_FULL + 2;
    auto bar = [&](int i) { return bar0 + 8u * i; };
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(bars + T_EMPTY + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = ptx::cluster_ctarank();
    const bool leader = (rank == 0);

    if (warp == 0 && lane == 0) {
        C1_STAMP(0);                                   // kernel entry
        ptx::prefetch_tensormap(&tm_a);
        ptx::prefetch_tensormap(&tm_w);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < C1_A_STAGES; ++i) {
            ptx::mbar_init(bar(A_FULL + i), 1);
            ptx::mbar_init(bar(A_EMPTY + i), 1);
        }
        ptx::mbar_init(bar(W_FULL), 1);
        for (int i = 0; i < 2; ++i) {
            ptx::mbar_init(bar(T_FULL + i), 1);
            ptx::mbar_init(bar(T_EMPTY + i), 2 * C1_EPI_WARPS);
        }
        ptx::fence_mbar_init();
    }
    if (warp == 2) {
        ptx::tmem_alloc_2sm(ptx::smem_u32(const_cast<uint32_t*>(tmem_slot)), 512);
        ptx::tmem_relinquish_2sm();
    }
    if (warp >= 4 && static_cast<int>(threadIdx.x) - 128 < p.cout)       // one element per thread: ONE global round trip
        sts_f32(s_bias + (threadIdx.x - 128) * 4, p.bias ? __ldg(p.bias + (threadIdx.x - 128)) : 0.f);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::cluster_sync_relaxed_arrive();   // the peer's barriers are initialised (and fenced) before anyone signals them
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (warp == 0 && lane == 0) C1_STAMP(1);           // set-up done (barriers, TMEM, cluster sync)

    const int n_kb = (p.kp + C1_BLOCK_K - 1) / C1_BLOCK_K;      // k-blocks (the last may be partial)
    const int n_ksteps = p.kp / 16;                              // UMMA k-steps over the whole K
    const int half = p.cout / 2;                                 // output channels whose weights this CTA holds
    const long long row_base = static_cast<long long>(blockIdx.x) * p.rows_per_cta;
    const int n_tiles = p.tiles_per_cta;

    if (warp == 0) {
        // ===================== TMA producer (both CTAs) =====================
        if (lane == 0) {
            if (leader) ptx::mbar_arrive_expect_tx(bar(W_FULL), 2u * n_kb * half * 128u);
            for (int kb = 0; kb < n_kb; ++kb)
                ptx::tma_load_3d_2sm(s_w + kb * C1_W_SLAB_BYTES, &tm_w, bar(W_FULL), kb * C1_BLOCK_K,
                                     static_cast<int>(rank) * half, 0);
            uint32_t a_it = 0;
            for (int t = 0; t < n_tiles; ++t) {
                long long m0 = row_base + static_cast<long long>(t) * C1_BLOCK_M;
                if (m0 > p.m_total - 1) m0 = (p.m_total - 1) & ~7LL;   // a range past the end: rows are masked in the epilogue
                for (int kb = 0; kb < n_kb; ++kb, ++a_it) {
                    const uint32_t st = a_it % C1_A_STAGES, ph = (a_it / C1_A_STAGES) & 1;
                    ptx::mbar_wait(bar(A_EMPTY + st), ph ^ 1);
                    if (leader) ptx::mbar_arrive_expect_tx(bar(A_FULL + st), 2 * C1_A_STAGE_BYTES);
                    // rows m0 .. m0 + 127 (m0 is a multiple of 8: ranges are multiples of 32), chunks 8 kb .. 8 kb + 7
                    ptx::tma_load_3d_2sm(s_a + st * C1_A_STAGE_BYTES, &tm_a, bar(A_FULL + st), 0,
                                         static_cast<int>(m0 >> 3), kb * (C1_BLOCK_K / 8));
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ===================== MMA issuer (leader CTA only; converged warp, tcgen05 under elect_one) =====================
        if (leader) {
            const uint32_t idesc = ptx::umma_idesc(2 * C1_BLOCK_M, p.cout, p.ab_format);
            ptx::mbar_wait(bar(W_FULL), 0);
            ptx::tc_fence_after();
            if (lane == 0) C1_STAMP(2);                // weights landed
            const uint64_t b_desc0 = ptx::umma_desc_k_sw128(s_w);
            uint32_t a_it = 0;
            for (int t = 0; t < n_tiles; ++t) {
                const uint32_t acc = t & 1, acc_ph = (t >> 1) & 1;
                ptx::mbar_wait(bar(T_EMPTY + acc), acc_ph ^ 1);
                ptx::tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * C1_MAX_COUT;
                for (int kb = 0; kb < n_kb; ++kb, ++a_it) {
                    const uint32_t st = a_it % C1_A_STAGES, ph = (a_it / C1_A_STAGES) & 1;
                    ptx::mbar_wait(bar(A_FULL + st), ph);
                    ptx::tc_fence_after();
                    if (lane == 0 && kb == 0) C1_STAMP(3 + t);          // first feature block of tile t landed (slots 3, 4)
                    if (lane == 0 && kb == n_kb - 1) C1_STAMP(5 + t);   // last one (slots 5, 6)
                    const uint64_t a_desc0 = ptx::umma_desc_k_nosw(s_a + st * C1_A_STAGE_BYTES, 2048, 128);
                    const int ks = n_ksteps - kb * 4;            // k-steps left: 4 for a full block
                    if (ptx::elect_one()) {
                        const uint64_t b_desc = b_desc0 + ((kb * C1_W_SLAB_BYTES) >> 4);
                        if (ks >= 4) {                            // a full k-block: four MMAs back to back
#pragma unroll
                            for (int k = 0; k < 4; ++k)
                                ptx::umma_bf16_2sm(d_tmem, a_desc0 + ((k * 4096) >> 4), b_desc + ((k * 32) >> 4), idesc,
                                                   (kb | k) != 0 ? 1u : 0u);          // A: two 2 KB chunk planes per k-step
                        } else {                                  // the partial last block (K = 352: two k-steps)
                            for (int k = 0; k < ks; ++k)
                                ptx::umma_bf16_2sm(d_tmem, a_desc0 + ((k * 4096) >> 4), b_desc + ((k * 32) >> 4), idesc,
                                                   (kb | k) != 0 ? 1u : 0u);
                        }
                        ptx::umma_commit_2sm(bar(A_EMPTY + st), 3);                   // ring slot free in both CTAs
                        if (kb == n_kb - 1) ptx::umma_commit_2sm(bar(T_FULL + acc), 3);  // accumulator ready in both
                    }
                    __syncwarp();
                }
            }
        }
        __syncwarp();
    } else if (warp >= 4) {
        // ===================== epilogue (both CTAs) =====================
        // warp 4 + e: TMEM lane quarter q = e % 4 (pixel rows 32 q .. 32 q + 31 of the tile), channel group e / 4
        // (a quarter of the channels, rounded up to 16).  Out of TMEM a thread is one pixel with 32 channels in
        // registers; the warp's 4 KB buffer turns that into "four consecutive pixels of one channel" per lane (see
        // the file header).  Shapes whose pixel count is not a multiple of 4 store one value per lane instead.
        const int e = warp - 4;
        const int q = e & 3;
        const int cpg = ((p.cout + 3) / 4 + 15) / 16 * 16;          // channels per warp group
        const int ch0 = (e >> 2) * cpg;
        const int nch_w = max(0, min(cpg, p.cout - ch0));            // this warp's channels (a multiple of 16; 0 = none)
        const uint32_t t_empty_leader0 = ptx::mapa(bar(T_EMPTY), 0);
        for (int t = 0; t < n_tiles; ++t) {
            const int row = t * C1_BLOCK_M + q * 32 + lane;                 // row inside this CTA's range
            const long long pix = row_base + row;
            const bool ok = (row < p.rows_per_cta) && (pix < p.m_total);
            // (32-bit: the ABI guarantees m_total < 2^31; a 64-bit division is a ~100-instruction subroutine)
            const long long b = ok ? static_cast<unsigned>(pix) / static_cast<unsigned>(p.n_pix) : 0;
            const long long qp = ok ? pix - b * p.n_pix : 0;
            OutT* o = static_cast<OutT*>(p.out) + (b * p.cout + ch0) * p.n_pix + qp;
            // vector path: after the shared-memory transpose lane l owns pixels 4 (l % 8) .. + 3 of channel row l / 8 (+ 4 k)
            const int px4 = (lane & 7) * 4, rsub = lane >> 3;
            const int row4 = t * C1_BLOCK_M + q * 32 + px4;
            const long long pix4 = row_base + row4;
            const bool ok4 = (row4 < p.rows_per_cta) && (pix4 < p.m_total);
            const long long b4 = ok4 ? static_cast<unsigned>(pix4) / static_cast<unsigned>(p.n_pix) : 0;
            OutT* o4 = static_cast<OutT*>(p.out) + (b4 * p.cout + ch0 + rsub) * p.n_pix + (ok4 ? pix4 - b4 * p.n_pix : 0);
            const long long step4 = 4LL * p.n_pix;
            const uint32_t stg = s_stg + e * C1_STG_BYTES;
            const uint32_t acc = t & 1, acc_ph = (t >> 1) & 1;
            ptx::mbar_wait(bar(T_FULL + acc), acc_ph);
            ptx::tc_fence_after();
            if (e == 0 && lane == 0) C1_STAMP(7 + t);                   // accumulator of tile t ready (slots 7, 8)
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * C1_MAX_COUT + ch0;
            if (nch_w == 0) {                                        // nothing to read: hand the accumulator straight back
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive_cluster_relaxed(t_empty_leader0 + 8u * acc);
            }
            for (int c = 0; c < nch_w; c += 32) {
                float v[32];
                const bool two = (c + 16 < nch_w);
                if (!C1_DBG(2)) {
                    ptx::tmem_ld_x16(taddr + c, v);
                    if (two) ptx::tmem_ld_x16(taddr + c + 16, v + 16);
                    ptx::tmem_ld_wait();
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i) v[i] = static_cast<float>(i + c);
                }
                if (e == 0 && lane == 0 && c == 0) C1_STAMP(13 + t);        // first chunk out of TMEM (slots 13, 14)
                if (c + 32 >= nch_w) {
                    // every TMEM read of this tile is done: hand the accumulator back (to the leader)
                    ptx::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) ptx::mbar_arrive_cluster_relaxed(t_empty_leader0 + 8u * acc);
                }
                const int nch = two ? 32 : 16;
                if constexpr (NHWC) {
                    if (ok && !C1_DBG(1)) {
#pragma unroll
                        for (int i = 0; i < 32; ++i) {
                            v[i] += lds_ro_f32(s_bias + min(ch0 + c + i, p.cout - 1) * 4);
                            if (p.relu) v[i] = fmaxf(v[i], 0.f);
                        }
                        OutT* d = static_cast<OutT*>(p.out) + pix * p.out_ps + ch0 + c;
                        c1_store16(d, v);
                        if (two) c1_store16(d + 16, v + 16);
                    }
                    continue;
                }
                if (p.vec4) {
                    // transpose through this warp's 4 KB buffer: [channel][pixel] fp32, a row is one conflict-free
                    // 128-byte st.shared; a quarter-warp then reads one row back as eight 16-byte pieces
#pragma unroll
                    for (int i = 0; i < 32; ++i)
                        if (i < nch) sts_f32(stg + (i * 32 + lane) * 4, v[i]);
                    __syncwarp();
                    OutT* d4 = o4 + static_cast<long long>(c) * p.n_pix;
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        if (4 * k < nch) {
                            const int r = 4 * k + rsub;
                            const float4 x = lds_f32x4(stg + (r * 32 + px4) * 4);
                            const float bb = lds_ro_f32(s_bias + (ch0 + c + r) * 4);
                            float a0 = x.x + bb, a1 = x.y + bb, a2 = x.z + bb, a3 = x.w + bb;
                            if (p.relu) { a0 = fmaxf(a0, 0.f); a1 = fmaxf(a1, 0.f); a2 = fmaxf(a2, 0.f); a3 = fmaxf(a3, 0.f); }
                            if (ok4 && !C1_DBG(1)) c1_store4(d4, a0, a1, a2, a3);
                            d4 += step4;
                        }
                    }
                    __syncwarp();                                    // the buffer is reused by the next chunk
                } else {
                    OutT* ds = o + static_cast<long long>(c) * p.n_pix;
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        if (i < nch) {
                            float x = v[i] + lds_ro_f32(s_bias + (ch0 + c + i) * 4);
                            if (p.relu) x = fmaxf(x, 0.f);
                            if (ok) *ds = c1_cvt<OutT>(x);
                            ds += p.n_pix;
                        }
                    }
                }
            }
            if (e == 0 && lane == 0) C1_STAMP(9 + t);                   // this warp's stores of tile t issued (slots 9, 10)
        }
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 0 && lane == 0) C1_STAMP(11);          // every warp of this CTA is done
    ptx::cluster_sync_all();          // the leader's MMAs read the peer's shared memory until the very end
    if (warp == 0 && lane == 0) C1_STAMP(12);
    if (warp == 2) ptx::tmem_dealloc_2sm(tmem_base, 512);
}

template <typename OutT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(C1_THREADS, 1)
corr_conv1x1_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_w,
                    const Conv1x1Params p) {
    corr_conv1x1_body<OutT, false>(tm_a, tm_w, p);
}

template <typename OutT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(C1_THREADS, 1)
corr_conv1x1_nhwc_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_w,
                         const Conv1x1Params p) {
    corr_conv1x1_body<OutT, true>(tm_a, tm_w, p);
}

}  // namespace rdvc
