// context_encoder_sm100.cuh -- RAFT's context encoder (torchvision FeatureEncoder with frozen BatchNorm,
// TV:raft.py:116-168) as tcgen05 implicit GEMMs over NHWC 16-bit activations, on the engine of update_conv_sm100.cuh.
// BatchNorm is folded into each convolution's weights and bias on the host (rdvc_corr_context_encoder_pack_weights).
//
//   unit  layer                                  geometry   Cin -> N       epilogue
//   0     convnormrelu (7x7 s2, 3 -> 64)         STEM       64 -> 64       bias, ReLU
//   1-4   layer1.{0,1}.convnormrelu{1,2}         S1         64 -> 64       bias, ReLU | relu(res + relu(acc + bias))
//   5     layer2.0.convnormrelu1 + downsample    S2         64 -> 128+128  bias, ReLU | bias (the residual)
//   6-8   layer2.0.convnormrelu2, layer2.1.*     S1        128 -> 128      as layer1
//   9     layer3.0.convnormrelu1 + downsample    S2        128 -> 128+128  as unit 5
//   10-12 layer3.0.convnormrelu2, layer3.1.*     S1        128 -> 128      as layer1
//   13    conv (1x1, 128 -> 256)                 1X1       128 -> 256      bias | tanh on 0-127, ReLU on 128-255
//
// layer2's 96 channels are stored at a 128-channel pixel stride: the padded weight rows and biases are zero, so the
// epilogue writes exact zeros to channels 96-127 and the next layer's padded K columns (zero weights) multiply zeros.
//
// Geometries (tile = 16 x 8 output pixels, M = 128; every tap is a descriptor offset of whole 1 KB swizzle atoms):
//   S1    3x3 stride 1: one box {64, 16, 10} per dx, the 3 dy taps are row offsets into its halo (as update_conv).
//   S2    3x3 stride 2: the input map has TMA element strides 2 along x and y, so a box {64, 32, 18} lands 16 x 9
//         pixels of one polyphase component.  Per dx two boxes: rows 2y - 1, 2y + 1, ... (dy = 0 at row offset 0,
//         dy = 2 at offset 1) and rows 2y, 2y + 2, ... (dy = 1).  The centre tap's A operand is exactly the 1x1
//         stride-2 downsample's input, so its MMAs into a second accumulator range (columns N..2N) ride on that box.
//   STEM  the 7x7 stride-2 stem over 3 channels is a 4x1 stride-1 convolution over the packed operand of
//         ce_stem_pack_kernel (per half-resolution pixel: 4 horizontal polyphase taps x 2 x 2 phases x 3 channels =
//         48 values, zero-padded to 64): one box {64, 16, 11}, the 4 vertical taps are row offsets (-2..+1).
//   1X1   one box {64, 16, 8}.
// Zero padding and tail tiles are TMA's out-of-bounds fill on the load side and a per-pixel mask on the store side.
// Weights stream from L2 as (k-block, slab) slabs of N x 64, packed [k-block][slab][N][64], each feeding UC_P tiles.
#pragma once
#include "update_conv_sm100.cuh"

namespace rdvc {

constexpr int CE_G_S1 = 0;
constexpr int CE_G_S2 = 1;
constexpr int CE_G_STEM = 2;
constexpr int CE_G_1X1 = 3;

constexpr int CE_EPI_RELU = 0;    // relu(acc + bias) -> OutT
constexpr int CE_EPI_RES = 1;     // relu(res + relu(acc + bias)) -> OutT; res: OpT NHWC at (res, res_ps)
constexpr int CE_EPI_DS = 2;      // columns 0..N-1: relu(acc + bias) -> out; N..2N-1: acc + bias -> out2
constexpr int CE_EPI_RAW = 3;     // acc + bias -> OutT
constexpr int CE_EPI_SPLIT = 4;   // tanh(acc + bias) on channels 0-127, relu(acc + bias) on the rest -> OutT

template <int G> struct CeGeom;
template <> struct CeGeom<CE_G_S1> { static constexpr int NL = 3, BOX_Y = UC_TY + 2, SLABS = 9; };
template <> struct CeGeom<CE_G_S2> { static constexpr int NL = 6, BOX_Y = UC_TY + 1, SLABS = 10; };
template <> struct CeGeom<CE_G_STEM> { static constexpr int NL = 1, BOX_Y = UC_TY + 3, SLABS = 4; };
template <> struct CeGeom<CE_G_1X1> { static constexpr int NL = 1, BOX_Y = UC_TY, SLABS = 1; };

// weight slabs that read box l (in issue order)
template <int G>
__device__ __forceinline__ int ce_n_slabs(int l) {
    if constexpr (G == CE_G_S1) return 3;
    else if constexpr (G == CE_G_S2) return ((l & 1) == 0 || l == 3) ? 2 : 1;   // l = 3: dy = 1, dx = 1 + downsample
    else if constexpr (G == CE_G_STEM) return 4;
    else return 1;
}

// slab i of box l: its index within the k-block
template <int G>
__device__ __forceinline__ int ce_slab(int l, int i) {
    if constexpr (G == CE_G_S1) return i * 3 + l;                                  // dy = i, dx = l
    else if constexpr (G == CE_G_S2) return (l & 1) == 0 ? (i == 0 ? 0 : 6) + (l >> 1) : (i == 0 ? 3 + (l >> 1) : 9);
    else if constexpr (G == CE_G_STEM) return i;
    else return 0;
}

// slab i of box l: its A operand's row offset into the box
template <int G>
__device__ __forceinline__ int ce_row(int l, int i) {
    if constexpr (G == CE_G_S2) return (l & 1) == 0 ? i : 0;
    else if constexpr (G == CE_G_1X1) return 0;
    else return i;
}

// box l of the tile at output (x0, y0): its first input coordinates (element coordinates of the map)
template <int G>
__device__ __forceinline__ void ce_box(int l, int x0, int y0, int& x, int& y) {
    if constexpr (G == CE_G_S1) { x = x0 + l - 1; y = y0 - 1; }
    else if constexpr (G == CE_G_S2) { x = 2 * x0 + (l >> 1) - 1; y = 2 * y0 - 1 + (l & 1); }
    else if constexpr (G == CE_G_STEM) { x = x0; y = y0 - 2; }
    else { x = x0; y = y0; }
}

template <int G, int N, bool DS>
struct CeCfg {
    static constexpr int NT = DS ? 2 * N : N;                        // accumulator columns per tile
    static constexpr int BOX_BYTES = UC_TX * CeGeom<G>::BOX_Y * 128;
    static constexpr int W_BYTES = N * 128;
    static constexpr int A_BYTES = UC_P * BOX_BYTES;
    static constexpr int SMEM_A = 0;
    static constexpr int SMEM_W = UC_A_STAGES * A_BYTES;
    static constexpr int SMEM_BAR = SMEM_W + UC_W_STAGES * W_BYTES;
    static constexpr int SMEM_TOTAL = SMEM_BAR + 256;
    static constexpr int SMEM_LAUNCH = SMEM_TOTAL + 1024;
    static constexpr int TMEM_COLS = UC_P * NT <= 128 ? 128 : UC_P * NT <= 256 ? 256 : 512;
    static_assert(N % 16 == 0 && N >= 16 && N <= 256, "UMMA N");
    static_assert(BOX_BYTES % 1024 == 0, "boxes must start on swizzle atoms");
    static_assert(SMEM_LAUNCH <= 227 * 1024, "shared memory");
    static_assert(UC_P * NT <= 512, "tensor memory");
};

struct CeParams {
    int B, H, W;                // output grid
    int n_kb;                   // 64-channel k-blocks of the input
    int n_tx, n_ty, n_tiles, n_super;
    const float* bias;          // NT floats (device)
    void* out;                  // OutT NHWC, pixel stride out_ps
    long long out_ps;
    void* out2;                 // CE_EPI_DS: OpT NHWC, pixel stride out_ps
    const void* res;            // CE_EPI_RES: OpT NHWC, pixel stride res_ps
    long long res_ps;
};

// tm_a: input {Cin, W, H, B}, box {64, 16, BOX_Y, 1} (S2: {64, 32, 18, 1} with element strides {1, 2, 2, 1});
// tm_w: weight slabs {64, N, n_kb * SLABS}, box {64, N, 1}.  128-byte swizzle.
template <int G, int N, int EPI, typename OutT, typename OpT>
__global__ void __launch_bounds__(UC_THREADS, 1)
context_conv_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_w, const CeParams p) {
    constexpr bool DS = (EPI == CE_EPI_DS);
    using Cfg = CeCfg<G, N, DS>;
    constexpr int NL = CeGeom<G>::NL;
    constexpr int NT = Cfg::NT;
    constexpr int WST = UC_W_STAGES;
    static_assert(!DS || G == CE_G_S2, "the fused downsample rides on the stride-2 centre tap");
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
    const UcParams tp{p.B, p.H, p.W, p.n_kb, p.n_tx, p.n_ty, p.n_tiles, p.n_super};   // uc_tile's view

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            uint32_t a_it = 0, w_it = 0;
            for (int s = blockIdx.x; s < p.n_super; s += gridDim.x) {
                int b[UC_P], x0[UC_P], y0[UC_P];
#pragma unroll
                for (int j = 0; j < UC_P; ++j)       // a missing last tile reloads the one before (its stores are masked)
                    uc_tile(tp, min(s * UC_P + j, p.n_tiles - 1), b[j], x0[j], y0[j]);
                for (int kb = 0; kb < p.n_kb; ++kb) {
                    for (int l = 0; l < NL; ++l, ++a_it) {
                        const uint32_t st = a_it % UC_A_STAGES, ph = (a_it / UC_A_STAGES) & 1;
                        ptx::mbar_wait(bar(A_EMPTY + st), ph ^ 1);
                        ptx::mbar_arrive_expect_tx(bar(A_FULL + st), Cfg::A_BYTES);
#pragma unroll
                        for (int j = 0; j < UC_P; ++j) {
                            int x, y;
                            ce_box<G>(l, x0[j], y0[j], x, y);
                            ptx::tma_load_4d(s_a + st * Cfg::A_BYTES + j * Cfg::BOX_BYTES, &tm_a, bar(A_FULL + st), kb * 64,
                                             x, y, b[j]);
                        }
                        const int ns = ce_n_slabs<G>(l);
                        for (int i = 0; i < ns; ++i, ++w_it) {
                            const uint32_t ws = w_it % WST, wph = (w_it / WST) & 1;
                            ptx::mbar_wait(bar(W_EMPTY + ws), wph ^ 1);
                            ptx::mbar_arrive_expect_tx(bar(W_FULL + ws), Cfg::W_BYTES);
                            ptx::tma_load_3d(s_w + ws * Cfg::W_BYTES, &tm_w, bar(W_FULL + ws), 0, 0,
                                             kb * CeGeom<G>::SLABS + ce_slab<G>(l, i));
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
                for (int l = 0; l < NL; ++l, ++a_it) {
                    const uint32_t st = a_it % UC_A_STAGES, ph = (a_it / UC_A_STAGES) & 1;
                    ptx::mbar_wait(bar(A_FULL + st), ph);
                    ptx::tc_fence_after();
                    const uint64_t a_desc0 = ptx::umma_desc_k_sw128(s_a + st * Cfg::A_BYTES);
                    const int ns = ce_n_slabs<G>(l);
#pragma unroll 1
                    for (int i = 0; i < ns; ++i, ++w_it) {
                        const uint32_t ws = w_it % WST, wph = (w_it / WST) & 1;
                        ptx::mbar_wait(bar(W_FULL + ws), wph);
                        ptx::tc_fence_after();
                        const uint64_t b_desc0 = ptx::umma_desc_k_sw128(s_w + ws * Cfg::W_BYTES);
                        const bool ds = DS && l == 3 && i == 1;                  // the downsample's slab
                        const uint32_t col = ds ? N : 0;
                        const bool first = ds ? kb == 0 : (kb | l | i) == 0;
                        const int row = ce_row<G>(l, i);
                        if (ptx::elect_one()) {
#pragma unroll
                            for (int j = 0; j < UC_P; ++j) {
#pragma unroll
                                for (int k = 0; k < 4; ++k)
                                    ptx::umma_bf16(tmem_base + j * NT + col,
                                                   a_desc0 + ((j * Cfg::BOX_BYTES + row * UC_DY_STEP + k * 32) >> 4),
                                                   b_desc0 + ((k * 32) >> 4), idesc, (first && k == 0) ? 0u : 1u);
                            }
                            ptx::umma_commit(bar(W_EMPTY + ws));                     // slab free when these MMAs retire
                            if (i == ns - 1) ptx::umma_commit(bar(A_EMPTY + st));
                            if (i == ns - 1 && l == NL - 1 && kb == p.n_kb - 1) ptx::umma_commit(bar(T_FULL));
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
            uc_tile(tp, min(tile, p.n_tiles - 1), b, x0, y0);
            const int x = x0 + (m & (UC_TX - 1)), y = y0 + m / UC_TX;
            const bool ok = (tile < p.n_tiles) && (x < p.W) && (y < p.H);
            const long long pix = (static_cast<long long>(b) * p.H + y) * p.W + x;
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + j * NT;
            ptx::mbar_wait(bar(T_FULL), t_it & 1);
            ptx::tc_fence_after();
            OutT* o = static_cast<OutT*>(p.out) + pix * p.out_ps;
#pragma unroll 1
            for (int c = 0; c < NT; c += 16) {
                float v[16];
                ptx::tmem_ld_x16(taddr + c, v);
                ptx::tmem_ld_wait();
                if (ok) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] += __ldg(p.bias + c + i);
                    if constexpr (EPI == CE_EPI_RELU) {
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.f);
                    } else if constexpr (EPI == CE_EPI_RES) {
                        float r[16];
                        GruVec<OpT>::load(static_cast<const OpT*>(p.res) + pix * p.res_ps + c, r);
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[i] = fmaxf(r[i] + fmaxf(v[i], 0.f), 0.f);
                    } else if constexpr (EPI == CE_EPI_SPLIT) {
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[i] = c < 128 ? tanhf(v[i]) : fmaxf(v[i], 0.f);
                    }
                    if constexpr (DS) {
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
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(bar(T_EMPTY));      // accumulators back to the MMA warp
        }
    }

    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 2) ptx::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
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
