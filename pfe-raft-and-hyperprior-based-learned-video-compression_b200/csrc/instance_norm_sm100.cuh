// instance_norm_sm100.cuh -- the CUDA-core half of RAFT's feature encoder (FeatureEncoder with InstanceNorm,
// TV:raft.py:116-168): tap_conv_in_kernel (tap_conv_sm100.cuh) stores each convolution's raw output and per-tile
// (mean, M2) partials; in_finalize_kernel turns a layer's partials into per-(sample, channel) mean and rstd, and
// in_apply_kernel normalises the raw output and closes the residual block.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>
#include <type_traits>

#include "tap_conv_sm100.cuh"

namespace rdvc {

// Per (sample, channel): Chan's parallel merge of the tiles' (mean, M2) in fp64, in a fixed order -> fp32 mean and
// rstd = 1 / sqrt(M2 / n + eps) (the biased variance, as InstanceNorm uses).  grid (NT / 32, B), block
// (32, IN_FIN_SLICES): thread (c, s) merges tiles s, s + IN_FIN_SLICES, ... of image blockIdx.y (a warp reads 32
// consecutive channels of one tile), then thread (c, 0) merges the slices in order.
constexpr int IN_FIN_SLICES = 16;

struct InFinParams {
    const float2* part;         // [n_tiles][NT] per-tile (mean, M2) of tap_conv_in_kernel; an image's tiles contiguous
    float* stats;               // [B][2][NT]: mean, then rstd
    int NT, N;                  // channels; channels >= N (the fused downsample's) use eps_hi
    int n_tx, n_ty, H, W;       // the convolution's tile grid and output size
    double eps_lo, eps_hi;
};

__device__ __forceinline__ void chan_merge(double& n, double& mean, double& m2, double nb, double mb, double m2b) {
    if (nb == 0.0) return;
    const double nn = n + nb, d = mb - mean;
    mean += d * (nb / nn);
    m2 += m2b + d * d * (n * nb / nn);
    n = nn;
}

__global__ void __launch_bounds__(32 * IN_FIN_SLICES) in_finalize_kernel(const InFinParams p) {
    __shared__ double sh[3][IN_FIN_SLICES][32];
    const int c = blockIdx.x * 32 + threadIdx.x, s = threadIdx.y, b = blockIdx.y;
    const int per_img = p.n_tx * p.n_ty;
    const float2* part = p.part + static_cast<long long>(b) * per_img * p.NT + c;
    double n = 0.0, mean = 0.0, m2 = 0.0;
    for (int t = s; t < per_img; t += IN_FIN_SLICES) {
        const int x0 = (t % p.n_tx) * TAP_TX, y0 = (t / p.n_tx) * TAP_TY;
        const float2 a = part[static_cast<long long>(t) * p.NT];
        chan_merge(n, mean, m2, static_cast<double>(min(TAP_TX, p.W - x0) * min(TAP_TY, p.H - y0)), a.x, a.y);
    }
    sh[0][s][threadIdx.x] = n; sh[1][s][threadIdx.x] = mean; sh[2][s][threadIdx.x] = m2;
    __syncthreads();
    if (s != 0) return;
    for (int k = 1; k < IN_FIN_SLICES; ++k)
        chan_merge(n, mean, m2, sh[0][k][threadIdx.x], sh[1][k][threadIdx.x], sh[2][k][threadIdx.x]);
    float* st = p.stats + static_cast<long long>(b) * 2 * p.NT + c;
    st[0] = static_cast<float>(mean);
    st[p.NT] = static_cast<float>(1.0 / sqrt(m2 / n + (c < p.N ? p.eps_lo : p.eps_hi)));
}

// Normalise one layer's raw output y (OpT NHWC) and close its block, one thread per 8 channels of a pixel:
constexpr int IN_APPLY_RELU = 0;      // relu(IN(y))                        stem, every convnormrelu1
constexpr int IN_APPLY_RES = 1;       // relu(z + relu(IN(y)))              convnormrelu2 of an identity block; z its input
constexpr int IN_APPLY_DS = 2;        // relu(IN(z) + relu(IN(y)))          convnormrelu2 of a stride-2 block; z the
                                      //                                    downsample's raw output
struct InApplyParams {
    const void* y;              // OpT, pixel stride y_ps
    const void* z;              // OpT, pixel stride z_ps
    long long y_ps, z_ps;
    const float* st;            // y's [B][2][st_nt] mean / rstd at channel 0
    const float* zst;           // DS: z's, [B][2][zst_nt] at channel 0 (the stride-2 unit's stats + N)
    int st_nt, zst_nt;
    void* out;                  // OpT, pixel stride out_ps
    long long out_ps;
    int C, Cs;                  // real channels; stored channels (multiples of 8): channels C..Cs-1 are written as zeros
    long long hw, n_pix;        // pixels per image, B * hw
};

template <typename OpT>
__device__ __forceinline__ void in_load8(const OpT* p, float* v) {
    const uint4 u = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        float2 f;
        if constexpr (std::is_same<OpT, __half>::value) f = __half22float2(*reinterpret_cast<const __half2*>(&w[j]));
        else f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[j]));
        v[2 * j] = f.x; v[2 * j + 1] = f.y;
    }
}

template <typename OpT>
__device__ __forceinline__ void in_store8(OpT* p, const float* v) {
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
    *reinterpret_cast<uint4*>(p) = make_uint4(w[0], w[1], w[2], w[3]);
}

template <int FORM, typename OpT>
__global__ void __launch_bounds__(256) in_apply_kernel(const InApplyParams p) {
    const int groups = p.Cs >> 3;
    const long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
    if (i >= p.n_pix * groups) return;
    const long long pix = i / groups;
    const int c0 = static_cast<int>(i - pix * groups) * 8;
    OpT* o = static_cast<OpT*>(p.out) + pix * p.out_ps + c0;
    if (c0 >= p.C) {                 // exact zeros whatever eps is (the raw channels are zero with zero variance)
        *reinterpret_cast<uint4*>(o) = make_uint4(0u, 0u, 0u, 0u);
        return;
    }
    const long long b = pix / p.hw;
    float v[8];
    in_load8(static_cast<const OpT*>(p.y) + pix * p.y_ps + c0, v);
    const float* st = p.st + b * 2 * p.st_nt + c0;
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = fmaxf((v[j] - __ldg(st + j)) * __ldg(st + p.st_nt + j), 0.f);
    if constexpr (FORM != IN_APPLY_RELU) {
        float z[8];
        in_load8(static_cast<const OpT*>(p.z) + pix * p.z_ps + c0, z);
        if constexpr (FORM == IN_APPLY_DS) {
            const float* zs = p.zst + b * 2 * p.zst_nt + c0;
#pragma unroll
            for (int j = 0; j < 8; ++j) z[j] = (z[j] - __ldg(zs + j)) * __ldg(zs + p.zst_nt + j);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = fmaxf(z[j] + v[j], 0.f);
    }
    in_store8(o, v);
}

}  // namespace rdvc
