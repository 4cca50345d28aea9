// corr_pack.cuh -- feature-map repack, one launch for both maps:
//   (B, D, h, w) {fp32|bf16|fp16}, NCHW as torchvision's encoder emits them (TV:raft.py:492-493)
//   -> K-major 16-bit rows [B][n_l][D] (D contiguous; bf16, or fp16 when the inputs are fp16), what the tcgen05 operand descriptors in
//      corr_build_sm100.cuh expect: fmap1 at level 0; fmap2 at level 0 and, for the linear
//      build mode, at the pooled levels 1..3.
// Level l row (Y, X) is the mean over the 2^l x 2^l block of the source map (= l nested
// floor-cropped 2x2 means, TV:raft.py:390-392), taken in fp32 and rounded to bf16 ONCE.
//
// One CTA = an 8 x 32 spatial block x 64 channels, fp32 in shared memory: global reads are
// 128-byte rows of the source, global writes are 128-byte pieces (64 channels) of the K-major
// rows.  Each map is read exactly once and each staged value is read from shared memory once
// (the pooled levels are register sums along a quad-ordered walk).  Small next to the volume
// write (67 MB in, 39 MB out at 1080p).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>

namespace rdvc {

constexpr int PACK_THREADS = 256;
constexpr int PACK_TY = 8, PACK_TX = 32, PACK_CG = 64;   // block: 8 rows x 32 px x 64 channels
constexpr int PACK_PITCH = PACK_TY * PACK_TX + 1;        // 257 floats per channel (bank spread)
constexpr int PACK_SMEM_BYTES = PACK_CG * PACK_PITCH * 4;

struct PackParams {
    const void* src[2];          // fmap1, fmap2
    __nv_bfloat16* dst[2][4];    // [map][level]
    int levels[2];               // levels to emit per map (fmap1: 1)
    int tiled[2];                // per map: rows in RDVC_LAYOUT_TILED order instead of raster order
    int twl, thl;                // log2 tile width / height of the tiled order
    int img[2][4];               // [map][level]: operand rows per batch item (pixels incl. layout padding)
    int f16;                     // operand format: 0 = bf16, 1 = fp16 (fp16 inputs keep their 11-bit mantissa)
    int B, D, h, w;
    long long ps;                // NHWC sources: pixel stride in elements (a multiple of 8, 16-byte aligned bases)
};

template <typename T> __device__ __forceinline__ float pack_to_float(T v);
template <> __device__ __forceinline__ float pack_to_float<float>(float v) { return v; }
template <> __device__ __forceinline__ float pack_to_float<__nv_bfloat16>(__nv_bfloat16 v) {
    return __bfloat162float(v);
}
template <> __device__ __forceinline__ float pack_to_float<__half>(__half v) {
    return __half2float(v);
}

// 4 consecutive elements (16-byte / 8-byte aligned) -> 4 floats
template <typename T> __device__ __forceinline__ void pack_ld4(const T* p, float* v);
template <> __device__ __forceinline__ void pack_ld4<float>(const float* p, float* v) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <> __device__ __forceinline__ void pack_ld4<__nv_bfloat16>(const __nv_bfloat16* p, float* v) {
    const uint2 t = __ldg(reinterpret_cast<const uint2*>(p));
    v[0] = __uint_as_float(t.x << 16); v[1] = __uint_as_float(t.x & 0xffff0000u);
    v[2] = __uint_as_float(t.y << 16); v[3] = __uint_as_float(t.y & 0xffff0000u);
}
template <> __device__ __forceinline__ void pack_ld4<__half>(const __half* p, float* v) {
    const uint2 t = __ldg(reinterpret_cast<const uint2*>(p));
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&t.x));
    const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&t.y));
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

// two floats -> one 32-bit operand pair (round to nearest even), bf16 or fp16
__device__ __forceinline__ uint32_t pack_pair(float a, float b, int f16) {
    if (f16) {
        const __half2 t = __floats2half2_rn(a, b);
        return *reinterpret_cast<const uint32_t*>(&t);
    }
    const __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&t);
}

// grid: (D/64 * ceil(w/32), ceil(h/8), 2 * B); block: 256 threads; dynamic smem: PACK_SMEM_BYTES.
// VEC: w % 4 == 0, rows can be fetched as 16-byte vectors.
// NHWC: the sources are NHWC 16-bit maps, pixel (b, y, x) at src + ((b * h + y) * w + x) * ps (the feature encoder's
// trunk, read in place); 16-byte loads of 8 channels, 8 lanes per pixel.  Same tile, same stores, same rows.
// QUICK: the layout is raster order or 4-row tiles 4 / 8 pixels wide (the defaults), so a warp's region maps onto
// whole layout tiles and pixel addresses are compile-time offsets from one base per level; !QUICK keeps the general
// per-pixel formula for other (experimental) tile shapes.  Two instantiations instead of a run-time choice: the
// general formula inlined 43 times made the kernel 4096 instructions long.
template <typename T, bool QUICK, bool VEC, bool NHWC = false>
__global__ void __launch_bounds__(PACK_THREADS)
corr_pack_kernel(const __grid_constant__ PackParams p) {
    extern __shared__ float tile[];  // [64][257], column = yy * 32 + xx
    const int D = p.D, h = p.h, w = p.w;
    // the D/64 channel groups of one spatial block are neighbours in dispatch order (fastest grid index):
    // the 128-byte pieces they write into the same 512-byte operand rows then meet in L2
    const int cgn = D / PACK_CG;
    const int cg = blockIdx.x % cgn;
    const int b = blockIdx.z % p.B;
    const int map = blockIdx.z / p.B;
    const int y0 = blockIdx.y * PACK_TY, x0 = (blockIdx.x / cgn) * PACK_TX;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const T* src = NHWC ? static_cast<const T*>(p.src[map]) + static_cast<size_t>(cg) * PACK_CG
                        : static_cast<const T*>(p.src[map]) +
                              (static_cast<size_t>(b) * D + static_cast<size_t>(cg) * PACK_CG) * h * w;

    // load.  Vector path (w % 4 == 0): one warp instruction fetches 4 pixels per lane for 4
    // consecutive channels at one row (4 x 128 B of fp32), PACK_MLP of them in flight per
    // thread before the first is consumed; the 4 channels land 257 floats apart, so the four
    // scalar smem stores are conflict-free.  Scalar path: one 32-pixel row per instruction.
    constexpr int NWARP = PACK_THREADS / 32, PACK_MLP = 8;
    if constexpr (NHWC) {
        static_assert(sizeof(T) == 2, "NHWC sources are 16-bit");
        constexpr int CHUNKS = PACK_TY * PACK_TX * (PACK_CG / 8);   // 16-byte pieces: 8 per pixel
        static_assert(CHUNKS % (PACK_THREADS * PACK_MLP) == 0, "load loop shape");
        for (int i0 = threadIdx.x; i0 < CHUNKS; i0 += PACK_THREADS * PACK_MLP) {
            uint4 v[PACK_MLP];
#pragma unroll
            for (int u = 0; u < PACK_MLP; ++u) {
                const int i = i0 + u * PACK_THREADS, q = i >> 3;
                const int y = y0 + q / PACK_TX, x = x0 + q % PACK_TX;
                v[u] = make_uint4(0, 0, 0, 0);
                if (y < h && x < w)
                    v[u] = __ldg(reinterpret_cast<const uint4*>(
                        src + ((static_cast<size_t>(b) * h + y) * w + x) * static_cast<size_t>(p.ps) + (i & 7) * 8));
            }
#pragma unroll
            for (int u = 0; u < PACK_MLP; ++u) {
                const int i = i0 + u * PACK_THREADS, q = i >> 3;
                const T* e = reinterpret_cast<const T*>(&v[u]);
                float* t = tile + (i & 7) * 8 * PACK_PITCH + q;
#pragma unroll
                for (int k = 0; k < 8; ++k) t[k * PACK_PITCH] = pack_to_float<T>(e[k]);
            }
        }
    } else if constexpr (VEC) {   // w % 4 == 0, chosen by the host: the two load loops are separate instantiations
        constexpr int ROWS4 = PACK_CG * PACK_TY / 4;   // 128 four-channel row groups
        static_assert(ROWS4 % (NWARP * PACK_MLP) == 0, "load loop shape");
        const int cl = lane >> 3, xq = (lane & 7) * 4;
        const int x = x0 + xq;
        for (int i0 = warp; i0 < ROWS4; i0 += NWARP * PACK_MLP) {
            float v[PACK_MLP][4];
#pragma unroll
            for (int u = 0; u < PACK_MLP; ++u) {
                const int i = i0 + u * NWARP;
                const int c = (i / PACK_TY) * 4 + cl, y = y0 + i % PACK_TY;
                v[u][0] = v[u][1] = v[u][2] = v[u][3] = 0.f;
                if (y < h && x < w) pack_ld4<T>(src + (static_cast<size_t>(c) * h + y) * w + x, v[u]);
            }
#pragma unroll
            for (int u = 0; u < PACK_MLP; ++u) {
                const int i = i0 + u * NWARP;
                float* t = tile + ((i / PACK_TY) * 4 + cl) * PACK_PITCH + (i % PACK_TY) * PACK_TX + xq;
                t[0] = v[u][0]; t[1] = v[u][1]; t[2] = v[u][2]; t[3] = v[u][3];
            }
        }
    } else {
        static_assert((PACK_CG * PACK_TY) % (NWARP * PACK_MLP) == 0, "load loop shape");
        const int x = x0 + lane;
        for (int i0 = warp; i0 < PACK_CG * PACK_TY; i0 += NWARP * PACK_MLP) {
            float v[PACK_MLP];
#pragma unroll
            for (int u = 0; u < PACK_MLP; ++u) {
                const int i = i0 + u * NWARP;
                const int c = i / PACK_TY, y = y0 + i % PACK_TY;
                v[u] = (y < h && x < w) ? pack_to_float<T>(__ldg(src + (static_cast<size_t>(c) * h + y) * w + x)) : 0.f;
            }
#pragma unroll
            for (int u = 0; u < PACK_MLP; ++u) {
                const int i = i0 + u * NWARP;
                tile[(i / PACK_TY) * PACK_PITCH + (i % PACK_TY) * PACK_TX + lane] = v[u];
            }
        }
    }
    __syncthreads();

    // store: one K-major row piece (64 channels = 128 B of bf16) per warp instruction, lane = channel
    // pair.  Warp wq owns the 4 x 8 pixel region (rows 4*(wq&1).., columns 8*(wq>>1)..) of the block and
    // walks it quad by quad (2x2 inside 4x4), so every level-0 value is read from shared memory ONCE:
    // the pooled levels are running sums in registers (level 1 = a quad, level 2 = four quads); the two
    // warps of an 8 x 8 block combine their halves of the level-3 sum through shared memory.
    const int L = p.levels[map];
    const int ry0 = (warp & 1) * 4, cx0 = (warp >> 1) * 8;
    const int f16 = p.f16;
    auto row_ptr = [&](int l, int Y, int X) -> uint32_t* {
        // operand row of pixel (Y, X) of level l: raster order, or tile by tile (see rdvc_corr.h); the
        // build's output columns follow the operand rows, so this IS the volume's layout
        const int wl = w >> l;
        size_t pix = static_cast<size_t>(Y) * wl + X;
        if (p.tiled[map]) {
            const int twl = p.twl, thl = p.thl;
            const int tiles_w = (wl + (1 << twl) - 1) >> twl;
            pix = (static_cast<size_t>((Y >> thl) * tiles_w + (X >> twl)) << (twl + thl)) +
                  ((Y & ((1 << thl) - 1)) << twl) + (X & ((1 << twl) - 1));
        }
        return reinterpret_cast<uint32_t*>(
                   p.dst[map][l] + (static_cast<size_t>(b) * p.img[map][l] + pix) * D + cg * PACK_CG) + lane;
    };
    const float* t0 = tile + (2 * lane) * PACK_PITCH + ry0 * PACK_TX + cx0;
    // Address of the region's first pixel per level once; the other pixels are compile-time row offsets from
    // it whenever the region maps onto whole layout tiles (raster order, or 4-row tiles 4 or 8 pixels wide --
    // the defaults); other tile shapes (experiments) take the general per-pixel formula.
    const int Yr = y0 + ry0, Xr = x0 + cx0;           // level-0 origin of this warp's 4 x 8 region
    const bool tl = p.tiled[map] != 0;
    constexpr bool quick = QUICK;
    const bool w4 = tl && p.twl == 2, w8 = tl && p.twl == 3;
    const size_t rstride = static_cast<size_t>(D) / 2;    // one operand row in 32-bit pairs
    uint32_t* const b0 = row_ptr(0, Yr, Xr);
    uint32_t* const b1 = (L > 1) ? row_ptr(1, Yr >> 1, Xr >> 1) : b0;
    uint32_t* const b2p = (L > 2) ? row_ptr(2, Yr >> 2, Xr >> 2) : b0;
    const int w0 = w, w1 = w >> 1;
    float s3a = 0.f, s3b = 0.f;                       // this warp's half of the level-3 sum (4 x 8 pixels)
#pragma unroll
    for (int b2 = 0; b2 < 2; ++b2) {                  // the two 4 x 4 blocks of the region
        float s2a = 0.f, s2b = 0.f;
#pragma unroll
        for (int qd = 0; qd < 4; ++qd) {              // 2 x 2 quads of a 4 x 4 block
            float s1a = 0.f, s1b = 0.f;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int yy = (qd >> 1) * 2 + (e >> 1), xx = b2 * 4 + (qd & 1) * 2 + (e & 1);
                const float v0 = t0[yy * PACK_TX + xx], v1 = t0[PACK_PITCH + yy * PACK_TX + xx];
                s1a += v0; s1b += v1;
                const int Y = Yr + yy, X = Xr + xx;
                if (Y < h && X < w) {
                    // row offset from b0: raster yy * w + xx; 4-wide tiles: next tile after 16; 8-wide: one tile
                    const int off = w4 ? (xx >> 2) * 16 + yy * 4 + (xx & 3) : w8 ? yy * 8 + xx : yy * w0 + xx;
                    uint32_t* dst;
                    if constexpr (quick) dst = b0 + off * rstride; else dst = row_ptr(0, Y, X);
                    *dst = pack_pair(v0, v1, f16);
                }
            }
            s2a += s1a; s2b += s1b;
            if (L > 1) {
                const int qy = qd >> 1, qx = b2 * 2 + (qd & 1);
                const int Y = (Yr >> 1) + qy, X = (Xr >> 1) + qx;
                if (Y < (h >> 1) && X < (w >> 1)) {
                    const int off = w4 ? qy * 4 + qx : w8 ? qy * 8 + qx : qy * w1 + qx;   // inside one tile
                    uint32_t* dst;
                    if constexpr (quick) dst = b1 + off * rstride; else dst = row_ptr(1, Y, X);
                    *dst = pack_pair(s1a * 0.25f, s1b * 0.25f, f16);
                }
            }
        }
        s3a += s2a; s3b += s2b;
        if (L > 2) {
            const int Y = Yr >> 2, X = (Xr >> 2) + b2;
            if (Y < (h >> 2) && X < (w >> 2)) {
                uint32_t* dst;                                                               // x neighbour, same tile
                if constexpr (quick) dst = b2p + b2 * rstride; else dst = row_ptr(2, Y, X);
                *dst = pack_pair(s2a * (1.0f / 16.0f), s2b * (1.0f / 16.0f), f16);
            }
        }
    }
    if (L > 3) {                                      // uniform over the block: all warps take it or none
        __syncthreads();                              // the tile has been consumed: reuse its first floats
        float2* part = reinterpret_cast<float2*>(tile);          // [4 blocks][32 lanes]
        if (warp & 1) part[(warp >> 1) * 32 + lane] = make_float2(s3a, s3b);
        __syncthreads();
        if (!(warp & 1)) {
            const float2 o = part[(warp >> 1) * 32 + lane];
            const int Y = y0 / 8, X = (x0 + cx0) / 8;
            if (Y < (h >> 3) && X < (w >> 3))
                *row_ptr(3, Y, X) = pack_pair((s3a + o.x) * (1.0f / 64.0f), (s3b + o.y) * (1.0f / 64.0f), f16);
        }
    }
}

}  // namespace rdvc
