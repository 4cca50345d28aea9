// rdvc_corr_abi.cu -- the C ABI of librdvc_corr.so (see include/rdvc_corr.h).
// Argument checking, pyramid layout arithmetic, TMA descriptor encoding and the
// kernel launches.  No torch, no C++ types across the boundary, no CPU fallback.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/rdvc_corr.h"
#include "corr_build_sm100.cuh"
#ifdef RDVC_EXPERIMENTS
#include "corr_build2_sm100.cuh"
#endif
#include "corr_conv1x1_sm100.cuh"
#include "corr_encoder_tail_sm100.cuh"
#include "corr_lookup.cuh"
#include "corr_pack.cuh"
#include "mask_upsample_sm100.cuh"
#include "tap_conv_sm100.cuh"
#include "instance_norm_sm100.cuh"
#include "entropy_coder.h"
#include "mcn_conv_sm100.cuh"
#include "mcn_convx_sm100.cuh"
#include "motion_warp.cuh"
#include "preprocess.cuh"
#include "raft_flow.cuh"

#ifndef RDVC_PAIR_DEFAULT
#define RDVC_PAIR_DEFAULT 0   // the CTA-pair build kernel is opt-in (option key 12 = 2) until it wins
#endif
// RDVC_EXPERIMENTS (off in the product build, `python -m ..._build --experiments` turns it on in a SEPARATE
// library, lib/librdvc_corr_exp.so): compiles in the knobs that skip work for timing experiments (level store
// mask, no-load / no-store lookups, L2 store policies) and the build variants that lost their measurements
// (fused pooling epilogue, CTA-pair kernel).  The product library accepts none of them.
#ifdef RDVC_EXPERIMENTS
#define RDVC_HAS_EXPERIMENTS 1
#else
#define RDVC_HAS_EXPERIMENTS 0
#endif
#ifndef RDVC_SRC_HASH
#define RDVC_SRC_HASH "unknown"
#endif
#define RDVC_STR2(x) #x
#define RDVC_STR(x) RDVC_STR2(x)

namespace {

thread_local char g_err[512] = "";
thread_local unsigned long long g_launches = 0;
thread_local cudaEvent_t g_prof_start = nullptr, g_prof_stop = nullptr;
std::atomic<int> g_opt_lookup{0};
std::atomic<int> g_opt_tile{0};
std::atomic<int> g_opt_msplit{0};
std::atomic<int> g_opt_store_mask{15};
std::atomic<int> g_opt_mode{0};
std::atomic<int> g_opt_tma_out{1};
std::atomic<int> g_opt_policy{0};
std::atomic<int> g_opt_twl{0};
std::atomic<int> g_opt_thl{0};
std::atomic<int> g_opt_epi_warps{0};
std::atomic<int> g_opt_pair{0};
std::atomic<int> g_opt_mcn_prefetch{0};
std::atomic<int> g_dbg_c1_flags{0};
std::atomic<unsigned long long*> g_dbg_timeline{nullptr};   // RDVC_EXPERIMENTS: device buffer for conv1x1 time stamps
std::atomic<int> g_opt_mcn_kernel{0};     // 0 = auto, 1 = three boxes per tile, 2 = one box per tile (x halo)   // measured: no effect at 1-4 tiles ahead, slower beyond (DESIGN 3.6)

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

int cuda_fail(cudaError_t e, const char* what) {
    snprintf(g_err, sizeof(g_err), "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
    return static_cast<int>(e);
}

size_t elem_size(int dt) {
    switch (dt) {
        case RDVC_DT_F32: return 4;
        case RDVC_DT_BF16: return 2;
        case RDVC_DT_F16: return 2;
        default: return 0;
    }
}

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// log2 tile shape of RDVC_LAYOUT_TILED: 16-byte rows x 4 rows (one 64-byte DRAM atom) unless
// overridden by the experiment options (keys 7 / 8)
void tile_log2(int vol_dtype, int* twl, int* thl) {
    const int ow = g_opt_twl.load(), oh = g_opt_thl.load();
    *twl = ow > 0 ? ow : (vol_dtype == RDVC_DT_F32 ? 2 : 3);
    *thl = oh > 0 ? oh : 2;
    if (vol_dtype != RDVC_DT_F32 && *twl < 3) *twl = 3;  // a 16-byte word must not straddle tiles
}

// elements of one level image in the given layout (TILED pads both sides to whole tiles)
size_t level_image_elems(int h, int w, int level, int vol_dtype, int layout) {
    if (vol_dtype != RDVC_DT_F32 && vol_dtype != RDVC_DT_BF16) return 0;   // size queries answer 0 for a bad enum
    if (h <= 0 || w <= 0 || level < 0 || level >= 31) return 0;
    const size_t hl = h >> level, wl = w >> level;
    if (layout != RDVC_LAYOUT_TILED) return hl * wl;
    int twl, thl;
    tile_log2(vol_dtype, &twl, &thl);
    const size_t tiles = (((hl + (1u << thl) - 1) >> thl) << thl) * (((wl + (1u << twl) - 1) >> twl) << twl);
    // whole 256-byte units per image row of the volume (a few all-zero tiles at the end): the build's
    // wide TMA boxes write 256 contiguous bytes per row visit, and a row pitch that keeps them
    // 256-byte aligned measures 6.1 instead of 5.7 TB/s (tools/micro/wbench3.cu, pitch sweep)
    const size_t per_line = 256 / elem_size(vol_dtype);
    return (tiles + per_line - 1) / per_line * per_line;
}

size_t level_bytes(int B, int h, int w, int level, int vol_dtype, int layout) {
    const size_t N = static_cast<size_t>(h) * w;
    return static_cast<size_t>(B) * N * level_image_elems(h, w, level, vol_dtype, layout) * elem_size(vol_dtype);
}

// upper bound of the K-major operand rows of fmap2 level l over every layout / tile option
size_t operand_rows_max(int h, int w, int level) {
    const size_t hl = h >> level, wl = w >> level;
    return ((hl + 15) / 16 * 16) * ((wl + 15) / 16 * 16);
}

int check_geometry(int B, int h, int w, int num_levels) {
    if (B <= 0 || h <= 0 || w <= 0) return fail(RDVC_E_SHAPE, "non-positive dimension B=%d h=%d w=%d", B, h, w);
    if (num_levels < 1 || num_levels > rdvc::BLD_MAX_LEVELS)
        return fail(RDVC_E_UNSUPPORTED, "num_levels=%d not in [1, %d]", num_levels, rdvc::BLD_MAX_LEVELS);
    const int min_size = 2 * (1 << (num_levels - 1));  // TV:raft.py:376
    if (h < min_size || w < min_size)
        return fail(RDVC_E_TOO_SMALL,
                    "Feature maps are too small to be down-sampled by the correlation pyramid. "
                    "H and W of feature maps should be at least %d; got: (%d, %d)", min_size, h, w);
    return RDVC_OK;
}

// ---- driver entry point for TMA descriptors (no -lcuda link dependency) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
    static std::once_flag once;
    static EncodeTiledFn fn = nullptr;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) ==
                cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    return fn;
}

// Tiled TMA descriptor, 128-byte swizzle, zero OOB fill (loads) / clipped (stores).
int make_tmap(CUtensorMap* m, CUtensorMapDataType dt, void* base, int rank, const cuuint64_t* dims,
              const cuuint64_t* strides_bytes, const cuuint32_t* box,
              CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B, const cuuint32_t* elem_strides = nullptr) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return fail(RDVC_E_DRIVER, "cuTensorMapEncodeTiled not available from the driver");
    const cuuint32_t ones[5] = {1, 1, 1, 1, 1};
    const cuuint32_t* estr = elem_strides ? elem_strides : ones;
    CUresult r = fn(m, dt, rank, base, dims, strides_bytes, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(RDVC_E_DRIVER, "cuTensorMapEncodeTiled failed: CUresult %d", (int)r);
    return RDVC_OK;
}

// per-device facts, cached per device id (a process may drive several GPUs)
constexpr int kMaxDevices = 64;

int current_device() {
    int dev = 0;
    cudaGetDevice(&dev);
    return dev;
}

int sm_count() {
    static std::atomic<int> cache[kMaxDevices];
    const int dev = current_device();
    int n = (dev >= 0 && dev < kMaxDevices) ? cache[dev].load() : 0;
    if (n == 0) {
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
        if (dev >= 0 && dev < kMaxDevices) cache[dev].store(n);
    }
    return n;
}

// cudaFuncSetAttribute(max dynamic smem) is per device: do it once per (kernel instantiation, device)
template <typename K>
int ensure_dynamic_smem(K kern, int bytes, std::atomic<unsigned long long>& done_mask, const char* what) {
    const int dev = current_device();
    const unsigned long long bit = (dev >= 0 && dev < kMaxDevices) ? (1ull << dev) : 0ull;
    if (bit && (done_mask.load() & bit)) return RDVC_OK;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return cuda_fail(e, what);
    if (bit) done_mask.fetch_or(bit);
    return RDVC_OK;
}

template <int MODE, int TY, int TX, typename OutT, int EW, int CL = 1>
int launch_build(const CUtensorMap& ta, const CUtensorMap* tb, const CUtensorMap* to, const rdvc::BuildParams& p,
                 cudaStream_t st) {
    auto kern = rdvc::corr_build_kernel<MODE, TY, TX, OutT, EW, CL>;
    using Cfg = rdvc::BuildCfg<EW>;
    static std::atomic<unsigned long long> attr_done{0};  // per instantiation, one bit per device
    if (int rc = ensure_dynamic_smem(kern, Cfg::SMEM_LAUNCH, attr_done, "cudaFuncSetAttribute(build, max dynamic smem)"))
        return rc;
    cudaError_t e;
    if constexpr (CL == 2) {
        // clusters of two CTAs that share the fmap1 stream (TMA multicast): items are PAIRS of fmap2 tiles
        long long grid = sm_count() & ~1;
        const long long n_items = static_cast<long long>(p.B) * ((p.ntiles + 1) / 2) * p.msplit;
        if (grid > 2 * n_items) grid = 2 * n_items;
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3(static_cast<unsigned>(grid));
        cfg.blockDim = dim3(Cfg::THREADS);
        cfg.dynamicSmemBytes = Cfg::SMEM_LAUNCH;
        cfg.stream = st;
        cudaLaunchAttribute attr;
        attr.id = cudaLaunchAttributeClusterDimension;
        attr.val.clusterDim.x = 2; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
        cfg.attrs = &attr;
        cfg.numAttrs = 1;
        if (g_prof_start) cudaEventRecord(g_prof_start, st);
        e = cudaLaunchKernelEx(&cfg, kern, ta, tb[0], tb[1], tb[2], tb[3], to[0], to[1], to[2], to[3], p);
        if (g_prof_stop) cudaEventRecord(g_prof_stop, st);
    } else {
        long long grid = sm_count();
        const long long n_items = static_cast<long long>(p.B) * p.ntiles * p.msplit;
        if (grid > n_items) grid = n_items;
        if (g_prof_start) cudaEventRecord(g_prof_start, st);
        kern<<<static_cast<unsigned>(grid), Cfg::THREADS, Cfg::SMEM_LAUNCH, st>>>(
            ta, tb[0], tb[1], tb[2], tb[3], to[0], to[1], to[2], to[3], p);
        if (g_prof_stop) cudaEventRecord(g_prof_stop, st);
        e = cudaGetLastError();
    }
    ++g_launches;
    if (e != cudaSuccess) return cuda_fail(e, "corr_build_kernel launch");
    return RDVC_OK;
}

#ifdef RDVC_EXPERIMENTS
template <typename OutT>
int launch_build_pair(const CUtensorMap& ta, const CUtensorMap* tb, const CUtensorMap* to, const rdvc::BuildParams& p,
                      cudaStream_t st) {
    auto kern = rdvc::corr_build2_kernel<OutT>;
    static std::atomic<unsigned long long> attr_done{0};
    if (int rc = ensure_dynamic_smem(kern, rdvc::B2_SMEM_LAUNCH, attr_done, "cudaFuncSetAttribute(build pair, max dynamic smem)"))
        return rc;
    long long grid = sm_count() & ~1;     // whole CTA pairs
    const long long n_items = static_cast<long long>(p.B) * p.ntiles * p.msplit;
    if (grid > 2 * n_items) grid = 2 * n_items;
    if (g_prof_start) cudaEventRecord(g_prof_start, st);
    kern<<<static_cast<unsigned>(grid), rdvc::B2_THREADS, rdvc::B2_SMEM_LAUNCH, st>>>(
        ta, tb[0], tb[1], tb[2], tb[3], to[0], to[1], to[2], to[3], p);
    if (g_prof_stop) cudaEventRecord(g_prof_stop, st);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "corr_build2_kernel launch");
    return RDVC_OK;
}

#endif

// both feature maps -> K-major bf16 rows (fmap2 at `levels2` pyramid levels), one launch
template <typename T, bool QUICK, bool VEC, bool NHWC = false>
int launch_pack_impl(const void* f1, const void* f2, void* a_km, void* const* b_km, int B, int D, int h, int w,
                int levels2, int layout, int twl, int thl, const size_t* nl_of, int f16, cudaStream_t st,
                long long ps = 0) {
    auto kern = rdvc::corr_pack_kernel<T, QUICK, VEC, NHWC>;
    static std::atomic<unsigned long long> attr_done{0};
    if (int rc = ensure_dynamic_smem(kern, rdvc::PACK_SMEM_BYTES, attr_done, "cudaFuncSetAttribute(pack, max dynamic smem)"))
        return rc;
    rdvc::PackParams pp;
    memset(&pp, 0, sizeof(pp));
    pp.src[0] = f1; pp.src[1] = f2;
    pp.dst[0][0] = static_cast<__nv_bfloat16*>(a_km);
    for (int l = 0; l < 4; ++l) pp.dst[1][l] = static_cast<__nv_bfloat16*>(b_km[l]);
    pp.levels[0] = 1; pp.levels[1] = levels2;
    pp.B = B; pp.D = D; pp.h = h; pp.w = w;
    pp.tiled[0] = 0; pp.tiled[1] = (layout == RDVC_LAYOUT_TILED);
    pp.twl = twl; pp.thl = thl;
    pp.f16 = f16;
    pp.ps = ps;
    pp.img[0][0] = h * w;
    for (int l = 0; l < 4; ++l) pp.img[1][l] = static_cast<int>(nl_of[l]);
    dim3 grid((D / rdvc::PACK_CG) * ((w + rdvc::PACK_TX - 1) / rdvc::PACK_TX), (h + rdvc::PACK_TY - 1) / rdvc::PACK_TY,
              2 * B);
    kern<<<grid, rdvc::PACK_THREADS, rdvc::PACK_SMEM_BYTES, st>>>(pp);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "corr_pack_kernel launch");
    return RDVC_OK;
}

// KIND: 0 / 1 = row-major layout, scalar / 128-bit loads; 2.. = tiled layout:
//       2 + DBG (DBG in 0..2)
template <typename T>
int launch_pack(const void* f1, const void* f2, void* a_km, void* const* b_km, int B, int D, int h, int w,
                int levels2, int layout, int twl, int thl, const size_t* nl_of, int f16, cudaStream_t st) {
    const bool quick = (layout != RDVC_LAYOUT_TILED) || (thl == 2 && (twl == 2 || twl == 3));
    // 4-element vector loads need w % 4 == 0 AND 4-element-aligned bases (a contiguous torch view can start at
    // an odd storage offset); anything else takes the scalar instantiation
    const uintptr_t amask = 4 * sizeof(T) - 1;
    const bool vec = (w % 4) == 0 && !((reinterpret_cast<uintptr_t>(f1) | reinterpret_cast<uintptr_t>(f2)) & amask);
    if (quick && vec) return launch_pack_impl<T, true, true>(f1, f2, a_km, b_km, B, D, h, w, levels2, layout, twl, thl, nl_of, f16, st);
    if (quick) return launch_pack_impl<T, true, false>(f1, f2, a_km, b_km, B, D, h, w, levels2, layout, twl, thl, nl_of, f16, st);
    if (vec) return launch_pack_impl<T, false, true>(f1, f2, a_km, b_km, B, D, h, w, levels2, layout, twl, thl, nl_of, f16, st);
    return launch_pack_impl<T, false, false>(f1, f2, a_km, b_km, B, D, h, w, levels2, layout, twl, thl, nl_of, f16, st);
}

// the same rows from NHWC 16-bit maps at pixel stride ps (elements)
template <typename T>
int launch_pack_nhwc(const void* f1, const void* f2, long long ps, void* a_km, void* const* b_km, int B, int D, int h,
                     int w, int levels2, int layout, int twl, int thl, const size_t* nl_of, int f16, cudaStream_t st) {
    const bool quick = (layout != RDVC_LAYOUT_TILED) || (thl == 2 && (twl == 2 || twl == 3));
    if (quick)
        return launch_pack_impl<T, true, false, true>(f1, f2, a_km, b_km, B, D, h, w, levels2, layout, twl, thl, nl_of, f16,
                                                      st, ps);
    return launch_pack_impl<T, false, false, true>(f1, f2, a_km, b_km, B, D, h, w, levels2, layout, twl, thl, nl_of, f16,
                                                   st, ps);
}

// row-major kernels: KIND 0 / 1 = scalar / 128-bit loads
template <int R, typename VolT, int KIND>
int launch_lookup(const rdvc::LookupParams& p, cudaStream_t st) {
    const unsigned grid = static_cast<unsigned>((p.total + 31) / 32);
    rdvc::corr_lookup_kernel<R, VolT, KIND == 1><<<grid, 32 * p.num_levels, 0, st>>>(p);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "corr_lookup_kernel launch");
    return RDVC_OK;
}

template <typename VolT, int KIND>
int dispatch_lookup_radius(int radius, const rdvc::LookupParams& p, cudaStream_t st) {
    switch (radius) {
        case 1: return launch_lookup<1, VolT, KIND>(p, st);
        case 2: return launch_lookup<2, VolT, KIND>(p, st);
        case 3: return launch_lookup<3, VolT, KIND>(p, st);
        case 4: return launch_lookup<4, VolT, KIND>(p, st);
        default: return fail(RDVC_E_UNSUPPORTED, "radius=%d not in [1, 4]", radius);
    }
}

// tiled kernel: OUT = output form (rdvc::LKP_OUT_*), DBG = timing experiments (RDVC_EXPERIMENTS builds only)
template <int R, typename VolT, int OUT, int DBG>
int launch_lookup_tiled(const rdvc::LookupParams& p, cudaStream_t st) {
    const unsigned grid = static_cast<unsigned>((p.total + 31) / 32);
    rdvc::corr_lookup_tiled_kernel<R, VolT, OUT, DBG><<<grid, 32 * p.num_levels, 0, st>>>(p);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "corr_lookup_tiled_kernel launch");
    return RDVC_OK;
}

template <typename VolT, int OUT, int DBG>
int dispatch_lookup_tiled_radius(int radius, const rdvc::LookupParams& p, cudaStream_t st) {
    switch (radius) {
        case 1: return launch_lookup_tiled<1, VolT, OUT, DBG>(p, st);
        case 2: return launch_lookup_tiled<2, VolT, OUT, DBG>(p, st);
        case 3: return launch_lookup_tiled<3, VolT, OUT, DBG>(p, st);
        case 4: return launch_lookup_tiled<4, VolT, OUT, DBG>(p, st);
        default: return fail(RDVC_E_UNSUPPORTED, "radius=%d not in [1, 4]", radius);
    }
}

template <typename VolT>
int dispatch_lookup_tiled(int out_mode, int dbg, int radius, const rdvc::LookupParams& p, cudaStream_t st) {
#ifdef RDVC_EXPERIMENTS
    if (dbg == 1 && out_mode == rdvc::LKP_OUT_NCHW_F32) return dispatch_lookup_tiled_radius<VolT, rdvc::LKP_OUT_NCHW_F32, 1>(radius, p, st);
    if (dbg == 2 && out_mode == rdvc::LKP_OUT_NCHW_F32) return dispatch_lookup_tiled_radius<VolT, rdvc::LKP_OUT_NCHW_F32, 2>(radius, p, st);
    if (dbg == 1 && out_mode == rdvc::LKP_OUT_KM_BF16) return dispatch_lookup_tiled_radius<VolT, rdvc::LKP_OUT_KM_BF16, 1>(radius, p, st);
    if (dbg == 2 && out_mode == rdvc::LKP_OUT_KM_BF16) return dispatch_lookup_tiled_radius<VolT, rdvc::LKP_OUT_KM_BF16, 2>(radius, p, st);
#else
    (void)dbg;
#endif
    switch (out_mode) {
        case rdvc::LKP_OUT_NCHW_F16: return dispatch_lookup_tiled_radius<VolT, rdvc::LKP_OUT_NCHW_F16, 0>(radius, p, st);
        case rdvc::LKP_OUT_KM_BF16: return dispatch_lookup_tiled_radius<VolT, rdvc::LKP_OUT_KM_BF16, 0>(radius, p, st);
        case rdvc::LKP_OUT_KM_F16: return dispatch_lookup_tiled_radius<VolT, rdvc::LKP_OUT_KM_F16, 0>(radius, p, st);
        default: return dispatch_lookup_tiled_radius<VolT, rdvc::LKP_OUT_NCHW_F32, 0>(radius, p, st);
    }
}

template <typename OutT, bool NHWC = false>
cudaError_t launch_conv1x1(const CUtensorMap& tm_a, const CUtensorMap& tm_w, const rdvc::Conv1x1Params& p, unsigned grid,
                           cudaStream_t st) {
    auto kern = [] {
        if constexpr (NHWC) return rdvc::corr_conv1x1_nhwc_kernel<OutT>;
        else return rdvc::corr_conv1x1_kernel<OutT>;
    }();
    static std::atomic<unsigned long long> attr_done{0};
    if (ensure_dynamic_smem(kern, rdvc::C1_SMEM_LAUNCH, attr_done, "cudaFuncSetAttribute(conv1x1, max dynamic smem)"))
        return cudaErrorInvalidValue;
    kern<<<grid, rdvc::C1_THREADS, rdvc::C1_SMEM_LAUNCH, st>>>(tm_a, tm_w, p);
    ++g_launches;
    return cudaGetLastError();
}

// ---- build plan: everything rdvc_corr_build derives from its arguments and the options, cached ----
struct BuildKey {            // compared with memcmp: no padding (2 pointers + 20 ints), zeroed before it is filled
    void* pyramid;
    void* workspace;
    int device, B, D, h, w, f16_ops, vol_dtype, layout, num_levels;
    int opt_mode, opt_tile, opt_msplit, opt_tma_out, opt_epi, opt_pair, opt_twl, opt_thl, opt_store_mask, opt_policy;
    int reserved;
};
static_assert(sizeof(BuildKey) == 2 * sizeof(void*) + 20 * sizeof(int), "BuildKey must have no padding");

struct BuildPlan {
    BuildKey key;
    void* a_km;                              // fmap1 as (B, N, D) 16-bit rows
    void* b_km[rdvc::BLD_MAX_LEVELS];        // fmap2 level l as (B, n_l, D)
    size_t nl_of[rdvc::BLD_MAX_LEVELS];      // pixels (operand rows / output columns) of level l in this layout
    int twl, thl;
    void* memset_ptr;
    size_t memset_bytes;
    bool linear, pair;
    bool cluster;                            // clusters of two CTAs sharing the fmap1 stream (TMA multicast)
    int tile, ew;
    CUtensorMap ta, tb[rdvc::BLD_MAX_LEVELS], to[rdvc::BLD_MAX_LEVELS], tb2[rdvc::BLD_MAX_LEVELS];
    rdvc::BuildParams p, p2;
};

constexpr size_t kPlanCacheSize = 8;
std::mutex g_plan_mutex;
std::vector<BuildPlan> g_plans;              // most recently used first
std::atomic<unsigned long long> g_plan_hits{0}, g_plan_misses{0};

bool plan_cache_get(const BuildKey& key, BuildPlan* out) {
    std::lock_guard<std::mutex> lock(g_plan_mutex);
    for (size_t i = 0; i < g_plans.size(); ++i)
        if (memcmp(&g_plans[i].key, &key, sizeof(key)) == 0) {
            if (i) std::swap(g_plans[0], g_plans[i]);
            *out = g_plans[0];
            ++g_plan_hits;
            return true;
        }
    ++g_plan_misses;
    return false;
}

void plan_cache_put(const BuildPlan& plan) {
    std::lock_guard<std::mutex> lock(g_plan_mutex);
    if (g_plans.size() >= kPlanCacheSize) g_plans.pop_back();
    g_plans.insert(g_plans.begin(), plan);
}

// m-range slices per fmap2 tile: enough (tile, slice) items to fill `G` CTAs (or pairs) in whole waves.
// cost = waves x (m-blocks per slice + ~0.5 for the tile reload); a mild bias toward few slices keeps
// concurrent CTAs on the same query rows (see the kernel).
int choose_msplit(long long units, int m_blks, int G, int forced) {
    int best = 1;
    double best_cost = 1e300;
    const int s_max = m_blks < 64 ? m_blks : 64;
    for (int S = 1; S <= s_max; ++S) {
        const long long waves = (units * S + G - 1) / G;
        const double cost = waves * ((m_blks + S - 1) / S + 0.5) * (1.0 + 0.005 * S);
        if (cost < best_cost) { best_cost = cost; best = S; }
    }
    return (forced > 0) ? (forced < m_blks ? forced : m_blks) : best;
}

// Where the K-major operand rows live inside a workspace of rdvc_corr_workspace_bytes(B, D, h, w): fmap1 rows first,
// then fmap2's rows per level (each block 256-byte aligned and sized for the largest layout), their row counts in this
// layout, and the byte range that must be zeroed before a pack (levels with layout padding).
struct WorkspaceLayout {
    void* a_km;
    void* b_km[rdvc::BLD_MAX_LEVELS];
    size_t nl_of[rdvc::BLD_MAX_LEVELS];
    int twl, thl;
    void* memset_ptr;
    size_t memset_bytes;
};

void workspace_layout(void* workspace, int B, int D, int h, int w, int vol_dtype, int layout, int num_levels,
                      WorkspaceLayout* out) {
    WorkspaceLayout& wl = *out;
    memset(&wl, 0, sizeof(wl));
    const int N = h * w;
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    wl.a_km = ws;
    size_t off = align_up(static_cast<size_t>(B) * N * D * 2, 256);
    for (int l = 0; l < rdvc::BLD_MAX_LEVELS; ++l) {
        wl.b_km[l] = ws + off;
        off += align_up(static_cast<size_t>(B) * operand_rows_max(h, w, l) * D * 2, 256);
    }
    for (int l = 0; l < rdvc::BLD_MAX_LEVELS; ++l) wl.nl_of[l] = level_image_elems(h, w, l, vol_dtype, layout);
    if (layout == RDVC_LAYOUT_TILED) {
        tile_log2(vol_dtype, &wl.twl, &wl.thl);
        int first = -1;
        for (int l = 0; l < num_levels && first < 0; ++l)
            if (wl.nl_of[l] != static_cast<size_t>(h >> l) * (w >> l)) first = l;
        if (first >= 0) {
            uint8_t* lo = static_cast<uint8_t*>(wl.b_km[first]);
            uint8_t* hi = static_cast<uint8_t*>(wl.b_km[num_levels - 1]) + static_cast<size_t>(B) * wl.nl_of[num_levels - 1] * D * 2;
            wl.memset_ptr = lo;
            wl.memset_bytes = static_cast<size_t>(hi - lo);
        }
    }
}

int make_build_plan(const BuildKey& k, BuildPlan* plan) {
    BuildPlan& pl = *plan;
    memset(&pl, 0, sizeof(pl));
    pl.key = k;
    const int B = k.B, D = k.D, h = k.h, w = k.w, num_levels = k.num_levels, vol_dtype = k.vol_dtype, layout = k.layout;
    const int N = h * w;
    int mode = k.opt_mode;
    if (mode == 0) mode = 2;  // default: linear (pooled fmap2 rows), see corr_build_sm100.cuh
    pl.linear = (mode == 2);
    if (!pl.linear && !RDVC_HAS_EXPERIMENTS)
        return fail(RDVC_E_UNSUPPORTED, "the fused-epilogue build mode exists in RDVC_EXPERIMENTS builds only");
    if (!pl.linear && layout != RDVC_LAYOUT_ROWMAJOR)
        return fail(RDVC_E_UNSUPPORTED, "the fused-epilogue build mode writes RDVC_LAYOUT_ROWMAJOR only");
    {
        WorkspaceLayout wl;
        workspace_layout(k.workspace, B, D, h, w, vol_dtype, layout, num_levels, &wl);
        pl.a_km = wl.a_km;
        for (int l = 0; l < rdvc::BLD_MAX_LEVELS; ++l) { pl.b_km[l] = wl.b_km[l]; pl.nl_of[l] = wl.nl_of[l]; }
        pl.twl = wl.twl; pl.thl = wl.thl;
        pl.memset_ptr = wl.memset_ptr; pl.memset_bytes = wl.memset_bytes;
    }
    // operand format: fp16 inputs (the reference's default autocast, R:codec_processing.py:1436) stay fp16
    // -- same tensor-core rate, 11 instead of 8 mantissa bits; everything else is multiplied as bf16
    const CUtensorMapDataType op_dt = k.f16_ops ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;

    // fused mode tile shape: 16x16 fmap2 pixels unless 8x32 wastes less padding
    int tile = k.opt_tile;
    auto padded = [&](int ty, int tx) {
        return static_cast<long long>((h + ty - 1) / ty) * ty * ((w + tx - 1) / tx) * tx;
    };
    if (tile == 0) tile = (padded(8, 32) < padded(16, 16)) ? 2 : 1;
    pl.tile = tile;
    const int TY = (tile == 1) ? 16 : 8, TX = (tile == 1) ? 16 : 32;

    // fmap1 multicast across CTA pairs (experiments library, option key 12 = 3): bit-identical, measured no faster
    // (1080p bf16 0.654 -> 0.646 ms, fp32 unchanged, 1440p 9 % slower: DESIGN.md 3.2) -- the L2 -> SM operand feed is
    // not what bounds the build
    pl.cluster = RDVC_HAS_EXPERIMENTS && pl.linear && sm_count() >= 2 && k.opt_pair == 3;
    // TMA descriptors over the repacked maps
    int rc;
    {
        cuuint64_t dims[3] = {(cuuint64_t)D, (cuuint64_t)N, (cuuint64_t)B};
        cuuint64_t str[2] = {(cuuint64_t)D * 2, (cuuint64_t)N * D * 2};
        cuuint32_t box[3] = {rdvc::BLD_BLOCK_K, static_cast<cuuint32_t>(pl.cluster ? rdvc::BLD_BLOCK_M / 2 : rdvc::BLD_BLOCK_M), 1};
        rc = make_tmap(&pl.ta, op_dt, pl.a_km, 3, dims, str, box);
        if (rc) return rc;
    }
    if (pl.linear) {
        for (int l = 0; l < rdvc::BLD_MAX_LEVELS; ++l) {
            const int ll = l < num_levels ? l : 0;  // unused slots alias level 0
            const cuuint64_t nl = (cuuint64_t)pl.nl_of[ll];
            cuuint64_t dims[3] = {(cuuint64_t)D, nl, (cuuint64_t)B};
            cuuint64_t str[2] = {(cuuint64_t)D * 2, nl * D * 2};
            cuuint32_t box[3] = {rdvc::BLD_BLOCK_K, rdvc::BLD_BLOCK_N, 1};
            rc = make_tmap(&pl.tb[l], op_dt, pl.b_km[ll], 3, dims, str, box);
            if (rc) return rc;
        }
    } else {
        cuuint64_t dims[4] = {(cuuint64_t)D, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)B};
        cuuint64_t str[3] = {(cuuint64_t)D * 2, (cuuint64_t)w * D * 2, (cuuint64_t)N * D * 2};
        cuuint32_t box[4] = {rdvc::BLD_BLOCK_K, (cuuint32_t)TX, (cuuint32_t)TY, 1};
        rc = make_tmap(&pl.tb[0], op_dt, pl.b_km[0], 4, dims, str, box);
        if (rc) return rc;
        pl.tb[1] = pl.tb[2] = pl.tb[3] = pl.tb[0];
    }

    rdvc::BuildParams& p = pl.p;
    for (int l = 0; l < num_levels; ++l) {
        p.lvl[l] = static_cast<uint8_t*>(k.pyramid) + rdvc_corr_level_offset_bytes(B, h, w, l, vol_dtype, layout);
        p.hl[l] = h >> l;
        p.wl[l] = w >> l;
        p.nl[l] = static_cast<int>(pl.nl_of[l]);
    }
    p.B = B; p.h = h; p.w = w; p.N = N;
    p.num_levels = num_levels;
    p.kc = D / 64;
    p.m_blks = (N + rdvc::BLD_BLOCK_M - 1) / rdvc::BLD_BLOCK_M;
    p.nty = (h + TY - 1) / TY;
    p.ntx = (w + TX - 1) / TX;
    if (pl.linear) {
        int t = 0;
        for (int l = 0; l < rdvc::BLD_MAX_LEVELS; ++l) {
            p.tile_start[l] = t;
            if (l < num_levels) t += (p.nl[l] + rdvc::BLD_BLOCK_N - 1) / rdvc::BLD_BLOCK_N;
        }
        p.ntiles = t;
    } else {
        p.ntiles = p.nty * p.ntx;
    }
    p.scale = static_cast<float>(1.0 / std::sqrt(static_cast<double>(D)));
    p.ab_format = k.f16_ops ? 0 : 1;
    p.dbg_store_mask = RDVC_HAS_EXPERIMENTS ? k.opt_store_mask : 15;
    p.dbg_policy = RDVC_HAS_EXPERIMENTS ? k.opt_policy : 0;
    p.msplit = pl.cluster ? choose_msplit(static_cast<long long>(B) * ((p.ntiles + 1) / 2), p.m_blks, sm_count() / 2, k.opt_msplit)
                          : choose_msplit(static_cast<long long>(B) * p.ntiles, p.m_blks, sm_count(), k.opt_msplit);

    // output descriptors (linear mode).  Row pitch a multiple of 128 bytes (always, in the tiled
    // layout): level l as a {128 B, pitch/128, N, B} tensor written in boxes of 16 query rows x 256
    // contiguous bytes.  Row pitch only 16-byte aligned: a {n_l, N, B} tensor, boxes of 32 rows x 128
    // bytes.  Anything else takes the staged-store path.  (option key 5: 0 = staged only, 1 = auto,
    // 2 = never the wide boxes)
    for (int l = 0; l < rdvc::BLD_MAX_LEVELS; ++l) pl.to[l] = pl.tb[0];     // placeholders for levels without a store map
    const int tma_opt = k.opt_tma_out;
    if (pl.linear && tma_opt) {
        const bool f32 = (vol_dtype == RDVC_DT_F32);
        const cuuint64_t es = f32 ? 4 : 2;
        const CUtensorMapDataType dt = f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
        for (int l = 0; l < num_levels; ++l) {
            const cuuint64_t nl = (cuuint64_t)p.nl[l];
            if ((nl * es) % 128 == 0 && tma_opt == 1) {
                cuuint64_t dims[4] = {128 / es, nl * es / 128, (cuuint64_t)N, (cuuint64_t)B};
                cuuint64_t str[3] = {128, nl * es, (cuuint64_t)N * nl * es};
                cuuint32_t box[4] = {(cuuint32_t)(128 / es), 2, 16, 1};
                rc = make_tmap(&pl.to[l], dt, p.lvl[l], 4, dims, str, box);
                if (rc) return rc;
                p.tma_out |= 2 << (2 * l);
            } else if ((nl * es) % 16 == 0) {
                cuuint64_t dims[3] = {nl, (cuuint64_t)N, (cuuint64_t)B};
                cuuint64_t str[2] = {nl * es, (cuuint64_t)N * nl * es};
                cuuint32_t box[3] = {(cuuint32_t)(128 / es), 32, 1};
                rc = make_tmap(&pl.to[l], dt, p.lvl[l], 3, dims, str, box);
                if (rc) return rc;
                p.tma_out |= 1 << (2 * l);
            }
        }
    }
    // epilogue shape per storage type: see BuildCfg (option key 9: 0 = auto, 4 / 8 = force)
    pl.ew = k.opt_epi ? k.opt_epi : ((vol_dtype == RDVC_DT_F32) ? 8 : 4);

#ifdef RDVC_EXPERIMENTS
    // CTA-pair kernel (cta_group::2): linear mode with every level on the wide-box path (always true for
    // the tiled layout).  Option key 12: 0 = auto, 1 = single-CTA kernel, 2 = pair kernel where possible.
    bool pair_ok = pl.linear && (sm_count() >= 2);
    for (int l = 0; l < num_levels; ++l) pair_ok = pair_ok && (((p.tma_out >> (2 * l)) & 3) == 2);
    if (pair_ok && (k.opt_pair == 2 || (k.opt_pair == 0 && RDVC_PAIR_DEFAULT))) {
        for (int l = 0; l < rdvc::BLD_MAX_LEVELS; ++l) {
            const int ll = l < num_levels ? l : 0;
            const cuuint64_t nl = (cuuint64_t)pl.nl_of[ll];
            cuuint64_t dims[3] = {(cuuint64_t)D, nl, (cuuint64_t)B};
            cuuint64_t str[2] = {(cuuint64_t)D * 2, nl * D * 2};
            cuuint32_t box[3] = {rdvc::BLD_BLOCK_K, rdvc::BLD_BLOCK_N / 2, 1};   // each CTA loads half the tile
            rc = make_tmap(&pl.tb2[l], op_dt, pl.b_km[ll], 3, dims, str, box);
            if (rc) return rc;
        }
        pl.p2 = p;
        pl.p2.m_blks = (N + 2 * rdvc::BLD_BLOCK_M - 1) / (2 * rdvc::BLD_BLOCK_M);
        pl.p2.msplit = choose_msplit(static_cast<long long>(B) * pl.p2.ntiles, pl.p2.m_blks, sm_count() / 2, k.opt_msplit);
        pl.pair = true;
    }
#endif
    return RDVC_OK;
}

struct HostArena {  // scratch owned by rdvc_corr_pair_host*, one per (thread, slot), bound to one device
    int device = -1;
    void* dev = nullptr;
    size_t bytes = 0;
    cudaStream_t compute = nullptr, copy = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};   // one per device-side result buffer: its D2H copy finished
    cudaEvent_t done[4] = {nullptr, nullptr, nullptr, nullptr}; // one per device-side result buffer: its lookup finished
    bool pending = false;   // a submitted pair has not been waited for yet
};
constexpr int kHostSlots = 2;
constexpr int kOutBufs = 4;     // lookups run ahead of their device->host copies by up to this many results
thread_local HostArena g_arena[kHostSlots];

void release_arena(HostArena& a) {
    if (a.compute) cudaStreamSynchronize(a.compute);
    if (a.copy) cudaStreamSynchronize(a.copy);
    if (a.dev) cudaFree(a.dev);
    if (a.compute) cudaStreamDestroy(a.compute);
    if (a.copy) cudaStreamDestroy(a.copy);
    for (auto& e : a.ev) if (e) cudaEventDestroy(e);
    for (auto& e : a.done) if (e) cudaEventDestroy(e);
    a = HostArena();
}

}  // namespace

extern "C" {

int rdvc_corr_version(void) { return RDVC_CORR_VERSION; }
const char* rdvc_corr_last_error(void) { return g_err; }
unsigned long long rdvc_corr_launch_count(void) { return g_launches; }

void rdvc_corr_set_profile_events(void* start, void* stop) {
    g_prof_start = static_cast<cudaEvent_t>(start);
    g_prof_stop = static_cast<cudaEvent_t>(stop);
}

int rdvc_corr_set_option(int key, int value) {
    const bool exp = RDVC_HAS_EXPERIMENTS;
    if (key == 0 && value >= 0 && value <= (exp ? 4 : 2)) { g_opt_lookup = value; return RDVC_OK; }
    if (key == 1 && value >= 0 && value <= 2) { g_opt_tile = value; return RDVC_OK; }
    if (key == 2 && value >= 0) { g_opt_msplit = value; return RDVC_OK; }
    if (key == 3 && value >= 0 && value <= 63 && (exp || value == 15)) { g_opt_store_mask = value; return RDVC_OK; }
    if (key == 4 && value >= 0 && value <= 2 && (exp || value != 1)) { g_opt_mode = value; return RDVC_OK; }
    if (key == 5 && value >= 0 && value <= 2) { g_opt_tma_out = value; return RDVC_OK; }
    if (key == 6 && value >= 0 && value <= 2 && (exp || value == 0)) { g_opt_policy = value; return RDVC_OK; }
    if (key == 7 && value >= 0 && value <= 4) { g_opt_twl = value; return RDVC_OK; }
    if (key == 8 && value >= 0 && value <= 4) { g_opt_thl = value; return RDVC_OK; }
    if (key == 9 && (value == 0 || value == 4 || value == 8)) { g_opt_epi_warps = value; return RDVC_OK; }
    if (key == 12 && value >= 0 && value <= 3 && (exp || value <= 1)) { g_opt_pair = value; return RDVC_OK; }
    if (key == 13 && value >= 0 && value <= 16) { g_opt_mcn_prefetch = value; return RDVC_OK; }
    if (key == 14 && value >= 0 && value <= 2) { g_opt_mcn_kernel = value; return RDVC_OK; }
    return fail(RDVC_E_UNSUPPORTED, "unknown option key=%d value=%d%s", key, value,
                exp ? "" : " (work-skipping knobs and the fused / CTA-pair build variants exist in RDVC_EXPERIMENTS builds only)");
}

const char* rdvc_corr_build_info(void) {
    // the marker lets _build.py read the hash out of the file without loading it
    return "RDVC_SRC_HASH=" RDVC_SRC_HASH " version=" RDVC_STR(RDVC_CORR_VERSION) " experiments=" RDVC_STR(RDVC_HAS_EXPERIMENTS);
}

unsigned long long rdvc_corr_plan_cache_hits(void) { return g_plan_hits.load(); }

#ifdef RDVC_EXPERIMENTS
// experiments library only (not in the header): 16 globaltimer stamps per CTA of the next rdvc_conv1x1 launches
void rdvc_exp_conv1x1_timeline(void* device_buffer) { g_dbg_timeline = static_cast<unsigned long long*>(device_buffer); }
void rdvc_exp_conv1x1_flags(int flags) { g_dbg_c1_flags = flags; }     // 1 = no output stores, 2 = no TMEM reads
#endif

size_t rdvc_corr_level_image_elems(int h, int w, int level, int vol_dtype, int layout) {
    if (elem_size(vol_dtype) == 0 || h <= 0 || w <= 0 || level < 0) return 0;
    return level_image_elems(h, w, level, vol_dtype, layout);
}

int rdvc_corr_tile_shape(int vol_dtype, int* tile_w, int* tile_h) {
    if (vol_dtype != RDVC_DT_F32 && vol_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "unsupported vol_dtype=%d", vol_dtype);
    if (!tile_w || !tile_h) return fail(RDVC_E_NULL, "null pointer argument");
    int twl, thl;
    tile_log2(vol_dtype, &twl, &thl);
    *tile_w = 1 << twl;
    *tile_h = 1 << thl;
    return RDVC_OK;
}

size_t rdvc_corr_level_offset_bytes(int B, int h, int w, int level, int vol_dtype, int layout) {
    if ((vol_dtype != RDVC_DT_F32 && vol_dtype != RDVC_DT_BF16) || B <= 0 || h <= 0 || w <= 0 || level < 0) return 0;
    size_t off = 0;
    for (int l = 0; l < level; ++l) off += align_up(level_bytes(B, h, w, l, vol_dtype, layout), 256);
    return off;
}

size_t rdvc_corr_pyramid_bytes(int B, int h, int w, int num_levels, int vol_dtype, int layout) {
    // every level padded to 256 bytes, so 16-byte gathers at a level's tail stay inside
    return rdvc_corr_level_offset_bytes(B, h, w, num_levels, vol_dtype, layout);
}

size_t rdvc_corr_workspace_bytes(int B, int D, int h, int w) {
    // fmap1 K-major + fmap2 K-major at every pyramid level (levels 1..3 are used by the
    // linear build mode only), each 256-byte aligned
    size_t total = align_up(static_cast<size_t>(B) * h * w * D * 2, 256);
    for (int l = 0; l < rdvc::BLD_MAX_LEVELS; ++l)
        total += align_up(static_cast<size_t>(B) * operand_rows_max(h, w, l) * D * 2, 256);
    return total;
}

}  // extern "C"

namespace {
// fmap1 == nullptr: the workspace already holds the K-major operand rows (rdvc_corr_build_packed)
int build_impl(const void* fmap1, const void* fmap2, int B, int D, int h, int w, int in_dtype,
               void* pyramid, int vol_dtype, int layout, int num_levels, void* workspace,
               size_t workspace_bytes, void* stream) {
    const bool packed = (fmap1 == nullptr);
    if ((!packed && !fmap2) || !pyramid || !workspace) return fail(RDVC_E_NULL, "null pointer argument");
    int rc = check_geometry(B, h, w, num_levels);
    if (rc) return rc;
    if (D <= 0) return fail(RDVC_E_SHAPE, "non-positive channel count D=%d", D);
    if (D % 64 != 0 || D > 64 * rdvc::BLD_MAX_KC)
        return fail(RDVC_E_UNSUPPORTED, "D=%d must be a multiple of 64 and <= %d", D, 64 * rdvc::BLD_MAX_KC);
    if (in_dtype != RDVC_DT_F32 && in_dtype != RDVC_DT_BF16 && in_dtype != RDVC_DT_F16)
        return fail(RDVC_E_DTYPE, "unsupported in_dtype=%d", in_dtype);
    if (vol_dtype != RDVC_DT_F32 && vol_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "unsupported vol_dtype=%d", vol_dtype);
    if (layout != RDVC_LAYOUT_ROWMAJOR && layout != RDVC_LAYOUT_TILED)
        return fail(RDVC_E_UNSUPPORTED, "unknown pyramid layout %d", layout);
    if (workspace_bytes < rdvc_corr_workspace_bytes(B, D, h, w))
        return fail(RDVC_E_WORKSPACE, "workspace %zu < required %zu", workspace_bytes,
                    rdvc_corr_workspace_bytes(B, D, h, w));
    if ((reinterpret_cast<uintptr_t>(pyramid) & 255) || (reinterpret_cast<uintptr_t>(workspace) & 255))
        return fail(RDVC_E_ALIGN, "pyramid and workspace must be 256-byte aligned");
    if (static_cast<long long>(h) * w > (1LL << 30) / 4)
        return fail(RDVC_E_UNSUPPORTED, "h*w too large for 32-bit pixel indices");

    cudaStream_t st = static_cast<cudaStream_t>(stream);
    BuildKey key;
    memset(&key, 0, sizeof(key));
    key.device = current_device();
    key.pyramid = pyramid; key.workspace = workspace;
    key.B = B; key.D = D; key.h = h; key.w = w; key.f16_ops = (in_dtype == RDVC_DT_F16) ? 1 : 0;
    key.vol_dtype = vol_dtype; key.layout = layout; key.num_levels = num_levels;
    key.opt_mode = g_opt_mode.load(); key.opt_tile = g_opt_tile.load(); key.opt_msplit = g_opt_msplit.load();
    key.opt_tma_out = g_opt_tma_out.load(); key.opt_epi = g_opt_epi_warps.load(); key.opt_pair = g_opt_pair.load();
    key.opt_twl = g_opt_twl.load(); key.opt_thl = g_opt_thl.load();
    key.opt_store_mask = g_opt_store_mask.load(); key.opt_policy = g_opt_policy.load();

    // The plan (pointers into the workspace, 9 TMA descriptors, work split) depends only on the key: a per-process,
    // mutex-guarded cache of the last few plans makes a repeated call (RAFT calls build once per frame pair with
    // the same buffers) skip the descriptor encoding and the m-split search.
    BuildPlan plan;
    if (!plan_cache_get(key, &plan)) {
        rc = make_build_plan(key, &plan);
        if (rc) return rc;
        plan_cache_put(plan);
    }

    if (plan.memset_bytes && !packed) {
        // padding pixels of a level must come out of the GEMM as exact zeros: clear the operand rows of
        // the levels that have any (the pack kernel writes only real pixels) -- ONE memset from the first
        // padded level to the end of the last level (the per-level buffers are contiguous)
        cudaError_t e = cudaMemsetAsync(plan.memset_ptr, 0, plan.memset_bytes, st);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(padded operand rows)");
    }
    // 1. repack to K-major 16-bit rows; the linear mode also needs the pooled fmap2 levels
    if (packed && !plan.linear) return fail(RDVC_E_UNSUPPORTED, "pre-packed operands need the linear build mode");
    if (!packed) {
        const int levels2 = plan.linear ? num_levels : 1;
        if (in_dtype == RDVC_DT_F32) rc = launch_pack<float>(fmap1, fmap2, plan.a_km, plan.b_km, B, D, h, w, levels2, layout, plan.twl, plan.thl, plan.nl_of, key.f16_ops, st);
        else if (in_dtype == RDVC_DT_BF16) rc = launch_pack<__nv_bfloat16>(fmap1, fmap2, plan.a_km, plan.b_km, B, D, h, w, levels2, layout, plan.twl, plan.thl, plan.nl_of, key.f16_ops, st);
        else rc = launch_pack<__half>(fmap1, fmap2, plan.a_km, plan.b_km, B, D, h, w, levels2, layout, plan.twl, plan.thl, plan.nl_of, key.f16_ops, st);
        if (rc) return rc;
    }
    // 2. the GEMM
    const CUtensorMap& ta = plan.ta;
    const CUtensorMap* tb = plan.tb;
    const CUtensorMap* to = plan.to;
    const rdvc::BuildParams& p = plan.p;
    using rdvc::MODE_LINEAR;
#ifdef RDVC_EXPERIMENTS
    using rdvc::MODE_FUSED;
    if (plan.pair)
        return (vol_dtype == RDVC_DT_F32) ? launch_build_pair<float>(ta, plan.tb2, to, plan.p2, st)
                                          : launch_build_pair<__nv_bfloat16>(ta, plan.tb2, to, plan.p2, st);
    if (!plan.linear) {
        if (vol_dtype == RDVC_DT_F32)
            return (plan.tile == 1) ? launch_build<MODE_FUSED, 16, 16, float, 8>(ta, tb, to, p, st)
                                    : launch_build<MODE_FUSED, 8, 32, float, 8>(ta, tb, to, p, st);
        return (plan.tile == 1) ? launch_build<MODE_FUSED, 16, 16, __nv_bfloat16, 8>(ta, tb, to, p, st)
                                : launch_build<MODE_FUSED, 8, 32, __nv_bfloat16, 8>(ta, tb, to, p, st);
    }
#endif
    // epilogue shape per storage type: see BuildCfg (option key 9: 0 = auto, 4 / 8 = force)
#ifdef RDVC_EXPERIMENTS
    if (plan.cluster) {
        if (vol_dtype == RDVC_DT_F32)
            return plan.ew == 8 ? launch_build<MODE_LINEAR, 16, 16, float, 8, 2>(ta, tb, to, p, st)
                                : launch_build<MODE_LINEAR, 16, 16, float, 4, 2>(ta, tb, to, p, st);
        return plan.ew == 8 ? launch_build<MODE_LINEAR, 16, 16, __nv_bfloat16, 8, 2>(ta, tb, to, p, st)
                            : launch_build<MODE_LINEAR, 16, 16, __nv_bfloat16, 4, 2>(ta, tb, to, p, st);
    }
#endif
    if (vol_dtype == RDVC_DT_F32)
        return plan.ew == 8 ? launch_build<MODE_LINEAR, 16, 16, float, 8>(ta, tb, to, p, st)
                            : launch_build<MODE_LINEAR, 16, 16, float, 4>(ta, tb, to, p, st);
    return plan.ew == 8 ? launch_build<MODE_LINEAR, 16, 16, __nv_bfloat16, 8>(ta, tb, to, p, st)
                        : launch_build<MODE_LINEAR, 16, 16, __nv_bfloat16, 4>(ta, tb, to, p, st);
}
}  // namespace

extern "C" {

int rdvc_corr_build(const void* fmap1, const void* fmap2, int B, int D, int h, int w, int in_dtype,
                    void* pyramid, int vol_dtype, int layout, int num_levels, void* workspace,
                    size_t workspace_bytes, void* stream) {
    if (!fmap1 || !fmap2) return fail(RDVC_E_NULL, "null pointer argument");
    return build_impl(fmap1, fmap2, B, D, h, w, in_dtype, pyramid, vol_dtype, layout, num_levels, workspace,
                      workspace_bytes, stream);
}

int rdvc_corr_build_packed(int B, int D, int h, int w, int op_dtype, void* pyramid, int vol_dtype, int layout,
                           int num_levels, void* workspace, size_t workspace_bytes, void* stream) {
    if (op_dtype != RDVC_DT_BF16 && op_dtype != RDVC_DT_F16)
        return fail(RDVC_E_DTYPE, "packed operands are BF16 or F16, got op_dtype=%d", op_dtype);
    return build_impl(nullptr, nullptr, B, D, h, w, op_dtype, pyramid, vol_dtype, layout, num_levels, workspace,
                      workspace_bytes, stream);
}

}  // extern "C"

namespace {
// pixel_stride 0: NCHW maps (rdvc_corr_pack); > 0: NHWC 16-bit maps at that pixel stride (rdvc_corr_pack_nhwc)
int pack_impl(const void* x1, const void* x2, long long pixel_stride, int B, int D, int h, int w, int in_dtype,
              int vol_dtype, int layout, int num_levels, void* workspace, size_t workspace_bytes, void* stream) {
    if (!x1 || !x2 || !workspace) return fail(RDVC_E_NULL, "null pointer argument");
    int rc = check_geometry(B, h, w, num_levels);
    if (rc) return rc;
    if (D <= 0 || D % 64 != 0 || D > 64 * rdvc::BLD_MAX_KC)
        return fail(RDVC_E_UNSUPPORTED, "D=%d must be a multiple of 64 and <= %d", D, 64 * rdvc::BLD_MAX_KC);
    if (in_dtype != RDVC_DT_F32 && in_dtype != RDVC_DT_BF16 && in_dtype != RDVC_DT_F16)
        return fail(RDVC_E_DTYPE, "unsupported in_dtype=%d", in_dtype);
    if (vol_dtype != RDVC_DT_F32 && vol_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "unsupported vol_dtype=%d", vol_dtype);
    if (layout != RDVC_LAYOUT_ROWMAJOR && layout != RDVC_LAYOUT_TILED)
        return fail(RDVC_E_UNSUPPORTED, "unknown pyramid layout %d", layout);
    if (workspace_bytes < rdvc_corr_workspace_bytes(B, D, h, w))
        return fail(RDVC_E_WORKSPACE, "workspace %zu < required %zu", workspace_bytes, rdvc_corr_workspace_bytes(B, D, h, w));
    if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail(RDVC_E_ALIGN, "workspace must be 256-byte aligned");
    if (pixel_stride) {
        if (in_dtype == RDVC_DT_F32) return fail(RDVC_E_DTYPE, "NHWC maps are F16 or BF16, got in_dtype=%d", in_dtype);
        if (pixel_stride < D) return fail(RDVC_E_UNSUPPORTED, "pixel_stride %lld < D=%d", pixel_stride, D);
        if ((pixel_stride % 8) || ((reinterpret_cast<uintptr_t>(x1) | reinterpret_cast<uintptr_t>(x2)) & 15))
            return fail(RDVC_E_ALIGN, "NHWC maps need 16-byte aligned bases and a pixel stride of a multiple of 8");
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    WorkspaceLayout wl;
    workspace_layout(workspace, B, D, h, w, vol_dtype, layout, num_levels, &wl);
    if (wl.memset_bytes) {
        cudaError_t e = cudaMemsetAsync(wl.memset_ptr, 0, wl.memset_bytes, st);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(padded operand rows)");
    }
    const int f16 = (in_dtype == RDVC_DT_F16) ? 1 : 0;
    if (pixel_stride)
        return f16 ? launch_pack_nhwc<__half>(x1, x2, pixel_stride, wl.a_km, wl.b_km, B, D, h, w, num_levels, layout, wl.twl,
                                              wl.thl, wl.nl_of, f16, st)
                   : launch_pack_nhwc<__nv_bfloat16>(x1, x2, pixel_stride, wl.a_km, wl.b_km, B, D, h, w, num_levels, layout,
                                                     wl.twl, wl.thl, wl.nl_of, f16, st);
    if (in_dtype == RDVC_DT_F32) return launch_pack<float>(x1, x2, wl.a_km, wl.b_km, B, D, h, w, num_levels, layout, wl.twl, wl.thl, wl.nl_of, f16, st);
    if (in_dtype == RDVC_DT_BF16) return launch_pack<__nv_bfloat16>(x1, x2, wl.a_km, wl.b_km, B, D, h, w, num_levels, layout, wl.twl, wl.thl, wl.nl_of, f16, st);
    return launch_pack<__half>(x1, x2, wl.a_km, wl.b_km, B, D, h, w, num_levels, layout, wl.twl, wl.thl, wl.nl_of, f16, st);
}
}  // namespace

extern "C" {

int rdvc_corr_pack(const void* x1, const void* x2, int B, int D, int h, int w, int in_dtype, int vol_dtype,
                   int layout, int num_levels, void* workspace, size_t workspace_bytes, void* stream) {
    return pack_impl(x1, x2, 0, B, D, h, w, in_dtype, vol_dtype, layout, num_levels, workspace, workspace_bytes, stream);
}

int rdvc_corr_pack_nhwc(const void* x1, const void* x2, long long pixel_stride, int B, int D, int h, int w, int in_dtype,
                        int vol_dtype, int layout, int num_levels, void* workspace, size_t workspace_bytes, void* stream) {
    if (pixel_stride <= 0) return fail(RDVC_E_UNSUPPORTED, "pixel_stride must be positive, got %lld", pixel_stride);
    return pack_impl(x1, x2, pixel_stride, B, D, h, w, in_dtype, vol_dtype, layout, num_levels, workspace, workspace_bytes,
                     stream);
}

size_t rdvc_linear_packed_weight_bytes(int cout, int cin) {
    if (cout <= 0 || cin <= 0) return 0;
    return static_cast<size_t>(cout) * cin * 2;
}

int rdvc_linear_pack_weights(const float* weight, int cout, int cin, int dtype, void* packed_host) {
    if (!weight || !packed_host) return fail(RDVC_E_NULL, "null pointer argument");
    if (dtype != RDVC_DT_BF16 && dtype != RDVC_DT_F16) return fail(RDVC_E_DTYPE, "dtype must be BF16 or F16, got %d", dtype);
    if (cout <= 0 || cin <= 0) return fail(RDVC_E_SHAPE, "non-positive dimension cout=%d cin=%d", cout, cin);
    uint16_t* out = static_cast<uint16_t*>(packed_host);
    for (size_t i = 0; i < static_cast<size_t>(cout) * cin; ++i) {
        if (dtype == RDVC_DT_F16) { const __half hv = __float2half_rn(weight[i]); memcpy(out + i, &hv, 2); }
        else { const __nv_bfloat16 bv = __float2bfloat16_rn(weight[i]); memcpy(out + i, &bv, 2); }
    }
    return RDVC_OK;
}

int rdvc_corr_encoder_tail(const void* ws_in, size_t ws_in_bytes, int D_in, const void* packed_w, const float* bias,
                           int D_out, int B, int h, int w, int op_dtype, int vol_dtype, int layout, int num_levels,
                           void* ws_out, size_t ws_out_bytes, void* stream) {
    if (!ws_in || !packed_w || !ws_out) return fail(RDVC_E_NULL, "null pointer argument");
    int rc = check_geometry(B, h, w, num_levels);
    if (rc) return rc;
    if (D_in != rdvc::ET_K || D_out != rdvc::ET_N)
        return fail(RDVC_E_UNSUPPORTED, "the encoder tail is a %d -> %d convolution, got %d -> %d", rdvc::ET_K, rdvc::ET_N, D_in, D_out);
    if (op_dtype != RDVC_DT_BF16 && op_dtype != RDVC_DT_F16)
        return fail(RDVC_E_DTYPE, "operands are BF16 or F16, got op_dtype=%d", op_dtype);
    if (vol_dtype != RDVC_DT_F32 && vol_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "unsupported vol_dtype=%d", vol_dtype);
    if (layout != RDVC_LAYOUT_ROWMAJOR && layout != RDVC_LAYOUT_TILED)
        return fail(RDVC_E_UNSUPPORTED, "unknown pyramid layout %d", layout);
    if (ws_in_bytes < rdvc_corr_workspace_bytes(B, D_in, h, w) || ws_out_bytes < rdvc_corr_workspace_bytes(B, D_out, h, w))
        return fail(RDVC_E_WORKSPACE, "workspaces must hold rdvc_corr_workspace_bytes for D = %d (in) and D = %d (out)", D_in, D_out);
    if ((reinterpret_cast<uintptr_t>(ws_in) & 255) || (reinterpret_cast<uintptr_t>(ws_out) & 255) ||
        (reinterpret_cast<uintptr_t>(packed_w) & 15))
        return fail(RDVC_E_ALIGN, "workspaces must be 256-byte aligned, packed weights 16-byte aligned");
    WorkspaceLayout li, lo;
    workspace_layout(const_cast<void*>(ws_in), B, D_in, h, w, vol_dtype, layout, num_levels, &li);
    workspace_layout(ws_out, B, D_out, h, w, vol_dtype, layout, num_levels, &lo);
    rdvc::EncoderTailParams p;
    memset(&p, 0, sizeof(p));
    const uint8_t* in0 = static_cast<const uint8_t*>(ws_in);
    const uint8_t* out0 = static_cast<const uint8_t*>(ws_out);
    const size_t in_row = static_cast<size_t>(D_in) * 2, out_row = static_cast<size_t>(D_out) * 2;
    int tiles = 0;
    auto add_seg = [&](const void* src, const void* dst, long long rows, int img, int hl, int wl_, int tiles_w) {
        const int s = p.n_segs++;
        p.in_row0[s] = static_cast<long long>((static_cast<const uint8_t*>(src) - in0) / in_row);
        p.out_row0[s] = static_cast<long long>((static_cast<const uint8_t*>(dst) - out0) / out_row);
        p.rows[s] = rows;
        p.tile0[s] = tiles;
        p.img[s] = img; p.hl[s] = hl; p.wl[s] = wl_; p.tiles_w[s] = tiles_w;
        tiles += static_cast<int>((rows + rdvc::ET_BLOCK_M - 1) / rdvc::ET_BLOCK_M);
    };
    add_seg(li.a_km, lo.a_km, static_cast<long long>(B) * h * w, h * w, h, w, 0);                 // image 1: every row real
    for (int l = 0; l < num_levels; ++l) {
        const int hl = h >> l, wl_ = w >> l;
        const bool padded = li.nl_of[l] != static_cast<size_t>(hl) * wl_;
        const int tiles_w = (layout == RDVC_LAYOUT_TILED && padded) ? ((wl_ + (1 << li.twl) - 1) >> li.twl) : 0;
        add_seg(li.b_km[l], lo.b_km[l], static_cast<long long>(B) * static_cast<long long>(li.nl_of[l]),
                static_cast<int>(li.nl_of[l]), hl, wl_, tiles_w);
    }
    p.tile0[p.n_segs] = tiles;
    p.n_tiles = tiles;
    p.twl = li.twl; p.thl = li.thl;
    p.out = ws_out; p.bias = bias; p.ab_format = (op_dtype == RDVC_DT_F16) ? 0 : 1;
    p.dbg_timeline = RDVC_HAS_EXPERIMENTS ? g_dbg_timeline.load() : nullptr;
    const CUtensorMapDataType op_dt = (op_dtype == RDVC_DT_F16) ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    CUtensorMap tm_a, tm_w;
    {
        const cuuint64_t total_rows = ws_in_bytes / in_row;
        if (total_rows >= (1ull << 31)) return fail(RDVC_E_UNSUPPORTED, "too many rows for 32-bit TMA coordinates");
        cuuint64_t dims[3] = {(cuuint64_t)D_in, total_rows, 1};
        cuuint64_t str[2] = {(cuuint64_t)in_row, total_rows * in_row};
        cuuint32_t box[3] = {64, rdvc::ET_BLOCK_M, 1};
        if ((rc = make_tmap(&tm_a, op_dt, const_cast<void*>(ws_in), 3, dims, str, box))) return rc;
    }
    {
        cuuint64_t dims[3] = {(cuuint64_t)D_in, (cuuint64_t)D_out, 1};
        cuuint64_t str[2] = {(cuuint64_t)in_row, (cuuint64_t)D_out * in_row};
        cuuint32_t box[3] = {64, (cuuint32_t)D_out, 1};
        if ((rc = make_tmap(&tm_w, op_dt, const_cast<void*>(packed_w), 3, dims, str, box))) return rc;
    }
    auto kern = rdvc::corr_encoder_tail_kernel;
    static std::atomic<unsigned long long> attr_done{0};
    if ((rc = ensure_dynamic_smem(kern, rdvc::ET_SMEM_LAUNCH, attr_done, "cudaFuncSetAttribute(encoder tail, max dynamic smem)"))) return rc;
    int grid = sm_count();
    if (grid > tiles) grid = tiles;
    kern<<<grid, rdvc::ET_THREADS, rdvc::ET_SMEM_LAUNCH, static_cast<cudaStream_t>(stream)>>>(tm_a, tm_w, p);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "corr_encoder_tail_kernel launch");
    return RDVC_OK;
}

size_t rdvc_corr_feat_pitch(int num_levels, int radius) {
    if (num_levels < 1 || num_levels > rdvc::LKP_MAX_LEVELS || radius < 1 || radius > 4) return 0;
    return static_cast<size_t>(rdvc::lkp_feat_pitch(num_levels, radius));
}

size_t rdvc_corr_feat_rows(int B, int h, int w) {
    if (B <= 0 || h <= 0 || w <= 0) return 0;
    return align_up(static_cast<size_t>(B) * h * w, 8);
}

size_t rdvc_corr_feat_bytes(int B, int h, int w, int num_levels, int radius) {
    return rdvc_corr_feat_pitch(num_levels, radius) * rdvc_corr_feat_rows(B, h, w) * 2;
}

int rdvc_corr_lookup_ex(const void* pyramid, int vol_dtype, int layout, const float* coords, int B, int h,
                        int w, int num_levels, int radius, void* out, int out_dtype, int out_form, void* stream) {
    if (!pyramid || !coords || !out) return fail(RDVC_E_NULL, "null pointer argument");
    int rc = check_geometry(B, h, w, num_levels);
    if (rc) return rc;
    if (vol_dtype != RDVC_DT_F32 && vol_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "unsupported vol_dtype=%d", vol_dtype);
    if (layout != RDVC_LAYOUT_ROWMAJOR && layout != RDVC_LAYOUT_TILED)
        return fail(RDVC_E_UNSUPPORTED, "unknown pyramid layout %d", layout);
    if (reinterpret_cast<uintptr_t>(pyramid) & 15)
        return fail(RDVC_E_ALIGN, "pyramid must be 16-byte aligned");
    if (radius < 1 || radius > 4) return fail(RDVC_E_UNSUPPORTED, "radius=%d not in [1, 4]", radius);
    int out_mode;
    if (out_form == RDVC_OUT_NCHW) {
        if (out_dtype == RDVC_DT_F32) out_mode = rdvc::LKP_OUT_NCHW_F32;
        else if (out_dtype == RDVC_DT_F16) out_mode = rdvc::LKP_OUT_NCHW_F16;
        else return fail(RDVC_E_DTYPE, "NCHW lookup output must be F32 or F16, got out_dtype=%d", out_dtype);
    } else if (out_form == RDVC_OUT_KMAJOR) {
        if (out_dtype == RDVC_DT_BF16) out_mode = rdvc::LKP_OUT_KM_BF16;
        else if (out_dtype == RDVC_DT_F16) out_mode = rdvc::LKP_OUT_KM_F16;
        else return fail(RDVC_E_DTYPE, "K-major feature rows must be BF16 or F16, got out_dtype=%d", out_dtype);
        if (reinterpret_cast<uintptr_t>(out) & 15) return fail(RDVC_E_ALIGN, "feature rows must be 16-byte aligned");
    } else {
        return fail(RDVC_E_UNSUPPORTED, "unknown lookup output form %d", out_form);
    }
    if (out_mode != rdvc::LKP_OUT_NCHW_F32 && layout != RDVC_LAYOUT_TILED)
        return fail(RDVC_E_UNSUPPORTED, "fp16 / K-major lookup outputs need RDVC_LAYOUT_TILED");
    rdvc::LookupParams p;
    memset(&p, 0, sizeof(p));
    for (int l = 0; l < num_levels; ++l) {
        p.lvl[l] = static_cast<const uint8_t*>(pyramid) + rdvc_corr_level_offset_bytes(B, h, w, l, vol_dtype, layout);
        p.hl[l] = h >> l;
        p.wl[l] = w >> l;
        p.img[l] = static_cast<long long>(level_image_elems(h, w, l, vol_dtype, layout));
    }
    if (layout == RDVC_LAYOUT_TILED) {
        tile_log2(vol_dtype, &p.twl, &p.thl);
        for (int l = 0; l < num_levels; ++l) p.tiles_w[l] = ((w >> l) + (1 << p.twl) - 1) >> p.twl;
    }
    p.coords = coords;
    p.out = out;
    p.feat_pitch = rdvc::lkp_feat_pitch(num_levels, radius);
    p.feat_rows = static_cast<long long>(rdvc_corr_feat_rows(B, h, w));
    p.B = B;
    p.N = h * w;
    p.num_levels = num_levels;
    p.total = static_cast<long long>(B) * p.N;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int variant = g_opt_lookup.load();
    if (layout == RDVC_LAYOUT_TILED) {
        const int dbg = variant >= 3 ? variant - 2 : 0;
        return (vol_dtype == RDVC_DT_F32) ? dispatch_lookup_tiled<float>(out_mode, dbg, radius, p, st)
                                          : dispatch_lookup_tiled<__nv_bfloat16>(out_mode, dbg, radius, p, st);
    }
    if (vol_dtype == RDVC_DT_F32) {
        if (variant == 1) return dispatch_lookup_radius<float, 0>(radius, p, st);
        return dispatch_lookup_radius<float, 1>(radius, p, st);
    }
    return dispatch_lookup_radius<__nv_bfloat16, 0>(radius, p, st);
}

int rdvc_corr_lookup(const void* pyramid, int vol_dtype, int layout, const float* coords, int B, int h,
                     int w, int num_levels, int radius, float* out, void* stream) {
    return rdvc_corr_lookup_ex(pyramid, vol_dtype, layout, coords, B, h, w, num_levels, radius, out, RDVC_DT_F32,
                               RDVC_OUT_NCHW, stream);
}

// ---- next row f-1: lookup + MotionEncoder.convcorr1 ------------------------------------------
size_t rdvc_conv1x1_packed_weight_bytes(int cout, int num_levels, int radius) {
    const size_t kp = rdvc_corr_feat_pitch(num_levels, radius);
    if (kp == 0 || cout <= 0 || cout > rdvc::C1_MAX_COUT || cout % 32 != 0) return 0;
    return static_cast<size_t>(cout) * align_up(kp, 64) * 2;
}

int rdvc_conv1x1_pack_weights(const float* weight, int cout, int num_levels, int radius, int feat_dtype,
                              void* packed_host) {
    if (!weight || !packed_host) return fail(RDVC_E_NULL, "null pointer argument");
    if (feat_dtype != RDVC_DT_BF16 && feat_dtype != RDVC_DT_F16)
        return fail(RDVC_E_DTYPE, "feat_dtype must be BF16 or F16, got %d", feat_dtype);
    const size_t kp = rdvc_corr_feat_pitch(num_levels, radius);
    if (kp == 0) return fail(RDVC_E_UNSUPPORTED, "num_levels=%d / radius=%d not supported", num_levels, radius);
    if (cout <= 0 || cout > rdvc::C1_MAX_COUT || cout % 32 != 0)
        return fail(RDVC_E_UNSUPPORTED, "cout=%d must be a multiple of 32 and <= %d", cout, rdvc::C1_MAX_COUT);
    const int S = 2 * radius + 1, PL = rdvc::lkp_level_pitch(radius);
    const size_t kpw = align_up(kp, 64);
    const int cin = num_levels * S * S;
    uint16_t* out = static_cast<uint16_t*>(packed_host);
    memset(out, 0, static_cast<size_t>(cout) * kpw * 2);
    for (int n = 0; n < cout; ++n)
        for (int l = 0; l < num_levels; ++l)
            for (int i = 0; i < S; ++i)          // torchvision channel = l*S*S + i*S + j  (i moves x, TV:raft.py:404-412)
                for (int j = 0; j < S; ++j) {
                    const float v = weight[static_cast<size_t>(n) * cin + l * S * S + i * S + j];
                    uint16_t bits;
                    if (feat_dtype == RDVC_DT_F16) { const __half hv = __float2half_rn(v); memcpy(&bits, &hv, 2); }
                    else { const __nv_bfloat16 bv = __float2bfloat16_rn(v); memcpy(&bits, &bv, 2); }
                    out[static_cast<size_t>(n) * kpw + l * PL + j * S + i] = bits;   // the lookup's column order
                }
    return RDVC_OK;
}

int rdvc_conv1x1(const void* feat, int feat_dtype, const void* packed_w, const float* bias, int B, int h, int w,
                 int num_levels, int radius, int cout, int act, void* out, int out_dtype, void* stream) {
    return rdvc_conv1x1_ex(feat, feat_dtype, packed_w, bias, B, h, w, num_levels, radius, cout, act, out, out_dtype, 0,
                           stream);
}

int rdvc_conv1x1_ex(const void* feat, int feat_dtype, const void* packed_w, const float* bias, int B, int h, int w,
                    int num_levels, int radius, int cout, int act, void* out, int out_dtype, long long out_pixel_stride,
                    void* stream) {
    if (!feat || !packed_w || !out) return fail(RDVC_E_NULL, "null pointer argument");
    if (B <= 0 || h <= 0 || w <= 0) return fail(RDVC_E_SHAPE, "non-positive dimension B=%d h=%d w=%d", B, h, w);
    if (feat_dtype != RDVC_DT_BF16 && feat_dtype != RDVC_DT_F16)
        return fail(RDVC_E_DTYPE, "feat_dtype must be BF16 or F16, got %d", feat_dtype);
    if (out_dtype != RDVC_DT_F32 && out_dtype != RDVC_DT_F16 && out_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "unsupported out_dtype=%d", out_dtype);
    if (act != RDVC_ACT_NONE && act != RDVC_ACT_RELU) return fail(RDVC_E_UNSUPPORTED, "unknown activation %d", act);
    const size_t kp = rdvc_corr_feat_pitch(num_levels, radius);
    if (kp == 0) return fail(RDVC_E_UNSUPPORTED, "num_levels=%d / radius=%d not supported", num_levels, radius);
    if (cout <= 0 || cout > rdvc::C1_MAX_COUT || cout % 32 != 0)
        return fail(RDVC_E_UNSUPPORTED, "cout=%d must be a multiple of 32 and <= %d", cout, rdvc::C1_MAX_COUT);
    if ((reinterpret_cast<uintptr_t>(feat) & 15) || (reinterpret_cast<uintptr_t>(packed_w) & 15))
        return fail(RDVC_E_ALIGN, "feature rows and packed weights must be 16-byte aligned");
    if (out_pixel_stride < 0) return fail(RDVC_E_UNSUPPORTED, "negative out_pixel_stride %lld", out_pixel_stride);
    if (out_pixel_stride > 0) {
        if (out_dtype == RDVC_DT_F32) return fail(RDVC_E_DTYPE, "the NHWC output is 16-bit (F16 or BF16)");
        if (out_pixel_stride < cout)
            return fail(RDVC_E_UNSUPPORTED, "out_pixel_stride %lld < cout %d", out_pixel_stride, cout);
        if ((out_pixel_stride % 8) || (reinterpret_cast<uintptr_t>(out) & 15))
            return fail(RDVC_E_ALIGN, "NHWC output: 16-byte aligned with a pixel stride that is a multiple of 8 elements");
    }
    const long long m_total = static_cast<long long>(B) * h * w;
    if (m_total >= (1LL << 31) - 256) return fail(RDVC_E_UNSUPPORTED, "too many pixels for 32-bit TMA coordinates");
    const size_t kpw = align_up(kp, 64);
    const CUtensorMapDataType op_dt = (feat_dtype == RDVC_DT_F16) ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    CUtensorMap tm_a, tm_w;
    {
        // chunk-major features [kp / 8][rows][8]: 8 consecutive rows of one chunk are 128 contiguous bytes, so the map
        // is {64 elements, rows / 8, chunks}; a box of {64, 16, 8} = 8 chunks x 128 rows lands in shared memory as
        // [chunk][row][16 B], the un-swizzled K-major core-matrix layout (corr_conv1x1_sm100.cuh)
        const cuuint64_t rows = (cuuint64_t)rdvc_corr_feat_rows(B, h, w);
        cuuint64_t dims[3] = {64, rows / 8, (cuuint64_t)kp / 8};
        cuuint64_t str[2] = {128, rows * 16};
        cuuint32_t box[3] = {64, rdvc::C1_BLOCK_M / 8, rdvc::C1_BLOCK_K / 8};
        if (int rc = make_tmap(&tm_a, op_dt, const_cast<void*>(feat), 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_NONE)) return rc;
    }
    {
        cuuint64_t dims[3] = {(cuuint64_t)kpw, (cuuint64_t)cout, 1};
        cuuint64_t str[2] = {(cuuint64_t)kpw * 2, (cuuint64_t)cout * kpw * 2};
        cuuint32_t box[3] = {rdvc::C1_BLOCK_K, (cuuint32_t)(cout / 2), 1};
        if (int rc = make_tmap(&tm_w, op_dt, const_cast<void*>(packed_w), 3, dims, str, box)) return rc;
    }
    rdvc::Conv1x1Params p;
    memset(&p, 0, sizeof(p));
    p.out = out; p.bias = bias; p.m_total = m_total; p.n_pix = h * w; p.cout = cout; p.kp = static_cast<int>(kp);
    p.relu = (act == RDVC_ACT_RELU); p.ab_format = (feat_dtype == RDVC_DT_F16) ? 0 : 1;
    p.dbg_timeline = RDVC_HAS_EXPERIMENTS ? g_dbg_timeline.load() : nullptr;
    p.dbg_flags = RDVC_HAS_EXPERIMENTS ? g_dbg_c1_flags.load() : 0;
    p.vec4 = ((h * w) % 4 == 0) && !(reinterpret_cast<uintptr_t>(out) & 15);
    // every CTA owns a contiguous range of pixel rows (a multiple of 32, one warp's rows), as equal as possible
    const int G = sm_count() & ~1;
    if (G < 2) return fail(RDVC_E_UNSUPPORTED, "the 1x1 convolution runs on CTA pairs: needs at least 2 SMs");
    long long rows = (m_total + G - 1) / G;
    rows = (rows + 31) / 32 * 32;
    p.rows_per_cta = static_cast<int>(rows);
    p.tiles_per_cta = static_cast<int>((rows + rdvc::C1_BLOCK_M - 1) / rdvc::C1_BLOCK_M);
    long long grid = (m_total + rows - 1) / rows;
    grid = (grid + 1) & ~1LL;                                  // whole CTA pairs (a trailing CTA may own no rows)
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    cudaError_t e;
    p.out_ps = out_pixel_stride;
    if (out_pixel_stride > 0 && out_dtype == RDVC_DT_F16)
        e = launch_conv1x1<__half, true>(tm_a, tm_w, p, static_cast<unsigned>(grid), st);
    else if (out_pixel_stride > 0) e = launch_conv1x1<__nv_bfloat16, true>(tm_a, tm_w, p, static_cast<unsigned>(grid), st);
    else if (out_dtype == RDVC_DT_F32) e = launch_conv1x1<float>(tm_a, tm_w, p, static_cast<unsigned>(grid), st);
    else if (out_dtype == RDVC_DT_F16) e = launch_conv1x1<__half>(tm_a, tm_w, p, static_cast<unsigned>(grid), st);
    else e = launch_conv1x1<__nv_bfloat16>(tm_a, tm_w, p, static_cast<unsigned>(grid), st);
    if (e != cudaSuccess) return cuda_fail(e, "corr_conv1x1_kernel launch");
    return RDVC_OK;
}

int rdvc_corr_lookup_conv1x1(const void* pyramid, int vol_dtype, int layout, const float* coords, int B, int h,
                             int w, int num_levels, int radius, const void* packed_w, const float* bias, int cout,
                             int act, int feat_dtype, void* feat_ws, size_t feat_ws_bytes, void* out, int out_dtype,
                             void* stream) {
    return rdvc_corr_lookup_conv1x1_ex(pyramid, vol_dtype, layout, coords, B, h, w, num_levels, radius, packed_w, bias, cout,
                                       act, feat_dtype, feat_ws, feat_ws_bytes, out, out_dtype, 0, stream);
}

int rdvc_corr_lookup_conv1x1_ex(const void* pyramid, int vol_dtype, int layout, const float* coords, int B, int h,
                                int w, int num_levels, int radius, const void* packed_w, const float* bias, int cout,
                                int act, int feat_dtype, void* feat_ws, size_t feat_ws_bytes, void* out, int out_dtype,
                                long long out_pixel_stride, void* stream) {
    if (!feat_ws) return fail(RDVC_E_NULL, "null pointer argument");
    const size_t kp = rdvc_corr_feat_pitch(num_levels, radius);
    if (kp == 0) return fail(RDVC_E_UNSUPPORTED, "num_levels=%d / radius=%d not supported", num_levels, radius);
    if (B <= 0 || h <= 0 || w <= 0) return fail(RDVC_E_SHAPE, "non-positive dimension B=%d h=%d w=%d", B, h, w);
    const size_t need = rdvc_corr_feat_bytes(B, h, w, num_levels, radius);
    if (feat_ws_bytes < need) return fail(RDVC_E_WORKSPACE, "feature workspace %zu < required %zu", feat_ws_bytes, need);
    int rc = rdvc_corr_lookup_ex(pyramid, vol_dtype, layout, coords, B, h, w, num_levels, radius, feat_ws, feat_dtype,
                                 RDVC_OUT_KMAJOR, stream);
    if (rc) return rc;
    return rdvc_conv1x1_ex(feat_ws, feat_dtype, packed_w, bias, B, h, w, num_levels, radius, cout, act, out, out_dtype,
                           out_pixel_stride, stream);
}

int rdvc_motion_warp(const float* prev, const float* flow, int B, int C, int H, int W, int h_in, int w_in,
                     float* warped, float* flow_out, void* stream) {
    if (!flow) return fail(RDVC_E_NULL, "null flow pointer");
    if ((prev == nullptr) != (warped == nullptr))
        return fail(RDVC_E_NULL, "prev and warped must both be given (warp) or both be NULL (resize only)");
    if (!warped && !flow_out) return fail(RDVC_E_NULL, "nothing to compute: warped and flow_out are both NULL");
    if (B <= 0 || H <= 0 || W <= 0 || h_in <= 0 || w_in <= 0 || (prev && C <= 0))
        return fail(RDVC_E_SHAPE, "non-positive dimension B=%d C=%d H=%d W=%d h_in=%d w_in=%d", B, C, H, W, h_in, w_in);
    if (H > 65535 || B > 65535) return fail(RDVC_E_UNSUPPORTED, "H and B must be <= 65535 (grid limits)");
    if (static_cast<long long>(H) * W >= (1LL << 31))
        return fail(RDVC_E_UNSUPPORTED, "H * W must fit 31 bits (in-plane offsets are 32-bit)");
    rdvc::WarpParams p;
    memset(&p, 0, sizeof(p));
    p.prev = prev; p.flow = flow; p.warped = warped; p.flow_out = flow_out;
    p.B = B; p.C = C; p.H = H; p.W = W; p.h_in = h_in; p.w_in = w_in;
    p.ry = static_cast<float>(h_in) / static_cast<float>(H);
    p.rx = static_cast<float>(w_in) / static_cast<float>(W);
    p.sh = static_cast<float>(static_cast<double>(H) / h_in);
    p.sw = static_cast<float>(static_cast<double>(W) / w_in);
    p.same_size = (h_in == H && w_in == W);
    const int per_block = rdvc::WARP_THREADS * rdvc::WARP_PIX;
    dim3 grid((W + per_block - 1) / per_block, H, B);
    rdvc::motion_warp_kernel<<<grid, rdvc::WARP_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(p);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "motion_warp_kernel launch");
    return RDVC_OK;
}

int rdvc_preprocess_frame(const unsigned char* frame_hwc, int H, int W, int C, float* out, int h_out, int w_out,
                          void* stream) {
    if (!frame_hwc || !out) return fail(RDVC_E_NULL, "null pointer argument");
    if (H <= 0 || W <= 0 || h_out <= 0 || w_out <= 0) return fail(RDVC_E_SHAPE, "non-positive dimension H=%d W=%d h_out=%d w_out=%d", H, W, h_out, w_out);
    if (C < 1 || C > 4) return fail(RDVC_E_UNSUPPORTED, "C=%d not in [1, 4]", C);
    if (h_out > 65535) return fail(RDVC_E_UNSUPPORTED, "h_out must be <= 65535 (grid limit)");
    const double sy = static_cast<double>(H) / h_out, sx = static_cast<double>(W) / w_out;
    if (2.0 * (sy > 1 ? sy : 1) + 2 > rdvc::PREP_MAX_TAPS || 2.0 * (sx > 1 ? sx : 1) + 2 > rdvc::PREP_MAX_TAPS)
        return fail(RDVC_E_UNSUPPORTED, "down-scaling by more than %dx is not supported", (rdvc::PREP_MAX_TAPS - 2) / 2);
    rdvc::PrepParams p;
    memset(&p, 0, sizeof(p));
    p.src = frame_hwc; p.dst = out; p.H = H; p.W = W; p.C = C; p.h_out = h_out; p.w_out = w_out;
    p.sy = static_cast<float>(H) / static_cast<float>(h_out);    // aten: area_pixel_compute_scale, fp32
    p.sx = static_cast<float>(W) / static_cast<float>(w_out);
    dim3 grid((w_out + 127) / 128, h_out);
    rdvc::preprocess_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(p);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "preprocess_kernel launch");
    return RDVC_OK;
}

void rdvc_corr_release(void) {
    for (auto& a : g_arena) release_arena(a);
}

int rdvc_corr_pair_host_submit_ex(const float* fmap1_host, const float* fmap2_host, const float* coords_host,
                                  void* out_host, int B, int D, int h, int w, int num_levels, int radius,
                                  int iters, int vol_dtype, int out_dtype, int slot) {
    if (!fmap1_host || !fmap2_host || !coords_host || !out_host) return fail(RDVC_E_NULL, "null pointer argument");
    if (slot < 0 || slot >= kHostSlots) return fail(RDVC_E_UNSUPPORTED, "slot=%d not in [0, %d)", slot, kHostSlots);
    // validated before any size arithmetic or allocation (a bad enum is an argument error, not a crash)
    if (vol_dtype != RDVC_DT_F32 && vol_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "unsupported vol_dtype=%d", vol_dtype);
    if (out_dtype != RDVC_DT_F32 && out_dtype != RDVC_DT_F16)
        return fail(RDVC_E_DTYPE, "out_dtype must be F32 or F16, got %d", out_dtype);
    int rc = check_geometry(B, h, w, num_levels);
    if (rc) return rc;
    if (iters <= 0 || D <= 0) return fail(RDVC_E_SHAPE, "iters=%d D=%d must be positive", iters, D);
    if (radius < 1 || radius > 4) return fail(RDVC_E_UNSUPPORTED, "radius=%d not in [1, 4]", radius);
    const size_t N = static_cast<size_t>(h) * w;
    const size_t S = 2 * radius + 1;
    const size_t oes = (out_dtype == RDVC_DT_F32) ? 4 : 2;
    const size_t fmap_bytes = align_up(static_cast<size_t>(B) * D * N * 4, 256);
    const size_t coords_bytes = align_up(static_cast<size_t>(B) * 2 * N * 4, 256);
    const size_t out_elems = static_cast<size_t>(B) * num_levels * S * S * N;
    const size_t out_bytes = align_up(out_elems * oes, 256);
    const int layout = (g_opt_mode.load() == 1) ? RDVC_LAYOUT_ROWMAJOR : RDVC_LAYOUT_TILED;
    const size_t pyr_bytes = rdvc_corr_pyramid_bytes(B, h, w, num_levels, vol_dtype, layout);
    const size_t ws_bytes = rdvc_corr_workspace_bytes(B, D, h, w);
    const size_t need = 2 * fmap_bytes + iters * coords_bytes + kOutBufs * out_bytes + pyr_bytes + ws_bytes;

    HostArena& a = g_arena[slot];
    cudaError_t e;
    if (a.pending) return fail(RDVC_E_UNSUPPORTED, "slot %d still has a submitted pair: call rdvc_corr_pair_host_wait first", slot);
    if (a.device != current_device()) {   // the caller switched GPUs: streams and scratch belong to the old one
        release_arena(a);
        a.device = current_device();
    }
    if (!a.compute) {
        if ((e = cudaStreamCreateWithFlags(&a.compute, cudaStreamNonBlocking)) != cudaSuccess) return cuda_fail(e, "stream create");
        if ((e = cudaStreamCreateWithFlags(&a.copy, cudaStreamNonBlocking)) != cudaSuccess) return cuda_fail(e, "stream create");
        for (auto& ev : a.ev)
            if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return cuda_fail(e, "event create");
        for (auto& ev : a.done)
            if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return cuda_fail(e, "event create");
    }
    if (a.bytes < need) {
        if (a.dev) cudaFree(a.dev);
        a.dev = nullptr; a.bytes = 0;
        if ((e = cudaMalloc(&a.dev, need)) != cudaSuccess) return cuda_fail(e, "cudaMalloc(scratch arena)");
        a.bytes = need;
    }
    uint8_t* base = static_cast<uint8_t*>(a.dev);
    uint8_t* d_f1 = base;
    uint8_t* d_f2 = d_f1 + fmap_bytes;
    uint8_t* d_co = d_f2 + fmap_bytes;
    uint8_t* d_out[kOutBufs];
    for (int k = 0; k < kOutBufs; ++k) d_out[k] = d_co + iters * coords_bytes + k * out_bytes;
    uint8_t* d_pyr = d_out[kOutBufs - 1] + out_bytes;
    uint8_t* d_ws = d_pyr + pyr_bytes;

    // inputs in (one copy each), then build
    const size_t fmap_raw = static_cast<size_t>(B) * D * N * 4;
    const size_t coords_raw = static_cast<size_t>(B) * 2 * N * 4;
    if ((e = cudaMemcpyAsync(d_f1, fmap1_host, fmap_raw, cudaMemcpyHostToDevice, a.compute)) != cudaSuccess) return cuda_fail(e, "H2D fmap1");
    if ((e = cudaMemcpyAsync(d_f2, fmap2_host, fmap_raw, cudaMemcpyHostToDevice, a.compute)) != cudaSuccess) return cuda_fail(e, "H2D fmap2");
    for (int it = 0; it < iters; ++it)
        if ((e = cudaMemcpyAsync(d_co + it * coords_bytes, coords_host + it * (coords_raw / 4), coords_raw,
                                 cudaMemcpyHostToDevice, a.compute)) != cudaSuccess) return cuda_fail(e, "H2D coords");
    a.pending = true;
    rc = rdvc_corr_build(d_f1, d_f2, B, D, h, w, RDVC_DT_F32, d_pyr, vol_dtype, layout, num_levels, d_ws, ws_bytes, a.compute);
    if (rc) return rc;
    // lookups rotate over kOutBufs device buffers; the copy stream drains them
    bool used[kOutBufs] = {};
    for (int it = 0; it < iters; ++it) {
        const int s = it % kOutBufs;
        if (used[s]) {  // the D2H that last read this buffer must have finished
            if ((e = cudaStreamWaitEvent(a.compute, a.ev[s], 0)) != cudaSuccess) return cuda_fail(e, "wait event");
        }
        rc = rdvc_corr_lookup_ex(d_pyr, vol_dtype, layout, reinterpret_cast<const float*>(d_co + it * coords_bytes), B, h, w,
                                 num_levels, radius, d_out[s], out_dtype, RDVC_OUT_NCHW, a.compute);
        if (rc) return rc;
        // lookup finished -> copy stream may read (the slot's own events, created once with the arena)
        if ((e = cudaEventRecord(a.done[s], a.compute)) != cudaSuccess) return cuda_fail(e, "event record");
        if ((e = cudaStreamWaitEvent(a.copy, a.done[s], 0)) != cudaSuccess) return cuda_fail(e, "wait event");
        if ((e = cudaMemcpyAsync(static_cast<uint8_t*>(out_host) + it * out_elems * oes, d_out[s], out_elems * oes,
                                 cudaMemcpyDeviceToHost, a.copy)) != cudaSuccess) return cuda_fail(e, "D2H out");
        cudaEventRecord(a.ev[s], a.copy);
        used[s] = true;
    }
    return RDVC_OK;
}

int rdvc_corr_pair_host_submit(const float* fmap1_host, const float* fmap2_host, const float* coords_host,
                               float* out_host, int B, int D, int h, int w, int num_levels, int radius,
                               int iters, int vol_dtype, int slot) {
    return rdvc_corr_pair_host_submit_ex(fmap1_host, fmap2_host, coords_host, out_host, B, D, h, w, num_levels, radius,
                                         iters, vol_dtype, RDVC_DT_F32, slot);
}

int rdvc_corr_pair_host_wait(int slot) {
    if (slot < 0 || slot >= kHostSlots) return fail(RDVC_E_UNSUPPORTED, "slot=%d not in [0, %d)", slot, kHostSlots);
    HostArena& a = g_arena[slot];
    if (!a.pending) return RDVC_OK;
    a.pending = false;
    cudaError_t e;
    if ((e = cudaStreamSynchronize(a.compute)) != cudaSuccess) return cuda_fail(e, "sync compute");
    if ((e = cudaStreamSynchronize(a.copy)) != cudaSuccess) return cuda_fail(e, "sync copy");
    return RDVC_OK;
}

int rdvc_corr_pair_host(const float* fmap1_host, const float* fmap2_host, const float* coords_host,
                        float* out_host, int B, int D, int h, int w, int num_levels, int radius,
                        int iters, int vol_dtype) {
    int rc = rdvc_corr_pair_host_wait(0);
    if (rc) return rc;
    rc = rdvc_corr_pair_host_submit(fmap1_host, fmap2_host, coords_host, out_host, B, D, h, w, num_levels, radius,
                                    iters, vol_dtype, 0);
    const int rw = rdvc_corr_pair_host_wait(0);
    return rc ? rc : rw;
}

}  // extern "C"

// ---- next row f-4 (cont.): motion compensation network ----------------------------------------
namespace {

int mcn_check_geometry(int B, int H, int W) {
    if (B <= 0 || H <= 0 || W <= 0) return fail(RDVC_E_SHAPE, "non-positive dimension B=%d H=%d W=%d", B, H, W);
    if (H > 65535 || B > 65535) return fail(RDVC_E_UNSUPPORTED, "H and B must be <= 65535 (grid limits)");
    if (static_cast<long long>(B) * ((H + 7) / 8) * (((W + 1) / 2 + rdvc::MCNX_TXO - 1) / rdvc::MCNX_TXO) >= (1LL << 31))
        return fail(RDVC_E_UNSUPPORTED, "too many tiles for 32-bit tile indices");
    return RDVC_OK;
}

// XH = false: mcn_conv_kernel (three boxes per tile); XH = true: mcn_convx_kernel (one box per tile, 14 output columns)
template <int R, int NOUT, int KPAT, bool XH>
int launch_mcn_conv_impl(const void* act_in, const void* packed_w, void* act_out, rdvc::McnConvParams& p, cudaStream_t st) {
    using Cfg = rdvc::McnCfg<R, NOUT>;
    constexpr int SMEM = XH ? rdvc::McnXCfg<R, NOUT>::SMEM_LAUNCH : Cfg::SMEM_LAUNCH;
    auto kern = XH ? rdvc::mcn_convx_kernel<R, NOUT, KPAT> : rdvc::mcn_conv_kernel<R, NOUT, KPAT>;
    static std::atomic<unsigned long long> attr_done{0};
    if (int rc = ensure_dynamic_smem(kern, SMEM, attr_done, "cudaFuncSetAttribute(mcn_conv, max dynamic smem)"))
        return rc;
    const int out_cols = XH ? rdvc::MCNX_TXO : rdvc::MCN_TX;
    p.ntx = (p.Wsp + out_cols - 1) / out_cols;
    const cuuint64_t Wsp = static_cast<cuuint64_t>(p.Wsp), H = static_cast<cuuint64_t>(p.H), B = static_cast<cuuint64_t>(p.B);
    CUtensorMap tm_in, tm_w, tm_out, tm_res;
    {
        const cuuint64_t dims[4] = {64, Wsp, H, B};
        const cuuint64_t strides[3] = {128, Wsp * 128, H * Wsp * 128};
        const cuuint32_t box_in[4] = {64, rdvc::MCN_TX, static_cast<cuuint32_t>(Cfg::BOX_ROWS), 1};
        if (int rc = make_tmap(&tm_in, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, const_cast<void*>(act_in), 4, dims, strides, box_in))
            return rc;
        // the last layer writes NCHW fp32 itself; its store map is a placeholder on the input tensor
        const cuuint32_t box_out[4] = {64, static_cast<cuuint32_t>(out_cols), 2, 1};
        if (int rc = make_tmap(&tm_out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, act_out ? act_out : const_cast<void*>(act_in), 4,
                               dims, strides, box_out))
            return rc;
        tm_res = tm_out;
        if (p.residual)
            if (int rc = make_tmap(&tm_res, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, const_cast<__half*>(p.residual), 4, dims,
                                   strides, box_out))
                return rc;
    }
    {
        const cuuint64_t dims[3] = {64, static_cast<cuuint64_t>(NOUT), static_cast<cuuint64_t>(Cfg::NTAPS)};
        const cuuint64_t strides[2] = {128, static_cast<cuuint64_t>(NOUT) * 128};
        const cuuint32_t box[3] = {64, static_cast<cuuint32_t>(NOUT), 1};
        if (int rc = make_tmap(&tm_w, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, const_cast<void*>(packed_w), 3, dims, strides, box))
            return rc;
    }
    long long grid = sm_count();
    const long long n_tiles = static_cast<long long>(p.B) * p.ntx * p.nty;
    if (grid > n_tiles) grid = n_tiles;
    kern<<<static_cast<unsigned>(grid), rdvc::MCN_THREADS, SMEM, st>>>(tm_in, tm_w, tm_out, tm_res, p);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "mcn_conv_kernel launch");
    return RDVC_OK;
}

template <int R, int NOUT, int KPAT>
int launch_mcn_conv(const void* act_in, const void* packed_w, void* act_out, rdvc::McnConvParams& p, cudaStream_t st) {
    // auto (measured at 1080p, us per layer, three boxes / one box): 3x3 68 / 58, first layer 103 / 89 -- but with a
    // residual 77 / 81 and for the output layer 88 / 98 (the one-box epilogue does more work per tile)
    const int k = g_opt_mcn_kernel.load();
    const bool xh = (k == 2) || (k == 0 && NOUT == 64 && p.residual == nullptr);
    return xh ? launch_mcn_conv_impl<R, NOUT, KPAT, true>(act_in, packed_w, act_out, p, st)
              : launch_mcn_conv_impl<R, NOUT, KPAT, false>(act_in, packed_w, act_out, p, st);
}

int mcn_fill_params(rdvc::McnConvParams& p, int B, int H, int W, const float* bias, int nbias) {
    memset(&p, 0, sizeof(p));
    p.B = B; p.H = H; p.W = W; p.Wsp = (W + 1) / 2;
    p.ntx = (p.Wsp + rdvc::MCN_TX - 1) / rdvc::MCN_TX;
    p.nty = (H + rdvc::MCN_TY - 1) / rdvc::MCN_TY;
    if (bias) for (int i = 0; i < nbias; ++i) p.bias[i] = bias[i];
    p.prefetch_dist = g_opt_mcn_prefetch.load();
    return RDVC_OK;
}

}  // namespace

extern "C" {

size_t rdvc_mcn_plane_bytes(int B, int H, int W) {
    if (B <= 0 || H <= 0 || W <= 0) return 0;
    return align_up(static_cast<size_t>(B) * H * ((W + 1) / 2) * 128, 1024);
}

size_t rdvc_mcn_workspace_bytes(int B, int H, int W) { return 3 * rdvc_mcn_plane_bytes(B, H, W); }

size_t rdvc_mcn_packed_weight_bytes(int ksize, int cout) {
    if ((ksize != 3 && ksize != 5) || cout <= 0 || cout > rdvc::MCN_C) return 0;
    const int nout = (cout > 8) ? 64 : 16;
    return static_cast<size_t>(ksize) * 3 * nout * 64 * 2;
}

int rdvc_mcn_pack_weights(const float* weight, int cout, int cin, int ksize, void* packed_host,
                          unsigned long long* kmask) {
    if (!weight || !packed_host || !kmask) return fail(RDVC_E_NULL, "null pointer argument");
    if (ksize != 3 && ksize != 5) return fail(RDVC_E_UNSUPPORTED, "kernel size %d not in {3, 5}", ksize);
    if (cin <= 0 || cin > rdvc::MCN_C || cout <= 0 || cout > rdvc::MCN_C)
        return fail(RDVC_E_UNSUPPORTED, "channel counts must be in [1, %d], got cin=%d cout=%d", rdvc::MCN_C, cin, cout);
    const int R = ksize / 2, nout = (cout > 8) ? 64 : 16, co_n = nout / 2;
    __half* out = static_cast<__half*>(packed_host);
    unsigned long long mask = 0;
    for (int dy = -R; dy <= R; ++dy)
        for (int dsx = -1; dsx <= 1; ++dsx) {
            const int t = (dy + R) * 3 + (dsx + 1);
            for (int n = 0; n < nout; ++n) {
                const int q = n / co_n, co = n % co_n;
                for (int k = 0; k < 64; ++k) {
                    const int pp = k / rdvc::MCN_C, ci = k % rdvc::MCN_C;
                    const int dx = 2 * dsx + pp - q;
                    float v = 0.f;
                    if (co < cout && ci < cin && dx >= -R && dx <= R)
                        v = weight[((static_cast<size_t>(co) * cin + ci) * ksize + (dy + R)) * ksize + (dx + R)];
                    const __half hv = __float2half_rn(v);
                    out[(static_cast<size_t>(t) * nout + n) * 64 + k] = hv;
                    if (__half2float(hv) != 0.f) mask |= 1ull << (4 * t + k / 16);
                }
            }
        }
    *kmask = mask;
    return RDVC_OK;
}

int rdvc_mcn_pack_input(const float* warped, const float* flow, const float* ref, int B, int c_warped, int c_flow,
                        int c_ref, int H, int W, void* act, void* stream) {
    if (!warped || !flow || !ref || !act) return fail(RDVC_E_NULL, "null pointer argument");
    if (int rc = mcn_check_geometry(B, H, W)) return rc;
    if (c_warped < 0 || c_flow < 0 || c_ref < 0 || c_warped + c_flow + c_ref > 8 || c_warped + c_flow + c_ref <= 0)
        return fail(RDVC_E_UNSUPPORTED, "input channels %d + %d + %d must sum to 1..8", c_warped, c_flow, c_ref);
    if (reinterpret_cast<uintptr_t>(act) % 16) return fail(RDVC_E_ALIGN, "activation buffer must be 16-byte aligned");
    rdvc::McnInputParams p;
    memset(&p, 0, sizeof(p));
    p.src[0] = warped; p.src[1] = flow; p.src[2] = ref;
    p.ch[0] = c_warped; p.ch[1] = c_flow; p.ch[2] = c_ref;
    p.dst = static_cast<__half*>(act);
    p.B = B; p.H = H; p.W = W; p.Wsp = (W + 1) / 2;
    dim3 grid((2 * p.Wsp + 127) / 128, H, B);
    rdvc::mcn_pack_input_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(p);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "mcn_pack_input_kernel launch");
    return RDVC_OK;
}

int rdvc_mcn_conv(const void* act_in, const void* packed_weights, unsigned long long kmask, const float* bias,
                  int ksize, int act, const void* residual, void* act_out, int B, int H, int W, void* stream) {
    if (!act_in || !packed_weights || !act_out) return fail(RDVC_E_NULL, "null pointer argument");
    if (ksize != 3 && ksize != 5) return fail(RDVC_E_UNSUPPORTED, "kernel size %d not in {3, 5}", ksize);
    const int reverse = (act & RDVC_MCN_REVERSE_ORDER) ? 1 : 0;
    act &= ~RDVC_MCN_REVERSE_ORDER;
    if (act != RDVC_MCN_ACT_NONE && act != RDVC_MCN_ACT_LEAKY) return fail(RDVC_E_UNSUPPORTED, "unknown activation %d", act);
    if (int rc = mcn_check_geometry(B, H, W)) return rc;
    if (act_in == act_out) return fail(RDVC_E_UNSUPPORTED, "a layer cannot run in place (neighbouring tiles read its input)");
    if (reinterpret_cast<uintptr_t>(act_in) % 16 || reinterpret_cast<uintptr_t>(act_out) % 16 ||
        reinterpret_cast<uintptr_t>(packed_weights) % 16 || reinterpret_cast<uintptr_t>(residual) % 16)
        return fail(RDVC_E_ALIGN, "activation / weight buffers must be 16-byte aligned");
    rdvc::McnConvParams p;
    mcn_fill_params(p, B, H, W, bias, rdvc::MCN_C);
    p.act = act;
    p.reverse = reverse;
    p.residual = static_cast<const __half*>(residual);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // the cheapest compile-time MMA schedule that covers the non-zero k-steps of these weights
    auto covered = [&](int kpat) { return (kmask & ~rdvc::mcn_pattern_mask(kpat, ksize)) == 0; };
    if (ksize == 3) {
        if (covered(rdvc::MCN_K_3X3)) return launch_mcn_conv<1, 64, rdvc::MCN_K_3X3>(act_in, packed_weights, act_out, p, st);
        return launch_mcn_conv<1, 64, rdvc::MCN_K_FULL>(act_in, packed_weights, act_out, p, st);
    }
    if (covered(rdvc::MCN_K_C16)) return launch_mcn_conv<2, 64, rdvc::MCN_K_C16>(act_in, packed_weights, act_out, p, st);
    return launch_mcn_conv<2, 64, rdvc::MCN_K_FULL>(act_in, packed_weights, act_out, p, st);
}

int rdvc_mcn_conv_out(const void* act_in, const void* packed_weights, unsigned long long kmask, const float* bias,
                      int ksize, int cout, const float* warped, float* out, int B, int H, int W, void* stream) {
    if (!act_in || !packed_weights || !warped || !out) return fail(RDVC_E_NULL, "null pointer argument");
    if (ksize != 5) return fail(RDVC_E_UNSUPPORTED, "the output layer is 5x5 (got %d)", ksize);
    if (cout <= 0 || cout > 8) return fail(RDVC_E_UNSUPPORTED, "output channels %d not in [1, 8]", cout);
    if (int rc = mcn_check_geometry(B, H, W)) return rc;
    if (reinterpret_cast<uintptr_t>(act_in) % 16 || reinterpret_cast<uintptr_t>(packed_weights) % 16)
        return fail(RDVC_E_ALIGN, "activation / weight buffers must be 16-byte aligned");
    if ((W % 2 == 0) && (reinterpret_cast<uintptr_t>(warped) % 8 || reinterpret_cast<uintptr_t>(out) % 8))
        return fail(RDVC_E_ALIGN, "warped / out must be 8-byte aligned");
    rdvc::McnConvParams p;
    mcn_fill_params(p, B, H, W, bias, cout);
    p.cout = cout;
    p.warped = warped;
    p.out = out;
    (void)kmask;   // the output layer always runs the full schedule
    return launch_mcn_conv<2, 16, rdvc::MCN_K_FULL>(act_in, packed_weights, nullptr, p, static_cast<cudaStream_t>(stream));
}

int rdvc_mcn_forward(const float* warped, const float* flow, const float* ref, int B, int H, int W,
                     int num_res_blocks, const void* const* packed_weights, const unsigned long long* kmasks,
                     const float* biases, void* workspace, size_t workspace_bytes, float* out, void* stream) {
    if (!warped || !flow || !ref || !packed_weights || !kmasks || !biases || !workspace || !out)
        return fail(RDVC_E_NULL, "null pointer argument");
    if (num_res_blocks < 0 || num_res_blocks > 64) return fail(RDVC_E_UNSUPPORTED, "num_res_blocks=%d", num_res_blocks);
    if (int rc = mcn_check_geometry(B, H, W)) return rc;
    const size_t plane = rdvc_mcn_plane_bytes(B, H, W);
    if (workspace_bytes < 3 * plane)
        return fail(RDVC_E_WORKSPACE, "workspace too small: %zu < %zu bytes", workspace_bytes, 3 * plane);
    if (reinterpret_cast<uintptr_t>(workspace) % 256) return fail(RDVC_E_ALIGN, "workspace must be 256-byte aligned");
    char* ws = static_cast<char*>(workspace);
    void* t = ws;                 // network input, then every block's middle activation
    void* x = ws + plane;         // block input (kept for the residual)
    void* y = ws + 2 * plane;     // block output
    const int n_layers = 2 + 2 * num_res_blocks;
    if (int rc = rdvc_mcn_pack_input(warped, flow, ref, B, 3, 2, 3, H, W, t, stream)) return rc;
    // Successive layers walk the tiles in opposite directions: a plane (133 MB at 1080p) is about the size of
    // the L2, so the part of it the previous launch wrote LAST is still cached when the next launch starts --
    // reading it first turns those loads into L2 hits.  The input pack writes first-to-last, so layer 0 runs
    // last-to-first; the output layer (odd index) runs first-to-last.
    const int REV = RDVC_MCN_REVERSE_ORDER;
    if (int rc = rdvc_mcn_conv(t, packed_weights[0], kmasks[0], biases, 5, RDVC_MCN_ACT_LEAKY | REV, nullptr, x, B, H, W, stream))
        return rc;
    for (int r = 0; r < num_res_blocks; ++r) {
        const int l = 1 + 2 * r;
        if (int rc = rdvc_mcn_conv(x, packed_weights[l], kmasks[l], biases + l * 32, 3, RDVC_MCN_ACT_LEAKY, nullptr, t,
                                   B, H, W, stream))                                   // odd layer: first-to-last
            return rc;
        if (int rc = rdvc_mcn_conv(t, packed_weights[l + 1], kmasks[l + 1], biases + (l + 1) * 32, 3, RDVC_MCN_ACT_LEAKY | REV,
                                   x, y, B, H, W, stream))                             // even layer: last-to-first
            return rc;
        void* tmp = x; x = y; y = tmp;
    }
    return rdvc_mcn_conv_out(x, packed_weights[n_layers - 1], kmasks[n_layers - 1], biases + (n_layers - 1) * 32, 5, 3,
                             warped, out, B, H, W, stream);
}

}  // extern "C"

// ---- the tap-convolution engine (tap_conv_sm100.cuh): tensor maps, tile grid, launches ----------------------------
namespace {

// {C, W, H, B} over NHWC 16-bit activations with pixel stride `ps` elements, box {64, box_x, box_y, 1}; `yx` lists y
// before x (the GRU's 1x5 pass convolves along the map's third dimension), `s2` reads every second pixel and row
int act_map(CUtensorMap* m, CUtensorMapDataType dt, const void* base, long long ps, int C, int B, int H, int W, int box_x,
            int box_y, bool yx = false, bool s2 = false) {
    const cuuint64_t px = static_cast<cuuint64_t>(ps) * 2, row = px * W;
    const cuuint64_t dims[4] = {static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(yx ? H : W),
                                static_cast<cuuint64_t>(yx ? W : H), static_cast<cuuint64_t>(B)};
    const cuuint64_t strides[3] = {yx ? row : px, yx ? px : row, row * H};
    const cuuint32_t box[4] = {64, static_cast<cuuint32_t>(box_x), static_cast<cuuint32_t>(box_y), 1};
    const cuuint32_t estr[4] = {1, 2, 2, 1};
    return make_tmap(m, dt, const_cast<void*>(base), 4, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B,
                     s2 ? estr : nullptr);
}

// `slabs` weight slabs of n x 64 16-bit values, one slab per box
int slab_map(CUtensorMap* m, CUtensorMapDataType dt, const void* base, int n, int slabs) {
    const cuuint64_t dims[3] = {64, static_cast<cuuint64_t>(n), static_cast<cuuint64_t>(slabs)};
    const cuuint64_t strides[2] = {128, static_cast<cuuint64_t>(n) * 128};
    const cuuint32_t box[3] = {64, static_cast<cuuint32_t>(n), 1};
    return make_tmap(m, dt, const_cast<void*>(base), 3, dims, strides, box);
}

CUtensorMapDataType op_map_dtype(int op_dtype) {
    return op_dtype == RDVC_DT_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
}

// parameters of one launch over the output grid B x H x W, with its tile grid; everything else zero
rdvc::TapParams tap_params(int B, int H, int W, int n_kb, int horiz = 0) {
    rdvc::TapParams p;
    memset(&p, 0, sizeof(p));
    p.B = B; p.H = H; p.W = W;
    p.n_kb = n_kb;
    p.horiz = horiz;
    p.n_tx = ((horiz ? H : W) + rdvc::TAP_TX - 1) / rdvc::TAP_TX;
    p.n_ty = ((horiz ? W : H) + rdvc::TAP_TY - 1) / rdvc::TAP_TY;
    const long long n_tiles = static_cast<long long>(B) * p.n_tx * p.n_ty;
    p.n_tiles = static_cast<int>(n_tiles);
    p.n_super = static_cast<int>((n_tiles + rdvc::TAP_P - 1) / rdvc::TAP_P);
    return p;
}

template <int G, int N, int EPI, typename OutT, typename OpT>
int launch_tap_conv(const rdvc::TapMaps<rdvc::TapGeom<G>::MAPS>& maps, const rdvc::TapParams& p, cudaStream_t st) {
    constexpr int SMEM = rdvc::TapCfg<G, N, EPI>::SMEM_LAUNCH;
    auto kern = rdvc::tap_conv_kernel<G, N, EPI, OutT, OpT>;
    static std::atomic<unsigned long long> attr_done{0};
    if (int rc = ensure_dynamic_smem(kern, SMEM, attr_done, "cudaFuncSetAttribute(tap_conv, max dynamic smem)")) return rc;
    const int grid = std::min(sm_count(), p.n_super);
    kern<<<grid, rdvc::TAP_THREADS, SMEM, st>>>(maps, p);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "tap_conv_kernel launch");
    return RDVC_OK;
}

template <int G, int N, int EPI, typename OpT>
int launch_tap_conv_in(const rdvc::TapMaps<rdvc::TapGeom<G>::MAPS>& maps, const rdvc::TapParams& p, cudaStream_t st) {
    constexpr int SMEM = rdvc::TapCfg<G, N, EPI>::SMEM_LAUNCH;
    auto kern = rdvc::tap_conv_in_kernel<G, N, EPI, OpT>;
    static std::atomic<unsigned long long> attr_done{0};
    if (int rc = ensure_dynamic_smem(kern, SMEM, attr_done, "cudaFuncSetAttribute(tap_conv_in, max dynamic smem)"))
        return rc;
    const int grid = std::min(sm_count(), p.n_super);
    kern<<<grid, rdvc::TAP_THREADS, SMEM, st>>>(maps, p);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "tap_conv_in_kernel launch");
    return RDVC_OK;
}

// Shared memory and TMEM columns of every (geometry, N, epilogue) the dispatch tables instantiate: the tile and ring
// sizes these kernels are measured with.  A change that moves one of them is a performance change.
template <int G, int N, int EPI>
constexpr bool tap_cfg_is(int smem, int tmem) {
    return rdvc::TapCfg<G, N, EPI>::SMEM_LAUNCH == smem && rdvc::TapCfg<G, N, EPI>::TMEM_COLS == tmem;
}
static_assert(tap_cfg_is<rdvc::TAP_G_GRU5, 256, rdvc::TAP_EPI_GRU_ZR>(197888, 512), "GRU z|r");
static_assert(tap_cfg_is<rdvc::TAP_G_GRU5, 128, rdvc::TAP_EPI_GRU_Q>(165120, 256), "GRU q");
static_assert(tap_cfg_is<rdvc::TAP_G_S1, 192, rdvc::TAP_EPI_RELU>(181504, 512), "convcorr2");
static_assert(tap_cfg_is<rdvc::TAP_G_S1, 64, rdvc::TAP_EPI_RELU>(115968, 128), "convflow2, layer1");
static_assert(tap_cfg_is<rdvc::TAP_G_S1, 256, rdvc::TAP_EPI_RELU>(214272, 512), "flow_head.conv1");
static_assert(tap_cfg_is<rdvc::TAP_G_S1, 128, rdvc::TAP_EPI_RELU_FLOW>(148736, 256), "conv");
static_assert(tap_cfg_is<rdvc::TAP_G_S1, 16, rdvc::TAP_EPI_FLOW2>(91392, 32), "flow_head.conv2");
static_assert(tap_cfg_is<rdvc::TAP_G_STEM, 64, rdvc::TAP_EPI_RELU>(124160, 128), "stem");
static_assert(tap_cfg_is<rdvc::TAP_G_S1, 64, rdvc::TAP_EPI_RES>(115968, 128), "layer1 residual");
static_assert(tap_cfg_is<rdvc::TAP_G_S1, 128, rdvc::TAP_EPI_RELU>(148736, 256), "layer2/3");
static_assert(tap_cfg_is<rdvc::TAP_G_S1, 128, rdvc::TAP_EPI_RES>(148736, 256), "layer2/3 residual");
static_assert(tap_cfg_is<rdvc::TAP_G_S2, 128, rdvc::TAP_EPI_DS>(140544, 512), "stride 2 + downsample");
static_assert(tap_cfg_is<rdvc::TAP_G_1X1, 256, rdvc::TAP_EPI_RAW>(197888, 512), "1x1");
static_assert(tap_cfg_is<rdvc::TAP_G_1X1, 256, rdvc::TAP_EPI_SPLIT>(197888, 512), "1x1 split");
// the feature encoder's statistics epilogues: the context encoder's rings plus 2 tiles x 4 warps x NT (mean, M2)
static_assert(tap_cfg_is<rdvc::TAP_G_STEM, 64, rdvc::TAP_EPI_STATS>(128256, 128), "stem, statistics");
static_assert(tap_cfg_is<rdvc::TAP_G_S1, 64, rdvc::TAP_EPI_STATS>(120064, 128), "layer1, statistics");
static_assert(tap_cfg_is<rdvc::TAP_G_S1, 128, rdvc::TAP_EPI_STATS>(156928, 256), "layer2/3, statistics");
static_assert(tap_cfg_is<rdvc::TAP_G_S2, 128, rdvc::TAP_EPI_DS_STATS>(156928, 512), "stride 2 + downsample, statistics");

// fp32 activations -> 16-bit NHWC operand copies (128 channels of each of the first n_src sources of cp)
int launch_gru_cast(const rdvc::GruCastParams& cp, int n_src, int op_dtype, cudaStream_t st) {
    const dim3 grid(static_cast<unsigned>((cp.n_pix * (rdvc::GRU_C / 8) + 255) / 256), n_src);
    if (op_dtype == RDVC_DT_F16) rdvc::convgru_cast_kernel<__half><<<grid, 256, 0, st>>>(cp);
    else rdvc::convgru_cast_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(cp);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "convgru_cast_kernel launch");
    return RDVC_OK;
}

}  // namespace

// ---- RAFT's recurrent block: one ConvGRU pass as two tcgen05 implicit GEMMs ------------------------------------
namespace {

size_t gru_plane_bytes(int B, int H, int W) {
    return align_up(static_cast<size_t>(B) * H * W * rdvc::GRU_C * 2, 256);
}

template <typename ActT, typename OpT>
int launch_convgru(const rdvc::TapMaps<3>& m_zr, const rdvc::TapMaps<3>& m_q, const rdvc::TapParams& p_zr,
                   const rdvc::TapParams& p_q, cudaStream_t st) {
    if (int rc = launch_tap_conv<rdvc::TAP_G_GRU5, rdvc::GRU_ZR_N, rdvc::TAP_EPI_GRU_ZR, ActT, OpT>(m_zr, p_zr, st))
        return rc;
    return launch_tap_conv<rdvc::TAP_G_GRU5, rdvc::GRU_Q_N, rdvc::TAP_EPI_GRU_Q, ActT, OpT>(m_q, p_q, st);
}

uint16_t gru_round16(float v, int op_dtype) {
    uint16_t bits;
    if (op_dtype == RDVC_DT_F16) { const __half hv = __float2half_rn(v); memcpy(&bits, &hv, 2); }
    else { const __nv_bfloat16 bv = __float2bfloat16_rn(v); memcpy(&bits, &bv, 2); }
    return bits;
}

}  // namespace

extern "C" {

size_t rdvc_corr_convgru_packed_weight_bytes(void) {
    return static_cast<size_t>(rdvc::GRU_W_ZR_ELEMS + rdvc::GRU_W_Q_ELEMS) * 2;
}

int rdvc_corr_convgru_pack_weights(const float* wz, const float* wr, const float* wq, int op_dtype, void* packed_host) {
    if (!wz || !wr || !wq || !packed_host) return fail(RDVC_E_NULL, "null pointer argument");
    if (op_dtype != RDVC_DT_F16 && op_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "op_dtype must be F16 or BF16, got %d", op_dtype);
    constexpr int CIN = rdvc::GRU_KB * 64, T = rdvc::GRU_TAPS;
    uint16_t* zr = static_cast<uint16_t*>(packed_host);
    uint16_t* qq = zr + rdvc::GRU_W_ZR_ELEMS;
    for (int kb = 0; kb < rdvc::GRU_KB; ++kb)
        for (int t = 0; t < T; ++t)
            for (int c = 0; c < 64; ++c) {
                const size_t src = static_cast<size_t>(kb * 64 + c) * T + t;     // w[co][ci][t] of a (1, 5) or (5, 1) kernel
                for (int n = 0; n < rdvc::GRU_ZR_N; ++n) {
                    const float v = (n < rdvc::GRU_C ? wz[static_cast<size_t>(n) * CIN * T + src]
                                                     : wr[static_cast<size_t>(n - rdvc::GRU_C) * CIN * T + src]);
                    zr[(static_cast<size_t>(kb * T + t) * rdvc::GRU_ZR_N + n) * 64 + c] = gru_round16(v, op_dtype);
                }
                for (int n = 0; n < rdvc::GRU_Q_N; ++n)
                    qq[(static_cast<size_t>(kb * T + t) * rdvc::GRU_Q_N + n) * 64 + c] =
                        gru_round16(wq[static_cast<size_t>(n) * CIN * T + src], op_dtype);
            }
    return RDVC_OK;
}

size_t rdvc_corr_convgru_workspace_bytes(int B, int H, int W, int act_dtype) {
    if (B <= 0 || H <= 0 || W <= 0) return 0;
    if (act_dtype != RDVC_DT_F32 && act_dtype != RDVC_DT_F16 && act_dtype != RDVC_DT_BF16) return 0;
    return (act_dtype == RDVC_DT_F32 ? 5 : 2) * gru_plane_bytes(B, H, W);
}

int rdvc_corr_convgru(const void* h, long long h_pixel_stride, const void* context, long long context_pixel_stride,
                 const void* motion, long long motion_pixel_stride, int act_dtype, int op_dtype, int axis, int B, int H,
                 int W, const void* packed_w, const float* bias_z, const float* bias_r, const float* bias_q,
                 void* workspace, size_t workspace_bytes, void* out, void* stream) {
    if (!h || !context || !motion || !packed_w || !bias_z || !bias_r || !bias_q || !workspace || !out)
        return fail(RDVC_E_NULL, "null pointer argument");
    if (B <= 0 || H <= 0 || W <= 0) return fail(RDVC_E_SHAPE, "non-positive dimension B=%d H=%d W=%d", B, H, W);
    if (act_dtype != RDVC_DT_F32 && act_dtype != RDVC_DT_F16 && act_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "unsupported act_dtype=%d", act_dtype);
    if (op_dtype != RDVC_DT_F16 && op_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "op_dtype must be F16 or BF16, got %d", op_dtype);
    if (act_dtype != RDVC_DT_F32 && act_dtype != op_dtype)
        return fail(RDVC_E_DTYPE, "16-bit activations are their own operands: act_dtype=%d needs op_dtype=%d", act_dtype,
                    act_dtype);
    if (axis != RDVC_GRU_HORIZONTAL && axis != RDVC_GRU_VERTICAL)
        return fail(RDVC_E_UNSUPPORTED, "axis=%d is neither RDVC_GRU_HORIZONTAL nor RDVC_GRU_VERTICAL", axis);
    const long long es = static_cast<long long>(elem_size(act_dtype));
    const long long ps[3] = {h_pixel_stride, context_pixel_stride, motion_pixel_stride};
    for (long long s : ps)
        if (s < rdvc::GRU_C) return fail(RDVC_E_UNSUPPORTED, "pixel stride %lld < %d channels", s, rdvc::GRU_C);
    const void* ptrs[5] = {h, context, motion, out, workspace};
    for (const void* q : ptrs)
        if (reinterpret_cast<uintptr_t>(q) & 15) return fail(RDVC_E_ALIGN, "activation buffers must be 16-byte aligned");
    for (long long s : ps)
        if ((s * es) % 16) return fail(RDVC_E_ALIGN, "pixel strides must be multiples of 16 bytes (got %lld elements)", s);
    if ((reinterpret_cast<uintptr_t>(packed_w) & 15) || (reinterpret_cast<uintptr_t>(workspace) & 255))
        return fail(RDVC_E_ALIGN, "packed weights must be 16-byte aligned, the workspace 256-byte aligned");
    if (out == h || out == context || out == motion) return fail(RDVC_E_UNSUPPORTED, "the pass cannot run in place");
    const long long n_pix = static_cast<long long>(B) * H * W;
    if (n_pix >= (1LL << 31) || H >= (1 << 24) || W >= (1 << 24))
        return fail(RDVC_E_UNSUPPORTED, "too many pixels for 32-bit TMA coordinates");
    const size_t need = rdvc_corr_convgru_workspace_bytes(B, H, W, act_dtype);
    if (workspace_bytes < need) return fail(RDVC_E_WORKSPACE, "workspace %zu < required %zu", workspace_bytes, need);

    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t plane = gru_plane_bytes(B, H, W);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    void* z = ws;
    void* rh = ws + plane;
    const void* a16[3] = {h, context, motion};          // the GEMMs' 16-bit operands
    long long ps16[3] = {ps[0], ps[1], ps[2]};
    if (act_dtype == RDVC_DT_F32) {
        rdvc::GruCastParams cp;
        memset(&cp, 0, sizeof(cp));
        for (int i = 0; i < 3; ++i) {
            cp.src[i] = static_cast<const float*>(a16[i]);
            cp.ps[i] = ps[i];
            cp.dst[i] = ws + (2 + i) * plane;
            a16[i] = cp.dst[i];
            ps16[i] = rdvc::GRU_C;
        }
        cp.n_pix = n_pix;
        if (int rc = launch_gru_cast(cp, 3, op_dtype, st)) return rc;
    }
    const int horiz = (axis == RDVC_GRU_HORIZONTAL) ? 1 : 0;
    const CUtensorMapDataType dt = op_map_dtype(op_dtype);
    rdvc::TapMaps<3> zr, q;                             // a: [h or r*h, context, motion]
    for (int i = 0; i < 3; ++i)
        if (int rc = act_map(&zr.a[i], dt, a16[i], ps16[i], rdvc::GRU_C, B, H, W, rdvc::TAP_TX,
                             rdvc::TapGeom<rdvc::TAP_G_GRU5>::BOX_Y, horiz))
            return rc;
    q.a[1] = zr.a[1];
    q.a[2] = zr.a[2];
    if (int rc = act_map(&q.a[0], dt, rh, rdvc::GRU_C, rdvc::GRU_C, B, H, W, rdvc::TAP_TX,
                         rdvc::TapGeom<rdvc::TAP_G_GRU5>::BOX_Y, horiz))
        return rc;
    constexpr int SLABS = rdvc::GRU_KB * rdvc::GRU_TAPS;
    if (int rc = slab_map(&zr.w, dt, packed_w, rdvc::GRU_ZR_N, SLABS)) return rc;
    if (int rc = slab_map(&q.w, dt, static_cast<const uint16_t*>(packed_w) + rdvc::GRU_W_ZR_ELEMS, rdvc::GRU_Q_N, SLABS))
        return rc;

    rdvc::TapParams p_zr = tap_params(B, H, W, rdvc::GRU_KB, horiz);
    p_zr.res = h; p_zr.res_ps = ps[0];
    rdvc::TapParams p_q = p_zr;
    p_zr.bias = bias_z; p_zr.bias_r = bias_r;
    p_zr.out = z; p_zr.out2 = rh;
    p_q.bias = bias_q;
    p_q.z = z; p_q.out = out;
    return (act_dtype == RDVC_DT_F32 && op_dtype == RDVC_DT_F16) ? launch_convgru<float, __half>(zr, q, p_zr, p_q, st)
           : (act_dtype == RDVC_DT_F32) ? launch_convgru<float, __nv_bfloat16>(zr, q, p_zr, p_q, st)
           : (op_dtype == RDVC_DT_F16)  ? launch_convgru<__half, __half>(zr, q, p_zr, p_q, st)
                                        : launch_convgru<__nv_bfloat16, __nv_bfloat16>(zr, q, p_zr, p_q, st);
}

}  // extern "C"

// ---- RAFT's motion encoder and flow head: 3x3 (and convflow1's 7x7) convolutions over NHWC 16-bit activations ---------
namespace {

struct UcLayer {
    int cin, cout, k, n;        // input / output channels, kernel size, GEMM width (cout padded to a multiple of 16)
};
// indexed by RDVC_UC_*: raft_large's MotionEncoder (TV:raft.py:184-196) and FlowHead (TV:raft.py:276-277)
constexpr UcLayer UC_LAYERS[6] = {
    {256, 192, 3, 192},     // RDVC_UC_CONVCORR2
    {2, 128, 7, 128},       // RDVC_UC_CONVFLOW1 (K = 98 padded to 128)
    {128, 64, 3, 64},       // RDVC_UC_CONVFLOW2
    {256, 126, 3, 128},     // RDVC_UC_CONV
    {128, 256, 3, 256},     // RDVC_UC_FH_CONV1
    {256, 2, 3, 16},        // RDVC_UC_FH_CONV2
};

size_t uc_packed_elems(int layer) {
    const UcLayer& L = UC_LAYERS[layer];
    if (layer == RDVC_UC_CONVFLOW1) return static_cast<size_t>(L.n) * rdvc::CF1_KP;
    return static_cast<size_t>(L.cin / 64) * 9 * L.n * 64;
}

size_t uc_plane_bytes(int B, int H, int W, int channels) {
    return align_up(static_cast<size_t>(B) * H * W * channels * 2, 256);
}

template <typename OpT>
int launch_convflow1(const rdvc::Cf1Params& p, cudaStream_t st) {
    auto kern = rdvc::convflow1_kernel<OpT>;
    static std::atomic<unsigned long long> attr_done{0};
    if (int rc = ensure_dynamic_smem(kern, rdvc::CF1_SMEM, attr_done, "cudaFuncSetAttribute(convflow1, max dynamic smem)"))
        return rc;
    const long long groups = (p.n_pix + 31) / 32;
    const long long grid = std::min<long long>(4LL * sm_count(), (groups + 1) / 2);
    kern<<<static_cast<unsigned>(grid), rdvc::CF1_THREADS, rdvc::CF1_SMEM, st>>>(p);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "convflow1_kernel launch");
    return RDVC_OK;
}

// the 3x3 layers' dispatch: one instantiation per (layer, output dtype, operand dtype)
template <typename OpT>
int dispatch_update_conv(int layer, int out_dtype, const rdvc::TapMaps<1>& m, const rdvc::TapParams& p, cudaStream_t st) {
    using namespace rdvc;
    const bool f32 = (out_dtype == RDVC_DT_F32);
    switch (layer) {
        case RDVC_UC_CONVCORR2: return launch_tap_conv<TAP_G_S1, 192, TAP_EPI_RELU, OpT, OpT>(m, p, st);
        case RDVC_UC_CONVFLOW2: return launch_tap_conv<TAP_G_S1, 64, TAP_EPI_RELU, OpT, OpT>(m, p, st);
        case RDVC_UC_FH_CONV1: return launch_tap_conv<TAP_G_S1, 256, TAP_EPI_RELU, OpT, OpT>(m, p, st);
        case RDVC_UC_CONV:
            return f32 ? launch_tap_conv<TAP_G_S1, 128, TAP_EPI_RELU_FLOW, float, OpT>(m, p, st)
                       : launch_tap_conv<TAP_G_S1, 128, TAP_EPI_RELU_FLOW, OpT, OpT>(m, p, st);
        default:
            return f32 ? launch_tap_conv<TAP_G_S1, 16, TAP_EPI_FLOW2, float, OpT>(m, p, st)
                       : launch_tap_conv<TAP_G_S1, 16, TAP_EPI_FLOW2, OpT, OpT>(m, p, st);
    }
}

// the 16-bit operand form of a 128-channel hidden state h (NHWC, pixel stride *ps): 16-bit h is used in place, fp32 h
// is rounded to op_dtype into dst (B * H * W x 128, pixel stride 128) and *h, *ps are pointed at it
int hidden_operand(const void** h, long long* ps, int act_dtype, int op_dtype, long long n_pix, void* dst, void* stream) {
    if (act_dtype != RDVC_DT_F32) return RDVC_OK;
    rdvc::GruCastParams cp;
    memset(&cp, 0, sizeof(cp));
    cp.src[0] = static_cast<const float*>(*h);
    cp.ps[0] = *ps;
    cp.dst[0] = dst;
    cp.n_pix = n_pix;
    if (int rc = launch_gru_cast(cp, 1, op_dtype, static_cast<cudaStream_t>(stream))) return rc;
    *h = dst;
    *ps = 128;
    return RDVC_OK;
}

// one 3x3 layer on the tap-convolution engine, arguments checked by the caller.  out2: FH_CONV2's coordinate update
// (out = coords1, out2 = flow, fp32 (B, 2, H, W); out_dtype is the dtype delta is rounded to), else NULL.
int launch_update_conv(int layer, const void* in, long long in_pixel_stride, const float* flow,
                       const long long* flow_strides, int B, int H, int W, int op_dtype, const void* packed_w,
                       const float* bias, void* out, long long out_pixel_stride, int out_dtype, void* out2,
                       cudaStream_t st) {
    const UcLayer& L = UC_LAYERS[layer];
    const CUtensorMapDataType dt = op_map_dtype(op_dtype);
    rdvc::TapMaps<1> m;
    if (int rc = act_map(&m.a[0], dt, in, in_pixel_stride, L.cin, B, H, W, rdvc::TAP_TX,
                         rdvc::TapGeom<rdvc::TAP_G_S1>::BOX_Y))
        return rc;
    if (int rc = slab_map(&m.w, dt, packed_w, L.n, L.cin / 64 * 9)) return rc;
    rdvc::TapParams p = tap_params(B, H, W, L.cin / 64);
    p.bias = bias; p.cout = L.cout;
    p.out = out; p.out_ps = out_pixel_stride;
    p.out2 = out2;
    if (flow) {
        p.flow = flow;
        p.fs_b = flow_strides[0]; p.fs_c = flow_strides[1]; p.fs_y = flow_strides[2]; p.fs_x = flow_strides[3];
    }
    return op_dtype == RDVC_DT_F16 ? dispatch_update_conv<__half>(layer, out_dtype, m, p, st)
                                   : dispatch_update_conv<__nv_bfloat16>(layer, out_dtype, m, p, st);
}

}  // namespace

extern "C" {

size_t rdvc_corr_update_conv_packed_weight_bytes(int layer) {
    if (layer < 0 || layer > RDVC_UC_FH_CONV2) return 0;
    return uc_packed_elems(layer) * 2;
}

int rdvc_corr_update_conv_pack_weights(int layer, const float* weight, int op_dtype, void* packed_host) {
    if (!weight || !packed_host) return fail(RDVC_E_NULL, "null pointer argument");
    if (layer < 0 || layer > RDVC_UC_FH_CONV2) return fail(RDVC_E_UNSUPPORTED, "unknown layer %d", layer);
    if (op_dtype != RDVC_DT_F16 && op_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "op_dtype must be F16 or BF16, got %d", op_dtype);
    const UcLayer& L = UC_LAYERS[layer];
    uint16_t* out = static_cast<uint16_t*>(packed_host);
    memset(out, 0, uc_packed_elems(layer) * 2);                 // padded rows (N > cout) and columns (K > 98) are zero
    const int kk = L.k * L.k;
    if (layer == RDVC_UC_CONVFLOW1) {                           // [n][(ky * 7 + kx) * 2 + ci]
        for (int n = 0; n < L.cout; ++n)
            for (int ci = 0; ci < L.cin; ++ci)
                for (int t = 0; t < kk; ++t)
                    out[static_cast<size_t>(n) * rdvc::CF1_KP + t * 2 + ci] =
                        gru_round16(weight[(static_cast<size_t>(n) * L.cin + ci) * kk + t], op_dtype);
        return RDVC_OK;
    }
    for (int kb = 0; kb < L.cin / 64; ++kb)                     // [k-block][dy * 3 + dx][n][64]
        for (int t = 0; t < 9; ++t)
            for (int n = 0; n < L.cout; ++n)
                for (int c = 0; c < 64; ++c)
                    out[((static_cast<size_t>(kb) * 9 + t) * L.n + n) * 64 + c] =
                        gru_round16(weight[(static_cast<size_t>(n) * L.cin + kb * 64 + c) * 9 + t], op_dtype);
    return RDVC_OK;
}

int rdvc_corr_update_conv(int layer, const void* in, long long in_pixel_stride, const float* flow, const long long* flow_strides,
                     int B, int H, int W, int op_dtype, const void* packed_w, const float* bias, void* out,
                     long long out_pixel_stride, int out_dtype, void* stream) {
    if (layer < 0 || layer > RDVC_UC_FH_CONV2) return fail(RDVC_E_UNSUPPORTED, "unknown layer %d", layer);
    const UcLayer& L = UC_LAYERS[layer];
    const bool uses_flow = (layer == RDVC_UC_CONVFLOW1 || layer == RDVC_UC_CONV);
    if (!packed_w || !bias || !out || (layer != RDVC_UC_CONVFLOW1 && !in) || (uses_flow && (!flow || !flow_strides)))
        return fail(RDVC_E_NULL, "null pointer argument");
    if (B <= 0 || H <= 0 || W <= 0) return fail(RDVC_E_SHAPE, "non-positive dimension B=%d H=%d W=%d", B, H, W);
    if (op_dtype != RDVC_DT_F16 && op_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "op_dtype must be F16 or BF16, got %d", op_dtype);
    const bool act_out = (layer == RDVC_UC_CONV || layer == RDVC_UC_FH_CONV2);    // written in the activation dtype
    if (act_out ? (out_dtype != RDVC_DT_F32 && out_dtype != op_dtype) : (out_dtype != op_dtype))
        return fail(RDVC_E_DTYPE, "layer %d cannot write out_dtype=%d with op_dtype=%d", layer, out_dtype, op_dtype);
    const long long n_pix = static_cast<long long>(B) * H * W;
    if (n_pix >= (1LL << 31) || H >= (1 << 24) || W >= (1 << 24))
        return fail(RDVC_E_UNSUPPORTED, "too many pixels for 32-bit TMA coordinates");
    if ((reinterpret_cast<uintptr_t>(packed_w) & 15) || (reinterpret_cast<uintptr_t>(out) & 15) ||
        (in && (reinterpret_cast<uintptr_t>(in) & 15)))
        return fail(RDVC_E_ALIGN, "input, output and packed weights must be 16-byte aligned");
    if (layer != RDVC_UC_CONVFLOW1) {
        if (in_pixel_stride < L.cin) return fail(RDVC_E_UNSUPPORTED, "in_pixel_stride %lld < %d", in_pixel_stride, L.cin);
        if (in_pixel_stride % 8) return fail(RDVC_E_ALIGN, "in_pixel_stride must be a multiple of 8 elements");
    }
    if (layer != RDVC_UC_FH_CONV2) {
        const long long es = (out_dtype == RDVC_DT_F32) ? 4 : 2;
        if (out_pixel_stride < L.n) return fail(RDVC_E_UNSUPPORTED, "out_pixel_stride %lld < %d", out_pixel_stride, L.n);
        if ((out_pixel_stride * es) % 16) return fail(RDVC_E_ALIGN, "out_pixel_stride must be a multiple of 16 bytes");
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (layer == RDVC_UC_CONVFLOW1) {
        rdvc::Cf1Params p;
        memset(&p, 0, sizeof(p));
        p.flow = flow;
        p.fs_b = flow_strides[0]; p.fs_c = flow_strides[1]; p.fs_y = flow_strides[2]; p.fs_x = flow_strides[3];
        p.w = packed_w; p.bias = bias; p.out = out; p.out_ps = out_pixel_stride;
        p.B = B; p.H = H; p.W = W; p.n_pix = n_pix;
        return op_dtype == RDVC_DT_F16 ? launch_convflow1<__half>(p, st) : launch_convflow1<__nv_bfloat16>(p, st);
    }
    return launch_update_conv(layer, in, in_pixel_stride, uses_flow ? flow : nullptr, flow_strides, B, H, W, op_dtype,
                              packed_w, bias, out, out_pixel_stride, out_dtype, nullptr, st);
}

size_t rdvc_corr_motion_encoder_workspace_bytes(int B, int H, int W) {
    if (B <= 0 || H <= 0 || W <= 0) return 0;
    return uc_plane_bytes(B, H, W, 128) + uc_plane_bytes(B, H, W, 256);
}

int rdvc_corr_motion_encoder(const void* c1, long long c1_pixel_stride, const float* flow, const long long* flow_strides, int B,
                        int H, int W, int op_dtype, const void* const* packed_w, const float* const* bias, void* workspace,
                        size_t workspace_bytes, void* out, long long out_pixel_stride, int out_dtype, void* stream) {
    if (!c1 || !flow || !flow_strides || !packed_w || !bias || !workspace || !out)
        return fail(RDVC_E_NULL, "null pointer argument");
    for (int i = 0; i < 4; ++i)
        if (!packed_w[i] || !bias[i]) return fail(RDVC_E_NULL, "null packed weight or bias pointer");
    if (B <= 0 || H <= 0 || W <= 0) return fail(RDVC_E_SHAPE, "non-positive dimension B=%d H=%d W=%d", B, H, W);
    const size_t need = rdvc_corr_motion_encoder_workspace_bytes(B, H, W);
    if (workspace_bytes < need) return fail(RDVC_E_WORKSPACE, "workspace %zu < required %zu", workspace_bytes, need);
    if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail(RDVC_E_ALIGN, "the workspace must be 256-byte aligned");
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    uint8_t* f1 = ws;                                            // convflow1 output (B, H, W, 128)
    uint8_t* cf = ws + uc_plane_bytes(B, H, W, 128);             // [convcorr2 | convflow2] (B, H, W, 256)
    // TV:raft.py:203-205: flo = convflow2(convflow1(flow)); cor = convcorr2(cor); the cat is two channel slices of cf
    if (int rc = rdvc_corr_update_conv(RDVC_UC_CONVFLOW1, nullptr, 0, flow, flow_strides, B, H, W, op_dtype, packed_w[1], bias[1],
                                  f1, 128, op_dtype, stream))
        return rc;
    if (int rc = rdvc_corr_update_conv(RDVC_UC_CONVFLOW2, f1, 128, nullptr, nullptr, B, H, W, op_dtype, packed_w[2], bias[2],
                                  cf + 192 * 2, 256, op_dtype, stream))
        return rc;
    if (int rc = rdvc_corr_update_conv(RDVC_UC_CONVCORR2, c1, c1_pixel_stride, nullptr, nullptr, B, H, W, op_dtype, packed_w[0],
                                  bias[0], cf, 256, op_dtype, stream))
        return rc;
    // TV:raft.py:207-210: conv(cat(cor, flo)), then cat with the flow: channels 126-127 written by the same epilogue
    return rdvc_corr_update_conv(RDVC_UC_CONV, cf, 256, flow, flow_strides, B, H, W, op_dtype, packed_w[3], bias[3], out,
                            out_pixel_stride, out_dtype, stream);
}

size_t rdvc_corr_flow_head_workspace_bytes(int B, int H, int W, int act_dtype) {
    if (B <= 0 || H <= 0 || W <= 0) return 0;
    if (act_dtype != RDVC_DT_F32 && act_dtype != RDVC_DT_F16 && act_dtype != RDVC_DT_BF16) return 0;
    return uc_plane_bytes(B, H, W, 256) + (act_dtype == RDVC_DT_F32 ? uc_plane_bytes(B, H, W, 128) : 0);
}

int rdvc_corr_flow_head(const void* h, long long h_pixel_stride, int act_dtype, int B, int H, int W, int op_dtype,
                   const void* const* packed_w, const float* const* bias, void* workspace, size_t workspace_bytes, void* out,
                   void* stream) {
    if (!h || !packed_w || !bias || !workspace || !out) return fail(RDVC_E_NULL, "null pointer argument");
    for (int i = 0; i < 2; ++i)
        if (!packed_w[i] || !bias[i]) return fail(RDVC_E_NULL, "null packed weight or bias pointer");
    if (B <= 0 || H <= 0 || W <= 0) return fail(RDVC_E_SHAPE, "non-positive dimension B=%d H=%d W=%d", B, H, W);
    if (act_dtype != RDVC_DT_F32 && act_dtype != RDVC_DT_F16 && act_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "unsupported act_dtype=%d", act_dtype);
    if (op_dtype != RDVC_DT_F16 && op_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "op_dtype must be F16 or BF16, got %d", op_dtype);
    if (act_dtype != RDVC_DT_F32 && act_dtype != op_dtype)
        return fail(RDVC_E_DTYPE, "16-bit activations are their own operands: act_dtype=%d needs op_dtype=%d", act_dtype,
                    act_dtype);
    if (h_pixel_stride < 128) return fail(RDVC_E_UNSUPPORTED, "h_pixel_stride %lld < 128 channels", h_pixel_stride);
    if ((reinterpret_cast<uintptr_t>(h) & 15) || ((h_pixel_stride * elem_size(act_dtype)) % 16))
        return fail(RDVC_E_ALIGN, "h must be 16-byte aligned with a pixel stride of a multiple of 16 bytes");
    const size_t need = rdvc_corr_flow_head_workspace_bytes(B, H, W, act_dtype);
    if (workspace_bytes < need) return fail(RDVC_E_WORKSPACE, "workspace %zu < required %zu", workspace_bytes, need);
    if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail(RDVC_E_ALIGN, "the workspace must be 256-byte aligned");
    const long long n_pix = static_cast<long long>(B) * H * W;
    if (n_pix >= (1LL << 31)) return fail(RDVC_E_UNSUPPORTED, "too many pixels for 32-bit TMA coordinates");
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    uint8_t* fh = ws;                                            // conv1 output (B, H, W, 256)
    const void* h16 = h;
    long long h16_ps = h_pixel_stride;
    if (int rc = hidden_operand(&h16, &h16_ps, act_dtype, op_dtype, n_pix, ws + uc_plane_bytes(B, H, W, 256), stream))
        return rc;
    // TV:raft.py:284-285: conv2(relu(conv1(x)))
    if (int rc = rdvc_corr_update_conv(RDVC_UC_FH_CONV1, h16, h16_ps, nullptr, nullptr, B, H, W, op_dtype, packed_w[0], bias[0],
                                  fh, 256, op_dtype, stream))
        return rc;
    return rdvc_corr_update_conv(RDVC_UC_FH_CONV2, fh, 256, nullptr, nullptr, B, H, W, op_dtype, packed_w[1], bias[1], out, 0,
                            act_dtype, stream);
}

}  // extern "C"

// ---- RAFT's mask predictor with the convex 8x upsampling fused into its 1x1 GEMM -------------------------------------
namespace {

template <int EPI, typename OutT, typename OpT>
int launch_mask_upsample(const CUtensorMap& a, const CUtensorMap& w, const rdvc::MuParams& p, cudaStream_t st) {
    auto kern = rdvc::mask_upsample_kernel<EPI, OutT, OpT>;
    static std::atomic<unsigned long long> attr_done{0};
    if (int rc = ensure_dynamic_smem(kern, rdvc::MU_SMEM_LAUNCH, attr_done,
                                     "cudaFuncSetAttribute(mask_upsample, max dynamic smem)"))
        return rc;
    const int grid = std::min(sm_count(), p.n_tiles);
    kern<<<grid, rdvc::MU_THREADS, rdvc::MU_SMEM_LAUNCH, st>>>(a, w, p);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "mask_upsample_kernel launch");
    return RDVC_OK;
}

template <typename OpT>
int dispatch_mask_upsample(int out_form, int act_dtype, const CUtensorMap& a, const CUtensorMap& w, const rdvc::MuParams& p,
                           cudaStream_t st) {
    if (out_form == RDVC_MASK_OUT_UPSAMPLED) return launch_mask_upsample<rdvc::MU_EPI_UPSAMPLED, float, OpT>(a, w, p, st);
    return act_dtype == RDVC_DT_F32 ? launch_mask_upsample<rdvc::MU_EPI_MASK, float, OpT>(a, w, p, st)
                                    : launch_mask_upsample<rdvc::MU_EPI_MASK, OpT, OpT>(a, w, p, st);
}

}  // namespace

extern "C" {

size_t rdvc_corr_mask_conv_packed_weight_bytes(void) { return static_cast<size_t>(rdvc::MU_COUT) * rdvc::MU_CIN * 2; }

int rdvc_corr_mask_conv_pack_weights(const float* weight, const float* bias, int op_dtype, void* packed_host,
                                     float* bias_host) {
    if (!weight || !bias || !packed_host || !bias_host) return fail(RDVC_E_NULL, "null pointer argument");
    if (op_dtype != RDVC_DT_F16 && op_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "op_dtype must be F16 or BF16, got %d", op_dtype);
    uint16_t* out = static_cast<uint16_t*>(packed_host);
    // GEMM row n = c * 144 + k * 16 + s  <-  stock channel k * 64 + 16 c + s;  packed [c][k-block][144][64]
    for (int c = 0; c < rdvc::MU_CHUNKS; ++c)
        for (int k = 0; k < 9; ++k)
            for (int s = 0; s < 16; ++s) {
                const int row = k * 16 + s, src = k * 64 + 16 * c + s;
                bias_host[c * rdvc::MU_NC + row] = bias[src];
                for (int kb = 0; kb < rdvc::MU_KB; ++kb)
                    for (int ch = 0; ch < 64; ++ch)
                        out[((static_cast<size_t>(c) * rdvc::MU_KB + kb) * rdvc::MU_NC + row) * 64 + ch] =
                            gru_round16(weight[static_cast<size_t>(src) * rdvc::MU_CIN + kb * 64 + ch], op_dtype);
            }
    return RDVC_OK;
}

size_t rdvc_corr_mask_predictor_workspace_bytes(int B, int H, int W, int act_dtype) {
    return rdvc_corr_flow_head_workspace_bytes(B, H, W, act_dtype);      // the same two buffers: convrelu's output, h16
}

int rdvc_corr_mask_predictor(const void* h, long long h_pixel_stride, int act_dtype, int B, int H, int W, int op_dtype,
                             const void* const* packed_w, const float* const* bias, float multiplier, const float* flow,
                             const long long* flow_strides, int out_form, void* workspace, size_t workspace_bytes, void* out,
                             void* stream) {
    if (!h || !packed_w || !bias || !workspace || !out) return fail(RDVC_E_NULL, "null pointer argument");
    for (int i = 0; i < 2; ++i)
        if (!packed_w[i] || !bias[i]) return fail(RDVC_E_NULL, "null packed weight or bias pointer");
    if (out_form != RDVC_MASK_OUT_UPSAMPLED && out_form != RDVC_MASK_OUT_MASK)
        return fail(RDVC_E_UNSUPPORTED, "unknown out_form %d", out_form);
    if (out_form == RDVC_MASK_OUT_UPSAMPLED && (!flow || !flow_strides))
        return fail(RDVC_E_NULL, "RDVC_MASK_OUT_UPSAMPLED needs the flow and its strides");
    if (B <= 0 || H <= 0 || W <= 0) return fail(RDVC_E_SHAPE, "non-positive dimension B=%d H=%d W=%d", B, H, W);
    if (act_dtype != RDVC_DT_F32 && act_dtype != RDVC_DT_F16 && act_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "unsupported act_dtype=%d", act_dtype);
    if (op_dtype != RDVC_DT_F16 && op_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "op_dtype must be F16 or BF16, got %d", op_dtype);
    if (act_dtype != RDVC_DT_F32 && act_dtype != op_dtype)
        return fail(RDVC_E_DTYPE, "16-bit activations are their own operands: act_dtype=%d needs op_dtype=%d", act_dtype,
                    act_dtype);
    if (h_pixel_stride < 128) return fail(RDVC_E_UNSUPPORTED, "h_pixel_stride %lld < 128 channels", h_pixel_stride);
    if ((reinterpret_cast<uintptr_t>(h) & 15) || ((h_pixel_stride * elem_size(act_dtype)) % 16))
        return fail(RDVC_E_ALIGN, "h must be 16-byte aligned with a pixel stride of a multiple of 16 bytes");
    if ((reinterpret_cast<uintptr_t>(out) & 15) || (reinterpret_cast<uintptr_t>(packed_w[1]) & 15))
        return fail(RDVC_E_ALIGN, "out and the packed 1x1 weights must be 16-byte aligned");
    const size_t need = rdvc_corr_mask_predictor_workspace_bytes(B, H, W, act_dtype);
    if (workspace_bytes < need) return fail(RDVC_E_WORKSPACE, "workspace %zu < required %zu", workspace_bytes, need);
    if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail(RDVC_E_ALIGN, "the workspace must be 256-byte aligned");
    const long long n_pix = static_cast<long long>(B) * H * W;
    if (n_pix >= (1LL << 31) || H >= (1 << 24) || W >= (1 << 24))
        return fail(RDVC_E_UNSUPPORTED, "too many pixels for 32-bit TMA coordinates");
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    uint8_t* hid = ws;                                           // convrelu output (B, H, W, 256), op_dtype
    const void* h16 = h;
    long long h16_ps = h_pixel_stride;
    if (int rc = hidden_operand(&h16, &h16_ps, act_dtype, op_dtype, n_pix, ws + uc_plane_bytes(B, H, W, 256), stream))
        return rc;
    // TV:raft.py:331: convrelu -- the 3x3 128 -> 256 + ReLU of flow_head.conv1's shape, same kernel
    if (int rc = rdvc_corr_update_conv(RDVC_UC_FH_CONV1, h16, h16_ps, nullptr, nullptr, B, H, W, op_dtype, packed_w[0], bias[0],
                                       hid, 256, op_dtype, stream))
        return rc;
    // TV:raft.py:332-333 (conv, x multiplier) and, UPSAMPLED, TV:_utils.py:39-48 in the epilogue
    const CUtensorMapDataType dt = op_map_dtype(op_dtype);
    CUtensorMap tm_a, tm_w;
    if (int rc = act_map(&tm_a, dt, hid, rdvc::MU_CIN, rdvc::MU_CIN, B, H, W, rdvc::MU_TX, rdvc::MU_TY)) return rc;
    if (int rc = slab_map(&tm_w, dt, packed_w[1], rdvc::MU_NC, rdvc::MU_CHUNKS * rdvc::MU_KB)) return rc;
    rdvc::MuParams p;
    memset(&p, 0, sizeof(p));
    p.B = B; p.H = H; p.W = W;
    p.n_tx = (W + rdvc::MU_TX - 1) / rdvc::MU_TX;
    p.n_ty = (H + rdvc::MU_TY - 1) / rdvc::MU_TY;
    p.n_tiles = static_cast<int>(static_cast<long long>(B) * p.n_tx * p.n_ty);
    p.bias = bias[1];
    p.multiplier = multiplier;
    p.out = out;
    if (out_form == RDVC_MASK_OUT_UPSAMPLED) {
        p.flow = flow;
        p.fs_b = flow_strides[0]; p.fs_c = flow_strides[1]; p.fs_y = flow_strides[2]; p.fs_x = flow_strides[3];
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    return op_dtype == RDVC_DT_F16 ? dispatch_mask_upsample<__half>(out_form, act_dtype, tm_a, tm_w, p, st)
                                   : dispatch_mask_upsample<__nv_bfloat16>(out_form, act_dtype, tm_a, tm_w, p, st);
}

}  // extern "C"

// ---- RAFT's context encoder: FeatureEncoder with frozen BatchNorm folded into tcgen05 convolutions ----------------
namespace {

struct CeLayer {
    int cin, cout, k;
};
// indexed like the pack arrays (parameter-tree order, see include/rdvc_corr.h)
constexpr CeLayer CE_LAYERS[RDVC_CE_LAYERS] = {
    {3, 64, 7},   {64, 64, 3},  {64, 64, 3},  {64, 64, 3},   {64, 64, 3},   {64, 96, 3},   {64, 96, 1},   {96, 96, 3},
    {96, 96, 3},  {96, 96, 3},  {96, 128, 3}, {96, 128, 1},  {128, 128, 3}, {128, 128, 3}, {128, 128, 3}, {128, 256, 1},
};

struct CeUnit {
    int geom, n, n_kb, epi;
    int conv, ds;               // layer index of the convolution and of the fused downsample (-1: none)
};
// one kernel launch each, in execution order
constexpr int CE_N_UNITS = 14;
constexpr CeUnit CE_UNITS[CE_N_UNITS] = {
    {rdvc::TAP_G_STEM, 64, 1, rdvc::TAP_EPI_RELU, 0, -1},
    {rdvc::TAP_G_S1, 64, 1, rdvc::TAP_EPI_RELU, 1, -1},   {rdvc::TAP_G_S1, 64, 1, rdvc::TAP_EPI_RES, 2, -1},
    {rdvc::TAP_G_S1, 64, 1, rdvc::TAP_EPI_RELU, 3, -1},   {rdvc::TAP_G_S1, 64, 1, rdvc::TAP_EPI_RES, 4, -1},
    {rdvc::TAP_G_S2, 128, 1, rdvc::TAP_EPI_DS, 5, 6},     {rdvc::TAP_G_S1, 128, 2, rdvc::TAP_EPI_RES, 7, -1},
    {rdvc::TAP_G_S1, 128, 2, rdvc::TAP_EPI_RELU, 8, -1},  {rdvc::TAP_G_S1, 128, 2, rdvc::TAP_EPI_RES, 9, -1},
    {rdvc::TAP_G_S2, 128, 2, rdvc::TAP_EPI_DS, 10, 11},   {rdvc::TAP_G_S1, 128, 2, rdvc::TAP_EPI_RES, 12, -1},
    {rdvc::TAP_G_S1, 128, 2, rdvc::TAP_EPI_RELU, 13, -1}, {rdvc::TAP_G_S1, 128, 2, rdvc::TAP_EPI_RES, 14, -1},
    {rdvc::TAP_G_1X1, 256, 2, rdvc::TAP_EPI_RAW, 15, -1},
};

// slabs per k-block and box height of a geometry
struct CeGeomSizes {
    int slabs, box_y;
};
CeGeomSizes ce_geom(int geom) {
    using namespace rdvc;
    switch (geom) {
        case TAP_G_S1: return {TapGeom<TAP_G_S1>::SLABS, TapGeom<TAP_G_S1>::BOX_Y};
        case TAP_G_S2: return {TapGeom<TAP_G_S2>::SLABS, TapGeom<TAP_G_S2>::BOX_Y};
        case TAP_G_STEM: return {TapGeom<TAP_G_STEM>::SLABS, TapGeom<TAP_G_STEM>::BOX_Y};
        default: return {TapGeom<TAP_G_1X1>::SLABS, TapGeom<TAP_G_1X1>::BOX_Y};
    }
}
size_t ce_unit_w_elems(const CeUnit& u) { return static_cast<size_t>(u.n_kb) * ce_geom(u.geom).slabs * u.n * 64; }
size_t ce_unit_b_floats(const CeUnit& u) { return static_cast<size_t>(u.n) * (u.ds >= 0 ? 2 : 1); }

size_t ce_w_elems_total() {
    size_t s = 0;
    for (const CeUnit& u : CE_UNITS) s += ce_unit_w_elems(u);
    return s;
}
size_t ce_b_floats_total() {
    size_t s = 0;
    for (const CeUnit& u : CE_UNITS) s += ce_unit_b_floats(u);
    return s;
}

uint16_t ce_round16(double v, int op_dtype) {         // one rounding, fp64 -> 16 bits
    uint16_t bits;
    if (op_dtype == RDVC_DT_F16) { const __half hv = __double2half(v); memcpy(&bits, &hv, 2); }
    else { const __nv_bfloat16 bv = __double2bfloat16(v); memcpy(&bits, &bv, 2); }
    return bits;
}

// w' = w s, b' = beta + (b - mean) s with s = gamma / sqrt(var + eps), in fp64 (layer 15 has no BatchNorm)
void ce_fold(int i, const float* const* conv_w, const float* const* conv_b, const float* const* bn_w,
             const float* const* bn_b, const float* const* bn_mean, const float* const* bn_var, const double* eps,
             std::vector<double>& w, std::vector<double>& b) {
    const CeLayer& L = CE_LAYERS[i];
    const size_t per = static_cast<size_t>(L.cin) * L.k * L.k;
    w.assign(conv_w[i], conv_w[i] + L.cout * per);
    b.assign(conv_b[i], conv_b[i] + L.cout);
    if (i == RDVC_CE_LAYERS - 1) return;
    for (int n = 0; n < L.cout; ++n) {
        const double s = static_cast<double>(bn_w[i][n]) / std::sqrt(static_cast<double>(bn_var[i][n]) + eps[i]);
        for (size_t e = 0; e < per; ++e) w[n * per + e] *= s;
        b[n] = static_cast<double>(bn_b[i][n]) + (b[n] - static_cast<double>(bn_mean[i][n])) * s;
    }
}

// one instantiation per (geometry, N, epilogue, output dtype, operand dtype) the unit table uses
template <typename OpT>
int dispatch_context_conv(const CeUnit& u, int epi, bool f32_out, const rdvc::TapMaps<1>& m, const rdvc::TapParams& p,
                          cudaStream_t st) {
    using namespace rdvc;
    switch (u.geom) {
        case TAP_G_STEM: return launch_tap_conv<TAP_G_STEM, 64, TAP_EPI_RELU, OpT, OpT>(m, p, st);
        case TAP_G_S2: return launch_tap_conv<TAP_G_S2, 128, TAP_EPI_DS, OpT, OpT>(m, p, st);
        case TAP_G_S1:
            if (u.n == 64)
                return epi == TAP_EPI_RES ? launch_tap_conv<TAP_G_S1, 64, TAP_EPI_RES, OpT, OpT>(m, p, st)
                                          : launch_tap_conv<TAP_G_S1, 64, TAP_EPI_RELU, OpT, OpT>(m, p, st);
            return epi == TAP_EPI_RES ? launch_tap_conv<TAP_G_S1, 128, TAP_EPI_RES, OpT, OpT>(m, p, st)
                                      : launch_tap_conv<TAP_G_S1, 128, TAP_EPI_RELU, OpT, OpT>(m, p, st);
        default:
            if (epi == TAP_EPI_SPLIT)
                return f32_out ? launch_tap_conv<TAP_G_1X1, 256, TAP_EPI_SPLIT, float, OpT>(m, p, st)
                               : launch_tap_conv<TAP_G_1X1, 256, TAP_EPI_SPLIT, OpT, OpT>(m, p, st);
            return f32_out ? launch_tap_conv<TAP_G_1X1, 256, TAP_EPI_RAW, float, OpT>(m, p, st)
                           : launch_tap_conv<TAP_G_1X1, 256, TAP_EPI_RAW, OpT, OpT>(m, p, st);
    }
}

// one unit's tensor maps and tile grid: input NHWC op_dtype (B, Hin, Win, n_kb * 64 of in_ps channels) -> output
// grid (Hout, Wout)
int context_unit_setup(const CeUnit& u, const void* in, long long in_ps, int B, int Hin, int Win, int Hout, int Wout,
                       int op_dtype, const void* w, rdvc::TapMaps<1>& m, rdvc::TapParams& p) {
    const CUtensorMapDataType dt = op_map_dtype(op_dtype);
    const CeGeomSizes g = ce_geom(u.geom);
    const int k = (u.geom == rdvc::TAP_G_S2) ? 2 : 1;      // stride 2: a box of {32, 18} lands 16 x 9 pixels
    if (int rc = act_map(&m.a[0], dt, in, in_ps, u.n_kb * 64, B, Hin, Win, k * rdvc::TAP_TX, k * g.box_y, false, k == 2))
        return rc;
    if (int rc = slab_map(&m.w, dt, w, u.n, u.n_kb * g.slabs)) return rc;
    p = tap_params(B, Hout, Wout, u.n_kb);
    return RDVC_OK;
}

// one unit: input NHWC op_dtype (B, Hin, Win, n_kb * 64 of in_ps channels) -> output grid (Hout, Wout)
int run_context_unit(const CeUnit& u, int epi, const void* in, long long in_ps, int B, int Hin, int Win, int Hout,
                     int Wout, int op_dtype, const void* w, const float* bias, void* out, long long out_ps,
                     int out_dtype, void* out2, const void* res, long long res_ps, cudaStream_t st) {
    rdvc::TapMaps<1> m;
    rdvc::TapParams p;
    if (int rc = context_unit_setup(u, in, in_ps, B, Hin, Win, Hout, Wout, op_dtype, w, m, p)) return rc;
    p.bias = bias;
    p.out = out; p.out_ps = out_ps;
    p.out2 = out2;
    p.res = res; p.res_ps = res_ps;
    const bool f32 = (out_dtype == RDVC_DT_F32);
    return op_dtype == RDVC_DT_F16 ? dispatch_context_conv<__half>(u, epi, f32, m, p, st)
                                   : dispatch_context_conv<__nv_bfloat16>(u, epi, f32, m, p, st);
}

template <typename InT, typename OpT>
int launch_ce_stem_pack(const rdvc::CeStemParams& p, cudaStream_t st) {
    const long long threads = p.n_pix * 8;
    rdvc::ce_stem_pack_kernel<InT, OpT><<<static_cast<unsigned>((threads + 255) / 256), 256, 0, st>>>(p);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "ce_stem_pack_kernel launch");
    return RDVC_OK;
}

template <typename OpT>
int dispatch_ce_stem_pack(int in_dtype, const rdvc::CeStemParams& p, cudaStream_t st) {
    if (in_dtype == RDVC_DT_F32) return launch_ce_stem_pack<float, OpT>(p, st);
    if (in_dtype == RDVC_DT_F16) return launch_ce_stem_pack<__half, OpT>(p, st);
    return launch_ce_stem_pack<__nv_bfloat16, OpT>(p, st);
}

struct CeSizes {
    int H1, W1, H2, W2, H3, W3;
    size_t p1, p2, p3;          // bytes of one activation buffer per level
};

CeSizes ce_sizes(int B, int H, int W) {
    CeSizes s;
    s.H1 = (H + 1) / 2; s.W1 = (W + 1) / 2;
    s.H2 = (s.H1 + 1) / 2; s.W2 = (s.W1 + 1) / 2;
    s.H3 = (s.H2 + 1) / 2; s.W3 = (s.W2 + 1) / 2;
    s.p1 = uc_plane_bytes(B, s.H1, s.W1, 64);
    s.p2 = uc_plane_bytes(B, s.H2, s.W2, 128);
    s.p3 = uc_plane_bytes(B, s.H3, s.W3, 128);
    return s;
}

bool ranges_overlap(const void* a, size_t a_bytes, const void* b, size_t b_bytes) {
    const uintptr_t x = reinterpret_cast<uintptr_t>(a), y = reinterpret_cast<uintptr_t>(b);
    return x < y + b_bytes && y < x + a_bytes;
}

}  // namespace

extern "C" {

size_t rdvc_corr_context_encoder_packed_weight_bytes(void) { return ce_w_elems_total() * 2; }

size_t rdvc_corr_context_encoder_packed_bias_bytes(void) { return ce_b_floats_total() * 4; }

int rdvc_corr_context_encoder_pack_weights(const float* const* conv_w, const float* const* conv_b,
                                           const float* const* bn_w, const float* const* bn_b,
                                           const float* const* bn_mean, const float* const* bn_var, const double* eps,
                                           int op_dtype, void* packed_host, float* bias_host) {
    if (!conv_w || !conv_b || !bn_w || !bn_b || !bn_mean || !bn_var || !eps || !packed_host || !bias_host)
        return fail(RDVC_E_NULL, "null pointer argument");
    for (int i = 0; i < RDVC_CE_LAYERS; ++i) {
        if (!conv_w[i] || !conv_b[i]) return fail(RDVC_E_NULL, "null weight or bias of layer %d", i);
        if (i < RDVC_CE_LAYERS - 1 && (!bn_w[i] || !bn_b[i] || !bn_mean[i] || !bn_var[i]))
            return fail(RDVC_E_NULL, "null BatchNorm vector of layer %d", i);
        if (i < RDVC_CE_LAYERS - 1 && !(eps[i] >= 0.0)) return fail(RDVC_E_UNSUPPORTED, "eps[%d] = %g", i, eps[i]);
    }
    if (op_dtype != RDVC_DT_F16 && op_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "op_dtype must be F16 or BF16, got %d", op_dtype);
    uint16_t* out = static_cast<uint16_t*>(packed_host);
    memset(out, 0, ce_w_elems_total() * 2);                  // padded rows, columns and stem taps are zero
    memset(bias_host, 0, ce_b_floats_total() * 4);
    std::vector<double> w, b;
    size_t wo = 0, bo = 0;
    for (const CeUnit& u : CE_UNITS) {
        const int S = ce_geom(u.geom).slabs;
        for (int part = 0; part < (u.ds >= 0 ? 2 : 1); ++part) {
            const int li = part ? u.ds : u.conv;
            const CeLayer& L = CE_LAYERS[li];
            ce_fold(li, conv_w, conv_b, bn_w, bn_b, bn_mean, bn_var, eps, w, b);
            for (int n = 0; n < L.cout; ++n) bias_host[bo + part * u.n + n] = static_cast<float>(b[n]);
            if (u.geom == rdvc::TAP_G_STEM) {                // [ty][n][k], k = tx * 12 + py * 6 + px * 3 + c
                for (int ty = 0; ty < 4; ++ty)
                    for (int n = 0; n < L.cout; ++n)
                        for (int k = 0; k < 48; ++k) {
                            const int tx = k / 12, py = k % 12 / 6, px = k % 6 / 3, c = k % 3;
                            const int ky = 2 * ty + py - 1, kx = 2 * tx + px - 1;
                            if (ky < 0 || kx < 0 || ky >= 7 || kx >= 7) continue;
                            out[wo + (static_cast<size_t>(ty) * u.n + n) * 64 + k] =
                                ce_round16(w[((static_cast<size_t>(n) * 3 + c) * 7 + ky) * 7 + kx], op_dtype);
                        }
                continue;
            }
            const int kk = L.k * L.k;
            for (int kb = 0; kb < u.n_kb; ++kb)               // [k-block][slab][n][64]
                for (int t = 0; t < kk; ++t) {
                    const int slab = part ? S - 1 : t;       // the downsample is the stride-2 unit's last slab
                    for (int n = 0; n < L.cout; ++n)
                        for (int c = 0; c < 64 && kb * 64 + c < L.cin; ++c)
                            out[wo + ((static_cast<size_t>(kb) * S + slab) * u.n + n) * 64 + c] =
                                ce_round16(w[(static_cast<size_t>(n) * L.cin + kb * 64 + c) * kk + t], op_dtype);
                }
        }
        wo += ce_unit_w_elems(u);
        bo += ce_unit_b_floats(u);
    }
    return RDVC_OK;
}

size_t rdvc_corr_context_encoder_workspace_bytes(int B, int H, int W, int act_dtype) {
    if (B <= 0 || H <= 0 || W <= 0) return 0;
    if (act_dtype != RDVC_DT_F32 && act_dtype != RDVC_DT_F16 && act_dtype != RDVC_DT_BF16) return 0;
    const CeSizes s = ce_sizes(B, H, W);
    return 6 * s.p1 + 5 * s.p2 + 5 * s.p3;
}

int rdvc_corr_context_encoder(const void* image, const long long* image_strides, int in_dtype, int B, int H, int W,
                              int op_dtype, const void* packed_w, const float* biases, int out_form, void* workspace,
                              size_t workspace_bytes, void* out, long long out_pixel_stride, int out_dtype, void* stream) {
    if (!image || !image_strides || !packed_w || !biases || !workspace || !out) return fail(RDVC_E_NULL, "null pointer argument");
    if (out_form != RDVC_CE_OUT_RAW && out_form != RDVC_CE_OUT_SPLIT) return fail(RDVC_E_UNSUPPORTED, "unknown out_form %d", out_form);
    if (B <= 0 || H <= 0 || W <= 0) return fail(RDVC_E_SHAPE, "non-positive dimension B=%d H=%d W=%d", B, H, W);
    if (in_dtype != RDVC_DT_F32 && in_dtype != RDVC_DT_F16 && in_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "unsupported in_dtype=%d", in_dtype);
    if (op_dtype != RDVC_DT_F16 && op_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "op_dtype must be F16 or BF16, got %d", op_dtype);
    if (out_dtype != RDVC_DT_F32 && out_dtype != op_dtype)
        return fail(RDVC_E_DTYPE, "out_dtype=%d must be F32 or op_dtype=%d", out_dtype, op_dtype);
    for (int i = 0; i < 4; ++i)
        if (image_strides[i] < 0) return fail(RDVC_E_UNSUPPORTED, "negative image stride %lld", image_strides[i]);
    if (H >= (1 << 24) || W >= (1 << 24) || static_cast<long long>(B) * ((H + 1) / 2) * ((W + 1) / 2) >= (1LL << 31))
        return fail(RDVC_E_UNSUPPORTED, "too many pixels for 32-bit TMA coordinates");
    const size_t in_es = elem_size(in_dtype), out_es = elem_size(out_dtype);
    if (reinterpret_cast<uintptr_t>(image) % in_es) return fail(RDVC_E_ALIGN, "the image must be aligned to its element size");
    if ((reinterpret_cast<uintptr_t>(packed_w) & 15) || (reinterpret_cast<uintptr_t>(biases) & 15) ||
        (reinterpret_cast<uintptr_t>(out) & 15))
        return fail(RDVC_E_ALIGN, "out, the packed weights and the biases must be 16-byte aligned");
    if (out_pixel_stride < 256) return fail(RDVC_E_UNSUPPORTED, "out_pixel_stride %lld < 256", out_pixel_stride);
    if ((out_pixel_stride * static_cast<long long>(out_es)) % 16)
        return fail(RDVC_E_ALIGN, "out_pixel_stride must be a multiple of 16 bytes");
    const size_t need = rdvc_corr_context_encoder_workspace_bytes(B, H, W, RDVC_DT_F32);
    if (workspace_bytes < need) return fail(RDVC_E_WORKSPACE, "workspace %zu < required %zu", workspace_bytes, need);
    if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail(RDVC_E_ALIGN, "the workspace must be 256-byte aligned");
    const CeSizes s = ce_sizes(B, H, W);
    const long long dims[4] = {B, 3, H, W};
    size_t img_elems = 1;
    for (int i = 0; i < 4; ++i) img_elems += static_cast<size_t>(dims[i] - 1) * static_cast<size_t>(image_strides[i]);
    const size_t out_bytes = (static_cast<size_t>(B) * s.H3 * s.W3 - 1) * out_pixel_stride * out_es + 256 * out_es;
    if (ranges_overlap(out, out_bytes, image, img_elems * in_es) || ranges_overlap(out, out_bytes, workspace, need))
        return fail(RDVC_E_UNSUPPORTED, "out overlaps the image or the workspace");

    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // every intermediate keeps its own buffer (the layout of include/rdvc_corr.h): level 1 (H1 x W1, 64 channels)
    // S X0 T0 X1 T1 X2, level 2 (H2 x W2, 128-channel stride) T R Y T' Z, level 3 the same
    void* l1[6];
    void* l2[5];
    void* l3[5];
    uint8_t* wsp = static_cast<uint8_t*>(workspace);
    for (void*& q : l1) { q = wsp; wsp += s.p1; }
    for (void*& q : l2) { q = wsp; wsp += s.p2; }
    for (void*& q : l3) { q = wsp; wsp += s.p3; }

    rdvc::CeStemParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.img = image;
    sp.sb = image_strides[0]; sp.sc = image_strides[1]; sp.sy = image_strides[2]; sp.sx = image_strides[3];
    sp.H = H; sp.W = W; sp.H1 = s.H1; sp.W1 = s.W1;
    sp.out = l1[0];
    sp.n_pix = static_cast<long long>(B) * s.H1 * s.W1;
    if (int rc = op_dtype == RDVC_DT_F16 ? dispatch_ce_stem_pack<__half>(in_dtype, sp, st)
                                         : dispatch_ce_stem_pack<__nv_bfloat16>(in_dtype, sp, st))
        return rc;

    const uint8_t* wp = static_cast<const uint8_t*>(packed_w);
    const float* bp = biases;
    auto unit = [&](int i, const void* in, long long in_ps, int Hin, int Win, int Hout, int Wout, void* o, long long o_ps,
                    void* o2, const void* res, long long res_ps) {
        const CeUnit& u = CE_UNITS[i];
        const int epi = (i == CE_N_UNITS - 1 && out_form == RDVC_CE_OUT_SPLIT) ? rdvc::TAP_EPI_SPLIT : u.epi;
        const int od = (i == CE_N_UNITS - 1) ? out_dtype : op_dtype;
        const int rc = run_context_unit(u, epi, in, in_ps, B, Hin, Win, Hout, Wout, op_dtype, wp, bp, o, o_ps, od, o2, res,
                                        res_ps, st);
        wp += ce_unit_w_elems(u) * 2;
        bp += ce_unit_b_floats(u);
        return rc;
    };
    const int H1 = s.H1, W1 = s.W1, H2 = s.H2, W2 = s.W2, H3 = s.H3, W3 = s.W3;
    int rc = 0;
    // TV:raft.py:145: convnormrelu; 146: layer1 = two residual blocks relu(x + relu(bn2(conv2(relu(bn1(conv1(x)))))))
    if ((rc = unit(0, l1[0], 64, H1, W1, H1, W1, l1[1], 64, nullptr, nullptr, 0))) return rc;
    if ((rc = unit(1, l1[1], 64, H1, W1, H1, W1, l1[2], 64, nullptr, nullptr, 0))) return rc;
    if ((rc = unit(2, l1[2], 64, H1, W1, H1, W1, l1[3], 64, nullptr, l1[1], 64))) return rc;
    if ((rc = unit(3, l1[3], 64, H1, W1, H1, W1, l1[4], 64, nullptr, nullptr, 0))) return rc;
    if ((rc = unit(4, l1[4], 64, H1, W1, H1, W1, l1[5], 64, nullptr, l1[3], 64))) return rc;
    // 147: layer2; its first block's downsample is the second accumulator of its stride-2 convolution
    if ((rc = unit(5, l1[5], 64, H1, W1, H2, W2, l2[0], 128, l2[1], nullptr, 0))) return rc;
    if ((rc = unit(6, l2[0], 128, H2, W2, H2, W2, l2[2], 128, nullptr, l2[1], 128))) return rc;
    if ((rc = unit(7, l2[2], 128, H2, W2, H2, W2, l2[3], 128, nullptr, nullptr, 0))) return rc;
    if ((rc = unit(8, l2[3], 128, H2, W2, H2, W2, l2[4], 128, nullptr, l2[2], 128))) return rc;
    // 148: layer3
    if ((rc = unit(9, l2[4], 128, H2, W2, H3, W3, l3[0], 128, l3[1], nullptr, 0))) return rc;
    if ((rc = unit(10, l3[0], 128, H3, W3, H3, W3, l3[2], 128, nullptr, l3[1], 128))) return rc;
    if ((rc = unit(11, l3[2], 128, H3, W3, H3, W3, l3[3], 128, nullptr, nullptr, 0))) return rc;
    if ((rc = unit(12, l3[3], 128, H3, W3, H3, W3, l3[4], 128, nullptr, l3[2], 128))) return rc;
    return unit(13, l3[4], 128, H3, W3, H3, W3, out, out_pixel_stride, nullptr, nullptr, 0);
}

}  // extern "C"

// ---- RAFT's feature encoder: FeatureEncoder with InstanceNorm, statistics in the convolution epilogues ------------
// The context encoder's units and packed weights (packed with the identity norm); every unit but the final 1x1 runs
// as tap_conv_in_kernel (raw output + per-tile partials), then in_finalize_kernel and in_apply_kernel.
namespace {

constexpr int FE_N_NORM_UNITS = CE_N_UNITS - 1;

int fe_unit_nt(int i) { return CE_UNITS[i].n * (CE_UNITS[i].ds >= 0 ? 2 : 1); }

// the workspace of include/rdvc_corr.h; with base == nullptr only .bytes is meaningful
struct FeLayout {
    uint8_t* l1[11];                     // S, then Y, A of units 0-4
    uint8_t* l2[9];                      // Y5 D5 A5 Y6 A6 Y7 A7 Y8 A8
    uint8_t* l3[9];                      // the same for units 9-12
    float2* part[FE_N_NORM_UNITS];
    float* stats[FE_N_NORM_UNITS];
    size_t bytes;
};

FeLayout fe_layout(int B, int H, int W, void* base) {
    const CeSizes s = ce_sizes(B, H, W);
    FeLayout L;
    uint8_t* q = static_cast<uint8_t*>(base);
    size_t off = 0;
    auto take = [&](size_t n) {
        uint8_t* r = q ? q + off : nullptr;
        off += align_up(n, 256);
        return r;
    };
    for (auto& x : L.l1) x = take(s.p1);
    for (auto& x : L.l2) x = take(s.p2);
    for (auto& x : L.l3) x = take(s.p3);
    for (int i = 0; i < FE_N_NORM_UNITS; ++i) {
        const int Ho = i < 5 ? s.H1 : i < 9 ? s.H2 : s.H3, Wo = i < 5 ? s.W1 : i < 9 ? s.W2 : s.W3;
        L.part[i] = reinterpret_cast<float2*>(take(static_cast<size_t>(tap_params(B, Ho, Wo, 1).n_tiles) * fe_unit_nt(i) * 8));
    }
    for (int i = 0; i < FE_N_NORM_UNITS; ++i)
        L.stats[i] = reinterpret_cast<float*>(take(static_cast<size_t>(B) * 2 * fe_unit_nt(i) * 4));
    L.bytes = off;
    return L;
}

template <typename OpT>
int dispatch_feature_conv(const CeUnit& u, const rdvc::TapMaps<1>& m, const rdvc::TapParams& p, cudaStream_t st) {
    using namespace rdvc;
    switch (u.geom) {
        case TAP_G_STEM: return launch_tap_conv_in<TAP_G_STEM, 64, TAP_EPI_STATS, OpT>(m, p, st);
        case TAP_G_S2: return launch_tap_conv_in<TAP_G_S2, 128, TAP_EPI_DS_STATS, OpT>(m, p, st);
        default:
            return u.n == 64 ? launch_tap_conv_in<TAP_G_S1, 64, TAP_EPI_STATS, OpT>(m, p, st)
                             : launch_tap_conv_in<TAP_G_S1, 128, TAP_EPI_STATS, OpT>(m, p, st);
    }
}

template <typename OpT>
int launch_in_apply(int form, const rdvc::InApplyParams& a, cudaStream_t st) {
    const unsigned blocks = static_cast<unsigned>((a.n_pix * (a.Cs / 8) + 255) / 256);
    if (form == rdvc::IN_APPLY_RELU) rdvc::in_apply_kernel<rdvc::IN_APPLY_RELU, OpT><<<blocks, 256, 0, st>>>(a);
    else if (form == rdvc::IN_APPLY_RES) rdvc::in_apply_kernel<rdvc::IN_APPLY_RES, OpT><<<blocks, 256, 0, st>>>(a);
    else rdvc::in_apply_kernel<rdvc::IN_APPLY_DS, OpT><<<blocks, 256, 0, st>>>(a);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "in_apply_kernel launch");
    return RDVC_OK;
}

}  // namespace

extern "C" {

size_t rdvc_corr_feature_encoder_workspace_bytes(int B, int H, int W, int act_dtype) {
    if (B <= 0 || H <= 0 || W <= 0) return 0;
    if (act_dtype != RDVC_DT_F32 && act_dtype != RDVC_DT_F16 && act_dtype != RDVC_DT_BF16) return 0;
    if ((H + 7) / 8 == 1 && (W + 7) / 8 == 1) return 0;          // a one-element plane cannot be normalised
    return fe_layout(B, H, W, nullptr).bytes;
}

int rdvc_corr_feature_encoder(const void* image, const long long* image_strides, int in_dtype, int B, int H, int W,
                              int op_dtype, const void* packed_w, const float* biases, const double* eps, int out_form,
                              void* workspace, size_t workspace_bytes, void* out, long long out_pixel_stride,
                              int out_dtype, void* stream) {
    if (!image || !image_strides || !packed_w || !biases || !eps || !workspace || !out)
        return fail(RDVC_E_NULL, "null pointer argument");
    if (out_form != RDVC_FE_OUT_FEATURES && out_form != RDVC_FE_OUT_TRUNK)
        return fail(RDVC_E_UNSUPPORTED, "unknown out_form %d", out_form);
    if (B <= 0 || H <= 0 || W <= 0) return fail(RDVC_E_SHAPE, "non-positive dimension B=%d H=%d W=%d", B, H, W);
    if ((H + 7) / 8 == 1 && (W + 7) / 8 == 1)
        return fail(RDVC_E_SHAPE, "H=%d W=%d: InstanceNorm expects more than 1 spatial element in layer3", H, W);
    if (in_dtype != RDVC_DT_F32 && in_dtype != RDVC_DT_F16 && in_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "unsupported in_dtype=%d", in_dtype);
    if (op_dtype != RDVC_DT_F16 && op_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "op_dtype must be F16 or BF16, got %d", op_dtype);
    const bool trunk = out_form == RDVC_FE_OUT_TRUNK;
    if (trunk ? out_dtype != op_dtype : (out_dtype != RDVC_DT_F32 && out_dtype != op_dtype))
        return fail(RDVC_E_DTYPE, "out_dtype=%d must be %sop_dtype=%d", out_dtype, trunk ? "" : "F32 or ", op_dtype);
    for (int i = 0; i < RDVC_FE_NORMS; ++i)
        if (!(eps[i] >= 0.0) || std::isinf(eps[i])) return fail(RDVC_E_UNSUPPORTED, "eps[%d] = %g", i, eps[i]);
    for (int i = 0; i < 4; ++i)
        if (image_strides[i] < 0) return fail(RDVC_E_UNSUPPORTED, "negative image stride %lld", image_strides[i]);
    if (H >= (1 << 24) || W >= (1 << 24) || static_cast<long long>(B) * ((H + 1) / 2) * ((W + 1) / 2) >= (1LL << 31))
        return fail(RDVC_E_UNSUPPORTED, "too many pixels for 32-bit TMA coordinates");
    const size_t in_es = elem_size(in_dtype), out_es = elem_size(out_dtype);
    if (reinterpret_cast<uintptr_t>(image) % in_es) return fail(RDVC_E_ALIGN, "the image must be aligned to its element size");
    if ((reinterpret_cast<uintptr_t>(packed_w) & 15) || (reinterpret_cast<uintptr_t>(biases) & 15) ||
        (reinterpret_cast<uintptr_t>(out) & 15))
        return fail(RDVC_E_ALIGN, "out, the packed weights and the biases must be 16-byte aligned");
    const int out_c = trunk ? 128 : 256;
    if (out_pixel_stride < out_c) return fail(RDVC_E_UNSUPPORTED, "out_pixel_stride %lld < %d", out_pixel_stride, out_c);
    if ((out_pixel_stride * static_cast<long long>(out_es)) % 16)
        return fail(RDVC_E_ALIGN, "out_pixel_stride must be a multiple of 16 bytes");
    const size_t need = rdvc_corr_feature_encoder_workspace_bytes(B, H, W, RDVC_DT_F32);
    if (workspace_bytes < need) return fail(RDVC_E_WORKSPACE, "workspace %zu < required %zu", workspace_bytes, need);
    if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail(RDVC_E_ALIGN, "the workspace must be 256-byte aligned");
    const CeSizes s = ce_sizes(B, H, W);
    const long long dims[4] = {B, 3, H, W};
    size_t img_elems = 1;
    for (int i = 0; i < 4; ++i) img_elems += static_cast<size_t>(dims[i] - 1) * static_cast<size_t>(image_strides[i]);
    const size_t out_bytes = (static_cast<size_t>(B) * s.H3 * s.W3 - 1) * out_pixel_stride * out_es + out_c * out_es;
    if (ranges_overlap(out, out_bytes, image, img_elems * in_es) || ranges_overlap(out, out_bytes, workspace, need))
        return fail(RDVC_E_UNSUPPORTED, "out overlaps the image or the workspace");

    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const FeLayout L = fe_layout(B, H, W, workspace);
    rdvc::CeStemParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.img = image;
    sp.sb = image_strides[0]; sp.sc = image_strides[1]; sp.sy = image_strides[2]; sp.sx = image_strides[3];
    sp.H = H; sp.W = W; sp.H1 = s.H1; sp.W1 = s.W1;
    sp.out = L.l1[0];
    sp.n_pix = static_cast<long long>(B) * s.H1 * s.W1;
    if (int rc = op_dtype == RDVC_DT_F16 ? dispatch_ce_stem_pack<__half>(in_dtype, sp, st)
                                         : dispatch_ce_stem_pack<__nv_bfloat16>(in_dtype, sp, st))
        return rc;

    const uint8_t* wp = static_cast<const uint8_t*>(packed_w);
    const float* bp = biases;
    // unit i: convolution of `in` -> raw y (and the downsample's raw y2), its statistics, then `form` -> a (a_ps);
    // z / zi: the residual input, or the stride-2 unit whose downsample this block adds
    auto unit = [&](int i, const void* in, long long in_ps, int Hin, int Win, int Ho, int Wo, void* y, void* y2,
                    int form, const void* z, long long z_ps, int zi, void* a, long long a_ps) {
        const CeUnit& u = CE_UNITS[i];
        const long long ps = u.n;                                   // 64, or 128 (layer2's 96 channels padded)
        rdvc::TapMaps<1> m;
        rdvc::TapParams p;
        if (int rc = context_unit_setup(u, in, in_ps, B, Hin, Win, Ho, Wo, op_dtype, wp, m, p)) return rc;
        p.out = y; p.out_ps = ps;
        p.out2 = y2;
        p.part = L.part[i];
        if (int rc = op_dtype == RDVC_DT_F16 ? dispatch_feature_conv<__half>(u, m, p, st)
                                             : dispatch_feature_conv<__nv_bfloat16>(u, m, p, st))
            return rc;
        wp += ce_unit_w_elems(u) * 2;
        bp += ce_unit_b_floats(u);
        const int nt = fe_unit_nt(i);
        rdvc::InFinParams f;
        f.part = L.part[i]; f.stats = L.stats[i];
        f.NT = nt; f.N = u.n;
        f.n_tx = p.n_tx; f.n_ty = p.n_ty; f.H = Ho; f.W = Wo;
        f.eps_lo = eps[u.conv]; f.eps_hi = u.ds >= 0 ? eps[u.ds] : 0.0;
        rdvc::in_finalize_kernel<<<dim3(nt / 32, B), dim3(32, rdvc::IN_FIN_SLICES), 0, st>>>(f);
        ++g_launches;
        if (cudaError_t e = cudaGetLastError()) return cuda_fail(e, "in_finalize_kernel launch");
        rdvc::InApplyParams ap;
        memset(&ap, 0, sizeof(ap));
        ap.y = y; ap.y_ps = ps;
        ap.z = z; ap.z_ps = ps;
        ap.st = L.stats[i]; ap.st_nt = nt;
        if (form == rdvc::IN_APPLY_DS) { ap.zst = L.stats[zi] + CE_UNITS[zi].n; ap.zst_nt = fe_unit_nt(zi); }
        ap.out = a; ap.out_ps = a_ps;
        ap.C = CE_LAYERS[u.conv].cout; ap.Cs = u.n;
        ap.hw = static_cast<long long>(Ho) * Wo;
        ap.n_pix = B * ap.hw;
        return op_dtype == RDVC_DT_F16 ? launch_in_apply<__half>(form, ap, st) : launch_in_apply<__nv_bfloat16>(form, ap, st);
    };
    using rdvc::IN_APPLY_RELU;
    using rdvc::IN_APPLY_RES;
    using rdvc::IN_APPLY_DS;
    const int H1 = s.H1, W1 = s.W1, H2 = s.H2, W2 = s.W2, H3 = s.H3, W3 = s.W3;
    uint8_t* const* l1 = L.l1;
    uint8_t* const* l2 = L.l2;
    uint8_t* const* l3 = L.l3;
    void* last = trunk ? out : static_cast<void*>(l3[8]);
    const long long last_ps = trunk ? out_pixel_stride : 128;
    int rc = 0;
    // TV:raft.py:145: convnormrelu; 146: layer1 = two residual blocks relu(x + relu(norm2(conv2(relu(norm1(conv1(x)))))))
    if ((rc = unit(0, l1[0], 64, H1, W1, H1, W1, l1[1], nullptr, IN_APPLY_RELU, nullptr, 0, 0, l1[2], 64))) return rc;
    if ((rc = unit(1, l1[2], 64, H1, W1, H1, W1, l1[3], nullptr, IN_APPLY_RELU, nullptr, 0, 0, l1[4], 64))) return rc;
    if ((rc = unit(2, l1[4], 64, H1, W1, H1, W1, l1[5], nullptr, IN_APPLY_RES, l1[2], 64, 0, l1[6], 64))) return rc;
    if ((rc = unit(3, l1[6], 64, H1, W1, H1, W1, l1[7], nullptr, IN_APPLY_RELU, nullptr, 0, 0, l1[8], 64))) return rc;
    if ((rc = unit(4, l1[8], 64, H1, W1, H1, W1, l1[9], nullptr, IN_APPLY_RES, l1[6], 64, 0, l1[10], 64))) return rc;
    // 147: layer2; its first block's downsample is the second accumulator of its stride-2 convolution, normalised in
    // the apply of the block's second convolution
    if ((rc = unit(5, l1[10], 64, H1, W1, H2, W2, l2[0], l2[1], IN_APPLY_RELU, nullptr, 0, 0, l2[2], 128))) return rc;
    if ((rc = unit(6, l2[2], 128, H2, W2, H2, W2, l2[3], nullptr, IN_APPLY_DS, l2[1], 128, 5, l2[4], 128))) return rc;
    if ((rc = unit(7, l2[4], 128, H2, W2, H2, W2, l2[5], nullptr, IN_APPLY_RELU, nullptr, 0, 0, l2[6], 128))) return rc;
    if ((rc = unit(8, l2[6], 128, H2, W2, H2, W2, l2[7], nullptr, IN_APPLY_RES, l2[4], 128, 0, l2[8], 128))) return rc;
    // 148: layer3
    if ((rc = unit(9, l2[8], 128, H2, W2, H3, W3, l3[0], l3[1], IN_APPLY_RELU, nullptr, 0, 0, l3[2], 128))) return rc;
    if ((rc = unit(10, l3[2], 128, H3, W3, H3, W3, l3[3], nullptr, IN_APPLY_DS, l3[1], 128, 9, l3[4], 128))) return rc;
    if ((rc = unit(11, l3[4], 128, H3, W3, H3, W3, l3[5], nullptr, IN_APPLY_RELU, nullptr, 0, 0, l3[6], 128))) return rc;
    if ((rc = unit(12, l3[6], 128, H3, W3, H3, W3, l3[7], nullptr, IN_APPLY_RES, l3[4], 128, 0, last, last_ps))) return rc;
    if (trunk) return RDVC_OK;
    // 150: conv, the context encoder's 1x1 instantiation
    return run_context_unit(CE_UNITS[13], rdvc::TAP_EPI_RAW, l3[8], 128, B, H3, W3, H3, W3, op_dtype, wp, bp, out,
                            out_pixel_stride, out_dtype, nullptr, nullptr, 0, st);
}

}  // extern "C"

// ---- the whole RAFT call: every network on the library's kernels, caller-owned memory, no allocation ------------
namespace {

constexpr int RAFT_LEVELS = 4, RAFT_RADIUS = 4;
constexpr uint32_t RAFT_MAGIC = 0x54464152u;     // "RAFT", little-endian
constexpr uint32_t RAFT_BLOB_VERSION = 1;
constexpr double RAFT_NORM_EPS = 1e-5;            // torchvision's BatchNorm2d / InstanceNorm2d default

// sections of the packed blob, in blob order (include/rdvc_corr.h)
enum {
    RS_FE_W, RS_FE_B, RS_CE_W, RS_CE_B, RS_TAIL_W, RS_TAIL_B, RS_CC1_W, RS_CC1_B,
    RS_ME_W, RS_ME_B = RS_ME_W + 4, RS_FH_W = RS_ME_B + 4, RS_FH_B = RS_FH_W + 2, RS_GRU_W = RS_FH_B + 2,
    RS_GRU_B = RS_GRU_W + 2, RS_MASK_W = RS_GRU_B + 6, RS_MASK_B = RS_MASK_W + 2, RS_COUNT = RS_MASK_B + 2
};
static_assert(RS_COUNT == RDVC_RAFT_SECTIONS, "section count of include/rdvc_corr.h");

struct RaftBlobHeader {
    uint32_t magic, version;
    int32_t op_dtype, sections;
    uint64_t offset[RS_COUNT], bytes[RS_COUNT];
};

constexpr int ME_LAYERS[4] = {RDVC_UC_CONVCORR2, RDVC_UC_CONVFLOW1, RDVC_UC_CONVFLOW2, RDVC_UC_CONV};

size_t raft_sections(uint64_t* off, uint64_t* bytes) {
    uint64_t b[RS_COUNT];
    b[RS_FE_W] = b[RS_CE_W] = rdvc_corr_context_encoder_packed_weight_bytes();
    b[RS_FE_B] = b[RS_CE_B] = rdvc_corr_context_encoder_packed_bias_bytes();
    b[RS_TAIL_W] = rdvc_linear_packed_weight_bytes(rdvc::ET_N, rdvc::ET_K);
    b[RS_TAIL_B] = rdvc::ET_N * 4;
    b[RS_CC1_W] = rdvc_conv1x1_packed_weight_bytes(256, RAFT_LEVELS, RAFT_RADIUS);
    b[RS_CC1_B] = 256 * 4;
    for (int i = 0; i < 4; ++i) {
        b[RS_ME_W + i] = rdvc_corr_update_conv_packed_weight_bytes(ME_LAYERS[i]);
        b[RS_ME_B + i] = UC_LAYERS[ME_LAYERS[i]].cout * 4;
    }
    b[RS_FH_W] = rdvc_corr_update_conv_packed_weight_bytes(RDVC_UC_FH_CONV1);
    b[RS_FH_W + 1] = rdvc_corr_update_conv_packed_weight_bytes(RDVC_UC_FH_CONV2);
    b[RS_FH_B] = 256 * 4;
    b[RS_FH_B + 1] = 2 * 4;
    b[RS_GRU_W] = b[RS_GRU_W + 1] = rdvc_corr_convgru_packed_weight_bytes();
    for (int i = 0; i < 6; ++i) b[RS_GRU_B + i] = rdvc::GRU_C * 4;
    b[RS_MASK_W] = rdvc_corr_update_conv_packed_weight_bytes(RDVC_UC_FH_CONV1);
    b[RS_MASK_W + 1] = rdvc_corr_mask_conv_packed_weight_bytes();
    b[RS_MASK_B] = 256 * 4;
    b[RS_MASK_B + 1] = rdvc::MU_COUT * 4;
    size_t o = align_up(sizeof(RaftBlobHeader), 256);
    for (int i = 0; i < RS_COUNT; ++i) {
        if (off) off[i] = o;
        if (bytes) bytes[i] = b[i];
        o = align_up(o + b[i], 256);
    }
    return o;
}

// state_dict keys of torchvision's raft_large and where each one goes
enum RaftKind { RK_IGNORE, RK_FE_W, RK_FE_B, RK_CE_W, RK_CE_B, RK_BN_W, RK_BN_B, RK_BN_M, RK_BN_V, RK_GRU_W, RK_SECTION };
struct RaftKey {
    std::string name;
    std::vector<long long> shape;
    int kind, index;              // RK_*; index: encoder layer, 3 * ConvGRU + (z, r, q), or the section of a lone tensor
};

const std::vector<RaftKey>& raft_keys() {
    static const std::vector<RaftKey> keys = [] {
        std::vector<RaftKey> k;
        // the encoders' 16 convolutions in the order of the context-encoder pack arrays: (module, cout, cin, kernel)
        struct Conv { const char* name; int cout, cin, ks; };
        static const Conv enc[RDVC_CE_LAYERS] = {
            {"convnormrelu", 64, 3, 7},
            {"layer1.0.convnormrelu1", 64, 64, 3}, {"layer1.0.convnormrelu2", 64, 64, 3},
            {"layer1.1.convnormrelu1", 64, 64, 3}, {"layer1.1.convnormrelu2", 64, 64, 3},
            {"layer2.0.convnormrelu1", 96, 64, 3}, {"layer2.0.downsample", 96, 64, 1},
            {"layer2.0.convnormrelu2", 96, 96, 3}, {"layer2.1.convnormrelu1", 96, 96, 3},
            {"layer2.1.convnormrelu2", 96, 96, 3},
            {"layer3.0.convnormrelu1", 128, 96, 3}, {"layer3.0.downsample", 128, 96, 1},
            {"layer3.0.convnormrelu2", 128, 128, 3}, {"layer3.1.convnormrelu1", 128, 128, 3},
            {"layer3.1.convnormrelu2", 128, 128, 3},
            {"conv", 256, 128, 1},
        };
        for (int e = 0; e < 2; ++e) {
            const std::string pre = e == 0 ? "feature_encoder." : "context_encoder.";
            for (int i = 0; i < RDVC_CE_LAYERS; ++i) {
                const Conv& c = enc[i];
                const std::string conv = pre + c.name + (i < RDVC_CE_LAYERS - 1 ? ".0" : "");
                k.push_back({conv + ".weight", {c.cout, c.cin, c.ks, c.ks}, e ? RK_CE_W : RK_FE_W, i});
                k.push_back({conv + ".bias", {c.cout}, e ? RK_CE_B : RK_FE_B, i});
                if (e == 1 && i < RDVC_CE_LAYERS - 1) {
                    const std::string bn = pre + c.name + ".1";
                    k.push_back({bn + ".weight", {c.cout}, RK_BN_W, i});
                    k.push_back({bn + ".bias", {c.cout}, RK_BN_B, i});
                    k.push_back({bn + ".running_mean", {c.cout}, RK_BN_M, i});
                    k.push_back({bn + ".running_var", {c.cout}, RK_BN_V, i});
                    k.push_back({bn + ".num_batches_tracked", {}, RK_IGNORE, i});
                }
            }
        }
        // single tensors, each packed into (weights) or copied to (biases) one section
        auto conv = [&](const std::string& name, int cout, int cin, int kh, int kw, int w_section, int b_section,
                        int w_kind = RK_SECTION) {
            k.push_back({name + ".weight", {cout, cin, kh, kw}, w_kind, w_section});
            k.push_back({name + ".bias", {cout}, RK_SECTION, b_section});
        };
        const std::string me = "update_block.motion_encoder.";
        conv(me + "convcorr1.0", 256, RAFT_LEVELS * (2 * RAFT_RADIUS + 1) * (2 * RAFT_RADIUS + 1), 1, 1, RS_CC1_W, RS_CC1_B);
        const char* me_names[4] = {"convcorr2.0", "convflow1.0", "convflow2.0", "conv.0"};
        for (int i = 0; i < 4; ++i) {
            const UcLayer& L = UC_LAYERS[ME_LAYERS[i]];
            conv(me + me_names[i], L.cout, L.cin, L.k, L.k, RS_ME_W + i, RS_ME_B + i);
        }
        for (int g = 0; g < 2; ++g)
            for (int q = 0; q < 3; ++q) {
                const std::string name = std::string("update_block.recurrent_block.convgru") + (g ? "2" : "1") + ".conv" + "zrq"[q];
                conv(name, rdvc::GRU_C, 3 * rdvc::GRU_C, g ? 5 : 1, g ? 1 : 5, 3 * g + q, RS_GRU_B + 3 * g + q, RK_GRU_W);
            }
        conv("update_block.flow_head.conv1", 256, 128, 3, 3, RS_FH_W, RS_FH_B);
        conv("update_block.flow_head.conv2", 2, 256, 3, 3, RS_FH_W + 1, RS_FH_B + 1);
        conv("mask_predictor.convrelu.0", 256, 128, 3, 3, RS_MASK_W, RS_MASK_B);
        conv("mask_predictor.conv", rdvc::MU_COUT, rdvc::MU_CIN, 1, 1, RS_MASK_W + 1, RS_MASK_B + 1);
        return k;
    }();
    return keys;
}

std::string shape_str(const long long* s, int nd) {
    std::string r = "(";
    for (int i = 0; i < nd; ++i) r += std::to_string(s[i]) + (i + 1 < nd ? ", " : nd == 1 ? "," : "");
    return r + ")";
}

// the workspace: persistent buffers first, then one scratch region shared by the three phases (encoders, context
// encoder, refinement loop), whose buffers' lifetimes do not overlap
struct RaftLayout {
    size_t pyr, hc, coords, flow, scratch;
    size_t trunk, enc_ws, tail_in, tail_out;          // phase 1: feature encoder, pack, encoder tail, build
    size_t ce_ws;                                     // phase 2: context encoder
    size_t feat, c1, motion, g1, hid, loop_ws;        // phase 3: the iterations and the mask predictor
    size_t total;
};

RaftLayout raft_layout(int n_images, int B, int H, int W, int act_dtype, int vol_dtype) {
    RaftLayout L;
    memset(&L, 0, sizeof(L));
    const int h = H / 8, w = W / 8;
    const size_t px = static_cast<size_t>(B) * h * w, aes = elem_size(act_dtype);
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t at = o; o = align_up(o + bytes, 256); return at; };
    L.pyr = take(rdvc_corr_pyramid_bytes(B, h, w, RAFT_LEVELS, vol_dtype, RDVC_LAYOUT_TILED));
    L.hc = take(px * 256 * aes);
    L.coords = take(px * 2 * 4);
    L.flow = take(px * 2 * 4);
    L.scratch = o;
    L.trunk = take(static_cast<size_t>(n_images) * h * w * rdvc::ET_K * 2);
    const size_t after_trunk = o;
    L.enc_ws = take(rdvc_corr_feature_encoder_workspace_bytes(n_images, H, W, act_dtype));
    size_t end1 = o;
    o = after_trunk;
    L.tail_in = take(rdvc_corr_workspace_bytes(B, rdvc::ET_K, h, w));
    L.tail_out = take(rdvc_corr_workspace_bytes(B, rdvc::ET_N, h, w));
    end1 = std::max(end1, o);
    o = L.scratch;
    L.ce_ws = take(rdvc_corr_context_encoder_workspace_bytes(B, H, W, act_dtype));
    const size_t end2 = o;
    o = L.scratch;
    L.feat = take(rdvc_corr_feat_bytes(B, h, w, RAFT_LEVELS, RAFT_RADIUS));
    L.c1 = take(px * 256 * 2);
    L.motion = take(px * 128 * aes);
    L.g1 = take(px * rdvc::GRU_C * aes);
    L.hid = take(px * rdvc::GRU_C * aes);
    L.loop_ws = take(std::max(std::max(rdvc_corr_convgru_workspace_bytes(B, h, w, act_dtype),
                                       rdvc_corr_motion_encoder_workspace_bytes(B, h, w)),
                              std::max(rdvc_corr_flow_head_workspace_bytes(B, h, w, act_dtype),
                                       rdvc_corr_mask_predictor_workspace_bytes(B, h, w, act_dtype))));
    L.total = std::max(std::max(end1, end2), o);
    return L;
}

int raft_check_sizes(int n_images, int B, int H, int W, int act_dtype, int vol_dtype) {
    if (B <= 0 || H <= 0 || W <= 0 || n_images <= B || n_images > 2 * B)
        return fail(RDVC_E_SHAPE, "bad sizes: %d images, %d pairs, H=%d W=%d", n_images, B, H, W);
    if (H % 8 || W % 8) return fail(RDVC_E_SHAPE, "input image H and W should be divisible by 8, got H=%d W=%d", H, W);
    const int min_fmap = 2 << (RAFT_LEVELS - 1);
    if (H / 8 < min_fmap || W / 8 < min_fmap)
        return fail(RDVC_E_TOO_SMALL, "feature maps %d x %d are under %d per side: H and W must be at least %d", H / 8, W / 8,
                    min_fmap, 8 * min_fmap);
    if (act_dtype != RDVC_DT_F32 && act_dtype != RDVC_DT_F16)
        return fail(RDVC_E_DTYPE, "act_dtype must be F32 or F16, got %d", act_dtype);
    if (vol_dtype != RDVC_DT_F32 && vol_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "vol_dtype must be F32 or BF16, got %d", vol_dtype);
    if (H >= (1 << 24) || W >= (1 << 24) || static_cast<long long>(n_images) * H * W >= (1LL << 31))
        return fail(RDVC_E_UNSUPPORTED, "too many pixels for 32-bit TMA coordinates");
    return RDVC_OK;
}

// one call of either form: the feature encoder sees `images` (one run of n_images frames, or image1 then image2),
// pair b is (trunk row b, trunk row b + pair_offset)
int raft_run(const void* image1, const void* image2, const long long* s, int in_dtype, int n_images, int B, int H, int W,
             int iters, int act_dtype, int vol_dtype, const void* packed_weights, float mask_multiplier, void* workspace,
             size_t workspace_bytes, float* flow_out, void* stream) {
    if (!image1 || !s || !packed_weights || !workspace || !flow_out) return fail(RDVC_E_NULL, "null pointer argument");
    if (int rc = raft_check_sizes(n_images, B, H, W, act_dtype, vol_dtype)) return rc;
    if (iters < 1) return fail(RDVC_E_SHAPE, "iters must be >= 1, got %d", iters);
    if (in_dtype != RDVC_DT_F32 && in_dtype != RDVC_DT_F16 && in_dtype != RDVC_DT_BF16)
        return fail(RDVC_E_DTYPE, "unsupported in_dtype=%d", in_dtype);
    for (int i = 0; i < 4; ++i)
        if (s[i] < 0) return fail(RDVC_E_UNSUPPORTED, "negative image stride %lld", s[i]);
    const size_t in_es = elem_size(in_dtype);
    if ((reinterpret_cast<uintptr_t>(image1) % in_es) || (reinterpret_cast<uintptr_t>(image2) % in_es))
        return fail(RDVC_E_ALIGN, "the images must be aligned to their element size");
    if ((reinterpret_cast<uintptr_t>(packed_weights) & 255) || (reinterpret_cast<uintptr_t>(workspace) & 255) ||
        (reinterpret_cast<uintptr_t>(flow_out) & 15))
        return fail(RDVC_E_ALIGN, "packed weights and workspace must be 256-byte aligned, flow_out 16-byte aligned");
    const RaftLayout L = raft_layout(n_images, B, H, W, act_dtype, vol_dtype);
    if (workspace_bytes < L.total) return fail(RDVC_E_WORKSPACE, "workspace %zu < required %zu", workspace_bytes, L.total);
    const long long n_in = image2 ? B : n_images;      // images per feature-encoder call
    const long long dims[4] = {n_in, 3, H, W};
    size_t img_elems = 1;
    for (int i = 0; i < 4; ++i) img_elems += static_cast<size_t>(dims[i] - 1) * static_cast<size_t>(s[i]);
    const size_t out_bytes = static_cast<size_t>(B) * 2 * H * W * 4;
    const void* imgs[2] = {image1, image2};
    for (const void* im : imgs)
        if (im && (ranges_overlap(im, img_elems * in_es, workspace, L.total) ||
                   ranges_overlap(im, img_elems * in_es, flow_out, out_bytes)))
            return fail(RDVC_E_UNSUPPORTED, "an image overlaps the workspace or flow_out");
    if (ranges_overlap(flow_out, out_bytes, workspace, L.total))
        return fail(RDVC_E_UNSUPPORTED, "flow_out overlaps the workspace");

    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int h = H / 8, w = W / 8, op = RDVC_DT_F16;
    const long long hw = static_cast<long long>(h) * w;
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    const uint8_t* pk = static_cast<const uint8_t*>(packed_weights);
    uint64_t off[RS_COUNT];
    raft_sections(off, nullptr);
    auto sec = [&](int i) { return static_cast<const void*>(pk + off[i]); };
    auto fsec = [&](int i) { return reinterpret_cast<const float*>(pk + off[i]); };
    void* pyr = ws + L.pyr;
    uint8_t* hc = ws + L.hc;
    float* coords = reinterpret_cast<float*>(ws + L.coords);
    float* flow = reinterpret_cast<float*>(ws + L.flow);
    __half* trunk = reinterpret_cast<__half*>(ws + L.trunk);
    const size_t enc_ws_bytes = rdvc_corr_feature_encoder_workspace_bytes(n_images, H, W, act_dtype);
    const size_t tail_in_bytes = rdvc_corr_workspace_bytes(B, rdvc::ET_K, h, w);
    const size_t tail_out_bytes = rdvc_corr_workspace_bytes(B, rdvc::ET_N, h, w);
    double eps[RDVC_FE_NORMS];
    for (double& e : eps) e = RAFT_NORM_EPS;

    // 1. feature encoder -> layer3's trunk, NHWC fp16; the encoder tail (pack + 1x1 GEMM) and the build on it
    for (int i = 0; i < (image2 ? 2 : 1); ++i)
        if (int rc = rdvc_corr_feature_encoder(imgs[i], s, in_dtype, static_cast<int>(n_in), H, W, op, sec(RS_FE_W),
                                               fsec(RS_FE_B), eps, RDVC_FE_OUT_TRUNK, ws + L.enc_ws, enc_ws_bytes,
                                               trunk + i * n_in * hw * rdvc::ET_K, rdvc::ET_K, op, stream))
            return rc;
    const long long pair_offset = (image2 ? B : 1) * hw * rdvc::ET_K;
    if (int rc = rdvc_corr_pack_nhwc(trunk, trunk + pair_offset, rdvc::ET_K, B, rdvc::ET_K, h, w, op, vol_dtype,
                                     RDVC_LAYOUT_TILED, RAFT_LEVELS, ws + L.tail_in, tail_in_bytes, stream))
        return rc;
    if (int rc = rdvc_corr_encoder_tail(ws + L.tail_in, tail_in_bytes, rdvc::ET_K, sec(RS_TAIL_W), fsec(RS_TAIL_B),
                                        rdvc::ET_N, B, h, w, op, vol_dtype, RDVC_LAYOUT_TILED, RAFT_LEVELS, ws + L.tail_out,
                                        tail_out_bytes, stream))
        return rc;
    if (int rc = rdvc_corr_build_packed(B, rdvc::ET_N, h, w, op, pyr, vol_dtype, RDVC_LAYOUT_TILED, RAFT_LEVELS,
                                        ws + L.tail_out, tail_out_bytes, stream))
        return rc;
    // 2. context encoder: tanh(hidden) | relu(context), one NHWC buffer in the activation dtype
    if (int rc = rdvc_corr_context_encoder(image1, s, in_dtype, B, H, W, op, sec(RS_CE_W), fsec(RS_CE_B), RDVC_CE_OUT_SPLIT,
                                           ws + L.ce_ws, rdvc_corr_context_encoder_workspace_bytes(B, H, W, act_dtype), hc,
                                           256, act_dtype, stream))
        return rc;
    // 3. coords1 = grid, flow = 0; then the iterations
    {
        const long long n = B * hw;
        const unsigned grid = static_cast<unsigned>(std::min<long long>((n + 255) / 256, 4LL * sm_count()));
        rdvc::raft_coords_init_kernel<<<grid, 256, 0, st>>>(coords, flow, B, h, w);
        ++g_launches;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return cuda_fail(e, "raft_coords_init_kernel launch");
    }
    const long long fs[4] = {2 * hw, hw, w, 1};
    const size_t aes = elem_size(act_dtype);
    const void* me_w[4] = {sec(RS_ME_W), sec(RS_ME_W + 1), sec(RS_ME_W + 2), sec(RS_ME_W + 3)};
    const float* me_b[4] = {fsec(RS_ME_B), fsec(RS_ME_B + 1), fsec(RS_ME_B + 2), fsec(RS_ME_B + 3)};
    void* loop_ws = ws + L.loop_ws;
    const size_t loop_ws_bytes = L.total - L.loop_ws;
    const void* ctx = hc + 128 * aes;
    void* hid = ws + L.hid;
    const void* hcur = hc;                               // iteration 0: the hidden half of the context encoder's output
    long long hps = 256;
    for (int it = 0; it < iters; ++it) {
        if (int rc = rdvc_corr_lookup_conv1x1_ex(pyr, vol_dtype, RDVC_LAYOUT_TILED, coords, B, h, w, RAFT_LEVELS, RAFT_RADIUS,
                                                 sec(RS_CC1_W), fsec(RS_CC1_B), 256, RDVC_ACT_RELU, op, ws + L.feat,
                                                 rdvc_corr_feat_bytes(B, h, w, RAFT_LEVELS, RAFT_RADIUS), ws + L.c1, op,
                                                 256, stream))
            return rc;
        if (int rc = rdvc_corr_motion_encoder(ws + L.c1, 256, flow, fs, B, h, w, op, me_w, me_b, loop_ws, loop_ws_bytes,
                                              ws + L.motion, 128, act_dtype, stream))
            return rc;
        for (int g = 0; g < 2; ++g)      // convgru1 (1 x 5) -> g1, convgru2 (5 x 1) -> hid
            if (int rc = rdvc_corr_convgru(g ? ws + L.g1 : hcur, g ? 128 : hps, ctx, 256, ws + L.motion, 128, act_dtype, op,
                                           g ? RDVC_GRU_VERTICAL : RDVC_GRU_HORIZONTAL, B, h, w, sec(RS_GRU_W + g),
                                           fsec(RS_GRU_B + 3 * g), fsec(RS_GRU_B + 3 * g + 1), fsec(RS_GRU_B + 3 * g + 2),
                                           loop_ws, loop_ws_bytes, g ? hid : ws + L.g1, stream))
                return rc;
        hcur = hid;
        hps = 128;
        // flow head; its conv2 epilogue adds delta (rounded to act_dtype) to coords1 and writes flow = coords1 - grid
        const void* h16 = hid;
        long long h16_ps = 128;
        uint8_t* fh = static_cast<uint8_t*>(loop_ws);
        if (int rc = hidden_operand(&h16, &h16_ps, act_dtype, op, B * hw, fh + uc_plane_bytes(B, h, w, 256), stream))
            return rc;
        if (int rc = rdvc_corr_update_conv(RDVC_UC_FH_CONV1, h16, h16_ps, nullptr, nullptr, B, h, w, op, sec(RS_FH_W),
                                           fsec(RS_FH_B), fh, 256, op, stream))
            return rc;
        if (int rc = launch_update_conv(RDVC_UC_FH_CONV2, fh, 256, nullptr, nullptr, B, h, w, op, sec(RS_FH_W + 1),
                                        fsec(RS_FH_B + 1), coords, 0, act_dtype, flow, st))
            return rc;
    }
    // 4. mask predictor + convex 8x upsampling of the last flow, straight into flow_out
    const void* mw[2] = {sec(RS_MASK_W), sec(RS_MASK_W + 1)};
    const float* mb[2] = {fsec(RS_MASK_B), fsec(RS_MASK_B + 1)};
    return rdvc_corr_mask_predictor(hid, 128, act_dtype, B, h, w, op, mw, mb, mask_multiplier, flow, fs,
                                    RDVC_MASK_OUT_UPSAMPLED, loop_ws, loop_ws_bytes, flow_out, stream);
}

}  // namespace

extern "C" {

size_t rdvc_corr_raft_packed_weight_bytes(int op_dtype) {
    return op_dtype == RDVC_DT_F16 ? raft_sections(nullptr, nullptr) : 0;
}

int rdvc_corr_raft_pack_weights(const char* const* names, const float* const* tensors, const int* ndims,
                           const long long* const* shapes, int n, int op_dtype, void* packed_host, size_t bytes) {
    if (!names || !tensors || !ndims || !shapes || !packed_host) return fail(RDVC_E_NULL, "null pointer argument");
    if (op_dtype != RDVC_DT_F16)
        return fail(RDVC_E_DTYPE, "op_dtype must be F16 (the operand type of both activation dtypes), got %d", op_dtype);
    if (n < 0) return fail(RDVC_E_SHAPE, "negative tensor count %d", n);
    uint64_t off[RS_COUNT], sz[RS_COUNT];
    const size_t need = raft_sections(off, sz);
    if (bytes < need) return fail(RDVC_E_WORKSPACE, "packed_host holds %zu bytes < required %zu", bytes, need);
    const std::vector<RaftKey>& keys = raft_keys();
    std::vector<const float*> found(keys.size(), nullptr);
    for (int i = 0; i < n; ++i) {
        if (!names[i]) return fail(RDVC_E_NULL, "names[%d] is NULL", i);
        size_t k = 0;
        while (k < keys.size() && keys[k].name != names[i]) ++k;
        if (k == keys.size()) return fail(RDVC_E_UNSUPPORTED, "unexpected key %s (not in raft_large's state_dict)", names[i]);
        const RaftKey& key = keys[k];
        if (key.kind == RK_IGNORE) continue;
        if (found[k]) return fail(RDVC_E_UNSUPPORTED, "duplicate key %s", names[i]);
        if (!tensors[i] || (ndims[i] > 0 && !shapes[i])) return fail(RDVC_E_NULL, "key %s: NULL tensor or shape", names[i]);
        const int nd = static_cast<int>(key.shape.size());
        bool same = ndims[i] == nd;
        for (int d = 0; same && d < nd; ++d) same = shapes[i][d] == key.shape[d];
        if (!same)
            return fail(RDVC_E_SHAPE, "key %s has shape %s, raft_large's is %s", names[i],
                        shape_str(ndims[i] > 0 ? shapes[i] : nullptr, std::max(ndims[i], 0)).c_str(),
                        shape_str(key.shape.data(), nd).c_str());
        found[k] = tensors[i];
    }
    const float* fe_w[RDVC_CE_LAYERS] = {}; const float* fe_b[RDVC_CE_LAYERS] = {};
    const float* ce_w[RDVC_CE_LAYERS] = {}; const float* ce_b[RDVC_CE_LAYERS] = {};
    const float* bn[4][RDVC_CE_LAYERS] = {};
    const float* single[RS_COUNT] = {};
    const float* gru[2][3] = {};
    for (size_t k = 0; k < keys.size(); ++k) {
        const RaftKey& key = keys[k];
        if (key.kind == RK_IGNORE) continue;
        if (!found[k]) return fail(RDVC_E_SHAPE, "missing key %s", key.name.c_str());
        switch (key.kind) {
            case RK_FE_W:                // feature_encoder.conv (the last layer) is also the encoder tail's weight
                fe_w[key.index] = found[k];
                if (key.index == RDVC_CE_LAYERS - 1) single[RS_TAIL_W] = found[k];
                break;
            case RK_FE_B:
                fe_b[key.index] = found[k];
                if (key.index == RDVC_CE_LAYERS - 1) single[RS_TAIL_B] = found[k];
                break;
            case RK_CE_W: ce_w[key.index] = found[k]; break;
            case RK_CE_B: ce_b[key.index] = found[k]; break;
            case RK_BN_W: case RK_BN_B: case RK_BN_M: case RK_BN_V: bn[key.kind - RK_BN_W][key.index] = found[k]; break;
            case RK_GRU_W: gru[key.index / 3][key.index % 3] = found[k]; break;
            default: single[key.index] = found[k];
        }
    }
    uint8_t* blob = static_cast<uint8_t*>(packed_host);
    memset(blob, 0, need);
    RaftBlobHeader hdr;
    memset(&hdr, 0, sizeof(hdr));
    hdr.magic = RAFT_MAGIC; hdr.version = RAFT_BLOB_VERSION; hdr.op_dtype = op_dtype; hdr.sections = RS_COUNT;
    for (int i = 0; i < RS_COUNT; ++i) { hdr.offset[i] = off[i]; hdr.bytes[i] = sz[i]; }
    memcpy(blob, &hdr, sizeof(hdr));
    auto fout = [&](int i) { return reinterpret_cast<float*>(blob + off[i]); };
    // feature encoder: the context encoder's packing with the identity norm (scale exactly 1, each weight rounded once)
    std::vector<float> ones(256, 1.f), zeros(256, 0.f);
    const float* one[RDVC_CE_LAYERS]; const float* zero[RDVC_CE_LAYERS];
    double eps0[RDVC_CE_LAYERS], eps[RDVC_CE_LAYERS];
    for (int i = 0; i < RDVC_CE_LAYERS; ++i) {
        one[i] = ones.data(); zero[i] = zeros.data();
        eps0[i] = 0.0; eps[i] = RAFT_NORM_EPS;
    }
    int rc = rdvc_corr_context_encoder_pack_weights(fe_w, fe_b, one, zero, zero, one, eps0, op_dtype, blob + off[RS_FE_W],
                                                    fout(RS_FE_B));
    if (!rc) rc = rdvc_corr_context_encoder_pack_weights(ce_w, ce_b, bn[0], bn[1], bn[2], bn[3], eps, op_dtype,
                                                         blob + off[RS_CE_W], fout(RS_CE_B));
    if (!rc) rc = rdvc_linear_pack_weights(single[RS_TAIL_W], rdvc::ET_N, rdvc::ET_K, op_dtype, blob + off[RS_TAIL_W]);
    if (!rc) rc = rdvc_conv1x1_pack_weights(single[RS_CC1_W], 256, RAFT_LEVELS, RAFT_RADIUS, op_dtype, blob + off[RS_CC1_W]);
    for (int i = 0; i < 4 && !rc; ++i)
        rc = rdvc_corr_update_conv_pack_weights(ME_LAYERS[i], single[RS_ME_W + i], op_dtype, blob + off[RS_ME_W + i]);
    for (int i = 0; i < 2 && !rc; ++i)
        rc = rdvc_corr_update_conv_pack_weights(i ? RDVC_UC_FH_CONV2 : RDVC_UC_FH_CONV1, single[RS_FH_W + i], op_dtype,
                                                blob + off[RS_FH_W + i]);
    for (int g = 0; g < 2 && !rc; ++g)
        rc = rdvc_corr_convgru_pack_weights(gru[g][0], gru[g][1], gru[g][2], op_dtype, blob + off[RS_GRU_W + g]);
    if (!rc) rc = rdvc_corr_update_conv_pack_weights(RDVC_UC_FH_CONV1, single[RS_MASK_W], op_dtype, blob + off[RS_MASK_W]);
    if (!rc) rc = rdvc_corr_mask_conv_pack_weights(single[RS_MASK_W + 1], single[RS_MASK_B + 1], op_dtype,
                                                   blob + off[RS_MASK_W + 1], fout(RS_MASK_B + 1));
    if (rc) return rc;
    // biases used as they are: fp32 copies
    const int copies[] = {RS_TAIL_B, RS_CC1_B, RS_ME_B, RS_ME_B + 1, RS_ME_B + 2, RS_ME_B + 3, RS_FH_B, RS_FH_B + 1,
                          RS_GRU_B, RS_GRU_B + 1, RS_GRU_B + 2, RS_GRU_B + 3, RS_GRU_B + 4, RS_GRU_B + 5, RS_MASK_B};
    for (int i : copies) memcpy(blob + off[i], single[i], sz[i]);
    return RDVC_OK;
}

size_t rdvc_corr_raft_workspace_bytes(int n_images, int n_pairs, int H, int W, int act_dtype, int vol_dtype) {
    if (raft_check_sizes(n_images, n_pairs, H, W, act_dtype, vol_dtype)) return 0;     // the reason: rdvc_corr_last_error
    return raft_layout(n_images, n_pairs, H, W, act_dtype, vol_dtype).total;
}

int rdvc_corr_raft_flow(const void* image1, const void* image2, const long long* image_strides, int in_dtype, int B, int H,
                   int W, int iters, int act_dtype, int vol_dtype, const void* packed_weights, float mask_multiplier,
                   void* workspace, size_t workspace_bytes, float* flow_out, void* stream) {
    if (!image2) return fail(RDVC_E_NULL, "null pointer argument");
    return raft_run(image1, image2, image_strides, in_dtype, 2 * B, B, H, W, iters, act_dtype, vol_dtype, packed_weights,
                    mask_multiplier, workspace, workspace_bytes, flow_out, stream);
}

int rdvc_corr_raft_flow_sequence(const void* frames, const long long* frame_strides, int in_dtype, int n_frames, int H, int W,
                            int iters, int act_dtype, int vol_dtype, const void* packed_weights, float mask_multiplier,
                            void* workspace, size_t workspace_bytes, float* flow_out, void* stream) {
    return raft_run(frames, nullptr, frame_strides, in_dtype, n_frames, n_frames - 1, H, W, iters, act_dtype, vol_dtype,
                    packed_weights, mask_multiplier, workspace, workspace_bytes, flow_out, stream);
}

}  // extern "C"

// ---- next row f-4 (last piece): entropy-coder stand-in (host only) ----------------------------
extern "C" {

size_t rdvc_ec_max_encoded_bytes(size_t n) { return rdvc::ec::max_encoded_bytes(n); }

size_t rdvc_ec_encode_with_indexes(const int* symbols, const int* indexes, size_t n, const unsigned int* cdfs,
                                   const int* cdf_lengths, const int* offsets, int n_tables, int max_len,
                                   unsigned char* out, size_t out_capacity) {
    if ((n && (!symbols || !indexes)) || !cdfs || !cdf_lengths || !offsets || !out) {
        fail(RDVC_E_NULL, "null pointer argument");
        return 0;
    }
    const size_t r = rdvc::ec::encode_with_indexes(symbols, indexes, n, cdfs, cdf_lengths, offsets, n_tables, max_len,
                                                   out, out_capacity);
    if (r == 0) fail(RDVC_E_UNSUPPORTED, "entropy encode failed: malformed CDF table / index, or output buffer too small");
    return r;
}

int rdvc_ec_decode_with_indexes(const unsigned char* in, size_t nbytes, const int* indexes, size_t n,
                                const unsigned int* cdfs, const int* cdf_lengths, const int* offsets, int n_tables,
                                int max_len, int* symbols_out) {
    if ((n && (!in || !indexes || !symbols_out)) || !cdfs || !cdf_lengths || !offsets)
        return fail(RDVC_E_NULL, "null pointer argument");
    if (rdvc::ec::decode_with_indexes(in, nbytes, indexes, n, cdfs, cdf_lengths, offsets, n_tables, max_len, symbols_out))
        return fail(RDVC_E_UNSUPPORTED, "entropy decode failed: truncated or malformed stream / table");
    return RDVC_OK;
}

}  // extern "C"
