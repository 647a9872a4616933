// rrt_b200.cu -- host side of librrt_b200.so: context, launch logic and the C ABI of include/rrt.h, plus the
// strict-contract instantiation of the kernels (this unit is compiled -fmad=false; rrt_fmad.cu holds the other).
//
// Replaces, for the hot path only, raymarch_kernel + launch_raymarch (reference src/raymarcher.cu:15-180).
//
// Where things are:
//   include/rrt_device.cuh   device math: the two rounding contracts, geodesic RHS, RK4, noise, densities
//   csrc/rrt_kernel.cuh      render_kernel (one 8x4 tile per persistent warp), per-ray helpers, shade_kernel,
//                            resolve_kernel, probe kernels
//   csrc/rrt_packed.cuh      render_kernel_p (two rays per thread, no medium), FMAD contract only
//   csrc/rrt_split.cuh       the split pipeline of launches with a medium: trace / media / fold kernels
//                            (every kernel that creates rays also has LENS variants: rrt_render_dof's per-sub-sample cameras
//                            and rrt_render_pano's equirectangular directions)
//   this file                band assembly, self-test / roofline probes, rrt_context, every extern "C" entry point
//
// Launch organisation (B200: 148 SMs, no tensor-core work on this path -- it is FP32 FMA-pipe bound):
//   * persistent warps: grid = SMs x resident CTAs (or 1/n of them with n frames in flight); each warp pulls
//     8x4-pixel tiles from a global atomic ticket until the frame is exhausted;
//   * ray state lives in registers for the whole ray; camera, effects and every derived constant arrive in the
//     kernel parameter block (constant bank) and are read as free FFMA/FMUL operands;
//   * the skybox is a texture object (wrap-x / clamp-y / linear), 33.5 MB, L2-resident;
//   * outputs: 4 B/pixel uchar4 (row-flipped like the reference) plus optional float4 parity planes.
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <climits>
#include <cstddef>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "../../include/rrt.h"
#include "../../include/rrt_device.cuh"

using rrt::Consts;
using rrt::V3;
using rrt::mk;

#include "rrt_kernel.cuh"

namespace {

// ---- band assembly on the encoding GPU ------------------------------------------------------------
__global__ void assemble_kernel(const uchar4* __restrict__ packed, int rows_per_rank, int w, int h, int nranks,
                                int group, uchar4* __restrict__ frame) {
    const size_t n = (size_t)w * h;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int y = (int)(i / w), x = (int)(i - (size_t)y * w);
        const int g = y / group, rank = g % nranks, lg = g / nranks;
        const int ly = lg * group + (y - g * group);
        frame[(size_t)(h - 1 - y) * w + x] = packed[((size_t)rank * rows_per_rank + ly) * w + x];
    }
}

// div_rn_fast / sqrt_rn_fast vs the IEEE intrinsics on random operands of the render loop's domain.
__device__ __forceinline__ unsigned long long mix64(unsigned long long z) {  // splitmix64 finaliser
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ float make_float(unsigned mant_bits, int exp2, bool neg) {
    return __uint_as_float((neg ? 0x80000000u : 0u) | ((unsigned)(exp2 + 127) << 23) | (mant_bits & 0x7fffffu));
}
__global__ void k_exact_math(unsigned long long seed, unsigned long long n, unsigned long long* bad) {
    unsigned long long bad_div = 0, bad_sqrt = 0;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const unsigned long long a = mix64(seed + 2 * i), b = mix64(seed + 2 * i + 1);
        // numerator: 0 (1/64 of draws) or +-2^[-60,40]; denominator: +-2^[-20,62]; sqrt argument: 2^[-40,80]
        float x = make_float((unsigned)a, (int)((a >> 23) % 101) - 60, (a >> 40) & 1);
        if (((a >> 41) & 63) == 0) x = 0.0f;
        const float y = make_float((unsigned)b, (int)((b >> 23) % 83) - 20, (b >> 40) & 1);
        const float s = make_float((unsigned)(a >> 8), (int)((b >> 41) % 121) - 40, false);
        if (!(rrt::div_rn_fast(x, y) == __fdiv_rn(x, y))) ++bad_div;
        if (!(rrt::sqrt_rn_fast(s) == __fsqrt_rn(s))) ++bad_sqrt;
    }
    if (bad_div) atomicAdd(bad + 0, bad_div);
    if (bad_sqrt) atomicAdd(bad + 1, bad_sqrt);
}

// pow_exp2(pow_log2(x), y) (include/rrt_device.cuh) vs libdevice's powf on random positive normal bases: the exponents the
// media code uses, and random ones.
__global__ void k_exact_pow(unsigned long long seed, unsigned long long n, unsigned long long* bad) {
    const float ys[8] = {0.5f, 0.4f, 1.5f, 1.6f, -0.75f, 4.0f, 1.2f, 0.2f};
    unsigned long long bad_used = 0, bad_rand = 0;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const unsigned long long a = mix64(seed + 2 * i), b = mix64(seed + 2 * i + 1);
        // base: half of the draws in the media code's range 2^[-8, 8], half in 2^[-60, 60]
        const int ex = (a >> 40) & 1 ? (int)((a >> 23) % 17) - 8 : (int)((a >> 23) % 121) - 60;
        const float x = make_float((unsigned)a, ex, false);
        const float y_used = ys[(b >> 50) & 7];
        const float y_rand = __uint_as_float((unsigned)b & 0x007fffffu | 0x3f800000u) * (float)((int)((b >> 30) % 9) - 3) * 0.73f + 0.011f;
        const rrt::PowLog L = rrt::pow_log2(x);
        const float g0 = rrt::pow_exp2(L, y_used), w0 = powf(x, y_used);
        const float g1 = rrt::pow_exp2(L, y_rand), w1 = powf(x, y_rand);
        if (__float_as_uint(g0) != __float_as_uint(w0)) ++bad_used;
        if (__float_as_uint(g1) != __float_as_uint(w1) && !(g1 != g1 && w1 != w1)) ++bad_rand;
    }
    if (bad_used) atomicAdd(bad + 0, bad_used);
    if (bad_rand) atomicAdd(bad + 1, bad_rand);
}

// FP32 roofline probe: 8 independent FFMA chains per thread, all operands in registers.
__global__ void __launch_bounds__(256) k_fp32_peak(int iters, float seed, float* sink) {
    float a0 = seed, a1 = seed + 1.f, a2 = seed + 2.f, a3 = seed + 3.f, a4 = seed + 4.f, a5 = seed + 5.f, a6 = seed + 6.f,
          a7 = seed + 7.f;
    const float m = 0.999f + seed * 1e-9f, c = 1e-3f + seed;
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            a0 = __fmaf_rn(a0, m, c); a1 = __fmaf_rn(a1, m, c); a2 = __fmaf_rn(a2, m, c); a3 = __fmaf_rn(a3, m, c);
            a4 = __fmaf_rn(a4, m, c); a5 = __fmaf_rn(a5, m, c); a6 = __fmaf_rn(a6, m, c); a7 = __fmaf_rn(a7, m, c);
        }
    }
    float s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 123456.789f) sink[0] = s;  // never true; keeps the chains alive
}

}  // namespace

// =================================== host side: context + C ABI ===================================

struct rrt_context {
    int device = -1;
    int sm_count = 0;
    unsigned long long* d_counters = nullptr;
    unsigned int* d_tickets = nullptr;
    unsigned ticket_next = 0;
    // fused FMAD launches without a medium use the packed f32x2 kernel (two rays per thread; measured,
    // profiles/r2_history.md) unless RRT_KERNEL=scalar pins the scalar one.  RRT_KERNEL=auto|scalar.
    bool scalar_kernel = false;
    // resident CTAs per SM of every kernel launched so far (carve-out applied): asked for once (resident_per_sm)
    std::vector<std::pair<const void*, int>> resident;
    void* d_frame[RRT_HOST_SLOTS] = {};  // device frames behind the host-destination calls, one per slot
    size_t d_frame_bytes[RRT_HOST_SLOTS] = {};
    unsigned long long* tile_log = nullptr;   // rrt_debug_tile_log: caller-owned device buffer, or null
    unsigned tile_log_cap = 0;
    bool probe_fmad = true;   // contract of the parameter-less probes (hash31 / noise3D / fbm): like rrt_default_params
    int frames_in_flight = 1; // render launches expected to run concurrently: each gets 1/n of the resident-CTA slots
    // split pipeline (csrc/rrt_split.cuh): trace / media / fold kernels over a sample pool, one pool per stream in flight
    int pipeline = RRT_PIPELINE_AUTO;
    int trace_choice = 0;                 // split pipeline's tracer: 0 auto (packed f32x2 under the FMAD contract), 1 scalar, 2 packed (RRT_TRACE)
    size_t pool_bytes_max = 16ull << 30;  // per pool (RRT_POOL_MB / rrt_set_sample_pool)
    int max_passes = 32;
    struct SamplePool {
        bool in_use = false;
        cudaStream_t stream = nullptr;
        uint4* d_slots = nullptr;
        size_t cap_slots = 0;
        char* d_ctrl = nullptr;           // PassCtrl[kMaxPasses + 1] | stats[8] | redo lists
        rrtk::TileDesc* d_desc = nullptr; // one per tile a pass can queue
        size_t desc_cap = 0;
        rrtk::WorkItem* d_work = nullptr; // media work items of one pass
        size_t work_cap = 0;
        unsigned* h_stats = nullptr;      // pinned copy of the stats of the last frame that completed on this pool
        cudaEvent_t done = nullptr;
        unsigned long long last_use = 0;
    };
    SamplePool pools[RRT_HOST_SLOTS];
    unsigned long long pool_clock = 0;
    int passes_hint = 2;                  // passes the last frame with history needed: the first guess of a pool without one
    // rrt_render_ss's supersampled hdr planes: stream-ordered allocations from this pool (created on first use), which
    // keeps freed blocks for the next frame instead of returning them to the device
    cudaMemPool_t ss_pool = nullptr;
    unsigned long long launches = 0;      // kernels this context has launched for rrt_render* / rrt_shade / rrt_resolve / rrt_assemble_bands
    std::string err;
    std::mutex mu;
};
struct rrt_sky {
    int device = -1;
    cudaArray_t arr = nullptr;
    cudaTextureObject_t tex = 0;
};

namespace {
constexpr int kMaxPasses = 32;          // split passes one frame can be cut into (then the sweep takes what is left)
constexpr unsigned kRedoCap = 16384;    // tiles one pass can give up: at most one per tracing warp
constexpr size_t kSlotBytes = 32;
constexpr size_t kPoolPadSlots = 64;    // fold_kernel reads a 33-slot window from any record header
constexpr size_t kCtrlHead = sizeof(rrtk::PassCtrl) * (kMaxPasses + 1) + 8 * sizeof(unsigned);   // zeroed per frame
constexpr size_t kCtrlBytes = kCtrlHead + sizeof(unsigned) * kRedoCap * (kMaxPasses + 1);
constexpr unsigned kTicketRing = 1024;
thread_local std::string g_create_err;

int fail(rrt_context* ctx, int code, const std::string& what, cudaError_t e = cudaSuccess) {
    std::string m = what;
    if (e != cudaSuccess) { m += ": "; m += cudaGetErrorString(e); }
    if (ctx) ctx->err = m; else g_create_err = m;
    return code;
}
#define RRT_CU(ctx, call)                                                    \
    do {                                                                     \
        cudaError_t e__ = (call);                                            \
        if (e__ != cudaSuccess) return fail(ctx, RRT_ERR_CUDA, #call, e__);  \
    } while (0)

// Derived constants in float, with the reference's own association (see include/rrt_device.cuh::Consts).
Consts make_consts(const rrt_params& P) {
    Consts C;
    std::memset(&C, 0, sizeof(C));
    C.horizon_r = P.event_horizon * 1.01f;
    C.acc_rmin = P.event_horizon * 0.5f;
    C.radial_k = -1.5f * P.event_horizon;
    C.drag_k = (2.0f * P.spin_a) * P.event_horizon;
    C.spin_a = P.spin_a;
    C.event_horizon = P.event_horizon;
    C.disk_zone_y = P.disk_h * 5.0f;
    C.disk_zone_r = P.disk_out + 5.0f;
    C.dust_zone_y = P.cloud_h * 1.5f;
    C.dust_zone_r = P.cloud_out;
    const float scale[4] = {1.0f, 0.1f, 0.3f, 0.5f};
    for (int i = 0; i < 4; ++i) {
        volatile float h = P.step_size;  // volatile: keep every intermediate in binary32
        if (i) h = h * scale[i];
        C.h[i] = h;
        volatile float hh = h * 0.5f;
        volatile float h6 = h / 6.0f;
        C.hh[i] = hh;
        C.h6[i] = h6;
    }
    C.isco = P.isco_radius;
    C.disk_out = P.disk_out;
    C.disk_h = P.disk_h;
    volatile float tf = P.disk_out * 0.85f;
    volatile float ts = P.disk_out - tf;
    C.taper_from = tf;
    C.taper_span = ts;
    C.dust_e1 = P.disk_out * 0.8f;
    C.dust_in_e1 = P.isco_radius + 5.0f;
    C.cloud_hh = P.cloud_h * 0.5f;
    C.disk_temp_ref = P.disk_temp_ref;
    C.disk_luminosity = P.disk_luminosity;
    C.disk_opacity = P.disk_opacity;
    C.cloud_luminosity = P.cloud_luminosity;
    C.cloud_opacity = P.cloud_opacity;
    C.exposure = P.exposure;
    C.max_steps = P.max_steps;
    C.flags = P.flags;
    C.neg_zero = -0.0f;
    return C;
}

struct DevGuard {
    int prev = -1;
    explicit DevGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// RAII device buffer for the probes
struct DBuf {
    void* p = nullptr;
    cudaError_t alloc(size_t n) { return cudaMalloc(&p, n ? n : 1); }
    ~DBuf() { if (p) cudaFree(p); }
};

const rrtk::KernelSet* kset(const rrt_params* prm) {
    return (prm->flags & RRT_FLAG_FMAD) ? rrtk::rrt_kernels_fmad() : rrtk::rrt_kernels_strict();
}
// hash31 / noise3D / fbm take no parameter block: rrt_set_probe_contract picks their contract per context
const rrtk::KernelSet* kset_noise(const rrt_context* ctx) {
    return ctx->probe_fmad ? rrtk::rrt_kernels_fmad() : rrtk::rrt_kernels_strict();
}

template <typename K, typename... Args>
int run_probe(rrt_context* ctx, int n, K kernel, Args... args) {
    if (n > 0) kernel<<<(n + 127) / 128, 128>>>(args...);
    RRT_CU(ctx, cudaGetLastError());
    RRT_CU(ctx, cudaDeviceSynchronize());
    return RRT_OK;
}
}  // namespace

extern "C" {

int rrt_abi_version(void) { return RRT_ABI_VERSION; }

const char* rrt_build_info(void) {
    return "librrt_b200 abi=1 arch=sm_100a prec-div=true prec-sqrt=true ftz=false; RRT_FLAG_FMAD (default contract) kernels: fmad=true, strict kernels: fmad=false (nvcc "
#define RRT_STR2(x) #x
#define RRT_STR(x) RRT_STR2(x)
           RRT_STR(__CUDACC_VER_MAJOR__) "." RRT_STR(__CUDACC_VER_MINOR__) ")";
}

const char* rrt_last_error(const rrt_context* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

int rrt_context_create(int device, rrt_context** out) {
    if (!out) return fail(nullptr, RRT_ERR_BAD_ARG, "rrt_context_create: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) return fail(nullptr, RRT_ERR_NO_DEVICE, "no CUDA device (this library has no CPU fallback)", e);
    if (device < 0 || device >= ndev) return fail(nullptr, RRT_ERR_BAD_ARG, "rrt_context_create: bad device ordinal");
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return fail(nullptr, RRT_ERR_CUDA, "cudaGetDeviceProperties", e);
    if (prop.major != 10) return fail(nullptr, RRT_ERR_NO_DEVICE, "device is not compute capability 10.x (library is built for sm_100a only)");
    rrt_context* ctx = new (std::nothrow) rrt_context();
    if (!ctx) return fail(nullptr, RRT_ERR_NOMEM, "out of host memory");
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    if (const char* k = std::getenv("RRT_KERNEL")) ctx->scalar_kernel = !std::strcmp(k, "scalar");
    if (const char* k = std::getenv("RRT_PIPELINE")) ctx->pipeline = !std::strcmp(k, "split") ? RRT_PIPELINE_SPLIT : (!std::strcmp(k, "fused") ? RRT_PIPELINE_FUSED : RRT_PIPELINE_AUTO);
    if (const char* k = std::getenv("RRT_TRACE")) ctx->trace_choice = !std::strcmp(k, "packed") ? 2 : (!std::strcmp(k, "scalar") ? 1 : 0);
    if (const char* k = std::getenv("RRT_POOL_MB")) { const long long mb = std::atoll(k); if (mb > 0) ctx->pool_bytes_max = (size_t)mb << 20; }
    if (const char* k = std::getenv("RRT_MAX_PASSES")) { const int n = std::atoi(k); if (n >= 1 && n <= kMaxPasses) ctx->max_passes = n; }
    DevGuard g(device);
    if ((e = cudaMalloc(&ctx->d_counters, sizeof(rrt_counters))) != cudaSuccess ||
        (e = cudaMemset(ctx->d_counters, 0, sizeof(rrt_counters))) != cudaSuccess ||
        (e = cudaMalloc(&ctx->d_tickets, kTicketRing * sizeof(unsigned))) != cudaSuccess ||
        (e = cudaMemset(ctx->d_tickets, 0, kTicketRing * sizeof(unsigned))) != cudaSuccess) {
        fail(nullptr, RRT_ERR_CUDA, "context allocation", e);
        rrt_context_destroy(ctx);
        return RRT_ERR_CUDA;
    }
    *out = ctx;
    return RRT_OK;
}

void rrt_context_destroy(rrt_context* ctx) {
    if (!ctx) return;
    DevGuard g(ctx->device);
    cudaDeviceSynchronize();
    if (ctx->d_counters) cudaFree(ctx->d_counters);
    if (ctx->d_tickets) cudaFree(ctx->d_tickets);
    for (void* f : ctx->d_frame)
        if (f) cudaFree(f);
    for (auto& pl : ctx->pools) {
        if (pl.d_slots) cudaFree(pl.d_slots);
        if (pl.d_ctrl) cudaFree(pl.d_ctrl);
        if (pl.d_desc) cudaFree(pl.d_desc);
        if (pl.d_work) cudaFree(pl.d_work);
        if (pl.h_stats) cudaFreeHost(pl.h_stats);
        if (pl.done) cudaEventDestroy(pl.done);
    }
    if (ctx->ss_pool) cudaMemPoolDestroy(ctx->ss_pool);
    delete ctx;
}

void rrt_default_params(rrt_params* o) {  // include/config.h
    if (!o) return;
    o->spin_a = 0.0f;
    o->event_horizon = 2.0f;
    o->isco_radius = 10.0f;
    o->disk_out = 25.0f;
    o->disk_h = 0.8f;
    o->disk_luminosity = 6.0f;
    o->disk_opacity = 0.4f;
    o->exposure = 0.8f;
    o->cloud_h = 0.5f;
    o->cloud_out = 25.0f;
    o->cloud_opacity = 0.3f;
    o->cloud_luminosity = 0.4f;
    o->step_size = 0.3f;
    o->disk_temp_ref = 1.5e7f;
    o->max_steps = 2000;
    o->flags = RRT_FLAG_DISK | RRT_FLAG_DUST | RRT_FLAG_FMAD;  // both media; the rounding contract of the reference's CUDA build
}

void rrt_default_effects(rrt_effects* o) {  // camera_settings.h:5-16
    if (!o) return;
    o->use_bloom = 1; o->bloom_threshold = 0.8f; o->bloom_intensity = 0.5f;
    o->use_vignette = 1; o->vignette_intensity = 0.4f;
    o->use_ca = 0; o->ca_amount = 0.005f;
    o->use_lens = 1; o->distortion_amount = 0.15f;
}

int rrt_sky_create(rrt_context* ctx, const uint8_t* host_rgba, int w, int h, rrt_sky** out) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!host_rgba || !out || w <= 0 || h <= 0) return fail(ctx, RRT_ERR_BAD_ARG, "rrt_sky_create: bad argument");
    *out = nullptr;
    DevGuard g(ctx->device);
    rrt_sky* s = new (std::nothrow) rrt_sky();
    if (!s) return fail(ctx, RRT_ERR_NOMEM, "out of host memory");
    s->device = ctx->device;
    // same recipe as the reference's loadSkybox (src/main.cpp:246-263)
    cudaChannelFormatDesc desc = cudaCreateChannelDesc(8, 8, 8, 8, cudaChannelFormatKindUnsigned);
    cudaError_t e = cudaMallocArray(&s->arr, &desc, (size_t)w, (size_t)h);
    if (e == cudaSuccess)
        e = cudaMemcpy2DToArray(s->arr, 0, 0, host_rgba, (size_t)w * 4, (size_t)w * 4, (size_t)h, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        cudaResourceDesc rd;
        std::memset(&rd, 0, sizeof(rd));
        rd.resType = cudaResourceTypeArray;
        rd.res.array.array = s->arr;
        cudaTextureDesc td;
        std::memset(&td, 0, sizeof(td));
        td.addressMode[0] = cudaAddressModeWrap;
        td.addressMode[1] = cudaAddressModeClamp;
        td.filterMode = cudaFilterModeLinear;
        td.readMode = cudaReadModeNormalizedFloat;
        td.normalizedCoords = 1;
        e = cudaCreateTextureObject(&s->tex, &rd, &td, nullptr);
    }
    if (e != cudaSuccess) {
        fail(ctx, RRT_ERR_CUDA, "rrt_sky_create", e);
        rrt_sky_destroy(s);
        return RRT_ERR_CUDA;
    }
    *out = s;
    return RRT_OK;
}

uint64_t rrt_sky_texture(const rrt_sky* sky) { return sky ? (uint64_t)sky->tex : 0; }

void rrt_sky_destroy(rrt_sky* s) {
    if (!s) return;
    DevGuard g(s->device);
    if (s->tex) cudaDestroyTextureObject(s->tex);
    if (s->arr) cudaFreeArray(s->arr);
    delete s;
}

int rrt_band_rows(const rrt_band* band, int h) {
    if (h <= 0) return 0;
    if (!band) return h;
    if (band->nranks <= 0 || band->group <= 0 || band->rank < 0 || band->rank >= band->nranks) return RRT_ERR_BAD_ARG;
    const int ngroups = (h + band->group - 1) / band->group;
    int rows = 0;
    for (int g = band->rank; g < ngroups; g += band->nranks) {
        int y0 = g * band->group, y1 = y0 + band->group;
        if (y1 > h) y1 = h;
        rows += y1 - y0;
    }
    return rows;
}

}  // extern "C"

// ---- launch geometry -----------------------------------------------------------------------------------------------
// Resident CTAs per SM of a kernel: a property of (kernel, device), asked for once per context, not per frame.
// max_shared: the carve-out stays at the shared-memory end although the persistent kernels declare no shared memory:
// every resident CTA still reserves 1 KB of it, and with one-warp CTAs (24-32 per SM) a small carve-out caps residency
// -- measured with cudaSharedmemCarveoutMaxL1: 4K C0 73.3 -> 80.7 ms, C3 133 -> 164 ms.  Negative: the error code.
// ctx->mu held, ctx->device current.
static int resident_per_sm(rrt_context* ctx, const void* kern, int block, bool max_shared) {
    for (const auto& k : ctx->resident)
        if (k.first == kern) return k.second;
    if (max_shared) RRT_CU(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    int per_sm = 0;
    RRT_CU(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, block, 0));
    per_sm = std::max(per_sm, 1);
    ctx->resident.push_back({kern, per_sm});
    return per_sm;
}

// The grid of a persistent launch of `kern`, at most `cap` CTAs.  A persistent launch normally fills every resident-CTA
// slot.  When the caller keeps n frames in flight, each launch takes 1/n of the slots so that the n kernels run side by
// side from the start: a launch then lasts n times longer than its critical path (one tile of disk-plane rays, ~17 ms at
// 4K) needs, instead of ending in a drain with most SMs idle (rrt_set_frames_in_flight).  Negative: the error code.
static long long persistent_grid(rrt_context* ctx, const void* kern, int block, bool max_shared, long long cap) {
    const int per_sm = resident_per_sm(ctx, kern, block, max_shared);
    if (per_sm < 0) return per_sm;
    return std::min(((long long)ctx->sm_count * per_sm + ctx->frames_in_flight - 1) / ctx->frames_in_flight, cap);
}

// ---- split pipeline: host side (csrc/rrt_split.cuh) ---------------------------------------------------------------
// Slots of a sample pool for one frame, at most max_bytes: ~128 samples per pixel before a frame is cut into passes, plus
// what the tracing warps hold in reserve: each takes the rows its tile could need in the worst case (max_steps + 1 rows of
// 1 KiB per ray of a thread) before it traces it.
static size_t pool_slots(size_t max_bytes, long long local_pixels, long long grid_trace, int rows_per_tile) {
    size_t want_bytes = (size_t)local_pixels * 4096 + (size_t)grid_trace * ((size_t)rows_per_tile + 256) * 1024;
    if (want_bytes < (64ull << 20)) want_bytes = 64ull << 20;
    if (want_bytes > max_bytes) want_bytes = max_bytes;
    size_t want_slots = want_bytes / kSlotBytes;
    if (want_slots > 0xfff00000ull) want_slots = 0xfff00000ull;   // slot indices are 32-bit
    if (want_slots < 1024) want_slots = 1024;
    return want_slots;
}

// The pool this stream renders through: its own if it has one, else a free one, else the least recently used one
// (stream-ordered behind that pool's last frame).  (Re)allocated when the frame needs more than it holds.  Returns null,
// with no error set, when the memory is not there: the caller renders fused.
static rrt_context::SamplePool* acquire_pool(rrt_context* ctx, cudaStream_t st, long long local_pixels, unsigned ntiles, long long grid_trace, int rows_per_tile) {
    rrt_context::SamplePool* pl = nullptr;
    for (auto& c : ctx->pools)
        if (c.in_use && c.stream == st) pl = &c;
    if (!pl)
        for (auto& c : ctx->pools)
            if (!c.in_use && !pl) pl = &c;
    if (!pl) {
        for (auto& c : ctx->pools)
            if (!pl || c.last_use < pl->last_use) pl = &c;
        if (pl->done && cudaStreamWaitEvent(st, pl->done, 0) != cudaSuccess) return nullptr;
    }
    const size_t want_slots = pool_slots(ctx->pool_bytes_max, local_pixels, grid_trace, rows_per_tile);
    const bool fresh = !pl->in_use;
    const size_t max_slots = ctx->pool_bytes_max / kSlotBytes;
    const bool resize = pl->cap_slots < want_slots || pl->cap_slots > (max_slots > want_slots ? max_slots : want_slots);   // grows; shrinks only below a lowered limit
    const size_t want_work = want_slots / kMediaBatch + ntiles + 64;   // every queued tile adds at most total / batch + 1 items
    if (resize || pl->desc_cap < ntiles || pl->work_cap < want_work || !pl->d_ctrl) {
        if (pl->done) cudaEventSynchronize(pl->done);
        if (resize) {
            if (pl->d_slots) cudaFree(pl->d_slots);
            pl->d_slots = nullptr; pl->cap_slots = 0;
            if (cudaMalloc(&pl->d_slots, (want_slots + kPoolPadSlots) * kSlotBytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
            pl->cap_slots = want_slots;
        }
        if (pl->desc_cap < ntiles) {
            if (pl->d_desc) cudaFree(pl->d_desc);
            pl->d_desc = nullptr; pl->desc_cap = 0;
            if (cudaMalloc(&pl->d_desc, (size_t)ntiles * sizeof(rrtk::TileDesc)) != cudaSuccess) { cudaGetLastError(); return nullptr; }
            pl->desc_cap = ntiles;
        }
        if (pl->work_cap < want_work) {
            if (pl->d_work) cudaFree(pl->d_work);
            pl->d_work = nullptr; pl->work_cap = 0;
            if (cudaMalloc(&pl->d_work, want_work * sizeof(rrtk::WorkItem)) != cudaSuccess) { cudaGetLastError(); return nullptr; }
            pl->work_cap = want_work;
        }
        if (!pl->d_ctrl) {
            if (cudaMalloc(&pl->d_ctrl, kCtrlBytes) != cudaSuccess || cudaMallocHost(&pl->h_stats, 8 * sizeof(unsigned)) != cudaSuccess ||
                cudaEventCreateWithFlags(&pl->done, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return nullptr; }
            std::memset(pl->h_stats, 0, 8 * sizeof(unsigned));
        }
    }
    if (fresh || pl->stream != st) std::memset(pl->h_stats, 0, 8 * sizeof(unsigned));   // another stream's history says nothing
    pl->in_use = true;
    pl->stream = st;
    pl->last_use = ++ctx->pool_clock;
    return pl;
}

// The pass arguments every split pass over a pool of cap_slots slots shares (pass, control block and redo lists are the caller's).
static rrtk::SplitArgs split_args(uint4* slots, size_t cap_slots, rrtk::TileDesc* desc, rrtk::WorkItem* work, size_t work_cap, bool packed_trace,
                                  int max_steps, long long grid_trace) {
    rrtk::SplitArgs S;
    std::memset(&S, 0, sizeof(S));
    S.slots = slots;
    S.capacity = (unsigned)cap_slots;
    // rows per chunk: as many as leave every tracing warp a few chunks, and few enough chunks per tile for a TileDesc
    unsigned rows = 128;
    const unsigned rows_min = (unsigned)(((packed_trace ? 2 : 1) * (max_steps + 1) + 1 + rrtk::kDescChunks - 3) / (rrtk::kDescChunks - 2));
    while (rows > 8 && rows / 2 >= rows_min && (unsigned long long)rows * 32ull * 8ull * (unsigned long long)grid_trace > cap_slots) rows >>= 1;
    S.chunk_rows = rows;
    S.chunk_shift = 0;
    while ((1u << S.chunk_shift) < rows) ++S.chunk_shift;
    S.high_water = 0xffffffffu;   // a warp takes its tile's worst-case rows before tracing it: a pass simply ends when the pool is used up
    S.desc = desc;
    S.work = work;
    S.work_cap = (unsigned)(work_cap > 0xffffffffull ? 0xffffffffull : work_cap);
    S.redo_cap = kRedoCap;
    S.tile16 = packed_trace ? 1u : 0u;
    return S;
}

// The split pipeline's kernels for a launch, as rrt_render picks them, and the tracer's persistent grid.
struct TracePlan {
    const rrtk::SplitKernels* sk;                         // the kernels of the launch's rounding contract
    bool packed;                                          // two rays per thread in packed f32x2 registers (FMAD contract)
    void (*trace)(const FrameArgs, const rrtk::SplitArgs, const rrtk::LensArgs);
    void (*sweep)(const FrameArgs, const rrtk::SplitArgs, const rrtk::LensArgs);
    long long grid;                                       // of the tracer, already divided by the frames in flight
    unsigned ntiles;                                      // tickets of the launch: 16x4 tiles (packed) or 8x4 tiles
    unsigned ngroups;                                     // groups of 32 rays a pass can queue
    int rows_per_tile;                                    // worst-case sample rows of one tile, exit states included
};
// Whether a launch with these parameters can go through the split pipeline: a tile's rows must fit a TileDesc.
static bool split_fits(const rrt_params* prm) { return prm->max_steps + 2 <= 128 * (rrtk::kDescChunks - 2); }
// lens: the ray source of the LENS variants (rrt_render: kRaysPinhole, rrt_render_dof: kRaysLens, rrt_render_pano: kRaysPano).
static int plan_trace(rrt_context* ctx, const rrt_params& prm, int w, int local_rows, int lens, TracePlan* t) {
    const bool spin = prm.spin_a != 0.0f;
    t->sk = (prm.flags & RRT_FLAG_FMAD) ? rrtk::rrt_split_kernels_fmad() : rrtk::rrt_split_kernels_strict();
    // the tracer: two rays per thread in packed f32x2 registers where that kernel exists (FMAD contract), else one per thread
    t->packed = t->sk->trace_packed[0][0] != nullptr && ctx->trace_choice != 1 && 2ll * (prm.max_steps + 1) + 2 <= 128ll * (rrtk::kDescChunks - 2);
    t->trace = (t->packed ? t->sk->trace_packed : t->sk->trace)[lens][spin];
    t->sweep = t->sk->sweep[lens][spin];
    const unsigned ntiles8 = (unsigned)(((w + kRTileW - 1) / kRTileW) * ((local_rows + kRTileH - 1) / kRTileH));
    const unsigned ntiles16 = (unsigned)(((w + kTile16W - 1) / kTile16W) * ((local_rows + kTile16H - 1) / kTile16H));
    t->ntiles = t->packed ? ntiles16 : ntiles8;
    t->ngroups = t->packed ? 2 * ntiles16 : ntiles8;
    t->grid = persistent_grid(ctx, (const void*)t->trace, kRenderBlock, true, std::min<long long>(t->ntiles, kRedoCap));
    t->rows_per_tile = (t->packed ? 2 : 1) * (prm.max_steps + 1) + 1;
    return t->grid < 0 ? (int)t->grid : RRT_OK;
}

// Everything a render kernel reads about the frame except the planes, counters, ticket and tile log.
static FrameArgs frame_args(const rrt_params& prm, const rrt_camera& cam, const rrt_effects& fx, uint64_t sky_texture, float time, int w,
                            int h, const rrt_band& b, int local_rows, int out_layout, void* d_out) {
    FrameArgs A;
    std::memset(&A, 0, sizeof(A));
    A.C = make_consts(prm);
    A.cam = cam;
    A.fx = fx;
    A.time = time;
    A.w = w;
    A.h = h;
    A.band_rank = b.rank;
    A.band_nranks = b.nranks;
    A.band_group = b.group;
    A.local_rows = local_rows;
    A.out_layout = out_layout;
    A.out = (uchar4*)d_out;
    A.sky = (cudaTextureObject_t)sky_texture;
    return A;
}

// The closing sweep of a split frame: the fused code over the tiles its passes left.  The caller checks the launch.
static int launch_sweep(rrt_context* ctx, const TracePlan& tp, const FrameArgs& A, const rrtk::SplitArgs& S, const rrtk::LensArgs& L,
                        cudaStream_t st) {
    const long long grid = persistent_grid(ctx, (const void*)tp.sweep, kRenderBlock, true, tp.ntiles);
    if (grid < 0) return (int)grid;
    tp.sweep<<<(unsigned)grid, kRenderBlock, 0, st>>>(A, S, L);
    return RRT_OK;
}

// One frame through trace / media / fold passes and the closing sweep.  A camera table (rrt_render_dof) or panorama table
// (rrt_render_pano) in L goes with the LENS tracers of the plan: the passes, the redo list and the sweep re-create every ray
// from it.
static int render_split(rrt_context* ctx, const FrameArgs& A, const rrtk::LensArgs& L, const TracePlan& tp, cudaStream_t st,
                        rrt_context::SamplePool* pl) {
    // passes to enqueue: what the last completed frame on this pool needed (the sweep renders whatever a wrong guess leaves)
    const unsigned* hs = pl->h_stats;   // [0] passes that took tiles [1] tiles swept [2] tiles taken by passes [3] passes enqueued [4] ntiles
    int passes = ctx->passes_hint;
    if (hs[3] != 0u) {
        if (hs[1] == 0u) passes = (int)hs[0];
        else passes = (int)(((unsigned long long)hs[3] * hs[4] + hs[2]) / (hs[2] ? hs[2] : 1u)) + 1;
        ctx->passes_hint = passes < 1 ? 1 : passes;
    }
    if (passes < 1) passes = 1;
    if (passes > ctx->max_passes) passes = ctx->max_passes;

    rrtk::SplitArgs S = split_args(pl->d_slots, pl->cap_slots, pl->d_desc, pl->d_work, pl->work_cap, tp.packed, A.C.max_steps, tp.grid);
    rrtk::PassCtrl* pcs = (rrtk::PassCtrl*)pl->d_ctrl;
    S.stats = (unsigned*)(pl->d_ctrl + sizeof(rrtk::PassCtrl) * (kMaxPasses + 1));
    unsigned* redo = (unsigned*)(pl->d_ctrl + kCtrlHead);

    RRT_CU(ctx, cudaMemsetAsync(pl->d_ctrl, 0, kCtrlHead, st));
    const int per_sm_media = resident_per_sm(ctx, (const void*)tp.sk->media, kMediaBlock, true);
    if (per_sm_media < 0) return per_sm_media;
    const int per_sm_fold = resident_per_sm(ctx, (const void*)tp.sk->fold, 128, false);
    if (per_sm_fold < 0) return per_sm_fold;
    for (int p = 0; p < passes; ++p) {
        S.pass = (unsigned)p;
        S.pc = pcs + p;
        S.pc_prev = p ? pcs + (p - 1) : nullptr;
        S.redo_in = p ? redo + (size_t)(p - 1) * kRedoCap : nullptr;
        S.redo_out = redo + (size_t)p * kRedoCap;
        tp.trace<<<(unsigned)tp.grid, kRenderBlock, 0, st>>>(A, S, L);
        tp.sk->media<<<(unsigned)(ctx->sm_count * per_sm_media), kMediaBlock, 0, st>>>(A, S);
        tp.sk->fold<<<(unsigned)(ctx->sm_count * per_sm_fold), 128, 0, st>>>(A, S);
    }
    S.pass = (unsigned)passes;
    S.pc = pcs + passes;
    S.pc_prev = pcs + (passes - 1);
    S.redo_in = redo + (size_t)(passes - 1) * kRedoCap;
    S.redo_out = redo + (size_t)passes * kRedoCap;
    if (int rc = launch_sweep(ctx, tp, A, S, L, st)) return rc;
    RRT_CU(ctx, cudaGetLastError());
    ctx->launches += 3ull * (unsigned)passes + 1ull;
    RRT_CU(ctx, cudaMemcpyAsync(pl->h_stats, S.stats, 8 * sizeof(unsigned), cudaMemcpyDeviceToHost, st));
    RRT_CU(ctx, cudaEventRecord(pl->done, st));
    return RRT_OK;
}

// ---- argument checks: every entry point runs them before it takes ctx->mu or enqueues anything ---------------------
// A destination: a known layout and at least one of the uchar4 frame and the hdr plane (or planes).
static bool outputs_ok(int out_layout, const void* d_out, const void* hdr) {
    return (out_layout == RRT_OUT_FRAME || out_layout == RRT_OUT_PACKED) && (d_out || hdr);
}

// The band of a call on a w x h frame: `band`, or the whole frame {0, 1, 1}, into *b and its rows into *local_rows.
// Traced with ss x ss rays per pixel it is the band {rank, nranks, ss*group} of the ss*w x ss*h frame, which must stay
// within rrt_render's 2^30 rays.
static int band_of(rrt_context* ctx, const std::string& what, const rrt_band* band, int w, int h, int ss, rrt_band* b, int* local_rows) {
    *b = band ? *band : rrt_band{0, 1, 1};
    const int rows = rrt_band_rows(b, h);
    if (rows < 0 || (long long)ss * b->group > INT_MAX) return fail(ctx, RRT_ERR_BAD_ARG, what + ": bad band");
    if ((long long)ss * ss * w * rows > (1ll << 30))
        return fail(ctx, RRT_ERR_BAD_ARG, what + (ss == 1 ? ": band larger than 2^30 pixels" : ": band larger than 2^30 sub-samples"));
    *local_rows = rows;
    return RRT_OK;
}

// A supersampling factor and the w x h frame it resolves to, whose ss*w x ss*h trace must have int sizes.
static bool ss_ok(int ss, int w, int h) {
    return ss >= 1 && ss <= 8 && w > 0 && h > 0 && (long long)ss * w <= INT_MAX && (long long)ss * h <= INT_MAX;
}

// What rrt_resolve_time, rrt_render_mb and rrt_capture_render_mb check: n, the frame, the band and a stack of n
// full-frame planes that fits the address space.
static int check_mb(rrt_context* ctx, const std::string& what, int n, int w, int h, const rrt_band* band, rrt_band* b, int* local_rows) {
    if (n < 1 || n > 64 || w <= 0 || h <= 0) return fail(ctx, RRT_ERR_BAD_ARG, what + ": bad argument");
    if (int rc = band_of(ctx, what, band, w, h, 1, b, local_rows)) return rc;
    if ((unsigned long long)w * h > SIZE_MAX / 16 / (unsigned)n)
        return fail(ctx, RRT_ERR_BAD_ARG, what + ": sub-frame stack larger than the address space");
    return RRT_OK;
}

// Whether float4 ranges [src, src + src_n) and [dst, dst + dst_n) share a byte.
static bool f4_overlap(const void* src, unsigned long long src_n, const void* dst, unsigned long long dst_n) {
    const uintptr_t a = (uintptr_t)src, b = (uintptr_t)dst;
    return b >= a ? (b - a) / 16 < src_n : (a - b) / 16 < dst_n;
}

// ---- bodies: arguments checked, ctx->mu held, ctx->device current ---------------------------------------------------
// rrt_render's body.  L.cams: null, or a DEVICE table of L.ss * L.ss cameras (rrt_render_dof) -- then the kRaysLens variant
// of the chosen kernel starts pixel (x, y)'s ray from L.cams[(y % L.ss) * L.ss + x % L.ss] and `cam` is not read by any
// kernel.  L.pano: null, or the DEVICE table of a w x h panorama (rrt_render_pano) -- then the kRaysPano variant starts
// every ray at cam.pos in the direction of pano_dir.  Launch choice, pipeline, counters and launch count are rrt_render's
// in every case.
static int render_frame(rrt_context* ctx, const rrt_params& prm, const rrt_camera& cam, const rrt_effects& fx, uint64_t sky_texture,
                        float time, int w, int h, const rrt_band& b, int local_rows, void* d_out, int out_layout, const rrt_planes* planes,
                        cudaStream_t st, const rrtk::LensArgs& L) {
    FrameArgs A = frame_args(prm, cam, fx, sky_texture, time, w, h, b, local_rows, out_layout, d_out);
    if (planes) A.planes = *planes;
    A.counters = ctx->d_counters;
    A.tile_log = ctx->tile_log;
    A.tile_log_cap = ctx->tile_log_cap;
    A.ticket = ctx->d_tickets + (ctx->ticket_next++ % kTicketRing);
    RRT_CU(ctx, cudaMemsetAsync(A.ticket, 0, sizeof(unsigned), st));

    const bool spin = prm.spin_a != 0.0f;
    const bool media = (prm.flags & (RRT_FLAG_DISK | RRT_FLAG_DUST)) != 0;
    const bool fmad = (prm.flags & RRT_FLAG_FMAD) != 0;
    const int lens = L.pano ? kRaysPano : (L.cams ? kRaysLens : kRaysPinhole);
    // A launch with a medium goes through the split pipeline (csrc/rrt_split.cuh) unless the caller pinned the fused
    // kernel, the tile log is selected, or the pool cannot be allocated.
    if (media && ctx->pipeline != RRT_PIPELINE_FUSED && (!ctx->tile_log || ctx->pipeline == RRT_PIPELINE_SPLIT) && split_fits(&prm)) {
        TracePlan tp;
        if (int rc = plan_trace(ctx, prm, w, local_rows, lens, &tp)) return rc;
        if (rrt_context::SamplePool* pl = acquire_pool(ctx, st, (long long)w * local_rows, tp.ngroups, tp.grid, tp.rows_per_tile))
            return render_split(ctx, A, L, tp, st, pl);
        if (ctx->pipeline == RRT_PIPELINE_SPLIT) return fail(ctx, RRT_ERR_NOMEM, "rrt_render: no memory for the sample pool of the split pipeline");
    }
    const rrtk::KernelSet* ks = kset(&prm);
    void (*kern)(const FrameArgs, const rrtk::LensArgs) = ks->render[lens][spin][media];
    long long rays_per_block = kRenderBlock;
    if (fmad && !media && !ctx->scalar_kernel) {
        kern = ks->render_packed[lens][spin];
        rays_per_block = 64;
    }
    const long long grid = persistent_grid(ctx, (const void*)kern, kRenderBlock, true, ((long long)w * local_rows + rays_per_block - 1) / rays_per_block);
    if (grid < 0) return (int)grid;
    kern<<<(unsigned)grid, kRenderBlock, 0, st>>>(A, L);
    RRT_CU(ctx, cudaGetLastError());
    ctx->launches += 1;
    return RRT_OK;
}

// The launch of rrt_resolve and rrt_resolve_time: resolve_kernel over the band's rows of the w x h frame, n planes of
// ss*w x ss*h from `src`, one plane_stride (float4) apart.
static int launch_resolve(rrt_context* ctx, const rrt_params& prm, const rrt_effects& fx, int ss, int n, int w, int h, const rrt_band& b,
                          int local_rows, const float* src, size_t plane_stride, void* d_out, int out_layout, float* hdr_out, cudaStream_t st) {
    // no camera, sky, counters, ticket or tile log: nothing is traced or sampled; the post step reads exposure only
    FrameArgs A = frame_args(prm, rrt_camera{}, fx, 0, 0.0f, w, h, b, local_rows, out_layout, d_out);
    A.planes.hdr = hdr_out;
    const long long npix = (long long)w * local_rows;
    kset(&prm)->resolve<<<(unsigned)((npix + kResolveBlock - 1) / kResolveBlock), kResolveBlock, 0, st>>>(
        A, (const float4*)src, ss, n, plane_stride);
    RRT_CU(ctx, cudaGetLastError());
    ctx->launches += 1;
    return RRT_OK;
}

// body(block) with a stream-ordered block of `bytes` from the context's scratch pool (created on first use), which keeps
// freed blocks for the next frame instead of returning them to the device: rrt_render_ss's supersampled plane, the
// sub-frame stacks of rrt_render_mb / rrt_capture_render_mb.  The block goes back to the pool behind whatever body
// enqueued; the first error wins.
template <typename Body>
static int with_scratch(rrt_context* ctx, const std::string& what, const char* block_name, size_t bytes, cudaStream_t st, Body body) {
    if (!ctx->ss_pool) {
        cudaMemPoolProps props;
        std::memset(&props, 0, sizeof(props));
        props.allocType = cudaMemAllocationTypePinned;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = ctx->device;
        RRT_CU(ctx, cudaMemPoolCreate(&ctx->ss_pool, &props));
        uint64_t keep = UINT64_MAX;   // hold freed blocks: the next frame of a sequence reuses them without a new allocation
        RRT_CU(ctx, cudaMemPoolSetAttribute(ctx->ss_pool, cudaMemPoolAttrReleaseThreshold, &keep));
    }
    float* block = nullptr;
    if (cudaMallocFromPoolAsync((void**)&block, bytes, ctx->ss_pool, st) != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, RRT_ERR_NOMEM, what + ": no memory for the " + block_name);
    }
    const int rc = body(block);
    const cudaError_t e = cudaFreeAsync(block, st);   // stream-ordered: the block goes back once the last kernel has read it
    if (rc == RRT_OK && e != cudaSuccess) return fail(ctx, RRT_ERR_CUDA, what + ": cudaFreeAsync", e);
    return rc;
}

extern "C" {

int rrt_render(rrt_context* ctx, const rrt_params* prm, const rrt_camera* cam, const rrt_effects* fx, uint64_t sky_texture,
               float time, int w, int h, const rrt_band* band, void* d_out, int out_layout, const rrt_planes* planes,
               void* stream) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!prm || !cam || !fx || w <= 0 || h <= 0 || sky_texture == 0 || prm->max_steps < 0 || !outputs_ok(out_layout, d_out, planes))
        return fail(ctx, RRT_ERR_BAD_ARG, "rrt_render: bad argument");
    rrt_band b;
    int local_rows = 0;
    if (int rc = band_of(ctx, "rrt_render", band, w, h, 1, &b, &local_rows)) return rc;
    if (local_rows == 0) return RRT_OK;

    std::lock_guard<std::mutex> lk(ctx->mu);
    DevGuard g(ctx->device);
    return render_frame(ctx, *prm, *cam, *fx, sky_texture, time, w, h, b, local_rows, d_out, out_layout, planes, (cudaStream_t)stream,
                        rrtk::LensArgs{});
}

int rrt_shade(rrt_context* ctx, const rrt_params* prm, const rrt_effects* fx, uint64_t sky_texture, int w, int h,
              const rrt_band* band, const rrt_planes* traced, void* d_out, int out_layout, float* hdr_out, void* stream) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!prm || !fx || w <= 0 || h <= 0 || sky_texture == 0 || !traced || !traced->vel || !traced->emis || !traced->hdr || !traced->cls ||
        !outputs_ok(out_layout, d_out, hdr_out))
        return fail(ctx, RRT_ERR_BAD_ARG, "rrt_shade: bad argument");
    rrt_band b;
    int local_rows = 0;
    if (int rc = band_of(ctx, "rrt_shade", band, w, h, 1, &b, &local_rows)) return rc;
    if (local_rows == 0) return RRT_OK;

    std::lock_guard<std::mutex> lk(ctx->mu);
    DevGuard g(ctx->device);
    // no camera, counters, ticket or tile log: nothing is traced; finish_ray_inl reads exposure only
    FrameArgs A = frame_args(*prm, rrt_camera{}, *fx, sky_texture, 0.0f, w, h, b, local_rows, out_layout, d_out);
    A.planes.hdr = hdr_out;
    const long long n = (long long)w * local_rows;
    kset(prm)->shade<<<(unsigned)((n + kShadeBlock - 1) / kShadeBlock), kShadeBlock, 0, (cudaStream_t)stream>>>(A, *traced);
    RRT_CU(ctx, cudaGetLastError());
    ctx->launches += 1;
    return RRT_OK;
}

int rrt_resolve(rrt_context* ctx, const rrt_params* prm, const rrt_effects* fx, int ss, int w, int h, const rrt_band* band,
                const float* hdr_hi, void* d_out, int out_layout, float* hdr_out, void* stream) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!prm || !fx || !hdr_hi || !ss_ok(ss, w, h) || !outputs_ok(out_layout, d_out, hdr_out))
        return fail(ctx, RRT_ERR_BAD_ARG, "rrt_resolve: bad argument");
    rrt_band b;
    int local_rows = 0;
    if (int rc = band_of(ctx, "rrt_resolve", band, w, h, ss, &b, &local_rows)) return rc;
    // the kernel reads hdr_hi while it writes hdr_out: the two must not share a byte
    if (hdr_out && f4_overlap(hdr_hi, (unsigned long long)ss * ss * w * h, hdr_out, (unsigned long long)w * h))
        return fail(ctx, RRT_ERR_BAD_ARG, "rrt_resolve: hdr_out overlaps hdr_hi");
    if (local_rows == 0) return RRT_OK;

    std::lock_guard<std::mutex> lk(ctx->mu);
    DevGuard g(ctx->device);
    return launch_resolve(ctx, *prm, *fx, ss, 1, w, h, b, local_rows, hdr_hi, 0, d_out, out_layout, hdr_out, (cudaStream_t)stream);
}

// rrt_render_ss and rrt_render_dof: the ss*w x ss*h trace into a scratch plane, then rrt_resolve's launch.  cams: null
// (every sub-sample from `cam`), or a HOST table of ss*ss cameras (rrt_render_dof), copied into the same scratch block
// behind the plane.
static int render_ss_frame(rrt_context* ctx, const char* what, const rrt_params* prm, const rrt_camera* cam, const rrt_camera* cams,
                           const rrt_effects* fx, uint64_t sky_texture, float time, int w, int h, int ss, const rrt_band* band,
                           void* d_out, int out_layout, float* hdr_out, void* stream) {
    const std::string m = what;
    if (!prm || !cam || !fx || sky_texture == 0 || prm->max_steps < 0 || !ss_ok(ss, w, h) || !outputs_ok(out_layout, d_out, hdr_out))
        return fail(ctx, RRT_ERR_BAD_ARG, m + ": bad argument");
    rrt_band b;
    int local_rows = 0;
    if (int rc = band_of(ctx, m, band, w, h, ss, &b, &local_rows)) return rc;
    bool cams_near = true;   // trace_ray's fast_ok for every camera of the table: |pos|^2 < 1e8
    if (cams)
        for (int k = 0; k < ss * ss; ++k) {
            const float* f = cams[k].pos;   // pos, forward, right, up: 12 consecutive floats
            for (int c = 0; c < 12; ++c)
                if (!std::isfinite(f[c])) return fail(ctx, RRT_ERR_BAD_ARG, m + ": non-finite camera field");
            cams_near = cams_near && (double)f[0] * f[0] + (double)f[1] * f[1] + (double)f[2] * f[2] < 1.0e8;
        }
    if (local_rows == 0) return RRT_OK;
    const unsigned long long n_hi = (unsigned long long)ss * ss * w * h;   // full-frame indexed like every plane of this ABI
    const size_t cam_bytes = cams ? sizeof(rrt_camera) * ss * ss : 0;
    if (n_hi > (SIZE_MAX - cam_bytes) / 16) return fail(ctx, RRT_ERR_NOMEM, m + ": supersampled hdr plane larger than the address space");

    std::lock_guard<std::mutex> lk(ctx->mu);
    DevGuard g(ctx->device);
    const cudaStream_t st = (cudaStream_t)stream;
    return with_scratch(ctx, m, "supersampled hdr plane", (size_t)16 * n_hi + cam_bytes, st, [&](float* hi) {
        rrtk::LensArgs L = {};
        if (cams) {
            // The table goes behind the plane (16-byte aligned).  The copy reads a pageable copy of the caller's table, which
            // the runtime stages before cudaMemcpyAsync returns: the caller may reuse its table at once, also when it is pinned.
            rrt_camera* d_cams = (rrt_camera*)(hi + 4 * n_hi);
            const std::vector<rrt_camera> staged(cams, cams + ss * ss);
            const cudaError_t e = cudaMemcpyAsync(d_cams, staged.data(), cam_bytes, cudaMemcpyHostToDevice, st);
            if (e != cudaSuccess) return fail(ctx, RRT_ERR_CUDA, m + ": copy of the camera table", e);
            L = {d_cams, ss, cams_near ? 1 : 0};
        }
        rrt_planes pl;
        std::memset(&pl, 0, sizeof(pl));
        pl.hdr = hi;
        // output group y / g is trace group (ss*y + j) / (ss*g): the band traces exactly the ss sub-rows of each of its rows
        const rrt_band tb = {b.rank, b.nranks, ss * b.group};
        if (int rc = render_frame(ctx, *prm, *cam, *fx, sky_texture, time, ss * w, ss * h, tb, ss * local_rows, nullptr, RRT_OUT_FRAME, &pl, st, L))
            return rc;
        return launch_resolve(ctx, *prm, *fx, ss, 1, w, h, b, local_rows, hi, 0, d_out, out_layout, hdr_out, st);
    });
}

int rrt_render_ss(rrt_context* ctx, const rrt_params* prm, const rrt_camera* cam, const rrt_effects* fx, uint64_t sky_texture,
                  float time, int w, int h, int ss, const rrt_band* band, void* d_out, int out_layout, float* hdr_out,
                  void* stream) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    return render_ss_frame(ctx, "rrt_render_ss", prm, cam, nullptr, fx, sky_texture, time, w, h, ss, band, d_out, out_layout, hdr_out,
                           stream);
}

int rrt_render_dof(rrt_context* ctx, const rrt_params* prm, const rrt_camera* cams, const rrt_effects* fx, uint64_t sky_texture,
                   float time, int w, int h, int ss, const rrt_band* band, void* d_out, int out_layout, float* hdr_out,
                   void* stream) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!cams) return fail(ctx, RRT_ERR_BAD_ARG, "rrt_render_dof: bad argument");
    return render_ss_frame(ctx, "rrt_render_dof", prm, cams, cams, fx, sky_texture, time, w, h, ss, band, d_out, out_layout, hdr_out,
                           stream);
}

int rrt_render_pano(rrt_context* ctx, const rrt_params* prm, const rrt_camera* cam, const rrt_effects* fx, uint64_t sky_texture,
                    float time, int w, int h, int ss, const rrt_band* band, void* d_out, int out_layout, const rrt_planes* planes,
                    void* stream) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    const std::string m = "rrt_render_pano";
    // ss > 1 offers the averaged hdr plane only, like rrt_render_ss
    const bool hdr_only = !planes || (!planes->dir && !planes->emis && !planes->pos && !planes->vel && !planes->cls && !planes->steps);
    if (!prm || !cam || !fx || sky_texture == 0 || prm->max_steps < 0 || !ss_ok(ss, w, h) || fx->use_lens != 0 ||
        !outputs_ok(out_layout, d_out, ss == 1 ? (const void*)planes : (const void*)(planes ? planes->hdr : nullptr)) ||
        (ss > 1 && !hdr_only))
        return fail(ctx, RRT_ERR_BAD_ARG, m + ": bad argument");
    rrt_band b;
    int local_rows = 0;
    if (int rc = band_of(ctx, m, band, w, h, ss, &b, &local_rows)) return rc;
    if (local_rows == 0) return RRT_OK;
    const int W = ss * w, H = ss * h;   // the traced panorama
    const unsigned long long n_hi = ss == 1 ? 0ull : (unsigned long long)W * H;   // the supersampled plane, full-frame indexed
    const size_t tab_bytes = sizeof(float2) * ((size_t)W + H);
    if (n_hi > (SIZE_MAX - tab_bytes) / 16) return fail(ctx, RRT_ERR_NOMEM, m + ": supersampled hdr plane larger than the address space");
    std::vector<float2> tab((size_t)W + H);   // pageable: staged by cudaMemcpyAsync before it returns
    rrtk::pano_table(W, H, (float*)tab.data());

    std::lock_guard<std::mutex> lk(ctx->mu);
    DevGuard g(ctx->device);
    const cudaStream_t st = (cudaStream_t)stream;
    return with_scratch(ctx, m, ss == 1 ? "panorama table" : "supersampled hdr plane", (size_t)16 * n_hi + tab_bytes, st, [&](float* blk) {
        float2* d_tab = (float2*)(blk + 4 * n_hi);   // behind the plane when there is one
        const cudaError_t e = cudaMemcpyAsync(d_tab, tab.data(), tab_bytes, cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) return fail(ctx, RRT_ERR_CUDA, m + ": copy of the panorama table", e);
        rrtk::LensArgs L = {};
        L.pano = d_tab;
        if (ss == 1)
            return render_frame(ctx, *prm, *cam, *fx, sky_texture, time, w, h, b, local_rows, d_out, out_layout, planes, st, L);
        rrt_planes pl;
        std::memset(&pl, 0, sizeof(pl));
        pl.hdr = blk;
        const rrt_band tb = {b.rank, b.nranks, ss * b.group};   // as in render_ss_frame: the ss sub-rows of each of the band's rows
        if (int rc = render_frame(ctx, *prm, *cam, *fx, sky_texture, time, W, H, tb, ss * local_rows, nullptr, RRT_OUT_FRAME, &pl, st, L))
            return rc;
        return launch_resolve(ctx, *prm, *fx, ss, 1, w, h, b, local_rows, blk, 0, d_out, out_layout, planes ? planes->hdr : nullptr, st);
    });
}

int rrt_resolve_time(rrt_context* ctx, const rrt_params* prm, const rrt_effects* fx, int n, int w, int h, const rrt_band* band,
                     const float* hdr_stack, void* d_out, int out_layout, float* hdr_out, void* stream) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!prm || !fx || !hdr_stack || !outputs_ok(out_layout, d_out, hdr_out))
        return fail(ctx, RRT_ERR_BAD_ARG, "rrt_resolve_time: bad argument");
    rrt_band b;
    int local_rows = 0;
    if (int rc = check_mb(ctx, "rrt_resolve_time", n, w, h, band, &b, &local_rows)) return rc;
    const unsigned long long plane = (unsigned long long)w * h;
    if (hdr_out && f4_overlap(hdr_stack, (unsigned long long)n * plane, hdr_out, plane))
        return fail(ctx, RRT_ERR_BAD_ARG, "rrt_resolve_time: hdr_out overlaps hdr_stack");
    if (local_rows == 0) return RRT_OK;

    std::lock_guard<std::mutex> lk(ctx->mu);
    DevGuard g(ctx->device);
    return launch_resolve(ctx, *prm, *fx, 1, n, w, h, b, local_rows, hdr_stack, (size_t)plane, d_out, out_layout, hdr_out,
                          (cudaStream_t)stream);
}

int rrt_render_mb(rrt_context* ctx, const rrt_params* prm, const rrt_camera* cams, const rrt_effects* fx, uint64_t sky_texture,
                  const float* times, int n, int w, int h, const rrt_band* band, void* d_out, int out_layout, float* hdr_out,
                  void* stream) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!prm || !cams || !fx || !times || sky_texture == 0 || prm->max_steps < 0 || !outputs_ok(out_layout, d_out, hdr_out))
        return fail(ctx, RRT_ERR_BAD_ARG, "rrt_render_mb: bad argument");
    rrt_band b;
    int local_rows = 0;
    if (int rc = check_mb(ctx, "rrt_render_mb", n, w, h, band, &b, &local_rows)) return rc;
    if (local_rows == 0) return RRT_OK;

    std::lock_guard<std::mutex> lk(ctx->mu);
    DevGuard g(ctx->device);
    const cudaStream_t st = (cudaStream_t)stream;
    const size_t plane = (size_t)w * h;   // full-frame indexed like every plane of this ABI, so full-frame sized even for a band
    return with_scratch(ctx, "rrt_render_mb", "sub-frame stack", 16 * n * plane, st, [&](float* stack) {
        rrt_planes pl;
        std::memset(&pl, 0, sizeof(pl));
        for (int i = 0; i < n; ++i) {
            pl.hdr = stack + 4 * plane * i;
            if (int rc = render_frame(ctx, *prm, cams[i], *fx, sky_texture, times[i], w, h, b, local_rows, nullptr, RRT_OUT_FRAME, &pl, st,
                                      rrtk::LensArgs{}))
                return rc;
        }
        return launch_resolve(ctx, *prm, *fx, 1, n, w, h, b, local_rows, stack, plane, d_out, out_layout, hdr_out, st);
    });
}

}  // extern "C"

// ---- captures (rrt_capture_*): one trace kept for renders at other times -----------------------------------------------
// The trace of a frame with a medium does not read the time: only the densities do, in media_kernel (and in sweep_kernel for
// tiles the pass could not hold).  A capture runs the split pipeline's trace pass once into a pool it owns and keeps what
// media + fold need afterwards; each render then evaluates the kept samples at its own time into a separate results array
// (media_kernel<true>), so the samples survive for the next render.
struct rrt_capture {
    rrt_context* ctx = nullptr;
    rrt_params prm;                   // what the trace used: a render takes prm with its own exposure
    rrt_camera cam;
    rrt_effects fx;
    rrt_band band = {0, 1, 1};
    int w = 0, h = 0, local_rows = 0;
    TracePlan plan;                   // the pass's kernels and tickets: 16x4 tiles (packed tracer) or 8x4 tiles
    unsigned tiles_left = 0;          // tickets the pass did not trace: its redo list + the tickets it never took
    rrtk::SplitArgs S;                // media / fold over what the capture holds; the sweep's pass derives from it
    char* d_ctrl = nullptr;           // PassCtrl[2] (the pass, the sweep) | stats[8] | ticket | ticket after the pass | redo list
    uint4* d_slots = nullptr;         // the used prefix of the pool (samples and exit states)
    uint4* d_results = nullptr;       // {e.rgb, s} per slot of the prefix
    rrtk::TileDesc* d_desc = nullptr;
    rrtk::WorkItem* d_work = nullptr;
    char* d_planes = nullptr;         // vel | emis | hdr (float4) | cls (u8), full frame: the rays the trace finished on the spot
    rrt_planes planes;
    uint64_t info[8] = {};
    cudaEvent_t done = nullptr;       // the last render enqueued
};

namespace {
constexpr size_t kCapStats = 2 * sizeof(rrtk::PassCtrl), kCapTicket = kCapStats + 8 * sizeof(unsigned), kCapRedo = 128;
constexpr size_t kCapCtrlBytes = kCapRedo + sizeof(unsigned) * kRedoCap;
static_assert(kCapTicket + 2 * sizeof(unsigned) <= kCapRedo, "capture control block layout");

void free_capture(rrt_capture* c) {
    DevGuard g(c->ctx->device);
    if (c->done) cudaEventSynchronize(c->done);
    for (void* p : {(void*)c->d_ctrl, (void*)c->d_slots, (void*)c->d_results, (void*)c->d_desc, (void*)c->d_work, (void*)c->d_planes})
        if (p) cudaFree(p);
    if (c->done) cudaEventDestroy(c->done);
    delete c;
}
// The device allocations of a capture under construction, released unless handed over.
struct DevAlloc {
    void* p = nullptr;
    bool get(size_t n) { if (cudaMalloc(&p, n ? n : 1) == cudaSuccess) return true; cudaGetLastError(); p = nullptr; return false; }
    void* take() { void* q = p; p = nullptr; return q; }
    ~DevAlloc() { if (p) cudaFree(p); }
};
}  // namespace

extern "C" {

// a failed CUDA call inside rrt_capture_create releases the partial capture
#define CAP_CU(call)                                                                    \
    do {                                                                                \
        if (cudaError_t e__ = (call)) return bail(RRT_ERR_CUDA, "rrt_capture_create: " #call, e__); \
    } while (0)
int rrt_capture_create(rrt_context* ctx, const rrt_params* prm, const rrt_camera* cam, const rrt_effects* fx, uint64_t sky_texture, int w,
                       int h, const rrt_band* band, size_t max_bytes, void* stream, rrt_capture** out) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!out || !prm || !cam || !fx || w <= 0 || h <= 0 || sky_texture == 0 || prm->max_steps < 0)
        return fail(ctx, RRT_ERR_BAD_ARG, "rrt_capture_create: bad argument");
    *out = nullptr;
    if (!(prm->flags & (RRT_FLAG_DISK | RRT_FLAG_DUST)))
        return fail(ctx, RRT_ERR_BAD_ARG, "rrt_capture_create: no medium (RRT_FLAG_DISK / RRT_FLAG_DUST): nothing depends on the time, re-shade with rrt_shade");
    if (!split_fits(prm)) return fail(ctx, RRT_ERR_BAD_ARG, "rrt_capture_create: max_steps too large for the split pipeline");
    rrt_band b;
    int local_rows = 0;
    if (int rc = band_of(ctx, "rrt_capture_create", band, w, h, 1, &b, &local_rows)) return rc;

    std::lock_guard<std::mutex> lk(ctx->mu);
    DevGuard g(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    rrt_capture* c = new (std::nothrow) rrt_capture();
    if (!c) return fail(ctx, RRT_ERR_NOMEM, "out of host memory");
    c->ctx = ctx;
    c->prm = *prm;
    c->cam = *cam;
    c->fx = *fx;
    c->band = b;
    c->w = w;
    c->h = h;
    c->local_rows = local_rows;
    auto bail = [&](int code, const char* what, cudaError_t e = cudaSuccess) { free_capture(c); return fail(ctx, code, what, e); };
    const size_t npix = (size_t)w * h;
    const size_t plane_bytes = npix * (3 * sizeof(float4) + 1);
    if (cudaEventCreateWithFlags(&c->done, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return bail(RRT_ERR_CUDA, "rrt_capture_create: event"); }
    DevAlloc ctrl, planes;
    if (!ctrl.get(kCapCtrlBytes) || !planes.get(plane_bytes)) return bail(RRT_ERR_NOMEM, "rrt_capture_create: no memory for the capture's planes");
    c->d_ctrl = (char*)ctrl.take();
    c->d_planes = (char*)planes.take();
    std::memset(&c->planes, 0, sizeof(c->planes));
    c->planes.vel = (float*)c->d_planes;
    c->planes.emis = (float*)(c->d_planes + npix * sizeof(float4));
    c->planes.hdr = (float*)(c->d_planes + 2 * npix * sizeof(float4));
    c->planes.cls = (uint8_t*)(c->d_planes + 3 * npix * sizeof(float4));
    CAP_CU(cudaMemsetAsync(c->d_ctrl, 0, kCapRedo, st));
    CAP_CU(cudaMemsetAsync(c->d_planes, 0, plane_bytes, st));   // pixels no kernel of the trace writes read as zeros
    if (local_rows == 0) {
        *out = c;
        return RRT_OK;
    }

    // the pass: rrt_render's tracer and grid, into a pool of this capture's own
    const TracePlan& tp = c->plan;
    if (int rc = plan_trace(ctx, *prm, w, local_rows, false, &c->plan)) {
        free_capture(c);
        return rc;
    }
    size_t cap_slots = pool_slots(ctx->pool_bytes_max, (long long)npix, tp.grid, tp.rows_per_tile);
    if (max_bytes) cap_slots = std::min<size_t>(std::max<size_t>(max_bytes / kSlotBytes, 1024), 0xfff00000ull);
    const size_t work_cap = cap_slots / kMediaBatch + tp.ngroups + 64;   // as acquire_pool sizes it
    DevAlloc pool, desc, work;
    if (!pool.get((cap_slots + kPoolPadSlots) * kSlotBytes) || !desc.get((size_t)tp.ngroups * sizeof(rrtk::TileDesc)) ||
        !work.get(work_cap * sizeof(rrtk::WorkItem)))
        return bail(RRT_ERR_NOMEM, "rrt_capture_create: no memory for the sample pool");
    FrameArgs A = frame_args(*prm, *cam, *fx, sky_texture, 0.0f, w, h, b, local_rows, RRT_OUT_FRAME, nullptr);
    A.planes = c->planes;
    A.counters = ctx->d_counters;
    A.ticket = (unsigned*)(c->d_ctrl + kCapTicket);
    rrtk::SplitArgs S = split_args((uint4*)pool.p, cap_slots, (rrtk::TileDesc*)desc.p, (rrtk::WorkItem*)work.p, work_cap, tp.packed,
                                   prm->max_steps, tp.grid);
    rrtk::PassCtrl* pcs = (rrtk::PassCtrl*)c->d_ctrl;
    S.pc = pcs;
    S.redo_out = (unsigned*)(c->d_ctrl + kCapRedo);
    S.stats = (unsigned*)(c->d_ctrl + kCapStats);
    tp.trace<<<(unsigned)tp.grid, kRenderBlock, 0, st>>>(A, S, rrtk::LensArgs{});
    CAP_CU(cudaGetLastError());
    ctx->launches += 1;
    CAP_CU(cudaMemcpyAsync(c->d_ctrl + kCapTicket + sizeof(unsigned), c->d_ctrl + kCapTicket, sizeof(unsigned), cudaMemcpyDeviceToDevice, st));
    unsigned char head[kCapRedo];
    CAP_CU(cudaMemcpyAsync(head, c->d_ctrl, kCapRedo, cudaMemcpyDeviceToHost, st));
    if (cudaError_t e = cudaStreamSynchronize(st)) return bail(RRT_ERR_CUDA, "rrt_capture_create: trace pass", e);
    rrtk::PassCtrl pc;
    std::memcpy(&pc, head, sizeof(pc));
    unsigned ticket;
    std::memcpy(&ticket, head + kCapTicket, sizeof(ticket));

    // keep the used prefix of the pool, the queued groups and their work items; free the rest (before the results array
    // is allocated: the peak is the pool plus its used prefix)
    const size_t used = std::min<size_t>(pc.cursor, cap_slots), held = used + kPoolPadSlots;
    const size_t n_desc = pc.pend_count, n_work = std::min<size_t>(pc.work_count, work_cap);
    DevAlloc slots, results, desc_held, work_held;
    if (!slots.get(held * kSlotBytes) || !desc_held.get(n_desc * sizeof(rrtk::TileDesc)) || !work_held.get(n_work * sizeof(rrtk::WorkItem)))
        return bail(RRT_ERR_NOMEM, "rrt_capture_create: no memory for the samples");
    CAP_CU(cudaMemcpyAsync(slots.p, pool.p, held * kSlotBytes, cudaMemcpyDeviceToDevice, st));
    if (n_desc) CAP_CU(cudaMemcpyAsync(desc_held.p, desc.p, n_desc * sizeof(rrtk::TileDesc), cudaMemcpyDeviceToDevice, st));
    if (n_work) CAP_CU(cudaMemcpyAsync(work_held.p, work.p, n_work * sizeof(rrtk::WorkItem), cudaMemcpyDeviceToDevice, st));
    uint64_t samples = 0;
    if (n_desc) {   // the `total` field of every queued group: a strided copy
        unsigned* tot = new (std::nothrow) unsigned[n_desc];
        if (!tot) return bail(RRT_ERR_NOMEM, "out of host memory");
        cudaError_t e = cudaMemcpy2DAsync(tot, sizeof(unsigned), (const char*)desc.p + offsetof(rrtk::TileDesc, total), sizeof(rrtk::TileDesc),
                                          sizeof(unsigned), n_desc, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        for (size_t i = 0; e == cudaSuccess && i < n_desc; ++i) samples += tot[i];
        delete[] tot;
        if (e != cudaSuccess) return bail(RRT_ERR_CUDA, "rrt_capture_create: copy of the queued groups", e);
    }
    if (cudaError_t e = cudaStreamSynchronize(st)) return bail(RRT_ERR_CUDA, "rrt_capture_create: copy of the samples", e);
    cudaFree(pool.take());
    if (!results.get(held * sizeof(uint4))) return bail(RRT_ERR_NOMEM, "rrt_capture_create: no memory for the media results");
    c->d_slots = (uint4*)slots.take();
    c->d_results = (uint4*)results.take();
    c->d_desc = (rrtk::TileDesc*)desc_held.take();
    c->d_work = (rrtk::WorkItem*)work_held.take();
    S.slots = c->d_slots;
    S.results = c->d_results;
    S.capacity = (unsigned)used;
    S.desc = c->d_desc;
    S.work = c->d_work;
    S.work_cap = (unsigned)n_work;
    S.redo_in = S.redo_out;
    S.redo_out = nullptr;
    c->S = S;
    const unsigned n_redo = std::min(pc.redo_out_count, kRedoCap);
    c->tiles_left = n_redo + (ticket < tp.ntiles ? tp.ntiles - ticket : 0u);
    const uint64_t bytes = held * (kSlotBytes + sizeof(uint4)) + n_desc * sizeof(rrtk::TileDesc) + n_work * sizeof(rrtk::WorkItem) + kCapCtrlBytes + plane_bytes;
    const uint64_t info[8] = {samples, used, bytes, n_desc, c->tiles_left, tp.packed ? 1u : 0u, tp.ntiles, (uint64_t)cap_slots * kSlotBytes};
    std::memcpy(c->info, info, sizeof(info));
    CAP_CU(cudaEventRecord(c->done, st));
    *out = c;
    return RRT_OK;
}

#undef CAP_CU

}  // extern "C"

// What rrt_capture_render and rrt_capture_render_mb check besides their own arguments: rrt_capture_render's rules.
static int check_capture_render(rrt_capture* cap, const char* what, const rrt_params* prm, const rrt_effects* fx, uint64_t sky_texture,
                                void* d_out, int out_layout, float* hdr_out) {
    const std::string m = what;
    if (!prm || !fx || sky_texture == 0 || !outputs_ok(out_layout, d_out, hdr_out))
        return fail(cap->ctx, RRT_ERR_BAD_ARG, m + ": bad argument");
    if (((prm->flags ^ cap->prm.flags) & RRT_FLAG_FMAD) || fx->use_lens != cap->fx.use_lens ||
        std::memcmp(&fx->distortion_amount, &cap->fx.distortion_amount, sizeof(float)) != 0)
        return fail(cap->ctx, RRT_ERR_BAD_ARG, m + ": the RRT_FLAG_FMAD bit, use_lens and distortion_amount must be the capture's");
    return RRT_OK;
}

// The kernels of one render of a capture at `time`, enqueued on `st`: shade, media, fold and, when the pass left tiles,
// the sweep.  Arguments checked, ctx->mu held, ctx->device current, `st` ordered after the capture's previous render.
static int capture_enqueue(rrt_capture* cap, float exposure, const rrt_effects* fx, uint64_t sky_texture, float time, void* d_out,
                           int out_layout, float* hdr_out, cudaStream_t st) {
    rrt_context* ctx = cap->ctx;
    rrt_params P = cap->prm;
    P.exposure = exposure;
    const rrtk::SplitKernels* sk = cap->plan.sk;
    FrameArgs A = frame_args(P, cap->cam, *fx, sky_texture, time, cap->w, cap->h, cap->band, cap->local_rows, out_layout, d_out);
    A.planes.hdr = hdr_out;
    A.counters = ctx->d_counters;
    A.ticket = (unsigned*)(cap->d_ctrl + kCapTicket);
    rrtk::PassCtrl* pcs = (rrtk::PassCtrl*)cap->d_ctrl;
    const int per_sm_media = resident_per_sm(ctx, (const void*)sk->media_results, kMediaBlock, true);
    if (per_sm_media < 0) return per_sm_media;
    const int per_sm_fold = resident_per_sm(ctx, (const void*)sk->fold_results, 128, false);
    if (per_sm_fold < 0) return per_sm_fold;
    // 1. every pixel from the planes; right for the rays the trace finished, overwritten below for the others
    const long long n = (long long)cap->w * cap->local_rows;
    kset(&P)->shade<<<(unsigned)((n + kShadeBlock - 1) / kShadeBlock), kShadeBlock, 0, st>>>(A, cap->planes);
    // 2.-4. the kept samples at this time, then fold + finish of the queued rays
    static_assert(offsetof(rrtk::PassCtrl, fold_ticket) == offsetof(rrtk::PassCtrl, media_ticket) + sizeof(unsigned), "PassCtrl layout");
    RRT_CU(ctx, cudaMemsetAsync(&pcs[0].media_ticket, 0, 2 * sizeof(unsigned), st));
    sk->media_results<<<(unsigned)(ctx->sm_count * per_sm_media), kMediaBlock, 0, st>>>(A, cap->S);
    sk->fold_results<<<(unsigned)(ctx->sm_count * per_sm_fold), 128, 0, st>>>(A, cap->S);
    int launches = 3;
    // 5. the tiles the pass could not hold, with the fused code: its redo list first, then the tickets it never took
    if (cap->tiles_left) {
        RRT_CU(ctx, cudaMemcpyAsync(A.ticket, A.ticket + 1, sizeof(unsigned), cudaMemcpyDeviceToDevice, st));
        RRT_CU(ctx, cudaMemsetAsync(&pcs[1], 0, sizeof(rrtk::PassCtrl), st));
        rrtk::SplitArgs S = cap->S;
        S.pass = 1;
        S.pc = pcs + 1;
        S.pc_prev = pcs;
        if (int rc = launch_sweep(ctx, cap->plan, A, S, rrtk::LensArgs{}, st)) return rc;
        ++launches;
    }
    RRT_CU(ctx, cudaGetLastError());
    ctx->launches += launches;
    return RRT_OK;
}

extern "C" {

int rrt_capture_render(rrt_capture* cap, const rrt_params* prm, const rrt_effects* fx, uint64_t sky_texture, float time, void* d_out,
                       int out_layout, float* hdr_out, void* stream) {
    if (!cap) return fail(nullptr, RRT_ERR_BAD_ARG, "rrt_capture_render: capture is NULL");
    if (int rc = check_capture_render(cap, "rrt_capture_render", prm, fx, sky_texture, d_out, out_layout, hdr_out)) return rc;
    if (cap->local_rows == 0) return RRT_OK;

    rrt_context* ctx = cap->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    DevGuard g(ctx->device);
    cudaStream_t st = (cudaStream_t)stream;
    RRT_CU(ctx, cudaStreamWaitEvent(st, cap->done, 0));   // one render at a time per capture, whatever the streams
    const int rc = capture_enqueue(cap, prm->exposure, fx, sky_texture, time, d_out, out_layout, hdr_out, st);
    // recorded even when the enqueue failed part-way: whatever it did enqueue stays ordered before the next render
    const cudaError_t e = cudaEventRecord(cap->done, st);
    if (rc != RRT_OK) return rc;
    if (e != cudaSuccess) return fail(ctx, RRT_ERR_CUDA, "rrt_capture_render: cudaEventRecord", e);
    return RRT_OK;
}

int rrt_capture_render_mb(rrt_capture* cap, const rrt_params* prm, const rrt_effects* fx, uint64_t sky_texture, const float* times,
                          int n, void* d_out, int out_layout, float* hdr_out, void* stream) {
    if (!cap) return fail(nullptr, RRT_ERR_BAD_ARG, "rrt_capture_render_mb: capture is NULL");
    rrt_context* ctx = cap->ctx;
    if (!times) return fail(ctx, RRT_ERR_BAD_ARG, "rrt_capture_render_mb: bad argument");
    if (int rc = check_capture_render(cap, "rrt_capture_render_mb", prm, fx, sky_texture, d_out, out_layout, hdr_out)) return rc;
    rrt_band b;
    int local_rows = 0;
    if (int rc = check_mb(ctx, "rrt_capture_render_mb", n, cap->w, cap->h, &cap->band, &b, &local_rows)) return rc;
    if (local_rows == 0) return RRT_OK;

    std::lock_guard<std::mutex> lk(ctx->mu);
    DevGuard g(ctx->device);
    const cudaStream_t st = (cudaStream_t)stream;
    const size_t plane = (size_t)cap->w * cap->h;   // full-frame, like the capture's own planes
    return with_scratch(ctx, "rrt_capture_render_mb", "sub-frame stack", 16 * n * plane, st, [&](float* stack) {
        // the capture's state is in use from the first sub-frame to the last: wait for its previous render once, record once
        if (cudaError_t e = cudaStreamWaitEvent(st, cap->done, 0)) return fail(ctx, RRT_ERR_CUDA, "rrt_capture_render_mb: cudaStreamWaitEvent", e);
        int rc = RRT_OK;
        for (int i = 0; i < n && rc == RRT_OK; ++i)
            rc = capture_enqueue(cap, prm->exposure, fx, sky_texture, times[i], nullptr, RRT_OUT_FRAME, stack + 4 * plane * i, st);
        // recorded even when a sub-frame failed: whatever was enqueued stays ordered before the capture's next render
        const cudaError_t e = cudaEventRecord(cap->done, st);
        if (rc != RRT_OK) return rc;
        if (e != cudaSuccess) return fail(ctx, RRT_ERR_CUDA, "rrt_capture_render_mb: cudaEventRecord", e);
        return launch_resolve(ctx, *prm, *fx, 1, n, cap->w, cap->h, b, local_rows, stack, plane, d_out, out_layout, hdr_out, st);
    });
}

int rrt_capture_info(const rrt_capture* cap, uint64_t out[8]) {
    if (!cap) return RRT_ERR_BAD_ARG;
    if (!out) return fail(cap->ctx, RRT_ERR_BAD_ARG, "rrt_capture_info: out is NULL");
    std::memcpy(out, cap->info, sizeof(cap->info));
    return RRT_OK;
}

void rrt_capture_destroy(rrt_capture* cap) {
    if (cap) free_capture(cap);
}

int rrt_render_host_async(rrt_context* ctx, const rrt_params* prm, const rrt_camera* cam, const rrt_effects* fx,
                          uint64_t sky_texture, float time, int w, int h, uint8_t* host_rgba, int slot, void* stream) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!host_rgba || w <= 0 || h <= 0 || slot < 0 || slot >= RRT_HOST_SLOTS)
        return fail(ctx, RRT_ERR_BAD_ARG, "rrt_render_host_async: bad argument");
    const size_t bytes = (size_t)w * h * 4;
    void* d_frame = nullptr;   // this slot's device frame, read while the context lock is held
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        DevGuard g(ctx->device);
        if (ctx->d_frame_bytes[slot] < bytes) {  // first use of this slot at this size (synchronous, like any cudaMalloc)
            if (ctx->d_frame[slot]) cudaFree(ctx->d_frame[slot]);
            ctx->d_frame[slot] = nullptr;
            ctx->d_frame_bytes[slot] = 0;
            RRT_CU(ctx, cudaMalloc(&ctx->d_frame[slot], bytes));
            ctx->d_frame_bytes[slot] = bytes;
        }
        d_frame = ctx->d_frame[slot];
    }
    int rc = rrt_render(ctx, prm, cam, fx, sky_texture, time, w, h, nullptr, d_frame, RRT_OUT_FRAME, nullptr, stream);
    if (rc != RRT_OK) return rc;
    DevGuard g(ctx->device);
    RRT_CU(ctx, cudaMemcpyAsync(host_rgba, d_frame, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return RRT_OK;
}

int rrt_render_host(rrt_context* ctx, const rrt_params* prm, const rrt_camera* cam, const rrt_effects* fx,
                    uint64_t sky_texture, float time, int w, int h, uint8_t* host_rgba) {
    int rc = rrt_render_host_async(ctx, prm, cam, fx, sky_texture, time, w, h, host_rgba, 0, nullptr);
    if (rc != RRT_OK) return rc;
    DevGuard g(ctx->device);
    RRT_CU(ctx, cudaStreamSynchronize(nullptr));
    return RRT_OK;
}

int rrt_assemble_bands(rrt_context* ctx, const void* d_packed, int rows_per_rank, int w, int h, int nranks, int group,
                       void* d_frame, void* stream) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!d_packed || !d_frame || w <= 0 || h <= 0 || nranks <= 0 || group <= 0 || rows_per_rank <= 0)
        return fail(ctx, RRT_ERR_BAD_ARG, "rrt_assemble_bands: bad argument");
    DevGuard g(ctx->device);
    assemble_kernel<<<ctx->sm_count * 8, 256, 0, (cudaStream_t)stream>>>((const uchar4*)d_packed, rows_per_rank, w, h,
                                                                         nranks, group, (uchar4*)d_frame);
    RRT_CU(ctx, cudaGetLastError());
    { std::lock_guard<std::mutex> lk(ctx->mu); ctx->launches += 1; }
    return RRT_OK;
}

int rrt_peer_frame_create(rrt_context* ctx, size_t bytes, void** d_frame, uint8_t handle[RRT_PEER_HANDLE_BYTES]) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!d_frame || !handle || bytes == 0) return fail(ctx, RRT_ERR_BAD_ARG, "rrt_peer_frame_create: bad argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == RRT_PEER_HANDLE_BYTES, "CUDA IPC handle size");
    DevGuard g(ctx->device);
    *d_frame = nullptr;
    void* p = nullptr;
    RRT_CU(ctx, cudaMalloc(&p, bytes));   // a raw allocation: an IPC handle names a whole cudaMalloc block
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaMemset(p, 0, bytes);
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return fail(ctx, RRT_ERR_CUDA, "rrt_peer_frame_create", e); }
    std::memcpy(handle, &h, sizeof(h));
    *d_frame = p;
    return RRT_OK;
}

int rrt_peer_frame_open(rrt_context* ctx, const uint8_t handle[RRT_PEER_HANDLE_BYTES], void** d_frame) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!d_frame || !handle) return fail(ctx, RRT_ERR_BAD_ARG, "rrt_peer_frame_open: bad argument");
    DevGuard g(ctx->device);
    *d_frame = nullptr;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof(h));
    RRT_CU(ctx, cudaIpcOpenMemHandle(d_frame, h, cudaIpcMemLazyEnablePeerAccess));
    return RRT_OK;
}

int rrt_peer_frame_read(rrt_context* ctx, const void* d_frame, size_t bytes, void* dst, void* stream) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!d_frame || !dst || bytes == 0) return fail(ctx, RRT_ERR_BAD_ARG, "rrt_peer_frame_read: bad argument");
    DevGuard g(ctx->device);
    RRT_CU(ctx, cudaMemcpyAsync(dst, d_frame, bytes, cudaMemcpyDefault, (cudaStream_t)stream));
    return RRT_OK;
}

int rrt_peer_frame_close(rrt_context* ctx, void* d_frame, int owner) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!d_frame) return RRT_OK;
    DevGuard g(ctx->device);
    RRT_CU(ctx, cudaDeviceSynchronize());
    if (owner) RRT_CU(ctx, cudaFree(d_frame));
    else RRT_CU(ctx, cudaIpcCloseMemHandle(d_frame));
    return RRT_OK;
}

int rrt_read_counters(rrt_context* ctx, rrt_counters* out, int reset) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!out) return fail(ctx, RRT_ERR_BAD_ARG, "rrt_read_counters: out is NULL");
    DevGuard g(ctx->device);
    RRT_CU(ctx, cudaDeviceSynchronize());
    RRT_CU(ctx, cudaMemcpy(out, ctx->d_counters, sizeof(rrt_counters), cudaMemcpyDeviceToHost));
    if (reset) RRT_CU(ctx, cudaMemset(ctx->d_counters, 0, sizeof(rrt_counters)));
    return RRT_OK;
}

// ---- probes -----------------------------------------------------------------------------------------
#define PROBE_PROLOGUE(cond)                                                  \
    if (!ctx) return RRT_ERR_BAD_ARG;                                         \
    if (!(cond) || n < 0) return fail(ctx, RRT_ERR_BAD_ARG, "probe: bad argument"); \
    DevGuard g__(ctx->device);

int rrt_geodesic_acc_batch(rrt_context* ctx, const rrt_params* prm, int n, const float* q, const float* v, float* out) {
    PROBE_PROLOGUE(prm && q && v && out)
    DBuf dq, dv, dout;
    const size_t b = (size_t)n * 3 * sizeof(float);
    RRT_CU(ctx, dq.alloc(b)); RRT_CU(ctx, dv.alloc(b)); RRT_CU(ctx, dout.alloc(b));
    RRT_CU(ctx, cudaMemcpy(dq.p, q, b, cudaMemcpyHostToDevice));
    RRT_CU(ctx, cudaMemcpy(dv.p, v, b, cudaMemcpyHostToDevice));
    int rc = run_probe(ctx, n, kset(prm)->acc, make_consts(*prm), n, (const float*)dq.p, (const float*)dv.p, (float*)dout.p);
    if (rc) return rc;
    RRT_CU(ctx, cudaMemcpy(out, dout.p, b, cudaMemcpyDeviceToHost));
    return RRT_OK;
}

static int step_batch(rrt_context* ctx, const rrt_params* prm, int n, float* p, float* v, const float* h, bool rk4) {
    PROBE_PROLOGUE(prm && p && v && h)
    DBuf dp, dv, dh;
    const size_t b = (size_t)n * 3 * sizeof(float);
    RRT_CU(ctx, dp.alloc(b)); RRT_CU(ctx, dv.alloc(b)); RRT_CU(ctx, dh.alloc((size_t)n * sizeof(float)));
    RRT_CU(ctx, cudaMemcpy(dp.p, p, b, cudaMemcpyHostToDevice));
    RRT_CU(ctx, cudaMemcpy(dv.p, v, b, cudaMemcpyHostToDevice));
    RRT_CU(ctx, cudaMemcpy(dh.p, h, (size_t)n * sizeof(float), cudaMemcpyHostToDevice));
    int rc = run_probe(ctx, n, rk4 ? kset(prm)->rk4 : kset(prm)->euler, make_consts(*prm), n, (float*)dp.p, (float*)dv.p, (const float*)dh.p);
    if (rc) return rc;
    RRT_CU(ctx, cudaMemcpy(p, dp.p, b, cudaMemcpyDeviceToHost));
    RRT_CU(ctx, cudaMemcpy(v, dv.p, b, cudaMemcpyDeviceToHost));
    return RRT_OK;
}
int rrt_rk4_step_batch(rrt_context* ctx, const rrt_params* prm, int n, float* p, float* v, const float* h) {
    return step_batch(ctx, prm, n, p, v, h, true);
}
int rrt_euler_step_batch(rrt_context* ctx, const rrt_params* prm, int n, float* p, float* v, const float* h) {
    return step_batch(ctx, prm, n, p, v, h, false);
}

int rrt_redshift_batch(rrt_context* ctx, const rrt_params* prm, int n, const float* q, const float* v, float* out) {
    PROBE_PROLOGUE(prm && q && v && out)
    DBuf dq, dv, dout;
    const size_t b = (size_t)n * 3 * sizeof(float);
    RRT_CU(ctx, dq.alloc(b)); RRT_CU(ctx, dv.alloc(b)); RRT_CU(ctx, dout.alloc((size_t)n * sizeof(float)));
    RRT_CU(ctx, cudaMemcpy(dq.p, q, b, cudaMemcpyHostToDevice));
    RRT_CU(ctx, cudaMemcpy(dv.p, v, b, cudaMemcpyHostToDevice));
    int rc = run_probe(ctx, n, kset(prm)->redshift, make_consts(*prm), n, (const float*)dq.p, (const float*)dv.p, (float*)dout.p);
    if (rc) return rc;
    RRT_CU(ctx, cudaMemcpy(out, dout.p, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
    return RRT_OK;
}

}  // extern "C"
// scalar-of-float3 probes share one shape: p[3n] -> out[n]
template <typename Launch>
static int p3_to_scalar(rrt_context* ctx, int n, const float* p, float* out, Launch launch) {
    PROBE_PROLOGUE(p && out)
    DBuf dp, dout;
    RRT_CU(ctx, dp.alloc((size_t)n * 3 * sizeof(float))); RRT_CU(ctx, dout.alloc((size_t)n * sizeof(float)));
    RRT_CU(ctx, cudaMemcpy(dp.p, p, (size_t)n * 3 * sizeof(float), cudaMemcpyHostToDevice));
    int rc = launch((const float*)dp.p, (float*)dout.p);
    if (rc) return rc;
    RRT_CU(ctx, cudaMemcpy(out, dout.p, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
    return RRT_OK;
}
extern "C" {
int rrt_hash31_batch(rrt_context* ctx, int n, const float* p, float* out) {
    return p3_to_scalar(ctx, n, p, out, [&](const float* dp, float* dout) { return run_probe(ctx, n, kset_noise(ctx)->hash31, n, dp, dout); });
}
int rrt_noise3d_batch(rrt_context* ctx, int n, const float* p, float* out) {
    return p3_to_scalar(ctx, n, p, out, [&](const float* dp, float* dout) { return run_probe(ctx, n, kset_noise(ctx)->noise3d, n, dp, dout); });
}
int rrt_fbm_batch(rrt_context* ctx, int n, const float* p, int octaves, float* out) {
    if (octaves < 0 || octaves > 16) return ctx ? fail(ctx, RRT_ERR_BAD_ARG, "rrt_fbm_batch: octaves out of range") : RRT_ERR_BAD_ARG;
    return p3_to_scalar(ctx, n, p, out, [&](const float* dp, float* dout) { return run_probe(ctx, n, kset_noise(ctx)->fbm, n, dp, octaves, dout); });
}
int rrt_disk_density_batch(rrt_context* ctx, const rrt_params* prm, int n, const float* q, float time, float* out) {
    if (!prm) return ctx ? fail(ctx, RRT_ERR_BAD_ARG, "probe: bad argument") : RRT_ERR_BAD_ARG;
    Consts C = make_consts(*prm);
    return p3_to_scalar(ctx, n, q, out, [&](const float* dp, float* dout) { return run_probe(ctx, n, kset(prm)->disk_density, C, n, dp, time, dout); });
}
int rrt_dust_density_batch(rrt_context* ctx, const rrt_params* prm, int n, const float* q, float time, float* out) {
    if (!prm) return ctx ? fail(ctx, RRT_ERR_BAD_ARG, "probe: bad argument") : RRT_ERR_BAD_ARG;
    Consts C = make_consts(*prm);
    return p3_to_scalar(ctx, n, q, out, [&](const float* dp, float* dout) { return run_probe(ctx, n, kset(prm)->dust_density, C, n, dp, time, dout); });
}
int rrt_disk_temperature_batch(rrt_context* ctx, const rrt_params* prm, int n, const float* r, float* out) {
    PROBE_PROLOGUE(prm && r && out)
    DBuf dr, dout;
    RRT_CU(ctx, dr.alloc((size_t)n * sizeof(float))); RRT_CU(ctx, dout.alloc((size_t)n * sizeof(float)));
    RRT_CU(ctx, cudaMemcpy(dr.p, r, (size_t)n * sizeof(float), cudaMemcpyHostToDevice));
    int rc = run_probe(ctx, n, kset(prm)->disk_temp, make_consts(*prm), n, (const float*)dr.p, (float*)dout.p);
    if (rc) return rc;
    RRT_CU(ctx, cudaMemcpy(out, dout.p, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
    return RRT_OK;
}
int rrt_sky_sample_batch(rrt_context* ctx, uint64_t sky_texture, int n, const float* tx, const float* ty, float* out4) {
    PROBE_PROLOGUE(sky_texture && tx && ty && out4)
    DBuf dx, dy, dout;
    RRT_CU(ctx, dx.alloc((size_t)n * sizeof(float))); RRT_CU(ctx, dy.alloc((size_t)n * sizeof(float)));
    RRT_CU(ctx, dout.alloc((size_t)n * 4 * sizeof(float)));
    RRT_CU(ctx, cudaMemcpy(dx.p, tx, (size_t)n * sizeof(float), cudaMemcpyHostToDevice));
    RRT_CU(ctx, cudaMemcpy(dy.p, ty, (size_t)n * sizeof(float), cudaMemcpyHostToDevice));
    int rc = run_probe(ctx, n, k_sky, (cudaTextureObject_t)sky_texture, n, (const float*)dx.p, (const float*)dy.p, (float4*)dout.p);
    if (rc) return rc;
    RRT_CU(ctx, cudaMemcpy(out4, dout.p, (size_t)n * 4 * sizeof(float), cudaMemcpyDeviceToHost));
    return RRT_OK;
}

uint64_t rrt_kernel_launches(rrt_context* ctx) {
    if (!ctx) return 0;
    std::lock_guard<std::mutex> lk(ctx->mu);
    return ctx->launches;
}

int rrt_set_pipeline(rrt_context* ctx, int mode) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (mode != RRT_PIPELINE_AUTO && mode != RRT_PIPELINE_FUSED && mode != RRT_PIPELINE_SPLIT) return fail(ctx, RRT_ERR_BAD_ARG, "rrt_set_pipeline: bad mode");
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->pipeline = mode;
    return RRT_OK;
}

int rrt_set_sample_pool(rrt_context* ctx, size_t max_bytes_per_stream, int max_passes) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (max_passes < 0 || max_passes > kMaxPasses) return fail(ctx, RRT_ERR_BAD_ARG, "rrt_set_sample_pool: max_passes out of range");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (max_bytes_per_stream) ctx->pool_bytes_max = max_bytes_per_stream;
    if (max_passes) ctx->max_passes = max_passes;
    return RRT_OK;
}

int rrt_split_stats(rrt_context* ctx, uint32_t out[8]) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!out) return fail(ctx, RRT_ERR_BAD_ARG, "rrt_split_stats: out is NULL");
    std::lock_guard<std::mutex> lk(ctx->mu);
    DevGuard g(ctx->device);
    RRT_CU(ctx, cudaDeviceSynchronize());
    const rrt_context::SamplePool* last = nullptr;
    for (const auto& pl : ctx->pools)
        if (pl.in_use && (!last || pl.last_use > last->last_use)) last = &pl;
    for (int i = 0; i < 8; ++i) out[i] = last ? last->h_stats[i] : 0u;
    if (last) {
        out[5] = (uint32_t)(last->cap_slots >> 10);   // pool size in Ki slots (32 B each)
    }
    return RRT_OK;
}

int rrt_set_frames_in_flight(rrt_context* ctx, int n) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (n < 1 || n > RRT_HOST_SLOTS) return fail(ctx, RRT_ERR_BAD_ARG, "rrt_set_frames_in_flight: n out of range");
    ctx->frames_in_flight = n;
    return RRT_OK;
}

int rrt_debug_tile_log(rrt_context* ctx, void* d_log, size_t entries) {
    if (!ctx) return RRT_ERR_BAD_ARG;
#ifndef RRT_WITH_TILE_LOG
    if (d_log) return fail(ctx, RRT_ERR_UNSUPPORTED, "rrt_debug_tile_log: this library was built without -DRRT_WITH_TILE_LOG (make -C csrc timeline)");
#endif
    if (entries > 0xffffffffull) return fail(ctx, RRT_ERR_BAD_ARG, "rrt_debug_tile_log: too many entries");
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->tile_log = d_log ? (unsigned long long*)d_log : nullptr;
    ctx->tile_log_cap = d_log ? (unsigned)entries : 0u;
    return RRT_OK;
}

int rrt_set_probe_contract(rrt_context* ctx, int fmad) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    ctx->probe_fmad = fmad != 0;
    return RRT_OK;
}

int rrt_exact_math_selftest(rrt_context* ctx, uint64_t seed, uint64_t n, uint64_t* div_mismatches, uint64_t* sqrt_mismatches) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!div_mismatches || !sqrt_mismatches) return fail(ctx, RRT_ERR_BAD_ARG, "rrt_exact_math_selftest: bad argument");
    DevGuard g(ctx->device);
    DBuf bad;
    RRT_CU(ctx, bad.alloc(2 * sizeof(unsigned long long)));
    RRT_CU(ctx, cudaMemset(bad.p, 0, 2 * sizeof(unsigned long long)));
    k_exact_math<<<ctx->sm_count * 16, 256>>>((unsigned long long)seed, (unsigned long long)n, (unsigned long long*)bad.p);
    RRT_CU(ctx, cudaGetLastError());
    RRT_CU(ctx, cudaDeviceSynchronize());
    unsigned long long h[2] = {0, 0};
    RRT_CU(ctx, cudaMemcpy(h, bad.p, sizeof(h), cudaMemcpyDeviceToHost));
    *div_mismatches = h[0];
    *sqrt_mismatches = h[1];
    return RRT_OK;
}

int rrt_exact_pow_selftest(rrt_context* ctx, uint64_t seed, uint64_t n, uint64_t* used_exponent_mismatches, uint64_t* random_exponent_mismatches) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (!used_exponent_mismatches || !random_exponent_mismatches) return fail(ctx, RRT_ERR_BAD_ARG, "rrt_exact_pow_selftest: bad argument");
    DevGuard g(ctx->device);
    DBuf bad;
    RRT_CU(ctx, bad.alloc(2 * sizeof(unsigned long long)));
    RRT_CU(ctx, cudaMemset(bad.p, 0, 2 * sizeof(unsigned long long)));
    k_exact_pow<<<ctx->sm_count * 16, 256>>>((unsigned long long)seed, (unsigned long long)n, (unsigned long long*)bad.p);
    RRT_CU(ctx, cudaGetLastError());
    RRT_CU(ctx, cudaDeviceSynchronize());
    unsigned long long h[2] = {0, 0};
    RRT_CU(ctx, cudaMemcpy(h, bad.p, sizeof(h), cudaMemcpyDeviceToHost));
    *used_exponent_mismatches = h[0];
    *random_exponent_mismatches = h[1];
    return RRT_OK;
}

int rrt_fp32_peak_probe(rrt_context* ctx, int iters, double* tflops, double* ms_out) {
    if (!ctx) return RRT_ERR_BAD_ARG;
    if (iters <= 0 || !tflops) return fail(ctx, RRT_ERR_BAD_ARG, "rrt_fp32_peak_probe: bad argument");
    DevGuard g(ctx->device);
    DBuf sink;
    RRT_CU(ctx, sink.alloc(sizeof(float)));
    const int blocks = ctx->sm_count * 8, threads = 256;
    cudaEvent_t e0, e1;
    RRT_CU(ctx, cudaEventCreate(&e0));
    RRT_CU(ctx, cudaEventCreate(&e1));
    k_fp32_peak<<<blocks, threads>>>(iters / 8 + 1, 1.0f, (float*)sink.p);  // warm-up
    double best = 1e30;
    for (int rep = 0; rep < 3; ++rep) {
        cudaEventRecord(e0);
        k_fp32_peak<<<blocks, threads>>>(iters, 1.0f, (float*)sink.p);
        cudaEventRecord(e1);
        cudaError_t e = cudaEventSynchronize(e1);
        if (e != cudaSuccess) { cudaEventDestroy(e0); cudaEventDestroy(e1); return fail(ctx, RRT_ERR_CUDA, "fp32 probe", e); }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    const double flop = (double)blocks * threads * (double)iters * 16.0 * 8.0 * 2.0;
    *tflops = flop / (best * 1e-3) / 1e12;
    if (ms_out) *ms_out = best;
    return RRT_OK;
}

}  // extern "C"
