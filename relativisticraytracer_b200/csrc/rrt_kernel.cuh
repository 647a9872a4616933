// rrt_kernel.cuh -- the render kernel (one 8x4-pixel tile per persistent warp), its per-ray helpers, the re-shading
// kernel (rrt_shade), the resolve kernel (rrt_resolve, rrt_resolve_time) and the function-level probe kernels.  Compiled
// TWICE, once per rounding contract (include/rrt_device.cuh):
//   rrt_b200.cu   RRT_FMAD = 0, nvcc -fmad=false   -> rrt_kernels_strict()
//   rrt_fmad.cu   RRT_FMAD = 1, nvcc -fmad=true    -> rrt_kernels_fmad()
// Everything with device code sits in an anonymous namespace (internal linkage per translation unit); the
// plain-data types both units and the host code share are in namespace rrtk.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rrt.h"
#include "../../include/rrt_device.cuh"

namespace rrtk {
using rrt::Consts;

struct FrameArgs {
    Consts C;
    rrt_camera cam;
    rrt_effects fx;
    float time;
    int w, h;
    int band_rank, band_nranks, band_group, local_rows;
    int out_layout;
    uchar4* out;
    rrt_planes planes;
    cudaTextureObject_t sky;
    unsigned long long* counters;  // rrt_counters, 8 x u64
    unsigned int* ticket;          // tile ticket for this launch
    unsigned long long* tile_log;  // optional profiling aid (rrt_debug_tile_log): 4 x u64 per tile, see render_kernel
    unsigned int tile_log_cap;     // entries the log can hold
};

// The ray source of a kernel that creates rays, its LENS template argument:
//   kRaysPinhole  the frame's camera, FrameArgs::cam (rrt_render)
//   kRaysLens     each pixel's camera of the table LensArgs::cams (rrt_render_dof)
//   kRaysPano     FrameArgs::cam's position, the equirectangular direction of the pixel from LensArgs::pano (rrt_render_pano)
enum : int { kRaysPinhole = 0, kRaysLens = 1, kRaysPano = 2, kRaySources = 3 };

// The tables of the other ray sources, the last parameter of every kernel that creates rays; read by their kRaysLens and kRaysPano
// variants only (zero for every other launch).  A separate parameter rather than more FrameArgs fields: appended at the
// end of the parameter block it moves no parameter of the existing kernels, and each member appended to it moves none of
// the members before it.
//   cams, ss, near: pixel (x, y) of the traced frame starts its ray from cams[(y % ss) * ss + x % ss] instead of
//     FrameArgs::cam.  near: every camera of the table lies in the branch-free domain (trace_ray's fast_ok), decided once
//     on the host so that the gate stays a launch constant as it is with one camera.
//   pano: w column entries (cos, sin) of the longitude, then h row entries (cos, sin) of the latitude (rrt_pano_directions).
struct LensArgs {
    const rrt_camera* cams;
    int ss;
    int near;
    const float2* pano;
};
// The w + h entries of LensArgs::pano for a w x h panorama, as 2 * (w + h) floats (host code, rrt_host.cpp).
void pano_table(int w, int h, float* out);

// kernels of one rounding contract
struct KernelSet {
    // [lens][spin != 0][media]; lens: the ray source (kRaysPinhole, kRaysLens, kRaysPano) of the LENS template argument
    void (*render[kRaySources][2][2])(const FrameArgs, const LensArgs);
    void (*render_packed[kRaySources][2])(const FrameArgs, const LensArgs);  // [lens][spin != 0]; two rays per thread in f32x2 registers, no medium (rrt_packed.cuh); FMAD contract only
    void (*acc)(Consts, int, const float*, const float*, float*);
    void (*rk4)(Consts, int, float*, float*, const float*);
    void (*euler)(Consts, int, float*, float*, const float*);
    void (*redshift)(Consts, int, const float*, const float*, float*);
    void (*hash31)(int, const float*, float*);
    void (*noise3d)(int, const float*, float*);
    void (*fbm)(int, const float*, int, float*);
    void (*disk_temp)(Consts, int, const float*, float*);
    void (*disk_density)(Consts, int, const float*, float, float*);
    void (*dust_density)(Consts, int, const float*, float, float*);
    void (*shade)(const FrameArgs, const rrt_planes);  // rrt_shade: the step after the ray loop, from traced planes
    // rrt_resolve / rrt_resolve_time: mean of ss x ss blocks of n hdr planes + post step
    void (*resolve)(const FrameArgs, const float4*, int, int, size_t);
};
const KernelSet* rrt_kernels_strict();
const KernelSet* rrt_kernels_fmad();
}  // namespace rrtk

using rrt::Consts;
using rrt::V3;
using rrt::mk;
using rrtk::FrameArgs;
using rrtk::LensArgs;
using rrtk::kRaysPinhole;
using rrtk::kRaysLens;
using rrtk::kRaysPano;

namespace {

// render_kernel's tile: 8x4 pixels, one warp (8x4 measured best or equal, profiles/r1_history.md)
constexpr int kRTileW = 8, kRTileH = 4;
// render_kernel's warps share nothing (no shared memory, no barrier), so its CTA is ONE warp: a CTA's slot is
// handed to the next launch the moment that warp runs out of tickets, instead of waiting for the slowest of four --
// which is what lets the frames of a sequence overlap cleanly (rrt_set_frames_in_flight, FramePipeline).
constexpr int kRenderBlock = 32;
// steps per unchecked vacuum burst of the render loop
constexpr int kBurst = 8;
// The media variant of the render kernel is asked to fit 24 warps per SM, i.e. <= 80 registers: the
// out-of-line media code stalls on libdevice call chains and MUFU latency, and six warps per scheduler hide
// that better than the four the unconstrained 109-register build gets (4K C0 78.5 -> 76.2 ms, C3 147.6 -> 135.4;
// 7 and 8 CTAs are no better).  The geodesic-only variant needs ~72 registers anyway.
constexpr int kMinBlocks = 1, kMinBlocksMedia = 24;
// The kRaysLens and kRaysPano variants (rrt_render_dof, rrt_render_pano) of the media kernels -- render_kernel<SPIN, true, LENS>
// and sweep_kernel<SPIN, LENS>, the fused fallbacks of such a frame -- are asked for 18 warps per SM (<= 112 registers), where
// none of them spills.
constexpr int kMinBlocksMediaLens = 18;

struct RayResult {
    float hdr[3], T, I[3];
    V3 d, p, v;
    float uvx, uvy;
    int steps;
    unsigned n_disk, n_dust, n_dense;
    bool captured, touched, exhausted;
};

// General-domain RK4 step (guarded div/sqrt, r < acc_rmin select): the rarely taken fallback of the loop.
struct PV {
    V3 p, v;
};
template <bool SPIN>
__device__ __noinline__ PV rk4_step_general(const Consts& C, V3 p, V3 v, float h, float hh, float h6) {
    const float r2 = rrt::norm2_loop(p);
    rrt::rk4_step<SPIN>(C, p, v, h, hh, h6, r2, sqrtf(r2));
    return PV{p, v};
}

// One in-zone sample of the participating media: densities at the PRE-step position, redshift with the
// POST-step velocity, emission colour and the step transmittance (reference raymarcher.cu:67-108).  Kept
// out of line so the vacuum step loop stays a few KB of straight-line FMA code in the instruction cache.
struct MediaOut {
    float er, eg, eb, s;
    int dense;
};
// Emission colour and step transmittance of one sample given both densities (reference :71-108).
__device__ __noinline__ MediaOut media_final(const Consts& C, V3 q, V3 v, float r, float h, float dd, float dc) {
    MediaOut o = {0.f, 0.f, 0.f, 1.0f, 0};
    if (dd > 0.001f || dc > 0.001f) {                                                     // :71
        o.dense = 1;
        float er = 0.f, eg = 0.f, eb = 0.f, kappa = 0.f;
        const float g = rrt::redshift(C, q, v);  // same arguments in both branches (:77, :92)
        if (dd > 0.001f) {                                                                // :76-88
            float Tk = rrt::disk_temperature(C, r);
            const rrt::PowBase TB = rrt::pow_base(Tk / C.disk_temp_ref);   // raised to 0.5 and to 0.4 (:79, :82)
            float tn = rrt::pow_of(TB, 0.5f);
            float bol = rrt::m_powf(g, 4.0f) * tn * dd * C.disk_luminosity;
            float ct = g * rrt::pow_of(TB, 0.4f) * 2.5f;
            er += 1.0f * bol;
            eg += fminf(0.25f, 0.12f * ct) * bol;
            eb += fmaxf(0.0f, 0.01f * (ct - 2.0f)) * bol;
            kappa += dd * C.disk_opacity;
        }
        if (dc > 0.001f) {                                                                // :91-105
            float light = 0.5f + 3.0f * rrt::m_powf(C.isco / fmaxf(r, C.isco), 1.2f);
            float J = dc * C.cloud_luminosity * light;
            float sh = rrt::sstep(0.7f, 1.3f, g);
            er += 0.60f * J * rrt::mixf(1.2f, 0.8f, sh);
            eg += 0.65f * J * rrt::mixf(0.8f, 1.1f, sh);
            eb += 0.80f * J * rrt::mixf(0.6f, 1.4f, sh);
            kappa += dc * C.cloud_opacity;
        }
        const float tau = kappa * h;                                                      // :107
        o.s = rrt::t_expf(-tau);
        o.er = er; o.eg = eg; o.eb = eb;
    }
    return o;
}
__device__ __forceinline__ MediaOut media_sample(const Consts& C, V3 q, V3 v, float r, float h, float time, unsigned zones) {
    const float dd = (zones & 1u) ? rrt::disk_density(C, q, time) : 0.0f;                 // :68
    const float dc = (zones & 2u) ? rrt::dust_density(C, q, time) : 0.0f;                 // :69
    return media_final(C, q, v, r, h, dd, dc);
}

// Image row of row ly of the band (groups of band_group rows dealt round-robin to the band's ranks).
__device__ __forceinline__ int band_row(const FrameArgs& A, int ly) {
    const int grp = ly / A.band_group;
    return (grp * A.band_nranks + A.band_rank) * A.band_group + (ly - grp * A.band_group);
}
// Tile row of the k-th of nty tile rows, handed out from the image centre outwards.
__device__ __forceinline__ int centre_out_row(int k, int nty) {
    const int c = nty >> 1, m = min(c, nty - 1 - c);
    if (k <= 2 * m) return (k & 1) ? c + ((k + 1) >> 1) : c - (k >> 1);
    return (c > nty - 1 - c) ? (c - m - 1) - (k - (2 * m + 1)) : (c + m + 1) + (k - (2 * m + 1));
}

// image-plane coordinate of a pixel after the optional lens distortion (reference :20-25)
__device__ __forceinline__ void pixel_uv(const FrameArgs& A, int x, int y, float& uvx, float& uvy) {
    using namespace rrt;
    uvx = (float)x / (float)A.w;
    uvy = (float)y / (float)A.h;
    if (A.fx.use_lens) {  // post_processing.h:19-24
        const float tu = sub(uvx, 0.5f), tv = sub(uvy, 0.5f);
        const float rr = mad2(tu, tu, tv, tv);
        const float f = mad(rr, A.fx.distortion_amount, 1.0f);
        uvx = mad(tu, f, 0.5f);
        uvy = mad(tv, f, 0.5f);
    }
}

// The camera a pixel's ray starts from: the frame's, or with kRaysLens (rrt_render_dof) its entry of the camera table.
template <int LENS>
__device__ __forceinline__ const rrt_camera& ray_camera(const FrameArgs& A, const LensArgs& L, int x, int y) {
    if (LENS != kRaysLens) return A.cam;
    return L.cams[(y % L.ss) * L.ss + x % L.ss];
}

__device__ __forceinline__ V3 cam_pos(const rrt_camera& c) { return mk(c.pos[0], c.pos[1], c.pos[2]); }

// initial ray of a pixel given its (distorted) image-plane coordinate (reference :27-34)
__device__ __forceinline__ V3 ray_dir_uv(const FrameArgs& A, const rrt_camera& cam, float uvx, float uvy) {
    using namespace rrt;
    float uc = mad(uvx, 2.0f, -1.0f);  // :27
    const float vc = mad(uvy, 2.0f, -1.0f);  // :28
    const float aspect = (float)A.w / (float)A.h;
    uc = mul(uc, aspect);  // :30
    // forward + (right*u + up*v)
    return unit3(mk(add(mad(cam.right[0], uc, mul(cam.up[0], vc)), cam.forward[0]),
                    add(mad(cam.right[1], uc, mul(cam.up[1], vc)), cam.forward[1]),
                    add(mad(cam.right[2], uc, mul(cam.up[2], vc)), cam.forward[2])));  // :33-34
}
__device__ __forceinline__ V3 ray_dir(const FrameArgs& A, const rrt_camera& cam, int x, int y) {
    float uvx, uvy;
    pixel_uv(A, x, y, uvx, uvy);
    return ray_dir_uv(A, cam, uvx, uvy);
}
// initial ray of pixel (x, y) of an equirectangular panorama (kRaysPano, rrt_render_pano): with (cl, sl) = pano[x] and
// (cp, sp) = pano[w + y], d = (cp*cl * forward + cp*sl * right) + sp * up, every operation rounded on its own in that
// order -- rrt_pano_directions' vector bit for bit -- then unit3 like the pinhole ray.  The pinhole ray of pixel (1, 1) of
// a 2 x 2 frame with forward = d is that same unit3(d).
__device__ __forceinline__ V3 pano_dir(const FrameArgs& A, const LensArgs& L, int x, int y) {
    using namespace rrt;
    const float2 lon = L.pano[x], lat = L.pano[A.w + y];
    const float a = mul(lat.x, lon.x), b = mul(lat.x, lon.y);
    const rrt_camera& c = A.cam;
    return unit3(mk(add(add(mul(a, c.forward[0]), mul(b, c.right[0])), mul(lat.y, c.up[0])),
                    add(add(mul(a, c.forward[1]), mul(b, c.right[1])), mul(lat.y, c.up[1])),
                    add(add(mul(a, c.forward[2]), mul(b, c.right[2])), mul(lat.y, c.up[2]))));
}
// the initial direction of pixel (x, y) from camera `cam` (ray_camera<LENS>), whatever the ray source
template <int LENS>
__device__ __forceinline__ V3 ray_dir_src(const FrameArgs& A, const LensArgs& L, const rrt_camera& cam, int x, int y) {
    if (LENS == kRaysPano) return pano_dir(A, L, x, y);
    return ray_dir(A, cam, x, y);
}

constexpr unsigned kEndCaptured = 1u, kEndTouched = 2u, kEndExhausted = 4u;

// The first half of finish_ray_inl: background, final assembly (reference :123-150) and the planes.  Returns final_hdr
// in (hr, hg, hb).
__device__ __forceinline__ void compose_ray_inl(const FrameArgs& A, int x, int y, float Ir, float Ig, float Ib, float T, V3 p,
                                                V3 v, int steps, unsigned end, float& hr, float& hg, float& hb) {
    using namespace rrt;
    float bg[3] = {0.f, 0.f, 0.f};
    V3 d = mk(0.f, 0.f, 0.f);
    const bool captured = (end & kEndCaptured) != 0;
    if (!captured) {
        d = unit3(v);
        const float off = A.fx.use_ca ? A.fx.ca_amount : 0.0f;
        const float theta = asinf(d.y);
        const float ty_ = 0.5f - theta / kPi;
        const float phi0 = atan2f(d.z, d.x);
        float4 sR = tex2D<float4>(A.sky, 0.5f + (phi0 + off) / (2.0f * kPi), ty_);
        float4 sG = tex2D<float4>(A.sky, 0.5f + (phi0 + 0.0f) / (2.0f * kPi), ty_);
        float4 sB = tex2D<float4>(A.sky, 0.5f + (phi0 + -off) / (2.0f * kPi), ty_);
        bg[0] = sR.x; bg[1] = sG.y; bg[2] = sB.z;
    }
    hr = mad(bg[0], T, Ir); hg = mad(bg[1], T, Ig); hb = mad(bg[2], T, Ib);  // :148-150
    const bool touched = (end & kEndTouched) != 0, exhausted = (end & kEndExhausted) != 0;
    const size_t pix = (size_t)y * A.w + x;
    const uint8_t cls = (uint8_t)((captured ? RRT_CLS_CAPTURED : (touched ? RRT_CLS_DISK_HIT : RRT_CLS_ESCAPED)) |
                                  (exhausted ? RRT_CLSF_EXHAUSTED : 0u) | (touched ? RRT_CLSF_TOUCHED : 0u));
    if (A.planes.hdr) reinterpret_cast<float4*>(A.planes.hdr)[pix] = make_float4(hr, hg, hb, T);
    if (A.planes.dir) reinterpret_cast<float4*>(A.planes.dir)[pix] = make_float4(d.x, d.y, d.z, 0.f);
    if (A.planes.emis) reinterpret_cast<float4*>(A.planes.emis)[pix] = make_float4(Ir, Ig, Ib, 0.f);
    if (A.planes.pos) reinterpret_cast<float4*>(A.planes.pos)[pix] = make_float4(p.x, p.y, p.z, 0.f);
    if (A.planes.vel) reinterpret_cast<float4*>(A.planes.vel)[pix] = make_float4(v.x, v.y, v.z, 0.f);
    if (A.planes.cls) A.planes.cls[pix] = cls;
    if (A.planes.steps) A.planes.steps[pix] = steps;
}
// The second half: bloom, vignette, exposure tonemap and the store of the pixel's final_hdr (reference :154-168).
// (uvx, uvy) is the distorted image-plane coordinate of the pixel.  Shared by every render kernel (through
// finish_ray_inl), shade_kernel and resolve_kernel.
__device__ __forceinline__ void post_ray_inl(const FrameArgs& A, int x, int y, int ly, float uvx, float uvy, float hr, float hg,
                                             float hb) {
    using namespace rrt;
    if (A.fx.use_bloom) {  // :154-157, post_processing.h:27-31
        const float lum = dot3(mk(hr, hg, hb), mk(0.2126f, 0.7152f, 0.0722f));
        float b0 = 0.f, b1 = 0.f, b2 = 0.f;
        if (lum > A.fx.bloom_threshold) { b0 = hr; b1 = hg; b2 = hb; }
        hr = mad(b0, A.fx.bloom_intensity, hr);
        hg = mad(b1, A.fx.bloom_intensity, hg);
        hb = mad(b2, A.fx.bloom_intensity, hb);
    }
    if (A.fx.use_vignette) {  // :159-161, post_processing.h:13-17; smoothstep(0.8, 0.2, d * intensity), math_utils.h:45-48
        const float dx = sub(uvx, 0.5f), dy = sub(uvy, 0.5f);
        const float dist = sqrtf(add(mad2(dx, dx, dy, dy), 0.0f));
        const float t = fminf(fmaxf(msub(dist, A.fx.vignette_intensity, 0.8f) / (0.2f - 0.8f), 0.0f), 1.0f);
        const float vg = mul(mul(t, t), sub(3.0f, mul(2.0f, t)));
        hr = mul(hr, vg); hg = mul(hg, vg); hb = mul(hb, vg);
    }
    const float o_r = 1.0f - expf(mul(-hr, A.C.exposure));  // :164-166
    const float o_g = 1.0f - expf(mul(-hg, A.C.exposure));
    const float o_b = 1.0f - expf(mul(-hb, A.C.exposure));
    const uchar4 px = make_uchar4((unsigned char)(o_r * 255), (unsigned char)(o_g * 255), (unsigned char)(o_b * 255), 255);
    if (A.out_layout == RRT_OUT_FRAME) A.out[(size_t)(A.h - 1 - y) * A.w + x] = px;  // :168
    else A.out[(size_t)ly * A.w + x] = px;
}
// Everything after the loop for one ray: background, final assembly, planes, effects, tonemap, store
// (reference :123-173).  (uvx, uvy) is the distorted image-plane coordinate of the pixel.
__device__ __forceinline__ void finish_ray_inl(const FrameArgs& A, int x, int y, int ly, float uvx, float uvy, float Ir, float Ig,
                                               float Ib, float T, V3 p, V3 v, int steps, unsigned end) {
    float hr, hg, hb;
    compose_ray_inl(A, x, y, Ir, Ig, Ib, T, p, v, steps, end, hr, hg, hb);
    if (!A.out) return;
    post_ray_inl(A, x, y, ly, uvx, uvy, hr, hg, hb);
}
// out-of-line copy for the kernels that finalise rays one at a time from several places
__device__ __noinline__ void finish_ray(const FrameArgs& A, int x, int y, int ly, float Ir, float Ig, float Ib, float T, V3 p,
                                        V3 v, int steps, unsigned end) {
    float uvx, uvy;
    pixel_uv(A, x, y, uvx, uvy);
    finish_ray_inl(A, x, y, ly, uvx, uvy, Ir, Ig, Ib, T, p, v, steps, end);
}

// What trace_ray does with an in-zone step's media sample (reference :67-115):
//   kMediaNone    nothing (no medium requested)
//   kMediaInline  evaluates it on the spot and folds it into I / T (the fused render_kernel)
//   kMediaEmit    hands (pre-step position, post-step velocity, radius, zone) to an emitter -- the split pipeline of
//                 rrt_split.cuh, where a second kernel evaluates the samples of many rays densely packed and a third
//                 folds the results in step order.  Samples do not feed back into the trajectory, so all three modes
//                 trace the same ray.
enum : int { kMediaNone = 0, kMediaInline = 1, kMediaEmit = 2 };
struct NoEmit {
    __device__ __forceinline__ void emit(V3, V3, float, int, unsigned) {}
};

// One ray: reference raymarch_kernel lines 20-150.  LENS: the ray source (ray_camera, pano_dir).
template <bool SPIN, int MEDIA, int LENS, class EM>
__device__ __forceinline__ void trace_ray(const FrameArgs& A, const LensArgs& L, int x, int y, RayResult& R, EM& em) {
    const Consts& C = A.C;
    const rrt_camera& cam = ray_camera<LENS>(A, L, x, y);
    float uvx, uvy;
    pixel_uv(A, x, y, uvx, uvy);                                       // :20-25
    V3 p = mk(cam.pos[0], cam.pos[1], cam.pos[2]);
    V3 v = LENS == kRaysPano ? pano_dir(A, L, x, y) : ray_dir_uv(A, cam, uvx, uvy);   // :27-34

    float Ir = 0.f, Ig = 0.f, Ib = 0.f, T = 1.0f;
    bool captured = false, touched = false, escaped = false;
    int it = 0;
    unsigned n_disk = 0, n_dust = 0, n_dense = 0;
    const int max_steps = C.max_steps;
    const bool want_disk = (C.flags & RRT_FLAG_DISK) != 0, want_dust = (C.flags & RRT_FLAG_DUST) != 0;
    // Domain of the branch-free div/sqrt (rrt_device.cuh): a ray that starts absurdly far out takes the
    // general path for its whole life.  Uniform per launch in practice (depends on the camera only); with kRaysLens decided
    // for the whole camera table (LensArgs::near), which keeps it a launch constant.  Both paths give the same bits where
    // the fast one is valid, so the gate decides only the speed.
    const bool fast_ok = (LENS == kRaysLens ? L.near != 0 : rrt::dot3(p, p) < 1.0e8f) && C.acc_rmin < C.horizon_r && C.horizon_r >= 1e-3f;
    const float zone_rmax = fmaxf(18.0f, fmaxf(C.disk_zone_r, C.dust_zone_r));
    // one compare per step for "redo with the general code": smallest stage radius below acc_rmin (or NaN), or
    // the whole ray outside the fast domain (+inf: every step is redone)
    const float redo_below = fast_ok ? C.acc_rmin : __int_as_float(0x7f800000);
    constexpr int kBurstUnroll = MEDIA == kMediaInline ? 1 : 4;   // steps per trip of the burst loop
    static_assert(kBurst % kBurstUnroll == 0, "burst length must be a multiple of its unroll factor");
    // every threshold a checked vacuum step compares a radius against from above: zones (:56-58), horizon (:47),
    // geodesics.h:33 through the redo guard
    const float burst_min = fmaxf(zone_rmax, fmaxf(C.horizon_r, redo_below));
    // entry window: kBurst steps of |v| ~ 1 (1.25 allowed) must fit between the zone sphere and the escape sphere
    const float burst_margin = 1.25f * (float)kBurst * C.h[0];
    const float burst_lo = burst_min + burst_margin, burst_hi = 250.0f - burst_margin;
    // Two-level loop.  The inner loop holds what (nearly) every step needs -- the branch-free RK4 step and, in
    // lock-step for the lanes that are inside a medium, the out-of-line media sample -- and nothing else; the
    // general-domain redo of a step (practically never taken) is done by the outer loop, which then re-enters,
    // so its call does not cost the hot loop registers or convergence barriers.  `it` counts executed
    // integrate_rk4 calls on every path.
    auto fold = [&](const MediaOut& m) {                                                      // :71, :107-115
        if (m.dense) {
            touched = true;
            ++n_dense;
            const float wgt = rrt::mul(rrt::sub(1.0f, m.s), T);                               // :109
            Ir = rrt::mad(m.er, wgt, Ir); Ig = rrt::mad(m.eg, wgt, Ig); Ib = rrt::mad(m.eb, wgt, Ib);   // :111-113
            T = rrt::mul(T, m.s);                                                             // :115
        }
    };
    enum : int { kRanOut = 0, kCaptured = 1, kEscaped = 2, kRedo = 3 };
    int burst_after = 0;   // no burst before this iteration count (set when one was rejected)
    for (;;) {
        int ev = kRanOut;
        V3 q = p, v_in = v;   // pre-step state: media and the escape test use q (:68-69, :120)
        float r = 0.0f;
        int zone_index = 0;   // which step size the step used (config.h:47 x {1, 0.1, 0.3, 0.5}); h itself stays in the loop
        unsigned zones = 0;
        // The loop is rotated: |p| of the NEXT iteration's header (:43-44) is computed right after the step, so
        // its multiply -> rsqrt -> refine chain overlaps the escape test and the loop bookkeeping instead of
        // standing alone at the top of every iteration (it was ~20 % of the stall samples there).
        float r2 = rrt::norm2_loop(p);
        r = rrt::sqrt_rn_fast(r2);                                                            // :44
        // ---- phase 1: vacuum bursts ------------------------------------------------------------------------------
        // Most steps (94 % of the headline frame's) happen outside every step-size zone, with the whole-warp step h[0]
        // and no medium; there the horizon test (:47), the zone logic (:54-62), the media branch (:67) and the escape test
        // (:120) are all false.  While the radii say the next kBurst steps will stay in that regime, take them straight-line
        // with none of those checks, tracking only the smallest radius any stage or state saw and the largest state radius
        // (FMNMX on the ALU pipe, off the FMA pipe), and validate afterwards: min >= every threshold the checks compare
        // against, max <= 250.  If the validation fails the state is rolled back.  Either way control goes on to the
        // checked steps of phase 2, so the result is the reference's on every path -- the entry margin only decides how
        // often a burst is wasted, never what is computed.
        //  * Warp-uniform on purpose: a burst is taken only when EVERY lane still in the loop qualifies.  A lane that
        //    burst on its own would finish its vacuum phase in 1/kBurst of the iterations -- alone, while its tile mates
        //    are still in a zone -- instead of sharing each execution of the step with the other vacuum lanes of the warp
        //    (measured with per-lane bursts: the media-heavy cameras, whose tiles are mixed, got 2-6 % slower).
        //    (__activemask: the vote only decides how the steps are scheduled, never what they compute.)
        //  * A loop of its own, in front of the checked loop rather than a block inside it: the zone / media iterations
        //    then do not jump over 3 KB of burst code every time (instruction-fetch stalls doubled on the media-heavy
        //    C3 frame with the block inside: ncu no_instruction 0.54 -> 1.05 warps per issue).
        {
            const unsigned in_loop = __activemask();
#pragma unroll 1
            while (r >= burst_lo && r <= burst_hi && it >= burst_after && it + kBurst < max_steps && __activemask() == in_loop) {
                const V3 ps = p, vs = v;
                const float r2s = r2, rs = r;
                float mn = r, mx = r;
                // kBurst steps as kBurst / kBurstUnroll trips of a rolled loop: the step is ~3 KB of code, and the media
                // kernels' instruction working set (noise, densities, libdevice) has no room for a fully unrolled burst
#pragma unroll 1
                for (int kb = 0; kb < kBurst / kBurstUnroll; ++kb) {
#pragma unroll
                    for (int ku = 0; ku < kBurstUnroll; ++ku) {
                        const float rm = rrt::rk4_step_fast<SPIN>(C, p, v, C.h[0], C.hh[0], C.h6[0], r2, r);   // :64
                        r2 = rrt::norm2_loop(p);
                        r = rrt::sqrt_rn_fast(r2);                                            // :44 of the next iteration
                        mn = fminf(mn, fminf(rm, r));
                        mx = fmaxf(mx, r);
                    }
                }
                // mn / mx include the radius of the state the next step starts from: its horizon test is covered too,
                // and its own escape test will see r <= 250
                if (mn >= burst_min && mx <= 250.0f) { it += kBurst; continue; }
                p = ps; v = vs; r2 = r2s; r = rs;
                burst_after = it + kBurst;   // a rejected burst (|v| well above 1): take the next steps one by one
                break;
            }
        }
        // ---- phase 2: checked steps, until the ray ends or the whole warp is back in the burst window ------------------
        bool rewind = false;
#pragma unroll 1
        while (it < max_steps) {                                                              // :41
            if (r < C.horizon_r) { ev = kCaptured; break; }                                   // :47-51
            unsigned z = 0;
            float rmin;
            q = p;
            v_in = v;
            // Which lanes take the general step below (step size from the zone table) and which the constant-step copy:
            // see the `else` branch.  With bursts in a media kernel the checked vacuum step is 1 in kBurst + 1, and the
            // instruction cache has no room for a third copy of the step next to the media code, so it uses this one.
            constexpr bool kOneCheckedStep = !RRT_FMAD || MEDIA == kMediaInline;
            if (kOneCheckedStep || r < zone_rmax) {
                float h = C.h[0], h6 = C.h6[0];
                int zsel = 0;
                if (r < zone_rmax) {  // one compare for the steps outside every zone
                    const bool near_bh = r < 18.0f;                                           // :56
                    const bool disk_zone = fabsf(p.y) < C.disk_zone_y && r < C.disk_zone_r;   // :57
                    const bool dust_zone = fabsf(p.y) < C.dust_zone_y && r < C.dust_zone_r;   // :58
                    const int zi = near_bh ? 1 : (disk_zone ? 2 : (dust_zone ? 3 : 0));       // :60-62
                    h = C.h[zi];
                    h6 = C.h6[zi];
                    zsel = zi;
                    if (MEDIA) z = (disk_zone && want_disk ? 1u : 0u) | (dust_zone && want_dust ? 2u : 0u);   // :67
                }
                zone_index = zsel;
                rmin = rrt::rk4_step_fast<SPIN>(C, p, v, h, h * 0.5f /* exact */, h6, r2, r);  // :64
            } else {
                // FMAD contract only.  3/4 of all steps are outside every zone; their step size is the same for the
                // whole warp, so this second copy of the step takes h, h/2 and h/6 as constant-bank operands and 24 of
                // its FFMAs read two registers instead of three.  The fused loop is bound by register-file operand
                // bandwidth (DESIGN.md): 4K C0 75.8 -> 74.1 ms.  The strict loop is issue bound and loses 3 % to the
                // larger code, so it keeps the single copy.
                zone_index = 0;
                rmin = rrt::rk4_step_fast<SPIN>(C, p, v, C.h[0], C.hh[0], C.h6[0], r2, r);    // :64
            }
            zones = z;
            if (!(rmin >= redo_below)) { ev = kRedo; break; }
            ++it;
            const float r2_next = rrt::norm2_loop(p);
            const float r_next = rrt::sqrt_rn_fast(r2_next);
            if (MEDIA != kMediaNone && z) {
                n_disk += z & 1u;
                n_dust += z >> 1;
                if (MEDIA == kMediaInline) fold(media_sample(C, q, v, r, C.h[zone_index], A.time, z));
                else em.emit(q, v, r, zone_index, z);
            }
            if (r > 250.0f && rrt::dot3(q, v) > 0.0f) { ev = kEscaped; break; }               // :120
            r2 = r2_next;
            r = r_next;
            {   // one VOTE per checked step: the lanes in the loop here, the qualifying ones inside the branch
                const unsigned in_loop = __activemask();
                if (r >= burst_lo && r <= burst_hi && it >= burst_after && it + kBurst < max_steps && __activemask() == in_loop) { rewind = true; break; }
            }
        }
        if (rewind) continue;   // back to phase 1 (p, v, it carry over; r2 / r are recomputed from p, bit for bit the same)
        if (ev == kRedo) {
            // outside the branch-free domain, or geodesics.h:33 can fire: redo this step with the general code
            const float h = C.h[zone_index];
            const PV s = rk4_step_general<SPIN>(C, q, v_in, h, h * 0.5f, C.h6[zone_index]);
            p = s.p; v = s.v;
            ++it;
            if (MEDIA != kMediaNone && zones) {
                n_disk += zones & 1u;
                n_dust += zones >> 1;
                if (MEDIA == kMediaInline) fold(media_sample(C, q, v, r, h, A.time, zones));
                else em.emit(q, v, r, zone_index, zones);
            }
            if (r > 250.0f && rrt::dot3(q, v) > 0.0f) { escaped = true; break; }              // :120
            continue;
        }
        if (ev == kCaptured) { captured = true; T = 0.0f; }
        escaped = ev == kEscaped;
        break;
    }
    R.exhausted = !captured && !escaped;  // the for loop ran out (:41)
    R.steps = it;
    R.captured = captured;
    R.touched = touched;
    R.n_disk = n_disk; R.n_dust = n_dust; R.n_dense = n_dense;
    R.p = p; R.v = v; R.T = T;
    R.I[0] = Ir; R.I[1] = Ig; R.I[2] = Ib;
    R.uvx = uvx; R.uvy = uvy;
}

template <bool SPIN, bool MEDIA, int LENS>
__global__ void __launch_bounds__(kRenderBlock, MEDIA ? (LENS != kRaysPinhole ? kMinBlocksMediaLens : kMinBlocksMedia) : kMinBlocks)
    render_kernel(const __grid_constant__ FrameArgs A, const __grid_constant__ LensArgs L) {
    const int lane = threadIdx.x & 31;
    const int ntx = (A.w + kRTileW - 1) / kRTileW;
    const int nty = (A.local_rows + kRTileH - 1) / kRTileH;
    const unsigned ntiles = (unsigned)(ntx * nty);
    unsigned long long c_steps = 0, c_disk = 0, c_dust = 0, c_dense = 0;
    unsigned c_cap = 0, c_esc = 0, c_exh = 0, c_touch = 0;

    for (;;) {
        unsigned tile = 0;
        if (lane == 0) tile = atomicAdd(A.ticket, 1u);
        tile = __shfl_sync(0xffffffffu, tile, 0);
        if (tile >= ntiles) break;
        // Tile rows are handed out from the image centre outwards: the rows that cross the hole and the
        // disk are the expensive ones, so they start first and the cheap sky rows fill the tail of the launch.
        const int tx = (int)(tile % (unsigned)ntx), k = (int)(tile / (unsigned)ntx);
        const int ty = centre_out_row(k, nty);
        const int x = tx * kRTileW + (lane & (kRTileW - 1));
        const int ly = ty * kRTileH + lane / kRTileW;
        if (x >= A.w || ly >= A.local_rows) continue;
        const int y = band_row(A, ly);
        if (y >= A.h) continue;

#ifdef RRT_WITH_TILE_LOG
        unsigned long long t_begin = 0;
        if (A.tile_log) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_begin));
#endif
        RayResult R;
        NoEmit no_emit;
        trace_ray<SPIN, MEDIA ? kMediaInline : kMediaNone, LENS>(A, L, x, y, R, no_emit);

        finish_ray_inl(A, x, y, ly, R.uvx, R.uvy, R.I[0], R.I[1], R.I[2], R.T, R.p, R.v, R.steps,
                       (R.captured ? kEndCaptured : 0u) | (R.touched ? kEndTouched : 0u) | (R.exhausted ? kEndExhausted : 0u));
        c_steps += (unsigned)R.steps;
        c_disk += R.n_disk; c_dust += R.n_dust; c_dense += R.n_dense;
        c_cap += R.captured; c_exh += R.exhausted; c_esc += (!R.captured && !R.exhausted); c_touch += R.touched;
#ifdef RRT_WITH_TILE_LOG   // (a build option, not a run-time one: the extra live values cost the step loop ~3 % through register allocation)
        if (A.tile_log) {   // who traced which tile from when to when (ns, %globaltimer) and how many steps its slowest ray took
            const int most = __reduce_max_sync(__activemask(), R.steps);
            if (lane == __ffs(__activemask()) - 1 && tile < A.tile_log_cap) {
                unsigned long long t_end;
                unsigned smid;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_end));
                asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
                unsigned long long* e = A.tile_log + 4ull * tile;
                e[0] = t_begin; e[1] = t_end; e[2] = ((unsigned long long)ty << 32) | (unsigned)tx;
                e[3] = ((unsigned long long)smid << 32) | (unsigned)most;
            }
        }
#endif
    }

    // one set of atomics per warp
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        c_steps += __shfl_xor_sync(0xffffffffu, c_steps, o);
        c_disk += __shfl_xor_sync(0xffffffffu, c_disk, o);
        c_dust += __shfl_xor_sync(0xffffffffu, c_dust, o);
        c_dense += __shfl_xor_sync(0xffffffffu, c_dense, o);
        c_cap += __shfl_xor_sync(0xffffffffu, c_cap, o);
        c_esc += __shfl_xor_sync(0xffffffffu, c_esc, o);
        c_exh += __shfl_xor_sync(0xffffffffu, c_exh, o);
        c_touch += __shfl_xor_sync(0xffffffffu, c_touch, o);
    }
    if (lane == 0 && A.counters) {
        atomicAdd(A.counters + 0, c_steps);
        atomicAdd(A.counters + 1, c_disk);
        atomicAdd(A.counters + 2, c_dust);
        atomicAdd(A.counters + 3, c_dense);
        atomicAdd(A.counters + 4, (unsigned long long)c_cap);
        atomicAdd(A.counters + 5, (unsigned long long)c_esc);
        atomicAdd(A.counters + 6, (unsigned long long)c_exh);
        atomicAdd(A.counters + 7, (unsigned long long)c_touch);
    }
}

// ---- re-shading (rrt_shade) -------------------------------------------------------------------------
// Everything after the ray loop again -- finish_ray_inl itself, so every byte is the one the render wrote for the same
// inputs -- from the planes a render left behind: I from `emis`, T from `hdr.w`, the exit velocity from `vel` (not
// `dir`: unit3 of an already normalised vector need not return the same bits) and the end bits from `cls`.  A.planes
// holds only the optional hdr output, which may be `traced.hdr` itself (each thread reads its pixel before it writes
// it).  One thread per pixel of the band, rows mapped like render_kernel's.
constexpr int kShadeBlock = 256;
__global__ void __launch_bounds__(kShadeBlock) shade_kernel(const __grid_constant__ FrameArgs A, const __grid_constant__ rrt_planes traced) {
    const int i = blockIdx.x * kShadeBlock + threadIdx.x;   // w * local_rows <= 2^30 (rrt_shade)
    if (i >= A.w * A.local_rows) return;
    const int ly = i / A.w, x = i - ly * A.w;
    const int y = band_row(A, ly);
    if (y >= A.h) return;
    const size_t pix = (size_t)y * A.w + x;
    const float4 v = reinterpret_cast<const float4*>(traced.vel)[pix];
    const float4 I = reinterpret_cast<const float4*>(traced.emis)[pix];
    const float4 hdr = reinterpret_cast<const float4*>(traced.hdr)[pix];
    const unsigned cls = traced.cls[pix];
    const unsigned end = ((cls & RRT_CLS_MASK) == RRT_CLS_CAPTURED ? kEndCaptured : 0u) |
                         ((cls & RRT_CLSF_TOUCHED) ? kEndTouched : 0u) | ((cls & RRT_CLSF_EXHAUSTED) ? kEndExhausted : 0u);
    float uvx, uvy;
    pixel_uv(A, x, y, uvx, uvy);
    finish_ray_inl(A, x, y, ly, uvx, uvy, I.x, I.y, I.z, hdr.w, mk(0.f, 0.f, 0.f), mk(v.x, v.y, v.z), 0, end);
}

// ---- resolve: supersample and shutter mean (rrt_resolve, rrt_render_ss, rrt_resolve_time, rrt_render_mb) ------------
// Box filter of n planes of ss*w x ss*h hdr values into the w x h frame of A.  Plane q starts at hi + q*plane_stride (in
// float4) and is indexed [Y * ss*w + X].  Output pixel (x, y) is the mean of sub-samples (ss*x + i, ss*y + j) of every
// plane, summed plane by plane (outer), then j, then i from (plane 0, 0, 0) and divided by n*ss*ss, with the explicit
// round-to-nearest intrinsics so that both contracts give the same bits (and numpy reproduces them).  rrt_resolve is
// n = 1, rrt_resolve_time is ss = 1.  The mean (.w = mean T) goes to A.planes.hdr, then the render's own post step
// (bloom, vignette at the output pixel's pixel_uv, tonemap, store) runs on it.  One thread per output pixel of the band,
// rows mapped like shade_kernel's; neighbouring threads read neighbouring ss*16-byte runs of each sub-row.
constexpr int kResolveBlock = 256;
__device__ __forceinline__ void add4_rn(float4& s, const float4 v) {
    s.x = __fadd_rn(s.x, v.x); s.y = __fadd_rn(s.y, v.y); s.z = __fadd_rn(s.z, v.z); s.w = __fadd_rn(s.w, v.w);
}
__global__ void __launch_bounds__(kResolveBlock) resolve_kernel(const __grid_constant__ FrameArgs A, const float4* __restrict__ hi, int ss,
                                                                int n, size_t plane_stride) {
    const int i = blockIdx.x * kResolveBlock + threadIdx.x;   // w * local_rows <= 2^30 (rrt_resolve, rrt_resolve_time)
    if (i >= A.w * A.local_rows) return;
    const int ly = i / A.w, x = i - ly * A.w;
    const int y = band_row(A, ly);
    if (y >= A.h) return;
    const size_t W = (size_t)ss * A.w;
    const float4* p = hi + (size_t)ss * y * W + (size_t)ss * x;
    float4 s = p[0];
    if (ss == 1) {   // one float4 per plane: unrolled so that the loads of several planes are in flight together
#pragma unroll 4
        for (int q = 1; q < n; ++q) add4_rn(s, p[q * plane_stride]);
    } else {
        for (int q = 0; q < n; ++q)
            for (int j = 0; j < ss; ++j)
                for (int k = q == 0 && j == 0 ? 1 : 0; k < ss; ++k) add4_rn(s, p[q * plane_stride + j * W + k]);
    }
    const float d = (float)(n * ss * ss);
    s = make_float4(__fdiv_rn(s.x, d), __fdiv_rn(s.y, d), __fdiv_rn(s.z, d), __fdiv_rn(s.w, d));
    if (A.planes.hdr) reinterpret_cast<float4*>(A.planes.hdr)[(size_t)y * A.w + x] = s;
    if (!A.out) return;
    float uvx, uvy;
    pixel_uv(A, x, y, uvx, uvy);
    post_ray_inl(A, x, y, ly, uvx, uvy, s.x, s.y, s.z);
}

// ---- probe kernels ---------------------------------------------------------------------------------
__device__ __forceinline__ V3 ld3(const float* a, int i) { return mk(a[3 * i], a[3 * i + 1], a[3 * i + 2]); }
__device__ __forceinline__ void st3(float* a, int i, V3 v) { a[3 * i] = v.x; a[3 * i + 1] = v.y; a[3 * i + 2] = v.z; }

__global__ void k_acc(Consts C, int n, const float* q, const float* v, float* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) st3(out, i, C.spin_a != 0.0f ? rrt::geodesic_acc<true>(C, ld3(q, i), ld3(v, i))
                                            : rrt::geodesic_acc<false>(C, ld3(q, i), ld3(v, i)));
}
__global__ void k_rk4(Consts C, int n, float* p, float* v, const float* h) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    V3 pp = ld3(p, i), vv = ld3(v, i);
    float hi = h[i], r2 = rrt::norm2_loop(pp);
    if (C.spin_a != 0.0f) rrt::rk4_step<true>(C, pp, vv, hi, hi * 0.5f, hi / 6.0f, r2, sqrtf(r2));
    else rrt::rk4_step<false>(C, pp, vv, hi, hi * 0.5f, hi / 6.0f, r2, sqrtf(r2));
    st3(p, i, pp);
    st3(v, i, vv);
}
__global__ void k_euler(Consts C, int n, float* p, float* v, const float* h) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    V3 pp = ld3(p, i), vv = ld3(v, i);
    if (C.spin_a != 0.0f) rrt::euler_step<true>(C, pp, vv, h[i]);
    else rrt::euler_step<false>(C, pp, vv, h[i]);
    st3(p, i, pp);
    st3(v, i, vv);
}
__global__ void k_redshift(Consts C, int n, const float* q, const float* v, float* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = rrt::redshift(C, ld3(q, i), ld3(v, i));
}
__global__ void k_hash31(int n, const float* p, float* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = rrt::hash31(ld3(p, i));
}
__global__ void k_noise3d(int n, const float* p, float* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = rrt::noise3d(ld3(p, i));
}
__global__ void k_fbm(int n, const float* p, int oct, float* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = rrt::fbm_rt(ld3(p, i), oct);
}
__global__ void k_disk_temp(Consts C, int n, const float* r, float* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = rrt::disk_temperature(C, r[i]);
}
__global__ void k_disk_density(Consts C, int n, const float* q, float time, float* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = rrt::disk_density(C, ld3(q, i), time);
}
__global__ void k_dust_density(Consts C, int n, const float* q, float time, float* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = rrt::dust_density(C, ld3(q, i), time);
}
__global__ void k_sky(cudaTextureObject_t sky, int n, const float* tx, const float* ty, float4* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = tex2D<float4>(sky, tx[i], ty[i]);
}

}  // namespace
#if RRT_FMAD
#include "rrt_packed.cuh"
#endif
#include "rrt_split.cuh"   // trace / media / fold kernels of the split pipeline (both contracts)
namespace {
const rrtk::KernelSet kKernelSet = {
    {{{render_kernel<false, false, 0>, render_kernel<false, true, 0>}, {render_kernel<true, false, 0>, render_kernel<true, true, 0>}},
     {{render_kernel<false, false, 1>, render_kernel<false, true, 1>}, {render_kernel<true, false, 1>, render_kernel<true, true, 1>}},
     {{render_kernel<false, false, 2>, render_kernel<false, true, 2>}, {render_kernel<true, false, 2>, render_kernel<true, true, 2>}}},
#if RRT_FMAD
    {{render_kernel_p<false, 0>, render_kernel_p<true, 0>}, {render_kernel_p<false, 1>, render_kernel_p<true, 1>},
     {render_kernel_p<false, 2>, render_kernel_p<true, 2>}},
#else
    {{nullptr, nullptr}, {nullptr, nullptr}, {nullptr, nullptr}},
#endif
    k_acc, k_rk4, k_euler, k_redshift, k_hash31, k_noise3d, k_fbm, k_disk_temp, k_disk_density, k_dust_density,
    shade_kernel, resolve_kernel,
};
}  // namespace

namespace rrtk {
#if RRT_FMAD
const KernelSet* rrt_kernels_fmad() { return &kKernelSet; }
#else
const KernelSet* rrt_kernels_strict() { return &kKernelSet; }
#endif
}  // namespace rrtk
