/*
 * rrt.h -- C ABI of the B200-native render path (librrt_b200.so).
 *
 * This is the drop-in boundary for ONE path of levi2234/RelativisticRayTracer: the per-pixel
 * geodesic integration + volumetric disk/dust march + skybox lookup that the reference runs in
 * raymarch_kernel (src/raymarcher.cu:15-174) behind launch_raymarch (include/raymarcher.h:19,
 * src/raymarcher.cu:176-180; sole caller renderFrame, src/main.cpp:467).
 *
 * Plain C: POD structs, raw pointers and sizes, int error codes.  No torch, no C++ types.
 * The C++ shim with the reference's exact launch_raymarch signature sits on top of this file in
 * include/compat/raymarcher.h + csrc/rrt_compat.cu (see INTEGRATION.md).
 *
 * There is no CPU fallback: every compute entry point needs a CUDA device of compute capability
 * 10.0 and fails with RRT_ERR_NO_DEVICE / RRT_ERR_CUDA otherwise.
 */
#ifndef RRT_H
#define RRT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RRT_ABI_VERSION 1

/* ---- error codes -------------------------------------------------------------------------------- */
#define RRT_OK 0
#define RRT_ERR_BAD_ARG (-1)   /* NULL pointer, non-positive size, bad band, ... */
#define RRT_ERR_CUDA (-2)      /* a CUDA runtime call or the kernel failed; see rrt_last_error() */
#define RRT_ERR_NO_DEVICE (-3) /* no usable sm_100 device */
#define RRT_ERR_NOMEM (-4)
#define RRT_ERR_UNSUPPORTED (-6) /* a valid file this build does not decode (see rrt_image_load) */
#define RRT_ERR_IO (-5)        /* frame sink: open / write / close failed */

/* ---- parameter surface ---------------------------------------------------------------------------
 * The reference bakes these in as macros (include/config.h); here they are run-time fields with the
 * same names in lower case, defaults = the reference's values (rrt_default_params). */
typedef struct rrt_params {
    float spin_a;           /* SPIN_A            config.h:21  (reference ships 0.0f) */
    float event_horizon;    /* EVENT_HORIZON     config.h:29 */
    float isco_radius;      /* ISCO_RADIUS       config.h:33 */
    float disk_out;         /* DISK_OUT_M        config.h:34 */
    float disk_h;           /* DISK_H_M          config.h:35 */
    float disk_luminosity;  /* DISK_LUMINOSITY   config.h:36 */
    float disk_opacity;     /* DISK_OPACITY      config.h:37 */
    float exposure;         /* EXPOSURE          config.h:38 */
    float cloud_h;          /* CLOUD_H_M         config.h:41 */
    float cloud_out;        /* CLOUD_OUT_M       config.h:42 */
    float cloud_opacity;    /* CLOUD_OPACITY     config.h:43 */
    float cloud_luminosity; /* CLOUD_LUMINOSITY  config.h:44 */
    float step_size;        /* STEP_SIZE_M       config.h:47 */
    float disk_temp_ref;    /* DISK_TEMP_REF     config.h:18 */
    int32_t max_steps;      /* MAX_STEPS         config.h:48 */
    uint32_t flags;         /* RRT_FLAG_* */
} rrt_params;

#define RRT_FLAG_DISK 1u /* accretion-disk medium  (getAccretionDensity, raymarcher.cu:68) */
#define RRT_FLAG_DUST 2u /* dust-cloud medium      (getDustCloudDensity, raymarcher.cu:69) */
/* Rounding contract.  Default (flag clear): every a*b+c is a rounded multiply followed by a rounded add --
 * the reference's expressions without contraction, bit-identical to its headers compiled for a host with
 * -ffp-contract=off.  RRT_FLAG_FMAD: the arithmetic of the reference's OWN CUDA build -- nvcc's default
 * -fmad=true fuses a*b+c into FMA, and the geodesic / ray-setup / noise code follows, operation by operation,
 * the fusion schedule nvcc 12.9 emits for the reference's sources on sm_100a (see DESIGN.md "Rounding
 * contracts"); ~1.3x fewer FP32 instructions per RK4 step. */
#define RRT_FLAG_FMAD 4u

/* struct CameraState, include/raymarcher.h:11-16: four packed float3, 48 bytes. */
typedef struct rrt_camera {
    float pos[3], forward[3], right[3], up[3];
} rrt_camera;

/* struct CameraEffects, include/camera_effects/camera_settings.h:4-17, as plain C (bool -> int32). */
typedef struct rrt_effects {
    int32_t use_bloom;
    float bloom_threshold, bloom_intensity;
    int32_t use_vignette;
    float vignette_intensity;
    int32_t use_ca;
    float ca_amount;
    int32_t use_lens;
    float distortion_amount;
} rrt_effects;

/* Row-band ownership for multi-GPU frames: image rows are cut into groups of `group` consecutive
 * rows and group k belongs to rank (k % nranks).  NULL / {0,1,1} = the whole frame. */
typedef struct rrt_band {
    int32_t rank, nranks, group;
} rrt_band;

/* Optional per-pixel DEVICE planes for parity checking, indexed [y*w + x] (not row-flipped).
 * Any pointer may be NULL.  float planes are float4 per pixel (16-byte aligned, coalesced). */
typedef struct rrt_planes {
    float* hdr;     /* final_hdr.rgb before camera effects (raymarcher.cu:148-150), w = transmittance */
    float* dir;     /* normalize(vel) at exit (raymarcher.cu:129); zeros for captured rays */
    float* emis;    /* accumulated emission I.rgb (raymarcher.cu:111-113) */
    float* pos;     /* final position */
    float* vel;     /* final (un-normalised) velocity */
    uint8_t* cls;   /* RRT_CLS_* | RRT_CLSF_* */
    int32_t* steps; /* RK4 steps taken */
} rrt_planes;

#define RRT_CLS_CAPTURED 0u /* r < 1.01*EVENT_HORIZON (raymarcher.cu:47-51) */
#define RRT_CLS_DISK_HIT 1u /* not captured and >= 1 sample passed the 0.001 density gate (raymarcher.cu:71) */
#define RRT_CLS_ESCAPED 2u  /* not captured, no medium touched */
#define RRT_CLS_MASK 3u
#define RRT_CLSF_EXHAUSTED 4u /* ran MAX_STEPS iterations (raymarcher.cu:41) */
#define RRT_CLSF_TOUCHED 8u

typedef struct rrt_counters {
    uint64_t rk4_steps;     /* integrate_rk4 calls -- the unit of the headline metric */
    uint64_t disk_evals;    /* disk-density evaluations */
    uint64_t dust_evals;    /* dust-density evaluations */
    uint64_t dense_samples; /* samples past the 0.001 gate */
    uint64_t n_captured, n_escaped, n_exhausted, n_touched;
} rrt_counters;

/* where the uchar4 pixels go */
#define RRT_OUT_FRAME 0  /* d_out is the full w*h frame; pixel (x,y) -> [(h-1-y)*w + x] as raymarcher.cu:168 */
#define RRT_OUT_PACKED 1 /* d_out holds only this band's rows, local row l -> [l*w + x], not flipped */

typedef struct rrt_context rrt_context; /* per-device scratch: counters, staging, default stream */
typedef struct rrt_sky rrt_sky;         /* cudaArray + texture object */

/* ---- lifetime ----------------------------------------------------------------------------------- */
int rrt_abi_version(void);
const char* rrt_build_info(void);                      /* arch + flags the library was compiled with */
int rrt_context_create(int device, rrt_context** out); /* device = CUDA ordinal */
void rrt_context_destroy(rrt_context* ctx);
const char* rrt_last_error(const rrt_context* ctx);    /* ctx may be NULL: last create failure */

void rrt_default_params(rrt_params* out);   /* the values of include/config.h */
void rrt_default_effects(rrt_effects* out); /* the default member initialisers of CameraEffects */

/* ---- skybox: replaces loadSkybox's device half, src/main.cpp:246-263 ----------------------------- */
/* RGBA8 rows top-down, exactly what stbi_load(...,4) returns; builds a cudaArray and a texture object
 * with addressMode {Wrap, Clamp}, linear filter, normalised-float read, normalised coordinates. */
int rrt_sky_create(rrt_context* ctx, const uint8_t* host_rgba, int w, int h, rrt_sky** out);
uint64_t rrt_sky_texture(const rrt_sky* sky); /* the cudaTextureObject_t, usable with launch_raymarch */

/* ---- skybox files: the host half of loadSkybox (src/main.cpp:237-245) ---------------------------------------------
 * The reference decodes its skybox with stbi_load(path, &w, &h, &c, 4) (stb_image v2.30, vendored there).  These entry
 * points decode PNG and baseline JPEG natively and return the SAME RGBA8 bytes stb_image returns for the file (for JPEG
 * that means stb_image's integer IDCT, chroma upsampling filters and fixed-point YCbCr->RGB, see csrc/rrt_image.cpp),
 * so a frame rendered from a file is the frame the reference renders from it.  Files outside that subset (progressive
 * or CMYK JPEG, 16-bit or interlaced PNG, other formats) fail with RRT_ERR_UNSUPPORTED; unreadable or corrupt files
 * with RRT_ERR_IO; the message is in rrt_image_last_error().  Pure host code, no device needed.
 * rrt_image_load / rrt_image_decode allocate *rgba (w*h*4 bytes, top row first); release it with rrt_image_free.
 * rrt_sky_load = rrt_image_load + rrt_sky_create (the whole loadSkybox). */
int rrt_image_load(const char* path, uint8_t** rgba, int* w, int* h);
int rrt_image_decode(const uint8_t* data, size_t size, uint8_t** rgba, int* w, int* h);
void rrt_image_free(uint8_t* rgba);
const char* rrt_image_last_error(void);
int rrt_sky_load(rrt_context* ctx, const char* path, rrt_sky** out);
void rrt_sky_destroy(rrt_sky* sky);

/* ---- the hot path: replaces launch_raymarch / raymarch_kernel ------------------------------------ */
/* Asynchronous on `stream` (a cudaStream_t; NULL = the legacy default stream, like the reference).
 * d_out: device uchar4 buffer (layout per out_layout).  planes: NULL or device planes.
 * RK4-step and class counters accumulate in the context until rrt_read_counters resets them. */
int rrt_render(rrt_context* ctx, const rrt_params* prm, const rrt_camera* cam, const rrt_effects* fx,
               uint64_t sky_texture, float time, int w, int h, const rrt_band* band, void* d_out, int out_layout,
               const rrt_planes* planes, void* stream);

/* Re-runs only the step after the ray loop (sky, final_hdr = I + bg*T, bloom, vignette, CA, tonemap, row-flipped store)
 * from the planes a previous rrt_render wrote: a new sky, exposure or bloom / vignette / CA setting without a new trace.
 * `traced` must carry vel, emis, hdr (only .w = T is read) and cls of that render, full-frame indexed [y*w + x] as
 * rrt_render writes them; other members are ignored.  Writes d_out (layout as in rrt_render, only the band's rows) and/or
 * hdr_out (float4 per pixel, full-frame indexed, the band's pixels only; may be traced->hdr itself).  Uses prm->exposure
 * and the contract bit prm->flags & RRT_FLAG_FMAD, and every rrt_effects field.  Asynchronous on `stream`; adds nothing
 * to the counters.
 * Contract: if the planes were written by rrt_render(P, cam, F, S, time, w, h, band, ...), then
 * rrt_shade(P', F', S', w, h, band, ...) writes exactly the bytes and hdr values of rrt_render(P*, cam, F*, S', time, w,
 * h, band, ...), where P* is P with P'.exposure and F* is F with the bloom, vignette and CA fields of F'.  This needs P'
 * to have the RRT_FLAG_FMAD bit of P and F' the use_lens / distortion_amount of F: those decide the rays and the
 * vignette's image-plane coordinate, and changing them needs a new trace. */
int rrt_shade(rrt_context* ctx, const rrt_params* prm, const rrt_effects* fx, uint64_t sky_texture, int w, int h,
              const rrt_band* band, const rrt_planes* traced, void* d_out, int out_layout, float* hdr_out, void* stream);

/* ---- supersampled (anti-aliased) frames: ss x ss rays per pixel, ss = 1 .. 8 --------------------------------------
 * Sub-sample (i, j) of output pixel (x, y) is pixel (ss*x + i, ss*y + j) of the ss*w x ss*h render with the same
 * parameters, camera, effects, sky and time, so its ray is that render's ray bit for bit (lens distortion and chromatic
 * aberration included: they act per sub-sample).  The pixel's linear final_hdr (and T, in .w) is the mean of its ss*ss
 * sub-samples, summed from (0,0) in row-major order (j outer, i inner) in round-to-nearest float32 and divided by
 * (float)(ss*ss); bloom, vignette (at the output pixel's own image-plane coordinate), exposure tonemap and the store
 * then run exactly as in rrt_render.  ss = 1 is rrt_render: same bytes, same hdr values.
 * Known shift: the sub-samples cover the pixel's footprint [x/w, (x+1)/w) while a 1-sample ray sits on its corner x/w,
 * so for ss > 1 the image moves by (ss-1)/(2*ss) of a pixel against a 1-sample render.  That is the price of being the
 * larger render exactly, which is what makes the result checkable bit for bit. */

/* Box-filters an ss*w x ss*h hdr plane (float4, [Y*ss*w + X], as rrt_render / rrt_shade write it) into a w x h frame:
 * mean of each ss x ss block in a fixed order, then bloom / vignette / tonemap / store exactly as rrt_render.
 * Writes d_out (layout as in rrt_render, only the band's rows) and/or hdr_out (float4 per pixel, w x h full-frame
 * indexed, the band's pixels only, the mean before bloom, like rrt_render's hdr plane); hdr_out must not overlap hdr_hi.
 * Reads only the sub-rows of the band's rows.  Uses prm->exposure and the contract bit prm->flags & RRT_FLAG_FMAD.
 * Asynchronous on `stream`; adds nothing to the counters and one launch.
 * Re-shading a supersampled frame: rrt_shade at ss*w x ss*h from the planes of rrt_render(ss*w, ss*h), with hdr_out
 * set to an ss*w x ss*h plane, followed by rrt_resolve of that plane, gives rrt_render_ss with the new sky, exposure and
 * effects. */
int rrt_resolve(rrt_context* ctx, const rrt_params* prm, const rrt_effects* fx, int ss, int w, int h,
                const rrt_band* band, const float* hdr_hi, void* d_out, int out_layout, float* hdr_out, void* stream);

/* rrt_render with ss x ss rays per pixel: traces the ss*w x ss*h frame into context-owned scratch (hdr plane only,
 * d_out = NULL, band {rank, nranks, ss*group}) and resolves it with rrt_resolve.  Same arguments as rrt_render plus ss;
 * planes other than the averaged hdr_out are not offered.
 * Band {r, N, g} traces band {r, N, ss*g} of the large frame: trace group (ss*y + j) / (ss*g) is y / g, so a rank traces
 * exactly the sub-rows of its own rows, and band-parallel frames (packed buffers or a peer frame) work as with rrt_render.
 * Scratch: one 16*ss*ss*w*h-byte plane per call (full-frame even for a band: 133 MB for 1920x1080 at ss = 2, 2.1 GB
 * for 3840x2160 at ss = 4), taken stream-ordered from a context-owned memory pool that keeps it for the next call, so
 * calls on different streams can be in flight together.  RRT_ERR_NOMEM, before anything is enqueued, when it cannot be
 * allocated.  Adds to the counters exactly what rrt_render(ss*w, ss*h) adds (they count sub-rays), and that render's
 * launches + 1 to rrt_kernel_launches. */
int rrt_render_ss(rrt_context* ctx, const rrt_params* prm, const rrt_camera* cam, const rrt_effects* fx,
                  uint64_t sky_texture, float time, int w, int h, int ss, const rrt_band* band,
                  void* d_out, int out_layout, float* hdr_out, void* stream);

/* ---- depth of field: each sub-sample of a supersampled pixel from its own camera --------------------------------------
 * rrt_render_ss with a HOST table cams[ss*ss] in place of cam.  Sub-sample (i, j) of output pixel (x, y) is pixel
 * (ss*x + i, ss*y + j) of rrt_render(P, cams[j*ss + i], F, S, time, ss*w, ss*h, band {r, N, ss*g}): its ray, step count,
 * media and sky are that render's bit for bit.  The pixel's hdr value (and T, in .w) is the mean of its ss*ss sub-samples,
 * summed and divided exactly as rrt_resolve does; bloom, vignette, tonemap and store then run exactly as in rrt_render.
 * So with every camera equal to cam it is rrt_render_ss(cam) (same bytes, same hdr values), and with ss = 1 it is
 * rrt_render(cams[0]); the (ss-1)/(2*ss)-pixel shift of rrt_render_ss applies unchanged.  With rrt_lens_cameras' table the
 * frame has the depth of field of a thin lens at the cost of rrt_render_ss: one trace of ss*ss rays per pixel.
 * Caveats of that lens: it is a flat-space thin lens at the camera; "in focus" is the plane at distance `focus` along
 * forward in the camera's local frame, before any bending of the rays; every pixel uses the same ss*ss lens points, so a
 * strongly defocused highlight (a star, the photon ring) shows as ss*ss discrete copies -- ss is the quality knob.
 * Bands, RRT_OUT_PACKED and a peer-frame d_out work as in rrt_render_ss; scratch, RRT_ERR_NOMEM and counters are
 * rrt_render_ss's (the camera table, 48*ss*ss bytes, rides in the same scratch block, copied on `stream`; the caller may
 * reuse its table as soon as the call returns); launches: the large trace's + 1.  RRT_ERR_BAD_ARG for a NULL table, a
 * non-finite camera field and everything rrt_render_ss refuses. */
int rrt_render_dof(rrt_context* ctx, const rrt_params* prm, const rrt_camera* cams, const rrt_effects* fx,
                   uint64_t sky_texture, float time, int w, int h, int ss, const rrt_band* band,
                   void* d_out, int out_layout, float* hdr_out, void* stream);

/* ---- panoramas: a 360 x 180 degree equirectangular frame -------------------------------------------------------------
 * Every direction around cam->pos in one w x h frame: column x is longitude lam = 2 pi ((x + 0.5) / w - 0.5) about up,
 * row y latitude phi = pi ((y + 0.5) / h - 0.5), and pixel (x, y) starts at cam->pos in the direction unit3(d), d being
 * rrt_pano_directions' vector of that pixel (forward at the centre, right at lam = pi/2, up at the top).  The contract:
 * pixel (x, y) of rrt_render_pano(P, cam, F, S, t, w, h, ss = 1) equals pixel (1, 1) of
 * rrt_render(P, {cam->pos, d, cam->right, cam->up}, F, S, t, 2, 2) -- whose ray is that same unit3(d) -- in cls, steps,
 * pos, vel, dir, emis and hdr, and in its byte when the vignette is off (the post step runs at pixel_uv (x/w, y/h): the
 * vignette darkens the panorama's edges as it does a pinhole frame's).  With the row-flipped RRT_OUT_FRAME store the
 * zenith is the first buffer row, the layout 360-degree players and environment maps expect.
 * ss = 1: rrt_render's pipeline choice, counters, launch count, bands, RRT_OUT_PACKED, peer-frame d_out and all seven planes.
 * ss = 2..8: the ss*w x ss*h panorama traced into scratch and resolved as rrt_render_ss does (band {r, N, ss*g}); only
 * planes->hdr, the w x h mean, is offered.  The result is bit for bit rrt_resolve(ss) of the hdr plane of
 * rrt_render_pano(ss*w, ss*h, ss = 1): the sub-samples are the cell centres of the large panorama, so unlike
 * rrt_render_ss there is no half-pixel shift.  Counters and launches: the large trace's, + 1 launch for the resolve.
 * The w + h (ss*w + ss*h) direction factors are computed on the host per call and copied on `stream` into a block of the
 * scratch pool (behind the supersampled plane when ss > 1); the caller's data is not involved.  Lens distortion has no
 * meaning here: RRT_ERR_BAD_ARG, before anything is enqueued, for fx->use_lens != 0, ss outside 1..8, a plane other than
 * hdr when ss > 1 and everything rrt_render / rrt_render_ss refuse; RRT_ERR_NOMEM when the scratch block cannot be had. */
int rrt_render_pano(rrt_context* ctx, const rrt_params* prm, const rrt_camera* cam, const rrt_effects* fx,
                    uint64_t sky_texture, float time, int w, int h, int ss, const rrt_band* band,
                    void* d_out, int out_layout, const rrt_planes* planes, void* stream);

/* ---- captures: one trace, renders at many times -------------------------------------------------------------------
 * With the camera fixed only the time moves, and the time enters only the disk and dust densities: trajectories, step
 * counts, classes and the positions of the media samples are the same at every time (a ray ends only at the horizon, on
 * escape or at max_steps).  A capture traces the frame once, keeps the media samples and the state of the rays the trace
 * finished, and renders it at any time by evaluating the media and folding them again, without a new trace.
 * Contract: let the capture be made from (P, cam, F, w, h, band).  rrt_capture_render(P', F', S', t, d_out, layout,
 * hdr_out) writes exactly the bytes and hdr values of rrt_render(P*, cam, F*, S', t, w, h, band, d_out, layout,
 * {hdr = hdr_out}), where P* is P with P'.exposure and F* is F with the bloom, vignette and CA fields of F' (the rules of
 * rrt_shade).  P' must carry P's RRT_FLAG_FMAD bit and F' F's use_lens / distortion_amount, else RRT_ERR_BAD_ARG; every
 * other field of P' is ignored (the capture keeps P).
 * Counters: rrt_capture_create adds the trace's (rk4 steps, disk / dust evaluations, classes); each render adds what
 * depends on the time (dense samples and touched rays of the folded rays) plus everything of the tiles the capture could
 * not hold, so the capture's counters plus one render's are those of one rrt_render.  Launches (rrt_kernel_launches):
 * 1 per capture; 3 per render (shade, media, fold), 4 when tiles were left to the fused sweep. */
typedef struct rrt_capture rrt_capture;
/* Traces the frame once (no time argument: the trace does not read it) and keeps what a later render needs.  The sky is
 * sampled by the trace but no render uses it.  Needs a medium (RRT_FLAG_DISK / RRT_FLAG_DUST; without one nothing depends
 * on the time: re-shade with rrt_shade) and a max_steps the split pipeline can describe; else RRT_ERR_BAD_ARG, as for the
 * arguments rrt_render refuses.  max_bytes: size of the sample pool the trace runs in (0: the context's sizing rule, as
 * rrt_render's pool, at most rrt_set_sample_pool's limit).  Tiles whose samples do not fit it are rendered by the fused
 * sweep at every render: correct for any max_bytes, fast when the frame fits.  Device memory held afterwards: the used
 * part of the pool (32 B per slot) plus 16 B of media results per slot, the queued ray groups, and four full-frame planes
 * of 49 B per pixel (vel, emis, hdr, cls; full-frame even for a band).  Synchronises `stream` (a cudaStream_t).
 * Destroy captures before their context. */
int rrt_capture_create(rrt_context* ctx, const rrt_params* prm, const rrt_camera* cam, const rrt_effects* fx,
                       uint64_t sky_texture, int w, int h, const rrt_band* band, size_t max_bytes, void* stream,
                       rrt_capture** out);
/* Evaluates the media at `time`, then folds, shades and stores: d_out (layout as in rrt_render, only the band's rows)
 * and/or hdr_out (float4 per pixel, full-frame indexed, the band's pixels only).  Asynchronous on `stream`.  One capture
 * serves one render at a time: each render waits for the capture's previous render, on whatever stream it was enqueued. */
int rrt_capture_render(rrt_capture* cap, const rrt_params* prm, const rrt_effects* fx, uint64_t sky_texture,
                       float time, void* d_out, int out_layout, float* hdr_out, void* stream);
/* [0] media samples kept, [1] pool slots held (32 B each), [2] device bytes held in all, [3] ray groups of 32 queued
 * for media + fold, [4] tiles left to the fused sweep (16x4 tiles for the packed tracer, else 8x4), [5] 1 if the
 * packed tracer traced it, [6] tiles of the frame (same unit as [4]), [7] bytes of the pool the trace ran in. */
int rrt_capture_info(const rrt_capture* cap, uint64_t out[8]);
void rrt_capture_destroy(rrt_capture* cap);

/* ---- motion-blurred frames: n sub-frames across the shutter interval, n = 1 .. 64 ---------------------------------
 * Sub-frame i has its own camera cams[i] and time times[i] (caller-supplied HOST arrays) and is exactly
 * rrt_render(P, cams[i], F, S, times[i], w, h, band, NULL, RRT_OUT_FRAME, {hdr = plane_i}): its ray, step count, media
 * and sky (chromatic aberration included) are that render's bit for bit.  The pixel's linear final_hdr (and T, in .w) is
 * the mean of the n planes, summed from plane 0 to plane n-1 in round-to-nearest float32 and divided by (float)n; bloom,
 * vignette (at the pixel's own image-plane coordinate: use_lens and distortion_amount are common to all sub-frames),
 * exposure tonemap and the store then run on the mean exactly as in rrt_render.  n = 1 is rrt_render: same bytes, same
 * hdr values.  rrt_shutter_times gives the times of a centred shutter.
 * Supersampled and motion-blurred: rrt_resolve_time at ss*w x ss*h with only hdr_out (an ss*w x ss*h plane), then
 * rrt_resolve(ss) of that plane, averages over time first and then over each pixel's ss x ss block. */

/* The time analogue of rrt_resolve: hdr_stack is n full-frame float4 planes back to back (plane i at i*w*h float4, each
 * [y*w + x] as rrt_render writes it).  Writes d_out (layout as in rrt_render, only the band's rows) and/or hdr_out (float4
 * per pixel, full-frame indexed, the band's pixels only, the mean before bloom); hdr_out must not overlap the stack.
 * Reads only the band's rows.  Uses prm->exposure and the contract bit prm->flags & RRT_FLAG_FMAD.  Asynchronous on
 * `stream`; adds nothing to the counters and one launch.  RRT_ERR_BAD_ARG for n outside 1..64, no output, a bad band or
 * layout, or a band of more than 2^30 pixels. */
int rrt_resolve_time(rrt_context* ctx, const rrt_params* prm, const rrt_effects* fx, int n, int w, int h, const rrt_band* band,
                     const float* hdr_stack, void* d_out, int out_layout, float* hdr_out, void* stream);

/* Renders the n sub-frames into a stack taken stream-ordered from the context's scratch pool (the one rrt_render_ss uses),
 * then rrt_resolve_time.  Same arguments as rrt_render with cams / times / n for cam / time, and hdr_out (the mean) for
 * the planes; bands, RRT_OUT_PACKED and a peer-frame d_out work as in rrt_render.  Scratch: 16*n*w*h bytes per call
 * (full-frame even for a band: 1.06 GB for 3840x2160 at n = 8); RRT_ERR_NOMEM, before anything is enqueued, when it
 * cannot be allocated.  Adds to the counters exactly what its n renders add, and their launches + 1. */
int rrt_render_mb(rrt_context* ctx, const rrt_params* prm, const rrt_camera* cams, const rrt_effects* fx, uint64_t sky_texture,
                  const float* times, int n, int w, int h, const rrt_band* band, void* d_out, int out_layout, float* hdr_out,
                  void* stream);

/* rrt_render_mb of a still camera through a capture: n rrt_capture_render calls into the stack (hdr only), then
 * rrt_resolve_time.  Writes exactly what rrt_render_mb writes with cams[i] = the capture's camera for every i, under
 * rrt_capture_render's rules: prm must carry the capture's RRT_FLAG_FMAD bit and fx its use_lens / distortion_amount, else
 * RRT_ERR_BAD_ARG; prm contributes only its exposure.  Waits for the capture's previous render once and is ordered before
 * its next one.  Scratch as rrt_render_mb.  Adds what n capture renders add to the counters; launches n * (3 or 4) + 1. */
int rrt_capture_render_mb(rrt_capture* cap, const rrt_params* prm, const rrt_effects* fx, uint64_t sky_texture, const float* times,
                          int n, void* d_out, int out_layout, float* hdr_out, void* stream);

/* Same call with a HOST destination: renders into a context-owned device frame, copies it to
 * host_rgba (w*h*4 bytes, reference layout) and synchronises.  This is the end-to-end entry point. */
int rrt_render_host(rrt_context* ctx, const rrt_params* prm, const rrt_camera* cam, const rrt_effects* fx,
                    uint64_t sky_texture, float time, int w, int h, uint8_t* host_rgba);

/* The same without the final synchronisation, for frame sequences (the recorder loop of src/main.cpp:505-528
 * renders frame after frame): enqueues the trace and the device->host copy on `stream` and returns.  `slot`
 * (0 .. RRT_HOST_SLOTS-1) picks the context-owned device frame, so that up to RRT_HOST_SLOTS frames can be in
 * flight on different streams; a slot may be reused once the work previously enqueued with it has completed
 * (stream order guarantees that when a slot is always used with the same stream).  host_rgba should be pinned
 * memory, otherwise the copy is staged and synchronous. */
#define RRT_HOST_SLOTS 4
int rrt_render_host_async(rrt_context* ctx, const rrt_params* prm, const rrt_camera* cam, const rrt_effects* fx,
                          uint64_t sky_texture, float time, int w, int h, uint8_t* host_rgba, int slot, void* stream);

/* How many rrt_render launches the caller keeps running concurrently on different streams (1 .. RRT_HOST_SLOTS,
 * default 1).  Each launch then occupies 1/n of the GPU's resident-CTA slots, so the n frames share the SMs from
 * the start instead of each filling the GPU and ending in a drain; results do not depend on it. */
int rrt_set_frames_in_flight(rrt_context* ctx, int n);

/* ---- render pipeline ------------------------------------------------------------------------------------------
 * A launch with a medium (RRT_FLAG_DISK / RRT_FLAG_DUST) can run as ONE fused kernel (every in-zone step evaluates
 * its media sample on the spot, like the reference's raymarch_kernel, src/raymarcher.cu:67-115) or SPLIT into three
 * kernels per pass over a sample pool in device memory: trace (trajectories; in-zone steps append their sample to the
 * pool), media (one thread per sample, densely packed) and fold (per ray, `I += e (1 - s) T; T *= s` in step order,
 * then background / effects / store).  Media samples do not feed back into the trajectory, so both produce the same
 * bits; the split form removes the frame's longest dependency chain (a disk-plane ray: 2000 x (step + both media))
 * and evaluates the media with every lane busy.  AUTO = split whenever a medium is on and the pool can be allocated.
 * RRT_PIPELINE=auto|fused|split in the environment sets the default of new contexts. */
#define RRT_PIPELINE_AUTO 0
#define RRT_PIPELINE_FUSED 1
#define RRT_PIPELINE_SPLIT 2
int rrt_set_pipeline(rrt_context* ctx, int mode);
/* Sample pool of the split pipeline: one pool per stream in flight (up to RRT_HOST_SLOTS), each at most
 * max_bytes_per_stream (default 16 GiB, RRT_POOL_MB; sized to the frame: 4 KiB per pixel plus ~2 MiB per resident tracing warp, at least 64 MiB).  A frame that
 * needs more is rendered in several passes (at most max_passes, default 32, RRT_MAX_PASSES; whatever is left after them
 * is rendered by the fused code), so any size gives the same frame.  0 leaves a value unchanged. */
int rrt_set_sample_pool(rrt_context* ctx, size_t max_bytes_per_stream, int max_passes);
/* Synchronises and reports the split pipeline's bookkeeping of the last frame that completed: [0] passes that traced
 * tiles, [1] tiles left to the closing fused sweep, [2] tiles traced by the passes, [3] passes enqueued, [4] tiles of
 * the launch, [5] pool size in Ki slots of 32 bytes; all 0 when no frame went through the split pipeline. */
int rrt_split_stats(rrt_context* ctx, uint32_t out[8]);
/* Kernels this context has launched so far for rrt_render*, rrt_shade, rrt_resolve*, rrt_capture_* and rrt_assemble_bands
 * (1 per fused frame; 3 per pass + 1 per split frame; 1 per rrt_shade, rrt_resolve or rrt_resolve_time; rrt_render_ss and
 * rrt_render_dof: their ss*w x ss*h render's + 1; rrt_render_pano: rrt_render's at ss = 1, its ss*w x ss*h render's + 1 at
 * ss > 1; rrt_render_mb: its n renders' + 1; 1 per rrt_capture_create, 3 or 4 per rrt_capture_render,
 * n * (3 or 4) + 1 per rrt_capture_render_mb):
 * what a benchmark reports as its launch count. */
uint64_t rrt_kernel_launches(rrt_context* ctx);

/* Number of rows a band owns in an h-row image (packed buffer height). */
int rrt_band_rows(const rrt_band* band, int h);

/* Scatter nranks packed band buffers (rank-major, each `rows_per_rank` rows of w uchar4) into the full
 * row-flipped frame -- the step after the NVLink gather on the encoding GPU. */
int rrt_assemble_bands(rrt_context* ctx, const void* d_packed, int rows_per_rank, int w, int h, int nranks,
                       int group, void* d_frame, void* stream);

/* ---- peer frames: the exchange step of a band-parallel frame without a gather --------------------------------
 * One process per GPU.  The encoding GPU's process (rank 0) creates the frame with rrt_peer_frame_create and hands
 * the 64-byte handle to the other processes (any channel: torch.distributed, a pipe ...); they map it with
 * rrt_peer_frame_open and pass the returned device pointer as d_out to rrt_render(band = their rows,
 * out_layout = RRT_OUT_FRAME).  The render kernel then stores each finished pixel straight into rank 0's row-flipped
 * frame over NVLink (4 B per ~220 kFLOP of tracing): no packed buffer, no NCCL gather, no rrt_assemble_bands --
 * the store that ends the path (src/raymarcher.cu:168) IS the exchange (the reference's exchange point is the mapped
 * PBO, src/main.cpp:463-469).  Ordering is the caller's: a stream-ordered barrier across the ranks (e.g. a 4-byte
 * NCCL all-reduce enqueued after the render) tells rank 0 that every band has landed.
 * CUDA IPC: processes must differ (a handle cannot be opened by the process that created it). */
#define RRT_PEER_HANDLE_BYTES 64
int rrt_peer_frame_create(rrt_context* ctx, size_t bytes, void** d_frame, uint8_t handle[RRT_PEER_HANDLE_BYTES]);
int rrt_peer_frame_open(rrt_context* ctx, const uint8_t handle[RRT_PEER_HANDLE_BYTES], void** d_frame);
/* Stream-ordered copy of a peer frame (or any device buffer) to `dst`, which may be pinned host memory or device
 * memory (cudaMemcpyDefault): how rank 0 hands the assembled frame on without wrapping the raw allocation. */
int rrt_peer_frame_read(rrt_context* ctx, const void* d_frame, size_t bytes, void* dst, void* stream);
/* owner != 0: the creating process frees the frame; owner == 0: a mapping process unmaps it */
int rrt_peer_frame_close(rrt_context* ctx, void* d_frame, int owner);

/* Synchronises the context's work, copies the counters out and optionally zeroes them. */
int rrt_read_counters(rrt_context* ctx, rrt_counters* out, int reset);

/* ---- function-level probes (HOST arrays in, HOST arrays out; float3 packed xyz) -------------------
 * Device implementations of the interfaces north_star names, callable one function at a time so each
 * can be checked against the oracle:
 *   getGeodesicAcc          geodesics.h:30-45        integrate_rk4   integrators.h:23-59
 *   calculateRedshiftFactor geodesics.h:11-25        integrate_euler integrators.h:12-18
 *   hash31/noise3D/fbm      math_utils.h:91-121      getDiskTemperature / getAccretionDensity /
 *   tex2D<float4>           raymarcher.cu:139        getDustCloudDensity  densities.h:12-132 */
int rrt_geodesic_acc_batch(rrt_context* ctx, const rrt_params* prm, int n, const float* q, const float* v, float* out);
int rrt_rk4_step_batch(rrt_context* ctx, const rrt_params* prm, int n, float* p, float* v, const float* h);
int rrt_euler_step_batch(rrt_context* ctx, const rrt_params* prm, int n, float* p, float* v, const float* h);
int rrt_redshift_batch(rrt_context* ctx, const rrt_params* prm, int n, const float* q, const float* v, float* out);
int rrt_hash31_batch(rrt_context* ctx, int n, const float* p, float* out);
int rrt_noise3d_batch(rrt_context* ctx, int n, const float* p, float* out);
int rrt_fbm_batch(rrt_context* ctx, int n, const float* p, int octaves, float* out);
int rrt_disk_temperature_batch(rrt_context* ctx, const rrt_params* prm, int n, const float* r, float* out);
int rrt_disk_density_batch(rrt_context* ctx, const rrt_params* prm, int n, const float* q, float time, float* out);
int rrt_dust_density_batch(rrt_context* ctx, const rrt_params* prm, int n, const float* q, float time, float* out);
int rrt_sky_sample_batch(rrt_context* ctx, uint64_t sky_texture, int n, const float* tx, const float* ty, float* out4);

/* ---- host camera + keyframe paths: the step before the hot path ---------------------------------------
 * Pure host code (no device needed).  rrt_camera_from replaces CameraController::getCUDAStateFrom
 * (src/main.cpp:141-167; angles in degrees, the reference's 3.14159f and float sinf/cosf).
 * rrt_path_state replaces PathController::getInterpolatedState (src/main.cpp:176-203) over the three
 * built-in keyframe tables of initDefaultPaths (src/camera_paths.cpp:31-73) with catmull_rom (:6-22) and
 * lerp_angle (:25-29).  rrt_path_clock reproduces the recorder's fixed clock: pathTime after `frame`
 * float accumulations of 1.0f/fps (src/main.cpp:511-516, 210-212). */
void rrt_camera_from(const float pos[3], float yaw_deg, float pitch_deg, rrt_camera* out);
int rrt_path_count(void);
const char* rrt_path_name(int path_index);
int rrt_path_num_keys(int path_index);
float rrt_path_duration(int path_index);
int rrt_path_state(int path_index, float t, rrt_camera* out, float pos_yaw_pitch[5]);
float rrt_path_clock(int frame, float fps);
/* The n sub-frame times of a shutter open for `shutter` (0 .. 1) of the frame interval 1/fps, centred on t:
 * d = shutter / fps, out[i] = t + d * ((i + 0.5f) / n - 0.5f), every operation rounded to float32 on its own (no
 * contraction).  n = 1 gives t and shutter = 0 gives t n times (a t of -0 may come back as +0).  RRT_ERR_BAD_ARG for shutter outside
 * [0, 1], fps <= 0, n outside 1..64 or out NULL. */
int rrt_shutter_times(float t, float shutter, float fps, int n, float* out);
/* The ss*ss cameras of a thin lens of radius `aperture` at cam->pos, focused on the plane at distance `focus` along
 * cam->forward (rrt_render_dof's table).  Lens sample k = j*ss + i is the centre of stratified cell (i, j),
 * (a, b) = (2(i+0.5)/ss - 1, 2(j+0.5)/ss - 1), mapped to the unit disk by Shirley & Chiu's concentric map ((0, 0) -> (0, 0))
 * and scaled by aperture: (ox, oy), the map evaluated in double precision and rounded to float32 once.  Camera k then is,
 * per component c and every operation rounded to float32 on its own (no contraction):
 *   o = right[c] * ox + up[c] * oy      (both products first, then the sum)
 *   pos[c] = cam->pos[c] + o,   forward[c] = cam->forward[c] - o / focus,   right and up unchanged.
 * Its ray for image-plane coordinate (u, v) passes through cam->pos + focus * (forward + right*u + up*v) for every lens
 * point, so that plane is sharp.  aperture == 0, ss == 1 and the centre cell of an odd ss give exact copies of *cam.
 * RRT_ERR_BAD_ARG for aperture < 0 or non-finite, focus <= 0 or non-finite, ss outside 1..8, or a NULL pointer.
 * out holds ss*ss cameras. */
int rrt_lens_cameras(const rrt_camera* cam, float aperture, float focus, int ss, rrt_camera* out);

/* The un-normalised direction of every pixel of a w x h rrt_render_pano frame: out[(y*w + x)*3 + c] = d[c].  With
 * lam = 2 pi ((x + 0.5) / w - 0.5) and phi = pi ((y + 0.5) / h - 0.5) evaluated in double (as pi (2x + 1 - w) / w and
 * pi/2 (2y + 1 - h) / h, so that mirrored columns and rows get exactly opposite angles) and (cos, sin) of each rounded to
 * float32 once, per component c and every operation rounded to float32 on its own (no contraction) in this order:
 *   a = cos phi * cos lam,   b = cos phi * sin lam,   d[c] = (a * forward[c] + b * right[c]) + sin phi * up[c].
 * The panorama's ray of that pixel is unit3(d) from cam->pos.  No orthonormality of the camera is assumed.
 * RRT_ERR_BAD_ARG for a NULL pointer, w or h <= 0, or w*h*3 floats beyond the address space. */
int rrt_pano_directions(const rrt_camera* cam, int w, int h, float* out);

/* ---- frame sink: the step after the hot path ----------------------------------------------------------
 * Pure host code.  Replaces, for headless use, the reference's ScreenRecorder (src/main.cpp:29-124): frames
 * are the host copies of what launch_raymarch / rrt_render_host wrote (w*h*4 bytes, buffer row 0 first --
 * which is what the recorder's glReadPixels returns for the 1:1 quad it draws).
 *   RRT_SINK_RGBA  the recorder's wire format byte for byte: raw rgba frames back to back (src/main.cpp:85-97).
 *                  With target "|<command>" the stream is popen()ed exactly like the reference does; the
 *                  reference's own command line is produced by rrt_sink_ffmpeg_command (src/main.cpp:61-72).
 *   RRT_SINK_Y4M   YUV4MPEG2 4:2:0 (BT.601 studio range), rows already flipped as `-vf vflip` would: a
 *                  self-describing file for boxes without ffmpeg.
 * target: a file path, or "|command". */
#define RRT_SINK_RGBA 0
#define RRT_SINK_Y4M 1
typedef struct rrt_sink rrt_sink;
int rrt_sink_open(const char* target, int format, int w, int h, int fps, rrt_sink** out);
int rrt_sink_write(rrt_sink* sink, const uint8_t* host_rgba);
int rrt_sink_frames(const rrt_sink* sink);          /* frames written so far */
int rrt_sink_close(rrt_sink* sink);                 /* RRT_ERR_IO if the file / pipe reported an error */
/* writes the reference recorder's ffmpeg command for this size into buf; returns its length or RRT_ERR_BAD_ARG */
int rrt_sink_ffmpeg_command(int w, int h, int fps, const char* out_name, char* buf, int buflen);

/* ---- measurement helper ---------------------------------------------------------------------------
 * Register-resident FFMA-chain microbenchmark: the FP32 roofline denominator MEASURED_PEAKS.json lacks.
 * Returns achieved FP32 TFLOP/s (2 flop per FFMA) over `iters` dependent-chain iterations. */
int rrt_fp32_peak_probe(rrt_context* ctx, int iters, double* tflops, double* ms);

/* Self-test of the branch-free correctly-rounded division / square root the render loop uses
 * (include/rrt_device.cuh: div_rn_fast, sqrt_rn_fast) against the IEEE intrinsics __fdiv_rn / __fsqrt_rn, on
 * `n` pseudo-random operand pairs drawn on the device from the loop's operand domain.  Outputs the number
 * of results that differ in value (expected: 0 and 0). */
int rrt_exact_math_selftest(rrt_context* ctx, uint64_t seed, uint64_t n, uint64_t* div_mismatches,
                            uint64_t* sqrt_mismatches);

/* Profiling aid: while d_log is non-NULL every render launch of this context writes, per 8x4-pixel tile (index =
 * the tile's ticket, tiles beyond `entries` are skipped), four uint64: %globaltimer at the start and at the end of the
 * tile (ns), (tile_row << 32 | tile_col), (sm_id << 32 | steps of the tile's longest ray).  d_log is a caller-owned device
 * buffer of entries * 32 bytes; pass NULL to switch the log off.  Only libraries built with -DRRT_WITH_TILE_LOG
 * (`make -C csrc timeline` -> build/timeline/librrt_b200_timeline.so) carry the instrumentation -- its extra live values
 * cost the step loop ~3 % through register allocation, so the product library returns RRT_ERR_UNSUPPORTED for a non-NULL
 * log.  Used by tools/tile_timeline.py to see what a launch's tail consists of. */
int rrt_debug_tile_log(rrt_context* ctx, void* d_log, size_t entries);

/* Self-test of the media code's split powf (include/rrt_device.cuh: pow_log2 + pow_exp2, libdevice's own algorithm cut
 * where the exponent enters so that one log2 serves several powers of the same base) against libdevice's powf on `n`
 * pseudo-random positive normal bases, with the exponents the media code uses and with random exponents.  Outputs the
 * number of results that differ in any bit (expected: 0 and 0). */
int rrt_exact_pow_selftest(rrt_context* ctx, uint64_t seed, uint64_t n, uint64_t* used_exponent_mismatches,
                           uint64_t* random_exponent_mismatches);

/* Rounding contract of the probes that take no rrt_params (hash31 / noise3D / fbm): 1 the RRT_FLAG_FMAD contract
 * (default, like rrt_default_params), 0 strict.  The other probes and rrt_render follow rrt_params.flags. */
int rrt_set_probe_contract(rrt_context* ctx, int fmad);

#ifdef __cplusplus
}
#endif
#endif /* RRT_H */
