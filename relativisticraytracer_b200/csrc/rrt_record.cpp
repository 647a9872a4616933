// rrt_record -- headless recorder: the reference's "P then R" session (camera-path playback under the recorder's
// fixed 1/24 s clock, src/main.cpp:171-220, 505-528) without a window, written against the C ABI only.
//
//   rrt_record <path 0..2> <frames> <width> <height> <target> [--spin a] [--y4m] [--pano] [--sky file.png|file.jpg] [--sky-raw file.rgba W H] [--device n]
//
// <target> is a file, or "|command" (e.g. the string rrt_sink_ffmpeg_command returns) which is popen()ed like the
// reference's recorder does.  Two frames are kept in flight (rrt_render_host_async on two streams, pinned host
// frames); frames reach the sink in order.  --sky decodes the file exactly like the reference's loadSkybox does
// (rrt_sky_load: the bytes stb_image returns, src/main.cpp:237-266); without a sky a smooth procedural RGBA8 map is used.
// --pano records 360-degree video: every frame is the width x height equirectangular panorama around the path camera
// (rrt_render_pano into a device frame, then a stream-ordered copy to the pinned host frame), with the default effects
// less lens distortion and vignette, which belong to a flat picture.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/rrt.h"

#define CHECK(call)                                                                            \
    do {                                                                                       \
        int rc__ = (call);                                                                     \
        if (rc__ != 0) {                                                                       \
            std::fprintf(stderr, "%s failed: %d (%s)\n", #call, rc__, rrt_last_error(ctx));    \
            return 1;                                                                          \
        }                                                                                      \
    } while (0)

int main(int argc, char** argv) {
    if (argc < 6) {
        std::fprintf(stderr, "usage: %s <path 0..%d> <frames> <width> <height> <target> [--spin a] [--y4m] [--pano] [--sky f.png|f.jpg] [--sky-raw f.rgba W H] [--device n]\n",
                     argv[0], rrt_path_count() - 1);
        return 2;
    }
    const int path = std::atoi(argv[1]), frames = std::atoi(argv[2]), w = std::atoi(argv[3]), h = std::atoi(argv[4]);
    const char* target = argv[5];
    float spin = 0.0f;  // SPIN_A of the reference's config.h
    int format = RRT_SINK_RGBA, device = 0, sky_w = 1024, sky_h = 512;
    const char* sky_file = nullptr;   // headerless RGBA8
    const char* sky_image = nullptr;  // PNG / JPEG, decoded by rrt_sky_load
    bool pano = false;
    for (int i = 6; i < argc; ++i) {
        if (!std::strcmp(argv[i], "--spin") && i + 1 < argc) spin = (float)std::atof(argv[++i]);
        else if (!std::strcmp(argv[i], "--y4m")) format = RRT_SINK_Y4M;
        else if (!std::strcmp(argv[i], "--pano")) pano = true;
        else if (!std::strcmp(argv[i], "--device") && i + 1 < argc) device = std::atoi(argv[++i]);
        else if (!std::strcmp(argv[i], "--sky") && i + 1 < argc) sky_image = argv[++i];
        else if (!std::strcmp(argv[i], "--sky-raw") && i + 3 < argc) { sky_file = argv[i + 1]; sky_w = std::atoi(argv[i + 2]); sky_h = std::atoi(argv[i + 3]); i += 3; }
        else { std::fprintf(stderr, "unknown option %s\n", argv[i]); return 2; }
    }
    if (path < 0 || path >= rrt_path_count() || frames <= 0 || w <= 0 || h <= 0 || sky_w <= 0 || sky_h <= 0) return 2;

    rrt_context* ctx = nullptr;
    if (int rc = rrt_context_create(device, &ctx)) {
        std::fprintf(stderr, "rrt_context_create: %d (%s)\n", rc, rrt_last_error(nullptr));
        return 1;
    }
    rrt_sky* sky = nullptr;
    std::vector<uint8_t> sky_px(sky_image ? 0 : (size_t)sky_w * sky_h * 4);
    if (sky_image) {
        if (int rc = rrt_sky_load(ctx, sky_image, &sky)) {
            std::fprintf(stderr, "rrt_sky_load(%s): %d (%s)\n", sky_image, rc, rc == RRT_ERR_CUDA ? rrt_last_error(ctx) : rrt_image_last_error());
            return 1;
        }
    } else if (sky_file) {
        FILE* f = std::fopen(sky_file, "rb");
        if (!f || std::fread(sky_px.data(), 1, sky_px.size(), f) != sky_px.size()) { std::fprintf(stderr, "cannot read %s\n", sky_file); return 1; }
        std::fclose(f);
    } else {
        for (int y = 0; y < sky_h; ++y)
            for (int x = 0; x < sky_w; ++x) {
                const float u = (x + 0.5f) / sky_w, v = (y + 0.5f) / sky_h;
                uint8_t* p = &sky_px[((size_t)y * sky_w + x) * 4];
                p[0] = (uint8_t)(255 * (0.30f + 0.20f * std::sin(6.2831853f * u) * std::sin(3.1415927f * v)));
                p[1] = (uint8_t)(255 * (0.28f + 0.18f * std::cos(6.2831853f * u + 1.0f) * std::sin(3.1415927f * v) * std::sin(3.1415927f * v)));
                p[2] = (uint8_t)(255 * (0.40f + 0.25f * std::cos(3.1415927f * v) * std::cos(12.566371f * u)));
                p[3] = 255;
            }
    }
    if (!sky) CHECK(rrt_sky_create(ctx, sky_px.data(), sky_w, sky_h, &sky));
    rrt_params prm;
    rrt_default_params(&prm);
    prm.spin_a = spin;
    rrt_effects fx;
    rrt_default_effects(&fx);
    if (pano) fx.use_lens = fx.use_vignette = 0;
    rrt_sink* sink = nullptr;
    if (int rc = rrt_sink_open(target, format, w, h, 24, &sink)) { std::fprintf(stderr, "rrt_sink_open(%s): %d\n", target, rc); return 1; }

    constexpr int kInFlight = 2;
    cudaSetDevice(device);
    cudaStream_t st[kInFlight];
    uint8_t* host[kInFlight];
    void* dev[kInFlight] = {};   // --pano: the device frame of each slot
    for (int k = 0; k < kInFlight; ++k) {
        if (cudaStreamCreateWithFlags(&st[k], cudaStreamNonBlocking) != cudaSuccess ||
            cudaMallocHost((void**)&host[k], (size_t)w * h * 4) != cudaSuccess ||
            (pano && cudaMalloc(&dev[k], (size_t)w * h * 4) != cudaSuccess)) { std::fprintf(stderr, "CUDA stream / frame allocation failed\n"); return 1; }
    }
    auto submit = [&](int frame) {   // frames are 1-based, like the recorder counts them
        const float t = rrt_path_clock(frame, 24.0f);                     // src/main.cpp:511-516
        rrt_camera cam;
        if (int rc = rrt_path_state(path, t, &cam, nullptr)) return rc;   // src/main.cpp:176-203
        const int k = frame % kInFlight;
        if (pano) {
            if (int rc = rrt_render_pano(ctx, &prm, &cam, &fx, rrt_sky_texture(sky), t, w, h, 1, nullptr, dev[k], RRT_OUT_FRAME, nullptr, st[k]))
                return rc;
            return cudaMemcpyAsync(host[k], dev[k], (size_t)w * h * 4, cudaMemcpyDeviceToHost, st[k]) == cudaSuccess ? 0 : RRT_ERR_CUDA;
        }
        return rrt_render_host_async(ctx, &prm, &cam, &fx, rrt_sky_texture(sky), /*simTime*/ t, w, h, host[k], k, st[k]);
    };
    for (int f = 1; f <= frames && f <= kInFlight; ++f) CHECK(submit(f));
    for (int f = 1; f <= frames; ++f) {
        const int k = f % kInFlight;
        if (cudaStreamSynchronize(st[k]) != cudaSuccess) { std::fprintf(stderr, "frame %d failed: %s\n", f, cudaGetErrorString(cudaGetLastError())); return 1; }
        CHECK(rrt_sink_write(sink, host[k]));
        if (f + kInFlight <= frames) CHECK(submit(f + kInFlight));
    }
    rrt_counters cnt;
    CHECK(rrt_read_counters(ctx, &cnt, 1));
    const int written = rrt_sink_frames(sink);
    CHECK(rrt_sink_close(sink));
    std::printf("%d frames %dx%d of \"%s\" -> %s   (%llu RK4 steps)\n", written, w, h, rrt_path_name(path), target,
                (unsigned long long)cnt.rk4_steps);
    for (int k = 0; k < kInFlight; ++k) { cudaFreeHost(host[k]); if (dev[k]) cudaFree(dev[k]); cudaStreamDestroy(st[k]); }
    rrt_sky_destroy(sky);
    rrt_context_destroy(ctx);
    return 0;
}
