// rrt_host.cpp -- host-side camera math and keyframe paths behind the C ABI (include/rrt.h).
//
// This is the step immediately before the hot path: it turns (position, yaw, pitch) or a path time
// into the CameraState the render kernel consumes.  It replaces, for headless use, the pieces of the
// reference that live in its GLFW application: CameraController::getCUDAStateFrom (src/main.cpp:141-167),
// PathController::getInterpolatedState (src/main.cpp:176-203) and the spline/angle helpers and keyframe
// tables of src/camera_paths.cpp.  Built with -ffp-contract=off: every operation is one binary32 op in
// the reference's order, so the basis vectors are bit-identical to the reference's on the same libm.
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/rrt.h"

namespace {

struct Vec { float x, y, z; };
struct Key { float t; Vec pos; float yaw, pitch; };
struct Path { const char* name; const Key* keys; int n; };

// src/camera_paths.cpp:33-72
const Key kGargantua[] = {
    {0.0f, {0.0f, 15.0f, -80.0f}, 0.0f, -10.6f},
    {6.0f, {15.0f, 3.0f, -30.0f}, -26.6f, -5.1f},
    {12.0f, {35.0f, 0.8f, 10.0f}, -106.0f, -1.2f},
    {18.0f, {5.0f, 1.5f, 50.0f}, -174.3f, -1.7f},
    {25.0f, {-20.0f, 12.0f, 70.0f}, -196.0f, -9.3f},
};
const Key kHorizonFocus[] = {
    {0.0f, {40.0f, 2.0f, 0.0f}, -90.0f, 0.0f},
    {8.0f, {0.0f, 5.0f, 40.0f}, -180.0f, -5.0f},
    {16.0f, {-40.0f, 2.0f, 0.0f}, -270.0f, 0.0f},
    {24.0f, {0.0f, -5.0f, -40.0f}, -360.0f, 5.0f},
    {32.0f, {40.0f, 2.0f, 0.0f}, -450.0f, 0.0f},
};
const Key kSkimmer[] = {
    {0.0f, {0.0f, 10.0f, -60.0f}, 0.0f, -9.5f},
    {8.0f, {15.0f, 2.0f, -15.0f}, -45.0f, -4.7f},
    {14.0f, {4.2f, 0.6f, 4.2f}, -90.0f, -5.7f},
    {20.0f, {-20.0f, 8.0f, -20.0f}, -225.0f, -20.0f},
    {26.0f, {-20.0f, 8.0f, -20.0f}, 20.0f, -10.0f},
    {29.0f, {-30.0f, 2.0f, -30.0f}, 45.0f, -2.7f},
};
const Path kPaths[] = {
    {"Gargantua Fly-By", kGargantua, 5},
    {"Event Horizon Focus", kHorizonFocus, 5},
    {"Horizon Skimmer", kSkimmer, 6},
};
constexpr int kNumPaths = 3;

// uniform Catmull-Rom, one coordinate (src/camera_paths.cpp:10-15)
float spline(float a, float b, float c, float d, float t, float t2, float t3) {
    return 0.5f * ((2.0f * b) + (-a + c) * t + (2.0f * a - 5.0f * b + 4.0f * c - d) * t2 +
                   (-a + 3.0f * b - 3.0f * c + d) * t3);
}

// shortest-arc interpolation in degrees (src/camera_paths.cpp:25-29)
float mix_angle(float a, float b, float t) {
    float diff = std::fmod(b - a + 180.0f, 360.0f) - 180.0f;
    if (diff < -180.0f) diff += 360.0f;
    return a + diff * t;
}

void basis_from(Vec pos, float yaw, float pitch, rrt_camera* out) {
    const float ry = yaw * 3.14159f / 180.0f;  // the reference's 5-digit pi (src/main.cpp:142-143)
    const float rp = pitch * 3.14159f / 180.0f;
    Vec f = {std::sin(ry) * std::cos(rp), std::sin(rp), std::cos(ry) * std::cos(rp)};
    const float fm = std::sqrt(f.x * f.x + f.y * f.y + f.z * f.z);
    f.x /= fm; f.y /= fm; f.z /= fm;
    const Vec wu = {0.0f, 1.0f, 0.0f};
    Vec r = {wu.y * f.z - wu.z * f.y, wu.z * f.x - wu.x * f.z, wu.x * f.y - wu.y * f.x};
    const float rm = std::sqrt(r.x * r.x + r.y * r.y + r.z * r.z);
    r.x /= rm; r.y /= rm; r.z /= rm;
    const Vec u = {f.y * r.z - f.z * r.y, f.z * r.x - f.x * r.z, f.x * r.y - f.y * r.x};  // not renormalised
    out->pos[0] = pos.x; out->pos[1] = pos.y; out->pos[2] = pos.z;
    out->forward[0] = f.x; out->forward[1] = f.y; out->forward[2] = f.z;
    out->right[0] = r.x; out->right[1] = r.y; out->right[2] = r.z;
    out->up[0] = u.x; out->up[1] = u.y; out->up[2] = u.z;
}

}  // namespace

namespace rrtk {
// rrt_render_pano's device table and rrt_pano_directions' factors: w entries (cos, sin) of each column's longitude
// lam = 2 pi ((x + 0.5) / w - 0.5), then h entries (cos, sin) of each row's latitude phi = pi ((y + 0.5) / h - 0.5), in
// double and rounded to float once.  The angle is taken as pi * (2x + 1 - w) / w (the same value): the integer numerator
// is exact, so mirrored columns and rows get exactly opposite angles, equal cosines and opposite sines.
void pano_table(int w, int h, float* out) {
    const double kPi = 3.14159265358979323846;
    for (int x = 0; x < w; ++x) {
        const double lam = kPi * ((double)(2ll * x + 1 - w) / w);
        out[2 * x] = (float)std::cos(lam);
        out[2 * x + 1] = (float)std::sin(lam);
    }
    for (int y = 0; y < h; ++y) {
        const double phi = 0.5 * kPi * ((double)(2ll * y + 1 - h) / h);
        out[2 * ((size_t)w + y)] = (float)std::cos(phi);
        out[2 * ((size_t)w + y) + 1] = (float)std::sin(phi);
    }
}
}  // namespace rrtk

extern "C" {

void rrt_camera_from(const float pos[3], float yaw_deg, float pitch_deg, rrt_camera* out) {
    if (!pos || !out) return;
    basis_from(Vec{pos[0], pos[1], pos[2]}, yaw_deg, pitch_deg, out);
}

int rrt_path_count(void) { return kNumPaths; }
const char* rrt_path_name(int i) { return (i >= 0 && i < kNumPaths) ? kPaths[i].name : nullptr; }
int rrt_path_num_keys(int i) { return (i >= 0 && i < kNumPaths) ? kPaths[i].n : RRT_ERR_BAD_ARG; }
float rrt_path_duration(int i) { return (i >= 0 && i < kNumPaths) ? kPaths[i].keys[kPaths[i].n - 1].t : -1.0f; }

int rrt_path_state(int path_index, float t, rrt_camera* out, float pyp[5]) {
    if (path_index < 0 || path_index >= kNumPaths || !out) return RRT_ERR_BAD_ARG;
    const Key* k = kPaths[path_index].keys;
    const int n = kPaths[path_index].n;
    Vec pos = k[0].pos;
    float yaw = k[0].yaw, pitch = k[0].pitch;
    if (t <= k[0].t) {
        // clamp to the first key (src/main.cpp:183)
    } else if (t >= k[n - 1].t) {  // clamp to the last key (:184)
        pos = k[n - 1].pos; yaw = k[n - 1].yaw; pitch = k[n - 1].pitch;
    } else {
        int seg = -1;
        for (int i = 0; i + 1 < n; ++i)
            if (t >= k[i].t && t <= k[i + 1].t) { seg = i; break; }  // first matching segment (:186-187)
        if (seg < 0) return RRT_ERR_BAD_ARG;
        const float s = (t - k[seg].t) / (k[seg + 1].t - k[seg].t);
        const int a = seg > 0 ? seg - 1 : 0, d = seg + 2 < n ? seg + 2 : n - 1;  // neighbour clamping (:190-193)
        const float s2 = s * s, s3 = s2 * s;
        pos.x = spline(k[a].pos.x, k[seg].pos.x, k[seg + 1].pos.x, k[d].pos.x, s, s2, s3);
        pos.y = spline(k[a].pos.y, k[seg].pos.y, k[seg + 1].pos.y, k[d].pos.y, s, s2, s3);
        pos.z = spline(k[a].pos.z, k[seg].pos.z, k[seg + 1].pos.z, k[d].pos.z, s, s2, s3);
        yaw = mix_angle(k[seg].yaw, k[seg + 1].yaw, s);
        pitch = mix_angle(k[seg].pitch, k[seg + 1].pitch, s);
    }
    basis_from(pos, yaw, pitch, out);
    if (pyp) { pyp[0] = pos.x; pyp[1] = pos.y; pyp[2] = pos.z; pyp[3] = yaw; pyp[4] = pitch; }
    return RRT_OK;
}

float rrt_path_clock(int frame, float fps) {
    // recording mode advances a float clock by dt = 1.0f / RECORDING_FPS every frame (src/main.cpp:511-516)
    volatile float t = 0.0f;
    const float dt = 1.0f / fps;
    for (int i = 0; i < frame; ++i) t = t + dt;
    return t;
}

int rrt_shutter_times(float t, float shutter, float fps, int n, float* out) {
    if (!out || !(shutter >= 0.0f && shutter <= 1.0f) || !(fps > 0.0f) || n < 1 || n > 64) return RRT_ERR_BAD_ARG;
    // a shutter open for `shutter` of the frame interval, centred on t; every operation one binary32 op (no contraction)
    const float d = shutter / fps;
    for (int i = 0; i < n; ++i) {
        const float u = ((float)i + 0.5f) / (float)n - 0.5f;
        out[i] = t + d * u;
    }
    return RRT_OK;
}

int rrt_lens_cameras(const rrt_camera* cam, float aperture, float focus, int ss, rrt_camera* out) {
    if (!cam || !out || !(aperture >= 0.0f) || !std::isfinite(aperture) || !(focus > 0.0f) || !std::isfinite(focus) || ss < 1 || ss > 8)
        return RRT_ERR_BAD_ARG;
    for (int j = 0; j < ss; ++j)
        for (int i = 0; i < ss; ++i) {
            rrt_camera& c = out[j * ss + i];
            c = *cam;
            // cell centre (a, b) = (na, nb) / ss in [-1, 1]^2; its image on the unit disk under Shirley & Chiu's concentric
            // map, in double and rounded to float once: the larger coordinate is the radius, the ratio of the two the angle
            const int na = 2 * i + 1 - ss, nb = 2 * j + 1 - ss;
            if (aperture == 0.0f || (na == 0 && nb == 0)) continue;   // the pinhole itself: an exact copy (keeps -0 fields)
            const double kPi4 = 0.78539816339744830962, a = (double)na / ss, b = (double)nb / ss;
            double x, y;
            if (std::abs(na) > std::abs(nb)) {
                const double t = kPi4 * ((double)nb / na);
                x = a * std::cos(t);
                y = a * std::sin(t);
            } else {   // phi = pi/2 - pi/4 * (a / b): cos(phi) = sin(pi/4 * a / b), sin(phi) = cos(pi/4 * a / b)
                const double t = kPi4 * ((double)na / nb);
                x = b * std::sin(t);
                y = b * std::cos(t);
            }
            const float ox = (float)((double)aperture * x), oy = (float)((double)aperture * y);
            // one binary32 operation each, in this order (no contraction): o = right * ox + up * oy, pos + o, forward - o / focus
            for (int k = 0; k < 3; ++k) {
                const float rx = cam->right[k] * ox, uy = cam->up[k] * oy;
                const float o = rx + uy;
                c.pos[k] = cam->pos[k] + o;
                const float tilt = o / focus;
                c.forward[k] = cam->forward[k] - tilt;
            }
        }
    return RRT_OK;
}

int rrt_pano_directions(const rrt_camera* cam, int w, int h, float* out) {
    if (!cam || !out || w <= 0 || h <= 0 || (unsigned long long)w * h > SIZE_MAX / (3 * sizeof(float))) return RRT_ERR_BAD_ARG;
    std::vector<float> t(2 * ((size_t)w + h));
    rrtk::pano_table(w, h, t.data());
    const float* lat = t.data() + 2 * (size_t)w;
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
            // one binary32 operation each, in this order (no contraction), as pano_dir does on the device
            const float a = lat[2 * y] * t[2 * x], b = lat[2 * y] * t[2 * x + 1];
            float* d = out + ((size_t)y * w + x) * 3;
            for (int c = 0; c < 3; ++c) {
                const float af = a * cam->forward[c], br = b * cam->right[c], su = lat[2 * y + 1] * cam->up[c];
                const float s = af + br;
                d[c] = s + su;
            }
        }
    return RRT_OK;
}

// ---- frame sink: the step immediately after the hot path --------------------------------------------------
// The reference's ScreenRecorder (src/main.cpp:29-124) reads the window back with glReadPixels -- which, for the
// 1:1 textured quad it draws (src/main.cpp:404-409, 471-479), returns exactly the bytes launch_raymarch wrote,
// buffer row 0 first -- and fwrite()s each frame to `ffmpeg -f rawvideo -pix_fmt rgba -s WxH -r 24 -i - -vf vflip
// ...` (src/main.cpp:61-72, 85-97).  RRT_SINK_RGBA writes that wire format byte for byte; a target that starts
// with '|' is popen()ed like the reference does, so "|ffmpeg ..." reproduces the recorder on a box that has
// ffmpeg.  RRT_SINK_Y4M writes a self-describing YUV4MPEG2 4:2:0 file with the rows already flipped (what
// -vf vflip -pix_fmt yuv420p would hand to the encoder), BT.601 studio range, for boxes without ffmpeg.
}  // extern "C"

struct rrt_sink {
    FILE* f = nullptr;
    bool piped = false;
    int format = 0, w = 0, h = 0, frames = 0;
    std::vector<uint8_t> yuv;
};

extern "C" {

int rrt_sink_ffmpeg_command(int w, int h, int fps, const char* out_name, char* buf, int buflen) {
    if (!buf || buflen <= 0 || !out_name || w <= 0 || h <= 0 || fps <= 0) return RRT_ERR_BAD_ARG;
    // src/main.cpp:61-72, same options in the same order
    const int n = std::snprintf(buf, (size_t)buflen,
                                "ffmpeg -y -f rawvideo -pix_fmt rgba -s %dx%d -r %d -i - -vf vflip -c:v libx264 -preset fast "
                                "-crf 18 -pix_fmt yuv420p \"%s\"",
                                w, h, fps, out_name);
    return (n < 0 || n >= buflen) ? RRT_ERR_BAD_ARG : n;
}

int rrt_sink_open(const char* target, int format, int w, int h, int fps, rrt_sink** out) {
    if (!out) return RRT_ERR_BAD_ARG;
    *out = nullptr;
    if (!target || !*target || w <= 0 || h <= 0 || fps <= 0 || (format != RRT_SINK_RGBA && format != RRT_SINK_Y4M))
        return RRT_ERR_BAD_ARG;
    rrt_sink* s = new (std::nothrow) rrt_sink();
    if (!s) return RRT_ERR_NOMEM;
    s->format = format; s->w = w; s->h = h;
    s->piped = target[0] == '|';
    s->f = s->piped ? popen(target + 1, "w") : std::fopen(target, "wb");
    if (!s->f) { delete s; return RRT_ERR_IO; }   // like the recorder's "Failed to start FFmpeg" (src/main.cpp:75-78)
    if (format == RRT_SINK_Y4M) {
        s->yuv.resize((size_t)w * h + 2 * (size_t)((w + 1) / 2) * ((h + 1) / 2));
        if (std::fprintf(s->f, "YUV4MPEG2 W%d H%d F%d:1 Ip A1:1 C420jpeg\n", w, h, fps) < 0) {
            rrt_sink_close(s);
            return RRT_ERR_IO;
        }
    }
    *out = s;
    return RRT_OK;
}

int rrt_sink_write(rrt_sink* s, const uint8_t* host_rgba) {
    if (!s || !s->f || !host_rgba) return RRT_ERR_BAD_ARG;
    const int w = s->w, h = s->h;
    if (s->format == RRT_SINK_RGBA) {
        const size_t n = (size_t)w * h * 4;
        if (std::fwrite(host_rgba, 1, n, s->f) != n) return RRT_ERR_IO;   // "Frame write incomplete", src/main.cpp:93-95
    } else {
        // vflip: output row j is buffer row h-1-j
        const int cw = (w + 1) / 2, ch = (h + 1) / 2;
        uint8_t* Y = s->yuv.data();
        uint8_t* U = Y + (size_t)w * h;
        uint8_t* V = U + (size_t)cw * ch;
        auto px = [&](int x, int j) { return host_rgba + ((size_t)(h - 1 - j) * w + x) * 4; };
        for (int j = 0; j < h; ++j)
            for (int x = 0; x < w; ++x) {
                const uint8_t* p = px(x, j);
                Y[(size_t)j * w + x] = (uint8_t)(((66 * p[0] + 129 * p[1] + 25 * p[2] + 128) >> 8) + 16);
            }
        for (int cj = 0; cj < ch; ++cj)
            for (int cx = 0; cx < cw; ++cx) {
                int r = 0, g = 0, b = 0;
                for (int dy = 0; dy < 2; ++dy)
                    for (int dx = 0; dx < 2; ++dx) {
                        const int x = 2 * cx + dx < w ? 2 * cx + dx : w - 1, j = 2 * cj + dy < h ? 2 * cj + dy : h - 1;
                        const uint8_t* p = px(x, j);
                        r += p[0]; g += p[1]; b += p[2];
                    }
                r = (r + 2) >> 2; g = (g + 2) >> 2; b = (b + 2) >> 2;
                U[(size_t)cj * cw + cx] = (uint8_t)(((-38 * r - 74 * g + 112 * b + 128) >> 8) + 128);
                V[(size_t)cj * cw + cx] = (uint8_t)(((112 * r - 94 * g - 18 * b + 128) >> 8) + 128);
            }
        if (std::fputs("FRAME\n", s->f) < 0 || std::fwrite(s->yuv.data(), 1, s->yuv.size(), s->f) != s->yuv.size())
            return RRT_ERR_IO;
    }
    ++s->frames;
    return RRT_OK;
}

int rrt_sink_frames(const rrt_sink* s) { return s ? s->frames : RRT_ERR_BAD_ARG; }

int rrt_sink_close(rrt_sink* s) {
    if (!s) return RRT_ERR_BAD_ARG;
    int rc = RRT_OK;
    if (s->f) {
        const int e = s->piped ? pclose(s->f) : std::fclose(s->f);
        if (e != 0) rc = RRT_ERR_IO;
    }
    delete s;
    return rc;
}

}  // extern "C"
