// Device helpers shared by the direct-gather (warp.cu) and the TMA-staged (warp_tma.cu) warp kernels.
#pragma once

#include "common.cuh"

namespace cf {

struct Taps {
    int o00, o01, o10, o11;  // offsets inside one channel plane
    float w00, w01, w10, w11;
};

// ATen reflect_coordinates(v, 0, 2*(size-1)) followed by clip_coordinates.
__device__ __forceinline__ float reflect_clip(float v, int size) {
    if (size == 1) return 0.f;
    const float span = (float)(size - 1);
    const float a = fabsf(v);
    // fast path (the sample lies inside the image): for a < span ATen's fmod(a, span) == a and
    // floor(a / span) == 0 exactly (a/span <= 1 - 2^-24 never rounds up to 1), so no division / fmod
    float r;
    if (a < span) {
        r = a;
    } else {
        const float extra = fmodf(a, span);
        const int flips = (int)floorf(a / span);
        r = (flips & 1) ? span - extra : extra;
    }
    return fminf(span, fmaxf(r, 0.f));
}

// Fused upflow8 + ImagePadder.unpad (SURVEY 8f rank 1; DCEIFlow/DCEIFlow.py:222-227, DCEIFlow/utils/sample_utils.py:66-68,
// utils/image_process.py:87-107): the flow network predicts at 1/8 of the x32-padded frame; the reference up-samples
// x8 bilinearly (align_corners=True, values x8), cuts the top/left padding off, and only then warps.  With `lr` set the
// full-resolution flow is never read: it is evaluated from the 1/8-resolution field on the fly (and optionally written
// out once, by the image part, because the model returns it as batch_flow['flow_final']).
struct FlowLR {
    const float *lr;       // [B,2,lh,lw] or nullptr (no fused up-sampling: the kernels read `flow`)
    int lh, lw, pad_h, pad_w;
    float sy, sx;          // ATen align_corners scales (lh-1)/(8*lh-1), (lw-1)/(8*lw-1)
    float *flow_out;       // optional [B,2,H,W]: upflow8 + unpad
};

// ATen upsample_bilinear2d(align_corners=True) at destination (X, Y) of the x8 grid, times 8; (x, y) un-padded
static __device__ __noinline__ float2 upflow8_at(const FlowLR &s, int b, int x, int y) {
    const float fy = s.sy * (float)(y + s.pad_h), fx = s.sx * (float)(x + s.pad_w);
    const int y0 = min((int)fy, s.lh - 1), x0 = min((int)fx, s.lw - 1);
    const int y1 = y0 + (y0 < s.lh - 1 ? 1 : 0), x1 = x0 + (x0 < s.lw - 1 ? 1 : 0);
    const float ly1 = fminf(fmaxf(fy - (float)y0, 0.f), 1.f), lx1 = fminf(fmaxf(fx - (float)x0, 0.f), 1.f);
    const float ly0 = 1.f - ly1, lx0 = 1.f - lx1;
    const float *c = s.lr + (size_t)b * 2 * s.lh * s.lw;
    float2 r;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const float p00 = __ldg(c + y0 * s.lw + x0), p01 = __ldg(c + y0 * s.lw + x1);
        const float p10 = __ldg(c + y1 * s.lw + x0), p11 = __ldg(c + y1 * s.lw + x1);
        const float v = 8.f * (ly0 * (lx0 * p00 + lx1 * p01) + ly1 * (lx0 * p10 + lx1 * p11));
        if (k == 0) r.x = v; else r.y = v;
        c += (size_t)s.lh * s.lw;
    }
    return r;
}

// Flow at output pixel (x, y).  half == false: flow has the output's size.
// half == true: x0.5 bilinear, align_corners=True from the [fH, fW] field
// (ATen upsample_bilinear2d: src = scale*dst, lambda clamped to [0,1]).
// `fb` is this batch item's [2,fH,fW] field; with lr.lr set the field is virtual (upflow8_at).
__device__ __forceinline__ float2 flow_at(const float *__restrict__ fb, int x, int y, int W,
                                          int fH, int fW, bool half, float sy, float sx, const FlowLR &lr, int b) {
    if (!half) {
        if (lr.lr) return upflow8_at(lr, b, x, y);
        const int p = y * W + x;
        return make_float2(__ldg(fb + p), __ldg(fb + (size_t)fH * fW + p));
    }
    const float fy = sy * (float)y, fx = sx * (float)x;
    int y0 = min((int)fy, fH - 1), x0 = min((int)fx, fW - 1);
    const int y1 = y0 + (y0 < fH - 1 ? 1 : 0), x1 = x0 + (x0 < fW - 1 ? 1 : 0);
    const float ly1 = fminf(fmaxf(fy - (float)y0, 0.f), 1.f), lx1 = fminf(fmaxf(fx - (float)x0, 0.f), 1.f);
    const float ly0 = 1.f - ly1, lx0 = 1.f - lx1;
    float2 r;
    if (lr.lr) {
        const float2 p00 = upflow8_at(lr, b, x0, y0), p01 = upflow8_at(lr, b, x1, y0);
        const float2 p10 = upflow8_at(lr, b, x0, y1), p11 = upflow8_at(lr, b, x1, y1);
        r.x = ly0 * (lx0 * p00.x + lx1 * p01.x) + ly1 * (lx0 * p10.x + lx1 * p11.x);
        r.y = ly0 * (lx0 * p00.y + lx1 * p01.y) + ly1 * (lx0 * p10.y + lx1 * p11.y);
        return r;
    }
    const float *c = fb;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const float p00 = __ldg(c + y0 * fW + x0), p01 = __ldg(c + y0 * fW + x1);
        const float p10 = __ldg(c + y1 * fW + x0), p11 = __ldg(c + y1 * fW + x1);
        const float v = ly0 * (lx0 * p00 + lx1 * p01) + ly1 * (lx0 * p10 + lx1 * p11);
        if (k == 0) r.x = v; else r.y = v;
        c += (size_t)fH * fW;
    }
    return r;
}

__device__ __forceinline__ Taps make_taps(float u, float v, int x, int y, int H, int W, float sign) {
    // utils/flow_utils.py:110-116 (sign=+1) / :180-186 (sign=-1), then ATen
    // grid_sampler_unnormalize(align_corners=True): ((g + 1) / 2) * (size - 1).
    const float gx = 2.f * (((float)x + sign * u) / (float)W - 0.5f);
    const float gy = 2.f * (((float)y + sign * v) / (float)H - 0.5f);
    const float ix = reflect_clip(((gx + 1.f) / 2.f) * (float)(W - 1), W);
    const float iy = reflect_clip(((gy + 1.f) / 2.f) * (float)(H - 1), H);
    const float fx0 = floorf(ix), fy0 = floorf(iy);
    const int x0 = (int)fx0, y0 = (int)fy0;
    // after the clip x0+1 == W only when ix == W-1 exactly, where its weight is 0
    const int x1 = min(x0 + 1, W - 1), y1 = min(y0 + 1, H - 1);
    // ATen weights: nw = (x_se - ix)(y_se - iy), ne = (ix - x_sw)(y_sw - iy), ...
    const float ax1 = (fx0 + 1.f) - ix, ax0 = ix - fx0;
    const float ay1 = (fy0 + 1.f) - iy, ay0 = iy - fy0;
    Taps t;
    t.o00 = y0 * W + x0; t.o01 = y0 * W + x1; t.o10 = y1 * W + x0; t.o11 = y1 * W + x1;
    t.w00 = ax1 * ay1;
    t.w01 = ax0 * ay1;
    t.w10 = ax1 * ay0;
    t.w11 = ax0 * ay0;
    return t;
}

// ---- adjoint of the warp (warp_backward.cu: atomic splat, warp_backward_det.cu: sort + gather) -------------------
// ATen reflect_coordinates_set_grad(v, 0, 2*(size-1)) + clip_coordinates_set_grad, after unnormalize (align_corners)
__device__ __forceinline__ float source_index_set_grad(float g, int size, float &mult) {
    const float unnorm = (float)(size - 1) / 2.f;
    float v = ((g + 1.f) / 2.f) * (float)(size - 1);
    float m = 1.f;
    if (size == 1) { mult = 0.f; return 0.f; }
    const float span = (float)(size - 1);
    if (v < 0.f) { v = -v; m = -1.f; }
    const float extra = fmodf(v, span);
    const int flips = (int)floorf(v / span);
    if (flips & 1) { v = span - extra; m = -m; } else { v = extra; }
    // clip: gradient 0 on and beyond the borders
    if (v <= 0.f) { v = 0.f; m = 0.f; }
    else if (v >= span) { v = span; m = 0.f; }
    mult = m * unnorm;
    return v;
}

struct GradPos {
    int x0, y0;               // top-left tap (floor of the sample position)
    float ax0, ax1, ay0, ay1; // ix - x0, (x0 + 1) - ix, ...
    float mx, my;             // d(ix)/d(gx), d(iy)/d(gy) incl. reflection sign and clipping
    bool xin1, yin1;          // the right / lower taps are inside (x0, y0 always are after the clip)
};

// sample position of output pixel (x, y) for flow (u, v) with the gradient multipliers of the backward pass
__device__ __forceinline__ GradPos grad_pos(float u, float v, int x, int y, int H, int W, float sign) {
    const float gx = 2.f * (((float)x + sign * u) / (float)W - 0.5f);
    const float gy = 2.f * (((float)y + sign * v) / (float)H - 0.5f);
    GradPos q;
    const float ix = source_index_set_grad(gx, W, q.mx), iy = source_index_set_grad(gy, H, q.my);
    const float fx0 = floorf(ix), fy0 = floorf(iy);
    q.x0 = (int)fx0;
    q.y0 = (int)fy0;
    q.ax1 = (fx0 + 1.f) - ix; q.ax0 = ix - fx0; q.ay1 = (fy0 + 1.f) - iy; q.ay0 = iy - fy0;
    q.xin1 = q.x0 + 1 < W;
    q.yin1 = q.y0 + 1 < H;
    return q;
}

// taps and lambdas of the x0.5 bilinear (align_corners=True) down-sampling at output pixel (x, y): those of flow_at()
struct HalfTaps {
    int y0, y1, x0, x1;
    float ly0, ly1, lx0, lx1;
};
__device__ __forceinline__ HalfTaps half_taps(int x, int y, int fH, int fW, float sy, float sx) {
    HalfTaps t;
    const float fy = sy * (float)y, fx = sx * (float)x;
    t.y0 = min((int)fy, fH - 1);
    t.x0 = min((int)fx, fW - 1);
    t.y1 = t.y0 + (t.y0 < fH - 1 ? 1 : 0);
    t.x1 = t.x0 + (t.x0 < fW - 1 ? 1 : 0);
    t.ly1 = fminf(fmaxf(fy - (float)t.y0, 0.f), 1.f);
    t.lx1 = fminf(fmaxf(fx - (float)t.x0, 0.f), 1.f);
    t.ly0 = 1.f - t.ly1;
    t.lx0 = 1.f - t.lx1;
    return t;
}

// Taps that reproduce the input pixel (weights 1, 0, 0, 0): what the reference's `if not flow_final.any()` branch
// returns (e2v/e2v_model.py:184-185).  Used when the device-side gate says the flow is all zero -- a zero flow is
// NOT the identity under the reference's 2*(x/W-0.5) normalisation (SURVEY.md F6), hence the explicit branch.
__device__ __forceinline__ Taps identity_taps(int x, int y, int W) {
    Taps t;
    t.o00 = t.o01 = t.o10 = t.o11 = y * W + x;
    t.w00 = 1.f;
    t.w01 = t.w10 = t.w11 = 0.f;
    return t;
}
// gate == nullptr: always warp; else *gate == 0 (written by cf_flow_any) means "flow is all zero": copy
__device__ __forceinline__ bool gate_closed(const int *__restrict__ gate) { return gate != nullptr && __ldg(gate) == 0; }

// One thread = one output pixel x CPT channels.  Addressing: the channel base is warp-uniform (one 64-bit add per
// channel on the uniform datapath); the four taps and the output are 32-bit byte offsets inside a plane (planes hold
// < 2^30 elements), so a tap costs one 64-bit add + one LDG.  (Written as `img_b + c * plane + t.o00` per tap the
// compiler produced ~80 instructions per output -- 55 % IMAD/LEA/MOV address arithmetic -- and the direct kernel was
// issue bound at 70 % issue-slot utilisation, 37 % of HBM.)
template <int CPT>
__device__ __forceinline__ void warp_pixel(const float *__restrict__ img_b, float *__restrict__ out_b,
                                           const Taps &t, int p, int c0, int C, size_t plane) {
    const unsigned b00 = 4u * (unsigned)t.o00, b01 = 4u * (unsigned)t.o01, b10 = 4u * (unsigned)t.o10, b11 = 4u * (unsigned)t.o11;
    const unsigned bo = 4u * (unsigned)p;
    const size_t pb = plane * sizeof(float);
    const char *src = reinterpret_cast<const char *>(img_b) + (size_t)c0 * pb;
    char *dst = reinterpret_cast<char *>(out_b) + (size_t)c0 * pb;
    if (c0 + CPT <= C) {   // whole batch of channels in range: no per-channel predicates (the common case, C % CPT == 0)
        float v[CPT][4];
        if (b01 == b00 + 4u && b11 == b10 + 4u) {
            // the right-hand taps are the next float (everywhere but on the clamped last column): two addresses per
            // channel, the +4 rides in the load's immediate offset
#pragma unroll
            for (int k = 0; k < CPT; ++k) {
                const float *top = reinterpret_cast<const float *>(src + (size_t)k * pb + b00);
                const float *bot = reinterpret_cast<const float *>(src + (size_t)k * pb + b10);
                v[k][0] = __ldg(top);
                v[k][1] = __ldg(top + 1);
                v[k][2] = __ldg(bot);
                v[k][3] = __ldg(bot + 1);
            }
        } else {
#pragma unroll
            for (int k = 0; k < CPT; ++k) {
                const char *s = src + (size_t)k * pb;
                v[k][0] = __ldg(reinterpret_cast<const float *>(s + b00));
                v[k][1] = __ldg(reinterpret_cast<const float *>(s + b01));
                v[k][2] = __ldg(reinterpret_cast<const float *>(s + b10));
                v[k][3] = __ldg(reinterpret_cast<const float *>(s + b11));
            }
        }
#pragma unroll
        for (int k = 0; k < CPT; ++k) {
            // ATen order: nw, ne, sw, se accumulated left to right
            float r = v[k][0] * t.w00;
            r += v[k][1] * t.w01;
            r += v[k][2] * t.w10;
            r += v[k][3] * t.w11;
            st_cs(reinterpret_cast<float *>(dst + (size_t)k * pb + bo), r);
        }
        return;
    }
#pragma unroll
    for (int k = 0; k < CPT; ++k) {
        if (c0 + k < C) {
            const char *s = src + (size_t)k * pb;
            float r = __ldg(reinterpret_cast<const float *>(s + b00)) * t.w00;
            r += __ldg(reinterpret_cast<const float *>(s + b01)) * t.w01;
            r += __ldg(reinterpret_cast<const float *>(s + b10)) * t.w10;
            r += __ldg(reinterpret_cast<const float *>(s + b11)) * t.w11;
            st_cs(reinterpret_cast<float *>(dst + (size_t)k * pb + bo), r);
        }
    }
}

struct WarpJob {
    const float *img; float *out;
    int C, H, W;          // geometry of img/out
    int half;             // 1: flow is [2, fH, fW] at twice the resolution
    float sy, sx;         // align_corners scales for the fused down-sampling
    int tiles_x;          // 32-pixel-wide tiles per row
    int blocks_x;         // pixel tiles (32x8) per (batch, channel group)
    int cpg;              // channels per group (one thread loops over them, CPT at a time)
    int groups;           // channel groups
};
constexpr int kTileW = 32, kTileH = 8;

template <int CPT>
__device__ __forceinline__ void run_job(const WarpJob &j, const float *__restrict__ flow,
                                        int fH, int fW, float sign, int tile, int group, int b, const int *__restrict__ gate,
                                        const FlowLR &lr, bool write_flow = false) {
    const int ty = tile / j.tiles_x, tx = tile - ty * j.tiles_x;
    const int x = tx * kTileW + (threadIdx.x & 31), y = ty * kTileH + (threadIdx.x >> 5);
    if (x >= j.W || y >= j.H) return;
    const int p = y * j.W + x;
    const float *fb = flow + (size_t)b * 2 * fH * fW;
    Taps t;
    if (gate_closed(gate)) {
        t = identity_taps(x, y, j.W);
    } else {
        const float2 uv = flow_at(fb, x, y, j.W, fH, fW, j.half != 0, j.sy, j.sx, lr, b);
        if (write_flow && lr.flow_out != nullptr && group == 0) {   // upflow8 + unpad, once per full-resolution pixel
            float *fo = lr.flow_out + (size_t)b * 2 * j.H * j.W;
            fo[p] = uv.x;
            fo[(size_t)j.H * j.W + p] = uv.y;
        }
        t = make_taps(uv.x, uv.y, x, y, j.H, j.W, sign);
    }
    const size_t plane = (size_t)j.H * j.W;
    const float *img_b = j.img + (size_t)b * j.C * plane;
    float *out_b = j.out + (size_t)b * j.C * plane;
    const int c_end = min(j.C, (group + 1) * j.cpg);
    for (int c0 = group * j.cpg; c0 < c_end; c0 += CPT) warp_pixel<CPT>(img_b, out_b, t, p, c0, c_end, plane);
}

}  // namespace cf
