// Deterministic adjoint of the flow-guided warp (include/cistaflow_det.h): the gradients of warp_backward.cu with
// every output element written once, by one thread, summing its terms in an order fixed by the inputs alone.
//
// The per-term arithmetic is warp_backward_kernel's (grad_pos / half_taps of warp_common.cuh: the same sample
// position, reflect/clip multipliers, 2*(x/W-0.5) chain rule and down-sampling lambdas); only the summation differs:
//   warp_backward_det_taps_kernel     one thread per output pixel p: the records (key = item*H*W + source pixel,
//                                     value = 4p + k, weight of tap k) of its valid taps -- invalid taps get the
//                                     key Bc*H*W and sort to the end -- and, for grad_flow, the sum over ALL
//                                     channels in channel order (written, or kept per pixel for the x0.5 adjoint);
//   rs_hist / rs_scan / rs_scatter    the stable LSB radix sort of radix_sort.cuh (records start in value order, so
//                                     a source pixel's bucket ends up in ascending (p, k) order);
//   warp_backward_det_bounds_kernel   bucket starts: the head of each run of equal keys writes the start of its own
//                                     bucket and of the empty buckets before it, every entry exactly once;
//   warp_backward_det_gather_kernel   one thread per (source pixel, 32 channels): walks its bucket in order,
//                                     accumulating w * grad_out[c, p], writes grad_img[c, s] (0 for an empty bucket);
//   warp_backward_det_flow_half_kernel  one thread per full-resolution flow pixel: gathers, in (y, x, tap) order, the
//                                     half-resolution pixels whose bilinear taps include it.
// The batch runs in chunks of Bc items such that the 4*Bc*H*W records fit 32-bit keys and values.  A flow that
// converges on one point puts all 4*H*W records of an item into one bucket: still correct, walked by one thread.
#include "cistaflow_det.h"
#include "radix_sort.cuh"
#include "warp_common.cuh"

namespace cf {
namespace wbd {
constexpr int THREADS = 256;
constexpr int CPG = 32;   // channels per gather thread

__global__ void __launch_bounds__(THREADS)
warp_backward_det_taps_kernel(const float *__restrict__ grad_out, const float *__restrict__ img,
                              const float *__restrict__ flow, int items, int C, int H, int W, int fH, int fW, int half,
                              float sy, float sx, float sign, uint4 *__restrict__ keys, uint4 *__restrict__ vals,
                              float4 *__restrict__ wts, float *__restrict__ grad_flow, float *__restrict__ gflow_half) {
    const int64_t plane = (int64_t)H * W;
    const int64_t i = (int64_t)blockIdx.x * THREADS + threadIdx.x;   // item-major output pixel of the chunk
    if (i >= items * plane) return;
    const int b = (int)(i / plane);
    const int p = (int)(i - b * plane);
    const int y = p / W, x = p - y * W;
    const float2 uv = flow_at(flow + (size_t)b * 2 * fH * fW, x, y, W, fH, fW, half != 0, sy, sx, FlowLR{}, 0);
    const GradPos q = grad_pos(uv.x, uv.y, x, y, H, W, sign);
    const int o00 = q.y0 * W + q.x0, o01 = o00 + 1, o10 = o00 + W, o11 = o10 + 1;
    if (keys) {
        const uint32_t base = (uint32_t)(b * plane), invalid = (uint32_t)(items * plane);
        keys[i] = make_uint4(base + o00, q.xin1 ? base + o01 : invalid, q.yin1 ? base + o10 : invalid,
                             (q.xin1 && q.yin1) ? base + o11 : invalid);
        const uint32_t v = 4u * (uint32_t)i;
        vals[i] = make_uint4(v, v + 1u, v + 2u, v + 3u);
        wts[i] = make_float4(q.ax1 * q.ay1, q.ax0 * q.ay1, q.ax1 * q.ay0, q.ax0 * q.ay0);
    }
    if (!grad_flow) return;
    const float *go = grad_out + (size_t)b * C * plane + p;
    const float *im = img + (size_t)b * C * plane;
    float gix = 0.f, giy = 0.f;
    for (int c = 0; c < C; ++c) {   // every channel, in order
        const float g = __ldg(go);
        const float v00 = __ldg(im + o00), v01 = q.xin1 ? __ldg(im + o01) : 0.f;
        const float v10 = q.yin1 ? __ldg(im + o10) : 0.f, v11 = (q.xin1 && q.yin1) ? __ldg(im + o11) : 0.f;
        gix += g * (-v00 * q.ay1 + v01 * q.ay1 - v10 * q.ay0 + v11 * q.ay0);
        giy += g * (-v00 * q.ax1 - v01 * q.ax0 + v10 * q.ax1 + v11 * q.ax0);
        go += plane;
        im += plane;
    }
    const float gu = sign * (2.f * (q.mx * gix)) / (float)W, gv = sign * (2.f * (q.my * giy)) / (float)H;
    if (!half) {
        float *gfb = grad_flow + (size_t)b * 2 * plane;
        gfb[p] = gu;
        gfb[plane + p] = gv;
    } else {
        float *gh = gflow_half + (size_t)b * 2 * plane;
        gh[p] = gu;
        gh[plane + p] = gv;
    }
}

// starts[s] = index of the first record with key >= s, for s = 0 .. M (M = the invalid key)
__global__ void __launch_bounds__(THREADS)
warp_backward_det_bounds_kernel(const uint32_t *__restrict__ keys, int64_t n, uint32_t M, uint32_t *__restrict__ starts) {
    const int64_t i = (int64_t)blockIdx.x * THREADS + threadIdx.x;
    if (i >= n) return;
    const int64_t k = keys[i];
    const int64_t prev = i > 0 ? (int64_t)keys[i - 1] : -1;
    for (int64_t s = prev + 1; s <= k; ++s) starts[s] = (uint32_t)i;
    if (i == n - 1)
        for (int64_t s = k + 1; s <= (int64_t)M; ++s) starts[s] = (uint32_t)n;
}

__global__ void __launch_bounds__(THREADS)
warp_backward_det_gather_kernel(const uint32_t *__restrict__ vals, const float *__restrict__ wts,
                                const uint32_t *__restrict__ starts, const float *__restrict__ grad_out,
                                float *__restrict__ grad_img, int items, int C, int64_t plane) {
    const int64_t s = (int64_t)blockIdx.x * THREADS + threadIdx.x;   // item-major source pixel of the chunk
    if (s >= items * plane) return;
    const int b = (int)(s / plane);
    const int64_t src = s - b * plane;
    const int c_begin = blockIdx.y * CPG, cn = min(C - c_begin, CPG);
    const float *go = grad_out + ((size_t)b * C + c_begin) * plane;
    const uint32_t pix0 = (uint32_t)(b * plane);
    float acc[CPG];
#pragma unroll
    for (int c = 0; c < CPG; ++c) acc[c] = 0.f;
    const uint32_t e = starts[s + 1];
    for (uint32_t j = starts[s]; j < e; ++j) {   // ascending (p, k)
        const uint32_t v = vals[j];
        const float w = wts[v];
        const float *g = go + ((v >> 2) - pix0);
#pragma unroll
        for (int c = 0; c < CPG; ++c)
            if (c < cn) acc[c] += __ldg(g + c * plane) * w;
    }
    float *gi = grad_img + ((size_t)b * C + c_begin) * plane + src;
#pragma unroll
    for (int c = 0; c < CPG; ++c)
        if (c < cn) gi[c * plane] = acc[c];
}

// candidate half-resolution coordinates whose down-sampling taps can reach full-resolution coordinate X (scale s >= 2,
// or 0 for a one-pixel axis); every candidate is then checked with the exact arithmetic of half_taps()
__device__ __forceinline__ void half_candidates(int X, float s, int n, int &lo, int &hi) {
    if (s > 0.f) {
        lo = max(0, (int)floorf((float)(X - 1) / s) - 1);
        hi = min(n - 1, (int)floorf((float)(X + 1) / s) + 1);
    } else {
        lo = 0;
        hi = n - 1;
    }
}

__global__ void __launch_bounds__(THREADS)
warp_backward_det_flow_half_kernel(const float *__restrict__ gflow_half, float *__restrict__ grad_flow, int items,
                                   int H, int W, int fH, int fW, float sy, float sx) {
    const int64_t fplane = (int64_t)fH * fW, plane = (int64_t)H * W;
    const int64_t i = (int64_t)blockIdx.x * THREADS + threadIdx.x;
    if (i >= items * fplane) return;
    const int b = (int)(i / fplane);
    const int P = (int)(i - b * fplane);
    const int Y = P / fW, X = P - Y * fW;
    int ylo, yhi, xlo, xhi;
    half_candidates(Y, sy, H, ylo, yhi);
    half_candidates(X, sx, W, xlo, xhi);
    const float *gh = gflow_half + (size_t)b * 2 * plane;
    float au = 0.f, av = 0.f;
    for (int y = ylo; y <= yhi; ++y) {
        for (int x = xlo; x <= xhi; ++x) {
            const HalfTaps t = half_taps(x, y, fH, fW, sy, sx);
            if (t.y0 != Y && t.y1 != Y) continue;
            if (t.x0 != X && t.x1 != X) continue;
            const float gu = __ldg(gh + y * W + x), gv = __ldg(gh + plane + y * W + x);
            // the four terms of warp_backward_kernel's splat, in its order (a clamped tap meets X or Y twice)
            if (t.y0 == Y && t.x0 == X) { au += gu * t.ly0 * t.lx0; av += gv * t.ly0 * t.lx0; }
            if (t.y0 == Y && t.x1 == X) { au += gu * t.ly0 * t.lx1; av += gv * t.ly0 * t.lx1; }
            if (t.y1 == Y && t.x0 == X) { au += gu * t.ly1 * t.lx0; av += gv * t.ly1 * t.lx0; }
            if (t.y1 == Y && t.x1 == X) { au += gu * t.ly1 * t.lx1; av += gv * t.ly1 * t.lx1; }
        }
    }
    float *gfb = grad_flow + (size_t)b * 2 * fplane;
    gfb[P] = au;
    gfb[fplane + P] = av;
}

struct Layout {
    int chunk;              // items per chunk
    int nblk;               // radix-sort CTAs for 4 * chunk * H * W records
    size_t keys0, vals0, keys1, vals1, wts, starts, hist, gflow, end;
};

static Layout layout(int B, int H, int W, bool half) {
    Layout L{};
    const int64_t plane = (int64_t)H * W;
    const int64_t fit = (int64_t)0xffffffffu / (4 * plane);   // 4 * chunk * plane < 2^32
    L.chunk = (int)(B < fit ? B : fit);
    const int64_t pix = (int64_t)L.chunk * plane, n = 4 * pix;
    L.nblk = (int)ceil_div(n, kRsTile);
    const size_t arr = align_up((size_t)n * 4, 256);
    L.keys0 = 0;
    L.vals0 = L.keys0 + arr;
    L.keys1 = L.vals0 + arr;
    L.vals1 = L.keys1 + arr;
    L.wts = L.vals1 + arr;
    L.starts = L.wts + arr;
    L.hist = L.starts + align_up((size_t)(pix + 1) * 4, 256);
    L.gflow = L.hist + align_up((size_t)256 * L.nblk * 4, 256);
    L.end = L.gflow + (half ? align_up((size_t)pix * 2 * 4, 256) : 0);
    return L;
}

// shape rules of cf_warp_backward; half / sy / sx of the fused x0.5 down-sampling
static int check_shape(int B, int C, int H, int W, int flowH, int flowW, int &half, float &sy, float &sx) {
    CF_REQUIRE(B >= 0 && C >= 0 && H > 0 && W > 0 && flowH > 0 && flowW > 0, CF_ERR_INVALID_ARG, "cf_warp_backward_det: bad shape");
    CF_REQUIRE((int64_t)H * W < (1ll << 30) && B <= 65535, CF_ERR_INVALID_ARG, "cf_warp_backward_det: too large");
    CF_REQUIRE(ceil_div(C, CPG) <= 65535, CF_ERR_INVALID_ARG, "cf_warp_backward_det: too many channels");
    half = 0;
    sy = sx = 0.f;
    if (flowH == H && flowW == W) return CF_OK;
    if (H == flowH / 2 && W == flowW / 2) {
        half = 1;
        sy = H > 1 ? (float)(flowH - 1) / (float)(H - 1) : 0.f;
        sx = W > 1 ? (float)(flowW - 1) / (float)(W - 1) : 0.f;
        return CF_OK;
    }
    set_error("cf_warp_backward_det: flow is %dx%d but the image is %dx%d (must be equal, or image == flow/2)", flowH, flowW, H, W);
    return CF_ERR_INVALID_ARG;
}
}  // namespace wbd
}  // namespace cf

extern "C" size_t cf_warp_backward_det_workspace_bytes(int B, int C, int H, int W, int flowH, int flowW) {
    using namespace cf;
    int half;
    float sy, sx;
    if (wbd::check_shape(B, C, H, W, flowH, flowW, half, sy, sx) != CF_OK || B == 0 || C == 0) return 0;
    return wbd::layout(B, H, W, half != 0).end + 256;
}

extern "C" int cf_warp_backward_det(const float *grad_out, const float *img, const float *flow, float *grad_img,
                                    float *grad_flow, int B, int C, int H, int W, int flowH, int flowW, float sign,
                                    void *workspace, size_t workspace_bytes, cf_stream_t stream_) {
    using namespace cf;
    if (int rc = check_device()) return rc;
    CF_REQUIRE(grad_out && flow, CF_ERR_NULL, "cf_warp_backward_det: null pointer");
    CF_REQUIRE(grad_img || grad_flow, CF_ERR_NULL, "cf_warp_backward_det: neither grad_img nor grad_flow requested");
    CF_REQUIRE(!grad_flow || img, CF_ERR_NULL, "cf_warp_backward_det: grad_flow needs img");
    int half;
    float sy, sx;
    if (int rc = wbd::check_shape(B, C, H, W, flowH, flowW, half, sy, sx)) return rc;
    CF_REQUIRE(sign == 1.f || sign == -1.f, CF_ERR_INVALID_ARG, "cf_warp_backward_det: sign must be +1 (backward warp) or -1 (forward warp)");
    cudaStream_t stream = (cudaStream_t)stream_;
    if (B == 0 || C == 0) {   // no channels: the flow gradient is zero (as cf_warp_backward's)
        if (grad_flow) CF_CUDA(cudaMemsetAsync(grad_flow, 0, sizeof(float) * (size_t)B * 2 * flowH * flowW, stream));
        return CF_OK;
    }
    const wbd::Layout L = wbd::layout(B, H, W, half != 0);
    CF_REQUIRE(workspace && workspace_bytes >= L.end + 256, CF_ERR_WORKSPACE,
               "cf_warp_backward_det: workspace too small (%zu < %zu)", workspace_bytes, L.end + 256);
    char *ws = reinterpret_cast<char *>(align_up(reinterpret_cast<uintptr_t>(workspace), 256));
    uint32_t *k0 = (uint32_t *)(ws + L.keys0), *v0 = (uint32_t *)(ws + L.vals0);
    uint32_t *k1 = (uint32_t *)(ws + L.keys1), *v1 = (uint32_t *)(ws + L.vals1);
    float *wts = (float *)(ws + L.wts);
    uint32_t *starts = (uint32_t *)(ws + L.starts), *hist = (uint32_t *)(ws + L.hist);
    float *gflow_half = half ? (float *)(ws + L.gflow) : nullptr;
    const int64_t plane = (int64_t)H * W, fplane = (int64_t)flowH * flowW;
    const unsigned groups = (unsigned)ceil_div(C, wbd::CPG);
    for (int b0 = 0; b0 < B; b0 += L.chunk) {
        const int items = B - b0 < L.chunk ? B - b0 : L.chunk;
        const int64_t pix = (int64_t)items * plane, n = 4 * pix;
        const float *go = grad_out + (size_t)b0 * C * plane;
        const unsigned pblk = (unsigned)ceil_div(pix, wbd::THREADS);
        wbd::warp_backward_det_taps_kernel<<<pblk, wbd::THREADS, 0, stream>>>(
            go, grad_flow ? img + (size_t)b0 * C * plane : nullptr, flow + (size_t)b0 * 2 * fplane, items, C, H, W,
            flowH, flowW, half, sy, sx, sign, grad_img ? (uint4 *)k0 : nullptr, (uint4 *)v0, (float4 *)wts,
            grad_flow ? grad_flow + (size_t)b0 * 2 * fplane : nullptr, gflow_half);
        CF_LAUNCH_CHECK("warp_backward_det_taps_kernel");
        if (grad_img) {
            const int nblk = (int)ceil_div(n, kRsTile);
            uint32_t *ka = k0, *va = v0, *kb = k1, *vb = v1;
            const int passes = (radix_bits((uint64_t)pix) + 7) / 8;   // keys 0 .. pix (pix = the invalid key)
            for (int p = 0; p < passes; ++p) {
                rs_hist_kernel<<<nblk, kRsThreads, 0, stream>>>(ka, n, 8 * p, hist, nblk);
                CF_LAUNCH_CHECK("rs_hist_kernel");
                rs_scan_kernel<<<1, 1024, 0, stream>>>(hist, (int64_t)256 * nblk);
                CF_LAUNCH_CHECK("rs_scan_kernel");
                rs_scatter_kernel<<<nblk, kRsThreads, 0, stream>>>(ka, va, kb, vb, n, 8 * p, hist, nblk);
                CF_LAUNCH_CHECK("rs_scatter_kernel");
                uint32_t *t = ka; ka = kb; kb = t;
                t = va; va = vb; vb = t;
            }
            wbd::warp_backward_det_bounds_kernel<<<(unsigned)ceil_div(n, wbd::THREADS), wbd::THREADS, 0, stream>>>(
                ka, n, (uint32_t)pix, starts);
            CF_LAUNCH_CHECK("warp_backward_det_bounds_kernel");
            wbd::warp_backward_det_gather_kernel<<<dim3(pblk, groups), wbd::THREADS, 0, stream>>>(
                va, wts, starts, go, grad_img + (size_t)b0 * C * plane, items, C, plane);
            CF_LAUNCH_CHECK("warp_backward_det_gather_kernel");
        }
        if (grad_flow && half) {
            wbd::warp_backward_det_flow_half_kernel<<<(unsigned)ceil_div((int64_t)items * fplane, wbd::THREADS), wbd::THREADS, 0, stream>>>(
                gflow_half, grad_flow + (size_t)b0 * 2 * fplane, items, H, W, flowH, flowW, sy, sx);
            CF_LAUNCH_CHECK("warp_backward_det_flow_half_kernel");
        }
    }
    return CF_OK;
}
