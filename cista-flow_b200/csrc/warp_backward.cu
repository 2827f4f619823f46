// Adjoint of the flow-guided warp (SURVEY.md section 8f rank 2): the true bilinear SPLAT.
//
// The reference trains through forwardWarp / backWarp with autograd (loss.py:147,155,208,217,241,247,336,
// 377,383,398,407; train.py:208-232): the backward of F.grid_sample(align_corners=True,
// padding_mode='reflection') w.r.t. the image is a scatter-add of grad_out * bilinear weight into the 4
// taps, and w.r.t. the flow the dot product of grad_out with the spatial differences of the taps, chained
// through reflect/clip (ATen grid_sampler_compute_source_index_set_grad) and the reference's
// g = 2 * ((x + sign * u) / W - 0.5) normalisation (utils/flow_utils.py:110-116,180-186).
//
// Round-1 version: one thread = one output pixel x a group of 32 channels; sample position, weights and
// gradient multipliers once; per channel 4 tap loads (for grad_flow), 4 fp32 RED.ADD into grad_img
// (resolved in L2) and, at the end, the pixel's flow gradient -- written, or added to the four
// full-resolution flow pixels when the x0.5 down-sampling of e2v/e2v_model.py:190 is fused (its adjoint).
// grad_img / grad_flow are zeroed here.  Sum order is unspecified (atomics), like ATen's CUDA backward; the
// fixed-order form, for torch.use_deterministic_algorithms(True), is warp_backward_det.cu.
// Next step (not done): privatise grad_img tiles in shared memory and flush once per tile.
#include "warp_common.cuh"

namespace cf {
namespace wb {
constexpr int THREADS = 256;
constexpr int CPG = 32;   // channels per thread

__global__ void __launch_bounds__(THREADS)
warp_backward_kernel(const float *__restrict__ grad_out, const float *__restrict__ img, const float *__restrict__ flow,
                     float *__restrict__ grad_img, float *__restrict__ grad_flow, int C, int H, int W, int fH, int fW,
                     int half, float sy, float sx, float sign) {
    const int b = blockIdx.z, group = blockIdx.y;
    const int64_t plane = (int64_t)H * W;
    const int p = blockIdx.x * THREADS + threadIdx.x;
    if (p >= plane) return;
    const int y = p / W, x = p - y * W;
    const float *fb = flow + (size_t)b * 2 * fH * fW;
    const float2 uv = flow_at(fb, x, y, W, fH, fW, half != 0, sy, sx, FlowLR{}, 0);
    const GradPos q = grad_pos(uv.x, uv.y, x, y, H, W, sign);
    const int x0 = q.x0, y0 = q.y0;
    const float ax1 = q.ax1, ax0 = q.ax0, ay1 = q.ay1, ay0 = q.ay0, mx = q.mx, my = q.my;
    const bool xin1 = q.xin1, yin1 = q.yin1;
    const int o00 = y0 * W + x0, o01 = o00 + 1, o10 = o00 + W, o11 = o10 + 1;
    const float w00 = ax1 * ay1, w01 = ax0 * ay1, w10 = ax1 * ay0, w11 = ax0 * ay0;

    const int c_begin = group * CPG, c_end = min(C, c_begin + CPG);
    const float *go = grad_out + ((size_t)b * C + c_begin) * plane + p;
    const float *im = img ? img + ((size_t)b * C + c_begin) * plane : nullptr;
    float *gi = grad_img ? grad_img + ((size_t)b * C + c_begin) * plane : nullptr;
    float gix = 0.f, giy = 0.f;
    for (int c = c_begin; c < c_end; ++c) {
        const float g = __ldg(go);
        if (gi) {
            atomicAdd(gi + o00, g * w00);
            if (xin1) atomicAdd(gi + o01, g * w01);
            if (yin1) atomicAdd(gi + o10, g * w10);
            if (xin1 && yin1) atomicAdd(gi + o11, g * w11);
            gi += plane;
        }
        if (grad_flow) {
            const float v00 = __ldg(im + o00), v01 = xin1 ? __ldg(im + o01) : 0.f;
            const float v10 = yin1 ? __ldg(im + o10) : 0.f, v11 = (xin1 && yin1) ? __ldg(im + o11) : 0.f;
            // ATen: gix -= nw*(iy_se - iy)*g; gix += ne*(iy_sw - iy)*g; gix -= sw*(iy - iy_ne)*g; gix += se*(iy - iy_nw)*g
            gix += g * (-v00 * ay1 + v01 * ay1 - v10 * ay0 + v11 * ay0);
            giy += g * (-v00 * ax1 - v01 * ax0 + v10 * ax1 + v11 * ax0);
            im += plane;
        }
        go += plane;
    }
    if (grad_flow) {
        // grad_grid = mult * g{ix,iy};  g = 2 * ((x + sign*u)/size - 0.5)  =>  d/du = sign * 2 / size
        const float gu = sign * (2.f * (mx * gix)) / (float)W, gv = sign * (2.f * (my * giy)) / (float)H;
        float *gfb = grad_flow + (size_t)b * 2 * fH * fW;
        const size_t fplane = (size_t)fH * fW;
        if (!half) {
            atomicAdd(gfb + p, gu);            // channel groups of the same pixel meet here
            atomicAdd(gfb + fplane + p, gv);
        } else {
            // adjoint of the x0.5 bilinear (align_corners=True) down-sampling: same taps / lambdas as flow_at()
            const HalfTaps t = half_taps(x, y, fH, fW, sy, sx);
            const int yy0 = t.y0, yy1 = t.y1, xx0 = t.x0, xx1 = t.x1;
            const float ly0 = t.ly0, ly1 = t.ly1, lx0 = t.lx0, lx1 = t.lx1;
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                float *c = gfb + k * fplane;
                const float g = k == 0 ? gu : gv;
                atomicAdd(c + yy0 * fW + xx0, g * ly0 * lx0);
                atomicAdd(c + yy0 * fW + xx1, g * ly0 * lx1);
                atomicAdd(c + yy1 * fW + xx0, g * ly1 * lx0);
                atomicAdd(c + yy1 * fW + xx1, g * ly1 * lx1);
            }
        }
    }
}
}  // namespace wb
}  // namespace cf

extern "C" int cf_warp_backward(const float *grad_out, const float *img, const float *flow, float *grad_img,
                                float *grad_flow, int B, int C, int H, int W, int flowH, int flowW, float sign,
                                cf_stream_t stream_) {
    using namespace cf;
    if (int rc = check_device()) return rc;
    CF_REQUIRE(grad_out && flow, CF_ERR_NULL, "cf_warp_backward: null pointer");
    CF_REQUIRE(grad_img || grad_flow, CF_ERR_NULL, "cf_warp_backward: neither grad_img nor grad_flow requested");
    CF_REQUIRE(!grad_flow || img, CF_ERR_NULL, "cf_warp_backward: grad_flow needs img");
    CF_REQUIRE(B >= 0 && C >= 0 && H > 0 && W > 0 && flowH > 0 && flowW > 0, CF_ERR_INVALID_ARG, "cf_warp_backward: bad shape");
    CF_REQUIRE(sign == 1.f || sign == -1.f, CF_ERR_INVALID_ARG, "cf_warp_backward: sign must be +1 (backward warp) or -1 (forward warp)");
    CF_REQUIRE((int64_t)H * W < (1ll << 30) && B <= 65535, CF_ERR_INVALID_ARG, "cf_warp_backward: too large");
    int half = 0;
    float sy = 0.f, sx = 0.f;
    if (flowH == H && flowW == W) {
        half = 0;
    } else if (H == flowH / 2 && W == flowW / 2) {
        half = 1;
        sy = H > 1 ? (float)(flowH - 1) / (float)(H - 1) : 0.f;
        sx = W > 1 ? (float)(flowW - 1) / (float)(W - 1) : 0.f;
    } else {
        set_error("cf_warp_backward: flow is %dx%d but the image is %dx%d (must be equal, or image == flow/2)", flowH, flowW, H, W);
        return CF_ERR_INVALID_ARG;
    }
    cudaStream_t stream = (cudaStream_t)stream_;
    if (grad_img) CF_CUDA(cudaMemsetAsync(grad_img, 0, sizeof(float) * (size_t)B * C * H * W, stream));
    if (grad_flow) CF_CUDA(cudaMemsetAsync(grad_flow, 0, sizeof(float) * (size_t)B * 2 * flowH * flowW, stream));
    if (B == 0 || C == 0) return CF_OK;
    const int groups = (int)ceil_div(C, wb::CPG);
    CF_REQUIRE(groups <= 65535, CF_ERR_INVALID_ARG, "cf_warp_backward: too many channels");
    dim3 grid((unsigned)ceil_div((int64_t)H * W, wb::THREADS), (unsigned)groups, (unsigned)B);
    wb::warp_backward_kernel<<<grid, wb::THREADS, 0, stream>>>(grad_out, img, flow, grad_img, grad_flow, C, H, W, flowH, flowW,
                                                               half, sy, sx, sign);
    CF_LAUNCH_CHECK("warp_backward_kernel");
    return CF_OK;
}
