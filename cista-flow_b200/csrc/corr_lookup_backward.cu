// Adjoint of the correlation pyramid lookup (SURVEY.md section 8f rank 2).
//
// The reference trains through CorrBlock.__call__ (ERAFT/corr.py:29-50, raft_corr.py:32-54) with autograd:
// grid_sample backward scatters into the pyramid and differentiates w.r.t. the sampling coordinates.
// Because every query owns its private h_l x w_l map and all (2r+1)^2 samples of a level share one pair of
// fractional weights, the gradient of a level's (2r+2)^2 patch is a 2x2 correlation of the (2r+1)^2 window
// of output gradients with the bilinear weights -- a GATHER: no atomics, every patch element is written
// once (the rest of the map stays zero from the memset).  The coordinate gradient is
//   d out[l,i,j] / d x = 2^-l * ((p01 - p00) (1 - fy) + (p11 - p10) fy)     (zeros padding, pixel coordinates:
//   the reference's 2x/(W-1)-1 normalisation and align_corners=True un-normalisation cancel).
// Channel l*(2r+1)^2 + i*(2r+1) + j moves i along x (the transposed window, SURVEY F7).
// One CTA = 16 queries of one batch item: patches (as in the forward kernel) and the queries' output
// gradients are staged in shared memory, then thread <-> patch element / thread <-> (query, channel).  Where 16
// queries' patches and gradients exceed the shared memory (6 levels at radius 8: 236 KB), a CTA takes 8 queries and
// 32 threads share each query's channels.  The threads of a query leave their partial coordinate gradients in shared
// memory and the query's owner thread adds them in thread order: the sum order is fixed, the result reproducible.
#include "common.cuh"

namespace cf {
namespace lb {
constexpr int THREADS = 256;
constexpr size_t SMEM_CAP = 200 * 1024;

struct Pyramid {
    const float *ptr[CF_CORR_MAX_LEVELS];
    float *grad[CF_CORR_MAX_LEVELS];
    int H[CF_CORR_MAX_LEVELS];
    int W[CF_CORR_MAX_LEVELS];
};

template <int QT>
__global__ void __launch_bounds__(THREADS)
corr_lookup_backward_kernel(const __grid_constant__ Pyramid pyr, const float *__restrict__ coords,
                            const float *__restrict__ grad_out, float *__restrict__ grad_coords, int N, int levels, int r,
                            int want_pyr) {
    extern __shared__ float smem[];
    const int K = 2 * r + 1, P = K + 1, KK = K * K, PP = P * P;
    const int LPP = levels * PP, CT = levels * KK;
    const int PS = LPP | 1, GS = CT | 1;        // odd strides between queries
    float *patch = smem;                        // [QT][PS]
    float *go = patch + (size_t)QT * PS;        // [QT][GS]
    float *cxy = go + (size_t)QT * GS;          // [QT][2]
    float *part = cxy + 2 * QT;                 // [THREADS][2] partial coordinate gradients
    const int tid = threadIdx.x, b = blockIdx.y, q0 = blockIdx.x * QT;
    const float *cb = coords + (size_t)b * 2 * N;
    if (tid < QT) {
        const int q = q0 + tid;
        cxy[2 * tid] = q < N ? fminf(fmaxf(__ldg(cb + q), -1.0e6f), 1.0e6f) : 0.f;
        cxy[2 * tid + 1] = q < N ? fminf(fmaxf(__ldg(cb + N + q), -1.0e6f), 1.0e6f) : 0.f;
    }
    // output gradients of the CTA's queries: 16 consecutive queries of a channel are 64 contiguous bytes
    const float *gob = grad_out + (size_t)b * CT * N;
    for (int idx = tid; idx < QT * CT; idx += THREADS) {
        const int c = idx / QT, qi = idx - c * QT;
        go[qi * GS + c] = q0 + qi < N ? __ldg(gob + (size_t)c * N + q0 + qi) : 0.f;
    }
    __syncthreads();
    // patches (zero outside the map), needed for the coordinate gradient
    if (grad_coords) {
        for (int idx = tid; idx < QT * LPP; idx += THREADS) {
            const int qi = idx / LPP, e = idx - qi * LPP;
            const int l = e / PP, rem = e - l * PP;
            const int py = rem / P, px = rem - py * P;
            const float inv = 1.f / (float)(1 << l);
            const int X = (int)floorf(cxy[2 * qi] * inv) - r + px, Y = (int)floorf(cxy[2 * qi + 1] * inv) - r + py;
            const int Hl = pyr.H[l], Wl = pyr.W[l], q = q0 + qi;
            float v = 0.f;
            if (q < N && X >= 0 && X < Wl && Y >= 0 && Y < Hl) v = __ldg(pyr.ptr[l] + (((size_t)b * N + q) * Hl + Y) * Wl + X);
            patch[qi * PS + e] = v;
        }
        __syncthreads();
        // thread <-> (query, channels c_first, c_first + c_step, ...) as in the forward kernel
        const int qi = tid % QT;
        float ax = 0.f, ay = 0.f;
        for (int l = 0; l < levels; ++l) {
            const float inv = 1.f / (float)(1 << l);
            const float sx = cxy[2 * qi] * inv, sy = cxy[2 * qi + 1] * inv;
            const float fx = sx - floorf(sx), fy = sy - floorf(sy);
            const float *pl = patch + qi * PS + l * PP;
            for (int c = tid / QT; c < KK; c += THREADS / QT) {
                const int i = c / K, j = c - i * K;
                const float *pp = pl + j * P + i;
                const float p00 = pp[0], p01 = pp[1], p10 = pp[P], p11 = pp[P + 1];
                const float g = go[qi * GS + l * KK + c] * inv;
                ax += g * ((p01 - p00) * (1.f - fy) + (p11 - p10) * fy);
                ay += g * ((p10 - p00) * (1.f - fx) + (p11 - p01) * fx);
            }
        }
        part[2 * tid] = ax;
        part[2 * tid + 1] = ay;
        __syncthreads();
        if (tid < QT && q0 + tid < N) {   // threads tid, tid + QT, tid + 2 QT, ... hold this query's partials
            float sx = 0.f, sy = 0.f;
            for (int t = tid; t < THREADS; t += QT) {
                sx += part[2 * t];
                sy += part[2 * t + 1];
            }
            grad_coords[(size_t)b * 2 * N + q0 + tid] = sx;
            grad_coords[(size_t)b * 2 * N + N + q0 + tid] = sy;
        }
    }
    // patch gradients: 2x2 correlation of the window of output gradients with the bilinear weights
    if (want_pyr) {
        for (int idx = tid; idx < QT * LPP; idx += THREADS) {
            const int qi = idx / LPP, e = idx - qi * LPP;
            const int l = e / PP, rem = e - l * PP;
            const int py = rem / P, px = rem - py * P;
            const int q = q0 + qi;
            if (q >= N) continue;
            const float inv = 1.f / (float)(1 << l);
            const float sx = cxy[2 * qi] * inv, sy = cxy[2 * qi + 1] * inv;
            const float fx = sx - floorf(sx), fy = sy - floorf(sy);
            const int X = (int)floorf(sx) - r + px, Y = (int)floorf(sy) - r + py;
            const int Hl = pyr.H[l], Wl = pyr.W[l];
            if (X < 0 || X >= Wl || Y < 0 || Y >= Hl) continue;
            const float *g = go + qi * GS + l * KK;
            float acc = 0.f;   // sample (i, j) reads patch (j + dy, i + dx) with weight w[dy][dx]
            if (px < K && py < K) acc += g[px * K + py] * ((1.f - fx) * (1.f - fy));
            if (px >= 1 && py < K) acc += g[(px - 1) * K + py] * (fx * (1.f - fy));
            if (px < K && py >= 1) acc += g[px * K + py - 1] * ((1.f - fx) * fy);
            if (px >= 1 && py >= 1) acc += g[(px - 1) * K + py - 1] * (fx * fy);
            pyr.grad[l][(((size_t)b * N + q) * Hl + Y) * Wl + X] = acc;
        }
    }
}
}  // namespace lb
}  // namespace cf

extern "C" int cf_corr_lookup_backward(const float *grad_out, const float *const *pyramid, const float *coords, int B, int h,
                                       int w, int levels, int radius, float *const *grad_pyramid, float *grad_coords,
                                       cf_stream_t stream_) {
    using namespace cf;
    if (int rc = check_device()) return rc;
    CF_REQUIRE(grad_out && coords, CF_ERR_NULL, "cf_corr_lookup_backward: null pointer");
    CF_REQUIRE(grad_pyramid || grad_coords, CF_ERR_NULL, "cf_corr_lookup_backward: no gradient requested");
    CF_REQUIRE(!grad_coords || pyramid, CF_ERR_NULL, "cf_corr_lookup_backward: grad_coords needs the pyramid");
    CF_REQUIRE(levels >= 1 && levels <= CF_CORR_MAX_LEVELS && radius >= 0 && radius <= 8, CF_ERR_INVALID_ARG,
               "cf_corr_lookup_backward: levels=%d radius=%d out of range", levels, radius);
    CF_REQUIRE(B >= 0 && B <= 65535 && h > 0 && w > 0 && (h >> (levels - 1)) >= 1 && (w >> (levels - 1)) >= 1, CF_ERR_INVALID_ARG,
               "cf_corr_lookup_backward: bad shape B=%d h=%d w=%d", B, h, w);
    if (B == 0) return CF_OK;
    cudaStream_t stream = (cudaStream_t)stream_;
    const int N = h * w;
    lb::Pyramid pyr{};
    for (int l = 0; l < levels; ++l) {
        pyr.H[l] = h >> l;
        pyr.W[l] = w >> l;
        pyr.ptr[l] = pyramid ? pyramid[l] : nullptr;
        CF_REQUIRE(!grad_coords || pyr.ptr[l], CF_ERR_NULL, "cf_corr_lookup_backward: pyramid[%d] is null", l);
        pyr.grad[l] = grad_pyramid ? grad_pyramid[l] : nullptr;
        if (grad_pyramid) {
            CF_REQUIRE(pyr.grad[l], CF_ERR_NULL, "cf_corr_lookup_backward: grad_pyramid[%d] is null", l);
            CF_CUDA(cudaMemsetAsync(pyr.grad[l], 0, sizeof(float) * (size_t)B * N * pyr.H[l] * pyr.W[l], stream));
        }
    }
    const int K = 2 * radius + 1, P = K + 1;
    auto smem_bytes = [&](int qt) {
        return ((size_t)qt * (((levels * P * P) | 1) + ((levels * K * K) | 1)) + 2 * qt + 2 * lb::THREADS) * sizeof(float);
    };
    const int qt = smem_bytes(16) <= lb::SMEM_CAP ? 16 : 8;
    const size_t smem = smem_bytes(qt);
    CF_REQUIRE(smem <= lb::SMEM_CAP, CF_ERR_INVALID_ARG, "cf_corr_lookup_backward: levels*radius too large for shared memory");
    int dev = 0;
    CF_CUDA(cudaGetDevice(&dev));
    static bool opt_in[64] = {};
    if (!opt_in[dev & 63]) {
        CF_CUDA(cudaFuncSetAttribute(lb::corr_lookup_backward_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lb::SMEM_CAP));
        CF_CUDA(cudaFuncSetAttribute(lb::corr_lookup_backward_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lb::SMEM_CAP));
        opt_in[dev & 63] = true;
    }
    dim3 grid((unsigned)ceil_div(N, qt), (unsigned)B);
    if (qt == 16)
        lb::corr_lookup_backward_kernel<16><<<grid, lb::THREADS, smem, stream>>>(pyr, coords, grad_out, grad_coords, N, levels,
                                                                             radius, grad_pyramid ? 1 : 0);
    else
        lb::corr_lookup_backward_kernel<8><<<grid, lb::THREADS, smem, stream>>>(pyr, coords, grad_out, grad_coords, N, levels,
                                                                            radius, grad_pyramid ? 1 : 0);
    CF_LAUNCH_CHECK("corr_lookup_backward_kernel");
    return CF_OK;
}
