// All-pairs correlation volume + average-pool pyramid (part 3a of the hot path).
//
// Replaces CorrBlock.__init__ / CorrBlock.corr of the reference
// (ERAFT/corr.py:13-27,52-60 == DCEIFlow/core/corr/raft_corr.py:16-30,56-65):
//   vol[b,i,j] = <fmap1[b,:,i], fmap2[b,:,j]> / sqrt(D)      (one GEMM per item)
//   level l+1  = avg_pool2d(level l, 2, stride 2) over the target dims (floor)
//
// Data layout: fmap [B,D,N] (N = h*w contiguous: both GEMM operands are
// "MN-major"), level l [B*N, h>>l, w>>l] fp32.
//
// This file holds the host entry point, the fp32 SIMT contraction
// (CF_CORR_FP32: the reference's arithmetic, used as the tight-tolerance
// cross-check) and the pooling kernel.  The tensor-core contraction
// (CF_CORR_TF32 / CF_CORR_3XTF32: TMA -> smem -> tcgen05.mma -> TMEM -> fused
// scale + level-1 pooling epilogue) lives in corr_build_tc.cu.
#include <cuda_fp16.h>
#include <stdlib.h>

#include "common.cuh"
#include "cistaflow_half.h"

namespace cf {

// implemented in corr_build_tc.cu
int corr_volume_tensor_core(const float *f1, const float *f2, int B, int D, int h, int w, float scale,
                            float *level0, float *level1, float *level2, float *level3, int precision, void *ws,
                            size_t ws_bytes, int flags, int *fused_levels, cudaStream_t stream, bool half_out);
bool corr_tensor_core_supported(int D, int h, int w);
size_t corr_tc_workspace_bytes(int B, int D, int h, int w);
size_t corr_x3_workspace_bytes(int B, int D, int h, int w);

// CF_TC_FLAGS (debug / experiments only, see corr_build_tc.cu)
static int tc_flags() {
    static int flags = -1;
    if (flags < 0) {
        const char *e = getenv("CF_TC_FLAGS");
        flags = e ? atoi(e) : 0;
    }
    return flags;
}

// ---- fp32 SIMT GEMM: 64x64 tile, 256 threads, 4x4 outputs per thread --------
constexpr int kTile = 64, kBK = 16;

__global__ void __launch_bounds__(256)
corr_volume_fp32_kernel(const float *__restrict__ f1, const float *__restrict__ f2, float *__restrict__ vol,
                        int D, int N, float scale) {
    __shared__ __align__(16) float As[kBK][kTile];
    __shared__ __align__(16) float Bs[kBK][kTile];
    const int b = blockIdx.z, i0 = blockIdx.y * kTile, j0 = blockIdx.x * kTile;
    const float *a = f1 + (size_t)b * D * N, *bm = f2 + (size_t)b * D * N;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    float acc[4][4] = {};
    for (int k0 = 0; k0 < D; k0 += kBK) {
#pragma unroll
        for (int r = 0; r < (kBK * kTile) / 256; ++r) {
            const int idx = threadIdx.x + r * 256;
            const int kk = idx / kTile, m = idx % kTile;
            const bool kin = k0 + kk < D;
            As[kk][m] = (kin && i0 + m < N) ? __ldg(a + (size_t)(k0 + kk) * N + i0 + m) : 0.f;
            Bs[kk][m] = (kin && j0 + m < N) ? __ldg(bm + (size_t)(k0 + kk) * N + j0 + m) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < kBK; ++kk) {
            const float4 av = *reinterpret_cast<const float4 *>(&As[kk][ty * 4]);
            const float4 bv = *reinterpret_cast<const float4 *>(&Bs[kk][tx * 4]);
            const float ar[4] = {av.x, av.y, av.z, av.w}, br[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[r][c] = fmaf(ar[r], br[c], acc[r][c]);
        }
        __syncthreads();
    }
    float *o = vol + (size_t)b * N * N;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int i = i0 + ty * 4 + r;
        if (i >= N) continue;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int j = j0 + tx * 4 + c;
            if (j < N) o[(size_t)i * N + j] = acc[r][c] * scale;
        }
    }
}

// ---- avg_pool2d(2, stride 2), floor on odd sizes -----------------------------
// maps: M images [Hi, Wi] -> [Ho, Wo];  ATen order: ((a + b) + c) + d, then / 4.
// The bodies are shared by the fp32 pyramid and the fp16 one (cf_corr_build_half): an fp16 level is read widened to fp32,
// summed in the same order and rounded to nearest once, so each level is the 2x2 mean of the level above AS STORED.
__device__ __forceinline__ float pool_ld(const float *p) { return __ldg(p); }
__device__ __forceinline__ float pool_ld(const __half *p) { return __half2float(__ldg(p)); }
__device__ __forceinline__ void pool_st(float *p, float v) { *p = v; }
__device__ __forceinline__ void pool_st(__half *p, float v) { *p = __float2half_rn(v); }
__device__ __forceinline__ float pool_stored(const float *, float v) { return v; }
__device__ __forceinline__ float pool_stored(const __half *, float v) { return __half2float(__float2half_rn(v)); }

template <typename T>
__device__ __forceinline__ void avg_pool2x2(const T *__restrict__ in, T *__restrict__ out, int64_t total_out,
                                            int Hi, int Wi, int Ho, int Wo) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; o < total_out; o += stride) {
        const int xo = (int)(o % Wo);
        const int64_t t = o / Wo;
        const int yo = (int)(t % Ho);
        const int64_t m = t / Ho;
        const T *p = in + (m * Hi + 2 * yo) * Wi + 2 * xo;
        float s = pool_ld(p) + pool_ld(p + 1);
        s += pool_ld(p + Wi);
        s += pool_ld(p + Wi + 1);
        pool_st(out + o, s / 4.f);
    }
}
__global__ void __launch_bounds__(256)
avg_pool2x2_kernel(const float *__restrict__ in, float *__restrict__ out, int64_t total_out,
                   int Hi, int Wi, int Ho, int Wo) {
    avg_pool2x2(in, out, total_out, Hi, Wi, Ho, Wo);
}
__global__ void __launch_bounds__(256)
avg_pool2x2_half_kernel(const __half *__restrict__ in, __half *__restrict__ out, int64_t total_out,
                        int Hi, int Wi, int Ho, int Wo) {
    avg_pool2x2(in, out, total_out, Hi, Wi, Ho, Wo);
}

// level l+1 AND level l+2 from level l in one launch (the two smallest pyramid levels): one thread
// per 2x2 group of level-(l+1) cells; floor semantics on odd sizes are kept exactly.
template <typename T>
__device__ __forceinline__ void avg_pool_two_levels(const T *__restrict__ in, T *__restrict__ out1, T *__restrict__ out2,
                                                    int64_t groups, int Hi, int Wi, int H1, int W1, int H2, int W2) {
    const int GH = (H1 + 1) / 2, GW = (W1 + 1) / 2;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += stride) {
        const int X = (int)(g % GW);
        const int64_t t = g / GW;
        const int Y = (int)(t % GH);
        const int64_t m = t / GH;
        float v[2][2] = {};
#pragma unroll
        for (int dy = 0; dy < 2; ++dy)
#pragma unroll
            for (int dx = 0; dx < 2; ++dx) {
                const int y1 = 2 * Y + dy, x1 = 2 * X + dx;
                if (y1 < H1 && x1 < W1) {
                    const T *p = in + (m * Hi + 2 * y1) * Wi + 2 * x1;
                    float s = pool_ld(p) + pool_ld(p + 1);
                    s += pool_ld(p + Wi);
                    s += pool_ld(p + Wi + 1);
                    v[dy][dx] = pool_stored(in, s / 4.f);
                    pool_st(out1 + (m * H1 + y1) * W1 + x1, v[dy][dx]);
                }
            }
        if (Y < H2 && X < W2) {
            float s = v[0][0] + v[0][1];
            s += v[1][0];
            s += v[1][1];
            pool_st(out2 + (m * H2 + Y) * W2 + X, s / 4.f);
        }
    }
}
__global__ void __launch_bounds__(256)
avg_pool_two_levels_kernel(const float *__restrict__ in, float *__restrict__ out1, float *__restrict__ out2, int64_t groups,
                           int Hi, int Wi, int H1, int W1, int H2, int W2) {
    avg_pool_two_levels(in, out1, out2, groups, Hi, Wi, H1, W1, H2, W2);
}
__global__ void __launch_bounds__(256)
avg_pool_two_levels_half_kernel(const __half *__restrict__ in, __half *__restrict__ out1, __half *__restrict__ out2,
                                int64_t groups, int Hi, int Wi, int H1, int W1, int H2, int W2) {
    avg_pool_two_levels(in, out1, out2, groups, Hi, Wi, H1, W1, H2, W2);
}

static void pool_launch(const float *in, float *out1, float *out2, int64_t n, unsigned g, int Hi, int Wi, int H1, int W1,
                        int H2, int W2, cudaStream_t stream) {
    if (out2) avg_pool_two_levels_kernel<<<g, 256, 0, stream>>>(in, out1, out2, n, Hi, Wi, H1, W1, H2, W2);
    else avg_pool2x2_kernel<<<g, 256, 0, stream>>>(in, out1, n, Hi, Wi, H1, W1);
}
static void pool_launch(const __half *in, __half *out1, __half *out2, int64_t n, unsigned g, int Hi, int Wi, int H1, int W1,
                        int H2, int W2, cudaStream_t stream) {
    if (out2) avg_pool_two_levels_half_kernel<<<g, 256, 0, stream>>>(in, out1, out2, n, Hi, Wi, H1, W1, H2, W2);
    else avg_pool2x2_half_kernel<<<g, 256, 0, stream>>>(in, out1, n, Hi, Wi, H1, W1);
}
static const char *pool_name(const float *, bool two) { return two ? "avg_pool_two_levels_kernel" : "avg_pool2x2_kernel"; }
static const char *pool_name(const __half *, bool two) { return two ? "avg_pool_two_levels_half_kernel" : "avg_pool2x2_half_kernel"; }

// levels first_pooled .. levels-1 by the pooling kernels, two per launch while two remain
template <typename T>
static int pool_levels(T *const *pyramid, int first_pooled, int levels, int B, int h, int w, cudaStream_t stream) {
    const int N = h * w;
    for (int l = first_pooled; l < levels; ++l) {
        const bool two = l + 1 < levels;
        const int Hi = h >> (l - 1), Wi = w >> (l - 1), H1 = h >> l, W1 = w >> l;
        const int H2 = two ? h >> (l + 1) : 0, W2 = two ? w >> (l + 1) : 0;
        const int64_t n = two ? (int64_t)B * N * ((H1 + 1) / 2) * ((W1 + 1) / 2) : (int64_t)B * N * H1 * W1;
        const int64_t blocks = ceil_div(n, 256);
        const unsigned g = (unsigned)(blocks < (int64_t)148 * 32 ? blocks : (int64_t)148 * 32);
        pool_launch(pyramid[l - 1], pyramid[l], two ? pyramid[l + 1] : nullptr, n, g, Hi, Wi, H1, W1, H2, W2, stream);
        CF_LAUNCH_CHECK(pool_name(pyramid[0], two));
        if (two) ++l;
    }
    return CF_OK;
}

}  // namespace cf

extern "C" size_t cf_corr_workspace_bytes(int B, int D, int h, int w, int, int precision) {
    if (B <= 0 || D <= 0 || h <= 0 || w <= 0) return 0;
    if (precision == CF_CORR_3XTF32) return cf::corr_x3_workspace_bytes(B, D, h, w);
    if (precision != CF_CORR_F16 && precision != CF_CORR_AUTO) return 0;
    return cf::corr_tc_workspace_bytes(B, D, h, w);
}

extern "C" int cf_corr_build(const float *fmap1, const float *fmap2, int B, int D, int h, int w, int levels,
                             float *const *pyramid, int precision, void *ws, size_t ws_bytes, cf_stream_t stream_) {
    using namespace cf;
    if (int rc = check_device()) return rc;
    CF_REQUIRE(fmap1 && fmap2 && pyramid, CF_ERR_NULL, "cf_corr_build: null pointer");
    CF_REQUIRE(levels >= 1 && levels <= CF_CORR_MAX_LEVELS, CF_ERR_INVALID_ARG,
               "cf_corr_build: levels=%d not in [1,%d]", levels, CF_CORR_MAX_LEVELS);
    CF_REQUIRE(B >= 0 && B <= 65535 && D > 0 && h > 0 && w > 0, CF_ERR_INVALID_ARG,
               "cf_corr_build: bad shape B=%d D=%d h=%d w=%d", B, D, h, w);
    CF_REQUIRE((h >> (levels - 1)) >= 1 && (w >> (levels - 1)) >= 1, CF_ERR_INVALID_ARG,
               "cf_corr_build: %dx%d feature map is too small for %d levels", h, w, levels);
    CF_REQUIRE(precision >= CF_CORR_TF32 && precision <= CF_CORR_AUTO, CF_ERR_INVALID_ARG,
               "cf_corr_build: bad precision %d", precision);
    for (int l = 0; l < levels; ++l) CF_REQUIRE(pyramid[l], CF_ERR_NULL, "cf_corr_build: pyramid[%d] is null", l);
    if (B == 0) return CF_OK;
    cudaStream_t stream = (cudaStream_t)stream_;
    const int N = h * w;
    CF_REQUIRE((int64_t)N * N < (1ll << 40), CF_ERR_INVALID_ARG, "cf_corr_build: volume too large");
    const float scale = 1.0f / sqrtf((float)D);

    int first_pooled = 1;  // first level the pooling kernel still has to produce
    if (precision == CF_CORR_FP32) {
        dim3 grid((unsigned)ceil_div(N, kTile), (unsigned)ceil_div(N, kTile), B);
        corr_volume_fp32_kernel<<<grid, 256, 0, stream>>>(fmap1, fmap2, pyramid[0], D, N, scale);
        CF_LAUNCH_CHECK("corr_volume_fp32_kernel");
    } else {
        CF_REQUIRE(corr_tensor_core_supported(D, h, w), CF_ERR_UNSUPPORTED,
                   "cf_corr_build: the tensor-core path needs D %% 32 == 0 and h*w %% 4 == 0 (got D=%d, h=%d, w=%d); "
                   "use CF_CORR_FP32", D, h, w);
        int fused = 0;  // pyramid levels beyond level 0 that the GEMM's epilogue produced
        if (int rc = corr_volume_tensor_core(fmap1, fmap2, B, D, h, w, scale, pyramid[0],
                                             levels > 1 ? pyramid[1] : nullptr, levels > 2 ? pyramid[2] : nullptr,
                                             levels > 3 ? pyramid[3] : nullptr, precision, ws, ws_bytes,
                                             tc_flags(), &fused, stream, false)) return rc;
        first_pooled = 1 + fused;
    }
    return pool_levels(pyramid, first_pooled, levels, B, h, w, stream);
}

extern "C" int cf_corr_build_half(const float *fmap1, const float *fmap2, int B, int D, int h, int w, int levels,
                                  uint16_t *const *pyramid, int precision, void *ws, size_t ws_bytes, cf_stream_t stream_) {
    using namespace cf;
    if (int rc = check_device()) return rc;
    CF_REQUIRE(fmap1 && fmap2 && pyramid, CF_ERR_NULL, "cf_corr_build_half: null pointer");
    CF_REQUIRE(levels >= 1 && levels <= CF_CORR_MAX_LEVELS, CF_ERR_INVALID_ARG,
               "cf_corr_build_half: levels=%d not in [1,%d]", levels, CF_CORR_MAX_LEVELS);
    CF_REQUIRE(B >= 0 && B <= 65535 && D > 0 && h > 0 && w > 0, CF_ERR_INVALID_ARG,
               "cf_corr_build_half: bad shape B=%d D=%d h=%d w=%d", B, D, h, w);
    CF_REQUIRE((h >> (levels - 1)) >= 1 && (w >> (levels - 1)) >= 1, CF_ERR_INVALID_ARG,
               "cf_corr_build_half: %dx%d feature map is too small for %d levels", h, w, levels);
    CF_REQUIRE(precision >= CF_CORR_TF32 && precision <= CF_CORR_AUTO, CF_ERR_INVALID_ARG,
               "cf_corr_build_half: bad precision %d", precision);
    CF_REQUIRE(precision != CF_CORR_FP32 && precision != CF_CORR_3XTF32, CF_ERR_UNSUPPORTED,
               "cf_corr_build_half: precision %d is fp32-accurate, which fp16 storage would lose; "
               "use CF_CORR_TF32, CF_CORR_F16 or CF_CORR_AUTO", precision);
    CF_REQUIRE(D % 32 == 0, CF_ERR_UNSUPPORTED, "cf_corr_build_half: needs D %% 32 == 0 (got D=%d)", D);
    CF_REQUIRE(((int64_t)h * w) % 8 == 0, CF_ERR_UNSUPPORTED,
               "cf_corr_build_half: needs h*w %% 8 == 0 for a 16-byte row pitch of the fp16 volume (got %dx%d)", h, w);
    for (int l = 0; l < levels; ++l) CF_REQUIRE(pyramid[l], CF_ERR_NULL, "cf_corr_build_half: pyramid[%d] is null", l);
    if (B == 0) return CF_OK;
    cudaStream_t stream = (cudaStream_t)stream_;
    const int N = h * w;
    CF_REQUIRE((int64_t)N * N < (1ll << 40), CF_ERR_INVALID_ARG, "cf_corr_build_half: volume too large");
    const float scale = 1.0f / sqrtf((float)D);
    float *lv[4] = {};
    for (int l = 0; l < 4 && l < levels; ++l) lv[l] = reinterpret_cast<float *>(pyramid[l]);
    int fused = 0;
    if (int rc = corr_volume_tensor_core(fmap1, fmap2, B, D, h, w, scale, lv[0], lv[1], lv[2], lv[3], precision, ws, ws_bytes,
                                         0, &fused, stream, true)) return rc;
    return pool_levels(reinterpret_cast<__half *const *>(pyramid), 1 + fused, levels, B, h, w, stream);
}
