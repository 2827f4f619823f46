// Correlation pyramid lookup (part 3b of the hot path).
//
// Replaces CorrBlock.__call__ (ERAFT/corr.py:29-50 == DCEIFlow/core/corr/
// raft_corr.py:32-54) and its bilinear_sampler (ERAFT/utils.py:7-21): for each
// query pixel q and pyramid level l the reference samples a (2r+1)^2 window
// around coords[q]/2^l with grid_sample(align_corners=True, zeros padding).
// The window offsets are integers, so all (2r+1)^2 samples of a level share
// one pair of fractional weights and read one (2r+2)^2 patch: the kernel loads
// the patch once (zero-filled outside the map) and forms the samples from
// shared memory.  The window is TRANSPOSED as in the reference (SURVEY.md F7):
// channel l*(2r+1)^2 + i*(2r+1) + j samples (x + i - r, y + j - r).
//
// Data layout: pyramid[l] [B*N, 1, h>>l, w>>l], coords [B,2,h,w], out
// [B, L*(2r+1)^2, h, w]; fp32.  Roofline: HBM (L2 when the pyramid was just
// built).  Algorithmic bytes per query: 4*L*(2r+1)^2 written + 8 read (coords)
// + 4*L*(2r+2)^2 read (patches) = 2904 B at L=4, r=4.
//
// Mapping: one CTA = QT (16 or 32) consecutive queries of one batch item.
//   phase A  all 256 threads fetch the QT*L patches (QT*400 independent 4-byte
//            loads at L=4, r=4, ~50 per thread, issued in unrolled batches so
//            that thousands of loads are in flight per SM: the kernel is
//            latency-bound, not bandwidth-bound, at feature-map sizes) into a
//            shared [query][level][P][P] array with an odd row stride;
//   phase B  thread <-> (query = lane, channel); the four weights of a level are
//            computed once per level and thread; every channel is 4 LDS + 4 FMA
//            and ONE coalesced store: the 32 lanes of a warp hold 32 consecutive
//            queries of the same channel = one 128-byte line of the
//            channel-major output.  No output staging, no bank conflicts (odd
//            stride => lanes hit distinct banks).
#include <cuda_fp16.h>
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"
#include "cistaflow_half.h"

namespace cf {

struct Pyramid {
    const float *ptr[CF_CORR_MAX_LEVELS];
    int H[CF_CORR_MAX_LEVELS];
    int W[CF_CORR_MAX_LEVELS];
};
// an fp16 pyramid (cf_corr_lookup_half): the kernels' bodies are shared, a tap is widened to fp32 as it is loaded
struct PyramidHalf {
    const __half *ptr[CF_CORR_MAX_LEVELS];
    int H[CF_CORR_MAX_LEVELS];
    int W[CF_CORR_MAX_LEVELS];
};
__device__ __forceinline__ float tap_ld(const float *p) { return __ldg(p); }
__device__ __forceinline__ float tap_ld(const __half *p) { return __half2float(__ldg(p)); }

constexpr int kLookupThreads = 256;

// ---- the models' configuration (4 levels, radius 4) -----------------------------------------
// The kernel is instruction-issue and latency bound at feature-map sizes (6 144 queries at
// configs[1]); both phases are written for few instructions per element:
//   phase A  warp <-> query, lane <-> (patch column = lane % 10, row group = lane / 10): a lane walks
//            rows rg, rg+3, rg+6, rg+9 of its column, so the x bound, the column address and the
//            shared-memory slot are loop constants and a row costs one compare + one predicated LDG;
//            the 16 loads of a query (two queries per pass: 32 per lane) are issued before the
//            first shared-memory store;
//   phase B  thread <-> (query = lane, level, group of window columns i): the 9 samples of a window
//            column share their horizontal interpolation, so a column is 20 LDS + 10 horizontal + 9
//            vertical lerps and 9 coalesced stores (32 lanes = 32 consecutive queries of one channel
//            = one 128-byte line of the channel-major output) instead of 36 LDS + 36 FMA.
// QT (queries per CTA, even, <= 32) is a run-time argument: the host picks the value that balances the CTAs over the
// SMs (see launch_lookup_r4l4).
// QT_CT = 16: compile-time value for the latency-bound small-problem case (5.2 against 5.5 us at configs[1]);
// QT_CT = 0: run-time value (compile-time values for the larger counts were measured slower: the unrolled
// multi-pair gather costs occupancy -- 64x24x32 34.7 against 31.5 us).
#define CF_LOOKUP_PYR Pyramid
#define CF_LOOKUP_T float
#define CF_LOOKUP_R4L4 corr_lookup_r4l4_kernel
#define CF_LOOKUP_GENERIC corr_lookup_kernel
#include "corr_lookup_kernels.cuh"
#undef CF_LOOKUP_PYR
#undef CF_LOOKUP_T
#undef CF_LOOKUP_R4L4
#undef CF_LOOKUP_GENERIC
#define CF_LOOKUP_PYR PyramidHalf
#define CF_LOOKUP_T __half
#define CF_LOOKUP_R4L4 corr_lookup_r4l4_half_kernel
#define CF_LOOKUP_GENERIC corr_lookup_half_kernel
#include "corr_lookup_kernels.cuh"
#undef CF_LOOKUP_PYR
#undef CF_LOOKUP_T
#undef CF_LOOKUP_R4L4
#undef CF_LOOKUP_GENERIC

CF_DEFINE_TRACE_SETTER(cf_trace_buffer_lookup)

static void r4l4_launch(const Pyramid &pyr, dim3 grid, size_t smem, const float *coords, float *out, int N, int qt,
                        cudaStream_t stream) {
    if (qt == 16) corr_lookup_r4l4_kernel<16><<<grid, kLookupThreads, smem, stream>>>(pyr, coords, out, N, qt);
    else corr_lookup_r4l4_kernel<0><<<grid, kLookupThreads, smem, stream>>>(pyr, coords, out, N, qt);
}
static void r4l4_launch(const PyramidHalf &pyr, dim3 grid, size_t smem, const float *coords, float *out, int N, int qt,
                        cudaStream_t stream) {
    if (qt == 16) corr_lookup_r4l4_half_kernel<16><<<grid, kLookupThreads, smem, stream>>>(pyr, coords, out, N, qt);
    else corr_lookup_r4l4_half_kernel<0><<<grid, kLookupThreads, smem, stream>>>(pyr, coords, out, N, qt);
}
static int r4l4_opt_in(const Pyramid &) {
    CF_CUDA(cudaFuncSetAttribute(corr_lookup_r4l4_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * 401 * (int)sizeof(float)));
    CF_CUDA(cudaFuncSetAttribute(corr_lookup_r4l4_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * 401 * (int)sizeof(float)));
    return CF_OK;
}
static int r4l4_opt_in(const PyramidHalf &) {
    CF_CUDA(cudaFuncSetAttribute(corr_lookup_r4l4_half_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * 401 * (int)sizeof(float)));
    CF_CUDA(cudaFuncSetAttribute(corr_lookup_r4l4_half_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * 401 * (int)sizeof(float)));
    return CF_OK;
}
static const char *kernel_name(const Pyramid &, bool r4l4) { return r4l4 ? "corr_lookup_r4l4_kernel" : "corr_lookup_kernel"; }
static const char *kernel_name(const PyramidHalf &, bool r4l4) { return r4l4 ? "corr_lookup_r4l4_half_kernel" : "corr_lookup_half_kernel"; }

template <typename PYR>
static int launch_lookup_r4l4(const PYR &pyr, const float *coords, float *out, int B, int N, cudaStream_t stream) {
    // queries per CTA.  Up to about one wave of 16-query CTAs the launch is latency bound and 16 is the measured
    // optimum (14 balances 6 144 queries better -- 3 CTAs on every SM -- but idles a gather warp and four lanes:
    // 5.4 against 5.2 us).  Beyond that: the even value in [16, 32] with the smallest per-SM maximum
    // ceil(CTAs / SMs) * QT (ties: larger).  Measured against fixed 32: 64x24x32 34.3 -> 31.9 us,
    // 64x36x44 83.4 -> 62.7 us, 8x60x80 42.9 -> 36.3 us.
    const int sms = sm_count();
    int qt = 16;
    if (ceil_div(N, 16) * B > 4 * (int64_t)sms) {
        int64_t best = -1;
        for (int cand = 32; cand >= 16; cand -= 2) {
            const int64_t ctas = ceil_div(N, cand) * B;
            const int64_t cost = ceil_div(ctas, sms) * cand;
            if (best < 0 || cost < best) { best = cost; qt = cand; }
        }
    }
    static const int forced_qt = [] { const char *e = getenv("CF_LOOKUP_QT"); return e ? atoi(e) : 0; }();  // experiments
    if (forced_qt >= 2 && forced_qt <= 32 && (forced_qt & 1) == 0) qt = forced_qt;
    const size_t smem = (size_t)qt * 401 * sizeof(float);
    int dev = 0;
    CF_CUDA(cudaGetDevice(&dev));
    static bool opt_in[64] = {};   // (one per instantiation: fp32 and fp16 pyramids)
    if (!opt_in[dev & 63]) {
        if (int rc = r4l4_opt_in(pyr)) return rc;
        opt_in[dev & 63] = true;
    }
    dim3 grid((unsigned)ceil_div(N, qt), B);
    // (programmatic dependent launch was tried here: with 12 lookups back to back in a graph it made
    //  each launch 1.4 us SLOWER on the B200 -- 8.8 vs 7.4 us -- so plain stream order is kept)
    r4l4_launch(pyr, grid, smem, coords, out, N, qt, stream);
    CF_LAUNCH_CHECK(kernel_name(pyr, true));
    return CF_OK;
}

// dynamic shared memory of corr_lookup_kernel<qt>: the patches plus the clamped coordinates
static size_t lookup_smem_bytes(int qt, int levels, int radius) {
    const int P = 2 * radius + 2;
    return ((size_t)qt * ((levels * P * P) | 1) + 2 * qt) * sizeof(float);
}
constexpr size_t kLookupSmemCap = 200 * 1024;

template <int QT>
static void* lookup_kernel_fn(const Pyramid &) { return reinterpret_cast<void *>(corr_lookup_kernel<QT>); }
template <int QT>
static void* lookup_kernel_fn(const PyramidHalf &) { return reinterpret_cast<void *>(corr_lookup_half_kernel<QT>); }

template <int QT, typename PYR>
static int launch_lookup(const PYR &pyr, const float *coords, float *out, int B, int N, int levels, int radius,
                         cudaStream_t stream) {
    const size_t smem = lookup_smem_bytes(QT, levels, radius);
    CF_REQUIRE(smem <= kLookupSmemCap, CF_ERR_INVALID_ARG, "cf_corr_lookup: levels*radius too large for shared memory");
    int dev = 0;
    CF_CUDA(cudaGetDevice(&dev));
    static bool opt_in[64] = {};
    if (!opt_in[dev & 63]) {
        CF_CUDA(cudaFuncSetAttribute(lookup_kernel_fn<QT>(pyr), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLookupSmemCap));
        opt_in[dev & 63] = true;
    }
    dim3 grid((unsigned)ceil_div(N, QT), B);
    void *args[] = {const_cast<PYR *>(&pyr), &coords, &out, &N, &levels, &radius};
    CF_CUDA(cudaLaunchKernel(lookup_kernel_fn<QT>(pyr), grid, dim3(kLookupThreads), args, smem, stream));
    CF_LAUNCH_CHECK(kernel_name(pyr, false));
    return CF_OK;
}

}  // namespace cf

namespace cf {
// argument checks and dispatch of cf_corr_lookup / cf_corr_lookup_half (PYR: Pyramid or PyramidHalf)
template <typename PYR, typename T>
static int corr_lookup_entry(const char *what, const T *const *pyramid, const float *coords, int B, int h, int w, int levels,
                             int radius, float *out, cudaStream_t stream) {
    if (int rc = check_device()) return rc;
    CF_REQUIRE(pyramid && coords && out, CF_ERR_NULL, "%s: null pointer", what);
    CF_REQUIRE(levels >= 1 && levels <= CF_CORR_MAX_LEVELS, CF_ERR_INVALID_ARG,
               "%s: levels=%d not in [1,%d]", what, levels, CF_CORR_MAX_LEVELS);
    CF_REQUIRE(radius >= 0 && radius <= 8, CF_ERR_INVALID_ARG, "%s: radius=%d not in [0,8]", what, radius);
    CF_REQUIRE(B >= 0 && B <= 65535 && h > 0 && w > 0, CF_ERR_INVALID_ARG, "%s: bad shape B=%d h=%d w=%d", what, B, h, w);
    CF_REQUIRE((h >> (levels - 1)) >= 1 && (w >> (levels - 1)) >= 1, CF_ERR_INVALID_ARG,
               "%s: %dx%d feature map has no level %d", what, h, w, levels - 1);
    if (B == 0) return CF_OK;
    PYR pyr{};
    for (int l = 0; l < levels; ++l) {
        CF_REQUIRE(pyramid[l], CF_ERR_NULL, "%s: pyramid[%d] is null", what, l);
        pyr.ptr[l] = reinterpret_cast<typename std::remove_reference<decltype(pyr.ptr[0])>::type>(pyramid[l]);
        pyr.H[l] = h >> l;
        pyr.W[l] = w >> l;
    }
    const int N = h * w;
    if (radius == 4 && levels == 4) {
        return launch_lookup_r4l4(pyr, coords, out, B, N, stream);
    }
    // 16 queries per CTA when the problem is small (more CTAs than SMs), else 32 (128-byte stores) -- unless 32 queries'
    // patches do not fit the shared memory (5 or 6 levels at radius 8).  Both do the same arithmetic per element, so the
    // result does not depend on which one runs.
    const bool small = (int64_t)B * ceil_div(N, 32) < 4 * (int64_t)sm_count();
    return (small || lookup_smem_bytes(32, levels, radius) > kLookupSmemCap)
               ? launch_lookup<16>(pyr, coords, out, B, N, levels, radius, stream)
               : launch_lookup<32>(pyr, coords, out, B, N, levels, radius, stream);
}
}  // namespace cf

extern "C" int cf_corr_lookup(const float *const *pyramid, const float *coords, int B, int h, int w,
                              int levels, int radius, float *out, cf_stream_t stream_) {
    return cf::corr_lookup_entry<cf::Pyramid>("cf_corr_lookup", pyramid, coords, B, h, w, levels, radius, out,
                                              (cudaStream_t)stream_);
}

extern "C" int cf_corr_lookup_half(const uint16_t *const *pyramid, const float *coords, int B, int h, int w, int levels,
                                   int radius, float *out, cf_stream_t stream_) {
    return cf::corr_lookup_entry<cf::PyramidHalf>("cf_corr_lookup_half", pyramid, coords, B, h, w, levels, radius, out,
                                                  (cudaStream_t)stream_);
}
