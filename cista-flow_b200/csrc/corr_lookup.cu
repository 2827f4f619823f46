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
#include <stdlib.h>

#include "common.cuh"

namespace cf {

struct Pyramid {
    const float *ptr[CF_CORR_MAX_LEVELS];
    int H[CF_CORR_MAX_LEVELS];
    int W[CF_CORR_MAX_LEVELS];
};

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
template <int QT_CT>
__global__ void __launch_bounds__(kLookupThreads)
corr_lookup_r4l4_kernel(const __grid_constant__ Pyramid pyr, const float *__restrict__ coords, float *__restrict__ out, int N,
                        int qt_rt) {
    const int QT = QT_CT > 0 ? QT_CT : qt_rt;
    extern __shared__ float smem[];
    constexpr int PS = 401;                    // 4 levels x 10 x 10, odd stride between queries
    constexpr int NW = kLookupThreads / 32;
    constexpr int U = 2;                       // queries in flight per pass (QT is even)
    float *patch = smem;                       // [QT][PS]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b = blockIdx.y;
    const int q0 = blockIdx.x * QT;
    const float *cb = coords + (size_t)b * 2 * N;
    if (tid == 0) CF_TRACE_AT(0);

    // phase-B coordinates of this lane's query: requested now, first used after the barrier
    const int TPW = 32 / QT;                   // tasks per warp pass in phase B
    const int qiB = lane % QT, tslot = lane / QT;
    const int qB = (tslot < TPW) ? q0 + qiB : N;   // lanes beyond TPW * QT idle in phase B
    float cxB = 0.f, cyB = 0.f;
    if (qB < N) {
        cxB = __ldg(cb + qB);
        cyB = __ldg(cb + N + qB);
    }

    // ---- phase A ---------------------------------------------------------------------------
    {
        // clamp keeps (int) conversions defined for wild coordinates; anything this far out samples
        // only zero padding anyway (NaN clamps to the bound)
        const int rg = lane / 10, col = lane - rg * 10;    // rg == 3: lanes 30, 31 idle
#pragma unroll 1
        for (int qq = U * warp; qq < QT; qq += U * NW) {   // this warp's query pairs
            float cxs[U], cys[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int q = q0 + qq + u;
                cxs[u] = q < N ? fminf(fmaxf(__ldg(cb + q), -1.0e6f), 1.0e6f) : 0.f;
                cys[u] = q < N ? fminf(fmaxf(__ldg(cb + N + q), -1.0e6f), 1.0e6f) : 0.f;
            }
            float *slot = patch + qq * PS + rg * 10 + col;
            float v[U][16];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int q = q0 + qq + u;
                const bool okq = q < N && rg < 3;
#pragma unroll
                for (int l = 0; l < 4; ++l) {
                    const float inv = 1.f / (float)(1 << l);  // exact: coords / 2**l
                    const int X = (int)floorf(cxs[u] * inv) - 4 + col;
                    const int Y = (int)floorf(cys[u] * inv) - 4 + rg;
                    const int Hl = pyr.H[l], Wl = pyr.W[l];
                    const bool okx = okq && (unsigned)X < (unsigned)Wl;
                    const float *p = pyr.ptr[l] + ((size_t)b * N + q) * (Hl * Wl) + (Y * Wl + X);
                    asm volatile("" : "+l"(p));  // one 64-bit column address per (query, level); rows are p + 3k*Wl
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const bool ok = okx && (unsigned)(Y + 3 * k) < (unsigned)Hl && (k < 3 || rg == 0);
                        v[u][l * 4 + k] = ok ? __ldg(p + 3 * k * Wl) : 0.f;
                    }
                }
            }
            if (rg < 3) {
#pragma unroll
                for (int u = 0; u < U; ++u)
#pragma unroll
                    for (int l = 0; l < 4; ++l)
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            if (k < 3 || rg == 0) slot[u * PS + l * 100 + 30 * k] = v[u][l * 4 + k];
            }
        }
    }
    if (tid == 0) CF_TRACE_AT(1);
    __syncthreads();
    if (tid == 0) CF_TRACE_AT(2);

    // ---- phase B ---------------------------------------------------------------------------
    if (qB < N) {
        // the NW * TPW (8 or 16) thread slots of a query split into 4 levels x G window-column groups: a thread's
        // level -- hence its fractions, patch and output base -- is fixed, its columns are ig, ig + G, ...
        // (the TPW lane groups of a warp take neighbouring column groups of the SAME level: their patch addresses then
        //  differ by one float, and with the odd query stride the 32 lanes hit 31-32 distinct banks; with different
        //  levels per lane group -- 100 floats = 4 banks apart -- nearly every LDS was a 2-way conflict)
        const int slot = warp * TPW + tslot, G = (NW * TPW) >> 2;
        const int l = slot / G, ig = slot - l * G;
        const float inv = __int_as_float(0x3f800000 - (l << 23));   // 2**-l, exact: coords / 2**l
        const float sx = fminf(fmaxf(cxB, -1.0e6f), 1.0e6f) * inv, sy = fminf(fmaxf(cyB, -1.0e6f), 1.0e6f) * inv;
        const float fx = sx - floorf(sx), fy = sy - floorf(sy);
        const float gx = 1.f - fx, gy = 1.f - fy;
        const float *pp = patch + qiB * PS + l * 100 + ig;
        float *o = out + (size_t)b * 324 * N + qB + (size_t)(l * 81 + ig * 9) * N;
        const size_t o_step = (size_t)(9 * G) * N;
#pragma unroll 1
        for (int i = ig; i < 9; i += G, pp += G, o += o_step) {   // i -> x offset (transposed window, SURVEY F7)
            float top = pp[0] * gx + pp[1] * fx;
#pragma unroll
            for (int j = 0; j < 9; ++j) {                       // j -> y offset
                const float bot = pp[(j + 1) * 10] * gx + pp[(j + 1) * 10 + 1] * fx;
                o[(size_t)j * N] = top * gy + bot * fy;
                top = bot;
            }
        }
    }
    if (tid == 0) CF_TRACE_AT(3);
#ifdef CF_TRACE
    if (tid == 0 && g_trace) {  // which SM ran this CTA (slot 4)
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        g_trace[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * kTraceSlots + 4] = smid + 1;
    }
#endif
}

// Generic radius / level count (runtime arguments): one element per thread and step.
template <int QT>
__global__ void __launch_bounds__(kLookupThreads)
corr_lookup_kernel(const __grid_constant__ Pyramid pyr, const float *__restrict__ coords, float *__restrict__ out,
                   int N, int levels, int r) {
    extern __shared__ float smem[];
    const int K = 2 * r + 1, P = K + 1, KK = K * K, PP = P * P;
    const int LPP = levels * PP;
    const int PS = LPP | 1;              // odd stride between queries
    float *patch = smem;                 // [QT][PS]
    float *cxy = smem + (size_t)QT * PS; // [QT][2]
    const int tid = threadIdx.x;
    const int b = blockIdx.y;
    const int q0 = blockIdx.x * QT;
    const float *cb = coords + (size_t)b * 2 * N;
    if (tid < QT) {
        const int q = q0 + tid;
        cxy[2 * tid] = q < N ? fminf(fmaxf(__ldg(cb + q), -1.0e6f), 1.0e6f) : 0.f;
        cxy[2 * tid + 1] = q < N ? fminf(fmaxf(__ldg(cb + N + q), -1.0e6f), 1.0e6f) : 0.f;
    }
    __syncthreads();

    // ---- phase A: gather the patches (zero outside the map) ----------------------
    const int total = QT * LPP;
#pragma unroll 5
    for (int idx = tid; idx < total; idx += kLookupThreads) {
        const int qi = idx / LPP, e = idx - qi * LPP;
        const int l = e / PP, rem = e - l * PP;
        const int py = rem / P, px = rem - py * P;
        const float inv = 1.f / (float)(1 << l);  // exact: coords / 2**l
        const int X = (int)floorf(cxy[2 * qi] * inv) - r + px;
        const int Y = (int)floorf(cxy[2 * qi + 1] * inv) - r + py;
        const int Hl = pyr.H[l], Wl = pyr.W[l];
        const int q = q0 + qi;
        float v = 0.f;
        if (q < N && X >= 0 && X < Wl && Y >= 0 && Y < Hl)
            v = __ldg(pyr.ptr[l] + (((size_t)b * N + q) * Hl + Y) * Wl + X);
        patch[qi * PS + e] = v;
    }
    __syncthreads();

    // ---- phase B: bilinear samples, coalesced channel-major stores ---------------
    constexpr int CPW = 32 / QT;                      // channels per warp-iteration
    const int warp = tid >> 5, lane = tid & 31;
    const int qi = lane % QT;
    const int q = q0 + qi;
    const int c_first = warp * CPW + lane / QT;
    constexpr int c_step = (kLookupThreads / 32) * CPW;
    const float cx = cxy[2 * qi], cy = cxy[2 * qi + 1];
    const float *pq = patch + qi * PS;
    float *ob = out + (size_t)b * levels * KK * N + q;
    if (q < N) {
        for (int l = 0; l < levels; ++l) {
            const float inv = 1.f / (float)(1 << l);
            const float sx = cx * inv, sy = cy * inv;
            const float fx = sx - floorf(sx), fy = sy - floorf(sy);
            const float w00 = (1.f - fx) * (1.f - fy), w01 = fx * (1.f - fy), w10 = (1.f - fx) * fy, w11 = fx * fy;
            const float *pl = pq + l * PP;
            float *ol = ob + (size_t)l * KK * N;
#pragma unroll 4
            for (int c = c_first; c < KK; c += c_step) {
                const int i = c / K, j = c - i * K;   // i -> x offset, j -> y offset (transposed window)
                const float *pp = pl + j * P + i;
                float acc = pp[0] * w00;
                acc += pp[1] * w01;
                acc += pp[P] * w10;
                acc += pp[P + 1] * w11;
                ol[(size_t)c * N] = acc;
            }
        }
    }
}

CF_DEFINE_TRACE_SETTER(cf_trace_buffer_lookup)

static int launch_lookup_r4l4(const Pyramid &pyr, const float *coords, float *out, int B, int N, cudaStream_t stream) {
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
    static bool opt_in[64] = {};
    if (!opt_in[dev & 63]) {
        CF_CUDA(cudaFuncSetAttribute(corr_lookup_r4l4_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * 401 * (int)sizeof(float)));
        CF_CUDA(cudaFuncSetAttribute(corr_lookup_r4l4_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * 401 * (int)sizeof(float)));
        opt_in[dev & 63] = true;
    }
    dim3 grid((unsigned)ceil_div(N, qt), B);
    // (programmatic dependent launch was tried here: with 12 lookups back to back in a graph it made
    //  each launch 1.4 us SLOWER on the B200 -- 8.8 vs 7.4 us -- so plain stream order is kept)
    if (qt == 16) corr_lookup_r4l4_kernel<16><<<grid, kLookupThreads, smem, stream>>>(pyr, coords, out, N, qt);
    else corr_lookup_r4l4_kernel<0><<<grid, kLookupThreads, smem, stream>>>(pyr, coords, out, N, qt);
    CF_LAUNCH_CHECK("corr_lookup_r4l4_kernel");
    return CF_OK;
}

// dynamic shared memory of corr_lookup_kernel<qt>: the patches plus the clamped coordinates
static size_t lookup_smem_bytes(int qt, int levels, int radius) {
    const int P = 2 * radius + 2;
    return ((size_t)qt * ((levels * P * P) | 1) + 2 * qt) * sizeof(float);
}
constexpr size_t kLookupSmemCap = 200 * 1024;

template <int QT>
static int launch_lookup(const Pyramid &pyr, const float *coords, float *out, int B, int N, int levels, int radius,
                         cudaStream_t stream) {
    const size_t smem = lookup_smem_bytes(QT, levels, radius);
    CF_REQUIRE(smem <= kLookupSmemCap, CF_ERR_INVALID_ARG, "cf_corr_lookup: levels*radius too large for shared memory");
    int dev = 0;
    CF_CUDA(cudaGetDevice(&dev));
    static bool opt_in[64] = {};
    if (!opt_in[dev & 63]) {
        CF_CUDA(cudaFuncSetAttribute(corr_lookup_kernel<QT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLookupSmemCap));
        opt_in[dev & 63] = true;
    }
    dim3 grid((unsigned)ceil_div(N, QT), B);
    corr_lookup_kernel<QT><<<grid, kLookupThreads, smem, stream>>>(pyr, coords, out, N, levels, radius);
    CF_LAUNCH_CHECK("corr_lookup_kernel");
    return CF_OK;
}

}  // namespace cf

extern "C" int cf_corr_lookup(const float *const *pyramid, const float *coords, int B, int h, int w,
                              int levels, int radius, float *out, cf_stream_t stream_) {
    using namespace cf;
    if (int rc = check_device()) return rc;
    CF_REQUIRE(pyramid && coords && out, CF_ERR_NULL, "cf_corr_lookup: null pointer");
    CF_REQUIRE(levels >= 1 && levels <= CF_CORR_MAX_LEVELS, CF_ERR_INVALID_ARG,
               "cf_corr_lookup: levels=%d not in [1,%d]", levels, CF_CORR_MAX_LEVELS);
    CF_REQUIRE(radius >= 0 && radius <= 8, CF_ERR_INVALID_ARG, "cf_corr_lookup: radius=%d not in [0,8]", radius);
    CF_REQUIRE(B >= 0 && B <= 65535 && h > 0 && w > 0, CF_ERR_INVALID_ARG, "cf_corr_lookup: bad shape B=%d h=%d w=%d", B, h, w);
    CF_REQUIRE((h >> (levels - 1)) >= 1 && (w >> (levels - 1)) >= 1, CF_ERR_INVALID_ARG,
               "cf_corr_lookup: %dx%d feature map has no level %d", h, w, levels - 1);
    if (B == 0) return CF_OK;
    Pyramid pyr{};
    for (int l = 0; l < levels; ++l) {
        CF_REQUIRE(pyramid[l], CF_ERR_NULL, "cf_corr_lookup: pyramid[%d] is null", l);
        pyr.ptr[l] = pyramid[l];
        pyr.H[l] = h >> l;
        pyr.W[l] = w >> l;
    }
    const int N = h * w;
    cudaStream_t stream = (cudaStream_t)stream_;
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
