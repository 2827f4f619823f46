// Packed event ingest (SURVEY.md section 8f rank 3): 8 bytes per event instead of the reference's
// 32-byte fp64 row (data_readers/event_readers.py:6-47 delivers [N,4] float64 (t, x, y, p)).
//
//   word 0  float32  t_rel = (float)(t - t_first_of_window): the fp64 subtraction happens BEFORE the
//                    rounding, so absolute stamps (~1e9 us, SURVEY F10) cost no precision
//   word 1  uint32   x | y << 16 | p << 31          (x < 65536, y < 32768, p = 1 for positive polarity)
//
// A row outside [offsets[0], offsets[B]) belongs to no window: both packers write the invalid record for it
// (x = 0xffff, t_rel = 0), and the voxel kernel does not visit it.
//
// cf_events_pack       device-side packer: fp64 rows -> packed (one pass, 32 B read + 8 B written per event)
// cf_voxel_bin_packed  ATOMIC-mode voxel grid (+ fused event_preprocess) from packed events: the kernel
//                      reads 8 B per event (4x fewer event bytes than cf_voxel_bin) and does the time
//                      normalisation t* = (nb-1) * t_rel / dT in fp32 (mul, then div, like
//                      utils/event_process.py:46-49).  Against the fp64 reference the bin position moves
//                      by <= ~4e-7 and, the temporal bilinear weights being continuous across bin
//                      boundaries, every cell stays within the atomic-mode tolerance 1e-5 * (sum|w| + 1).
//                      There is no deterministic (bit-exact) mode for packed input: the fp64 stamps
//                      that define the reference's bins are gone.
#include "voxel_common.cuh"

namespace cf {

// from voxel.cu: statistics -> normalise, shared with the fp64 path
int run_preprocess(const float *in, float *out, int B, int64_t cells, int preprocess, float hot_thr, void *ws,
                   size_t ws_bytes, cudaStream_t stream);

namespace vp {
constexpr int THREADS = 256;
constexpr int UNROLL = 4;

__device__ __forceinline__ int find_window(int64_t i, const int64_t *__restrict__ off, int B) {
    int lo = 0, hi = B - 1;  // last b with off[b] <= i
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(off + mid) <= i) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__global__ void __launch_bounds__(THREADS)
events_pack_kernel(const double *__restrict__ ev, const int64_t *__restrict__ off, int64_t total, int B,
                   uint2 *__restrict__ packed) {
    const int64_t ev_first = __ldg(off), ev_end = __ldg(off + B);
    int b = -1;
    int64_t begin = 0, end = 0;
    double t0 = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * THREADS + threadIdx.x; i < total; i += (int64_t)gridDim.x * THREADS) {
        if (i < ev_first || i >= ev_end) {   // a row of no window: the invalid record (x = 0xffff, t_rel = 0)
            packed[i] = make_uint2(0u, 0xffffu);
            continue;
        }
        const Event e = load_event(ev, i);
        if (b < 0 || i < begin || i >= end) {
            b = find_window(i, off, B);
            begin = __ldg(off + b);
            end = __ldg(off + b + 1);
            t0 = __ldg(ev + 4 * begin);
        }
        // out-of-range coordinates are kept representable and marked invalid (x = 0xffff): the voxel kernel
        // drops them like cf_voxel_bin drops out-of-grid events
        const bool ok = e.x >= 0.0 && e.x < 65535.0 && e.y >= 0.0 && e.y < 32768.0;
        const uint32_t x = ok ? (uint32_t)e.x : 0xffffu, y = ok ? (uint32_t)e.y : 0u;
        const uint32_t p = e.p > 0.0 ? 1u : 0u;
        packed[i] = make_uint2(__float_as_uint((float)__dsub_rn(e.t, t0)), x | (y << 16) | (p << 31));
    }
}

__global__ void __launch_bounds__(THREADS)
voxel_scatter_packed_kernel(const uint2 *__restrict__ packed, const int64_t *__restrict__ off, int B, int nb, int H, int W,
                            float *__restrict__ out) {
    const int64_t ev_first = __ldg(off), ev_end = __ldg(off + B);   // rows outside the windows are not visited
    const int64_t plane = (int64_t)H * W;
    constexpr int64_t kTile = THREADS * UNROLL;
    int b = -1;
    int64_t begin = 0, end = 0;
    float span = 1.f;
    for (int64_t tile = ev_first + (int64_t)blockIdx.x * kTile; tile < ev_end; tile += (int64_t)gridDim.x * kTile) {
        uint2 e[UNROLL];
#pragma unroll
        for (int k = 0; k < UNROLL; ++k) {  // all loads in flight first
            const int64_t i = tile + k * THREADS + threadIdx.x;
            if (i < ev_end) e[k] = __ldg(packed + i);
        }
#pragma unroll
        for (int k = 0; k < UNROLL; ++k) {
            const int64_t i = tile + k * THREADS + threadIdx.x;
            if (i >= ev_end) break;
            if (b < 0 || i < begin || i >= end) {
                b = find_window(i, off, B);
                begin = __ldg(off + b);
                end = __ldg(off + b + 1);
                span = __uint_as_float(__ldg(packed + end - 1).x);   // t_rel of the window's last event
                if (span == 0.f) span = 1.f;                          // event_process.py:43-44
            }
            const float tn = __fdiv_rn(__fmul_rn((float)(nb - 1), __uint_as_float(e[k].x)), span);
            const float lo = floorf(tn);
            const int x = (int)(e[k].y & 0xffffu), y = (int)((e[k].y >> 16) & 0x7fffu);
            if (!(lo >= 0.f && lo < (float)nb) || x >= W || y >= H) continue;
            const int bin = (int)lo;
            const float f = __fsub_rn(tn, lo);
            const float s = (e[k].y >> 31) ? 1.f : -1.f;             // event_process.py:51 (p == 0 -> -1)
            float *cell = out + ((int64_t)b * nb + bin) * plane + (int64_t)y * W + x;
            atomicAdd(cell, __fmul_rn(s, __fsub_rn(1.f, f)));
            if (bin + 1 < nb) atomicAdd(cell + plane, __fmul_rn(s, f));
        }
    }
}
}  // namespace vp
}  // namespace cf

extern "C" int cf_events_pack(const double *events, const int64_t *offsets, int64_t total, int B, void *packed,
                              cf_stream_t stream_) {
    using namespace cf;
    if (int rc = check_device()) return rc;
    CF_REQUIRE(offsets && packed, CF_ERR_NULL, "cf_events_pack: null pointer");
    CF_REQUIRE(total == 0 || events, CF_ERR_NULL, "cf_events_pack: events is null");
    CF_REQUIRE(B >= 1 && total >= 0, CF_ERR_INVALID_ARG, "cf_events_pack: bad sizes B=%d total=%lld", B, (long long)total);
    CF_REQUIRE(total == 0 || aligned16(events), CF_ERR_ALIGN, "cf_events_pack: events not 16-byte aligned");
    CF_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 7u) == 0, CF_ERR_ALIGN, "cf_events_pack: packed not 8-byte aligned");
    if (total == 0) return CF_OK;
    int64_t blocks = ceil_div(total, vp::THREADS);
    const int64_t cap = (int64_t)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    vp::events_pack_kernel<<<(unsigned)blocks, vp::THREADS, 0, (cudaStream_t)stream_>>>(events, offsets, total, B,
                                                                                        reinterpret_cast<uint2 *>(packed));
    CF_LAUNCH_CHECK("events_pack_kernel");
    return CF_OK;
}

extern "C" int cf_voxel_bin_packed(const void *packed, const int64_t *offsets, int64_t total, int B, int nb, int H, int W,
                                   int preprocess, float hot_thr, float *out, void *ws, size_t ws_bytes,
                                   cf_stream_t stream_) {
    using namespace cf;
    if (int rc = check_device()) return rc;
    CF_REQUIRE(out && offsets, CF_ERR_NULL, "cf_voxel_bin_packed: null pointer");
    CF_REQUIRE(total == 0 || packed, CF_ERR_NULL, "cf_voxel_bin_packed: packed is null");
    CF_REQUIRE(nb > 0 && H > 0 && W > 0 && H <= 32768 && W <= 65535, CF_ERR_INVALID_ARG,
               "cf_voxel_bin_packed: num_bins > 0, 0 < width <= 65535, 0 < height <= 32768 required");
    CF_REQUIRE(B >= 0 && total >= 0, CF_ERR_INVALID_ARG, "cf_voxel_bin_packed: negative size");
    CF_REQUIRE(preprocess >= CF_PRE_NONE && preprocess <= CF_PRE_MAXMIN, CF_ERR_INVALID_ARG, "cf_voxel_bin_packed: bad preprocess %d", preprocess);
    CF_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 7u) == 0, CF_ERR_ALIGN, "cf_voxel_bin_packed: packed not 8-byte aligned");
    if (B == 0) return CF_OK;
    cudaStream_t stream = (cudaStream_t)stream_;
    const int64_t cells = (int64_t)nb * H * W;
    CF_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)B * cells, stream));
    if (total > 0) {
        int64_t blocks = ceil_div(total, vp::THREADS * vp::UNROLL);
        const int64_t cap = (int64_t)sm_count() * 8;
        if (blocks > cap) blocks = cap;
        vp::voxel_scatter_packed_kernel<<<(unsigned)blocks, vp::THREADS, 0, stream>>>(
            reinterpret_cast<const uint2 *>(packed), offsets, B, nb, H, W, out);
        CF_LAUNCH_CHECK("voxel_scatter_packed_kernel");
    }
    if (preprocess != CF_PRE_NONE) return run_preprocess(out, out, B, cells, preprocess, hot_thr, ws, ws_bytes, stream);
    return CF_OK;
}

namespace cf {

// ---------------------------------------------------------------- device-side windowing ---
// What the reference's readers do on the host with pandas / NumPy before every frame
// (data_readers/video_readers.py:208-232, data_readers/event_readers.py:6-47), on the device:
//   cf_events_filter      keeps the rows with x < width and y < height (video_readers.py:208-209, in this order, no lower
//                         bound -- like the reference), STABLE, compacted into `out`; the kept count goes to a device
//                         int64 so that nothing is read back;
//   cf_event_window_offsets   offsets[0..n] of the frame's windows from a DEVICE-resident event count:
//                         CF_WINDOWS_FIXED  non-overlapping windows of `param` events, the last one keeps the remainder
//                                           (FixedSizeEventReader with k_shift <= 0: pandas get_chunk)
//                         CF_WINDOWS_SPLIT  np.array_split(events, max(1, round(n / param))): n // k + 1 events in the first
//                                           n % k windows, n // k in the others (limit_num_events > 0, video_readers.py:219-224)
//                         offsets beyond the last window are filled with n, so a fixed-size offsets array (max_windows + 1)
//                         feeds cf_voxel_bin with B = max_windows and empty trailing windows -- graph-capturable.
namespace vw {
constexpr int THREADS = 256;
constexpr int ITEMS = 8;                      // rows per thread
constexpr int TILE = THREADS * ITEMS;         // 2048 rows per CTA

__device__ __forceinline__ bool keep_row(const double *__restrict__ ev, int64_t i, double W, double H) {
    const double x = __ldg(ev + 4 * i + 1), y = __ldg(ev + 4 * i + 2);
    return x < W && y < H;
}

// kept rows per CTA tile -> counts[blockIdx.x]
__global__ void __launch_bounds__(THREADS) filter_count_kernel(const double *__restrict__ ev, int64_t total, double W, double H,
                                                               uint32_t *__restrict__ counts) {
    const int64_t base = (int64_t)blockIdx.x * TILE + (int64_t)threadIdx.x * ITEMS;
    int n = 0;
#pragma unroll
    for (int k = 0; k < ITEMS; ++k)
        if (base + k < total && keep_row(ev, base + k, W, H)) ++n;
    n = warp_sum(n);
    __shared__ int sh[THREADS / 32];
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = n;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int k = 0; k < THREADS / 32; ++k) t += sh[k];
        counts[blockIdx.x] = (uint32_t)t;
    }
}

// exclusive scan of `n` CTA counts in place (single CTA of 1024 threads); total -> *kept
__global__ void __launch_bounds__(1024) filter_scan_kernel(uint32_t *__restrict__ data, int64_t n, int64_t *__restrict__ kept) {
    __shared__ uint32_t warp_tot[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t per = (n + 1023) / 1024;
    const int64_t s = (int64_t)tid * per, e = min(n, s + per);
    uint32_t sum = 0;
    for (int64_t i = s; i < e; ++i) sum += data[i];
    uint32_t inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += v;
    }
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint32_t t = warp_tot[lane], ti = t;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, ti, o);
            if (lane >= o) ti += v;
        }
        warp_tot[lane] = ti - t;
        if (lane == 31) *kept = (int64_t)ti;
    }
    __syncthreads();
    uint32_t run = warp_tot[warp] + inc - sum;
    for (int64_t i = s; i < e; ++i) {
        const uint32_t v = data[i];
        data[i] = run;
        run += v;
    }
}

// stable scatter: thread-local ranks + warp scan + warp totals, on top of the scanned CTA base
__global__ void __launch_bounds__(THREADS) filter_scatter_kernel(const double *__restrict__ ev, int64_t total, double W, double H,
                                                                 const uint32_t *__restrict__ bases, double *__restrict__ out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t base = (int64_t)blockIdx.x * TILE + (int64_t)threadIdx.x * ITEMS;
    bool keep[ITEMS];
    int n = 0;
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        keep[k] = base + k < total && keep_row(ev, base + k, W, H);
        n += keep[k];
    }
    int inc = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += v;
    }
    __shared__ int sh[THREADS / 32];
    if (lane == 31) sh[warp] = inc;
    __syncthreads();
    int before = inc - n;
    for (int k = 0; k < warp; ++k) before += sh[k];
    int64_t dst = (int64_t)bases[blockIdx.x] + before;
    const double2 *src2 = reinterpret_cast<const double2 *>(ev);
    double2 *out2 = reinterpret_cast<double2 *>(out);
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        if (keep[k]) {
            out2[2 * dst] = __ldg(src2 + 2 * (base + k));
            out2[2 * dst + 1] = __ldg(src2 + 2 * (base + k) + 1);
            ++dst;
        }
    }
}

__global__ void __launch_bounds__(256) window_offsets_kernel(const int64_t *__restrict__ count, int policy, int64_t param,
                                                             int64_t *__restrict__ offsets, int max_windows, int *__restrict__ n_windows) {
    const int64_t n = *count;
    int64_t k;      // number of windows
    if (policy == CF_WINDOWS_FIXED) {
        k = (n + param - 1) / param;
    } else {
        // Python round(): half to even, on the fp64 quotient (video_readers.py:220)
        k = (int64_t)rint((double)n / (double)param);
        if (k == 0) k = 1;
    }
    // the caller sized the array: FIXED keeps windows of `param` events and the last one keeps the rest; SPLIT splits
    // the n events evenly over max_windows windows (np.array_split with k = max_windows)
    if (k > max_windows) k = max_windows;
    const int64_t q = k > 0 ? n / k : 0, r = k > 0 ? n % k : 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i <= max_windows; i += gridDim.x * blockDim.x) {
        int64_t o;
        if (i >= k) o = n;
        else if (policy == CF_WINDOWS_FIXED) o = (int64_t)i * param < n ? (int64_t)i * param : n;
        else o = (int64_t)i * q + (i < r ? i : r);          // np.array_split: the first n % k sections get one more
        offsets[i] = o;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0 && n_windows) *n_windows = (int)k;
}
}  // namespace vw
}  // namespace cf

extern "C" size_t cf_events_filter_workspace_bytes(int64_t total_events) {
    const int64_t tiles = ((total_events > 0 ? total_events : 1) + cf::vw::TILE - 1) / cf::vw::TILE;
    return cf::align_up((size_t)tiles * sizeof(uint32_t), 256);
}

extern "C" int cf_events_filter(const double *events, int64_t total, int W, int H, double *out, int64_t *kept,
                                void *ws, size_t ws_bytes, cf_stream_t stream_) {
    using namespace cf;
    if (int rc = check_device()) return rc;
    CF_REQUIRE(kept && (total == 0 || (events && out)), CF_ERR_NULL, "cf_events_filter: null pointer");
    CF_REQUIRE(total >= 0 && W > 0 && H > 0, CF_ERR_INVALID_ARG, "cf_events_filter: bad size");
    CF_REQUIRE(total < (1ll << 32), CF_ERR_INVALID_ARG, "cf_events_filter: more than 2^32 events in one call");
    CF_REQUIRE(total == 0 || (aligned16(events) && aligned16(out)), CF_ERR_ALIGN, "cf_events_filter: events not 16-byte aligned");
    cudaStream_t stream = (cudaStream_t)stream_;
    if (total == 0) {
        CF_CUDA(cudaMemsetAsync(kept, 0, sizeof(int64_t), stream));
        return CF_OK;
    }
    const int64_t tiles = ceil_div(total, vw::TILE);
    CF_REQUIRE(ws && ws_bytes >= (size_t)tiles * sizeof(uint32_t), CF_ERR_WORKSPACE, "cf_events_filter: workspace too small");
    uint32_t *counts = reinterpret_cast<uint32_t *>(ws);
    vw::filter_count_kernel<<<(unsigned)tiles, vw::THREADS, 0, stream>>>(events, total, (double)W, (double)H, counts);
    CF_LAUNCH_CHECK("filter_count_kernel");
    vw::filter_scan_kernel<<<1, 1024, 0, stream>>>(counts, tiles, kept);
    CF_LAUNCH_CHECK("filter_scan_kernel");
    vw::filter_scatter_kernel<<<(unsigned)tiles, vw::THREADS, 0, stream>>>(events, total, (double)W, (double)H, counts, out);
    CF_LAUNCH_CHECK("filter_scatter_kernel");
    return CF_OK;
}

extern "C" int cf_event_window_offsets(const int64_t *count, int policy, int64_t param, int64_t *offsets, int max_windows,
                                       int *n_windows, cf_stream_t stream_) {
    using namespace cf;
    if (int rc = check_device()) return rc;
    CF_REQUIRE(count && offsets, CF_ERR_NULL, "cf_event_window_offsets: null pointer");
    CF_REQUIRE(policy == CF_WINDOWS_FIXED || policy == CF_WINDOWS_SPLIT, CF_ERR_INVALID_ARG, "cf_event_window_offsets: bad policy %d", policy);
    CF_REQUIRE(param > 0 && max_windows > 0, CF_ERR_INVALID_ARG, "cf_event_window_offsets: param and max_windows must be > 0");
    vw::window_offsets_kernel<<<(unsigned)ceil_div(max_windows + 1, 256), 256, 0, (cudaStream_t)stream_>>>(count, policy, param, offsets,
                                                                                                    max_windows, n_windows);
    CF_LAUNCH_CHECK("window_offsets_kernel");
    return CF_OK;
}
