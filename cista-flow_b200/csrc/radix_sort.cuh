// Stable LSB radix sort of (uint32 key, uint32 value) pairs, 8 bits per pass:
//   for each pass p: rs_hist_kernel (per-CTA digit counts) -> rs_scan_kernel (exclusive scan, digit-major) ->
//   rs_scatter_kernel (stable scatter), then swap the in/out buffers.
// Stable: equal keys keep their input order whatever the launch configuration, which is what the deterministic
// voxel mode (voxel.cu) and the deterministic warp adjoint (warp_backward_det.cu) build their fixed summation
// orders on.  The kernels are static: each translation unit that includes this header gets its own copy.
#pragma once

#include "common.cuh"

namespace cf {

constexpr int kRsThreads = 256;
constexpr int kRsItems = 16;
constexpr int kRsTile = kRsThreads * kRsItems;  // 4096 keys per CTA
constexpr int kRsWarps = kRsThreads / 32;

static __global__ void __launch_bounds__(kRsThreads)
rs_hist_kernel(const uint32_t *__restrict__ keys, int64_t n, int shift, uint32_t *__restrict__ hist, int nblk) {
    __shared__ uint32_t h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * kRsTile;
#pragma unroll
    for (int k = 0; k < kRsItems; ++k) {
        const int64_t i = base + k * kRsThreads + threadIdx.x;
        if (i < n) atomicAdd(&h[(keys[i] >> shift) & 255u], 1u);  // integer: order-independent
    }
    __syncthreads();
    hist[(size_t)threadIdx.x * nblk + blockIdx.x] = h[threadIdx.x];
}

// exclusive scan of `n` counters in place, single CTA of 1024 threads
static __global__ void __launch_bounds__(1024) rs_scan_kernel(uint32_t *__restrict__ data, int64_t n) {
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
    }
    __syncthreads();
    uint32_t run = warp_tot[warp] + inc - sum;
    for (int64_t i = s; i < e; ++i) {
        const uint32_t v = data[i];
        data[i] = run;
        run += v;
    }
}

// Stable scatter of one 8-bit digit.  Order inside a CTA tile: warp-major,
// round-major, lane-minor == global index order; __match_any_sync ranks the
// lanes of a round, a per-warp running count ranks the rounds, a scan over the
// warps ranks the warps, the scanned histogram ranks the CTAs.
static __global__ void __launch_bounds__(kRsThreads)
rs_scatter_kernel(const uint32_t *__restrict__ keys_in, const uint32_t *__restrict__ vals_in,
                  uint32_t *__restrict__ keys_out, uint32_t *__restrict__ vals_out, int64_t n, int shift,
                  const uint32_t *__restrict__ hist, int nblk) {
    __shared__ uint32_t warp_cnt[kRsWarps][256];
    __shared__ uint32_t gbase[256];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int k = tid; k < kRsWarps * 256; k += kRsThreads) (&warp_cnt[0][0])[k] = 0;
    __syncthreads();
    const int64_t wbase = (int64_t)blockIdx.x * kRsTile + (int64_t)warp * (kRsItems * 32);
    uint32_t key[kRsItems], rnk[kRsItems];
#pragma unroll
    for (int r = 0; r < kRsItems; ++r) {
        const int64_t i = wbase + r * 32 + lane;
        const bool valid = i < n;
        key[r] = valid ? keys_in[i] : 0u;
        const uint32_t d = valid ? ((key[r] >> shift) & 255u) : (256u + lane);  // invalid lanes never match
        const uint32_t peers = __match_any_sync(0xffffffffu, d);
        const uint32_t before = __popc(peers & ((1u << lane) - 1u));
        uint32_t prev = 0;
        if (valid) prev = warp_cnt[warp][d];
        __syncwarp();
        if (valid && before == 0) warp_cnt[warp][d] = prev + __popc(peers);
        __syncwarp();
        rnk[r] = prev + before;
    }
    __syncthreads();
    {
        uint32_t run = 0;
#pragma unroll
        for (int w = 0; w < kRsWarps; ++w) {
            const uint32_t c = warp_cnt[w][tid];
            warp_cnt[w][tid] = run;
            run += c;
        }
        gbase[tid] = hist[(size_t)tid * nblk + blockIdx.x];
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kRsItems; ++r) {
        const int64_t i = wbase + r * 32 + lane;
        if (i < n) {
            const uint32_t d = (key[r] >> shift) & 255u;
            const uint32_t dst = gbase[d] + warp_cnt[warp][d] + rnk[r];
            keys_out[dst] = key[r];
            vals_out[dst] = vals_in[i];
        }
    }
}

// significant bits of max_key (at least 1): the sort takes ceil(bits / 8) passes
static inline int radix_bits(uint64_t max_key) {
    int bits = 1;
    while (bits < 32 && (max_key >> bits) != 0) ++bits;
    return bits;
}

}  // namespace cf
