// Event stream -> voxel grid binning + normalisation (part 1 of the hot path).
//
// Replaces events_to_voxel_grid / _pytorch / _pol and event_preprocess(_pytorch)
// of the reference (utils/event_process.py:15-72, 127-190, 75-123, 193-239).
//
// Data layout in HBM: events float64 [total,4] rows (t,x,y,p), B windows
// concatenated + int64 offsets[B+1]; out float32 [B,nb,H,W] ([B,nb,2,H,W] for
// the polarity flavour).  One event is one 32-byte row = two 128-bit loads.
// Roofline: HBM.  Algorithmic bytes per window = 32*N_events + 4*nb*H*W.
//
// Two accumulation modes:
//   ATOMIC         sum order unspecified -> agrees with the reference to <= 1e-5.
//                  fp32 RED.ADD resolved in L2; the batch is processed in chunks
//                  of windows whose grids + events fit in L2 (kL2ChunkBytes), each
//                  chunk running zero -> scatter -> statistics -> normalise-in-place
//                  back to back, so a grid is read and written in L2 and reaches
//                  HBM exactly once.
//   DETERMINISTIC  bit-exact.  The reference accumulates every cell
//                  sequentially in event order, all bin-ti ("left")
//                  contributions before all bin-ti+1 ("right") ones (two
//                  scatter-adds).  We reproduce exactly that order: a stable
//                  LSB radix sort of (cell-column key, event index) groups the
//                  events of each pixel in event order, then one thread per
//                  pixel walks its run bin by bin with un-contracted IEEE
//                  adds (__fadd_rn / fp64 add + round for the NumPy flavour).
// Measured and dropped (round 1): taking the std statistics out of the scatter itself -- returning atomics
// (ATOMG instead of RED) give each add's previous value o, and sum f(o + w) - f(o) telescopes to the final
// grid's sum / sum of squares / non-zero count, so the separate statistics pass disappears.  Correct (all parity
// tests green) but 1.4-4x SLOWER end to end on the B200 (8x180x240: 24.4 against 16.6 us; 64x260x346: 543 against
// 132 us): returning atomics cost far more than the pass over the L2-resident grid they save.  Rebuilt in round 2
// with per-warp fp64 accumulators and measured again, then removed: 419 against 367 us at 64x480x640, 56 against
// 30 us at 1x624x970 -- every add becomes a round trip its thread waits for.
// Also measured and dropped: statistics + normalisation as ONE pass (a CTA keeps its <= 32 KB slice of a window in
// registers, publishes its partial, waits on a per-window arrival counter -- tickets make the wait deadlock-free --
// and normalises out of registers: one read, one write, one launch).  Parity-green but slower than the two
// kernels at every shape (8x180x240: 18.7 against 16.6 us; 8x480x640: 55.2 against 43.6 us): the ticket atomic
// sits in front of every load address and the waiting CTAs hold their SM slots idle.
// Also measured and removed:
//   - privatising the grid in the distributed shared memory of a thread-block cluster and scattering with
//     red.shared::cluster.add.f32.  DSMEM atomics sustain ~19 G adds/s chip-wide vs ~69 G/s for L2 atomics on a
//     B200, so that path was 2-4x SLOWER than the L2 one (timed with scripts/voxel_microbench.py).
//   - the four L2 stages (zero, scatter, statistics, normalise) of four consecutive chunks fused horizontally into
//     one launch per step: 573 against 365 us at 64x480x640, 78 against 43 us at 8x480x640 -- the stages did not
//     overlap usefully inside one launch.
// Time normalisation is fp64 with the reference's operation order
// (mul, then div) in both modes, so bin assignment is identical.
#include "radix_sort.cuh"
#include "voxel_common.cuh"

namespace cf {

// ------------------------------------------------------------ atomic mode ---
constexpr int kScatterThreads = 256;
constexpr int kScatterUnroll = 4;
constexpr size_t kL2ChunkBytes = (size_t)96 << 20;  // grids + events of one chunk of windows (of the B200's 126 MB L2)

__global__ void __launch_bounds__(kScatterThreads)
voxel_scatter_atomic_kernel(const double *__restrict__ ev, const int64_t *__restrict__ off,
                            int B, int nb, int H, int W, int flavour, float *__restrict__ out, int b_first, int b_end) {
    // the events of windows [b_first, b_end) (one L2-sized chunk of the batch), grid-stride over
    // tiles of 1024 events: the host does not know the chunk's event count (offsets are on the device)
    const int64_t ev_first = __ldg(off + b_first), ev_end = __ldg(off + b_end);
    const int64_t plane = (int64_t)H * W;
    const int planes_per_bin = flavour == CF_FLAVOUR_POL ? 2 : 1;
    constexpr int64_t kTileEvents = kScatterThreads * kScatterUnroll;
    Window w;
    w.b = -1;
    for (int64_t tile = ev_first + (int64_t)blockIdx.x * kTileEvents; tile < ev_end; tile += (int64_t)gridDim.x * kTileEvents) {
        Event e[kScatterUnroll];
#pragma unroll
        for (int k = 0; k < kScatterUnroll; ++k) {  // all loads in flight first
            const int64_t i = tile + k * kScatterThreads + threadIdx.x;
            if (i < ev_end) e[k] = load_event(ev, i);
        }
#pragma unroll
        for (int k = 0; k < kScatterUnroll; ++k) {
            const int64_t i = tile + k * kScatterThreads + threadIdx.x;
            if (i >= ev_end) break;
            locate_window(w, i, off, ev, B);
            const Binned b = bin_event(e[k], w, nb, H, W, flavour);
            if (!b.ok) continue;
            float wl, wr;
            if (flavour == CF_FLAVOUR_TORCH) {
                weights_f32(b, wl, wr);
            } else {
                double dl, dr;
                weights_wide(b, flavour, dl, dr);
                wl = (float)dl;
                wr = (float)dr;
            }
            float *cell = out + (((int64_t)w.b * nb + b.bin) * planes_per_bin + b.chan) * plane + (int64_t)b.y * W + b.x;
            atomicAdd(cell, wl);  // result unused -> REDG.E.ADD.F32
            if (b.bin + 1 < nb) atomicAdd(cell + planes_per_bin * plane, wr);
        }
    }
}

// ------------------------------------------------------ deterministic mode ---
// key = pixel column of the output ((b*planes + chan)*H*W + y*W + x); events
// that contribute nothing get key == invalid_key (sorted to the very end).
__global__ void __launch_bounds__(256)
det_make_keys_kernel(const double *__restrict__ ev, const int64_t *__restrict__ off, int64_t total,
                     int B, int nb, int H, int W, int flavour, uint32_t invalid_key,
                     uint32_t *__restrict__ keys, uint32_t *__restrict__ vals) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    // rows outside [off[0], off[B]) belong to no window: a row past the last one (a device-side filter kept fewer
    // rows than the buffer holds), or a row before the first (offsets sliced from a longer stream, not rebased)
    if (i < __ldg(off) || i >= __ldg(off + B)) {
        keys[i] = invalid_key;
        vals[i] = (uint32_t)i;
        return;
    }
    Window w;
    w.b = -1;
    locate_window(w, i, off, ev, B);
    const Binned b = bin_event(load_event(ev, i), w, nb, H, W, flavour);
    const int planes = flavour == CF_FLAVOUR_POL ? 2 : 1;
    uint32_t key = invalid_key;
    if (b.ok) key = (uint32_t)(((int64_t)w.b * planes + b.chan) * ((int64_t)H * W) + (int64_t)b.y * W + b.x);
    keys[i] = key;
    vals[i] = (uint32_t)i;
}

// One thread per run of equal keys (= one output pixel column).  The run is in
// event order; for time-sorted events bin indices are non-decreasing along it (runs that are not take
// the order-agnostic walk at the top of the kernel).  For each bin: first
// the left weights of the events with ti == bin, then the right weights of the
// events with ti == bin-1 -- the order of the reference's two scatter-adds.
__global__ void __launch_bounds__(256)
det_accumulate_kernel(const uint32_t *__restrict__ keys, const uint32_t *__restrict__ vals, int64_t n,
                      uint32_t invalid_key, const double *__restrict__ ev, const int64_t *__restrict__ off,
                      int B, int nb, int H, int W, int flavour, float *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t k = keys[i];
    if (k == invalid_key) return;
    if (i > 0 && keys[i - 1] == k) return;  // not the head of its run

    const int64_t plane = (int64_t)H * W;
    const int planes = flavour == CF_FLAVOUR_POL ? 2 : 1;
    const int64_t col = (int64_t)k / plane;  // b*planes + chan
    const int64_t pix = (int64_t)k - col * plane;
    const int b = (int)(col / planes), chan = (int)(col - (int64_t)b * planes);
    Window w;
    w.b = -1;
    locate_window(w, vals[i], off, ev, B);
    float *cell0 = out + ((int64_t)b * nb * planes + chan) * plane + pix;  // bin 0 of this column

    // The fast walk below needs the run's bin indices to be non-decreasing (time-sorted events).  The reference's
    // scatter-adds do not depend on that, so a run that breaks it (jittered / unsorted stamps, concatenated packs)
    // takes the order-agnostic walk: per bin, the whole run in event order.
    {
        int64_t e = i;
        int last_bin = -1;
        bool monotone = true;
        while (e < n && keys[e] == k) {
            const Binned bb = bin_event(load_event(ev, vals[e]), w, nb, H, W, flavour);
            monotone = monotone && bb.bin >= last_bin;
            last_bin = bb.bin;
            ++e;
        }
        if (!monotone) {
            for (int bin = 0; bin < nb; ++bin) {
                float acc = 0.f;
                bool touched = false;
                if (flavour == CF_FLAVOUR_MVSEC) {  // one index_put_ per bin: left and right weights interleave in event order
                    for (int64_t j = i; j < e; ++j) {
                        const Binned bb = bin_event(load_event(ev, vals[j]), w, nb, H, W, flavour);
                        if (bb.bin != bin && bb.bin != bin - 1) continue;
                        double wl, wr;
                        weights_mvsec(bb, wl, wr);
                        acc = __fadd_rn(acc, (float)(bb.bin == bin ? wl : wr));
                        touched = true;
                    }
                } else {
                    for (int pass = 0; pass < 2; ++pass) {  // all left weights (ti == bin), then all right ones (ti == bin-1)
                        for (int64_t j = i; j < e; ++j) {
                            const Binned bb = bin_event(load_event(ev, vals[j]), w, nb, H, W, flavour);
                            if (bb.bin != bin - pass) continue;
                            if (flavour == CF_FLAVOUR_TORCH) {
                                float wl, wr;
                                weights_f32(bb, wl, wr);
                                acc = __fadd_rn(acc, pass ? wr : wl);
                            } else {
                                double wl, wr;
                                weights_f64(bb, wl, wr);
                                acc = (float)__dadd_rn((double)acc, pass ? wr : wl);
                            }
                            touched = true;
                        }
                    }
                }
                if (touched) cell0[(int64_t)bin * planes * plane] = acc;
            }
            return;
        }
    }

    int64_t pos = i, prev_s = i, prev_e = i;
    for (int bin = 0; bin < nb; ++bin) {
        float acc = 0.f;
        bool touched = false;
        int64_t e = pos;
        if (flavour == CF_FLAVOUR_MVSEC) {
            // one index_put_ per bin over the time-sorted events (MVSEC_utils.py:283-292): the events of bin-1 (their
            // right weights) precede the events of this bin (their left weights); fp32 adds of fp32-cast weights
            for (int64_t j = prev_s; j < prev_e; ++j) {
                const Binned bb = bin_event(load_event(ev, vals[j]), w, nb, H, W, flavour);
                double wl, wr;
                weights_mvsec(bb, wl, wr);
                acc = __fadd_rn(acc, (float)wr);
                touched = true;
            }
            while (e < n && keys[e] == k) {
                const Binned bb = bin_event(load_event(ev, vals[e]), w, nb, H, W, flavour);
                if (bb.bin != bin) break;
                double wl, wr;
                weights_mvsec(bb, wl, wr);
                acc = __fadd_rn(acc, (float)wl);
                touched = true;
                ++e;
            }
            if (touched) cell0[(int64_t)bin * planes * plane] = acc;
            prev_s = pos;
            prev_e = e;
            pos = e;
            if (prev_s == prev_e && (pos >= n || keys[pos] != k)) break;
            continue;
        }
        while (e < n && keys[e] == k) {  // left weights, ti == bin
            const Binned bb = bin_event(load_event(ev, vals[e]), w, nb, H, W, flavour);
            if (bb.bin != bin) break;
            if (flavour == CF_FLAVOUR_TORCH) {
                float wl, wr;
                weights_f32(bb, wl, wr);
                acc = __fadd_rn(acc, wl);
            } else {
                double wl, wr;
                weights_f64(bb, wl, wr);
                acc = (float)__dadd_rn((double)acc, wl);
            }
            touched = true;
            ++e;
        }
        for (int64_t j = prev_s; j < prev_e; ++j) {  // right weights, ti == bin-1
            const Binned bb = bin_event(load_event(ev, vals[j]), w, nb, H, W, flavour);
            if (flavour == CF_FLAVOUR_TORCH) {
                float wl, wr;
                weights_f32(bb, wl, wr);
                acc = __fadd_rn(acc, wr);
            } else {
                double wl, wr;
                weights_f64(bb, wl, wr);
                acc = (float)__dadd_rn((double)acc, wr);
            }
            touched = true;
        }
        if (touched) cell0[(int64_t)bin * planes * plane] = acc;
        prev_s = pos;
        prev_e = e;
        pos = e;
        if (prev_s == prev_e && (pos >= n || keys[pos] != k)) break;
    }
}

// ---------------------------------------------- statistics + normalisation ---
constexpr int kStatThreads = 256;

// Both kernels: one CTA = one chunk of a window; a thread streams its float4s with 4 loads in flight.
// (Round-1a sized them for 296 CTAs with one load in flight per thread: 43 of 70 us at 8 x 480x640.)
__global__ void __launch_bounds__(kStatThreads)
voxel_stats_kernel(const float *__restrict__ grid, int64_t cells, int64_t chunk_len, float hot_thr,
                   Partial *__restrict__ partials, int chunks) {
    const int b = (int)blockIdx.y, c = (int)blockIdx.x;
    const float *g = grid + (int64_t)b * cells;
    const int64_t s = (int64_t)c * chunk_len, e = min(cells, s + chunk_len);
    // fp64 partials per thread: a thread takes chunk_len / 256 terms, ~300 at 64 x 5x480x640 and thousands for
    // larger batches, and fp32 running sums of a grid whose mean is large against its spread lose the variance
    double fs = 0.0, fq = 0.0;
    int fn = 0;
    float mn = INFINITY, mx = -INFINITY;
    auto take = [&](float raw) {
        const float v = hot_filter(raw, hot_thr);
        fs += (double)v;
        fq = fma((double)v, (double)v, fq);   // the square of an fp32 value is exact in fp64
        fn += (v != 0.f);
        mn = fminf(mn, v);
        mx = fmaxf(mx, v);
    };
    if (((cells | chunk_len) & 3) == 0) {  // 128-bit loads (chunk starts stay 16-byte aligned)
        const float4 *g4 = reinterpret_cast<const float4 *>(g);
        const int64_t e4 = e >> 2;
        for (int64_t i = (s >> 2) + threadIdx.x; i < e4; i += 4 * kStatThreads) {
            float4 q[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int64_t j = i + (int64_t)u * kStatThreads;
                q[u] = j < e4 ? __ldg(g4 + j) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (i + (int64_t)u * kStatThreads < e4) { take(q[u].x); take(q[u].y); take(q[u].z); take(q[u].w); }
            }
        }
    } else {
        for (int64_t i = s + threadIdx.x; i < e; i += kStatThreads) take(__ldg(g + i));
    }
    // fixed-shape tree: deterministic for a given launch geometry
    double sum = warp_sum(fs), sumsq = warp_sum(fq);
    long long nnz = warp_sum((long long)fn);
    mn = warp_min(mn); mx = warp_max(mx);
    __shared__ Partial sh[kStatThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) sh[warp] = Partial{sum, sumsq, nnz, mn, mx};
    __syncthreads();
    if (threadIdx.x == 0) {
        Partial t = sh[0];
        for (int k = 1; k < kStatThreads / 32; ++k) {
            t.sum += sh[k].sum; t.sumsq += sh[k].sumsq; t.nnz += sh[k].nnz;
            t.mn = fminf(t.mn, sh[k].mn); t.mx = fmaxf(t.mx, sh[k].mx);
        }
        partials[(size_t)b * chunks + c] = t;
    }
}

__global__ void __launch_bounds__(kStatThreads)
voxel_normalise_kernel(const float *in, float *out /* may alias in */, int64_t cells, int64_t chunk_len,
                       float hot_thr, int mode, const Partial *__restrict__ partials, int chunks) {
    const int b = (int)blockIdx.y, c = (int)blockIdx.x;
    const float *g = in + (int64_t)b * cells;
    float *o = out + (int64_t)b * cells;
    const int64_t s = (int64_t)c * chunk_len, e = min(cells, s + chunk_len);
    const bool vec = ((cells | chunk_len) & 3) == 0;
    // this thread's first loads go out before the window's partials are reduced
    const float4 *g4 = reinterpret_cast<const float4 *>(g);
    float4 *o4 = reinterpret_cast<float4 *>(o);
    const int64_t e4 = e >> 2, i0 = (s >> 2) + threadIdx.x;
    float4 q[4];
    if (vec) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t j = i0 + (int64_t)u * kStatThreads;
            q[u] = j < e4 ? g4[j] : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    __shared__ float s_a, s_b;   // out = (v - s_a) * s_b
    __shared__ int s_identity;
    if (threadIdx.x < 32) {
        // every CTA of a window re-reduces the window's partials in the same fixed order
        const Partial *p = partials + (size_t)b * chunks;
        double sum = 0.0, sumsq = 0.0;
        long long nnz = 0;
        float mn = INFINITY, mx = -INFINITY;
        for (int k = threadIdx.x; k < chunks; k += 32) {
            sum += p[k].sum; sumsq += p[k].sumsq; nnz += p[k].nnz;
            mn = fminf(mn, p[k].mn); mx = fmaxf(mx, p[k].mx);
        }
        sum = warp_sum(sum); sumsq = warp_sum(sumsq); nnz = warp_sum(nnz);
        mn = warp_min(mn); mx = warp_max(mx);
        if (threadIdx.x == 0) {
            if (mode == CF_PRE_STD) {
                s_identity = nnz == 0;  // event_process.py:205 -- untouched when there is no non-zero entry
                const double mean = nnz ? sum / (double)nnz : 0.0;
                const double var = nnz ? sumsq / (double)nnz - mean * mean : 0.0;
                s_a = (float)mean;
                s_b = (float)(1.0 / (sqrt(fmax(var, 0.0)) + 1e-8));
            } else {
                s_identity = 0;
                s_a = mn;
                s_b = (float)(1.0 / ((double)mx - (double)mn + 1e-8));
            }
        }
    }
    __syncthreads();
    const float a = s_a, inv = s_b;
    const bool identity = s_identity != 0;
    // mean and 1/(std+eps) are formed in fp64 once per window; the per-cell map is fp32 (1 ulp of the
    // fp64 formula rounded to fp32; a true fp64 divide per cell made this kernel 3x slower than the scatter)
    auto norm = [&](float raw) -> float {
        const float v = hot_filter(raw, hot_thr);
        if (identity) return v;
        const float r = (v - a) * inv;
        return (mode == CF_PRE_STD && v == 0.f) ? 0.f : r;
    };
    // in place, std mode: zero cells stay zero (event_process.py:207-210) -- an all-zero float4 is not rewritten
    const bool skip_zero = (in == out) && mode == CF_PRE_STD;
    if (vec) {
        for (int64_t i = i0; i < e4; i += 4 * kStatThreads) {
            if (i != i0) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int64_t j = i + (int64_t)u * kStatThreads;
                    q[u] = j < e4 ? g4[j] : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int64_t j = i + (int64_t)u * kStatThreads;
                if (j < e4) {
                    if (skip_zero && q[u].x == 0.f && q[u].y == 0.f && q[u].z == 0.f && q[u].w == 0.f) continue;
                    o4[j] = make_float4(norm(q[u].x), norm(q[u].y), norm(q[u].z), norm(q[u].w));
                }
            }
        }
    } else {
        for (int64_t i = s + threadIdx.x; i < e; i += kStatThreads) o[i] = norm(g[i]);
    }
}

static void stat_geometry(int B, int64_t cells, int &chunks, int64_t &chunk_len) {
    // ~8 CTAs per SM over the batch, chunks of >= 2048 cells (2 float4 per thread), <= kMaxChunks per window
    int64_t want = ceil_div(8 * 148, B > 0 ? B : 1);
    int64_t cap = ceil_div(cells, 2048);
    chunks = (int)(want < 1 ? 1 : want);
    if (chunks > cap) chunks = (int)(cap < 1 ? 1 : cap);
    if (chunks > kMaxChunks) chunks = kMaxChunks;
    chunk_len = ceil_div(cells, chunks);
    chunk_len = (chunk_len + 3) & ~(int64_t)3;  // keeps every chunk start 16-byte aligned
}

// statistics + normalisation of B grids; also used by the packed-event path (voxel_packed.cu)
int run_preprocess(const float *in, float *out, int B, int64_t cells, int preprocess, float hot_thr, void *ws,
                   size_t ws_bytes, cudaStream_t stream) {
    CF_REQUIRE(B <= 65535, CF_ERR_INVALID_ARG, "preprocess: B > 65535");
    CF_REQUIRE(ws && ws_bytes >= (size_t)B * kMaxChunks * sizeof(Partial), CF_ERR_WORKSPACE,
               "preprocess: workspace too small (%zu < %zu)", ws_bytes, (size_t)B * kMaxChunks * sizeof(Partial));
    CF_REQUIRE(aligned16(ws), CF_ERR_ALIGN, "preprocess: workspace not 16-byte aligned");
    int chunks;
    int64_t chunk_len;
    stat_geometry(B, cells, chunks, chunk_len);
    Partial *partials = reinterpret_cast<Partial *>(ws);
    dim3 grid(chunks, B);
    voxel_stats_kernel<<<grid, kStatThreads, 0, stream>>>(in, cells, chunk_len, hot_thr, partials, chunks);
    CF_LAUNCH_CHECK("voxel_stats_kernel");
    voxel_normalise_kernel<<<grid, kStatThreads, 0, stream>>>(in, out, cells, chunk_len, hot_thr, preprocess, partials, chunks);
    CF_LAUNCH_CHECK("voxel_normalise_kernel");
    return CF_OK;
}

// implemented in voxel_tiled.cu (CF_VOXEL_ATOMIC_TILED)
size_t voxel_tiled_workspace_bytes(int64_t total, int B, int nb, int H, int W, int flavour);
int launch_voxel_tiled(const double *events, const int64_t *offsets, int64_t total, int B, int nb, int H, int W,
                       int flavour, int preprocess, float hot_thr, float *out, void *ws, size_t ws_bytes,
                       cudaStream_t stream);

// ATOMIC mode has two data paths with identical numerics (sum order unspecified in both):
//   L2 atomics (this file, the default): zero -> RED.ADD into the L2-resident grid -> statistics ->
//     normalise in place;
//   tiled (voxel_tiled.cu, CF_VOXEL_ATOMIC_TILED): partition into 12-byte records -> accumulate tiles in
//     shared memory -> statistics, normalisation and the only write of the grid out of shared memory.
// Measured on the B200 (scripts/scale_bench.py, us per launch, fused std normalisation, round 1):
//                 8x180x240  64x180x240  1x260x346  64x260x346  8x480x640  1x624x970
//   L2 atomics       16.4       50.8       10.3       132.0       43.8       30.0
//   tiled            19.4      107.5       15.4       160.1       57.1       49.6
// The tiled path issues no global atomic, but its two kernels are each a chain of dependent steps
// (window lookup -> event loads -> fp64 decode -> counting sort -> write; run bounds -> records ->
// shared-memory atomics -> statistics -> per-window barrier -> normalise -> write: timelines from
// scripts/voxel_trace.py in profiles/), two waves are needed as soon as the batch's grids exceed the
// chip's 33 MB of shared memory, and the ~100 G/s of L2 atomics it avoids were not the bound once the
// statistics/normalise kernels were given enough loads in flight.  So the L2 path is the default and the
// tiled path stays selectable (and tested) for the next round's work on it.
struct DetLayout {
    size_t keys0, vals0, keys1, vals1, hist, end;
    int nblk;
};
static DetLayout det_layout(int64_t total, size_t base) {
    DetLayout L;
    L.nblk = (int)ceil_div(total > 0 ? total : 1, kRsTile);
    const size_t arr = align_up((size_t)(total > 0 ? total : 1) * sizeof(uint32_t), 256);
    L.keys0 = base;
    L.vals0 = L.keys0 + arr;
    L.keys1 = L.vals0 + arr;
    L.vals1 = L.keys1 + arr;
    L.hist = L.vals1 + arr;
    L.end = L.hist + align_up((size_t)256 * L.nblk * sizeof(uint32_t), 256);
    return L;
}

}  // namespace cf

extern "C" size_t cf_preprocess_workspace_bytes(int B, int64_t) {
    return (size_t)(B > 0 ? B : 1) * cf::kMaxChunks * sizeof(cf::Partial);
}

extern "C" size_t cf_voxel_workspace_bytes(int64_t total_events, int B, int nb, int H, int W, int mode, int flavour, int) {
    size_t base = cf::align_up(cf_preprocess_workspace_bytes(B, 0), 256);
    if (mode == CF_VOXEL_DETERMINISTIC) return cf::det_layout(total_events, base).end;
    // CF_VOXEL_ATOMIC runs the L2 path (cf_voxel_bin): only the forced tiled path needs its records and tables
    if (mode == CF_VOXEL_ATOMIC_TILED && nb > 0 && H > 0 && W > 0)
        base += cf::voxel_tiled_workspace_bytes(total_events, B, nb, H, W, flavour);
    return base;
}

extern "C" int cf_voxel_preprocess(const float *in, float *out, int B, int64_t cells, int preprocess, float hot_thr,
                                   void *ws, size_t ws_bytes, cf_stream_t stream_) {
    using namespace cf;
    if (int rc = check_device()) return rc;
    CF_REQUIRE(in && out, CF_ERR_NULL, "cf_voxel_preprocess: null pointer");
    CF_REQUIRE(B >= 0 && cells > 0, CF_ERR_INVALID_ARG, "cf_voxel_preprocess: bad shape");
    CF_REQUIRE(preprocess == CF_PRE_STD || preprocess == CF_PRE_MAXMIN, CF_ERR_INVALID_ARG,
               "cf_voxel_preprocess: mode must be CF_PRE_STD or CF_PRE_MAXMIN");
    if (B == 0) return CF_OK;
    return run_preprocess(in, out, B, cells, preprocess, hot_thr, ws, ws_bytes, (cudaStream_t)stream_);
}

extern "C" int cf_voxel_bin(const double *events, const int64_t *offsets, int64_t total, int B, int nb, int H, int W,
                            int mode, int flavour, int preprocess, float hot_thr, float *out,
                            void *ws, size_t ws_bytes, cf_stream_t stream_) {
    using namespace cf;
    if (int rc = check_device()) return rc;
    CF_REQUIRE(out && offsets, CF_ERR_NULL, "cf_voxel_bin: null pointer");
    CF_REQUIRE(total == 0 || events, CF_ERR_NULL, "cf_voxel_bin: events is null");
    CF_REQUIRE(nb > 0 && H > 0 && W > 0, CF_ERR_INVALID_ARG, "cf_voxel_bin: num_bins, width, height must be > 0");
    CF_REQUIRE(B >= 0 && total >= 0, CF_ERR_INVALID_ARG, "cf_voxel_bin: negative size");
    CF_REQUIRE(mode >= CF_VOXEL_ATOMIC && mode <= CF_VOXEL_ATOMIC_TILED, CF_ERR_INVALID_ARG, "cf_voxel_bin: bad mode %d", mode);
    const bool force_l2 = mode == CF_VOXEL_ATOMIC_L2, force_tiled = mode == CF_VOXEL_ATOMIC_TILED;
    if (force_l2 || force_tiled) mode = CF_VOXEL_ATOMIC;
    CF_REQUIRE(flavour >= CF_FLAVOUR_TORCH && flavour <= CF_FLAVOUR_MVSEC, CF_ERR_INVALID_ARG, "cf_voxel_bin: bad flavour %d", flavour);
    CF_REQUIRE(!(force_tiled && flavour == CF_FLAVOUR_MVSEC), CF_ERR_UNSUPPORTED,
               "cf_voxel_bin: CF_VOXEL_ATOMIC_TILED does not implement CF_FLAVOUR_MVSEC");
    CF_REQUIRE(preprocess >= CF_PRE_NONE && preprocess <= CF_PRE_MAXMIN, CF_ERR_INVALID_ARG, "cf_voxel_bin: bad preprocess %d", preprocess);
    CF_REQUIRE(total == 0 || aligned16(events), CF_ERR_ALIGN, "cf_voxel_bin: events not 16-byte aligned");
    CF_REQUIRE(total < (1ll << 32), CF_ERR_INVALID_ARG, "cf_voxel_bin: more than 2^32 events in one call");
    if (B == 0) return CF_OK;
    cudaStream_t stream = (cudaStream_t)stream_;
    const int planes = flavour == CF_FLAVOUR_POL ? 2 : 1;
    const int64_t cells = (int64_t)nb * planes * H * W;
    if (force_tiled) {
        const size_t base = align_up(cf_preprocess_workspace_bytes(B, 0), 256);
        const size_t need = voxel_tiled_workspace_bytes(total, B, nb, H, W, flavour);
        if (need > 0 && total > 0) {
            CF_REQUIRE(ws && ws_bytes >= base + need, CF_ERR_WORKSPACE, "cf_voxel_bin: workspace too small (%zu < %zu)",
                       ws_bytes, base + need);
            const int rc = launch_voxel_tiled(events, offsets, total, B, nb, H, W, flavour, preprocess, hot_thr, out,
                                              reinterpret_cast<char *>(ws) + base, ws_bytes - base, stream);
            if (rc != 1) return rc;  // 1 = geometry not covered
        }
        // an empty batch takes the L2-atomic path below (zero-fill + normalise)
        CF_REQUIRE(total == 0, CF_ERR_UNSUPPORTED,
                   "cf_voxel_bin: CF_VOXEL_ATOMIC_TILED does not cover B=%d, %dx%d, nb=%d", B, H, W, nb);
    }
    if (mode == CF_VOXEL_ATOMIC) {
        // Chunks of windows that stay L2-resident from the zero-fill to the normalised write-back.
        // The host does not know the per-window event counts (offsets live on the device), so the
        // events of a chunk are budgeted with the batch average; kernels take device offsets.
        const size_t per_window = (size_t)cells * sizeof(float) + (size_t)(total / B + 1) * 32;
        int chunk = (int)(kL2ChunkBytes / per_window);
        if (chunk < 1) chunk = 1;
        if (chunk > B) chunk = B;
        if (preprocess != CF_PRE_NONE) {
            CF_REQUIRE(ws && ws_bytes >= (size_t)B * kMaxChunks * sizeof(Partial), CF_ERR_WORKSPACE,
                       "cf_voxel_bin: workspace too small (%zu < %zu)", ws_bytes, (size_t)B * kMaxChunks * sizeof(Partial));
            CF_REQUIRE(aligned16(ws), CF_ERR_ALIGN, "cf_voxel_bin: workspace not 16-byte aligned");
        }
        for (int b0 = 0; b0 < B; b0 += chunk) {
            const int nbat = B - b0 < chunk ? B - b0 : chunk;
            float *o = out + (size_t)b0 * cells;
            CF_CUDA(cudaMemsetAsync(o, 0, sizeof(float) * (size_t)nbat * cells, stream));
            if (total > 0) {
                // grid sized for the chunk's expected share of the events, capped at 8 CTAs per SM;
                // the kernel grid-strides, so a longer-than-average chunk is still fully processed
                int64_t blocks = ceil_div(ceil_div(total * nbat, B), kScatterThreads * kScatterUnroll);
                const int64_t cap = (int64_t)sm_count() * 8;
                if (blocks > cap) blocks = cap;
                if (blocks < 1) blocks = 1;
                voxel_scatter_atomic_kernel<<<(unsigned)blocks, kScatterThreads, 0, stream>>>(
                    events, offsets, B, nb, H, W, flavour, out, b0, b0 + nbat);
                CF_LAUNCH_CHECK("voxel_scatter_atomic_kernel");
            }
            if (preprocess != CF_PRE_NONE) {
                if (int rc = run_preprocess(o, o, nbat, cells, preprocess, hot_thr,
                                            reinterpret_cast<char *>(ws) + (size_t)b0 * kMaxChunks * sizeof(Partial),
                                            ws_bytes - (size_t)b0 * kMaxChunks * sizeof(Partial), stream)) return rc;
            }
        }
        return CF_OK;
    }
    CF_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)B * cells, stream));
    if (total > 0) {
        const uint64_t columns = (uint64_t)B * planes * H * W;  // invalid key == columns
        CF_REQUIRE(columns < 0xffffffffull, CF_ERR_INVALID_ARG, "cf_voxel_bin: B*H*W too large for the deterministic mode");
        const size_t base = align_up(cf_preprocess_workspace_bytes(B, 0), 256);
        const DetLayout L = det_layout(total, base);
        CF_REQUIRE(ws && ws_bytes >= L.end, CF_ERR_WORKSPACE, "cf_voxel_bin: workspace too small (%zu < %zu)", ws_bytes, L.end);
        CF_REQUIRE(aligned16(ws), CF_ERR_ALIGN, "cf_voxel_bin: workspace not 16-byte aligned");
        char *w8 = reinterpret_cast<char *>(ws);
        uint32_t *k0 = (uint32_t *)(w8 + L.keys0), *v0 = (uint32_t *)(w8 + L.vals0);
        uint32_t *k1 = (uint32_t *)(w8 + L.keys1), *v1 = (uint32_t *)(w8 + L.vals1);
        uint32_t *hist = (uint32_t *)(w8 + L.hist);
        const unsigned eb = (unsigned)ceil_div(total, 256);
        det_make_keys_kernel<<<eb, 256, 0, stream>>>(events, offsets, total, B, nb, H, W, flavour, (uint32_t)columns, k0, v0);
        CF_LAUNCH_CHECK("det_make_keys_kernel");
        const int passes = (radix_bits(columns) + 7) / 8;
        for (int p = 0; p < passes; ++p) {
            rs_hist_kernel<<<L.nblk, kRsThreads, 0, stream>>>(k0, total, 8 * p, hist, L.nblk);
            CF_LAUNCH_CHECK("rs_hist_kernel");
            rs_scan_kernel<<<1, 1024, 0, stream>>>(hist, (int64_t)256 * L.nblk);
            CF_LAUNCH_CHECK("rs_scan_kernel");
            rs_scatter_kernel<<<L.nblk, kRsThreads, 0, stream>>>(k0, v0, k1, v1, total, 8 * p, hist, L.nblk);
            CF_LAUNCH_CHECK("rs_scatter_kernel");
            uint32_t *t = k0; k0 = k1; k1 = t;
            t = v0; v0 = v1; v1 = t;
        }
        det_accumulate_kernel<<<eb, 256, 0, stream>>>(k0, v0, total, (uint32_t)columns, events, offsets, B, nb, H, W, flavour, out);
        CF_LAUNCH_CHECK("det_accumulate_kernel");
    }
    if (preprocess != CF_PRE_NONE)
        return run_preprocess(out, out, B, cells, preprocess, hot_thr, ws, ws_bytes, stream);
    return CF_OK;
}
