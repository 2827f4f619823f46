// On-demand correlation lookup (AlternateCorrBlock, include/cistaflow_altcorr.h) for sm_100a.
//
// Replaces DCEIFlow/core/corr/raft_corr.py:175-203 (RAFT's AlternateCorrBlock, whose alt_cuda_corr extension the
// reference does not ship).  No all-pairs volume: the state holds fmap1 and the pooled levels of fmap2, channel-last
// ([B, h_l, w_l, D]: every pixel is one K-major row), and each lookup computes the (2r+2)^2 dot products of every
// query's bilinear patches itself.  avg_pool2d is linear, so the pooled feature map gives the pooled correlation.
//
// State (cf_corr_alt_workspace_bytes): [fmap1 as B,h,w,D] [level 0 of fmap2] [level 1] ... each region rounded up to
// 256 bytes: 2.33 x the bytes of one feature map at 4 levels, against B*N^2*4*1.33 for the pyramid.
//
// Lookup, tensor cores (corr_alt_tc_kernel, one CTA per tile of 16x8 queries = the 128 TMEM lanes):
//   prologue   the 128 query threads reduce, per level, the bounds of the tile's patch origins
//              floor(coords / 2^l) - r.  Their union is a box of targets; the tile is served here when every level's
//              box is at most bw_l targets wide and 8 * bh_l rows high (bw_l * bh_l = 256, the UMMA N limit), else
//              the CTA exits and the fp32 kernel, which evaluates the same predicate (tile_box), serves it.
//   producer   per level and band of bh_l box rows, per 32 channels: one TMA box of the 128 queries
//              {32 ch, 16 x, 8 y} and one of the band {32 ch, bw_l, bh_l}, 128-byte swizzle, TF32 rounding in the
//              TMA unit (CU_TENSOR_MAP_DATA_TYPE_TFLOAT32); targets outside the map are zero-filled by the TMA unit,
//              which is grid_sample's zero padding.
//   MMA        tcgen05.mma kind::tf32, M = 128 queries, N = 256 band targets, K = D; two TMEM accumulators.
//   epilogue   each thread owns one query (its TMEM lane): for every band row inside its patch it copies the row
//              from TMEM to a private strip of shared memory (dynamic indexing), forms the 2r+1 horizontal lerps and,
//              with the previous patch row's lerps (kept in shared memory), the 2r+1 outputs of one window row.
// Lookup, fp32 (corr_alt_simt_kernel): a warp per query, a lane per patch target, fp32 FMA dot products.  It serves
// the tiles the tensor cores leave, precision FP32, and D % 32 != 0.
#include <algorithm>
#include <climits>

#include "cistaflow_altcorr.h"
#include "tcgen05.cuh"
#include "tma.cuh"

namespace cf {
namespace alt {

constexpr int TX = 16, TY = 8;                  // query tile (TX * TY = 128 = UMMA M)
constexpr int MAX_BANDS = 8;                    // box rows per level at most MAX_BANDS * bh_l (32 rows at bw_l = 64)
constexpr int BAND_N = 256;                     // UMMA N: targets of one band
constexpr int KC = 32;                          // channels per stage: one 128-byte row per query / target
constexpr int STAGES = 3;
constexpr int A_BYTES = tc::BM * KC * 4;        // 16 KB
constexpr int B_BYTES = BAND_N * KC * 4;        // 32 KB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int MAX_BW = 64;                      // widest box (radius 8)
constexpr int STG_STRIDE = MAX_BW + 1;          // odd: a TMEM row lands in 32 distinct banks
constexpr int MAX_K = 17;                       // 2r+1 at radius 8
constexpr int TC_THREADS = 192;                 // warps 0-3 epilogue, 4 TMA producer, 5 TMEM allocator + MMA issuer
constexpr int TC_SMEM = STAGES * STAGE_BYTES + 4 * 32 * STG_STRIDE * 4 + MAX_K * tc::BM * 4 + 1024;
constexpr int SIMT_THREADS = 256;
constexpr float COORD_CLAMP = 1.0e6f;           // cf_corr_lookup's clamp: keeps float -> int defined (NaN -> -1e6)

struct Args {
    const float *f1;                            // [B, h, w, D]
    const float *lv[CF_CORR_MAX_LEVELS];        // level l of fmap2, [B, h_l, w_l, D]
    const float *coords;                        // [B, 2, h, w]
    float *out;                                 // [B, levels*(2r+1)^2, h, w]
    int D, h, w, levels, r;
    int hl[CF_CORR_MAX_LEVELS], wl[CF_CORR_MAX_LEVELS];
    int bw[CF_CORR_MAX_LEVELS], bh[CF_CORR_MAX_LEVELS];   // box width and band height of level l (bw * bh = 256)
    int tiles_x;
    int tc;                                     // 1: corr_alt_tc_kernel serves the tiles whose boxes fit
    float scale;                                // 1 / sqrt(D)
};

struct Maps {
    CUtensorMap m[1 + CF_CORR_MAX_LEVELS];      // [0] fmap1, [1 + l] level l
};

struct TileBox {
    int x0[CF_CORR_MAX_LEVELS], y0[CF_CORR_MAX_LEVELS];  // box origin (smallest patch origin) per level
    int rows[CF_CORR_MAX_LEVELS];                        // box rows per level
    int fits;
};

__device__ __forceinline__ float clamp_coord(float c) { return fminf(fmaxf(c, -COORD_CLAMP), COORD_CLAMP); }

// Called by every thread of the block; threads 0..127 own the tile's queries.  Both lookup kernels evaluate this
// with the same arithmetic, so each tile is served by exactly one of them without a read-back.
__device__ void tile_box(const Args &a, int b, int qx0, int qy0, int *red, TileBox &tb) {
    const int t = threadIdx.x;
    if (t < 4 * CF_CORR_MAX_LEVELS) red[t] = (t & 1) ? INT_MIN : INT_MAX;   // [l][min x, max x, min y, max y]
    __syncthreads();
    const int qx = qx0 + (t & (TX - 1)), qy = qy0 + t / TX;
    if (t < tc::BM && qx < a.w && qy < a.h) {
        const size_t N = (size_t)a.h * a.w, q = (size_t)qy * a.w + qx;
        const float *cb = a.coords + (size_t)b * 2 * N;
        const float cx = clamp_coord(cb[q]), cy = clamp_coord(cb[N + q]);
        for (int l = 0; l < a.levels; ++l) {
            const float inv = 1.f / (float)(1 << l);
            const int bx = (int)floorf(cx * inv) - a.r, by = (int)floorf(cy * inv) - a.r;
            atomicMin(&red[4 * l], bx);
            atomicMax(&red[4 * l + 1], bx);
            atomicMin(&red[4 * l + 2], by);
            atomicMax(&red[4 * l + 3], by);
        }
    }
    __syncthreads();
    if (t == 0) {
        int fits = a.tc;
        for (int l = 0; l < a.levels; ++l) {
            const int wd = red[4 * l + 1] - red[4 * l] + 2 * a.r + 2, ht = red[4 * l + 3] - red[4 * l + 2] + 2 * a.r + 2;
            fits &= (wd <= a.bw[l] && ht <= MAX_BANDS * a.bh[l]) ? 1 : 0;
            tb.x0[l] = red[4 * l];
            tb.y0[l] = red[4 * l + 2];
            tb.rows[l] = ht;
        }
        tb.fits = fits;
    }
    __syncthreads();
}

__global__ void __launch_bounds__(TC_THREADS, 1)
corr_alt_tc_kernel(const __grid_constant__ Maps maps, const __grid_constant__ Args a) {
    using namespace tc;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *ring = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    float *stg = reinterpret_cast<float *>(ring + STAGES * STAGE_BYTES);   // [128 queries][STG_STRIDE]
    float *hp = stg + tc::BM * STG_STRIDE;                                  // [2r+1][128]: previous patch row's lerps
    __shared__ int red[4 * CF_CORR_MAX_LEVELS];
    __shared__ TileBox tb;
    __shared__ uint64_t full[STAGES], empty[STAGES], tfull[2], tempty[2];
    __shared__ uint32_t tmem_slot;

    const int b = blockIdx.y;
    const int qx0 = (int)(blockIdx.x % (unsigned)a.tiles_x) * TX, qy0 = (int)(blockIdx.x / (unsigned)a.tiles_x) * TY;
    tile_box(a, b, qx0, qy0, red, tb);
    if (!tb.fits) return;   // uniform: the fp32 kernel serves this tile

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 5) {
        if (lane == 0) {
            for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
            for (int s = 0; s < 2; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], tc::BM); }
            fence_barrier_init();
        }
        __syncwarp();
        tmem_alloc(&tmem_slot, 2 * BAND_N);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;
    const int kchunks = a.D / KC;

    if (warp == 4) {
        // ------------------------------------------------------------ TMA producer
        if (lane == 0) {
            for (int l = 0; l <= a.levels; ++l) tma_prefetch_desc(&maps.m[l]);
        }
        int stage = 0;
        uint32_t phase = 0;
        for (int l = 0; l < a.levels; ++l) {
            const int bands = (tb.rows[l] + a.bh[l] - 1) / a.bh[l];
            for (int band = 0; band < bands; ++band) {
                for (int kc = 0; kc < kchunks; ++kc) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    if (elect_one()) {
                        uint8_t *sa = ring + stage * STAGE_BYTES;
                        mbar_expect_tx(&full[stage], STAGE_BYTES);
                        tma_load_4d(sa, &maps.m[0], kc * KC, qx0, qy0, b, &full[stage]);
                        tma_load_4d(sa + A_BYTES, &maps.m[1 + l], kc * KC, tb.x0[l], tb.y0[l] + band * a.bh[l], b, &full[stage]);
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 5) {
        // -------------------------------------------------------------- MMA issuer
        const uint32_t idesc = make_idesc_tf32_kmajor(BAND_N);
        const uint32_t ring_base = smem_u32(ring);
        int stage = 0, acc = 0;
        uint32_t phase = 0, acc_phase = 0;
        for (int l = 0; l < a.levels; ++l) {
            const int bands = (tb.rows[l] + a.bh[l] - 1) / a.bh[l];
            for (int band = 0; band < bands; ++band) {
                mbar_wait(&tempty[acc], acc_phase ^ 1);   // the epilogue drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BAND_N);
                for (int kc = 0; kc < kchunks; ++kc) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t sa = ring_base + (uint32_t)(stage * STAGE_BYTES);
                    if (elect_one()) {
#pragma unroll
                        for (int kk = 0; kk < KC / 8; ++kk)
                            umma_tf32(d_tmem, make_desc_k_sw128(sa + 32 * kk), make_desc_k_sw128(sa + A_BYTES + 32 * kk), idesc,
                                      (uint32_t)((kc | kk) != 0));
                        umma_commit(&empty[stage]);                    // frees the stage once these MMAs have read it
                        if (kc == kchunks - 1) umma_commit(&tfull[acc]);  // the band's accumulator is complete
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                acc ^= 1;
                if (acc == 0) acc_phase ^= 1;
            }
        }
    } else {
        // ---------------------------------------------------------------- epilogue
        const int t = threadIdx.x;
        const int qx = qx0 + (t & (TX - 1)), qy = qy0 + t / TX;
        const bool valid = qx < a.w && qy < a.h;
        const int N = a.h * a.w, K = 2 * a.r + 1;
        float cx = 0.f, cy = 0.f;
        if (valid) {
            const float *cb = a.coords + (size_t)b * 2 * N;
            cx = clamp_coord(cb[qy * a.w + qx]);
            cy = clamp_coord(cb[N + qy * a.w + qx]);
        }
        float *st = stg + t * STG_STRIDE;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int l = 0; l < a.levels; ++l) {
            const float inv = 1.f / (float)(1 << l);
            const float sx = cx * inv, sy = cy * inv;
            const float fsx = floorf(sx), fsy = floorf(sy);
            const float fx = sx - fsx, fy = sy - fsy, gx = 1.f - fx, gy = 1.f - fy;
            const int ox = (int)fsx - a.r - tb.x0[l];          // patch origin inside the box
            const int py0 = (int)fsy - a.r - tb.y0[l];
            const int bw = a.bw[l], bh = a.bh[l];
            const int bands = (tb.rows[l] + bh - 1) / bh;
            float *ob = a.out + ((size_t)b * a.levels * K * K + (size_t)l * K * K) * N + (size_t)qy * a.w + qx;
            for (int band = 0; band < bands; ++band) {
                mbar_wait(&tfull[acc], acc_phase);
                tc_fence_after();
                const int rows = min(bh, tb.rows[l] - band * bh);
                const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(acc * BAND_N);
                for (int rr = 0; rr < rows; ++rr) {
                    for (int c0 = 0; c0 < bw; c0 += 16) {   // warp-uniform: tcgen05.ld is .sync.aligned
                        uint32_t v[16];
                        tmem_ld16(trow + (uint32_t)(rr * bw + c0), v);
#pragma unroll
                        for (int j = 0; j < 16; ++j) st[c0 + j] = __uint_as_float(v[j]) * a.scale;
                    }
                    const int py = band * bh + rr - py0;            // row of this query's patch
                    if (valid && py >= 0 && py <= K) {
                        for (int i = 0; i < K; ++i) {               // i -> x offset (transposed window, SURVEY F7)
                            const float hcur = st[ox + i] * gx + st[ox + i + 1] * fx;
                            if (py > 0) ob[(size_t)(i * K + py - 1) * N] = hp[i * tc::BM + t] * gy + hcur * fy;
                            hp[i * tc::BM + t] = hcur;
                        }
                    }
                }
                tc_fence_before();
                mbar_arrive(&tempty[acc]);
                acc ^= 1;
                if (acc == 0) acc_phase ^= 1;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 5) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 2 * BAND_N);
    }
}

// fp32 SIMT lookup: a warp per query, a lane per patch target.  Shared memory per warp: the query's fmap1 row [D]
// and the level's patch [(2r+2)^2].
__global__ void __launch_bounds__(SIMT_THREADS)
corr_alt_simt_kernel(const __grid_constant__ Args a) {
    extern __shared__ float sm[];
    __shared__ int red[4 * CF_CORR_MAX_LEVELS];
    __shared__ TileBox tb;
    const int b = blockIdx.y;
    const int qx0 = (int)(blockIdx.x % (unsigned)a.tiles_x) * TX, qy0 = (int)(blockIdx.x / (unsigned)a.tiles_x) * TY;
    if (a.tc) {
        tile_box(a, b, qx0, qy0, red, tb);
        if (tb.fits) return;   // the tensor-core kernel serves this tile
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int D = a.D, K = 2 * a.r + 1, P = K + 1, PP = P * P, N = a.h * a.w;
    float *f1s = sm + (size_t)warp * (D + PP);
    float *pat = f1s + D;
    const bool vec4 = (D & 3) == 0;
    for (int i = warp; i < tc::BM; i += SIMT_THREADS / 32) {
        const int qx = qx0 + (i & (TX - 1)), qy = qy0 + i / TX;
        if (qx >= a.w || qy >= a.h) continue;   // warp-uniform
        const int q = qy * a.w + qx;
        const float *fr = a.f1 + ((size_t)b * N + q) * D;
        for (int c = lane; c < D; c += 32) f1s[c] = fr[c];
        const float *cb = a.coords + (size_t)b * 2 * N;
        const float cx = clamp_coord(cb[q]), cy = clamp_coord(cb[N + q]);
        __syncwarp();
        for (int l = 0; l < a.levels; ++l) {
            const float inv = 1.f / (float)(1 << l);
            const float sx = cx * inv, sy = cy * inv;
            const float fsx = floorf(sx), fsy = floorf(sy);
            const float fx = sx - fsx, fy = sy - fsy, gx = 1.f - fx, gy = 1.f - fy;
            const int bx = (int)fsx - a.r, by = (int)fsy - a.r;
            const int Hl = a.hl[l], Wl = a.wl[l];
            for (int e = lane; e < PP; e += 32) {
                const int py = e / P, px = e - py * P;
                const int X = bx + px, Y = by + py;
                float s = 0.f;
                if (X >= 0 && X < Wl && Y >= 0 && Y < Hl) {
                    const float *tr = a.lv[l] + (((size_t)b * Hl + Y) * Wl + X) * D;
                    if (vec4) {
                        for (int c = 0; c < D; c += 4) {
                            const float4 u = *reinterpret_cast<const float4 *>(f1s + c);
                            const float4 v = __ldg(reinterpret_cast<const float4 *>(tr + c));
                            s = fmaf(u.x, v.x, s);
                            s = fmaf(u.y, v.y, s);
                            s = fmaf(u.z, v.z, s);
                            s = fmaf(u.w, v.w, s);
                        }
                    } else {
                        for (int c = 0; c < D; ++c) s = fmaf(f1s[c], __ldg(tr + c), s);
                    }
                }
                pat[e] = s * a.scale;
            }
            __syncwarp();
            float *ol = a.out + ((size_t)b * a.levels * K * K + (size_t)l * K * K) * N + q;
            for (int c = lane; c < K * K; c += 32) {
                const int ii = c / K, j = c - ii * K;      // ii -> x offset, j -> y offset (transposed window)
                const float *pp = pat + j * P + ii;
                const float top = pp[0] * gx + pp[1] * fx, bot = pp[P] * gx + pp[P + 1] * fx;
                ol[(size_t)c * N] = top * gy + bot * fy;
            }
            __syncwarp();
        }
        __syncwarp();
    }
}

// [B, D, N] -> [B, N, D] for both feature maps (blockIdx.y = 2 * channel block + map, blockIdx.z = b), 32x32 tiles
// through shared memory
__global__ void corr_alt_transpose_kernel(const float *__restrict__ f1, const float *__restrict__ f2, float *__restrict__ o1,
                                          float *__restrict__ o2, int D, int N) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z;
    const float *src = ((blockIdx.y & 1) ? f2 : f1) + (size_t)b * D * N;
    float *dst = ((blockIdx.y & 1) ? o2 : o1) + (size_t)b * D * N;
    const int n0 = blockIdx.x * 32, d0 = (blockIdx.y >> 1) * 32;
    for (int k = threadIdx.y; k < 32; k += blockDim.y) {
        const int d = d0 + k, n = n0 + threadIdx.x;
        if (d < D && n < N) tile[k][threadIdx.x] = src[(size_t)d * N + n];
    }
    __syncthreads();
    for (int k = threadIdx.y; k < 32; k += blockDim.y) {
        const int n = n0 + k, d = d0 + threadIdx.x;
        if (d < D && n < N) dst[(size_t)n * D + d] = tile[threadIdx.x][k];
    }
}

// level l+1 = avg_pool2d(level l, 2, 2) on [B, h, w, D] maps (odd sizes floored)
__global__ void corr_alt_pool_kernel(const float *__restrict__ in, float *__restrict__ out, int B, int D, int hi, int wi, int ho,
                                     int wo) {
    const size_t total = (size_t)B * ho * wo * D;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int d = (int)(idx % D);
        const size_t pix = idx / D;
        const int x = (int)(pix % wo), y = (int)((pix / wo) % ho), b = (int)(pix / ((size_t)wo * ho));
        const float *p = in + (((size_t)b * hi + 2 * y) * wi + 2 * x) * D + d;
        const size_t row = (size_t)wi * D;
        out[idx] = (p[0] + p[D] + p[row] + p[row + D]) * 0.25f;
    }
}

struct Layout {
    size_t f1, lv[CF_CORR_MAX_LEVELS], total;
};

static Layout layout(int B, int D, int h, int w, int levels) {
    Layout L{};
    size_t off = 0;
    auto region = [&](int hh, int ww) { const size_t o = off; off += align_up((size_t)B * D * hh * ww * sizeof(float), 256); return o; };
    L.f1 = region(h, w);
    for (int l = 0; l < levels; ++l) L.lv[l] = region(h >> l, w >> l);
    L.total = off;
    return L;
}

static int check_args(const char *fn, int B, int D, int h, int w, int levels, int precision) {
    CF_REQUIRE(levels >= 1 && levels <= CF_CORR_MAX_LEVELS, CF_ERR_INVALID_ARG, "%s: levels=%d not in [1,%d]", fn, levels,
               CF_CORR_MAX_LEVELS);
    CF_REQUIRE(B >= 0 && B <= 65535 && D > 0 && D <= 65536 && h > 0 && w > 0, CF_ERR_INVALID_ARG,
               "%s: bad shape B=%d D=%d h=%d w=%d", fn, B, D, h, w);
    CF_REQUIRE((h >> (levels - 1)) >= 1 && (w >> (levels - 1)) >= 1, CF_ERR_INVALID_ARG,
               "%s: %dx%d feature map has no level %d", fn, h, w, levels - 1);
    CF_REQUIRE((int64_t)h * w * D < (1ll << 31), CF_ERR_INVALID_ARG, "%s: feature map too large", fn);
    CF_REQUIRE(precision != CF_CORR_F16 && precision != CF_CORR_3XTF32, CF_ERR_UNSUPPORTED,
               "%s: the on-demand lookup has TF32 (AUTO) and FP32 forms only, not precision %d", fn, precision);
    CF_REQUIRE(precision == CF_CORR_TF32 || precision == CF_CORR_FP32 || precision == CF_CORR_AUTO, CF_ERR_INVALID_ARG,
               "%s: bad precision %d", fn, precision);
    return CF_OK;
}

// box of level l: the narrowest of 16 / 32 / 64 targets that holds a tile's patches with a few pixels of flow variation
static int box_width(int l, int r) {
    const int need = (TX >> l) + 2 * r + 4;
    return need <= 16 ? 16 : (need <= 32 ? 32 : 64);
}

static int encode(CUtensorMap *m, const float *base, int D, int ww, int hh, int B, int box_w, int box_h) {
    TensorMapEncodeTiledFn fn = tensor_map_encoder();
    CF_REQUIRE(fn, CF_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
    const cuuint64_t dims[4] = {(cuuint64_t)D, (cuuint64_t)ww, (cuuint64_t)hh, (cuuint64_t)B};
    const cuuint64_t strides[3] = {(cuuint64_t)D * 4, (cuuint64_t)ww * D * 4, (cuuint64_t)hh * ww * D * 4};
    const cuuint32_t box[4] = {(cuuint32_t)KC, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    const CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_TFLOAT32, 4, const_cast<float *>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CF_REQUIRE(r == CUDA_SUCCESS, CF_ERR_CUDA, "cuTensorMapEncodeTiled (on-demand correlation) failed with CUresult %d", (int)r);
    return CF_OK;
}

}  // namespace alt
}  // namespace cf

extern "C" size_t cf_corr_alt_workspace_bytes(int B, int D, int h, int w, int levels, int precision) {
    using namespace cf;
    if (B <= 0 || alt::check_args("cf_corr_alt_workspace_bytes", B, D, h, w, levels, precision) != CF_OK) return 0;
    return alt::layout(B, D, h, w, levels).total;
}

extern "C" int cf_corr_alt_prepare(const float *fmap1, const float *fmap2, int B, int D, int h, int w, int levels,
                                   int precision, void *state, size_t state_bytes, cf_stream_t stream_) {
    using namespace cf;
    if (int rc = check_device()) return rc;
    if (int rc = alt::check_args("cf_corr_alt_prepare", B, D, h, w, levels, precision)) return rc;
    CF_REQUIRE(fmap1 && fmap2, CF_ERR_NULL, "cf_corr_alt_prepare: null pointer");
    CF_REQUIRE(aligned16(fmap1) && aligned16(fmap2), CF_ERR_ALIGN, "cf_corr_alt_prepare: feature maps must be 16-byte aligned");
    if (B == 0) return CF_OK;
    const alt::Layout L = alt::layout(B, D, h, w, levels);
    CF_REQUIRE(state && state_bytes >= L.total, CF_ERR_WORKSPACE,
               "cf_corr_alt_prepare: state of %zu bytes, %zu needed (cf_corr_alt_workspace_bytes)", state ? state_bytes : (size_t)0,
               L.total);
    CF_REQUIRE(aligned16(state), CF_ERR_ALIGN, "cf_corr_alt_prepare: state must be 16-byte aligned");
    cudaStream_t stream = (cudaStream_t)stream_;
    uint8_t *base = static_cast<uint8_t *>(state);
    const int N = h * w;
    dim3 tgrid((unsigned)ceil_div(N, 32), 2u * (unsigned)ceil_div(D, 32), (unsigned)B);
    alt::corr_alt_transpose_kernel<<<tgrid, dim3(32, 8), 0, stream>>>(fmap1, fmap2, reinterpret_cast<float *>(base + L.f1),
                                                                      reinterpret_cast<float *>(base + L.lv[0]), D, N);
    CF_LAUNCH_CHECK("corr_alt_transpose_kernel");
    for (int l = 1; l < levels; ++l) {
        const size_t total = (size_t)B * (h >> l) * (w >> l) * D;
        const unsigned blocks = (unsigned)std::min<int64_t>(ceil_div((int64_t)total, 256), 16 * (int64_t)sm_count());
        alt::corr_alt_pool_kernel<<<blocks, 256, 0, stream>>>(reinterpret_cast<const float *>(base + L.lv[l - 1]),
                                                              reinterpret_cast<float *>(base + L.lv[l]), B, D, h >> (l - 1),
                                                              w >> (l - 1), h >> l, w >> l);
        CF_LAUNCH_CHECK("corr_alt_pool_kernel");
    }
    return CF_OK;
}

extern "C" int cf_corr_alt_lookup(const void *state, const float *coords, int B, int D, int h, int w, int levels, int radius,
                                  int precision, float *out, cf_stream_t stream_) {
    using namespace cf;
    using namespace cf::alt;
    if (int rc = check_device()) return rc;
    if (int rc = check_args("cf_corr_alt_lookup", B, D, h, w, levels, precision)) return rc;
    CF_REQUIRE(radius >= 0 && radius <= 8, CF_ERR_INVALID_ARG, "cf_corr_alt_lookup: radius=%d not in [0,8]", radius);
    CF_REQUIRE(coords && out, CF_ERR_NULL, "cf_corr_alt_lookup: null pointer");
    CF_REQUIRE(aligned16(coords) && aligned16(out), CF_ERR_ALIGN, "cf_corr_alt_lookup: coords and out must be 16-byte aligned");
    if (B == 0) return CF_OK;
    CF_REQUIRE(state, CF_ERR_WORKSPACE, "cf_corr_alt_lookup: no state (cf_corr_alt_prepare)");
    CF_REQUIRE(aligned16(state), CF_ERR_ALIGN, "cf_corr_alt_lookup: state must be 16-byte aligned");
    cudaStream_t stream = (cudaStream_t)stream_;
    const Layout L = layout(B, D, h, w, levels);
    const uint8_t *base = static_cast<const uint8_t *>(state);
    Args a{};
    a.f1 = reinterpret_cast<const float *>(base + L.f1);
    a.coords = coords;
    a.out = out;
    a.D = D;
    a.h = h;
    a.w = w;
    a.levels = levels;
    a.r = radius;
    for (int l = 0; l < levels; ++l) {
        a.lv[l] = reinterpret_cast<const float *>(base + L.lv[l]);
        a.hl[l] = h >> l;
        a.wl[l] = w >> l;
        a.bw[l] = box_width(l, radius);
        a.bh[l] = BAND_N / a.bw[l];
    }
    a.tiles_x = (int)ceil_div(w, TX);
    a.scale = 1.0f / sqrtf((float)D);
    a.tc = (precision != CF_CORR_FP32 && D % KC == 0) ? 1 : 0;
    const dim3 grid((unsigned)(a.tiles_x * ceil_div(h, TY)), (unsigned)B);

    const size_t simt_smem = (size_t)(SIMT_THREADS / 32) * (D + (2 * radius + 2) * (2 * radius + 2)) * sizeof(float);
    CF_REQUIRE(simt_smem <= 200 * 1024, CF_ERR_INVALID_ARG, "cf_corr_alt_lookup: D=%d too large", D);
    int dev = 0;
    CF_CUDA(cudaGetDevice(&dev));
    static bool opt_in[64] = {};
    if (!opt_in[dev & 63]) {
        CF_CUDA(cudaFuncSetAttribute(corr_alt_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        CF_CUDA(cudaFuncSetAttribute(corr_alt_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
        opt_in[dev & 63] = true;
    }
    // the fp32 kernel first: with the tensor cores in use it serves only the tiles whose boxes do not fit
    corr_alt_simt_kernel<<<grid, SIMT_THREADS, simt_smem, stream>>>(a);
    CF_LAUNCH_CHECK("corr_alt_simt_kernel");
    if (!a.tc) return CF_OK;
    Maps maps;
    if (int rc = encode(&maps.m[0], a.f1, D, w, h, B, TX, TY)) return rc;
    for (int l = 0; l < levels; ++l)
        if (int rc = encode(&maps.m[1 + l], a.lv[l], D, w >> l, h >> l, B, a.bw[l], a.bh[l])) return rc;
    corr_alt_tc_kernel<<<grid, TC_THREADS, TC_SMEM, stream>>>(maps, a);
    CF_LAUNCH_CHECK("corr_alt_tc_kernel");
    return CF_OK;
}
