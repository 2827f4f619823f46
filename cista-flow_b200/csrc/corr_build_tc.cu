// Tensor-core all-pairs correlation for sm_100a:
//   TMA (cp.async.bulk.tensor, 128B swizzle) -> shared memory ring ->
//   tcgen05.mma kind::tf32 (accumulators in TMEM) -> tcgen05.ld epilogue with
//   fused 1/sqrt(D) scale and fused level-1 (2x2) average pooling.
//
// Replaces the torch.matmul + first avg_pool2d of CorrBlock.__init__
// (ERAFT/corr.py:19-27,52-60; DCEIFlow/core/corr/raft_corr.py:22-30,56-65).
//
// GEMM view, per batch item b:   C[i, j] = sum_k A[k, i] * Bm[k, j]
//   A = fmap1[b] (D x N), Bm = fmap2[b] (D x N), N = h*w contiguous: BOTH
//   operands are "MN-major" (the reference's fmap1.transpose(1,2) is free).
//   The tiles are loaded as TMA boxes of 32 (MN, 128 bytes) x 32 (K rows) with
//   CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, which lands them in the only shared
//   memory layout tcgen05 accepts for MN-major 32-bit operands: UMMA layout type
//   1, "128B swizzle with 32-byte atoms" (Swizzle<2,5,2>: the 32-byte chunk index
//   of a 128-byte row is XORed with row % 4).  Canonical form, in 16-byte units:
//   ((8,n),(4,k)) : ((1,LBO),(8,SBO)) -- LBO = 4096 B between 32-column atoms
//   (one TMA box each), SBO = 512 B between groups of 4 K rows.  One tcgen05.mma
//   kind::tf32 has K = 8 = two 4-row groups, so the descriptor start address
//   advances by 1024 B per MMA.  (The plain SWIZZLE_128B layout is silently
//   computed as zeros for MN-major tf32; scripts/tc_probe.cu is the single-tile
//   probe that established this on a B200.)
//
// Tile: 128 queries (M, TMEM lanes) x BN targets (TMEM columns).  With pooling
// fused, BN = R*w covers R (even) whole rows of the target map so that each 2x2
// pooling window lives inside one accumulator row; the epilogue thread that owns
// query i reads row y and row y+1 of its TMEM lane, stores both level-0 rows and
// the pooled level-1 row.  Level 0 (N^2 floats) is therefore written once and
// never re-read: the volume is HBM-write bound (96 FLOP/B, SURVEY.md H2).
//
// Persistent, warp-specialised CTA (1 per SM, 192 threads):
//   warps 0-3  epilogue (TMEM lane quarter = warp id): TMEM -> registers -> swizzled smem -> TMA store
//   warp  4    TMA producer (one elected lane)
//   warp  5    TMEM allocator + MMA issuer (one elected lane)
// Two TMEM accumulator stages (2 x 256 columns) let the MMA of tile t+1 overlap
// the epilogue of tile t; a 4-stage shared-memory ring feeds the MMA.
//
// Operand precision: tcgen05 kind::tf32 reads fp32 words and ignores the low 13
// mantissa bits (truncation), which biases every product low (measured: signed
// relative bias -7e-4, max|err| 7.7e-4*max|ref| at D=256).  Encoding the tensor
// maps with CU_TENSOR_MAP_DATA_TYPE_TFLOAT32 makes the TMA unit round the
// operands to TF32 (nearest) on their way into shared memory -- measured
// identical to a cvt.rna.tf32.f32 pre-pass: bias -5e-7, max|err| 2.8e-4*max|ref|
// -- so no extra pass over the feature maps and no workspace are needed.
//
// State at the end of round 2 (the notes below and at launch_tc() are the history that led here): on wide maps the default
// is kind::f16 on fp16 operand copies, two 128-K-row stages per tile (fmap1 slice: one 128B-swizzled 3-D box; fmap2 slice:
// one 64B-swizzled 3-D box of exactly BN columns), eight epilogue warps, levels 1 and 2 pooled in the epilogue.  At 64 x
// 60x80 the GEMM kernel runs 3.4 us per 128x160 tile = 1.65 ms (ncu) and writes at 4.7-5.0 TB/s.  Its period is the SM's
// TMA unit: four operand boxes (~0.32 us each) + twenty 4 KB store boxes (~0.12 us each) per tile queue in ONE unit
// (scripts/experiments/write_probe.cu); the epilogue warps are busy ~3.0 us of it, the MMAs ~1.5 us.
#include <cuda.h>
#include <cuda_fp16.h>

#include <type_traits>

#include "tcgen05.cuh"

namespace cf {

namespace tc {

constexpr int BK = 32;           // K rows per pipeline stage (4 MMAs of K=8)
// fp16 operands: 64 K rows per stage.  One SM's TMA unit retires a 3-D box instruction of these shapes about every
// 320 ns WHATEVER its size between 20 and 40 KB (profiles/r02/tma_probe.txt: {64 cols, 32 rows, 5 atoms} and
// {64, 64, 5} both 320 ns), and a stage is two instructions (fmap1 box + fmap2 box): with 32-row stages the fp16
// kernel spent 8 x 2 x 320 ns = 5.1 us per tile on operand loads alone -- exactly what it measured, and why halving
// the operand bytes had bought nothing in round 1.  64-row stages: 3.0 us of loads per tile (ablation: loads only), 305 us at
// 8 x 60x80; 128-row stages (two per tile, 80 KB each, ring of two): loads + MMAs 2.45 us per tile, 290 us.
constexpr int BK_F16 = 128;
constexpr int BK_TF32 = 32;      // TF32 stages.  64-row stages (ring of two) measured the same within 2 % at every shape (64 x 60x80 2595
                                 // against 2580 us): the TF32 kernel is bound by its MMAs (3.0 us per 128x160 tile), not by TMA issue
constexpr int MAX_STAGES = 8;     // ring depth = as many stages of (fmap1 tile + this shape's fmap2 tile) as fit, at most 6
constexpr int MAX_BN = 256;      // UMMA N limit
constexpr int BOX_BYTES = 32 * 32 * 4;                 // one TMA box: 32 cols x 32 rows fp32
constexpr int A_BYTES = (BM / 32) * BOX_BYTES;         // 16 KB
constexpr int EPI_BUF_BYTES = 32 * 32 * 4;               // one 32x32 fp32 output box, 128B swizzle
// Epilogue warps per TMEM lane quarter.  2 (eight epilogue warps splitting the tile's work items) was measured
// SLOWER on the B200 (8 x 60x80: 362 against 334 us; with loads and stores ablated 258 against 238 us): the
// epilogue is not the critical path, the tf32 MMAs are (operand fetch from shared memory, see DESIGN.md).
// (the kernel's template parameter ES; the TF32 kernel uses 1.  With fp16 operands the stages are half the size, the
//  64 KB of epilogue buffers fit beside a deep ring, and the epilogue IS the critical path: one tile's epilogue takes
//  3.7 us on four warps while the MMAs of a 128x160 tile need 1.5 us -- see the kernel's header.)
constexpr int SMEM_LIMIT = 227 * 1024;
__host__ __device__ constexpr int epi_bytes(int es) { return 4 * es * 2 /*double buffer*/ * EPI_BUF_BYTES; }   // 32 KB per ES
__host__ __device__ constexpr int smem_fixed(int es) { return epi_bytes(es) + 1024 /*align slack*/ + 256 /*barriers*/; }
__host__ __device__ constexpr int threads(int es) { return 32 * (4 * es + 2); }

struct Params {
    int B, D, N, h, w;
    int BN;        // valid target columns per tile
    int BN_mma;    // UMMA N (BN rounded up to 16)
    int n_boxes_b; // TMA boxes per stage for the B operand
    int R;         // target rows per tile when pooling is fused (0 = not fused)
    int tiles_m, tiles_n, total_tiles;
    int tiles_nv;  // target tiles per query block in the tile index (= tiles_n, rounded up to 4 with quad3: indices with
                   // nb >= tiles_n are skipped by every role)
    int quad3;     // 1 (with pair2): a CTA takes the tiles of FOUR consecutive target-row pairs back to back and the epilogue pools
                   // level 3 from two level-2 rows (the first one parked in free TMEM columns, like pair2's level-1 row)
    int tiles_mp;  // pair kernel: pairs of query tiles per batch item (= ceil(tiles_m / 2)); total_tiles counts pairs
    int stages;      // shared-memory ring depth
    int stage_bytes; // A_BYTES + n_boxes_b * BOX_BYTES
    int qbox_h0;     // qbox: level-0 chunks of the first warp of a lane quarter
    int frag_stores; // 1: level 0 leaves straight from registers in the tcgen05.ld.16x256b fragment layout (32-byte runs, no shared
                     // memory, no TMA store) -- see launch_tc()
    int qbox;        // 1 (two epilogue warps per lane quarter): level 0 leaves as ONE {32 cols, 32 rows, BN/32 atoms} box per lane
                     // quarter and tile (tmap_c is then that 3-D map over {32, B*N rows, N/32 atoms}) -- see launch_tc()
    int epi_bytes;   // bytes of epilogue buffers between the operand ring and the barriers
    int l1_scratch;  // byte offset (from the epilogue buffers) of a level-1 scratch area of 2 KB per epilogue warp that is NOT a
                     // level-0 box buffer (0: none, the strips borrow a box buffer and wait for its store)
    int b_sw64;      // fp16 operands, BN_mma an odd multiple of 32: the fmap2 slice as {32 cols, K rows, BN_mma / 32 atoms} with the
                     // 64-byte swizzle -- exactly BN_mma columns per stage instead of the next multiple of 64 (160: 40 KB, not 48)
    int ablate;    // experiments (CF_TC_FLAGS bits 8-10): 1 = no level-0/1 stores, 2 = no MMAs, 4 = no operand loads, 16 = no epilogue at all, 32 = no pooling part, 64 = no level-0 part
    int b_half;    // pair kernel: fmap2 boxes per stage and CTA (half of the tile's columns each)
    int h1, w1;    // level-1 map size
    float scale;
    int stream_l0; // 1: level 0 is larger than L2 can hold -> evict-first stores
    int b3d;       // as atoms3d, for the B operand: also needs tile origins on atom boundaries (BN % 32 == 0)
    int atoms3d;   // 1: N % 32 == 0 -> the tensor maps are 3-D {32 cols, rows, 32-column atoms}: ONE TMA instruction
                   //    per operand and stage.  One thread issues a cp.async.bulk.tensor about every 100 cycles, and
                   //    9-12 per-atom boxes per stage made that issue rate the bound of the main loop (timeline)
    float *l0;
    float *l1;
    int l1_staged;           // 1: level-1 rows are transposed through shared memory into 64-byte runs (w1 % 4 == 0)
    int lsu_stores;          // 1: level-0 rows leave through the LSU (transposed in shared memory), 0: TMA bulk stores
    const float *inv_scale;  // F16 operands: [2*B] powers of two that undo the per-item operand scaling (else nullptr)
    // deep fusion (tiles of 8k whole target rows, i.e. feature maps up to 32 wide -- the 180x240 / DAVIS240 case):
    // levels 2 and 3 are pooled from the level-1 rows while they are still in registers
    int pair2;     // 1: a CTA takes tiles in PAIRS of consecutive target-row pairs (nb, nb+1) and the epilogue pools level 2 from
                   //    the two level-1 rows (the first one parked in free TMEM columns) -- maps too wide for `deep`, R == 2
    int deep;      // 0: none, 1: level 2, 2: levels 2 and 3
    int h2, w2, h3, w3;
    float *l2;
    float *l3;
};

// Debug timeline of CTA 0's first tile (clock64 stamps), read back with cf_debug_tc_timeline().
__device__ unsigned long long g_tc_timeline[32];
__device__ __forceinline__ void stamp(int slot) {
    if (blockIdx.x == 0) g_tc_timeline[slot] = (unsigned long long)clock64();
}

// experiment builds (-DCF_TRACE, scripts/corr_trace.py): per-CTA, per-tile globaltimer stamps, 16 slots per tile:
//  0 first load issued, 1 last load issued | 2 accumulator free (MMA), 3..10 stage kb landed, 11 last commit |
//  12 accumulator ready (epilogue), 13 level-0 chunks issued, 14 epilogue done
#ifdef CF_TRACE
#define TC_TRACE(tile_no, slot) do { if ((tile_no) < 15) CF_TRACE_AT(16 + 16 * (tile_no) + (slot)); } while (0)
#else
#define TC_TRACE(tile_no, slot) ((void)0)
#endif

__device__ __forceinline__ void decode_tile(const Params &p, int tile, int &b, int &mb, int &nb) {
    nb = tile % p.tiles_nv;
    const int t = tile / p.tiles_nv;
    mb = t % p.tiles_m;
    b = t / p.tiles_m;
}
// pair kernel: `tile` indexes a pair of vertically adjacent query tiles; CTA `rank` owns query tile 2*pair + rank,
// which may lie entirely below the volume when tiles_m is odd (its loads are zero-filled, its stores clipped)
__device__ __forceinline__ void decode_pair_tile(const Params &p, int tile, int rank, int &b, int &mb, int &nb) {
    nb = tile % p.tiles_n;
    const int t = tile / p.tiles_n;
    mb = 2 * (t % p.tiles_mp) + rank;
    b = t / p.tiles_mp;
}

template <bool STREAM>
__device__ __forceinline__ void store_row_chunk_impl(float *dst, const uint32_t (&v)[32], float scale, int nvalid, bool vec4) {
    // nvalid in [0,32], multiple of 4 when vec4
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        if (vec4) {
            if (4 * q < nvalid) {
                const float4 o = make_float4(__uint_as_float(v[4 * q]) * scale, __uint_as_float(v[4 * q + 1]) * scale,
                                             __uint_as_float(v[4 * q + 2]) * scale, __uint_as_float(v[4 * q + 3]) * scale);
                if (STREAM) __stcs(reinterpret_cast<float4 *>(dst) + q, o);
                else *(reinterpret_cast<float4 *>(dst) + q) = o;
            }
        } else {
#pragma unroll
            for (int r = 0; r < 4; ++r)
                if (4 * q + r < nvalid) {
                    const float o = __uint_as_float(v[4 * q + r]) * scale;
                    if (STREAM) __stcs(dst + 4 * q + r, o);
                    else dst[4 * q + r] = o;
                }
        }
    }
}
__device__ __forceinline__ void store_row_chunk(float *dst, const uint32_t (&v)[32], float scale, int nvalid, bool vec4, bool stream) {
    if (stream) store_row_chunk_impl<true>(dst, v, scale, nvalid, vec4);
    else store_row_chunk_impl<false>(dst, v, scale, nvalid, vec4);
}

// ---- fp16 pyramid (cf_corr_build_half) ----
// RN_f16 of an fp32 value, widened back (exact): what a pooled level is summed from
__device__ __forceinline__ float round_half(float x) { return __half2float(__float2half_rn(x)); }
template <bool HALF>
__device__ __forceinline__ float stored(float x) {   // a pooled value as the pyramid stores it
    if constexpr (HALF) return round_half(x);
    else return x;
}
__device__ __forceinline__ uint32_t pack_half2(float lo, float hi) {
    const __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<const uint32_t *>(&h);
}
// widest store (8, 4, 2 or 1 halves) that keeps every run of a level aligned: the base pointer, the per-query map (`map`
// halves) and the row start (`row` halves) all fall on its boundary
__device__ __forceinline__ int half_vec(const void *base, int map, int row) {
    int v = 8;
    while (v > 1 && (((reinterpret_cast<uintptr_t>(base) & (uintptr_t)(2 * v - 1)) != 0) || map % v != 0 || row % v != 0)) v >>= 1;
    return v;
}
// the first nvalid of M values (already fp16-representable) as halves at dst, `vec` halves per store; nvalid is a
// multiple of vec or the end of the run
template <int M>
__device__ __forceinline__ void store_halves(__half *dst, const float (&o)[M], int nvalid, int vec, bool stream) {
    if (M >= 8 && vec == 8) {
#pragma unroll
        for (int q = 0; q < M / 8; ++q)
            if (8 * q < nvalid) {
                const uint4 u = make_uint4(pack_half2(o[8 * q], o[8 * q + 1]), pack_half2(o[8 * q + 2], o[8 * q + 3]),
                                           pack_half2(o[8 * q + 4], o[8 * q + 5]), pack_half2(o[8 * q + 6], o[8 * q + 7]));
                if (stream) __stcs(reinterpret_cast<uint4 *>(dst) + q, u);
                else *(reinterpret_cast<uint4 *>(dst) + q) = u;
            }
    } else if (M >= 4 && vec == 4) {
#pragma unroll
        for (int q = 0; q < M / 4; ++q)
            if (4 * q < nvalid)
                *(reinterpret_cast<uint2 *>(dst) + q) = make_uint2(pack_half2(o[4 * q], o[4 * q + 1]), pack_half2(o[4 * q + 2], o[4 * q + 3]));
    } else if (vec == 2) {
#pragma unroll
        for (int q = 0; q < M / 2; ++q)
            if (2 * q < nvalid) *(reinterpret_cast<uint32_t *>(dst) + q) = pack_half2(o[2 * q], o[2 * q + 1]);
    } else {
#pragma unroll
        for (int q = 0; q < M; ++q)
            if (q < nvalid) dst[q] = __float2half_rn(o[q]);
    }
}

// CL = 1: one CTA per tile.  CL = 2 (tcgen05 cta_group::2): a cluster of two CTAs owns two vertically adjacent
// query tiles of the same target tile = one 256 x BN UMMA.  Each CTA loads its own 128 fmap1 rows and HALF of the
// fmap2 columns; the leader (rank 0) issues the MMAs for the pair, each CTA's accumulator rows land in its own TMEM
// and are drained by its own epilogue.  Per SM and K step this moves and reads (128 + BN/2) x 32 B instead of
// (128 + BN) x 32 B: the single-CTA tf32 MMA is bound by operand fetch from shared memory (measured: ~50 B/clk,
// i.e. 181 cycles for 128x160x8 and 243 for 128x256x8 with loads and stores ablated; K-major descriptors on the
// same bytes change nothing).  Barriers: both producers' bytes complete on the LEADER's `full`; the leader's
// commits arrive on `empty` / `tfull` of both CTAs; both epilogues arrive on the leader's `tempty`.
// (A first pair variant only multicast the fmap2 tile to two independent cta_group::1 MMAs: L2 traffic -33 %,
//  time unchanged -- L2 bandwidth was not the bound.)
// OM_F16: the operands are fp16 copies of the feature maps (same 11-bit significand as TF32, scaled per batch item by a
// power of two so that any finite input fits; made by fmap_to_half_kernel).  kind::f16 covers K = 16 per MMA where
// kind::tf32 covers 8 at the same ~1 accumulator column per clock, and every stage moves half the bytes: the GEMM
// stops being MMA / load-latency bound and runs at the HBM write rate of the volume.
// OM_3XTF32: each operand is split x = hi + lo into two exact TF32 values (fmap_split_tf32_kernel, workspace) and every
// K = 8 step issues lo.hi + hi.lo + hi.hi into the same accumulator: within ~2^-22 of the exact products, fp32-level
// accuracy at three times the MMA work.  A stage holds both slices of every 32-column atom side by side
// ([atom][hi, lo][K rows][32 cols], one 4-D TMA box per operand), so the UMMA descriptors see LBO = two boxes and
// address the lo slice one box behind the hi slice.  Only the producer and the MMA issuer differ; the epilogue is the TF32 one.
enum OperandMode { OM_TF32 = 0, OM_F16 = 1, OM_3XTF32 = 2 };
#define CF_TC_KERNEL corr_tc_kernel
#define CF_TC_OUT float
#include "corr_tc_kernel.cuh"
#undef CF_TC_KERNEL
#undef CF_TC_OUT
#define CF_TC_KERNEL corr_tc_half_kernel
#define CF_TC_OUT __half
#include "corr_tc_kernel.cuh"
#undef CF_TC_KERNEL
#undef CF_TC_OUT

// ---- measured and dropped: A-resident variant --------------------------------------------------
// Round 1 also built a variant that keeps the 128 x D slice of fmap1 resident in shared memory (128 KB)
// for a whole range of target tiles, streaming only fmap2 (operand traffic per 128x160 tile 160 KB
// instead of 288 KB).  It was SLOWER (8 x 60x80: 426 us against 327 us; 1 x 80x124: 248 against 198):
// with 128 KB pinned only ~64 KB are left for the fmap2 ring, and at ~1.6 us of loaded TMA latency
// 60 KB in flight sustain ~37 KB/us per SM -- the streaming kernel keeps 144 KB in flight.  The per-tile
// timeline (scripts/corr_trace.py at that commit) showed the main loop waiting on loads, the epilogue
// (3.4-3.9 us per tile) hidden behind it.  What did help both variants: ONE 3-D TMA instruction per
// operand and stage (atoms3d / b3d above) instead of 9-12 per-atom boxes -- a single thread issues a
// cp.async.bulk.tensor only about every 100 cycles, which was the main-loop bound (368 -> 327 us).
// Next lever (not done): cta_group::2 pairs (M = 256 across two SMs, each loading half of the fmap2 tile).

CF_DEFINE_TRACE_SETTER(cf_trace_buffer_corr)

// ---- fp16 operand copies ---------------------------------------------------------------------------------
// amax[t * B + b] = max |x| over batch item b of feature map t (t = 0, 1), as the bit pattern of a non-negative float
// (integer max == float max); zeroed by the host side before the launch.
__global__ void __launch_bounds__(256)
fmap_absmax_kernel(const float *__restrict__ f1, const float *__restrict__ f2, int64_t per_item, int B, int b0, int nbc,
                   unsigned *__restrict__ amax) {
    // this launch covers batch items [b0, b0 + nbc) of both maps: blockIdx.y = t * nbc + (b - b0)
    const int t = (int)blockIdx.y / nbc, b = b0 + (int)blockIdx.y % nbc;
    const int item = t * B + b;
    const float *src = (t == 0 ? f1 : f2) + (int64_t)b * per_item;
    float m = 0.f;
    const int64_t n4 = per_item >> 2;
    const float4 *s4 = reinterpret_cast<const float4 *>(src);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 v = __ldg(s4 + i);
        m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
    }
    m = warp_max(m);
    __shared__ float sh[8];
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < 8; ++k) m = fmaxf(m, sh[k]);
        if (m > 0.f) atomicMax(amax + item, __float_as_uint(fminf(m, 3.0e38f)));
    }
}
// x -> fp16(x * 2^shift), shift chosen per batch item so that the largest magnitude lands in [2^13, 2^14): every finite
// input fits fp16 (round to nearest: the same 11-bit significand a TF32 operand keeps), the scaling is exact, and
// inv_scale[item] = 2^-shift lets the GEMM epilogue undo it.  per_item % 4 == 0.
__global__ void __launch_bounds__(256)
fmap_to_half_kernel(const float *__restrict__ f1, const float *__restrict__ f2, int64_t per_item, int B, int b0, int nbc,
                    const unsigned *__restrict__ amax, __half *__restrict__ h1, __half *__restrict__ h2,
                    float *__restrict__ inv_scale) {
    const int t = (int)blockIdx.y / nbc, b = b0 + (int)blockIdx.y % nbc;
    const int item = t * B + b;
    const bool first = t == 0;
    const int64_t base = (int64_t)b * per_item;
    const float *src = (first ? f1 : f2) + base;
    __half *dst = (first ? h1 : h2) + base;
    const float mx = __uint_as_float(__ldg(amax + item));
    const int shift = mx > 0.f ? 13 - ilogbf(mx) : 0;
    const float up = ldexpf(1.f, shift > 126 ? 126 : shift);      // (a tiny maximum: clamp the exponent, still exact)
    if (blockIdx.x == 0 && threadIdx.x == 0) inv_scale[item] = 1.f / up;
    const int64_t n4 = per_item >> 2;
    const float4 *s4 = reinterpret_cast<const float4 *>(src);
    uint2 *d4 = reinterpret_cast<uint2 *>(dst);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 v = __ldg(s4 + i);
        const __half2 lo = __floats2half2_rn(v.x * up, v.y * up), hi = __floats2half2_rn(v.z * up, v.w * up);
        uint2 o;
        o.x = *reinterpret_cast<const unsigned *>(&lo);
        o.y = *reinterpret_cast<const unsigned *>(&hi);
        d4[i] = o;
    }
}

// One pass instead of two (round 2): a CTA keeps its 32 KB slice of a feature map in REGISTERS (8 float4 per thread),
// publishes the slice's maximum (atomicMax on the item's slot + an arrival counter), waits until all slices of the item have
// arrived, then scales and narrows out of registers -- the fp32 maps cross the HBM interface once.  The two-kernel form
// (maximum pass, then conversion pass, chunked so that the second read hit the L2) measured 342 us for 64 x 2 maps of 256 x
// 60x80 under ncu -- 15 % of the whole pyramid build.  Units are ordered by item and there are no more slices per item
// than CTAs, so a CTA never waits for a slice that is queued behind its own (all CTAs of the launch fit on the chip at once).
constexpr int CV_THREADS = 256, CV_F4 = 8;
// (round 2, later: the loads of a CTA's NEXT slice are issued before it waits for the current item's arrival counter --
//  without that all resident CTAs loaded, waited and stored in lockstep waves, reads and writes taking turns on the bus)
__global__ void __launch_bounds__(CV_THREADS, 3)
fmap_to_half_fused_kernel(const float *__restrict__ f1, const float *__restrict__ f2, int64_t per_item, int B, int parts,
                          unsigned *amax, int *arrived, __half *__restrict__ h1, __half *__restrict__ h2,
                          float *__restrict__ inv_scale) {
    __shared__ float s_red[2][CV_THREADS / 32];
    __shared__ float s_up[2];
    const int64_t units = (int64_t)2 * B * parts, n4 = per_item >> 2;
    struct Unit {
        const float4 *s4;
        uint2 *d4;
        int64_t i0;
        int item, part;
    };
    auto unit_of = [&](int64_t u) {
        Unit t;
        t.item = (int)(u / parts);
        t.part = (int)(u - (int64_t)t.item * parts);
        const bool first = t.item < B;
        const int64_t base = (int64_t)(first ? t.item : t.item - B) * per_item;
        t.s4 = reinterpret_cast<const float4 *>((first ? f1 : f2) + base);
        t.d4 = reinterpret_cast<uint2 *>((first ? h1 : h2) + base);
        t.i0 = (int64_t)t.part * (CV_THREADS * CV_F4) + threadIdx.x;
        return t;
    };
    auto load = [&](const Unit &t, float4 (&v)[CV_F4]) {
#pragma unroll
        for (int k = 0; k < CV_F4; ++k) {
            const int64_t i = t.i0 + (int64_t)k * CV_THREADS;
            v[k] = i < n4 ? __ldg(t.s4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    // the slice's maximum -> the item's slot, arrival counted (thread 0 of the CTA); `slot` alternates between units
    auto publish = [&](const Unit &t, const float4 (&v)[CV_F4], int slot) {
        float m = 0.f;
#pragma unroll
        for (int k = 0; k < CV_F4; ++k)
            m = fmaxf(fmaxf(m, fmaxf(fabsf(v[k].x), fabsf(v[k].y))), fmaxf(fabsf(v[k].z), fabsf(v[k].w)));
        m = warp_max(m);
        if ((threadIdx.x & 31) == 0) s_red[slot][threadIdx.x >> 5] = m;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int k = 1; k < CV_THREADS / 32; ++k) m = fmaxf(m, s_red[slot][k]);
            if (m > 0.f) atomicMax(amax + t.item, __float_as_uint(fminf(m, 3.0e38f)));
            __threadfence();
            atomicAdd(arrived + t.item, 1);
        }
    };
    // wait until every slice of the item has arrived, then scale and narrow out of registers
    auto finish = [&](const Unit &t, const float4 (&v)[CV_F4], int slot) {
        if (threadIdx.x == 0) {
            unsigned spins = 0;
            while (*reinterpret_cast<volatile int *>(arrived + t.item) < parts) {
                __nanosleep(64);
                if (++spins > (1u << 24)) __trap();
            }
            __threadfence();
            const float mx = __uint_as_float(*reinterpret_cast<volatile unsigned *>(amax + t.item));
            const int shift = mx > 0.f ? 13 - ilogbf(mx) : 0;
            const float up = ldexpf(1.f, shift > 126 ? 126 : shift);      // (a tiny maximum: clamp the exponent, still exact)
            s_up[slot] = up;
            if (t.part == 0) inv_scale[t.item] = 1.f / up;
        }
        __syncthreads();
        const float up = s_up[slot];
#pragma unroll
        for (int k = 0; k < CV_F4; ++k) {
            const int64_t i = t.i0 + (int64_t)k * CV_THREADS;
            if (i < n4) {
                const __half2 lo = __floats2half2_rn(v[k].x * up, v[k].y * up), hi = __floats2half2_rn(v[k].z * up, v[k].w * up);
                uint2 o;
                o.x = *reinterpret_cast<const unsigned *>(&lo);
                o.y = *reinterpret_cast<const unsigned *>(&hi);
                t.d4[i] = o;
            }
        }
    };
    // two register sets in turn: publish(cur) -> load(next) -> finish(cur)
    float4 va[CV_F4], vb[CV_F4];
    int64_t u = blockIdx.x;
    if (u >= units) return;
    Unit ta = unit_of(u), tb = ta;
    load(ta, va);
    for (;;) {
        publish(ta, va, 0);
        const bool more_b = u + gridDim.x < units;
        if (more_b) { tb = unit_of(u + gridDim.x); load(tb, vb); }
        finish(ta, va, 0);
        if (!more_b) break;
        u += gridDim.x;
        publish(tb, vb, 1);
        const bool more_a = u + gridDim.x < units;
        if (more_a) { ta = unit_of(u + gridDim.x); load(ta, va); }
        finish(tb, vb, 1);
        if (!more_a) break;
        u += gridDim.x;
    }
}

// ---- 3xTF32 operand split ----------------------------------------------------------------------------------
// hi = rn_tf32(x) and lo = rn_tf32(x - hi) for both feature maps (x - hi is exact in fp32).  Both are TF32 values exactly,
// so the tensor maps read them as plain FLOAT32 and the result does not depend on how the TMA or the MMA treats the low
// 13 mantissa bits.  No scaling: the fp32 range is kept.  n4 = float4 per map.
__device__ __forceinline__ float rna_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r & 0xFFFFE000u);
}
__device__ __forceinline__ void split_tf32(float x, float &hi, float &lo) {
    hi = rna_tf32(x);
    lo = rna_tf32(x - hi);
}
__global__ void __launch_bounds__(256)
fmap_split_tf32_kernel(const float4 *__restrict__ f1, const float4 *__restrict__ f2, int64_t n4, float4 *__restrict__ hi1,
                       float4 *__restrict__ lo1, float4 *__restrict__ hi2, float4 *__restrict__ lo2) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < 2 * n4; i += stride) {
        const bool first = i < n4;
        const int64_t j = first ? i : i - n4;
        const float4 v = __ldg((first ? f1 : f2) + j);
        float4 h, l;
        split_tf32(v.x, h.x, l.x);
        split_tf32(v.y, h.y, l.y);
        split_tf32(v.z, h.z, l.z);
        split_tf32(v.w, h.w, l.w);
        (first ? hi1 : hi2)[j] = h;
        (first ? lo1 : lo2)[j] = l;
    }
}

// ---- host side --------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// 2-D map over a feature map viewed as [B*D rows, N cols], box 32 x 32, 128B swizzle / 32B atoms
// (fp16 operand copies: 2-byte elements, boxes of 64 columns, plain 128B swizzle)
static int make_fmap_tmap(CUtensorMap *m, const void *base, int B, int D, int N, CUtensorMapDataType dt, int box_rows = 32) {
    EncodeTiledFn fn = encode_fn();
    CF_REQUIRE(fn, CF_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
    const bool half = dt == CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    const size_t elt = half ? 2 : 4;
    cuuint64_t dims[2] = {(cuuint64_t)N, (cuuint64_t)B * D};
    cuuint64_t strides[1] = {(cuuint64_t)N * elt};
    cuuint32_t box[2] = {(cuuint32_t)(128 / elt), (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(m, dt, 2, const_cast<void *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    half ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CF_REQUIRE(r == CUDA_SUCCESS, CF_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return CF_OK;
}

// The same feature map as a 3-D tensor {32 cols, B*D rows, N/32 column atoms} (N % 32 == 0): a box
// {32, rows, atoms} lands in shared memory as [atom][row][32 cols] -- the UMMA MN-major layout -- in ONE instruction
static int make_fmap_tmap3(CUtensorMap *m, const void *base, int B, int D, int N, CUtensorMapDataType dt, int box_rows,
                           int box_atoms) {
    EncodeTiledFn fn = encode_fn();
    CF_REQUIRE(fn, CF_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
    const bool half = dt == CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    const size_t elt = half ? 2 : 4;
    const cuuint32_t bc = (cuuint32_t)(128 / elt);
    cuuint64_t dims[3] = {bc, (cuuint64_t)B * D, (cuuint64_t)N / bc};
    cuuint64_t strides[2] = {(cuuint64_t)N * elt, 128};
    cuuint32_t box[3] = {bc, (cuuint32_t)box_rows, (cuuint32_t)box_atoms};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(m, dt, 3, const_cast<void *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    half ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CF_REQUIRE(r == CUDA_SUCCESS, CF_ERR_CUDA, "cuTensorMapEncodeTiled (3-D feature map) failed with CUresult %d", (int)r);
    return CF_OK;
}

// the level-0 volume as {32 cols, B*N rows, N/32 column atoms} (N % 32 == 0): a box {32, 32, atoms} stores `atoms` swizzled
// 32 x 32 images that lie side by side in shared memory with ONE instruction
static int make_volume_tmap_atoms(CUtensorMap *m, float *base, int B, int N, int atoms) {
    EncodeTiledFn fn = encode_fn();
    CF_REQUIRE(fn, CF_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
    cuuint64_t dims[3] = {32, (cuuint64_t)B * N, (cuuint64_t)N / 32};
    cuuint64_t strides[2] = {(cuuint64_t)N * sizeof(float), 128};
    cuuint32_t box[3] = {32, 32, (cuuint32_t)atoms};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CF_REQUIRE(r == CUDA_SUCCESS, CF_ERR_CUDA, "cuTensorMapEncodeTiled (volume, atoms) failed with CUresult %d", (int)r);
    return CF_OK;
}

// fp16 feature map as {32 cols, B*D rows, N/32 atoms of 64 bytes}, 64-byte swizzle (N % 32 == 0)
static int make_fmap_tmap3_sw64(CUtensorMap *m, const void *base, int B, int D, int N, int box_rows, int box_atoms) {
    EncodeTiledFn fn = encode_fn();
    CF_REQUIRE(fn, CF_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
    cuuint64_t dims[3] = {32, (cuuint64_t)B * D, (cuuint64_t)N / 32};
    cuuint64_t strides[2] = {(cuuint64_t)N * 2, 64};
    cuuint32_t box[3] = {32, (cuuint32_t)box_rows, (cuuint32_t)box_atoms};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void *>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CF_REQUIRE(r == CUDA_SUCCESS, CF_ERR_CUDA, "cuTensorMapEncodeTiled (64B-swizzled feature map) failed with CUresult %d", (int)r);
    return CF_OK;
}

// 3xTF32 operands: the hi copy of a feature map and its lo copy `lo_off` bytes behind it as ONE tensor whose third
// dimension selects the slice.  box_atoms > 0 (N % 32 == 0): {32 cols, B*D rows, 2 slices, N/32 atoms}, a box {32, rows, 2,
// box_atoms} lands as [atom][hi, lo][row][32 cols]; box_atoms == 0: {N cols, B*D rows, 2 slices}, one box {32, rows, 2} per atom
static int make_split_tmap(CUtensorMap *m, const float *hi, size_t lo_off, int B, int D, int N, int box_rows, int box_atoms) {
    EncodeTiledFn fn = encode_fn();
    CF_REQUIRE(fn, CF_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
    const bool atoms = box_atoms > 0;
    const cuuint32_t rank = atoms ? 4 : 3;
    cuuint64_t dims[4] = {atoms ? 32u : (cuuint64_t)N, (cuuint64_t)B * D, 2, (cuuint64_t)N / 32};
    cuuint64_t strides[3] = {(cuuint64_t)N * sizeof(float), (cuuint64_t)lo_off, 128};
    cuuint32_t box[4] = {32, (cuuint32_t)box_rows, 2, (cuuint32_t)box_atoms};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, rank, const_cast<float *>(hi), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CF_REQUIRE(r == CUDA_SUCCESS, CF_ERR_CUDA, "cuTensorMapEncodeTiled (split feature map) failed with CUresult %d", (int)r);
    return CF_OK;
}

// 3-D map over the level-0 volume [B][N][N], box {32 cols, 32 rows, 1}, 128B swizzle (store side)
static int make_volume_tmap(CUtensorMap *m, float *base, int B, int N) {
    EncodeTiledFn fn = encode_fn();
    CF_REQUIRE(fn, CF_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
    cuuint64_t dims[3] = {(cuuint64_t)N, (cuuint64_t)N, (cuuint64_t)B};
    cuuint64_t strides[2] = {(cuuint64_t)N * sizeof(float), (cuuint64_t)N * N * sizeof(float)};
    cuuint32_t box[3] = {32, 32, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CF_REQUIRE(r == CUDA_SUCCESS, CF_ERR_CUDA, "cuTensorMapEncodeTiled (volume) failed with CUresult %d", (int)r);
    return CF_OK;
}

// the fp16 level-0 volume [B][N][N] (N % 8 == 0: 16-byte row pitch), box {64 cols, 32 rows, 1}: 128-byte rows, 128B swizzle
static int make_volume_tmap_half(CUtensorMap *m, void *base, int B, int N) {
    EncodeTiledFn fn = encode_fn();
    CF_REQUIRE(fn, CF_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
    cuuint64_t dims[3] = {(cuuint64_t)N, (cuuint64_t)N, (cuuint64_t)B};
    cuuint64_t strides[2] = {(cuuint64_t)N * sizeof(__half), (cuuint64_t)N * N * sizeof(__half)};
    cuuint32_t box[3] = {64, 32, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CF_REQUIRE(r == CUDA_SUCCESS, CF_ERR_CUDA, "cuTensorMapEncodeTiled (fp16 volume) failed with CUresult %d", (int)r);
    return CF_OK;
}

}  // namespace tc

bool corr_tensor_core_supported(int D, int h, int w) {
    return D % tc::BK == 0 && ((int64_t)h * w) % 4 == 0;
}

// fp16 operand copies of both feature maps + per-item maxima and inverse scales (CF_CORR_F16 / CF_CORR_AUTO)
size_t corr_tc_workspace_bytes(int B, int D, int h, int w) {
    const size_t per_map = align_up((size_t)B * D * h * w * sizeof(__half), 256);
    return 2 * per_map + align_up((size_t)6 * B * sizeof(float), 256);   // maxima, inverse scales, arrival counters
}

// 3xTF32: hi and lo copies of both feature maps, [hi1 | lo1 | hi2 | lo2], each B*D*h*w floats rounded up to 256 bytes
size_t corr_x3_workspace_bytes(int B, int D, int h, int w) {
    return 4 * align_up((size_t)B * D * h * w * sizeof(float), 256);
}

// half_out: the levels are fp16 ([B*N][h>>l][w>>l] halves behind the float pointers; cf_corr_build_half, flags == 0).
// flags (debug/experiments, env CF_TC_FLAGS): bit1 = encode the tensor maps as plain FLOAT32 (operands are
// then truncated, not rounded, to TF32), bit2 = never fuse the pooling, bit3 = fuse level 1 only, bit4 = per-atom 2-D TMA boxes even when N % 32 == 0.
int corr_volume_tensor_core(const float *f1, const float *f2, int B, int D, int h, int w, float scale, float *level0,
                            float *level1, float *level2, float *level3, int precision, void *ws, size_t ws_bytes, int flags,
                            int *fused_levels, cudaStream_t stream, bool half_out) {
    using namespace tc;
    CF_REQUIRE(!half_out || (flags == 0 && precision != CF_CORR_3XTF32), CF_ERR_UNSUPPORTED,
               "cf_corr_build_half: no fp16 pyramid for precision %d", precision);
    CF_REQUIRE(precision == CF_CORR_TF32 || precision == CF_CORR_F16 || precision == CF_CORR_AUTO || precision == CF_CORR_3XTF32,
               CF_ERR_UNSUPPORTED, "cf_corr_build: precision %d has no tensor-core path", precision);
    CF_REQUIRE(aligned16(f1) && aligned16(f2) && aligned16(level0), CF_ERR_ALIGN, "cf_corr_build: tensors must be 16-byte aligned");
    const int N = h * w;
    // AUTO (round 2): fp16 operands where they measured faster on the B200 -- wide maps whose N is a whole number of
    // 64-column fp16 boxes and enough tiles to amortise the conversion pass (8 x 60x80: 288 against 319 us, 64 x 60x80: 2375
    // against 2580 us) -- TF32 elsewhere (64 x 24x32: 61 against 108 us, 64 x 36x44: 336 against 374, 1 x 80x124: 183 against 205)
    if (precision == CF_CORR_AUTO)
        precision = (N % 64 == 0 && N >= 2048 && (int64_t)B * N >= 19200 && D % BK_F16 == 0 && ws != nullptr &&
                     ws_bytes >= corr_tc_workspace_bytes(B, D, h, w)) ? CF_CORR_F16 : CF_CORR_TF32;
    if (precision == CF_CORR_F16 && D % BK_F16 != 0) precision = CF_CORR_TF32;   // the fp16 stages hold 128 K rows
    const bool f16 = precision == CF_CORR_F16, x3 = precision == CF_CORR_3XTF32;
    const int BC = f16 ? 64 : 32;   // operand columns per TMA box
    const void *a = f1, *bm = f2;
    const float *inv_scale = nullptr;
    size_t lo_off = 0;              // 3xTF32: bytes from a hi copy to its lo copy
    if (x3) {
        const size_t need = corr_x3_workspace_bytes(B, D, h, w);
        CF_REQUIRE(ws && ws_bytes >= need, CF_ERR_WORKSPACE, "cf_corr_build: workspace too small for CF_CORR_3XTF32 (%zu < %zu)",
                   ws_bytes, need);
        CF_REQUIRE(aligned16(ws), CF_ERR_ALIGN, "cf_corr_build: workspace not 16-byte aligned");
        lo_off = need / 4;
        char *base = reinterpret_cast<char *>(ws);
        float4 *hi1 = reinterpret_cast<float4 *>(base), *lo1 = reinterpret_cast<float4 *>(base + lo_off);
        float4 *hi2 = reinterpret_cast<float4 *>(base + 2 * lo_off), *lo2 = reinterpret_cast<float4 *>(base + 3 * lo_off);
        const int64_t n4 = (int64_t)B * D * N / 4;   // N % 4 == 0 (corr_tensor_core_supported)
        const int64_t blocks = ceil_div(2 * n4, 256);
        const int64_t cap = 8 * (int64_t)sm_count();
        fmap_split_tf32_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, stream>>>(
            reinterpret_cast<const float4 *>(f1), reinterpret_cast<const float4 *>(f2), n4, hi1, lo1, hi2, lo2);
        CF_LAUNCH_CHECK("fmap_split_tf32_kernel");
        a = hi1; bm = hi2;
    }
    if (f16) {
        const size_t need = corr_tc_workspace_bytes(B, D, h, w);
        CF_REQUIRE(ws && ws_bytes >= need, CF_ERR_WORKSPACE, "cf_corr_build: workspace too small for CF_CORR_F16 (%zu < %zu)",
                   ws_bytes, need);
        CF_REQUIRE(aligned16(ws), CF_ERR_ALIGN, "cf_corr_build: workspace not 16-byte aligned");
        const int64_t per_item = (int64_t)D * N;   // N % 4 == 0 (corr_tensor_core_supported)
        const size_t per_map = align_up((size_t)B * per_item * sizeof(__half), 256);
        __half *h1 = reinterpret_cast<__half *>(ws), *h2 = reinterpret_cast<__half *>(reinterpret_cast<char *>(ws) + per_map);
        unsigned *amax = reinterpret_cast<unsigned *>(reinterpret_cast<char *>(ws) + 2 * per_map);
        float *inv = reinterpret_cast<float *>(amax + 2 * B);
        int *arrived = reinterpret_cast<int *>(inv + 2 * B);
        const int parts = (int)ceil_div(per_item / 4, CV_THREADS * CV_F4);
        int resident = 0;
        CF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, fmap_to_half_fused_kernel, CV_THREADS, 0));
        const int64_t cap = (int64_t)resident * sm_count();
        if (parts <= cap && !(flags & (1 << 16))) {   // (flags bit16: the two-pass form)
            // one pass: every slice of an item is in flight at once (parts <= CTAs of the launch)
            CF_CUDA(cudaMemsetAsync(amax, 0, sizeof(unsigned) * 2 * B, stream));
            CF_CUDA(cudaMemsetAsync(arrived, 0, sizeof(int) * 2 * B, stream));
            const int64_t units = (int64_t)2 * B * parts;
            fmap_to_half_fused_kernel<<<(unsigned)(units < cap ? units : cap), CV_THREADS, 0, stream>>>(f1, f2, per_item, B, parts, amax,
                                                                                                   arrived, h1, h2, inv);
            CF_LAUNCH_CHECK("fmap_to_half_fused_kernel");
        } else {
        CF_CUDA(cudaMemsetAsync(amax, 0, sizeof(unsigned) * 2 * B, stream));
        // groups of batch items whose fp32 maps fit the L2 together (<= 48 MB): the conversion pass re-reads what the
        // maximum pass just read out of L2, so the feature maps cross the HBM interface once, not twice
        int nbc = (int)((48ll << 20) / (2 * per_item * (int64_t)sizeof(float)));
        if (nbc < 1) nbc = 1;
        if (nbc > B) nbc = B;
        for (int b0 = 0; b0 < B; b0 += nbc) {
            const int nb_ = B - b0 < nbc ? B - b0 : nbc;
            int64_t bx = ceil_div(per_item / 4, 256 * 8);
            const int64_t cap = ceil_div(8 * (int64_t)sm_count(), 2 * nb_);
            if (bx > cap) bx = cap;
            if (bx < 1) bx = 1;
            dim3 grid((unsigned)bx, (unsigned)(2 * nb_));
            fmap_absmax_kernel<<<grid, 256, 0, stream>>>(f1, f2, per_item, B, b0, nb_, amax);
            CF_LAUNCH_CHECK("fmap_absmax_kernel");
            fmap_to_half_kernel<<<grid, 256, 0, stream>>>(f1, f2, per_item, B, b0, nb_, amax, h1, h2, inv);
            CF_LAUNCH_CHECK("fmap_to_half_kernel");
        }
        }
        a = h1; bm = h2; inv_scale = inv;
    }
    Params p{};
    p.B = B; p.D = D; p.N = N; p.h = h; p.w = w; p.scale = scale; p.l0 = level0; p.l1 = level1;
    p.inv_scale = inv_scale;
    p.h1 = h / 2; p.w1 = w / 2;
    // R = number of whole target rows per tile (even).  The epilogue reads 32-column chunks, so the
    // last chunk of the last row must stay inside the 256-column accumulator stage.
    int R = 0;
    if (level1 != nullptr && !(flags & 4) && (w % 4 == 0) && (h % 2 == 0) && 2 * w <= MAX_BN) {
        R = 2 * (MAX_BN / (2 * w));
        if (R > h) R = h;
        while (R > 0 && (R - 1) * w + (int)align_up(w, 32) > MAX_BN) R -= 2;
        // narrow maps: whole groups of 8 (or 4) rows per tile, so that levels 2 and 3 can be pooled in the epilogue too
        if (!(flags & 8) && w <= 32 && w % 8 == 0) {
            if (R >= 8 && h % 8 == 0) R &= ~7;
            else if (R >= 4 && h % 4 == 0) R &= ~3;
        }
    }
    // levels this launch produces beyond level 0.  Levels 2 / 3 ride along when a tile holds whole groups of 4 / 8
    // target rows (R % 4 == 0 / R % 8 == 0: maps up to 64 / 32 wide) and the widths halve evenly (flags bit3: off)
    p.deep = 0;
    if (R > 0 && !(flags & 8) && w <= 32 && level2 != nullptr && aligned16(level2) && R % 4 == 0 && w % 8 == 0 && h % 4 == 0) {
        p.deep = 1;
        if (level3 != nullptr && R % 8 == 0 && w % 8 == 0 && h % 8 == 0) p.deep = 2;
    }
    p.h2 = h / 4; p.w2 = w / 4; p.h3 = h / 8; p.w3 = w / 8;
    p.l2 = level2; p.l3 = level3;
    // wide maps (R == 2): level 2 out of pairs of tiles (kernel: pair2).  Needs an even number of target-row pairs, level-2
    // rows that start 16-byte aligned per 32-column strip, and w1 free TMEM columns behind stage 0's accumulator
    p.pair2 = 0;
    if (R == 2 && p.deep == 0 && !(flags & 8) && !(flags & 64) && level2 != nullptr && aligned16(level2) && h % 4 == 0 && w % 16 == 0 &&
        (int)align_up(R * w, 16) + w / 2 <= MAX_BN)
        p.pair2 = 1;
    // ... and level 3 out of quads of tiles (kernel: quad3): needs level-2 rows that pool inside a 32-column strip (w % 16 == 0
    // gives 4 or 8 level-2 values per strip) and w2 more free TMEM columns; h / 8 level-3 rows (a last half quad only parks)
    // MEASURED SLOWER (64 x 60x80: 2571 against 2007-2026 us, 8 x 60x80: 293 against 255): it saves the 89 us pooling kernel, but a
    // lane's four level-3 values are 16 bytes of a 280-byte per-query map -- 32 scattered partial-sector writes per store
    // instruction where the pooling kernel writes level 3 as one dense stream.  Parity-tested, on request only (flags bit25).
    p.quad3 = 0;
    if (p.pair2 && level3 != nullptr && (flags & (1 << 25)) && h >= 8 && w >= 8 &&
        (int)align_up(R * w, 16) + 24 * (int)ceil_div(w, 32) <= MAX_BN)
        p.quad3 = 1;
    *fused_levels = R > 0 ? 1 + (p.quad3 ? 2 : (p.pair2 ? 1 : p.deep)) : 0;
    p.stream_l0 = (int64_t)B * N * N * (half_out ? 2 : 4) > (64ll << 20);
    if (R > 0) {
        p.R = R;
        p.BN = R * w;
        p.tiles_n = (int)ceil_div(h, R);
    } else {
        p.R = 0;
        p.BN = N < MAX_BN ? (int)align_up(N, 16) : MAX_BN;
        p.tiles_n = (int)ceil_div(N, p.BN);
    }
    p.BN_mma = (int)align_up(p.BN, 16);
    p.n_boxes_b = (int)ceil_div(p.BN_mma, BC);
    p.tiles_m = (int)ceil_div(N, BM);
    p.tiles_nv = p.quad3 ? (int)align_up(p.tiles_n, 4) : p.tiles_n;
    const int64_t total = (int64_t)B * p.tiles_m * p.tiles_nv;
    CF_REQUIRE(total < (1ll << 31), CF_ERR_INVALID_ARG, "cf_corr_build: too many tiles");
    p.total_tiles = (int)total;

    const CUtensorMapDataType dt = f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                       : ((flags & 2) ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_TFLOAT32);
    p.atoms3d = (N % BC == 0) && !(flags & 16);
    p.b3d = p.atoms3d && (p.BN % BC == 0 || p.tiles_n == 1);
    const bool pair_req = (flags & 64) && !f16 && !x3;
    const int bk = f16 ? BK_F16 : ((pair_req || D % BK_TF32 != 0) ? BK : BK_TF32);          // K rows per stage
    const int boxb = 128 * bk;                 // bytes per TMA box
    const int a_bytes = (x3 ? 2 : 1) * (BM / BC) * boxb;
    p.stage_bytes = a_bytes + (x3 ? 2 : 1) * p.n_boxes_b * boxb;
    p.b_sw64 = 0;
    // (the 128-byte-swizzled slice is one 3-D box only when tiles start on 64-column boundaries -- b3d; with 160-column tiles
    //  it took three 2-D boxes per stage)
    if (f16 && p.atoms3d && N % 32 == 0 && !pair_req && !(flags & (1 << 17)) && p.BN_mma % 64 == 32 && p.BN % 32 == 0) {
        p.b_sw64 = 1;
        p.stage_bytes = a_bytes + (p.BN_mma / 32) * bk * 64;
    }
    // two epilogue warps per TMEM lane quarter when the ring still gets >= 5 stages beside their 64 KB of buffers (fp16
    // operands); the deep pooling keeps per-thread row state and stays on one warp per quarter (flags bit7: force 1)
    // (measured slower again, also with the half-size fp16 stages: 396 against 359 us at 8 x 60x80 -- only on request)
    // round 2: with 64-row fp16 stages the operand loads take 4 x 0.45 us and the MMAs 1.9 us per 128x160 tile; the
    // epilogue on four warps (3.6 us per tile, corr_trace) became the critical path -> two warps per lane quarter by
    // default for fp16 operands (flags bit7 now forces one)
    const int es = (f16 && p.deep == 0 && !(flags & 128) && (SMEM_LIMIT - smem_fixed(2)) / p.stage_bytes >= 2) ? 2 : 1;
    p.stages = (SMEM_LIMIT - smem_fixed(es)) / p.stage_bytes;
    if (p.stages > MAX_STAGES) p.stages = MAX_STAGES;
    // 3xTF32 stages are twice the TF32 ones (72 KB at BN = 160, 96 KB at BN = 256): a ring of two beside the epilogue
    CF_REQUIRE(!x3 || p.stages >= 2, CF_ERR_UNSUPPORTED, "cf_corr_build: %d-byte operand stages leave room for %d in shared memory",
               p.stage_bytes, p.stages);
    // pairs of query tiles as one 256-row UMMA across two CTAs: measured slower than one CTA per tile on the B200
    // (8 x 60x80: 359 against 322 us, see the kernel's header), so only on request (flags bit6)
    const bool pair = (flags & 64) && p.tiles_m >= 2 && !f16 && !x3;
    p.ablate = (flags >> 8) & 255;
    // level-0 rows through the LSU instead of TMA bulk stores: helps where the operand loads already need many TMA
    // instructions per stage (N % 32 != 0: 64 x 36x44 398 -> 367 us), costs 2-5 % elsewhere (flags bit0: always TMA)
    p.lsu_stores = (!(flags & 1) && !p.atoms3d && N % 4 == 0 && !half_out) ? 1 : 0;   // (fp16 level 0: always {64 x 32} boxes)
    // round 2, measured and NOT adopted for fp16 operands: (a) level-0 rows through the LSU (flags bit5): 64 x 60x80 2617
    // against 2515 us; (b) one bulk store per 32-column chunk for all 128 rows of the tile (box {32, 128}, the four
    // epilogue warps of a lane-quarter group meeting at a named barrier; 5 store instructions per tile instead of 20):
    // 2704 against 2375 us (TF32: 2744 against 2580) -- the stores' instruction count is not what holds the epilogue up
    if (f16 && N % 4 == 0 && (flags & 32)) p.lsu_stores = 1;
    // (d) what the data movement alone costs (scripts/experiments/write_probe.cu -> profiles/r02/write_probe.txt, no MMAs, no
    // epilogue arithmetic, per 128x160 tile and SM): the two 80 KB operand stages 1.12 us; the 20 level-0 boxes 2.4-2.5 us
    // (4.9-5.0 TB/s chip-wide, the same with 2 CTAs per SM or 2-atom boxes: ~3.75 ns per 128-byte box row); both together
    // 3.27 us -- the TMA unit mostly serialises them, and the kernel's 3.75 us per tile (with levels 1-2 on top) is within 15 %
    // of that.  A write-only stream reaches 6.1-6.2 TB/s (memset 7.0), one bulk store per whole 640-byte tile row 5.9 TB/s,
    // loads + row stores 2.5 us per tile.  Two epilogues built on row stores (padded row-major staging, 16 rows per lane
    // quarter single-buffered / 8 rows double-buffered, the warp pair of a quarter meeting at a named barrier, lanes issuing
    // their rows) passed the parity tests and were SLOWER: 2685 / 3350 against 2100-2190 us at 64 x 60x80 -- beside two 80 KB
    // operand stages only 64 KB are left, a lane quarter's rows (20 KB) cannot all be staged at once, and the extra passes
    // (barriers, TMEM re-reads at the register cap of 168) lengthen the epilogue's serial chain more than the cheaper stores
    // shorten the TMA queue.  (e) level-0 chunks split between TMA (half-0 warps) and LSU (half-1 warps) or the reverse:
    // 2280 / 2318 against 2190 us.  (f) other splits of the 5 chunks between the two warps of a lane quarter than the
    // alternating 3 | 2 (the second warp also takes 2 of the 3 pooling strips): 4 | 1 2256-2276, 2 | 3 2240, 5 | 0 2372 against
    // 2197 us.  All removed again.  What the per-tile timeline shows (scripts/corr_trace.py with the stamps of four epilogue
    // warps, profiles/r02/corr_trace_f16_8x60x80.txt): an epilogue warp is busy 2.75-3.0 us per tile and then WAITS 0.6-0.9 us for
    // the next accumulator; the tile period (3.6-3.9 us) is the chain  accumulator drained by all 8 warps -> operand stages
    // of the tile after next land (the ring of two 80 KB stages holds exactly one tile's K, and these loads queue in the TMA
    // unit behind the store boxes) -> its MMAs run (~2 us, bound by the operand fetch from shared memory) -> epilogue.
    // (c) one epilogue pass per 32-column strip of an R == 2 tile -- both level-0 boxes, level 1 and level 2 from ONE pair of
    // TMEM loads instead of 5 chunk loads + 6 strip loads per warp, no drain between the phases: SLOWER on the same box
    // (64 x 60x80: fp16 2668 against 2558 us, TF32 2482 against 2392 us) -- each warp then has a single pair of staging
    // buffers in flight and waits for its bulk stores once per strip.  Removed again; the two-phase epilogue stays.
    // level-1 rows through shared memory into 64-byte runs (flags bit13: per-lane 16-byte stores): 64 x 24x32
    // 66.7 -> 60.8 us, 8 x 60x80 314 -> 309 us
    p.l1_staged = (p.R > 0 && p.w1 % 2 == 0 && !(flags & 8192) && !(flags & (1 << 24)) && !half_out) ? 1 : 0;   // (bit24: off, without bit13's ablation side effect; fp16: per-lane stores)
    // level 0 as one multi-atom box per lane quarter (kernel: qbox).  Needs whole tiles (h % R == 0), 32-column atoms that
    // start on atom boundaries, whole lane quarters (N % 32 == 0) and the tile's level 0 (BN x 128 x 4 B) inside the shared
    // memory left beside the operand ring -- for 160 columns that takes the 64-byte-swizzled fmap2 slice (b_sw64).  The
    // level-1 scratch has no room then: level-1 rows leave as per-lane 16-byte stores.  Measured SLOWER at 64 x 60x80: 2476
    // against 1985 us for the twenty single boxes on the same box (one buffer per lane quarter: every tile waits for its
    // predecessor's box to leave, and two named barriers) -- only on request (flags bit19).  flags bit17 switches b_sw64 off.
    // (Also measured: the epilogue's shared-memory accesses as explicit st.shared / ld.shared asm instead of the generic ST.E / LD.E
    //  the compiler emits for the aligned-up buffer pointer: 2545-2568 against 2221-2243 us on one box -- volatile asm with a memory
    //  clobber pins every store in program order between the TMEM loads and fences; the plain C++ dereferences stay.)
    // Most of that loss is the level-1 rows: per-lane 16-byte stores alone (flags bit24, single boxes) cost 2485 against 2015 us
    // at this shape.  A variant with one {32 x 32 x 3 | 2} box per WARP (no barrier, 8 stores per tile; write_probe: 5.8 against
    // 4.9 TB/s for the stores alone, 4.3 against 3.7 with the operand loads) measured 2630 us with the same level-1 stores,
    // i.e. still behind the single boxes -- removed again.
    p.frag_stores = (R > 0 && (flags & (1 << 26)) && h % R == 0 && N % 8 == 0 && p.BN % 32 == 0 && !pair) ? 1 : 0;
    p.qbox = 0;
    if (es == 2 && R > 0 && (flags & (1 << 19)) && h % R == 0 && N % 32 == 0 && p.BN % 32 == 0 && !p.lsu_stores && !pair &&
        p.stages * p.stage_bytes + 4 * (p.BN / 32) * EPI_BUF_BYTES + 1024 + 256 <= SMEM_LIMIT) {
        p.qbox = 1;
        p.l1_staged = 0;
        const int nch = p.BN / 32, ns = (R / 2) * (int)ceil_div(w, 32);
        // a pooling strip costs a warp about twice a chunk (timeline): the second warp gets one strip more when their count is odd
        p.qbox_h0 = (nch + 1) / 2 + ((ns & 1) ? 1 : 0);
        if (p.qbox_h0 > nch) p.qbox_h0 = nch;
        if ((flags >> 20) & 15) p.qbox_h0 = min(nch, ((flags >> 20) & 15) - 1);
    }
    p.tiles_mp = (int)ceil_div(p.tiles_m, 2);
    p.b_half = (int)ceil_div(p.BN_mma / 2, 32);
    if (pair) {
        p.total_tiles = B * p.tiles_mp * p.tiles_n;
        p.b3d = p.b3d && (p.BN_mma / 2) % 32 == 0;
        p.stage_bytes = A_BYTES + p.b_half * BOX_BYTES;
        p.stages = (SMEM_LIMIT - smem_fixed(1)) / p.stage_bytes;
        if (p.stages > MAX_STAGES) p.stages = MAX_STAGES;
    }
    p.epi_bytes = p.qbox ? 4 * (p.BN / 32) * EPI_BUF_BYTES : epi_bytes(es);
    p.l1_scratch = 0;
    if (es == 2 && !p.qbox && p.l1_staged && p.stages * p.stage_bytes + epi_bytes(2) + 8 * 2048 + 1024 + 256 <= SMEM_LIMIT) {
        p.l1_scratch = epi_bytes(2);
        p.epi_bytes += 8 * 2048;
    }
    const int smem_bytes = p.stages * p.stage_bytes + p.epi_bytes + 1024 + 256;
    CUtensorMap ta, tb, tcm;
    if (x3) {
        if (int rc = make_split_tmap(&ta, static_cast<const float *>(a), lo_off, B, D, N, bk, p.atoms3d ? BM / 32 : 0)) return rc;
    } else if (p.atoms3d) {
        if (int rc = make_fmap_tmap3(&ta, a, B, D, N, dt, bk, BM / BC)) return rc;
    } else {
        if (int rc = make_fmap_tmap(&ta, a, B, D, N, dt, bk)) return rc;
    }
    if (x3) {
        if (int rc = make_split_tmap(&tb, static_cast<const float *>(bm), lo_off, B, D, N, bk, p.b3d ? p.n_boxes_b : 0)) return rc;
    } else if (p.b_sw64) {
        if (int rc = make_fmap_tmap3_sw64(&tb, bm, B, D, N, bk, p.BN_mma / 32)) return rc;
    } else if (p.b3d) {
        if (int rc = make_fmap_tmap3(&tb, bm, B, D, N, dt, bk, pair ? p.b_half : p.n_boxes_b)) return rc;
    } else {
        if (int rc = make_fmap_tmap(&tb, bm, B, D, N, dt, bk)) return rc;
    }
    if (half_out) {
        if (int rc = make_volume_tmap_half(&tcm, level0, B, N)) return rc;
    } else if (p.qbox) {
        if (int rc = make_volume_tmap_atoms(&tcm, level0, B, N, p.BN / 32)) return rc;
    } else if (int rc = make_volume_tmap(&tcm, level0, B, N)) return rc;

    int dev = 0;
    CF_CUDA(cudaGetDevice(&dev));
    static bool opt_in[64] = {};
    if (!opt_in[dev & 63]) {
        CF_CUDA(cudaFuncSetAttribute(corr_tc_kernel<1, OM_TF32, 1, BK_TF32>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
        CF_CUDA(cudaFuncSetAttribute(corr_tc_kernel<1, OM_TF32, 1, BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
        CF_CUDA(cudaFuncSetAttribute(corr_tc_kernel<2, OM_TF32, 1, BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
        CF_CUDA(cudaFuncSetAttribute(corr_tc_kernel<1, OM_F16, 1, BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
        CF_CUDA(cudaFuncSetAttribute(corr_tc_kernel<1, OM_F16, 2, BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
        CF_CUDA(cudaFuncSetAttribute(corr_tc_kernel<1, OM_3XTF32, 1, BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
        opt_in[dev & 63] = true;
    }
    const int sms = sm_count();
    if (pair) {
        const int clusters = p.total_tiles < sms / 2 ? p.total_tiles : sms / 2;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(2 * clusters));
        cfg.blockDim = dim3(threads(1));
        cfg.dynamicSmemBytes = smem_bytes;
        cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        CF_CUDA(cudaLaunchKernelEx(&cfg, corr_tc_kernel<2, OM_TF32, 1, BK>, ta, tb, tcm, p));
        CF_LAUNCH_CHECK("corr_tc_kernel<pair>");
        return CF_OK;
    }
    const int grid = p.total_tiles < sms ? p.total_tiles : sms;
    if (half_out) {
        static bool opt_in_half[64] = {};
        if (!opt_in_half[dev & 63]) {
            CF_CUDA(cudaFuncSetAttribute(corr_tc_half_kernel<1, OM_TF32, 1, BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
            CF_CUDA(cudaFuncSetAttribute(corr_tc_half_kernel<1, OM_F16, 1, BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
            CF_CUDA(cudaFuncSetAttribute(corr_tc_half_kernel<1, OM_F16, 2, BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
            opt_in_half[dev & 63] = true;
        }
        if (f16 && es == 2) corr_tc_half_kernel<1, OM_F16, 2, BK><<<grid, threads(2), smem_bytes, stream>>>(ta, tb, tcm, p);
        else if (f16) corr_tc_half_kernel<1, OM_F16, 1, BK><<<grid, threads(1), smem_bytes, stream>>>(ta, tb, tcm, p);
        else corr_tc_half_kernel<1, OM_TF32, 1, BK><<<grid, threads(1), smem_bytes, stream>>>(ta, tb, tcm, p);
        CF_LAUNCH_CHECK(f16 ? "corr_tc_half_kernel<f16>" : "corr_tc_half_kernel");
        return CF_OK;
    }
    if (f16) {
        if (es == 2) corr_tc_kernel<1, OM_F16, 2, BK><<<grid, threads(2), smem_bytes, stream>>>(ta, tb, tcm, p);
        else corr_tc_kernel<1, OM_F16, 1, BK><<<grid, threads(1), smem_bytes, stream>>>(ta, tb, tcm, p);
        CF_LAUNCH_CHECK("corr_tc_kernel<f16>");
        return CF_OK;
    }
    if (x3) {
        corr_tc_kernel<1, OM_3XTF32, 1, BK><<<grid, threads(1), smem_bytes, stream>>>(ta, tb, tcm, p);
        CF_LAUNCH_CHECK("corr_tc_kernel<3xtf32>");
        return CF_OK;
    }
    if (bk == BK_TF32) corr_tc_kernel<1, OM_TF32, 1, BK_TF32><<<grid, threads(1), smem_bytes, stream>>>(ta, tb, tcm, p);
    else corr_tc_kernel<1, OM_TF32, 1, BK><<<grid, threads(1), smem_bytes, stream>>>(ta, tb, tcm, p);
    CF_LAUNCH_CHECK("corr_tc_kernel");
    return CF_OK;
}

}  // namespace cf

// debug only (not part of include/cistaflow.h): copies the 32 clock64 stamps of the last launch
extern "C" __attribute__((visibility("default"))) int cf_debug_tc_timeline(unsigned long long *host_out) {
    return cudaMemcpyFromSymbol(host_out, cf::tc::g_tc_timeline, sizeof(unsigned long long) * 32) == cudaSuccess ? 0 : -6;
}
