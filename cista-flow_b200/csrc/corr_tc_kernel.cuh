// The tensor-core correlation kernel (see corr_build_tc.cu), included twice by corr_build_tc.cu:
//   CF_TC_KERNEL = corr_tc_kernel,      CF_TC_OUT = float    the fp32 pyramid (cf_corr_build)
//   CF_TC_KERNEL = corr_tc_half_kernel, CF_TC_OUT = __half   the fp16 pyramid (cf_corr_build_half)
// The fp16 pyramid's code sits in `if constexpr (HO)` branches: level 0 is rounded to fp16 in registers and leaves as
// {64 cols x 32 rows} fp16 boxes (128-byte rows, the staging image of one fp32 {32 x 32} box: half the boxes per tile);
// the fused levels are pooled from the rounded values and stored as fp16 with the widest store their alignment allows.
// (A textual include, not a shared __device__ function: the fp32 kernel compiles to the same code as before the fp16
// pyramid existed -- a function boundary alone changed its register allocation.)
template <int CL, int OM, int ES, int BKT>
__global__ void __launch_bounds__(threads(ES), 1)
CF_TC_KERNEL(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
             const __grid_constant__ CUtensorMap tmap_c, const Params p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    constexpr bool F16 = OM == OM_F16, X3 = OM == OM_3XTF32;
    constexpr bool HO = std::is_same<CF_TC_OUT, __half>::value;
    static_assert(!HO || (CL == 1 && !X3), "the fp16 pyramid is built by the single-CTA TF32 and fp16-operand kernels");
    static_assert(OM == OM_TF32 || CL == 1, "the CTA-pair variant is tf32 only");
    constexpr int EPI_SPLIT = ES, EPI_WARPS = 4 * ES, EPI_BYTES = epi_bytes(ES);
#ifdef CF_SWAP_SERVICE_WARPS   // experiment: which warp scheduler (warp % 4) hosts the producer / the MMA issuer
    constexpr int PRODUCER_WARP = EPI_WARPS + 1, MMA_WARP = EPI_WARPS;
#else
    constexpr int PRODUCER_WARP = EPI_WARPS, MMA_WARP = EPI_WARPS + 1;
#endif
    constexpr int BC = F16 ? 64 : 32;                   // operand columns per TMA box (128 bytes)
    constexpr int BKK = F16 ? BK_F16 : BKT;             // K rows per stage (TF32: 64, or 32 for D % 64 != 0 and the CTA-pair kernel)
    constexpr int BOXB = 128 * BKK;                     // bytes of one TMA box: 128-byte rows x BKK
    constexpr int PARTS = X3 ? 2 : 1;                   // slices per 32-column atom (3xTF32: hi, lo)
    constexpr int ABYTES = PARTS * (BM / BC) * BOXB;    // fmap1 part of a stage
    constexpr int MMAS = F16 ? BKK / 16 : BKK / 8;      // MMAs per stage
    constexpr int KSTEP = F16 ? 2048 : 1024;            // descriptor start-address advance per MMA
    const int STAGES = p.stages, STAGE_BYTES = p.stage_bytes;
    uint8_t *epi = smem + STAGES * STAGE_BYTES;  // [EPI_WARPS][2][EPI_BUF_BYTES]
    uint64_t *bars = reinterpret_cast<uint64_t *>(epi + p.epi_bytes);
    uint64_t *full = bars, *empty = bars + MAX_STAGES;
    uint64_t *tfull = bars + 2 * MAX_STAGES, *tempty = bars + 2 * MAX_STAGES + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * MAX_STAGES + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kblocks = p.D / BKK;
    const int rank = CL == 2 ? (int)cluster_ctarank() : 0;
    const int first_tile = (int)blockIdx.x / CL, tile_step = (int)gridDim.x / CL;
    // the s-th tile of this CTA: tile indices have the target-row pair nb fastest, so with pair2 a CTA takes the two tiles
    // 2u, 2u+1 of unit u back to back (same batch item, same query rows, target rows 4u' .. 4u'+3)
    const int GS = p.quad3 ? 4 : (p.pair2 ? 2 : 1), gs_shift = p.quad3 ? 2 : (p.pair2 ? 1 : 0);
    auto tile_of = [&](int sq) { return ((first_tile + (sq >> gs_shift) * tile_step) << gs_shift) + (sq & (GS - 1)); };
    // (b, mb, nb) of the next tile of this CTA without integer divisions (three of them per tile, twice with the look-ahead
    // of the fp16 epilogue, were ~0.5 us of every tile's serial chain): the step from the last tile of a group to the first
    // of the next is a constant, decomposed once
    const int jump = GS * tile_step - (GS - 1);
    const int jump_n = jump % p.tiles_nv, jump_m = (jump / p.tiles_nv) % p.tiles_m, jump_b = (jump / p.tiles_nv) / p.tiles_m;
    auto advance = [&](int sq, int &tile, int &b, int &mb, int &nb) {   // tile of sequence number sq -> sq + 1   (CL == 1)
        if ((sq & (GS - 1)) != GS - 1) {   // next tile of the group: the next target-row pair (tiles_nv is a multiple of GS)
            ++tile;
            ++nb;
            return;
        }
        tile += jump;
        nb += jump_n;
        int c = nb >= p.tiles_nv ? 1 : 0;
        nb -= c ? p.tiles_nv : 0;
        mb += jump_m + c;
        c = mb >= p.tiles_m ? 1 : 0;
        mb -= c ? p.tiles_m : 0;
        b += jump_b + c;
    };
    if (threadIdx.x == 0) stamp(0);

    if (warp == PRODUCER_WARP && lane == 0) {
        tma_prefetch_desc(&tmap_a);
        tma_prefetch_desc(&tmap_b);
        tma_prefetch_desc(&tmap_c);
    }
    if (warp == MMA_WARP) {
        if (lane == 0) {
            for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
            for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 32 * EPI_WARPS * CL); }
            fence_barrier_init();
        }
        __syncwarp();
        if (CL == 2) tmem_alloc_2sm(tmem_slot, 512);
        else tmem_alloc(tmem_slot, 512);
    }
    tc_fence_before();
    __syncthreads();
    if (CL == 2) cluster_sync_all();  // the peer's barriers are initialised (and its TMEM allocated) before anything targets them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (threadIdx.x == 0) stamp(1);

    if (warp == PRODUCER_WARP) {
        // ------------------------------------------------------------ TMA producer
        // (whole warp convergent, an elected lane issues -- see the MMA issuer below: under `if (lane == 0)` every
        //  cp.async.bulk.tensor cost an ELECT / R2UR / BRA.U.ANY sequence, the "one TMA issue per ~100 cycles" measured
        //  earlier)
        {
            int stage = 0;
            uint32_t phase = 0;
            // pair kernel: the leader's barrier counts the bytes of BOTH CTAs' boxes
            const uint32_t tx_bytes = (F16 && p.b_sw64) ? (uint32_t)p.stage_bytes
                                                       : (uint32_t)(CL * PARTS * (BM / BC + (CL == 2 ? p.b_half : p.n_boxes_b))) * BOXB;
            const int jr = CL == 2 ? rank * (p.BN_mma / 2) : 0;  // first fmap2 column of this CTA inside the tile
            int tile_no = 0;
            int tile = tile_of(0), b = 0, mb = 0, nb = 0;
            if (CL == 1 && tile < p.total_tiles) decode_tile(p, tile, b, mb, nb);
            for (; tile < p.total_tiles; ++tile_no) {
                if (CL == 2) decode_pair_tile(p, tile, rank, b, mb, nb);
                if (CL == 1 && nb >= p.tiles_n) {   // (quad3: padding index, no such tile)
                    advance(tile_no, tile, b, mb, nb);
                    continue;
                }
                const int i0 = mb * BM, j0 = nb * p.BN;
                for (int kb = 0; kb < kblocks; ++kb) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    if (lane == 0) {
                        if (kb == 0) TC_TRACE(tile_no, 0);
                        if (kb == kblocks - 1) TC_TRACE(tile_no, 1);
                    }
                    uint8_t *sa = smem + stage * STAGE_BYTES, *sb = sa + ABYTES;
                    const int krow = b * p.D + kb * BKK;
                    const bool issuer = elect_one();
                    if (!issuer) {
                        __syncwarp();
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                        continue;
                    }
                    if (p.ablate & 4) {
                        if (rank == 0) mbar_arrive(&full[stage]);
                        __syncwarp();
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                        continue;
                    }
                    if (CL == 2) {
                        if (rank == 0) mbar_expect_tx(&full[stage], tx_bytes);
                        const uint32_t lead_full = mapa_rank0(&full[stage]);
                        if (p.atoms3d) {
                            tma_load_3d_2sm(sa, &tmap_a, 0, krow, i0 >> 5, lead_full);
                        } else {
#pragma unroll
                            for (int a = 0; a < BM / 32; ++a) tma_load_2d_2sm(sa + a * BOX_BYTES, &tmap_a, i0 + 32 * a, krow, lead_full);
                        }
                        if (p.b3d) {
                            tma_load_3d_2sm(sb, &tmap_b, 0, krow, (j0 + jr) >> 5, lead_full);
                        } else {
                            for (int a = 0; a < p.b_half; ++a) tma_load_2d_2sm(sb + a * BOX_BYTES, &tmap_b, j0 + jr + 32 * a, krow, lead_full);
                        }
                        __syncwarp();
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                        continue;
                    }
                    mbar_expect_tx(&full[stage], tx_bytes);
                    if (X3) {   // both slices of each atom in one box: {32 cols, K rows, hi/lo, atoms} (per atom when N % 32 != 0)
                        if (p.atoms3d) {
                            tma_load_4d(sa, &tmap_a, 0, krow, 0, i0 / BC, &full[stage]);
                        } else {
#pragma unroll
                            for (int a = 0; a < BM / BC; ++a) tma_load_3d(sa + 2 * a * BOXB, &tmap_a, i0 + BC * a, krow, 0, &full[stage]);
                        }
                        if (p.b3d) {
                            tma_load_4d(sb, &tmap_b, 0, krow, 0, j0 / BC, &full[stage]);
                        } else {
                            for (int a = 0; a < p.n_boxes_b; ++a) tma_load_3d(sb + 2 * a * BOXB, &tmap_b, j0 + BC * a, krow, 0, &full[stage]);
                        }
                        __syncwarp();
                        if (++stage == STAGES) { stage = 0; phase ^= 1; }
                        continue;
                    }
                    if (p.atoms3d) {
                        tma_load_3d(sa, &tmap_a, 0, krow, i0 / BC, &full[stage]);
                    } else {
#pragma unroll
                        for (int a = 0; a < BM / BC; ++a) tma_load_2d(sa + a * BOXB, &tmap_a, i0 + BC * a, krow, &full[stage]);
                    }
                    if (F16 && p.b_sw64) {
                        tma_load_3d(sb, &tmap_b, 0, krow, j0 / 32, &full[stage]);
                    } else if (p.b3d) {
                        tma_load_3d(sb, &tmap_b, 0, krow, j0 / BC, &full[stage]);
                    } else {
                        for (int a = 0; a < p.n_boxes_b; ++a) tma_load_2d(sb + a * BOXB, &tmap_b, j0 + BC * a, krow, &full[stage]);
                    }
                    if (tile_no == 0 && kb == 0) stamp(2);
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                if (CL == 2) tile = tile_of(tile_no + 1);
                else advance(tile_no, tile, b, mb, nb);
            }
        }
    } else if (warp == MMA_WARP) {
        // -------------------------------------------------------------- MMA issuer
        // The WHOLE warp walks the loop (convergent, every value warp-uniform) and one elected lane issues: written as
        // `if (lane == 0) { ... }` the compiler wrapped every tcgen05.mma in an ELECT / R2UR.BROADCAST / BRA.U.ANY
        // sequence and rebuilt both 64-bit descriptors in front of it -- ~30 dependent uniform-datapath instructions
        // per MMA, i.e. an issue interval of ~180 cycles for an MMA that occupies the tensor pipe for ~90.
        if (rank == 0) {
            int stage = 0, acc = 0;
            uint32_t phase = 0, acc_phase = 0;
            const uint32_t idesc = F16 ? make_idesc_f16(p.BN_mma) : make_idesc_tf32(p.BN_mma, CL * BM);
            // descriptor high words are constants of the layout; the low word = start address >> 4 | LBO << 16
            const uint32_t desc_hi = F16 ? (uint32_t)((1024u >> 4) | (1u << 14) | (2u << 29))
                                         : (uint32_t)((512u >> 4) | (1u << 14) | (1u << 29));
            const uint32_t lbo_bits = ((uint32_t)(PARTS * BOXB) >> 4) << 16;   // bytes between column atoms = one TMA box per slice
            // fmap2 slice in the 64-byte swizzle (b_sw64): atoms of 32 columns x 64 B rows, 8-row groups 512 B apart, one
            // atom = BKK x 64 B, and a K step of 16 rows is 1024 B
            const bool sw64 = F16 && p.b_sw64;
            const uint32_t desc_hi_b = sw64 ? (uint32_t)((512u >> 4) | (1u << 14) | (4u << 29)) : desc_hi;
            const uint32_t lbo_bits_b = sw64 ? (((uint32_t)(BKK * 64) >> 4) << 16) : lbo_bits;
            const uint32_t kstep_b = sw64 ? (1024u >> 4) : (uint32_t)(KSTEP >> 4);
            const uint32_t smem_base = smem_u32(smem);
            int tile_no = 0;
            int wb_ = 0, wmb_ = 0, wnb_ = 0, wtile_ = tile_of(0);          // (b, mb, nb) carried only to skip quad3's padding indices
            if (CL == 1 && wtile_ < p.total_tiles) decode_tile(p, wtile_, wb_, wmb_, wnb_);
            for (int tile = tile_of(0); tile < p.total_tiles; tile = tile_of(++tile_no)) {
                if (CL == 1) {
                    const bool skip = wnb_ >= p.tiles_n;
                    advance(tile_no, wtile_, wb_, wmb_, wnb_);
                    if (skip) continue;
                }
                mbar_wait(&tempty[acc], acc_phase ^ 1);  // epilogue drained this accumulator
                tc_fence_after();
                if (lane == 0) TC_TRACE(tile_no, 2);
                const uint32_t d_tmem = tmem_base + (uint32_t)acc * MAX_BN;
                for (int kb = 0; kb < kblocks; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    if (lane == 0) {
                        if (tile_no == 0 && kb < 16) stamp(3 + kb);
                        if (kb < 8) TC_TRACE(tile_no, 3 + kb);
                    }
                    const uint32_t sa = smem_base + (uint32_t)(stage * STAGE_BYTES);
                    const uint32_t a_lo = (((sa & 0x3FFFFu) >> 4) | lbo_bits), b_lo = ((((sa + ABYTES) & 0x3FFFFu) >> 4) | lbo_bits_b);
                    if (elect_one()) {
                        if (!(p.ablate & 2)) {
#pragma unroll
                            for (int kk = 0; kk < MMAS; ++kk) {
                                const uint64_t da = ((uint64_t)desc_hi << 32) | (uint64_t)(a_lo + (uint32_t)(kk * (KSTEP >> 4)));
                                const uint64_t db = ((uint64_t)desc_hi_b << 32) | (uint64_t)(b_lo + (uint32_t)kk * kstep_b);
                                if (X3) {   // the small cross terms first, hi.hi last; only the tile's first MMA clears
                                    constexpr uint32_t LO = (uint32_t)BOXB >> 4;   // the lo slice: one box behind the hi slice
                                    umma_tf32(d_tmem, da + LO, db, idesc, (uint32_t)((kb | kk) != 0));
                                    umma_tf32(d_tmem, da, db + LO, idesc, 1u);
                                    umma_tf32(d_tmem, da, db, idesc, 1u);
                                } else if (F16) umma_f16(d_tmem, da, db, idesc, (uint32_t)((kb | kk) != 0));
                                else if (CL == 2) umma_tf32_2sm(d_tmem, da, db, idesc, (uint32_t)((kb | kk) != 0));
                                else umma_tf32(d_tmem, da, db, idesc, (uint32_t)((kb | kk) != 0));
                            }
                        }
                        // frees the smem slot once these MMAs have read it (pair kernel: in both CTAs)
                        if (CL == 2) umma_commit_2sm(&empty[stage], (uint16_t)3);
                        else umma_commit(&empty[stage]);
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                if (elect_one()) {
                    if (CL == 2) umma_commit_2sm(&tfull[acc], (uint16_t)3);  // accumulator complete -> both epilogues
                    else umma_commit(&tfull[acc]);
                }
                __syncwarp();
                if (lane == 0) {
                    if (tile_no == 0) stamp(19);
                    TC_TRACE(tile_no, 11);
                }
                acc ^= 1;
                if (acc == 0) acc_phase ^= 1;
            }
        }
    } else {
        // ---------------------------------------------------------------- epilogue
        // warp <-> TMEM lane quarter warp % 4 (a warp may only read those lanes); with EPI_SPLIT > 1 the warps of a
        // quarter take the tile's work items (32-column level-0 chunks, 32-column pooling strips) in turn
        int acc = 0;
        uint32_t acc_phase = 0, chunk_count = 0;
        const int quarter = warp & 3, half = warp >> 2;
        const int row = 32 * quarter + lane;
        const bool vec4_l0 = (p.N % 4) == 0 && (p.w % 4) == 0;
        const bool vec4_l1 = (p.w1 % 4) == 0;
        uint8_t *my_epi = epi + warp * 2 * EPI_BUF_BYTES;
        int tile_no = 0;
        // F16: 1/sqrt(D) times the powers of two that undo the per-item scaling of the operands.  The two factors of the NEXT
        // tile's item are fetched while this tile is drained: the volume streams through the L2, so these loads are DRAM
        // misses, and fetched at the top of their own tile they put ~0.9 us into every tile of the slowest epilogue warp --
        // which sets the tile period (corr_trace, round 2)
        float inv_a = 1.f, inv_b = 1.f;
        int tile = tile_of(0), b = 0, mb = 0, nb = 0;
        if (CL == 1 && tile < p.total_tiles) decode_tile(p, tile, b, mb, nb);
        int tile_nx = tile, b_nx = b, mb_nx = mb, nb_nx = nb;      // the tile after this one (CL == 1)
        if (CL == 1) advance(0, tile_nx, b_nx, mb_nx, nb_nx);
        if (F16 && tile < p.total_tiles) {
            inv_a = __ldg(p.inv_scale + b);
            inv_b = __ldg(p.inv_scale + p.B + b);
        }
        auto next_tile = [&]() {
            ++tile_no;
            if (CL == 2) { tile = tile_of(tile_no); return; }
            tile = tile_nx; b = b_nx; mb = mb_nx; nb = nb_nx;
            advance(tile_no, tile_nx, b_nx, mb_nx, nb_nx);
        };
        for (; tile < p.total_tiles; next_tile()) {
            if (CL == 2) decode_pair_tile(p, tile, rank, b, mb, nb);
            const int i = mb * BM + row;
            const bool row_ok = i < p.N;
            const float scale = F16 ? p.scale * inv_a * inv_b : p.scale;
            if (F16 && tile_nx < p.total_tiles) {
                inv_a = __ldg(p.inv_scale + b_nx);
                inv_b = __ldg(p.inv_scale + p.B + b_nx);
            }
            if (CL == 1 && nb >= p.tiles_n) continue;   // (quad3: padding index -- after the look-ahead, which every index owes its successor)
            mbar_wait(&tfull[acc], acc_phase);
            tc_fence_after();
            if (tile_no == 0 && threadIdx.x == 0) stamp(20);
            if (threadIdx.x == 0) TC_TRACE(tile_no, 12);
            if (p.ablate & 16) {  // experiment: the epilogue reads nothing (MMA issue rate without TMEM read traffic)
                tc_fence_before();
                if (CL == 2) mbar_arrive_cluster(mapa_rank0(&tempty[acc]));
                else mbar_arrive(&tempty[acc]);
                acc ^= 1;
                if (acc == 0) acc_phase ^= 1;
                continue;
            }
            const uint32_t taddr = tmem_base + ((uint32_t)(32 * quarter) << 16) + (uint32_t)acc * MAX_BN;
            const int j0 = nb * p.BN;
            const int bn_valid = min(p.BN, p.N - j0);  // accumulator column c <-> target index j0 + c
            // ---- level 0: TMEM -> registers (x scale) -> swizzled smem box -> TMA bulk store.
            // A warp-wide st.global of this fragment would touch 32 different rows per instruction
            // (measured: 18k cycles per tile); the TMA writes whole 128-byte lines instead.
            if constexpr (HO) {
                __half *l0h = reinterpret_cast<__half *>(p.l0);
                if (bn_valid >= 64) {
                    // ---- fp16 level 0: two 32-column chunks -> one 4 KB image of 32 rows x 64 halves (128-byte rows, the
                    // swizzle of the fp32 box) -> one {64 x 32} store box.  The last box overlaps its neighbour (same values).
                    const int nboxes = (bn_valid + 63) / 64;
                    for (int ci = half; ci < nboxes; ci += EPI_SPLIT) {
                        const int c0 = min(ci * 64, bn_valid - 64);
                        uint32_t v[32], u[32];
                        tmem_ld32(taddr + c0, v);
                        tmem_ld32(taddr + c0 + 32, u);
                        tmem_ld_wait();
                        uint8_t *buf = my_epi + (chunk_count & 1) * EPI_BUF_BYTES;
                        if (chunk_count >= 2) {  // the store issued two boxes ago has finished reading this buffer
                            if (lane == 0) tma_store_wait_read<1>();
                            __syncwarp();
                        }
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const uint4 o = make_uint4(pack_half2(__uint_as_float(v[8 * q]) * scale, __uint_as_float(v[8 * q + 1]) * scale),
                                                       pack_half2(__uint_as_float(v[8 * q + 2]) * scale, __uint_as_float(v[8 * q + 3]) * scale),
                                                       pack_half2(__uint_as_float(v[8 * q + 4]) * scale, __uint_as_float(v[8 * q + 5]) * scale),
                                                       pack_half2(__uint_as_float(v[8 * q + 6]) * scale, __uint_as_float(v[8 * q + 7]) * scale));
                            *reinterpret_cast<uint4 *>(buf + lane * 128 + ((q ^ (lane & 7)) << 4)) = o;
                        }
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const uint4 o = make_uint4(pack_half2(__uint_as_float(u[8 * q]) * scale, __uint_as_float(u[8 * q + 1]) * scale),
                                                       pack_half2(__uint_as_float(u[8 * q + 2]) * scale, __uint_as_float(u[8 * q + 3]) * scale),
                                                       pack_half2(__uint_as_float(u[8 * q + 4]) * scale, __uint_as_float(u[8 * q + 5]) * scale),
                                                       pack_half2(__uint_as_float(u[8 * q + 6]) * scale, __uint_as_float(u[8 * q + 7]) * scale));
                            *reinterpret_cast<uint4 *>(buf + lane * 128 + (((q + 4) ^ (lane & 7)) << 4)) = o;
                        }
                        fence_async_smem();
                        __syncwarp();
                        if (lane == 0) {
                            if (mb * BM + 32 * quarter < p.N && !(p.ablate & 1))
                                tma_store_3d(&tmap_c, buf, j0 + c0, mb * BM + 32 * quarter, b);
                            tma_store_commit();   // one bulk group per box, empty or not (see the fp32 chunks below)
                        }
                        ++chunk_count;
                    }
                } else if (half == 0) {
                    // tiles narrower than one box (maps of fewer than 64 targets, short last tiles): each lane its own row
                    const int vec0 = half_vec(l0h, p.N, j0);
                    __half *l0row = l0h + ((size_t)b * p.N + (row_ok ? i : 0)) * p.N + j0;
                    for (int c0 = 0; c0 < bn_valid; c0 += 32) {
                        uint32_t v[32];
                        tmem_ld32(taddr + c0, v);
                        tmem_ld_wait();
                        float o[32];
#pragma unroll
                        for (int q = 0; q < 32; ++q) o[q] = round_half(__uint_as_float(v[q]) * scale);
                        if (row_ok && !(p.ablate & 1)) store_halves<32>(l0row + c0, o, min(32, bn_valid - c0), vec0, p.stream_l0 != 0);
                    }
                }
            } else if (p.frag_stores && bn_valid == p.BN && !(p.ablate & 64)) {
                // ---- level 0 straight from registers: the 16x256b fragment gives four neighbouring threads one 32-byte run of
                // a row, so a warp-wide st.global.v2 writes eight whole sectors -- no staging in shared memory, no fence, and
                // no store box in the TMA unit, which then carries only the operand stages (write_probe: loads + these stores
                // 4.1 TB/s against 3.6 with the twenty boxes).  MEASURED SLOWER in the kernel (64 x 60x80, same box: 2565-2600 against
                // 2222-2227 us): the LSU already carries the level-1 and level-2 rows.  Experiment, flags bit26, parity-tested.
                for (int ci = half; ci < p.BN / 32; ci += EPI_SPLIT) {
#pragma unroll
                    for (int hr = 0; hr < 2; ++hr) {
                        uint32_t v[16];
                        tmem_ld_16x256b_x4(tmem_base + ((uint32_t)(32 * quarter + 16 * hr) << 16) + (uint32_t)acc * MAX_BN + (uint32_t)(32 * ci), v);
                        tmem_ld_wait();
                        const int r = mb * BM + 32 * quarter + 16 * hr + (lane >> 2);
                        float *dst = p.l0 + ((size_t)b * p.N + r) * p.N + j0 + 32 * ci + 2 * (lane & 3);
                        if (!(p.ablate & 1)) {
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const float2 lo = make_float2(__uint_as_float(v[4 * j]) * scale, __uint_as_float(v[4 * j + 1]) * scale);
                                const float2 hi = make_float2(__uint_as_float(v[4 * j + 2]) * scale, __uint_as_float(v[4 * j + 3]) * scale);
                                float2 *d0 = reinterpret_cast<float2 *>(dst + 8 * j), *d1 = reinterpret_cast<float2 *>(dst + (size_t)8 * p.N + 8 * j);
                                if (r < p.N) { if (p.stream_l0) __stcs(d0, lo); else *d0 = lo; }
                                if (r + 8 < p.N) { if (p.stream_l0) __stcs(d1, hi); else *d1 = hi; }
                            }
                        }
                    }
                }
            } else if (p.qbox && !(p.ablate & 64)) {
                // ---- level 0, one box per lane quarter: the SM's TMA unit carries the operand stages and the volume's stores
                // and is ~90 % busy (profiles/r02/write_probe.txt, corr_trace_f16_8x60x80.txt); twenty {32 x 32} boxes per tile cost
                // it 2.4 us, four {32 x 32 x 5} boxes 1.5 us.  The two warps of the quarter stage their chunks (same swizzled
                // 4 KB images as below) side by side, meet, and one lane stores all of them.
                uint8_t *qb = epi + quarter * (p.BN / 32) * EPI_BUF_BYTES;
                const bool issuer = half == 0 && lane == 0;
                if (issuer) tma_store_wait_read<0>();      // the previous tile's box has left the buffer
                quarter_barrier(quarter);
                // chunks [0, qbox_h0) to the first warp, the rest to the second (which also takes the odd pooling strip)
                for (int ci = half ? p.qbox_h0 : 0; ci < (half ? p.BN / 32 : p.qbox_h0); ++ci) {
                    uint32_t v[32];
                    tmem_ld32(taddr + 32 * ci, v);
                    tmem_ld_wait();
                    uint8_t *buf = qb + ci * EPI_BUF_BYTES;
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const float4 o = make_float4(__uint_as_float(v[4 * q]) * scale, __uint_as_float(v[4 * q + 1]) * scale,
                                                     __uint_as_float(v[4 * q + 2]) * scale, __uint_as_float(v[4 * q + 3]) * scale);
                        *reinterpret_cast<float4 *>(buf + lane * 128 + ((q ^ (lane & 7)) << 4)) = o;
                    }
                }
                fence_async_smem();
                quarter_barrier(quarter);
                if (issuer) {
                    if (mb * BM + 32 * quarter < p.N && !(p.ablate & 1))
                        tma_store_3d(&tmap_c, qb, 0, b * p.N + mb * BM + 32 * quarter, j0 >> 5);
                    tma_store_commit();
                }
            } else if (bn_valid >= 32 && !(p.ablate & 64)) {
                const int nchunks = (bn_valid + 31) / 32;
                for (int ci = half; ci < nchunks; ci += EPI_SPLIT) {
                    const int c0 = min(ci * 32, bn_valid - 32);  // last chunk overlaps its neighbour (same values)
                    uint32_t v[32];
                    tmem_ld32(taddr + c0, v);
                    tmem_ld_wait();
                    uint8_t *buf = my_epi + (chunk_count & 1) * EPI_BUF_BYTES;
                    if (p.lsu_stores) {
                        // transpose through the (swizzled) buffer, then whole 128-byte rows with plain vector stores:
                        // lane <-> (row = 4*it + lane/8, 16-byte piece = lane%8), four rows per instruction.  These go
                        // through the LSU, not the TMA unit, so the operand loads never queue behind the volume's
                        // HBM-paced write stream (with TMA bulk stores the tile period was store time + MMA time)
                        __syncwarp();   // the previous chunk's reads of this buffer (two chunks ago) are done
#pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const float4 o = make_float4(__uint_as_float(v[4 * q]) * scale, __uint_as_float(v[4 * q + 1]) * scale,
                                                         __uint_as_float(v[4 * q + 2]) * scale, __uint_as_float(v[4 * q + 3]) * scale);
                            *reinterpret_cast<float4 *>(buf + lane * 128 + ((q ^ (lane & 7)) << 4)) = o;
                        }
                        __syncwarp();
                        const int piece = lane & 7;
                        float *dst0 = p.l0 + ((size_t)b * p.N + (size_t)(mb * BM + 32 * quarter)) * p.N + j0 + c0 + 4 * piece;
                        float4 rowv[8];
#pragma unroll
                        for (int it = 0; it < 8; ++it) {
                            const int r = 4 * it + (lane >> 3);
                            rowv[it] = *reinterpret_cast<const float4 *>(buf + r * 128 + ((piece ^ (r & 7)) << 4));
                        }
                        if (!(p.ablate & 1)) {
#pragma unroll
                            for (int it = 0; it < 8; ++it) {
                                const int r = 4 * it + (lane >> 3);
                                if (mb * BM + 32 * quarter + r < p.N) {
                                    float4 *d = reinterpret_cast<float4 *>(dst0 + (size_t)r * p.N);
                                    if (p.stream_l0) __stcs(d, rowv[it]); else *d = rowv[it];
                                }
                            }
                        }
                        ++chunk_count;
                        continue;
                    }
                    if (chunk_count >= 2) {  // the store issued two chunks ago has finished reading this buffer
                        if (lane == 0) tma_store_wait_read<1>();
                        __syncwarp();
                    }
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const float4 o = make_float4(__uint_as_float(v[4 * q]) * scale, __uint_as_float(v[4 * q + 1]) * scale,
                                                     __uint_as_float(v[4 * q + 2]) * scale, __uint_as_float(v[4 * q + 3]) * scale);
                        *reinterpret_cast<float4 *>(buf + lane * 128 + ((q ^ (lane & 7)) << 4)) = o;
                    }
                    fence_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        if (mb * BM + 32 * quarter < p.N && !(p.ablate & 1))   // (rows below the volume: nothing to store)
                            tma_store_3d(&tmap_c, buf, j0 + c0, mb * BM + 32 * quarter, b);
                        // one bulk group per chunk, empty when nothing was stored: the wait_read<1> above counts groups, and
                        // a skipped commit let a chunk overwrite a buffer whose store was still reading it (the last query
                        // tile's rows below the volume, then a store of the next tile: zeros in the earlier tile's box)
                        tma_store_commit();
                    }
                    ++chunk_count;
                }
            } else if (half == 0) {
                float *l0row = p.l0 + ((size_t)b * p.N + (row_ok ? i : 0)) * p.N;
                uint32_t v[32];
                tmem_ld32(taddr, v);
                tmem_ld_wait();
                if (row_ok && bn_valid > 0) store_row_chunk(l0row + j0, v, scale, bn_valid, vec4_l0 && (bn_valid % 4 == 0), false);
            }
            if (threadIdx.x == 0) TC_TRACE(tile_no, 13);
            // ---- level 1: 2x2 means straight from the accumulator rows
            if (p.R != 0 && !(p.ablate & 32)) {
                const int y0 = nb * p.R;
                float *l1map = p.l1 + ((size_t)b * p.N + (row_ok ? i : 0)) * p.h1 * p.w1;
                float prev1[16], prev2[8];   // deep fusion: the previous level-1 / level-2 row of this query
                int item = EPI_SPLIT - 1;  // an odd chunk count leaves the last warp of a quarter one item short: it starts here
                for (int pr = 0; pr < p.R; pr += 2) {
                    const int y = y0 + pr;
                    if (y + 1 >= p.h) break;  // warp-uniform
                    for (int xc = 0; xc < p.w; xc += 32) {
                        if (((item++) % EPI_SPLIT) != half) continue;
                        uint32_t ra[32], rc[32];
                        tmem_ld32(taddr + pr * p.w + xc, ra);
                        tmem_ld32(taddr + (pr + 1) * p.w + xc, rc);
                        tmem_ld_wait();
                        // ATen avg_pool2d: ((a + b) + c) + d, then / 4, on the stored (scaled) values
                        float o[16];
                        if constexpr (HO) {   // from the stored (rounded) level-0 values, ((a + b) + c) + d, x 0.25, rounded
#pragma unroll
                            for (int q = 0; q < 16; ++q) {
                                float s = round_half(__uint_as_float(ra[2 * q]) * scale) + round_half(__uint_as_float(ra[2 * q + 1]) * scale);
                                s += round_half(__uint_as_float(rc[2 * q]) * scale);
                                s += round_half(__uint_as_float(rc[2 * q + 1]) * scale);
                                o[q] = round_half(s * 0.25f);
                            }
                            if (row_ok && !(p.ablate & 1))
                                store_halves<16>(reinterpret_cast<__half *>(p.l1) + ((size_t)b * p.N + i) * p.h1 * p.w1 + (size_t)(y >> 1) * p.w1 + (xc >> 1),
                                                 o, min(16, p.w1 - (xc >> 1)), half_vec(p.l1, p.h1 * p.w1, p.w1), false);
                        } else {
#pragma unroll
                        for (int q = 0; q < 16; ++q) {
                            float s = __uint_as_float(ra[2 * q]) * scale + __uint_as_float(ra[2 * q + 1]) * scale;
                            s += __uint_as_float(rc[2 * q]) * scale;
                            s += __uint_as_float(rc[2 * q + 1]) * scale;
                            o[q] = s * 0.25f;
                        }
                        if (p.l1_staged && p.w1 - (xc >> 1) >= 8) {   // (a narrow last strip is not worth the round trip)
                            // the lane's 16 values (64 B of ITS row) -> shared memory -> whole 64-byte runs, 8 rows per
                            // store instruction (lane <-> row 8*it + lane/4, piece lane%4) instead of 32 rows x 16 B
                            const int npool = min(16, p.w1 - (xc >> 1));
                            float *stg = p.l1_scratch ? reinterpret_cast<float *>(epi + p.l1_scratch + warp * 2048)
                                                      : reinterpret_cast<float *>(my_epi);
                            if (!p.l1_scratch && !p.lsu_stores && lane == 0) tma_store_wait_read<0>();   // the level-0 boxes have left the buffers
                            __syncwarp();
#pragma unroll
                            for (int q = 0; q < 4; ++q)
                                *reinterpret_cast<float4 *>(stg + lane * 16 + 4 * ((q + (lane >> 1)) & 3)) =
                                    make_float4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
                            __syncwarp();
                            const int row0 = mb * BM + 32 * quarter;
                            if (vec4_l1) {
                                const int pc = lane & 3;
#pragma unroll
                                for (int it = 0; it < 4; ++it) {
                                    const int rr = 8 * it + (lane >> 2);
                                    const float4 val = *reinterpret_cast<const float4 *>(stg + rr * 16 + 4 * ((pc + (rr >> 1)) & 3));
                                    if (row0 + rr < p.N && 4 * pc < npool && !(p.ablate & 1))
                                        *reinterpret_cast<float4 *>(p.l1 + ((size_t)b * p.N + row0 + rr) * p.h1 * p.w1 +
                                                                    (size_t)(y >> 1) * p.w1 + (xc >> 1) + 4 * pc) = val;
                                }
                            } else {   // w1 even but not a multiple of 4: rows are only 8-byte aligned -> float2 pieces, 4 rows per store
                                const int pc = lane & 7;
#pragma unroll
                                for (int it = 0; it < 8; ++it) {
                                    const int rr = 4 * it + (lane >> 3);
                                    const float2 val = *reinterpret_cast<const float2 *>(
                                        stg + rr * 16 + 4 * (((pc >> 1) + (rr >> 1)) & 3) + 2 * (pc & 1));
                                    if (row0 + rr < p.N && 2 * pc < npool && !(p.ablate & 1))
                                        *reinterpret_cast<float2 *>(p.l1 + ((size_t)b * p.N + row0 + rr) * p.h1 * p.w1 +
                                                                    (size_t)(y >> 1) * p.w1 + (xc >> 1) + 2 * pc) = val;
                                }
                            }
                            __syncwarp();
                        } else if (row_ok && !(p.ablate & 1)) {
                            float *dst = l1map + (size_t)(y >> 1) * p.w1 + (xc >> 1);
                            const int npool = min(16, p.w1 - (xc >> 1));
                            if (vec4_l1) {
#pragma unroll
                                for (int q = 0; q < 4; ++q)
                                    if (4 * q < npool)
                                        *(reinterpret_cast<float4 *>(dst) + q) = make_float4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
                            } else {
#pragma unroll
                                for (int q = 0; q < 8; ++q)
                                    if (2 * q < npool) *(reinterpret_cast<float2 *>(dst) + q) = make_float2(o[2 * q], o[2 * q + 1]);
                            }
                        }
                        }
                        if (p.pair2) {
                            // level 2 across the tile pair: the first tile parks its level-1 strip in TMEM columns
                            // [BN_mma, BN_mma + w1) of stage 0's window (free: BN_mma + w1 <= 256), the second tile pools
                            // ATen-style ((a + b) + c) + d, / 4 and stores 8 level-2 values per query and strip
                            const uint32_t park = tmem_base + ((uint32_t)(32 * quarter) << 16) + (uint32_t)p.BN_mma + (uint32_t)(xc >> 1);
                            if ((nb & 1) == 0) {
                                uint32_t ov[16];
#pragma unroll
                                for (int q = 0; q < 16; ++q) ov[q] = __float_as_uint(o[q]);
                                tmem_st16(park, ov);
                            } else {
                                uint32_t pv[16];
                                tmem_ld16(park, pv);
                                float l2v[8];
#pragma unroll
                                for (int q = 0; q < 8; ++q) {
                                    float s2 = __uint_as_float(pv[2 * q]) + __uint_as_float(pv[2 * q + 1]);
                                    s2 += o[2 * q];
                                    s2 += o[2 * q + 1];
                                    l2v[q] = stored<HO>(s2 * 0.25f);
                                }
                                const int r2g = nb >> 1, n2 = min(8, p.w2 - (xc >> 2));
                                if constexpr (HO) {
                                    if (row_ok && r2g < p.h2 && !(p.ablate & 1))
                                        store_halves<8>(reinterpret_cast<__half *>(p.l2) + (((size_t)b * p.N + i) * p.h2 + r2g) * p.w2 + (xc >> 2),
                                                        l2v, n2, half_vec(p.l2, p.h2 * p.w2, p.w2), false);
                                } else if (row_ok && r2g < p.h2 && !(p.ablate & 1)) {
                                    float *d2 = p.l2 + (((size_t)b * p.N + i) * p.h2 + r2g) * p.w2 + (xc >> 2);   // w2 % 4 == 0
#pragma unroll
                                    for (int q = 0; q < 2; ++q)
                                        if (4 * q < n2)
                                            *(reinterpret_cast<float4 *>(d2) + q) = make_float4(l2v[4 * q], l2v[4 * q + 1], l2v[4 * q + 2], l2v[4 * q + 3]);
                                }
                                if constexpr (!HO) if (p.quad3) {
                                    // level 3 across the quad: the second tile parks this level-2 strip behind the level-1
                                    // park (16 columns per strip there, 8 per strip here), the fourth pools 4 level-3 values per query and strip
                                    const uint32_t park2 = tmem_base + ((uint32_t)(32 * quarter) << 16) + (uint32_t)(p.BN_mma + 16 * ((p.w + 31) >> 5)) + (uint32_t)(xc >> 2);
                                    if ((nb & 3) == 1) {
                                        uint32_t ov[8];
#pragma unroll
                                        for (int q = 0; q < 8; ++q) ov[q] = __float_as_uint(l2v[q]);
                                        tmem_st8(park2, ov);
                                    } else {
                                        uint32_t qv[8];
                                        tmem_ld8(park2, qv);
                                        const int r3g = nb >> 2, n3 = min(4, p.w3 - (xc >> 3));
                                        if (row_ok && r3g < p.h3 && !(p.ablate & 1)) {
                                            float *d3 = p.l3 + (((size_t)b * p.N + i) * p.h3 + r3g) * p.w3 + (xc >> 3);
#pragma unroll
                                            for (int q = 0; q < 4; ++q) {
                                                float s3 = __uint_as_float(qv[2 * q]) + __uint_as_float(qv[2 * q + 1]);
                                                s3 += l2v[2 * q];
                                                s3 += l2v[2 * q + 1];
                                                if (q < n3) d3[q] = s3 * 0.25f;
                                            }
                                        }
                                    }
                                }
                            }
                        }
                        if (p.deep) {   // w <= 32: this is the only 32-column strip of the row pair
                            // ATen avg_pool2d again, on the level-1 (then level-2) values just stored
                            const int r1g = y >> 1;
                            if (r1g & 1) {
                                float l2v[8];
#pragma unroll
                                for (int q = 0; q < 8; ++q) {
                                    float s2 = prev1[2 * q] + prev1[2 * q + 1];
                                    s2 += o[2 * q];
                                    s2 += o[2 * q + 1];
                                    l2v[q] = stored<HO>(s2 * 0.25f);
                                }
                                const int r2g = r1g >> 1;
                                if constexpr (HO) {
                                    if (row_ok && r2g < p.h2 && !(p.ablate & 1))
                                        store_halves<8>(reinterpret_cast<__half *>(p.l2) + (((size_t)b * p.N + i) * p.h2 + r2g) * p.w2, l2v, p.w2,
                                                        half_vec(p.l2, p.h2 * p.w2, p.w2), false);
                                } else if (row_ok && r2g < p.h2 && !(p.ablate & 1)) {
                                    float *d2 = p.l2 + (((size_t)b * p.N + i) * p.h2 + r2g) * p.w2;   // w2 is even
                                    if ((p.w2 & 3) == 0) {   // 16-byte aligned rows: w2 = 4 or 8
#pragma unroll
                                        for (int q = 0; q < 2; ++q)
                                            if (4 * q < p.w2)
                                                *(reinterpret_cast<float4 *>(d2) + q) = make_float4(l2v[4 * q], l2v[4 * q + 1], l2v[4 * q + 2], l2v[4 * q + 3]);
                                    } else {
#pragma unroll
                                        for (int q = 0; q < 4; ++q)
                                            if (2 * q < p.w2) *(reinterpret_cast<float2 *>(d2) + q) = make_float2(l2v[2 * q], l2v[2 * q + 1]);
                                    }
                                }
                                if (p.deep > 1) {
                                    if (r2g & 1) {
                                        const int r3g = r2g >> 1;
                                        float l3v[4];
#pragma unroll
                                        for (int q = 0; q < 4; ++q) {
                                            float s3 = prev2[2 * q] + prev2[2 * q + 1];
                                            s3 += l2v[2 * q];
                                            s3 += l2v[2 * q + 1];
                                            l3v[q] = stored<HO>(s3 * 0.25f);
                                        }
                                        if constexpr (HO) {
                                            if (row_ok && r3g < p.h3 && !(p.ablate & 1))
                                                store_halves<4>(reinterpret_cast<__half *>(p.l3) + (((size_t)b * p.N + i) * p.h3 + r3g) * p.w3, l3v, p.w3,
                                                                half_vec(p.l3, p.h3 * p.w3, p.w3), false);
                                        } else if (row_ok && r3g < p.h3 && !(p.ablate & 1)) {
                                            float *d3 = p.l3 + (((size_t)b * p.N + i) * p.h3 + r3g) * p.w3;
                                            if (p.w3 == 4 && (reinterpret_cast<uintptr_t>(p.l3) & 15u) == 0) {
                                                *reinterpret_cast<float4 *>(d3) = make_float4(l3v[0], l3v[1], l3v[2], l3v[3]);
                                            } else {
#pragma unroll
                                                for (int q = 0; q < 4; ++q)
                                                    if (q < p.w3) d3[q] = l3v[q];
                                            }
                                        }
                                    } else {
#pragma unroll
                                        for (int q = 0; q < 8; ++q) prev2[q] = l2v[q];
                                    }
                                }
                            } else {
#pragma unroll
                                for (int q = 0; q < 16; ++q) prev1[q] = o[q];
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            if (CL == 2) mbar_arrive_cluster(mapa_rank0(&tempty[acc]));
            else mbar_arrive(&tempty[acc]);
            if (tile_no == 0 && threadIdx.x == 0) stamp(21);
            if (threadIdx.x == 0) TC_TRACE(tile_no, 14);
            if (kblocks <= 2 && lane == 0 && warp > 0) TC_TRACE(tile_no, warp == 3 ? 15 : (warp < 3 ? 4 + warp : 3 + warp));   // (slots of K blocks 2.. are free: epilogue done, warps 1,2 -> 5,6; 4..7 -> 7..10; 3 -> 15)
            acc ^= 1;
            if (acc == 0) acc_phase ^= 1;
        }
    }
    if (warp < EPI_WARPS && lane == 0) tma_store_wait_all();  // bulk stores must drain before the CTA's smem goes away
    tc_fence_before();
    __syncthreads();
    __syncwarp();
    if (CL == 2) cluster_sync_all();  // the peer may still commit onto this CTA's barriers until its own loop ends
    if (warp == MMA_WARP) {
        tc_fence_after();
        if (CL == 2) tmem_dealloc_2sm(tmem_base, 512);
        else tmem_dealloc(tmem_base, 512);
    }
    if (threadIdx.x == 0) stamp(22);
}
