// The two lookup kernels (see corr_lookup.cu), included twice by corr_lookup.cu:
//   CF_LOOKUP_PYR = Pyramid,     CF_LOOKUP_T = float    corr_lookup_r4l4_kernel,      corr_lookup_kernel        (cf_corr_lookup)
//   CF_LOOKUP_PYR = PyramidHalf, CF_LOOKUP_T = __half   corr_lookup_r4l4_half_kernel, corr_lookup_half_kernel   (cf_corr_lookup_half)
// tap_ld widens an fp16 tap to fp32 as it is loaded; everything after the load is the same code.  (A textual include,
// not a shared __device__ function: the fp32 kernels compile to the same code as before the fp16 pyramid existed.)
template <int QT_CT>
__global__ void __launch_bounds__(kLookupThreads)
CF_LOOKUP_R4L4(const __grid_constant__ CF_LOOKUP_PYR pyr, const float *__restrict__ coords, float *__restrict__ out, int N,
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
                    const CF_LOOKUP_T *p = pyr.ptr[l] + ((size_t)b * N + q) * (Hl * Wl) + (Y * Wl + X);
                    asm volatile("" : "+l"(p));  // one 64-bit column address per (query, level); rows are p + 3k*Wl
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const bool ok = okx && (unsigned)(Y + 3 * k) < (unsigned)Hl && (k < 3 || rg == 0);
                        v[u][l * 4 + k] = ok ? tap_ld(p + 3 * k * Wl) : 0.f;
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
CF_LOOKUP_GENERIC(const __grid_constant__ CF_LOOKUP_PYR pyr, const float *__restrict__ coords, float *__restrict__ out,
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
            v = tap_ld(pyr.ptr[l] + (((size_t)b * N + q) * Hl + Y) * Wl + X);
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
