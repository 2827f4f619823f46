"""Event binning, its normalisation and the event ingest on every dispatch branch, element by element against float64.

The reference is one vectorised numpy restatement of bin_event and the weights (voxel_common.cuh) with the window
semantics of include/cistaflow.h: window b is rows [offsets[b], offsets[b+1]); rows outside [offsets[0], offsets[B])
belong to no window; x < 0, y < 0, x >= W, y >= H, NaN and floor(t*) outside [0, nb) are dropped.  t* is the fp64
operation sequence of the kernels ((nb-1) * (t - t0) / dT, or ((t - t0) / dT) * (nb-1) for MVSEC), so the reference has
the kernels' bins and fractions bit for bit.  The TORCH weights are restated in np.float32 bit for bit, the other
flavours' in float64.  (The C oracle voxel_seq.c keeps x in (-1, 0) through its integer cast; it is used only where
its semantics agree, in the CPU self-tests.)

Bounds (u = 2^-24, gamma(k) = k u / (1 - k u); gamma64 the same with 2^-53).  Each is asserted per cell, and a zero
bound demands an exact zero:
  * deterministic, all four flavours: bit-exact against the sequential restatement (per cell, the left weights in
    event order then the right ones; MVSEC: one pass per bin in event order; fp32 adds, or fp64 add and round).
  * atomic (L2, tiled), TORCH:  |got - ref| <= gamma(n-1) M, ref the float64 sum of the kernel's fp32 weights, n the
    number of adds into the cell and M their sum of magnitudes: n - 1 fp32 additions in any order.
  * atomic, NUMPY / POL / MVSEC:  (u + gamma(n-1)(1+u)) M, ref the float64 sum of the fp64 weights: every weight is
    rounded to fp32 once before the additions.
  * packed (cf_voxel_bin_packed): the atomic term plus L = sum over the events that can reach the cell of |s| dt*.
    dt* = 6u |t*| bounds the fp32 time normalisation against the fp64 one: t_rel and dT each round once in fp64 and
    once to fp32, then one fp32 mul and one fp32 div -- a relative error of at most 4u + 2^-51 + O(u^2).  An event's
    contribution to bin k is s * max(0, 1 - |t* - k|), 1-Lipschitz in t* and continuous across bins, including the drop
    past nb - 1 (the hat of bin nb-1 is 0 at t* = nb) -- so a change of t* by dt* moves every contribution by at most
    |s| dt*; sorted windows have t* >= 0 in both, so the drop below 0 is never crossed.  An event can reach bins
    floor(t*) - 1 .. floor(t*) + 2, and both n and M count those.
  * normalisation (fused in each path, and cf_voxel_preprocess), against float64 statistics of the float32 grid the
    same call produced (read back from a NONE call on inputs whose cell sums are exact in fp32 in any order, or from
    the deterministic grid) and a float64 map.  STD: the kernel forms a = fl(m), i = fl(1/(s + 1e-8)) from its fp64
    statistics m, s and maps fl(fl(v - a) * i).  Its statistics are fp64 sums of depth k (terms per thread plus the
    fixed trees), so |m - mean| <= em = gamma64(k) A1 / N + 2^-52 |mean| and the variance moves by
    ev = gamma64(k) A2 / N + 2 |mean| em + em^2 + 2^-51 (Q / N + mean^2), with A1 = sum |v|, A2 = sum v^2 (for the
    telescoped tiled statistics: the sums of |old| + |new| over all adds).  Then |s - std| <= es = min(sqrt(ev),
    ev / (2 std)), |i - inv| <= ei = es / (sd (sd - es)) + 2^-51 inv with sd = std + 1e-8, and
        |got - ref| <= (em + u(|mean| + em))(inv + ei) + |v - mean| ei + gamma(3)(|v - mean| + em + u(|mean| + em))(inv + ei).
    The k of the reference's own float64 sums is included.  MAXMIN: min and max are exact, |got - ref| <= gamma(3) |ref|
    + 2^-50 |ref|.  A window with no non-zero cell is the identity, and cells the hot-pixel filter zeroes are 0: exact.
  * cf_events_pack, cf_events_filter, cf_event_window_offsets: bit-exact against numpy / Python round / np.array_split.

Outputs go into NaN-filled views with guard regions (guarded_buffers.py).  Every row names its branch and proves it:
cf_last_kernel() and the return code, the number of launches where it tells the branches apart (radix passes, L2
chunks), and the restated host predicates (stat_geometry of voxel.cu, geometry of voxel_tiled.cu, the L2 chunking of
cf_voxel_bin) where the kernel name is not enough."""
import math
import os
import zlib

import numpy as np
import pytest
import torch

from guarded_buffers import assert_written_and_guarded, guarded

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32
U = 2.0 ** -24
U64 = 2.0 ** -53
TORCH, NUMPY, POL, MVSEC = 0, 1, 2, 3
ATOMIC, DET, L2, TILED = 0, 1, 2, 3
NONE, STD, MAXMIN = 0, 1, 2
FIXED, SPLIT = 0, 1
OK, INVALID_ARG, UNSUPPORTED = 0, -1, -7
SMS = 148                      # B200
K_MAX_CHUNKS = 512             # voxel_common.cuh
CHUNK, MAX_T, TILE_BYTES_MAX = 2048, 1024, 108 * 1024   # voxel_tiled.cu
L2_CHUNK_BYTES = 96 << 20      # voxel.cu kL2ChunkBytes
FLAVOURS = {TORCH: "torch", NUMPY: "numpy", POL: "pol", MVSEC: "mvsec"}


def seed(*parts):
    return zlib.crc32(repr(parts).encode())


def gamma(k, u=U):
    k = np.maximum(np.asarray(k, np.float64), 0.0)
    return k * u / (1.0 - k * u)


def ceil_div(a, b):
    return -(-a // b)


# ------------------------------------------------------------------------------------------ restated predicates ---
def stat_geometry(B, cells):
    """voxel.cu stat_geometry: (chunks, chunk_len) of the statistics / normalise kernels."""
    want = ceil_div(8 * 148, B if B > 0 else 1)
    cap = ceil_div(cells, 2048)
    chunks = max(want, 1)
    if chunks > cap:
        chunks = max(cap, 1)
    chunks = min(chunks, K_MAX_CHUNKS)
    chunk_len = ceil_div(cells, chunks)
    return chunks, (chunk_len + 3) & ~3


def stat_depth(B, cells):
    """Additions along the longest path of voxel_stats_kernel + voxel_normalise_kernel: the terms of one thread, the
    warp and CTA trees, the per-lane chunk loop and its warp tree; +160 for the reference's own pairwise sums."""
    chunks, chunk_len = stat_geometry(B, cells)
    return chunk_len // 256 + 4 + 5 + 8 + ceil_div(chunks, 32) + 5 + 160


def tiled_geometry(total, B, nb, H, W, flavour, sms=SMS):
    """voxel_tiled.cu geometry: None when the tiled path does not cover the shape, else dict(P, T, max_c)."""
    HW = H * W
    planes = nb * (2 if flavour == POL else 1)
    if B < 1 or B > (1 << 20) or HW >= (1 << 28) or total < 0:
        return None
    pmax = (TILE_BYTES_MAX // (4 * planes)) & ~3
    if pmax < 64:
        return None
    t0 = ceil_div(HW, pmax)
    want = min(ceil_div(2 * sms, B), CHUNK // 16, HW // 256)
    T = max(t0, want, 1)
    P = (ceil_div(HW, T) + 3) & ~3
    T = ceil_div(HW, P)
    if T > MAX_T or 2 * planes * P * 4 > 2 * TILE_BYTES_MAX or T > 2 * sms:
        return None
    mc = min(max(ceil_div(ceil_div(total if total > 0 else 1, B), CHUNK), 1), 65536)
    return dict(P=P, T=T, t0=t0, want=want, max_c=mc)


def l2_chunk(total, B, cells):
    """Windows per L2-resident chunk of cf_voxel_bin's atomic path."""
    per_window = cells * 4 + (total // B + 1) * 32
    return max(1, min(B, L2_CHUNK_BYTES // per_window))


def window_offsets_ref(n, policy, param, max_windows):
    """cf_event_window_offsets restated: (offsets [max_windows + 1], n_windows)."""
    if policy == FIXED:
        k = ceil_div(n, param)
    else:
        k = max(1, round(n / param))           # Python round: half to even
    k = min(k, max_windows)
    if policy == FIXED:
        o = [min(i * param, n) for i in range(k)]
    else:
        sizes = [len(a) for a in np.array_split(np.arange(n), k)]
        o = list(np.concatenate([[0], np.cumsum(sizes)])[:k])
    return np.array(o + [n] * (max_windows + 1 - k), np.int64), k


# ------------------------------------------------------------------------------------------- float64 reference ---
def binned(ev, off, nb, H, W, flavour):
    """bin_event of every row with window semantics: dict of per-row arrays (fp64 t*, floor, fraction, sign, ...)."""
    ev = np.asarray(ev, np.float64)
    n = len(ev)
    off = np.asarray(off, np.int64)
    win = np.full(n, -1, np.int64)
    t0 = np.zeros(n)
    span = np.ones(n)
    for b in range(len(off) - 1):
        s, e = int(off[b]), int(off[b + 1])
        if e > s:
            win[s:e] = b
            t0[s:e] = ev[s, 0]
            sp = ev[e - 1, 0] - ev[s, 0]
            span[s:e] = 1.0 if sp == 0.0 else sp
    t, x, y, p = ev.T if n else (np.zeros(0),) * 4
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        d = t - t0
        tn = (d / span) * float(nb - 1) if flavour == MVSEC else (float(nb - 1) * d) / span
        lo = np.floor(tn)
        ok = (win >= 0) & (lo >= 0) & (lo < nb) & (x >= 0) & (y >= 0) & (x < W) & (y < H)
        if flavour == POL:
            ok &= (p >= 0) & (p < 2)
        dt = tn - lo
    if flavour == POL:
        sgn = np.where(p == 0, 1.0, p)
    elif flavour == MVSEC:
        sgn = p.copy()
    else:
        sgn = np.where(p == 0, -1.0, p)
    z = np.zeros(n, np.int64)
    return dict(ok=ok, win=np.where(ok, win, 0), lo=np.where(ok, lo, 0).astype(np.int64), dt=np.where(ok, dt, 0.0),
                tn=np.where(ok, tn, 0.0), sgn=np.where(ok, sgn, 0.0),
                x=np.where(ok, x, 0).astype(np.int64) if n else z, y=np.where(ok, y, 0).astype(np.int64) if n else z,
                chan=np.where(ok, p, 0).astype(np.int64) if (n and flavour == POL) else z)


def weights(r, flavour):
    """(left, right) weights as the kernels form them: float32 for TORCH, float64 otherwise."""
    if flavour == TORCH:
        s, f = r["sgn"].astype(F32), r["dt"].astype(F32)
        return (s * (F32(1) - f)).astype(F32), (s * f).astype(F32)
    if flavour == MVSEC:
        om = 1.0 - r["dt"]
        return r["sgn"] * om, r["sgn"] * (1.0 - om)
    return r["sgn"] * (1.0 - r["dt"]), r["sgn"] * r["dt"]


def grid_shape(B, nb, H, W, flavour):
    return (B, nb, 2, H, W) if flavour == POL else (B, nb, H, W)


def contributions(ev, off, nb, H, W, flavour):
    """Every add the binning makes: (flat cell, weight, sequential order key).  Weights as the kernels form them
    (TORCH float32, else float64)."""
    r = binned(ev, off, nb, H, W, flavour)
    n = len(ev)
    planes = 2 if flavour == POL else 1
    plane = H * W
    idx = np.arange(n)
    base = ((r["win"] * nb + r["lo"]) * planes + r["chan"]) * plane + r["y"] * W + r["x"]
    wl, wr = weights(r, flavour)
    L = r["ok"]
    R = r["ok"] & (r["lo"] + 1 < nb)
    key_r = idx if flavour == MVSEC else idx + n       # MVSEC: one pass per bin in event order; else left then right
    cell = np.concatenate([base[L], base[R] + planes * plane])
    w = np.concatenate([wl[L], wr[R]])
    key = np.concatenate([idx[L], key_r[R]])
    return cell, w, key


def seq_grid(ev, off, nb, H, W, flavour):
    """Deterministic mode restated: per cell, the adds in their sequential order, fp32 adds (TORCH; MVSEC adds
    fp32-cast weights) or fp64 add rounded to fp32 (NUMPY, POL).  Vectorised over cells, one round per add rank."""
    B = len(off) - 1
    shape = grid_shape(B, nb, H, W, flavour)
    out = np.zeros(math.prod(shape), F32)
    cell, w, key = contributions(ev, off, nb, H, W, flavour)
    if len(cell) == 0:
        return out.reshape(shape)
    if flavour == MVSEC:
        w = w.astype(F32)
    order = np.lexsort((key, cell))
    c, wv = cell[order], w[order]
    head = np.r_[True, c[1:] != c[:-1]]
    run = np.cumsum(head) - 1
    starts = np.flatnonzero(head)
    rank = np.arange(len(c)) - starts[run]
    by_rank = np.argsort(rank, kind="stable")
    acc = np.zeros(len(starts), F32)
    pos = 0
    for cnt in np.bincount(rank):
        sel = by_rank[pos:pos + cnt]
        pos += cnt
        ru = run[sel]
        if flavour in (NUMPY, POL):
            acc[ru] = (acc[ru].astype(np.float64) + wv[sel]).astype(F32)
        else:
            acc[ru] = acc[ru] + wv[sel]
    out[c[starts]] = acc
    return out.reshape(shape)


def atomic_ref(ev, off, nb, H, W, flavour):
    """(float64 grid, per-cell bound, adds per cell, sum |w| per cell) of the atomic paths."""
    B = len(off) - 1
    shape = grid_shape(B, nb, H, W, flavour)
    size = math.prod(shape)
    cell, w, _ = contributions(ev, off, nb, H, W, flavour)
    w = w.astype(np.float64)
    ref = np.zeros(size)
    M = np.zeros(size)
    np.add.at(ref, cell, w)
    np.add.at(M, cell, np.abs(w))
    n = np.bincount(cell, minlength=size).astype(np.float64)
    if flavour == TORCH:
        bound = gamma(n - 1) * M
    else:
        bound = (U + gamma(n - 1) * (1 + U)) * M
    return ref.reshape(shape), bound.reshape(shape), n.reshape(shape), M.reshape(shape)


def packed_ref(ev, off, nb, H, W):
    """cf_voxel_bin_packed against the fp64 events: (float64 grid, per-cell bound).  Sign +1 for p > 0, else -1."""
    evs = np.array(ev, np.float64, copy=True)
    evs[:, 3] = np.where(evs[:, 3] > 0, 1.0, 0.0)        # p -> +-1 through the NUMPY flavour's p == 0 -> -1
    B = len(off) - 1
    shape = (B, nb, H, W)
    size = math.prod(shape)
    ref, _, _, _ = atomic_ref(evs, off, nb, H, W, NUMPY)
    r = binned(evs, off, nb, H, W, NUMPY)
    wl, wr = weights(r, NUMPY)
    ok = r["ok"]
    dts = 6 * U * np.abs(r["tn"])
    pix = r["win"] * nb * H * W + r["y"] * W + r["x"]
    n = np.zeros(size)
    Mx = np.zeros(size)
    L = np.zeros(size)
    for k in (-1, 0, 1, 2):
        b = r["lo"] + k
        sel = ok & (b >= 0) & (b < nb)
        cell = pix[sel] + b[sel] * H * W
        wk = np.where(k == 0, np.abs(wl), np.where(k == 1, np.abs(wr), 0.0))[sel]
        np.add.at(n, cell, 1.0)
        np.add.at(Mx, cell, wk + dts[sel])
        np.add.at(L, cell, dts[sel])
    bound = (U + gamma(n - 1) * (1 + U)) * Mx + L
    return ref.reshape(shape), bound.reshape(shape)


def norm_ref(G, mode, thr, k, A1=None, A2=None):
    """float64 normalisation of one window's fp32 grid G and its per-cell bound (module docstring)."""
    g = np.array(G, F32, copy=True).reshape(-1)
    if thr > 0:
        g[np.abs(g) > F32(thr)] = 0
    v = g.astype(np.float64)
    if mode == MAXMIN:
        mn, mx = v.min(), v.max()
        ref = (v - mn) / (mx - mn + 1e-8)
        return ref, (gamma(3) + 2.0 ** -50) * np.abs(ref) * (1 + 1e-9)
    nz = v != 0
    N = int(nz.sum())
    if N == 0:
        return v, np.zeros_like(v)
    S, Q = v.sum(), (v * v).sum()
    mean = S / N
    var = Q / N - mean * mean
    std = math.sqrt(max(var, 0.0))
    sd = std + 1e-8
    inv = 1.0 / sd
    A1 = np.abs(v).sum() if A1 is None else A1
    A2 = Q if A2 is None else A2
    gk = float(gamma(k, U64))
    em = gk * A1 / N + 2 * U64 * abs(mean)
    ev_ = gk * A2 / N + 2 * abs(mean) * em + em * em + 4 * U64 * (Q / N + mean * mean)
    es = min(math.sqrt(ev_), ev_ / (2 * std) if std > 0 else math.inf)
    ref = np.where(nz, (v - mean) * inv, 0.0)
    if es >= sd:            # the spread is within the statistics' error: no finite bound (rows assert such cells)
        return ref, np.where(nz, np.inf, 0.0)
    ei = es / (sd * (sd - es)) + 4 * U64 * inv
    dv = np.abs(v - mean)
    da = em + U * (abs(mean) + em)
    bound = da * (inv + ei) + dv * ei + gamma(3) * (dv + da) * (inv + ei)
    return ref, np.where(nz, bound * (1 + 1e-9), 0.0)


# --------------------------------------------------------------------------------------------- event builders ---
T0 = 1.0e9     # absolute stamps: t - t0 is exact for the dyadic builders below


def dyadic_window(rng, n, nb, H, W, pmode="01"):
    """n sorted events with t* = t - T0 a multiple of 1/8 in [0, nb-1] (first at 0, last at nb-1): every weight is a
    multiple of 1/8 and every cell sum is exact in fp32, in any order -- and, with nb - 1 a power of two, in the fp32
    time normalisation of the packed path too."""
    tt = np.sort(rng.integers(0, 8 * (nb - 1) + 1, n)) / 8.0
    if n >= 2:
        tt[0], tt[-1] = 0.0, float(nb - 1)
    x = rng.integers(0, W, n).astype(np.float64)
    y = rng.integers(0, H, n).astype(np.float64)
    p = rng.integers(0, 2, n).astype(np.float64)
    return np.stack([T0 + tt, x, y, p], axis=1)


def random_window(rng, n, H, W, p_values=(0.0, 1.0)):
    t = T0 + np.sort(rng.random(n)) * 5.0e4
    x = rng.integers(0, W, n) + rng.random(n) * 0.999
    y = rng.integers(0, H, n) + rng.random(n) * 0.999
    p = rng.choice(np.asarray(p_values, np.float64), n)
    return np.stack([t, x, y, p], axis=1)


def concat(windows, lead=None, tail=None):
    parts = ([lead] if lead is not None else []) + list(windows) + ([tail] if tail is not None else [])
    ev = np.concatenate(parts, axis=0) if parts else np.zeros((0, 4))
    first = 0 if lead is None else len(lead)
    off = np.r_[first, first + np.cumsum([len(w) for w in windows])].astype(np.int64)
    return np.ascontiguousarray(ev), off


def layout(name, rng, H, W, p_values=(0.0, 1.0)):
    """Window layouts: (events, offsets)."""
    if name == "lead_rows":          # offsets[0] > 0, the leading rows' stamps inside window 0's span, on its pixels
        w0 = random_window(rng, 300, H, W, p_values)
        lead = w0[rng.integers(1, 299, 40)].copy()
        lead[:, 0] = np.sort(lead[:, 0])
        return concat([w0, random_window(rng, 200, H, W, p_values)], lead=lead)
    if name == "tail_rows":          # rows past offsets[B]
        return concat([random_window(rng, 300, H, W, p_values), random_window(rng, 200, H, W, p_values)],
                      tail=random_window(rng, 77, H, W, p_values))
    if name == "empty_windows":      # empty first, in the middle and last
        z = np.zeros((0, 4))
        return concat([z, random_window(rng, 300, H, W, p_values), z, z, random_window(rng, 250, H, W, p_values), z])
    if name == "one_event_and_span0":
        one = random_window(rng, 1, H, W, p_values)
        same = random_window(rng, 120, H, W, p_values)
        same[:, 0] = T0 + 7.0                     # span 0 -> 1: every t* = 0
        return concat([one, same, random_window(rng, 200, H, W, p_values)])
    raise KeyError(name)


LAYOUTS = ["lead_rows", "tail_rows", "empty_windows", "one_event_and_span0"]


def edge_window(flavour, nb=5, H=6, W=7):
    """One window of edge events: t* on bin edges (dt = 0), the last at t* = nb-1, a stamp 2^-30 below an edge (TORCH:
    f32(dt) = 1, a +-0 left weight), x = W-1+0.999 (kept), x = W, -0.5 (dropped), -0.0 (kept), NaN in t and in x of
    middle rows, and every polarity of p_values(flavour)."""
    rows = []
    ps = [0.0, 1.0, -1.0, 0.5, 2.0, 1.5]
    k = 0

    def add(ts, x, y):
        nonlocal k
        rows.append([1000.0 + ts, x, y, ps[k % len(ps)]])     # small t0: 2^-30 below an edge is representable
        k += 1
    add(0.0, 0, 0)
    for ts in np.linspace(0, nb - 1, 4 * (nb - 1) + 1):     # quarter steps: bin edges and midpoints
        for x in (0.0, 3.5, W - 1 + 0.999, -0.0):
            add(ts, x, (k * 3) % H)
    add(2.0 - 2.0 ** -30, 1, 1)
    add(2.0 - 2.0 ** -30, 1, 1)
    add(2.5, float(W), 2)
    add(2.5, -0.5, 2)
    add(2.6, 3, float(H))
    add(float("nan"), 2, 2)
    add(2.7, float("nan"), 2)
    add(3.0, 2, 2)
    add(float(nb - 1), 4, 4)
    ev = np.array(rows)
    ev[1:-1] = ev[1:-1][np.argsort(ev[1:-1, 0], kind="stable")]      # sorted (NaN sorts last: move it inside)
    nan_rows = np.isnan(ev[:, 0])
    ev = np.concatenate([ev[~nan_rows][:-1], ev[nan_rows], ev[~nan_rows][-1:]])
    return ev


def unsorted(ev, rng):
    """The rows between the first and the last shuffled: t0 and dT stay, bin order along a pixel breaks."""
    ev = ev.copy()
    mid = ev[1:-1].copy()
    ev[1:-1] = mid[rng.permutation(len(mid))]
    return ev


def runs_not_monotone(ev, off, nb, H, W, flavour):
    """The restated predicate of det_accumulate_kernel's order-agnostic walk: some pixel column whose valid events'
    bins, in event order, decrease somewhere."""
    r = binned(ev, off, nb, H, W, flavour)
    planes = 2 if flavour == POL else 1
    col = ((r["win"] * planes + r["chan"]) * H + r["y"]) * W + r["x"]
    idx = np.flatnonzero(r["ok"])
    o = np.lexsort((idx, col[idx]))
    c, lo = col[idx][o], r["lo"][idx][o]
    return bool(np.any((c[1:] == c[:-1]) & (lo[1:] < lo[:-1])))


# ------------------------------------------------------------------------------------------- CPU self-tests ---
@pytest.mark.parametrize("flavour", [TORCH, NUMPY, POL])
@pytest.mark.parametrize("case", ["base", "dense_hot", "single", "two_same_t", "empty"])
def test_reference_reproduces_the_c_oracle_and_the_golden(golden, flavour, case):
    """The restatement equals voxel_seq.c and the voxel.npz golden bit for bit (in-grid events, p in {0, 1})."""
    from oracle import explicit
    g = golden("voxel")
    ev = g[f"{case}/events"]
    nb, w, h = (int(v) for v in g[f"{case}/dims"])
    mine = seq_grid(ev, [0, len(ev)], nb, h, w, flavour)[0]
    oracle = explicit.voxel_grid_sequential(ev, nb, w, h, flavour)
    assert np.array_equal(mine.view(np.uint32), oracle.view(np.uint32))
    assert np.array_equal(mine.view(np.uint32), g[f"{case}/{FLAVOURS[flavour]}"].view(np.uint32))


def test_reference_reproduces_the_c_oracle_on_random_windows():
    from oracle import explicit
    rng = np.random.default_rng(11)
    for flavour in (TORCH, NUMPY, POL):
        for n in (1, 2, 500, 3000):
            ev = random_window(rng, n, 9, 13, (0.0, 1.0, 0.25) if flavour != POL else (0.0, 1.0, 1.5))
            ev[rng.random(n) < 0.3, 1] = 4.0                # long runs on a few pixels
            mine = seq_grid(ev, [0, n], 5, 9, 13, flavour)[0]
            assert np.array_equal(mine.view(np.uint32), explicit.voxel_grid_sequential(ev, 5, 13, 9, flavour).view(np.uint32))


def test_reference_reproduces_the_mvsec_port():
    import torch as th
    from oracle import ref_port
    rng = np.random.default_rng(12)
    for n, nb in ((400, 5), (3000, 9), (2, 3)):
        ev = random_window(rng, n, 7, 11, (-1.0, 1.0, 0.5))
        got = seq_grid(ev, [0, n], nb, 7, 11, MVSEC)[0]
        want = ref_port.mvsec_voxel_torch(th.from_numpy(ev[:, 1]), th.from_numpy(ev[:, 2]), th.from_numpy(ev[:, 0]),
                                          th.from_numpy(ev[:, 3]), nb, 7, 11).numpy()
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("mode", ["std", "maxmin"])
@pytest.mark.parametrize("thr", [0.0, 1.0])
def test_normalisation_reference_agrees_with_explicit_preprocess(mode, thr):
    from oracle import explicit
    rng = np.random.default_rng(13)
    g = seq_grid(random_window(rng, 4000, 30, 40), [0, 4000], 5, 30, 40, NUMPY)[0]
    ref, bound = norm_ref(g, STD if mode == "std" else MAXMIN, thr, 200)
    want = explicit.preprocess(g, mode, thr).reshape(-1)
    assert np.array_equal(ref.astype(F32), want)
    assert (bound >= 0).all() and np.isfinite(bound).all()


def test_restated_host_predicates():
    """Hand-computed cases of stat_geometry (voxel.cu), the tiled geometry (voxel_tiled.cu) and the window offsets."""
    assert stat_geometry(1, 5 * 480 * 640) == (512, 3000)          # the 512-chunk cap
    assert stat_geometry(64, 5 * 480 * 640) == (19, 80844)         # 315 terms per thread
    assert stat_geometry(1184, 5 * 480 * 640) == (1, 1536000)
    assert stat_geometry(1, 5) == (1, 8)
    assert stat_geometry(3, 5735) == (3, 1912)
    g = tiled_geometry(64 * 100000, 64, 5, 480, 640, TORCH)
    assert g["T"] == 56 and g["P"] == 5488 and g["want"] == 5           # the window's size sets the tiles
    g = tiled_geometry(100000, 1, 5, 480, 640, TORCH)
    assert g["want"] == 128 and g["T"] == 128 and g["P"] == 2400        # small batch: more, smaller tiles
    assert tiled_geometry(300 * 200, 300, 5, 30, 40, TORCH)["T"] == 1
    assert tiled_geometry(10, 1, 5, 2000, 2000, TORCH) is None          # T = 724 > 2 * 148
    assert tiled_geometry(20300, 4, 5, 30, 40, TORCH)["max_c"] == 3
    o, k = window_offsets_ref(5, SPLIT, 2, 8)                            # 2.5 -> 2 (half to even)
    assert k == 2 and list(o) == [0, 3, 5, 5, 5, 5, 5, 5, 5]
    o, k = window_offsets_ref(7, SPLIT, 2, 8)                            # 3.5 -> 4
    assert k == 4 and list(o[:5]) == [0, 2, 4, 6, 7]
    o, k = window_offsets_ref(1000, FIXED, 100, 4)                       # clamped: the last window keeps the rest
    assert k == 4 and list(o) == [0, 100, 200, 300, 1000]
    o, k = window_offsets_ref(1000, SPLIT, 100, 4)                       # clamped: an even split over 4 windows
    assert k == 4 and list(o) == [0, 250, 500, 750, 1000]
    assert window_offsets_ref(0, FIXED, 10, 3)[1] == 0 and window_offsets_ref(0, SPLIT, 10, 3)[1] == 1
    c, cl = stat_geometry(1, SHORT_TAIL_CELLS)
    assert c == 498 and cl == 2048 and SHORT_TAIL_CELLS - (c - 1) * cl == 60
    # No geometry has an EMPTY trailing chunk: that needs cells <= 4 c (c - 1) (chunk_len rounds up by < 4), while
    # c <= ceil(cells / 2048) and c <= 512 keep cells > 2048 (c - 1) >= 4 c (c - 1).  Sampled here.
    for B in (1, 3, 64, 1184):
        for cells in range(1, 1 << 21, 997):
            c, cl = stat_geometry(B, cells)
            assert (c - 1) * cl < cells <= c * cl


SHORT_TAIL_CELLS = 1017916     # B = 1: 498 chunks of 2048 cells, the last one holds 60 (15 float4, fewer than threads)


def test_packers_agree_on_the_host_contract():
    """pack_events_host writes the invalid record for rows outside [offsets[0], offsets[B])."""
    from cistaflow_b200 import event_process as ep
    rng = np.random.default_rng(14)
    ev, off = layout("lead_rows", rng, 20, 30)
    ev = np.concatenate([ev, random_window(rng, 5, 20, 30)])
    rec = ep.pack_events_host(ev, off)
    outside = np.r_[0:off[0], off[-1]:len(ev)]
    assert (rec[outside] == np.uint64(0xffff) << np.uint64(32)).all()


# ----------------------------------------------------------------------------------------------- GPU plumbing ---
def _lib():
    from cistaflow_b200 import _lib as L
    return L


def lib():
    return _lib().load()


def last_kernel():
    return lib().cf_last_kernel().decode()


def launches():
    return int(lib().cf_launch_count())


def stream():
    return torch.cuda.current_stream().cuda_stream


class Call:
    pass


def run_bin(ev, off, nb, H, W, mode, flavour, pre=NONE, thr=0.0, dev="cuda"):
    ev = np.ascontiguousarray(ev, np.float64)
    B = len(off) - 1
    total = len(ev)
    ev_d = torch.from_numpy(ev).to(dev) if total else None
    off_d = torch.from_numpy(np.asarray(off, np.int64)).to(dev)
    shape = grid_shape(B, nb, H, W, flavour)
    buf, (out,) = guarded([shape], dev)
    need = lib().cf_voxel_workspace_bytes(total, B, nb, H, W, mode, flavour, pre)
    ws = torch.empty(max(need, 16), dtype=torch.uint8, device=dev)
    n0 = launches()
    rc = lib().cf_voxel_bin(ev_d.data_ptr() if total else None, off_d.data_ptr(), total, B, nb, H, W, mode, flavour,
                            pre, thr, out.data_ptr(), ws.data_ptr(), need, stream())
    torch.cuda.synchronize()
    c = Call()
    c.rc, c.kernel, c.launches, c.buf, c.view = rc, last_kernel(), launches() - n0, buf, out
    c.out = out.cpu().numpy() if rc == OK else None
    return c


def check_bits(c, want, what):
    assert c.rc == OK, (what, c.rc, lib().cf_last_error())
    assert_written_and_guarded(c.buf, [c.view], what)
    got = c.out.view(np.uint32)
    bad = got != want.view(np.uint32)
    assert not bad.any(), f"{what}: {int(bad.sum())} cells differ, first at {np.argwhere(bad)[0]}"


def check_bound(c, ref, bound, what, report=None, family=None):
    assert c.rc == OK, (what, c.rc, lib().cf_last_error())
    assert_written_and_guarded(c.buf, [c.view], what)
    err = np.abs(c.out.astype(np.float64) - ref)
    zero = bound == 0
    assert (err[zero] == 0).all(), f"{what}: {int((err[zero] != 0).sum())} cells with a zero bound are not exact"
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(zero, 0.0, err / bound)
    assert not np.isnan(ratio).any(), f"{what}: NaN in the output or the bound"
    worst = float(ratio.max()) if ratio.size else 0.0
    if report is not None:
        report.add(f"voxel_branches/{family}", case=what, max_err_over_bound=worst)
    assert worst <= 1.0, f"{what}: err/bound {worst:.3g} at {np.unravel_index(int(ratio.argmax()), ratio.shape)}"
    return worst


MODE_KERNEL = {DET: "det_accumulate_kernel", L2: "voxel_scatter_atomic_kernel", ATOMIC: "voxel_scatter_atomic_kernel",
               TILED: "voxel_tile_kernel"}


def check_binning(c, ev, off, nb, H, W, mode, flavour, what, report):
    assert c.kernel == MODE_KERNEL[mode], (what, c.kernel)
    if mode == DET:
        check_bits(c, seq_grid(ev, off, nb, H, W, flavour), what)
        report.add("voxel_branches/deterministic", case=what, max_err_over_bound=0.0)
    else:
        ref, bound, _, _ = atomic_ref(ev, off, nb, H, W, flavour)
        check_bound(c, ref, bound, what, report, "atomic_torch" if flavour == TORCH else "atomic_wide")


# ----------------------------------------------------------------------------------------------- window layout ---
@gpu
@pytest.mark.parametrize("name", LAYOUTS)
@pytest.mark.parametrize("mode,flavour", [(DET, f) for f in (TORCH, NUMPY, POL, MVSEC)] +
                         [(L2, f) for f in (TORCH, NUMPY, POL, MVSEC)] + [(TILED, f) for f in (TORCH, NUMPY, POL)] +
                         [(ATOMIC, TORCH)])
def test_window_layout(cuda_device, parity_report, name, mode, flavour):
    rng = np.random.default_rng(seed(name, mode, flavour))
    H, W, nb = 12, 17, 5
    ev, off = layout(name, rng, H, W, (0.0, 1.0) if flavour != MVSEC else (-1.0, 1.0, 0.5))
    c = run_bin(ev, off, nb, H, W, mode, flavour)
    check_binning(c, ev, off, nb, H, W, mode, flavour, f"{name}/mode{mode}/{FLAVOURS[flavour]}", parity_report)


@gpu
@pytest.mark.parametrize("mode", [DET, L2])
def test_ragged_batch_across_l2_chunks(cuda_device, parity_report, mode):
    """Ragged windows (0 .. 30 000 events) over 20 windows of 5x480x640: two L2-resident chunks."""
    rng = np.random.default_rng(21)
    nb, H, W, B = 5, 480, 640, 20
    sizes = rng.integers(0, 3000, B)
    sizes[3], sizes[14], sizes[15] = 30000, 0, 1
    ev, off = concat([random_window(rng, int(s), H, W) for s in sizes])
    chunk = l2_chunk(len(ev), B, nb * H * W)
    assert chunk < B and B % chunk and ceil_div(B, chunk) == 2
    c = run_bin(ev, off, nb, H, W, mode, TORCH)
    if mode == L2:
        assert c.launches == ceil_div(B, chunk)            # one scatter per chunk
    check_binning(c, ev, off, nb, H, W, mode, TORCH, f"ragged/mode{mode}", parity_report)


# ----------------------------------------------------------------------------------------------- edge events ---
@gpu
@pytest.mark.parametrize("order", ["sorted", "unsorted"])
@pytest.mark.parametrize("mode,flavour", [(DET, f) for f in (TORCH, NUMPY, POL, MVSEC)] +
                         [(L2, f) for f in (TORCH, NUMPY, POL, MVSEC)] + [(TILED, f) for f in (TORCH, NUMPY, POL)])
def test_edge_events(cuda_device, parity_report, order, mode, flavour):
    nb, H, W = 5, 6, 7
    ev = edge_window(flavour, nb, H, W)
    if order == "unsorted":
        ev = unsorted(ev, np.random.default_rng(22))
    off = np.array([0, len(ev)], np.int64)
    if mode == DET:
        assert runs_not_monotone(ev, off, nb, H, W, flavour) == (order == "unsorted")
    c = run_bin(ev, off, nb, H, W, mode, flavour)
    check_binning(c, ev, off, nb, H, W, mode, flavour, f"edges/{order}/mode{mode}/{FLAVOURS[flavour]}", parity_report)


def test_edge_window_covers_the_polarity_rules():
    """POL: p = 1.5 goes to channel 1 with weight 1.5, p = 2 and p = -1 are dropped; MVSEC: p = 0 adds +0."""
    ev = edge_window(POL)
    r = binned(ev, [0, len(ev)], 5, 6, 7, POL)
    p = ev[:, 3]
    assert not r["ok"][(p == 2) | (p == -1)].any()
    sel = r["ok"] & (p == 1.5)
    assert sel.any() and (r["chan"][sel] == 1).all() and (r["sgn"][sel] == 1.5).all()
    rm = binned(ev, [0, len(ev)], 5, 6, 7, MVSEC)
    wl, wr = weights(rm, MVSEC)
    z = rm["ok"] & (p == 0)
    assert z.any() and (wl[z] == 0).all() and not np.signbit(wl[z]).any()
    rt = binned(ev, [0, len(ev)], 5, 6, 7, TORCH)
    assert ((rt["dt"] == 0) & rt["ok"]).sum() > 8 and (rt["tn"] == 4.0).any()
    assert (weights(rt, TORCH)[0][rt["ok"] & (rt["dt"] > 0.99)] == 0).any()     # f32(dt) = 1: a +-0 left weight


# --------------------------------------------------------------------------------------------- deterministic ---
@gpu
@pytest.mark.parametrize("passes,B,H,W", [(1, 1, 8, 8), (2, 1, 100, 100), (3, 4, 480, 640), (4, 64, 480, 640)])
def test_deterministic_radix_passes(cuda_device, parity_report, passes, B, H, W):
    rng = np.random.default_rng(31 + passes)
    nb = 5
    columns = B * H * W
    bits = max(1, int(columns).bit_length())
    assert (bits + 7) // 8 == passes
    ev, off = concat([random_window(rng, 3000 if B > 1 else 20000, H, W) for _ in range(B)])
    c = run_bin(ev, off, nb, H, W, DET, TORCH)
    assert c.launches == 1 + 3 * passes + 1                 # keys, (hist, scan, scatter) per pass, accumulate
    check_binning(c, ev, off, nb, H, W, DET, TORCH, f"radix{passes}", parity_report)


@gpu
@pytest.mark.parametrize("flavour", [TORCH, NUMPY, POL, MVSEC])
def test_deterministic_long_single_pixel_runs(cuda_device, parity_report, flavour):
    rng = np.random.default_rng(41)
    ev = random_window(rng, 6000, 4, 5, (0.0, 1.0) if flavour != MVSEC else (-1.0, 0.5, 1.0))
    ev[:, 1], ev[:, 2] = 3.25, 2.5
    ev[::7, 1] = 1.0
    ev2, off = concat([ev, random_window(rng, 100, 4, 5)])
    c = run_bin(ev2, off, 7, 4, 5, DET, flavour)
    check_binning(c, ev2, off, 7, 4, 5, DET, flavour, f"long_run/{FLAVOURS[flavour]}", parity_report)


def _filter_offsets_bin(ev_d, total, W, H, param, max_windows, nb, policy, bufs):
    L = lib()
    filt, kept, fws, offs, nwin, out, vws = bufs
    s = stream()
    assert L.cf_events_filter(ev_d.data_ptr(), total, W, H, filt.data_ptr(), kept.data_ptr(), fws.data_ptr(), fws.numel(), s) == OK
    assert L.cf_event_window_offsets(kept.data_ptr(), policy, param, offs.data_ptr(), max_windows, nwin.data_ptr(), s) == OK
    assert L.cf_voxel_bin(filt.data_ptr(), offs.data_ptr(), total, max_windows, nb, H, W, DET, TORCH, NONE, 0.0,
                          out.data_ptr(), vws.data_ptr(), vws.numel(), s) == OK


@gpu
@pytest.mark.parametrize("policy", [FIXED, SPLIT])
def test_deterministic_repeatable_on_streams_and_in_a_graph(cuda_device, policy):
    """Bit for bit: again, on a side stream, and the chain filter -> window_offsets -> cf_voxel_bin(B = max_windows)
    captured as one CUDA graph against the eager chain; all equal the restatement of the filtered windows."""
    rng = np.random.default_rng(51)
    H, W, nb, param, max_windows = 30, 40, 5, 700, 6
    ev = random_window(rng, 3000, H + 3, W + 3)          # some rows outside the grid: filtered out
    total = len(ev)
    dev = cuda_device
    ev_d = torch.from_numpy(ev).to(dev)

    def bufs():
        return (torch.empty_like(ev_d), torch.empty(1, dtype=torch.int64, device=dev),
                torch.empty(lib().cf_events_filter_workspace_bytes(total), dtype=torch.uint8, device=dev),
                torch.empty(max_windows + 1, dtype=torch.int64, device=dev), torch.empty(1, dtype=torch.int32, device=dev),
                torch.full((max_windows, nb, H, W), float("nan"), device=dev),
                torch.empty(lib().cf_voxel_workspace_bytes(total, max_windows, nb, H, W, DET, TORCH, NONE), dtype=torch.uint8, device=dev))
    keep = (ev[:, 1] < W) & (ev[:, 2] < H)
    kev = ev[keep]
    off, k = window_offsets_ref(len(kev), policy, param, max_windows)
    want = seq_grid(kev, off, nb, H, W, TORCH)
    results = []
    for where in ("eager", "again", "side"):
        b = bufs()
        if where == "side":
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                _filter_offsets_bin(ev_d, total, W, H, param, max_windows, nb, policy, b)
            torch.cuda.current_stream().wait_stream(side)
        else:
            _filter_offsets_bin(ev_d, total, W, H, param, max_windows, nb, policy, b)
        torch.cuda.synchronize()
        assert int(b[4].item()) == k and list(b[3].cpu().numpy()) == list(off)
        results.append(b[5].cpu().numpy())
    b = bufs()
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            _filter_offsets_bin(ev_d, total, W, H, param, max_windows, nb, policy, b)
    graph.replay()
    torch.cuda.synchronize()
    results.append(b[5].cpu().numpy())
    for r in results:
        assert np.array_equal(r.view(np.uint32), want.view(np.uint32))


# ------------------------------------------------------------------------------------------------------ tiled ---
def tiled_case(name, rng):
    """(events, offsets, nb, H, W) of the tiled geometry rows."""
    if name == "one_tile_per_window":
        return (*concat([random_window(rng, 200, 30, 40) for _ in range(300)]), 5, 30, 40)
    if name == "many_tiles_small_batch":
        return (*concat([random_window(rng, 60000, 480, 640)]), 5, 480, 640)
    if name == "many_tiles":
        return (*concat([random_window(rng, 20000, 480, 640) for _ in range(8)]), 5, 480, 640)
    if name == "hw_not_multiple_of_4":
        return (*concat([random_window(rng, 3000, 31, 37) for _ in range(3)]), 5, 31, 37)
    if name == "hot_pixel":
        w = random_window(rng, 5000, 30, 40)
        w[:4500, 1], w[:4500, 2] = 7.0, 9.0
        return (*concat([w, random_window(rng, 300, 30, 40)]), 5, 30, 40)
    if name == "window_longer_than_max_c":
        return (*concat([random_window(rng, s, 30, 40) for s in (20000, 100, 100, 100)]), 5, 30, 40)
    if name == "chunk_edges":
        return (*concat([random_window(rng, s, 30, 40) for s in (CHUNK - 1, CHUNK, CHUNK + 1)]), 5, 30, 40)
    raise KeyError(name)


TILED_CASES = ["one_tile_per_window", "many_tiles_small_batch", "many_tiles", "hw_not_multiple_of_4", "hot_pixel",
               "window_longer_than_max_c", "chunk_edges"]


@gpu
@pytest.mark.parametrize("name", TILED_CASES)
@pytest.mark.parametrize("flavour", [TORCH, POL])
def test_tiled_geometry(cuda_device, parity_report, name, flavour):
    rng = np.random.default_rng(seed(name, flavour))
    ev, off, nb, H, W = tiled_case(name, rng)
    if flavour == POL:
        ev[:, 3] = rng.choice([0.0, 1.0], len(ev))
    B = len(off) - 1
    g = tiled_geometry(len(ev), B, nb, H, W, flavour)
    assert g is not None
    sizes = np.diff(off)
    proof = {"one_tile_per_window": g["T"] == 1,
             "many_tiles_small_batch": g["want"] > g["t0"] and g["T"] > 1,
             "many_tiles": g["t0"] >= g["want"] and g["T"] > 1,
             "hw_not_multiple_of_4": (H * W) % 4 != 0,
             "hot_pixel": True,
             "window_longer_than_max_c": sizes.max() > g["max_c"] * CHUNK,
             "chunk_edges": set(sizes) == {CHUNK - 1, CHUNK, CHUNK + 1}}[name]
    assert proof, (name, g)
    if name == "hot_pixel":
        r = binned(ev, off, nb, H, W, flavour)
        assert np.bincount(r["y"][:CHUNK] * W + r["x"][:CHUNK]).max() > 64
    c = run_bin(ev, off, nb, H, W, TILED, flavour)
    check_binning(c, ev, off, nb, H, W, TILED, flavour, f"tiled/{name}/{FLAVOURS[flavour]}", parity_report)


@gpu
def test_tiled_refusals_and_the_empty_batch(cuda_device):
    ev = random_window(np.random.default_rng(61), 100, 30, 40)
    c = run_bin(ev, [0, 100], 5, 30, 40, TILED, MVSEC)
    assert c.rc == UNSUPPORTED and "MVSEC" in lib().cf_last_error().decode()
    ev = random_window(np.random.default_rng(62), 100, 2000, 2000)
    assert tiled_geometry(100, 1, 5, 2000, 2000, TORCH) is None
    c = run_bin(ev, [0, 100], 5, 2000, 2000, TILED, TORCH)
    assert c.rc == UNSUPPORTED
    for pre in (NONE, STD):                       # an empty batch: the L2 zero-fill (+ normalise) path
        c = run_bin(np.zeros((0, 4)), [0, 0, 0], 5, 30, 40, TILED, TORCH, pre)
        assert c.rc == OK and (c.out == 0).all() and not np.signbit(c.out).any()
        assert_written_and_guarded(c.buf, [c.view], "tiled empty")
        assert c.launches == (0 if pre == NONE else 2)


# --------------------------------------------------------------------------------- fused normalisation paths ---
def fused_case(rng, B, nb, H, W, n):
    return concat([dyadic_window(rng, n, nb, H, W) for _ in range(B)])


@gpu
@pytest.mark.parametrize("pre", [STD, MAXMIN])
@pytest.mark.parametrize("thr", [0.0, 0.75])
@pytest.mark.parametrize("mode,flavour", [(L2, TORCH), (L2, NUMPY), (TILED, TORCH), (TILED, POL), (DET, TORCH),
                                          (DET, MVSEC)])
def test_fused_normalisation(cuda_device, parity_report, pre, thr, mode, flavour):
    """Dyadic events: the grid of the fused call equals the NONE call's, whatever the summation order."""
    rng = np.random.default_rng(71)
    B, nb, H, W = 5, 5, 31, 37
    ev, off = fused_case(rng, B, nb, H, W, 2500)
    ev, off = concat([ev[off[b]:off[b + 1]] for b in range(B)] + [np.zeros((0, 4))])    # + an all-zero window
    B += 1
    base = run_bin(ev, off, nb, H, W, mode, flavour)
    c = run_bin(ev, off, nb, H, W, mode, flavour, pre, thr)
    assert c.kernel == ("voxel_tile_kernel" if mode == TILED else "voxel_normalise_kernel")
    cells = base.out[0].size
    refs, bounds = [], []
    _, _, n, M = atomic_ref(ev, off, nb, H, W, flavour)
    for b in range(B):
        if mode == TILED:           # telescoped statistics: depth = every add of the window, magnitudes of old + new
            k = int(n[b].sum()) + ceil_div(tiled_geometry(len(ev), B, nb, H, W, flavour)["T"], 32) + 64 + 160
            A1 = float((2 * n[b] * M[b]).sum())
            A2 = float((2 * n[b] * M[b] ** 2).sum())
            r, bd = norm_ref(base.out[b], pre, thr, k, A1, A2)
        else:
            r, bd = norm_ref(base.out[b], pre, thr, stat_depth(B, cells))
        refs.append(r)
        bounds.append(bd)
    ref = np.stack(refs).reshape(c.out.shape)
    bound = np.stack(bounds).reshape(c.out.shape)
    if pre == STD:
        assert np.array_equal(c.out[-1], base.out[-1])       # the all-zero window is the identity
    check_bound(c, ref, bound, f"fused/mode{mode}/{FLAVOURS[flavour]}/pre{pre}/thr{thr}", parity_report, "normalise")


@gpu
@pytest.mark.parametrize("mode", [L2, DET])
def test_fused_shifted_grid(cuda_device, parity_report, mode):
    """The shifted grid (every cell 3 + 0.01 N(0, 1)) through a fused path: MVSEC with nb = 1 puts f32(p) of one event
    into each cell, so the grid is exact and equals the NONE call's."""
    rng = np.random.default_rng(81)
    H, W = 480, 640
    yy, xx = np.divmod(np.arange(H * W), W)
    ev = np.stack([np.full(H * W, T0), xx + 0.5, yy + 0.5, 3.0 + 0.01 * rng.standard_normal(H * W)], axis=1)
    off = np.array([0, H * W], np.int64)
    base = run_bin(ev, off, 1, H, W, mode, MVSEC)
    c = run_bin(ev, off, 1, H, W, mode, MVSEC, STD)
    assert c.kernel == "voxel_normalise_kernel"
    ref, bound = norm_ref(base.out[0], STD, 0.0, stat_depth(1, H * W))
    check_bound(c, ref.reshape(c.out.shape), bound.reshape(c.out.shape), f"fused_shifted/mode{mode}", parity_report,
                "normalise")


# ---------------------------------------------------------------------------------------- cf_voxel_preprocess ---
def run_preprocess(g, pre, thr, inplace=False, dev="cuda"):
    B = g.shape[0]
    cells = g[0].size
    shape = (B, cells)
    buf, (inp, outp) = guarded([shape, shape], dev)
    inp.copy_(torch.from_numpy(np.ascontiguousarray(g.reshape(shape), F32)))
    out = inp if inplace else outp
    if inplace:
        outp.fill_(0.0)         # unused view: keep the guard check meaningful
    need = lib().cf_preprocess_workspace_bytes(B, cells)
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    n0 = launches()
    rc = lib().cf_voxel_preprocess(inp.data_ptr(), out.data_ptr(), B, cells, pre, thr, ws.data_ptr(), need, stream())
    torch.cuda.synchronize()
    c = Call()
    c.rc, c.kernel, c.launches, c.buf, c.view = rc, last_kernel(), launches() - n0, buf, out
    c.views = [inp, outp]
    c.out = out.cpu().numpy()
    return c


def check_preprocess(c, g, pre, thr, what, report):
    assert c.rc == OK and c.kernel == "voxel_normalise_kernel" and c.launches == 2, (what, c.rc, c.kernel)
    assert_written_and_guarded(c.buf, c.views, what)
    B = g.shape[0]
    cells = g[0].size
    worst = 0.0
    for b in range(B):
        ref, bound = norm_ref(g[b], pre, thr, stat_depth(B, cells))
        got = c.out[b].astype(np.float64)
        zero = bound == 0
        assert np.array_equal(got[zero], ref[zero]), f"{what}: window {b}: exact cells differ"
        with np.errstate(divide="ignore", invalid="ignore"):
            r = np.where(zero, 0.0, np.abs(got - ref) / bound)
        assert not np.isnan(r).any(), f"{what}: window {b}: NaN in the output or the bound"
        worst = max(worst, float(r.max()))
    report.add("voxel_branches/normalise", case=what, max_err_over_bound=worst)
    assert worst <= 1.0, f"{what}: err/bound {worst:.3g}"


def event_like(rng, B, cells, dens=0.2):
    g = np.where(rng.random((B, cells)) < dens, rng.standard_normal((B, cells)), 0.0)
    return g.astype(F32)


@gpu
@pytest.mark.parametrize("case", ["cells_not_multiple_of_4", "chunk_cap_512", "short_trailing_chunk",
                                  "shifted_b1", "shifted_b64_315_terms", "event_like_b64", "hot_thr_ties",
                                  "zero_and_single_nonzero"])
@pytest.mark.parametrize("inplace", [False, True])
@pytest.mark.parametrize("pre", [STD, MAXMIN])
def test_preprocess(cuda_device, parity_report, case, inplace, pre):
    rng = np.random.default_rng(seed(case))
    thr = 0.0
    if case == "cells_not_multiple_of_4":
        g = event_like(rng, 3, 5735)
        assert g.shape[1] % 4
    elif case == "chunk_cap_512":
        g = event_like(rng, 1, 5 * 480 * 640)
        assert stat_geometry(1, g.shape[1])[0] == K_MAX_CHUNKS
    elif case == "short_trailing_chunk":
        g = event_like(rng, 1, SHORT_TAIL_CELLS, 0.5)
    elif case == "shifted_b1":
        g = (3.0 + 0.01 * rng.standard_normal((1, 5 * 480 * 640))).astype(F32)
    elif case == "shifted_b64_315_terms":
        if pre == MAXMIN or inplace:
            pytest.skip("one configuration of this size is enough")
        g = (3.0 + 0.01 * rng.standard_normal((64, 5 * 480 * 640))).astype(F32)
        assert stat_geometry(64, g.shape[1])[1] // 256 == 315
    elif case == "event_like_b64":
        if pre == MAXMIN or inplace:
            pytest.skip("one configuration of this size is enough")
        g = event_like(rng, 64, 5 * 480 * 640)
    elif case == "hot_thr_ties":
        thr = 1.25
        g = event_like(rng, 2, 4096)
        g[:, ::7] = F32(thr)
        g[:, 3::7] = -F32(thr)
        g[:, 5::11] = F32(2.5)
    else:
        g = np.zeros((3, 4099), F32)
        g[1, 1234] = F32(-2.5)
        g[2] = event_like(rng, 1, 4099)[0]
    c = run_preprocess(g, pre, thr, inplace)
    if case == "hot_thr_ties" and pre == STD:        # |v| == thr is kept (the comparison is strict), 2.5 is zeroed
        assert (c.out[np.abs(g) == F32(thr)] != 0).all() and (c.out[np.abs(g) > F32(thr)] == 0).all()
    if case == "zero_and_single_nonzero" and pre == STD:
        assert np.array_equal(c.out[0], g[0]) and c.out[1, 1234] == 0 and (c.out[1] == 0).all()
    check_preprocess(c, g, pre, thr, f"preprocess/{case}/pre{pre}/inplace{int(inplace)}", parity_report)


@gpu
def test_preprocess_rejects_more_than_65535_windows(cuda_device):
    g = torch.zeros((65536, 4), device=cuda_device)
    rc = lib().cf_voxel_preprocess(g.data_ptr(), g.data_ptr(), 65536, 4, STD, 0.0, None, 0, stream())
    assert rc == INVALID_ARG and "65535" in lib().cf_last_error().decode()


@gpu
def test_preprocess_python_wrappers(cuda_device):
    """The drop-in wrappers reach the same kernel with the reference's thresholds (25/nb numpy, 20/nb torch)."""
    from cistaflow_b200 import event_process as ep
    rng = np.random.default_rng(91)
    g = (event_like(rng, 1, 5 * 30 * 40)[0] * 8).reshape(5, 30, 40)
    for fn, thr in ((ep.event_preprocess, 25.0 / 5), (ep.event_preprocess_pytorch, 20.0 / 5)):
        arg = g if fn is ep.event_preprocess else torch.from_numpy(g).to(cuda_device)
        got = fn(arg, "std", True)
        got = got.cpu().numpy() if torch.is_tensor(got) else got
        assert last_kernel() == "voxel_normalise_kernel"
        ref, bound = norm_ref(g, STD, thr, stat_depth(1, g.size))
        assert (np.abs(got.reshape(-1) - ref) <= bound).all()


# --------------------------------------------------------------------------------------------------- routing ---
@gpu
def test_atomic_mode_runs_and_sizes_the_l2_path(cuda_device):
    """CF_VOXEL_ATOMIC asks only for the L2 path's workspace, and runs it at a small and at the bench shape."""
    L = lib()
    for (B, nb, H, W, n) in ((2, 5, 30, 40, 500), (64, 5, 480, 640, 100000)):
        total = B * n
        base = ceil_div(B * K_MAX_CHUNKS * 32, 256) * 256
        for pre in (NONE, STD):
            assert L.cf_voxel_workspace_bytes(total, B, nb, H, W, ATOMIC, TORCH, pre) == base
            assert L.cf_voxel_workspace_bytes(total, B, nb, H, W, L2, TORCH, pre) == base
        assert L.cf_voxel_workspace_bytes(total, B, nb, H, W, TILED, TORCH, NONE) >= base + 12 * total
    rng = np.random.default_rng(95)
    for (B, H, W, n) in ((2, 30, 40, 500), (64, 480, 640, 2000)):
        ev, off = concat([random_window(rng, n, H, W) for _ in range(B)])
        c = run_bin(ev, off, 5, H, W, ATOMIC, TORCH)
        assert c.kernel == "voxel_scatter_atomic_kernel" and c.launches == ceil_div(B, l2_chunk(len(ev), B, 5 * H * W))
        c = run_bin(ev, off, 5, H, W, ATOMIC, TORCH, STD)
        assert c.kernel == "voxel_normalise_kernel"


@gpu
def test_python_wrappers_ignore_rows_outside_the_windows(cuda_device):
    """events_to_voxel_grid_batched with offsets[0] > 0: 'deterministic' and 'atomic' agree with the restatement."""
    from cistaflow_b200 import event_process as ep
    rng = np.random.default_rng(96)
    ev, off = layout("lead_rows", rng, 12, 17)
    ev_d, off_d = torch.from_numpy(ev).to(cuda_device), torch.from_numpy(off).to(cuda_device)
    for flav, fid in (("numpy", NUMPY), ("torch", TORCH)):
        det = ep.events_to_voxel_grid_batched(ev_d, off_d, 5, 17, 12, flavour=flav, mode="deterministic").cpu().numpy()
        assert np.array_equal(det.view(np.uint32), seq_grid(ev, off, 5, 12, 17, fid).view(np.uint32))
        atom = ep.events_to_voxel_grid_batched(ev_d, off_d, 5, 17, 12, flavour=flav, mode="atomic").cpu().numpy()
        ref, bound, _, _ = atomic_ref(ev, off, 5, 12, 17, fid)
        assert (np.abs(atom - ref) <= bound).all()


# ----------------------------------------------------------------------------------------------------- packed ---
def run_pack(ev, off, dev="cuda"):
    ev_d = torch.from_numpy(np.ascontiguousarray(ev, np.float64)).to(dev)
    off_d = torch.from_numpy(np.asarray(off, np.int64)).to(dev)
    rec = torch.full((len(ev),), -1, dtype=torch.int64, device=dev)
    rc = lib().cf_events_pack(ev_d.data_ptr(), off_d.data_ptr(), len(ev), len(off) - 1, rec.data_ptr(), stream())
    torch.cuda.synchronize()
    assert rc == OK and last_kernel() == "events_pack_kernel"
    return rec.cpu().numpy().view(np.uint64)


def run_packed_bin(rec, off, nb, H, W, pre=NONE, thr=0.0, dev="cuda"):
    rec_d = torch.from_numpy(rec.view(np.int64)).to(dev)
    off_d = torch.from_numpy(np.asarray(off, np.int64)).to(dev)
    B = len(off) - 1
    buf, (out,) = guarded([(B, nb, H, W)], dev)
    need = lib().cf_preprocess_workspace_bytes(B, nb * H * W)
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    rc = lib().cf_voxel_bin_packed(rec_d.data_ptr(), off_d.data_ptr(), len(rec), B, nb, H, W, pre, thr, out.data_ptr(),
                                   ws.data_ptr(), need, stream())
    torch.cuda.synchronize()
    c = Call()
    c.rc, c.kernel, c.buf, c.view = rc, last_kernel(), buf, out
    c.out = out.cpu().numpy()
    return c


@gpu
@pytest.mark.parametrize("name", LAYOUTS + ["coords"])
def test_packers_agree_bit_for_bit(cuda_device, name):
    from cistaflow_b200 import event_process as ep
    rng = np.random.default_rng(seed(name))
    if name == "coords":
        ev = random_window(rng, 40, 20, 30, (0.0, 1.0, -1.0, 0.5))
        ev[:, 1] = [65534.9, 65535.0, 70000.0, -0.5, -0.0, float("nan"), 3.0, 65534.0] * 5
        ev[:, 2] = [32767.5, 3.0, 1.0, 2.0, 32768.0, 1.0, -1.0, float("nan")] * 5
        off = np.array([0, 20, 40], np.int64)
    else:
        ev, off = layout(name, rng, 20, 30, (0.0, 1.0, -1.0, 0.5))
    host = ep.pack_events_host(ev, off)
    dev = run_pack(ev, off)
    assert np.array_equal(host, dev)
    outside = np.r_[0:off[0], off[-1]:len(ev)]
    assert (dev[outside] == np.uint64(0xffff) << np.uint64(32)).all()


@gpu
@pytest.mark.parametrize("name", LAYOUTS + ["random", "x_limit_65535", "y_limit_32768"])
def test_packed_binning(cuda_device, parity_report, name):
    rng = np.random.default_rng(seed(name))
    nb, H, W = 5, 12, 17
    if name == "random":
        ev, off = concat([random_window(rng, 5000, H, W, (0.0, 1.0, -1.0, 0.5)) for _ in range(3)])
    elif name == "x_limit_65535":
        nb, H, W = 5, 1, 65535
        ev, off = concat([random_window(rng, 4000, H, W)])
        ev[:5, 1] = [65534.5, 65535.0, -0.5, 0.0, 70000.0]
    elif name == "y_limit_32768":
        nb, H, W = 5, 32768, 1
        ev, off = concat([random_window(rng, 4000, H, W)])
        ev[:5, 2] = [32767.5, 32768.0, -0.5, 0.0, 40000.0]
    else:
        ev, off = layout(name, rng, H, W, (0.0, 1.0, -1.0, 0.5))
    c = run_packed_bin(run_pack(ev, off), off, nb, H, W)
    assert c.rc == OK and c.kernel == "voxel_scatter_packed_kernel"
    ref, bound = packed_ref(ev, off, nb, H, W)
    check_bound(c, ref, bound, f"packed/{name}", parity_report, "packed")


@gpu
@pytest.mark.parametrize("pre", [STD, MAXMIN])
def test_packed_fused(cuda_device, parity_report, pre):
    rng = np.random.default_rng(101)
    nb, H, W, B = 5, 31, 37, 4
    ev, off = fused_case(rng, B, nb, H, W, 2500)
    rec = run_pack(ev, off)
    base = run_packed_bin(rec, off, nb, H, W)
    ref0, _ = packed_ref(ev, off, nb, H, W)
    assert np.array_equal(base.out.astype(np.float64), ref0)           # dyadic: exact in fp32
    c = run_packed_bin(rec, off, nb, H, W, pre, 0.75)
    assert c.rc == OK and c.kernel == "voxel_normalise_kernel"
    cells = nb * H * W
    rb = [norm_ref(base.out[b], pre, 0.75, stat_depth(B, cells)) for b in range(B)]
    check_bound(c, np.stack([r for r, _ in rb]).reshape(c.out.shape), np.stack([b for _, b in rb]).reshape(c.out.shape),
                f"packed_fused/pre{pre}", parity_report, "normalise")


# ---------------------------------------------------------------------------------------- filter and offsets ---
@gpu
@pytest.mark.parametrize("total", [0, 2047, 2048, 2049, 2048 * 1100 + 5])
def test_events_filter(cuda_device, total):
    rng = np.random.default_rng(total)
    H, W = 20, 30
    ev = random_window(rng, total, H + 2, W + 2) if total else np.zeros((0, 4))
    if total:
        ev[rng.random(total) < 0.05, 1] = W                     # x == W: dropped
        ev[rng.random(total) < 0.05, 1] = float("nan")          # NaN: dropped
        ev[rng.random(total) < 0.05, 2] = -3.0                  # negative: kept (no lower bound)
    tiles = ceil_div(max(total, 1), 2048)
    if total > 2048 * 1024:
        assert ceil_div(tiles, 1024) > 1                        # the scan kernel's per > 1
    dev = cuda_device
    ev_d = torch.from_numpy(ev).to(dev) if total else torch.zeros((1, 4), dtype=torch.float64, device=dev)
    out = torch.full((max(total, 1), 4), float("nan"), dtype=torch.float64, device=dev)
    kept = torch.full((1,), -1, dtype=torch.int64, device=dev)
    need = lib().cf_events_filter_workspace_bytes(total)
    ws = torch.empty(need, dtype=torch.uint8, device=dev)
    rc = lib().cf_events_filter(ev_d.data_ptr(), total, W, H, out.data_ptr(), kept.data_ptr(), ws.data_ptr(), need, stream())
    torch.cuda.synchronize()
    assert rc == OK
    want = ev[(ev[:, 1] < W) & (ev[:, 2] < H)] if total else ev
    assert int(kept.item()) == len(want)
    got = out[:len(want)].cpu().numpy()
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
    if total:
        assert last_kernel() == "filter_scatter_kernel"
        assert torch.isnan(out[len(want):]).all()


@gpu
@pytest.mark.parametrize("n,policy,param,max_windows", [
    (5, SPLIT, 2, 8), (7, SPLIT, 2, 8), (0, FIXED, 10, 3), (0, SPLIT, 10, 3), (1000, FIXED, 100, 4),
    (1000, SPLIT, 100, 4), (999, FIXED, 100, 12), (1049, SPLIT, 100, 12), (1050, SPLIT, 100, 12), (1, FIXED, 1, 1)])
@pytest.mark.parametrize("with_count", [True, False])
def test_window_offsets(cuda_device, n, policy, param, max_windows, with_count):
    dev = cuda_device
    cnt = torch.tensor([n], dtype=torch.int64, device=dev)
    offs = torch.full((max_windows + 1,), -7, dtype=torch.int64, device=dev)
    nw = torch.full((1,), -7, dtype=torch.int32, device=dev)
    rc = lib().cf_event_window_offsets(cnt.data_ptr(), policy, param, offs.data_ptr(), max_windows,
                                       nw.data_ptr() if with_count else None, stream())
    torch.cuda.synchronize()
    assert rc == OK and last_kernel() == "window_offsets_kernel"
    want, k = window_offsets_ref(n, policy, param, max_windows)
    assert list(offs.cpu().numpy()) == list(want)
    assert int(nw.item()) == (k if with_count else -7)
