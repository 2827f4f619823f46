/*
 * cistaflow_altcorr.h -- on-demand correlation lookup of libcistaflow.so (AlternateCorrBlock).
 *
 * replaces  DCEIFlow/core/corr/raft_corr.py:175-203  AlternateCorrBlock (RAFT's design; its CUDA extension
 *           alt_cuda_corr is not part of the reference checkout, SURVEY.md F1)
 *
 * Instead of the O(B*N^2) all-pairs pyramid of cf_corr_build, a caller keeps an O(B*D*N) state -- fmap1 and the
 * average-pooled levels of fmap2, channel-last -- and every lookup computes only the dot products around each query.
 * avg_pool2d is linear, so level l of the pyramid at target (y, x) equals <fmap1[:, q], P^l(fmap2)[:, y, x]> / sqrt(D)
 * with P^l = avg_pool2d(., 2, 2) applied l times (odd sizes floored): the output is that of cf_corr_lookup on the
 * pyramid of cf_corr_build, up to fp32 summation order and operand rounding.
 *
 * Conventions are those of cistaflow.h: device pointers only, no allocation, no host synchronisation (a prepare and
 * its lookups can be captured in a CUDA graph), CF_OK or a negative cf_status.
 */
#ifndef CISTAFLOW_ALTCORR_H_
#define CISTAFLOW_ALTCORR_H_

#include "cistaflow.h"

#ifdef __cplusplus
extern "C" {
#endif

/*
 * Bytes of state for fmap1 / fmap2 [B, D, h, w]: fmap1 as [B, h, w, D] and levels 0 .. levels-1 of fmap2 as
 * [B, h>>l, w>>l, D], each region rounded up to 256 bytes (at most 3 * B*D*h*w*4 + 256 * (levels + 1)).
 * 0 for B == 0 and for arguments cf_corr_alt_prepare rejects.
 */
CF_API size_t cf_corr_alt_workspace_bytes(int B, int D, int h, int w, int levels, int precision);

/*
 * Writes the state (16-byte aligned, at least cf_corr_alt_workspace_bytes bytes).  Level l+1 of fmap2 is pooled
 * from level l, as the reference's repeated avg_pool2d does.  CF_ERR_WORKSPACE for a missing or short state,
 * CF_ERR_ALIGN for a misaligned pointer, CF_ERR_INVALID_ARG for levels outside 1..6 or a map without level
 * levels-1, CF_ERR_UNSUPPORTED for CF_CORR_F16 and CF_CORR_3XTF32.
 */
CF_API int cf_corr_alt_prepare(const float *fmap1, const float *fmap2, int B, int D, int h, int w, int levels,
                               int precision, void *state, size_t state_bytes, cf_stream_t stream);

/*
 * coords [B, 2, h, w], out [B, levels*(2r+1)^2, h, w]: the layout and window of cf_corr_lookup (channel
 * l*(2r+1)^2 + i*(2r+1) + j samples (x/2^l + i - r, y/2^l + j - r), zero outside the map).  The shape arguments
 * are those the state was prepared with (a smaller `levels` is allowed); radius 0..8.
 *   CF_CORR_TF32, CF_CORR_AUTO  tcgen05.mma kind::tf32 on tiles of 16x8 queries whose windows fit one box of
 *                               targets per level (TF32 operands, rounded to nearest, as CorrBlock's default);
 *                               the other tiles (noise flow, wild coordinates) and maps with D % 32 != 0 go
 *                               to the fp32 kernel.  The split is decided on the device, per tile.
 *   CF_CORR_FP32                every tile on the fp32 SIMT kernel.
 * The state is only read: lookups on several streams may share it.
 */
CF_API int cf_corr_alt_lookup(const void *state, const float *coords, int B, int D, int h, int w, int levels,
                              int radius, int precision, float *out, cf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CISTAFLOW_ALTCORR_H_ */
