/*
 * cistaflow_half.h -- opt-in fp16 correlation pyramid of libcistaflow.so.
 *
 * The pyramid of cf_corr_build in IEEE binary16 instead of float32: half the bytes of the largest tensor of the
 * flow network (7.8 GB -> 3.9 GB for 64 x 60x80, D = 256, 4 levels), half the bytes written by the build and half the
 * patch bytes read by every lookup.  The caller takes the precision decision (the reference's HalfCorrBlock,
 * DCEIFlow/core/corr/raft_corr.py:68-118, for the same reason); cf_corr_build keeps the fp32 pyramid.  Inference
 * only: there is no adjoint of this pyramid.
 *
 * Contract (same shapes as cf_corr_build: level l is [B*h*w, 1, h>>l, w>>l], here as binary16 bit patterns):
 *   - level 0 = RN_f16(v), v the fp32 value cf_corr_build stores for the same precision (TF32, F16 or AUTO
 *     operands, fp32 accumulation, x 1/sqrt(D));
 *   - level l+1 = RN_f16((((a + b) + c) + d) * 0.25) with a, b, c, d the four STORED level-l values of the 2x2 window
 *     (rows 2y, 2y, 2y+1, 2y+1; columns 2x, 2x+1, 2x, 2x+1), widened to fp32 and summed in fp32 in that order; odd
 *     sizes are floored.  Each level is therefore avg_pool2d of the level above as stored, whether the build's epilogue
 *     or a pooling kernel produced it;
 *   - overflow is IEEE: |v| >= 65520 is stored as +-inf, and NaN stays NaN.  Nothing is clamped;
 *   - the absolute error of level 0 is that of cf_corr_build plus half an fp16 ulp: <= 2^-11 * |v| + 2^-25.
 *
 * Conventions are those of cistaflow.h: device pointers only, no allocation, no host synchronisation (graph-capturable),
 * CF_OK or a negative cf_status.
 */
#ifndef CISTAFLOW_HALF_H_
#define CISTAFLOW_HALF_H_

#include "cistaflow.h"

#ifdef __cplusplus
extern "C" {
#endif

/*
 * fmap1, fmap2 [B, D, h, w] float32;  pyramid[l] [B*h*w, 1, h>>l, w>>l] binary16 (host array of `levels` device
 * pointers, 16-byte aligned).  The workspace is cf_corr_workspace_bytes(B, D, h, w, levels, precision) bytes.
 *   precision  CF_CORR_TF32, CF_CORR_F16 or CF_CORR_AUTO (the same choice of operands as cf_corr_build);
 *              CF_CORR_FP32 and CF_CORR_3XTF32 return CF_ERR_UNSUPPORTED: fp16 storage would lose their fp32 accuracy.
 *   shapes     D % 32 == 0 and h*w % 8 == 0 (the fp16 volume's row pitch must be a multiple of 16 bytes for its
 *              tensor map); otherwise CF_ERR_UNSUPPORTED.  All of 24x32, 36x44, 60x80, 80x124 and 92x160 qualify.
 * The experiment switches of CF_TC_FLAGS are not honoured: the build always takes the library's default tiling.
 */
CF_API int cf_corr_build_half(const float *fmap1, const float *fmap2, int B, int D, int h, int w, int levels,
                              uint16_t *const *pyramid, int precision, void *workspace, size_t workspace_bytes,
                              cf_stream_t stream);

/*
 * cf_corr_lookup on an fp16 pyramid: same coords [B, 2, h, w], same fp32 output [B, levels*(2r+1)^2, h, w], same
 * levels (1..6) and radii (0..8).  Each tap is widened to fp32 as it is loaded and everything after that is the
 * arithmetic of cf_corr_lookup, so the output equals cf_corr_lookup on the widened pyramid bit for bit.
 */
CF_API int cf_corr_lookup_half(const uint16_t *const *pyramid, const float *coords, int B, int h, int w, int levels,
                               int radius, float *out, cf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CISTAFLOW_HALF_H_ */
