/*
 * cistaflow_det.h -- deterministic adjoint of the warp in libcistaflow.so.
 *
 * cf_warp_backward (cistaflow.h) splats the image gradient into the four taps of every sample with fp32 atomics, so
 * two identical backward passes can differ in the last bits.  cf_warp_backward_det computes the same gradients with
 * the same per-term arithmetic but sums them in an order fixed by the inputs alone:
 *   1. one record per (output pixel p, valid tap k): key = item * H*W + source pixel, value = 4p + k, weight;
 *   2. a stable radix sort by key, so the records of a source pixel are in ascending (p, k) order;
 *   3. one thread per (source pixel, group of channels) walks its records in that order and writes grad_img once;
 *   4. grad_flow is summed per output pixel over the channels in order; with the fused x0.5 down-sampling, each
 *      full-resolution flow pixel gathers the half-resolution pixels whose bilinear taps include it, in order.
 * No floating-point atomics and no memset of the outputs.
 *
 * Properties:
 *   - bitwise identical results for identical inputs, whatever the stream, and inside or outside a CUDA graph;
 *   - no host synchronisation: a call can be captured in a CUDA graph;
 *   - the caller provides the workspace (see cf_warp_backward_det_workspace_bytes; any alignment).
 */
#ifndef CISTAFLOW_DET_H_
#define CISTAFLOW_DET_H_

#include "cistaflow.h"

#ifdef __cplusplus
extern "C" {
#endif

/*
 * Upper bound of the workspace bytes cf_warp_backward_det needs for these shapes (0 for B == 0, C == 0 and for
 * shapes it rejects).  The batch is processed in chunks of Bc = min(B, floor((2^32 - 1) / (4*H*W))) items, so that
 * the n = 4*Bc*H*W tap records fit 32-bit keys and values.  Per chunk: four arrays of n uint32 (keys and values,
 * double-buffered by the sort), n float weights, Bc*H*W + 1 bucket starts, 256 * ceil(n / 4096) histogram counters
 * and, when the flow is at twice the image's resolution, 2*Bc*H*W floats of per-pixel flow gradients; each region
 * rounded up to 256 bytes, plus 256 bytes of alignment slack.  About 21 bytes per tap record (23 with the
 * half-resolution flow): 0.46 GB for the codes warp of 64 x 240x320 items, computed from this formula.
 */
CF_API size_t cf_warp_backward_det_workspace_bytes(int B, int C, int H, int W, int flowH, int flowW);

/*
 * The gradients of cf_warp_backward (same arguments, NULL rules and error codes), summed in a fixed order.
 * CF_ERR_WORKSPACE when the workspace is missing or shorter than cf_warp_backward_det_workspace_bytes.
 */
CF_API int cf_warp_backward_det(const float *grad_out, const float *img, const float *flow, float *grad_img,
                                float *grad_flow, int B, int C, int H, int W, int flowH, int flowW, float sign,
                                void *workspace, size_t workspace_bytes, cf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CISTAFLOW_DET_H_ */
