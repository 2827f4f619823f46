/*
 * cistaflow.h -- C ABI of libcistaflow.so: the CISTA-Flow per-frame
 * motion-compensation hot path as hand-written sm_100a (B200) CUDA.
 *
 * The reference (lsying009/CISTA-Flow) is pure Python: it has no FFI of its own
 * (SURVEY.md F1), its boundary is a set of Python functions/classes.  Each entry
 * point below names the reference interface it replaces (file:line, relative to
 * the reference checkout).  The Python mirror of those interfaces lives in
 * cista-flow_b200/ and binds this header through ctypes (INTEGRATION.md shows the
 * stub a reference maintainer would add).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the parameter is documented as
 *     "host array"; the library never allocates or frees device memory and never
 *     synchronises the host: all work is enqueued on `stream` (graph-capturable);
 *   - tensors are dense, row-major ("NCHW"), float32 unless stated;
 *   - float32/float64 tensors must be 16-byte aligned (torch allocations are);
 *   - return value: CF_OK (0) or a negative cf_status; cf_last_error() returns a
 *     thread-local human-readable message for the last failure;
 *   - there is no CPU fallback: on a device that is not compute capability 10.x
 *     every compute entry point returns CF_ERR_ARCH.
 */
#ifndef CISTAFLOW_H_
#define CISTAFLOW_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CISTAFLOW_VERSION 100 /* major*10000 + minor*100 + patch */

#if defined(__GNUC__)
#define CF_API __attribute__((visibility("default")))
#else
#define CF_API
#endif

typedef void *cf_stream_t; /* a cudaStream_t */

typedef enum cf_status {
    CF_OK = 0,
    CF_ERR_INVALID_ARG = -1, /* bad shape / size / enum value              */
    CF_ERR_NULL = -2,        /* required pointer is NULL                    */
    CF_ERR_ALIGN = -3,       /* pointer not 16-byte aligned                 */
    CF_ERR_ARCH = -4,        /* current device is not sm_100 (B200)         */
    CF_ERR_WORKSPACE = -5,   /* workspace missing or too small              */
    CF_ERR_CUDA = -6,        /* a CUDA runtime/driver call failed           */
    CF_ERR_UNSUPPORTED = -7  /* valid request this build does not implement */
} cf_status;

CF_API int cf_version(void);
CF_API const char *cf_last_error(void);
/* CF_OK when the CURRENT device can run the kernels (compute capability 10.x). */
CF_API int cf_device_check(void);
/* Number of CUDA kernels this library has launched (or recorded into a graph
 * capture) in this process so far; benchmarks report it as evidence that the
 * hand-written kernels -- not a fallback -- did the work. */
CF_API int64_t cf_launch_count(void);
/* Name of the kernel this process launched last ("" before the first launch): lets tests assert
 * WHICH of the data-movement variants of an entry point ran (e.g. the TMA-staged warp kernel
 * vs the direct gather it falls back to on discontinuous flow). */
CF_API const char *cf_last_kernel(void);

/* ------------------------------------------------------------------------- *
 * Part 1: event stream -> voxel grid (+ normalisation)
 * replaces  utils/event_process.py:15-72    events_to_voxel_grid        (flavour NUMPY)
 *           utils/event_process.py:127-190  events_to_voxel_grid_pytorch (flavour TORCH)
 *           utils/event_process.py:75-123   events_to_voxel_grid_pol     (flavour POL)
 *           utils/event_process.py:193-239  event_preprocess(_pytorch)   (preprocess != NONE)
 *           data_readers/MVSEC_utils.py:253-303  events_to_voxel_torch   (flavour MVSEC; SURVEY.md 8f rank 4;
 *                                                same code in DCEIFlow/utils/event_uitls.py:91-141)
 * ------------------------------------------------------------------------- */
typedef enum cf_voxel_mode {
    CF_VOXEL_ATOMIC = 0,        /* fast: fp32 atomics, sum order unspecified (<= 1e-5 rel.);  */
                                /* runs the L2 path (the tiled one only when forced, below)   */
    CF_VOXEL_DETERMINISTIC = 1, /* bit-exact: per-cell sums in the reference's event order    */
    CF_VOXEL_ATOMIC_L2 = 2,     /* ATOMIC, forced path: RED.ADD into the L2-resident grid     */
    CF_VOXEL_ATOMIC_TILED = 3   /* ATOMIC, forced path: partition + shared-memory tiles;      */
                                /* CF_ERR_UNSUPPORTED when the geometry does not fit          */
} cf_voxel_mode;

typedef enum cf_voxel_flavour {
    CF_FLAVOUR_TORCH = 0, /* fp32 weights, fp32 adds                  (event_process.py:166-187) */
    CF_FLAVOUR_NUMPY = 1, /* fp64 weights, fp64 add rounded to fp32    (event_process.py:56-66)   */
    CF_FLAVOUR_POL = 2,   /* [nb,2,H,W], channel = polarity, |weights| (event_process.py:104-119) */
    CF_FLAVOUR_MVSEC = 3  /* the second voxeliser: t* = ((t-t0)/dT)*(nb-1) (divide first), weight p*max(0,1-|t*-bin|)
                             with p used AS IS (0 contributes nothing), fp64 weights cast to fp32, fp32 adds; per cell
                             and bin the sequential order is "events of bin-1 (right weights) before events of bin"
                             (MVSEC_utils.py:283-292: one index_put_ per bin over the time-sorted events) */
} cf_voxel_flavour;

typedef enum cf_preprocess {
    CF_PRE_NONE = 0,
    CF_PRE_STD = 1,   /* mask*(v-mean)/(std+1e-8) over the NON-ZERO entries of each window */
    CF_PRE_MAXMIN = 2 /* (v-min)/(max-min+1e-8)                                            */
} cf_preprocess;

/*
 * events   float64 [total_events, 4] rows (t, x, y, p); the windows are
 *          concatenated, each sorted by t; p == 0 means negative polarity.
 *          fp64 is part of the contract: absolute stamps do not fit fp32
 *          (data_readers/event_readers.py:15-20, SURVEY.md F10).
 * offsets  int64 [B+1] (DEVICE), window b = rows [offsets[b], offsets[b+1]).
 *          Rows outside [offsets[0], offsets[B]) belong to no window and are
 *          ignored by every mode (offsets need not start at 0 nor end at
 *          total_events).
 * out      float32 [B, nb, H, W]   (flavour POL: [B, nb, 2, H, W]).
 * hot_thr  > 0: entries with |v| > hot_thr are zeroed before the statistics
 *          (25/nb in event_preprocess, 20/nb in event_preprocess_pytorch);
 *          <= 0 disables.  Ignored when preprocess == CF_PRE_NONE.
 * Events whose (x, y) fall outside the grid are dropped (the reference would
 * raise IndexError; its callers pre-filter, data_readers/video_readers.py:208).
 * An empty window yields an all-zero grid (event_process.py:36-37).
 * The window statistics of preprocess != NONE (sum, sum of squares, count)
 * are accumulated in fp64; only the per-cell map is fp32.
 */
CF_API size_t cf_voxel_workspace_bytes(int64_t total_events, int B, int nb, int H, int W,
                                int mode, int flavour, int preprocess);
CF_API int cf_voxel_bin(const double *events, const int64_t *offsets, int64_t total_events,
                 int B, int nb, int H, int W, int mode, int flavour,
                 int preprocess, float hot_thr, float *out,
                 void *workspace, size_t workspace_bytes, cf_stream_t stream);

/* event_preprocess(_pytorch) on an existing batch of grids [B, C, H, W]
 * (utils/event_process.py:193-239).  in == out is allowed. */
CF_API size_t cf_preprocess_workspace_bytes(int B, int64_t cells_per_window);
CF_API int cf_voxel_preprocess(const float *in, float *out, int B, int64_t cells_per_window,
                        int preprocess, float hot_thr,
                        void *workspace, size_t workspace_bytes, cf_stream_t stream);

/* ------------------------------------------------------------------------- *
 * Part 1b: packed event ingest (SURVEY.md section 8f, rank 3) -- 8 bytes per event
 * narrows the fp64 rows of data_readers/event_readers.py:6-47 to
 *   word 0  float32 t_rel = (float)(t - t_first_of_window)   (fp64 subtraction first)
 *   word 1  uint32  x | y << 16 | p << 31                    (x < 65535, y < 32768)
 * ------------------------------------------------------------------------- */
/* events float64 [total,4] + offsets int64 [B+1] (as cf_voxel_bin) -> packed uint64 [total].
 * A row outside [offsets[0], offsets[B]) gets the invalid record (x = 0xffff, t_rel = 0), which
 * cf_voxel_bin_packed never visits; pack_events_host writes the same bits. */
CF_API int cf_events_pack(const double *events, const int64_t *offsets, int64_t total_events, int B,
                   void *packed, cf_stream_t stream);
/* Device-side windowing (what data_readers/video_readers.py:208-232 and data_readers/event_readers.py:6-47 do on the host
 * before every frame), so that a raw event stream uploaded once is cut into voxel windows without a read-back:
 *   cf_events_filter   rows with x < W and y < H (video_readers.py:208-209; no lower bound, like the reference), stable,
 *                      compacted into out [<= total,4]; *kept (device int64) = rows kept.
 *                      workspace: cf_events_filter_workspace_bytes(total).
 *   cf_event_window_offsets   offsets [max_windows+1] from a DEVICE-resident count:
 *                      CF_WINDOWS_FIXED  windows of `param` events, the last keeps the remainder (FixedSizeEventReader)
 *                      CF_WINDOWS_SPLIT  np.array_split into max(1, round(count / param)) windows (limit_num_events)
 *                      more windows than max_windows: FIXED keeps max_windows windows of `param` events and the last
 *                      keeps the rest; SPLIT splits the count evenly over max_windows windows;
 *                      entries past the last window = count (empty windows); *n_windows (device int, may be NULL). */
enum cf_window_policy { CF_WINDOWS_FIXED = 0, CF_WINDOWS_SPLIT = 1 };
CF_API size_t cf_events_filter_workspace_bytes(int64_t total_events);
CF_API int cf_events_filter(const double *events, int64_t total_events, int W, int H, double *out, int64_t *kept,
                     void *workspace, size_t workspace_bytes, cf_stream_t stream);
CF_API int cf_event_window_offsets(const int64_t *count, int policy, int64_t param, int64_t *offsets, int max_windows,
                            int *n_windows, cf_stream_t stream);
/* Voxel grid [B, nb, H, W] (+ fused event_preprocess) from packed events; ATOMIC numerics
 * (|err| <= 1e-5 * (sum|w| + 1) per cell against the fp64 reference), polarity 0 -> -1 like
 * events_to_voxel_grid.  workspace: cf_preprocess_workspace_bytes(B, nb*H*W) when preprocess != NONE. */
CF_API int cf_voxel_bin_packed(const void *packed, const int64_t *offsets, int64_t total_events,
                        int B, int nb, int H, int W, int preprocess, float hot_thr, float *out,
                        void *workspace, size_t workspace_bytes, cf_stream_t stream);

/* ------------------------------------------------------------------------- *
 * Part 2: flow-guided bilinear warp (a gather in BOTH warp modes)
 * replaces  utils/flow_utils.py:153-190  forwardWarp.forward  (sign = -1)
 *           utils/flow_utils.py:83-120   backWarp.forward     (sign = +1)
 *           utils/flow_utils.py:212-221  FrameWarp.warp_frame
 * ------------------------------------------------------------------------- */
/*
 * img   [B, C, H, W];  out [B, C, H, W];  flow [B, 2, flowH, flowW], ch0 = u (x).
 * flowH == H && flowW == W : flow is used as is.
 * H == flowH/2 && W == flowW/2 (integer division) : the x0.5 bilinear
 *   align_corners=True down-sampling of e2v/e2v_model.py:190 is fused into the
 *   kernel (flow values are NOT rescaled, as in the reference).
 * Sample position ((x + sign*u) * (W-1)/W, (y + sign*v) * (H-1)/H) -- the
 * reference's 2*(x/W-0.5) normalisation under align_corners=True -- reflected
 * about [0, W-1] x [0, H-1] (padding_mode='reflection').
 */
CF_API int cf_warp(const float *img, const float *flow, float *out, int B, int C, int H, int W,
            int flowH, int flowW, float sign, cf_stream_t stream);

/* The per-frame step of e2v/e2v_model.py:188-191 in one launch: warps the
 * previous reconstruction img [B,Ci,H,W] with the full-resolution flow and the
 * sparse codes [B,Cz,H/2,W/2] with the fused half-resolution flow. */
CF_API int cf_warp_frame_and_codes(const float *img, const float *codes, const float *flow,
                            float *img_out, float *codes_out, int B, int Ci, int Cz,
                            int H, int W, float sign, cf_stream_t stream);

/* Device-side form of `if not flow_final.any(): warped_I = rec_img0 (states untouched)`
 * (e2v/e2v_model.py:184-191, 236-243; SURVEY.md section 8f rank 1): the reference reads the predicate back to
 * the host -- a synchronisation in every frame, and the reason the frame step cannot be captured in a CUDA graph.
 *   cf_flow_any       flag[0] = 1 iff any of the n floats of flow is non-zero (NaN counts, -0.0 does not:
 *                     torch.Tensor.any()); flag is a device int, zeroed and written on `stream`.
 *   ..._gated         as cf_warp_frame_and_codes, but when gate != NULL and *gate == 0 the outputs are COPIES of
 *                     img / codes (what the reference's branch returns; a zero flow is not the identity under its
 *                     grid normalisation).  gate == NULL: always warp.  No host synchronisation, graph-capturable. */
CF_API int cf_flow_any(const float *flow, int64_t n, int *flag, cf_stream_t stream);
CF_API int cf_warp_frame_and_codes_gated(const float *img, const float *codes, const float *flow,
                                  float *img_out, float *codes_out, int B, int Ci, int Cz,
                                  int H, int W, float sign, const int *gate, cf_stream_t stream);

/* The frame step from the flow network's own output (SURVEY.md section 8f rank 1, completed in round 2): DCEIFlow
 * predicts the flow at 1/8 of the x32-padded frame; the reference up-samples it with upflow8
 * (DCEIFlow/DCEIFlow.py:222, DCEIFlow/utils/sample_utils.py:66-68: x8 bilinear, align_corners=True, values x8), cuts the
 * top/left padding off (ImagePadder.unpad, utils/image_process.py:103-107), and only then warps the previous frame and
 * -- after another x0.5 bilinear down-sampling -- the sparse codes (e2v/e2v_model.py:188-191).  One launch does all of it:
 *   flow_lr   [B,2,lh,lw]  coords1 - coords0 of the last refinement iteration, lh = (H + pad_h)/8, lw = (W + pad_w)/8
 *   flow_out  [B,2,H,W] or NULL: the up-sampled, un-padded flow (what the model returns as batch_flow['flow_final'])
 *   img [B,Ci,H,W], codes [B,Cz,H/2,W/2] and their outputs as in cf_warp_frame_and_codes.
 * Same arithmetic, operation by operation, as the reference's three ATen calls followed by cf_warp_frame_and_codes. */
CF_API int cf_warp_frame_and_codes_upflow8(const float *img, const float *codes, const float *flow_lr, float *img_out,
                                    float *codes_out, float *flow_out, int B, int Ci, int Cz, int H, int W,
                                    int lh, int lw, int pad_h, int pad_w, float sign, cf_stream_t stream);

/* Adjoint of cf_warp (SURVEY.md section 8f, rank 2): what autograd runs through forwardWarp / backWarp in
 * training (loss.py:147,336,398; train.py:208-232).  grad_out [B,C,H,W];
 *   grad_img  [B,C,H,W]           <- bilinear SPLAT of grad_out into the 4 taps (may be NULL)
 *   grad_flow [B,2,flowH,flowW]   <- through reflect/clip and the 2*(x/W-0.5) normalisation; with the fused x0.5
 *                                    down-sampling (H == flowH/2) its adjoint is applied too (may be NULL; needs img)
 * Both outputs are zeroed by the call; accumulation order is unspecified (fp32 atomics), as in ATen's CUDA backward. */
CF_API int cf_warp_backward(const float *grad_out, const float *img, const float *flow, float *grad_img,
                     float *grad_flow, int B, int C, int H, int W, int flowH, int flowW, float sign,
                     cf_stream_t stream);

/* Flow-warp of a voxel grid for the FWL metric (SURVEY.md section 8f, rank 4)
 * replaces  loss.py:27-83  voxel_warping_flow_loss   (call sites test_wo_flow.py:161, test_mvsec.py:180)
 * voxel [B,C,H,W], displacement [B,2,H,W] (ch0 = x).  Channel i is sampled (bilinear, zeros padding,
 * align_corners=True, grid 2*coord/size - 1) at (x + dx*r_i, y + dy*r_i), r_i = i/(C-1), or 1 - i/(C-1)
 * with the displacement negated when reverse_time != 0.
 * warped   [B,C,H,W] the warped channels (may be NULL);  summed [B,1,H,W] their sum;
 * mean_var device double[2] <- mean and UNBIASED variance of `summed` over the batch (may be NULL;
 *          needs cf_voxel_flow_warp_workspace_bytes(B, H, W) bytes of workspace). */
CF_API size_t cf_voxel_flow_warp_workspace_bytes(int B, int H, int W);
CF_API int cf_voxel_flow_warp(const float *voxel, const float *displacement, int B, int C, int H, int W,
                       int reverse_time, float *warped, float *summed, double *mean_var,
                       void *workspace, size_t workspace_bytes, cf_stream_t stream);

/* ------------------------------------------------------------------------- *
 * Part 3: all-pairs correlation volume, pyramid and lookup
 * replaces  ERAFT/corr.py:13-27,52-60  CorrBlock.__init__ / CorrBlock.corr
 *           ERAFT/corr.py:29-50        CorrBlock.__call__
 *           DCEIFlow/core/corr/raft_corr.py:16-65 (identical maths)
 * ------------------------------------------------------------------------- */
typedef enum cf_corr_precision {
    CF_CORR_TF32 = 0, /* tcgen05.mma kind::tf32, fp32 accumulate in TMEM (default)  */
    CF_CORR_FP32 = 1, /* SIMT FFMA, fp32 operands (reference arithmetic)             */
    CF_CORR_3XTF32 = 2, /* tcgen05.mma kind::tf32 on split operands (workspace): x = hi + lo, hi = rn_tf32(x),
                           lo = rn_tf32(x - hi), three MMAs per K step (lo.hi + hi.lo + hi.hi) into one fp32 accumulator.
                           Within ~2^-22 of the exact products: fp32 accuracy at three times the TF32 MMA work.  Same
                           shapes as TF32 (CF_ERR_UNSUPPORTED elsewhere).  Workspace: 4 * round_up(B*D*h*w*4, 256) bytes */
    CF_CORR_F16 = 3,    /* tcgen05.mma kind::f16 on fp16 operand COPIES (workspace): same 11-bit significand as a TF32
                           operand, scaled per batch item by a power of two so that every finite input fits; K = 16
                           per MMA and half the operand bytes.  Within fp32 summation-order noise of TF32; faster than
                           TF32 on wide maps with many tiles, which is where CF_CORR_AUTO selects it */
    CF_CORR_AUTO = 4    /* the library's choice by shape: fp16 operand copies for wide maps (N % 64 == 0, many tiles), else TF32 */
} cf_corr_precision;

#define CF_CORR_MAX_LEVELS 6

/*
 * fmap1, fmap2  [B, D, h, w];  pyramid[l]  [B*h*w, 1, h>>l, w>>l]  (host array of
 * `levels` device pointers).  pyramid[0][b*N+i, 0, y, x] =
 * <fmap1[b,:,i], fmap2[b,:,y*w+x]> / sqrt(D); level l+1 = avg_pool2d(level l, 2, 2)
 * (odd sizes are floored).
 */
CF_API size_t cf_corr_workspace_bytes(int B, int D, int h, int w, int levels, int precision);
CF_API int cf_corr_build(const float *fmap1, const float *fmap2, int B, int D, int h, int w,
                  int levels, float *const *pyramid, int precision,
                  void *workspace, size_t workspace_bytes, cf_stream_t stream);

/*
 * coords [B, 2, h, w] (ch0 = x, ch1 = y, level-0 feature-map pixels);
 * out [B, levels*(2r+1)^2, h, w]; channel l*(2r+1)^2 + i*(2r+1) + j is level l
 * sampled bilinearly (zero outside) at (x/2^l + i - r, y/2^l + j - r): i runs
 * along X -- the reference's transposed window (ERAFT/corr.py:37-43).
 */
CF_API int cf_corr_lookup(const float *const *pyramid, const float *coords, int B, int h, int w,
                   int levels, int radius, float *out, cf_stream_t stream);

/* Adjoint of cf_corr_lookup (SURVEY.md section 8f, rank 2; training through CorrBlock.__call__).
 * grad_out [B, levels*(2r+1)^2, h, w];
 *   grad_pyramid[l] [B*h*w, 1, h>>l, w>>l]  (host array of device pointers; zeroed by the call; may be NULL)
 *   grad_coords     [B, 2, h, w]            (may be NULL; needs `pyramid`)
 * No atomics: every query owns its maps, each patch element is written once. */
CF_API int cf_corr_lookup_backward(const float *grad_out, const float *const *pyramid, const float *coords,
                            int B, int h, int w, int levels, int radius, float *const *grad_pyramid,
                            float *grad_coords, cf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CISTAFLOW_H_ */
