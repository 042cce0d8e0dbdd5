/* vlg_b200.h -- C ABI of the B200-native flow-guided warp + per-pixel loss path.
 *
 * One shared library (libvlg_b200.so), built for sm_100a only, no torch types in any signature.
 * Every entry point is stateless, re-entrant, stream-ordered and never synchronises the host;
 * the caller owns all buffers (device pointers unless stated) and the workspace.
 *
 * The reference (gongaa/video-layout-generation) has NO plugin / operator / FFI layer for this
 * path: its boundary is a set of Python call signatures (SURVEY.md section 8b).  Each entry point
 * below names the reference interface it stands behind:
 *
 *   vlg_pixel_loss_*      <- criterionL1(img, frame3)                 src/trainer.py:130,248,329
 *                            loss(output=img, target=frame3)          src/loss.py:20-25 (GradientLoss),
 *                                                                     src/loss.py:64-91 (SsimLoss), :61-62
 *                            cross_entropy_loss(input=seg, target=seg3)  src/trainer.py:124,250,331
 *                            composition 40/20/10                     src/trainer.py:248-251
 *   vlg_warp_fwd          <- (absent upstream) F.grid_sample(bilinear, align_corners=True) on the
 *                            src/models/modules.py:69 grid + torch.argmax(seg, 1) src/trainer.py:342,467
 *   vlg_warp_loss_*       <- the fused op that replaces src/trainer.py:248-258 when the producer
 *                            emits flow instead of pixels (SURVEY.md section 3.5)
 *   vlg_warp_loss_labels_fwd_bwd <- the same with the layout source as the class-id map the reference
 *                            actually holds (one_hot(label): src/models/net_utils.py:14-24, src/trainer.py:461)
 *   vlg_ingest            <- ToTensor src/data.py:33-35 + renormalisation src/trainer.py:193-195 + flip :200-206
 *                            + seg casts src/folder.py:97-100 + one-hot, from the dataset's uint8 arrays
 *   vlg_reduce_partials   <- the scalar losses handed to Trainer.sync  src/trainer.py:381-386
 *
 * Memory layout: activations are NHWC ("channels_last" storage of an NCHW-logical tensor),
 * dense, 16-byte aligned base pointers.  coords / d_coords are [N,H,W,2] fp32 (x/u first),
 * labels and argmax are int64 [N,H,W] (src/folder.py:100).
 */
#ifndef VLG_B200_H
#define VLG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VLG_VERSION 200 /* major*100 + minor */

/* activation dtype (coords, d_coords, loss outputs are always fp32; labels int64) */
#define VLG_F32 0
#define VLG_BF16 1

/* padding_mode of the sampler (SURVEY Appendix A.4; oracle default = border) */
#define VLG_PAD_ZEROS 0
#define VLG_PAD_BORDER 1

/* what `coords` holds */
#define VLG_COORD_FLOW 0 /* pixel-unit flow; grid = base + flow*2/(S-1) is built in-kernel */
#define VLG_COORD_GRID 1 /* a ready normalised sampling grid (align_corners=True)          */

/* flags */
#define VLG_FLAG_NO_FAR_PATH 1u /* caller asserts |displacement| < VLG_NEAR_RADIUS; far taps raise status */
#define VLG_FLAG_NO_TMA 2u      /* stage the source-layout window with cp.async instead of a TMA tensor map   */
#define VLG_FLAG_TILE_RGB 4u    /* evaluate the rgb terms in the tile kernel instead of the column-strip kernel */
#define VLG_FLAG_TILE_LAYOUT 8u /* evaluate the layout terms in the first (non-persistent) tile kernel            */
#define VLG_FLAG_FAR_WIDE 64u     /* far path: always one 64-bit accumulator per channel (default: two 32-bit lanes per 64-bit word in
                                   * every source-tile row that receives at most 512 far pixels)                                 */
#define VLG_FLAG_PASS2_COORDS 32u /* pass 2 re-derives the tap cells and weights from the coordinates and scans (pass2_kernel)
                                   * instead of registering the tap records pass 1 wrote (pass2_rec_kernel)            */

/* term_mask bits */
#define VLG_TERM_L1 1u
#define VLG_TERM_GD 2u
#define VLG_TERM_SSIM 4u
#define VLG_TERM_CE 8u
#define VLG_TERM_TV 16u
#define VLG_TERM_ALL 31u

/* ce_norm */
#define VLG_CE_NORM_TORCH 0u /* sum_p w[l_p] nll_p / sum_p w[l_p]   (torch 'mean'; w == 1 without weights) */
#define VLG_CE_NORM_COUNT 1u /* sum_p w[l_p] nll_p / #{labels != ignore_index}    (src/models/simple.py:56-59) */

/* error codes (negative) */
#define VLG_OK 0
#define VLG_ERR_ARG (-1)
#define VLG_ERR_UNSUPPORTED (-2)
#define VLG_ERR_CUDA (-3)
#define VLG_ERR_WORKSPACE (-4)

/* bits of the device status word (see vlg_read_status) */
#define VLG_STATUS_BAD_LABEL 1u  /* label outside [0,K) and != ignore_index */
#define VLG_STATUS_FAR_TAPS 2u   /* displacement >= VLG_NEAR_RADIUS while VLG_FLAG_NO_FAR_PATH was set */

/* Displacements below this many pixels take the atomics-free gather; larger ones the
 * fixed-point (integer, hence order-independent) far path. */
#define VLG_NEAR_RADIUS 3

/* slots of the fp32 loss vector written by vlg_reduce_partials */
#define VLG_LOSS_L1 0
#define VLG_LOSS_GD 1
#define VLG_LOSS_SSIM 2
#define VLG_LOSS_CE 3
#define VLG_LOSS_TV 4
#define VLG_LOSS_TOTAL 5   /* w_l1*L1 + w_gd*GD + w_ssim*SSIM + w_ce*CE + w_tv*TV (src/trainer.py:248-251) */
#define VLG_LOSS_NVALID 6  /* number of labels != ignore_index                                       */
#define VLG_LOSS_MAXDISP 7 /* max |sampling displacement| in pixels seen by the pass                */
#define VLG_LOSS_SLOTS 8

typedef struct vlg_problem {
    uint32_t struct_size; /* sizeof(vlg_problem_t) as the CALLER compiled it; checked by every entry point, so a
                           * stale binding (older, shorter struct) is refused instead of read out of bounds    */
    uint32_t abi_version; /* VLG_VERSION the caller was written against (major must match)               */
    int64_t N, H, W, K;   /* batch, output height/width (== source size), layout classes          */
    int32_t dtype;        /* VLG_F32 | VLG_BF16                                                    */
    int32_t padding;      /* VLG_PAD_*                                                             */
    int32_t coord_mode;   /* VLG_COORD_*                                                           */
    uint32_t flags;       /* VLG_FLAG_*                                                            */
    int64_t ignore_index; /* nn.CrossEntropyLoss default -100 (src/trainer.py:124)                 */
    float w_l1, w_gd, w_ssim, w_ce, w_tv; /* 40, 20, 20, 10 (src/trainer.py:248-250) + TV weight  */
    uint32_t term_mask;   /* VLG_TERM_* bits to evaluate; 0 = all.  Skipped terms read as 0 and add
                           * nothing to the total or to any gradient, whatever their weight.        */
    uint32_t ce_norm;     /* VLG_CE_NORM_*: divisor of the (weighted) cross-entropy sum                 */
    /* Divisors of the means.  0 = derive from N,H,W (single GPU).  Data-parallel ranks pass the
     * GLOBAL batch here so that per-rank loss vectors and gradients simply add (SURVEY 8e). */
    int64_t global_N;
    /* Optional per-class CE weights (device pointer, K floats; NULL = unweighted).  The reference's
     * class-weighted variant: F.cross_entropy(weight=w, reduction='sum') / n_known, src/models/simple.py:56-59
     * (= VLG_CE_NORM_COUNT); nn.CrossEntropyLoss(weight=w) semantics are VLG_CE_NORM_TORCH. */
    const float *ce_class_weight;
} vlg_problem_t;

int vlg_version(void);
/* Thread-local description of the last error returned on this thread ("" if none). */
const char *vlg_last_error(void);

/* Bytes of caller-supplied device workspace needed by the vlg_warp_loss_* / vlg_pixel_loss_*
 * entry points for this problem (16-byte aligned; contents need no initialisation).
 * `with_src_grad` != 0 adds the d_out staging the deterministic source-gradient pass reads. */
size_t vlg_workspace_bytes(const vlg_problem_t *prob, int with_src_grad);

/* Forward warp only (validation / rollout, src/trainer.py:329-342,460-469):
 *   out_rgb    [N,H,W,3]  = warp(src_rgb)         (nullable)
 *   out_layout [N,H,W,K]  = warp(src_layout)      (nullable)
 *   out_argmax [N,H,W] i64 = argmax_k out_layout  (nullable; first max on ties)
 *   dbg_x0y0   [N,H,W,2] i32 floor source indices (nullable; bit-exact index witness) */
int vlg_warp_fwd(const vlg_problem_t *prob, const void *src_rgb, const void *src_layout,
                 const float *coords, void *out_rgb, void *out_layout, int64_t *out_argmax,
                 int32_t *dbg_x0y0, void *stream);

/* Rollout warp with LABEL sources (autoregressive feedback of src/trainer.py:460-469: the layout fed
 * back is argmax -> one-hot, so the K-channel gather collapses to four int64 taps):
 *   out_rgb   [N,H,W,3]   = warp(src_rgb)                                   (nullable with src_rgb)
 *   out_label [N,H,W] i64 = argmax_k warp(one_hot(src_label))_k, bit-exact with the dense path
 * prob->K is only validated, not used. */
int vlg_warp_fwd_labels(const vlg_problem_t *prob, const void *src_rgb, const int64_t *src_label,
                        const float *coords, void *out_rgb, int64_t *out_label, void *stream);

/* Layout visualisation (src/trainer.py:416-427 vis_seg_mask, src/val.py:178): colour = lut[class]/255.
 *   layout [N,H,W,K] (argmax taken here, first max on ties)  XOR  label [N,H,W] i64
 *   lut_rgb: K*3 bytes on the device;  out_rgb [N,H,W,3];  out_label nullable (argmax output) */
int vlg_colorize(const vlg_problem_t *prob, const void *layout, const int64_t *label,
                 const uint8_t *lut_rgb, void *out_rgb, int64_t *out_label, void *stream);

/* One-hot layout encoding (src/models/net_utils.py:14-24 transform_seg_one_hot:
 * torch.eye(K)[seg.long()].permute(0,3,1,2)): label [N,H,W] as int64 XOR float32 class ids (the dataset
 * hands float maps, src/folder.py:97-99; values are truncated like .long()) -> layout [N,H,W,K] of the
 * problem's dtype.  Labels outside [0,K) raise VLG_STATUS_BAD_LABEL in `workspace`'s status word when a
 * workspace is given and produce an all-zero pixel. */
int vlg_one_hot(const vlg_problem_t *prob, const int64_t *label_i64, const float *label_f32,
                void *out_layout, void *workspace, void *stream);

/* Boundary fusion around the path (SURVEY 8a-10, 8f-3): per-channel affine renormalisation of rgb frames,
 * horizontal flip and NCHW -> NHWC re-layout in one pass; bit-identical to the reference's torch ops.
 *   denormalize == 0:  out = (in - a[c]) / b[c]   src/trainer.py:193-195 (img_mean_arr, img_std_arr), :212,:324
 *   denormalize != 0:  out = in * b[c] + a[c]     src/trainer.py:215
 *   flip_w: torch.flip(frame, [3]) and torch.flip(seg3, [2])   src/trainer.py:200-206
 *   in_rgb  fp32, [N,3,H,W] contiguous (in_is_nchw != 0, what the DataLoader hands) or [N,H,W,3]
 *   a3, b3  HOST pointers to 3 floats each (passed to the kernel by value)
 *   out_rgb [N,H,W,3] of the problem's dtype;  label_in/label_out [N,H,W] i64 (nullable pair)
 * prob->K, padding, coord_mode are ignored. */
int vlg_frame_affine(const vlg_problem_t *prob, const float *in_rgb, int32_t in_is_nchw, const float *a3,
                     const float *b3, int32_t denormalize, int32_t flip_w, void *out_rgb,
                     const int64_t *label_in, int64_t *label_out, void *stream);

/* Pass 1 of the fused op: warp + all loss terms + d(loss)/d(warped) + d(loss)/d(coords) in one
 * kernel.  Gradients are for an upstream grad of 1.0 (see vlg_scale_grads).
 *   tgt_rgb [N,H,W,3], tgt_label [N,H,W] i64
 *   d_coords [N,H,W,2] fp32 (nullable = forward/validation only: no gradient work, no d_out)
 *   out_argmax nullable.
 * Writes per-block partial sums and (if with_src_grad) d_out into `workspace`. */
int vlg_warp_loss_bwd_out(const vlg_problem_t *prob, const void *src_rgb, const void *src_layout,
                          const float *coords, const void *tgt_rgb, const int64_t *tgt_label,
                          float *d_coords, int64_t *out_argmax, int with_src_grad,
                          void *workspace, size_t workspace_bytes, void *stream);

/* vlg_warp_loss_bwd_out with the final reduction fused in: the last pass-1 CTA writes loss_out[VLG_LOSS_SLOTS]
 * (nullable), so the loss vector is complete BEFORE pass 2 starts -- a data-parallel caller issues its one
 * all-reduce of the loss vector (src/trainer.py:381-386) here and lets it overlap vlg_warp_bwd_src. */
int vlg_warp_loss_pass1(const vlg_problem_t *prob, const void *src_rgb, const void *src_layout,
                        const float *coords, const void *tgt_rgb, const int64_t *tgt_label, float *loss_out,
                        float *d_coords, int64_t *out_argmax, int with_src_grad, void *workspace,
                        size_t workspace_bytes, void *stream);

/* Pass 2: deterministic source gradient (no float atomics): every source pixel gathers, in a
 * fixed order, the d_out of the output pixels whose bilinear footprint covers it.
 *   d_src_rgb [N,H,W,3], d_src_layout [N,H,W,K] (either nullable) */
int vlg_warp_bwd_src(const vlg_problem_t *prob, const float *coords, void *d_src_rgb,
                     void *d_src_layout, void *workspace, size_t workspace_bytes, void *stream);

/* Fixed-order fp64 reduction of the per-block partials into loss_out[VLG_LOSS_SLOTS] (fp32). */
int vlg_reduce_partials(const vlg_problem_t *prob, float *loss_out, void *workspace,
                        size_t workspace_bytes, void *stream);

/* Convenience: pass 1 + reduce (+ pass 2 when d_src_* given) on one stream. */
int vlg_warp_loss_fwd_bwd(const vlg_problem_t *prob, const void *src_rgb, const void *src_layout,
                          const float *coords, const void *tgt_rgb, const int64_t *tgt_label,
                          float *loss_out, float *d_coords, void *d_src_rgb, void *d_src_layout,
                          int64_t *out_argmax, void *workspace, size_t workspace_bytes, void *stream);

/* The fused op with a LABEL layout source (SURVEY 8f-2): src_label [N,H,W] i64 stands for one_hot(src_label)
 * (src/models/net_utils.py:14-24; the rollout feeds argmax maps back the same way, src/trainer.py:461,467).  Sources are
 * data here, as in the reference: the gradient goes to the coordinates only (d_coords nullable = validation).
 *   out_argmax == argmax_k warp(one_hot(src_label))_k bit for bit; losses / d_coords equal the dense path's on
 *   one-hot inputs to fp32 rounding (same formulas, sums over the <= 4 non-zero channels instead of K).
 * Workspace: vlg_workspace_bytes(prob, 0). */
int vlg_warp_loss_labels_fwd_bwd(const vlg_problem_t *prob, const void *src_rgb, const int64_t *src_label,
                                 const float *coords, const void *tgt_rgb, const int64_t *tgt_label, float *loss_out,
                                 float *d_coords, int64_t *out_argmax, void *workspace, size_t workspace_bytes,
                                 void *stream);

/* Ingest of what the dataset holds (src/folder.py:85-104: uint8 RGB frames [N,H,W,3] from cv2, uint8 class maps
 * [N,H,W]) in one pass per tensor, bit-identical to the reference's torch expressions:
 *   out_frames [N,H,W,3] of the problem's dtype = ((u8 / 255) - mean[c]) / std[c]   ToTensor src/data.py:33-35, then
 *              src/trainer.py:193-195; mean3 == NULL: u8 / 255 only.  mean3 / std3 are HOST pointers to 3 floats.
 *   flip_w     torch.flip(frame, [3]) / torch.flip(seg, [2])                         src/trainer.py:200-206
 *   out_label  [N,H,W] i64 = seg.long()                       src/folder.py:100      (nullable)
 *   out_seg_f32 [N,H,W] f32 = seg.float()                     src/folder.py:97-99    (nullable)
 *   out_onehot [N,H,W,K] of the problem's dtype               src/models/net_utils.py:14-24 (nullable)
 * Either of (frames_u8, out_frames) / (seg_u8, outputs) may be NULL pairs.  `workspace` (nullable) receives
 * VLG_STATUS_BAD_LABEL for class ids >= K when a one-hot layout is written. */
int vlg_ingest(const vlg_problem_t *prob, const uint8_t *frames_u8, const float *mean3, const float *std3, int32_t flip_w,
               void *out_frames, const uint8_t *seg_u8, int64_t *out_label, float *out_seg_f32, void *out_onehot,
               void *workspace, void *stream);

/* The reference's own loss call sites without a warp: `output` rgb [N,H,W,3] vs `target`,
 * `logits` [N,H,W,K] vs `tgt_label`.  Any of (out_rgb+tgt_rgb) / (logits+tgt_label) may be NULL
 * to evaluate a single criterion.  d_out_rgb / d_logits nullable (validation).  prob->coord_mode
 * and padding are ignored. */
int vlg_pixel_loss_fwd_bwd(const vlg_problem_t *prob, const void *out_rgb, const void *tgt_rgb,
                           const void *logits, const int64_t *tgt_label, float *loss_out,
                           void *d_out_rgb, void *d_logits, int64_t *out_argmax, void *workspace,
                           size_t workspace_bytes, void *stream);

/* g <- g * (*scale) for n fp32/bf16 elements; exits at once when *scale == 1.0f (the common
 * `loss.backward()` case), so autograd semantics cost one empty launch.  `scale` is a device ptr. */
int vlg_scale_grads(void *g, int64_t n, int32_t dtype, const float *scale, void *stream);

/* The same for `count` (<= 4) buffers in one launch: g[b] has n[b] elements of dtype[b] (HOST arrays of device
 * pointers / sizes / dtypes, read at call time).  What `loss.backward()` (src/trainer.py:257) costs the fused op: one
 * launch that finds *scale == 1.0f and exits, instead of one per gradient tensor. */
int vlg_scale_grads_multi(int32_t count, void *const *g, const int64_t *n, const int32_t *dtype, const float *scale,
                          void *stream);

/* Copies the device status word (VLG_STATUS_*) to *host_status.  Synchronises `stream`. */
int vlg_read_status(void *workspace, size_t workspace_bytes, uint32_t *host_status, void *stream);

/* Number of kernels the library has launched in this process (for bench.py's gpu_launches). */
int64_t vlg_launch_count(void);

/* Measurement aid (bench.py's per-kernel roofline; no reference counterpart).  While armed on the calling thread
 * (on != 0), vlg_warp_loss_* / vlg_warp_bwd_src record CUDA events on their launch stream right before and after the
 * three main kernels of the step.  vlg_timeline_read waits for the last recorded event and returns device times in
 * milliseconds of the most recent armed call sequence: ms4[0] rgb_strip_kernel, ms4[1] lay_tile_kernel, ms4[2] the
 * pass-2 gather kernel, ms4[3] first event to last event; -1 where a kernel did not run.  Do not arm while the
 * stream is being captured into a CUDA graph. */
int vlg_timeline_arm(int on);
int vlg_timeline_read(float *ms4);

#ifdef __cplusplus
}
#endif
#endif /* VLG_B200_H */
