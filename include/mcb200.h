/*
 * mcb200.h — C-ABI of libmcb200.so: the B200 (sm_100a) hot path of
 * AnishDelft/ModelCompression (pruned YOLOv2-VOC forward, pruning masks, region decode + NMS).
 *
 * The reference has no FFI layer: its hot path is PyTorch/NumPy library calls made from Python
 * (SURVEY.md §8b).  Each entry point below names the reference call site it replaces
 * (paths under the reference repo root).  The Python package `modelcompression_b200` binds these
 * with ctypes and re-exposes the reference's own function/class names.
 *
 * Conventions
 *   - every pointer named d_* is a DEVICE pointer owned by the caller; h_* is a HOST pointer.
 *   - the library never allocates or frees device memory; scratch is passed as (d_ws, ws_bytes)
 *     and sized by the matching mc_workspace_bytes_* function.
 *   - `stream` is a cudaStream_t passed as void*; all calls are asynchronous on it.
 *   - return 0 on success; <0 on error: -1 bad argument, -2 unsupported shape,
 *     -3 workspace too small, -(1000+cudaError_t) CUDA failure.
 *     mc_last_error_string() gives the thread-local message for the last failure.
 *   - sm_100a only.  There is no CPU fallback.
 */
#ifndef MCB200_H_
#define MCB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MCB200_VERSION 100
#define MC_MAX_SEGMENTS 64 /* max tensors per multi-tensor launch (YOLOv2-VOC has 23 conv weights) */

int mc_version(void);
const char* mc_last_error_string(void);
/* 1 if the current device is compute capability 10.x, else 0 (or <0 on CUDA error). */
int mc_device_ok(void);

/* ------------------------------------------------------------------------------------------
 * Magnitude (weight) pruner — replaces src/pruning/weightPruning/methods.py:9-26 (weight_prune):
 *   all_weights = concat(|p| for p in params if p.dim()!=1); thr = np.percentile(all_weights, perc)
 *   mask = (|p| > thr).float()
 * and the apply half of MaskedConv2d.set_mask (src/pruning/weightPruning/layers.py:41-47).
 * -------------------------------------------------------------------------------------------- */

/* Exact order statistics of |w| over `nseg` fp32 tensors (n = sum of h_sizes):
 *   a = sorted(|w|)[k], b = sorted(|w|)[min(k+1, n-1)]
 *   d_out[0] = thr = NumPy's _lerp(a, b, gamma) in float32 (gamma==0 -> a); d_out[1] = a; d_out[2] = b.
 * k and gamma are the data-independent "virtual index" pieces of np.percentile, computed by the host
 * (modelcompression_b200/pruning/weightPruning/methods.py).  Radix select on the fp32 bit pattern of |w|
 * (monotone as uint32), so the result is bit-exact.                                                    */
int mc_kth_abs_select(const float* const* h_seg_ptrs, const int64_t* h_seg_sizes, int nseg,
                      int64_t k, float gamma, float* d_out3,
                      void* d_ws, size_t ws_bytes, void* stream);
size_t mc_workspace_bytes_kth_abs_select(int64_t n_total);

/* The whole of weight_prune in ONE cooperative launch: the order statistics as above (same d_out3) AND
 * mask[i] = (|w[i]| > thr) ? 1.f : 0.f for every segment.  Fast path: pivots from a sample bracket the rank-k key,
 * one pass over W writes provisional masks and collects the bracketed ~5 % as candidates, the exact rank is resolved
 * on the candidates and only their masks are fixed up (HBM traffic 8n bytes: read W once, write masks once).  A missed
 * bracket falls back, inside the same launch, to an exact 12+10+9-bit radix select and a full mask pass.
 * Workspace: mc_workspace_bytes_kth_abs_select(n).                                                    */
int mc_weight_prune_masks(const float* const* h_w_ptrs, float* const* h_mask_ptrs, const int64_t* h_seg_sizes,
                          int nseg, int64_t k, float gamma, float* d_out3, void* d_ws, size_t ws_bytes,
                          void* stream);
/* Diagnostics (synchronises the stream): 1 if the last select on this workspace took the sample-pivot fast path. */
int mc_debug_select_used_fast(const void* d_ws, void* stream);
/* Diagnostics (synchronises): globaltimer (ns) of block 0 at the phase boundaries of the last launch, 12 values. */
int mc_debug_select_tstamps(const void* d_ws, unsigned long long* h_out12, void* stream);

/* mask[i] = (|w[i]| > *d_thr) ? 1.f : 0.f for every segment; if apply!=0 also w[i] *= mask[i]
 * (set_mask).  h_mask_ptrs may be NULL when apply!=0 (apply only).                                  */
int mc_mask_apply_gt(float* const* h_w_ptrs, float* const* h_mask_ptrs, const int64_t* h_seg_sizes,
                     int nseg, const float* d_thr, int apply, void* stream);

/* w[i] *= mask[i] for every segment — MaskedConv2d.set_mask, layers.py:46.                          */
int mc_apply_masks(float* const* h_w_ptrs, const float* const* h_mask_ptrs,
                   const int64_t* h_seg_sizes, int nseg, void* stream);

/* Counts exact zeros per segment into d_counts[nseg] (int64) — prune_rate, utils.py:59-93.          */
int mc_count_zeros(const float* const* h_w_ptrs, const int64_t* h_seg_sizes, int nseg,
                   int64_t* d_counts, void* stream);

/* d_out[s] = sum_i w[i] * |mask[i] - 1| per segment, fp64 accumulation — are_masks_consistent,
 * utils.py:122-133 (the reference only tests the total against 0).                                  */
int mc_masked_residual(const float* const* h_w_ptrs, const float* const* h_mask_ptrs,
                       const int64_t* h_seg_sizes, int nseg, double* d_out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Filter pruner — replaces methods.py:28-78 (quick_filter_prune).
 * Layer l has weight [O_l, C_l, kh_l, kw_l] fp32, contiguous.
 * -------------------------------------------------------------------------------------------- */

/* Step 1 (methods.py:43-44 / 64-65): d_values[off_l + o] = (sum_{c,h,w} w^2) / (C*kh*kw) in float32, with
 * NumPy's exact summation order (sequential over c, then h, then w for kh*kw>1; pairwise over c for 1x1).
 * Step 2 (methods.py:46-51): v /= sqrt(pairwise_sum(v^2)); v /= max(v), per layer, float32 (up to 51,200 filters
 * per layer).  off_l = sum of O of the previous layers.                                             */
int mc_filter_values(const float* const* h_w_ptrs, const int* h_O, const int* h_C, const int* h_kh,
                     const int* h_kw, int nlayers, float* d_values, void* stream);

/* The whole of quick_filter_prune in one call.  Step 1 and 2 as above; step 3 (methods.py:55): *d_thr = float64
 * np.percentile(values, perc), method 'linear': _lerp(sorted[k], sorted[min(k+1,n-1)], gamma); step 4 (methods.py:75):
 * d_keep[off_l + o] = !((double)v < *d_thr) and full-shape masks (fp32 1/0 per weight).  d_values [sum O] float32,
 * d_keep [sum O] (may be NULL), h_mask_ptrs may be NULL.  ONE cooperative launch: persistent blocks take filter groups
 * from an atomic queue (3x3 layers through a cp.async shared-memory ring); the block that completes the last group
 * normalises every layer, selects the percentile (counting rounds on the top byte of the bit patterns, then radix
 * passes) and publishes threshold + keep flags while the other blocks pre-fill their masks; every block then fixes up
 * its masks.  (More than 26,368 filters: three launches, up to 51,200.)  d_ws: mc_workspace_bytes_filter_prune()
 * bytes, any content.                                                                                                 */
int mc_filter_prune(const float* const* h_w_ptrs, const int* h_O, const int* h_C, const int* h_kh, const int* h_kw,
                    int nlayers, int64_t k, double gamma, float* d_values, double* d_thr,
                    float* const* h_mask_ptrs, uint8_t* d_keep, void* d_ws, size_t ws_bytes, void* stream);
size_t mc_workspace_bytes_filter_prune(void);

/* Greedy filter pruning — replaces methods.py:81-126 (prune_one_filter) and :129-142 (filter_prune), arXiv:1611.06440.
 * Per layer v = raw / sqrt(pairwise_sum(raw^2)) (raw as in step 1 above, float32, NumPy's order); each layer offers
 * arg_nonzero_min(v) (utils.py:96-120, with its tie rules; (inf, inf) when nothing or only index 0 is nonzero); the
 * pick is np.argmin over those float64 values (the first NaN, else the first minimum); the picked filter's raw value
 * becomes 0 and its nonzero weights are added to the zero count.  After each pick the walk stops when
 * !(100. * zeros / total_params < perc) (float64; zeros starts at zeros0, so at least one filter is picked), or
 * after max_picks picks (1 <= max_picks <= sum O).  sum O <= 20,480.
 *   d_picks  [max_picks][2] int32, 8-byte aligned: (filter index over all layers, its count of nonzero weights)
 *   d_result [3] int64: picks made, final zero count, status: 0 target reached, 1 max_picks made first, 2 a NaN pick
 *            (it changes no value: the reference repeats it forever), 3 every layer reports (inf, inf) (no pick is
 *            made), 4 a raw value is not finite (no pick is made)
 * Full-shape masks (1 = kept, 0 = picked) are written when h_mask_ptrs != NULL.
 * d_ws: mc_workspace_bytes_filter_prune_greedy(sum O) bytes, any content.                                         */
int mc_filter_prune_greedy(const float* const* h_w_ptrs, const int* h_O, const int* h_C, const int* h_kh,
                           const int* h_kw, int nlayers, int64_t zeros0, int64_t total_params, double perc,
                           int max_picks, int32_t* d_picks, int64_t* d_result, float* const* h_mask_ptrs,
                           void* d_ws, size_t ws_bytes, void* stream);
size_t mc_workspace_bytes_filter_prune_greedy(int n_filters);

/* ------------------------------------------------------------------------------------------
 * Region decode + NMS — replaces src/nets2_utils.py:141-234 (get_region_boxes) and :236-259 (nms),
 * :63-98 (bbox_iou, centre format).
 * -------------------------------------------------------------------------------------------- */

/* d_head: [B, A*(5+nc), H, W] fp32 (raw Darknet.forward output).  For every image, candidates are
 * emitted in the reference's list order (cy, cx, anchor) into
 *   d_boxes  [B, H*W*A, 8] : x/W, y/H, w/W, h/H, conf, cls_max_conf, (float)cls_max_id, (float)src_pos
 *   d_cls    [B, H*W*A, nc]: softmax class probabilities of each candidate (may be NULL)
 *   d_counts [B]           : number of candidates per image
 * Candidate iff conf > thresh (only_objectness) or conf*cls_max_conf > thresh.                       */
int mc_decode_region(const float* d_head, int B, int H, int W, int A, int nc, const float* h_anchors,
                     float conf_thresh, int only_objectness,
                     float* d_boxes, float* d_cls, int* d_counts, void* stream);

/* Greedy class-agnostic NMS per image on centre-format boxes (stride 8 floats as above, `cap` boxes per
 * image, counts[b] valid).  Sort key 1-conf ascending, ties by ascending candidate index (the
 * reference's torch.sort is unstable; SURVEY.md §8c shim 3 pins the stable order).
 * d_keep[b, 0..d_keep_counts[b]) = candidate indices of the kept boxes in sorted order.
 * Boxes suppressed get conf (element 4) set to 0 in d_boxes, as the reference mutates its input.     */
int mc_nms_batched(float* d_boxes, const int* d_counts, int B, int cap, float nms_thresh,
                   int* d_keep, int* d_keep_counts, void* stream);

/* mc_nms_batched plus what the batched evaluator needs from the same pass (src/predict.py:148-173):
 *   d_counts == NULL: `d_boxes` is a DENSE slot table [B, cap, 8] (one row per (cy*W+cx)*A + a, element 7 = slot index
 *                     for a candidate, -1 for a non-candidate — the output of the fused decode epilogue MC_EPI_DECODE);
 *                     `d_keep` then holds slot indices.  Slot order == the reference's list order, so ties break alike.
 *   d_row_counts [B] (may be NULL): rows image b contributes to the detection table — one per kept box, plus, when
 *                     d_cls [B, cap, nc] is given (validation mode, nets2_utils.py:223-228), one per other class c
 *                     with conf*cls[c] > conf_thresh.
 *   d_cand_counts [B] (may be NULL): number of candidates per image.                                    */
int mc_nms_detect(float* d_boxes, const int* d_counts, int B, int cap, float nms_thresh, int* d_keep,
                  int* d_keep_counts, const float* d_cls, int nc, float conf_thresh, int* d_row_counts,
                  int* d_cand_counts, void* stream);

/* Detection rows [img, x, y, w, h, box_conf, cls_conf, cls_id] of B images written straight from the NMS output —
 * replaces the per-class row emission of src/predict.py:157-173.  Image b's rows start at d_row_offsets[b] (int64,
 * exclusive prefix sums of mc_nms_detect's d_row_counts) and are in NMS order; with d_cls (validation mode) the arg-max
 * class row comes first, then the other passing classes in ascending order.  img = first_image + b.               */
int mc_compact_detections(const float* d_boxes, const int* d_keep, const int* d_keep_counts, const float* d_cls,
                          int B, int cap, int nc, float conf_thresh, int first_image,
                          const int64_t* d_row_offsets, float* d_out, void* stream);

/* Element-wise IoU of two box sets laid out [4, n] (row i = coordinate i of every box) — replaces bbox_ious,
 * src/nets2_utils.py:100-131 (x1y1x2y2 != 0: corner format; 0: centre format).  d_out[n].  fp32, reference op order. */
int mc_bbox_ious(const float* d_boxes1, const float* d_boxes2, int64_t n, int x1y1x2y2, float* d_out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Darknet-19 forward — replaces the F.conv2d + BatchNorm2d + LeakyReLU + MaxPool2d + Reorg + cat
 * call sites of src/nets.py:720-774 / src/pruning/weightPruning/layers.py:53-64.
 *
 * Activation layout ("PNHWC"): bf16, row-major [rows, C] with rows = B*(H+1)*(W+1); pixel (b,y,x) is row
 * b*(H+1)*(W+1) + y*(W+1) + x; column x==W of every line and line y==H of every image are zero, so a
 * 3x3 tap is a constant row offset dy*(W+1)+dx and the implicit GEMM needs no bounds logic.
 * -------------------------------------------------------------------------------------------- */

enum { MC_EPI_PNHWC = 0,      /* bf16 PNHWC at the same resolution, channel offset ch_off, row pitch ldc   */
       MC_EPI_REORG2 = 1,     /* bf16 PNHWC at (H/2,W/2): channel ((y&1)*2+(x&1))*N + n + ch_off (Reorg)   */
       MC_EPI_NCHW_F32 = 2,   /* fp32 NCHW [B,N,H,W] (network head)                                        */
       /* (3 is unused: a 2x2/2 max-pool is fused by the thin-layer kernels below, whose GEMM row is a pool window — */
       /* mc_conv_im2col_fwd / mc_conv_window_fwd / mc_conv_thin_fwd with pool=1 —, not by this row-tiled kernel:  */
       /* DESIGN.md §9)                                                                                            */
       MC_EPI_DECODE = 4 };   /* network head + region decode fused: see mc_decode_params                  */

/* MC_EPI_DECODE — get_region_boxes (src/nets2_utils.py:158-205) applied to the head convolution's accumulators in its
 * epilogue: the thread that owns pixel (b, cy, cx) holds all A*(5+nc) logits of the cell, so sigmoid / exp / softmax /
 * arg-max / threshold run there and the raw head never makes a round trip through HBM.  Output is the DENSE slot table
 *   d_boxes [B, H*W*A, 8]: slot (cy*W+cx)*A + a = x/W, y/H, w/W, h/H, conf, cls_max_conf, (float)cls_max_id,
 *                          (float)slot for a candidate (conf > thresh, or conf*cls_max_conf > thresh) else -1
 *   d_cls   [B, H*W*A, nc] softmax probabilities of the candidates (may be NULL)
 *   d_head  fp32 NCHW [B, A*(5+nc), H, W]: the raw head as MC_EPI_NCHW_F32 would store it (may be NULL)
 * which mc_nms_detect consumes directly (d_counts = NULL).  Slot order is the reference's list order (cy, cx, anchor).
 * Needs N == A*(5+nc) <= 256 (one N tile).  Arithmetic identical to mc_decode_region on the same fp32 logits.      */
typedef struct mc_decode_params {
  float* d_boxes;
  float* d_cls;
  float* d_head;
  int A, nc;
  float conf_thresh;
  int only_objectness;
  float anchors[32];     /* (w, h) pairs, A of them                                                      */
} mc_decode_params;

typedef struct mc_conv_desc {
  const void* d_in;      /* bf16 PNHWC [B*(H+1)*(W+1), Cin_ld]                                           */
  const void* d_wpack;   /* bf16 [Npad, ntaps*Kc] K-major, Kc = round_up(Cin, block_k); from mc_pack_conv_weights */
  const float* d_scale;  /* [Npad] per-output-channel multiplier (folded BN gamma/sqrt(var+eps), or 1)     */
  const float* d_shift;  /* [Npad] per-output-channel addend (folded BN beta - mean*scale, or conv bias)   */
  void* d_out;
  int B, H, W;           /* input (= conv output) resolution                                              */
  int Cin, Cin_ld;       /* channels read, row pitch (elements) of d_in; both multiples of 8              */
  int N, Npad;           /* output channels, padded to a multiple of 16                                   */
  int ksize;             /* 1 or 3 (stride 1, 'same' padding)                                             */
  int leaky;             /* 1: y = max(y, 0.1y)                                                           */
  int epi_mode;          /* MC_EPI_*                                                                      */
  int ldc, ch_off;       /* output row pitch (elements) and channel offset (bf16 modes)                   */
  int block_n;           /* 0 = auto; else 16..256 multiple of 16                                         */
  int stages;            /* 0 = auto                                                                      */
  int block_k;           /* k-block: 0/64 = 64 bf16 (d_wpack Kc = round_up(Cin,64)); 32 = 32 bf16 with 64-byte   */
                         /* swizzle (Kc = round_up(Cin,32)): less zero padding for Cin like 32, 69, 91             */
  int in_cols;           /* 0 = Cin.  Else Cin <= in_cols <= Cin_ld: columns of a d_in row TMA may READ.  Columns    */
                         /* >= Cin meet zero weights and must hold finite values (the engine's pad channels are 0).  */
                         /* A box that lies wholly inside the tensor takes TMA's fast path: a partly out-of-bounds   */
                         /* inner box costs 28 us instead of 20 us on a 17-channel 1x1 layer at 104x104, batch 64.   */
  const mc_decode_params* decode; /* MC_EPI_DECODE only (host pointer, copied at launch); d_out is unused then      */
  void* d_ws;            /* optional scratch (256-byte aligned, mc_workspace_bytes_conv_fwd bytes, its first 2 KB ZERO   */
  size_t ws_bytes;       /* before the first use; launches leave them zero): lets the CTA-pair kernel split the partial  */
                         /* last wave of tiles along K (stream-K).  NULL: whole tiles only.                             */
  float* d_stat_sum;     /* optional, MC_EPI_PNHWC with N > 32 only (training forward): per-output-channel sum and sum of */
  float* d_stat_sumsq;   /* squares of the STORED bf16 values over all rows are ADDED here (atomics; the caller zeroes    */
                         /* them) — nn.BatchNorm2d's batch statistics (src/nets.py:802) without a pass over the output.   */
} mc_conv_desc;

int mc_conv_fwd(const mc_conv_desc* desc, void* stream);
/* Scratch bytes mc_conv_fwd can use for this layer shape (0 = none).  The same buffer may serve every layer of a network
 * (launches on one stream are ordered); contents are meaningless between calls.                                  */
size_t mc_workspace_bytes_conv_fwd(const mc_conv_desc* desc);

/* A chain of 2..4 wide 3x3 layers in which member i+1 reads member i's output, as ONE launch of the CTA-pair kernel.
 * Each member computes exactly what its own mc_conv_fwd call would (same plan, same arithmetic, bit-identical output);
 * only the schedule changes: the (member, m-pair, n-tile) units are tickets in layer-major, m-major order, which the
 * clusters claim with one atomic each, so the idle clusters of one member's partial last wave start the next member's
 * first units, and the launches, drains and pipeline fills between the members disappear.  A unit of member i+1 starts
 * once every unit of member i over its rows (3x3 halo included) is stored; a counter per (member, m-pair) in the
 * workspace tracks that.  Returns an error WITHOUT launching unless: 2 <= n <= 4; every member takes the CTA-pair
 * kernel under mc_conv_fwd's own rules with the TMA-store PNHWC epilogue and the same tile width, ring and activation;
 * all members share B, H, W; no member asks for statistics; member i+1 reads member i's output allocation
 * (d_in == previous d_out, Cin_ld == previous ldc) and no member reads or rewrites another member's output otherwise.
 * Workspace: descs[0].d_ws / ws_bytes, 16-byte aligned, mc_workspace_bytes_conv_chain bytes, ZERO before the first
 * launch; every launch leaves it zero again, except the status word (uint32 index 2), which becomes nonzero if a unit
 * waited for its inputs longer than a second (never expected: a dependency bug).  d_ws of the other members is ignored. */
int mc_conv_chain_fwd(const mc_conv_desc* descs, int n, void* stream);
/* Workspace bytes of that chain, or 0 when mc_conv_chain_fwd would reject these descriptors (the same checks, no
 * launch: callers use it to find the runs of layers the chain takes at a given batch size).                        */
size_t mc_workspace_bytes_conv_chain(const mc_conv_desc* descs, int n);

/* Which launch configuration the LAST mc_conv_fwd call of this host thread chose (tests / bench reporting):
 * info[0] = 1 CTA-pair kernel (tcgen05 cta_group::2, 256-row tiles, half of each weight tile per CTA), 0 single CTA
 * info[1] = tile width block_n      info[2] = resident CTAs per SM requested (1..3)
 * info[3] = CTA pair: units in the stream-K tail; 0 otherwise
 * info[4] = 1 shared activation box (3x3)
 * info[5] = smem ring stages         info[6] = grid size                   info[7] = k-block (32 or 64)           */
int mc_conv_last_plan(int info[8]);

/* What mc_conv_fwd would launch for this descriptor on the current device, without launching (tests / reporting).
 * The descriptor is checked as mc_conv_fwd checks it (same errors); buffers are not touched.
 * info[0]  = 1 CTA-pair kernel, 0 single CTA       info[1]  = CTAs per SM (1..3; 1 for the pair)
 * info[2]  = block_n                               info[3]  = block_k (32 or 64)
 * info[4]  = B-tile (or A | B) ring stages         info[5]  = activation-box ring stages (0: no shared box)
 * info[6]  = 1 shared activation box               info[7]  = CTAs launched
 * info[8]  = 128-row m-tiles                       info[9]  = n-tiles
 * info[10] = CTA pair: units in the stream-K tail (0: whole units only)
 * info[11] = PNHWC store path: 2 TMA-store slabs, 1 staged through shared memory, 0 direct (and every other mode)
 * info[12] = TMA-store slabs per epilogue warp     info[13] = 1: the epilogue loads 64 accumulator columns at a time
 * info[14] = 1: 16-byte stores allowed (8-aligned ldc and ch_off; REORG2 also N % 8 == 0), 0: scalar stores
 * info[15] = UMMA K steps (16 channels) issued for the last channel block of a tap                                  */
int mc_conv_fwd_plan(const mc_conv_desc* desc, int info[16]);

/* Small-channel direct convolution on CUDA cores, for layers too thin for a 128xNx64 tensor-core tile: the 3-channel
 * first layer (in_is_nchw_f32=1: d_in is the fp32 NCHW image [B,Cin,H,W]) and the first blocks of a filter-pruned
 * network (d_in PNHWC bf16, pitch Cin_ld).  d_w: fp32 [N,Cin,k,k] (already masked / gathered).  Fused scale/shift,
 * leaky and optional 2x2/2 max-pool; writes channels [0,N) of the interior rows of a PNHWC bf16 buffer at (H,W) or
 * (H/2,W/2) — the destination's pad line/column must already be zero.  Limits: mc_conv_direct_supported().        */
int mc_conv_direct_supported(int Cin, int N, int ksize);
int mc_conv_direct_fwd(const void* d_in, int in_is_nchw_f32, const float* d_w, const float* d_scale,
                       const float* d_shift, void* d_out, int B, int H, int W, int Cin, int Cin_ld, int N, int ldc,
                       int ksize, int leaky, int pool, void* stream);

/* Degenerate layers of a filter-pruned network on CUDA cores (csrc/conv_thin.cu): MaskedConv2d + folded BatchNorm +
 * leaky [+ 2x2/2 max-pool] (src/nets.py:779-821) for a 3x3 layer with <= 8 input channels or a 1x1 layer with <= 32
 * input channels and <= 8 outputs, a few hundred multiply-adds per pixel at most.  One thread per output pixel (or pool
 * window); the weights are passed as KERNEL PARAMETERS, so h_w / h_scale / h_shift (and the *2 arrays) are HOST pointers:
 *   h_w   fp32 [(tap*ct + c)*nt + n] = w[n,c,tap/k,tap%k] (bf16-rounded by the caller, zero padded), h_scale/h_shift [nt]
 *   N2 > 0: the 1x1 layer behind a 3x3 layer is applied in the same thread to the bf16-rounded activations:
 *   h_w2  fp32 [n*n2t + o] = w2[o,n], h_scale2/h_shift2 [n2t]; the output then has N2 channels.
 * mc_conv_thin_geometry returns 1 and the padded sizes (ct channels read per input pixel, nt, n2t) when the shape is
 * taken, 0 otherwise.  d_in: bf16 PNHWC with pitch Cin_ld >= ct; d_out: interior rows of a bf16 PNHWC buffer at (H,W) or
 * (H/2,W/2) whose pad line/column are already zero; channels up to the next multiple of 8 are written (zeros).      */
int mc_conv_thin_geometry(int ksize, int Cin, int N, int pool, int N2, int* ct, int* nt, int* n2t);
int mc_conv_thin_fwd(const void* d_in, const float* h_w, const float* h_scale, const float* h_shift, const float* h_w2,
                     const float* h_scale2, const float* h_shift2, void* d_out, int B, int H, int W, int Cin, int Cin_ld,
                     int N, int ldc, int ksize, int leaky, int pool, int N2, int leaky2, void* stream);

/* Thin 3x3 layers on the tensor cores with the im2col tile built in shared memory (csrc/conv_im2col_tc.cu): the
 * 3-channel first layer (in_is_nchw_f32=1, Cin<=4) or a PNHWC bf16 input with pitch == CL (8 for Cin<=8, 16 for
 * Cin<=16).  pool=1 fuses the 2x2/2 max-pool ("pool-window GEMM").  d_wexp is the expanded bf16 weight matrix
 * [nb_pad, kpad] described by mc_conv_im2col_geometry():
 *   pool=0: row n,            column (r*3+s)*CL + c         = w[n,c,r,s]
 *   pool=1: row pos*npos + n, column (py*4+px)*CL + c       = w[n,c,py-dy,px-dx]  (pos = dy*2+dx; 0 outside the 3x3)
 * Writes channels [0,N) of the interior rows of a PNHWC bf16 buffer whose pad line/column are already zero.       */
int mc_conv_im2col_supported(int Cin, int in_is_nchw_f32, int N, int pool);
int mc_conv_im2col_geometry(int Cin, int in_is_nchw_f32, int N, int pool, int* cl, int* npos, int* nb, int* kpad);
int mc_conv_im2col_fwd(const void* d_in, int in_is_nchw_f32, const void* d_wexp, const float* d_scale,
                       const float* d_shift, void* d_out, int B, int H, int W, int Cin, int Cin_ld, int N, int ldc,
                       int leaky, int pool, void* stream);

/* Thin 3x3 layers on the tensor cores WITHOUT an im2col build (csrc/conv_window.cu): un-swizzled UMMA descriptors read
 * the overlapping receptive-field windows of a 16x8 output tile straight out of a shared-memory pixel patch.
 *   in_kind 0: d_in bf16 PNHWC with pitch 8 (Cin <= 8), N <= 128, optional 2x2/2 max-pool taken across lanes in the
 *              epilogue.  d_w: bf16 [nb][80], row n, column tap*8 + c = w[n,c,tap/3,tap%3] (columns 72..79 zero).
 *   in_kind 1 / 2: d_in fp32 / uint8 NCHW image [B,3,H,W] (uint8 is scaled by 1/255 like ToTensor), pool = 1 required:
 *              pool-window GEMM, d_w in mc_conv_im2col_fwd's expanded layout with CL = 4 and 64 columns:
 *              row pos*npos + n, column (py*4+px)*4 + c = w[n,c,py-dy,px-dx] (pos = dy*2+dx).
 * mc_conv_window_geometry reports npos, nb (rows of d_w, multiple of 16) and the column count of d_w.
 * Writes channels [0,N) of the interior rows of a PNHWC bf16 buffer whose pad line/column are already zero.       */
int mc_conv_window_supported(int Cin, int in_kind, int N, int pool);
int mc_conv_window_geometry(int Cin, int in_kind, int N, int pool, int* npos, int* nb, int* kcols);
int mc_conv_window_fwd(const void* d_in, int in_kind, const void* d_w, const float* d_scale, const float* d_shift,
                       void* d_out, int B, int H, int W, int Cin, int N, int ldc, int leaky, int pool, void* stream);

/* Debug aid: later single-CTA mc_conv_fwd launches record globaltimer stamps (32 x uint64 per CTA: entry, set-up done,
 * first operands landed, per-tile MMA issue / accumulator ready / epilogue done, exit) into d_buf (32*8*grid bytes);
 * NULL switches it off.  tools/trace_conv.py prints the timelines.                                              */
int mc_debug_conv_trace(void* d_buf);

/* Debug aid: code of the first mbarrier wait that timed out inside mc_conv_im2col_fwd kernels (0 = none). */
int mc_debug_im2col_timeout(void);

/* fp32 [O,C,kh,kw] (optionally * mask, optionally gathered by h_oidx/h_cidx surviving-index lists)
 * -> bf16 [Npad, kh*kw*Kc] with column (tap*Kc + c).  d_oidx/d_cidx are device int32 arrays or NULL. */
int mc_pack_conv_weights(const float* d_w, const float* d_mask, int O, int C, int ksize,
                         const int* d_oidx, int n_o, const int* d_cidx, int n_c,
                         void* d_wpack, int Npad, int Kc, void* stream);

/* 2x2/2 max-pool on PNHWC bf16: in [B,(H+1),(W+1),C] -> out [B,(H/2+1),(W/2+1),C].                   */
int mc_maxpool2x2(const void* d_in, void* d_out, int B, int H, int W, int C, int ld_in, int ld_out,
                  void* stream);

/* PNHWC bf16 -> NCHW fp32 [B,C,H,W] (debug / per-block parity checks). */
int mc_unpack_pnhwc(const void* d_in, float* d_out, int B, int H, int W, int C, int ld_in, int ch_off,
                    void* stream);

/* Stand-alone Reorg — replaces Reorg.forward, src/nets.py:648-667, on the reference's layout: fp32 NCHW [B,C,H,W] ->
 * fp32 NCHW [B, s*s*C, H/s, W/s], out[b,(i*s+j)*C+c,y,x] = in[b,c,s*y+i,s*x+j].  (Inside Darknet.forward the shuffle is
 * the MC_EPI_REORG2 store addressing of the producing conv.)                                           */
int mc_reorg_nchw(const float* d_in, float* d_out, int B, int C, int H, int W, int stride, void* stream);

/* NCHW fp32 [B,C,H,W] -> PNHWC bf16 (channels >= C up to ld zeroed; pad rows/cols zeroed). */
int mc_pack_pnhwc(const float* d_in, void* d_out, int B, int H, int W, int C, int ld_out, void* stream);


/* ------------------------------------------------------------------------------------------
 * Masked retrain step — replaces, for model.train(), the autograd graph of src/train.py:221-235 over the Darknet of
 * src/nets.py:779-822: F.conv2d(x, weight*mask) forward/dgrad/wgrad (layers.py:53-64), nn.BatchNorm2d in training mode
 * (batch statistics, eps 1e-5, running stats momentum 0.1; nets.py:802), nn.LeakyReLU(0.1) (:809), nn.MaxPool2d(2,2)
 * (:821) and their backward.  Convolutions (forward and data gradient) reuse mc_conv_fwd; the weight gradient is
 * mc_conv_wgrad.  All activations / gradients are PNHWC bf16, per-channel statistics and weight gradients fp32.
 * -------------------------------------------------------------------------------------------- */

/* The BatchNorm / pool passes below move 8 channels per 16-byte access, for any C up to 2048 (a ragged last group
 * of C % 8 channels is handled; columns past C are never written).  They return an argument error unless
 * C <= 2048, every pitch (ld*) and ch_off is a multiple of 8, every tensor pointer is 16-byte aligned and
 * B*(H+1)*(W+1) (rows for mc_col_stats) is below 2^31.  Pitches of round_up(C, 8) and torch allocations meet this.    */

/* d_sum[c] = sum over rows of z[row, ch_off+c]; d_sumsq[c] likewise of z^2 (may be NULL).  Pad rows are zero.       */
int mc_col_stats(const void* d_z, int64_t rows, int C, int ld, int ch_off, float* d_sum, float* d_sumsq, void* stream);

/* Batch statistics -> per-channel (scale, shift) of y = z*scale + shift, mean, invstd; running stats updated in place
 * (running = (1-momentum)*running + momentum*batch, unbiased variance) when the pointers are not NULL.              */
int mc_bn_finalize(const float* d_sum, const float* d_sumsq, int C, double count, const float* d_gamma,
                   const float* d_beta, float eps, float momentum, float* d_running_mean, float* d_running_var,
                   float* d_scale, float* d_shift, float* d_mean, float* d_invstd, void* stream);

/* out = act(z*scale + shift) at interior pixels, 0 at pads.  reorg=0: out[row, ch_off + c]; reorg=1: the Reorg(2)
 * shuffle into a (H/2, W/2) buffer, channel ((y&1)*2+(x&1))*C + c + ch_off (interior rows only).                   */
int mc_bn_apply(const void* d_z, int ld_z, int B, int H, int W, int C, const float* d_scale, const float* d_shift,
                int leaky, void* d_out, int ld_out, int ch_off, int reorg, void* stream);

/* BatchNorm(training) + leaky backward: g = da * leaky'(.), dbeta = sum g, dgamma = sum g*xhat,
 * dz = gamma*invstd*(g - dbeta/N - xhat*dgamma/N) (0 at pads).  da is read through (ld_da, ch_off, reorg) so a concat
 * slice / reorg'd gradient needs no un-shuffling copy.                                                              */
int mc_bn_backward(const void* d_z, int ld_z, const void* d_da, int ld_da, int ch_off, int reorg, int B, int H, int W,
                   int C, const float* d_mean, const float* d_invstd, const float* d_gamma, const float* d_beta,
                   int leaky, float* d_dbeta, float* d_dgamma, void* d_dz, int ld_dz, void* stream);

/* d_full[b,y,x,c] (+)= d_pooled[b,y/2,x/2,c] where a_full[b,y,x,c] is the first maximum of its 2x2 window.          */
int mc_maxpool2x2_backward(const void* d_a_full, int ld_a, const void* d_dpooled, int ld_dp, int B, int H, int W, int C,
                           void* d_dfull, int ld_df, int accumulate, void* stream);

/* BatchNorm(training) + leaky + MaxPool2d(2,2) in one pass each way, for layers whose un-pooled activation only feeds
 * the pool (nn.BatchNorm2d / nn.LeakyReLU / nn.MaxPool2d of src/nets.py:802-821 and their autograd backward): the
 * forward writes pooled = maxpool(bf16(act(z*scale + shift))) straight from z; the backward recomputes the window
 * from z, routes d_pooled to the first maximum and produces dbeta / dgamma / dz like mc_bn_backward — the un-pooled
 * activation and its gradient never exist.  Needs C = 8 * 2^k <= 2048 (mc_bn_pool_supported), even H and W, and the
 * pitch / alignment / row-count conditions above.                                                                   */
int mc_bn_pool_supported(int C);
int mc_bn_apply_pool(const void* d_z, int ld_z, int B, int H, int W, int C, const float* d_scale, const float* d_shift,
                     int leaky, void* d_pooled, int ld_p, void* stream);
int mc_bn_pool_backward(const void* d_z, int ld_z, const void* d_dpooled, int ld_dp, int B, int H, int W, int C,
                        const float* d_scale, const float* d_shift, const float* d_mean, const float* d_invstd,
                        const float* d_gamma, const float* d_beta, int leaky, float* d_dbeta, float* d_dgamma, void* d_dz,
                        int ld_dz, void* stream);

/* YOLOv2 region loss — replaces RegionLoss.forward + build_targets (src/nets.py:282-440, 468-610) and the backward of
 * the loss expression: d_output fp32 [nB, nA*(5+nC), nH, nW] (the head), d_target fp32 [nB, 50*5] rows of
 * (cls, x, y, w, h) normalised and zero padded (dataloader.py:82-96), h_anchors 2*nA HOST doubles (the cfg's floats).
 * Writes *d_loss (float32 scalar), d_grad = d loss / d output (same shape as the head), d_counts = {nGT, nCorrect}.
 * The reference's quirks are kept (w/h exp()-ed twice for the IoU boxes, tw = gw/anchor_w, list ends at the first
 * x == 0, later box overwrites an earlier one on the same (anchor, cell), no positive anchor IoU -> last anchor).   */
size_t mc_workspace_bytes_region_loss(int nB);
int mc_region_loss(const float* d_output, const float* d_target, int nB, int nA, int nC, int nH, int nW,
                   const double* h_anchors, float coord_scale, float noobject_scale, float object_scale,
                   float class_scale, float thresh, float* d_grad, float* d_loss, int* d_counts, void* d_ws,
                   size_t ws_bytes, void* stream);

/* PASCAL-VOC scorer pieces — replace the '%f' detection files of the eval loop (src/predict.py:157-173) and the
 * per-detection matching loop of voc_eval (src/predict.py:305-380).  mc_voc_table: rows (image, x, y, w, h, box_conf,
 * cls_conf, cls) -> image / class ids, score and corner boxes after the reference's float32 arithmetic and the 6-decimal
 * text round trip (float64); d_sizes [n_images, 2] (width, height) or NULL (def_w x def_h).  mc_voc_match: detections in
 * (class, descending score) order with key = class*K + image, ground-truth boxes sorted by the same key (float64
 * corners, difficult flags) -> tp / fp flags (float64 0/1) by the reference's rule: best-overlap box (first maximum),
 * > ovthresh, difficult boxes ignored, the first detection in order that reaches a box is its true positive.        */
int mc_voc_table(const float* d_dets, int64_t n, const float* d_sizes, float def_w, float def_h, int64_t* d_img,
                 int64_t* d_cls, double* d_conf, double* d_corners, void* stream);
size_t mc_workspace_bytes_voc_match(int64_t n, int64_t m);
int mc_voc_match(const int64_t* d_key, const double* d_corners, int64_t n, const int64_t* d_gkey, const double* d_gbox,
                 const uint8_t* d_gdiff, int64_t m, double ovthresh, double* d_tp, double* d_fp, void* d_ws,
                 size_t ws_bytes, void* stream);

/* dgrad weights for mc_conv_fwd: bf16 [Cpad, taps*Ko], row c, column tap'*Ko + o = (w*mask)[o, c, taps-1-tap'].      */
int mc_pack_conv_weights_dgrad(const float* d_w, const float* d_mask, int O, int C, int ksize, void* d_wpack, int Cpad,
                               int Ko, void* stream);

/* dW[O,C,k,k] (fp32, PyTorch layout) = mask * sum_p dZ[p, o] * A[p + off(tap), c]  on tcgen05 (both operands
 * MN-major from TMA); split over the pixel rows, partials in the workspace.  accumulate!=0 adds the masked gradient
 * to d_dw: dW = dW_old + mask * grad, so masked entries keep their old value (they are not zeroed).                */
int mc_conv_wgrad(const void* d_a, int lda, int C, const void* d_dz, int ld_dz, int O, int B, int H, int W, int ksize,
                  const float* d_mask, float* d_dw, int accumulate, void* d_ws, size_t ws_bytes, void* stream);
size_t mc_workspace_bytes_conv_wgrad(int B, int H, int W, int C, int O, int ksize);
/* What mc_conv_wgrad does for this shape on the current device (no launch; tests / reporting):
 * info[0] = nsplit (CTAs along the pixel rows)   info[1] = m_tiles (128 filters)   info[2] = n_tiles
 * info[3] = block_n (input channels per tile)    info[4] = share3 (3x3: one CTA per filter row)
 * info[5] = merge3 (the three dx taps as one N = 192 MMA)
 * info[6] = split reduction: 1 rows<9>, 2 rows<1>, 3 small<1>, 4 small<4>, 5 small<8>
 *           (wgrad_reduce_rows_kernel<TAPS> / wgrad_reduce_small_kernel<split groups>)
 * info[7] = num_kb (64-row k-blocks of the whole reduction)                                                     */
int mc_conv_wgrad_plan(int B, int H, int W, int C, int O, int ksize, int info[8]);

/* Weight gradient of the first layer: x is the fp32 NCHW image [B,C,H,W], 3x3.  With a workspace of
 * mc_workspace_bytes_conv_wgrad_first() bytes (256-byte aligned; C*9 <= 32): the image is expanded to bf16 im2col rows
 * [B*(H+1)*(W+1), 32] and dW = the 1x1 tcgen05 weight gradient over them (mc_conv_wgrad).  Without one (d_ws NULL):
 * CUDA-core kernel, C <= 4, O <= 32 and a multiple of 4.                                                            */
size_t mc_workspace_bytes_conv_wgrad_first(int B, int H, int W, int C, int O);
int mc_conv_wgrad_first(const float* d_x, const void* d_dz, int ld_dz, int B, int H, int W, int C, int O,
                        const float* d_mask, float* d_dw, void* d_ws, size_t ws_bytes, void* stream);

/* Momentum SGD over `nseg` parameter tensors in one launch — replaces torch.optim.SGD.step() as the reference
 * configures it (src/train.py:144-147, stepped at :233-235; dampening 0, no nesterov): per element
 *   d = g + weight_decay*p;  buf = first_step ? d : momentum*buf + d;  p -= lr*buf      (fp32, torch's operation order).
 * Pruned weights have exactly zero gradients (mc_conv_wgrad multiplies by the mask) and therefore stay exactly zero. */
int mc_sgd_momentum_step(float* const* h_param_ptrs, const float* const* h_grad_ptrs, float* const* h_buf_ptrs,
                         const int64_t* h_sizes, int nseg, float lr, float momentum, float weight_decay,
                         int first_step, void* stream);

/* ------------------------------------------------------------------------------------------
 * Filter-shrunk retrain step (model.b200_shrink_train): the convolutions run over the ALIVE filters only (a filter is
 * dead when its mask is zero over [C,kh,kw]).  A dead filter is not inert in training: its activation is the constant
 * leaky(beta) inside the image (batch mean = var = 0), beta gets a gradient and the consumers' weights on it train.
 * Each consumer therefore reads two extra "ones" input columns (1 at interior pixels, 0 at pads) whose packed weights
 * are the high and low bf16 halves of S = sum over dead inputs c of bf16((W*mask)[o,c,tap]) * bf16(leaky(beta_c))
 * (fp32; the dense step's products), and whose weight gradient G1[o,tap] gives
 *   dW[o, c_dead, tap] = mask * leaky(beta_c) * G1[o,tap]
 *   dbeta_c (dead)     = leaky'(beta_c) * sum over consumers of sum_{o,tap} (W*mask)[o, c_in, tap] * G1[o,tap]
 * (c_in = every consumer input column carrying channel c: one per consumer, four through a Reorg).  DESIGN.md §1 a-12.
 *
 * One segment per convolution, in a device array built once per plan; per-step buffers are passed as base pointers and
 * the segment holds offsets into them.  Index lists are offsets into one int32 device array `idx`.
 * Every entry point is ONE launch over all segments (nseg <= MC_MAX_SEGMENTS).                                       */
typedef struct mc_shrink_seg {
  const float* w;          /* [O, C, taps] fp32 conv weight                                                       */
  const float* mask;       /* same shape, or NULL                                                                 */
  const float* gamma;      /* [O] BatchNorm weight / bias, NULL for a layer without BatchNorm                    */
  const float* beta;
  float* rmean;            /* [O] running statistics, NULL when not tracked                                       */
  float* rvar;
  float momentum;          /* running-statistics momentum                                                         */
  int leaky;               /* 1: leaky(0.1) activation, 0: linear                                                 */
  int O, C, taps;          /* full shape                                                                          */
  int n_o;                 /* compact (alive) filters                                                             */
  int n_col;               /* physical input columns (contraction width of the compact conv / wgrad)             */
  int ones_col;            /* physical column of the first of the two ones columns, -1 none                       */
  int npad, kc;            /* forward pack [npad, taps*kc] (kc = 0: this layer packs its weights itself)          */
  int cpad, ko;            /* data-gradient pack [cpad, taps*ko]                                                  */
  int n_dead;              /* dead input channels (length of dead_in)                                             */
  int pad_;
  int64_t oidx;            /* idx offset: [n_o] compact row -> filter                                             */
  int64_t orow;            /* idx offset: [O] filter -> compact row, -1 dead                                      */
  int64_t colmap;          /* idx offset: [n_col] physical column -> input channel, -1 zero column, -2 ones column */
  int64_t cphys;           /* idx offset: [C] input channel -> physical column, -1 dead input                    */
  int64_t clk;             /* idx offset: [C] dead input channel -> index into lk, -1 otherwise                  */
  int64_t dead_in;         /* idx offset: [n_dead] the dead input channels                                        */
  int64_t cons_ptr;        /* idx offset: [O+1] CSR row pointers of the consumer inputs of each dead filter       */
  int64_t cons;            /* idx offset: pairs (consumer segment, consumer input channel)                        */
  int64_t lk_off;          /* lk[lk_off + f] = act(beta[f]) for this layer's filters (BatchNorm layers)           */
  int64_t cbn_off;         /* compact gamma, beta, running mean, running var at cbn_off + {0,1,2,3} * cbn_ld      */
  int64_t cbn_ld;
  int64_t wp_off, wpd_off; /* bf16 element offsets of the forward / data-gradient packs                           */
  int64_t dwc_off;         /* float offset of the compact weight gradient [n_o, n_col, taps]                      */
  int64_t cdgb_off;        /* float offset of the compact dbeta [n_o], then dgamma [n_o] (mc_bn_backward output)  */
  int64_t dw_off;          /* float offset of the full dW [O, C, taps]                                            */
  int64_t dbn_off;         /* float offset of the full dbeta [O], then dgamma [O]                                 */
} mc_shrink_seg;

/* Per training forward, first: lk[lk_off+f] = bf16(act(beta[f])) (a dead channel's stored activation) and the compact gamma/beta/running statistics gathered at
 * cbn_off (which mc_bn_finalize / mc_bn_backward then use unchanged).                                                */
int mc_shrink_prepare(const mc_shrink_seg* d_segs, int nseg, const int* d_idx, float* d_cbn, float* d_lk, void* stream);
/* Forward weights: wp[wp_off + n*taps*kc + tap*kc + j] = bf16((W*mask)[oidx[n], colmap[j], tap]); the ones columns
 * hold hi = bf16(S), lo = bf16(S - hi) of S above; zero rows / columns elsewhere.  d_wpd (may be NULL):
 * the data-gradient weights at wpd_off, row = physical column (ones / zero columns get zero rows), column
 * tap'*ko + n = (W*mask)[oidx[n], colmap[row], taps-1-tap'].                                                         */
int mc_shrink_pack(const mc_shrink_seg* d_segs, int nseg, const int* d_idx, const float* d_lk, void* d_wp, void* d_wpd,
                   void* stream);
/* End of the training forward: compact running statistics (updated by mc_bn_finalize) back into the full buffers;
 * dead channels decay as nn.BatchNorm2d with batch mean = var = 0, in mc_bn_finalize's fp32 operation order.         */
int mc_shrink_stats(const mc_shrink_seg* d_segs, int nseg, const int* d_idx, const float* d_cbn, void* stream);
/* End of the backward: full dW (alive entries from the compact gradient, dead input columns by the G1 rule, the mask
 * applied, dead filters exactly 0) and full dgamma / dbeta (alive from the compact ones, dead: dgamma = 0 and dbeta by
 * the rule above) into d_grad.                                                                                      */
int mc_shrink_finish(const mc_shrink_seg* d_segs, int nseg, const int* d_idx, const float* d_lk, const float* d_dwc,
                     float* d_grad, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MCB200_H_ */
