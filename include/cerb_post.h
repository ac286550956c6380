/*
 * cerb_post.h -- C ABI of libcerb_post.so, the B200 (sm_100a) post-head path for
 * CerberusDet: Detect decode + per-task non_max_suppression.
 *
 * The reference (ai-forever/CerberusDet) is pure Python and has no FFI; its "operator
 * interface" for this path is three Python symbols.  Each entry point below names the
 * reference code it replaces (paths relative to the reference root).  INTEGRATION.md
 * shows the ctypes binding and the monkey-patch a maintainer adds on the reference side.
 *
 * Conventions
 *  - Plain pointers and sizes only.  Pointer *arrays* (lvl, y, pred, nc, H, W, strides,
 *    classes) are HOST arrays; what they point to (tensors, dets, counts, workspace) is
 *    DEVICE memory owned by the caller.  The library never allocates, frees or keeps a
 *    pointer after the call returns.
 *  - All work is enqueued on `stream` (a cudaStream_t passed as void*); no call
 *    synchronises the device.  Re-entrant; safe from several host threads on
 *    different streams: the only mutable state (last error, test knobs) is thread-local.
 *  - Return 0 on success, a negative CERB_E* code otherwise; cerb_last_error() gives the
 *    calling thread's message.  There is no CPU fallback.
 *  - dtype: CERB_F16 (IEEE half) or CERB_F32; tensors are contiguous.
 */
#ifndef CERB_POST_H
#define CERB_POST_H
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CERB_F16 0
#define CERB_F32 1

#define CERB_MAX_TASKS_ABI 8
#define CERB_MAX_LEVELS_ABI 4

#define CERB_EINVAL (-1)  /* bad argument (message says which) */
#define CERB_ECUDA (-2)   /* CUDA runtime error at launch */
#define CERB_ENOSPC (-3)  /* workspace too small */

/* Library version, major*10000 + minor*100 + patch. */
int cerb_version(void);

/* Message of the last error raised on the calling thread ("" if none). */
const char* cerb_last_error(void);

/*
 * Detect-head decode for T task heads in one launch.
 * Replaces the eval branch of Detect.forward after the conv towers
 * (cerberusdet/models/yolo.py:93-99) together with make_anchors
 * (cerberusdet/utils/tal.py:181-193), DFL.forward (models/yolo.py:57-59) and
 * dist2bbox(xywh=True) (utils/tal.py:196-205).
 *
 *   lvl[t*L + l]  raw head tensor of task t, level l: [B, 64 + nc[t], H[l], W[l]]
 *   y[t]          output [B, 4 + nc[t], A], A = sum_l H[l]*W[l]; rows cx, cy, w, h (pixels),
 *                 then sigmoid class scores -- the layout Detect.forward returns.
 *   strides[l]    pixel stride of level l (8, 16, 32 for P3..P5).
 */
int cerb_decode(const void* const* lvl, const int* nc, int T, int L, int B, const int* H, const int* W,
                const float* strides, int dtype, void* const* y, void* const* smax, int* summary_written,
                void* stream);

/*
 * The same decode reading SPLIT heads: the box channels and the class channels of every (task, level) stay in the
 * two tensors the conv towers wrote, so the reference's channel concat
 * `x[i] = torch.cat((self.cv2[i](x[i]), self.cv3[i](x[i])), 1)` (cerberusdet/models/yolo.py:89-90, a full copy of
 * the raw heads) is never materialised.  For callers that do not need the raw `x` Detect.forward returns next to y
 * (CerberusDetInference.predict drops it, cerberusdet_inference.py:119).
 *
 *   box_lvl[t*L + l]  [B, 64, H[l], W[l]]       (cv2[l]'s output)
 *   cls_lvl[t*L + l]  [B, nc[t], H[l], W[l]]    (cv3[l]'s output)
 * Everything else as cerb_decode; results are bit-identical to cerb_decode on the concatenated tensors.
 */
int cerb_decode_split(const void* const* box_lvl, const void* const* cls_lvl, const int* nc, int T, int L, int B,
                      const int* H, const int* W, const float* strides, int dtype, void* const* y, void* const* smax,
                      int* summary_written, void* stream);

/*
 * Head-tail fusion (fp16 only): the LAST 1x1 convolution of both conv towers of every (task, level)
 *   box = cv2[l][-1](u2), cls = cv3[l][-1](u3)   (cerberusdet/models/yolo.py:81-84, applied at :89-90)
 * fused with the channel concat (:90) and the eval decode (:93-99) in one persistent tcgen05 kernel: the raw head
 * tensor [B, 64+nc, H, W] is neither written nor re-read.  Per 128-anchor tile the two GEMMs
 * [128 x c2] x [c2 x 64] and [128 x c3] x [c3 x nc] run on the tensor cores (fp32 accumulators in TMEM, operands
 * brought in by TMA), and every epilogue thread decodes the anchor whose logits it reads back.
 *
 *   box_feat[t*L + l]  [B, c2[t], H[l], W[l]]  input of cv2[l][-1]      cls_feat[t*L + l]  [B, c3[t], H[l], W[l]]
 *   box_w[t*L + l]     [64, c2[t]] (the 1x1 kernel squeezed), box_b [64]; cls_w [nc[t], c3[t]], cls_b [nc[t]]
 *   y, smax, summary_written as in cerb_decode.
 * Needs c2, c3 multiples of 16, every H[l]*W[l] a multiple of 8 (16-byte rows for TMA), nc <= 192, 16-byte aligned
 * tensors; otherwise CERB_EINVAL (run the convolutions and cerb_decode_split instead).  The convolution output is
 * rounded to half (fp32 accumulation + bias, one rounding) before the decode, like the reference's half conv.
 */
int cerb_head_tail(const void* const* box_feat, const void* const* cls_feat, const void* const* box_w,
                   const void* const* box_b, const void* const* cls_w, const void* const* cls_b, const int* c2,
                   const int* c3, const int* nc, int T, int L, int B, const int* H, const int* W, const float* strides,
                   int dtype, void* const* y, void* const* smax, int* summary_written, void* stream);

/*
 * Score summary (optional by-product of cerb_decode, optional input of cerb_nms).
 *   smax[t]   [B, nc[t], R] in the tensor dtype, R = cerb_summary_row_len(A, dtype): entry (b, c, i) is
 *             the maximum of the 16-byte score vector i of class c, i.e. of the scores of anchors
 *             [i*V, i*V+V), V = 8 (fp16) / 4 (fp32); rows are padded to a multiple of V entries.
 * cerb_decode fills it when `smax` is non-NULL and the tensors allow the 128-bit path (every
 * H[l]*W[l] a multiple of V, 16-byte aligned pointers) and then sets *summary_written = 1.
 * cerb_nms uses it only to skip score vectors that cannot hold a candidate; results are identical
 * with and without it.  It must describe exactly the `pred` passed.
 */
size_t cerb_summary_row_len(int A, int dtype);

/* Bytes of device workspace cerb_nms / cerb_decode_nms need (0 unless max_det is large). */
size_t cerb_nms_workspace_bytes(int T, int B, int max_det);

/*
 * Confidence filter, best-class / multi-label candidate expansion, top-k (max_nms)
 * ordering, class-offset greedy NMS and the max_det cut for T task heads, every image
 * of the batch, in one launch.
 * Replaces non_max_suppression(prediction, conf_thres, iou_thres, classes, agnostic,
 * multi_label, labels=(), max_det, nm=0)  (cerberusdet/utils/general.py:360-481),
 * xywh2xyxy (:272-288) and the torchvision.ops.nms call at :464, as called per task by
 * cerberusdet/cerberusdet_inference.py:125-135, val.py:318 and detect.py:99.
 *
 *   pred[t]     [B, 4 + nc[t], A] prediction of task t (what Detect.forward returns)
 *   conf_thres, iou_thres   the Python floats; rounded inside exactly as torch does
 *               (conf to the tensor dtype; IoU quotient compared in double)
 *   classes     optional host list of class ids to keep (NULL / 0 = all)
 *   max_nms     30000 in the reference (:416); max_wh 7680 (:415)
 *   smax        optional score summaries from cerb_decode for exactly these predictions, or NULL
 *   dets        out [T, B, max_det, 6] fp32 rows (x1, y1, x2, y2, conf, cls), score order;
 *               only the first counts[t*B + b] rows of a segment are written
 *   counts      out [T, B] int32
 * Candidate order is "score descending, then (anchor, class) ascending" -- the stable
 * form of the reference's sort at :459, whose tie order is unspecified.
 */
int cerb_nms(const void* const* pred, const int* nc, int T, int B, int A, int dtype, double conf_thres,
             double iou_thres, const int* classes, int n_classes, int agnostic, int multi_label, int max_det,
             int max_nms, double max_wh, const void* const* smax, float* dets, int* counts, void* workspace,
             size_t workspace_bytes, void* stream);

/*
 * cerb_nms with per-segment statistics: stats is a device array [T*B][2] of 64-bit counters that receives, per
 * (task, image) segment, the number of IoU tests made and the number of candidates consumed from the sorted order
 * (bench.py reports IoU pairs/s from it; SURVEY 8d).  stats == NULL is exactly cerb_nms.
 */
int cerb_nms_stats(const void* const* pred, const int* nc, int T, int B, int A, int dtype, double conf_thres,
                   double iou_thres, const int* classes, int n_classes, int agnostic, int multi_label, int max_det,
                   int max_nms, double max_wh, const void* const* smax, float* dets, int* counts, void* workspace,
                   size_t workspace_bytes, unsigned long long* stats, void* stream);

/*
 * Multi-GPU delivery without a collective (SURVEY 8e: the one exchange of the path -- the padded detections of every
 * rank's images reach rank dst).  Rank dst owns, per (slot, rank), a region of device memory that is peer-mapped into
 * every writer (NVLink), and a writer signals / dst acknowledges through two 32-bit words per slot:
 *   flag    in dst's memory (peer-mapped into the writer): batches the writer has delivered into the slot.  Stored with
 *           release semantics at system scope by the LAST CTA of the delivering kernel, after every CTA has ordered its
 *           stores before its completion count at GPU scope (PTX causality order is transitive across the two scopes);
 *   ack     in the writer's memory, stored remotely by dst: batches dst has taken out of the slot.  A writer waits
 *           (bounded, ~2 s: a lost peer must not hang the GPU) until ack >= the batches it has written there before
 *           its first store, so a slot is never overwritten before dst has seen it;
 *   seq, done   local counters owned by the delivering kernel (zero-initialised once by the caller);
 *   collected   local counter owned by dst's kernel.
 * All of it is stream-ordered kernels, capturable in CUDA graphs: no NCCL kernel and no host synchronisation is on the
 * data path.  Three forms:
 *
 * cerb_nms_deliver, piggyback (push_src != NULL; what shard.PeerDelivery uses): cerb_nms writing LOCAL `dets` / `counts`
 *   as on one GPU; the launch gets up to 16 EXTRA CTAs that push the PREVIOUS batch's packed words (dets rows then
 *   counts, left in local staging by the previous launch: push_src -> push_dst, push_words 32-bit words, a multiple of
 *   4, both 16-byte aligned) with 128-bit stores and publish that slot's flag when they are done.  They run beside the
 *   segment CTAs, so the NVLink round trips of their fences are on nobody's critical path, and the step graph has no
 *   extra node.  On rank dst (collect_flags != NULL) one extra CTA takes the batch the writers pushed during the
 *   previous step: thread r waits for collect_flags[r] to exceed *collect_count and stores the acknowledgement into
 *   collect_ack[r] (rank r's ack word, peer-mapped).
 * cerb_nms_deliver, direct (push_src == NULL, flag_remote != NULL): `dets` / `counts` ARE dst's slot; rows cross NVLink
 *   one by one and the fences sit at the end of the NMS kernel (+7 us per step at N=2).
 * cerb_deliver_push / cerb_deliver_collect: the two sides as kernels of their own (the last batches of a run, and
 *   tools/side_probe.py).
 */
typedef struct cerb_delivery {
    const void* push_src;    /* writer, piggyback: previous batch in local staging, or NULL */
    void* push_dst;          /* ... its slot in dst's memory (peer-mapped) */
    size_t push_words;
    void* flag_remote;       /* writer: the slot's flag word in dst's memory; NULL = this launch delivers nothing */
    const void* ack_local;
    void* seq_local;
    void* done_local;
    const void* collect_flags;   /* dst: local [world] flag words of the slot to take, or NULL */
    void* collect_ack[16];       /* dst: rank r's ack word of that slot (peer-mapped); entry dst unused */
    void* collect_count;         /* dst: local counter of that slot */
    int world, dst;
} cerb_delivery;
int cerb_nms_deliver(const void* const* pred, const int* nc, int T, int B, int A, int dtype, double conf_thres,
                     double iou_thres, const int* classes, int n_classes, int agnostic, int multi_label, int max_det,
                     int max_nms, double max_wh, const void* const* smax, float* dets, int* counts, void* workspace,
                     size_t workspace_bytes, const cerb_delivery* delivery, void* stream);
int cerb_deliver_push(const void* src_local, void* dst_remote, size_t n_words, void* flag_remote, const void* ack_local,
                      void* seq_local, void* done_local, void* stream);
int cerb_deliver_collect(const void* flags_local, void* const* ack_remote, void* collected_local, int world, int dst,
                         void* stream);

/*
 * Decode + NMS for T task heads in one call (two launches on `stream`, no host work in between): the raw head
 * tensors go in, the padded detections come out; `y` (and `smax`, may be NULL) are caller-provided buffers that
 * receive the decoded predictions / score summary on the way (they are what Detect.forward would have returned).
 * Replaces the pair Detect.forward -> non_max_suppression as driven by
 * cerberusdet/cerberusdet_inference.py:117-135.  Arguments as in cerb_decode and cerb_nms.
 */
int cerb_decode_nms(const void* const* lvl, const int* nc, int T, int L, int B, const int* H, const int* W,
                    const float* strides, int dtype, void* const* y, void* const* smax, double conf_thres,
                    double iou_thres, const int* classes, int n_classes, int agnostic, int multi_label, int max_det,
                    int max_nms, double max_wh, float* dets, int* counts, void* workspace, size_t workspace_bytes,
                    void* stream);

/*
 * Cross-task merge of the per-task NMS results for a whole batch in one launch (one CTA per image).
 * Replaces the per-image host loop of CerberusDetInference.predict
 * (cerberusdet/cerberusdet_inference.py:140-155): _combine_output (:72-83, local -> global class ids),
 * nms_between_tasks (cerberusdet/utils/general.py:484-554, with box_iou of utils/metrics.py:415-433) and the
 * optional scale_boxes(...).round() (utils/general.py:313-357).
 *
 *   dets, counts   the outputs of cerb_nms: [T, B, max_det, 6], [T, B]
 *   class_offset   host [T]: global id = local id + class_offset[t]
 *   scale          optional device [B, 5] = (gain, pad_x, pad_y, orig_w, orig_h) per image, or NULL
 *   out            [B, T*max_det, 6] merged rows (x1, y1, x2, y2, conf, global cls), task order kept;
 *   out_counts     [B]
 * cerb_cross_task needs T*max_det <= 1024 (the per-image tables then always fit shared memory); cerb_cross_task_ws lifts
 * that (the reference's detect.py:124 runs max_det = 1000): images whose rows (the sum of the tasks' counts) exceed 1024
 * keep their tables in `workspace` (device memory, cerb_cross_task_workspace_bytes(T, B, max_det) bytes, 0 when
 * T*max_det <= 1024), every other image still runs out of shared memory.  max_det <= 65535.
 */
int cerb_cross_task(const float* dets, const int* counts, int T, int B, int max_det, const int* class_offset,
                    double iou_thres, const float* scale, float* out, int* out_counts, void* stream);
size_t cerb_cross_task_workspace_bytes(int T, int B, int max_det);
int cerb_cross_task_ws(const float* dets, const int* counts, int T, int B, int max_det, const int* class_offset,
                       double iou_thres, const float* scale, float* out, int* out_counts, void* workspace,
                       size_t workspace_bytes, void* stream);

/*
 * Which detections are correct at each IoU threshold, for a whole batch of ONE task in one launch (one CTA per image).
 * Replaces process_batch (cerberusdet/val.py:32-54) as called per image by the validation loop (val.py:321-357).
 *
 *   dets, counts     [B, max_det, 6] / [B]: detections already in native image space (scale_boxes applied)
 *   labels           device [sum_b M_b, 5] rows (cls, x1, y1, x2, y2), native space, images concatenated
 *   label_offsets    device [B + 1] row offsets into labels; max_labels_per_image = max_b M_b (<= 1024)
 *   iouv             host [K] thresholds (K <= 16; the reference uses linspace(0.5, 0.95, 10))
 *   correct          out [B, max_det, K] bytes (0/1); rows past counts[b] are 0
 * Equal IoUs of one detection with two labels resolve to the lower label index (the reference's numpy sort is
 * unstable there).
 */
int cerb_val_match(const float* dets, const int* counts, int B, int max_det, const float* labels,
                   const int* label_offsets, int max_labels_per_image, const float* iouv, int K,
                   unsigned char* correct, void* stream);

/*
 * Training-time sibling of the decode (SURVEY 8f row 4): Loss.bbox_decode (cerberusdet/utils/loss.py:126-131) =
 * softmax over the reg_max bins of each side, expectation with proj = arange(reg_max), then
 * dist2bbox(xywh=False) (cerberusdet/utils/tal.py:196-205).
 *
 *   pred_dist       [n_rows, 4 * reg_max], n_rows = B * A, the bins of a side contiguous (loss.py:139-146), fp16 | fp32
 *   anchor_points   [A, 2] (x, y) in grid units, same dtype (make_anchors, tal.py:181-193)
 *   out             [n_rows, 4] = (x1, y1, x2, y2) in grid units, same dtype
 * reg_max must be 16 (models/yolo.py:75).  Half tensors round where the reference's do (softmax output, the
 * expectation, the corner).
 */
int cerb_bbox_decode_fwd(const void* pred_dist, const void* anchor_points, long n_rows, int A, int reg_max, int dtype,
                         void* out, void* stream);

/*
 * Its backward: grad_pred_dist [n_rows, 4 * reg_max] from grad_out [n_rows, 4] -- the fused autograd of
 * dist2bbox (sign), matmul (g * k, rounded in the tensor dtype) and softmax (p_j * (gp_j - sum_k gp_k p_k));
 * the probabilities are recomputed from pred_dist.
 */
int cerb_bbox_decode_bwd(const void* pred_dist, const void* grad_out, long n_rows, int reg_max, int dtype,
                         void* grad_pred_dist, void* stream);

/*
 * The training-time sibling's caller (SURVEY 8f row 4): TaskAlignedAssigner.forward (cerberusdet/utils/tal.py:56-178, with
 * select_candidates_in_gts :13-28, select_highest_overlaps :31-53 and bbox_iou(CIoU=True) of utils/metrics.py:373-408), as
 * called by the loss at cerberusdet/utils/loss.py:160-162, in three launches.
 *
 *   pd_scores     [B, A, C] sigmoid scores, fp16 | fp32 (score_dtype)      pd_bboxes   [B, A, 4] xyxy pixels, fp32
 *   anc_points    [A, 2] anchor centres in pixels, fp32
 *   gt_labels     [B, G] class ids as floats, gt_bboxes [B, G, 4] xyxy pixels, mask_gt [B, G] 1 = real box, 0 = padding
 *   topk (<= 16), alpha, beta, eps: the assigner's attributes (10, 0.5, 6.0, 1e-9 in the reference, loss.py:100-105)
 *   out: target_labels [B, A] int64, target_bboxes [B, A, 4] fp32, target_scores [B, A, C] fp32, fg_mask [B, A] bool
 *        (one byte each), target_gt_idx [B, A] int64 -- exactly the five tensors forward returns
 *   workspace: cerb_tal_workspace_bytes(B, A, G, topk) bytes of device memory
 * G >= 1 (the reference returns early for G == 0, tal.py:89-93: the caller keeps that branch), G <= 1024.
 * Equal metrics rank by anchor index ascending -- the reference's torch.topk (:140) leaves their order unspecified; it
 * only matters for boxes with fewer than topk positive-metric anchors AND anchors inside whose CIoU is <= 0.
 */
size_t cerb_tal_workspace_bytes(int B, int A, int G, int topk);
int cerb_tal_assign(const void* pd_scores, const float* pd_bboxes, const float* anc_points, const float* gt_labels,
                    const float* gt_bboxes, const float* mask_gt, int B, int A, int C, int G, int topk, double alpha,
                    double beta, double eps, int score_dtype, long long* target_labels, float* target_bboxes,
                    float* target_scores, unsigned char* fg_mask, long long* target_gt_idx, void* workspace,
                    size_t workspace_bytes, void* stream);

/*
 * The box-regression term of the training loss (SURVEY 8f row 4, the step after the assigner): BboxLoss.forward
 * (cerberusdet/utils/loss.py:12-44) with use_dfl and 16 bins, i.e. the CIoU loss (bbox_iou(xywh=False, CIoU=True),
 * utils/metrics.py:373-408) and the distribution focal loss against bbox2dist(anchor_points, target_bboxes, 15)
 * (utils/tal.py:208-211), both summed over the foreground anchors, weighted by the target-score row sums and divided by
 * target_scores_sum.  One launch; no host synchronisation (the reference's boolean-mask indexing costs five).
 *
 *   pred_dist      [B, A, 4 * reg_max] (bins of a side contiguous), dtype, 32-byte aligned
 *   pred_bboxes    [B, A, 4] xyxy grid units, dtype        anchor_points [A, 2] grid units, dtype
 *   target_bboxes  [B, A, 4] xyxy grid units, fp32        target_scores [B, A, C] fp32      fg_mask [B, A] bool bytes
 *   target_scores_sum   device fp32 scalar, or NULL: target_scores_sum_host is used
 *   dtype          CERB_F32: every tensor above fp32.  CERB_F16: the trainer's fp16 autocast case -- half predictions and
 *                  anchors, fp32 targets; the reference's half roundings (w1, h1, w1*h1, w1/h1, atan(w1/h1), the
 *                  cross-entropy's log-probabilities) are kept
 *   loss_iou, loss_dfl   out: device fp32 scalars
 *   per_anchor     optional out [B, A, 2] fp32: (1 - CIoU) * weight and DFL * weight per anchor (0 at background), or NULL
 *   workspace      cerb_bbox_loss_workspace_bytes(B, A) bytes, 16-byte aligned, ZEROED before its first use (the
 *                  kernel leaves it reusable: it resets its counter, so CUDA-graph replays need nothing else)
 * Sums are reduced in a fixed order: equal inputs give equal bits.  reg_max must be 16; CERB_EINVAL for another value,
 * an unknown dtype, misaligned rows or B*A beyond 2^31 - 1.
 */
size_t cerb_bbox_loss_workspace_bytes(int B, int A);
int cerb_bbox_loss_fwd(const void* pred_dist, const void* pred_bboxes, const void* anchor_points, const float* target_bboxes,
                       const float* target_scores, const unsigned char* fg_mask, const float* target_scores_sum,
                       double target_scores_sum_host, int B, int A, int C, int reg_max, int dtype, float* loss_iou,
                       float* loss_dfl, float* per_anchor, void* workspace, size_t workspace_bytes, void* stream);

/*
 * Its backward (loss.py:12-44, tal.py:208-211, metrics.py:373-408), recomputed from the same inputs: grad_iou and
 * grad_dfl are the device fp32 gradients of the two scalars; out grad_pred_dist [B, A, 64] (dense: zeros at background
 * anchors, 32-byte aligned) and grad_pred_bboxes [B, A, 4], both in dtype.  Autograd's conventions: CIoU's alpha is a
 * constant, minimum / maximum split the gradient in half on exact ties, clamp(0) passes it at exactly 0, and the
 * cross-entropy gradient is softmax - onehot in fp32, rounded once to dtype.
 */
int cerb_bbox_loss_bwd(const void* pred_dist, const void* pred_bboxes, const void* anchor_points, const float* target_bboxes,
                       const float* target_scores, const unsigned char* fg_mask, const float* target_scores_sum,
                       double target_scores_sum_host, int B, int A, int C, int reg_max, int dtype, const float* grad_iou,
                       const float* grad_dfl, void* grad_pred_dist, void* grad_pred_bboxes, void* stream);

/*
 * Per-class average precision of the validation statistics: ap_per_class (cerberusdet/utils/metrics.py:56-120) with
 * compute_ap (np.interp of the precision envelope at np.linspace(0, 1, 101), np.trapz), up to the per-class arrays; the
 * caller does the O(nc * 1000) tail (f1, smooth, argmax, rounded tp / fp).  Detections are ordered by conf descending,
 * ties by row index ascending: np.argsort(-conf, kind="stable"), with -0.0 == 0.0 (the reference's unstable argsort has
 * no defined order on ties).  Every float64 value is the reference's own IEEE operation, so the outputs equal numpy's
 * bit for bit.
 *
 *   tp        [n, K] bytes, nonzero = true positive at IoU threshold j     conf, pred_cls   [n] fp32
 *   classes   HOST [nc] fp32, strictly ascending (np.unique of the target classes); a detection whose class is not
 *             among them (or NaN) is ignored, as `pred_cls == c` ignores it
 *   n_labels  HOST [nc] labels per class (np.unique's counts)                eps              the reference's 1e-16
 *   ap        out [nc, K] fp64      p, r   out [nc, 1000] fp64: precision / recall at px = np.linspace(0, 1, 1000) of
 *             column 0, np.interp(-px, -conf, ., left=1 | 0).  A class with no detection or no label keeps zero rows.
 *   workspace cerb_ap_workspace_bytes(n, K, nc) bytes, 256-byte aligned (0 returned: the size cannot be computed,
 *             e.g. without a CUDA device)
 * Requires what process_batch guarantees: per class and column, at most n_labels true positives (recall <= 1).
 * CERB_EINVAL for n outside 0..2^31-1, K outside 1..32, nc < 0, classes not strictly ascending or NaN, negative
 * n_labels; CERB_ENOSPC for a workspace that is too small.  n == 0 or nc == 0 is valid (zero outputs).
 */
size_t cerb_ap_workspace_bytes(long n, int K, int nc);
int cerb_ap_per_class(const unsigned char* tp, int K, const float* conf, const float* pred_cls, long n, const float* classes,
                      const long long* n_labels, int nc, double eps, double* ap, double* p, double* r, void* workspace,
                      size_t workspace_bytes, void* stream);

/*
 * Test / tools hooks.  cerb_debug_set(name, value) overrides one internal choice FOR THE CALLING THREAD (so the
 * library stays re-entrant); cerb_debug_reset() drops every override of the calling thread.  Results never depend
 * on a knob: the parity tests run the alternatives against each other.  Knobs: "decode_pipe" (0 = register-resident
 * decode kernel instead of the pipelined one), "decode_order", "decode_vec", "decode_l2hint", "nms_minb" (1 | 2: the
 * 128- / 64-register NMS build), "nms_pdl" (0 = no programmatic dependent launch), "decode_pdl" (1 = the decode
 * launch carries the programmatic-serialization attribute: behind an NMS launch of another batch in the same stream it starts
 * as soon as every NMS CTA is running -- the single-stream overlapped schedule of pipeline.py; the decode reads nothing the
 * kernel before it writes), "chunk_cap", "chunk_first",
 * "hist_sample", "ht_order" (head-tail kernel: 0 = tiles dealt round-robin to the CTAs, 1 = contiguous runs), "ht_stages"
 * (cap on its activation ring depth), "ht_groups" (its epilogue warp groups, 1 | 2).
 */
int cerb_debug_set(const char* name, int value);
int cerb_debug_reset(void);

/*
 * Test hook: override the chunk capacity (16..4096) and first-chunk target of the lazy
 * top-k so small inputs exercise the multi-chunk and radix-refinement paths.
 * (0, 0) restores the defaults.  Results never depend on these values.
 */
int cerb_debug_set_chunking(int chunk_cap, int chunk_first);

/*
 * Test hook: stride (in 16-byte score vectors) of the estimating histogram that sizes the
 * chunks of large multi-label segments; 1 = always exact, 0 = default (8).  Results never
 * depend on it.
 */
int cerb_debug_set_hist_sample(int stride);

#ifdef __cplusplus
}
#endif
#endif /* CERB_POST_H */
