// Kernel parameter blocks and launchers shared by decode.cu / nms.cu / api.cu.
#pragma once
#include "cerb_common.cuh"


// ------------------------------------------------------------------ decode
struct DecodeParams {
    const void* lvl[CERB_MAX_TASKS][CERB_MAX_LEVELS];  // raw head tensors [B, 64+nc, H_l, W_l]
    // optional split heads: class channels [B, nc, H_l, W_l] of each (task, level) in their own tensor (the cv3 tower's
    // output) and lvl = the box channels [B, 64, H_l, W_l] alone (cv2's output) -- the reference's channel concat
    // (models/yolo.py:90) is then never materialised.  null = lvl holds both, concatenated
    const void* cls[CERB_MAX_TASKS][CERB_MAX_LEVELS];
    void* y[CERB_MAX_TASKS];                           // decoded [B, 4+nc, A]
    int nc[CERB_MAX_TASKS];
    int hw[CERB_MAX_LEVELS];
    int w[CERB_MAX_LEVELS];
    int aoff[CERB_MAX_LEVELS];  // first anchor of each level inside A
    float stride[CERB_MAX_LEVELS];
    int B, A, T, L;
    int nrows;                                                  // T * L
    int row_start[2 * CERB_MAX_TASKS * CERB_MAX_LEVELS + 1];    // first block of each row ((task, level), or (kind, task, level) in box-first order)
    int row_blocks_per_part[CERB_MAX_TASKS * CERB_MAX_LEVELS];  // ceil(B * nvecp / threads)
    void* smax[CERB_MAX_TASKS];  // optional score summary [B, nc, A/V]: max of every 16-byte score vector
    int l2_evict_first;          // pipelined kernel: read the raw heads with an L2 evict-first policy (outputs fit in L2)
    int pdl;                     // host only: launch with programmatic stream serialization -- the grid may start as soon as the
                                 // kernel before it in the stream has released its dependents (the NMS kernel of the PREVIOUS
                                 // batch does so at entry); the decode reads nothing that kernel writes, so it never waits
    int interleave_parts;        // block order: 0 parts contiguous per (task, level), 1 interleaved, 2 all DFL blocks first, then all class blocks
};
cudaError_t cerb_launch_decode(DecodeParams& P, int dtype, int vec, cudaStream_t stream);
// software-pipelined variant (cp.async prefetch into per-thread shared-memory slots, ipt items per thread);
// needs vec == 16 / sizeof(T); cudaErrorInvalidConfiguration = use the other one
cudaError_t cerb_launch_decode_pipe(const DecodeParams& P, int dtype, int ipt, cudaStream_t stream);

// ------------------------------------------------------------------ select + NMS
#define CERB_MAX_CLASS_WORDS 32  // class filter bitmask: nc <= 1024

struct NmsParams {
    const void* pred[CERB_MAX_TASKS];  // [B, 4+nc, A], dtype below
    int nc[CERB_MAX_TASKS];
    int T, B, A;
    float conf_thr;   // already rounded to the prediction dtype (reference general.py:411)
    float iou_thr;    // largest float <= the double threshold: (double)ovr > thr  <=>  ovr > iou_thr
    float class_gap;  // max_wh (7680) or 0 when agnostic (general.py:462)
    int multi_label;
    int max_det, max_nms;
    int use_class_filter;
    unsigned class_mask[CERB_MAX_CLASS_WORDS];
    float* dets;     // [T, B, max_det, 6]
    int* counts;     // [T, B]
    float* kept_ws;  // global kept-list storage [T*B, max_det, 5] when max_det is too large for smem, else null
    int chunk_cap;   // candidates sorted per chunk (<= NMS_CAP); tests shrink it to force the rare paths
    int chunk_first; // size target of the first chunk
    int hist_sample; // stride (in 16-byte vectors) of the estimating histogram; 1 = exact
    int class_shortcut; // 1 if different-class tame boxes provably never intersect after the offset
    const void* smax[CERB_MAX_TASKS];  // optional score summary [B, nc, A/V] from the decode kernel (else null)
    float tame_lo, tame_hi; // the window of "tame" un-offset coordinates, tame_hi - tame_lo == class_gap
    unsigned long long* pair_counts;  // optional [T*B][2]: IoU tests made, candidates consumed (statistics), else null
    int force_minb;         // host only: 0 = pick the register build per launch, 1 / 2 = force it (tests, tools)
    int pdl;                // host only: launch with programmatic stream serialization (default 1)
    // Multi-GPU delivery without a collective (shard.py: PeerDelivery): `dets` / `counts` point into rank dst's
    // peer-mapped memory; the kernel itself tells dst when the batch is complete and waits for dst before it reuses the
    // slot.  All four null = off.
    unsigned* deliver_flag;        // dst's memory (peer-mapped): batches this rank has delivered into this slot
    const unsigned* deliver_ack;   // local, written remotely by dst: batches dst has taken out of this slot
    unsigned* deliver_seq;         // local: batches this rank has written into this slot (kept by the kernel)
    unsigned* deliver_done;        // local: CTA completion counter of the running launch (zero between launches)
    // piggyback form (default of shard.PeerDelivery): `dets` / `counts` are LOCAL; the launch additionally pushes the
    // PREVIOUS batch's packed words (left in local staging by the previous launch) into dst's slot at its start -- the
    // four words above then describe that slot -- so the remote stores have ~50 us to land before the fences at the end
    const float* push_src;         // local staging of the previous batch (16-byte aligned), null = direct form
    float* push_dst;               // dst's slot (peer-mapped)
    unsigned push_words;           // multiple of 4
    int deliver_ctas;              // host only -> kernel: extra CTAs of the launch that do the delivery (0 = none)
    // rank dst: CTA 0 takes the batch the other ranks pushed during the previous step (cerb_deliver_collect's job)
    const unsigned* col_flags;     // local [world], null = off
    unsigned* col_ack[16];         // peer-mapped
    unsigned* col_collected;       // local counter of that slot
    int col_world, col_dst;
};
cudaError_t cerb_launch_nms(const NmsParams& P, int dtype, cudaStream_t stream);
// dst's side of the delivery: one CTA; thread r waits until rank r's flag reaches (*collected + 1), then acknowledges
// into rank r's memory (ack[r], peer-mapped); *collected is advanced at the end
#define CERB_MAX_RANKS 16
struct CollectParams {
    const unsigned* flags;            // local [world]
    unsigned* ack[CERB_MAX_RANKS];    // peer-mapped, entry dst unused
    unsigned* collected;              // local counter of this slot
    int world, dst;
};
cudaError_t cerb_launch_deliver_collect(const CollectParams& P, cudaStream_t stream);
struct PushParams {
    const float* src;      // local: one batch's packed words (dets rows, then counts), 16-byte aligned
    float* dst;            // rank dst's slot (peer-mapped), 16-byte aligned
    size_t n_words;        // 32-bit words to copy, a multiple of 4
    unsigned* flag;        // dst's memory (peer-mapped)
    const unsigned* ack;   // local, written remotely by dst
    unsigned* seq;         // local
    unsigned* done;        // local
    int mode;              // 0; tools only: 1 = skip the fences and the flag, 2 = skip the copy
};
cudaError_t cerb_launch_deliver_push(const PushParams& P, int ctas, cudaStream_t stream);
size_t cerb_nms_kept_ws_bytes(int T, int B, int max_det);

// ------------------------------------------------------------------ cross-task merge (SURVEY 8f-1)
struct CrossTaskParams {
    const float* dets;       // [T, B, max_det, 6] per-task NMS rows (local class ids)
    const int* counts;       // [T, B]
    int T, B, max_det;
    int class_offset[CERB_MAX_TASKS];  // local -> global class id
    float iou_thr;           // (float)iou_thres_between_tasks: compared like the reference's fp32 matrix > python float
    const float* scale;      // optional [B, 5]: gain, pad_x, pad_y, orig_w, orig_h (scale_boxes + round), else null
    float* out;              // [B, T*max_det, 6] merged rows, global class ids
    int* out_counts;         // [B]
    unsigned char* workspace;  // global tables for images with more than 1024 rows (cerb_cross_task_ws_bytes), else null
};
cudaError_t cerb_launch_cross_task(const CrossTaskParams& P, cudaStream_t stream);
size_t cerb_cross_task_ws_bytes(int T, int B, int max_det);

// ------------------------------------------------------------------ validation matching (SURVEY 8f-2)
struct ValMatchParams {
    const float* dets;          // [B, max_det, 6] native-space detections of ONE task (x1, y1, x2, y2, conf, cls)
    const int* counts;          // [B]
    const float* labels;        // [sum M_b, 5] (cls, x1, y1, x2, y2), images concatenated
    const int* label_offsets;   // device [B + 1]
    int B, max_det, K;
    float iouv[16];             // IoU thresholds (val.py: linspace(0.5, 0.95, 10))
    unsigned char* correct;     // [B, max_det, K]
};
cudaError_t cerb_launch_val_match(const ValMatchParams& P, int max_labels_per_image, cudaStream_t stream);

// box_iou (utils/metrics.py:415-433) of one label row q = (cls, x1, y1, x2, y2) and one detection (x1, y1, x2, y2) whose
// area ad = (x2 - x1) * (y2 - y1) the caller computed: fp32, one rounding per operation, + 1e-7 in the denominator
__device__ __forceinline__ float cerb_box_iou(const float* q, float x1, float y1, float x2, float y2, float ad) {
    const float iw = fmaxf(__fsub_rn(fminf(q[3], x2), fmaxf(q[1], x1)), 0.f);
    const float ih = fmaxf(__fsub_rn(fminf(q[4], y2), fmaxf(q[2], y1)), 0.f);
    const float inter = __fmul_rn(iw, ih);
    const float al = __fmul_rn(__fsub_rn(q[3], q[1]), __fsub_rn(q[4], q[2]));
    return __fdiv_rn(inter, __fadd_rn(__fsub_rn(__fadd_rn(al, ad), inter), 1e-7f));
}

// ------------------------------------------------------------------ validation confusion matrix (confusion.cu)
#define CERB_CM_MAX_LABELS 1024
#define CERB_CM_MAX_DETS 30000
#define CERB_CM_MAX_NC 32767         // (nc + 1)^2 cells index in 32 bits
#define CERB_CM_CLASS_RANGE 1        // status: a label or conf-passing detection has a class outside [0, nc)
#define CERB_CM_LABEL_COUNT 2        // status: the image's label rows are not within [0, 1024] / inside labels
struct ConfusionParams {
    const float* dets;           // [B, max_det, 6] (x1, y1, x2, y2, conf, cls)
    const int* counts;           // [B], or null: every image has max_det detections
    const float* labels;         // [n_labels, 5] (cls, x1, y1, x2, y2), images concatenated
    const int* label_offsets;    // device [B + 1], or null (B == 1): all n_labels rows are image 0's
    int B, max_det, n_labels, nc;
    float conf, iou_thr;         // the Python floats rounded to fp32, as torch compares an fp32 tensor with them
    unsigned long long* matrix;  // optional [nc + 1, nc + 1] int64, added to
    int* cells;                  // optional [n_labels + B * max_det]: the cell each label / detection row adds to, or -1
    int* status;                 // [B]
};
cudaError_t cerb_launch_confusion(const ConfusionParams& P, cudaStream_t stream);

// ------------------------------------------------------------------ training-time sibling decode (SURVEY 8f-4)
// Loss.bbox_decode forward / backward on pred_dist [n_rows = B * A, 64] (bins contiguous); train_decode.cu
cudaError_t cerb_launch_bbox_decode_fwd(const void* pred, const void* anchor_points, long n_rows, int A, int dtype, void* out,
                                        cudaStream_t stream);
cudaError_t cerb_launch_bbox_decode_bwd(const void* pred, const void* grad_out, long n_rows, int dtype, void* grad_in,
                                        cudaStream_t stream);

// ------------------------------------------------------------------ letterbox preprocessing (SURVEY row 10)
#define CERB_LB_MAX_IMAGES 256  // images per launch (the table travels in the kernel parameters: 40 B each)
#define CERB_LB_MAX_SIDE 32768  // longest image or output side (keeps every offset of the kernel in 32 bits)
struct LbImage {
    const unsigned char* src;  // uint8 HWC BGR rows
    long long pitch;           // bytes between rows, >= 3 * w
    int h, w;                  // source size
    int uh, uw;                // resized size (cv2.resize's dsize)
    int top, left;             // border above / left of the resized image
};
struct LetterboxParams {
    LbImage img[CERB_LB_MAX_IMAGES];
    void* out;  // [n_images, 3, out_h, out_w] dtype: RGB planes, value / 255
    int out_h, out_w;
};
// letterbox.cu; one CTA column per image of P.img[0 .. n_images)
cudaError_t cerb_launch_letterbox(const LetterboxParams& P, int n_images, int dtype, cudaStream_t stream);
