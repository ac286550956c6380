// The validation confusion matrix: ConfusionMatrix.process_batch (cerberusdet/utils/metrics.py:273-370), which the
// validation loop calls per image when plots are on, for a whole batch in one launch, one CTA per image.  The reference
// does it with numpy argsort / unique and two Python loops that read the class of every row back from the device.
//
// Per image: keep the detections with conf > thr_conf (order preserved, so "lowest filtered index" is "lowest original
// index" and no compaction is needed); a detection's best label is the highest IoU > thr_iou, ties -> lowest label
// index; a label's winner among the detections that chose it is the highest IoU, ties -> lowest detection index (the
// canonical form of the reference's two unstable argsorts).  Then every label adds [cls(winner), cls(label)] or
// [nc, cls(label)], and -- only when some pair survived, the reference's `if n:` -- every unmatched conf-passing
// detection adds [cls(det), nc].  Classes are the fp32 values truncated to int (`.int()`).
#include "cerb_kernels.h"

#define CM_THREADS 256
#define CM_FILTERED -2  // best[d] of a detection at or below the conf threshold (-1: passes, no label above thr_iou)

__device__ __forceinline__ bool cm_class_ok(float c, int nc) { return c > -1.f && c < (float)nc; }  // trunc(c) in [0, nc)

__global__ void __launch_bounds__(CM_THREADS) confusion_kernel(const __grid_constant__ ConfusionParams P) {
    extern __shared__ short best[];                        // [max_det]: best label of each detection, -1 or CM_FILTERED
    __shared__ unsigned long long win[CERB_CM_MAX_LABELS];  // per label: (IoU bits << 32) | ~index of its winner, 0 = none
    __shared__ int s_flags, s_any;
    const int b = blockIdx.x, tid = threadIdx.x, nc = P.nc, W = nc + 1;
    const int l0 = P.label_offsets ? P.label_offsets[b] : 0;
    const int M = P.label_offsets ? P.label_offsets[b + 1] - l0 : P.n_labels;
    const int N = P.counts ? min(max(P.counts[b], 0), P.max_det) : P.max_det;
    const bool labels_ok = l0 >= 0 && M >= 0 && M <= CERB_CM_MAX_LABELS && l0 + M <= P.n_labels;
    const float* dets = P.dets + (size_t)b * P.max_det * 6;
    const float* labels = P.labels + (size_t)l0 * 5;
    int* label_cells = P.cells ? P.cells + l0 : nullptr;
    int* det_cells = P.cells ? P.cells + P.n_labels + (size_t)b * P.max_det : nullptr;
    if (tid == 0) {
        s_flags = labels_ok ? 0 : CERB_CM_LABEL_COUNT;
        s_any = 0;
    }
    __syncthreads();
    // every class the reference indexes the matrix with: all labels', the conf-passing detections'
    bool bad = false;
    if (labels_ok) {
        for (int l = tid; l < M; l += CM_THREADS) {
            bad |= !cm_class_ok(labels[(size_t)l * 5], nc);
            win[l] = 0ull;
        }
        for (int d = tid; d < N; d += CM_THREADS)
            if (dets[(size_t)d * 6 + 4] > P.conf) bad |= !cm_class_ok(dets[(size_t)d * 6 + 5], nc);
    }
    if (bad) atomicOr(&s_flags, CERB_CM_CLASS_RANGE);
    __syncthreads();
    const int flags = s_flags;
    if (flags) {  // the image adds nothing; its rows say so
        if (tid == 0) P.status[b] = flags;
        if (label_cells && labels_ok)
            for (int l = tid; l < M; l += CM_THREADS) label_cells[l] = -1;
        if (det_cells)
            for (int d = tid; d < P.max_det; d += CM_THREADS) det_cells[d] = -1;
        return;
    }
    // per conf-passing detection: its best label with IoU > thr_iou, and that label's atomicMax claim
    for (int d = tid; d < N; d += CM_THREADS) {
        const float* r = dets + (size_t)d * 6;
        int bl = CM_FILTERED;
        if (r[4] > P.conf) {
            const float x1 = r[0], y1 = r[1], x2 = r[2], y2 = r[3];
            const float ad = __fmul_rn(__fsub_rn(x2, x1), __fsub_rn(y2, y1));
            float biou = P.iou_thr;
            bl = -1;
            for (int l = 0; l < M; ++l) {
                const float iou = cerb_box_iou(labels + (size_t)l * 5, x1, y1, x2, y2, ad);
                if (iou > biou) { biou = iou; bl = l; }  // strict: only IoU > thr_iou, and the lowest label wins ties
            }
            if (bl >= 0) {  // IoU > thr_iou >= 0: a positive float, whose bits order as unsigned
                atomicMax(&win[bl], ((unsigned long long)__float_as_uint(biou) << 32) | (unsigned)~d);
                s_any = 1;
            }
        }
        best[d] = (short)bl;
    }
    __syncthreads();
    const bool any = s_any;
    if (tid == 0) P.status[b] = 0;
    for (int l = tid; l < M; l += CM_THREADS) {
        const unsigned long long k = win[l];
        const int row = k ? (int)dets[(size_t)(~(unsigned)k) * 6 + 5] : nc;
        const int cell = row * W + (int)labels[(size_t)l * 5];
        if (label_cells) label_cells[l] = cell;
        if (P.matrix) atomicAdd(P.matrix + cell, 1ull);
    }
    if (!det_cells && !any) return;
    for (int d = tid; d < P.max_det; d += CM_THREADS) {
        int cell = -1;
        if (d < N && any) {
            const int bl = best[d];
            if (bl == -1 || (bl >= 0 && (unsigned)win[bl] != (unsigned)~d)) cell = (int)dets[(size_t)d * 6 + 5] * W + nc;
        }
        if (det_cells) det_cells[d] = cell;
        if (cell >= 0 && P.matrix) atomicAdd(P.matrix + cell, 1ull);
    }
}

cudaError_t cerb_launch_confusion(const ConfusionParams& P, cudaStream_t stream) {
    if (P.B == 0) return cudaSuccess;
    const size_t smem = (size_t)(P.max_det > 0 ? P.max_det : 1) * sizeof(short);
    cudaError_t e = cudaFuncSetAttribute(confusion_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    confusion_kernel<<<P.B, CM_THREADS, smem, stream>>>(P);
    return cudaGetLastError();
}
