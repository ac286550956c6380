// Which detections are correct at each IoU threshold -- the statistics step right after NMS in the reference
// validation loop (SURVEY section 8f row 2): process_batch (cerberusdet/val.py:32-54), for a whole batch in one
// launch, one CTA per image.  The reference does it per image with numpy argsort/unique on the host.
//
// Per threshold t: pairs (label, detection) with iou >= t and equal class, sorted by IoU descending; a detection
// keeps its best label; per label the lowest detection index survives (val.py:48-51).  The best label of a
// detection does not depend on t (it is the arg-max IoU over the class-matching labels; ties -> lowest label, the
// canonical form of the reference's unstable sort), so one pass finds it and K atomicMin tables resolve the labels.
// IoU: cerb_box_iou (cerb_kernels.h), box_iou's arithmetic.
#include "cerb_kernels.h"

#define VM_THREADS 256
#define VM_MAX_LABELS 1024
#define VM_MAX_THR 16

__global__ void __launch_bounds__(VM_THREADS) val_match_kernel(const __grid_constant__ ValMatchParams P) {
    extern __shared__ int first[];  // [K][labels of this image]: lowest detection index claiming the label
    const int b = blockIdx.x, tid = threadIdx.x;
    const int l0 = P.label_offsets[b], M = P.label_offsets[b + 1] - l0;
    const int N = min(max(P.counts[b], 0), P.max_det);
    const int K = P.K;
    for (int i = tid; i < K * M; i += VM_THREADS) first[i] = 0x7fffffff;
    __syncthreads();
    const float* dets = P.dets + (size_t)b * P.max_det * 6;
    unsigned char* out = P.correct + (size_t)b * P.max_det * K;
    // per detection: best class-matching label
    for (int d0 = 0; d0 < N; d0 += VM_THREADS) {
        const int d = d0 + tid;
        float biou = -1.f;
        int bl = -1;
        if (d < N) {
            const float* r = dets + (size_t)d * 6;
            const float x1 = r[0], y1 = r[1], x2 = r[2], y2 = r[3], cls = r[5];
            const float ad = __fmul_rn(__fsub_rn(x2, x1), __fsub_rn(y2, y1));
            for (int l = 0; l < M; ++l) {
                const float* q = P.labels + (size_t)(l0 + l) * 5;
                if (q[0] != cls) continue;
                const float iou = cerb_box_iou(q, x1, y1, x2, y2, ad);
                if (iou > biou) { biou = iou; bl = l; }  // strict: the lowest label wins ties
            }
            if (bl >= 0)
                for (int i = 0; i < K; ++i)
                    if (biou >= P.iouv[i]) atomicMin(&first[i * M + bl], d);
        }
        __syncthreads();  // (N <= max_det: all rounds' claims are in before anyone reads -- see the second loop)
        (void)biou;
    }
    __syncthreads();
    for (int d0 = 0; d0 < N; d0 += VM_THREADS) {
        const int d = d0 + tid;
        if (d >= N) continue;
        // recompute the best label (cheaper than keeping per-detection state across the barrier for N > 256)
        const float* r = dets + (size_t)d * 6;
        const float x1 = r[0], y1 = r[1], x2 = r[2], y2 = r[3], cls = r[5];
        const float ad = __fmul_rn(__fsub_rn(x2, x1), __fsub_rn(y2, y1));
        float biou = -1.f;
        int bl = -1;
        for (int l = 0; l < M; ++l) {
            const float* q = P.labels + (size_t)(l0 + l) * 5;
            if (q[0] != cls) continue;
            const float iou = cerb_box_iou(q, x1, y1, x2, y2, ad);
            if (iou > biou) { biou = iou; bl = l; }
        }
        for (int i = 0; i < K; ++i)
            out[(size_t)d * K + i] = (bl >= 0 && biou >= P.iouv[i] && first[i * M + bl] == d) ? 1 : 0;
    }
    for (int i = N * K + tid; i < P.max_det * K; i += VM_THREADS) out[i] = 0;  // padding rows
}

cudaError_t cerb_launch_val_match(const ValMatchParams& P, int max_labels_per_image, cudaStream_t stream) {
    if (P.B == 0) return cudaSuccess;
    if (max_labels_per_image > VM_MAX_LABELS || P.K > VM_MAX_THR) return cudaErrorInvalidConfiguration;
    const size_t smem = (size_t)P.K * (max_labels_per_image > 0 ? max_labels_per_image : 1) * sizeof(int);
    cudaError_t e = cudaFuncSetAttribute(val_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    val_match_kernel<<<P.B, VM_THREADS, smem, stream>>>(P);
    return cudaGetLastError();
}
