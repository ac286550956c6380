// SURVEY 8f row 4 (the training-time sibling's caller): TaskAlignedAssigner.forward (reference utils/tal.py:56-178 with
// select_candidates_in_gts :13-28, select_highest_overlaps :31-53, bbox_iou(CIoU) utils/metrics.py:373-408) in three
// launches instead of the reference's ~60 elementwise / topk / one_hot / gather launches over [B, G, A] tensors (five of
// them materialised: 43 MB each at B=64, G=20, A=8400).
//
//   tal_topk_kernel    one CTA per (image, ground-truth box): the topk anchors by  metric = score^alpha * CIoU^beta * inside
//                      (only anchors INSIDE the box need the CIoU; every thread keeps the best topk of its own anchors in
//                      registers, the CTA merges them).  Ties go to the lower anchor index (the reference's torch.topk
//                      leaves them unspecified; oracle/ref_port.tal_assign_port uses the same rule).
//   tal_assign_kernel  one CTA per image: anchors claimed by several boxes go to the box with the highest overlap (over ALL
//                      boxes, like the reference), per-box maxima of metric and overlap over the final positives, then
//                      labels, boxes, foreground mask, box index of every anchor.
//   tal_scores_kernel  the normalised one-hot scores [B, A, C], the one big output, written by the whole GPU.
// Arithmetic: fp32, one rounding per reference op (no FMA contraction), libdevice atanf / powf / sqrtf like the ATen
// kernels the reference runs, so indices and values match the reference on the same GPU bit for bit.
// bf16 scores (the trainer under bf16 autocast) take tal_topk_bf16_kernel and tal_assign_bf16_kernel, built from the same
// source as the fp16 / fp32 kernels (tal_stages.cuh) with a bf16 load and no rounding of the power (see align_metric).
#include "../../include/cerb_post.h"
#include "cerb_common.cuh"

#define TAL_MAX_TOPK 16
#define TAL_THREADS_A 256
#define TAL_THREADS_B 512
#define TAL_MAX_GT 1024

struct TalParams {
    const void* scores;      // [B, A, C] fp32 | fp16 | bf16 (sigmoid scores)
    const float* pd;         // [B, A, 4] xyxy, pixels
    const float* anc;        // [A, 2] anchor centres, pixels
    const float* gt_labels;  // [B, G]
    const float* gt_boxes;   // [B, G, 4]
    const float* mask_gt;    // [B, G]
    int B, A, C, G, topk, score_half;
    float alpha, beta, eps;
    int* topk_idx;           // workspace [B, G, topk]
    int* cnt;                // workspace [B, A]: boxes claiming the anchor
    int* gsel;               // workspace [B, A]: the box the anchor ends up with
    float* aval;             // workspace [B, A]: metric of (that box, anchor)
    float* pos;              // workspace [B, G, 2]: per-box maxima of metric and overlap over its final positives
    long long* target_labels;   // [B, A]
    float* target_bboxes;       // [B, A, 4]
    float* target_scores;       // [B, A, C]
    unsigned char* fg_mask;     // [B, A] bool
    long long* target_gt_idx;   // [B, A]
};

// torch.pow(tensor, python scalar) on CUDA (ATen PowKernel.cu): a few exponents are special-cased, the rest is powf
__device__ __forceinline__ float pow_like_torch(float x, float e) {
    if (e == 0.5f) return sqrtf(x);
    if (e == 1.f) return powf(x, 1.f);
    if (e == 2.f) return __fmul_rn(x, x);
    if (e == 3.f) return __fmul_rn(__fmul_rn(x, x), x);
    if (e == -0.5f) return rsqrtf(x);
    if (e == -1.f) return __fdiv_rn(1.f, x);
    if (e == -2.f) return __fdiv_rn(1.f, __fmul_rn(x, x));
    return powf(x, e);
}

// bbox_iou(box1 = ground truth, box2 = prediction, xywh=False, CIoU=True), then .clamp(0) (utils/tal.py:128)
__device__ __forceinline__ float ciou_clamped(const float4 g, const float4 p) {
    const float eps = 1e-7f;
    const float w1 = __fsub_rn(g.z, g.x), h1 = __fadd_rn(__fsub_rn(g.w, g.y), eps);
    const float w2 = __fsub_rn(p.z, p.x), h2 = __fadd_rn(__fsub_rn(p.w, p.y), eps);
    const float iw = fmaxf(__fsub_rn(fminf(g.z, p.z), fmaxf(g.x, p.x)), 0.f);
    const float ih = fmaxf(__fsub_rn(fminf(g.w, p.w), fmaxf(g.y, p.y)), 0.f);
    const float inter = __fmul_rn(iw, ih);
    const float uni = __fadd_rn(__fsub_rn(__fadd_rn(__fmul_rn(w1, h1), __fmul_rn(w2, h2)), inter), eps);
    const float iou = __fdiv_rn(inter, uni);
    const float cw = __fsub_rn(fmaxf(g.z, p.z), fminf(g.x, p.x));
    const float ch = __fsub_rn(fmaxf(g.w, p.w), fminf(g.y, p.y));
    const float c2 = __fadd_rn(__fadd_rn(__fmul_rn(cw, cw), __fmul_rn(ch, ch)), eps);
    const float dx = __fsub_rn(__fsub_rn(__fadd_rn(p.x, p.z), g.x), g.z);
    const float dy = __fsub_rn(__fsub_rn(__fadd_rn(p.y, p.w), g.y), g.w);
    const float rho2 = __fmul_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), 0.25f);  // "/ 4" = * (1 / 4) on CUDA, exact
    const float at = __fsub_rn(atanf(__fdiv_rn(w2, h2)), atanf(__fdiv_rn(w1, h1)));
    const float v = __fmul_rn((float)(4.0 / (3.141592653589793 * 3.141592653589793)), __fmul_rn(at, at));
    const float al = __fdiv_rn(v, __fadd_rn(__fsub_rn(v, iou), (float)(1.0 + 1e-7)));
    const float ciou = __fsub_rn(iou, __fadd_rn(__fdiv_rn(rho2, c2), __fmul_rn(v, al)));
    return fmaxf(ciou, 0.f);
}
__device__ __forceinline__ bool inside_gt(const float4 g, float ax, float ay, float eps) {
    const float m = fminf(fminf(__fsub_rn(ax, g.x), __fsub_rn(ay, g.y)), fminf(__fsub_rn(g.z, ax), __fsub_rn(g.w, ay)));
    return m > eps;
}
// BF16 = false: fp16 or fp32 scores as P.score_half says; true: bf16 scores (the *_bf16 kernels)
template <bool BF16> __device__ __forceinline__ float load_score(const TalParams& P, int b, int a, int c) {
    const size_t i = ((size_t)b * P.A + a) * P.C + c;
    if constexpr (BF16) return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(P.scores)[i]);
    return P.score_half ? __half2float(reinterpret_cast<const __half*>(P.scores)[i]) : reinterpret_cast<const float*>(P.scores)[i];
}
// align_metric of (box, anchor) BEFORE the inside mask: score^alpha * overlap^beta, with the reference's type promotion
// (half scores: the power is rounded to half, then multiplied in fp32).  bf16 scores come from bf16 autocast, whose fp32
// op list has pow: the power runs in fp32 on the widened score and is not rounded, so bf16 is the fp32 path after the load.
template <bool BF16> __device__ __forceinline__ float align_metric(const TalParams& P, float score, float ov) {
    float sp = pow_like_torch(score, P.alpha);
    if (!BF16 && P.score_half) sp = __half2float(__float2half_rn(sp));
    return __fmul_rn(sp, pow_like_torch(ov, P.beta));
}

#define TAL_BF16 false
#define TAL_KERNEL(stage) stage##_kernel
#include "tal_stages.cuh"
#undef TAL_BF16
#undef TAL_KERNEL
#define TAL_BF16 true
#define TAL_KERNEL(stage) stage##_bf16_kernel
#include "tal_stages.cuh"
#undef TAL_BF16
#undef TAL_KERNEL

// target_scores [B, A, C] = one_hot(label) * fg * norm (tal.py:174-177, :107-108): the one big output (43 MB at B=64,
// A=8400, C=20), written by the whole GPU with consecutive threads on consecutive elements
__global__ void __launch_bounds__(256) tal_scores_kernel(const __grid_constant__ TalParams P) {
    const size_t n = (size_t)P.B * P.A * P.C;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t o = i / P.C;  // (image, anchor)
        const int c = (int)(i - o * P.C);
        float v = 0.f;
        if (P.cnt[o] > 0) {
            const int b = (int)(o / P.A), g = P.gsel[o];
            if ((int)P.gt_labels[(size_t)b * P.G + g] == c) {
                const float* ps = P.pos + ((size_t)b * P.G + g) * 2;
                v = __fdiv_rn(__fmul_rn(P.aval[o], ps[1]), __fadd_rn(ps[0], P.eps));
            }
        }
        P.target_scores[i] = v;
    }
}

size_t cerb_tal_workspace_bytes_impl(int B, int A, int G, int topk) {
    return ((size_t)B * G * topk + (size_t)B * A * 3 + (size_t)B * G * 2) * 4;
}

extern "C" size_t cerb_tal_workspace_bytes(int B, int A, int G, int topk) { return cerb_tal_workspace_bytes_impl(B, A, G, topk); }

extern "C" int cerb_tal_assign(const void* pd_scores, const float* pd_bboxes, const float* anc_points, const float* gt_labels,
                               const float* gt_bboxes, const float* mask_gt, int B, int A, int C, int G, int topk, double alpha,
                               double beta, double eps, int score_dtype, long long* target_labels, float* target_bboxes,
                               float* target_scores, unsigned char* fg_mask, long long* target_gt_idx, void* workspace,
                               size_t workspace_bytes, void* stream) {
    cerb_clear_error();
    CERB_REQUIRE(pd_scores && pd_bboxes && anc_points && gt_labels && gt_bboxes && mask_gt && target_labels && target_bboxes &&
                     target_scores && fg_mask && target_gt_idx,
                 "cerb_tal_assign: null argument");
    CERB_REQUIRE(B >= 1 && A >= 1 && C >= 1, "cerb_tal_assign: empty problem (B=%d A=%d C=%d)", B, A, C);
    CERB_REQUIRE(G >= 1 && G <= TAL_MAX_GT, "cerb_tal_assign: G=%d outside [1, %d] (no boxes at all is the caller's early return, tal.py:89-93)", G, TAL_MAX_GT);
    CERB_REQUIRE(topk >= 1 && topk <= TAL_MAX_TOPK && topk <= A, "cerb_tal_assign: topk=%d outside [1, min(%d, A)]", topk, TAL_MAX_TOPK);
    CERB_REQUIRE(score_dtype == CERB_F16 || score_dtype == CERB_BF16 || score_dtype == CERB_F32,
                 "cerb_tal_assign: unsupported score dtype %d", score_dtype);
    CERB_REQUIRE(cerb_aligned(pd_bboxes, 16) && cerb_aligned(gt_bboxes, 16) && cerb_aligned(target_bboxes, 16) && cerb_aligned(anc_points, 8),
                 "cerb_tal_assign: box tensors must be 16-byte aligned, anchor points 8-byte aligned");
    const size_t need = cerb_tal_workspace_bytes_impl(B, A, G, topk);
    if (const int rc = cerb_require_workspace("cerb_tal_assign", workspace, workspace_bytes, need)) return rc;
    TalParams P;
    P.scores = pd_scores; P.pd = pd_bboxes; P.anc = anc_points; P.gt_labels = gt_labels; P.gt_boxes = gt_bboxes; P.mask_gt = mask_gt;
    P.B = B; P.A = A; P.C = C; P.G = G; P.topk = topk; P.score_half = score_dtype == CERB_F16;
    P.alpha = (float)alpha; P.beta = (float)beta; P.eps = (float)eps;
    int* ws = (int*)workspace;
    P.topk_idx = ws; ws += (size_t)B * G * topk;
    P.cnt = ws; ws += (size_t)B * A;
    P.gsel = ws; ws += (size_t)B * A;
    P.aval = (float*)ws; ws += (size_t)B * A;
    P.pos = (float*)ws;
    P.target_labels = target_labels; P.target_bboxes = target_bboxes; P.target_scores = target_scores; P.fg_mask = fg_mask;
    P.target_gt_idx = target_gt_idx;
    if (score_dtype == CERB_BF16) {
        tal_topk_bf16_kernel<<<B * G, TAL_THREADS_A, 0, (cudaStream_t)stream>>>(P);
        tal_assign_bf16_kernel<<<B, TAL_THREADS_B, 0, (cudaStream_t)stream>>>(P);
    } else {
        tal_topk_kernel<<<B * G, TAL_THREADS_A, 0, (cudaStream_t)stream>>>(P);
        tal_assign_kernel<<<B, TAL_THREADS_B, 0, (cudaStream_t)stream>>>(P);
    }
    const size_t n_out = (size_t)B * A * C;
    const int blocks = (int)((n_out + 255) / 256 < 148 * 16 ? (n_out + 255) / 256 : 148 * 16);
    tal_scores_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(P);
    return cerb_launch_status("cerb_tal_assign", cudaGetLastError());
}
