// The box-regression term of the training loss (SURVEY 8f row 4, the step after the assigner): BboxLoss.forward
// (reference cerberusdet/utils/loss.py:12-44) = CIoU loss + distribution focal loss over the foreground anchors, with
// bbox2dist (utils/tal.py:208-211) and bbox_iou(xywh=False, CIoU=True) (utils/metrics.py:373-408), reg_max 16 bins.
//
//   bbox_loss_fwd_kernel  one launch, both scalars.  Work unit (anchor, side) as in train_decode.cu.  A background
//                         anchor reads its fg_mask byte and nothing else; a positive one reads its 16 bins per side, its
//                         two boxes and its target-score row.  Per-CTA partial sums go to a workspace; the last CTA
//                         (ticket counter, reset by that CTA) adds them in CTA order and divides by target_scores_sum:
//                         the result does not depend on scheduling, and no host value is needed.
//   bbox_loss_bwd_kernel  recomputes everything from the inputs (nothing saved by the forward) and writes the dense
//                         grad_pred_dist [B, A, 64] (zeros at background anchors, 256-bit stores) and grad_pred_bboxes.
//
// Rounding follows the reference's ops: fp32, one rounding per op (no FMA contraction), libdevice atanf / expf / logf as
// in the ATen kernels.  The cross-entropy restates ATen's warp softmax for 16 classes (max, then exp(x - max) summed by a
// butterfly over 16 lanes, log_softmax = (x - max) - log(sum)).  Half mode is the trainer's fp16 autocast case
// (trainers/averaging.py:158): pred_dist, pred_bboxes and anchor_points are fp16, the targets fp32; type promotion then
// rounds w1, h1 (twice), w1 * h1, w1 / h1 and atan(w1 / h1) to half, everything that meets a target coordinate is fp32,
// and the cross-entropy's log_softmax keeps the half dtype (fp32 inside, output rounded to half) before nll_loss reads it
// in fp32 -- what autocast does with F.cross_entropy on half logits, measured against the reference on the B200.
// The backward follows autograd's conventions: alpha = v / (v - iou + 1 + eps) is a constant (computed under no_grad), minimum / maximum split
// the gradient in half on exact ties, clamp(min=0) passes it at exactly 0, the gradient of a half intermediate is rounded
// to half where autograd keeps it as a half tensor, and the cross-entropy gradient is (softmax - onehot) in fp32.
#include "../../include/cerb_post.h"
#include "train_common.cuh"

#define BL_THREADS 256
#define BL_MAX_CTAS (148 * 8)  // forward grid cap (grid-stride): one partial pair per CTA in the workspace

struct BboxLossParams {
    const void* pred_dist;       // [B, A, 64] T
    const void* pred_bboxes;     // [B, A, 4] T, xyxy grid units
    const void* anchor_points;   // [A, 2] T
    const float* target_bboxes;  // [B, A, 4] xyxy grid units
    const float* target_scores;  // [B, A, C]
    const unsigned char* fg_mask;  // [B, A]
    const float* tss_dev;        // target_scores_sum on the device, or null: tss_host
    float tss_host;
    long n_rows;                 // B * A
    int A, C;
};

template <typename T> struct BoxT;
template <> struct BoxT<float> {
    static __device__ __forceinline__ float4 load(const void* p, long row) { return reinterpret_cast<const float4*>(p)[row]; }
};
template <> struct BoxT<__half> {
    static __device__ __forceinline__ float4 load(const void* p, long row) {
        const uint2 u = reinterpret_cast<const uint2*>(p)[row];
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
        const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
        return make_float4(a.x, a.y, b.x, b.y);
    }
};

// round to the pred dtype where the reference keeps a half tensor (identity in fp32 mode)
template <typename T> __device__ __forceinline__ float rh(float v) { return rnd<T>(v); }

// the four lanes of one anchor (lanes 4k .. 4k+3 of a warp): sum of the lanes' values, the same bits in every lane
__device__ __forceinline__ unsigned quad_mask() { return 0xFu << (threadIdx.x & 28); }
__device__ __forceinline__ float quad_sum(float v) {
    const unsigned m = quad_mask();
    v = __fadd_rn(v, __shfl_xor_sync(m, v, 1));
    return __fadd_rn(v, __shfl_xor_sync(m, v, 2));
}

// weight = target_scores.sum(-1) (loss.py:14): the row is one-hot times a norm, so any order gives the exact sum
__device__ __forceinline__ float score_weight(const BboxLossParams& P, long row, int side) {
    const float* s = P.target_scores + row * P.C;
    float acc = 0.f;
    for (int c = side; c < P.C; c += 4) acc = __fadd_rn(acc, s[c]);
    return quad_sum(acc);
}

// CIoU forward of box1 = prediction p, box2 = target t, with every intermediate the backward needs
struct Ciou {
    float w1, h1, w2, h2, ix, iy, cix, ciy, inter, w1h1, uni, iou, cw, ch, c2, dx, dy, rho2, r1, at, v, alpha, ciou;
};
template <typename T> __device__ __forceinline__ Ciou ciou_fwd(const float4 p, const float4 t) {
    const float eps = 1e-7f;
    Ciou c;
    c.w1 = rh<T>(__fsub_rn(p.z, p.x));
    c.h1 = rh<T>(__fadd_rn(rh<T>(__fsub_rn(p.w, p.y)), eps));
    c.w2 = __fsub_rn(t.z, t.x);
    c.h2 = __fadd_rn(__fsub_rn(t.w, t.y), eps);
    c.ix = __fsub_rn(fminf(p.z, t.z), fmaxf(p.x, t.x));
    c.iy = __fsub_rn(fminf(p.w, t.w), fmaxf(p.y, t.y));
    c.cix = fmaxf(c.ix, 0.f);
    c.ciy = fmaxf(c.iy, 0.f);
    c.inter = __fmul_rn(c.cix, c.ciy);
    c.w1h1 = rh<T>(__fmul_rn(c.w1, c.h1));
    c.uni = __fadd_rn(__fsub_rn(__fadd_rn(c.w1h1, __fmul_rn(c.w2, c.h2)), c.inter), eps);
    c.iou = __fdiv_rn(c.inter, c.uni);
    c.cw = __fsub_rn(fmaxf(p.z, t.z), fminf(p.x, t.x));
    c.ch = __fsub_rn(fmaxf(p.w, t.w), fminf(p.y, t.y));
    c.c2 = __fadd_rn(__fadd_rn(__fmul_rn(c.cw, c.cw), __fmul_rn(c.ch, c.ch)), eps);
    c.dx = __fsub_rn(__fsub_rn(__fadd_rn(t.x, t.z), p.x), p.z);  // b2_x1 + b2_x2 - b1_x1 - b1_x2
    c.dy = __fsub_rn(__fsub_rn(__fadd_rn(t.y, t.w), p.y), p.w);
    c.rho2 = __fmul_rn(__fadd_rn(__fmul_rn(c.dx, c.dx), __fmul_rn(c.dy, c.dy)), 0.25f);  // "/ 4": exact either way
    c.r1 = rh<T>(__fdiv_rn(c.w1, c.h1));
    c.at = __fsub_rn(atanf(__fdiv_rn(c.w2, c.h2)), rh<T>(atanf(c.r1)));
    c.v = __fmul_rn((float)(4.0 / (3.141592653589793 * 3.141592653589793)), __fmul_rn(c.at, c.at));
    c.alpha = __fdiv_rn(c.v, __fadd_rn(__fsub_rn(c.v, c.iou), (float)(1.0 + 1e-7)));
    c.ciou = __fsub_rn(c.iou, __fadd_rn(__fdiv_rn(c.rho2, c.c2), __fmul_rn(c.v, c.alpha)));
    return c;
}

// d(ciou)/d(box1) * G for box1 = (x1, y1, x2, y2), returned in that order
// autograd's split of minimum(a, b) / maximum(a, b) onto a: all of it, half of it on a tie, none
__device__ __forceinline__ float pick_min(float a, float b, float g) { return a < b ? g : (a == b ? __fmul_rn(g, 0.5f) : 0.f); }
__device__ __forceinline__ float pick_max(float a, float b, float g) { return a > b ? g : (a == b ? __fmul_rn(g, 0.5f) : 0.f); }

template <typename T> __device__ __forceinline__ float4 ciou_bwd(const Ciou& c, const float4 p, const float4 t, float G) {
    const float gS = -G;  // ciou = iou - (rho2 / c2 + v * alpha)
    // iou = inter / union;  union = ((w1h1 + w2h2) - inter) + eps
    const float g_union = __fmul_rn(-G, __fdiv_rn(c.iou, c.uni));
    const float g_inter = __fadd_rn(__fdiv_rn(G, c.uni), -g_union);
    const float g_ix = c.ix >= 0.f ? __fmul_rn(g_inter, c.ciy) : 0.f;  // clamp(min=0) passes the gradient at 0
    const float g_iy = c.iy >= 0.f ? __fmul_rn(g_inter, c.cix) : 0.f;
    // rho2 / c2
    const float g_rho2 = __fdiv_rn(gS, c.c2);
    const float g_c2 = __fmul_rn(-gS, __fdiv_rn(__fdiv_rn(c.rho2, c.c2), c.c2));
    const float g_sq = __fmul_rn(g_rho2, 0.25f);
    const float g_dx = __fmul_rn(g_sq, 2.f * c.dx), g_dy = __fmul_rn(g_sq, 2.f * c.dy);
    const float g_cw = __fmul_rn(g_c2, 2.f * c.cw), g_ch = __fmul_rn(g_c2, 2.f * c.ch);
    // v = K * (atan(w2 / h2) - atan(w1 / h1))^2, alpha constant; the w1 / h1 branch is half in the autocast case
    const float g_v = __fmul_rn(gS, c.alpha);
    const float g_at = __fmul_rn(__fmul_rn(g_v, (float)(4.0 / (3.141592653589793 * 3.141592653589793))), 2.f * c.at);
    const float g_a1 = rh<T>(-g_at);
    const float g_r1 = rh<T>(__fdiv_rn(g_a1, rh<T>(__fadd_rn(rh<T>(__fmul_rn(c.r1, c.r1)), 1.f))));
    const float g_u = rh<T>(g_union);  // the gradient reaching the (half) product w1 * h1
    const float g_w1 = rh<T>(__fadd_rn(rh<T>(__fmul_rn(g_u, c.h1)), rh<T>(__fdiv_rn(g_r1, c.h1))));
    const float g_h1 = rh<T>(__fadd_rn(rh<T>(__fmul_rn(g_u, c.w1)), rh<T>(__fmul_rn(-g_r1, rh<T>(__fdiv_rn(c.r1, c.h1))))));
    // each coordinate: w1 / h1, the intersection's min / max, the enclosing box's min / max, the centre distance
    float4 g;
    g.x = __fadd_rn(__fadd_rn(__fadd_rn(-g_w1, rh<T>(pick_max(p.x, t.x, -g_ix))), rh<T>(pick_min(p.x, t.x, -g_cw))), rh<T>(-g_dx));
    g.y = __fadd_rn(__fadd_rn(__fadd_rn(-g_h1, rh<T>(pick_max(p.y, t.y, -g_iy))), rh<T>(pick_min(p.y, t.y, -g_ch))), rh<T>(-g_dy));
    g.z = __fadd_rn(__fadd_rn(__fadd_rn(g_w1, rh<T>(pick_min(p.z, t.z, g_ix))), rh<T>(pick_max(p.z, t.z, g_cw))), rh<T>(-g_dx));
    g.w = __fadd_rn(__fadd_rn(__fadd_rn(g_h1, rh<T>(pick_min(p.w, t.w, g_iy))), rh<T>(pick_max(p.w, t.w, g_ch))), rh<T>(-g_dy));
    return g;
}

// bbox2dist (tal.py:208-211) for one side: (anchor - x1y1, x2y2 - anchor).clamp(0, reg_max - 0.01), reg_max = 15
__device__ __forceinline__ float dfl_target(float4 t, float ax, float ay, int side) {
    const float d = side == 0 ? __fsub_rn(ax, t.x) : side == 1 ? __fsub_rn(ay, t.y) : side == 2 ? __fsub_rn(t.z, ax) : __fsub_rn(t.w, ay);
    return fminf(fmaxf(d, 0.f), 14.99f);
}

// log_softmax of the 16 bins as ATen's warp softmax computes it: (x - max) - log(sum exp(x - max)), the sum a butterfly,
// the output in the tensor dtype
template <typename T> __device__ __forceinline__ void log_softmax16(const Row16<T>& r, float (&ls)[CERB_REG_MAX]) {
    float m = r.get(0);
#pragma unroll
    for (int k = 1; k < CERB_REG_MAX; ++k) m = fmaxf(m, r.get(k));
    float e[CERB_REG_MAX];
#pragma unroll
    for (int k = 0; k < CERB_REG_MAX; ++k) {
        ls[k] = __fsub_rn(r.get(k), m);
        e[k] = expf(ls[k]);
    }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1)
#pragma unroll
        for (int k = 0; k < o; ++k) e[k] = __fadd_rn(e[k], e[k + o]);
    const float lse = logf(e[0]);
#pragma unroll
    for (int k = 0; k < CERB_REG_MAX; ++k) ls[k] = rh<T>(__fsub_rn(ls[k], lse));
}

// the per-anchor quantities both kernels need, for a positive anchor
struct Pos {
    float4 p, t;
    float w, target;
};
template <typename T> __device__ __forceinline__ Pos load_pos(const BboxLossParams& P, long row, int side) {
    Pos q;
    q.p = BoxT<T>::load(P.pred_bboxes, row);
    q.t = reinterpret_cast<const float4*>(P.target_bboxes)[row];
    const int a = (int)(row % P.A);
    const T* ap = reinterpret_cast<const T*>(P.anchor_points) + 2 * (long)a;
    q.target = dfl_target(q.t, to_f32<T>(ap[0]), to_f32<T>(ap[1]), side);
    q.w = score_weight(P, row, side);
    return q;
}

__device__ __forceinline__ float tss_of(const BboxLossParams& P) { return P.tss_dev ? *P.tss_dev : P.tss_host; }

// deterministic sum of one value per thread over the CTA (fixed shuffle tree, warps in order); valid in thread 0
__device__ __forceinline__ float2 block_sum2(float2 v, float2* sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        v.x = __fadd_rn(v.x, __shfl_down_sync(0xffffffffu, v.x, o));
        v.y = __fadd_rn(v.y, __shfl_down_sync(0xffffffffu, v.y, o));
    }
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    float2 s = make_float2(0.f, 0.f);
    if (threadIdx.x == 0)
        for (int w = 0; w < BL_THREADS / 32; ++w) s = make_float2(__fadd_rn(s.x, sh[w].x), __fadd_rn(s.y, sh[w].y));
    return s;
}

template <typename T>
__global__ void __launch_bounds__(BL_THREADS) bbox_loss_fwd_kernel(const __grid_constant__ BboxLossParams P, float* __restrict__ loss_iou,
                                                                    float* __restrict__ loss_dfl, float* __restrict__ per_anchor,
                                                                    float2* __restrict__ partials, unsigned* __restrict__ ticket) {
    __shared__ float2 sh[BL_THREADS / 32];
    __shared__ bool last;
    const long n_sides = P.n_rows * 4;
    const long stride = (long)gridDim.x * BL_THREADS;  // a multiple of 4: the four lanes of an anchor stay together
    float2 acc = make_float2(0.f, 0.f);
    for (long idx = (long)blockIdx.x * BL_THREADS + threadIdx.x; idx < n_sides; idx += stride) {
        const long row = idx >> 2;
        const int side = (int)(idx & 3);
        float t_iou = 0.f, t_dfl = 0.f;
        if (P.fg_mask[row]) {  // the four lanes of the anchor take this branch together
            const Pos q = load_pos<T>(P, row, side);
            Row16<T> r;
            load_row<T, true>(reinterpret_cast<const T*>(P.pred_dist) + idx * CERB_REG_MAX, r);
            float ls[CERB_REG_MAX];
            log_softmax16<T>(r, ls);
            const int tl = (int)q.target;  // target.long(); target >= 0
            const float wl = __fsub_rn((float)(tl + 1), q.target), wr = __fsub_rn(1.f, wl);
            // F.cross_entropy(.., tl) * wl + F.cross_entropy(.., tr) * wr  (loss.py:39-44); selects, not a dynamic index,
            // keep ls[] in registers
            float cel = 0.f, cer = 0.f;
#pragma unroll
            for (int k = 0; k < CERB_REG_MAX; ++k) {
                cel = k == tl ? -ls[k] : cel;
                cer = k == tl + 1 ? -ls[k] : cer;
            }
            const float side_term = __fadd_rn(__fmul_rn(cel, wl), __fmul_rn(cer, wr));
            // .mean(-1) over the four sides, then * weight (loss.py:19)
            const unsigned m = quad_mask();
            const float s1 = __shfl_sync(m, side_term, 1, 4), s2 = __shfl_sync(m, side_term, 2, 4), s3 = __shfl_sync(m, side_term, 3, 4);
            const float s0 = __shfl_sync(m, side_term, 0, 4);
            const float mean = __fmul_rn(__fadd_rn(__fadd_rn(__fadd_rn(s0, s1), s2), s3), 0.25f);
            if (side == 0) {
                const Ciou c = ciou_fwd<T>(q.p, q.t);
                t_iou = __fmul_rn(__fsub_rn(1.f, c.ciou), q.w);  // (1.0 - iou) * weight (loss.py:16)
                t_dfl = __fmul_rn(mean, q.w);
            }
        }
        if (side == 0) {
            acc.x = __fadd_rn(acc.x, t_iou);
            acc.y = __fadd_rn(acc.y, t_dfl);
            if (per_anchor) reinterpret_cast<float2*>(per_anchor)[row] = make_float2(t_iou, t_dfl);
        }
    }
    const float2 s = block_sum2(acc, sh);
    if (threadIdx.x == 0) {
        partials[blockIdx.x] = s;
        __threadfence();
        last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    float2 tot = make_float2(0.f, 0.f);
    for (int i = threadIdx.x; i < (int)gridDim.x; i += BL_THREADS) {
        const float2 v = __ldcg(partials + i);
        tot.x = __fadd_rn(tot.x, v.x);
        tot.y = __fadd_rn(tot.y, v.y);
    }
    __syncthreads();  // (sh is reused)
    const float2 all = block_sum2(tot, sh);
    if (threadIdx.x == 0) {
        const float tss = tss_of(P);
        *loss_iou = __fdiv_rn(all.x, tss);  // .sum() / target_scores_sum (loss.py:17, :20)
        *loss_dfl = __fdiv_rn(all.y, tss);
        *ticket = 0u;  // ready for the next launch (CUDA-graph replays reuse the workspace)
    }
}

template <typename T>
__global__ void __launch_bounds__(BL_THREADS) bbox_loss_bwd_kernel(const __grid_constant__ BboxLossParams P, const float* __restrict__ grad_iou,
                                                                    const float* __restrict__ grad_dfl, T* __restrict__ grad_pred_dist,
                                                                    T* __restrict__ grad_pred_bboxes) {
    const long idx = (long)blockIdx.x * BL_THREADS + threadIdx.x;
    if (idx >= P.n_rows * 4) return;
    const long row = idx >> 2;
    const int side = (int)(idx & 3);
    Row16<T> r;
    if (!P.fg_mask[row]) {
#pragma unroll
        for (int i = 0; i < Row16<T>::NV; ++i) r.v[i] = U8x32{};
        store_row<T, true>(grad_pred_dist + idx * CERB_REG_MAX, r);
        grad_pred_bboxes[idx] = from_f32<T>(0.f);
        return;
    }
    const Pos q = load_pos<T>(P, row, side);
    const float tss = tss_of(P);
    // DFL: loss_dfl = sum(mean_sides(ce_l * wl + ce_r * wr) * weight) / tss
    {
        load_row<T, true>(reinterpret_cast<const T*>(P.pred_dist) + idx * CERB_REG_MAX, r);
        float ls[CERB_REG_MAX];
        log_softmax16<T>(r, ls);
        const int tl = (int)q.target;
        const float wl = __fsub_rn((float)(tl + 1), q.target), wr = __fsub_rn(1.f, wl);
        const float gq = __fmul_rn(__fmul_rn(__fdiv_rn(*grad_dfl, tss), q.w), 0.25f);  // sum, * weight, mean backward
        const float gl = __fmul_rn(gq, wl), gr = __fmul_rn(gq, wr);
        // nll_loss backward (-g at the target, in the log-probabilities' dtype), then log_softmax backward of each
        // cross-entropy: g_j = [j == t] * (-g) - exp(ls_j) * (-g); the two gradients add up in the tensor dtype
        const float gL = rh<T>(-gl), gR = rh<T>(-gr);
#pragma unroll
        for (int k = 0; k < CERB_REG_MAX; ++k) {
            const float p = expf(ls[k]);
            const float a = __fsub_rn(k == tl ? gL : 0.f, __fmul_rn(p, gL));
            const float b = __fsub_rn(k == tl + 1 ? gR : 0.f, __fmul_rn(p, gR));
            r.set(k, rh<T>(__fadd_rn(rh<T>(a), rh<T>(b))));
        }
        store_row<T, true>(grad_pred_dist + idx * CERB_REG_MAX, r);
    }
    // CIoU: loss_iou = sum((1 - ciou) * weight) / tss
    const Ciou c = ciou_fwd<T>(q.p, q.t);
    const float G = -__fmul_rn(__fdiv_rn(*grad_iou, tss), q.w);
    const float4 g = ciou_bwd<T>(c, q.p, q.t, G);
    grad_pred_bboxes[idx] = from_f32<T>(side == 0 ? g.x : side == 1 ? g.y : side == 2 ? g.z : g.w);
}

static unsigned fwd_ctas(long n_rows) {
    const long n = (n_rows * 4 + BL_THREADS - 1) / BL_THREADS;
    return (unsigned)(n < 1 ? 1 : (n > BL_MAX_CTAS ? BL_MAX_CTAS : n));
}

extern "C" size_t cerb_bbox_loss_workspace_bytes(int B, int A) {
    if (B < 0 || A < 0) return 0;
    return 16 + (size_t)fwd_ctas((long)B * A) * sizeof(float2);
}

#define BL_REQUIRE(cond, ...)            \
    do {                                 \
        if (!(cond)) {                   \
            cerb_set_error(__VA_ARGS__); \
            return CERB_EINVAL;          \
        }                                \
    } while (0)

static bool bl_aligned(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }

static int bl_params(const char* fn, const void* pred_dist, const void* pred_bboxes, const void* anchor_points,
                     const float* target_bboxes, const float* target_scores, const unsigned char* fg_mask,
                     const float* tss_dev, double tss_host, int B, int A, int C, int reg_max, int dtype, BboxLossParams& P) {
    cerb_set_error("%s", "");
    BL_REQUIRE(reg_max == CERB_REG_MAX, "%s: reg_max=%d bins, only %d is supported (loss.py:96, BboxLoss(m.reg_max - 1))", fn, reg_max, CERB_REG_MAX);
    BL_REQUIRE(dtype == CERB_F16 || dtype == CERB_F32, "%s: unsupported dtype %d", fn, dtype);
    BL_REQUIRE(B >= 0 && A >= 0 && C >= 1, "%s: bad sizes B=%d A=%d C=%d", fn, B, A, C);
    BL_REQUIRE((long long)B * A <= 0x7fffffffLL && (long long)B * A * C <= (1LL << 40), "%s: B*A overflows (B=%d A=%d C=%d)", fn, B, A, C);
    if ((long long)B * A > 0) {
        BL_REQUIRE(pred_dist && pred_bboxes && anchor_points && target_bboxes && target_scores && fg_mask, "%s: null argument", fn);
        const size_t e = dtype == CERB_F16 ? 2 : 4;
        BL_REQUIRE(bl_aligned(pred_dist, 32) && bl_aligned(pred_bboxes, 4 * e) && bl_aligned(anchor_points, e) &&
                       bl_aligned(target_bboxes, 16) && bl_aligned(target_scores, 4),
                   "%s: misaligned rows (pred_dist needs 32 bytes, box rows 4 elements)", fn);
    }
    P.pred_dist = pred_dist; P.pred_bboxes = pred_bboxes; P.anchor_points = anchor_points;
    P.target_bboxes = target_bboxes; P.target_scores = target_scores; P.fg_mask = fg_mask;
    P.tss_dev = tss_dev; P.tss_host = (float)tss_host;
    P.n_rows = (long)B * A; P.A = A; P.C = C;
    return 0;
}

extern "C" int cerb_bbox_loss_fwd(const void* pred_dist, const void* pred_bboxes, const void* anchor_points, const float* target_bboxes,
                                  const float* target_scores, const unsigned char* fg_mask, const float* target_scores_sum,
                                  double target_scores_sum_host, int B, int A, int C, int reg_max, int dtype, float* loss_iou,
                                  float* loss_dfl, float* per_anchor, void* workspace, size_t workspace_bytes, void* stream) {
    BboxLossParams P;
    const int rc = bl_params("cerb_bbox_loss_fwd", pred_dist, pred_bboxes, anchor_points, target_bboxes, target_scores, fg_mask,
                             target_scores_sum, target_scores_sum_host, B, A, C, reg_max, dtype, P);
    if (rc) return rc;
    BL_REQUIRE(loss_iou && loss_dfl, "cerb_bbox_loss_fwd: null argument");
    BL_REQUIRE(per_anchor == nullptr || bl_aligned(per_anchor, 8), "cerb_bbox_loss_fwd: per_anchor must be 8-byte aligned");
    const size_t need = cerb_bbox_loss_workspace_bytes(B, A);
    if (workspace == nullptr || workspace_bytes < need) {
        cerb_set_error("cerb_bbox_loss_fwd: workspace of %zu bytes required, got %zu", need, workspace_bytes);
        return CERB_ENOSPC;
    }
    BL_REQUIRE(bl_aligned(workspace, 16), "cerb_bbox_loss_fwd: workspace must be 16-byte aligned");
    unsigned* ticket = (unsigned*)workspace;
    float2* partials = (float2*)((char*)workspace + 16);
    const unsigned ctas = fwd_ctas(P.n_rows);
    if (dtype == CERB_F16)
        bbox_loss_fwd_kernel<__half><<<ctas, BL_THREADS, 0, (cudaStream_t)stream>>>(P, loss_iou, loss_dfl, per_anchor, partials, ticket);
    else
        bbox_loss_fwd_kernel<float><<<ctas, BL_THREADS, 0, (cudaStream_t)stream>>>(P, loss_iou, loss_dfl, per_anchor, partials, ticket);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        cerb_set_error("cerb_bbox_loss_fwd: launch failed: %s", cudaGetErrorString(e));
        return CERB_ECUDA;
    }
    return 0;
}

extern "C" int cerb_bbox_loss_bwd(const void* pred_dist, const void* pred_bboxes, const void* anchor_points, const float* target_bboxes,
                                  const float* target_scores, const unsigned char* fg_mask, const float* target_scores_sum,
                                  double target_scores_sum_host, int B, int A, int C, int reg_max, int dtype, const float* grad_iou,
                                  const float* grad_dfl, void* grad_pred_dist, void* grad_pred_bboxes, void* stream) {
    BboxLossParams P;
    const int rc = bl_params("cerb_bbox_loss_bwd", pred_dist, pred_bboxes, anchor_points, target_bboxes, target_scores, fg_mask,
                             target_scores_sum, target_scores_sum_host, B, A, C, reg_max, dtype, P);
    if (rc) return rc;
    if (P.n_rows == 0) return 0;
    BL_REQUIRE(grad_iou && grad_dfl && grad_pred_dist && grad_pred_bboxes, "cerb_bbox_loss_bwd: null argument");
    BL_REQUIRE(bl_aligned(grad_pred_dist, 32) && bl_aligned(grad_pred_bboxes, dtype == CERB_F16 ? 8 : 16),
               "cerb_bbox_loss_bwd: misaligned rows (grad_pred_dist needs 32 bytes, box rows 4 elements)");
    const unsigned blocks = (unsigned)((P.n_rows * 4 + BL_THREADS - 1) / BL_THREADS);
    if (dtype == CERB_F16)
        bbox_loss_bwd_kernel<__half><<<blocks, BL_THREADS, 0, (cudaStream_t)stream>>>(P, grad_iou, grad_dfl, (__half*)grad_pred_dist, (__half*)grad_pred_bboxes);
    else
        bbox_loss_bwd_kernel<float><<<blocks, BL_THREADS, 0, (cudaStream_t)stream>>>(P, grad_iou, grad_dfl, (float*)grad_pred_dist, (float*)grad_pred_bboxes);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        cerb_set_error("cerb_bbox_loss_bwd: launch failed: %s", cudaGetErrorString(e));
        return CERB_ECUDA;
    }
    return 0;
}
