// Training-time sibling of the Detect decode (SURVEY 8f row 4): Loss.bbox_decode, forward and backward.
//
// Reference: cerberusdet/utils/loss.py:126-131
//     pred_dist.view(b, a, 4, 16).softmax(3).matmul(proj)          proj = arange(16)
//     dist2bbox(pred_dist, anchor_points, xywh=False)              utils/tal.py:196-205 -> (x1, y1, x2, y2), grid units
// The layout differs from the inference path: pred_dist is [B, A, 64], the 16 bins of a side are contiguous
// (loss.py:139-146 permutes the raw heads), so a thread owns one (anchor, side): 16 contiguous values in
// (1 or 2 256-bit loads, a warp reads 1 KB contiguous per instruction), one value out.  Same rounding points as the
// inference kernel for half tensors (dfl_expectation<T>): probabilities rounded to half, fp32 accumulation
// rounded once, the corner rounded once.  bfloat16 tensors round at the same points, in bf16.
//
// Backward (the autograd of the three reference ops, fused): with p = softmax(x), d = sum_k k p_k and g the
// incoming gradient of this side's corner (negated for the l, t sides: x1y1 = anchor - lt),
//     matmul backward   gp_k = g * k                  (rounded to the tensor dtype, as the reference's tensor is)
//     softmax backward  gx_j = p_j * (gp_j - sum_k gp_k p_k)
// p is recomputed from x instead of being saved by the forward (64 B re-read instead of 32 B saved + 32 B read).
#include "train_common.cuh"

#define TD_THREADS 256

// softmax probabilities (rounded like the reference's softmax output) and the expectation before its rounding
template <typename T> __device__ __forceinline__ void softmax16(const Row16<T>& r, float (&p)[CERB_REG_MAX]) {
    float m = r.get(0);
#pragma unroll
    for (int k = 1; k < CERB_REG_MAX; ++k) m = fmaxf(m, r.get(k));
    const float mb = m * CERB_LOG2E;
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < CERB_REG_MAX; ++k) {
        p[k] = fast_ex2(fmaf(r.get(k), CERB_LOG2E, -mb));
        s += p[k];
    }
    const float inv = fast_rcp(s);
#pragma unroll
    for (int k = 0; k < CERB_REG_MAX; ++k) p[k] = rnd<T>(p[k] * inv);
}

template <typename T, bool ALIGNED>
__global__ void __launch_bounds__(TD_THREADS) bbox_decode_fwd_kernel(const T* __restrict__ pred, const T* __restrict__ anchor_points,
                                                                      long n_sides, int A, T* __restrict__ out) {
    const long idx = (long)blockIdx.x * TD_THREADS + threadIdx.x;  // (row = b * A + a, side)
    if (idx >= n_sides) return;
    Row16<T> r;
    load_row<T, ALIGNED>(pred + idx * CERB_REG_MAX, r);
    float x[CERB_REG_MAX];
#pragma unroll
    for (int k = 0; k < CERB_REG_MAX; ++k) x[k] = r.get(k);
    const float d = dfl_expectation<T>(x);  // rounded to T
    const int side = (int)(idx & 3);
    const int a = (int)((idx >> 2) % A);
    const float ap = to_f32<T>(anchor_points[a * 2 + (side & 1)]);
    out[idx] = from_f32<T>(side < 2 ? ap - d : ap + d);  // x1y1 = a - lt, x2y2 = a + rb (tal.py:198-200)
}

template <typename T, bool ALIGNED>
__global__ void __launch_bounds__(TD_THREADS) bbox_decode_bwd_kernel(const T* __restrict__ pred, const T* __restrict__ grad_out,
                                                                      long n_sides, T* __restrict__ grad_in) {
    const long idx = (long)blockIdx.x * TD_THREADS + threadIdx.x;
    if (idx >= n_sides) return;
    Row16<T> r;
    load_row<T, ALIGNED>(pred + idx * CERB_REG_MAX, r);
    float p[CERB_REG_MAX];
    softmax16<T>(r, p);
    const int side = (int)(idx & 3);
    const float go = to_f32<T>(grad_out[idx]);
    const float g = side < 2 ? -go : go;
    float gp[CERB_REG_MAX];
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int k = 0; k < CERB_REG_MAX; k += 2) {
        gp[k] = rnd<T>(g * (float)k);
        gp[k + 1] = rnd<T>(g * (float)(k + 1));
        s0 = fmaf(gp[k], p[k], s0);
        s1 = fmaf(gp[k + 1], p[k + 1], s1);
    }
    const float s = s0 + s1;
#pragma unroll
    for (int k = 0; k < CERB_REG_MAX; ++k) r.set(k, p[k] * (gp[k] - s));
    store_row<T, ALIGNED>(grad_in + idx * CERB_REG_MAX, r);
}

static bool td_aligned(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 31) == 0; }

cudaError_t cerb_launch_bbox_decode_fwd(const void* pred, const void* anchor_points, long n_rows, int A, int dtype, void* out,
                                        cudaStream_t stream) {
    const long n_sides = n_rows * 4;
    if (n_sides == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)((n_sides + TD_THREADS - 1) / TD_THREADS);
    const bool al = td_aligned(pred);
    if (dtype == CERB_DTYPE_BF16) {
        if (al) bbox_decode_fwd_kernel<__nv_bfloat16, true><<<blocks, TD_THREADS, 0, stream>>>((const __nv_bfloat16*)pred, (const __nv_bfloat16*)anchor_points, n_sides, A, (__nv_bfloat16*)out);
        else bbox_decode_fwd_kernel<__nv_bfloat16, false><<<blocks, TD_THREADS, 0, stream>>>((const __nv_bfloat16*)pred, (const __nv_bfloat16*)anchor_points, n_sides, A, (__nv_bfloat16*)out);
    } else if (dtype == CERB_DTYPE_F16) {
        if (al) bbox_decode_fwd_kernel<__half, true><<<blocks, TD_THREADS, 0, stream>>>((const __half*)pred, (const __half*)anchor_points, n_sides, A, (__half*)out);
        else bbox_decode_fwd_kernel<__half, false><<<blocks, TD_THREADS, 0, stream>>>((const __half*)pred, (const __half*)anchor_points, n_sides, A, (__half*)out);
    } else {
        if (al) bbox_decode_fwd_kernel<float, true><<<blocks, TD_THREADS, 0, stream>>>((const float*)pred, (const float*)anchor_points, n_sides, A, (float*)out);
        else bbox_decode_fwd_kernel<float, false><<<blocks, TD_THREADS, 0, stream>>>((const float*)pred, (const float*)anchor_points, n_sides, A, (float*)out);
    }
    return cudaGetLastError();
}

cudaError_t cerb_launch_bbox_decode_bwd(const void* pred, const void* grad_out, long n_rows, int dtype, void* grad_in,
                                        cudaStream_t stream) {
    const long n_sides = n_rows * 4;
    if (n_sides == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)((n_sides + TD_THREADS - 1) / TD_THREADS);
    const bool al = td_aligned(pred) && td_aligned(grad_in);
    if (dtype == CERB_DTYPE_BF16) {
        if (al) bbox_decode_bwd_kernel<__nv_bfloat16, true><<<blocks, TD_THREADS, 0, stream>>>((const __nv_bfloat16*)pred, (const __nv_bfloat16*)grad_out, n_sides, (__nv_bfloat16*)grad_in);
        else bbox_decode_bwd_kernel<__nv_bfloat16, false><<<blocks, TD_THREADS, 0, stream>>>((const __nv_bfloat16*)pred, (const __nv_bfloat16*)grad_out, n_sides, (__nv_bfloat16*)grad_in);
    } else if (dtype == CERB_DTYPE_F16) {
        if (al) bbox_decode_bwd_kernel<__half, true><<<blocks, TD_THREADS, 0, stream>>>((const __half*)pred, (const __half*)grad_out, n_sides, (__half*)grad_in);
        else bbox_decode_bwd_kernel<__half, false><<<blocks, TD_THREADS, 0, stream>>>((const __half*)pred, (const __half*)grad_out, n_sides, (__half*)grad_in);
    } else {
        if (al) bbox_decode_bwd_kernel<float, true><<<blocks, TD_THREADS, 0, stream>>>((const float*)pred, (const float*)grad_out, n_sides, (float*)grad_in);
        else bbox_decode_bwd_kernel<float, false><<<blocks, TD_THREADS, 0, stream>>>((const float*)pred, (const float*)grad_out, n_sides, (float*)grad_in);
    }
    return cudaGetLastError();
}
