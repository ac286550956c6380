// Letterbox preprocessing (SURVEY row 10): the inference front end of CerberusPreprocessor.preprocess
// (cerberusdet/cerberusdet_preprocessor.py:42-74) for a batch of images of any sizes in one launch --
//     letterbox (data/augmentations.py:59-90): cv2.resize(INTER_LINEAR) to unpad_w x unpad_h, copyMakeBorder(114)
//     [:, :, ::-1].transpose(2, 0, 1): BGR -> RGB, HWC -> CHW
//     np.stack, upload, / 255
// Input: uint8 HWC BGR rows (any pitch).  Output: one [B, 3, out_h, out_w] fp16 | fp32 tensor.
//
// The resize is cv2's uint8 arithmetic (imgproc/src/resize.cpp), not a float bilinear, so the pixels equal cv2's bit for
// bit (tests/letterbox_port.py restates it in numpy):
//   coefficients   scale = 1 / (dst / src) (double); f = (float)((d + 0.5) * scale - 0.5), s = floor(f), f -= s;
//                  weights rint((1 - f) * 2048), rint(f * 2048).  Columns clamp s and zero f at both borders, rows keep
//                  the weights and clamp the two source rows.
//   horizontal     exact int: S[s] * a0 + S[s + 1] * a1
//   vertical       cv2's fixed-point rounding ((((r0 >> 4) * b0) >> 16) + (((r1 >> 4) * b1) >> 16) + 2) >> 2
//   exact 2x       cv2 switches to INTER_AREA: (a + b + c + d + 2) >> 2
//   same size      a copy (letterbox skips cv2.resize)
// The double and float steps use __d*_rn / __f*_rn intrinsics: no FMA contraction changes a coefficient.  The / 255 is
// what ATen does for a CUDA tensor divided by a Python scalar: a multiply by the fp32 reciprocal, rounded to the dtype.
//
// Memory-bound.  One thread owns one output column (its horizontal coefficients are computed once) and walks
// LB_ROWS / LB_TY rows; a warp writes 32 consecutive values of each RGB plane.  The source bytes a warp gathers for a
// row span a few 128-byte lines and come through L1.
#include "cerb_kernels.h"

#define LB_TX 128   // output columns per CTA, one per thread
#define LB_TY 2     // rows handled at once by a CTA
#define LB_ROWS 16  // output rows per CTA

// cv2's source index pair and 11-bit weights of output index d along an axis of n source pixels (scale = n / dst)
struct LbTap {
    int s0, s1, w0, w1;
};
__device__ __forceinline__ LbTap lb_tap(int d, double scale, int n, bool column) {
    const float f = __double2float_rn(__dsub_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), 0.5));
    int s = (int)floorf(f);
    float fr = __fsub_rn(f, (float)s);
    LbTap t;
    if (column) {  // xofs / alpha clamping of resizeGeneric: fx = 0 outside [0, n - 1)
        if (s < 0) { s = 0; fr = 0.f; }
        if (s >= n - 1) { s = n - 1; fr = 0.f; }
        t.s0 = s;
        t.s1 = min(s + 1, n - 1);
    } else {  // rows: the weights stay, the rows are clipped to the image
        t.s0 = min(max(s, 0), n - 1);
        t.s1 = min(max(s + 1, 0), n - 1);
    }
    t.w0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, fr), 2048.f));
    t.w1 = __float2int_rn(__fmul_rn(fr, 2048.f));
    return t;
}

template <typename T> __device__ __forceinline__ T lb_norm(int v);
// 0x3b808081 = fp32(1 / 255): x / 255.0 on a CUDA tensor is x * (1.f / 255.f) in fp32 (ATen's div_true_kernel_cuda)
template <> __device__ __forceinline__ float lb_norm<float>(int v) { return __fmul_rn((float)v, __int_as_float(0x3b808081)); }
template <> __device__ __forceinline__ __half lb_norm<__half>(int v) { return __float2half_rn(lb_norm<float>(v)); }

template <typename T>
__global__ void __launch_bounds__(LB_TX * LB_TY) letterbox_kernel(const __grid_constant__ LetterboxParams P) {
    const LbImage& im = P.img[blockIdx.z];
    const int x = blockIdx.x * LB_TX + threadIdx.x;
    if (x >= P.out_w) return;
    const size_t plane = (size_t)P.out_h * P.out_w;
    T* out = (T*)P.out + (size_t)blockIdx.z * 3 * plane + x;
    const unsigned char* __restrict__ src = im.src;
    // 0 = same size (copy), 1 = exact 2x in both axes (INTER_AREA), 2 = INTER_LINEAR
    const int mode = (im.uw == im.w && im.uh == im.h) ? 0 : (im.w == 2 * im.uw && im.h == 2 * im.uh) ? 1 : 2;
    const int dx = x - im.left;
    const bool xin = dx >= 0 && dx < im.uw;
    int xo0 = 0, xo1 = 0, a0 = 0, a1 = 0;  // byte offsets of the two source columns, their weights
    double scale_y = 0.0;
    if (xin) {
        if (mode == 0) {
            xo0 = dx * 3;
        } else if (mode == 1) {
            xo0 = dx * 6;
            xo1 = xo0 + 3;
        } else {
            const LbTap t = lb_tap(dx, __ddiv_rn(1.0, __ddiv_rn((double)im.uw, (double)im.w)), im.w, true);
            xo0 = t.s0 * 3;
            xo1 = t.s1 * 3;
            a0 = t.w0;
            a1 = t.w1;
            scale_y = __ddiv_rn(1.0, __ddiv_rn((double)im.uh, (double)im.h));
        }
    }
    const int y_end = min((int)(blockIdx.y + 1) * LB_ROWS, P.out_h);
    for (int y = blockIdx.y * LB_ROWS + threadIdx.y; y < y_end; y += LB_TY) {
        const int dy = y - im.top;
        int bgr[3] = {114, 114, 114};
        if (xin && dy >= 0 && dy < im.uh) {
            if (mode == 0) {
                const unsigned char* r = src + (long long)dy * im.pitch + xo0;
#pragma unroll
                for (int c = 0; c < 3; ++c) bgr[c] = __ldg(r + c);
            } else if (mode == 1) {
                const unsigned char* r0 = src + (long long)(2 * dy) * im.pitch;
                const unsigned char* r1 = r0 + im.pitch;
#pragma unroll
                for (int c = 0; c < 3; ++c)
                    bgr[c] = (__ldg(r0 + xo0 + c) + __ldg(r0 + xo1 + c) + __ldg(r1 + xo0 + c) + __ldg(r1 + xo1 + c) + 2) >> 2;
            } else {
                const LbTap t = lb_tap(dy, scale_y, im.h, false);
                const unsigned char* r0 = src + (long long)t.s0 * im.pitch;
                const unsigned char* r1 = src + (long long)t.s1 * im.pitch;
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const int h0 = __ldg(r0 + xo0 + c) * a0 + __ldg(r0 + xo1 + c) * a1;
                    const int h1 = __ldg(r1 + xo0 + c) * a0 + __ldg(r1 + xo1 + c) * a1;
                    const int v = ((((h0 >> 4) * t.w0) >> 16) + (((h1 >> 4) * t.w1) >> 16) + 2) >> 2;
                    bgr[c] = min(max(v, 0), 255);
                }
            }
        }
        T* o = out + (size_t)y * P.out_w;
        o[0] = lb_norm<T>(bgr[2]);  // R
        o[plane] = lb_norm<T>(bgr[1]);
        o[2 * plane] = lb_norm<T>(bgr[0]);
    }
}

cudaError_t cerb_launch_letterbox(const LetterboxParams& P, int n_images, int dtype, cudaStream_t stream) {
    const dim3 grid((P.out_w + LB_TX - 1) / LB_TX, (P.out_h + LB_ROWS - 1) / LB_ROWS, n_images);
    const dim3 block(LB_TX, LB_TY);
    if (dtype == CERB_DTYPE_F16) letterbox_kernel<__half><<<grid, block, 0, stream>>>(P);
    else letterbox_kernel<float><<<grid, block, 0, stream>>>(P);
    return cudaGetLastError();
}
