// Helpers shared by the decode kernels (decode.cu, decode_pipe.cu): 128-bit packs, streaming accesses,
// the DFL side reduction.  sm_100a only.
#pragma once
#include "cerb_kernels.h"

#ifndef DEC_THREADS
#define DEC_THREADS 128
#endif
#ifndef DEC_MINB
#define DEC_MINB 5  // 96 registers -> 20 warps per SM: best of the measured variants (profiles/r01_decode.md)
#endif
#define CLS_CHUNK 32
#define LOG2E_F 1.4426950408889634f

template <int BYTES> struct RawOf;
template <> struct RawOf<16> { typedef uint4 type; };
template <> struct RawOf<8> { typedef uint2 type; };
template <> struct RawOf<4> { typedef uint32_t type; };
template <> struct RawOf<2> { typedef uint16_t type; };

template <typename T, int VEC> union Pack {
    typename RawOf<sizeof(T) * VEC>::type raw;
    T e[VEC];
};

template <typename T, int VEC> __device__ __forceinline__ Pack<T, VEC> load_pack(const T* p) {
    Pack<T, VEC> r;
    if constexpr (sizeof(T) * VEC == 16) {
        r.raw = ldg_stream16(p);
    } else {
        r.raw = __ldg(reinterpret_cast<const typename RawOf<sizeof(T) * VEC>::type*>(p));
    }
    return r;
}
template <typename T, int VEC> __device__ __forceinline__ void store_pack(T* p, const Pack<T, VEC>& v) {
    if constexpr (sizeof(T) * VEC == 16) {
        stg_stream16(p, v.raw);
    } else {
        *reinterpret_cast<typename RawOf<sizeof(T) * VEC>::type*>(p) = v.raw;
    }
}

// maximum of the VEC stored (already rounded) scores of one vector; scores are sigmoids, so no NaN unless the
// logit was NaN, which fmaxf / __hmax2 drop -- a NaN score is never a candidate either
template <typename T, int VEC> __device__ __forceinline__ T pack_max(const Pack<T, VEC>& v);
template <> __device__ __forceinline__ __half pack_max<__half, 8>(const Pack<__half, 8>& v) {
    const __half2* h = reinterpret_cast<const __half2*>(&v.raw);
    const __half2 m = __hmax2(__hmax2(h[0], h[1]), __hmax2(h[2], h[3]));
    return __hmax(__low2half(m), __high2half(m));
}
template <> __device__ __forceinline__ __nv_bfloat16 pack_max<__nv_bfloat16, 8>(const Pack<__nv_bfloat16, 8>& v) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v.raw);
    const __nv_bfloat162 m = __hmax2(__hmax2(h[0], h[1]), __hmax2(h[2], h[3]));
    return __hmax(__low2bfloat16(m), __high2bfloat16(m));
}
template <> __device__ __forceinline__ float pack_max<float, 4>(const Pack<float, 4>& v) {
    return fmaxf(fmaxf(v.e[0], v.e[1]), fmaxf(v.e[2], v.e[3]));
}
template <typename T, int VEC> __device__ __forceinline__ T pack_max(const Pack<T, VEC>& v) { return v.e[0]; }

// Expected DFL distances of one box side for VEC anchors: sum_k k * softmax(logits)_k (reference DFL.forward,
// models/yolo.py:57-59).  Rounding points follow the reference for half tensors: probabilities are rounded to
// half (softmax output), the 1x1 conv accumulates in fp32 and rounds once; bfloat16 tensors likewise in bf16.
// DVec holds the VEC rounded distances: as floats, or -- 16-bit tensors, even VEC -- as packed half2 / bfloat162 pairs
// (anchors i, i+1), so that the rounding of two anchors is ONE F2FP.PACK_AB and the box arithmetic after it runs on pairs.
#ifndef CERB_HALF2_EPILOGUE
#define CERB_HALF2_EPILOGUE 1
#endif
template <typename T, int VEC> struct DVecTraits {
    static constexpr bool packed = CERB_HALF2_EPILOGUE && sizeof(T) == 2 && (VEC % 2) == 0;
};
template <typename T, int VEC, bool PACKED = DVecTraits<T, VEC>::packed> struct DVec { float f[VEC]; };
template <typename T, int VEC> struct DVec<T, VEC, true> { uint32_t h2[VEC / 2]; };

template <typename T, int VEC>
__device__ __forceinline__ void dfl_load(const T* __restrict__ side_base, int hw, Pack<T, VEC> (&v)[CERB_REG_MAX]) {
#pragma unroll
    for (int k = 0; k < CERB_REG_MAX; ++k) v[k] = load_pack<T, VEC>(side_base + (size_t)k * hw);
}
template <typename T, int VEC>
__device__ __forceinline__ void dfl_reduce(const Pack<T, VEC> (&v)[CERB_REG_MAX], DVec<T, VEC>& d) {
    if constexpr (DVecTraits<T, VEC>::packed) {
#pragma unroll
        for (int i = 0; i < VEC; i += 2) {
            float x0[CERB_REG_MAX], x1[CERB_REG_MAX];
#pragma unroll
            for (int k = 0; k < CERB_REG_MAX; ++k) {
                x0[k] = to_f32<T>(v[k].e[i]);
                x1[k] = to_f32<T>(v[k].e[i + 1]);
            }
            const float e0 = dfl_expectation_acc<T>(x0);
            const float e1 = dfl_expectation_acc<T>(x1);
            d.h2[i / 2] = Pair<T>::pack2_rn(e0, e1);
        }
    } else {
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            float x[CERB_REG_MAX];
#pragma unroll
            for (int k = 0; k < CERB_REG_MAX; ++k) x[k] = to_f32<T>(v[k].e[i]);
            d.f[i] = dfl_expectation<T>(x);
        }
    }
}
template <typename T, int VEC>
__device__ __forceinline__ void dfl_side(const T* __restrict__ side_base, int hw, DVec<T, VEC>& d) {
    Pack<T, VEC> v[CERB_REG_MAX];
    dfl_load<T, VEC>(side_base, hw, v);
    dfl_reduce<T, VEC>(v, d);
}

// dist2bbox(xywh) on ONE axis for VEC consecutive anchors starting at anchor a0 of a level of width W
// (reference utils/tal.py:198-204), then * stride (models/yolo.py:98):
//     ac = arange(dtype) + 0.5 (tal.py:188-189);  p1 = ac - dlo;  p2 = ac + dhi;  centre = (p1 + p2) / 2;  size = p2 - p1
// every operation rounded in the tensor dtype.  For half tensors the whole chain runs on half2 pairs: an IEEE half
// add/sub/mul IS "compute exactly, round once to half", and the operands here (|value| < 2^16, products by powers of
// two or of two halves) never differ from the reference's "fp32 operation, then round to half" except on a tie that
// only appears after the fp32 rounding -- which needs an operand below 2^-13 of the other AND an exact midpoint.
// bfloat16 tensors run the same chain on bfloat162 pairs, with no exception: fp32 carries 24 >= 2 * 8 + 2 significant
// bits, so rounding the fp32 result of an add/sub/mul to bf16 always equals the single rounding of the exact result.
// The anchor centres round too: bf16(k) + 0.5 is exact only below 128 (128.5 -> 128, 129.5 -> 130), as in the reference.
template <typename T, int VEC>
__device__ __forceinline__ void axis_boxes(const DVec<T, VEC>& dlo, const DVec<T, VEC>& dhi, int a0, int W, bool x_axis, float st,
                                           Pack<T, VEC>& centre, Pack<T, VEC>& size) {
    int gx = a0 % W, gy = a0 / W;  // one division per thread; the VEC anchors then walk the grid row by row
    if constexpr (DVecTraits<T, VEC>::packed) {
        typedef typename Pair<T>::type T2;
        const T2 half = Pair<T>::splat(0.5f), st2 = Pair<T>::splat(st);
        T2* oc = reinterpret_cast<T2*>(&centre.raw);
        T2* os = reinterpret_cast<T2*>(&size.raw);
#pragma unroll
        for (int i = 0; i < VEC; i += 2) {
            const int g0 = x_axis ? gx : gy;
            if (++gx >= W) { gx = 0; ++gy; }
            const int g1 = x_axis ? gx : gy;
            if (++gx >= W) { gx = 0; ++gy; }
            const T2 ac = __hadd2(Pair<T>::of_floats((float)g0, (float)g1), half);
            const T2 lo = *reinterpret_cast<const T2*>(&dlo.h2[i / 2]);
            const T2 hi = *reinterpret_cast<const T2*>(&dhi.h2[i / 2]);
            const T2 p1 = __hsub2(ac, lo), p2 = __hadd2(ac, hi);
            oc[i / 2] = __hmul2(__hmul2(__hadd2(p1, p2), half), st2);
            os[i / 2] = __hmul2(__hsub2(p2, p1), st2);
        }
    } else {
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            const int g = x_axis ? gx : gy;
            if (++gx >= W) { gx = 0; ++gy; }
            const float ac = rnd<T>(rnd<T>((float)g) + 0.5f);
            const float p1 = rnd<T>(ac - dlo.f[i]);
            const float p2 = rnd<T>(ac + dhi.f[i]);
            const float c = rnd<T>(rnd<T>(p1 + p2) * 0.5f);
            const float sz = rnd<T>(p2 - p1);
            centre.e[i] = from_f32<T>(c * st);
            size.e[i] = from_f32<T>(sz * st);
        }
    }
}

// class scores of one 16-byte (or narrower) vector, in place: sigmoid in fp32, rounded to the tensor dtype (yolo.py:99)
template <typename T, int VEC> __device__ __forceinline__ void sigmoid_pack(Pack<T, VEC>& v) {
    if constexpr ((VEC % 2) == 0) {
#pragma unroll
        for (int i = 0; i < VEC; i += 2) {
            const float2 s = sigmoid2(make_float2(to_f32<T>(v.e[i]), to_f32<T>(v.e[i + 1])));
            if constexpr (sizeof(T) == 2) {
                reinterpret_cast<uint32_t*>(&v.raw)[i / 2] = Pair<T>::pack2_rn(s.x, s.y);
            } else {
                v.e[i] = from_f32<T>(s.x);
                v.e[i + 1] = from_f32<T>(s.y);
            }
        }
    } else {
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            const float x = to_f32<T>(v.e[i]);
            v.e[i] = from_f32<T>(fast_rcp(1.f + fast_ex2(-x * LOG2E_F)));
        }
    }
}
