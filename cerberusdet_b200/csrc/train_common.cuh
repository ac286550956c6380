// Row access shared by the training-time kernels (train_decode.cu, bbox_loss.cu): pred_dist is [B, A, 64] with the 16
// bins of a side contiguous, so a thread that owns one (anchor, side) moves its 16 values in one (fp16) or two (fp32)
// 256-bit accesses.  sm_100a only.
#pragma once
#include "cerb_kernels.h"

// 256-bit global accesses (sm_100a: LDG.E.256 / STG.E.256): a thread's 16 half bins are exactly one 32-byte sector, so
// a warp reads 1 KB contiguous per instruction with every sector requested once
struct __align__(32) U8x32 { uint32_t w[8]; };
__device__ __forceinline__ U8x32 ldg_stream32(const void* p) {
    U8x32 r;
    asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r.w[0]), "=r"(r.w[1]), "=r"(r.w[2]), "=r"(r.w[3]), "=r"(r.w[4]), "=r"(r.w[5]), "=r"(r.w[6]), "=r"(r.w[7])
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream32(void* p, const U8x32& r) {
    asm volatile("st.global.L1::no_allocate.v8.u32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(r.w[0]), "r"(r.w[1]),
                 "r"(r.w[2]), "r"(r.w[3]), "r"(r.w[4]), "r"(r.w[5]), "r"(r.w[6]), "r"(r.w[7])
                 : "memory");
}

template <typename T> struct Row16;  // the 16 bins of one (anchor, side)
template <> struct Row16<__half> {
    static constexpr int NV = 1;
    U8x32 v[1];
    __device__ __forceinline__ float get(int k) const { return __half2float(reinterpret_cast<const __half*>(v)[k]); }
    __device__ __forceinline__ void set(int k, float f) { reinterpret_cast<__half*>(v)[k] = from_f32<__half>(f); }
};
template <> struct Row16<float> {
    static constexpr int NV = 2;
    U8x32 v[2];
    __device__ __forceinline__ float get(int k) const { return reinterpret_cast<const float*>(v)[k]; }
    __device__ __forceinline__ void set(int k, float f) { reinterpret_cast<float*>(v)[k] = f; }
};

template <typename T, bool ALIGNED> __device__ __forceinline__ void load_row(const T* p, Row16<T>& r) {
    if constexpr (ALIGNED) {
#pragma unroll
        for (int i = 0; i < Row16<T>::NV; ++i) r.v[i] = ldg_stream32(reinterpret_cast<const U8x32*>(p) + i);
    } else {
#pragma unroll
        for (int k = 0; k < CERB_REG_MAX; ++k) reinterpret_cast<T*>(r.v)[k] = p[k];
    }
}
template <typename T, bool ALIGNED> __device__ __forceinline__ void store_row(T* p, const Row16<T>& r) {
    if constexpr (ALIGNED) {
#pragma unroll
        for (int i = 0; i < Row16<T>::NV; ++i) stg_stream32(reinterpret_cast<U8x32*>(p) + i, r.v[i]);
    } else {
#pragma unroll
        for (int k = 0; k < CERB_REG_MAX; ++k) p[k] = reinterpret_cast<const T*>(r.v)[k];
    }
}
