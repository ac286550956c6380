// Shared definitions for the cerb_post kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#define CERB_MAX_TASKS 8
#define CERB_MAX_LEVELS 4
#define CERB_REG_MAX 16  // DFL bins per side, reference models/yolo.py:75
#define CERB_DTYPE_F16 0
#define CERB_DTYPE_F32 1
#define CERB_DTYPE_BF16 2

// ---- rounding helpers: the reference computes every elementwise op in the tensor
// dtype, i.e. for half inputs each op is "compute in fp32, round to half".  rnd<T>()
// marks those rounding points (identity for float).
template <typename T> __device__ __forceinline__ float rnd(float v);
template <> __device__ __forceinline__ float rnd<float>(float v) { return v; }
// (packed convert: F2FP runs on the ALU pipes, the scalar F2F.F16.F32 on the SFU pipe the exps already load)
template <> __device__ __forceinline__ float rnd<__half>(float v) { return __low2float(__floats2half2_rn(v, 0.f)); }
template <> __device__ __forceinline__ float rnd<__nv_bfloat16>(float v) { return __low2float(__floats2bfloat162_rn(v, 0.f)); }

// two roundings at once: for half one F2FP.PACK_AB packs both values (the compiler does not pair scalar
// conversions by itself), for float nothing happens
template <typename T> __device__ __forceinline__ void rnd2(float a, float b, float& ra, float& rb);
template <> __device__ __forceinline__ void rnd2<float>(float a, float b, float& ra, float& rb) { ra = a; rb = b; }
template <> __device__ __forceinline__ void rnd2<__half>(float a, float b, float& ra, float& rb) {
    const float2 f = __half22float2(__floats2half2_rn(a, b));
    ra = f.x;
    rb = f.y;
}
template <> __device__ __forceinline__ void rnd2<__nv_bfloat16>(float a, float b, float& ra, float& rb) {
    const float2 f = __bfloat1622float2(__floats2bfloat162_rn(a, b));
    ra = f.x;
    rb = f.y;
}

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __low2half(__floats2half2_rn(v, 0.f)); }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) {
    return __low2bfloat16(__floats2bfloat162_rn(v, 0.f));
}

__device__ __forceinline__ float fast_ex2(float x) {
#ifdef CERB_EXPERIMENT_NO_MUFU  // tools/ only: where does the time go without the SFU?
    return x * 0.5f + 1.0f;
#else
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#endif
}
__device__ __forceinline__ float fast_rcp(float x) {
#ifdef CERB_EXPERIMENT_NO_MUFU
    return 2.0f - x;
#else
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#endif
}

// ---- mixed-precision FMA (sm_100a, PTX fma.rn.f32.f16 -> SASS FHFMA, fma.rn.f32.bf16 -> FHFMA.BF16): d = a * b + c.f32
// with a and b 16-bit values picked from the low / high half of a packed register, one rounding in fp32
__device__ __forceinline__ float fhfma_lo(uint32_t a2, uint32_t b2, float c) {
    float d;
    asm("{\n\t.reg .b16 al, ah, bl, bh;\n\tmov.b32 {al, ah}, %1;\n\tmov.b32 {bl, bh}, %2;\n\t"
        "fma.rn.f32.f16 %0, al, bl, %3;\n\t}"
        : "=f"(d) : "r"(a2), "r"(b2), "f"(c));
    return d;
}
__device__ __forceinline__ float fhfma_hi(uint32_t a2, uint32_t b2, float c) {
    float d;
    asm("{\n\t.reg .b16 al, ah, bl, bh;\n\tmov.b32 {al, ah}, %1;\n\tmov.b32 {bl, bh}, %2;\n\t"
        "fma.rn.f32.f16 %0, ah, bh, %3;\n\t}"
        : "=f"(d) : "r"(a2), "r"(b2), "f"(c));
    return d;
}
__device__ __forceinline__ float fbfma_lo(uint32_t a2, uint32_t b2, float c) {
    float d;
    asm("{\n\t.reg .b16 al, ah, bl, bh;\n\tmov.b32 {al, ah}, %1;\n\tmov.b32 {bl, bh}, %2;\n\t"
        "fma.rn.f32.bf16 %0, al, bl, %3;\n\t}"
        : "=f"(d) : "r"(a2), "r"(b2), "f"(c));
    return d;
}
__device__ __forceinline__ float fbfma_hi(uint32_t a2, uint32_t b2, float c) {
    float d;
    asm("{\n\t.reg .b16 al, ah, bl, bh;\n\tmov.b32 {al, ah}, %1;\n\tmov.b32 {bl, bh}, %2;\n\t"
        "fma.rn.f32.bf16 %0, ah, bh, %3;\n\t}"
        : "=f"(d) : "r"(a2), "r"(b2), "f"(c));
    return d;
}
__device__ __forceinline__ uint32_t pack_half2_rn(float lo, float hi) {
    const __half2 h = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack_bf162_rn(float lo, float hi) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&h);
}
// packed half2 bit pattern of two small non-negative integers (exact in half), a compile-time constant after unrolling
__host__ __device__ constexpr uint32_t half_bits_of_int(int k) {
    // k in [0, 2048): sign 0, exponent 15 + floor(log2 k), mantissa = the bits below the leading one
    if (k == 0) return 0u;
    int e = 0;
    for (int t = k; t > 1; t >>= 1) ++e;
    return (uint32_t)((15 + e) << 10) | (((uint32_t)k << (10 - e)) & 0x3FFu);
}
__host__ __device__ constexpr uint32_t half2_bits_of_ints(int lo, int hi) {
    return half_bits_of_int(lo) | (half_bits_of_int(hi) << 16);
}
static_assert(half_bits_of_int(1) == 0x3C00 && half_bits_of_int(3) == 0x4200 && half_bits_of_int(9) == 0x4880 &&
              half_bits_of_int(15) == 0x4B80, "half encoding of the DFL bin weights");
// the same for bfloat16 (k in [0, 256): exact with 8 significant bits): exponent 127 + floor(log2 k), 7 mantissa bits
__host__ __device__ constexpr uint32_t bf16_bits_of_int(int k) {
    if (k == 0) return 0u;
    int e = 0;
    for (int t = k; t > 1; t >>= 1) ++e;
    return (uint32_t)((127 + e) << 7) | (((uint32_t)k << (7 - e)) & 0x7Fu);
}
__host__ __device__ constexpr uint32_t bf162_bits_of_ints(int lo, int hi) {
    return bf16_bits_of_int(lo) | (bf16_bits_of_int(hi) << 16);
}
static_assert(bf16_bits_of_int(1) == 0x3F80 && bf16_bits_of_int(3) == 0x4040 && bf16_bits_of_int(9) == 0x4110 &&
              bf16_bits_of_int(15) == 0x4170, "bfloat16 encoding of the DFL bin weights");

// The packed forms of the two 16-bit tensor dtypes, for code that is written once for both: Pair<T>::type is the
// two-lane vector type, pack2_rn rounds two floats into one, mixfma_lo / _hi is the mixed-precision FMA on a lane and
// bits2_of_ints the packed pattern of two small integers.
template <typename T> struct Pair;
template <> struct Pair<__half> {
    typedef __half2 type;
    static __device__ __forceinline__ uint32_t pack2_rn(float lo, float hi) { return pack_half2_rn(lo, hi); }
    static __device__ __forceinline__ __half2 splat(float v) { return __float2half2_rn(v); }
    static __device__ __forceinline__ __half2 of_floats(float lo, float hi) { return __floats2half2_rn(lo, hi); }
    static __device__ __forceinline__ float mixfma_lo(uint32_t a2, uint32_t b2, float c) { return fhfma_lo(a2, b2, c); }
    static __device__ __forceinline__ float mixfma_hi(uint32_t a2, uint32_t b2, float c) { return fhfma_hi(a2, b2, c); }
    static __host__ __device__ constexpr uint32_t bits2_of_ints(int lo, int hi) { return half2_bits_of_ints(lo, hi); }
};
template <> struct Pair<__nv_bfloat16> {
    typedef __nv_bfloat162 type;
    static __device__ __forceinline__ uint32_t pack2_rn(float lo, float hi) { return pack_bf162_rn(lo, hi); }
    static __device__ __forceinline__ __nv_bfloat162 splat(float v) { return __float2bfloat162_rn(v); }
    static __device__ __forceinline__ __nv_bfloat162 of_floats(float lo, float hi) { return __floats2bfloat162_rn(lo, hi); }
    static __device__ __forceinline__ float mixfma_lo(uint32_t a2, uint32_t b2, float c) { return fbfma_lo(a2, b2, c); }
    static __device__ __forceinline__ float mixfma_hi(uint32_t a2, uint32_t b2, float c) { return fbfma_hi(a2, b2, c); }
    static __host__ __device__ constexpr uint32_t bits2_of_ints(int lo, int hi) { return bf162_bits_of_ints(lo, hi); }
};

// ---- packed fp32 pairs (sm_100a: PTX fma.rn.f32x2 / add.rn.f32x2 / mul.rn.f32x2 -> SASS FFMA2 / FADD2 / FMUL2): two
// IEEE fp32 operations (each rounded exactly like the scalar instruction) for one issue slot.  The decode kernels are
// issue-bound for half inputs (profiles/r01_decode.md), so every elementwise fp32 step is done on pairs.
#ifndef CERB_F32X2
#define CERB_F32X2 1
#endif
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
#if CERB_F32X2
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
        "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return d;
#else
    return make_float2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y));
#endif
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
#if CERB_F32X2
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tadd.rn.f32x2 rd, ra, rb;\n\t"
        "mov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
#else
    return make_float2(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y));
#endif
}
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
#if CERB_F32X2
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmul.rn.f32x2 rd, ra, rb;\n\t"
        "mov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
#else
    return make_float2(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y));
#endif
}

// Expected DFL distance of one box side: sum_k k * softmax(x)_k over the 16 bins (reference DFL.forward,
// models/yolo.py:57-59).  Rounding points follow the reference for half tensors: probabilities are rounded
// to half (softmax output), the frozen 1x1 conv accumulates in fp32 and rounds once.  Max, sum and the
// weighted sum are short trees / 4 partial sums (instruction-level parallelism instead of three 16-long
// dependency chains); the scale-and-shift before the exponentials, the sum and the normalisation run on
// packed fp32 pairs (bins k, k+1).  dfl_expectation_acc returns the fp32 accumulator BEFORE its final rounding.
// bfloat16 follows the same rules with bf16 in place of half.
#define CERB_LOG2E 1.4426950408889634f
template <typename T> __device__ __forceinline__ float dfl_expectation_acc(float (&x)[CERB_REG_MAX]) {
#ifdef CERB_EXPERIMENT_COPY_ONLY  // tools/ only: memory floor of this access pattern
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < CERB_REG_MAX; ++k) t += x[k];
    return t;
#endif
    float m0 = fmaxf(fmaxf(x[0], x[1]), fmaxf(x[2], x[3]));
    float m1 = fmaxf(fmaxf(x[4], x[5]), fmaxf(x[6], x[7]));
    float m2 = fmaxf(fmaxf(x[8], x[9]), fmaxf(x[10], x[11]));
    float m3 = fmaxf(fmaxf(x[12], x[13]), fmaxf(x[14], x[15]));
    const float nmb = -(fmaxf(fmaxf(m0, m1), fmaxf(m2, m3)) * CERB_LOG2E);
    float2 e[CERB_REG_MAX / 2];
#pragma unroll
    for (int k = 0; k < CERB_REG_MAX / 2; ++k) {
        const float2 u = ffma2(make_float2(x[2 * k], x[2 * k + 1]), make_float2(CERB_LOG2E, CERB_LOG2E), make_float2(nmb, nmb));
        e[k] = make_float2(fast_ex2(u.x), fast_ex2(u.y));
    }
    const float2 s01 = fadd2(fadd2(e[0], e[1]), fadd2(e[2], e[3]));
    const float2 s23 = fadd2(fadd2(e[4], e[5]), fadd2(e[6], e[7]));
    const float2 s = fadd2(s01, s23);
    const float inv = fast_rcp(s.x + s.y);
    const float2 inv2 = make_float2(inv, inv);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#ifndef CERB_NO_FHFMA
    if constexpr (sizeof(T) == 2) {
        // half / bf16: the rounded probabilities stay packed and feed the mixed-precision FMA (FHFMA: f16 x f16 + f32,
        // one rounding) -- the same value as fmaf((float)k, (float)p, acc) without the two unpacking converts per pair
        typedef Pair<T> P2;
#pragma unroll
        for (int k = 0; k < CERB_REG_MAX; k += 4) {
            const float2 q01 = fmul2(e[k / 2], inv2), q23 = fmul2(e[k / 2 + 1], inv2);
            const uint32_t p01 = P2::pack2_rn(q01.x, q01.y);
            const uint32_t p23 = P2::pack2_rn(q23.x, q23.y);
            if (k != 0) a0 = P2::mixfma_lo(p01, P2::bits2_of_ints(k, k + 1), a0);  // 0 * p0 + 0 == +0
            a1 = P2::mixfma_hi(p01, P2::bits2_of_ints(k, k + 1), a1);
            a2 = P2::mixfma_lo(p23, P2::bits2_of_ints(k + 2, k + 3), a2);
            a3 = P2::mixfma_hi(p23, P2::bits2_of_ints(k + 2, k + 3), a3);
        }
        return (a0 + a1) + (a2 + a3);
    } else
#endif
    {
        float2 a01 = make_float2(0.f, 0.f), a23 = make_float2(0.f, 0.f);
#pragma unroll
        for (int k = 0; k < CERB_REG_MAX; k += 4) {
            float2 q01 = fmul2(e[k / 2], inv2), q23 = fmul2(e[k / 2 + 1], inv2);
            rnd2<T>(q01.x, q01.y, q01.x, q01.y);
            rnd2<T>(q23.x, q23.y, q23.x, q23.y);
            a01 = ffma2(make_float2((float)k, (float)(k + 1)), q01, a01);
            a23 = ffma2(make_float2((float)(k + 2), (float)(k + 3)), q23, a23);
        }
        const float2 a = fadd2(a01, a23);
        return a.x + a.y;
    }
}
template <typename T> __device__ __forceinline__ float dfl_expectation(float (&x)[CERB_REG_MAX]) {
    return rnd<T>(dfl_expectation_acc<T>(x));
}

// sigmoid of two logits at once (reference models/yolo.py:99): 1 / (1 + 2^(-x log2 e)), the scale and the "+ 1" on
// packed fp32 pairs; the caller rounds to the tensor dtype
__device__ __forceinline__ float2 sigmoid2(float2 x) {
    const float2 t = fmul2(x, make_float2(-CERB_LOG2E, -CERB_LOG2E));
    const float2 u = fadd2(make_float2(fast_ex2(t.x), fast_ex2(t.y)), make_float2(1.f, 1.f));
    return make_float2(fast_rcp(u.x), fast_rcp(u.y));
}

// streaming 128-bit / 64-bit / scalar accesses (read once, write once: keep them out of L1)
__device__ __forceinline__ uint4 ldg_stream16(const void* p) {
    uint4 r;
#if defined(CERB_LD_L2_256)
    asm volatile("ld.global.nc.L1::no_allocate.L2::256B.v4.u32 {%0,%1,%2,%3}, [%4];"
#elif defined(CERB_LD_L2_128)
    asm volatile("ld.global.nc.L1::no_allocate.L2::128B.v4.u32 {%0,%1,%2,%3}, [%4];"
#elif defined(CERB_LD_PLAIN)
    asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];"
#else
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
#endif
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream16(void* p, uint4 v) {
#ifdef CERB_L2_STORE_HINT  // experiment: keep the decode outputs in L2 for the NMS kernel (profiles/r01_decode.md)
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v4.u32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(p), "r"(v.x), "r"(v.y),
                 "r"(v.z), "r"(v.w), "l"(pol)
                 : "memory");
#else
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w)
                 : "memory");
#endif
}

// host-side error plumbing of the C ABI (api.cu): the message cerb_last_error() returns is thread-local
void cerb_set_error(const char* fmt, ...);
void cerb_clear_error();
// 0, or CERB_ECUDA with "<fn>: launch failed: <msg>"
int cerb_launch_status(const char* fn, cudaError_t e);
// 0 when the call needs no workspace or gets enough, else CERB_ENOSPC with "<fn>: workspace of N bytes required, got M"
int cerb_require_workspace(const char* fn, const void* ws, size_t have, size_t need);
inline bool cerb_aligned(const void* p, size_t bytes) { return reinterpret_cast<uintptr_t>(p) % bytes == 0; }
// argument check of an entry point: on failure set the message and return CERB_EINVAL
#define CERB_REQUIRE(cond, ...)          \
    do {                                 \
        if (!(cond)) {                   \
            cerb_set_error(__VA_ARGS__); \
            return CERB_EINVAL;          \
        }                                \
    } while (0)
bool cerb_debug_knob(const char* name, int* out);  // thread-local / environment test knob, false when unset
