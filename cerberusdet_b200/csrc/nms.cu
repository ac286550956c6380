// Per-task confidence filter, candidate expansion, lazy top-k ordering and class-offset
// greedy NMS -- one CTA per (task, image) segment, all segments in ONE launch.
//
// Replaces reference non_max_suppression (utils/general.py:360-481) incl. xywh2xyxy
// (:272-288) and the third-party torchvision.ops.nms it calls (:464).  The reference
// runs ~25 ATen launches and ~4 host syncs per (image, task) and materialises every
// candidate; this kernel never materialises the candidate table:
//
//  * Candidates are implicit: (anchor a, class c) pairs of the prediction whose score
//    passes the threshold (multi-label, :444-446) or the best class of an anchor
//    (:447-449).  Each gets a unique 64-bit key  score_bits << 32 | ~(a*nc + c), so that
//    descending key order == "score descending, candidate index ascending", the
//    canonical form of the reference's sort at :459 (ties there are unspecified).  score_bits
//    are the fp32 bits of the score: a half or bfloat16 score widens exactly (bf16: its own
//    bits << 16), and the non-negative sigmoid outputs order as unsigned integers.
//  * Greedy NMS is order-causal and stops at max_det (:465), so only a prefix of the
//    sorted order is ever needed.  A 2048-bin histogram of the top 12 key bits locates
//    successive chunks of <= CAP keys; each chunk is gathered, bitonic-sorted (registers +
//    shuffles + shared memory) and consumed; the kernel stops as soon as max_det boxes are
//    kept or max_nms candidates (:459) were consumed.  The histogram only steers chunk
//    sizes, so it may be an estimate: from the score summary the decode kernel leaves (one
//    maximum per 16-byte score vector), or from every 8th score vector; what a chunk
//    contains, its order and every count that matters are exact.  An overflowing chunk
//    switches the segment to an exact histogram; a single bin that exceeds CAP (massive
//    ties) is refined by deeper 12-bit radix levels down to unique keys.
//  * Scans.  With a summary, pass 1 reads it (1/8 of the scores) and lists the score
//    vectors whose maximum reaches the chunk's lower bound, pass 2 reads only those; list
//    and key slots are reserved per warp (count, prefix-sum, one atomic).  Without a
//    summary, or when the candidates are dense, the class planes are scanned with 128-bit
//    loads and a packed-half2 range prefilter.
//  * Suppression (:462-465): candidates are taken in tiles of 512, one per thread; a
//    candidate is first tested against the kept list (shared memory), then the tile is
//    resolved internally with a per-thread suppressor bitmask and a ballot fixpoint
//    iteration (equal to the sequential sweep).  Per-class chains skip the pairs that the
//    class offset makes disjoint.  IoU arithmetic reproduces torchvision's CPU kernel:
//    separately rounded fp32 ops on class-offset boxes, strict '>' against the threshold
//    (the double-precision compare is folded into iou_thr).
//  History, counters and the experiments that did not work: profiles/r01_nms.md.
#include <stdlib.h>

#include "cerb_kernels.h"

#define NMS_THREADS 512
#define NMS_TILE 512         // == NMS_THREADS: one candidate per thread
#define NMS_TILE_WORDS (NMS_TILE / 64)
#define NMS_CAP 4096         // max keys sorted at once
#define NMS_BINS 4096        // 12-bit radix digits
#define NMS_KEPT_SMEM 1024   // kept list lives in smem up to this max_det
#define NMS_BUCKETS 1024     // class buckets of the kept-list chains (class & 1023)

typedef unsigned long long u64;

// Optional per-CTA wall times (-DNMS_BLOCK_TIMES, tools/nms_block_times.py only): start / end %globaltimer and SM id of
// every CTA of the last launch -- shows whether the kernel's duration is one slow segment or all of them.
#ifdef NMS_BLOCK_TIMES
__device__ unsigned long long g_nms_block_t[3][4096];
__device__ __forceinline__ unsigned long long nms_globaltimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
extern "C" int cerb_debug_read_block_times(unsigned long long* out, int n) {
    cudaDeviceSynchronize();
    if (n > 4096) n = 4096;
    for (int k = 0; k < 3; ++k)
        if (cudaMemcpyFromSymbol(out + (size_t)k * n, g_nms_block_t, sizeof(unsigned long long) * n,
                                 sizeof(unsigned long long) * 4096 * k) != cudaSuccess)
            return -1;
    return 0;
}
#define BLOCK_T_START                                                                      \
    if (threadIdx.x == 0 && blockIdx.x < 4096) {                                            \
        unsigned smid;                                                                      \
        asm volatile("mov.u32 %0, %smid;" : "=r"(smid));                                    \
        g_nms_block_t[0][blockIdx.x] = nms_globaltimer();                                   \
        g_nms_block_t[2][blockIdx.x] = smid;                                                \
    }
#define BLOCK_T_END \
    if (threadIdx.x == 0 && blockIdx.x < 4096) g_nms_block_t[1][blockIdx.x] = nms_globaltimer();
#else
#define BLOCK_T_START
#define BLOCK_T_END
#endif

// Optional phase timers (-DNMS_PROFILE, tools/ only): thread 0 of EVERY block accumulates clock64() deltas per phase in
// registers/local memory (no global traffic at the stamps, so short phases are not inflated) and adds them to the global
// totals once, at the end of the kernel.  g_nms_prof[0..9] phases, [10] blocks, [11] consumed, [12..14] collect sub-steps,
// [15] fixpoint rounds, [16] chunks collected, [17] tiles, [18] score vectors listed by summary pass 1, [19] chunks that
// fell back to the plain scan, [20] exact-histogram rebuilds, [21] / [22] fixpoint settle-loop iterations / cycles summed
// over the warps.  The collect sub-steps, [18], [21] and [22] are global atomics at the stamp (PROFX / PROF_GADD).
#ifdef NMS_PROFILE
#define NMS_PROF_SLOTS 24
__device__ unsigned long long g_nms_prof[NMS_PROF_SLOTS];
__shared__ long long s_profx_t;
#define PROF_DECL long long prof_t = clock64(); unsigned long long prof_acc[NMS_PROF_SLOTS] = {0};
#define PROF_COUNT(slot, n) do { if (threadIdx.x == 0) prof_acc[slot] += (n); } while (0)
#define PROF_GADD(slot, n) do { if (threadIdx.x == 0) atomicAdd(&g_nms_prof[slot], (unsigned long long)(n)); } while (0)
#define PROFX_START do { if (threadIdx.x == 0) s_profx_t = clock64(); } while (0)
#define PROFX(slot)                                                              \
    do {                                                                         \
        if (threadIdx.x == 0) {                                                  \
            const long long now_ = clock64();                                    \
            atomicAdd(&g_nms_prof[slot], (unsigned long long)(now_ - s_profx_t)); \
            s_profx_t = now_;                                                    \
        }                                                                        \
    } while (0)
#define PROF(slot)                                                        \
    do {                                                                  \
        if (threadIdx.x == 0) {                                           \
            const long long now = clock64();                              \
            prof_acc[slot] += (unsigned long long)(now - prof_t);         \
            prof_t = now;                                                 \
        }                                                                 \
    } while (0)
#define PROF_FLUSH(consumed_)                                             \
    do {                                                                  \
        if (threadIdx.x == 0) {                                           \
            prof_acc[10] = 1; prof_acc[11] = (consumed_);                 \
            for (int i_ = 0; i_ < NMS_PROF_SLOTS; ++i_) if (prof_acc[i_]) atomicAdd(&g_nms_prof[i_], prof_acc[i_]); \
        }                                                                 \
    } while (0)
// out receives NMS_PROF_SLOTS (24) counters
extern "C" int cerb_debug_read_profile(unsigned long long* out, int reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, g_nms_prof, sizeof(unsigned long long) * NMS_PROF_SLOTS);
    if (reset) { unsigned long long z[NMS_PROF_SLOTS] = {0}; cudaMemcpyToSymbol(g_nms_prof, z, sizeof(z)); }
    return 0;
}
#else
#define PROF_DECL
#define PROF(slot) do {} while (0)
#define PROF_COUNT(slot, n) do {} while (0)
#define PROF_GADD(slot, n) do {} while (0)
#define PROFX_START do {} while (0)
#define PROFX(slot) do {} while (0)
#define PROF_FLUSH(c) do {} while (0)
#endif

struct __align__(16) NmsSmem {
    unsigned g0[NMS_BINS + 8];   // level-0: G0[d] = #keys with digit >= d (histogram units); G0[4096] = 0
    unsigned g1[NMS_BINS + 8];   // scratch for deeper levels
    u64 keys[NMS_CAP];
    float4 tbox[NMS_TILE];       // class-offset corners of the tile's candidates
    float tarea[NMS_TILE];
    int tcode[NMS_TILE];         // class id if the box is "tame" (see class shortcut), -1 wild, -2 padding
    int tprev[NMS_TILE];         // previous candidate of the same class inside the tile, or -1
    unsigned keep32[2][NMS_TILE / 32];
    unsigned char tdead[NMS_TILE];
    unsigned warp_tot[NMS_THREADS / 32];
    unsigned counter, nhits;
    int tile_wild, kept_wild;
    int khead[NMS_BUCKETS];      // newest kept box of each class bucket, or -1
    int knext_s[NMS_KEPT_SMEM];  // next kept box of the same bucket
    float4 kbox[NMS_KEPT_SMEM];
    float karea[NMS_KEPT_SMEM];
};

// ---- IoU test exactly as torchvision's CPU kernel does it (std::max/std::min semantics,
// one rounding per operation, no FMA).  box i is the earlier (kept) box.
__device__ __forceinline__ bool suppresses(const float4 bi, const float ai, const float4 bj, const float aj,
                                           const float thr) {
    const float xx1 = (bi.x < bj.x) ? bj.x : bi.x;
    const float yy1 = (bi.y < bj.y) ? bj.y : bi.y;
    const float xx2 = (bj.z < bi.z) ? bj.z : bi.z;
    const float yy2 = (bj.w < bi.w) ? bj.w : bi.w;
    const float dw = __fsub_rn(xx2, xx1), dh = __fsub_rn(yy2, yy1);
    const float w = (0.f < dw) ? dw : 0.f;
    const float h = (0.f < dh) ? dh : 0.f;
    const float inter = __fmul_rn(w, h);
    if (!(inter > 0.f)) return false;  // quotient would be 0 (or NaN): never > thr >= 0
    const float uni = __fsub_rn(__fadd_rn(ai, aj), inter);
    return __fdiv_rn(inter, uni) > thr;
}

// ---- enumerate the candidates of one segment; f(score_bits, anchor, class) is called once per
// candidate.  Scores are read with 128-bit loads (the class planes of one image are one contiguous
// [nc*A] array) whenever A is a multiple of the vector width and the base is 16-byte aligned.
__device__ __forceinline__ unsigned make_sbits(float s) { return __float_as_uint(s); }
__device__ __forceinline__ u64 make_key(unsigned sbits, unsigned idx) {
    return ((u64)sbits << 32) | (u64)(0xFFFFFFFFu - idx);
}

// Warp-aggregated shared-memory atomics: many lanes of a warp hitting ONE address serialise otherwise.
__device__ __forceinline__ unsigned lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}
// all currently active lanes take consecutive slots of *counter; returns this lane's slot
__device__ __forceinline__ unsigned warp_take_slot(unsigned* counter) {
    const unsigned active = __activemask();
    const int leader = __ffs(active) - 1;
    unsigned base = 0;
    if ((int)(threadIdx.x & 31) == leader) base = atomicAdd(counter, (unsigned)__popc(active));
    base = __shfl_sync(active, base, leader);
    return base + __popc(active & lanemask_lt());
}
// every active lane adds 1 to hist[bin]; lanes with equal bins are merged into one atomic
__device__ __forceinline__ void warp_hist_add(unsigned* hist, unsigned bin) {
    const unsigned active = __activemask();
    const unsigned peers = __match_any_sync(active, bin);
    if ((int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[bin], (unsigned)__popc(peers));
}

// Slot reservation without a returning atomic per item: a shared-memory atomicAdd that returns a value costs ~13
// cycles and same-address ones serialise across the whole CTA (1.2 k list pushes = 15 k cycles, measured), so every
// lane first counts its items, the warp prefix-sums the counts and ONE lane reserves the warp's total.  Must be
// called by all 32 lanes; returns this lane's first slot.
__device__ __forceinline__ unsigned warp_reserve(unsigned* counter, unsigned n) {
    const unsigned lane = threadIdx.x & 31u;
    unsigned inc = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += t;
    }
    const unsigned total = __shfl_sync(0xffffffffu, inc, 31);
    unsigned base = 0;
    if (total) {
        if (lane == 31u) base = atomicAdd(counter, total);
        base = __shfl_sync(0xffffffffu, base, 31);
    }
    return base + inc - n;
}

template <typename T> struct ScoreVec {
    static constexpr int V = 16 / sizeof(T);
    union { uint4 raw; T e[16 / sizeof(T)]; };
};

#define SCAN_UNROLL 4

// padded length of one class row of the score summary: roundup(A / V, V) entries (rows stay 16-byte aligned)
template <typename T> __host__ __device__ __forceinline__ size_t summary_row_len(int A) {
    const size_t V = 16 / sizeof(T);
    return ((size_t)A / V + V - 1) / V * V;
}

// Per-dtype form of the score-bit range [sb_lo, sb_hi] (positive floats: bit order == value order).
template <typename T> struct RangeBounds;
template <> struct RangeBounds<float> { unsigned lo, span; };
template <> struct RangeBounds<__half> { __half2 lo2, hi2; };
template <> struct RangeBounds<__nv_bfloat16> { __nv_bfloat162 lo2, hi2; };
template <typename T> __device__ __forceinline__ RangeBounds<T> make_range_bounds(unsigned sb_lo, unsigned sb_hi);
template <> __device__ __forceinline__ RangeBounds<float> make_range_bounds<float>(unsigned sb_lo, unsigned sb_hi) {
    RangeBounds<float> r;
    r.lo = sb_lo;
    r.span = sb_hi - sb_lo;
    return r;
}
template <> __device__ __forceinline__ RangeBounds<__half> make_range_bounds<__half>(unsigned sb_lo, unsigned sb_hi) {
    // smallest half >= lo and largest half <= hi: for half data  lo <= float(s) <= hi  <=>  lo_h <= s <= hi_h
    RangeBounds<__half> r;
    r.lo2 = __half2half2(__float2half_ru(__uint_as_float(sb_lo)));
    r.hi2 = __half2half2(__float2half_rd(__uint_as_float(sb_hi)));
    return r;
}
template <>
__device__ __forceinline__ RangeBounds<__nv_bfloat16> make_range_bounds<__nv_bfloat16>(unsigned sb_lo, unsigned sb_hi) {
    // smallest bf16 >= lo and largest bf16 <= hi, as for half
    RangeBounds<__nv_bfloat16> r;
    r.lo2 = __bfloat162bfloat162(__float2bfloat16_ru(__uint_as_float(sb_lo)));
    r.hi2 = __bfloat162bfloat162(__float2bfloat16_rd(__uint_as_float(sb_hi)));
    return r;
}
// bit k set iff element k of the vector has its score bits in [sb_lo, sb_hi]
template <typename T>
__device__ __forceinline__ unsigned range_hits(const ScoreVec<T>& v, unsigned sb_lo, unsigned sb_hi, const RangeBounds<T>& rb);
template <>
__device__ __forceinline__ unsigned range_hits<float>(const ScoreVec<float>& v, unsigned, unsigned, const RangeBounds<float>& rb) {
    unsigned h = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) h |= ((__float_as_uint(v.e[k]) - rb.lo) <= rb.span ? 1u : 0u) << k;
    return h;
}
template <>
__device__ __forceinline__ unsigned range_hits<__half>(const ScoreVec<__half>& v, unsigned, unsigned, const RangeBounds<__half>& rb) {
    const __half2* h2 = reinterpret_cast<const __half2*>(&v.raw);
    unsigned m[4], any = 0;
#pragma unroll
    for (int p = 0; p < 4; ++p) { m[p] = __hge2_mask(h2[p], rb.lo2) & __hle2_mask(h2[p], rb.hi2); any |= m[p]; }
    if (!any) return 0u;
    unsigned h = 0;
#pragma unroll
    for (int p = 0; p < 4; ++p) h |= ((m[p] & 1u) | ((m[p] >> 15) & 2u)) << (2 * p);
    return h;
}
template <>
__device__ __forceinline__ unsigned range_hits<__nv_bfloat16>(const ScoreVec<__nv_bfloat16>& v, unsigned, unsigned,
                                                               const RangeBounds<__nv_bfloat16>& rb) {
    const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&v.raw);
    unsigned m[4], any = 0;
#pragma unroll
    for (int p = 0; p < 4; ++p) { m[p] = __hge2_mask(h2[p], rb.lo2) & __hle2_mask(h2[p], rb.hi2); any |= m[p]; }
    if (!any) return 0u;
    unsigned h = 0;
#pragma unroll
    for (int p = 0; p < 4; ++p) h |= ((m[p] & 1u) | ((m[p] >> 15) & 2u)) << (2 * p);
    return h;
}

template <typename T, bool MULTI, typename F>
__device__ __forceinline__ void for_each_candidate(const T* __restrict__ img, int nc, int A, float thr,
                                                   const NmsParams& P, F f, unsigned sb_lo = 0u,
                                                   unsigned sb_hi = 0x7F800000u, const unsigned vstride = 1) {
    // Only candidates whose score bits lie in [sb_lo, sb_hi] are reported (a whole vector is rejected with
    // a few packed compares).  vstride > 1 visits only every vstride-th 16-byte vector (multi-label vector
    // path only): used for the *estimating* histogram; every exact pass uses vstride == 1.
    constexpr int V = ScoreVec<T>::V;
    {   // fold the strict "score > conf_thres" (thr >= 0, so it is a bit-pattern compare) into the range
        const unsigned tb = __float_as_uint(thr) + 1u;
        sb_lo = sb_lo > tb ? sb_lo : tb;
        sb_hi = sb_hi < 0x7F800000u ? sb_hi : 0x7F800000u;  // excludes NaN
    }
    if (sb_lo > sb_hi) return;
    const T* __restrict__ sc = img + (size_t)4 * A;
    const bool vec_ok = (A % V == 0) && ((reinterpret_cast<uintptr_t>(sc) & 15) == 0);
    const bool filt = P.use_class_filter != 0;
    if (MULTI) {
        if (vec_ok) {
            const unsigned nvec = (unsigned)(((u64)nc * (u64)A) / V);
            const unsigned nvis = (nvec + vstride - 1) / vstride;  // vectors visited
            const RangeBounds<T> rb = make_range_bounds<T>(sb_lo, sb_hi);
            for (unsigned q0 = threadIdx.x; q0 < nvis; q0 += NMS_THREADS * SCAN_UNROLL) {
                ScoreVec<T> v[SCAN_UNROLL];
#pragma unroll
                for (int u = 0; u < SCAN_UNROLL; ++u) {
                    const unsigned q = q0 + u * NMS_THREADS;
                    if (q < nvis) v[u].raw = __ldg(reinterpret_cast<const uint4*>(sc) + (size_t)q * vstride);
                }
#pragma unroll
                for (int u = 0; u < SCAN_UNROLL; ++u) {
                    const unsigned q = q0 + u * NMS_THREADS;
                    if (q >= nvis) break;
                    const unsigned hits = range_hits<T>(v[u], sb_lo, sb_hi, rb);
                    if (!hits) continue;
                    const unsigned e0 = q * vstride * V;
                    const unsigned c = e0 / (unsigned)A;
                    const unsigned a0 = e0 - c * (unsigned)A;
                    if (filt && !((P.class_mask[c >> 5] >> (c & 31)) & 1u)) continue;
#pragma unroll
                    for (int k = 0; k < V; ++k)
                        if ((hits >> k) & 1u) f(make_sbits(to_f32<T>(v[u].e[k])), (int)(a0 + k), (int)c);
                }
            }
        } else {
            for (int c = 0; c < nc; ++c) {
                if (filt && !((P.class_mask[c >> 5] >> (c & 31)) & 1u)) continue;
                const T* __restrict__ row = sc + (size_t)c * A;
                for (int a = threadIdx.x; a < A; a += NMS_THREADS) {
                    const unsigned sb = make_sbits(to_f32<T>(__ldg(row + a)));
                    if (sb - sb_lo <= sb_hi - sb_lo) f(sb, a, c);
                }
            }
        }
    } else {
        if (vec_ok) {
            const int nv = A / V;
            for (int i = threadIdx.x; i < nv; i += NMS_THREADS) {
                const uint4* __restrict__ col = reinterpret_cast<const uint4*>(sc) + i;
                float best[V];
                int bc[V];
                {
                    ScoreVec<T> v0;
                    v0.raw = __ldg(col);
#pragma unroll
                    for (int k = 0; k < V; ++k) { best[k] = to_f32<T>(v0.e[k]); bc[k] = 0; }
                }
                int c = 1;
                for (; c + SCAN_UNROLL <= nc; c += SCAN_UNROLL) {
                    ScoreVec<T> v[SCAN_UNROLL];
#pragma unroll
                    for (int u = 0; u < SCAN_UNROLL; ++u) v[u].raw = __ldg(col + (size_t)(c + u) * nv);
#pragma unroll
                    for (int u = 0; u < SCAN_UNROLL; ++u)
#pragma unroll
                        for (int k = 0; k < V; ++k) {
                            const float s = to_f32<T>(v[u].e[k]);
                            if (s > best[k]) { best[k] = s; bc[k] = c + u; }  // lowest index wins ties (torch.max)
                        }
                }
                for (; c < nc; ++c) {
                    ScoreVec<T> v1;
                    v1.raw = __ldg(col + (size_t)c * nv);
#pragma unroll
                    for (int k = 0; k < V; ++k) {
                        const float s = to_f32<T>(v1.e[k]);
                        if (s > best[k]) { best[k] = s; bc[k] = c; }
                    }
                }
#pragma unroll
                for (int k = 0; k < V; ++k) {
                    const unsigned sb = make_sbits(best[k]);
                    if (sb - sb_lo <= sb_hi - sb_lo) {
                        if (filt && !((P.class_mask[bc[k] >> 5] >> (bc[k] & 31)) & 1u)) continue;
                        f(sb, i * V + k, bc[k]);
                    }
                }
            }
        } else {
            for (int a = threadIdx.x; a < A; a += NMS_THREADS) {
                float best = to_f32<T>(__ldg(sc + a));
                int bc = 0;
                for (int c = 1; c < nc; ++c) {
                    const float s = to_f32<T>(__ldg(sc + (size_t)c * A + a));
                    if (s > best) { best = s; bc = c; }  // lowest index wins ties (torch.max)
                }
                const unsigned sb = make_sbits(best);
                if (sb - sb_lo <= sb_hi - sb_lo) {
                    if (filt && !((P.class_mask[bc >> 5] >> (bc & 31)) & 1u)) continue;
                    f(sb, a, bc);
                }
            }
        }
    }
}

// ---- the same enumeration guided by the score summary written by the decode kernel: smax[c][vi] is the
// maximum of score vector vi (V consecutive anchors) of class c, rows padded to SNV = roundup(A/V, V) entries.
// Pass 1 reads the summary and lists the score vectors whose maximum reaches sb_lo (shared-memory list `hits`,
// NMS_BINS entries); pass 2 reads just those.  Returns false -- having reported nothing -- when the list
// overflows: then the candidates are dense and the caller runs the plain scan instead.
// WITH_SCORES == false stops after pass 1 and reports one pseudo-candidate per listed vector (its maximum):
// that is the estimating histogram.
template <typename T, bool MULTI, bool WITH_SCORES, typename F>
__device__ __forceinline__ bool for_each_candidate_summary(const T* __restrict__ img, const T* __restrict__ smax,
                                                           int nc, int A, float thr, const NmsParams& P, F f,
                                                           unsigned sb_lo, unsigned sb_hi, unsigned* hits,
                                                           unsigned* nhits, u64 lo = 0, u64 hi = 0, u64* keys = nullptr,
                                                           unsigned* counter = nullptr) {
    // WITH_SCORES: the keys in [lo, hi) are appended to keys[] / *counter (slots reserved per warp, see
    // warp_reserve).  !WITH_SCORES: f(max_bits, 0, 0) per summary entry in range (the estimating histogram).
    constexpr int V = ScoreVec<T>::V;
    const T* __restrict__ sc = img + (size_t)4 * A;
    const unsigned NV = (unsigned)A / V;          // score vectors per class row
    const unsigned SNV = (NV + V - 1) / V * V;    // padded summary row length
    const unsigned SV = SNV / V;                  // 16-byte summary vectors per row
    const bool filt = P.use_class_filter != 0;
    {
        const unsigned tb = __float_as_uint(thr) + 1u;
        sb_lo = sb_lo > tb ? sb_lo : tb;
        sb_hi = sb_hi < 0x7F800000u ? sb_hi : 0x7F800000u;
    }
    if (sb_lo > sb_hi) return true;
    const RangeBounds<T> rb = make_range_bounds<T>(sb_lo, sb_hi);
    const RangeBounds<T> rb_any = make_range_bounds<T>(sb_lo, 0x7F800000u);  // "maximum reaches sb_lo"
    const unsigned nsv = MULTI ? (unsigned)nc * SV : SV;
    if (WITH_SCORES) {
        __syncthreads();
        if (threadIdx.x == 0) *nhits = 0;
        __syncthreads();
        PROFX_START;
    }
    // ---- pass 1: the summary (block-uniform trip count: warp_reserve needs whole warps)
    for (unsigned qb = 0; qb < nsv; qb += NMS_THREADS * SCAN_UNROLL) {
        const unsigned q0 = qb + threadIdx.x;
        ScoreVec<T> m[SCAN_UNROLL];
#pragma unroll
        for (int u = 0; u < SCAN_UNROLL; ++u) {
            // rows are SV vectors apart (SNV == SV * V), so summary vector q sits at smax + q * V.  The index is clamped
            // rather than tested: behind a branch per load the compiler parks each loaded vector in local memory, which
            // serialises the loads and, with 2 CTAs of 109 KB per SM, sends every reload to L2.
            const unsigned q = min(q0 + u * NMS_THREADS, nsv - 1u);
            m[u].raw = __ldg(reinterpret_cast<const uint4*>(smax) + q);
        }
        unsigned h[SCAN_UNROLL], ebase[SCAN_UNROLL], cnt = 0;
#pragma unroll
        for (int u = 0; u < SCAN_UNROLL; ++u) {
            h[u] = 0;
            ebase[u] = 0;
            const unsigned q = q0 + u * NMS_THREADS;
            if (q >= nsv) continue;
            const unsigned c = MULTI ? q / SV : 0u;
            const unsigned j0 = (MULTI ? q - c * SV : q) * V;  // first entry of this summary vector in its row
            if (MULTI) {
                if (filt && !((P.class_mask[c >> 5] >> (c & 31)) & 1u)) continue;
            } else {
                for (int cc = 1; cc < nc; ++cc) {
                    ScoreVec<T> o;
                    o.raw = __ldg(reinterpret_cast<const uint4*>(smax + (size_t)cc * SNV + j0));
#pragma unroll
                    for (int k = 0; k < V; ++k)
                        if (to_f32<T>(o.e[k]) > to_f32<T>(m[u].e[k])) m[u].e[k] = o.e[k];
                }
            }
            unsigned hm = range_hits<T>(m[u], sb_lo, 0x7F800000u, rb_any);
            if (j0 + V > NV) hm &= (1u << (NV - j0)) - 1u;  // row padding
            h[u] = hm;
            ebase[u] = c * NV + j0;
            cnt += __popc(hm);
        }
        if (WITH_SCORES) {
            unsigned pos = warp_reserve(nhits, cnt);
#pragma unroll
            for (int u = 0; u < SCAN_UNROLL; ++u)
                // set bits only: most summary vectors list nothing, and with 2 CTAs per SM this phase is bound by issue
                for (unsigned hm = h[u]; hm; hm &= hm - 1u) {
                    if (pos < NMS_BINS) hits[pos] = ebase[u] + (unsigned)(__ffs(hm) - 1);
                    ++pos;
                }
        } else {
#pragma unroll
            for (int u = 0; u < SCAN_UNROLL; ++u)
#pragma unroll
                for (int k = 0; k < V; ++k)
                    if ((h[u] >> k) & 1u) {
                        const unsigned sbm = make_sbits(to_f32<T>(m[u].e[k]));
                        if (sbm <= sb_hi) f(sbm, 0, 0);
                    }
        }
    }
    if (!WITH_SCORES) return true;
    PROFX(12);  // collect: pass 1 (this thread)
    __syncthreads();
    const unsigned nh = *nhits;
    __syncthreads();
    PROFX(13);  // collect: wait for the block
    PROF_GADD(18, nh);
    if (nh > NMS_BINS) return false;  // dense: not worth (and not possible) to list
    // ---- pass 2: the listed score vectors
    if (MULTI) {
        for (unsigned ib = 0; ib < nh; ib += NMS_THREADS * SCAN_UNROLL) {
            const unsigned i0 = ib + threadIdx.x;
            ScoreVec<T> v[SCAN_UNROLL];
            unsigned e_[SCAN_UNROLL];
#pragma unroll
            for (int u = 0; u < SCAN_UNROLL; ++u) {
                e_[u] = hits[min(i0 + u * NMS_THREADS, nh - 1u)];  // clamped: unconditional loads, as in pass 1
                const unsigned c = e_[u] / NV;
                v[u].raw = __ldg(reinterpret_cast<const uint4*>(sc + (size_t)c * A + (size_t)(e_[u] - c * NV) * V));
            }
            unsigned hv[SCAN_UNROLL], cnt = 0;
#pragma unroll
            for (int u = 0; u < SCAN_UNROLL; ++u) {
                hv[u] = 0;
                const unsigned i = i0 + u * NMS_THREADS;
                if (i >= nh) continue;
                unsigned hm = range_hits<T>(v[u], sb_lo, sb_hi, rb);
                if (hm && ((unsigned)lo | (unsigned)hi)) {  // bounds not digit-aligned (refinement): full key compare
                    const unsigned c = e_[u] / NV, a_s = (e_[u] - c * NV) * V;
#pragma unroll
                    for (int k = 0; k < V; ++k)
                        if ((hm >> k) & 1u) {
                            const u64 key = make_key(make_sbits(to_f32<T>(v[u].e[k])), (a_s + k) * (unsigned)nc + c);
                            if (!(key >= lo && key < hi)) hm &= ~(1u << k);
                        }
                }
                hv[u] = hm;
                cnt += __popc(hm);
            }
            unsigned pos = warp_reserve(counter, cnt);
#pragma unroll
            for (int u = 0; u < SCAN_UNROLL; ++u) {
                if (!hv[u]) continue;
                const unsigned c = e_[u] / NV, a_s = (e_[u] - c * NV) * V;
#pragma unroll
                for (int k = 0; k < V; ++k)
                    if ((hv[u] >> k) & 1u) {
                        if (pos < NMS_CAP) keys[pos] = make_key(make_sbits(to_f32<T>(v[u].e[k])), (a_s + k) * (unsigned)nc + c);
                        ++pos;
                    }
            }
        }
    } else {
        for (unsigned ib = 0; ib < nh; ib += NMS_THREADS) {
            const unsigned i = ib + threadIdx.x;
            u64 mykeys[V];
            unsigned cnt = 0;
            if (i < nh) {
                const unsigned a_s = hits[i] * V;
                const uint4* __restrict__ col = reinterpret_cast<const uint4*>(sc + a_s);
                const size_t rowv = (size_t)A / V;
                float best[V];
                int bc[V];
#pragma unroll
                for (int k = 0; k < V; ++k) { best[k] = -INFINITY; bc[k] = 0; }
                int cc = 0;
                for (; cc + SCAN_UNROLL <= nc; cc += SCAN_UNROLL) {
                    ScoreVec<T> v[SCAN_UNROLL];
#pragma unroll
                    for (int u = 0; u < SCAN_UNROLL; ++u) v[u].raw = __ldg(col + (size_t)(cc + u) * rowv);
#pragma unroll
                    for (int u = 0; u < SCAN_UNROLL; ++u)
#pragma unroll
                        for (int k = 0; k < V; ++k) {
                            const float sv = to_f32<T>(v[u].e[k]);
                            if ((cc + u) == 0 || sv > best[k]) { best[k] = sv; bc[k] = cc + u; }  // lowest index wins ties
                        }
                }
                for (; cc < nc; ++cc) {
                    ScoreVec<T> v1;
                    v1.raw = __ldg(col + (size_t)cc * rowv);
#pragma unroll
                    for (int k = 0; k < V; ++k) {
                        const float sv = to_f32<T>(v1.e[k]);
                        if (cc == 0 || sv > best[k]) { best[k] = sv; bc[k] = cc; }
                    }
                }
#pragma unroll
                for (int k = 0; k < V; ++k) {
                    mykeys[k] = 0ull;
                    const unsigned sb = make_sbits(best[k]);
                    if (sb - sb_lo <= sb_hi - sb_lo) {
                        if (filt && !((P.class_mask[bc[k] >> 5] >> (bc[k] & 31)) & 1u)) continue;
                        const u64 key = make_key(sb, (a_s + k) * (unsigned)nc + (unsigned)bc[k]);
                        if (key >= lo && key < hi) { mykeys[k] = key; ++cnt; }
                    }
                }
            } else {
#pragma unroll
                for (int k = 0; k < V; ++k) mykeys[k] = 0ull;
            }
            unsigned pos = warp_reserve(counter, cnt);
#pragma unroll
            for (int k = 0; k < V; ++k)
                if (mykeys[k]) {
                    if (pos < NMS_CAP) keys[pos] = mykeys[k];
                    ++pos;
                }
        }
    }
    PROFX(14);  // collect: pass 2 (this thread)
    return true;
}

__device__ __forceinline__ int level_shift(int lvl) { return lvl < 5 ? 52 - 12 * lvl : 0; }
__device__ __forceinline__ unsigned level_digit(u64 key, int lvl) {
    return lvl < 5 ? (unsigned)(key >> (52 - 12 * lvl)) & 0xFFFu : (unsigned)key & 0xFu;
}

// in-place: h[d] (counts) -> G[d] = sum_{d' >= d} h[d'], G[NMS_BINS] = 0.  All threads call.
__device__ void suffix_scan(unsigned* h, unsigned* warp_tot) {
    constexpr int PER = NMS_BINS / NMS_THREADS;  // 8
    const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
    // thread t owns reversed positions r in [PER*t, PER*t+PER), bin = NMS_BINS-1-r
    unsigned v[PER], sum = 0;
#pragma unroll
    for (int i = 0; i < PER; ++i) { v[i] = h[NMS_BINS - 1 - (PER * t + i)]; sum += v[i]; }
    unsigned inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned n = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += n;
    }
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    unsigned base = 0;
    for (int w = 0; w < wid; ++w) base += warp_tot[w];
    unsigned run = base + inc - sum;
#pragma unroll
    for (int i = 0; i < PER; ++i) { run += v[i]; h[NMS_BINS - 1 - (PER * t + i)] = run; }
    if (t == 0) h[NMS_BINS] = 0;
    __syncthreads();
}

// largest digit d in [0, hi) with G[d] - base >= need   (G non-increasing in d; caller guarantees G[0]-base >= need)
__device__ __forceinline__ int find_digit(const unsigned* G, int hi, unsigned base, unsigned need) {
    int lo = 0, up = hi;  // invariant: G[lo]-base >= need ; (up == hi or G[up]-base < need)
    while (up - lo > 1) {
        const int mid = (lo + up) >> 1;
        if (G[mid] - base >= need) lo = mid; else up = mid;
    }
    return lo;
}

// Bitonic sort (descending) of E * NMS_THREADS 64-bit keys held in shared memory.  Element i = e * 512 + tid
// lives in register e of thread tid: partners at distance j < 32 are reached with warp shuffles, at
// 32 <= j < 512 through shared memory, at j >= 512 inside the thread -- 10 block barriers pairs instead
// of one per network stage.
template <int E> __device__ __forceinline__ void block_sort_desc(u64* keys) {
    const unsigned tid = threadIdx.x;
    u64 r[E];
#pragma unroll
    for (int e = 0; e < E; ++e) r[e] = keys[e * NMS_THREADS + tid];
    for (unsigned k = 2; k <= (unsigned)E * NMS_THREADS; k <<= 1) {
        for (unsigned j = k >> 1; j > 0; j >>= 1) {
            if (j >= NMS_THREADS) {
                const int je = j / NMS_THREADS;
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const int pe = e ^ je;
                    if (pe > e) {
                        const unsigned i = e * NMS_THREADS + tid;
                        const bool desc = ((i & k) == 0);
                        const u64 x = r[e], y = r[pe];
                        if (desc ? (x < y) : (x > y)) { r[e] = y; r[pe] = x; }
                    }
                }
            } else if (j >= 32) {
                __syncthreads();
#pragma unroll
                for (int e = 0; e < E; ++e) keys[e * NMS_THREADS + tid] = r[e];
                __syncthreads();
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const unsigned i = e * NMS_THREADS + tid;
                    const u64 y = keys[i ^ j];
                    const bool lower = (i & j) == 0;          // i < partner
                    const bool desc = ((i & k) == 0);
                    const bool take_max = (lower == desc);    // this slot keeps the larger key
                    const u64 x = r[e];
                    r[e] = take_max ? (x > y ? x : y) : (x < y ? x : y);
                }
            } else {
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const unsigned i = e * NMS_THREADS + tid;
                    const u64 x = r[e];
                    const u64 y = __shfl_xor_sync(0xffffffffu, x, j);
                    const bool lower = (i & j) == 0;
                    const bool desc = ((i & k) == 0);
                    const bool take_max = (lower == desc);
                    r[e] = take_max ? (x > y ? x : y) : (x < y ? x : y);
                }
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int e = 0; e < E; ++e) keys[e * NMS_THREADS + tid] = r[e];
    __syncthreads();
}

__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned ld_relaxed_sys(const unsigned* p) {
    unsigned v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// MINB = CTAs per SM the registers are budgeted for: 2 (64 registers; needed when there are more segments than SMs) or
// 1 (128 registers, no spills: 26 % faster per segment, used when every segment gets an SM of its own -- cerb_launch_nms)
template <typename T, bool MULTI, int MINB>
__global__ void __launch_bounds__(NMS_THREADS, MINB) nms_kernel(const __grid_constant__ NmsParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    NmsSmem& S = *reinterpret_cast<NmsSmem*>(smem_raw);

    // a kernel launched behind this one with the programmatic attribute (the NEXT batch's decode in the single-stream
    // overlapped schedule) may start as soon as every CTA of this grid is running
    asm volatile("griddepcontrol.launch_dependents;");
    if ((int)blockIdx.x >= P.T * P.B) {
        // The launch's extra CTAs (only present with a piggyback delivery descriptor): this rank's side of the delivery of
        // an earlier batch, beside the segment CTAs and on nobody's critical path.
        const int d = (int)blockIdx.x - P.T * P.B;  // 0 .. P.deliver_ctas - 1
        if (P.push_src != nullptr) {
            // writer: push the PREVIOUS batch (complete in local staging since the previous launch) into rank dst's slot
            // with 128-bit stores, then publish the slot's new batch count in dst's flag word: every delivery CTA orders
            // its stores before its count at GPU scope, the last one releases at system scope (the NVLink round trips
            // of the fences are paid by these CTAs only, ~10 us into a ~50 us kernel).  dst must have taken the batch
            // that was in the slot (never spins in steady state; bounded: a lost peer must not hang the GPU).
            if (threadIdx.x == 0) {
                const unsigned need = *reinterpret_cast<volatile unsigned*>(P.deliver_seq);
                for (unsigned spins = 0; ld_relaxed_sys(P.deliver_ack) < need && spins < 8000000u; ++spins) __nanosleep(256);
            }
            __syncthreads();
            const float4* __restrict__ src = reinterpret_cast<const float4*>(P.push_src);
            float4* __restrict__ dst4 = reinterpret_cast<float4*>(P.push_dst);
            for (unsigned i = (unsigned)d * NMS_THREADS + threadIdx.x; i < P.push_words / 4; i += (unsigned)P.deliver_ctas * NMS_THREADS)
                dst4[i] = src[i];
            __syncthreads();
            if (threadIdx.x == 0) {
                __threadfence();
                if (atomicAdd(P.deliver_done, 1u) == (unsigned)P.deliver_ctas - 1u) {
                    __threadfence();
                    *reinterpret_cast<volatile unsigned*>(P.deliver_done) = 0u;
                    const unsigned n = *reinterpret_cast<volatile unsigned*>(P.deliver_seq) + 1u;
                    *reinterpret_cast<volatile unsigned*>(P.deliver_seq) = n;
                    st_release_sys(P.deliver_flag, n);
                }
            }
        }
        if (P.col_flags != nullptr && d == 0) {
            // rank dst: take the batch the other ranks pushed during the previous step and acknowledge it (one thread per
            // rank); a late writer delays this CTA only
            const int r = threadIdx.x;
            const unsigned need = *reinterpret_cast<volatile unsigned*>(P.col_collected) + 1u;
            if (r < P.col_world && r != P.col_dst) {
                for (unsigned spins = 0; ld_relaxed_sys(P.col_flags + r) < need && spins < 8000000u; ++spins) __nanosleep(256);
                (void)ld_acquire_sys(P.col_flags + r);
                st_release_sys(P.col_ack[r], need);
            }
            __syncthreads();
            if (r == 0) *reinterpret_cast<volatile unsigned*>(P.col_collected) = need;
        }
        return;
    }
    BLOCK_T_START
    const int seg = blockIdx.x;
    const int task = seg / P.B, b = seg - task * P.B;
    const int nc = P.nc[task], A = P.A;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const T* __restrict__ img = reinterpret_cast<const T*>(P.pred[task]) + (size_t)b * (4 + nc) * A;
    float* __restrict__ dets = P.dets + (size_t)seg * P.max_det * 6;
    const float thr = P.conf_thr, iou_thr = P.iou_thr;
    const int max_det = P.max_det;
    const unsigned cap = (unsigned)P.chunk_cap;

    float4* kbox = S.kbox;
    float* karea = S.karea;
    if (max_det > NMS_KEPT_SMEM) {
        float* ws = P.kept_ws + (size_t)seg * max_det * 5;
        kbox = reinterpret_cast<float4*>(ws);
        karea = ws + (size_t)max_det * 4;
    }
    // Class shortcut.  Boxes are offset by class * max_wh before NMS (general.py:462-463), so two boxes
    // of different classes whose un-offset corners all lie in the window [tame_lo, tame_hi) of width
    // max_wh can never intersect (the host checked that the fp32 offsets are exact, P.class_shortcut).
    // While every box involved is such a "tame" box, a candidate is only tested against the kept /
    // earlier boxes of its own class, found through per-class chains; one wild box anywhere (or
    // agnostic mode, or a kept list too large for shared memory) switches to testing all pairs.
    const bool shortcut = P.class_shortcut != 0 && max_det <= NMS_KEPT_SMEM;
    bool kept_wild = false;
    for (int i = tid; i < NMS_BUCKETS; i += NMS_THREADS) S.khead[i] = -1;
    if (tid == 0) S.kept_wild = 0;

    // ---------------- level-0 histogram (top 12 key bits).  For large multi-label segments it is an
    // ESTIMATE built from every hstride-th score vector: chunk boundaries only steer how much is
    // gathered at once; what a chunk contains, its order and every count that matters (collect)
    // are exact.  A chunk that turns out too large switches the segment to the exact histogram.
    PROF_DECL
    const unsigned max_nms = (unsigned)max(P.max_nms, 0);
    const T* __restrict__ smax =
        P.smax[task] ? reinterpret_cast<const T*>(P.smax[task]) + (size_t)b * nc * summary_row_len<T>(A) : nullptr;
    unsigned hstride = 1;  // > 1: the histogram is a 1/hstride sample
    if (!smax && MULTI && P.hist_sample > 1) {
        const u64 nvec = ((u64)nc * (u64)A) / ScoreVec<T>::V;
        if (nvec >= 8192 && (A % ScoreVec<T>::V) == 0) hstride = (unsigned)P.hist_sample;
    }
    bool exact = (hstride == 1) && !smax;  // histogram counts every candidate
    bool summary_dense = false;
    auto build_hist = [&](unsigned stride, unsigned below_digit) {
        for (int i = tid; i < NMS_BINS; i += NMS_THREADS) S.g0[i] = 0;
        __syncthreads();
        for_each_candidate<T, MULTI>(img, nc, A, thr, P, [&](unsigned sb, int, int) {
            atomicAdd(&S.g0[sb >> 20], 1u);
        }, 0u, below_digit >= 2048u ? 0x7F800000u : (below_digit << 20) - 1u, stride);
        __syncthreads();
        suffix_scan(S.g0, S.warp_tot);
    };
    // with a score summary the histogram counts score VECTORS by their maximum: a lower bound on the candidates
    // of every digit range (each vector contributes at least its maximum), which is all the chunk search needs
    auto build_hist_summary = [&]() {
        for (int i = tid; i < NMS_BINS; i += NMS_THREADS) S.g0[i] = 0;
        __syncthreads();
        for_each_candidate_summary<T, MULTI, false>(img, smax, nc, A, thr, P, [&](unsigned sb, int, int) {
            atomicAdd(&S.g0[sb >> 20], 1u);
        }, 0u, 0x7F800000u, S.g1, &S.nhits);
        __syncthreads();
        suffix_scan(S.g0, S.warp_tot);
    };
    PROF(0);  // setup
    // Programmatic dependent launch: this grid may have been started while the kernel before it in the stream (the
    // decode kernel) was still draining; nothing above touched global memory.  Wait for that kernel's results here.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    // direct delivery (cerb_nms_deliver): the output slot lives in rank dst's memory, and dst must have taken the batch this
    // rank wrote there last time (two batches ago, so this never spins in steady state).  A relaxed load is enough: no
    // data is read on the strength of it, it only gates stores (which are never speculated).  Bounded: a lost peer
    // must not hang the GPU.
    if (P.deliver_flag != nullptr && P.push_src == nullptr && tid == 0) {
        const unsigned need = *reinterpret_cast<volatile unsigned*>(P.deliver_seq);
        for (unsigned spins = 0; ld_relaxed_sys(P.deliver_ack) < need && spins < 8000000u; ++spins) __nanosleep(256);
    }
    // (every path below passes a __syncthreads before the first store to dets)
    if (smax) build_hist_summary(); else build_hist(hstride, NMS_BINS);
    PROF(1);  // first histogram

    unsigned consumed = 0;
    int kept = 0;
    unsigned target = min((unsigned)max(P.chunk_first, 1), cap);
    unsigned npairs = 0;  // IoU tests made by this thread (reported per segment when P.pair_counts is set)

    // -------- consume the sorted chunk in S.keys[0..n) (first `take` entries) ; returns updated kept
    auto consume_chunk = [&](unsigned n, unsigned take) {
        // bitonic sort, descending, padded with zeros (keys are never 0); see block_sort_desc
        {
            unsigned n2 = NMS_THREADS;
            while (n2 < n) n2 <<= 1;
            for (unsigned i = n + tid; i < n2; i += NMS_THREADS) S.keys[i] = 0ull;
            __syncthreads();
            switch (n2 / NMS_THREADS) {
                case 1: block_sort_desc<1>(S.keys); break;
                case 2: block_sort_desc<2>(S.keys); break;
                case 4: block_sort_desc<4>(S.keys); break;
                default: block_sort_desc<8>(S.keys); break;
            }
        }
        PROF(3);  // sort
        // tiles: one candidate per thread
        for (unsigned t0 = 0; t0 < take && kept < max_det; t0 += NMS_TILE) {
            const int nt = (int)min((unsigned)NMS_TILE, take - t0);
            // A: materialise the tile's boxes  (general.py:443 xywh2xyxy in dtype, :462-463 class offset in fp32)
            float4 raw = make_float4(0.f, 0.f, 0.f, 0.f), box = raw;
            float area = 0.f, score = 0.f;
            int cls = 0, code = -1;
            bool dead = true;
            if (tid == 0) S.tile_wild = 0;
            PROF_COUNT(17, 1);
            __syncthreads();
            if (tid < nt) {
                const u64 key = S.keys[t0 + tid];
                const unsigned idx = 0xFFFFFFFFu - (unsigned)key;
                const int a = idx / nc;
                cls = idx - a * nc;
                const float cx = to_f32<T>(__ldg(img + a));
                const float cy = to_f32<T>(__ldg(img + (size_t)A + a));
                const float bw = to_f32<T>(__ldg(img + (size_t)2 * A + a));
                const float bh = to_f32<T>(__ldg(img + (size_t)3 * A + a));
                const float hw_ = rnd<T>(bw * 0.5f), hh_ = rnd<T>(bh * 0.5f);
                raw.x = rnd<T>(__fsub_rn(cx, hw_));
                raw.y = rnd<T>(__fsub_rn(cy, hh_));
                raw.z = rnd<T>(__fadd_rn(cx, hw_));
                raw.w = rnd<T>(__fadd_rn(cy, hh_));
                const float off = __fmul_rn((float)cls, P.class_gap);
                box.x = __fadd_rn(raw.x, off);
                box.y = __fadd_rn(raw.y, off);
                box.z = __fadd_rn(raw.z, off);
                box.w = __fadd_rn(raw.w, off);
                area = __fmul_rn(__fsub_rn(box.z, box.x), __fsub_rn(box.w, box.y));
                score = __uint_as_float((unsigned)(key >> 32));
                const float lo = P.tame_lo, hi = P.tame_hi;
                const bool tame = raw.x >= lo && raw.y >= lo && raw.z >= lo && raw.w >= lo &&
                                  raw.x < hi && raw.y < hi && raw.z < hi && raw.w < hi;
                code = tame ? cls : -1;
                if (!tame) S.tile_wild = 1;
                dead = false;
            }
            S.tbox[tid] = box;
            S.tarea[tid] = area;
            S.tcode[tid] = dead ? -2 : code;  // -2: padding, never equal to a class
            __syncthreads();
            PROF(4);  // tile A (gather)
            // Per-class chains are valid while every box involved is tame (see the class shortcut above).
            const bool fast = shortcut && !S.tile_wild && !kept_wild;
            int prev = -1;
            if (fast && !dead) {  // previous candidate of the same class inside the tile
                int p = tid - 1;
                while (p >= 0 && S.tcode[p] != code) --p;
                prev = p;
            }
            S.tprev[tid] = prev;
            // B: against the kept list
            if (!dead && kept > 0) {
                if (fast) {
                    for (int k = S.khead[cls & (NMS_BUCKETS - 1)]; k >= 0; k = S.knext_s[k]) {
                        ++npairs;
                        if (suppresses(kbox[k], karea[k], box, area, iou_thr)) { dead = true; break; }
                    }
                } else {
                    for (int k = 0; k < kept; ++k) {
                        ++npairs;
                        if (suppresses(kbox[k], karea[k], box, area, iou_thr)) { dead = true; break; }
                    }
                }
            }
            S.tdead[tid] = dead ? 1 : 0;
            __syncthreads();
            PROF(5);  // tile B (prev chain + kept list)
            // C: m[w] = bits of the earlier candidates i in word w (alive) that would suppress this one
            u64 m0 = 0, m1 = 0, m2 = 0, m3 = 0, m4 = 0, m5 = 0, m6 = 0, m7 = 0;
#define NMS_SETBIT(i)                                        \
    do {                                                     \
        const u64 bit_ = 1ull << ((i) & 63);                 \
        switch ((i) >> 6) {                                  \
            case 0: m0 |= bit_; break;                       \
            case 1: m1 |= bit_; break;                       \
            case 2: m2 |= bit_; break;                       \
            case 3: m3 |= bit_; break;                       \
            case 4: m4 |= bit_; break;                       \
            case 5: m5 |= bit_; break;                       \
            case 6: m6 |= bit_; break;                       \
            default: m7 |= bit_; break;                      \
        }                                                    \
    } while (0)
            if (!dead) {
                if (fast) {
                    for (int i = prev; i >= 0; i = S.tprev[i]) {
                        if (!S.tdead[i]) {
                            ++npairs;
                            if (suppresses(S.tbox[i], S.tarea[i], box, area, iou_thr)) NMS_SETBIT(i);
                        }
                    }
                } else {
                    for (int i = 0; i < tid; ++i) {
                        if (!S.tdead[i]) {
                            ++npairs;
                            if (suppresses(S.tbox[i], S.tarea[i], box, area, iou_thr)) NMS_SETBIT(i);
                        }
                    }
                }
            }
            {
                const unsigned al = __ballot_sync(0xffffffffu, !dead);
                if (lane == 0) S.keep32[0][wid] = al;
            }
            __syncthreads();
            PROF(6);  // tile C (pairwise)
            // D: greedy result as the fixpoint of  keep[j] = alive[j] && no kept earlier i suppresses j.
            //    It is unique (keep[j] depends only on lower indices).  Every block round lets each warp
            //    settle its own 32 candidates to their fixpoint given the other warps' current words, so
            //    after round r the first r warps are final: <= 16 rounds, in practice 2-3.
            int cur = 0;
            {
                const int myw = wid >> 1;          // 64-bit word holding this warp's 32 candidates
                const bool upper = (wid & 1) != 0; // which half of it
                const u64 mw[NMS_TILE_WORDS] = {m0, m1, m2, m3, m4, m5, m6, m7};
                u64 mown = 0ull;
#pragma unroll
                for (int w = 0; w < NMS_TILE_WORDS; ++w)
                    if (w == myw) mown = mw[w];
                for (;;) {
                    const unsigned* K = S.keep32[cur];
                    u64 others = 0ull;
#pragma unroll
                    for (int w = 0; w < NMS_TILE_WORDS; ++w)
                        if (w != myw) others |= mw[w] & (((u64)K[2 * w + 1] << 32) | (u64)K[2 * w]);
                    const unsigned sibling = K[wid ^ 1];
                    unsigned mine = K[wid];
#ifdef NMS_PROFILE
                    const long long settle_t0 = clock64();
                    unsigned settle_it = 0;
#endif
                    for (;;) {  // warp-local settle
                        const u64 own = upper ? (((u64)mine << 32) | (u64)sibling) : (((u64)sibling << 32) | (u64)mine);
                        const bool kj = !dead && (others | (mown & own)) == 0ull;
                        const unsigned nw = __ballot_sync(0xffffffffu, kj);
#ifdef NMS_PROFILE
                        ++settle_it;
#endif
                        if (nw == mine) break;
                        mine = nw;
                    }
#ifdef NMS_PROFILE
                    if (lane == 0) {  // [21] settle iterations, [22] settle cycles: summed over the warps of the block
                        atomicAdd(&g_nms_prof[21], (unsigned long long)settle_it);
                        atomicAdd(&g_nms_prof[22], (unsigned long long)(clock64() - settle_t0));
                    }
#endif
                    int changed = 0;
                    if (lane == 0) { S.keep32[cur ^ 1][wid] = mine; changed = (mine != K[wid]); }
                    cur ^= 1;
#ifdef NMS_PROFILE
                    if (tid == 0) prof_acc[15] += 1;  // fixpoint block rounds
#endif
                    if (!__syncthreads_or(changed)) break;
                }
            }
            PROF(7);  // tile D (fixpoint)
            // E: the first `budget` kept candidates (greedy stops at max_det, general.py:465) are appended,
            //    in order, to the kept list and to the output
            {
                const unsigned* K = S.keep32[cur];
                int before = 0, total = 0;
#pragma unroll
                for (int w = 0; w < NMS_THREADS / 32; ++w) {
                    const int c = __popc(K[w]);
                    if (w < wid) before += c;
                    total += c;
                }
                const bool mine = (K[wid] >> lane) & 1u;
                const int pos = kept + before + __popc(K[wid] & ((1u << lane) - 1u));
                if (mine && pos < max_det) {
                    kbox[pos] = box;
                    karea[pos] = area;
                    float* o = dets + (size_t)pos * 6;  // general.py:474 rows (x1,y1,x2,y2,conf,cls)
                    o[0] = raw.x; o[1] = raw.y; o[2] = raw.z; o[3] = raw.w;
                    o[4] = score;
                    o[5] = (float)cls;
                    if (code < 0) S.kept_wild = 1;
                    if (max_det <= NMS_KEPT_SMEM) {  // chain the box into its class bucket (any order is fine)
                        const int old = atomicExch(&S.khead[cls & (NMS_BUCKETS - 1)], pos);
                        S.knext_s[pos] = old;
                    }
                }
                kept = min(kept + total, max_det);
            }
            __syncthreads();
            kept_wild = kept_wild || (S.kept_wild != 0);
            PROF(8);  // tile E (append)
        }
    };

    // -------- gather the keys in [lo, hi) into S.keys ; returns count (uniform)
    auto collect = [&](u64 lo, u64 hi) -> unsigned {
        if (tid == 0) S.counter = 0;
        __syncthreads();
        const unsigned sb_lo = (unsigned)(lo >> 32), sb_hi = (unsigned)((hi - 1) >> 32);
        auto put = [&](unsigned sb, int a, int c) {
            const u64 key = make_key(sb, (unsigned)(a * nc + c));
            if (key >= lo && key < hi) {
                const unsigned p = atomicAdd(&S.counter, 1u);
                if (p < NMS_CAP) S.keys[p] = key;
            }
        };
        bool done = false;
        if (smax && !summary_dense)
            done = for_each_candidate_summary<T, MULTI, true>(img, smax, nc, A, thr, P, put, sb_lo, sb_hi, S.g1, &S.nhits,
                                                              lo, hi, S.keys, &S.counter);
        PROF_COUNT(16, 1);
        if (!done) {
            PROF_COUNT(19, 1);
            summary_dense = true;  // candidates are dense in this segment: the plain scan is the better tool
            for_each_candidate<T, MULTI>(img, nc, A, thr, P, put, sb_lo, sb_hi);
        }
        __syncthreads();
        const unsigned n = S.counter;
        __syncthreads();
        PROF(2);  // collect (and chunk search before it)
        return n;
    };

    // -------- a level-0 bin that alone exceeds the chunk capacity: refine by deeper digits
    auto overflow_bin = [&](int bin) {
        const u64 lowlim = (u64)bin << 52;
        u64 bnd = (u64)(bin + 1) << 52;
        while (consumed < max_nms && kept < max_det) {
            u64 lo = lowlim, hi = bnd, L = lowlim;
            int lvl = 1;
            bool empty = false;
            for (;;) {
                for (int i = tid; i < NMS_BINS; i += NMS_THREADS) S.g1[i] = 0;
                __syncthreads();
                const unsigned sb_lo = (unsigned)(lo >> 32), sb_hi = (unsigned)((hi - 1) >> 32);
                for_each_candidate<T, MULTI>(img, nc, A, thr, P, [&](unsigned sb, int a, int c) {
                    const u64 key = make_key(sb, (unsigned)(a * nc + c));
                    if (key >= lo && key < hi) atomicAdd(&S.g1[level_digit(key, lvl)], 1u);
                }, sb_lo, sb_hi);
                __syncthreads();
                suffix_scan(S.g1, S.warp_tot);
                const unsigned tot = S.g1[0];
                if (tot == 0) { empty = true; break; }
                if (tot <= cap) { L = lo; break; }
                const unsigned need = min(cap, max_nms - consumed);
                const int nb = lvl < 5 ? NMS_BINS : 16;
                const int sh = level_shift(lvl);
                const u64 parent = lvl < 5 ? (lo >> (sh + 12)) << (sh + 12) : (lo >> 4) << 4;
                const int d = find_digit(S.g1, nb, 0u, min(need, tot));
                const unsigned cnt = S.g1[d];
                if (cnt <= cap) { L = parent | ((u64)d << sh); break; }
                const unsigned c1 = S.g1[d + 1];
                if (c1 > 0) { L = parent | ((u64)(d + 1) << sh); break; }
                const u64 blo = parent | ((u64)d << sh);
                const u64 bhi = blo + (1ull << sh);
                lo = lo > blo ? lo : blo;
                hi = hi < bhi ? hi : bhi;
                ++lvl;
                __syncthreads();
            }
            __syncthreads();
            if (empty) return;
            if (L < lowlim) L = lowlim;
            const unsigned n = collect(L, bnd);
            const unsigned take = min(n, max_nms - consumed);
            consume_chunk(n, take);
            consumed += take;
            bnd = L;
            if (L == lowlim) return;
        }
    };

    // ---------------- main loop over level-0 digit ranges, from the top
    int hi0 = NMS_BINS / 2;  // float sign bit is 0: digits < 2048, so (hi0 << 52) never overflows
    while (hi0 > 0 && consumed < max_nms && kept < max_det) {
        const unsigned base = S.g0[hi0];
        const unsigned rem_s = S.g0[0] - base;  // candidates left below hi0, in histogram units
        if (exact && rem_s == 0) break;
        unsigned need = min(target, max_nms - consumed);
        // an estimating histogram (summary: a lower bound; sample: noisy) must leave head-room below the capacity,
        // or the gather overflows and the segment pays for an exact histogram
        if (!exact) need = min(need, cap - cap / 4 - cap / 8);
        const unsigned need_s = hstride == 1 ? need : (need + need / 4 + hstride - 1) / hstride;  // sample: +25% margin
        int lo0 = 0;
        bool single_heavy = false;
        if (rem_s > need_s) {
            const int d = find_digit(S.g0, hi0, base, need_s);
            lo0 = d;
            const unsigned est = (S.g0[d] - base) * hstride;
            if (est > (exact ? cap : cap - cap / 4)) {
                if (S.g0[d + 1] - base > 0) lo0 = d + 1;
                else single_heavy = exact;  // exact: digit d alone exceeds the capacity
            }
        }
        if (single_heavy) {
            overflow_bin(lo0);
            hi0 = lo0;
            target = cap;
            continue;
        }
        const unsigned n = collect((u64)lo0 << 52, (u64)hi0 << 52);
        if (n > cap) {
            // estimate was off (or ties piled up): count exactly what is left and retry
            PROF_COUNT(20, 1);
            build_hist(1u, (unsigned)hi0);
            hstride = 1;
            exact = true;
            continue;
        }
        const unsigned take = min(n, max_nms - consumed);
        consume_chunk(n, take);
        consumed += take;
        hi0 = lo0;
        // next chunk: as many candidates as the keep rate seen so far says are needed to fill max_det (+25 %),
        // at least double, at most the capacity
        {
            const unsigned missing = (unsigned)max(max_det - kept, 0);
            const unsigned long long want = (unsigned long long)missing * consumed / (unsigned)max(kept, 1);
            const unsigned adaptive = (unsigned)min(want + want / 4ull + 64ull, (unsigned long long)cap);
            target = min(max(adaptive, min(target * 2u, cap)), cap);
        }
    }

    if (tid == 0) P.counts[seg] = kept;
    if (P.pair_counts != nullptr) {  // statistics for bench.py / profiles: IoU tests and candidates consumed, per segment
        unsigned v = npairs;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        __syncthreads();
        if (lane == 0) S.warp_tot[wid] = v;
        __syncthreads();
        if (tid == 0) {
            unsigned long long tot = 0;
            for (int w = 0; w < NMS_THREADS / 32; ++w) tot += S.warp_tot[w];
            P.pair_counts[2 * seg] = tot;
            P.pair_counts[2 * seg + 1] = consumed;
        }
    }
    // rows past the count are zero so the padded [T, B, max_det, 6] output is deterministic without a separate fill
    for (int i = kept * 6 + tid; i < max_det * 6; i += NMS_THREADS) dets[i] = 0.f;
    if (P.deliver_flag != nullptr && P.push_src == nullptr) {
        // direct form: tell rank dst that this rank's batch is complete.  Every CTA orders its stores before its count at GPU scope
        // (fence + atomic = release; the per-CTA fence is the cheap one); the last CTA -- which has observed every count
        // (acquire at GPU scope) -- fences ONCE at system scope and releases the slot's new sequence number into dst's
        // flag.  PTX causality order is transitive across the two scopes, so a reader on dst that acquires the flag sees
        // every CTA's rows.
        __syncthreads();
        if (tid == 0) {
            __threadfence();
            if (atomicAdd(P.deliver_done, 1u) == (unsigned)(P.T * P.B) - 1u) {
                __threadfence();
                *reinterpret_cast<volatile unsigned*>(P.deliver_done) = 0u;
                const unsigned n = *reinterpret_cast<volatile unsigned*>(P.deliver_seq) + 1u;
                *reinterpret_cast<volatile unsigned*>(P.deliver_seq) = n;
                st_release_sys(P.deliver_flag, n);  // (release = system-scope fence + store)
            }
        }
    }
    PROF(9);  // rest
    PROF_FLUSH(consumed);
    BLOCK_T_END
}

// rank dst's side of the peer delivery (cerb_kernels.h: CollectParams)
__global__ void deliver_collect_kernel(const __grid_constant__ CollectParams P) {
    const int r = threadIdx.x;
    const unsigned need = *reinterpret_cast<volatile unsigned*>(P.collected) + 1u;
    if (r < P.world && r != P.dst) {
        // poll with relaxed loads (an acquire load is a load plus a system-scope fence: not something to repeat every
        // 256 ns beside a memory-bound kernel), then acquire once
        for (unsigned spins = 0; ld_relaxed_sys(P.flags + r) < need && spins < 8000000u; ++spins) __nanosleep(256);
        (void)ld_acquire_sys(P.flags + r);
        st_release_sys(P.ack[r], need);
    }
    __syncthreads();
    if (r == 0) *reinterpret_cast<volatile unsigned*>(P.collected) = need;
}
// a writer's side of the peer delivery, off the critical path: the NMS kernel left the padded rows of one batch in LOCAL
// memory; this small kernel pushes them into rank dst's slot over NVLink (128-bit stores) and runs the hand-shake -- wait
// for dst's acknowledgement of the batch that was in the slot, copy, order the stores (GPU-scope release per CTA, one
// system-scope release by the last CTA) and publish the slot's new sequence number in dst's flag word.  The fences'
// NVLink round trips cost this kernel a few microseconds and nobody else anything: it runs beside the next batch's
// decode / NMS kernels.
__global__ void __launch_bounds__(256) deliver_push_kernel(const __grid_constant__ PushParams P) {
    const int tid = threadIdx.x;
    if (tid == 0) {
        const unsigned need = *reinterpret_cast<volatile unsigned*>(P.seq);
        for (unsigned spins = 0; ld_relaxed_sys(P.ack) < need && spins < 8000000u; ++spins) __nanosleep(256);
    }
    __syncthreads();
    const size_t n4 = P.n_words / 4;
    const float4* __restrict__ src = reinterpret_cast<const float4*>(P.src);
    float4* __restrict__ dst = reinterpret_cast<float4*>(P.dst);
    if (P.mode != 2)
        for (size_t i = (size_t)blockIdx.x * blockDim.x + tid; i < n4; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
    __syncthreads();
    if (tid == 0 && P.mode != 1) {
        __threadfence();
        if (atomicAdd(P.done, 1u) == gridDim.x - 1) {
            __threadfence();
            *reinterpret_cast<volatile unsigned*>(P.done) = 0u;
            const unsigned n = *reinterpret_cast<volatile unsigned*>(P.seq) + 1u;
            *reinterpret_cast<volatile unsigned*>(P.seq) = n;
            st_release_sys(P.flag, n);
        }
    }
}
cudaError_t cerb_launch_deliver_push(const PushParams& P, int ctas, cudaStream_t stream) {
    deliver_push_kernel<<<ctas, 256, 0, stream>>>(P);
    return cudaGetLastError();
}

cudaError_t cerb_launch_deliver_collect(const CollectParams& P, cudaStream_t stream) {
    deliver_collect_kernel<<<1, 32, 0, stream>>>(P);
    return cudaGetLastError();
}

size_t cerb_nms_kept_ws_bytes(int T, int B, int max_det) {
    if (max_det <= NMS_KEPT_SMEM) return 0;
    return (size_t)T * B * max_det * 5 * sizeof(float);
}

template <typename T, bool MULTI, int MINB> static cudaError_t launch_nms_t(const NmsParams& P, cudaStream_t stream) {
    const size_t smem = sizeof(NmsSmem);
    cudaError_t e = cudaFuncSetAttribute(nms_kernel<T, MULTI, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    // launched with programmatic stream serialization: the CTAs may be scheduled as soon as every CTA of the previous
    // kernel has started (the decode kernels signal launch_dependents at entry) and block in griddepcontrol.wait until
    // it has completed -- hides the launch latency and the prologue behind the decode kernel's tail
    const bool pdl = P.pdl != 0;
    cudaLaunchConfig_t cfg = {};
    // (+ the delivery CTAs of the piggyback form, see the top of the kernel)
    cfg.gridDim = dim3((unsigned)(P.T * P.B) + (unsigned)P.deliver_ctas);
    cfg.blockDim = dim3(NMS_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, nms_kernel<T, MULTI, MINB>, P);
}

template <typename T, bool MULTI> static cudaError_t launch_nms_v(const NmsParams& P, cudaStream_t stream) {
    // One CTA per (task, image) segment.  With at most one segment per SM the 128-register build runs (config 2:
    // 63.5 -> 47.1 us, config 4: 79.9 -> 70.7 us); with more segments two CTAs must share an SM and the 64-register
    // build is the faster one (config 3, 192 segments: 59.4 vs 69.6 us) -- profiles/r01_nms.md
    int minb = 2, dev = 0, sms = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess &&
        P.T * P.B <= sms)
        minb = 1;
    if (P.force_minb) minb = P.force_minb == 1 ? 1 : 2;  // tests and tools
    return minb == 1 ? launch_nms_t<T, MULTI, 1>(P, stream) : launch_nms_t<T, MULTI, 2>(P, stream);
}

cudaError_t cerb_launch_nms(const NmsParams& P, int dtype, cudaStream_t stream) {
    if (P.T * P.B == 0) return cudaSuccess;
    // multi_label &= nc > 1 (general.py:419): with nc == 1 both modes select the same candidates
    const bool multi = P.multi_label != 0;
    if (dtype == CERB_DTYPE_F16)
        return multi ? launch_nms_v<__half, true>(P, stream) : launch_nms_v<__half, false>(P, stream);
    if (dtype == CERB_DTYPE_BF16)
        return multi ? launch_nms_v<__nv_bfloat16, true>(P, stream) : launch_nms_v<__nv_bfloat16, false>(P, stream);
    return multi ? launch_nms_v<float, true>(P, stream) : launch_nms_v<float, false>(P, stream);
}
