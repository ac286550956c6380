// Per-class average precision of the validation statistics: ap_per_class (reference utils/metrics.py:56-120) and the
// compute_ap it calls, on the GPU.  The host keeps only the O(nc * 1000) tail (f1, smooth, argmax, the rounded tp/fp).
//
// Work decomposition (all deterministic: no atomics, max / integer sums only):
//   1. ap_key_kernel      dense class of every detection (exact float binary search in the ascending classes; not found
//                         or NaN -> nc, ignored), a 64-bit key (class, order-preserving bits of -conf with -0 folded to
//                         +0), the row index and the tp row packed into a 32-bit mask.
//   2. cub radix sort     stable, on the 32 + bitwidth(nc) bits in use: per class, conf descending, ties by row index --
//                         the reference's per-class subsequence under np.argsort(-conf, kind="stable").
//   3. ap_segment_kernel  class offsets in the sorted order (binary search of the keys) and the class-aligned tiling:
//                         a class of n_c detections owns ceil(n_c / AP_TILE) tiles, so no tile straddles two classes and
//                         a class of any size is spread over as many CTAs as it has tiles.
//   4. ap_tile_count      per tile and IoU column: true positives in the tile;
//      ap_tile_base       per (class, column): exclusive scan of those counts over the class's tiles;
//      ap_tile_tpc        per tile: tpc = cumulative true positives of every position (int32 [K, n], the only per-row
//                         array: recall and precision are recomputed from it), and the tile's largest precision;
//      ap_tile_suffix     per (class, column): suffix maximum of those over the class's tiles.
//   5. ap_column_kernel   per (class, column): compute_ap's 101 interpolations in mrec = [0, recall..., 1] against the
//                         precision envelope, then np.trapz's sum in numpy's pairwise order.
//   6. ap_curve_kernel    per (class, point of px): the p and r curves of column 0, np.interp(-px, -conf, ., left=0|1).
//
// Bit-exactness: every float64 value is one IEEE operation of the reference's (recall = tpc / (n_l + eps), precision =
// tpc / position, interpolation slope * (x - xp[j]) + fp[j] without FMA); np.interp's search returns the last knot
// j with xp[j] <= x, which on a non-decreasing knot array is the count of knots <= x minus one, the binary search here.
#include <cub/cub.cuh>

#include "../../include/cerb_post.h"
#include "cerb_common.cuh"

namespace {

constexpr int AP_TILE = 512;       // positions per tile = threads of the tile kernels
constexpr int AP_WARPS_TILE = AP_TILE / 32;
constexpr int AP_SCAN_THREADS = 256;
constexpr int AP_COL_WARPS = 8;    // warps of a (class, column) CTA of ap_column_kernel
constexpr int AP_POINTS = 101;     // compute_ap: x = np.linspace(0, 1, 101)
constexpr int AP_CURVE = 1000;     // px = np.linspace(0, 1, 1000)
constexpr int AP_CURVE_THREADS = 256;

struct ApParams {
    const unsigned long long* keys;  // sorted keys
    const int* rows;                 // sorted row indices (the permutation)
    const unsigned* mask;            // [n] tp rows, bit j = column j
    const long long* n_labels;       // [nc] device copy
    int* tpc;                        // [K, n] cumulative true positives at each sorted position (within its class)
    int* offsets;                    // [nc + 1] first sorted position of each class (offsets[nc] = rows with a class)
    int* tile_first;                 // [nc + 1] first tile of each class (tile_first[nc] = tiles in use)
    int* tile_cnt;                   // [tiles, K] true positives per tile, then the class's count before the tile
    double* tile_max;                // [tiles, K] largest precision in the tile, then the suffix maximum over the class
    double eps;
    double *ap, *p, *r;
    int n, K, nc;
};

struct MaxOp {
    __device__ __forceinline__ double operator()(double a, double b) const { return a > b ? a : b; }
};

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// np.linspace(0, 1, num)[i] == i * (1.0 / (num - 1)), with the last point exactly 1.0
__device__ __forceinline__ double linspace01(int i, int num) {
    return i == num - 1 ? 1.0 : __dmul_rn((double)i, __ddiv_rn(1.0, (double)(num - 1)));
}

// -conf as the reference's float32 negation widened to float64, from the sort key (-0.0 comes back as +0.0; the
// interpolations below give the same result for either zero)
__device__ __forceinline__ double key_neg_conf(unsigned long long key) {
    const unsigned u = (unsigned)key;
    return (double)__uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

__global__ void ap_key_kernel(const unsigned char* __restrict__ tp, int K, const float* __restrict__ conf,
                              const float* __restrict__ pred_cls, int n, const float* __restrict__ classes, int nc,
                              unsigned long long* __restrict__ keys, int* __restrict__ rows, unsigned* __restrict__ mask) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float v = pred_cls[i];
        int lo = 0, hi = nc;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (classes[mid] < v) lo = mid + 1; else hi = mid;
        }
        const unsigned c = (lo < nc && classes[lo] == v) ? (unsigned)lo : (unsigned)nc;  // `pred_cls == c`, NaN matches none
        float f = -conf[i];
        if (f == 0.f) f = 0.f;  // numpy compares -0.0 == 0.0: one key for both
        unsigned u = __float_as_uint(f);
        u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);  // ascending -conf = descending conf
        keys[i] = ((unsigned long long)c << 32) | u;
        rows[i] = i;
        const unsigned char* row = tp + (size_t)i * K;
        unsigned m = 0;
        for (int j = 0; j < K; ++j) m |= (row[j] != 0 ? 1u : 0u) << j;
        mask[i] = m;
    }
}

__global__ void __launch_bounds__(1024) ap_segment_kernel(ApParams P) {
    const int n = P.n, nc = P.nc;
    for (int c = threadIdx.x; c <= nc; c += blockDim.x) {
        const unsigned long long want = (unsigned long long)c << 32;
        int lo = 0, hi = n;
        while (lo < hi) {
            const int mid = lo + ((hi - lo) >> 1);
            if (P.keys[mid] < want) lo = mid + 1; else hi = mid;
        }
        P.offsets[c] = lo;
    }
    __syncthreads();
    typedef cub::BlockScan<int, 1024> Scan;
    __shared__ typename Scan::TempStorage tmp;
    int carry = 0;
    for (int base = 0; base < nc; base += 1024) {
        const int c = base + threadIdx.x;
        const int t = c < nc ? (P.offsets[c + 1] - P.offsets[c] + AP_TILE - 1) / AP_TILE : 0;
        int excl, total;
        Scan(tmp).ExclusiveSum(t, excl, total);
        if (c < nc) P.tile_first[c] = carry + excl;
        carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) P.tile_first[nc] = carry;
}

// the class owning tile b < tile_first[nc]: the last c with tile_first[c] <= b
__device__ __forceinline__ int tile_class(const int* tile_first, int nc, int b) {
    int lo = 0, hi = nc;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (tile_first[mid] <= b) lo = mid + 1; else hi = mid;
    }
    return lo - 1;
}

__global__ void __launch_bounds__(AP_TILE) ap_tile_count_kernel(ApParams P) {
    const int b = blockIdx.x;
    if (b >= P.tile_first[P.nc]) return;
    const int c = tile_class(P.tile_first, P.nc, b);
    const int q = P.offsets[c] + (b - P.tile_first[c]) * AP_TILE + threadIdx.x;
    const unsigned m = q < P.offsets[c + 1] ? P.mask[P.rows[q]] : 0u;
    __shared__ int warp_cnt[AP_WARPS_TILE][32];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int j = 0; j < P.K; ++j) {
        const unsigned bal = __ballot_sync(0xffffffffu, (m >> j) & 1u);
        if (lane == j) warp_cnt[w][j] = __popc(bal);
    }
    __syncthreads();
    if (threadIdx.x < P.K) {
        int s = 0;
        for (int v = 0; v < AP_WARPS_TILE; ++v) s += warp_cnt[v][threadIdx.x];
        P.tile_cnt[(size_t)b * P.K + threadIdx.x] = s;
    }
}

__global__ void __launch_bounds__(AP_SCAN_THREADS) ap_tile_base_kernel(ApParams P) {
    const int c = blockIdx.x / P.K, j = blockIdx.x % P.K;
    const int t0 = P.tile_first[c], t1 = P.tile_first[c + 1];
    typedef cub::BlockScan<int, AP_SCAN_THREADS> Scan;
    __shared__ typename Scan::TempStorage tmp;
    int carry = 0;
    for (int base = t0; base < t1; base += AP_SCAN_THREADS) {
        const int b = base + threadIdx.x;
        const int v = b < t1 ? P.tile_cnt[(size_t)b * P.K + j] : 0;
        int excl, total;
        Scan(tmp).ExclusiveSum(v, excl, total);
        if (b < t1) P.tile_cnt[(size_t)b * P.K + j] = carry + excl;
        carry += total;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(AP_TILE) ap_tile_tpc_kernel(ApParams P) {
    const int b = blockIdx.x;
    if (b >= P.tile_first[P.nc]) return;
    const int c = tile_class(P.tile_first, P.nc, b);
    const int off = P.offsets[c];
    const int ql = (b - P.tile_first[c]) * AP_TILE + threadIdx.x;  // position within the class
    const int q = off + ql;
    const bool live = q < P.offsets[c + 1];
    const unsigned m = live ? P.mask[P.rows[q]] : 0u;
    __shared__ int warp_pre[AP_WARPS_TILE][32];
    __shared__ double warp_top[AP_WARPS_TILE][32];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned le = 0xffffffffu >> (31 - lane);
    for (int j = 0; j < P.K; ++j) {
        const unsigned bal = __ballot_sync(0xffffffffu, (m >> j) & 1u);
        if (lane == j) warp_pre[w][j] = __popc(bal);
    }
    __syncthreads();
    if (threadIdx.x < P.K) {  // exclusive scan of the warp counts, plus the class's count before this tile
        int s = P.tile_cnt[(size_t)b * P.K + threadIdx.x];
        for (int v = 0; v < AP_WARPS_TILE; ++v) {
            const int t = warp_pre[v][threadIdx.x];
            warp_pre[v][threadIdx.x] = s;
            s += t;
        }
    }
    __syncthreads();
    const double pos = (double)(ql + 1);
    for (int j = 0; j < P.K; ++j) {
        const unsigned bal = __ballot_sync(0xffffffffu, (m >> j) & 1u);
        const int tpc = warp_pre[w][j] + __popc(bal & le);
        double prec = 0.0;  // the envelope's appended 0 bounds it from below anyway
        if (live) {
            P.tpc[(size_t)j * P.n + q] = tpc;
            prec = __ddiv_rn((double)tpc, pos);
        }
        prec = warp_max(prec);
        if (lane == 0) warp_top[w][j] = prec;
    }
    __syncthreads();
    if (threadIdx.x < P.K) {
        double mx = 0.0;
        for (int v = 0; v < AP_WARPS_TILE; ++v) mx = fmax(mx, warp_top[v][threadIdx.x]);
        P.tile_max[(size_t)b * P.K + threadIdx.x] = mx;
    }
}

__global__ void __launch_bounds__(AP_SCAN_THREADS) ap_tile_suffix_kernel(ApParams P) {
    const int c = blockIdx.x / P.K, j = blockIdx.x % P.K;
    const int t0 = P.tile_first[c], t1 = P.tile_first[c + 1];
    typedef cub::BlockScan<double, AP_SCAN_THREADS> Scan;
    __shared__ typename Scan::TempStorage tmp;
    double carry = 0.0;
    for (int top = t1; top > t0; top -= AP_SCAN_THREADS) {
        const int b = top - 1 - threadIdx.x;  // thread 0 takes the class's last tile
        const double v = b >= t0 ? P.tile_max[(size_t)b * P.K + j] : 0.0;
        double incl, total;
        Scan(tmp).InclusiveScan(v, incl, MaxOp(), total);
        if (b >= t0) P.tile_max[(size_t)b * P.K + j] = fmax(incl, carry);
        carry = fmax(carry, total);
        __syncthreads();
    }
}

struct ClassColumn {
    const int* tpc;        // the class's tpc of this column
    const double* suffix;  // tile_max of the class's first tile, this column (stride K)
    double nl_eps;
    int np, K;
    __device__ __forceinline__ double recall(int q) const { return __ddiv_rn((double)tpc[q], nl_eps); }
    __device__ __forceinline__ double precision(int q) const { return __ddiv_rn((double)tpc[q], (double)(q + 1)); }
    // max(precision[q:]) of the class, by the whole warp (q < np)
    __device__ double suffix_max(int q, int lane) const {
        const int t = q / AP_TILE;
        const int tend = min((t + 1) * AP_TILE, np);
        double m = 0.0;
        for (int k = q + lane; k < tend; k += 32) m = fmax(m, precision(k));
        m = warp_max(m);
        return tend < np ? fmax(m, suffix[(size_t)(t + 1) * K]) : m;
    }
};

// np.interp(x, mrec, mpre) of compute_ap, mrec = [0, recall..., 1], mpre = its precision envelope [1, ..., 0]
__device__ double ap_point(const ClassColumn& cc, double x, int lane) {
    if (x >= 1.0) return 0.0;  // the last knot (mrec = 1) is <= x: mpre's last value
    int lo = 0, hi = cc.np;    // J = the last knot <= x = the count of recall values <= x
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (cc.recall(mid) <= x) lo = mid + 1; else hi = mid;
    }
    const int J = lo;
    const double xj = J == 0 ? 0.0 : cc.recall(J - 1);
    const double yj1 = J < cc.np ? cc.suffix_max(J, lane) : 0.0;
    const double yj = J == 0 ? 1.0 : fmax(cc.precision(J - 1), yj1);
    if (xj == x) return yj;
    const double xj1 = J < cc.np ? cc.recall(J) : 1.0;
    const double slope = __ddiv_rn(__dsub_rn(yj1, yj), __dsub_rn(xj1, xj));
    return __dadd_rn(__dmul_rn(slope, __dsub_rn(x, xj)), yj);
}

__global__ void __launch_bounds__(AP_COL_WARPS * 32) ap_column_kernel(ApParams P) {
    const int c = blockIdx.x / P.K, j = blockIdx.x % P.K;
    const int off = P.offsets[c];
    const long long nl = P.n_labels[c];
    ClassColumn cc;
    cc.np = P.offsets[c + 1] - off;
    cc.K = P.K;
    if (cc.np == 0 || nl == 0) {
        if (threadIdx.x == 0) P.ap[(size_t)c * P.K + j] = 0.0;
        return;
    }
    cc.tpc = P.tpc + (size_t)j * P.n + off;
    cc.suffix = P.tile_max + (size_t)P.tile_first[c] * P.K + j;
    cc.nl_eps = __dadd_rn((double)nl, P.eps);
    __shared__ double y[AP_POINTS];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = w; i < AP_POINTS; i += AP_COL_WARPS) {
        const double v = ap_point(cc, linspace01(i, AP_POINTS), lane);
        if (lane == 0) y[i] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        // np.trapz: diff(x) * (y[1:] + y[:-1]) / 2.0, summed as numpy's pairwise sum does for 100 elements: 8
        // accumulators over elements 0..95, combined as a tree, then 96..99 in order
        double acc[8];
        double term[AP_POINTS - 1];
        for (int i = 0; i < AP_POINTS - 1; ++i) {
            const double d = __dsub_rn(linspace01(i + 1, AP_POINTS), linspace01(i, AP_POINTS));
            term[i] = __ddiv_rn(__dmul_rn(d, __dadd_rn(y[i + 1], y[i])), 2.0);
        }
        for (int k = 0; k < 8; ++k) acc[k] = term[k];
        for (int i = 8; i < 96; i += 8)
            for (int k = 0; k < 8; ++k) acc[k] = __dadd_rn(acc[k], term[i + k]);
        double s = __dadd_rn(__dadd_rn(__dadd_rn(acc[0], acc[1]), __dadd_rn(acc[2], acc[3])),
                             __dadd_rn(__dadd_rn(acc[4], acc[5]), __dadd_rn(acc[6], acc[7])));
        for (int i = 96; i < AP_POINTS - 1; ++i) s = __dadd_rn(s, term[i]);
        P.ap[(size_t)c * P.K + j] = s;
    }
}

// r[c] = np.interp(-px, -conf, recall[:, 0], left=0), p[c] = np.interp(-px, -conf, precision[:, 0], left=1)
__global__ void __launch_bounds__(AP_CURVE_THREADS) ap_curve_kernel(ApParams P) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)P.nc * AP_CURVE) return;
    const int c = (int)(idx / AP_CURVE), k = (int)(idx % AP_CURVE);
    const int off = P.offsets[c], np = P.offsets[c + 1] - off;
    const long long nl = P.n_labels[c];
    double pv = 0.0, rv = 0.0;
    if (np > 0 && nl > 0) {
        const unsigned long long* keys = P.keys + off;
        const int* tpc = P.tpc + off;  // column 0
        const double nl_eps = __dadd_rn((double)nl, P.eps);
        const double x = -linspace01(k, AP_CURVE);
        int lo = 0, hi = np;  // count of knots -conf <= x
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (key_neg_conf(keys[mid]) <= x) lo = mid + 1; else hi = mid;
        }
        const int jj = lo - 1;
        if (jj < 0) {
            rv = 0.0;
            pv = 1.0;
        } else {
            const double t0 = (double)tpc[jj];
            const double r0 = __ddiv_rn(t0, nl_eps), p0 = __ddiv_rn(t0, (double)(jj + 1));
            const double x0 = key_neg_conf(keys[jj]);
            if (jj == np - 1 || x0 == x) {  // the last knot (also x past it: right = fp[-1]), or an exact knot
                rv = r0;
                pv = p0;
            } else {
                const double t1 = (double)tpc[jj + 1];
                const double r1 = __ddiv_rn(t1, nl_eps), p1 = __ddiv_rn(t1, (double)(jj + 2));
                const double dx = __dsub_rn(key_neg_conf(keys[jj + 1]), x0), u = __dsub_rn(x, x0);
                rv = __dadd_rn(__dmul_rn(__ddiv_rn(__dsub_rn(r1, r0), dx), u), r0);
                pv = __dadd_rn(__dmul_rn(__ddiv_rn(__dsub_rn(p1, p0), dx), u), p0);
            }
        }
    }
    P.p[idx] = pv;
    P.r[idx] = rv;
}

// ---------------------------------------------------------------------------------------------------------- host side
int bitwidth(int v) {  // bits to hold 0..v
    int b = 0;
    while (b < 31 && (1 << b) <= v) ++b;
    return b;
}

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

struct ApLayout {
    size_t keys[2], rows[2], mask, tpc, offsets, tile_first, tile_cnt, tile_max, classes, n_labels, temp, temp_bytes, total;
    long tiles;
    int end_bit;
};

// sub-buffer offsets of the workspace; false if the sort's temporary size cannot be queried
bool ap_layout(long n, int K, int nc, ApLayout& L) {
    L.tiles = (n + AP_TILE - 1) / AP_TILE + nc;
    L.end_bit = 32 + bitwidth(nc);
    L.temp_bytes = 0;
    if (n > 0) {
        cub::DoubleBuffer<unsigned long long> k(nullptr, nullptr);
        cub::DoubleBuffer<int> v(nullptr, nullptr);
        if (cub::DeviceRadixSort::SortPairs(nullptr, L.temp_bytes, k, v, (int)n, 0, L.end_bit) != cudaSuccess) {
            cudaGetLastError();
            return false;
        }
    }
    size_t o = 0;
    auto take = [&o](size_t bytes) { const size_t at = o; o += align256(bytes); return at; };
    L.keys[0] = take(n * sizeof(unsigned long long));
    L.keys[1] = take(n * sizeof(unsigned long long));
    L.rows[0] = take(n * sizeof(int));
    L.rows[1] = take(n * sizeof(int));
    L.mask = take(n * sizeof(unsigned));
    L.tpc = take((size_t)K * n * sizeof(int));
    L.offsets = take((nc + 1) * sizeof(int));
    L.tile_first = take((nc + 1) * sizeof(int));
    L.tile_cnt = take((size_t)L.tiles * K * sizeof(int));
    L.tile_max = take((size_t)L.tiles * K * sizeof(double));
    L.classes = take(nc * sizeof(float));
    L.n_labels = take(nc * sizeof(long long));
    L.temp = take(L.temp_bytes);
    L.total = o;
    return true;
}

#define AP_CUDA(call)                                                                        \
    do {                                                                                     \
        const cudaError_t e_ = (call);                                                       \
        if (e_ != cudaSuccess) {                                                             \
            cerb_set_error("cerb_ap_per_class: %s failed: %s", #call, cudaGetErrorString(e_)); \
            return CERB_ECUDA;                                                               \
        }                                                                                    \
    } while (0)

}  // namespace

extern "C" size_t cerb_ap_workspace_bytes(long n, int K, int nc) {
    if (n < 0 || n > 0x7fffffffL || K < 1 || K > 32 || nc < 0) return 0;
    ApLayout L;
    return ap_layout(n, K, nc, L) ? L.total : 0;
}

extern "C" int cerb_ap_per_class(const unsigned char* tp, int K, const float* conf, const float* pred_cls, long n,
                                 const float* classes, const long long* n_labels, int nc, double eps, double* ap, double* p,
                                 double* r, void* workspace, size_t workspace_bytes, void* stream) {
    cerb_clear_error();
    CERB_REQUIRE(n >= 0 && n <= 0x7fffffffL, "cerb_ap_per_class: n=%ld detections, 0 <= n < 2^31 required", n);
    CERB_REQUIRE(K >= 1 && K <= 32, "cerb_ap_per_class: K=%d IoU thresholds, 1..32 supported", K);
    CERB_REQUIRE(nc >= 0, "cerb_ap_per_class: nc=%d", nc);
    CERB_REQUIRE(n == 0 || (tp && conf && pred_cls), "cerb_ap_per_class: null argument (tp, conf, pred_cls)");
    CERB_REQUIRE(nc == 0 || (classes && n_labels && ap && p && r), "cerb_ap_per_class: null argument (classes, n_labels, ap, p, r)");
    for (int c = 0; c < nc; ++c) {
        CERB_REQUIRE(c == 0 || classes[c - 1] < classes[c], "cerb_ap_per_class: classes must be strictly ascending (and not NaN) at %d", c);
        CERB_REQUIRE(classes[c] == classes[c], "cerb_ap_per_class: classes[%d] is NaN", c);
        CERB_REQUIRE(n_labels[c] >= 0, "cerb_ap_per_class: n_labels[%d] < 0", c);
    }
    if (nc == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    if (n == 0) {  // no detection: every class is skipped by the reference and keeps its zero rows
        AP_CUDA(cudaMemsetAsync(ap, 0, (size_t)nc * K * sizeof(double), s));
        AP_CUDA(cudaMemsetAsync(p, 0, (size_t)nc * AP_CURVE * sizeof(double), s));
        AP_CUDA(cudaMemsetAsync(r, 0, (size_t)nc * AP_CURVE * sizeof(double), s));
        return 0;
    }
    ApLayout L;
    if (!ap_layout(n, K, nc, L)) {
        cerb_set_error("cerb_ap_per_class: cannot size the radix sort (no CUDA device?)");
        return CERB_ECUDA;
    }
    if (const int rc = cerb_require_workspace("cerb_ap_per_class", workspace, workspace_bytes, L.total)) return rc;
    CERB_REQUIRE(cerb_aligned(workspace, 256), "cerb_ap_per_class: workspace must be 256-byte aligned");
    char* ws = (char*)workspace;
    float* classes_d = (float*)(ws + L.classes);
    long long* n_labels_d = (long long*)(ws + L.n_labels);
    // host arrays -> workspace, on the stream (small; the copy is staged before the call returns)
    AP_CUDA(cudaMemcpyAsync(classes_d, classes, nc * sizeof(float), cudaMemcpyHostToDevice, s));
    AP_CUDA(cudaMemcpyAsync(n_labels_d, n_labels, nc * sizeof(long long), cudaMemcpyHostToDevice, s));

    cub::DoubleBuffer<unsigned long long> keys((unsigned long long*)(ws + L.keys[0]), (unsigned long long*)(ws + L.keys[1]));
    cub::DoubleBuffer<int> rows((int*)(ws + L.rows[0]), (int*)(ws + L.rows[1]));
    const int key_blocks = (int)((n + 255) / 256 < 148 * 16 ? (n + 255) / 256 : 148 * 16);
    ap_key_kernel<<<key_blocks, 256, 0, s>>>(tp, K, conf, pred_cls, (int)n, classes_d, nc, keys.Current(), rows.Current(),
                                             (unsigned*)(ws + L.mask));
    AP_CUDA(cudaGetLastError());
    size_t temp_bytes = L.temp_bytes;
    AP_CUDA(cub::DeviceRadixSort::SortPairs(ws + L.temp, temp_bytes, keys, rows, (int)n, 0, L.end_bit, s));

    ApParams P;
    P.keys = keys.Current();
    P.rows = rows.Current();
    P.mask = (const unsigned*)(ws + L.mask);
    P.n_labels = n_labels_d;
    P.tpc = (int*)(ws + L.tpc);
    P.offsets = (int*)(ws + L.offsets);
    P.tile_first = (int*)(ws + L.tile_first);
    P.tile_cnt = (int*)(ws + L.tile_cnt);
    P.tile_max = (double*)(ws + L.tile_max);
    P.eps = eps;
    P.ap = ap;
    P.p = p;
    P.r = r;
    P.n = (int)n;
    P.K = K;
    P.nc = nc;
    const unsigned tiles = (unsigned)L.tiles, columns = (unsigned)nc * K;
    ap_segment_kernel<<<1, 1024, 0, s>>>(P);
    ap_tile_count_kernel<<<tiles, AP_TILE, 0, s>>>(P);
    ap_tile_base_kernel<<<columns, AP_SCAN_THREADS, 0, s>>>(P);
    ap_tile_tpc_kernel<<<tiles, AP_TILE, 0, s>>>(P);
    ap_tile_suffix_kernel<<<columns, AP_SCAN_THREADS, 0, s>>>(P);
    ap_column_kernel<<<columns, AP_COL_WARPS * 32, 0, s>>>(P);
    ap_curve_kernel<<<(unsigned)(((long long)nc * AP_CURVE + AP_CURVE_THREADS - 1) / AP_CURVE_THREADS), AP_CURVE_THREADS, 0, s>>>(P);
    AP_CUDA(cudaGetLastError());
    return 0;
}
