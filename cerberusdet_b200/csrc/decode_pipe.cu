// Fused Detect-head decode, software-pipelined variant: every thread keeps its NEXT loads in flight
// (cp.async into a private shared-memory slot) while it reduces the rows it already holds in registers.
//
// Why: decode.cu's threads alternate "issue 16 loads, wait for HBM" and "~1100 instructions of exp/convert
// work with nothing in flight"; at 96 registers only 5 warps per scheduler are there to cover the wait, and
// register double buffering costs more occupancy than it wins (profiles/r01_decode.md).  cp.async needs no
// destination registers, so the prefetch is free in registers: 16 rows x 16 bytes = 256 bytes of shared
// memory per thread (32 KB per 128-thread CTA, 5 CTAs per SM).  A thread only ever touches its own slot, so
// there is no barrier anywhere; the only ordering is cp.async.wait_group in the issuing thread.
//
// Same arithmetic and rounding points as decode.cu (reference models/yolo.py:93-99, utils/tal.py:181-205).
//
// Work decomposition.  A "row" is one (task, level, kind): kind 0 = DFL sides l,r -> (cx, w); kind 1 = sides
// t,b -> (cy, h); kind 2 = every class channel (sigmoid + score summary).  An item is VEC consecutive anchors
// of one image (one 128-bit access per channel); a CTA owns DEC_THREADS * IPT consecutive items of a row and
// a thread the items first + i * DEC_THREADS, so a warp still reads 512 contiguous bytes per channel.
//   DFL thread:   groups = the 2 * IPT sides of its items; group g+1 streams in while group g is reduced.
//   class thread: groups of 4 channels in a 4-deep ring (16 vectors in flight), across its CIPT items (class CTAs come
//                 last in the grid, so fewer items per thread = shorter CTAs = a shorter tail).
#include "decode_common.cuh"

#ifndef PIPE_MINB
#define PIPE_MINB 5
#endif
#define PIPE_SLOT_VECS CERB_REG_MAX  // 16-byte vectors per thread slot
#define PIPE_MAX_ROWS (3 * CERB_MAX_TASKS * CERB_MAX_LEVELS)

struct PipeParams {
    DecodeParams d;
    int nrows;
    int row_start[PIPE_MAX_ROWS + 1];      // first CTA of each row
    unsigned char row_kind[PIPE_MAX_ROWS];  // 0, 1 = DFL part, 2 = classes
    unsigned char row_trow[PIPE_MAX_ROWS];  // task * L + level
};

// cp_async16_pred: 16-byte cp.async with a source size.  src_bytes = 0 reads nothing (the slot is zero-filled): a
// branch-free "maybe prefetch" that the scheduler cannot sink below the arithmetic the way it sinks a conditional block.
#ifndef CERB_NO_L2_HINTS
// raw heads are read exactly once: mark their lines evict-first so that y and the score summary (written here, read by
// the NMS kernel right after) stay in the 126 MB L2 instead of being pushed out by 261 MB of streaming input
// (only when the outputs fit: with fp32 inputs at B=64 -- 152 MB of outputs -- the same hint costs 7 us, so the host
// decides per launch, DecodeParams::l2_evict_first)
__device__ __forceinline__ uint64_t l2_policy(bool evict_first) {
    uint64_t pol;
    if (evict_first) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void cp_async16_pred(uint32_t dst, const void* src, int src_bytes, uint64_t pol) {
    asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2, %3;" ::"r"(dst), "l"(src), "r"(src_bytes), "l"(pol)
                 : "memory");
}
#else
__device__ __forceinline__ void cp_async16_pred(uint32_t dst, const void* src, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
#endif
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

template <typename T, int VEC, int IPT, int CIPT>
__global__ void __launch_bounds__(DEC_THREADS, PIPE_MINB) decode_pipe_kernel(const __grid_constant__ PipeParams Q) {
    static_assert(sizeof(T) * VEC == 16, "the pipelined kernel moves 16-byte vectors");
    // the next kernel in the stream (NMS, launched with programmatic stream serialization) may be scheduled as this
    // grid drains; it waits for this grid's completion (griddepcontrol.wait) before it reads y
    asm volatile("griddepcontrol.launch_dependents;");
    extern __shared__ uint4 pipe_smem[];  // [PIPE_SLOT_VECS][DEC_THREADS]: conflict-free for 128-bit accesses
    const DecodeParams& P = Q.d;
    uint4* const my = pipe_smem + threadIdx.x;
    const uint32_t my_s = (uint32_t)__cvta_generic_to_shared(my);
    constexpr uint32_t SLOT_STRIDE = DEC_THREADS * 16;
#ifndef CERB_NO_L2_HINTS
    const uint64_t pol = l2_policy(Q.d.l2_evict_first != 0);
#define CERB_POL , pol
#else
#define CERB_POL
#endif

    // ---- block -> row; uniform per block
    int row = 0;
    {
        int lo = 0, hi = Q.nrows;  // row_start[lo] <= blockIdx.x < row_start[hi]
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if ((int)blockIdx.x >= Q.row_start[mid]) lo = mid; else hi = mid;
        }
        row = lo;
    }
    const int kind = Q.row_kind[row];
    const int trow = Q.row_trow[row];
    const int task = trow / P.L, level = trow - task * P.L;
    const int hw = P.hw[level];
    const int nvec = hw / VEC;
    const int n_items = P.B * nvec;
    const int ipt = kind < 2 ? IPT : CIPT;
    const int first = ((int)blockIdx.x - Q.row_start[row]) * (DEC_THREADS * ipt) + (int)threadIdx.x;
    if (first >= n_items) return;
    const int cnt = min(ipt, (n_items - first + DEC_THREADS - 1) / DEC_THREADS);  // my items: first + i * DEC_THREADS

    const int nc = P.nc[task];
    // concatenated heads: box and class channels share one tensor; split heads: two tensors (models/yolo.py:90 unmaterialised)
    const T* __restrict__ clsp = reinterpret_cast<const T*>(P.cls[task][level]);
    const bool use_cls = kind == 2 && clsp != nullptr;
    const size_t img_stride = (size_t)(clsp == nullptr ? 4 * CERB_REG_MAX + nc : (kind == 2 ? nc : 4 * CERB_REG_MAX)) * hw;
    const T* __restrict__ lbase = use_cls ? clsp : reinterpret_cast<const T*>(P.lvl[task][level]);
    const size_t cls_off = use_cls ? 0 : (size_t)(4 * CERB_REG_MAX) * hw;  // first class channel inside an image
    T* __restrict__ ybase = reinterpret_cast<T*>(P.y[task]) + P.aoff[level];
    const size_t y_img = (size_t)(4 + nc) * P.A;

    if (kind < 2) {
        // ------------------------------------------------ DFL sides -> (centre, size) of one axis
        auto side_ptr = [&](int g) -> const T* {
            const int it = first + (g >> 1) * DEC_THREADS;
            const int b = it / nvec, v = it - b * nvec;
            return lbase + (size_t)b * img_stride + (size_t)((kind + ((g & 1) << 1)) * CERB_REG_MAX) * hw + v * VEC;
        };
        auto issue = [&](const T* p, int bytes) {
#pragma unroll
            for (int k = 0; k < CERB_REG_MAX; ++k) cp_async16_pred(my_s + k * SLOT_STRIDE, p + (size_t)k * hw, bytes CERB_POL);
            cp_async_commit();
        };
        issue(side_ptr(0), 16);
        const int G = 2 * cnt;
        DVec<T, VEC> dlo;
#pragma unroll 1
        for (int g = 0; g < G; ++g) {
            const bool more = g + 1 < G;
            const T* nxt = side_ptr(more ? g + 1 : g);  // (a valid address either way)
            cp_async_wait<0>();
            Pack<T, VEC> v[CERB_REG_MAX];
#pragma unroll
            for (int k = 0; k < CERB_REG_MAX; ++k) v[k].raw = my[k * DEC_THREADS];
            issue(nxt, more ? 16 : 0);  // streams in while this side is reduced
            DVec<T, VEC> d;
            dfl_reduce<T, VEC>(v, d);
            if ((g & 1) == 0) {
                dlo = d;
            } else {
                // dist2bbox(xywh) on one axis (utils/tal.py:198-204), * stride (yolo.py:98)
                const int it = first + (g >> 1) * DEC_THREADS;
                const int b = it / nvec, vv = it - b * nvec;
                const int a0 = vv * VEC;
                T* __restrict__ out = ybase + (size_t)b * y_img + a0;
                Pack<T, VEC> oc, os;
                axis_boxes<T, VEC>(dlo, d, a0, P.w[level], kind == 0, P.stride[level], oc, os);
                store_pack<T, VEC>(out + (size_t)kind * P.A, oc);
                store_pack<T, VEC>(out + (size_t)(kind + 2) * P.A, os);
            }
        }
    } else {
        // ------------------------------------------------ class sigmoids (+ score summary), yolo.py:99
        const size_t srow = ((size_t)(P.A / VEC) + VEC - 1) / VEC * VEC;
        T* __restrict__ sbase = P.smax[task] != nullptr ? reinterpret_cast<T*>(P.smax[task]) : nullptr;
        auto class_ptr = [&](int i) -> const T* {
            const int it = first + i * DEC_THREADS;
            const int b = it / nvec, v = it - b * nvec;
            return lbase + (size_t)b * img_stride + cls_off + v * VEC;
        };
        // issue cursor: 4-channel groups in item order; an exhausted cursor still commits (zero-byte) groups so
        // that wait_group<3> always means "the group consumed now has landed"
        int ii = 0, ic = 0;
        const T* ip = class_ptr(0);
        auto issue_next = [&](int slot) {
            const bool live = ii < cnt;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int c = min(ic + u, nc - 1);  // (a valid address either way)
                cp_async16_pred(my_s + (slot * 4 + u) * SLOT_STRIDE, ip + (size_t)c * hw, (live && ic + u < nc) ? 16 : 0 CERB_POL);
            }
            cp_async_commit();
            ic += 4;
            if (live && ic >= nc) {
                ic = 0;
                if (++ii < cnt) ip = class_ptr(ii);
            }
        };
#pragma unroll
        for (int s = 0; s < 4; ++s) issue_next(s);

        const int G = cnt * ((nc + 3) >> 2);
        int ci = 0, cc = 0;
        T* __restrict__ cout = nullptr;
        T* __restrict__ smax = nullptr;
        auto set_out = [&](int i) {
            const int it = first + i * DEC_THREADS;
            const int b = it / nvec, v = it - b * nvec;
            cout = ybase + (size_t)b * y_img + (size_t)4 * P.A + v * VEC;
            if (sbase != nullptr) smax = sbase + (size_t)b * nc * srow + (P.aoff[level] + v * VEC) / VEC;
        };
        set_out(0);
#pragma unroll 1
        for (int g = 0; g < G; ++g) {
            cp_async_wait<3>();
            const int slot = g & 3;
            Pack<T, VEC> vv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (cc + u < nc) vv[u].raw = my[(slot * 4 + u) * DEC_THREADS];
            issue_next(slot);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (cc + u < nc) {
                    sigmoid_pack<T, VEC>(vv[u]);
                    store_pack<T, VEC>(cout + (size_t)(cc + u) * P.A, vv[u]);
                    if (smax != nullptr) smax[(size_t)(cc + u) * srow] = pack_max<T, VEC>(vv[u]);
                }
            }
            cc += 4;
            if (cc >= nc) {
                cc = 0;
                if (++ci < cnt) set_out(ci);
            }
        }
    }
}

template <typename T, int VEC, int IPT, int CIPT> static cudaError_t launch_pipe_t(const DecodeParams& P, cudaStream_t stream) {
    PipeParams q;
    q.d = P;
    int blocks = 0, r = 0;
    // block order (profiles/r01_decode.md): 2 = every DFL row of the launch first, then every class row (the
    // short streaming CTAs fill the tail); anything else = per (task, level): [l,r][t,b][classes]
    const bool box_first = P.interleave_parts == 2;
    for (int pass = 0; pass < (box_first ? 2 : 1); ++pass)
        for (int t = 0; t < P.T; ++t)
            for (int l = 0; l < P.L; ++l) {
                const long items = (long)P.B * (P.hw[l] / VEC);
                const int k0 = box_first ? (pass == 0 ? 0 : 2) : 0;
                const int k1 = box_first ? (pass == 0 ? 2 : 3) : 3;
                for (int k = k0; k < k1; ++k) {
                    const int per_block = DEC_THREADS * (k < 2 ? IPT : CIPT);
                    q.row_start[r] = blocks;
                    q.row_kind[r] = (unsigned char)k;
                    q.row_trow[r] = (unsigned char)(t * P.L + l);
                    blocks += (int)((items + per_block - 1) / per_block);
                    ++r;
                }
            }
    q.nrows = r;
    q.row_start[r] = blocks;
    if (blocks == 0) return cudaSuccess;
    constexpr size_t smem = (size_t)PIPE_SLOT_VECS * DEC_THREADS * 16;
    // per launch, like launch_nms_t: function attributes are per device, and a process may drive several
    // (32 KB fits the default dynamic limit; the carve-out is what lets 5 CTAs = 165 KB share an SM)
    cudaError_t e = cudaFuncSetAttribute(decode_pipe_kernel<T, VEC, IPT, CIPT>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                         cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    if (!P.pdl) {
        decode_pipe_kernel<T, VEC, IPT, CIPT><<<blocks, DEC_THREADS, smem, stream>>>(q);
        return cudaGetLastError();
    }
    // overlapped schedule on ONE stream (pipeline.py): NMS(k-1), then this launch with the programmatic attribute -- its CTAs
    // are dispatched once every CTA of the NMS kernel has started, never before (the order that overlaps best, made
    // deterministic), and run beside it
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)blocks);
    cfg.blockDim = dim3(DEC_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, decode_pipe_kernel<T, VEC, IPT, CIPT>, q);
}

// Items per thread (DFL rows, class rows) of the shipped instantiations: fp16 2 / PIPE_CIPT_F16, fp32 1 / 1
// (profiles/r02_decode.md); bf16 takes fp16's (it moves the same bytes and runs the same packed arithmetic).  -DCERB_DECODE_VARIANTS also builds the other combinations for tools/ A/B runs
// (ipt = 10 * IPT + CIPT selects one).
#ifndef PIPE_IPT_F16
#define PIPE_IPT_F16 2
#endif
#ifndef PIPE_CIPT_F16
#define PIPE_CIPT_F16 1
#endif
// needs vec == 16 / sizeof(T); cudaErrorInvalidConfiguration = use decode.cu's kernel
cudaError_t cerb_launch_decode_pipe(const DecodeParams& P, int dtype, int ipt, cudaStream_t stream) {
    if (dtype == CERB_DTYPE_F16) {
        switch (ipt) {
#ifdef CERB_DECODE_VARIANTS
            case 11: return launch_pipe_t<__half, 8, 1, 1>(P, stream);
            case 21: return launch_pipe_t<__half, 8, 2, 1>(P, stream);
            case 22: return launch_pipe_t<__half, 8, 2, 2>(P, stream);
            case 42: return launch_pipe_t<__half, 8, 4, 2>(P, stream);
            case 41: return launch_pipe_t<__half, 8, 4, 1>(P, stream);
#endif
            case 0: return cudaErrorInvalidConfiguration;
            default: return launch_pipe_t<__half, 8, PIPE_IPT_F16, PIPE_CIPT_F16>(P, stream);
        }
    }
    if (dtype == CERB_DTYPE_BF16) return ipt == 0 ? cudaErrorInvalidConfiguration
                                                  : launch_pipe_t<__nv_bfloat16, 8, PIPE_IPT_F16, PIPE_CIPT_F16>(P, stream);
    switch (ipt) {
#ifdef CERB_DECODE_VARIANTS
        case 21: return launch_pipe_t<float, 4, 2, 1>(P, stream);
        case 22: return launch_pipe_t<float, 4, 2, 2>(P, stream);
#endif
        case 0: return cudaErrorInvalidConfiguration;
        default: return launch_pipe_t<float, 4, 1, 1>(P, stream);
    }
}
