// Fused Detect-head decode for every task head in ONE launch.
//
// Replaces the eval branch of the reference Detect.forward after the conv towers
// (reference models/yolo.py:93-99): make_anchors (utils/tal.py:181-193), the
// [B,no,A] concat/split (yolo.py:97), DFL softmax-expectation (yolo.py:57-59),
// dist2bbox(xywh) (utils/tal.py:196-205), * stride (yolo.py:98) and the class
// sigmoid + concat (yolo.py:99).  ~15 ATen launches and ~4.5x the algorithmic HBM
// traffic there; here each raw element is read once and each y element written once.
//
// Work decomposition.  A "row" is one (task, level).  Inside a row the blocks are laid
// out as [part][vector-block]: part 0 owns DFL sides l,r -> (cx, w); part 1 owns sides
// t,b -> (cy, h); parts 2.. own chunks of CLS_CHUNK class channels.  A thread owns VEC
// consecutive anchors of one image (one 128-bit access per channel), so a warp reads
// 512 contiguous bytes per channel.  Anchors are computed analytically.
#include "cerb_kernels.h"

#include "decode_common.cuh"


template <typename T, int VEC>
__global__ void __launch_bounds__(DEC_THREADS, DEC_MINB) decode_kernel(const __grid_constant__ DecodeParams P) {
    // ---- block -> (row, part, vector block); uniform per block
    // the next kernel in the stream (NMS, launched with programmatic stream serialization) may be scheduled as this
    // grid drains; it waits for this grid's completion (griddepcontrol.wait) before it reads y
    asm volatile("griddepcontrol.launch_dependents;");
    int row = 0;
    {
        int lo = 0, hi = P.nrows;  // row_start[lo] <= blockIdx.x < row_start[hi]
        while (hi - lo > 1) {
            int mid = (lo + hi) >> 1;
            if ((int)blockIdx.x >= P.row_start[mid]) lo = mid; else hi = mid;
        }
        row = lo;
    }
    const int TL = P.T * P.L;
    const bool cls_row = row >= TL;  // box-first order only: rows TL.. are the class rows
    const int trow = cls_row ? row - TL : row;
    const int task = trow / P.L, level = trow - task * P.L;
    const int in_row = blockIdx.x - P.row_start[row];
    const int bpp = P.row_blocks_per_part[trow];
    // Block order of the parts (profiles/r01_decode.md): 0 = contiguous per (task, level): [l,r blocks][t,b][classes];
    // 1 = interleaved (DFL and class blocks share every SM at all times; best for fp32, which is HBM-bound);
    // 2 = every DFL block of the launch first, then every class block (the short streaming blocks fill the tail).
    int part, vblk;
    if (P.interleave_parts == 1) {
        const int nparts = 2 + (P.nc[task] + CLS_CHUNK - 1) / CLS_CHUNK;
        vblk = in_row / nparts;
        part = in_row - vblk * nparts;
    } else {
        part = in_row / bpp;
        vblk = in_row - part * bpp;
        if (cls_row) part += 2;
    }

    const int hw = P.hw[level];
    const int nvec = hw / VEC;
    const int item = vblk * DEC_THREADS + threadIdx.x;
    if (item >= P.B * nvec) return;
    const int b = item / nvec;
    const int v = item - b * nvec;
    const int a0 = v * VEC;  // first anchor inside the level

    const int nc = P.nc[task];
    const int no = 4 * CERB_REG_MAX + nc;
    const T* __restrict__ clsp = reinterpret_cast<const T*>(P.cls[task][level]);  // split heads, or null
    const T* __restrict__ in = reinterpret_cast<const T*>(P.lvl[task][level]) +
                               (size_t)b * (clsp ? 4 * CERB_REG_MAX : no) * hw + a0;
    T* __restrict__ out = reinterpret_cast<T*>(P.y[task]) + (size_t)b * (4 + nc) * P.A + P.aoff[level] + a0;

    if (part < 2) {
        // sides (l, r) -> cx, w   or   (t, b) -> cy, h      (utils/tal.py:198-204)
        DVec<T, VEC> dlo, dhi;
        dfl_side<T, VEC>(in + (size_t)(part * CERB_REG_MAX) * hw, hw, dlo);
        dfl_side<T, VEC>(in + (size_t)((part + 2) * CERB_REG_MAX) * hw, hw, dhi);
        Pack<T, VEC> oc, os;
        axis_boxes<T, VEC>(dlo, dhi, a0, P.w[level], part == 0, P.stride[level], oc, os);
        store_pack<T, VEC>(out + (size_t)part * P.A, oc);
        store_pack<T, VEC>(out + (size_t)(part + 2) * P.A, os);
    } else {
        // class scores: sigmoid (yolo.py:99).  Optionally also the score summary: the maximum of each
        // 16-byte vector of scores (one value per class and VEC consecutive anchors), which lets the NMS
        // kernel read only the vectors that can hold a candidate.
        const int c0 = (part - 2) * CLS_CHUNK;
        const int c1 = min(nc, c0 + CLS_CHUNK);
        const T* __restrict__ cin = clsp ? clsp + (size_t)b * nc * hw + a0 : in + (size_t)(4 * CERB_REG_MAX) * hw;
        T* __restrict__ cout = out + (size_t)4 * P.A;
        T* __restrict__ smax = nullptr;  // [B, nc, srow], srow = roundup(A / VEC, VEC)
        const size_t srow = ((size_t)(P.A / VEC) + VEC - 1) / VEC * VEC;
        if (sizeof(T) * VEC == 16 && P.smax[task] != nullptr)
            smax = reinterpret_cast<T*>(P.smax[task]) + (size_t)b * nc * srow + (P.aoff[level] + a0) / VEC;
        int c = c0;
        for (; c + 4 <= c1; c += 4) {
            Pack<T, VEC> vv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) vv[u] = load_pack<T, VEC>(cin + (size_t)(c + u) * hw);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                sigmoid_pack<T, VEC>(vv[u]);
                store_pack<T, VEC>(cout + (size_t)(c + u) * P.A, vv[u]);
                if (smax != nullptr) smax[(size_t)(c + u) * srow] = pack_max<T, VEC>(vv[u]);
            }
        }
        for (; c < c1; ++c) {
            Pack<T, VEC> v1 = load_pack<T, VEC>(cin + (size_t)c * hw);
            sigmoid_pack<T, VEC>(v1);
            store_pack<T, VEC>(cout + (size_t)c * P.A, v1);
            if (smax != nullptr) smax[(size_t)c * srow] = pack_max<T, VEC>(v1);
        }
    }
}

template <typename T, int VEC> static cudaError_t launch_decode_t(DecodeParams& P, cudaStream_t stream) {
    int blocks = 0;
    const int TL = P.T * P.L;
    const int passes = P.interleave_parts == 2 ? 2 : 1;  // box-first: DFL rows, then class rows
    for (int pass = 0; pass < passes; ++pass)
        for (int t = 0; t < P.T; ++t)
            for (int l = 0; l < P.L; ++l) {
                const int trow = t * P.L + l;
                const long items = (long)P.B * (P.hw[l] / VEC);
                const int bpp = (int)((items + DEC_THREADS - 1) / DEC_THREADS);
                const int cls_parts = (P.nc[t] + CLS_CHUNK - 1) / CLS_CHUNK;
                const int parts = passes == 1 ? 2 + cls_parts : (pass == 0 ? 2 : cls_parts);
                P.row_start[pass * TL + trow] = blocks;
                P.row_blocks_per_part[trow] = bpp > 0 ? bpp : 1;
                blocks += bpp * parts;
            }
    P.nrows = passes * TL;
    P.row_start[P.nrows] = blocks;
    if (blocks == 0) return cudaSuccess;
    decode_kernel<T, VEC><<<blocks, DEC_THREADS, 0, stream>>>(P);
    return cudaGetLastError();
}

// vec = anchors per thread the caller proved legal (alignment + divisibility)
cudaError_t cerb_launch_decode(DecodeParams& P, int dtype, int vec, cudaStream_t stream) {
    if (dtype == CERB_DTYPE_F16) {
        switch (vec) {
            case 8: return launch_decode_t<__half, 8>(P, stream);
            case 4: return launch_decode_t<__half, 4>(P, stream);
            case 2: return launch_decode_t<__half, 2>(P, stream);
            default: return launch_decode_t<__half, 1>(P, stream);
        }
    } else if (dtype == CERB_DTYPE_BF16) {
        switch (vec) {
            case 8: return launch_decode_t<__nv_bfloat16, 8>(P, stream);
            case 4: return launch_decode_t<__nv_bfloat16, 4>(P, stream);
            case 2: return launch_decode_t<__nv_bfloat16, 2>(P, stream);
            default: return launch_decode_t<__nv_bfloat16, 1>(P, stream);
        }
    } else {
        switch (vec) {
            case 4: return launch_decode_t<float, 4>(P, stream);
            case 2: return launch_decode_t<float, 2>(P, stream);
            default: return launch_decode_t<float, 1>(P, stream);
        }
    }
}
