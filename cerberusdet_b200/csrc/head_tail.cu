// SURVEY 8f row 3, head-tail fusion: the LAST 1x1 convolutions of the two towers of every (task, level)
//     box = cv2[l][-1](u2)   [B, c2, H, W] -> [B, 64, H, W]        reference models/yolo.py:81-84, 89-90
//     cls = cv3[l][-1](u3)   [B, c3, H, W] -> [B, nc, H, W]
// fused with the eval decode (models/yolo.py:93-99): the raw head tensor [B, 64+nc, H, W] is never written or re-read.
// fp16 only (tcgen05 kind::f16, fp32 accumulation in TMEM); one persistent launch for all task heads and levels.
//
// Shape of the problem.  Per image the activations are [channels][anchors] with the anchors contiguous, so with the
// anchors on the MMA's M axis the A operand is MN-major.  A tile = 128 consecutive anchors of one image and level:
//     D1[128 x 64]  = U2^T[128 x c2] * W2^T[c2 x 64]      tcgen05.mma.cta_group::1.kind::f16, M = 128, N = 64
//     D2[128 x NCP] = U3^T[128 x c3] * W3^T[c3 x NCP]     NCP = nc rounded up to 16
// It is memory-bound (the tile reads (c2+c3)*256 B and needs 2*128*(c2*64 + c3*NCP) flop: ~30 flop/B at yolov8x widths),
// so the design goal is to keep TMA loads in flight, not tensor throughput.
//
// A (activations): TMA boxes {64 anchors (128 B inner), RB channel rows}, SWIZZLE_128B -> rows of 128 B, 8 rows = one
//   1024-byte swizzle atom = the canonical MN-major SW128 layout ((8,8,m),(8,k)):((1,8,LBO),(64,SBO)) (elements; CUTLASS
//   cute/atom/mma_traits_sm100.hpp): SBO = 1024 B (next 8 channels), LBO = bytes between the two 64-anchor halves of a
//   stage; one MMA (K = 16) consumes 16 rows = 2048 B.
// B (weights [N][K] row-major = K-major): TMA boxes {64 k, N rows}, SWIZZLE_128B -> the K-major SW128 image (row n at
//   n*128 B inside a 64-wide K block, 16-byte chunks XOR-swizzled by n & 7), SBO = 1024 B; a K = 16 step advances the
//   start address by 32 B inside the swizzled row.  Rows >= nc and columns >= K are zero-filled by TMA.
// D: TMEM, lane = anchor, column = output channel, up to four accumulator buffers (tiles i+1.. are multiplied while
//   tile i is decoded).  tcgen05.ld.32x32b hands each epilogue thread the logits of ITS anchor, so the epilogue is the per-anchor
//   decode math of decode.cu after "conv output = half(acc + bias)".
//
// Warp roles (576 threads, 1 CTA per SM): warp 0 = TMA producer (one lane), warp 1 = TMEM allocation + MMA issue (one
// lane), warps 2-17 = epilogue in two groups of 8 that take alternate tiles; inside a group two warps per TMEM lane
// quadrant, the first takes DFL sides l,r (x axis) and the even 8-class chunks, the second sides t,b (y axis) and the
// odd chunks.
// Pipelines: activation ring full[s]/empty[s] (TMA -> MMA -> TMA), weights wfull/wempty (reloaded when the CTA's tile
// sequence enters another (task, level)), accumulators tfull[b]/tempty[b] over up to 4 TMEM buffers (MMA -> epilogue
// -> MMA).
#include <cuda.h>

#include "../../include/cerb_post.h"
#include "decode_common.cuh"

#define HT_TILE 128
#define HT_EPI_WARPS 8    // epilogue warps per group: two per TMEM lane quadrant
#define HT_EPI_GROUPS 2   // at most; groups take alternate tiles.  One group decodes a tile in ~2.9 us, which is slower than
                          // the memory stream delivers one below ~384 input channels: the host launches 2 groups
                          // there and 1 above (profiles/r02_head_tail.md)
#define HT_MAX_BUFS 4     // TMEM accumulator buffers (as many as fit 512 columns, at least 2)
#define HT_THREADS (64 + 32 * HT_EPI_WARPS * HT_EPI_GROUPS)
#define HT_MAX_ROWS 12   // (task, level) pairs per launch; more are split over several launches
#define HT_MAX_STAGES 8
#define HT_MAX_NCP 192   // two accumulator buffers of 64 + NCP columns must fit the 512 TMEM columns

struct HtRow {
    const __half* b2;   // [64]
    const __half* b3;   // [nc]
    __half* y;          // [B, 4 + nc, A] of this row's task
    __half* smax;       // optional score summary of this row's task
    int c2, c3, nc, ncp;
    int rb2, rb3;       // channel rows per ring stage (divide c2 / c3, multiples of 16)
    int hw, W, aoff;
    int tiles_per_image, tile_start;
    float stride;
};
struct HeadTailParams {
    CUtensorMap map[HT_MAX_ROWS][4];  // u2 [B*c2, hw], u3 [B*c3, hw], w2 [64, c2], w3 [nc, c3]
    HtRow row[HT_MAX_ROWS];
    int nrows, total_tiles, B, A;
    int nstages, stage_bytes;
    int off_w2, off_w3, off_bias, off_bar;  // byte offsets inside the (1024-aligned) dynamic shared memory
    int tmem_cols, buf_cols, nbufs;
    int ngroups;                            // epilogue groups launched (blockDim = 64 + 256 * ngroups)
    int srow;                               // score-summary row length (cerb_summary_row_len)
    int chunked;                            // 1: CTA i owns one contiguous run of tiles (few (task, level) changes, so few
                                            // weight reloads); 0: tiles dealt round-robin
};

// ---- PTX wrappers
__device__ __forceinline__ uint32_t ht_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ht_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void ht_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void ht_mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void ht_mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!ok);
}
// the same with a pause between polls: the 8-16 epilogue warps wait here for most of a memory-bound tile and must
// not take issue slots from the single producer / MMA lanes
__device__ __forceinline__ void ht_mbar_wait_backoff(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    for (;;) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
        if (ok) break;
        __nanosleep(40);
    }
}
#define HT_EVICT_FIRST 0x12F0000000000000ull  // L2 cache-hint encodings (CUTLASS cute/arch/copy_sm90_tma.hpp)
#define HT_EVICT_LAST 0x14F0000000000000ull
__device__ __forceinline__ void ht_tma_load_2d(uint32_t dst, const CUtensorMap* map, int col, int row, uint32_t bar, uint64_t hint) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(dst),
        "l"(map), "r"(bar), "r"(col), "r"(row), "l"(hint)
        : "memory");
}
__device__ __forceinline__ void ht_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void ht_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, cute/arch/mma_sm100_desc.hpp): start >> 4 in bits [0,14),
// LBO >> 4 in [16,30), SBO >> 4 in [32,46), version 1 in [46,48), layout type in [61,64) (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t ht_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 = 1 at [4,6), a/b format F16 = 0 at [7,10) / [10,13),
// a_major (1 = MN-major) at 15, b_major (0 = K-major) at 16, N >> 3 at [17,23), M >> 4 at [24,29)
__device__ __forceinline__ uint32_t ht_instr_desc(int M, int N) {
    return (1u << 4) | (1u << 15) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void ht_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void ht_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 16 / 8 consecutive accumulator columns of this thread's TMEM lane (issue only; ht_tmem_wait() before use)
__device__ __forceinline__ void ht_tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void ht_tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void ht_tmem_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// (task, level) row of global tile g; rows are sorted by tile_start and r only ever moves forward
__device__ __forceinline__ int ht_row_of(const HeadTailParams& P, int g, int r) {
    while (r + 1 < P.nrows && g >= P.row[r + 1].tile_start) ++r;
    return r;
}

__global__ void __launch_bounds__(HT_THREADS, 1) head_tail_kernel(const __grid_constant__ HeadTailParams P) {
    extern __shared__ __align__(1024) unsigned char ht_smem_raw[];
    // the dynamic window is only guaranteed 16-byte aligned: round up to the 1024 B the 128-byte swizzle needs
    unsigned char* const smem = ht_smem_raw + ((1024u - (ht_smem_u32(ht_smem_raw) & 1023u)) & 1023u);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int S = P.nstages;
    unsigned char* const sW2 = smem + P.off_w2;
    unsigned char* const sW3 = smem + P.off_w3;
    float* const sbias_all = reinterpret_cast<float*>(smem + P.off_bias);  // [HT_EPI_GROUPS][64 + HT_MAX_NCP]
    uint64_t* const bars = reinterpret_cast<uint64_t*>(smem + P.off_bar);
    // barrier map: full[0..S), empty[S..2S), wfull, wempty, tfull[HT_MAX_BUFS], tempty[HT_MAX_BUFS], then the TMEM base address slot
    const uint32_t bar0 = ht_smem_u32(bars);
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (S + s); };
    const uint32_t wfull = bar0 + 8u * (2 * S), wempty = wfull + 8u;
    auto tfull_bar = [&](int b) { return wfull + 16u + 8u * b; };
    auto tempty_bar = [&](int b) { return wfull + 16u + 8u * (HT_MAX_BUFS + b); };
    uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * S + 2 + 2 * HT_MAX_BUFS);
    const int NB = P.nbufs;

    if (tid == 0) {
        for (int s = 0; s < S; ++s) { ht_mbar_init(full_bar(s), 1); ht_mbar_init(empty_bar(s), 1); }
        ht_mbar_init(wfull, 1);
        ht_mbar_init(wempty, 1);
        for (int b = 0; b < HT_MAX_BUFS; ++b) { ht_mbar_init(tfull_bar(b), 1); ht_mbar_init(tempty_bar(b), HT_EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {  // TMEM: one warp allocates, the base address lands in shared memory
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(ht_smem_u32(tmem_slot)), "r"(P.tmem_cols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    ht_fence_before();
    __syncthreads();
    ht_fence_after();
    const uint32_t tmem = *tmem_slot;
    // this CTA's tile sequence: tile(i) = t0 + i * tstep for i in [0, n_my)
    const int G = gridDim.x;
    int t0, tstep, n_my;
    if (P.chunked) {
        const int q = P.total_tiles / G, rem = P.total_tiles - q * G;
        t0 = (int)blockIdx.x * q + min((int)blockIdx.x, rem);
        n_my = q + ((int)blockIdx.x < rem ? 1 : 0);
        tstep = 1;
    } else {
        t0 = blockIdx.x;
        tstep = G;
        n_my = (P.total_tiles - t0 + G - 1) / G;
    }

    if (warp == 0) {
        if (lane == 0) {
            // ------------------------------------------------ TMA producer
            int s = 0, cur = -1, r = 0;
            uint32_t ph = 0, wloads = 0;
            for (int i = 0; i < n_my; ++i) {
                const int g = t0 + i * tstep;
                r = ht_row_of(P, g, r);
                const HtRow& R = P.row[r];
                if (r != cur) {  // weights of a new (task, level): wait until the MMAs that read the old ones are done
                    ht_mbar_wait(wempty, (wloads & 1) ^ 1);
                    const int kb2 = (R.c2 + 63) >> 6, kb3 = (R.c3 + 63) >> 6;
                    ht_mbar_expect_tx(wfull, (uint32_t)(kb2 * 64 + kb3 * R.ncp) * 128u);
                    for (int kb = 0; kb < kb2; ++kb)
                        ht_tma_load_2d(ht_smem_u32(sW2) + kb * 64 * 128, &P.map[r][2], kb * 64, 0, wfull, HT_EVICT_LAST);
                    for (int kb = 0; kb < kb3; ++kb)
                        ht_tma_load_2d(ht_smem_u32(sW3) + kb * R.ncp * 128, &P.map[r][3], kb * 64, 0, wfull, HT_EVICT_LAST);
                    ++wloads;
                    cur = r;
                }
                const int lt = g - R.tile_start;
                const int b = lt / R.tiles_per_image, a0 = (lt - b * R.tiles_per_image) * HT_TILE;
                for (int op = 0; op < 2; ++op) {  // anchors past hw are zero-filled by TMA
                    const int c = op ? R.c3 : R.c2, rb = op ? R.rb3 : R.rb2;
                    const CUtensorMap* map = &P.map[r][op];
                    for (int k0 = 0; k0 < c; k0 += rb) {
                        ht_mbar_wait(empty_bar(s), ph ^ 1);
                        const uint32_t dst = ht_smem_u32(smem) + (uint32_t)s * P.stage_bytes;
                        ht_mbar_expect_tx(full_bar(s), (uint32_t)rb * 256u);
                        ht_tma_load_2d(dst, map, a0, b * c + k0, full_bar(s), HT_EVICT_FIRST);
                        ht_tma_load_2d(dst + rb * 128, map, a0 + 64, b * c + k0, full_bar(s), HT_EVICT_FIRST);
                        if (++s == S) { s = 0; ph ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // ------------------------------------------------ MMA issue: D1 in columns [0, 64) of a buffer, D2 in [64, 64 + ncp)
            int s = 0, cur = -1, r = 0, it = 0;
            uint32_t ph = 0, wloads = 0;
            for (; it < n_my; ++it) {
                const int g = t0 + it * tstep;
                r = ht_row_of(P, g, r);
                const HtRow& R = P.row[r];
                const int buf = it % NB;
                ht_mbar_wait(tempty_bar(buf), ((it / NB) & 1) ^ 1);  // the epilogue has drained this accumulator buffer
                if (r != cur) {
                    ht_mbar_wait(wfull, wloads & 1);
                    ++wloads;
                    cur = r;
                }
                ht_fence_after();
                const uint32_t d1 = tmem + (uint32_t)buf * P.buf_cols;
                for (int op = 0; op < 2; ++op) {
                    const int c = op ? R.c3 : R.c2, rb = op ? R.rb3 : R.rb2;
                    const int nrows_w = op ? R.ncp : 64;  // rows of one 64-wide K block of the weight image
                    const uint32_t wbase = ht_smem_u32(op ? sW3 : sW2);
                    const uint32_t idesc = ht_instr_desc(HT_TILE, nrows_w);
                    const uint32_t d = d1 + (op ? 64u : 0u);
                    int kk = 0;
                    for (int k0 = 0; k0 < c; k0 += rb) {
                        ht_mbar_wait(full_bar(s), ph);
                        ht_fence_after();
                        const uint32_t abase = ht_smem_u32(smem) + (uint32_t)s * P.stage_bytes;
                        for (int j = 0; j < rb / 16; ++j, ++kk) {
                            const uint64_t ad = ht_smem_desc(abase + j * 2048, (uint32_t)rb * 128u, 1024);
                            const uint64_t bd = ht_smem_desc(wbase + (kk >> 2) * nrows_w * 128 + (kk & 3) * 32, 0, 1024);
                            ht_mma(d, ad, bd, idesc, kk > 0);
                        }
                        ht_commit(empty_bar(s));  // the stage is free once these MMAs have read it
                        if (++s == S) { s = 0; ph ^= 1; }
                    }
                }
                if (it + 1 >= n_my || ht_row_of(P, g + tstep, r) != r) ht_commit(wempty);
                ht_commit(tfull_bar(buf));
            }
        }
    } else {
        // ------------------------------------------------ epilogue: thread = TMEM lane = anchor
        const int q = warp & 3;                 // a warp may only read the TMEM lane quadrant warp % 4
        const int grp = (warp - 2) / HT_EPI_WARPS;  // epilogue group: takes the tiles it = grp, grp + HT_EPI_GROUPS, ...
        const int h = ((warp - 2) >> 2) & 1;    // 0: sides l,r -> (cx, w) + even class chunks; 1: t,b -> (cy, h) + odd chunks
        const int etid = tid - 64 - grp * 32 * HT_EPI_WARPS;
        float* const sbias = sbias_all + grp * (64 + HT_MAX_NCP);
        int cur = -1, r = 0, it = grp;
        for (; it < n_my; it += P.ngroups) {
            const int g = t0 + it * tstep;
            r = ht_row_of(P, g, r);
            const HtRow& R = P.row[r];
            if (r != cur) {  // biases of the new (task, level) as floats (all epilogue threads are between tiles here)
                asm volatile("bar.sync %0, %1;" ::"r"(1 + grp), "n"(32 * HT_EPI_WARPS) : "memory");
                for (int i = etid; i < 64 + R.ncp; i += 32 * HT_EPI_WARPS)
                    sbias[i] = i < 64 ? __half2float(R.b2[i]) : (i - 64 < R.nc ? __half2float(R.b3[i - 64]) : 0.f);
                asm volatile("bar.sync %0, %1;" ::"r"(1 + grp), "n"(32 * HT_EPI_WARPS) : "memory");
                cur = r;
            }
            const int lt = g - R.tile_start;
            const int b = lt / R.tiles_per_image;
            const int a = (lt - b * R.tiles_per_image) * HT_TILE + q * 32 + lane;  // anchor inside the level
            const bool live = a < R.hw;
            const int buf = it % NB;
            const uint32_t trow = tmem + (uint32_t)buf * P.buf_cols + ((uint32_t)(q * 32) << 16);
            __half* __restrict__ yb = R.y + (size_t)b * (4 + R.nc) * P.A + R.aoff + a;
            ht_mbar_wait_backoff(tfull_bar(buf), (it / NB) & 1);
            ht_fence_after();
            {   // DFL sides h and h + 2 of this anchor -> centre and size on axis h (tal.py:198-204, yolo.py:98)
                uint32_t r0[16], r1[16];
                ht_tmem_ld16(trow + h * 16, r0);
                ht_tmem_ld16(trow + (h + 2) * 16, r1);
                ht_tmem_wait();
                float x0[CERB_REG_MAX], x1[CERB_REG_MAX];
#pragma unroll
                for (int k = 0; k < CERB_REG_MAX; k += 2) {  // conv output = half(acc + bias), like the reference's half conv
                    rnd2<__half>(__uint_as_float(r0[k]) + sbias[h * 16 + k], __uint_as_float(r0[k + 1]) + sbias[h * 16 + k + 1], x0[k], x0[k + 1]);
                    rnd2<__half>(__uint_as_float(r1[k]) + sbias[(h + 2) * 16 + k], __uint_as_float(r1[k + 1]) + sbias[(h + 2) * 16 + k + 1], x1[k], x1[k + 1]);
                }
                DVec<__half, 1> dlo, dhi;
                dlo.f[0] = dfl_expectation<__half>(x0);
                dhi.f[0] = dfl_expectation<__half>(x1);
                Pack<__half, 1> oc, os;
                axis_boxes<__half, 1>(dlo, dhi, live ? a : 0, R.W, h == 0, R.stride, oc, os);
                if (live) {
                    yb[(size_t)h * P.A] = oc.e[0];
                    yb[(size_t)(h + 2) * P.A] = os.e[0];
                }
            }
            // class sigmoids (yolo.py:99) + score summary; addresses advance by pointer, nothing is multiplied per class
            const size_t Astr = (size_t)P.A;
            __half* __restrict__ ycls = yb + 4 * Astr + (size_t)(h * 8) * Astr;
            const bool sm_on = R.smax != nullptr;
            __half* __restrict__ smp = sm_on ? R.smax + ((size_t)b * R.nc + h * 8) * P.srow + ((R.aoff + a) >> 3) : nullptr;
            const bool sm_writer = sm_on && live && (lane & 7) == 0;
            const float* __restrict__ bcls = sbias + 64;
            for (int c0 = h * 8; c0 < R.nc; c0 += 16, ycls += 16 * Astr, smp += 16 * (size_t)P.srow) {
                uint32_t rc[8];
                ht_tmem_ld8(trow + 64 + c0, rc);
                ht_tmem_wait();
#pragma unroll
                for (int k = 0; k < 8; k += 2) {
                    const int c = c0 + k;
                    if (c < R.nc) {  // (warp-uniform)
                        const bool two = c + 1 < R.nc;
                        float l0, l1;
                        rnd2<__half>(__uint_as_float(rc[k]) + bcls[c], __uint_as_float(rc[k + 1]) + bcls[c + 1], l0, l1);
                        const float2 sg = sigmoid2(make_float2(l0, l1));
                        const __half2 s2 = __floats2half2_rn(sg.x, sg.y);
                        if (live) {
                            ycls[k * Astr] = __low2half(s2);
                            if (two) ycls[(k + 1) * Astr] = __high2half(s2);
                        }
                        if (sm_on) {  // maximum over the 8 anchors of a 16-byte score vector (decode_pipe.cu)
                            __half2 m = live ? s2 : __floats2half2_rn(0.f, 0.f);
                            m = __hmax2(m, __shfl_xor_sync(0xffffffffu, m, 1));
                            m = __hmax2(m, __shfl_xor_sync(0xffffffffu, m, 2));
                            m = __hmax2(m, __shfl_xor_sync(0xffffffffu, m, 4));
                            if (sm_writer) {
                                smp[k * (size_t)P.srow] = __low2half(m);
                                if (two) smp[(k + 1) * (size_t)P.srow] = __high2half(m);
                            }
                        }
                    }
                }
            }
            ht_fence_before();
            __syncwarp();
            if (lane == 0) ht_mbar_arrive(tempty_bar(buf));
        }
    }
    // ---- teardown: every MMA has completed (the epilogue waited for the last tfull) and every TMEM read is done
    ht_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(P.tmem_cols));
    }
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*HtEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static HtEncodeTiledFn ht_encoder() {
    static HtEncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<HtEncodeTiledFn>(p);
    }();
    return fn;
}
// 2-D fp16 tensor [rows, cols] (cols contiguous), box {64 cols, box_rows}, 128-byte swizzle, out-of-range elements read as 0
static bool ht_encode(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
    const cuuint64_t gdim[2] = {cols, rows};
    const cuuint64_t gstride[1] = {cols * 2};
    const cuuint32_t box[2] = {64, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return ht_encoder()(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// channel rows per ring stage: the largest divisor of c that is a multiple of 16 and at most 128
static int ht_stage_rows(int c) {
    for (int d = 128; d >= 16; d -= 16)
        if (c % d == 0) return d;
    return 0;
}

extern "C" int cerb_head_tail(const void* const* box_feat, const void* const* cls_feat, const void* const* box_w,
                              const void* const* box_b, const void* const* cls_w, const void* const* cls_b, const int* c2,
                              const int* c3, const int* nc, int T, int L, int B, const int* H, const int* W,
                              const float* strides, int dtype, void* const* y, void* const* smax, int* summary_written,
                              void* stream) {
    cerb_clear_error();
    CERB_REQUIRE(box_feat && cls_feat && box_w && box_b && cls_w && cls_b && c2 && c3 && nc && H && W && strides && y,
                 "cerb_head_tail: null argument");
    CERB_REQUIRE(dtype == CERB_F16, "cerb_head_tail: fp16 only (tcgen05 kind::f16); run the convolutions and cerb_decode for fp32");
    CERB_REQUIRE(T >= 1 && T <= CERB_MAX_TASKS, "cerb_head_tail: T=%d outside [1, %d]", T, CERB_MAX_TASKS);
    CERB_REQUIRE(L >= 1 && L <= CERB_MAX_LEVELS, "cerb_head_tail: L=%d outside [1, %d]", L, CERB_MAX_LEVELS);
    CERB_REQUIRE(B >= 1, "cerb_head_tail: B=%d", B);
    CERB_REQUIRE(ht_encoder() != nullptr, "cerb_head_tail: cuTensorMapEncodeTiled is not available in this driver");
    int A = 0, aoff[CERB_MAX_LEVELS];
    for (int l = 0; l < L; ++l) {
        CERB_REQUIRE(H[l] >= 1 && W[l] >= 1, "cerb_head_tail: level %d is %dx%d", l, H[l], W[l]);
        CERB_REQUIRE((H[l] * W[l]) % 8 == 0, "cerb_head_tail: H*W of level %d (%d) must be a multiple of 8 (16-byte rows for TMA)", l, H[l] * W[l]);
        aoff[l] = A;
        A += H[l] * W[l];
    }
    int max_ncp = 0;
    for (int t = 0; t < T; ++t) {
        CERB_REQUIRE(nc[t] >= 1 && ((nc[t] + 15) & ~15) <= HT_MAX_NCP, "cerb_head_tail: nc[%d]=%d outside [1, %d]", t, nc[t], HT_MAX_NCP);
        CERB_REQUIRE(c2[t] >= 16 && c2[t] % 16 == 0 && c3[t] >= 16 && c3[t] % 16 == 0,
                     "cerb_head_tail: c2[%d]=%d / c3[%d]=%d must be multiples of 16", t, c2[t], t, c3[t]);
        CERB_REQUIRE((size_t)B * c2[t] < (1ull << 31) && (size_t)B * c3[t] < (1ull << 31), "cerb_head_tail: B * channels too large");
        CERB_REQUIRE(y[t] != nullptr, "cerb_head_tail: y[%d] is null", t);
        max_ncp = max(max_ncp, (nc[t] + 15) & ~15);
    }
    bool want_summary = smax != nullptr;
    for (int t = 0; t < T && want_summary; ++t) want_summary = smax[t] != nullptr;
    if (summary_written) *summary_written = want_summary ? 1 : 0;

    int dev = 0, smem_max = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);

    // launches of at most HT_MAX_ROWS (task, level) rows, whole tasks per launch
    const int tasks_per_launch = max(1, HT_MAX_ROWS / L);
    for (int t0 = 0; t0 < T; t0 += tasks_per_launch) {
        const int t1 = min(T, t0 + tasks_per_launch);
        HeadTailParams P;
        memset(&P, 0, sizeof(P));
        int r = 0, tiles = 0, stage_rows = 0, w2_bytes = 0, w3_bytes = 0, ncp_max = 0;
        for (int t = t0; t < t1; ++t)
            for (int l = 0; l < L; ++l, ++r) {
                HtRow& R = P.row[r];
                const int i = t * L + l, hw = H[l] * W[l];
                CERB_REQUIRE(box_feat[i] && cls_feat[i] && box_w[i] && box_b[i] && cls_w[i] && cls_b[i], "cerb_head_tail: null tensor (task %d, level %d)", t, l);
                CERB_REQUIRE(cerb_aligned(box_feat[i], 16) && cerb_aligned(cls_feat[i], 16) && cerb_aligned(box_w[i], 16) &&
                                 cerb_aligned(cls_w[i], 16),
                             "cerb_head_tail: tensors must be 16-byte aligned (task %d, level %d)", t, l);
                R.b2 = (const __half*)box_b[i];
                R.b3 = (const __half*)cls_b[i];
                R.y = (__half*)y[t];
                R.smax = want_summary ? (__half*)smax[t] : nullptr;
                R.c2 = c2[t]; R.c3 = c3[t]; R.nc = nc[t]; R.ncp = (nc[t] + 15) & ~15;
                R.rb2 = ht_stage_rows(c2[t]); R.rb3 = ht_stage_rows(c3[t]);
                R.hw = hw; R.W = W[l]; R.aoff = aoff[l]; R.stride = strides[l];
                R.tiles_per_image = (hw + HT_TILE - 1) / HT_TILE;
                R.tile_start = tiles;
                tiles += B * R.tiles_per_image;
                stage_rows = max(stage_rows, max(R.rb2, R.rb3));
                w2_bytes = max(w2_bytes, ((R.c2 + 63) / 64) * 64 * 128);
                w3_bytes = max(w3_bytes, ((R.c3 + 63) / 64) * R.ncp * 128);
                ncp_max = max(ncp_max, R.ncp);
                if (!ht_encode(&P.map[r][0], box_feat[i], (uint64_t)B * c2[t], hw, R.rb2) ||
                    !ht_encode(&P.map[r][1], cls_feat[i], (uint64_t)B * c3[t], hw, R.rb3) ||
                    !ht_encode(&P.map[r][2], box_w[i], 64, c2[t], 64) ||
                    !ht_encode(&P.map[r][3], cls_w[i], nc[t], c3[t], R.ncp)) {
                    cerb_set_error("cerb_head_tail: cuTensorMapEncodeTiled failed (task %d, level %d)", t, l);
                    return CERB_ECUDA;
                }
            }
        P.nrows = r; P.total_tiles = tiles; P.B = B; P.A = A;
        P.stage_bytes = stage_rows * 256;
        P.srow = (int)cerb_summary_row_len(A, CERB_F16);
        P.buf_cols = 64 + ncp_max;
        P.nbufs = 512 / P.buf_cols;  // >= 2 because ncp <= HT_MAX_NCP
        if (P.nbufs > HT_MAX_BUFS) P.nbufs = HT_MAX_BUFS;
        P.tmem_cols = 32;
        while (P.tmem_cols < P.nbufs * P.buf_cols) P.tmem_cols <<= 1;
        const int bias_bytes = HT_EPI_GROUPS * (64 + HT_MAX_NCP) * 4, bar_bytes = (2 * HT_MAX_STAGES + 2 + 2 * HT_MAX_BUFS + 2) * 8;
        const int fixed = w2_bytes + w3_bytes + bias_bytes + bar_bytes + 1024 /* alignment slack */;
        int S = (smem_max - fixed) / P.stage_bytes;
        if (S > HT_MAX_STAGES) S = HT_MAX_STAGES;
        int kv = 0;
        if (cerb_debug_knob("ht_stages", &kv) && kv >= 2 && kv < S) S = kv;
        P.chunked = cerb_debug_knob("ht_order", &kv) ? (kv != 0) : 1;
        int min_ch = 1 << 30;
        for (int i = 0; i < P.nrows; ++i) min_ch = min(min_ch, P.row[i].c2 + P.row[i].c3);
        P.ngroups = min_ch >= 384 ? 1 : HT_EPI_GROUPS;
        if (cerb_debug_knob("ht_groups", &kv) && kv >= 1 && kv <= HT_EPI_GROUPS) P.ngroups = kv;
        if (S < 2) {
            cerb_set_error("cerb_head_tail: %d + %d weight bytes and %d-byte stages do not fit %d bytes of shared memory", w2_bytes, w3_bytes, P.stage_bytes, smem_max);
            return CERB_ENOSPC;
        }
        P.nstages = S;
        P.off_w2 = S * P.stage_bytes;
        P.off_w3 = P.off_w2 + w2_bytes;
        P.off_bias = P.off_w3 + w3_bytes;
        P.off_bar = P.off_bias + bias_bytes;
        int smem = P.off_bar + bar_bytes + 1024;
        if (smem < 120 * 1024) smem = 120 * 1024;  // one CTA per SM whatever the model width (the TMEM allocation assumes it)
        if (want_summary && P.srow == 0) {
            cerb_set_error("cerb_head_tail: the score summary needs A %% 8 == 0 (A=%d)", A);
            return CERB_EINVAL;
        }
        cudaError_t e = cudaFuncSetAttribute(head_tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e == cudaSuccess) {
            head_tail_kernel<<<min(tiles, sms), 64 + 32 * HT_EPI_WARPS * P.ngroups, smem, (cudaStream_t)stream>>>(P);
            e = cudaGetLastError();
        }
        if (const int rc = cerb_launch_status("cerb_head_tail", e)) return rc;
    }
    return 0;
}
