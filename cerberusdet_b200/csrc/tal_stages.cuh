// The two score-reading stages of the TAL assigner (tal_assign.cu), included there once per score kind: TAL_BF16 false
// gives tal_topk_kernel / tal_assign_kernel (fp16 or fp32 scores, as TalParams::score_half says), true gives
// tal_topk_bf16_kernel / tal_assign_bf16_kernel (bf16 scores).  TAL_KERNEL(stage) names the kernel.  One source for both
// keeps them from drifting apart; kernels rather than a device function keep the fp16 / fp32 code exactly what it was
// (a body inlined from a device function schedules differently).

__global__ void __launch_bounds__(TAL_THREADS_A) TAL_KERNEL(tal_topk)(const __grid_constant__ TalParams P) {
    __shared__ unsigned long long skeys[(TAL_THREADS_A / 32) * TAL_MAX_TOPK];
    const int b = blockIdx.x / P.G, g = blockIdx.x - b * P.G, tid = threadIdx.x;
    int* out = P.topk_idx + ((size_t)b * P.G + g) * P.topk;
    if (!(P.mask_gt[(size_t)b * P.G + g] > 0.f)) {  // padded box: the reference zeroes its topk (tal.py:146-150)
        if (tid < P.topk) out[tid] = -1;
        return;
    }
    const float4 gt = reinterpret_cast<const float4*>(P.gt_boxes)[(size_t)b * P.G + g];
    const int label = (int)P.gt_labels[(size_t)b * P.G + g];
    // key = metric bits (metric >= 0: bit order = value order) in the high word, ~anchor in the low word:
    // descending key = metric descending, then anchor ascending
    unsigned long long best[TAL_MAX_TOPK];
#pragma unroll
    for (int i = 0; i < TAL_MAX_TOPK; ++i) best[i] = 0ull;  // (no real key is 0: ~anchor != 0)
    const int K = P.topk;
    for (int a = tid; a < P.A; a += TAL_THREADS_A) {
        const float2 pt = reinterpret_cast<const float2*>(P.anc)[a];
        float metric = 0.f;
        if (inside_gt(gt, pt.x, pt.y, P.eps)) {
            const float4 pb = reinterpret_cast<const float4*>(P.pd)[(size_t)b * P.A + a];
            metric = align_metric<TAL_BF16>(P, load_score<TAL_BF16>(P, b, a, label), ciou_clamped(gt, pb));
            if (!(metric >= 0.f)) metric = 0.f;  // NaN guard (scores are sigmoids, overlaps >= 0)
        }
        unsigned long long key = ((unsigned long long)__float_as_uint(metric) << 32) | (unsigned)(~a);
        if (key > best[K - 1]) {  // insertion into the descending list (fully unrolled: registers)
#pragma unroll
            for (int i = 0; i < TAL_MAX_TOPK; ++i) {
                if (i < K && key > best[i]) { const unsigned long long t = best[i]; best[i] = key; key = t; }
            }
        }
    }
    // merge without block-wide rounds: every warp pops the K largest heads of its 32 sorted lists with shuffles (keys are
    // unique, so exactly one lane owns each maximum and shifts its list), then warp 0 does the same over the 8 * K survivors
    const int lane = tid & 31, warp = tid >> 5;
    unsigned long long mine = 0ull;  // lane r ends up with the warp's r-th largest key
    for (int r = 0; r < K; ++r) {
        unsigned long long m = best[0];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long t = __shfl_xor_sync(0xffffffffu, m, o);
            m = t > m ? t : m;
        }
        if (best[0] == m && m != 0ull) {
#pragma unroll
            for (int i = 0; i + 1 < TAL_MAX_TOPK; ++i) best[i] = best[i + 1];
            best[TAL_MAX_TOPK - 1] = 0ull;
        }
        if (lane == r) mine = m;
    }
    if (lane < K) skeys[warp * TAL_MAX_TOPK + lane] = mine;
    __syncthreads();
    if (warp == 0) {
        constexpr int NW = TAL_THREADS_A / 32;
        unsigned long long k[(NW * TAL_MAX_TOPK + 31) / 32];
#pragma unroll
        for (int j = 0; j < (NW * TAL_MAX_TOPK + 31) / 32; ++j) {
            const int idx = lane + 32 * j, w = idx / TAL_MAX_TOPK, i = idx - w * TAL_MAX_TOPK;
            k[j] = (w < NW && i < K) ? skeys[idx] : 0ull;
        }
        for (int r = 0; r < K; ++r) {
            unsigned long long m = 0ull;
#pragma unroll
            for (int j = 0; j < (NW * TAL_MAX_TOPK + 31) / 32; ++j) m = k[j] > m ? k[j] : m;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long t = __shfl_xor_sync(0xffffffffu, m, o);
                m = t > m ? t : m;
            }
#pragma unroll
            for (int j = 0; j < (NW * TAL_MAX_TOPK + 31) / 32; ++j)
                if (k[j] == m) k[j] = 0ull;
            if (lane == 0) out[r] = m != 0ull ? (int)(~(unsigned)(m & 0xffffffffull)) : -1;
        }
    }
}

__global__ void __launch_bounds__(TAL_THREADS_B) TAL_KERNEL(tal_assign)(const __grid_constant__ TalParams P) {
    __shared__ float pos_align[TAL_MAX_GT], pos_ov[TAL_MAX_GT];
    const int b = blockIdx.x, tid = threadIdx.x;
    int* cnt = P.cnt + (size_t)b * P.A;
    int* gsel = P.gsel + (size_t)b * P.A;
    float* aval = P.aval + (size_t)b * P.A;
    const float4* gts = reinterpret_cast<const float4*>(P.gt_boxes) + (size_t)b * P.G;
    const float4* pds = reinterpret_cast<const float4*>(P.pd) + (size_t)b * P.A;
    for (int a = tid; a < P.A; a += TAL_THREADS_B) { cnt[a] = 0; gsel[a] = 0; }
    for (int g = tid; g < P.G; g += TAL_THREADS_B) { pos_align[g] = 0.f; pos_ov[g] = 0.f; }
    __syncthreads();
    // mask_pos = is_in_topk * mask_in_gts * mask_gt (tal.py:118): the (box, anchor) pairs of the topk lists that lie inside
    for (int i = tid; i < P.G * P.topk; i += TAL_THREADS_B) {
        const int g = i / P.topk;
        const int a = P.topk_idx[((size_t)b * P.G + g) * P.topk + (i - g * P.topk)];
        if (a < 0) continue;
        const float2 pt = reinterpret_cast<const float2*>(P.anc)[a];
        if (!inside_gt(gts[g], pt.x, pt.y, P.eps)) continue;
        atomicAdd(&cnt[a], 1);
        gsel[a] = g;  // unique writer when exactly one box claims the anchor; recomputed below otherwise
    }
    __syncthreads();
    // select_highest_overlaps (tal.py:31-53): an anchor claimed by several boxes goes to argmax over ALL boxes of the
    // overlap (first maximum), padded boxes included
    for (int a = tid; a < P.A; a += TAL_THREADS_B) {
        if (cnt[a] > 1) {
            const float4 pb = pds[a];
            float bestv = -1.f;
            int bestg = 0;
            for (int g = 0; g < P.G; ++g) {
                const float ov = ciou_clamped(gts[g], pb);
                if (ov > bestv) { bestv = ov; bestg = g; }
            }
            gsel[a] = bestg;
        }
    }
    __syncthreads();
    // per-box maxima of metric and overlap over the final positives (tal.py:103-106); values are >= 0, so the integer
    // order of their bit patterns is their order
    for (int a = tid; a < P.A; a += TAL_THREADS_B) {
        if (cnt[a] > 0) {
            const int g = gsel[a];
            const float ov = ciou_clamped(gts[g], pds[a]);
            float al = align_metric<TAL_BF16>(P, load_score<TAL_BF16>(P, b, a, (int)P.gt_labels[(size_t)b * P.G + g]), ov);
            if (!(al >= 0.f)) al = 0.f;
            aval[a] = al;
            atomicMax(reinterpret_cast<int*>(&pos_align[g]), __float_as_int(al));
            atomicMax(reinterpret_cast<int*>(&pos_ov[g]), __float_as_int(ov));
        }
    }
    __syncthreads();
    // get_targets (tal.py:153-178) + normalisation (:107-108); background anchors point at box 0 like the reference's argmax
    for (int a = tid; a < P.A; a += TAL_THREADS_B) {
        const bool fg = cnt[a] > 0;
        const int g = fg ? gsel[a] : 0;
        const size_t o = (size_t)b * P.A + a;
        P.target_labels[o] = (long long)P.gt_labels[(size_t)b * P.G + g];
        reinterpret_cast<float4*>(P.target_bboxes)[o] = gts[g];
        P.fg_mask[o] = fg ? 1 : 0;
        P.target_gt_idx[o] = g;
    }
    for (int g = tid; g < P.G; g += TAL_THREADS_B) {
        P.pos[((size_t)b * P.G + g) * 2] = pos_align[g];
        P.pos[((size_t)b * P.G + g) * 2 + 1] = pos_ov[g];
    }
}
