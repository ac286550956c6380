// C ABI of libcerb_post.so (declared in include/cerb_post.h).
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/cerb_post.h"
#include "cerb_kernels.h"

static thread_local char g_err[512] = "";

// ---- test / tools knobs.  Results never depend on any of them (the parity tests run the paths they select against
// each other).  A knob set through cerb_debug_set() is THREAD-LOCAL: it affects only calls made by the thread that set
// it, so the library stays re-entrant; the CERB_DEBUG_* environment variables (tools/ A/B runs, one process per
// variant) are read ONCE per process.
enum Knob {
    K_DECODE_PIPE,    // 0 = register kernel (decode.cu), otherwise the pipelined kernel (value = variant id in CERB_DECODE_VARIANTS builds)
    K_DECODE_ORDER,   // DecodeParams::interleave_parts
    K_DECODE_VEC,     // cap on the anchors per thread
    K_DECODE_L2HINT,  // force the L2 evict-first input policy on / off
    K_NMS_MINB,       // 1 = 128-register NMS build, 2 = 64-register build
    K_NMS_PDL,        // 0 = launch the NMS kernel without programmatic stream serialization
    K_DECODE_PDL,     // 1 = launch the (pipelined) decode kernel WITH it: the single-stream overlapped schedule of pipeline.py
    K_CHUNK_CAP,      // lazy top-k: chunk capacity (16..4096)
    K_CHUNK_FIRST,    // lazy top-k: first chunk target
    K_HIST_SAMPLE,    // stride of the estimating histogram
    K_HT_ORDER,       // head-tail kernel: 0 = tiles dealt round-robin to the CTAs, 1 = one contiguous run of tiles per CTA
    K_HT_STAGES,      // head-tail kernel: cap on the activation ring depth (2..8)
    K_HT_GROUPS,      // head-tail kernel: epilogue groups (1 | 2)
    K_PUSH_CTAS,      // delivery push kernel: CTAs (tools/side_probe.py)
    K_PUSH_MODE,      // delivery push kernel: 0 = normal, 1 = no fences / flag (timing experiments only), 2 = no copy
    K_COUNT
};
static const char* const kKnobName[K_COUNT] = {"decode_pipe", "decode_order", "decode_vec", "decode_l2hint", "nms_minb",
                                               "nms_pdl",     "decode_pdl",     "chunk_cap",    "chunk_first", "hist_sample",  "ht_order",
                                               "ht_stages",   "ht_groups",   "push_ctas",
                                               "push_mode"};
static const char* const kKnobEnv[K_COUNT] = {"CERB_DEBUG_DECODE_PIPE", "CERB_DEBUG_DECODE_ORDER", "CERB_DEBUG_DECODE_VEC",
                                              "CERB_DEBUG_DECODE_L2HINT", "CERB_DEBUG_NMS_MINB", "CERB_DEBUG_NMS_PDL", "CERB_DEBUG_DECODE_PDL",
                                              nullptr, nullptr, nullptr, "CERB_DEBUG_HT_ORDER", "CERB_DEBUG_HT_STAGES",
                                              "CERB_DEBUG_HT_GROUPS", "CERB_DEBUG_PUSH_CTAS", "CERB_DEBUG_PUSH_MODE"};
struct KnobTable {
    int v[K_COUNT];
    bool set[K_COUNT];
};
static const KnobTable& env_knobs() {
    static const KnobTable t = [] {
        KnobTable k;
        memset(&k, 0, sizeof(k));
        for (int i = 0; i < K_COUNT; ++i)
            if (kKnobEnv[i])
                if (const char* ev = getenv(kKnobEnv[i])) { k.v[i] = atoi(ev); k.set[i] = true; }
        return k;
    }();
    return t;
}
static thread_local KnobTable g_knobs = {};
static bool knob(Knob k, int* out) {
    if (g_knobs.set[k]) { *out = g_knobs.v[k]; return true; }
    const KnobTable& e = env_knobs();
    if (e.set[k]) { *out = e.v[k]; return true; }
    return false;
}

// knob lookup by name for the other translation units (head_tail.cu)
bool cerb_debug_knob(const char* name, int* out) {
    for (int i = 0; i < K_COUNT; ++i)
        if (strcmp(name, kKnobName[i]) == 0) return knob((Knob)i, out);
    return false;
}

void cerb_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

void cerb_clear_error() { g_err[0] = 0; }

int cerb_launch_status(const char* fn, cudaError_t e) {
    if (e == cudaSuccess) return 0;
    cerb_set_error("%s: launch failed: %s", fn, cudaGetErrorString(e));
    return CERB_ECUDA;
}

int cerb_require_workspace(const char* fn, const void* ws, size_t have, size_t need) {
    if (need == 0 || (ws != nullptr && have >= need)) return 0;
    cerb_set_error("%s: workspace of %zu bytes required, got %zu", fn, need, have);
    return CERB_ENOSPC;
}

extern "C" int cerb_version(void) { return 100; }
extern "C" const char* cerb_last_error(void) { return g_err; }

extern "C" int cerb_debug_set(const char* name, int value) {
    CERB_REQUIRE(name != nullptr, "cerb_debug_set: null knob name");
    for (int i = 0; i < K_COUNT; ++i)
        if (strcmp(name, kKnobName[i]) == 0) {
            g_knobs.v[i] = value;
            g_knobs.set[i] = true;
            return 0;
        }
    cerb_set_error("cerb_debug_set: unknown knob '%s'", name);
    return CERB_EINVAL;
}
extern "C" int cerb_debug_reset(void) {
    memset(&g_knobs, 0, sizeof(g_knobs));
    return 0;
}

extern "C" int cerb_debug_set_chunking(int chunk_cap, int chunk_first) {
    if (chunk_cap == 0 && chunk_first == 0) { g_knobs.set[K_CHUNK_CAP] = g_knobs.set[K_CHUNK_FIRST] = false; return 0; }
    CERB_REQUIRE(chunk_cap >= 16 && chunk_cap <= 4096, "chunk_cap must be in [16, 4096], got %d", chunk_cap);
    CERB_REQUIRE(chunk_first >= 1, "chunk_first must be >= 1, got %d", chunk_first);
    g_knobs.v[K_CHUNK_CAP] = chunk_cap; g_knobs.set[K_CHUNK_CAP] = true;
    g_knobs.v[K_CHUNK_FIRST] = chunk_first; g_knobs.set[K_CHUNK_FIRST] = true;
    return 0;
}

extern "C" int cerb_debug_set_hist_sample(int stride) {
    CERB_REQUIRE(stride >= 0 && stride <= 64, "hist sample stride must be in [0, 64], got %d", stride);
    g_knobs.v[K_HIST_SAMPLE] = stride;
    g_knobs.set[K_HIST_SAMPLE] = stride != 0;
    return 0;
}

// bytes per element of a dtype code the post-head kernels take (fp16 / bf16 / fp32), 0 for any other
static size_t post_elt(int dtype) { return dtype == CERB_F16 || dtype == CERB_BF16 ? 2 : dtype == CERB_F32 ? 4 : 0; }

extern "C" size_t cerb_summary_row_len(int A, int dtype) {
    if (post_elt(dtype) == 0) return 0;
    const size_t V = 16 / post_elt(dtype);
    if (A <= 0 || (size_t)A % V) return 0;
    return ((size_t)A / V + V - 1) / V * V;
}

static int decode_common(const void* const* lvl, const void* const* cls_lvl, const int* nc, int T, int L, int B,
                         const int* H, const int* W, const float* strides, int dtype, void* const* y, void* const* smax,
                         int* summary_written, void* stream) {
    cerb_clear_error();
    CERB_REQUIRE(lvl && nc && H && W && strides && y, "cerb_decode: null argument");
    CERB_REQUIRE(T >= 1 && T <= CERB_MAX_TASKS, "cerb_decode: T=%d outside [1, %d]", T, CERB_MAX_TASKS);
    CERB_REQUIRE(L >= 1 && L <= CERB_MAX_LEVELS, "cerb_decode: L=%d outside [1, %d]", L, CERB_MAX_LEVELS);
    CERB_REQUIRE(B >= 0, "cerb_decode: negative batch");
    CERB_REQUIRE(post_elt(dtype) != 0, "cerb_decode: unsupported dtype %d", dtype);
    DecodeParams P;
    memset(&P, 0, sizeof(P));
    P.T = T; P.L = L; P.B = B; P.nrows = T * L;
    P.interleave_parts = dtype == CERB_F32 ? 1 : 2;  // measured best per dtype (profiles/r01_decode.md; bf16 takes fp16's)
    (void)knob(K_DECODE_ORDER, &P.interleave_parts);
    const size_t elt = post_elt(dtype);
    int vec = (int)(16 / elt);
    long A = 0;
    if (summary_written) *summary_written = 0;
    for (int l = 0; l < L; ++l) {
        CERB_REQUIRE(H[l] > 0 && W[l] > 0, "cerb_decode: level %d has empty shape %dx%d", l, H[l], W[l]);
        const long hw = (long)H[l] * W[l];
        CERB_REQUIRE(hw < (1l << 30), "cerb_decode: level %d too large", l);
        P.hw[l] = (int)hw; P.w[l] = W[l]; P.aoff[l] = (int)A; P.stride[l] = strides[l];
        A += hw;
        while (vec > 1 && hw % vec) vec >>= 1;
    }
    CERB_REQUIRE(A < (1l << 30), "cerb_decode: too many anchors");
    P.A = (int)A;
    for (int t = 0; t < T; ++t) {
        CERB_REQUIRE(nc[t] >= 1, "cerb_decode: task %d has nc=%d", t, nc[t]);
        P.nc[t] = nc[t];
        CERB_REQUIRE(y[t] != nullptr || B == 0, "cerb_decode: y[%d] is null", t);
        P.y[t] = y[t];
        while (vec > 1 && !cerb_aligned(y[t], vec * elt)) vec >>= 1;
        for (int l = 0; l < L; ++l) {
            const void* p = lvl[t * L + l];
            CERB_REQUIRE(p != nullptr || B == 0, "cerb_decode: lvl[%d][%d] is null", t, l);
            P.lvl[t][l] = p;
            while (vec > 1 && !cerb_aligned(p, vec * elt)) vec >>= 1;
            if (cls_lvl != nullptr) {
                const void* c = cls_lvl[t * L + l];
                CERB_REQUIRE(c != nullptr || B == 0, "cerb_decode_split: cls_lvl[%d][%d] is null", t, l);
                P.cls[t][l] = c;
                while (vec > 1 && !cerb_aligned(c, vec * elt)) vec >>= 1;
            }
        }
    }
    { int v = 0; if (knob(K_DECODE_VEC, &v) && v >= 1 && v < vec) vec = v; }
    if (B == 0) return 0;
    // the score summary (one maximum per 16-byte score vector) needs the full 128-bit path
    if (smax != nullptr && vec == (int)(16 / elt)) {
        bool all = true;
        for (int t = 0; t < T; ++t) all = all && smax[t] != nullptr && cerb_aligned(smax[t], 16);
        if (all) {
            for (int t = 0; t < T; ++t) P.smax[t] = smax[t];
            if (summary_written) *summary_written = 1;
        }
    }
    {
        // y and the score summary are read by the NMS kernel right after: when they fit in L2 with room to spare, the raw
        // heads (read once) are streamed with an evict-first policy so that they do not push the outputs out
        // (profiles/r01_decode.md: fp16 B=64 gains 2 us in decode and 1.4 us in NMS; fp32 B=64, whose outputs do not fit,
        // loses 7 us with the same hint)
        size_t out_bytes = 0;
        for (int t = 0; t < T; ++t)  // y [B, 4+nc, A] + score summary [B, nc, ~A/V]
            out_bytes += (size_t)B * ((size_t)(4 + nc[t]) * (size_t)P.A + (size_t)nc[t] * ((size_t)P.A / (16 / elt) + 8)) * elt;
        int dev = 0, l2 = 0;
        if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, dev) == cudaSuccess)
            P.l2_evict_first = out_bytes <= (size_t)l2 / 4 * 3;
        (void)knob(K_DECODE_L2HINT, &P.l2_evict_first);
        P.pdl = 0;
        (void)knob(K_DECODE_PDL, &P.pdl);
    }
    cudaError_t e = cudaErrorInvalidConfiguration;
    // software-pipelined kernel (decode_pipe.cu) whenever every row allows 16-byte vectors, else (or with the
    // decode_pipe knob at 0) the register-resident kernel of decode.cu.  (The persistent TMA variant measured in round 1
    // is slower on B200 and no longer part of the library: csrc/experiments/decode_tma.cu, profiles/r01_decode.md.)
    int pipe = 1;
    (void)knob(K_DECODE_PIPE, &pipe);
    if (pipe != 0 && vec == (int)(16 / elt)) e = cerb_launch_decode_pipe(P, dtype, pipe, (cudaStream_t)stream);
    if (e == cudaErrorInvalidConfiguration) {
        (void)cudaGetLastError();
        e = cerb_launch_decode(P, dtype, vec, (cudaStream_t)stream);
    }
    return cerb_launch_status("cerb_decode", e);
}

extern "C" int cerb_decode(const void* const* lvl, const int* nc, int T, int L, int B, const int* H, const int* W,
                           const float* strides, int dtype, void* const* y, void* const* smax, int* summary_written,
                           void* stream) {
    return decode_common(lvl, nullptr, nc, T, L, B, H, W, strides, dtype, y, smax, summary_written, stream);
}

extern "C" int cerb_decode_split(const void* const* box_lvl, const void* const* cls_lvl, const int* nc, int T, int L, int B,
                                 const int* H, const int* W, const float* strides, int dtype, void* const* y,
                                 void* const* smax, int* summary_written, void* stream) {
    CERB_REQUIRE(cls_lvl != nullptr, "cerb_decode_split: null argument");
    return decode_common(box_lvl, cls_lvl, nc, T, L, B, H, W, strides, dtype, y, smax, summary_written, stream);
}

extern "C" size_t cerb_nms_workspace_bytes(int T, int B, int max_det) {
    if (T <= 0 || B <= 0 || max_det <= 0) return 0;
    return cerb_nms_kept_ws_bytes(T, B, max_det);
}

// torch compares a half tensor with a Python scalar after casting the scalar to half
// (double -> float -> half), a bfloat16 tensor after casting it to bfloat16 (double -> float -> bf16, round to nearest
// even, as c10::BFloat16 does: bf16(0.3) = 0.30078125), a float tensor after casting it to float (general.py:411).
static float round_conf_to_dtype(double conf, int dtype) {
    float f = (float)conf;
    if (dtype == CERB_F16) f = __half2float(__float2half_rn(f));
    if (dtype == CERB_BF16) f = __bfloat162float(__float2bfloat16_rn(f));
    return f;
}
// torchvision's CPU kernel widens the fp32 quotient and compares with the double threshold:
// (double)q > thr  <=>  q > (largest float <= thr).
static float iou_threshold_as_float(double thr) {
    float f = (float)thr;
    if ((double)f > thr) f = nextafterf(f, -INFINITY);
    return f;
}

extern "C" int cerb_nms(const void* const* pred, const int* nc, int T, int B, int A, int dtype, double conf_thres,
                        double iou_thres, const int* classes, int n_classes, int agnostic, int multi_label,
                        int max_det, int max_nms, double max_wh, const void* const* smax, float* dets, int* counts, void* workspace, size_t workspace_bytes, void* stream) {
    return cerb_nms_stats(pred, nc, T, B, A, dtype, conf_thres, iou_thres, classes, n_classes, agnostic, multi_label, max_det,
                          max_nms, max_wh, smax, dets, counts, workspace, workspace_bytes, nullptr, stream);
}

static int nms_impl(const void* const* pred, const int* nc, int T, int B, int A, int dtype, double conf_thres, double iou_thres,
                    const int* classes, int n_classes, int agnostic, int multi_label, int max_det, int max_nms, double max_wh,
                    const void* const* smax, float* dets, int* counts, void* workspace, size_t workspace_bytes,
                    unsigned long long* stats, const cerb_delivery* dv, void* stream);

extern "C" int cerb_nms_stats(const void* const* pred, const int* nc, int T, int B, int A, int dtype, double conf_thres,
                              double iou_thres, const int* classes, int n_classes, int agnostic, int multi_label,
                              int max_det, int max_nms, double max_wh, const void* const* smax, float* dets, int* counts,
                              void* workspace, size_t workspace_bytes, unsigned long long* stats, void* stream) {
    return nms_impl(pred, nc, T, B, A, dtype, conf_thres, iou_thres, classes, n_classes, agnostic, multi_label, max_det, max_nms,
                    max_wh, smax, dets, counts, workspace, workspace_bytes, stats, nullptr, stream);
}

extern "C" int cerb_nms_deliver(const void* const* pred, const int* nc, int T, int B, int A, int dtype, double conf_thres,
                                double iou_thres, const int* classes, int n_classes, int agnostic, int multi_label,
                                int max_det, int max_nms, double max_wh, const void* const* smax, float* dets, int* counts,
                                void* workspace, size_t workspace_bytes, const cerb_delivery* dv, void* stream) {
    CERB_REQUIRE(dv != nullptr, "cerb_nms_deliver: null delivery");
    if (dv->flag_remote != nullptr) {
        CERB_REQUIRE(dv->ack_local && dv->seq_local && dv->done_local, "cerb_nms_deliver: null protocol word");
        CERB_REQUIRE(cerb_aligned(dv->flag_remote, 4) && cerb_aligned(dv->ack_local, 4) && cerb_aligned(dv->seq_local, 4) && cerb_aligned(dv->done_local, 4),
                     "cerb_nms_deliver: protocol words must be 4-byte aligned");
    }
    if (dv->push_src != nullptr) {
        CERB_REQUIRE(dv->flag_remote != nullptr && dv->push_dst != nullptr, "cerb_nms_deliver: push_src needs push_dst and the protocol words");
        CERB_REQUIRE(cerb_aligned(dv->push_src, 16) && cerb_aligned(dv->push_dst, 16) && dv->push_words % 4 == 0 && dv->push_words < (1ull << 32),
                     "cerb_nms_deliver: push buffers must be 16-byte aligned and hold a multiple of 4 words");
    }
    if (dv->collect_flags != nullptr) {
        CERB_REQUIRE(dv->collect_count != nullptr && dv->world >= 1 && dv->world <= 16 && dv->dst >= 0 && dv->dst < dv->world,
                     "cerb_nms_deliver: bad collect side (world=%d dst=%d)", dv->world, dv->dst);
        for (int r = 0; r < dv->world; ++r)
            CERB_REQUIRE(r == dv->dst || dv->collect_ack[r] != nullptr, "cerb_nms_deliver: collect_ack[%d] is null", r);
    }
    return nms_impl(pred, nc, T, B, A, dtype, conf_thres, iou_thres, classes, n_classes, agnostic, multi_label, max_det, max_nms,
                    max_wh, smax, dets, counts, workspace, workspace_bytes, nullptr, dv, stream);
}

extern "C" int cerb_deliver_push(const void* src_local, void* dst_remote, size_t n_words, void* flag_remote, const void* ack_local,
                                 void* seq_local, void* done_local, void* stream) {
    cerb_clear_error();
    CERB_REQUIRE(src_local && dst_remote && flag_remote && ack_local && seq_local && done_local, "cerb_deliver_push: null argument");
    CERB_REQUIRE(cerb_aligned(src_local, 16) && cerb_aligned(dst_remote, 16) && n_words % 4 == 0,
                 "cerb_deliver_push: buffers must be 16-byte aligned and hold a multiple of 4 words");
    PushParams P;
    P.src = (const float*)src_local;
    P.dst = (float*)dst_remote;
    P.n_words = n_words;
    P.flag = (unsigned*)flag_remote;
    P.ack = (const unsigned*)ack_local;
    P.seq = (unsigned*)seq_local;
    P.done = (unsigned*)done_local;
    // 16 bytes per thread and sweep: enough CTAs to cover the batch in ~4 sweeps, at most 32 (it shares the GPU with the
    // next batch's kernels)
    size_t ctas = (n_words / 4 + 4 * 256 - 1) / (4 * 256);
    if (ctas < 1) ctas = 1;
    if (ctas > 32) ctas = 32;
    int kv = 0;
    if (knob(K_PUSH_CTAS, &kv) && kv >= 1 && kv <= 1024) ctas = (size_t)kv;
    P.mode = knob(K_PUSH_MODE, &kv) ? kv : 0;
    return cerb_launch_status("cerb_deliver_push", cerb_launch_deliver_push(P, (int)ctas, (cudaStream_t)stream));
}

extern "C" int cerb_deliver_collect(const void* flags_local, void* const* ack_remote, void* collected_local, int world, int dst,
                                    void* stream) {
    cerb_clear_error();
    CERB_REQUIRE(flags_local && ack_remote && collected_local, "cerb_deliver_collect: null argument");
    CERB_REQUIRE(world >= 1 && world <= CERB_MAX_RANKS && dst >= 0 && dst < world, "cerb_deliver_collect: world=%d dst=%d (at most %d ranks)", world, dst, CERB_MAX_RANKS);
    CollectParams P;
    memset(&P, 0, sizeof(P));
    P.flags = (const unsigned*)flags_local;
    P.collected = (unsigned*)collected_local;
    P.world = world;
    P.dst = dst;
    for (int r = 0; r < world; ++r) {
        CERB_REQUIRE(r == dst || ack_remote[r] != nullptr, "cerb_deliver_collect: ack_remote[%d] is null", r);
        P.ack[r] = (unsigned*)ack_remote[r];
    }
    return cerb_launch_status("cerb_deliver_collect", cerb_launch_deliver_collect(P, (cudaStream_t)stream));
}

static int nms_impl(const void* const* pred, const int* nc, int T, int B, int A, int dtype, double conf_thres, double iou_thres,
                    const int* classes, int n_classes, int agnostic, int multi_label, int max_det, int max_nms, double max_wh,
                    const void* const* smax, float* dets, int* counts, void* workspace, size_t workspace_bytes,
                    unsigned long long* stats, const cerb_delivery* dv, void* stream) {
    cerb_clear_error();
    CERB_REQUIRE(pred && nc, "cerb_nms: null argument");
    CERB_REQUIRE(T >= 1 && T <= CERB_MAX_TASKS, "cerb_nms: T=%d outside [1, %d]", T, CERB_MAX_TASKS);
    CERB_REQUIRE(B >= 0 && A >= 0, "cerb_nms: negative size");
    CERB_REQUIRE(post_elt(dtype) != 0, "cerb_nms: unsupported dtype %d", dtype);
    CERB_REQUIRE(conf_thres >= 0.0 && conf_thres <= 1.0, "Invalid Confidence threshold %g, valid values are between 0.0 and 1.0", conf_thres);
    CERB_REQUIRE(iou_thres >= 0.0 && iou_thres <= 1.0, "Invalid IoU %g, valid values are between 0.0 and 1.0", iou_thres);
    CERB_REQUIRE(max_det >= 0 && max_nms >= 0, "cerb_nms: negative max_det/max_nms");
    if (B == 0) return 0;
    CERB_REQUIRE(counts != nullptr, "cerb_nms: counts is null");
    CERB_REQUIRE(dets != nullptr || max_det == 0, "cerb_nms: dets is null");
    NmsParams P;
    memset(&P, 0, sizeof(P));
    P.T = T; P.B = B; P.A = A;
    for (int t = 0; t < T; ++t) {
        CERB_REQUIRE(nc[t] >= 1, "cerb_nms: task %d has nc=%d", t, nc[t]);
        CERB_REQUIRE((double)A * nc[t] < 4294967295.0, "cerb_nms: A*nc overflows the 32-bit candidate index");
        CERB_REQUIRE(pred[t] != nullptr || A == 0, "cerb_nms: pred[%d] is null", t);
        P.pred[t] = pred[t];
        P.nc[t] = nc[t];
    }
    if (classes != nullptr && n_classes >= 0) {
        P.use_class_filter = 1;
        for (int i = 0; i < n_classes; ++i) {
            const int c = classes[i];
            if (c < 0 || c >= 32 * CERB_MAX_CLASS_WORDS) continue;  // can never match a class id
            P.class_mask[c >> 5] |= 1u << (c & 31);
        }
        for (int t = 0; t < T; ++t)
            CERB_REQUIRE(nc[t] <= 32 * CERB_MAX_CLASS_WORDS, "cerb_nms: class filter supports nc <= %d", 32 * CERB_MAX_CLASS_WORDS);
    }
    if (smax != nullptr) {
        const int V = (int)(16 / post_elt(dtype));
        CERB_REQUIRE(A % V == 0, "cerb_nms: a score summary needs A (%d) to be a multiple of %d", A, V);
        for (int t = 0; t < T; ++t) {
            CERB_REQUIRE(smax[t] != nullptr && cerb_aligned(smax[t], 16), "cerb_nms: smax[%d] is null or misaligned", t);
            CERB_REQUIRE(cerb_aligned(pred[t], 16), "cerb_nms: summary path needs 16-byte aligned predictions");
            P.smax[t] = smax[t];
        }
    }
    P.conf_thr = round_conf_to_dtype(conf_thres, dtype);
    P.iou_thr = iou_threshold_as_float(iou_thres);
    P.class_gap = agnostic ? 0.f : (float)max_wh;
    P.multi_label = multi_label ? 1 : 0;
    P.max_det = max_det;
    P.max_nms = max_nms;
    P.dets = dets;
    P.counts = counts;
    P.pair_counts = stats;
    if (dv != nullptr) {
        P.deliver_flag = (unsigned*)dv->flag_remote;
        P.deliver_ack = (const unsigned*)dv->ack_local;
        P.deliver_seq = (unsigned*)dv->seq_local;
        P.deliver_done = (unsigned*)dv->done_local;
        P.push_src = (const float*)dv->push_src;
        P.push_dst = (float*)dv->push_dst;
        P.push_words = (unsigned)dv->push_words;
        if (dv->push_src != nullptr) {  // <= 16 sweeps of 8 KB per delivery CTA, at most 16 CTAs (they take NMS-sized slots)
            size_t n = (dv->push_words / 4 + 512 * 16 - 1) / (512 * 16);
            P.deliver_ctas = (int)(n < 1 ? 1 : (n > 16 ? 16 : n));
        } else if (dv->collect_flags != nullptr) {
            P.deliver_ctas = 1;
        }
        if (dv->collect_flags != nullptr) {
            P.col_flags = (const unsigned*)dv->collect_flags;
            for (int r = 0; r < dv->world; ++r) P.col_ack[r] = (unsigned*)dv->collect_ack[r];
            P.col_collected = (unsigned*)dv->collect_count;
            P.col_world = dv->world;
            P.col_dst = dv->dst;
        }
    }
    const size_t need = cerb_nms_kept_ws_bytes(T, B, max_det);
    if (const int rc = cerb_require_workspace("cerb_nms", workspace, workspace_bytes, need)) return rc;
    if (need) {
        CERB_REQUIRE(cerb_aligned(workspace, 16), "cerb_nms: workspace must be 16-byte aligned");
        P.kept_ws = (float*)workspace;
    }
    P.chunk_cap = 4096;
    (void)knob(K_CHUNK_CAP, &P.chunk_cap);
    int first = max_det + max_det / 8 + 32;
    if (first < 128) first = 128;
    (void)knob(K_CHUNK_FIRST, &first);
    if (first > P.chunk_cap) first = P.chunk_cap;
    P.chunk_first = first;
    P.hist_sample = 8;
    (void)knob(K_HIST_SAMPLE, &P.hist_sample);
    P.force_minb = 0;
    (void)knob(K_NMS_MINB, &P.force_minb);
    P.pdl = 1;
    (void)knob(K_NMS_PDL, &P.pdl);
    // Class shortcut (see nms.cu): exact when the offsets and the window ends are integers small enough
    // for every fp32 sum  coordinate-bound + class * gap  to be exact (true for the reference's 7680).
    P.class_shortcut = 0;
    if (!agnostic && P.class_gap >= 8.f) {
        int ncmax = 0;
        for (int t = 0; t < T; ++t) ncmax = nc[t] > ncmax ? nc[t] : ncmax;
        const double gap = (double)P.class_gap;
        const double lo = -floor(gap / 8.0);
        if (gap == floor(gap) && gap * (double)(ncmax + 1) < 8388608.0) {
            P.class_shortcut = 1;
            P.tame_lo = (float)lo;
            P.tame_hi = (float)(lo + gap);
        }
    }
    return cerb_launch_status("cerb_nms", cerb_launch_nms(P, dtype, (cudaStream_t)stream));
}

extern "C" size_t cerb_cross_task_workspace_bytes(int T, int B, int max_det) {
    if (T <= 0 || B <= 0 || max_det <= 0) return 0;
    return cerb_cross_task_ws_bytes(T, B, max_det);
}

extern "C" int cerb_cross_task_ws(const float* dets, const int* counts, int T, int B, int max_det, const int* class_offset,
                                  double iou_thres, const float* scale, float* out, int* out_counts, void* workspace,
                                  size_t workspace_bytes, void* stream) {
    cerb_clear_error();
    CERB_REQUIRE(T >= 1 && T <= CERB_MAX_TASKS, "cerb_cross_task: T=%d outside [1, %d]", T, CERB_MAX_TASKS);
    CERB_REQUIRE(B >= 0 && max_det >= 0, "cerb_cross_task: negative size");
    CERB_REQUIRE(max_det <= 65535, "cerb_cross_task: max_det=%d exceeds 65535", max_det);
    if (B == 0) return 0;
    CERB_REQUIRE(counts && class_offset && out_counts && (dets || max_det == 0) && (out || max_det == 0), "cerb_cross_task: null argument");
    const size_t need = cerb_cross_task_ws_bytes(T, B, max_det);
    if (need && (workspace == nullptr || workspace_bytes < need)) {
        cerb_set_error("cerb_cross_task: T*max_det=%ld rows per image need a workspace of %zu bytes, got %zu", (long)T * max_det, need,
                       workspace ? workspace_bytes : (size_t)0);
        return CERB_ENOSPC;
    }
    CERB_REQUIRE(!need || cerb_aligned(workspace, 16), "cerb_cross_task: workspace must be 16-byte aligned");
    CrossTaskParams P;
    memset(&P, 0, sizeof(P));
    P.dets = dets; P.counts = counts; P.T = T; P.B = B; P.max_det = max_det;
    for (int t = 0; t < T; ++t) P.class_offset[t] = class_offset[t];
    P.iou_thr = (float)iou_thres;
    P.scale = scale; P.out = out; P.out_counts = out_counts;
    P.workspace = need ? (unsigned char*)workspace : nullptr;
    return cerb_launch_status("cerb_cross_task", cerb_launch_cross_task(P, (cudaStream_t)stream));
}

extern "C" int cerb_cross_task(const float* dets, const int* counts, int T, int B, int max_det, const int* class_offset,
                               double iou_thres, const float* scale, float* out, int* out_counts, void* stream) {
    return cerb_cross_task_ws(dets, counts, T, B, max_det, class_offset, iou_thres, scale, out, out_counts, nullptr, 0, stream);
}

extern "C" int cerb_decode_nms(const void* const* lvl, const int* nc, int T, int L, int B, const int* H, const int* W,
                               const float* strides, int dtype, void* const* y, void* const* smax, double conf_thres,
                               double iou_thres, const int* classes, int n_classes, int agnostic, int multi_label,
                               int max_det, int max_nms, double max_wh, float* dets, int* counts, void* workspace,
                               size_t workspace_bytes, void* stream) {
    int written = 0;
    int rc = cerb_decode(lvl, nc, T, L, B, H, W, strides, dtype, y, smax, &written, stream);
    if (rc) return rc;
    long A = 0;
    for (int l = 0; l < L; ++l) A += (long)H[l] * W[l];
    return cerb_nms((const void* const*)y, nc, T, B, (int)A, dtype, conf_thres, iou_thres, classes, n_classes, agnostic,
                    multi_label, max_det, max_nms, max_wh, written ? (const void* const*)smax : nullptr, dets, counts,
                    workspace, workspace_bytes, stream);
}

extern "C" int cerb_val_match(const float* dets, const int* counts, int B, int max_det, const float* labels,
                              const int* label_offsets, int max_labels_per_image, const float* iouv, int K,
                              unsigned char* correct, void* stream) {
    cerb_clear_error();
    CERB_REQUIRE(B >= 0 && max_det >= 0, "cerb_val_match: negative size");
    CERB_REQUIRE(K >= 1 && K <= 16, "cerb_val_match: K=%d thresholds outside [1, 16]", K);
    CERB_REQUIRE(max_labels_per_image >= 0 && max_labels_per_image <= 1024, "cerb_val_match: more than 1024 labels per image (%d)", max_labels_per_image);
    if (B == 0 || max_det == 0) return 0;
    CERB_REQUIRE(dets && counts && label_offsets && iouv && correct, "cerb_val_match: null argument");
    ValMatchParams P;
    memset(&P, 0, sizeof(P));
    P.dets = dets; P.counts = counts; P.labels = labels; P.label_offsets = label_offsets;
    P.B = B; P.max_det = max_det; P.K = K; P.correct = correct;
    for (int i = 0; i < K; ++i) P.iouv[i] = iouv[i];
    return cerb_launch_status("cerb_val_match", cerb_launch_val_match(P, max_labels_per_image, (cudaStream_t)stream));
}

// ConfusionMatrix.process_batch (cerberusdet/utils/metrics.py:273-370) for a batch of images
extern "C" int cerb_confusion_matrix(const float* dets, const int* counts, int B, int max_det, const float* labels,
                                     const int* label_offsets, int n_labels, int nc, double conf, double iou_thres,
                                     long long* matrix, int* cells, int* status, void* stream) {
    cerb_clear_error();
    CERB_REQUIRE(B >= 0 && n_labels >= 0, "cerb_confusion_matrix: negative size");
    CERB_REQUIRE(max_det >= 0 && max_det <= CERB_CM_MAX_DETS, "cerb_confusion_matrix: max_det=%d outside [0, %d]", max_det, CERB_CM_MAX_DETS);
    CERB_REQUIRE(nc >= 1 && nc <= CERB_CM_MAX_NC, "cerb_confusion_matrix: nc=%d outside [1, %d]", nc, CERB_CM_MAX_NC);
    CERB_REQUIRE(iou_thres >= 0.0, "cerb_confusion_matrix: iou_thres=%g must be >= 0", iou_thres);
    CERB_REQUIRE(label_offsets || (B <= 1 && n_labels <= CERB_CM_MAX_LABELS),
                 "cerb_confusion_matrix: without label_offsets, one image of at most %d labels (B=%d, n_labels=%d)",
                 CERB_CM_MAX_LABELS, B, n_labels);
    if (B == 0) return 0;
    CERB_REQUIRE(status && (dets || max_det == 0) && (labels || n_labels == 0), "cerb_confusion_matrix: null argument");
    ConfusionParams P;
    memset(&P, 0, sizeof(P));
    P.dets = dets; P.counts = counts; P.labels = labels; P.label_offsets = label_offsets;
    P.B = B; P.max_det = max_det; P.n_labels = n_labels; P.nc = nc;
    P.conf = (float)conf; P.iou_thr = (float)iou_thres;
    P.matrix = (unsigned long long*)matrix; P.cells = cells; P.status = status;
    return cerb_launch_status("cerb_confusion_matrix", cerb_launch_confusion(P, (cudaStream_t)stream));
}

// ------------------------------------------------------------------ training-time sibling decode (SURVEY 8f-4)
extern "C" int cerb_bbox_decode_fwd(const void* pred_dist, const void* anchor_points, long n_rows, int A, int reg_max,
                                    int dtype, void* out, void* stream) {
    cerb_clear_error();
    CERB_REQUIRE(post_elt(dtype) != 0, "cerb_bbox_decode_fwd: unsupported dtype %d", dtype);
    CERB_REQUIRE(reg_max == CERB_REG_MAX, "cerb_bbox_decode_fwd: reg_max=%d, only %d is supported (models/yolo.py:75)", reg_max, CERB_REG_MAX);
    CERB_REQUIRE(n_rows >= 0 && n_rows < (1l << 40) && A >= 0, "cerb_bbox_decode_fwd: bad sizes n_rows=%ld A=%d", n_rows, A);
    if (n_rows == 0) return 0;
    CERB_REQUIRE(A >= 1 && n_rows % A == 0, "cerb_bbox_decode_fwd: n_rows=%ld is not a multiple of A=%d", n_rows, A);
    CERB_REQUIRE(pred_dist && anchor_points && out, "cerb_bbox_decode_fwd: null argument");
    return cerb_launch_status("cerb_bbox_decode_fwd",
                              cerb_launch_bbox_decode_fwd(pred_dist, anchor_points, n_rows, A, dtype, out, (cudaStream_t)stream));
}

extern "C" int cerb_bbox_decode_bwd(const void* pred_dist, const void* grad_out, long n_rows, int reg_max, int dtype,
                                    void* grad_pred_dist, void* stream) {
    cerb_clear_error();
    CERB_REQUIRE(post_elt(dtype) != 0, "cerb_bbox_decode_bwd: unsupported dtype %d", dtype);
    CERB_REQUIRE(reg_max == CERB_REG_MAX, "cerb_bbox_decode_bwd: reg_max=%d, only %d is supported (models/yolo.py:75)", reg_max, CERB_REG_MAX);
    CERB_REQUIRE(n_rows >= 0 && n_rows < (1l << 40), "cerb_bbox_decode_bwd: bad n_rows=%ld", n_rows);
    if (n_rows == 0) return 0;
    CERB_REQUIRE(pred_dist && grad_out && grad_pred_dist, "cerb_bbox_decode_bwd: null argument");
    return cerb_launch_status("cerb_bbox_decode_bwd",
                              cerb_launch_bbox_decode_bwd(pred_dist, grad_out, n_rows, dtype, grad_pred_dist, (cudaStream_t)stream));
}

// ------------------------------------------------------------------ letterbox preprocessing (SURVEY row 10)
extern "C" int cerb_letterbox(const void* const* src, const int* h, const int* w, const long* pitch, const int* unpad_h,
                              const int* unpad_w, const int* top, const int* left, int B, int out_h, int out_w, int dtype,
                              void* out, void* stream) {
    cerb_clear_error();
    CERB_REQUIRE(B >= 0, "cerb_letterbox: negative batch %d", B);
    CERB_REQUIRE(out_h > 0 && out_w > 0 && out_h <= CERB_LB_MAX_SIDE && out_w <= CERB_LB_MAX_SIDE,
                 "cerb_letterbox: output size %dx%d outside [1, %d]", out_h, out_w, CERB_LB_MAX_SIDE);
    CERB_REQUIRE(dtype == CERB_F16 || dtype == CERB_F32, "cerb_letterbox: unsupported dtype %d", dtype);
    if (B == 0) return 0;
    CERB_REQUIRE(src && h && w && pitch && unpad_h && unpad_w && top && left && out, "cerb_letterbox: null argument");
    for (int i = 0; i < B; ++i) {
        CERB_REQUIRE(src[i] != nullptr, "cerb_letterbox: image %d is null", i);
        CERB_REQUIRE(h[i] > 0 && w[i] > 0 && h[i] <= CERB_LB_MAX_SIDE && w[i] <= CERB_LB_MAX_SIDE,
                     "cerb_letterbox: image %d has size %dx%d outside [1, %d]", i, h[i], w[i], CERB_LB_MAX_SIDE);
        CERB_REQUIRE(pitch[i] >= 3l * w[i], "cerb_letterbox: image %d has a row pitch of %ld bytes < 3 * width %d", i, pitch[i], w[i]);
        CERB_REQUIRE(unpad_h[i] > 0 && unpad_w[i] > 0, "cerb_letterbox: image %d resizes to an empty %dx%d", i, unpad_h[i], unpad_w[i]);
        CERB_REQUIRE(top[i] >= 0 && left[i] >= 0 && (long)top[i] + unpad_h[i] <= out_h && (long)left[i] + unpad_w[i] <= out_w,
                     "cerb_letterbox: image %d: %dx%d at top %d, left %d does not fit the %dx%d output", i, unpad_h[i],
                     unpad_w[i], top[i], left[i], out_h, out_w);
    }
    const size_t image_bytes = (size_t)3 * out_h * out_w * (dtype == CERB_F16 ? 2 : 4);
    LetterboxParams P;
    memset(&P, 0, sizeof(P));
    P.out_h = out_h;
    P.out_w = out_w;
    for (int b0 = 0; b0 < B; b0 += CERB_LB_MAX_IMAGES) {  // one launch up to CERB_LB_MAX_IMAGES images
        const int n = B - b0 < CERB_LB_MAX_IMAGES ? B - b0 : CERB_LB_MAX_IMAGES;
        for (int k = 0; k < n; ++k) {
            const int i = b0 + k;
            P.img[k] = LbImage{(const unsigned char*)src[i], (long long)pitch[i], h[i], w[i], unpad_h[i], unpad_w[i], top[i], left[i]};
        }
        P.out = (char*)out + (size_t)b0 * image_bytes;
        if (const int rc = cerb_launch_status("cerb_letterbox", cerb_launch_letterbox(P, n, dtype, (cudaStream_t)stream))) return rc;
    }
    return 0;
}
