// proposals.cu -- pre-NMS top-k, NMS and the fused proposal stage, one CTA per image.
//
// Replaces tf.nn.top_k + tf.gather (predictor.py:58-60), non_max_suppression ->
// tf.image.combined_non_max_suppression (utils/bbox_utils.py:48-70) and their composition
// (SURVEY.md 8a row P).
//
// Order: every entry gets the unique 64-bit composite  (orderable(score) << 32) | ~index , so
// "larger composite" == "higher score, and among equal scores the LOWER index" -- the order of
// tf.nn.top_k and the order in which TF's NMS pops candidates ([TF-internal]; ties documented in
// the oracle).  NMS is lazy: it consumes candidates in BATCHES of at most 1024 ranks and usually stops
// (max_output_size kept) inside the first batch, so the other ~5000 of the pre-NMS top-6000 are
// never sorted, gathered or decoded.  Per batch, inside the CTA (proposal_kernel):
//   1 SELECT a threshold tau with 11-bit histograms (the first one built while the keys are staged):
//     the batch is every remaining composite >= tau, between 768 and 1024 of them (fewer: all that remain)
//   2 the batch's entries, from a short candidate list the select copied out, or one compaction sweep
//   3 COUNTING SORT on 11 key bits, entries of a bin ranked by comparison (bitonic network for long bins)
//   4 top-k outputs, or greedy NMS rounds of 128 candidates: test against the kept list, build
//     predecessor masks inside the round, resolve them in one warp with ballots.
//   In the fused mode boxes are decoded (+clipped) on the fly, for the examined candidates only.
//
// Kernels of this file:
//   proposal_kernel<T>             one CTA of T = 512 (two per SM) or 1024 threads per image (the default above 8
//                                  images per launch; launch_one picks T)
//   proposal_cluster_kernel<CL,T>  the same algorithm on a thread-block cluster per image (<= 8 images per launch;
//                                  also MODE_RANK / presorted launches of the host pipeline's two-phase transfer)
//   nms_mask_kernel, nms_sweep_kernel   matrix NMS over the ranks of a MODE_RANK launch (opt-in, TFRPN_NMS_PATH=matrix)
//   gather_rows_kernel             candidate rows of a page-locked host tensor -> compact device array (pipeline.cu)
//   pre_hist / pre_count / pre_scatter_kernel   large-N prefilter (N >= 40 000)
//   nms_mc_stage_kernel / nms_mc_row_count + nms_mc_row_scatter_kernel, nms_mc_merge_kernel   multi-class combined
//                                  NMS around proposal_kernel (tfrpn_nms_multiclass)
// The NMS pair test runs behind a cheap conservative pre-test (nms_maybe / nms_maybe2): see there.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include <cooperative_groups.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace tfrpn {

constexpr int BATCH = 1024;         // ranks sorted per batch: BATCH / T composites per thread of proposal_kernel<T>
constexpr int NMS_CHUNK = 128;

enum { MODE_TOPK = 0, MODE_NMS = 1, MODE_PROPOSALS = 2, MODE_RANK = 3 };

#ifdef TFRPN_PHASE_TIMING
// debug build only (make EXTRA=-DTFRPN_PHASE_TIMING): cycles per phase of CTA 0, read with tfrpn_debug_phase_cycles
__device__ long long g_phase[32];
__device__ long long g_img[4096];   // per CTA: start clock (globaltimer ns), end, rounds
__device__ __forceinline__ long long gtimer() { long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define PH_DECL __shared__ long long ph_acc[32]; __shared__ long long ph_last; \
    if (threadIdx.x == 0) { for (int q_ = 0; q_ < 32; ++q_) ph_acc[q_] = 0; ph_last = clock64(); if (blockIdx.x < 1024) g_img[blockIdx.x * 4] = gtimer(); }
#define PH(id) do { if (threadIdx.x == 0 && blockIdx.x == 0) { const long long t_ = clock64(); ph_acc[id] += t_ - ph_last; ph_last = t_; } } while (0)
#define PH_FLUSH do { if (threadIdx.x == 0 && blockIdx.x < 1024) g_img[blockIdx.x * 4 + 1] = gtimer(); \
    if (threadIdx.x == 0 && blockIdx.x == 0) { for (int q_ = 0; q_ < 32; ++q_) g_phase[q_] = ph_acc[q_]; } } while (0)
#else
#define PH_DECL
#define PH(id) do {} while (0)
#define PH_FLUSH do {} while (0)
#endif



struct PropParams {
    int mode;
    int N;       // entries per image
    int k;       // requested top-k (<= N)
    int staged;  // score keys staged in shared memory (N * 4 bytes)
    const float* scores;  // (B,N)
    int use_sthr;
    float score_threshold;
    const float4* boxes;   // MODE_TOPK gather source / MODE_NMS input
    long long box_stride;  // elements between images (0 = shared (N,4))
    const float4* reg;     // MODE_PROPOSALS: (B,N,4) head regression output
    const float4* anchors; // MODE_PROPOSALS: (N,4)
    const AnchorGen* gen;  //   ... or null `anchors` and the generator: anchors are regenerated in registers
    float4 var;
    int clip_decoded;
    float* values;   // MODE_TOPK (B,k)
    int* indices;    // MODE_TOPK (B,k)
    float4* gathered;
    int rows, max_out;
    int mo_pad;  // max_out rounded up to a multiple of 4 (keeps the carve 16-byte aligned)
    IouThreshold iou_thr;
    int clip_out;
    float4* out_boxes;
    float* out_scores;
    float* out_classes;
    int* valid;
    int* keep_idx;
    // large-N prefilter (launch_prefiltered): per-image entry counts over a compacted candidate array
    const int* counts;        // entries of image b (null: N)
    const int* remap;         // (B,N) candidate position -> index in the caller's arrays (null: identity)
    int anchors_batched;      // MODE_PROPOSALS / predict_topk: anchors are (B,N,4) (gathered candidates)
    const int* flags;         // (B,) 1 = the candidate array of this image overflowed
    int flag_mode;            // 0: run every image; 1: skip flagged images; 2: run flagged images only
    int* flags_out;           // NMS over a TRUNCATED candidate set: raise flags[b] when the candidates ran out
    int full_n;               //   before max_out boxes were kept and the image has more than its candidates
    unsigned long long* rows_fetched;   // optional device counter: rows of `reg` / `boxes` the launch loaded
    // two-phase flow (pipeline.cu, cluster kernel only): a MODE_RANK launch writes the first batch of ranks of every
    // image; the host gathers those rows of `reg`; a `presorted` launch then runs NMS over that batch alone.
    int* rank_idx;              // MODE_RANK out / presorted in: (B, BATCH) entry index by rank
    int* rank_n;                // (B,) ranks in the batch
    int* rank_more;             // (B,) 1: ranks beyond the batch exist and may be consumed
    int presorted;
    const float4* reg_compact;  // presorted: rows of `reg` in rank order, (B, compact_stride); null: read `reg`
    int compact_rows;           //   ranks >= compact_rows read `reg`, or end the batch when `reg` is null
    int compact_stride;
    int* redo_flags;            // presorted out (B,): 1 = the batch ran out before max_out boxes were kept (the
                                //   unfiltered kernel must redo the image), else 0
    // matrix NMS (nms_mask_kernel + nms_sweep_kernel) over the first nms_rows ranks of the rank launch
    unsigned int* nms_mask;     // (B, nms_rows, mask_words): bit j%32 of word j/32 of row i set iff j < i and j suppresses i
    int nms_rows, mask_words;
};

// proposal_kernel front end (see there): 11-bit digits, 2048-bin shared histograms scanned two bins per thread
constexpr int SEL_BITS = 11;
constexpr int SEL_NB = 1 << SEL_BITS;
constexpr int SEL_FLOOR = BATCH * 3 / 4;   // a batch may end at a histogram bin edge once it holds this many entries
constexpr int SEL_LIST = 2 * BATCH;        // candidate-list capacity: the sort buffer
constexpr int SEG_MAX = 32;                // longest counting-sort bin ordered by comparisons; longer -> bitonic network

struct PropShared {
    unsigned int wtot[32], wmax[32];
    unsigned int digit, excl, bin_count;
    unsigned int count;      // entries above the score threshold
    unsigned int lcount;     // candidate-list cursor
    unsigned int kmax;       // largest key of the image
    int nk;
    int nalive;
};

// anchor i of the image: read from the (N,4) tensor, or regenerated (utils/bbox_utils.py:23-46)
__device__ __forceinline__ float4 anchor_of(const PropParams& p, const float4* anc, uint32_t i) {
    return p.gen ? anchor_at(*p.gen, (int)i) : ldg_f4(anc + i);
}

// score -> sortable key; entries at or below the score threshold get key 0 (below every real key)
__device__ __forceinline__ uint32_t score_key(float s, int use_sthr, float sthr) {
    if (use_sthr && !(s > sthr)) return 0u;
    return orderable(s);
}
__device__ __forceinline__ unsigned long long make_comp(uint32_t key, int i) {
    return ((unsigned long long)key << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)i);
}

// Histogram bins of thread t of a T-thread CTA, scanned from the top: PER = SEL_NB / T bins, c[q] = bin
// SEL_NB-1-PER*t-q.  Four bins are one aligned 16-byte word (read and written as one).
template <int T>
__device__ __forceinline__ void own_bins_load(const unsigned int* hist, unsigned (&c)[SEL_NB / T]) {
    constexpr int PER = SEL_NB / T;
    const int t = threadIdx.x;
    if constexpr (PER == 4) {
        const uint4 v = reinterpret_cast<const uint4*>(hist)[SEL_NB / 4 - 1 - t];
        c[0] = v.w; c[1] = v.z; c[2] = v.y; c[3] = v.x;
    } else {
#pragma unroll
        for (int q = 0; q < PER; ++q) c[q] = hist[SEL_NB - 1 - PER * t - q];
    }
}
template <int T>
__device__ __forceinline__ void own_bins_store(unsigned int* hist, const unsigned (&c)[SEL_NB / T]) {
    constexpr int PER = SEL_NB / T;
    const int t = threadIdx.x;
    if constexpr (PER == 4) {
        reinterpret_cast<uint4*>(hist)[SEL_NB / 4 - 1 - t] = make_uint4(c[3], c[2], c[1], c[0]);
    } else {
#pragma unroll
        for (int q = 0; q < PER; ++q) hist[SEL_NB - 1 - PER * t - q] = c[q];
    }
}

// Block-wide scan of SEL_NB histogram bins from the top over the own bins c[] (own_bins_load).
// excl = entries in the bins above c[0], total = all entries, cmax = the fullest bin.  One barrier inside; sh->wtot /
// sh->wmax may be rewritten only after another barrier.
template <int T>
__device__ __forceinline__ void hist_scan_desc(const unsigned int* hist, unsigned (&c)[SEL_NB / T], unsigned& excl,
                                               unsigned& total, unsigned& cmax, PropShared* sh) {
    constexpr int WARPS = T / 32;
    const int lane = lane_id(), warp = warp_id();
    own_bins_load<T>(hist, c);
    unsigned s = 0, m = 0;
#pragma unroll
    for (int q = 0; q < SEL_NB / T; ++q) { s += c[q]; m = max(m, c[q]); }
    const unsigned incl = (unsigned)warp_incl_scan((int)s);
    m = __reduce_max_sync(0xffffffffu, m);
    if (lane == 31) { sh->wtot[warp] = incl; sh->wmax[warp] = m; }
    __syncthreads();
    const unsigned w = lane < WARPS ? sh->wtot[lane] : 0u;
    const unsigned wi = (unsigned)warp_incl_scan((int)w);
    total = __shfl_sync(0xffffffffu, wi, 31);
    excl = __shfl_sync(0xffffffffu, wi - w, warp) + incl - s;
    cmax = __reduce_max_sync(0xffffffffu, lane < WARPS ? sh->wmax[lane] : 0u);
}

// TF CombinedNonMaxSuppression IOU on canonicalised boxes ([TF-internal]); c = (ymin,xmin,ymax,xmax).
// Returns IOU(i,j) > thr exactly as TF evaluates it: 0 if either area <= 0; otherwise
// RN(inter / ((ai + aj) - inter)) > thr, decided without the division (common.cuh: iou_exceeds).
__device__ __forceinline__ bool nms_suppresses(float4 ci, float ai, float4 cj, float aj, const IouThreshold& t) {
    if (ai > 0.0f && aj > 0.0f) {
        float iymin = fmaxf(ci.x, cj.x), ixmin = fmaxf(ci.y, cj.y);
        float iymax = fminf(ci.z, cj.z), ixmax = fminf(ci.w, cj.w);
        float inter = __fmul_rn(fmaxf(__fsub_rn(iymax, iymin), 0.0f), fmaxf(__fsub_rn(ixmax, ixmin), 0.0f));
        // inter == 0  =>  IOU == +0 exactly (union >= max(ai, aj) > 0)
        if (inter != 0.0f) return iou_exceeds(inter, __fsub_rn(__fadd_rn(ai, aj), inter), t);
    }
    return 0.0f > t.thr;
}

// The same decision for SANITISED boxes and a normal positive threshold (t.fast): a box whose area is not
// > 0 has been replaced by FAR_BOX with area 0 when it was staged, so its intersection with anything is
// +0 and the area guards leave the loop; the two float pre-filters of iou_exceeds are evaluated without
// branches and only a quotient within 2^-12 of the threshold (or a degenerate pair) takes the exact path.
__device__ __forceinline__ bool nms_suppresses_fast(float4 ci, float ai, float4 cj, float aj, const IouThreshold& t) {
    const float iymin = fmaxf(ci.x, cj.x), ixmin = fmaxf(ci.y, cj.y);
    const float iymax = fminf(ci.z, cj.z), ixmax = fminf(ci.w, cj.w);
    const float inter = __fmul_rn(fmaxf(__fsub_rn(iymax, iymin), 0.0f), fmaxf(__fsub_rn(ixmax, ixmin), 0.0f));
    const float uni = __fsub_rn(__fadd_rn(ai, aj), inter);
    const bool sure = inter > __fmul_rn(t.hi_f, uni);
    const bool maybe = inter >= __fmul_rn(t.lo_f, uni);
    if (maybe && !sure) {
        if (inter == 0.0f) return false;   // degenerate pair (union 0): IOU is 0, and 0 > thr is false for thr > 0
        const double prod = __dmul_rn(t.mid, (double)uni);
        const double di = (double)inter;
        return di > prod || (di == prod && t.tie_up);
    }
    return sure;
}
#define TFRPN_FAR_BOX make_float4(3.0e38f, 3.0e38f, -3.0e38f, -3.0e38f)

// Cheap conservative pre-test for SANITISED boxes and t.fast: `false` means IoU is certainly not > thr, so the pair
// test above is only evaluated for the few pairs that pass (a candidate meets at most a handful of boxes it really
// overlaps that much).  IoU = inter / (S - inter) > thr  <=>  inter > thr / (1 + thr) * S with S = ai + aj; lo_s
// carries a 2^-10 margin, three orders of magnitude above the rounding of either side, so no true suppression can
// fail it.  Only the height is clamped at 0: a negative width makes the product <= 0 (or NaN for the far-away empty
// box: -inf * 0), which fails `>=` as well.  11 instructions instead of 19 -- and 17 for two kept boxes in the packed
// form (FADD2 / FMUL2; the min / max have no packed form).
__device__ __forceinline__ bool nms_maybe(float4 ci, float ai, float4 cj, float aj, float lo_s) {
    const float h = fmaxf(__fsub_rn(fminf(ci.z, cj.z), fmaxf(ci.x, cj.x)), 0.0f);
    const float w = __fsub_rn(fminf(ci.w, cj.w), fmaxf(ci.y, cj.y));
    return __fmul_rn(h, w) >= __fmul_rn(lo_s, __fadd_rn(ai, aj));
}
// bit 0: box k0 may suppress / be suppressed by c, bit 1: box k1
__device__ __forceinline__ unsigned nms_maybe2(float4 c, f32x2 ca2, float4 k0, float a0, float4 k1, float a1, f32x2 lo2) {
    const f32x2 y_top = pack2(fmaxf(c.x, k0.x), fmaxf(c.x, k1.x)), y_bot = pack2(fminf(c.z, k0.z), fminf(c.z, k1.z));
    const f32x2 x_top = pack2(fmaxf(c.y, k0.y), fmaxf(c.y, k1.y)), x_bot = pack2(fminf(c.w, k0.w), fminf(c.w, k1.w));
    float h0, h1, i0, i1, b0, b1;
    unpack2(sub2(y_bot, y_top), h0, h1);
    unpack2(mul2(pack2(fmaxf(h0, 0.0f), fmaxf(h1, 0.0f)), sub2(x_bot, x_top)), i0, i1);
    unpack2(mul2(lo2, add2(ca2, pack2(a0, a1))), b0, b1);
    return (i0 >= b0 ? 1u : 0u) | (i1 >= b1 ? 2u : 0u);
}
// the exact decision behind the pre-test
__device__ __forceinline__ bool nms_suppresses_filtered(float4 ci, float ai, float4 cj, float aj, const IouThreshold& t) {
    return nms_maybe(ci, ai, cj, aj, t.lo_s) && nms_suppresses_fast(ci, ai, cj, aj, t);
}
// the pair test for boxes staged by canonical_box
__device__ __forceinline__ bool pair_suppresses(const IouThreshold& thr, float4 ci, float ai, float4 cj, float aj) {
    return thr.fast ? nms_suppresses_filtered(ci, ai, cj, aj, thr) : nms_suppresses(ci, ai, cj, aj, thr);
}

// canonical box (ymin, xmin, ymax, xmax) and area of a raw box, as the pair tests take them
__device__ __forceinline__ void canonical_box(float4 raw, const IouThreshold& thr, float4& c, float& ca) {
    c = make_float4(fminf(raw.x, raw.z), fminf(raw.y, raw.w), fmaxf(raw.x, raw.z), fmaxf(raw.y, raw.w));
    ca = __fmul_rn(__fsub_rn(c.z, c.x), __fsub_rn(c.w, c.y));
    if (thr.fast && !(ca > 0.0f)) { c = TFRPN_FAR_BOX; ca = 0.0f; }   // see nms_suppresses_fast
}

// candidate (cb, ca) against the kept boxes j = first, first + stride, ... < nkept: G (2 or 4) independent tests per
// iteration (the tests are latency chains; the early exit is checked once per group)
template <int G>
__device__ __forceinline__ bool kept_list_suppresses(float4 cb, float ca, const float4* kbox, const float* karea, int first,
                                                     int stride, int nkept, const IouThreshold& thr) {
    static_assert(G == 2 || G == 4, "kept_list_suppresses: groups of 2 or 4");
    bool dead = false;
    int j = first;
    if (thr.fast) {
        const f32x2 ca2 = pack2(ca, ca), lo2 = pack2(thr.lo_s, thr.lo_s);
        for (; j + (G - 1) * stride < nkept && !dead; j += G * stride) {
            unsigned m = nms_maybe2(cb, ca2, kbox[j], karea[j], kbox[j + stride], karea[j + stride], lo2);
            if (G == 4)
                m |= nms_maybe2(cb, ca2, kbox[j + 2 * stride], karea[j + 2 * stride], kbox[j + 3 * stride], karea[j + 3 * stride],
                                lo2) << 2;
            if (m != 0u) {   // rare: the exact test for the pairs that passed
#pragma unroll
                for (int u = 0; u < G; ++u)
                    if (!dead && ((m >> u) & 1u)) dead = nms_suppresses_fast(cb, ca, kbox[j + u * stride], karea[j + u * stride], thr);
            }
        }
        if (G == 2) { if (!dead && j < nkept) dead = nms_suppresses_filtered(cb, ca, kbox[j], karea[j], thr); }
        else for (; j < nkept && !dead; j += stride) dead = nms_suppresses_filtered(cb, ca, kbox[j], karea[j], thr);
    } else {
        for (; j < nkept && !dead; j += stride) dead = nms_suppresses(cb, ca, kbox[j], karea[j], thr);
    }
    return dead;
}

// Resolves a round of NMS_CHUNK candidates in warp 0, in parallel sweeps (same result as the sequential greedy loop):
// an undecided candidate is REMOVED if a kept predecessor suppresses it, KEPT if no undecided predecessor does, else
// stays undecided.  Lane l owns candidates l, 32+l, 64+l, 96+l, so ballot word q is exactly bits [32q, 32q+32).
// m4[c]: the predecessor words of candidate c inside the round; U: the candidates that enter the sweeps (those the kept
// list suppresses are left out).  Kept candidates take consecutive output slots from nkept in score order, capped at
// max_out: slot[c] = its slot or -1, kept[0..3] (if not null) = the kept words after the cap.  Returns the number of
// candidates kept.
__device__ __forceinline__ int resolve_round(const uint4* m4, unsigned (&U)[4], int nkept, int max_out, int* slot,
                                             unsigned* kept) {
    const int lane = lane_id();
    uint4 pr[4];
    unsigned Kp[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int q = 0; q < 4; ++q) pr[q] = m4[q * 32 + lane];
    while ((U[0] | U[1] | U[2] | U[3]) != 0u) {
        unsigned nU[4], nK[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const bool und = (U[q] >> lane) & 1u;
            const unsigned hitK = (pr[q].x & Kp[0]) | (pr[q].y & Kp[1]) | (pr[q].z & Kp[2]) | (pr[q].w & Kp[3]);
            const unsigned hitU = (pr[q].x & U[0]) | (pr[q].y & U[1]) | (pr[q].z & U[2]) | (pr[q].w & U[3]);
            nK[q] = __ballot_sync(0xffffffffu, und && hitK == 0u && hitU == 0u);
            nU[q] = __ballot_sync(0xffffffffu, und && hitK == 0u && hitU != 0u);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) { Kp[q] |= nK[q]; U[q] = nU[q]; }
    }
    const int allowed = max_out - nkept;
    int before = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int rank = before + __popc(Kp[q] & ((1u << lane) - 1u));
        const bool k = ((Kp[q] >> lane) & 1u) && rank < allowed;
        slot[q * 32 + lane] = k ? nkept + rank : -1;
        if (kept) kept[q] = __ballot_sync(0xffffffffu, k);
        before += __popc(Kp[q]);
    }
    return min(before, allowed);
}

// warp-aggregated append: the lanes with `pred` store `v` at consecutive positions of dst, reserved with one atomicAdd
// on *cursor (all lanes call)
__device__ __forceinline__ void warp_append(bool pred, unsigned long long v, unsigned int* cursor, unsigned long long* dst) {
    const int lane = lane_id();
    const unsigned bal = __ballot_sync(0xffffffffu, pred);
    if (bal != 0u) {
        unsigned int pos0 = 0;
        if (lane == __ffs(bal) - 1) pos0 = atomicAdd(cursor, (unsigned)__popc(bal));
        pos0 = __shfl_sync(0xffffffffu, pos0, __ffs(bal) - 1);
        if (pred) dst[pos0 + __popc(bal & ((1u << lane) - 1u))] = v;
    }
}

// decoded box of an entry (predictor.py:55-56): decode(anchor, delta * variances), clipped to [0, 1] if asked
__device__ __forceinline__ float4 decoded_box(const PropParams& p, float4 anchor, float4 delta) {
    const float4 raw = decode_ref(anchor, mul4(delta, p.var));
    return p.clip_decoded ? clip01(raw) : raw;
}
// raw (decoded, optionally clipped) box of the entry `idx` at rank `rank` of image b; ranks below compact_rows read
// their regression row from reg_compact
__device__ __forceinline__ float4 ranked_raw_box(const PropParams& p, int b, int rank, uint32_t idx) {
    if (p.mode == MODE_PROPOSALS) {
        const float4 row = (p.reg_compact && rank < p.compact_rows)
                               ? ldg_f4(p.reg_compact + (long long)b * p.compact_stride + rank)
                               : ldg_f4(p.reg + (long long)b * p.N + idx);
        const float4* anc = p.anchors + (p.anchors_batched ? (long long)b * p.N : 0LL);
        return decoded_box(p, anchor_of(p, anc, idx), row);
    }
    return ldg_f4(p.boxes + (long long)b * p.box_stride + idx);
}

// MODE_TOPK output row o of image b: score and index of entry i, and its gathered or decoded box if asked
__device__ __forceinline__ void write_topk_row(const PropParams& p, int b, long long o, uint32_t i, const float* scores,
                                               const float4* anc, const int* remap) {
    p.values[o] = scores[i];
    p.indices[o] = remap ? remap[i] : (int)i;
    if (p.gathered) {
        if (p.reg) p.gathered[o] = decoded_box(p, anchor_of(p, anc, i), ldg_f4(p.reg + (long long)b * p.N + i));
        else p.gathered[o] = ldg_f4(p.boxes + (long long)b * p.box_stride + i);
    }
}
// output slot s of image b for the kept entry idx with raw box `raw`
__device__ __forceinline__ void write_kept_row(const PropParams& p, int b, int s, float4 raw, const float* scores, uint32_t idx,
                                               const int* remap) {
    const long long o = (long long)b * p.rows + s;
    p.out_boxes[o] = p.clip_out ? clip01(raw) : raw;
    p.out_scores[o] = scores[idx];
    if (p.keep_idx) p.keep_idx[o] = remap ? remap[idx] : (int)idx;
}
// output rows first, first + stride, ... of image b: zero padding past nkept (TF pads boxes/scores/classes with 0;
// keep_idx pads with -1), and the class column
__device__ __forceinline__ void pad_outputs(const PropParams& p, int b, int nkept, int first, int stride) {
    for (int rnk = first; rnk < p.rows; rnk += stride) {
        const long long o = (long long)b * p.rows + rnk;
        if (rnk >= nkept) {
            p.out_boxes[o] = make_float4(0.f, 0.f, 0.f, 0.f);
            p.out_scores[o] = 0.0f;
            if (p.keep_idx) p.keep_idx[o] = -1;
        }
        if (p.out_classes) p.out_classes[o] = 0.0f;
    }
}

// descending bitonic sort of BATCH composites, one per thread of a BATCH-thread CTA; thread t ends with rank t.
// Strides < 32 use shuffles; strides >= 32 go through a double-buffered shared array (1 barrier each).
__device__ __forceinline__ unsigned long long bitonic_sort_desc(unsigned long long v, unsigned long long* buf) {
    const int t = threadIdx.x;
    int flip = 0;
    for (int k = 2; k <= BATCH; k <<= 1) {
        const bool desc = (t & k) == 0;
        for (int j = k >> 1; j > 0; j >>= 1) {
            unsigned long long pv;
            if (j >= 32) {
                unsigned long long* bb = buf + flip * BATCH;
                bb[t] = v;
                __syncthreads();
                pv = bb[t ^ j];
                flip ^= 1;
            } else {
                pv = __shfl_xor_sync(0xffffffffu, v, j);
            }
            const bool lower = (t & j) == 0;
            const bool keep_max = (lower == desc);
            v = keep_max ? max(v, pv) : min(v, pv);
        }
    }
    return v;
}

// the same network over BATCH composites in shared memory, sorted in place by a CTA of T < BATCH threads: one
// compare-exchange per pair and step, a barrier after each step
template <int T>
__device__ __forceinline__ void bitonic_sort_desc_shared(unsigned long long* buf) {
    for (int k = 2; k <= BATCH; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int q = threadIdx.x; q < BATCH / 2; q += T) {
                const int i = ((q & ~(j - 1)) << 1) | (q & (j - 1)), l = i + j;
                const unsigned long long a = buf[i], c = buf[l];
                if (((i & k) == 0) == (a < c)) { buf[i] = c; buf[l] = a; }   // descending where bit k of i is 0
            }
            __syncthreads();
        }
    }
}

// One CTA of T threads per image (T = 1024 or 512).  The algorithm and every order are the same for both builds; only
// the mapping of work to threads differs: sweeps stride T, thread t owns SEL_NB / T histogram bins of a scan, holds
// list entries t + q T and ranks t + q T of the batch, and the kept-list test splits a candidate into T / 128 parts.
// Two 512-thread CTAs share an SM (64 registers per thread) and fill each other's barrier gaps.
template <int T>
__global__ void __launch_bounds__(T, BATCH / T) proposal_kernel(PropParams p) {
    constexpr int PER_BIN = SEL_NB / T;       // histogram bins per thread in a scan
    constexpr int PER_LIST = SEL_LIST / T;    // candidate-list entries per thread
    constexpr int PER_RANK = BATCH / T;       // ranks of a batch per thread
    constexpr int NMS_PARTS = T / NMS_CHUNK;  // kept-list parts per candidate
    static_assert((T == 512 || T == 1024) && T >= NMS_CHUNK * 4, "proposal_kernel: 512 or 1024 threads");
    extern __shared__ float4 smem4[];
    __shared__ PropShared sh;
    PH_DECL
    const int tid = threadIdx.x, lane = lane_id(), warp = warp_id();
    const int b = blockIdx.x;
    if (p.flag_mode == 1 && p.flags[b] != 0) return;
    if (p.flag_mode == 2 && p.flags[b] == 0) return;
    const long long SN = p.N;                          // row stride of scores / reg / remap
    const int N = p.counts ? p.counts[b] : p.N;        // entries of this image
    const float* scores = p.scores + (long long)b * SN;
    const float4* anc = p.anchors + (p.anchors_batched ? (long long)b * SN : 0LL);
    const int* remap = p.remap ? p.remap + (long long)b * SN : nullptr;

    unsigned long long* sortbuf = reinterpret_cast<unsigned long long*>(smem4);   // [2 * BATCH] list, then the batch
    uint32_t* sidx = reinterpret_cast<uint32_t*>(sortbuf + 2 * BATCH);            // [BATCH] sorted indices
    float4* kbox = reinterpret_cast<float4*>(sidx + BATCH);                       // [mo_pad]
    float4* cbox = kbox + p.mo_pad;                                               // [NMS_CHUNK]
    float* karea = reinterpret_cast<float*>(cbox + NMS_CHUNK);                    // [mo_pad]
    float* carea = karea + p.mo_pad;                                              // [NMS_CHUNK]
    unsigned int* alive = reinterpret_cast<unsigned int*>(carea + NMS_CHUNK);     // [NMS_CHUNK]
    int* slot = reinterpret_cast<int*>(alive + NMS_CHUNK);                        // [NMS_CHUNK]
    unsigned int* mask32 = reinterpret_cast<unsigned int*>(slot + NMS_CHUNK);       // [NMS_CHUNK][4]
    unsigned int* hist = mask32 + NMS_CHUNK * 4;                                  // [SEL_NB]
    uint32_t* skeys = hist + SEL_NB;                                              // [N] when staged

    // Entries at or below the score threshold (key 0) can never be consumed (K <= M below), so with a threshold
    // they take no part in any batch: composites with key 0 are <= cmin.
    const unsigned long long cmin = p.use_sthr ? 0xFFFFFFFFull : 0ull;

    // ---- phase 0: stage keys; count entries above the score threshold, the largest key and the first select
    //      histogram (key bits [31:21]) in the same sweep, four loads in flight per thread --------------------
#pragma unroll
    for (int q = 0; q < PER_BIN; ++q) hist[q * T + tid] = 0u;
    if (tid == 0) { sh.count = 0u; sh.kmax = 0u; }
    __syncthreads();
    unsigned int my_valid = 0, my_max = 0;
    for (int base = 0; base < N; base += 4 * T) {
        float sc[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + u * T + tid;
            sc[u] = i < N ? __ldg(scores + i) : 0.0f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + u * T + tid;
            if (i < N) {
                const uint32_t key = score_key(sc[u], p.use_sthr, p.score_threshold);
                if (p.staged) skeys[i] = key;
                my_max = max(my_max, key);
                if (key != 0u || !p.use_sthr) {
                    ++my_valid;
                    atomicAdd(&hist[key >> (32 - SEL_BITS)], 1u);
                }
            }
        }
    }
    my_valid = __reduce_add_sync(0xffffffffu, my_valid);
    my_max = __reduce_max_sync(0xffffffffu, my_max);
    if (lane == 0) { atomicAdd(&sh.count, my_valid); atomicMax(&sh.kmax, my_max); }
    __syncthreads();
    const int M = (int)sh.count;   // N without a score threshold
    const uint32_t kmax = sh.kmax;
    const int K = min(p.k, M);  // ranks that may be consumed
    PH(1);
    int nkept = 0;
    const IouThreshold thr = p.iou_thr;

    auto key_at = [&](int i) -> uint32_t {
        return p.staged ? skeys[i] : score_key(scores[i], p.use_sthr, p.score_threshold);
    };

    // Batches by threshold: a batch is every eligible entry with composite >= tau, where tau is a histogram bin
    // edge chosen so that the batch holds at most BATCH entries, and at least SEL_FLOOR unless it holds every
    // eligible entry.  Entries of earlier batches (composite >= lo_tau) are no longer eligible.  The batch is
    // ordered in full, so its first K - lo ranks end exactly at rank K.
    unsigned long long lo_tau = 0ull;
    bool have_lo = false;
    for (int lo = 0; lo < K;) {
        auto eligible = [&](unsigned long long c) -> bool { return c > cmin && (!have_lo || c < lo_tau); };
        // ---- 1. select tau: 11-bit digits from the top of the composite, refined inside the bin that holds
        //      rank BATCH.  Once the eligible entries >= the bin's lower edge fit SEL_LIST, the next full sweep
        //      also copies them into sortbuf and every later pass (and the batch) reads only that list. ----------
        unsigned long long tau = 0ull, prefix = 0ull;   // tau 0: every eligible entry
        int top = 63;                                   // digit bits [top - 10, top] below the common prefix
        unsigned int r = BATCH;                         // rank of the boundary among entries matching `prefix`
        int nl = -1;                                    // entries in the list (-1: none, sweep all N)
        bool listing = false;
        for (int pass = 0;; ++pass) {
            const int shift = max(top - (SEL_BITS - 1), 0);
            const unsigned int dmask = (2u << (top - shift)) - 1u;
            const unsigned long long himask = top >= 63 ? 0ull : (~0ull << (top + 1));
            if (nl >= 0) {
                for (int q = tid; q < nl; q += T) {
                    const unsigned long long c = sortbuf[q];
                    if (((c ^ prefix) & himask) == 0ull) atomicAdd(&hist[(unsigned)(c >> shift) & dmask], 1u);
                }
            } else if (pass > 0 || have_lo) {           // (the first batch's first histogram comes from phase 0)
                for (int base = 0; base < N; base += T) {
                    const int i = base + tid;
                    unsigned long long c = 0ull;
                    bool in = false;                    // eligible and >= prefix: above the bin, or in it
                    if (i < N) {
                        c = make_comp(key_at(i), i);
                        in = eligible(c) && c >= prefix;
                    }
                    if (in && ((c ^ prefix) & himask) == 0ull) atomicAdd(&hist[(unsigned)(c >> shift) & dmask], 1u);
                    if (listing) warp_append(in, c, &sh.lcount, sortbuf);
                }
            }
            __syncthreads();                            // histogram (and list) complete
            if (listing) nl = (int)sh.lcount;
            unsigned total;
            {
                unsigned c[PER_BIN], ex, cmax;
                hist_scan_desc<T>(hist, c, ex, total, cmax, &sh);
                const unsigned zero[PER_BIN] = {};
                own_bins_store<T>(hist, zero);          // own bins, for the next histogram (after the barrier below)
#pragma unroll
                for (int q = 0; q < PER_BIN; ++q) {     // the bin that holds rank r
                    if (ex < r && r <= ex + c[q]) {
                        sh.digit = (unsigned)(SEL_NB - 1 - PER_BIN * tid - q);
                        sh.excl = ex;
                        sh.bin_count = c[q];
                    }
                    ex += c[q];
                }
            }
            if (tid == 0) sh.lcount = 0u;
            __syncthreads();
            if (total < r) break;                       // (first pass only) fewer than BATCH eligible entries: all of them
            const unsigned int d = sh.digit, ex = sh.excl, bc = sh.bin_count;
            const unsigned long long edge = prefix | ((unsigned long long)d << shift);   // lower edge of the boundary bin
            const unsigned int above = BATCH - r + ex;  // eligible entries above the boundary bin
            if (bc == r - ex) { tau = edge; break; }    // the whole bin makes exactly BATCH
            if (above >= (unsigned)SEL_FLOOR) { tau = edge + (1ull << shift); break; }
            listing = nl < 0 && above + bc <= (unsigned)SEL_LIST;
            prefix = edge;
            r -= ex;
            top = shift - 1;                            // (shift == 0 cannot get here: its bins are single composites)
        }
        PH(2);
        // ---- 2. the batch: up to PER_LIST list entries per thread (without a list, one compaction sweep makes it) ----
        if (nl < 0) {
            for (int base = 0; base < N; base += T) {
                const int i = base + tid;
                bool take = false;
                unsigned long long c = 0ull;
                if (i < N) {
                    c = make_comp(key_at(i), i);
                    take = eligible(c) && c >= tau;
                }
                warp_append(take, c, &sh.lcount, sortbuf);
            }
            __syncthreads();
            nl = (int)sh.lcount;
        }
        // list entries are eligible and >= tau's bin edge or better; composites of entries are > 0
        unsigned long long le[PER_LIST];
#pragma unroll
        for (int q = 0; q < PER_LIST; ++q) le[q] = q * T + tid < nl ? sortbuf[q * T + tid] : 0ull;
        PH(3);
        // ---- 3. order the batch: counting sort on the 11 key bits below the common prefix of its key range
        //      [key(tau), upper bound]; a bin's entries find their place by comparing composites within it ---------
        const uint32_t khi = have_lo ? (uint32_t)(lo_tau >> 32) : kmax, kdiff = khi ^ (uint32_t)(tau >> 32);
        const int sshift = kdiff ? max(31 - __clz(kdiff) - (SEL_BITS - 1), 0) : 0;
        unsigned ds[PER_LIST];                          // (bin << 16) | place in the bin; ~0u: not in the batch
#pragma unroll
        for (int q = 0; q < PER_LIST; ++q) {
            ds[q] = ~0u;
            if (le[q] != 0ull && le[q] >= tau) {
                const unsigned d = ((uint32_t)(le[q] >> 32) >> sshift) & (SEL_NB - 1);
                ds[q] = (d << 16) | atomicAdd(&hist[d], 1u);
            }
        }
        __syncthreads();                                // bin counts complete; the list has been read
        unsigned total, cmax;
        {
            unsigned c[PER_BIN], ex;
            hist_scan_desc<T>(hist, c, ex, total, cmax, &sh);
#pragma unroll
            for (int q = 0; q < PER_BIN; ++q) { const unsigned n = c[q]; c[q] = (ex << 16) | n; ex += n; }
            own_bins_store<T>(hist, c);                 // (first position, count) of the own bins
        }
        __syncthreads();
        const int nb_all = (int)total;                  // entries of this batch, <= BATCH
        unsigned long long* bybin = sortbuf;            // [BATCH] the batch grouped by bin
        unsigned long long* ranked = sortbuf + BATCH;   // [BATCH] the batch in rank order
#pragma unroll
        for (int q = 0; q < PER_LIST; ++q)
            if (ds[q] != ~0u) bybin[(hist[ds[q] >> 16] >> 16) + (ds[q] & 0xFFFFu)] = le[q];
        __syncthreads();
        unsigned long long mine[PER_RANK];              // thread t holds ranks t + q T of the batch
        if (cmax <= (unsigned)SEG_MAX) {
            auto place = [&](unsigned long long v, unsigned d) {
                const unsigned hv = hist[d], first = hv >> 16, n = hv & 0xFFFFu;
                unsigned gt = 0;
                for (unsigned q = 0; q < n; ++q) gt += bybin[first + q] > v ? 1u : 0u;
                ranked[first + gt] = v;
            };
#pragma unroll
            for (int q = 0; q < PER_LIST; ++q)
                if (ds[q] != ~0u) place(le[q], ds[q] >> 16);
            __syncthreads();
#pragma unroll
            for (int q = 0; q < PER_RANK; ++q) mine[q] = q * T + tid < nb_all ? ranked[q * T + tid] : 0ull;
        } else if constexpr (T == BATCH) {              // long bins (tie groups, clustered scores): bitonic network
            mine[0] = tid < nb_all ? bybin[tid] : 0ull; // padding sorts last
            __syncthreads();
            mine[0] = bitonic_sort_desc(mine[0], sortbuf);
        } else {
#pragma unroll
            for (int q = 0; q < PER_RANK; ++q) ranked[q * T + tid] = q * T + tid < nb_all ? bybin[q * T + tid] : 0ull;
            __syncthreads();
            bitonic_sort_desc_shared<T>(ranked);
#pragma unroll
            for (int q = 0; q < PER_RANK; ++q) mine[q] = ranked[q * T + tid];
        }
#pragma unroll
        for (int q = 0; q < PER_BIN; ++q) hist[q * T + tid] = 0u;   // for the next batch: its first histogram follows a barrier
        const int blo = lo;                             // thread t holds ranks blo + t + q T
        const int nb = min(nb_all, K - lo);             // entries of this batch that may be consumed
        lo += nb_all;
        lo_tau = tau;
        have_lo = true;
        PH(4);
        uint32_t my_i[PER_RANK];
#pragma unroll
        for (int q = 0; q < PER_RANK; ++q) my_i[q] = 0xFFFFFFFFu - (uint32_t)(mine[q] & 0xFFFFFFFFull);

        // ---- 4a. top-k outputs (predictor.py:58-60) -------------------------------------------
        if (p.mode == MODE_TOPK) {
#pragma unroll
            for (int q = 0; q < PER_RANK; ++q) {
                const int rk = q * T + tid;
                if (rk < nb) write_topk_row(p, b, (long long)b * p.k + blo + rk, my_i[q], scores, anc, remap);
            }
            __syncthreads();   // sortbuf is rewritten by the next batch
            continue;
        }

        // ---- 4b. greedy NMS rounds over this batch ---------------------------------------------
#pragma unroll
        for (int q = 0; q < PER_RANK; ++q) sidx[q * T + tid] = my_i[q];
        __syncthreads();
        auto fetch = [&](int pos, float4& a, float4& d, uint32_t& idx) {
            if (p.rows_fetched && tid == 0 && pos < nb) atomicAdd(p.rows_fetched, (unsigned long long)min(NMS_CHUNK, nb - pos));
            if (tid < NMS_CHUNK && pos + tid < nb) {
                idx = sidx[pos + tid];
                if (p.mode == MODE_PROPOSALS) {
                    d = ldg_f4(p.reg + (long long)b * SN + idx);
                    a = anchor_of(p, anc, idx);
                } else {
                    a = ldg_f4(p.boxes + (long long)b * p.box_stride + idx);
                }
            }
        };
        float4 na = make_float4(0.f, 0.f, 0.f, 0.f), nd = na;
        uint32_t nidx = 0u;
        fetch(0, na, nd, nidx);
        for (int pos = 0; pos < nb && nkept < p.max_out; pos += NMS_CHUNK) {
            const int C = min(NMS_CHUNK, nb - pos);
            float4 raw = na;
            const uint32_t my_idx = nidx;
            if (tid < C) {
                if (p.mode == MODE_PROPOSALS) raw = decoded_box(p, na, nd);
                float4 c;
                float ca;
                canonical_box(raw, thr, c, ca);
                cbox[tid] = c;
                carea[tid] = ca;
                alive[tid] = 1u;
            }
            if (tid < NMS_CHUNK * 4) mask32[tid] = 0u;
            __syncthreads();
            PH(6);
            fetch(pos + NMS_CHUNK, na, nd, nidx);   // in flight during the tests below
            {   // candidates vs kept list: thread = (candidate c, part), kept j strided by NMS_PARTS
                const int c = tid & (NMS_CHUNK - 1), part = tid >> 7;
                if (c < C && kept_list_suppresses<2>(cbox[c], carea[c], kbox, karea, part, NMS_PARTS, nkept, thr)) alive[c] = 0u;
            }
            __syncthreads();
            PH(7);
            if (warp == 0) {   // compact the candidates that survived the kept list (order preserved) into slot[]
                int before = 0;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int c = q * 32 + lane;
                    const bool a = c < C && alive[c] != 0u;
                    const unsigned bal = __ballot_sync(0xffffffffu, a);
                    if (a) slot[before + __popc(bal & ((1u << lane) - 1u))] = c;
                    before += __popc(bal);
                }
                if (lane == 0) sh.nalive = before;
            }
            __syncthreads();
            PH(8);
            {   // intra-round predecessor masks over the A survivors: bit j of row i set iff j < i and j suppresses i.
                // The triangle is folded so that every 16-thread team gets the same number of pairs:
                // team r takes row iA = r + 1 (iA pairs) and row iB = A - 1 - r (iB pairs) of the compact order.
                // With T / 16 < 64 teams, team r also takes the folded pair r + T / 16.
                const int A = sh.nalive;
                const int sub = tid & 15;
                for (int r = tid >> 4; r < NMS_CHUNK / 2; r += T / 16) {
                    const int iA = r + 1, iB = A - 1 - r;
                    const int len = (iA < iB) ? iA + iB : (iA == iB ? iA : 0);
                    for (int e = sub; e < len; e += 16) {
                        const int i = slot[e < iA ? iA : iB];
                        const int j = slot[e < iA ? e : e - iA];
                        if (pair_suppresses(thr, cbox[j], carea[j], cbox[i], carea[i])) atomicOr(&mask32[i * 4 + (j >> 5)], 1u << (j & 31));
                    }
                }
            }
            __syncthreads();
            PH(9);
            if (warp == 0) {   // the round's greedy order, over the candidates that survived the kept list
                unsigned U[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int c = q * 32 + lane;
                    U[q] = __ballot_sync(0xffffffffu, c < C && alive[c] != 0u);
                }
                const int nk = resolve_round(reinterpret_cast<const uint4*>(mask32), U, nkept, p.max_out, slot, nullptr);
                if (lane == 0) sh.nk = nk;
            }
            __syncthreads();
            PH(10);
            if (tid < C && slot[tid] >= 0) {
                const int s = slot[tid];
                kbox[s] = cbox[tid];
                karea[s] = carea[tid];
                write_kept_row(p, b, s, raw, scores, my_idx, remap);
            }
            nkept += sh.nk;
            __syncthreads();
            PH(11);
        }
        if (nkept >= p.max_out) break;
    }
    if (p.mode == MODE_TOPK) return;
    if (p.flags_out && nkept < p.max_out && N < p.full_n) {   // the unfiltered kernel redoes this image
        if (tid == 0) p.flags_out[b] = 1;
        return;
    }
    pad_outputs(p, b, nkept, tid, T);
    if (tid == 0) p.valid[b] = nkept;
    PH(12);
    PH_FLUSH;
}


// ------------------------------------------------------------------------------------------------
// proposal_cluster_kernel<CL>: the same algorithm with an image spread over a thread-block CLUSTER of
// CL CTAs x (1024 / CL) threads (distributed shared memory).  The one-CTA kernel is bound by the latency
// of its serial phases with 32 warps contending for one SM's schedulers; here every phase keeps its
// per-thread work and runs on CL SMs, and the phases are cut so that CTAs meet as rarely as possible
// (a cluster barrier costs ~400 cycles): two barriers per batch of ranks + ONE per NMS round.
//
//   scores      CTA r owns the 32-entry chunks c with c % CL == r (coalesced loads, balanced slices)
//   select      LOCAL: every CTA radix-selects (11 bits per pass, shared-memory histogram) a threshold
//               tau_r such that its slice holds between T/2 and T = 1024 / CL composites >= tau_r
//               (everything when the slice has fewer), compacts them and bitonic-sorts them, one per thread
//   merge       the sorted lists and the tau_r meet through DSMEM (barrier 1).  tau = max tau_r: every
//               entry >= tau of the image is in some list, so the entries >= tau ARE the next ranks, in
//               order; an entry's rank = its local rank + its lower bound in each peer's list.  Entries
//               below tau wait for the next batch (its eligibility rule is "composite < tau").
//   boxes       every entry's owner decodes its box and writes (canonical box, area) to slot `rank` of a
//               replicated array in every CTA (barrier 2)
//   NMS rounds  128 candidates per round.  The tests against the kept list AND the predecessor triangle of
//               the round (over all its candidates: independent of the kept-list outcome) are split over
//               all CL x T threads in one phase; the suppressed bits and the triangle rows meet through
//               DSMEM (one barrier per round, parity-double-buffered), and every CTA resolves the round and
//               appends to its own copy of the kept list redundantly.
// Results are bit-identical to proposal_kernel: same composites, same order, same pair test.
// ------------------------------------------------------------------------------------------------
constexpr int CL_NBITS = 11;
constexpr int CL_NB = 1 << CL_NBITS;
constexpr int CL_MAX = 8;

struct ClShared {
    unsigned long long tau;            // this CTA's threshold of the batch (read by the peers)
    unsigned int wtot[32], wtot2[32];
    unsigned int digit, excl, bin_count, total;
    unsigned int count;                // compaction cursor, then the batch's entry count
    unsigned int valid_all[CL_MAX];    // [0]: this CTA's count of entries above the score threshold (peers read it after the first barrier)
    unsigned int dead_all[2][CL_MAX][4];  // [round parity][CTA]: "suppressed by the kept list" bits
    unsigned int dead_w[4];            // the bits found inside this CTA
    int nk;
};

template <int CL>
__device__ __forceinline__ void cl_sync() {
    if (CL == 1) __syncthreads();
    else cg::this_cluster().sync();
}
template <int CL, class P>
__device__ __forceinline__ P* cl_peer(P* local, unsigned q) {
    if (CL == 1) return local;
    return cg::this_cluster().map_shared_rank(local, q);
}

// descending bitonic sort of S composites held by the threads t < S of the CTA, one each (all T threads call);
// thread t < S ends with local rank t.  Strides < 32 use shuffles, the others a double-buffered shared array.
template <int S>
__device__ __forceinline__ unsigned long long bitonic_sort_desc_s(unsigned long long v, unsigned long long* buf) {
    const int t = threadIdx.x;
    const bool active = t < S;
    int flip = 0;
    for (int k = 2; k <= S; k <<= 1) {
        const bool desc = (t & k) == 0;
        for (int j = k >> 1; j > 0; j >>= 1) {
            unsigned long long pv;
            if (j >= 32) {
                unsigned long long* bb = buf + flip * S;
                if (active) bb[t] = v;
                __syncthreads();
                pv = active ? bb[t ^ j] : 0ull;
                flip ^= 1;
            } else {
                pv = __shfl_xor_sync(0xffffffffu, v, j);
            }
            const bool lower = (t & j) == 0;
            const bool keep_max = (lower == desc);
            v = keep_max ? max(v, pv) : min(v, pv);
        }
    }
    return v;
}

// CL CTAs x T threads per image; S = 1024 / CL sort slots per CTA (T >= S, T >= 128)
template <int CL, int T>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(T, (T <= 512 && CL > 1) ? 2 : 1) proposal_cluster_kernel(PropParams p) {
    constexpr int S = BATCH / CL;           // sort slots per CTA
    constexpr int WARPS = T / 32;
    constexpr int PER = CL_NB / T;          // histogram bins per thread in the scan
    constexpr int NT = CL * T;              // threads per image
    constexpr int PARTS = NT / NMS_CHUNK;   // kept-list parts over the whole cluster
    constexpr int TS = NT / 64;             // threads per team of the folded triangle (64 teams)
    static_assert(T >= S && T >= NMS_CHUNK && PER >= 1 && TS >= 1, "bad cluster shape");
    extern __shared__ float4 smem4[];
    __shared__ ClShared sh;
    PH_DECL
    const int tid = threadIdx.x, lane = lane_id(), warp = warp_id();
    unsigned crank = 0;
    if (CL > 1) crank = cg::this_cluster().block_rank();
    const int b = blockIdx.x / CL;
    if (p.flag_mode == 1 && p.flags[b] != 0) return;     // uniform over the cluster
    if (p.flag_mode == 2 && p.flags[b] == 0) return;
    const long long SN = p.N;
    const int N = p.counts ? p.counts[b] : p.N;
    const float* scores = p.scores + (long long)b * SN;
    const float4* anc = p.anchors + (p.anchors_batched ? (long long)b * SN : 0LL);
    const int* remap = p.remap ? p.remap + (long long)b * SN : nullptr;

    // ---- shared memory carve -----------------------------------------------------------------------
    unsigned int* hist = reinterpret_cast<unsigned int*>(smem4);                                 // [CL_NB]
    unsigned long long* lists = reinterpret_cast<unsigned long long*>(hist + CL_NB);             // [CL][S]: mine, then copies of the peers'
    unsigned long long* sortbuf = lists + BATCH;                                                 // [2][S]
    float4* cbox_all = reinterpret_cast<float4*>(sortbuf + 2 * S);                               // [BATCH] canonical boxes by rank
    float4* kbox = cbox_all + BATCH;                                                             // [mo_pad]
    float* carea_all = reinterpret_cast<float*>(kbox + p.mo_pad);                                // [BATCH]
    float* karea = carea_all + BATCH;                                                            // [mo_pad]
    int* slot = reinterpret_cast<int*>(karea + p.mo_pad);                                        // [NMS_CHUNK]
    unsigned int* mask32 = reinterpret_cast<unsigned int*>(slot + NMS_CHUNK);                    // [2][NMS_CHUNK][4]
    uint32_t* skeys = mask32 + 2 * NMS_CHUNK * 4;                                                // [Lmax] when staged

    // local slice: local index li <-> entry i
    const int nchunks = (N + 31) >> 5;
    const int Lmax = ((nchunks + CL - 1) / CL) << 5;
    auto entry_of = [&](int li) -> int { return (((li >> 5) * CL + (int)crank) << 5) + (li & 31); };
    auto key_at = [&](int li, int i) -> uint32_t {
        return p.staged ? skeys[li] : score_key(scores[i], p.use_sthr, p.score_threshold);
    };

    // ---- phase 0: stage keys (four loads in flight per thread), count entries above the score threshold ----
    unsigned int my_valid = 0;
    for (int base = 0; base < Lmax && !p.presorted; base += 4 * T) {
        float sc[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int li = base + u * T + tid;
            const int i = entry_of(li);
            sc[u] = (li < Lmax && i < N) ? __ldg(scores + i) : 0.0f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int li = base + u * T + tid;
            if (li < Lmax && entry_of(li) < N) {
                const uint32_t key = score_key(sc[u], p.use_sthr, p.score_threshold);
                if (p.staged) skeys[li] = key;
                my_valid += (key != 0u) ? 1u : 0u;
            }
        }
    }
    for (int k = tid; k < 2 * NMS_CHUNK * 4; k += T) mask32[k] = 0u;
    if (tid < 4) sh.dead_w[tid] = 0u;
    int M = N;
    if (p.use_sthr) {
        my_valid = __reduce_add_sync(0xffffffffu, my_valid);
        if (lane == 0) sh.wtot[warp] = my_valid;
        __syncthreads();
        if (tid == 0) {   // this CTA's count stays LOCAL until the barrier: a peer may not have started yet
            unsigned int tot = 0;
            for (int w = 0; w < WARPS; ++w) tot += sh.wtot[w];
            sh.valid_all[0] = tot;
        }
    }
    // (every CTA of the cluster must be running before the first remote shared-memory access)
    cl_sync<CL>();
    if (p.use_sthr) {
        M = 0;
        for (int q = 0; q < CL; ++q) M += (int)*cl_peer<CL>(&sh.valid_all[0], (unsigned)q);
    }
    int K = min(p.k, M);                    // ranks that may be consumed
    bool cut = false;                       // presorted: the launch cannot serve every rank of the batch
    if (p.presorted) {
        K = p.rank_n[b];
        if (p.reg_compact && K > p.compact_rows) { K = p.compact_rows; cut = true; }   // only the gathered rows are served
    }
    int nkept = 0;
    const IouThreshold thr = p.iou_thr;
    PH(1);

    unsigned long long lo_tau = 0ull;       // entries already consumed: composite >= lo_tau
    bool have_lo = false;
    int par = 0;                            // parity of the NMS round (cluster-uniform)
    if (p.mode == MODE_RANK && K <= 0 && tid == 0 && crank == 0) { p.rank_n[b] = 0; p.rank_more[b] = 0; }   // no rank at all

    for (int lo = 0; lo < K;) {
        auto eligible = [&](unsigned long long c) -> bool { return !have_lo || c < lo_tau; };
        unsigned long long mine = 0ull, tau = 0ull;
        int nb_all = K, nb = K, rank = (int)crank * S + tid;     // presorted: thread t of CTA r owns rank r * S + t
        if (!p.presorted) {
        // ---- 1. local select: tau_r with 7S/8 <= #{eligible local composites >= tau_r} <= S (0: all of them) ----
        unsigned long long tau_r = 0ull;
        {
            // leading bits every eligible key shares carry no information: the digit windows start below them
            uint32_t kor = 0u, kand = 0xFFFFFFFFu;
            for (int li = tid; li < Lmax; li += T) {
                const int i = entry_of(li);
                if (i < N) {
                    const uint32_t key = key_at(li, i);
                    if (eligible(make_comp(key, i))) { kor |= key; kand &= key; }
                }
            }
            kor = __reduce_or_sync(0xffffffffu, kor);
            kand = __reduce_and_sync(0xffffffffu, kand);
            if (lane == 0) { sh.wtot[warp] = kor; sh.wtot2[warp] = kand; }
            __syncthreads();
            kor = 0u; kand = 0xFFFFFFFFu;
            for (int w = 0; w < WARPS; ++w) { kor |= sh.wtot[w]; kand &= sh.wtot2[w]; }
            __syncthreads();
            const uint32_t diff = kor ^ kand;
            int top = diff ? 63 - __clz(diff) : 31;                      // highest composite bit that varies
            unsigned long long prefix = top >= 32 ? ((unsigned long long)(kand & ~((2u << (top - 32)) - 1u)) << 32)
                                                  : ((unsigned long long)kand << 32);
            if (kor == 0u && kand == 0xFFFFFFFFu) { top = 63; prefix = 0ull; }   // no eligible entry here
            unsigned int r = (unsigned int)S;        // looking for the r-th largest among the entries matching `prefix`
            for (int pass = 0; pass < 8; ++pass) {
                const int bot = max(top - (CL_NBITS - 1), 0);
                const int shift = bot, width = top - bot + 1;
                for (int k = tid; k < CL_NB; k += T) hist[k] = 0u;
                __syncthreads();
                const unsigned long long himask = top >= 63 ? 0ull : (~0ull << (top + 1));
                const unsigned int dmask = (1u << width) - 1u;
                for (int li = tid; li < Lmax; li += T) {
                    const int i = entry_of(li);
                    if (i < N) {
                        const unsigned long long c = make_comp(key_at(li, i), i);
                        if (eligible(c) && ((c ^ prefix) & himask) == 0ull) atomicAdd(&hist[(unsigned)(c >> shift) & dmask], 1u);
                    }
                }
                __syncthreads();
                // thread t owns the PER digits CL_NB-1 - (t*PER + q), q = 0..PER-1, scanned from the top
                unsigned int c[PER], s = 0;
#pragma unroll
                for (int q = 0; q < PER; ++q) { c[q] = hist[CL_NB - 1 - (tid * PER + q)]; s += c[q]; }
                const unsigned int incl_w = (unsigned int)warp_incl_scan((int)s);
                if (lane == 31) sh.wtot[warp] = incl_w;
                if (tid == 0) sh.bin_count = 0u;     // stays 0 when fewer than r entries match
                __syncthreads();
                unsigned int woff = 0, total = 0;
                for (int w = 0; w < WARPS; ++w) {
                    const unsigned int v = sh.wtot[w];
                    woff += (w < warp) ? v : 0u;
                    total += v;
                }
                const unsigned int excl = woff + incl_w - s;
                if (excl < r && r <= excl + s) {
                    unsigned int acc = excl;
#pragma unroll
                    for (int q = 0; q < PER; ++q) {
                        if (acc < r && r <= acc + c[q]) {
                            sh.digit = (unsigned)(CL_NB - 1 - (tid * PER + q));
                            sh.excl = acc;
                            sh.bin_count = c[q];
                        }
                        acc += c[q];
                    }
                }
                __syncthreads();
                const unsigned int d = sh.digit, ex = sh.excl, bc = sh.bin_count;
                __syncthreads();
                if (total < r) break;                                  // (first pass only) fewer than S eligible entries: all of them
                const unsigned long long edge = prefix | ((unsigned long long)d << shift);   // lower edge of the boundary bin
                if (bc == r - ex) { tau_r = edge; break; }             // the whole bin is taken: exactly S entries
                if ((unsigned int)S - r + ex >= (unsigned int)(S - S / 8)) {  // leave the (small) boundary bin to the next batch
                    tau_r = edge + (1ull << shift);
                    break;
                }
                prefix = edge;
                r -= ex;
                top = bot - 1;                                         // (bot == 0 cannot get here: its bins are singletons)
            }
        }
        PH(2);
        // ---- 2. local compaction (<= S entries by construction): one reservation per warp -------------------
        if (tid < S) sortbuf[tid] = 0ull;       // padding sorts last
        if (tid == 0) sh.count = 0u;
        __syncthreads();
        {
            unsigned int wtotal = 0;
            for (int base = 0; base < Lmax; base += T) {
                const int li = base + tid;
                const int i = entry_of(li);
                bool take = false;
                if (li < Lmax && i < N) {
                    const unsigned long long c = make_comp(key_at(li, i), i);
                    take = eligible(c) && c >= tau_r;
                }
                wtotal += __popc(__ballot_sync(0xffffffffu, take));
            }
            unsigned int wbase = 0;
            if (lane == 0 && wtotal != 0u) wbase = atomicAdd(&sh.count, wtotal);
            wbase = __shfl_sync(0xffffffffu, wbase, 0);
            if (wtotal != 0u) {
                for (int base = 0; base < Lmax; base += T) {
                    const int li = base + tid;
                    const int i = entry_of(li);
                    bool take = false;
                    unsigned long long c = 0ull;
                    if (li < Lmax && i < N) {
                        c = make_comp(key_at(li, i), i);
                        take = eligible(c) && c >= tau_r;
                    }
                    const unsigned bal = __ballot_sync(0xffffffffu, take);
                    if (take) sortbuf[wbase + __popc(bal & ((1u << lane) - 1u))] = c;
                    wbase += __popc(bal);
                }
            }
        }
        __syncthreads();
        PH(3);
        mine = tid < S ? sortbuf[tid] : 0ull;
        __syncthreads();
        mine = bitonic_sort_desc_s<S>(mine, sortbuf);
        if (tid < S) lists[tid] = mine;         // my sorted list, read by the peers
        if (tid == 0) { sh.tau = tau_r; sh.count = 0u; }
        PH(4);
        cl_sync<CL>();                          // barrier 1
        // ---- 3. tau, the batch's entry count and every entry's rank ------------------------------------------
        tau = tau_r;
        if (CL > 1) {
#pragma unroll
            for (int q = 1; q < CL; ++q) tau = max(tau, *cl_peer<CL>(&sh.tau, (crank + q) % CL));
        }
        unsigned int cnt = (mine != 0ull && mine >= tau) ? 1u : 0u;
        if (CL > 1 && tid < S) {
#pragma unroll
            for (int q = 1; q < CL; ++q) {
                const unsigned long long v = cl_peer<CL>(lists, (crank + q) % CL)[tid];
                lists[q * S + tid] = v;
                cnt += (v != 0ull && v >= tau) ? 1u : 0u;
            }
        }
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        if (lane == 0 && cnt != 0u) atomicAdd(&sh.count, cnt);
        __syncthreads();
        nb_all = (int)sh.count;                             // entries of this batch (all >= tau)
        nb = min(nb_all, K - lo);                           // ... that may be consumed
        rank = tid;
        if (CL > 1 && tid < S) {
            // composites are unique (padding zeros excepted, which nobody looks at): rank = #entries greater
#pragma unroll
            for (int q = 1; q < CL; ++q) {
                const unsigned long long* lst = lists + q * S;
                int lo_i = 0, n_i = S;          // first position whose value is < mine (the list is descending)
                while (n_i > 0) {
                    const int half = n_i >> 1;
                    const bool gt = lst[lo_i + half] > mine;
                    lo_i = gt ? lo_i + half + 1 : lo_i;
                    n_i = gt ? n_i - half - 1 : half;
                }
                rank += lo_i;
            }
        }
        }   // !presorted
        const bool real = p.presorted ? (tid < S && rank < nb) : (tid < S && mine != 0ull && mine >= tau && rank < nb);
        const uint32_t my_i = p.presorted ? (real ? (uint32_t)p.rank_idx[(long long)b * BATCH + rank] : 0u)
                                          : 0xFFFFFFFFu - (uint32_t)(mine & 0xFFFFFFFFull);
        PH(5);
        if (p.mode == MODE_RANK) {   // the first batch is all this launch computes
            if (real) p.rank_idx[(long long)b * BATCH + rank] = (int)my_i;
            if (tid == 0 && crank == 0) { p.rank_n[b] = nb; p.rank_more[b] = (nb_all < K) ? 1 : 0; }
            break;
        }

        // ---- 4a. top-k outputs (predictor.py:58-60) -------------------------------------------------
        if (p.mode == MODE_TOPK) {
            if (real) write_topk_row(p, b, (long long)b * p.k + lo + rank, my_i, scores, anc, remap);
            lo += nb_all; lo_tau = tau; have_lo = true;
            cl_sync<CL>();   // my list / tau are rewritten by the next batch while peers may still be copying them
            continue;
        }

        // ---- 4b. boxes of the batch, replicated by rank ------------------------------------------------
        float4 raw = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.rows_fetched && tid == 0 && crank == 0)
            atomicAdd(p.rows_fetched, (unsigned long long)((p.presorted && p.reg_compact) ? max(nb - p.compact_rows, 0) : nb));
        if (real) {
            // reg_compact is only set for a presorted launch (proposals_presorted_enqueue), so ranked_raw_box reads it
            // in presorted launches only
            raw = ranked_raw_box(p, b, rank, my_i);
            float4 c;
            float ca;
            canonical_box(raw, thr, c, ca);
#pragma unroll
            for (int q = 0; q < CL; ++q) {
                cl_peer<CL>(cbox_all, (crank + q) % CL)[rank] = c;
                cl_peer<CL>(carea_all, (crank + q) % CL)[rank] = ca;
            }
        }
        cl_sync<CL>();                          // barrier 2
        PH(6);

        // ---- 4c. greedy NMS rounds over this batch ---------------------------------------------------
        for (int pos = 0; pos < nb && nkept < p.max_out; pos += NMS_CHUNK, par ^= 1) {
            const int C = min(NMS_CHUNK, nb - pos);
            unsigned int* mk = mask32 + par * (NMS_CHUNK * 4);
            // the other parity's mask serves the NEXT round: no peer writes to it before the barrier below
            for (int k = tid; k < NMS_CHUNK * 4; k += T) mask32[(par ^ 1) * (NMS_CHUNK * 4) + k] = 0u;
            const int gt = (int)crank * T + tid;
            if (nkept > 0) {   // candidates vs kept list: thread = (candidate c, part), kept j strided by PARTS
                const int c = gt & (NMS_CHUNK - 1), part = gt >> 7;
                if (c < C && kept_list_suppresses<4>(cbox_all[pos + c], carea_all[pos + c], kbox, karea, part, PARTS, nkept, thr))
                    atomicOr(&sh.dead_w[c >> 5], 1u << (c & 31));
            }
            {   // predecessor masks of the round: bit j of row i set iff j < i and j suppresses i.  Folded triangle
                // over ALL candidates of the round (independent of the kept-list outcome): TS-thread team r takes
                // rows r + 1 and C - 1 - r
                const int r = gt / TS, sub = gt % TS;
                const int iA = r + 1, iB = C - 1 - r;
                const int len = (iA < iB) ? iA + iB : (iA == iB ? iA : 0);
                auto pair = [&](int e, int& i, int& j) -> bool {
                    i = e < iA ? iA : iB;
                    j = e < iA ? e : e - iA;
                    return pair_suppresses(thr, cbox_all[pos + j], carea_all[pos + j], cbox_all[pos + i], carea_all[pos + i]);
                };
                int e = sub;
                for (; e + TS < len; e += 2 * TS) {      // two independent tests in flight
                    int i0, j0, i1, j1;
                    const bool s0 = pair(e, i0, j0), s1 = pair(e + TS, i1, j1);
                    if (s0) atomicOr(&mk[i0 * 4 + (j0 >> 5)], 1u << (j0 & 31));
                    if (s1) atomicOr(&mk[i1 * 4 + (j1 >> 5)], 1u << (j1 & 31));
                }
                if (e < len) {
                    int i0, j0;
                    if (pair(e, i0, j0)) atomicOr(&mk[i0 * 4 + (j0 >> 5)], 1u << (j0 & 31));
                }
            }
            __syncthreads();
            PH(7);
            if (tid < 4 * CL) {   // my suppressed bits -> every CTA's dead_all[par][crank]
                const int q = tid >> 2, w = tid & 3;
                cl_peer<CL>(&sh.dead_all[par][crank][0], (unsigned)q)[w] = sh.dead_w[w];
            }
            if (CL > 1) {
                // publish the rows my teams own (rows are disjoint between CTAs): T/TS teams x 2 rows x 4 words
                for (int k = tid; k < (T / TS) * 8; k += T) {
                    const int team = (int)crank * (T / TS) + (k >> 3), which = (k >> 2) & 1, w = k & 3;
                    const int rA = team + 1, rB = C - 1 - team;
                    if (rA < rB || (rA == rB && which == 0)) {
                        const int row = which == 0 ? rA : rB;
                        const unsigned int v = mk[row * 4 + w];
                        if (v != 0u) {
#pragma unroll
                            for (int q = 1; q < CL; ++q) cl_peer<CL>(mk, (crank + q) % CL)[row * 4 + w] = v;
                        }
                    }
                }
            }
            cl_sync<CL>();                      // the round's barrier
            PH(9);
            if (warp == 0) {   // the round's greedy order; candidates suppressed by the kept list do not enter it
                unsigned U[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    unsigned dead_w = 0u;
                    if (nkept > 0) {
#pragma unroll
                        for (int g = 0; g < CL; ++g) dead_w |= sh.dead_all[par][g][q];
                    }
                    U[q] = __ballot_sync(0xffffffffu, q * 32 + lane < C) & ~dead_w;
                }
                const int nk = resolve_round(reinterpret_cast<const uint4*>(mk), U, nkept, p.max_out, slot, nullptr);
                if (lane == 0) sh.nk = nk;
                if (lane < 4) sh.dead_w[lane] = 0u;
            }
            __syncthreads();
            PH(10);
            if (tid < C && slot[tid] >= 0) {      // every CTA appends to its own copy of the kept list
                const int s = slot[tid];
                kbox[s] = cbox_all[pos + tid];
                karea[s] = carea_all[pos + tid];
            }
            if (real && rank >= pos && rank < pos + C) {   // the owner of a kept candidate writes its outputs
                const int s = slot[rank - pos];
                if (s >= 0) write_kept_row(p, b, s, raw, scores, my_i, remap);
            }
            nkept += sh.nk;
            __syncthreads();
            PH(11);
        }
        lo += nb_all; lo_tau = tau; have_lo = true;
        if (nkept >= p.max_out) break;
    }
    if (CL > 1) cg::this_cluster().sync();   // no CTA leaves while a peer may still access its shared memory
    if (p.mode == MODE_TOPK || p.mode == MODE_RANK) return;
    if (p.presorted) {
        const bool redo = nkept < p.max_out && (cut || p.rank_more[b] != 0);
        if (tid == 0 && crank == 0) p.redo_flags[b] = redo ? 1 : 0;
        if (redo) return;
    }
    if (p.flags_out && nkept < p.max_out && N < p.full_n) {   // the unfiltered kernel redoes this image
        if (tid == 0 && crank == 0) p.flags_out[b] = 1;
        return;
    }
    pad_outputs(p, b, nkept, (int)crank * T + tid, NT);
    if (tid == 0 && crank == 0) p.valid[b] = nkept;
    PH(12);
    PH_FLUSH;
}

// ------------------------------------------------------------------------------------------------
// Matrix NMS over the ranks a MODE_RANK launch produced.  The lazy kernels above do the minimum number of pair
// tests but on one or two SMs per image with a barrier between every phase (25 % of the issue capacity of
// the SMs they hold).  Here the pair tests of the first T = nms_rows ranks are done up front by the whole GPU,
//   nms_mask_kernel    CTA (word w, image b): the 32 boxes of ranks [32w, 32w+32) in shared memory; every thread
//                      owns a later rank i and packs "j suppresses i" of those 32 predecessors into one word
//   nms_sweep_kernel   one 128-thread CTA per image walks the ranks in chunks of 128: a candidate is dead if a row
//                      word ANDed with the kept bits of the earlier chunks is non-zero, the chunk itself is resolved
//                      with the same parallel sweeps as above, kept boxes are decoded again and written out
// ~1.5x the pair tests of the lazy kernel (205 k instead of 138 k per image at C2, T = 640), no dependency
// between them.  An image that has not filled max_out when the T ranks are used up raises redo_flags[b] and
// the lazy kernel redoes it.  Results are bit-identical: same composites, same order, same pair test.
// Measured at C2 (profiles/r2g_*): rank launch 11.7 us + mask 31 us (14.0 M warp instructions, 34 per pair test)
// + sweep 19 us against 43.6 us for the lazy kernel, and MORE instructions in total (20 M vs 12 M per launch), so
// with several steps in flight the GPU -- which is issue-bound -- loses throughput (1.28 M vs 1.37 M images/s).
// The path is therefore opt-in (TFRPN_NMS_PATH=matrix); the lazy kernels stay the default.
// ------------------------------------------------------------------------------------------------
constexpr int MASK_THREADS = 256;
constexpr int SWEEP_THREADS = NMS_CHUNK;   // 128

// ranks of image b the matrix covers, and whether the image has ranks beyond them
__device__ __forceinline__ int matrix_rows(const PropParams& p, int b, bool& more) {
    int n = p.rank_n[b];
    more = p.rank_more[b] != 0;
    int cap = p.nms_rows;
    if (p.reg_compact && p.compact_rows < cap) cap = p.compact_rows;   // only the gathered rows can be decoded
    if (n > cap) { n = cap; more = true; }
    return n;
}

__global__ void __launch_bounds__(MASK_THREADS) nms_mask_kernel(const __grid_constant__ PropParams p) {
    __shared__ float4 jbox[32];
    __shared__ float jarea[32];
    const int b = blockIdx.y, w = blockIdx.x, tid = threadIdx.x;
    bool more;
    const int n = matrix_rows(p, b, more);
    if (32 * w + 1 >= n) return;                 // no rank of this image has a predecessor in this word
    const IouThreshold thr = p.iou_thr;
    const int* ridx = p.rank_idx + (long long)b * BATCH;
    if (tid < 32) {
        const int j = 32 * w + tid;
        float4 c = TFRPN_FAR_BOX;
        float ca = 0.0f;
        if (j < n) canonical_box(ranked_raw_box(p, b, j, (uint32_t)ridx[j]), thr, c, ca);
        jbox[tid] = c;
        jarea[tid] = ca;
    }
    __syncthreads();
    unsigned int* mrow = p.nms_mask + (long long)b * p.nms_rows * p.mask_words + w;
    for (int i = 32 * w + 1 + tid; i < n; i += MASK_THREADS) {
        float4 ci;
        float ai;
        canonical_box(ranked_raw_box(p, b, i, (uint32_t)ridx[i]), thr, ci, ai);
        const int jmax = min(32, i - 32 * w);    // predecessors of i inside this word
        unsigned int word = 0u;
        if (thr.fast) {
            if (jmax == 32) {
                const f32x2 ai2 = pack2(ai, ai), lo2 = pack2(thr.lo_s, thr.lo_s);
                unsigned int cand = 0u;              // pairs that pass the cheap pre-test ...
#pragma unroll 8
                for (int jj = 0; jj < 32; jj += 2)
                    cand |= nms_maybe2(ci, ai2, jbox[jj], jarea[jj], jbox[jj + 1], jarea[jj + 1], lo2) << jj;
                while (cand != 0u) {                 // ... get the exact test (a handful per row)
                    const int jj = __ffs(cand) - 1;
                    cand &= cand - 1u;
                    word |= nms_suppresses_fast(jbox[jj], jarea[jj], ci, ai, thr) ? (1u << jj) : 0u;
                }
            } else {
                for (int jj = 0; jj < jmax; ++jj)
                    word |= nms_suppresses_filtered(jbox[jj], jarea[jj], ci, ai, thr) ? (1u << jj) : 0u;
            }
        } else {
            for (int jj = 0; jj < jmax; ++jj)
                word |= nms_suppresses(jbox[jj], jarea[jj], ci, ai, thr) ? (1u << jj) : 0u;
        }
        mrow[(long long)i * p.mask_words] = word;
    }
}

__global__ void __launch_bounds__(SWEEP_THREADS) nms_sweep_kernel(const __grid_constant__ PropParams p) {
    __shared__ unsigned int kw[BATCH / 32];      // kept bits by rank
    __shared__ uint4 pr_s[NMS_CHUNK];            // predecessor words of the chunk's candidates (inside the chunk)
    __shared__ unsigned int dead_s[4];
    __shared__ int slot[NMS_CHUNK];
    __shared__ int s_nk;
    const int b = blockIdx.x, tid = threadIdx.x, lane = lane_id(), warp = warp_id();
    bool more;
    const int n = matrix_rows(p, b, more);
    const int W = p.mask_words;
    const int* ridx = p.rank_idx + (long long)b * BATCH;
    const float* scores = p.scores + (long long)b * p.N;
    const unsigned int* mimg = p.nms_mask + (long long)b * p.nms_rows * W;
    if (tid < BATCH / 32) kw[tid] = 0u;
    if (tid < 4) dead_s[tid] = 0u;
    __syncthreads();
    int nkept = 0;
    for (int pos = 0; pos < n && nkept < p.max_out; pos += NMS_CHUNK) {
        const int C = min(NMS_CHUNK, n - pos);
        const int i = pos + tid;
        const int w0 = pos >> 5;                 // first word of this chunk
        bool dead = false;
        uint4 pr = make_uint4(0u, 0u, 0u, 0u);
        if (tid < C) {
            const unsigned int* row = mimg + (long long)i * W;
            const int wlast = (i - 1) >> 5;      // last word the mask kernel wrote for row i (i >= 1), -1 for i == 0
            unsigned int hit = 0u;
            for (int w = 0; w < w0; ++w) hit |= row[w] & kw[w];
            dead = hit != 0u;
            if (i > 0) {
                pr.x = (w0 <= wlast) ? row[w0] : 0u;
                pr.y = (w0 + 1 <= wlast) ? row[w0 + 1] : 0u;
                pr.z = (w0 + 2 <= wlast) ? row[w0 + 2] : 0u;
                pr.w = (w0 + 3 <= wlast) ? row[w0 + 3] : 0u;
            }
            pr_s[tid] = pr;
            if (dead) atomicOr(&dead_s[tid >> 5], 1u << (tid & 31));
        }
        __syncthreads();
        if (warp == 0) {   // the chunk's greedy order; candidates dead by the earlier chunks do not enter it
            unsigned U[4], kept[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) U[q] = __ballot_sync(0xffffffffu, q * 32 + lane < C) & ~dead_s[q];
            const int nk = resolve_round(pr_s, U, nkept, p.max_out, slot, kept);
            __syncwarp();   // every lane has read dead_s[] above
            if (lane < 4) {
                kw[w0 + lane] = lane == 0 ? kept[0] : lane == 1 ? kept[1] : lane == 2 ? kept[2] : kept[3];
                dead_s[lane] = 0u;
            }
            if (lane == 0) s_nk = nk;
        }
        __syncthreads();
        if (tid < C && slot[tid] >= 0) {         // (matrix_applies excludes remapped launches)
            const uint32_t idx = (uint32_t)ridx[i];
            write_kept_row(p, b, slot[tid], ranked_raw_box(p, b, i, idx), scores, idx, nullptr);
        }
        nkept += s_nk;
        __syncthreads();
    }
    const bool redo = nkept < p.max_out && more;
    if (tid == 0) p.redo_flags[b] = redo ? 1 : 0;
    if (redo) return;                            // the lazy kernel redoes this image and writes all of its outputs
    pad_outputs(p, b, nkept, tid, SWEEP_THREADS);
    if (tid == 0) p.valid[b] = nkept;
}

// ------------------------------------------------------------------------------------------------
// Multi-class combined NMS (tfrpn_nms_multiclass): C classes of (B,K,C) scores with shared (q = 1) or
// class-specific (q = C) boxes.  Three launches:
//   nms_mc_stage_kernel   one CTA per (image, class): the class's candidates (score > threshold, or all) in
//                         ASCENDING original index -> compact scores / remap / boxes, the interface of the
//                         large-N prefilter, so proposal_kernel's composite breaks ties to the lower index
//                         (column layout: reads column c with stride C).  The same arrays from coalesced score
//                         rows: nms_mc_row_count_kernel + nms_mc_row_scatter_kernel (row layout, see there)
//   proposal_kernel       MODE_NMS on the B*C segments (launch_one), keep lists into the workspace
//   nms_mc_merge_kernel   G CTAs per image: merge the C keep lists by rank, scatter and pad the outputs
// ------------------------------------------------------------------------------------------------
constexpr int MC_STAGE_THREADS = 256;
constexpr int MC_STAGE_ITEMS = 4;      // consecutive positions per thread and sweep step (40 registers: 6 CTAs per SM)
constexpr int MC_MERGE_THREADS = 512;

struct McStageParams {
    const float* scores;   // (B,K,C)
    const float4* boxes;   // (B,K,q)
    int K, C, q, use_sthr;
    float sthr;
    float* cand_scores;    // (B*C, K) per segment, ascending original index
    int* remap;            // (B*C, K)
    float4* cand_boxes;    // (B*C, K)
    int* counts;           // (B*C)
};

__global__ void __launch_bounds__(MC_STAGE_THREADS) nms_mc_stage_kernel(McStageParams p) {
    __shared__ unsigned int wtot[MC_STAGE_THREADS / 32];
    const int seg = blockIdx.x, b = seg / p.C, c = seg - b * p.C;   // the classes of an image run side by side
    const int tid = threadIdx.x, lane = lane_id(), warp = warp_id();
    const float* sc = p.scores + (long long)b * p.K * p.C + c;
    const float4* bx = p.boxes + (long long)b * p.K * p.q + (p.q == 1 ? 0 : c);
    float* os = p.cand_scores + (long long)seg * p.K;
    int* orm = p.remap + (long long)seg * p.K;
    float4* ob = p.cand_boxes + (long long)seg * p.K;
    unsigned int run = 0;
    for (int base = 0; base < p.K; base += MC_STAGE_THREADS * MC_STAGE_ITEMS) {
        const int k0 = base + tid * MC_STAGE_ITEMS;
        float s[MC_STAGE_ITEMS];
        unsigned int take = 0;
#pragma unroll
        for (int u = 0; u < MC_STAGE_ITEMS; ++u) {
            s[u] = 0.0f;
            if (k0 + u < p.K) {
                s[u] = __ldg(sc + (long long)(k0 + u) * p.C);
                if (!p.use_sthr || s[u] > p.sthr) take |= 1u << u;   // score_key's rule
            }
        }
        const unsigned int n = __popc(take);
        const unsigned int incl = (unsigned int)warp_incl_scan((int)n);
        if (lane == 31) wtot[warp] = incl;
        __syncthreads();
        unsigned int woff = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < MC_STAGE_THREADS / 32; ++w) {
            const unsigned int t = wtot[w];
            woff += w < warp ? t : 0u;
            tot += t;
        }
        __syncthreads();                                // wtot is rewritten by the next step
        unsigned int o = run + woff + incl - n;
#pragma unroll
        for (int u = 0; u < MC_STAGE_ITEMS; ++u) {
            if ((take >> u) & 1u) {
                const int k = k0 + u;
                os[o] = s[u];
                orm[o] = k;
                ob[o] = ldg_f4(bx + (long long)k * p.q);
                ++o;
            }
        }
        run += tot;
    }
    if (tid == 0) p.counts[seg] = (int)run;
}

// Row layout of the staging: grid (slices, B) over coalesced (K, C) score rows, like pre_count / pre_scatter_kernel.
// Warp w of slice s owns rows [r_lo, r_hi) (flat elements [r_lo * C, r_hi * C), read 32 consecutive at a time).
// count: candidates per (image, slice, warp, class) -> row_cnt; scatter: each CTA turns the counts of the
// (slice, warp) pairs before its own into per-warp, per-class offsets (the last slice also writes counts[]), then
// every warp walks its range in order; lanes with the same class rank themselves with __match_any_sync.
constexpr int MC_ROW_THREADS = 256;
constexpr int MC_ROW_WARPS = MC_ROW_THREADS / 32;
constexpr int MC_ROW_MAX_C = 1024;     // the per-warp, per-class table lives in shared memory (32 KB)
struct McRowParams {
    McStageParams g;
    int slices, slice_rows;
    int* row_cnt;          // (B, slices, MC_ROW_WARPS, C)
};
__device__ __forceinline__ void mc_row_range(const McRowParams& p, int& lo, int& hi) {
    const int slo = blockIdx.x * p.slice_rows, shi = min(p.g.K, slo + p.slice_rows);
    const int sub = (p.slice_rows + MC_ROW_WARPS - 1) / MC_ROW_WARPS;
    const int rlo = min(shi, slo + warp_id() * sub), rhi = min(shi, rlo + sub);
    lo = rlo * p.g.C;
    hi = rhi * p.g.C;
}
__global__ void __launch_bounds__(MC_ROW_THREADS) nms_mc_row_count_kernel(McRowParams p) {
    extern __shared__ unsigned int wc[];   // [MC_ROW_WARPS][C]
    const int b = blockIdx.y, lane = lane_id(), warp = warp_id(), Cn = p.g.C;
    unsigned int* mine = wc + warp * Cn;
    for (int c = lane; c < Cn; c += 32) mine[c] = 0u;
    __syncwarp();
    int lo, hi;
    mc_row_range(p, lo, hi);
    const float* sc = p.g.scores + (long long)b * p.g.K * Cn;
    for (int f = lo + lane; f - lane < hi; f += 32) {
        const bool in = f < hi;
        const float s = in ? __ldg(sc + f) : 0.0f;
        const bool take = in && (!p.g.use_sthr || s > p.g.sthr);
        const int c = f % Cn;
        const unsigned m = __match_any_sync(0xffffffffu, take ? c : -1);
        if (take && lane == __ffs(m) - 1) mine[c] += __popc(m);
        __syncwarp();
    }
    int* out = p.row_cnt + (((long long)b * p.slices + blockIdx.x) * MC_ROW_WARPS + warp) * Cn;
    for (int c = lane; c < Cn; c += 32) out[c] = (int)mine[c];
}
__global__ void __launch_bounds__(MC_ROW_THREADS) nms_mc_row_scatter_kernel(McRowParams p) {
    extern __shared__ unsigned int off[];   // [MC_ROW_WARPS][C]
    const int b = blockIdx.y, s = blockIdx.x, lane = lane_id(), warp = warp_id(), Cn = p.g.C;
    const int* cnt = p.row_cnt + (long long)b * p.slices * MC_ROW_WARPS * Cn;
    const bool last = s == p.slices - 1;
    for (int c = threadIdx.x; c < Cn; c += MC_ROW_THREADS) {
        int run = 0;
        for (int q = 0; q < s * MC_ROW_WARPS; ++q) run += cnt[(long long)q * Cn + c];
        for (int w = 0; w < MC_ROW_WARPS; ++w) {
            off[w * Cn + c] = (unsigned)run;
            run += cnt[(long long)(s * MC_ROW_WARPS + w) * Cn + c];
        }
        if (last) p.g.counts[(long long)b * Cn + c] = run;
    }
    __syncthreads();
    unsigned int* mine = off + warp * Cn;
    int lo, hi;
    mc_row_range(p, lo, hi);
    const float* sc = p.g.scores + (long long)b * p.g.K * Cn;
    for (int f = lo + lane; f - lane < hi; f += 32) {
        const bool in = f < hi;
        const float v = in ? __ldg(sc + f) : 0.0f;
        const bool take = in && (!p.g.use_sthr || v > p.g.sthr);
        const int k = f / Cn, c = f - k * Cn;
        const unsigned m = __match_any_sync(0xffffffffu, take ? c : -1);
        if (take) {
            const long long o = ((long long)b * Cn + c) * p.g.K + mine[c] + __popc(m & ((1u << lane) - 1u));
            p.g.cand_scores[o] = v;
            p.g.remap[o] = k;
            p.g.cand_boxes[o] = ldg_f4(p.g.boxes + ((long long)b * p.g.K + k) * p.g.q + (p.g.q == 1 ? 0 : c));
        }
        __syncwarp();
        if (take && lane == __ffs(m) - 1) mine[c] += __popc(m);
        __syncwarp();
    }
}

struct McMergeParams {
    const float* ks;       // (B*C, P) keep lists of the per-class NMS: scores, boxes, original indices, lengths
    const float4* kb;
    const int* ki;
    const int* kv;
    int C, P, rows, lmax;  // lmax = min(P, rows): no entry at a list position >= rows can reach an output row
    int use_smem;          // scratch in dynamic shared memory, else in `gscratch` (per image: scratch_bytes)
    char* gscratch;
    long long scratch_bytes;
    float4* out_boxes;     // (B, rows)
    float* out_scores;
    float* out_classes;
    int* valid;
    int* keep_idx;
};

// Merge key: score by VALUE, descending, as a stable torch.sort compares it: +0 == -0, and NaN (either sign) above
// +inf, every NaN equal.  A keep list is in the kernel's order of orderable(score), which agrees with this key except
// that -NaN sorts last there: the list read as [+NaN run][-NaN run][rest] (the "virtual" order) is non-increasing.
__device__ __forceinline__ uint32_t mc_merge_key(float s) {
    if (isnan(s)) return 0xFFFFFFFFu;
    return s == 0.0f ? 0x80000000u : orderable(s);
}
__device__ __forceinline__ int mc_phys(int v, int m, int a, int bn) {   // virtual -> physical list position
    return v < a ? v : (v < a + bn ? m - bn + (v - a) : v - bn);
}

// Grid (B, G): every CTA of an image builds the keys (cheap: <= C * min(P, rows) loads) and ranks every G-th slice of
// the entries; CTA 0 writes the padding and valid.
__global__ void __launch_bounds__(MC_MERGE_THREADS) nms_mc_merge_kernel(McMergeParams p) {
    extern __shared__ float4 smem4[];
    __shared__ unsigned int s_total;
    const int b = blockIdx.x, tid = threadIdx.x, lane = lane_id(), warp = warp_id();
    constexpr int WARPS = MC_MERGE_THREADS / 32;
    char* base = p.use_smem ? reinterpret_cast<char*>(smem4)
                            : p.gscratch + ((long long)b * gridDim.y + blockIdx.y) * p.scratch_bytes;
    int4* meta = reinterpret_cast<int4*>(base);                            // [C] (m, a, bn, L)
    uint32_t* keys = reinterpret_cast<uint32_t*>(meta + p.C);              // [C][lmax] merge keys, virtual order
    const long long seg0 = (long long)b * p.C;
    if (tid == 0) s_total = 0u;
    __syncthreads();
    // ---- 1. per list (one warp each): its NaN runs, then its first L = min(m, lmax) merge keys in virtual order
    unsigned int live = 0;
    for (int c = warp; c < p.C; c += WARPS) {
        const long long seg = seg0 + c;
        const int m = p.kv[seg];
        const float* s = p.ks + seg * p.P;
        int a = 0, bn = 0;
        for (int j = lane; j < m; j += 32) {
            const float v = s[j];
            const bool nan = isnan(v);
            a += (nan && !signbit(v)) ? 1 : 0;
            bn += (nan && signbit(v)) ? 1 : 0;
        }
        a = __reduce_add_sync(0xffffffffu, a);
        bn = __reduce_add_sync(0xffffffffu, bn);
        const int L = min(m, p.lmax);
        if (lane == 0) { meta[c] = make_int4(m, a, bn, L); live += (unsigned int)m; }
        for (int v = lane; v < L; v += 32) keys[(long long)c * p.lmax + v] = mc_merge_key(s[mc_phys(v, m, a, bn)]);
    }
    if (lane == 0 && live) atomicAdd(&s_total, live);
    __syncthreads();
    const int nvalid = min((int)s_total, p.rows);
    // ---- 2. rank of entry (c, v): v + entries of lists c' < c with key >= its key + of lists c' > c with key >
    //      its key (each list is non-increasing in virtual order: a binary search).  Equal keys go to the lower
    //      class, then to the earlier position in the class's list.  Entries ranked >= rows are dropped.
    const long long items = (long long)p.C * p.lmax;
    for (long long it = (long long)blockIdx.y * MC_MERGE_THREADS + tid; it < items; it += (long long)gridDim.y * MC_MERGE_THREADS) {
        const int c = (int)(it / p.lmax), v = (int)(it - (long long)c * p.lmax);
        const int4 mc = meta[c];
        if (v >= mc.w) continue;
        const uint32_t key = keys[it];
        int rank = v;
        for (int c2 = 0; c2 < p.C && rank < p.rows; ++c2) {
            if (c2 == c) continue;
            const uint32_t* kl = keys + (long long)c2 * p.lmax;
            int lo = 0, hi = meta[c2].w;                // first position whose entry does not precede (c, v)
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                const uint32_t k2 = kl[mid];
                if (c2 < c ? k2 >= key : k2 > key) lo = mid + 1; else hi = mid;
            }
            rank += lo;
        }
        if (rank < p.rows) {
            const long long src = (seg0 + c) * p.P + mc_phys(v, mc.x, mc.y, mc.z);
            const long long o = (long long)b * p.rows + rank;
            p.out_boxes[o] = p.kb[src];
            p.out_scores[o] = p.ks[src];
            p.out_classes[o] = (float)c;
            if (p.keep_idx) p.keep_idx[o] = p.ki[src];
        }
    }
    // ---- 3. padding rows (TF pads with 0; keep_idx with -1)
    if (blockIdx.y != 0) return;
    for (int r = nvalid + tid; r < p.rows; r += MC_MERGE_THREADS) {
        const long long o = (long long)b * p.rows + r;
        p.out_boxes[o] = make_float4(0.f, 0.f, 0.f, 0.f);
        p.out_scores[o] = 0.0f;
        p.out_classes[o] = 0.0f;
        if (p.keep_idx) p.keep_idx[o] = -1;
    }
    if (tid == 0) p.valid[b] = nvalid;
}

static size_t cluster_smem_bytes(int cl, int n_staged, int max_out) {
    max_out = (max_out + 3) & ~3;
    const int T = 1024 / cl;                        // (sort slots per CTA)
    const int nchunks = (n_staged + 31) / 32;
    const size_t lmax = (size_t)((nchunks + cl - 1) / cl) * 32;
    size_t s = (size_t)CL_NB * 4;                   // histogram
    s += (size_t)BATCH * 8;                         // my sorted list + the peers'
    s += (size_t)2 * T * 8;                         // sortbuf (double buffer)
    s += (size_t)(BATCH + max_out) * (16 + 4);      // boxes + areas: batch by rank, kept list
    s += (size_t)NMS_CHUNK * (4 + 2 * 16);          // slot, mask32 (two parities)
    s += lmax * 4;                                  // staged score keys of the slice
    return s + 16;
}

int set_attributes_proposals() {
    const int lim = (int)(227 * 1024 - 4096);
    TFRPN_CHECK_CUDA(cudaFuncSetAttribute(proposal_kernel<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    TFRPN_CHECK_CUDA(cudaFuncSetAttribute(proposal_kernel<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    TFRPN_CHECK_CUDA(cudaFuncSetAttribute(proposal_cluster_kernel<1, 1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    TFRPN_CHECK_CUDA(cudaFuncSetAttribute(proposal_cluster_kernel<2, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    TFRPN_CHECK_CUDA(cudaFuncSetAttribute(proposal_cluster_kernel<2, 1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    TFRPN_CHECK_CUDA(cudaFuncSetAttribute(proposal_cluster_kernel<4, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    TFRPN_CHECK_CUDA(cudaFuncSetAttribute(proposal_cluster_kernel<4, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    TFRPN_CHECK_CUDA(cudaFuncSetAttribute(proposal_cluster_kernel<8, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    TFRPN_CHECK_CUDA(cudaFuncSetAttribute(proposal_cluster_kernel<8, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    TFRPN_CHECK_CUDA(cudaFuncSetAttribute(nms_mc_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    return 0;
}

// Shape of the proposal stage for a batch of B images.  Measured (profiles/r2l_prop_shapes.txt): alone on the GPU the
// cluster kernels are faster (C2, B = 64: 2 x 512 = 41 us against 48.8 us; C1, B = 1: 8 x 256 = 28 us against 46 us),
// but they execute more instructions (16.4 M against 13.8 M warp instructions at C2) and hold twice the SMs, so as soon
// as the batch alone can fill the GPU -- and with the target kernels and other steps running beside it -- the one-CTA
// kernel gives more images/s AND the lower step latency (bench.py at C2: 1.42 M images/s, p50 67.6 us against 1.34 M,
// 71.7 us with 2 x 512; C4, B = 32: 196 k against 173 k with 8 x 256).  Hence: B <= 8 -> 8 CTAs x 256 threads per
// image, larger batches -> one CTA per image (proposal_kernel<T>, T picked in launch_one).  TFRPN_PROP_CLUSTER = 10 * t + cl forces a shape (A/B
// switch): cl = 0 one-CTA kernel, 1 / 2 / 4 / 8 CTAs per image; t selects the threads per CTA.
static void pick_cluster(tfrpn_handle h, int B, int& cl, int& threads) {
    const int v = h->opts.prop_cluster;
    if (v >= 0) {
        cl = v % 10;
        const int t = v / 10;
        if (cl != 1 && cl != 2 && cl != 4 && cl != 8) { cl = 0; threads = 1024; return; }
        threads = cl == 1 ? 1024 : cl == 2 ? (t == 1 ? 512 : 1024) : cl == 4 ? (t == 1 ? 256 : 512) : (t == 2 ? 512 : 256);
        return;
    }
    if (B <= 8) { cl = 8; threads = 256; }
    else { cl = 0; threads = 1024; }
}

static IouThreshold make_threshold(float thr) {
    IouThreshold t;
    t.thr = thr;
    t.fast = (thr >= 1e-30f && thr <= 1e30f) ? 1 : 0;
    const float nxt = nextafterf(thr, INFINITY);
    t.mid = ((double)thr + (double)nxt) * 0.5;   // exact: 25 significant bits
    t.lo_f = (float)((double)thr * (1.0 - 1.0 / 4096.0));
    t.hi_f = (float)((double)thr * (1.0 + 1.0 / 4096.0));
    t.lo_s = (float)((double)thr / (1.0 + (double)thr) * (1.0 - 1.0 / 1024.0));
    uint32_t nb;
    memcpy(&nb, &nxt, 4);
    t.tie_up = ((nb & 1u) == 0u) ? 1 : 0;        // a tie rounds to the even mantissa
    return t;
}
// The IoU threshold range TF's CombinedNonMaxSuppression accepts, [0, 1] (-0.0 included).  Outside it NaN would turn
// NMS off, and a negative threshold would let zero-area boxes suppress everything (0 > thr).
int check_iou_threshold(const char* fn, float thr) {
    if (!(thr >= 0.0f && thr <= 1.0f))
        return fail(TFRPN_ERR_BAD_ARG, "%s: iou_threshold = %g must be in [0, 1]", fn, (double)thr);
    return 0;
}

static size_t prop_smem_bytes(int n_staged, int max_out) {
    max_out = (max_out + 3) & ~3;
    size_t s = (size_t)2 * BATCH * 8;               // sortbuf (double buffer)
    s += (size_t)BATCH * 4;                         // sidx
    s += (size_t)(max_out + NMS_CHUNK) * (16 + 4);  // kbox+cbox, karea+carea
    s += (size_t)NMS_CHUNK * (4 + 4 + 16);          // alive, slot, mask16
    s += (size_t)SEL_NB * 4;                        // select / counting-sort histogram
    s += (size_t)n_staged * 4;                      // staged score keys
    return s + 16;
}
constexpr size_t PROP_SMEM_LIMIT = 227 * 1024 - 4096;   // leaves room for the static PropShared
// the kept list lives in shared memory, which bounds max_out
static int check_prop_smem(size_t smem, int max_out) {
    if (smem > PROP_SMEM_LIMIT)
        return fail(TFRPN_ERR_UNSUPPORTED, "NMS: %d output rows need %zu B of shared memory (> %zu)", max_out, smem,
                    PROP_SMEM_LIMIT);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Large-N prefilter.  One CTA per image cannot stream hundreds of thousands of scores several times,
// so when N is large and only the top k << N ranks can ever be consumed, all SMs first cut every image
// down to the entries whose key is >= T, the 22-bit prefix of the key at rank k:
//   pre_hist_kernel pass 0 / 1   2048-bin histograms of key bits [31:21], then [20:10] inside the bin
//                                that holds rank k (shared-memory bins per slice, flushed with global
//                                atomics; the last CTA of an image scans them and publishes the digit)
//   pre_count_kernel             entries >= T per warp sub-slice; the last CTA turns them into offsets
//   pre_scatter_kernel           STABLE compaction (ascending original index, so the lower-index-first
//                                tie rule survives) of scores, original indices and the gathered
//                                boxes / deltas / anchors into (B, Mcap) arrays
// proposal_kernel then runs on the compact arrays (counts / remap above).  An image whose candidate set
// does not fit Mcap (a tie group of thousands of equal keys) is flagged and handled by a second launch
// of the unfiltered kernel, which returns immediately for every other image.
// ------------------------------------------------------------------------------------------------
constexpr int PRE_THREADS = 512;
constexpr int PRE_WARPS = PRE_THREADS / 32;
constexpr int PRE_BINS = 2048;
constexpr int PRE_MIN_N = 40000;      // below this the one-CTA kernel stages every key in shared memory
constexpr int PRE_SLACK = 8192;       // Mcap = k + PRE_SLACK
// NMS over "all" K boxes (or a very large pre-NMS k) rarely looks past the first few thousand ranks: the
// prefilter then keeps only the top PRE_NMS_CAP ranks, and an image whose NMS runs out of candidates
// before max_out boxes are kept raises its flag and is redone by the unfiltered kernel.
constexpr int PRE_NMS_CAP = 6144;
constexpr int PRE_NMS_CAP_MAX_OUT = 384;

struct PreState {
    unsigned int ticket[3];
    unsigned int d1, rem1, above1;
    unsigned int T;
    unsigned int pad[9];
};

struct PreParams {
    const float* scores;
    int N, k, use_sthr;
    float sthr;
    int slices, slice_len, Mcap;
    unsigned int* hist;        // [B][2][PRE_BINS]
    PreState* state;           // [B]
    unsigned int* slice_cnt;   // [B][slices][PRE_WARPS]  per-warp counts, then exclusive offsets
    int* counts;               // [B]
    int* flags;                // [B]
    float* cand_scores;        // [B][Mcap]
    int* remap;                // [B][Mcap]
    const float4* boxes;       // MODE_TOPK gather source / MODE_NMS input (or null)
    long long box_stride;
    float4* cand_boxes;
    const float4* reg;         // (B,N,4) or null
    float4* cand_reg;
    const float4* anchors;     // (N,4)
    float4* cand_anchors;
};

// exclusive block scan of one unsigned per thread (PRE_THREADS threads); returns the exclusive prefix,
// *total gets the block sum
__device__ __forceinline__ unsigned int pre_block_excl_scan(unsigned int v, unsigned int* wtot, unsigned int* total) {
    const unsigned int incl = (unsigned int)warp_incl_scan((int)v);
    if (lane_id() == 31) wtot[warp_id()] = incl;
    __syncthreads();
    unsigned int woff = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < PRE_WARPS; ++w) {
        const unsigned int t = wtot[w];
        woff += (w < warp_id()) ? t : 0u;
        tot += t;
    }
    __syncthreads();
    *total = tot;
    return woff + incl - v;
}

__global__ void __launch_bounds__(PRE_THREADS) pre_hist_kernel(PreParams p, int pass) {
    __shared__ unsigned int sh[PRE_BINS];
    __shared__ unsigned int wtot[PRE_WARPS];
    __shared__ unsigned int s_last;
    const int b = blockIdx.y, tid = threadIdx.x;
    PreState* st = p.state + b;
    for (int i = tid; i < PRE_BINS; i += PRE_THREADS) sh[i] = 0u;
    __syncthreads();
    const unsigned int d1 = pass ? st->d1 : 0u;
    const float* sc = p.scores + (long long)b * p.N;
    const int lo = blockIdx.x * p.slice_len, hi = min(p.N, lo + p.slice_len);
    for (int i = lo + tid; i < hi; i += PRE_THREADS) {
        const uint32_t key = score_key(sc[i], p.use_sthr, p.sthr);
        if (pass == 0) atomicAdd(&sh[key >> 21], 1u);
        else if ((key >> 21) == d1) atomicAdd(&sh[(key >> 10) & (PRE_BINS - 1)], 1u);
    }
    __syncthreads();
    unsigned int* gh = p.hist + ((long long)b * 2 + pass) * PRE_BINS;
    for (int i = tid; i < PRE_BINS; i += PRE_THREADS)
        if (sh[i] != 0u) atomicAdd(&gh[i], sh[i]);
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(&st->ticket[pass], 1u) == gridDim.x - 1) ? 1u : 0u;
    __syncthreads();
    if (s_last == 0u) return;
    __threadfence();
    // last CTA of this image: find the bin that holds rank r, scanning from the top (thread 0 = top bins)
    const unsigned int r = pass ? st->rem1 : (unsigned int)min(p.k, p.N);
    constexpr int PER = PRE_BINS / PRE_THREADS;   // 4
    unsigned int c[PER], sum = 0;
#pragma unroll
    for (int q = 0; q < PER; ++q) {
        c[q] = __ldcg(gh + (PRE_BINS - 1 - (tid * PER + q)));
        sum += c[q];
    }
    unsigned int total;
    const unsigned int excl = pre_block_excl_scan(sum, wtot, &total);
    if (excl < r && r <= excl + sum) {
        unsigned int acc = excl;
#pragma unroll
        for (int q = 0; q < PER; ++q) {
            if (acc < r && r <= acc + c[q]) {
                const unsigned int d = (unsigned int)(PRE_BINS - 1 - (tid * PER + q));
                if (pass == 0) {
                    st->d1 = d;
                    st->rem1 = r - acc;
                    st->above1 = acc;
                } else {
                    st->T = (st->d1 << 21) | (d << 10);
                    const unsigned int M = st->above1 + acc + c[q];     // entries with key >= T
                    const bool over = M > (unsigned int)p.Mcap;
                    p.flags[b] = over ? 1 : 0;
                    p.counts[b] = over ? 0 : (int)M;
                }
            }
            acc += c[q];
        }
    }
}

// count / scatter work on per-WARP sub-slices (warp w of slice s owns entries [lo + w*sub, lo + (w+1)*sub)), so
// neither needs a block-wide scan per chunk: a warp counts with ballots, and scatters from its own offset.
__device__ __forceinline__ void pre_warp_range(const PreParams& p, int slice, int& lo, int& hi) {
    const int slo = slice * p.slice_len, shi = min(p.N, slo + p.slice_len);
    const int sub = (((p.slice_len + PRE_WARPS - 1) / PRE_WARPS) + 31) & ~31;
    lo = min(shi, slo + warp_id() * sub);
    hi = min(shi, lo + sub);
}

__global__ void __launch_bounds__(PRE_THREADS) pre_count_kernel(PreParams p) {
    __shared__ unsigned int wtot[PRE_WARPS];
    __shared__ unsigned int s_last;
    const int b = blockIdx.y, tid = threadIdx.x, lane = lane_id();
    if (p.flags[b] != 0) return;
    PreState* st = p.state + b;
    const unsigned int T = st->T;
    const float* sc = p.scores + (long long)b * p.N;
    int lo, hi;
    pre_warp_range(p, blockIdx.x, lo, hi);
    unsigned int mine = 0;
    for (int i = lo + lane; i < hi; i += 32) mine += (score_key(sc[i], p.use_sthr, p.sthr) >= T) ? 1u : 0u;
    mine = __reduce_add_sync(0xffffffffu, mine);
    unsigned int* cnt = p.slice_cnt + (long long)b * p.slices * PRE_WARPS;
    if (lane == 0) cnt[blockIdx.x * PRE_WARPS + warp_id()] = mine;
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(&st->ticket[2], 1u) == gridDim.x - 1) ? 1u : 0u;
    __syncthreads();
    if (s_last == 0u) return;
    __threadfence();
    // last CTA: exclusive scan over all sub-slices; thread t owns the PRE_WARPS entries of slice t
    unsigned int v[PRE_WARPS], sum = 0;
#pragma unroll
    for (int w = 0; w < PRE_WARPS; ++w) {
        v[w] = tid < p.slices ? __ldcg(cnt + tid * PRE_WARPS + w) : 0u;
        sum += v[w];
    }
    unsigned int total;
    unsigned int run = pre_block_excl_scan(sum, wtot, &total);
    if (tid < p.slices) {
#pragma unroll
        for (int w = 0; w < PRE_WARPS; ++w) {
            cnt[tid * PRE_WARPS + w] = run;
            run += v[w];
        }
    }
}

__global__ void __launch_bounds__(PRE_THREADS) pre_scatter_kernel(PreParams p) {
    const int b = blockIdx.y, lane = lane_id();
    if (p.flags[b] != 0) return;
    const unsigned int T = p.state[b].T;
    const float* sc = p.scores + (long long)b * p.N;
    int lo, hi;
    pre_warp_range(p, blockIdx.x, lo, hi);
    unsigned int running = p.slice_cnt[((long long)b * p.slices + blockIdx.x) * PRE_WARPS + warp_id()];
    const long long ob = (long long)b * p.Mcap;
    for (int base = lo; base < hi; base += 32) {
        const int i = base + lane;
        float s = 0.0f;
        bool take = false;
        if (i < hi) {
            s = sc[i];
            take = score_key(s, p.use_sthr, p.sthr) >= T;
        }
        const unsigned int bal = __ballot_sync(0xffffffffu, take);
        if (take) {
            const long long o = ob + running + __popc(bal & ((1u << lane) - 1u));
            p.cand_scores[o] = s;
            p.remap[o] = i;
            if (p.boxes) p.cand_boxes[o] = ldg_f4(p.boxes + (long long)b * p.box_stride + i);
            if (p.reg) {
                p.cand_reg[o] = ldg_f4(p.reg + (long long)b * p.N + i);
                p.cand_anchors[o] = ldg_f4(p.anchors + i);
            }
        }
        running += __popc(bal);
    }
}

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }
static int pre_slices(int B, int N) {
    int s = (592 + B - 1) / B;                           // ~4 CTAs per SM over the batch
    s = min(s, (N + 2047) / 2048);                       // at least 2048 entries per slice
    return max(1, min(s, PRE_THREADS));
}
static bool pre_applies(int N, int k) {
    static const bool off = getenv("TFRPN_NO_PREFILTER") != nullptr;   // A/B switch
    return !off && k > 0 && N >= PRE_MIN_N && (long long)k * 4 <= N;
}
static size_t prefilter_bytes_for(int B, int N, int k);
size_t matrix_workspace_bytes(int B);
size_t prefilter_workspace_bytes(int B, int N, int k) {   // = the proposal side's workspace: prefilter arrays or the NMS matrix
    if (k <= 0) k = N;
    const size_t a = prefilter_bytes_for(B, N, k), b = prefilter_bytes_for(B, N, min(k, PRE_NMS_CAP));
    const size_t c = B > 0 ? matrix_workspace_bytes(B) : 0;
    return std::max(std::max(a, b), c);
}
static size_t prefilter_bytes_for(int B, int N, int k) {
    if (B <= 0 || !pre_applies(N, k)) return 0;
    const size_t Mcap = (size_t)min(N, k + PRE_SLACK);
    size_t b = 0;
    b += align256((size_t)B * 2 * PRE_BINS * 4 + (size_t)B * sizeof(PreState));   // hist + state (one memset)
    b += align256((size_t)B * PRE_THREADS * PRE_WARPS * 4);   // sub-slice counts / offsets
    b += align256((size_t)B * 4) * 2;                  // counts, flags
    b += align256((size_t)B * Mcap * 4) * 2;           // scores, remap
    b += align256((size_t)B * Mcap * 16) * 2;          // boxes | (reg, anchors)
    return b + 256;
}

static int launch_one(tfrpn_handle h, PropParams& p, int B, cudaStream_t st);
static int launch_cluster(tfrpn_handle h, PropParams& p, int B, int cl, int threads, cudaStream_t st);

static int launch_prefiltered(tfrpn_handle h, PropParams& p, int k_eff, int B, cudaStream_t st) {
    const int N = p.N, Mcap = min(N, k_eff + PRE_SLACK);
    const bool truncated = k_eff < p.k;
    char* ws = nullptr;
    if (int rc = ensure_workspace_prop(h, prefilter_bytes_for(B, N, k_eff), st, &ws)) return rc;
    PreParams q = {};
    q.scores = p.scores; q.N = N; q.k = k_eff; q.use_sthr = p.use_sthr; q.sthr = p.score_threshold;
    q.slices = pre_slices(B, N);
    q.slice_len = (N + q.slices - 1) / q.slices;
    q.Mcap = Mcap;
    char* c = ws;
    const size_t zero_bytes = (size_t)B * 2 * PRE_BINS * 4 + (size_t)B * sizeof(PreState);
    q.hist = reinterpret_cast<unsigned int*>(c);
    q.state = reinterpret_cast<PreState*>(c + (size_t)B * 2 * PRE_BINS * 4);
    c += align256(zero_bytes);
    q.slice_cnt = reinterpret_cast<unsigned int*>(c); c += align256((size_t)B * PRE_THREADS * PRE_WARPS * 4);
    q.counts = reinterpret_cast<int*>(c); c += align256((size_t)B * 4);
    q.flags = reinterpret_cast<int*>(c); c += align256((size_t)B * 4);
    q.cand_scores = reinterpret_cast<float*>(c); c += align256((size_t)B * Mcap * 4);
    q.remap = reinterpret_cast<int*>(c); c += align256((size_t)B * Mcap * 4);
    float4* arr0 = reinterpret_cast<float4*>(c); c += align256((size_t)B * Mcap * 16);
    float4* arr1 = reinterpret_cast<float4*>(c);
    if (p.reg) { q.reg = p.reg; q.cand_reg = arr0; q.anchors = p.anchors; q.cand_anchors = arr1; }
    else if (p.boxes) { q.boxes = p.boxes; q.box_stride = p.box_stride; q.cand_boxes = arr0; }
    TFRPN_CHECK_CUDA(cudaMemsetAsync(q.hist, 0, zero_bytes, st));
    const dim3 grid(q.slices, B);
    pre_hist_kernel<<<grid, PRE_THREADS, 0, st>>>(q, 0);
    TFRPN_AFTER_LAUNCH("pre_hist_kernel");
    pre_hist_kernel<<<grid, PRE_THREADS, 0, st>>>(q, 1);
    TFRPN_AFTER_LAUNCH("pre_hist_kernel");
    pre_count_kernel<<<grid, PRE_THREADS, 0, st>>>(q);
    TFRPN_AFTER_LAUNCH("pre_count_kernel");
    pre_scatter_kernel<<<grid, PRE_THREADS, 0, st>>>(q);
    TFRPN_AFTER_LAUNCH("pre_scatter_kernel");
    // the one-CTA-per-image kernel on the compact arrays ...
    PropParams c1 = p;
    c1.N = Mcap; c1.scores = q.cand_scores; c1.counts = q.counts; c1.remap = q.remap;
    c1.flags = q.flags; c1.flag_mode = 1;
    if (truncated) {   // every candidate may be consumed, up to the caller's k; full_n = ranks an unfiltered run may use
        c1.k = min(Mcap, p.k);
        c1.flags_out = q.flags;
        c1.full_n = min(N, p.k);
    }
    if (p.reg) { c1.reg = arr0; c1.anchors = arr1; c1.anchors_batched = 1; }
    else if (p.boxes) { c1.boxes = arr0; c1.box_stride = Mcap; }
    if (int rc = launch_one(h, c1, B, st)) return rc;
    // ... and the unfiltered kernel for the images whose candidates did not fit (normally none)
    PropParams c2 = p;
    c2.flags = q.flags; c2.flag_mode = 2;
    return launch_one(h, c2, B, st);
}

// ---- matrix NMS launch sequence (small N): rank launch -> mask -> sweep -> lazy kernel for flagged images ----
static int matrix_rows_of(tfrpn_handle h) {
    int r = h->opts.nms_rows > 0 ? h->opts.nms_rows : 640;
    r = (r + 31) & ~31;
    return r < 32 ? 32 : (r > BATCH ? BATCH : r);
}
size_t matrix_workspace_bytes(int B) {   // sized for the largest row count, so TFRPN_NMS_ROWS never outgrows a reservation
    return align256((size_t)B * BATCH * 4) + 3 * align256((size_t)B * 4) + align256((size_t)B * BATCH * (BATCH / 32) * 4) + 256;
}
static bool matrix_applies(tfrpn_handle h, const PropParams& p) {
    if (!h || h->opts.nms_lazy || p.mode == MODE_TOPK || p.counts || p.remap || p.flag_mode != 0 || p.presorted) return false;
    return p.max_out >= 1 && cluster_smem_bytes(2, p.N, p.max_out) <= PROP_SMEM_LIMIT;   // the rank launch stages every key
}
// mask + sweep over ranks already produced (rank_idx / rank_n / rank_more set in p); `mask` holds B * rows * rows/32 words
static int launch_mask_sweep(tfrpn_handle h, PropParams& p, int B, int rows, unsigned int* mask, cudaStream_t st) {
    p.nms_mask = mask; p.nms_rows = rows; p.mask_words = rows / 32;
    prof_begin(h, TFRPN_K_NMS_MASK, st);
    nms_mask_kernel<<<dim3(p.mask_words, B), MASK_THREADS, 0, st>>>(p);
    prof_end(h, st);
    TFRPN_AFTER_LAUNCH("nms_mask_kernel");
    prof_begin(h, TFRPN_K_NMS_SWEEP, st);
    nms_sweep_kernel<<<B, SWEEP_THREADS, 0, st>>>(p);
    prof_end(h, st);
    TFRPN_AFTER_LAUNCH("nms_sweep_kernel");
    return 0;
}
static void two_phase_shape(tfrpn_handle h, int B, int& cl, int& threads);
static int launch_matrix(tfrpn_handle h, PropParams& p, int B, cudaStream_t st) {
    char* ws = nullptr;
    if (int rc = ensure_workspace_prop(h, matrix_workspace_bytes(B), st, &ws)) return rc;
    int32_t* rank_idx = reinterpret_cast<int32_t*>(ws); ws += align256((size_t)B * BATCH * 4);
    int32_t* rank_n = reinterpret_cast<int32_t*>(ws); ws += align256((size_t)B * 4);
    int32_t* rank_more = reinterpret_cast<int32_t*>(ws); ws += align256((size_t)B * 4);
    int32_t* redo = reinterpret_cast<int32_t*>(ws); ws += align256((size_t)B * 4);
    unsigned int* mask = reinterpret_cast<unsigned int*>(ws);
    PropParams r = p;
    r.mode = MODE_RANK; r.rank_idx = rank_idx; r.rank_n = rank_n; r.rank_more = rank_more;
    int cl, threads;
    two_phase_shape(h, B, cl, threads);
    if (int rc = launch_cluster(h, r, B, cl, threads, st)) return rc;
    PropParams m = p;
    m.rank_idx = rank_idx; m.rank_n = rank_n; m.rank_more = rank_more; m.redo_flags = redo;
    if (int rc = launch_mask_sweep(h, m, B, matrix_rows_of(h), mask, st)) return rc;
    PropParams c2 = p;   // images that used up the matrix rows before max_out boxes were kept (rare)
    c2.flags = redo; c2.flag_mode = 2;
    return launch_one(h, c2, B, st);
}

static int launch(tfrpn_handle h, PropParams& p, int B, cudaStream_t st) {
    int k_eff = p.k;
    if (p.mode != MODE_TOPK && p.max_out <= PRE_NMS_CAP_MAX_OUT) k_eff = min(p.k, PRE_NMS_CAP);
    if (h && pre_applies(p.N, k_eff)) return launch_prefiltered(h, p, k_eff, B, st);
    if (matrix_applies(h, p)) return launch_matrix(h, p, B, st);
    return launch_one(h, p, B, st);
}

static int launch_cluster(tfrpn_handle h, PropParams& p, int B, int cl, int threads, cudaStream_t st) {
    p.mo_pad = (p.max_out + 3) & ~3;
    // (a presorted launch never looks at the scores' order: no staged keys)
    p.staged = (!p.presorted && cluster_smem_bytes(cl, p.N, p.max_out) <= PROP_SMEM_LIMIT) ? 1 : 0;
    const size_t smem = cluster_smem_bytes(cl, p.staged ? p.N : 0, p.max_out);
    if (int rc = check_prop_smem(smem, p.max_out)) return rc;
    prof_begin(h, TFRPN_K_PROPOSAL_CLUSTER, st);
    if (cl == 8 && threads == 512) proposal_cluster_kernel<8, 512><<<B * 8, 512, smem, st>>>(p);
    else if (cl == 8) proposal_cluster_kernel<8, 256><<<B * 8, 256, smem, st>>>(p);
    else if (cl == 4 && threads == 256) proposal_cluster_kernel<4, 256><<<B * 4, 256, smem, st>>>(p);
    else if (cl == 4) proposal_cluster_kernel<4, 512><<<B * 4, 512, smem, st>>>(p);
    else if (cl == 2 && threads == 512) proposal_cluster_kernel<2, 512><<<B * 2, 512, smem, st>>>(p);
    else if (cl == 2) proposal_cluster_kernel<2, 1024><<<B * 2, 1024, smem, st>>>(p);
    else proposal_cluster_kernel<1, 1024><<<B, 1024, smem, st>>>(p);
    prof_end(h, st);
    TFRPN_AFTER_LAUNCH("proposal_cluster_kernel");
    return 0;
}

// Device-side variant of the two-phase gather (pipeline.cu): the candidate rows of a PAGE-LOCKED host tensor, in rank
// order, into a compact device array.  Every row is an independent 16-byte read over PCIe (~0.55 G rows/s,
// tools/src/pcie_gather.cu): slower than the host-side gather + one bulk copy when host cores are free, but it
// costs no host time at all.  Lane pairs read the two halves of the row's 32-byte sector (one request per pair).
__global__ void __launch_bounds__(256) gather_rows_kernel(const float4* __restrict__ reg, const int* __restrict__ rank_idx,
                                                          const int* __restrict__ rank_n, int N, int rows, int cap,
                                                          float4* __restrict__ dst, int stride, unsigned long long* counter) {
    const int b = blockIdx.y;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int r = t >> 1, half = t & 1;
    const int n = min(rank_n[b], rows);
    const bool live = r < n;
    const int i = live ? rank_idx[(long long)b * cap + r] : 0;
    const bool pair_ok = ((i & ~1) + 1) < N || (i & 1);      // the sector's other half exists (the last row of an odd N may not)
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4* src = reg + (long long)b * N;
    if (live) v = pair_ok ? __ldg(src + (i & ~1) + half) : (half == 0 ? __ldg(src + i) : v);
    const float4 o = make_float4(__shfl_xor_sync(0xffffffffu, v.x, 1), __shfl_xor_sync(0xffffffffu, v.y, 1),
                                 __shfl_xor_sync(0xffffffffu, v.z, 1), __shfl_xor_sync(0xffffffffu, v.w, 1));
    if (live && half == 0) dst[(long long)b * stride + r] = (pair_ok && (i & 1)) ? o : v;
    if (counter && t == 0) atomicAdd(counter, (unsigned long long)n);
}

// Every launch of the one-CTA kernel comes through here: the proposal stage, tfrpn_topk / tfrpn_nms (the large-N
// prefilter's compact launch and its redo of flagged images included) and the per-class launch of
// tfrpn_nms_multiclass.  Threads per CTA: 512 whenever two such CTAs, each with this launch's dynamic shared memory,
// fit one SM -- an image then holds half an SM's threads and registers, and the two CTAs fill each other's barrier
// gaps -- else 1024 (large staged N, large max_out).  TFRPN_PROP_THREADS = 512 | 1024 forces one build (A/B switch).
static int launch_one(tfrpn_handle h, PropParams& p, int B, cudaStream_t st) {
    p.mo_pad = (p.max_out + 3) & ~3;
    int cl = 0, threads = 1024;
    pick_cluster(h, B, cl, threads);
    if (cl) return launch_cluster(h, p, B, cl, threads, st);
    p.staged = prop_smem_bytes(p.N, p.max_out) <= PROP_SMEM_LIMIT ? 1 : 0;
    const size_t smem = prop_smem_bytes(p.staged ? p.N : 0, p.max_out);
    if (int rc = check_prop_smem(smem, p.max_out)) return rc;
    threads = h->opts.prop_threads;
    if (threads != 512 && threads != 1024) {
        int per_sm = 0;
        TFRPN_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, proposal_kernel<512>, 512, smem));
        threads = per_sm >= 2 ? 512 : 1024;
    }
    prof_begin(h, TFRPN_K_PROPOSAL, st);
    if (threads == 512) proposal_kernel<512><<<B, 512, smem, st>>>(p);
    else proposal_kernel<1024><<<B, 1024, smem, st>>>(p);
    prof_end(h, st);
    TFRPN_AFTER_LAUNCH("proposal_kernel");
    return 0;
}

}  // namespace tfrpn

using namespace tfrpn;

extern "C" int tfrpn_topk(tfrpn_handle h, const float* scores, int B, int N, int k, float* values, int32_t* indices,
                          const float* boxes_or_null, int boxes_batched, float* gathered_or_null, tfrpn_stream s) {
    if (!scores || !values || !indices) return fail(TFRPN_ERR_BAD_ARG, "topk: null pointer");
    if (B < 0 || N < 0 || k < 0) return fail(TFRPN_ERR_BAD_ARG, "topk: negative shape");
    if (k > N) return fail(TFRPN_ERR_BAD_ARG, "topk: k=%d > N=%d (tf.nn.top_k raises InvalidArgumentError too)", k, N);
    if ((gathered_or_null != nullptr) != (boxes_or_null != nullptr))
        return fail(TFRPN_ERR_BAD_ARG, "topk: boxes and gathered must be given together");
    if (boxes_or_null && (!aligned16(boxes_or_null) || !aligned16(gathered_or_null)))
        return fail(TFRPN_ERR_MISALIGNED, "topk: boxes must be 16-byte aligned");
    if (B == 0 || k == 0) return 0;
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "topk: null handle");
    TFRPN_ENTER(h);
    TFRPN_CHECK_ON_DEVICE(h, scores, "topk: scores");
    PropParams p = {};
    p.mode = MODE_TOPK; p.N = N; p.k = k; p.scores = scores; p.use_sthr = 0;
    p.boxes = reinterpret_cast<const float4*>(boxes_or_null); p.box_stride = boxes_batched ? N : 0;
    p.values = values; p.indices = indices; p.gathered = reinterpret_cast<float4*>(gathered_or_null);
    p.max_out = 0; p.rows = 0;
    return launch(h, p, B, as_stream(s));
}

extern "C" int tfrpn_predict_topk(tfrpn_handle h, const float* rpn_reg, const float* rpn_cls, const float* anchors, int B,
                                  int N, int k, const float* variances_host, int clip, float* out_boxes,
                                  float* out_scores, int32_t* out_indices, tfrpn_stream s) {
    if (!rpn_reg || !rpn_cls || !anchors || !variances_host || !out_boxes || !out_scores || !out_indices)
        return fail(TFRPN_ERR_BAD_ARG, "predict_topk: null pointer");
    if (B < 0 || N < 0 || k < 0) return fail(TFRPN_ERR_BAD_ARG, "predict_topk: negative shape");
    if (k > N) return fail(TFRPN_ERR_BAD_ARG, "predict_topk: k=%d > N=%d (tf.nn.top_k raises InvalidArgumentError too)", k, N);
    if (!aligned16(rpn_reg) || !aligned16(anchors) || !aligned16(out_boxes))
        return fail(TFRPN_ERR_MISALIGNED, "predict_topk: rpn_reg / anchors / out_boxes must be 16-byte aligned");
    if (B == 0 || k == 0) return 0;
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "predict_topk: null handle");
    TFRPN_ENTER(h);
    TFRPN_CHECK_ON_DEVICE(h, rpn_reg, "predict_topk: rpn_reg");
    PropParams p = {};
    p.mode = MODE_TOPK; p.N = N; p.k = k; p.scores = rpn_cls; p.use_sthr = 0;
    p.reg = reinterpret_cast<const float4*>(rpn_reg); p.anchors = reinterpret_cast<const float4*>(anchors);
    p.var = make_float4(variances_host[0], variances_host[1], variances_host[2], variances_host[3]);
    p.clip_decoded = clip;
    p.values = out_scores; p.indices = out_indices; p.gathered = reinterpret_cast<float4*>(out_boxes);
    p.max_out = 0; p.rows = 0;
    return launch(h, p, B, as_stream(s));
}

extern "C" int tfrpn_nms(tfrpn_handle h, const float* boxes, const float* scores, int B, int K, const tfrpn_nms_cfg* cfg,
                         float* out_boxes, float* out_scores, float* out_classes, int32_t* valid,
                         int32_t* keep_idx_or_null, tfrpn_stream s) {
    if (!boxes || !scores || !cfg || !out_boxes || !out_scores || !valid) return fail(TFRPN_ERR_BAD_ARG, "nms: null pointer");
    if (B < 0 || K < 0) return fail(TFRPN_ERR_BAD_ARG, "nms: negative shape");
    if (cfg->max_output_size_per_class <= 0 || cfg->max_total_size <= 0)
        return fail(TFRPN_ERR_BAD_ARG, "nms: max_output_size_per_class and max_total_size must be > 0");
    if (int rc = check_iou_threshold("nms", cfg->iou_threshold)) return rc;
    if (!aligned16(boxes) || !aligned16(out_boxes)) return fail(TFRPN_ERR_MISALIGNED, "nms: boxes must be 16-byte aligned");
    if (B == 0) return 0;
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "nms: null handle");
    TFRPN_ENTER(h);
    TFRPN_CHECK_ON_DEVICE(h, boxes, "nms: boxes");
    PropParams p = {};
    if (cfg->pre_nms_topn < 0) return fail(TFRPN_ERR_BAD_ARG, "nms: pre_nms_topn must be >= 0");
    p.mode = MODE_NMS; p.N = K; p.k = cfg->pre_nms_topn > 0 ? min(K, cfg->pre_nms_topn) : K; p.scores = scores;
    p.use_sthr = !(cfg->score_threshold == -INFINITY);
    p.score_threshold = cfg->score_threshold;
    p.boxes = reinterpret_cast<const float4*>(boxes); p.box_stride = K;
    p.rows = cfg->pad_per_class ? min(cfg->max_total_size, cfg->max_output_size_per_class) : cfg->max_total_size;
    p.max_out = min(cfg->max_output_size_per_class, p.rows);
    p.iou_thr = make_threshold(cfg->iou_threshold); p.clip_out = cfg->clip_boxes;
    p.out_boxes = reinterpret_cast<float4*>(out_boxes); p.out_scores = out_scores; p.out_classes = out_classes;
    p.valid = valid; p.keep_idx = keep_idx_or_null;
    return launch(h, p, B, as_stream(s));
}

namespace tfrpn {
static void fill_proposal_params(PropParams& p, const float* rpn_reg, const float* rpn_cls, const float* anchors, int N,
                                 const tfrpn_proposal_cfg* cfg, float* out_boxes, float* out_scores, int32_t* valid,
                                 int32_t* keep_idx_or_null) {
    p.mode = MODE_PROPOSALS; p.N = N; p.k = min(cfg->pre_nms_topn, N); p.scores = rpn_cls; p.use_sthr = 0;
    p.reg = reinterpret_cast<const float4*>(rpn_reg); p.anchors = reinterpret_cast<const float4*>(anchors);
    p.var = make_float4(cfg->variances[0], cfg->variances[1], cfg->variances[2], cfg->variances[3]);
    p.clip_decoded = cfg->clip;
    p.rows = cfg->post_nms_topn; p.max_out = cfg->post_nms_topn;
    p.iou_thr = make_threshold(cfg->nms_iou_threshold); p.clip_out = 1;  // combined NMS default clip_boxes=True
    p.out_boxes = reinterpret_cast<float4*>(out_boxes); p.out_scores = out_scores; p.out_classes = nullptr;
    p.valid = valid; p.keep_idx = keep_idx_or_null;
}

// ---- two-phase flow of the host pipeline (pipeline.cu) ------------------------------------------------------
// A host step's rpn_reg tensor is 80 % of its H2D bytes, and NMS decodes only the rows of the candidates it
// examines (~550 of 8649 per image at C2).  So: (1) rank launch over the scores alone -> the entry index of the
// first batch of ranks (<= 1024 per image, sorted); (2) the host gathers those rows of rpn_reg into a compact
// array and copies it; (3) presorted launch = the NMS rounds of that batch, rows read by rank.  An image whose
// NMS needs more than that batch raises redo_flags[b] and is redone by the unfiltered kernel (proposals_redo).
constexpr int RANK_CAP = BATCH;
int proposals_rank_cap() { return RANK_CAP; }
bool proposals_two_phase_applies(int B, int N, const tfrpn_proposal_cfg* cfg) {
    const int k = min(cfg->pre_nms_topn, N);
    int k_eff = k;
    if (cfg->post_nms_topn <= PRE_NMS_CAP_MAX_OUT) k_eff = min(k, PRE_NMS_CAP);
    if (pre_applies(N, k_eff)) return false;                           // large N: the prefilter path
    return B > 0 && cluster_smem_bytes(2, 0, cfg->post_nms_topn) <= PROP_SMEM_LIMIT;
}
static void two_phase_shape(tfrpn_handle h, int B, int& cl, int& threads) {
    pick_cluster(h, B, cl, threads);
    if (cl == 0) { cl = 2; threads = 512; }                            // the one-CTA kernel has no rank / presorted modes
}
int proposals_rank_enqueue(tfrpn_handle h, const float* rpn_cls, int B, int N, const tfrpn_proposal_cfg* cfg,
                           int32_t* rank_idx, int32_t* rank_n, int32_t* rank_more, cudaStream_t st) {
    PropParams p = {};
    fill_proposal_params(p, nullptr, rpn_cls, nullptr, N, cfg, nullptr, nullptr, nullptr, nullptr);
    p.mode = MODE_RANK;
    p.rank_idx = rank_idx; p.rank_n = rank_n; p.rank_more = rank_more;
    int cl, threads;
    two_phase_shape(h, B, cl, threads);
    return launch_cluster(h, p, B, cl, threads, st);
}
// reg_compact: (B, compact_stride, 4) rows of rpn_reg in rank order, the first compact_rows of every image valid;
// ranks beyond them end the batch (and raise the image's redo flag if max_out boxes were not kept by then).
// reg_compact null: rows are read from rpn_reg_or_null by entry index (device-resident two-phase run, tests).
int proposals_presorted_enqueue(tfrpn_handle h, const float* rpn_reg_or_null, const float* reg_compact, int compact_rows,
                                int compact_stride, const float* rpn_cls, const float* anchors, int B, int N,
                                const tfrpn_proposal_cfg* cfg, int32_t* rank_idx, int32_t* rank_n, int32_t* rank_more,
                                float* out_boxes, float* out_scores, int32_t* valid, int32_t* keep_idx_or_null,
                                int32_t* redo_flags, unsigned int* mask_ws_or_null, cudaStream_t st) {
    PropParams p = {};
    fill_proposal_params(p, rpn_reg_or_null, rpn_cls, anchors, N, cfg, out_boxes, out_scores, valid, keep_idx_or_null);
    p.rank_idx = rank_idx; p.rank_n = rank_n; p.rank_more = rank_more;
    p.reg_compact = reinterpret_cast<const float4*>(reg_compact); p.compact_rows = reg_compact ? compact_rows : 0;
    p.compact_stride = compact_stride;
    p.redo_flags = redo_flags;
    if (mask_ws_or_null && !h->opts.nms_lazy) {   // matrix NMS over the gathered rows (the caller owns the mask buffer)
        int rows = (min(compact_rows, BATCH) + 31) & ~31;
        return launch_mask_sweep(h, p, B, rows, mask_ws_or_null, st);
    }
    p.presorted = 1;                              // the lazy cluster kernel's rounds over the same ranks
    int cl, threads;
    two_phase_shape(h, B, cl, threads);
    return launch_cluster(h, p, B, cl, threads, st);
}
size_t proposals_mask_bytes(int B, int rows) { rows = (min(rows, BATCH) + 31) & ~31; return (size_t)B * rows * (rows / 32) * 4; }
int proposals_gather_enqueue(const float* reg_pinned_dev, const int32_t* rank_idx, const int32_t* rank_n, int B, int N,
                             int rows, float* dst, int stride, unsigned long long* counter_or_null, cudaStream_t st) {
    const dim3 grid((2 * rows + 255) / 256, B);
    gather_rows_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const float4*>(reg_pinned_dev), rank_idx, rank_n, N, rows, RANK_CAP,
                                             reinterpret_cast<float4*>(dst), stride, counter_or_null);
    TFRPN_AFTER_LAUNCH("gather_rows_kernel");
    return 0;
}
// the unfiltered kernel for the images whose redo flag is set (it returns at once for the others)
int proposals_redo_enqueue(tfrpn_handle h, const float* rpn_reg, const float* rpn_cls, const float* anchors, int B, int N,
                           const tfrpn_proposal_cfg* cfg, float* out_boxes, float* out_scores, int32_t* valid,
                           int32_t* keep_idx_or_null, const int32_t* redo_flags, unsigned long long* rows_fetched_or_null,
                           cudaStream_t st) {
    PropParams p = {};
    fill_proposal_params(p, rpn_reg, rpn_cls, anchors, N, cfg, out_boxes, out_scores, valid, keep_idx_or_null);
    p.rows_fetched = rows_fetched_or_null;
    p.flags = redo_flags; p.flag_mode = 2;
    return launch_one(h, p, B, st);
}

// The fused stage after argument checks.  `rpn_reg` may also be PAGE-LOCKED HOST memory (pipeline.cu): the kernels
// touch only the rows of the candidates they examine (<= ~1000 of the N rows per image), so those rows are
// pulled over PCIe by the loads themselves instead of copying the whole tensor to the device first.
int proposals_enqueue(tfrpn_handle h, const float* rpn_reg, const float* rpn_cls, const float* anchors, int B, int N,
                      const tfrpn_proposal_cfg* cfg, float* out_boxes, float* out_scores, int32_t* valid,
                      int32_t* keep_idx_or_null, unsigned long long* rows_fetched_or_null, cudaStream_t st) {
    PropParams p = {};
    fill_proposal_params(p, rpn_reg, rpn_cls, anchors, N, cfg, out_boxes, out_scores, valid, keep_idx_or_null);
    p.rows_fetched = rows_fetched_or_null;
    return launch(h, p, B, st);
}
}  // namespace tfrpn

extern "C" int tfrpn_proposals(tfrpn_handle h, const float* rpn_reg, const float* rpn_cls, const float* anchors, int B,
                               int N, const tfrpn_proposal_cfg* cfg, float* out_boxes, float* out_scores,
                               int32_t* valid, int32_t* keep_idx_or_null, tfrpn_stream s) {
    if (!rpn_reg || !rpn_cls || !anchors || !cfg || !out_boxes || !out_scores || !valid)
        return fail(TFRPN_ERR_BAD_ARG, "proposals: null pointer");
    if (B < 0 || N < 0) return fail(TFRPN_ERR_BAD_ARG, "proposals: negative shape");
    if (cfg->pre_nms_topn <= 0 || cfg->post_nms_topn <= 0) return fail(TFRPN_ERR_BAD_ARG, "proposals: topn must be > 0");
    if (int rc = check_iou_threshold("proposals", cfg->nms_iou_threshold)) return rc;
    if (!aligned16(rpn_reg) || !aligned16(anchors) || !aligned16(out_boxes))
        return fail(TFRPN_ERR_MISALIGNED, "proposals: rpn_reg / anchors / out_boxes must be 16-byte aligned");
    if (B == 0) return 0;
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "proposals: null handle");
    TFRPN_ENTER(h);
    TFRPN_CHECK_ON_DEVICE(h, rpn_reg, "proposals: rpn_reg");
    return proposals_enqueue(h, rpn_reg, rpn_cls, anchors, B, N, cfg, out_boxes, out_scores, valid, keep_idx_or_null,
                             nullptr, as_stream(s));
}

// The same stage with the anchors regenerated in registers from the hyper-parameters (north star: fused
// anchor-generate + decode + clip): no (N,4) anchor tensor is read.  N = fm_h * fm_w * n_scales * n_ratios.
extern "C" int tfrpn_proposals_anchor_cfg(tfrpn_handle h, const float* rpn_reg, const float* rpn_cls,
                                          const tfrpn_anchor_cfg* acfg, int B, const tfrpn_proposal_cfg* cfg, float* out_boxes,
                                          float* out_scores, int32_t* valid, int32_t* keep_idx_or_null, tfrpn_stream s) {
    if (!rpn_reg || !rpn_cls || !acfg || !cfg || !out_boxes || !out_scores || !valid)
        return fail(TFRPN_ERR_BAD_ARG, "proposals_anchor_cfg: null pointer");
    if (B < 0) return fail(TFRPN_ERR_BAD_ARG, "proposals_anchor_cfg: negative shape");
    if (cfg->pre_nms_topn <= 0 || cfg->post_nms_topn <= 0) return fail(TFRPN_ERR_BAD_ARG, "proposals_anchor_cfg: topn must be > 0");
    if (int rc = check_iou_threshold("proposals_anchor_cfg", cfg->nms_iou_threshold)) return rc;
    if (!aligned16(rpn_reg) || !aligned16(out_boxes))
        return fail(TFRPN_ERR_MISALIGNED, "proposals_anchor_cfg: rpn_reg / out_boxes must be 16-byte aligned");
    AnchorGen gen;
    long long N = 0;
    if (int rc = make_anchor_gen(acfg, &gen, &N)) return rc;
    if (B == 0) return 0;
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "proposals_anchor_cfg: null handle");
    TFRPN_ENTER(h);
    TFRPN_CHECK_ON_DEVICE(h, rpn_reg, "proposals_anchor_cfg: rpn_reg");
    cudaStream_t st = as_stream(s);
    if (!h->anchor_gen) TFRPN_CHECK_CUDA(cudaMalloc(&h->anchor_gen, sizeof(AnchorGen)));
    if (memcmp(&h->anchor_gen_cfg, acfg, sizeof(*acfg)) != 0) {
        // the generator lives in device memory of the handle; uploaded again only when the configuration changes
        // (a copy from pageable memory returns once the source has been staged, so `gen` may go out of scope)
        TFRPN_CHECK_CUDA(cudaMemcpyAsync(h->anchor_gen, &gen, sizeof(gen), cudaMemcpyHostToDevice, st));
        TFRPN_CHECK_CUDA(cudaStreamSynchronize(st));
        h->anchor_gen_cfg = *acfg;
    }
    PropParams p = {};
    fill_proposal_params(p, rpn_reg, rpn_cls, nullptr, (int)N, cfg, out_boxes, out_scores, valid, keep_idx_or_null);
    p.gen = static_cast<const AnchorGen*>(h->anchor_gen);
    int k_eff = p.k;
    if (p.max_out <= PRE_NMS_CAP_MAX_OUT) k_eff = min(p.k, PRE_NMS_CAP);
    if (pre_applies(p.N, k_eff))   // the large-N prefilter gathers anchors from a tensor: materialise them for it
        return fail(TFRPN_ERR_UNSUPPORTED, "proposals_anchor_cfg: N = %lld takes the prefilter path, which reads an anchor tensor; "
                                           "call tfrpn_anchors + tfrpn_proposals", N);
    return launch_one(h, p, B, st);
}

// ---- multi-class combined NMS (kernels: see nms_mc_stage_kernel) -------------------------------------------------
namespace tfrpn {
struct McLayout {
    int rows, lmax;
    int G;               // merge CTAs per image
    int row_layout, slices, slice_rows;   // staging: row layout (count + scatter) and its slices, or the column layout
    long long scratch;   // merge scratch per CTA: C * 16 + C * lmax * 4 bytes, rounded up to 16
    size_t cand_scores, remap, cand_boxes, counts, ks, ki, kb, kv, gscratch, row_cnt, total;   // byte offsets, total size
};
// Staging layout: TFRPN_NMS_MC_STAGE=column|rows forces one (A/B switch).  Otherwise the column layout once its B*C
// CTAs fill the 148 SMs, the row layout below that (measured, DESIGN.md section 4: column 62 against 95 us at SSD-VOC,
// B*C = 640; rows 60 against 150 us at 4 x 100000 x 4, B*C = 16).  The row layout needs C <= MC_ROW_MAX_C.
static bool mc_rows_apply(int mode, int B, int K, int C) {
    if (C > MC_ROW_MAX_C || (long long)K * C > 0x7FFFFFFFLL || mode == 1) return false;
    return mode == 2 || (long long)B * C < 148;
}
// row_classes: the classes of the output-row rule (C; C - 1 for the box-head detections, whose class 0 never has a
// candidate).  The sizes do not depend on it: lmax = min(P, total) for any row_classes >= 1.
static void mc_layout(int B, int K, int C, const tfrpn_nms_cfg* cfg, McLayout* L, int stage_mode = 0, int row_classes = 0) {
    const int P = cfg->max_output_size_per_class;
    const long long rc = row_classes > 0 ? row_classes : C;
    L->rows = cfg->pad_per_class ? (int)std::min((long long)cfg->max_total_size, (long long)P * rc) : cfg->max_total_size;
    L->lmax = min(P, L->rows);
    L->scratch = ((long long)C * 16 + (long long)C * L->lmax * 4 + 15) & ~15LL;
    // ~2 CTAs per SM over the batch, no more than there are slices of MC_MERGE_THREADS entries
    const long long slices = ((long long)C * L->lmax + MC_MERGE_THREADS - 1) / MC_MERGE_THREADS;
    L->G = (int)std::max(1LL, std::min({slices, (long long)(296 + B - 1) / B, 64LL}));
    const size_t S = (size_t)B * C;
    size_t o = 0;
    L->cand_scores = o; o += align256(S * K * 4);
    L->remap = o;       o += align256(S * K * 4);
    L->cand_boxes = o;  o += align256(S * K * 16);
    L->counts = o;      o += align256(S * 4);
    L->ks = o;          o += align256(S * P * 4);
    L->ki = o;          o += align256(S * P * 4);
    L->kb = o;          o += align256(S * P * 16);
    L->kv = o;          o += align256(S * 4);
    L->gscratch = o;    o += align256((size_t)B * L->G * L->scratch);
    // row layout: ~4 CTAs per SM over the batch, at least 256 rows per slice
    L->row_layout = mc_rows_apply(stage_mode, B, K, C) ? 1 : 0;
    L->slices = std::max(1, std::min((592 + B - 1) / B, (K + 255) / 256));
    L->slice_rows = (K + L->slices - 1) / L->slices;
    L->row_cnt = o;     o += align256((size_t)B * L->slices * MC_ROW_WARPS * C * 4);   // (counted in every mode)
    L->total = o + 256;
}
int mc_check_sizes(const char* fn, int B, int K, int C, const tfrpn_nms_cfg* cfg) {
    if (!cfg) return fail(TFRPN_ERR_BAD_ARG, "%s: null cfg", fn);
    if (B <= 0 || K <= 0 || C < 1) return fail(TFRPN_ERR_BAD_ARG, "%s: B=%d, K=%d, C=%d must be > 0", fn, B, K, C);
    if ((long long)B * C > 0x7FFFFFFFLL) return fail(TFRPN_ERR_BAD_ARG, "%s: B * C = %lld segments", fn, (long long)B * C);
    if (cfg->max_output_size_per_class <= 0 || cfg->max_total_size <= 0)
        return fail(TFRPN_ERR_BAD_ARG, "%s: max_output_size_per_class and max_total_size must be > 0", fn);
    if (cfg->pre_nms_topn < 0) return fail(TFRPN_ERR_BAD_ARG, "%s: pre_nms_topn must be >= 0", fn);
    return check_iou_threshold(fn, cfg->iou_threshold);
}
}  // namespace tfrpn

extern "C" size_t tfrpn_nms_multiclass_workspace_bytes(int B, int K, int C, const tfrpn_nms_cfg* cfg) {
    if (!cfg || B <= 0 || K <= 0 || C < 1 || cfg->max_output_size_per_class <= 0 || cfg->max_total_size <= 0) return 0;
    McLayout L;
    mc_layout(B, K, C, cfg, &L);
    return L.total;
}

extern "C" int tfrpn_reserve_nms_multiclass(tfrpn_handle h, int B, int K, int C, const tfrpn_nms_cfg* cfg) {
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "reserve_nms_multiclass: null handle");
    if (int rc = mc_check_sizes("reserve_nms_multiclass", B, K, C, cfg)) return rc;
    TFRPN_ENTER(h);
    char* ws;
    return ensure_workspace_prop(h, tfrpn_nms_multiclass_workspace_bytes(B, K, C, cfg), nullptr, &ws);
}

namespace tfrpn {
// the per-class kernel's shared-memory carve bounds max_output_size_per_class, as in tfrpn_nms
int nms_mc_check_smem(tfrpn_handle h, int B, int C, int P) {
    int cl = 0, threads = 1024;
    pick_cluster(h, B * C, cl, threads);
    return check_prop_smem(cl ? cluster_smem_bytes(cl, 0, P) : prop_smem_bytes(0, P), P);
}

// The body of tfrpn_nms_multiclass after its argument checks, shared with tfrpn_roi_head_detections (roi_detect.cu).
// Candidates are the entries with score > sthr (use_sthr) or all of them; output rows follow the rule with
// row_classes classes.  The layout starts ws_offset bytes into the proposal-side workspace: the bytes before it are
// the caller's (the detections' staged scores and boxes, written before this call).
int nms_mc_run(tfrpn_handle h, const float* boxes, int q, const float* scores, int B, int K, int C,
               const tfrpn_nms_cfg* cfg, int row_classes, int use_sthr, float sthr, size_t ws_offset, float* out_boxes,
               float* out_scores, float* out_classes, int32_t* valid, int32_t* keep_idx_or_null, cudaStream_t st) {
    const int S = B * C, P = cfg->max_output_size_per_class;
    if (int rc = nms_mc_check_smem(h, B, C, P)) return rc;
    McLayout L;
    mc_layout(B, K, C, cfg, &L, h->opts.nms_mc_stage, row_classes);
    char* ws = nullptr;
    if (int rc = ensure_workspace_prop(h, ws_offset + L.total, st, &ws)) return rc;
    ws += ws_offset;

    McStageParams g = {};
    g.scores = scores; g.boxes = reinterpret_cast<const float4*>(boxes); g.K = K; g.C = C; g.q = q;
    g.use_sthr = use_sthr; g.sthr = sthr;
    g.cand_scores = reinterpret_cast<float*>(ws + L.cand_scores); g.remap = reinterpret_cast<int*>(ws + L.remap);
    g.cand_boxes = reinterpret_cast<float4*>(ws + L.cand_boxes); g.counts = reinterpret_cast<int*>(ws + L.counts);
    prof_begin(h, TFRPN_K_NMS_MC_STAGE, st);
    if (L.row_layout) {
        McRowParams r = {};
        r.g = g; r.slices = L.slices; r.slice_rows = L.slice_rows; r.row_cnt = reinterpret_cast<int*>(ws + L.row_cnt);
        const size_t smem = (size_t)MC_ROW_WARPS * C * 4;
        nms_mc_row_count_kernel<<<dim3(L.slices, B), MC_ROW_THREADS, smem, st>>>(r);
        TFRPN_AFTER_LAUNCH("nms_mc_row_count_kernel");
        nms_mc_row_scatter_kernel<<<dim3(L.slices, B), MC_ROW_THREADS, smem, st>>>(r);
    } else {
        nms_mc_stage_kernel<<<S, MC_STAGE_THREADS, 0, st>>>(g);
    }
    prof_end(h, st);
    TFRPN_AFTER_LAUNCH("nms_mc_stage_kernel");

    PropParams p = {};
    p.mode = MODE_NMS; p.N = K; p.k = cfg->pre_nms_topn > 0 ? min(K, cfg->pre_nms_topn) : K;
    p.scores = g.cand_scores; p.counts = g.counts; p.remap = g.remap;
    p.use_sthr = g.use_sthr; p.score_threshold = g.sthr;
    p.boxes = g.cand_boxes; p.box_stride = K;
    p.rows = P; p.max_out = P;
    p.iou_thr = make_threshold(cfg->iou_threshold); p.clip_out = cfg->clip_boxes;
    p.out_boxes = reinterpret_cast<float4*>(ws + L.kb); p.out_scores = reinterpret_cast<float*>(ws + L.ks);
    p.out_classes = nullptr; p.valid = reinterpret_cast<int*>(ws + L.kv); p.keep_idx = reinterpret_cast<int*>(ws + L.ki);
    if (int rc = launch_one(h, p, S, st)) return rc;

    McMergeParams m = {};
    m.ks = p.out_scores; m.kb = p.out_boxes; m.ki = p.keep_idx; m.kv = p.valid;
    m.C = C; m.P = P; m.rows = L.rows; m.lmax = L.lmax;
    m.use_smem = (size_t)L.scratch <= PROP_SMEM_LIMIT ? 1 : 0;
    m.gscratch = ws + L.gscratch; m.scratch_bytes = L.scratch;
    m.out_boxes = reinterpret_cast<float4*>(out_boxes); m.out_scores = out_scores; m.out_classes = out_classes;
    m.valid = valid; m.keep_idx = keep_idx_or_null;
    prof_begin(h, TFRPN_K_NMS_MC_MERGE, st);
    nms_mc_merge_kernel<<<dim3(B, L.G), MC_MERGE_THREADS, m.use_smem ? (size_t)L.scratch : 0, st>>>(m);
    prof_end(h, st);
    TFRPN_AFTER_LAUNCH("nms_mc_merge_kernel");
    return 0;
}
}  // namespace tfrpn

extern "C" int tfrpn_nms_multiclass(tfrpn_handle h, const float* boxes, int q, const float* scores, int B, int K, int C,
                                    const tfrpn_nms_cfg* cfg, float* out_boxes, float* out_scores, float* out_classes,
                                    int32_t* valid, int32_t* keep_idx_or_null, tfrpn_stream s) {
    if (!boxes || !scores || !cfg || !out_boxes || !out_scores || !out_classes || !valid)
        return fail(TFRPN_ERR_BAD_ARG, "nms_multiclass: null pointer");
    if (int rc = mc_check_sizes("nms_multiclass", B, K, C, cfg)) return rc;
    if (q != 1 && q != C) return fail(TFRPN_ERR_BAD_ARG, "nms_multiclass: q = %d must be 1 or C = %d", q, C);
    if (!aligned16(boxes) || !aligned16(out_boxes))
        return fail(TFRPN_ERR_MISALIGNED, "nms_multiclass: boxes must be 16-byte aligned");
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "nms_multiclass: null handle");
    TFRPN_ENTER(h);
    TFRPN_CHECK_ON_DEVICE(h, boxes, "nms_multiclass: boxes");
    return nms_mc_run(h, boxes, q, scores, B, K, C, cfg, C, !(cfg->score_threshold == -INFINITY), cfg->score_threshold, 0,
                      out_boxes, out_scores, out_classes, valid, keep_idx_or_null, as_stream(s));
}

#ifdef TFRPN_PHASE_TIMING
extern "C" __attribute__((visibility("default"))) int tfrpn_debug_phase_cycles(long long* out32) {
    return cudaMemcpyFromSymbol(out32, tfrpn::g_phase, sizeof(long long) * 32) == cudaSuccess ? 0 : -3;
}
extern "C" __attribute__((visibility("default"))) int tfrpn_debug_cta_times(long long* out4096) {
    return cudaMemcpyFromSymbol(out4096, tfrpn::g_img, sizeof(long long) * 4096) == cudaSuccess ? 0 : -3;
}
#endif
