// evaluate.cu -- proposal recall against ground truth (the quality measure of an RPN; the reference has none):
// for every limit k and IoU threshold t, the number of valid GT boxes that the first k proposals of their image
// cover at IoU >= t, and the number of valid GT boxes.  AR@k is the mean over t of hits / n_gt (host side).
//
//   recall_kernel  grid (L, B) x 512 threads, one CTA per (limit, image).  The image's GT boxes and its first k_eff =
//                  min(k, valid[b], P) proposals (with their areas) are staged in dynamic shared memory.
//     round 0      warp w takes the valid GT rows w, w+16, ...: the row's best pair over the k_eff ranks as a key
//                  (IoU bits | 0xFFFF - g | 0xFFFF - p).  Scores are clamped to >= +0, so the IoU bits order like the
//                  values; a key of 0 means "out of the competition" (invalid, assigned, or no positive pair left).
//                  Coverage matching stops here.
//     greedy       one round per match: a block max over the keys picks the pair with the largest IoU, then the
//                  lowest GT, then the lowest rank -- the global maximum of the remaining pairs, because every key
//                  is its row's maximum.  The GT is assigned, the rank is marked used, and only the GT rows whose
//                  key pointed at that rank are recomputed over the unused ranks (one warp per row).  A row whose
//                  best is +0 can never match again and leaves; the loop ends when no key is left.
//     counting     ballots per warp, shared-memory sums, then one 64-bit atomicAdd per counter and CTA.
//                  n_gt is added by the l = 0 CTAs only.  Every value is an integer or an exact float compare, so
//                  the counts do not depend on the order in which the CTAs run.
// The IoU is utils/bbox_utils.py:141-150 with the proposal as `bboxes`: iou_nice (range-check-free division, the same
// bits as __fdiv_rn) when every valid GT box of the CTA is a nice box and every staged proposal is nice or degenerate
// (per-CTA vote), iou_ref otherwise.  No workspace and no host synchronisation: the call can be graph-captured.
#include "common.cuh"

namespace tfrpn {

constexpr int RC_THREADS = 512;
constexpr int RC_WARPS = RC_THREADS / 32;
constexpr int RC_MAX_G = 1024;
constexpr int RC_MAX_K = 8192;

struct RecallParams {
    const float4* prop;    // (B,P,4)
    const int32_t* valid;  // (B,) or null
    const float4* gt;      // (B,G,4)
    const int32_t* labels; // (B,G) or null
    float* gt_iou;         // (L,B,G) or null
    unsigned long long* counts;   // (L*T + 1)
    int B, P, G, L, T, kcap, coverage;
    float thr[16];
    int lim[8];
};

// dynamic shared memory of a launch whose CTAs stage at most kcap proposals
static size_t recall_smem_bytes(int kcap, int G) {
    return (size_t)(kcap + G) * 16 + (size_t)(kcap + 2 * G) * 4 + (size_t)G * 8 + 4 * (size_t)(kcap / 32 + 1) + 8;
}

__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long w = __shfl_xor_sync(0xffffffffu, v, o);
        v = w > v ? w : v;
    }
    return v;
}

// The best remaining pair of GT box g (box gb, area ga) over the ranks [0, k) that are not used and not `skip`, as
// (IoU bits << 32) | (0xFFFF - rank), lowest rank on ties; 0 when no pair has a positive IoU.  Called by a whole warp.
template <bool NICE, bool SKIP>
__device__ __forceinline__ unsigned long long row_best(float4 gb, float ga, const float4* sp, const float* spa, int k,
                                                       const uint32_t* used, int skip) {
    uint32_t bs = 0u;   // bits of the best score of this lane (+0 never counts)
    int bp = 0;
    for (int p = lane_id(); p < k; p += 32) {   // a lane's ranks ascend: '>' keeps its lowest rank of a tie
        if (SKIP && (p == skip || ((used[p >> 5] >> (p & 31)) & 1u))) continue;
        float v = NICE ? iou_nice(gb, ga, sp[p], spa[p]) : iou_ref(sp[p], spa[p], gb, ga);
        v = v > 0.0f ? v : 0.0f;   // NaN, negative and -0 score +0
        const uint32_t u = __float_as_uint(v);
        if (u > bs) { bs = u; bp = p; }
    }
    const uint32_t m = __reduce_max_sync(0xffffffffu, bs);
    if (m == 0u) return 0ull;
    const uint32_t pmin = __reduce_min_sync(0xffffffffu, bs == m ? (uint32_t)bp : 0xFFFFFFFFu);
    return ((unsigned long long)m << 32) | (0xFFFFu - pmin);
}

__device__ __forceinline__ unsigned long long gt_key(unsigned long long row, int g) {
    return row ? row | ((unsigned long long)(0xFFFFu - (uint32_t)g) << 16) : 0ull;
}

template <bool NICE>
__device__ __forceinline__ void greedy_rounds(const float4* sp, const float* spa, int k, const float4* sg, const float* sga,
                                              float* siou, unsigned long long* key, uint32_t* used, int G,
                                              unsigned long long* s_red) {
    const int lane = lane_id(), warp = warp_id();
    for (;;) {
        unsigned long long m = 0ull;
        for (int g = threadIdx.x; g < G; g += RC_THREADS) m = key[g] > m ? key[g] : m;
        m = warp_max_u64(m);
        if (lane == 0) s_red[warp] = m;
        __syncthreads();
        m = s_red[0];
#pragma unroll
        for (int w = 1; w < RC_WARPS; ++w) m = s_red[w] > m ? s_red[w] : m;
        if (m == 0ull) break;
        const int gs = 0xFFFF - (int)((m >> 16) & 0xFFFFu);
        const uint32_t rank_field = (uint32_t)(m & 0xFFFFu);
        const int ps = 0xFFFF - (int)rank_field;
        // the winner is assigned by the lane that owns it; the rows whose best was rank ps look again.  Each key is
        // read and written only by its owner warp here, and read by everyone only after the next barrier.  GT g
        // belongs to warp g % 16, so neighbouring GT (which tend to share their best proposal) spread over the warps.
        for (int base = warp; base < G; base += RC_THREADS) {
            const int g = base + lane * RC_WARPS;
            bool again = false;
            if (g == gs) {
                siou[g] = __uint_as_float((uint32_t)(m >> 32));
                key[g] = 0ull;
            } else if (g < G) {
                const unsigned long long kg = key[g];
                again = kg != 0ull && (uint32_t)(kg & 0xFFFFu) == rank_field;
            }
            unsigned bal = __ballot_sync(0xffffffffu, again);
            while (bal) {
                const int j = __ffs(bal) - 1;
                bal &= bal - 1u;
                const int gg = base + j * RC_WARPS;
                const unsigned long long r = row_best<NICE, true>(sg[gg], sga[gg], sp, spa, k, used, ps);
                if (lane == j) key[gg] = gt_key(r, gg);
            }
        }
        __syncthreads();   // keys final, s_red read by every thread
        if (threadIdx.x == 0) used[ps >> 5] |= 1u << (ps & 31);   // read by the next round after its first barrier
    }
}

__global__ void __launch_bounds__(RC_THREADS) recall_kernel(RecallParams q) {
    extern __shared__ float4 rc_smem[];
    __shared__ unsigned long long s_red[RC_WARPS];
    __shared__ int s_cnt[17];
    const int l = blockIdx.x, b = blockIdx.y, G = q.G, kcap = q.kcap;
    float4* sp = rc_smem;                                              // [kcap] proposals
    float4* sg = sp + kcap;                                            // [G]    GT boxes
    unsigned long long* key = reinterpret_cast<unsigned long long*>(sg + G);   // [G]
    float* spa = reinterpret_cast<float*>(key + G);                    // [kcap] proposal areas
    float* sga = spa + kcap;                                           // [G]    GT areas
    float* siou = sga + G;                                             // [G]    matched IoU; -1 = invalid GT
    uint32_t* used = reinterpret_cast<uint32_t*>(siou + G);            // [kcap/32 + 1] ranks taken by a match

    const int nv = q.valid ? min(max(q.valid[b], 0), q.P) : q.P;
    const int k = min(min(q.lim[l], nv), q.P);
    bool ok = true;
    const float4* pb = q.prop + (long long)b * q.P;
    for (int p = threadIdx.x; p < k; p += RC_THREADS) {
        const float4 v = ldg_f4(pb + p);
        sp[p] = v;
        spa[p] = box_area(v);
        ok = ok && nice_coords(v) && v.z >= v.x && v.w >= v.y;
    }
    for (int w = threadIdx.x; w <= kcap / 32; w += RC_THREADS) used[w] = 0u;
    const float4* gb = q.gt + (long long)b * G;
    for (int g = threadIdx.x; g < G; g += RC_THREADS) {
        const float4 v = ldg_f4(gb + g);
        const float a = box_area(v);
        const bool valid = a > 0.0f && (!q.labels || q.labels[(long long)b * G + g] >= 0);
        sg[g] = v;
        sga[g] = a;
        siou[g] = valid ? 0.0f : -1.0f;
        ok = ok && (!valid || nice_box(v));
    }
    if (threadIdx.x < 17) s_cnt[threadIdx.x] = 0;
    const bool nice = __syncthreads_and(ok) != 0;

    // round 0: every valid GT row's best pair
    const int warp = warp_id(), lane = lane_id();
    for (int g = warp; g < G; g += RC_WARPS) {
        unsigned long long r = 0ull;
        if (siou[g] == 0.0f)
            r = nice ? row_best<true, false>(sg[g], sga[g], sp, spa, k, used, -1)
                     : row_best<false, false>(sg[g], sga[g], sp, spa, k, used, -1);
        if (lane == 0) key[g] = gt_key(r, g);
    }
    __syncthreads();
    if (q.coverage) {
        for (int g = threadIdx.x; g < G; g += RC_THREADS)
            if (key[g]) siou[g] = __uint_as_float((uint32_t)(key[g] >> 32));
    } else if (nice) {
        greedy_rounds<true>(sp, spa, k, sg, sga, siou, key, used, G, s_red);
    } else {
        greedy_rounds<false>(sp, spa, k, sg, sga, siou, key, used, G, s_red);
    }
    __syncthreads();

    // counting (and the matched IoUs)
    float* out = q.gt_iou ? q.gt_iou + ((long long)l * q.B + b) * G : nullptr;
    for (int base = warp * 32; base < G; base += RC_THREADS) {
        const int g = base + lane;
        const float v = g < G ? siou[g] : -1.0f;
        if (out && g < G) out[g] = v;
        const unsigned nval = __popc(__ballot_sync(0xffffffffu, v >= 0.0f));
        for (int t = 0; t < q.T; ++t) {
            const unsigned h = __popc(__ballot_sync(0xffffffffu, v >= q.thr[t]));
            if (lane == 0 && h) atomicAdd(&s_cnt[t], (int)h);
        }
        if (lane == 0 && nval) atomicAdd(&s_cnt[16], (int)nval);
    }
    __syncthreads();
    if (threadIdx.x < q.T) {
        const int c = s_cnt[threadIdx.x];
        if (c) atomicAdd(q.counts + (long long)l * q.T + threadIdx.x, (unsigned long long)c);
    } else if (threadIdx.x == 16 && l == 0) {
        const int c = s_cnt[16];
        if (c) atomicAdd(q.counts + (long long)q.L * q.T, (unsigned long long)c);
    }
}

int set_attributes_evaluate() {
    TFRPN_CHECK_CUDA(cudaFuncSetAttribute(recall_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)recall_smem_bytes(RC_MAX_K, RC_MAX_G)));
    return 0;
}

}  // namespace tfrpn

using namespace tfrpn;

extern "C" int tfrpn_proposal_recall(tfrpn_handle h, const float* proposals, const int32_t* valid, const float* gt_boxes,
                                     const int32_t* gt_labels, int B, int P, int G, const tfrpn_recall_cfg* cfg,
                                     float* gt_iou, int64_t* counts, tfrpn_stream s) {
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "proposal_recall: null handle");
    if (!cfg || !counts) return fail(TFRPN_ERR_BAD_ARG, "proposal_recall: null cfg or counts");
    if (B < 0 || P < 0 || G < 0) return fail(TFRPN_ERR_BAD_ARG, "proposal_recall: negative shape");
    if ((P > 0 && B > 0 && !proposals) || (G > 0 && B > 0 && !gt_boxes))
        return fail(TFRPN_ERR_BAD_ARG, "proposal_recall: null proposals or gt_boxes");
    if (cfg->n_thresholds < 1 || cfg->n_thresholds > 16)
        return fail(TFRPN_ERR_BAD_ARG, "proposal_recall: n_thresholds = %d, must be 1..16", cfg->n_thresholds);
    if (cfg->n_limits < 1 || cfg->n_limits > 8)
        return fail(TFRPN_ERR_BAD_ARG, "proposal_recall: n_limits = %d, must be 1..8", cfg->n_limits);
    if (cfg->matching != 0 && cfg->matching != 1)
        return fail(TFRPN_ERR_BAD_ARG, "proposal_recall: matching = %d, must be 0 (greedy) or 1 (coverage)", cfg->matching);
    RecallParams q = {};
    int kmax = 0;
    for (int t = 0; t < cfg->n_thresholds; ++t) {
        const float v = cfg->thresholds[t];
        if (!(v > 0.0f && v <= 1.0f)) return fail(TFRPN_ERR_BAD_ARG, "proposal_recall: threshold %d = %g, must be in (0, 1]", t, v);
        q.thr[t] = v;
    }
    for (int i = 0; i < cfg->n_limits; ++i) {
        const int v = cfg->limits[i];
        if (v <= 0) return fail(TFRPN_ERR_BAD_ARG, "proposal_recall: limit %d = %d, must be > 0", i, v);
        q.lim[i] = v;
        kmax = v > kmax ? v : kmax;
    }
    if (G > RC_MAX_G) return fail(TFRPN_ERR_UNSUPPORTED, "proposal_recall: G = %d, at most %d GT boxes per image", G, RC_MAX_G);
    if (kmax > RC_MAX_K) return fail(TFRPN_ERR_UNSUPPORTED, "proposal_recall: limit %d, at most %d", kmax, RC_MAX_K);
    if ((proposals && !aligned16(proposals)) || (gt_boxes && !aligned16(gt_boxes)) ||
        (reinterpret_cast<uintptr_t>(counts) & 7u) || (reinterpret_cast<uintptr_t>(gt_iou) & 3u) ||
        (reinterpret_cast<uintptr_t>(valid) & 3u) || (reinterpret_cast<uintptr_t>(gt_labels) & 3u))
        return fail(TFRPN_ERR_MISALIGNED, "proposal_recall: boxes must be 16-byte aligned, counts 8-byte, the rest 4-byte");
    TFRPN_ENTER(h);
    TFRPN_CHECK_ON_DEVICE(h, counts, "proposal_recall: counts");
    if (B == 0 || G == 0) return 0;   // nothing to count
    TFRPN_CHECK_ON_DEVICE(h, gt_boxes, "proposal_recall: gt_boxes");
    if (P > 0) TFRPN_CHECK_ON_DEVICE(h, proposals, "proposal_recall: proposals");
    if (valid) TFRPN_CHECK_ON_DEVICE(h, valid, "proposal_recall: valid");
    if (gt_labels) TFRPN_CHECK_ON_DEVICE(h, gt_labels, "proposal_recall: gt_labels");
    if (gt_iou) TFRPN_CHECK_ON_DEVICE(h, gt_iou, "proposal_recall: gt_iou");
    q.prop = reinterpret_cast<const float4*>(proposals);
    q.valid = valid;
    q.gt = reinterpret_cast<const float4*>(gt_boxes);
    q.labels = gt_labels;
    q.gt_iou = gt_iou;
    q.counts = reinterpret_cast<unsigned long long*>(counts);
    q.B = B; q.P = P; q.G = G; q.L = cfg->n_limits; q.T = cfg->n_thresholds;
    q.kcap = kmax < P ? kmax : P;
    q.coverage = cfg->matching;
    cudaStream_t st = as_stream(s);
    prof_begin(h, TFRPN_K_RECALL, st);
    recall_kernel<<<dim3(q.L, B), RC_THREADS, recall_smem_bytes(q.kcap, G), st>>>(q);
    prof_end(h, st);
    TFRPN_AFTER_LAUNCH("recall_kernel");
    return 0;
}
