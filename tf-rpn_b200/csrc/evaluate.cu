// evaluate.cu -- quality measures the reference does not have: detection mAP (below, after recall_kernel) and
// proposal recall against ground truth (the quality measure of an RPN):
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
#include <algorithm>

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

// ---- detection mAP (tfrpn_map_update / tfrpn_map_compute, include/tfrpn.h) ------------------------------------------
//   map_match_kernel    grid B x 512 threads, one CTA per image.  The image's detections (boxes, areas, 64-bit keys
//                       (class | score key | row)) and GT (boxes, areas, 32-bit keys (label | ignore | crowd | index))
//                       are staged in dynamic shared memory and bitonic-sorted there, so each class is one segment of
//                       detections in (score descending, row) order and one segment of GT.  Warp w takes the (class,
//                       threshold) items w, w+16, ...: the class's GT are spread over the lanes (at most 32 each, so
//                       the matched state is one 32-bit mask per lane), every detection in order is matched by
//                       __reduce_max_sync over the IoU bits (IoUs are >= +0, so bits order like values) and a max
//                       (coco) or min (voc) reduction over the GT index among the equal ones.  The outcome goes into
//                       the detection's TP / ignore bit t (shared atomicOr).  Then one record per slot of the image
//                       (the sorted order, so equal scores keep the row order), and one 64-bit atomic per class to n_gt.
//   map_cursor_kernel   one thread: advances the cursor by B*R, or sets overflow when the batch did not fit (the match
//                       kernel read the same cursor and wrote nothing then).
//   map_hist / map_scan / map_scatter_kernel   one pass of a stable LSD radix sort of the records over 11-bit digits:
//                       the score key in three digits, then the class (the sentinel 2047 last).  A tile is 2048
//                       records of one warp: per-tile histograms, a per-digit scan over the tiles (16 x 128 threads),
//                       then a scatter in which every warp walks its tile in order and ranks equal digits with
//                       __match_any_sync.  Stability keeps the insertion order of equal scores; the class digit's
//                       totals (tot) are the class segments.
//   map_ap_kernel       grid (T, C) x 512 threads, one CTA per (threshold, class), walking the class segment in chunks
//                       of 512.  Pass A: block scans give TP / FP, the chunk maxima of the precision go to the
//                       workspace; thread 0 turns them into suffix maxima; pass B: the same scans again, a block suffix
//                       max with the carry of the later chunks gives the envelope, each entry writes the recall points
//                       it covers (coco / voc07) or its area term (voc, added in order by one thread per chunk).
// Every count is an integer and every float64 sum has one order, so the results are bit-identical to
// oracle/map_oracle.py and do not depend on launch order or batching.
constexpr int MP_THREADS = 512;
constexpr int MP_WARPS = MP_THREADS / 32;
constexpr int MP_MAX_R = 4096;
constexpr int MP_MAX_G = 1024;
constexpr int MP_MAX_C = 1024;
constexpr uint32_t MP_SENTINEL = 2047u;   // class of a slot that takes no part: the largest class digit
constexpr int MP_DIGITS = 2048;
constexpr int MP_SORT_THREADS = 128;
constexpr int MP_SORT_WARPS = MP_SORT_THREADS / 32;
constexpr int MP_TILE = 2048;             // records per warp in a sort pass
constexpr int MP_AP_THREADS = 512;        // = entries per chunk of map_ap_kernel
constexpr int MP_AP_WARPS = MP_AP_THREADS / 32;

struct MapMatchParams {
    const float4* det;      // (B,R,4)
    const float* scores;    // (B,R)
    const float* classes;   // (B,R)
    const int32_t* valid;   // (B,) or null
    const float4* gt;       // (B,G,4)
    const int32_t* labels;  // (B,G)
    const uint8_t* flags;   // (B,G) or null
    uint4* records;         // (capacity) x {score key, class, tp bits | ignore bits << 16, 0}
    const long long* cursor;
    unsigned long long* n_gt;
    long long capacity;
    int B, R, G, C, T, protocol, max_dets, NP, NG;
    float thr[16];
};

static int pow2_at_least(int n) {
    int p = 1;
    while (p < n) p <<= 1;
    return p;
}
static size_t map_match_smem(int R, int G, int C) {
    return (size_t)(R + G) * 16 + (size_t)pow2_at_least(R) * 8 + (size_t)R * 8 + (size_t)pow2_at_least(G) * 4 +
           (size_t)G * 4 + (size_t)C * 20;
}

// ascending key of "score descending, compared by value": NaN first, +0 and -0 equal
__device__ __forceinline__ uint32_t map_score_key(float s) {
    if (s != s) return 0u;
    uint32_t u = __float_as_uint(s);
    if ((u << 1) == 0u) u = 0u;
    return ~orderable(__uint_as_float(u));
}

// COCO crowd region: inter / area(det), +0 when area(det) <= 0.  A GT whose area is NaN has a NaN or an inf - inf
// in its coordinates, where the reference's max / min would carry the NaN into inter (fmaxf drops it): +0 as well.
__device__ __forceinline__ float crowd_iou(float4 d, float da, float4 g, float ga) {
    if (!(da > 0.0f) || ga != ga) return 0.0f;
    const float x_top = fmaxf(d.y, g.y), y_top = fmaxf(d.x, g.x);
    const float x_bot = fminf(d.w, g.w), y_bot = fminf(d.z, g.z);
    const float inter = __fmul_rn(fmaxf(__fsub_rn(x_bot, x_top), 0.0f), fmaxf(__fsub_rn(y_bot, y_top), 0.0f));
    return __fdiv_rn(inter, da);
}

template <typename K>
__device__ void block_bitonic(K* a, int n) {   // n a power of two, ascending; called by the whole CTA
    for (int k = 2; k <= n; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n; i += blockDim.x) {
                const int p = i ^ j;
                if (p > i) {
                    const K x = a[i], y = a[p];
                    if (((i & k) == 0) == (x > y)) { a[i] = y; a[p] = x; }
                }
            }
            __syncthreads();
        }
}

// The matching score of detection (db, da) against the GT of sorted position p (key gk).
__device__ __forceinline__ float map_pair_iou(float4 db, float da, uint32_t gk, const float4* sgb, const float* sga,
                                              bool nice, bool coco) {
    const int g = (int)(gk & 1023u);
    float v;
    if (coco && ((gk >> 10) & 1u)) v = crowd_iou(db, da, sgb[g], sga[g]);
    else v = nice ? iou_nice(sgb[g], sga[g], db, da) : iou_ref(db, da, sgb[g], sga[g]);
    return v > 0.0f ? v : 0.0f;   // NaN, negative and -0 score +0
}

// One detection against the m GT of its class (sorted positions g0.., lane-strided), at threshold thr.
// -> 0 FP, 1 TP, 2 ignored (warp-uniform); `matched` bit k is the lane's k-th GT.
__device__ __forceinline__ int match_coco(float4 db, float da, const uint32_t* gk, int m, const float4* sgb,
                                          const float* sga, bool nice, float thr, uint32_t& matched) {
    uint32_t b1 = 0u, b2 = 0u;
    int j1 = -1, j2 = -1, k1 = 0, k2 = 0;
    for (int k = 0, p = lane_id(); p < m; ++k, p += 32) {
        const uint32_t key = gk[p];
        const float v = map_pair_iou(db, da, key, sgb, sga, nice, true);
        if (!(v >= thr)) continue;
        const uint32_t u = __float_as_uint(v);
        const int g = (int)(key & 1023u);
        const bool taken = (matched >> k) & 1u;
        if (!((key >> 11) & 1u)) {
            if (!taken && (u > b1 || (u == b1 && g > j1))) { b1 = u; j1 = g; k1 = k; }
        } else if (!taken || ((key >> 10) & 1u)) {
            if (u > b2 || (u == b2 && g > j2)) { b2 = u; j2 = g; k2 = k; }
        }
    }
    const uint32_t m1 = __reduce_max_sync(0xffffffffu, b1);
    if (m1) {   // a non-ignored GT: the largest IoU, ties to the highest index
        const int j = (int)__reduce_max_sync(0xffffffffu, b1 == m1 ? (uint32_t)(j1 + 1) : 0u) - 1;
        if (b1 == m1 && j1 == j) matched |= 1u << k1;
        return 1;
    }
    const uint32_t m2 = __reduce_max_sync(0xffffffffu, b2);
    if (m2) {   // an ignored GT that is free or a crowd
        const int j = (int)__reduce_max_sync(0xffffffffu, b2 == m2 ? (uint32_t)(j2 + 1) : 0u) - 1;
        if (b2 == m2 && j2 == j) matched |= 1u << k2;
        return 2;
    }
    return 0;
}

__device__ __forceinline__ int match_voc(float4 db, float da, const uint32_t* gk, int m, const float4* sgb,
                                         const float* sga, bool nice, float thr, uint32_t& matched) {
    uint32_t bu = 0u, bj = 0xFFFFFFFFu;
    int bk = 0;
    bool bign = false;
    for (int k = 0, p = lane_id(); p < m; ++k, p += 32) {
        const uint32_t key = gk[p];
        const uint32_t u = __float_as_uint(map_pair_iou(db, da, key, sgb, sga, nice, false));
        const uint32_t g = key & 1023u;
        if (u > bu || (u == bu && g < bj)) { bu = u; bj = g; bk = k; bign = (key >> 11) & 1u; }
    }
    const uint32_t s = __reduce_max_sync(0xffffffffu, bu);   // the best IoU over all GT of the class ...
    const uint32_t j = __reduce_min_sync(0xffffffffu, bu == s ? bj : 0xFFFFFFFFu);   // ... at its lowest index
    if (!(__uint_as_float(s) > thr)) return 0;
    int out = 0;
    if (bu == s && bj == j) {
        if (bign) out = 2;
        else if (!((matched >> bk) & 1u)) { out = 1; matched |= 1u << bk; }
    }
    return (int)__reduce_max_sync(0xffffffffu, (uint32_t)out);
}

__global__ void __launch_bounds__(MP_THREADS) map_match_kernel(MapMatchParams q) {
    extern __shared__ float4 mp_smem[];
    const int b = blockIdx.x, R = q.R, G = q.G, C = q.C, NP = q.NP, NG = q.NG;
    const long long base = *q.cursor;
    if (base + (long long)q.B * R > q.capacity) return;   // the batch does not fit: it records nothing
    float4* sdb = mp_smem;                                                    // [R]  detection boxes (by row)
    float4* sgb = sdb + R;                                                    // [G]  GT boxes (by index)
    unsigned long long* dkey = reinterpret_cast<unsigned long long*>(sgb + G);   // [NP] class << 44 | score key << 12 | row
    float* sda = reinterpret_cast<float*>(dkey + NP);                         // [R]  detection areas
    uint32_t* msk = reinterpret_cast<uint32_t*>(sda + R);                     // [R]  tp | ignore << 16, sorted position
    uint32_t* gkey = msk + R;                                                 // [NG] label << 12 | ign << 11 | crowd << 10 | g
    float* sga = reinterpret_cast<float*>(gkey + NG);                         // [G]  GT areas
    int* dlo = reinterpret_cast<int*>(sga + G);                               // [C]  class segments of dkey
    int* dhi = dlo + C;
    int* glo = dhi + C;                                                       // [C]  class segments of gkey
    int* ghi = glo + C;
    int* gni = ghi + C;                                                       // [C]  non-ignored GT per class
    for (int c = threadIdx.x; c < C; c += MP_THREADS) dlo[c] = dhi[c] = glo[c] = ghi[c] = gni[c] = 0;
    const int nv = q.valid ? min(max(q.valid[b], 0), R) : R;
    const bool coco = q.protocol == 0;
    bool ok = true;
    for (int r = threadIdx.x; r < NP; r += MP_THREADS) {
        unsigned long long k = ~0ull;
        if (r < R) {
            const long long o = (long long)b * R + r;
            const float4 v = ldg_f4(q.det + o);
            sdb[r] = v;
            sda[r] = box_area(v);
            msk[r] = 0u;
            const float cf = q.classes[o];
            uint32_t cls = MP_SENTINEL, sk = 0u;
            if (r < nv && cf == floorf(cf) && cf >= 0.0f && cf < (float)C) {
                cls = (uint32_t)cf;
                sk = map_score_key(q.scores[o]);
                ok = ok && nice_coords(v) && v.z >= v.x && v.w >= v.y;
            }
            k = ((unsigned long long)cls << 44) | ((unsigned long long)sk << 12) | (unsigned long long)r;
        }
        dkey[r] = k;
    }
    for (int g = threadIdx.x; g < NG; g += MP_THREADS) {
        uint32_t k = ~0u;
        if (g < G) {
            const long long o = (long long)b * G + g;
            const float4 v = ldg_f4(q.gt + o);
            sgb[g] = v;
            sga[g] = box_area(v);
            const int lab = q.labels[o];
            if (lab >= 0 && lab < C) {
                const uint32_t f = q.flags ? q.flags[o] : 0u;
                const uint32_t crowd = (f >> 1) & 1u, ign = (f | crowd) & 1u;
                k = ((uint32_t)lab << 12) | (ign << 11) | (crowd << 10) | (uint32_t)g;
                ok = ok && nice_box(v);
            }
        }
        gkey[g] = k;
    }
    const bool nice = __syncthreads_and(ok) != 0;
    block_bitonic(dkey, NP);
    block_bitonic(gkey, NG);
    for (int i = threadIdx.x; i < R; i += MP_THREADS) {
        const uint32_t c = (uint32_t)(dkey[i] >> 44);
        if (c < (uint32_t)C) {
            if (i == 0 || (uint32_t)(dkey[i - 1] >> 44) != c) dlo[c] = i;
            if (i == R - 1 || (uint32_t)(dkey[i + 1] >> 44) != c) dhi[c] = i + 1;
        }
    }
    for (int i = threadIdx.x; i < G; i += MP_THREADS) {
        const uint32_t c = gkey[i] >> 12;
        if (c < (uint32_t)C) {
            if (i == 0 || (gkey[i - 1] >> 12) != c) glo[c] = i;
            if (i == G - 1 || (gkey[i + 1] >> 12) != c) ghi[c] = i + 1;
            if (!((gkey[i] >> 11) & 1u)) atomicAdd(&gni[c], 1);
        }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += MP_THREADS)
        if (gni[c]) atomicAdd(q.n_gt + c, (unsigned long long)gni[c]);

    for (int item = warp_id(); item < C * q.T; item += MP_WARPS) {
        const int c = item / q.T, t = item - c * q.T;
        const int d0 = dlo[c];
        int d1 = dhi[c];
        if (d1 == d0) continue;
        if (coco && q.max_dets > 0) d1 = min(d1, d0 + q.max_dets);
        const int m = ghi[c] - glo[c];
        if (m == 0) continue;   // every detection is FP
        const uint32_t* gk = gkey + glo[c];
        const float thr = q.thr[t];
        uint32_t matched = 0u;
        for (int i = d0; i < d1; ++i) {
            const int row = (int)(dkey[i] & 0xFFFu);
            const int out = coco ? match_coco(sdb[row], sda[row], gk, m, sgb, sga, nice, thr, matched)
                                 : match_voc(sdb[row], sda[row], gk, m, sgb, sga, nice, thr, matched);
            if (lane_id() == 0 && out) atomicOr(&msk[i], 1u << (out == 1 ? t : 16 + t));
        }
    }
    __syncthreads();
    uint4* out = q.records + base + (long long)b * R;
    for (int i = threadIdx.x; i < R; i += MP_THREADS) {
        const unsigned long long k = dkey[i];
        const uint32_t c = (uint32_t)(k >> 44);
        uint4 rec = make_uint4(~0u, MP_SENTINEL, 0u, 0u);
        if (c < (uint32_t)C && !(coco && q.max_dets > 0 && i - dlo[c] >= q.max_dets))
            rec = make_uint4((uint32_t)(k >> 12), c, msk[i], 0u);
        out[i] = rec;
    }
}

__global__ void map_cursor_kernel(long long* cursor, int* overflow, long long n, long long capacity) {
    const long long base = *cursor;
    if (base + n <= capacity) *cursor = base + n;
    else *overflow = 1;
}

struct MapSortParams {
    const uint4* src;
    uint4* dst;
    const long long* cursor;
    unsigned* hist;   // (tiles, 2048): per tile, then (after map_scan_kernel) its exclusive prefix per digit
    unsigned* tot;    // (2048) records per digit
    long long capacity;
    int pass;
};
__device__ __forceinline__ long long map_count(const MapSortParams& p) {
    const long long n = *p.cursor;
    return n < p.capacity ? n : p.capacity;
}
__device__ __forceinline__ uint32_t map_digit(uint4 r, int pass) {
    return pass == 3 ? r.y : (r.x >> (11 * pass)) & 2047u;
}

__global__ void __launch_bounds__(MP_SORT_THREADS) map_hist_kernel(MapSortParams p) {
    __shared__ unsigned cnt[MP_SORT_WARPS][MP_DIGITS];
    const int lane = lane_id();
    const long long n = map_count(p), tile = (long long)blockIdx.x * MP_SORT_WARPS + warp_id(), lo = tile * MP_TILE;
    if (lo >= n) return;
    unsigned* mine = cnt[warp_id()];
    for (int d = lane; d < MP_DIGITS; d += 32) mine[d] = 0u;
    __syncwarp();
    const long long hi = min(n, lo + MP_TILE);
    for (long long i = lo + lane; i - lane < hi; i += 32) {
        const bool in = i < hi;
        const uint32_t d = in ? map_digit(p.src[i], p.pass) : 0xFFFFFFFFu;
        const unsigned m = __match_any_sync(0xffffffffu, d);
        if (in && lane == __ffs(m) - 1) mine[d] += __popc(m);
        __syncwarp();
    }
    unsigned* h = p.hist + tile * MP_DIGITS;
    for (int d = lane; d < MP_DIGITS; d += 32) h[d] = mine[d];
}

__global__ void __launch_bounds__(MP_SORT_THREADS) map_scan_kernel(MapSortParams p) {
    const int d = blockIdx.x * MP_SORT_THREADS + threadIdx.x;
    const long long tiles = (map_count(p) + MP_TILE - 1) / MP_TILE;
    unsigned run = 0u;
    long long t = 0;
    for (; t + 8 <= tiles; t += 8) {   // the loads of 8 tiles in flight together
        unsigned v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = p.hist[(t + j) * MP_DIGITS + d];
#pragma unroll
        for (int j = 0; j < 8; ++j) { p.hist[(t + j) * MP_DIGITS + d] = run; run += v[j]; }
    }
    for (; t < tiles; ++t) {
        const unsigned v = p.hist[t * MP_DIGITS + d];
        p.hist[t * MP_DIGITS + d] = run;
        run += v;
    }
    p.tot[d] = run;
}

__global__ void __launch_bounds__(MP_SORT_THREADS) map_scatter_kernel(MapSortParams p) {
    __shared__ unsigned off[MP_SORT_WARPS][MP_DIGITS];
    __shared__ unsigned dbase[MP_DIGITS];
    __shared__ int wsum[MP_SORT_WARPS];
    constexpr int PER = MP_DIGITS / MP_SORT_THREADS;
    const int lane = lane_id(), warp = warp_id();
    // exclusive scan of the digit totals: where each digit's records start
    unsigned v[PER];
    int s = 0;
#pragma unroll
    for (int j = 0; j < PER; ++j) { v[j] = p.tot[threadIdx.x * PER + j]; s += (int)v[j]; }
    const int incl = warp_incl_scan(s);
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    unsigned run = (unsigned)(incl - s);
    for (int w = 0; w < warp; ++w) run += (unsigned)wsum[w];
#pragma unroll
    for (int j = 0; j < PER; ++j) { dbase[threadIdx.x * PER + j] = run; run += v[j]; }
    __syncthreads();
    const long long n = map_count(p), tile = (long long)blockIdx.x * MP_SORT_WARPS + warp, lo = tile * MP_TILE;
    if (lo >= n) return;
    unsigned* mine = off[warp];
    const unsigned* h = p.hist + tile * MP_DIGITS;
    for (int d = lane; d < MP_DIGITS; d += 32) mine[d] = dbase[d] + h[d];
    __syncwarp();
    const long long hi = min(n, lo + MP_TILE);
    for (long long i = lo + lane; i - lane < hi; i += 32) {
        const bool in = i < hi;
        uint4 r = make_uint4(0u, 0u, 0u, 0u);
        if (in) r = p.src[i];
        const uint32_t d = in ? map_digit(r, p.pass) : 0xFFFFFFFFu;
        const unsigned m = __match_any_sync(0xffffffffu, d);
        if (in) p.dst[mine[d] + __popc(m & ((1u << lane) - 1u))] = r;
        __syncwarp();
        if (in && lane == __ffs(m) - 1) mine[d] += __popc(m);
        __syncwarp();
    }
}

struct MapApParams {
    const uint4* rec;          // sorted records
    const unsigned* tot;       // records per class (the class digit's totals)
    const long long* n_gt;     // (C)
    double* chunk_max;         // (16, slots)
    double* ap;                // (C,T)
    double* recall;            // (C,T)
    long long slots;
    int C, T, protocol;
};

// inclusive block scan (sum); `total` = the CTA's sum.  Every thread of the CTA calls it.
__device__ __forceinline__ int ap_block_scan(int v, int* s_w, int& total) {
    const int x = warp_incl_scan(v);
    if (lane_id() == 31) s_w[warp_id()] = x;
    __syncthreads();
    int off = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < MP_AP_WARPS; ++w) {
        const int s = s_w[w];
        off += w < warp_id() ? s : 0;
        tot += s;
    }
    __syncthreads();
    total = tot;
    return x + off;
}
// max over this thread and every later thread of the CTA (values >= 0)
__device__ __forceinline__ double ap_block_suffix_max(double v, double* s_w) {
    const int lane = lane_id(), warp = warp_id();
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double y = __shfl_down_sync(0xffffffffu, v, o);
        if (lane + o < 32) v = fmax(v, y);
    }
    if (lane == 0) s_w[warp] = v;
    __syncthreads();
    for (int w = warp + 1; w < MP_AP_WARPS; ++w) v = fmax(v, s_w[w]);
    __syncthreads();
    return v;
}

__device__ __forceinline__ double ap_precision(long long tp, long long n, int protocol) {
    const double T = (double)tp;
    return protocol == 0 ? __ddiv_rn(T, __dadd_rn((double)n, 0x1p-52))   // (FP + TP) + np.spacing(1)
                         : __ddiv_rn(T, fmax((double)n, 0x1p-52));
}

__global__ void __launch_bounds__(MP_AP_THREADS, 1) map_ap_kernel(MapApParams p) {
    __shared__ double s_q[101];
    __shared__ double s_term[MP_AP_THREADS];
    __shared__ double s_dw[MP_AP_WARPS];
    __shared__ int s_w[MP_AP_WARPS];
    __shared__ long long s_start[MP_AP_WARPS];
    const int t = blockIdx.x, c = blockIdx.y, tid = threadIdx.x;
    const long long o = (long long)c * p.T + t, ng = p.n_gt[c];
    if (ng == 0) {
        if (tid == 0) p.ap[o] = p.recall[o] = __longlong_as_double(0x7ff8000000000000ll);   // NaN: no GT
        return;
    }
    long long st = 0;
    for (int d = tid; d < c; d += MP_AP_THREADS) st += p.tot[d];
#pragma unroll
    for (int w = 16; w > 0; w >>= 1) st += __shfl_xor_sync(0xffffffffu, st, w);
    if (lane_id() == 0) s_start[warp_id()] = st;
    if (tid <= 100) s_q[tid] = 0.0;
    __syncthreads();
    long long start = 0;
#pragma unroll
    for (int w = 0; w < MP_AP_WARPS; ++w) start += s_start[w];
    const long long len = p.tot[c];
    const int nch = (int)((len + MP_AP_THREADS - 1) / MP_AP_THREADS);
    double* cm = p.chunk_max + (long long)t * p.slots + start / MP_AP_THREADS + c;
    const bool coco = p.protocol == 0, voc = p.protocol == 1;
    const int npts = coco ? 101 : 11;
    const double step = coco ? 0.01 : 0.1;
    const double dng = (double)ng;

    // pass A: the precision of every entry; the chunk maxima
    long long cTP = 0, cN = 0;
    for (int j = 0; j < nch; ++j) {
        const long long i = start + (long long)j * MP_AP_THREADS + tid;
        const uint32_t z = i < start + len ? p.rec[i].z : (1u << (16 + t));
        const int ni = !((z >> (16 + t)) & 1u), tp = ni & (int)((z >> t) & 1u);
        int tot;
        const int inc = ap_block_scan((ni << 16) | tp, s_w, tot);
        const long long TP = cTP + (inc & 0xFFFF), N = cN + (inc >> 16);
        const double m = ap_block_suffix_max(ni ? ap_precision(TP, N, p.protocol) : 0.0, s_dw);
        if (tid == 0) cm[j] = m;
        cTP += tot & 0xFFFF;
        cN += tot >> 16;
    }
    __syncthreads();
    if (tid == 0) {   // chunk j -> the envelope carried in from the chunks after it
        double s = 0.0;
        for (int j = nch - 1; j >= 0; --j) {
            const double v = cm[j];
            cm[j] = s;
            s = fmax(s, v);
        }
    }
    __syncthreads();

    // pass B: envelope, recall points / area terms
    const long long TPall = cTP;
    cTP = cN = 0;
    double area = 0.0;
    for (int j = 0; j < nch; ++j) {
        const long long i = start + (long long)j * MP_AP_THREADS + tid;
        const uint32_t z = i < start + len ? p.rec[i].z : (1u << (16 + t));
        const int ni = !((z >> (16 + t)) & 1u), tp = ni & (int)((z >> t) & 1u);
        int tot;
        const int inc = ap_block_scan((ni << 16) | tp, s_w, tot);
        const long long TP = cTP + (inc & 0xFFFF), N = cN + (inc >> 16);
        const double e = fmax(ap_block_suffix_max(ni ? ap_precision(TP, N, p.protocol) : 0.0, s_dw), cm[j]);
        if (ni) {
            const double rc = __ddiv_rn((double)TP, dng);
            const double prev = __ddiv_rn((double)(TP - tp), dng);
            if (voc) {
                if (tp) s_term[(inc & 0xFFFF) - 1] = __dmul_rn(__dsub_rn(rc, prev), e);
            } else {
                // the points k with rc_prev < r_k <= rc; the first entry also takes r_0 = 0
                const double lo = N == 1 ? -1.0 : prev;
                int k = lo < 0.0 ? 0 : max(0, (int)(lo / step) - 2);
                while (k < npts && __dmul_rn((double)k, step) <= lo) ++k;
                for (; k < npts && __dmul_rn((double)k, step) <= rc; ++k) s_q[k] = e;
            }
        }
        __syncthreads();
        if (voc && tid == 0)
            for (int k = 0; k < (tot & 0xFFFF); ++k) area = __dadd_rn(area, s_term[k]);
        __syncthreads();
        cTP += tot & 0xFFFF;
        cN += tot >> 16;
    }
    if (tid == 0) {
        if (!voc) {
            for (int k = 0; k < npts; ++k) area = __dadd_rn(area, coco ? s_q[k] : __ddiv_rn(s_q[k], 11.0));
            if (coco) area = __ddiv_rn(area, 101.0);
        }
        p.ap[o] = area;
        p.recall[o] = __ddiv_rn((double)TPall, dng);
    }
}

size_t map_workspace_bytes(long long capacity, int C) {
    auto a = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t tiles = (size_t)((capacity + MP_TILE - 1) / MP_TILE);
    return 2 * a((size_t)capacity * 16) + a(tiles * MP_DIGITS * 4) + a(MP_DIGITS * 4) +
           a((size_t)16 * (size_t)(capacity / MP_AP_THREADS + C + 2) * 8);
}

int set_attributes_evaluate() {
    TFRPN_CHECK_CUDA(cudaFuncSetAttribute(recall_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)recall_smem_bytes(RC_MAX_K, RC_MAX_G)));
    TFRPN_CHECK_CUDA(cudaFuncSetAttribute(map_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)map_match_smem(MP_MAX_R, MP_MAX_G, MP_MAX_C)));
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

static int map_check_cfg(const tfrpn_map_cfg* cfg, const char* fn) {
    if (!cfg) return fail(TFRPN_ERR_BAD_ARG, "%s: null cfg", fn);
    if (cfg->protocol < 0 || cfg->protocol > 2)
        return fail(TFRPN_ERR_BAD_ARG, "%s: protocol = %d, must be 0 (coco), 1 (voc) or 2 (voc07)", fn, cfg->protocol);
    if (cfg->num_classes < 1) return fail(TFRPN_ERR_BAD_ARG, "%s: num_classes = %d, must be >= 1", fn, cfg->num_classes);
    if (cfg->n_thresholds < 1 || cfg->n_thresholds > 16)
        return fail(TFRPN_ERR_BAD_ARG, "%s: n_thresholds = %d, must be 1..16", fn, cfg->n_thresholds);
    for (int t = 0; t < cfg->n_thresholds; ++t) {
        const float v = cfg->thresholds[t];
        if (!(v > 0.0f && v <= 1.0f)) return fail(TFRPN_ERR_BAD_ARG, "%s: threshold %d = %g, must be in (0, 1]", fn, t, v);
    }
    if (cfg->max_dets < 0) return fail(TFRPN_ERR_BAD_ARG, "%s: max_dets = %d, must be >= 0", fn, cfg->max_dets);
    if (cfg->num_classes > MP_MAX_C)
        return fail(TFRPN_ERR_UNSUPPORTED, "%s: num_classes = %d, at most %d", fn, cfg->num_classes, MP_MAX_C);
    return 0;
}

static int map_check_state(const tfrpn_map_state* st, const char* fn) {
    if (!st || !st->cursor || !st->n_gt || !st->overflow || (st->capacity > 0 && !st->records))
        return fail(TFRPN_ERR_BAD_ARG, "%s: null state, cursor, n_gt, overflow or records", fn);
    if (st->capacity < 0) return fail(TFRPN_ERR_BAD_ARG, "%s: capacity = %lld, must be >= 0", fn, (long long)st->capacity);
    if (st->capacity > INT32_MAX)
        return fail(TFRPN_ERR_UNSUPPORTED, "%s: capacity = %lld, at most %d records", fn, (long long)st->capacity, INT32_MAX);
    if (!aligned16(st->records) || (reinterpret_cast<uintptr_t>(st->cursor) & 7u) ||
        (reinterpret_cast<uintptr_t>(st->n_gt) & 7u) || (reinterpret_cast<uintptr_t>(st->overflow) & 3u))
        return fail(TFRPN_ERR_MISALIGNED, "%s: records must be 16-byte aligned, cursor and n_gt 8-byte, overflow 4-byte", fn);
    return 0;
}

extern "C" size_t tfrpn_map_workspace_bytes(int64_t capacity, int C) {
    return map_workspace_bytes(capacity < 0 ? 0 : capacity, C < 0 ? 0 : C);
}

extern "C" int tfrpn_map_update(tfrpn_handle h, const float* det_boxes, const float* det_scores,
                                const float* det_classes, const int32_t* valid, const float* gt_boxes,
                                const int32_t* gt_labels, const uint8_t* gt_flags, int B, int R, int G,
                                const tfrpn_map_cfg* cfg, const tfrpn_map_state* state, tfrpn_stream s) {
    static const char* fn = "map_update";
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "map_update: null handle");
    if (int rc = map_check_cfg(cfg, fn)) return rc;
    if (int rc = map_check_state(state, fn)) return rc;
    if (B < 0 || R < 0 || G < 0) return fail(TFRPN_ERR_BAD_ARG, "map_update: negative shape");
    if (B > 0 && R > 0 && (!det_boxes || !det_scores || !det_classes))
        return fail(TFRPN_ERR_BAD_ARG, "map_update: null det_boxes, det_scores or det_classes");
    if (B > 0 && G > 0 && (!gt_boxes || !gt_labels)) return fail(TFRPN_ERR_BAD_ARG, "map_update: null gt_boxes or gt_labels");
    if (R > MP_MAX_R) return fail(TFRPN_ERR_UNSUPPORTED, "map_update: R = %d, at most %d detections per image", R, MP_MAX_R);
    if (G > MP_MAX_G) return fail(TFRPN_ERR_UNSUPPORTED, "map_update: G = %d, at most %d GT boxes per image", G, MP_MAX_G);
    if ((det_boxes && !aligned16(det_boxes)) || (gt_boxes && !aligned16(gt_boxes)) ||
        (reinterpret_cast<uintptr_t>(det_scores) & 3u) || (reinterpret_cast<uintptr_t>(det_classes) & 3u) ||
        (reinterpret_cast<uintptr_t>(valid) & 3u) || (reinterpret_cast<uintptr_t>(gt_labels) & 3u))
        return fail(TFRPN_ERR_MISALIGNED, "map_update: boxes must be 16-byte aligned, scores, classes, valid and labels 4-byte");
    TFRPN_ENTER(h);
    if (B == 0) return 0;
    TFRPN_CHECK_ON_DEVICE(h, state->cursor, "map_update: cursor");
    TFRPN_CHECK_ON_DEVICE(h, state->n_gt, "map_update: n_gt");
    TFRPN_CHECK_ON_DEVICE(h, state->overflow, "map_update: overflow");
    if (state->capacity > 0) TFRPN_CHECK_ON_DEVICE(h, state->records, "map_update: records");
    if (R > 0) {
        TFRPN_CHECK_ON_DEVICE(h, det_boxes, "map_update: det_boxes");
        TFRPN_CHECK_ON_DEVICE(h, det_scores, "map_update: det_scores");
        TFRPN_CHECK_ON_DEVICE(h, det_classes, "map_update: det_classes");
        if (valid) TFRPN_CHECK_ON_DEVICE(h, valid, "map_update: valid");
    }
    if (G > 0) {
        TFRPN_CHECK_ON_DEVICE(h, gt_boxes, "map_update: gt_boxes");
        TFRPN_CHECK_ON_DEVICE(h, gt_labels, "map_update: gt_labels");
        if (gt_flags) TFRPN_CHECK_ON_DEVICE(h, gt_flags, "map_update: gt_flags");
    }
    MapMatchParams q = {};
    q.det = reinterpret_cast<const float4*>(det_boxes);
    q.scores = det_scores;
    q.classes = det_classes;
    q.valid = valid;
    q.gt = reinterpret_cast<const float4*>(gt_boxes);
    q.labels = gt_labels;
    q.flags = gt_flags;
    q.records = reinterpret_cast<uint4*>(state->records);
    q.cursor = reinterpret_cast<const long long*>(state->cursor);
    q.n_gt = reinterpret_cast<unsigned long long*>(state->n_gt);
    q.capacity = state->capacity;
    q.B = B; q.R = R; q.G = G; q.C = cfg->num_classes; q.T = cfg->n_thresholds;
    q.protocol = cfg->protocol;
    q.max_dets = cfg->max_dets;
    q.NP = pow2_at_least(R);
    q.NG = pow2_at_least(G);
    for (int t = 0; t < q.T; ++t) q.thr[t] = cfg->thresholds[t];
    cudaStream_t st = as_stream(s);
    prof_begin(h, TFRPN_K_MAP_MATCH, st);
    map_match_kernel<<<B, MP_THREADS, map_match_smem(R, G, q.C), st>>>(q);
    TFRPN_AFTER_LAUNCH("map_match_kernel");
    map_cursor_kernel<<<1, 1, 0, st>>>(reinterpret_cast<long long*>(state->cursor), state->overflow, (long long)B * R,
                                       state->capacity);
    TFRPN_AFTER_LAUNCH("map_cursor_kernel");
    prof_end(h, st);
    return 0;
}

extern "C" int tfrpn_map_compute(tfrpn_handle h, const tfrpn_map_cfg* cfg, const tfrpn_map_state* state, double* ap,
                                 double* recall, tfrpn_stream s) {
    static const char* fn = "map_compute";
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "map_compute: null handle");
    if (int rc = map_check_cfg(cfg, fn)) return rc;
    if (int rc = map_check_state(state, fn)) return rc;
    if (!ap || !recall) return fail(TFRPN_ERR_BAD_ARG, "map_compute: null ap or recall");
    if ((reinterpret_cast<uintptr_t>(ap) & 7u) || (reinterpret_cast<uintptr_t>(recall) & 7u))
        return fail(TFRPN_ERR_MISALIGNED, "map_compute: ap and recall must be 8-byte aligned");
    TFRPN_ENTER(h);
    TFRPN_CHECK_ON_DEVICE(h, state->cursor, "map_compute: cursor");
    TFRPN_CHECK_ON_DEVICE(h, ap, "map_compute: ap");
    TFRPN_CHECK_ON_DEVICE(h, recall, "map_compute: recall");
    const long long cap = state->capacity;
    const int C = cfg->num_classes;
    cudaStream_t st = as_stream(s);
    char* ws = nullptr;
    if (int rc = ensure_workspace_prop(h, map_workspace_bytes(cap, C), st, &ws)) return rc;
    auto a = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const long long tiles = (cap + MP_TILE - 1) / MP_TILE;
    uint4* bufA = reinterpret_cast<uint4*>(ws);
    uint4* bufB = reinterpret_cast<uint4*>(ws + a((size_t)cap * 16));
    unsigned* hist = reinterpret_cast<unsigned*>(ws + 2 * a((size_t)cap * 16));
    unsigned* tot = reinterpret_cast<unsigned*>(reinterpret_cast<char*>(hist) + a((size_t)tiles * MP_DIGITS * 4));
    double* cmax = reinterpret_cast<double*>(reinterpret_cast<char*>(tot) + a(MP_DIGITS * 4));
    MapSortParams sp = {};
    sp.cursor = reinterpret_cast<const long long*>(state->cursor);
    sp.hist = hist;
    sp.tot = tot;
    sp.capacity = cap;
    const int grid = (int)std::max<long long>(1, (tiles + MP_SORT_WARPS - 1) / MP_SORT_WARPS);
    const uint4* src[4] = {reinterpret_cast<const uint4*>(state->records), bufA, bufB, bufA};
    uint4* dst[4] = {bufA, bufB, bufA, bufB};
    prof_begin(h, TFRPN_K_MAP_AP, st);
    for (int pass = 0; pass < 4; ++pass) {
        sp.src = src[pass];
        sp.dst = dst[pass];
        sp.pass = pass;
        map_hist_kernel<<<grid, MP_SORT_THREADS, 0, st>>>(sp);
        TFRPN_AFTER_LAUNCH("map_hist_kernel");
        map_scan_kernel<<<MP_DIGITS / MP_SORT_THREADS, MP_SORT_THREADS, 0, st>>>(sp);
        TFRPN_AFTER_LAUNCH("map_scan_kernel");
        map_scatter_kernel<<<grid, MP_SORT_THREADS, 0, st>>>(sp);
        TFRPN_AFTER_LAUNCH("map_scatter_kernel");
    }
    MapApParams p = {};
    p.rec = bufB;
    p.tot = tot;
    p.n_gt = reinterpret_cast<const long long*>(state->n_gt);
    p.chunk_max = cmax;
    p.ap = ap;
    p.recall = recall;
    p.slots = cap / MP_AP_THREADS + C + 2;
    p.C = C;
    p.T = cfg->n_thresholds;
    p.protocol = cfg->protocol;
    map_ap_kernel<<<dim3(p.T, C), MP_AP_THREADS, 0, st>>>(p);
    prof_end(h, st);
    TFRPN_AFTER_LAUNCH("map_ap_kernel");
    return 0;
}
