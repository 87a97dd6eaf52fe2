// roi_detect.cu -- the box head's detections at inference (tfrpn_roi_head_detections): softmax, per-class decode of
// the RoIs, the size filter and class-aware NMS, torchvision's RoIHeads.postprocess_detections on the device.
//
//   roi_det_score_kernel<G>  G lanes per row (roi_row_lanes(C), as roi_loss_partial_kernel<G>), grid-stride over the
//                            B*S rows.  The row's max and exp-sum come from roi_row_stats<G> (logits only), so p has
//                            the bits of the losses' softmax.  Each lane then walks its 4-class chunks: p, probs when
//                            asked, the score test, and the staged score (B,S,C): p where the test passes, -inf
//                            otherwise (class 0 and rows that take no part included).  A second pass decodes the boxes
//                            of the entries that passed only (for q = 1 the row's one box), writes them into the
//                            staged (B,S,q) and sets the score of a box below min_size back to -inf.  So the boxes
//                            cost memory traffic per candidate, not per B*S*C, and the decode stays out of the
//                            softmax loop.
//   then the multi-class NMS of proposals.cu (nms_mc_run), unchanged, on the staged arrays as (B,K = S,C) scores and
//   (B,S,q) boxes with the candidates "score > -inf": exactly the candidates above, in ascending s.  Class 0's empty
//   keep lists take no output rank, so the merge writes the class ids 1..C-1 with no offset.
#include <algorithm>
#include <cmath>

#include "roi_rows.cuh"

namespace tfrpn {

constexpr int DET_THREADS = 256;
constexpr int DET_MAX_CTAS = 1184;   // 8 CTAs of 256 threads on each of 148 SMs; the rows are grid-strided

struct RoiDetParams {
    const float4* rois;    // (B,S)
    const int* valid;      // (B,) or null
    const float* x;        // (B,S,C) logits or probabilities
    const float4* deltas;  // (B,S,q)
    long long rows;        // B*S
    int S, C, q, logits, clip;
    bool vec_in, vec_out, vec_st;
    float4 var;
    float max_log_scale, min_size, sthr;
    float* probs;          // (B,S,C) or null
    float* st_scores;      // (B,S,C)
    float4* st_boxes;      // (B,S,q)
};

// box k of row r: deltas * variances, dh / dw clamped from above (NaN stays NaN), decode_ref, clip01
__device__ __forceinline__ float4 det_box(const RoiDetParams& p, float4 roi, long long r, int k) {
    float4 d = mul4(ldg_f4(p.deltas + r * p.q + k), p.var);
    d.z = d.z > p.max_log_scale ? p.max_log_scale : d.z;
    d.w = d.w > p.max_log_scale ? p.max_log_scale : d.w;
    const float4 b = decode_ref(roi, d);
    return p.clip ? clip01(b) : b;
}
// torchvision's remove_small_boxes: a NaN extent fails the comparison and drops the box
__device__ __forceinline__ bool det_keeps_size(float4 b, float min_size) {
    return !(min_size > 0.0f) || (__fsub_rn(b.z, b.x) >= min_size && __fsub_rn(b.w, b.y) >= min_size);
}

template <int G>
__global__ void __launch_bounds__(DET_THREADS) roi_det_score_kernel(RoiDetParams p) {
    constexpr int RPW = 32 / G;   // rows per warp and pass
    const int g = lane_id() % G;
    const long long stride = (long long)gridDim.x * (DET_THREADS / 32) * RPW;
    for (long long r0 = ((long long)blockIdx.x * (DET_THREADS / 32) + warp_id()) * RPW; r0 < p.rows; r0 += stride) {
        const long long r = r0 + lane_id() / G;
        const bool in = r < p.rows;
        const int b = in ? (int)(r / p.S) : 0;
        const int s = in ? (int)(r - (long long)b * p.S) : 0;
        const bool part = in && s < (p.valid ? min(max(__ldg(p.valid + b), 0), p.S) : p.S);
        const float* x = p.x + (in ? r : 0) * p.C;
        float m = 0.0f, sum = 1.0f;
        if (p.logits) {
            int first;
            bool nan;
            roi_row_stats<G>(x, in ? p.C : 0, p.vec_in, g, m, sum, first, nan);
        }
        // pass 1: p, probs, and the staged score of every class; bit 4i + j of `pass` marks class c0 + j of the lane's
        // i-th chunk as above the score threshold (i < 8: C <= 1024 and G = 32 give at most 8 chunks per lane)
        unsigned pass = 0u;
        for (int c0 = 4 * g, i = 0; in && c0 < p.C; c0 += 4 * G, ++i) {
            float v[4], o[4];
            load_chunk(x, c0, p.C, p.vec_in, v);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = c0 + j;
                if (p.logits) v[j] = __fdiv_rn(expf(__fsub_rn(v[j], m)), sum);
                const bool hit = part && c >= 1 && c < p.C && v[j] > p.sthr;
                pass |= hit ? 1u << (4 * i + j) : 0u;
                o[j] = hit ? v[j] : -INFINITY;
            }
            float* sc = p.st_scores + r * p.C + c0;
            if (p.vec_st) {
                *reinterpret_cast<float4*>(sc) = make_float4(o[0], o[1], o[2], o[3]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (c0 + j < p.C) sc[j] = o[j];
            }
            if (p.probs) {
                float* pr = p.probs + r * p.C + c0;
                if (p.vec_out) {
                    stg_f4_stream(reinterpret_cast<float4*>(pr), make_float4(v[0], v[1], v[2], v[3]));
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (c0 + j < p.C) stg_f1_stream(pr + j, v[j]);
                }
            }
        }
        if (!pass) continue;
        // pass 2: the boxes of the marked entries only; a box below min_size takes its entry out again
        const float4 roi = ldg_f4(p.rois + r);
        if (p.q == 1) {   // one box per row: every lane with a mark decodes it and writes the same bits
            const float4 bx = det_box(p, roi, r, 0);
            const bool keep = det_keeps_size(bx, p.min_size);
            if (keep) p.st_boxes[r] = bx;
            for (unsigned mk = keep ? 0u : pass; mk; mk &= mk - 1u) {
                const int bit = __ffs(mk) - 1;
                p.st_scores[r * p.C + 4 * g + (bit >> 2) * 4 * G + (bit & 3)] = -INFINITY;
            }
        } else {
            for (unsigned mk = pass; mk; mk &= mk - 1u) {
                const int bit = __ffs(mk) - 1;
                const int c = 4 * g + (bit >> 2) * 4 * G + (bit & 3);
                const float4 bx = det_box(p, roi, r, c);
                if (det_keeps_size(bx, p.min_size)) p.st_boxes[r * p.q + c] = bx;
                else p.st_scores[r * p.C + c] = -INFINITY;
            }
        }
    }
}

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// the staged scores and boxes, in front of the multi-class NMS's own layout
static size_t det_staged_bytes(int B, int S, int C, int q) {
    const size_t rows = (size_t)B * S;
    return align256(rows * C * 4) + align256(rows * q * 16);
}

// shape and configuration checks shared by the call and the reserve
static int det_check(const char* fn, int B, int S, const tfrpn_roi_det_cfg* cfg) {
    if (!cfg) return fail(TFRPN_ERR_BAD_ARG, "%s: null cfg", fn);
    if (B < 1 || S < 1) return fail(TFRPN_ERR_BAD_ARG, "%s: B = %d and S = %d must be >= 1", fn, B, S);
    const int C = cfg->num_classes, q = cfg->box_classes;
    if (C < 2) return fail(TFRPN_ERR_BAD_ARG, "%s: num_classes must be >= 2, got %d", fn, C);
    if (q != 1 && q != C) return fail(TFRPN_ERR_BAD_ARG, "%s: box_classes must be 1 or %d, got %d", fn, C, q);
    for (int i = 0; i < 4; ++i)
        if (!std::isfinite(cfg->variances[i])) return fail(TFRPN_ERR_BAD_ARG, "%s: variances must be finite", fn);
    if (std::isnan(cfg->max_log_scale)) return fail(TFRPN_ERR_BAD_ARG, "%s: max_log_scale is NaN", fn);
    if (cfg->score_input != 0 && cfg->score_input != 1)
        return fail(TFRPN_ERR_BAD_ARG, "%s: score_input must be 0 or 1, got %d", fn, cfg->score_input);
    if (int rc = mc_check_sizes(fn, B, S, C, &cfg->nms)) return rc;
    if (C > 1024 || S > 8192 || B > 65535)
        return fail(TFRPN_ERR_UNSUPPORTED, "%s: C = %d, S = %d, B = %d beyond 1024, 8192, 65535", fn, C, S, B);
    return 0;
}

template <int G>
int launch_det_scores(const RoiDetParams& p, cudaStream_t st) {
    const long long per_cta = (DET_THREADS / 32) * (32 / G);
    const int ctas = (int)std::max(1LL, std::min((p.rows + per_cta - 1) / per_cta, (long long)DET_MAX_CTAS));
    roi_det_score_kernel<G><<<ctas, DET_THREADS, 0, st>>>(p);
    TFRPN_AFTER_LAUNCH("roi_det_score_kernel");
    return 0;
}

}  // namespace tfrpn

using namespace tfrpn;

extern "C" size_t tfrpn_roi_head_detections_workspace_bytes(int B, int S, const tfrpn_roi_det_cfg* cfg) {
    if (!cfg || B < 1 || S < 1 || cfg->num_classes < 2) return 0;
    const int C = cfg->num_classes, q = cfg->box_classes;
    if (q != 1 && q != C) return 0;
    const size_t mc = tfrpn_nms_multiclass_workspace_bytes(B, S, C, &cfg->nms);
    return mc ? det_staged_bytes(B, S, C, q) + mc : 0;
}

extern "C" int tfrpn_reserve_roi_head_detections(tfrpn_handle h, int B, int S, const tfrpn_roi_det_cfg* cfg) {
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "reserve_roi_head_detections: null handle");
    if (int rc = det_check("reserve_roi_head_detections", B, S, cfg)) return rc;
    TFRPN_ENTER(h);
    char* ws;
    return ensure_workspace_prop(h, tfrpn_roi_head_detections_workspace_bytes(B, S, cfg), nullptr, &ws);
}

extern "C" int tfrpn_roi_head_detections(tfrpn_handle h, const float* rois, const int32_t* valid_or_null,
                                         const float* cls_scores, const float* box_deltas, int B, int S,
                                         const tfrpn_roi_det_cfg* cfg, float* out_boxes, float* out_scores,
                                         float* out_classes, int32_t* valid, int32_t* keep_idx_or_null,
                                         float* probs_or_null, tfrpn_stream s) {
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "roi_head_detections: null handle");
    if (!rois || !cls_scores || !box_deltas || !out_boxes || !out_scores || !out_classes || !valid)
        return fail(TFRPN_ERR_BAD_ARG, "roi_head_detections: null rois, cls_scores, box_deltas or output");
    if (int rc = det_check("roi_head_detections", B, S, cfg)) return rc;
    if (probs_or_null && cfg->score_input != 0)
        return fail(TFRPN_ERR_BAD_ARG, "roi_head_detections: probs are only written for logits input (score_input 0)");
    if (!aligned16(rois) || !aligned16(box_deltas) || !aligned16(out_boxes))
        return fail(TFRPN_ERR_MISALIGNED, "roi_head_detections: rois, box_deltas and out_boxes must be 16-byte aligned");
    const auto a4 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3u) == 0; };
    if (!a4(cls_scores) || !a4(probs_or_null))
        return fail(TFRPN_ERR_MISALIGNED, "roi_head_detections: cls_scores and probs must be 4-byte aligned");
    TFRPN_ENTER(h);
    TFRPN_CHECK_ON_DEVICE(h, rois, "roi_head_detections: rois");
    TFRPN_CHECK_ON_DEVICE(h, cls_scores, "roi_head_detections: cls_scores");
    cudaStream_t st = as_stream(s);
    const int C = cfg->num_classes, q = cfg->box_classes;
    // refuse before anything is launched what the NMS would refuse after the score kernel
    if (int rc = nms_mc_check_smem(h, B, C, cfg->nms.max_output_size_per_class)) return rc;
    char* ws = nullptr;
    if (int rc = ensure_workspace_prop(h, tfrpn_roi_head_detections_workspace_bytes(B, S, cfg), st, &ws)) return rc;

    RoiDetParams p = {};
    p.rois = reinterpret_cast<const float4*>(rois);
    p.valid = valid_or_null;
    p.x = cls_scores;
    p.deltas = reinterpret_cast<const float4*>(box_deltas);
    p.rows = (long long)B * S;
    p.S = S; p.C = C; p.q = q; p.logits = cfg->score_input == 0 ? 1 : 0; p.clip = cfg->clip;
    p.vec_in = C % 4 == 0 && aligned16(cls_scores);
    p.vec_out = C % 4 == 0 && aligned16(probs_or_null);
    p.vec_st = C % 4 == 0;
    p.var = make_float4(cfg->variances[0], cfg->variances[1], cfg->variances[2], cfg->variances[3]);
    p.max_log_scale = cfg->max_log_scale; p.min_size = cfg->min_size; p.sthr = cfg->nms.score_threshold;
    p.probs = probs_or_null;
    p.st_scores = reinterpret_cast<float*>(ws);
    p.st_boxes = reinterpret_cast<float4*>(ws + align256(p.rows * C * 4));
    int rc;
    switch (roi_row_lanes(C)) {
        case 4: rc = launch_det_scores<4>(p, st); break;
        case 8: rc = launch_det_scores<8>(p, st); break;
        case 16: rc = launch_det_scores<16>(p, st); break;
        default: rc = launch_det_scores<32>(p, st); break;
    }
    if (rc) return rc;
    return nms_mc_run(h, reinterpret_cast<const float*>(p.st_boxes), q, p.st_scores, B, S, C,
                      &cfg->nms, C - 1, 1, -INFINITY, det_staged_bytes(B, S, C, q), out_boxes, out_scores, out_classes,
                      valid, keep_idx_or_null, st);
}
