// losses.cu -- the RPN losses that consume the target-assignment outputs (SURVEY 8f rank 1):
//   cls_loss  utils/train_utils.py:146-161  BinaryCrossentropy over the entries with label != -1
//   reg_loss  utils/train_utils.py:163-185  Huber (delta 1) summed over the 4 coordinates of the
//             rows whose true delta is not all-zero, divided by max(1, #such rows)
// and, optionally, their gradients with respect to the predictions (what TF's autograd derives
// from the same ops), so that the pair can back a tf.custom_gradient.
//
//   L1 rpn_loss_partial_kernel  one pass over (labels, true deltas); the predictions are only
//                               read where a term exists (~3 % of the scores, ~1.5 % of the
//                               regression rows), so the kernel is HBM-bound on 20*B*N bytes.
//                               Per-element terms in float32 in the reference's op order;
//                               sums to float64 accuracy (float32 two-sum pairs inside a
//                               warp, doubles above), one partial per CTA; the last CTA
//                               sums the partials in a fixed order (deterministic) and divides.
//   L2 rpn_loss_grad_kernel     elementwise gradients, scaled by the counts L1 left on the device.
#include "roi_rows.cuh"

namespace tfrpn {

constexpr int LOSS_THREADS = 256;

// [TF-internal] Keras backend.binary_crossentropy(from_logits=False), TF 2.0.0:
//   p = clip_by_value(p, eps, 1 - eps); bce = t*log(p + eps); bce += (1 - t)*log(1 - p + eps); -bce
__device__ __forceinline__ float bce_term(float t, float p) {
    const float eps = 1e-7f;
    const float hi = __fsub_rn(1.0f, eps);
    p = fminf(fmaxf(p, eps), hi);
    float bce = __fmul_rn(t, logf(__fadd_rn(p, eps)));
    bce = __fadd_rn(bce, __fmul_rn(__fsub_rn(1.0f, t), logf(__fadd_rn(__fsub_rn(1.0f, p), eps))));
    return -bce;
}
// d bce / d p (clip_by_value passes the gradient where eps <= p <= 1 - eps)
__device__ __forceinline__ float bce_grad(float t, float p) {
    const float eps = 1e-7f;
    const float hi = __fsub_rn(1.0f, eps);
    if (!(p >= eps && p <= hi)) return 0.0f;
    const float a = __fdiv_rn(t, __fadd_rn(p, eps));
    const float b = __fdiv_rn(__fsub_rn(1.0f, t), __fadd_rn(__fsub_rn(1.0f, p), eps));
    return __fsub_rn(b, a);
}
// [TF-internal] keras huber_loss, TF 2.0.0 (elementwise; no mean over the last axis before 2.1):
//   e = pred - true; q = min(|e|, delta); lin = |e| - q; 0.5*q*q + delta*lin
__device__ __forceinline__ float huber_term(float t, float p, float delta) {
    const float ae = fabsf(__fsub_rn(p, t));
    const float q = fminf(ae, delta);
    const float lin = __fsub_rn(ae, q);
    return __fadd_rn(__fmul_rn(0.5f, __fmul_rn(q, q)), __fmul_rn(delta, lin));
}
__device__ __forceinline__ float huber_grad(float t, float p, float delta) {
    const float e = __fsub_rn(p, t);
    const float ae = fabsf(e);
    if (ae <= delta) return e;                       // minimum(x, y) routes the gradient to x when x <= y
    return e > 0.0f ? delta : -delta;
}

// per-CTA partial: the two sums as (hi, lo) float pairs and the two counts
struct LossPartial {
    float4 sums;   // reg.hi, reg.lo, cls.hi, cls.lo
    uint2 counts;  // n_pos, n_cls
    uint2 pad;
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// Non-tensor FP64 is slow on this part, so the hot path stays in float32: a thread adds its <= LOSS_EPT terms
// in float32, and the warp combines them as (hi, lo) pairs with the error-free two-sum, i.e. to float64-like
// accuracy without FP64 instructions.  Only one thread per CTA (and the last CTA) touches doubles.
__device__ __forceinline__ float2 pair_add(float2 a, float2 b) {
    const float s = __fadd_rn(a.x, b.x);
    const float bb = __fsub_rn(s, a.x);
    const float err = __fadd_rn(__fsub_rn(a.x, __fsub_rn(s, bb)), __fsub_rn(b.x, bb));
    return make_float2(s, __fadd_rn(err, __fadd_rn(a.y, b.y)));
}
__device__ __forceinline__ float2 warp_pair_sum(float v) {
    float2 p = make_float2(v, 0.0f);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        float2 q;
        q.x = __shfl_xor_sync(0xffffffffu, p.x, o);
        q.y = __shfl_xor_sync(0xffffffffu, p.y, o);
        p = pair_add(p, q);
    }
    return p;
}
__device__ __forceinline__ unsigned warp_sum(unsigned v) { return __reduce_add_sync(0xffffffffu, v); }

// One element (one anchor of one image) per thread and LOSS_EPT independent elements per thread, all of
// whose unconditional loads are issued before anything is consumed.  The last CTA to finish (a ticket in
// handle-owned memory, reset for the next call) sums the per-CTA partials in a fixed order, so the result
// does not depend on the order in which the CTAs ran.
constexpr int LOSS_EPT = 4;

__global__ void __launch_bounds__(LOSS_THREADS) rpn_loss_partial_kernel(
    const float4* __restrict__ true_deltas, const float4* __restrict__ pred_deltas,
    const float* __restrict__ true_labels, const float* __restrict__ pred_scores, long long total, float delta,
    LossPartial* __restrict__ partials, unsigned int* __restrict__ ticket, tfrpn_loss_out* __restrict__ out) {
    float reg = 0.0f, cls = 0.0f;
    unsigned npos = 0u, ncls = 0u;
    const long long base = (long long)blockIdx.x * (LOSS_THREADS * LOSS_EPT) + threadIdx.x;
    float tl[LOSS_EPT];
    float4 td[LOSS_EPT];
#pragma unroll
    for (int u = 0; u < LOSS_EPT; ++u) {
        const long long i = base + (long long)u * LOSS_THREADS;
        tl[u] = -1.0f;
        td[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < total) {
            if (true_labels) tl[u] = __ldg(true_labels + i);
            if (true_deltas) td[u] = ldg_f4_stream(true_deltas + i);
        }
    }
    // second wave of loads: the predictions, only where a term exists -- all issued before any is used
    // (a load inside each divergent branch would serialise LOSS_EPT memory latencies per warp)
    float ps[LOSS_EPT];
    float4 pp[LOSS_EPT];
    bool pos[LOSS_EPT];
#pragma unroll
    for (int u = 0; u < LOSS_EPT; ++u) {
        const long long i = base + (long long)u * LOSS_THREADS;
        const float4 t = td[u];
        pos[u] = t.x != 0.0f || t.y != 0.0f || t.z != 0.0f || t.w != 0.0f;      // train_utils.py:180
        ps[u] = 0.5f;
        pp[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (tl[u] != -1.0f) ps[u] = __ldg(pred_scores + i);                     // train_utils.py:156
        if (pos[u]) pp[u] = ldg_f4(pred_deltas + i);
    }
#pragma unroll
    for (int u = 0; u < LOSS_EPT; ++u) {
        if (tl[u] != -1.0f) {
            cls = __fadd_rn(cls, bce_term(tl[u], ps[u]));
            ++ncls;
        }
        if (pos[u]) {
            const float4 t = td[u], p = pp[u];
            float row = huber_term(t.x, p.x, delta);                      // reduce_sum(axis=-1), :178
            row = __fadd_rn(row, huber_term(t.y, p.y, delta));
            row = __fadd_rn(row, huber_term(t.z, p.z, delta));
            row = __fadd_rn(row, huber_term(t.w, p.w, delta));
            reg = __fadd_rn(reg, row);
            ++npos;
        }
    }
    __shared__ float2 s_reg[LOSS_THREADS / 32], s_cls[LOSS_THREADS / 32];
    __shared__ unsigned s_np[LOSS_THREADS / 32], s_nc[LOSS_THREADS / 32];
    __shared__ bool s_last;
    const float2 reg2 = warp_pair_sum(reg);
    const float2 cls2 = warp_pair_sum(cls);
    npos = warp_sum(npos);
    ncls = warp_sum(ncls);
    if (lane_id() == 0) {
        s_reg[warp_id()] = reg2; s_cls[warp_id()] = cls2; s_np[warp_id()] = npos; s_nc[warp_id()] = ncls;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float2 r = s_reg[0], c = s_cls[0];
        unsigned np = s_np[0], nc = s_nc[0];
        for (int w = 1; w < LOSS_THREADS / 32; ++w) {
            r = pair_add(r, s_reg[w]); c = pair_add(c, s_cls[w]); np += s_np[w]; nc += s_nc[w];
        }
        LossPartial p;
        p.sums = make_float4(r.x, r.y, c.x, c.y);
        p.counts = make_uint2(np, nc);
        p.pad = make_uint2(0u, 0u);
        partials[blockIdx.x] = p;
        __threadfence();
        s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    // the last CTA: fixed-order sum of all partials (thread t takes t, t+256, ...; then fixed trees)
    __threadfence();
    float2 r2 = make_float2(0.f, 0.f), c2 = make_float2(0.f, 0.f);
    unsigned long long np2 = 0ull, nc2 = 0ull;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += LOSS_THREADS) {
        const float4 q = __ldcg(&partials[i].sums);
        const uint2 k = __ldcg(&partials[i].counts);
        r2 = pair_add(r2, make_float2(q.x, q.y));
        c2 = pair_add(c2, make_float2(q.z, q.w));
        np2 += k.x; nc2 += k.y;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        float2 q;
        q.x = __shfl_xor_sync(0xffffffffu, r2.x, o); q.y = __shfl_xor_sync(0xffffffffu, r2.y, o);
        r2 = pair_add(r2, q);
        q.x = __shfl_xor_sync(0xffffffffu, c2.x, o); q.y = __shfl_xor_sync(0xffffffffu, c2.y, o);
        c2 = pair_add(c2, q);
        np2 += __shfl_xor_sync(0xffffffffu, np2, o);
        nc2 += __shfl_xor_sync(0xffffffffu, nc2, o);
    }
    __shared__ float2 t_reg[LOSS_THREADS / 32], t_cls[LOSS_THREADS / 32];
    __shared__ unsigned long long t_np[LOSS_THREADS / 32], t_nc[LOSS_THREADS / 32];
    if (lane_id() == 0) { t_reg[warp_id()] = r2; t_cls[warp_id()] = c2; t_np[warp_id()] = np2; t_nc[warp_id()] = nc2; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double R = 0.0, Cs = 0.0;
        unsigned long long NP = 0ull, NC = 0ull;
        for (int w = 0; w < LOSS_THREADS / 32; ++w) {
            R += (double)t_reg[w].x + (double)t_reg[w].y;
            Cs += (double)t_cls[w].x + (double)t_cls[w].y;
            NP += t_np[w]; NC += t_nc[w];
        }
        tfrpn_loss_out r;
        // :183-185  loc_loss / max(1, #pos);   :159-161  mean over the gathered entries (0/0 -> NaN, as TF)
        r.reg_loss = true_deltas ? (float)(R / (double)(NP > 0ull ? NP : 1ull)) : 0.0f;
        r.cls_loss = true_labels ? (float)(Cs / (double)NC) : 0.0f;
        r.n_pos = (int32_t)NP;
        r.n_cls = (int32_t)NC;
        *out = r;
        *ticket = 0u;     // ready for the next call on this handle
    }
}

constexpr int GRAD_EPT = 4;
__global__ void __launch_bounds__(LOSS_THREADS) rpn_loss_grad_kernel(
    const float4* __restrict__ true_deltas, const float4* __restrict__ pred_deltas,
    const float* __restrict__ true_labels, const float* __restrict__ pred_scores, long long total, float delta,
    const tfrpn_loss_out* __restrict__ res, float4* __restrict__ grad_deltas, float* __restrict__ grad_scores) {
    const long long base = (long long)blockIdx.x * (LOSS_THREADS * GRAD_EPT) + threadIdx.x;
    float tl[GRAD_EPT];
    float4 td[GRAD_EPT];
#pragma unroll
    for (int u = 0; u < GRAD_EPT; ++u) {
        const long long i = base + (long long)u * LOSS_THREADS;
        tl[u] = -1.0f;
        td[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < total) {
            if (grad_scores) tl[u] = __ldg(true_labels + i);
            if (grad_deltas) td[u] = ldg_f4_stream(true_deltas + i);
        }
    }
    float ps[GRAD_EPT];
    float4 pp[GRAD_EPT];
    bool pos[GRAD_EPT];
#pragma unroll
    for (int u = 0; u < GRAD_EPT; ++u) {   // the predictions, only where a term exists, all in flight together
        const long long i = base + (long long)u * LOSS_THREADS;
        const float4 t = td[u];
        pos[u] = t.x != 0.0f || t.y != 0.0f || t.z != 0.0f || t.w != 0.0f;
        ps[u] = 0.5f;
        pp[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (tl[u] != -1.0f) ps[u] = __ldg(pred_scores + i);
        if (pos[u]) pp[u] = ldg_f4(pred_deltas + i);
    }
    const float inv_pos = __fdiv_rn(1.0f, (float)max(res->n_pos, 1));
    const float inv_cls = __fdiv_rn(1.0f, (float)res->n_cls);
#pragma unroll
    for (int u = 0; u < GRAD_EPT; ++u) {
        const long long i = base + (long long)u * LOSS_THREADS;
        if (i >= total) continue;
        if (grad_scores) {
            float g = 0.0f;
            if (tl[u] != -1.0f) g = __fmul_rn(bce_grad(tl[u], ps[u]), inv_cls);
            stg_f1_stream(grad_scores + i, g);
        }
        if (grad_deltas) {
            const float4 t = td[u], p = pp[u];
            float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
            if (pos[u])
                g = make_float4(__fmul_rn(huber_grad(t.x, p.x, delta), inv_pos), __fmul_rn(huber_grad(t.y, p.y, delta), inv_pos),
                                __fmul_rn(huber_grad(t.z, p.z, delta), inv_pos), __fmul_rn(huber_grad(t.w, p.w, delta), inv_pos));
            stg_f4_stream(grad_deltas + i, g);
        }
    }
}

size_t losses_workspace_bytes(long long total) {
    return (size_t)((total + LOSS_THREADS * LOSS_EPT - 1) / (LOSS_THREADS * LOSS_EPT) + 1) * sizeof(LossPartial) + 256;
}

// ---- the second stage's box-head losses (tfrpn_roi_head_losses) ------------------------------------------------------
//   L1 roi_loss_partial_kernel<G>  a group of G lanes per row: the lanes stride over the row's logits in chunks of 4
//                                  classes (lane g takes chunks g, g + G, ...; a float4 load where the row is 16-byte
//                                  aligned, 4 scalar loads otherwise: the same values in the same order) for the max,
//                                  then the exp-sum and the argmax; lane 0 of the group adds the row's terms.  The box
//                                  deltas are read for fg rows only, 16 bytes per row.  The sums and counts go through
//                                  the partial / last-CTA scheme of rpn_loss_partial_kernel (ticket word 1).
//   L2 roi_loss_grad_kernel<G>     recomputes each row's max and exp-sum with the same code, so e_c / s has the bits
//                                  L1 saw, and writes both gradients everywhere, scaled by the counts L1 left in out.
// G (4, 8, 16 or 32) is the smallest that covers the ceil(C / 4) chunks, 32 above: C = 21 takes 8 lanes per row, C = 81
// takes 32.  The grid is capped at a constant, so the partition of the sums depends on the shape alone.
constexpr int ROI_LOSS_MAX_CTAS = 1184;   // 8 CTAs of 256 threads on each of 148 SMs

struct RoiLossPartial {
    float4 sums;    // cls.hi, cls.lo, reg.hi, reg.lo
    uint4 counts;   // n_rows, n_fg, n_correct, n_fg_correct
};

__device__ __forceinline__ float huber_row(float4 t, float4 p, float delta) {   // reduce_sum over the 4 coordinates
    float row = huber_term(t.x, p.x, delta);
    row = __fadd_rn(row, huber_term(t.y, p.y, delta));
    row = __fadd_rn(row, huber_term(t.z, p.z, delta));
    return __fadd_rn(row, huber_term(t.w, p.w, delta));
}

template <int G>
__global__ void __launch_bounds__(LOSS_THREADS) roi_loss_partial_kernel(
    const float* __restrict__ logits, const float4* __restrict__ box_deltas, const int* __restrict__ labels,
    const float4* __restrict__ targets, long long rows, int C, int q, float delta, int norm_rows, bool vec,
    RoiLossPartial* __restrict__ partials, unsigned int* __restrict__ ticket, tfrpn_roi_loss_out* __restrict__ out) {
    constexpr int RPW = 32 / G;   // rows per warp and pass
    const int g = lane_id() % G;
    float2 cls = make_float2(0.f, 0.f), reg = make_float2(0.f, 0.f);
    unsigned n_rows = 0u, n_fg = 0u, n_ok = 0u, n_fg_ok = 0u;
    const long long stride = (long long)gridDim.x * (LOSS_THREADS / 32) * RPW;
    for (long long r0 = ((long long)blockIdx.x * (LOSS_THREADS / 32) + warp_id()) * RPW; r0 < rows; r0 += stride) {
        const long long r = r0 + lane_id() / G;
        const int label = r < rows ? __ldg(labels + r) : -1;
        const bool part = label >= 0 && label < C;
        const float* x = logits + (part ? r : 0) * C;
        float m, s;
        int first;
        bool nan;
        roi_row_stats<G>(x, part ? C : 0, vec, g, m, s, first, nan);
        if (part && g == 0) {
            const float term = __fsub_rn(logf(s), __fsub_rn(__ldg(x + label), m));
            const unsigned ok = (!nan && first == label) ? 1u : 0u;
            cls = pair_add(cls, make_float2(term, 0.0f));
            ++n_rows;
            n_ok += ok;
            if (label >= 1) {
                const float4 t = ldg_f4(targets + r);
                const float4 p = ldg_f4(box_deltas + r * q + (q == C ? label : 0));
                reg = pair_add(reg, make_float2(huber_row(t, p, delta), 0.0f));
                ++n_fg;
                n_fg_ok += ok;
            }
        }
    }
    __shared__ float2 s_cls[LOSS_THREADS / 32], s_reg[LOSS_THREADS / 32];
    __shared__ uint4 s_n[LOSS_THREADS / 32];
    __shared__ bool s_last;
    const float2 cls2 = warp_pair_sum(cls.x), cls2lo = warp_pair_sum(cls.y);
    const float2 reg2 = warp_pair_sum(reg.x), reg2lo = warp_pair_sum(reg.y);
    const uint4 n = make_uint4(warp_sum(n_rows), warp_sum(n_fg), warp_sum(n_ok), warp_sum(n_fg_ok));
    if (lane_id() == 0) {
        s_cls[warp_id()] = pair_add(cls2, cls2lo);
        s_reg[warp_id()] = pair_add(reg2, reg2lo);
        s_n[warp_id()] = n;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float2 c = s_cls[0], rg = s_reg[0];
        uint4 k = s_n[0];
        for (int w = 1; w < LOSS_THREADS / 32; ++w) {
            c = pair_add(c, s_cls[w]);
            rg = pair_add(rg, s_reg[w]);
            k.x += s_n[w].x; k.y += s_n[w].y; k.z += s_n[w].z; k.w += s_n[w].w;
        }
        RoiLossPartial p;
        p.sums = make_float4(c.x, c.y, rg.x, rg.y);
        p.counts = k;
        partials[blockIdx.x] = p;
        __threadfence();
        s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    // the last CTA: the partials in a fixed order (grid <= ROI_LOSS_MAX_CTAS, so one warp walks them), then doubles
    __threadfence();
    if (threadIdx.x >= 32) return;
    float2 c2 = make_float2(0.f, 0.f), r2 = make_float2(0.f, 0.f);
    unsigned long long k2[4] = {0ull, 0ull, 0ull, 0ull};
    for (int i = lane_id(); i < (int)gridDim.x; i += 32) {
        const float4 v = __ldcg(&partials[i].sums);
        const uint4 k = __ldcg(&partials[i].counts);
        c2 = pair_add(c2, make_float2(v.x, v.y));
        r2 = pair_add(r2, make_float2(v.z, v.w));
        k2[0] += k.x; k2[1] += k.y; k2[2] += k.z; k2[3] += k.w;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        float2 t;
        t.x = __shfl_xor_sync(0xffffffffu, c2.x, o); t.y = __shfl_xor_sync(0xffffffffu, c2.y, o);
        c2 = pair_add(c2, t);
        t.x = __shfl_xor_sync(0xffffffffu, r2.x, o); t.y = __shfl_xor_sync(0xffffffffu, r2.y, o);
        r2 = pair_add(r2, t);
#pragma unroll
        for (int j = 0; j < 4; ++j) k2[j] += __shfl_xor_sync(0xffffffffu, k2[j], o);
    }
    if (lane_id() == 0) {
        const double Cs = (double)c2.x + (double)c2.y, R = (double)r2.x + (double)r2.y;
        const unsigned long long norm = norm_rows ? k2[0] : k2[1];
        tfrpn_roi_loss_out res;
        res.cls_loss = (float)(Cs / (double)k2[0]);                      // 0/0 -> NaN
        res.reg_loss = (float)(R / (double)(norm > 0ull ? norm : 1ull));
        res.n_rows = (int32_t)k2[0];
        res.n_fg = (int32_t)k2[1];
        res.n_correct = (int32_t)k2[2];
        res.n_fg_correct = (int32_t)k2[3];
        res.reserved[0] = res.reserved[1] = 0;
        *out = res;
        *ticket = 0u;     // ready for the next call on this handle
    }
}

template <int G>
__global__ void __launch_bounds__(LOSS_THREADS) roi_loss_grad_kernel(
    const float* __restrict__ logits, const float4* __restrict__ box_deltas, const int* __restrict__ labels,
    const float4* __restrict__ targets, long long rows, int C, int q, float delta, int norm_rows, bool vec_in,
    bool vec_out, const tfrpn_roi_loss_out* __restrict__ res, const float* __restrict__ scale,
    float* __restrict__ grad_logits, float4* __restrict__ grad_deltas) {
    constexpr int RPW = 32 / G;
    const int g = lane_id() % G;
    const int n_rows = res->n_rows;
    const float inv_rows = __fdiv_rn(1.0f, (float)n_rows);
    const float inv_reg = __fdiv_rn(1.0f, (float)max(norm_rows ? n_rows : res->n_fg, 1));
    const float s_cls = scale ? scale[0] : 1.0f, s_reg = scale ? scale[1] : 1.0f;
    const long long stride = (long long)gridDim.x * (LOSS_THREADS / 32) * RPW;
    for (long long r0 = ((long long)blockIdx.x * (LOSS_THREADS / 32) + warp_id()) * RPW; r0 < rows; r0 += stride) {
        const long long r = r0 + lane_id() / G;
        const bool in = r < rows;
        const int label = in ? __ldg(labels + r) : -1;
        const bool part = label >= 0 && label < C;
        if (grad_logits) {
            const float* x = logits + (part ? r : 0) * C;
            float m, s;
            int first;
            bool nan;
            roi_row_stats<G>(x, part ? C : 0, vec_in, g, m, s, first, nan);
            float* gx = grad_logits + (in ? r : 0) * C;
            for (int c0 = 4 * g; in && c0 < C; c0 += 4 * G) {
                float v[4] = {0.f, 0.f, 0.f, 0.f};
                if (part) {
                    load_chunk(x, c0, C, vec_in, v);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float p = __fdiv_rn(expf(__fsub_rn(v[j], m)), s);
                        v[j] = __fmul_rn(__fmul_rn(__fsub_rn(p, c0 + j == label ? 1.0f : 0.0f), inv_rows), s_cls);
                    }
                }
                if (vec_out) {
                    stg_f4_stream(reinterpret_cast<float4*>(gx + c0), make_float4(v[0], v[1], v[2], v[3]));
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (c0 + j < C) stg_f1_stream(gx + c0 + j, v[j]);
                }
            }
        }
        if (grad_deltas && in) {
            float4 gsel = make_float4(0.f, 0.f, 0.f, 0.f);
            int sel = -1;
            if (label >= 1 && label < C) {
                sel = q == C ? label : 0;
                const float4 t = ldg_f4(targets + r), p = ldg_f4(box_deltas + r * q + sel);
                gsel = make_float4(__fmul_rn(__fmul_rn(huber_grad(t.x, p.x, delta), inv_reg), s_reg),
                                   __fmul_rn(__fmul_rn(huber_grad(t.y, p.y, delta), inv_reg), s_reg),
                                   __fmul_rn(__fmul_rn(huber_grad(t.z, p.z, delta), inv_reg), s_reg),
                                   __fmul_rn(__fmul_rn(huber_grad(t.w, p.w, delta), inv_reg), s_reg));
            }
            for (int k = g; k < q; k += G)
                stg_f4_stream(grad_deltas + r * q + k, k == sel ? gsel : make_float4(0.f, 0.f, 0.f, 0.f));
        }
    }
}

}  // namespace tfrpn

using namespace tfrpn;

extern "C" int tfrpn_rpn_losses(tfrpn_handle h, const float* true_deltas, const float* pred_deltas,
                                const float* true_labels, const float* pred_scores, int B, int N, float huber_delta,
                                tfrpn_loss_out* out, float* grad_deltas_or_null, float* grad_scores_or_null,
                                tfrpn_stream s) {
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "rpn_losses: null handle");
    if (!out) return fail(TFRPN_ERR_BAD_ARG, "rpn_losses: out is null");
    if ((true_deltas != nullptr) != (pred_deltas != nullptr) || (true_labels != nullptr) != (pred_scores != nullptr))
        return fail(TFRPN_ERR_BAD_ARG, "rpn_losses: true / predicted tensors must be given in pairs");
    if (!true_deltas && !true_labels) return fail(TFRPN_ERR_BAD_ARG, "rpn_losses: nothing to do");
    if ((grad_deltas_or_null && !true_deltas) || (grad_scores_or_null && !true_labels))
        return fail(TFRPN_ERR_BAD_ARG, "rpn_losses: gradient requested for a loss that is not computed");
    if (B < 0 || N < 0) return fail(TFRPN_ERR_BAD_ARG, "rpn_losses: negative shape");
    if (!(huber_delta > 0.0f)) return fail(TFRPN_ERR_BAD_ARG, "rpn_losses: huber_delta must be > 0");
    if (true_deltas && (!aligned16(true_deltas) || !aligned16(pred_deltas) || (grad_deltas_or_null && !aligned16(grad_deltas_or_null))))
        return fail(TFRPN_ERR_MISALIGNED, "rpn_losses: delta tensors must be 16-byte aligned");
    TFRPN_ENTER(h);
    TFRPN_CHECK_ON_DEVICE(h, out, "rpn_losses: out");
    cudaStream_t st = as_stream(s);
    const long long total = (long long)B * N;
    if (total > (1LL << 38)) return fail(TFRPN_ERR_UNSUPPORTED, "rpn_losses: tensor too large");
    char* ws = nullptr;
    if (int rc = ensure_workspace(h, losses_workspace_bytes(total), st, &ws)) return rc;
    LossPartial* partials = reinterpret_cast<LossPartial*>(ws);
    if (!h->ticket) return fail(TFRPN_ERR_CUDA, "rpn_losses: the handle has no device counter");
    const long long want = (total + LOSS_THREADS * LOSS_EPT - 1) / (LOSS_THREADS * LOSS_EPT);
    const int ctas = (int)(want < 1 ? 1 : want);
    const float4* td = reinterpret_cast<const float4*>(true_deltas);
    const float4* pd = reinterpret_cast<const float4*>(pred_deltas);
    prof_begin(h, TFRPN_K_LOSS, st);
    rpn_loss_partial_kernel<<<ctas, LOSS_THREADS, 0, st>>>(td, pd, true_labels, pred_scores, total, huber_delta, partials,
                                                           h->ticket, out);
    prof_end(h, st);
    TFRPN_AFTER_LAUNCH("rpn_loss_partial_kernel");
    if ((grad_deltas_or_null || grad_scores_or_null) && total > 0) {
        const int gctas = (int)((total + LOSS_THREADS * GRAD_EPT - 1) / (LOSS_THREADS * GRAD_EPT));
        rpn_loss_grad_kernel<<<gctas, LOSS_THREADS, 0, st>>>(td, pd, true_labels, pred_scores, total, huber_delta, out,
                                                            reinterpret_cast<float4*>(grad_deltas_or_null),
                                                            grad_scores_or_null);
        TFRPN_AFTER_LAUNCH("rpn_loss_grad_kernel");
    }
    return 0;
}

namespace {
long long roi_loss_ctas(long long rows, int G) {
    const long long per_cta = (LOSS_THREADS / 32) * (32 / G);
    return std::max(1LL, std::min((rows + per_cta - 1) / per_cta, (long long)ROI_LOSS_MAX_CTAS));
}

template <int G>
int launch_roi_losses(const float* logits, const float4* bd, const int32_t* labels, const float4* td, long long rows,
                      const tfrpn_roi_loss_cfg& cfg, char* ws, unsigned int* ticket, tfrpn_roi_loss_out* out,
                      const float* scale, float* grad_logits, float4* grad_deltas, cudaStream_t st) {
    const int C = cfg.num_classes, q = cfg.box_classes;
    const int ctas = (int)roi_loss_ctas(rows, G);
    const bool vec_in = C % 4 == 0 && aligned16(logits);
    roi_loss_partial_kernel<G><<<ctas, LOSS_THREADS, 0, st>>>(logits, bd, labels, td, rows, C, q, cfg.huber_delta,
                                                              cfg.reg_normalizer, vec_in,
                                                              reinterpret_cast<RoiLossPartial*>(ws), ticket, out);
    TFRPN_AFTER_LAUNCH("roi_loss_partial_kernel");
    if ((grad_logits || grad_deltas) && rows > 0) {
        const bool vec_out = C % 4 == 0 && aligned16(grad_logits);
        roi_loss_grad_kernel<G><<<ctas, LOSS_THREADS, 0, st>>>(logits, bd, labels, td, rows, C, q, cfg.huber_delta,
                                                               cfg.reg_normalizer, vec_in, vec_out, out, scale,
                                                               grad_logits, grad_deltas);
        TFRPN_AFTER_LAUNCH("roi_loss_grad_kernel");
    }
    return 0;
}
}  // namespace

extern "C" int tfrpn_roi_head_losses(tfrpn_handle h, const float* cls_logits, const float* box_deltas,
                                     const int32_t* labels, const float* target_deltas, int B, int S,
                                     const tfrpn_roi_loss_cfg* cfg, tfrpn_roi_loss_out* out,
                                     const float* grad_scale_or_null, float* grad_logits_or_null,
                                     float* grad_deltas_or_null, tfrpn_stream s) {
    if (!h) return fail(TFRPN_ERR_BAD_ARG, "roi_head_losses: null handle");
    if (!cls_logits || !box_deltas || !labels || !target_deltas || !cfg || !out)
        return fail(TFRPN_ERR_BAD_ARG, "roi_head_losses: null cls_logits, box_deltas, labels, target_deltas, cfg or out");
    if (B < 0 || S < 0) return fail(TFRPN_ERR_BAD_ARG, "roi_head_losses: negative shape");
    const int C = cfg->num_classes, q = cfg->box_classes;
    if (C < 2) return fail(TFRPN_ERR_BAD_ARG, "roi_head_losses: num_classes must be >= 2, got %d", C);
    if (q != 1 && q != C) return fail(TFRPN_ERR_BAD_ARG, "roi_head_losses: box_classes must be 1 or %d, got %d", C, q);
    if (!(cfg->huber_delta > 0.0f)) return fail(TFRPN_ERR_BAD_ARG, "roi_head_losses: huber_delta must be > 0");
    if (cfg->reg_normalizer != 0 && cfg->reg_normalizer != 1)
        return fail(TFRPN_ERR_BAD_ARG, "roi_head_losses: reg_normalizer must be 0 or 1, got %d", cfg->reg_normalizer);
    if (C > 1024 || S > 8192 || B > 65535)
        return fail(TFRPN_ERR_UNSUPPORTED, "roi_head_losses: C = %d, S = %d, B = %d beyond 1024, 8192, 65535", C, S, B);
    if (!aligned16(box_deltas) || !aligned16(target_deltas) || (grad_deltas_or_null && !aligned16(grad_deltas_or_null)))
        return fail(TFRPN_ERR_MISALIGNED, "roi_head_losses: box_deltas, target_deltas and grad_deltas must be 16-byte aligned");
    const auto a4 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3u) == 0; };
    if (!a4(cls_logits) || !a4(labels) || !a4(grad_logits_or_null))
        return fail(TFRPN_ERR_MISALIGNED, "roi_head_losses: cls_logits, labels and grad_logits must be 4-byte aligned");
    TFRPN_ENTER(h);
    TFRPN_CHECK_ON_DEVICE(h, out, "roi_head_losses: out");
    TFRPN_CHECK_ON_DEVICE(h, cls_logits, "roi_head_losses: cls_logits");
    cudaStream_t st = as_stream(s);
    const long long rows = (long long)B * S;
    const int G = roi_row_lanes(C);
    char* ws = nullptr;
    if (int rc = ensure_workspace(h, (size_t)roi_loss_ctas(rows, G) * sizeof(RoiLossPartial) + 256, st, &ws)) return rc;
    if (!h->ticket) return fail(TFRPN_ERR_CUDA, "roi_head_losses: the handle has no device counter");
    const float4* bd = reinterpret_cast<const float4*>(box_deltas);
    const float4* td = reinterpret_cast<const float4*>(target_deltas);
    float4* gd = reinterpret_cast<float4*>(grad_deltas_or_null);
    unsigned int* ticket = h->ticket + 1;
    switch (G) {
        case 4: return launch_roi_losses<4>(cls_logits, bd, labels, td, rows, *cfg, ws, ticket, out, grad_scale_or_null,
                                            grad_logits_or_null, gd, st);
        case 8: return launch_roi_losses<8>(cls_logits, bd, labels, td, rows, *cfg, ws, ticket, out, grad_scale_or_null,
                                            grad_logits_or_null, gd, st);
        case 16: return launch_roi_losses<16>(cls_logits, bd, labels, td, rows, *cfg, ws, ticket, out, grad_scale_or_null,
                                              grad_logits_or_null, gd, st);
        default: return launch_roi_losses<32>(cls_logits, bd, labels, td, rows, *cfg, ws, ticket, out, grad_scale_or_null,
                                              grad_logits_or_null, gd, st);
    }
}
