// roi_rows.cuh -- the per-row softmax statistics of the box head's class scores, shared by the box-head losses
// (losses.cu) and the box-head detections (roi_detect.cu), so both see the same max, exp-sum and therefore the same
// probability bits.  A group of G lanes (4, 8, 16 or 32) owns one row; lane g takes the 4-class chunks g, g + G, ...
#pragma once

#include "common.cuh"

namespace tfrpn {

template <int G>
__device__ __forceinline__ float group_max(float v) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
template <int G>
__device__ __forceinline__ float group_sum(float v) {   // a butterfly: every lane of the group gets the same bits
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
template <int G>
__device__ __forceinline__ int group_min(int v) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// classes c0 .. c0 + 3 of a row (those < C); vec: C % 4 == 0 and the row is 16-byte aligned
__device__ __forceinline__ void load_chunk(const float* __restrict__ x, int c0, int C, bool vec, float v[4]) {
    if (vec) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(x + c0));
        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
        return;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = c0 + j < C ? __ldg(x + c0 + j) : 0.0f;
}

// One row's softmax statistics, the same on every lane of the group: m = max (NaN ignored), s = sum of
// expf(x_c - m) (NaN when any logit is NaN), first = the first c with x_c == m, nan = any logit is NaN.  C_eff = 0
// (a row that takes no part) reads nothing but keeps the group in step with the shuffles.
template <int G>
__device__ __forceinline__ void roi_row_stats(const float* __restrict__ x, int C_eff, bool vec, int g, float& m,
                                              float& s, int& first, bool& nan) {
    float mx = -INFINITY;
    bool bad = false;
    for (int c0 = 4 * g; c0 < C_eff; c0 += 4 * G) {
        float v[4];
        load_chunk(x, c0, C_eff, vec, v);
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (c0 + j < C_eff) { bad |= isnan(v[j]); mx = fmaxf(mx, v[j]); }
    }
    m = group_max<G>(mx);
    nan = group_min<G>(bad ? 0 : 1) == 0;
    float sum = 0.0f;
    int arg = C_eff;
    for (int c0 = 4 * g; c0 < C_eff; c0 += 4 * G) {
        float v[4];
        load_chunk(x, c0, C_eff, vec, v);
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (c0 + j < C_eff) {
                sum = __fadd_rn(sum, expf(__fsub_rn(v[j], m)));
                if (v[j] == m && arg == C_eff) arg = c0 + j;
            }
    }
    s = group_sum<G>(sum);
    first = group_min<G>(arg);
}

// lanes per row: the smallest G that covers the ceil(C / 4) chunks, 32 above (C = 21 takes 8, C = 81 takes 32)
inline int roi_row_lanes(int C) {
    const int chunks = (C + 3) / 4;
    return chunks <= 4 ? 4 : chunks <= 8 ? 8 : chunks <= 16 ? 16 : 32;
}

}  // namespace tfrpn
