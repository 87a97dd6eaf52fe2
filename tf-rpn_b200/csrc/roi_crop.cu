// roi_crop.cu -- tf.image.crop_and_resize (bilinear) and its image gradient: tfrpn_crop_and_resize and
// tfrpn_crop_and_resize_grad_image, definition in include/tfrpn.h.
//   crop_kernel       one CTA per (box, output row): the row's and the columns' sample coordinates once, then the
//                     threads run over (column, channel) in float4 (C % 4 == 0) or scalar channels
//   crop_grad_kernel  one CTA per (image, 4 x 4 pixel tile, channel slice), one warp per pixel, a lane per channel
//                     group: a gather over the image's boxes in ascending order with no atomics, so every gradient
//                     element is the float32 sum of its terms in the order (box, y, x, term) of TF's CPU loop
#include "common.cuh"

namespace tfrpn {
namespace {

constexpr int CR_MAX_C = 4096, CR_MAX_CROP = 32, CR_MAX_HW = 8192, CR_MAX_M = 1 << 24;
constexpr int CR_THREADS = 128;                 // crop_kernel
constexpr int CG_TILE = 4, CG_THREADS = 512;    // crop_grad_kernel: 16 warps = the 4 x 4 pixels of a tile

struct CropArgs {
    const float* src;          // image (forward) | grad_out (gradient)
    const float4* boxes;       // (M,4) [y1,x1,y2,x2]
    const int32_t* box_index;  // (M,) or NULL: box m belongs to image m / per_image
    float* dst;                // out (forward) | grad_image (gradient)
    int B, H, W, C, M, ch, cw, per_image;
    float extrapolation;
};

__device__ __forceinline__ int image_of(const CropArgs& p, int m) {
    return p.box_index ? p.box_index[m] : m / p.per_image;
}

// The sample grid of one box along one axis of length L with n samples (crop_and_resize_op.cc, bilinear):
//   n > 1:  in(i) = lo*(L-1) + i*s,  s = (hi-lo)*(L-1)/(n-1), every operation in float32;
//   n == 1: in = 0.5*(lo+hi)*(L-1): lo+hi in float32, the rest in float64 (0.5 is a double literal), rounded once.
struct Axis {
    float a, s, lmax;
    int n;
};
__device__ __forceinline__ Axis make_axis(float lo, float hi, int L, int n) {
    Axis ax;
    ax.n = n;
    ax.lmax = (float)(L - 1);
    if (n > 1) {
        ax.a = __fmul_rn(lo, ax.lmax);
        ax.s = __fdiv_rn(__fmul_rn(__fsub_rn(hi, lo), ax.lmax), (float)(n - 1));
    } else {
        ax.a = __double2float_rn(__dmul_rn(__dmul_rn(0.5, (double)__fadd_rn(lo, hi)), (double)(L - 1)));
        ax.s = 0.0f;
    }
    return ax;
}
__device__ __forceinline__ float sample_at(const Axis& ax, int i) {
    return ax.n > 1 ? __fadd_rn(ax.a, __fmul_rn((float)i, ax.s)) : ax.a;
}
// a sample inside [0, L-1] is interpolated, any other (NaN included) extrapolated
__device__ __forceinline__ bool inside(float v, float lmax) { return v >= 0.0f && v <= lmax; }

__device__ __forceinline__ float lerp_tf(float a, float b, float t) { return __fadd_rn(a, __fmul_rn(__fsub_rn(b, a), t)); }

template <int VEC>
struct Vec;
template <>
struct Vec<4> {
    using T = float4;
};
template <>
struct Vec<1> {
    using T = float;
};
__device__ __forceinline__ float4 ld_vec(const float4* p) { return __ldg(p); }
__device__ __forceinline__ float ld_vec(const float* p) { return __ldg(p); }
__device__ __forceinline__ void st_vec(float4* p, float4 v) { stg_f4_stream(p, v); }
__device__ __forceinline__ void st_vec(float* p, float v) { stg_f1_stream(p, v); }
__device__ __forceinline__ float4 splat(float v, float4*) { return make_float4(v, v, v, v); }
__device__ __forceinline__ float splat(float v, float*) { return v; }
__device__ __forceinline__ float4 bilinear(float4 tl, float4 tr, float4 bl, float4 br, float xl, float yl) {
    return make_float4(lerp_tf(lerp_tf(tl.x, tr.x, xl), lerp_tf(bl.x, br.x, xl), yl),
                       lerp_tf(lerp_tf(tl.y, tr.y, xl), lerp_tf(bl.y, br.y, xl), yl),
                       lerp_tf(lerp_tf(tl.z, tr.z, xl), lerp_tf(bl.z, br.z, xl), yl),
                       lerp_tf(lerp_tf(tl.w, tr.w, xl), lerp_tf(bl.w, br.w, xl), yl));
}
__device__ __forceinline__ float bilinear(float tl, float tr, float bl, float br, float xl, float yl) {
    return lerp_tf(lerp_tf(tl, tr, xl), lerp_tf(bl, br, xl), yl);
}

template <int VEC>
__global__ void __launch_bounds__(CR_THREADS) crop_kernel(CropArgs p) {
    using V = typename Vec<VEC>::T;
    __shared__ int s_left[CR_MAX_CROP], s_right[CR_MAX_CROP];
    __shared__ float s_xlerp[CR_MAX_CROP];
    const int m = blockIdx.x / p.ch, y = blockIdx.x - m * p.ch;
    const float4 bx = p.boxes[m];
    const int b = image_of(p, m);
    if (threadIdx.x < p.cw) {
        const Axis ax = make_axis(bx.y, bx.w, p.W, p.cw);
        const float u = sample_at(ax, threadIdx.x);
        const bool ok = inside(u, ax.lmax);
        const int l = (int)floorf(u);
        s_left[threadIdx.x] = ok ? l : -1;
        s_right[threadIdx.x] = ok ? (int)ceilf(u) : -1;
        s_xlerp[threadIdx.x] = __fsub_rn(u, (float)l);
    }
    const Axis ay = make_axis(bx.x, bx.z, p.H, p.ch);
    const float v = sample_at(ay, y);
    const bool bad = b < 0 || b >= p.B;
    const bool row_ok = inside(v, ay.lmax);
    const int top = row_ok ? (int)floorf(v) : 0, bottom = row_ok ? (int)ceilf(v) : 0;
    const float ylerp = __fsub_rn(v, (float)top);
    __syncthreads();
    const int CV = p.C / VEC;
    const V* img_top = reinterpret_cast<const V*>(p.src + (size_t)((long long)(bad ? 0 : b) * p.H + top) * p.W * p.C);
    const V* img_bot = reinterpret_cast<const V*>(p.src + (size_t)((long long)(bad ? 0 : b) * p.H + bottom) * p.W * p.C);
    V* out = reinterpret_cast<V*>(p.dst + (size_t)blockIdx.x * p.cw * p.C);
    const V fill = splat(bad ? __int_as_float(0x7fc00000) : p.extrapolation, (V*)nullptr);
    int x = 0, cv = threadIdx.x;
    while (cv >= CV) { cv -= CV; ++x; }
    for (; x < p.cw; ) {
        V r = fill;
        const int left = s_left[x];
        if (!bad && row_ok && left >= 0) {
            const size_t lo = (size_t)left * CV + cv, ro = (size_t)s_right[x] * CV + cv;
            r = bilinear(ld_vec(img_top + lo), ld_vec(img_top + ro), ld_vec(img_bot + lo), ld_vec(img_bot + ro),
                         s_xlerp[x], ylerp);
        }
        st_vec(out + (size_t)x * CV + cv, r);
        cv += CR_THREADS;
        while (cv >= CV) { cv -= CV; ++x; }
    }
}

// First and last sample i whose floor or ceil is tile line t0 + r (r < 4), as byte r of lo / hi (lo 255, hi 0 when
// none).  The samples are monotone in i, so those touching one line are contiguous.
__device__ __forceinline__ bool line_ranges(const Axis& ax, int t0, uint32_t& lo_bytes, uint32_t& hi_bytes) {
    int lo[CG_TILE], hi[CG_TILE];
#pragma unroll
    for (int r = 0; r < CG_TILE; ++r) { lo[r] = 255; hi[r] = 0; }
    bool any = false;
    for (int i = 0; i < ax.n; ++i) {
        const float v = sample_at(ax, i);
        if (!inside(v, ax.lmax)) continue;
        const int f = (int)floorf(v) - t0, c = (int)ceilf(v) - t0;
#pragma unroll
        for (int r = 0; r < CG_TILE; ++r) {
            if (f == r || c == r) {
                lo[r] = min(lo[r], i);
                hi[r] = i;
                any = true;
            }
        }
    }
    lo_bytes = hi_bytes = 0;
#pragma unroll
    for (int r = 0; r < CG_TILE; ++r) {
        lo_bytes |= (uint32_t)lo[r] << (8 * r);
        hi_bytes |= (uint32_t)hi[r] << (8 * r);
    }
    return any;
}

template <int VEC>
__device__ __forceinline__ void add_terms(float (&acc)[VEC], const float* g, float wtop, float ylerp, float wleft,
                                          float xlerp, bool tl, bool tr, bool bl, bool br) {
    float gv[VEC];
    if constexpr (VEC == 4) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(g));
        gv[0] = t.x; gv[1] = t.y; gv[2] = t.z; gv[3] = t.w;
    } else {
        gv[0] = __ldg(g);
    }
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
        const float dtop = __fmul_rn(wtop, gv[k]), dbot = __fmul_rn(ylerp, gv[k]);
        if (tl) acc[k] = __fadd_rn(acc[k], __fmul_rn(wleft, dtop));
        if (tr) acc[k] = __fadd_rn(acc[k], __fmul_rn(xlerp, dtop));
        if (bl) acc[k] = __fadd_rn(acc[k], __fmul_rn(wleft, dbot));
        if (br) acc[k] = __fadd_rn(acc[k], __fmul_rn(xlerp, dbot));
    }
}

// grid (tiles, channel slices of 32*VEC*CPL, B).  Per chunk of CG_THREADS candidate boxes (the image's range of the
// batched layout, or all M filtered by box_index): each thread tests one box exactly against the tile's 4 rows and
// 4 columns, the boxes that touch the tile are compacted in ascending order into shared memory, then every warp
// walks that list for its pixel, visiting only the samples (y, x) whose row and column touch it.
template <int VEC, int CPL>
__global__ void __launch_bounds__(CG_THREADS, 2) crop_grad_kernel(CropArgs p) {
    constexpr int NW = CG_THREADS / 32;
    __shared__ float4 s_geo[CG_THREADS];   // a_y, s_y, a_x, s_x
    __shared__ uint4 s_rng[CG_THREADS];    // row lo, row hi, column lo, column hi (a byte per tile line)
    __shared__ int s_m[CG_THREADS];
    __shared__ int s_count[NW];
    const int tiles_x = (p.W + CG_TILE - 1) / CG_TILE;
    const int ty0 = (blockIdx.x / tiles_x) * CG_TILE, tx0 = (blockIdx.x % tiles_x) * CG_TILE;
    const int b = blockIdx.z, warp = warp_id(), lane = lane_id();
    const int ry = warp / CG_TILE, rx = warp % CG_TILE;
    const int py = ty0 + ry, px = tx0 + rx;
    const bool mine = py < p.H && px < p.W;
    const int c0 = blockIdx.y * (32 * VEC * CPL) + lane * VEC;
    float acc[CPL][VEC];
#pragma unroll
    for (int j = 0; j < CPL; ++j)
#pragma unroll
        for (int k = 0; k < VEC; ++k) acc[j][k] = 0.0f;
    const int m_begin = p.box_index ? 0 : b * p.per_image, m_end = p.box_index ? p.M : m_begin + p.per_image;
    const size_t row_stride = (size_t)p.cw * p.C;
    for (int base = m_begin; base < m_end; base += CG_THREADS) {
        const int m = base + threadIdx.x;
        bool hit = false;
        float4 geo;
        uint4 rng;
        if (m < m_end && (!p.box_index || p.box_index[m] == b)) {
            const float4 bx = p.boxes[m];
            const Axis ay = make_axis(bx.x, bx.z, p.H, p.ch), ax = make_axis(bx.y, bx.w, p.W, p.cw);
            hit = line_ranges(ay, ty0, rng.x, rng.y);
            hit = line_ranges(ax, tx0, rng.z, rng.w) && hit;
            geo = make_float4(ay.a, ay.s, ax.a, ax.s);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) s_count[warp] = __popc(bal);
        __syncthreads();
        int off = 0, total = 0;
#pragma unroll
        for (int w = 0; w < NW; ++w) {
            const int c = s_count[w];
            off += w < warp ? c : 0;
            total += c;
        }
        if (hit) {
            const int k = off + __popc(bal & ((1u << lane) - 1u));
            s_geo[k] = geo;
            s_rng[k] = rng;
            s_m[k] = m;
        }
        __syncthreads();
        if (mine) {
            for (int k = 0; k < total; ++k) {
                const uint4 rg = s_rng[k];
                const int ylo = (rg.x >> (8 * ry)) & 255, yhi = (rg.y >> (8 * ry)) & 255;
                const int xlo = (rg.z >> (8 * rx)) & 255, xhi = (rg.w >> (8 * rx)) & 255;
                if (ylo > yhi || xlo > xhi) continue;
                const float4 geo_k = s_geo[k];
                Axis ay, ax;
                ay.a = geo_k.x; ay.s = geo_k.y; ay.n = p.ch;
                ax.a = geo_k.z; ax.s = geo_k.w; ax.n = p.cw;
                const float* g_box = p.src + (size_t)s_m[k] * p.ch * row_stride;
                for (int y = ylo; y <= yhi; ++y) {
                    const float v = sample_at(ay, y);
                    const int top = (int)floorf(v);
                    const float ylerp = __fsub_rn(v, (float)top), wtop = __fsub_rn(1.0f, ylerp);
                    const bool is_top = top == py, is_bot = (int)ceilf(v) == py;
                    const float* g_row = g_box + (size_t)y * row_stride;
                    for (int x = xlo; x <= xhi; ++x) {
                        const float u = sample_at(ax, x);
                        const int left = (int)floorf(u);
                        const float xlerp = __fsub_rn(u, (float)left), wleft = __fsub_rn(1.0f, xlerp);
                        const bool is_l = left == px, is_r = (int)ceilf(u) == px;
                        const float* g = g_row + (size_t)x * p.C;
#pragma unroll
                        for (int j = 0; j < CPL; ++j) {
                            const int c = c0 + j * 32 * VEC;
                            if (c < p.C)
                                add_terms<VEC>(acc[j], g + c, wtop, ylerp, wleft, xlerp, is_top && is_l, is_top && is_r,
                                               is_bot && is_l, is_bot && is_r);
                        }
                    }
                }
            }
        }
        __syncthreads();
    }
    if (!mine) return;
    float* dst = p.dst + (((size_t)b * p.H + py) * p.W + px) * p.C;
#pragma unroll
    for (int j = 0; j < CPL; ++j) {
        const int c = c0 + j * 32 * VEC;
        if (c >= p.C) continue;
        if constexpr (VEC == 4)
            st_vec(reinterpret_cast<float4*>(dst + c), make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]));
        else
            st_vec(dst + c, acc[j][0]);
    }
}

int check_args(const char* what, const void* src, const float* boxes, const int32_t* box_index, const void* dst, int B,
               int H, int W, int C, int M, int crop_h, int crop_w) {
    if (!src || !boxes || !dst) return fail(TFRPN_ERR_BAD_ARG, "%s: null pointer", what);
    if (B < 1 || H < 1 || W < 1 || C < 1 || M < 1 || crop_h < 1 || crop_w < 1)
        return fail(TFRPN_ERR_BAD_ARG, "%s: B = %d, H = %d, W = %d, C = %d, M = %d, crop %d x %d (all must be >= 1)", what,
                    B, H, W, C, M, crop_h, crop_w);
    if (!box_index && M % B != 0)
        return fail(TFRPN_ERR_BAD_ARG, "%s: M = %d is not a multiple of B = %d (box_index is NULL)", what, M, B);
    if (C > CR_MAX_C || crop_h > CR_MAX_CROP || crop_w > CR_MAX_CROP || H > CR_MAX_HW || W > CR_MAX_HW || B > 65535 ||
        M > CR_MAX_M)
        return fail(TFRPN_ERR_UNSUPPORTED,
                    "%s: C = %d, crop %d x %d, H = %d, W = %d, B = %d, M = %d (at most %d, %d x %d, %d, %d, 65535, %d)", what,
                    C, crop_h, crop_w, H, W, B, M, CR_MAX_C, CR_MAX_CROP, CR_MAX_CROP, CR_MAX_HW, CR_MAX_HW, CR_MAX_M);
    if (!aligned16(boxes)) return fail(TFRPN_ERR_MISALIGNED, "%s: boxes must be 16-byte aligned", what);
    return 0;
}

CropArgs make_args(const float* src, const float* boxes, const int32_t* box_index, float* dst, int B, int H, int W,
                   int C, int M, int crop_h, int crop_w, float extrapolation) {
    CropArgs p;
    p.src = src;
    p.boxes = reinterpret_cast<const float4*>(boxes);
    p.box_index = box_index;
    p.dst = dst;
    p.B = B; p.H = H; p.W = W; p.C = C; p.M = M; p.ch = crop_h; p.cw = crop_w;
    p.per_image = box_index ? 0 : M / B;
    p.extrapolation = extrapolation;
    return p;
}

template <int VEC>
void launch_grad(const CropArgs& p, dim3 grid_base, cudaStream_t st) {
    const int groups = (p.C + VEC - 1) / VEC;   // channel groups; 32 lanes x CPL per slice
    const int cpl = groups <= 32 ? 1 : groups <= 64 ? 2 : 4;
    dim3 grid(grid_base.x, (groups + 32 * cpl - 1) / (32 * cpl), p.B);
    if (cpl == 1) crop_grad_kernel<VEC, 1><<<grid, CG_THREADS, 0, st>>>(p);
    else if (cpl == 2) crop_grad_kernel<VEC, 2><<<grid, CG_THREADS, 0, st>>>(p);
    else crop_grad_kernel<VEC, 4><<<grid, CG_THREADS, 0, st>>>(p);
}

}  // namespace
}  // namespace tfrpn

using namespace tfrpn;

extern "C" int tfrpn_crop_and_resize(const float* image, int B, int H, int W, int C, const float* boxes,
                                     const int32_t* box_index_or_null, int M, int crop_h, int crop_w,
                                     float extrapolation_value, float* out, tfrpn_stream s) {
    if (int rc = check_args("crop_and_resize", image, boxes, box_index_or_null, out, B, H, W, C, M, crop_h, crop_w))
        return rc;
    TFRPN_ENTER_PTR(out, "crop_and_resize: out");
    const CropArgs p = make_args(image, boxes, box_index_or_null, out, B, H, W, C, M, crop_h, crop_w, extrapolation_value);
    const unsigned blocks = (unsigned)M * (unsigned)crop_h;
    // float4 channels need C % 4 == 0 and 16-byte aligned rows of image and out
    if (C % 4 == 0 && aligned16(image) && aligned16(out)) crop_kernel<4><<<blocks, CR_THREADS, 0, as_stream(s)>>>(p);
    else crop_kernel<1><<<blocks, CR_THREADS, 0, as_stream(s)>>>(p);
    TFRPN_AFTER_LAUNCH("crop_kernel");
    return 0;
}

extern "C" int tfrpn_crop_and_resize_grad_image(const float* grad_out, const float* boxes,
                                                const int32_t* box_index_or_null, int M, int B, int H, int W, int C,
                                                int crop_h, int crop_w, float* grad_image, tfrpn_stream s) {
    if (int rc = check_args("crop_and_resize_grad_image", grad_out, boxes, box_index_or_null, grad_image, B, H, W, C, M,
                            crop_h, crop_w))
        return rc;
    TFRPN_ENTER_PTR(grad_image, "crop_and_resize_grad_image: grad_image");
    const CropArgs p = make_args(grad_out, boxes, box_index_or_null, grad_image, B, H, W, C, M, crop_h, crop_w, 0.0f);
    const dim3 tiles((unsigned)(((H + CG_TILE - 1) / CG_TILE) * ((W + CG_TILE - 1) / CG_TILE)));
    if (C % 4 == 0 && aligned16(grad_out) && aligned16(grad_image)) launch_grad<4>(p, tiles, as_stream(s));
    else launch_grad<1>(p, tiles, as_stream(s));
    TFRPN_AFTER_LAUNCH("crop_grad_kernel");
    return 0;
}
