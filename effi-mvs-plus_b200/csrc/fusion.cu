// Geometric-consistency filter: ref -> src -> ref reprojection with a bilinear sample of the
// source depth, the ladder of distance / depth thresholds, view votes, masked depth average and
// back-projection to world points -- one thread per reference pixel, one pass over the v source
// depth maps, nothing but the final mask / depth / points written back.
//
//   get_pixel_grids, idx_img2cam, idx_cam2world, idx_world2cam, idx_cam2img
//                                       upstream misc/fusion.py:8-47
//   get_reproj_dynamic                  upstream misc/fusion.py:117-154
//   vis_filter_dynamic                  upstream misc/fusion.py:157-181
//   vote / average / back-projection    upstream test_tank.py:473-515
//
// HBM-bound: per reference view it reads (1 + v) depth maps + the confidence map once and
// writes 1 + 4 + 12 bytes per pixel.  fusion_views_kernel runs the same per-pixel body (fusion_pixel) for all of a
// scene's reference views in one launch, reading the maps in place from one depth stack through index rows.
#include "common.cuh"

namespace effimvs {
namespace {

constexpr int MAXV = EFFIMVS_MAX_SRC_VIEWS;

struct alignas(16) Cam {   // one camera in shared memory; every matrix row is one 128-bit record
    float4 E[4];           // world -> camera
    float4 Ei[4];          // inverse(E)
    float4 K[3];           // rows of the 3x3 intrinsics (w unused)
    float4 Ki[3];
    // last row exactly (0,0,0,1) / (0,0,1): the homogeneous coordinate is then exactly 1 and
    // x / (1 + 1e-9f) == x bit for bit, so upstream's renormalising divisions can be skipped
    int affE, affEi, affK, affKi;
};
struct RefCam { float4 E[4]; float4 K[3]; int affE; };   // what the per-view loop needs of the reference camera: in registers

__device__ bool invert_n(const double* A, double* inv, int n) {
    double M[4][8];
    for (int r = 0; r < n; ++r)
        for (int c = 0; c < n; ++c) {
            M[r][c] = A[r * n + c];
            M[r][c + n] = (r == c) ? 1.0 : 0.0;
        }
    for (int col = 0; col < n; ++col) {
        int piv = col;
        double best = fabs(M[col][col]);
        for (int r = col + 1; r < n; ++r)
            if (fabs(M[r][col]) > best) { best = fabs(M[r][col]); piv = r; }
        if (best == 0.0) return false;
        if (piv != col)
            for (int c = 0; c < 2 * n; ++c) { double t = M[col][c]; M[col][c] = M[piv][c]; M[piv][c] = t; }
        double s = 1.0 / M[col][col];
        for (int c = 0; c < 2 * n; ++c) M[col][c] *= s;
        for (int r = 0; r < n; ++r) {
            if (r == col) continue;
            double f = M[r][col];
            for (int c = 0; c < 2 * n; ++c) M[r][c] -= f * M[col][c];
        }
    }
    for (int r = 0; r < n; ++r)
        for (int c = 0; c < n; ++c) inv[r * n + c] = M[r][c + n];
    return true;
}

// cam: (2,4,4) fp32.  inv: (2,4,4) holding inverse(E), inverse(K) padded.  INVERT: inv may be nullptr -> invert here
// (fp64 Gauss-Jordan with pivoting; its local arrays are why the <true> instantiation has a stack frame -- the torch
// binding always passes the inverses, from torch's LU or from effimvs_fusion_invert_cameras_f32).
template <bool INVERT>
__device__ void load_cam(Cam& c, const float* __restrict__ cam, const float* __restrict__ inv) {
    float E[16], Ei[16], K[9], Ki[9];
    for (int i = 0; i < 16; ++i) E[i] = cam[i];
    for (int r = 0; r < 3; ++r)
        for (int k = 0; k < 3; ++k) K[r * 3 + k] = cam[16 + r * 4 + k];
    if (!INVERT || inv) {
        for (int i = 0; i < 16; ++i) Ei[i] = inv[i];
        for (int r = 0; r < 3; ++r)
            for (int k = 0; k < 3; ++k) Ki[r * 3 + k] = inv[16 + r * 4 + k];
    } else {
        double A[16], I[16];
        for (int i = 0; i < 16; ++i) A[i] = E[i];
        bool ok = invert_n(A, I, 4);
        for (int i = 0; i < 16; ++i) Ei[i] = ok ? (float)I[i] : __int_as_float(0x7fc00000);
        for (int i = 0; i < 9; ++i) A[i] = K[i];
        ok = invert_n(A, I, 3);
        for (int i = 0; i < 9; ++i) Ki[i] = ok ? (float)I[i] : __int_as_float(0x7fc00000);
    }
    for (int r = 0; r < 4; ++r) {
        c.E[r] = make_float4(E[r * 4], E[r * 4 + 1], E[r * 4 + 2], E[r * 4 + 3]);
        c.Ei[r] = make_float4(Ei[r * 4], Ei[r * 4 + 1], Ei[r * 4 + 2], Ei[r * 4 + 3]);
    }
    for (int r = 0; r < 3; ++r) {
        c.K[r] = make_float4(K[r * 3], K[r * 3 + 1], K[r * 3 + 2], 0.0f);
        c.Ki[r] = make_float4(Ki[r * 3], Ki[r * 3 + 1], Ki[r * 3 + 2], 0.0f);
    }
    c.affE = E[12] == 0.0f && E[13] == 0.0f && E[14] == 0.0f && E[15] == 1.0f;
    c.affEi = Ei[12] == 0.0f && Ei[13] == 0.0f && Ei[14] == 0.0f && Ei[15] == 1.0f;
    c.affK = K[6] == 0.0f && K[7] == 0.0f && K[8] == 1.0f;
    c.affKi = Ki[6] == 0.0f && Ki[7] == 0.0f && Ki[8] == 1.0f;
}

__device__ __forceinline__ void mat3(const float4* M, float x, float y, float z, float o[3]) {
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const float4 m = M[r];
        o[r] = fmaf(m.z, z, fmaf(m.y, y, __fmul_rn(m.x, x)));
    }
}
__device__ __forceinline__ void mat4(const float4* M, const float p[4], float o[4]) {
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const float4 m = M[r];
        o[r] = fmaf(m.w, p[3], fmaf(m.z, p[2], fmaf(m.y, p[1], __fmul_rn(m.x, p[0]))));
    }
}

// idx_img2cam + idx_cam2world (fusion.py:23-34): pixel (u,v,1), depth -> homogeneous world point
__device__ __forceinline__ void img_to_world(const Cam& c, float u, float v, float depth, float pw[4]) {
    float k[3];
    mat3(c.Ki, u, v, 1.0f, k);
    float pc[4];
    if (c.affKi) {   // k[2] == 1 exactly
        pc[0] = __fmul_rn(k[0], depth); pc[1] = __fmul_rn(k[1], depth); pc[2] = depth;
    } else {
        float zz = __fadd_rn(k[2], 1e-9f);
        pc[0] = __fmul_rn(__fdiv_rn(k[0], zz), depth); pc[1] = __fmul_rn(__fdiv_rn(k[1], zz), depth);
        pc[2] = __fmul_rn(__fdiv_rn(k[2], zz), depth);
    }
    pc[3] = 1.0f;
    float w[4];
    mat4(c.Ei, pc, w);
    if (c.affEi) {   // w[3] == 1 exactly
#pragma unroll
        for (int i = 0; i < 4; ++i) pw[i] = w[i];
    } else {
        float ww = __fadd_rn(w[3], 1e-9f);
#pragma unroll
        for (int i = 0; i < 4; ++i) pw[i] = __fdiv_rn(w[i], ww);
    }
}

// idx_world2cam (fusion.py:37-40)
__device__ __forceinline__ void world_to_cam(const float4* E, int affE, const float pw[4], float pc[4]) {
    if (affE && pw[3] == 1.0f) {   // last row (0,0,0,1) and w == 1: t[3] == 1 exactly, x / (1 + 1e-9f) == x: three rows, no division
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float4 m = E[r];
            pc[r] = fmaf(m.w, pw[3], fmaf(m.z, pw[2], fmaf(m.y, pw[1], __fmul_rn(m.x, pw[0]))));
        }
        pc[3] = 1.0f;
        return;
    }
    float t[4];
    mat4(E, pw, t);
    {
        float ww = __fadd_rn(t[3], 1e-9f);
#pragma unroll
        for (int i = 0; i < 4; ++i) pc[i] = __fdiv_rn(t[i], ww);
    }
}

// idx_cam2img (fusion.py:43-47)
__device__ __forceinline__ void cam_to_img(const float4* K, const float pc[4], float& u, float& v) {
    float k[3];
    if (pc[3] == 1.0f) {             // (1 + 1e-9f) == 1: the division is the identity
        mat3(K, pc[0], pc[1], pc[2], k);
    } else {
        float ww = __fadd_rn(pc[3], 1e-9f);
        mat3(K, __fdiv_rn(pc[0], ww), __fdiv_rn(pc[1], ww), __fdiv_rn(pc[2], ww), k);
    }
    div2_rn(k[0], k[1], __fadd_rn(k[2], 1e-9f), u, v);
}

// bilinear sample, zeros padding, align_corners=True, pixel coordinates (u,v) normalised the way
// fusion.py:134-139 + ATen do it on a CUDA device
__device__ __forceinline__ float sample_depth(const float* __restrict__ img, int h, int w, float u, float v,
                                              float inv_half_w, float inv_half_h) {
    float gx = __fsub_rn(__fmul_rn(u, inv_half_w), 1.0f);
    float gy = __fsub_rn(__fmul_rn(v, inv_half_h), 1.0f);
    float ix = __fmul_rn(__fadd_rn(gx, 1.0f), 0.5f * (float)(w - 1));    // = ((g + 1) / 2) * (w - 1) bit for bit (exact halving)
    float iy = __fmul_rn(__fadd_rn(gy, 1.0f), 0.5f * (float)(h - 1));
    float fx = floorf(ix), fy = floorf(iy);
    bool x0 = (fx >= 0.0f) && (fx <= (float)(w - 1));
    bool x1 = (fx >= -1.0f) && (fx <= (float)(w - 2));
    bool y0 = (fy >= 0.0f) && (fy <= (float)(h - 1));
    bool y1 = (fy >= -1.0f) && (fy <= (float)(h - 2));
    if (!((x0 || x1) && (y0 || y1))) return 0.0f;
    int xi = (int)fx, yi = (int)fy;
    const float* p = img + (ptrdiff_t)yi * w + xi;
    float ex = __fsub_rn(__fadd_rn(fx, 1.0f), ix), ey = __fsub_rn(__fadd_rn(fy, 1.0f), iy);
    float dx = __fsub_rn(ix, fx), dy = __fsub_rn(iy, fy);
    float out = 0.0f;
    if (x0 && y0) out = __fmul_rn(__ldg(p), __fmul_rn(ex, ey));
    if (x1 && y0) out = fmaf(__ldg(p + 1), __fmul_rn(dx, ey), out);
    if (x0 && y1) out = fmaf(__ldg(p + w), __fmul_rn(ex, dy), out);
    if (x1 && y1) out = fmaf(__ldg(p + w + 1), __fmul_rn(dx, dy), out);
    return out;
}

struct Reproj { float x, y, d; };

// Number of ladder rungs k in [0, K) with e < thr[k], thr[k] = fl((tv + k) / base) (fusion.py:172-176).  The
// thresholds are non-decreasing in k, so the rungs passed are exactly k >= idx with idx the first rung passed:
// idx is estimated from e * base - tv and settled with the same comparisons upstream makes (typically one or two
// instead of all K).  NaN passes no rung, like the comparison chain it replaces.
__device__ __forceinline__ int ladder_count(float e, const float* __restrict__ thr, int K, float base, float tv) {
    // thr has K + 2 entries: thr[0] = -inf, thr[1 + k] = rung k, thr[K + 1] = +inf, so the neighbours of the estimate can be
    // read without bounds checks.  The estimate floor(e * base - tv) + 1 is the exact first rung passed up to the rounding of
    // one product and one quotient, i.e. off by at most one: one look at each neighbour settles it with upstream's own
    // comparisons (e < thr[k]); the two loops stay as the (never iterating) safety net for pathological bases.
    int idx = (int)fminf(fmaxf(floorf(fmaf(e, base, -tv)) + 1.0f, 0.0f), (float)K);
    const float below = thr[idx], at = thr[idx + 1];      // rung idx - 1, rung idx
    idx += (e < below) ? -1 : ((e < at) ? 0 : 1);
    idx = max(0, min(idx, K));
    while (idx > 0 && e < thr[idx]) --idx;
    while (idx < K && !(e < thr[idx + 1])) ++idx;
    return K - idx;
}

__device__ __forceinline__ Reproj reproject(const RefCam& ref, const Cam& src, const float ref_world[4],
                                            const float* __restrict__ src_depth, int h, int w,
                                            float inv_half_w, float inv_half_h) {
    float pc[4], u, v;
    world_to_cam(src.E, src.affE, ref_world, pc);
    cam_to_img(src.K, pc, u, v);
    float ds = sample_depth(src_depth, h, w, u, v, inv_half_w, inv_half_h);
    float pw[4], back[4];
    img_to_world(src, u, v, ds, pw);
    world_to_cam(ref.E, ref.affE, pw, back);
    Reproj r;
    r.d = back[2];
    cam_to_img(ref.K, back, r.x, r.y);
    return r;
}

// One reference pixel of the filter (view n of the launch, cameras and ladder already in shared memory).  `ref_of()` is
// the view's (h,w) reference depth map and `src_of(s)` its source view s's, so the body never knows how the maps are
// laid out.  conf is (n,hc,wc); the outputs are indexed by n as (n,1,h,w) / (n,3,h,w) / (n,v,3,h,w) / (n,v,K,h,w),
// and reproj_xyd, final_mask (with depth_avg / points) and masks_out may be null.
template <class RefOf, class SrcOf>
__device__ __forceinline__ void fusion_pixel(int n, int pix, const Cam* cams, const float* thr_xy,
                                             const float* thr_d, RefOf ref_of, SrcOf src_of,
                                             const float* conf, int v, int K, int h, int w, int hc, int wc,
                                             float dist_base, float rel_diff_base, int thres_view, float prob_threshold,
                                             int relative, float inv_half_w, float inv_half_h, float* reproj_xyd,
                                             uint8_t* final_mask, float* depth_avg,
                                             float* points, uint8_t* masks_out) {
    const int hw = h * w;
    const int yi = pix / w, xi = pix - yi * w;
    const float cx = (float)xi + 0.5f, cy = (float)yi + 0.5f;
    const float dref = __ldg(ref_of() + pix);
    float ref_world[4];
    img_to_world(cams[0], cx, cy, dref, ref_world);
    RefCam rc;
#pragma unroll
    for (int r = 0; r < 4; ++r) rc.E[r] = cams[0].E[r];
#pragma unroll
    for (int r = 0; r < 3; ++r) rc.K[r] = cams[0].K[r];
    rc.affE = cams[0].affE;

    // The ladder thresholds grow with k, so a view passes rungs K-c .. K-1 where c = min(#rungs its pixel
    // error passes, #rungs its depth error passes).  hist packs the per-view c values: 17 bins of 5 bits.
    unsigned long long hist_lo = 0ull, hist_hi = 0ull;   // bins 0..11 | bins 12..16
    float sum_d = 0.0f;
    int n_last = 0;
    for (int s = 0; s < v; ++s) {
        Reproj r = reproject(rc, cams[s + 1], ref_world, src_of(s), h, w, inv_half_w, inv_half_h);
        if (reproj_xyd) {
            float* o = reproj_xyd + (((size_t)n * v + s) * 3) * hw + pix;
            o[0] = r.x; o[(size_t)hw] = r.y; o[(size_t)2 * hw] = r.d;
        }
        if (!final_mask) continue;
        float ex = __fsub_rn(r.x, cx), ey = __fsub_rn(r.y, cy);
        float e_xy = sqrtf(__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)));
        float e_d = fabsf(__fsub_rn(dref, r.d));
        if (relative) e_d = __fdiv_rn(e_d, dref);
        const int c = min(ladder_count(e_xy, thr_xy, K, dist_base, (float)thres_view),
                          ladder_count(e_d, thr_d, K, rel_diff_base, (float)thres_view));
        if (c < 12) hist_lo += 1ull << (5 * c);
        else hist_hi += 1ull << (5 * (c - 12));
        if (masks_out)
            for (int k = 0; k < K; ++k) masks_out[(((size_t)n * v + s) * K + k) * hw + pix] = (k >= K - c) ? 1 : 0;
        if (c >= 1) { sum_d = __fadd_rn(sum_d, r.d); n_last += 1; }
    }
    if (!final_mask) return;
    // votes[k] = #views with c >= K - k; geo = any k with votes[k] >= thres_view + k
    bool geo = false;
    int votes = 0;
    for (int k = 0; k < K; ++k) {
        const int bin = K - k;   // views whose c equals K - k start passing at rung k
        votes += bin < 12 ? (int)((hist_lo >> (5 * bin)) & 31ull) : (int)((hist_hi >> (5 * (bin - 12))) & 31ull);
        geo = geo || (votes >= thres_view + k);
    }
    // nearest resize of the confidence map: src index = floor(dst * in / out)  (F.interpolate 'nearest')
    int sy = (int)floorf((float)yi * ((float)hc / (float)h)), sx = (int)floorf((float)xi * ((float)wc / (float)w));
    sy = sy < hc - 1 ? sy : hc - 1; sx = sx < wc - 1 ? sx : wc - 1;
    bool prob = __ldg(conf + ((size_t)n * hc + sy) * wc + sx) > prob_threshold;
    float avg = __fdiv_rn(__fadd_rn(sum_d, dref), (float)(n_last + 1));
    float pw[4];
    img_to_world(cams[0], cx, cy, avg, pw);
    final_mask[(size_t)n * hw + pix] = (prob && geo) ? 1 : 0;
    depth_avg[(size_t)n * hw + pix] = avg;
    points[((size_t)n * 3 + 0) * hw + pix] = pw[0];
    points[((size_t)n * 3 + 1) * hw + pix] = pw[1];
    points[((size_t)n * 3 + 2) * hw + pix] = pw[2];
}

// the ladder k / dist_base, k / rel_diff_base (fusion.py:172-176) of thres_view <= k < thres_view + K between -inf and +inf,
// written by threads 32 .. 32 + MAXV + 1 of the block
__device__ __forceinline__ void fill_ladder(float* __restrict__ thr_xy, float* __restrict__ thr_d, int K, float dist_base,
                                            float rel_diff_base, int thres_view) {
    const int j = threadIdx.x - 32, k = j - 1;
    const float kk = (float)(thres_view + k);
    thr_xy[j] = j == 0 ? -INFINITY : (k < K ? __fdiv_rn(kk, dist_base) : INFINITY);
    thr_d[j] = j == 0 ? -INFINITY : (k < K ? __fdiv_rn(kk, rel_diff_base) : INFINITY);
}

template <bool INVERT>
__global__ void __launch_bounds__(128, 6)
fusion_kernel(const float* __restrict__ ref_depth, const float* __restrict__ srcs_depth, const float* __restrict__ conf,
              const float* __restrict__ ref_cam, const float* __restrict__ srcs_cam, const float* __restrict__ inv_cams,
              int v, int h, int w, int hc, int wc, float dist_base, float rel_diff_base, int thres_view,
              float prob_threshold, int relative, float inv_half_w, float inv_half_h, float* __restrict__ reproj_xyd, uint8_t* __restrict__ final_mask,
              float* __restrict__ depth_avg, float* __restrict__ points, uint8_t* __restrict__ masks_out) {
    __shared__ Cam cams[MAXV + 1];
    __shared__ float thr_xy[MAXV + 2], thr_d[MAXV + 2];   // the ladder between -inf and +inf
    const int n = blockIdx.y;
    const int K = v - thres_view + 1;
    if (threadIdx.x <= v) {
        const float* cam = threadIdx.x == 0 ? ref_cam + (size_t)n * 32 : srcs_cam + ((size_t)n * v + threadIdx.x - 1) * 32;
        const float* inv = inv_cams ? inv_cams + ((size_t)n * (v + 1) + threadIdx.x) * 32 : nullptr;
        load_cam<INVERT>(cams[threadIdx.x], cam, inv);
    } else if (threadIdx.x >= 32 && threadIdx.x < 32 + MAXV + 2) {
        fill_ladder(thr_xy, thr_d, K, dist_base, rel_diff_base, thres_view);
    }
    __syncthreads();
    const int hw = h * w;
    const int pix = blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= hw) return;
    fusion_pixel(n, pix, cams, thr_xy, thr_d, [=] { return ref_depth + (size_t)n * hw; },
                 [=](int s) { return srcs_depth + ((size_t)n * v + s) * hw; }, conf, v, K, h, w, hc, wc, dist_base,
                 rel_diff_base, thres_view, prob_threshold, relative, inv_half_w, inv_half_h, reproj_xyd, final_mask, depth_avg,
                 points, masks_out);
}

// Several reference views of one scene in one launch: grid (pixel tiles of 128, n views).  Block y filters reference view
// y: its reference map is row ref_idx[y] of the one (N,h,w) depth stack, its sources are rows src_idx[y][0 .. src_count[y]),
// all read in place; the cameras of those rows come from the scene table cams (N,2,4,4) and their inverses from inv_cams
// (N,2,4,4, as invert_cameras_kernel writes them).  The ladder is the view's own (K = src_count[y] - thres_view + 1).
// Every view's results are those of fusion_kernel<false> on that view alone with the same cameras and inverses.
__global__ void __launch_bounds__(128, 6)
fusion_views_kernel(const float* __restrict__ depths, const int* __restrict__ ref_idx, const int* __restrict__ src_idx,
                    const int* __restrict__ src_count, int vmax, const float* __restrict__ cam_tab,
                    const float* __restrict__ inv_tab, const float* __restrict__ conf, int h, int w, int hc, int wc,
                    float dist_base, float rel_diff_base, int thres_view, float prob_threshold, int relative,
                    float inv_half_w, float inv_half_h, uint8_t* __restrict__ final_mask, float* __restrict__ depth_avg,
                    float* __restrict__ points) {
    __shared__ Cam cams[MAXV + 1];
    __shared__ float thr_xy[MAXV + 2], thr_d[MAXV + 2];
    __shared__ int rows[MAXV + 1];                         // stack rows of the reference map, then of the source maps
    const int n = blockIdx.y;
    const int v = src_count[n];
    const int K = v - thres_view + 1;
    if (threadIdx.x <= v) {
        const int r = threadIdx.x == 0 ? ref_idx[n] : src_idx[(size_t)n * vmax + threadIdx.x - 1];
        rows[threadIdx.x] = r;
        load_cam<false>(cams[threadIdx.x], cam_tab + (size_t)r * 32, inv_tab + (size_t)r * 32);
    } else if (threadIdx.x >= 32 && threadIdx.x < 32 + MAXV + 2) {
        fill_ladder(thr_xy, thr_d, K, dist_base, rel_diff_base, thres_view);
    }
    __syncthreads();
    const int hw = h * w;
    const int pix = blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= hw) return;
    fusion_pixel(n, pix, cams, thr_xy, thr_d, [=] { return depths + (size_t)rows[0] * hw; },
                 [=](int s) { return depths + (size_t)rows[s + 1] * hw; }, conf, v, K, h, w, hc, wc, dist_base, rel_diff_base,
                 thres_view, prob_threshold, relative, inv_half_w, inv_half_h, nullptr, final_mask, depth_avg, points, nullptr);
}

// inverse(E), inverse(K) of the 1 + v cameras of every batch item -> inv (n, 1+v, 2, 4, 4), the layout fusion_kernel reads
__global__ void invert_cameras_kernel(const float* __restrict__ ref_cam, const float* __restrict__ srcs_cam, int v, float* __restrict__ inv) {
    const int n = blockIdx.x, i = threadIdx.x;
    if (i > v) return;
    const float* cam = i == 0 ? ref_cam + (size_t)n * 32 : srcs_cam + ((size_t)n * v + i - 1) * 32;
    float* o = inv + ((size_t)n * (v + 1) + i) * 32;
    double A[16], I[16];
    for (int k = 0; k < 16; ++k) A[k] = cam[k];
    bool ok = invert_n(A, I, 4);
    for (int k = 0; k < 16; ++k) o[k] = ok ? (float)I[k] : __int_as_float(0x7fc00000);
    for (int r = 0; r < 3; ++r)
        for (int k = 0; k < 3; ++k) A[r * 3 + k] = cam[16 + r * 4 + k];
    ok = invert_n(A, I, 3);
    for (int k = 0; k < 16; ++k) o[16 + k] = 0.0f;
    for (int r = 0; r < 3; ++r)
        for (int k = 0; k < 3; ++k) o[16 + r * 4 + k] = ok ? (float)I[r * 3 + k] : __int_as_float(0x7fc00000);
}

// vis_filter_dynamic (misc/fusion.py:157-181) on an existing reproj_xyd (n,v,3,h,w) -> masks (n,v,K,h,w)
__global__ void fusion_masks_kernel(const float* __restrict__ ref_depth, const float* __restrict__ xyd, int v, int h, int w,
                                    float dist_base, float rel_diff_base, int thres_view, int relative, uint8_t* __restrict__ masks) {
    const int n = blockIdx.z, s = blockIdx.y;
    const int hw = h * w;
    const int pix = blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= hw) return;
    const int yi = pix / w, xi = pix - yi * w;
    const float cx = (float)xi + 0.5f, cy = (float)yi + 0.5f;
    const float* p = xyd + (((size_t)n * v + s) * 3) * hw + pix;
    const float dref = __ldg(ref_depth + (size_t)n * hw + pix);
    const float ex = __fsub_rn(__ldg(p), cx), ey = __fsub_rn(__ldg(p + hw), cy);
    const float e_xy = sqrtf(__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)));
    float e_d = fabsf(__fsub_rn(dref, __ldg(p + 2 * (size_t)hw)));
    if (relative) e_d = __fdiv_rn(e_d, dref);
    const int K = v - thres_view + 1;
    for (int k = 0; k < K; ++k) {
        const float kk = (float)(thres_view + k);
        masks[(((size_t)n * v + s) * K + k) * hw + pix] = (e_xy < __fdiv_rn(kk, dist_base)) && (e_d < __fdiv_rn(kk, rel_diff_base));
    }
}

}  // namespace
}  // namespace effimvs

using namespace effimvs;

extern "C" int effimvs_fusion_reproject_f32(const float* ref_depth, const float* srcs_depth, const float* ref_cam,
                                            const float* srcs_cam, const float* inv_cams, int n, int v, int h, int w,
                                            float* reproj_xyd, void* stream) {
    EFFI_REQUIRE(ref_depth && srcs_depth && ref_cam && srcs_cam && reproj_xyd, EFFIMVS_EINVAL, "fusion_reproject: null pointer");
    EFFI_REQUIRE(n > 0 && v >= 1 && v <= MAXV && h > 1 && w > 1, EFFIMVS_EINVAL, "fusion_reproject: bad sizes (v in [1,%d])", MAXV);
    dim3 block(128), grid(ceil_div(h * w, 128), n);
    const float ihw = 1.0f / (float)((double)(w - 1) / 2.0), ihh = 1.0f / (float)((double)(h - 1) / 2.0);   // as __fdiv_rn on the device
    if (inv_cams)
        fusion_kernel<false><<<grid, block, 0, (cudaStream_t)stream>>>(ref_depth, srcs_depth, nullptr, ref_cam, srcs_cam, inv_cams, v, h, w,
                                                                      1, 1, 1.0f, 1.0f, 1, 0.0f, 0, ihw, ihh, reproj_xyd, nullptr, nullptr, nullptr, nullptr);
    else
        fusion_kernel<true><<<grid, block, 0, (cudaStream_t)stream>>>(ref_depth, srcs_depth, nullptr, ref_cam, srcs_cam, inv_cams, v, h, w,
                                                                     1, 1, 1.0f, 1.0f, 1, 0.0f, 0, ihw, ihh, reproj_xyd, nullptr, nullptr, nullptr, nullptr);
    return check_launch("fusion_kernel(reproject)");
}

extern "C" int effimvs_fusion_filter_f32(const float* ref_depth, const float* srcs_depth, const float* conf,
                                         const float* ref_cam, const float* srcs_cam, const float* inv_cams,
                                         int n, int v, int h, int w, int hc, int wc,
                                         float dist_base, float rel_diff_base, int thres_view, float prob_threshold,
                                         int relative, uint8_t* final_mask, float* depth_avg, float* points,
                                         uint8_t* masks_out, void* stream) {
    EFFI_REQUIRE(ref_depth && srcs_depth && conf && ref_cam && srcs_cam && final_mask && depth_avg && points, EFFIMVS_EINVAL,
                 "fusion_filter: null pointer");
    EFFI_REQUIRE(n > 0 && v >= 1 && v <= MAXV && h > 1 && w > 1 && hc > 0 && wc > 0, EFFIMVS_EINVAL,
                 "fusion_filter: bad sizes (v in [1,%d])", MAXV);
    EFFI_REQUIRE(thres_view >= 1 && thres_view <= v, EFFIMVS_EINVAL, "fusion_filter: thres_view=%d outside [1,%d]", thres_view, v);
    EFFI_REQUIRE(dist_base > 0.0f && rel_diff_base > 0.0f, EFFIMVS_EINVAL, "fusion_filter: thresholds must be positive");
    dim3 block(128), grid(ceil_div(h * w, 128), n);
    const float ihw = 1.0f / (float)((double)(w - 1) / 2.0), ihh = 1.0f / (float)((double)(h - 1) / 2.0);   // as __fdiv_rn on the device
    if (inv_cams)
        fusion_kernel<false><<<grid, block, 0, (cudaStream_t)stream>>>(ref_depth, srcs_depth, conf, ref_cam, srcs_cam, inv_cams, v, h, w, hc, wc,
                                                                      dist_base, rel_diff_base, thres_view, prob_threshold, relative, ihw, ihh,
                                                                      nullptr, final_mask, depth_avg, points, masks_out);
    else
        fusion_kernel<true><<<grid, block, 0, (cudaStream_t)stream>>>(ref_depth, srcs_depth, conf, ref_cam, srcs_cam, inv_cams, v, h, w, hc, wc,
                                                                     dist_base, rel_diff_base, thres_view, prob_threshold, relative, ihw, ihh,
                                                                     nullptr, final_mask, depth_avg, points, masks_out);
    return check_launch("fusion_kernel(filter)");
}

extern "C" int effimvs_fusion_invert_cameras_f32(const float* ref_cam, const float* srcs_cam, int n, int v, float* inv_out, void* stream) {
    EFFI_REQUIRE(ref_cam && srcs_cam && inv_out, EFFIMVS_EINVAL, "fusion_invert_cameras: null pointer");
    EFFI_REQUIRE(n > 0 && v >= 1 && v <= MAXV, EFFIMVS_EINVAL, "fusion_invert_cameras: bad sizes (v in [1,%d])", MAXV);
    invert_cameras_kernel<<<n, 32, 0, (cudaStream_t)stream>>>(ref_cam, srcs_cam, v, inv_out);
    return check_launch("invert_cameras_kernel");
}

extern "C" int effimvs_fusion_masks_f32(const float* ref_depth, const float* reproj_xyd, int n, int v, int h, int w,
                                        float dist_base, float rel_diff_base, int thres_view, int relative,
                                        uint8_t* masks_out, void* stream) {
    EFFI_REQUIRE(ref_depth && reproj_xyd && masks_out, EFFIMVS_EINVAL, "fusion_masks: null pointer");
    EFFI_REQUIRE(n > 0 && v >= 1 && v <= 65535 && h > 0 && w > 0 && thres_view >= 1 && thres_view <= v, EFFIMVS_EINVAL, "fusion_masks: bad sizes");
    EFFI_REQUIRE(dist_base > 0.0f && rel_diff_base > 0.0f, EFFIMVS_EINVAL, "fusion_masks: thresholds must be positive");
    dim3 block(128), grid(ceil_div(h * w, 128), v, n);
    fusion_masks_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(ref_depth, reproj_xyd, v, h, w, dist_base, rel_diff_base, thres_view,
                                                                relative, masks_out);
    return check_launch("fusion_masks_kernel");
}

extern "C" int effimvs_fusion_filter_views_f32(const float* depths, int n_depths, const int* ref_idx, const int* src_idx,
                                               const int* src_count, int vmax, const float* cams, const float* inv_cams,
                                               const float* conf, int hc, int wc, float dist_base, float rel_diff_base,
                                               int thres_view, float prob_threshold, int relative, int n, int h, int w,
                                               uint8_t* final_mask, float* depth_avg, float* points, void* stream) {
    EFFI_REQUIRE(depths && ref_idx && src_idx && src_count && cams && inv_cams && conf && final_mask && depth_avg && points,
                 EFFIMVS_EINVAL, "fusion_filter_views: null pointer");
    EFFI_REQUIRE(n_depths >= 1 && vmax >= 1 && vmax <= MAXV && n >= 1 && n <= 65535 && h > 1 && w > 1 && hc > 0 && wc > 0 &&
                 (long long)h * w <= 0x7fffffffLL - 127, EFFIMVS_EINVAL,
                 "fusion_filter_views: bad sizes (N=%d, vmax=%d in [1,%d], n=%d in [1,65535], h=%d, w=%d, hc=%d, wc=%d)",
                 n_depths, vmax, MAXV, n, h, w, hc, wc);
    EFFI_REQUIRE(thres_view >= 1 && thres_view <= vmax, EFFIMVS_EINVAL, "fusion_filter_views: thres_view=%d outside [1,%d]", thres_view, vmax);
    EFFI_REQUIRE(dist_base > 0.0f && rel_diff_base > 0.0f, EFFIMVS_EINVAL, "fusion_filter_views: thresholds must be positive");
    dim3 block(128), grid(ceil_div(h * w, 128), n);
    const float ihw = 1.0f / (float)((double)(w - 1) / 2.0), ihh = 1.0f / (float)((double)(h - 1) / 2.0);   // as __fdiv_rn on the device
    fusion_views_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(depths, ref_idx, src_idx, src_count, vmax, cams, inv_cams, conf, h, w,
                                                                 hc, wc, dist_base, rel_diff_base, thres_view, prob_threshold, relative,
                                                                 ihw, ihh, final_mask, depth_avg, points);
    return check_launch("fusion_views_kernel");
}
