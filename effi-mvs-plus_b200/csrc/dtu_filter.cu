// DTU geometric-consistency filter (SURVEY section 8(f) row 2): the NumPy + cv2.remap variant upstream's DTU
// pipeline uses, one thread per reference pixel, one pass over the v source depth maps.
//
//   reproject_with_depth          upstream test_dtu_dypcd.py:164-204
//   check_geometric_consistency   upstream test_dtu_dypcd.py:207-233
//   filter_depth (aggregation)    upstream test_dtu_dypcd.py:261-309, 320-337
//
// Arithmetic as NumPy's promotion rules produce it upstream: camera matrices, inverses and relative
// poses are float32 (prepared by the caller exactly as upstream forms them), everything multiplied
// with the integer pixel grid is float64, the sampled / reprojected depths and reprojected pixel
// positions are rounded to float32 where upstream casts them.  cv2.remap(INTER_LINEAR) on a float32
// image is restated from OpenCV's remapBilinear: coordinates rounded to 1/32 pixel (half to even),
// table weights (1-fy)(1-fx), (1-fy)fx, fy(1-fx), fy fx in float32, taps accumulated left to right
// without contraction, constant border 0.
#include "common.cuh"

namespace effimvs {
namespace {

constexpr int MAX_RUNGS = 32;

struct Ladder {
    double dist[MAX_RUNGS];   // i * dist_base (compared in float64)
    float diff[MAX_RUNGS];    // log10(max(i, 1.05)) * diff_base rounded to float32 (compared in float32)
};

__device__ __forceinline__ void mat3d(const float* __restrict__ M, double x, double y, double z, double o[3]) {
#pragma unroll
    for (int r = 0; r < 3; ++r)
        o[r] = __dadd_rn(__dadd_rn(__dmul_rn((double)M[r * 3], x), __dmul_rn((double)M[r * 3 + 1], y)), __dmul_rn((double)M[r * 3 + 2], z));
}
// first three rows of a 4x4 applied to (x, y, z, 1)
__device__ __forceinline__ void mat4d(const float* __restrict__ M, const double p[3], double o[3]) {
#pragma unroll
    for (int r = 0; r < 3; ++r)
        o[r] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn((double)M[r * 4], p[0]), __dmul_rn((double)M[r * 4 + 1], p[1])),
                                   __dmul_rn((double)M[r * 4 + 2], p[2])), (double)M[r * 4 + 3]);
}

// cv2.remap(img, x, y, INTER_LINEAR), float32 image, BORDER_CONSTANT 0
__device__ __forceinline__ float remap_bilinear(const float* __restrict__ img, int h, int w, float x, float y) {
    if (!(fabsf(x) < 6.0e7f) || !(fabsf(y) < 6.0e7f)) return 0.0f;   // NaN / beyond int32 after the x32 scaling: outside
    const int sx = __float2int_rn(__fmul_rn(x, 32.0f)), sy = __float2int_rn(__fmul_rn(y, 32.0f));
    const int x0 = sx >> 5, y0 = sy >> 5;
    const float fx = (float)(sx & 31) * 0.03125f, fy = (float)(sy & 31) * 0.03125f;
    const float gx = __fsub_rn(1.0f, fx), gy = __fsub_rn(1.0f, fy);
    const bool xa = x0 >= 0 && x0 < w, xb = x0 + 1 >= 0 && x0 + 1 < w;
    const bool ya = y0 >= 0 && y0 < h, yb = y0 + 1 >= 0 && y0 + 1 < h;
    const float* p = img + (ptrdiff_t)y0 * w + x0;
    const float t00 = (xa && ya) ? __ldg(p) : 0.0f, t01 = (xb && ya) ? __ldg(p + 1) : 0.0f;
    const float t10 = (xa && yb) ? __ldg(p + w) : 0.0f, t11 = (xb && yb) ? __ldg(p + w + 1) : 0.0f;
    float out = __fmul_rn(t00, __fmul_rn(gy, gx));
    out = __fadd_rn(out, __fmul_rn(t01, __fmul_rn(gy, fx)));
    out = __fadd_rn(out, __fmul_rn(t10, __fmul_rn(fy, gx)));
    out = __fadd_rn(out, __fmul_rn(t11, __fmul_rn(fy, fx)));
    return out;
}

// mats: [Kinv_ref 9][K_ref 9][Einv_ref 16] then per source view [E_src @ inv(E_ref) 16][K_src 9][Kinv_src 9][E_ref @ inv(E_src) 16]
constexpr int REF_FLOATS = 34, SRC_FLOATS = 50;

// One reference pixel of the filter.  `src_of(s)` is source view s's (h,w) depth map; the output pointers are the
// view's own (h,w) / (3,h,w) planes; geo_mask, masks_out and reproj_depth_out may be null.
template <class SrcOf>
__device__ __forceinline__ void dtu_filter_pixel(int pix, const float* __restrict__ sm, const float* __restrict__ ref_depth,
                                                 SrcOf src_of, const float* __restrict__ conf, const Ladder& lad, int K, int S,
                                                 int E, float conf_thres, float conf_keep, int v, int h, int w,
                                                 uint8_t* __restrict__ final_mask, uint8_t* __restrict__ geo_mask,
                                                 float* __restrict__ depth_avg, float* __restrict__ points,
                                                 uint8_t* __restrict__ masks_out, float* __restrict__ reproj_depth_out) {
    const int hw = h * w;
    const int yi = pix / w, xi = pix - yi * w;
    const double xd = (double)xi, yd = (double)yi;
    const float dref = __ldg(ref_depth + pix);
    const double dd = (double)dref;
    const float* Kinv_ref = sm, * K_ref = sm + 9, * Einv_ref = sm + 18;

    double pr[3];
    mat3d(Kinv_ref, __dmul_rn(xd, dd), __dmul_rn(yd, dd), dd, pr);   // inv(K_ref) @ ((x, y, 1) * depth)

    unsigned long long hist_lo = 0ull, hist_hi = 0ull, hist_top = 0ull;   // 33 bins of 5 bits: c = rungs passed by a view
    float sum_rep = 0.0f;
    int n_last = 0;
    for (int s = 0; s < v; ++s) {
        const float* R1 = sm + REF_FLOATS + s * SRC_FLOATS, * K_src = R1 + 16, * Kinv_src = R1 + 25, * R2 = R1 + 34;
        double ps[3], ks[3];
        mat4d(R1, pr, ps);
        mat3d(K_src, ps[0], ps[1], ps[2], ks);
        const double u = __ddiv_rn(ks[0], ks[2]), t = __ddiv_rn(ks[1], ks[2]);
        const float sampled = remap_bilinear(src_of(s), h, w, (float)u, (float)t);
        const double sd = (double)sampled;
        double q[3], back[3], kb[3];
        mat3d(Kinv_src, __dmul_rn(u, sd), __dmul_rn(t, sd), sd, q);
        mat4d(R2, q, back);
        const float depth_rep = (float)back[2];
        mat3d(K_ref, back[0], back[1], back[2], kb);
        if (kb[2] == 0.0) kb[2] = __dadd_rn(kb[2], 0.00001);
        const float xr = (float)__ddiv_rn(kb[0], kb[2]), yr = (float)__ddiv_rn(kb[1], kb[2]);
        const double ex = __dsub_rn((double)xr, xd), ey = __dsub_rn((double)yr, yd);
        const double dist = sqrt(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)));
        const float diff = fabsf(__fsub_rn(depth_rep, dref));
        int c_dist = 0, c_diff = 0;   // both ladders grow with the rung, so a view passes the top min(c_dist, c_diff) rungs
        for (int k = 0; k < K; ++k) {
            c_dist += (dist < lad.dist[k]) ? 1 : 0;
            c_diff += (diff < lad.diff[k]) ? 1 : 0;
        }
        const int c = min(c_dist, c_diff);
        if (c < 12) hist_lo += 1ull << (5 * c);
        else if (c < 24) hist_hi += 1ull << (5 * (c - 12));
        else hist_top += 1ull << (5 * (c - 24));
        if (masks_out)
            for (int k = 0; k < K; ++k) masks_out[((size_t)s * K + k) * hw + pix] = (k >= K - c) ? 1 : 0;
        const bool last = c >= 1;
        if (reproj_depth_out) reproj_depth_out[(size_t)s * hw + pix] = last ? depth_rep : 0.0f;
        sum_rep = __fadd_rn(sum_rep, last ? depth_rep : 0.0f);
        n_last += last ? 1 : 0;
    }
    bool geo = n_last >= E;
    int votes = 0;
    for (int k = 0; k < K; ++k) {
        const int bin = K - k;
        const unsigned long long word = bin < 12 ? hist_lo >> (5 * bin) : (bin < 24 ? hist_hi >> (5 * (bin - 12)) : hist_top >> (5 * (bin - 24)));
        votes += (int)(word & 31ull);
        geo = geo || (votes >= S + k);
    }
    const float cf = __ldg(conf + pix);
    double avg = __ddiv_rn((double)__fadd_rn(sum_rep, dref), (double)(n_last + 1));
    if (cf > conf_keep) avg = dd;
    double pa[3], pw[3];
    mat3d(Kinv_ref, __dmul_rn(xd, avg), __dmul_rn(yd, avg), avg, pa);
    mat4d(Einv_ref, pa, pw);
    final_mask[pix] = (cf > conf_thres && geo) ? 1 : 0;
    if (geo_mask) geo_mask[pix] = geo ? 1 : 0;
    depth_avg[pix] = (float)avg;
    points[pix] = (float)pw[0];
    points[(size_t)hw + pix] = (float)pw[1];
    points[(size_t)2 * hw + pix] = (float)pw[2];
}

__global__ void __launch_bounds__(128)
dtu_filter_kernel(const float* __restrict__ ref_depth, const float* __restrict__ srcs_depth, const float* __restrict__ conf,
                  const float* __restrict__ mats, const __grid_constant__ Ladder lad, int K, int S, int E, float conf_thres,
                  float conf_keep, int v, int h, int w, uint8_t* __restrict__ final_mask, uint8_t* __restrict__ geo_mask,
                  float* __restrict__ depth_avg, float* __restrict__ points, uint8_t* __restrict__ masks_out,
                  float* __restrict__ reproj_depth_out) {
    extern __shared__ float sm[];   // REF_FLOATS + v * SRC_FLOATS
    for (int i = threadIdx.x; i < REF_FLOATS + v * SRC_FLOATS; i += blockDim.x) sm[i] = mats[i];
    __syncthreads();
    const int hw = h * w;
    const int pix = blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= hw) return;
    dtu_filter_pixel(pix, sm, ref_depth, [&](int s) { return srcs_depth + (size_t)s * hw; }, conf, lad, K, S, E, conf_thres,
                     conf_keep, v, h, w, final_mask, geo_mask, depth_avg, points, masks_out, reproj_depth_out);
}

// Several reference views in one launch: grid (pixel tiles of 128, n views).  Block y filters reference view y, whose
// depth map and source maps are rows ref_idx[y] and src_idx[y][0 .. src_count[y]) of the one (N,h,w) depth stack, read
// in place; its camera pack is row y of `mats` (REF_FLOATS + vmax * SRC_FLOATS floats, the single-view layout padded to
// vmax sources).  Every view's results are those of dtu_filter_kernel on that view alone.
__global__ void __launch_bounds__(128)
dtu_filter_views_kernel(const float* __restrict__ depths, const int* __restrict__ ref_idx, const int* __restrict__ src_idx,
                        const int* __restrict__ src_count, int vmax, const float* __restrict__ mats,
                        const float* __restrict__ conf, const __grid_constant__ Ladder lad, int K, int S, int E,
                        float conf_thres, float conf_keep, int h, int w, uint8_t* __restrict__ final_mask,
                        uint8_t* __restrict__ geo_mask, float* __restrict__ depth_avg, float* __restrict__ points) {
    extern __shared__ float sm[];   // REF_FLOATS + vmax * SRC_FLOATS floats, then vmax source rows (int)
    int* rows = reinterpret_cast<int*>(sm + REF_FLOATS + vmax * SRC_FLOATS);
    const int view = blockIdx.y;
    const int v = src_count[view];
    const float* pack = mats + (size_t)view * (REF_FLOATS + vmax * SRC_FLOATS);
    for (int i = threadIdx.x; i < REF_FLOATS + v * SRC_FLOATS; i += blockDim.x) sm[i] = pack[i];
    for (int i = threadIdx.x; i < v; i += blockDim.x) rows[i] = src_idx[(size_t)view * vmax + i];
    __syncthreads();
    const int hw = h * w;
    const int pix = blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= hw) return;
    const size_t plane = (size_t)view * hw;
    dtu_filter_pixel(pix, sm, depths + (size_t)ref_idx[view] * hw, [&](int s) { return depths + (size_t)rows[s] * hw; },
                     conf + plane, lad, K, S, E, conf_thres, conf_keep, v, h, w, final_mask + plane,
                     geo_mask ? geo_mask + plane : nullptr, depth_avg + plane, points + 3 * plane, nullptr, nullptr);
}

// the rung thresholds as the kernels' parameter block; fails unless both ladders are non-decreasing
int make_ladder(const double* thr_dist_host, const float* thr_diff_host, int n_rungs, Ladder* lad) {
    for (int k = 0; k < MAX_RUNGS; ++k) {
        lad->dist[k] = k < n_rungs ? thr_dist_host[k] : 0.0;
        lad->diff[k] = k < n_rungs ? thr_diff_host[k] : 0.0f;
        if (k > 0 && k < n_rungs)
            EFFI_REQUIRE(lad->dist[k] >= lad->dist[k - 1] && lad->diff[k] >= lad->diff[k - 1], EFFIMVS_EUNSUPPORTED,
                         "dtu_filter: the threshold ladder must be non-decreasing");
    }
    return EFFIMVS_OK;
}

}  // namespace
}  // namespace effimvs

using namespace effimvs;

extern "C" int effimvs_dtu_filter_f32(const float* ref_depth, const float* srcs_depth, const float* conf, const float* mats,
                                      const double* thr_dist_host, const float* thr_diff_host, int n_rungs, int first_rung,
                                      int full_count, float conf_thres, float conf_keep, int v, int h, int w,
                                      uint8_t* final_mask, uint8_t* geo_mask, float* depth_avg, float* points, uint8_t* masks_out,
                                      float* reproj_depth_out, void* stream) {
    EFFI_REQUIRE(ref_depth && srcs_depth && conf && mats && thr_dist_host && thr_diff_host && final_mask && depth_avg && points,
                 EFFIMVS_EINVAL, "dtu_filter: null pointer");
    EFFI_REQUIRE(v >= 1 && v <= 31 && h > 1 && w > 1, EFFIMVS_EINVAL, "dtu_filter: bad sizes (v in [1,31])");
    EFFI_REQUIRE(n_rungs >= 1 && n_rungs <= MAX_RUNGS && first_rung >= 0, EFFIMVS_EINVAL, "dtu_filter: n_rungs=%d outside [1,%d]", n_rungs, MAX_RUNGS);
    Ladder lad;
    if (const int rc = make_ladder(thr_dist_host, thr_diff_host, n_rungs, &lad)) return rc;
    dim3 block(128), grid(ceil_div(h * w, 128));
    const size_t smem = (size_t)(REF_FLOATS + v * SRC_FLOATS) * sizeof(float);
    dtu_filter_kernel<<<grid, block, smem, (cudaStream_t)stream>>>(ref_depth, srcs_depth, conf, mats, lad, n_rungs, first_rung, full_count,
                                                                  conf_thres, conf_keep, v, h, w, final_mask, geo_mask, depth_avg, points,
                                                                  masks_out, reproj_depth_out);
    return check_launch("dtu_filter_kernel");
}

extern "C" int effimvs_dtu_filter_views_f32(const float* depths, int n_depths, const int* ref_idx, const int* src_idx,
                                            const int* src_count, int vmax, const float* mats, const float* conf,
                                            const double* thr_dist_host, const float* thr_diff_host, int n_rungs, int first_rung,
                                            int full_count, float conf_thres, float conf_keep, int n, int h, int w,
                                            uint8_t* final_mask, uint8_t* geo_mask, float* depth_avg, float* points, void* stream) {
    EFFI_REQUIRE(depths && ref_idx && src_idx && src_count && mats && conf && thr_dist_host && thr_diff_host && final_mask &&
                 depth_avg && points, EFFIMVS_EINVAL, "dtu_filter_views: null pointer");
    EFFI_REQUIRE(n_depths >= 1 && vmax >= 1 && vmax <= 31 && n >= 1 && n <= 65535 && h > 1 && w > 1 &&
                 (long long)h * w <= 0x7fffffffLL - 127, EFFIMVS_EINVAL,
                 "dtu_filter_views: bad sizes (N=%d, vmax=%d in [1,31], n=%d in [1,65535], h=%d, w=%d)", n_depths, vmax, n, h, w);
    EFFI_REQUIRE(n_rungs >= 1 && n_rungs <= MAX_RUNGS && first_rung >= 0, EFFIMVS_EINVAL, "dtu_filter_views: n_rungs=%d outside [1,%d]", n_rungs, MAX_RUNGS);
    Ladder lad;
    if (const int rc = make_ladder(thr_dist_host, thr_diff_host, n_rungs, &lad)) return rc;
    dim3 block(128), grid(ceil_div(h * w, 128), n);
    const size_t smem = (size_t)(REF_FLOATS + vmax * SRC_FLOATS) * sizeof(float) + (size_t)vmax * sizeof(int);
    dtu_filter_views_kernel<<<grid, block, smem, (cudaStream_t)stream>>>(depths, ref_idx, src_idx, src_count, vmax, mats, conf, lad,
                                                                        n_rungs, first_rung, full_count, conf_thres, conf_keep, h, w,
                                                                        final_mask, geo_mask, depth_avg, points);
    return check_launch("dtu_filter_views_kernel");
}
