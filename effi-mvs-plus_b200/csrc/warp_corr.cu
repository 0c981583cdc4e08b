// Fused homography warp + group-wise correlation (+ view aggregation / softmax entropy).
//
// Replaces, without ever materialising the warped (B,C,D,H,W) volume:
//   homo_warping_new                 upstream models/module.py:303-344
//   group-wise correlation           upstream models/Effi_MVS_plus.py:39-40, 222-224
//   weighted view aggregation        upstream models/Effi_MVS_plus.py:52-53, 67, 233-234, 244
//   softmax entropy of a view        upstream models/Effi_MVS_plus.py:43-44
//   local hypothesis generation      upstream models/module.py:554-570
//
// Thread mapping: a warp owns 32 consecutive reference pixels, so every bilinear tap of a channel is
// one (nearly) contiguous 128-byte request on a planar (NCHW) source map, or C/4 128-bit loads per
// lane on a channels-last map; the C reference-feature values of the pixel live in registers and
// are reused across source views and depth planes.
// Reductions over the channels of a group and over the views stay in registers; the stage-1
// kernel reduces softmax statistics over D through shared memory.
#include "common.cuh"
#include "warp_coords.cuh"

namespace effimvs {
namespace {

constexpr int DT = 8;  // depth lanes per block

struct Taps {
    int o_nw;               // linear offset of the north-west corner (y0 * W + x0), clamped to be loadable
    float w_nw, w_ne, w_sw, w_se;
    bool v_nw, v_ne, v_sw, v_se;
    bool any;
};

__device__ __forceinline__ Taps make_taps(const Ray& r, float depth, int H, int W, float inv_half_w, float inv_half_h) {
    float ix, iy;
    sample_coords(r, depth, H, W, inv_half_w, inv_half_h, ix, iy);
    float fx = floorf(ix), fy = floorf(iy);
    Taps t;
    // comparisons are false for NaN/inf -> every corner contributes zero (ATen CUDA behaviour)
    bool x0 = (fx >= 0.0f) && (fx <= (float)(W - 1));
    bool x1 = (fx >= -1.0f) && (fx <= (float)(W - 2));
    bool y0 = (fy >= 0.0f) && (fy <= (float)(H - 1));
    bool y1 = (fy >= -1.0f) && (fy <= (float)(H - 2));
    t.v_nw = x0 && y0; t.v_ne = x1 && y0; t.v_sw = x0 && y1; t.v_se = x1 && y1;
    t.any = t.v_nw || t.v_ne || t.v_sw || t.v_se;
    float ex = __fsub_rn(__fadd_rn(fx, 1.0f), ix);   // ix_se - ix
    float ey = __fsub_rn(__fadd_rn(fy, 1.0f), iy);   // iy_se - iy
    float dx = __fsub_rn(ix, fx);
    float dy = __fsub_rn(iy, fy);
    t.w_nw = __fmul_rn(ex, ey); t.w_ne = __fmul_rn(dx, ey);
    t.w_sw = __fmul_rn(ex, dy); t.w_se = __fmul_rn(dx, dy);
    int xi = t.any ? (int)fx : 0;
    int yi = t.any ? (int)fy : 0;
    t.o_nw = yi * W + xi;
    return t;
}

template <int C, int G>
__device__ __forceinline__ void correlate(const float* __restrict__ src, int HW, int W, const Taps& t,
                                          const float (&ref)[C], float (&sim)[G]) {
    constexpr int CG = C / G;
#pragma unroll
    for (int g = 0; g < G; ++g) sim[g] = 0.0f;
    if (!t.any) return;
    const float* p = src + t.o_nw;
#pragma unroll
    for (int g = 0; g < G; ++g) {
        float acc = 0.0f;
#pragma unroll
        for (int cc = 0; cc < CG; ++cc) {
            const float* q = p + (size_t)(g * CG + cc) * HW;
            float a = t.v_nw ? __ldg(q) : 0.0f;
            float b = t.v_ne ? __ldg(q + 1) : 0.0f;
            float c = t.v_sw ? __ldg(q + W) : 0.0f;
            float d = t.v_se ? __ldg(q + W + 1) : 0.0f;
            float w = a * t.w_nw;
            w = fmaf(b, t.w_ne, w);
            w = fmaf(c, t.w_sw, w);
            w = fmaf(d, t.w_se, w);
            acc = fmaf(w, ref[g * CG + cc], acc);
        }
        sim[g] = acc * (1.0f / CG);
    }
}

// Channels-last (NHWC) feature maps -- what cuDNN's channels_last FPN emits: the C values of a tap
// are contiguous, so a tap is C/4 128-bit loads at immediate offsets from one address and the
// correlation is formed per tap (dot over the channels of a group, then one FMA with the bilinear
// weight): 4x fewer load and address instructions than the planar path.
template <int C, int G>
__device__ __forceinline__ void tap_dot(const float4* __restrict__ p, const float (&ref)[C], float w, float (&sim)[G]) {
    constexpr int CG = C / G;
    float dot[G];
#pragma unroll
    for (int g = 0; g < G; ++g) dot[g] = 0.0f;
#pragma unroll
    for (int cq = 0; cq < C / 4; ++cq) {
        const float4 v = __ldg(p + cq);
        dot[(cq * 4 + 0) / CG] = fmaf(v.x, ref[cq * 4 + 0], dot[(cq * 4 + 0) / CG]);
        dot[(cq * 4 + 1) / CG] = fmaf(v.y, ref[cq * 4 + 1], dot[(cq * 4 + 1) / CG]);
        dot[(cq * 4 + 2) / CG] = fmaf(v.z, ref[cq * 4 + 2], dot[(cq * 4 + 2) / CG]);
        dot[(cq * 4 + 3) / CG] = fmaf(v.w, ref[cq * 4 + 3], dot[(cq * 4 + 3) / CG]);
    }
#pragma unroll
    for (int g = 0; g < G; ++g) sim[g] = fmaf(dot[g], w, sim[g]);
}

template <int C, int G>
__device__ __forceinline__ void correlate_nhwc(const float* __restrict__ src, int W, const Taps& t, const float (&ref)[C],
                                               float (&sim)[G]) {
#pragma unroll
    for (int g = 0; g < G; ++g) sim[g] = 0.0f;
    if (!t.any) return;
    const float4* p = reinterpret_cast<const float4*>(src) + (ptrdiff_t)t.o_nw * (C / 4);
    if (t.v_nw) tap_dot<C, G>(p, ref, t.w_nw, sim);
    if (t.v_ne) tap_dot<C, G>(p + C / 4, ref, t.w_ne, sim);
    if (t.v_sw) tap_dot<C, G>(p + (ptrdiff_t)W * (C / 4), ref, t.w_sw, sim);
    if (t.v_se) tap_dot<C, G>(p + (ptrdiff_t)(W + 1) * (C / 4), ref, t.w_se, sim);
#pragma unroll
    for (int g = 0; g < G; ++g) sim[g] *= (1.0f / (C / G));
}

template <int C, bool NHWC>
__device__ __forceinline__ void load_ref(const float* __restrict__ ref_fea, int b, int pix, int HW, float (&ref)[C]) {
    if (NHWC) {
        const float4* rp = reinterpret_cast<const float4*>(ref_fea + ((size_t)b * HW + pix) * C);
#pragma unroll
        for (int cq = 0; cq < C / 4; ++cq) {
            const float4 v = __ldg(rp + cq);
            ref[cq * 4] = v.x; ref[cq * 4 + 1] = v.y; ref[cq * 4 + 2] = v.z; ref[cq * 4 + 3] = v.w;
        }
    } else {
        const float* rp = ref_fea + (size_t)b * C * HW + pix;
#pragma unroll
        for (int c = 0; c < C; ++c) ref[c] = __ldg(rp + (size_t)c * HW);
    }
}

// One thread owns one reference pixel and DPT consecutive depth planes (8 for G = 1): the reference
// features, the per-view ray rot @ (x,y,1), the view weight and the whole prologue are amortised over
// the planes, and the planes' independent tap loads give the memory system work to overlap.
constexpr int AGG_THREADS = 128;
template <int G> struct PlanesPerThread { static constexpr int value = G >= 4 ? 4 : 8; };   // accumulators: planes x G <= 32

template <int C, int G, bool NHWC>
__global__ void __launch_bounds__(AGG_THREADS)
warp_corr_agg_kernel(const float* __restrict__ ref_fea, SrcPtrs srcs, int n_src, const float* __restrict__ proj,
                     const float* __restrict__ hyp, int hyp_mode, const float* __restrict__ interval,
                     const float* __restrict__ weights, int ray_unfused, int H, int W, int D,
                     float* __restrict__ sim_out, float* __restrict__ hyp_out) {
    pdl_enter();
    constexpr int DPT = PlanesPerThread<G>::value;
    __shared__ float sP[EFFIMVS_MAX_SRC_VIEWS * 12];
    __shared__ const float* sSrc[EFFIMVS_MAX_SRC_VIEWS];
    const int b = blockIdx.z;
    const int HW = H * W;
    const int tid = threadIdx.x;
    for (int i = tid; i < n_src * 12; i += AGG_THREADS) sP[i] = proj[(size_t)b * n_src * 12 + i];
    if (tid < EFFIMVS_MAX_SRC_VIEWS) sSrc[tid] = srcs.p[tid];
    __syncthreads();
    const int pix = blockIdx.x * AGG_THREADS + tid;
    const int d0 = blockIdx.y * DPT;
    if (pix >= HW) return;
    const int yi = pix / W, xi = pix - yi * W;
    const float x = (float)xi, y = (float)yi;
    const float inv_half_w = __fdiv_rn(1.0f, (float)((double)(W - 1) / 2.0));
    const float inv_half_h = __fdiv_rn(1.0f, (float)((double)(H - 1) / 2.0));

    float ref[C];
    load_ref<C, NHWC>(ref_fea, b, pix, HW, ref);

    float depth[DPT], num[DPT][G];
#pragma unroll
    for (int k = 0; k < DPT; ++k) {
        depth[k] = (d0 + k < D) ? fetch_hypothesis(hyp, hyp_mode, interval, b, d0 + k, D, pix, HW) : 1.0f;
        if (hyp_out && d0 + k < D) hyp_out[((size_t)b * D + d0 + k) * HW + pix] = depth[k];
#pragma unroll
        for (int g = 0; g < G; ++g) num[k][g] = 0.0f;
    }
    float den = 0.0f;
    for (int v = 0; v < n_src; ++v) {
        const Ray ray = make_ray(sP + v * 12, x, y, ray_unfused != 0);
        const float* src = sSrc[v] + (size_t)b * C * HW;
        const float w = weights ? __ldg(weights + ((size_t)b * n_src + v) * HW + pix) : 1.0f;
#pragma unroll
        for (int k = 0; k < DPT; ++k) {
            if (d0 + k < D) {
                Taps t = make_taps(ray, depth[k], H, W, inv_half_w, inv_half_h);
                float sim[G];
                if (NHWC) correlate_nhwc<C, G>(src, W, t, ref, sim);
                else correlate<C, G>(src, HW, W, t, ref, sim);
#pragma unroll
                for (int g = 0; g < G; ++g)
                    num[k][g] = weights ? __fadd_rn(num[k][g], __fmul_rn(sim[g], w)) : __fadd_rn(num[k][g], sim[g]);
            }
        }
        den = __fadd_rn(den, w);
    }
    const float div = weights ? __fadd_rn(den, 1e-6f) : (float)n_src;
#pragma unroll
    for (int k = 0; k < DPT; ++k)
        if (d0 + k < D) {
#pragma unroll
            for (int g = 0; g < G; ++g)
                sim_out[(((size_t)b * G + g) * D + d0 + k) * HW + pix] = __fdiv_rn(num[k][g], div);
        }
}

// Stage-1 form: one source view per blockIdx.y; all D planes of 32 pixels per block so that the
// softmax entropy over D can be reduced on chip.
template <int C, bool NHWC>
__global__ void __launch_bounds__(32 * DT)
warp_corr_views_kernel(const float* __restrict__ ref_fea, SrcPtrs srcs, int n_src, const float* __restrict__ proj,
                       const float* __restrict__ hyp, int hyp_mode, int ray_unfused, int H, int W, int D,
                       float* __restrict__ sims_out, float* __restrict__ entropy_out) {
    pdl_enter();
    extern __shared__ float s_sim[];  // [D][32]
    __shared__ float sP[12];
    const int b = blockIdx.z, v = blockIdx.y;
    const int HW = H * W;
    const int tid = threadIdx.y * 32 + threadIdx.x;
    __shared__ const float* sSrc;
    if (tid < 12) sP[tid] = proj[((size_t)b * n_src + v) * 12 + tid];
    if (tid < EFFIMVS_MAX_SRC_VIEWS && tid == v) sSrc = srcs.p[tid];
    __syncthreads();
    const int pix = blockIdx.x * 32 + threadIdx.x;
    const bool live = pix < HW;
    if (live) {
        const int yi = pix / W, xi = pix - yi * W;
        const float x = (float)xi, y = (float)yi;
        const float inv_half_w = __fdiv_rn(1.0f, (float)((double)(W - 1) / 2.0));
        const float inv_half_h = __fdiv_rn(1.0f, (float)((double)(H - 1) / 2.0));
        float ref[C];
        load_ref<C, NHWC>(ref_fea, b, pix, HW, ref);
        const float* src = sSrc + (size_t)b * C * HW;
        float* out = sims_out + (((size_t)b * n_src + v) * D) * HW + pix;
        for (int d = threadIdx.y; d < D; d += DT) {
            const float depth = fetch_hypothesis(hyp, hyp_mode, nullptr, b, d, D, pix, HW);
            Taps t = make_taps(make_ray(sP, x, y, ray_unfused != 0), depth, H, W, inv_half_w, inv_half_h);
            float sim[1];
            if (NHWC) correlate_nhwc<C, 1>(src, W, t, ref, sim);
            else correlate<C, 1>(src, HW, W, t, ref, sim);
            out[(size_t)d * HW] = sim[0];
            s_sim[d * 32 + threadIdx.x] = sim[0];
        }
    }
    __syncthreads();
    if (threadIdx.y == 0 && live) {
        float m = -INFINITY;
        for (int d = 0; d < D; ++d) m = fmaxf(m, s_sim[d * 32 + threadIdx.x]);
        float z = 0.0f;
        for (int d = 0; d < D; ++d) z += expf(s_sim[d * 32 + threadIdx.x] - m);
        float ent = 0.0f;
        for (int d = 0; d < D; ++d) {
            float p = __fdiv_rn(expf(s_sim[d * 32 + threadIdx.x] - m), z);
            ent -= p * logf(p + 1e-7f);
        }
        entropy_out[((size_t)b * n_src + v) * HW + pix] = ent;
    }
}

// homo_warping_new itself (models/module.py:303-344): materialises the warped volume (B,C,D,H,W).  Only
// for callers that need upstream's intermediate; the fused kernels above never write it.
__global__ void __launch_bounds__(128)
homo_warp_kernel(const float* __restrict__ src_fea, const float* __restrict__ proj, const float* __restrict__ hyp, int hyp_mode,
                 int ray_unfused, int C, int H, int W, int D, float* __restrict__ out) {
    pdl_enter();
    __shared__ float sP[12];
    const int b = blockIdx.z, d = blockIdx.y;
    const int HW = H * W;
    if (threadIdx.x < 12) sP[threadIdx.x] = proj[(size_t)b * 12 + threadIdx.x];
    __syncthreads();
    const int pix = blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= HW) return;
    const int yi = pix / W, xi = pix - yi * W;
    const float inv_half_w = __fdiv_rn(1.0f, (float)((double)(W - 1) / 2.0));
    const float inv_half_h = __fdiv_rn(1.0f, (float)((double)(H - 1) / 2.0));
    const float depth = fetch_hypothesis(hyp, hyp_mode, nullptr, b, d, D, pix, HW);
    const Taps t = make_taps(make_ray(sP, (float)xi, (float)yi, ray_unfused != 0), depth, H, W, inv_half_w, inv_half_h);
    const float* p = src_fea + (size_t)b * C * HW + t.o_nw;
    float* o = out + (((size_t)b * C) * D + d) * HW + pix;
    for (int c = 0; c < C; ++c) {
        float v = 0.0f;
        if (t.any) {
            const float* q = p + (size_t)c * HW;
            const float a = t.v_nw ? __ldg(q) : 0.0f, e = t.v_ne ? __ldg(q + 1) : 0.0f;
            const float f = t.v_sw ? __ldg(q + W) : 0.0f, g = t.v_se ? __ldg(q + W + 1) : 0.0f;
            v = fmaf(g, t.w_se, fmaf(f, t.w_sw, fmaf(e, t.w_ne, a * t.w_nw)));
        }
        o[(size_t)c * D * HW] = v;
    }
}

__global__ void weighted_agg_kernel(const float* __restrict__ sims, const float* __restrict__ weights,
                                    int n_src, int D, int HW, float* __restrict__ out) {
    pdl_enter();
    const int b = blockIdx.z;
    const int pix = blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= HW) return;
    float w[EFFIMVS_MAX_SRC_VIEWS];
    float den = 0.0f;
#pragma unroll
    for (int v = 0; v < EFFIMVS_MAX_SRC_VIEWS; ++v) {
        if (v < n_src) {
            w[v] = __ldg(weights + ((size_t)b * n_src + v) * HW + pix);
            den = __fadd_rn(den, w[v]);
        }
    }
    den = __fadd_rn(den, 1e-6f);
    for (int d = blockIdx.y; d < D; d += gridDim.y) {
        float num = 0.0f;
#pragma unroll
        for (int v = 0; v < EFFIMVS_MAX_SRC_VIEWS; ++v)
            if (v < n_src) num = __fadd_rn(num, __fmul_rn(__ldg(sims + (((size_t)b * n_src + v) * D + d) * HW + pix), w[v]));
        out[((size_t)b * D + d) * HW + pix] = __fdiv_rn(num, den);
    }
}

template <int C, int G>
int launch_agg(const float* ref, const SrcPtrs& srcs, int n_src, const float* proj, const float* hyp, int hyp_mode,
               const float* interval, const float* weights, int B, int H, int W, int D, int nhwc, float* sim_out,
               float* hyp_out, cudaStream_t st) {
    dim3 block(AGG_THREADS), grid(ceil_div(H * W, AGG_THREADS), ceil_div(D, PlanesPerThread<G>::value), B);
    if (nhwc)
        launch_kernel(warp_corr_agg_kernel<C, G, true>, grid, block, 0, st, ref, srcs, n_src, proj, hyp, hyp_mode, interval, weights,
                                                                 ray_unfused_for(H, W), H, W, D, sim_out, hyp_out);
    else
        launch_kernel(warp_corr_agg_kernel<C, G, false>, grid, block, 0, st, ref, srcs, n_src, proj, hyp, hyp_mode, interval, weights,
                                                                  ray_unfused_for(H, W), H, W, D, sim_out, hyp_out);
    return check_launch("warp_corr_agg_kernel");
}

template <int C>
int dispatch_g(int G, const float* ref, const SrcPtrs& srcs, int n_src, const float* proj, const float* hyp,
               int hyp_mode, const float* interval, const float* weights, int B, int H, int W, int D, int nhwc,
               float* sim_out, float* hyp_out, cudaStream_t st) {
    switch (G) {
        case 1: return launch_agg<C, 1>(ref, srcs, n_src, proj, hyp, hyp_mode, interval, weights, B, H, W, D, nhwc, sim_out, hyp_out, st);
        case 2: return launch_agg<C, 2>(ref, srcs, n_src, proj, hyp, hyp_mode, interval, weights, B, H, W, D, nhwc, sim_out, hyp_out, st);
        case 4: return launch_agg<C, 4>(ref, srcs, n_src, proj, hyp, hyp_mode, interval, weights, B, H, W, D, nhwc, sim_out, hyp_out, st);
        case 8: return launch_agg<C, 8>(ref, srcs, n_src, proj, hyp, hyp_mode, interval, weights, B, H, W, D, nhwc, sim_out, hyp_out, st);
    }
    set_error("warp_corr_agg: G=%d not in {1,2,4,8}", G);
    return EFFIMVS_EUNSUPPORTED;
}

int fill_srcs(SrcPtrs& s, const float* const* src_fea, int n_src) {
    EFFI_REQUIRE(src_fea && n_src >= 1 && n_src <= EFFIMVS_MAX_SRC_VIEWS, EFFIMVS_EINVAL,
                 "n_src=%d must be in [1,%d]", n_src, EFFIMVS_MAX_SRC_VIEWS);
    for (int i = 0; i < EFFIMVS_MAX_SRC_VIEWS; ++i) s.p[i] = i < n_src ? src_fea[i] : nullptr;
    for (int i = 0; i < n_src; ++i) EFFI_REQUIRE(s.p[i], EFFIMVS_EINVAL, "src_fea[%d] is NULL", i);
    return EFFIMVS_OK;
}

}  // namespace
}  // namespace effimvs

namespace effimvs {
int warp_corr_agg_tile(const float* ref_fea, const SrcPtrs& srcs, int n_src, const float* proj, const float* hyp, int hyp_mode,
                       const float* interval, const float* weights, int B, int C, int H, int W, int D, int G, float* sim_out,
                       float* hyp_out, cudaStream_t st);
int warp_corr_views_tile(const float* ref_fea, const SrcPtrs& srcs, int n_src, const float* proj, const float* hyp, int hyp_mode,
                         int B, int C, int H, int W, int D, float* sims_out, float* entropy_out, cudaStream_t st);
}

using namespace effimvs;

extern "C" int effimvs_warp_corr_agg_f32(const float* ref_fea, const float* const* src_fea, int n_src,
                                         const float* proj, const float* hyp, int hyp_mode, const float* interval,
                                         const float* weights, int B, int C, int H, int W, int D, int G,
                                         int fea_layout, float* sim_out, float* hyp_out, void* stream) {
    EFFI_REQUIRE(ref_fea && proj && hyp && sim_out, EFFIMVS_EINVAL, "warp_corr_agg: null pointer");
    EFFI_REQUIRE(B > 0 && C > 0 && H > 1 && W > 1 && D > 0 && G > 0, EFFIMVS_EINVAL, "warp_corr_agg: bad sizes");
    EFFI_REQUIRE(hyp_mode >= 0 && hyp_mode <= 2, EFFIMVS_EINVAL, "warp_corr_agg: hyp_mode=%d", hyp_mode);
    EFFI_REQUIRE(hyp_mode != EFFIMVS_HYP_LOCAL || (interval && D > 1), EFFIMVS_EINVAL,
                 "warp_corr_agg: HYP_LOCAL needs interval and D > 1");
    EFFI_REQUIRE(C % G == 0, EFFIMVS_EINVAL, "warp_corr_agg: C=%d not divisible by G=%d", C, G);
    EFFI_REQUIRE(fea_layout == EFFIMVS_FEA_NCHW || fea_layout == EFFIMVS_FEA_NHWC, EFFIMVS_EINVAL, "warp_corr_agg: fea_layout=%d", fea_layout);
    const int nhwc = fea_layout == EFFIMVS_FEA_NHWC;
    EFFI_REQUIRE(B <= 65535, EFFIMVS_EUNSUPPORTED, "warp_corr_agg: B too large");
    SrcPtrs s;
    int rc = fill_srcs(s, src_fea, n_src);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (nhwc && (C == 8 || C == 16 || C == 32) && ((uintptr_t)ref_fea & 31) == 0) {
        bool aligned = true;
        for (int i = 0; i < n_src; ++i) aligned = aligned && ((uintptr_t)s.p[i] & 31) == 0;   // 256-bit ld.global.nc.v4.b64 in the tile kernels
        if (aligned)
            return warp_corr_agg_tile(ref_fea, s, n_src, proj, hyp, hyp_mode, interval, weights, B, C, H, W, D, G, sim_out, hyp_out, st);
    }
    switch (C) {
        case 8: return dispatch_g<8>(G, ref_fea, s, n_src, proj, hyp, hyp_mode, interval, weights, B, H, W, D, nhwc, sim_out, hyp_out, st);
        case 16: return dispatch_g<16>(G, ref_fea, s, n_src, proj, hyp, hyp_mode, interval, weights, B, H, W, D, nhwc, sim_out, hyp_out, st);
        case 32: return dispatch_g<32>(G, ref_fea, s, n_src, proj, hyp, hyp_mode, interval, weights, B, H, W, D, nhwc, sim_out, hyp_out, st);
    }
    set_error("warp_corr_agg: C=%d not in {8,16,32}", C);
    return EFFIMVS_EUNSUPPORTED;
}

extern "C" int effimvs_warp_corr_views_f32(const float* ref_fea, const float* const* src_fea, int n_src,
                                           const float* proj, const float* hyp, int hyp_mode,
                                           int B, int C, int H, int W, int D, int fea_layout,
                                           float* sims_out, float* entropy_out, void* stream) {
    EFFI_REQUIRE(ref_fea && proj && hyp && sims_out && entropy_out, EFFIMVS_EINVAL, "warp_corr_views: null pointer");
    EFFI_REQUIRE(B > 0 && H > 1 && W > 1 && D > 0, EFFIMVS_EINVAL, "warp_corr_views: bad sizes");
    EFFI_REQUIRE(hyp_mode == EFFIMVS_HYP_TENSOR || hyp_mode == EFFIMVS_HYP_PLANES, EFFIMVS_EINVAL,
                 "warp_corr_views: hyp_mode=%d", hyp_mode);
    EFFI_REQUIRE(D <= 1024 && B <= 65535, EFFIMVS_EUNSUPPORTED, "warp_corr_views: D=%d > 1024", D);
    EFFI_REQUIRE(fea_layout == EFFIMVS_FEA_NCHW || fea_layout == EFFIMVS_FEA_NHWC, EFFIMVS_EINVAL, "warp_corr_views: fea_layout=%d", fea_layout);
    SrcPtrs s;
    int rc = fill_srcs(s, src_fea, n_src);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (fea_layout == EFFIMVS_FEA_NHWC && (C == 8 || C == 16 || C == 32) && ((uintptr_t)ref_fea & 31) == 0) {
        bool aligned = true;
        for (int i = 0; i < n_src; ++i) aligned = aligned && ((uintptr_t)s.p[i] & 31) == 0;   // 256-bit ld.global.nc.v4.b64 in the tile kernels
        if (aligned) return warp_corr_views_tile(ref_fea, s, n_src, proj, hyp, hyp_mode, B, C, H, W, D, sims_out, entropy_out, st);
    }
    dim3 block(32, DT), grid(ceil_div(H * W, 32), n_src, B);
    size_t smem = (size_t)D * 32 * sizeof(float);
#define EFFI_VIEWS_CASE(CC, L)                                                                                                   \
    {                                                                                                                            \
        if (smem > 48 * 1024) cudaFuncSetAttribute(warp_corr_views_kernel<CC, L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        launch_kernel(warp_corr_views_kernel<CC, L>, grid, block, smem, st, ref_fea, s, n_src, proj, hyp, hyp_mode, ray_unfused_for(H, W), H, W, D, sims_out, entropy_out); \
    }
    const bool nhwc = fea_layout == EFFIMVS_FEA_NHWC;
    switch (C) {
        case 8: if (nhwc) EFFI_VIEWS_CASE(8, true) else EFFI_VIEWS_CASE(8, false) break;
        case 16: if (nhwc) EFFI_VIEWS_CASE(16, true) else EFFI_VIEWS_CASE(16, false) break;
        case 32: if (nhwc) EFFI_VIEWS_CASE(32, true) else EFFI_VIEWS_CASE(32, false) break;
        default:
            set_error("warp_corr_views: C=%d not in {8,16,32}", C);
            return EFFIMVS_EUNSUPPORTED;
    }
#undef EFFI_VIEWS_CASE
    return check_launch("warp_corr_views_kernel");
}

extern "C" int effimvs_weighted_agg_f32(const float* sims, const float* weights, int B, int n_src, int D, int H, int W,
                                        float* out, void* stream) {
    EFFI_REQUIRE(sims && weights && out, EFFIMVS_EINVAL, "weighted_agg: null pointer");
    EFFI_REQUIRE(B > 0 && D > 0 && H > 0 && W > 0 && n_src >= 1 && n_src <= EFFIMVS_MAX_SRC_VIEWS, EFFIMVS_EINVAL,
                 "weighted_agg: bad sizes");
    dim3 block(256), grid(ceil_div(H * W, 256), D < 8 ? D : 8, B);
    launch_kernel(weighted_agg_kernel, grid, block, 0, (cudaStream_t)stream, sims, weights, n_src, D, H * W, out);
    return check_launch("weighted_agg_kernel");
}

extern "C" int effimvs_homo_warp_f32(const float* src_fea, const float* proj, const float* hyp, int hyp_mode,
                                     int B, int C, int H, int W, int D, float* warped_out, void* stream) {
    EFFI_REQUIRE(src_fea && proj && hyp && warped_out, EFFIMVS_EINVAL, "homo_warp: null pointer");
    EFFI_REQUIRE(B > 0 && C > 0 && H > 1 && W > 1 && D > 0 && D <= 65535 && B <= 65535, EFFIMVS_EINVAL, "homo_warp: bad sizes");
    EFFI_REQUIRE(hyp_mode == EFFIMVS_HYP_TENSOR || hyp_mode == EFFIMVS_HYP_PLANES, EFFIMVS_EINVAL, "homo_warp: hyp_mode=%d", hyp_mode);
    dim3 block(128), grid(ceil_div(H * W, 128), D, B);
    launch_kernel(homo_warp_kernel, grid, block, 0, (cudaStream_t)stream, src_fea, proj, hyp, hyp_mode, ray_unfused_for(H, W), C, H, W, D, warped_out);
    return check_launch("homo_warp_kernel");
}
