// Stream compaction of the fusion filters' dense outputs into a coloured point cloud (upstream's vertex / colour
// collection, test_tank.py:517-570, test_dtu_dypcd.py:339-350): every kept pixel's world point, and optionally its colour
// from the reference image, in view order and within a view in raster order.
//
// Three launches for any number of views, in two entry points:
//   effimvs_point_offsets     count_kernel  popcount of the mask per (view, 4096-pixel tile), mask read as 16-byte words
//                             scan_kernel   one CTA: exclusive scan of the tile counts -> tile offsets, view offsets, total
//   effimvs_gather_points_f32 gather_kernel one CTA per tile: the tile's kept points (and colours) compacted in shared
//                             memory, then written as vector stores to the tile's contiguous output range
// Offsets come from the scan, never from atomics, so the output is the same bits on every run.
#include "common.cuh"

namespace effimvs {
namespace {

constexpr int kTile = 4096;                      // pixels per tile
constexpr int kThreads = 256;                    // 16 pixels (one 16-byte mask word) per thread
constexpr int kPix = kTile / kThreads;
constexpr int kScanThreads = 1024;
constexpr int kScanItems = 8;                    // tiles per scan thread and pass
constexpr size_t kGatherSmem = (size_t)kTile * 3 * sizeof(float) + (size_t)kTile * 3;

// bit j of the result: pixel j of the thread's 16 is kept (a nonzero mask byte)
template <bool VEC>
__device__ __forceinline__ unsigned keep_bits(const uint8_t* mask, int npx) {
    unsigned keep = 0;
    if (VEC) {
        if (npx >= kPix) {
            const uint4 m = __ldg(reinterpret_cast<const uint4*>(mask));
            const unsigned words[4] = {m.x, m.y, m.z, m.w};
#pragma unroll
            for (int k = 0; k < 16; ++k) keep |= (((words[k >> 2] >> (8 * (k & 3))) & 0xffu) != 0u) << k;
        }
    } else {
#pragma unroll
        for (int k = 0; k < 16; ++k)
            if (k < npx && mask[k] != 0) keep |= 1u << k;
    }
    return keep;
}

// exclusive block scan of one int per thread (kThreads threads); *total gets the block's sum
__device__ __forceinline__ int block_exclusive_scan(int x, int* s_warp, int* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += y;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int v = lane < kThreads / 32 ? s_warp[lane] : 0;
#pragma unroll
        for (int d = 1; d < kThreads / 32; d <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, v, d);
            if (lane >= d) v += y;
        }
        if (lane < kThreads / 32) s_warp[lane] = v;      // inclusive sums of the warps
    }
    __syncthreads();
    *total = s_warp[kThreads / 32 - 1];
    return inc - x + (warp ? s_warp[warp - 1] : 0);
}

// counts[view * tiles + tile] = kept pixels of that tile
template <bool VEC>
__global__ void __launch_bounds__(kThreads) count_kernel(const uint8_t* __restrict__ mask, long long P, int tiles,
                                                          long long* __restrict__ counts) {
    __shared__ int s_warp[kThreads / 32];
    const int b = blockIdx.x / tiles, t = blockIdx.x - b * tiles;
    const long long p0 = (long long)t * kTile;
    const int npx = (int)min((long long)kTile, P - p0) - (int)threadIdx.x * kPix;
    const unsigned keep = keep_bits<VEC>(mask + (long long)b * P + p0 + threadIdx.x * kPix, npx);
    int total;
    block_exclusive_scan(__popc(keep), s_warp, &total);
    if (threadIdx.x == 0) counts[blockIdx.x] = total;
}

// in place: counts (m) -> exclusive tile offsets; view_offsets[b] = offset of view b's first tile, view_offsets[n] = total
__global__ void __launch_bounds__(kScanThreads) scan_kernel(long long* __restrict__ tile_off, int m, int tiles, int n,
                                                             long long* __restrict__ view_offsets) {
    __shared__ long long s_warp[kScanThreads / 32];
    __shared__ long long s_carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < m; base += kScanThreads * kScanItems) {
        const int first = base + threadIdx.x * kScanItems;
        long long v[kScanItems], sum = 0;
#pragma unroll
        for (int k = 0; k < kScanItems; ++k) {
            v[k] = first + k < m ? tile_off[first + k] : 0;
            sum += v[k];
        }
        long long inc = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const long long y = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += y;
        }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            long long w = s_warp[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const long long y = __shfl_up_sync(0xffffffffu, w, d);
                if (lane >= d) w += y;
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        long long run = s_carry + inc - sum + (warp ? s_warp[warp - 1] : 0);
#pragma unroll
        for (int k = 0; k < kScanItems; ++k) {
            const int g = first + k;
            if (g < m) {
                tile_off[g] = run;
                if (g % tiles == 0) view_offsets[g / tiles] = run;
            }
            run += v[k];
        }
        __syncthreads();                                  // every thread has read s_carry and s_warp
        if (threadIdx.x == 0) s_carry += s_warp[31];
        __syncthreads();
    }
    if (threadIdx.x == 0) view_offsets[n] = s_carry;
}

// The colour rule: trunc(clamp(x * 255, 0, 255)) with an IEEE multiply; fmaxf returns 0 for a NaN product.  On [0,1] this
// is NumPy's (x * 255).astype(np.uint8); outside [0,1] (where that cast is undefined) the clamp is this library's rule.
__device__ __forceinline__ uint8_t color_byte(float x) {
    return (uint8_t)__float2uint_rz(fminf(fmaxf(__fmul_rn(x, 255.0f), 0.0f), 255.0f));
}

// the thread's 16 values of one plane; VEC: one 16-pixel group, fully inside the view (P % 16 == 0) and 16-byte aligned
template <bool VEC>
__device__ __forceinline__ void load16(const float* __restrict__ src, int npx, float (&v)[kPix]) {
    if (VEC) {
        if (npx >= kPix) {
#pragma unroll
            for (int k = 0; k < kPix / 4; ++k) {
                const float4 q = __ldg(reinterpret_cast<const float4*>(src) + k);
                v[4 * k] = q.x, v[4 * k + 1] = q.y, v[4 * k + 2] = q.z, v[4 * k + 3] = q.w;
            }
        }
    } else {
#pragma unroll
        for (int k = 0; k < kPix; ++k) v[k] = k < npx ? __ldg(src + k) : 0.0f;
    }
}

template <bool VEC, bool COLOR>
__global__ void __launch_bounds__(kThreads) gather_kernel(const uint8_t* __restrict__ mask, const float* __restrict__ points,
                                                           const float* __restrict__ images, const int* __restrict__ image_rows,
                                                           long long P, int tiles, const long long* __restrict__ tile_off,
                                                           float* __restrict__ points_out, uint8_t* __restrict__ colors_out) {
    extern __shared__ __align__(16) unsigned char smem[];
    float* s_pts = reinterpret_cast<float*>(smem);                      // (k,3) rows of the tile
    uint8_t* s_col = smem + (size_t)kTile * 3 * sizeof(float);          // (k,3) bytes
    __shared__ int s_warp[kThreads / 32];
    const int b = blockIdx.x / tiles, t = blockIdx.x - b * tiles;
    const long long p0 = (long long)t * kTile + threadIdx.x * kPix;      // the thread's first pixel in the view
    const int npx = (int)min((long long)kPix, P - p0);                   // <= 0: the thread is past the view's end
    const unsigned keep = keep_bits<VEC>(mask + (long long)b * P + p0, npx);
    int k;
    const int at = block_exclusive_scan(__popc(keep), s_warp, &k);
    if (keep) {
        float v[3][kPix];
#pragma unroll
        for (int c = 0; c < 3; ++c) load16<VEC>(points + ((long long)b * 3 + c) * P + p0, npx, v[c]);
        int r = at;
#pragma unroll
        for (int j = 0; j < kPix; ++j)
            if (keep >> j & 1u) {
                s_pts[3 * r] = v[0][j], s_pts[3 * r + 1] = v[1][j], s_pts[3 * r + 2] = v[2][j];
                ++r;
            }
        if (COLOR) {
            const long long row = image_rows[b];
#pragma unroll
            for (int c = 0; c < 3; ++c) load16<VEC>(images + (row * 3 + c) * P + p0, npx, v[c]);
            r = at;
#pragma unroll
            for (int j = 0; j < kPix; ++j)
                if (keep >> j & 1u) {
                    s_col[3 * r] = color_byte(v[0][j]), s_col[3 * r + 1] = color_byte(v[1][j]), s_col[3 * r + 2] = color_byte(v[2][j]);
                    ++r;
                }
        }
    }
    __syncthreads();
    if (k == 0) return;
    const long long first = tile_off[blockIdx.x] * 3;                   // the tile's first output element
    const int e = 3 * k;
    {   // points: scalar head up to a 16-byte boundary of points_out (16-byte aligned), float4 body, scalar tail
        float* dst = points_out + first;
        const int head = min(e, (int)((4 - (first & 3)) & 3));
        const int body = (e - head) >> 2;
        if ((int)threadIdx.x < head) dst[threadIdx.x] = s_pts[threadIdx.x];
        for (int q = threadIdx.x; q < body; q += kThreads) {
            const float* s = s_pts + head + 4 * q;
            reinterpret_cast<float4*>(dst + head)[q] = make_float4(s[0], s[1], s[2], s[3]);
        }
        const int tail = head + 4 * body;
        if ((int)threadIdx.x < e - tail) dst[tail + threadIdx.x] = s_pts[tail + threadIdx.x];
    }
    if (COLOR) {   // colours: the same with 16-byte words
        uint8_t* dst = colors_out + first;
        const int head = min(e, (int)((16 - (first & 15)) & 15));
        const int body = (e - head) >> 4;
        if ((int)threadIdx.x < head) dst[threadIdx.x] = s_col[threadIdx.x];
        for (int q = threadIdx.x; q < body; q += kThreads) {
            const uint8_t* s = s_col + head + 16 * q;
            unsigned w[4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
                w[i] = (unsigned)s[4 * i] | (unsigned)s[4 * i + 1] << 8 | (unsigned)s[4 * i + 2] << 16 | (unsigned)s[4 * i + 3] << 24;
            reinterpret_cast<uint4*>(dst + head)[q] = make_uint4(w[0], w[1], w[2], w[3]);
        }
        const int tail = head + 16 * body;
        if ((int)threadIdx.x < e - tail) dst[tail + threadIdx.x] = s_col[tail + threadIdx.x];
    }
}

inline bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

// tiles per view, or -1 when n * tiles does not fit a grid
int tiles_per_view(int n, int h, int w) {
    if (n < 1 || h < 1 || w < 1) return -1;
    const long long P = (long long)h * w, tiles = (P + kTile - 1) / kTile;
    return (long long)n * tiles <= 0x7fffffffLL ? (int)tiles : -1;
}

template <bool VEC, bool COLOR>
int launch_gather(const uint8_t* mask, const float* points, const float* images, const int* image_rows, long long P, int tiles,
                  int grid, const long long* tile_off, float* points_out, uint8_t* colors_out, cudaStream_t stream) {
    auto fn = gather_kernel<VEC, COLOR>;
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGatherSmem);
    EFFI_REQUIRE(e == cudaSuccess, EFFIMVS_ECUDA, "gather_points: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    launch_kernel(fn, dim3(grid), dim3(kThreads), kGatherSmem, stream, mask, points, images, image_rows, P, tiles, tile_off,
                  points_out, colors_out);
    return check_launch("gather_points_kernel");
}

}  // namespace
}  // namespace effimvs

using namespace effimvs;

extern "C" size_t effimvs_point_offsets_workspace_bytes(int n, int h, int w) {
    const int tiles = tiles_per_view(n, h, w);
    return tiles < 0 ? 0 : (size_t)n * tiles * sizeof(long long);
}

extern "C" int effimvs_point_offsets(const uint8_t* final_mask, int n, int h, int w, void* workspace, size_t workspace_bytes,
                                     int64_t* view_offsets, void* stream) {
    EFFI_REQUIRE(final_mask && workspace && view_offsets, EFFIMVS_EINVAL, "point_offsets: null pointer");
    const int tiles = tiles_per_view(n, h, w);
    EFFI_REQUIRE(tiles > 0, EFFIMVS_EINVAL, "point_offsets: bad sizes n=%d h=%d w=%d", n, h, w);
    EFFI_REQUIRE(aligned16(workspace), EFFIMVS_EINVAL, "point_offsets: workspace must be 16-byte aligned");
    const size_t need = effimvs_point_offsets_workspace_bytes(n, h, w);
    EFFI_REQUIRE(workspace_bytes >= need, EFFIMVS_EWORKSPACE, "point_offsets: workspace of %zu bytes, %zu needed", workspace_bytes, need);
    const long long P = (long long)h * w;
    const int m = n * tiles;
    long long* tile_off = static_cast<long long*>(workspace);
    const cudaStream_t s = (cudaStream_t)stream;
    if (P % 16 == 0 && aligned16(final_mask))
        launch_kernel(count_kernel<true>, dim3(m), dim3(kThreads), 0, s, final_mask, P, tiles, tile_off);
    else
        launch_kernel(count_kernel<false>, dim3(m), dim3(kThreads), 0, s, final_mask, P, tiles, tile_off);
    int rc = check_launch("point_count_kernel");
    if (rc != EFFIMVS_OK) return rc;
    launch_kernel(scan_kernel, dim3(1), dim3(kScanThreads), 0, s, tile_off, m, tiles, n, reinterpret_cast<long long*>(view_offsets));
    return check_launch("point_scan_kernel");
}

extern "C" int effimvs_gather_points_f32(const uint8_t* final_mask, const float* points, const float* images, int n_images,
                                         const int* image_rows, int n, int h, int w, const void* workspace,
                                         size_t workspace_bytes, float* points_out, uint8_t* colors_out, void* stream) {
    EFFI_REQUIRE(final_mask && points && workspace && points_out, EFFIMVS_EINVAL, "gather_points: null pointer");
    EFFI_REQUIRE(!images || (image_rows && colors_out && n_images >= 1), EFFIMVS_EINVAL,
                 "gather_points: images need image_rows, colors_out and n_images >= 1");
    const int tiles = tiles_per_view(n, h, w);
    EFFI_REQUIRE(tiles > 0, EFFIMVS_EINVAL, "gather_points: bad sizes n=%d h=%d w=%d", n, h, w);
    EFFI_REQUIRE(aligned16(workspace) && aligned16(points_out) && (!images || aligned16(colors_out)), EFFIMVS_EINVAL,
                 "gather_points: workspace, points_out and colors_out must be 16-byte aligned");
    const size_t need = effimvs_point_offsets_workspace_bytes(n, h, w);
    EFFI_REQUIRE(workspace_bytes >= need, EFFIMVS_EWORKSPACE, "gather_points: workspace of %zu bytes, %zu needed", workspace_bytes, need);
    const long long P = (long long)h * w;
    const bool vec = P % 16 == 0 && aligned16(final_mask) && aligned16(points) && (!images || aligned16(images));
    const long long* tile_off = static_cast<const long long*>(workspace);
    const cudaStream_t s = (cudaStream_t)stream;
    const int grid = n * tiles;
    if (images)
        return vec ? launch_gather<true, true>(final_mask, points, images, image_rows, P, tiles, grid, tile_off, points_out, colors_out, s)
                   : launch_gather<false, true>(final_mask, points, images, image_rows, P, tiles, grid, tile_off, points_out, colors_out, s);
    return vec ? launch_gather<true, false>(final_mask, points, nullptr, nullptr, P, tiles, grid, tile_off, points_out, nullptr, s)
               : launch_gather<false, false>(final_mask, points, nullptr, nullptr, P, tiles, grid, tile_off, points_out, nullptr, s);
}
