// Implicit-GEMM 3x3 convolution (stride 1, zero padding 1) on channels-last fp32 maps for the 2-D convolutions of the
// ConvGRU update block (SURVEY section 8(f) row 3), on the 5th-generation tensor cores (tcgen05, fp32 accumulation in
// tensor memory), with the per-pixel glue that follows each convolution in upstream as the epilogue:
//
//   ProjectionInput.convc2 / convd2 / convd / convc   upstream models/update.py:69-99
//   ConvGRU.convz / convr / convq + gate arithmetic   upstream models/update.py:33-49
//   DepthHead.conv1                                   upstream models/update.py:10-27
//   BasicUpdateBlock.mask[0]                          upstream models/update.py:106-110
//
// Precision: the arithmetic class of TF32 -- operands carry 11 significant bits (1 + 10 mantissa), products are exact,
// accumulation is fp32 -- which is what PyTorch's cuDNN convolutions use for these layers under its default
// torch.backends.cudnn.allow_tf32 = True.  The operands are fed to the tensor core as IEEE half (fp16: the same 10 mantissa
// bits as TF32 in half the bytes, so an MMA covers K = 16 channels instead of 8; measured, an MMA of this shape costs the
// tensor pipe ~130-170 clk of A-operand streaming whatever its N, so halving their number is what counts).  Activations are
// rounded to nearest when staged (cvt.rn.satfinite: |x| > 65504 saturates -- the inputs of these layers are tanh / sigmoid
// / relu outputs of O(1) -- and |x| < 6e-5 goes gradually to an absolute error of 3e-8), weights when packed.  Callers
// that need fp32 products use the bf16x3 instantiations below or keep cuDNN.
//
// Precision bf16x3 (effimvs_conv2d_bf16x3*, opt-in): the arithmetic class of the 3-D nets' default mode (conv3d_tc.cu).
// Every operand is carried as a pair hi = bf16_rn(x), lo = bf16_rn(x - hi) (x - hi is exact in fp32; together ~2^-16
// relative), and each K step issues hi.hi + hi.lo + lo.hi into the same fp32 accumulator -- fp32's exponent range, no
// saturation.  A staged input row holds the hi copy followed by the lo copy (each in the layout below), the packed
// weights the hi image followed by the lo image (36 Cin Cout bytes, both resident); K phases are at most 32 channels so
// that 64 -> 64 (147 KB of weights) fits one CTA per SM with three stages.  Operand precision is a template parameter:
// the f16 instantiations compile to the same instructions as without it.
//
// Formulation ("row sweep", input stationary).  A unit is a strip of 128 output pixels x R consecutive output rows of
// one image.  Input row i of the strip (130 pixels with the x halo, zero beyond the image) is staged ONCE in shared
// memory as [channel group of 8][pixel][8 halves]: for every x tap the 128 x 16-channel operand is then the canonical
// K-major / no-swizzle UMMA matrix at a 16-byte shifted address (no im2col), and the row is multiplied once against
// the STACKED weights [w(ky=2) ; w(ky=1) ; w(ky=0)] -- one MMA of N = 3 Cout writes the partial sums of output rows
// i-1, i, i+1, whose accumulators sit side by side in a ring of TMEM slots.  So every input row is read from global
// memory once per unit, streamed through the tensor pipe once per x tap, and an output row is complete when input
// row i+1 has passed.  The whole weight tensor (18 Cin Cout bytes) is resident in shared memory.
//
// Warp roles of a 416-thread CTA (persistent over units; one or two CTAs per SM):
//   warps 5-12 producers : 2 x 128-bit global loads per lane (8 channels of a pixel; two channel segments = a virtual
//                          concat, so cat[h, x] / cat[r*h, x] are never materialised; zero outside the image), fp32 -> fp16,
//                          conflict-free 128-bit shared stores, fence.proxy.async, one mbarrier arrival per warp
//                                                                             (3- or 4-stage ring, K phases of <= 64 channels)
//   warp 4     MMA issuer: warp-uniform loops, one lane issues tcgen05.mma kind::f16 and commits -> stage empty / row complete
//   warps 0-3  epilogue  : TMEM lanes 32w..32w+31 = pixels; tcgen05.ld, transpose through shared memory, then per mode
//                          BIAS / BIAS_RELU    out = [relu](acc + bias)
//                          ADD_RELU            out = relu(acc + addend[pixel])                (encoder tail: context term)
//                          GRU_GATES           z = sigmoid(acc[:h] + b) -> zbuf;  out = sigmoid(acc[h:] + b) * h_prev
//                          GRU_UPDATE          out = (1 - z) * out + z * tanh(acc + b)        (in place on the hidden state)
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cstdlib>

#include "common.cuh"

namespace effimvs {
namespace {

constexpr int C2_TM = 128;                       // output pixels of a row tile = MMA M
constexpr int C2_ROWPX = 136;                    // staged pixels of an input row: 128 + 2 halo, padded to a multiple of 8
constexpr int C2_CG_BYTES = C2_ROWPX * 16;       // one channel group (8 halves per pixel) of a staged row
constexpr int C2_STAGES = 4;                     // input-row ring (at most; 3 when shared memory is short)
constexpr int C2_RING = 16;                      // TMEM accumulator slots (output rows in flight), at most; a power of two >= 4
constexpr int C2_PROD_WARPS = 8;
constexpr int C2_PROD_GROUPS = 2;                  // producer warps work in groups that take alternate fills: two fills' loads in flight
constexpr int C2_GROUP_WARPS = C2_PROD_WARPS / C2_PROD_GROUPS;
constexpr int C2_MMA_WARP = 4, C2_PROD_WARP0 = 5;
constexpr int C2_THREADS = (C2_PROD_WARP0 + C2_PROD_WARPS) * 32;   // 416
constexpr int C2_EPI_STRIDE = 144;                // bytes per pixel row of an epilogue warp's transpose buffer (32 channels + 16 pad)
constexpr int C2_EPI_BYTES = 4 * 32 * C2_EPI_STRIDE;
constexpr int C2_MAX_COUT = 128;
constexpr int C2_F16 = 0, C2_BF16X3 = 1;          // operand precision (template parameter of the kernel)

struct C2Params {
    const float* in0; long long ps0; int c0;     // channel segment 0: pointer to (pixel 0, channel 0), pixel stride in floats
    const float* in1; long long ps1; int c1;     // channel segment 1 (c1 = 0: none)
    int cin, cout, coutp;                        // coutp = cout rounded up to a multiple of 16
    int B, H, W;
    int kc, n_phases;                            // channels per K phase (16, 32 or 64), cin / kc
    int strips, R, chunks, n_units;              // unit = (image, row chunk, strip)
    int mode;
    const float* bias;
    float* out; long long out_ps;
    const float* aux0; long long aux0_ps;        // ADD_RELU: addend; GRU_GATES: h_prev; GRU_UPDATE: z
    float* aux1; long long aux1_ps;              // GRU_GATES: z out
    int tmem_cols, w_bytes, stage_bytes, n_stages;
    int gw;                                      // producer warps per group (2 groups): 4 (416-thread CTA) or 2 (288 threads, three CTAs per SM)
    int ring;                                    // accumulator slots in use: the fewer wrap-arounds, the fewer split MMAs
    long long* tl;                               // profiling: timeline buffer [3 roles][64 steps][4 events] of clock64, written by CTA 0
    int debug;                                   // EFFIMVS_CONV2D_DEBUG bits (builds with -DEFFIMVS_CONV2D_PROFILING only; results wrong): 1 no MMAs, 2 no operand loads, 4 no epilogue body, 8 no TMEM reads,
                                                 // 16 producers do not wait for free stages, 32 plain arrives instead of tcgen05.commit, 64 epilogue = wait + arrive
};

// ------------------------------------------------------------------------------------------------
// PTX wrappers (same conventions as conv3d_tc.cu)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// try_wait parks the thread in hardware for a short, system-defined time; between polls the lane sleeps.  Tried and measured:
// a long suspend-time hint on try_wait itself makes threads wake late (32 -> 32 at 800 x 592: 41 -> 64 us with a 20 us hint);
// backoffs of 32 / 64 / 200 ns between polls are indistinguishable; pure test_wait polling is no faster.
// A barrier that never completes must surface as a launch failure, not as a hung GPU.
__device__ __forceinline__ uint32_t mbar_try(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return done;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    for (uint32_t spin = 0; spin < (1u << 24); ++spin) {
        if (mbar_try(bar, parity)) return;
        if (spin > 4) __nanosleep(32);
    }
    __trap();
}
// The same for a whole warp: ONE lane polls (an mbarrier poll is a shared-memory atomic; 32 lanes polling one address
// serialise in the shared-memory pipe and starve the stores of the working warps -- measured), and the warp leaves on a vote
// so that the compiler sees warp-uniform control flow after the wait.
__device__ __forceinline__ void mbar_wait_warp(uint64_t* bar, uint32_t parity) {
    const bool poller = (threadIdx.x & 31) == 0;
    for (uint32_t spin = 0; spin < (1u << 24); ++spin) {
        const uint32_t done = poller ? mbar_try(bar, parity) : 0u;
        if (__any_sync(0xffffffffu, done)) return;
        if (spin > 4) __nanosleep(32);
    }
    __trap();
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// K-major, no-swizzle shared-memory matrix descriptor: core matrix = 8 rows x 16 bytes (8 halves) contiguous;
// LBO = byte distance between the two 8-element K halves of an MMA (K = 16), SBO = distance between 8-row groups.
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
    return d;
}
// kind::f16 instruction descriptor: D = f32, A = B = f16 (format 0), both K-major, M = 128, N = n
__device__ __forceinline__ uint32_t umma_idesc_tf32(int n) {
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(C2_TM >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accum) : "memory");
}
// bf16x3: three MMAs into one accumulator -- hi.hi, hi.lo (B's lo image blo16 units on), lo.hi (A's lo copy alo16 units
// on); f16: the one MMA.  A and B are descriptors, the offsets in 16-byte units.
template <int PREC>
__device__ __forceinline__ void umma_op(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum, uint32_t alo16, uint32_t blo16) {
    umma_tf32(tmem_d, da, db, idesc, accum);
    if (PREC == C2_BF16X3) {
        umma_tf32(tmem_d, da, db + blo16, idesc, 1u);
        umma_tf32(tmem_d, da + alo16, db, idesc, 1u);
    }
}
// instruction descriptor per precision: bf16x3 sets A and B format to bf16 (bits 7-9, 10-12 = 1)
template <int PREC>
__device__ __forceinline__ uint32_t umma_idesc_p(int n) {
    return umma_idesc_tf32(n) | (PREC == C2_BF16X3 ? (1u << 7) | (1u << 10) : 0u);
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                   "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
                 "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                   "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
                   "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
                   "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
// eight consecutive floats with one 256-bit load (one request per 32-byte sector)
struct F8 { unsigned long long a, b, c, d; };
__device__ __forceinline__ F8 ldg_nc8(const float* p) {
    F8 o;
    asm volatile("ld.global.nc.v4.b64 {%0, %1, %2, %3}, [%4];" : "=l"(o.a), "=l"(o.b), "=l"(o.c), "=l"(o.d) : "l"(p));
    return o;
}
// two floats (a 64-bit pair, low word first) -> packed IEEE halves, round to nearest, saturating at +-65504
__device__ __forceinline__ uint32_t pack_half2(unsigned long long pair) {
    float lo, hi;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(pair));
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
// two floats (low word first) -> packed bf16 hi = bf16_rn(x) and lo = bf16_rn(x - hi); no saturation (fp32's exponent range)
__device__ __forceinline__ void split_bf16x2(unsigned long long pair, uint32_t& hi, uint32_t& lo) {
    float a, b;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(pair));
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));
    const float ra = a - __uint_as_float(hi << 16), rb = b - __uint_as_float(hi & 0xffff0000u);
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(rb), "f"(ra));
}
__device__ __forceinline__ float to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
__device__ __forceinline__ float4 ldg_nc4(const float* p) {
    float4 v;
    asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
// Gate activations of the epilogue: 1 / (1 + e^-x) and 1 - 2 / (1 + e^2x) on the special-function unit (ex2 + rcp, absolute
// error ~1e-7 -- three orders below the operand rounding of the convolution that feeds them).  The IEEE expf / division /
// tanhf sequences of update_glue.cu cost ~30 instructions per element, and the four epilogue warps of a CTA would spend
// longer on them than the tensor pipe spends on the row.
__device__ __forceinline__ float sigmoid_t(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float tanh_t(float x) { return 1.0f - __fdividef(2.0f, 1.0f + __expf(2.0f * x)); }
// The same two functions on channel pairs with packed fp32 arithmetic (add / mul / fma .f32x2: one issue slot for two lanes of
// work -- the epilogue warps are instruction bound); the exponentials and reciprocals stay scalar special-function ops.
typedef unsigned long long pk2;
__device__ __forceinline__ pk2 pk(float lo, float hi) { pk2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void unpk(pk2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ pk2 add2(pk2 a, pk2 b) { pk2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ pk2 mul2(pk2 a, pk2 b) { pk2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ pk2 fma2(pk2 a, pk2 b, pk2 c) { pk2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ float ex2f(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcpf(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// 1 / (1 + 2^(s * x)) per channel of a pair: s = -log2(e) gives sigmoid(x), s = 2 log2(e) gives (1 - tanh(x)) / 2
__device__ __forceinline__ pk2 inv1pexp2(pk2 x, float s) {
    float e0, e1;
    unpk(mul2(x, pk(s, s)), e0, e1);
    float d0, d1;
    unpk(add2(pk(ex2f(e0), ex2f(e1)), pk(1.0f, 1.0f)), d0, d1);
    return pk(rcpf(d0), rcpf(d1));
}

#ifdef EFFIMVS_CONV2D_TIMELINE   // profiling builds only: clock64 stamps of CTA 0's roles (tools/conv2d_check.py timeline)
#define C2_TL(role, step, ev) do { if (P.tl && blockIdx.x == 0 && (step) < 64) P.tl[((role) * 64 + (step)) * 4 + (ev)] = clock64(); } while (0)
#else
#define C2_TL(role, step, ev) do { } while (0)
#endif

// Second half of the epilogue for one chunk of 4 * CPP columns of a warp's 32 pixels: lane = (pixel within a pass, 4-channel
// group), 32 / (32 / CPP) passes, four at a time so that the shared-memory reads, the aux-map loads and the stores of
// different pixels overlap.  Every role of this kernel is a single-warp chain whose speed is its instruction count (measured:
// ~6 clk per executed instruction), hence the compile-time mode, the pointer-increment addressing and the predicate-free
// path for warps whose 32 pixels all lie inside the image.
template <int CPP, int MODE, bool FULL>
__device__ __forceinline__ void epilogue_rows_m(const C2Params& P, const uint8_t* __restrict__ ebuf, const float* __restrict__ sbias, int lane,
                                                int cb, int h, long long rowpix, int xw0, int W) {
    constexpr int PPP = 32 / CPP, NPASS = 32 / PPP;
    const int sub = lane & (CPP - 1), pxl = lane / CPP;
    const int ch = cb + sub * 4;
    if (ch >= P.cout) return;
    const float4 b4 = *reinterpret_cast<const float4*>(sbias + ch);
    const long long pix0 = rowpix + xw0 + pxl;
    const uint8_t* src = ebuf + pxl * C2_EPI_STRIDE + sub * 16;
    const bool gate_r = MODE == EFFIMVS_CONV2D_GRU_GATES && ch >= h;
    // main output pointer and the aux map read per pixel (none for the plain modes and the z half of the gates)
    float* o;
    long long o_step;                                   // floats between the pixels of consecutive passes
    if (MODE == EFFIMVS_CONV2D_GRU_GATES) {
        o = gate_r ? P.out + pix0 * P.out_ps + (ch - h) : P.aux1 + pix0 * P.aux1_ps + ch;
        o_step = (gate_r ? P.out_ps : P.aux1_ps) * PPP;
    } else {
        o = P.out + pix0 * P.out_ps + ch;
        o_step = P.out_ps * PPP;
    }
    constexpr bool AUX = MODE == EFFIMVS_CONV2D_ADD_RELU || MODE == EFFIMVS_CONV2D_GRU_UPDATE || MODE == EFFIMVS_CONV2D_GRU_GATES;
    const bool has_aux = MODE == EFFIMVS_CONV2D_GRU_GATES ? gate_r : AUX;
    const float* ax = AUX ? P.aux0 + pix0 * P.aux0_ps + (gate_r ? ch - h : ch) : nullptr;
    const long long ax_step = AUX ? P.aux0_ps * PPP : 0;
    const int n_ok = FULL ? NPASS : (W - xw0 - pxl + PPP - 1) / PPP;      // passes whose pixel lies inside the image
#pragma unroll
    for (int g0 = 0; g0 < NPASS; g0 += 4) {
        float4 a[4], d[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            a[j] = *reinterpret_cast<const float4*>(src + (g0 + j) * PPP * C2_EPI_STRIDE);
            if (AUX) {
                d[j] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                if (has_aux && (FULL || g0 + j < n_ok)) d[j] = ldg_nc4(ax + (g0 + j) * ax_step);
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (!FULL && g0 + j >= n_ok) continue;
            float* op = o + (g0 + j) * o_step;
            float4 w;
            if (MODE == EFFIMVS_CONV2D_BIAS || MODE == EFFIMVS_CONV2D_BIAS_RELU) {
                w.x = __fadd_rn(a[j].x, b4.x); w.y = __fadd_rn(a[j].y, b4.y); w.z = __fadd_rn(a[j].z, b4.z); w.w = __fadd_rn(a[j].w, b4.w);
                if (MODE == EFFIMVS_CONV2D_BIAS_RELU) { w.x = fmaxf(w.x, 0.0f); w.y = fmaxf(w.y, 0.0f); w.z = fmaxf(w.z, 0.0f); w.w = fmaxf(w.w, 0.0f); }
            } else if (MODE == EFFIMVS_CONV2D_ADD_RELU) {
                w.x = fmaxf(__fadd_rn(a[j].x, d[j].x), 0.0f); w.y = fmaxf(__fadd_rn(a[j].y, d[j].y), 0.0f);
                w.z = fmaxf(__fadd_rn(a[j].z, d[j].z), 0.0f); w.w = fmaxf(__fadd_rn(a[j].w, d[j].w), 0.0f);
            } else if (MODE == EFFIMVS_CONV2D_GRU_GATES) {
                // z = sigmoid(z_pre + b_z)  |  sigmoid(r_pre + b_r) * h_prev
                pk2 s01 = inv1pexp2(add2(pk(a[j].x, a[j].y), pk(b4.x, b4.y)), -1.4426950408889634f);
                pk2 s23 = inv1pexp2(add2(pk(a[j].z, a[j].w), pk(b4.z, b4.w)), -1.4426950408889634f);
                if (gate_r) { s01 = mul2(s01, pk(d[j].x, d[j].y)); s23 = mul2(s23, pk(d[j].z, d[j].w)); }
                unpk(s01, w.x, w.y);
                unpk(s23, w.z, w.w);
            } else {
                // GRU_UPDATE: out = (1 - z) * out + z * tanh(q_pre + b_q), z = d
                const float4 hq = *reinterpret_cast<const float4*>(op);
                // tanh(t) = 1 - 2 u with u = 1 / (1 + e^(2t));  h' = (1 - z) h + z tanh(t)
                const pk2 one = pk(1.0f, 1.0f), m2 = pk(-2.0f, -2.0f), m1 = pk(-1.0f, -1.0f);
                const pk2 z01 = pk(d[j].x, d[j].y), z23 = pk(d[j].z, d[j].w);
                const pk2 q01 = fma2(inv1pexp2(add2(pk(a[j].x, a[j].y), pk(b4.x, b4.y)), 2.8853900817779268f), m2, one);
                const pk2 q23 = fma2(inv1pexp2(add2(pk(a[j].z, a[j].w), pk(b4.z, b4.w)), 2.8853900817779268f), m2, one);
                unpk(fma2(z01, q01, mul2(fma2(z01, m1, one), pk(hq.x, hq.y))), w.x, w.y);
                unpk(fma2(z23, q23, mul2(fma2(z23, m1, one), pk(hq.z, hq.w))), w.z, w.w);
            }
            *reinterpret_cast<float4*>(op) = w;
        }
    }
}
template <int CPP, int MODE>
__device__ __forceinline__ void epilogue_rows(const C2Params& P, const uint8_t* __restrict__ ebuf, const float* __restrict__ sbias, int lane,
                                              int cb, int h, long long rowpix, int xw0, int W) {
    if (xw0 + 32 <= W) epilogue_rows_m<CPP, MODE, true>(P, ebuf, sbias, lane, cb, h, rowpix, xw0, W);
    else epilogue_rows_m<CPP, MODE, false>(P, ebuf, sbias, lane, cb, h, rowpix, xw0, W);
}

struct Unit { int b, y0, y1, x0; };
__device__ __forceinline__ Unit unit_of(const C2Params& P, int u) {
    Unit t;
    const int per_img = P.strips * P.chunks;
    t.b = u / per_img;
    const int r = u - t.b * per_img;
    const int chunk = r / P.strips, strip = r - chunk * P.strips;   // strips fastest: neighbouring CTAs share halo rows in L2
    t.y0 = chunk * P.R;
    t.y1 = min(t.y0 + P.R, P.H);
    t.x0 = strip * C2_TM;
    return t;
}

// One instantiation per (epilogue mode, channel groups of a K phase, operand precision): every role of the kernel is a single-warp chain whose speed
// is its instruction count, and three CTAs x three roles share the SM's instruction cache -- a run-time mode switch, a generic item
// mapping and the profiling switches of the first version cost measurably (see DESIGN, appendix A), so they are compile-time here.
template <int MODE, int GROUPS, int PREC>
__global__ void __launch_bounds__(C2_THREADS, 2)
conv2d_tc_kernel(const __grid_constant__ C2Params P, const uint8_t* __restrict__ wpk) {
#ifdef EFFIMVS_CONV2D_PROFILING
    const int dbg = dbg;             // EFFIMVS_CONV2D_DEBUG switches (tools/conv2d_check.py probe / scale / rows) only in profiling builds
#else
    constexpr int dbg = 0;
#endif
    constexpr int KC = GROUPS * 8;       // channels per K phase
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) uint64_t bar_afull[C2_STAGES], bar_aempty[C2_STAGES], bar_tfull[C2_RING], bar_tempty[C2_RING], bar_w;
    __shared__ uint32_t tmem_base_s;
    __shared__ __align__(16) float sbias[C2_MAX_COUT];
    // warp index through a shuffle: tells the compiler that it is warp-uniform, so the role branches below are uniform control flow
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
    uint8_t* wsm = smem;
    uint8_t* astage = smem + P.w_bytes;

    if (warp == C2_MMA_WARP) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"((uint32_t)P.tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        for (int s = 0; s < C2_STAGES; ++s) { mbar_init(&bar_afull[s], P.gw); mbar_init(&bar_aempty[s], 1); }
        for (int a = 0; a < C2_RING; ++a) { mbar_init(&bar_tfull[a], 1); mbar_init(&bar_tempty[a], 4); }   // (only P.ring of them are used)
        mbar_init(&bar_w, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    // the packed weights are a constant of the model (effimvs_conv2d_tf32_pack, once per layer): their copy into shared memory
    // starts before the programmatic-launch wait, together with the TMEM allocation and barrier set-up above -- the part of
    // this kernel that overlaps the tail of its predecessor.  Maps and bias are only touched after the wait.
    if (tid == C2_PROD_WARP0 * 32) {
        mbar_expect_tx(&bar_w, (uint32_t)P.w_bytes);
        bulk_g2s(wsm, wpk, (uint32_t)P.w_bytes, &bar_w);
    }
    pdl_trigger();
    pdl_wait();
    if (tid < C2_MAX_COUT) sbias[tid] = (P.bias && tid < P.cout) ? __ldg(P.bias + tid) : 0.0f;
    __syncthreads();
    const uint32_t tmem = tmem_base_s;
    const int H = P.H, W = P.W;

    if (warp >= C2_PROD_WARP0) {
        // ---------------- producers ----------------
        // A lane owns (pixel, group of 8 channels) items: two 128-bit global loads, four packed conversions, one 128-bit
        // shared store, up to 5 items = 10 loads in flight per lane.  The warps form two groups that take alternate fills, so
        // the global-memory round trips of consecutive fills overlap.
        const int pw = warp - C2_PROD_WARP0, grp = pw / P.gw, pwg = pw - grp * P.gw;
        const int S = P.n_stages;
        constexpr int groups = GROUPS;                                 // 16-byte channel groups per phase: 2, 4 or 8
        // groups >= 4: an item = 8 pixels x 4 groups (a pixel's 32 channels = 128 contiguous bytes); groups == 2: 16 pixels x 2 groups
        const int pxl = groups >= 4 ? (lane & 7) : (lane & 15), cgl0 = groups >= 4 ? (lane >> 3) : (lane >> 4);
        const int px_per_item = groups >= 4 ? 8 : 16, px_items = (C2_ROWPX + px_per_item - 1) / px_per_item;
        const int n_items = px_items * (groups >= 4 ? groups >> 2 : 1);
        const int ps0i = (int)P.ps0, ps1i = (int)P.ps1;                  // a row of a map is < 2^31 floats
        constexpr int NIT = PREC == C2_BF16X3 ? 4 : 5;                    // items in flight per lane (bf16x3: two stores each)
        uint32_t fill = 0;
        for (int u = blockIdx.x; u < P.n_units; u += gridDim.x) {
            const Unit t = unit_of(P, u);
            const int i_lo = max(t.y0 - 1, 0), i_hi = min(t.y1, H - 1);
            for (int i = i_lo; i <= i_hi; ++i) {
                const long long rowpix = ((long long)t.b * H + i) * W;
                for (int p = 0; p < P.n_phases; ++p, ++fill) {
                    if ((int)(fill % C2_PROD_GROUPS) != grp) continue;     // the other group's fill
                    const uint32_t s = fill % S, n = fill / S;
                    if (lane == 0) mbar_wait(&bar_aempty[s], (n & 1) ^ 1);
                    __syncwarp();
                    if (pw == 0 && lane == 0) C2_TL(0, fill, 0);
                    uint8_t* dst = astage + (size_t)s * P.stage_bytes;
                    const float* r0 = P.in0 + rowpix * P.ps0;          // (pixel 0 of the row, channel 0) of the two segments
                    const float* r1 = P.in1 + rowpix * P.ps1 - P.c0;
                    const int ch0 = p * KC + cgl0 * 8, xb = t.x0 - 1 + pxl;
                    for (int it0 = pwg; it0 < n_items; it0 += NIT * P.gw) {
                        F8 v[NIT];
                        uint32_t off[NIT];
#pragma unroll
                        for (int k = 0; k < NIT; ++k) {
                            const int it = it0 + P.gw * k;
                            v[k].a = v[k].b = v[k].c = v[k].d = 0ull;
                            off[k] = 0xffffffffu;
                            if (it < n_items && !(dbg & 2)) {
                                const int cgq = it >= px_items ? 1 : 0, g = it - (cgq ? px_items : 0);   // n_items <= 2 px_items
                                const int pxo = g * px_per_item, px = pxo + pxl, x = xb + pxo;
                                if (px < C2_ROWPX) off[k] = (uint32_t)((cgq * 4 + cgl0) * C2_CG_BYTES + px * 16);
                                if (px < C2_TM + 2 && (unsigned)x < (unsigned)W) {
                                    const int gc = ch0 + cgq * 32;
                                    v[k] = ldg_nc8(gc < P.c0 ? r0 + (x * ps0i + gc) : r1 + (x * ps1i + gc));
                                }
                            }
                        }
#pragma unroll
                        for (int k = 0; k < NIT; ++k) {
                            if (off[k] != 0xffffffffu) {
                                uint4 q;
                                if (PREC == C2_BF16X3) {
                                    uint4 l;    // the lo copy sits GROUPS channel groups after the hi copy
                                    split_bf16x2(v[k].a, q.x, l.x); split_bf16x2(v[k].b, q.y, l.y);
                                    split_bf16x2(v[k].c, q.z, l.z); split_bf16x2(v[k].d, q.w, l.w);
                                    *reinterpret_cast<uint4*>(dst + off[k] + GROUPS * C2_CG_BYTES) = l;
                                } else {
                                    q.x = pack_half2(v[k].a); q.y = pack_half2(v[k].b); q.z = pack_half2(v[k].c); q.w = pack_half2(v[k].d);
                                }
                                *reinterpret_cast<uint4*>(dst + off[k]) = q;
                            }
                        }
                    }
                    if (dbg & 512) {
                        __syncwarp();
                        if (lane == 0) { fence_async_smem(); mbar_arrive(&bar_afull[s]); }
                    } else {
                        if (!(dbg & 256)) fence_async_smem();           // generic-proxy stores -> visible to the tensor core's async proxy
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&bar_afull[s]);
                    }
                    if (pw == 0 && lane == 0) C2_TL(0, fill, 1);
                }
            }
        }
    } else if (warp == C2_MMA_WARP) {
        // ---------------- MMA issuer ----------------
        // The whole warp walks the loops (warp-uniform control flow: descriptors and addresses stay in uniform registers,
        // which is where tcgen05.mma takes them from -- inside one big `if (lane == 0)` every operand of every MMA costs an R2UR
        // move, measured ~170 clk per MMA; the barrier waits exit on a warp vote for the same reason); lane 0 issues the MMAs
        // and commits.
        {
            const bool leader = lane == 0;
            const int S = P.n_stages;
            const uint32_t coutp = (uint32_t)P.coutp;
            const uint32_t blk16 = (96u * coutp) >> 4;                // a packed weight block [2 K halves][3 coutp rows][16 B] in 16-byte units
            const uint64_t bdesc0 = umma_desc(smem_u32(wsm), 3u * coutp * 16u, 128);
            constexpr int ksteps = KC >> 4;
            const bool two_max = 3 * P.coutp > 256;                   // an MMA spans at most two of the three stacked row blocks
            const bool mma_on = !(dbg & 1);
            const uint32_t rm = (uint32_t)P.ring - 1u, rs = (uint32_t)__ffs(P.ring) - 1u;
            constexpr uint32_t alo16 = (GROUPS * C2_CG_BYTES) >> 4;                 // bf16x3: lo copy of a staged row
            const uint32_t blo16 = PREC == C2_BF16X3 ? (uint32_t)P.w_bytes >> 5 : 0u;  // bf16x3: lo weight image (second half)
            mbar_wait_warp(&bar_w, 0);
            __syncwarp();
            uint32_t fill = 0, seq_base = 0;
            for (int u = blockIdx.x; u < P.n_units; u += gridDim.x) {
                const Unit t = unit_of(P, u);
                const int i_lo = max(t.y0 - 1, 0), i_hi = min(t.y1, H - 1);
                for (int i = i_lo; i <= i_hi; ++i) {
                    // output rows r_lo..r_hi are fed by input row i through weight row blocks kyb0.. (ky = 2 - kyb); their
                    // accumulators are the ring slots (seq0 + k) & (ring - 1).  A row is fresh (first partial sum) when it is i + 1, or row 0.
                    const int r_lo = max(i - 1, t.y0), r_hi = min(i + 1, t.y1 - 1), nt = r_hi - r_lo + 1;
                    const uint32_t seq0 = seq_base + (uint32_t)(r_lo - t.y0);
                    const uint32_t kyb0 = (uint32_t)(r_lo - (i - 1));
                    uint32_t fresh = 0;
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        if (k < nt && ((r_lo + k == i + 1) || (i == 0 && r_lo + k == 0))) {
                            fresh |= 1u << k;
                            mbar_wait_warp(&bar_tempty[(seq0 + k) & rm], (((seq0 + k) >> rs) & 1u) ^ 1u);   // slot drained by the epilogue
                        }
                    }
                    tc_fence_after();
                    if (leader) C2_TL(1, fill, 0);
                    // runs of stacked blocks: split where the ring wraps (slot 3 -> 0) and, for wide layers, after two blocks
                    const bool brk1 = nt > 1 && ((seq0 + 1) & rm) == 0;
                    const bool brk2 = nt > 2 && ((((seq0 + 2) & rm) == 0) || (two_max && !brk1));
                    const int lenA = (nt > 1 && !brk1) ? ((nt > 2 && !brk2) ? 3 : 2) : 1;
                    const int lenB = nt - lenA;
                    const uint32_t dA = tmem + (seq0 & rm) * coutp, dB = tmem + ((seq0 + (uint32_t)lenA) & rm) * coutp;
                    const uint32_t boffA = kyb0 * coutp, boffB = (kyb0 + (uint32_t)lenA) * coutp;          // 16-byte units (one per row)
                    const uint32_t idA = umma_idesc_p<PREC>(lenA * P.coutp), idB = umma_idesc_p<PREC>(lenB * P.coutp), id1 = umma_idesc_p<PREC>(P.coutp);
                    for (int p = 0; p < P.n_phases; ++p, ++fill) {
                        const uint32_t s = fill % S, n = fill / S;
                        mbar_wait_warp(&bar_afull[s], n & 1);
                        if (leader) C2_TL(1, fill, 1);
                        if (!(dbg & 2048)) tc_fence_after();
                        const uint64_t adesc0 = umma_desc(smem_u32(astage + (size_t)s * P.stage_bytes), C2_CG_BYTES, 128);
                        uint64_t bstep = bdesc0 + (uint64_t)((uint32_t)(p * ksteps * 3) * blk16);
                        if (leader && mma_on) {
                            int q0 = 0;
                            if (p == 0 && fresh) {
                                // first K step of a row with fresh accumulators: one MMA per output row, overwriting where fresh
#pragma unroll
                                for (int k = 0; k < 3; ++k)
                                    if (k < nt)
                                        umma_op<PREC>(tmem + ((seq0 + k) & rm) * coutp, adesc0, bstep + (uint64_t)((kyb0 + k) * coutp), id1, ((fresh >> k) & 1u) ^ 1u, alo16, blo16);
                                q0 = 1;
                                bstep += blk16;
                            }
                            // K steps q = j * 3 + kx: channel groups 2j, 2j + 1 of the stage, x tap kx (a 16-byte shift)
                            const uint64_t bA = bstep + (uint64_t)boffA, bB = bstep + (uint64_t)boffB;
                            uint32_t boff = 0;
                            for (int q = q0; q < 3 * ksteps; ++q, boff += blk16) {
                                const int j = q / 3, kx = q - 3 * j;
                                const uint64_t adesc = adesc0 + (uint64_t)(uint32_t)(j * 2 * (C2_CG_BYTES >> 4) + kx);
                                umma_op<PREC>(dA, adesc, bA + boff, idA, 1u, alo16, blo16);
                                if (lenB > 0) umma_op<PREC>(dB, adesc, bB + boff, idB, 1u, alo16, blo16);
                            }
                        }
                        if (leader) {
                            C2_TL(1, fill, 2);
                            if (dbg & 32) mbar_arrive(&bar_aempty[s]);
                            else umma_commit(&bar_aempty[s]);                 // stage reusable once these MMAs retire
                            C2_TL(1, fill, 3);
                        }
                        __syncwarp();
                    }
                    if (!leader) {
                    } else if (dbg & 32) {
                        if (i - 1 >= t.y0 && i - 1 < t.y1) mbar_arrive(&bar_tfull[(seq_base + (uint32_t)(i - 1 - t.y0)) & rm]);
                        if (i == H - 1 && i < t.y1) mbar_arrive(&bar_tfull[(seq_base + (uint32_t)(i - t.y0)) & rm]);
                    } else {
                        if (i - 1 >= t.y0 && i - 1 < t.y1) umma_commit(&bar_tfull[(seq_base + (uint32_t)(i - 1 - t.y0)) & rm]);
                        if (i == H - 1 && i < t.y1) umma_commit(&bar_tfull[(seq_base + (uint32_t)(i - t.y0)) & rm]);
                    }
                }
                seq_base += (uint32_t)(t.y1 - t.y0);
            }
        }
        __syncwarp();
    } else {
        // ---------------- epilogue ----------------
        // TMEM lane = pixel: a thread reads the accumulators of ITS pixel (32 columns at a time), but a channels-last map
        // wants a warp to write whole pixels side by side.  So the raw sums go through a per-warp transpose buffer
        // (144-byte pixel rows: conflict-free 128-bit accesses both ways) and come back as (pixel, 4-channel group) per lane:
        // every global access of the epilogue -- the stores and the aux maps of the fused modes -- then covers full 128-byte lines.
        uint8_t* ebuf = astage + (size_t)P.n_stages * P.stage_bytes + (size_t)warp * (32 * C2_EPI_STRIDE);
        uint32_t seq = 0;
        const int h = MODE == EFFIMVS_CONV2D_GRU_GATES ? P.cout / 2 : P.cout;
        for (int u = blockIdx.x; u < P.n_units; u += gridDim.x) {
            const Unit t = unit_of(P, u);
            const int xw0 = t.x0 + warp * 32;
            for (int r = t.y0; r < t.y1; ++r, ++seq) {
                const uint32_t slot = seq & (uint32_t)(P.ring - 1);
                const long long rowpix = ((long long)t.b * H + r) * W;
                if (tid == 0) C2_TL(2, seq, 0);
                // the aux maps of the fused modes are read once the accumulators arrive: ask for their lines now (a lane per
                // pixel: 32 pixels x h channels of this warp), so that the reads in epilogue_rows hit L1 instead of waiting on L2
                if (MODE >= EFFIMVS_CONV2D_ADD_RELU && xw0 + lane < W && !(dbg & 4096)) {
                    const float* a0 = P.aux0 + (rowpix + xw0 + lane) * P.aux0_ps;
                    for (int c = 0; c < h; c += 32) asm volatile("prefetch.global.L1 [%0];" ::"l"(a0 + c));
                    if (MODE == EFFIMVS_CONV2D_GRU_UPDATE) {
                        const float* o0 = P.out + (rowpix + xw0 + lane) * P.out_ps;
                        for (int c = 0; c < h; c += 32) asm volatile("prefetch.global.L1 [%0];" ::"l"(o0 + c));
                    }
                }
                if (lane == 0) mbar_wait(&bar_tfull[slot], (seq >> (__ffs(P.ring) - 1)) & 1u);
                __syncwarp();
                if (tid == 0) C2_TL(2, seq, 1);
                if (!(dbg & 1024)) tc_fence_after();
                const uint32_t lane_base = tmem + slot * (uint32_t)P.coutp + ((uint32_t)(warp * 32) << 16);
                if (dbg & 64) {
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bar_tempty[slot]);
                    continue;
                }
                for (int cb = 0; cb < P.coutp; cb += 32) {
                    const int ncol = min(32, P.coutp - cb);
                    {
                        float4* mine = reinterpret_cast<float4*>(ebuf + lane * C2_EPI_STRIDE);
                        if (ncol == 32) {
                            float v[32];
                            if (!(dbg & 8)) tmem_ld32(lane_base + (uint32_t)cb, v);
                            else for (int q = 0; q < 32; ++q) v[q] = 0.0f;
#pragma unroll
                            for (int q = 0; q < 8; ++q) mine[q] = make_float4(v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
                        } else {
                            float v[16];
                            if (!(dbg & 8)) tmem_ld16(lane_base + (uint32_t)cb, v);
                            else for (int q = 0; q < 16; ++q) v[q] = 0.0f;
#pragma unroll
                            for (int q = 0; q < 4; ++q) mine[q] = make_float4(v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
                        }
                    }
                    const bool last = cb + 32 >= P.coutp;
                    if (last && !(dbg & 1024)) tc_fence_before();
                    __syncwarp();
                    if (last && lane == 0) mbar_arrive(&bar_tempty[slot]);     // last TMEM read of this row: the slot goes back to the MMA warp
                    if (last && tid == 0) C2_TL(2, seq, 2);
                    if (!(dbg & 4)) {
                        if (ncol == 32) epilogue_rows<8, MODE>(P, ebuf, sbias, lane, cb, h, rowpix, xw0, W);
                        else epilogue_rows<4, MODE>(P, ebuf, sbias, lane, cb, h, rowpix, xw0, W);
                    }
                    __syncwarp();      // the buffer is rewritten by the next chunk / row
                }
                if (tid == 0) C2_TL(2, seq, 3);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == C2_MMA_WARP)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)P.tmem_cols) : "memory");
}

// packed weights = the shared-memory image: block ((p * kc/16 + j) * 3 + kx) = [K half (2)][row (3 coutp)][8 halves],
// row = kyb * coutp + co with ky = 2 - kyb, channel = (p * kc/16 + j) * 16 + half * 8 + e; fp16 (round to nearest), zero beyond cout.
__global__ void conv2d_pack_kernel(const float* __restrict__ w, int cin, int cout, int coutp, __half* __restrict__ dst) {
    const int total = 9 * cin * coutp;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int e = i & 7;
        const int row = (i >> 3) % (3 * coutp);
        const int half = (i / (8 * 3 * coutp)) & 1;
        const int blk = i / (16 * 3 * coutp);
        const int kx = blk % 3, c16 = blk / 3;
        const int kyb = row / coutp, co = row - kyb * coutp;
        const int ci = c16 * 16 + half * 8 + e;
        float v = 0.0f;
        if (co < cout) v = w[(((size_t)co * cin + ci) * 3 + (2 - kyb)) * 3 + kx];
        dst[i] = __float2half_rn(fminf(fmaxf(v, -65504.0f), 65504.0f));
    }
}
// bf16x3: the same layout twice -- dst[0, n) = bf16_rn(w), dst[n, 2n) = bf16_rn(w - bf16_rn(w)), n = 9 cin coutp; no saturation.
__global__ void conv2d_pack_bf16x3_kernel(const float* __restrict__ w, int cin, int cout, int coutp, __nv_bfloat16* __restrict__ dst) {
    const int total = 9 * cin * coutp;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int e = i & 7;
        const int row = (i >> 3) % (3 * coutp);
        const int half = (i / (8 * 3 * coutp)) & 1;
        const int blk = i / (16 * 3 * coutp);
        const int kx = blk % 3, c16 = blk / 3;
        const int kyb = row / coutp, co = row - kyb * coutp;
        const int ci = c16 * 16 + half * 8 + e;
        float v = 0.0f;
        if (co < cout) v = w[(((size_t)co * cin + ci) * 3 + (2 - kyb)) * 3 + kx];
        const __nv_bfloat16 hi = __float2bfloat16_rn(v);
        dst[i] = hi;
        dst[total + i] = __float2bfloat16_rn(v - __bfloat162float(hi));
    }
}

int pow2_cols(int n) { int c = 32; while (c < n) c <<= 1; return c; }
// channels per K phase: the whole input when it is 16, 32 or 64 channels, else 32- or 16-channel phases; bf16x3 (a stage holds
// two copies): at most 32
int phase_channels(int cin) { return (cin == 16 || cin == 32 || cin == 64) ? cin : (cin % 32 == 0 ? 32 : 16); }
int phase_channels(int cin, int prec) { return prec == C2_BF16X3 ? (cin % 32 == 0 ? 32 : 16) : phase_channels(cin); }
// copies of each operand: the bf16x3 weight image and staged rows hold hi and lo
int operand_copies(int prec) { return prec == C2_BF16X3 ? 2 : 1; }

size_t packed_bytes(int cin, int cout, int prec) {
    if (cin <= 0 || cout <= 0) return 0;
    const int coutp = (cout + 15) / 16 * 16;
    return (size_t)18 * operand_copies(prec) * cin * coutp;
}

int supported(int cin, int cout, int prec) {
    if (cin < 16 || cin % 16 != 0 || cout < 4 || cout % 4 != 0 || cout > C2_MAX_COUT) return 0;
    const int coutp = (cout + 15) / 16 * 16;
    const int kc = phase_channels(cin, prec);
    const size_t smem = packed_bytes(cin, cout, prec) + (size_t)3 * operand_copies(prec) * (kc / 8) * C2_CG_BYTES + C2_EPI_BYTES;
    if (smem > 224 * 1024) return 0;
    if (4 * coutp > 512) return 0;
    return 1;
}

int pack(const char* name, int prec, const float* w, int cin, int cout, void* packed, void* stream) {
    EFFI_REQUIRE(w && packed, EFFIMVS_EINVAL, "%s: null pointer", name);
    EFFI_REQUIRE(supported(cin, cout, prec), EFFIMVS_EUNSUPPORTED, "%s: cin=%d cout=%d not supported", name, cin, cout);
    const int coutp = (cout + 15) / 16 * 16;
    const int total = 9 * cin * coutp;
    const int grid = std::min(ceil_div(total, 256), 1024);
    if (prec == C2_BF16X3) {
        conv2d_pack_bf16x3_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(w, cin, cout, coutp, (__nv_bfloat16*)packed);
        return check_launch("conv2d_pack_bf16x3_kernel");
    }
    conv2d_pack_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(w, cin, cout, coutp, (__half*)packed);
    return check_launch("conv2d_pack_kernel");
}

long long* g_conv2d_timeline = nullptr;

// the host side of both families: validation, budgets and the launch of the instantiation for (mode, K phase, precision)
int launch(const char* name, int prec, const float* in0, long long in0_ps, int c0, const float* in1, long long in1_ps, int c1,
           const void* packed, const float* bias, int cout, int B, int H, int W, int mode,
           float* out, long long out_ps, const float* aux0, long long aux0_ps, float* aux1,
           long long aux1_ps, void* stream) {
    EFFI_REQUIRE(in0 && packed && out, EFFIMVS_EINVAL, "%s: null pointer", name);
    EFFI_REQUIRE(B > 0 && H >= 2 && W >= 1, EFFIMVS_EINVAL, "%s: bad shape %dx%dx%d", name, B, H, W);
    EFFI_REQUIRE(c0 > 0 && c0 % 8 == 0 && c1 >= 0 && c1 % 8 == 0 && (c1 == 0 || in1), EFFIMVS_EINVAL, "%s: bad channel segments %d + %d", name, c0, c1);
    const int cin = c0 + c1;
    EFFI_REQUIRE(supported(cin, cout, prec), EFFIMVS_EUNSUPPORTED, "%s: cin=%d cout=%d not supported", name, cin, cout);
    EFFI_REQUIRE(mode >= EFFIMVS_CONV2D_BIAS && mode <= EFFIMVS_CONV2D_GRU_UPDATE, EFFIMVS_EINVAL, "%s: bad mode %d", name, mode);
    EFFI_REQUIRE(in0_ps >= c0 && in0_ps % 8 == 0 && (c1 == 0 || (in1_ps >= c1 && in1_ps % 8 == 0)) && out_ps % 4 == 0,
                 EFFIMVS_EINVAL, "%s: input pixel strides must be multiples of 8 floats, the output's of 4", name);
    EFFI_REQUIRE((((uintptr_t)in0 | (uintptr_t)in1) & 31) == 0 && (((uintptr_t)out | (uintptr_t)aux0 | (uintptr_t)aux1 | (uintptr_t)packed) & 15) == 0,
                 EFFIMVS_EINVAL, "%s: input maps must be 32-byte aligned, the other pointers 16-byte aligned", name);
    EFFI_REQUIRE((long long)W * in0_ps < (1ll << 31) && (long long)W * in1_ps < (1ll << 31), EFFIMVS_EUNSUPPORTED, "%s: a row of a map must be below 2^31 floats", name);
    if (mode == EFFIMVS_CONV2D_ADD_RELU) EFFI_REQUIRE(aux0 && aux0_ps % 4 == 0, EFFIMVS_EINVAL, "%s: ADD_RELU needs the addend map", name);
    if (mode == EFFIMVS_CONV2D_GRU_GATES)
        EFFI_REQUIRE(aux0 && aux1 && bias && cout % 32 == 0 && aux0_ps % 4 == 0 && aux1_ps % 4 == 0, EFFIMVS_EINVAL,
                     "%s: GRU_GATES needs h_prev, the z buffer, the bias and cout = 2h with h a multiple of 16", name);
    if (mode == EFFIMVS_CONV2D_GRU_UPDATE) EFFI_REQUIRE(aux0 && bias && aux0_ps % 4 == 0, EFFIMVS_EINVAL, "%s: GRU_UPDATE needs z and the bias", name);

    C2Params P;
    P.in0 = in0; P.ps0 = in0_ps; P.c0 = c0;
    P.in1 = in1 ? in1 : in0; P.ps1 = in1 ? in1_ps : in0_ps; P.c1 = c1;
    P.cin = cin; P.cout = cout; P.coutp = (cout + 15) / 16 * 16;
    P.B = B; P.H = H; P.W = W;
    P.kc = phase_channels(cin, prec);
    P.n_phases = cin / P.kc;
    P.mode = mode;
    P.tl = g_conv2d_timeline;
    P.debug = getenv("EFFIMVS_CONV2D_DEBUG") ? atoi(getenv("EFFIMVS_CONV2D_DEBUG")) : 0;
    P.bias = bias;
    P.out = out; P.out_ps = out_ps;
    P.aux0 = aux0; P.aux0_ps = aux0_ps;
    P.aux1 = aux1; P.aux1_ps = aux1_ps;
    P.w_bytes = (int)packed_bytes(cin, cout, prec);
    P.stage_bytes = operand_copies(prec) * (P.kc / 8) * C2_CG_BYTES;
    // CTAs per SM: three 288-thread CTAs (two producer warps per group) when shared memory, registers and TMEM allow -- every
    // role of this kernel is a chain of per-row latencies, so resident CTAs are what fills the SM --, else two or one
    // 416-thread CTAs.  The accumulator ring takes the TMEM columns that is left per CTA (the fewer wrap-arounds, the fewer
    // split MMAs), at least 4 slots.
    const size_t fixed = (size_t)P.w_bytes + C2_EPI_BYTES;
    const size_t smem3 = fixed + 3 * (size_t)P.stage_bytes;
    int per_sm = smem3 + 1024 <= 75 * 1024 && 4 * P.coutp <= 128 ? 3 : (smem3 + 1024 <= 113 * 1024 && 4 * P.coutp <= 256 ? 2 : 1);
    if (const char* e = getenv("EFFIMVS_CONV2D_CTAS")) per_sm = std::max(1, std::min(per_sm, atoi(e)));
    P.gw = per_sm == 3 ? 2 : 4;
    const int tmem_budget = per_sm == 3 ? 128 : (per_sm == 2 ? 256 : 512);
    P.ring = 4;
    while (P.ring < C2_RING && 2 * P.ring * P.coutp <= tmem_budget) P.ring *= 2;
    if (const char* e = getenv("EFFIMVS_CONV2D_RING")) { int r = atoi(e); if ((r == 4 || r == 8 || r == 16) && r * P.coutp <= tmem_budget) P.ring = r; }
    P.tmem_cols = pow2_cols(P.ring * P.coutp);
    // a fourth stage where it is free
    const size_t smem_budget = per_sm == 3 ? 75 * 1024 : (per_sm == 2 ? 113 * 1024 : 225 * 1024);
    P.n_stages = (smem3 + P.stage_bytes + 1024 <= smem_budget) ? 4 : 3;
    if (const char* e = getenv("EFFIMVS_CONV2D_STAGES")) { int n = atoi(e); if (n == 3 || (n == 4 && smem3 + P.stage_bytes + 1024 <= smem_budget)) P.n_stages = n; }
    const size_t smem = fixed + (size_t)P.n_stages * P.stage_bytes;
    const int G = kNumSMs * per_sm;
    P.strips = ceil_div(W, C2_TM);
    // rows per unit: about one unit per CTA, at least 4 rows (each unit re-reads two halo rows)
    int chunks = std::max(1, (G + B * P.strips / 2) / (B * P.strips));
    if (const char* e = getenv("EFFIMVS_CONV2D_ROWS")) chunks = ceil_div(H, std::max(1, atoi(e)));
    int min_rows = 4;
    if (const char* e = getenv("EFFIMVS_CONV2D_MINROWS")) min_rows = std::max(1, atoi(e));
    P.R = std::max(std::min(min_rows, H), ceil_div(H, chunks));
    P.chunks = ceil_div(H, P.R);
    P.n_units = B * P.strips * P.chunks;

    typedef void (*KernelFn)(C2Params, const uint8_t*);
#define C2_ROW(M) {{conv2d_tc_kernel<M, 2, C2_F16>, conv2d_tc_kernel<M, 4, C2_F16>, conv2d_tc_kernel<M, 8, C2_F16>}, \
                   {conv2d_tc_kernel<M, 2, C2_BF16X3>, conv2d_tc_kernel<M, 4, C2_BF16X3>, nullptr}}
    static const KernelFn table[5][2][3] = {C2_ROW(EFFIMVS_CONV2D_BIAS), C2_ROW(EFFIMVS_CONV2D_BIAS_RELU), C2_ROW(EFFIMVS_CONV2D_ADD_RELU),
                                            C2_ROW(EFFIMVS_CONV2D_GRU_GATES), C2_ROW(EFFIMVS_CONV2D_GRU_UPDATE)};
#undef C2_ROW
    const int gi = P.kc == 16 ? 0 : (P.kc == 32 ? 1 : 2);
    const KernelFn fn = table[mode][prec][gi];      // (bf16x3 phases are at most 32 channels: gi < 2)
    static bool attr_set[64][5][2][3] = {};   // per device and instantiation; idempotent, a race only repeats the call
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !attr_set[dev][mode][prec][gi]) {
        cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024);
        EFFI_REQUIRE(e == cudaSuccess, EFFIMVS_ECUDA, "%s: cudaFuncSetAttribute: %s", name, cudaGetErrorString(e));
        if (dev >= 0 && dev < 64) attr_set[dev][mode][prec][gi] = true;
    }
    launch_kernel(fn, dim3(std::min(G, P.n_units)), dim3((C2_PROD_WARP0 + C2_PROD_GROUPS * P.gw) * 32), smem, (cudaStream_t)stream, P,
                  (const uint8_t*)packed);
    return check_launch("conv2d_tc_kernel");
}

}  // namespace
}  // namespace effimvs

using namespace effimvs;

/* profiling hook (not part of include/effimvs.h): device buffer of 3 * 64 * 4 int64 that CTA 0 of the following launches fills */
extern "C" void effimvs_conv2d_debug_timeline(void* buf) { g_conv2d_timeline = (long long*)buf; }

extern "C" size_t effimvs_conv2d_tf32_packed_bytes(int cin, int cout) { return packed_bytes(cin, cout, C2_F16); }
extern "C" int effimvs_conv2d_tf32_supported(int cin, int cout) { return supported(cin, cout, C2_F16); }
extern "C" int effimvs_conv2d_tf32_pack(const float* w, int cin, int cout, void* packed, void* stream) {
    return pack("conv2d_tf32_pack", C2_F16, w, cin, cout, packed, stream);
}
extern "C" int effimvs_conv2d_tf32(const float* in0, long long in0_ps, int c0, const float* in1, long long in1_ps, int c1,
                                   const void* packed, const float* bias, int cout, int B, int H, int W, int mode,
                                   float* out, long long out_ps, const float* aux0, long long aux0_ps, float* aux1,
                                   long long aux1_ps, void* stream) {
    return launch("conv2d_tf32", C2_F16, in0, in0_ps, c0, in1, in1_ps, c1, packed, bias, cout, B, H, W, mode, out, out_ps,
                  aux0, aux0_ps, aux1, aux1_ps, stream);
}

extern "C" size_t effimvs_conv2d_bf16x3_packed_bytes(int cin, int cout) { return packed_bytes(cin, cout, C2_BF16X3); }
extern "C" int effimvs_conv2d_bf16x3_supported(int cin, int cout) { return supported(cin, cout, C2_BF16X3); }
extern "C" int effimvs_conv2d_bf16x3_pack(const float* w, int cin, int cout, void* packed, void* stream) {
    return pack("conv2d_bf16x3_pack", C2_BF16X3, w, cin, cout, packed, stream);
}
extern "C" int effimvs_conv2d_bf16x3(const float* in0, long long in0_ps, int c0, const float* in1, long long in1_ps, int c1,
                                     const void* packed, const float* bias, int cout, int B, int H, int W, int mode,
                                     float* out, long long out_ps, const float* aux0, long long aux0_ps, float* aux1,
                                     long long aux1_ps, void* stream) {
    return launch("conv2d_bf16x3", C2_BF16X3, in0, in0_ps, c0, in1, in1_ps, c1, packed, bias, cout, B, H, W, mode, out, out_ps,
                  aux0, aux0_ps, aux1, aux1_ps, stream);
}
