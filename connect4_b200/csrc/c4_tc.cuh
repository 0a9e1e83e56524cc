// c4_tc.cuh -- building blocks of the tcgen05 / TMEM network tower (oinkoink/neural/pytorch/model.py:20-134, eval mode),
// shared by the batch kernel k_net_tc (c4_net.cu) and the fused persistent self-play engine (c4_fused.cu): operand
// types, strip geometry, UMMA / mbarrier / TMEM helpers, the per-layer epilogue and the fused head tails.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <math.h>

#include "c4_common.cuh"

#define NPX 66            // padded pixel rows: q in [-1, 64], row index q + 1
#define LEAKY 0.01f
#define SCRATCH_BYTES 512 // per-warp head scratch (126 floats)

// offsets inside the fp32 head block
#define HO_VW 0           // value conv weight [F] (max 64)
#define HO_PW 64          // policy conv weight [2][F] (max 128)
#define HO_VB 192         // value conv bias
#define HO_PB 193         // policy conv bias [2]
#define HO_FC1B 195
#define HO_W1 196
#define HO_W2 197
#define HO_FCB 200        // [42]
#define HO_FC1W 242       // [42]
#define HO_POLB 284       // [7]
#define HO_FCT 292        // [42][42] transposed: FCT[j*42+i] = W_eff[i][j]
#define HO_POLW 2056      // [7][84]
#define HEAD_FLOATS 2656  // fp32 head parameter block (2644 used)

struct c4_net {
    int device;
    int F, R, n_fc;
    unsigned long long uid;  // unique per created network (the engine's evaluation memo is keyed on it)
    bool fp16;            // operand element type of the conv GEMMs (false: bf16)
    bool use_tc;          // tcgen05 kernel instead of the mma.sync kernels
    void *image_tc;       // device: [L][WSTAGE_BYTES] weights + biases + head block (tcgen05 kernel)
    void *image;          // device: smem image (kernel A) / per-layer weight images (kernel B)
    size_t image_bytes;
    double flops;
    int scale_log2;       // fp16 operands: the trunk runs at activations * 2^-scale_log2 (chosen by calibration at creation)
    float calib_max;      // largest |activation| (scaled units) the calibration positions produced
    c4_eval_fn ext_fn;    // caller-served network (c4_net_create_external): F = R = 0, no images, no kernel of ours
    void *ext_user;
    int32_t *ext_count;   // pinned host copy of a device leaf count
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ldsm4(uint32_t addr, uint32_t &r0, uint32_t &r1, uint32_t &r2, uint32_t &r3)
{
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void mma16816(float *c, const uint32_t *a, uint32_t b0, uint32_t b1)
{
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void mma16816h(float *c, const uint32_t *a, uint32_t b0, uint32_t b1)
{
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float leaky(float x) { return x > 0.f ? x : LEAKY * x; }

// operand element type of the tensor-core GEMMs (accumulation is always fp32).  fp16 is the default: on the
// reference's trained checkpoint bf16 operands give max |dvalue| 5.4e-2 (> the 1e-2 parity bound), fp16 6.6e-3, at the
// same tensor-core rate (DESIGN.md, "operand precision").
struct OpBF16 {
    static constexpr uint32_t ONE = 0x3F80u;
    static constexpr uint32_t FMT = 1u;   // tcgen05 instruction-descriptor a/b format
    __device__ static __forceinline__ void mma(float *c, const uint32_t *a, uint32_t b0, uint32_t b1) { mma16816(c, a, b0, b1); }
    __device__ static __forceinline__ uint32_t pack(float lo, float hi)
    {
        __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
        return *reinterpret_cast<uint32_t *>(&v);
    }
    __device__ static __forceinline__ float2 unpack(uint32_t u)
    {
        return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162 *>(&u));
    }
};
struct OpFP16 {
    static constexpr uint32_t ONE = 0x3C00u;
    static constexpr uint32_t FMT = 0u;
    __device__ static __forceinline__ void mma(float *c, const uint32_t *a, uint32_t b0, uint32_t b1) { mma16816h(c, a, b0, b1); }
    __device__ static __forceinline__ uint32_t pack(float lo, float hi)
    {
        __half2 v = __floats2half2_rn(lo, hi);
        return *reinterpret_cast<uint32_t *>(&v);
    }
    __device__ static __forceinline__ float2 unpack(uint32_t u) { return __half22float2(*reinterpret_cast<__half2 *>(&u)); }
};

// head tails for one board (model.py:83-91,112-117): scratch[0..41] = value-conv activations, scratch[42..125] =
// policy-conv activations (channel-major); writes {prior[7], value} to out[0..7].  One warp.
__device__ __forceinline__ void head_tail(const float *scratch, const float *hp, float *out, int lane)
{
    // value: (pre-multiplied) Linear(42,42) stack -> LeakyReLU -> Linear(42,1) -> tanh -> (x + w1) * w2
    float part = 0.f;
    for (int i = lane; i < 42; i += 32) {
        float a = hp[HO_FCB + i];
#pragma unroll 6
        for (int j = 0; j < 42; j++) a = fmaf(hp[HO_FCT + j * 42 + i], scratch[j], a);
        part = fmaf(hp[HO_FC1W + i], leaky(a), part);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
    const float value = (tanhf(part + hp[HO_FC1B]) + hp[HO_W1]) * hp[HO_W2];
    // policy: Linear(84,7) on the channel-major flatten -> softmax
    float lg[7];
#pragma unroll
    for (int k = 0; k < 7; k++) lg[k] = 0.f;
    for (int m = lane; m < 84; m += 32) {
        float xv = scratch[42 + m];
#pragma unroll
        for (int k = 0; k < 7; k++) lg[k] = fmaf(hp[HO_POLW + k * 84 + m], xv, lg[k]);
    }
#pragma unroll
    for (int k = 0; k < 7; k++) {
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) lg[k] += __shfl_xor_sync(0xffffffffu, lg[k], off);
        lg[k] += hp[HO_POLB + k];
    }
    float mx = lg[0];
#pragma unroll
    for (int k = 1; k < 7; k++) mx = fmaxf(mx, lg[k]);
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < 7; k++) { lg[k] = expf(lg[k] - mx); sum += lg[k]; }
    float mine = value;
#pragma unroll
    for (int k = 0; k < 7; k++) if (lane == k) mine = lg[k] / sum;
    if (lane < 8) out[lane] = mine;
    __syncwarp();
}

// ------------------------------------------------------------------------------------------------ kernel C (tcgen05)
// Blackwell-native tower for filters = 32: tcgen05.mma with TMEM accumulators, one persistent CTA per SM.
//
//  * STRIP: up to 16 boards stacked in one 8-wide padded pixel strip (7 row-blocks of 8 pixels per board: one shared
//    zero row-block + 6 board rows; pixel column 0 of every row-block is a shared zero column).  112 row-blocks = 896
//    rows = exactly 7 M-tiles of 128.
//  * GEMM: the three dx taps are folded into N:  E_dx[r] = sum_dy A[r + 8 dy] . W[dy][dx]  is ONE accumulation chain
//    of 3 (dy) x Cin/16 MMAs of shape M128 x N96 x K16 whose A operand is only ever shifted by +-8 rows = whole
//    core matrices, done with the descriptor start address.  A is read 3x per conv instead of 9x, which is what
//    makes the small-N conv tensor-bound instead of shared-memory-operand-bound (tools/umma_test.cu: 56 cycles per MMA
//    against a 48-cycle tensor floor).  The epilogue finishes the conv:  out[q] = E_-1[q-1] + E_0[q] + E_+1[q+1],
//    a one-lane shuffle because TMEM lane = strip row.
//  * shared memory: activations [k-chunk][row][8 x 16-bit] (K-major, SWIZZLE_NONE core matrices; a thread's 16-byte
//    store per k-chunk is conflict-free); weights [dy][k-chunk][n = dx*32+co][8] streamed per layer through a 3-stage
//    ring with cp.async.bulk + mbarrier (generic in depth; 18 KB per layer).
//  * TMEM (512 columns): fp32 residual stream of the 7 tiles (224 columns) + 3 accumulator slots of 96 columns, so
//    the MMA warp runs up to 3 tiles ahead of the epilogue.
//  * warp roles: warp 0 = weight producer, warp 1 = MMA issuer (one thread), warps 2..9 = epilogue (TMEM lane
//    quadrant = warp % 4, channel half = (warp - 2) / 4).  MMA(layer l+1, tile t) only waits for epilogue(l, tile t+1),
//    so layers overlap tile by tile; no CTA-wide barrier inside a strip.
// Geometry of the kernel for one filter count.  F = 32: 16-board strips of 7 tiles, whole-layer weight stages (18 KB) in a
// 3-deep ring, 3 accumulator slots, two epilogue groups of 8 warps (4 TMEM lane quadrants x 2 channel slices of 16) on
// alternate tiles.  F = 64 (the reference's example_config network): N = 192 and K = 64 per tap row give 12 MMAs of 96
// tensor cycles per tile -- four times the tensor work per hand-shake -- so one group of 16 warps (4 quadrants x 4 channel
// slices) and a single accumulator slot keep up; strips are 6 boards (3 tiles) so that two activation buffers, one
// 72 KB weight stage and the fp32 residual of the strip (3 x 64 TMEM columns) fit.
template <int F_> struct TcC;
// SLICED: the single weight stage is refilled one dy slice at a time -- the next layer's slice dy is requested as soon as
// the last tile of this layer has issued its dy MMAs, so the reload runs under the rest of that tile and its epilogue.
template <> struct TcC<32> { static constexpr int F = 32, NB = 16, T = 7, ROWS = 912, WSTAGES = 3, ACC_SLOTS = 3, GROUPS = 2, EPI_WARPS = 16; static constexpr bool SLICED = false; };
template <> struct TcC<64> { static constexpr int F = 64, NB = 6, T = 3, ROWS = 400, WSTAGES = 1, ACC_SLOTS = 1, GROUPS = 1, EPI_WARPS = 16; static constexpr bool SLICED = true; };
#define TC_CH 16                       // channels per epilogue thread (one slice)
#define TC_THREADS 576                 // warp 0 weight producer, warp 1 MMA issuer, warps 2..17 epilogue
#define TC_EPI_WARPS 16
// derived constants and the shared-memory map of one geometry (TcC<F> for the batch kernel, c4_fused.cu has its own)
template <class C_> struct TcKc : C_ {
    using C = C_;
    static constexpr int KC = C::F / 8;                                    // 16-byte k-chunks per pixel
    static constexpr int NN = 3 * C::F;                                    // N = 3 dx x F output channels
    static constexpr int SLICES = C::F / TC_CH;                            // channel slices of 16
    static constexpr int GROUP_WARPS = 4 * SLICES;
    static constexpr int ACT_BYTES = KC * C::ROWS * 16;
    static constexpr int WSTAGE_BYTES = 3 * KC * NN * 16;
    static constexpr int WSLICE_BYTES = KC * NN * 16;                      // one dy slice of a layer
    static constexpr int WBARS = C::SLICED ? 3 : C::WSTAGES;               // weight barriers: per dy slice / per stage
    static constexpr int STEM_KC = C::SLICED ? KC : 2;                     // k-chunk pitch of the stem's packed weights
    static constexpr int ACC_COL0 = C::T * C::F;                           // TMEM: residual stream first, then the slots
    static_assert(GROUP_WARPS * C::GROUPS == C::EPI_WARPS, "epilogue warps = groups x (4 lane quadrants x channel slices)");
    static_assert(ACC_COL0 + C::ACC_SLOTS * NN <= 512, "TMEM columns");
    static_assert(16 * C::T >= 7 * C::NB && C::ROWS == 128 * C::T + 16, "strip geometry");
    // shared memory map
    static constexpr int X = 0;
    static constexpr int H = X + ACT_BYTES;
    static constexpr int W = H + ACT_BYTES;
    static constexpr int SMALL = W + C::WSTAGES * WSTAGE_BYTES;            // biases + head params (fp32)
    __host__ __device__ static constexpr int scratch(int R) { return SMALL + ((1 + 2 * R) * C::F + HEAD_FLOATS) * 4; }
    __host__ __device__ static constexpr int bars(int R) { return scratch(R) + SLICES * C::NB * 128 * 4; }   // [slice][board][128]
    __host__ __device__ static constexpr int total(int R) { return bars(R) + 256; }
};
template <int F_> using TcK = TcKc<TcC<F_>>;

__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46);
}
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                 :: "r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
template <int ACC>
__device__ __forceinline__ void umma_f16c(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc)
{
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                 :: "r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "n"(ACC) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t}\n" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0u;
}
// Spin until the phase completes.  A wait that lasts ~5 s of SM cycles can only be a protocol bug: trap (the launch
// fails with an error) instead of hanging the device.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    if (mbar_try(bar, parity)) return;
    const long long t0 = clock64();
    for (uint32_t it = 1;; it++) {
        if (mbar_try(bar, parity)) return;
        if ((it & 0xfu) == 0u && clock64() - t0 > 10000000000LL) __trap();
    }
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float *r)
{
    uint32_t u[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
                 : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
                   "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
                 : "r"(taddr) : "memory");
#pragma unroll
    for (int i = 0; i < 16; i++) r[i] = __uint_as_float(u[i]);
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float *r)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};\n"
                 :: "r"(taddr), "r"(__float_as_uint(r[0])), "r"(__float_as_uint(r[1])), "r"(__float_as_uint(r[2])),
                    "r"(__float_as_uint(r[3])), "r"(__float_as_uint(r[4])), "r"(__float_as_uint(r[5])),
                    "r"(__float_as_uint(r[6])), "r"(__float_as_uint(r[7])), "r"(__float_as_uint(r[8])),
                    "r"(__float_as_uint(r[9])), "r"(__float_as_uint(r[10])), "r"(__float_as_uint(r[11])),
                    "r"(__float_as_uint(r[12])), "r"(__float_as_uint(r[13])), "r"(__float_as_uint(r[14])),
                    "r"(__float_as_uint(r[15])) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float *r)
{
    uint32_t u[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
                 : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7])
                 : "r"(taddr) : "memory");
#pragma unroll
    for (int i = 0; i < 8; i++) r[i] = __uint_as_float(u[i]);
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float *r)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};\n"
                 :: "r"(taddr), "r"(__float_as_uint(r[0])), "r"(__float_as_uint(r[1])), "r"(__float_as_uint(r[2])),
                    "r"(__float_as_uint(r[3])), "r"(__float_as_uint(r[4])), "r"(__float_as_uint(r[5])),
                    "r"(__float_as_uint(r[6])), "r"(__float_as_uint(r[7])) : "memory");
}
#define TC_FENCE_BEFORE() asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory")
#define TC_FENCE_AFTER() asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory")
#define TC_PROXY_FENCE() asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory")
#define EPI_BAR() asm volatile("bar.sync 1, 512;\n" ::: "memory")      // the 16 epilogue warps only

// Epilogue of one layer, specialised on the layer kind so the tile loop carries no layer-type branches:
//   KIND 0 = stem (result -> residual stream + X), 1 = first conv of a block (-> H),
//   2 = second conv (+= residual, -> residual stream + X), 3 = the last conv of the tower (+= residual, -> head partials).
// The per-tile epilogue is a serial chain of long-latency steps (barrier wake-up, TMEM loads, shuffles, TMEM / shared
// stores, fences, arrive: ~1100 cycles), so the 16 epilogue warps form TWO groups that take alternate tiles of the
// global tile sequence: two chains are always in flight.  A tile's residual columns are touched in layers 0, 2, 4, ...
// whose tile counters differ by a multiple of 2T, i.e. always by the same group and the same thread.
struct EpiCtx {
    uint32_t b_accfull, b_accempty, b_epi;
    uint32_t tmem_acc;        // tmem + lane quadrant + ACC_COL0 + 16 * slice
    uint32_t tmem_res;        // tmem + lane quadrant + 16 * slice
    unsigned char *dst_x, *dst_h;   // smem row of this thread in tile 0, k-chunk 2 * slice
    const float *bias, *hp;
    float *scratch;           // + slice * NB * 128
    uint32_t valid_mask;      // bit t: this thread's row of tile t is a real pixel of a board of this strip
    int lane, lm, lp, half, group, rb0, col8;
    unsigned *calib;          // calibration launches only: running max of the bits of |activation|
};

template <typename OP, int F, int KIND, bool CALIB = false>
__device__ __forceinline__ void tc_epilogue_layer(const EpiCtx &E, int l, int T, int c0)
{
    using K = TcK<F>;
    constexpr bool TO_RES = (KIND == 0 || KIND == 2), ADD_RES = (KIND == 2 || KIND == 3), LAST = (KIND == 3);
    unsigned char *dst = (KIND == 1) ? E.dst_h : E.dst_x;
    const float *bl = E.bias + l * F + TC_CH * E.half;
#pragma unroll 1
    for (int t = (E.group + K::GROUPS - c0 % K::GROUPS) % K::GROUPS; t < T; t += K::GROUPS) {   // tiles c = c0 + t with c % GROUPS == group
        const int c = c0 + t, slot = c % K::ACC_SLOTS;
        mbar_wait(E.b_accfull + 8 * slot, (uint32_t)(c / K::ACC_SLOTS) & 1u);
        TC_FENCE_AFTER();
        const uint32_t ta = E.tmem_acc + slot * K::NN;
        const uint32_t tr = E.tmem_res + F * t;
        float em[TC_CH], ez[TC_CH], ep[TC_CH], rs[TC_CH];
        tmem_ld16(ta, em);
        tmem_ld16(ta + F, ez);
        tmem_ld16(ta + 2 * F, ep);
        if (ADD_RES) tmem_ld16(tr, rs);
        asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
        TC_FENCE_BEFORE();
        __syncwarp();
        if (E.lane == 0) mbar_arrive(E.b_accempty + 8 * slot);            // accumulator slot free for the MMA warp
        // out[q] = E_-1[q-1] + E_0[q] + E_+1[q+1].  Rotating shuffles need no edge fix-up: lane 0 is a pad-column row
        // (its result is discarded) and lane 31 wraps to lane 0 whose E is exactly 0 (A is zero on pad rows).
        // Packed fp32x2 adds / muls (FADD2 / FMUL2 on sm_100).
        float v[TC_CH];
#pragma unroll
        for (int j = 0; j < TC_CH; j += 2) {
            float2 m1 = make_float2(__shfl_sync(0xffffffffu, em[j], E.lm), __shfl_sync(0xffffffffu, em[j + 1], E.lm));
            float2 p1 = make_float2(__shfl_sync(0xffffffffu, ep[j], E.lp), __shfl_sync(0xffffffffu, ep[j + 1], E.lp));
            float2 y = __fadd2_rn(__fadd2_rn(m1, make_float2(ez[j], ez[j + 1])), __fadd2_rn(p1, make_float2(bl[j], bl[j + 1])));
            if (ADD_RES) y = __fadd2_rn(y, make_float2(rs[j], rs[j + 1]));
            float2 z = __fmul2_rn(y, make_float2(LEAKY, LEAKY));
            v[j] = fmaxf(y.x, z.x);
            v[j + 1] = fmaxf(y.y, z.y);
        }
        const bool valid = (E.valid_mask >> t) & 1u;
        if (CALIB && valid) {
            // range calibration (c4_net_create): integer max of the bit patterns, so Inf / NaN read as "too large"
            unsigned mu = 0u;
#pragma unroll
            for (int j = 0; j < TC_CH; j++) mu = max(mu, __float_as_uint(fabsf(v[j])));
            atomicMax(E.calib, mu);
        }
        if (TO_RES) tmem_st16(tr, v);
        if (!LAST) {
            if (valid) {
                unsigned char *p = dst + (size_t)t * (128 * 16);
                *reinterpret_cast<uint4 *>(p) =
                    make_uint4(OP::pack(v[0], v[1]), OP::pack(v[2], v[3]), OP::pack(v[4], v[5]), OP::pack(v[6], v[7]));
                *reinterpret_cast<uint4 *>(p + K::ROWS * 16) =
                    make_uint4(OP::pack(v[8], v[9]), OP::pack(v[10], v[11]), OP::pack(v[12], v[13]), OP::pack(v[14], v[15]));
            }
        } else if (valid) {
            // head 1x1 convs (model.py:77-79,107-109): this thread's 16 channels of one pixel; the two channel halves are
            // summed in a fixed order by the head tail (deterministic, no atomics)
            float a = 0.f, p0 = 0.f, p1 = 0.f;
#pragma unroll
            for (int j = 0; j < TC_CH; j++) {
                a = fmaf(v[j], E.hp[HO_VW + TC_CH * E.half + j], a);
                p0 = fmaf(v[j], E.hp[HO_PW + TC_CH * E.half + j], p0);
                p1 = fmaf(v[j], E.hp[HO_PW + F + TC_CH * E.half + j], p1);
            }
            const int rb = 16 * t + E.rb0, b = rb / 7;
            float *sc = E.scratch + b * 128 + (rb - 7 * b - 1) * 7 + (E.col8 - 1);
            sc[0] = a; sc[42] = p0; sc[84] = p1;
        }
        if (TO_RES) asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
        if (!LAST) TC_PROXY_FENCE();
        __syncwarp();
        if (E.lane == 0) mbar_arrive(E.b_epi + 8 * t);
    }
}

// mbarrier wait for warps that may wait LONG (the fused engine's tower idles while its SM has no leaves): after a few
// failed polls the warp sleeps between polls so that it does not take issue slots from the tree warps of the same SM
__device__ __forceinline__ void mbar_wait_idle(uint32_t bar, uint32_t parity)
{
    if (mbar_try(bar, parity)) return;
    const long long t0 = clock64();
    for (uint32_t it = 1;; it++) {
        if (mbar_try(bar, parity)) return;
        if (it > 8u) __nanosleep(it > 64u ? 256 : 32);
        if ((it & 0xfu) == 0u && clock64() - t0 > 10000000000LL) __trap();
    }
}

// The same epilogue in two steps of 8 channels: at most 40 accumulator / residual / result values are live per thread,
// so it fits the 64 registers of the 1024-thread fused engine (c4_fused.cu) without spilling.  Every output element goes
// through exactly the same operations in the same order as in tc_epilogue_layer (the head partial sums are carried
// across the two steps), so both kernels produce bit-identical network answers.
template <typename OP, typename K, int KIND>
__device__ __forceinline__ void tc_epilogue_layer8(const EpiCtx &E, int l, int T, int c0)
{
    constexpr int F = K::F;
    constexpr bool TO_RES = (KIND == 0 || KIND == 2), ADD_RES = (KIND == 2 || KIND == 3), LAST = (KIND == 3);
    unsigned char *dst = (KIND == 1) ? E.dst_h : E.dst_x;
    const float *bl = E.bias + l * F + TC_CH * E.half;
#pragma unroll 1
    for (int t = (E.group + K::GROUPS - c0 % K::GROUPS) % K::GROUPS; t < T; t += K::GROUPS) {
        const int c = c0 + t, slot = c % K::ACC_SLOTS;
        mbar_wait_idle(E.b_accfull + 8 * slot, (uint32_t)(c / K::ACC_SLOTS) & 1u);
        TC_FENCE_AFTER();
        const uint32_t ta = E.tmem_acc + slot * K::NN;
        const uint32_t tr = E.tmem_res + F * t;
        const bool valid = (E.valid_mask >> t) & 1u;
        float a = 0.f, p0 = 0.f, p1 = 0.f;
#pragma unroll
        for (int h0 = 0; h0 < TC_CH; h0 += 8) {
            float em[8], ez[8], ep[8], rs[8];
            tmem_ld8(ta + h0, em);
            tmem_ld8(ta + F + h0, ez);
            tmem_ld8(ta + 2 * F + h0, ep);
            if (ADD_RES) tmem_ld8(tr + h0, rs);
            asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
            if (h0 + 8 == TC_CH) {
                TC_FENCE_BEFORE();
                __syncwarp();
                if (E.lane == 0) mbar_arrive(E.b_accempty + 8 * slot);    // accumulator slot free for the MMA warp
            }
            float v[8];
#pragma unroll
            for (int j = 0; j < 8; j += 2) {
                float2 m1 = make_float2(__shfl_sync(0xffffffffu, em[j], E.lm), __shfl_sync(0xffffffffu, em[j + 1], E.lm));
                float2 q1 = make_float2(__shfl_sync(0xffffffffu, ep[j], E.lp), __shfl_sync(0xffffffffu, ep[j + 1], E.lp));
                float2 y = __fadd2_rn(__fadd2_rn(m1, make_float2(ez[j], ez[j + 1])),
                                      __fadd2_rn(q1, make_float2(bl[h0 + j], bl[h0 + j + 1])));
                if (ADD_RES) y = __fadd2_rn(y, make_float2(rs[j], rs[j + 1]));
                float2 z = __fmul2_rn(y, make_float2(LEAKY, LEAKY));
                v[j] = fmaxf(y.x, z.x);
                v[j + 1] = fmaxf(y.y, z.y);
            }
            if (TO_RES) tmem_st8(tr + h0, v);
            if (!LAST) {
                if (valid)
                    *reinterpret_cast<uint4 *>(dst + (size_t)t * (128 * 16) + (size_t)(h0 / 8) * (K::ROWS * 16)) =
                        make_uint4(OP::pack(v[0], v[1]), OP::pack(v[2], v[3]), OP::pack(v[4], v[5]), OP::pack(v[6], v[7]));
            } else {
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    a = fmaf(v[j], E.hp[HO_VW + TC_CH * E.half + h0 + j], a);
                    p0 = fmaf(v[j], E.hp[HO_PW + TC_CH * E.half + h0 + j], p0);
                    p1 = fmaf(v[j], E.hp[HO_PW + F + TC_CH * E.half + h0 + j], p1);
                }
            }
        }
        if (LAST && valid) {
            const int rb = 16 * t + E.rb0, b = rb / 7;
            float *sc = E.scratch + b * 128 + (rb - 7 * b - 1) * 7 + (E.col8 - 1);
            sc[0] = a; sc[42] = p0; sc[84] = p1;
        }
        if (TO_RES) asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
        if (!LAST) TC_PROXY_FENCE();
        __syncwarp();
        if (E.lane == 0) mbar_arrive(E.b_epi + 8 * t);
    }
}
