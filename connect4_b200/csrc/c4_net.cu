// c4_net.cu -- fused residual value/policy network forward (oinkoink/neural/pytorch/model.py:20-134, eval mode).
//
// One launch evaluates a whole leaf batch: bitboards in (16 B/position), {prior[7], value} out (32 B/position);
// every intermediate activation stays on chip.
//
// Kernel A (filters = 32, the default NetConfig): WARP-PER-BOARD fused tower.
//   * all BN-folded bf16 conv weights (stem + 2R residual convs, 123 KB) and the fp32 head parameters stay resident
//     in shared memory for the life of the CTA; a persistent grid of 148 CTAs x 8 warps strides over the batch.
//   * a board is laid out as an 8-wide padded pixel strip (row stride 8 = 7 columns + one shared zero column), so a
//     3x3 tap is a constant row offset and every conv is 9 shifted [48 x Cin] x [Cin x 32] bf16 GEMMs
//     (mma.sync m16n8k16, fp32 accumulate, operands via ldmatrix from conflict-free padded rows).
//   * the residual stream is kept in fp32 registers (same fragment layout for every layer); shared memory only holds
//     the bf16 operand copy.  No block-level barrier anywhere: a warp only touches its own board.
//   * heads are fused: 1x1 convs straight from the fp32 fragments (quad shuffles), the (pre-multiplied) value MLP,
//     tanh, the policy linear and the 7-way softmax.
// Kernel B (filters = 64, example_config): same math, but weights do not fit on chip (897 KB): the CTA walks the layers
//   together and streams each layer's weights L2 -> shared memory; the residual is re-read from the bf16 copy.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "c4_common.cuh"

#include "c4_tc.cuh"
#include "c4_layers.cuh"

// One 3x3 convolution of one board as implicit GEMM: acc[t][j][.] (+)= sum over taps/channels.
//   src: padded activation strip (row stride AS bytes), W: [F][9*CIN + 8] bf16 rows (stride WS bytes)
template <typename OP, int F, int CIN>
__device__ __forceinline__ void conv3x3(float (&acc)[3][F / 8][4], uint32_t src, uint32_t W, int lane)
{
    constexpr int AS = F * 2 + 16;
    constexpr int WS = (9 * CIN + 8) * 2;
    constexpr int NT = F / 8;
#pragma unroll
    for (int t = 0; t < 3; t++)
#pragma unroll
        for (int j = 0; j < NT; j++)
#pragma unroll
            for (int e = 0; e < 4; e++) acc[t][j][e] = 0.f;
    // per-lane ldmatrix row addresses
    const int arow = (lane & 7) + ((lane >> 3) & 1) * 8;       // A: matrices 0/1 = rows 0-7 / 8-15, 2/3 = k+8
    const uint32_t a_base = src + (uint32_t)((8 + arow + 1) * AS + (lane >> 4) * 16);
    const uint32_t b_base = W + (uint32_t)((((lane >> 4) & 1) * 8 + (lane & 7)) * WS + ((lane >> 3) & 1) * 16);
#pragma unroll 1
    for (int tap = 0; tap < 9; tap++) {
        const int off = (tap / 3 - 1) * 8 + (tap % 3 - 1);
#pragma unroll
        for (int kc = 0; kc < CIN / 16; kc++) {
            uint32_t a[3][4];
#pragma unroll
            for (int t = 0; t < 3; t++)
                ldsm4(a_base + (uint32_t)((16 * t + off) * AS + kc * 32), a[t][0], a[t][1], a[t][2], a[t][3]);
#pragma unroll
            for (int jp = 0; jp < NT / 2; jp++) {
                uint32_t b0, b1, b2, b3;
                ldsm4(b_base + (uint32_t)(jp * 16 * WS + (tap * CIN + kc * 16) * 2), b0, b1, b2, b3);
#pragma unroll
                for (int t = 0; t < 3; t++) {
                    OP::mma(acc[t][2 * jp], a[t], b0, b1);
                    OP::mma(acc[t][2 * jp + 1], a[t], b2, b3);
                }
            }
        }
    }
}

// board -> bf16 input planes (Board.to_array, oinkoink/board.py:147-154) in channels 0..15 of the strip
template <typename OP, int F>
__device__ __forceinline__ void write_input(unsigned char *buf, u64 c0, u64 c1, int lane)
{
    constexpr int AS = F * 2 + 16;
    const uint32_t tomove = ((__popcll(c0 | c1) & 1) == 0) ? OP::ONE : 0u;
    for (int px = lane; px < 42; px += 32) {
        int r = px / 7, c = px - r * 7;
        int bit = 7 * c + (5 - r);
        uint32_t o = (uint32_t)((c0 >> bit) & 1ULL) * OP::ONE, x = (uint32_t)((c1 >> bit) & 1ULL) * OP::ONE;
        uint4 v0 = make_uint4(tomove | (o << 16), x, 0u, 0u), v1 = make_uint4(0u, 0u, 0u, 0u);
        unsigned char *row = buf + (size_t)(((r + 1) * 8 + (c + 1)) + 1) * AS;
        *reinterpret_cast<uint4 *>(row) = v0;
        *reinterpret_cast<uint4 *>(row + 16) = v1;
    }
}

// store the activated fp32 fragments as the bf16 operand copy (valid pixels only: pad column rows stay zero)
template <typename OP, int F>
__device__ __forceinline__ void store_act(unsigned char *buf, const float (&v)[3][F / 8][4], int lane)
{
    constexpr int AS = F * 2 + 16;
    const int g = lane >> 2, tq = lane & 3;
    if (g == 0) return;
#pragma unroll
    for (int t = 0; t < 3; t++)
#pragma unroll
        for (int j = 0; j < F / 8; j++) {
            unsigned char *p = buf + (size_t)((8 + 16 * t + g) + 1) * AS + (j * 8 + 2 * tq) * 2;
            *reinterpret_cast<uint32_t *>(p) = OP::pack(v[t][j][0], v[t][j][1]);
            *reinterpret_cast<uint32_t *>(p + 8 * AS) = OP::pack(v[t][j][2], v[t][j][3]);
        }
}

// value + policy heads from the fp32 trunk fragments (model.py:77-91,107-117); scratch: >= 126 floats of shared memory
template <int F>
__device__ __forceinline__ void heads(const float (&x)[3][F / 8][4], const float *hp, float *scratch, float *out, int lane)
{
    const int g = lane >> 2, tq = lane & 3;
    float pv[3][2], p0[3][2], p1[3][2];
#pragma unroll
    for (int t = 0; t < 3; t++)
#pragma unroll
        for (int h = 0; h < 2; h++) {
            float a = 0.f, b = 0.f, c = 0.f;
#pragma unroll
            for (int j = 0; j < F / 8; j++) {
                int co = j * 8 + 2 * tq;
                float x0 = x[t][j][2 * h], x1 = x[t][j][2 * h + 1];
                a = fmaf(x0, hp[HO_VW + co], a); a = fmaf(x1, hp[HO_VW + co + 1], a);
                b = fmaf(x0, hp[HO_PW + co], b); b = fmaf(x1, hp[HO_PW + co + 1], b);
                c = fmaf(x0, hp[HO_PW + F + co], c); c = fmaf(x1, hp[HO_PW + F + co + 1], c);
            }
            pv[t][h] = a; p0[t][h] = b; p1[t][h] = c;
        }
#pragma unroll
    for (int t = 0; t < 3; t++)
#pragma unroll
        for (int h = 0; h < 2; h++) {
            pv[t][h] += __shfl_xor_sync(0xffffffffu, pv[t][h], 1); pv[t][h] += __shfl_xor_sync(0xffffffffu, pv[t][h], 2);
            p0[t][h] += __shfl_xor_sync(0xffffffffu, p0[t][h], 1); p0[t][h] += __shfl_xor_sync(0xffffffffu, p0[t][h], 2);
            p1[t][h] += __shfl_xor_sync(0xffffffffu, p1[t][h], 1); p1[t][h] += __shfl_xor_sync(0xffffffffu, p1[t][h], 2);
        }
    __syncwarp();
    if (tq == 0 && g != 0) {
#pragma unroll
        for (int t = 0; t < 3; t++)
#pragma unroll
            for (int h = 0; h < 2; h++) {
                int q = 8 + 16 * t + g + 8 * h;
                int idx = ((q >> 3) - 1) * 7 + ((q & 7) - 1);
                scratch[idx] = leaky(pv[t][h] + hp[HO_VB]);
                scratch[42 + idx] = leaky(p0[t][h] + hp[HO_PB]);
                scratch[84 + idx] = leaky(p1[t][h] + hp[HO_PB + 1]);
            }
    }
    __syncwarp();
    head_tail(scratch, hp, out, lane);
}

// ------------------------------------------------------------------------------------------------ kernel A (F = 32)
// shared-memory image: [stem W 32x(144+8) bf16][2R conv W 32x(288+8) bf16][biases (1+2R) x 32 f32][head f32]
template <int F>
struct ImageA {
    static constexpr int WS_STEM = (9 * 16 + 8) * 2;
    static constexpr int WS = (9 * F + 8) * 2;
    __host__ __device__ static constexpr size_t stem_bytes() { return (size_t)F * WS_STEM; }
    __host__ __device__ static constexpr size_t conv_bytes() { return (size_t)F * WS; }
    __host__ __device__ static constexpr size_t bias_off(int R) { return stem_bytes() + 2 * R * conv_bytes(); }
    __host__ __device__ static constexpr size_t head_off(int R) { return bias_off(R) + (size_t)(1 + 2 * R) * F * 4; }
    __host__ __device__ static constexpr size_t total(int R) { return head_off(R) + HEAD_FLOATS * 4; }
};

template <typename OP, int F, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, 1)
k_net_resident(const unsigned char *__restrict__ image, int image_bytes, int R, const u64 *__restrict__ c0,
               const u64 *__restrict__ c1, int n, const int *__restrict__ count, float *__restrict__ out)
{
    extern __shared__ __align__(16) unsigned char smem[];
    constexpr int AS = F * 2 + 16;
    constexpr int ACT = NPX * AS;
    if (count) { int m = *count; n = m < n ? m : n; }
    if ((int)blockIdx.x * WARPS >= n) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // resident parameters
    for (int i = threadIdx.x; i < image_bytes / 16; i += blockDim.x)
        reinterpret_cast<uint4 *>(smem)[i] = reinterpret_cast<const uint4 *>(image)[i];
    unsigned char *X = smem + image_bytes + (size_t)warp * (2 * ACT + SCRATCH_BYTES);
    unsigned char *H = X + ACT;
    float *scratch = reinterpret_cast<float *>(H + ACT);   // NOT inside the strips: their pad rows must stay zero
    for (int i = lane; i < 2 * ACT / 16; i += 32) reinterpret_cast<uint4 *>(X)[i] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    const uint32_t sX = smem_u32(X), sH = smem_u32(H), sW = smem_u32(smem);
    const float *bias = reinterpret_cast<const float *>(smem + ImageA<F>::stem_bytes() + 2 * R * ImageA<F>::conv_bytes());
    const float *hp = bias + (1 + 2 * R) * F;
    const int tq = lane & 3;

    for (int b = blockIdx.x * WARPS + warp; b < n; b += gridDim.x * WARPS) {
        const u64 bc0 = c0[b], bc1 = c1[b];
        write_input<OP, F>(H, bc0, bc1, lane);
        __syncwarp();
        float acc[3][F / 8][4], res[3][F / 8][4];
        // stem: conv3x3(3->F) + BN + LeakyReLU (model.py:20-31)
        conv3x3<OP, F, 16>(acc, sH, sW, lane);
#pragma unroll
        for (int t = 0; t < 3; t++)
#pragma unroll
            for (int j = 0; j < F / 8; j++) {
                float b0 = bias[j * 8 + 2 * tq], b1 = bias[j * 8 + 2 * tq + 1];
                res[t][j][0] = leaky(acc[t][j][0] + b0); res[t][j][1] = leaky(acc[t][j][1] + b1);
                res[t][j][2] = leaky(acc[t][j][2] + b0); res[t][j][3] = leaky(acc[t][j][3] + b1);
            }
        store_act<OP, F>(X, res, lane);
        __syncwarp();
        // residual tower (model.py:45-55)
#pragma unroll 1
        for (int r = 0; r < R; r++) {
            const uint32_t w1 = sW + (uint32_t)(ImageA<F>::stem_bytes() + (size_t)(2 * r) * ImageA<F>::conv_bytes());
            const uint32_t w2 = w1 + (uint32_t)ImageA<F>::conv_bytes();
            const float *bb1 = bias + (1 + 2 * r) * F, *bb2 = bb1 + F;
            conv3x3<OP, F, F>(acc, sX, w1, lane);
#pragma unroll
            for (int t = 0; t < 3; t++)
#pragma unroll
                for (int j = 0; j < F / 8; j++) {
                    float b0 = bb1[j * 8 + 2 * tq], b1 = bb1[j * 8 + 2 * tq + 1];
                    acc[t][j][0] = leaky(acc[t][j][0] + b0); acc[t][j][1] = leaky(acc[t][j][1] + b1);
                    acc[t][j][2] = leaky(acc[t][j][2] + b0); acc[t][j][3] = leaky(acc[t][j][3] + b1);
                }
            store_act<OP, F>(H, acc, lane);
            __syncwarp();
            conv3x3<OP, F, F>(acc, sH, w2, lane);
#pragma unroll
            for (int t = 0; t < 3; t++)
#pragma unroll
                for (int j = 0; j < F / 8; j++) {
                    float b0 = bb2[j * 8 + 2 * tq], b1 = bb2[j * 8 + 2 * tq + 1];
                    res[t][j][0] = leaky(acc[t][j][0] + b0 + res[t][j][0]); res[t][j][1] = leaky(acc[t][j][1] + b1 + res[t][j][1]);
                    res[t][j][2] = leaky(acc[t][j][2] + b0 + res[t][j][2]); res[t][j][3] = leaky(acc[t][j][3] + b1 + res[t][j][3]);
                }
            if (r + 1 < R) store_act<OP, F>(X, res, lane);
            __syncwarp();
        }
        heads<F>(res, hp, scratch, out + (size_t)b * 8, lane);
    }
}

// ------------------------------------------------------------------------------------------------ kernel B (F = 64)
// global image: [stem W][2R conv W][biases][head]; shared: one layer's weights + biases + head + per-warp strips
template <typename OP, int F, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, 1)
k_net_streamed(const unsigned char *__restrict__ image, int R, const u64 *__restrict__ c0, const u64 *__restrict__ c1,
               int n, const int *__restrict__ count, float *__restrict__ out)
{
    extern __shared__ __align__(16) unsigned char smem[];
    constexpr int AS = F * 2 + 16;
    constexpr int ACT = NPX * AS;
    constexpr int NT = F / 8;
    if (count) { int m = *count; n = m < n ? m : n; }
    if ((int)blockIdx.x * WARPS >= n) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, tq = lane & 3, g = lane >> 2;
    const size_t conv_b = ImageA<F>::conv_bytes(), stem_b = ImageA<F>::stem_bytes();
    unsigned char *Wbuf = smem;                                               // conv_b bytes
    float *small = reinterpret_cast<float *>(smem + conv_b);                  // biases + head
    const int small_bytes = (1 + 2 * R) * F * 4 + HEAD_FLOATS * 4;
    unsigned char *X = smem + conv_b + small_bytes + (size_t)warp * (2 * ACT + SCRATCH_BYTES);
    unsigned char *H = X + ACT;
    float *scratch = reinterpret_cast<float *>(H + ACT);
    {
        const unsigned char *src = image + ImageA<F>::bias_off(R);
        for (int i = threadIdx.x; i < small_bytes / 16; i += blockDim.x)
            reinterpret_cast<uint4 *>(small)[i] = reinterpret_cast<const uint4 *>(src)[i];
    }
    for (int i = lane; i < 2 * ACT / 16; i += 32) reinterpret_cast<uint4 *>(X)[i] = make_uint4(0u, 0u, 0u, 0u);
    const float *bias = small, *hp = small + (1 + 2 * R) * F;
    const uint32_t sX = smem_u32(X), sH = smem_u32(H), sW = smem_u32(Wbuf);

    const int per_round = gridDim.x * WARPS;
    for (int base = 0; base < n; base += per_round) {                         // CTA-uniform trip count
        const int b = base + blockIdx.x * WARPS + warp;
        const bool active = b < n;
        float acc[3][NT][4];
        // layer 0: stem
        __syncthreads();
        for (int i = threadIdx.x; i < (int)(stem_b / 16); i += blockDim.x)
            reinterpret_cast<uint4 *>(Wbuf)[i] = reinterpret_cast<const uint4 *>(image)[i];
        if (active) write_input<OP, F>(H, c0[b], c1[b], lane);
        __syncthreads();
        if (active) {
            conv3x3<OP, F, 16>(acc, sH, sW, lane);
#pragma unroll
            for (int t = 0; t < 3; t++)
#pragma unroll
                for (int j = 0; j < NT; j++) {
                    float b0 = bias[j * 8 + 2 * tq], b1 = bias[j * 8 + 2 * tq + 1];
                    acc[t][j][0] = leaky(acc[t][j][0] + b0); acc[t][j][1] = leaky(acc[t][j][1] + b1);
                    acc[t][j][2] = leaky(acc[t][j][2] + b0); acc[t][j][3] = leaky(acc[t][j][3] + b1);
                }
            store_act<OP, F>(X, acc, lane);
        }
#pragma unroll 1
        for (int l = 0; l < 2 * R; l++) {
            __syncthreads();
            const unsigned char *src = image + stem_b + (size_t)l * conv_b;
            for (int i = threadIdx.x; i < (int)(conv_b / 16); i += blockDim.x)
                reinterpret_cast<uint4 *>(Wbuf)[i] = reinterpret_cast<const uint4 *>(src)[i];
            __syncthreads();
            if (!active) continue;
            const float *bb = bias + (1 + l) * F;
            const bool second = (l & 1);
            conv3x3<OP, F, F>(acc, second ? sH : sX, sW, lane);
#pragma unroll
            for (int t = 0; t < 3; t++)
#pragma unroll
                for (int j = 0; j < NT; j++) {
                    float b0 = bb[j * 8 + 2 * tq], b1 = bb[j * 8 + 2 * tq + 1];
                    float r0 = 0.f, r1 = 0.f, r2 = 0.f, r3 = 0.f;
                    if (second && g != 0) {                                      // residual from the bf16 copy
                        const unsigned char *p = X + (size_t)((8 + 16 * t + g) + 1) * AS + (j * 8 + 2 * tq) * 2;
                        float2 lo = OP::unpack(*reinterpret_cast<const uint32_t *>(p));
                        float2 hi = OP::unpack(*reinterpret_cast<const uint32_t *>(p + 8 * AS));
                        r0 = lo.x; r1 = lo.y; r2 = hi.x; r3 = hi.y;
                    }
                    acc[t][j][0] = leaky(acc[t][j][0] + b0 + r0); acc[t][j][1] = leaky(acc[t][j][1] + b1 + r1);
                    acc[t][j][2] = leaky(acc[t][j][2] + b0 + r2); acc[t][j][3] = leaky(acc[t][j][3] + b1 + r3);
                }
            __syncwarp();
            if (l + 1 < 2 * R) store_act<OP, F>(second ? X : H, acc, lane);
            __syncwarp();
        }
        if (active) heads<F>(acc, hp, scratch, out + (size_t)b * 8, lane);
    }
}

// global image: [L layers][WSTAGE_BYTES] weights, then biases [(1+2R)*F] fp32, then head block [HEAD_FLOATS] fp32
template <typename OP, int F, bool CALIB = false>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_net_tc(const unsigned char *__restrict__ image, int R, const u64 *__restrict__ c0, const u64 *__restrict__ c1, int n,
         const int *__restrict__ count, float *__restrict__ out, long long *__restrict__ dbg)
{
#ifdef C4_TC_PROFILE   // per-role cycle accounting (build with -DC4_TC_PROFILE, run with C4_TC_DEBUG=1)
#define DBG_T(var) if (dbg) { long long _now = clock64(); var += _now - tmark; tmark = _now; }
    long long tmark = clock64(), d0 = 0, d1 = 0, d2 = 0, d3 = 0, d4 = 0, d5 = 0, d6 = 0, d7 = 0;
#else
#define DBG_T(var)
#endif
    using K = TcK<F>;
    extern __shared__ __align__(16) unsigned char smem[];
    if (count) { int m = *count; n = m < n ? m : n; }
    // static, even partition of the batch over the grid
    const int per = n / (int)gridDim.x, extra = n % (int)gridDim.x;
    const int my_n = per + ((int)blockIdx.x < extra ? 1 : 0);
    const int my_first = (int)blockIdx.x * per + min((int)blockIdx.x, extra);
    if (my_n == 0) return;
    const int n_strips = (my_n + K::NB - 1) / K::NB;
    const int L = 1 + 2 * R;
    // warp index through a broadcast so the compiler knows the role branches below are warp-uniform (otherwise every
    // shuffle of the epilogue is wrapped in WARPSYNC.COLLECTIVE)
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;

    unsigned char *sX = smem + K::X, *sH = smem + K::H, *sW = smem + K::W;
    float *small = reinterpret_cast<float *>(smem + K::SMALL);
    const float *bias = small, *hp = small + L * F;
    float *scratch = reinterpret_cast<float *>(smem + K::scratch(R));
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + K::bars(R));
    const uint32_t b_wfull = smem_u32(bars), b_wempty = b_wfull + 8 * K::WBARS;
    const uint32_t b_accfull = b_wempty + 8 * K::WBARS, b_accempty = b_accfull + 8 * K::ACC_SLOTS;
    const uint32_t b_epi = b_accempty + 8 * K::ACC_SLOTS;                   // T barriers
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * K::WBARS + 2 * K::ACC_SLOTS + K::T);

    // ---- one-time setup: zero the strips (pad rows/columns stay zero for ever), small params, barriers, TMEM
    for (int i = threadIdx.x; i < 2 * K::ACT_BYTES / 16; i += blockDim.x)
        reinterpret_cast<uint4 *>(sX)[i] = make_uint4(0u, 0u, 0u, 0u);
    {
        const unsigned char *src = image + (size_t)L * K::WSTAGE_BYTES;
        const int nb16 = (L * F + HEAD_FLOATS) * 4 / 16;
        for (int i = threadIdx.x; i < nb16; i += blockDim.x)
            reinterpret_cast<uint4 *>(small)[i] = reinterpret_cast<const uint4 *>(src)[i];
    }
    if (threadIdx.x == 0) {
        for (int i = 0; i < K::WBARS; i++) { mbar_init(b_wfull + 8 * i, 1); mbar_init(b_wempty + 8 * i, 1); }
        for (int i = 0; i < K::ACC_SLOTS; i++) { mbar_init(b_accfull + 8 * i, 1); mbar_init(b_accempty + 8 * i, K::GROUP_WARPS); }
        for (int i = 0; i < K::T; i++) mbar_init(b_epi + 8 * i, K::GROUP_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;\n" :: "r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    TC_PROXY_FENCE();
    TC_FENCE_BEFORE();
    __syncthreads();
    TC_FENCE_AFTER();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        // ================= weight producer: layer g of the (strip, layer) sequence -> ring stage g % WSTAGES
        if (lane == 0 && K::SLICED) {
            const int total = n_strips * L;
            for (int g = 0; g < total; g++)
                for (int dy = 0; dy < 3; dy++) {                              // slice dy of layer g -> its third of the stage
                    if (g > 0) mbar_wait(b_wempty + 8 * dy, (g - 1) & 1);
                    mbar_expect_tx(b_wfull + 8 * dy, K::WSLICE_BYTES);
                    bulk_g2s(smem_u32(sW + dy * K::WSLICE_BYTES), image + (size_t)(g % L) * K::WSTAGE_BYTES + dy * K::WSLICE_BYTES,
                             K::WSLICE_BYTES, b_wfull + 8 * dy);
                }
        } else if (lane == 0) {
            const int total = n_strips * L;
            for (int g = 0; g < total; g++) {
                const int st = g % K::WSTAGES, use = g / K::WSTAGES;
                if (use > 0) mbar_wait(b_wempty + 8 * st, (use - 1) & 1);
                mbar_expect_tx(b_wfull + 8 * st, K::WSTAGE_BYTES);
                bulk_g2s(smem_u32(sW + st * K::WSTAGE_BYTES), image + (size_t)(g % L) * K::WSTAGE_BYTES, K::WSTAGE_BYTES,
                         b_wfull + 8 * st);
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | ((uint32_t)OP::FMT << 7) | ((uint32_t)OP::FMT << 10) |
                                   ((uint32_t)(K::NN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
            int g = 0, c = 0;                                   // (strip, layer) counter, (strip, layer, tile) counter
            for (int s = 0; s < n_strips; s++) {
                const int nb = min(K::NB, my_n - s * K::NB);
                const int T = (7 * nb + 15) / 16;
                for (int l = 0; l < L; l++, g++) {
                    const int st = g % K::WSTAGES;
                    if (!K::SLICED) mbar_wait(b_wfull + 8 * st, (g / K::WSTAGES) & 1);
                    DBG_T(d0)
                    const uint32_t wbase = smem_u32(sW + st * K::WSTAGE_BYTES);
                    const uint32_t abase = smem_u32((l == 0 || (l & 1) == 0) ? sH : sX);   // stem and conv2 read H
                    const uint64_t a_l = umma_desc(abase, K::ROWS * 16, 128);      // tile 0, dy = -1: buffer row 8 - 8
                    const uint64_t b_l = umma_desc(wbase, K::NN * 16, 128);
                    // epilogue arrivals seen so far on each tile barrier: (L + 1) per finished strip, l + 1 needed now
                    const uint32_t ep_par = (uint32_t)(s * (L + 1) + l) & 1u;
#pragma unroll
                    for (int t = 0; t < K::T; t++, c++) {                      // fully unrolled: per-tile constants fold away
                        if (t >= T) break;
                        // rows of tiles t-1, t, t+1 of the previous layer are read; the two epilogue groups finish
                        // tiles out of order, so every tile is waited for once (tile t+1 here, tile 0 at t == 0)
                        if (t == 0) mbar_wait(b_epi, ep_par);
                        if (t + 1 < T) mbar_wait(b_epi + 8 * (t + 1), ep_par);
                        DBG_T(d1)
                        const int slot = c % K::ACC_SLOTS, use = c / K::ACC_SLOTS;
                        if (use > 0) mbar_wait(b_accempty + 8 * slot, (use - 1) & 1);
                        DBG_T(d2)
                        TC_FENCE_AFTER();
                        const uint32_t d = tmem + K::ACC_COL0 + slot * K::NN;
                        // descriptors advance by adding 16-byte units to the start-address field:
                        //   A: +8 per dy (8 rows), +2*ROWS per 16-channel k-step;  B: +kc*NN per dy, +2*NN per k-step
                        const uint64_t a = a_l + (uint64_t)(128 * t);
                        // (the layer-kind branch stays OUTSIDE the unrolled tap loops: this thread is the serial resource of
                        //  the kernel and every extra instruction per tile shows up in the step time)
                        if (l != 0) {
#pragma unroll
                            for (int dy = 0; dy < 3; dy++) {
                                if (K::SLICED && t == 0) mbar_wait(b_wfull + 8 * dy, (uint32_t)g & 1u);
#pragma unroll
                                for (int ks = 0; ks < K::KC / 2; ks++) {
                                    const uint64_t aa = a + 8 * dy + 2 * K::ROWS * ks, bb = b_l + (dy * K::KC + 2 * ks) * K::NN;
                                    if (dy == 0 && ks == 0) umma_f16c<0>(d, aa, bb, idesc); else umma_f16c<1>(d, aa, bb, idesc);
                                }
                                if (K::SLICED && t == T - 1) umma_commit(b_wempty + 8 * dy);  // slice free for the next layer
                            }
                        } else {                                              // stem: 16 (padded) input channels = one k-step
#pragma unroll
                            for (int dy = 0; dy < 3; dy++) {
                                if (K::SLICED && t == 0) mbar_wait(b_wfull + 8 * dy, (uint32_t)g & 1u);
                                const uint64_t aa = a + 8 * dy, bb = b_l + dy * K::STEM_KC * K::NN;
                                if (dy == 0) umma_f16c<0>(d, aa, bb, idesc); else umma_f16c<1>(d, aa, bb, idesc);
                                if (K::SLICED && t == T - 1) umma_commit(b_wempty + 8 * dy);
                            }
                        }
                        umma_commit(b_accfull + 8 * slot);
                        DBG_T(d3)
                    }
                    if (!K::SLICED) umma_commit(b_wempty + 8 * st);
                }
            }
#ifdef C4_TC_PROFILE
            if (dbg && blockIdx.x == 0) { dbg[0] = d0; dbg[1] = d1; dbg[2] = d2; dbg[3] = d3; }
#endif
        }
    } else {
        // ================= epilogue warps
        const int e = warp - 2, quad = warp & 3, half = (e >> 2) % K::SLICES, group = e / K::GROUP_WARPS;   // half = channel slice
        const int et = threadIdx.x - 64;                                     // 0..511
        EpiCtx E;
        E.b_accfull = b_accfull; E.b_accempty = b_accempty; E.b_epi = b_epi;
        E.tmem_acc = tmem + ((uint32_t)(quad * 32) << 16) + K::ACC_COL0 + TC_CH * half;
        E.tmem_res = tmem + ((uint32_t)(quad * 32) << 16) + TC_CH * half;
        E.dst_x = sX + (size_t)(2 * half * K::ROWS + 8 + 32 * quad + lane) * 16;
        E.dst_h = sH + (size_t)(2 * half * K::ROWS + 8 + 32 * quad + lane) * 16;
        E.bias = bias; E.hp = hp;
        E.scratch = scratch + half * K::NB * 128;
        E.lane = lane; E.lm = (lane + 31) & 31; E.lp = (lane + 1) & 31; E.half = half; E.group = group;
        E.rb0 = 4 * quad + (lane >> 3); E.col8 = lane & 7;
        E.calib = CALIB ? reinterpret_cast<unsigned *>(dbg) : nullptr;
        int c = 0;                                                           // global (strip, layer, tile) counter
        for (int s = 0; s < n_strips; s++) {
            const int nb = min(K::NB, my_n - s * K::NB);
            const int T = (7 * nb + 15) / 16;
            const int first = my_first + s * K::NB;
            E.valid_mask = 0;
            for (int t = 0; t < T; t++) {
                const int rb = 16 * t + E.rb0, b = rb / 7;
                if (E.col8 != 0 && rb - 7 * b != 0 && b < nb) E.valid_mask |= 1u << t;
            }
            // ---- input planes (Board.to_array) -> channels 0..15 of H
            for (int i = et; i < nb * 42; i += 32 * TC_EPI_WARPS) {
                const int b = i / 42, px = i - b * 42, r = px / 7, col = px - r * 7;
                const u64 a0 = c0[first + b], a1 = c1[first + b];
                const int bit = 7 * col + (5 - r);
                const uint32_t tomove = ((__popcll(a0 | a1) & 1) == 0) ? OP::ONE : 0u;
                const uint32_t o = (uint32_t)((a0 >> bit) & 1ULL) * OP::ONE, x = (uint32_t)((a1 >> bit) & 1ULL) * OP::ONE;
                const int row = 8 + (7 * b + 1 + r) * 8 + (col + 1);
                *reinterpret_cast<uint4 *>(sH + (size_t)row * 16) = make_uint4(tomove | (o << 16), x, 0u, 0u);
                *reinterpret_cast<uint4 *>(sH + (size_t)(K::ROWS + row) * 16) = make_uint4(0u, 0u, 0u, 0u);
            }
            TC_PROXY_FENCE();
            EPI_BAR();
            if (lane == 0 && e < K::GROUP_WARPS)                             // GROUP_WARPS arrivals per tile barrier and epoch
                for (int t = 0; t < T; t++) mbar_arrive(b_epi + 8 * t);

            tc_epilogue_layer<OP, F, 0, CALIB>(E, 0, T, c); c += T;
            for (int l = 1; l < L - 1; l += 2) {
                tc_epilogue_layer<OP, F, 1, CALIB>(E, l, T, c); c += T;
                if (l + 1 < L - 1) { tc_epilogue_layer<OP, F, 2, CALIB>(E, l + 1, T, c); c += T; }
            }
            tc_epilogue_layer<OP, F, 3, CALIB>(E, L - 1, T, c); c += T;

            // ---- head tails: one warp per board
            EPI_BAR();
            for (int b = e; b < nb; b += TC_EPI_WARPS) {
                float *sc = scratch + b * 128;
                for (int i = lane; i < 126; i += 32) {
                    float bb = i < 42 ? hp[HO_VB] : (i < 84 ? hp[HO_PB] : hp[HO_PB + 1]);
                    float acc = sc[i];                                       // channel slices summed in a fixed order
#pragma unroll
                    for (int q = 1; q < K::SLICES; q++) acc += sc[q * K::NB * 128 + i];
                    sc[i] = leaky(acc + bb);
                }
                __syncwarp();
                head_tail(sc, hp, out + (size_t)(first + b) * 8, lane);
            }
            EPI_BAR();
        }
    }
    TC_FENCE_BEFORE();
    __syncthreads();
    if (warp == 0) {
        __syncwarp();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" :: "r"(tmem) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------ host side
int c4_net_forward_ex(c4_net *net, const uint64_t *c0, const uint64_t *c1, int64_t n, const int32_t *count, float *out,
                      void *stream, int max_ctas, const c4_ly_scratch *scratch);
static uint16_t f2bf(float f)
{
    uint32_t u;
    memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);   // NaN
    uint32_t r = 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)((u + r) >> 16);
}

static uint16_t f2h(float f)
{
    __half h = __float2half_rn(f);
    uint16_t u;
    memcpy(&u, &h, 2);
    return u;
}

uint16_t c4_f2op(float f, bool fp16) { return fp16 ? f2h(f) : f2bf(f); }

// head parameters of the blob (from the value head's 1x1 conv on) -> the fp32 head block; the 1x1 conv weights go to vw [F]
// and pw [2][F]
void c4_pack_heads(const float *p, int F, float *hp, float *vw, float *pw)
{
    memcpy(vw, p, F * 4); p += F;
    hp[HO_VB] = *p++;
    for (int i = 0; i < 42; i++)
        for (int j = 0; j < 42; j++) hp[HO_FCT + j * 42 + i] = p[i * 42 + j];
    p += 42 * 42;
    memcpy(hp + HO_FCB, p, 42 * 4); p += 42;
    memcpy(hp + HO_FC1W, p, 42 * 4); p += 42;
    hp[HO_FC1B] = *p++;
    hp[HO_W1] = *p++; hp[HO_W2] = *p++;
    memcpy(pw, p, F * 4); memcpy(pw + F, p + F, F * 4); p += 2 * F;
    hp[HO_PB] = *p++; hp[HO_PB + 1] = *p++;
    memcpy(hp + HO_POLW, p, 7 * 84 * 4); p += 7 * 84;
    memcpy(hp + HO_POLB, p, 7 * 4);
}

// pack W[co][ci][ky][kx] (fp32) into [co][k = (ky*3+kx)*CINP + ci] 16-bit rows of (9*CINP + 8) elements
static void pack_conv(const float *W, int F, int cin, int cinp, uint16_t *dst, bool fp16)
{
    const int ws = 9 * cinp + 8;
    for (int co = 0; co < F; co++)
        for (int ci = 0; ci < cin; ci++)
            for (int ky = 0; ky < 3; ky++)
                for (int kx = 0; kx < 3; kx++)
                {
                    float w = W[((co * cin + ci) * 3 + ky) * 3 + kx];
                    dst[(size_t)co * ws + (ky * 3 + kx) * cinp + ci] = fp16 ? f2h(w) : f2bf(w);
                }
}

template <int F, int WARPS>
static size_t smem_resident(int R) { return ImageA<F>::total(R) + (size_t)WARPS * (2 * NPX * (F * 2 + 16) + SCRATCH_BYTES); }
template <int F, int WARPS>
static size_t smem_streamed(int R)
{
    return ImageA<F>::conv_bytes() + (size_t)(1 + 2 * R) * F * 4 + HEAD_FLOATS * 4 +
           (size_t)WARPS * (2 * NPX * (F * 2 + 16) + SCRATCH_BYTES);
}

#define WARPS_A 8
#define WARPS_B 6

// blob sections in front of the heads: [4 header][stem W F*27][stem b F] + 2R x ([W F*F*9][b F])
// The blob with the trunk running at activations * s (s = 2^-k): LeakyReLU is positively homogeneous, so scaling the stem's
// weights and EVERY conv bias by s scales every trunk activation by exactly s (power of two: the roundings do not move),
// and dividing the heads' 1x1 conv weights by s gives the original head inputs back.  Returns false if a scaled weight
// does not fit the operand type (fp16: |w| > 65504).
static bool scaled_blob(const float *blob, int64_t n, int F, int R, int k, bool fp16, std::vector<float> &out)
{
    out.assign(blob, blob + n);
    const float s = ldexpf(1.f, -k), inv = ldexpf(1.f, k);
    float *p = out.data() + 4;
    for (int i = 0; i < F * 27 + F; i++) p[i] *= s;                                // stem weights + bias
    p += F * 27 + F;
    for (int l = 0; l < 2 * R; l++) {
        p += (size_t)F * F * 9;
        for (int i = 0; i < F; i++) p[i] *= s;                                     // conv bias (BN folded)
        p += F;
    }
    for (int i = 0; i < F; i++) p[i] *= inv;                                       // value head 1x1 conv weights
    float *q = p + F + 1 + 42 * 42 + 42 + 42 + 1 + 2;
    for (int i = 0; i < 2 * F; i++) q[i] *= inv;                                   // policy head 1x1 conv weights
    // conv weights are the 16-bit operands (biases and heads stay fp32): every one must be finite and fit the operand type
    const float lim = fp16 ? 65504.f : 3.38e38f;
    const float *w = out.data() + 4;
    for (int i = 0; i < F * 27; i++)
        if (!(fabsf(w[i]) <= lim)) return false;
    w += F * 27 + F;
    for (int l = 0; l < 2 * R; l++) {
        for (size_t i = 0; i < (size_t)F * F * 9; i++)
            if (!(fabsf(w[i]) <= lim)) return false;
        w += (size_t)F * F * 9 + F;
    }
    return true;
}

// (re)build and upload the device images of the network from a (scaled) blob
static int upload_images(c4_net *net, const float *blob)
{
    const int F = net->F, R = net->R;
    const bool fp16 = net->fp16;
    const size_t total = (F == 32) ? ImageA<32>::total(R) : ImageA<64>::total(R);
    const size_t stem_b = (F == 32) ? ImageA<32>::stem_bytes() : ImageA<64>::stem_bytes();
    const size_t conv_b = (F == 32) ? ImageA<32>::conv_bytes() : ImageA<64>::conv_bytes();
    std::vector<unsigned char> img(total, 0);
    const float *p = blob + 4;
    float *bias = reinterpret_cast<float *>(img.data() + stem_b + 2 * R * conv_b);
    float *hp = bias + (1 + 2 * R) * F;
    pack_conv(p, F, 3, 16, reinterpret_cast<uint16_t *>(img.data()), fp16);
    p += F * 27;
    memcpy(bias, p, F * 4);
    p += F;
    for (int l = 0; l < 2 * R; l++) {
        pack_conv(p, F, F, F, reinterpret_cast<uint16_t *>(img.data() + stem_b + l * conv_b), fp16);
        p += (size_t)F * F * 9;
        memcpy(bias + (1 + l) * F, p, F * 4);
        p += F;
    }
    c4_pack_heads(p, F, hp, hp + HO_VW, hp + HO_PW);
    net->image_bytes = total;
    if (!net->image && cudaMalloc(&net->image, total) != cudaSuccess) { c4_set_error("cudaMalloc failed"); return -2; }
    C4_CUDA(cudaMemcpy(net->image, img.data(), total, cudaMemcpyHostToDevice));
    if (net->use_tc) {
        // tcgen05 image: per layer [dy][k-chunk][n = dx*F + co][8 ci] 16-bit, K-major SWIZZLE_NONE core matrices
        const int L = 1 + 2 * R;
        const int KC = F / 8, NN = 3 * F;
        const size_t stage = (size_t)3 * KC * NN * 16;
        const size_t small_bytes = (size_t)(L * F + HEAD_FLOATS) * 4;
        std::vector<unsigned char> tc((size_t)L * stage + small_bytes, 0);
        const float *q = blob + 4;
        for (int l = 0; l < L; l++) {
            const int cin = l == 0 ? 3 : F, kc = (l == 0 && F == 32) ? 2 : KC;    // = TcK<F>::STEM_KC for the stem
            uint16_t *dst = reinterpret_cast<uint16_t *>(tc.data() + (size_t)l * stage);
            for (int co = 0; co < F; co++)
                for (int ci = 0; ci < cin; ci++)
                    for (int ky = 0; ky < 3; ky++)
                        for (int kx = 0; kx < 3; kx++) {
                            float w = q[((co * cin + ci) * 3 + ky) * 3 + kx];
                            size_t idx = ((size_t)(ky * kc + ci / 8) * NN + (kx * F + co)) * 8 + (ci % 8);
                            dst[idx] = fp16 ? f2h(w) : f2bf(w);
                        }
            q += (size_t)F * cin * 9 + F;
        }
        memcpy(tc.data() + (size_t)L * stage, bias, small_bytes);               // biases + head block, as in image A
        if (!net->image_tc && cudaMalloc(&net->image_tc, tc.size()) != cudaSuccess) { c4_set_error("cudaMalloc failed"); return -2; }
        C4_CUDA(cudaMemcpy(net->image_tc, tc.data(), tc.size(), cudaMemcpyHostToDevice));
    }
    return 0;
}

// Largest |activation| any trunk layer produces on a fixed set of 512 calibration positions (random stones of both colours,
// 0..40 plies, deterministic), measured with the kernel that runs the network (tcgen05 tower or layered kernels).  Inf / NaN
// come back as a huge value.
static int calibrate_range(c4_net *net, float *max_abs)
{
    const int n = 512;
    std::vector<u64> c0(n), c1(n);
    u64 rng = 0x9E3779B97F4A7C15ULL;
    for (int i = 0; i < n; i++) {
        int h[7] = {0, 0, 0, 0, 0, 0, 0};
        u64 a = 0, b = 0;
        rng = rng * 6364136223846793005ULL + 1442695040888963407ULL;
        const int plies = (int)((rng >> 33) % 41);
        for (int k = 0; k < plies; k++) {
            rng = rng * 6364136223846793005ULL + 1442695040888963407ULL;
            int col = (int)((rng >> 33) % 7);
            for (int t = 0; t < 7 && h[col] == 6; t++) col = (col + 1) % 7;
            if (h[col] == 6) break;
            const u64 bit = 1ULL << (7 * col + h[col]++);
            if (k & 1) b |= bit; else a |= bit;
        }
        c0[i] = a; c1[i] = b;
    }
    u64 *d0 = nullptr, *d1 = nullptr;
    float *out = nullptr;
    unsigned *mx = nullptr;
    C4_CUDA(cudaMalloc(&d0, n * 8)); C4_CUDA(cudaMalloc(&d1, n * 8)); C4_CUDA(cudaMalloc(&out, n * 32));
    C4_CUDA(cudaMalloc(&mx, 64));
    C4_CUDA(cudaMemcpy(d0, c0.data(), n * 8, cudaMemcpyHostToDevice));
    C4_CUDA(cudaMemcpy(d1, c1.data(), n * 8, cudaMemcpyHostToDevice));
    C4_CUDA(cudaMemset(mx, 0, 64));
    if (net->layers) {
        const int rc = c4_ly_forward(net, (const uint64_t *)d0, (const uint64_t *)d1, n, nullptr, out, 0, 148, nullptr, mx);
        if (rc) return rc;
    } else {
        const int tc_smem = net->F == 32 ? TcK<32>::total(net->R) : TcK<64>::total(net->R);
        auto k = net->F == 32 ? k_net_tc<OpFP16, 32, true> : k_net_tc<OpFP16, 64, true>;
        C4_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem));
        k<<<32, TC_THREADS, tc_smem>>>((const unsigned char *)net->image_tc, net->R, d0, d1, n, nullptr, out,
                                       reinterpret_cast<long long *>(mx));
        C4_CUDA(cudaGetLastError());
    }
    unsigned bits = 0;
    C4_CUDA(cudaMemcpy(&bits, mx, 4, cudaMemcpyDeviceToHost));
    cudaFree(d0); cudaFree(d1); cudaFree(out); cudaFree(mx);
    memcpy(max_abs, &bits, 4);
    return 0;
}

static unsigned long long next_net_uid = 1;   // c4_net::uid of the next network created

extern "C" int c4_net_create(int device, const float *blob, int64_t n_floats, c4_net **out)
{
    C4_REQUIRE(blob && out, "c4_net_create: null pointer");
    C4_REQUIRE(n_floats >= 4 && (int)blob[0] == 0xC4B2, "c4_net_create: bad blob magic");
    const int F = (int)blob[1], R = (int)blob[2], n_fc = (int)blob[3] & 0xff;
    const bool fp16 = (((int)blob[3] >> 8) & 0xff) != 1;        // header[3] = n_fc | (operand dtype << 8) | (kernel << 16)
    const int kernel_sel = ((int)blob[3] >> 16) & 0xff;         // 0 = auto (tcgen05 when filters == 32), 1 = mma.sync,
                                                                // 2 = layer by layer (c4_layers.cu)
    if (kernel_sel == 2) {
        C4_REQUIRE(F >= 16 && F <= 256 && F % 16 == 0,
                   "c4_net_create: the layered kernels need filters a multiple of 16 in 16..256");
        C4_REQUIRE(R >= 1 && R <= 40, "c4_net_create: the layered kernels need n_residuals in 1..40");
    } else {
        C4_REQUIRE(F == 32 || F == 64, "c4_net_create: filters must be 32 or 64");
        C4_REQUIRE(R >= 1 && R <= 16, "c4_net_create: n_residuals out of range");
    }
    const int64_t expect = 4 + (int64_t)F * 27 + F + (int64_t)2 * R * ((int64_t)F * F * 9 + F) + F + 1 + 42 * 42 + 42 +
                           42 + 1 + 2 + 2 * F + 2 + 7 * 84 + 7;
    C4_REQUIRE(n_floats == expect, "c4_net_create: blob size does not match its header");
    int ndev = 0;
    C4_CUDA(cudaGetDeviceCount(&ndev));
    C4_REQUIRE(device >= 0 && device < ndev, "no such CUDA device (there is no CPU fallback)");
    C4_CUDA(cudaSetDevice(device));

    c4_net *net = new c4_net();
    net->uid = next_net_uid++;
    net->device = device; net->F = F; net->R = R; net->n_fc = n_fc; net->fp16 = fp16;
    net->image = nullptr; net->image_tc = nullptr;
    net->layers = kernel_sel == 2; net->ly = nullptr;
    net->scale_log2 = 0; net->calib_max = 0.f;
    net->flops = 2.0 * (42.0 * 27 * F + 2.0 * R * 42 * 9 * F * F + 42.0 * F + (double)n_fc * 42 * 42 + 42 + 42.0 * F * 2 +
                        84.0 * 7);
    const int tc_smem = (F == 32) ? TcK<32>::total(R) : TcK<64>::total(R);
    net->use_tc = kernel_sel != 1 && !net->layers && tc_smem <= 227 * 1024;
    int rc = 0;
    if (net->layers) {
        if ((rc = c4_ly_setup(net))) { c4_net_destroy(net); return rc; }
    } else if (net->use_tc) {
        if (F == 32) {
            C4_CUDA(cudaFuncSetAttribute(k_net_tc<OpFP16, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem));
            C4_CUDA(cudaFuncSetAttribute(k_net_tc<OpBF16, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem));
        } else {
            C4_CUDA(cudaFuncSetAttribute(k_net_tc<OpFP16, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem));
            C4_CUDA(cudaFuncSetAttribute(k_net_tc<OpBF16, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem));
        }
    }
    if (net->layers) {
        // (no mma.sync kernel: c4_ly_setup above)
    } else if (F == 32) {
        // the mma.sync kernel for 32 filters keeps every layer's weights resident in shared memory (up to 4 residual blocks);
        // deeper 32-filter networks run on the tcgen05 kernel only, which streams the weights layer by layer
        const bool resident_ok = smem_resident<32, WARPS_A>(R) <= 227 * 1024;
        if (!net->use_tc && !resident_ok) {
            c4_net_destroy(net);
            c4_set_error("invalid argument: c4_net_create: this 32-filter network is too deep for the mma.sync kernel (use kernel auto)");
            return -1;
        }
        if (resident_ok) {
            C4_CUDA(cudaFuncSetAttribute(k_net_resident<OpFP16, 32, WARPS_A>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem_resident<32, WARPS_A>(R)));
            C4_CUDA(cudaFuncSetAttribute(k_net_resident<OpBF16, 32, WARPS_A>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem_resident<32, WARPS_A>(R)));
        }
    } else {
        C4_CUDA(cudaFuncSetAttribute(k_net_streamed<OpFP16, 64, WARPS_B>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)smem_streamed<64, WARPS_B>(R)));
        C4_CUDA(cudaFuncSetAttribute(k_net_streamed<OpBF16, 64, WARPS_B>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)smem_streamed<64, WARPS_B>(R)));
    }

    // fp16 operands have 5 exponent bits: a trunk whose activations (or BN-folded weights) leave +-65504 would turn into
    // Inf / NaN.  The trunk is therefore run at activations * 2^-k, k chosen here: calibrate on 512 positions with the
    // kernel itself and keep a 16x margin.  Networks in the usual range (the reference's checkpoint peaks below 4) get
    // k = 0, i.e. exactly the unscaled arithmetic.  What calibration cannot foresee is caught at run time: a non-finite
    // network answer never enters a tree and makes the engine call fail (c4_search.cu / c4_fused.cu).
    std::vector<float> sb;
    int k = 0;
    bool ok = false;
    for (int attempt = 0; attempt < 12 && !ok; attempt++) {
        if (!scaled_blob(blob, n_floats, F, R, k, fp16, sb)) { k += 12; continue; }     // a weight overflows fp16
        if ((rc = net->layers ? c4_ly_upload(net, sb.data()) : upload_images(net, sb.data()))) { c4_net_destroy(net); return rc; }
        if (!fp16 || !(net->use_tc || net->layers) || getenv("C4_NET_NO_CALIBRATION")) { ok = true; break; }
        float m = 0.f;
        if ((rc = calibrate_range(net, &m))) { c4_net_destroy(net); return rc; }
        net->calib_max = m;
        if (m <= 4096.f) ok = true;                                                    // NaN compares false
        else if (m < 3.0e38f) k += (int)ceilf(log2f(m / 2048.f));
        else k += 12;
    }
    if (!ok) {
        c4_net_destroy(net);
        c4_set_error("invalid argument: c4_net_create: this network's weights / activations do not fit fp16 operands at any "
                     "power-of-two scale (NaN weights?); use operand_dtype='bf16'");
        return -1;
    }
    net->scale_log2 = k;
    *out = net;
    return 0;
}

extern "C" int c4_net_create_external(int device, c4_eval_fn fn, void *user, c4_net **out)
{
    C4_REQUIRE(fn && out, "c4_net_create_external: null pointer");
    int ndev = 0;
    C4_CUDA(cudaGetDeviceCount(&ndev));
    C4_REQUIRE(device >= 0 && device < ndev, "no such CUDA device (there is no CPU fallback)");
    C4_CUDA(cudaSetDevice(device));
    c4_net *net = new c4_net();
    if (cudaMallocHost((void **)&net->ext_count, sizeof(int32_t)) != cudaSuccess) {
        delete net;
        c4_set_error("cudaMallocHost failed");
        return -2;
    }
    net->uid = next_net_uid++;
    net->device = device;
    net->ext_fn = fn;
    net->ext_user = user;
    *out = net;
    return 0;
}

extern "C" int c4_net_destroy(c4_net *net)
{
    if (!net) return 0;
    cudaSetDevice(net->device);
    if (net->image) cudaFree(net->image);
    if (net->image_tc) cudaFree(net->image_tc);
    if (net->ext_count) cudaFreeHost(net->ext_count);
    c4_ly_destroy(net);
    delete net;
    return 0;
}

extern "C" double c4_net_flops_per_position(const c4_net *net) { return net ? net->flops : 0.0; }
extern "C" double c4_net_get(const c4_net *net, int key)
{
    if (!net) return -1.0;
    if (net->ext_fn) return 0.0;                                 // a caller-served network has none of these
    switch (key) {
    case 0: return net->F;
    case 1: return net->R;
    case 2: return net->fp16 ? 0.0 : 1.0;
    case 3: return net->scale_log2;
    case 4: return net->use_tc ? 1.0 : 0.0;
    case 5: return net->calib_max;
    case 6: return net->layers ? 2.0 : net->use_tc ? 1.0 : 0.0;
    default: return -1.0;
    }
}
unsigned long long c4_net_uid(const c4_net *net) { return net ? net->uid : 0ULL; }   // internal (not part of the C ABI)
int c4_net_filters(const c4_net *net) { return net ? net->F : 0; }                  // internal
int c4_net_device(const c4_net *net) { return net ? net->device : -1; }             // internal
bool c4_net_external(const c4_net *net) { return net && net->ext_fn; }             // internal
bool c4_net_layered(const c4_net *net) { return net && net->layers; }              // internal

extern "C" int c4_net_forward(c4_net *net, const uint64_t *c0, const uint64_t *c1, int64_t n, const int32_t *count,
                              float *out, void *stream)
{
    return c4_net_forward_ex(net, c0, c1, n, count, out, stream, 148, nullptr);
}

// internal: same, with a cap on the number of CTAs (the self-play engine leaves SMs to the concurrent tree pass) and, for
// a layered network, the activation scratch of the caller (null: the network's own, c4_ly_forward)
int c4_net_forward_ex(c4_net *net, const uint64_t *c0, const uint64_t *c1, int64_t n, const int32_t *count, float *out,
                      void *stream, int max_ctas, const c4_ly_scratch *scratch)
{
    C4_REQUIRE(net && (n == 0 || (c0 && c1 && out)), "c4_net_forward: null pointer");
    C4_REQUIRE(n >= 0 && n < (1LL << 31), "c4_net_forward: n out of range");
    if (n == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    C4_CUDA(cudaSetDevice(net->device));
    if (net->ext_fn) {
        // caller-served network: the host needs the leaf count to hand over the batch, hence one synchronise per call
        if (count) {
            C4_CUDA(cudaMemcpyAsync(net->ext_count, count, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
            C4_CUDA(cudaStreamSynchronize(s));
            n = std::min<int64_t>(n, std::max(0, *net->ext_count));
            if (n == 0) return 0;
        }
        const int rc = net->ext_fn(net->ext_user, c0, c1, n, out, stream);
        if (rc) {
            c4_set_error("the caller's evaluator failed (c4_eval_fn returned " + std::to_string(rc) + ")");
            return -5;
        }
        C4_CUDA(cudaSetDevice(net->device));                    // (the callback may have switched devices)
        return 0;
    }
    if (net->layers) {
        return c4_ly_forward(net, c0, c1, n, count, out, s, max_ctas, scratch, nullptr);
    } else if (net->use_tc) {
        int grid = (int)std::min<int64_t>(std::max(1, std::min(max_ctas, 148)), n);
        auto k = net->F == 32 ? (net->fp16 ? k_net_tc<OpFP16, 32> : k_net_tc<OpBF16, 32>)
                              : (net->fp16 ? k_net_tc<OpFP16, 64> : k_net_tc<OpBF16, 64>);
        const int tc_smem = net->F == 32 ? TcK<32>::total(net->R) : TcK<64>::total(net->R);
        static long long *dbg = nullptr;
        static bool dbg_on = getenv("C4_TC_DEBUG") != nullptr;
        if (dbg_on && !dbg) { cudaMalloc(&dbg, 16 * sizeof(long long)); cudaMemset(dbg, 0, 16 * sizeof(long long)); }
        k<<<grid, TC_THREADS, tc_smem, s>>>((const unsigned char *)net->image_tc, net->R, (const u64 *)c0,
                                                         (const u64 *)c1, (int)n, count, out, dbg);
        if (dbg_on) {
            long long h[16];
            cudaStreamSynchronize(s);
            cudaMemcpy(h, dbg, sizeof(h), cudaMemcpyDeviceToHost);
            cudaMemset(dbg, 0, 16 * sizeof(long long));
            fprintf(stderr, "[tc dbg] mma: wait_w %lld wait_epi %lld wait_accempty %lld issue %lld | epi warp0: wait_accfull %lld ld %lld "
                            "sts/heads %lld store-wait+fence %lld loop %lld | arrive_accempty %lld shfl+fp %lld sttm %lld\n", h[0], h[1], h[2], h[3], h[8], h[9], h[10], h[11], h[12], h[13], h[14], h[15]);
        }
    } else if (net->F == 32) {
        int grid = (int)std::min<int64_t>(148, (n + WARPS_A - 1) / WARPS_A);
        auto k = net->fp16 ? k_net_resident<OpFP16, 32, WARPS_A> : k_net_resident<OpBF16, 32, WARPS_A>;
        k<<<grid, WARPS_A * 32, smem_resident<32, WARPS_A>(net->R), s>>>(
            (const unsigned char *)net->image, (int)net->image_bytes, net->R, (const u64 *)c0, (const u64 *)c1, (int)n,
            count, out);
    } else {
        int grid = (int)std::min<int64_t>(148, (n + WARPS_B - 1) / WARPS_B);
        auto k = net->fp16 ? k_net_streamed<OpFP16, 64, WARPS_B> : k_net_streamed<OpBF16, 64, WARPS_B>;
        k<<<grid, WARPS_B * 32, smem_streamed<64, WARPS_B>(net->R), s>>>(
            (const unsigned char *)net->image, net->R, (const u64 *)c0, (const u64 *)c1, (int)n, count, out);
    }
    C4_CUDA(cudaGetLastError());
    return 0;
}
