// c4_layers.cu -- the network one layer per launch (kernel "layers": any F = 16..256 in steps of 16, R = 1..40).
//
// The fused tower (k_net_tc) keeps a strip's whole tower on chip, which limits it to 32 and 64 filters.  Here every 3x3
// conv is its own launch of k_layers_conv and the activations live in global memory between launches (at 128 filters a
// 2,400-board pass is 34 MB per 16-bit copy: L2-resident on a B200):
//
//  * layout: the padded pixel strip of c4_tc.cuh over the whole batch.  Board b owns rows LY_GUARD + 56 b .. + 55: 7
//    row-blocks of 8 pixels, row-block 0 and pixel column 0 are zero.  16-bit operand copies are [k-chunk][row][8]
//    (K-major core matrices), the fp32 trunk stream is [F/16][row][16].  Pad rows are zeroed once at allocation and
//    never written, so a board's valid outputs only ever read its own pixels and zeros: its answer does not depend on
//    the batch, its neighbours, the CTA count or stale rows of an earlier, larger batch.
//  * k_layers_conv: implicit GEMM, M = 128 rows per tile, N = F, K = 9 taps x Cin.  A CTA takes MT tiles at a time
//    (MT x F <= 256 TMEM columns per accumulator slot, two slots) and loads their rows plus 16 rows either side once
//    per k-chunk with cp.async.bulk; a tap (dy, dx) is the descriptor start address moved by 8 dy + dx rows (16-byte
//    rows, SWIZZLE_NONE: any row offset is a valid start).  Weights stream through a 3-stage ring of 32 KB stages.
//    tcgen05.mma kind::f16, fp32 accumulation in TMEM, one fixed MMA order per output row.
//    Epilogue (8 warps, one row per thread): bias, residual add where a block closes, LeakyReLU, then the 16-bit copy
//    for the next layer and / or the fp32 trunk stream.
//  * k_layers_heads: value / policy 1x1 convs from the fp32 trunk stream, then head_tail, one warp per board.
// Warp roles of k_layers_conv: warp 0 = loads (A windows + weight ring), warp 1 = MMA issuer, warps 2..9 = epilogue.
#include <algorithm>
#include <mutex>
#include <string>
#include <vector>

#include "c4_common.cuh"
#include "c4_tc.cuh"
#include "c4_layers.cuh"

#define LY_THREADS 320
#define LY_EPI_WARPS 8
#define LY_WSTAGES 3
#define LY_WSTAGE_BYTES 32768
// at least half an SM's shared memory: two layered CTAs (of one forward or of two concurrent ones) never share an SM, so
// none waits for another's TMEM allocation
#define LY_MIN_SMEM (120 * 1024)

__host__ __device__ static inline int ly_mt(int F) { return F <= 64 ? 4 : 256 / F; }      // tiles per CTA step
__host__ __device__ static inline int ly_wrows(int F) { return 128 * ly_mt(F) + 32; }      // A window rows
static int ly_smem(int F)
{
    return std::max(LY_MIN_SMEM, (F / 8) * ly_wrows(F) * 16 + LY_WSTAGES * LY_WSTAGE_BYTES + 256);
}
#define LY_MAX_SMEM (32 * (128 + 32) * 16 + LY_WSTAGES * LY_WSTAGE_BYTES + 256)   // F = 256

struct LyConv {
    const unsigned char *w;    // this layer's weights: 9 x Cin/16 blocks (tap-major) of [2 k-chunks][F][8] 16-bit
    const float *bias;         // [F]
    const unsigned char *src;  // [kcin][rows][8] 16-bit
    unsigned char *dst;        // [F/8][rows][8] 16-bit, or null (last layer)
    float *res;                // [F/16][rows][16] fp32 trunk stream
    unsigned *calib;           // range calibration only: running max of the bits of |activation|
    const int *count;          // device position count (or null)
    size_t rows;
    int F, kcin, kind;         // kind: 0 stem, 1 first conv of a block, 2 second conv, 3 second conv of the last block
    int base, n;               // positions [base, base + n) of the call; count caps it
};

template <typename OP>
__global__ void __launch_bounds__(LY_THREADS, 1) k_layers_conv(const LyConv a)
{
    extern __shared__ __align__(128) unsigned char smem[];
    int n = a.n;
    if (a.count) n = min(n, *a.count - a.base);
    if (n <= 0) return;
    const int F = a.F, MT = ly_mt(F), WROWS = ly_wrows(F);
    const int G = ((56 * n + 127) / 128 + MT - 1) / MT;                       // groups of MT tiles
    if ((int)blockIdx.x >= G) return;
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int KS = a.kcin / 2, NBLK = 9 * KS, BLK = F * 32;                 // 16-channel k-steps, weight blocks
    const int SPS = LY_WSTAGE_BYTES / BLK, NST = (NBLK + SPS - 1) / SPS;     // blocks per stage, stages per layer
    unsigned char *sA = smem, *sW = smem + (F / 8) * WROWS * 16;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sW + LY_WSTAGES * LY_WSTAGE_BYTES);
    const uint32_t b_afull = smem_u32(bars), b_aempty = b_afull + 8, b_wfull = b_afull + 16;
    const uint32_t b_wempty = b_wfull + 8 * LY_WSTAGES, b_accfull = b_wempty + 8 * LY_WSTAGES, b_accempty = b_accfull + 16;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 + 2 * LY_WSTAGES + 4);
    const int SLOT = MT * F;
    uint32_t ncols = 32;
    while (ncols < (uint32_t)(2 * SLOT)) ncols <<= 1;

    if (threadIdx.x == 0) {
        mbar_init(b_afull, 1); mbar_init(b_aempty, 1);
        for (int i = 0; i < LY_WSTAGES; i++) { mbar_init(b_wfull + 8 * i, 1); mbar_init(b_wempty + 8 * i, 1); }
        for (int i = 0; i < 2; i++) { mbar_init(b_accfull + 8 * i, 1); mbar_init(b_accempty + 8 * i, LY_EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" :: "r"(smem_u32(tmem_slot)), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    TC_FENCE_BEFORE();
    __syncthreads();
    TC_FENCE_AFTER();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        // ================= loads: per group the A window (every k-chunk), then the layer's weights stage by stage
        if (lane == 0) {
            int wuse = 0;
            for (int i = 0, g = blockIdx.x; g < G; g += gridDim.x, i++) {
                if (i > 0) mbar_wait(b_aempty, (i - 1) & 1);
                mbar_expect_tx(b_afull, (uint32_t)(a.kcin * WROWS * 16));
                // window row 0 = board-space row 128 MT g - 16 = buffer row 128 MT g (LY_GUARD = 16)
                for (int kc = 0; kc < a.kcin; kc++)
                    bulk_g2s(smem_u32(sA + kc * WROWS * 16), a.src + ((size_t)kc * a.rows + (size_t)g * MT * 128) * 16,
                             WROWS * 16, b_afull);
                for (int s = 0; s < NST; s++, wuse++) {
                    const int st = wuse % LY_WSTAGES, u = wuse / LY_WSTAGES;
                    if (u > 0) mbar_wait(b_wempty + 8 * st, (u - 1) & 1);
                    const uint32_t bytes = (uint32_t)(min(SPS, NBLK - s * SPS) * BLK);
                    mbar_expect_tx(b_wfull + 8 * st, bytes);
                    bulk_g2s(smem_u32(sW + st * LY_WSTAGE_BYTES), a.w + (size_t)s * SPS * BLK, bytes, b_wfull + 8 * st);
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | ((uint32_t)OP::FMT << 7) | ((uint32_t)OP::FMT << 10) |
                                   ((uint32_t)(F >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
            const uint32_t a0 = smem_u32(sA), w0 = smem_u32(sW);
            int wuse = 0;
            for (int i = 0, g = blockIdx.x; g < G; g += gridDim.x, i++) {
                const int slot = i & 1;
                if (i >= 2) mbar_wait(b_accempty + 8 * slot, ((i >> 1) - 1) & 1);
                mbar_wait(b_afull, i & 1);
                TC_FENCE_AFTER();
                const uint32_t d = tmem + slot * SLOT;
                for (int s = 0; s < NST; s++, wuse++) {
                    const int st = wuse % LY_WSTAGES;
                    mbar_wait(b_wfull + 8 * st, (wuse / LY_WSTAGES) & 1);
                    TC_FENCE_AFTER();
                    const int nb = min(SPS, NBLK - s * SPS);
                    for (int j = 0; j < nb; j++) {
                        const int blk = s * SPS + j, tap = blk / KS, ks = blk - tap * KS;
                        const int shift = 16 + 8 * (tap / 3 - 1) + (tap % 3 - 1);
                        const uint64_t bd = umma_desc(w0 + st * LY_WSTAGE_BYTES + j * BLK, F * 16, 128);
                        for (int mt = 0; mt < MT; mt++) {
                            const uint64_t ad = umma_desc(a0 + (uint32_t)((2 * ks * WROWS + shift + 128 * mt) * 16), WROWS * 16, 128);
                            umma_f16(d + mt * F, ad, bd, idesc, blk > 0 ? 1u : 0u);
                        }
                    }
                    umma_commit(b_wempty + 8 * st);
                }
                umma_commit(b_aempty);
                umma_commit(b_accfull + 8 * slot);
            }
        }
    } else {
        // ================= epilogue: TMEM lane quadrant = warp % 4, channel slices of 16 alternate between two warps
        const int quad = warp & 3, half = (warp - 2) >> 2;
        const bool to_res = a.kind != 1, add_res = a.kind >= 2;
        for (int i = 0, g = blockIdx.x; g < G; g += gridDim.x, i++) {
            const int slot = i & 1;
            mbar_wait(b_accfull + 8 * slot, (i >> 1) & 1);
            TC_FENCE_AFTER();
            for (int mt = 0; mt < MT; mt++) {
                const int r = (g * MT + mt) * 128 + 32 * quad + lane, b = r / 56, rr = r - 56 * b;
                const bool valid = b < n && rr >= 8 && (rr & 7) != 0;
                const size_t row = (size_t)(LY_GUARD + r);
                const uint32_t ta = tmem + ((uint32_t)(quad * 32) << 16) + slot * SLOT + mt * F;
                for (int c16 = half; c16 < F / 16; c16 += 2) {
                    float v[16];
                    tmem_ld16(ta + 16 * c16, v);
                    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
                    if (valid) {
                    float4 *rp = reinterpret_cast<float4 *>(a.res + ((size_t)c16 * a.rows + row) * 16);
                    const float4 *bp = reinterpret_cast<const float4 *>(a.bias + 16 * c16);
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const float4 bb = bp[q];
                        float4 y = make_float4(v[4 * q] + bb.x, v[4 * q + 1] + bb.y, v[4 * q + 2] + bb.z, v[4 * q + 3] + bb.w);
                        if (add_res) {
                            const float4 rs = rp[q];
                            y.x += rs.x; y.y += rs.y; y.z += rs.z; y.w += rs.w;
                        }
                        v[4 * q] = leaky(y.x); v[4 * q + 1] = leaky(y.y); v[4 * q + 2] = leaky(y.z); v[4 * q + 3] = leaky(y.w);
                    }
                    if (a.calib) {
                        unsigned mu = 0u;
#pragma unroll
                        for (int j = 0; j < 16; j++) mu = max(mu, __float_as_uint(fabsf(v[j])));
                        atomicMax(a.calib, mu);
                    }
                    if (to_res)
#pragma unroll
                        for (int q = 0; q < 4; q++) rp[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
                    if (a.dst) {
                        unsigned char *p = a.dst + ((size_t)(2 * c16) * a.rows + row) * 16;
                        *reinterpret_cast<uint4 *>(p) =
                            make_uint4(OP::pack(v[0], v[1]), OP::pack(v[2], v[3]), OP::pack(v[4], v[5]), OP::pack(v[6], v[7]));
                        *reinterpret_cast<uint4 *>(p + a.rows * 16) =
                            make_uint4(OP::pack(v[8], v[9]), OP::pack(v[10], v[11]), OP::pack(v[12], v[13]), OP::pack(v[14], v[15]));
                    }
                    }
                    __syncwarp();
                }
            }
            TC_FENCE_BEFORE();
            __syncwarp();
            if (lane == 0) mbar_arrive(b_accempty + 8 * slot);                // accumulator slot free for the MMA warp
        }
    }
    __syncwarp();
    TC_FENCE_BEFORE();
    __syncthreads();
    if (warp == 0) {
        TC_FENCE_AFTER();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" :: "r"(tmem), "r"(ncols) : "memory");
    }
}

// bitboards -> input planes (Board.to_array, oinkoink/board.py:147-154) in channels 0..15 of the stem's operand
template <typename OP>
__global__ void k_layers_input(const u64 *__restrict__ c0, const u64 *__restrict__ c1, int base, int n,
                               const int *__restrict__ count, unsigned char *__restrict__ in, size_t rows)
{
    if (count) n = min(n, *count - base);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n * 42; i += gridDim.x * blockDim.x) {
        const int b = i / 42, px = i - b * 42, r = px / 7, col = px - r * 7;
        const u64 a0 = c0[base + b], a1 = c1[base + b];
        const int bit = 7 * col + (5 - r);
        const uint32_t tomove = ((__popcll(a0 | a1) & 1) == 0) ? OP::ONE : 0u;
        const uint32_t o = (uint32_t)((a0 >> bit) & 1ULL) * OP::ONE, x = (uint32_t)((a1 >> bit) & 1ULL) * OP::ONE;
        const size_t row = LY_GUARD + 56 * (size_t)b + (r + 1) * 8 + (col + 1);
        *reinterpret_cast<uint4 *>(in + row * 16) = make_uint4(tomove | (o << 16), x, 0u, 0u);
        *reinterpret_cast<uint4 *>(in + (rows + row) * 16) = make_uint4(0u, 0u, 0u, 0u);
    }
}

// value / policy heads (model.py:77-91,107-117) from the fp32 trunk stream; one warp per board, fixed summation order
#define LY_HEAD_WARPS 8
__global__ void __launch_bounds__(LY_HEAD_WARPS * 32)
k_layers_heads(const float *__restrict__ res, size_t rows, int F, const float *__restrict__ w1x1,
               const float *__restrict__ head, int base, int n, const int *__restrict__ count, float *__restrict__ out)
{
    __shared__ float hp[HEAD_FLOATS];
    __shared__ float w[3 * 256];                 // value conv [F], policy conv [2][F]
    __shared__ float sc[LY_HEAD_WARPS][128];
    if (count) n = min(n, *count - base);
    if (n <= 0 || (int)blockIdx.x * LY_HEAD_WARPS >= n) return;
    for (int i = threadIdx.x; i < HEAD_FLOATS; i += blockDim.x) hp[i] = head[i];
    for (int i = threadIdx.x; i < 3 * F; i += blockDim.x) w[i] = w1x1[i];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float *s = sc[warp];
    for (int b = blockIdx.x * LY_HEAD_WARPS + warp; b < n; b += gridDim.x * LY_HEAD_WARPS) {
        for (int px = lane; px < 42; px += 32) {
            const int r = px / 7, col = px - r * 7;
            const size_t row = LY_GUARD + 56 * (size_t)b + (r + 1) * 8 + (col + 1);
            float v = 0.f, p0 = 0.f, p1 = 0.f;
            for (int c16 = 0; c16 < F / 16; c16++) {
                const float4 *rp = reinterpret_cast<const float4 *>(res + ((size_t)c16 * rows + row) * 16);
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const float4 x = rp[q];
                    const int c = 16 * c16 + 4 * q;
                    v = fmaf(x.x, w[c], v); v = fmaf(x.y, w[c + 1], v); v = fmaf(x.z, w[c + 2], v); v = fmaf(x.w, w[c + 3], v);
                    p0 = fmaf(x.x, w[F + c], p0); p0 = fmaf(x.y, w[F + c + 1], p0);
                    p0 = fmaf(x.z, w[F + c + 2], p0); p0 = fmaf(x.w, w[F + c + 3], p0);
                    p1 = fmaf(x.x, w[2 * F + c], p1); p1 = fmaf(x.y, w[2 * F + c + 1], p1);
                    p1 = fmaf(x.z, w[2 * F + c + 2], p1); p1 = fmaf(x.w, w[2 * F + c + 3], p1);
                }
            }
            s[px] = leaky(v + hp[HO_VB]);
            s[42 + px] = leaky(p0 + hp[HO_PB]);
            s[84 + px] = leaky(p1 + hp[HO_PB + 1]);
        }
        __syncwarp();
        head_tail(s, hp, out + (size_t)(base + b) * 8, lane);
    }
}

// ------------------------------------------------------------------------------------------------ host side
// device image: per layer its weight blocks, then biases [L][F], the head 1x1 convs [3][F] and the head block
static size_t ly_stem_bytes(int F) { return (size_t)9 * F * 32; }
static size_t ly_conv_bytes(int F) { return (size_t)9 * (F / 16) * F * 32; }
static size_t ly_weight_bytes(int F, int R) { return ly_stem_bytes(F) + (size_t)2 * R * ly_conv_bytes(F); }

size_t c4_ly_scratch_bytes(int F, int cap) { return ((size_t)2 * 16 + (size_t)2 * F * 2 + (size_t)F * 4) * ly_rows(cap); }

struct c4_ly_net {
    c4_ly_scratch own;        // scratch of the public c4_net_forward
    std::mutex mu;            // serialises public forwards on the host ...
    cudaEvent_t done;         // ... and orders each after the previous one's use of `own` on the device
};

int c4_ly_scratch_alloc(int F, int cap, c4_ly_scratch *s)
{
    s->F = F; s->cap = cap; s->rows = ly_rows(cap);
    const size_t bytes = c4_ly_scratch_bytes(F, cap);
    if (cudaMalloc(&s->base, bytes) != cudaSuccess) {
        cudaGetLastError();
        s->base = nullptr;
        c4_set_error("cudaMalloc of the layered network's activations failed");
        return -2;
    }
    C4_CUDA(cudaMemset(s->base, 0, bytes));                     // pad rows stay zero for ever
    unsigned char *p = (unsigned char *)s->base;
    s->in = p; p += (size_t)2 * 16 * s->rows;
    s->x = p; p += (size_t)F * 2 * s->rows;
    s->h = p; p += (size_t)F * 2 * s->rows;
    s->res = (float *)p;
    return 0;
}

void c4_ly_scratch_free(c4_ly_scratch *s)
{
    if (s->base) cudaFree(s->base);
    s->base = nullptr;
}

int c4_ly_setup(c4_net *net)
{
    C4_CUDA(cudaFuncSetAttribute(k_layers_conv<OpFP16>, cudaFuncAttributeMaxDynamicSharedMemorySize, LY_MAX_SMEM));
    C4_CUDA(cudaFuncSetAttribute(k_layers_conv<OpBF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, LY_MAX_SMEM));
    c4_ly_net *ly = new c4_ly_net();
    net->ly = ly;
    ly->own.base = nullptr;
    C4_CUDA(cudaEventCreateWithFlags(&ly->done, cudaEventDisableTiming));
    // public forwards work through larger batches in chunks of about 256 MB of activations
    const int per = (int)(c4_ly_scratch_bytes(net->F, 1024) / 1024);
    const int cap = std::max(1024, std::min(16384, (256 << 20) / per)) & ~1023;
    return c4_ly_scratch_alloc(net->F, cap, &ly->own);
}

void c4_ly_destroy(c4_net *net)
{
    if (!net->ly) return;
    c4_ly_scratch_free(&net->ly->own);
    if (net->ly->done) cudaEventDestroy(net->ly->done);
    delete net->ly;
    net->ly = nullptr;
}

int c4_ly_upload(c4_net *net, const float *blob)
{
    const int F = net->F, R = net->R, L = 1 + 2 * R;
    const size_t wb = ly_weight_bytes(F, R);
    std::vector<unsigned char> img(wb + ((size_t)L * F + 3 * F + HEAD_FLOATS) * 4, 0);
    float *bias = reinterpret_cast<float *>(img.data() + wb), *w1x1 = bias + L * F, *hp = w1x1 + 3 * F;
    const float *p = blob + 4;
    for (int l = 0; l < L; l++) {
        const int cin = l == 0 ? 3 : F, cinp = l == 0 ? 16 : F;
        uint16_t *dst = reinterpret_cast<uint16_t *>(img.data() + (l == 0 ? 0 : ly_stem_bytes(F) + (l - 1) * ly_conv_bytes(F)));
        for (int co = 0; co < F; co++)
            for (int ci = 0; ci < cin; ci++)
                for (int ky = 0; ky < 3; ky++)
                    for (int kx = 0; kx < 3; kx++) {
                        // block (tap, 16-channel k-step), inside it [k-chunk][co][8]
                        const size_t blk = (size_t)(ky * 3 + kx) * (cinp / 16) + ci / 16;
                        const size_t idx = ((blk * 2 + (ci % 16) / 8) * F + co) * 8 + ci % 8;
                        dst[idx] = c4_f2op(p[((co * cin + ci) * 3 + ky) * 3 + kx], net->fp16);
                    }
        p += (size_t)F * cin * 9;
        memcpy(bias + l * F, p, F * 4);
        p += F;
    }
    c4_pack_heads(p, F, hp, w1x1, w1x1 + F);
    if (!net->image && cudaMalloc(&net->image, img.size()) != cudaSuccess) { c4_set_error("cudaMalloc failed"); return -2; }
    net->image_bytes = img.size();
    C4_CUDA(cudaMemcpy(net->image, img.data(), img.size(), cudaMemcpyHostToDevice));
    return 0;
}

template <typename OP>
static int ly_chain(const c4_net *net, const u64 *c0, const u64 *c1, int64_t n, const int *count, float *out,
                    cudaStream_t s, int max_ctas, const c4_ly_scratch &scr, unsigned *calib)
{
    const int F = net->F, R = net->R, L = 1 + 2 * R, MT = ly_mt(F), smem = ly_smem(F);
    const unsigned char *img = (const unsigned char *)net->image;
    const float *bias = reinterpret_cast<const float *>(img + ly_weight_bytes(F, R));
    const float *w1x1 = bias + L * F, *hp = w1x1 + 3 * F;
    for (int64_t base = 0; base < n; base += scr.cap) {
        const int nc = (int)std::min<int64_t>(scr.cap, n - base);
        k_layers_input<OP><<<std::min(1024, (nc * 42 + 255) / 256), 256, 0, s>>>(c0, c1, (int)base, nc, count, scr.in,
                                                                                    scr.rows);
        const int groups = ((56 * nc + 127) / 128 + MT - 1) / MT;
        const int grid = std::min(groups, std::max(1, std::min(max_ctas, 148)));
        LyConv a;
        a.bias = bias; a.res = scr.res; a.calib = calib; a.count = count; a.rows = scr.rows;
        a.F = F; a.base = (int)base; a.n = nc;
        for (int l = 0; l < L; l++) {
            a.w = img + (l == 0 ? 0 : ly_stem_bytes(F) + (l - 1) * ly_conv_bytes(F));
            a.bias = bias + l * F;
            a.kind = l == 0 ? 0 : (l & 1) ? 1 : (l == L - 1 ? 3 : 2);
            a.kcin = l == 0 ? 2 : F / 8;
            a.src = l == 0 ? scr.in : (a.kind == 1 ? scr.x : scr.h);
            a.dst = a.kind == 1 ? scr.h : (a.kind == 3 ? nullptr : scr.x);
            k_layers_conv<OP><<<grid, LY_THREADS, smem, s>>>(a);
        }
        k_layers_heads<<<std::min(4 * 148, (nc + LY_HEAD_WARPS - 1) / LY_HEAD_WARPS), LY_HEAD_WARPS * 32, 0, s>>>(
            scr.res, scr.rows, F, w1x1, hp, (int)base, nc, count, out);
    }
    C4_CUDA(cudaGetLastError());
    return 0;
}

int c4_ly_forward(c4_net *net, const uint64_t *c0, const uint64_t *c1, int64_t n, const int32_t *count, float *out,
                  cudaStream_t s, int max_ctas, const c4_ly_scratch *scratch, unsigned *calib)
{
    auto run = [&](const c4_ly_scratch &scr) {
        return net->fp16 ? ly_chain<OpFP16>(net, (const u64 *)c0, (const u64 *)c1, n, count, out, s, max_ctas, scr, calib)
                         : ly_chain<OpBF16>(net, (const u64 *)c0, (const u64 *)c1, n, count, out, s, max_ctas, scr, calib);
    };
    if (scratch) {
        C4_REQUIRE(scratch->base && scratch->F == net->F, "c4_net_forward: no activation scratch for this layered network");
        return run(*scratch);
    }
    c4_ly_net *ly = net->ly;
    std::lock_guard<std::mutex> lock(ly->mu);
    C4_CUDA(cudaStreamWaitEvent(s, ly->done, 0));
    const int rc = run(ly->own);
    C4_CUDA(cudaEventRecord(ly->done, s));
    return rc;
}
