// c4_board.cu -- batched bitboard engine kernels + their C-ABI entry points (include/c4b200.h).
// One thread per position, grid-stride, 64-bit coalesced loads; pure integer work, HBM-bound (16-32 B/position).
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "c4_common.cuh"

static thread_local std::string g_err;
void c4_set_error(const std::string &msg) { g_err = msg; }
extern "C" const char *c4_last_error(void) { return g_err.c_str(); }
extern "C" int c4_abi_version(void) { return C4_ABI_VERSION; }
extern "C" int c4_device_count(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { c4_set_error(cudaGetErrorString(e)); return -2; }
    return n;
}

static inline int grid_for(int64_t n, int block)
{
    int64_t g = (n + block - 1) / block;
    const int64_t cap = 148 * 16;             // a few waves on 148 SMs, grid-stride beyond
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}
#define GRID_STRIDE(i, n) \
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (n); i += (int64_t)gridDim.x * blockDim.x)

__global__ void k_legal_mask(const u64 *__restrict__ c0, const u64 *__restrict__ c1, const int8_t *__restrict__ res,
                             uint8_t *__restrict__ mask, int64_t n)
{
    GRID_STRIDE(i, n) {
        int m = c4_legal_mask(c0[i], c1[i]);
        if (res && res[i] != C4_RES_NONE) m = 0;
        mask[i] = (uint8_t)m;
    }
}

__global__ void k_drop(u64 *__restrict__ c0, u64 *__restrict__ c1, const int8_t *__restrict__ move,
                       int8_t *__restrict__ res, int64_t n)
{
    GRID_STRIDE(i, n) {
        int mv = move[i];
        if (mv < 0) continue;
        u64 a = c0[i], b = c1[i];
        int r = c4_drop(a, b, c4_age(a, b), mv);
        c0[i] = a; c1[i] = b;
        if (res) res[i] = (int8_t)r;
    }
}

__global__ void k_has_win(const u64 *__restrict__ bb, uint8_t *__restrict__ out, int64_t n)
{
    GRID_STRIDE(i, n) out[i] = c4_has_win(bb[i]) ? 1 : 0;
}

__global__ void k_result(const u64 *__restrict__ c0, const u64 *__restrict__ c1, int8_t *__restrict__ res, int64_t n)
{
    GRID_STRIDE(i, n) res[i] = (int8_t)c4_result_of(c0[i], c1[i]);
}

__global__ void k_fliplr(const u64 *__restrict__ c0, const u64 *__restrict__ c1, u64 *__restrict__ f0,
                         u64 *__restrict__ f1, int64_t n)
{
    GRID_STRIDE(i, n) { f0[i] = c4_fliplr(c0[i]); f1[i] = c4_fliplr(c1[i]); }
}

// Board.to_array (oinkoink/board.py:147-154).  HBM-write bound (126 plane values out per 16 bytes in).  A block stages
// TP positions in shared memory -- one thread per (position, channel, row) task writes that row's 7 values -- and then
// streams the tile to global memory with 128-bit stores (a tile of TP positions is a multiple of 16 bytes).
#define TP 64
template <typename T> __device__ __forceinline__ T plane_value(unsigned v) { return (T)v; }
template <> __device__ __forceinline__ __half plane_value<__half>(unsigned v) { return __uint2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 plane_value<__nv_bfloat16>(unsigned v) { return __uint2bfloat16_rn(v); }
template <typename T>
__global__ void __launch_bounds__(256) k_to_planes(const u64 *__restrict__ c0, const u64 *__restrict__ c1, T *__restrict__ planes,
                                                  int64_t n)
{
    __shared__ __align__(16) T tile[TP * 126];
    for (int64_t p0 = (int64_t)blockIdx.x * TP; p0 < n; p0 += (int64_t)gridDim.x * TP) {
        const int np = (int)((n - p0 < TP) ? (n - p0) : TP);
        for (int task = threadIdx.x; task < np * 18; task += blockDim.x) {
            const int p = task / 18, cr = task - p * 18, ch = cr / 6, r = cr - ch * 6;
            const u64 a = c0[p0 + p], b = c1[p0 + p];
            T *dst = tile + p * 126 + cr * 7;
            if (ch == 0) {
                const T tm = plane_value<T>((c4_age(a, b) & 1) == 0);
#pragma unroll
                for (int c = 0; c < 7; c++) dst[c] = tm;
            } else {
                const u64 row = ((ch == 1 ? a : b) >> (5 - r));               // column c of this row at bit 7c
#pragma unroll
                for (int c = 0; c < 7; c++) dst[c] = plane_value<T>((unsigned)((row >> (7 * c)) & 1ULL));
            }
        }
        __syncthreads();
        const int nbytes = np * 126 * (int)sizeof(T);
        char *g = reinterpret_cast<char *>(planes + p0 * 126);
        const char *sm = reinterpret_cast<const char *>(tile);
        const int nv = nbytes / 16;
        for (int v = threadIdx.x; v < nv; v += blockDim.x)
            reinterpret_cast<uint4 *>(g)[v] = reinterpret_cast<const uint4 *>(sm)[v];
        for (int t = nv * 16 + threadIdx.x; t < nbytes; t += blockDim.x) g[t] = sm[t];     // tail of the last tile
        __syncthreads();
    }
}

__global__ void k_from_planes(const uint8_t *__restrict__ o, const uint8_t *__restrict__ x, u64 *__restrict__ c0,
                              u64 *__restrict__ c1, int64_t n)
{
    GRID_STRIDE(i, n) {
        u64 a = 0, b = 0;
        for (int r = 0; r < 6; r++)
            for (int c = 0; c < 7; c++) {
                int bit = 7 * c + (5 - r);
                if (o[i * 42 + r * 7 + c]) a |= 1ULL << bit;
                if (x[i * 42 + r * 7 + c]) b |= 1ULL << bit;
            }
        c0[i] = a; c1[i] = b;
    }
}

__global__ void k_evaluate_centre(const u64 *__restrict__ c0, const u64 *__restrict__ c1, double *__restrict__ v,
                                  int64_t n)
{
    GRID_STRIDE(i, n) v[i] = c4_evaluate_centre(c0[i], c1[i]);
}

#define LAUNCH_CHECK() C4_CUDA(cudaGetLastError())

extern "C" int c4_board_legal_mask(const uint64_t *c0, const uint64_t *c1, const int8_t *result, uint8_t *mask,
                                   int64_t n, void *stream)
{
    C4_REQUIRE(n >= 0 && (n == 0 || (c0 && c1 && mask)), "c4_board_legal_mask: null pointer");
    if (n == 0) return 0;
    k_legal_mask<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const u64 *)c0, (const u64 *)c1, result, mask, n);
    LAUNCH_CHECK();
    return 0;
}
extern "C" int c4_board_drop(uint64_t *c0, uint64_t *c1, const int8_t *move, int8_t *result_out, int64_t n,
                             void *stream)
{
    C4_REQUIRE(n >= 0 && (n == 0 || (c0 && c1 && move)), "c4_board_drop: null pointer");
    if (n == 0) return 0;
    k_drop<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((u64 *)c0, (u64 *)c1, move, result_out, n);
    LAUNCH_CHECK();
    return 0;
}
extern "C" int c4_board_has_win(const uint64_t *bb, uint8_t *out, int64_t n, void *stream)
{
    C4_REQUIRE(n >= 0 && (n == 0 || (bb && out)), "c4_board_has_win: null pointer");
    if (n == 0) return 0;
    k_has_win<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const u64 *)bb, out, n);
    LAUNCH_CHECK();
    return 0;
}
extern "C" int c4_board_result(const uint64_t *c0, const uint64_t *c1, int8_t *result_out, int64_t n, void *stream)
{
    C4_REQUIRE(n >= 0 && (n == 0 || (c0 && c1 && result_out)), "c4_board_result: null pointer");
    if (n == 0) return 0;
    k_result<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const u64 *)c0, (const u64 *)c1, result_out, n);
    LAUNCH_CHECK();
    return 0;
}
extern "C" int c4_board_fliplr(const uint64_t *c0, const uint64_t *c1, uint64_t *f0, uint64_t *f1, int64_t n,
                               void *stream)
{
    C4_REQUIRE(n >= 0 && (n == 0 || (c0 && c1 && f0 && f1)), "c4_board_fliplr: null pointer");
    if (n == 0) return 0;
    k_fliplr<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const u64 *)c0, (const u64 *)c1, (u64 *)f0,
                                                                 (u64 *)f1, n);
    LAUNCH_CHECK();
    return 0;
}
extern "C" int c4_board_to_planes(const uint64_t *c0, const uint64_t *c1, void *planes, int dtype, int64_t n,
                                  void *stream)
{
    C4_REQUIRE(n >= 0 && (n == 0 || (c0 && c1 && planes)), "c4_board_to_planes: null pointer");
    C4_REQUIRE(dtype >= 0 && dtype <= 3, "c4_board_to_planes: dtype must be 0 (uint8), 1 (float32), 2 (float16) or 3 (bfloat16)");
    if (n == 0) return 0;
    C4_REQUIRE(((uintptr_t)planes & 15) == 0, "c4_board_to_planes: planes must be 16-byte aligned");
    const int64_t tiles = (n + TP - 1) / TP;
    const int blocks = (int)(tiles < 148 * 8 ? tiles : 148 * 8);
    const cudaStream_t s = (cudaStream_t)stream;
    if (dtype == 0)
        k_to_planes<uint8_t><<<blocks, 256, 0, s>>>((const u64 *)c0, (const u64 *)c1, (uint8_t *)planes, n);
    else if (dtype == 1)
        k_to_planes<float><<<blocks, 256, 0, s>>>((const u64 *)c0, (const u64 *)c1, (float *)planes, n);
    else if (dtype == 2)
        k_to_planes<__half><<<blocks, 256, 0, s>>>((const u64 *)c0, (const u64 *)c1, (__half *)planes, n);
    else
        k_to_planes<__nv_bfloat16><<<blocks, 256, 0, s>>>((const u64 *)c0, (const u64 *)c1, (__nv_bfloat16 *)planes, n);
    LAUNCH_CHECK();
    return 0;
}
extern "C" int c4_board_from_planes(const uint8_t *o, const uint8_t *x, uint64_t *c0, uint64_t *c1, int64_t n,
                                    void *stream)
{
    C4_REQUIRE(n >= 0 && (n == 0 || (o && x && c0 && c1)), "c4_board_from_planes: null pointer");
    if (n == 0) return 0;
    k_from_planes<<<grid_for(n, 128), 128, 0, (cudaStream_t)stream>>>(o, x, (u64 *)c0, (u64 *)c1, n);
    LAUNCH_CHECK();
    return 0;
}
extern "C" int c4_board_evaluate_centre(const uint64_t *c0, const uint64_t *c1, double *value, int64_t n, void *stream)
{
    C4_REQUIRE(n >= 0 && (n == 0 || (c0 && c1 && value)), "c4_board_evaluate_centre: null pointer");
    if (n == 0) return 0;
    k_evaluate_centre<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>((const u64 *)c0, (const u64 *)c1, value, n);
    LAUNCH_CHECK();
    return 0;
}
