// c4_layers.cuh -- host interface of the layer-by-layer network kernels (c4_layers.cu), used by c4_net.cu and the
// lock-step engine (c4_search.cu).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

struct c4_net;

#define LY_GUARD 16               // zero rows in front of board 0 (a tap reads up to 9 rows back)

// global activations of one forward for up to `cap` positions per launch chain; two forwards in flight at once must
// never share one
struct c4_ly_scratch {
    int F, cap;
    size_t rows;                  // rows of every plane: guard + 56 per position + the last group's window overhang
    unsigned char *in, *x, *h;    // 16-bit operand copies [k-chunk][rows][8]: stem input (2 k-chunks), block input, mid-block
    float *res;                   // fp32 trunk stream [F/16][rows][16]
    void *base;                   // the one allocation behind them (null: none)
};

static inline size_t ly_rows(int cap) { return LY_GUARD + (size_t)56 * cap + 1024; }
size_t c4_ly_scratch_bytes(int F, int cap);
int c4_ly_scratch_alloc(int F, int cap, c4_ly_scratch *s);    // zeroed; 0 or a C4 error code
void c4_ly_scratch_free(c4_ly_scratch *s);

bool c4_net_layered(const c4_net *net);                       // c4_net.cu
int c4_ly_setup(c4_net *net);                                 // kernel attributes + the public forward's scratch
void c4_ly_destroy(c4_net *net);
int c4_ly_upload(c4_net *net, const float *blob);             // (scaled) blob -> device image
// `scratch` null: the network's own scratch, ordered after its previous use.  `calib` non-null: also record the largest
// |activation| bits (range calibration).  No host synchronise and no allocation.
int c4_ly_forward(c4_net *net, const uint64_t *c0, const uint64_t *c1, int64_t n, const int32_t *count, float *out,
                  cudaStream_t s, int max_ctas, const c4_ly_scratch *scratch, unsigned *calib);

// shared with the other network images (c4_net.cu)
uint16_t c4_f2op(float f, bool fp16);
void c4_pack_heads(const float *p, int F, float *hp, float *vw, float *pw);
