// c4_fused.cu -- the fused persistent self-play engine: ONE launch plays a whole generation.
//
// What it replaces: the reference's free-running runtime -- game threads that never wait for an unrelated game
// (oinkoink/neural/game_pool.py:15-49) and an inference server that batches whatever requests are there
// (oinkoink/neural/inference_server.py:37-63) -- and this package's own first engine, the lock-step pass
// (c4_search.cu: one tree launch + one network launch per pass, a pool-wide barrier between them).
//
// Design (SURVEY.md section 7, "persistent CTA-per-game-group megakernel ... no grid-wide sync"):
//   * one persistent CTA per SM (1024 threads), each OWNING a contiguous group of game slots for the whole launch;
//     CTAs never talk to each other (the evaluation memo and the generation counters in HBM are the only shared
//     state, both lock-free), so there is no cooperative launch, no grid barrier and no cross-SM spin.
//   * warps 18..31 = TREE warps.  A tree warp picks any runnable game of the CTA (status word in shared memory, CAS),
//     consumes its evaluator answer if one is waiting, and runs select / expand / backup (c4_tree.cuh -- the same device
//     functions as the lock-step pass, hence bit-identical trees) until the game needs an evaluation that is not in the
//     memo.  It then pushes {c0, c1, game} into the CTA's leaf ring in shared memory and picks the NEXT runnable game:
//     a game that waits for the network never holds a warp, and no game ever waits for an unrelated game.
//   * warps 0..17 = the tcgen05 / TMEM network tower of c4_tc.cuh, running on THIS SM for THIS CTA's leaves: warp 0
//     streams the layer weights L2 -> shared memory (cp.async.bulk ring), warp 1 issues the tcgen05.mma chain, warps 2..17
//     are the epilogue.  Epilogue warp 0 is also the dispatcher: whenever the tower is idle it takes up to 16 published
//     leaves from the ring (no batching delay: when the network is the bottleneck the ring is full by the time a strip
//     ends, when it is not, latency matters more than strip fill) and the strip's answers go straight to shared memory,
//     where they flip the games' status words to ANSWERED.
//   * the PUCT tables (log / sqrt / reciprocal, 19 KB at 800 simulations) are staged in shared memory; the network
//     needs 200 KB, which leaves only ~28 KB of L1 for the node records (DESIGN.md discusses the trade).
// Every inter-warp hand-off is CTA-local (shared-memory words + mbarriers), bounded by a watchdog that makes the call
// fail with an error code instead of hanging the device.
//
// Lock-free hand-offs, all inside one CTA (what a race checker would flag, and why each is safe):
//   * status[gl]: claimed by a tree warp with atomicCAS (READY / ANSWERED / NEWROOT -> RUNNING); written back by the
//     owner only (RUNNING -> WAIT / READY / IDLE / DONE) after a __threadfence_block(); flipped WAIT -> ANSWERED by the one
//     epilogue warp that holds the game's board, after the answer is in ans[gl] and a fence.  WAIT is published BEFORE the
//     leaf enters the ring, so an answer can never be overwritten by a late WAIT.
//   * leaf ring: slot reserved with atomicAdd(q_tail); entry written; fence; q_seq[idx] = slot + 1.  The dispatcher reads
//     q_seq with volatile loads and takes only the leading run of complete entries.  Capacity >= games per CTA and a game has
//     at most one leaf pending, so a slot is never reused before it was consumed (C4_DEV_ASSERT in fz_run_game).
//   * strip_*: written by the dispatcher before the epilogue warps' named barrier, read after it; each warp copies the game
//     of its board into a register at once, because the dispatcher refills strip_game for the next strip while other warps
//     are still in their head tails.
//   * stop / quit / abort: monotone 0 -> 1 flags, volatile stores and loads; seeing one late costs one more simulation or
//     poll, never a result.
//   * the evaluation memo in HBM is shared by all CTAs: see memo_insert in c4_tree.cuh (checksummed entries).
//
// Not in this engine: the de-duplication of evaluations in flight (PENDING tags in the memo, c4_tree.cuh) that the lock-step
// engine uses.  It was built here too (a parked game re-probes the memo with exponential back-off) and removed 27 % of the
// network evaluations of the benchmark generation, but the re-probing tree warps slowed the tower on the same SM by more
// than the saved evaluations were worth (252k vs 265k positions/s in the same build, profiles/README.md); a PENDING tag
// written by the other engine simply reads as a miss here.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <thread>

#include "c4_fz.cuh"

// Strip geometry of the tower inside the fused engine (c4_tc.cuh: TcC<32> is the batch kernel's).  The engine is bound by
// the tree warps, not by the tower (profiles/README.md), so the tower is kept small: strips of FZ_NB boards, FZ_GROUPS
// epilogue groups of 8 warps -- every warp and every KB of shared memory it does not take goes to the tree (warps that run
// games, L1 for the node records).
#ifndef FZ_NB
#define FZ_NB 9
#endif
#ifndef FZ_GROUPS
#define FZ_GROUPS 1
#endif
struct TcFz {
    static constexpr int F = 32, NB = FZ_NB, T = (7 * FZ_NB + 15) / 16, ROWS = 128 * T + 16, WSTAGES = 3, ACC_SLOTS = 3,
                         GROUPS = FZ_GROUPS, EPI_WARPS = 8 * FZ_GROUPS;
    static constexpr bool SLICED = false;
};
typedef TcKc<TcFz> FzK32;
// 64 filters (the reference's example_config network): the batch kernel's geometry as it is -- 6-board strips, one
// 72 KB weight stage refilled slice by slice, 16 epilogue warps (4 lane quadrants x 4 channel slices)
typedef TcKc<TcC<64>> FzK64;

#define FZ_THREADS 1024
// Warp ids = issue priority (the SM's arbiter prefers HIGH warp ids): the single-thread issuer and producer on top; then
// the tree warps (their simulations are dependent chains -- every lost issue slot is latency of a game) and the epilogue
// warps at the bottom (FZ_TREE_HIGH), or the other way round.
#ifndef FZ_TREE_HIGH
#define FZ_TREE_HIGH 1
#endif
template <class K> struct FzW {
    static constexpr int EPI_WARPS = K::EPI_WARPS;
    static constexpr int TREE_WARPS = FZ_THREADS / 32 - 2 - EPI_WARPS;
    static constexpr int EPI_WARP0 = FZ_TREE_HIGH ? 0 : TREE_WARPS;
    static constexpr int TREE_WARP0 = FZ_TREE_HIGH ? EPI_WARPS : 0;
    static constexpr int PRODUCER = FZ_THREADS / 32 - 2, ISSUER = FZ_THREADS / 32 - 1;
    static constexpr int BOARDS_PER_WARP = (K::NB + EPI_WARPS - 1) / EPI_WARPS;
};
#define FZ_EPI_BAR() asm volatile("bar.sync 1, %0;\n" :: "n"(32 * W::EPI_WARPS) : "memory")
#define FZ_GC_MAX 128                                     // game slots per CTA
#define FZ_QCAP 128                                       // leaf ring entries (>= FZ_GC_MAX: one pending leaf per game)

struct FzParams {
    int n_slots;                        // game slots of the pool
    int table_entries;                  // entries of each PUCT table staged in shared memory (0: read them from HBM)
    unsigned long long stop_games;      // leave once ctr->games_finished reaches this (0 = never)
    unsigned long long stop_ns;         // leave after this much run time (0 = never)
    const int *host_abort;              // mapped host word: non-zero = the host gave up waiting, leave at once
    int *dbg;                           // [CTA][32 warps] last checkpoint of every warp (host-side hang diagnosis), or null
    unsigned long long *prof;           // [16] cycle / event sums of CTA 0 (C4_FZ_DEBUG), or null
    int tree_warps;                     // tree warps that work (tuning knob C4_FZ_TREE_WARPS)
};

struct FzCtl {
    unsigned q_tail, q_head;            // leaf ring: requests reserved / consumed
    int quit, abort, stop, tree_exited;
    int strip_nb;
    int wake;                           // bumped whenever a game becomes runnable or a flag changes: idle tree warps poll this one word
    int strip_game[16];
    u64 strip_c0[16], strip_c1[16];
    unsigned q_seq[FZ_QCAP];            // slot number + 1 once the entry is complete
    int q_game[FZ_QCAP];
    u64 q_c0[FZ_QCAP], q_c1[FZ_QCAP];
    int status[FZ_GC_MAX];              // ST_* / FZ_*: authoritative while the kernel runs
    float ans[FZ_GC_MAX][8];            // evaluator answers {prior[7], value} of ANSWERED games
    long long t_push[FZ_GC_MAX], t_ans[FZ_GC_MAX];   // clock64 stamps of the last request / answer of a game (profiling)
};

#define FZ_PROF(i, v) do { if (P.prof && blockIdx.x == 0 && lane == 0) atomicAdd(&P.prof[i], (unsigned long long)(v)); } while (0)
#define FZ_DBG(code) do { if (P.dbg && lane == 0) *reinterpret_cast<volatile int *>(&P.dbg[blockIdx.x * 32 + warp]) = (code); } while (0)

template <class K> __host__ __device__ constexpr int fz_ctl_off(int R) { return (K::total(R) + 15) & ~15; }
template <class K> __host__ __device__ constexpr int fz_tab_off(int R) { return (fz_ctl_off<K>(R) + (int)sizeof(FzCtl) + 15) & ~15; }
template <class K> __host__ __device__ constexpr int fz_total(int R, int table_entries) { return fz_tab_off<K>(R) + 3 * 8 * table_entries; }

// the fused engine's port: answers and the leaf ring live in the CTA's shared memory
struct FzPort {
    static constexpr int GC_MAX = FZ_GC_MAX;
    static constexpr bool DEDUP = false;                                  // measured slower in this engine (header comment)
    typedef Game GameType;
    FzCtl *S;
    __device__ __forceinline__ void stage(Game &, int) const {}
    __device__ __forceinline__ bool impatient(int) const { return true; }
    __device__ __forceinline__ int stopping() const { return ld_vol(&S->stop); }
    __device__ __forceinline__ float answer(int, int gl, int lane) const { return (lane < 8) ? S->ans[gl][lane] : 0.f; }
    __device__ __forceinline__ void publish(int, int gl, int st, bool request, u64 rc0, u64 rc1) const
    {
        __threadfence_block();
        st_vol(&S->status[gl], st);                                       // WAIT must be visible before the request is
        if (st == ST_IDLE || st == ST_DONE) atomicAdd(&S->wake, 1);       // idle warps re-check whether anything is left
        if (request) {
            S->t_push[gl] = clock64();
            const unsigned slot = atomicAdd(&S->q_tail, 1u);
            const unsigned idx = slot % FZ_QCAP;
            C4_DEV_ASSERT(slot - *reinterpret_cast<volatile unsigned *>(&S->q_head) < FZ_QCAP);   // one pending leaf per game
            S->q_c0[idx] = rc0; S->q_c1[idx] = rc1; S->q_game[idx] = gl;
            __threadfence_block();
            *reinterpret_cast<volatile unsigned *>(&S->q_seq[idx]) = slot + 1u;
        }
    }
};

template <typename OP, class K, bool SELFPLAY>
__global__ void __launch_bounds__(FZ_THREADS, 1)
k_fused(const C4Dev dg, const unsigned char *__restrict__ image, int R, FzParams P)
{
    using W = FzW<K>;
    constexpr int F = K::F;
    extern __shared__ __align__(16) unsigned char smem[];
    const int L = 1 + 2 * R;
    const int warp = __shfl_sync(FULL, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    // this CTA's game slots
    const int per = P.n_slots / (int)gridDim.x, extra = P.n_slots % (int)gridDim.x;
    const int Gc = per + ((int)blockIdx.x < extra ? 1 : 0);
    const int g0 = (int)blockIdx.x * per + min((int)blockIdx.x, extra);

    unsigned char *sX = smem + K::X, *sH = smem + K::H, *sW = smem + K::W;
    float *small = reinterpret_cast<float *>(smem + K::SMALL);
    const float *bias = small, *hp = small + L * F;
    float *scratch = reinterpret_cast<float *>(smem + K::scratch(R));
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + K::bars(R));
    const uint32_t b_wfull = smem_u32(bars), b_wempty = b_wfull + 8 * K::WBARS;
    const uint32_t b_accfull = b_wempty + 8 * K::WBARS, b_accempty = b_accfull + 8 * K::ACC_SLOTS;
    const uint32_t b_epi = b_accempty + 8 * K::ACC_SLOTS;                   // T barriers
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * K::WBARS + 2 * K::ACC_SLOTS + K::T);
    FzCtl *S = reinterpret_cast<FzCtl *>(smem + fz_ctl_off<K>(R));
    double *tab = reinterpret_cast<double *>(smem + fz_tab_off<K>(R));

    // ---- one-time setup
    for (int i = threadIdx.x; i < 2 * K::ACT_BYTES / 16; i += blockDim.x)
        reinterpret_cast<uint4 *>(sX)[i] = make_uint4(0u, 0u, 0u, 0u);
    {
        const unsigned char *src = image + (size_t)L * K::WSTAGE_BYTES;
        const int nb16 = (L * F + HEAD_FLOATS) * 4 / 16;
        for (int i = threadIdx.x; i < nb16; i += blockDim.x)
            reinterpret_cast<uint4 *>(small)[i] = reinterpret_cast<const uint4 *>(src)[i];
    }
    for (int i = threadIdx.x; i < (int)(sizeof(FzCtl) / 4); i += blockDim.x) reinterpret_cast<uint32_t *>(S)[i] = 0u;
    for (int i = threadIdx.x; i < P.table_entries; i += blockDim.x) {
        tab[i] = dg.pbc[i]; tab[P.table_entries + i] = dg.sqt[i]; tab[2 * P.table_entries + i] = dg.rcp[i];
    }
    if (threadIdx.x == 0) {
        for (int i = 0; i < K::WBARS; i++) { mbar_init(b_wfull + 8 * i, 1); mbar_init(b_wempty + 8 * i, 1); }
        for (int i = 0; i < K::ACC_SLOTS; i++) { mbar_init(b_accfull + 8 * i, 1); mbar_init(b_accempty + 8 * i, K::GROUP_WARPS); }
        for (int i = 0; i < K::T; i++) mbar_init(b_epi + 8 * i, K::GROUP_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == W::PRODUCER) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;\n" :: "r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    __syncthreads();                                                      // FzCtl zeroed before the statuses go in
    for (int i = threadIdx.x; i < FZ_GC_MAX; i += blockDim.x) S->status[i] = (i < Gc) ? fz_entry_status(dg, g0 + i) : (int)ST_IDLE;
    TC_PROXY_FENCE();
    TC_FENCE_BEFORE();
    __syncthreads();
    TC_FENCE_AFTER();
    const uint32_t tmem = *tmem_slot;
    const unsigned long long t_begin = fz_globaltimer();

    if (warp == W::PRODUCER) {
        // ================= weight producer: layer g of the endless (strip, layer) sequence -> ring stage g % WSTAGES.
        // It runs up to WSTAGES layers ahead of the issuer, i.e. the first layers of the NEXT strip are already on chip
        // while the tower idles.
        if (lane == 0 && K::SLICED) {
            // one weight stage, refilled one dy slice at a time: slice dy of layer g is requested as soon as the issuer has
            // released slice dy of layer g - 1 (c4_net.cu)
            int g = 0, last[3] = {-1, -1, -1};
            bool live = true;
            for (; live; g++) {
                FZ_DBG(0x100000 | g);
                for (int dy = 0; dy < 3 && live; dy++) {
                    if (g > 0) {
                        const uint32_t bar = b_wempty + 8 * dy, par = (uint32_t)(g - 1) & 1u;
                        for (uint32_t it = 0; !mbar_try(bar, par); it++) {
                            if (it > 4u) __nanosleep(it > 64u ? 500 : 100);
                            if ((it & 15u) == 15u && (ld_vol(&S->quit) || ld_vol(&S->abort))) { live = false; break; }
                        }
                        if (!live) break;
                    }
                    mbar_expect_tx(b_wfull + 8 * dy, K::WSLICE_BYTES);
                    bulk_g2s(smem_u32(sW + dy * K::WSLICE_BYTES), image + (size_t)(g % L) * K::WSTAGE_BYTES + dy * K::WSLICE_BYTES,
                             K::WSLICE_BYTES, b_wfull + 8 * dy);
                    last[dy] = g;
                }
            }
            FZ_DBG(0x1f0000 | g);
            for (int dy = 0; dy < 3; dy++)                                        // no bulk copy in flight at exit
                if (last[dy] >= 0) mbar_wait(b_wfull + 8 * dy, (uint32_t)last[dy] & 1u);
            FZ_DBG(0x1ff000);
        } else if (lane == 0) {
            int g = 0;
            bool live = true;
            for (; live; g++) {
                const int st = g % K::WSTAGES, use = g / K::WSTAGES;
                FZ_DBG(0x100000 | g);
                if (use > 0) {
                    const uint32_t bar = b_wempty + 8 * st, par = (uint32_t)(use - 1) & 1u;
                    for (uint32_t it = 0; !mbar_try(bar, par); it++) {
                        if (it > 4u) __nanosleep(it > 64u ? 500 : 100);
                        if ((it & 15u) == 15u && (ld_vol(&S->quit) || ld_vol(&S->abort))) { live = false; break; }
                    }
                    if (!live) break;
                }
                mbar_expect_tx(b_wfull + 8 * st, K::WSTAGE_BYTES);
                bulk_g2s(smem_u32(sW + st * K::WSTAGE_BYTES), image + (size_t)(g % L) * K::WSTAGE_BYTES, K::WSTAGE_BYTES,
                         b_wfull + 8 * st);
            }
            FZ_DBG(0x1f0000 | g);
            // no bulk copy may be in flight when the CTA exits: wait for the stages requested last
            for (int i = max(0, g - K::WSTAGES); i < g; i++) mbar_wait(b_wfull + 8 * (i % K::WSTAGES), (uint32_t)(i / K::WSTAGES) & 1u);
            FZ_DBG(0x1ff000);
        }
    } else if (warp == W::ISSUER) {
        // ================= MMA issuer (one thread): the strip loop of k_net_tc with strips that arrive at run time
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | ((uint32_t)OP::FMT << 7) | ((uint32_t)OP::FMT << 10) |
                                   ((uint32_t)(K::NN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
            int g = 0, c = 0;                                   // (strip, layer) counter, (strip, layer, tile) counter
            bool live = true;
            for (int s = 0; live; s++) {
                FZ_DBG(0x200000 | (s & 0xffff));
                // every strip completes L + 1 phases on EVERY tile barrier (input planes + L epilogues)
                if (!fz_wait(b_epi, (uint32_t)(s * (L + 1)) & 1u, &S->abort)) break;
                const int nb = ld_vol(&S->strip_nb);
                if (nb == 0) break;                                             // the dispatcher said quit
                const int T = (7 * nb + 15) / 16;
                for (int l = 0; l < L && live; l++, g++) {
                    const int st = g % K::WSTAGES;
                    FZ_DBG(0x210000 | ((s & 0xff) << 8) | l);
                    if (!K::SLICED && !fz_wait(b_wfull + 8 * st, (uint32_t)(g / K::WSTAGES) & 1u, &S->abort)) { live = false; break; }
                    const uint32_t wbase = smem_u32(sW + st * K::WSTAGE_BYTES);
                    const uint32_t abase = smem_u32((l == 0 || (l & 1) == 0) ? sH : sX);   // stem and conv2 read H
                    const uint64_t a_l = umma_desc(abase, K::ROWS * 16, 128);
                    const uint64_t b_l = umma_desc(wbase, K::NN * 16, 128);
                    const uint32_t ep_par = (uint32_t)(s * (L + 1) + l) & 1u;
#pragma unroll
                    for (int t = 0; t < K::T; t++, c++) {
                        if (t >= T) break;
                        if (t == 0 && !fz_wait(b_epi, ep_par, &S->abort)) { live = false; break; }
                        if (t + 1 < T && !fz_wait(b_epi + 8 * (t + 1), ep_par, &S->abort)) { live = false; break; }
                        const int slot = c % K::ACC_SLOTS, use = c / K::ACC_SLOTS;
                        if (use > 0 && !fz_wait(b_accempty + 8 * slot, (uint32_t)(use - 1) & 1u, &S->abort)) { live = false; break; }
                        TC_FENCE_AFTER();
                        const uint32_t dcol = tmem + K::ACC_COL0 + slot * K::NN;
                        const uint64_t a = a_l + (uint64_t)(128 * t);
                        if (l != 0) {
#pragma unroll
                            for (int dy = 0; dy < 3; dy++) {
                                if (K::SLICED && t == 0 && !fz_wait(b_wfull + 8 * dy, (uint32_t)g & 1u, &S->abort)) { live = false; break; }
#pragma unroll
                                for (int ks = 0; ks < K::KC / 2; ks++) {
                                    const uint64_t aa = a + 8 * dy + 2 * K::ROWS * ks, bb = b_l + (dy * K::KC + 2 * ks) * K::NN;
                                    if (dy == 0 && ks == 0) umma_f16c<0>(dcol, aa, bb, idesc); else umma_f16c<1>(dcol, aa, bb, idesc);
                                }
                                if (K::SLICED && t == T - 1) umma_commit(b_wempty + 8 * dy);  // slice free for the next layer
                            }
                        } else {                                              // stem: 16 (padded) input channels = one k-step
#pragma unroll
                            for (int dy = 0; dy < 3; dy++) {
                                if (K::SLICED && t == 0 && !fz_wait(b_wfull + 8 * dy, (uint32_t)g & 1u, &S->abort)) { live = false; break; }
                                const uint64_t aa = a + 8 * dy, bb = b_l + dy * K::STEM_KC * K::NN;
                                if (dy == 0) umma_f16c<0>(dcol, aa, bb, idesc); else umma_f16c<1>(dcol, aa, bb, idesc);
                                if (K::SLICED && t == T - 1) umma_commit(b_wempty + 8 * dy);
                            }
                        }
                        if (!live) break;
                        umma_commit(b_accfull + 8 * slot);
                    }
                    if (live && !K::SLICED) umma_commit(b_wempty + 8 * st);
                }
                // observe the LAST epilogue phase of tile 0 too: a parity wait only tells "not the phase in progress", so
                // with a one-tile strip the wait for the next strip's input phase (same parity as this strip's phase L - 1)
                // would fall through while phase L is still in progress
                if (live && !fz_wait(b_epi, (uint32_t)(s * (L + 1) + L) & 1u, &S->abort)) break;
            }
            FZ_DBG(0x2ff000);
        }
    } else if (warp >= W::EPI_WARP0 && warp < W::EPI_WARP0 + W::EPI_WARPS) {
        // ================= epilogue warps (+ the dispatcher in the first of them)
        const int e = warp - W::EPI_WARP0, quad = warp & 3, half = (e >> 2) % K::SLICES, group = e / K::GROUP_WARPS;
        const int et = threadIdx.x - 32 * W::EPI_WARP0;                      // 0..511
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
        int c = 0;                                                           // global (strip, layer, tile) counter
        for (;;) {
            FZ_DBG(0x300000 | (c & 0xffff));
            const long long t_d0 = clock64();
            // ---- dispatch: take what the leaf ring holds (up to one strip)
            if (e == 0) {
                const unsigned head = S->q_head;                             // written by this warp only
                if (lane == 0 && !ld_vol(&S->stop)) {
                    if (P.stop_games && __ldcg(&dg.ctr->games_finished) >= P.stop_games) { st_vol(&S->stop, 1); atomicAdd(&S->wake, 1); }
                    if (P.stop_ns && fz_globaltimer() - t_begin > P.stop_ns) { st_vol(&S->stop, 1); atomicAdd(&S->wake, 1); }
                }
                int k = 0;
                for (uint32_t it = 1;; it++) {
                    if (*reinterpret_cast<volatile unsigned *>(&S->q_tail) == head) {     // nothing requested: one word read
                        if (ld_vol(&S->quit) | ld_vol(&S->abort)) break;
                        if ((it & 1023u) == 0u && lane == 0 && *reinterpret_cast<const volatile int *>(P.host_abort)) { st_vol(&S->abort, 1); atomicAdd(&S->wake, 1); }
                        if ((it & 31u) == 0u && lane == 0 && !ld_vol(&S->stop)) {
                            if (P.stop_games && __ldcg(&dg.ctr->games_finished) >= P.stop_games) { st_vol(&S->stop, 1); atomicAdd(&S->wake, 1); }
                            if (P.stop_ns && fz_globaltimer() - t_begin > P.stop_ns) { st_vol(&S->stop, 1); atomicAdd(&S->wake, 1); }
                        }
                        __nanosleep(it > 32u ? 400 : 100);
                        continue;
                    }
                    const bool ok = lane < K::NB &&
                        *reinterpret_cast<volatile unsigned *>(&S->q_seq[(head + lane) % FZ_QCAP]) == head + (unsigned)lane + 1u;
                    const unsigned m = __ballot_sync(FULL, ok);
                    k = __ffs((int)~m) - 1;                                  // leading complete entries (m only has bits < NB)
                    if (k > 0) break;
                    if (__any_sync(FULL, ld_vol(&S->quit) | ld_vol(&S->abort))) break;
                    __nanosleep(50);                                         // an entry is reserved but not complete yet
                }
                __threadfence_block();
                if (lane < k) {
                    const unsigned idx = (head + lane) % FZ_QCAP;
                    S->strip_game[lane] = S->q_game[idx]; S->strip_c0[lane] = S->q_c0[idx]; S->strip_c1[lane] = S->q_c1[idx];
                }
                if (lane == 0) { S->strip_nb = k; S->q_head = head + (unsigned)k; }
            }
            FZ_EPI_BAR();
            const int nb = ld_vol(&S->strip_nb);
            // (one board per epilogue warp at most: the dispatcher overwrites strip_game for the next strip while other
            //  warps are still in their head tails, so the game of THIS warp's board is read now)
            int my_gl[W::BOARDS_PER_WARP];
#pragma unroll
            for (int i = 0; i < W::BOARDS_PER_WARP; i++) my_gl[i] = S->strip_game[(e + i * W::EPI_WARPS) & 15];
            const long long t_d1 = clock64();
            FZ_DBG(0x310000 | nb);
            if (nb == 0) {                                                   // quit: wake the issuer so it reads strip_nb == 0
                if (lane == 0 && e < K::GROUP_WARPS)
                    for (int t = 0; t < K::T; t++) mbar_arrive(b_epi + 8 * t);
                break;
            }
            const int T = (7 * nb + 15) / 16;
            E.valid_mask = 0;
            for (int t = 0; t < T; t++) {
                const int rb = 16 * t + E.rb0, b = rb / 7;
                if (E.col8 != 0 && rb - 7 * b != 0 && b < nb) E.valid_mask |= 1u << t;
            }
            // ---- input planes (Board.to_array) -> channels 0..15 of H
            for (int i = et; i < nb * 42; i += 32 * W::EPI_WARPS) {
                const int b = i / 42, px = i - b * 42, r = px / 7, col = px - r * 7;
                const u64 a0 = S->strip_c0[b], a1 = S->strip_c1[b];
                const int bit = 7 * col + (5 - r);
                const uint32_t tomove = ((__popcll(a0 | a1) & 1) == 0) ? OP::ONE : 0u;
                const uint32_t o = (uint32_t)((a0 >> bit) & 1ULL) * OP::ONE, x = (uint32_t)((a1 >> bit) & 1ULL) * OP::ONE;
                const int row = 8 + (7 * b + 1 + r) * 8 + (col + 1);
                *reinterpret_cast<uint4 *>(sH + (size_t)row * 16) = make_uint4(tomove | (o << 16), x, 0u, 0u);
                *reinterpret_cast<uint4 *>(sH + (size_t)(K::ROWS + row) * 16) = make_uint4(0u, 0u, 0u, 0u);
            }
            TC_PROXY_FENCE();
            FZ_EPI_BAR();
            const long long t_d2 = clock64();
            // every phase completes on ALL tile barriers (also those of tiles this strip does not have), so that the
            // phase parity of a tile barrier is a function of (strip, layer) only
            if (lane == 0 && e < K::GROUP_WARPS)
                for (int t = 0; t < K::T; t++) mbar_arrive(b_epi + 8 * t);
#define FZ_SKIPPED_TILES() if (lane == 0 && e < K::GROUP_WARPS) for (int t = T; t < K::T; t++) mbar_arrive(b_epi + 8 * t)
            tc_epilogue_layer8<OP, K, 0>(E, 0, T, c); c += T; FZ_SKIPPED_TILES();
            for (int l = 1; l < L - 1; l += 2) {
                tc_epilogue_layer8<OP, K, 1>(E, l, T, c); c += T; FZ_SKIPPED_TILES();
                if (l + 1 < L - 1) { tc_epilogue_layer8<OP, K, 2>(E, l + 1, T, c); c += T; FZ_SKIPPED_TILES(); }
            }
            tc_epilogue_layer8<OP, K, 3>(E, L - 1, T, c); c += T; FZ_SKIPPED_TILES();
#undef FZ_SKIPPED_TILES

            // ---- head tails: one warp per board; the answer goes to the game's slot and flips its status word
            FZ_DBG(0x320000 | nb);
            FZ_EPI_BAR();
            const long long t_d3 = clock64();
#pragma unroll
            for (int bi = 0; bi < W::BOARDS_PER_WARP; bi++) {
                const int b = e + bi * W::EPI_WARPS;
                if (b >= nb) break;
                float *sc = scratch + b * 128;
                for (int i = lane; i < 126; i += 32) {
                    float bb = i < 42 ? hp[HO_VB] : (i < 84 ? hp[HO_PB] : hp[HO_PB + 1]);
                    float acc = sc[i];                                       // channel slices summed in a fixed order
#pragma unroll
                    for (int q = 1; q < K::SLICES; q++) acc += sc[q * K::NB * 128 + i];
                    sc[i] = leaky(acc + bb);
                }
                __syncwarp();
                const int gl = my_gl[bi];
                C4_DEV_ASSERT(gl >= 0 && gl < Gc && ld_vol(&S->status[gl]) == ST_WAIT);
                float *ans = S->ans[gl];
                head_tail(sc, hp, ans, lane);
                const float o = (lane < 8) ? ans[lane] : 0.f;
                if (__any_sync(FULL, !isfinite(o))) {
                    // operand overflow (fp16) or NaN weights: never into the tree -- neutral answer + a flag that makes the
                    // host call fail (the reference asserts, oinkoink/neural/pytorch/model.py:258-263,275-280)
                    if (lane < 8) ans[lane] = (lane < 7) ? (1.f / 7.f) : 0.5f;
                    if (lane == 0) dg.ctr->net_nonfinite = 1;
                }
                __syncwarp();
                if (lane == 0) { S->t_ans[gl] = clock64(); __threadfence_block(); st_vol(&S->status[gl], FZ_ANSWERED); atomicAdd(&S->wake, 1); }
            }
            if (e == 0) {
                FZ_PROF(0, 1); FZ_PROF(1, nb); FZ_PROF(2, t_d1 - t_d0); FZ_PROF(3, t_d2 - t_d1); FZ_PROF(4, t_d3 - t_d2);
                FZ_PROF(5, clock64() - t_d3);
            }
        }
    } else {
        // ================= tree warps
        C4Dev d = dg;
        if (P.table_entries) { d.pbc = tab; d.sqt = tab + P.table_entries; d.rcp = tab + 2 * P.table_entries; }
        const int tw = warp - W::TREE_WARP0;
        int rot = (tw * 9) % Gc;
        bool idle = false;
        long long idle_t0 = 0;
        uint32_t idle_it = 0;
        for (; tw < P.tree_warps;) {
            const int seen = ld_vol(&S->wake);                             // read BEFORE the scan: no wake-up is lost
            const int aborting = ld_vol(&S->abort);
            const int stop = ld_vol(&S->stop) | aborting;
            FZ_DBG(0x400000);
            int cand = -1, n_wait = 0, n_ans = 0, n_ready = 0;
            bool cand_ans = false;
            for (int base = 0; base < Gc; base += 32) {
                const int i = base + lane;
                int idx = i + rot;
                if (idx >= Gc) idx -= Gc;
                const int s = (i < Gc) ? ld_vol(&S->status[idx]) : ST_IDLE;
                const unsigned ma = __ballot_sync(FULL, s == FZ_ANSWERED);
                const unsigned mr = __ballot_sync(FULL, s == ST_READY || s == ST_NEWROOT);
                const unsigned mw = __ballot_sync(FULL, s == ST_WAIT);
                n_wait += __popc(mw); n_ans += __popc(ma); n_ready += __popc(mr);
                if (ma && !cand_ans) { cand = __shfl_sync(FULL, idx, __ffs((int)ma) - 1); cand_ans = true; }
                else if (mr && cand < 0 && !stop) cand = __shfl_sync(FULL, idx, __ffs((int)mr) - 1);
            }
            if (aborting) break;
            if (cand >= 0) {
                int s = 0, ok = 0;
                if (lane == 0) {
                    s = ld_vol(&S->status[cand]);
                    if (s == FZ_ANSWERED || (!stop && (s == ST_READY || s == ST_NEWROOT)))
                        ok = atomicCAS(&S->status[cand], s, (int)FZ_RUNNING) == s;
                }
                ok = __shfl_sync(FULL, ok, 0);
                s = __shfl_sync(FULL, s, 0);
                if (ok) {
                    __threadfence_block();
                    FZ_DBG(0x410000 | (s << 8) | cand);
                    const long long t_r0 = clock64();
                    if (s == FZ_ANSWERED) { FZ_PROF(8, 1); FZ_PROF(9, S->t_ans[cand] - S->t_push[cand]); FZ_PROF(10, t_r0 - S->t_ans[cand]); }
                    fz_run_game<SELFPLAY>(d, FzPort{S}, g0 + cand, cand, s, lane);
                    FZ_PROF(6, 1); FZ_PROF(7, clock64() - t_r0);
                    FZ_DBG(0x420000 | cand);
                    idle = false;
                    rot = cand + 1 < Gc ? cand + 1 : 0;
                }
                continue;
            }
            if (n_wait == 0 && n_ans == 0 && (stop || n_ready == 0)) break;    // nothing left that needs this warp
            FZ_DBG(0x430000 | (n_wait << 8) | n_ans);
            // idle: wait until something is published.  ONE shared-memory word is polled (an ncu instruction profile of the
            // first version, which re-scanned the status array every 0.25-2 us, showed 45 % of the kernel's executed
            // instructions in that loop -- taken from the tower on the same SM).
            if (!idle) { idle = true; idle_t0 = clock64(); idle_it = 0; }
            bool dead = false;
            while (ld_vol(&S->wake) == seen) {
                __nanosleep(idle_it < 16u ? 100 : 400);
                if ((++idle_it & 1023u) == 0u) {
                    if (lane == 0 && *reinterpret_cast<const volatile int *>(P.host_abort)) { st_vol(&S->abort, 1); atomicAdd(&S->wake, 1); }
                    if (clock64() - idle_t0 > FZ_WATCHDOG_CYCLES) {
                        if (lane == 0) { dg.ctr->engine_error = 1; st_vol(&S->abort, 1); atomicAdd(&S->wake, 1); }
                        dead = true;
                        break;
                    }
                }
            }
            if (dead) break;
        }
        __syncwarp();
        FZ_DBG(0x4ff000);
        if (lane == 0 && atomicAdd(&S->tree_exited, 1) == W::TREE_WARPS - 1) { __threadfence_block(); st_vol(&S->quit, 1); }
    }
    TC_FENCE_BEFORE();
    __syncthreads();
    if (warp == W::PRODUCER) {
        __syncwarp();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" :: "r"(tmem) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------ host side
// internal interface used by c4_search.cu
// can the fused engine run this network on a pool of this size at all?
bool c4_fused_supported(const c4_net *net, int max_games)
{
    // (a network served by the caller, c4_net_create_external, has F = 0 and no images: it runs lock-step only)
    if (!net || (net->F != 32 && net->F != 64) || !net->use_tc || !net->image_tc) return false;
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return false;
    const int grid = std::min(sms, max_games);
    if ((max_games + grid - 1) / grid > FZ_GC_MAX) return false;
    return (net->F == 32 ? fz_total<FzK32>(net->R, 0) : fz_total<FzK64>(net->R, 0)) <= 227 * 1024;
}

// ... and is it the engine to use for `live_games` games in flight?  env C4_ENGINE = "fused" / "lockstep" forces one.
bool c4_fused_eligible(const c4_net *net, int max_games, long long live_games)
{
    const char *want = getenv("C4_ENGINE");
    if (want && !strcmp(want, "lockstep")) return false;
    if (!c4_fused_supported(net, max_games)) return false;
    if (want && !strcmp(want, "fused")) return true;
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // auto: the fused engine up to 16 games per SM (2,368 on a B200).  Measured crossover, cold generation, positions/s
    // (profiles/README.md): 256 games 52k vs 23k (lock-step), 1,024 games 123k vs 96k, 2,048 games 189k vs 181k, 4,096 games
    // 291k vs 318k, 8,192 games 315k vs 427k -- with many games per SM the lock-step pass, which gives every phase the
    // whole SM and de-duplicates the evaluations in flight, is ahead
    return live_games <= 16LL * sms;
}

// Run the pool until every game slot is idle / done, `stop_games` games have finished (counter in d.ctr) or `stop_ms`
// have passed, and wait for it.  The host keeps a deadline (env C4_FZ_TIMEOUT_S, default 900 s): when it passes, the
// mapped abort word makes the kernel leave; C4_FZ_DEBUG=1 additionally prints the last checkpoint of every warp of the
// first CTAs if even that does not end the launch.  The caller reads d.ctr afterwards (engine_error / net_nonfinite).
int c4_fused_run(const C4Dev &d, const c4_net *net, int max_games, int simulations, bool selfplay,
                 unsigned long long stop_games, double stop_ms, cudaStream_t stream)
{
    int dev = 0, sms = 0;
    C4_CUDA(cudaGetDevice(&dev));
    C4_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    static int *h_abort = nullptr, *d_abort = nullptr, *dbg = nullptr;
    static unsigned long long *prof = nullptr;
    static cudaStream_t side = nullptr;
    static const bool debug = getenv("C4_FZ_DEBUG") != nullptr;
    if (!h_abort) {
        C4_CUDA(cudaHostAlloc((void **)&h_abort, 64, cudaHostAllocMapped));
        C4_CUDA(cudaHostGetDevicePointer((void **)&d_abort, h_abort, 0));
        C4_CUDA(cudaStreamCreateWithFlags(&side, cudaStreamNonBlocking));
        if (debug) {
            C4_CUDA(cudaMalloc((void **)&dbg, 256 * 32 * sizeof(int))); C4_CUDA(cudaMemset(dbg, 0, 256 * 32 * sizeof(int)));
            C4_CUDA(cudaMalloc((void **)&prof, 16 * sizeof(unsigned long long)));
        }
    }
    *reinterpret_cast<volatile int *>(h_abort) = 0;
    FzParams P;
    P.n_slots = max_games;
    // PUCT tables in shared memory: off by default -- without them the CTA fits the 164 KB shared-memory configuration and
    // the SM keeps 92 KB of L1 for the node records, which is worth more (profiles/README.md)
    const bool f32 = net->F == 32;
    auto total = [&](int entries) { return f32 ? fz_total<FzK32>(net->R, entries) : fz_total<FzK64>(net->R, entries); };
    P.table_entries = (getenv("C4_FZ_SMEM_TABLES") && total(simulations + 2) <= 227 * 1024) ? simulations + 2 : 0;
    P.stop_games = stop_games;
    P.stop_ns = stop_ms > 0.0 ? (unsigned long long)(stop_ms * 1e6) : 0ULL;
    P.host_abort = d_abort;
    P.dbg = dbg;
    P.prof = prof;
    const int tree_warps = f32 ? FzW<FzK32>::TREE_WARPS : FzW<FzK64>::TREE_WARPS;
    P.tree_warps = getenv("C4_FZ_TREE_WARPS") ? std::max(1, std::min(tree_warps, atoi(getenv("C4_FZ_TREE_WARPS")))) : tree_warps;
    if (prof) C4_CUDA(cudaMemsetAsync(prof, 0, 16 * sizeof(unsigned long long), stream));
    const int smem = total(P.table_entries);
    const int grid = std::min(sms, max_games);
    void (*k)(const C4Dev, const unsigned char *, int, FzParams);
    if (f32) k = selfplay ? (net->fp16 ? k_fused<OpFP16, FzK32, true> : k_fused<OpBF16, FzK32, true>)
                          : (net->fp16 ? k_fused<OpFP16, FzK32, false> : k_fused<OpBF16, FzK32, false>);
    else k = selfplay ? (net->fp16 ? k_fused<OpFP16, FzK64, true> : k_fused<OpBF16, FzK64, true>)
                      : (net->fp16 ? k_fused<OpFP16, FzK64, false> : k_fused<OpBF16, FzK64, false>);
    C4_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    k<<<grid, FZ_THREADS, smem, stream>>>(d, (const unsigned char *)net->image_tc, net->R, P);
    C4_CUDA(cudaGetLastError());
    const double limit_s = getenv("C4_FZ_TIMEOUT_S") ? atof(getenv("C4_FZ_TIMEOUT_S")) : 900.0;
    const auto t0 = std::chrono::steady_clock::now();
    bool asked = false;
    for (long long it = 0;; it++) {
        cudaError_t q = cudaStreamQuery(stream);
        if (q == cudaSuccess) break;
        if (q != cudaErrorNotReady) { C4_CUDA(q); }
        const double el = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        if (!asked && el > limit_s) { *reinterpret_cast<volatile int *>(h_abort) = 1; asked = true; }
        if (asked && el > limit_s + 5.0) {
            if (debug && dbg) {
                static int hd[256 * 32];
                if (cudaMemcpyAsync(hd, dbg, sizeof(hd), cudaMemcpyDeviceToHost, side) == cudaSuccess && cudaStreamSynchronize(side) == cudaSuccess)
                    for (int c = 0; c < std::min(grid, 4); c++) {
                        fprintf(stderr, "[fused dbg] cta %d:", c);
                        for (int w = 0; w < 32; w++) fprintf(stderr, " %x", hd[c * 32 + w]);
                        fprintf(stderr, "\n");
                    }
            }
            fprintf(stderr, "[fused] the launch did not end %.0f s after the abort request; giving up\n", 5.0);
            fflush(stderr);
            _exit(86);
        }
        if (it > 2000) std::this_thread::sleep_for(std::chrono::microseconds(el > 1.0 ? 2000 : 50));
    }
    if (prof) {
        unsigned long long h[16];
        C4_CUDA(cudaMemcpy(h, prof, sizeof(h), cudaMemcpyDeviceToHost));
        const double ns = (double)std::max(1ULL, h[0]), nr = (double)std::max(1ULL, h[6]), na = (double)std::max(1ULL, h[8]);
        fprintf(stderr, "[fused prof cta0] strips %llu boards/strip %.2f | cycles per strip: dispatch-wait %.0f input %.0f layers %.0f heads %.0f | "
                        "tree runs %llu cycles/run %.0f | answered %llu push->answer %.0f answer->pick %.0f\n",
                h[0], h[1] / ns, h[2] / ns, h[3] / ns, h[4] / ns, h[5] / ns, h[6], h[7] / nr, h[8], h[9] / na, h[10] / na);
    }
    if (asked) { c4_set_error("fused engine: host deadline passed (C4_FZ_TIMEOUT_S); the launch was aborted"); return -4; }
    return 0;
}
