// c4_split.cu -- the split persistent self-play engine: tree CTAs and tower CTAs on SEPARATE SMs, one leaf ring per tower in HBM.
//
// What it replaces: the same free-running runtime of the reference as the fused engine (game threads that never wait for
// an unrelated game, oinkoink/neural/game_pool.py:15-49; an inference server that batches whatever requests are there,
// oinkoink/neural/inference_server.py:37-63).  The fused engine (c4_fused.cu) puts tree warps AND a tower on every SM; its
// ncu profile shows the price: the two roles share the SM's issue slots, registers (64 per thread for both) and L1, the
// tower runs 1,850 cycles per tile-layer instead of 950, strips are 9 boards.  Here every SM has ONE role:
//   * tree CTAs (1,024 threads): 31 tree warps run the CTA's own games exactly as in the fused engine (fz_run_game,
//     c4_fz.cuh -- the same device functions as the lock-step pass, hence identical records); a leaf that misses the
//     evaluation memo goes into a tower's leaf ring (16-byte entries in HBM / L2).  Warp 31 is the CTA's mail warp: it polls
//     the answer slots of the CTA's waiting games and the memo entries other games wait for, flips their status words in
//     shared memory and keeps the stop / abort flags.
//   * tower CTAs = the batch kernel's tower (c4_net.cu: 16-board strips, two epilogue groups of 8 warps at 96 registers,
//     200 KB of shared memory; 6-board strips for 64 filters) as a server with its OWN leaf ring: the dispatcher (epilogue
//     warp 0) takes what its ring holds -- up to a strip; no batching delay -- and the strip's answers go to the games'
//     answer slots.
//   * requests are dealt round-robin: ONE atomicAdd on a global ticket counter gives a request both its tower (ticket %
//     n_net) and its slot in that tower's ring (ticket / n_net); a tower learns how many entries it owns from the same
//     counter.  Single consumer per ring: no CAS, no contention between the towers (the first version had one shared ring
//     claimed with a CAS on its head: 16k cycles per strip went into the claim).
// ONE launch (k_sp_one): CTAs 0 .. n_tree - 1 are tree CTAs, the rest tower CTAs; one CTA of 1,024 threads per SM and
// n_tree + n_net <= number of SMs, so all of them are resident at once -- the form a kernel that waits must have.  A launch
// has one block size and one register count (64 at 1,024 threads): a tower CTA reshapes its register file with setmaxnreg --
// the 12 warps without a role drop to 24 registers and leave, the producer / issuer warpgroup drops to 56, the 16 epilogue warps
// rise to the 96 the batch kernel's epilogue needs.  A launch also has one shared-memory size, so the tree CTAs carry the
// tower's 200 KB and keep ~28 KB of L1 (cost: 420k instead of 428k positions/s).  The two-launch form (k_sp_tree + k_sp_net on two
// streams, env C4_SP_LAUNCH=two) keeps the tree CTAs' L1 whole, but CUDA does not promise that two launches run side by
// side -- a tool that serialises launches (ncu, CUDA_LAUNCH_BLOCKING=1) deadlocks it until the watchdog -- so it is opt-in
// and gated by a co-residency probe.  All cross-SM hand-offs are polls of L2-resident words with a back-off; every wait is
// bounded (tree-warp watchdog -> abort flag -> all CTAs leave; host deadline through a mapped word), so a protocol bug ends
// in an error code, not in a hung device.
//
// Last part of round 2 (DESIGN.md section 4.0): the tree CTAs of the one-launch form keep the PUCT tables in the shared memory they
// carry anyway (GameTab, c4_tree.cuh: compile-time offsets, plain LDS) and descend without the lock-step pass's speculative prefetch
// (GameNP); and the split of the SMs between the roles is ADAPTIVE: a run is cut into time slices (SpParams::slice_ns), each slice is
// one launch, and the host picks the next slice's tower count from the load signals of the last one (sp_adapt_next).
//
// NO gpu-scope fence on the data path: __threadfence() invalidates the SM's whole L1 (CCTL.IVALL) -- in a tree CTA that
// is the cache of the node records, and the first version paid it on every request and every answer.  Instead every
// cross-SM message is made of self-validating 8-byte words (aligned 8-byte stores and loads are single transactions):
//   * ring entry = two words {c0 (48 bits) | game << 48 | stamp << 62} {c1 (48 bits) | tag << 48 | stamp << 62}; stamp = 1 +
//     lap parity of the slot (0 = never written; rings are zeroed per launch).  The consumer spins until both stamps are
//     those of the lap it expects.  Ring capacity >= game slots and a game has at most one leaf pending, so a slot is never
//     overwritten before it was read.
//   * answer = eight words {float bits | tag << 32} in the game's answer slot, stored by eight lanes of the tower's head
//     warp.  tag = the game's request number (14 bits, never 0).  The mail warp looks at the LAST word only (a hint); the
//     tree warp that claims the game reads all eight with ld.global.cg and spins until every tag matches.
//   * status words, stop / abort flags: as in the fused engine (c4_fused.cu).
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include <algorithm>
#include <type_traits>
#include <chrono>
#include <mutex>
#include <thread>

#include "c4_fz.cuh"

#define SP_GMAX 16384                                     // game slots the engine accepts
#define SP_GC_MAX 256                                     // game slots per tree CTA
#define SP_TREE_THREADS 1024
#define SP_TREE_WARPS 31                                  // warps 0..30 run games, warp 31 is the mail warp
#define SP_NB 16                                          // boards per strip (TcC<32>::NB)
#define SP_PATIENCE 4                                     // watch time-outs after which a parked game asks for itself
#define SP_WATCH_SWEEPS 2048                              // mail-warp sweeps (~150 ns each) until a watch times out

struct SpHeader {                                         // (what the host reads back after a launch)
    unsigned ticket; unsigned pad0[31];                   // requests issued so far (dealt round-robin to the towers)
    int quit, abort, trees_exited, sliced; int pad2[28];  // sliced: a tree CTA ended this launch because its time slice was over
    unsigned long long prof[32];
    unsigned long long sig[16];                           // load signals of the launch (always on): [0] strips, [1] boards in them,
                                                          // [2] tree-warp cycles in runs, [3] tree-warp cycles idle between runs
};
struct SpGlobal : SpHeader {
    unsigned long long ans[SP_GMAX][8];                   // per game slot: {float bits | tag << 32} x {prior[7], value}
    // followed by the rings: [n_net][ring_cap][2] words
};
__host__ __device__ constexpr size_t sp_rings_off() { return (sizeof(SpGlobal) + 255) & ~(size_t)255; }

struct SpParams {
    int n_slots;                        // game slots of the pool
    unsigned long long stop_games;      // leave once ctr->games_finished reaches this (0 = never)
    unsigned long long stop_ns;         // leave after this much run time (0 = never)
    unsigned long long slice_ns;        // leave after this much run time AND tell the host (SpGlobal::sliced) that the launch is to be
                                        // continued by another one, possibly with another tower count (0 = no slices)
    const int *host_abort;              // mapped host word: non-zero = the host gave up waiting, leave at once
    int prof;                           // accumulate cycle / event sums in SpGlobal::prof (C4_FZ_DEBUG)
    int batch_ns;                       // a dispatcher that finds less than a strip waits up to this long for more
    int n_tree;                         // tree CTAs (the first n_tree CTAs of a single launch)
    int n_net;                          // tower CTAs = rings
    unsigned ring_cap;                  // entries per ring (power of two >= game slots)
    int stage_nodes;                    // node records per game that a tree CTA keeps in shared memory (multiple of 8; 0 = none)
    int table_entries;                  // entries of each PUCT table (log / sqrt / reciprocal) a tree CTA of the ONE-launch form keeps in
                                        // the shared memory it carries anyway (0: read them through L1 from HBM)
};

// tree CTA control block (shared memory)
struct SpCtl {
    int abort, stop, tree_exited, wake;
    int status[SP_GC_MAX];              // ST_* / FZ_*: authoritative while the kernel runs
    unsigned req[SP_GC_MAX];            // request number of the game's last leaf (= its answer tag)
    // ST_WAITMEMO games: the memo entry's check word the mail warp watches, the PENDING tag it holds while the owner's
    // evaluation is in flight, the mail-warp sweep at which the game was parked, and how often the watch timed out
    const unsigned long long *watch[SP_GC_MAX];
    unsigned long long watch_tag[SP_GC_MAX];
    unsigned watch_t0[SP_GC_MAX];
    int watch_timeouts[SP_GC_MAX];
    unsigned sweep;                     // the mail warp's sweep counter
};

__device__ __forceinline__ unsigned ld_volu(const unsigned *p) { return *reinterpret_cast<const volatile unsigned *>(p); }
__device__ __forceinline__ unsigned long long ld_vol64(const unsigned long long *p) { return *reinterpret_cast<const volatile unsigned long long *>(p); }
__device__ __forceinline__ unsigned sp_tag(unsigned request_no) { return request_no % 16383u + 1u; }   // 14 bits, never 0
__device__ __forceinline__ unsigned long long *sp_ring(SpGlobal *G, unsigned cap, int r)
{
    return reinterpret_cast<unsigned long long *>(reinterpret_cast<unsigned char *>(G) + sp_rings_off()) + (size_t)r * cap * 2;
}
__device__ __forceinline__ void st_volu(unsigned *p, unsigned v) { *reinterpret_cast<volatile unsigned *>(p) = v; }
// PUCT tables in a tree CTA's dynamic shared memory (one-launch form): behind the control block, SP_TAB_STRIDE entries apart
#define SP_TAB_OFF ((uint32_t)((sizeof(SpCtl) + 127) & ~(size_t)127))
#define SP_TAB_STRIDE 4096u

#define SP_PROF(i, v) do { if (P.prof) atomicAdd(&G->prof[i], (unsigned long long)(v)); } while (0)

// the split engine's port: the answer comes from the game's answer slot in HBM / L2 (written by a tower CTA), the request goes
// to the ring of the tower its ticket names
template <bool TAB>
struct SpPort {
    static constexpr int GC_MAX = SP_GC_MAX;
    static constexpr bool DEDUP = true;
    SpCtl *S;
    SpGlobal *G;
#ifdef C4_SP_STAGE_TOP
    typedef GameS GameType;
    uint32_t stage_base32;              // .shared address of [game of the CTA][stage_nodes] node records (or stage_nodes == 0)
    uint32_t stage_nodes;
    __device__ __forceinline__ void stage(GameS &g, int gl) const { g.sp32 = stage_base32 + (uint32_t)gl * stage_nodes * 32u; g.sp_nodes = stage_nodes; }
#else
    typedef typename std::conditional<TAB, GameTab<SP_TAB_OFF, SP_TAB_STRIDE>, GameNP>::type GameType;
    __device__ __forceinline__ void stage(Game &, int) const {}
#endif
    const uint32_t *memo;
    uint32_t memo_mask, memo_epoch;
    unsigned n_net, ring_cap;
    __device__ __forceinline__ int stopping() const { return ld_vol(&S->stop); }
    // all eight words of the answer must carry the tag of the game's request (the mail warp only saw the last one)
    __device__ __forceinline__ float answer(int g, int gl, int lane) const
    {
        const unsigned tag = sp_tag(S->req[gl]);
        const unsigned long long *a = &G->ans[g][lane & 7];
        unsigned long long v = __ldcg(a);
        while (!__all_sync(FULL, (unsigned)(v >> 32) == tag)) v = ld_vol64(a);
        return (lane < 8) ? __uint_as_float((unsigned)v) : 0.f;
    }
    // a parked game whose watch timed out SP_PATIENCE times (the owner of the tag never answered) asks for itself
    __device__ __forceinline__ bool impatient(int gl) const { return S->watch_timeouts[gl] >= SP_PATIENCE; }
    __device__ __forceinline__ void publish(int g, int gl, int st, bool request, u64 rc0, u64 rc1) const
    {
        unsigned tag = 0u;
        if (request) {
            const unsigned no = S->req[gl] + 1u;
            *reinterpret_cast<volatile unsigned *>(&S->req[gl]) = no;
            tag = sp_tag(no);
            S->watch_timeouts[gl] = 0;
        }
        if (st == ST_WAITMEMO) {
            S->watch[gl] = reinterpret_cast<const unsigned long long *>(memo + (size_t)memo_index(rc0, rc1, memo_mask) * 16 + 12);
            S->watch_tag[gl] = memo_pending_tag(memo_epoch, rc0, rc1);
            S->watch_t0[gl] = ld_volu(&S->sweep);
        }
        __threadfence_block();
        st_vol(&S->status[gl], st);                                       // WAIT (and its request number) visible before the request is
        if (st == ST_IDLE || st == ST_DONE) atomicAdd(&S->wake, 1);       // idle warps re-check whether anything is left
        if (request) {
            const unsigned n = atomicAdd(&G->ticket, 1u);
            const unsigned r = n % n_net, k = n / n_net;
            const unsigned long long stamp = 1ULL + ((k / ring_cap) & 1u);
            unsigned long long *e = sp_ring(G, ring_cap, (int)r) + (size_t)(k & (ring_cap - 1u)) * 2;
            C4_DEV_ASSERT((rc0 >> 48) == 0 && (rc1 >> 48) == 0 && g < (1 << 14));
            __stcg(reinterpret_cast<ulonglong2 *>(e), make_ulonglong2(rc0 | ((unsigned long long)g << 48) | (stamp << 62),
                                                                       rc1 | ((unsigned long long)tag << 48) | (stamp << 62)));
        }
    }
};

// ------------------------------------------------------------------------------------------------ tree CTAs
// (body of a tree CTA: CTAs 0 .. n_tree - 1 of the launch)
// (TAB: the PUCT tables are read from the CTA's dynamic shared memory -- one-launch form only)
template <bool SELFPLAY, bool TAB>
__device__ __forceinline__ void sp_tree_body(const C4Dev &dg, SpGlobal *G, const SpParams &P, SpCtl *S)
{
    const int warp = __shfl_sync(FULL, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    // this CTA's game slots
    const int per = P.n_slots / P.n_tree, extra = P.n_slots % P.n_tree;
    const int Gc = per + ((int)blockIdx.x < extra ? 1 : 0);
    const int g0 = (int)blockIdx.x * per + min((int)blockIdx.x, extra);

    for (int i = threadIdx.x; i < (int)(sizeof(SpCtl) / 4); i += blockDim.x) reinterpret_cast<uint32_t *>(S)[i] = 0u;
    __syncthreads();
    for (int i = threadIdx.x; i < SP_GC_MAX; i += blockDim.x) S->status[i] = (i < Gc) ? fz_entry_status(dg, g0 + i) : (int)ST_IDLE;
    if (TAB) {
        // PUCT tables (19 KB at 800 simulations; every level of every descent reads all three): a tree CTA of the one-launch form
        // carries the tower's 200 KB of shared memory and has only ~28 KB of L1, which the tables would share with the node records
        double *tab = reinterpret_cast<double *>(reinterpret_cast<unsigned char *>(S) + SP_TAB_OFF);
        for (int i = threadIdx.x; i < P.table_entries; i += blockDim.x) {
            tab[i] = dg.pbc[i]; tab[SP_TAB_STRIDE + i] = dg.sqt[i]; tab[2 * SP_TAB_STRIDE + i] = dg.rcp[i];
        }
    }
#ifdef C4_SP_STAGE_TOP
    // shared-memory staging of the top of each tree: the first stage_nodes node records of every game of this CTA (the blocks
    // created first: root, its children, the first expansions) are copied in here, live in shared memory while the launch
    // runs (GameS in c4_tree.cuh) and are copied back at the end -- a game never leaves its CTA
    C4Node *stage_base = reinterpret_cast<C4Node *>(reinterpret_cast<unsigned char *>(S) + ((sizeof(SpCtl) + 127) & ~(size_t)127));
    {
        const int per_game = P.stage_nodes * 2;                              // 16-byte units (a node record is 32 bytes)
        for (int i = threadIdx.x; i < Gc * per_game; i += blockDim.x) {
            const int gl = i / per_game, k = i - gl * per_game;
            reinterpret_cast<uint4 *>(stage_base)[i] =
                __ldcg(reinterpret_cast<const uint4 *>(dg.pool + (size_t)(g0 + gl) * dg.blocks_per_game * C4_SLOTS) + k);
        }
    }
#endif
    __syncthreads();
    const unsigned long long t_begin = fz_globaltimer();

    if (warp == SP_TREE_WARPS) {
        // ================= mail warp: answer tags of the waiting games -> status words; stop / abort flags
        for (uint32_t it = 0;; it++) {
            if (lane == 0 && (it & 7u) == 0u) {
                if (!ld_vol(&S->stop)) {
                    bool stop = false;
                    if (P.stop_games && __ldcg(&dg.ctr->games_finished) >= P.stop_games) stop = true;
                    if (P.stop_ns && fz_globaltimer() - t_begin > P.stop_ns) stop = true;
                    if (!stop && P.slice_ns && fz_globaltimer() - t_begin > P.slice_ns) { stop = true; st_vol(&G->sliced, 1); }
                    if (stop) { st_vol(&S->stop, 1); atomicAdd(&S->wake, 1); }
                }
                if ((it & 8191u) == 0u && *reinterpret_cast<const volatile int *>(P.host_abort)) st_vol(&G->abort, 1);
                if (!ld_vol(&S->abort) && ld_vol(&G->abort)) { st_vol(&S->abort, 1); atomicAdd(&S->wake, 1); }
            }
            int n_wait = 0;
            const bool look = (it & 7u) == 0u;                                // the memo watches are looked at every 8th sweep
            for (int base = 0; base < Gc; base += 32) {
                const int i = base + lane;
                const int st = i < Gc ? ld_vol(&S->status[i]) : (int)ST_IDLE;
                const bool w = st == ST_WAIT, wm = st == ST_WAITMEMO;
                bool hit = false;
                if (w) {
                    const unsigned tag = sp_tag(ld_volu(&S->req[i]));
                    hit = (unsigned)(ld_vol64(&G->ans[g0 + i][7]) >> 32) == tag;
                    if (hit) { __threadfence_block(); st_vol(&S->status[i], FZ_ANSWERED); }
                } else if (wm && look) {
                    // the PENDING tag is gone: the owner's answer is in (or a colliding key took the entry) -- probe again
                    const bool timeout = it - S->watch_t0[i] > SP_WATCH_SWEEPS;
                    hit = *reinterpret_cast<const volatile unsigned long long *>(S->watch[i]) != S->watch_tag[i] || timeout;
                    if (hit) { if (timeout) S->watch_timeouts[i]++; __threadfence_block(); st_vol(&S->status[i], FZ_MEMOREADY); }
                }
                n_wait += __popc(__ballot_sync(FULL, w || wm));
                if (__any_sync(FULL, hit) && lane == 0) { __threadfence_block(); atomicAdd(&S->wake, 1); }
            }
            if (lane == 0) st_volu(&S->sweep, it + 1u);
            if (ld_vol(&S->tree_exited) == SP_TREE_WARPS) break;
            __nanosleep(n_wait ? 150 : 1000);
        }
        __syncwarp();
        if (lane == 0 && atomicAdd(&G->trees_exited, 1) == P.n_tree - 1) { __threadfence(); st_vol(&G->quit, 1); }
    } else {
        // ================= tree warps (the picker loop of the fused engine)
#ifdef C4_SP_STAGE_TOP
        uint32_t stage_base32;                                                // (volatile: computed once, not re-derived from the window base at every access)
        asm volatile("{ .reg .u64 t; cvta.to.shared.u64 t, %1; cvt.u32.u64 %0, t; }" : "=r"(stage_base32) : "l"(stage_base));
        const SpPort<false> port{S, G, stage_base32, (uint32_t)P.stage_nodes, dg.memo, dg.memo_mask, dg.memo_epoch, (unsigned)P.n_net, P.ring_cap};
#else
        const SpPort<TAB> port{S, G, dg.memo, dg.memo_mask, dg.memo_epoch, (unsigned)P.n_net, P.ring_cap};
#endif
        int rot = (warp * 9) % Gc;
        bool idle = false;
        long long idle_t0 = 0;
        uint32_t idle_it = 0;
        long long t_run = 0, n_run = 0, t_idle = 0;
        for (;;) {
            const int seen = ld_vol(&S->wake);                             // read BEFORE the scan: no wake-up is lost
            const int aborting = ld_vol(&S->abort);
            const int stop = ld_vol(&S->stop) | aborting;
            int cand = -1, n_wait = 0, n_ans = 0, n_ready = 0;
            bool cand_ans = false;
            for (int base = 0; base < Gc; base += 32) {
                const int i = base + lane;
                int idx = i + rot;
                if (idx >= Gc) idx -= Gc;
                const int s = (i < Gc) ? ld_vol(&S->status[idx]) : ST_IDLE;
                const unsigned ma = __ballot_sync(FULL, s == FZ_ANSWERED);
                const unsigned mr = __ballot_sync(FULL, s == ST_READY || s == ST_NEWROOT || s == FZ_MEMOREADY);
                const unsigned mw = __ballot_sync(FULL, s == ST_WAIT);
                n_wait += __popc(mw); n_ans += __popc(ma); n_ready += __popc(mr);
                n_ready += __popc(__ballot_sync(FULL, s == ST_WAITMEMO));   // parked on another game's evaluation: will be handed back
                if (ma && !cand_ans) { cand = __shfl_sync(FULL, idx, __ffs((int)ma) - 1); cand_ans = true; }
                else if (mr && cand < 0 && !stop) cand = __shfl_sync(FULL, idx, __ffs((int)mr) - 1);
            }
            if (aborting) break;
            if (cand >= 0) {
                int s = 0, ok = 0;
                if (lane == 0) {
                    s = ld_vol(&S->status[cand]);
                    if (s == FZ_ANSWERED || (!stop && (s == ST_READY || s == ST_NEWROOT || s == FZ_MEMOREADY)))
                        ok = atomicCAS(&S->status[cand], s, (int)FZ_RUNNING) == s;
                }
                ok = __shfl_sync(FULL, ok, 0);
                s = __shfl_sync(FULL, s, 0);
                if (ok) {
                    __threadfence_block();
                    const long long t_r0 = clock64();
                    if (idle) { t_idle += t_r0 - idle_t0; idle = false; }
                    fz_run_game<SELFPLAY>(dg, port, g0 + cand, cand, s, lane);
                    t_run += clock64() - t_r0; n_run++;
                    rot = cand + 1 < Gc ? cand + 1 : 0;
                }
                continue;
            }
            if (n_wait == 0 && n_ans == 0 && (stop || n_ready == 0)) break;    // nothing left that needs this warp
            // idle: wait until something is published (one shared-memory word is polled, see c4_fused.cu)
            if (!idle) { idle = true; idle_t0 = clock64(); idle_it = 0; }
            bool dead = false;
            while (ld_vol(&S->wake) == seen) {
                __nanosleep(idle_it < 16u ? 100 : 400);
                if ((++idle_it & 1023u) == 0u && clock64() - idle_t0 > FZ_WATCHDOG_CYCLES) {
                    if (lane == 0) { dg.ctr->engine_error = 1; st_vol(&G->abort, 1); st_vol(&S->abort, 1); atomicAdd(&S->wake, 1); }
                    dead = true;
                    break;
                }
            }
            if (dead) break;
        }
        __syncwarp();
        if (lane == 0) {
            if (P.prof) { SP_PROF(8, n_run); SP_PROF(9, t_run); SP_PROF(10, t_idle); }
            atomicAdd(&G->sig[2], (unsigned long long)t_run); atomicAdd(&G->sig[3], (unsigned long long)t_idle);
            __threadfence_block();
            atomicAdd(&S->tree_exited, 1);
        }
    }
#ifdef C4_SP_STAGE_TOP
    // every warp of the CTA is done with the games: the staged tree tops go back to the pool in HBM (read-outs, tree export,
    // the next launch and the other engines read it there)
    __syncthreads();
    {
        const int per_game = P.stage_nodes * 2;
        for (int i = threadIdx.x; i < Gc * per_game; i += blockDim.x) {
            const int gl = i / per_game, k = i - gl * per_game;
            reinterpret_cast<uint4 *>(dg.pool + (size_t)(g0 + gl) * dg.blocks_per_game * C4_SLOTS)[k] = reinterpret_cast<const uint4 *>(stage_base)[i];
        }
    }
#endif
}

// ------------------------------------------------------------------------------------------------ tower CTAs
struct SpNetCtl {
    int strip_nb, quit, abort, pad;
    int strip_game[SP_NB];
    unsigned strip_tag[SP_NB];
    u64 strip_c0[SP_NB], strip_c1[SP_NB];
    float ans[SP_NB][8];
};
template <int F> __host__ __device__ constexpr int sp_ctl_off(int R) { return (TcK<F>::total(R) + 15) & ~15; }
template <int F> __host__ __device__ constexpr int sp_net_smem(int R) { return sp_ctl_off<F>(R) + (int)sizeof(SpNetCtl); }

// (body of tower CTA `tower`.  Warp roles: EPI0 .. EPI0 + 15 epilogue, PRODUCER, ISSUER.  ONE_LAUNCH: the CTA has 1,024
//  threads at 64 registers like the tree CTAs of the same launch; the 16 epilogue warps raise their register limit to 96 with
//  setmaxnreg from what the 12 warps without a role and the producer / issuer warpgroup give back:
//  16 x 32 x 96 + 4 x 32 x 56 + 12 x 32 x 24 = 65,536.)
template <typename OP, int F, int EPI0, int PRODUCER, int ISSUER, bool ONE_LAUNCH>
__device__ __forceinline__ void sp_net_body(const unsigned char *__restrict__ image, int R, SpGlobal *G, C4Counters *ctr,
                                            const SpParams &P, unsigned char *smem, const unsigned tower)
{
    using K = TcK<F>;                                                      // the batch kernel's geometry (c4_tc.cuh)
    static_assert(K::NB <= SP_NB && K::EPI_WARPS == TC_EPI_WARPS, "strip control block / epilogue warps");
    static_assert(EPI0 % 4 == 0 || !ONE_LAUNCH, "setmaxnreg works on warpgroups");
    const int L = 1 + 2 * R;
    const int warp = __shfl_sync(FULL, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;

    unsigned char *sX = smem + K::X, *sH = smem + K::H, *sW = smem + K::W;
    float *small = reinterpret_cast<float *>(smem + K::SMALL);
    const float *bias = small, *hp = small + L * F;
    float *scratch = reinterpret_cast<float *>(smem + K::scratch(R));
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + K::bars(R));
    const uint32_t b_wfull = smem_u32(bars), b_wempty = b_wfull + 8 * K::WBARS;
    const uint32_t b_accfull = b_wempty + 8 * K::WBARS, b_accempty = b_accfull + 8 * K::ACC_SLOTS;
    const uint32_t b_epi = b_accempty + 8 * K::ACC_SLOTS;                   // T barriers
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * K::WBARS + 2 * K::ACC_SLOTS + K::T);
    SpNetCtl *S = reinterpret_cast<SpNetCtl *>(smem + sp_ctl_off<F>(R));

    // ---- one-time setup (k_net_tc): zero the strips, small params, barriers, TMEM
    for (int i = threadIdx.x; i < 2 * K::ACT_BYTES / 16; i += blockDim.x)
        reinterpret_cast<uint4 *>(sX)[i] = make_uint4(0u, 0u, 0u, 0u);
    {
        const unsigned char *src = image + (size_t)L * K::WSTAGE_BYTES;
        const int nb16 = (L * F + HEAD_FLOATS) * 4 / 16;
        for (int i = threadIdx.x; i < nb16; i += blockDim.x)
            reinterpret_cast<uint4 *>(small)[i] = reinterpret_cast<const uint4 *>(src)[i];
    }
    for (int i = threadIdx.x; i < (int)(sizeof(SpNetCtl) / 4); i += blockDim.x) reinterpret_cast<uint32_t *>(S)[i] = 0u;
    if (threadIdx.x == 0) {
        for (int i = 0; i < K::WBARS; i++) { mbar_init(b_wfull + 8 * i, 1); mbar_init(b_wempty + 8 * i, 1); }
        for (int i = 0; i < K::ACC_SLOTS; i++) { mbar_init(b_accfull + 8 * i, 1); mbar_init(b_accempty + 8 * i, K::GROUP_WARPS); }
        for (int i = 0; i < K::T; i++) mbar_init(b_epi + 8 * i, K::GROUP_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == PRODUCER) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;\n" :: "r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    TC_PROXY_FENCE();
    TC_FENCE_BEFORE();
    __syncthreads();
    TC_FENCE_AFTER();
    const uint32_t tmem = *tmem_slot;
    if (ONE_LAUNCH) {
        if (warp >= EPI0 + 16 && (warp < (PRODUCER & ~3) || warp >= (PRODUCER & ~3) + 4)) {
            asm volatile("setmaxnreg.dec.sync.aligned.u32 24;\n");          // no role in a tower CTA
            return;
        }
        if (warp >= (PRODUCER & ~3) && warp < (PRODUCER & ~3) + 4) {
            asm volatile("setmaxnreg.dec.sync.aligned.u32 56;\n");          // producer / issuer warpgroup (single threads at work)
            if (warp != PRODUCER && warp != ISSUER) return;
        } else {
            asm volatile("setmaxnreg.inc.sync.aligned.u32 96;\n");          // epilogue warps
        }
    }

    if (warp == PRODUCER) {
        // ================= weight producer: layer g of the endless (strip, layer) sequence -> ring stage g % WSTAGES; it
        // runs up to WSTAGES layers ahead of the issuer, so the first layers of the NEXT strip are on chip while the tower idles
        if (lane == 0 && K::SLICED) {
            // one weight stage, refilled one dy slice at a time: slice dy of layer g is requested as soon as the issuer has
            // released slice dy of layer g - 1 (c4_net.cu)
            int g = 0, last[3] = {-1, -1, -1};
            bool live = true;
            for (; live; g++)
                for (int dy = 0; dy < 3 && live; dy++) {
                    if (g > 0) {
                        const uint32_t bar = b_wempty + 8 * dy, par = (uint32_t)(g - 1) & 1u;
                        for (uint32_t it = 0; !mbar_try(bar, par); it++) {
                            if (it > 4u) __nanosleep(it > 64u ? 500 : 100);
                            if ((it & 15u) == 15u && ld_vol(&S->quit)) { live = false; break; }
                        }
                        if (!live) break;
                    }
                    mbar_expect_tx(b_wfull + 8 * dy, K::WSLICE_BYTES);
                    bulk_g2s(smem_u32(sW + dy * K::WSLICE_BYTES), image + (size_t)(g % L) * K::WSTAGE_BYTES + dy * K::WSLICE_BYTES,
                             K::WSLICE_BYTES, b_wfull + 8 * dy);
                    last[dy] = g;
                }
            for (int dy = 0; dy < 3; dy++)                                        // no bulk copy in flight at exit
                if (last[dy] >= 0) mbar_wait(b_wfull + 8 * dy, (uint32_t)last[dy] & 1u);
        } else if (lane == 0) {
            int g = 0;
            bool live = true;
            for (; live; g++) {
                const int st = g % K::WSTAGES, use = g / K::WSTAGES;
                if (use > 0) {
                    const uint32_t bar = b_wempty + 8 * st, par = (uint32_t)(use - 1) & 1u;
                    for (uint32_t it = 0; !mbar_try(bar, par); it++) {
                        if (it > 4u) __nanosleep(it > 64u ? 500 : 100);
                        if ((it & 15u) == 15u && ld_vol(&S->quit)) { live = false; break; }
                    }
                    if (!live) break;
                }
                mbar_expect_tx(b_wfull + 8 * st, K::WSTAGE_BYTES);
                bulk_g2s(smem_u32(sW + st * K::WSTAGE_BYTES), image + (size_t)(g % L) * K::WSTAGE_BYTES, K::WSTAGE_BYTES,
                         b_wfull + 8 * st);
            }
            // no bulk copy may be in flight when the CTA exits: wait for the stages requested last
            for (int i = max(0, g - K::WSTAGES); i < g; i++) mbar_wait(b_wfull + 8 * (i % K::WSTAGES), (uint32_t)(i / K::WSTAGES) & 1u);
        }
    } else if (warp == ISSUER) {
        // ================= MMA issuer (one thread): the strip loop of k_net_tc with strips that arrive at run time
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | ((uint32_t)OP::FMT << 7) | ((uint32_t)OP::FMT << 10) |
                                   ((uint32_t)(K::NN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
            int g = 0, c = 0;                                   // (strip, layer) counter, (strip, layer, tile) counter
            bool live = true;
            for (int s = 0; live; s++) {
                // every strip completes L + 1 phases on EVERY tile barrier (input planes + L epilogues)
                if (!fz_wait(b_epi, (uint32_t)(s * (L + 1)) & 1u, &S->abort)) break;
                const int nb = ld_vol(&S->strip_nb);
                if (nb == 0) break;                                             // the dispatcher said quit
                const int T = (7 * nb + 15) / 16;
                for (int l = 0; l < L && live; l++, g++) {
                    const int st = g % K::WSTAGES;
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
                // observe the LAST epilogue phase of tile 0 too (c4_fused.cu: with a one-tile strip the wait for the next
                // strip's input phase would otherwise alias this strip's phase L - 1)
                if (live && !fz_wait(b_epi, (uint32_t)(s * (L + 1) + L) & 1u, &S->abort)) break;
            }
        }
    } else {
        // ================= epilogue warps (+ the dispatcher in the first of them)
        const int e = warp - EPI0, quad = warp & 3, half = (e >> 2) % K::SLICES, group = e / K::GROUP_WARPS;
        const int et = threadIdx.x - 32 * EPI0;                              // 0..511
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
        E.calib = nullptr;
        int c = 0;                                                           // global (strip, layer, tile) counter
        unsigned ring_head = 0u;                                             // dispatcher: entries of this tower's ring consumed
        unsigned sig_strips = 0u;                                            // dispatcher: strips served (boards = ring_head)
        const unsigned long long *ring = sp_ring(G, P.ring_cap, (int)tower);
        for (;;) {
            const long long t_d0 = clock64();
            long long t_work = t_d0;                                         // dispatcher: first look that found leaves
            if (e == 0) {
                // ---- dispatch: take what this tower's ring holds (up to one strip).  The ring's entries are the tickets
                // n = k * n_net + tower; `ticket` tickets have been issued so far.
                int k = 0;
                long long t_first = 0;
                for (uint32_t it = 1;; it++) {
                    unsigned issued = 0;
                    int q = 0;
                    if (lane == 0) {
                        const unsigned t = ld_volu(&G->ticket);
                        issued = (t + (unsigned)P.n_net - 1u - tower) / (unsigned)P.n_net;
                        q = ld_vol(&G->quit) | (ld_vol(&G->abort) << 1);
                    }
                    issued = __shfl_sync(FULL, issued, 0); q = __shfl_sync(FULL, q, 0);
                    const int avail = (int)(issued - ring_head);
                    if (q & 2) break;                                        // abort: leave at once
                    if (avail <= 0) {
                        if (q) break;                                        // every tree CTA has left: nothing can be pending
                        if ((it & 4095u) == 0u && lane == 0 && *reinterpret_cast<const volatile int *>(P.host_abort)) st_vol(&G->abort, 1);
                        t_first = 0;
                        __nanosleep(it > 64u ? 300 : 60);
                        continue;
                    }
                    if (avail < K::NB && P.batch_ns > 0) {                   // optional batching window
                        const long long now = (long long)fz_globaltimer();
                        if (t_first == 0) t_first = now;
                        if (now - t_first < P.batch_ns) { __nanosleep(100); continue; }
                    }
                    if (P.prof) t_work = clock64();
                    k = min(avail, K::NB);
                    if (lane < k) {
                        const unsigned idx = ring_head + (unsigned)lane;
                        const unsigned long long stamp = 1ULL + ((idx / P.ring_cap) & 1u);
                        const unsigned long long *en = ring + (size_t)(idx & (P.ring_cap - 1u)) * 2;
                        unsigned long long a = 0, b = 0;
                        for (uint32_t w = 0;; w++) {                         // ticket taken, words not written yet
                            a = ld_vol64(en); b = ld_vol64(en + 1);
                            if ((a >> 62) == stamp && (b >> 62) == stamp) break;
                            __nanosleep(40);
                            if ((w & 255u) == 255u && ld_vol(&G->abort)) break;
                        }
                        S->strip_c0[lane] = a & 0xFFFFFFFFFFFFULL;
                        S->strip_c1[lane] = b & 0xFFFFFFFFFFFFULL;
                        S->strip_game[lane] = (int)((a >> 48) & 0x3FFFu);
                        S->strip_tag[lane] = (unsigned)((b >> 48) & 0x3FFFu);
                    }
                    ring_head += (unsigned)k;
                    sig_strips++;
                    break;
                }
                __syncwarp();
                if (lane == 0) {
                    if (k == 0) { st_vol(&S->quit, 1); atomicAdd(&G->sig[0], (unsigned long long)sig_strips); atomicAdd(&G->sig[1], (unsigned long long)ring_head); }
                    __threadfence_block();
                    st_vol(&S->strip_nb, k);
                }
            }
            EPI_BAR();
            const int nb = ld_vol(&S->strip_nb);
            // (the dispatcher overwrites strip_game for the next strip while other warps are still in their head tails, so
            //  the game of THIS warp's board is read now)
            const int my_game = S->strip_game[e];
            const unsigned my_tag = S->strip_tag[e];
            const long long t_d1 = clock64();
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
            for (int i = et; i < nb * 42; i += 32 * TC_EPI_WARPS) {
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
            EPI_BAR();
            const long long t_d2 = clock64();
            // every phase completes on ALL tile barriers (also those of tiles this strip does not have), so that the
            // phase parity of a tile barrier is a function of (strip, layer) only
            if (lane == 0 && e < K::GROUP_WARPS)
                for (int t = 0; t < K::T; t++) mbar_arrive(b_epi + 8 * t);
#define SP_SKIPPED_TILES() if (lane == 0 && e < K::GROUP_WARPS) for (int t = T; t < K::T; t++) mbar_arrive(b_epi + 8 * t)
            tc_epilogue_layer<OP, F, 0>(E, 0, T, c); c += T; SP_SKIPPED_TILES();
            for (int l = 1; l < L - 1; l += 2) {
                tc_epilogue_layer<OP, F, 1>(E, l, T, c); c += T; SP_SKIPPED_TILES();
                if (l + 1 < L - 1) { tc_epilogue_layer<OP, F, 2>(E, l + 1, T, c); c += T; SP_SKIPPED_TILES(); }
            }
            tc_epilogue_layer<OP, F, 3>(E, L - 1, T, c); c += T; SP_SKIPPED_TILES();
#undef SP_SKIPPED_TILES

            // ---- head tails: one warp per board; the answer goes to the game's answer slot, every word tagged
            EPI_BAR();
            const long long t_d3 = clock64();
            if (e < nb) {
                float *sc = scratch + e * 128;
                for (int i = lane; i < 126; i += 32) {
                    float bb = i < 42 ? hp[HO_VB] : (i < 84 ? hp[HO_PB] : hp[HO_PB + 1]);
                    float acc = sc[i];                                       // channel slices summed in a fixed order
#pragma unroll
                    for (int q = 1; q < K::SLICES; q++) acc += sc[q * K::NB * 128 + i];
                    sc[i] = leaky(acc + bb);
                }
                __syncwarp();
                float *ans = S->ans[e];
                head_tail(sc, hp, ans, lane);
                float o = (lane < 8) ? ans[lane] : 0.f;
                if (__any_sync(FULL, !isfinite(o))) {
                    // operand overflow (fp16) or NaN weights: never into the tree -- neutral answer + a flag that makes the
                    // host call fail (the reference asserts, oinkoink/neural/pytorch/model.py:258-263,275-280)
                    o = (lane < 7) ? (1.f / 7.f) : 0.5f;
                    if (lane == 0) ctr->net_nonfinite = 1;
                }
                if (lane < 8) __stcg(&G->ans[my_game][lane], (unsigned long long)__float_as_uint(o) | ((unsigned long long)my_tag << 32));
            }
            if (P.prof && e == 0 && lane == 0) {
                SP_PROF(0, 1); SP_PROF(1, nb); SP_PROF(2, t_work - t_d0); SP_PROF(3, clock64() - t_work);
                SP_PROF(4, t_d1 - t_work); SP_PROF(5, t_d2 - t_d1); SP_PROF(6, t_d3 - t_d2); SP_PROF(7, clock64() - t_d3);
            }
        }
    }
    TC_FENCE_BEFORE();
    asm volatile("bar.sync 2, 576;\n" ::: "memory");                       // the 18 warps with a role
    if (warp == PRODUCER) {
        __syncwarp();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" :: "r"(tmem) : "memory");
    }
}

// ---- the kernels.  Two launches on two streams (tree CTAs: 2 KB of shared memory, the rest of the SM's 256 KB is L1 for the
// node records) ...
template <bool SELFPLAY>
__global__ void __launch_bounds__(SP_TREE_THREADS, 1)
k_sp_tree(const C4Dev dg, SpGlobal *G, SpParams P)
{
    __shared__ SpCtl Sm;
    sp_tree_body<SELFPLAY, false>(dg, G, P, &Sm);
}
template <typename OP, int F>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_sp_net(const unsigned char *__restrict__ image, int R, SpGlobal *G, C4Counters *ctr, SpParams P)
{
    extern __shared__ __align__(16) unsigned char smem[];
    sp_net_body<OP, F, 2, 0, 1, false>(image, R, G, ctr, P, smem, blockIdx.x);
}
// ... or ONE launch whose CTAs take a role by index (co-resident by construction: one CTA per SM, grid <= SMs; this is the
// form ncu can profile).  Every CTA then has the tower's shared memory, so the tree CTAs keep only ~28 KB (32 filters) of L1.
template <typename OP, int F, bool SELFPLAY>
__global__ void __launch_bounds__(SP_TREE_THREADS, 1)
k_sp_one(const C4Dev dg, const unsigned char *__restrict__ image, int R, SpGlobal *G, SpParams P)
{
    extern __shared__ __align__(16) unsigned char smem[];
    if ((int)blockIdx.x < P.n_tree) {
#ifndef C4_SP_STAGE_TOP
        if (P.table_entries) sp_tree_body<SELFPLAY, true>(dg, G, P, reinterpret_cast<SpCtl *>(smem));
        else
#endif
        sp_tree_body<SELFPLAY, false>(dg, G, P, reinterpret_cast<SpCtl *>(smem));
    }
    else sp_net_body<OP, F, 0, 16, 17, true>(image, R, G, dg.ctr, P, smem, blockIdx.x - (unsigned)P.n_tree);
}

// ------------------------------------------------------------------------------------------------ host side
// internal interface used by c4_search.cu
static int sp_sms()
{
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
    return sms;
}

// tower CTAs (env C4_SP_NET_CTAS overrides); the rest of the SMs run trees.  Measured on a B200 (148 SMs), cold generation,
// positions/s by tower count (profiles/README.md): 4,096 games 64: 417k, 72: 431k, 80: 421k, 88: 384k; 2,048 games 56: 291k,
// 72: 308k, 88: 294k; 1,024 games 56: 181k, 72 / 88: 185k; 256 games 72: 56k, 104: 59k; 8,192 games 56: 486k, 72: 484k --
// just under half of the SMs at every pool size.
static int sp_net_ctas(int sms, int filters)
{
    // (a 64-filter evaluation is 8x the tensor work of a 32-filter one: most SMs run towers)
    int n = getenv("C4_SP_NET_CTAS") ? atoi(getenv("C4_SP_NET_CTAS")) : (filters == 64 ? (sms * 112 + 74) / 148 : (sms * 72 + 74) / 148);
    return std::max(1, std::min(n, sms - 1));
}

struct SpDevice {
    int *h_abort = nullptr, *d_abort = nullptr;
    SpGlobal *G = nullptr;
    cudaStream_t side = nullptr, side2 = nullptr;
    cudaEvent_t ev_a = nullptr, ev_b = nullptr;
    int coresident = 0;                 // 0 = not probed yet, 1 = two kernels on two streams run side by side, -1 = they do not
    int adapt_n_net = 0;                // adaptive tower count: where the last sliced run ended (0 = no such run yet)
    int last_launches = 0;              // kernels launched by the last run
    std::mutex run;                     // one run per device at a time: the rings and answer slots are per device
};
static SpDevice g_sp_device[64];
static std::mutex g_sp_init;

__global__ void k_sp_probe_wait(int *flag, int *result)
{
    const unsigned long long t0 = fz_globaltimer();
    while (ld_vol(flag) == 0) {
        if (fz_globaltimer() - t0 > 200000000ULL) { *result = -1; return; }      // 0.2 s: the other kernel is not running
        __nanosleep(1000);
    }
    *result = 1;
}
__global__ void k_sp_probe_set(int *flag) { st_vol(flag, 1); }

// Per-device buffers of the engine (control block, answer slots, rings; mapped abort word; side streams)
static SpDevice *sp_device()
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    SpDevice &pd = g_sp_device[dev];
    std::lock_guard<std::mutex> lock(g_sp_init);
    if (pd.G) return &pd;
    const int sms = sp_sms();
    if (sms < 8) return nullptr;
    SpGlobal *G = nullptr;
    if (cudaHostAlloc((void **)&pd.h_abort, 64, cudaHostAllocMapped) != cudaSuccess) return nullptr;
    if (cudaHostGetDevicePointer((void **)&pd.d_abort, pd.h_abort, 0) != cudaSuccess) return nullptr;
    if (cudaStreamCreateWithFlags(&pd.side, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaStreamCreateWithFlags(&pd.side2, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&pd.ev_a, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&pd.ev_b, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    if (cudaMalloc((void **)&G, sp_rings_off() + (size_t)sms * SP_GMAX * 16) != cudaSuccess) return nullptr;   // rings for any tower count / pool size
    pd.G = G;
    return &pd;
}

// The two-launch form needs two kernels that wait for each other to run at the same time.  Nothing in CUDA guarantees that
// for two launches; it holds when both are launched by one process into two streams of one context and together need no more
// SMs than the device has -- but a tool that serialises launches (ncu kernel replay, compute-sanitizer,
// CUDA_LAUNCH_BLOCKING=1) breaks it.  So before its first use a 1-thread kernel waits (at most 0.2 s) for a flag set by a
// second 1-thread kernel on another stream; if the flag never arrives the engine stays with ONE launch.
static bool sp_coresident(SpDevice &pd)
{
    std::lock_guard<std::mutex> lock(g_sp_init);
    if (pd.coresident != 0) return pd.coresident == 1;
    pd.coresident = -1;
    cudaFuncAttributes fa;
    if (cudaFuncGetAttributes(&fa, k_sp_probe_wait) != cudaSuccess || cudaFuncGetAttributes(&fa, k_sp_probe_set) != cudaSuccess) return false;
    int *w = reinterpret_cast<int *>(pd.G);                               // two scratch words of the control block (no run is active)
    if (cudaMemsetAsync(w, 0, 8, pd.side) != cudaSuccess || cudaStreamSynchronize(pd.side) != cudaSuccess) return false;
    k_sp_probe_wait<<<1, 1, 0, pd.side>>>(w, w + 1);
    k_sp_probe_set<<<1, 1, 0, pd.side2>>>(w);
    int result = 0;
    if (cudaStreamSynchronize(pd.side) != cudaSuccess || cudaStreamSynchronize(pd.side2) != cudaSuccess) return false;
    if (cudaMemcpy(&result, w + 1, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return false;
    pd.coresident = result == 1 ? 1 : -1;
    if (pd.coresident < 0) fprintf(stderr, "[split] two kernels on two streams do not run side by side here (serialising tool?): one launch\n");
    return pd.coresident == 1;
}

// ---- adaptive tower count.  The best split of the SMs between trees and towers moves with the state of a generation (time profile
// in profiles/README.md: a cold generation at 4,096 games goes through a cold start with hardly any evaluations, a middle phase at
// ~81 % memo hits in which 72 saturated towers hold the trees back -- best constant count there: 80 -- and a tail at > 90 % hits
// in which 56 towers are enough and every further tree SM counts).  A constant count (72) is a compromise; the hand-made
// schedule 64 -> 80 -> 56 towers measured +5 %.  So a run is cut into slices (SpParams::slice_ns): a slice ends like any stop (tree
// warps finish the answers in flight, every game's state is in HBM), the host reads the slice's load signals and launches the
// next slice with the tower count they ask for.  Signals: boards per strip b (a tower takes what its ring holds, so b says how
// far from saturated the towers are: capacity use u = throughput(b) / throughput(NB), strip time ~ 1 + gamma b) and the share i
// of their time the tree warps found no runnable game.  Balance: evaluations asked per busy tree SM = evaluations a saturated
// tower serves, n_net' / n_tree' = n_net u / (n_tree (1 - i)).  Records do not depend on any of this (tests/test_gpu_split.py).
struct SpAdapt {
    bool on = false;
    int lo = 0, hi = 0;
    double slice_ms = 25.0;
};
// 40..96 of 148 SMs as towers, and never so many that a tree CTA would own more than SP_GC_MAX game slots
static void sp_adapt_bounds(SpAdapt &a, int max_games, int sms)
{
    a.lo = (sms * 40 + 74) / 148;
    a.hi = std::min((sms * 96 + 74) / 148, sms - (max_games + SP_GC_MAX - 1) / SP_GC_MAX);
}
static SpAdapt sp_adapt_config(const c4_net *net, int max_games, int sms, bool two)
{
    SpAdapt a;
    const char *e = getenv("C4_SP_ADAPT");                                // "0" = off, "1" = on, "<ms>" = on with this slice length
    if (e && atof(e) <= 0.0) return a;
    if (two || getenv("C4_SP_NET_CTAS") || net->F != 32 || max_games < 1024) return a;    // (measured for 32-filter networks only)
    a.on = true;
    if (e && atof(e) > 1.0) a.slice_ms = atof(e);
    sp_adapt_bounds(a, max_games, sms);
    if (a.hi < a.lo) a.on = false;
    return a;
}
static int sp_adapt_next(const SpAdapt &a, int sms, int n_net, int n_tree, const unsigned long long *sig)
{
    const double NB = SP_NB, gamma = 0.145;                               // strip time ~ T0 (1 + gamma b): 16.5k cycles at 1 board, 47k at 16
    const double b = sig[0] ? (double)sig[1] / (double)sig[0] : 0.0;
    const double u = b >= NB - 1.0 ? 1.0 : b * (1.0 + gamma * NB) / (NB * (1.0 + gamma * b));
    const double idle = (sig[2] + sig[3]) ? (double)sig[3] / (double)(sig[2] + sig[3]) : 0.0;
    const double rho = std::max(1e-3, n_net * u) / std::max(1e-3, n_tree * (1.0 - idle));
    double target = sms * rho / (1.0 + rho);
    if (target < n_net && idle > 0.05) target = n_net;                    // trees wait although the towers are not full: latency, not capacity
    target = std::max((double)n_net - 16.0, std::min((double)n_net + 16.0, target));
    int n = (int)(target / 4.0 + 0.5) * 4;
    n = std::max(a.lo, std::min(a.hi, n));
    return n;
}

// Test hook (tests/test_host_logic.py; host arithmetic only, no GPU): the tower count the controller picks after a slice with
// `n_net` towers on a device of `sms` SMs that served `boards` boards in `strips` strips while the tree warps spent
// `run_cycles` in runs and `idle_cycles` without a runnable game.
extern "C" int c4_split_adapt_next(int sms, int max_games, int n_net, unsigned long long strips, unsigned long long boards,
                                   unsigned long long run_cycles, unsigned long long idle_cycles)
{
    SpAdapt a;
    a.on = true;
    sp_adapt_bounds(a, max_games, sms);
    const unsigned long long sig[4] = {strips, boards, run_cycles, idle_cycles};
    return sp_adapt_next(a, sms, n_net, std::min(sms - n_net, max_games), sig);
}

static bool c4_split_supported(const c4_net *net, int max_games)
{
    // (a network served by the caller, c4_net_create_external, has F = 0 and no images: it runs lock-step only)
    if (!net || (net->F != 32 && net->F != 64) || !net->use_tc || !net->image_tc) return false;
    if (getenv("C4_SP_DISABLE")) return false;                            // (tests of the other engines' auto policy)
    const int sms = sp_sms();
    if (sms < 8 || max_games > SP_GMAX || max_games < 1) return false;
    const int n_tree = std::min(sms - sp_net_ctas(sms, net->F), max_games);
    if ((max_games + n_tree - 1) / n_tree > SP_GC_MAX) return false;
    if ((net->F == 32 ? sp_net_smem<32>(net->R) : sp_net_smem<64>(net->R)) > 227 * 1024) return false;
    const SpDevice *pd = sp_device();
    return pd != nullptr;
}

// ONE launch by default.  env C4_SP_LAUNCH=two: two launches on two streams, if the device runs them side by side (probe) --
// the tree CTAs then keep the SM's whole L1 (428k instead of 420k positions/s on the benchmark generation), at the price of
// relying on co-residency that CUDA does not promise.
static bool sp_two_launches(SpDevice &pd)
{
    const char *want = getenv("C4_SP_LAUNCH");
    return want && !strcmp(want, "two") && sp_coresident(pd);
}

// ... and is it the engine to use?  env C4_ENGINE = "split" / "fused" / "lockstep" forces one.  Auto: whenever it is supported --
// measured cold generations, positions/s (profiles/README.md), split / fused / lock-step: 256 games 59k / 52k / 23k; 1,024 games
// 185k / 123k / 96k; 2,048 games 308k / 201k / 181k; 4,096 games 431k / 310k / 336k; 8,192 games 486k / 315k / 427k.
bool c4_split_eligible(const c4_net *net, int max_games, long long live_games)
{
    (void)live_games;
    const char *want = getenv("C4_ENGINE");
    if (want && (!strcmp(want, "fused") || !strcmp(want, "lockstep"))) return false;
    return c4_split_supported(net, max_games);
}

// kernels launched by the last c4_split_run on the current device (one per slice; two in the two-launch form)
int c4_split_last_launches()
{
    SpDevice *pd = sp_device();
    return pd ? pd->last_launches : 0;
}

// Run the pool until every game slot is idle / done, `stop_games` games have finished (counter in d.ctr) or `stop_ms` have
// passed, and wait for it (same contract as c4_fused_run).
int c4_split_run(const C4Dev &d, const c4_net *net, int max_games, int simulations, bool selfplay,
                 unsigned long long stop_games, double stop_ms, cudaStream_t stream)
{
    const int sms = sp_sms();
    C4_REQUIRE(c4_split_supported(net, max_games), "split engine: network, pool size or device not supported");
    SpDevice &pd = *sp_device();
    std::lock_guard<std::mutex> run_lock(pd.run);
    static const bool debug = getenv("C4_FZ_DEBUG") != nullptr;
    const bool adapt_log = getenv("C4_SP_ADAPT_LOG") != nullptr;
    *reinterpret_cast<volatile int *>(pd.h_abort) = 0;
    SpParams P;
    P.n_slots = max_games;
    P.stop_games = stop_games;
    P.stop_ns = stop_ms > 0.0 ? (unsigned long long)(stop_ms * 1e6) : 0ULL;
    P.host_abort = pd.d_abort;
    P.prof = debug ? 1 : 0;
    P.batch_ns = getenv("C4_SP_BATCH_NS") ? atoi(getenv("C4_SP_BATCH_NS")) : 0;
    unsigned cap = 64;
    while ((int)cap < max_games) cap <<= 1;
    P.ring_cap = cap;
    const int smem = net->F == 32 ? sp_net_smem<32>(net->R) : sp_net_smem<64>(net->R);
    const bool two = sp_two_launches(pd);                                 // (may run the probe, which uses the control block: before the reset)
    const SpAdapt adapt = sp_adapt_config(net, max_games, sms, two);
    int n_net = sp_net_ctas(sms, net->F);
    if (adapt.on) n_net = std::max(adapt.lo, std::min(adapt.hi, pd.adapt_n_net ? pd.adapt_n_net : (sms * 64 + 74) / 148));
    const double limit_s = getenv("C4_FZ_TIMEOUT_S") ? atof(getenv("C4_FZ_TIMEOUT_S")) : 900.0;
    const auto t_call = std::chrono::steady_clock::now();
    bool asked = false;
    pd.last_launches = 0;
    for (int slice = 0;; slice++) {
        const int n_tree = std::min(sms - n_net, max_games);
        P.n_net = n_net;
        P.n_tree = n_tree;
        // time limits of this launch: what is left of the caller's limit, and the slice of the adaptive tower count
        P.slice_ns = 0ULL;
        if (stop_ms > 0.0) {
            const double left_ms = stop_ms - std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_call).count();
            if (slice > 0 && left_ms <= 0.0) break;
            P.stop_ns = (unsigned long long)(std::max(left_ms, 0.01) * 1e6);
            if (adapt.on && left_ms > adapt.slice_ms) P.slice_ns = (unsigned long long)(adapt.slice_ms * 1e6);
        } else if (adapt.on) P.slice_ns = (unsigned long long)(adapt.slice_ms * 1e6);
        P.stage_nodes = 0;
#ifdef C4_SP_STAGE_TOP
        // ONE launch: every CTA has the tower's shared memory; a tree CTA uses it for the top of its games' trees (env
        // C4_SP_STAGE=0 turns that off; C4_SP_STAGE=n caps the node records per game).  Compiled in with -DC4_SP_STAGE_TOP only:
        // measured slower than no staging (profiles/README.md, "shared-memory staging of the tree top")
        {
            const int gc_max = (max_games + n_tree - 1) / n_tree;
            const int avail = smem - (int)((sizeof(SpCtl) + 127) & ~(size_t)127);
            int nodes = std::min(avail / (gc_max * 32), std::min(512, d.blocks_per_game * C4_SLOTS)) & ~7;
            if (getenv("C4_SP_STAGE")) nodes = std::min(nodes, atoi(getenv("C4_SP_STAGE")) & ~7);
            P.stage_nodes = std::max(0, nodes);
        }
#endif
        // PUCT tables in the tree CTAs' shared memory (one-launch form only; env C4_SP_SMEM_TABLES=0/1 overrides the default)
        P.table_entries = 0;
#ifndef C4_SP_STAGE_TOP
        {
            const bool want = getenv("C4_SP_SMEM_TABLES") ? atoi(getenv("C4_SP_SMEM_TABLES")) != 0 : true;
            const size_t need = SP_TAB_OFF + (size_t)3 * 8 * SP_TAB_STRIDE;
            if (want && !two && simulations + 2 <= (int)SP_TAB_STRIDE && need <= (size_t)smem) P.table_entries = simulations + 2;
        }
#endif
        if (two) P.stage_nodes = 0;                                           // (the tree kernel of the two-launch form has no dynamic shared memory)
        // ticket counter, flags, answer slots and the rings' stamps all start from zero
        C4_CUDA(cudaMemsetAsync(pd.G, 0, sp_rings_off() + (size_t)n_net * cap * 16, stream));
        if (two) {
            auto kn = net->F == 32 ? (net->fp16 ? k_sp_net<OpFP16, 32> : k_sp_net<OpBF16, 32>) : (net->fp16 ? k_sp_net<OpFP16, 64> : k_sp_net<OpBF16, 64>);
            auto kt = selfplay ? k_sp_tree<true> : k_sp_tree<false>;
            C4_CUDA(cudaFuncSetAttribute(kn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            // Both kernels must be LOADED before the first of them starts: with lazy module loading (the CUDA 12 default) the
            // first launch of a function loads it, and that load can wait for running kernels -- here for a tower kernel that
            // itself waits for the tree kernel: a deadlock, and it was the first thing the bring-up hit.
            {
                cudaFuncAttributes fa;
                C4_CUDA(cudaFuncGetAttributes(&fa, kn));
                C4_CUDA(cudaFuncGetAttributes(&fa, kt));
            }
            C4_CUDA(cudaEventRecord(pd.ev_a, stream));
            C4_CUDA(cudaStreamWaitEvent(pd.side, pd.ev_a, 0));
            kn<<<n_net, TC_THREADS, smem, pd.side>>>((const unsigned char *)net->image_tc, net->R, pd.G, d.ctr, P);
            C4_CUDA(cudaGetLastError());
            kt<<<n_tree, SP_TREE_THREADS, 0, stream>>>(d, pd.G, P);
            C4_CUDA(cudaGetLastError());
            C4_CUDA(cudaEventRecord(pd.ev_b, pd.side));
            C4_CUDA(cudaStreamWaitEvent(stream, pd.ev_b, 0));
            pd.last_launches += 2;
        } else {
            void (*k1)(const C4Dev, const unsigned char *, int, SpGlobal *, SpParams);
            if (net->F == 32) k1 = selfplay ? (net->fp16 ? k_sp_one<OpFP16, 32, true> : k_sp_one<OpBF16, 32, true>)
                                            : (net->fp16 ? k_sp_one<OpFP16, 32, false> : k_sp_one<OpBF16, 32, false>);
            else k1 = selfplay ? (net->fp16 ? k_sp_one<OpFP16, 64, true> : k_sp_one<OpBF16, 64, true>)
                               : (net->fp16 ? k_sp_one<OpFP16, 64, false> : k_sp_one<OpBF16, 64, false>);
            C4_CUDA(cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            k1<<<n_tree + n_net, SP_TREE_THREADS, smem, stream>>>(d, (const unsigned char *)net->image_tc, net->R, pd.G, P);
            C4_CUDA(cudaGetLastError());
            pd.last_launches += 1;
        }
        const auto t0 = std::chrono::steady_clock::now();
        for (long long it = 0;; it++) {
            cudaError_t q = cudaStreamQuery(stream);
            if (q == cudaSuccess) break;
            if (q != cudaErrorNotReady) { C4_CUDA(q); }
            const double el = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_call).count();
            if (!asked && el > limit_s) { *reinterpret_cast<volatile int *>(pd.h_abort) = 1; asked = true; }
            if (asked && el > limit_s + 5.0) {
                fprintf(stderr, "[split] the launches did not end %.0f s after the abort request; giving up\n", 5.0);
                fflush(stderr);
                _exit(86);
            }
            if (it > 2000) std::this_thread::sleep_for(std::chrono::microseconds(
                std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > 1.0 ? 2000 : 50));
        }
        if (debug) {
            unsigned long long h[32];
            C4_CUDA(cudaMemcpy(h, pd.G->prof, sizeof(h), cudaMemcpyDeviceToHost));
            const double ns = (double)std::max(1ULL, h[0]), nr = (double)std::max(1ULL, h[8]);
            fprintf(stderr, "[split prof] %d tree CTAs + %d tower CTAs, %s | strips %llu boards/strip %.2f | tower cycles per strip: idle %.0f busy %.0f "
                            "(busy share %.2f) = claim %.0f + input %.0f + layers %.0f + heads %.0f | tree runs %llu cycles/run %.0f tree-warp idle share %.2f\n",
                    n_tree, n_net, two ? "two launches" : "one launch", h[0], h[1] / ns, h[2] / ns, h[3] / ns, h[3] / (double)std::max(1ULL, h[2] + h[3]),
                    h[4] / ns, h[5] / ns, h[6] / ns, h[7] / ns, h[8], h[9] / nr, h[10] / (double)std::max(1ULL, h[9] + h[10]));
        }
        if (!adapt.on || asked) break;
        // the slice's flags and load signals; a launch that no CTA ended for its slice is the last one
        SpHeader hd;
        C4_CUDA(cudaMemcpy(&hd, pd.G, sizeof(hd), cudaMemcpyDeviceToHost));
        if (!hd.sliced || hd.abort) break;
        const unsigned long long *sig = hd.sig;
        const int n_prev = n_net;
        n_net = sp_adapt_next(adapt, sms, n_net, n_tree, sig);
        if (adapt_log)
            fprintf(stderr, "[split adapt] slice %d: %d towers, boards/strip %.2f, tree-warp idle share %.3f -> %d towers\n", slice, n_prev,
                    sig[0] ? (double)sig[1] / (double)sig[0] : 0.0, (sig[2] + sig[3]) ? (double)sig[3] / (double)(sig[2] + sig[3]) : 0.0, n_net);
        pd.adapt_n_net = n_net;
        C4_REQUIRE(slice < (1 << 24), "split engine: did not terminate");
    }
    if (asked) { c4_set_error("split engine: host deadline passed (C4_FZ_TIMEOUT_S); the launches were aborted"); return -4; }
    return 0;
}
