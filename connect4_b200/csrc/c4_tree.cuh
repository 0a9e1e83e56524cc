// c4_tree.cuh -- device pieces of the warp-per-game MCTS engine (select / expand / evaluate / backup, the self-play
// state machine, the evaluation memo), shared by the lock-step pass kernel (c4_search.cu) and the fused persistent
// engine (c4_fused.cu).  Reference semantics cited per function (paths relative to the reference root).
#pragma once
#include <math.h>

#include "c4_common.cuh"

unsigned long long c4_net_uid(const c4_net *net);     // c4_net.cu (internal)
int c4_net_filters(const c4_net *net);
int c4_net_device(const c4_net *net);
bool c4_net_external(const c4_net *net);              // served by the caller (c4_net_create_external)

enum { ST_IDLE = 0, ST_READY = 1, ST_WAIT = 2, ST_DONE = 3, ST_NEWROOT = 4,
       ST_WAITMEMO = 7 };     // the leaf is being evaluated for ANOTHER game: re-probe the memo instead of asking again
#define PATH_CAP 48
#define MAX_PLY 42
#define FULL 0xffffffffu

struct C4Counters {
    unsigned long long next_game;       // next local game number to seed
    unsigned long long games_finished;
    unsigned long long n_records;
    unsigned long long n_done;          // stand-alone searches finished
    unsigned long long overflow;        // records dropped (records_out too small)
    int leaf_count[2][2];               // [pool][parity] ping-pong leaf batch counters
    int busy_count[2][2];               // ... leaves + games that wait for another game's leaf (the pass's stop rule)
    int engine_error;                   // fused engine: non-zero = the kernel gave up (watchdog), see c4_fused.cu
    int net_nonfinite;                  // a network answer was not finite (fp16 operand overflow): the call fails loudly
    int pad[32 - 20];
    int stop_flag[2][2];                // [pool][parity], on its own 128-byte line: set by the warp whose request makes
                                        // the batch reach the pass's stop count, polled (read-only) by the running warps
    int pad2[28];
};
static_assert(sizeof(C4Counters) == 256, "counters: two 128-byte lines");
static_assert(sizeof(c4_record) == 64, "position record must be 64 bytes");

struct C4Dev {
    C4Node *pool;
    int blocks_per_game;
    const double *pbc;                  // pbc[N] = log((N + base + 1)/base) + init
    const double *sqt;                  // sqt[N] = sqrt(N)  (correctly rounded, = math.sqrt)
    const double *rcp;                  // rcp[m] = 1.0 / m  (correctly rounded); rcp[0] unused
    int fastdiv;                        // sqrt(N)/(n+1) by reciprocal table + two FMAs, verified exhaustively on the host
    int sims;
    double frac, one_minus_frac;
    float one_minus_frac_f;
    double alpha;
    int noise_on;                       // alpha != 0 && frac != 0   (oinkoink/mcts.py:174)
    int n_sampling;
    int rng_mode;
    int rng_record;
    u64 seed;
    double *noise;                      // [G][42][7]
    double *uniform;                    // [G][42]
    // per game slot
    u64 *root_c0, *root_c1;
    int *status, *sims_done, *n_blocks, *pending_node, *pending_slot, *path_len, *ply;
    u64 *pend_c0, *pend_c1;
    uint32_t *path;                     // [G][PATH_CAP]
    long long *game_id;
    unsigned long long *stat_evals, *stat_positions;
    c4_record *staging;                 // [G][42]
    // leaf batch
    u64 *leaf_c0, *leaf_c1;
    int *leaf_game;
    // evaluation memo (the reference's Evaluator.position_table, oinkoink/evaluators.py:18-25): direct-mapped table of
    // 64-byte entries {c0, c1, out[8], check64}; looked up before a leaf is sent to the network, filled when the
    // network's answer is consumed.  Pure cache: a hit returns bit-identical numbers to a network evaluation.
    uint32_t *memo;                     // [memo_mask + 1][16] words, or nullptr
    uint32_t memo_mask;
    int memo_dedup;                     // a game that misses claims the entry (PENDING tag): later askers wait for its answer
    uint32_t memo_epoch;                // mixed into the PENDING tags: a new pool / search batch never waits on the tags of an
                                        // abandoned one (their owners are gone and would never answer)
    unsigned long long *stat_hits;      // [G]
    // evaluator answers
    const float *net_out;               // [G][8] {prior[7], value}
    const double *ext_value;            // [G]
    const void *ext_prior;              // [G][7] fp64 or fp32
    int ext_prior_dtype;
    // self-play control
    C4Counters *ctr;
    long long n_games_target;
    long long game_id_base, game_id_stride;
    const u64 *start_c0, *start_c1;
    c4_record *records_out;
    long long max_records;
};

// ------------------------------------------------------------------------------------------------ device pieces
__device__ __forceinline__ C4NodeA ld_a(const C4Node *n)
{
    C4NodeA a;
    uint4 v = *reinterpret_cast<const uint4 *>(&n->a);
    a.vsum = __hiloint2double((int)v.y, (int)v.x);
    a.visits = v.z; a.meta = v.w;
    return a;
}
__device__ __forceinline__ C4NodeB ld_b(const C4Node *n)
{
    C4NodeB b;
    uint4 v = *reinterpret_cast<const uint4 *>(&n->b);
    b.prior = __hiloint2double((int)v.y, (int)v.x);
    b.vsel = __hiloint2double((int)v.w, (int)v.z);
    return b;
}
__device__ __forceinline__ void st_a(C4Node *n, double vsum, uint32_t visits, uint32_t meta)
{
    uint4 v;
    v.x = (uint32_t)__double2loint(vsum); v.y = (uint32_t)__double2hiint(vsum); v.z = visits; v.w = meta;
    *reinterpret_cast<uint4 *>(&n->a) = v;
}
__device__ __forceinline__ void st_b(C4Node *n, double prior, double vsel)
{
    uint4 v;
    v.x = (uint32_t)__double2loint(prior); v.y = (uint32_t)__double2hiint(prior);
    v.z = (uint32_t)__double2loint(vsel); v.w = (uint32_t)__double2hiint(vsel);
    *reinterpret_cast<uint4 *>(&n->b) = v;
}
// block header (slot 7), second half of B: number of children and the parent's node id
__device__ __forceinline__ double pack_header(uint32_t n_children, uint32_t parent)
{
    return __hiloint2double((int)parent, (int)n_children);
}
__device__ __forceinline__ uint32_t header_children(const C4NodeB &b) { return (uint32_t)__double2loint(b.vsel); }
__device__ __forceinline__ uint32_t header_parent(const C4NodeB &b) { return (uint32_t)__double2hiint(b.vsel); }

// sequential sum of the 7 per-lane values, left to right from 0.0 (numpy's add.reduce for n < 8)
__device__ __forceinline__ double seq_sum7(double v)
{
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 7; i++) s = __dadd_rn(s, shfl_d(v, i));
    return s;
}
__device__ __forceinline__ float seq_sum7f(float v)
{
    float s = 0.0f;
#pragma unroll
    for (int i = 0; i < 7; i++) s = __fadd_rn(s, __shfl_sync(FULL, v, i));
    return s;
}

// gamma(alpha, 1) variate (Marsaglia-Tsang, with the U^(1/alpha) boost for alpha < 1); replaces np.random.gamma of
// oinkoink/mcts.py:175 -- distributionally, not draw-for-draw (the reference's global MT19937 stream is not
// reproducible across threads anyway, SURVEY.md section 7).
static __device__ double c4_gamma(Philox &ph, double alpha)
{
    double a = alpha < 1.0 ? alpha + 1.0 : alpha;
    double d = a - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
    double x, v, u3, u4;
    for (int it = 0; it < 64; it++) {
        uint32_t r[4], q[4];
        ph.next(r);
        ph.next(q);
        double u1 = ph.uniform_from(r[0], r[1]), u2 = ph.uniform_from(r[2], r[3]);
        u3 = ph.uniform_from(q[0], q[1]);
        u4 = ph.uniform_from(q[2], q[3]);
        x = sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
        v = 1.0 + c * x;
        if (v <= 0.0) continue;
        v = v * v * v;
        if (log(u3) < 0.5 * x * x + d - d * v + d * log(v)) break;
    }
    double g = d * v;
    if (alpha < 1.0) g *= pow(u4, 1.0 / alpha);
    return g;
}

__device__ __forceinline__ u64 memo_mix(u64 x)
{
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
    return x;
}
__device__ __forceinline__ uint32_t memo_index(u64 c0, u64 c1, uint32_t mask)
{
    return (uint32_t)(memo_mix(c0 * 0x9E3779B97F4A7C15ULL ^ c1 * 0xC2B2AE3D27D4EB4FULL) >> 20) & mask;
}
// 64-bit checksum over key and payload: a torn entry (two warps writing the same slot) reads as a miss
__device__ __forceinline__ u64 memo_check(u64 c0, u64 c1, uint32_t payload_xor_rot)
{
    return memo_mix(c0 ^ memo_mix(c1 + 0x632BE59BD9B4E019ULL) ^ ((u64)payload_xor_rot * 0xD6E8FEB86659FD93ULL)) | 1ULL;
}
// lanes 0..7 hold the payload words (out[lane] bits); returns a warp-uniform digest of them
__device__ __forceinline__ uint32_t memo_payload_digest(uint32_t w, int lane)
{
    uint32_t x = (lane < 8) ? __funnelshift_l(w, w, 3 * lane) + (uint32_t)lane * 0x9E3779B9u : 0u;
#pragma unroll
    for (int off = 4; off >= 1; off >>= 1) x ^= __shfl_xor_sync(FULL, x, off);
    return __shfl_sync(FULL, x, 0);
}
// store {c0, c1, out[8]} (lane l < 8 holds out[l]); one coalesced 64-byte store.
// INTENTIONAL RACE (1 of 3 in the lock-step engine): warps of different games may write the same slot at the same time, and a
// reader may see a half-written entry.  No lock: the 64-bit checksum over key AND payload turns every torn or mixed entry
// into a miss, and two writers of the same key write identical bytes.
__device__ __forceinline__ void memo_insert(const C4Dev &d, u64 c0, u64 c1, float out_lane, int lane)
{
    const uint32_t w = __float_as_uint(out_lane);
    const u64 chk = memo_check(c0, c1, memo_payload_digest(w, lane));
    uint32_t *e = d.memo + (size_t)memo_index(c0, c1, d.memo_mask) * 16;
    const uint32_t pw = __shfl_sync(FULL, w, (lane - 4) & 31);         // lane 4 + l <- out[l]
    uint32_t v = 0u;
    if (lane < 2) v = (uint32_t)(c0 >> (32 * lane));
    else if (lane < 4) v = (uint32_t)(c1 >> (32 * (lane - 2)));
    else if (lane < 12) v = pw;
    else if (lane < 14) v = (uint32_t)(chk >> (32 * (lane - 12)));
    if (lane < 16) e[lane] = v;
}
// true on a hit; out_lane (lanes 0..7) receives out[lane]
__device__ __forceinline__ bool memo_lookup(const C4Dev &d, u64 c0, u64 c1, float &out_lane, int lane)
{
    const uint32_t *e = d.memo + (size_t)memo_index(c0, c1, d.memo_mask) * 16;
    const uint32_t v = (lane < 16) ? __ldcg(e + lane) : 0u;
    const u64 k0 = (u64)__shfl_sync(FULL, v, 0) | ((u64)__shfl_sync(FULL, v, 1) << 32);
    const u64 k1 = (u64)__shfl_sync(FULL, v, 2) | ((u64)__shfl_sync(FULL, v, 3) << 32);
    const u64 chk = (u64)__shfl_sync(FULL, v, 12) | ((u64)__shfl_sync(FULL, v, 13) << 32);
    const uint32_t w = __shfl_sync(FULL, v, (lane + 4) & 31);          // lane l < 8 <- word 4 + l
    const uint32_t dig = memo_payload_digest(w, lane);
    out_lane = __uint_as_float(w);
    return k0 == c0 && k1 == c1 && chk == memo_check(c0, c1, dig);
}

// ---- de-duplication of evaluations in flight.  Measured on the benchmark generation (tools/memo_dups.py): 1.45 network
// evaluations per DISTINCT position (2.3 in the first 256 games) -- thousands of games walk the same openings at the same
// time, and all of them miss the memo until the first answer is in.  So the game that misses first CLAIMS the entry: it
// swaps a PENDING tag (a function of the key, bit 0 clear -- checksums have bit 0 set, empty entries are 0) into the
// entry's check word with a 64-bit CAS and asks the network; every later asker finds the tag, parks its leaf
// (ST_WAITMEMO) and re-probes until the owner's answer has replaced the tag.  Pure work elimination: a waiter ends up with
// the bit-identical numbers it would have got from its own evaluation.  No dead end: whoever wins a claim evaluates and
// inserts; if a colliding key overwrites the tag or the entry, the waiters simply miss and claim again; the tags carry the
// epoch of the pool that wrote them, so the tags of an abandoned pool (a stream that was stopped and reset: their owners
// will never answer) read as plain misses; and a waiter that has looked WAITMEMO_PATIENCE times asks for itself.
#define WAITMEMO_PATIENCE 64
enum { MEMO_MISS = 0, MEMO_HIT = 1, MEMO_PENDING = 2 };
__device__ __forceinline__ u64 memo_pending_tag(uint32_t epoch, u64 c0, u64 c1)
{
    return (memo_mix(c1 * 0x9E3779B97F4A7C15ULL ^ memo_mix(c0 + 0xD6E8FEB86659FD93ULL + ((u64)epoch << 50))) & ~3ULL) | 2ULL;
}
__device__ __forceinline__ u64 memo_pending_tag(const C4Dev &d, u64 c0, u64 c1) { return memo_pending_tag(d.memo_epoch, c0, c1); }
// like memo_lookup, three-valued; `seen` = the check word that was read (the CAS of memo_claim expects it)
__device__ __forceinline__ int memo_probe(const C4Dev &d, u64 c0, u64 c1, float &out_lane, int lane, u64 &seen)
{
    const uint32_t *e = d.memo + (size_t)memo_index(c0, c1, d.memo_mask) * 16;
    const uint32_t v = (lane < 16) ? __ldcg(e + lane) : 0u;
    const u64 k0 = (u64)__shfl_sync(FULL, v, 0) | ((u64)__shfl_sync(FULL, v, 1) << 32);
    const u64 k1 = (u64)__shfl_sync(FULL, v, 2) | ((u64)__shfl_sync(FULL, v, 3) << 32);
    const u64 chk = (u64)__shfl_sync(FULL, v, 12) | ((u64)__shfl_sync(FULL, v, 13) << 32);
    const uint32_t w = __shfl_sync(FULL, v, (lane + 4) & 31);
    const uint32_t dig = memo_payload_digest(w, lane);
    out_lane = __uint_as_float(w);
    seen = chk;
    if (k0 == c0 && k1 == c1 && chk == memo_check(c0, c1, dig)) return MEMO_HIT;
#ifdef C4_NO_DEDUP_BUILD
    return MEMO_MISS;
#else
    return (d.memo_dedup && chk == memo_pending_tag(d, c0, c1)) ? MEMO_PENDING : MEMO_MISS;
#endif
}
// after a MEMO_MISS: true = this game evaluates the position (it won the claim, or the slot is contended by another key
// and nothing is marked), false = another game claimed the same position a moment ago: wait for its answer
__device__ __forceinline__ bool memo_claim(const C4Dev &d, u64 c0, u64 c1, u64 seen, int lane)
{
    int own = 1;
#ifdef C4_NO_DEDUP_BUILD
    return true;
#endif
    if (lane == 0) {
        unsigned long long *chk = reinterpret_cast<unsigned long long *>(d.memo + (size_t)memo_index(c0, c1, d.memo_mask) * 16 + 12);
        const u64 tag = memo_pending_tag(d, c0, c1);
        const u64 old = atomicCAS(chk, (unsigned long long)seen, (unsigned long long)tag);
        own = !(old != seen && old == tag);
    }
    return __shfl_sync(FULL, own, 0) != 0;
}

struct Game {
    C4Node *gp;          // this game's node pool
    int g;               // slot
    int lane;
    int n_blocks;
    int sims_done;
    u64 c0, c1;          // root board
    int age;             // root age
    static constexpr bool SMEM_TABLES = false;   // the PUCT tables are read from HBM (through L1) via C4Dev::pbc / sqt / rcp
    static constexpr bool PREFETCH = true;       // descend() pulls every child's own block towards L2 while the warp decides
    // node accessors (node i of this game): every read / write of the tree goes through these
    __device__ __forceinline__ C4NodeA lda(uint32_t i) const { return ld_a(gp + i); }
    __device__ __forceinline__ C4NodeB ldb(uint32_t i) const { return ld_b(gp + i); }
    // both halves of node i (what select reads of a child): two 128-bit loads through L1.  Measured in the split engine and not
    // kept (profiles/README.md): ONE 256-bit load (`ld.global.v4.u64` = LDG.E.ENL2.256 on sm_100a) 446.7k against 450k positions/s,
    // two `ld.global.cg` loads 442k -- the 28 KB of L1 the tree CTAs have left still serve 37-41 % of the node reads
    __device__ __forceinline__ void ldab(uint32_t i, C4NodeA &a, C4NodeB &b) const { a = ld_a(gp + i); b = ld_b(gp + i); }
    __device__ __forceinline__ void sta(uint32_t i, double vsum, uint32_t visits, uint32_t meta) const { st_a(gp + i, vsum, visits, meta); }
    __device__ __forceinline__ void stb(uint32_t i, double prior, double vsel) const { st_b(gp + i, prior, vsel); }
    __device__ __forceinline__ void st_vsel(uint32_t i, double vsel) const { gp[i].b.vsel = vsel; }
    __device__ __forceinline__ bool in_hbm(uint32_t) const { return true; }
};
// A game of a CTA that keeps the three PUCT tables (C4Dev::pbc / sqt / rcp) in its DYNAMIC shared memory, table k at byte
// OFF + k * 8 * STRIDE: compile-time offsets from the dynamic shared-memory base, so a table read is one LDS with an immediate
// and costs no pointer register (three generic pointers instead spilled the 64-register tree warps).  Used by the tree CTAs
// of the one-launch split engine (c4_split.cu), which carry the tower's shared memory and have little L1.
// (no speculative prefetch of the grandchildren's blocks: tuned in round 1 for the lock-step pass, where a warp's lines have to come
//  back from L2 / HBM at every pass; in the persistent split engine a game stays on its SM and the 14 prefetch instructions per level
//  only take issue slots and L1 / L2 request bandwidth from the 31 tree warps: 434k -> 449k positions/s without them)
struct GameNP : Game { static constexpr bool PREFETCH = false; };
template <uint32_t OFF, uint32_t STRIDE>
struct GameTab : GameNP {
    static constexpr bool SMEM_TABLES = true;
    static __device__ __forceinline__ const double *table(int k)
    {
        extern __shared__ __align__(16) unsigned char c4_dyn_smem[];
        return reinterpret_cast<const double *>(c4_dyn_smem + OFF) + (size_t)k * STRIDE;
    }
};
// A game whose FIRST `sp_nodes` nodes (the blocks created first = the top of the tree, the records every simulation reads
// and writes) live in shared memory for the length of a persistent launch ("shared-memory staging of the hot top of each
// tree"; c4_split.cu copies them in at launch entry and back at exit).  Same functions, other addresses: the select /
// expand / backup code below is templated on the game type, and with `Game` it compiles to what it was.  The shared copy
// is addressed with 32-bit .shared addresses and explicit ld.shared / st.shared: a generic pointer costs a 64-bit select
// plus the window-base arithmetic (S2UR) at every access, which measured slower than no staging at all.
struct GameS : Game {
    uint32_t sp32;       // .shared address of the copy of nodes 0 .. sp_nodes - 1
    uint32_t sp_nodes;
    // 16 bytes of node i (half 0 = A, half 1 = B).  Both addresses are computed up front and the two loads are predicated:
    // as a branch, the compiler sank the 64-bit address arithmetic (with its constant-bank loads) under the predicate, onto the
    // dependent chain of the descent
    __device__ __forceinline__ uint4 ld16(uint32_t i, uint32_t half) const
    {
        const char *pg = reinterpret_cast<const char *>(gp + i) + half * 16u;
        const uint32_t ps = sp32 + i * 32u + half * 16u;
        uint4 v;
        asm volatile("{\n\t.reg .pred p;\n\tsetp.lt.u32 p, %6, %7;\n\t"
                     "@p ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];\n\t"
                     "@!p ld.global.v4.u32 {%0,%1,%2,%3}, [%5];\n\t}"
                     : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(ps), "l"(pg), "r"(i), "r"(sp_nodes) : "memory");
        return v;
    }
    __device__ __forceinline__ C4NodeA lda(uint32_t i) const
    {
        const uint4 v = ld16(i, 0u);
        C4NodeA a;
        a.vsum = __hiloint2double((int)v.y, (int)v.x); a.visits = v.z; a.meta = v.w;
        return a;
    }
    __device__ __forceinline__ void ldab(uint32_t i, C4NodeA &a, C4NodeB &b) const { a = lda(i); b = ldb(i); }
    __device__ __forceinline__ C4NodeB ldb(uint32_t i) const
    {
        const uint4 v = ld16(i, 1u);
        C4NodeB b;
        b.prior = __hiloint2double((int)v.y, (int)v.x); b.vsel = __hiloint2double((int)v.w, (int)v.z);
        return b;
    }
    __device__ __forceinline__ void sta(uint32_t i, double vsum, uint32_t visits, uint32_t meta) const
    {
        if (i >= sp_nodes) { st_a(gp + i, vsum, visits, meta); return; }
        asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" :: "r"(sp32 + i * 32u), "r"((uint32_t)__double2loint(vsum)),
                     "r"((uint32_t)__double2hiint(vsum)), "r"(visits), "r"(meta) : "memory");
    }
    __device__ __forceinline__ void stb(uint32_t i, double prior, double vsel) const
    {
        if (i >= sp_nodes) { st_b(gp + i, prior, vsel); return; }
        asm volatile("st.shared.v4.u32 [%0+16], {%1,%2,%3,%4};" :: "r"(sp32 + i * 32u), "r"((uint32_t)__double2loint(prior)),
                     "r"((uint32_t)__double2hiint(prior)), "r"((uint32_t)__double2loint(vsel)), "r"((uint32_t)__double2hiint(vsel)) : "memory");
    }
    __device__ __forceinline__ void st_vsel(uint32_t i, double vsel) const
    {
        if (i >= sp_nodes) { gp[i].b.vsel = vsel; return; }
        asm volatile("st.shared.f64 [%0+24], %1;" :: "r"(sp32 + i * 32u), "d"(vsel) : "memory");
    }
    __device__ __forceinline__ bool in_hbm(uint32_t block) const { return block * C4_SLOTS >= sp_nodes; }
};

// Evaluate node `node` (board c0,c1 at `age`): store the value, normalise the prior over the legal moves in its own
// dtype (oinkoink/mcts.py:129-135,197-202), optionally mix root noise (mcts.py:171-181) and create the child block
// (oinkoink/tree.py:119-132 -- one child per legal move, each with its terminal result).
// p64 / p32: lane c (<7) holds the raw prior of column c.
template <bool F32, class GAME>
__device__ __forceinline__ void apply_eval(const C4Dev &d, GAME &G, uint32_t node, u64 c0, u64 c1, int age, double value,
                                           double p64, float p32, bool is_root, int ply)
{
    const int lane = G.lane;
    const int legal = c4_legal_mask(c0, c1);
    const bool mine = lane < 7 && ((legal >> lane) & 1);
    double p;
    float pf = 0.f;
    if (F32) {
        pf = (lane < 7) ? p32 : 0.f;
        if (legal != 127 && !mine) pf = 0.f;
        float s = seq_sum7f(pf);
        pf = __fdiv_rn(pf, s);
        p = (double)pf;
    } else {
        p = (lane < 7) ? p64 : 0.0;
        if (legal != 127 && !mine) p = 0.0;
        double s = seq_sum7(p);
        p = __ddiv_rn(p, s);
    }
    if (is_root && d.noise_on) {
        double nz = 0.0;
        if (d.rng_mode == C4_RNG_PHILOX) {
            if (lane < 7) {
                Philox ph(d.seed, (u64)d.game_id[G.g], (u64)(ply * 8 + lane));
                nz = c4_gamma(ph, d.alpha);
            }
            if (d.rng_record && d.noise && lane < 7) d.noise[((size_t)G.g * MAX_PLY + ply) * 7 + lane] = nz;
        } else if (d.rng_mode == C4_RNG_INJECTED) {
            if (lane < 7) nz = d.noise[((size_t)G.g * MAX_PLY + ply) * 7 + lane];
        }
        if (d.rng_mode != C4_RNG_NONE) {
            __syncwarp();
            if (legal != 127 && !mine) nz = 0.0;
            double s = seq_sum7(nz);
            nz = __ddiv_rn(nz, s);
            // prior * (1 - frac) + noise * frac ; a float32 prior times the python float stays float32
            double a = F32 ? (double)__fmul_rn(pf, d.one_minus_frac_f) : __dmul_rn(p, d.one_minus_frac);
            p = __dadd_rn(a, __dmul_rn(nz, d.frac));
        }
    }
    const uint32_t blk = (uint32_t)G.n_blocks;
    C4_DEV_ASSERT((int)blk < d.blocks_per_game && node < blk * C4_SLOTS);
    G.n_blocks++;
    const uint32_t slot = blk * C4_SLOTS + (uint32_t)lane;
    if (lane < 7) {
        int res = C4_RES_NONE;
        if (mine) { u64 a = c0, b = c1; res = c4_drop(a, b, age, lane); }
        const uint32_t m = c4_make_meta(mine, res);
        G.sta(slot, 0.0, 0u, m);
        // a terminal child is worth its result to the mover here; an unvisited one 0.0 ("assume lost", tree.py:42-44)
        G.stb(slot, mine ? p : 0.0, (m & C4_META_TERMINAL) ? c4_side_value(c4_meta_value(m), age) : 0.0);
    } else if (lane == 7) {
        G.sta(slot, value, 0u, 0u);                                    // block header: position value, #children, parent id
        G.stb(slot, 0.0, pack_header((uint32_t)__popc(legal), node));
    }
    if (lane == 0) {
        const double vs = __dadd_rn(0.0, value);                      // SearchEvaluation(): 0.0 + value, count 1
        G.sta(node, vs, 1u, C4_META_EXISTS | (blk << C4_META_CB_SHIFT));
        if (node != 0u) G.st_vsel(node, c4_side_value(vs, age - 1));       // mean of one visit, seen by the parent's mover
    }
    __syncwarp();
}

// add `value` to one path node and refresh the side-relative mean select reads (depth = its distance from the root)
template <class GAME>
__device__ __forceinline__ void backup_node(const GAME &G, uint32_t id, int depth, double value)
{
    C4NodeA a = G.lda(id);
    const double vs = __dadd_rn(a.vsum, value);
    const uint32_t vis = a.visits + 1u;
    G.sta(id, vs, vis, a.meta);
    // float(search_value) = value_sum / visit_count (mcts.py:56-57), flipped for the mover at the PARENT (age + depth - 1);
    // a terminal node keeps its result (NodeData.absolute_value, tree.py:27-38); the root is never selected
    if (depth > 0 && !(a.meta & C4_META_TERMINAL))
        G.st_vsel(id, c4_side_value(__ddiv_rn(vs, (double)vis), G.age + depth - 1));
}
// add `value` to the first `count` path nodes (lane i owns path entry i / i+32): oinkoink/mcts.py:164-168
template <class GAME>
__device__ __forceinline__ void backup(GAME &G, uint32_t path_lo, uint32_t path_hi, int count, double value)
{
    if (G.lane < count) backup_node(G, path_lo, G.lane, value);
    if (G.lane + 32 < count) backup_node(G, path_hi, G.lane + 32, value);
    __syncwarp();
}

struct Leaf {
    uint32_t node;
    uint32_t meta;
    u64 c0, c1;
    int age;
    int depth;            // number of moves below the root; path has depth+1 entries
    uint32_t path_lo, path_hi;
};

// order-preserving map of a finite double to an unsigned 64-bit key (+0.0 and -0.0 share a key)
__device__ __forceinline__ u64 score_key(double x)
{
    u64 b = (u64)__double_as_longlong(x);
    if ((b << 1) == 0ULL) b = 0ULL;
    return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}

// One descent from the root to a leaf: oinkoink/mcts.py:108-116 (the `while node.children` loop plus the
// expand-then-select step, merged by eager expansion) with select_child / ucb_score (mcts.py:138-161).
// The per-level dependent chain is what bounds the tree pass (profiles/README.md), so it is kept short:
//   load {A,B} of the own child -> sqrt(N)/(n+1) -> two multiplies, one add -> 64-bit key -> two REDUX.MAX + one vote.
template <class GAME>
__device__ __forceinline__ Leaf descend(const C4Dev &d, const GAME &G)
{
    const int lane = G.lane;
    Leaf L;
    L.c0 = G.c0; L.c1 = G.c1; L.age = G.age; L.depth = 0;
    L.path_lo = 0u; L.path_hi = 0u; L.node = 0u;
    C4NodeA ra = G.lda(0u);
    uint32_t visits = ra.visits, meta = ra.meta;
    while (!(meta & C4_META_TERMINAL) && visits > 0u) {
        const uint32_t blk = c4_meta_child_block(meta);
        C4_DEV_ASSERT(blk > 0u && (int)blk < G.n_blocks && L.depth < PATH_CAP - 1);
        const uint32_t cn = blk * C4_SLOTS + (uint32_t)(lane & 7);
        C4NodeA a;
        C4NodeB b;
        G.ldab(cn, a, b);
        // exploration factor of the parent: log((N+base+1)/base)+init and sqrt(N) from host-built tables (glibc log / sqrt)
        double pbc, sq;
        if constexpr (GAME::SMEM_TABLES) { pbc = GAME::table(0)[visits]; sq = GAME::table(1)[visits]; }
        else { pbc = d.pbc[visits]; sq = d.sqt[visits]; }
        const bool exists = (lane < 7) && (a.meta & C4_META_EXISTS);
        // speculative prefetch: every lane pulls ITS child's block (two 128-byte lines) towards L2 while the warp decides;
        // HBM bandwidth is nowhere near a limit for this kernel (profiles/README.md)
        if (GAME::PREFETCH && exists && c4_meta_child_block(a.meta) != 0u && G.in_hbm(c4_meta_child_block(a.meta))) {
            const char *pf = reinterpret_cast<const char *>(G.gp + (size_t)c4_meta_child_block(a.meta) * C4_SLOTS);
            asm volatile("prefetch.global.L2 [%0];" :: "l"(pf));
            asm volatile("prefetch.global.L2 [%0];" :: "l"(pf + 128));
        }
        // ucb_score: pb_c = (log(..)+init) * (sqrt(N)/(n+1)); score = pb_c*prior + value   (two roundings, no FMA)
        const double den = (double)(a.visits + 1u);
        double q;
        if (d.fastdiv) {
            // correctly rounded sqrt(N)/(n+1) from the correctly rounded reciprocal and two FMAs (Markstein's
            // sequence); upload_config checked it against IEEE division for EVERY (N, n) pair this context can meet
            double y;
            if constexpr (GAME::SMEM_TABLES) y = GAME::table(2)[a.visits + 1u]; else y = d.rcp[a.visits + 1u];
            const double q0 = __dmul_rn(sq, y);
            q = __fma_rn(__fma_rn(-den, q0, sq), y, q0);
        } else {
            q = __ddiv_rn(sq, den);
        }
        const double score = __dadd_rn(__dmul_rn(__dmul_rn(pbc, q), b.prior), b.vsel);
        // argmax over (score, column); equal scores -> highest column (Node.__gt__ on names, tree.py:11-15)
        const u64 key = exists ? score_key(score) : 0ULL;
        const uint32_t hi = (uint32_t)(key >> 32), lo = (uint32_t)key;
        const uint32_t mhi = __reduce_max_sync(FULL, hi);
        const bool cand = exists && hi == mhi;
        const uint32_t mlo = __reduce_max_sync(FULL, cand ? lo : 0u);
        const unsigned win = __ballot_sync(FULL, cand && lo == mlo);
        const int col = 31 - __clz((int)win);
        C4_DEV_ASSERT(win != 0u && col < 7);
        visits = __shfl_sync(FULL, a.visits, col);
        meta = __shfl_sync(FULL, a.meta, col);
        // replay the move on the register-resident board
        u64 bit = 1ULL << c4_drop_bit(L.c0 | L.c1, col);
        if (L.age & 1) L.c1 |= bit; else L.c0 |= bit;
        L.age++;
        L.depth++;
        uint32_t nid = blk * C4_SLOTS + (uint32_t)col;
        L.node = nid;
        if (lane == L.depth) L.path_lo = nid;
        if (lane + 32 == L.depth) L.path_hi = nid;
    }
    L.meta = meta;
    return L;
}

// side-relative value and absolute value of root child in lane c (oinkoink/tree.py:27-44, utils.py:33-34)
__device__ __forceinline__ void child_values(const C4NodeA &a, bool exists, int side, double &v_side, double &v_abs)
{
    v_side = 0.0;
    v_abs = nan("");
    if (!exists) return;
    if (a.meta & C4_META_TERMINAL) v_abs = c4_meta_value(a.meta);
    else if (a.visits > 0u) v_abs = __ddiv_rn(a.vsum, (double)a.visits);
    else return;
    v_side = side ? __dsub_rn(1.0, v_abs) : v_abs;
}

// Tree._normalise_policy (oinkoink/tree.py:139-147) on the per-lane raw policy entries
__device__ __forceinline__ double normalise_policy(double v, bool exists)
{
    double s = seq_sum7(v);
    unsigned m = __ballot_sync(FULL, exists) & 127u;
    if (s == 0.0) return exists ? __ddiv_rn(1.0, (double)__popc(m)) : __ddiv_rn(0.0, (double)__popc(m));
    return __ddiv_rn(v, s);
}

// argmax of (value, column) over existing children, ties -> highest column (Tree.best_move, tree.py:69-73)
__device__ __forceinline__ int best_child(double v, bool exists, int lane)
{
    double s = exists ? v : -1.0;
    int col = lane & 7;
    if (lane >= 7) s = -1.0;
#pragma unroll
    for (int off = 4; off >= 1; off >>= 1) {
        double os = __shfl_xor_sync(FULL, s, off);
        int oc = __shfl_xor_sync(FULL, col, off);
        if (os > s || (os == s && oc > col)) { s = os; col = oc; }
    }
    return __shfl_sync(FULL, col, 0);
}

// Tree.sample_value_fn(lambda x: x**2) (oinkoink/tree.py:75-82) with np.random.choice's inverse-cdf draw
__device__ __forceinline__ int sample_child(double v, bool exists, int lane, double u)
{
    double w = exists ? __dmul_rn(v, v) : 0.0;
    if (lane >= 7) w = 0.0;
    double s = seq_sum7(w);
    if (!(s > 0.0)) return best_child(v, exists, lane);   // reference raises here (NaN probabilities)
    double p = __ddiv_rn(w, s);
    const unsigned m = __ballot_sync(FULL, lane < 7 && exists) & 127u;
    double cdf = 0.0, mine = 0.0, last = 0.0;
#pragma unroll
    for (int i = 0; i < 7; i++) {
        cdf = __dadd_rn(cdf, shfl_d(p, i));
        if (i == lane) mine = cdf;
        if ((m >> i) & 1u) last = cdf;
    }
    mine = __ddiv_rn(mine, last);
    unsigned hit = __ballot_sync(FULL, lane < 7 && exists && mine > u) & 127u;
    if (hit) return __ffs(hit) - 1;
    return 31 - __clz(m);
}

// the pass's stop rule: one more game of the pool waits (for the network, or for another game's leaf)
__device__ __forceinline__ void count_busy(const C4Dev &d, int pool, int parity, int stop_count)
{
    const int b = atomicAdd(&d.ctr->busy_count[pool][parity], 1);
    if (stop_count > 0 && b + 1 == stop_count) d.ctr->stop_flag[pool][parity] = 1;
}
// park the pending leaf of a game (consumed when the answer is there): node, board, path
__device__ __forceinline__ void save_pending(const C4Dev &d, const Game &G, u64 c0, u64 c1, uint32_t node, int path_len,
                                             uint32_t path_lo, uint32_t path_hi)
{
    if (G.lane == 0) {
        d.pend_c0[G.g] = c0; d.pend_c1[G.g] = c1;
        d.pending_node[G.g] = (int)node; d.path_len[G.g] = path_len;
    }
    if (G.lane < path_len) d.path[(size_t)G.g * PATH_CAP + G.lane] = path_lo;
    if (G.lane + 32 < path_len) d.path[(size_t)G.g * PATH_CAP + G.lane + 32] = path_hi;
}
// append a (parked) leaf to the pool's batch
__device__ __forceinline__ void emit_request(const C4Dev &d, Game &G, int pool, int g0, int parity, u64 c0, u64 c1,
                                             int stop_count = 0)
{
    if (G.lane == 0) {
        // INTENTIONAL RACES (2 and 3 of 3 in the lock-step engine): the leaf counter is bumped with an atomic while the
        // network kernel of the PREVIOUS pass may still read its ping-pong twin (two counters per pool, reset one pass late),
        // and the stop flag is a plain store polled with plain loads: a warp that sees it one simulation late only plays
        // one more simulation of its own game -- pass length never changes results (tests/test_gpu_edges.py)
        const int k = atomicAdd(&d.ctr->leaf_count[pool][parity], 1);               // a pool's batch lives at [g0, g0 + n)
        C4_DEV_ASSERT(k >= 0 && g0 + k < g0 + (1 << 20));
        count_busy(d, pool, parity, stop_count);
        const int slot = g0 + k;
        d.leaf_c0[slot] = c0; d.leaf_c1[slot] = c1; d.leaf_game[slot] = G.g;
        d.pending_slot[G.g] = slot;
        d.stat_evals[G.g] += 1ULL;
    }
}

// End of a search inside a self-play game: pick the move, log the position, play it, finish / re-seed the game.
// oinkoink/mcts.py:78-88 (MCTS.make_move) + neural/training_game.py:8-19 (training_game).  Returns the new status.
template <class GAME>
__device__ __forceinline__ int finalize_move(const C4Dev &d, GAME &G)
{
    const int lane = G.lane;
    const int side = G.age & 1;
    const uint32_t blk = c4_meta_child_block(G.lda(0u).meta);
    C4NodeA a = G.lda(blk * C4_SLOTS + (uint32_t)(lane & 7));
    const bool exists = lane < 7 && (a.meta & C4_META_EXISTS);
    double v_side, v_abs;
    child_values(a, exists, side, v_side, v_abs);
    double pol = normalise_policy(lane < 7 ? v_side : 0.0, exists);
    int ply = d.ply[G.g];
    C4_DEV_ASSERT(ply >= 0 && ply < MAX_PLY && exists == (lane < 7 && ((c4_legal_mask(G.c0, G.c1) >> lane) & 1)));
    int mv;
    if (G.age < d.n_sampling && d.rng_mode != C4_RNG_NONE) {
        double u;
        if (d.rng_mode == C4_RNG_PHILOX) {
            Philox ph(d.seed, (u64)d.game_id[G.g], (u64)(ply * 8 + 7));
            uint32_t r[4];
            ph.next(r);
            u = ph.uniform_from(r[0], r[1]);
            if (d.rng_record && d.uniform && lane == 0) d.uniform[(size_t)G.g * MAX_PLY + ply] = u;
        } else {
            u = d.uniform[(size_t)G.g * MAX_PLY + ply];
        }
        mv = sample_child(v_side, exists, lane, u);
    } else {
        mv = best_child(v_side, exists, lane);
    }
    double mv_abs = shfl_d(v_abs, mv);
    c4_record *rec = d.staging + (size_t)G.g * MAX_PLY + ply;
    if (lane < 7) rec->policy[lane] = (float)pol;
    if (lane == 0) {
        rec->c0 = G.c0; rec->c1 = G.c1;
        rec->result_value = 0.f;
        rec->search_value = (float)mv_abs;
        rec->game_id = (int32_t)d.game_id[G.g];
        rec->move = (int8_t)mv; rec->ply = (int8_t)ply; rec->n_moves = 0; rec->result = C4_RES_NONE; rec->reserved = 0;
        d.stat_positions[G.g] += 1ULL;
    }
    C4_DEV_ASSERT(mv >= 0 && mv < 7 && ((c4_legal_mask(G.c0, G.c1) >> mv) & 1));
    int res = c4_drop(G.c0, G.c1, G.age, mv);
    G.age++;
    ply++;
    __syncwarp();
    if (res == C4_RES_NONE) {
        if (lane == 0) d.ply[G.g] = ply;
        return ST_NEWROOT;
    }
    // game over: flush the staged records with the final result, then re-seed the slot
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(&d.ctr->n_records, (unsigned long long)ply);
    base = shfl_u64(base, 0);
    if (d.records_out) {
        if ((long long)(base + ply) <= d.max_records) {
            for (int r = lane; r < ply; r += 32) {
                c4_record t = d.staging[(size_t)G.g * MAX_PLY + r];
                t.result_value = (float)(res * 0.5);
                t.n_moves = (int8_t)ply;
                t.result = (int8_t)res;
                t.reserved = 0;
                d.records_out[base + r] = t;
            }
        } else if (lane == 0) {
            atomicAdd(&d.ctr->overflow, 1ULL);
        }
    }
    unsigned long long nxt = 0;
    if (lane == 0) {
        atomicAdd(&d.ctr->games_finished, 1ULL);
        nxt = atomicAdd(&d.ctr->next_game, 1ULL);
    }
    nxt = shfl_u64(nxt, 0);
    if ((long long)nxt >= d.n_games_target) return ST_IDLE;
    G.c0 = d.start_c0 ? d.start_c0[nxt] : 0ULL;
    G.c1 = d.start_c1 ? d.start_c1[nxt] : 0ULL;
    G.age = c4_age(G.c0, G.c1);
    if (lane == 0) {
        d.game_id[G.g] = d.game_id_base + (long long)nxt * d.game_id_stride;
        d.ply[G.g] = 0;
    }
    __syncwarp();
    return ST_NEWROOT;
}

