// c4_search.cu -- warp-per-game MCTS engine: select / expand / evaluate / backup and the self-play state machine.
//
// Reference semantics reproduced bit-for-bit (deterministic evaluator): oinkoink/mcts.py:94-202 (search,
// evaluate_node, select_child, ucb_score, backpropagate, add_exploration_noise, normalise), oinkoink/tree.py:18-147
// (NodeData.value, best_move, sample_value_fn, get_values_policy), oinkoink/neural/training_game.py:8-19.
//
// B200 design (NOT the reference's structure):
//  * one warp owns one game for the whole kernel; lanes 0..6 are the seven columns.  One descent level = lanes 0..6
//    each reading their 32-byte child record (two 128-bit loads, two fully used 128-byte lines per level), fp64 PUCT
//    per lane from select-ready fields (the side-relative mean is maintained by backup, the division by n+1 is a table
//    reciprocal + two FMAs verified against IEEE division on the host), argmax on (score, column) by two REDUX.MAX
//    over an order-preserving 64-bit key and one vote.
//  * children are allocated EAGERLY when a node is evaluated (one 8-slot block), which is observably identical to the
//    reference's lazy expand-on-second-visit (a node's children cannot be reached before its second visit) but lets
//    the evaluation result (prior) be scattered straight into the child records.
//  * boards are not stored per node: the descent replays the moves on the root bitboards held in registers; only the
//    terminal result of each child is stored (2 bits), computed by the drop + 4-in-a-row test at block creation.
//  * a game advances until it needs an evaluator answer; pending leaves of all games are compacted into one batch
//    (atomic slot counter), evaluated by the network kernel (c4_net.cu) or the host, and consumed by the next pass.
//    Terminal revisits and hits of the evaluation memo (the reference's Evaluator.position_table, here a checksummed
//    hash table in HBM) need no evaluator and are played through inside the same pass (bounded by `budget`, a cycle
//    limit, and the share of games already waiting for the network).
//  * all PUCT arithmetic uses explicit round-to-nearest intrinsics (__dmul_rn/__dadd_rn/__ddiv_rn/__dsqrt_rn) so no
//    FMA contraction can change the reference's two-rounding  pb_c*prior + value ; log() comes from a host-built
//    table (glibc, the same libm Python's math.log calls).
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <vector>

#include "c4_common.cuh"

#include "c4_tree.cuh"

// c4_fused.cu: the persistent engine (one launch per generation); c4_search.cu keeps the lock-step pass engine
bool c4_fused_eligible(const c4_net *net, int max_games, long long live_games);
int c4_fused_run(const C4Dev &d, const c4_net *net, int max_games, int simulations, bool selfplay,
                 unsigned long long stop_games, double stop_ms, cudaStream_t stream);
// c4_split.cu: the persistent engine with tree CTAs and tower CTAs on separate SMs (same contract)
bool c4_split_eligible(const c4_net *net, int max_games, long long live_games);
int c4_split_last_launches();
int c4_split_run(const C4Dev &d, const c4_net *net, int max_games, int simulations, bool selfplay,
                 unsigned long long stop_games, double stop_ms, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------ the pass kernel
// A game needs an evaluation that is not in the memo: park the leaf, then either append it to the pool's batch (ST_WAIT) or,
// if another game claimed the same position a moment ago, wait for that game's answer (ST_WAITMEMO; c4_tree.cuh).
template <int MODE>
__device__ __forceinline__ int request_or_wait(const C4Dev &d, Game &G, int pool, int g0, int parity, int stop_count, u64 c0,
                                               u64 c1, uint32_t node, int path_len, uint32_t path_lo, uint32_t path_hi,
                                               int probe, u64 seen)
{
    save_pending(d, G, c0, c1, node, path_len, path_lo, path_hi);
    if (MODE == C4_EVAL_NET && d.memo && d.memo_dedup && (probe == MEMO_PENDING || !memo_claim(d, c0, c1, seen, G.lane))) {
        if (G.lane == 0) { count_busy(d, pool, parity, stop_count); d.pending_slot[G.g] = 0; }   // looks at the memo so far
        return ST_WAITMEMO;
    }
    emit_request(d, G, pool, g0, parity, c0, c1, stop_count);
    return ST_WAIT;
}

// MODE: C4_EVAL_EXTERNAL / C4_EVAL_CENTRE / C4_EVAL_NET.  One warp per game slot.
template <int MODE, bool SELFPLAY>
#ifndef C4_ADV_MIN_BLOCKS
#define C4_ADV_MIN_BLOCKS 8
#endif
__global__ void __launch_bounds__(128, C4_ADV_MIN_BLOCKS) k_advance(C4Dev d, int g0, int n_games, int pool, int parity, int budget, long long cycle_limit, int stop_count)
{
    const int gi = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int g = g0 + gi;
    const int lane = threadIdx.x & 31;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        d.ctr->leaf_count[pool][parity ^ 1] = 0; d.ctr->busy_count[pool][parity ^ 1] = 0; d.ctr->stop_flag[pool][parity ^ 1] = 0;
    }
    if (gi >= n_games) return;
    const long long t_start = clock64();
    int st = d.status[g];
    if (st == ST_IDLE || st == ST_DONE) return;

    Game G;
    G.g = g; G.lane = lane;
    G.gp = d.pool + (size_t)g * d.blocks_per_game * C4_SLOTS;
    G.n_blocks = d.n_blocks[g];
    G.sims_done = d.sims_done[g];
    G.c0 = d.root_c0[g]; G.c1 = d.root_c1[g];
    G.age = c4_age(G.c0, G.c1);

    if (st == ST_WAIT || st == ST_WAITMEMO) {
        // consume the evaluator's answer for the pending leaf (oinkoink/mcts.py:129-135), then backpropagate
        const uint32_t node = (uint32_t)d.pending_node[g];
        const int plen = d.path_len[g];
        const u64 lc0 = d.pend_c0[g], lc1 = d.pend_c1[g];
        const int lage = c4_age(lc0, lc1);
        const bool is_root = (plen == 0);
        const int ply = SELFPLAY ? d.ply[g] : 0;
        if (MODE == C4_EVAL_NET) {
            float ov;
            if (st == ST_WAIT) {
                const float *o = d.net_out + (size_t)d.pending_slot[g] * 8;
                ov = (lane < 8) ? o[lane] : 0.f;
                if (__any_sync(FULL, !isfinite(ov))) {
                    // operand overflow (fp16) or NaN weights: neutral answer + a flag that makes the host call fail
                    // (the reference asserts on every evaluation, oinkoink/neural/pytorch/model.py:258-263,275-280)
                    ov = (lane < 7) ? (1.f / 7.f) : 0.5f;
                    if (lane == 0) d.ctr->net_nonfinite = 1;
                }
                if (d.memo) memo_insert(d, lc0, lc1, ov, lane);          // replaces this game's PENDING tag
            } else {
                // the leaf was being evaluated for another game.  Its owner consumes the answer at the start of this very
                // pass and puts it into the memo a microsecond or two from now: look a few times (bounded -- the owner's
                // warp may not be running yet), then leave it for the next pass
                u64 seen;
                int pr = memo_probe(d, lc0, lc1, ov, lane, seen);
                for (int k = 0; k < 6 && pr == MEMO_PENDING; k++) { __nanosleep(500); pr = memo_probe(d, lc0, lc1, ov, lane, seen); }
                if (pr == MEMO_HIT) {
                    if (lane == 0) d.stat_hits[g] += 1ULL;
                } else if (budget < 0 || (d.pending_slot[g] < WAITMEMO_PATIENCE &&
                                          (pr == MEMO_PENDING || !memo_claim(d, lc0, lc1, seen, lane)))) {
                    if (lane == 0) { count_busy(d, pool, parity, stop_count); d.pending_slot[g] += 1; }   // still waiting
                    return;                         // (a consume-only pass never asks for anything new)
                } else {                            // the tag is gone (a colliding key took the entry): evaluate it ourselves
                    emit_request(d, G, pool, g0, parity, lc0, lc1, stop_count);
                    if (lane == 0) d.status[g] = ST_WAIT;
                    return;
                }
            }
            float pf = (lane < 7) ? ov : 0.f;
            double value = (double)__shfl_sync(FULL, ov, 7);
            apply_eval<true>(d, G, node, lc0, lc1, lage, value, 0.0, pf, is_root, ply);
            if (!is_root) {
                uint32_t plo = (lane < plen) ? d.path[(size_t)g * PATH_CAP + lane] : 0u;
                uint32_t phi = (lane + 32 < plen) ? d.path[(size_t)g * PATH_CAP + lane + 32] : 0u;
                backup(G, plo, phi, plen - 1, value);
                G.sims_done++;
            }
        } else if (MODE == C4_EVAL_EXTERNAL) {
            const int slot = d.pending_slot[g];
            double value = d.ext_value[slot];
            if (d.ext_prior_dtype == 1) {
                float pf = (lane < 7) ? ((const float *)d.ext_prior)[(size_t)slot * 7 + lane] : 0.f;
                apply_eval<true>(d, G, node, lc0, lc1, lage, value, 0.0, pf, is_root, ply);
            } else {
                double p = (lane < 7) ? ((const double *)d.ext_prior)[(size_t)slot * 7 + lane] : 0.0;
                apply_eval<false>(d, G, node, lc0, lc1, lage, value, p, 0.f, is_root, ply);
            }
            if (!is_root) {
                uint32_t plo = (lane < plen) ? d.path[(size_t)g * PATH_CAP + lane] : 0u;
                uint32_t phi = (lane + 32 < plen) ? d.path[(size_t)g * PATH_CAP + lane + 32] : 0u;
                backup(G, plo, phi, plen - 1, value);
                G.sims_done++;
            }
        }
        st = ST_READY;
    }

    bool first_descent_done = false;
    int waiting_seen = 0;
    for (;;) {
        if (budget < 0) break;                                            // consume-only pass (hand-over to the fused engine)
        if (st == ST_NEWROOT) {
            // Tree(board) + evaluate root (oinkoink/mcts.py:98-105): fresh pool, root = node 0 of block 0
            G.n_blocks = 1;
            G.sims_done = 0;
            if (lane == 0) { st_a(G.gp, 0.0, 0u, C4_META_EXISTS); st_b(G.gp, 0.0, 0.0); }
            __syncwarp();
            if (MODE == C4_EVAL_CENTRE) {
                const int ply = SELFPLAY ? d.ply[g] : 0;
                apply_eval<false>(d, G, 0u, G.c0, G.c1, G.age, c4_evaluate_centre(G.c0, G.c1), __ddiv_rn(1.0, 7.0),
                                  0.f, true, ply);
                if (lane == 0) d.stat_evals[g] += 1ULL;
                st = ST_READY;
            } else {
                float ov;
                u64 seen = 0;
                const int pr = (MODE == C4_EVAL_NET && d.memo) ? memo_probe(d, G.c0, G.c1, ov, lane, seen) : MEMO_MISS;
                if (pr == MEMO_HIT) {
                    // the new root was evaluated before (usually as a leaf of the previous move's search)
                    const int ply = SELFPLAY ? d.ply[g] : 0;
                    apply_eval<true>(d, G, 0u, G.c0, G.c1, G.age, (double)__shfl_sync(FULL, ov, 7), 0.0,
                                     (lane < 7) ? ov : 0.f, true, ply);
                    if (lane == 0) d.stat_hits[g] += 1ULL;
                    st = ST_READY;
                } else {
                    st = request_or_wait<MODE>(d, G, pool, g0, parity, stop_count, G.c0, G.c1, 0u, 0, 0u, 0u, pr, seen);
                    break;
                }
            }
        }
        if (G.sims_done >= d.sims) {
            if (!SELFPLAY) {
                st = ST_DONE;
                if (lane == 0) atomicAdd(&d.ctr->n_done, 1ULL);
                break;
            }
            st = finalize_move(d, G);
            if (st == ST_IDLE) break;
            continue;
        }
        if (budget-- <= 0) break;
        // bound the tail of the pass: the first descent is always allowed, later ones (after terminal re-visits) only
        // while the warp is inside its cycle budget
        if (cycle_limit > 0 && first_descent_done && clock64() - t_start > cycle_limit) break;
        // ... and the pass ends for everybody once `stop_count` games of the pool wait for the network: the games still
        // running would only keep the waiting ones from their answers (cold memo: most games miss at once and the
        // pass lasts a simulation or two; warm memo: it runs until the usual share of games has missed)
        // (the counter is read one simulation ahead of its use, so its L2 round trip is off the critical path)
        if (stop_count > 0) {
            if (first_descent_done && waiting_seen != 0) break;
            waiting_seen = __ldcg(&d.ctr->stop_flag[pool][parity]);           // one broadcast L2 read per warp
        }
        first_descent_done = true;
        Leaf L = descend(d, G);
        if (L.meta & C4_META_TERMINAL) {
            // terminal branch of evaluate_node (mcts.py:125-128) + backpropagate: leaf and all ancestors get the result
            backup(G, L.path_lo, L.path_hi, L.depth + 1, c4_meta_value(L.meta));
            G.sims_done++;
            continue;
        }
        if (MODE == C4_EVAL_CENTRE) {
            double value = c4_evaluate_centre(L.c0, L.c1);
            apply_eval<false>(d, G, L.node, L.c0, L.c1, L.age, value, __ddiv_rn(1.0, 7.0), 0.f, false, 0);
            backup(G, L.path_lo, L.path_hi, L.depth, value);
            if (lane == 0) d.stat_evals[g] += 1ULL;
            G.sims_done++;
            continue;
        }
        int pr = MEMO_MISS;
        u64 seen = 0;
        if (MODE == C4_EVAL_NET && d.memo) {
            float ov;
            pr = memo_probe(d, L.c0, L.c1, ov, lane, seen);
            if (pr == MEMO_HIT) {
                const double value = (double)__shfl_sync(FULL, ov, 7);
                apply_eval<true>(d, G, L.node, L.c0, L.c1, L.age, value, 0.0, (lane < 7) ? ov : 0.f, false, 0);
                backup(G, L.path_lo, L.path_hi, L.depth, value);
                if (lane == 0) d.stat_hits[g] += 1ULL;
                G.sims_done++;
                continue;
            }
        }
        st = request_or_wait<MODE>(d, G, pool, g0, parity, stop_count, L.c0, L.c1, L.node, L.depth + 1, L.path_lo, L.path_hi, pr, seen);
        break;
    }
    if (lane == 0) {
        d.status[g] = st;
        d.n_blocks[g] = G.n_blocks;
        d.sims_done[g] = G.sims_done;
        d.root_c0[g] = G.c0; d.root_c1[g] = G.c1;
    }
}

// ------------------------------------------------------------------------------------------------ small kernels
__global__ void k_search_begin(C4Dev d, const u64 *c0, const u64 *c1, int n, int max_games)
{
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g == 0) {
        d.ctr->leaf_count[0][0] = 0; d.ctr->leaf_count[0][1] = 0; d.ctr->leaf_count[1][0] = 0; d.ctr->leaf_count[1][1] = 0;
        d.ctr->busy_count[0][0] = 0; d.ctr->busy_count[0][1] = 0; d.ctr->busy_count[1][0] = 0; d.ctr->busy_count[1][1] = 0;
        d.ctr->stop_flag[0][0] = 0; d.ctr->stop_flag[0][1] = 0; d.ctr->stop_flag[1][0] = 0; d.ctr->stop_flag[1][1] = 0;
        d.ctr->n_done = 0; d.ctr->engine_error = 0; d.ctr->net_nonfinite = 0;
    }
    if (g >= max_games) return;
    if (g < n) {
        d.root_c0[g] = c0[g]; d.root_c1[g] = c1[g];
        d.status[g] = ST_NEWROOT;
        d.game_id[g] = g;
    } else {
        d.status[g] = ST_IDLE;
    }
    d.sims_done[g] = 0; d.n_blocks[g] = 1; d.ply[g] = 0; d.path_len[g] = 0;
}

__global__ void k_selfplay_init(C4Dev d, int max_games)
{
    int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g == 0) {
        d.ctr->leaf_count[0][0] = 0; d.ctr->leaf_count[0][1] = 0; d.ctr->leaf_count[1][0] = 0; d.ctr->leaf_count[1][1] = 0;
        d.ctr->busy_count[0][0] = 0; d.ctr->busy_count[0][1] = 0; d.ctr->busy_count[1][0] = 0; d.ctr->busy_count[1][1] = 0;
        d.ctr->stop_flag[0][0] = 0; d.ctr->stop_flag[0][1] = 0; d.ctr->stop_flag[1][0] = 0; d.ctr->stop_flag[1][1] = 0;
        d.ctr->games_finished = 0; d.ctr->n_records = 0; d.ctr->overflow = 0; d.ctr->n_done = 0;
        d.ctr->engine_error = 0; d.ctr->net_nonfinite = 0;
        long long first = d.n_games_target < (long long)max_games ? d.n_games_target : (long long)max_games;
        d.ctr->next_game = (unsigned long long)first;
    }
    if (g >= max_games) return;
    d.sims_done[g] = 0; d.n_blocks[g] = 1; d.ply[g] = 0; d.path_len[g] = 0;
    d.stat_evals[g] = 0; d.stat_positions[g] = 0; d.stat_hits[g] = 0;
    if ((long long)g < d.n_games_target) {
        d.root_c0[g] = d.start_c0 ? d.start_c0[g] : 0ULL;
        d.root_c1[g] = d.start_c1 ? d.start_c1[g] : 0ULL;
        d.game_id[g] = d.game_id_base + (long long)g * d.game_id_stride;
        d.status[g] = ST_NEWROOT;
    } else {
        d.status[g] = ST_IDLE;
    }
}

// root read-out: one warp per game (Tree.get_values_policy / get_visit_count_policy / best_move + reference node count)
__global__ void k_readout(C4Dev d, int n, int32_t *visits, double *value_sum, int8_t *child_result,
                          int32_t *root_visits, double *root_value_sum, double *root_prior, double *values_policy,
                          double *visit_policy, int8_t *best_move, double *best_value, int32_t *n_nodes)
{
    const int g = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (g >= n) return;
    C4Node *gp = d.pool + (size_t)g * d.blocks_per_game * C4_SLOTS;
    const u64 c0 = d.root_c0[g], c1 = d.root_c1[g];
    const int side = c4_age(c0, c1) & 1;
    C4NodeA ra = ld_a(gp);
    const uint32_t blk = c4_meta_child_block(ra.meta);
    C4NodeA a; a.vsum = 0.0; a.visits = 0; a.meta = 0;
    C4NodeB b; b.prior = 0.0; b.vsel = 0.0;
    if (blk != 0u) { a = ld_a(gp + (size_t)blk * C4_SLOTS + (lane & 7)); b = ld_b(gp + (size_t)blk * C4_SLOTS + (lane & 7)); }
    const bool exists = lane < 7 && (a.meta & C4_META_EXISTS);
    // the reference creates the root's children during the first simulation only
    const bool expanded = ra.visits >= 2u;
    const bool ex = exists && expanded;
    double v_side, v_abs;
    child_values(a, ex, side, v_side, v_abs);
    double vp = normalise_policy(lane < 7 ? v_side : 0.0, ex);
    double cnt = (ex && a.visits > 0u) ? (double)a.visits : 0.0;
    double cp = normalise_policy(lane < 7 ? cnt : 0.0, ex);
    int bm = best_child(v_side, ex, lane);
    double bv = shfl_d(v_abs, bm);
    if (lane < 7) {
        size_t o = (size_t)g * 7 + lane;
        if (visits) visits[o] = ex ? (int32_t)a.visits : 0;
        if (value_sum) value_sum[o] = ex ? a.vsum : 0.0;
        if (child_result) child_result[o] = ex ? (int8_t)c4_meta_result(a.meta) : (int8_t)-2;
        if (root_prior) root_prior[o] = exists ? b.prior : 0.0;
        if (values_policy) values_policy[o] = vp;
        if (visit_policy) visit_policy[o] = cp;
    }
    if (lane == 0) {
        if (root_visits) root_visits[g] = (int32_t)ra.visits;
        if (root_value_sum) root_value_sum[g] = ra.vsum;
        if (best_move) best_move[g] = expanded ? (int8_t)bm : (int8_t)-1;
        if (best_value) best_value[g] = bv;
    }
    if (n_nodes) {
        // nodes of the reference's lazily expanded tree: root + children of every node visited at least twice
        int nb = d.n_blocks[g], total = 0;
        for (int bI = 1 + lane; bI < nb; bI += 32) {
            C4NodeB h = ld_b(gp + (size_t)bI * C4_SLOTS + 7);
            C4NodeA pa = ld_a(gp + header_parent(h));
            if (pa.visits >= 2u) total += (int)header_children(h);
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) total += __shfl_xor_sync(FULL, total, off);
        if (lane == 0) n_nodes[g] = total + 1;
    }
}

__global__ void k_sum_stats(const unsigned long long *evals, const unsigned long long *positions,
                            const unsigned long long *hits, int n, unsigned long long *out)
{
    unsigned long long e = 0, p = 0, h = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) { e += evals[i]; p += positions[i]; h += hits[i]; }
    __shared__ unsigned long long se[256], sp[256], sh[256];
    se[threadIdx.x] = e; sp[threadIdx.x] = p; sh[threadIdx.x] = h;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) {
            se[threadIdx.x] += se[threadIdx.x + s]; sp[threadIdx.x] += sp[threadIdx.x + s]; sh[threadIdx.x] += sh[threadIdx.x + s];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) { out[0] = se[0]; out[1] = sp[0]; out[2] = sh[0]; }
}

// occupied entries of the evaluation memo (diagnostics: distinct positions evaluated ~ occupied entries)
__global__ void k_memo_count(const uint32_t *memo, size_t n_entries, unsigned long long *out)
{
    unsigned long long c = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_entries; i += (size_t)gridDim.x * blockDim.x)
        c += (memo[i * 16 + 12] | memo[i * 16 + 13]) != 0u;
    for (int off = 16; off >= 1; off >>= 1) c += __shfl_xor_sync(0xffffffffu, c, off);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

// generation sink: native_to_pytorch(add_fliplr=True) (oinkoink/neural/pytorch/data.py:78-105); originals first, then
// mirrors.  HBM-write bound (536 B out per 64 B record).  Two consecutive rows of 126 plane floats are 63 aligned
// float4, so one thread produces one float4 and a warp writes 512 contiguous bytes per store; where a plane float comes
// from (to-move flag, or which bit of which colour) is a 126-entry table in shared memory; the 64-byte record is read
// through L1 by the threads of its row.
__global__ void __launch_bounds__(256) k_augment_pack(const c4_record *__restrict__ rec, long long n, float *__restrict__ boards,
                                                     float *__restrict__ values, float *__restrict__ priors)
{
    __shared__ unsigned char tab[126];                                    // (channel << 6) | bit index (board.py:147-154)
    for (int k = threadIdx.x; k < 126; k += blockDim.x) {
        const int ch = k / 42, px = k - ch * 42, rr = px / 7, c = px - rr * 7;
        tab[k] = (unsigned char)((ch << 6) | (7 * c + (5 - rr)));
    }
    __syncthreads();
    const long long total = n * 63;                                       // float4 units: 2n rows / 2 rows per 63 float4
    float4 *out4 = reinterpret_cast<float4 *>(boards);
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long pair = e / 63;
        const int f0 = 4 * (int)(e - pair * 63);                          // first of 4 floats inside the 252-float row pair
        float v[4];
        long long row_prev = -1;
        u64 a = 0, b = 0;
        float tomove = 0.f;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int f = f0 + i;
            const long long row = 2 * pair + (f >= 126);
            const int k = f >= 126 ? f - 126 : f;
            if (row != row_prev) {                                        // at most two records per thread
                const bool flip = row >= n;
                const c4_record &r = rec[flip ? row - n : row];
                a = r.c0; b = r.c1;
                if (flip) { a = c4_fliplr(a); b = c4_fliplr(b); }
                tomove = ((__popcll(a | b) & 1) == 0) ? 1.f : 0.f;
                row_prev = row;
            }
            const unsigned t = tab[k];
            const u64 src = (t & 64u) ? a : b;
            v[i] = (t < 64u) ? tomove : (float)((src >> (t & 63u)) & 1ULL);
        }
        out4[e] = make_float4(v[0], v[1], v[2], v[3]);
    }
    // values and priors: 8 floats per row, one thread per row
    for (long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x; row < 2 * n; row += (long long)gridDim.x * blockDim.x) {
        const bool flip = row >= n;
        const c4_record &r = rec[flip ? row - n : row];
        values[row] = r.result_value;
#pragma unroll
        for (int j = 0; j < 7; j++) priors[row * 7 + j] = flip ? r.policy[6 - j] : r.policy[j];
    }
}

// ------------------------------------------------------------------------------------------------ host side
struct c4_ctx {
    int device;
    int max_games;
    int sims_cap;
    c4_mcts_config cfg;
    C4Dev d;
    c4_net *net;
    std::vector<void *> allocs;
    double *pbc_dev;
    double *sqt_dev;
    double *rcp_dev;
    float *net_out;
    double *ext_value;
    void *ext_prior;
    unsigned long long *stats_dev;      // [2]
    unsigned long long *pinned;         // host pinned scratch (64 words: counters copy + stats at [40..])
    int parity;                         // single-pool paths (stand-alone searches)
    int pool_parity[2];                 // self-play half pools
    int n_pools;                        // 2: the tree pass of one half overlaps the network launch of the other
    int net_ctas;                       // CTA cap of a half-pool network launch (leaves SMs for the concurrent tree pass)
    cudaStream_t pool_stream[2];
    cudaEvent_t ev_fork, ev_join[2];
    int n_search;                       // searches started by the last c4_search_begin
    long long cycle_limit;
    double stop_frac;                   // a NET pass ends once this share of the live games waits for the network (0 = off)
    long long live_games;               // upper bound of the games still being played (self-play tail)
    unsigned long long memo_net_uid;    // network whose outputs the memo currently holds
    long long last_memo_hits;           // memo hits during the last c4_selfplay_bench call
    int memo_log2;                      // log2(entries) of the evaluation memo, 0 = disabled
    int budget_net;                     // terminal re-visits a game may play through per pass (NET / EXTERNAL)
    int last_pending;
    bool supplied;
    bool search_failed;                 // the network call of the last c4_search_run failed: its games wait for answers
                                        // that never came, so only a new c4_search_begin may run searches again
    bool pool_fresh;                    // bench pool initialised
    long long last_launches;            // kernels launched by the last c4_selfplay_stream call
    cudaGraphExec_t chunk_graph[2];     // 64 lock-step passes of the re-seeding / generation pool captured once (no per-launch
    unsigned long long chunk_key[2][4]; // host work, no gaps between the 128 launches); re-captured when its parameters change;
                                        // [1] = the same with the launches of pass 32 bracketed by events (eva / evs [0..1])
    float last_tree_ms, last_net_ms;    // lock-step engine: mean sampled launch durations of the last c4_selfplay_stream call
    long long last_passes;
    int pool_engine;                    // engine that owns the re-seeding pool's state: 0 none, 1 lock-step, 2 fused
    cudaEvent_t ev0, ev1;
    cudaEvent_t evs[2 * 64];            // sampled (start, stop) pairs around network launches
    cudaEvent_t eva[2 * 64];            // sampled (start, stop) pairs around tree-pass launches
};
#define N_SAMPLES 64

template <typename T>
static int dev_alloc(c4_ctx *ctx, T **p, size_t n)
{
    void *q = nullptr;
    C4_CUDA(cudaMalloc(&q, n * sizeof(T)));
    C4_CUDA(cudaMemset(q, 0, n * sizeof(T)));
    ctx->allocs.push_back(q);
    *p = (T *)q;
    return 0;
}

// The select loop divides sqrt(N) by (n+1) with a table reciprocal and two FMAs.  That sequence is checked here against
// IEEE division for every (N, n+1) pair a search of this capacity can produce (N, n+1 <= simulations + 1); if a single
// pair differed (none does up to the 4096-simulation limit of the check) the kernel uses __ddiv_rn instead.
static bool fastdiv_verified(int sims_cap)
{
    static std::mutex mu;
    static int ok_cap = -1;             // every pair up to this capacity verified equal
    static int bad_cap = 1 << 30;       // a pair below this capacity differed
    if (sims_cap > 4096 || getenv("C4_NO_FASTDIV")) return false;
    std::lock_guard<std::mutex> lock(mu);
    if (sims_cap <= ok_cap) return true;
    if (sims_cap >= bad_cap) return false;
    const int n = sims_cap + 2;
    std::vector<double> q(n), r(n);
    for (int i = 0; i < n; i++) { q[i] = sqrt((double)i); r[i] = i ? 1.0 / (double)i : 0.0; }
    for (int N = 0; N < n; N++)
        for (int m = 1; m < n; m++) {
            if (N <= ok_cap + 1 && m <= ok_cap + 1) continue;
            const double den = (double)m, q0 = q[N] * r[m];
            const double qq = fma(fma(-den, q0, q[N]), r[m], q0);
            if (qq != q[N] / den) { bad_cap = sims_cap; return false; }
        }
    ok_cap = sims_cap;
    return true;
}

static int upload_config(c4_ctx *ctx, const c4_mcts_config *cfg)
{
    C4_REQUIRE(cfg->simulations >= 0 && cfg->simulations <= ctx->sims_cap, "simulations exceeds the context capacity");
    C4_REQUIRE(cfg->pb_c_base > 0, "pb_c_base must be positive");
    ctx->cfg = *cfg;
    std::vector<double> t(ctx->sims_cap + 2), q(ctx->sims_cap + 2), r(ctx->sims_cap + 2);
    for (int n = 0; n < (int)t.size(); n++) {                  // oinkoink/mcts.py:150-154, host libm log / sqrt
        t[n] = log(((double)n + cfg->pb_c_base + 1.0) / cfg->pb_c_base) + cfg->pb_c_init;
        q[n] = sqrt((double)n);
        r[n] = n ? 1.0 / (double)n : 0.0;
    }
    C4_CUDA(cudaMemcpy(ctx->pbc_dev, t.data(), t.size() * sizeof(double), cudaMemcpyHostToDevice));
    C4_CUDA(cudaMemcpy(ctx->sqt_dev, q.data(), q.size() * sizeof(double), cudaMemcpyHostToDevice));
    C4_CUDA(cudaMemcpy(ctx->rcp_dev, r.data(), r.size() * sizeof(double), cudaMemcpyHostToDevice));
    ctx->d.fastdiv = fastdiv_verified(ctx->sims_cap) ? 1 : 0;
    ctx->d.sims = cfg->simulations;
    ctx->d.alpha = cfg->root_dirichlet_alpha;
    ctx->d.frac = cfg->root_exploration_fraction;
    ctx->d.one_minus_frac = 1.0 - cfg->root_exploration_fraction;
    ctx->d.one_minus_frac_f = (float)(1.0 - cfg->root_exploration_fraction);
    ctx->d.noise_on = (cfg->root_dirichlet_alpha != 0.0 && cfg->root_exploration_fraction != 0.0) ? 1 : 0;
    ctx->d.n_sampling = cfg->num_sampling_moves;
    return 0;
}

extern "C" int c4_ctx_create(int device, int32_t max_games, const c4_mcts_config *cfg, c4_ctx **out)
{
    C4_REQUIRE(out && cfg, "c4_ctx_create: null pointer");
    C4_REQUIRE(max_games > 0 && max_games <= (1 << 20), "max_games out of range");
    C4_REQUIRE(cfg->simulations >= 0 && cfg->simulations <= (1 << 20), "simulations out of range");
    int ndev = 0;
    C4_CUDA(cudaGetDeviceCount(&ndev));
    C4_REQUIRE(device >= 0 && device < ndev, "no such CUDA device (there is no CPU fallback)");
    C4_CUDA(cudaSetDevice(device));
    c4_ctx *ctx = new c4_ctx();
    ctx->device = device;
    ctx->max_games = max_games;
    ctx->sims_cap = cfg->simulations;
    ctx->net = nullptr;
    ctx->parity = 0;
    ctx->n_search = 0;
    ctx->budget_net = getenv("C4_BUDGET") ? atoi(getenv("C4_BUDGET")) : 96;
    ctx->n_pools = getenv("C4_POOLS") ? atoi(getenv("C4_POOLS")) : 1;
    if (ctx->n_pools < 1 || ctx->n_pools > 2) ctx->n_pools = 1;
    ctx->net_ctas = getenv("C4_NET_CTAS") ? atoi(getenv("C4_NET_CTAS")) : 112;
    ctx->pool_parity[0] = ctx->pool_parity[1] = 0;
    ctx->last_pending = 0;
    ctx->supplied = true;
    ctx->search_failed = false;
    ctx->pool_fresh = false;
    ctx->pool_engine = 0;
    ctx->chunk_graph[0] = ctx->chunk_graph[1] = nullptr;
    memset(ctx->chunk_key, 0, sizeof(ctx->chunk_key));
    memset(&ctx->d, 0, sizeof(ctx->d));
    C4Dev &d = ctx->d;
    // a warp starts no further descent in a NET pass after this many SM cycles (bounds the tail of the pass; 0 = off)
    ctx->cycle_limit = getenv("C4_CYCLE_LIMIT") ? atoll(getenv("C4_CYCLE_LIMIT")) : 160000;
    ctx->stop_frac = getenv("C4_STOP_FRAC") ? atof(getenv("C4_STOP_FRAC")) : 0.5;
    ctx->live_games = max_games;
    ctx->last_memo_hits = 0;
    ctx->memo_net_uid = 0;
    {   // evaluation memo: 65536 entries per game slot, 2^14 .. 2^28 entries of 64 B (<= 16 GiB of the 180 GB HBM; the hit
        // rate keeps rising with the size because 4096 games share openings); C4_MEMO_LOG2=0 disables
        int lg = 14;
        while (lg < 28 && (1LL << lg) < (long long)max_games * 65536) lg++;
        if (getenv("C4_MEMO_LOG2")) lg = atoi(getenv("C4_MEMO_LOG2"));
        ctx->memo_log2 = (lg >= 10 && lg <= 30) ? lg : 0;   // (29 and 30 through the environment only: 34 / 69 GB)
    }
    const size_t G = (size_t)max_games;
    d.blocks_per_game = cfg->simulations + 2;
    int rc = 0;
#define A(ptr, n) if ((rc = dev_alloc(ctx, &(ptr), (n))) != 0) { c4_ctx_destroy(ctx); return rc; }
    A(d.pool, G * d.blocks_per_game * C4_SLOTS);
    A(ctx->pbc_dev, (size_t)cfg->simulations + 2);
    A(ctx->sqt_dev, (size_t)cfg->simulations + 2);
    A(ctx->rcp_dev, (size_t)cfg->simulations + 2);
    d.pbc = ctx->pbc_dev;
    d.sqt = ctx->sqt_dev;
    d.rcp = ctx->rcp_dev;
    A(d.root_c0, G); A(d.root_c1, G); A(d.status, G); A(d.sims_done, G); A(d.n_blocks, G);
    A(d.pending_node, G); A(d.pending_slot, G); A(d.path_len, G); A(d.ply, G);
    A(d.pend_c0, G); A(d.pend_c1, G); A(d.path, G * PATH_CAP); A(d.game_id, G);
    A(d.stat_evals, G); A(d.stat_positions, G); A(d.stat_hits, G); A(d.staging, G * MAX_PLY);
    A(d.leaf_c0, G); A(d.leaf_c1, G); A(d.leaf_game, G);
    A(ctx->net_out, G * 8); A(ctx->ext_value, G);
    double *extp = nullptr;
    A(extp, G * 7);
    ctx->ext_prior = extp;
    A(d.ctr, 1); A(ctx->stats_dev, 4);
#undef A
    d.net_out = ctx->net_out;
    d.ext_value = ctx->ext_value;
    d.ext_prior = ctx->ext_prior;
    d.rng_mode = C4_RNG_NONE;
    if (cudaMallocHost((void **)&ctx->pinned, 64 * sizeof(unsigned long long)) != cudaSuccess) {
        c4_set_error("cudaMallocHost failed");
        c4_ctx_destroy(ctx);
        return -2;
    }
    cudaEventCreate(&ctx->ev0); cudaEventCreate(&ctx->ev1);
    cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming);
    for (int i = 0; i < 2; i++) {
        cudaStreamCreateWithFlags(&ctx->pool_stream[i], cudaStreamNonBlocking);
        cudaEventCreateWithFlags(&ctx->ev_join[i], cudaEventDisableTiming);
    }
    for (int i = 0; i < 2 * N_SAMPLES; i++) { cudaEventCreate(&ctx->evs[i]); cudaEventCreate(&ctx->eva[i]); }
    rc = upload_config(ctx, cfg);
    if (rc) { c4_ctx_destroy(ctx); return rc; }
    *out = ctx;
    return 0;
}

extern "C" int c4_ctx_destroy(c4_ctx *ctx)
{
    if (!ctx) return 0;
    cudaSetDevice(ctx->device);
    for (int i = 0; i < 2; i++) if (ctx->chunk_graph[i]) cudaGraphExecDestroy(ctx->chunk_graph[i]);
    for (void *p : ctx->allocs) cudaFree(p);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    if (ctx->ev0) {
        cudaEventDestroy(ctx->ev0); cudaEventDestroy(ctx->ev1); cudaEventDestroy(ctx->ev_fork);
        for (int i = 0; i < 2; i++) { cudaStreamDestroy(ctx->pool_stream[i]); cudaEventDestroy(ctx->ev_join[i]); }
        for (int i = 0; i < 2 * N_SAMPLES; i++) { cudaEventDestroy(ctx->evs[i]); cudaEventDestroy(ctx->eva[i]); }
    }
    delete ctx;
    return 0;
}

extern "C" int c4_ctx_set_config(c4_ctx *ctx, const c4_mcts_config *cfg)
{
    C4_REQUIRE(ctx && cfg, "c4_ctx_set_config: null pointer");
    C4_CUDA(cudaSetDevice(ctx->device));
    return upload_config(ctx, cfg);
}

extern "C" int c4_ctx_get(c4_ctx *ctx, int key)
{
    if (!ctx) return -1;
    switch (key) {
    case 0: return ctx->n_pools;
    case 1: return ctx->net_ctas;
    case 2: return ctx->budget_net;
    case 3: return ctx->max_games;
    case 4: return ctx->d.memo ? ctx->memo_log2 : 0;
    case 5: return (int)std::min<long long>(ctx->last_memo_hits, 0x7fffffff);
    case 6: return (int)std::min<long long>(ctx->last_launches, 0x7fffffff);
    case 8: return (int)(ctx->last_tree_ms * 1e6f);     // ns, mean tree-pass launch of the last stream call (lock-step)
    case 9: return (int)(ctx->last_net_ms * 1e6f);      // ns, mean network launch
    case 10: return (int)std::min<long long>(ctx->last_passes, 0x7fffffff);
    case 7: {                                           // occupied entries of the evaluation memo (synchronises the device)
        if (!ctx->d.memo) return 0;
        cudaSetDevice(ctx->device);
        cudaMemset(ctx->stats_dev + 3, 0, sizeof(unsigned long long));
        k_memo_count<<<148 * 8, 256>>>(ctx->d.memo, (size_t)1 << ctx->memo_log2, ctx->stats_dev + 3);
        unsigned long long h = 0;
        if (cudaMemcpy(&h, ctx->stats_dev + 3, sizeof(h), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
        return (int)std::min<unsigned long long>(h, 0x7fffffffULL);
    }
    default: return -1;
    }
}

extern "C" int c4_ctx_set_net(c4_ctx *ctx, c4_net *net)
{
    C4_REQUIRE(ctx, "c4_ctx_set_net: null context");
    C4_REQUIRE(!net || c4_net_device(net) == ctx->device, "c4_ctx_set_net: the network lives on another CUDA device than the context");
    C4_CUDA(cudaSetDevice(ctx->device));
    if (ctx->memo_log2 > 0) {
        // the memo caches THIS network's outputs: (re)start empty whenever the evaluator changes
        if (!ctx->d.memo) {
            // the memo is a cache: when the device cannot spare the preferred size it is halved down to 2^18 entries
            uint32_t *m = nullptr;
            while (cudaMalloc((void **)&m, ((size_t)1 << ctx->memo_log2) * 64) != cudaSuccess) {
                cudaGetLastError();
                m = nullptr;
                if (--ctx->memo_log2 < 18) { c4_set_error("cudaMalloc of the evaluation memo failed"); ctx->memo_log2 = 0; return -2; }
            }
            ctx->allocs.push_back(m);
            ctx->d.memo = m;
            ctx->d.memo_mask = (uint32_t)(((size_t)1 << ctx->memo_log2) - 1);
        }
        const size_t bytes = ((size_t)1 << ctx->memo_log2) * 64;
        if (c4_net_uid(net) != ctx->memo_net_uid) C4_CUDA(cudaMemset(ctx->d.memo, 0, bytes));
        ctx->memo_net_uid = c4_net_uid(net);
    }
    ctx->net = net;
    ctx->d.memo_dedup = (ctx->d.memo && !getenv("C4_MEMO_NO_DEDUP")) ? 1 : 0;
    // Self-play with a 64-filter network is network-bound (124 us network vs 41 us tree per pass): there the two half
    // pools on two streams pay -- the tree pass of one half runs under the network launch of the other (+7-9 %,
    // tools/ramp64.py) -- while with the 32-filter network the game chains are the limit and one pool is faster.
    if (!getenv("C4_POOLS")) ctx->n_pools = (c4_net_filters(net) == 64 && ctx->max_games >= 512) ? 2 : 1;
    if (!getenv("C4_NET_CTAS")) ctx->net_ctas = (ctx->n_pools == 2 && c4_net_filters(net) == 64) ? 96 : 112;
    return 0;
}

extern "C" int c4_ctx_set_rng(c4_ctx *ctx, int mode, uint64_t seed, double *noise, double *uniform, int record)
{
    C4_REQUIRE(ctx, "c4_ctx_set_rng: null context");
    C4_REQUIRE(mode >= 0 && mode <= 2, "rng mode must be 0 (none), 1 (philox) or 2 (injected)");
    C4_REQUIRE(mode != C4_RNG_INJECTED || (noise && uniform), "injected rng needs noise and uniform buffers");
    C4_REQUIRE(!record || (noise && uniform), "recording needs noise and uniform buffers");
    ctx->d.rng_mode = mode; ctx->d.seed = seed; ctx->d.noise = noise; ctx->d.uniform = uniform;
    ctx->d.rng_record = record;
    return 0;
}

int c4_net_forward_ex(c4_net *net, const uint64_t *c0, const uint64_t *c1, int64_t n, const int32_t *count, float *out,
                      void *stream, int max_ctas);

// a NET self-play pass ends once this many games of the pool wait (stop_frac of the live games; steps of 64 so that the
// captured launch graphs survive the slow decline of the live games in the drain of a generation)
static int pass_stop_count(const c4_ctx *ctx, int n_games)
{
    if (ctx->stop_frac <= 0.0) return 0;
    const long long live = std::min<long long>(ctx->live_games, (long long)n_games);
    const int stop = std::max(1, (int)(ctx->stop_frac * (double)live));
    return stop > 64 ? stop & ~63 : stop;
}

// one tree pass over games [g0, g0 + n_games) of pool `pool`
template <bool SP>
static int launch_advance_pool(c4_ctx *ctx, int mode, int g0, int n_games, int pool, int parity, int budget, cudaStream_t s)
{
    const int threads = 128, wpb = threads / 32;
    const int blocks = (n_games + wpb - 1) / wpb;
    switch (mode) {
    case C4_EVAL_EXTERNAL: k_advance<C4_EVAL_EXTERNAL, SP><<<blocks, threads, 0, s>>>(ctx->d, g0, n_games, pool, parity, budget, 0LL, 0); break;
    case C4_EVAL_CENTRE: k_advance<C4_EVAL_CENTRE, SP><<<blocks, threads, 0, s>>>(ctx->d, g0, n_games, pool, parity, budget, 0LL, 0); break;
    case C4_EVAL_NET: {
        const int stop = SP ? pass_stop_count(ctx, n_games) : 0;
        k_advance<C4_EVAL_NET, SP><<<blocks, threads, 0, s>>>(ctx->d, g0, n_games, pool, parity, budget, ctx->cycle_limit, stop);
        break;
    }
    default: c4_set_error("bad eval kind"); return -1;
    }
    C4_CUDA(cudaGetLastError());
    return 0;
}

template <bool SP>
static int launch_advance(c4_ctx *ctx, int mode, int n_games, int budget, cudaStream_t s)
{
    ctx->parity ^= 1;
    return launch_advance_pool<SP>(ctx, mode, 0, n_games, 0, ctx->parity, budget, s);
}

// A failed network call (the caller's evaluator of an external net) leaves games waiting for answers that never came and
// PENDING memo tags nobody will replace: the pool and the search batch must not be continued.  The next
// c4_search_begin / c4_selfplay_run / c4_selfplay_stream starts from fresh slots and a new memo epoch (the abandoned tags
// then read as misses).
static int net_failed(c4_ctx *ctx, int rc)
{
    ctx->pool_fresh = false;
    ctx->search_failed = true;
    return rc;
}

static int run_net(c4_ctx *ctx, cudaStream_t s)
{
    const int rc = c4_net_forward(ctx->net, (const uint64_t *)ctx->d.leaf_c0, (const uint64_t *)ctx->d.leaf_c1,
                                  ctx->max_games, &ctx->d.ctr->leaf_count[0][ctx->parity], ctx->net_out, s);
    return rc ? net_failed(ctx, rc) : 0;
}

static inline void pool_range(const c4_ctx *ctx, int pool, int *g0, int *n)
{
    if (ctx->n_pools == 1) { *g0 = 0; *n = ctx->max_games; return; }
    const int half = (ctx->max_games + 1) / 2;
    *g0 = pool ? half : 0;
    *n = pool ? ctx->max_games - half : half;
}

extern "C" int c4_search_begin(c4_ctx *ctx, const uint64_t *c0, const uint64_t *c1, int32_t n, void *stream)
{
    C4_REQUIRE(ctx && (n == 0 || (c0 && c1)), "c4_search_begin: null pointer");
    C4_REQUIRE(n >= 0 && n <= ctx->max_games, "c4_search_begin: n exceeds max_games");
    C4_CUDA(cudaSetDevice(ctx->device));
    ctx->d.n_games_target = 0;
    ctx->d.records_out = nullptr;
    ctx->pool_fresh = false;
    ctx->d.memo_epoch++;
    k_search_begin<<<(ctx->max_games + 127) / 128, 128, 0, (cudaStream_t)stream>>>(ctx->d, (const u64 *)c0,
                                                                                   (const u64 *)c1, n, ctx->max_games);
    C4_CUDA(cudaGetLastError());
    ctx->parity = 0;
    ctx->n_search = n;
    ctx->last_pending = 0;
    ctx->supplied = true;
    ctx->search_failed = false;
    return 0;
}

extern "C" int c4_search_pending(c4_ctx *ctx, uint64_t *leaf_c0, uint64_t *leaf_c1, int32_t *leaf_game,
                                 int32_t *n_pending, void *stream)
{
    C4_REQUIRE(ctx && n_pending, "c4_search_pending: null pointer");
    C4_REQUIRE(ctx->supplied || ctx->last_pending == 0, "c4_search_pending: previous leaves were not supplied");
    cudaStream_t s = (cudaStream_t)stream;
    C4_CUDA(cudaSetDevice(ctx->device));
    int rc = launch_advance<false>(ctx, C4_EVAL_EXTERNAL, ctx->max_games, 0x7fffffff, s);
    if (rc) return rc;
    C4_CUDA(cudaMemcpyAsync(ctx->pinned, &ctx->d.ctr->leaf_count[0][ctx->parity], sizeof(int), cudaMemcpyDeviceToHost, s));
    C4_CUDA(cudaStreamSynchronize(s));
    int m = *(int *)ctx->pinned;
    if (m > 0) {
        if (leaf_c0) C4_CUDA(cudaMemcpyAsync(leaf_c0, ctx->d.leaf_c0, m * sizeof(u64), cudaMemcpyDeviceToDevice, s));
        if (leaf_c1) C4_CUDA(cudaMemcpyAsync(leaf_c1, ctx->d.leaf_c1, m * sizeof(u64), cudaMemcpyDeviceToDevice, s));
        if (leaf_game) C4_CUDA(cudaMemcpyAsync(leaf_game, ctx->d.leaf_game, m * sizeof(int), cudaMemcpyDeviceToDevice, s));
    }
    *n_pending = m;
    ctx->last_pending = m;
    ctx->supplied = (m == 0);
    return 0;
}

extern "C" int c4_search_supply(c4_ctx *ctx, const double *value, const void *prior, int prior_dtype, int32_t m,
                                void *stream)
{
    C4_REQUIRE(ctx && value && prior, "c4_search_supply: null pointer");
    C4_REQUIRE(m == ctx->last_pending, "c4_search_supply: m must equal the last pending count");
    C4_REQUIRE(prior_dtype == 0 || prior_dtype == 1, "prior_dtype must be 0 (fp64) or 1 (fp32)");
    cudaStream_t s = (cudaStream_t)stream;
    C4_CUDA(cudaSetDevice(ctx->device));
    C4_CUDA(cudaMemcpyAsync(ctx->ext_value, value, (size_t)m * sizeof(double), cudaMemcpyDeviceToDevice, s));
    C4_CUDA(cudaMemcpyAsync(ctx->ext_prior, prior, (size_t)m * 7 * (prior_dtype ? 4 : 8), cudaMemcpyDeviceToDevice, s));
    ctx->d.ext_prior_dtype = prior_dtype;
    ctx->supplied = true;
    return 0;
}

static int read_counters(c4_ctx *ctx, C4Counters *host, cudaStream_t s)
{
    C4_CUDA(cudaMemcpyAsync(ctx->pinned, ctx->d.ctr, sizeof(C4Counters), cudaMemcpyDeviceToHost, s));
    C4_CUDA(cudaStreamSynchronize(s));
    memcpy(host, ctx->pinned, sizeof(C4Counters));
    return 0;
}

// the two device-side failure words: a network answer that was not finite, and the fused engine's watchdog
static int check_device_errors(const c4_ctx *ctx, const C4Counters &c)
{
    if (c.net_nonfinite && c4_net_external(ctx->net)) {
        c4_set_error("the caller's evaluator returned a non-finite value or prior: oinkoink/neural/pytorch/model.py:258-263 "
                     "asserts here");
        return -3;
    }
    if (c.net_nonfinite) {
        c4_set_error("the network produced a non-finite value or prior (fp16 operand overflow or NaN weights; try "
                     "operand_dtype='bf16'): oinkoink/neural/pytorch/model.py:258-263 asserts here");
        return -3;
    }
    if (c.engine_error) { c4_set_error("fused engine watchdog: games waited for the network for seconds (internal error)"); return -4; }
    return 0;
}

// a persistent engine (split or fused) instead of lock-step passes for `live_games` games in flight?
static bool use_fused(const c4_ctx *ctx, int eval_kind, long long live_games)
{
    return eval_kind == C4_EVAL_NET &&
           (c4_split_eligible(ctx->net, ctx->max_games, live_games) || c4_fused_eligible(ctx->net, ctx->max_games, live_games));
}

// one persistent launch (pair) over the pool; *engine = 3 (split) or 2 (fused)
static int persistent_run(c4_ctx *ctx, long long live_games, bool selfplay, unsigned long long stop_games, double stop_ms,
                          cudaStream_t s, int *engine = nullptr)
{
    const bool split = c4_split_eligible(ctx->net, ctx->max_games, live_games);
    if (engine) *engine = split ? 3 : 2;
    return split ? c4_split_run(ctx->d, ctx->net, ctx->max_games, ctx->cfg.simulations, selfplay, stop_games, stop_ms, s)
                 : c4_fused_run(ctx->d, ctx->net, ctx->max_games, ctx->cfg.simulations, selfplay, stop_games, stop_ms, s);
}

extern "C" int c4_search_run(c4_ctx *ctx, int eval_kind, void *stream)
{
    C4_REQUIRE(ctx, "c4_search_run: null context");
    C4_REQUIRE(eval_kind == C4_EVAL_CENTRE || eval_kind == C4_EVAL_NET, "c4_search_run: eval_kind must be CENTRE or NET");
    C4_REQUIRE(eval_kind != C4_EVAL_NET || ctx->net, "c4_search_run: no network attached (c4_ctx_set_net)");
    C4_REQUIRE(!ctx->search_failed, "c4_search_run: the network failed during the last search; start again with c4_search_begin");
    cudaStream_t s = (cudaStream_t)stream;
    C4_CUDA(cudaSetDevice(ctx->device));
    int rc;
    if (eval_kind == C4_EVAL_CENTRE) {
        // the whole search of every game in one launch: evaluator fused into the tree kernel
        if ((rc = launch_advance<false>(ctx, C4_EVAL_CENTRE, ctx->max_games, 0x7fffffff, s))) return rc;
        C4_CUDA(cudaStreamSynchronize(s));
        return 0;
    }
    C4Counters c;
    if (use_fused(ctx, eval_kind, ctx->n_search)) {
        // every search of the batch in ONE persistent launch (c4_fused.cu)
        if ((rc = persistent_run(ctx, ctx->n_search, false, 0ULL, 0.0, s))) return rc;
        if ((rc = read_counters(ctx, &c, s))) return rc;
        if ((rc = check_device_errors(ctx, c))) return rc;
        C4_REQUIRE((long long)c.n_done >= ctx->n_search, "c4_search_run: the fused engine left searches unfinished");
        return 0;
    }
    const int chunk = 32;
    for (long long it = 0;; it++) {
        for (int k = 0; k < chunk; k++) {
            if ((rc = launch_advance<false>(ctx, C4_EVAL_NET, ctx->max_games, ctx->budget_net, s))) return rc;
            if ((rc = run_net(ctx, s))) return rc;
        }
        if ((rc = read_counters(ctx, &c, s))) return rc;
        if ((rc = check_device_errors(ctx, c))) return rc;
        if ((long long)c.n_done >= ctx->n_search) break;
        C4_REQUIRE(it < (1 << 20), "c4_search_run: did not terminate");
    }
    return 0;
}

extern "C" int c4_search_readout(c4_ctx *ctx, int32_t n, int32_t *visits, double *value_sum, int8_t *child_result,
                                 int32_t *root_visits, double *root_value_sum, double *root_prior,
                                 double *values_policy, double *visit_policy, int8_t *best_move, double *best_value,
                                 int32_t *n_nodes, void *stream)
{
    C4_REQUIRE(ctx, "c4_search_readout: null context");
    C4_REQUIRE(n >= 0 && n <= ctx->max_games, "c4_search_readout: n exceeds max_games");
    if (n == 0) return 0;
    C4_CUDA(cudaSetDevice(ctx->device));
    k_readout<<<(n + 3) / 4, 128, 0, (cudaStream_t)stream>>>(ctx->d, n, visits, value_sum, child_result, root_visits,
                                                            root_value_sum, root_prior, values_policy, visit_policy,
                                                            best_move, best_value, n_nodes);
    C4_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int c4_search_export_tree(c4_ctx *ctx, int32_t game, void *nodes_out, int64_t capacity_slots,
                                     int64_t *n_slots, void *stream)
{
    C4_REQUIRE(ctx && nodes_out && n_slots, "c4_search_export_tree: null pointer");
    C4_REQUIRE(game >= 0 && game < ctx->max_games, "c4_search_export_tree: bad game index");
    cudaStream_t s = (cudaStream_t)stream;
    C4_CUDA(cudaSetDevice(ctx->device));
    C4_CUDA(cudaMemcpyAsync(ctx->pinned, ctx->d.n_blocks + game, sizeof(int), cudaMemcpyDeviceToHost, s));
    C4_CUDA(cudaStreamSynchronize(s));
    int64_t slots = (int64_t)(*(int *)ctx->pinned) * C4_SLOTS;
    C4_REQUIRE(slots <= capacity_slots, "c4_search_export_tree: output buffer too small");
    C4_CUDA(cudaMemcpyAsync(nodes_out, ctx->d.pool + (size_t)game * ctx->d.blocks_per_game * C4_SLOTS,
                            (size_t)slots * sizeof(C4Node), cudaMemcpyDeviceToHost, s));
    C4_CUDA(cudaStreamSynchronize(s));
    *n_slots = slots;
    return 0;
}

// `sample_every` > 0: bracket every sample_every-th pass's launches (of half pool 0) with CUDA events (<= N_SAMPLES samples).
// With two half pools the launches go to two internal streams (forked from / joined to the caller's stream), so the
// tree pass of one half overlaps the network launch of the other; the network launch is capped at net_ctas CTAs so
// the tree blocks find free SMs.
static int selfplay_passes(c4_ctx *ctx, int eval_kind, int n_passes, cudaStream_t s, int sample_every = 0,
                           int *n_sampled = nullptr, int first_sample = 0, bool capturing = false)
{
    int rc, ns = first_sample;
    // (inside a stream capture an event that is read from the host afterwards must be recorded as an external one)
    const unsigned ev_flags = capturing ? cudaEventRecordExternal : cudaEventRecordDefault;
    const bool two = ctx->n_pools == 2 && eval_kind == C4_EVAL_NET;
    if (two) {
        C4_CUDA(cudaEventRecord(ctx->ev_fork, s));
        for (int p = 0; p < 2; p++) C4_CUDA(cudaStreamWaitEvent(ctx->pool_stream[p], ctx->ev_fork, 0));
    }
    for (int k = 0; k < n_passes; k++) {
        const bool sample = sample_every > 0 && (k % sample_every) == sample_every / 2 && ns < N_SAMPLES;
        if (!two) {
            if (sample) C4_CUDA(cudaEventRecordWithFlags(ctx->eva[2 * ns], s, ev_flags));
            if (eval_kind == C4_EVAL_CENTRE) {
                if ((rc = launch_advance<true>(ctx, C4_EVAL_CENTRE, ctx->max_games, 512, s))) return rc;
                if (sample) C4_CUDA(cudaEventRecordWithFlags(ctx->eva[2 * ns + 1], s, ev_flags));
            } else {
                if ((rc = launch_advance<true>(ctx, C4_EVAL_NET, ctx->max_games, ctx->budget_net, s))) return rc;
                if (sample) { C4_CUDA(cudaEventRecordWithFlags(ctx->eva[2 * ns + 1], s, ev_flags)); C4_CUDA(cudaEventRecordWithFlags(ctx->evs[2 * ns], s, ev_flags)); }
                if ((rc = run_net(ctx, s))) return rc;
                if (sample) C4_CUDA(cudaEventRecordWithFlags(ctx->evs[2 * ns + 1], s, ev_flags));
            }
        } else {
            for (int p = 0; p < 2; p++) {
                cudaStream_t ps = ctx->pool_stream[p];
                int g0, n;
                pool_range(ctx, p, &g0, &n);
                ctx->pool_parity[p] ^= 1;
                const bool smp = sample && p == 0;
                if (smp) C4_CUDA(cudaEventRecordWithFlags(ctx->eva[2 * ns], ps, ev_flags));
                if ((rc = launch_advance_pool<true>(ctx, C4_EVAL_NET, g0, n, p, ctx->pool_parity[p], ctx->budget_net, ps))) return rc;
                if (smp) { C4_CUDA(cudaEventRecordWithFlags(ctx->eva[2 * ns + 1], ps, ev_flags)); C4_CUDA(cudaEventRecordWithFlags(ctx->evs[2 * ns], ps, ev_flags)); }
                if ((rc = c4_net_forward_ex(ctx->net, (const uint64_t *)(ctx->d.leaf_c0 + g0), (const uint64_t *)(ctx->d.leaf_c1 + g0),
                                            n, &ctx->d.ctr->leaf_count[p][ctx->pool_parity[p]], ctx->net_out + (size_t)g0 * 8, ps,
                                            ctx->net_ctas))) return net_failed(ctx, rc);
                if (smp) C4_CUDA(cudaEventRecordWithFlags(ctx->evs[2 * ns + 1], ps, ev_flags));
            }
        }
        if (sample) ns++;
    }
    if (two) {
        for (int p = 0; p < 2; p++) {
            C4_CUDA(cudaEventRecord(ctx->ev_join[p], ctx->pool_stream[p]));
            C4_CUDA(cudaStreamWaitEvent(s, ctx->ev_join[p], 0));
        }
    }
    if (n_sampled) *n_sampled = ns;
    return 0;
}

// One chunk of 64 lock-step passes.  With one pool and the network evaluator the 128 launches are replayed from a CUDA
// graph captured the first time (and again whenever a launch parameter changes: the stop count follows the number of
// live games in the drain of a generation, the kernel arguments hold the context's device pointers and RNG settings): the
// launches then follow each other on the device without host work in between.  C4_NO_GRAPH=1 keeps the plain launches.
// A network served by the caller is host code between the launches, so its passes are never captured.
static int selfplay_chunk(c4_ctx *ctx, int eval_kind, cudaStream_t s, bool sampled = false)
{
    static const bool no_graph = getenv("C4_NO_GRAPH") != nullptr;
    const bool two = ctx->n_pools == 2 && eval_kind == C4_EVAL_NET;
    int ns = 0;
    if (no_graph || two || eval_kind != C4_EVAL_NET || ctx->parity != 0 || c4_net_external(ctx->net))
        return selfplay_passes(ctx, eval_kind, 64, s, sampled ? 64 : 0, &ns, 0);
    const int gi = sampled ? 1 : 0;
    const int stop = pass_stop_count(ctx, ctx->max_games);
    // everything the captured kernel arguments depend on (C4Dev is passed by value)
    unsigned long long h = 1469598103934665603ULL;
    const unsigned char *raw = reinterpret_cast<const unsigned char *>(&ctx->d);
    for (size_t i = 0; i < sizeof(C4Dev); i++) h = (h ^ raw[i]) * 1099511628211ULL;
    const unsigned long long key[4] = {h, (unsigned long long)stop | ((unsigned long long)ctx->budget_net << 32),
                                       (unsigned long long)ctx->cycle_limit, c4_net_uid(ctx->net)};
    // capture and replay on an internal stream (the caller's may be the legacy default stream, which cannot be captured),
    // forked from / joined to the caller's stream with events
    cudaStream_t cs = ctx->pool_stream[0];
    if (!ctx->chunk_graph[gi] || memcmp(key, ctx->chunk_key[gi], sizeof(key))) {
        if (ctx->chunk_graph[gi]) { cudaGraphExecDestroy(ctx->chunk_graph[gi]); ctx->chunk_graph[gi] = nullptr; }
        cudaGraph_t g = nullptr;
        C4_CUDA(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
        int rc = selfplay_passes(ctx, eval_kind, 64, cs, sampled ? 64 : 0, &ns, 0, true);
        cudaError_t e = cudaStreamEndCapture(cs, &g);
        if (rc) { if (g) cudaGraphDestroy(g); return rc; }
        C4_CUDA(e);
        e = cudaGraphInstantiate(&ctx->chunk_graph[gi], g, 0);
        cudaGraphDestroy(g);
        C4_CUDA(e);
        memcpy(ctx->chunk_key[gi], key, sizeof(key));
    }
    C4_CUDA(cudaEventRecord(ctx->ev_fork, s));
    C4_CUDA(cudaStreamWaitEvent(cs, ctx->ev_fork, 0));
    C4_CUDA(cudaGraphLaunch(ctx->chunk_graph[gi], cs));
    C4_CUDA(cudaEventRecord(ctx->ev_join[0], cs));
    C4_CUDA(cudaStreamWaitEvent(s, ctx->ev_join[0], 0));
    return 0;
}

extern "C" int c4_selfplay_run(c4_ctx *ctx, int eval_kind, int64_t n_games, int64_t game_id_base,
                               int64_t game_id_stride, const uint64_t *start_c0, const uint64_t *start_c1,
                               c4_record *records_out, int64_t max_records, int64_t *n_records_out, void *stream)
{
    C4_REQUIRE(ctx && records_out && n_records_out, "c4_selfplay_run: null pointer");
    C4_REQUIRE(eval_kind == C4_EVAL_CENTRE || eval_kind == C4_EVAL_NET, "c4_selfplay_run: eval_kind must be CENTRE or NET");
    C4_REQUIRE(eval_kind != C4_EVAL_NET || ctx->net, "c4_selfplay_run: no network attached (c4_ctx_set_net)");
    C4_REQUIRE(n_games >= 0 && max_records >= 0, "c4_selfplay_run: negative size");
    C4_REQUIRE(ctx->d.rng_mode != C4_RNG_NONE || (!ctx->d.noise_on && ctx->d.n_sampling <= 0),
               "c4_selfplay_run: the config asks for root noise or sampled moves but no RNG is set (c4_ctx_set_rng): every "
               "slot would play the same game");
    cudaStream_t s = (cudaStream_t)stream;
    C4_CUDA(cudaSetDevice(ctx->device));
    C4Dev &d = ctx->d;
    d.n_games_target = n_games;
    d.game_id_base = game_id_base; d.game_id_stride = game_id_stride;
    d.start_c0 = (const u64 *)start_c0; d.start_c1 = (const u64 *)start_c1;
    d.records_out = records_out; d.max_records = max_records;
    ctx->pool_fresh = false;
    d.memo_epoch++;
    k_selfplay_init<<<(ctx->max_games + 127) / 128, 128, 0, s>>>(d, ctx->max_games);
    C4_CUDA(cudaGetLastError());
    ctx->parity = 0;
    ctx->pool_parity[0] = ctx->pool_parity[1] = 0;
    int rc;
    C4Counters c;
    ctx->pool_engine = 0;
    if (use_fused(ctx, eval_kind, std::min<long long>(n_games, ctx->max_games))) {
        // the whole generation in ONE persistent launch: slots go idle when no game is left to seed, CTAs leave when
        // all their slots are idle (c4_fused.cu)
        if ((rc = persistent_run(ctx, std::min<long long>(n_games, ctx->max_games), true, 0ULL, 0.0, s))) return rc;
        if ((rc = read_counters(ctx, &c, s))) return rc;
        if ((rc = check_device_errors(ctx, c))) return rc;
        C4_REQUIRE((long long)c.games_finished >= n_games, "c4_selfplay_run: the fused engine left games unfinished");
    } else {
        ctx->live_games = std::min<long long>(n_games, ctx->max_games);
        for (long long it = 0;; it++) {
            if ((rc = selfplay_chunk(ctx, eval_kind, s))) return rc;
            if ((rc = read_counters(ctx, &c, s))) return rc;
            if ((rc = check_device_errors(ctx, c))) return rc;
            ctx->live_games = std::max<long long>(1, std::min<long long>(n_games - (long long)c.games_finished, ctx->max_games));
            if ((long long)c.games_finished >= n_games) break;
            if (use_fused(ctx, eval_kind, ctx->live_games)) {
                // the drain of a generation: few games are left in flight, and a pass costs the same launches and the same
                // network latency for 500 games as for 4,096.  Hand the pool over to the fused engine: one consume-only
                // pass (every answered leaf is applied, nothing new is requested), then one persistent launch to the end.
                if (ctx->n_pools == 2 && eval_kind == C4_EVAL_NET) {
                    for (int p = 0; p < 2; p++) {
                        int g0, n;
                        pool_range(ctx, p, &g0, &n);
                        ctx->pool_parity[p] ^= 1;
                        if ((rc = launch_advance_pool<true>(ctx, eval_kind, g0, n, p, ctx->pool_parity[p], -1, s))) return rc;
                    }
                } else if ((rc = launch_advance<true>(ctx, eval_kind, ctx->max_games, -1, s))) return rc;
                if ((rc = persistent_run(ctx, ctx->live_games, true, 0ULL, 0.0, s))) return rc;
                if ((rc = read_counters(ctx, &c, s))) return rc;
                if ((rc = check_device_errors(ctx, c))) return rc;
                C4_REQUIRE((long long)c.games_finished >= n_games, "c4_selfplay_run: the fused engine left games unfinished");
                break;
            }
            C4_REQUIRE(it < (1LL << 24), "c4_selfplay_run: did not terminate");
        }
    }
    C4_REQUIRE(c.overflow == 0, "c4_selfplay_run: records_out too small");
    *n_records_out = (int64_t)c.n_records;
    return 0;
}

extern "C" int c4_selfplay_reset(c4_ctx *ctx, void *stream)
{
    C4_REQUIRE(ctx, "c4_selfplay_reset: null context");
    ctx->pool_fresh = false;
    return 0;
}

extern "C" int c4_selfplay_bench(c4_ctx *ctx, int eval_kind, int64_t iterations, int64_t *positions, int64_t *evals,
                                 int64_t *sims, int64_t *games, float *device_ms, float *net_ms, float *tree_ms,
                                 void *stream)
{
    C4_REQUIRE(ctx, "c4_selfplay_bench: null context");
    C4_REQUIRE(eval_kind == C4_EVAL_CENTRE || eval_kind == C4_EVAL_NET, "c4_selfplay_bench: eval_kind must be CENTRE or NET");
    C4_REQUIRE(eval_kind != C4_EVAL_NET || ctx->net, "c4_selfplay_bench: no network attached (c4_ctx_set_net)");
    cudaStream_t s = (cudaStream_t)stream;
    C4_CUDA(cudaSetDevice(ctx->device));
    C4Dev &d = ctx->d;
    int rc;
    if (ctx->pool_engine != 1) ctx->pool_fresh = false;      // the pool state of another engine cannot be continued
    ctx->pool_engine = 1;
    if (!ctx->pool_fresh) {
        d.n_games_target = (long long)1 << 60;
        ctx->live_games = ctx->max_games;
        d.game_id_base = 0; d.game_id_stride = 1;
        d.start_c0 = nullptr; d.start_c1 = nullptr;
        d.records_out = nullptr; d.max_records = 0;
        d.memo_epoch++;
    k_selfplay_init<<<(ctx->max_games + 127) / 128, 128, 0, s>>>(d, ctx->max_games);
        C4_CUDA(cudaGetLastError());
        ctx->parity = 0;
        ctx->pool_parity[0] = ctx->pool_parity[1] = 0;
        ctx->pool_fresh = true;
    }
    unsigned long long before[4], after[4];
    C4Counters c;
    k_sum_stats<<<1, 256, 0, s>>>(d.stat_evals, d.stat_positions, d.stat_hits, ctx->max_games, ctx->stats_dev);
    C4_CUDA(cudaMemcpyAsync(ctx->pinned + 40, ctx->stats_dev, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    if ((rc = read_counters(ctx, &c, s))) return rc;
    before[0] = ctx->pinned[40]; before[1] = ctx->pinned[41]; before[2] = c.games_finished; before[3] = ctx->pinned[42];
    int n_sampled = 0;
    const int sample_every = (net_ms || tree_ms) ? (int)std::max<int64_t>(1, iterations / N_SAMPLES) : 0;
    C4_CUDA(cudaEventRecord(ctx->ev0, s));
    if ((rc = selfplay_passes(ctx, eval_kind, (int)iterations, s, sample_every, &n_sampled))) return rc;
    C4_CUDA(cudaEventRecord(ctx->ev1, s));
    k_sum_stats<<<1, 256, 0, s>>>(d.stat_evals, d.stat_positions, d.stat_hits, ctx->max_games, ctx->stats_dev);
    C4_CUDA(cudaMemcpyAsync(ctx->pinned + 40, ctx->stats_dev, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    if ((rc = read_counters(ctx, &c, s))) return rc;
    after[0] = ctx->pinned[40]; after[1] = ctx->pinned[41]; after[2] = c.games_finished; after[3] = ctx->pinned[42];
    ctx->last_memo_hits = (long long)(after[3] - before[3]);
    float ms = 0.f;
    C4_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    if (evals) *evals = (int64_t)(after[0] - before[0]);
    if (positions) *positions = (int64_t)(after[1] - before[1]);
    if (sims) *sims = (int64_t)(after[1] - before[1]) * ctx->cfg.simulations;
    if (games) *games = (int64_t)(after[2] - before[2]);
    if (device_ms) *device_ms = ms;
    // mean duration of the sampled launches (events on the launching stream)
    float nsum = 0.f, tsum = 0.f;
    for (int i = 0; i < n_sampled; i++) {
        float t = 0.f;
        if (eval_kind == C4_EVAL_NET) { C4_CUDA(cudaEventElapsedTime(&t, ctx->evs[2 * i], ctx->evs[2 * i + 1])); nsum += t; }
        C4_CUDA(cudaEventElapsedTime(&t, ctx->eva[2 * i], ctx->eva[2 * i + 1]));
        tsum += t;
    }
    if (net_ms) *net_ms = n_sampled ? nsum / n_sampled : 0.f;
    if (tree_ms) *tree_ms = n_sampled ? tsum / n_sampled : 0.f;
    return 0;
}

extern "C" int c4_ctx_clear_memo(c4_ctx *ctx, void *stream)
{
    C4_REQUIRE(ctx, "c4_ctx_clear_memo: null context");
    C4_CUDA(cudaSetDevice(ctx->device));
    if (ctx->d.memo) C4_CUDA(cudaMemsetAsync(ctx->d.memo, 0, ((size_t)1 << ctx->memo_log2) * 64, (cudaStream_t)stream));
    return 0;
}

extern "C" int c4_selfplay_stream(c4_ctx *ctx, int eval_kind, int reset, int64_t stop_games, double max_ms,
                                  int64_t *positions, int64_t *evals, int64_t *memo_hits, int64_t *games,
                                  float *device_ms, int32_t *engine, void *stream)
{
    C4_REQUIRE(ctx, "c4_selfplay_stream: null context");
    C4_REQUIRE(eval_kind == C4_EVAL_CENTRE || eval_kind == C4_EVAL_NET, "c4_selfplay_stream: eval_kind must be CENTRE or NET");
    C4_REQUIRE(eval_kind != C4_EVAL_NET || ctx->net, "c4_selfplay_stream: no network attached (c4_ctx_set_net)");
    C4_REQUIRE(stop_games > 0 || max_ms > 0.0, "c4_selfplay_stream: needs a game count or a time limit");
    C4_REQUIRE(ctx->d.rng_mode != C4_RNG_NONE || (!ctx->d.noise_on && ctx->d.n_sampling <= 0),
               "c4_selfplay_stream: the config asks for root noise or sampled moves but no RNG is set (c4_ctx_set_rng)");
    cudaStream_t s = (cudaStream_t)stream;
    C4_CUDA(cudaSetDevice(ctx->device));
    C4Dev &d = ctx->d;
    const bool fused = use_fused(ctx, eval_kind, ctx->max_games);
    const int eng = fused ? (c4_split_eligible(ctx->net, ctx->max_games, ctx->max_games) ? 3 : 2) : 1;
    int rc;
    if (reset || !ctx->pool_fresh || ctx->pool_engine != eng) {
        d.n_games_target = (long long)1 << 60;
        ctx->live_games = ctx->max_games;
        d.game_id_base = 0; d.game_id_stride = 1;
        d.start_c0 = nullptr; d.start_c1 = nullptr;
        d.records_out = nullptr; d.max_records = 0;
        d.memo_epoch++;
    k_selfplay_init<<<(ctx->max_games + 127) / 128, 128, 0, s>>>(d, ctx->max_games);
        C4_CUDA(cudaGetLastError());
        ctx->parity = 0;
        ctx->pool_parity[0] = ctx->pool_parity[1] = 0;
        ctx->pool_fresh = true;
        ctx->pool_engine = eng;
    }
    unsigned long long before[4], after[4];
    C4Counters c;
    k_sum_stats<<<1, 256, 0, s>>>(d.stat_evals, d.stat_positions, d.stat_hits, ctx->max_games, ctx->stats_dev);
    C4_CUDA(cudaMemcpyAsync(ctx->pinned + 40, ctx->stats_dev, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    if ((rc = read_counters(ctx, &c, s))) return rc;
    before[0] = ctx->pinned[40]; before[1] = ctx->pinned[41]; before[2] = c.games_finished; before[3] = ctx->pinned[42];
    const unsigned long long games_goal = stop_games > 0 ? before[2] + (unsigned long long)stop_games : 0ULL;
    C4_CUDA(cudaEventRecord(ctx->ev0, s));
    ctx->last_launches = 2;                                  // k_sum_stats before and after
    ctx->last_tree_ms = ctx->last_net_ms = 0.f;
    ctx->last_passes = 0;
    int n_sampled = 0;
    float tree_sum = 0.f, net_sum = 0.f;
    if (fused) {
        if ((rc = persistent_run(ctx, ctx->max_games, true, games_goal, max_ms, s))) return rc;
        ctx->last_launches += eng == 3 ? c4_split_last_launches() : 1;
    } else {
        // lock-step engine: chunks of passes with a host look at the counters in between
        for (long long it = 0;; it++) {
            // one pass of some chunks is bracketed with CUDA events (<= 64 samples over the call): launch durations of the
            // tree pass and the network kernel for the roofline figures
            // (every 8th chunk, up to 64 of them, carries event records around the launches of its pass 32)
            const bool sampled = (it & 7) == 3 && n_sampled < N_SAMPLES;
            if ((rc = selfplay_chunk(ctx, eval_kind, s, sampled))) return rc;
            ctx->last_launches += 64 * (eval_kind == C4_EVAL_NET ? 2 * ctx->n_pools : 1);
            ctx->last_passes += 64;
            C4_CUDA(cudaEventRecord(ctx->ev1, s));
            if ((rc = read_counters(ctx, &c, s))) return rc;
            float ms = 0.f;
            C4_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
            if (sampled) {
                float t = 0.f;
                C4_CUDA(cudaEventElapsedTime(&t, ctx->eva[0], ctx->eva[1]));
                tree_sum += t;
                if (eval_kind == C4_EVAL_NET) { C4_CUDA(cudaEventElapsedTime(&t, ctx->evs[0], ctx->evs[1])); net_sum += t; }
                n_sampled++;
            }
            if (games_goal && c.games_finished >= games_goal) break;
            if (max_ms > 0.0 && ms >= max_ms) break;
            C4_REQUIRE(it < (1LL << 24), "c4_selfplay_stream: did not terminate");
        }
    }
    C4_CUDA(cudaEventRecord(ctx->ev1, s));
    k_sum_stats<<<1, 256, 0, s>>>(d.stat_evals, d.stat_positions, d.stat_hits, ctx->max_games, ctx->stats_dev);
    C4_CUDA(cudaMemcpyAsync(ctx->pinned + 40, ctx->stats_dev, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    if ((rc = read_counters(ctx, &c, s))) return rc;
    if ((rc = check_device_errors(ctx, c))) return rc;
    after[0] = ctx->pinned[40]; after[1] = ctx->pinned[41]; after[2] = c.games_finished; after[3] = ctx->pinned[42];
    float ms = 0.f;
    C4_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    if (!fused && n_sampled > 0) {
        ctx->last_tree_ms = tree_sum / n_sampled;
        ctx->last_net_ms = net_sum / n_sampled;
    }
    if (evals) *evals = (int64_t)(after[0] - before[0]);
    if (positions) *positions = (int64_t)(after[1] - before[1]);
    if (games) *games = (int64_t)(after[2] - before[2]);
    if (memo_hits) *memo_hits = (int64_t)(after[3] - before[3]);
    if (device_ms) *device_ms = ms;
    if (engine) *engine = eng;
    return 0;
}

extern "C" int c4_records_augment_pack(const c4_record *records, int64_t n, float *boards, float *values,
                                       float *priors, void *stream)
{
    C4_REQUIRE(n >= 0 && (n == 0 || (records && boards && values && priors)), "c4_records_augment_pack: null pointer");
    if (n == 0) return 0;
    long long total = n * 63;
    long long blocks = (total + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    k_augment_pack<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(records, n, boards, values, priors);
    C4_CUDA(cudaGetLastError());
    return 0;
}
