/*
 * c4b200.h -- C ABI of libc4b200.so: the B200 (sm_100a) implementation of oinkoink's self-play hot path.
 *
 * The reference (willis-richard/connect4) is pure Python and has no FFI; its boundary for this path is a set of
 * Python call protocols (SURVEY.md 8b).  Every entry point below names the reference interface it replaces
 * (file:line relative to the reference root).  INTEGRATION.md shows the ctypes binding a maintainer would add.
 *
 * Conventions
 *  - plain C: pointers + sizes, no torch / C++ types.  Pointers marked DEVICE are device pointers on the context's
 *    GPU (e.g. tensor.data_ptr()); pointers marked HOST are ordinary host memory.
 *  - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls taking a stream are asynchronous
 *    unless documented otherwise.
 *  - return value: 0 = ok, negative = error (message via c4_last_error(), thread-local).
 *  - there is NO CPU fallback: every compute entry point launches sm_100a kernels and fails if no device is usable.
 *  - bitboards: two uint64 per position, bit c*7+h (column c, height h from the bottom), exactly the reference's
 *    layout (oinkoink/board.py:9-32).  Side to move / age are derived: age = popcount(c0|c1), o moves at even age.
 *  - result codes (int8): -1 = game not over, 0 = x_win, 1 = draw, 2 = o_win; reference Result value = code * 0.5
 *    (oinkoink/utils.py:19-22).
 */
#ifndef C4B200_H
#define C4B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define C4_ABI_VERSION 1

typedef struct c4_ctx c4_ctx;   /* one self-play / search engine on one GPU */
typedef struct c4_net c4_net;   /* one folded value/policy network resident on one GPU */

const char *c4_last_error(void);
int c4_abi_version(void);
/* number of CUDA devices visible; negative on driver error */
int c4_device_count(void);

/* ------------------------------------------------------------------------------------------------------------
 * Bitboard engine (batched; all pointers DEVICE, n positions)
 * ------------------------------------------------------------------------------------------------------------ */
/* Board.valid_moves / _isplayable (oinkoink/board.py:88-92,186-188): bit c of mask[i] set iff column c is
 * playable; 0 when result[i] != -1 (result may be NULL = all games running). */
int c4_board_legal_mask(const uint64_t *c0, const uint64_t *c1, const int8_t *result, uint8_t *mask, int64_t n,
                        void *stream);
/* Board.make_move (oinkoink/board.py:160-170), in place, no legality check (like the reference); entries whose
 * move[i] is negative are left untouched.  result_out[i] receives the new result code. */
int c4_board_drop(uint64_t *c0, uint64_t *c1, const int8_t *move, int8_t *result_out, int64_t n, void *stream);
/* Board._check_terminal_position (oinkoink/board.py:173-184): out[i] = 1 iff bb[i] holds four in a row. */
int c4_board_has_win(const uint64_t *bb, uint8_t *out, int64_t n, void *stream);
/* result derivation of Board.from_pieces (oinkoink/board.py:56-61): o-win, then x-win, then full board. */
int c4_board_result(const uint64_t *c0, const uint64_t *c1, int8_t *result_out, int64_t n, void *stream);
/* Board.create_fliplr / flip_color (oinkoink/board.py:115-145) */
int c4_board_fliplr(const uint64_t *c0, const uint64_t *c1, uint64_t *f0, uint64_t *f1, int64_t n, void *stream);
/* Board.to_array (oinkoink/board.py:147-154): planes [n][3][6][7], row 0 = top; dtype 0 = uint8, 1 = float32,
 * 2 = float16, 3 = bfloat16 (the operand type of a caller-served network, see c4_net_create_external) */
int c4_board_to_planes(const uint64_t *c0, const uint64_t *c1, void *planes, int dtype, int64_t n, void *stream);
/* Board.from_pieces colour part (oinkoink/board.py:43-50): uint8 planes o[n][6][7], x[n][6][7] -> bitboards */
int c4_board_from_planes(const uint8_t *o, const uint8_t *x, uint64_t *c0, uint64_t *c1, int64_t n, void *stream);
/* evaluate_centre (oinkoink/evaluators.py:28-33,47-63): fp64 value per position */
int c4_board_evaluate_centre(const uint64_t *c0, const uint64_t *c1, double *value, int64_t n, void *stream);

/* ------------------------------------------------------------------------------------------------------------
 * Value / policy network (replaces ModelWrapper.__call__/_call_list, oinkoink/neural/pytorch/model.py:171-178,
 * 252-282, and Net.forward, model.py:120-134)
 * ------------------------------------------------------------------------------------------------------------ */
/* `blob` (HOST, float32) is the BN-folded parameter image built by connect4_b200.neural.weights.fold_state_dict:
 *   [0] magic 0xC4B2 [1] filters F [2] n_residuals R [3] n_fc | (operand dtype << 8) | (kernel << 16)
 *       (dtype 0 = fp16, 1 = bf16; kernel 0 = auto: tcgen05 tower for F = 32, 1 = force the mma.sync kernels,
 *       2 = "layers": the layer-by-layer tcgen05 kernels, one launch per conv with the activations in global memory), then
 *   stem W[F][3][3][3] (co,ci,ky,kx), stem b[F]; per residual conv (2R of them): W[F][F][3][3], b[F];
 *   value head: wv[F], bv; fc W[42][42] (the n_fc affine layers pre-multiplied), fc b[42]; fc1 w[42], b; w1, w2;
 *   policy head: wp[2][F], bp[2]; fc W[7][84], b[7].
 * Supported: kernels 0 and 1: F in {32, 64}, 1 <= R <= 16; kernel 2: F a multiple of 16 in 16..256, 1 <= R <= 40, any
 * n_fc.  A geometry outside these is refused before any device is looked for.
 * Kernel 2 networks run on the lock-step pass engine only (the split / fused engines refuse them, also under C4_ENGINE):
 * from 512 game slots on two half pools on two streams (measured faster than one pool), else one pool whose passes are
 * captured into CUDA graphs like the tower's.  An engine context keeps their activations in scratch of its own, one per
 * half pool (allocated by c4_ctx_set_net), so two contexts may share one network. */
int c4_net_create(int device, const float *blob, int64_t n_floats, c4_net **out);
/* A network the CALLER serves (any geometry, any framework): the engine keeps the tree passes, the evaluation memo and
 * its de-duplication, leaf compaction, Philox noise and the records, and hands each compacted leaf batch to `fn`.
 *   fn(user, c0, c1, n, out, stream): c0/c1 (DEVICE, n >= 1 leaves) -> out[i] = {prior[0..6], value} (DEVICE, the rows
 *   c4_net_forward writes).  It is called on the thread that made the engine call, between the tree pass that compacted
 *   the leaves and the next pass; its work must be enqueued on `stream` (a cudaStream_t, NULL = default stream) or
 *   finished before it returns.  A non-zero return fails the engine call ("the caller's evaluator failed"); the context
 *   stays usable: the next c4_search_begin / c4_selfplay_run / c4_selfplay_stream(reset=1) starts clean.
 * The result is an ordinary c4_net: c4_ctx_set_net attaches it (with a fresh memo key), c4_net_forward calls `fn`
 * (after reading a device `count`, which synchronises the stream; n = 0 leaves make no call), c4_net_destroy frees it.
 * c4_net_get and c4_net_flops_per_position return 0 for it.
 * Engine policy: an external network always runs on the lock-step pass engine (the persistent split / fused engines
 * cannot call back into the host in the middle of a launch; C4_ENGINE=split|fused is ignored for it), with one host
 * synchronise per pass, and no pass is captured into a CUDA graph.  A non-finite answer fails the call like one of the
 * built-in tower. */
typedef int (*c4_eval_fn)(void *user, const uint64_t *c0, const uint64_t *c1, int64_t n, float *out, void *stream);
int c4_net_create_external(int device, c4_eval_fn fn, void *user, c4_net **out);
int c4_net_destroy(c4_net *net);
/* out[i] = {prior[0..6], value} as 8 float32 (DEVICE, 32 B per position); `count` (DEVICE int32, may be NULL)
 * overrides n with a device-side position count <= n. 16-bit tensor-core tower (fp16 operands by default, bf16
 * selectable in the blob header), fp32 accumulation, fp32 residual stream.  A layered network (kernel 2) works through
 * the batch in chunks in global scratch owned by the network: calls on different streams or threads are ordered one after
 * the other on the device.  No host synchronise and no allocation on any built-in network. */
int c4_net_forward(c4_net *net, const uint64_t *c0, const uint64_t *c1, int64_t n, const int32_t *count, float *out,
                   void *stream);
/* FLOPs (2*MAC, convs + linears) per position of this network: the roofline numerator (SURVEY.md 8d) */
double c4_net_flops_per_position(const c4_net *net);
/* Network read-out: key 0 = filters, 1 = residual blocks, 2 = operand type of the conv GEMMs (0 fp16, 1 bf16), 3 = k of
 * the power-of-two trunk scale 2^-k chosen at creation so that fp16 operands cannot overflow (0 for networks in the usual
 * range: exactly the unscaled arithmetic), 4 = 1 if the tcgen05 kernel runs it, 5 = largest |activation| (scaled units)
 * of the 512 calibration positions, 6 = kernel that runs it (0 mma.sync, 1 fused tcgen05 tower, 2 layered kernels; key 4
 * is 0 for a layered network).  A non-finite network answer at run time never enters a search tree and makes the
 * engine call fail (the reference asserts: oinkoink/neural/pytorch/model.py:258-263,275-280). */
double c4_net_get(const c4_net *net, int key);

/* ------------------------------------------------------------------------------------------------------------
 * Search / self-play engine (replaces mcts.search + MCTS.make_move, oinkoink/mcts.py:78-202; tree.py:61-147;
 * training_game, neural/training_game.py:8-19; game_pool + InferenceServer, neural/game_pool.py:15-49,
 * neural/inference_server.py:15-76)
 * ------------------------------------------------------------------------------------------------------------ */
typedef struct {
    int32_t simulations;          /* MCTSConfig.simulations        (oinkoink/mcts.py:13-26) */
    double pb_c_base;             /* MCTSConfig.pb_c_base          */
    double pb_c_init;             /* MCTSConfig.pb_c_init          */
    double root_dirichlet_alpha;  /* MCTSConfig.root_dirichlet_alpha       (0 = no noise) */
    double root_exploration_fraction; /* MCTSConfig.root_exploration_fraction */
    int32_t num_sampling_moves;   /* MCTSConfig.num_sampling_moves */
} c4_mcts_config;

enum { C4_EVAL_EXTERNAL = 0, C4_EVAL_CENTRE = 1, C4_EVAL_NET = 2 };
enum { C4_RNG_NONE = 0, C4_RNG_PHILOX = 1, C4_RNG_INJECTED = 2 };

/* One engine = one node pool for `max_games` concurrent trees on `device` (32 B nodes, 8-slot child blocks,
 * simulations+2 blocks per game). */
int c4_ctx_create(int device, int32_t max_games, const c4_mcts_config *cfg, c4_ctx **out);
int c4_ctx_destroy(c4_ctx *ctx);
int c4_ctx_set_config(c4_ctx *ctx, const c4_mcts_config *cfg);   /* simulations must not exceed the created size */
int c4_ctx_set_net(c4_ctx *ctx, c4_net *net);                    /* evaluator for C4_EVAL_NET */
/* engine tuning read-out: key 0 = number of half pools self-play runs (2 = the tree pass of one half overlaps the
 * network launch of the other; env C4_POOLS), 1 = CTA cap of a half-pool network launch (env C4_NET_CTAS),
 * 2 = terminal re-visits played through per pass (env C4_BUDGET), 3 = max_games, 4 = log2(entries) of the evaluation
 * memo (0 = off; env C4_MEMO_LOG2), 5 = memo hits during the last c4_selfplay_bench call, 6 = kernels launched by the
 * last c4_selfplay_stream call, 7 = occupied entries of the evaluation memo (~ distinct positions evaluated so far),
 * 8 / 9 = mean duration in ns of the tree-pass / network launches sampled with CUDA events during the last
 * c4_selfplay_stream call of the lock-step engine, 10 = its number of passes.
 * The evaluation memo mirrors Evaluator.position_table (oinkoink/evaluators.py:18-25; shared by all games of a
 * process for a whole generation, neural/game_pool.py:21-27): network outputs are cached by position and re-used across
 * moves and games; it is emptied by c4_ctx_set_net.  A hit is bit-identical to a network evaluation. */
int c4_ctx_get(c4_ctx *ctx, int key);
/* root-noise / move-sampling randomness (oinkoink/mcts.py:171-181, tree.py:75-82).
 * PHILOX: counter-based, keyed by (seed, global game id, ply).  INJECTED: noise[g][ply][7] raw gamma draws and
 * uniform[g][ply] (DEVICE fp64, g = game slot), e.g. recorded from the reference.  If `record` is non-zero in
 * PHILOX mode the draws used are written to the same two arrays so a run can be replayed by the oracle. */
int c4_ctx_set_rng(c4_ctx *ctx, int mode, uint64_t seed, double *noise, double *uniform, int record);

/* --- stand-alone searches (MCTS.make_move protocol) --- */
/* Start n (<= max_games) searches from the given roots (DEVICE). Roots must not be terminal (the reference never
 * searches a terminal root: mcts.py:102). */
int c4_search_begin(c4_ctx *ctx, const uint64_t *c0, const uint64_t *c1, int32_t n, void *stream);
/* External-evaluator stepping (parity vehicle; lets the host plug ANY evaluator with the reference's protocol
 * `evaluator(board) -> (value, prior[7])`, evaluators.py:18-25):
 *   c4_search_pending: advance every tree until it needs an evaluation; the pending leaves are compacted into
 *     leaf_c0/leaf_c1/leaf_game (DEVICE, capacity n) and their number is returned through n_pending (HOST; this
 *     call synchronises the stream).  0 pending = all searches finished.
 *   c4_search_supply: answers for the leaves of the last c4_search_pending, in the same order: value fp64 [m];
 *     prior [m][7] fp64 (prior_dtype 0) or fp32 (prior_dtype 1); unnormalised over illegal moves (mcts.py:197-202
 *     is applied on the device in the prior's own dtype). */
int c4_search_pending(c4_ctx *ctx, uint64_t *leaf_c0, uint64_t *leaf_c1, int32_t *leaf_game, int32_t *n_pending,
                      void *stream);
int c4_search_supply(c4_ctx *ctx, const double *value, const void *prior, int prior_dtype, int32_t m, void *stream);
/* Run all started searches to completion on the device with the built-in evaluator `eval_kind`
 * (C4_EVAL_CENTRE = evaluators.evaluate_centre_with_prior, fused in the tree kernel; C4_EVAL_NET = the attached
 * c4_net).  Synchronises the stream. */
int c4_search_run(c4_ctx *ctx, int eval_kind, void *stream);
/* Root read-out for the first n games (all DEVICE, any pointer may be NULL):
 *   visits[n][7] int32, value_sum[n][7] fp64, child_result[n][7] int8 (-2 no child, -1 running, else code),
 *   root_visits[n] int32, root_value_sum[n] fp64, root_prior[n][7] fp64,
 *   values_policy[n][7] fp64 (Tree.get_values_policy, tree.py:104-109), visit_policy[n][7] fp64 (tree.py:111-117),
 *   best_move[n] int8 (Tree.best_move, tree.py:69-73), best_value[n] fp64 (child.absolute_value, NaN = None),
 *   n_nodes[n] int32 (node count of the reference's lazily expanded tree). */
int c4_search_readout(c4_ctx *ctx, int32_t n, int32_t *visits, double *value_sum, int8_t *child_result,
                      int32_t *root_visits, double *root_value_sum, double *root_prior, double *values_policy,
                      double *visit_policy, int8_t *best_move, double *best_value, int32_t *n_nodes, void *stream);
/* Copy the node pool of one game to HOST memory (for Tree/NodeData views). nodes_out: capacity*32 bytes;
 * returns the number of 32-byte node slots written through n_slots (8 per block; block 0 slot 0 is the root).
 * Slot layout (little endian): f64 value_sum, u32 visit_count, u32 meta (bit0 exists, bit1 terminal, bits2-3 result code,
 * bits 4.. block index of the children, 0 = not evaluated), f64 prior, f64 side-relative value used by select;
 * slot 7 of a block is its header: f64 position value, 8 zero bytes, f64 0, u32 number of children, u32 parent slot. */
int c4_search_export_tree(c4_ctx *ctx, int32_t game, void *nodes_out, int64_t capacity_slots, int64_t *n_slots,
                          void *stream);

/* --- self-play generation (training_game / game_pool protocol) --- */
/* 64-byte position record, the unit of the generation sink (neural/pytorch/data.py:52-64,78-105). */
typedef struct {
    uint64_t c0, c1;      /* board BEFORE the move (GameData.boards)                         */
    float policy[7];      /* Tree.get_values_policy() (GameData.priors), float32 like data.pth */
    float result_value;   /* game result value for every position (training_game.py:57-60)   */
    float search_value;   /* child.absolute_value returned by make_move (GameData.values); NaN = None */
    int32_t game_id;      /* global game index                                               */
    int8_t move;          /* GameData.moves                                                  */
    int8_t ply;
    int8_t n_moves;       /* length of the finished game                                     */
    int8_t result;        /* result code                                                     */
    int32_t reserved;     /* always 0 (keeps the record 64 bytes and a generation byte-reproducible) */
} c4_record;

/* Play `n_games` complete games (global ids game_id_base + i*game_id_stride) on the context's `max_games` slots,
 * re-seeding a slot as soon as its game ends, every move searched with cfg.simulations simulations and evaluator
 * `eval_kind` (CENTRE or NET).  start_c0/start_c1 (DEVICE, may be NULL = empty board) give per-game start positions
 * indexed by local game number.  Records are appended to records_out (DEVICE, capacity max_records; a game's
 * records are contiguous and in ply order).  n_records_out / n_positions_out (HOST) receive the totals.
 * Synchronises the stream. */
int c4_selfplay_run(c4_ctx *ctx, int eval_kind, int64_t n_games, int64_t game_id_base, int64_t game_id_stride,
                    const uint64_t *start_c0, const uint64_t *start_c1, c4_record *records_out, int64_t max_records,
                    int64_t *n_records_out, void *stream);
/* Steady-state throughput mode for benchmarks: keeps every slot busy (unbounded re-seeding) for `iterations`
 * lock-step passes (one leaf batch each) and reports what was done (HOST outputs): positions = root moves played,
 * evals = evaluator calls, sims = simulations, games = games finished.  Records are discarded.  The pool state
 * persists across calls, so warm-up calls bring it to steady state.  device_ms = CUDA-event time of all passes;
 * net_ms / tree_ms = mean duration of the network launch / tree-pass launch over <= 64 evenly sampled passes
 * (CUDA events on the launching stream; pass NULL for both to disable sampling).  Synchronises the stream. */
int c4_selfplay_bench(c4_ctx *ctx, int eval_kind, int64_t iterations, int64_t *positions, int64_t *evals,
                      int64_t *sims, int64_t *games, float *device_ms, float *net_ms, float *tree_ms, void *stream);
int c4_selfplay_reset(c4_ctx *ctx, void *stream);
/* Continuous self-play on the re-seeding pool, engine-agnostic -- the reference's free-running runtime
 * (neural/game_pool.py:15-49 game threads + neural/inference_server.py:37-63 request loop) as ONE call:
 * `reset` != 0 starts a fresh pool (every slot at ply 0 of a new game, counters zero); otherwise the pool continues where
 * the last call left it.  Runs until `stop_games` more games have finished (0 = no game limit) or `max_ms` device
 * milliseconds have passed (0 = no time limit); at least one of the two must be given.  HOST outputs (any may be NULL):
 * positions = root moves played, evals = network evaluations, memo_hits = leaves answered by the evaluation memo, games =
 * games finished, device_ms = CUDA-event time, engine = 3 when the split persistent engine ran (c4_split.cu, the default for
 * 32- and 64-filter networks: one launch, tree CTAs and tcgen05 tower CTAs on separate SMs, no pass barrier), 2 for the fused
 * persistent engine (c4_fused.cu: tree warps and a tower on every SM), 1 for the lock-step pass engine (env
 * C4_ENGINE=split|fused|lockstep forces one).  Records are discarded.  Synchronises the stream. */
int c4_selfplay_stream(c4_ctx *ctx, int eval_kind, int reset, int64_t stop_games, double max_ms, int64_t *positions,
                       int64_t *evals, int64_t *memo_hits, int64_t *games, float *device_ms, int32_t *engine,
                       void *stream);
/* Empty the evaluation memo (Evaluator.position_table of a new generation, oinkoink/neural/game_pool.py:21-27). */
int c4_ctx_clear_memo(c4_ctx *ctx, void *stream);

/* Generation sink: records -> the reference's data.pth tensors with left-right flip augmentation
 * (native_to_pytorch(add_fliplr=True), neural/pytorch/data.py:78-105): boards [2n][3][6][7] f32, values [2n] f32,
 * priors [2n][7] f32; originals first, mirrors second. All DEVICE. */
int c4_records_augment_pack(const c4_record *records, int64_t n, float *boards, float *values, float *priors,
                            void *stream);

#ifdef __cplusplus
}
#endif
#endif /* C4B200_H */
