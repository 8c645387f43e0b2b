/*
 * gmz.h -- C ABI of the B200-native batched Gumbel-MCTS self-play engine.
 *
 * This is the drop-in boundary for the reference's search hot path
 * (Datou/Datou-gomoku-muzero).  The reference has no FFI: its seam is the Python
 * class pair AlphaZeroMCTS / MuZeroMCTS (mcts.py:191-362) plus the inference
 * queue protocol (mcts.py:73-85, workers.py:314-373).  Each entry point below
 * names the reference code it replaces; datou_gomoku_muzero_b200/{mcts,engine}.py
 * rebuild the reference classes on top through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer unless
 *    the parameter name ends in _host.  The caller (PyTorch) owns every buffer,
 *    including the engine workspace; the library never allocates device memory.
 *  - every call that launches work takes the cudaStream_t to launch on
 *    (gmz_stream, passed as void*) and is asynchronous with respect to the host.
 *  - return value: 0 = OK, non-zero = error; gmz_last_error() gives the text
 *    (thread-local).  There is no CPU fallback behind any entry point.
 *  - G = num_games, A = board_size^2, S = num_simulations, K = num_top_actions.
 *    Actions are r*board_size + c.  "None" last move = -1.
 */
#ifndef GMZ_H
#define GMZ_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GMZ_VERSION 200
#define GMZ_MODE_ALPHAZERO 0 /* AlphaZeroMCTS, mcts.py:191-280 */
#define GMZ_MODE_MUZERO 1    /* MuZeroMCTS,   mcts.py:283-362 */
#define GMZ_MAX_BOARD 19
#define GMZ_MAX_TOP_ACTIONS 32
#define GMZ_WINNER_NONE 2 /* get_game_ended() returned None (game.py:60-63) */

#define GMZ_F32 0  /* values: float32;  observations: float32, NCHW [G,3,N,N] */
#define GMZ_F64 1  /* values: float64 */
#define GMZ_BF16 2 /* observations only: bfloat16, NHWC [G,N,N,3] (channels_last: the network's input format) */
#define GMZ_ACCUM_F64 0 /* gmz_config.accum_dtype */
#define GMZ_ACCUM_F32 1

typedef struct gmz_engine gmz_engine;
typedef void *gmz_stream;

/* The subset of config.py the search reads (config.py:18-34). */
typedef struct gmz_config {
    int32_t board_size;      /* BOARD_SIZE  <= GMZ_MAX_BOARD */
    int32_t n_in_row;        /* N_IN_ROW */
    int32_t num_simulations; /* NUM_SIMULATIONS, 1..32767 */
    int32_t num_top_actions; /* NUM_TOP_ACTIONS, 1..GMZ_MAX_TOP_ACTIONS */
    int32_t mode;            /* GMZ_MODE_* (MCTS_IMPLEMENTATION) */
    int32_t num_games;       /* G: concurrent game trees held by this engine */
    int32_t max_moves;       /* trajectory capacity per game (0 = board_size^2) */
    int32_t accum_dtype;     /* GMZ_ACCUM_*: the dtype the reference's tree arithmetic runs in.  It follows
                              * the evaluator's value scalars (SURVEY.md App. A.7): Python floats (the upstream test
                              * mock) -> float64 = GMZ_ACCUM_F64; np.float32 (the reference's inference server,
                              * workers.py:355,368, NumPy >= 2) -> value_sum / backed-up value / Q / MinMaxStats in
                              * float32 = GMZ_ACCUM_F32.  Visit counts are bit-exact against the reference in
                              * either mode only if the mode matches what the evaluator hands the reference. */
    double c_visit;          /* C_VISIT */
    double c_scale;          /* C_SCALE */
    double minmax_delta;     /* VALUE_MINMAX_DELTA */
    double discount;         /* DISCOUNT */
} gmz_config;

int gmz_version(void);
const char *gmz_last_error(void);

/* Bytes of device workspace gmz_create needs (node pools + per-game state). */
size_t gmz_workspace_bytes(const gmz_config *cfg);

/* Replaces AlphaZeroMCTS(...) / MuZeroMCTS(...) construction (mcts.py:51-56,
 * workers.py:134-142).  `workspace` must stay alive until gmz_destroy and be
 * 256-byte aligned; it is zero-initialised by gmz_create on `stream`. */
int gmz_create(const gmz_config *cfg, void *workspace, size_t workspace_bytes, gmz_stream stream, gmz_engine **out);
int gmz_destroy(gmz_engine *e);

/* ---- root positions ------------------------------------------------------ */
/* Load G root positions: what search() reads off `game` (mcts.py:203,213):
 * boards int8 [G,A] in {-1,0,+1}, players int8 [G] (+-1), last_moves int32 [G]
 * (-1 = None), move_counts int32 [G].  A full board makes that game inactive
 * (search() sentinel, mcts.py:214-215). */
int gmz_set_roots(gmz_engine *e, const int8_t *boards, const int8_t *players, const int32_t *last_moves,
                  const int32_t *move_counts, gmz_stream stream);
/* GomokuGame.reset() (game.py:8-11) for every game with mask[g] != 0 (NULL = all). */
int gmz_games_reset(gmz_engine *e, const uint8_t *mask, gmz_stream stream);
/* GomokuGame.get_board_state at the roots (game.py:12-17): obs [G,3,N,N] float32 (GMZ_F32) or the same
 * planes as bfloat16 in NHWC order (GMZ_BF16). */
int gmz_root_obs(gmz_engine *e, void *obs, int obs_dtype, gmz_stream stream);
/* Read the root positions back (boards int8 [G,A], players, last_moves, move_counts; any may be NULL). */
int gmz_get_roots(gmz_engine *e, int8_t *boards, int8_t *players, int32_t *last_moves, int32_t *move_counts,
                  gmz_stream stream);

/* ---- one search, step by step (external evaluator) ------------------------ */
/* Root expansion + first backup + Gumbel top-k + halving schedule
 * (mcts.py:217-226): logits f32 [G,A], values [G] (value_dtype GMZ_F32/F64),
 * gumbel f64 [G,A] = the np.random.gumbel(0,1,A) draw of each search. */
int gmz_root_expand(gmz_engine *e, const float *logits, const void *values, int value_dtype,
                    const double *gumbel, gmz_stream stream);
/* AlphaZero mode: _select_leaf + path replay on the real board + leaf
 * observation (mcts.py:232-251).  leaf_obs [G,3,N,N] (obs_dtype as gmz_root_obs); optional int32 [G]
 * out_leaf_action / out_leaf_depth for tracing.  Games whose search is
 * complete (sim_count >= S) or inactive write a zero observation. */
int gmz_select(gmz_engine *e, void *leaf_obs, int obs_dtype, int32_t *out_leaf_action, int32_t *out_leaf_depth,
               gmz_stream stream);
/* MuZero mode: the len(selected_children_actions) identical selections of
 * mcts.py:326-332, deduplicated.  Outputs int32 [G]: parent_slot (index of the
 * parent's hidden state, g*S + node), action, child_slot (where the evaluator's
 * next hidden state belongs), or -1 for games with nothing to evaluate;
 * out_reps = len(selected_children_actions), the number of identical rows the
 * reference would have sent and of backups the leaf will receive. */
int gmz_select_mz(gmz_engine *e, int32_t *out_parent_slot, int32_t *out_action, int32_t *out_child_slot,
                  int32_t *out_leaf_depth, int32_t *out_reps, gmz_stream stream);
/* leaf.expand + _backpropagate + sim_count update + sequential halving
 * (mcts.py:260-268 / 340-350): logits f32 [G,A], values [G], rewards [G]
 * (same dtype as values; NULL = 0.0, AlphaZero mode). */
int gmz_expand_backup(gmz_engine *e, const float *logits, const void *values, const void *rewards,
                      int value_dtype, gmz_stream stream);
/* Decision phase (mcts.py:271-280): policy f64 [G,A], value f64 [G], action
 * int32 [G] (-1 for inactive games), optional visits int32 [G,A] (root child
 * visit counts).  Any output may be NULL. */
int gmz_finalize(gmz_engine *e, double *policy, double *value, int32_t *action, int32_t *visits, gmz_stream stream);

/* ---- E0, the fixed deterministic evaluator (DESIGN.md) --------------------- */
/* Stand-alone evaluator kernel over observations obs f32 [B,3,N,N] ->
 * logits f32 [B,A], values f64 [B] (the device twin of tests/golden/e0_py.py).
 * logit_div > 0: quantised logits (k-32)/logit_div, k in 0..63, values k/16; logit_div = 0: DENSE
 * logits (24 random mantissa bits in [-4, 4)) and values in [-1, 1) -- what a network's outputs look
 * like to the search.  Every value / reward E0 produces is exactly representable in float32.
 * The fused kernels (gmz_search_e0, gmz_selfplay_e0) take logit_div = 0 or a power of two (the logit is then
 * one exact multiply); gmz_e0_eval_obs takes any logit_div >= 0. */
int gmz_e0_eval_obs(const float *obs, int batch, int board_size, uint64_t seed, int logit_div,
                    float *logits, double *values, gmz_stream stream);
/* Whole search (root evaluation + S-1 simulations) in ONE persistent kernel
 * with E0 inlined: the tree-only fast path.  In a MuZero-mode engine the in-tree
 * evaluator is E0's recurrent half (hidden state = 64-bit hash per node, reward
 * from the hash) and every evaluation receives len(selected) backups.  gumbel f64 [G,A]; optional int32
 * [G,S] traces (leaf action / depth per evaluation).  Follow with gmz_finalize. */
int gmz_search_e0(gmz_engine *e, const double *gumbel, uint64_t seed, int logit_div,
                  int32_t *trace_leaf_action, int32_t *trace_leaf_depth, gmz_stream stream);
/* Gumbel(0,1) noise on device from a counter-based generator: out f64 [n],
 * element i uses counter (offset + i).  (Parity runs pass NumPy's draw instead.) */
int gmz_fill_gumbel(double *out, size_t n, uint64_t seed, uint64_t offset, gmz_stream stream);

/* ---- persistent self-play (workers.py:162-189 for G games, no host in the loop) ---- */
/* Caller-owned trajectory storage; every pointer is a device pointer.  A game records into
 * one slot; when it ends the slot is pushed on fin_queue (what the reference puts on
 * data_queue, workers.py:230) and the game continues in a fresh slot from the free stack. */
typedef struct gmz_traj {
    int32_t n_slots;       /* >= G */
    int32_t max_moves;     /* moves recorded per game (board_size^2 covers any game from reset) */
    int32_t fin_cap;       /* entries of fin_queue, >= n_slots */
    int32_t reserved;
    double *policy;        /* [n_slots][max_moves][A]  search policies (float64, like the reference) */
    double *value;         /* [n_slots][max_moves]     root search values */
    int32_t *action;       /* [n_slots][max_moves]     moves played */
    uint64_t *start_board; /* [n_slots][2][8]          bitboards (+1 / -1 stones) at the first recorded move */
    int32_t *start_info;   /* [n_slots][4]             player to move, move_count, last_move, game index */
    int32_t *free_slots;   /* [n_slots]                stack of free slot ids */
    int32_t *free_top;     /* [1]                      ids on the stack */
    int32_t *fin_queue;    /* [fin_cap][4]             slot, game, length, winner */
    int32_t *fin_count;    /* [1] */
} gmz_traj;
/* Slot g -> game g, remaining slots on the free stack, queues cleared. */
int gmz_traj_init(gmz_engine *e, const gmz_traj *traj, gmz_stream stream);
/* Play `total_moves` self-play moves (one move = Gumbel noise + a full S-simulation search with
 * E0 + decision + do_move + get_game_ended) spread over the G games by a ticket counter, in ONE
 * persistent kernel.  Noise of game g's k-th search = gmz_fill_gumbel(noise_seed, offset =
 * (k*G + g)*A).  Finished games restart inside the launch if `restart` (and a free slot exists);
 * otherwise they park until gmz_selfplay_unpark.  traj may be NULL (no recording). */
int gmz_selfplay_e0(gmz_engine *e, const gmz_traj *traj, uint64_t eval_seed, int logit_div, uint64_t noise_seed,
                    int64_t total_moves, int restart, gmz_stream stream);
int gmz_selfplay_unpark(gmz_engine *e, const gmz_traj *traj, gmz_stream stream);
/* The same move bookkeeping for the stepwise path (any evaluator): after gmz_finalize, record
 * (policy f64 [G,A], value f64 [G], action int32 [G]) in each game's trajectory slot, do_move,
 * get_game_ended, queue finished games and restart them (workers.py:172-189, 230).  traj may be
 * NULL (no recording); out_winner int32 [G] may be NULL. */
int gmz_selfplay_step(gmz_engine *e, const gmz_traj *traj, const double *policy, const double *value,
                      const int32_t *action, int restart, int32_t *out_winner, gmz_stream stream);
/* out (device, uint64 [4]) = moves played, games finished, tickets that found no playable game,
 * tickets whose game produced no move -- all since gmz_create. */
int gmz_play_counters(gmz_engine *e, uint64_t *out2, gmz_stream stream);
/* out (device, uint64 [3]) = interior selections (_select_action, mcts.py:106-117) that the certified
 * float32 candidate path could not decide and handed to the exact float64 path; and, in builds with
 * -DGMZ_VERIFY_FAST only (every certified decision re-derived by the exact path), the number of
 * certified decisions and how many of them the exact path contradicted (must be 0). */
int gmz_select_counters(gmz_engine *e, uint64_t *out3, gmz_stream stream);

/* ---- MuZero-mode hidden-state pool (Node.hidden_state, mcts.py:21, 40-41; queue hops mcts.py:77-85) ---- */
/* The pool holds one row per tree node, row(g, node) = g*nodes_per_game + node, each row `positions`
 * cells of pos_bytes (NHWC: board cells x channels).  Slots are what gmz_select_mz emits
 * (g*sims_per_game + node, or -1 = nothing to do for that game).
 * gather: x[g] = per cell [ pool row cell | embed if cell == action[g] else zeros ] -- the dynamics
 *   net's input, hidden state and one-hot action embedding concatenated along channels
 *   (network.py:70-73).  embed_bytes may be 0 (then embed/action may be NULL).  slot < 0 writes zeros.
 * scatter: pool[row(slot[g])] = hidden[g] (row_bytes each); slot < 0 is skipped.
 * Byte sizes and pointers must be multiples of 4; 16-byte multiples take the 128-bit copy path. */
int gmz_hidden_gather(const void *pool, const int32_t *slot, const int32_t *action, int num_games, int sims_per_game,
                      int nodes_per_game, int positions, int pos_bytes, const void *embed, int embed_bytes, void *x,
                      gmz_stream stream);
int gmz_hidden_scatter(void *pool, const int32_t *slot, int num_games, int sims_per_game, int nodes_per_game,
                       int row_bytes, const void *hidden, gmz_stream stream);

/* ---- self-play game step --------------------------------------------------- */
/* game.do_move(action) + game.get_game_ended() on the roots (workers.py:178-181,
 * game.py:20-63): actions int32 [G] (<0 = skip that game); out_winner int32 [G]
 * = +-1, 0 (draw) or GMZ_WINNER_NONE. */
int gmz_game_step(gmz_engine *e, const int32_t *actions, int32_t *out_winner, gmz_stream stream);

/* ---- packed move records: the device-side trajectory hand-off (workers.py:172-230, 399-433) ---- */
/* One fixed-stride record per move of a finished game: everything the reference's self-play loop emits for
 * that move.  Layout (stride = gmz_move_record_bytes(board_size), a multiple of 16):
 *   bytes 0..63   gmz_move_record header (below)
 *   then          policy f64 [A]   the search policy (policies.append, workers.py:174)
 *   then          obs    f32 [3A]  game.get_board_state before the move (workers.py:173)
 *   then          board  i8  [A]   np.copy(game.board) before the move (workers.py:177)
 * The same bytes are (a) viewed as GameRecord / TrainingSlice arrays on the host, (b) gathered across ranks
 * as raw bytes, (c) appended to the device replay ring gmz_records_batch samples from. */
typedef struct gmz_move_record {
    int32_t game_seq;     /* index of the game in the gmz_traj_pack call */
    int32_t t;            /* move number within the recorded game, 0-based */
    int32_t length;       /* moves recorded for the game */
    int32_t winner;       /* get_game_ended(): +-1, 0 = draw */
    int32_t action;       /* the move played */
    int32_t to_move;      /* current_player before the move */
    int32_t last_move;    /* last_move before the move, -1 = None */
    int32_t move_count;   /* move_count before the move */
    float reward;         /* final_rewards[t], workers.py:183-187 */
    float value_target;   /* compute_n_step_returns(...)[t], workers.py:144-152, 205 */
    double search_value;  /* root value of the search for this move */
    int32_t game;         /* engine game index that played it */
    int32_t slot;         /* trajectory slot it was recorded in */
    int32_t reserved[2];
} gmz_move_record;
size_t gmz_move_record_bytes(int board_size);
/* Expand n_games finished games into records.  fin int32 [n_games][4] = (slot, game, length, winner) rows of the
 * store's fin_queue; move_offset int64 [n_games] = record index of each game's first move (exclusive prefix sum of
 * min(length, max_moves)); discount_pow f64 [n_steps+1] = discount**i as the host computes them;
 * out_records = total_moves * stride bytes.  All pointers are device pointers. */
int gmz_traj_pack(const gmz_traj *traj, int board_size, const int32_t *fin, int n_games, const int64_t *move_offset,
                  const double *discount_pow, int n_steps, void *out_records, gmz_stream stream);
/* A training batch (workers.py:430-433) gathered from a RING of `capacity` records: sample b is the record at
 * ring position positions[b] (the reference's data index, replay_buffer.py:80) plus the next `unroll` records of
 * the same game, padded past its end like workers.py:208-222; rot_k / flip = the trainer's D4 augmentation
 * (loss.py:37-51): planes and policies turned rot_k (0..3) quarter turns as torch.rot90 does, then flipped
 * left-right if `flip`; actions by the reference's own index formula (loss.py:46-51), padded entries stay -1.
 * Outputs: obs f32 [B,U+1,3,N,N], act i32 [B,U] (padding -1), rew f32 [B,U], pi f64 [B,U+1,A], val f32 [B,U+1]
 * -- the tuple data_loader_worker stacks (workers.py:430-433). */
int gmz_records_batch(const void *ring, int64_t capacity, int board_size, const int64_t *positions, int batch, int unroll,
                      int rot_k, int flip, float *obs, int32_t *act, float *rew, double *pi, float *val, gmz_stream stream);
/* Missed-win flags of n_records consecutive records (a packed block or a stretch of the ring), read in place: the
 * record's board is classified like gmz_tactics_classify for the side in its to_move, out_flags uint8 [n_records] =
 * bit 0: the mover had a winning move, bit 1: the mover had a five, bit 2: the played action was one of them
 * (an action outside [0, A) is not).  A missed win (workers.py:191-203) is bit 0 without bit 2, a missed five
 * additionally has bit 1.  n_records = 0 is a no-op. */
int gmz_records_tactics(const void *records, int64_t n_records, int board_size, int n_in_row, uint8_t *out_flags,
                        gmz_stream stream);
/* Re-analysis of a stretch of the ring in place (workers.py:243-305).  A stretch is (first, n): record k sits at ring
 * position (first + k) % capacity, 0 <= first < capacity, 0 <= n <= capacity; n = 0 is a no-op.
 * gmz_set_roots_from_records: the engine's roots straight from records, n <= G.  Game k < n takes record k's board
 *   (before the move), and its header's to_move (not move parity), last_move and move_count -- what gmz_set_roots does
 *   with those fields; games n..G-1 become inactive (full-board padding, as reanalyse_positions pads).
 * gmz_records_writeback: policy f64 [n,A] row k and value f64 [n] entry k (gmz_finalize's outputs) replace record k's
 *   policy and header search_value; nothing else is written.
 * gmz_records_retarget: record k's value_target from its own header (t, length, winner) and the search_value of the
 *   record n_steps later in the same game, with re-analysis arithmetic (float32 rewards, workers.py:291-292): reward
 *   terms (float)discount_pow[i] * r in float32, summed in float32 for i = 0..n_steps-1, plus the float32 bootstrap
 *   (float)search_value * (float)discount_pow[n_steps].  The stretch must hold whole live games (their later moves are
 *   read).  discount_pow f64 [n_steps+1] = discount**i as the host computes them. */
int gmz_set_roots_from_records(gmz_engine *e, const void *ring, int64_t capacity, int64_t first, int64_t n, gmz_stream stream);
int gmz_records_writeback(void *ring, int64_t capacity, int board_size, int64_t first, int64_t n, const double *policy,
                          const double *value, gmz_stream stream);
int gmz_records_retarget(void *ring, int64_t capacity, int board_size, int64_t first, int64_t n, const double *discount_pow,
                         int n_steps, gmz_stream stream);
/* Checkpoint form of the ring: only a record's header and policy carry information -- its board follows from the previous
 * record's board and action, its observation planes from the board and the header.  A SEGMENT is a run of consecutive
 * records that starts at k = 0 or at a header t = 0 (games sit whole and in move order in the ring).
 * gmz_records_compact: the stretch (first, n) -> out_headers u8 [n][64] and out_policy f64 [n][A], verbatim, and
 *   out_flags u8 [n]: bit 0 = record k starts a segment; bit 1 = record k is NOT rebuildable by gmz_records_expand: its
 *   board holds a value outside {-1, 0, 1}, its planes are not (board == own, board == -own, cell == last_move) as
 *   0.0f / 1.0f with own = to_move > 0 ? +1 : -1, or (not a segment start) its board is not record k-1's board with record
 *   k-1's action played for record k-1's to_move (an action outside [0, A) changes nothing).
 * gmz_records_expand: n compact records (headers, policy as above), seg_start int64 [n_seg] (the k of each segment's
 *   first record, 1 <= n_seg <= n when n > 0) and base_boards int8 [n_seg][A] (those records' boards) -> record k, for
 *   every k >= skip (0 <= skip <= n, n - skip <= capacity), as a full record at ring position (first + k - skip) % capacity:
 *   header and policy verbatim, board replayed from the segment's base board with every earlier record's action played
 *   for that record's to_move, planes derived from it, tail padding zero.  Segments are clamped to [0, n).
 * n = 0 is a no-op for both.  All pointers are device pointers. */
int gmz_records_compact(const void *ring, int64_t capacity, int board_size, int64_t first, int64_t n, void *out_headers,
                        double *out_policy, uint8_t *out_flags, gmz_stream stream);
int gmz_records_expand(const void *headers, const double *policy, int64_t n, const int64_t *seg_start, const int8_t *base_boards,
                       int64_t n_seg, int64_t skip, int board_size, void *ring, int64_t capacity, int64_t first, gmz_stream stream);

/* ---- tactics classifier (find_winning_moves_rebuilt, workers.py:49-123) ---- */
/* boards int8 [B,A], players int8 [B] (the side to move) -> out_cls int8 [B,A]: per empty cell
 * 1 = 'five', 2 = 'open_four', 3 = 'combo', 0 = none (occupied cells: 0).  Feeds the missed-win
 * statistics of the self-play and re-analysis loops (workers.py:191-203, 270-289). */
int gmz_tactics_classify(const int8_t *boards, const int8_t *players, int batch, int board_size, int n_in_row,
                         int8_t *out_cls, gmz_stream stream);

/* ---- prioritized replay: SumTree (replay_buffer.py:4-106) ------------------- */
/* tree f64 [2*capacity-1] lives in caller memory.  Sequential reference
 * semantics are preserved bit for bit (each node receives its += in batch order). */
/* update_priorities / add: tree_idx int64 [n], priorities f64 [n], applied in order. */
int gmz_per_update(double *tree, int64_t capacity, const int64_t *tree_idx, const double *priorities, int n,
                   gmz_stream stream);
/* add(): n priorities written at ring positions write_ptr, write_ptr+1, ... (mod capacity), applied in
 * order (replay_buffer.py:21-25); scratch_idx int64 [n] is caller-owned scratch.  The caller advances
 * write_ptr / count like SumTree.add does. */
int gmz_per_add(double *tree, int64_t capacity, int64_t write_ptr, const double *priorities, int n,
                int64_t *scratch_idx, gmz_stream stream);
/* sample(): u01 f64 [B] uniform draws; outputs tree_idx int64 [B], priority f64 [B],
 * is_weights f32 [B] (already divided by the batch max). */
int gmz_per_sample(const double *tree, int64_t capacity, int64_t count, const double *u01, int batch, double beta,
                   int64_t *out_tree_idx, double *out_priority, float *out_weights, gmz_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* GMZ_H */
