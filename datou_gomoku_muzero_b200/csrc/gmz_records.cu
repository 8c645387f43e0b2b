// gmz_records.cu -- device-side trajectory hand-off (reference workers.py:172-230, 399-433).
//
// A finished game leaves the trajectory store as PACKED MOVE RECORDS: one fixed-stride record per move holding
// everything the reference's self-play loop emits for that move -- the observation planes (game.py:12-17), the
// search policy (float64, as the reference keeps it), the board before the move, and the scalars (action, root
// search value, final reward workers.py:183-187, n-step value target workers.py:144-152).  The same bytes serve
//   * the host: GameRecord / TrainingSlice objects are numpy views of the copied block (no per-move arithmetic),
//   * the wire: ranks gather them with one collective of raw bytes (replaces data_queue, workers.py:230, 399),
//   * the replay ring on the device: a TrainingSlice is U+1 consecutive records of one game, so a training batch
//     (workers.py:430-433) is gathered straight from the ring, D4 augmentation (loss.py:37-51) included.
// Record layout (gmz_move_record_bytes): 64-byte header | policy f64[A] | obs f32[3A] | board i8[A] | pad to 16.
#include <stdint.h>
#include <stdio.h>

#include "../../include/gmz.h"
#include "gmz_common.cuh"
#include "gmz_records.cuh"
#include "gmz_tactics.cuh"

extern "C" void gmz_set_error_(const char *msg);
static int rc_fail(const char *m) { gmz_set_error_(m); return 1; }

extern "C" size_t gmz_move_record_bytes(int board_size)
{
    if (board_size < 1 || board_size > GMZ_MAX_BOARD) return 0;
    return rec_stride(board_size * board_size);
}

// Missed-win flags of packed move records (workers.py:191-203): one CTA per record, one thread per cell.  The record's
// board (before the move, absolute colours) is classified for the side in the header's to_move -- not move parity,
// so a game started from a mid-game position gets the right colour -- and reduced to one byte:
//   bit 0: the mover had a winning move (some cell class > 0), bit 1: the mover had a five (some cell class == 1),
//   bit 2: the played cell (header action; outside [0, A) counts as class 0) has class > 0.
__global__ void __launch_bounds__(512)
k_records_tactics(const unsigned char *records, size_t stride, int N, int n_in_row, uint8_t *out_flags)
{
    __shared__ int8_t sb[GMZ_MAX_BOARD * GMZ_MAX_BOARD];
    const int A = N * N;
    const unsigned char *rec = records + (size_t)blockIdx.x * stride;
    const int8_t *brd = reinterpret_cast<const int8_t *>(rec + 64 + (size_t)20 * A);
    for (int i = threadIdx.x; i < A; i += blockDim.x) sb[i] = brd[i];
    const RecHeader *h = reinterpret_cast<const RecHeader *>(rec);
    const int P = h->to_move >= 0 ? 1 : -1, action = h->action;
    __syncthreads();
    int any = 0, five = 0, played = 0;
    for (int cell = threadIdx.x; cell < A; cell += blockDim.x) {
        const int cls = gmz_tactics_cell_class(sb, N, n_in_row, P, cell);
        any |= cls > 0;
        five |= cls == 1;
        played |= cell == action && cls > 0;
    }
    any = __syncthreads_or(any);
    five = __syncthreads_or(five);
    played = __syncthreads_or(played);
    if (threadIdx.x == 0) out_flags[blockIdx.x] = (uint8_t)((any ? 1 : 0) | (five ? 2 : 0) | (played ? 4 : 0));
}

extern "C" int gmz_records_tactics(const void *records, int64_t n_records, int board_size, int n_in_row, uint8_t *out_flags,
                                   gmz_stream stream)
{
    if (!records || !out_flags) return rc_fail("gmz_records_tactics: null argument");
    if (board_size < 1 || board_size > GMZ_MAX_BOARD) return rc_fail("gmz_records_tactics: board_size out of range");
    if (n_in_row < 1) return rc_fail("gmz_records_tactics: n_in_row must be >= 1");
    if (n_records < 0 || n_records > 0x7fffffff) return rc_fail("gmz_records_tactics: n_records out of range");
    if (n_records == 0) return 0;
    const int A = board_size * board_size;
    int threads = ((A + 31) / 32) * 32;          // the block-size rule of gmz_tactics_classify
    if (threads > 512) threads = 512;
    k_records_tactics<<<(unsigned)n_records, threads, 0, (cudaStream_t)stream>>>((const unsigned char *)records, rec_stride(A),
                                                                               board_size, n_in_row, out_flags);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : rc_fail(cudaGetErrorString(e));
}

__device__ __forceinline__ float rec_final_reward(int i, int T, int winner)   // workers.py:183-187
{
    if (winner == 0 || i < 0 || i >= T) return 0.0f;
    const int j = (T - 1 - i) & 3;
    return (j == 0 || j == 3) ? 1.0f : -1.0f;
}
__device__ __forceinline__ void rec_apply(u64 &P, u64 &M, int colour, int a, int lane)
{
    if (lane == (a >> 6)) { const u64 bit = 1ull << (a & 63); if (colour > 0) { P |= bit; M &= ~bit; } else { M |= bit; P &= ~bit; } }
}

// A record's observation planes (game.py:12-17) and board (before the move) from the position's bitboards: P / M hold
// the stones of +1 / -1, 64 cells per lane; the own plane is P if colour (the side to move) > 0, else M; the third plane
// marks `last` (-1 or any value outside [0, A): no cell).  Called by the whole warp: every lane takes part in the shuffles.
__device__ __forceinline__ void rec_write_position(unsigned char *rec, int A, u64 P, u64 M, int colour, int last, int lane)
{
    float *obs = reinterpret_cast<float *>(rec + 64 + (size_t)8 * A);
    int8_t *brd = reinterpret_cast<int8_t *>(rec + 64 + (size_t)20 * A);
    const u64 own = colour > 0 ? P : M, opp = colour > 0 ? M : P;
    for (int c0 = 0; c0 < A; c0 += 32) {
        const int c = c0 + lane, cw = min(c, A - 1) >> 6;
        const u64 ow = __shfl_sync(GMZ_FULL, own, cw), pw = __shfl_sync(GMZ_FULL, opp, cw);
        const u64 bp = __shfl_sync(GMZ_FULL, P, cw), bm = __shfl_sync(GMZ_FULL, M, cw);
        if (c < A) {
            obs[c] = (float)((ow >> (c & 63)) & 1ull);
            obs[A + c] = (float)((pw >> (c & 63)) & 1ull);
            obs[2 * A + c] = c == last ? 1.0f : 0.0f;
            brd[c] = (int8_t)((int)((bp >> (c & 63)) & 1ull) - (int)((bm >> (c & 63)) & 1ull));
        }
    }
}

// One CTA per finished game, warp w emits moves w, w + 4, ... (each warp replays the game on its own bitboards).
__global__ void __launch_bounds__(128)
k_traj_pack(int N, int A, size_t stride, int max_moves, const double *policy, const double *value, const int32_t *action,
            const u64 *start_board, const int32_t *start_info, const int32_t *fin, int n_games, const int64_t *move_offset,
            const double *dpow, int n_steps, unsigned char *out)
{
    const int gi = blockIdx.x, lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
    if (gi >= n_games) return;
    const int slot = fin[4 * gi + 0], game = fin[4 * gi + 1], T = min(fin[4 * gi + 2], max_moves), winner = fin[4 * gi + 3];
    u64 P = lane < GMZ_WORDS ? start_board[((size_t)slot * 2 + 0) * GMZ_WORDS + lane] : 0ull;
    u64 M = lane < GMZ_WORDS ? start_board[((size_t)slot * 2 + 1) * GMZ_WORDS + lane] : 0ull;
    int colour = start_info[(size_t)slot * 4 + 0], mc = start_info[(size_t)slot * 4 + 1], last = start_info[(size_t)slot * 4 + 2];
    const int32_t *acts = action + (size_t)slot * max_moves;
    const double *vals = value + (size_t)slot * max_moves;
    const float gn = (float)dpow[n_steps];
    int m = 0;
    for (int t = wi; t < T; t += 4) {
        for (; m < t; ++m) { const int a = acts[m]; rec_apply(P, M, colour, a, lane); colour = -colour; last = a; ++mc; }
        unsigned char *rec = out + (size_t)(move_offset[gi] + t) * stride;
        double *pol = reinterpret_cast<double *>(rec + 64);
        const double *psrc = policy + ((size_t)slot * max_moves + t) * A;
        rec_write_position(rec, A, P, M, colour, last, lane);
        for (int c = lane; c < A; c += 32) pol[c] = psrc[c];
        if (lane == 0) {
            // compute_n_step_returns (workers.py:144-152): Python-float reward sum, float32 bootstrap, float32 add
            double acc = 0.0;
            for (int i = 0; i < n_steps; ++i)
                if (t + i < T) acc = __dadd_rn(acc, __dmul_rn(dpow[i], (double)rec_final_reward(t + i, T, winner)));
            const int b = t + n_steps;
            RecHeader h;
            h.game_seq = gi; h.t = t; h.length = T; h.winner = winner;
            h.action = acts[t]; h.to_move = colour; h.last_move = last; h.move_count = mc;
            h.reward = rec_final_reward(t, T, winner);
            h.value_target = b < T ? __fadd_rn((float)acc, __fmul_rn((float)vals[b], gn)) : (float)acc;
            h.search_value = vals[t];
            h.game = game; h.slot = slot; h.pad0 = 0; h.pad1 = 0;
            *reinterpret_cast<RecHeader *>(rec) = h;
        }
    }
}

extern "C" int gmz_traj_pack(const gmz_traj *traj, int board_size, const int32_t *fin, int n_games, const int64_t *move_offset,
                             const double *discount_pow, int n_steps, void *out_records, gmz_stream stream)
{
    if (!traj || !fin || !move_offset || !discount_pow || !out_records) return rc_fail("gmz_traj_pack: null argument");
    if (n_games <= 0) return 0;
    if (board_size < 1 || board_size > GMZ_MAX_BOARD || n_steps < 0) return rc_fail("gmz_traj_pack: bad size");
    const int A = board_size * board_size;
    k_traj_pack<<<n_games, 128, 0, (cudaStream_t)stream>>>(board_size, A, rec_stride(A), traj->max_moves, traj->policy, traj->value,
                                                           traj->action, (const u64 *)traj->start_board, traj->start_info, fin, n_games,
                                                           move_offset, discount_pow, n_steps, (unsigned char *)out_records);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : rc_fail(cudaGetErrorString(e));
}

// ---------------------------------------------------------------------------------------------------------
// Training batches from a ring of records (DeviceReplayBuffer): sample b is the record at ring position pos[b]
// (= the reference's data index, replay_buffer.py:50-55, 80); its slice is that record and the next U of the same
// game (they sit at the following ring positions: records are appended game by game in move order, and a ring
// overwrites oldest first, so the successors of a live record are live), padded past the game's end like
// workers.py:208-222 (zero planes / policies / values / rewards, action -1).
__device__ __forceinline__ int rec_sym_cell(int c, int N, int rk, int fl)      // loss.py:39-44, as torch.rot90 / flip
{
    const int r = c / N, q = c - r * N;
    int i = r, j = q;
    if (rk == 1) { i = N - 1 - q; j = r; }
    else if (rk == 2) { i = N - 1 - r; j = N - 1 - q; }
    else if (rk == 3) { i = q; j = N - 1 - r; }
    if (fl) j = N - 1 - j;
    return i * N + j;
}
__device__ __forceinline__ int rec_sym_action(int a, int N, int rk, int fl)     // loss.py:46-51, as written
{
    if (a < 0) return a;
    int rows = a / N, cols = a - rows * N;
    if (rk == 1) { const int t = rows; rows = cols; cols = N - 1 - t; }
    else if (rk == 2) { rows = N - 1 - rows; cols = N - 1 - cols; }
    else if (rk == 3) { const int t = rows; rows = N - 1 - cols; cols = t; }
    if (fl) cols = N - 1 - cols;
    return rows * N + cols;
}

__global__ void __launch_bounds__(128)
k_records_batch(int N, int A, size_t stride, int64_t capacity, const unsigned char *ring, const int64_t *pos, int B, int U,
                int rk, int fl, float *obs, int32_t *act, float *rew, double *pi, float *val)
{
    const int lane = threadIdx.x & 31, b = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (b >= B) return;
    const int64_t p0 = pos[b];
    const RecHeader h0 = *reinterpret_cast<const RecHeader *>(ring + (size_t)p0 * stride);
    for (int k = 0; k <= U; ++k) {
        float *o = obs + ((size_t)b * (U + 1) + k) * 3 * A;
        double *pk = pi + ((size_t)b * (U + 1) + k) * A;
        if (h0.t + k < h0.length) {
            const unsigned char *rec = ring + (size_t)((p0 + k) % capacity) * stride;
            const RecHeader *h = reinterpret_cast<const RecHeader *>(rec);
            const double *pol = reinterpret_cast<const double *>(rec + 64);
            const float *ob = reinterpret_cast<const float *>(rec + 64 + (size_t)8 * A);
            for (int c = lane; c < A; c += 32) {
                const int d = rec_sym_cell(c, N, rk, fl);
                o[d] = ob[c]; o[A + d] = ob[A + c]; o[2 * A + d] = ob[2 * A + c];
                pk[d] = pol[c];
            }
            if (lane == 0) {
                val[(size_t)b * (U + 1) + k] = h->value_target;
                if (k < U) { act[(size_t)b * U + k] = rec_sym_action(h->action, N, rk, fl); rew[(size_t)b * U + k] = h->reward; }
            }
        } else {
            for (int c = lane; c < A; c += 32) { o[c] = 0.f; o[A + c] = 0.f; o[2 * A + c] = 0.f; pk[c] = 0.0; }
            if (lane == 0) {
                val[(size_t)b * (U + 1) + k] = 0.0f;
                if (k < U) { act[(size_t)b * U + k] = -1; rew[(size_t)b * U + k] = 0.0f; }
            }
        }
    }
}

extern "C" int gmz_records_batch(const void *ring, int64_t capacity, int board_size, const int64_t *positions, int batch, int unroll,
                                 int rot_k, int flip, float *obs, int32_t *act, float *rew, double *pi, float *val, gmz_stream stream)
{
    if (!ring || !positions || !obs || !act || !rew || !pi || !val) return rc_fail("gmz_records_batch: null argument");
    if (batch <= 0) return 0;
    if (board_size < 1 || board_size > GMZ_MAX_BOARD || unroll < 0 || capacity < 1) return rc_fail("gmz_records_batch: bad size");
    if (rot_k < 0 || rot_k > 3) return rc_fail("gmz_records_batch: rot_k must be 0..3");
    const int A = board_size * board_size;
    k_records_batch<<<(batch + 3) / 4, 128, 0, (cudaStream_t)stream>>>(board_size, A, rec_stride(A), capacity, (const unsigned char *)ring,
                                                                       positions, batch, unroll, rot_k, flip ? 1 : 0, obs, act, rew, pi, val);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : rc_fail(cudaGetErrorString(e));
}

// ---------------------------------------------------------------------------------------------------------
// Re-analysis of a stretch of the ring in place (workers.py:243-305): record k of the stretch sits at ring position
// (first + k) % capacity.  gmz_set_roots_from_records (gmz_engine.cu) loads the roots, the search runs, then the two
// kernels below put the results back.
static int rc_fail2(const char *name, const char *m)
{
    char buf[256];
    snprintf(buf, sizeof(buf), "%s: %s", name, m);
    gmz_set_error_(buf);
    return 1;
}

// The re-searched policy row k and root value k replace the record's policy bytes and header search_value; nothing
// else in the record is written.  One warp per record.
__global__ void __launch_bounds__(128)
k_records_writeback(unsigned char *ring, size_t stride, int64_t capacity, int64_t first, int64_t n, int A, const double *policy,
                    const double *value)
{
    const int lane = threadIdx.x & 31;
    const int64_t k = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (k >= n) return;
    unsigned char *rec = ring + (size_t)((first + k) % capacity) * stride;
    double *pol = reinterpret_cast<double *>(rec + 64);
    const double *src = policy + (size_t)k * A;
    for (int c = lane; c < A; c += 32) pol[c] = src[c];
    if (lane == 0) reinterpret_cast<RecHeader *>(rec)->search_value = value[k];
}

extern "C" int gmz_records_writeback(void *ring, int64_t capacity, int board_size, int64_t first, int64_t n, const double *policy,
                                     const double *value, gmz_stream stream)
{
    const char *name = "gmz_records_writeback";
    if (!ring || !policy || !value) return rc_fail2(name, "null argument");
    if (board_size < 1 || board_size > GMZ_MAX_BOARD) return rc_fail2(name, "board_size out of range (1..19)");
    if (const char *m = rec_stretch_check(capacity, first, n)) return rc_fail2(name, m);
    if (n == 0) return 0;
    const int A = board_size * board_size;
    k_records_writeback<<<(unsigned)((n + 3) / 4), 128, 0, (cudaStream_t)stream>>>((unsigned char *)ring, rec_stride(A), capacity,
                                                                                   first, n, A, policy, value);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : rc_fail2(name, cudaGetErrorString(e));
}

// New n-step value targets from the re-searched root values, with re-analysis arithmetic (reanalysis.reanalyse ->
// compute_n_step_returns on float32 rewards, workers.py:291-292): each reward term a float32 product, summed in float32
// in order, the bootstrap a float32 product, one float32 add.  (Self-play's k_traj_pack sums the rewards in float64.)
// A record reads its own header and the search_value of the record n_steps later in the same game, which is live and
// already rewritten: games sit whole and in move order in the ring, and the stretch covers whole games.
__global__ void __launch_bounds__(256)
k_records_retarget(unsigned char *ring, size_t stride, int64_t capacity, int64_t first, int64_t n, const double *dpow, int n_steps)
{
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int64_t p = (first + k) % capacity;
    RecHeader *h = reinterpret_cast<RecHeader *>(ring + (size_t)p * stride);
    const int t = h->t, T = h->length, winner = h->winner;
    float acc = 0.0f;
    for (int i = 0; i < n_steps && t + i < T; ++i) acc = __fadd_rn(acc, __fmul_rn((float)dpow[i], rec_final_reward(t + i, T, winner)));
    float boot = 0.0f;
    if ((int64_t)t + n_steps < T) {
        const RecHeader *hb = reinterpret_cast<const RecHeader *>(ring + (size_t)((p + n_steps) % capacity) * stride);
        boot = __fmul_rn((float)hb->search_value, (float)dpow[n_steps]);
    }
    h->value_target = __fadd_rn(acc, boot);
}

extern "C" int gmz_records_retarget(void *ring, int64_t capacity, int board_size, int64_t first, int64_t n, const double *discount_pow,
                                    int n_steps, gmz_stream stream)
{
    const char *name = "gmz_records_retarget";
    if (!ring || !discount_pow) return rc_fail2(name, "null argument");
    if (board_size < 1 || board_size > GMZ_MAX_BOARD) return rc_fail2(name, "board_size out of range (1..19)");
    if (const char *m = rec_stretch_check(capacity, first, n)) return rc_fail2(name, m);
    if (n_steps < 0) return rc_fail2(name, "n_steps must be >= 0");
    if (n == 0) return 0;
    const int A = board_size * board_size;
    k_records_retarget<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((unsigned char *)ring, rec_stride(A), capacity,
                                                                                     first, n, discount_pow, n_steps);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : rc_fail2(name, cudaGetErrorString(e));
}

// ---------------------------------------------------------------------------------------------------------
// Checkpoint form of the ring (DeviceReplayBuffer.state_dict / load_state_dict).  Of a record only the header and the
// policy carry information: the board follows from the previous record's board and action, the observation planes from
// the board and the header.  A stretch is saved as headers u8 [n][64] + policies f64 [n][A], plus the board of the first
// record of every segment (a run of records that starts at k = 0 or at a header t = 0: games sit whole and in move order
// in the ring, only the oldest live game can be cut).

// Saving: record k of the stretch (one warp per record) -> its header and policy bytes verbatim, and a flag byte:
//   bit 0: the record starts a segment (k == 0 or t == 0),
//   bit 1: the record is NOT rebuildable -- its board or observation planes differ from what k_records_expand writes:
//          the board holds a value outside {-1, 0, 1}; the planes are not (board == own, board == -own, cell == last_move)
//          as 0.0f / 1.0f bit patterns, own = to_move > 0 ? +1 : -1; or (no segment start) the board is not record k-1's
//          board with record k-1's action played for record k-1's to_move (rec_apply: overwrite the cell, an action
//          outside [0, A) changes nothing).
// Each record is compared with its predecessor only, so the check needs no sequential replay.
__global__ void __launch_bounds__(128)
k_records_compact(const unsigned char *ring, size_t stride, int64_t capacity, int64_t first, int64_t n, int A,
                  unsigned char *out_headers, double *out_policy, uint8_t *out_flags)
{
    const int lane = threadIdx.x & 31;
    const int64_t k = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (k >= n) return;
    const unsigned char *rec = ring + (size_t)((first + k) % capacity) * stride;
    const RecHeader *h = reinterpret_cast<const RecHeader *>(rec);
    if (lane < 16) reinterpret_cast<uint32_t *>(out_headers + (size_t)k * 64)[lane] = reinterpret_cast<const uint32_t *>(rec)[lane];
    const double *pol = reinterpret_cast<const double *>(rec + 64);
    double *dst = out_policy + (size_t)k * A;
    for (int c = lane; c < A; c += 32) dst[c] = pol[c];

    const bool start = k == 0 || h->t == 0;
    const int own = h->to_move > 0 ? 1 : -1, last = h->last_move;
    const uint32_t *obs = reinterpret_cast<const uint32_t *>(rec + 64 + (size_t)8 * A);
    const int8_t *brd = reinterpret_cast<const int8_t *>(rec + 64 + (size_t)20 * A);
    const int8_t *pbrd = nullptr;
    int pa = -1, pown = 0;
    if (!start) {
        const unsigned char *prv = ring + (size_t)((first + k - 1) % capacity) * stride;
        const RecHeader *hp = reinterpret_cast<const RecHeader *>(prv);
        pa = hp->action;
        pown = hp->to_move > 0 ? 1 : -1;
        pbrd = reinterpret_cast<const int8_t *>(prv + 64 + (size_t)20 * A);
    }
    const uint32_t one = 0x3f800000u;                   // 1.0f
    bool bad = false;
    for (int c = lane; c < A; c += 32) {
        const int b = brd[c];
        bad |= b < -1 || b > 1;
        bad |= obs[c] != (b == own ? one : 0u);
        bad |= obs[A + c] != (b == -own ? one : 0u);
        bad |= obs[2 * A + c] != (c == last ? one : 0u);
        if (pbrd) bad |= b != (c == pa ? pown : (int)pbrd[c]);
    }
    bad = __any_sync(GMZ_FULL, bad);
    if (lane == 0) out_flags[k] = (uint8_t)((start ? 1 : 0) | (bad ? 2 : 0));
}

extern "C" int gmz_records_compact(const void *ring, int64_t capacity, int board_size, int64_t first, int64_t n, void *out_headers,
                                   double *out_policy, uint8_t *out_flags, gmz_stream stream)
{
    const char *name = "gmz_records_compact";
    if (!ring || !out_headers || !out_policy || !out_flags) return rc_fail2(name, "null argument");
    if (board_size < 1 || board_size > GMZ_MAX_BOARD) return rc_fail2(name, "board_size out of range (1..19)");
    if (const char *m = rec_stretch_check(capacity, first, n)) return rc_fail2(name, m);
    if (n == 0) return 0;
    const int A = board_size * board_size;
    k_records_compact<<<(unsigned)((n + 3) / 4), 128, 0, (cudaStream_t)stream>>>((const unsigned char *)ring, rec_stride(A), capacity,
                                                                                 first, n, A, (unsigned char *)out_headers, out_policy,
                                                                                 out_flags);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : rc_fail2(name, cudaGetErrorString(e));
}

// Loading: one CTA per segment, segment s = records [seg_start[s], seg_start[s+1]) (the last one up to n), clamped to
// [0, n).  Warp w replays the segment from its base board on its own bitboards, every record's action played for that
// record's own header to_move (the exact inverse of the check above), and emits records w, w + 4, ...: record k >= skip
// becomes a full record at ring position (first + k - skip) % capacity -- header and policy verbatim, board and
// observation planes rebuilt (rec_write_position, as k_traj_pack writes them), tail padding zero.  Records below skip
// are replayed but not written.  No memory is indexed by a header field, so any table contents stay in bounds.
__global__ void __launch_bounds__(128)
k_records_expand(const unsigned char *headers, const double *policy, int64_t n, const int64_t *seg_start, const int8_t *base_boards,
                 int64_t n_seg, int64_t skip, int A, size_t stride, unsigned char *ring, int64_t capacity, int64_t first)
{
    const int64_t s = blockIdx.x;
    const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
    const int64_t lo = min(max(seg_start[s], (int64_t)0), n);
    const int64_t hi = s + 1 < n_seg ? min(max(seg_start[s + 1], lo), n) : n;
    if (lo >= hi) return;
    const int8_t *bb = base_boards + (size_t)s * A;
    u64 P = 0, M = 0;
    for (int w = 0; w < (A + 63) / 64; ++w) {          // ballots pack 32 cells at a time (root_load, gmz_engine.cu)
        u64 pw = 0, mw = 0;
        for (int h = 0; h < 2; ++h) {
            const int a = 64 * w + 32 * h + lane;
            const int c = a < A ? (int)bb[a] : 0;
            pw |= (u64)__ballot_sync(GMZ_FULL, c == 1) << (32 * h);
            mw |= (u64)__ballot_sync(GMZ_FULL, c == -1) << (32 * h);
        }
        if (lane == w) { P = pw; M = mw; }
    }
    const size_t body = (size_t)64 + (size_t)21 * A;
    int64_t m = lo;
    for (int64_t k = lo + wi; k < hi; k += 4) {
        for (; m < k; ++m) {
            const RecHeader *hm = reinterpret_cast<const RecHeader *>(headers + (size_t)m * 64);
            rec_apply(P, M, hm->to_move, hm->action, lane);
        }
        if (k < skip) continue;
        const unsigned char *src = headers + (size_t)k * 64;
        const RecHeader *hk = reinterpret_cast<const RecHeader *>(src);
        unsigned char *rec = ring + (size_t)((first + k - skip) % capacity) * stride;
        if (lane < 16) reinterpret_cast<uint32_t *>(rec)[lane] = reinterpret_cast<const uint32_t *>(src)[lane];
        double *pol = reinterpret_cast<double *>(rec + 64);
        const double *psrc = policy + (size_t)k * A;
        for (int c = lane; c < A; c += 32) pol[c] = psrc[c];
        rec_write_position(rec, A, P, M, hk->to_move, hk->last_move, lane);
        for (size_t i = body + lane; i < stride; i += 32) rec[i] = 0;
    }
}

extern "C" int gmz_records_expand(const void *headers, const double *policy, int64_t n, const int64_t *seg_start,
                                  const int8_t *base_boards, int64_t n_seg, int64_t skip, int board_size, void *ring, int64_t capacity,
                                  int64_t first, gmz_stream stream)
{
    const char *name = "gmz_records_expand";
    if (!headers || !policy || !seg_start || !base_boards || !ring) return rc_fail2(name, "null argument");
    if (board_size < 1 || board_size > GMZ_MAX_BOARD) return rc_fail2(name, "board_size out of range (1..19)");
    if (capacity < 1) return rc_fail2(name, "capacity must be >= 1");
    if (n < 0) return rc_fail2(name, "n must be >= 0");
    if (skip < 0 || skip > n) return rc_fail2(name, "skip must be in 0..n");
    if (n - skip > capacity) return rc_fail2(name, "n - skip exceeds the ring capacity");
    if (first < 0 || first >= capacity) return rc_fail2(name, "first outside the ring [0, capacity)");
    if (n > 0 && (n_seg < 1 || n_seg > n || n_seg > 0x7fffffff)) return rc_fail2(name, "n_seg must be in 1..n when n > 0");
    if (n == 0) return 0;
    const int A = board_size * board_size;
    k_records_expand<<<(unsigned)n_seg, 128, 0, (cudaStream_t)stream>>>((const unsigned char *)headers, policy, n, seg_start, base_boards,
                                                                        n_seg, skip, A, rec_stride(A), (unsigned char *)ring, capacity,
                                                                        first);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : rc_fail2(name, cudaGetErrorString(e));
}
