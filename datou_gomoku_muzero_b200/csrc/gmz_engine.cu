// gmz_engine.cu -- kernels and C ABI (include/gmz.h) of the batched Gumbel-MCTS engine.
// sm_100a only; build: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -lineinfo ...
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <unordered_set>

#include "gmz_internal.h"
#include "gmz_engine.cuh"
#include "gmz_records.cuh"
#include "gmz_tree.cuh"
#include "gmz_play.cuh"

// one warp (= one game) per CTA, as in the play kernel (gmz_play.cuh): warp-uniform state is then CTA-uniform and the
// compiler keeps it on the uniform datapath (k_select: 96 -> 80 registers; stepwise search 19.8 -> 18.9 ms)
#ifndef WARPS_PER_CTA
#define WARPS_PER_CTA 1
#endif
#define CTA_THREADS (32 * WARPS_PER_CTA)

static thread_local char g_err[512] = "";
int gmz_fail(const char *fmt, const char *a)
{
    snprintf(g_err, sizeof(g_err), fmt, a);
    return 1;
}
int gmz_check_launch(const char *what)
{
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e)); return 1; }
    return 0;
}
#define fail gmz_fail
#define check_launch gmz_check_launch

// Live engine handles.  Threading contract (as the reference's engines, SURVEY 8b: "one engine per process,
// single-threaded, not re-entrant"): calls on DIFFERENT engines may run concurrently from different host
// threads; calls on ONE engine must be serialised by the caller.  gmz_destroy on a handle that is not (or no
// longer) live is a no-op returning 0; every other entry point rejects such a handle.
static std::mutex g_live_mu;
static std::unordered_set<const gmz_engine *> g_live;
static bool engine_live(const gmz_engine *e)
{
    if (!e) return false;
    std::lock_guard<std::mutex> lk(g_live_mu);
    return g_live.count(e) != 0;
}

int gmz_engine_live(const gmz_engine *e) { return engine_live(e) ? 1 : 0; }

// ---------------------------------------------------------------------------------------------
// root positions (root_load: gmz_engine.cuh)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS)
k_set_roots(Params p, const int8_t *boards, const int8_t *players, const int32_t *last_moves, const int32_t *move_counts)
{
    const int lane = threadIdx.x & 31, g = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= p.G) return;
    root_load(p, g, lane, boards + (size_t)g * p.A, players[g], last_moves[g], move_counts[g]);
}

// Roots from packed move records (re-analysis, workers.py:254-263): game g < n takes the record at ring position
// (first + g) % capacity -- its board (before the move, absolute colours), and from the header the side to move (not
// move parity: games started mid-game keep their colour), last move and move count.  Games n..G-1 get the full-board
// padding root, inactive.
__global__ void __launch_bounds__(CTA_THREADS)
k_set_roots_records(Params p, const unsigned char *ring, size_t stride, int64_t capacity, int64_t first, int n)
{
    const int lane = threadIdx.x & 31, g = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= p.G) return;
    if (g >= n) { root_load(p, g, lane, nullptr, 1, -1, 0); return; }
    const unsigned char *rec = rec_at(ring, stride, capacity, first, g);
    const gmz_move_record *h = rec_header(rec);
    root_load(p, g, lane, rec_board(rec, p.A), h->to_move, h->last_move, h->move_count);
}

__global__ void __launch_bounds__(CTA_THREADS)
k_games_reset(const __grid_constant__ Params p, const __grid_constant__ BookDev book, const uint8_t *mask)
{
    const int lane = threadIdx.x & 31, g = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= p.G) return;
    if (mask && !mask[g]) return;
    game_deal(p, book, p.gs + g, g, lane);
}

__global__ void __launch_bounds__(CTA_THREADS)
k_get_roots(Params p, int8_t *boards, int8_t *players, int32_t *last_moves, int32_t *move_counts)
{
    const int lane = threadIdx.x & 31, g = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= p.G) return;
    const GState *s = p.gs + g;
    if (boards) {
        for (int a = lane; a < p.A; a += 32) {
            const u64 b = 1ull << (a & 63);
            boards[(size_t)g * p.A + a] = (s->p1[a >> 6] & b) ? 1 : ((s->m1[a >> 6] & b) ? -1 : 0);
        }
    }
    if (lane == 0) {
        if (players) players[g] = (int8_t)s->to_move;
        if (last_moves) last_moves[g] = s->last_move;
        if (move_counts) move_counts[g] = s->move_count;
    }
}

// T = float: NCHW float32 planes; T = unsigned short: NHWC bf16 (channels_last), see obs_write_nhwc_bf16
template <int NC, typename T>
__device__ __forceinline__ void obs_emit(T *obs, int A, u64 own, u64 opp, int last, int lane)
{
    if constexpr (sizeof(T) == 2) obs_write_nhwc_bf16<NC>((unsigned short *)obs, A, own, opp, last, lane);
    else obs_write<NC, T>(obs, A, own, opp, last, lane);
}
template <int NC, typename T>
__global__ void __launch_bounds__(CTA_THREADS) k_root_obs(Params p, T *obs)
{
    const int lane = threadIdx.x & 31, g = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= p.G) return;
    const GState *s = p.gs + g;
    const u64 P = lane < GMZ_WORDS ? s->p1[lane] : 0ull, M = lane < GMZ_WORDS ? s->m1[lane] : 0ull;
    const int tm = s->to_move;
    obs_emit<NC, T>(obs + (size_t)g * 3 * p.A, p.A, tm > 0 ? P : M, tm > 0 ? M : P, s->last_move, lane);
}

// ---------------------------------------------------------------------------------------------
// stepwise search kernels (external evaluator)
// ---------------------------------------------------------------------------------------------
template <int NC>
__device__ __forceinline__ void load_lane_logits(const float *src, int A, int lane, float *lg)
{
#pragma unroll
    for (int i = 0; i < 4 * NC; ++i) {
        const int a = 128 * (i >> 2) + 4 * lane + (i & 3);
        lg[i] = a < A ? __fadd_rn(src[a], 0.0f) : 0.0f;      // -0.0 -> +0.0: equal logits have equal bits (unvisited_summary)
    }
}
__device__ __forceinline__ double load_value(const void *v, int dtype, int g)
{
    return dtype == GMZ_F64 ? ((const double *)v)[g] : (double)((const float *)v)[g];
}

template <int NC>
__global__ void __launch_bounds__(CTA_THREADS)
k_root_expand(Params p, const float *logits, const void *values, int vdtype, const double *gumbel)
{
    const int lane = threadIdx.x & 31, g = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= p.G) return;
    __shared__ WG s_wg[WARPS_PER_CTA];
    WG &w = s_wg[threadIdx.x >> 5];
    wg_load(p, g, lane, w);
    if (!w.active) return;
    wg_valid_bits<NC>(p, w, lane);
    float lg[4 * NC]; double gum[4 * NC];
    load_lane_logits<NC>(logits + (size_t)g * p.A, p.A, lane, lg);
#pragma unroll
    for (int i = 0; i < 4 * NC; ++i) {
        const int a = 128 * (i >> 2) + 4 * lane + (i & 3);
        gum[i] = a < p.A ? gumbel[(size_t)g * p.A + a] : 0.0;
    }
    root_init<NC>(p, w, lg, gum, load_value(values, vdtype, g), lane);
    wg_store_search(p, lane, w);
    if (lane == 0) p.gs[g].leaf_depth = 0;
}

template <int NC, bool MZ, bool F32, typename T>
__global__ void __launch_bounds__(CTA_THREADS)
k_select(const __grid_constant__ Params p, T *leaf_obs, int32_t *out_a, int32_t *out_b, int32_t *out_c, int32_t *out_depth, int32_t *out_reps)
{
    // AZ: out_a = leaf action (trace).  MZ: out_a = parent slot, out_b = action, out_c = child slot.
    const int lane = threadIdx.x & 31, g = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= p.G) return;
    __shared__ WG s_wg[WARPS_PER_CTA];
    WG &w = s_wg[threadIdx.x >> 5];
    wg_load(p, g, lane, w);
    const bool run = w.active && w.sim_count >= 1 && w.sim_count < p.S;
    if (!run) {
        if (!MZ && leaf_obs) {
            T *o = leaf_obs + (size_t)g * 3 * p.A;
            for (int a = lane; a < 3 * p.A; a += 32) o[a] = (T)0.0f;
        }
        if (lane == 0) {
            if (out_a) out_a[g] = -1;
            if (out_b) out_b[g] = -1;
            if (out_c) out_c[g] = -1;
            if (out_depth) out_depth[g] = 0;
            if (out_reps) out_reps[g] = 0;
            p.gs[g].leaf_depth = 0;
        }
        return;
    }
    wg_valid_bits<NC>(p, w, lane);
    __shared__ SelSmem s_sel[WARPS_PER_CTA];
    __shared__ DescSmem s_desc[WARPS_PER_CTA];
    DescSmem &ds = s_desc[threadIdx.x >> 5];
    int2 *path = p.path + (size_t)g * (p.S + 2);
    int lp, la;
    const int depth = descend<NC, MZ, F32>(p, w, path, ds, s_sel[threadIdx.x >> 5], blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5), lane,
                                      lp, la);
    if (!MZ && leaf_obs) { // the replayed position as the player to move at the leaf sees it; last move = la
        u64 own, opp;
        replay_path(p, w, path, ds, depth, la, lane, own, opp);
        obs_emit<NC, T>(leaf_obs + (size_t)g * 3 * p.A, p.A, own, opp, la, lane);
    }
    if (lane < min(depth, 32)) path[lane] = lane == 0 ? make_int2(0, 0) : make_int2(ds.path[lane].node, ds.path[lane].mir);   // for k_expand_backup
    if (lane == 0) {
        GState *s = p.gs + g;
        s->leaf_parent = lp; s->leaf_action = la; s->leaf_depth = depth; s->leaf_reps = MZ ? w.n_surv : 1;
        if (MZ) {
            if (out_a) out_a[g] = (int32_t)(w.nbase + (size_t)lp);
            if (out_b) out_b[g] = la;
            if (out_c) out_c[g] = (int32_t)(w.nbase + (size_t)w.num_nodes);
        } else if (out_a) out_a[g] = la;
        if (out_depth) out_depth[g] = depth;
        if (out_reps) out_reps[g] = MZ ? w.n_surv : 1;
    }
}

template <int NC, bool MZ, bool F32>
__global__ void __launch_bounds__(CTA_THREADS)
k_expand_backup(const __grid_constant__ Params p, const float *logits, const void *values, const void *rewards, int vdtype)
{
    const int lane = threadIdx.x & 31, g = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= p.G) return;
    const GState *s = p.gs + g;
    const int depth = s->leaf_depth;
    if (!s->active || depth <= 0) return;
    __shared__ WG s_wg[WARPS_PER_CTA];
    WG &w = s_wg[threadIdx.x >> 5];
    wg_load(p, g, lane, w);
    const int lp = s->leaf_parent, la = s->leaf_action, reps = s->leaf_reps;
    const int2 *path = p.path + (size_t)g * (p.S + 2);
    float lg[4 * NC];
    load_lane_logits<NC>(logits + (size_t)g * p.A, p.A, lane, lg);
    const double value = load_value(values, vdtype, g);
    const double reward = (MZ && rewards) ? load_value(rewards, vdtype, g) : 0.0;
    const int nn = w.num_nodes;
    wg_valid_bits<NC>(p, w, lane);
    node_write_row<NC>(p, w, nn, lg, lane);
    node_init_hdr<NC>(p, w, nn, lg, lane);
    const int nmir = node_link<NC>(p, w, lp, la, nn, lane);
    wg_set(w.num_nodes, nn + 1);
    PathReg pr; pr.node = 0; pr.mir = 0; pr.n = 0; pr.W = 0.0; pr.R = 0.0;
    if (lane < min(depth, 32)) {        // the statistics the fused kernel keeps in registers: re-read them here
        const int2 t = path[lane]; pr.node = t.x; pr.mir = t.y;
        const size_t li = w.nbase + (size_t)t.x;
        pr.n = p.nN[li]; pr.W = p.nW[li]; if (MZ) pr.R = p.nR[li];
    }
    backup<MZ, F32>(p, w, path, pr, depth, nn, nmir, value, reward, reps, lane);
    survivor_visit(w, depth, pr.node, nn, la, reps, lane);
    const int sc = w.sim_count + reps;
    wg_set(w.sim_count, sc);
    if (halving_ready(p, w, sc)) sequential_halving<MZ, F32>(p, w, lane);
    wg_store_search(p, lane, w);
    if (lane == 0) p.gs[g].leaf_depth = 0;
}

template <int NC, bool MZ, bool F32>
__global__ void __launch_bounds__(CTA_THREADS)
k_finalize(const __grid_constant__ Params p, double *policy, double *value, int32_t *action, int32_t *visits)
{
    __shared__ short s_nvis[WARPS_PER_CTA][128 * NC];
    const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5, g = blockIdx.x * WARPS_PER_CTA + wi;
    if (g >= p.G) return;
    __shared__ WG s_wg[WARPS_PER_CTA];
    WG &w = s_wg[threadIdx.x >> 5];
    wg_load(p, g, lane, w);
    double v; int a;
    finalize_root<NC, MZ, F32>(p, w, lane, policy ? policy + (size_t)g * p.A : nullptr, visits ? visits + (size_t)g * p.A : nullptr,
                          s_nvis[wi], p.pyset + ((size_t)blockIdx.x * WARPS_PER_CTA + wi) * 4096, v, a);
    if (lane == 0) { if (value) value[g] = v; if (action) action[g] = a; }
}

// ---------------------------------------------------------------------------------------------
// E0 evaluator kernels
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS)
k_e0_eval_obs(const float *obs, int B, int N, E0Spec e0, float *logits, double *values)
{
    const int lane = threadIdx.x & 31, b = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5);
    if (b >= B) return;
    const int A = N * N, nw = (A + 63) / 64;
    const float *o = obs + (size_t)b * 3 * A;
    u64 own = 0, opp = 0; int last = -1;
    for (int w = 0; w < nw; ++w) {
        u64 ow = 0, pw = 0;
        for (int h = 0; h < 2; ++h) {
            const int a = 64 * w + 32 * h + lane;
            const bool in = a < A;
            ow |= (u64)__ballot_sync(GMZ_FULL, in && o[a] > 0.5f) << (32 * h);
            pw |= (u64)__ballot_sync(GMZ_FULL, in && o[A + a] > 0.5f) << (32 * h);
            const unsigned lb = __ballot_sync(GMZ_FULL, in && o[2 * A + a] > 0.5f);
            if (lb && last < 0) last = 64 * w + 32 * h + (__ffs(lb) - 1);
        }
        if (lane == w) { own = ow; opp = pw; }
    }
    const u64 h = e0_hash_planes(e0.h0, own, opp, nw, last, lane);
    for (int a = lane; a < A; a += 32) logits[(size_t)b * A + a] = e0_logit(h, a, e0);
    if (lane == 0) values[b] = e0_value(h, e0.dense);
}

// Gumbel(0,1) = -log(-log(u)), u from a counter-based splitmix64 stream, 53-bit mantissa in (0,1).
__global__ void k_fill_gumbel(double *out, size_t n, u64 seed, u64 offset)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = gumbel_at(mix64(seed ^ E0_GOLD), offset + i);
}

// Stepwise self-play move (external evaluator): what k_play_e0 does after its search, as a kernel of
// its own -- record (policy, value, action) in the game's trajectory slot, do_move, get_game_ended,
// hand finished games to the host queue and restart them in a fresh slot (workers.py:172-189, 230).
__global__ void __launch_bounds__(CTA_THREADS)
k_selfplay_step(const __grid_constant__ Params p, const __grid_constant__ TrajDev t, const __grid_constant__ BookDev book, int use_traj,
                int restart, const double *policy, const double *value, const int32_t *action, int32_t *out_winner)
{
    const int lane = threadIdx.x & 31, g = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= p.G) return;
    GState *s = p.gs + g;
    const int a = action[g];
    if (s->parked || a < 0 || a >= p.A || s->winner != GMZ_WINNER_NONE) {
        if (lane == 0 && out_winner) out_winner[g] = s->winner;
        return;
    }
    int slot = -1, tl = 0;
    if (use_traj) {
        slot = s->traj_slot; tl = s->traj_len;
        if (tl == 0) traj_open(t, s, slot, g, s->to_move, s->last_move, lane);
        if (tl < t.max_moves) {
            double *dst = t.policy + ((size_t)slot * t.max_moves + tl) * (size_t)p.A;
            for (int c = lane; c < p.A; c += 32) dst[c] = policy[(size_t)g * p.A + c];
        }
    }
    const int wv = move_commit(p, t, s, use_traj, slot, tl, use_traj ? value[g] : 0.0, a, lane);   // value: null without a store
    if (lane == 0 && out_winner) out_winner[g] = wv;
    if (wv != GMZ_WINNER_NONE) game_finish(p, t, book, s, g, use_traj, restart, slot, tl + 1, wv, lane);
}

// parked games (finished, no free trajectory slot at the time): take a slot and restart
__global__ void __launch_bounds__(CTA_THREADS)
k_unpark(const __grid_constant__ Params p, const __grid_constant__ TrajDev t, const __grid_constant__ BookDev book)
{
    const int lane = threadIdx.x & 31, g = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= p.G) return;
    GState *s = p.gs + g;
    if (!s->parked) return;
    int ok = 0, slot = -1;
    if (lane == 0) ok = traj_pop_slot(t, slot);
    if (__shfl_sync(GMZ_FULL, ok, 0)) game_redeal(p, book, s, g, 1, slot, lane);
}
// give every game its initial trajectory slot (slot g) and clear the play bookkeeping
__global__ void k_traj_init(Params p, TrajDev t)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < p.G) { GState *s = p.gs + i; s->traj_slot = i; s->traj_len = 0; s->parked = 0; s->busy = 0; }
    if (i < t.n_slots - p.G) t.free_slots[i] = p.G + i;
    if (i == 0) { *t.free_top = t.n_slots - p.G; *t.fin_count = 0; }
}

// ---------------------------------------------------------------------------------------------
// self-play game step: do_move + get_game_ended on the roots (game.py:20-63)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS) k_game_step(Params p, const int32_t *actions, int32_t *out_winner)
{
    const int lane = threadIdx.x & 31, g = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5);
    if (g >= p.G) return;
    GState *s = p.gs + g;
    const int a = actions[g];
    if (a < 0 || a >= p.A) { if (lane == 0 && out_winner) out_winner[g] = s->winner; return; }
    const int wv = game_do_move(p, s, a, lane);
    if (lane == 0 && out_winner) out_winner[g] = wv;
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct Layout { size_t gs, logits, child, nN, nW, nR, nH, path, pyset, selov, ctl, blk, total; };

static int validate(const gmz_config *c)
{
    if (!c) return fail("null config");
    if (c->board_size < 1 || c->board_size > GMZ_MAX_BOARD) return fail("board_size out of range (1..19)");
    if (c->num_simulations < 1 || c->num_simulations > 32767) return fail("num_simulations out of range (1..32767)");
    if (c->num_top_actions < 1 || c->num_top_actions > GMZ_MAX_TOP_ACTIONS) return fail("num_top_actions out of range (1..32)");
    if (c->mode != GMZ_MODE_ALPHAZERO && c->mode != GMZ_MODE_MUZERO) return fail("unknown mode");
    if (c->accum_dtype != GMZ_ACCUM_F64 && c->accum_dtype != GMZ_ACCUM_F32) return fail("unknown accum_dtype");
    if (c->num_games < 1) return fail("num_games must be >= 1");
    if (c->n_in_row < 1 || c->n_in_row > 14) return fail("n_in_row out of range (1..14)");
    if (c->max_moves < 0) return fail("max_moves must be >= 0");
    return 0;
}
static Layout make_layout(const gmz_config *c)
{
    const size_t A = (size_t)c->board_size * c->board_size, NC = (A + 127) / 128, AP = 128 * NC;
    const size_t G = c->num_games, S = c->num_simulations;
    Layout L; size_t o = 0;
    L.gs = o; o = align_up(o + G * sizeof(GState), 256);
    L.logits = o; o = align_up(o + G * S * AP * sizeof(float), 256);
    L.child = o; o = align_up(o + G * S * AP * sizeof(short), 256);
    L.nN = o; o = align_up(o + G * S * sizeof(int), 256);
    L.nW = o; o = align_up(o + G * S * sizeof(double), 256);
    L.nR = o; if (c->mode == GMZ_MODE_MUZERO) o = align_up(o + G * S * sizeof(double), 256);
    L.nH = o; if (c->mode == GMZ_MODE_MUZERO) o = align_up(o + G * S * sizeof(u64), 256);
    L.path = o; o = align_up(o + G * (S + 2) * sizeof(int2), 256);
    L.pyset = o; o = align_up(o + ((G + 3) / 4 * 4) * 4096 * sizeof(short), 256);
    L.selov = o; o = align_up(o + ((G + 3) / 4 * 4) * AP * 20, 256);
    L.ctl = o; o = align_up(o + sizeof(PlayCtl), 256);
    L.blk = o; o = align_up(o + G * S * (size_t)kBlkBytes, 1024);
    L.total = o;
    return L;
}

extern "C" int gmz_version(void) { return GMZ_VERSION; }
extern "C" const char *gmz_last_error(void) { return g_err; }

extern "C" size_t gmz_workspace_bytes(const gmz_config *cfg)
{
    if (validate(cfg)) return 0;
    return make_layout(cfg).total;
}

extern "C" int gmz_create(const gmz_config *cfg, void *workspace, size_t workspace_bytes, gmz_stream stream, gmz_engine **out)
{
    if (validate(cfg)) return 1;
    if (!out) return fail("null out pointer");
    const Layout L = make_layout(cfg);
    if (!workspace || workspace_bytes < L.total) return fail("workspace too small");
    if ((uintptr_t)workspace % 256) return fail("workspace must be 256-byte aligned");
    gmz_engine *e = (gmz_engine *)calloc(1, sizeof(gmz_engine));
    if (!e) return fail("out of host memory");
    e->magic = GMZ_ENGINE_MAGIC; e->cfg = *cfg; e->workspace = workspace; e->bytes = L.total;
    cudaGetDevice(&e->device);
    Params &p = e->p;
    p.G = cfg->num_games; p.N = cfg->board_size; p.A = p.N * p.N; p.S = cfg->num_simulations; p.K = cfg->num_top_actions;
    p.NW = (p.A + 63) / 64; e->NC = (p.A + 127) / 128; p.AP = 128 * e->NC; p.mode = cfg->mode;
    p.n_in_row = cfg->n_in_row; p.max_moves = cfg->max_moves > 0 ? cfg->max_moves : p.A;
    p.c_visit = cfg->c_visit; p.c_scale = cfg->c_scale; p.delta = cfg->minmax_delta; p.discount = cfg->discount;
    p.discf = (float)cfg->discount; p.deltaf = (float)cfg->minmax_delta; p.f32acc = cfg->accum_dtype == GMZ_ACCUM_F32; p.pad0 = 0;
    // sequential-halving schedule (mcts.py:158-181), same double arithmetic as the reference
    {
        const int n = p.S, m = p.K;
        const double lg2 = log2((double)m);
        if (m <= 1 || lg2 <= 0) p.first_thr = n;
        else { double v = floor((double)n / (lg2 * (double)m)) * (double)m; if ((double)n < v) v = (double)n; p.first_thr = (int)v; }
        double used = 0.0; int cm = m; p.n_phases = 0;
        for (int ph = 1; ph < GMZ_MAX_PHASES; ++ph) {
            cm /= 2;
            if (cm < 1) break;
            double extra = (cm <= 1 || lg2 <= 0) ? (double)n - used : floor((double)n / (lg2 * (double)cm)) * (double)cm;
            used += extra;
            p.m_of_phase[ph] = cm; p.extra_of_phase[ph] = (int)extra; p.n_phases = ph;
        }
    }
    char *base = (char *)workspace;
    p.gs = (GState *)(base + L.gs); p.logits = (float *)(base + L.logits); p.child = (short *)(base + L.child);
    p.nN = (int *)(base + L.nN); p.nW = (double *)(base + L.nW);
    p.nR = cfg->mode == GMZ_MODE_MUZERO ? (double *)(base + L.nR) : nullptr;
    p.nH = cfg->mode == GMZ_MODE_MUZERO ? (u64 *)(base + L.nH) : nullptr;
    p.path = (int2 *)(base + L.path);
    p.pyset = (short *)(base + L.pyset); p.sel_overflow = base + L.selov; p.ctl = (PlayCtl *)(base + L.ctl);
    p.nBlk = base + L.blk;
    cudaError_t err = cudaMemsetAsync(base + L.gs, 0, (size_t)p.G * sizeof(GState), (cudaStream_t)stream);
    if (err == cudaSuccess) err = cudaMemsetAsync(base + L.ctl, 0, sizeof(PlayCtl), (cudaStream_t)stream);
    if (err != cudaSuccess) { free(e); return fail("cudaMemsetAsync: %s", cudaGetErrorString(err)); }
    { std::lock_guard<std::mutex> lk(g_live_mu); g_live.insert(e); }
    *out = e;
    return 0;
}

// Idempotent: destroying a handle that is not live (already destroyed, or never created) does nothing.
extern "C" int gmz_destroy(gmz_engine *e)
{
    if (!e) return 0;
    {
        std::lock_guard<std::mutex> lk(g_live_mu);
        if (!g_live.erase(e)) return 0;
    }
    e->magic = 0;
    free(e);
    return 0;
}

#define GRID(e) dim3(((e)->p.G + WARPS_PER_CTA - 1) / WARPS_PER_CTA), dim3(CTA_THREADS)
#define LIVE(e, name) do { if (!engine_live(e)) return fail("%s: invalid or destroyed engine handle", name); } while (0)
#define DISPATCH_NC(e, ...)                                      \
    switch ((e)->NC) {                                           \
        case 1: { constexpr int NC = 1; __VA_ARGS__; } break;    \
        case 2: { constexpr int NC = 2; __VA_ARGS__; } break;    \
        default: { constexpr int NC = 3; __VA_ARGS__; } break;   \
    }
// NC x (MuZero mode) x (float32 accumulation)
#define DISPATCH_ALL(e, ...)                                                                      \
    do {                                                                                          \
        const int mz_ = (e)->p.mode == GMZ_MODE_MUZERO, f_ = (e)->p.f32acc;                       \
        if (mz_ && f_) { constexpr bool MZ = true, F32 = true; DISPATCH_NC(e, __VA_ARGS__) }      \
        else if (mz_) { constexpr bool MZ = true, F32 = false; DISPATCH_NC(e, __VA_ARGS__) }      \
        else if (f_) { constexpr bool MZ = false, F32 = true; DISPATCH_NC(e, __VA_ARGS__) }       \
        else { constexpr bool MZ = false, F32 = false; DISPATCH_NC(e, __VA_ARGS__) }              \
    } while (0)

extern "C" int gmz_set_roots(gmz_engine *e, const int8_t *boards, const int8_t *players, const int32_t *last_moves,
                             const int32_t *move_counts, gmz_stream stream)
{
    LIVE(e, "gmz_set_roots");
    if (!boards || !players || !last_moves || !move_counts) return fail("gmz_set_roots: null argument");
    k_set_roots<<<GRID(e), 0, (cudaStream_t)stream>>>(e->p, boards, players, last_moves, move_counts);
    return check_launch("k_set_roots");
}
extern "C" int gmz_set_roots_from_records(gmz_engine *e, const void *ring, int64_t capacity, int64_t first, int64_t n,
                                          gmz_stream stream)
{
    if (!ring) return fail("gmz_set_roots_from_records: null argument");
    if (const char *m = rec_stretch_check(capacity, first, n)) return fail("gmz_set_roots_from_records: %s", m);
    LIVE(e, "gmz_set_roots_from_records");
    if (n > e->p.G) return fail("gmz_set_roots_from_records: n exceeds the engine's num_games");
    if (n == 0) return 0;
    k_set_roots_records<<<GRID(e), 0, (cudaStream_t)stream>>>(e->p, (const unsigned char *)ring, rec_stride(e->p.A), capacity, first,
                                                              (int)n);
    return check_launch("k_set_roots_records");
}
extern "C" int gmz_games_reset(gmz_engine *e, const uint8_t *mask, gmz_stream stream)
{
    LIVE(e, "gmz_games_reset");
    k_games_reset<<<GRID(e), 0, (cudaStream_t)stream>>>(e->p, e->book, mask);
    return check_launch("k_games_reset");
}
extern "C" int gmz_get_roots(gmz_engine *e, int8_t *boards, int8_t *players, int32_t *last_moves, int32_t *move_counts,
                             gmz_stream stream)
{
    LIVE(e, "gmz_get_roots");
    k_get_roots<<<GRID(e), 0, (cudaStream_t)stream>>>(e->p, boards, players, last_moves, move_counts);
    return check_launch("k_get_roots");
}
extern "C" int gmz_root_obs(gmz_engine *e, void *obs, int obs_dtype, gmz_stream stream)
{
    LIVE(e, "gmz_root_obs");
    if (!obs) return fail("gmz_root_obs: null argument");
    if (obs_dtype == GMZ_F32) { DISPATCH_NC(e, k_root_obs<NC, float><<<GRID(e), 0, (cudaStream_t)stream>>>(e->p, (float *)obs)); }
    else if (obs_dtype == GMZ_BF16) { DISPATCH_NC(e, k_root_obs<NC, unsigned short><<<GRID(e), 0, (cudaStream_t)stream>>>(e->p, (unsigned short *)obs)); }
    else return fail("gmz_root_obs: obs_dtype must be GMZ_F32 (NCHW float32) or GMZ_BF16 (NHWC bfloat16)");
    return check_launch("k_root_obs");
}
extern "C" int gmz_root_expand(gmz_engine *e, const float *logits, const void *values, int value_dtype,
                               const double *gumbel, gmz_stream stream)
{
    LIVE(e, "gmz_root_expand");
    if (!logits || !values || !gumbel) return fail("gmz_root_expand: null argument");
    if (value_dtype != GMZ_F32 && value_dtype != GMZ_F64) return fail("gmz_root_expand: bad value dtype");
    DISPATCH_NC(e, k_root_expand<NC><<<GRID(e), 0, (cudaStream_t)stream>>>(e->p, logits, values, value_dtype, gumbel));
    return check_launch("k_root_expand");
}
extern "C" int gmz_select(gmz_engine *e, void *leaf_obs, int obs_dtype, int32_t *out_leaf_action, int32_t *out_leaf_depth,
                          gmz_stream stream)
{
    LIVE(e, "gmz_select");
    if (e->p.mode != GMZ_MODE_ALPHAZERO) return fail("gmz_select: engine is in MuZero mode, use gmz_select_mz");
    if (obs_dtype != GMZ_F32 && obs_dtype != GMZ_BF16)
        return fail("gmz_select: obs_dtype must be GMZ_F32 (NCHW float32) or GMZ_BF16 (NHWC bfloat16)");
#define GMZ_SEL(F, T) DISPATCH_NC(e, k_select<NC, false, F, T><<<GRID(e), 0, (cudaStream_t)stream>>>(e->p, (T *)leaf_obs, out_leaf_action, \
                                                                                           nullptr, nullptr, out_leaf_depth, nullptr))
    if (obs_dtype == GMZ_F32) { if (e->p.f32acc) { GMZ_SEL(true, float); } else { GMZ_SEL(false, float); } }
    else { if (e->p.f32acc) { GMZ_SEL(true, unsigned short); } else { GMZ_SEL(false, unsigned short); } }
#undef GMZ_SEL
    return check_launch("k_select");
}
extern "C" int gmz_select_mz(gmz_engine *e, int32_t *out_parent_slot, int32_t *out_action, int32_t *out_child_slot,
                             int32_t *out_leaf_depth, int32_t *out_reps, gmz_stream stream)
{
    LIVE(e, "gmz_select_mz");
    if (e->p.mode != GMZ_MODE_MUZERO) return fail("gmz_select_mz: engine is in AlphaZero mode, use gmz_select");
    if (e->p.f32acc) {
        DISPATCH_NC(e, k_select<NC, true, true, float><<<GRID(e), 0, (cudaStream_t)stream>>>(e->p, nullptr, out_parent_slot, out_action,
                                                                                           out_child_slot, out_leaf_depth, out_reps));
    } else {
        DISPATCH_NC(e, k_select<NC, true, false, float><<<GRID(e), 0, (cudaStream_t)stream>>>(e->p, nullptr, out_parent_slot, out_action,
                                                                                            out_child_slot, out_leaf_depth, out_reps));
    }
    return check_launch("k_select_mz");
}
extern "C" int gmz_expand_backup(gmz_engine *e, const float *logits, const void *values, const void *rewards,
                                 int value_dtype, gmz_stream stream)
{
    LIVE(e, "gmz_expand_backup");
    if (!logits || !values) return fail("gmz_expand_backup: null argument");
    if (value_dtype != GMZ_F32 && value_dtype != GMZ_F64) return fail("gmz_expand_backup: bad value dtype");
    DISPATCH_ALL(e, k_expand_backup<NC, MZ, F32><<<GRID(e), 0, (cudaStream_t)stream>>>(e->p, logits, values, rewards, value_dtype));
    return check_launch("k_expand_backup");
}
extern "C" int gmz_finalize(gmz_engine *e, double *policy, double *value, int32_t *action, int32_t *visits, gmz_stream stream)
{
    LIVE(e, "gmz_finalize");
    DISPATCH_ALL(e, k_finalize<NC, MZ, F32><<<GRID(e), 0, (cudaStream_t)stream>>>(e->p, policy, value, action, visits));
    return check_launch("k_finalize");
}
extern "C" int gmz_e0_eval_obs(const float *obs, int batch, int board_size, uint64_t seed, int logit_div,
                               float *logits, double *values, gmz_stream stream)
{
    if (!obs || !logits || !values) return fail("gmz_e0_eval_obs: null argument");
    if (batch <= 0) return 0;
    if (board_size < 1 || board_size > GMZ_MAX_BOARD) return fail("gmz_e0_eval_obs: board_size out of range");
    if (logit_div < 0) return fail("gmz_e0_eval_obs: logit_div must be >= 0 (0 = dense logits)");
    k_e0_eval_obs<<<(batch + WARPS_PER_CTA - 1) / WARPS_PER_CTA, CTA_THREADS, 0, (cudaStream_t)stream>>>(
        obs, batch, board_size, e0_spec((u64)seed, logit_div), logits, values);
    return check_launch("k_e0_eval_obs");
}
static int launch_play(gmz_engine *e, const PlayArgs &a, cudaStream_t st)
{
    const bool f = e->p.f32acc != 0;
    if (e->p.mode == GMZ_MODE_MUZERO) return f ? gmz_launch_play_mz1_f1(e, a, st) : gmz_launch_play_mz1_f0(e, a, st);
    return f ? gmz_launch_play_mz0_f1(e, a, st) : gmz_launch_play_mz0_f0(e, a, st);
}
static TrajDev traj_dev(const gmz_traj *t)
{
    TrajDev d; memset(&d, 0, sizeof(d));
    if (!t) return d;
    d.n_slots = t->n_slots; d.max_moves = t->max_moves; d.fin_cap = t->fin_cap;
    d.policy = t->policy; d.value = t->value; d.action = t->action;
    d.start_board = (u64 *)t->start_board; d.start_info = t->start_info;
    d.free_slots = t->free_slots; d.free_top = t->free_top; d.fin_queue = t->fin_queue; d.fin_count = t->fin_count;
    d.start_opening = t->start_opening;
    return d;
}
static int check_traj(const gmz_engine *e, const gmz_traj *t)
{
    if (!t->policy || !t->value || !t->action || !t->start_board || !t->start_info || !t->free_slots || !t->free_top ||
        !t->fin_queue || !t->fin_count) return fail("gmz_traj: null buffer");
    if (t->n_slots < e->p.G) return fail("gmz_traj: n_slots must be >= num_games");
    if (t->fin_cap < t->n_slots) return fail("gmz_traj: fin_cap must be >= n_slots");
    if (t->max_moves < 1) return fail("gmz_traj: max_moves must be >= 1");
    return 0;
}

extern "C" int gmz_search_e0(gmz_engine *e, const double *gumbel, uint64_t seed, int logit_div,
                             int32_t *trace_leaf_action, int32_t *trace_leaf_depth, gmz_stream stream)
{
    LIVE(e, "gmz_search_e0");
    if (!gumbel) return fail("gmz_search_e0: null argument");
    if (logit_div < 0 || (logit_div & (logit_div - 1))) return fail("gmz_search_e0: logit_div must be 0 (dense logits) or a power of two");
    PlayArgs a; memset(&a, 0, sizeof(a));
    a.e0 = e0_spec((u64)seed, logit_div);
    a.total_tickets = e->p.G; a.do_step = 0; a.gumbel_in = gumbel;
    a.trace_a = trace_leaf_action; a.trace_d = trace_leaf_depth;
    return launch_play(e, a, (cudaStream_t)stream);
}
extern "C" int gmz_traj_init(gmz_engine *e, const gmz_traj *traj, gmz_stream stream)
{
    LIVE(e, "gmz_traj_init");
    if (!traj) return fail("gmz_traj_init: null argument");
    if (check_traj(e, traj)) return 1;
    const int n = traj->n_slots > e->p.G ? traj->n_slots : e->p.G;
    k_traj_init<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(e->p, traj_dev(traj));
    return check_launch("k_traj_init");
}
extern "C" int gmz_selfplay_e0(gmz_engine *e, const gmz_traj *traj, uint64_t eval_seed, int logit_div, uint64_t noise_seed,
                               int64_t total_moves, int restart, gmz_stream stream)
{
    LIVE(e, "gmz_selfplay_e0");
    if (traj && check_traj(e, traj)) return 1;
    if (logit_div < 0 || (logit_div & (logit_div - 1))) return fail("gmz_selfplay_e0: logit_div must be 0 (dense logits) or a power of two");
    if (total_moves <= 0) return 0;
    PlayArgs a; memset(&a, 0, sizeof(a));
    a.e0 = e0_spec((u64)eval_seed, logit_div); a.noise_seed = noise_seed;
    a.total_tickets = total_moves; a.do_step = 1; a.restart = restart ? 1 : 0; a.use_traj = traj ? 1 : 0;
    a.traj = traj_dev(traj); a.book = e->book;
    return launch_play(e, a, (cudaStream_t)stream);
}
extern "C" int gmz_selfplay_step(gmz_engine *e, const gmz_traj *traj, const double *policy, const double *value,
                                 const int32_t *action, int restart, int32_t *out_winner, gmz_stream stream)
{
    LIVE(e, "gmz_selfplay_step");
    if (!action) return fail("gmz_selfplay_step: null argument");
    if (traj && (check_traj(e, traj) || !policy || !value)) return traj && policy && value ? 1 : fail("gmz_selfplay_step: policy/value required with a trajectory store");
    k_selfplay_step<<<GRID(e), 0, (cudaStream_t)stream>>>(e->p, traj_dev(traj), e->book, traj ? 1 : 0, restart ? 1 : 0, policy, value, action, out_winner);
    return check_launch("k_selfplay_step");
}
extern "C" int gmz_selfplay_unpark(gmz_engine *e, const gmz_traj *traj, gmz_stream stream)
{
    LIVE(e, "gmz_selfplay_unpark");
    if (!traj) return fail("gmz_selfplay_unpark: null argument");
    if (check_traj(e, traj)) return 1;
    k_unpark<<<GRID(e), 0, (cudaStream_t)stream>>>(e->p, traj_dev(traj), e->book);
    return check_launch("k_unpark");
}
extern "C" int gmz_set_openings(gmz_engine *e, const gmz_openings *book, gmz_stream stream)
{
    if (book && book->n_openings < 1) return fail("gmz_set_openings: n_openings must be >= 1");
    if (book && (!book->boards || !book->players || !book->last_moves || !book->move_counts))
        return fail("gmz_set_openings: null array");
    LIVE(e, "gmz_set_openings");
    // every game's deal counter k back to 0: one 4-byte field per 1 KiB GState
    cudaError_t err = cudaMemset2DAsync(&e->p.gs->deals, sizeof(GState), 0, sizeof(unsigned), e->p.G, (cudaStream_t)stream);
    if (err != cudaSuccess) return fail("gmz_set_openings: %s", cudaGetErrorString(err));
    memset(&e->book, 0, sizeof(e->book));
    if (book) {
        e->book.n = book->n_openings; e->book.boards = book->boards; e->book.players = book->players;
        e->book.last_moves = book->last_moves; e->book.move_counts = book->move_counts;
    }
    return 0;
}
extern "C" int gmz_play_counters(gmz_engine *e, uint64_t *out2, gmz_stream stream)
{
    LIVE(e, "gmz_play_counters");
    if (!out2) return fail("gmz_play_counters: null argument");
    cudaError_t err = cudaMemcpyAsync(out2, &e->p.ctl->moves_played, 4 * sizeof(uint64_t), cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
    if (err != cudaSuccess) return fail("gmz_play_counters: %s", cudaGetErrorString(err));
    return 0;
}
extern "C" int gmz_select_counters(gmz_engine *e, uint64_t *out3, gmz_stream stream)
{
    LIVE(e, "gmz_select_counters");
    if (!out3) return fail("gmz_select_counters: null argument");
    cudaError_t err = cudaMemcpyAsync(out3, &e->p.ctl->sel_fallback, 3 * sizeof(uint64_t), cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
    if (err != cudaSuccess) return fail("gmz_select_counters: %s", cudaGetErrorString(err));
    return 0;
}
extern "C" int gmz_fill_gumbel(double *out, size_t n, uint64_t seed, uint64_t offset, gmz_stream stream)
{
    if (!out) return fail("gmz_fill_gumbel: null argument");
    if (n == 0) return 0;
    k_fill_gumbel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(out, n, (u64)seed, (u64)offset);
    return check_launch("k_fill_gumbel");
}
extern "C" int gmz_game_step(gmz_engine *e, const int32_t *actions, int32_t *out_winner, gmz_stream stream)
{
    LIVE(e, "gmz_game_step");
    if (!actions) return fail("gmz_game_step: null argument");
    k_game_step<<<GRID(e), 0, (cudaStream_t)stream>>>(e->p, actions, out_winner);
    return check_launch("k_game_step");
}
