// gmz_play.cuh -- decision phase, game step, and the persistent "play" kernel that runs whole
// searches / whole self-play moves for one game per warp with E0 inlined.
//
// Work distribution: per-search work is heavy tailed (a few games grow 100-ply-deep chains and
// take 5x the mean), so a static game->warp mapping leaves most SMs idle while the slowest games
// finish.  k_play_e0 instead hands out TICKETS from a global atomic counter: a ticket is "one
// search (+ one self-play move) of one game"; a warp that finishes takes the next ticket.  Games
// are protected by a busy flag (acquire / release with device-scope fences), and everything a
// game owns lives in global memory (GState + its node pool), so any warp on any SM can continue it.
#pragma once
#include "gmz_tree.cuh"
#include "gmz_engine.cuh"

// CPython set iteration order over the valid actions, to break ties of the final
// max(visit_counts, key=visit_counts.get) the way the reference does (mcts.py:274-275).
// Runs on one lane, only when the maximum visit count is not unique.  Restates
// Objects/setobject.c (set_add_entry / set_table_resize / set_insert_clean, CPython >= 3.7).
// `table` = 4096 shorts of scratch (two 2048-entry halves).
static __device__ __noinline__ int pyset_first_max(const u64 *vw, int A, const short *nvis, int maxn, short *table)
{
    int mask = 7, fill = 0;
    for (int i = 0; i < 8; ++i) table[i] = -1;
    short *cur = table, *alt = table + 2048;
    for (int a = 0; a < A; ++a) {
        if (!((vw[a >> 6] >> (a & 63)) & 1ull)) continue;
        unsigned i = (unsigned)a & mask, perturb = (unsigned)a, e;
        for (;;) {
            e = i;
            int probes = (i + 9 <= (unsigned)mask) ? 9 : 0; bool found = false;
            do { if (cur[e] < 0) { found = true; break; } ++e; } while (probes--);
            if (found) break;
            perturb >>= 5; i = (i * 5 + 1 + perturb) & mask;
        }
        cur[e] = (short)a; ++fill;
        if (fill * 5 >= mask * 3) {
            int newsize = 8; const int minused = fill * 4;
            while (newsize <= minused) newsize <<= 1;
            const int nmask = newsize - 1;
            for (int j = 0; j < newsize; ++j) alt[j] = -1;
            for (int j = 0; j <= mask; ++j) {
                if (cur[j] < 0) continue;
                const unsigned h2 = (unsigned)cur[j];
                unsigned ii = h2 & nmask, pp = h2, ee;
                for (;;) {
                    ee = ii;
                    if (alt[ee] < 0) break;
                    bool ok = false;
                    if (ii + 9 <= (unsigned)nmask) { for (int q = 0; q < 9; ++q) { ++ee; if (alt[ee] < 0) { ok = true; break; } } }
                    if (ok) break;
                    pp >>= 5; ii = (ii * 5 + 1 + pp) & nmask;
                }
                alt[ee] = cur[j];
            }
            short *t = cur; cur = alt; alt = t; mask = nmask;
        }
    }
    for (int j = 0; j <= mask; ++j) if (cur[j] >= 0 && nvis[cur[j]] == maxn) return cur[j];
    return -1;
}

// Decision phase (mcts.py:271-280): improved policy at the root, root value, most-visited action.
// policy / visits point at this game's [A] output rows (may be null).  nvis: 128*NC shorts of
// per-warp shared scratch; table: 4096 shorts of per-warp global scratch (tie-break only).
template <int NC, bool MZ, bool F32>
__device__ __noinline__ void finalize_root(const Params &p, WG &w, int lane, double *policy, int32_t *visits,
                                           short *nvis, short *table, double &value, int &action)
{
    if (!w.active || w.sim_count < 1) {   // sentinel (np.zeros(A), 0.0, -1), mcts.py:214-215
        for (int a = lane; a < p.A; a += 32) {
            if (policy) policy[a] = 0.0;
            if (visits) visits[a] = 0;
        }
        value = 0.0; action = -1;
        return;
    }
    wg_valid_bits<NC>(p, w, lane);
    Row<NC> r;
    row_load<NC, MZ, F32>(p, w, 0, lane, r);
    double x[4 * NC];
    const double inv = row_softmax<NC, F32>(p, w, r, x, lane);
    const unsigned wvb = w.vb[lane];
    int bn = -1, ba = 0x7fffffff;
#pragma unroll
    for (int i = 0; i < 4 * NC; ++i) {
        const int a = 128 * (i >> 2) + 4 * lane + (i & 3);
        nvis[a] = (short)r.n[i];
        if (a < p.A) {
            if (policy) policy[a] = __dmul_rn(x[i], inv);
            if (visits) visits[a] = r.n[i];
            if (((wvb >> i) & 1u) && r.n[i] > bn) { bn = r.n[i]; ba = a; }
        }
    }
    const int maxn = __reduce_max_sync(GMZ_FULL, bn);
    int ties = 0;
#pragma unroll
    for (int i = 0; i < 4 * NC; ++i) ties += (((wvb >> i) & 1u) && r.n[i] == maxn) ? 1 : 0;
    ties = __reduce_add_sync(GMZ_FULL, ties);
    int best = __reduce_min_sync(GMZ_FULL, bn == maxn ? ba : 0x7fffffff);
    __syncwarp();
    if (ties > 1) {
        u64 vw[GMZ_WORDS];
#pragma unroll
        for (int k = 0; k < GMZ_WORDS; ++k) vw[k] = p.gs[w.g].valid[k];
        if (lane == 0) best = pyset_first_max(vw, p.A, nvis, maxn, table);
        best = __shfl_sync(GMZ_FULL, best, 0);
    }
    value = F32 ? (double)__fdiv_rn((float)p.nW[w.nbase], (float)p.nN[w.nbase])       // root.get_value(), mcts.py:273
                : __ddiv_rn(p.nW[w.nbase], (double)p.nN[w.nbase]);
    action = best;
    __syncwarp();
}

// game.do_move(a) + game.get_game_ended() on a root (game.py:20-63, workers.py:178-181).
// check_win: 4 directions through the last move, up to n_in_row+1 stones each way; lane l tests
// the cell at offset (l - span) along the direction and the ballot is the line's bit pattern.
// Returns +-1 (winner's colour), 0 (draw) or GMZ_WINNER_NONE; updates the GState.
__device__ __forceinline__ int game_do_move(const Params &p, GState *s, int a, int lane)
{
    const int colour = s->to_move;
    u64 P = lane < GMZ_WORDS ? s->p1[lane] : 0ull, M = lane < GMZ_WORDS ? s->m1[lane] : 0ull;
    bb_do_move(P, M, colour, a, lane);
    const int mc = s->move_count + 1;
    const int r = a / p.N, c = a % p.N, span = p.n_in_row + 1;
    const int off = lane - span;
    bool win = false;
    const int DR[4] = {0, 1, 1, 1}, DC[4] = {1, 0, 1, -1};
#pragma unroll
    for (int d = 0; d < 4; ++d) {
        const int rr = r + off * DR[d], cc = c + off * DC[d];
        const bool in = lane <= 2 * span && rr >= 0 && rr < p.N && cc >= 0 && cc < p.N;
        const int cell = in ? rr * p.N + cc : 0;
        const u64 mine = shfl_u64(colour > 0 ? P : M, cell >> 6);
        const unsigned line = __ballot_sync(GMZ_FULL, in && ((mine >> (cell & 63)) & 1ull));
        const unsigned up = line >> (span + 1);               // cells after the stone
        const int fwd = __ffs(~up) - 1;
        const unsigned dn = __brev(line << (32 - span));      // cells before the stone, nearest first
        const int bwd = __ffs(~dn) - 1;
        win = win || (1 + min(fwd, span) + min(bwd, span)) >= p.n_in_row;
    }
    const int wv = win ? colour : (mc >= p.A ? 0 : GMZ_WINNER_NONE);
    if (lane < GMZ_WORDS) {
        s->p1[lane] = P; s->m1[lane] = M;
        u64 fullm = 0; const int lo = 64 * lane;
        if (lo < p.A) fullm = (p.A - lo >= 64) ? ~0ull : ((1ull << (p.A - lo)) - 1ull);
        s->valid[lane] = ~(P | M) & fullm;
    }
    if (lane == 0) {
        s->to_move = -colour; s->last_move = a; s->move_count = mc; s->winner = wv;
        s->active = (wv == GMZ_WINNER_NONE);
        s->sim_count = 0; s->leaf_depth = 0;
    }
    return wv;
}

// Gumbel(0,1) noise from a counter-based splitmix64 stream: -log(-log(u)), u in (0,1) with 53 bits.
// (z >> 11) + 0.5 rounds to even once z >> 11 >= 2^52, so z >> 11 = 2^53 - 1 would give u = 1 and +inf noise:
// that draw is clamped to 1 - 2^-53, a value no other draw produces.
__device__ __forceinline__ double gumbel_at(u64 seed_mixed, u64 counter)
{
    const u64 z = mix64(seed_mixed + counter * E0_GOLD);
    const double u = fmin(((double)(z >> 11) + 0.5) * (1.0 / 9007199254740992.0), 1.0 - 1.0 / 9007199254740992.0);
    return -log(-log(u));
}

// Caller-owned trajectory storage (gmz_traj in include/gmz.h), device pointers.
struct TrajDev {
    int n_slots, max_moves, fin_cap, pad;
    double *policy;      // [n_slots][max_moves][A]
    double *value;       // [n_slots][max_moves]
    int32_t *action;     // [n_slots][max_moves]
    u64 *start_board;    // [n_slots][2][GMZ_WORDS]  p1 / m1 at the first recorded move
    int32_t *start_info; // [n_slots][4]  player to move, move_count, last_move, game index
    int32_t *free_slots; // stack of free slot ids
    int32_t *free_top;   // number of ids on the stack
    int32_t *fin_queue;  // [fin_cap][4] = slot, game, length, winner
    int32_t *fin_count;
    int32_t *start_opening;   // [n_slots]  book opening + 1 of the game recorded in a slot, 0 = none (may be null)
};

struct PlayArgs {
    E0Spec e0;            // the fixed evaluator (seed, quantised / dense heads)
    u64 noise_seed;
    long long total_tickets;
    int do_step;          // 1: self-play move (decision + record + do_move + restart); 0: search only
    int restart;          // self-play: restart finished games inside the launch
    int use_traj;
    const double *gumbel_in;   // search-only: external noise [G][A] (nullptr = generate)
    double *out_policy; double *out_value; int32_t *out_action; int32_t *out_visits;   // search-only outputs
    int32_t *trace_a, *trace_d;   // [G][S] leaf action / depth per evaluation (search-only, optional)
    TrajDev traj;
    BookDev book;         // self-play deals (game_deal)
};

// The self-play move commit (workers.py:172-189), shared by k_play_e0, k_selfplay_step and k_unpark.  Each caller
// writes the move's policy row itself; to_move / last_move are the root's, passed in by the caller.

// First recorded move of the game in `slot`: remember the position it started from and its opening label.
__device__ __forceinline__ void traj_open(const TrajDev &t, const GState *s, int slot, int g, int to_move, int last_move,
                                          int lane)
{
    if (lane < GMZ_WORDS) {
        t.start_board[((size_t)slot * 2 + 0) * GMZ_WORDS + lane] = s->p1[lane];
        t.start_board[((size_t)slot * 2 + 1) * GMZ_WORDS + lane] = s->m1[lane];
    }
    if (lane == 0) {
        int32_t *si = t.start_info + (size_t)slot * 4;
        si[0] = to_move; si[1] = s->move_count; si[2] = last_move; si[3] = g;
        if (t.start_opening) t.start_opening[slot] = s->opening;
    }
}

// Record value and action as move tl of `slot` (moves past max_moves are played, not recorded), play the move and count
// it.  Returns game_do_move's winner.
__device__ __forceinline__ int move_commit(const Params &p, const TrajDev &t, GState *s, int use_traj, int slot, int tl,
                                           double value, int action, int lane)
{
    if (use_traj && lane == 0 && tl < t.max_moves) {
        t.value[(size_t)slot * t.max_moves + tl] = value;
        t.action[(size_t)slot * t.max_moves + tl] = action;
    }
    __syncwarp();
    const int wv = game_do_move(p, s, action, lane);
    if (lane == 0) {
        s->noise_ctr += 1; s->traj_len = tl + 1;
        atomicAdd(&p.ctl->moves_played, 1ull);
    }
    return wv;
}

// Pop a free trajectory slot (lane 0); false when the free stack is empty.
__device__ __forceinline__ bool traj_pop_slot(const TrajDev &t, int &slot)
{
    const int idx = atomicSub(t.free_top, 1) - 1;
    if (idx < 0) { atomicAdd(t.free_top, 1); return false; }
    slot = t.free_slots[idx];
    return true;
}

// Deal game g a new game, recorded into `slot` when there is a store.
__device__ __forceinline__ void game_redeal(const Params &p, const BookDev &b, GState *s, int g, int use_traj, int slot, int lane)
{
    game_deal(p, b, s, g, lane);
    if (lane == 0 && use_traj) s->traj_slot = slot;
}

// Game g has ended (winner wv after len moves): hand its slot to the host through the finish queue, then deal it a new
// game if `restart` and a free slot allow.  Otherwise it parks with a store (k_unpark deals it once slots are released)
// and stays finished without one.  A full finish queue drops the row and parks the game.
__device__ __forceinline__ void game_finish(const Params &p, const TrajDev &t, const BookDev &b, GState *s, int g,
                                            int use_traj, int restart, int slot, int len, int wv, int lane)
{
    int ok = 1, nslot = -1;
    if (lane == 0) {
        atomicAdd(&p.ctl->games_finished, 1ull);
        if (use_traj) {
            const int qi = atomicAdd(t.fin_count, 1);
            if (qi < t.fin_cap) { int32_t *q = t.fin_queue + (size_t)qi * 4; q[0] = slot; q[1] = g; q[2] = len; q[3] = wv; }
            ok = (qi < t.fin_cap) && restart && traj_pop_slot(t, nslot);
            if (qi >= t.fin_cap) atomicSub(t.fin_count, 1);
        } else ok = restart;
    }
    ok = __shfl_sync(GMZ_FULL, ok, 0);
    nslot = __shfl_sync(GMZ_FULL, nslot, 0);
    __syncwarp();
    if (ok) game_redeal(p, b, s, g, use_traj, nslot, lane);
    else if (lane == 0) s->parked = use_traj ? 1 : 0;
}

struct PlayArgs;
// Root of a search inside the play kernel: evaluate the root with E0, draw (or load) the Gumbel
// noise, expand + top-k (mcts.py:203-226).  Out of line: it runs once per 400 simulations, and
// keeping its registers out of the simulation loop's allocation is worth more than the call.
template <int NC>
__device__ __noinline__ u64 play_root(const Params &p, const PlayArgs &a, WG &w, unsigned noise_ctr, u64 noise_mixed, int lane);

// Launch shape: ONE warp (= one game) per CTA, 28 CTAs per SM (72 registers; 28 x 148 = 4144 warps >= the 4096 games of
// the headline configuration, so every game is resident).  A warp is the unit of everything here -- no CTA-wide
// barrier, no data shared between warps -- so a CTA of several warps only ties unrelated games together.  With one
// warp per CTA (a) everything warp-uniform (game index, pool bases, counters, the shared-memory addresses of the game
// view) is CTA-uniform, which the compiler can prove: it moves to the uniform datapath and out of the 72 vector
// registers (local-memory instructions per simulation 47 -> 14); (b) a search-only launch frees a CTA slot the moment
// its search ends, not when the slowest of four does.  Measured against 4 warps x 7 CTAs, same sources: 580 vs 514 M
// sims/s in the persistent self-play launch, 538 vs 462 M end to end from host batches (6 launches in flight).
#ifndef GMZ_PLAY_MIN_CTAS
#define GMZ_PLAY_MIN_CTAS 28
#endif
#ifndef GMZ_PLAY_WARPS
#define GMZ_PLAY_WARPS 1
#endif

template <int NC>
__device__ __noinline__ u64 play_root(const Params &p, const PlayArgs &a, WG &w, unsigned noise_ctr, u64 noise_mixed, int lane)
{
    const int g = w.g;
    const GState *gs = p.gs + g;
    const u64 rP = lane < GMZ_WORDS ? gs->p1[lane] : 0ull, rM = lane < GMZ_WORDS ? gs->m1[lane] : 0ull;
    const u64 h = e0_hash_planes(a.e0.h0, w.to_move > 0 ? rP : rM, w.to_move > 0 ? rM : rP, p.NW, w.last_move, lane);
    const u64 nctr = ((u64)noise_ctr * (u64)p.G + (u64)g) * (u64)p.A;
    float lg[4 * NC]; double gum[4 * NC];
#pragma unroll 1
    for (int i = 0; i < 4 * NC; ++i) {
        const int ac = 128 * (i >> 2) + 4 * lane + (i & 3);
        lg[i] = ac < p.A ? e0_logit(h, ac, a.e0) : 0.0f;
        gum[i] = ac < p.A ? (a.gumbel_in ? a.gumbel_in[(size_t)g * p.A + ac] : gumbel_at(noise_mixed, nctr + ac)) : 0.0;
    }
    root_init<NC>(p, w, lg, gum, e0_value(h, a.e0.dense), lane);
    return h;
}

// One search (mcts.py:197-280) -- and in self-play mode one whole move (workers.py:168-189) --
// per ticket, one game per warp, E0 inlined.
template <int NC, bool MZ, bool F32>
__global__ void __launch_bounds__(32 * GMZ_PLAY_WARPS, GMZ_PLAY_MIN_CTAS)
k_play_e0(const __grid_constant__ Params p, const __grid_constant__ PlayArgs a)
{
    __shared__ SelSmem s_sel[GMZ_PLAY_WARPS];
    __shared__ DescSmem s_desc[GMZ_PLAY_WARPS];
    __shared__ WG s_wg[GMZ_PLAY_WARPS];
    __shared__ short s_nvis[GMZ_PLAY_WARPS][128 * NC];
    const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
    const int warp_slot = blockIdx.x * GMZ_PLAY_WARPS + wi;
    short *table = p.pyset + (size_t)warp_slot * 4096;
    const u64 noise_mixed = mix64(a.noise_seed ^ E0_GOLD);
    for (;;) {
        // Pick a game: every attempt draws the next position of ONE global cursor that sweeps the
        // games round-robin, so the cursor always points at the game that has been idle longest
        // (a per-warp linear probe instead can run in lock-step with the window of busy games and
        // starve).  A busy / parked game is simply skipped; a move is only counted once a game is held.
        int g = 0;
        bool got = false, done = false;
        for (int tries = 0; tries < 4 * p.G; ++tries) {
            unsigned long long t = 0;
            int ok = 0;
            if (lane == 0) {
                t = atomicAdd(&p.ctl->next_ticket, 1ull);
                if (!a.do_step && (long long)t >= a.total_tickets) ok = -1;      // search-only: one ticket per game
                else {
                    GState *s = p.gs + (int)(t % (unsigned long long)p.G);
                    if (atomicCAS(&s->busy, 0, 1) == 0) {
                        __threadfence();
                        const volatile GState *vs = s;
                        ok = 1;
                        if (a.do_step && (vs->parked || (vs->winner != GMZ_WINNER_NONE && !a.restart))) ok = 0;
                        if (ok && a.do_step && (long long)atomicAdd(&p.ctl->moves_started, 1ull) >= a.total_tickets) ok = -1;
                        if (ok != 1) atomicExch(&s->busy, 0);
                    }
                }
            }
            ok = __shfl_sync(GMZ_FULL, ok, 0);
            t = __shfl_sync(GMZ_FULL, t, 0);
            g = (int)(t % (unsigned long long)p.G);
            if (ok == 1) { got = true; break; }
            if (ok < 0) { done = true; break; }
        }
        if (done) break;
        if (!got) {                          // nothing playable (everything parked): give up
            if (lane == 0) atomicAdd(&p.ctl->tickets_unserved, 1ull);
            break;
        }
        __threadfence();                    // acquire: everything the previous owner wrote is visible
        GState *s = p.gs + g;
        int2 *path = p.path + (size_t)g * (p.S + 2);    // descent path past depth 31 (rare)

        if (a.do_step && s->winner != GMZ_WINNER_NONE) {   // finished earlier, could not restart then
            game_deal(p, a.book, s, g, lane);
            __syncwarp();
        }
        WG &w = s_wg[wi];
        wg_load(p, g, lane, w);
        double value = 0.0; int action = -1;
        if (w.active) {
            wg_valid_bits<NC>(p, w, lane);
            u64 h_root;
            h_root = play_root<NC>(p, a, w, s->noise_ctr, noise_mixed, lane);
            if (MZ && lane == 0) p.nH[w.nbase] = h_root;         // root hidden state = hash of the root observation
            __syncwarp();
            int ev = 0;
            while (w.sim_count < p.S) {
                int lp, la;
                DescSmem &ds = s_desc[wi];
                const int depth = descend<NC, MZ, F32>(p, w, path, ds, s_sel[wi], warp_slot, lane, lp, la);
                PathReg pr;
                path_load<MZ>(p, w, ds, depth, pr, lane);
                prefetch_parent_rows<NC>(p, w, lp, lane);
                u64 own = 0, opp = 0;
                if (!MZ) replay_path(p, w, path, ds, depth, la, lane, own, opp);
                // AlphaZero mode: evaluate the replayed board (mcts.py:251-253).  MuZero mode: the learned
                // dynamics, here E0's recurrent half on the parent's hidden state (mcts.py:336-343).
                const u64 h = MZ ? e0_child_hidden(p.nH[w.nbase + (size_t)lp], la)
                                 : e0_hash_planes(a.e0.h0, own, opp, p.NW, la, lane);
                const int reps = MZ ? w.n_surv : 1;            // MuZero: len(selected) identical selections -> that many backups
                const int nn = w.num_nodes;
                {   // evaluate + leaf.expand fused: logits go straight into the new node's row
                    float lg[4 * NC];
                    const unsigned xb = e0_seed32(h) + (unsigned)(4 * lane + 1) * E0_GOLD32;   // seed + (a + 1) * G for this lane's first action
#pragma unroll
                    for (int i = 0; i < 4 * NC; ++i) {                       // (power-of-two divisor / dense: one exact multiply -- the entry points reject other divisors)
                        const int off = 128 * (i >> 2) + (i & 3);
                        const unsigned x = e0_action_hash(xb + (unsigned)off * E0_GOLD32);
                        lg[i] = __fmul_rn((float)((int)(x >> a.e0.lshift) - a.e0.lbias), a.e0.lmul);   // (padding past A: never read, the valid mask covers it)
                    }
                    node_write_row<NC>(p, w, nn, lg, lane);
                    node_init_hdr<NC>(p, w, nn, lg, lane);
                }
                const int nmir = node_link<NC>(p, w, lp, la, nn, lane);
                if (MZ && lane == 0) p.nH[w.nbase + (size_t)nn] = h;
                if ((a.trace_a != nullptr || a.trace_d != nullptr) && lane == 0) {      // parity tests only
                    if (a.trace_a) a.trace_a[(size_t)g * p.S + ev] = la;
                    if (a.trace_d) a.trace_d[(size_t)g * p.S + ev] = depth;
                }
                wg_set(w.num_nodes, nn + 1); ++ev;
                __syncwarp();
                backup<MZ, F32>(p, w, path, pr, depth, nn, nmir, e0_value(h, a.e0.dense), MZ ? e0_reward(h, a.e0.dense) : 0.0, reps, lane);
                survivor_visit(w, depth, pr.node, nn, la, reps, lane);
                const int sc = w.sim_count + reps;
                wg_set(w.sim_count, sc);
                if (halving_ready(p, w, sc)) sequential_halving<MZ, F32>(p, w, lane);
            }
            wg_store_search(p, lane, w);
            __syncwarp();
        }
        // ---- decision phase
        double *pol = nullptr; int32_t *vis = nullptr;
        int slot = -1, tl = 0;
        if (a.do_step) {
            if (a.use_traj) {
                slot = s->traj_slot; tl = s->traj_len;
                if (tl == 0 && w.active) traj_open(a.traj, s, slot, g, w.to_move, w.last_move, lane);
                if (tl < a.traj.max_moves) pol = a.traj.policy + ((size_t)slot * a.traj.max_moves + tl) * (size_t)p.A;
            }
        } else {
            if (a.out_policy) pol = a.out_policy + (size_t)g * p.A;
            if (a.out_visits) vis = a.out_visits + (size_t)g * p.A;
        }
        finalize_root<NC, MZ, F32>(p, w, lane, pol, vis, s_nvis[wi], table, value, action);
        if (!a.do_step) {
            if (lane == 0) { if (a.out_value) a.out_value[g] = value; if (a.out_action) a.out_action[g] = action; }
        } else if (action < 0) {
            if (lane == 0) atomicAdd(&p.ctl->tickets_idle, 1ull);
        } else {
            const int wv = move_commit(p, a.traj, s, a.use_traj, slot, tl, value, action, lane);
            if (wv != GMZ_WINNER_NONE) game_finish(p, a.traj, a.book, s, g, a.use_traj, a.restart, slot, tl + 1, wv, lane);
        }
        __syncwarp();
        __threadfence();                    // release
        if (lane == 0) atomicExch(&s->busy, 0);
    }
}
