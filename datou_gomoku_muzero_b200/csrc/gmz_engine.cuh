// gmz_engine.cuh -- what gmz_engine.cu shares with the other translation units that drive an engine's roots.
#pragma once
#include "gmz_internal.h"

// Non-zero if `e` is a live handle (created and not yet destroyed); defined in gmz_engine.cu.
int gmz_engine_live(const gmz_engine *e);

// A new root for the GState: the bitboards (lane w < GMZ_WORDS holds word w of P, M and the valid cells V) and every
// field a new root resets.  The opening label is left to the callers that deal games.
__device__ __forceinline__ void root_write(GState *s, int lane, u64 P, u64 M, u64 V, int to_move, int last_move, int move_count,
                                           bool active)
{
    if (lane < GMZ_WORDS) { s->p1[lane] = P; s->m1[lane] = M; s->valid[lane] = V; }
    if (lane == 0) {
        s->to_move = to_move; s->last_move = last_move; s->move_count = move_count; s->active = active;
        s->sim_count = 0; s->num_nodes = 0; s->leaf_depth = 0; s->n_surv = 0; s->n_init = 0;
        s->winner = GMZ_WINNER_NONE;
    }
}

// board int8 [A] -> game g's bitboards; one warp per game, ballots pack 32 cells at a time.  b == NULL: a full board
// of +1 stones (an inactive padding root).
__device__ __forceinline__ void root_load(const Params &p, int g, int lane, const int8_t *b, int player, int last_move,
                                          int move_count)
{
    u64 P = 0, M = 0, V = 0;
    int nvalid = 0;
    for (int w = 0; w < GMZ_WORDS; ++w) {
        u64 pw = 0, mw = 0, vw = 0;
        for (int h = 0; h < 2; ++h) {
            const int a = 64 * w + 32 * h + lane;
            const int c = a < p.A ? (b ? (int)b[a] : 1) : 2;
            pw |= (u64)__ballot_sync(GMZ_FULL, c == 1) << (32 * h);
            mw |= (u64)__ballot_sync(GMZ_FULL, c == -1) << (32 * h);
            vw |= (u64)__ballot_sync(GMZ_FULL, c == 0) << (32 * h);
        }
        nvalid += __popcll(vw);
        if (lane == w) { P = pw; M = mw; V = vw; }
    }
    GState *s = p.gs + g;
    root_write(s, lane, P, M, V, player >= 0 ? 1 : -1, last_move, move_count, nvalid > 0);
    if (lane == 0) s->opening = 0;
}

// GomokuGame.reset() on a GState (game.py:8-11).
__device__ __forceinline__ void game_reset(const Params &p, GState *s, int lane)
{
    u64 v = 0;
    const int lo = 64 * lane;
    if (lo < p.A) v = (p.A - lo >= 64) ? ~0ull : ((1ull << (p.A - lo)) - 1ull);
    root_write(s, lane, 0ull, 0ull, v, 1, -1, 0, true);
}

// A new self-play game for game g: its k-th deal since the book was bound (k = s->deals) takes opening (k*G + g) mod O,
// so the games of an index depend on g and k only, not on which warp or launch deals them.  Without a book: the empty
// board, labelled "none".  Every lane takes part (root_load ballots).  Out of line: in the play kernel a deal is rare next
// to the simulations, and its code stays out of the simulation loop's instruction stream and registers.  Callers pass
// __grid_constant__ kernel parameters: a by-value Params would be copied to a 360-byte stack frame for every call.
static __device__ __noinline__ void game_deal(const Params &p, const BookDev &b, GState *s, int g, int lane)
{
    const unsigned k = s->deals;
    int label = 0;
    if (b.n > 0) {
        const int o = (int)(((u64)k * (u64)p.G + (u64)g) % (u64)b.n);
        root_load(p, g, lane, b.boards + (size_t)o * p.A, b.players[o], b.last_moves[o], b.move_counts[o]);
        label = o + 1;
    } else game_reset(p, s, lane);
    __syncwarp();
    if (lane == 0) { s->traj_len = 0; s->parked = 0; s->deals = k + 1; s->opening = label; }
}
