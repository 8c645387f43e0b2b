// gmz_engine.cuh -- what gmz_engine.cu shares with the other translation units that drive an engine's roots.
#pragma once
#include "gmz_internal.h"

// Non-zero if `e` is a live handle (created and not yet destroyed); defined in gmz_engine.cu.
int gmz_engine_live(const gmz_engine *e);

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
    if (lane < GMZ_WORDS) { s->p1[lane] = P; s->m1[lane] = M; s->valid[lane] = V; }
    if (lane == 0) {
        s->to_move = player >= 0 ? 1 : -1;
        s->last_move = last_move;
        s->move_count = move_count;
        s->active = nvalid > 0;
        s->sim_count = 0; s->num_nodes = 0; s->leaf_depth = 0; s->n_surv = 0; s->n_init = 0;
        s->winner = GMZ_WINNER_NONE; s->opening = 0;
    }
}

// GomokuGame.reset() on a GState (game.py:8-11).
__device__ __forceinline__ void game_reset(const Params &p, GState *s, int lane)
{
    if (lane < GMZ_WORDS) {
        u64 v = 0;
        const int lo = 64 * lane;
        if (lo < p.A) v = (p.A - lo >= 64) ? ~0ull : ((1ull << (p.A - lo)) - 1ull);
        s->p1[lane] = 0; s->m1[lane] = 0; s->valid[lane] = v;
    }
    if (lane == 0) {
        s->to_move = 1; s->last_move = -1; s->move_count = 0; s->active = 1;
        s->sim_count = 0; s->num_nodes = 0; s->leaf_depth = 0; s->n_surv = 0; s->n_init = 0;
        s->winner = GMZ_WINNER_NONE; s->traj_len = 0; s->parked = 0;
    }
}

// A new self-play game for game g: its k-th deal since the book was bound (k = s->deals) takes opening (k*G + g) mod O,
// so the games of an index depend on g and k only, not on which warp or launch deals them.  Without a book: the empty
// board, labelled "none".  Every lane takes part (root_load ballots).
__device__ __forceinline__ void game_deal(const Params &p, const BookDev &b, GState *s, int g, int lane)
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
