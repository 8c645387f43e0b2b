// gmz_match.cu -- matches between two engines (include/gmz.h, "matches"): the per-ply glue that deals openings into
// the slots of both engines, draws each game's Gumbel noise from its (opening, ply), plays both engines' decisions and
// hands every game over to the other engine, with no host read inside a ply.  One warp per slot g, which owns slot g of
// both engines, so the hand-over is a register swap inside the warp.
#include <stdint.h>
#include <string.h>

#include "gmz_internal.h"
#include "gmz_engine.cuh"
#include "gmz_play.cuh"

#define MATCH_WARPS 4
#define MATCH_THREADS (32 * MATCH_WARPS)

// Slot g of engine q (0 = a, 1 = b) takes the next opening of q's queue (ticket 2o + q: q's player moves first, with
// the opening's side to move), or the inactive full-board root once the queue is empty.
__device__ __forceinline__ void slot_deal(const Params &p, const gmz_match &m, int q, int g, int lane)
{
    int o = 0;
    if (lane == 0) o = atomicAdd(m.cursor + q, 1);
    o = __shfl_sync(GMZ_FULL, o, 0);
    int32_t *tk = m.slot_ticket + (size_t)q * p.G + g, *ply = m.slot_ply + (size_t)q * p.G + g;
    if (o >= m.n_openings) {
        root_load(p, g, lane, nullptr, 1, -1, 0);
        if (lane == 0) { *tk = -1; *ply = 0; }
        return;
    }
    const int t = 2 * o + q, pl = m.open_players[o];
    root_load(p, g, lane, m.open_boards + (size_t)o * p.A, pl, m.open_last[o], m.open_mc[o]);
    for (int a = lane; a < p.A; a += 32) m.moves[(size_t)t * p.A + a] = -1;
    if (lane == 0) {
        int32_t *r = m.results + (size_t)t * 4;
        r[0] = GMZ_WINNER_NONE; r[1] = 0; r[2] = q; r[3] = q == 0 ? pl : -pl;
        *tk = t; *ply = 0;
    }
}

__global__ void __launch_bounds__(MATCH_THREADS) k_match_start(Params pa, Params pb, gmz_match m)
{
    const int lane = threadIdx.x & 31, g = blockIdx.x * MATCH_WARPS + (threadIdx.x >> 5);
    if (g >= pa.G) return;
    slot_deal(pa, m, 0, g, lane);
    slot_deal(pb, m, 1, g, lane);
}

// Noise of ply k of opening o: counters (o*A + k)*A + a of the match seed, gmz_fill_gumbel's generator.
__global__ void __launch_bounds__(MATCH_THREADS)
k_match_noise(int G, int A, gmz_match m, u64 seed_mixed, double *gum_a, double *gum_b)
{
    const int lane = threadIdx.x & 31, g = blockIdx.x * MATCH_WARPS + (threadIdx.x >> 5);
    if (g >= G) return;
    for (int q = 0; q < 2; ++q) {
        const int t = m.slot_ticket[(size_t)q * G + g];
        double *out = (q ? gum_b : gum_a) + (size_t)g * A;
        const u64 base = t < 0 ? 0 : ((u64)(t >> 1) * (u64)A + (u64)m.slot_ply[(size_t)q * G + g]) * (u64)A;
        for (int a = lane; a < A; a += 32) out[a] = t < 0 ? 0.0 : gumbel_at(seed_mixed, base + (u64)a);
    }
}

__global__ void __launch_bounds__(MATCH_THREADS)
k_match_step(Params pa, Params pb, gmz_match m, const int32_t *act_a, const int32_t *act_b)
{
    const int lane = threadIdx.x & 31, g = blockIdx.x * MATCH_WARPS + (threadIdx.x >> 5);
    const int G = pa.G, A = pa.A;
    if (g >= G) return;
    int tk[2], ply[2];
    bool live[2];
    for (int q = 0; q < 2; ++q) {
        const Params &p = q ? pb : pa;
        tk[q] = m.slot_ticket[(size_t)q * G + g];
        ply[q] = m.slot_ply[(size_t)q * G + g];
        live[q] = false;
        if (tk[q] < 0) continue;
        const int a = (q ? act_b : act_a)[g];
        const bool ok = a >= 0 && a < A;
        const int wv = ok ? game_do_move(p, p.gs + g, a, lane) : GMZ_WINNER_NONE;
        if (lane == 0 && ok && ply[q] < A) m.moves[(size_t)tk[q] * A + ply[q]] = a;
        if (ok) ply[q] += 1;
        if (ok && wv == GMZ_WINNER_NONE) { live[q] = true; continue; }
        if (lane == 0) {
            int32_t *r = m.results + (size_t)tk[q] * 4;
            r[0] = wv; r[1] = ply[q];
            atomicAdd(m.finished, 1);
        }
    }
    __syncwarp();
    // read both games as they stand after the moves, then hand each to the other engine's slot g
    u64 P[2] = {0, 0}, M[2] = {0, 0}, V[2] = {0, 0};
    int tm[2] = {0, 0}, lm[2] = {0, 0}, mc[2] = {0, 0};
    for (int q = 0; q < 2; ++q) {
        const GState *s = (q ? pb : pa).gs + g;
        if (lane < GMZ_WORDS) { P[q] = s->p1[lane]; M[q] = s->m1[lane]; V[q] = s->valid[lane]; }
        tm[q] = s->to_move; lm[q] = s->last_move; mc[q] = s->move_count;
    }
    __syncwarp();
    for (int q = 0; q < 2; ++q) {           // q = the receiving engine, 1 - q = where its incoming game comes from
        const Params &p = q ? pb : pa;
        const int src = 1 - q;
        if (!live[src]) { slot_deal(p, m, q, g, lane); continue; }
        root_write(p.gs + g, lane, P[src], M[src], V[src], tm[src], lm[src], mc[src],
                   __any_sync(GMZ_FULL, lane < GMZ_WORDS && V[src] != 0ull));
        if (lane == 0) { m.slot_ticket[(size_t)q * G + g] = tk[src]; m.slot_ply[(size_t)q * G + g] = ply[src]; }
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static int check_match(const char *name, gmz_engine *a, gmz_engine *b, const gmz_match *m)
{
    if (!gmz_engine_live(a) || !gmz_engine_live(b)) return gmz_fail("%s: invalid or destroyed engine handle", name);
    if (a == b) return gmz_fail("%s: the two players need two different engines", name);
    if (a->p.G != b->p.G) return gmz_fail("%s: the engines hold different numbers of games (num_games)", name);
    if (a->p.N != b->p.N) return gmz_fail("%s: the engines have different board sizes", name);
    if (a->p.n_in_row != b->p.n_in_row) return gmz_fail("%s: the engines have different n_in_row", name);
    if (a->device != b->device) return gmz_fail("%s: the engines live on different devices", name);
    if (!m) return gmz_fail("%s: null match", name);
    if (m->n_openings < 1) return gmz_fail("%s: a match needs at least one opening", name);
    if (!m->open_boards || !m->open_players || !m->open_last || !m->open_mc || !m->cursor || !m->slot_ticket ||
        !m->slot_ply || !m->results || !m->moves || !m->finished)
        return gmz_fail("%s: null buffer in the match", name);
    return 0;
}
#define MATCH_GRID(e) dim3(((e)->p.G + MATCH_WARPS - 1) / MATCH_WARPS), dim3(MATCH_THREADS)

extern "C" int gmz_match_start(gmz_engine *a, gmz_engine *b, const gmz_match *m, gmz_stream stream)
{
    if (check_match("gmz_match_start", a, b, m)) return 1;
    cudaError_t err = cudaMemsetAsync(m->cursor, 0, 2 * sizeof(int32_t), (cudaStream_t)stream);
    if (err == cudaSuccess) err = cudaMemsetAsync(m->finished, 0, sizeof(int32_t), (cudaStream_t)stream);
    if (err != cudaSuccess) return gmz_fail("gmz_match_start: cudaMemsetAsync: %s", cudaGetErrorString(err));
    k_match_start<<<MATCH_GRID(a), 0, (cudaStream_t)stream>>>(a->p, b->p, *m);
    return gmz_check_launch("k_match_start");
}

extern "C" int gmz_match_noise(gmz_engine *a, gmz_engine *b, const gmz_match *m, uint64_t seed, double *gumbel_a,
                               double *gumbel_b, gmz_stream stream)
{
    if (check_match("gmz_match_noise", a, b, m)) return 1;
    if (!gumbel_a || !gumbel_b) return gmz_fail("gmz_match_noise: null argument");
    k_match_noise<<<MATCH_GRID(a), 0, (cudaStream_t)stream>>>(a->p.G, a->p.A, *m, mix64((u64)seed ^ E0_GOLD), gumbel_a,
                                                              gumbel_b);
    return gmz_check_launch("k_match_noise");
}

extern "C" int gmz_match_step(gmz_engine *a, gmz_engine *b, const gmz_match *m, const int32_t *action_a,
                              const int32_t *action_b, gmz_stream stream)
{
    if (check_match("gmz_match_step", a, b, m)) return 1;
    if (!action_a || !action_b) return gmz_fail("gmz_match_step: null argument");
    k_match_step<<<MATCH_GRID(a), 0, (cudaStream_t)stream>>>(a->p, b->p, *m, action_a, action_b);
    return gmz_check_launch("k_match_step");
}
