// gmz_inspect.cu -- search inspection (include/gmz.h, "search inspection"): copy each game's search tree, its root's
// Gumbel top-k with the halving round that eliminated each entry, and the per-game search state out of the engine's
// workspace into caller buffers.  It only reads the workspace and only copies stored values: nothing here computes a
// search quantity, so an exported tree is bit for bit what the search kernels left behind.
#include <math.h>
#include <stdint.h>

#include "gmz_internal.h"
#include "gmz_engine.cuh"

// Round of the sequential halving (mcts.py:183-185) that dropped top-k position i.  sequential_halving permutes only
// the first n_surv entries, so an entry stays where the halving that removed it left it: after round r the survivors are
// positions 0 .. min(m_of_phase[r], n_init) - 1, and position i >= n_surv left in the first round whose cut is <= i.
__device__ __forceinline__ int eliminated_in(const Params &p, int i, int n_surv, int n_init, int phase)
{
    if (i < n_surv) return phase;
    const int last = min(phase, p.n_phases);
    for (int r = 1; r <= last; ++r)
        if (i >= min(p.m_of_phase[r], n_init)) return r;
    return -1;
}

// One warp per game.  A game's tree is current iff sim_count > 0 (root_load / game_do_move / game_reset set it to 0),
// otherwise it exports as empty.  Shared memory: the parent and the action of every node, short [S] each.
__global__ void __launch_bounds__(32) k_tree_export(const __grid_constant__ Params p, const __grid_constant__ gmz_tree_out o)
{
    extern __shared__ short s_tree[];
    short *par = s_tree, *act = s_tree + p.S;
    const int lane = threadIdx.x, g = blockIdx.x;
    const GState *s = p.gs + g;
    const int sim = s->sim_count;
    const int n = sim > 0 ? s->num_nodes : 0;
    const int phase = n ? s->phase : 0, n_surv = n ? s->n_surv : 0, n_init = n ? s->n_init : 0;
    const size_t nb = (size_t)g * (size_t)p.S;

    if (lane == 0) {
        if (o.num_nodes) o.num_nodes[g] = n;
        if (o.sim_count) o.sim_count[g] = sim;
        if (o.root) { int32_t *r = o.root + (size_t)g * 3; r[0] = s->to_move; r[1] = s->last_move; r[2] = s->move_count; }
        if (o.minmax) { o.minmax[2 * (size_t)g] = n ? s->mm_min : INFINITY; o.minmax[2 * (size_t)g + 1] = n ? s->mm_max : -INFINITY; }
        if (o.halving) { int32_t *h = o.halving + (size_t)g * 3; h[0] = phase; h[1] = n_surv; h[2] = n_init; }
    }
    for (int i = lane; i < p.K; i += 32) {
        const bool in = i < n_init;
        const size_t t = (size_t)g * p.K + i;
        if (o.topk_action) o.topk_action[t] = in ? s->surv_act[i] : -1;
        if (o.topk_gumbel) o.topk_gumbel[t] = in ? s->surv_g[i] : 0.0;
        if (o.topk_logit) o.topk_logit[t] = in ? s->surv_logit[i] : 0.0f;
        if (o.topk_round) o.topk_round[t] = in ? eliminated_in(p, i, n_surv, n_init, phase) : -1;
    }
    if (o.root_logits) {
        const float *lrow = p.logits + nb * (size_t)p.AP;
        for (int a = lane; a < p.A; a += 32) o.root_logits[(size_t)g * p.A + a] = n ? lrow[a] : __int_as_float(0x7fc00000);
    }

    // node statistics as stored; entries past num_nodes read -1 / 0
    for (int k = lane; k < p.S; k += 32) {
        const bool in = k < n;
        if (o.visits) o.visits[nb + k] = in ? p.nN[nb + k] : -1;
        if (o.value_sum) o.value_sum[nb + k] = in ? p.nW[nb + k] : 0.0;
        if (o.reward) o.reward[nb + k] = (in && p.nR) ? p.nR[nb + k] : 0.0;
        if (o.prior_logit && (k == 0 || !in)) o.prior_logit[nb + k] = in ? __int_as_float(0x7fc00000) : 0.0f;   // root: no edge
        if (in) { par[k] = -1; act[k] = -1; }
    }
    if (n == 0) {
        for (int k = lane; k < p.S; k += 32) {
            if (o.parent) o.parent[nb + k] = -1;
            if (o.action) o.action[nb + k] = -1;
            if (o.depth) o.depth[nb + k] = -1;
        }
        return;
    }
    __syncwarp();
    // Structure from the child rows (Params::child is authoritative; the block slots mirror only the first 31 children):
    // row k names every child of node k.  Lane l reads actions 128 j + 4 l .. + 3 of each row, one short4 per chunk.
    const int nc = p.AP >> 7;
#pragma unroll 4
    for (int k = 0; k < n; ++k) {
        const short *crow = p.child + (nb + k) * (size_t)p.AP;
        const float *lrow = p.logits + (nb + k) * (size_t)p.AP;
        for (int j = 0; j < nc; ++j) {
            const short4 c4 = __ldg(reinterpret_cast<const short4 *>(crow + 128 * j + 4 * lane));
            const short cs[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int c = cs[t], a = 128 * j + 4 * lane + t;
                if (c > 0 && c < n) {
                    par[c] = (short)k; act[c] = (short)a;
                    if (o.prior_logit) o.prior_logit[nb + c] = __ldg(lrow + a);
                }
            }
        }
    }
    __syncwarp();
    for (int k = lane; k < p.S; k += 32) {
        if (o.parent) o.parent[nb + k] = k < n ? par[k] : -1;
        if (o.action) o.action[nb + k] = k < n ? act[k] : -1;
    }
    __syncwarp();
    // depth: one in-order pass, in place over the parents (a parent's id is below its child's)
    if (lane == 0) {
        par[0] = 0;
        for (int k = 1; k < n; ++k) {
            const int pk = par[k];
            par[k] = pk >= 0 ? (short)(par[pk] + 1) : (short)-1;
        }
    }
    __syncwarp();
    if (o.depth)
        for (int k = lane; k < p.S; k += 32) o.depth[nb + k] = k < n ? par[k] : -1;
}

extern "C" int gmz_tree_export(gmz_engine *e, const gmz_tree_out *out, gmz_stream stream)
{
    if (!gmz_engine_live(e)) return gmz_fail("%s: invalid or destroyed engine handle", "gmz_tree_export");
    if (!out) return gmz_fail("gmz_tree_export: null out");
    const size_t smem = (size_t)4 * e->p.S;
    if (smem > 48 * 1024) {
        const cudaError_t err = cudaFuncSetAttribute(k_tree_export, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err != cudaSuccess) return gmz_fail("gmz_tree_export: cudaFuncSetAttribute: %s", cudaGetErrorString(err));
    }
    k_tree_export<<<e->p.G, 32, smem, (cudaStream_t)stream>>>(e->p, *out);
    return gmz_check_launch("k_tree_export");
}
