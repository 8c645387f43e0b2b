// gmz_tree.cuh -- warp-cooperative device functions of the Gumbel-MCTS simulation step.
// Each function restates one piece of the reference search (file:line cited) for a warp that
// owns one game; see gmz_common.cuh for the lane <-> action mapping.
#pragma once
#include "gmz_common.cuh"

// View of the game a warp is searching, IN SHARED MEMORY (one per warp).  "U" = warp-uniform field: every lane
// stores the same value; "L" = one element per lane.  It used to be a register struct; at 72 registers most of it
// was spilled, and a third of those local-memory reloads missed the L1 (67 MB of stack for 4096 warps) -- in
// shared memory the same accesses cost an LDS.  The select loop keeps what it needs (nbase, mn, rden) in registers.
struct __align__(16) WG {
    double mm_min, mm_max; // U  MinMaxStats
    size_t nbase;          // U  g * S : index of this game's node 0 in the per-node arrays
    int g;                 // U
    int sim_count, num_nodes, phase, next_thr, n_surv, n_init, to_move, last_move, active;  // U
    u64 rP[GMZ_WORDS], rM[GMZ_WORDS];   // the root's +1 / -1 bitboards (word w at index w): every replay starts from them
    unsigned vb[32];       // L  valid bits of this lane's actions (bit 4*j + t)
    int s_act[32], s_child[32], s_n[32];  // L  lane i < n_init: survivor i
    // (the survivors' gumbel noise / root logits and the valid bitboard stay in GState: they are only
    //  needed at the <= 5 halvings and at the decision)
};
// A uniform field must not be read by one lane after another lane already stored its update: read (before the
// call), wait for every lane, store, make the store visible.
template <typename T>
__device__ __forceinline__ void wg_set(T &field, T value) { __syncwarp(); field = value; __syncwarp(); }

__device__ __forceinline__ void wg_load(const Params &p, int g, int lane, WG &w)
{
    const GState *s = p.gs + g;
    w.g = g; w.nbase = (size_t)g * (size_t)p.S;
    w.mm_min = s->mm_min; w.mm_max = s->mm_max;
    w.sim_count = s->sim_count; w.num_nodes = s->num_nodes; w.phase = s->phase; w.next_thr = s->next_thr;
    w.n_surv = s->n_surv; w.n_init = s->n_init; w.to_move = s->to_move; w.last_move = s->last_move;
    w.active = s->active;
    w.s_act[lane] = s->surv_act[lane]; w.s_child[lane] = s->surv_child[lane]; w.s_n[lane] = s->surv_n[lane];
    if (lane < GMZ_WORDS) { w.rP[lane] = s->p1[lane]; w.rM[lane] = s->m1[lane]; }
    __syncwarp();
}
template <int NC>
__device__ __forceinline__ void wg_valid_bits(const Params &p, WG &w, int lane)
{
    const u64 V = lane < GMZ_WORDS ? p.gs[w.g].valid[lane] : 0ull;
    unsigned vb = 0;
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        u64 word = shfl_u64(V, 2 * j + (lane >> 4));
        vb |= (unsigned)((word >> ((lane & 15) * 4)) & 0xFull) << (4 * j);
    }
    w.vb[lane] = vb;
}
__device__ __forceinline__ void wg_store_search(const Params &p, int lane, const WG &w)
{
    GState *s = p.gs + w.g;
    if (lane == 0) {
        s->mm_min = w.mm_min; s->mm_max = w.mm_max;
        s->sim_count = w.sim_count; s->num_nodes = w.num_nodes; s->phase = w.phase; s->next_thr = w.next_thr;
        s->n_surv = w.n_surv; s->n_init = w.n_init;
    }
    s->surv_act[lane] = (short)w.s_act[lane]; s->surv_child[lane] = (short)w.s_child[lane]; s->surv_n[lane] = w.s_n[lane];
}

// GomokuGame.do_move on the lane-distributed bitboards (game.py:20-23): the stone OVERWRITES
// whatever is on the cell (the reference's in-tree replay has no legality check).
__device__ __forceinline__ void bb_do_move(u64 &P, u64 &M, int colour, int a, int lane)
{
    const u64 b = lane == (a >> 6) ? 1ull << (a & 63) : 0ull;     // branch-free: every lane runs the same few LOP3
    const u64 bp = colour > 0 ? b : 0ull, bm = b ^ bp;
    P = (P | bp) & ~bm;
    M = (M | bm) & ~bp;
}

// Per-warp shared scratch of the simulation in flight: the descent path with the action taken into each node and
// the statistics read on the way down (handed to the backup).  Kept in shared memory, not registers: the select
// needs ~30 temporaries per level, and anything live across it in registers is spilled and reloaded every level.
struct PathEntry { int node, mir, n, act; double W, R; };      // 32 bytes, see PathReg; act = the move that led here
struct DescSmem {
    PathEntry path[32];
};

// utils.MinMaxStats.normalize (utils.py:16-25) with the range test hoisted.
__device__ __forceinline__ double mm_norm(double q, bool rng, double mn, double denom)
{
    if (!rng) return 0.0;
    double n = __ddiv_rn(__dsub_rn(q, mn), denom);
    n = n < 1.0 ? n : 1.0;
    return n > 0.0 ? n : 0.0;
}

// Arithmetic mode.  F32 = false: the evaluator handed Python floats, everything is float64 (the upstream
// test mock).  F32 = true: it handed np.float32 scalars (the reference's inference server, workers.py:355,368);
// under NumPy >= 2 value_sum, the backed-up value, get_value / get_qsa and the MinMaxStats bounds are then
// float32 (one float32 rounding per operation, DISCOUNT and VALUE_MINMAX_DELTA rounded to float32 first), while
// normalize()'s numerator / division, sigma, the softmax and the scores stay float64 (SURVEY.md App. A.7;
// pinned by the vdtype = 1 goldens of tests/golden/).  Values are stored widened in the
// same double arrays.
// Node.get_qsa for a visited child (mcts.py:35-38): child.reward + DISCOUNT * (value_sum / visit_count)
template <bool F32>
__device__ __forceinline__ double q_of(const Params &p, double W, int n, double R)
{
    if (F32) return (double)__fadd_rn((float)R, __fmul_rn(p.discf, __fdiv_rn((float)W, (float)n)));
    return __dadd_rn(R, __dmul_rn(p.discount, __ddiv_rn(W, (double)n)));
}
// denominator of MinMaxStats.normalize (utils.py:19): maximum - minimum + minmax_delta
template <bool F32>
__device__ __forceinline__ double mm_denom(const Params &p, double mn, double mx)
{
    if (F32) return (double)__fadd_rn(__fsub_rn((float)mx, (float)mn), p.deltaf);
    return __dadd_rn(__dsub_rn(mx, mn), p.delta);
}

// Loaded view of one expanded node's row: logits, child ids, child visit counts and q values.
template <int NC>
struct Row {
    float lg[4 * NC];
    short ch[4 * NC];
    int n[4 * NC];
    double q[4 * NC];
    int maxN, sumN;
};

// Node.get_qsa for every action of `node` (mcts.py:35-38) + max / sum of child visits
// (mcts.py:144-147, 110).  Only visited children (child id >= 0) touch memory beyond the row.
template <int NC, bool MZ, bool F32>
__device__ __forceinline__ void row_load(const Params &p, const WG &w, int node, int lane, Row<NC> &r)
{
    const size_t ni = w.nbase + (size_t)node;
    const float *lrow = p.logits + ni * (size_t)p.AP;
    const short *crow = p.child + ni * (size_t)p.AP;
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        const float4 t = *reinterpret_cast<const float4 *>(lrow + 128 * j + 4 * lane);
        const short4 c = *reinterpret_cast<const short4 *>(crow + 128 * j + 4 * lane);
        r.lg[4 * j + 0] = t.x; r.lg[4 * j + 1] = t.y; r.lg[4 * j + 2] = t.z; r.lg[4 * j + 3] = t.w;
        r.ch[4 * j + 0] = c.x; r.ch[4 * j + 1] = c.y; r.ch[4 * j + 2] = c.z; r.ch[4 * j + 3] = c.w;
    }
    int lmax = 0, lsum = 0;
#pragma unroll
    for (int i = 0; i < 4 * NC; ++i) {
        r.n[i] = 0; r.q[i] = 0.0;
        if (r.ch[i] >= 0) {
            const size_t ci = w.nbase + (size_t)r.ch[i];
            const int nn = p.nN[ci];
            r.q[i] = q_of<F32>(p, p.nW[ci], nn, MZ ? p.nR[ci] : 0.0);
            r.n[i] = nn; lmax = max(lmax, nn); lsum += nn;
        }
    }
    r.maxN = __reduce_max_sync(GMZ_FULL, lmax);
    r.sumN = __reduce_add_sync(GMZ_FULL, lsum);
}

// softmax over the root-valid actions of logits + sigma(q) (mcts.py:141-156): on return
// x[i] = exp(logit + sigma - max) (0 for invalid actions) and the return value is 1/sum.
template <int NC, bool F32>
__device__ __forceinline__ double row_softmax(const Params &p, const WG &w, const Row<NC> &r, double *x, int lane)
{
    const unsigned wvb = w.vb[lane];
    const double scale = __dmul_rn(__dadd_rn(p.c_visit, (double)r.maxN), p.c_scale);
    const bool rng = w.mm_max > w.mm_min;
    const double denom = mm_denom<F32>(p, w.mm_min, w.mm_max);
    const double sig0 = __dmul_rn(scale, mm_norm(0.0, rng, w.mm_min, denom));   // unvisited: q = 0.0
    double lmx = -INFINITY;
#pragma unroll
    for (int i = 0; i < 4 * NC; ++i) {
        if ((wvb >> i) & 1u) {
            const double sig = r.ch[i] >= 0 ? __dmul_rn(scale, mm_norm(r.q[i], rng, w.mm_min, denom)) : sig0;
            x[i] = __dadd_rn((double)r.lg[i], sig);
            lmx = dmax2(lmx, x[i]);
        } else x[i] = -INFINITY;
    }
    const double mx = warp_max_f64(lmx);
    double ls = 0.0;
#pragma unroll
    for (int i = 0; i < 4 * NC; ++i) {
        x[i] = ((wvb >> i) & 1u) ? exp(__dsub_rn(x[i], mx)) : 0.0;
        ls = __dadd_rn(ls, x[i]);
    }
    const double sum = warp_sum_f64(ls);
    return __ddiv_rn(1.0, sum);
}

// Per-warp scratch of the EXACT select (select_interior_exact / _big; the certified path below needs no
// shared memory).  Nodes almost always have <= 32 visited children: then child k is handed to lane k through
// 256 bytes of shared memory and scored in registers.  The rare bigger node takes select_interior_big,
// which loops over this warp's slice of a global overflow area (Params::sel_overflow).
// Shared memory is kept small on purpose: it is carved out of the same 228 KB as the L1 cache
// that serves the node-header gathers.
#ifndef GMZ_EXP_UNROLL
#define GMZ_EXP_UNROLL 2
#endif
constexpr int kExpUnroll = GMZ_EXP_UNROLL;
struct SelSmem {
    double dx[256];                // dense pass: element i of lane l at [32*i + l] (NC <= 2; NC = 3 keeps registers)
    int key[32];                   // visited child k -> (action << 16) | child node id   (<= 32 children)
    float lg[32];                  // logit of that action
};
// Working pointers for one select call (shared or global, chosen per node).
struct SelPtr { int *key; float *lg; int *n; double *x; };
template <int NC>
__device__ __forceinline__ SelPtr sel_global(const Params &p, int warp_slot)
{   // layout per warp: x[128*NC] doubles, then key / lg / n [128*NC] each
    char *base = p.sel_overflow + (size_t)warp_slot * (size_t)(128 * NC * 20);
    SelPtr s;
    s.x = reinterpret_cast<double *>(base);
    s.key = reinterpret_cast<int *>(base + 128 * NC * 8);
    s.lg = reinterpret_cast<float *>(base + 128 * NC * 12);
    s.n = reinterpret_cast<int *>(base + 128 * NC * 16);
    return s;
}

// What the out-of-line exact select needs of the game, passed BY VALUE: a reference to the caller's WG
// would pin the whole register-resident game view in local memory.
struct SelCtx { size_t nbase; double mm_min, mm_max; unsigned vb; };
__device__ __forceinline__ SelCtx sel_ctx(const WG &w, int lane) { SelCtx c; c.nbase = w.nbase; c.mm_min = w.mm_min; c.mm_max = w.mm_max; c.vb = w.vb[lane]; return c; }
__device__ __forceinline__ int sel_pack(int action, int child) { return (action << 16) | (child & 0xffff); }
__device__ __forceinline__ void sel_unpack(int packed, int &action, int &child)
{
    action = packed >> 16;
    child = (packed & 0xffff) == 0xffff ? -1 : (packed & 0xffff);
}

// The exact _select_action at an interior node (mcts.py:106-117):
// argmax_a  softmax(logits + sigma)[a] - N(a) / (1 + sum_b N(b))   over the ROOT-valid actions.
// Most of a node's A children are unvisited (q = 0, N = 0, same sigma): those are scored in a
// branch-free dense pass from the row alone.  The few visited children are compacted into
// `sc` (one per lane) and scored in a sparse pass that gathers their N / W.
template <int NC, bool MZ, bool F32>
__device__ __noinline__ int select_interior_big(const Params &p, const SelCtx w, int node, int lane, SelSmem &sm, int warp_slot)
{
    int action, child;
    constexpr int E = 4 * NC;
    const size_t ni = w.nbase + (size_t)node;
    const float *lrow = p.logits + ni * (size_t)p.AP;
    const short *crow = p.child + ni * (size_t)p.AP;
    float lg[E]; short ch[E];
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        const float4 t = *reinterpret_cast<const float4 *>(lrow + 128 * j + 4 * lane);
        const short4 c = *reinterpret_cast<const short4 *>(crow + 128 * j + 4 * lane);
        lg[4 * j + 0] = t.x; lg[4 * j + 1] = t.y; lg[4 * j + 2] = t.z; lg[4 * j + 3] = t.w;
        ch[4 * j + 0] = c.x; ch[4 * j + 1] = c.y; ch[4 * j + 2] = c.z; ch[4 * j + 3] = c.w;
    }
    unsigned vm = 0;
#pragma unroll
    for (int i = 0; i < E; ++i) vm |= (ch[i] >= 0 ? 1u : 0u) << i;
    // compact the visited children: lane prefix over popc(vm)
    int total = 0;
    SelPtr sc = sel_global<NC>(p, warp_slot);
    if (__any_sync(GMZ_FULL, vm != 0)) {
        const int cnt = __popc(vm);
        int inc = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(GMZ_FULL, inc, o); if (lane >= o) inc += t; }
        total = __shfl_sync(GMZ_FULL, inc, 31);
        int pos = inc - cnt;
#pragma unroll
        for (int i = 0; i < E; ++i) {
            if ((vm >> i) & 1u) {
                sc.key[pos] = ((128 * (i >> 2) + 4 * lane + (i & 3)) << 16) | (int)ch[i];
                sc.lg[pos] = lg[i];
                ++pos;
            }
        }
        __syncwarp();
    }
    // sparse pass A: gather N and W of the visited children (one memory round trip)
    int lmax = 0, lsum = 0;
    for (int k = lane; k < total; k += 32) {
        const size_t ci = w.nbase + (size_t)(sc.key[k] & 0xffff);
        const int nn = p.nN[ci];
        sc.n[k] = nn; sc.x[k] = p.nW[ci];
        lmax = max(lmax, nn); lsum += nn;
    }
    int maxN = 0, sumN = 0;
    if (total > 0) { maxN = __reduce_max_sync(GMZ_FULL, lmax); sumN = __reduce_add_sync(GMZ_FULL, lsum); }
    const double scale = __dmul_rn(__dadd_rn(p.c_visit, (double)maxN), p.c_scale);
    const bool rng = w.mm_max > w.mm_min;
    const double denom = mm_denom<F32>(p, w.mm_min, w.mm_max);
    const double sig0 = __dmul_rn(scale, mm_norm(0.0, rng, w.mm_min, denom));   // unvisited: q = 0.0
    double lmx = -INFINITY;
    // sparse pass B: q -> sigma -> x
    for (int k = lane; k < total; k += 32) {
        const double rew = MZ ? p.nR[w.nbase + (size_t)(sc.key[k] & 0xffff)] : 0.0;
        const double q = q_of<F32>(p, sc.x[k], sc.n[k], rew);
        const double x = __dadd_rn((double)sc.lg[k], __dmul_rn(scale, mm_norm(q, rng, w.mm_min, denom)));
        sc.x[k] = x; lmx = dmax2(lmx, x);
    }
    const unsigned dv = w.vb & ~vm;      // valid and unvisited: the dense set
    double best = -INFINITY; int ba = 0x7fffffff, bc = -1;
    double inv;
    if (NC <= 2) {
        // Rolled loops over this lane's E elements, staged in shared memory: the kernel is bound by
        // instruction fetch (every warp is at a different PC of a ~30 KB loop), so the exp / score
        // bodies are kept small enough to be re-served by the L0 instruction cache.
        double *dx = sm.dx + lane;
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const double xi = __dadd_rn((double)lg[i], sig0);
            dx[32 * i] = xi;
            if ((dv >> i) & 1u) lmx = dmax2(lmx, xi);
        }
        const double mx = warp_max_f64(lmx);
        double ls = 0.0;
#pragma unroll kExpUnroll
        for (int i = 0; i < E; ++i) {
            double e = exp_nonpos(dmin2(__dsub_rn(dx[32 * i], mx), 0.0));
            e = ((dv >> i) & 1u) ? e : 0.0;
            dx[32 * i] = e;
            ls = __dadd_rn(ls, e);
        }
        for (int k = lane; k < total; k += 32) {
            const double e = exp_nonpos(__dsub_rn(sc.x[k], mx));
            sc.x[k] = e; ls = __dadd_rn(ls, e);
        }
        inv = __ddiv_rn(1.0, warp_sum_f64(ls));
        int bi = -1;
#pragma unroll 2
        for (int i = 0; i < E; ++i) {
            const double s = __dmul_rn(dx[32 * i], inv);
            if (((dv >> i) & 1u) && s > best) { best = s; bi = i; }
        }
        if (bi >= 0) ba = 128 * (bi >> 2) + 4 * lane + (bi & 3);
    } else {
        double x[E];
#pragma unroll
        for (int i = 0; i < E; ++i) {
            x[i] = __dadd_rn((double)lg[i], sig0);
            if ((dv >> i) & 1u) lmx = dmax2(lmx, x[i]);
        }
        const double mx = warp_max_f64(lmx);
        double ls = 0.0;
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const double e = exp_nonpos(dmin2(__dsub_rn(x[i], mx), 0.0));
            x[i] = ((dv >> i) & 1u) ? e : 0.0;
            ls = __dadd_rn(ls, x[i]);
        }
        for (int k = lane; k < total; k += 32) {
            const double e = exp_nonpos(__dsub_rn(sc.x[k], mx));
            sc.x[k] = e; ls = __dadd_rn(ls, e);
        }
        inv = __ddiv_rn(1.0, warp_sum_f64(ls));
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const double s = __dmul_rn(x[i], inv);
            if (((dv >> i) & 1u) && s > best) { best = s; ba = 128 * (i >> 2) + 4 * lane + (i & 3); }
        }
    }
    if (total > 0) {
        const double dn = (double)(1 + sumN);
        for (int k = lane; k < total; k += 32) {
            const double s = __dsub_rn(__dmul_rn(sc.x[k], inv), __ddiv_rn((double)sc.n[k], dn));
            const int a = sc.key[k] >> 16;
            if (s > best || (s == best && a < ba)) { best = s; ba = a; bc = sc.key[k] & 0xffff; }
        }
    }
    // warp argmax, lowest action wins ties (np.argmax, mcts.py:117)
    const u64 mk = warp_max_key(f64_key(best));
    const int a = __reduce_min_sync(GMZ_FULL, f64_key(best) == mk ? ba : 0x7fffffff);
    const unsigned own = __ballot_sync(GMZ_FULL, f64_key(best) == mk && ba == a);
    action = a;
    child = __shfl_sync(GMZ_FULL, bc, __ffs(own) - 1);
    __syncwarp();
    return sel_pack(action, child);
}

// The exact _select_action (mcts.py:106-117) for nodes with <= 32 visited children: lane k owns
// visited child k in registers (N, W -> q -> sigma -> exp -> score), every lane owns 4*NC dense
// (unvisited) actions.  Same arithmetic, same order of operations per element as the big variant.
// Out of line: it only runs when the certified path below cannot decide.
template <int NC, bool MZ, bool F32>
__device__ __noinline__ int select_interior_exact(const Params &p, const SelCtx w, int node, int lane, SelSmem &sm, int warp_slot)
{
    int action, child;
    constexpr int E = 4 * NC;
    const size_t ni = w.nbase + (size_t)node;
    const float *lrow = p.logits + ni * (size_t)p.AP;
    const short *crow = p.child + ni * (size_t)p.AP;
    float lg[E]; short ch[E];
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        const float4 t = *reinterpret_cast<const float4 *>(lrow + 128 * j + 4 * lane);
        const short4 c = *reinterpret_cast<const short4 *>(crow + 128 * j + 4 * lane);
        lg[4 * j + 0] = t.x; lg[4 * j + 1] = t.y; lg[4 * j + 2] = t.z; lg[4 * j + 3] = t.w;
        ch[4 * j + 0] = c.x; ch[4 * j + 1] = c.y; ch[4 * j + 2] = c.z; ch[4 * j + 3] = c.w;
    }
    unsigned vm = 0;
#pragma unroll
    for (int i = 0; i < E; ++i) vm |= (ch[i] >= 0 ? 1u : 0u) << i;
    int total = 0;
    if (__any_sync(GMZ_FULL, vm != 0)) {
        const int cnt = __popc(vm);
        int inc = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(GMZ_FULL, inc, o); if (lane >= o) inc += t; }
        total = __shfl_sync(GMZ_FULL, inc, 31);
        if (total > 32) return select_interior_big<NC, MZ, F32>(p, w, node, lane, sm, warp_slot);
        int pos = inc - cnt;
#pragma unroll
        for (int i = 0; i < E; ++i) {
            if ((vm >> i) & 1u) {
                sm.key[pos] = ((128 * (i >> 2) + 4 * lane + (i & 3)) << 16) | (int)ch[i];
                sm.lg[pos] = lg[i];
                ++pos;
            }
        }
        __syncwarp();
    }
    // sparse: lane k < total owns visited child k
    const bool sp = lane < total;
    int key = 0, nn = 0; float slg = 0.f; double W = 0.0, rew = 0.0;
    if (sp) {
        key = sm.key[lane]; slg = sm.lg[lane];
        const size_t ci = w.nbase + (size_t)(key & 0xffff);
        nn = p.nN[ci]; W = p.nW[ci];
        if (MZ) rew = p.nR[ci];
    }
    const int maxN = __reduce_max_sync(GMZ_FULL, nn), sumN = __reduce_add_sync(GMZ_FULL, nn);
    const double scale = __dmul_rn(__dadd_rn(p.c_visit, (double)maxN), p.c_scale);
    const bool rng = w.mm_max > w.mm_min;
    const double denom = mm_denom<F32>(p, w.mm_min, w.mm_max);
    const double sig0 = __dmul_rn(scale, mm_norm(0.0, rng, w.mm_min, denom));   // unvisited: q = 0.0
    double lmx = -INFINITY, xs = -INFINITY;
    if (sp) {
        const double q = q_of<F32>(p, W, nn, rew);
        xs = __dadd_rn((double)slg, __dmul_rn(scale, mm_norm(q, rng, w.mm_min, denom)));
        lmx = xs;
    }
    const unsigned dv = w.vb & ~vm;      // valid and unvisited: the dense set
    double best = -INFINITY; int ba = 0x7fffffff, bc = -1;
    double inv;
    if (NC <= 2) {
        // rolled loops over this lane's E elements staged in shared memory: small code (the loop is
        // bound by instruction fetch / dependent-issue latency, not by the extra LDS/STS)
        double *dx = sm.dx + lane;
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const double xi = __dadd_rn((double)lg[i], sig0);
            dx[32 * i] = xi;
            if ((dv >> i) & 1u) lmx = dmax2(lmx, xi);
        }
        const double mx = warp_max_f64(lmx);
        double ls = 0.0;
#pragma unroll kExpUnroll
        for (int i = 0; i < E; ++i) {
            double e = exp_nonpos(dmin2(__dsub_rn(dx[32 * i], mx), 0.0));
            e = ((dv >> i) & 1u) ? e : 0.0;
            dx[32 * i] = e;
            ls = __dadd_rn(ls, e);
        }
        if (sp) { xs = exp_nonpos(__dsub_rn(xs, mx)); ls = __dadd_rn(ls, xs); }
        inv = __ddiv_rn(1.0, warp_sum_f64(ls));
        int bi = -1;
#pragma unroll 2
        for (int i = 0; i < E; ++i) {
            const double s = __dmul_rn(dx[32 * i], inv);
            if (((dv >> i) & 1u) && s > best) { best = s; bi = i; }
        }
        if (bi >= 0) ba = 128 * (bi >> 2) + 4 * lane + (bi & 3);
    } else {
        double x[E];
#pragma unroll
        for (int i = 0; i < E; ++i) {
            x[i] = __dadd_rn((double)lg[i], sig0);
            if ((dv >> i) & 1u) lmx = dmax2(lmx, x[i]);
        }
        const double mx = warp_max_f64(lmx);
        double ls = 0.0;
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const double e = exp_nonpos(dmin2(__dsub_rn(x[i], mx), 0.0));
            x[i] = ((dv >> i) & 1u) ? e : 0.0;
            ls = __dadd_rn(ls, x[i]);
        }
        if (sp) { xs = exp_nonpos(__dsub_rn(xs, mx)); ls = __dadd_rn(ls, xs); }
        inv = __ddiv_rn(1.0, warp_sum_f64(ls));
#pragma unroll
        for (int i = 0; i < E; ++i) {
            const double s = __dmul_rn(x[i], inv);
            if (((dv >> i) & 1u) && s > best) { best = s; ba = 128 * (i >> 2) + 4 * lane + (i & 3); }
        }
    }
    if (sp) {
        const double s = __dsub_rn(__dmul_rn(xs, inv), __ddiv_rn((double)nn, (double)(1 + sumN)));
        const int a = key >> 16;
        if (s > best || (s == best && a < ba)) { best = s; ba = a; bc = key & 0xffff; }
    }
    // warp argmax, lowest action wins ties (np.argmax, mcts.py:117)
    const u64 mk = warp_max_key(f64_key(best));
    const int a = __reduce_min_sync(GMZ_FULL, f64_key(best) == mk ? ba : 0x7fffffff);
    const unsigned own = __ballot_sync(GMZ_FULL, f64_key(best) == mk && ba == a);
    action = a;
    child = __shfl_sync(GMZ_FULL, bc, __ffs(own) - 1);
    __syncwarp();
    return sel_pack(action, child);
}

// ---------------------------------------------------------------------------------------------
// Certified select.  At an interior node every UNVISITED action has q = 0 and N = 0, so its score is
// just its softmax probability: among the unvisited root-valid actions the winner is always the one
// with the highest logit (lowest index among equals), whatever sigma and the MinMaxStats are.  Each
// node therefore carries a 16-byte summary of its unvisited set,
//     ub  = that best unvisited action,  lub = its logit,
//     U   = sum over the unvisited valid actions of exp(logit - lub)       (float32, in [1, A])
// and the list of its children in creation order WITH THEIR EDGE STATISTICS MIRRORED IN: one 1 KiB block per
// node (Params::nBlk) of 32 slots x 32 bytes -- slot 0 the summary, slot j (1..31) child j-1 as
//     { (action << 16) | child id,  logit,  N(child),  -,  W(child) f64,  x f64 },   x = reward(child) in MuZero mode,
//     x = get_qsa(child) in AlphaZero mode (exact: the backup computes it for the MinMaxStats anyway).
// The candidates of a select are then the <= 31 visited children plus `ub`: one per lane, no pass over the A
// logits, ONE memory round trip per tree level (lane j reads its own slot while every lane reads slot 0; the
// canonical per-node arrays nN / nW / nR are only read by the exact path, the root and the halving), and the
// softmax denominator is
//     sum_visited exp(x_c - mx) + exp(x_ub - mx) * U.
// The backup keeps the mirror current: it already holds each path node's statistics in registers (handed
// over by the descent that read them), so it needs no loads at all -- it stores N / W to the node's own
// arrays and to its slot in the parent's block.
// The summary is float32 (relative error ~3e-6 on the probabilities), so the decision is CERTIFIED:
// it is taken only if the best score clears every other candidate by more than that error, or ties
// with candidates whose inputs are bit-identical (then the lowest action wins, as np.argmax); otherwise
// the exact float64 path above decides.  Visit counts stay bit-exact; the summary is rebuilt (one pass
// over the parent's logits, float32 exp) once per simulation, when a child is added.
constexpr int kBlkBytes = 1024;       // per-node block (Params::nBlk): 32 slots of 32 bytes
constexpr int kSlotBytes = 32;
#ifndef GMZ_LIST_SPEC
#define GMZ_LIST_SPEC 8
#endif
constexpr int kListSpec = GMZ_LIST_SPEC;   // slots loaded speculatively with the header (one per lane; 5 of 6 nodes have < 8 children)
constexpr int kFastMaxVisited = 31;   // visited children (slots 1..31) + the best unvisited action fit one warp

// Per-lane view of the descent path: lane d holds the node at depth d (depths >= 32 spill to Params::path) with
// the statistics the descent read for it, i.e. BEFORE this simulation's backup.  mir = (parent node << 5) | slot
// of this node in the parent's block (slot 0 = not mirrored: root children, children past the 31st).
struct PathReg { int node, mir, n; double W, R; };
__device__ __forceinline__ char *blk_of(const Params &p, size_t ni) { return p.nBlk + ni * (size_t)kBlkBytes; }
constexpr double kCertEps = 4.5e-5;   // > 2x the error bound of a probability on this path, ~1.8e-5: float32 exp at
                                      // |d| <= 87.4 ~1.2e-5 (grows with |d|), softmax denominator with U's share ~6e-6,
                                      // rcp_approx + two float32 roundings ~2e-7 (tests/test_numerics_gpu.py budget)

// ub / lub / U / "ambiguous" for the candidate set `cand` (bit i = this lane's action i).  Ambiguous:
// two different unvisited logits closer than 1e-6 -- float64 rounding of logit + sigma could merge
// them, so such a node always takes the exact path.
// WITH_U = false: a freshly expanded node.  Its U is never read -- the first select at the node has no
// visited child and returns `ub` outright, and adding that child rebuilds the summary -- so only ub / lub /
// amb are computed.
template <int NC, bool WITH_U>
__device__ __forceinline__ void unvisited_summary(const float *lg, unsigned cand, int lane, int &ub, float &lub, float &U, bool &amb)
{
    constexpr int E = 4 * NC;
    // rows never hold -0.0 (canonicalised when they are written), so equal logits have equal bits
    float v[E], best = -INFINITY;
#pragma unroll
    for (int i = 0; i < E; ++i) { v[i] = ((cand >> i) & 1u) ? lg[i] : -INFINITY; best = fmaxf(best, v[i]); }
    const unsigned mk = __reduce_max_sync(GMZ_FULL, f32_key(best));
    lub = f32_unkey(mk);
    int bi = E;
#pragma unroll
    for (int i = E - 1; i >= 0; --i) bi = (v[i] == lub) ? i : bi;
    ub = __reduce_min_sync(GMZ_FULL, (bi < E && cand != 0u) ? 128 * (bi >> 2) + 4 * lane + (bi & 3) : 0x7fffffff);
    if (ub == 0x7fffffff) { ub = -1; lub = 0.0f; U = 0.0f; amb = false; return; }
    float u = 0.0f; bool am = false;
#pragma unroll
    for (int i = 0; i < E; ++i) {
        const float d = __fsub_rn(v[i], lub);                          // <= 0, -inf for non-candidates (exp -> 0)
        if (WITH_U) u = __fadd_rn(u, exp_approx(d));
        am |= (d < 0.0f) && (d > -1e-6f);
    }
    U = WITH_U ? warp_sum_fx(u) : 0.0f;              // <= 12 terms per lane (NC = 3), each <= 1: one fixed-point REDUX (error <= 2e-6 of U >= 1)
    amb = __any_sync(GMZ_FULL, am);
}

__device__ __forceinline__ int4 hdr_pack(float U, float lub, int ub, int nvis, int flags)
{
    return make_int4(__float_as_int(U), __float_as_int(lub), (ub & 0xffff) | (nvis << 16), flags);
}

// Header of a freshly expanded node: nothing visited yet.
template <int NC>
__device__ __forceinline__ void node_init_hdr(const Params &p, const WG &w, int node, const float *lg, int lane)
{
    int ub; float lub, U; bool amb;
    unvisited_summary<NC, false>(lg, w.vb[lane], lane, ub, lub, U, amb);
    if (lane == 0) *reinterpret_cast<int4 *>(blk_of(p, w.nbase + (size_t)node)) = hdr_pack(U, lub, ub, 0, amb ? 1 : 0);
}

// node.children[action] = new_node (mcts.py:27-30, 109): the child-row link, and for a non-root parent
// the block slot (key + logit; the backup fills in N / W / reward) + the refreshed summary of what is still
// unvisited.  Returns the new node's mirror word (parent << 5) | slot, slot 0 = not mirrored.
template <int NC>
__device__ __forceinline__ int node_link(const Params &p, const WG &w, int parent, int action, int new_node, int lane)
{
    constexpr int E = 4 * NC;
    const size_t pi = w.nbase + (size_t)parent;
    short *crow = p.child + pi * (size_t)p.AP;
    if (parent == 0) { if (lane == 0) crow[action] = (short)new_node; return 0; }
    const float *lrow = p.logits + pi * (size_t)p.AP;
    float lg[E]; unsigned vm = 0;
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        const float4 t = *reinterpret_cast<const float4 *>(lrow + 128 * j + 4 * lane);
        const short4 c = *reinterpret_cast<const short4 *>(crow + 128 * j + 4 * lane);
        lg[4 * j + 0] = t.x; lg[4 * j + 1] = t.y; lg[4 * j + 2] = t.z; lg[4 * j + 3] = t.w;
        vm |= ((c.x >= 0 ? 1u : 0u) | (c.y >= 0 ? 2u : 0u) | (c.z >= 0 ? 4u : 0u) | (c.w >= 0 ? 8u : 0u)) << (4 * j);
    }
    char *blk = blk_of(p, pi);
    const int4 h = *reinterpret_cast<const int4 *>(blk);
    const int owner = (action & 127) >> 2, idx = 4 * (action >> 7) + (action & 3);
    if (lane == owner) vm |= 1u << idx;
    float la = __int_as_float(h.y);                       // the new child is normally the summary's best unvisited action
    if (action != (int)(short)(h.z & 0xffff)) {           // (not when the exact path broke a near-tie differently)
        la = 0.0f;
        if (lane == owner) {
#pragma unroll
            for (int i = 0; i < E; ++i) if (i == idx) la = lg[i];
        }
        la = __shfl_sync(GMZ_FULL, la, owner);
    }
    __syncwarp();
    const int nvis = (h.z >> 16) + 1;
    const int slot = nvis <= kFastMaxVisited ? nvis : 0;
    if (lane == 0) {
        crow[action] = (short)new_node;
        if (slot) *reinterpret_cast<int2 *>(blk + kSlotBytes * slot) = make_int2((action << 16) | new_node, __float_as_int(la));
    }
    int ub; float lub, U; bool amb;
    unvisited_summary<NC, true>(lg, w.vb[lane] & ~vm, lane, ub, lub, U, amb);
    if (lane == 0) *reinterpret_cast<int4 *>(blk) = hdr_pack(U, lub, ub, min(nvis, 32767), (amb || nvis > kFastMaxVisited) ? 1 : 0);
    return (parent << 5) | slot;
}

// One slot of a node's block: the first 16 bytes (key, logit, N) and the statistics behind them
// (R = the child's reward in MuZero mode, its q in AlphaZero mode).
// One 32-byte slot of a node block with ONE 256-bit load (sm_100: ld.global.v8.b32) carrying the L2 eviction hint
// evict_last: the blocks are the re-read part of a tree -- the hot set is ~200 MB against 126 MB of L2 -- while
// the logits / child rows are written once with streaming stores (node_write_row).  466 -> 472 M sims/s.
__device__ __forceinline__ void ld_slot(const char *ptr, int4 &a, int4 &b)
{
#ifndef GMZ_NO_BLK_EVICT_LAST
    asm volatile("ld.global.L2::evict_last.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
#else
    asm volatile("ld.global.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
#endif
                 : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(ptr));
}
template <bool MZ>
__device__ __forceinline__ void slot_load(const char *slot, int4 &e, double &W, double &R)
{
    int4 t;
    ld_slot(slot, e, t);
    W = __hiloint2double(t.y, t.x); R = __hiloint2double(t.w, t.z);
}

// Returns the chosen action, the child it leads to (-1 = not created yet) and -- for an existing child --
// its slot in this node's block (0 = not mirrored) and its statistics N / W / reward as of now.
template <int NC, bool MZ, bool F32>
__device__ __forceinline__ void select_interior(const Params &p, const WG &w, size_t nbase, int node, int lane, SelSmem &sm, int warp_slot,
                                                double mn, double rden, int &action, int &child, int &slot, int &cn, double &cW, double &cR)
{
    const size_t ni = nbase + (size_t)node;
    const char *blk = blk_of(p, ni);
    const char *mine = blk + kSlotBytes * lane;
    int4 h, hspare;
    ld_slot(blk, h, hspare);
    // slots 1..7 are fetched alongside the summary: one round trip for 5 of 6 nodes
    int4 e = make_int4(0, 0, 0, 0); double eW = 0.0, eR = 0.0;
    if (lane >= 1 && lane < kListSpec) slot_load<MZ>(mine, e, eW, eR);
    const int nvis = h.z >> 16, ub = (int)(short)(h.z & 0xffff);
    bool loaded_all = false;
    if (h.w == 0) {
        if (nvis == 0) { action = ub; child = -1; slot = 0; cn = 0; cW = 0.0; cR = 0.0; return; }   // nothing visited: the highest logit wins outright
        const bool vis = lane >= 1 && lane <= nvis, un = lane == 0 && ub >= 0, cand = vis || un;
        if (vis && lane >= kListSpec) slot_load<MZ>(mine, e, eW, eR);
        loaded_all = true;
        int key = (ub << 16) | 0xffff, nn = 0; float slg = __int_as_float(h.y); double W = 0.0, rew = 0.0;
        if (vis) { key = e.x; slg = __int_as_float(e.y); nn = e.z; W = eW; rew = MZ ? eR : 0.0; }
#if defined(GMZ_PREFETCH_CHILD_L1) || defined(GMZ_PREFETCH_CHILD_L2)
        if (vis) {      // the next level reads the chosen child's block: start pulling every candidate's first line now
            const char *cb = blk_of(p, w.nbase + (size_t)(key & 0xffff));
#ifdef GMZ_PREFETCH_CHILD_L1
            asm volatile("prefetch.global.L1 [%0];" ::"l"(cb));
#else
            asm volatile("prefetch.global.L2 [%0];" ::"l"(cb));
#endif
        }
#endif
        const int maxN = __reduce_max_sync(GMZ_FULL, nn), sumN = __reduce_add_sync(GMZ_FULL, nn);
        const double scale = (p.c_visit + (double)maxN) * p.c_scale;
        double xs = -INFINITY;
        if (cand) {
            // AlphaZero mode: q comes with the slot.  MuZero mode, float32: q IS float32 arithmetic in the reference -> exact here too
            const double q = !vis ? 0.0 : (!MZ ? eR : (F32 ? q_of<true>(p, W, nn, rew) : rew + p.discount * (W * rcp_newton((double)nn))));
            double nrm = (q - mn) * rden;                       // (mn, rden) = (0, 0) while max <= min: normalize() is 0 then
            const int hi = __double2hiint(nrm);                  // clamp to [0, 1] on the high word
            nrm = hi < 0 ? 0.0 : (hi >= 0x3ff00000 ? 1.0 : nrm);
            xs = (double)slg + scale * nrm;
        }
        // any common shift near the maximum will do on this path: take it in float32 (one REDUX)
        const double mx = (double)f32_unkey(__reduce_max_sync(GMZ_FULL, f32_key(cand ? (float)xs : -INFINITY)));
        const float ef = cand ? exp_approx((float)(xs - mx)) : 0.0f;
        const float sum = warp_sum_fx(un ? __fmul_rn(ef, __int_as_float(h.x)) : ef);
        const float pf = __fmul_rn(ef, rcp_approx(sum));
        const double s = (double)pf - (double)nn * rcp_newton((double)(1 + sumN));
        // the winner is FOUND in float32 (one REDUX; lowest action among float32 ties) and then CERTIFIED in float64
        // against every other candidate: a candidate that beats it by less than float32 resolution fails the margin
        // below like any other near-tie
        // (key = the score's float32 bits with the low 9 replaced by 511 - action: ONE REDUX orders by score, then by
        //  lowest action; candidates closer than 2^-14 relative merge into a "tie" and go through the margin test)
        const unsigned k32 = cand ? ((f32_key((float)s) & 0xFFFFFE00u) | (unsigned)(511 - (key >> 16))) : 0u;
        const unsigned mk = __reduce_max_sync(GMZ_FULL, k32);
        const int a = 511 - (int)(mk & 511u);
        const int bl = __ffs(__ballot_sync(GMZ_FULL, cand && k32 == mk)) - 1;
        const double sb = __shfl_sync(GMZ_FULL, s, bl);
        const float pb = __shfl_sync(GMZ_FULL, pf, bl);
        bool near = cand && lane != bl && !(sb - s > kCertEps * (double)(pb + pf));
        if (__any_sync(GMZ_FULL, near)) {      // a near-tie is fine only between bit-identical inputs (a true tie)
            const int nb = __shfl_sync(GMZ_FULL, nn, bl);
            const float lb = __shfl_sync(GMZ_FULL, slg, bl);
            const double Wb = __shfl_sync(GMZ_FULL, W, bl), rb = __shfl_sync(GMZ_FULL, rew, bl);
            near = near && !(nn == nb && nn > 0 && slg == lb && W == Wb && rew == rb);      // (AlphaZero mode: W and N fix q)
            near = __any_sync(GMZ_FULL, near);
        } else near = false;
        if (!near) {
            const int wkey = __shfl_sync(GMZ_FULL, key, bl);
            action = a; child = (wkey & 0xffff) == 0xffff ? -1 : (wkey & 0xffff);
            slot = bl;                                            // lane j scored slot j; lane 0 (the unvisited candidate) -> no slot
            cn = __shfl_sync(GMZ_FULL, nn, bl); cW = __shfl_sync(GMZ_FULL, W, bl);
            cR = MZ ? __shfl_sync(GMZ_FULL, rew, bl) : 0.0;
#ifdef GMZ_VERIFY_FAST
            int ea, ec;
            sel_unpack(select_interior_exact<NC, MZ, F32>(p, sel_ctx(w, lane), node, lane, sm, warp_slot), ea, ec);
            if (lane == 0) atomicAdd(&p.ctl->sel_fast, 1ull);
            if (ea == action && ec == child) return;
            if (lane == 0) atomicAdd(&p.ctl->sel_mismatch, 1ull);
            action = ea; child = ec;                              // the exact decision stands; locate it below
#else
            return;
#endif
        } else {
            if (lane == 0) atomicAdd(&p.ctl->sel_fallback, 1ull);
            sel_unpack(select_interior_exact<NC, MZ, F32>(p, sel_ctx(w, lane), node, lane, sm, warp_slot), action, child);
        }
    } else sel_unpack(select_interior_exact<NC, MZ, F32>(p, sel_ctx(w, lane), node, lane, sm, warp_slot), action, child);
    // the exact path decided: find the child among the mirrored slots (or read its own arrays)
    slot = 0; cn = 0; cW = 0.0; cR = 0.0;
    if (child >= 0) {
        const bool vis = lane >= 1 && lane <= min(nvis, kFastMaxVisited);
        if (vis && !loaded_all && lane >= kListSpec) slot_load<MZ>(mine, e, eW, eR);
        const unsigned hit = __ballot_sync(GMZ_FULL, vis && (e.x >> 16) == action);
        if (hit) {
            slot = __ffs(hit) - 1;
            cn = __shfl_sync(GMZ_FULL, e.z, slot); cW = __shfl_sync(GMZ_FULL, eW, slot);
            cR = MZ ? __shfl_sync(GMZ_FULL, eR, slot) : 0.0;
        } else {
            const size_t ci = nbase + (size_t)child;
            cn = p.nN[ci]; cW = p.nW[ci]; cR = MZ ? p.nR[ci] : 0.0;
        }
    }
}

// _select_leaf (mcts.py:88-104): root = first least-visited survivor (strict <, list order),
// then interior selection until an unexpanded child is reached.  In AlphaZero mode the path
// is replayed on the bitboards while descending (mcts.py:236-248).  Returns depth (edges).
// ds.path[d] <- the node at depth d, the action that led to it and its statistics.
template <int NC, bool MZ, bool F32>
__device__ __forceinline__ int descend(const Params &p, const WG &w, int2 *path, DescSmem &ds, SelSmem &sc, int warp_slot, int lane,
                                       int &leaf_parent, int &leaf_action)
{
    const unsigned key = lane < w.n_surv ? (((unsigned)w.s_n[lane] << 5) | (unsigned)lane) : 0xffffffffu;
    const int bl = (int)(__reduce_min_sync(GMZ_FULL, key) & 31u);
    int a = w.s_act[bl];
    int node = w.s_child[bl];
    const size_t nbase = w.nbase;
    int cn = 0, slot = 0;
    double cW = 0.0, cR = 0.0;
    // (the root and the chosen root child get their statistics from path_load() after the descent: only the
    //  backup consumes them, and loading them here would stall the first level on them)
    int parent = 0, depth = 1;
    // MinMaxStats only change in the backup: 1 / (max - min + delta) is the same at every level of this descent
    const bool rng = w.mm_max > w.mm_min;
    const double rden = rng ? rcp_newton(F32 ? mm_denom<true>(p, w.mm_min, w.mm_max) : (w.mm_max - w.mm_min) + p.delta) : 0.0, mn = rng ? w.mm_min : 0.0;
    while (node >= 0) {
        const int mir = (parent << 5) | slot;
        if (depth < 32) {          // (every lane stores the same entry: cheaper than electing one)
            PathEntry &e = ds.path[depth];
            e.node = node; e.mir = mir; e.n = cn; e.act = a; e.W = cW;
            if (MZ) e.R = cR;
        } else if (lane == 0) path[depth] = make_int2(node, mir | (a << 20));
        int c;
        select_interior<NC, MZ, F32>(p, w, nbase, node, lane, sc, warp_slot, mn, rden, a, c, slot, cn, cW, cR);
        parent = node; node = c; ++depth;
    }
    __syncwarp();
    leaf_parent = parent; leaf_action = a;
    return depth;
}

// The position at the leaf (AlphaZero mode, mcts.py:236-248): the root bitboards with the path's moves replayed on
// them, AFTER the descent -- nothing of it is live across the selects, and the actions come out of shared memory
// as independent loads.  The boards are kept RELATIVE to the player about to move (`mine`, `theirs`): a move sets the
// mover's bit and clears the other's (GomokuGame.do_move overwrites, game.py:20-23), then the roles swap -- two plies per
// iteration make the swap a renaming.  Lane w ends up with word w of the planes the evaluator sees at the leaf:
// own = the stones of the player to move there, opp = the other's (game.py:12-17).
__device__ __forceinline__ void bb_place(u64 &mover, u64 &other, int a, int lane)
{
    const u64 b = lane == (a >> 6) ? 1ull << (a & 63) : 0ull;
    mover |= b; other &= ~b;
}
__device__ __forceinline__ void replay_path(const Params &p, const WG &w, const int2 *path, const DescSmem &ds, int depth, int leaf_action,
                                            int lane, u64 &own, u64 &opp)
{
    const u64 rP = lane < GMZ_WORDS ? w.rP[lane] : 0ull, rM = lane < GMZ_WORDS ? w.rM[lane] : 0ull;
    u64 mine = w.to_move > 0 ? rP : rM, theirs = w.to_move > 0 ? rM : rP;
    // moves 1 .. depth-1 are the path's, move `depth` is the leaf action
    auto move_at = [&](int d) { return d < depth ? (d < 32 ? ds.path[d].act : (path[d].y >> 20)) : leaf_action; };
    int d = 1;
    for (; d < depth; d += 2) {
        bb_place(mine, theirs, move_at(d), lane);
        bb_place(theirs, mine, move_at(d + 1), lane);
    }
    if (d == depth) { bb_place(mine, theirs, leaf_action, lane); own = theirs; opp = mine; }     // odd number of plies: the roles end swapped
    else { own = mine; opp = theirs; }
}

// The descent's path into registers for the backup: lane d <- position d.  The root (lane 0) and the root child
// on the path (lane 1) have no slot in a parent's block, so their statistics come from the nodes' own arrays --
// issued here, right after the descent, consumed by the backup after the evaluation.
template <bool MZ>
__device__ __forceinline__ void path_load(const Params &p, const WG &w, const DescSmem &ds, int depth, PathReg &pr, int lane)
{
    const PathEntry e = ds.path[lane];                 // (lanes >= depth read stale entries; the backup ignores them)
    pr.node = lane == 0 ? 0 : e.node; pr.mir = lane == 0 ? 0 : e.mir; pr.n = e.n; pr.W = e.W; pr.R = MZ ? e.R : 0.0;
    if (lane == 0 || (lane == 1 && depth > 1)) {
        const size_t li = w.nbase + (size_t)pr.node;
        pr.n = p.nN[li]; pr.W = p.nW[li];
        if (MZ) pr.R = p.nR[li];
    }
}

// The leaf's parent is refreshed (node_link) after the evaluation: start pulling its logits / child rows
// into L1 now, so that the refresh does not pay the memory round trip.
template <int NC>
__device__ __forceinline__ void prefetch_parent_rows(const Params &p, const WG &w, int parent, int lane)
{
    if (parent == 0) return;
#ifdef GMZ_NO_PREFETCH
    return;
#endif
    const size_t pi = (w.nbase + (size_t)parent) * (size_t)(128 * NC);          // row index * AP
    const char *a = lane < 4 * NC ? (const char *)(p.logits + pi) + 128 * lane   // 4*NC lines of logits, 2*NC of child ids
                                  : (const char *)(p.child + pi) + 128 * (lane - 4 * NC);
    if (lane < 6 * NC) asm volatile("prefetch.global.L1 [%0];" ::"l"(a));
}

// leaf.expand (mcts.py:24-25, 260): write the new node's row (logits, no children) and link it.
template <int NC>
__device__ __forceinline__ void node_write_row(const Params &p, const WG &w, int node, const float *lg, int lane)
{
    const size_t ni = w.nbase + (size_t)node;
    float *lrow = p.logits + ni * (size_t)p.AP;
    short *crow = p.child + ni * (size_t)p.AP;
#pragma unroll
    for (int j = 0; j < NC; ++j) {
#ifndef GMZ_NO_STREAM_ROWS
        // a node's rows are written once and read at most a few times much later: keep them from evicting the blocks
        __stcs(reinterpret_cast<float4 *>(lrow + 128 * j + 4 * lane), make_float4(lg[4 * j], lg[4 * j + 1], lg[4 * j + 2], lg[4 * j + 3]));
        __stcs(reinterpret_cast<short4 *>(crow + 128 * j + 4 * lane), make_short4(-1, -1, -1, -1));
#else
        *reinterpret_cast<float4 *>(lrow + 128 * j + 4 * lane) = make_float4(lg[4 * j], lg[4 * j + 1], lg[4 * j + 2], lg[4 * j + 3]);
        *reinterpret_cast<short4 *>(crow + 128 * j + 4 * lane) = make_short4(-1, -1, -1, -1);
#endif
    }
}

// _backpropagate for one leaf, `reps` times in sequence (mcts.py:119-138; MuZero applies the
// same value len(selected) times, mcts.py:345).  Positions 0..depth-1 are the descent path, position
// `depth` is the new node.  Lane l owns position 32 c + l of chunk c; chunk 0 comes from the descent's
// registers (no loads), deeper chunks (paths longer than a warp) from Params::path and the nodes' own arrays.
// Also maintains the mirrored statistics in the parents' blocks and the MinMaxStats (min/max are
// order-independent).
template <bool MZ, bool F32>
__device__ __forceinline__ void backup(const Params &p, WG &w, const int2 *path, const PathReg &pr, int depth, int new_node, int new_mir,
                                       double value, double reward, int reps, int lane)
{
    double v = dclip1(value);
    double qmin = INFINITY, qmax = -INFINITY;
    const bool noclip = p.discount <= 1.0 && p.discount >= -1.0;      // (float32(discount) then is in [-1, 1] too)

    for (int c = depth >> 5; c >= 0; --c) {
        const int base = c << 5, top = min(depth, base + 31);
        const int pos = base + lane;
        const bool act = pos <= top;
        const bool is_new = pos == depth;
        int node = pr.node, mir = pr.mir, n = pr.n; double W = pr.W, R = MZ ? pr.R : 0.0;
        if (c > 0 && act && !is_new) {
            const int2 t = path[pos]; node = t.x; mir = t.y & 0xfffff;
            const size_t li = w.nbase + (size_t)node;
            n = p.nN[li]; W = p.nW[li]; if (MZ) R = p.nR[li];
        }
        if (is_new) { node = new_node; mir = new_mir; n = 0; W = 0.0; R = MZ ? reward : 0.0; }
        double myv = 0.0;
        if (!MZ && noclip) {            // no rewards, |discount| <= 1: after the first clip |v| can only shrink
            for (int l = top - base; l >= 0; --l) {
                if (lane == l) myv = v;
                v = F32 ? (double)__fmul_rn(p.discf, (float)v) : __dadd_rn(0.0, __dmul_rn(p.discount, v));
            }
        } else {
            for (int l = top - base; l >= 0; --l) {
                const double Rl = MZ ? __shfl_sync(GMZ_FULL, R, l) : 0.0;
                if (lane == l) myv = v;
                v = dclip1(F32 ? (double)__fadd_rn((float)Rl, __fmul_rn(p.discf, (float)v))
                               : __dadd_rn(Rl, __dmul_rn(p.discount, v)));   // value = node.reward + DISCOUNT * value; clip
            }
        }
        if (act) {
            double myq = 0.0;
            for (int r = 0; r < reps; ++r) {
                W = F32 ? (double)__fadd_rn((float)W, (float)myv) : __dadd_rn(W, myv); n += 1;
                if (pos > 0) {   // min_max_stats.update(parent.get_qsa(node.action))
                    myq = q_of<F32>(p, W, n, R);
                    qmin = dmin2(qmin, myq); qmax = dmax2(qmax, myq);
                }
            }
            const size_t ni = w.nbase + (size_t)node;
            p.nN[ni] = n; p.nW[ni] = W;
            if (MZ && is_new) p.nR[ni] = R;
            if (mir & 31) {              // the copy the parent's selects read
                char *e = blk_of(p, w.nbase + (size_t)(mir >> 5)) + kSlotBytes * (mir & 31);
                *reinterpret_cast<int *>(e + 8) = n;
                if (MZ) {
                    *reinterpret_cast<double *>(e + 16) = W;
                    if (is_new) *reinterpret_cast<double *>(e + 24) = R;
                } else *reinterpret_cast<double2 *>(e + 16) = make_double2(W, myq);   // W and get_qsa(child), read by the parent's selects
            }
        }
    }
    if (__any_sync(GMZ_FULL, qmin < w.mm_min || qmax > w.mm_max)) {      // rare once the range has settled
        qmin = warp_min_f64(qmin); qmax = warp_max_f64(qmax);
        const double nmin = dmin2(w.mm_min, qmin), nmax = dmax2(w.mm_max, qmax);
        __syncwarp();
        w.mm_min = nmin; w.mm_max = nmax;
        __syncwarp();
    }
}

// _ready_for_next_gumbel_phase (mcts.py:166-181), tables precomputed on the host.
__device__ __forceinline__ bool halving_ready(const Params &p, WG &w, int sim_count)
{
    const int thr = w.next_thr;
    if (sim_count < thr) return false;
    const int ph = w.phase + 1;
    if (ph > p.n_phases) { wg_set(w.phase, p.n_phases + 1); return false; }   // current_num_top_actions < 1
    __syncwarp();
    w.phase = ph; w.next_thr = min(thr + p.extra_of_phase[ph], p.S);
    __syncwarp();
    return true;
}

// _sequential_halving (mcts.py:183-185): survivors = first m of the current survivors sorted
// (stable, descending) by gumbel + logit + sigma(q) at the root.
template <bool MZ, bool F32>
__device__ __forceinline__ void sequential_halving(const Params &p, WG &w, int lane)
{
    const bool mine = lane < w.n_init;
    double q = 0.0;
    const int n = mine ? w.s_n[lane] : 0;
    if (mine && w.s_child[lane] >= 0) {
        const size_t ci = w.nbase + (size_t)w.s_child[lane];
        q = q_of<F32>(p, p.nW[ci], n, MZ ? p.nR[ci] : 0.0);
    }
    const int maxN = __reduce_max_sync(GMZ_FULL, n);
    const double scale = __dmul_rn(__dadd_rn(p.c_visit, (double)maxN), p.c_scale);
    const bool rng = w.mm_max > w.mm_min;
    const double denom = mm_denom<F32>(p, w.mm_min, w.mm_max);
    const double sig = __dmul_rn(scale, mm_norm(q, rng, w.mm_min, denom));
    GState *gs = p.gs + w.g;
    double s_g = gs->surv_g[lane]; float s_logit = gs->surv_logit[lane];
    const double score = __dadd_rn(__dadd_rn(s_g, (double)s_logit), sig);
    int rank = 0;
    for (int j = 0; j < w.n_surv; ++j) {
        const double sj = __shfl_sync(GMZ_FULL, score, j);
        if (sj > score || (sj == score && j < lane)) ++rank;
    }
    if (lane >= w.n_surv) rank = lane;
    int src = lane;
    for (int j = 0; j < 32; ++j) {
        const int rj = __shfl_sync(GMZ_FULL, rank, j);
        if (rj == lane) src = j;
    }
    {
        const int na = w.s_act[src], nc = w.s_child[src], nn = w.s_n[src];
        __syncwarp();
        w.s_act[lane] = na; w.s_child[lane] = nc; w.s_n[lane] = nn;
        __syncwarp();
    }
    s_g = __shfl_sync(GMZ_FULL, s_g, src);
    s_logit = __shfl_sync(GMZ_FULL, s_logit, src);
    gs->surv_g[lane] = s_g; gs->surv_logit[lane] = s_logit;
    wg_set(w.n_surv, min(p.m_of_phase[w.phase], w.n_surv));
}

// After a backup through root child `first_node` (depth-1 node on the path): bump the
// survivor's visit count (and record the child id if it was just created).
__device__ __forceinline__ void survivor_visit(WG &w, int depth, int path_node, int new_node, int leaf_action, int reps, int lane)
{
    const int first = __shfl_sync(GMZ_FULL, path_node, 1);     // every lane takes part: no shuffle behind a short-circuit
    bool hit;
    if (depth == 1) hit = lane < w.n_surv && w.s_act[lane] == leaf_action;
    else hit = lane < w.n_surv && w.s_child[lane] == first;
    if (hit) { w.s_n[lane] += reps; if (depth == 1) w.s_child[lane] = new_node; }
    __syncwarp();
}

// Root initialisation (mcts.py:217-226): expand root, first backup, halving schedule, Gumbel
// top-k = first K valid actions by (gumbel + logit, action) descending.
template <int NC>
__device__ __forceinline__ void root_init(const Params &p, WG &w, const float *lg, const double *gum, double value, int lane)
{
    node_write_row<NC>(p, w, 0, lg, lane);
    w.mm_min = INFINITY; w.mm_max = -INFINITY;
    if (lane == 0) {   // backup of the root alone: N = 1, W = clip(v)
        p.nN[w.nbase] = 1; p.nW[w.nbase] = dclip1(value);
        if (p.nR) p.nR[w.nbase] = 0.0;
    }
    w.num_nodes = 1; w.sim_count = 1; w.phase = 0; w.next_thr = p.first_thr;
    double sc[4 * NC];
    unsigned rem = w.vb[lane];
#pragma unroll
    for (int i = 0; i < 4 * NC; ++i) sc[i] = __dadd_rn(gum[i], (double)lg[i]);
    w.s_act[lane] = -1; w.s_child[lane] = -1; w.s_n[lane] = 0;
    GState *gs = p.gs + w.g;
    gs->surv_g[lane] = 0.0; gs->surv_logit[lane] = 0.f;
    __syncwarp();
    int cnt = 0;
    for (int r = 0; r < p.K; ++r) {
        double best = -INFINITY; int ba = -1;
#pragma unroll
        for (int i = 0; i < 4 * NC; ++i) {
            if ((rem >> i) & 1u) {
                const int a = 128 * (i >> 2) + 4 * lane + (i & 3);
                if (ba < 0 || sc[i] > best || (sc[i] == best && a > ba)) { best = sc[i]; ba = a; }
            }
        }
        if (ba < 0) best = -INFINITY;
        // lanes without candidates must lose: use (-inf, -1)
        warp_argmax_highidx(best, ba);
        if (ba < 0) break;
        const int owner = (ba & 127) >> 2;
        double gsel = 0.0; float lsel = 0.f;
        if (lane == owner) {
#pragma unroll
            for (int i = 0; i < 4 * NC; ++i)
                if (128 * (i >> 2) + 4 * lane + (i & 3) == ba) { gsel = gum[i]; lsel = lg[i]; rem &= ~(1u << i); }
        }
        gsel = __shfl_sync(GMZ_FULL, gsel, owner); lsel = __shfl_sync(GMZ_FULL, lsel, owner);
        if (lane == r) { w.s_act[lane] = ba; gs->surv_g[r] = gsel; gs->surv_logit[r] = lsel; }
        ++cnt;
    }
    w.n_init = cnt; w.n_surv = cnt;
    __syncwarp();
}

// The same planes as bf16 in NHWC order ([cell][own, opp, last]): what the network's first convolution reads
// (channels_last), written by the select itself so no cast / re-layout kernel sits between tree and network.
// Lane l writes the 4 cells x 3 channels x 2 bytes = 24 contiguous bytes of each chunk: adjacent lanes, adjacent bytes.
template <int NC>
__device__ __forceinline__ void obs_write_nhwc_bf16(unsigned short *obs, int A, u64 own_w, u64 opp_w, int last, int lane)
{
    constexpr unsigned short ONE = 0x3F80;      // bf16(1.0)
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        const u64 ow = shfl_u64(own_w, 2 * j + (lane >> 4)) >> ((lane & 15) * 4);
        const u64 pw = shfl_u64(opp_w, 2 * j + (lane >> 4)) >> ((lane & 15) * 4);
        const int a0 = 128 * j + 4 * lane;
        unsigned short v[12];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            v[3 * t + 0] = ((ow >> t) & 1ull) ? ONE : 0;
            v[3 * t + 1] = ((pw >> t) & 1ull) ? ONE : 0;
            v[3 * t + 2] = (a0 + t == last) ? ONE : 0;
        }
        // 16-bit stores: a game's block starts at g * 3A * 2 bytes, which is only 2-byte aligned for odd 3A
#pragma unroll
        for (int t = 0; t < 4; ++t)
            if (a0 + t < A) { obs[(size_t)(a0 + t) * 3] = v[3 * t]; obs[(size_t)(a0 + t) * 3 + 1] = v[3 * t + 1]; obs[(size_t)(a0 + t) * 3 + 2] = v[3 * t + 2]; }
    }
}

// Observation planes of a position (game.py:12-17) for this lane's actions, from the
// lane-distributed bitboards: own / opp relative to `to_move`, last-move one-hot.
template <int NC, typename T>
__device__ __forceinline__ void obs_write(T *obs, int A, u64 own_w, u64 opp_w, int last, int lane)
{
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        const u64 ow = shfl_u64(own_w, 2 * j + (lane >> 4)) >> ((lane & 15) * 4);
        const u64 pw = shfl_u64(opp_w, 2 * j + (lane >> 4)) >> ((lane & 15) * 4);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int a = 128 * j + 4 * lane + t;
            if (a < A) {
                obs[a] = (T)(float)((ow >> t) & 1ull);
                obs[A + a] = (T)(float)((pw >> t) & 1ull);
                obs[2 * A + a] = (T)(a == last ? 1.0f : 0.0f);
            }
        }
    }
}
