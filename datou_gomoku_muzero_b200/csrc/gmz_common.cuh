// gmz_common.cuh -- shared types and warp-level helpers of the batched Gumbel-MCTS engine.
//
// Execution model: ONE WARP OWNS ONE GAME TREE.  Simulations inside a game are sequential
// (the reference has exactly one simulation in flight per search, mcts.py:229-268, and visit
// counts must be bit-exact), so the parallelism is across the G concurrent games.  Within a
// warp the A actions of a node are spread over the 32 lanes: lane l owns actions
// 128*j + 4*l + t (j < NC chunks, t < 4), i.e. one float4 of logits and one short4 of child
// indices per chunk -- every row access is a fully coalesced 512-byte / 256-byte transaction.
//
// All parity-critical arithmetic is IEEE double with one rounding per operation
// (__dadd_rn/__dmul_rn/__ddiv_rn; the file is also compiled with -fmad=false), mirroring the
// reference's Python-float / NumPy-float64 arithmetic (SURVEY.md App. A.7).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

typedef unsigned long long u64;

#define GMZ_FULL 0xffffffffu
#define GMZ_MAX_PHASES 16
#define GMZ_WORDS 8  // 64-bit words per bitboard held in GState (A <= 384 uses <= 6)

// Per-game search + game state, one 1 KiB record per game (lane-indexed arrays so a warp
// loads/stores it with coalesced accesses).
struct __align__(128) GState {
    u64 p1[GMZ_WORDS];        // stones of player +1 at the root        game.py:9 board
    u64 m1[GMZ_WORDS];        // stones of player -1 at the root
    u64 valid[GMZ_WORDS];     // empty cells at the root = valid_moves   mcts.py:213
    double surv_g[32];        // gumbel noise of the initial top-k actions  mcts.py:221
    int surv_n[32];           // visit count of the root child of each survivor
    float surv_logit[32];     // root logit of each survivor
    short surv_act[32];       // selected_children_actions (first n_surv) + eliminated ones (up to n_init)
    short surv_child[32];     // node index of that root child, -1 if not created yet
    double mm_min, mm_max;    // utils.MinMaxStats                          utils.py:6-25
    int sim_count;            // mcts.py:228
    int num_nodes;            // nodes allocated in this game's pool (root = node 0)
    int phase;                // current_phase                              mcts.py:159
    int next_thr;             // visit_num_for_next_phase
    int n_surv;               // len(selected_children_actions)
    int n_init;               // length of the initial top-k list
    int to_move;              // game.current_player (+1 / -1)
    int last_move;            // game.last_move as an action index, -1 = None
    int move_count;           // game.move_count
    int active;               // 0: no valid moves -> search() sentinel (mcts.py:214-215)
    int leaf_parent;          // pending leaf (between select and expand_backup)
    int leaf_action;
    int leaf_depth;           // edges root -> leaf, 0 = nothing pending
    int leaf_reps;            // number of backups the pending leaf receives (MuZero: n_surv)
    int winner;               // get_game_ended(): +-1, 0 draw, 2 = None
    int busy;                 // play kernel: game is owned by a warp (acquire/release flag)
    int parked;               // finished, waiting for the host to hand out a trajectory slot
    int traj_slot;            // trajectory slot this game records into
    int traj_len;             // moves recorded in the current game
    unsigned noise_ctr;       // searches done by this game (Gumbel noise counter)
    unsigned deals;           // games dealt to this game index since the opening book was bound (gmz_set_openings)
    int opening;              // book opening the current game was dealt, + 1; 0 = not dealt from a book
    char pad1[88];
};
static_assert(sizeof(GState) == 1024, "GState must be 1 KiB");

// Kernel parameters (passed by value).
struct Params {
    int G, N, A, S, K, NW, AP, mode;   // NW = ceil(A/64) words in use, AP = padded row length (128*NC)
    int n_in_row, max_moves, first_thr, n_phases;
    int m_of_phase[GMZ_MAX_PHASES];      // current_num_top_actions after p halvings (mcts.py:168-169)
    int extra_of_phase[GMZ_MAX_PHASES];  // int(extra_visit) of phase p            (mcts.py:173-180)
    double c_visit, c_scale, delta, discount;
    float discf, deltaf;                 // float32(DISCOUNT), float32(VALUE_MINMAX_DELTA): float32 accumulation mode
    int f32acc, pad0;                    // gmz_config.accum_dtype == GMZ_F32
    GState *gs;
    float *logits;   // [G*S][AP]  node.policy_logits
    short *child;    // [G*S][AP]  node.children -> node index, -1 = absent
    int *nN;         // [G*S]      node.visit_count
    double *nW;      // [G*S]      node.value_sum
    double *nR;      // [G*S]      node.reward (MuZero mode only)
    u64 *nH;         // [G*S]      E0 hidden state of a node (MuZero mode + fixed evaluator only)
    int2 *path;      // [G][S+2]   (node id, mirror word) root..leaf-parent of the pending simulation (see PathReg)
    short *pyset;    // [ceil(G/4)*4][4096] scratch for the CPython-set tie-break (rare path)
    char *sel_overflow;   // [ceil(G/4)*4][128*NC*20 B] select scratch for nodes with > 64 visited children
    struct PlayCtl *ctl;   // play-kernel ticket counter + statistics
    char *nBlk;      // [G*S][1 KiB]  per node: summary of its unvisited actions + its children with their edge
                     //               statistics mirrored in, 32 slots of 32 bytes (see gmz_tree.cuh)
};

// Device-side control block of the play kernel (+ select statistics).
struct PlayCtl {
    unsigned long long next_ticket;        // round-robin game cursor of the current launch
    unsigned long long moves_started;      // moves handed out in the current launch
    unsigned long long moves_played;
    unsigned long long games_finished;
    unsigned long long tickets_unserved;   // no playable game found (everything busy / parked)
    unsigned long long tickets_idle;       // game acquired but no move came out of it
    unsigned long long sel_fallback;       // interior selects the certified path handed to the exact one
    unsigned long long sel_fast;           // (GMZ_VERIFY_FAST builds) selects decided by the certified path
    unsigned long long sel_mismatch;       // (GMZ_VERIFY_FAST builds) ... that the exact path decided differently
    unsigned long long pad[3];
};

// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double dclip1(double v) { return v < -1.0 ? -1.0 : (v > 1.0 ? 1.0 : v); }  // np.clip(v,-1,1)

// Order-preserving map double -> u64 (no NaNs on this path): a < b  <=>  key(a) < key(b).
__device__ __forceinline__ u64 f64_key(double v)
{
    const u64 b = (u64)__double_as_longlong(v);
    return b ^ ((b >> 63) ? ~0ull : 0x8000000000000000ull);
}
__device__ __forceinline__ double f64_unkey(u64 k)
{
    return __longlong_as_double((long long)(k ^ ((k >> 63) ? 0x8000000000000000ull : ~0ull)));
}
// warp max of keys with two 32-bit REDUX instead of ten shuffles
__device__ __forceinline__ u64 warp_max_key(u64 k)
{
    const unsigned hi = __reduce_max_sync(GMZ_FULL, (unsigned)(k >> 32));
    const unsigned lo = __reduce_max_sync(GMZ_FULL, (unsigned)(k >> 32) == hi ? (unsigned)k : 0u);
    return ((u64)hi << 32) | lo;
}
__device__ __forceinline__ double warp_max_f64(double v) { return f64_unkey(warp_max_key(f64_key(v))); }
__device__ __forceinline__ double warp_min_f64(double v) { return -f64_unkey(warp_max_key(f64_key(-v))); }
__device__ __forceinline__ double dmax2(double a, double b) { return b > a ? b : a; }
__device__ __forceinline__ double dmin2(double a, double b) { return b < a ? b : a; }

// exp(x) for x <= 0 (softmax arguments after subtracting the max), ~1 ulp: Cody-Waite range
// reduction + degree-11 polynomial, 2^k applied to the exponent field.  A pure function of x,
// so equal inputs give equal outputs (exact ties stay exact).  Far tail -> libdevice exp.
static __device__ __noinline__ double exp_far_tail(double x) { return exp(x); }
// Coefficients live in the constant bank so each Horner step is ONE DFMA with a c[][] operand
// (as 64-bit immediates ptxas rebuilds them with two moves per step, tripling the exp's cost).
static __constant__ double c_exp[16] = {
    1.4426950408889634, 6755399441055744.0, -6.93147180559945286e-01, -2.31904681384629956e-17,
    2.5052097064908941e-08, 2.7626262793835868e-07, 2.7557414788000726e-06, 2.4801504602132958e-05,
    1.9841269707468915e-04, 1.3888888932258898e-03, 8.3333333333978320e-03, 4.1666666666573905e-02,
    1.6666666666666563e-01, 5.0000000000000056e-01, 1.0, 1.0};
__device__ __forceinline__ double exp_nonpos(double x)
{
    if (x < -700.0) return exp_far_tail(x);
    double t = fma(x, c_exp[0], c_exp[1]);
    const int k = __double2loint(t);
    t -= c_exp[1];
    double r = fma(t, c_exp[2], x);
    r = fma(t, c_exp[3], r);
    double q = c_exp[4];
#pragma unroll
    for (int i = 5; i < 16; ++i) q = fma(q, r, c_exp[i]);
    return __hiloint2double(__double2hiint(q) + (int)((unsigned)k << 20), __double2loint(q));
}
// Order-preserving map float -> u32 and back.
__device__ __forceinline__ unsigned f32_key(float v)
{
    const unsigned b = __float_as_uint(v);
    return b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u);
}
__device__ __forceinline__ float f32_unkey(unsigned k) { return __uint_as_float(k ^ ((k >> 31) ? 0x80000000u : 0xffffffffu)); }
__device__ __forceinline__ float warp_sum_f32(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = __fadd_rn(v, __shfl_xor_sync(GMZ_FULL, v, o));
    return v;
}
// Sum of non-negative terms (lane total <= ~400, at least one == 1 up to rounding) in 2^-23 fixed point: ONE integer
// REDUX instead of a five-step shuffle tree (the largest legal total, 392 * 2^23, stays below 2^32).  Error: <= 2^-24
// per lane from the fixed point, plus one float32 rounding of the integer total (exact for totals below 2), i.e.
// <= 33 * 2^-24 relative on a sum >= 1 (certified select only; tests/test_numerics_gpu.py).
__device__ __forceinline__ float warp_sum_fx(float v)
{
    const unsigned q = __float2uint_rn(__fmul_rn(v, 8388608.0f));
    return __fmul_rn((float)__reduce_add_sync(GMZ_FULL, q), 1.1920928955078125e-07f);
}
// 1/x for x in the float range, to <= 4e-14 relative (1.4e-14 measured on a B200): float reciprocal + one Newton
// step (the certified select path only needs ~1e-9; the exact path keeps the correctly rounded division).
__device__ __forceinline__ float rcp_approx(float x)
{
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// exp(x) for x <= 0: one multiply and MUFU.EX2 (results below 2^-126 flush to +0).  Relative error <= 2^-22 + 1.3e-7 |x|
// for x = (float)d: the float32 roundings of d and of d * log2(e) each move the exponent by up to 2^-24 |d|, so the
// error grows with |d| (bound ~1.2e-5 at d = -87.4, measured 7.5e-6 on a B200); only near 0 is it ex2.approx's ~2^-22.
__device__ __forceinline__ float exp_approx(float x)
{
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(__fmul_rn(x, 1.4426950408889634f)));
    return r;
}
__device__ __forceinline__ double rcp_newton(double x)
{
    const double r = (double)rcp_approx((float)x);           // ~1.5 * 2^-23; one Newton step squares it: <= 4e-14 relative,
    return fma(r, fma(-x, r, 1.0), r);                       // nine orders below what the certificate tolerates
}
// xor-butterfly sum: a+b == b+a exactly, so every lane ends with the same bits
__device__ __forceinline__ double warp_sum_f64(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = __dadd_rn(v, __shfl_xor_sync(GMZ_FULL, v, o));
    return v;
}
// argmax with lowest-index tie-break (np.argmax, mcts.py:117)
__device__ __forceinline__ void warp_argmax_lowidx(double &s, int &a)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double s2 = __shfl_xor_sync(GMZ_FULL, s, o);
        int a2 = __shfl_xor_sync(GMZ_FULL, a, o);
        if (s2 > s || (s2 == s && a2 < a)) { s = s2; a = a2; }
    }
}
// argmax with highest-index tie-break (sorted(zip(scores, actions), reverse=True), mcts.py:225)
__device__ __forceinline__ void warp_argmax_highidx(double &s, int &a)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double s2 = __shfl_xor_sync(GMZ_FULL, s, o);
        int a2 = __shfl_xor_sync(GMZ_FULL, a, o);
        if (s2 > s || (s2 == s && a2 > a)) { s = s2; a = a2; }
    }
}
__device__ __forceinline__ u64 shfl_u64(u64 v, int src) { return __shfl_sync(GMZ_FULL, v, src); }

// ---------------------------------------------------------------------------------------------
// E0, the fixed deterministic evaluator (DESIGN.md; device twin of tests/golden/e0_py.py):
//   h0 = mix64(seed ^ GOLD)
//   h  = mix64( XOR_w [ ((own_w ^ h0) + (2w+1) GOLD) K1 ^ rot32(((opp_w ^ h0) + (2w+2) GOLD) K2) ] + (last+1) CV )
//   y = (lo32(h) ^ hi32(h)) + (a+1) * 0x9E3779B1;  x_a = (y ^ (y >> 16)) * 0x7FEB352D   (one multiply, high bits used)
//   quantised (logit_div > 0): logit = ((x_a >> 26) - 32) / logit_div,  value = ((h >> 40) % 33 - 16) / 16,
//                              reward = (((h >> 16) & 0xFFFFFF) % 5 - 2) / 16
//   dense (logit_div = 0):     logit = ((x_a >> 8) - 2^23) 2^-21,  value = ((h >> 40) - 2^23) 2^-23,
//                              reward = (((h >> 16) & 0xFFFFFF) - 2^23) 2^-25
//   MuZero mode: h_child = mix64(h_parent + (a+1) CA)
// The per-word terms are XOR-combined, so lane w hashes word w and a REDUX finishes the board hash; a word term is
// one odd-constant multiply (a bijection of the word), the single mix64 after the REDUX gives the avalanche.
#define E0_GOLD 0x9E3779B97F4A7C15ULL
#define E0_CV 0xD1B54A32D192ED03ULL
#define E0_CA 0x8CB92BA72F3D8DD7ULL
#define E0_GOLD32 0x9E3779B1u

#define E0_K1 0xBF58476D1CE4E5B9ULL
#define E0_K2 0x94D049BB133111EBULL

__host__ __device__ __forceinline__ u64 mix64(u64 z)
{
    z ^= z >> 30; z *= E0_K1;
    z ^= z >> 27; z *= E0_K2;
    z ^= z >> 31;
    return z;
}
// How E0's integers become numbers (host-prepared, passed by value to the kernels).
struct E0Spec {
    u64 h0;            // mix64(seed ^ GOLD)
    int lshift, lbias; // k = (x >> lshift) - lbias
    float lmul, ldiv;  // logit = lmul != 0 ? k * lmul : k / ldiv   (lmul = exact reciprocal of a power-of-two divisor)
    int dense;         // 0: quantised value / reward, 1: dense 24-bit value / reward
    int pad;
};
static inline E0Spec e0_spec(u64 seed, int logit_div)
{
    E0Spec s;
    s.h0 = mix64(seed ^ E0_GOLD); s.pad = 0;
    if (logit_div > 0) {
        s.lshift = 26; s.lbias = 32; s.dense = 0; s.ldiv = (float)logit_div;
        s.lmul = (logit_div & (logit_div - 1)) == 0 ? 1.0f / (float)logit_div : 0.0f;
    } else { s.lshift = 8; s.lbias = 1 << 23; s.dense = 1; s.ldiv = 1.0f; s.lmul = 4.76837158203125e-07f; /* 2^-21 */ }
    return s;
}
__device__ __forceinline__ u64 warp_xor_u64(u64 v)
{
    const unsigned lo = __reduce_xor_sync(GMZ_FULL, (unsigned)v), hi = __reduce_xor_sync(GMZ_FULL, (unsigned)(v >> 32));
    return ((u64)hi << 32) | lo;
}
// own_w / opp_w: lane w holds word w of the plane.  All lanes return the same hash.
__device__ __forceinline__ u64 e0_hash_planes(u64 h0, u64 own_w, u64 opp_w, int nw, int last, int lane)
{
    u64 t = 0;
    if (lane < nw) {
        const u64 b = ((opp_w ^ h0) + (u64)(2 * lane + 2) * E0_GOLD) * E0_K2;
        t = (((own_w ^ h0) + (u64)(2 * lane + 1) * E0_GOLD) * E0_K1) ^ ((b << 32) | (b >> 32));
    }
    return mix64(warp_xor_u64(t) + (u64)(long long)(last + 1) * E0_CV);
}
__device__ __forceinline__ unsigned e0_seed32(u64 h) { return (unsigned)h ^ (unsigned)(h >> 32); }
__device__ __forceinline__ unsigned e0_action_hash(unsigned x)      // x = seed32 + (a + 1) * E0_GOLD32
{
    x ^= x >> 16; x *= 0x7FEB352Du;
    return x;
}
__device__ __forceinline__ float e0_logit_of(unsigned x, const E0Spec &e)
{
    const float k = (float)((int)(x >> e.lshift) - e.lbias);
    return e.lmul != 0.0f ? __fmul_rn(k, e.lmul) : __fdiv_rn(k, e.ldiv);
}
__device__ __forceinline__ float e0_logit(u64 h, int a, const E0Spec &e)
{
    return e0_logit_of(e0_action_hash(e0_seed32(h) + (unsigned)(a + 1) * E0_GOLD32), e);
}
__device__ __forceinline__ u64 e0_child_hidden(u64 h_parent, int action) { return mix64(h_parent + (u64)(action + 1) * E0_CA); }
__device__ __forceinline__ double e0_value(u64 h, int dense)
{
    const int vk = (int)((h >> 40) & 0xFFFFFFull);
    return dense ? (double)(vk - (1 << 23)) * 1.1920928955078125e-07 : (double)(vk % 33 - 16) * 0.0625;
}
__device__ __forceinline__ double e0_reward(u64 h, int dense)
{
    const int rk = (int)((h >> 16) & 0xFFFFFFull);
    return dense ? (double)(rk - (1 << 23)) * 2.98023223876953125e-08 : (double)(rk % 5 - 2) * 0.0625;
}
