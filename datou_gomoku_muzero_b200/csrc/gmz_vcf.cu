// gmz_vcf.cu -- forced wins: the VCF (victory by continuous fours) and VCT (threats of three) solvers of include/gmz.h,
// for a batch of boards (k_vcf, k_vct) and in place on packed move records (k_records_vcf, k_records_vct).  The
// definitions, the visiting orders and the node counts are those gmz.h states; tests/csrc/vcf_ref.c and vct_ref.c
// restate them on the CPU.
//
// One warp per position.  The attacker's and the defender's stones are two bitboards of VW words in shared memory, and
// so is the depth-first stack: per level, the candidates not tried yet, the attacker's move and the forced reply.
// Expanding a position is one warp pass over the cells (lane l owns cells 32j + l), each cell walking its four
// directions; moves are set and cleared in the shared bitboards, so the search itself touches no global memory.
#include <stdint.h>

#include "gmz_internal.h"
#include "gmz_records.cuh"

namespace {

constexpr int VW = (GMZ_MAX_BOARD * GMZ_MAX_BOARD + 63) / 64;   // words of a bitboard and of `first` (6)
constexpr int VCF_MAX_ATTACKS = 32;
constexpr int VCF_WARPS = 4;                                     // warps (positions) per CTA
static_assert(VW == 6, "gmz.h documents first as uint64 [6]");

struct VcfWarp {
    u64 bb[2][VW];                   // [0] attacker (side to move), [1] defender
    u64 cand[VCF_MAX_ATTACKS][VW];   // per level of the inner search: candidates not tried yet
    u64 root[VW];                    // the root's candidates not tried yet
    short m[VCF_MAX_ATTACKS], c[VCF_MAX_ATTACKS];   // per level: attacker's move and the forced reply below it
};

struct Geo {
    int N, A, n, budget;
};

__device__ __forceinline__ bool has(const u64 *b, int cell) { return (b[cell >> 6] >> (cell & 63)) & 1ull; }

// Lane 0 sets / clears a stone; the warp sees it after the __syncwarp.
__device__ __forceinline__ void put(u64 *b, int cell, bool on, int lane)
{
    if (lane == 0) {
        const u64 bit = 1ull << (cell & 63);
        b[cell >> 6] = on ? (b[cell >> 6] | bit) : (b[cell >> 6] & ~bit);
    }
    __syncwarp();
}

// Stones of `s` in a row from (r, c), stepping (dr, dc), not counting (r, c), at most n; (r, c) becomes the cell
// after the run (possibly off the board).  EXTRA: `extra` counts as one more stone of `s` (a move not on the board).
template <bool EXTRA = false>
__device__ __forceinline__ int run(const u64 *s, const Geo &g, int &r, int &c, int dr, int dc, int extra = -1)
{
    int k = 0;
    r += dr; c += dc;
    while (k < g.n && r >= 0 && r < g.N && c >= 0 && c < g.N && (has(s, r * g.N + c) || (EXTRA && r * g.N + c == extra))) {
        ++k; r += dr; c += dc;
    }
    return k;
}

template <bool EXTRA = false, class W>
__device__ __forceinline__ bool empty_on_board(const W &w, const Geo &g, int r, int c, int extra = -1)
{
    if (r < 0 || r >= g.N || c < 0 || c >= g.N) return false;
    const int cell = r * g.N + c;
    return !has(w.bb[0], cell) && !has(w.bb[1], cell) && !(EXTRA && cell == extra);
}

// direction d: (0, 1), (1, 0), (1, 1), (1, -1)
__device__ __forceinline__ int dir_r(int d) { return d != 0; }
__device__ __forceinline__ int dir_c(int d) { return d == 1 ? 0 : (d == 3 ? -1 : 1); }

// The completion cells a stone of side s (0 attacker, 1 defender) at `cell` would add in direction d: the first cell
// not of s on each side, if it is empty and closes a run of >= n through `cell`.  Valid while s has no completion
// cell (then every new one lies on a line through `cell`, next to the run that holds it).  EXTRA: a stone of s at
// `extra` (off `cell`'s position) counts as played.
template <bool EXTRA = false, class W>
__device__ __forceinline__ void four_ends(const W &w, const Geo &g, int cell, int d, bool &okL, int &eL, bool &okR, int &eR,
                                          int s = 0, int extra = -1)
{
    const int r = cell / g.N, c = cell % g.N, dr = dir_r(d), dc = dir_c(d);
    int rl = r, cl = c, rr = r, cr = c;
    const int aL = run<EXTRA>(w.bb[s], g, rl, cl, -dr, -dc, extra), aR = run<EXTRA>(w.bb[s], g, rr, cr, dr, dc, extra);
    okL = okR = false;
    eL = rl * g.N + cl; eR = rr * g.N + cr;
    if (empty_on_board<EXTRA>(w, g, rl, cl, extra)) {
        int r2 = rl, c2 = cl;
        okL = 2 + aL + aR + run<EXTRA>(w.bb[s], g, r2, c2, -dr, -dc, extra) >= g.n;
    }
    if (empty_on_board<EXTRA>(w, g, rr, cr, extra)) {
        int r2 = rr, c2 = cr;
        okR = 2 + aL + aR + run<EXTRA>(w.bb[s], g, r2, c2, dr, dc, extra) >= g.n;
    }
}

// Does a stone of side s (0 attacker, 1 defender) on the empty `cell` make a run of >= n?
template <class W>
__device__ __forceinline__ bool completes(const W &w, const Geo &g, int s, int cell, int d)
{
    const int r = cell / g.N, c = cell % g.N, dr = dir_r(d), dc = dir_c(d);
    int r1 = r, c1 = c, r2 = r, c2 = c;
    return 1 + run(w.bb[s], g, r1, c1, -dr, -dc) + run(w.bb[s], g, r2, c2, dr, dc) >= g.n;
}

// One expansion: the attacker's completion cells and four moves (lane w < VW holds word w of each mask), whether the
// attacker has a completion cell, and the defender's completion cells (count capped at 2, and the lowest one).
struct Scan {
    u64 compl_x, four;
    bool any_x;
    int n_y, y_cell;
};

__device__ Scan scan(const VcfWarp &w, const Geo &g, int lane)
{
    Scan s{0ull, 0ull, false, 0, -1};
    for (int j = 0; j * 32 < g.A; ++j) {
        const int cell = j * 32 + lane;
        bool cx = false, cy = false, f = false;
        if (cell < g.A && !has(w.bb[0], cell) && !has(w.bb[1], cell)) {
            for (int d = 0; d < 4; ++d) {
                cx |= completes(w, g, 0, cell, d);
                cy |= completes(w, g, 1, cell, d);
                bool okL, okR;
                int eL, eR;
                four_ends(w, g, cell, d, okL, eL, okR, eR);
                f |= okL || okR;
            }
        }
        const unsigned bx = __ballot_sync(GMZ_FULL, cx), by = __ballot_sync(GMZ_FULL, cy), bf = __ballot_sync(GMZ_FULL, f);
        if (lane == (j >> 1)) {
            s.compl_x |= (u64)bx << ((j & 1) * 32);
            s.four |= (u64)bf << ((j & 1) * 32);
        }
        s.any_x |= bx != 0u;
        if (by && s.y_cell < 0) s.y_cell = j * 32 + __ffs(by) - 1;
        s.n_y += __popc(by);
    }
    if (s.n_y > 2) s.n_y = 2;
    return s;
}

// Lowest candidate of `cand` (removed from it), -1 if none.
__device__ int pop(u64 *cand, int lane)
{
    const u64 v = lane < VW ? cand[lane] : 0ull;
    const unsigned nz = __ballot_sync(GMZ_FULL, v != 0ull);
    if (!nz) return -1;
    const int fw = __ffs(nz) - 1;
    int m = 0;
    if (lane == fw) { m = fw * 64 + __ffsll((long long)v) - 1; cand[lane] = v & (v - 1ull); }
    m = __shfl_sync(GMZ_FULL, m, fw);
    __syncwarp();
    return m;
}

// Side s's completion cells after it plays m (it had none before): their number, and the lowest-lane one.
template <class W>
__device__ int threats(const W &w, const Geo &g, int m, int lane, int &cell, int s = 0)
{
    bool okL = false, okR = false;
    int eL = -1, eR = -1;
    if (lane < 4) four_ends(w, g, m, lane, okL, eL, okR, eR, s);
    const int cnt = __reduce_add_sync(GMZ_FULL, (int)okL + (int)okR);
    const unsigned who = __ballot_sync(GMZ_FULL, okL || okR);
    cell = who ? __shfl_sync(GMZ_FULL, okL ? eL : eR, __ffs(who) - 1) : -1;
    return cnt;
}

// Does the defender's stone on `cell` make a run of >= n (attacker's move already on the board)?
template <class W>
__device__ __forceinline__ bool defender_completes(const W &w, const Geo &g, int cell, int lane)
{
    return __any_sync(GMZ_FULL, lane < 4 && completes(w, g, 1, cell, lane));
}

// Candidates of an expanded position into cand (lane w < VW writes word w): the four moves, or only the defender's
// completion cell if it has one and it is a four move.
__device__ __forceinline__ void store_candidates(u64 *cand, const Scan &s, int lane)
{
    u64 v = s.four;
    if (s.n_y == 1) v &= lane == (s.y_cell >> 6) ? 1ull << (s.y_cell & 63) : 0ull;
    if (lane < VW) cand[lane] = v;
    __syncwarp();
}

// vcf(current board, L0), depth first; the board is as it was when this returns.  1 true, 0 false, -1 budget cut.
// nodes counts expansions; limit_hit is set when a position is refused by "L <= 1".
__device__ int search(VcfWarp &w, const Geo &g, int L0, int empties, int &nodes, bool &limit_hit, int lane)
{
    int d = 0, res = 0;
    for (;;) {
        if (nodes == g.budget) { res = -1; break; }
        ++nodes;
        const Scan s = scan(w, g, lane);
        if (s.any_x) { res = 1; break; }
        const int L = L0 - d;
        if (L <= 1) limit_hit = true;
        if (L <= 1 || s.n_y >= 2) {
            if (lane < VW) w.cand[d][lane] = 0ull;
            __syncwarp();
        } else {
            store_candidates(w.cand[d], s, lane);
        }
        // next candidate of level d, backing up through exhausted levels
        bool down = false, done = false;
        while (!down && !done) {
            const int m = pop(w.cand[d], lane);
            if (m < 0) {
                if (d == 0) { res = 0; done = true; break; }
                --d;
                put(w.bb[0], w.m[d], false, lane);
                put(w.bb[1], w.c[d], false, lane);
                continue;
            }
            int c;
            if (threats(w, g, m, lane, c) >= 2) { res = 1; done = true; break; }
            put(w.bb[0], m, true, lane);
            if (empties - 2 * d - 2 == 0 || defender_completes(w, g, c, lane)) { put(w.bb[0], m, false, lane); continue; }
            put(w.bb[1], c, true, lane);
            if (lane == 0) { w.m[d] = (short)m; w.c[d] = (short)c; }
            __syncwarp();
            ++d;
            down = true;
        }
        if (done) break;
    }
    while (d > 0) {
        --d;
        put(w.bb[0], w.m[d], false, lane);
        put(w.bb[1], w.c[d], false, lane);
    }
    return res;
}

struct Result {
    int length, nodes;
    u64 first;   // lane w < VW: word w
};

// The whole solve of the position in w.bb (gmz.h: length, first, nodes).
__device__ Result solve(VcfWarp &w, const Geo &g, int max_attacks, int lane)
{
    int stones = 0;
    for (int k = 0; k < VW; ++k) stones += __popcll(w.bb[0][k]) + __popcll(w.bb[1][k]);
    const int empties = g.A - stones;
    Result out{0, 1, 0ull};
    const Scan s = scan(w, g, lane);
    if (s.any_x) { out.length = 1; out.first = s.compl_x; return out; }
    if (max_attacks <= 1 || s.n_y >= 2) return out;
    store_candidates(w.root, s, lane);
    int best = VCF_MAX_ATTACKS + 1;
    for (int m; (m = pop(w.root, lane)) >= 0;) {
        int c;
        bool wins = threats(w, g, m, lane, c) >= 2;
        int len = 2;
        if (!wins) {
            put(w.bb[0], m, true, lane);
            if (empties - 2 > 0 && !defender_completes(w, g, c, lane)) {
                put(w.bb[1], c, true, lane);
                for (len = 2; len <= max_attacks; ++len) {
                    bool limit_hit = false;
                    const int r = search(w, g, len - 1, empties - 2, out.nodes, limit_hit, lane);
                    if (r < 0) {
                        put(w.bb[1], c, false, lane);
                        put(w.bb[0], m, false, lane);
                        return Result{-1, out.nodes, 0ull};
                    }
                    if (r > 0) { wins = true; break; }
                    if (!limit_hit) break;
                }
                put(w.bb[1], c, false, lane);
            }
            put(w.bb[0], m, false, lane);
        }
        if (wins) {
            if (lane == (m >> 6)) out.first |= 1ull << (m & 63);
            best = min(best, len);
        }
    }
    out.length = best <= max_attacks ? best : 0;
    return out;
}

// The board (values by sign) into the shared bitboards, `P` (+-1) the attacker.
template <class W>
__device__ void load(W &w, const int8_t *board, int A, int P, int lane)
{
    u64 x = 0ull, y = 0ull;
    for (int j = 0; j * 32 < A; ++j) {
        const int cell = j * 32 + lane;
        const int v = cell < A ? board[cell] : 0;
        const unsigned bx = __ballot_sync(GMZ_FULL, v != 0 && (v > 0) == (P > 0));
        const unsigned by = __ballot_sync(GMZ_FULL, v != 0 && (v > 0) != (P > 0));
        if (lane == (j >> 1)) { x |= (u64)bx << ((j & 1) * 32); y |= (u64)by << ((j & 1) * 32); }
    }
    if (lane < VW) { w.bb[0][lane] = x; w.bb[1][lane] = y; }
    __syncwarp();
}

// A record's flag byte (gmz.h gmz_records_vcf / gmz_records_vct): bit 0 a forced win, bit 1 the played action starts
// one, bit 2 the budget cut the search.  The action indexes nothing before its range check.
__device__ __forceinline__ uint8_t record_flags(const Result &r, int action, int A, int lane)
{
    const bool played = __any_sync(GMZ_FULL, action >= 0 && action < A && lane == (action >> 6) &&
                                                 ((r.first >> (action & 63)) & 1ull));
    return (uint8_t)((r.length > 0 ? 1 : 0) | (played ? 2 : 0) | (r.length < 0 ? 4 : 0));
}

__global__ void __launch_bounds__(VCF_WARPS * 32)
k_vcf(const int8_t *boards, const int8_t *players, int batch, Geo g, int max_attacks, int32_t *out_length, u64 *out_first,
      int32_t *out_nodes)
{
    __shared__ VcfWarp sw[VCF_WARPS];
    const int lane = threadIdx.x & 31, b = blockIdx.x * VCF_WARPS + (threadIdx.x >> 5);
    if (b >= batch) return;                      // whole warps leave; nothing below synchronises the CTA
    VcfWarp &w = sw[threadIdx.x >> 5];
    load(w, boards + (size_t)b * g.A, g.A, players[b] >= 0 ? 1 : -1, lane);
    const Result r = solve(w, g, max_attacks, lane);
    if (lane < VW) out_first[(size_t)b * VW + lane] = r.first;
    if (lane == 0) { out_length[b] = r.length; out_nodes[b] = r.nodes; }
}

__global__ void __launch_bounds__(VCF_WARPS * 32)
k_records_vcf(const unsigned char *records, size_t stride, int n_records, Geo g, int max_attacks, uint8_t *out_flags)
{
    __shared__ VcfWarp sw[VCF_WARPS];
    const int lane = threadIdx.x & 31, k = blockIdx.x * VCF_WARPS + (threadIdx.x >> 5);
    if (k >= n_records) return;
    VcfWarp &w = sw[threadIdx.x >> 5];
    const unsigned char *rec = records + (size_t)k * stride;
    const gmz_move_record *h = rec_header(rec);
    const int action = h->action;
    load(w, rec_board(rec, g.A), g.A, h->to_move >= 0 ? 1 : -1, lane);
    const uint8_t f = record_flags(solve(w, g, max_attacks, lane), action, g.A, lane);
    if (lane == 0) out_flags[k] = f;
}

const char *check_limits(int board_size, int n_in_row, int max_attacks, int node_budget)
{
    if (board_size < 1 || board_size > GMZ_MAX_BOARD) return "board_size out of range";
    if (n_in_row < 1) return "n_in_row must be >= 1";
    if (max_attacks < 1 || max_attacks > VCF_MAX_ATTACKS) return "max_attacks must be in [1, 32]";
    if (node_budget < 1) return "node_budget must be >= 1";
    return nullptr;
}

// ---- VCT: forced wins through threats of three (gmz.h gmz_vct_solve) ----
// The same warp layout: bitboards and the stack in shared memory, one warp pass per expansion.  The search alternates
// X nodes (X to move: its threat moves) and Y nodes (Y to move: the forced block of X's four, or the replies R = D | K
// to X's three).  A path holds at most 2 L - 1 open levels below a Y node with L stones left (each X level and each Y
// level that blocks spends an attacker stone; a Y level that does not block is followed by an X level), so
// 2 * VCF_MAX_ATTACKS levels hold any search the limit allows.
constexpr int VCT_LEVELS = 2 * VCF_MAX_ATTACKS;
enum { KX = 0, KY_FORCED = 1, KY_REPLY = 2 };

struct VctWarp {
    u64 bb[2][VW];                   // [0] attacker X (side to move at the root), [1] defender Y
    u64 cand[VCT_LEVELS][VW];        // per level: X's threat moves or Y's replies not tried yet
    u64 root[VW];                    // the root's candidates not tried yet
    u64 tmp[VW];                     // the cells a pass tests: three-move candidates, or F2 for the defences
    short m[VCT_LEVELS], c[VCT_LEVELS];           // per level: the stone of the child searched, X's forced block (-1)
    signed char kind[VCT_LEVELS], L[VCT_LEVELS];  // per level: KX / KY_FORCED / KY_REPLY, attacker stones left
    unsigned char ends[GMZ_MAX_BOARD * GMZ_MAX_BOARD];   // per empty f: |C_X(B+X@f)| per direction, 2 bits each
};

// One expansion (lane w < VW holds word w of each mask): X's completion cells, four moves and F2 cells, the empty
// cells, and Y's four moves (YNODE); counts capped at 2 with the lowest cell.  An X node also leaves each empty
// cell's completion counts per direction in w.ends for the three-move pass.
struct VScan {
    u64 compl_x, four, f2, empty, yfour;
    int n_x, x_cell, n_y, y_cell, n_f2, f2_cell;
};

__device__ __forceinline__ void tally(unsigned b, int j, int &n, int &low)
{
    if (b && low < 0) low = j * 32 + __ffs(b) - 1;
    n = min(2, n + __popc(b));
}

__device__ __forceinline__ void gather(u64 &word, unsigned b, int j, int lane)
{
    if (lane == (j >> 1)) word |= (u64)b << ((j & 1) * 32);
}

template <bool YNODE>
__device__ __forceinline__ VScan vct_scan(VctWarp &w, const Geo &g, int lane)
{
    VScan s{0ull, 0ull, 0ull, 0ull, 0ull, 0, -1, 0, -1, 0, -1};
    for (int j = 0; j * 32 < g.A; ++j) {
        const int cell = j * 32 + lane;
        const bool e = cell < g.A && !has(w.bb[0], cell) && !has(w.bb[1], cell);
        bool cx = false, cy = false, yf = false;
        int cnt = 0, ends = 0;
        if (e) {
            for (int d = 0; d < 4; ++d) {
                cx |= completes(w, g, 0, cell, d);
                if (!YNODE) cy |= completes(w, g, 1, cell, d);
                bool okL, okR;
                int eL, eR;
                four_ends(w, g, cell, d, okL, eL, okR, eR);
                cnt += (int)okL + (int)okR;
                ends |= ((int)okL + (int)okR) << (2 * d);
                if (YNODE) {
                    four_ends(w, g, cell, d, okL, eL, okR, eR, 1);
                    yf |= okL || okR;
                }
            }
            if (!YNODE) w.ends[cell] = (unsigned char)ends;
        }
        const unsigned bx = __ballot_sync(GMZ_FULL, cx), by = __ballot_sync(GMZ_FULL, cy);
        const unsigned bf = __ballot_sync(GMZ_FULL, cnt >= 1), b2 = __ballot_sync(GMZ_FULL, cnt >= 2);
        gather(s.compl_x, bx, j, lane);
        gather(s.four, bf, j, lane);
        gather(s.f2, b2, j, lane);
        gather(s.empty, __ballot_sync(GMZ_FULL, e), j, lane);
        if (YNODE) gather(s.yfour, __ballot_sync(GMZ_FULL, yf), j, lane);
        tally(bx, j, s.n_x, s.x_cell);
        tally(by, j, s.n_y, s.y_cell);
        tally(b2, j, s.n_f2, s.f2_cell);
    }
    __syncwarp();
    return s;
}

__device__ __forceinline__ int sum_ends(int e) { return (e & 3) + (e >> 2 & 3) + (e >> 4 & 3) + (e >> 6 & 3); }

// X's three moves among the cells of w.tmp (empty, not four moves; X has no completion cell).  An X stone never
// removes an X completion cell except the one it lands on, so every cell's count rises or stays, and F2 minus m stays
// in F2(B+X@m) (if m completed B+X@f, f would complete B+X@m, a four).  A cell f gains only through a new completion
// cell e whose run holds m, f and e: only its count along the line through m and f changes, and the cells strictly
// between m and f are X stones or e -- so f is the first or second empty cell from m on one of m's lines, at most
// n - 1 away (farther, the cells from f up to m would already be a run of n with e, or f would complete B).
__device__ __forceinline__ u64 three_moves(const VctWarp &w, const Geo &g, const VScan &s, int lane)
{
    u64 out = 0ull;
    for (int j = 0; j * 32 < g.A; ++j) {
        const int m = j * 32 + lane;
        bool three = false;
        if (m < g.A && has(w.tmp, m)) {
            three = s.n_f2 >= 2 || (s.n_f2 == 1 && s.f2_cell != m);
            const int r = m / g.N, c = m % g.N;
            for (int d = 0; d < 4 && !three; ++d) {
                const int dr = dir_r(d), dc = dir_c(d);
                for (int sg = -1; sg <= 1 && !three; sg += 2) {
                    int rr = r, cc = c, gaps = 0;
                    for (int i = 1; i < g.n && !three; ++i) {
                        rr += sg * dr; cc += sg * dc;
                        if (rr < 0 || rr >= g.N || cc < 0 || cc >= g.N) break;
                        const int f = rr * g.N + cc;
                        if (has(w.bb[1], f)) break;
                        if (has(w.bb[0], f)) continue;
                        const int e = w.ends[f];
                        bool okL, okR;
                        int eL, eR;
                        four_ends<true>(w, g, f, d, okL, eL, okR, eR, 0, m);
                        three = sum_ends(e) - (e >> (2 * d) & 3) + (int)okL + (int)okR >= 2;
                        if (++gaps == 2) break;
                    }
                }
            }
        }
        gather(out, __ballot_sync(GMZ_FULL, three), j, lane);
    }
    return out;
}

// X's threat moves (X has no completion cell), restricted to Y's completion cell when Y has one.
__device__ __forceinline__ u64 threat_moves(VctWarp &w, const Geo &g, const VScan &s, int lane)
{
    const u64 only = s.n_y == 1 ? (lane == (s.y_cell >> 6) ? 1ull << (s.y_cell & 63) : 0ull) : ~0ull;
    if (lane < VW) w.tmp[lane] = s.empty & ~s.four & only;
    __syncwarp();
    return (s.four | three_moves(w, g, s, lane)) & only;
}

// Y's defences D (X has no completion cell, F2 in w.tmp, f0 its lowest cell).  A Y stone at d lowers f's count only by
// filling f or one of the completion cells of B+X@f -- the other cells of those runs are X stones -- and those lie on
// different lines, so by at most one; it creates no X completion cell.  So d is a defence iff for every f in F2,
// d == f or (|C_X(B+X@f)| == 2 and d is one of them): D lies within f0 and its completion cells, 9 candidates.
__device__ __forceinline__ u64 defences(const VctWarp &w, const Geo &g, int f0, int lane)
{
    bool okL = false, okR = false;
    int eL = -1, eR = -1;
    if (lane < 4) four_ends(w, g, f0, lane, okL, eL, okR, eR);
    int kc[9];
    kc[0] = f0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        kc[1 + 2 * i] = __shfl_sync(GMZ_FULL, okL ? eL : -1, i);
        kc[2 + 2 * i] = __shfl_sync(GMZ_FULL, okR ? eR : -1, i);
    }
    unsigned bad = 0u;               // bit i: candidate i leaves one of this lane's F2 cells standing
    for (int j = 0; j * 32 < g.A; ++j) {
        const int f = j * 32 + lane;
        if (f >= g.A || !has(w.tmp, f)) continue;
        int e[8], cnt = 0;
#pragma unroll
        for (int d = 0; d < 4; ++d) {
            four_ends(w, g, f, d, okL, eL, okR, eR);
            e[2 * d] = okL ? eL : -1;
            e[2 * d + 1] = okR ? eR : -1;
            cnt += (int)okL + (int)okR;
        }
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            bool kills = kc[i] == f;
#pragma unroll
            for (int k = 0; k < 8; ++k) kills |= cnt == 2 && kc[i] >= 0 && kc[i] == e[k];
            if (!kills) bad |= 1u << i;
        }
    }
    bad = __reduce_or_sync(GMZ_FULL, bad);
    u64 out = 0ull;
#pragma unroll
    for (int i = 0; i < 9; ++i)
        if (kc[i] >= 0 && !(bad >> i & 1u) && lane == (kc[i] >> 6)) out |= 1ull << (kc[i] & 63);
    return out;
}

// Expand the node at level d (an X node, or a Y node, with L attacker stones left): its value (1 / 0), or 2 with the
// level's kind, L and candidates stored.
__device__ __forceinline__ int vct_expand(VctWarp &w, const Geo &g, int d, bool xnode, int L, int empties, bool &limit_hit, int lane)
{
    int kind;
    u64 cand;
    if (xnode) {
        const VScan s = vct_scan<false>(w, g, lane);
        if (s.n_x) return 1;
        if (L <= 1) { limit_hit = true; return 0; }
        if (s.n_y == 0 && s.n_f2) return 1;
        if (s.n_y >= 2) return 0;
        cand = threat_moves(w, g, s, lane);
        kind = KX;
    } else {
        const VScan s = vct_scan<true>(w, g, lane);
        if (s.n_x >= 2) return 1;
        if (s.n_x == 1) {
            if (empties == 1 || defender_completes(w, g, s.x_cell, lane)) return 0;
            cand = lane == (s.x_cell >> 6) ? 1ull << (s.x_cell & 63) : 0ull;
            kind = KY_FORCED;
        } else {
            if (!s.n_f2) return 0;
            if (L < 2) { limit_hit = true; return 0; }
            if (lane < VW) w.tmp[lane] = s.f2;
            __syncwarp();
            cand = defences(w, g, s.f2_cell, lane) | s.yfour;
            kind = KY_REPLY;
        }
    }
    if (lane < VW) w.cand[d][lane] = cand;
    if (lane == 0) { w.kind[d] = (signed char)kind; w.L[d] = (signed char)L; }
    __syncwarp();
    return 2;
}

__device__ __forceinline__ void set_level(VctWarp &w, int d, int m, int c, int lane)
{
    if (lane == 0) { w.m[d] = (short)m; w.c[d] = (short)c; }
    __syncwarp();
}

// Play level d's candidate m and what it forces.  2: the child (xnode, L) is to be expanded at level d + 1; 0: the
// child is false without an expansion (its stones already taken back).
__device__ __forceinline__ int vct_enter(VctWarp &w, const Geo &g, int d, int m, int &empties, bool &xnode, int &L, int lane)
{
    const int kind = w.kind[d], Ld = w.L[d];
    if (kind == KX) {
        put(w.bb[0], m, true, lane);
        --empties;
        set_level(w, d, m, -1, lane);
        xnode = false; L = Ld - 1;
        return 2;
    }
    put(w.bb[1], m, true, lane);
    --empties;
    if (kind == KY_FORCED) {
        set_level(w, d, m, -1, lane);
        xnode = true; L = Ld;
        return 2;
    }
    int c = -1;
    const int k = empties == 0 ? 2 : threats(w, g, m, lane, c, 1);   // a full board is false like a double four of Y
    if (k == 1) {
        put(w.bb[0], c, true, lane);
        if (empties - 1 > 0) {
            --empties;
            set_level(w, d, m, c, lane);
            xnode = false; L = Ld - 1;
            return 2;
        }
        put(w.bb[0], c, false, lane);
    }
    if (k >= 1) {
        put(w.bb[1], m, false, lane);
        ++empties;
        return 0;
    }
    set_level(w, d, m, -1, lane);
    xnode = true; L = Ld;
    return 2;
}

// Take back level d's child stones.
__device__ __forceinline__ void vct_leave(VctWarp &w, int d, int &empties, int lane)
{
    const int c = w.c[d];
    put(w.bb[w.kind[d] == KX ? 0 : 1], w.m[d], false, lane);
    ++empties;
    if (c >= 0) { put(w.bb[0], c, false, lane); ++empties; }
}

// A child's value cv seen from its parent of `kind`: decided (an X node's first true, a Y node's first false, a cut),
// or 2 to try the parent's next candidate.
__device__ __forceinline__ int settle(int kind, int cv) { return cv < 0 || (kind == KX) == (cv == 1) ? cv : 2; }

// ynode(current board, L0), depth first; the board is as it was when this returns.  1 true, 0 false, -1 budget cut.
__device__ __forceinline__ int vct_search(VctWarp &w, const Geo &g, int L0, int empties, int &nodes, bool &limit_hit, int lane)
{
    int d = 0, L = L0;
    bool xnode = false;
    for (;;) {
        int v = -1;
        if (nodes < g.budget) {
            ++nodes;
            v = vct_expand(w, g, d, xnode, L, empties, limit_hit, lane);
        }
        for (;;) {                   // until a child is to be expanded: v == 2 level d is open, else node d's value
            if (v == 2) {
                const int m = pop(w.cand[d], lane);
                if (m < 0) {
                    v = w.kind[d] == KX ? 0 : 1;
                } else {
                    const int cv = vct_enter(w, g, d, m, empties, xnode, L, lane);
                    if (cv == 2) { ++d; break; }
                    v = settle(w.kind[d], cv);
                    continue;
                }
            }
            if (d == 0) return v;
            --d;
            vct_leave(w, d, empties, lane);
            v = settle(w.kind[d], v);
        }
    }
}

__device__ __forceinline__ Result vct_solve(VctWarp &w, const Geo &g, int max_attacks, int lane)
{
    int stones = 0;
    for (int k = 0; k < VW; ++k) stones += __popcll(w.bb[0][k]) + __popcll(w.bb[1][k]);
    const int empties = g.A - stones;
    const VScan s = vct_scan<false>(w, g, lane);
    if (s.n_x) return Result{1, 1, s.compl_x};
    if (max_attacks <= 1 || s.n_y >= 2) return Result{0, 1, 0ull};
    if (s.n_y == 0 && s.n_f2) return Result{2, 1, s.f2};
    const u64 cand = threat_moves(w, g, s, lane);
    if (lane < VW) w.root[lane] = cand;
    __syncwarp();
    int best = VCF_MAX_ATTACKS + 1, nodes = 1;
    u64 first = 0ull;
    for (int m; (m = pop(w.root, lane)) >= 0;) {
        put(w.bb[0], m, true, lane);
        bool wins = false;
        int len;
        for (len = 2; len <= max_attacks; ++len) {
            bool limit_hit = false;
            const int r = vct_search(w, g, len - 1, empties - 1, nodes, limit_hit, lane);
            if (r < 0) {
                put(w.bb[0], m, false, lane);
                return Result{-1, nodes, 0ull};
            }
            if (r > 0) { wins = true; break; }
            if (!limit_hit) break;
        }
        put(w.bb[0], m, false, lane);
        if (wins) {
            if (lane == (m >> 6)) first |= 1ull << (m & 63);
            best = min(best, len);
        }
    }
    return Result{best <= max_attacks ? best : 0, nodes, first};
}

__global__ void __launch_bounds__(VCF_WARPS * 32, 1)
k_vct(const int8_t *boards, const int8_t *players, int batch, Geo g, int max_attacks, int32_t *out_length, u64 *out_first,
      int32_t *out_nodes)
{
    __shared__ VctWarp sw[VCF_WARPS];
    const int lane = threadIdx.x & 31, b = blockIdx.x * VCF_WARPS + (threadIdx.x >> 5);
    if (b >= batch) return;
    VctWarp &w = sw[threadIdx.x >> 5];
    load(w, boards + (size_t)b * g.A, g.A, players[b] >= 0 ? 1 : -1, lane);
    const Result r = vct_solve(w, g, max_attacks, lane);
    if (lane < VW) out_first[(size_t)b * VW + lane] = r.first;
    if (lane == 0) { out_length[b] = r.length; out_nodes[b] = r.nodes; }
}

__global__ void __launch_bounds__(VCF_WARPS * 32, 1)
k_records_vct(const unsigned char *records, size_t stride, int n_records, Geo g, int max_attacks, uint8_t *out_flags)
{
    __shared__ VctWarp sw[VCF_WARPS];
    const int lane = threadIdx.x & 31, k = blockIdx.x * VCF_WARPS + (threadIdx.x >> 5);
    if (k >= n_records) return;
    VctWarp &w = sw[threadIdx.x >> 5];
    const unsigned char *rec = records + (size_t)k * stride;
    const gmz_move_record *h = rec_header(rec);
    const int action = h->action;
    load(w, rec_board(rec, g.A), g.A, h->to_move >= 0 ? 1 : -1, lane);
    const uint8_t f = record_flags(vct_solve(w, g, max_attacks, lane), action, g.A, lane);
    if (lane == 0) out_flags[k] = f;
}

}  // namespace

extern "C" int gmz_vcf_solve(const int8_t *boards, const int8_t *players, int batch, int board_size, int n_in_row,
                             int max_attacks, int node_budget, int32_t *out_length, uint64_t *out_first, int32_t *out_nodes,
                             gmz_stream stream)
{
    if (!boards || !players || !out_length || !out_first || !out_nodes) return gmz_fail("gmz_vcf_solve: null argument");
    if (const char *bad = check_limits(board_size, n_in_row, max_attacks, node_budget)) return gmz_fail("gmz_vcf_solve: %s", bad);
    if (batch < 0) return gmz_fail("gmz_vcf_solve: batch must be >= 0");
    if (batch == 0) return 0;
    const Geo g{board_size, board_size * board_size, n_in_row, node_budget};
    k_vcf<<<(unsigned)((batch + VCF_WARPS - 1) / VCF_WARPS), VCF_WARPS * 32, 0, (cudaStream_t)stream>>>(
        boards, players, batch, g, max_attacks, out_length, (u64 *)out_first, out_nodes);
    return gmz_check_launch("k_vcf");
}

extern "C" int gmz_records_vcf(const void *records, int64_t n_records, int board_size, int n_in_row, int max_attacks,
                               int node_budget, uint8_t *out_flags, gmz_stream stream)
{
    if (!records || !out_flags) return gmz_fail("gmz_records_vcf: null argument");
    if (const char *bad = check_limits(board_size, n_in_row, max_attacks, node_budget)) return gmz_fail("gmz_records_vcf: %s", bad);
    if (n_records < 0 || n_records > 0x7fffffff) return gmz_fail("gmz_records_vcf: n_records out of range");
    if (n_records == 0) return 0;
    const Geo g{board_size, board_size * board_size, n_in_row, node_budget};
    k_records_vcf<<<(unsigned)((n_records + VCF_WARPS - 1) / VCF_WARPS), VCF_WARPS * 32, 0, (cudaStream_t)stream>>>(
        (const unsigned char *)records, rec_stride(g.A), (int)n_records, g, max_attacks, out_flags);
    return gmz_check_launch("k_records_vcf");
}

extern "C" int gmz_vct_solve(const int8_t *boards, const int8_t *players, int batch, int board_size, int n_in_row,
                             int max_attacks, int node_budget, int32_t *out_length, uint64_t *out_first, int32_t *out_nodes,
                             gmz_stream stream)
{
    if (!boards || !players || !out_length || !out_first || !out_nodes) return gmz_fail("gmz_vct_solve: null argument");
    if (const char *bad = check_limits(board_size, n_in_row, max_attacks, node_budget)) return gmz_fail("gmz_vct_solve: %s", bad);
    if (batch < 0) return gmz_fail("gmz_vct_solve: batch must be >= 0");
    if (batch == 0) return 0;
    const Geo g{board_size, board_size * board_size, n_in_row, node_budget};
    k_vct<<<(unsigned)((batch + VCF_WARPS - 1) / VCF_WARPS), VCF_WARPS * 32, 0, (cudaStream_t)stream>>>(
        boards, players, batch, g, max_attacks, out_length, (u64 *)out_first, out_nodes);
    return gmz_check_launch("k_vct");
}

extern "C" int gmz_records_vct(const void *records, int64_t n_records, int board_size, int n_in_row, int max_attacks,
                               int node_budget, uint8_t *out_flags, gmz_stream stream)
{
    if (!records || !out_flags) return gmz_fail("gmz_records_vct: null argument");
    if (const char *bad = check_limits(board_size, n_in_row, max_attacks, node_budget)) return gmz_fail("gmz_records_vct: %s", bad);
    if (n_records < 0 || n_records > 0x7fffffff) return gmz_fail("gmz_records_vct: n_records out of range");
    if (n_records == 0) return 0;
    const Geo g{board_size, board_size * board_size, n_in_row, node_budget};
    k_records_vct<<<(unsigned)((n_records + VCF_WARPS - 1) / VCF_WARPS), VCF_WARPS * 32, 0, (cudaStream_t)stream>>>(
        (const unsigned char *)records, rec_stride(g.A), (int)n_records, g, max_attacks, out_flags);
    return gmz_check_launch("k_records_vct");
}
