// gmz_vcf.cu -- forced wins: the VCF (victory by continuous fours) solver of include/gmz.h, for a batch of boards
// (k_vcf) and in place on packed move records (k_records_vcf).  The definition, the visiting order and the node count
// are those gmz.h states; tests/csrc/vcf_ref.c restates them on the CPU.
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
// after the run (possibly off the board).
__device__ __forceinline__ int run(const u64 *s, const Geo &g, int &r, int &c, int dr, int dc)
{
    int k = 0;
    r += dr; c += dc;
    while (k < g.n && r >= 0 && r < g.N && c >= 0 && c < g.N && has(s, r * g.N + c)) { ++k; r += dr; c += dc; }
    return k;
}

__device__ __forceinline__ bool empty_on_board(const VcfWarp &w, const Geo &g, int r, int c)
{
    if (r < 0 || r >= g.N || c < 0 || c >= g.N) return false;
    const int cell = r * g.N + c;
    return !has(w.bb[0], cell) && !has(w.bb[1], cell);
}

// direction d: (0, 1), (1, 0), (1, 1), (1, -1)
__device__ __forceinline__ int dir_r(int d) { return d != 0; }
__device__ __forceinline__ int dir_c(int d) { return d == 1 ? 0 : (d == 3 ? -1 : 1); }

// The attacker's completion cells an attacker stone at `cell` would add in direction d: the first non-attacker cell on
// each side, if it is empty and closes a run of >= n through `cell`.  Valid while the attacker has no completion
// cell (then every new one lies on a line through `cell`, next to the run that holds it).
__device__ __forceinline__ void four_ends(const VcfWarp &w, const Geo &g, int cell, int d, bool &okL, int &eL, bool &okR,
                                          int &eR)
{
    const int r = cell / g.N, c = cell % g.N, dr = dir_r(d), dc = dir_c(d);
    int rl = r, cl = c, rr = r, cr = c;
    const int aL = run(w.bb[0], g, rl, cl, -dr, -dc), aR = run(w.bb[0], g, rr, cr, dr, dc);
    okL = okR = false;
    eL = rl * g.N + cl; eR = rr * g.N + cr;
    if (empty_on_board(w, g, rl, cl)) { int r2 = rl, c2 = cl; okL = 2 + aL + aR + run(w.bb[0], g, r2, c2, -dr, -dc) >= g.n; }
    if (empty_on_board(w, g, rr, cr)) { int r2 = rr, c2 = cr; okR = 2 + aL + aR + run(w.bb[0], g, r2, c2, dr, dc) >= g.n; }
}

// Does a stone of side s (0 attacker, 1 defender) on the empty `cell` make a run of >= n?
__device__ __forceinline__ bool completes(const VcfWarp &w, const Geo &g, int s, int cell, int d)
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

// The attacker's completion cells after it plays the four move m: their number, and the cell when there is one.
__device__ int threats(const VcfWarp &w, const Geo &g, int m, int lane, int &cell)
{
    bool okL = false, okR = false;
    int eL = -1, eR = -1;
    if (lane < 4) four_ends(w, g, m, lane, okL, eL, okR, eR);
    const int cnt = __reduce_add_sync(GMZ_FULL, (int)okL + (int)okR);
    const unsigned who = __ballot_sync(GMZ_FULL, okL || okR);
    cell = who ? __shfl_sync(GMZ_FULL, okL ? eL : eR, __ffs(who) - 1) : -1;
    return cnt;
}

// Does the defender's stone on `cell` make a run of >= n (attacker's move already on the board)?
__device__ __forceinline__ bool defender_completes(const VcfWarp &w, const Geo &g, int cell, int lane)
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
__device__ void load(VcfWarp &w, const int8_t *board, int A, int P, int lane)
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
    const Result r = solve(w, g, max_attacks, lane);
    const bool played = __any_sync(GMZ_FULL, action >= 0 && action < g.A && lane == (action >> 6) &&
                                                 ((r.first >> (action & 63)) & 1ull));
    if (lane == 0) out_flags[k] = (uint8_t)((r.length > 0 ? 1 : 0) | (played ? 2 : 0) | (r.length < 0 ? 4 : 0));
}

const char *check_limits(int board_size, int n_in_row, int max_attacks, int node_budget)
{
    if (board_size < 1 || board_size > GMZ_MAX_BOARD) return "board_size out of range";
    if (n_in_row < 1) return "n_in_row must be >= 1";
    if (max_attacks < 1 || max_attacks > VCF_MAX_ATTACKS) return "max_attacks must be in [1, 32]";
    if (node_budget < 1) return "node_budget must be >= 1";
    return nullptr;
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
