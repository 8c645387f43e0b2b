/* vcf_ref.c -- TEST INFRASTRUCTURE: a plain CPU restatement of the VCF solver include/gmz.h defines (gmz_vcf_solve),
 * written straight from the definition: an int8 board, recursion, and completion cells found by counting runs.  It is
 * the reference tests/test_vcf_*.py pin the CUDA solver against, node counts included. */
#include <stdint.h>
#include <string.h>

#define MAXA 361
#define MAX_ATTACKS 32

typedef struct {
    int N, A, n, budget;
    int nodes, limit_hit;
    int8_t b[MAXA];   /* +1 attacker, -1 defender, 0 empty */
} Ctx;

static const int DR[4] = {0, 1, 1, 1}, DC[4] = {1, 0, 1, -1};

/* stones of `who` in a row next to (r, c) in direction (dr, dc), not counting (r, c) */
static int run(const Ctx *x, int r, int c, int dr, int dc, int who)
{
    int k = 0;
    for (r += dr, c += dc; r >= 0 && r < x->N && c >= 0 && c < x->N && x->b[r * x->N + c] == who; r += dr, c += dc) ++k;
    return k;
}

/* an empty cell where a stone of `who` makes a run of >= n */
static int completion(const Ctx *x, int cell, int who)
{
    if (x->b[cell] != 0) return 0;
    const int r = cell / x->N, c = cell % x->N;
    for (int d = 0; d < 4; ++d)
        if (1 + run(x, r, c, DR[d], DC[d], who) + run(x, r, c, -DR[d], -DC[d], who) >= x->n) return 1;
    return 0;
}

/* number of completion cells of `who` (and the lowest), stopping at `cap` */
static int completions(const Ctx *x, int who, int cap, int *first)
{
    int k = 0;
    *first = -1;
    for (int a = 0; a < x->A && k < cap; ++a)
        if (completion(x, a, who)) {
            if (k == 0) *first = a;
            ++k;
        }
    return k;
}

/* The attacker's completion cells after its stone at m (already on the board), given it had none before: each lies on
 * one of the four lines through m, so those lines are scanned whole.  Returns their number (up to 2) and one of them. */
static int threats_after(const Ctx *x, int m, int *cell)
{
    const int r = m / x->N, c = m % x->N;
    int k = 0;
    *cell = -1;
    for (int d = 0; d < 4; ++d)
        for (int s = -1; s <= 1; s += 2)
            for (int i = 1; i < x->N; ++i) {
                const int rr = r + s * i * DR[d], cc = c + s * i * DC[d];
                if (rr < 0 || rr >= x->N || cc < 0 || cc >= x->N) break;
                if (completion(x, rr * x->N + cc, 1)) {
                    if (k == 0) *cell = rr * x->N + cc;
                    ++k;
                }
            }
    return k;
}

/* a four move: an empty cell after which the attacker has a completion cell.  For n >= 3 it needs an attacker stone
 * within n - 1 cells on one of its lines (the n cells that make the run hold m, the completion cell and n - 2 attacker
 * stones), which rules most cells out cheaply. */
static int four_move(Ctx *x, int m, int *cnt, int *cell)
{
    if (x->b[m] != 0) return 0;
    if (x->n >= 3) {
        const int r = m / x->N, c = m % x->N;
        int near = 0;
        for (int d = 0; d < 4 && !near; ++d)
            for (int s = -1; s <= 1 && !near; s += 2)
                for (int i = 1; i <= x->n - 1; ++i) {
                    const int rr = r + s * i * DR[d], cc = c + s * i * DC[d];
                    if (rr < 0 || rr >= x->N || cc < 0 || cc >= x->N) break;
                    if (x->b[rr * x->N + cc] == 1) { near = 1; break; }
                }
        if (!near) return 0;
    }
    x->b[m] = 1;
    *cnt = threats_after(x, m, cell);
    x->b[m] = 0;
    return *cnt > 0;
}

static int empties(const Ctx *x)
{
    int e = 0;
    for (int a = 0; a < x->A; ++a) e += x->b[a] == 0;
    return e;
}

/* The branch of candidate m (a four move with cnt completion cells, `cell` one of them): 1 = wins now (cnt >= 2), 0 =
 * fails (the reply makes the defender's run or fills the board), 2 = the reply is played (caller undoes m and cell). */
static int branch(Ctx *x, int m, int cnt, int cell)
{
    if (cnt >= 2) return 1;
    x->b[m] = 1;
    if (completion(x, cell, -1) || empties(x) == 1) { x->b[m] = 0; return 0; }
    x->b[cell] = -1;
    return 2;
}

/* vcf(board, L): 1 true, 0 false, -1 budget cut */
static int vcf(Ctx *x, int L)
{
    if (x->nodes == x->budget) return -1;
    x->nodes++;
    int y_cell, cell, cnt;
    if (completions(x, 1, 1, &cell)) return 1;
    if (L <= 1) { x->limit_hit = 1; return 0; }
    const int ny = completions(x, -1, 2, &y_cell);
    if (ny >= 2) return 0;
    for (int m = 0; m < x->A; ++m) {
        if (ny == 1 && m != y_cell) continue;
        if (!four_move(x, m, &cnt, &cell)) continue;
        const int br = branch(x, m, cnt, cell);
        if (br == 1) return 1;
        if (br == 0) continue;
        const int r = vcf(x, L - 1);
        x->b[m] = 0;
        x->b[cell] = 0;
        if (r != 0) return r;
    }
    return 0;
}

/* One position: board int8 [A] (values by sign), player the side to move.  first uint64 [6]. */
static void solve_one(Ctx *x, const int8_t *board, int player, int max_attacks, int32_t *length, uint64_t *first,
                      int32_t *nodes)
{
    const int P = player >= 0 ? 1 : -1;
    for (int a = 0; a < x->A; ++a) x->b[a] = board[a] == 0 ? 0 : ((board[a] > 0) == (P > 0) ? 1 : -1);
    memset(first, 0, 6 * sizeof(uint64_t));
    x->nodes = 1;
    *length = 0;
    int cell, cnt, y_cell;
    if (completions(x, 1, 1, &cell)) {
        for (int a = 0; a < x->A; ++a)
            if (completion(x, a, 1)) first[a >> 6] |= 1ull << (a & 63);
        *length = 1;
        *nodes = x->nodes;
        return;
    }
    const int ny = completions(x, -1, 2, &y_cell);
    int best = MAX_ATTACKS + 1;
    if (max_attacks >= 2 && ny < 2)
        for (int m = 0; m < x->A; ++m) {
            if (ny == 1 && m != y_cell) continue;
            if (!four_move(x, m, &cnt, &cell)) continue;
            const int br = branch(x, m, cnt, cell);
            int len = 2, wins = br == 1;
            if (br == 2) {
                for (len = 2; len <= max_attacks; ++len) {
                    x->limit_hit = 0;
                    const int r = vcf(x, len - 1);
                    if (r < 0) {
                        memset(first, 0, 6 * sizeof(uint64_t));
                        *length = -1;
                        *nodes = x->nodes;
                        return;
                    }
                    if (r > 0) { wins = 1; break; }
                    if (!x->limit_hit) break;
                }
                x->b[m] = 0;
                x->b[cell] = 0;
            }
            if (wins) {
                first[m >> 6] |= 1ull << (m & 63);
                if (len < best) best = len;
            }
        }
    *length = best <= max_attacks ? best : 0;
    *nodes = x->nodes;
}

/* The batch form of gmz_vcf_solve's arguments (host arrays); 0 or 1 for a refused argument. */
int vcf_ref_solve(const int8_t *boards, const int8_t *players, int batch, int board_size, int n_in_row, int max_attacks,
                  int node_budget, int32_t *length, uint64_t *first, int32_t *nodes)
{
    if (board_size < 1 || board_size > 19 || n_in_row < 1 || max_attacks < 1 || max_attacks > MAX_ATTACKS || node_budget < 1)
        return 1;
    const int A = board_size * board_size;
#pragma omp parallel for schedule(dynamic, 16)
    for (int i = 0; i < batch; ++i) {
        Ctx x;
        x.N = board_size; x.A = A; x.n = n_in_row; x.budget = node_budget; x.limit_hit = 0;
        solve_one(&x, boards + (size_t)i * A, players[i], max_attacks, length + i, first + (size_t)i * 6, nodes + i);
    }
    return 0;
}
