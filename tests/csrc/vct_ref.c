/* vct_ref.c -- TEST INFRASTRUCTURE: a plain CPU restatement of the VCT solver include/gmz.h defines (gmz_vct_solve),
 * written straight from the definition: an int8 board, recursion, and completion cells found by counting runs.  It
 * reuses vcf_ref.c's board helpers and has two modes that must agree on length, first and nodes:
 *   brute force -- every four move, three move, F2, D and K set is found by placing a stone and rescanning the whole
 *                  board;
 *   filtered    -- the same sets through the board-level facts the CUDA kernel relies on (stated where they are used).
 * tests/test_vct_cpu.py pins the two against each other; tests/test_vct_gpu.py pins the kernel against this file. */
#include "vcf_ref.c"

typedef struct {
    Ctx x;
    int filtered;
} V;

/* X's completion cells after an X stone at the empty f (taken back), capped at 2: brute force rescans the board;
 * filtered scans f's four lines only (valid while X has no completion cell: a new one is on a run through f). */
static int compl_after_x(V *v, int f)
{
    Ctx *x = &v->x;
    int cell;
    x->b[f] = 1;
    const int k = v->filtered ? threats_after(x, f, &cell) : completions(x, 1, 2, &cell);
    x->b[f] = 0;
    return k;
}

/* F2: the empty cells f where an X stone leaves >= 2 completion cells (X has none).  Returns their number capped at 2,
 * and the lowest. */
static int f2_cells(V *v, int *lowest)
{
    int k = 0;
    *lowest = -1;
    for (int f = 0; f < v->x.A && k < 2; ++f)
        if (v->x.b[f] == 0 && compl_after_x(v, f) >= 2) {
            if (k == 0) *lowest = f;
            ++k;
        }
    return k;
}

/* Is the empty m (X has no completion cell) a threat move of X: a four move, or a three move -- X@m leaves no
 * completion cell but a non-empty F2?  f2_n / f2_low describe F2 of the board without m. */
static int threat_move(V *v, int m, int f2_n, int f2_low)
{
    Ctx *x = &v->x;
    if (x->b[m] != 0) return 0;
    int cnt, cell;
    if (v->filtered) {
        if (four_move(x, m, &cnt, &cell)) return 1;
    } else {
        x->b[m] = 1;
        const int four = completions(x, 1, 1, &cell) > 0;
        x->b[m] = 0;
        if (four) return 1;
    }
    int three = 0;
    x->b[m] = 1;
    if (!v->filtered) {
        int low;
        three = f2_cells(v, &low) > 0;
    } else {
        /* Fact 2.  An X stone never removes an X completion cell except the cell it lands on, so the count of every
         * f rises or stays; it can stay only at m itself if m completed B+X@f, and then f would complete B+X@m, a
         * four.  So F2(B) minus m stays in F2(B+X@m).  A cell f gains only through a new completion cell e whose run
         * holds m, f and e; two cells share one line, so only f's count along the line through m and f changes, and
         * the cells strictly between m and f are X stones or e, so f is within n - 1 of m on one of m's four lines
         * (were it farther, the cells from f up to m minus one would already be a run of n with e, or f would
         * complete B). */
        three = f2_n >= 2 || (f2_n == 1 && f2_low != m);
        const int r = m / x->N, c = m % x->N;
        for (int d = 0; d < 4 && !three; ++d)
            for (int s = -1; s <= 1 && !three; s += 2)
                for (int i = 1; i <= x->n - 1; ++i) {
                    const int rr = r + s * i * DR[d], cc = c + s * i * DC[d];
                    if (rr < 0 || rr >= x->N || cc < 0 || cc >= x->N) break;
                    const int f = rr * x->N + cc;
                    if (x->b[f] == 0 && compl_after_x(v, f) >= 2) { three = 1; break; }
                }
    }
    x->b[m] = 0;
    return three;
}

/* Is the empty d a defence of Y: after Y@d, X has no completion cell and F2 is empty? */
static int defence(V *v, int d)
{
    Ctx *x = &v->x;
    int low, cell;
    x->b[d] = -1;
    const int ok = (v->filtered || completions(x, 1, 1, &cell) == 0) && f2_cells(v, &low) == 0;
    x->b[d] = 0;
    return ok;
}

/* Fact 1.  A Y stone at d lowers f's count only by filling f or one of the completion cells of B+X@f: the other cells
 * of those runs are X stones.  So a defence lies on a cell of F2 or on a completion cell of B+X@f for some f in F2. */
static int defence_candidate(V *v, int d)
{
    Ctx *x = &v->x;
    const int r = d / x->N, c = d % x->N;
    if (x->b[d] != 0) return 0;
    if (compl_after_x(v, d) >= 2) return 1;
    /* d completes B+X@f: f is on one of d's lines; try each F2 cell there */
    for (int k = 0; k < 4; ++k)
        for (int s = -1; s <= 1; s += 2)
            for (int i = 1; i < x->N; ++i) {
                const int rr = r + s * i * DR[k], cc = c + s * i * DC[k];
                if (rr < 0 || rr >= x->N || cc < 0 || cc >= x->N) break;
                const int f = rr * x->N + cc;
                if (x->b[f] != 0 || compl_after_x(v, f) < 2) continue;
                x->b[f] = 1;
                const int hit = completion(x, d, 1);
                x->b[f] = 0;
                if (hit) return 1;
            }
    return 0;
}

/* Is the empty k a counter-four of Y: after Y@k, Y has a completion cell (it has none before)? */
static int counter_four(V *v, int k)
{
    Ctx *x = &v->x;
    int cell, n;
    x->b[k] = -1;
    if (v->filtered) {          /* Y's new completion cells lie on k's lines (the VCF fact, for Y) */
        for (int a = 0; a < x->A; ++a) x->b[a] = -x->b[a];
        n = threats_after(x, k, &cell);
        for (int a = 0; a < x->A; ++a) x->b[a] = -x->b[a];
    } else {
        n = completions(x, -1, 1, &cell);
    }
    x->b[k] = 0;
    return n > 0;
}

static int ynode(V *v, int L);

/* xnode(B, L), X to move: 1 true, 0 false, -1 budget cut */
static int xnode(V *v, int L)
{
    Ctx *x = &v->x;
    if (x->nodes == x->budget) return -1;
    x->nodes++;
    int cell, y_cell, f2_low;
    if (completions(x, 1, 1, &cell)) return 1;
    if (L <= 1) { x->limit_hit = 1; return 0; }
    const int ny = completions(x, -1, 2, &y_cell);
    const int nf = f2_cells(v, &f2_low);
    if (ny == 0 && nf > 0) return 1;
    if (ny >= 2) return 0;
    for (int m = 0; m < x->A; ++m) {
        if (ny == 1 && m != y_cell) continue;
        if (!threat_move(v, m, nf, f2_low)) continue;
        x->b[m] = 1;
        const int r = ynode(v, L - 1);
        x->b[m] = 0;
        if (r != 0) return r;
    }
    return 0;
}

/* ynode(B, L), Y to move, Y has no completion cell */
static int ynode(V *v, int L)
{
    Ctx *x = &v->x;
    if (x->nodes == x->budget) return -1;
    x->nodes++;
    int c, f2_low;
    const int nx = completions(x, 1, 2, &c);
    if (nx >= 2) return 1;
    if (nx == 1) {
        if (completion(x, c, -1) || empties(x) == 1) return 0;
        x->b[c] = -1;
        const int r = xnode(v, L);
        x->b[c] = 0;
        return r;
    }
    if (f2_cells(v, &f2_low) == 0) return 0;
    if (L < 2) { x->limit_hit = 1; return 0; }
    for (int r = 0; r < x->A; ++r) {
        if (x->b[r] != 0) continue;
        const int in_d = v->filtered ? defence_candidate(v, r) && defence(v, r) : defence(v, r);
        if (!in_d && !counter_four(v, r)) continue;
        x->b[r] = -1;
        int res, yc;
        if (empties(x) == 0) res = 0;
        else {
            const int ny = completions(x, -1, 2, &yc);
            if (ny >= 2) res = 0;
            else if (ny == 1) {
                x->b[yc] = 1;
                res = empties(x) == 0 ? 0 : ynode(v, L - 1);
                x->b[yc] = 0;
            } else {
                res = xnode(v, L);
            }
        }
        x->b[r] = 0;
        if (res <= 0) return res;
    }
    return 1;
}

static void vct_one(V *v, const int8_t *board, int player, int max_attacks, int32_t *length, uint64_t *first,
                    int32_t *nodes)
{
    Ctx *x = &v->x;
    const int P = player >= 0 ? 1 : -1;
    for (int a = 0; a < x->A; ++a) x->b[a] = board[a] == 0 ? 0 : ((board[a] > 0) == (P > 0) ? 1 : -1);
    memset(first, 0, 6 * sizeof(uint64_t));
    x->nodes = 1;
    *length = 0;
    int cell, y_cell, f2_low;
    if (completions(x, 1, 1, &cell)) {
        for (int a = 0; a < x->A; ++a)
            if (completion(x, a, 1)) first[a >> 6] |= 1ull << (a & 63);
        *length = 1;
        *nodes = x->nodes;
        return;
    }
    if (max_attacks <= 1) { *nodes = x->nodes; return; }
    const int ny = completions(x, -1, 2, &y_cell);
    const int nf = f2_cells(v, &f2_low);
    if (ny == 0 && nf > 0) {
        for (int f = 0; f < x->A; ++f)
            if (x->b[f] == 0 && compl_after_x(v, f) >= 2) first[f >> 6] |= 1ull << (f & 63);
        *length = 2;
        *nodes = x->nodes;
        return;
    }
    int best = MAX_ATTACKS + 1;
    if (ny < 2)
        for (int m = 0; m < x->A; ++m) {
            if (ny == 1 && m != y_cell) continue;
            if (!threat_move(v, m, nf, f2_low)) continue;
            x->b[m] = 1;
            int len, wins = 0;
            for (len = 2; len <= max_attacks; ++len) {
                x->limit_hit = 0;
                const int r = ynode(v, len - 1);
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
            if (wins) {
                first[m >> 6] |= 1ull << (m & 63);
                if (len < best) best = len;
            }
        }
    *length = best <= max_attacks ? best : 0;
    *nodes = x->nodes;
}

/* The batch form of gmz_vct_solve's arguments (host arrays), in brute-force (filtered = 0) or filtered mode; 0 or 1
 * for a refused argument. */
int vct_ref_solve(const int8_t *boards, const int8_t *players, int batch, int board_size, int n_in_row, int max_attacks,
                  int node_budget, int filtered, int32_t *length, uint64_t *first, int32_t *nodes)
{
    if (board_size < 1 || board_size > 19 || n_in_row < 1 || max_attacks < 1 || max_attacks > MAX_ATTACKS || node_budget < 1)
        return 1;
    const int A = board_size * board_size;
#pragma omp parallel for schedule(dynamic, 4)
    for (int i = 0; i < batch; ++i) {
        V v;
        v.x.N = board_size; v.x.A = A; v.x.n = n_in_row; v.x.budget = node_budget; v.x.limit_hit = 0;
        v.filtered = filtered;
        vct_one(&v, boards + (size_t)i * A, players[i], max_attacks, length + i, first + (size_t)i * 6, nodes + i);
    }
    return 0;
}

/* The candidate sets of one position, for the hand-built tests (board +1 = X, -1 = Y, X without a completion cell):
 * threats = X's threat moves as xnode step 5 takes them, replies = Y's R = D | K as ynode step 5 builds it (meaningful
 * when F2 is non-empty and Y has no completion cell).  uint64 [6] each. */
void vct_ref_sets(const int8_t *board, int board_size, int n_in_row, int filtered, uint64_t *threats, uint64_t *replies)
{
    V v;
    v.x.N = board_size; v.x.A = board_size * board_size; v.x.n = n_in_row; v.x.budget = 1; v.x.nodes = 0;
    v.filtered = filtered;
    memcpy(v.x.b, board, (size_t)v.x.A);
    memset(threats, 0, 6 * sizeof(uint64_t));
    memset(replies, 0, 6 * sizeof(uint64_t));
    int y_cell, f2_low;
    const int ny = completions(&v.x, -1, 2, &y_cell);
    const int nf = f2_cells(&v, &f2_low);
    for (int m = 0; m < v.x.A; ++m) {
        if ((ny == 0 || m == y_cell) && threat_move(&v, m, nf, f2_low)) threats[m >> 6] |= 1ull << (m & 63);
        if (v.x.b[m] == 0 && ((filtered ? defence_candidate(&v, m) && defence(&v, m) : defence(&v, m)) || counter_four(&v, m)))
            replies[m >> 6] |= 1ull << (m & 63);
    }
}
