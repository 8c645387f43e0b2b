// gmz_tactics.cuh -- per-cell body of the reference's find_winning_moves_rebuilt (workers.py:49-123), shared by
// k_tactics (gmz_tactics.cu, a batch of boards) and k_records_tactics (gmz_records.cu, packed move records).
// Class of one cell for the side P (+-1) to move: 1 = 'five' (placing the stone wins, game.py:25-58), 2 = 'open_four',
// 3 = 'combo' (>= 2 blocked fours, blocked four + open three, or >= 2 open threes), 0 = none or occupied.
// Patterns are matched anywhere inside the 9-cell line centred on the move, off-board cells count as opponent
// stones, each pattern at most once per direction -- exactly as the reference does.
#pragma once
#include <stdint.h>

// sb: the N x N board (row-major, +1 / -1 / 0), normally in shared memory.
__device__ __forceinline__ int gmz_tactics_cell_class(const int8_t *sb, int N, int n_in_row, int P, int cell)
{
    if (sb[cell] != 0) return 0;
    const int O = -P;
    const int DR[4] = {0, 1, 1, 1}, DC[4] = {1, 0, 1, -1};
    const int r = cell / N, c = cell % N;
    bool five = false;
    int open_four = 0, blocked_four = 0, open_three = 0;
    for (int d = 0; d < 4; ++d) {
        // the 9-cell line as two bit masks (mine / empty), the stone placed at bit 4; everything else is a block
        unsigned mine = 0, empty = 0;
        for (int i = -4; i <= 4; ++i) {
            const int rr = r + i * DR[d], cc = c + i * DC[d];
            int v = O;
            if (rr >= 0 && rr < N && cc >= 0 && cc < N) v = (i == 0) ? P : sb[rr * N + cc];
            if (v == P) mine |= 1u << (i + 4); else if (v == 0) empty |= 1u << (i + 4);
        }
        // check_win with the stone placed: a contiguous run of n_in_row through (r,c).  For n_in_row <= 5 such a run
        // lies inside the 9-cell line: some window of n_in_row mine bits starting at bit 5-n_in_row .. 4.
        if (n_in_row >= 1 && n_in_row <= 5) {
            unsigned run = mine;
            for (int k = 1; k < n_in_row; ++k) run &= mine >> k;
            if (run & (0x1fu & ~((1u << (5 - n_in_row)) - 1u))) five = true;
        } else {                             // longer rows: walk the run up to n_in_row+1 each way, as the reference does
            int cnt = 1;
            for (int s = -1; s <= 1; s += 2)
                for (int i = 1; i < n_in_row + 2; ++i) {
                    const int rr = r + s * i * DR[d], cc = c + s * i * DC[d];
                    if (rr >= 0 && rr < N && cc >= 0 && cc < N && sb[rr * N + cc] == P) ++cnt; else break;
                }
            if (cnt >= n_in_row) five = true;
        }
        // the patterns at every offset i of the line at once (bit i of each mask = pattern starting at cell i)
        const unsigned block = ~(mine | empty) & 0x1ffu;
        const unsigned mid = (mine >> 1) & (mine >> 2) & (mine >> 3);                        // P,P,P at i+1..i+3
        open_four += (empty & (empty >> 5) & mid & (mine >> 4) & 0xfu) != 0;                 // (0,P,P,P,P,0)
        blocked_four += (mid & ((block & (empty >> 4)) | (empty & (block >> 4))) & 0x1fu) != 0;   // (X,P,P,P,0) / (0,P,P,P,X)
        open_three += (mid & empty & (empty >> 4) & 0x1fu) != 0;                             // (0,P,P,P,0)
    }
    if (five) return 1;
    if (open_four > 0) return 2;
    if (blocked_four >= 2 || (blocked_four >= 1 && open_three >= 1) || open_three >= 2) return 3;
    return 0;
}
