// gmz_tactics.cu -- the reference's tactical move classifier find_winning_moves_rebuilt
// (workers.py:49-123) for a batch of boards: one CTA per board, one thread per cell.
// The per-cell classes (gmz_tactics_cell_class) are defined in gmz_tactics.cuh.
#include <stdint.h>

#include "../../include/gmz.h"
#include "gmz_common.cuh"
#include "gmz_tactics.cuh"

extern "C" void gmz_set_error_(const char *msg);

__global__ void __launch_bounds__(512)
k_tactics(const int8_t *boards, const int8_t *players, int N, int n_in_row, int8_t *out)
{
    __shared__ int8_t sb[GMZ_MAX_BOARD * GMZ_MAX_BOARD];
    const int A = N * N, b = blockIdx.x;
    for (int i = threadIdx.x; i < A; i += blockDim.x) sb[i] = boards[(size_t)b * A + i];
    __syncthreads();
    const int P = players[b] >= 0 ? 1 : -1;
    for (int cell = threadIdx.x; cell < A; cell += blockDim.x) {
        const int cls = gmz_tactics_cell_class(sb, N, n_in_row, P, cell);
        out[(size_t)b * A + cell] = (int8_t)cls;
    }
}

extern "C" int gmz_tactics_classify(const int8_t *boards, const int8_t *players, int batch, int board_size, int n_in_row,
                                    int8_t *out_cls, gmz_stream stream)
{
    if (!boards || !players || !out_cls) { gmz_set_error_("gmz_tactics_classify: null argument"); return 1; }
    if (batch <= 0) return 0;
    if (board_size < 1 || board_size > GMZ_MAX_BOARD) { gmz_set_error_("gmz_tactics_classify: board_size out of range"); return 1; }
    int threads = ((board_size * board_size + 31) / 32) * 32;
    if (threads > 512) threads = 512;
    k_tactics<<<batch, threads, 0, (cudaStream_t)stream>>>(boards, players, board_size, n_in_row, out_cls);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { gmz_set_error_(cudaGetErrorString(e)); return 1; }
    return 0;
}
