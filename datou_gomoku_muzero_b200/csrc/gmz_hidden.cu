// MuZero-mode hidden-state pool: one row per tree node, resident in HBM.
//
// The reference keeps `hidden_state` on every Node (mcts.py:21, 40-41) and ships it through two
// mp.Queue hops per recurrent batch (mcts.py:77-85, workers.py:357-369).  Here a row of the pool is the
// node's hidden state in NHWC order (A positions x C channels), and one simulation step moves
//   gather : x[g] = [ pool[row(parent_slot[g])] | action plane ]   -> the dynamics net's input
//   scatter: pool[row(child_slot[g])] = next_hidden[g]              <- the dynamics net's output
// Both are pure byte movement (SURVEY 8d: 2 * C * A * elt bytes per distinct evaluation), written as
// 16-byte vector copies with four loads in flight per thread; rows are independent, so the grid is
// (chunks per row, games).  The action plane is the dynamics net's one-hot action embedding
// (network.py:70-73: a 1x1 conv without bias of a one-hot plane == `embed` at the action's cell, zeros
// elsewhere), written by the same pass so the concatenated input is never built by a separate kernel.
#include <stdint.h>

#include "gmz_internal.h"

namespace {

constexpr int kThreads = 256, kUnroll = 8;

// engine slot g*S + node -> pool row g*nodes + node
__device__ __forceinline__ long long pool_row(int slot, int S, int nodes) { return (long long)(slot / S) * nodes + (slot % S); }

template <typename V> __device__ __forceinline__ V vzero();
template <> __device__ __forceinline__ uint4 vzero<uint4>() { return make_uint4(0u, 0u, 0u, 0u); }
template <> __device__ __forceinline__ uint2 vzero<uint2>() { return make_uint2(0u, 0u); }
template <> __device__ __forceinline__ unsigned vzero<unsigned>() { return 0u; }

// x row = A positions of (vin + ve) vectors; pool row = A positions of vin vectors.  V = the widest
// vector (16, 8 or 4 bytes) every size and pointer is a multiple of.
// CVIN / CVE: compile-time vector counts per position for the common shapes (the division by their sum
// then costs a multiply-high), 0 = take the run-time values.
template <typename V, int CVIN, int CVE>
__global__ void __launch_bounds__(kThreads)
k_hidden_gather(const V *__restrict__ pool, const int32_t *__restrict__ slot, const int32_t *__restrict__ action,
                int S, int nodes, int A, int vin_rt, int ve_rt, const V *__restrict__ embed, V *__restrict__ x)
{
    const int vin = CVIN ? CVIN : vin_rt, ve = CVIN ? CVE : ve_rt;
    const int g = blockIdx.y, s = slot[g], a = ve ? action[g] : -1;
    const int vo = vin + ve, total = A * vo;
    const V *src = pool + (s >= 0 ? pool_row(s, S, nodes) : 0) * (long long)A * vin;
    V *dst = x + (long long)g * total;
    const int base = blockIdx.x * (kThreads * kUnroll) + threadIdx.x;
    V v[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
        const int i = base + u * kThreads;
        v[u] = vzero<V>();
        if (i < total) {
            const int p = i / vo, q = i - p * vo;
            if (q < vin) { if (s >= 0) v[u] = __ldg(src + p * vin + q); }
            else if (p == a) v[u] = __ldg(embed + (q - vin));
        }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
        const int i = base + u * kThreads;
        if (i < total) dst[i] = v[u];
    }
}

template <typename V>
__global__ void __launch_bounds__(kThreads)
k_hidden_scatter(V *__restrict__ pool, const int32_t *__restrict__ slot, int S, int nodes, int total, const V *__restrict__ h)
{
    const int g = blockIdx.y, s = slot[g];
    if (s < 0) return;
    V *dst = pool + pool_row(s, S, nodes) * (long long)total;
    const V *src = h + (long long)g * total;
    const int base = blockIdx.x * (kThreads * kUnroll) + threadIdx.x;
    V v[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
        const int i = base + u * kThreads;
        if (i < total) v[u] = __ldg(src + i);
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
        const int i = base + u * kThreads;
        if (i < total) dst[i] = v[u];
    }
}

}  // namespace

template <typename V>
static void launch_gather(const void *pool, const int32_t *slot, const int32_t *action, int G, int S, int nodes, int A,
                          int pos_bytes, const void *embed, int embed_bytes, void *x, cudaStream_t st)
{
    const int vin = pos_bytes / (int)sizeof(V), ve = embed_bytes / (int)sizeof(V);
    const long long total = (long long)A * (vin + ve);
    dim3 grid((unsigned)((total + kThreads * kUnroll - 1) / (kThreads * kUnroll)), (unsigned)G);
    if (sizeof(V) == 16 && vin == 16 && ve == 2)        // 128 bf16 channels + 16-channel action embedding (GomokuNetEZ)
        k_hidden_gather<V, 16, 2><<<grid, kThreads, 0, st>>>((const V *)pool, slot, action, S, nodes, A, vin, ve, (const V *)embed, (V *)x);
    else if (sizeof(V) == 16 && vin == 16 && ve == 0)
        k_hidden_gather<V, 16, 0><<<grid, kThreads, 0, st>>>((const V *)pool, slot, action, S, nodes, A, vin, ve, (const V *)embed, (V *)x);
    else
        k_hidden_gather<V, 0, 0><<<grid, kThreads, 0, st>>>((const V *)pool, slot, action, S, nodes, A, vin, ve, (const V *)embed, (V *)x);
}

template <typename V>
static void launch_scatter(void *pool, const int32_t *slot, int G, int S, int nodes, int row_bytes, const void *h, cudaStream_t st)
{
    const int total = row_bytes / (int)sizeof(V);
    dim3 grid((unsigned)((total + kThreads * kUnroll - 1) / (kThreads * kUnroll)), (unsigned)G);
    k_hidden_scatter<V><<<grid, kThreads, 0, st>>>((V *)pool, slot, S, nodes, total, (const V *)h);
}

extern "C" int gmz_hidden_gather(const void *pool, const int32_t *slot, const int32_t *action, int num_games,
                                 int sims_per_game, int nodes_per_game, int positions, int pos_bytes,
                                 const void *embed, int embed_bytes, void *x, gmz_stream stream)
{
    if (!pool || !slot || !x) return gmz_fail("gmz_hidden_gather: null argument");
    if (embed_bytes && (!embed || !action)) return gmz_fail("gmz_hidden_gather: embed_bytes > 0 needs embed and action");
    if (num_games <= 0) return 0;
    if (sims_per_game < 1 || nodes_per_game < 1 || positions < 1 || pos_bytes < 4 || embed_bytes < 0)
        return gmz_fail("gmz_hidden_gather: sizes must be positive");
    const uintptr_t bits = (uintptr_t)pool | (uintptr_t)x | (uintptr_t)embed | (uintptr_t)pos_bytes | (uintptr_t)embed_bytes;
    if (bits & 3) return gmz_fail("gmz_hidden_gather: sizes and pointers must be multiples of 4 bytes");
    if ((long long)positions * (pos_bytes + embed_bytes) > (1ll << 30) || num_games > 65535)
        return gmz_fail("gmz_hidden_gather: row or batch too large");
    cudaStream_t st = (cudaStream_t)stream;
    if (!(bits & 15)) launch_gather<uint4>(pool, slot, action, num_games, sims_per_game, nodes_per_game, positions, pos_bytes, embed, embed_bytes, x, st);
    else if (!(bits & 7)) launch_gather<uint2>(pool, slot, action, num_games, sims_per_game, nodes_per_game, positions, pos_bytes, embed, embed_bytes, x, st);
    else launch_gather<unsigned>(pool, slot, action, num_games, sims_per_game, nodes_per_game, positions, pos_bytes, embed, embed_bytes, x, st);
    return gmz_check_launch("k_hidden_gather");
}

extern "C" int gmz_hidden_scatter(void *pool, const int32_t *slot, int num_games, int sims_per_game, int nodes_per_game,
                                  int row_bytes, const void *hidden, gmz_stream stream)
{
    if (!pool || !slot || !hidden) return gmz_fail("gmz_hidden_scatter: null argument");
    if (num_games <= 0) return 0;
    if (sims_per_game < 1 || nodes_per_game < 1 || row_bytes < 4) return gmz_fail("gmz_hidden_scatter: sizes must be positive");
    const uintptr_t bits = (uintptr_t)pool | (uintptr_t)hidden | (uintptr_t)row_bytes;
    if (bits & 3) return gmz_fail("gmz_hidden_scatter: row_bytes and pointers must be multiples of 4 bytes");
    if (num_games > 65535) return gmz_fail("gmz_hidden_scatter: batch too large");
    cudaStream_t st = (cudaStream_t)stream;
    if (!(bits & 15)) launch_scatter<uint4>(pool, slot, num_games, sims_per_game, nodes_per_game, row_bytes, hidden, st);
    else if (!(bits & 7)) launch_scatter<uint2>(pool, slot, num_games, sims_per_game, nodes_per_game, row_bytes, hidden, st);
    else launch_scatter<unsigned>(pool, slot, num_games, sims_per_game, nodes_per_game, row_bytes, hidden, st);
    return gmz_check_launch("k_hidden_scatter");
}
