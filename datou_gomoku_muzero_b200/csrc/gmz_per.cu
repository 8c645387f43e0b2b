// gmz_per.cu -- prioritized-replay SumTree kernels (reference replay_buffer.py:4-106).
//
// The reference applies priority updates one after another in Python; each update adds
// `change` to every ancestor (replay_buffer.py:11-19), so a tree node's float64 value depends
// on the ORDER its += arrive in.  To stay bit-exact the update kernel keeps that order while
// running every tree depth in parallel: warp d owns all nodes of depth d, walks the batch in
// order 32 updates at a time, groups lanes that hit the same node (__match_any_sync) and lets
// the group leader accumulate the group's changes in lane (= batch) order.
#include <math.h>
#include <stdint.h>

#include "gmz_internal.h"

#define PER_MAX_CHUNK 2048
// k_per_update's 32 warps own tree depths 0..31, so the deepest leaf may sit at depth 32: 2*capacity - 2 < 2^33 - 1.
#define PER_MAX_CAPACITY (1ll << 32)

__device__ __forceinline__ int node_depth(long long k) { return 63 - __clzll((unsigned long long)(k + 1)); }

// One CTA of 1024 threads (32 warps).  Stage 1 (warp 0): leaf writes and `change` per update,
// in batch order (a repeated leaf sees the previous write).  Stage 2 (warp d): depth-d ancestors.
// An index outside [0, len) is an inactive lane in both stages: it writes nothing.
__global__ void __launch_bounds__(1024)
k_per_update(double *tree, long long len, const long long *tree_idx, const double *prio, int n)
{
    extern __shared__ double s_change[];           // [n]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (warp == 0) {
        for (int base = 0; base < n; base += 32) {
            const int i = base + lane;
            const long long k = i < n ? tree_idx[i] : -1;
            const bool act = k >= 0 && k < len;
            const long long key = act ? k : -1 - lane;
            const double p = act ? prio[i] : 0.0;
            const unsigned grp = __match_any_sync(GMZ_FULL, key);
            const int leader = __ffs(grp) - 1;
            double cur = 0.0;
            if (act && lane == leader) cur = __ldcg(tree + key);
            cur = __shfl_sync(GMZ_FULL, cur, leader);
            // walk the group in lane order: change_b = p_b - cur; cur = p_b
            double my_change = 0.0, last = cur;
            for (int b = 0; b < 32; ++b) {
                const long long kb = __shfl_sync(GMZ_FULL, key, b);
                const double pb = __shfl_sync(GMZ_FULL, p, b);
                if (kb == key) {
                    if (b == lane) my_change = __dsub_rn(pb, last);
                    last = pb;
                }
            }
            if (act) {
                s_change[i] = my_change;
                if (lane == leader) __stcg(tree + key, last);   // value after the group's last write
            }
            __syncwarp();
        }
    }
    __syncthreads();
    const int d = warp;                              // this warp's tree depth (0 = root)
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        long long key = -1 - lane;
        double ch = 0.0;
        const long long leaf = i < n ? tree_idx[i] : -1;
        if (leaf >= 0 && leaf < len) {
            const int D = node_depth(leaf);
            if (D > d) { key = ((leaf + 1) >> (D - d)) - 1; ch = s_change[i]; }
        }
        const bool act = key >= 0;
        const unsigned grp = __match_any_sync(GMZ_FULL, key);
        if (__ballot_sync(GMZ_FULL, act) == 0) continue;
        const int leader = __ffs(grp) - 1;
        double acc = 0.0;
        if (act && lane == leader) acc = __ldcg(tree + key);
        if (__all_sync(GMZ_FULL, grp == (1u << lane))) {
            // every lane hits a different node (the common case away from the root): one += each
            if (act) acc = __dadd_rn(acc, ch);
        } else {
            // walk only the lanes that share a node with someone, in lane (= batch) order
            unsigned shared = __ballot_sync(GMZ_FULL, act && grp != (1u << lane));
            if (act && grp == (1u << lane)) acc = __dadd_rn(acc, ch);
            while (shared) {
                const int b = __ffs(shared) - 1; shared &= shared - 1;
                const long long kb = __shfl_sync(GMZ_FULL, key, b);
                const double cb = __shfl_sync(GMZ_FULL, ch, b);
                if (act && lane == leader && kb == key) acc = __dadd_rn(acc, cb);   // self.tree[parent] += change
            }
        }
        if (act && lane == leader) __stcg(tree + key, acc);
        __syncwarp();
    }
}

// InMemoryReplayBuffer.sample, PER branch (replay_buffer.py:60-86).  Single CTA: stratified
// draw + get_leaf descent per sample, then the batch-max normalisation of the IS weights.
__global__ void __launch_bounds__(1024)
k_per_sample(const double *tree, long long capacity, long long count, const double *u01, int B, double beta,
             long long *out_idx, double *out_prio, float *out_w)
{
    __shared__ float s_max[32];
    const long long len = 2 * capacity - 1;
    const double total = tree[0];
    const double segment = __ddiv_rn(total, (double)B);
    float lmax = -INFINITY;
    for (int i = threadIdx.x; i < B; i += blockDim.x) {
        const double lo = __dmul_rn(segment, (double)i), hi = __dmul_rn(segment, (double)(i + 1));
        double v = __dadd_rn(lo, __dmul_rn(__dsub_rn(hi, lo), u01[i]));   // np.random.uniform(lo, hi)
        long long parent = 0;
        for (;;) {                                                        // SumTree.get_leaf
            const long long left = 2 * parent + 1;
            if (left >= len) break;
            const double lv = tree[left];
            if (v <= lv) parent = left; else { v = __dsub_rn(v, lv); parent = left + 1; }
        }
        const double p = tree[parent];
        const double prob = __ddiv_rn(p, total);
        const float wgt = (float)pow(__dmul_rn((double)count, prob), -beta);
        out_idx[i] = parent; out_prio[i] = p; out_w[i] = wgt;
        lmax = fmaxf(lmax, wgt);
    }
    for (int o = 16; o > 0; o >>= 1) lmax = fmaxf(lmax, __shfl_xor_sync(GMZ_FULL, lmax, o));
    if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = lmax;
    __syncthreads();
    float m = (threadIdx.x & 31) < (blockDim.x >> 5) ? s_max[threadIdx.x & 31] : -INFINITY;
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(GMZ_FULL, m, o));
    if (m > 0.0f)
        for (int i = threadIdx.x; i < B; i += blockDim.x) out_w[i] = __fdiv_rn(out_w[i], m);
}

extern "C" int gmz_per_update(double *tree, int64_t capacity, const int64_t *tree_idx, const double *priorities, int n,
                              gmz_stream stream)
{
    if (!tree || !tree_idx || !priorities) return gmz_fail("gmz_per_update: null argument");
    if (capacity < 1 || capacity > PER_MAX_CAPACITY) return gmz_fail("gmz_per_update: capacity out of range (1 .. 2^32)");
    static bool attr_set = false;
    if (!attr_set) {
        cudaFuncSetAttribute(k_per_update, cudaFuncAttributeMaxDynamicSharedMemorySize, PER_MAX_CHUNK * (int)sizeof(double));
        attr_set = true;
    }
    for (int off = 0; off < n; off += PER_MAX_CHUNK) {     // chunks run in stream order = batch order
        const int m = n - off < PER_MAX_CHUNK ? n - off : PER_MAX_CHUNK;
        k_per_update<<<1, 1024, m * sizeof(double), (cudaStream_t)stream>>>(tree, 2 * capacity - 1, (const long long *)tree_idx + off,
                                                                           priorities + off, m);
    }
    return gmz_check_launch("k_per_update");
}

// SumTree.add for a batch (replay_buffer.py:21-25): leaf i goes to ring position (write_ptr + i) % capacity.
__global__ void k_per_add_idx(long long *idx, long long capacity, long long write_ptr, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) idx[i] = (write_ptr + i) % capacity + capacity - 1;
}

// Bulk add (n <= capacity consecutive ring positions, so no leaf repeats): the same bits as n sequential add()s, on
// the whole GPU.  A tree node's value after the batch is its old value with the `change`s of the batch leaves below
// it added ONE BY ONE IN BATCH ORDER (replay_buffer.py:11-19) -- and for consecutive ring positions those leaves are
// at most four runs of consecutive batch indices (two leaf levels of the heap x the ring's wrap-around).  So every
// internal node is independent: one thread per node folds its runs in order.  The root's fold is n dependent adds
// long (the floor bit-exactness sets); everything else hides under it.
__global__ void k_per_add_leaves(double *tree, long long capacity, long long write_ptr, const double *prio, int n, double *change)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long j = (write_ptr + i) % capacity + capacity - 1;
    const double p = prio[i];
    change[i] = __dsub_rn(p, tree[j]);          // change = priority - self.tree[tree_idx]
    tree[j] = p;
}
__global__ void k_per_add_nodes(double *tree, long long capacity, long long write_ptr, int n, const double *change)
{
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= capacity - 1) return;                // internal nodes only
    const int d = node_depth(k), Dmax = node_depth(2 * capacity - 2);
    long long rs[4], re[4];
    int nr = 0;
    for (int t = max(d, Dmax - 1); t <= Dmax; ++t) {          // the (at most two) levels that hold leaves
        long long lo = ((k + 1) << (t - d)) - 1, hi = ((k + 2) << (t - d)) - 2;
        if (t == Dmax) { lo = max(lo, (1ll << Dmax) - 1); hi = min(hi, 2 * capacity - 2); }
        else { lo = max(lo, capacity - 1); hi = min(hi, (1ll << Dmax) - 2); }
        if (lo > hi) continue;
        const long long plo = lo - (capacity - 1), phi = hi - (capacity - 1);      // ring positions under this node
        // batch index of ring position q: q - write_ptr (first part), q + capacity - write_ptr (after the wrap)
        const long long a0 = max(plo, write_ptr), a1 = min(phi, min(capacity - 1, write_ptr + n - 1));
        if (a0 <= a1) { rs[nr] = a0 - write_ptr; re[nr] = a1 - write_ptr; ++nr; }
        const long long wrapped = write_ptr + n - capacity;                        // positions 0 .. wrapped-1 come after the wrap
        const long long b0 = plo, b1 = min(phi, wrapped - 1);
        if (wrapped > 0 && b0 <= b1) { rs[nr] = b0 + capacity - write_ptr; re[nr] = b1 + capacity - write_ptr; ++nr; }
    }
    if (nr == 0) return;
    for (int a = 1; a < nr; ++a)                  // batch order
        for (int b = a; b > 0 && rs[b] < rs[b - 1]; --b) {
            const long long ts = rs[b], te = re[b]; rs[b] = rs[b - 1]; re[b] = re[b - 1]; rs[b - 1] = ts; re[b - 1] = te;
        }
    double acc = tree[k];
    for (int a = 0; a < nr; ++a) {
        long long i = rs[a];
        if (i + 15 <= re[a]) {                    // software pipeline: the next 16 changes load while these 16 are added, in order
            double c[16], nx[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) c[u] = __ldg(change + i + u);
            for (; i + 31 <= re[a]; i += 16) {
#pragma unroll
                for (int u = 0; u < 16; ++u) nx[u] = __ldg(change + i + 16 + u);
#pragma unroll
                for (int u = 0; u < 16; ++u) acc = __dadd_rn(acc, c[u]);
#pragma unroll
                for (int u = 0; u < 16; ++u) c[u] = nx[u];
            }
#pragma unroll
            for (int u = 0; u < 16; ++u) acc = __dadd_rn(acc, c[u]);
            i += 16;
        }
        for (; i <= re[a]; ++i) acc = __dadd_rn(acc, change[i]);   // self.tree[parent] += change
    }
    tree[k] = acc;
}

extern "C" int gmz_per_add(double *tree, int64_t capacity, int64_t write_ptr, const double *priorities, int n,
                           int64_t *scratch_idx, gmz_stream stream)
{
    if (!tree || !priorities || !scratch_idx) return gmz_fail("gmz_per_add: null argument");
    if (capacity < 1 || capacity > PER_MAX_CAPACITY) return gmz_fail("gmz_per_add: capacity out of range (1 .. 2^32)");
    if (n <= 0) return 0;
    if (write_ptr < 0 || write_ptr >= capacity) return gmz_fail("gmz_per_add: write_ptr outside the ring");
    if (n >= 64 && (int64_t)n <= capacity && capacity >= 2) {     // bulk path: node-parallel, whole GPU
        double *change = reinterpret_cast<double *>(scratch_idx);  // the caller's int64 [n] scratch, reused as float64 [n]
        k_per_add_leaves<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(tree, capacity, write_ptr, priorities, n, change);
        if (gmz_check_launch("k_per_add_leaves")) return 1;
        const long long nodes = capacity - 1;
        k_per_add_nodes<<<(unsigned)((nodes + 127) / 128), 128, 0, (cudaStream_t)stream>>>(tree, capacity, write_ptr, n, change);
        return gmz_check_launch("k_per_add_nodes");
    }
    k_per_add_idx<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>((long long *)scratch_idx, capacity, write_ptr, n);
    if (gmz_check_launch("k_per_add_idx")) return 1;
    return gmz_per_update(tree, capacity, scratch_idx, priorities, n, stream);
}

extern "C" int gmz_per_sample(const double *tree, int64_t capacity, int64_t count, const double *u01, int batch, double beta,
                              int64_t *out_tree_idx, double *out_priority, float *out_weights, gmz_stream stream)
{
    if (!tree || !u01 || !out_tree_idx || !out_priority || !out_weights) return gmz_fail("gmz_per_sample: null argument");
    if (capacity < 1 || capacity > PER_MAX_CAPACITY) return gmz_fail("gmz_per_sample: capacity out of range (1 .. 2^32)");
    if (batch <= 0) return 0;
    k_per_sample<<<1, 1024, 0, (cudaStream_t)stream>>>(tree, capacity, count, u01, batch, beta,
                                                        (long long *)out_tree_idx, out_priority, out_weights);
    return gmz_check_launch("k_per_sample");
}
