// gmz_play_inst.cu -- one instantiation family of the persistent play kernel k_play_e0<NC, MZ, F32>.
// Compiled four times (-DGMZ_PLAY_MZ=0|1 -DGMZ_PLAY_F32=0|1) so the big kernels build in parallel.
#include "gmz_internal.h"
#include "gmz_tree.cuh"
#include "gmz_play.cuh"

#if !defined(GMZ_PLAY_MZ) || !defined(GMZ_PLAY_F32)
#error "compile with -DGMZ_PLAY_MZ=0|1 -DGMZ_PLAY_F32=0|1"
#endif
#define GMZ_CAT_(a, b, c, d) a##b##c##d
#define GMZ_CAT(a, b, c, d) GMZ_CAT_(a, b, c, d)
#define GMZ_LAUNCH_NAME GMZ_CAT(gmz_launch_play_mz, GMZ_PLAY_MZ, _f, GMZ_PLAY_F32)

// grid = what fits on the GPU at once (persistent), capped by the game count.  The occupancy is a
// property of (device, NC) for this translation unit's (MZ, F32): cached per device, filled under a mutex.
#include <mutex>
#include <stdlib.h>
template <int NC>
static int launch_t(gmz_engine *e, const PlayArgs &a, cudaStream_t st)
{
    constexpr bool MZ = GMZ_PLAY_MZ != 0, F32 = GMZ_PLAY_F32 != 0;
    static std::mutex mu;
    static int cache[64];                    // resident CTAs per device ordinal, 0 = unknown
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return gmz_fail("cudaGetDevice failed");
    int resident = 0;
    {
        std::lock_guard<std::mutex> lk(mu);
        if (dev >= 0 && dev < 64) resident = cache[dev];
        if (!resident) {
            int occ = 0, sms = 0;
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_play_e0<NC, MZ, F32>, 32 * GMZ_PLAY_WARPS, 0);
            resident = (occ > 0 ? occ : 1) * (sms > 0 ? sms : 148);
            if (dev >= 0 && dev < 64) cache[dev] = resident;
        }
    }
    int grid = (e->p.G + GMZ_PLAY_WARPS - 1) / GMZ_PLAY_WARPS;
    if (grid > resident) grid = resident;
    if (const char *cap = getenv("GMZ_PLAY_GRID_CAP")) { const int c = atoi(cap); if (c > 0 && c < grid) grid = c; }   // development: occupancy sweeps
    if (cudaMemsetAsync(&e->p.ctl->next_ticket, 0, 2 * sizeof(unsigned long long), st) != cudaSuccess) return gmz_fail("cudaMemsetAsync(ctl)");
    k_play_e0<NC, MZ, F32><<<grid, 32 * GMZ_PLAY_WARPS, 0, st>>>(e->p, a);
    return gmz_check_launch("k_play_e0");
}

int GMZ_LAUNCH_NAME(gmz_engine *e, const PlayArgs &a, cudaStream_t st)
{
    switch (e->NC) {
        case 1: return launch_t<1>(e, a, st);
        case 2: return launch_t<2>(e, a, st);
        default: return launch_t<3>(e, a, st);
    }
}
