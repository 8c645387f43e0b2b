// gmz_internal.h -- declarations shared by the translation units of libgmz.so (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include "../../include/gmz.h"
#include "gmz_common.cuh"

// The opening book self-play deals from (gmz_openings in include/gmz.h); n == 0: no book, deals are empty boards.
struct BookDev {
    int n, pad;
    const int8_t *boards;      // [n][A]
    const int8_t *players;     // [n]
    const int32_t *last_moves; // [n]
    const int32_t *move_counts;// [n]
};

struct gmz_engine {
    unsigned magic;          // GMZ_ENGINE_MAGIC while alive (gmz_destroy is idempotent per handle value)
    gmz_config cfg;
    Params p;
    int NC;
    int device;              // CUDA device the engine was created on
    size_t bytes;
    void *workspace;
    BookDev book;            // the bound opening book (n == 0: none)
};
#define GMZ_ENGINE_MAGIC 0x474d5a32u

// error text behind gmz_last_error() (thread-local, defined in gmz_engine.cu); both return 1
int gmz_fail(const char *fmt, const char *a = "");
int gmz_check_launch(const char *what);

// ticketed persistent play kernel, one translation unit per (MuZero mode, float32 accumulation)
struct PlayArgs;
int gmz_launch_play_mz0_f0(gmz_engine *e, const PlayArgs &a, cudaStream_t st);
int gmz_launch_play_mz0_f1(gmz_engine *e, const PlayArgs &a, cudaStream_t st);
int gmz_launch_play_mz1_f0(gmz_engine *e, const PlayArgs &a, cudaStream_t st);
int gmz_launch_play_mz1_f1(gmz_engine *e, const PlayArgs &a, cudaStream_t st);
