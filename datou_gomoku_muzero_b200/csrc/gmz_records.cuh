// gmz_records.cuh -- the packed move record layout, shared by the translation units that read or write records
// (gmz_records.cu, and gmz_engine.cu for roots loaded from records).  Not part of the C ABI: include/gmz.h
// gmz_move_record is the public description of the same bytes.
// Record layout (gmz_move_record_bytes): 64-byte header | policy f64[A] | obs f32[3A] | board i8[A] | pad to 16.
#pragma once
#include <stddef.h>
#include <stdint.h>

struct RecHeader {            // 64 bytes, see include/gmz.h gmz_move_record
    int32_t game_seq, t, length, winner;
    int32_t action, to_move, last_move, move_count;
    float reward, value_target;
    double search_value;
    int32_t game, slot, opening, pad1;   // opening: book opening + 1, 0 = none
};
static_assert(sizeof(RecHeader) == 64, "record header must be 64 bytes");

static inline size_t rec_stride(int A) { return ((size_t)64 + (size_t)21 * A + 15) / 16 * 16; }

// A stretch of a ring of `capacity` records: record k at ring position (first + k) % capacity, k < n.  NULL if valid,
// else what is wrong with it.
static inline const char *rec_stretch_check(int64_t capacity, int64_t first, int64_t n)
{
    if (capacity < 1) return "capacity must be >= 1";
    if (n < 0) return "n must be >= 0";
    if (n > capacity) return "n exceeds the ring capacity";
    if (first < 0 || first >= capacity) return "first outside the ring [0, capacity)";
    return nullptr;
}
