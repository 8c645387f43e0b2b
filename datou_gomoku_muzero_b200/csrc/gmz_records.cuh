// gmz_records.cuh -- the packed move record layout, shared by the translation units that read or write records
// (gmz_records.cu, and gmz_engine.cu for roots loaded from records).  The only place in C that knows where a field sits:
// kernels address a record through the accessors below.
// Record layout (gmz_move_record_bytes): header gmz_move_record | policy f64[A] | obs f32[3A] | board i8[A] | pad to 16.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include <type_traits>

#include "../../include/gmz.h"

static_assert(sizeof(gmz_move_record) == 64, "record header must be 64 bytes");
static_assert(offsetof(gmz_move_record, t) == 4 && offsetof(gmz_move_record, length) == 8 &&
              offsetof(gmz_move_record, winner) == 12 && offsetof(gmz_move_record, action) == 16 &&
              offsetof(gmz_move_record, to_move) == 20 && offsetof(gmz_move_record, last_move) == 24 &&
              offsetof(gmz_move_record, move_count) == 28 && offsetof(gmz_move_record, reward) == 32 &&
              offsetof(gmz_move_record, value_target) == 36 && offsetof(gmz_move_record, search_value) == 40 &&
              offsetof(gmz_move_record, opening) == 56,
              "gmz_move_record fields moved: the Python header dtype (trajectory.RECORD_HEADER) must move with them");

constexpr size_t REC_HEADER = sizeof(gmz_move_record);

// bytes of a record before its padding, and the record stride
__host__ __device__ __forceinline__ size_t rec_body(int A)
{
    return REC_HEADER + (sizeof(double) + 3 * sizeof(float) + sizeof(int8_t)) * (size_t)A;
}
__host__ __device__ __forceinline__ size_t rec_stride(int A) { return (rec_body(A) + 15) / 16 * 16; }

// T, const if the record bytes U are
template <class U, class T> using rec_ptr = typename std::conditional<std::is_const<U>::value, const T, T>::type *;

template <class U> __host__ __device__ __forceinline__ rec_ptr<U, gmz_move_record> rec_header(U *rec)
{
    return reinterpret_cast<rec_ptr<U, gmz_move_record>>(rec);
}
template <class U> __host__ __device__ __forceinline__ rec_ptr<U, double> rec_policy(U *rec)
{
    return reinterpret_cast<rec_ptr<U, double>>(rec + REC_HEADER);
}
template <class U> __host__ __device__ __forceinline__ rec_ptr<U, float> rec_obs(U *rec, int A)
{
    return reinterpret_cast<rec_ptr<U, float>>(rec + REC_HEADER + sizeof(double) * (size_t)A);
}
template <class U> __host__ __device__ __forceinline__ rec_ptr<U, int8_t> rec_board(U *rec, int A)
{
    return reinterpret_cast<rec_ptr<U, int8_t>>(rec + REC_HEADER + (sizeof(double) + 3 * sizeof(float)) * (size_t)A);
}

// Record k of a stretch of a ring of `capacity` records: ring position (first + k) % capacity.
template <class U> __host__ __device__ __forceinline__ U *rec_at(U *ring, size_t stride, int64_t capacity, int64_t first, int64_t k)
{
    return ring + (size_t)((first + k) % capacity) * stride;
}

// Copy a record header, one 32-bit word per lane (lanes below 16 copy).
__device__ __forceinline__ void rec_copy_header(unsigned char *dst, const unsigned char *src, int lane)
{
    if (lane < (int)(REC_HEADER / sizeof(uint32_t)))
        reinterpret_cast<uint32_t *>(dst)[lane] = reinterpret_cast<const uint32_t *>(src)[lane];
}

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
