// primitives.cuh -- hand-written device-wide building blocks: exclusive scan, stable LSD radix
// sort of (key, payload) pairs, index narrowing.  All run on ctx().stream.
#pragma once
#include "common.cuh"

namespace cpb {

// out[i] = sum_{t<i} in[i]  (u32, n entries).  in == out allowed.
void exclusive_scan_u32(const u32* in, u32* out, size_t n);

// Stable sort of (key, payload) by the low `bits` bits of key, 8 or 10 bits per pass.  Buffers are
// ping-ponged; returns 0 if the result is in (keys, vals), 1 if in (keys_tmp, vals_tmp).
int radix_sort_pairs(u32* keys, u32* vals, u32* keys_tmp, u32* vals_tmp, size_t n, int bits);
// same with payload = element index, generated on the fly (vals need not be initialised); the keys are read from the
// read-only keys_src in the first pass (keys is scratch and need not be initialised either)
int radix_sort_pairs_iota(const u32* keys_src, u32* keys, u32* vals, u32* keys_tmp, u32* vals_tmp, size_t n, int bits);

// dst[i] = (u32)(src[i] - 1); flags[0] |= 1 if any src[i] outside [lo, hi]
void narrow_minus1(const i64* src, u32* dst, size_t n, i64 lo, i64 hi, u32* flags);
void narrow32_minus1(const int* src, u32* dst, size_t n, i64 lo, i64 hi, u32* flags);  // the same from Int32 indices
// in place: v[i] -= 1; flags[0] |= 1 if any v[i] (before the decrement) outside [lo, hi]
void dec_check_u32(u32* v, size_t n, i64 lo, i64 hi, u32* flags);
// flags[0] |= 2 if pos is not non-decreasing
void check_monotone(const u32* pos, size_t n, u32* flags);
void iota_u32(u32* dst, size_t n);
// colidx[q] = 0-based column of nonzero q, from pos[0..ncol] (pos[ncol] == N)
void expand_columns(const u32* pos, u32 ncol, u32* colidx, size_t N);
// P[x] = first index p with keys[p] >= x, for x = 0..domain  (keys sorted ascending, P has domain+1 entries)
void segment_starts(const u32* sorted_keys, size_t n, u32* P, u32 domain);
// dst[i] = (i64)src[i] + add
void widen_plus(const u32* src, i64* dst, size_t n, i64 add);

int bits_for(u64 max_value);  // number of bits needed to represent max_value (>= 1)

}  // namespace cpb
