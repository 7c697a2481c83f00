// onesweep.cuh -- one-read-one-write radix passes on packed (key << 32 | payload) pairs and the link construction built
// on them (onesweep.cu).
#pragma once
#include "primitives.cuh"

namespace cpb {

// Stable sort of (keys[i] << 32 | i) by the low `bits` key bits, 0 < n < 2^31; a, b: n entries each (ping-pong); returns
// the one that holds the result.
u64* onesweep_sort_iota(const u32* keys, size_t n, int bits, u64* a, u64* b);

// prev[q] = link of nonzero q, 0 < N < 2^31, from row[q] (SparseColorArrays.jl:103-118 as a sort): 1 + q_off + position of the previous
// nonzero of the same row (as_pos) or 1 + its column (colidx), 0 if none.  first_count += number of zero links;
// last_local (optional, zero-initialised by the caller): last_local[r] = q_off + 1 + last position of row r.  Inputs of at
// least window_min nonzeros (0 = never) group the links by windows of `prev` before scattering.  Returns the sorted
// (row << 32 | position) pairs (in a or b).
u64* onesweep_links(const u32* row, size_t N, int row_bits, const u32* colidx, bool as_pos, u32 q_off, u32* prev, u32* first_count, u32* last_local,
                    size_t window_min, u64* a, u64* b);

}  // namespace cpb
