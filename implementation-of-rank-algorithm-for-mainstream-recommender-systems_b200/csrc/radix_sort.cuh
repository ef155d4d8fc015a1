// radix_sort.cuh — the multi-CTA LSD radix sort of plan_sort.cu (tile histogram, per-digit scan,
// stable scatter) on caller-given arrays, for library code other than rk_plan_build.
#pragma once
#include "common.cuh"

namespace rk {

// Scratch radix_sort_u32 needs for n pairs: one ping-pong pair of arrays plus the tile histograms.
size_t radix_sort_ws_bytes(int64_t n);

// Stable sort of (keys, vals) by the low `bits` bits of keys (1 <= bits <= 32), n < 2^31, into
// (keys_out, vals_out).  keys / vals are clobbered (they are the other half of the ping-pong);
// the outputs must not alias them.  Enqueued on `s`, no synchronisation, no allocation.
int radix_sort_u32(uint32_t* keys, uint32_t* vals, uint32_t* keys_out, uint32_t* vals_out, int64_t n,
                   int bits, void* ws, cudaStream_t s);

}  // namespace rk
