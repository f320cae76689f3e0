// prims.cuh — small device-wide primitives written for this engine (no CUB/Thrust):
// exclusive scan, bitmap → ordered index list, stable LSD radix sort of (u32 key, u32 value).
// They implement what the reference gets from BTreeSet / Vec ordering on the CPU
// (common/witness.rs:10,30-32; proofs/generator.rs:34,85-88; events/utils.rs:56-91).
#pragma once
#include "common.cuh"

namespace ipcfp {

// out[i] = sum_{j<i} in[j] (u64 accumulators); *total_dev (device u64) receives the grand total.
// scratch must hold scan_scratch_elems(n) u64. fixed_launches: the same two launches for every n ≥ 1 up to 16.7 M (no one-CTA
// shortcut for small n), for callers whose launch count must not depend on the size.
size_t scan_scratch_elems(uint64_t n);
void exclusive_scan_u32(const uint32_t* in, uint64_t* out, uint64_t n, uint64_t* total_dev, uint64_t* scratch, cudaStream_t st,
                        bool fixed_launches = false);

// Ordered list of set-bit positions of a bitmap of nbits bits (nbits rounded up to 32 must be allocated).
// word_prefix: u64[nwords] scratch. out: u32[≥ popcount]. *total_dev receives the count.
void bitmap_to_indices(const uint32_t* bits, uint64_t nbits, uint32_t* out, uint64_t* total_dev, uint64_t* word_prefix,
                       uint64_t* scratch, cudaStream_t st, bool fixed_launches = false);

// Stable radix sort of n (key,val) pairs by the `nbits` low bits of key (8-bit digits, LSD).
// keys/vals are sorted in place using the alt buffers as ping-pong space.
// hist: u32[256 * radix_blocks(n) + 256] scratch.
unsigned radix_blocks(uint64_t n);
void radix_sort_pairs(uint32_t* keys, uint32_t* vals, uint32_t* keys_alt, uint32_t* vals_alt, uint64_t n, int nbits,
                      uint32_t* hist, uint64_t* scan_tmp, uint64_t* scratch, cudaStream_t st);

}  // namespace ipcfp
