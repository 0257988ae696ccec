// Open-addressing table of int64 keys in device memory (linear probing, splitmix64 hash, -1 = empty slot), shared by the
// voxelizer (csrc/voxelize.cu) and the nearest-neighbour grid (csrc/nn_grid.cu).  capacity is a power of two; cap_mask =
// capacity - 1.  Keys are never removed, so a slot once set never changes.
#pragma once
#include "common.cuh"

namespace ps {

constexpr long long kEmptyKey = -1;

__device__ __forceinline__ uint64_t mix64(uint64_t k) {   // splitmix64 finaliser
    k ^= k >> 30; k *= 0xbf58476d1ce4e5b9ull;
    k ^= k >> 27; k *= 0x94d049bb133111ebull;
    k ^= k >> 31;
    return k;
}

// slot of `key` (inserted if absent; *fresh = it was absent), or -1 when the table is full
__device__ __forceinline__ long long table_insert(long long* __restrict__ keys, uint64_t cap_mask, long long key,
                                                  bool& fresh) {
    fresh = false;
    uint64_t s = mix64((uint64_t)key) & cap_mask;
    for (uint64_t probe = 0; probe <= cap_mask; ++probe) {
        const long long seen = __ldcg(keys + s);                   // a set key never changes: no atomic needed to skip it
        if (seen == key) return (long long)s;
        if (seen == kEmptyKey) {
            const long long prev = (long long)atomicCAS(reinterpret_cast<unsigned long long*>(keys + s),
                                                        (unsigned long long)kEmptyKey, (unsigned long long)key);
            if (prev == kEmptyKey) { fresh = true; return (long long)s; }
            if (prev == key) return (long long)s;
        }
        s = (s + 1) & cap_mask;
    }
    return -1;
}

// slot of `key`, or -1 when it is not in the table
__device__ __forceinline__ long long table_find(const long long* __restrict__ keys, uint64_t cap_mask, long long key) {
    uint64_t s = mix64((uint64_t)key) & cap_mask;
    for (uint64_t probe = 0; probe <= cap_mask; ++probe) {
        const long long seen = keys[s];
        if (seen == key) return (long long)s;
        if (seen == kEmptyKey) return -1;
        s = (s + 1) & cap_mask;
    }
    return -1;
}

}  // namespace ps
