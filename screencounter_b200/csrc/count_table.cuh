// Device-side inserts into the count tables of libdev.hpp (random barcodes, sparse combinations): the GPU hash that
// replaces the reference's unordered_map<string, int> (handlers/RandomBarcodeSingleEnd.hpp:93-104) and its vector of
// combinations (handlers/CombinatorialBarcodesSingleEnd.hpp:188-199).  Shared by the nvcc-built and the run-time
// compiled kernels.
#pragma once

#include "libdev.hpp"

namespace scg {

// after this many probes an insert gives up and raises the table's overflow flag (the host sizes tables for a load
// factor of at most 1/2, where probe sequences are a handful of slots long)
constexpr unsigned long long COUNT_MAX_PROBES = 1ull << 16;

// Home of a key: an EVEN slot, so that the home and the slot after it share one aligned 32-byte sector -- a kernel that
// requested that sector ahead of time has, for most keys, everything it needs (bucketised linear probing, buckets of two).
__device__ __forceinline__ unsigned long long count_home(const CountTable64& t, unsigned long long key) {
    return count_hash(key) & t.mask & ~1ull;
}

// Adds `add` to the count of `key`, inserting it when new, starting at slot `pos` whose key was already seen as `seen`
// (callers that requested the slot earlier pass what they loaded; others pass the slot's current key).  Returns true
// when the key was new; the caller accounts for it in t.live[0] (count_insert64 does, one atomic per key; kernels that
// insert many keys add them up per warp first).
__device__ __forceinline__ bool count_insert64_from(const CountTable64& t, unsigned long long key, uint32_t add, unsigned long long pos,
                                                    unsigned long long seen) {
    bool fresh = false;
    for (unsigned long long probes = 0;; ++probes) {
        if (seen == key) break;
        if (seen == ~0ull) {
            const unsigned long long old = atomicCAS(&t.slots[pos].key, ~0ull, key);
            if (old == ~0ull) {
                fresh = true;
                break;
            }
            if (old == key) break;
        }
        if (probes >= COUNT_MAX_PROBES || probes > t.mask) {
            atomicExch(t.live + 1, 1ull);
            return false;
        }
        pos = (pos + 1) & t.mask;
        seen = __ldcg(&t.slots[pos].key);
    }
    atomicAdd(&t.slots[pos].count, add);
    return fresh;
}

__device__ __forceinline__ void count_insert64(const CountTable64& t, unsigned long long key, uint32_t add) {
    const unsigned long long pos = count_home(t, key);
    if (count_insert64_from(t, key, add, pos, __ldcg(&t.slots[pos].key))) atomicAdd(t.live, 1ull);
}

// 128-bit compare-and-swap (atom.cas.b128, sm_90+).
__device__ __forceinline__ ulonglong2 cas128(ulonglong2* addr, ulonglong2 expected, ulonglong2 desired) {
    ulonglong2 old;
    asm volatile(
        "{\n\t"
        ".reg .b128 e, d, o;\n\t"
        "mov.b128 e, {%2, %3};\n\t"
        "mov.b128 d, {%4, %5};\n\t"
        "atom.cas.b128 o, [%6], e, d;\n\t"
        "mov.b128 {%0, %1}, o;\n\t"
        "}"
        : "=l"(old.x), "=l"(old.y)
        : "l"(expected.x), "l"(expected.y), "l"(desired.x), "l"(desired.y), "l"(addr)
        : "memory");
    return old;
}

// Home of a 128-bit key: an EVEN slot, as count_home, so that the home and the slot after it are one aligned 32-byte sector
// of keys.  Every kernel that inserts into a wide table starts at this home and probes slot by slot from it.
__device__ __forceinline__ unsigned long long count_home128(const CountTable128& t, ulonglong2 key) {
    return count_hash(key.x ^ count_hash(key.y)) & t.mask & ~1ull;
}

// Adds `add` to the count of `key`, inserting it when new.  Returns true when the key was new; the caller accounts for it
// in t.live[0].
__device__ __forceinline__ bool count_add128(const CountTable128& t, ulonglong2 key, uint32_t add) {
    unsigned long long pos = count_home128(t, key);
    const ulonglong2 empty = make_ulonglong2(~0ull, ~0ull);
    bool fresh = false;
    for (unsigned long long probes = 0;; ++probes) {
        const ulonglong2 old = cas128(t.keys + pos, empty, key);
        if (old.x == ~0ull && old.y == ~0ull) {
            fresh = true;
            break;
        }
        if (old.x == key.x && old.y == key.y) break;
        if (probes >= COUNT_MAX_PROBES || probes > t.mask) {
            atomicExch(t.live + 1, 1ull);
            return false;
        }
        pos = (pos + 1) & t.mask;
    }
    atomicAdd(t.counts + pos, add);
    return fresh;
}

__device__ __forceinline__ void count_insert128(const CountTable128& t, ulonglong2 key, uint32_t add) {
    if (count_add128(t, key, add)) atomicAdd(t.live, 1ull);
}

__device__ __forceinline__ void combo_count(const ComboSink& k, int id0, int id1) {
    if (k.dense) {
        atomicAdd(k.dense + (size_t)id0 * k.n2 + id1, 1);
    } else {
        count_insert64(k.sparse, ((unsigned long long)(uint32_t)id0 << 32) | (uint32_t)id1, 1u);
    }
}

// packed key of a random barcode of up to 21 bases: H | L << 21 | N << 42 (bit i of a plane = base i)
__device__ __forceinline__ unsigned long long random_key64(uint32_t h, uint32_t l, uint32_t n) {
    return (unsigned long long)h | ((unsigned long long)l << 21) | ((unsigned long long)n << 42);
}

// packed key of a random barcode of 22 to 42 bases: the planes H, L, N (bit i = base i) in 42-bit fields of 128 bits,
// x = H | L << 42, y = L >> 22 | N << 20 (y < 2^62, so no key is the empty slot's (~0, ~0))
__device__ __forceinline__ ulonglong2 random_key128(unsigned long long h, unsigned long long l, unsigned long long n) {
    return make_ulonglong2(h | (l << 42), (l >> 22) | (n << 20));
}

} // namespace scg
