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

// ---- keys of three words or more (CountTableLong) ----
// tag: bits 34..63 the key's fingerprint (the top bits of its hash), bit 33 set in every occupied slot, bit 32 while the key
// is FRESH (its words are still in the staging row of bits 0..31)
constexpr unsigned long long LONG_PRINT = ~((1ull << 34) - 1);
constexpr unsigned long long LONG_OCCUPIED = 1ull << 33;
constexpr unsigned long long LONG_FRESH = 1ull << 32;
constexpr unsigned long long LONG_ROW = 0xFFFFFFFFull;

// hash of a key word by word (long_hash_step over the words from a seed of 0, then long_hash_final)
__device__ __forceinline__ unsigned long long long_hash_step(unsigned long long h, unsigned long long word) {
    h = (h ^ word) * 0x9E3779B97F4A7C15ull;
    return h ^ (h >> 29);
}
__device__ __forceinline__ unsigned long long long_hash_final(unsigned long long h) {
    h = (h ^ (h >> 32)) * 0xD6E8FEB86659FD93ull;
    return h ^ (h >> 32);
}
__device__ __forceinline__ unsigned long long long_key_hash(const unsigned long long* key, int words) {
    unsigned long long h = 0;
    for (int w = 0; w < words; ++w) h = long_hash_step(h, key[w]);
    return long_hash_final(h);
}

// a tag as every thread of the grid sees it (no stale copy in L1)
__device__ __forceinline__ unsigned long long load_tag(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ bool long_rows_equal(const unsigned long long* a, const unsigned long long* b, int words) {
    for (int w = 0; w < words; ++w) {
        if (__ldcg(a + w) != __ldcg(b + w)) return false;
    }
    return true;
}

// Adds `add` to the count of the key in staging row `row` (hash h), claiming a slot when the key is new (*fresh).  Returns the
// slot, or ~0 when the probe limit was reached (the overflow flag is raised and nothing is counted).  The row must have been
// written and fenced (__threadfence) before the call: a claim publishes it to every other thread.
__device__ __forceinline__ unsigned long long count_add_long(const CountTableLong& t, unsigned long long h, unsigned long long row, uint32_t add,
                                                             bool& fresh) {
    const unsigned long long words = (unsigned long long)t.words;
    const unsigned long long* own = t.staging + row * words;
    const unsigned long long print = h & LONG_PRINT;
    unsigned long long pos = h & t.mask & ~1ull;
    fresh = false;
    for (unsigned long long probes = 0;; ++probes) {
        unsigned long long tag = load_tag(t.tags + pos);
        if (tag == 0) {
            tag = atomicCAS(t.tags + pos, 0ull, print | LONG_OCCUPIED | LONG_FRESH | row);
            if (tag == 0) {
                fresh = true;
                break;
            }
        }
        if ((tag & LONG_PRINT) == print) {
            const unsigned long long* other;
            if (tag & LONG_FRESH) {
                __threadfence();   // pairs with the claimer's fence between writing its row and publishing the tag
                other = t.staging + (tag & LONG_ROW) * words;
            } else {
                other = t.keys + pos * words;
            }
            if (long_rows_equal(own, other, t.words)) break;
        }
        if (probes >= COUNT_MAX_PROBES || probes > t.mask) {
            atomicExch(t.live + 1, 1ull);
            return ~0ull;
        }
        pos = (pos + 1) & t.mask;
    }
    atomicAdd(t.counts + pos, add);
    return pos;
}

// count_add_long of one read's key, the slots claimed by the warp listed in t.fresh and counted in t.live[0] with one atomic
// each per warp
__device__ __forceinline__ void count_insert_long(const CountTableLong& t, unsigned long long h, unsigned long long row) {
    bool fresh;
    const unsigned long long pos = count_add_long(t, h, row, 1u, fresh);
    const uint32_t active = __activemask();
    const uint32_t m = __ballot_sync(active, fresh);
    if (!m) return;
    const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
    unsigned long long base = 0;
    if (lane == leader) {
        base = atomicAdd(t.fresh_count, (unsigned long long)__popc(m));
        atomicAdd(t.live, (unsigned long long)__popc(m));
    }
    base = __shfl_sync(active, base, leader);
    if (fresh) t.fresh[base + __popc(m & ((1u << lane) - 1u))] = pos;
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
