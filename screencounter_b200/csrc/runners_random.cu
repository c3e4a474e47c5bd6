// countRandomBarcodes (reference src/count_random_barcodes.cpp:12-60) and the device count tables
// (GPU open-addressing hash of packed keys) shared with the sparse combination tally.
#include <algorithm>
#include <chrono>
#include <cstring>
#include <map>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "api_common.hpp"
#include "handlers.cuh"
#include "hostpool.hpp"
#include "launchers.hpp"
#include "matchers.hpp"

namespace scg {

static double now_s() {
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// ---------------------------------------------------------------------------------------
// CountTable
// ---------------------------------------------------------------------------------------
__global__ void fill_slots_kernel(CountSlot* p, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        p[i] = CountSlot{ ~0ull, 0u, 0u };
    }
}

__global__ void fill_u64_kernel(unsigned long long* p, unsigned long long v, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}

// re-insert the live entries of an old count table into a larger one
__global__ void rehash64_kernel(const CountSlot* slots, size_t n, CountTable64 dst) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const CountSlot s = slots[i];
        if (s.key != ~0ull) count_insert64(dst, s.key, s.count);
    }
}

__global__ void rehash128_kernel(const ulonglong2* keys, const uint32_t* counts, size_t n, CountTable128 dst) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        if (!(keys[i].x == ~0ull && keys[i].y == ~0ull)) count_insert128(dst, keys[i], counts[i]);
    }
}

// re-insert the entries of an old long-key table (every one RESIDENT: keys distinct, so only empty slots are claimed)
__global__ void rehash_long_kernel(const unsigned long long* tags, const uint32_t* counts, const unsigned long long* keys, size_t n,
                                   CountTableLong dst) {
    const size_t words = (size_t)dst.words;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        if (!tags[i]) continue;
        const unsigned long long* key = keys + i * words;
        const unsigned long long h = long_key_hash(key, dst.words);
        unsigned long long pos = h & dst.mask & ~1ull;
        for (unsigned long long probes = 0;; ++probes) {
            if (atomicCAS(dst.tags + pos, 0ull, (h & LONG_PRINT) | LONG_OCCUPIED) == 0) break;
            if (probes > dst.mask) {
                atomicExch(dst.live + 1, 1ull);
                return;
            }
            pos = (pos + 1) & dst.mask;
        }
        for (size_t w = 0; w < words; ++w) dst.keys[pos * words + w] = key[w];
        dst.counts[pos] = counts[i];
        atomicAdd(dst.live, 1ull);
    }
}

// the slots a counting launch claimed: their keys from the staging rows into the key store, their tags RESIDENT
__global__ void promote_fresh_kernel(CountTableLong t) {
    const unsigned long long n = *t.fresh_count;
    const size_t words = (size_t)t.words;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long pos = t.fresh[i];
        const unsigned long long tag = t.tags[pos];
        const unsigned long long* row = t.staging + (tag & LONG_ROW) * words;
        for (size_t w = 0; w < words; ++w) t.keys[pos * words + w] = row[w];
        t.tags[pos] = tag & (LONG_PRINT | LONG_OCCUPIED);
    }
}

// Rank of every base in the byte order of its letter (A < C < G < N < T, what R's order() sees,
// R/countRandomBarcodes.R:73), three bits per base, first base most significant: sorting these integers sorts the
// barcodes as text.  Bases [from, to) of the planes H, L, N (bit b = base b).
__device__ __forceinline__ unsigned long long text_order_bits(unsigned long long H, unsigned long long L, unsigned long long N, int from, int to) {
    unsigned long long s = 0;
    for (int b = from; b < to; ++b) {
        const uint32_t code = (uint32_t)((((H >> b) & 1ull) << 1) | ((L >> b) & 1ull));
        const uint32_t rank = ((N >> b) & 1ull) ? 3u : (code == 3u ? 4u : code);
        s = (s << 3) | rank;
    }
    return s;
}

// Keys of up to 21 bases (random_key64: H | L << 21 | N << 42).
__device__ __forceinline__ unsigned long long text_order_key(unsigned long long k, int len) {
    return text_order_bits(k & 0x1FFFFFull, (k >> 21) & 0x1FFFFFull, (k >> 42) & 0x1FFFFFull, 0, len);
}

// compact the live entries of a narrow table (key_len > 0: keys re-coded to text order on the way); one atomic per warp
__global__ void compact64_kernel(const CountSlot* slots, size_t n, int key_len, unsigned long long* out_keys, uint32_t* out_counts,
                                 unsigned long long* cursor) {
    const int lane = threadIdx.x & 31;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t rounds = (n + stride - 1) / stride;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (size_t r = 0; r < rounds; ++r, i += stride) {
        CountSlot s{ ~0ull, 0u, 0u };
        if (i < n) s = slots[i];
        const bool livep = s.key != ~0ull;
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, livep);
        if (!m) continue;
        unsigned long long base = 0;
        const int leader = __ffs(m) - 1;
        if (lane == leader) base = atomicAdd(cursor, (unsigned long long)__popc(m));
        base = __shfl_sync(0xFFFFFFFFu, base, leader);
        if (livep) {
            const unsigned long long at = base + __popc(m & ((1u << lane) - 1u));
            out_keys[at] = key_len > 0 ? text_order_key(s.key, key_len) : s.key;
            out_counts[at] = s.count;
        }
    }
}

// A row of a wide sorted table (SortedTable: two text-order words), and how the radix sort sees it: word 0 most significant.
struct WideKey {
    unsigned long long w0, w1;
};
__device__ __forceinline__ bool operator<(const WideKey& a, const WideKey& b) { return a.w0 < b.w0 || (a.w0 == b.w0 && a.w1 < b.w1); }
__device__ __forceinline__ bool operator==(const WideKey& a, const WideKey& b) { return a.w0 == b.w0 && a.w1 == b.w1; }
struct WideKeyDecomposer {
    __host__ __device__ ::cuda::std::tuple<unsigned long long&, unsigned long long&> operator()(WideKey& k) const { return { k.w0, k.w1 }; }
};

// compact the live entries of a wide table, one atomic per warp, keys re-coded on the way to the two text-order words, word 1
// shifted up by `shift1` bits: the 3 * key_len bits in use are then the contiguous bits [shift1, 127) of (word 0, word 1),
// the only ones the radix sort has to look at
__global__ void compact128_kernel(const ulonglong2* keys, const uint32_t* counts, size_t n, int key_len, int shift1, WideKey* out_keys,
                                  uint32_t* out_counts, unsigned long long* cursor) {
    const int lane = threadIdx.x & 31;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t rounds = (n + stride - 1) / stride;
    const unsigned long long m42 = (1ull << 42) - 1;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (size_t r = 0; r < rounds; ++r, i += stride) {
        ulonglong2 k = make_ulonglong2(~0ull, ~0ull);
        if (i < n) k = keys[i];
        const bool livep = !(k.x == ~0ull && k.y == ~0ull);
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, livep);
        if (!m) continue;
        unsigned long long base = 0;
        const int leader = __ffs(m) - 1;
        if (lane == leader) base = atomicAdd(cursor, (unsigned long long)__popc(m));
        base = __shfl_sync(0xFFFFFFFFu, base, leader);
        if (livep) {
            const unsigned long long at = base + __popc(m & ((1u << lane) - 1u));
            const unsigned long long H = k.x & m42, L = ((k.x >> 42) | (k.y << 22)) & m42, N = (k.y >> 20) & m42;
            out_keys[at] = WideKey{ text_order_bits(H, L, N, 0, 21), text_order_bits(H, L, N, 21, key_len) << shift1 };
            out_counts[at] = counts[i];
        }
    }
}

__global__ void unshift_word1_kernel(WideKey* keys, size_t n, int shift1) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) keys[i].w1 >>= shift1;
}

// compact the live entries of a long-key table (keys already in text order), one atomic per warp
__global__ void compact_long_kernel(const unsigned long long* tags, const uint32_t* counts, const unsigned long long* keys, size_t n, int words,
                                    unsigned long long* out_keys, uint32_t* out_counts, unsigned long long* cursor) {
    const int lane = threadIdx.x & 31;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t rounds = (n + stride - 1) / stride;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (size_t r = 0; r < rounds; ++r, i += stride) {
        const bool livep = i < n && tags[i] != 0;
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, livep);
        if (!m) continue;
        unsigned long long base = 0;
        const int leader = __ffs(m) - 1;
        if (lane == leader) base = atomicAdd(cursor, (unsigned long long)__popc(m));
        base = __shfl_sync(0xFFFFFFFFu, base, leader);
        if (livep) {
            const unsigned long long at = base + __popc(m & ((1u << lane) - 1u));
            for (int w = 0; w < words; ++w) out_keys[at * words + w] = keys[i * words + w];
            out_counts[at] = counts[i];
        }
    }
}

// LSD sort of a long-key table: word w of every row, in the order of the permutation so far
__global__ void gather_word_kernel(const unsigned long long* __restrict__ keys, const uint32_t* __restrict__ perm, size_t n, int words, int w,
                                   unsigned long long* __restrict__ out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        out[i] = keys[(size_t)perm[i] * words + w];
    }
}

__global__ void iota_kernel(uint32_t* p, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = (uint32_t)i;
}

// rows and counts in the order of the finished permutation
__global__ void gather_rows_kernel(const unsigned long long* __restrict__ keys, const uint32_t* __restrict__ counts, const uint32_t* __restrict__ perm,
                                   size_t n, int words, unsigned long long* __restrict__ out_keys, uint32_t* __restrict__ out_counts) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t from = perm[i];
        for (int w = 0; w < words; ++w) out_keys[i * words + w] = keys[from * words + w];
        out_counts[i] = counts[from];
    }
}

static int fill_grid(Context& ctx, size_t n) { return (int)std::max<size_t>(1, std::min<size_t>((n + 255) / 256, (size_t)ctx.sm_count * 32)); }

void CountTable::init(Context& ctx, bool wide128, size_t initial, int nwords) {
    wide = wide128;
    long_words = nwords;
    size_t cap = 1024;
    while (cap < initial && cap < (1ull << 33)) cap <<= 1;
    capacity = cap;
    if (long_words) {
        slots.alloc(capacity * sizeof(unsigned long long), false);
        keys.alloc(capacity * (size_t)long_words * sizeof(unsigned long long), false);
        fresh_count.alloc(sizeof(unsigned long long), true);
    } else {
        slots.alloc(capacity * 16, false);
    }
    if (wide || long_words) counts.alloc(capacity * sizeof(uint32_t), false);
    live.alloc(2 * sizeof(unsigned long long), false);
    reset(ctx, ctx.stream);
}

void CountTable::reset(Context& ctx, cudaStream_t stream) {
    if (long_words) {
        SCG_CUDA_CHECK(cudaMemsetAsync(slots.ptr, 0, capacity * sizeof(unsigned long long), stream));
        SCG_CUDA_CHECK(cudaMemsetAsync(counts.ptr, 0, capacity * sizeof(uint32_t), stream));
    } else if (wide) {
        fill_u64_kernel<<<fill_grid(ctx, capacity * 2), 256, 0, stream>>>(slots.as<unsigned long long>(), ~0ull, capacity * 2);
        SCG_CUDA_CHECK(cudaMemsetAsync(counts.ptr, 0, capacity * sizeof(uint32_t), stream));
    } else {
        fill_slots_kernel<<<fill_grid(ctx, capacity), 256, 0, stream>>>(slots.as<CountSlot>(), capacity);
    }
    SCG_CUDA_CHECK(cudaGetLastError());
    SCG_CUDA_CHECK(cudaMemsetAsync(live.ptr, 0, 2 * sizeof(unsigned long long), stream));
    ++ctx.launches;
    live_known = 0;
    pending = 0;
}

CountTable64 CountTable::view64() const {
    CountTable64 v;
    v.slots = slots.as<CountSlot>();
    v.mask = capacity - 1;
    v.live = live.as<unsigned long long>();
    return v;
}

CountTable128 CountTable::view128() const {
    CountTable128 v;
    v.keys = slots.as<ulonglong2>();
    v.counts = counts.as<uint32_t>();
    v.mask = capacity - 1;
    v.live = live.as<unsigned long long>();
    return v;
}

CountTableLong CountTable::view_long(size_t rows) {
    if (rows > staging_rows) {
        staging.alloc(rows * (size_t)long_words * sizeof(unsigned long long), false);
        fresh.alloc(rows * sizeof(unsigned long long), false);
        staging_rows = rows;
    }
    CountTableLong v;
    v.tags = slots.as<unsigned long long>();
    v.counts = counts.as<uint32_t>();
    v.keys = keys.as<unsigned long long>();
    v.staging = staging.as<unsigned long long>();
    v.fresh = fresh.as<unsigned long long>();
    v.fresh_count = fresh_count.as<unsigned long long>();
    v.mask = capacity - 1;
    v.live = live.as<unsigned long long>();
    v.words = long_words;
    return v;
}

void CountTable::promote_fresh(Context& ctx, cudaStream_t stream) {
    promote_fresh_kernel<<<ctx.sm_count * 4, 256, 0, stream>>>(view_long(0));
    SCG_CUDA_CHECK(cudaGetLastError());
    SCG_CUDA_CHECK(cudaMemsetAsync(fresh_count.ptr, 0, sizeof(unsigned long long), stream));
    ++ctx.launches;
    ++ctx.timing.launches;
}

void CountTable::check_overflow(Context& ctx) {
    unsigned long long state[2] = { 0, 0 };
    SCG_CUDA_CHECK(cudaMemcpyAsync(state, live.ptr, sizeof state, cudaMemcpyDeviceToHost, ctx.stream));
    SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
    live_known = (long long)state[0];
    pending = 0;
    if (state[1]) throw Error("the device count table overflowed (more distinct keys than it was sized for)");
}

void CountTable::ensure(Context& ctx, long long upcoming) {
    if (fixed) {
        pending += upcoming;
        return;
    }
    // Every insert MAY be a new key.  While that pessimistic bound fits, nothing happens; when it does not, the true number
    // of distinct keys is read back (the table then follows the distinct keys, not the reads), and only if that does not fit
    // either the table grows: at least twofold, by re-inserting its live entries.
    if (2ull * (unsigned long long)(live_known + pending + upcoming) > capacity) {
        check_overflow(ctx);
        const unsigned long long need = 2ull * (unsigned long long)(live_known + upcoming);
        if (need > capacity) {
            size_t ncap = capacity * 2;
            while (ncap < need) ncap *= 2;
            if (ncap > (1ull << 34)) throw Error("the device count table would exceed 2^34 slots");
            DeviceBuffer nslots, ncounts, nkeys, nlive;
            nslots.alloc(ncap * (long_words ? sizeof(unsigned long long) : 16), false);
            nlive.alloc(2 * sizeof(unsigned long long), true);
            if (long_words) {
                const size_t words = (size_t)long_words;
                nkeys.alloc(ncap * words * sizeof(unsigned long long), false);
                ncounts.alloc(ncap * sizeof(uint32_t), true);
                SCG_CUDA_CHECK(cudaMemsetAsync(nslots.ptr, 0, ncap * sizeof(unsigned long long), ctx.stream));
                CountTableLong dst{ nslots.as<unsigned long long>(), ncounts.as<uint32_t>(), nkeys.as<unsigned long long>(), nullptr, nullptr, nullptr,
                                    ncap - 1, nlive.as<unsigned long long>(), long_words };
                rehash_long_kernel<<<fill_grid(ctx, capacity), 256, 0, ctx.stream>>>(slots.as<unsigned long long>(), counts.as<uint32_t>(),
                                                                                   keys.as<unsigned long long>(), capacity, dst);
            } else if (wide) {
                ncounts.alloc(ncap * sizeof(uint32_t), true);
                fill_u64_kernel<<<fill_grid(ctx, ncap * 2), 256, 0, ctx.stream>>>(nslots.as<unsigned long long>(), ~0ull, ncap * 2);
                CountTable128 dst{ nslots.as<ulonglong2>(), ncounts.as<uint32_t>(), ncap - 1, nlive.as<unsigned long long>() };
                rehash128_kernel<<<fill_grid(ctx, capacity), 256, 0, ctx.stream>>>(slots.as<ulonglong2>(), counts.as<uint32_t>(), capacity, dst);
            } else {
                fill_slots_kernel<<<fill_grid(ctx, ncap), 256, 0, ctx.stream>>>(nslots.as<CountSlot>(), ncap);
                CountTable64 dst{ nslots.as<CountSlot>(), ncap - 1, nlive.as<unsigned long long>() };
                rehash64_kernel<<<fill_grid(ctx, capacity), 256, 0, ctx.stream>>>(slots.as<CountSlot>(), capacity, dst);
            }
            SCG_CUDA_CHECK(cudaGetLastError());
            ctx.launches += 2;
            SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
            slots = std::move(nslots);
            counts = std::move(ncounts);
            if (long_words) keys = std::move(nkeys);
            live = std::move(nlive);
            capacity = ncap;
        }
    }
    pending += upcoming;
}

// Live entries as (key, count) sorted by key ON THE DEVICE (radix sort), left there in the layout of SortedTable.
void CountTable::sorted(Context& ctx, int key_len, SortedTable& out) {
    const int words = table_key_words(key_len);
    if (wide != (words == 2) || (long_words != 0) != (words > 2) || (long_words && long_words != words)) {
        throw Error("internal error: count table and key length disagree on the key width");
    }
    check_overflow(ctx);
    const size_t nlive = (size_t)live_known;
    out.rows = nlive;
    out.key_len = key_len;
    const size_t key_bytes = 8 * (size_t)out.words();
    out.keys.alloc(std::max<size_t>(nlive, 1) * key_bytes, false);
    out.counts.alloc(std::max<size_t>(nlive, 1) * sizeof(uint32_t), false);
    if (nlive == 0) return;
    DeviceBuffer d_keys, d_counts, d_cursor, d_temp;
    d_keys.alloc(nlive * key_bytes, false);
    d_counts.alloc(nlive * sizeof(uint32_t), false);
    d_cursor.alloc(sizeof(unsigned long long), true);
    size_t temp_bytes = 0;
    if (long_words) {
        // LSD over the words, last word first: a stable radix sort of each word's 3 * (bases in it) bits carries the permutation
        if (nlive >= (1ull << 32)) throw Error("long-key tables of 2^32 rows or more cannot be sorted");
        compact_long_kernel<<<fill_grid(ctx, capacity), 256, 0, ctx.stream>>>(slots.as<unsigned long long>(), counts.as<uint32_t>(),
                                                                             keys.as<unsigned long long>(), capacity, words, d_keys.as<unsigned long long>(),
                                                                             d_counts.as<uint32_t>(), d_cursor.as<unsigned long long>());
        SCG_CUDA_CHECK(cudaGetLastError());
        DeviceBuffer word_in, word_out, perm_in, perm_out;
        word_in.alloc(nlive * sizeof(unsigned long long), false);
        word_out.alloc(nlive * sizeof(unsigned long long), false);
        perm_in.alloc(nlive * sizeof(uint32_t), false);
        perm_out.alloc(nlive * sizeof(uint32_t), false);
        iota_kernel<<<fill_grid(ctx, nlive), 256, 0, ctx.stream>>>(perm_in.as<uint32_t>(), nlive);
        SCG_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, word_in.as<unsigned long long>(), word_out.as<unsigned long long>(),
                                                       perm_in.as<uint32_t>(), perm_out.as<uint32_t>(), (long long)nlive, 0, 63, ctx.stream));
        d_temp.alloc(temp_bytes, false);
        for (int w = words - 1; w >= 0; --w) {
            const int bases = std::min(21, key_len - 21 * w);
            gather_word_kernel<<<fill_grid(ctx, nlive), 256, 0, ctx.stream>>>(d_keys.as<unsigned long long>(), perm_in.as<uint32_t>(), nlive, words, w,
                                                                            word_in.as<unsigned long long>());
            SCG_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(d_temp.ptr, temp_bytes, word_in.as<unsigned long long>(), word_out.as<unsigned long long>(),
                                                           perm_in.as<uint32_t>(), perm_out.as<uint32_t>(), (long long)nlive, 0, 3 * bases,
                                                           ctx.stream));
            std::swap(perm_in, perm_out);
        }
        gather_rows_kernel<<<fill_grid(ctx, nlive), 256, 0, ctx.stream>>>(d_keys.as<unsigned long long>(), d_counts.as<uint32_t>(), perm_in.as<uint32_t>(),
                                                                        nlive, words, out.keys.as<unsigned long long>(), out.counts.as<uint32_t>());
        SCG_CUDA_CHECK(cudaGetLastError());
        ctx.launches += 3 + 2 * words;
    } else if (wide) {
        const int shift1 = 64 - 3 * (key_len - 21);
        compact128_kernel<<<fill_grid(ctx, capacity), 256, 0, ctx.stream>>>(slots.as<ulonglong2>(), counts.as<uint32_t>(), capacity, key_len, shift1,
                                                                          d_keys.as<WideKey>(), d_counts.as<uint32_t>(), d_cursor.as<unsigned long long>());
        SCG_CUDA_CHECK(cudaGetLastError());
        SCG_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, d_keys.as<WideKey>(), out.keys.as<WideKey>(), d_counts.as<uint32_t>(),
                                                       out.counts.as<uint32_t>(), (long long)nlive, WideKeyDecomposer{}, shift1, 127, ctx.stream));
        d_temp.alloc(temp_bytes, false);
        SCG_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(d_temp.ptr, temp_bytes, d_keys.as<WideKey>(), out.keys.as<WideKey>(), d_counts.as<uint32_t>(),
                                                       out.counts.as<uint32_t>(), (long long)nlive, WideKeyDecomposer{}, shift1, 127, ctx.stream));
        unshift_word1_kernel<<<fill_grid(ctx, nlive), 256, 0, ctx.stream>>>(out.keys.as<WideKey>(), nlive, shift1);
        SCG_CUDA_CHECK(cudaGetLastError());
        ctx.launches += 4;
    } else {
        compact64_kernel<<<fill_grid(ctx, capacity), 256, 0, ctx.stream>>>(slots.as<CountSlot>(), capacity, key_len, d_keys.as<unsigned long long>(),
                                                                         d_counts.as<uint32_t>(), d_cursor.as<unsigned long long>());
        SCG_CUDA_CHECK(cudaGetLastError());
        const int end_bit = key_len > 0 ? 3 * key_len : 64;
        SCG_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, d_keys.as<unsigned long long>(), out.keys.as<unsigned long long>(),
                                                       d_counts.as<uint32_t>(), out.counts.as<uint32_t>(), (long long)nlive, 0, end_bit, ctx.stream));
        d_temp.alloc(temp_bytes, false);
        SCG_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(d_temp.ptr, temp_bytes, d_keys.as<unsigned long long>(), out.keys.as<unsigned long long>(),
                                                       d_counts.as<uint32_t>(), out.counts.as<uint32_t>(), (long long)nlive, 0, end_bit, ctx.stream));
        ctx.launches += 3;
    }
    SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));   // the scratch buffers above go back to the block cache
}

// ---------------------------------------------------------------------------------------
// sorted tables: rendering and merging on the device
// ---------------------------------------------------------------------------------------
// one row per thread; word w renders bases [21w, min(21w + 21, len))
__global__ void render_barcodes_kernel(const unsigned long long* __restrict__ keys, const uint32_t* __restrict__ counts, size_t n, int len,
                                       int words, char* __restrict__ strings, int32_t* __restrict__ freq) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const unsigned long long* row = keys + i * (size_t)words;
        char* out = strings + i * (size_t)len;
        for (int w = 0; w < words; ++w) {
            unsigned long long k = row[w];
            for (int b = min(len, 21 * w + 21) - 1; b >= 21 * w; --b) {
                out[b] = "ACGNT"[k & 7ull];
                k >>= 3;
            }
        }
        freq[i] = (int32_t)counts[i];
    }
}

void render_barcodes(Context& ctx, const SortedTable& t, DeviceBuffer& strings, DeviceBuffer& freq) {
    strings.alloc(std::max<size_t>(t.rows * (size_t)t.key_len, 16), false);
    freq.alloc(std::max<size_t>(t.rows, 4) * sizeof(int32_t), false);
    if (t.rows == 0) return;
    render_barcodes_kernel<<<fill_grid(ctx, t.rows), 256, 0, ctx.stream>>>(t.keys.as<unsigned long long>(), t.counts.as<uint32_t>(), t.rows, t.key_len,
                                                                          t.words(), strings.as<char>(), freq.as<int32_t>());
    SCG_CUDA_CHECK(cudaGetLastError());
    ++ctx.launches;
}

__global__ void render_combinations_kernel(const unsigned long long* __restrict__ keys, const uint32_t* __restrict__ counts, size_t n,
                                           int32_t* __restrict__ out, int32_t* __restrict__ freq) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const unsigned long long k = keys[i];
        out[2 * i] = (int32_t)(k >> 32);
        out[2 * i + 1] = (int32_t)(k & 0xFFFFFFFFull);
        freq[i] = (int32_t)counts[i];
    }
}

void render_combinations(Context& ctx, const SortedTable& t, DeviceBuffer& keys, DeviceBuffer& freq) {
    keys.alloc(std::max<size_t>(t.rows, 2) * 2 * sizeof(int32_t), false);
    freq.alloc(std::max<size_t>(t.rows, 4) * sizeof(int32_t), false);
    if (t.rows == 0) return;
    render_combinations_kernel<<<fill_grid(ctx, t.rows), 256, 0, ctx.stream>>>(t.keys.as<unsigned long long>(), t.counts.as<uint32_t>(), t.rows,
                                                                              keys.as<int32_t>(), freq.as<int32_t>());
    SCG_CUDA_CHECK(cudaGetLastError());
    ++ctx.launches;
}

void device_table_result(Context& ctx, const SortedTable& t, scg_result& out) {
    if (t.key_len > 0) {
        out.width = t.key_len;
        render_barcodes(ctx, t, out.d_strings, out.d_freq);
    } else {
        out.width = 2;
        render_combinations(ctx, t, out.d_keys, out.d_freq);
    }
    SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
    out.on_device = true;
    out.device = ctx.device;
    out.d_rows = t.rows;
}

// Merge of two sorted tables (the device-side reduce() of handlers/RandomBarcodeSingleEnd.hpp:197-207 and of the
// combinations' append + sort, handlers/CombinatorialBarcodesSingleEnd.hpp:268-305): every row finds its place in the
// output by a binary search in the OTHER table -- rank = own index + rows of the other table that sort before it, minus
// the keys both tables hold that sort before it (those collapse into one row).  K: the row's key, one word
// (unsigned long long) or two (WideKey).
template <class K>
__device__ __forceinline__ size_t lower_bound_dev(const K* __restrict__ a, size_t n, K key) {
    size_t lo = 0, hi = n;
    while (lo < hi) {
        const size_t mid = (lo + hi) >> 1;
        if (a[mid] < key) {
            lo = mid + 1;
        } else {
            hi = mid;
        }
    }
    return lo;
}

// pass 1: for every row of a, 1 if b also holds its key (those rows of b are dropped)
template <class K>
__global__ void merge_mark_kernel(const K* __restrict__ ak, size_t na, const K* __restrict__ bk, size_t nb, uint32_t* __restrict__ a_pos_in_b,
                                  uint32_t* __restrict__ b_dup) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < na; i += (size_t)gridDim.x * blockDim.x) {
        const K key = ak[i];
        const size_t p = lower_bound_dev(bk, nb, key);
        a_pos_in_b[i] = (uint32_t)p;
        if (p < nb && bk[p] == key) b_dup[p] = 1;
    }
}

// pass 2 (after an exclusive scan of b_dup): scatter
template <class K>
__global__ void merge_scatter_a_kernel(const K* __restrict__ ak, const uint32_t* __restrict__ ac, size_t na, const K* __restrict__ bk,
                                       const uint32_t* __restrict__ bc, size_t nb, const uint32_t* __restrict__ a_pos_in_b,
                                       const uint32_t* __restrict__ dup_before, K* __restrict__ ck, uint32_t* __restrict__ cc) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < na; i += (size_t)gridDim.x * blockDim.x) {
        const size_t p = a_pos_in_b[i];
        // rows of b before p that survive = p - duplicates among them
        const size_t at = i + p - dup_before[p];
        const K key = ak[i];
        uint32_t count = ac[i];
        if (p < nb && bk[p] == key) count += bc[p];
        ck[at] = key;
        cc[at] = count;
    }
}

template <class K>
__global__ void merge_scatter_b_kernel(const K* __restrict__ ak, size_t na, const K* __restrict__ bk, const uint32_t* __restrict__ bc, size_t nb,
                                       const uint32_t* __restrict__ b_dup, const uint32_t* __restrict__ dup_before, K* __restrict__ ck,
                                       uint32_t* __restrict__ cc) {
    for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < nb; j += (size_t)gridDim.x * blockDim.x) {
        if (b_dup[j]) continue;
        const size_t q = lower_bound_dev(ak, na, bk[j]);   // rows of a before it (its key is not in a)
        const size_t at = q + j - dup_before[j];
        ck[at] = bk[j];
        cc[at] = bc[j];
    }
}

// A row of a long-key sorted table (N >= 3 text-order words), compared word 0 first.
template <int N>
struct LongKey {
    unsigned long long w[N];
};
template <int N>
__device__ __forceinline__ bool operator<(const LongKey<N>& a, const LongKey<N>& b) {
    for (int i = 0; i < N; ++i) {
        if (a.w[i] != b.w[i]) return a.w[i] < b.w[i];
    }
    return false;
}
template <int N>
__device__ __forceinline__ bool operator==(const LongKey<N>& a, const LongKey<N>& b) {
    for (int i = 0; i < N; ++i) {
        if (a.w[i] != b.w[i]) return false;
    }
    return true;
}

// the longest barcode a template holds (MAX_TEMPLATE bases) takes this many words
constexpr int MAX_TABLE_WORDS = (MAX_TEMPLATE + 20) / 21;

template <int N, class F>
static void with_long_key(int words, F&& f) {
    if constexpr (N > MAX_TABLE_WORDS) {
        throw Error("internal error: sorted table of " + std::to_string(words) + " words per row");
    } else if (words == N) {
        f(LongKey<N>{});
    } else {
        with_long_key<N + 1>(words, f);
    }
}

// f(K{}) with the key type of tables of `words` words per row
template <class F>
static void with_key_type(int words, F&& f) {
    if (words == 2) {
        f(WideKey{});
    } else if (words > 2) {
        with_long_key<3>(words, f);
    } else {
        f(0ull);
    }
}

void merge_sorted_tables(Context& ctx, const SortedTable& a, const SortedTable& b, SortedTable& c) {
    c.key_len = a.rows ? a.key_len : b.key_len;
    const size_t na = a.rows, nb = b.rows;
    if (na >= (1ull << 32) || nb >= (1ull << 32)) throw Error("sorted tables of 2^32 rows or more cannot be merged");
    DeviceBuffer pos, dup, dup_scan, d_temp;
    pos.alloc(std::max<size_t>(na, 1) * sizeof(uint32_t), false);
    dup.alloc((nb + 1) * sizeof(uint32_t), false);
    dup_scan.alloc((nb + 1) * sizeof(uint32_t), false);
    SCG_CUDA_CHECK(cudaMemsetAsync(dup.ptr, 0, (nb + 1) * sizeof(uint32_t), ctx.stream));
    with_key_type(c.words(), [&](auto key) {
        using K = decltype(key);
        if (na) {
            merge_mark_kernel<K><<<fill_grid(ctx, na), 256, 0, ctx.stream>>>(a.keys.as<K>(), na, b.keys.as<K>(), nb, pos.as<uint32_t>(), dup.as<uint32_t>());
            SCG_CUDA_CHECK(cudaGetLastError());
        }
        size_t temp_bytes = 0;
        SCG_CUDA_CHECK(cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, dup.as<uint32_t>(), dup_scan.as<uint32_t>(), (long long)(nb + 1), ctx.stream));
        d_temp.alloc(temp_bytes, false);
        SCG_CUDA_CHECK(cub::DeviceScan::ExclusiveSum(d_temp.ptr, temp_bytes, dup.as<uint32_t>(), dup_scan.as<uint32_t>(), (long long)(nb + 1), ctx.stream));
        uint32_t ndup = 0;
        SCG_CUDA_CHECK(cudaMemcpyAsync(&ndup, dup_scan.as<uint32_t>() + nb, sizeof ndup, cudaMemcpyDeviceToHost, ctx.stream));
        SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        c.rows = na + nb - ndup;
        c.keys.alloc(std::max<size_t>(c.rows, 1) * sizeof(K), false);
        c.counts.alloc(std::max<size_t>(c.rows, 1) * sizeof(uint32_t), false);
        if (na) {
            merge_scatter_a_kernel<K><<<fill_grid(ctx, na), 256, 0, ctx.stream>>>(a.keys.as<K>(), a.counts.as<uint32_t>(), na, b.keys.as<K>(),
                                                                                b.counts.as<uint32_t>(), nb, pos.as<uint32_t>(), dup_scan.as<uint32_t>(),
                                                                                c.keys.as<K>(), c.counts.as<uint32_t>());
        }
        if (nb) {
            merge_scatter_b_kernel<K><<<fill_grid(ctx, nb), 256, 0, ctx.stream>>>(a.keys.as<K>(), na, b.keys.as<K>(), b.counts.as<uint32_t>(), nb,
                                                                                dup.as<uint32_t>(), dup_scan.as<uint32_t>(), c.keys.as<K>(),
                                                                                c.counts.as<uint32_t>());
        }
    });
    SCG_CUDA_CHECK(cudaGetLastError());
    ctx.launches += 5;
    SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
}

// What validate_table_kernel found wrong with a table, one bit per kind of fault (messages in validate_sorted_table)
enum : uint32_t { TABLE_UNSORTED = 1, TABLE_DUPLICATE = 2, TABLE_RANK = 4, TABLE_HIGH_BITS = 8, TABLE_COMBO_INDEX = 16, TABLE_COUNT = 32 };

// faults of one word of a barcode key that holds `groups` (1..21) bases: a 3-bit rank above 4 (the renderer indexes "ACGNT"
// with it), or bits set above the bases
__device__ __forceinline__ uint32_t barcode_word_faults(unsigned long long w, int groups) {
    const unsigned long long used = (1ull << (3 * groups)) - 1;
    const unsigned long long low = 0x1249249249249249ull & used;   // bit 0 of every group in use
    uint32_t e = (w & ~used) ? TABLE_HIGH_BITS : 0u;
    if ((w >> 2) & (w | (w >> 1)) & low) e |= TABLE_RANK;       // bit 2 set and bit 1 or 0 set: 5, 6 or 7
    return e;
}

// one row per thread: the row's key and count, and its order against the row before it; faults are or-ed into *err
__global__ void validate_table_kernel(const unsigned long long* __restrict__ keys, const uint32_t* __restrict__ counts, size_t n, int key_len,
                                      uint32_t* err) {
    const int words = key_len > 21 ? 2 : 1;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const unsigned long long* row = keys + i * (size_t)words;
        const unsigned long long k0 = row[0], k1 = words == 2 ? row[1] : 0ull;
        uint32_t e = 0;
        if (key_len == 0) {
            if (k0 & 0x8000000080000000ull) e |= TABLE_COMBO_INDEX;
        } else {
            e |= barcode_word_faults(k0, min(key_len, 21));
            if (words == 2) e |= barcode_word_faults(k1, key_len - 21);
        }
        if (counts[i] >> 31) e |= TABLE_COUNT;
        if (i > 0) {
            const unsigned long long p0 = row[-words], p1 = words == 2 ? row[-1] : 0ull;
            if (p0 == k0 && p1 == k1) {
                e |= TABLE_DUPLICATE;
            } else if (p0 > k0 || (p0 == k0 && p1 > k1)) {
                e |= TABLE_UNSORTED;
            }
        }
        if (e) atomicOr(err, e);
    }
}

void validate_sorted_table(Context& ctx, const SortedTable& t) {
    if (t.rows == 0) return;
    DeviceBuffer d_err;
    d_err.alloc(sizeof(uint32_t), true);
    validate_table_kernel<<<fill_grid(ctx, t.rows), 256, 0, ctx.stream>>>(t.keys.as<unsigned long long>(), t.counts.as<uint32_t>(), t.rows, t.key_len,
                                                                         d_err.as<uint32_t>());
    SCG_CUDA_CHECK(cudaGetLastError());
    ++ctx.launches;
    uint32_t err = 0;
    SCG_CUDA_CHECK(cudaMemcpyAsync(&err, d_err.ptr, sizeof err, cudaMemcpyDeviceToHost, ctx.stream));
    SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
    if (!err) return;
    static const char* const what[] = { "rows are not in ascending key order", "a key appears in two rows",
                                        "a key holds a base rank above 4", "a key has bits set beyond its key length",
                                        "a combination index is 2^31 or more", "a count is 2^31 or more" };
    std::string msg = "malformed sorted table:";
    for (int b = 0; b < 6; ++b) {
        if (err & (1u << b)) msg += std::string(msg.back() == ':' ? " " : "; ") + what[b];
    }
    throw Error(msg);
}

// column[i] = count of all_keys[i] in table t, 0 where t does not hold the key (every key of t is in all_keys)
template <class K>
__global__ void scatter_column_kernel(const K* __restrict__ uk, size_t nu, const K* __restrict__ tk, const uint32_t* __restrict__ tc, size_t nt,
                                      int32_t* __restrict__ column) {
    for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < nt; j += (size_t)gridDim.x * blockDim.x) {
        const K key = tk[j];
        const size_t p = lower_bound_dev(uk, nu, key);
        if (p < nu && uk[p] == key) column[p] = (int32_t)tc[j];
    }
}

void scatter_table_column(Context& ctx, const SortedTable& all_keys, const SortedTable& t, int32_t* column) {
    if (t.rows == 0) return;
    with_key_type(t.words(), [&](auto key) {
        using K = decltype(key);
        scatter_column_kernel<K><<<fill_grid(ctx, t.rows), 256, 0, ctx.stream>>>(all_keys.keys.as<K>(), all_keys.rows, t.keys.as<K>(),
                                                                                t.counts.as<uint32_t>(), t.rows, column);
    });
    SCG_CUDA_CHECK(cudaGetLastError());
    ++ctx.launches;
}

// ---------------------------------------------------------------------------------------
// ComboTally
// ---------------------------------------------------------------------------------------
void ComboTally::init(Context& ctx, int a, int b) {
    n1 = a;
    n2 = b;
    dense = (long long)n1 * n2 <= (1ll << 24);
    // SCG_COMBO_FORCE_SPARSE=1: tally in the device hash whatever the pool sizes (measurement: BASELINE configs[3] asks for it)
    if (const char* env = std::getenv("SCG_COMBO_FORCE_SPARSE")) {
        if (env[0] && env[0] != '0') dense = false;
    }
    if (dense) {
        matrix.alloc((size_t)std::max<long long>((long long)n1 * n2, 1) * sizeof(int32_t), true);
    } else {
        table.init(ctx, false, 1u << 20);
    }
}

void ComboTally::reset(Context& ctx, cudaStream_t stream) {
    if (dense) {
        SCG_CUDA_CHECK(cudaMemsetAsync(matrix.ptr, 0, (size_t)std::max<long long>((long long)n1 * n2, 1) * sizeof(int32_t), stream));
    } else {
        table.reset(ctx, stream);
    }
}

ComboSink ComboTally::sink(Context& ctx, long long upcoming) {
    ComboSink s;
    std::memset(&s, 0, sizeof s);
    s.n2 = n2;
    if (dense) {
        s.dense = matrix.as<int32_t>();
    } else {
        table.ensure(ctx, upcoming);
        s.sparse = table.view64();
    }
    return s;
}

// non-zero cells of the dense matrix, in row-major order, as (first << 32 | second, count)
__global__ void dense_cells_kernel(const int32_t* __restrict__ matrix, size_t cells, int n2, unsigned long long* __restrict__ keys,
                                   uint32_t* __restrict__ counts, unsigned long long* cursor_by_block, int phase) {
    // phase 0: count the non-zero cells of each block's contiguous span; phase 1: write them at the block's offset
    const size_t per_block = (cells + gridDim.x - 1) / gridDim.x;
    const size_t begin = (size_t)blockIdx.x * per_block, end = min(cells, begin + per_block);
    __shared__ unsigned long long base;
    __shared__ uint32_t warp_tot[8];
    if (threadIdx.x == 0) base = phase ? cursor_by_block[blockIdx.x] : 0ull;
    __syncthreads();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    unsigned long long total = 0;
    for (size_t at = begin; at < end; at += blockDim.x) {
        const size_t i = at + threadIdx.x;
        const int32_t v = i < end ? matrix[i] : 0;
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, v != 0);
        if (lane == 0) warp_tot[wib] = __popc(m);
        __syncthreads();
        uint32_t before = 0, all = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
            if (w < wib) before += warp_tot[w];
            all += warp_tot[w];
        }
        if (phase && v != 0) {
            const unsigned long long o = base + total + before + __popc(m & ((1u << lane) - 1u));
            keys[o] = ((unsigned long long)(i / n2) << 32) | (unsigned long long)(i % n2);
            counts[o] = (uint32_t)v;
        }
        total += all;
        __syncthreads();
    }
    if (!phase && threadIdx.x == 0) cursor_by_block[blockIdx.x] = total;
}

void ComboTally::sorted(Context& ctx, SortedTable& out) {
    if (!dense) {
        table.sorted(ctx, 0, out);
        return;
    }
    const size_t cells = (size_t)n1 * n2;
    out.key_len = 0;
    const int blocks = (int)std::max<size_t>(1, std::min<size_t>((cells + 4095) / 4096, 1024));
    DeviceBuffer per_block, scanned, d_temp;
    per_block.alloc((size_t)(blocks + 1) * sizeof(unsigned long long), true);
    scanned.alloc((size_t)(blocks + 1) * sizeof(unsigned long long), false);
    dense_cells_kernel<<<blocks, 256, 0, ctx.stream>>>(matrix.as<int32_t>(), cells, n2, nullptr, nullptr, per_block.as<unsigned long long>(), 0);
    SCG_CUDA_CHECK(cudaGetLastError());
    size_t temp_bytes = 0;
    SCG_CUDA_CHECK(cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, per_block.as<unsigned long long>(), scanned.as<unsigned long long>(), blocks + 1,
                                                 ctx.stream));
    d_temp.alloc(temp_bytes, false);
    SCG_CUDA_CHECK(cub::DeviceScan::ExclusiveSum(d_temp.ptr, temp_bytes, per_block.as<unsigned long long>(), scanned.as<unsigned long long>(), blocks + 1,
                                                 ctx.stream));
    unsigned long long rows = 0;
    SCG_CUDA_CHECK(cudaMemcpyAsync(&rows, scanned.as<unsigned long long>() + blocks, sizeof rows, cudaMemcpyDeviceToHost, ctx.stream));
    SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
    out.rows = (size_t)rows;
    out.keys.alloc(std::max<size_t>(out.rows, 1) * 8, false);
    out.counts.alloc(std::max<size_t>(out.rows, 1) * sizeof(uint32_t), false);
    if (rows) {
        dense_cells_kernel<<<blocks, 256, 0, ctx.stream>>>(matrix.as<int32_t>(), cells, n2, out.keys.as<unsigned long long>(), out.counts.as<uint32_t>(),
                                                          scanned.as<unsigned long long>(), 1);
        SCG_CUDA_CHECK(cudaGetLastError());
    }
    ctx.launches += 3;
    SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
}

// sort_combinations + count_combinations (reference inst/include/kaori/utils.hpp:173-198, src/utils.h:14-45):
// rows sorted ascending by (first, second), one frequency per distinct combination.  Sorted and rendered on the device;
// the table stays there until scg_result_copy_table copies it into the caller's arrays.
void ComboTally::harvest(Context& ctx, scg_result& out) {
    SortedTable t;
    sorted(ctx, t);
    device_table_result(ctx, t, out);
}

} // namespace scg

using namespace scg;

extern "C" {

} // extern "C"

namespace scg {

// countRandomBarcodes over one reader.  The barcodes stay on the device as a sorted table (rank-coded, text order); only when
// some were taken from raw read text is the result rendered on the host.
void count_random_reader(Context& c, FastqReader* reader, const RandomMatcher& m, int nthreads, SparseCounts& result) {
    const TemplateSpec& tmpl = m.tmpl;
    const int key_len = m.key_len;
    const bool wide = m.wide;

    c.ensure_ready();
    CountTable tab;
    tab.init(c, wide, (wide || m.long_words) ? (1u << 20) : (1u << 23), m.long_words);   // 8 M slots (128 MB) to start with: a few million distinct barcodes need no rehash
    DeviceBuffer d_odd_out, d_odd_count;
    d_odd_count.alloc(sizeof(unsigned long long), true);
    std::map<std::string, int> extra;   // keys of reads that need their raw text

    ReadPipeline pipe(c, reader, nullptr, nthreads, true);
    ReadPipeline::Batch b;
    long long nreads = 0;
    std::vector<OddOutcome> odd_host;
    while (pipe.next(b)) {
        {
            const double t0 = now_s();
            tab.ensure(c, b.n);
            c.timing.setup_s += now_s() - t0;
        }
        // reads flagged odd get their outcome reported back; the device-side reader only knows on the device how many
        // there are (count_odd < 0), so room is made for all
        const long long nodd_host = pipe.count_odd(b);
        const long long nodd = nodd_host < 0 ? b.n : nodd_host;
        d_odd_out.reserve((size_t)std::max<long long>(nodd, 1) * sizeof(OddOutcome));
        SCG_CUDA_CHECK(cudaMemsetAsync(d_odd_count.ptr, 0, sizeof(unsigned long long), c.stream));
        launch_random(c, b.reads1, m, tab, b.odd1, d_odd_out.as<OddOutcome>(), d_odd_count.as<unsigned long long>(), nullptr, c.stream);
        pipe.submitted(b);
        if (nodd > 0) {
            // reads holding lower-case letters or symbols other than N: the device decided where the
            // barcode sits, the host renders it from the raw read text exactly as the reference would
            unsigned long long got = 0;
            SCG_CUDA_CHECK(cudaMemcpyAsync(&got, d_odd_count.ptr, sizeof got, cudaMemcpyDeviceToHost, c.stream));
            SCG_CUDA_CHECK(cudaStreamSynchronize(c.stream));
            odd_host.resize(got);
            if (got) {
                SCG_CUDA_CHECK(cudaMemcpyAsync(odd_host.data(), d_odd_out.ptr, got * sizeof(OddOutcome), cudaMemcpyDeviceToHost, c.stream));
                SCG_CUDA_CHECK(cudaStreamSynchronize(c.stream));
            }
            std::sort(odd_host.begin(), odd_host.end(), [](const OddOutcome& x, const OddOutcome& y) { return x.read < y.read; });
            std::string key(key_len, ' ');
            std::string seq;
            for (const auto& o : odd_host) {
                pipe.raw_read(b, (long long)o.read, seq);
                const char* start = seq.data() + o.position + tmpl.fwd_regions[0].start;
                if (!o.reverse) {  // forward_match: raw characters (handlers/RandomBarcodeSingleEnd.hpp:93-104)
                    key.assign(start, key_len);
                } else {  // reverse_match: complement_base<true> (:106-120, utils.hpp:41-62)
                    for (int j = 0; j < key_len; ++j) {
                        const char ch = start[key_len - j - 1];
                        char out;
                        switch (ch) {
                            case 'A': case 'a': out = 'T'; break;
                            case 'C': case 'c': out = 'G'; break;
                            case 'G': case 'g': out = 'C'; break;
                            case 'T': case 't': out = 'A'; break;
                            case 'N': case 'n': out = 'N'; break;
                            default: throw Error(std::string("cannot complement unknown base '") + ch + "'");
                        }
                        key[j] = out;
                    }
                }
                ++extra[key];
            }
        }
        nreads += b.n;
    }
    const double t_harvest = now_s();
    result.reads = nreads;
    // sorted as text ON THE DEVICE (radix sort of rank-coded keys)
    SortedTable sorted;
    tab.sorted(c, key_len, sorted);
    if (extra.empty()) {
        result.table = std::move(sorted);
        c.timing.harvest_s = now_s() - t_harvest;
        return;
    }
    // a few keys came from raw read text (lower case, IUPAC letters): merged on the host in text order
    const size_t n = sorted.rows;
    const int words = sorted.words();
    std::vector<unsigned long long> order_keys(n * (size_t)words);
    std::vector<uint32_t> cnt(n);
    if (n) {
        SCG_CUDA_CHECK(cudaMemcpyAsync(order_keys.data(), sorted.keys.ptr, order_keys.size() * 8, cudaMemcpyDeviceToHost, c.stream));
        SCG_CUDA_CHECK(cudaMemcpyAsync(cnt.data(), sorted.counts.ptr, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, c.stream));
        SCG_CUDA_CHECK(cudaStreamSynchronize(c.stream));
    }
    // one row of the table as text: word w holds bases [21w, min(21w + 21, key_len))
    auto render = [&](const unsigned long long* row, char* out) {
        for (int w = 0; w < words; ++w) {
            unsigned long long k = row[w];
            for (int b = std::min(key_len, 21 * w + 21) - 1; b >= 21 * w; --b) {
                out[b] = "ACGNT"[k & 7ull];
                k >>= 3;
            }
        }
    };
    std::unique_ptr<scg_result> r(new scg_result);
    r->width = key_len;
    r->strings.reserve((n + extra.size()) * (size_t)key_len);
    r->freq.reserve(n + extra.size());
    std::string cur(key_len, ' ');
    auto it = extra.begin();
    auto emit = [&](const std::string& k, int f) {
        r->strings.insert(r->strings.end(), k.begin(), k.end());
        r->freq.push_back(f);
    };
    for (size_t i = 0; i < n; ++i) {
        render(&order_keys[i * (size_t)words], &cur[0]);
        while (it != extra.end() && it->first < cur) {
            emit(it->first, it->second);
            ++it;
        }
        int f = (int)cnt[i];
        if (it != extra.end() && it->first == cur) {
            f += it->second;
            ++it;
        }
        emit(cur, f);
    }
    for (; it != extra.end(); ++it) emit(it->first, it->second);
    c.timing.harvest_s = now_s() - t_harvest;
    result.rendered = std::move(r);
}

void count_random_file(scg_ctx* ctx, const scg_source* src, const char* constant, int strand, int mismatches, int use_first, int nthreads,
                       bool split_over_devices, SparseCounts& out) {
    Context& c = ctx->impl;
    const double t_start = now_s();
    c.timing = Timing();
    Source source(src);
    RandomMatcher m;
    m.prepare(constant, strand, mismatches, use_first != 0);
    c.ensure_ready();
    if (!(split_over_devices && !ctx->peers.empty() &&
          count_random_multi(ctx, *source.reader, constant, strand, mismatches, use_first, nthreads, out))) {
        count_random_reader(c, source.reader.get(), m, nthreads, out);
        c.timing.parse_s = source.reader->parse_seconds();
    }
    c.timing.total_s = now_s() - t_start;
    c.finish_timing();
}

} // namespace scg

extern "C" {

int scg_count_random(scg_ctx* ctx, const scg_source* src, const char* constant, int strand, int mismatches, int use_first,
                     int nthreads, scg_result** table, int32_t* total) {
    return guarded(ctx, [&] {
        SparseCounts counts;
        count_random_file(ctx, src, constant, strand, mismatches, use_first, nthreads, true, counts);
        if (!counts.rendered) {
            // the table was sorted on the device: rendered there too, and left there (scg_result_copy_table copies the finished
            // table straight into the caller's arrays, no host image in between)
            counts.rendered.reset(new scg_result);
            device_table_result(ctx->impl, counts.table, *counts.rendered);
        }
        *table = counts.rendered.release();
        *total = (int32_t)counts.reads;
    });
}

} // extern "C"
