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

// Rank of every base in the byte order of its letter (A < C < G < N < T, what R's order() sees,
// R/countRandomBarcodes.R:73), three bits per base, first base most significant: sorting these integers sorts the
// barcodes as text.  Keys of up to 21 bases (random_key64: H | L << 21 | N << 42).
__device__ __forceinline__ unsigned long long text_order_key(unsigned long long k, int len) {
    const uint32_t H = (uint32_t)(k & 0x1FFFFFull), L = (uint32_t)((k >> 21) & 0x1FFFFFull), N = (uint32_t)((k >> 42) & 0x1FFFFFull);
    unsigned long long s = 0;
    for (int b = 0; b < len; ++b) {
        const uint32_t code = (((H >> b) & 1u) << 1) | ((L >> b) & 1u);
        const uint32_t rank = ((N >> b) & 1u) ? 3u : (code == 3u ? 4u : code);
        s = (s << 3) | rank;
    }
    return s;
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

__global__ void compact128_kernel(const ulonglong2* keys, const uint32_t* counts, size_t n,
                                  ulonglong2* out_keys, uint32_t* out_counts, unsigned long long* cursor) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        if (!(keys[i].x == ~0ull && keys[i].y == ~0ull)) {
            const unsigned long long at = atomicAdd(cursor, 1ull);
            out_keys[at] = keys[i];
            out_counts[at] = counts[i];
        }
    }
}

static int fill_grid(Context& ctx, size_t n) { return (int)std::max<size_t>(1, std::min<size_t>((n + 255) / 256, (size_t)ctx.sm_count * 32)); }

void CountTable::init(Context& ctx, bool wide128, size_t initial) {
    wide = wide128;
    size_t cap = 1024;
    while (cap < initial && cap < (1ull << 33)) cap <<= 1;
    capacity = cap;
    slots.alloc(capacity * 16, false);
    if (wide) counts.alloc(capacity * sizeof(uint32_t), false);
    live.alloc(2 * sizeof(unsigned long long), false);
    reset(ctx, ctx.stream);
}

void CountTable::reset(Context& ctx, cudaStream_t stream) {
    if (wide) {
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
            DeviceBuffer nslots, ncounts, nlive;
            nslots.alloc(ncap * 16, false);
            nlive.alloc(2 * sizeof(unsigned long long), true);
            if (wide) {
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
            live = std::move(nlive);
            capacity = ncap;
        }
    }
    pending += upcoming;
}

void CountTable::download(Context& ctx, std::vector<unsigned long long>& keys_lo, std::vector<unsigned long long>& keys_hi,
                          std::vector<uint32_t>& out_counts) {
    check_overflow(ctx);
    const size_t nlive = (size_t)live_known;
    keys_lo.resize(nlive);
    keys_hi.clear();
    out_counts.resize(nlive);
    if (nlive == 0) return;
    DeviceBuffer d_keys, d_counts, d_cursor;
    d_keys.alloc(nlive * 16, false);
    d_counts.alloc(nlive * sizeof(uint32_t), false);
    d_cursor.alloc(sizeof(unsigned long long), true);
    if (wide) {
        compact128_kernel<<<fill_grid(ctx, capacity), 256, 0, ctx.stream>>>(slots.as<ulonglong2>(), counts.as<uint32_t>(), capacity,
                                                                          d_keys.as<ulonglong2>(), d_counts.as<uint32_t>(),
                                                                          d_cursor.as<unsigned long long>());
    } else {
        compact64_kernel<<<fill_grid(ctx, capacity), 256, 0, ctx.stream>>>(slots.as<CountSlot>(), capacity, 0, d_keys.as<unsigned long long>(),
                                                                         d_counts.as<uint32_t>(), d_cursor.as<unsigned long long>());
    }
    SCG_CUDA_CHECK(cudaGetLastError());
    ++ctx.launches;
    SCG_CUDA_CHECK(cudaMemcpyAsync(out_counts.data(), d_counts.ptr, nlive * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx.stream));
    if (wide) {
        std::vector<ulonglong2> tmp(nlive);
        SCG_CUDA_CHECK(cudaMemcpyAsync(tmp.data(), d_keys.ptr, nlive * 16, cudaMemcpyDeviceToHost, ctx.stream));
        SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        keys_hi.resize(nlive);
        for (size_t i = 0; i < nlive; ++i) {
            keys_lo[i] = tmp[i].x;
            keys_hi[i] = tmp[i].y;
        }
    } else {
        SCG_CUDA_CHECK(cudaMemcpyAsync(keys_lo.data(), d_keys.ptr, nlive * 8, cudaMemcpyDeviceToHost, ctx.stream));
        SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
    }
}

// Live entries of a narrow table as (key, count) sorted by key ON THE DEVICE (radix sort), left there.
void CountTable::sorted(Context& ctx, int key_len, SortedTable& out) {
    if (wide) throw Error("internal error: only narrow count tables are sorted on the device");
    check_overflow(ctx);
    const size_t nlive = (size_t)live_known;
    out.rows = nlive;
    out.key_len = key_len;
    out.keys.alloc(std::max<size_t>(nlive, 1) * 8, false);
    out.counts.alloc(std::max<size_t>(nlive, 1) * sizeof(uint32_t), false);
    if (nlive == 0) return;
    DeviceBuffer d_keys, d_counts, d_cursor, d_temp;
    d_keys.alloc(nlive * 8, false);
    d_counts.alloc(nlive * sizeof(uint32_t), false);
    d_cursor.alloc(sizeof(unsigned long long), true);
    compact64_kernel<<<fill_grid(ctx, capacity), 256, 0, ctx.stream>>>(slots.as<CountSlot>(), capacity, key_len, d_keys.as<unsigned long long>(),
                                                                     d_counts.as<uint32_t>(), d_cursor.as<unsigned long long>());
    SCG_CUDA_CHECK(cudaGetLastError());
    const int end_bit = key_len > 0 ? 3 * key_len : 64;
    size_t temp_bytes = 0;
    SCG_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, d_keys.as<unsigned long long>(), out.keys.as<unsigned long long>(),
                                                   d_counts.as<uint32_t>(), out.counts.as<uint32_t>(), (long long)nlive, 0, end_bit, ctx.stream));
    d_temp.alloc(temp_bytes, false);
    SCG_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(d_temp.ptr, temp_bytes, d_keys.as<unsigned long long>(), out.keys.as<unsigned long long>(),
                                                   d_counts.as<uint32_t>(), out.counts.as<uint32_t>(), (long long)nlive, 0, end_bit, ctx.stream));
    ctx.launches += 3;
    SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));   // the scratch buffers above go back to the block cache
}

// ---------------------------------------------------------------------------------------
// sorted tables: rendering and merging on the device
// ---------------------------------------------------------------------------------------
__global__ void render_barcodes_kernel(const unsigned long long* __restrict__ keys, const uint32_t* __restrict__ counts, size_t n, int len,
                                       char* __restrict__ strings, int32_t* __restrict__ freq) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        unsigned long long k = keys[i];
        char* out = strings + i * (size_t)len;
        for (int b = len - 1; b >= 0; --b) {
            out[b] = "ACGNT"[k & 7ull];
            k >>= 3;
        }
        freq[i] = (int32_t)counts[i];
    }
}

void render_barcodes(Context& ctx, const SortedTable& t, DeviceBuffer& strings, DeviceBuffer& freq) {
    strings.alloc(std::max<size_t>(t.rows * (size_t)t.key_len, 16), false);
    freq.alloc(std::max<size_t>(t.rows, 4) * sizeof(int32_t), false);
    if (t.rows == 0) return;
    render_barcodes_kernel<<<fill_grid(ctx, t.rows), 256, 0, ctx.stream>>>(t.keys.as<unsigned long long>(), t.counts.as<uint32_t>(), t.rows, t.key_len,
                                                                          strings.as<char>(), freq.as<int32_t>());
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
// the keys both tables hold that sort before it (those collapse into one row).
__device__ __forceinline__ size_t lower_bound_dev(const unsigned long long* __restrict__ a, size_t n, unsigned long long key) {
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
__global__ void merge_mark_kernel(const unsigned long long* __restrict__ ak, size_t na, const unsigned long long* __restrict__ bk, size_t nb,
                                  uint32_t* __restrict__ a_pos_in_b, uint32_t* __restrict__ b_dup) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < na; i += (size_t)gridDim.x * blockDim.x) {
        const size_t p = lower_bound_dev(bk, nb, ak[i]);
        a_pos_in_b[i] = (uint32_t)p;
        if (p < nb && bk[p] == ak[i]) b_dup[p] = 1;
    }
}

// pass 2 (after an exclusive scan of b_dup): scatter
__global__ void merge_scatter_a_kernel(const unsigned long long* __restrict__ ak, const uint32_t* __restrict__ ac, size_t na,
                                       const unsigned long long* __restrict__ bk, const uint32_t* __restrict__ bc, size_t nb,
                                       const uint32_t* __restrict__ a_pos_in_b, const uint32_t* __restrict__ dup_before,
                                       unsigned long long* __restrict__ ck, uint32_t* __restrict__ cc) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < na; i += (size_t)gridDim.x * blockDim.x) {
        const size_t p = a_pos_in_b[i];
        // rows of b before p that survive = p - duplicates among them
        const size_t at = i + p - dup_before[p];
        uint32_t count = ac[i];
        if (p < nb && bk[p] == ak[i]) count += bc[p];
        ck[at] = ak[i];
        cc[at] = count;
    }
}

__global__ void merge_scatter_b_kernel(const unsigned long long* __restrict__ ak, size_t na, const unsigned long long* __restrict__ bk,
                                       const uint32_t* __restrict__ bc, size_t nb, const uint32_t* __restrict__ b_dup,
                                       const uint32_t* __restrict__ dup_before, unsigned long long* __restrict__ ck, uint32_t* __restrict__ cc) {
    for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < nb; j += (size_t)gridDim.x * blockDim.x) {
        if (b_dup[j]) continue;
        const size_t q = lower_bound_dev(ak, na, bk[j]);   // rows of a before it (its key is not in a)
        const size_t at = q + j - dup_before[j];
        ck[at] = bk[j];
        cc[at] = bc[j];
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
    if (na) {
        merge_mark_kernel<<<fill_grid(ctx, na), 256, 0, ctx.stream>>>(a.keys.as<unsigned long long>(), na, b.keys.as<unsigned long long>(), nb,
                                                                     pos.as<uint32_t>(), dup.as<uint32_t>());
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
    c.keys.alloc(std::max<size_t>(c.rows, 1) * 8, false);
    c.counts.alloc(std::max<size_t>(c.rows, 1) * sizeof(uint32_t), false);
    if (na) {
        merge_scatter_a_kernel<<<fill_grid(ctx, na), 256, 0, ctx.stream>>>(a.keys.as<unsigned long long>(), a.counts.as<uint32_t>(), na,
                                                                          b.keys.as<unsigned long long>(), b.counts.as<uint32_t>(), nb, pos.as<uint32_t>(),
                                                                          dup_scan.as<uint32_t>(), c.keys.as<unsigned long long>(), c.counts.as<uint32_t>());
    }
    if (nb) {
        merge_scatter_b_kernel<<<fill_grid(ctx, nb), 256, 0, ctx.stream>>>(a.keys.as<unsigned long long>(), na, b.keys.as<unsigned long long>(),
                                                                          b.counts.as<uint32_t>(), nb, dup.as<uint32_t>(), dup_scan.as<uint32_t>(),
                                                                          c.keys.as<unsigned long long>(), c.counts.as<uint32_t>());
    }
    SCG_CUDA_CHECK(cudaGetLastError());
    ctx.launches += 5;
    SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
}

// column[i] = count of all_keys[i] in table t, 0 where t does not hold the key (every key of t is in all_keys)
__global__ void scatter_column_kernel(const unsigned long long* __restrict__ uk, size_t nu, const unsigned long long* __restrict__ tk,
                                      const uint32_t* __restrict__ tc, size_t nt, int32_t* __restrict__ column) {
    for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < nt; j += (size_t)gridDim.x * blockDim.x) {
        const size_t p = lower_bound_dev(uk, nu, tk[j]);
        if (p < nu && uk[p] == tk[j]) column[p] = (int32_t)tc[j];
    }
}

void scatter_table_column(Context& ctx, const SortedTable& all_keys, const SortedTable& t, int32_t* column) {
    if (t.rows == 0) return;
    scatter_column_kernel<<<fill_grid(ctx, t.rows), 256, 0, ctx.stream>>>(all_keys.keys.as<unsigned long long>(), all_keys.rows,
                                                                         t.keys.as<unsigned long long>(), t.counts.as<uint32_t>(), t.rows, column);
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

namespace {

// Decodes a packed random-barcode key (random_kernel's layout) to text.
std::string decode_key(unsigned long long lo, unsigned long long hi, int len, bool wide) {
    unsigned long long H, L, N;
    if (!wide) {
        H = lo & ((1ull << 21) - 1);
        L = (lo >> 21) & ((1ull << 21) - 1);
        N = (lo >> 42) & ((1ull << 21) - 1);
    } else {
        const unsigned long long m42 = (1ull << 42) - 1;
        H = lo & m42;
        L = ((lo >> 42) | (hi << 22)) & m42;
        N = (hi >> 20) & m42;
    }
    std::string s(len, 'A');
    for (int i = 0; i < len; ++i) {
        if ((N >> i) & 1ull) {
            s[i] = 'N';
        } else {
            s[i] = "ACGT"[(((H >> i) & 1ull) << 1) | ((L >> i) & 1ull)];
        }
    }
    return s;
}

} // namespace

} // namespace scg

using namespace scg;

extern "C" {

} // extern "C"

namespace scg {

// countRandomBarcodes over one reader.  Barcodes of up to 21 bases, none taken from raw read text, stay on the device as a
// sorted table (rank-coded, text order); any other result is rendered on the host.
void count_random_reader(Context& c, FastqReader* reader, const RandomMatcher& m, int nthreads, SparseCounts& result) {
    const TemplateSpec& tmpl = m.tmpl;
    const int key_len = m.key_len;
    const bool wide = m.wide;

    c.ensure_ready();
    CountTable tab;
    tab.init(c, wide, wide ? (1u << 20) : (1u << 23));   // 8 M slots (128 MB) to start with: a few million distinct barcodes need no rehash
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
    std::unique_ptr<scg_result> r(new scg_result);
    r->width = key_len;
    if (!wide) {
        // barcodes of up to 21 bases: sorted as text ON THE DEVICE (radix sort of rank-coded keys)
        SortedTable sorted;
        tab.sorted(c, key_len, sorted);
        if (extra.empty()) {
            result.table = std::move(sorted);
            c.timing.harvest_s = now_s() - t_harvest;
            return;
        }
        {
            // a few keys came from raw read text (lower case, IUPAC letters): merged on the host in text order
            const size_t n = sorted.rows;
            std::vector<unsigned long long> order_keys(n);
            std::vector<uint32_t> cnt(n);
            if (n) {
                SCG_CUDA_CHECK(cudaMemcpyAsync(order_keys.data(), sorted.keys.ptr, n * 8, cudaMemcpyDeviceToHost, c.stream));
                SCG_CUDA_CHECK(cudaMemcpyAsync(cnt.data(), sorted.counts.ptr, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, c.stream));
                SCG_CUDA_CHECK(cudaStreamSynchronize(c.stream));
            }
            auto render = [&](unsigned long long k, char* out) {
                for (int b = key_len - 1; b >= 0; --b) {
                    out[b] = "ACGNT"[k & 7ull];
                    k >>= 3;
                }
            };
            r->strings.reserve((n + extra.size()) * (size_t)key_len);
            r->freq.reserve(n + extra.size());
            std::string cur(key_len, ' ');
            auto it = extra.begin();
            auto emit = [&](const std::string& k, int f) {
                r->strings.insert(r->strings.end(), k.begin(), k.end());
                r->freq.push_back(f);
            };
            for (size_t i = 0; i < n; ++i) {
                render(order_keys[i], &cur[0]);
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
        }
    } else {
        std::vector<unsigned long long> lo, hi;
        std::vector<uint32_t> cnt;
        tab.download(c, lo, hi, cnt);
        std::map<std::string, int> merged(std::move(extra));
        for (size_t i = 0; i < lo.size(); ++i) merged[decode_key(lo[i], hi[i], key_len, wide)] += (int)cnt[i];
        r->strings.reserve(merged.size() * (size_t)key_len);
        r->freq.reserve(merged.size());
        for (const auto& kv : merged) {  // std::map iterates in byte order = R's order(sequences) for ACGTN text
            r->strings.insert(r->strings.end(), kv.first.begin(), kv.first.end());
            r->freq.push_back(kv.second);
        }
    }
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
