// Launchers of the dual / combinatorial / random-barcode kernels -- the run-time specialised ones of spec_handlers.cuh
// with their follow-up kernels where the batch allows, the generic ones of handlers.cuh otherwise -- and the resident
// plans of include/scg.h built on them (scg_dual_plan_*, scg_combo_plan_*, scg_random_plan_*).
#include <algorithm>
#include <cstring>
#include <sstream>

#include "api_common.hpp"
#include "handlers.cuh"
#include "jit.hpp"
#include "launchers.hpp"
#include "matchers.hpp"

namespace scg {

// ---------------------------------------------------------------------------------------
// follow-up kernels of the specialised handlers: LOOKUPS ONLY, on the keys the main kernel left in its deferred list
// ---------------------------------------------------------------------------------------

// countDualBarcodes: the segmented mismatch-tolerant search (SegmentedBarcodeSearch<2>::search after its exact probe,
// BarcodeSearch.hpp:478-487) for pairs whose concatenated key missed the exact table or holds an N.
template <int KW>
__global__ void __launch_bounds__(128) dual_deferred_kernel(DeferredList def, const LibDev* __restrict__ lib, int32_t* __restrict__ counts,
                                                            int32_t* __restrict__ out_index) {
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t r = warp; r < def.regions; r += nwarps) {
        const uint32_t cnt = def.warp_counts[r];
        for (uint32_t e0 = 0; e0 < cnt; e0 += 32) {
            const uint32_t e = e0 + lane;
            if (e >= cnt) continue;
            const unsigned long long at = (unsigned long long)r * def.per_warp + e;
            const uint32_t i = def.words[at], x = def.words[def.stride + at], y = def.words[2 * def.stride + at],
                           z = def.words[3 * def.stride + at], n_lo = def.words[4 * def.stride + at], w = def.words[5 * def.stride + at];
            Key<KW> q;
            q.h[0] = x;
            q.l[0] = y;
            q.n[0] = n_lo;
            if (KW > 1) {
                q.h[KW - 1] = z & 0xFFFFu;
                q.l[KW - 1] = z >> 16;
                q.n[KW - 1] = w & 0xFFFFu;
            }
            const Hit h = lookup_segmented_inexact<KW>(lib, q, (int)((w >> 16) & 0xFFu), (int)(w >> 24));
            if (h.index >= 0) atomicAdd(counts + h.index, 1);
            if (out_index) out_index[i] = h.index;
        }
    }
}

// The same search with its dependent chains flattened (libdev.hpp DualFlat; budgets of at most one mismatch per read): the
// root-rule probe and the seed buckets of ALL seeds are requested together, each bucket arriving with its first candidate; only
// a bucket with several candidates costs further loads.  Outcomes equal lookup_segmented_inexact's.
template <int KW>
__global__ void __launch_bounds__(128) dual_deferred_flat_kernel(DeferredList def, DualFlat F, int32_t* __restrict__ counts,
                                                                 int32_t* __restrict__ out_index) {
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t r = warp; r < def.regions; r += nwarps) {
        const uint32_t cnt = def.warp_counts[r];
        for (uint32_t e0 = 0; e0 < cnt; e0 += 32) {
            const uint32_t e = e0 + lane;
            if (e >= cnt) continue;
            const unsigned long long at = (unsigned long long)r * def.per_warp + e;
            const uint32_t i = def.words[at], x = def.words[def.stride + at], y = def.words[2 * def.stride + at],
                           z = def.words[3 * def.stride + at], n_lo = def.words[4 * def.stride + at], w = def.words[5 * def.stride + at];
            const uint32_t zh = KW > 1 ? (z & 0xFFFFu) : 0u, zl = KW > 1 ? (z >> 16) : 0u, n_hi = KW > 1 ? (w & 0xFFFFu) : 0u;
            const int c1 = min((int)((w >> 16) & 0xFFu), F.seg1), c2 = min((int)(w >> 24), F.L - F.seg1);
            int index = -1;
            if (c1 > 0 || c2 > 0) {
                // root rule (SURVEY 8.1 T8): second cap 0, first cap 1 -- the exact chain down to the last base makes the search miss
                bool phantom = false;
                if (c2 == 0 && c1 >= 1) {
                    uint32_t ph[KW], pl[KW], pn = 0;
                    const int lw = (F.L - 1) >> 5;
                    const uint32_t lastbit = 1u << ((F.L - 1) & 31);
                    ph[0] = x;
                    pl[0] = y;
                    uint32_t nn0 = n_lo, nn1 = n_hi;
                    if (KW > 1) {
                        ph[KW - 1] = zh;
                        pl[KW - 1] = zl;
                    }
                    if (lw == 0) {
                        ph[0] &= ~lastbit;
                        pl[0] &= ~lastbit;
                        nn0 &= ~lastbit;
                    } else if (KW > 1) {
                        ph[KW - 1] &= ~lastbit;
                        pl[KW - 1] &= ~lastbit;
                        nn1 &= ~lastbit;
                    }
                    pn = nn0 | nn1;
                    phantom = !pn && probe_table<KW>(F.prefix_slots, F.prefix_mask, F.slot_words, F.kw, ph, pl) >= 0;
                }
                if (!phantom) {
                    uint4 first[4], meta[4];
#pragma unroll
                    for (int sd = 0; sd < 4; ++sd) {
                        first[sd] = meta[sd] = make_uint4(0, 0, 0, 0);
                        if (sd < F.nseeds) {
                            const uint32_t mlo = F.seed_lo[sd], mhi = F.seed_hi[sd];
                            if (!((n_lo & mlo) | (n_hi & mhi))) {   // an N inside the seed: no row agrees with the key there
                                uint32_t mh[KW], ml[KW];
                                mh[0] = x & mlo;
                                ml[0] = y & mlo;
                                if (KW > 1) {
                                    mh[KW - 1] = zh & mhi;
                                    ml[KW - 1] = zl & mhi;
                                }
                                const uint32_t b = hash_key(mh, ml, F.kw, 0x5EED0000u + sd) & F.bucket_mask;
                                const uint4* __restrict__ bucket = F.ibuckets + 2 * ((size_t)sd * (F.bucket_mask + 1) + b);
                                first[sd] = __ldg(bucket);
                                meta[sd] = __ldg(bucket + 1);
                            }
                        }
                    }
                    int best = c1 + c2 + 1, bidx = -1;
                    bool ambiguous = false;
                    auto consider = [&](const uint4 row) {
                        const uint32_t dlo = (row.x ^ x) | (row.y ^ y) | n_lo;
                        const uint32_t dhi = KW > 1 ? (((row.z & 0xFFFFu) ^ zh) | ((row.z >> 16) ^ zl) | n_hi) : 0u;
                        const int d1 = __popc(dlo & F.seg1_lo) + __popc(dhi & F.seg1_hi);
                        const int d2 = __popc(dlo & ~F.seg1_lo) + __popc(dhi & ~F.seg1_hi);
                        if (d1 > c1 || d2 > c2) return;
                        const int d = d1 + d2;
                        if (d > best) return;
                        const int idx = (int)row.w;
                        if (d < best) {
                            best = d;
                            bidx = idx;
                            ambiguous = false;
                        } else if (idx != bidx) {
                            if (F.dup_first) {
                                bidx = min(bidx, idx);
                            } else {
                                ambiguous = true;
                            }
                        }
                    };
#pragma unroll
                    for (int sd = 0; sd < 4; ++sd) {
                        if (meta[sd].y == 0) continue;
                        consider(first[sd]);
                        for (uint32_t c = 1; c < meta[sd].y; ++c) consider(__ldg(F.rows + (size_t)sd * F.nentries + meta[sd].x + c));
                    }
                    if (bidx >= 0 && !ambiguous) index = bidx;
                }
            }
            if (index >= 0) atomicAdd(counts + index, 1);
            if (out_index) out_index[i] = index;
        }
    }
}

// Best-unique bookkeeping of the mismatch-tolerant search over candidate rows (h, l, pool index, -): the rules of
// MismatchTrie.hpp:266-343 as lookup_seeded_body applies them.
struct BestRow {
    int dist, index;
    bool ambiguous;
    __device__ __forceinline__ void consider(const uint4 row, uint32_t kh, uint32_t kl, uint32_t kn, int cap, bool valid, bool dup_first) {
        if (!valid) return;
        const int d = __popc((row.x ^ kh) | (row.y ^ kl) | kn);
        if (d > cap || d > dist) return;
        const int idx = (int)row.z;
        if (d < dist) {
            dist = d;
            index = idx;
            ambiguous = false;
        } else if (idx != index) {
            if (dup_first) {
                index = min(index, idx);
            } else {
                ambiguous = true;
            }
        }
    }
};

// countComboBarcodes with libraries of one word per plane, two seeds and inline buckets (a budget of one mismatch -- the
// usual design): the same search as combo_deferred_kernel with the dependent chains flattened.  The exact probes of BOTH
// regions go out together (four loads), then the seed buckets of every region that missed (up to four loads, each carrying
// its first candidate); only a bucket with more than one candidate costs further loads.  Two round trips to the tables
// where the generic search walks bucket -> candidate list -> entry keys -> entry index per seed and per region.
__global__ void __launch_bounds__(128) combo_deferred_flat_kernel(DeferredList def, ComboParams P, ComboSink sink, int32_t* __restrict__ out_pairs) {
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t r = warp; r < def.regions; r += nwarps) {
        const uint32_t cnt = def.warp_counts[r];
        for (uint32_t e0 = 0; e0 < cnt; e0 += 32) {
            const uint32_t e = e0 + lane;
            if (e >= cnt) continue;
            const unsigned long long at = (unsigned long long)r * def.per_warp + e;
            const uint32_t i = def.words[at], m = def.words[def.stride + at];
            const bool rev = (m & 0x100u) != 0;
            const int obs0 = (int)(m & 0xFFu);
            uint32_t kh[2], kl[2], kn[2];
#pragma unroll
            for (int reg = 0; reg < 2; ++reg) {
                kh[reg] = def.words[(2 + 3 * reg) * def.stride + at];
                kl[reg] = def.words[(3 + 3 * reg) * def.stride + at];
                kn[reg] = def.words[(4 + 3 * reg) * def.stride + at];
            }
            const LibDev* __restrict__ libs = P.libs + (rev ? 2 : 0);
            // ---- round 1: exact probes of both regions ----
            uint4 ea[2], eb[2];
#pragma unroll
            for (int reg = 0; reg < 2; ++reg) {
                ea[reg] = eb[reg] = make_uint4(0, 0, 0xFFFFFFFFu, 0);
                if (kn[reg] == 0) {
                    const uint4* __restrict__ slots = reinterpret_cast<const uint4*>(libs[reg].slots);
                    const uint32_t mask = libs[reg].slot_mask;
                    const uint32_t acc = hash_key(&kh[reg], &kl[reg], 1, 0);
                    ea[reg] = __ldg(slots + (acc & mask));
                    eb[reg] = __ldg(slots + (size_t)(mask + 1) + (hash_second(acc) & mask));
                }
            }
            int exact[2];
#pragma unroll
            for (int reg = 0; reg < 2; ++reg) {
                const int ra = (kn[reg] == 0 && ea[reg].x == kh[reg] && ea[reg].y == kl[reg]) ? (int)ea[reg].z : -1;
                const int rb = (kn[reg] == 0 && eb[reg].x == kh[reg] && eb[reg].y == kl[reg]) ? (int)eb[reg].z : -1;
                exact[reg] = max(ra, rb);
            }
            // ---- round 2: the seed buckets (first candidate inline) of the regions that missed ----
            const int cap0 = P.max_mm - obs0;
            uint4 first[2][2];
            uint2 bk[2][2];
#pragma unroll
            for (int reg = 0; reg < 2; ++reg) {
                const bool search = exact[reg] < 0 && cap0 >= 1 && __popc(kn[reg]) <= cap0;
                const uint32_t bmask = libs[reg].bucket_mask;
#pragma unroll
                for (int sd = 0; sd < 2; ++sd) {
                    first[reg][sd] = make_uint4(0, 0, 0, 0);
                    const uint32_t sm = __ldg(libs[reg].seed_masks + sd);
                    const uint32_t mh = kh[reg] & sm, ml = kl[reg] & sm;
                    if (search && !(kn[reg] & sm)) {
                        const uint32_t b = hash_key(&mh, &ml, 1, 0x5EED0000u + sd) & bmask;
                        first[reg][sd] = __ldg(libs[reg].ibuckets + (size_t)sd * (bmask + 1) + b);
                    }
                    bk[reg][sd] = make_uint2(first[reg][sd].w & 0xFFFFFFu, first[reg][sd].w >> 24);
                }
            }
            // ---- the regions in read order with the shared budget (find_match, :149-186) ----
            int obs = obs0;
            int ids[2] = { -1, -1 };
            bool ok = true;
#pragma unroll
            for (int reg = 0; reg < 2; ++reg) {
                if (!ok) continue;
                int found = exact[reg], dist = 0;
                if (found < 0) {
                    const int cap = min(P.max_mm - obs, libs[reg].L);
                    if (cap >= 1 && __popc(kn[reg]) <= cap) {
                        const bool dup_first = libs[reg].dup_first != 0;
                        BestRow best{ cap + 1, -1, false };
#pragma unroll
                        for (int sd = 0; sd < 2; ++sd) {
                            best.consider(first[reg][sd], kh[reg], kl[reg], kn[reg], cap, bk[reg][sd].y > 0, dup_first);
                            for (uint32_t c = 1; c < bk[reg][sd].y; ++c) {
                                best.consider(__ldg(libs[reg].cand_rows + (size_t)sd * libs[reg].nentries + bk[reg][sd].x + c), kh[reg], kl[reg],
                                              kn[reg], cap, true, dup_first);
                            }
                        }
                        if (best.index >= 0 && !best.ambiguous) {
                            found = best.index;
                            dist = best.dist;
                        }
                    }
                }
                if (found < 0) {
                    ok = false;
                } else {
                    obs += dist;
                    ids[rev ? 1 - reg : reg] = found;
                }
            }
            if (ok) combo_count(sink, ids[0], ids[1]);
            if (out_pairs) __stcs(reinterpret_cast<int2*>(out_pairs) + i, ok ? make_int2(ids[0], ids[1]) : make_int2(-1, -1));
        }
    }
}

// countComboBarcodes: both regions of the read's one verified window through the mismatch-tolerant lookups, in read
// order with the shared budget (find_match, handlers/CombinatorialBarcodesSingleEnd.hpp:149-186).
__global__ void __launch_bounds__(128) combo_deferred_kernel(DeferredList def, ComboParams P, ComboSink sink, int32_t* __restrict__ out_pairs) {
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t r = warp; r < def.regions; r += nwarps) {
        const uint32_t cnt = def.warp_counts[r];
        for (uint32_t e0 = 0; e0 < cnt; e0 += 32) {
            const uint32_t e = e0 + lane;
            if (e >= cnt) continue;
            const unsigned long long at = (unsigned long long)r * def.per_warp + e;
            const uint32_t i = def.words[at], m = def.words[def.stride + at];
            const bool rev = (m & 0x100u) != 0;
            int obs = (int)(m & 0xFFu);
            int ids[2] = { -1, -1 };
            bool ok = true;
#pragma unroll
            for (int reg = 0; reg < 2; ++reg) {
                if (!ok) continue;
                Key<1> key;
                key.h[0] = def.words[(2 + 3 * reg) * def.stride + at];
                key.l[0] = def.words[(3 + 3 * reg) * def.stride + at];
                key.n[0] = def.words[(4 + 3 * reg) * def.stride + at];
                const Hit h = lookup_any<1>(P.libs + (rev ? 2 : 0) + reg, key, P.max_mm - obs);
                if (h.index < 0) {
                    ok = false;
                } else {
                    obs += h.dist;
                    ids[rev ? 1 - reg : reg] = h.index;
                }
            }
            if (ok) combo_count(sink, ids[0], ids[1]);
            if (out_pairs) {
                out_pairs[2 * (size_t)i] = ok ? ids[0] : -1;
                out_pairs[2 * (size_t)i + 1] = ok ? ids[1] : -1;
            }
        }
    }
}

// countRandomBarcodes: the barcodes the main kernel did not find in their home sector -- new ones, and ones a collision
// pushed further along -- inserted (or found) with the full probing loop.  Every entry is independent of every other, so the
// compare-and-swap round trips of thousands of lanes overlap; new keys are added up per warp before they reach the
// table's counter of distinct keys.
// U barcodes per lane through the count table at once: the two slots of every barcode's home sector are requested together
// (bucketised linear probing, count_table.cuh), then the sector's slots are visited in probing order -- a match is counted, an
// empty slot claimed by compare-and-swap (the claims of the U barcodes overlap) -- and only a barcode whose home sector is taken
// by two others walks on, slot by slot.  Returns the number of new keys this lane inserted.
template <int U>
__device__ __forceinline__ unsigned int count_batch(const CountTable64& table, const unsigned long long (&key)[U], const bool (&valid)[U]) {
    unsigned long long pos[U], ka[U], kb[U];
    int at[U];   // -1: not settled yet, 0 / 1: the barcode's slot is home + 0 / 1
    unsigned int fresh = 0;
#pragma unroll
    for (int u = 0; u < U; ++u) {
        pos[u] = count_home(table, key[u]);
        ka[u] = kb[u] = 0ull;
        at[u] = -1;
        if (valid[u]) {
            // the home sector (two 16-byte slots, 32 aligned bytes) in ONE 256-bit load: half the requests of two 8-byte loads
            uint32_t w0, w1, w2, w3, w4, w5, w6, w7;
            asm volatile("ld.global.cg.v8.u32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                         : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3), "=r"(w4), "=r"(w5), "=r"(w6), "=r"(w7)
                         : "l"(table.slots + pos[u]));
            ka[u] = (unsigned long long)w0 | ((unsigned long long)w1 << 32);
            kb[u] = (unsigned long long)w4 | ((unsigned long long)w5 << 32);
        }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        if (!valid[u]) continue;
        if (ka[u] == ~0ull) {
            ka[u] = atomicCAS(&table.slots[pos[u]].key, ~0ull, key[u]);
            if (ka[u] == ~0ull) {
                ++fresh;
                ka[u] = key[u];
            }
        }
        if (ka[u] == key[u]) at[u] = 0;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        if (!valid[u] || at[u] >= 0) continue;
        if (kb[u] == ~0ull) {
            kb[u] = atomicCAS(&table.slots[pos[u] + 1].key, ~0ull, key[u]);
            if (kb[u] == ~0ull) {
                ++fresh;
                kb[u] = key[u];
            }
        }
        if (kb[u] == key[u]) at[u] = 1;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        if (!valid[u]) continue;
        if (at[u] >= 0) {
            atomicAdd(&table.slots[pos[u] + (unsigned)at[u]].count, 1u);
        } else {
            const unsigned long long next = (pos[u] + 2) & table.mask;
            if (count_insert64_from(table, key[u], 1u, next, __ldcg(&table.slots[next].key))) ++fresh;
        }
    }
    return fresh;
}

__global__ void __launch_bounds__(256) random_insert_kernel(DeferredList def, CountTable64 table) {
    constexpr int U = 4;   // entries per lane in flight: their slot loads, then their compare-and-swaps, overlap
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
    unsigned long long fresh = 0;
    for (uint32_t r = warp; r < def.regions; r += nwarps) {
        const uint32_t cnt = def.warp_counts[r];
        const unsigned long long base = (unsigned long long)r * def.per_warp;
        for (uint32_t e0 = 0; e0 < cnt; e0 += 32 * U) {
            unsigned long long key[U];
            bool valid[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint32_t e = e0 + 32 * u + lane;
                valid[u] = e < cnt;
                key[u] = valid[u] ? ((unsigned long long)def.words[base + e] | ((unsigned long long)def.words[def.stride + base + e] << 32)) : 0ull;
            }
            fresh += count_batch<U>(table, key, valid);
            __syncwarp();
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) fresh += __shfl_xor_sync(0xFFFFFFFFu, fresh, d);
    if (lane == 0 && fresh) atomicAdd(table.live, fresh);
}

// The same for a wide table (barcodes of 22 to 42 bases): an entry is the 128-bit key in four words, inserted (or found) by
// the full probing loop from its even home (count_add128), the loop the generic kernel's inserts take.
__global__ void __launch_bounds__(256) random_insert128_kernel(DeferredList def, CountTable128 table) {
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
    unsigned long long fresh = 0;
    for (uint32_t r = warp; r < def.regions; r += nwarps) {
        const uint32_t cnt = def.warp_counts[r];
        const unsigned long long base = (unsigned long long)r * def.per_warp;
        for (uint32_t e = lane; e < cnt; e += 32) {
            const unsigned long long at = base + e;
            const ulonglong2 key = make_ulonglong2((unsigned long long)def.words[at] | ((unsigned long long)def.words[def.stride + at] << 32),
                                                   (unsigned long long)def.words[2 * def.stride + at] |
                                                       ((unsigned long long)def.words[3 * def.stride + at] << 32));
            if (count_add128(table, key, 1u)) ++fresh;
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) fresh += __shfl_xor_sync(0xFFFFFFFFu, fresh, d);
    if (lane == 0 && fresh) atomicAdd(table.live, fresh);
}

// countRandomBarcodes, partitioned (libdev.hpp PartitionedKeys): the lists of table part 0 are counted first, then part 1's, ...
// -- regions are numbered part-major and the warps take them in that order, so at any moment the kernel works on one or two
// parts of the table, which stay in L2: the random traffic of the inserts never reaches HBM.  Four keys per lane in flight.
template <int U>
__global__ void __launch_bounds__(256) random_count_parts_kernel(PartitionedKeys parts, CountTable64 table) {
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t nwarps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t regions = parts.nparts * parts.nwarps;
    unsigned long long fresh = 0;
    for (uint32_t r = warp; r < regions; r += nwarps) {
        const uint32_t cnt = parts.counts[r];
        const unsigned long long* __restrict__ list = parts.keys + (size_t)r * parts.cap;
        for (uint32_t e0 = 0; e0 < cnt; e0 += 32 * U) {
            unsigned long long key[U];
            bool valid[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint32_t e = e0 + 32 * u + lane;
                valid[u] = e < cnt;
                key[u] = valid[u] ? __ldcs(list + e) : 0ull;
            }
            fresh += count_batch<U>(table, key, valid);
            __syncwarp();   // lanes that walked a probe sequence rejoin here: the warp stays on one part of the table
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) fresh += __shfl_xor_sync(0xFFFFFFFFu, fresh, d);
    if (lane == 0 && fresh) atomicAdd(table.live, fresh);
}

namespace {

// ---- program text of a specialised handler kernel ----
bool template_fits(const TemplateSpec& t, const ScanSpec& s, const ReadsDev& reads, std::string* why) {
    auto no = [&](const char* msg) {
        if (why) *why = msg;
        return false;
    };
    if (reads.lens != nullptr) return no("reads of different lengths use the generic kernel");
    if (reads.n > 0x7FFFFFC0ll) return no("batch too large for 32-bit read indices");
    const int nwin = reads.uniform_len - t.length + 1;
    if (nwin < 1) return no("reads shorter than the template use the generic kernel");
    if (reads.W > 5) return no("reads longer than 160 bases use the generic kernel");
    if (t.length > 128) return no("templates longer than 128 bases use the generic kernel");
    if (reads.W + 2 < (t.length + 31) / 32 + 1) return no("template too long for the read");
    int nconst = 0;
    for (char ch : t.fwd_seq) nconst += ch != '-';
    if (s.mm < 0 || s.mm > 3 || nconst < 4 * (s.mm + 1)) return no("mismatch budget too large for the pigeonhole filter");
    return true;
}

void template_macros(std::ostringstream& o, const char* P, const TemplateSpec& t, const ScanSpec& s, int maxmm, const ReadsDev& reads) {
    const std::string rb = t.rev ? t.rev_seq : std::string(t.length, '-');
    const std::string fb = t.fwd ? t.fwd_seq : std::string(t.length, '-');
    o << "#define SPH_" << P << "_T " << t.length << "\n"
      << "#define SPH_" << P << "_FB \"" << fb << "\"\n"
      << "#define SPH_" << P << "_RB \"" << rb << "\"\n"
      << "#define SPH_" << P << "_FWD " << (t.fwd ? 1 : 0) << "\n"
      << "#define SPH_" << P << "_REV " << (t.rev ? 1 : 0) << "\n"
      << "#define SPH_" << P << "_MM " << s.mm << "\n"
      << "#define SPH_" << P << "_MAXMM " << maxmm << "\n"
      << "#define SPH_" << P << "_ULEN " << reads.uniform_len << "\n"
      << "#define SPH_" << P << "_W " << reads.W << "\n";
    for (int r = 0; r < s.nreg && r < 2; ++r) {
        o << "#define SPH_" << P << "_FSTART" << r << " " << s.fstart[r] << "\n"
          << "#define SPH_" << P << "_FLEN" << r << " " << s.rlen_f[r] << "\n"
          << "#define SPH_" << P << "_RSTART" << r << " " << s.rstart[r] << "\n"
          << "#define SPH_" << P << "_RLEN" << r << " " << s.rlen_r[r] << "\n";
    }
}

void common_macros(std::ostringstream& o, int kind, int min_blocks, int group, int use_first, int has_index) {
    o << "#define SPH_KIND " << kind << "\n"
      << "#define SPH_MIN_BLOCKS " << jit_env_int("SCG_SPH_MIN_BLOCKS", min_blocks, 1, 16) << "\n"
      << "#define SPH_STAGES " << jit_env_int("SCG_SPH_STAGES", 2, 1, 8) << "\n"
      << "#define SPH_GROUP " << jit_env_int("SCG_SPH_GROUP", group, 1, 8) << "\n"
      << "#define SPH_SAMPLES " << jit_env_int("SCG_SPEC_SAMPLES", 8, 1, 32) << "\n"
      << "#define SPH_USE_FIRST " << use_first << "\n"
      << "#define SPH_HAS_INDEX " << has_index << "\n";
}

// counters of at most this many cells are privatised per block in shared memory (4 bytes a cell: 4 KB keep 8 blocks per SM resident)
int hist_cells(long long cells) {
    const long long most = jit_env_int("SCG_SPEC_HIST_MAX", 1024, 0, 8192);
    return cells > 0 && cells <= most ? (int)((cells + 31) / 32 * 32) : 0;
}

JitProgram dual_program(const TemplateSpec& t1, const ScanSpec& s1, int mm1, const ReadsDev& r1, const TemplateSpec& t2, const ScanSpec& s2,
                        int mm2, const ReadsDev& r2, int use_first, int has_index, int hist) {
    std::ostringstream src;
    common_macros(src, 1, 8, 1, use_first, has_index);
    src << "#define SPH_HIST " << hist << "\n";
    template_macros(src, "A", t1, s1, mm1, r1);
    template_macros(src, "B", t2, s2, mm2, r2);
    src << "#include \"spec_handlers.cuh\"\n";
    JitProgram prog;
    prog.name = "spec_dual_pe_jit.cu";
    prog.text = src.str();
    prog.kernels = { "spec_dual_pe_kernel" };
    return prog;
}

JitProgram combo_program(const TemplateSpec& t, const ScanSpec& s, int mm, const ReadsDev& r, int use_first, int has_index, int hist) {
    std::ostringstream src;
    common_macros(src, 2, 8, 2, use_first, has_index);
    src << "#define SPH_HIST " << hist << "\n";
    template_macros(src, "A", t, s, mm, r);
    src << "#include \"spec_handlers.cuh\"\n";
    JitProgram prog;
    prog.name = "spec_combo_jit.cu";
    prog.text = src.str();
    prog.kernels = { "spec_combo_kernel" };
    return prog;
}

JitProgram random_program(const TemplateSpec& t, const ScanSpec& s, int mm, const ReadsDev& r, int use_first, int has_index, int partitioned) {
    std::ostringstream src;
    common_macros(src, 3, 8, 2, use_first, has_index);
    src << "#define SPH_PARTITIONED " << partitioned << "\n";
    template_macros(src, "A", t, s, mm, r);
    src << "#include \"spec_handlers.cuh\"\n";
    JitProgram prog;
    prog.name = "spec_random_jit.cu";
    prog.text = src.str();
    prog.kernels = { "spec_random_kernel" };
    return prog;
}

bool spec_disabled() {
    const char* env = std::getenv("SCG_NO_SPEC_HANDLERS");
    return env && env[0] && env[0] != '0';
}

// Per-context scratch of the specialised handlers: one region of deferred entries per warp of the launch, the slow list.
struct Scratch {
    DeferredList def;
    SlowList slow;
};
Scratch prepare_scratch(Context& ctx, long long n, int grid, int group, int nwords, cudaStream_t stream) {
    const long long ntiles = (n + TILE - 1) / TILE;
    const long long ngroups = (ntiles + group - 1) / group;
    const long long nwarps = (long long)grid * 4;
    const long long groups_per_warp = (ngroups + nwarps - 1) / nwarps;
    Scratch s;
    s.def.per_warp = (uint32_t)(groups_per_warp * group * TILE);
    s.def.regions = (uint32_t)nwarps;
    s.def.stride = (unsigned long long)nwarps * s.def.per_warp;
    ctx.defer_words.reserve(std::max<size_t>((size_t)nwords * s.def.stride * sizeof(uint32_t), 16));
    ctx.defer_counts.reserve((size_t)nwarps * sizeof(uint32_t));
    ctx.slow_list.reserve((size_t)(ntiles * TILE) * sizeof(uint32_t));
    ctx.slow_count.reserve(sizeof(uint32_t));
    s.def.words = ctx.defer_words.as<uint32_t>();
    s.def.warp_counts = ctx.defer_counts.as<uint32_t>();
    s.slow.list = ctx.slow_list.as<uint32_t>();
    s.slow.count = ctx.slow_count.as<uint32_t>();
    // regions of warps that end up without work keep a count of zero
    SCG_CUDA_CHECK(cudaMemsetAsync(s.def.warp_counts, 0, (size_t)nwarps * sizeof(uint32_t), stream));
    SCG_CUDA_CHECK(cudaMemsetAsync(s.slow.count, 0, sizeof(uint32_t), stream));
    return s;
}

int spec_grid(Context& ctx, cudaKernel_t k, long long n, int group) {
    const long long ntiles = (n + TILE - 1) / TILE;
    const long long ngroups = (ntiles + group - 1) / group;
    const int resident = specialised_blocks_per_sm(k);
    return (int)std::max<long long>(1, std::min<long long>((ngroups + 3) / 4, (long long)ctx.sm_count * resident));
}

int followup_grid(Context& ctx, long long n) {
    const long long ntiles = (n + TILE - 1) / TILE;
    return (int)std::max<long long>(1, std::min<long long>((ntiles + 3) / 4, (long long)ctx.sm_count * 8));
}

} // namespace

// ---------------------------------------------------------------------------------------
// countDualBarcodes, paired-end
// ---------------------------------------------------------------------------------------
static void launch_dual_pe_generic(Context& ctx, const ReadsDev& r1, const ReadsDev& r2, const DualPEMatcher& m, int32_t* d_counts,
                                   int32_t* d_index, ReadList visit, int grid, cudaStream_t stream) {
    const int cb = std::max(m.params.spec1.cbits, m.params.spec2.cbits);
    dispatch_cb(cb, [&](auto CB) {
        dispatch_kw(m.params.kw, [&](auto KW) {
            dual_pe_kernel<decltype(CB)::value, decltype(KW)::value><<<grid, 128, 0, stream>>>(r1, r2, m.params, d_counts, d_index, visit);
        });
    });
    SCG_CUDA_CHECK(cudaGetLastError());
    ++ctx.launches;
    ++ctx.timing.launches;
}

void launch_dual_pe(Context& ctx, const ReadsDev& r1, const ReadsDev& r2, const DualPEMatcher& m, int32_t* d_counts, int32_t* d_index,
                    cudaStream_t stream) {
    if (r1.n <= 0) return;
    const long long ntiles = (r1.n + TILE - 1) / TILE;
    std::string why;
    const JitModule* mod = nullptr;
    int group = 1;
    if (spec_disabled()) {
        why = "disabled by SCG_NO_SPEC_HANDLERS";
    } else if (m.params.randomized) {
        why = "randomized designs use the generic kernel";
    } else if (!m.exact16.ptr || m.exact16_shift == 0) {
        why = "variable regions of more than 48 bases in total use the generic kernel";
    } else if (m.params.len1 > 32 || m.params.len2 > 32) {
        why = "variable regions longer than 32 bases use the generic kernel";
    } else if (template_fits(m.t1, m.params.spec1, r1, &why) && template_fits(m.t2, m.params.spec2, r2, &why)) {
        group = jit_env_int("SCG_SPH_GROUP", 1, 1, 8);
        mod = jit_module(dual_program(m.t1, m.params.spec1, m.params.mm1, r1, m.t2, m.params.spec2, m.params.mm2, r2, m.params.use_first,
                                      d_index ? 1 : 0, hist_cells((long long)m.lib.host.nchoices)),
                         ctx.device, &why);
    }
    if (!mod) {
        launch_dual_pe_generic(ctx, r1, r2, m, d_counts, d_index, ReadList{ nullptr, nullptr }, ctx.grid_for(ntiles), stream);
        ctx.kernel_note = "generic dual_pe_kernel (" + why + ")";
        return;
    }
    cudaKernel_t k = mod->kernels[0];
    const int grid = spec_grid(ctx, k, r1.n, group);
    Scratch sc = prepare_scratch(ctx, r1.n, grid, group, DUAL_DEFER_WORDS, stream);
    ReadsDev a1 = r1, a2 = r2;
    DualTables tb{ m.exact16.as<uint4>(), m.exact16_shift };
    void* args[] = { &a1, &a2, &tb, &d_counts, &d_index, &sc.def, &sc.slow };
    SCG_CUDA_CHECK(cudaLaunchKernel(reinterpret_cast<const void*>(k), dim3(grid), dim3(128), args, 0, stream));
    const int fgrid = followup_grid(ctx, r1.n);
    const bool flat = m.flat.nseeds > 0 && !std::getenv("SCG_DUAL_NO_FLAT");
    if (m.params.kw <= 1) {
        if (flat) {
            dual_deferred_flat_kernel<1><<<fgrid, 128, 0, stream>>>(sc.def, m.flat, d_counts, d_index);
        } else {
            dual_deferred_kernel<1><<<fgrid, 128, 0, stream>>>(sc.def, m.params.lib, d_counts, d_index);
        }
    } else {
        if (flat) {
            dual_deferred_flat_kernel<2><<<fgrid, 128, 0, stream>>>(sc.def, m.flat, d_counts, d_index);
        } else {
            dual_deferred_kernel<2><<<fgrid, 128, 0, stream>>>(sc.def, m.params.lib, d_counts, d_index);
        }
    }
    SCG_CUDA_CHECK(cudaGetLastError());
    ctx.launches += 2;
    ctx.timing.launches += 2;
    // pairs with several verified windows: the full per-pair search of the generic kernel on exactly those
    launch_dual_pe_generic(ctx, r1, r2, m, d_counts, d_index, ReadList{ sc.slow.list, sc.slow.count }, ctx.sm_count * 2, stream);
    ctx.kernel_note = "specialised (NVRTC) spec_dual_pe_kernel, filter+verify on both mates, " + std::to_string(specialised_blocks_per_sm(k)) +
                      " blocks/SM; + " + (flat ? "dual_deferred_flat_kernel" : "dual_deferred_kernel") + " (mismatch lookups) + dual_pe_kernel on the multi-window pairs";
}

// ---------------------------------------------------------------------------------------
// countComboBarcodes, single-end
// ---------------------------------------------------------------------------------------
static void launch_combo_generic(Context& ctx, const ReadsDev& reads, const ComboParams& P, const ComboSink& sink, const int32_t* skip_if_found,
                                 int32_t* out_pairs, ReadList visit, int grid, cudaStream_t stream) {
    dispatch_cb(P.spec.cbits, [&](auto CB) {
        dispatch_kw(P.kw, [&](auto KW) {
            combo_kernel<decltype(CB)::value, decltype(KW)::value><<<grid, 128, 0, stream>>>(reads, P, sink, skip_if_found, out_pairs, visit);
        });
    });
    SCG_CUDA_CHECK(cudaGetLastError());
    ++ctx.launches;
    ++ctx.timing.launches;
}

void launch_combo(Context& ctx, const ReadsDev& reads, const ComboMatcher& m, const ComboSink& sink, const int32_t* skip_if_found,
                  int32_t* out_pairs, cudaStream_t stream) {
    if (reads.n <= 0) return;
    const long long ntiles = (reads.n + TILE - 1) / TILE;
    const ComboParams& P = m.params;
    std::string why;
    const JitModule* mod = nullptr;
    int group = 2;
    bool ok = !spec_disabled();
    if (!ok) why = "disabled by SCG_NO_SPEC_HANDLERS";
    if (ok && skip_if_found) {
        ok = false;
        why = "the diagnostics pass uses the generic kernel";
    }
    if (ok && P.kw > 1) {
        ok = false;
        why = "variable regions longer than 32 bases use the generic kernel";
    }
    if (ok) ok = template_fits(m.tmpl, P.spec, reads, &why);
    if (ok) {
        group = jit_env_int("SCG_SPH_GROUP", 2, 1, 8);
        mod = jit_module(combo_program(m.tmpl, P.spec, P.max_mm, reads, P.use_first, out_pairs ? 1 : 0,
                                       sink.dense ? hist_cells((long long)P.n1 * P.n2) : 0),
                         ctx.device, &why);
    }
    if (!mod) {
        launch_combo_generic(ctx, reads, P, sink, skip_if_found, out_pairs, ReadList{ nullptr, nullptr }, ctx.grid_for(ntiles), stream);
        ctx.kernel_note = "generic combo_kernel (" + why + ")";
        return;
    }
    cudaKernel_t k = mod->kernels[0];
    const int grid = spec_grid(ctx, k, reads.n, group);
    Scratch sc = prepare_scratch(ctx, reads.n, grid, group, COMBO_DEFER_WORDS, stream);
    ReadsDev a = reads;
    ComboTables tb;
    std::memset(&tb, 0, sizeof tb);
    for (int l = 0; l < 4; ++l) {
        const bool used = l < 2 ? m.tmpl.fwd : m.tmpl.rev;
        if (!used) continue;
        tb.slots[l] = reinterpret_cast<const uint4*>(m.lib[l].dev.slots);
        tb.mask[l] = m.lib[l].dev.slot_mask;
    }
    ComboSink sk = sink;
    void* args[] = { &a, &tb, &sk, &out_pairs, &sc.def, &sc.slow };
    SCG_CUDA_CHECK(cudaLaunchKernel(reinterpret_cast<const void*>(k), dim3(grid), dim3(128), args, 0, stream));
    ++ctx.launches;
    ++ctx.timing.launches;
    if (P.max_mm > 0) {
        // libraries of one word per plane with two seeds and inline buckets (a budget of one mismatch): the flattened search
        bool flat = P.max_mm == 1 && !std::getenv("SCG_COMBO_NO_FLAT");
        for (int k = 0; k < 4 && flat; ++k) {
            const bool used = k < 2 ? m.tmpl.fwd : m.tmpl.rev;
            if (used) flat = m.lib[k].dev.KW == 1 && m.lib[k].dev.nseeds == 2 && m.lib[k].dev.ibuckets != nullptr && m.lib[k].dev.slot_words == 4;
        }
        if (flat) {
            combo_deferred_flat_kernel<<<followup_grid(ctx, reads.n), 128, 0, stream>>>(sc.def, P, sink, out_pairs);
        } else {
            combo_deferred_kernel<<<followup_grid(ctx, reads.n), 128, 0, stream>>>(sc.def, P, sink, out_pairs);
        }
        SCG_CUDA_CHECK(cudaGetLastError());
        ++ctx.launches;
        ++ctx.timing.launches;
    }
    launch_combo_generic(ctx, reads, P, sink, nullptr, out_pairs, ReadList{ sc.slow.list, sc.slow.count }, ctx.sm_count * 2, stream);
    ctx.kernel_note = "specialised (NVRTC) spec_combo_kernel, filter+verify, " + std::to_string(specialised_blocks_per_sm(k)) + " blocks/SM" +
                      (P.max_mm > 0 ? "; + combo_deferred_kernel (mismatch lookups)" : "") + " + combo_kernel on the multi-window reads";
}

// ---------------------------------------------------------------------------------------
// countRandomBarcodes
// ---------------------------------------------------------------------------------------
static void launch_random_generic(Context& ctx, const ReadsDev& reads, const RandomMatcher& m, CountTable& tab, const uint8_t* odd,
                                  OddOutcome* odd_out, unsigned long long* odd_count, int32_t* out_index, ReadList visit, int grid,
                                  cudaStream_t stream) {
    const RandomParams& P = m.params;
    CountTable64 t64 = m.wide ? CountTable64{ nullptr, 0, nullptr } : tab.view64();
    CountTable128 t128 = m.wide ? tab.view128() : CountTable128{ nullptr, nullptr, 0, nullptr };
    CountTableLong tl{};
    dispatch_cb(P.spec.cbits, [&](auto CB) {
        if (m.key_len <= 32) {
            random_kernel<decltype(CB)::value, 1><<<grid, 128, 0, stream>>>(reads, P, t64, t128, tl, odd, 0, odd_out, odd_count, out_index, visit);
        } else {
            random_kernel<decltype(CB)::value, 2><<<grid, 128, 0, stream>>>(reads, P, t64, t128, tl, odd, 0, odd_out, odd_count, out_index, visit);
        }
    });
    SCG_CUDA_CHECK(cudaGetLastError());
    ++ctx.launches;
    ++ctx.timing.launches;
}

// Barcodes of 43 bases or more: the generic kernel into the long-key table (libdev.hpp CountTableLong), over slices of at most
// LONG_SLICE_READS reads, each followed by the kernel that moves its fresh keys from the staging rows into the key store -- so the
// staging buffer holds one slice (at most 2^21 rows of up to 13 words, 208 MiB) however many reads the batch has.
static constexpr long long LONG_SLICE_READS = 1ll << 21;

static void launch_random_long(Context& ctx, const ReadsDev& reads, const RandomMatcher& m, CountTable& tab, const uint8_t* odd,
                               OddOutcome* odd_out, unsigned long long* odd_count, int32_t* out_index, cudaStream_t stream) {
    const RandomParams& P = m.params;
    const CountTable64 t64{ nullptr, 0, nullptr };
    const CountTable128 t128{ nullptr, nullptr, 0, nullptr };
    for (long long first = 0; first < reads.n; first += LONG_SLICE_READS) {
        // a slice starts on a tile boundary (LONG_SLICE_READS is a multiple of TILE)
        ReadsDev slice = reads;
        slice.n = std::min(LONG_SLICE_READS, reads.n - first);
        slice.data = reads.data + (size_t)(first / TILE) * tile_words(reads.W);
        if (reads.lens) slice.lens = reads.lens + first;
        const CountTableLong tl = tab.view_long((size_t)slice.n);
        const uint8_t* slice_odd = odd ? odd + first : nullptr;
        int32_t* slice_index = out_index ? out_index + first : nullptr;
        const int grid = ctx.grid_for((slice.n + TILE - 1) / TILE);
        dispatch_cb(P.spec.cbits, [&](auto CB) {
            if (m.key_len <= 64) {
                random_kernel<decltype(CB)::value, 2><<<grid, 128, 0, stream>>>(slice, P, t64, t128, tl, slice_odd, first, odd_out, odd_count, slice_index,
                                                                                ReadList{ nullptr, nullptr });
            } else {
                random_kernel<decltype(CB)::value, 8><<<grid, 128, 0, stream>>>(slice, P, t64, t128, tl, slice_odd, first, odd_out, odd_count, slice_index,
                                                                                ReadList{ nullptr, nullptr });
            }
        });
        SCG_CUDA_CHECK(cudaGetLastError());
        ++ctx.launches;
        ++ctx.timing.launches;
        tab.promote_fresh(ctx, stream);
    }
}

void launch_random(Context& ctx, const ReadsDev& reads, const RandomMatcher& m, CountTable& tab, const uint8_t* odd, OddOutcome* odd_out,
                   unsigned long long* odd_count, int32_t* out_index, cudaStream_t stream) {
    if (reads.n <= 0) return;
    if (m.long_words) {
        launch_random_long(ctx, reads, m, tab, odd, odd_out, odd_count, out_index, stream);
        ctx.kernel_note = "generic random_kernel into the long-key count table (barcodes of " + std::to_string(m.key_len) +
                          " bases: staged keys, tag claims, promote_fresh_kernel)";
        return;
    }
    const long long ntiles = (reads.n + TILE - 1) / TILE;
    std::string why;
    const JitModule* mod = nullptr;
    int group = 2;
    int nparts = 0;
    bool ok = !spec_disabled();
    if (!ok) why = "disabled by SCG_NO_SPEC_HANDLERS";
    if (ok) ok = template_fits(m.tmpl, m.params.spec, reads, &why);
    if (ok) {
        group = jit_env_int("SCG_SPH_GROUP", 2, 1, 8);
        // a table too large to live in L2 is filled part by part (libdev.hpp PartitionedKeys); SCG_RANDOM_PARTS = 0 / 2..32 overrides
        const size_t table_bytes = tab.capacity * sizeof(CountSlot);
        nparts = 0;
        if (table_bytes > ((size_t)48 << 20)) {
            nparts = 2;
            while (nparts < 32 && table_bytes / (size_t)nparts > ((size_t)12 << 20)) nparts *= 2;
        }
        if (const char* env = std::getenv("SCG_RANDOM_PARTS")) {
            const int want = std::atoi(env);
            nparts = want <= 1 ? 0 : 2;
            while (nparts && nparts < std::min(want, 32)) nparts *= 2;
        }
        while (nparts > 0 && (size_t)nparts * 2 > tab.capacity) nparts /= 2;
        if (nparts < 2 || m.wide) nparts = 0;   // a wide table takes the home-sector route at every size
        mod = jit_module(random_program(m.tmpl, m.params.spec, m.params.max_mm, reads, m.params.use_first, out_index ? 1 : 0, nparts ? 1 : 0),
                         ctx.device, &why);
    }
    if (!mod) {
        launch_random_generic(ctx, reads, m, tab, odd, odd_out, odd_count, out_index, ReadList{ nullptr, nullptr }, ctx.grid_for(ntiles), stream);
        ctx.kernel_note = "generic random_kernel (" + why + ")";
        return;
    }
    cudaKernel_t k = mod->kernels[0];
    const int grid = spec_grid(ctx, k, reads.n, group);
    // (the partitioned route keeps its key lists where the other route keeps its deferred entries: two words per read at most)
    Scratch sc = prepare_scratch(ctx, reads.n, grid, group, nparts ? 0 : (m.wide ? 4 : 2), stream);
    SlowList slow = sc.slow;
    ReadsDev a = reads;
    CountTable64 t64 = tab.view64();
    CountTable128 t128 = tab.view128();
    long long read_offset = 0;
    PartitionedKeys parts{ nullptr, nullptr, 0, 0, 0, 0 };
    if (nparts) {
        // a warp's reads spread evenly over the parts (the part is a hash of the barcode): half as much again, and a margin
        const unsigned long long per_warp = sc.def.per_warp;
        parts.nwarps = sc.def.regions;
        parts.nparts = (uint32_t)nparts;
        parts.cap = (uint32_t)(per_warp / (unsigned)nparts + per_warp / (2u * (unsigned)nparts) + 64);
        ctx.part_keys.reserve((size_t)parts.cap * parts.nparts * parts.nwarps * sizeof(unsigned long long));
        int log2cap = 0;
        while (((size_t)1 << log2cap) < tab.capacity) ++log2cap;
        int log2parts = 0;
        while ((1 << log2parts) < nparts) ++log2parts;
        parts.shift = (uint32_t)(log2cap - log2parts);
        parts.keys = ctx.part_keys.as<unsigned long long>();
        ctx.part_counts.reserve((size_t)parts.nparts * parts.nwarps * sizeof(uint32_t));
        parts.counts = ctx.part_counts.as<uint32_t>();
        SCG_CUDA_CHECK(cudaMemsetAsync(parts.counts, 0, (size_t)parts.nparts * parts.nwarps * sizeof(uint32_t), stream));
    }
    void* table_arg = m.wide ? static_cast<void*>(&t128) : static_cast<void*>(&t64);
    void* args[] = { &a, table_arg, &odd, &read_offset, &odd_out, &odd_count, &out_index, &sc.def, &slow, &parts };
    SCG_CUDA_CHECK(cudaLaunchKernel(reinterpret_cast<const void*>(k), dim3(grid), dim3(128), args, 0, stream));
    if (nparts) {
        // exactly the blocks that are resident together: every warp then walks the parts in the same order at the same pace, and
        // the slices of the table pass through L2 one after the other
        // (keys per lane in flight: SCG_RANDOM_UNROLL = 2 / 4 / 8, measured in DESIGN.md 5.2)
        static const int unroll = jit_env_int("SCG_RANDOM_UNROLL", 4, 2, 8);
        auto launch = [&](auto kernel) {
            int blocks_per_sm = 0;
            SCG_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kernel, 256, 0));
            kernel<<<ctx.sm_count * std::max(1, blocks_per_sm), 256, 0, stream>>>(parts, t64);
        };
        if (unroll <= 2) {
            launch(random_count_parts_kernel<2>);
        } else if (unroll >= 8) {
            launch(random_count_parts_kernel<8>);
        } else {
            launch(random_count_parts_kernel<4>);
        }
    } else if (m.wide) {
        random_insert128_kernel<<<ctx.sm_count * 8, 256, 0, stream>>>(sc.def, t128);
    } else {
        // barcodes that were not in their home sector yet: inserted (or found further along) by the follow-up kernel
        random_insert_kernel<<<ctx.sm_count * 8, 256, 0, stream>>>(sc.def, t64);
    }
    SCG_CUDA_CHECK(cudaGetLastError());
    ctx.launches += 2;
    ctx.timing.launches += 2;
    if (!m.params.use_first) {
        // best mode: reads with several verified windows take the full scan (the minimum must be attained once)
        launch_random_generic(ctx, reads, m, tab, odd, odd_out, odd_count, out_index, ReadList{ slow.list, slow.count }, ctx.sm_count * 2, stream);
    }
    ctx.kernel_note = nparts ? "specialised (NVRTC) spec_random_kernel, filter+verify, barcodes listed by table part (" + std::to_string(nparts) + " parts), " +
                                   std::to_string(specialised_blocks_per_sm(k)) + " blocks/SM; + random_count_parts_kernel (16-byte-slot count table filled part by part in L2)"
                  : m.wide ? "specialised (NVRTC) spec_random_kernel, filter+verify + 128-bit-key count table (home sector requested a tile ahead), " +
                                   std::to_string(specialised_blocks_per_sm(k)) + " blocks/SM; + random_insert128_kernel (new and displaced barcodes)"
                             : "specialised (NVRTC) spec_random_kernel, filter+verify + 16-byte-slot count table (home sector requested a tile ahead), " +
                                   std::to_string(specialised_blocks_per_sm(k)) + " blocks/SM; + random_insert_kernel (new and displaced barcodes)";
    if (!m.params.use_first) ctx.kernel_note += " + random_kernel on the multi-window reads";
}

} // namespace scg

// ---------------------------------------------------------------------------------------
// resident plans (include/scg.h)
// ---------------------------------------------------------------------------------------
using namespace scg;

namespace {
cudaStream_t plan_stream(Context& c, void* cuda_stream) {
    return cuda_stream == SCG_STREAM_OWN ? c.stream : static_cast<cudaStream_t>(cuda_stream);
}
} // namespace

extern "C" {

// Compiles the run-time specialised kernel of a handler (NVRTC) for a template and read length; no device needed for the
// compile step.  kind: 1 dual paired-end (both templates), 2 combinatorial single-end, 3 random barcodes.
// Returns 0 = compiled and loaded, 2 = compiled but no device to load it on, 1 = failed; `message` has the details.
int scg_jit_selftest_handler(int kind, const char* constant_a, int strand_a, int mismatches_a, const char* constant_b, int strand_b,
                             int mismatches_b, int read_len, int use_first, char* message, size_t capacity) {
    std::string msg;
    int status = 1;
    try {
        ReadsDev fake;
        std::memset(&fake, 0, sizeof fake);
        fake.uniform_len = read_len;
        fake.W = std::max(1, (read_len + 31) / 32);
        fake.n = 1;
        TemplateSpec ta(constant_a, strand_a);
        const ScanSpec sa = ta.scan_spec(mismatches_a);
        std::string why;
        if (!template_fits(ta, sa, fake, &why)) throw Error(why);
        JitProgram prog;
        if (kind == 1) {
            TemplateSpec tb(constant_b, strand_b);
            const ScanSpec sb = tb.scan_spec(mismatches_b);
            if (!template_fits(tb, sb, fake, &why)) throw Error(why);
            prog = dual_program(ta, sa, mismatches_a, fake, tb, sb, mismatches_b, fake, use_first, 1, read_len % 2 ? 64 : 0);
        } else if (kind == 2) {
            if (ta.fwd_regions.size() != 2) throw Error("expected 2 variable regions in the constant template");
            prog = combo_program(ta, sa, mismatches_a, fake, use_first, 1, read_len % 2 ? 64 : 0);
        } else if (kind == 3 || kind == 4) {   // 4 = the variant that lists the barcodes by table part
            if (ta.fwd_regions.empty()) throw Error("expected at least one variable region in the constant template");
            prog = random_program(ta, sa, mismatches_a, fake, use_first, 1, kind == 4 ? 1 : 0);
        } else {
            throw Error("unknown handler kind");
        }
        const JitModule* mod = jit_module(prog, 0, &why);
        if (mod) {
            msg = "ok: " + jit_status();
            status = 0;
        } else {
            msg = why + " [" + jit_status() + "]";
            status = why.rfind("cudaLibraryLoadData", 0) == 0 ? 2 : 1;
        }
    } catch (const std::exception& e) {
        msg = e.what();
    }
    if (message && capacity) {
        std::snprintf(message, capacity, "%s", msg.c_str());   // (strncpy would zero-fill the whole buffer)
    }
    return status;
}

int scg_dual_plan_create(scg_ctx* ctx, const char* constant1, int reverse1, int mismatches1, const char* const* pool1, int npool1,
                         const char* constant2, int reverse2, int mismatches2, const char* const* pool2, int npool2, int randomized,
                         int use_first, scg_plan** out) {
    return guarded(ctx, [&] {
        Context& c = ctx->impl;
        Pool p1(pool1, npool1), p2(pool2, npool2);
        std::unique_ptr<scg_plan> plan(new scg_plan);
        plan->owner = ctx;
        plan->kind = scg_plan::DUAL;
        plan->npool = npool1;
        plan->dual = std::make_shared<DualPEMatcher>();
        plan->dual->prepare(constant1, reverse1 != 0, mismatches1, p1, constant2, reverse2 != 0, mismatches2, p2, randomized != 0, use_first != 0);
        c.ensure_ready();
        plan->dual->upload(c);
        *out = plan.release();
    });
}

int scg_dual_plan_run(scg_plan* plan, const scg_reads* reads1, const scg_reads* reads2, int32_t* d_counts, int32_t* d_index, void* cuda_stream) {
    if (!plan || !reads1 || !reads2) return 1;
    return guarded(plan->owner, [&] {
        Context& c = plan->owner->impl;
        if (plan->kind != scg_plan::DUAL) throw Error("not a dual-barcode plan");
        if (reads1->n != reads2->n || reads1->batches.size() != reads2->batches.size()) {
            throw Error("different number of reads in paired FASTQ files");   // process_data.hpp:284-285
        }
        SCG_CUDA_CHECK(cudaSetDevice(c.device));
        cudaStream_t st = plan_stream(c, cuda_stream);
        long long at = 0;
        for (size_t k = 0; k < reads1->batches.size(); ++k) {
            const ReadsDev& a = reads1->batches[k].view;
            const ReadsDev& b = reads2->batches[k].view;
            if (a.n != b.n) throw Error("the two mates' resident batches differ in size");
            launch_dual_pe(c, a, b, *plan->dual, d_counts, d_index ? d_index + at : nullptr, st);
            at += a.n;
        }
        plan->kernel_note = c.kernel_note;
    });
}

int scg_combo_plan_create(scg_ctx* ctx, const char* constant, int strand, const char* const* pool1, int npool1, const char* const* pool2,
                          int npool2, int mismatches, int use_first, scg_plan** out) {
    return guarded(ctx, [&] {
        Context& c = ctx->impl;
        Pool p1(pool1, npool1), p2(pool2, npool2);
        std::unique_ptr<scg_plan> plan(new scg_plan);
        plan->owner = ctx;
        plan->kind = scg_plan::COMBO;
        plan->combo = std::make_shared<ComboMatcher>();
        plan->combo->prepare(constant, strand, p1, p2, mismatches, use_first != 0, Duplicates::ERROR);
        c.ensure_ready();
        plan->combo->upload(c);
        plan->tally.init(c, npool1, npool2);
        SCG_CUDA_CHECK(cudaStreamSynchronize(c.stream));
        *out = plan.release();
    });
}

int scg_combo_plan_run(scg_plan* plan, const scg_reads* reads, int32_t* d_pairs, void* cuda_stream) {
    if (!plan || !reads) return 1;
    return guarded(plan->owner, [&] {
        Context& c = plan->owner->impl;
        if (plan->kind != scg_plan::COMBO) throw Error("not a combinatorial-barcode plan");
        SCG_CUDA_CHECK(cudaSetDevice(c.device));
        cudaStream_t st = plan_stream(c, cuda_stream);
        long long at = 0;
        for (const auto& b : reads->batches) {
            launch_combo(c, b.view, *plan->combo, plan->tally.sink(c, b.view.n), nullptr, d_pairs ? d_pairs + 2 * at : nullptr, st);
            at += b.view.n;
        }
        plan->kernel_note = c.kernel_note;
    });
}

int scg_random_plan_create(scg_ctx* ctx, const char* constant, int strand, int mismatches, int use_first, long long expected_distinct,
                           scg_plan** out) {
    return guarded(ctx, [&] {
        Context& c = ctx->impl;
        std::unique_ptr<scg_plan> plan(new scg_plan);
        plan->owner = ctx;
        plan->kind = scg_plan::RANDOM;
        plan->random = std::make_shared<RandomMatcher>();
        plan->random->prepare(constant, strand, mismatches, use_first != 0);
        c.ensure_ready();
        // sized once for the distinct barcodes the caller expects (load factor <= 1/2; a table twice the size keeps more barcodes
        // inside their home sector but measured slower: its footprint costs more than the displaced keys do); 0 = grow as the
        // reference's map does
        plan->table.init(c, plan->random->wide, expected_distinct > 0 ? (size_t)(2 * expected_distinct) : (size_t)1 << 20, plan->random->long_words);
        plan->table.fixed = expected_distinct > 0;
        SCG_CUDA_CHECK(cudaStreamSynchronize(c.stream));
        *out = plan.release();
    });
}

int scg_random_plan_run(scg_plan* plan, const scg_reads* reads, int32_t* d_index, void* cuda_stream) {
    if (!plan || !reads) return 1;
    return guarded(plan->owner, [&] {
        Context& c = plan->owner->impl;
        if (plan->kind != scg_plan::RANDOM) throw Error("not a random-barcode plan");
        SCG_CUDA_CHECK(cudaSetDevice(c.device));
        cudaStream_t st = plan_stream(c, cuda_stream);
        long long at = 0;
        for (const auto& b : reads->batches) {
            plan->table.ensure(c, b.view.n);
            // resident reads are packed bases: no read needs its raw text
            launch_random(c, b.view, *plan->random, plan->table, nullptr, nullptr, nullptr, d_index ? d_index + at : nullptr, st);
            at += b.view.n;
        }
        plan->kernel_note = c.kernel_note;
    });
}

int scg_plan_reset(scg_plan* plan, void* cuda_stream) {
    if (!plan) return 1;
    return guarded(plan->owner, [&] {
        Context& c = plan->owner->impl;
        SCG_CUDA_CHECK(cudaSetDevice(c.device));
        cudaStream_t st = plan_stream(c, cuda_stream);
        if (plan->kind == scg_plan::COMBO) plan->tally.reset(c, st);
        if (plan->kind == scg_plan::RANDOM) plan->table.reset(c, st);
    });
}

int scg_plan_harvest(scg_plan* plan, scg_result** table) {
    if (!plan || !table) return 1;
    return guarded(plan->owner, [&] {
        Context& c = plan->owner->impl;
        SCG_CUDA_CHECK(cudaSetDevice(c.device));
        SCG_CUDA_CHECK(cudaDeviceSynchronize());   // the runs may have been enqueued on the caller's stream
        std::unique_ptr<scg_result> r(new scg_result);
        if (plan->kind == scg_plan::COMBO) {
            plan->tally.harvest(c, *r);
        } else if (plan->kind == scg_plan::RANDOM) {
            SortedTable sorted;
            plan->table.sorted(c, plan->random->key_len, sorted);
            r->width = plan->random->key_len;
            render_barcodes(c, sorted, r->d_strings, r->d_freq);
            SCG_CUDA_CHECK(cudaStreamSynchronize(c.stream));
            r->on_device = true;
            r->device = c.device;
            r->d_rows = sorted.rows;
        } else {
            throw Error("only combinatorial and random-barcode plans hold a table");
        }
        *table = r.release();
    });
}

// ---- sorted tables resident on the device: what the GPUs exchange when a sparse result is merged across them ----

int scg_plan_sorted_table(scg_plan* plan, scg_table** out) {
    if (!plan || !out) return 1;
    return guarded(plan->owner, [&] {
        Context& c = plan->owner->impl;
        SCG_CUDA_CHECK(cudaSetDevice(c.device));
        SCG_CUDA_CHECK(cudaDeviceSynchronize());   // the runs may have been enqueued on the caller's stream
        std::unique_ptr<scg_table> t(new scg_table);
        t->owner = plan->owner;
        if (plan->kind == scg_plan::COMBO) {
            plan->tally.sorted(c, t->table);
        } else if (plan->kind == scg_plan::RANDOM) {
            // what this interface hands out it must be able to take back (scg_table_from_device: key lengths 0..42)
            if (plan->random->key_len > 42) throw Error("sorted tables hold random barcodes of at most 42 bases");
            plan->table.sorted(c, plan->random->key_len, t->table);
        } else {
            throw Error("only combinatorial and random-barcode plans hold a table");
        }
        *out = t.release();
    });
}

int scg_plan_dense_tally(scg_plan* plan, void** d_matrix, long long* cells) {
    if (!plan || !d_matrix || !cells) return 1;
    return guarded(plan->owner, [&] {
        *d_matrix = nullptr;
        *cells = 0;
        if (plan->kind == scg_plan::COMBO && plan->tally.dense) {
            *d_matrix = plan->tally.matrix.ptr;
            *cells = (long long)plan->tally.n1 * plan->tally.n2;
        }
    });
}

long long scg_table_rows(const scg_table* t) { return t ? (long long)t->table.rows : 0; }
int scg_table_key_len(const scg_table* t) { return t ? t->table.key_len : 0; }
int scg_table_key_words(const scg_table* t) { return t ? t->table.words() : 0; }
void* scg_table_keys(const scg_table* t) { return t ? t->table.keys.ptr : nullptr; }
void* scg_table_counts(const scg_table* t) { return t ? t->table.counts.ptr : nullptr; }
void scg_table_free(scg_table* t) { delete t; }

int scg_table_from_device(scg_ctx* ctx, const void* d_keys, const void* d_counts, long long rows, int key_len, scg_table** out) {
    return guarded(ctx, [&] {
        Context& c = ctx->impl;
        c.ensure_ready();
        if (rows < 0) throw Error("negative number of rows");
        if (key_len < 0 || key_len > 42) throw Error("key length " + std::to_string(key_len) + " is outside 0..42");
        std::unique_ptr<scg_table> t(new scg_table);
        t->owner = ctx;
        t->table.rows = (size_t)rows;
        t->table.key_len = key_len;
        const size_t key_bytes = (size_t)rows * 8 * (size_t)t->table.words();
        t->table.keys.alloc(std::max<size_t>(key_bytes, 8), false);
        t->table.counts.alloc(std::max<size_t>((size_t)rows, 1) * sizeof(uint32_t), false);
        if (rows) {
            SCG_CUDA_CHECK(cudaMemcpyAsync(t->table.keys.ptr, d_keys, key_bytes, cudaMemcpyDeviceToDevice, c.stream));
            SCG_CUDA_CHECK(cudaMemcpyAsync(t->table.counts.ptr, d_counts, (size_t)rows * sizeof(uint32_t), cudaMemcpyDeviceToDevice, c.stream));
        }
        // foreign rows: the merge's binary searches and the renderer rely on what a table promises (include/scg.h);
        // synchronises the copies; a refused table is freed with t
        validate_sorted_table(c, t->table);
        *out = t.release();
    });
}

int scg_table_merge(scg_ctx* ctx, const scg_table* a, const scg_table* b, scg_table** out) {
    return guarded(ctx, [&] {
        Context& c = ctx->impl;
        c.ensure_ready();
        if (!a || !b) throw Error("null table");
        if (a->table.key_len != b->table.key_len) {
            throw Error("cannot merge tables of different key lengths (" + std::to_string(a->table.key_len) + " and " +
                        std::to_string(b->table.key_len) + ")");
        }
        std::unique_ptr<scg_table> t(new scg_table);
        t->owner = ctx;
        merge_sorted_tables(c, a->table, b->table, t->table);
        *out = t.release();
    });
}

int scg_table_render(scg_ctx* ctx, const scg_table* t, scg_result** out) {
    return guarded(ctx, [&] {
        Context& c = ctx->impl;
        c.ensure_ready();
        if (!t) throw Error("null table");
        std::unique_ptr<scg_result> r(new scg_result);
        if (t->table.key_len > 0) {
            r->width = t->table.key_len;
            render_barcodes(c, t->table, r->d_strings, r->d_freq);
        } else {
            r->width = 2;
            render_combinations(c, t->table, r->d_keys, r->d_freq);
        }
        SCG_CUDA_CHECK(cudaStreamSynchronize(c.stream));
        r->on_device = true;
        r->device = c.device;
        r->d_rows = t->table.rows;
        *out = r.release();
    });
}

} // extern "C"
