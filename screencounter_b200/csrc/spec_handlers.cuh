// Handler kernels with their TEMPLATES FOLDED IN AT COMPILE TIME (NVRTC, jit.cpp), for batches of uniform-length reads:
//
//   SPH_KIND 1   countDualBarcodes, paired-end      DualBarcodesPairedEnd::process        handlers/DualBarcodesPairedEnd.hpp:216-381
//   SPH_KIND 2   countComboBarcodes, single-end     CombinatorialBarcodesSingleEnd        handlers/CombinatorialBarcodesSingleEnd.hpp:149-258
//   SPH_KIND 3   countRandomBarcodes                RandomBarcodeSingleEnd::process       handlers/RandomBarcodeSingleEnd.hpp:93-181
//
// Shape shared by the three (the recipe of the single-barcode kernel, DESIGN.md 5.1b): one warp per tile of 32 reads
// (pairs), persistent warps; tiles arrive by 1-D TMA bulk copies into a per-warp ring in shared memory (both mates of a
// pair on ONE mbarrier); the constant flanks are scanned with the filter + verify of spec_scan.cuh; a read with exactly
// one verified window (per mate) is settled by the kernel itself:
//   dual    the two variable regions, concatenated, are probed in a 16-byte-slot cuckoo table of the library rows; the two
//           slots are requested after the scan and looked at ONE TILE LATER, so their latency hides behind the next scan;
//   combo   each region is probed in its pool's exact table;
//   random  the barcode's slot in the count table is requested and, one tile later, counted (or inserted).
// What the kernel cannot settle goes to global lists, so that the registers of the heavy searches do not cap THIS kernel's
// occupancy:
//   * exact probe missed with mismatch budget left, or an N inside a region: the keys are appended to the warp's own
//     region of a DeferredList and a follow-up kernel runs the mismatch-tolerant lookups (lookups only, no rescan);
//   * several verified windows: the read's index goes to a SlowList and the generic kernel of the handler
//     (handlers.cuh) runs the full per-read search on exactly those reads.
// Per-read outcomes are identical to the generic kernels'; tests/test_gpu_plans.py compares both with the reference.
//
// Macros (all required): SPH_KIND; SPH_MIN_BLOCKS, SPH_STAGES, SPH_GROUP (tiles per bulk copy), SPH_SAMPLES; SPH_USE_FIRST,
// SPH_HAS_INDEX; template A: SPH_A_T, SPH_A_FB, SPH_A_RB, SPH_A_FWD, SPH_A_REV, SPH_A_MM (scan budget), SPH_A_MAXMM (the
// caller's budget), SPH_A_ULEN, SPH_A_W, SPH_A_FSTART0/FLEN0/RSTART0/RLEN0 and, for two regions, ...1; kind 1 also template
// B the same way (SPH_B_*), read 2's template.
#pragma once

#include "count_table.cuh"
#include "spec_scan.cuh"

#ifndef SPH_PARTITIONED
#define SPH_PARTITIONED 0
#endif
#ifndef SPH_HIST
#define SPH_HIST 0   // > 0: the design's counters (pool rows / cells of the dense combination matrix) privatised per block in shared memory
#endif
#ifndef SPH_A_FSTART1
#define SPH_A_FSTART1 0
#define SPH_A_FLEN1 1
#define SPH_A_RSTART1 0
#define SPH_A_RLEN1 1
#endif

namespace scg {
namespace sph {

using namespace scg::sscan;

struct TrA {
    static constexpr int T = SPH_A_T;
    static constexpr char FB[] = SPH_A_FB;
    static constexpr char RB[] = SPH_A_RB;
    static constexpr bool FWD = SPH_A_FWD != 0, REV = SPH_A_REV != 0;
    static constexpr int MM = SPH_A_MM;
    static constexpr int ULEN = SPH_A_ULEN, W = SPH_A_W;
    static constexpr int SAMPLES = SPH_SAMPLES;
};
#if SPH_KIND == 1
struct TrB {
    static constexpr int T = SPH_B_T;
    static constexpr char FB[] = SPH_B_FB;
    static constexpr char RB[] = SPH_B_RB;
    static constexpr bool FWD = SPH_B_FWD != 0, REV = SPH_B_REV != 0;
    static constexpr int MM = SPH_B_MM;
    static constexpr int ULEN = SPH_B_ULEN, W = SPH_B_W;
    static constexpr int SAMPLES = SPH_SAMPLES;
};
#endif

constexpr int BLOCK = 128;
constexpr int WARPS = BLOCK / 32;
constexpr int STAGES = SPH_STAGES;
constexpr int GROUP = SPH_GROUP;

// flags of the word a lane carries from one tile to the next, beside sscan's SM_CAND / SM_REV
constexpr uint32_t PM_INRANGE = 1u << 26;       // the lane holds a real read
constexpr uint32_t PM_PROBED = 1u << 30;        // table slots were requested
constexpr uint32_t PM_MISS_DEFERS = 1u << 25;   // if the probe misses (or was not possible), the read is deferred
constexpr uint32_t PM_SLOW = 1u << 24;          // several verified windows: the full per-read search

__host__ __device__ constexpr uint32_t low_mask(int len) { return len >= 32 ? 0xFFFFFFFFu : ((1u << len) - 1u); }

// appends one entry per flagged lane to the warp's region of a deferred list; `cursor` is warp-uniform
template <int NWORDS>
__device__ __forceinline__ void defer_append(const DeferredList& def, uint32_t region_base, uint32_t& cursor, bool flag, int lane,
                                             const uint32_t (&entry)[NWORDS]) {
    const uint32_t dm = __ballot_sync(0xFFFFFFFFu, flag);
    if (dm) {
        if (flag) {
            const unsigned long long at = (unsigned long long)region_base + cursor + __popc(dm & ((1u << lane) - 1u));
#pragma unroll
            for (int k = 0; k < NWORDS; ++k) def.words[(unsigned long long)k * def.stride + at] = entry[k];
        }
        cursor += __popc(dm);
    }
}

// appends the flagged lanes' read indices to the slow list: one atomic per warp batch
__device__ __forceinline__ void slow_append(const SlowList& slow, bool flag, int lane, uint32_t index) {
    const uint32_t hard = __ballot_sync(0xFFFFFFFFu, flag);
    if (hard) {
        const int leader = __ffs(hard) - 1;
        uint32_t base = 0;
        if (lane == leader) base = atomicAdd(slow.count, (uint32_t)__popc(hard));
        base = __shfl_sync(0xFFFFFFFFu, base, leader);
        if (flag) slow.list[base + __popc(hard & ((1u << lane) - 1u))] = index;
    }
}

} // namespace sph
} // namespace scg

// =====================================================================================================================
// countDualBarcodes, paired-end
// =====================================================================================================================
#if SPH_KIND == 1
extern "C" __global__ void __launch_bounds__(128, SPH_MIN_BLOCKS)
    spec_dual_pe_kernel(const scg::ReadsDev reads1, const scg::ReadsDev reads2, const scg::DualTables tb, int32_t* __restrict__ counts,
                        int32_t* __restrict__ out_index, const scg::DeferredList def, const scg::SlowList slow) {
    using namespace scg;
    using namespace scg::sph;
    using DA = Dims<TrA>;
    using DB = Dims<TrB>;
    static_assert(TrA::FWD != TrA::REV && TrB::FWD != TrB::REV, "each read of a paired design is searched on exactly one strand");
    constexpr int START_A = TrA::FWD ? SPH_A_FSTART0 : SPH_A_RSTART0, LEN_A = TrA::FWD ? SPH_A_FLEN0 : SPH_A_RLEN0;
    constexpr int START_B = TrB::FWD ? SPH_B_FSTART0 : SPH_B_RSTART0, LEN_B = TrB::FWD ? SPH_B_FLEN0 : SPH_B_RLEN0;
    static_assert(LEN_A >= 1 && LEN_A <= 32 && LEN_B >= 1 && LEN_B <= 32 && LEN_A + LEN_B <= DUAL_MAX_KEYLEN, "variable regions too long");
    constexpr uint32_t BYTES_A = GROUP * DA::TILE_BYTES, BYTES_B = GROUP * DB::TILE_BYTES;
    __shared__ __align__(128) uint32_t stage_a[WARPS][STAGES][GROUP * DA::TILE_WORDS];
    __shared__ __align__(128) uint32_t stage_b[WARPS][STAGES][GROUP * DB::TILE_WORDS];
    __shared__ __align__(8) unsigned long long bar_all[WARPS][STAGES];
#if SPH_HIST
    __shared__ int32_t hist[SPH_HIST];
    for (int k = threadIdx.x; k < SPH_HIST; k += BLOCK) hist[k] = 0;
    __syncthreads();
#endif

    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int warp = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int nwarps = (int)((gridDim.x * blockDim.x) >> 5);
    const uint32_t n = (uint32_t)reads1.n;
    const int ntiles = (int)((n + TILE - 1) / TILE);
    const int ngroups = (ntiles + GROUP - 1) / GROUP;

    const uint32_t base_a = smem_addr(&stage_a[wib][0][0]), base_b = smem_addr(&stage_b[wib][0][0]);
    const uint32_t bar_base = smem_addr(&bar_all[wib][0]);
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) mbar_init(bar_base + 8u * s, 1);
        fence_barrier_init();
    }
    __syncwarp();
    const uint64_t policy = evict_first_policy();
    auto fetch = [&](int g, uint32_t stage) {
        const uint32_t tiles = (uint32_t)min(GROUP, ntiles - GROUP * g);
        const uint32_t bar = bar_base + 8u * stage;
        tma_fetch(bar, base_a + stage * BYTES_A, reinterpret_cast<const char*>(reads1.data) + (size_t)g * BYTES_A, tiles * DA::TILE_BYTES,
                  tiles * (DA::TILE_BYTES + DB::TILE_BYTES), policy);
        tma_fetch_more(bar, base_b + stage * BYTES_B, reinterpret_cast<const char*>(reads2.data) + (size_t)g * BYTES_B, tiles * DB::TILE_BYTES,
                       policy);
    };
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
        if (warp + s * nwarps < ngroups) fetch(warp + s * nwarps, (uint32_t)s);
    }

    const uint32_t region_base = (uint32_t)warp * def.per_warp;
    uint32_t cursor = 0;   // warp-uniform: entries in this warp's region

    // carried from one tile to the next: the two slots of the pair's key, the key, the flags
    uint4 pa = make_uint4(0, 0, 0, 0), pb = make_uint4(0, 0, 0, 0);
    uint32_t pmeta = 0, px = 0, py = 0, pz = 0, pn_lo = 0, pn_hi_caps = 0, pi = 0;

    uint32_t stage = 0, parity = 0;
    int group = warp, tile_in_group = 0, tiles_here = 0;
    bool have = group < ngroups;
    if (have) {
        mbar_wait(bar_base, 0);
        tiles_here = min(GROUP, ntiles - GROUP * group);
    }
    for (;;) {
        uint32_t meta = 0, x = 0, y = 0, z = 0, n_lo = 0, n_hi_caps = 0, i = 0;
        if (have) {
            i = (uint32_t)(group * GROUP + tile_in_group) * TILE + lane;
            const bool inrange = i < n;
            // ---- read 1: template A ----
            uint32_t metaA = 0, ah = 0, al = 0, an = 0;
            int ncandA = 0;
            {
                Words<TrA::W> R;
                load_words<TrA::W>(stage_a[wib][stage] + tile_in_group * DA::TILE_WORDS + lane, R);
                Planes<TrA::W> P;
                make_planes<TrA::W>(R, P);
                scan_blocks<TrA, 0>(R, P, inrange, ncandA, metaA, [&](const uint32_t(&wh)[DA::TW + 1], const uint32_t(&wl)[DA::TW + 1],
                                                                     const uint32_t(&wn)[DA::TW + 1], bool) {
                    ah = window_bits<START_A, LEN_A>(wh);
                    al = window_bits<START_A, LEN_A>(wl);
                    an = window_bits<START_A, LEN_A>(wn);
                });
            }
            // ---- read 2: template B ----
            uint32_t metaB = 0, bh = 0, bl = 0, bn = 0;
            int ncandB = 0;
            {
                Words<TrB::W> R;
                load_words<TrB::W>(stage_b[wib][stage] + tile_in_group * DB::TILE_WORDS + lane, R);
                Planes<TrB::W> P;
                make_planes<TrB::W>(R, P);
                scan_blocks<TrB, 0>(R, P, inrange, ncandB, metaB, [&](const uint32_t(&wh)[DB::TW + 1], const uint32_t(&wl)[DB::TW + 1],
                                                                     const uint32_t(&wn)[DB::TW + 1], bool) {
                    bh = window_bits<START_B, LEN_B>(wh);
                    bl = window_bits<START_B, LEN_B>(wl);
                    bn = window_bits<START_B, LEN_B>(wn);
                });
            }
            // the buffers go back to the TMA once every lane has consumed the group's last tile
            if (++tile_in_group == tiles_here) {
                __syncwarp();
                const int ahead = group + STAGES * nwarps;
                if (ahead < ngroups) fetch(ahead, stage);
            }
            // ---- the pair's key: region of read 1, then region of read 2 (DualBarcodesPairedEnd.hpp:139-164) ----
            const bool both = (metaA & SM_CAND) && (metaB & SM_CAND);
            const bool many = both && (ncandA > 1 || ncandB > 1);
            const int c1 = (int)((metaA >> 16) & 0xFFu), c2 = (int)((metaB >> 16) & 0xFFu);
            const int cap1 = SPH_A_MAXMM - c1, cap2 = SPH_B_MAXMM - c2;
            constexpr int HI_SHIFT = LEN_A >= 32 ? 0 : 32 - LEN_A;   // bits of read 2's region that do not fit the low word
            const uint32_t hl = LEN_A >= 32 ? ah : (ah | (bh << (LEN_A & 31)));
            const uint32_t ll = LEN_A >= 32 ? al : (al | (bl << (LEN_A & 31)));
            const uint32_t nl = LEN_A >= 32 ? an : (an | (bn << (LEN_A & 31)));
            const uint32_t hh = LEN_A >= 32 ? bh : (LEN_A + LEN_B > 32 ? bh >> HI_SHIFT : 0u);
            const uint32_t lh = LEN_A >= 32 ? bl : (LEN_A + LEN_B > 32 ? bl >> HI_SHIFT : 0u);
            const uint32_t nh = LEN_A >= 32 ? bn : (LEN_A + LEN_B > 32 ? bn >> HI_SHIFT : 0u);
            x = hl;
            y = ll;
            z = hh | (lh << 16);
            n_lo = nl;
            n_hi_caps = nh | ((uint32_t)(cap1 & 0xFF) << 16) | ((uint32_t)(cap2 & 0xFF) << 24);
            const bool budget = cap1 >= 1 || cap2 >= 1;
            meta = (inrange ? PM_INRANGE : 0u) + (both ? SM_CAND : 0u) + (many ? PM_SLOW : 0u) +
                   ((both && !many && budget) ? PM_MISS_DEFERS : 0u);
        }

        // ---- settle the PREVIOUS tile: its slots were requested one scan ago ----
        {
            const uint32_t m = pmeta;
            int index = -1;
            if (m & PM_PROBED) {
                const int ra = (pa.x == px && pa.y == py && pa.z == pz) ? (int)pa.w : -1;
                const int rb = (pb.x == px && pb.y == py && pb.z == pz) ? (int)pb.w : -1;
                index = max(ra, rb);
            }
            const bool slowp = (m & PM_SLOW) != 0;
            const bool defer = (m & PM_MISS_DEFERS) && index < 0;
            if ((m & PM_INRANGE) && !defer && !slowp) {
#if SPH_HIST
                if (index >= 0) atomicAdd(&hist[index], 1);
#else
                if (index >= 0) atomicAdd(counts + index, 1);
#endif
                if (SPH_HAS_INDEX) __stcs(out_index + pi, index);
            }
            const uint32_t entry[DUAL_DEFER_WORDS] = { pi, px, py, pz, pn_lo, pn_hi_caps };
            defer_append<DUAL_DEFER_WORDS>(def, region_base, cursor, defer, lane, entry);
            slow_append(slow, slowp, lane, pi);
        }

        // ---- this tile: request the two slots of the pair's key ----
        pmeta = meta;
        pi = i;
        px = x;
        py = y;
        pz = z;
        pn_lo = n_lo;
        pn_hi_caps = n_hi_caps;
        if ((meta & SM_CAND) && !(meta & PM_SLOW) && n_lo == 0 && (n_hi_caps & 0xFFFFu) == 0) {
            const uint32_t h = dual_hash(x, y, z);
            const uint32_t second = (1u << (32 - tb.shift)) + (dual_hash2(h) >> tb.shift);
            pa = __ldcg(tb.exact + (h >> tb.shift));
            pb = __ldcg(tb.exact + second);
            pmeta = meta + PM_PROBED;
        }

        if (!have) break;
        if (tile_in_group == tiles_here) {
            group += nwarps;
            tile_in_group = 0;
            if (++stage == STAGES) {
                stage = 0;
                parity ^= 1u;
            }
            have = group < ngroups;
            if (have) {
                mbar_wait(bar_base + 8u * stage, parity);
                tiles_here = min(GROUP, ntiles - GROUP * group);
            }
        }
    }
    if (lane == 0) def.warp_counts[warp] = cursor;
#if SPH_HIST
    // flush the block's private counters: one global atomic per row that was hit
    __syncthreads();
    for (int k = threadIdx.x; k < SPH_HIST; k += BLOCK) {
        const int32_t v = hist[k];
        if (v) atomicAdd(counts + k, v);
    }
#endif
}
#endif  // SPH_KIND == 1

// =====================================================================================================================
// countComboBarcodes, single-end, two variable regions
// =====================================================================================================================
#if SPH_KIND == 2
extern "C" __global__ void __launch_bounds__(128, SPH_MIN_BLOCKS)
    spec_combo_kernel(const scg::ReadsDev reads, const scg::ComboTables tb, const scg::ComboSink sink, int32_t* __restrict__ out_pairs,
                      const scg::DeferredList def, const scg::SlowList slow) {
    using namespace scg;
    using namespace scg::sph;
    using DA = Dims<TrA>;
    static_assert(SPH_A_FLEN0 <= 32 && SPH_A_FLEN1 <= 32 && SPH_A_RLEN0 <= 32 && SPH_A_RLEN1 <= 32, "variable regions too long");
    constexpr uint32_t BYTES_A = GROUP * DA::TILE_BYTES;
    __shared__ __align__(128) uint32_t stage_a[WARPS][STAGES][GROUP * DA::TILE_WORDS];
    __shared__ __align__(8) unsigned long long bar_all[WARPS][STAGES];
#if SPH_HIST
    __shared__ int32_t hist[SPH_HIST];   // the dense n1 x n2 matrix of a small design
    for (int k = threadIdx.x; k < SPH_HIST; k += BLOCK) hist[k] = 0;
    __syncthreads();
#endif

    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int warp = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int nwarps = (int)((gridDim.x * blockDim.x) >> 5);
    const uint32_t n = (uint32_t)reads.n;
    const int ntiles = (int)((n + TILE - 1) / TILE);
    const int ngroups = (ntiles + GROUP - 1) / GROUP;

    const uint32_t base_a = smem_addr(&stage_a[wib][0][0]);
    const uint32_t bar_base = smem_addr(&bar_all[wib][0]);
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) mbar_init(bar_base + 8u * s, 1);
        fence_barrier_init();
    }
    __syncwarp();
    const uint64_t policy = evict_first_policy();
    auto fetch = [&](int g, uint32_t stage) {
        const uint32_t bytes = (uint32_t)min(GROUP, ntiles - GROUP * g) * DA::TILE_BYTES;
        tma_fetch(bar_base + 8u * stage, base_a + stage * BYTES_A, reinterpret_cast<const char*>(reads.data) + (size_t)g * BYTES_A, bytes, bytes,
                  policy);
    };
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
        if (warp + s * nwarps < ngroups) fetch(warp + s * nwarps, (uint32_t)s);
    }
    const uint32_t region_base = (uint32_t)warp * def.per_warp;
    uint32_t cursor = 0;

    // carried from one tile to the next: the four slots requested for the two regions, the regions, the flags
    constexpr uint32_t PM_PROBED1 = 1u << 29;   // region 1's slots were requested (PM_PROBED: region 0's)
    uint4 pa0 = make_uint4(0, 0, 0, 0), pb0 = pa0, pa1 = pa0, pb1 = pa0;
    uint32_t pmeta = 0, pi = 0, pk0h = 0, pk0l = 0, pk0n = 0, pk1h = 0, pk1l = 0, pk1n = 0;

    uint32_t stage = 0, parity = 0;
    int group = warp, tile_in_group = 0, tiles_here = 0;
    bool have = group < ngroups;
    if (have) {
        mbar_wait(bar_base, 0);
        tiles_here = min(GROUP, ntiles - GROUP * group);
    }
    for (;;) {
        uint32_t meta = 0, i = 0, k0h = 0, k0l = 0, k0n = 0, k1h = 0, k1l = 0, k1n = 0;   // regions in READ order
        if (have) {
            i = (uint32_t)(group * GROUP + tile_in_group) * TILE + lane;
            const bool inrange = i < n;
            int ncand = 0;
            {
                Words<TrA::W> R;
                load_words<TrA::W>(stage_a[wib][stage] + tile_in_group * DA::TILE_WORDS + lane, R);
                Planes<TrA::W> P;
                make_planes<TrA::W>(R, P);
                scan_blocks<TrA, 0>(R, P, inrange, ncand, meta, [&](const uint32_t(&wh)[DA::TW + 1], const uint32_t(&wl)[DA::TW + 1],
                                                                   const uint32_t(&wn)[DA::TW + 1], bool rev) {
                    if (TrA::FWD && (!TrA::REV || !rev)) {
                        k0h = window_bits<SPH_A_FSTART0, SPH_A_FLEN0>(wh);
                        k0l = window_bits<SPH_A_FSTART0, SPH_A_FLEN0>(wl);
                        k0n = window_bits<SPH_A_FSTART0, SPH_A_FLEN0>(wn);
                        k1h = window_bits<SPH_A_FSTART1, SPH_A_FLEN1>(wh);
                        k1l = window_bits<SPH_A_FSTART1, SPH_A_FLEN1>(wl);
                        k1n = window_bits<SPH_A_FSTART1, SPH_A_FLEN1>(wn);
                    }
                    if (TrA::REV && (!TrA::FWD || rev)) {
                        k0h = window_bits<SPH_A_RSTART0, SPH_A_RLEN0>(wh);
                        k0l = window_bits<SPH_A_RSTART0, SPH_A_RLEN0>(wl);
                        k0n = window_bits<SPH_A_RSTART0, SPH_A_RLEN0>(wn);
                        k1h = window_bits<SPH_A_RSTART1, SPH_A_RLEN1>(wh);
                        k1l = window_bits<SPH_A_RSTART1, SPH_A_RLEN1>(wl);
                        k1n = window_bits<SPH_A_RSTART1, SPH_A_RLEN1>(wn);
                    }
                });
            }
            // the buffers go back to the TMA once every lane has consumed the group's last tile
            if (++tile_in_group == tiles_here) {
                __syncwarp();
                const int ahead = group + STAGES * nwarps;
                if (ahead < ngroups) fetch(ahead, stage);
            }
            meta = (meta & (SM_CAND | SM_REV | 0x00FF0000u)) + (inrange ? PM_INRANGE : 0u) + (((meta & SM_CAND) && ncand > 1) ? PM_SLOW : 0u);
        }

        // ---- settle the PREVIOUS tile: its slots were requested one scan ago (find_match, :149-186) ----
        {
            const uint32_t m = pmeta;
            const bool cand = (m & SM_CAND) != 0, many = (m & PM_SLOW) != 0, rev = (m & SM_REV) != 0;
            const int c = (int)((m >> 16) & 0xFFu);
            int id_a = -1, id_b = -1;   // pool indices found for region 0 / region 1 (read order)
            if (m & PM_PROBED) {
                const int ra = (pa0.x == pk0h && pa0.y == pk0l) ? (int)pa0.z : -1;
                const int rb = (pb0.x == pk0h && pb0.y == pk0l) ? (int)pb0.z : -1;
                id_a = max(ra, rb);
            }
            if (m & PM_PROBED1) {
                const int ra = (pa1.x == pk1h && pa1.y == pk1l) ? (int)pa1.z : -1;
                const int rb = (pb1.x == pk1h && pb1.y == pk1l) ? (int)pb1.z : -1;
                id_b = max(ra, rb);
            }
            const bool found = id_a >= 0 && id_b >= 0;
            const bool defer = cand && !many && !found && (SPH_A_MAXMM - c >= 1);
            const bool slowp = cand && many;
            // reverse strand: region r of the read is pool 1 - r (:111-116)
            const int id0 = rev ? id_b : id_a, id1 = rev ? id_a : id_b;
            if ((m & PM_INRANGE) && !defer && !slowp) {
#if SPH_HIST
                if (found) atomicAdd(&hist[id0 * sink.n2 + id1], 1);
#else
                if (found) combo_count(sink, id0, id1);
#endif
                if (SPH_HAS_INDEX) {
                    __stcs(reinterpret_cast<int2*>(out_pairs) + pi, found ? make_int2(id0, id1) : make_int2(-1, -1));
                }
            }
            const uint32_t entry[COMBO_DEFER_WORDS] = { pi, (rev ? 0x100u : 0u) | (uint32_t)c, pk0h, pk0l, pk0n, pk1h, pk1l, pk1n };
            defer_append<COMBO_DEFER_WORDS>(def, region_base, cursor, defer, lane, entry);
            slow_append(slow, slowp, lane, pi);
        }

        // ---- this tile: request the two slots of each region in its pool's exact table ----
        pmeta = meta;
        pi = i;
        pk0h = k0h;
        pk0l = k0l;
        pk0n = k0n;
        pk1h = k1h;
        pk1l = k1l;
        pk1n = k1n;
        if ((meta & SM_CAND) && !(meta & PM_SLOW)) {
            const int l0 = (meta & SM_REV) ? 2 : 0;
            const uint4* __restrict__ s0 = tb.slots[l0];
            const uint4* __restrict__ s1 = tb.slots[l0 + 1];
            const uint32_t m0 = tb.mask[l0], m1 = tb.mask[l0 + 1];
            if (k0n == 0) {
                const uint32_t acc0 = hash_key(&k0h, &k0l, 1, 0);
                pa0 = __ldg(s0 + (acc0 & m0));
                pb0 = __ldg(s0 + (size_t)(m0 + 1) + (hash_second(acc0) & m0));
                pmeta += PM_PROBED;
            }
            if (k1n == 0) {
                const uint32_t acc1 = hash_key(&k1h, &k1l, 1, 0);
                pa1 = __ldg(s1 + (acc1 & m1));
                pb1 = __ldg(s1 + (size_t)(m1 + 1) + (hash_second(acc1) & m1));
                pmeta += PM_PROBED1;
            }
        }

        if (!have) break;
        if (tile_in_group == tiles_here) {
            group += nwarps;
            tile_in_group = 0;
            if (++stage == STAGES) {
                stage = 0;
                parity ^= 1u;
            }
            have = group < ngroups;
            if (have) {
                mbar_wait(bar_base + 8u * stage, parity);
                tiles_here = min(GROUP, ntiles - GROUP * group);
            }
        }
    }
    if (lane == 0) def.warp_counts[warp] = cursor;
#if SPH_HIST
    __syncthreads();
    for (int k = threadIdx.x; k < SPH_HIST; k += BLOCK) {
        const int32_t v = hist[k];
        if (v) atomicAdd(sink.dense + k, v);
    }
#endif
}
#endif  // SPH_KIND == 2

// =====================================================================================================================
// countRandomBarcodes
// =====================================================================================================================
#if SPH_KIND == 3
// barcodes of 22 to 42 bases: 128-bit keys (random_key128) in the wide count table, whose keys and counts are separate arrays
#define SPH_WIDE (SPH_A_FLEN0 > 21)
namespace scg {
namespace sph {
// bits [START, START + LEN) of a window given as words, LEN <= 64
template <int START, int LEN, int NW>
__device__ __forceinline__ unsigned long long window_bits64(const uint32_t (&w)[NW]) {
    if constexpr (LEN <= 32) {
        return window_bits<START, LEN>(w);
    } else {
        return (unsigned long long)window_bits<START, 32>(w) | ((unsigned long long)window_bits<START + 32, LEN - 32>(w) << 32);
    }
}
} // namespace sph
} // namespace scg

extern "C" __global__ void __launch_bounds__(128, SPH_MIN_BLOCKS)
#if SPH_WIDE
    spec_random_kernel(const scg::ReadsDev reads, const scg::CountTable128 table, const uint8_t* __restrict__ odd, long long read_offset,
#else
    spec_random_kernel(const scg::ReadsDev reads, const scg::CountTable64 table, const uint8_t* __restrict__ odd, long long read_offset,
#endif
                       scg::OddOutcome* __restrict__ odd_out, unsigned long long* __restrict__ odd_count, int32_t* __restrict__ out_index,
                       const scg::DeferredList def, const scg::SlowList slow, const scg::PartitionedKeys parts) {
    using namespace scg;
    using namespace scg::sph;
    using DA = Dims<TrA>;
    constexpr int KEYLEN = SPH_A_FLEN0;
#if SPH_WIDE
    static_assert(KEYLEN <= 42, "barcodes of up to 42 bases fit the 128-bit table");
    static_assert(!SPH_PARTITIONED, "wide tables are not filled part by part");
    using KeyT = ulonglong2;
    using PlaneT = unsigned long long;
    constexpr unsigned long long KMASK = (1ull << KEYLEN) - 1ull;
#else
    static_assert(KEYLEN >= 1 && KEYLEN <= 21, "barcodes of up to 21 bases fit the 64-bit table");
    using KeyT = unsigned long long;
    using PlaneT = uint32_t;
    constexpr uint32_t KMASK = low_mask(KEYLEN);
#endif
    constexpr uint32_t BYTES_A = GROUP * DA::TILE_BYTES;
    __shared__ __align__(128) uint32_t stage_a[WARPS][STAGES][GROUP * DA::TILE_WORDS];
    __shared__ __align__(8) unsigned long long bar_all[WARPS][STAGES];
#if SPH_PARTITIONED
    __shared__ uint32_t part_cursor[WARPS][32];   // keys this warp has appended to each part's list
#endif

    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int warp = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int nwarps = (int)((gridDim.x * blockDim.x) >> 5);
    const uint32_t n = (uint32_t)reads.n;
    const int ntiles = (int)((n + TILE - 1) / TILE);
    const int ngroups = (ntiles + GROUP - 1) / GROUP;

    const uint32_t base_a = smem_addr(&stage_a[wib][0][0]);
    const uint32_t bar_base = smem_addr(&bar_all[wib][0]);
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) mbar_init(bar_base + 8u * s, 1);
        fence_barrier_init();
    }
#if SPH_PARTITIONED
    part_cursor[wib][lane] = 0;
#endif
    __syncwarp();
    const uint64_t policy = evict_first_policy();
    auto fetch = [&](int g, uint32_t stage) {
        const uint32_t bytes = (uint32_t)min(GROUP, ntiles - GROUP * g) * DA::TILE_BYTES;
        tma_fetch(bar_base + 8u * stage, base_a + stage * BYTES_A, reinterpret_cast<const char*>(reads.data) + (size_t)g * BYTES_A, bytes, bytes,
                  policy);
    };
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
        if (warp + s * nwarps < ngroups) fetch(warp + s * nwarps, (uint32_t)s);
    }

    // carried from one tile to the next: the barcode, its home in the count table and what the home's two slots (one
    // 32-byte sector: two 16-byte slots of a narrow table, two 16-byte keys of a wide one) held when requested
    KeyT pkey{};
    unsigned long long ppos = 0;
    uint4 pa = make_uint4(0, 0, 0, 0), pb = make_uint4(0, 0, 0, 0);
    bool pinsert = false;
    const uint32_t region_base = (uint32_t)warp * def.per_warp;
    uint32_t cursor = 0;   // warp-uniform: entries in this warp's region of the deferred list

    uint32_t stage = 0, parity = 0;
    int group = warp, tile_in_group = 0, tiles_here = 0;
    bool have = group < ngroups;
    if (have) {
        mbar_wait(bar_base, 0);
        tiles_here = min(GROUP, ntiles - GROUP * group);
    }
    for (;;) {
        KeyT key{};
        bool insert = false;
        if (have) {
            const uint32_t i = (uint32_t)(group * GROUP + tile_in_group) * TILE + lane;
            const bool inrange = i < n;
            uint32_t meta = 0;
            PlaneT kh = 0, kl = 0, kn = 0;
            int ncand = 0;
            {
                Words<TrA::W> R;
                load_words<TrA::W>(stage_a[wib][stage] + tile_in_group * DA::TILE_WORDS + lane, R);
                Planes<TrA::W> P;
                make_planes<TrA::W>(R, P);
                // the barcode is cut at the FORWARD coordinates on both strands (:106-108; SURVEY 8.1 T9)
                scan_blocks<TrA, 0>(R, P, inrange, ncand, meta, [&](const uint32_t(&wh)[DA::TW + 1], const uint32_t(&wl)[DA::TW + 1],
                                                                   const uint32_t(&wn)[DA::TW + 1], bool) {
#if SPH_WIDE
                    kh = window_bits64<SPH_A_FSTART0, KEYLEN>(wh);
                    kl = window_bits64<SPH_A_FSTART0, KEYLEN>(wl);
                    kn = window_bits64<SPH_A_FSTART0, KEYLEN>(wn);
#else
                    kh = window_bits<SPH_A_FSTART0, KEYLEN>(wh);
                    kl = window_bits<SPH_A_FSTART0, KEYLEN>(wl);
                    kn = window_bits<SPH_A_FSTART0, KEYLEN>(wn);
#endif
                });
            }
            if (++tile_in_group == tiles_here) {
                __syncwarp();
                const int ahead = group + STAGES * nwarps;
                if (ahead < ngroups) fetch(ahead, stage);
            }
            const bool cand = (meta & SM_CAND) != 0;
            // first mode: the first window (:126-137); best mode: the minimum of the constant mismatches must be attained once
            // (:139-177) -- one verified window is that minimum, several go through the full scan
            const bool slowp = cand && !SPH_USE_FIRST && ncand > 1;
            const bool counted = cand && !slowp;
            const bool rev = (meta & SM_REV) != 0;
            if (rev) {
                // reverse complement of the KEYLEN bases; an N stays an N
#if SPH_WIDE
                const PlaneT rh = __brevll(kh) >> (64 - KEYLEN), rl = __brevll(kl) >> (64 - KEYLEN), rn = __brevll(kn) >> (64 - KEYLEN);
#else
                const uint32_t rh = __brev(kh) >> (32 - KEYLEN), rl = __brev(kl) >> (32 - KEYLEN), rn = __brev(kn) >> (32 - KEYLEN);
#endif
                kh = ~rh & KMASK & ~rn;
                kl = ~rl & KMASK & ~rn;
                kn = rn;
            }
            const bool is_odd = odd != nullptr && inrange && odd[i] != 0;
            if (inrange && !slowp) {
                if (SPH_HAS_INDEX) __stcs(out_index + i, counted ? (int)((meta & 0xFFFFu) * 2u + (rev ? 1u : 0u)) : -1);
                if (counted && is_odd) {
                    // characters the packed planes cannot render: the host formats the barcode from the raw read (:93-120)
                    const unsigned long long at = atomicAdd(odd_count, 1ull);
                    odd_out[at] = OddOutcome{ read_offset + (long long)i, (int)(meta & 0xFFFFu), rev ? 1 : 0 };
                }
            }
            slow_append(slow, slowp && inrange, lane, i);
            insert = inrange && counted && !is_odd;
#if SPH_WIDE
            key = random_key128(kh, kl, kn);
#else
            key = random_key64(kh, kl, kn);
#endif
        }

#if SPH_PARTITIONED
        // ---- this tile's barcodes go to the lists of the table parts they live in (libdev.hpp PartitionedKeys): lanes with
        // the same part line up behind that part's cursor; nothing here touches the table ----
        {
            const uint32_t part = insert ? (uint32_t)(count_home(table, key) >> parts.shift) : 0xFFFFFFFFu;
            const uint32_t peers = __match_any_sync(0xFFFFFFFFu, part);
            const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
            const uint32_t base = insert ? part_cursor[wib][part] : 0u;
            __syncwarp();
            if (insert) {
                if (rank == 0) part_cursor[wib][part] = base + __popc(peers);
                const uint32_t at = base + rank;
                if (at < parts.cap) {
                    __stcs(parts.keys + ((size_t)part * parts.nwarps + warp) * parts.cap + at, key);
                } else {
                    count_insert64(table, key, 1u);   // the list is full (a very uneven batch): straight to the table
                }
            }
            __syncwarp();
        }
        if (!have) break;
#else
        // ---- count the PREVIOUS tile's barcodes: their homes were requested one scan ago.  A barcode found in its home
        // sector is counted with one fire-and-forget atomic; one that is not there yet (new, or pushed further along by a
        // collision) goes to the deferred list and the follow-up kernel inserts it -- no compare-and-swap round trip, no
        // probing loop, nothing this warp has to wait for ----
#if SPH_WIDE
        {
            const uint32_t x0 = (uint32_t)pkey.x, x1 = (uint32_t)(pkey.x >> 32), y0 = (uint32_t)pkey.y, y1 = (uint32_t)(pkey.y >> 32);
            const bool hit_a = pinsert && pa.x == x0 && pa.y == x1 && pa.z == y0 && pa.w == y1;
            const bool hit_b = pinsert && pb.x == x0 && pb.y == x1 && pb.z == y0 && pb.w == y1;
            if (hit_a || hit_b) atomicAdd(table.counts + ppos + (hit_a ? 0u : 1u), 1u);
            const uint32_t entry[4] = { x0, x1, y0, y1 };
            defer_append<4>(def, region_base, cursor, pinsert && !hit_a && !hit_b, lane, entry);
        }

        // ---- this tile's barcodes: request their home sectors ----
        pinsert = insert;
        pkey = key;
        if (insert) {
            ppos = count_home128(table, key);
            const uint4* __restrict__ home = reinterpret_cast<const uint4*>(table.keys + ppos);
            pa = __ldcg(home);
            pb = __ldcg(home + 1);
        }
#else
        {
            const unsigned long long ka = (unsigned long long)pa.x | ((unsigned long long)pa.y << 32);
            const unsigned long long kb = (unsigned long long)pb.x | ((unsigned long long)pb.y << 32);
            const bool hit_a = pinsert && ka == pkey, hit_b = pinsert && kb == pkey;
            if (hit_a || hit_b) atomicAdd(&table.slots[ppos + (hit_a ? 0u : 1u)].count, 1u);
            const uint32_t entry[2] = { (uint32_t)pkey, (uint32_t)(pkey >> 32) };
            defer_append<2>(def, region_base, cursor, pinsert && !hit_a && !hit_b, lane, entry);
        }

        // ---- this tile's barcodes: request their home sectors ----
        pinsert = insert;
        pkey = key;
        if (insert) {
            ppos = count_home(table, key);
            const uint4* __restrict__ home = reinterpret_cast<const uint4*>(table.slots + ppos);
            pa = __ldcg(home);
            pb = __ldcg(home + 1);
        }
#endif

        if (!have) break;
#endif
        if (tile_in_group == tiles_here) {
            group += nwarps;
            tile_in_group = 0;
            if (++stage == STAGES) {
                stage = 0;
                parity ^= 1u;
            }
            have = group < ngroups;
            if (have) {
                mbar_wait(bar_base + 8u * stage, parity);
                tiles_here = min(GROUP, ntiles - GROUP * group);
            }
        }
    }
#if SPH_PARTITIONED
    if ((uint32_t)lane < parts.nparts) parts.counts[(size_t)lane * parts.nwarps + warp] = min(part_cursor[wib][lane], parts.cap);
    (void)pa; (void)pb; (void)ppos; (void)pkey; (void)pinsert; (void)region_base; (void)cursor;
#else
    if (lane == 0) def.warp_counts[warp] = cursor;
#endif
}
#endif  // SPH_KIND == 3
