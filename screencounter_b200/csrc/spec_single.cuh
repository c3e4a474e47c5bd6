// countSingleBarcodes kernel with the TEMPLATE FOLDED IN AT COMPILE TIME.
//
// One warp owns a tile of 32 reads (layout.hpp), one lane one read.  Work per tile:
//
//   FAST PATH (every lane, no divergence)
//     1. the read's bit planes (3 x W words) arrive with coalesced 128-byte loads, the next tile's
//        words are requested before this tile is processed (software prefetch);
//     2. four "is not base X" planes are derived once; the constant-flank scan is then, per constant
//        template position and strand, ONE funnel shift (the 32-window view of that base's plane) plus
//        a carry-save update of a bit-sliced saturating counter -- bit p of every register is window p
//        (replaces ScanTemplate::next / strand_match, ScanTemplate.hpp:183-252);
//     3. the first window that passes (positions ascending, forward before reverse,
//        SimpleSingleMatch.hpp:226-242) has its variable region cut out of the registers and probed
//        in the exact table (one 16-byte load); an exact hit resolves the read on the spot.
//        The two table slots are requested right after the scan and looked at one tile later, so the
//        L2 latency of the probe hides behind the next tile's scan.
//   SLOW PATH (compacted)
//     Reads the fast path cannot settle -- the exact probe missed with budget left for the
//     mismatch-tolerant search, an N inside the variable region, several candidate windows -- are
//     appended, with their variable region, to a per-warp queue in shared memory.  Whenever 32 are
//     waiting the warp runs the mismatch-tolerant search (pigeonhole seeds, every candidate row one
//     16-byte load, best-unique / tie rules of MismatchTrie.hpp:266-343) with all 32 lanes busy on 32
//     different deferred reads, instead of a few lanes of every tile dragging the rest of the warp
//     through the long path.  The rare read with several candidate windows gets the full per-read
//     search (every window, first / best rules) out of line.
//
// This file is compiled twice:
//   * by nvcc at build time for the default configuration below (BASELINE configs[1]'s template),
//     which proves it builds for sm_100a and gives that configuration a precompiled kernel;
//   * by NVRTC at run time (jit.cpp) with the SPEC_* macros of the template in use.
//
// Macros (all required when SPEC_CUSTOM is defined):
//   SPEC_T template length, SPEC_FBASES / SPEC_RBASES the forward / reverse-complemented template
//   as a string of A C G T and '-', SPEC_FWD / SPEC_REV strands searched, SPEC_W words per plane of
//   the batch, SPEC_NB window blocks (ceil((32*W - T + 1) / 32)), SPEC_CB counter planes, SPEC_MM
//   clamped scan budget, SPEC_MAXMM the caller's budget, SPEC_USE_FIRST, SPEC_FSTART / SPEC_RSTART /
//   SPEC_KEYLEN the variable region (at most 32 bases), SPEC_NSEEDS / SPEC_SEEDMASKS the libraries' pigeonhole
//   seeds (0 = deferred reads all take the generic search), SPEC_NAME the kernel's name.
#pragma once

#include "device_keys.cuh"

#ifndef SPEC_CUSTOM
#define SPEC_T 44
#define SPEC_FBASES "CAGCTACGTACG--------------------CCAGCTCGATCG"
#define SPEC_RBASES "CGATCGAGCTGG--------------------CGTACGTAGCTG"
#define SPEC_FWD 1
#define SPEC_REV 1
#define SPEC_W 3
#define SPEC_NB 2
#define SPEC_CB 1
#define SPEC_MM 1
#define SPEC_MAXMM 1
#define SPEC_USE_FIRST 1
#define SPEC_FSTART 12
#define SPEC_RSTART 12
#define SPEC_KEYLEN 20
#define SPEC_NAME spec_single_kernel_default
#endif

#ifndef SPEC_BLOCK
#define SPEC_BLOCK 128
#endif
#ifndef SPEC_MIN_BLOCKS
#define SPEC_MIN_BLOCKS 6
#endif
#ifndef SPEC_STAGES
#define SPEC_STAGES 2
#endif
// pigeonhole seeds of the libraries (library.cpp): number (0 = none usable here) and base-position masks
#ifndef SPEC_NSEEDS
#define SPEC_NSEEDS 2
#define SPEC_SEEDMASKS { 0x3FFu, 0xFFC00u }
#endif
#ifndef SPEC_DUP_FIRST
#define SPEC_DUP_FIRST 0
#endif
// Every read of the batch has this length (0 = lengths differ): enables the second kernel of this file,
// `SPEC_NAME_U`, whose windows, masks and loop bounds are all compile-time constants.
#ifndef SPEC_ULEN
#ifdef SPEC_CUSTOM
#define SPEC_ULEN 0
#else
#define SPEC_ULEN 75
#endif
#endif
#ifndef SPEC_NAME_U
#define SPEC_NAME_U spec_single_kernel_u_default
#endif
#ifndef SPEC_NAME_SLOW
#define SPEC_NAME_SLOW spec_single_kernel_slow_default
#endif
// tiles fetched by one bulk copy of the uniform-length kernel
#ifndef SPEC_GROUP
#define SPEC_GROUP 2
#endif
// whether the uniform-length kernel is ever asked for the per-read info word (traces)
#ifndef SPEC_INFO
#define SPEC_INFO 1
#endif
// the joint exact table of both strands (libdev.hpp SpecTables::joint) is there: same table for every lane, cheap hash
#ifndef SPEC_JOINT
#define SPEC_JOINT 0
#endif
// the caller asks for the per-read index (always, in practice; without it the stores and their null checks go away)
#ifndef SPEC_HAS_INDEX
#define SPEC_HAS_INDEX 1
#endif
// the seed buckets with their first candidate inline (libdev.hpp SpecTables::ibuckets) are there
#ifndef SPEC_IBUCKETS
#define SPEC_IBUCKETS 0
#endif
// the batch of the "uniform-length" kernel has per-read lengths after all (trimmed reads): SPEC_ULEN is then the longest read,
// and every lane masks, block by block, the windows its own read does not have
#ifndef SPEC_RAGGED
#define SPEC_RAGGED 0
#endif
// > 0: the pool is small enough for the counters to be PRIVATISED IN SHARED MEMORY (one histogram of SPEC_HIST ints per block,
// shared-memory atomics per matched read, one global atomic per non-zero counter and block at the end) -- the reference's
// per-thread counter + reduce() of handlers/SingleBarcodeSingleEnd.hpp:93-104,119-125.  Uniform-length kernel only.
#ifndef SPEC_UWARP
#define SPEC_UWARP 0
#endif
#ifndef SPEC_HIST
#define SPEC_HIST 0
#endif

namespace scg {
namespace spec {

constexpr int T = SPEC_T;
constexpr int W = SPEC_W;
constexpr int NB = SPEC_NB;
constexpr int CB = SPEC_CB;
constexpr int KEYLEN = SPEC_KEYLEN;
constexpr int WARPS = SPEC_BLOCK / 32;
constexpr int QCAP = 64;   // per-warp queue of deferred reads: < 32 waiting + at most 32 new ones
constexpr int STAGES = SPEC_STAGES;                 // tiles in flight per warp
constexpr int TILE_WORDS = 3 * W * TILE;            // one tile = 3 planes x W words x 32 lanes, contiguous
constexpr uint32_t TILE_BYTES = TILE_WORDS * 4u;    // a multiple of 16, as the bulk copy requires
constexpr char FB[] = SPEC_FBASES;
constexpr char RB[] = SPEC_RBASES;

__host__ __device__ constexpr int count_constant(const char* s) {
    int n = 0;
    for (int j = 0; j < T; ++j) n += s[j] != '-';
    return n;
}
// template position of the k-th constant base of a strand
__host__ __device__ constexpr int kth_constant(const char* s, int k) {
    int n = 0;
    for (int j = 0; j < T; ++j) {
        if (s[j] != '-') {
            if (n == k) return j;
            ++n;
        }
    }
    return 0;
}
constexpr int NCF = SPEC_FWD ? count_constant(FB) : 0;
constexpr int NCR = SPEC_REV ? count_constant(RB) : 0;

// The read's words in registers; two zero guard words so that every funnel shift has a partner.
struct Words {
    uint32_t h[W + 2], l[W + 2], n[W + 2];
};

// mismatch planes of one read: bit i of x?[w] is set when base 32*w + i is NOT that base
// (an N, or anything else that is not ACGT, mismatches all four)
struct Planes {
    uint32_t xa[W + 2], xc[W + 2], xg[W + 2], xt[W + 2];
};

__device__ __forceinline__ void make_planes(const Words& R, Planes& P) {
#pragma unroll
    for (int w = 0; w < W; ++w) {
        const uint32_t h = R.h[w], l = R.l[w], n = R.n[w];
        P.xa[w] = h | l | n;
        P.xc[w] = h | ~l | n;
        P.xg[w] = ~h | l | n;
        P.xt[w] = ~h | ~l | n;
    }
    P.xa[W] = P.xc[W] = P.xg[W] = P.xt[W] = 0;
    P.xa[W + 1] = P.xc[W + 1] = P.xg[W + 1] = P.xt[W + 1] = 0;
}

template <char B>
__device__ __forceinline__ uint32_t window(const Planes& P, int word, int shift) {
    const uint32_t* x = B == 'A' || B == 'a' ? P.xa : (B == 'C' || B == 'c' ? P.xc : (B == 'G' || B == 'g' ? P.xg : P.xt));
    return __funnelshift_r(x[word], x[word + 1], shift);
}

// 32-window mismatch plane of the K-th constant position of a strand, window block pb
template <bool REV, int K>
__device__ __forceinline__ uint32_t cplane(const Planes& P, int pb) {
    constexpr int j = REV ? kth_constant(RB, K) : kth_constant(FB, K);
    constexpr char b = REV ? RB[j] : FB[j];
    return window<b>(P, pb + j / 32, j % 32);
}

// one LOP3 with a chosen truth table (a = 0xF0, b = 0xCC, c = 0xAA)
template <int LUT>
__device__ __forceinline__ uint32_t lop3(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(d) : "r"(a), "r"(b), "r"(c), "n"(LUT));
    return d;
}
__device__ __forceinline__ uint32_t xor3(uint32_t a, uint32_t b, uint32_t c) { return lop3<0x96>(a, b, c); }
__device__ __forceinline__ uint32_t maj3(uint32_t a, uint32_t b, uint32_t c) { return lop3<0xE8>(a, b, c); }
__device__ __forceinline__ uint32_t or3(uint32_t a, uint32_t b, uint32_t c) { return lop3<0xFE>(a, b, c); }

// counts[index]++ : a shared-memory reduction into the block's private histogram when there is one, else a global one
__device__ __forceinline__ void count_hit(int32_t* __restrict__ counts, uint32_t hist_saddr, int index) {
#if SPEC_HIST
    asm volatile("red.shared.add.s32 [%0], 1;" ::"r"(hist_saddr + 4u * (uint32_t)index) : "memory");
#else
    atomicAdd(counts + index, 1);
#endif
}

// ---- TMA (1-D bulk copy global -> shared) signalled on an mbarrier ----
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// dst, bar: shared-memory addresses; src: global pointer, 16-byte aligned
__device__ __forceinline__ void tma_tile(uint32_t dst, const void* src, uint32_t bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(TILE_BYTES) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(TILE_BYTES), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.b32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!done);
}

// Accumulates constant positions K .. N-1 of a strand into the bit-sliced counter.
//   CB == 0 (no mismatch allowed): only "any mismatch" is kept            -> 1/2 LOP3 per position
//   CB == 1 (budget 1): ones / "two or more" planes, carry-save, 4 at once -> 5/4 LOP3 per position
//   otherwise: ripple add, one position at a time
template <bool REV, int K, int N>
struct Accumulate {
    static __device__ __forceinline__ void run(const Planes& P, int pb, Counter<CB>& c) {
        if constexpr (K < N) {
            if constexpr (CB == 0) {
                if constexpr (N - K >= 2) {
                    c.ovf = or3(c.ovf, cplane<REV, K>(P, pb), cplane<REV, K + 1>(P, pb));
                    Accumulate<REV, K + 2, N>::run(P, pb, c);
                } else {
                    c.ovf |= cplane<REV, K>(P, pb);
                }
            } else if constexpr (CB == 1) {
                if constexpr (N - K >= 4) {
                    const uint32_t a = cplane<REV, K>(P, pb), b = cplane<REV, K + 1>(P, pb), d = cplane<REV, K + 2>(P, pb),
                                   e = cplane<REV, K + 3>(P, pb);
                    const uint32_t s = xor3(a, b, d);
                    const uint32_t t = maj3(a, b, d);
                    c.ovf = or3(c.ovf, t, maj3(s, e, c.c[0]));
                    c.c[0] = xor3(c.c[0], s, e);
                    Accumulate<REV, K + 4, N>::run(P, pb, c);
                } else if constexpr (N - K >= 2) {
                    const uint32_t a = cplane<REV, K>(P, pb), b = cplane<REV, K + 1>(P, pb);
                    c.ovf |= maj3(a, b, c.c[0]);
                    c.c[0] = xor3(c.c[0], a, b);
                    Accumulate<REV, K + 2, N>::run(P, pb, c);
                } else {
                    const uint32_t a = cplane<REV, K>(P, pb);
                    c.ovf |= a & c.c[0];
                    c.c[0] ^= a;
                }
            } else {
                c.add(cplane<REV, K>(P, pb));
                Accumulate<REV, K + 1, N>::run(P, pb, c);
            }
        }
    }
};

// value of arr[base + d] for a run-time d in [0, DMAX]; arr lives in registers
template <int DMAX, int LEN>
__device__ __forceinline__ uint32_t pick(const uint32_t (&arr)[LEN], int base, int d) {
    uint32_t v = arr[base];
#pragma unroll
    for (int k = 1; k <= DMAX; ++k) {
        if (base + k < LEN) v = (d == k) ? arr[base + k] : v;
    }
    return v;
}

// the variable region's first word index is one of a few consecutive values known at compile time
__host__ __device__ constexpr int cmin(int a, int b) { return a < b ? a : b; }
__host__ __device__ constexpr int cmax(int a, int b) { return a > b ? a : b; }
constexpr int SMIN = (SPEC_FWD && SPEC_REV) ? cmin(SPEC_FSTART, SPEC_RSTART) : (SPEC_FWD ? SPEC_FSTART : SPEC_RSTART);
constexpr int SMAX = (SPEC_FWD && SPEC_REV) ? cmax(SPEC_FSTART, SPEC_RSTART) : (SPEC_FWD ? SPEC_FSTART : SPEC_RSTART);

// The full per-read search (every window, mismatch-tolerant lookups, first / best rules): the
// reference's SimpleSingleMatch::search_first / search_best (SimpleSingleMatch.hpp:200-306) for one
// read, reading its words from global memory.  Run by a full warp on 32 deferred reads.
__device__ __noinline__ void slow_single(const ReadsDev& reads, const LibDev* __restrict__ libs, long long i, bool active,
                                         int32_t* __restrict__ counts, int32_t* __restrict__ out_index, uint32_t* __restrict__ out_info) {
    if (!active) return;
    const ReadView rd = read_view(reads, i / TILE, (int)(i % TILE));
    Words R;
    Planes P;
#pragma unroll
    for (int w = 0; w < W; ++w) {
        R.h[w] = rd.word(PLANE_H, w);
        R.l[w] = rd.word(PLANE_L, w);
        R.n[w] = rd.word(PLANE_N, w);
    }
    R.h[W] = R.l[W] = R.n[W] = 0;
    R.h[W + 1] = R.l[W + 1] = R.n[W + 1] = 0;
    make_planes(R, P);

    SingleOut out{ false, -1, 0, false, 0, 0 };
    int best = SPEC_MAXMM + 1;
    bool done = false;
    const int nblocks = window_blocks(rd.len, T);
#pragma unroll
    for (int pb = 0; pb < NB; ++pb) {
        if (pb >= nblocks || done) continue;
        Counter<CB> cf, cr;
        cf.clear();
        cr.clear();
        if constexpr (SPEC_FWD) Accumulate<false, 0, NCF>::run(P, pb, cf);
        if constexpr (SPEC_REV) Accumulate<true, 0, NCR>::run(P, pb, cr);
        const uint32_t valid = valid_windows(rd.len, T, pb);
        uint32_t okf = SPEC_FWD ? (cf.le(SPEC_MM) & valid) : 0u;
        uint32_t okr = SPEC_REV ? (cr.le(SPEC_MM) & valid) : 0u;
        // hits in the reference's order: positions ascending, forward before reverse
        // (SimpleSingleMatch.hpp:226-242); the strand is per-lane data
        while ((okf | okr) && !done) {
            const int p = __ffs(okf | okr) - 1;
            const bool rev = !((okf >> p) & 1u);
            if (rev) {
                okr &= ~(1u << p);
            } else {
                okf &= ~(1u << p);
            }
            const int c = rev ? cr.get(p) : cf.get(p);
            Key<1> key;
            extract_region<1>(rd, 32 * pb + p + (rev ? SPEC_RSTART : SPEC_FSTART), KEYLEN, key);
            const Hit h = lookup_any<1>(libs + (rev ? 1 : 0), key, SPEC_MAXMM - c);
            if (h.index < 0) continue;
            const int total = c + h.dist;
            if (SPEC_USE_FIRST) {
                out.found = true;
                out.index = h.index;
                out.position = 32 * pb + p;
                out.reverse = rev;
                out.mismatches = total;
                out.var_mismatches = h.dist;
                done = true;
            } else if (total == best) {  // SimpleSingleMatch.hpp:270-275
                if (out.index != h.index) {
                    out.found = false;
                    out.index = -1;
                }
            } else if (total < best) {
                best = total;
                out.found = true;
                out.index = h.index;
                out.position = 32 * pb + p;
                out.reverse = rev;
                out.mismatches = total;
                out.var_mismatches = h.dist;
            }
        }
    }
    if (out.found) atomicAdd(counts + out.index, 1);
    if (out_index) out_index[i] = out.found ? out.index : -1;
    if (out_info) out_info[i] = pack_info(out.found, out.reverse, out.mismatches, out.var_mismatches, out.position);
}


// What a lane remembers about its read between the scan and the arrival of the table slots.
struct Pending {
    uint4 a, b;        // the two cuckoo slots of the first candidate's variable region (a.x = its N plane when not probed)
    uint32_t kh, kl;   // that region, packed
    uint32_t meta;     // PM_* flags | constant mismatches << 16 | window position
    uint32_t i;        // read index inside the batch
};
constexpr uint32_t PM_CAND = 1u << 31;    // at least one window passed the constant-flank filter
constexpr uint32_t PM_PROBED = 1u << 30;  // slots a, b were requested (the region holds no N and sits in the first block)
constexpr uint32_t PM_MANY = 1u << 29;    // more than one candidate window
constexpr uint32_t PM_REV = 1u << 28;     // the first candidate is on the reverse strand
constexpr uint32_t PM_LATE = 1u << 27;    // the first candidate lies beyond the first window block
constexpr uint32_t PM_INRANGE = 1u << 26; // the lane holds a real read

constexpr int NSEEDS = SPEC_NSEEDS;
__host__ __device__ constexpr uint32_t seed_mask(int sd) {
    constexpr uint32_t masks[] = SPEC_SEEDMASKS;   // at least one element (a dummy when there are no seeds)
    return masks[sd];
}
constexpr uint32_t KEYMASK = KEYLEN >= 32 ? 0xFFFFFFFFu : ((1u << KEYLEN) - 1u);

// best-unique bookkeeping of the mismatch-tolerant search (MismatchTrie.hpp:266-343)
struct Best {
    int dist, index;
    bool ambiguous;
    __device__ __forceinline__ void consider(const uint4 row, uint32_t kh, uint32_t kl, uint32_t kn, int cap, bool valid) {
        const int d = __popc(((kh ^ row.x) | (kl ^ row.y) | kn) & KEYMASK);
        if (!valid || d > cap || d > dist) return;
        const int idx = (int)row.z;
        if (d < dist) {
            dist = d;
            index = idx;
            ambiguous = false;
        } else if (idx != index) {
            if (SPEC_DUP_FIRST) {
                index = min(index, idx);
            } else {
                ambiguous = true;
            }
        }
    }
};

// AnyMismatches::search (MismatchTrie.hpp:446-501) for a region whose exact probe already missed (or that holds an
// N): a barcode within `cap` substitutions agrees with the region on at least one of the cap + 1 seeds, so one
// bucket per seed enumerates every candidate.  Uniform control flow: the bucket loads of all seeds go out
// together, then the first candidate row of each; further rows of a bucket are rare.
__device__ __forceinline__ Hit seeded_search(const SpecTables& tb, bool rev, uint32_t kh, uint32_t kl, uint32_t kn, int cap, bool active) {
    Hit out{ -1, 0 };
    cap = min(cap, KEYLEN);
    active = active && cap > 0 && __popc(kn) <= cap;
    const uint2* __restrict__ buckets = rev ? tb.buckets[1] : tb.buckets[0];
    const uint4* __restrict__ rows = rev ? tb.cand_rows[1] : tb.cand_rows[0];
    const uint32_t bmask = rev ? tb.bucket_mask[1] : tb.bucket_mask[0];
    const int nent = rev ? tb.nentries[1] : tb.nentries[0];
    uint2 bk[NSEEDS > 0 ? NSEEDS : 1];
    uint4 first[NSEEDS > 0 ? NSEEDS : 1], second[NSEEDS > 0 ? NSEEDS : 1];
#if SPEC_IBUCKETS
    // buckets that carry their first candidate: one round of loads settles nine deferred reads in ten
    const uint4* __restrict__ ibuckets = rev ? tb.ibuckets[1] : tb.ibuckets[0];
#pragma unroll
    for (int sd = 0; sd < NSEEDS; ++sd) {
        const uint32_t m = seed_mask(sd);
        const uint32_t mh = kh & m, ml = kl & m;
        first[sd] = make_uint4(0, 0, 0, 0);
        // an N inside the seed: no barcode agrees with the region there
        if (active && !(kn & m)) {
            const uint32_t b = hash_key(&mh, &ml, 1, 0x5EED0000u + sd) & bmask;
            first[sd] = __ldg(ibuckets + (size_t)sd * (bmask + 1) + b);
        }
        bk[sd] = make_uint2(first[sd].w & 0xFFFFFFu, first[sd].w >> 24);
    }
#pragma unroll
    for (int sd = 0; sd < NSEEDS; ++sd) {
        second[sd] = make_uint4(0, 0, 0, 0);
        if (bk[sd].y > 1) second[sd] = __ldg(rows + (size_t)sd * nent + bk[sd].x + 1);
    }
#else
#pragma unroll
    for (int sd = 0; sd < NSEEDS; ++sd) {
        const uint32_t m = seed_mask(sd);
        const uint32_t mh = kh & m, ml = kl & m;
        bk[sd] = make_uint2(0, 0);
        // an N inside the seed: no barcode agrees with the region there
        if (active && !(kn & m)) {
            const uint32_t b = hash_key(&mh, &ml, 1, 0x5EED0000u + sd) & bmask;
            bk[sd] = __ldg(buckets + (size_t)sd * (bmask + 1) + b);
        }
    }
    // the first two candidate rows of every bucket go out together (a bucket with an entry holds a second one 7 % of
    // the time, a third one almost never)
#pragma unroll
    for (int sd = 0; sd < NSEEDS; ++sd) {
        first[sd] = second[sd] = make_uint4(0, 0, 0, 0);
        if (bk[sd].y > 0) first[sd] = __ldg(rows + (size_t)sd * nent + bk[sd].x);
        if (bk[sd].y > 1) second[sd] = __ldg(rows + (size_t)sd * nent + bk[sd].x + 1);
    }
#endif
    Best best{ cap + 1, -1, false };
#pragma unroll
    for (int sd = 0; sd < NSEEDS; ++sd) {
        best.consider(first[sd], kh, kl, kn, cap, bk[sd].y > 0);
        best.consider(second[sd], kh, kl, kn, cap, bk[sd].y > 1);
    }
#pragma unroll
    for (int sd = 0; sd < NSEEDS; ++sd) {
        for (uint32_t c = 2; c < bk[sd].y; ++c) best.consider(__ldg(rows + (size_t)sd * nent + bk[sd].x + c), kh, kl, kn, cap, true);
    }
    if (best.index >= 0 && !best.ambiguous) {
        out.index = best.index;
        out.dist = best.dist;
    }
    return out;
}

} // namespace spec
} // namespace scg

#ifndef SPEC_SKIP_GENERAL
#define SPEC_SKIP_GENERAL 0
#endif
#if !SPEC_SKIP_GENERAL
extern "C" __global__ void __launch_bounds__(SPEC_BLOCK, SPEC_MIN_BLOCKS)
    SPEC_NAME(const scg::ReadsDev reads, const scg::SpecTables tb, int32_t* __restrict__ counts, int32_t* __restrict__ out_index,
              uint32_t* __restrict__ out_info) {
    using namespace scg;
    using namespace scg::spec;
    static_assert(KEYLEN <= 32, "the specialised kernel handles variable regions of at most 32 bases");
    // per warp: a ring of STAGES tile buffers filled by the TMA (1-D bulk copies, one per tile, issued by
    // lane 0 and signalled on an mbarrier), and the queue of deferred reads (index, meta word, variable region)
    __shared__ __align__(128) uint32_t stage_all[WARPS][STAGES][TILE_WORDS];
    __shared__ __align__(8) unsigned long long bar_all[WARPS][STAGES];
    __shared__ uint32_t queue_all[WARPS][5][QCAP];
    const int wib = threadIdx.x >> 5;
    uint32_t(*queue)[QCAP] = queue_all[wib];
    int waiting = 0;   // warp-uniform

    const int lane = threadIdx.x & 31;
    const uint32_t lanes_below = (1u << lane) - 1u;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long ntiles = (reads.n + TILE - 1) / TILE;

    const uint32_t stage_base = smem_addr(&stage_all[wib][0][0]);
    const uint32_t bar_base = smem_addr(&bar_all[wib][0]);
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) mbar_init(bar_base + 8u * s, 1);
        fence_barrier_init();
    }
    __syncwarp();
    const char* src = reinterpret_cast<const char*>(reads.data) + (size_t)warp * TILE_BYTES;
    const size_t src_stride = (size_t)nwarps * TILE_BYTES;
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) {
            if (warp + s * nwarps < ntiles) tma_tile(stage_base + s * TILE_BYTES, src + s * src_stride, bar_base + 8u * s);
        }
    }
    src += STAGES * src_stride;   // the next tile to request

    Pending pend;
    pend.meta = 0;
    pend.a = pend.b = make_uint4(0, 0, 0, 0);
    pend.kh = pend.kl = pend.i = 0;
    long long tile = warp;
    uint32_t stage = 0, parity = 0;
    for (;;) {
        const bool have = tile < ntiles;   // warp-uniform
        Words R;
        uint32_t meta = 0;
        if (have) {
            // ---- this tile's words: wait for the TMA, registers <- shared memory ----
            mbar_wait(bar_base + 8u * stage, parity);
            const uint32_t* buf = stage_all[wib][stage] + lane;
#pragma unroll
            for (int w = 0; w < W; ++w) {
                R.h[w] = buf[(PLANE_H * W + w) * TILE];
                R.l[w] = buf[(PLANE_L * W + w) * TILE];
                R.n[w] = buf[(PLANE_N * W + w) * TILE];
            }
            R.h[W] = R.l[W] = R.n[W] = 0;
            R.h[W + 1] = R.l[W + 1] = R.n[W + 1] = 0;

            const long long i = tile * TILE + lane;
            const bool inrange = i < reads.n;
            const int len = inrange ? (reads.lens ? (int)reads.lens[i] : reads.uniform_len) : 0;
            Planes P;
            make_planes(R, P);

            // ---- scan: every window of every block, both strands ----
            int ncand = 0;            // windows (position, strand) that pass the constant-flank filter
            int fp = 0, fc = 0;       // first candidate in the reference's order: position, constant mismatches
            bool frev = false;
            const int nblocks = window_blocks(len, T);
#pragma unroll
            for (int pb = 0; pb < NB; ++pb) {
                // later blocks only exist for reads longer than T + 31 bases: skipped when no lane has one
                if (pb > 0 && !__any_sync(0xFFFFFFFFu, pb < nblocks)) continue;
                Counter<CB> cf, cr;
                cf.clear();
                cr.clear();
                if constexpr (SPEC_FWD) Accumulate<false, 0, NCF>::run(P, pb, cf);
                if constexpr (SPEC_REV) Accumulate<true, 0, NCR>::run(P, pb, cr);
                const uint32_t valid = valid_windows(len, T, pb);
                const uint32_t okf = SPEC_FWD ? (cf.le(SPEC_MM) & valid) : 0u;
                const uint32_t okr = SPEC_REV ? (cr.le(SPEC_MM) & valid) : 0u;
                const uint32_t any = okf | okr;
                if (any && ncand == 0) {
                    const int p = __ffs(any) - 1;
                    frev = !((okf >> p) & 1u);
                    fc = frev ? cr.get(p) : cf.get(p);
                    fp = 32 * pb + p;
                }
                ncand += __popc(okf) + __popc(okr);
            }
            // the buffer goes back to the TMA once every lane has consumed the words it read from it
            __syncwarp();
            if (lane == 0 && tile + (long long)STAGES * nwarps < ntiles) {
                tma_tile(stage_base + stage * TILE_BYTES, src, bar_base + 8u * stage);
            }
            src += src_stride;
            if (++stage == STAGES) {
                stage = 0;
                parity ^= 1u;
            }
            meta = (inrange ? PM_INRANGE : 0u) | (ncand > 0 ? PM_CAND : 0u) | (ncand > 1 ? PM_MANY : 0u) | (frev ? PM_REV : 0u) |
                   ((NB > 1 && fp >= 32) ? PM_LATE : 0u) | ((uint32_t)fc << 16) | (uint32_t)fp;
        }

        // ---- settle the PREVIOUS tile: its table slots were requested one scan ago ----
        if (__any_sync(0xFFFFFFFFu, pend.meta != 0)) {
            const uint32_t m = pend.meta;
            int index = -1;
            if (m & PM_PROBED) {
                const int ra = (pend.a.x == pend.kh && pend.a.y == pend.kl) ? (int)pend.a.z : -1;
                const int rb = (pend.b.x == pend.kh && pend.b.y == pend.kl) ? (int)pend.b.z : -1;
                index = max(ra, rb);
            }
            const int pfc = (int)((m >> 16) & 0xFFu), pfp = (int)(m & 0xFFFFu);
            // an exact hit at the first window is the answer in first mode, and in best mode when it is the only window
            const bool found = index >= 0 && (SPEC_USE_FIRST || !(m & PM_MANY));
            // otherwise the mismatch-tolerant search may still find something there (budget left), or another window may
            const bool defer = (m & PM_CAND) && !found && ((SPEC_MAXMM - pfc >= 1) || (m & (PM_MANY | PM_LATE)));
            if ((m & PM_INRANGE) && !defer) {
                if (found) atomicAdd(counts + index, 1);
                if (out_index) out_index[pend.i] = found ? index : -1;
                if (out_info) out_info[pend.i] = pack_info(found, (m & PM_REV) != 0, pfc, 0, pfp);
            }
            const uint32_t dm = __ballot_sync(0xFFFFFFFFu, defer);
            if (dm) {
                if (defer) {
                    const int at = waiting + __popc(dm & lanes_below);
                    queue[0][at] = pend.i;
                    queue[1][at] = m;
                    queue[2][at] = pend.kh;
                    queue[3][at] = pend.kl;
                    queue[4][at] = (m & PM_PROBED) ? 0u : pend.a.x;
                }
                waiting += __popc(dm);
                __syncwarp();
            }
        }

        // ---- this tile's first candidate: cut the variable region out of the registers, request its two slots ----
        pend.meta = meta;
        if (have) {
            pend.i = (uint32_t)(tile * TILE + lane);
            if ((meta & PM_CAND) && !(meta & PM_LATE)) {
                const bool frev = (meta & PM_REV) != 0;
                const int start = (int)(meta & 0xFFFFu) + (frev ? SPEC_RSTART : SPEC_FSTART);
                const int a = start >> 5, sh = start & 31;
                // a - base is in [0, DMAX] inside the first block; candidates of later blocks (long reads) take the slow path
                constexpr int base = SMIN >> 5;
                constexpr int DMAX = ((SMAX + 31) >> 5) - base;
                const int d = a - base;
                const uint32_t kh = __funnelshift_r(pick<DMAX>(R.h, base, d), pick<DMAX>(R.h, base + 1, d), sh) & KEYMASK;
                const uint32_t kl = __funnelshift_r(pick<DMAX>(R.l, base, d), pick<DMAX>(R.l, base + 1, d), sh) & KEYMASK;
                const uint32_t kn = __funnelshift_r(pick<DMAX>(R.n, base, d), pick<DMAX>(R.n, base + 1, d), sh) & KEYMASK;
                pend.kh = kh;
                pend.kl = kl;
                pend.a.x = kn;
                if (kn == 0) {
                    // library.cpp CuckooTable: a key sits in T1 at hash & mask or in T2 (mask + 1 slots on) at hash_second(hash) & mask
                    const uint4* __restrict__ slots = frev ? tb.slots[1] : tb.slots[0];
                    const uint32_t mask = frev ? tb.slot_mask[1] : tb.slot_mask[0];
                    const uint32_t acc = hash_key(&kh, &kl, 1, 0);
                    // scattered 16-byte loads that never hit L1: .cg keeps them out of it
                    pend.a = __ldcg(slots + (acc & mask));
                    pend.b = __ldcg(slots + (size_t)(mask + 1) + (hash_second(acc) & mask));
                    pend.meta |= PM_PROBED;
                }
            }
        }

        // ---- deferred reads: searched when a warp's worth is waiting, and whatever is left at the end ----
        while (waiting >= 32 || (!have && waiting > 0)) {
            const int take = waiting < 32 ? waiting : 32;
            waiting -= take;
            const bool active = lane < take;
            const uint32_t qi = active ? queue[0][waiting + lane] : 0u;
            const uint32_t qm = active ? queue[1][waiting + lane] : 0u;
            const uint32_t qh = active ? queue[2][waiting + lane] : 0u;
            const uint32_t ql = active ? queue[3][waiting + lane] : 0u;
            const uint32_t qn = active ? queue[4][waiting + lane] : 0u;
            __syncwarp();
            // one candidate window in the first block: only its variable region is still open
            const bool simple = active && NSEEDS > 0 && !(qm & (PM_MANY | PM_LATE));
            if (NSEEDS > 0) {
                const bool rev = (qm & PM_REV) != 0;
                const int fc = (int)((qm >> 16) & 0xFFu);
                const Hit h = seeded_search(tb, rev, qh, ql, qn, SPEC_MAXMM - fc, simple);
                if (simple) {
                    const bool found = h.index >= 0;
                    if (found) atomicAdd(counts + h.index, 1);
                    if (out_index) out_index[qi] = h.index;
                    if (out_info) out_info[qi] = pack_info(found, rev, fc + h.dist, h.dist, (int)(qm & 0xFFFFu));
                }
            }
            // several candidate windows (or one beyond the first block): the full per-read search
            if (__any_sync(0xFFFFFFFFu, active && !simple)) {
                slow_single(reads, tb.libs, (long long)qi, active && !simple, counts, out_index, out_info);
            }
        }
        if (!have) break;
        tile += nwarps;
    }
}
#endif  // !SPEC_SKIP_GENERAL


// =====================================================================================================================
// Uniform-length variant.  Same per-read outcomes as the kernel above, for batches whose reads all have SPEC_ULEN
// bases (the sequencing-run case: BASELINE configs[1] is 75-base reads, 44-base template, exactly 32 windows = one
// window block; longer reads go through their blocks of 32 windows in turn).  What changes:
//   * FILTER + VERIFY instead of counting every constant position in every window.  A window with at most MM
//     constant mismatches is mismatch-free in at least one of MM + 1 groups of constant positions (pigeonhole), so
//     the bit-sliced pass only ORs the mismatch planes of up to 8 sampled positions per group (one funnel shift and
//     about half a LOP3 per sampled position) and keeps the windows where some group stayed clean.  Each lane then
//     cuts its candidate window out of its registers (funnel shifts by the lane's own position) and counts the
//     constant mismatches exactly with XOR / mask / POPC against the template's words, which are immediates; the
//     variable region falls out of the same window words.  False candidates (about 0.2 % of random reads at 8
//     sampled positions per group) cost another round of the verify loop for their warp.
//   * several tiles per bulk copy, 32-bit read indices, no per-read length loads, no window-validity masks.
// The exact-table probe carried across tiles, the deferred queue and the searches behind it are the ones above.
// =====================================================================================================================
#if SPEC_ULEN > 0

namespace scg {
namespace spec {

constexpr int ULEN = SPEC_ULEN;
constexpr int NWIN = ULEN - T + 1;
static_assert(NWIN >= 1, "the uniform-length kernel needs reads at least as long as the template");
constexpr int NBLOCKS = (NWIN + 31) / 32;   // window blocks: block b holds windows [32 b, 32 b + 32)
// windows of block PB that exist in a read of ULEN bases
template <int PB>
__host__ __device__ constexpr uint32_t block_mask() {
    return NWIN - 32 * PB >= 32 ? 0xFFFFFFFFu : ((1u << (NWIN - 32 * PB)) - 1u);
}
constexpr int TW = (T + 31) / 32;           // words per window
constexpr int GROUP = SPEC_GROUP;           // tiles per bulk copy
constexpr int NGROUPS = SPEC_MM + 1;        // pigeonhole groups of constant positions
#ifndef SPEC_SAMPLES
#define SPEC_SAMPLES 8
#endif
constexpr int SAMPLES = SPEC_SAMPLES;       // sampled positions per group
static_assert(W + 2 >= TW + 1, "window words plus their funnel partner must exist");
static_assert(NBLOCKS - 1 + TW <= W, "the last block's window words and their funnel partners lie within the guarded words");

// constant positions [lo, hi) of a strand's group g
template <bool REV, int G>
struct Group {
    static constexpr int NC = REV ? NCR : NCF;
    static constexpr int lo = NC * G / NGROUPS, hi = NC * (G + 1) / NGROUPS, size = hi - lo;
    static constexpr int S = size < SAMPLES ? size : SAMPLES;
    // the K-th sampled constant position (index among the strand's constant positions), evenly spread
    __host__ __device__ static constexpr int sample(int k) { return lo + (S > 0 ? k * size / S : 0); }
};

// OR of the mismatch planes of a group's sampled positions: bit p set = window p mismatches at a sampled position
template <bool REV, int PB, int G, int K>
__device__ __forceinline__ uint32_t group_any(const Planes& P) {
    using Gr = Group<REV, G>;
    if constexpr (K >= Gr::S) {
        return 0u;
    } else if constexpr (K + 3 <= Gr::S) {
        return cplane<REV, Gr::sample(K)>(P, PB) | cplane<REV, Gr::sample(K + 1)>(P, PB) |
               cplane<REV, Gr::sample(K + 2)>(P, PB) | group_any<REV, PB, G, K + 3>(P);
    } else if constexpr (K + 2 <= Gr::S) {
        return cplane<REV, Gr::sample(K)>(P, PB) | cplane<REV, Gr::sample(K + 1)>(P, PB) | group_any<REV, PB, G, K + 2>(P);
    } else {
        return cplane<REV, Gr::sample(K)>(P, PB) | group_any<REV, PB, G, K + 1>(P);
    }
}

// windows in which EVERY group shows a mismatch among its samples (those cannot be within the budget)
template <bool REV, int PB, int G>
__device__ __forceinline__ uint32_t all_groups_dirty(const Planes& P) {
    if constexpr (G >= NGROUPS) {
        return 0xFFFFFFFFu;
    } else if constexpr (Group<REV, G>::S == 0) {
        return 0u;   // an empty group is trivially clean: nothing can be excluded
    } else {
        return group_any<REV, PB, G, 0>(P) & all_groups_dirty<REV, PB, G + 1>(P);
    }
}

// candidate windows of block PB
template <bool REV, int PB>
__device__ __forceinline__ uint32_t candidate_windows(const Planes& P, uint32_t live) {
    return ~all_groups_dirty<REV, PB, 0>(P) & live;
}

// word k of a strand's template: what = 0 constant-position mask, 1 high bits of the bases, 2 low bits
__host__ __device__ constexpr uint32_t template_word(const char* s, int k, int what) {
    uint32_t w = 0;
    for (int j = 0; j < 32; ++j) {
        const int pos = 32 * k + j;
        if (pos >= T || s[pos] == '-') continue;
        const char c = s[pos];
        const uint32_t code = (c == 'A' || c == 'a') ? 0u : ((c == 'C' || c == 'c') ? 1u : ((c == 'G' || c == 'g') ? 2u : 3u));
        const uint32_t bit = what == 0 ? 1u : (what == 1 ? (code >> 1) : (code & 1u));
        w |= bit << j;
    }
    return w;
}

// Exact constant-mismatch count of window 32 PB + p on a strand; leaves the window's words in wh / wl / wn.
template <int K, int PB>
__device__ __forceinline__ int verify_words(const Words& R, int p, bool rev, uint32_t (&wh)[TW + 1], uint32_t (&wl)[TW + 1],
                                            uint32_t (&wn)[TW + 1]) {
    if constexpr (K >= TW) {
        return 0;
    } else {
        constexpr uint32_t fth = template_word(FB, K, 1), ftl = template_word(FB, K, 2), fcm = template_word(FB, K, 0);
        constexpr uint32_t rth = template_word(RB, K, 1), rtl = template_word(RB, K, 2), rcm = template_word(RB, K, 0);
        wh[K] = __funnelshift_r(R.h[PB + K], R.h[PB + K + 1], p);
        wl[K] = __funnelshift_r(R.l[PB + K], R.l[PB + K + 1], p);
        wn[K] = __funnelshift_r(R.n[PB + K], R.n[PB + K + 1], p);
        const uint32_t th = (SPEC_FWD && SPEC_REV) ? (rev ? rth : fth) : (SPEC_REV ? rth : fth);
        const uint32_t tl = (SPEC_FWD && SPEC_REV) ? (rev ? rtl : ftl) : (SPEC_REV ? rtl : ftl);
        const uint32_t cm = (SPEC_FWD && SPEC_REV) ? (rev ? rcm : fcm) : (SPEC_REV ? rcm : fcm);
        return __popc(((wh[K] ^ th) | (wl[K] ^ tl) | wn[K]) & cm) + verify_words<K + 1, PB>(R, p, rev, wh, wl, wn);
    }
}
template <int PB>
__device__ __forceinline__ int verify_window(const Words& R, int p, bool rev, uint32_t (&wh)[TW + 1], uint32_t (&wl)[TW + 1],
                                             uint32_t (&wn)[TW + 1]) {
    wh[TW] = wl[TW] = wn[TW] = 0;
    return verify_words<0, PB>(R, p, rev, wh, wl, wn);
}

// bits [START, START + KEYLEN) of a window given as words
template <int START>
__device__ __forceinline__ uint32_t window_key(const uint32_t (&w)[TW + 1]) {
    constexpr int a = START >> 5, sh = START & 31;
    const uint32_t lo = w[a], hi = a + 1 <= TW ? w[a + 1] : 0u;
    return (sh == 0 ? lo : __funnelshift_r(lo, hi, sh)) & KEYMASK;
}

// Filter + verify of window block PB (and, recursively, the blocks after it): exact constant mismatches of each candidate, in
// the reference's order (positions ascending, forward before reverse at a position).  `npos` is the lane's number of windows.
// The first block's first round runs unconditionally (nine reads in ten have a candidate); further rounds only while some lane
// still has one.  The first verified window's strand, mismatches, position and variable region go to meta / kh / kl / kn.
template <int PB>
__device__ __forceinline__ void scan_blocks(const Words& R, const Planes& P, int npos, int& ncand, uint32_t& meta, uint32_t& kh,
                                            uint32_t& kl, uint32_t& kn) {
    if constexpr (PB < NBLOCKS) {
#if SPEC_RAGGED
        const int left = npos - 32 * PB;
        const uint32_t live = left <= 0 ? 0u : (left >= 32 ? 0xFFFFFFFFu : ((1u << left) - 1u));
#else
        const uint32_t live = npos > 0 ? block_mask<PB>() : 0u;
#endif
        uint32_t cf = SPEC_FWD ? candidate_windows<false, PB>(P, live) : 0u;
        uint32_t cr = SPEC_REV ? candidate_windows<true, PB>(P, live) : 0u;
        bool more = PB == 0 ? true : __any_sync(0xFFFFFFFFu, (cf | cr) != 0u);
        while (more) {
            const uint32_t any = cf | cr;
            const uint32_t lowest = any & (0u - any);   // 0 when the lane has no candidate left
            const int p = 31 - __clz(lowest | 1u);
            const bool rev = SPEC_FWD ? !(cf & lowest) : true;
            if (rev) {
                cr &= ~lowest;
            } else {
                cf &= ~lowest;
            }
            uint32_t wh[TW + 1], wl[TW + 1], wn[TW + 1];
            const int c = verify_window<PB>(R, p, rev, wh, wl, wn);
            const bool ok = lowest != 0u && c <= SPEC_MM;
            if (ok && ncand == 0) {
                meta = PM_CAND + (rev ? PM_REV : 0u) + ((uint32_t)c << 16) + (uint32_t)(32 * PB + p);
                if (SPEC_FSTART == SPEC_RSTART || !SPEC_REV || !SPEC_FWD) {
                    constexpr int START = (SPEC_FWD && SPEC_REV) ? SPEC_FSTART : (SPEC_FWD ? SPEC_FSTART : SPEC_RSTART);
                    kh = window_key<START>(wh);
                    kl = window_key<START>(wl);
                    kn = window_key<START>(wn);
                } else {
                    kh = rev ? window_key<SPEC_RSTART>(wh) : window_key<SPEC_FSTART>(wh);
                    kl = rev ? window_key<SPEC_RSTART>(wl) : window_key<SPEC_FSTART>(wl);
                    kn = rev ? window_key<SPEC_RSTART>(wn) : window_key<SPEC_FSTART>(wn);
                }
            }
            ncand += ok ? 1 : 0;
            more = __any_sync(0xFFFFFFFFu, (cf | cr) != 0u);
        }
        scan_blocks<PB + 1>(R, P, npos, ncand, meta, kh, kl, kn);
    }
}

// One warp's worth of deferred reads (lane < take holds one): the seeded search for reads with a single candidate
// window.  Reads with several candidate windows need the full per-read search, whose register appetite would
// halve this kernel's occupancy: their indices go to a list in global memory that `SPEC_NAME_SLOW` works off
// right after this kernel, on the same stream.
__device__ __forceinline__ void drain_deferred(const SpecTables& tb, const uint32_t (*queue)[QCAP], int at, int take, int lane,
                                               int32_t* __restrict__ counts, uint32_t hist_saddr, int32_t* __restrict__ out_index,
                                               uint32_t* __restrict__ out_info, uint32_t* __restrict__ slow_list,
                                               uint32_t* __restrict__ slow_count) {
    const bool active = lane < take;
    const uint32_t qi = active ? queue[0][at + lane] : 0u;
    const uint32_t qm = active ? queue[1][at + lane] : 0u;
    const uint32_t qh = active ? queue[2][at + lane] : 0u;
    const uint32_t ql = active ? queue[3][at + lane] : 0u;
    const uint32_t qn = active ? queue[4][at + lane] : 0u;
    __syncwarp();
    const bool simple = active && NSEEDS > 0 && !(qm & PM_MANY);
    if (NSEEDS > 0) {
        const bool rev = (qm & PM_REV) != 0;
        const int fc = (int)((qm >> 16) & 0xFFu);
        const Hit h = seeded_search(tb, rev, qh, ql, qn, SPEC_MAXMM - fc, simple);
        if (simple) {
            const bool found = h.index >= 0;
            if (found) count_hit(counts, hist_saddr, h.index);
            if (out_index) out_index[qi] = h.index;
            if (SPEC_INFO && out_info) out_info[qi] = pack_info(found, rev, fc + h.dist, h.dist, (int)(qm & 0xFFFFu));
        }
    }
    const uint32_t hard = __ballot_sync(0xFFFFFFFFu, active && !simple);
    if (hard) {
        const int leader = __ffs(hard) - 1;
        uint32_t base = 0;
        if (lane == leader) base = atomicAdd(slow_count, (uint32_t)__popc(hard));
        base = __shfl_sync(0xFFFFFFFFu, base, leader);
        if (active && !simple) slow_list[base + __popc(hard & ((1u << lane) - 1u))] = qi;
    }
}

} // namespace spec
} // namespace scg

extern "C" __global__ void __launch_bounds__(SPEC_BLOCK, SPEC_MIN_BLOCKS)
    SPEC_NAME_U(const scg::ReadsDev reads, const scg::SpecTables tb, int32_t* __restrict__ counts, int32_t* __restrict__ out_index,
                uint32_t* __restrict__ out_info, uint32_t* __restrict__ slow_list, uint32_t* __restrict__ slow_count) {
    using namespace scg;
    using namespace scg::spec;
    static_assert(KEYLEN <= 32, "the specialised kernel handles variable regions of at most 32 bases");
    constexpr uint32_t GROUP_BYTES = GROUP * TILE_BYTES;
    __shared__ __align__(128) uint32_t stage_all[WARPS][STAGES][GROUP * TILE_WORDS];
    __shared__ __align__(8) unsigned long long bar_all[WARPS][STAGES];
    __shared__ uint32_t queue_all[WARPS][5][QCAP];
#if SPEC_HIST
    __shared__ int32_t hist[SPEC_HIST];
    for (int k = threadIdx.x; k < SPEC_HIST; k += SPEC_BLOCK) hist[k] = 0;
    __syncthreads();
    const uint32_t hist_saddr = smem_addr(hist);
#else
    const uint32_t hist_saddr = 0;
#endif
#if SPEC_UWARP
    // An experiment (SCG_SPEC_UWARP=1, DESIGN.md 5.1b): the number of the warp read from lane 0, so that the compiler can prove what is
    // warp-uniform.  It then drops the R2UR traffic and a third of the BSSY/BSYNC pairs (316 instead of 341 instructions per tile,
    // 48 registers) but moves the bookkeeping of the loop to the uniform datapath: MIO-throttle and scoreboard stalls, 51.9
    // against 66.9 G reads/s.
    const int wib = __shfl_sync(0xFFFFFFFFu, (int)(threadIdx.x >> 5), 0);
#else
    const int wib = threadIdx.x >> 5;
#endif
    uint32_t(*queue)[QCAP] = queue_all[wib];
    int waiting = 0;   // warp-uniform

    const int lane = threadIdx.x & 31;
    const uint32_t lanes_below = (1u << lane) - 1u;
#if SPEC_UWARP
    const int warp = (int)(blockIdx.x * (blockDim.x >> 5)) + wib;
#else
    const int warp = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
#endif
    const int nwarps = (int)((gridDim.x * blockDim.x) >> 5);
    const uint32_t n = (uint32_t)reads.n;                       // the host sends at most 2^31 - 64 reads per launch
    const int ntiles = (int)((n + TILE - 1) / TILE);
    const int ngroups = (ntiles + GROUP - 1) / GROUP;

    const uint32_t stage_base = smem_addr(&stage_all[wib][0][0]);
    const uint32_t bar_base = smem_addr(&bar_all[wib][0]);
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) mbar_init(bar_base + 8u * s, 1);
        fence_barrier_init();
    }
    __syncwarp();
    // group g = tiles [GROUP * g, GROUP * g + GROUP) (the last group may be short): one bulk copy each
    // The packed reads pass through L2 once: their lines are marked evict-first so that the tables stay resident.
    uint64_t stream_policy;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(stream_policy));
    // one elected lane arms the barrier and issues the copy (called by the whole warp, converged)
    auto fetch = [&](int g, uint32_t stage) {
        const int tiles = min(GROUP, ntiles - GROUP * g);
        const uint32_t bytes = (uint32_t)tiles * TILE_BYTES;
        const uint32_t bar = bar_base + 8u * stage;
        const char* src = reinterpret_cast<const char*>(reads.data) + (size_t)g * GROUP_BYTES;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "elect.sync _|p, 0xFFFFFFFF;\n\t"
            "@p mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t"
            "@p cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%2], [%3], %1, [%0], %4;\n\t}"
            ::"r"(bar), "r"(bytes), "r"(stage_base + stage * GROUP_BYTES), "l"(src), "l"(stream_policy)
            : "memory");
    };
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
        if (warp + s * nwarps < ngroups) fetch(warp + s * nwarps, (uint32_t)s);
    }

    // What a lane carries from one tile to the next: the slots of its candidate's variable region (requested after the scan,
    // looked at one tile later), the region itself, and the flags below.
    //   PM_CAND     a window passed the verify         PM_PROBED  the slots were requested (no N in the region)
    //   PM_MANY     more than one verified window      PM_REV     the first one is on the reverse strand
    //   PM_INRANGE  the lane holds a real read
    //   PU_MISS_DEFERS  (bit 25) if the probe misses, the read is deferred (budget left for the seeded search, or other windows)
    //   PU_ALWAYS_DEFERS (bit 24) deferred whatever the probe says (best mode with several windows)
    constexpr uint32_t PU_MISS_DEFERS = 1u << 25, PU_ALWAYS_DEFERS = 1u << 24;
    Pending pend;
    pend.meta = 0;
    pend.a = pend.b = make_uint4(0, 0, 0, 0);
    pend.kh = pend.kl = pend.i = 0;
    uint32_t stage = 0, parity = 0;
    int group = warp;
    int tile_in_group = 0, tiles_here = 0;
    bool have = group < ngroups;   // warp-uniform
    if (have) {
        mbar_wait(bar_base, 0);
        tiles_here = min(GROUP, ntiles - GROUP * group);
    }
    for (;;) {
        uint32_t meta = 0, kh = 0, kl = 0, kn = 0, i = 0;
        if (have) {
            Words R;
            const uint32_t* buf = stage_all[wib][stage] + tile_in_group * TILE_WORDS + lane;
#pragma unroll
            for (int w = 0; w < W; ++w) {
                R.h[w] = buf[(PLANE_H * W + w) * TILE];
                R.l[w] = buf[(PLANE_L * W + w) * TILE];
                R.n[w] = buf[(PLANE_N * W + w) * TILE];
            }
            R.h[W] = R.l[W] = R.n[W] = 0;
            R.h[W + 1] = R.l[W + 1] = R.n[W + 1] = 0;
            i = (uint32_t)(group * GROUP + tile_in_group) * TILE + lane;
            const bool inrange = i < n;
            Planes P;
            make_planes(R, P);

            // ---- filter + verify, window block by window block ----
#if SPEC_RAGGED
            // windows p with p + T <= this read's length (ScanTemplate.hpp:153,168-170: a read shorter than the template has none)
            const int npos = inrange ? (int)reads.lens[i] - T + 1 : 0;
#else
            const int npos = inrange ? NWIN : 0;
#endif
            int ncand = 0;
            scan_blocks<0>(R, P, npos, ncand, meta, kh, kl, kn);
            // what the settle step will need to know, decided here once
            {
                const bool many = ncand > 1;
                const int fc = (int)((meta >> 16) & 0xFFu);
                const bool cand = (meta & PM_CAND) != 0;
                const bool miss_defers = cand && ((SPEC_MAXMM - fc >= 1) || many);
                const bool always_defers = cand && many && !SPEC_USE_FIRST;
                meta += (inrange ? PM_INRANGE : 0u) + (many ? PM_MANY : 0u) + (miss_defers ? PU_MISS_DEFERS : 0u) +
                        (always_defers ? PU_ALWAYS_DEFERS : 0u);
            }

            // the group's buffer goes back to the TMA once every lane has consumed its last tile
            if (++tile_in_group == tiles_here) {
                __syncwarp();
                const int ahead = group + STAGES * nwarps;
                if (ahead < ngroups) fetch(ahead, stage);
            }
        }

        // ---- settle the PREVIOUS tile: its table slots were requested one scan ago ----
        {
            const uint32_t m = pend.meta;
            int index = -1;
            if (m & PM_PROBED) {
                const int ra = (pend.a.x == pend.kh && pend.a.y == pend.kl) ? (int)pend.a.z : -1;
                const int rb = (pend.b.x == pend.kh && pend.b.y == pend.kl) ? (int)pend.b.z : -1;
                index = max(ra, rb);
            }
            const bool defer = (m & PU_ALWAYS_DEFERS) || ((m & PU_MISS_DEFERS) && index < 0);
            if ((m & PM_INRANGE) && !defer) {
                if (index >= 0) count_hit(counts, hist_saddr, index);
                if (SPEC_HAS_INDEX) __stcs(out_index + pend.i, index);
                if (SPEC_INFO && out_info) {
                    __stcs(out_info + pend.i, pack_info(index >= 0, (m & PM_REV) != 0, (int)((m >> 16) & 0xFFu), 0, (int)(m & 0xFFFFu)));
                }
            }
            const uint32_t dm = __ballot_sync(0xFFFFFFFFu, defer);
            if (dm) {
                if (defer) {
                    const int at = waiting + __popc(dm & lanes_below);
                    queue[0][at] = pend.i;
                    queue[1][at] = m;
#if SPEC_JOINT
                    queue[2][at] = pend.kh & 0x7FFFFFFFu;
#else
                    queue[2][at] = pend.kh;
#endif
                    queue[3][at] = pend.kl;
                    queue[4][at] = (m & PM_PROBED) ? 0u : pend.a.x;
                }
                waiting += __popc(dm);
                __syncwarp();
            }
        }

        // ---- this tile's first candidate: request the two slots of its variable region ----
        pend.meta = meta;
        pend.i = i;
        pend.kl = kl;
        pend.a.x = kn;
#if SPEC_JOINT
        // one table for both strands: the strand is bit 31 of the H word, the homes are the top bits of two multiply-adds
        pend.kh = kh + ((meta & PM_REV) ? 0x80000000u : 0u);
        if ((meta & PM_CAND) && kn == 0) {
            const uint32_t x = joint_hash(pend.kh, kl);
            const uint32_t second = (1u << (32 - tb.joint_shift)) + (joint_hash2(x) >> tb.joint_shift);
            // scattered 16-byte loads that never hit L1: .cg keeps them out of it (measured + 1.7 %)
            pend.a = __ldcg(tb.joint + (x >> tb.joint_shift));
            pend.b = __ldcg(tb.joint + second);
            pend.meta = meta + PM_PROBED;
        }
#else
        pend.kh = kh;
        if ((meta & PM_CAND) && kn == 0) {
            const bool frev = (meta & PM_REV) != 0;
            const uint4* __restrict__ slots = frev ? tb.slots[1] : tb.slots[0];
            const uint32_t mask = frev ? tb.slot_mask[1] : tb.slot_mask[0];
            const uint32_t acc = hash_key(&kh, &kl, 1, 0);
            pend.a = __ldcg(slots + (acc & mask));
            pend.b = __ldcg(slots + (size_t)(mask + 1) + (hash_second(acc) & mask));
            pend.meta = meta + PM_PROBED;
        }
#endif

        // ---- deferred reads: searched when a warp's worth is waiting, and whatever is left at the end ----
        while (waiting >= 32 || (!have && waiting > 0)) {
            const int take = waiting < 32 ? waiting : 32;
            waiting -= take;
            drain_deferred(tb, queue, waiting, take, lane, counts, hist_saddr, out_index, out_info, slow_list, slow_count);
        }
        if (!have) break;
        // ---- next tile: the same group, or the warp's next group ----
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
#if SPEC_HIST
    // flush the block's private histogram: one global atomic per counter that was hit
    __syncthreads();
    for (int k = threadIdx.x; k < SPEC_HIST; k += SPEC_BLOCK) {
        const int32_t v = hist[k];
        if (v) atomicAdd(counts + k, v);
    }
#endif
}

// The reads the kernel above could not settle (several candidate windows): the full per-read search, one lane per
// listed read, any grid.
extern "C" __global__ void __launch_bounds__(128)
    SPEC_NAME_SLOW(const scg::ReadsDev reads, const scg::LibDev* __restrict__ libs, const uint32_t* __restrict__ slow_list,
                   const uint32_t* __restrict__ slow_count, int32_t* __restrict__ counts, int32_t* __restrict__ out_index,
                   uint32_t* __restrict__ out_info) {
    using namespace scg;
    using namespace scg::spec;
    const uint32_t total = *slow_count;
    const uint32_t stride = gridDim.x * blockDim.x;
    // whole warps enter the search together (it votes); lanes past the end of the list idle through it
    for (uint32_t base = (blockIdx.x * blockDim.x + threadIdx.x) & ~31u; base < total; base += stride) {
        const uint32_t k = base + (threadIdx.x & 31);
        const bool active = k < total;
        const uint32_t i = active ? slow_list[k] : 0u;
        slow_single(reads, libs, (long long)i, active, counts, out_index, out_info);
    }
}

#endif  // SPEC_ULEN > 0
