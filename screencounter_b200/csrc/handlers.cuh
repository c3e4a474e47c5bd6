// Per-read decision logic of each barcode design, as device functions over the building blocks
// of device_scan.cuh, plus the kernels that run them: one thread per read (pair), one warp per
// tile of 32 reads, a grid of persistent warps striding over the tiles.
//
// Reference logic restated here (inst/include/kaori/...):
//   single       SimpleSingleMatch::search_first / search_best        SimpleSingleMatch.hpp:200-306
//   random       RandomBarcodeSingleEnd::process                      handlers/RandomBarcodeSingleEnd.hpp:122-181
//   combo (SE)   CombinatorialBarcodesSingleEnd::process_first/best   handlers/CombinatorialBarcodesSingleEnd.hpp:149-258
//   dual (SE)    DualBarcodesSingleEnd::process_first/best            handlers/DualBarcodesSingleEnd.hpp:144-231
//   combo (PE)   CombinatorialBarcodesPairedEnd::process              handlers/CombinatorialBarcodesPairedEnd.hpp:167-242
//   dual (PE)    DualBarcodesPairedEnd::process                       handlers/DualBarcodesPairedEnd.hpp:229-381
#pragma once

#include "count_table.cuh"
#include "device_scan.cuh"
#include "handlers_params.hpp"

namespace scg {

// Which reads a kernel visits: every read of the batch (list == nullptr), or the reads whose indices a specialised
// kernel listed as needing the full per-read search (spec_handlers.cuh; *list_count entries).
struct ReadList {
    const uint32_t* list;
    const uint32_t* list_count;
};
__device__ __forceinline__ long long visit_rounds(const ReadList& v, long long n) {
    const long long items = v.list ? (long long)*v.list_count : n;
    return (items + TILE - 1) / TILE;
}
// the read (pair) index this lane handles in round t, or -1
__device__ __forceinline__ long long visit_index(const ReadList& v, long long n, long long t, int lane) {
    const long long k = t * TILE + lane;
    if (v.list) return k < (long long)*v.list_count ? (long long)v.list[k] : -1;
    return k < n ? k : -1;
}
__device__ __forceinline__ ReadView read_view_at(const ReadsDev& r, long long i) {
    if (i < 0) {
        ReadView v;
        v.ptr = r.data;
        v.W = r.W;
        v.len = 0;
        return v;
    }
    return read_view(r, i / TILE, (int)(i % TILE));
}

// -------------------------------------------------------------------------------------------
// single barcode (also the building block of the paired combinatorial design)
// -------------------------------------------------------------------------------------------


template <int CB, int KW>
__device__ __forceinline__ SingleOut single_search(const ReadView& rd, const SingleParams& P, bool use_first) {
    SingleOut out{ false, -1, 0, false, 0, 0 };
    const ScanSpec& s = P.spec;
    int best = P.max_mm + 1;
    const int nblocks = window_blocks(rd.len, s.T);
    for (int pb = 0; pb < nblocks; ++pb) {
        Counter<CB> cf, cr;
        scan_block<CB>(rd, s, pb, cf, cr);
        const uint32_t valid = valid_windows(rd.len, s.T, pb);
        uint32_t okf = s.fwd ? (cf.le(s.mm) & valid) : 0u;
        uint32_t okr = s.rev ? (cr.le(s.mm) & valid) : 0u;
        // hits in the reference's order: positions ascending, forward before reverse at each
        // position (SimpleSingleMatch.hpp:226-242); each lane walks its own list, one hit per trip,
        // the strand being per-lane data so that forward and reverse hits share the instructions
        while (okf | okr) {
            const int p = __ffs(okf | okr) - 1;
            const bool rev = !((okf >> p) & 1u);
            if (rev) {
                okr &= ~(1u << p);
            } else {
                okf &= ~(1u << p);
            }
            const int c = rev ? cr.get(p) : cf.get(p);
            Key<KW> key;
            extract_region<KW>(rd, 32 * pb + p + (rev ? s.rstart[0] : s.fstart[0]), s.rlen_f[0], key);
            const Hit h = lookup_any<KW>(P.libs + (rev ? 1 : 0), key, P.max_mm - c);
            if (h.index < 0) continue;
            const int total = c + h.dist;
            if (use_first) {
                out.found = true;
                out.index = h.index;
                out.position = 32 * pb + p;
                out.reverse = rev;
                out.mismatches = total;
                out.var_mismatches = h.dist;
                return out;
            }
            if (total == best) {  // SimpleSingleMatch.hpp:270-275: equal total, different barcode -> ambiguous, sticky
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
    return out;
}

// counts[index]++ fused into the search (SingleBarcodeSingleEnd::process, handlers/SingleBarcodeSingleEnd.hpp:93-104)
template <int CB, int KW>
__global__ void __launch_bounds__(128) single_kernel(ReadsDev reads, SingleParams P, int32_t* __restrict__ counts,
                                                     int32_t* __restrict__ out_index, uint32_t* __restrict__ out_info) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long ntiles = (reads.n + TILE - 1) / TILE;
    for (long long tile = warp; tile < ntiles; tile += nwarps) {
        const long long i = tile * TILE + lane;
        const ReadView rd = read_view(reads, tile, lane);
        const SingleOut o = single_search<CB, KW>(rd, P, P.use_first != 0);
        if (i < reads.n) {
            if (o.found) atomicAdd(counts + o.index, 1);
            if (out_index) out_index[i] = o.found ? o.index : -1;
            if (out_info) out_info[i] = pack_info(o.found, o.reverse, o.mismatches, o.var_mismatches, o.position);
        }
    }
}

// -------------------------------------------------------------------------------------------
// random barcodes
// -------------------------------------------------------------------------------------------


// A key of more than 42 bases as the text-order words of SortedTable (three bits a base, 21 bases a word, the first base most
// significant) into its staging row; returns the key's hash (long_key_hash of those words).
template <int KW>
__device__ __forceinline__ unsigned long long store_long_key(const Key<KW>& key, int len, unsigned long long* row) {
    unsigned long long h = 0, s = 0;
    int in_word = 0, w = 0;
#pragma unroll
    for (int pw = 0; pw < KW; ++pw) {
        const uint32_t H = key.h[pw], L = key.l[pw], N = key.n[pw];
        const int end = min(32, len - 32 * pw);
        for (int j = 0; j < end; ++j) {
            const uint32_t code = (((H >> j) & 1u) << 1) | ((L >> j) & 1u);
            const uint32_t rank = ((N >> j) & 1u) ? 3u : (code == 3u ? 4u : code);
            s = (s << 3) | rank;
            if (++in_word == 21) {
                row[w++] = s;
                h = long_hash_step(h, s);
                s = 0;
                in_word = 0;
            }
        }
    }
    if (in_word) {
        row[w] = s;
        h = long_hash_step(h, s);
    }
    return long_hash_final(h);
}

template <int CB, int KW>
__global__ void __launch_bounds__(128) random_kernel(ReadsDev reads, RandomParams P, CountTable64 t64, CountTable128 t128, CountTableLong tl,
                                                     const uint8_t* __restrict__ odd, long long read_offset,
                                                     OddOutcome* __restrict__ odd_out, unsigned long long* __restrict__ odd_count,
                                                     int32_t* __restrict__ out_index, ReadList visit) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long ntiles = visit_rounds(visit, reads.n);
    const ScanSpec& s = P.spec;
    for (long long tile = warp; tile < ntiles; tile += nwarps) {
        const long long i = visit_index(visit, reads.n, tile, lane);
        const ReadView rd = read_view_at(reads, i);
        int best = P.max_mm + 1, best_pos = 0;
        bool best_rev = false, tied = false, have = false;
        const int nblocks = window_blocks(rd.len, s.T);
        for (int pb = 0; pb < nblocks && !(P.use_first && have); ++pb) {
            Counter<CB> cf, cr;
            scan_block<CB>(rd, s, pb, cf, cr);
            const uint32_t valid = valid_windows(rd.len, s.T, pb);
            const uint32_t okf = s.fwd ? (cf.le(s.mm) & valid) : 0u;
            const uint32_t okr = s.rev ? (cr.le(s.mm) & valid) : 0u;
            uint32_t both = okf | okr;
            if (P.use_first) {  // first window, forward before reverse (:126-137)
                if (both) {
                    const int p = __ffs(both) - 1;
                    have = true;
                    best_pos = 32 * pb + p;
                    best_rev = !((okf >> p) & 1u);
                }
                continue;
            }
            while (both) {  // minimum constant mismatches, must be attained once (:139-177)
                const int p = __ffs(both) - 1;
                both &= both - 1;
                for (int rev = 0; rev < 2; ++rev) {
                    if (!(((rev ? okr : okf) >> p) & 1u)) continue;
                    const int c = rev ? cr.get(p) : cf.get(p);
                    if (c < best) {
                        best = c;
                        best_pos = 32 * pb + p;
                        best_rev = rev != 0;
                        tied = false;
                    } else if (c == best) {
                        tied = true;
                    }
                }
            }
        }
        const bool counted = P.use_first ? have : (!tied && best <= P.max_mm);
        if (i >= 0) {
            if (out_index) out_index[i] = counted ? (best_pos * 2 + (best_rev ? 1 : 0)) : -1;
            if (counted) {
                if (odd && odd[i]) {
                    const unsigned long long slot = atomicAdd(odd_count, 1ull);
                    odd_out[slot] = OddOutcome{ read_offset + i, best_pos, best_rev ? 1 : 0 };
                } else {
                    Key<KW> key;
                    // forward coordinates on BOTH strands (:106-108, SURVEY 8.1 T9 "Quirk B")
                    extract_region<KW>(rd, best_pos + s.fstart[0], P.key_len, key);
                    if (best_rev) key_revcomp<KW>(key, P.key_len);
                    if (KW == 1 && P.key_len <= 21) {
                        count_insert64(t64, random_key64(key.h[0], key.l[0], key.n[0]), 1u);
                    } else if (KW > 1 && P.key_len > 42) {
                        // the key's row of the staging buffer is read i of this launch; written before the probe (CountTableLong)
                        const unsigned long long h = store_long_key<KW>(key, P.key_len, tl.staging + (unsigned long long)i * (unsigned)tl.words);
                        __threadfence();
                        count_insert_long(tl, h, (unsigned long long)i);
                    } else {
                        // up to 42 bases: H, L, N in 42-bit fields of a 128-bit word
                        unsigned long long H = key.h[0], L = key.l[0], N = key.n[0];
                        if (KW > 1) {
                            H |= (unsigned long long)key.h[KW > 1 ? 1 : 0] << 32;
                            L |= (unsigned long long)key.l[KW > 1 ? 1 : 0] << 32;
                            N |= (unsigned long long)key.n[KW > 1 ? 1 : 0] << 32;
                        }
                        count_insert128(t128, random_key128(H, L, N), 1u);
                    }
                }
            }
        }
    }
}

// -------------------------------------------------------------------------------------------
// combinatorial barcodes, single-end (two variable regions) -- also the "invalid combination"
// tabulator of the dual single-end diagnostics
// -------------------------------------------------------------------------------------------

struct ComboOut {
    bool found;
    int id0, id1;
};

template <int CB, int KW>
__device__ __forceinline__ ComboOut combo_search(const ReadView& rd, const ComboParams& P) {
    ComboOut out{ false, -1, -1 };
    const ScanSpec& s = P.spec;
    int best = P.max_mm + 1;
    const int nblocks = window_blocks(rd.len, s.T);
    for (int pb = 0; pb < nblocks; ++pb) {
        Counter<CB> cf, cr;
        scan_block<CB>(rd, s, pb, cf, cr);
        const uint32_t valid = valid_windows(rd.len, s.T, pb);
        uint32_t okf = s.fwd ? (cf.le(s.mm) & valid) : 0u;
        uint32_t okr = s.rev ? (cr.le(s.mm) & valid) : 0u;
        while (okf | okr) {
            const int p = __ffs(okf | okr) - 1;
            const bool rev = !((okf >> p) & 1u);
            if (rev) {
                okr &= ~(1u << p);
            } else {
                okf &= ~(1u << p);
            }
            int obs = rev ? cr.get(p) : cf.get(p);
            int ids[2] = { -1, -1 };
            bool ok = true;
            // regions in read order with the remaining budget (find_match, :149-186)
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                if (!ok) continue;
                Key<KW> key;
                extract_region<KW>(rd, 32 * pb + p + (rev ? s.rstart[r] : s.fstart[r]), rev ? s.rlen_r[r] : s.rlen_f[r], key);
                const Hit h = lookup_any<KW>(P.libs + (rev ? 2 : 0) + r, key, P.max_mm - obs);
                if (h.index < 0) {
                    ok = false;
                } else {
                    obs += h.dist;
                    if (rev) {
                        ids[1 - r] = h.index;
                    } else {
                        ids[r] = h.index;
                    }
                }
            }
            if (!ok) continue;
            if (P.use_first) {
                out.found = true;
                out.id0 = ids[0];
                out.id1 = ids[1];
                return out;
            }
            if (obs == best) {  // :225-241
                if (out.id0 != ids[0] || out.id1 != ids[1]) out.found = false;
            } else if (obs < best) {
                out.found = true;
                best = obs;
                out.id0 = ids[0];
                out.id1 = ids[1];
            }
        }
    }
    return out;
}

template <int CB, int KW>
__global__ void __launch_bounds__(128) combo_kernel(ReadsDev reads, ComboParams P, ComboSink sink,
                                                    const int32_t* __restrict__ skip_if_found, int32_t* __restrict__ out_pairs, ReadList visit) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long ntiles = visit_rounds(visit, reads.n);
    for (long long tile = warp; tile < ntiles; tile += nwarps) {
        const long long i = visit_index(visit, reads.n, tile, lane);
        ReadView rd = read_view_at(reads, i);
        // diagnostics: only reads the dual handler failed on are tabulated
        // (handlers/DualBarcodesSingleEndWithDiagnostics.hpp:99-104)
        if (skip_if_found && i >= 0 && skip_if_found[i] >= 0) rd.len = 0;
        const ComboOut o = combo_search<CB, KW>(rd, P);
        if (i >= 0) {
            if (o.found) combo_count(sink, o.id0, o.id1);
            if (out_pairs) {
                out_pairs[2 * i] = o.found ? o.id0 : -1;
                out_pairs[2 * i + 1] = o.found ? o.id1 : -1;
            }
        }
    }
}

// -------------------------------------------------------------------------------------------
// dual barcodes, single-end: all variable regions concatenated, ONE any-mismatch search
// -------------------------------------------------------------------------------------------

template <int CB, int KW>
__global__ void __launch_bounds__(128) dual_se_kernel(ReadsDev reads, DualSEParams P, int32_t* __restrict__ counts,
                                                      int32_t* __restrict__ out_index) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long ntiles = (reads.n + TILE - 1) / TILE;
    const ScanSpec& s = P.spec;
    for (long long tile = warp; tile < ntiles; tile += nwarps) {
        const long long i = tile * TILE + lane;
        const ReadView rd = read_view(reads, tile, lane);
        bool found = false, done = false;
        int best = P.max_mm + 1, best_id = -1;
        const int nblocks = window_blocks(rd.len, s.T);
        for (int pb = 0; pb < nblocks && !done; ++pb) {
            Counter<CB> cf, cr;
            scan_block<CB>(rd, s, pb, cf, cr);
            const uint32_t valid = valid_windows(rd.len, s.T, pb);
            uint32_t okf = s.fwd ? (cf.le(s.mm) & valid) : 0u;
            uint32_t okr = s.rev ? (cr.le(s.mm) & valid) : 0u;
            while ((okf | okr) && !done) {
                const int p = __ffs(okf | okr) - 1;
                const bool rev = !((okf >> p) & 1u);
                if (rev) {
                    okr &= ~(1u << p);
                } else {
                    okf &= ~(1u << p);
                }
                const int c = rev ? cr.get(p) : cf.get(p);
                Key<KW> key;
                key_clear(key);
                int off = 0;
                for (int r = 0; r < s.nreg; ++r) {  // find_match, :144-160
                    const int rl = rev ? s.rlen_r[r] : s.rlen_f[r];
                    extract_into<KW>(rd, 32 * pb + p + (rev ? s.rstart[r] : s.fstart[r]), rl, off, key);
                    off += rl;
                }
                const Hit h = lookup_any<KW>(P.libs + (rev ? 1 : 0), key, P.max_mm - c);
                if (h.index < 0) continue;
                if (P.use_first) {
                    found = true;
                    best_id = h.index;
                    done = true;
                    continue;
                }
                const int tot = c + h.dist;
                if (tot == best) {  // :205-222
                    if (best_id != h.index) found = false;
                } else if (tot < best) {
                    found = true;
                    best = tot;
                    best_id = h.index;
                }
            }
        }
        if (i < reads.n) {
            if (found) atomicAdd(counts + best_id, 1);
            if (out_index) out_index[i] = found ? best_id : -1;
        }
    }
}

// -------------------------------------------------------------------------------------------
// combinatorial barcodes, paired-end: two independent single searches per pair
// -------------------------------------------------------------------------------------------

// counters[0] = barcode1_only, counters[1] = barcode2_only
template <int CB, int KW>
__global__ void __launch_bounds__(128) combo_pe_kernel(ReadsDev reads1, ReadsDev reads2, ComboPEParams P, ComboSink sink,
                                                       int32_t* __restrict__ counters, const int32_t* __restrict__ skip_if_found,
                                                       int32_t* __restrict__ out_pairs, int32_t* __restrict__ out_code) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long ntiles = (reads1.n + TILE - 1) / TILE;
    const bool first = P.use_first != 0;
    for (long long tile = warp; tile < ntiles; tile += nwarps) {
        const long long i = tile * TILE + lane;
        ReadView r1 = read_view(reads1, tile, lane);
        ReadView r2 = read_view(reads2, tile, lane);
        const bool skipped = skip_if_found && i < reads1.n && skip_if_found[i] >= 0;
        if (skipped) r1.len = r2.len = 0;
        int code = 0, id0 = -1, id1 = -1;  // 1 pair, 2 barcode1 only, 3 barcode2 only
        const SingleOut a = single_search<CB, KW>(r1, P.m1, first);
        const SingleOut b = single_search<CB, KW>(r2, P.m2, first);
        if (first) {  // handlers/CombinatorialBarcodesPairedEnd.hpp:168-192
            if (a.found && b.found) {
                code = 1; id0 = a.index; id1 = b.index;
            } else if (P.randomized) {
                const SingleOut n1 = single_search<CB, KW>(r2, P.m1, true);
                const SingleOut n2 = single_search<CB, KW>(r1, P.m2, true);
                if (n1.found && n2.found) {
                    code = 1; id0 = n1.index; id1 = n2.index;
                } else if (a.found || n1.found) {
                    code = 2;
                } else if (b.found || n2.found) {
                    code = 3;
                }
            } else if (a.found) {
                code = 2;
            } else if (b.found) {
                code = 3;
            }
        } else if (!P.randomized) {  // :196-203
            if (a.found && b.found) {
                code = 1; id0 = a.index; id1 = b.index;
            } else if (a.found) {
                code = 2;
            } else if (b.found) {
                code = 3;
            }
        } else {  // :204-239
            const SingleOut n1 = single_search<CB, KW>(r2, P.m1, false);
            const SingleOut n2 = single_search<CB, KW>(r1, P.m2, false);
            if (a.found && b.found) {
                const int mm = a.mismatches + b.mismatches;
                if (n1.found && n2.found) {
                    const int rmm = n1.mismatches + n2.mismatches;
                    if (mm > rmm) {
                        code = 1; id0 = n1.index; id1 = n2.index;
                    } else if (mm < rmm) {
                        code = 1; id0 = a.index; id1 = b.index;
                    } else if (a.index == n1.index && b.index == n2.index) {
                        code = 1; id0 = a.index; id1 = b.index;
                    }
                } else {
                    code = 1; id0 = a.index; id1 = b.index;
                }
            } else if (n1.found && n2.found) {
                code = 1; id0 = n1.index; id1 = n2.index;
            } else if (a.found || n1.found) {
                code = 2;
            } else if (b.found || n2.found) {
                code = 3;
            }
        }
        if (i < reads1.n && !skipped) {
            if (code == 1) combo_count(sink, id0, id1);
            if (code == 2) atomicAdd(counters + 0, 1);
            if (code == 3) atomicAdd(counters + 1, 1);
        }
        if (i < reads1.n) {
            if (out_pairs) {
                out_pairs[2 * i] = code == 1 ? id0 : -1;
                out_pairs[2 * i + 1] = code == 1 ? id1 : -1;
            }
            if (out_code) out_code[i] = skipped ? 0 : code;
        }
    }
}

// -------------------------------------------------------------------------------------------
// dual barcodes, paired-end: one template per mate, ONE segmented search over (var1, var2)
// -------------------------------------------------------------------------------------------

struct DualOut {
    int index;   // chosen pool row or -1
    int score;   // total mismatches of the chosen pair (best mode)
};

// One orientation: template 1 on read `ra`, template 2 on read `rb`
// (process_first :258-308, process_best :310-347).
template <int CB, int KW>
__device__ __forceinline__ DualOut dual_pe_search(const ReadView& ra, const ReadView& rb, const DualPEParams& P) {
    DualOut out{ -1, P.mm1 + P.mm2 + 1 };
    const ScanSpec& s1 = P.spec1;
    const ScanSpec& s2 = P.spec2;
    const bool rev1 = s1.rev != 0, rev2 = s2.rev != 0;
    const int nb1 = window_blocks(ra.len, s1.T), nb2 = window_blocks(rb.len, s2.T);
    for (int pb1 = 0; pb1 < nb1; ++pb1) {
        Counter<CB> c1f, c1r;
        scan_block<CB>(ra, s1, pb1, c1f, c1r);
        const Counter<CB>& c1 = rev1 ? c1r : c1f;
        uint32_t ok1 = c1.le(s1.mm) & valid_windows(ra.len, s1.T, pb1);
        while (ok1) {
            const int p1 = __ffs(ok1) - 1;
            ok1 &= ok1 - 1;
            const int m1 = c1.get(p1);
            Key<KW> key1;
            extract_region<KW>(ra, 32 * pb1 + p1 + (rev1 ? s1.rstart[0] : s1.fstart[0]), P.len1, key1);
            // every hit of template 2 on the other read, in position order
            for (int pb2 = 0; pb2 < nb2; ++pb2) {
                Counter<CB> c2f, c2r;
                scan_block<CB>(rb, s2, pb2, c2f, c2r);
                const Counter<CB>& c2 = rev2 ? c2r : c2f;
                uint32_t ok2 = c2.le(s2.mm) & valid_windows(rb.len, s2.T, pb2);
                while (ok2) {
                    const int p2 = __ffs(ok2) - 1;
                    ok2 &= ok2 - 1;
                    const int m2 = c2.get(p2);
                    Key<KW> key = key1;
                    extract_into<KW>(rb, 32 * pb2 + p2 + (rev2 ? s2.rstart[0] : s2.fstart[0]), P.len2, P.len1, key);
                    const Hit h = lookup_segmented<KW>(P.lib, key, P.mm1 - m1, P.mm2 - m2);
                    if (h.index < 0) continue;
                    if (P.use_first) {
                        out.index = h.index;
                        out.score = 0;
                        return out;
                    }
                    const int cur = h.dist + m1 + m2;
                    if (cur < out.score) {
                        out.index = h.index;
                        out.score = cur;
                    } else if (cur == out.score && out.index != h.index) {
                        out.index = -1;
                    }
                }
            }
        }
    }
    return out;
}

template <int CB, int KW>
__global__ void __launch_bounds__(128) dual_pe_kernel(ReadsDev reads1, ReadsDev reads2, DualPEParams P,
                                                      int32_t* __restrict__ counts, int32_t* __restrict__ out_index, ReadList visit) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long ntiles = visit_rounds(visit, reads1.n);
    for (long long tile = warp; tile < ntiles; tile += nwarps) {
        const long long i = visit_index(visit, reads1.n, tile, lane);
        const ReadView r1 = read_view_at(reads1, i);
        const ReadView r2 = read_view_at(reads2, i);
        DualOut best = dual_pe_search<CB, KW>(r1, r2, P);  // process, :353-381
        if (P.randomized) {
            if (P.use_first) {
                if (best.index < 0) best = dual_pe_search<CB, KW>(r2, r1, P);
            } else {
                const DualOut other = dual_pe_search<CB, KW>(r2, r1, P);
                if (best.index < 0 || best.score > other.score) {
                    best = other;
                } else if (best.score == other.score && best.index != other.index) {
                    best.index = -1;
                }
            }
        }
        if (i >= 0) {
            if (best.index >= 0) atomicAdd(counts + best.index, 1);
            if (out_index) out_index[i] = best.index;
        }
    }
}

// -------------------------------------------------------------------------------------------
// small utility kernels
// -------------------------------------------------------------------------------------------

// matchBarcodes: one thread per query key (src/match_barcodes.cpp:7-37)
template <int KW>
__global__ void match_kernel(const uint32_t* __restrict__ qkeys /* n * 3KW: h, l, n */, int nq, const LibDev* lib, int cap,
                             int32_t* __restrict__ index, int32_t* __restrict__ mm) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    Key<KW> q;
#pragma unroll
    for (int w = 0; w < KW; ++w) {
        q.h[w] = qkeys[(size_t)i * 3 * KW + w];
        q.l[w] = qkeys[(size_t)i * 3 * KW + KW + w];
        q.n[w] = qkeys[(size_t)i * 3 * KW + 2 * KW + w];
    }
    const Hit h = lookup_any<KW>(lib, q, cap);
    index[i] = h.index;
    mm[i] = h.index >= 0 ? h.dist : -1;
}

// the segmented search on its own, one thread per query, caps per query (tests)
template <int KW>
__global__ void segmented_probe_kernel(const uint32_t* __restrict__ qkeys /* n * 3KW: h, l, n */, int nq, const LibDev* lib,
                                       const int32_t* __restrict__ caps, int32_t* __restrict__ index, int32_t* __restrict__ mm) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    Key<KW> q;
#pragma unroll
    for (int w = 0; w < KW; ++w) {
        q.h[w] = qkeys[(size_t)i * 3 * KW + w];
        q.l[w] = qkeys[(size_t)i * 3 * KW + KW + w];
        q.n[w] = qkeys[(size_t)i * 3 * KW + 2 * KW + w];
    }
    const Hit h = lookup_segmented<KW>(lib, q, caps[2 * i], caps[2 * i + 1]);
    index[i] = h.index;
    mm[i] = h.index >= 0 ? h.dist : -1;
}

} // namespace scg
