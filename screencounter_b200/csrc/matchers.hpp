// The handlers' matchers: templates + libraries validated on the host (the reference's handler constructors, with their
// error texts) and resident on the device.  Shared by the file-level entry points (runners_*.cu) and the resident plans
// (runners_spec.cu).
#pragma once

#include <algorithm>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "api_common.hpp"

namespace scg {

constexpr int TRIE_MAX_KEY = 64;   // device_keys.cuh TRIE_MAX_LEN: longest key the trie walk handles

// CombinatorialBarcodesPairedEnd (reference handlers/CombinatorialBarcodesPairedEnd.hpp:58-98): two
// independent single-barcode matchers, each on its own configured strand.
struct ComboPEMatcher {
    SingleMatcher m1, m2;
    ComboPEParams params;

    void prepare(const std::string& c1, bool rev1, int mm1, const Pool& p1, const std::string& c2, bool rev2, int mm2, const Pool& p2,
                 bool randomized, bool use_first, Duplicates dup) {
        if (std::max(c1.size(), c2.size()) > (size_t)MAX_TEMPLATE) {
            throw Error("lacking compile-time support for constant regions longer than 256 bp");
        }
        m1.prepare(c1, rev1 ? 1 : 0, p1, mm1, use_first, dup);
        m2.prepare(c2, rev2 ? 1 : 0, p2, mm2, use_first, dup);
        std::memset(&params, 0, sizeof params);
        params.randomized = randomized ? 1 : 0;
        params.use_first = use_first ? 1 : 0;
    }

    void upload(Context& ctx) {
        m1.upload(ctx);
        m2.upload(ctx);
        params.m1 = m1.params;
        params.m2 = m2.params;
    }
};

// DualBarcodesPairedEnd (reference handlers/DualBarcodesPairedEnd.hpp:92-179).
struct DualPEMatcher {
    TemplateSpec t1, t2;
    DeviceLibrary lib;
    DeviceBuffer lib_dev;
    DualPEParams params;

    void prepare(const std::string& c1, bool rev1, int mm1, const Pool& p1, const std::string& c2, bool rev2, int mm2, const Pool& p2,
                 bool randomized, bool use_first) {
        if (std::max(c1.size(), c2.size()) > (size_t)MAX_TEMPLATE) {
            throw Error("lacking compile-time support for constant regions longer than 256 bp");
        }
        t1 = TemplateSpec(c1, rev1 ? 1 : 0);
        t2 = TemplateSpec(c2, rev2 ? 1 : 0);
        if (p1.seqs.size() != p2.seqs.size()) throw Error("both barcode pools should be of the same length");
        if (t1.fwd_regions.size() != 1) throw Error("expected one variable region in the first constant template");
        const int len1 = t1.fwd_regions[0].end - t1.fwd_regions[0].start;
        if (len1 != p1.length) {
            throw Error("length of variable sequences (" + std::to_string(p1.length) + ") should be the same as the variable region (" +
                        std::to_string(len1) + ")");
        }
        if (t2.fwd_regions.size() != 1) throw Error("expected one variable region in the second constant template");
        const int len2 = t2.fwd_regions[0].end - t2.fwd_regions[0].start;
        if (len2 != p2.length) {
            throw Error("length of variable sequences (" + std::to_string(p2.length) + ") should be the same as the variable region (" +
                        std::to_string(len2) + ")");
        }
        // rows = each half reverse-complemented on its own when its strand is reverse (:139-164)
        std::vector<std::string> combined;
        combined.reserve(p1.seqs.size());
        for (size_t i = 0; i < p1.seqs.size(); ++i) {
            combined.push_back((rev1 ? reverse_complement_iupac(p1.seqs[i]) : p1.seqs[i]) +
                               (rev2 ? reverse_complement_iupac(p2.seqs[i]) : p2.seqs[i]));
        }
        // The reference's segmented trie search has a phantom result when the second cap is 0 (SURVEY.md 8.1 T8).  The
        // table search reproduces it for first-segment caps 0 and 1; with 2 or more substitutions on read 1 the library also
        // carries the reference's trie and caps [>= 2, 0] are answered by walking it (device_keys.cuh trie_search_segmented).
        if (mm1 >= 2 && len1 + len2 > TRIE_MAX_KEY) {
            throw Error("countDualBarcodes with 2 or more substitutions on the first read needs variable regions of at most " +
                        std::to_string(TRIE_MAX_KEY) + " bp in total in this engine");
        }
        LibraryOptions opt;
        opt.segmented = true;
        opt.seg1 = len1;
        opt.max_mismatches1 = mm1;
        opt.max_mismatches2 = mm2;
        opt.duplicates = Duplicates::ERROR;
        lib.host = Library(combined, len1 + len2, opt);
        std::memset(&params, 0, sizeof params);
        params.spec1 = t1.scan_spec(mm1);
        params.spec2 = t2.scan_spec(mm2);
        params.mm1 = mm1;
        params.mm2 = mm2;
        params.randomized = randomized ? 1 : 0;
        params.use_first = use_first ? 1 : 0;
        params.len1 = len1;
        params.len2 = len2;
    }

    void upload(Context& ctx) {
        lib.upload(ctx);
        params.lib = upload_lib_array(ctx, std::vector<LibDev>{ lib.dev }, lib_dev);
        params.kw = lib.dev.KW;
        build_exact16(ctx);
        build_flat(ctx);
    }

    // The flattened mismatch-tolerant tables of the follow-up kernel (libdev.hpp DualFlat); flat.nseeds == 0 when the library does
    // not qualify (keys over 48 bases, two or more mismatches on a read, a seed without positions).
    DeviceBuffer flat_ibuckets, flat_rows;
    DualFlat flat;
    void build_flat(Context& ctx) {
        std::memset(&flat, 0, sizeof flat);
        flat_ibuckets.release();
        flat_rows.release();
        const Library& host = lib.host;
        if (host.L > DUAL_MAX_KEYLEN || host.L < 1 || host.KW > 2 || host.nseeds < 1 || host.nseeds > 4 || host.opt.max_mismatches1 > 1 ||
            host.opt.max_mismatches2 > 1 || host.nentries() >= (1u << 24) || host.nbuckets == 0) {
            return;
        }
        const int kw = host.KW;
        for (int sd = 0; sd < host.nseeds; ++sd) {
            uint32_t any = 0;
            for (int w = 0; w < kw; ++w) any |= host.seed_masks[(size_t)sd * kw + w];
            if (!any) return;
        }
        const size_t E = host.nentries(), B = host.nbuckets;
        std::vector<uint32_t> rows((size_t)host.nseeds * E * 4, 0), ib((size_t)host.nseeds * B * 8, 0);
        for (size_t k = 0; k < (size_t)host.nseeds * E; ++k) {
            const size_t e = (size_t)host.cands[k];
            const uint32_t* ek = &host.ent_keys[e * 2 * kw];
            rows[4 * k + 0] = ek[0];
            rows[4 * k + 1] = ek[kw];
            rows[4 * k + 2] = kw > 1 ? (ek[1] | (ek[kw + 1] << 16)) : 0u;
            rows[4 * k + 3] = (uint32_t)host.ent_idx[e];
        }
        for (size_t b = 0; b < (size_t)host.nseeds * B; ++b) {
            const uint2 bk = host.buckets[b];
            if (bk.y == 0) continue;
            const size_t sd = b / B;
            std::memcpy(&ib[8 * b], &rows[4 * (sd * E + bk.x)], 16);
            ib[8 * b + 4] = bk.x;
            ib[8 * b + 5] = bk.y;
        }
        flat_rows.upload(rows.data(), rows.size() * sizeof(uint32_t), ctx.stream);
        flat_ibuckets.upload(ib.data(), ib.size() * sizeof(uint32_t), ctx.stream);
        SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        flat.ibuckets = flat_ibuckets.as<uint4>();
        flat.rows = flat_rows.as<uint4>();
        flat.bucket_mask = (uint32_t)B - 1;
        flat.nentries = (int)E;
        flat.nseeds = host.nseeds;
        for (int sd = 0; sd < host.nseeds; ++sd) {
            flat.seed_lo[sd] = host.seed_masks[(size_t)sd * kw];
            flat.seed_hi[sd] = kw > 1 ? host.seed_masks[(size_t)sd * kw + 1] : 0u;
        }
        const int s1 = host.opt.seg1;
        flat.seg1_lo = s1 >= 32 ? 0xFFFFFFFFu : ((1u << s1) - 1u);
        flat.seg1_hi = s1 > 32 ? ((1u << (s1 - 32)) - 1u) : 0u;
        flat.kw = kw;
        flat.seg1 = s1;
        flat.L = host.L;
        flat.dup_first = host.opt.duplicates == Duplicates::FIRST;
        flat.prefix_slots = lib.dev.prefix_slots;
        flat.prefix_mask = lib.dev.prefix_mask;
        flat.slot_words = lib.dev.slot_words;
    }

    // The 16-byte-slot exact table of the specialised kernel (libdev.hpp DualTables), filled from the library's own cuckoo
    // table so that a lookup answers exactly what the generic probe answers.  Keys of up to 48 bases.
    DeviceBuffer exact16;
    uint32_t exact16_shift = 0;
    void build_exact16(Context& ctx) {
        exact16.release();
        exact16_shift = 0;
        const Library& host = lib.host;
        if (host.L > DUAL_MAX_KEYLEN || host.KW > 2 || host.L < 1) return;
        struct Entry {
            uint32_t x, y, z;
            int32_t value;
        };
        std::vector<Entry> entries;
        const int kw = host.KW;
        const size_t nslots = host.slot_words ? host.slots.size() / host.slot_words : 0;
        for (size_t k = 0; k < nslots; ++k) {
            const uint32_t* slot = &host.slots[k * host.slot_words];
            if ((int32_t)slot[2 * kw] < 0) continue;   // empty
            const uint32_t hh = kw > 1 ? slot[1] : 0u, lh = kw > 1 ? slot[kw + 1] : 0u;
            entries.push_back(Entry{ slot[0], slot[kw], hh | (lh << 16), (int32_t)slot[2 * kw] });
        }
        uint32_t bits = 4;
        while ((1ull << bits) < entries.size() + 1 && bits < 28) ++bits;
        std::vector<uint32_t> table;
        for (;; ++bits) {
            if (bits > 29) return;   // no table: the generic kernel serves the design
            const size_t n = (size_t)1 << bits;
            table.assign(2 * n * 4, 0);
            for (size_t k = 0; k < 2 * n; ++k) table[4 * k + 3] = 0xFFFFFFFFu;
            auto home = [&](const Entry& e, int t) {
                const uint32_t h = dual_hash(e.x, e.y, e.z);
                return (size_t)t * n + ((t == 0 ? h : dual_hash2(h)) >> (32 - bits));
            };
            bool ok = true;
            for (size_t i = 0; i < entries.size() && ok; ++i) {
                Entry cur = entries[i];
                int t = 0;
                ok = false;
                for (int kicks = 0; kicks < 2000; ++kicks) {
                    uint32_t* slot = &table[4 * home(cur, t)];
                    if ((int32_t)slot[3] < 0) {
                        slot[0] = cur.x; slot[1] = cur.y; slot[2] = cur.z; slot[3] = (uint32_t)cur.value;
                        ok = true;
                        break;
                    }
                    if (kicks == 0) {   // try the other home before evicting anyone
                        uint32_t* other = &table[4 * home(cur, 1)];
                        if ((int32_t)other[3] < 0) {
                            other[0] = cur.x; other[1] = cur.y; other[2] = cur.z; other[3] = (uint32_t)cur.value;
                            ok = true;
                            break;
                        }
                    }
                    const Entry evicted{ slot[0], slot[1], slot[2], (int32_t)slot[3] };
                    slot[0] = cur.x; slot[1] = cur.y; slot[2] = cur.z; slot[3] = (uint32_t)cur.value;
                    cur = evicted;
                    t ^= 1;
                }
            }
            if (ok) break;
        }
        exact16.upload(table.data(), table.size() * sizeof(uint32_t), ctx.stream);
        SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        exact16_shift = 32 - bits;
    }
};

// CombinatorialBarcodesSingleEnd<_, 2> (reference handlers/CombinatorialBarcodesSingleEnd.hpp:66-119).
struct ComboMatcher {
    TemplateSpec tmpl;
    DeviceLibrary lib[4];   // [2 * reverse + region]
    DeviceBuffer libs_dev;
    ComboParams params;

    void prepare(const std::string& constant, int strand, const Pool& p1, const Pool& p2, int mismatches, bool use_first, Duplicates dup) {
        tmpl = TemplateSpec(constant, strand);
        const Pool* pools[2] = { &p1, &p2 };
        if (tmpl.fwd_regions.size() != 2) throw Error("expected 2 variable regions in the constant template");
        for (int i = 0; i < 2; ++i) {
            const int rlen = tmpl.fwd_regions[i].end - tmpl.fwd_regions[i].start;
            if (pools[i]->length != rlen) {
                throw Error("length of variable region " + std::to_string(i + 1) + " (" + std::to_string(rlen) +
                            ") should be the same as its sequences (" + std::to_string(pools[i]->length) + ")");
            }
        }
        LibraryOptions opt;
        opt.max_mismatches = mismatches;
        opt.duplicates = dup;
        if (tmpl.fwd) {
            for (int r = 0; r < 2; ++r) lib[r].host = Library(pools[r]->seqs, pools[r]->length, opt);
        }
        if (tmpl.rev) {  // reversed pool order on the reverse strand (:111-116)
            for (int r = 0; r < 2; ++r) lib[2 + r].host = Library(pools[1 - r]->reverse_complemented(), pools[1 - r]->length, opt);
        }
        std::memset(&params, 0, sizeof params);
        params.spec = tmpl.scan_spec(mismatches);
        params.max_mm = mismatches;
        params.use_first = use_first ? 1 : 0;
        params.n1 = (int)p1.seqs.size();
        params.n2 = (int)p2.seqs.size();
    }

    void upload(Context& ctx) {
        std::vector<LibDev> libs(4);
        std::memset(libs.data(), 0, 4 * sizeof(LibDev));
        params.kw = 1;
        for (int k = 0; k < 4; ++k) {
            const bool used = k < 2 ? tmpl.fwd : tmpl.rev;
            if (!used) continue;
            lib[k].upload(ctx);
            libs[k] = lib[k].dev;
            params.kw = std::max(params.kw, lib[k].dev.KW);
        }
        params.libs = upload_lib_array(ctx, libs, libs_dev);
    }
};

// DualBarcodesSingleEnd (reference handlers/DualBarcodesSingleEnd.hpp:64-124).
struct DualSEMatcher {
    TemplateSpec tmpl;
    DeviceLibrary lib[2];
    DeviceBuffer libs_dev;
    DualSEParams params;
    int nchoices = 0;

    void prepare(const std::string& constant, const std::vector<Pool>& pools, int nchoices_, int strand, int mismatches, bool use_first) {
        tmpl = TemplateSpec(constant, strand);
        nchoices = nchoices_;
        if (pools.size() != tmpl.fwd_regions.size()) throw Error("length of 'barcode_pools' should equal the number of variable regions");
        int klen = 0;
        for (size_t i = 0; i < pools.size(); ++i) {
            const int rlen = tmpl.fwd_regions[i].end - tmpl.fwd_regions[i].start;
            if (pools[i].length != rlen) {
                throw Error("length of variable region " + std::to_string(i + 1) + " (" + std::to_string(rlen) +
                            ") should be the same as its sequences (" + std::to_string(pools[i].length) + ")");
            }
            klen += rlen;
        }
        std::vector<std::string> combined(nchoices);  // rows concatenated across the pools (:99-108)
        for (const auto& p : pools) {
            for (int c = 0; c < nchoices; ++c) combined[c] += p.seqs[c];
        }
        LibraryOptions opt;
        opt.max_mismatches = mismatches;
        opt.duplicates = Duplicates::ERROR;
        if (tmpl.fwd) lib[0].host = Library(combined, klen, opt);
        if (tmpl.rev) {  // reverse complement of the whole row (:117-120)
            std::vector<std::string> rc;
            rc.reserve(combined.size());
            for (const auto& s : combined) rc.push_back(reverse_complement_iupac(s));
            lib[1].host = Library(rc, klen, opt);
        }
        std::memset(&params, 0, sizeof params);
        params.spec = tmpl.scan_spec(mismatches);
        params.max_mm = mismatches;
        params.use_first = use_first ? 1 : 0;
    }

    void upload(Context& ctx) {
        std::vector<LibDev> libs(2);
        std::memset(libs.data(), 0, 2 * sizeof(LibDev));
        params.kw = 1;
        for (int k = 0; k < 2; ++k) {
            const bool used = k == 0 ? tmpl.fwd : tmpl.rev;
            if (!used) continue;
            lib[k].upload(ctx);
            libs[k] = lib[k].dev;
            params.kw = std::max(params.kw, lib[k].dev.KW);
        }
        params.libs = upload_lib_array(ctx, libs, libs_dev);
    }
};

// RandomBarcodeSingleEnd (reference handlers/RandomBarcodeSingleEnd.hpp:51-80): a template and nothing else.
struct RandomMatcher {
    TemplateSpec tmpl;
    RandomParams params;
    int key_len = 0;
    bool wide = false;   // barcodes of 22 to 42 bases: 128-bit table keys
    int long_words = 0;  // barcodes of 43 bases or more: a long-key table of this many words per key (CountTableLong)

    void prepare(const std::string& constant, int strand, int mismatches, bool use_first) {
        tmpl = TemplateSpec(constant, strand);
        // the reference dereferences variable_regions()[0] unconditionally (handlers/RandomBarcodeSingleEnd.hpp:93-96, :212-214)
        if (tmpl.fwd_regions.empty()) throw Error("expected at least one variable region in the constant template");
        key_len = tmpl.fwd_regions[0].end - tmpl.fwd_regions[0].start;
        std::memset(&params, 0, sizeof params);
        params.spec = tmpl.scan_spec(mismatches);
        params.max_mm = mismatches;
        params.use_first = use_first ? 1 : 0;
        params.key_len = key_len;
        wide = key_len > 21 && key_len <= 42;
        long_words = key_len > 42 ? table_key_words(key_len) : 0;
    }
};

} // namespace scg

// A compiled handler resident on the device (include/scg.h scg_*_plan_*).
struct scg_plan {
    enum Kind { SINGLE = 0, DUAL = 1, COMBO = 2, RANDOM = 3 };
    scg_ctx* owner = nullptr;
    Kind kind = SINGLE;
    int npool = 0;
    scg::SingleMatcher matcher;                    // SINGLE
    std::shared_ptr<scg::DualPEMatcher> dual;      // DUAL
    std::shared_ptr<scg::ComboMatcher> combo;      // COMBO: the plan owns the tally of combinations
    scg::ComboTally tally;
    std::shared_ptr<scg::RandomMatcher> random;    // RANDOM: the plan owns the count table
    scg::CountTable table;
    std::string kernel_note;
};

// A sorted (key, count) table resident on the device (include/scg.h scg_table_*).
struct scg_table {
    scg_ctx* owner = nullptr;
    scg::SortedTable table;
};
