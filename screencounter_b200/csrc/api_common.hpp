// Glue shared by the C-ABI translation units: exception -> status code, pool marshalling,
// template-instantiation dispatch.
#pragma once

#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/scg.h"
#include "engine.hpp"
#include "pipeline.hpp"

namespace scg {

std::string& creation_error();   // message of a failed scg_ctx_create

// Runs f(); any exception becomes status 1 + ctx->last_error (BEGIN_RCPP/END_RCPP equivalent,
// reference src/RcppExports.cpp:16,33).
template <class F>
int guarded(scg_ctx* ctx, F&& f) {
    try {
        if (!ctx) throw Error("null context");
        f();
        return 0;
    } catch (const std::exception& e) {
        if (ctx) {
            ctx->impl.last_error = e.what();
        } else {
            creation_error() = e.what();
        }
        return 1;
    } catch (...) {
        if (ctx) ctx->impl.last_error = "unknown error";
        return 1;
    }
}

// format_pointers (reference src/utils.cpp:5-23): every sequence of a pool has the same length.
struct Pool {
    std::vector<std::string> seqs;
    int length = 0;
    Pool() {}
    Pool(const char* const* p, int n);
    std::vector<std::string> reverse_complemented() const;
};

// Owns one FASTQ input.
struct Source {
    std::unique_ptr<FastqReader> reader;
    explicit Source(const scg_source* s);
};

template <int V>
struct IntC {
    static constexpr int value = V;
};

// Counter planes compiled: 0 (no mismatch allowed), 1 (<= 1), 2 (<= 3), 9 (anything up to 256).
template <class F>
void dispatch_cb(int cbits, F&& f) {
    if (cbits <= 0) {
        f(IntC<0>());
    } else if (cbits == 1) {
        f(IntC<1>());
    } else if (cbits == 2) {
        f(IntC<2>());
    } else {
        f(IntC<9>());
    }
}

// Key words per plane compiled: 1 (<= 32 bases), 2 (<= 64), 8 (<= 256), 16 (<= 512).
template <class F>
void dispatch_kw(int kw, F&& f) {
    if (kw <= 1) {
        f(IntC<1>());
    } else if (kw == 2) {
        f(IntC<2>());
    } else if (kw <= 8) {
        f(IntC<8>());
    } else {
        f(IntC<16>());
    }
}

// 128-bit key over everything that defines a matcher (handler kind, templates, options, the pools' sequences): calls that
// repeat it (one call per FASTQ file of a screen, R/countDualBarcodes.R matrixOf* loops) find the tables already on the
// device.  Only successfully built matchers are cached, so validation errors are raised every time.
struct CacheKey {
    unsigned long long k1 = 1469598103934665603ull, k2 = 0x9E3779B97F4A7C15ull;
    unsigned long long fed = 0;   // bytes fed so far (kept beside the hash as a cheap secondary check of a cache hit)
    void feed(const void* data, size_t n) {
        const char* p = static_cast<const char*>(data);
        fed += n;
        k1 = mix64(k1 ^ n);
        k2 = (k2 ^ (0xA24BAED4963EE407ull + n)) * 1099511628211ull + (k2 >> 29);   // the length goes into both words
        size_t i = 0;
        for (; i + 8 <= n; i += 8) {
            unsigned long long w;
            std::memcpy(&w, p + i, 8);
            k1 = mix64(k1 ^ w);
            k2 = (k2 ^ w) * 1099511628211ull + (k2 >> 29);
        }
        unsigned long long w = 0;
        if (i < n) std::memcpy(&w, p + i, n - i);
        k1 = mix64(k1 ^ w);
        k2 = (k2 ^ w) * 1099511628211ull + (k2 >> 29);
    }
    void feed(int v) { feed(&v, sizeof v); }
    void feed(const std::string& s) { feed(s.data(), s.size()); }
    void feed(const Pool& p) {
        feed((int)p.seqs.size());
        for (const auto& s : p.seqs) feed(s);
    }
};

template <class M, class Build>
std::shared_ptr<M> cached_matcher(Context& ctx, const CacheKey& key, Build&& build) {
    for (auto& e : ctx.matcher_cache) {
        if (e.key1 == key.k1 && e.key2 == key.k2 && e.fed_bytes == key.fed) return std::static_pointer_cast<M>(e.object);
    }
    std::shared_ptr<M> m = build();
    if (ctx.matcher_cache.size() >= 6) ctx.matcher_cache.erase(ctx.matcher_cache.begin());
    Context::CachedObject entry;
    entry.key1 = key.k1;
    entry.key2 = key.k2;
    entry.fed_bytes = key.fed;
    entry.object = m;
    ctx.matcher_cache.push_back(entry);
    return m;
}

// Device scratch for per-read outputs of one batch, copied back after each batch when tracing.
struct TraceSink {
    bool enabled = false;
    int width = 1;
    DeviceBuffer d_index, d_info;
    std::vector<int32_t> index;
    std::vector<uint32_t> info;
    void prepare(long long n, bool want_info);
    void collect(Context& ctx, long long n, bool want_info);
};

// Copies an array of library descriptors to the device (the kernels index it per lane).
const LibDev* upload_lib_array(Context& ctx, const std::vector<LibDev>& libs, DeviceBuffer& storage);

// A single-barcode matcher (template + forward/reverse libraries) resident on the device.
struct SingleMatcher {
    TemplateSpec tmpl;
    DeviceLibrary lib_f, lib_r;
    DeviceBuffer libs_dev;   // LibDev[2] on the device: forward, reverse
    DeviceBuffer joint;      // exact table of both strands (libdev.hpp SpecTables::joint), keys of up to 31 bases
    uint32_t joint_shift = 0;
    DeviceBuffer ibuckets[2]; // seed buckets with the first candidate inline, per strand (SpecTables::ibuckets)
    bool have_ibuckets = false;
    SingleParams params;
    int npool = 0;
    mutable std::string kernel_note;   // which kernel the last launch used, and why
    // SimpleSingleMatch constructor (reference inst/include/kaori/SimpleSingleMatch.hpp:61-97): host-only, throws
    // the reference's validation errors; upload() then moves the tables to the device.
    void prepare(const std::string& constant, int strand, const Pool& pool, int mismatches, bool use_first, Duplicates dup);
    void upload(Context& ctx);
};

// A matcher for these arguments from the context's cache, built and uploaded on a miss (runners_single.cu).
std::shared_ptr<SingleMatcher> cached_single_matcher(Context& ctx, const char* constant, int strand, const char* const* pool, int npool,
                                                     int mismatches, bool use_first);

// Runs the single-barcode kernel over one batch: the run-time specialised kernel (jit.hpp) when it
// can be had, the generic one otherwise.
void launch_single(Context& ctx, const ReadsDev& reads, const SingleMatcher& m, int32_t* d_counts, int32_t* d_index,
                   uint32_t* d_info, cudaStream_t stream);

// A sparse result resident on the device, sorted: what scg_result hands out on demand (scg_result_copy_table) and what the
// multi-GPU merge exchanges.  keys: one 64-bit word per row, ascending -- combinations as first << 32 | second, random
// barcodes as three bits per base in text order (A < C < G < N < T), first base most significant.
struct SortedTable {
    DeviceBuffer keys, counts;   // unsigned long long[rows], uint32_t[rows]
    size_t rows = 0;
    int key_len = 0;             // > 0: random barcodes of this length; 0: combinations
};

// Device count table (libdev.hpp: 16-byte slots for 64-bit keys, separate arrays for 128-bit keys).  Sized for a load
// factor of at most 1/2 of the keys it may hold; how many distinct keys it holds is tracked ON THE DEVICE (a counter bumped
// by every first insert), so the table follows the number of distinct keys, not the number of reads.
struct CountTable {
    bool wide = false;
    DeviceBuffer slots;    // narrow: CountSlot[capacity]; wide: ulonglong2[capacity]
    DeviceBuffer counts;   // wide only: uint32_t[capacity]
    DeviceBuffer live;     // device: [0] distinct keys inserted, [1] overflow flag
    size_t capacity = 0;
    long long live_known = 0;   // distinct keys at the last read-back
    long long pending = 0;      // inserts launched since (each may be a new key)
    bool fixed = false;         // sized by the caller (resident plans): ensure() never grows it
    void init(Context& ctx, bool wide128, size_t initial);
    void reset(Context& ctx, cudaStream_t stream);            // empties the table, asynchronously
    void ensure(Context& ctx, long long upcoming_inserts);    // keeps (distinct keys + upcoming) <= capacity / 2; may synchronise
    void check_overflow(Context& ctx);                        // throws when inserts were dropped (synchronises)
    CountTable64 view64() const;
    CountTable128 view128() const;
    // live entries to the host, unsorted (wide tables)
    void download(Context& ctx, std::vector<unsigned long long>& keys_lo, std::vector<unsigned long long>& keys_hi,
                  std::vector<uint32_t>& counts);
    // narrow tables: live entries sorted on the device.  key_len > 0: keys are random barcodes (random_key64), re-coded to
    // text order before the sort; key_len == 0: sorted as they are (combinations).
    void sorted(Context& ctx, int key_len, SortedTable& out);
};

// device-side helpers on sorted tables (runners_random.cu)
void render_barcodes(Context& ctx, const SortedTable& t, DeviceBuffer& strings, DeviceBuffer& freq);   // rows * key_len chars, int32 freq
void render_combinations(Context& ctx, const SortedTable& t, DeviceBuffer& keys, DeviceBuffer& freq);  // rows * 2 int32 (first, second), int32 freq
// out = t rendered (barcodes when t.key_len > 0, combinations otherwise) and left on the device for scg_result_copy_table
void device_table_result(Context& ctx, const SortedTable& t, scg_result& out);
// c = sorted merge of a and b with the counts of equal keys added (a and b sorted ascending, keys unique within each)
void merge_sorted_tables(Context& ctx, const SortedTable& a, const SortedTable& b, SortedTable& c);

// column[i] = count of all_keys' row i in t (0 where t lacks the key): one column of a many-files count matrix
void scatter_table_column(Context& ctx, const SortedTable& all_keys, const SortedTable& t, int32_t* column);

// Tally of (i, j) combinations: dense matrix when small, count table otherwise.
struct ComboTally {
    int n1 = 0, n2 = 0;
    bool dense = false;
    DeviceBuffer matrix;
    CountTable table;
    void init(Context& ctx, int n1, int n2);
    ComboSink sink(Context& ctx, long long upcoming);
    void reset(Context& ctx, cudaStream_t stream);
    void harvest(Context& ctx, scg_result& out);   // sorted (i, j) rows + freq (reference src/utils.h:14-45)
    void sorted(Context& ctx, SortedTable& out);   // the same on the device, keys = first << 32 | second
};

} // namespace scg
