// countComboBarcodes (reference src/count_combo_barcodes_single.cpp:12-70) and
// countDualBarcodesSingleEnd (src/count_dual_barcodes_single_end.cpp:12-88).
#include <algorithm>
#include <chrono>
#include <cstring>

#include "api_common.hpp"
#include "handlers.cuh"
#include "launchers.hpp"
#include "matchers.hpp"

namespace scg {

static double now_s() {
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

} // namespace scg

using namespace scg;

extern "C" {

} // extern "C"

namespace scg {

std::shared_ptr<ComboMatcher> cached_combo_matcher(Context& c, const char* constant, int strand, const Pool& p1, const Pool& p2, int mismatches,
                                                   int use_first) {
    CacheKey key;
    const int header[5] = { /* combo single */ 3, strand, mismatches, use_first, 0 };
    key.feed(header, sizeof header);
    key.feed(std::string(constant));
    key.feed(p1);
    key.feed(p2);
    return cached_matcher<ComboMatcher>(c, key, [&] {
        auto built = std::make_shared<ComboMatcher>();
        built->prepare(constant, strand, p1, p2, mismatches, use_first != 0, Duplicates::ERROR);
        c.ensure_ready();
        built->upload(c);
        return built;
    });
}

DualSEMatchers cached_dual_se_matchers(Context& c, const char* constant, const std::vector<Pool>& pools, int nchoices, int strand, int mismatches,
                                       int use_first, bool diagnostics) {
    const int npools = (int)pools.size();
    auto key_for = [&](int kind, int dup) {
        CacheKey k;
        const int header[6] = { kind, strand, mismatches, use_first, dup, npools };
        k.feed(header, sizeof header);
        k.feed(std::string(constant));
        for (const auto& p : pools) k.feed(p);
        return k;
    };
    DualSEMatchers m;
    m.dual = cached_matcher<DualSEMatcher>(c, key_for(/* dual single-end */ 4, 0), [&] {
        auto built = std::make_shared<DualSEMatcher>();
        built->prepare(constant, pools, nchoices, strand, mismatches, use_first != 0);
        if (diagnostics && npools != 2) throw Error("expected 2 variable regions in the constant template");
        c.ensure_ready();
        built->upload(c);
        return built;
    });
    if (diagnostics) {
        // DualBarcodesSingleEndWithDiagnostics<_, 2> (reference handlers/DualBarcodesSingleEndWithDiagnostics.hpp:44-58):
        // two variable regions, each pool searched on its own with DuplicateAction::FIRST
        if (npools != 2) throw Error("expected 2 variable regions in the constant template");
        m.diagnostics = cached_matcher<ComboMatcher>(c, key_for(/* combo single */ 3, 1), [&] {
            auto built = std::make_shared<ComboMatcher>();
            built->prepare(constant, strand, pools[0], pools[1], mismatches, use_first != 0, Duplicates::FIRST);
            c.ensure_ready();
            built->upload(c);
            return built;
        });
    }
    return m;
}

// countComboBarcodes over one reader: the tally (dense matrix or device hash) as a sorted table (first << 32 | second) on the device
void count_combo_reader(Context& c, FastqReader* reader, const ComboMatcher& m, int npool1, int npool2, int nthreads, bool want_trace,
                        SparseCounts& out) {
    c.ensure_ready();
    ComboTally tally;
    tally.init(c, npool1, npool2);
    TraceSink trace;
    trace.enabled = want_trace;
    trace.width = 2;

    ReadPipeline pipe(c, reader, nullptr, nthreads, false);
    ReadPipeline::Batch b;
    long long nreads = 0;
    while (pipe.next(b)) {
        trace.prepare(b.n, false);
        launch_combo(c, b.reads1, m, tally.sink(c, b.n), nullptr, trace.enabled ? trace.d_index.as<int32_t>() : nullptr, c.stream);
        pipe.submitted(b);
        trace.collect(c, b.n, false);
        nreads += b.n;
    }
    tally.sorted(c, out.table);
    out.trace.swap(trace.index);
    out.reads = nreads;
}

void count_combo_file(scg_ctx* ctx, const scg_source* src, const char* constant, int strand, const char* const* pool1, int npool1,
                      const char* const* pool2, int npool2, int mismatches, int use_first, int nthreads, bool want_trace,
                      bool split_over_devices, SparseCounts& out) {
    Context& c = ctx->impl;
    const double t_start = now_s();
    c.timing = Timing();
    Source source(src);
    Pool p1(pool1, npool1), p2(pool2, npool2);
    const std::shared_ptr<ComboMatcher> m = cached_combo_matcher(c, constant, strand, p1, p2, mismatches, use_first);
    c.ensure_ready();
    if (!(split_over_devices && !ctx->peers.empty() &&
          count_combo_multi(ctx, *source.reader, constant, strand, p1, p2, mismatches, use_first, nthreads, want_trace, out))) {
        count_combo_reader(c, source.reader.get(), *m, npool1, npool2, nthreads, want_trace, out);
        c.timing.parse_s = source.reader->parse_seconds();
    }
    c.timing.total_s = now_s() - t_start;
    c.finish_timing();
}

// countDualBarcodesSingleEnd over one reader: counts of the valid pairs and, with diagnostics, the tally of the others
void count_dual_se_reader(Context& c, FastqReader* reader, const DualSEMatchers& matchers, int nchoices, int nthreads, bool want_trace,
                          DualSECounts& out) {
    const DualSEMatcher& m = *matchers.dual;
    const bool diagnostics = matchers.diagnostics != nullptr;
    c.ensure_ready();
    ComboTally tally;
    if (diagnostics) tally.init(c, nchoices, nchoices);
    DeviceBuffer d_index;
    out.counts.alloc((size_t)std::max(nchoices, 1) * sizeof(int32_t), true);
    const bool need_index = diagnostics || want_trace;

    ReadPipeline pipe(c, reader, nullptr, nthreads, false);
    ReadPipeline::Batch b;
    long long nreads = 0;
    while (pipe.next(b)) {
        if (need_index) d_index.reserve((size_t)b.n * sizeof(int32_t));
        const long long ntiles = (b.n + TILE - 1) / TILE;
        const int grid = c.grid_for(ntiles);
        dispatch_cb(m.params.spec.cbits, [&](auto CB) {
            dispatch_kw(m.params.kw, [&](auto KW) {
                dual_se_kernel<decltype(CB)::value, decltype(KW)::value><<<grid, 128, 0, c.stream>>>(
                    b.reads1, m.params, out.counts.as<int32_t>(), need_index ? d_index.as<int32_t>() : nullptr);
            });
        });
        SCG_CUDA_CHECK(cudaGetLastError());
        ++c.launches;
        ++c.timing.launches;
        c.kernel_note = "generic dual_se_kernel (all variable regions concatenated, one any-mismatch search)";
        if (diagnostics) {
            // only reads without a valid pair are tabulated (:99-104)
            launch_combo(c, b.reads1, *matchers.diagnostics, tally.sink(c, b.n), d_index.as<int32_t>(), nullptr, c.stream);
            c.kernel_note = "generic dual_se_kernel; diagnostics: " + c.kernel_note;
        }
        pipe.submitted(b);
        if (want_trace) {
            const size_t at = out.trace.size();
            out.trace.resize(at + (size_t)b.n);
            SCG_CUDA_CHECK(cudaMemcpyAsync(out.trace.data() + at, d_index.ptr, (size_t)b.n * sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
            SCG_CUDA_CHECK(cudaStreamSynchronize(c.stream));
        }
        nreads += b.n;
    }
    if (diagnostics) tally.sorted(c, out.invalid);
    out.reads = nreads;
}

} // namespace scg

extern "C" {

int scg_count_combo_single(scg_ctx* ctx, const scg_source* src, const char* constant, int strand, const char* const* pool1, int npool1,
                           const char* const* pool2, int npool2, int mismatches, int use_first, int nthreads, int want_trace,
                           scg_result** table, int32_t* total) {
    return guarded(ctx, [&] {
        SparseCounts counts;
        count_combo_file(ctx, src, constant, strand, pool1, npool1, pool2, npool2, mismatches, use_first, nthreads, want_trace != 0, true, counts);
        std::unique_ptr<scg_result> r(new scg_result);
        device_table_result(ctx->impl, counts.table, *r);
        if (want_trace) {
            r->trace_width = 2;
            r->trace_index.swap(counts.trace);
        }
        *table = r.release();
        *total = (int32_t)counts.reads;
    });
}

int scg_count_dual_single_end(scg_ctx* ctx, const scg_source* src, const char* constant, const char* const* pools_flat, int npools,
                              int nchoices, int strand, int mismatches, int use_first, int diagnostics, int nthreads, int want_trace,
                              int32_t* counts, int32_t* total, scg_result** table) {
    return guarded(ctx, [&] {
        Context& c = ctx->impl;
        const double t_start = now_s();
        c.timing = Timing();
        Source source(src);
        std::vector<Pool> pools;
        for (int p = 0; p < npools; ++p) pools.emplace_back(pools_flat + (size_t)p * nchoices, nchoices);
        const DualSEMatchers m = cached_dual_se_matchers(c, constant, pools, nchoices, strand, mismatches, use_first, diagnostics != 0);
        c.ensure_ready();
        DualSECounts out;
        if (!(!ctx->peers.empty() && count_dual_se_multi(ctx, *source.reader, constant, pools, nchoices, strand, mismatches, use_first,
                                                         diagnostics != 0, nthreads, want_trace != 0, out))) {
            count_dual_se_reader(c, source.reader.get(), m, nchoices, nthreads, want_trace != 0, out);
            c.timing.parse_s = source.reader->parse_seconds();
        }
        SCG_CUDA_CHECK(cudaMemcpyAsync(counts, out.counts.ptr, (size_t)nchoices * sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
        SCG_CUDA_CHECK(cudaStreamSynchronize(c.stream));
        *total = (int32_t)out.reads;
        if (table) {
            std::unique_ptr<scg_result> r(new scg_result);
            if (diagnostics) device_table_result(c, out.invalid, *r);
            if (want_trace) {
                r->trace_width = 1;
                r->trace_index.swap(out.trace);
            }
            *table = r.release();
        }
        c.timing.total_s = now_s() - t_start;
        c.finish_timing();
    });
}

} // extern "C"
