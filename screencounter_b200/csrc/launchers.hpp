// Kernel launchers shared by the file-level entry points and the resident plans: each picks the run-time specialised
// kernel (spec_handlers.cuh, with its follow-up kernels) when the batch allows and the generic kernel otherwise, and
// records which in Context::kernel_note.  Everything is enqueued on `stream`; nothing synchronises.
#pragma once

#include "api_common.hpp"
#include "matchers.hpp"

namespace scg {

// countDualBarcodes over one batch of pairs (DualBarcodesPairedEnd::process, handlers/DualBarcodesPairedEnd.hpp:353-381)
void launch_dual_pe(Context& ctx, const ReadsDev& r1, const ReadsDev& r2, const DualPEMatcher& m, int32_t* d_counts, int32_t* d_index,
                    cudaStream_t stream);

// countComboBarcodes over one batch (CombinatorialBarcodesSingleEnd::process, handlers/CombinatorialBarcodesSingleEnd.hpp:200-258);
// skip_if_found: the diagnostics pass of the dual single-end design
void launch_combo(Context& ctx, const ReadsDev& reads, const ComboMatcher& m, const ComboSink& sink, const int32_t* skip_if_found,
                  int32_t* out_pairs, cudaStream_t stream);

// countRandomBarcodes over one batch (RandomBarcodeSingleEnd::process, handlers/RandomBarcodeSingleEnd.hpp:122-181);
// the caller has made room in `tab` (CountTable::ensure)
void launch_random(Context& ctx, const ReadsDev& reads, const RandomMatcher& m, CountTable& tab, const uint8_t* odd, OddOutcome* odd_out,
                   unsigned long long* odd_count, int32_t* out_index, cudaStream_t stream);

// countSingleBarcodes over one input on one device (runners_single.cu); counts stay on the device
long long count_single_core(Context& c, FastqReader* reader, const SingleMatcher& m, int nthreads, int32_t* d_counts, TraceSink& sink);

// A sparse result (combinations, random barcodes) of one input or one part of it: a sorted table on the device, or -- random
// barcodes taken from raw read text or longer than 21 bases -- a table rendered on the host.
struct SparseCounts {
    SortedTable table;
    std::unique_ptr<scg_result> rendered;   // set instead of `table`
    std::vector<int32_t> trace;             // per-read trace (want_trace), trace width ints per read
    long long reads = 0;
};

// countDualBarcodesSingleEnd's result over one input or one part of it, left on the device.
struct DualSECounts {
    DeviceBuffer counts;          // nchoices int32
    SortedTable invalid;          // diagnostics: the combinations of reads without a valid pair
    std::vector<int32_t> trace;   // want_trace: one index per read
    long long reads = 0;
};

// The matchers of the sparse designs from the context's cache, built and uploaded on a miss (runners_combo.cu).  Throw the
// reference's validation errors.
std::shared_ptr<ComboMatcher> cached_combo_matcher(Context& c, const char* constant, int strand, const Pool& p1, const Pool& p2, int mismatches,
                                                   int use_first);
struct DualSEMatchers {
    std::shared_ptr<DualSEMatcher> dual;
    std::shared_ptr<ComboMatcher> diagnostics;   // null without diagnostics
};
DualSEMatchers cached_dual_se_matchers(Context& c, const char* constant, const std::vector<Pool>& pools, int nchoices, int strand, int mismatches,
                                       int use_first, bool diagnostics);

// countComboBarcodes / countDualBarcodesSingleEnd / countRandomBarcodes over one reader on one device (runners_combo.cu,
// runners_random.cu): the reader's whole text, or one part of a text cut over several devices.
void count_combo_reader(Context& c, FastqReader* reader, const ComboMatcher& m, int npool1, int npool2, int nthreads, bool want_trace,
                        SparseCounts& out);
void count_dual_se_reader(Context& c, FastqReader* reader, const DualSEMatchers& m, int nchoices, int nthreads, bool want_trace,
                          DualSECounts& out);
void count_random_reader(Context& c, FastqReader* reader, const RandomMatcher& m, int nthreads, SparseCounts& out);

// The same for one input: on the context's first device, or -- split_over_devices, a context of several devices and an input that
// can be cut -- on all of them (runners_multi.cu).  Then the result sits on the first device as if that device had done it all.
void count_combo_file(scg_ctx* ctx, const scg_source* src, const char* constant, int strand, const char* const* pool1, int npool1,
                      const char* const* pool2, int npool2, int mismatches, int use_first, int nthreads, bool want_trace,
                      bool split_over_devices, SparseCounts& out);
void count_random_file(scg_ctx* ctx, const scg_source* src, const char* constant, int strand, int mismatches, int use_first, int nthreads,
                       bool split_over_devices, SparseCounts& out);

// countSingleBarcodes for one input (runners_single.cu): on the context's first device, or cut over all its devices
void count_single_file(scg_ctx* ctx, const scg_source* src, const char* constant, int strand, const char* const* pool, int npool,
                       int mismatches, int use_first, int nthreads, int32_t* counts, int32_t* total, scg_result** trace,
                       bool split_over_devices);

// The single-end designs over SEVERAL devices (runners_multi.cu): the text is cut at record boundaries into one contiguous part
// per device, every device counts its part on its own host thread, and the parts' results are merged on the first device
// (count vectors added, sorted tables merged, traces joined in read order).  false = the input cannot be split (a gzip stream,
// too small, no safe cut, or a part did not parse cleanly): the caller runs the single-device path, which also produces the
// reference's error text where there is one.
bool count_single_multi(scg_ctx* ctx, FastqReader& reader, const char* constant, int strand, const char* const* pool, int npool,
                        int mismatches, bool use_first, int nthreads, int32_t* counts, int32_t* total, scg_result** trace);
bool count_combo_multi(scg_ctx* ctx, FastqReader& reader, const char* constant, int strand, const Pool& p1, const Pool& p2, int mismatches,
                       int use_first, int nthreads, bool want_trace, SparseCounts& out);
bool count_dual_se_multi(scg_ctx* ctx, FastqReader& reader, const char* constant, const std::vector<Pool>& pools, int nchoices, int strand,
                         int mismatches, int use_first, bool diagnostics, int nthreads, bool want_trace, DualSECounts& out);
bool count_random_multi(scg_ctx* ctx, FastqReader& reader, const char* constant, int strand, int mismatches, int use_first, int nthreads,
                        SparseCounts& out);

} // namespace scg
