// Several devices behind ONE context, and several files behind ONE call.
//
// The reference parallelises inside a call (a thread pool over blocks of reads, inst/include/kaori/process_data.hpp:131-177)
// and across files in R (bplapply over files + cbind / union of the per-file results: R/countSingleBarcodes.R:112-126,
// R/combineComboCounts.R:31-57, R/countRandomBarcodes.R:84-105).  Here:
//   * scg_ctx_create_multi binds one context to several GPUs.  The single-end entry points (scg_count_single,
//     scg_count_combo_single, scg_count_dual_single_end, scg_count_random) on such a context cut the text of ONE file at record
//     boundaries into one contiguous part per device (every read is counted on its own, so the parts' results add up to the
//     file's); every device reads, packs and counts its part on its own host thread and stream, and the parts' results are
//     merged on the first device: count vectors added (peer copies + one kernel), sorted tables merged (merge kernels),
//     per-read traces joined in read order.
//   * scg_count_{single,combo,random}_many take a list of files, deal them to the devices (one file per device at a time; the
//     library tables stay resident in every device's matcher cache) and return the count matrix the R wrappers assemble:
//     dense columns for single barcodes; for combinations and random barcodes the sorted union of the files' keys, built on
//     the device from the files' sorted tables (merge kernels), and one column per file scattered by binary search.
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <map>
#include <thread>

#include "api_common.hpp"
#include "bgzf.hpp"
#include "ingest.hpp"
#include "launchers.hpp"
#include "matchers.hpp"

namespace scg {

namespace {

double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

__global__ void add_counts_kernel(int32_t* __restrict__ into, const int32_t* __restrict__ from, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) into[i] += from[i];
}

std::vector<scg_ctx*> device_contexts(scg_ctx* ctx) {
    std::vector<scg_ctx*> all{ ctx };
    for (auto& p : ctx->peers) all.push_back(p.get());
    return all;
}

size_t split_threshold() {
    // below this many bytes of text per device a file is not worth cutting up (SCG_MULTI_MIN_BYTES overrides, for tests)
    if (const char* env = std::getenv("SCG_MULTI_MIN_BYTES")) return (size_t)std::strtoull(env, nullptr, 10);
    return (size_t)8 << 20;
}

// Stage timings of a call that ran on several devices: the slowest device's stages, the sums of what was moved and launched.
void combine_timing(Context& into, const std::vector<scg_ctx*>& all, double total_s) {
    Timing t;
    t.reader = all[0]->impl.timing.reader;
    for (scg_ctx* c : all) {
        const Timing& s = c->impl.timing;
        t.parse_s = std::max(t.parse_s, s.parse_s);
        t.pack_s = std::max(t.pack_s, s.pack_s);
        t.h2d_s = std::max(t.h2d_s, s.h2d_s);
        t.device_s = std::max(t.device_s, s.device_s);
        t.setup_s = std::max(t.setup_s, s.setup_s);
        t.harvest_s = std::max(t.harvest_s, s.harvest_s);
        t.reads += s.reads;
        t.bytes_h2d += s.bytes_h2d;
        t.launches += s.launches;
    }
    t.total_s = total_s;
    into.timing = t;
    into.kernel_note += "; " + std::to_string(all.size()) + " devices";
    into.finish_timing();
}

// Where the text of one input is cut: part d is the text [at[d], at[d + 1]).
struct TextCuts {
    const char* text = nullptr;         // raw text in memory, or
    const BgzfIndex* image = nullptr;   // a block-gzip image, cut in the coordinates of its text
    std::vector<size_t> at;
};

// Cuts for `ndev` parts, each at a likely record start; false = the input cannot be cut (a plain gzip stream, too little text
// per device, no record start found near a cut).
bool plan_cuts(FastqReader& reader, int ndev, TextCuts& cuts) {
    size_t size = 0;
    const bool raw = reader.memory_text(&cuts.text, &size);
    if (!raw) {
        // a block-gzip file is cut the same way, in the coordinates of its TEXT: a part begins inside some member, at a record
        // start guessed on that member's (and the next one's) text, inflated here on the host; a plain gzip stream cannot be cut
        size_t b = 0;
        cuts.text = nullptr;
        if (!device_inflate_enabled() || !reader.bgzf_image(&cuts.image, &b, &size) || b != 0) return false;
    }
    if (size < split_threshold() * (size_t)ndev) return false;
    const BgzfIndex* image = cuts.image;
    cuts.at.assign(1, 0);
    std::vector<char> around;
    for (int k = 1; k < ndev; ++k) {
        const size_t target = size / ndev * k;
        size_t g = (size_t)-1;
        if (raw) {
            g = guess_fastq_record_start(cuts.text, size, target);
        } else {
            const size_t blk = image->block_of(target);
            if (blk >= image->blocks.size()) return false;
            const size_t n0 = image->blocks[blk].isize, n1 = blk + 1 < image->blocks.size() ? image->blocks[blk + 1].isize : 0;
            around.resize(n0 + n1 + 1);
            if (!bgzf_inflate_block(*image, blk, around.data()) || (n1 && !bgzf_inflate_block(*image, blk + 1, around.data() + n0))) return false;
            const size_t local = guess_fastq_record_start(around.data(), n0 + n1, target - image->text_off[blk]);
            if (local != (size_t)-1) g = image->text_off[blk] + local;
        }
        if (g == (size_t)-1 || g <= cuts.at.back() || g >= size) return false;
        cuts.at.push_back(g);
    }
    cuts.at.push_back(size);
    return true;
}

// Runs job(device context, part reader, d) for every part d, one host thread per device.  false = some part threw: nothing of
// the parts may be used.  Otherwise the call's timing on the first device is that of the parts (combine_timing).
template <class Job>
bool run_parts(scg_ctx* ctx, const TextCuts& cuts, Job&& job) {
    const std::vector<scg_ctx*> all = device_contexts(ctx);
    const int ndev = (int)all.size();
    std::vector<char> failed(ndev, 0);
    const double t_start = now_s();
    auto work = [&](int d) {
        Context& c = all[d]->impl;
        try {
            c.timing = Timing();
            c.ensure_ready();
            // A part is a FASTQ text of its own.  Part 0 starts at a record boundary; a part that parses cleanly to its very
            // end proves that the next cut is one too (the parser never looks behind a record's start), so by induction the
            // parts are exactly the records of the whole file.  Anything else throws here and the caller starts over on one
            // device, which also raises the reference's error with the right line number.
            const size_t b = cuts.at[d], e = cuts.at[d + 1];
            FastqReader sub(nullptr, cuts.text ? cuts.text + b : reinterpret_cast<const char*>(cuts.image->image),
                            cuts.text ? e - b : cuts.image->image_size);
            if (!cuts.text) sub.set_text_range(b, e);
            job(c, sub, d);
            SCG_CUDA_CHECK(cudaStreamSynchronize(c.stream));
            c.timing.parse_s = sub.parse_seconds();
        } catch (const std::exception&) {
            failed[d] = 1;
            cudaGetLastError();
        }
    };
    {
        std::vector<std::thread> threads;
        for (int d = 1; d < ndev; ++d) threads.emplace_back(work, d);
        work(0);
        for (auto& t : threads) t.join();
    }
    for (char f : failed) {
        if (f) return false;
    }
    combine_timing(ctx->impl, all, now_s() - t_start);
    return true;
}

// counts[d] (n int32 on device d) added up into counts[0] on the first device
void add_up_counts(const std::vector<scg_ctx*>& all, const std::vector<int32_t*>& counts, int n) {
    Context& c0 = all[0]->impl;
    c0.ensure_ready();
    if (n == 0) return;
    DeviceBuffer landing;
    landing.alloc((size_t)n * sizeof(int32_t), false);
    for (size_t d = 1; d < all.size(); ++d) {
        SCG_CUDA_CHECK(cudaMemcpyPeerAsync(landing.ptr, c0.device, counts[d], all[d]->impl.device, (size_t)n * sizeof(int32_t), c0.stream));
        add_counts_kernel<<<(n + 255) / 256, 256, 0, c0.stream>>>(counts[0], landing.as<int32_t>(), n);
        SCG_CUDA_CHECK(cudaGetLastError());
        ++c0.launches;
        ++c0.timing.launches;
    }
}

// A table that lives on another device, brought to the context's device.
void bring_home(Context& c0, SortedTable& t) {
    if (t.rows == 0 || t.keys.device == c0.device) return;
    SortedTable here;
    here.rows = t.rows;
    here.key_len = t.key_len;
    const size_t key_bytes = t.rows * 8 * (size_t)t.words();
    here.keys.alloc(key_bytes, false);
    here.counts.alloc(t.rows * sizeof(uint32_t), false);
    SCG_CUDA_CHECK(cudaMemcpyPeerAsync(here.keys.ptr, c0.device, t.keys.ptr, t.keys.device, key_bytes, c0.stream));
    SCG_CUDA_CHECK(cudaMemcpyPeerAsync(here.counts.ptr, c0.device, t.counts.ptr, t.counts.device, t.rows * sizeof(uint32_t), c0.stream));
    SCG_CUDA_CHECK(cudaStreamSynchronize(c0.stream));
    t = std::move(here);
}

// The union of sorted device tables on the first device: keys ascending, the counts of equal keys added.  Every table is
// brought to the first device on the way; a single table is its own union (moved into u).
void union_on_device(Context& c0, std::vector<SortedTable>& tables, SortedTable& u) {
    for (size_t f = 0; f < tables.size(); ++f) {
        bring_home(c0, tables[f]);
        if (f == 0) continue;
        SortedTable merged;
        merge_sorted_tables(c0, f == 1 ? tables[0] : u, tables[f], merged);
        u = std::move(merged);
    }
    if (tables.size() == 1) u = std::move(tables[0]);
}

// The union made on the host, for tables of which some could only be rendered there (random barcodes read from raw text):
// key -> its count in every table.  std::map iterates strings in byte order = sort(union) of R for
// ACGTN text; combinations are keyed big-endian, so that byte order is (first, second) order.
using HostUnion = std::map<std::string, std::vector<int32_t>>;
HostUnion union_on_host(Context& c0, std::vector<SortedTable>& tables, std::vector<std::unique_ptr<scg_result>>& rendered, int width,
                        bool strings) {
    HostUnion rows;
    const int ntables = (int)tables.size();
    const size_t unit = strings ? (size_t)width : (size_t)width * sizeof(int32_t);
    for (int f = 0; f < ntables; ++f) {
        std::unique_ptr<scg_result> mine;
        const scg_result* r = rendered[f].get();
        if (!r) {
            mine.reset(new scg_result);
            bring_home(c0, tables[f]);
            device_table_result(c0, tables[f], *mine);
            r = mine.get();
        }
        const size_t n = r->rows();
        std::vector<char> keys(std::max<size_t>(n * unit, 1));
        std::vector<int32_t> freq(std::max<size_t>(n, 1));
        if (scg_result_copy_table(r, strings ? nullptr : reinterpret_cast<int32_t*>(keys.data()), strings ? keys.data() : nullptr, freq.data()) != 0) {
            throw Error("could not read a table back");
        }
        for (size_t i = 0; i < n; ++i) {
            std::string k(keys.data() + i * unit, unit);
            if (!strings) {
                for (int w = 0; w < width; ++w) {
                    uint32_t v;
                    std::memcpy(&v, keys.data() + i * unit + (size_t)w * 4, 4);
                    v = __builtin_bswap32(v);
                    std::memcpy(&k[(size_t)w * 4], &v, 4);
                }
            }
            auto& row = rows[k];
            if (row.empty()) row.assign(ntables, 0);
            row[f] += freq[i];
        }
    }
    return rows;
}

// A host union as a result: its rows in key order with their summed counts and, with `columns`, one column of counts per table.
void host_union_result(const HostUnion& rows, int ntables, int width, bool strings, bool columns, scg_result& out) {
    const size_t nrows = rows.size();
    out.width = width;
    if (columns) out.matrix.assign(nrows * (size_t)ntables, 0);
    size_t at = 0;
    for (const auto& kv : rows) {
        int32_t sum = 0;
        for (int f = 0; f < ntables; ++f) {
            if (columns) out.matrix[(size_t)f * nrows + at] = kv.second[f];
            sum += kv.second[f];
        }
        out.freq.push_back(sum);
        if (strings) {
            out.strings.insert(out.strings.end(), kv.first.begin(), kv.first.end());
        } else {
            for (int w = 0; w < width; ++w) {
                uint32_t v;
                std::memcpy(&v, kv.first.data() + (size_t)w * 4, 4);
                out.keys.push_back((int32_t)__builtin_bswap32(v));
            }
        }
        ++at;
    }
}

// The parts' sparse results as the result of the whole input, on the first device: what one device would have left there.
void unite_parts(scg_ctx* ctx, std::vector<SparseCounts>& parts, bool strings, SparseCounts& out) {
    Context& c0 = ctx->impl;
    const double t0 = now_s();
    c0.ensure_ready();
    std::vector<SortedTable> tables;
    std::vector<std::unique_ptr<scg_result>> rendered;
    bool host_union = false;
    int width = strings ? 0 : 2;
    out.reads = 0;
    out.trace.clear();
    for (SparseCounts& p : parts) {
        out.reads += p.reads;
        out.trace.insert(out.trace.end(), p.trace.begin(), p.trace.end());
        if (strings) width = std::max(width, p.rendered ? p.rendered->width : p.table.key_len);
        host_union = host_union || p.rendered;
        tables.push_back(std::move(p.table));
        rendered.push_back(std::move(p.rendered));
    }
    if (!host_union) {
        union_on_device(c0, tables, out.table);
    } else {
        out.rendered.reset(new scg_result);
        host_union_result(union_on_host(c0, tables, rendered, width, strings), (int)tables.size(), width, strings, false, *out.rendered);
    }
    c0.timing.merge_s = now_s() - t0;
}

} // namespace

bool count_single_multi(scg_ctx* ctx, FastqReader& reader, const char* constant, int strand, const char* const* pool, int npool,
                        int mismatches, bool use_first, int nthreads, int32_t* counts, int32_t* total, scg_result** trace) {
    const std::vector<scg_ctx*> all = device_contexts(ctx);
    const int ndev = (int)all.size();
    TextCuts cuts;
    if (!plan_cuts(reader, ndev, cuts)) return false;
    struct Part {
        long long reads = 0;
        TraceSink sink;
        DeviceBuffer d_counts;
    };
    std::vector<Part> parts(ndev);
    const bool ok = run_parts(ctx, cuts, [&](Context& c, FastqReader& sub, int d) {
        Part& part = parts[d];
        const double t0 = now_s();
        const std::shared_ptr<SingleMatcher> m = cached_single_matcher(c, constant, strand, pool, npool, mismatches, use_first);
        c.timing.setup_s = now_s() - t0;
        part.d_counts.alloc((size_t)std::max(npool, 1) * sizeof(int32_t), true);
        part.sink.enabled = trace != nullptr;
        part.reads = count_single_core(c, &sub, *m, nthreads, part.d_counts.as<int32_t>(), part.sink);
    });
    if (!ok) return false;

    // the parts' count vectors, added up on the first device
    Context& c0 = ctx->impl;
    const double t_merge = now_s();
    std::vector<int32_t*> d_counts;
    long long nreads = 0;
    for (Part& p : parts) {
        d_counts.push_back(p.d_counts.as<int32_t>());
        nreads += p.reads;
    }
    add_up_counts(all, d_counts, npool);
    SCG_CUDA_CHECK(cudaMemcpyAsync(counts, parts[0].d_counts.ptr, (size_t)npool * sizeof(int32_t), cudaMemcpyDeviceToHost, c0.stream));
    SCG_CUDA_CHECK(cudaStreamSynchronize(c0.stream));
    c0.timing.merge_s = now_s() - t_merge;
    *total = (int32_t)nreads;
    if (trace) {
        auto* r = new scg_result;
        r->trace_width = 1;
        for (Part& p : parts) {
            r->trace_index.insert(r->trace_index.end(), p.sink.index.begin(), p.sink.index.end());
            r->trace_info.insert(r->trace_info.end(), p.sink.info.begin(), p.sink.info.end());
        }
        *trace = r;
    }
    return true;
}

bool count_combo_multi(scg_ctx* ctx, FastqReader& reader, const char* constant, int strand, const Pool& p1, const Pool& p2, int mismatches,
                       int use_first, int nthreads, bool want_trace, SparseCounts& out) {
    TextCuts cuts;
    if (!plan_cuts(reader, (int)device_contexts(ctx).size(), cuts)) return false;
    std::vector<SparseCounts> parts(device_contexts(ctx).size());
    const bool ok = run_parts(ctx, cuts, [&](Context& c, FastqReader& sub, int d) {
        const double t0 = now_s();
        const std::shared_ptr<ComboMatcher> m = cached_combo_matcher(c, constant, strand, p1, p2, mismatches, use_first);
        c.timing.setup_s = now_s() - t0;
        count_combo_reader(c, &sub, *m, (int)p1.seqs.size(), (int)p2.seqs.size(), nthreads, want_trace, parts[d]);
    });
    if (!ok) return false;
    unite_parts(ctx, parts, false, out);
    return true;
}

bool count_dual_se_multi(scg_ctx* ctx, FastqReader& reader, const char* constant, const std::vector<Pool>& pools, int nchoices, int strand,
                         int mismatches, int use_first, bool diagnostics, int nthreads, bool want_trace, DualSECounts& out) {
    const std::vector<scg_ctx*> all = device_contexts(ctx);
    TextCuts cuts;
    if (!plan_cuts(reader, (int)all.size(), cuts)) return false;
    std::vector<DualSECounts> parts(all.size());
    const bool ok = run_parts(ctx, cuts, [&](Context& c, FastqReader& sub, int d) {
        const double t0 = now_s();
        const DualSEMatchers m = cached_dual_se_matchers(c, constant, pools, nchoices, strand, mismatches, use_first, diagnostics);
        c.timing.setup_s = now_s() - t0;
        count_dual_se_reader(c, &sub, m, nchoices, nthreads, want_trace, parts[d]);
    });
    if (!ok) return false;

    Context& c0 = ctx->impl;
    const double t_merge = now_s();
    std::vector<int32_t*> d_counts;
    std::vector<SortedTable> invalid;
    out.reads = 0;
    out.trace.clear();
    for (DualSECounts& p : parts) {
        d_counts.push_back(p.counts.as<int32_t>());
        out.reads += p.reads;
        out.trace.insert(out.trace.end(), p.trace.begin(), p.trace.end());
        invalid.push_back(std::move(p.invalid));
    }
    add_up_counts(all, d_counts, nchoices);
    if (diagnostics) union_on_device(c0, invalid, out.invalid);
    SCG_CUDA_CHECK(cudaStreamSynchronize(c0.stream));
    out.counts = std::move(parts[0].counts);
    c0.timing.merge_s = now_s() - t_merge;
    return true;
}

bool count_random_multi(scg_ctx* ctx, FastqReader& reader, const char* constant, int strand, int mismatches, int use_first, int nthreads,
                        SparseCounts& out) {
    TextCuts cuts;
    if (!plan_cuts(reader, (int)device_contexts(ctx).size(), cuts)) return false;
    std::vector<SparseCounts> parts(device_contexts(ctx).size());
    const bool ok = run_parts(ctx, cuts, [&](Context& c, FastqReader& sub, int d) {
        RandomMatcher m;
        m.prepare(constant, strand, mismatches, use_first != 0);
        count_random_reader(c, &sub, m, nthreads, parts[d]);
    });
    if (!ok) return false;
    unite_parts(ctx, parts, true, out);
    return true;
}

namespace {

// Runs job(device context, file) for every file, the files dealt to the devices in turn, one host thread per device.
// The first failing file (lowest index) gives the call's error.
template <class Job>
void deal_files(scg_ctx* ctx, int nfiles, Job&& job) {
    const std::vector<scg_ctx*> all = device_contexts(ctx);
    const int ndev = (int)std::min<size_t>(all.size(), (size_t)std::max(nfiles, 1));
    std::vector<std::string> errors(nfiles);
    std::vector<char> failed(nfiles, 0);
    auto work = [&](int d) {
        for (int f = d; f < nfiles; f += ndev) {
            try {
                job(all[d], f);
            } catch (const std::exception& e) {
                failed[f] = 1;
                errors[f] = e.what();
                cudaGetLastError();
            }
        }
    };
    std::vector<std::thread> threads;
    for (int d = 1; d < ndev; ++d) threads.emplace_back(work, d);
    work(0);
    for (auto& t : threads) t.join();
    for (int f = 0; f < nfiles; ++f) {
        if (failed[f]) throw Error(errors[f]);
    }
}

void status_or_throw(scg_ctx* c, int status) {
    if (status != 0) throw Error(c->impl.last_error);
}

// The files' results as one matrix over the union of their keys.  tables[f] is file f's sorted device table, or empty with
// rendered[f] set where a file's result could only be had on the host: then the union is made on the host.
void unite(scg_ctx* ctx, std::vector<SortedTable>& tables, std::vector<std::unique_ptr<scg_result>>& rendered, int width, bool strings,
           scg_result& out) {
    Context& c0 = ctx->impl;
    c0.ensure_ready();
    const int nfiles = (int)tables.size();
    out.width = width;
    out.columns = nfiles;
    bool host_union = false;
    for (int f = 0; f < nfiles; ++f) host_union = host_union || rendered[f];
    if (!host_union) {
        SortedTable u;
        union_on_device(c0, tables, u);
        out.d_matrix.alloc(std::max<size_t>(u.rows * (size_t)nfiles, 1) * sizeof(int32_t), true);
        for (int f = 0; f < nfiles; ++f) scatter_table_column(c0, u, nfiles == 1 ? u : tables[f], out.d_matrix.as<int32_t>() + (size_t)f * u.rows);
        device_table_result(c0, u, out);
        return;
    }
    host_union_result(union_on_host(c0, tables, rendered, width, strings), nfiles, width, strings, true, out);
}

} // namespace

} // namespace scg

using namespace scg;

extern "C" {

int scg_ctx_create_multi(scg_ctx** out, const int* devices, int n_devices) {
    try {
        if (!out || !devices || n_devices < 1) throw Error("scg_ctx_create_multi needs at least one device");
        std::unique_ptr<scg_ctx> ctx(new scg_ctx(devices[0]));
        for (int d = 1; d < n_devices; ++d) ctx->peers.emplace_back(new scg_ctx(devices[d]));
        *out = ctx.release();
        return 0;
    } catch (const std::exception& e) {
        creation_error() = e.what();
        return 1;
    }
}

int scg_ctx_devices(const scg_ctx* ctx) { return ctx ? 1 + (int)ctx->peers.size() : 0; }

int scg_result_columns(const scg_result* r) { return r ? r->columns : 0; }

int scg_result_copy_matrix(const scg_result* r, int32_t* matrix) {
    if (!r || !matrix) return 1;
    const size_t cells = r->rows() * (size_t)r->columns;
    if (cells == 0) return 0;
    if (r->on_device) {
        int current = -1;
        cudaGetDevice(&current);
        bool ok = cudaSetDevice(r->device) == cudaSuccess;
        ok = ok && r->d_matrix.ptr && cudaMemcpy(matrix, r->d_matrix.ptr, cells * sizeof(int32_t), cudaMemcpyDeviceToHost) == cudaSuccess;
        if (current >= 0 && current != r->device) cudaSetDevice(current);
        if (!ok) {
            cudaGetLastError();
            return 1;
        }
        return 0;
    }
    if (r->matrix.size() != cells) return 1;
    std::memcpy(matrix, r->matrix.data(), cells * sizeof(int32_t));
    return 0;
}

// matrixOfSingleBarcodes (reference R/countSingleBarcodes.R:112-126): one column of counts per file.
int scg_count_single_many(scg_ctx* ctx, const scg_source* sources, int nfiles, const char* constant, int strand, const char* const* pool,
                          int npool, int mismatches, int use_first, int nthreads, int32_t* matrix, int32_t* totals) {
    return guarded(ctx, [&] {
        if (nfiles < 0 || (nfiles && (!sources || !totals))) throw Error("invalid list of files");
        const double t_start = now_s();
        const std::vector<scg_ctx*> all = device_contexts(ctx);
        if (nfiles < (int)all.size()) {
            // fewer files than devices: one file at a time, each cut over all the devices
            for (int f = 0; f < nfiles; ++f) {
                status_or_throw(ctx, scg_count_single(ctx, &sources[f], constant, strand, pool, npool, mismatches, use_first, nthreads,
                                                      matrix + (size_t)f * npool, &totals[f], nullptr));
            }
            return;
        }
        // one file per device at a time, each on that device alone (its tables are cached in that device's context)
        deal_files(ctx, nfiles, [&](scg_ctx* dc, int f) {
            count_single_file(dc, &sources[f], constant, strand, pool, npool, mismatches, use_first, nthreads, matrix + (size_t)f * npool,
                              &totals[f], nullptr, false);
        });
        if (all.size() > 1) combine_timing(ctx->impl, all, now_s() - t_start);
    });
}

// countComboBarcodes per file + combineComboCounts (reference R/combineComboCounts.R:31-57): the sorted union of the files'
// combinations and one column of counts per file.
int scg_count_combo_many(scg_ctx* ctx, const scg_source* sources, int nfiles, const char* constant, int strand, const char* const* pool1,
                         int npool1, const char* const* pool2, int npool2, int mismatches, int use_first, int nthreads, scg_result** table,
                         int32_t* totals) {
    return guarded(ctx, [&] {
        if (nfiles < 1 || !sources || !totals || !table) throw Error("invalid list of files");
        std::vector<SortedTable> tables(nfiles);
        std::vector<std::unique_ptr<scg_result>> rendered(nfiles);
        deal_files(ctx, nfiles, [&](scg_ctx* dc, int f) {
            SparseCounts counts;
            count_combo_file(dc, &sources[f], constant, strand, pool1, npool1, pool2, npool2, mismatches, use_first, nthreads, false, false, counts);
            tables[f] = std::move(counts.table);
            totals[f] = (int32_t)counts.reads;
        });
        std::unique_ptr<scg_result> out(new scg_result);
        unite(ctx, tables, rendered, 2, false, *out);
        *table = out.release();
    });
}

// matrixOfRandomBarcodes (reference R/countRandomBarcodes.R:84-105): sort(union of the files' barcodes), one column per file.
int scg_count_random_many(scg_ctx* ctx, const scg_source* sources, int nfiles, const char* constant, int strand, int mismatches,
                          int use_first, int nthreads, scg_result** table, int32_t* totals) {
    return guarded(ctx, [&] {
        if (nfiles < 1 || !sources || !totals || !table) throw Error("invalid list of files");
        std::vector<SortedTable> tables(nfiles);
        std::vector<std::unique_ptr<scg_result>> rendered(nfiles);
        int width = 0;
        deal_files(ctx, nfiles, [&](scg_ctx* dc, int f) {
            SparseCounts counts;
            count_random_file(dc, &sources[f], constant, strand, mismatches, use_first, nthreads, false, counts);
            tables[f] = std::move(counts.table);
            rendered[f] = std::move(counts.rendered);
            totals[f] = (int32_t)counts.reads;
        });
        for (int f = 0; f < nfiles; ++f) width = std::max(width, rendered[f] ? rendered[f]->width : tables[f].key_len);
        std::unique_ptr<scg_result> out(new scg_result);
        unite(ctx, tables, rendered, width, true, *out);
        *table = out.release();
    });
}

} // extern "C"
