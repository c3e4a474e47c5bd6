// countSingleBarcodes / matchBarcodes / the resident single-barcode plan, plus the context and
// result plumbing of the C ABI.
#include <algorithm>
#include <chrono>
#include <cstring>
#include <exception>
#include <thread>

#include "api_common.hpp"
#include "hostpool.hpp"
#include "handlers.cuh"
#include "jit.hpp"
#include "launchers.hpp"
#include "matchers.hpp"

namespace scg {

std::string& creation_error() {
    static thread_local std::string msg;
    return msg;
}

static double now_s() {
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

Pool::Pool(const char* const* p, int n) {
    seqs.reserve(n);
    size_t size = 0;
    for (int i = 0; i < n; ++i) {
        size_t cur = std::strlen(p[i]);
        if (i == 0) {
            size = cur;
        } else if (cur != size) {
            throw Error("variable regions should all have the same length (" + std::to_string(size) + ")");
        }
        seqs.emplace_back(p[i], cur);
    }
    length = (int)size;
}

std::vector<std::string> Pool::reverse_complemented() const {
    std::vector<std::string> out;
    out.reserve(seqs.size());
    for (const auto& s : seqs) out.push_back(reverse_complement_iupac(s));
    return out;
}

Source::Source(const scg_source* s) {
    if (!s) throw Error("null FASTQ source");
    reader.reset(new FastqReader(s->path, s->data, s->size));
}

void TraceSink::prepare(long long n, bool want_info) {
    if (!enabled) return;
    d_index.reserve((size_t)std::max<long long>(n, 1) * width * sizeof(int32_t));
    if (want_info) d_info.reserve((size_t)std::max<long long>(n, 1) * sizeof(uint32_t));
}

void TraceSink::collect(Context& ctx, long long n, bool want_info) {
    if (!enabled) return;
    size_t at = index.size();
    index.resize(at + (size_t)n * width);
    SCG_CUDA_CHECK(cudaMemcpyAsync(index.data() + at, d_index.ptr, (size_t)n * width * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx.stream));
    if (want_info) {
        size_t ai = info.size();
        info.resize(ai + (size_t)n);
        SCG_CUDA_CHECK(cudaMemcpyAsync(info.data() + ai, d_info.ptr, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx.stream));
    }
    SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
}

// SimpleSingleMatch constructor (reference inst/include/kaori/SimpleSingleMatch.hpp:61-97).
void SingleMatcher::prepare(const std::string& constant, int strand, const Pool& pool, int mismatches, bool use_first, Duplicates dup) {
    tmpl = TemplateSpec(constant, strand);
    if (tmpl.fwd_regions.size() != 1) throw Error("expected one variable region in the constant template");
    const int var_length = tmpl.fwd_regions[0].end - tmpl.fwd_regions[0].start;
    if (var_length != pool.length) {
        throw Error("length of barcode_pool sequences (" + std::to_string(pool.length) + ") should be the same as the barcode_pool region (" +
                    std::to_string(var_length) + ")");
    }
    npool = (int)pool.seqs.size();
    LibraryOptions opt;
    opt.max_mismatches = mismatches;
    opt.duplicates = dup;
    std::memset(&params, 0, sizeof params);
    // the two strands' tables are independent: build them side by side (errors surface in the reference's order,
    // forward library first, SimpleSingleMatch.hpp:88-96)
    std::exception_ptr err_f, err_r;
    std::thread side;
    if (tmpl.fwd && tmpl.rev) {
        side = std::thread([&] {
            try {
                lib_r.host = Library(pool.reverse_complemented(), pool.length, opt);
            } catch (...) {
                err_r = std::current_exception();
            }
        });
    }
    try {
        if (tmpl.fwd) lib_f.host = Library(pool.seqs, pool.length, opt);
    } catch (...) {
        err_f = std::current_exception();
    }
    if (side.joinable()) {
        side.join();
    } else if (tmpl.rev) {
        lib_r.host = Library(pool.reverse_complemented(), pool.length, opt);
    }
    if (err_f) std::rethrow_exception(err_f);
    if (err_r) std::rethrow_exception(err_r);
    params.spec = tmpl.scan_spec(mismatches);
    params.max_mm = mismatches;
    params.use_first = use_first ? 1 : 0;
}

const LibDev* upload_lib_array(Context& ctx, const std::vector<LibDev>& libs, DeviceBuffer& storage) {
    storage.upload(libs.data(), libs.size() * sizeof(LibDev), ctx.stream);
    SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
    return storage.as<LibDev>();
}

void SingleMatcher::upload(Context& ctx) {
    std::vector<LibDev> libs(2);
    std::memset(libs.data(), 0, 2 * sizeof(LibDev));
    params.kw = 1;
    if (tmpl.fwd) {
        lib_f.upload(ctx);
        libs[0] = lib_f.dev;
        params.kw = std::max(params.kw, lib_f.dev.KW);
    }
    if (tmpl.rev) {
        lib_r.upload(ctx);
        libs[1] = lib_r.dev;
        params.kw = std::max(params.kw, lib_r.dev.KW);
    }
    params.libs = upload_lib_array(ctx, libs, libs_dev);

    // Seed buckets with the first candidate inline (uniform-length kernel's seeded search)
    have_ibuckets = false;
    {
        const Library* strands[2] = { tmpl.fwd ? &lib_f.host : nullptr, tmpl.rev ? &lib_r.host : nullptr };
        bool ok = true;
        for (const Library* lib : strands) {
            if (!lib) continue;
            if (lib->KW != 1 || lib->nseeds < 1 || lib->cand_rows.empty() || lib->nentries() >= (1u << 24)) ok = false;
            if (ok) {
                for (const uint2& b : lib->buckets) ok = ok && b.y < 255;
            }
        }
        if (ok && (strands[0] || strands[1])) {
            for (int k = 0; k < 2; ++k) {
                ibuckets[k].release();
                const Library* lib = strands[k];
                if (!lib) continue;
                std::vector<uint32_t> rows(lib->buckets.size() * 4, 0);
                const size_t per_seed = lib->nbuckets, E = lib->nentries();
                for (size_t b = 0; b < lib->buckets.size(); ++b) {
                    const uint2 bk = lib->buckets[b];
                    if (bk.y == 0) continue;
                    const size_t sd = b / per_seed;
                    const uint32_t* first = &lib->cand_rows[4 * (sd * E + bk.x)];
                    rows[4 * b + 0] = first[0];
                    rows[4 * b + 1] = first[1];
                    rows[4 * b + 2] = first[2];
                    rows[4 * b + 3] = bk.x | (bk.y << 24);
                }
                ibuckets[k].upload(rows.data(), rows.size() * sizeof(uint32_t), ctx.stream);
            }
            SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
            have_ibuckets = true;
        }
    }

    // Joint exact table of both strands (libdev.hpp): filled from the strands' own cuckoo tables, so a lookup answers exactly
    // what they answer.
    joint.release();
    joint_shift = 0;
    const Library* both[2] = { tmpl.fwd ? &lib_f.host : nullptr, tmpl.rev ? &lib_r.host : nullptr };
    const Library* any = both[0] ? both[0] : both[1];
    if (any && any->KW == 1 && any->L <= JOINT_MAX_KEYLEN) {
        struct Entry {
            uint32_t kh, kl;
            int32_t value;
        };
        std::vector<Entry> entries;
        for (int strand = 0; strand < 2; ++strand) {
            const Library* lib = both[strand];
            if (!lib) continue;
            const size_t nslots = lib->slots.size() / lib->slot_words;
            for (size_t k = 0; k < nslots; ++k) {
                const uint32_t* slot = &lib->slots[k * lib->slot_words];
                if ((int32_t)slot[2] < 0) continue;   // empty
                entries.push_back(Entry{ slot[0] | ((uint32_t)strand << 31), slot[1], (int32_t)slot[2] });
            }
        }
        uint32_t bits = 4;
        while ((1ull << bits) < entries.size() + 1 && bits < 28) ++bits;
        std::vector<uint32_t> table;
        for (;; ++bits) {
            if (bits > 29) throw Error("could not build the joint barcode hash table");
            const size_t n = (size_t)1 << bits;
            table.assign(2 * n * 4, 0);
            for (size_t k = 0; k < 2 * n; ++k) table[4 * k + 2] = 0xFFFFFFFFu;
            auto home = [&](const Entry& e, int t) {
                const uint32_t x = joint_hash(e.kh, e.kl);
                return (size_t)t * n + ((t == 0 ? x : joint_hash2(x)) >> (32 - bits));
            };
            bool ok = true;
            for (size_t i = 0; i < entries.size() && ok; ++i) {
                Entry cur = entries[i];
                int t = 0;
                ok = false;
                for (int kicks = 0; kicks < 2000; ++kicks) {
                    uint32_t* slot = &table[4 * home(cur, t)];
                    if ((int32_t)slot[2] < 0) {
                        slot[0] = cur.kh;
                        slot[1] = cur.kl;
                        slot[2] = (uint32_t)cur.value;
                        ok = true;
                        break;
                    }
                    if (kicks == 0) {   // try the other home before evicting anyone
                        uint32_t* other = &table[4 * home(cur, 1)];
                        if ((int32_t)other[2] < 0) {
                            other[0] = cur.kh;
                            other[1] = cur.kl;
                            other[2] = (uint32_t)cur.value;
                            ok = true;
                            break;
                        }
                    }
                    const Entry evicted{ slot[0], slot[1], (int32_t)slot[2] };
                    slot[0] = cur.kh;
                    slot[1] = cur.kl;
                    slot[2] = (uint32_t)cur.value;
                    cur = evicted;
                    t ^= 1;
                }
            }
            if (ok) break;
        }
        joint.upload(table.data(), table.size() * sizeof(uint32_t), ctx.stream);
        SCG_CUDA_CHECK(cudaStreamSynchronize(ctx.stream));
        joint_shift = 32 - bits;
    }
}

// A matcher for these arguments, from the context's cache when an earlier call (another file of the same screen)
// already built and uploaded it.  Only successful builds are cached, so validation errors are raised every time.
// A matcher of a recent call with the same template, options and pool (compared by a 128-bit hash of the pool's raw
// C strings, eight bytes at a time): a hit skips marshalling the pool altogether -- the same content went through
// every validation when the entry was made.  A miss marshals the pool, validates, builds and uploads.
std::shared_ptr<SingleMatcher> cached_single_matcher(Context& ctx, const char* constant, int strand, const char* const* pool, int npool,
                                                     int mismatches, bool use_first) {
    // The pool's strings are separate allocations (one cache miss each): pieces of the pool are hashed on the host threads,
    // every piece into its own pair of words, and the pairs are folded in order.
    struct Pair {
        unsigned long long k1, k2;
    };
    auto feed = [](Pair& h, const char* data, size_t n) {
        h.k1 = mix64(h.k1 ^ n);
        h.k2 = (h.k2 ^ (0xA24BAED4963EE407ull + n)) * 1099511628211ull + (h.k2 >> 29);   // the length goes into both words
        size_t i = 0;
        for (; i + 8 <= n; i += 8) {
            unsigned long long w;
            std::memcpy(&w, data + i, 8);
            h.k1 = mix64(h.k1 ^ w);
            h.k2 = (h.k2 ^ w) * 1099511628211ull + (h.k2 >> 29);
        }
        unsigned long long w = 0;
        if (i < n) std::memcpy(&w, data + i, n - i);
        h.k1 = mix64(h.k1 ^ w);
        h.k2 = (h.k2 ^ w) * 1099511628211ull + (h.k2 >> 29);
    };
    Pair total{ 1469598103934665603ull, 0x9E3779B97F4A7C15ull };
    const int header[4] = { strand, mismatches, use_first ? 1 : 0, npool };
    feed(total, reinterpret_cast<const char*>(header), sizeof header);
    feed(total, constant, std::strlen(constant));
    {
        const int pieces = npool >= 4096 ? 16 : 1;
        std::vector<Pair> part((size_t)pieces);
        auto work = [&](int k) {
            Pair h{ 1469598103934665603ull + (unsigned long long)k, 0x9E3779B97F4A7C15ull };
            const int b = (int)((long long)npool * k / pieces), e = (int)((long long)npool * (k + 1) / pieces);
            for (int i = b; i < e; ++i) feed(h, pool[i], std::strlen(pool[i]));
            part[(size_t)k] = h;
        };
        if (pieces > 1) {
            HostPool::instance().parallel_for(pieces, pieces, work);
        } else {
            work(0);
        }
        for (const Pair& h : part) feed(total, reinterpret_cast<const char*>(&h), sizeof h);
    }
    const unsigned long long k1 = total.k1, k2 = total.k2;
    // a hit also has to agree on what can be compared without marshalling the pool: its size, the template, and the first
    // and last sequences (a 128-bit collision between two real libraries would otherwise return the wrong tables silently)
    const std::string first_seq = npool > 0 ? pool[0] : "", last_seq = npool > 0 ? pool[npool - 1] : "";
    for (auto& e : ctx.single_cache) {
        if (e.key1 == k1 && e.key2 == k2 && e.npool == npool && e.constant == constant && e.first_seq == first_seq && e.last_seq == last_seq) {
            return e.matcher;
        }
    }
    const Pool p(pool, npool);
    auto m = std::make_shared<SingleMatcher>();
    m->prepare(constant, strand, p, mismatches, use_first, Duplicates::ERROR);  // all validation happens on the host
    ctx.ensure_ready();
    m->upload(ctx);
    if (ctx.single_cache.size() >= 4) ctx.single_cache.erase(ctx.single_cache.begin());
    Context::CachedMatcher entry;
    entry.key1 = k1;
    entry.key2 = k2;
    entry.npool = npool;
    entry.constant = constant;
    entry.first_seq = first_seq;
    entry.last_seq = last_seq;
    entry.matcher = m;
    ctx.single_cache.push_back(entry);
    return m;
}

// The pigeonhole seeds the specialised kernel may fold in: both strands' libraries have the same ones (same length,
// same budget); more than four seeds, or the "every entry is a candidate" seed, leave the list empty and the
// kernel sends its deferred reads through the generic search.
static void spec_seeds(const SingleMatcher& m, SpecSingleConfig& cfg) {
    cfg.seed_masks.clear();
    const Library& lib = m.tmpl.fwd ? m.lib_f.host : m.lib_r.host;
    cfg.dup_first = lib.opt.duplicates == Duplicates::FIRST ? 1 : 0;
    if (lib.KW != 1 || lib.nseeds < 1 || lib.nseeds > 4 || lib.cand_rows.empty()) return;
    for (int s = 0; s < lib.nseeds; ++s) {
        if (lib.seed_masks[s] == 0) {
            cfg.seed_masks.clear();
            return;
        }
        cfg.seed_masks.push_back(lib.seed_masks[s]);
    }
}

void launch_single(Context& ctx, const ReadsDev& reads, const SingleMatcher& m, int32_t* d_counts, int32_t* d_index, uint32_t* d_info,
                   cudaStream_t stream) {
    if (reads.n <= 0) return;
    const SingleParams& P = m.params;
    const long long ntiles = (reads.n + TILE - 1) / TILE;
    const int grid = ctx.grid_for(ntiles);

    // the template folded into the kernel at run time (spec_single.cuh via NVRTC)
    SpecSingleConfig cfg;
    cfg.fbases = m.tmpl.fwd_seq;
    cfg.rbases = m.tmpl.rev ? m.tmpl.rev_seq : std::string(m.tmpl.length, '-');
    cfg.T = m.tmpl.length;
    cfg.fwd = m.tmpl.fwd ? 1 : 0;
    cfg.rev = m.tmpl.rev ? 1 : 0;
    cfg.W = reads.W;
    // uniform_len is the longest read of the batch (also when per-read lengths are present)
    cfg.nb = std::max(1, (reads.uniform_len - m.tmpl.length + 1 + 31) / 32);
    cfg.cb = P.spec.cbits;
    cfg.mm = P.spec.mm;
    cfg.maxmm = P.max_mm;
    cfg.use_first = P.use_first;
    cfg.fstart = P.spec.fstart[0];
    cfg.rstart = P.spec.rstart[0];
    cfg.keylen = P.spec.rlen_f[0];
    spec_seeds(m, cfg);
    // the uniform-length kernel: reads no longer than 320 bases with at least one window, a budget the pigeonhole filter
    // is worth having for (at least four constant positions per group), indices that fit 32 bits
    {
        const int nwin = reads.uniform_len - m.tmpl.length + 1;
        int nconst = 0;
        for (char ch : m.tmpl.fwd_seq) nconst += ch != '-';
        const bool want_u = !std::getenv("SCG_SPEC_NO_UNIFORM");
        if (want_u && nwin >= 1 && P.spec.mm >= 0 && P.spec.mm <= 3 && nconst >= 4 * (P.spec.mm + 1) &&
            cfg.T <= 128 && reads.W + 2 >= (cfg.T + 31) / 32 + 1 && reads.n <= 0x7FFFFFC0ll) {
            cfg.ulen = reads.uniform_len;
            cfg.ragged = reads.lens != nullptr ? 1 : 0;   // trimmed reads: per-lane window masks
            cfg.info = d_info ? 1 : 0;
            cfg.joint = (m.joint.ptr != nullptr && m.joint_shift != 0 && !std::getenv("SCG_SPEC_NO_JOINT")) ? 1 : 0;
            cfg.has_index = d_index ? 1 : 0;
            cfg.ibuckets = (m.have_ibuckets && !std::getenv("SCG_SPEC_NO_IBUCKETS")) ? 1 : 0;
            // small pools: counters privatised in shared memory (4 bytes per barcode and block; up to 1024 barcodes keep the
            // kernel's 8 blocks per SM resident)
            const int hist_max = jit_env_int("SCG_SPEC_HIST_MAX", 1024, 0, 8192);
            if (m.npool > 0 && m.npool <= hist_max) cfg.hist = (m.npool + 31) / 32 * 32;
        }
    }
    std::string why;
    cudaKernel_t slow = nullptr;
    cudaKernel_t spec = (P.spec.mm >= 0 && cfg.T > 0) ? specialised_single_kernel(cfg, ctx.device, &why, &slow) : nullptr;
    if (spec) {
        ReadsDev reads_arg = reads;
        SpecTables tables;
        std::memset(&tables, 0, sizeof tables);
        const DeviceLibrary* both[2] = { m.tmpl.fwd ? &m.lib_f : nullptr, m.tmpl.rev ? &m.lib_r : nullptr };
        for (int s = 0; s < 2; ++s) {
            if (!both[s]) continue;
            tables.slots[s] = reinterpret_cast<const uint4*>(both[s]->dev.slots);
            tables.buckets[s] = both[s]->dev.buckets;
            tables.cand_rows[s] = both[s]->dev.cand_rows;
            tables.slot_mask[s] = both[s]->dev.slot_mask;
            tables.bucket_mask[s] = both[s]->dev.bucket_mask;
            tables.nentries[s] = both[s]->dev.nentries;
        }
        tables.libs = P.libs;
        tables.joint = m.joint.as<uint4>();
        tables.ibuckets[0] = m.ibuckets[0].as<uint4>();
        tables.ibuckets[1] = m.ibuckets[1].as<uint4>();
        tables.joint_shift = m.joint_shift;
        // persistent warps: as many blocks as are resident at once, each warp strides over the tiles
        const int resident = specialised_blocks_per_sm(spec);
        const int spec_grid = (int)std::max<long long>(1, std::min<long long>((ntiles + 3) / 4, (long long)ctx.sm_count * resident));
        if (cfg.ulen > 0) {
            // reads with several candidate windows are listed by the main kernel and finished by the follow-up kernel
            ctx.slow_list.reserve((size_t)(ntiles * TILE) * sizeof(uint32_t));
            ctx.slow_count.reserve(sizeof(uint32_t));
            uint32_t* d_list = ctx.slow_list.as<uint32_t>();
            uint32_t* d_count = ctx.slow_count.as<uint32_t>();
            SCG_CUDA_CHECK(cudaMemsetAsync(d_count, 0, sizeof(uint32_t), stream));
            void* args[] = { &reads_arg, &tables, &d_counts, &d_index, &d_info, &d_list, &d_count };
            SCG_CUDA_CHECK(cudaLaunchKernel(reinterpret_cast<const void*>(spec), dim3(spec_grid), dim3(128), args, 0, stream));
            const LibDev* libs = P.libs;
            void* slow_args[] = { &reads_arg, &libs, &d_list, &d_count, &d_counts, &d_index, &d_info };
            const int slow_grid = (int)std::max<long long>(1, std::min<long long>((ntiles + 3) / 4, (long long)ctx.sm_count * 2));
            SCG_CUDA_CHECK(cudaLaunchKernel(reinterpret_cast<const void*>(slow), dim3(slow_grid), dim3(128), slow_args, 0, stream));
            ++ctx.launches;
        } else {
            void* args[] = { &reads_arg, &tables, &d_counts, &d_index, &d_info };
            SCG_CUDA_CHECK(cudaLaunchKernel(reinterpret_cast<const void*>(spec), dim3(spec_grid), dim3(128), args, 0, stream));
        }
        m.kernel_note = cfg.ulen > 0 ? std::string("specialised (NVRTC), ") + (cfg.ragged ? "trimmed reads, " : "uniform-length ") +
                                           "filter+verify, " + std::to_string(resident) + " blocks/SM"
                                     : "specialised (NVRTC)";
        ctx.kernel_note = m.kernel_note;
    } else {
        dispatch_cb(P.spec.cbits, [&](auto CB) {
            dispatch_kw(P.kw, [&](auto KW) {
                single_kernel<decltype(CB)::value, decltype(KW)::value><<<grid, 128, 0, stream>>>(reads, P, d_counts, d_index, d_info);
            });
        });
        m.kernel_note = "generic (" + why + ")";
        ctx.kernel_note = m.kernel_note;
    }
    SCG_CUDA_CHECK(cudaGetLastError());
    ++ctx.launches;
    ++ctx.timing.launches;
}

} // namespace scg

using namespace scg;

extern "C" {

const char* scg_version(void) { return "screencounter_b200 0.1.0 (sm_100a)"; }

int scg_ctx_create(scg_ctx** out, int device) {
    try {
        *out = new scg_ctx(device);
        return 0;
    } catch (const std::exception& e) {
        creation_error() = e.what();
        return 1;
    }
}

void scg_ctx_destroy(scg_ctx* ctx) { delete ctx; }

const char* scg_last_error(const scg_ctx* ctx) { return ctx ? ctx->impl.last_error.c_str() : creation_error().c_str(); }

const char* scg_timing_json(const scg_ctx* ctx) { return ctx ? ctx->impl.timing_json.c_str() : "{}"; }

long long scg_kernel_launches(const scg_ctx* ctx) {
    if (!ctx) return 0;
    long long n = ctx->impl.launches;
    for (const auto& p : ctx->peers) n += p->impl.launches;
    return n;
}

size_t scg_result_rows(const scg_result* r) { return r ? r->rows() : 0; }
int scg_result_width(const scg_result* r) { return r ? r->width : 0; }
size_t scg_result_reads(const scg_result* r) { return (r && r->trace_width) ? r->trace_index.size() / r->trace_width : 0; }
int scg_result_trace_width(const scg_result* r) { return r ? r->trace_width : 0; }

int scg_result_copy_table(const scg_result* r, int32_t* keys, char* strings, int32_t* freq) {
    if (!r) return 1;
    if (r->on_device) {
        // the table was sorted and rendered on the device and waits there: straight into the caller's arrays
        int current = -1;
        cudaGetDevice(&current);
        bool ok = cudaSetDevice(r->device) == cudaSuccess;
        const size_t n = r->d_rows;
        if (ok && n && keys && r->d_keys.ptr) ok = cudaMemcpy(keys, r->d_keys.ptr, n * (size_t)r->width * sizeof(int32_t), cudaMemcpyDeviceToHost) == cudaSuccess;
        if (ok && n && strings && r->d_strings.ptr) ok = cudaMemcpy(strings, r->d_strings.ptr, n * (size_t)r->width, cudaMemcpyDeviceToHost) == cudaSuccess;
        if (ok && n && freq && r->d_freq.ptr) ok = cudaMemcpy(freq, r->d_freq.ptr, n * sizeof(int32_t), cudaMemcpyDeviceToHost) == cudaSuccess;
        if (current >= 0 && current != r->device) cudaSetDevice(current);
        if (!ok) {
            cudaGetLastError();
            return 1;
        }
        return 0;
    }
    if (keys && !r->keys.empty()) std::memcpy(keys, r->keys.data(), r->keys.size() * sizeof(int32_t));
    if (strings && !r->strings.empty()) std::memcpy(strings, r->strings.data(), r->strings.size());
    if (freq && !r->freq.empty()) std::memcpy(freq, r->freq.data(), r->freq.size() * sizeof(int32_t));
    return 0;
}

int scg_result_copy_trace(const scg_result* r, int32_t* index, uint32_t* info) {
    if (!r) return 1;
    if (index && !r->trace_index.empty()) std::memcpy(index, r->trace_index.data(), r->trace_index.size() * sizeof(int32_t));
    if (info && !r->trace_info.empty()) std::memcpy(info, r->trace_info.data(), r->trace_info.size() * sizeof(uint32_t));
    return 0;
}

void scg_result_free(scg_result* r) { delete r; }

// ---- countSingleBarcodes (reference src/count_single_barcodes.cpp:12-50) --------------------
} // extern "C"

namespace scg {

// SingleBarcodeSingleEnd over one input on one device: every batch of the reader through the kernels, counts accumulated
// in d_counts (left on the device).  Returns the number of reads.
long long count_single_core(Context& c, FastqReader* reader, const SingleMatcher& m, int nthreads, int32_t* d_counts, TraceSink& sink) {
    ReadPipeline pipe(c, reader, nullptr, nthreads, false);
    ReadPipeline::Batch b;
    long long nreads = 0;
    while (pipe.next(b)) {
        sink.prepare(b.n, true);
        launch_single(c, b.reads1, m, d_counts, sink.enabled ? sink.d_index.as<int32_t>() : nullptr,
                      sink.enabled ? sink.d_info.as<uint32_t>() : nullptr, c.stream);
        pipe.submitted(b);
        sink.collect(c, b.n, true);
        nreads += b.n;
    }
    return nreads;
}

} // namespace scg

extern "C" {

} // extern "C"

namespace scg {

// countSingleBarcodes on the context's first device, or -- split_over_devices, a context of several devices and an input that
// can be cut -- on all of them (runners_multi.cu).  Throws; the C entry points wrap it.
void count_single_file(scg_ctx* ctx, const scg_source* src, const char* constant, int strand, const char* const* pool, int npool,
                       int mismatches, int use_first, int nthreads, int32_t* counts, int32_t* total, scg_result** trace,
                       bool split_over_devices) {
    {
        Context& c = ctx->impl;
        const double t_start = now_s();
        c.timing = Timing();
        // same order as the reference glue: open the file, marshal the pool, build the handler, then read
        Source source(src);
        const double t_setup = now_s();
        const std::shared_ptr<SingleMatcher> matcher = cached_single_matcher(c, constant, strand, pool, npool, mismatches, use_first != 0);
        const SingleMatcher& m = *matcher;
        c.ensure_ready();
        c.timing.setup_s += now_s() - t_setup;

        // several devices (scg_ctx_create_multi): the file's text is cut at record boundaries and every device counts its part
        if (split_over_devices && !ctx->peers.empty() &&
            count_single_multi(ctx, *source.reader, constant, strand, pool, npool, mismatches, use_first != 0, nthreads, counts, total, trace)) {
            c.timing.total_s = now_s() - t_start;
            c.finish_timing();
            return;
        }

        DeviceBuffer d_counts;
        d_counts.alloc((size_t)std::max(npool, 1) * sizeof(int32_t), true);
        TraceSink sink;
        sink.enabled = trace != nullptr;
        const long long nreads = count_single_core(c, source.reader.get(), m, nthreads, d_counts.as<int32_t>(), sink);
        double t0 = now_s();
        SCG_CUDA_CHECK(cudaMemcpyAsync(counts, d_counts.ptr, (size_t)npool * sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
        SCG_CUDA_CHECK(cudaStreamSynchronize(c.stream));
        c.timing.device_s += now_s() - t0;
        *total = (int32_t)nreads;  // SingleBarcodeSingleEnd::process counts every read, matched or not (:103)
        if (trace) {
            auto* r = new scg_result;
            r->trace_width = 1;
            r->trace_index.swap(sink.index);
            r->trace_info.swap(sink.info);
            *trace = r;
        }
        c.timing.parse_s = source.reader->parse_seconds();
        c.timing.total_s = now_s() - t_start;
        c.finish_timing();
    }
}

} // namespace scg

extern "C" {

int scg_count_single(scg_ctx* ctx, const scg_source* src, const char* constant, int strand, const char* const* pool, int npool,
                     int mismatches, int use_first, int nthreads, int32_t* counts, int32_t* total, scg_result** trace) {
    return guarded(ctx, [&] {
        count_single_file(ctx, src, constant, strand, pool, npool, mismatches, use_first, nthreads, counts, total, trace, true);
    });
}

// ---- matchBarcodes (reference src/match_barcodes.cpp:7-37) -----------------------------------
int scg_match_barcodes(scg_ctx* ctx, const char* const* sequences, int nsequences, const char* const* choices, int nchoices,
                       int substitutions, int reverse, int32_t* index, int32_t* mismatches) {
    return guarded(ctx, [&] {
        Context& c = ctx->impl;
        Pool lib_pool(choices, nchoices);
        LibraryOptions opt;
        opt.max_mismatches = substitutions;
        opt.duplicates = Duplicates::ERROR;
        Library host(reverse ? lib_pool.reverse_complemented() : lib_pool.seqs, lib_pool.length, opt);
        Pool queries(sequences, nsequences);  // format_pointers on the queries too (:19)
        if (nsequences == 0) return;
        c.ensure_ready();
        DeviceLibrary lib;
        lib.host = std::move(host);
        lib.upload(c);
        // The reference hands each query's C string to a search of the library's length; queries are
        // packed at that length (shorter queries would read past their terminator in the reference).
        const int L = lib.host.L, KW = lib.host.KW;
        // (a longer query is matched on its first L characters, as the trie walk does; a shorter one
        // makes the reference read past the string's end, which is refused here)
        if (queries.length < L) {
            throw Error("sequences (" + std::to_string(queries.length) + " bp) are shorter than the choices (" + std::to_string(L) + " bp)");
        }
        std::vector<uint32_t> qk((size_t)nsequences * 3 * KW, 0);
        for (int i = 0; i < nsequences; ++i) {
            uint32_t* base = &qk[(size_t)i * 3 * KW];
            pack_key(queries.seqs[i].data(), L, base, base + KW, base + 2 * KW);
        }
        DeviceBuffer d_q, d_idx, d_mm, d_lib;
        const LibDev* libp = upload_lib_array(c, std::vector<LibDev>{ lib.dev }, d_lib);
        d_q.upload(qk.data(), qk.size() * sizeof(uint32_t), c.stream);
        d_idx.alloc((size_t)nsequences * sizeof(int32_t), false);
        d_mm.alloc((size_t)nsequences * sizeof(int32_t), false);
        const int grid = (nsequences + 127) / 128;
        dispatch_kw(KW, [&](auto KWC) {
            constexpr int K = decltype(KWC)::value;
            if (K == KW) {
                match_kernel<K><<<grid, 128, 0, c.stream>>>(d_q.as<uint32_t>(), nsequences, libp, substitutions, d_idx.as<int32_t>(),
                                                            d_mm.as<int32_t>());
            } else {
                // repack to the compiled width
                std::vector<uint32_t> wide((size_t)nsequences * 3 * K, 0);
                for (int i = 0; i < nsequences; ++i) {
                    for (int pl = 0; pl < 3; ++pl) {
                        std::memcpy(&wide[((size_t)i * 3 + pl) * K], &qk[((size_t)i * 3 + pl) * KW], KW * sizeof(uint32_t));
                    }
                }
                d_q.upload(wide.data(), wide.size() * sizeof(uint32_t), c.stream);
                SCG_CUDA_CHECK(cudaStreamSynchronize(c.stream));
                match_kernel<K><<<grid, 128, 0, c.stream>>>(d_q.as<uint32_t>(), nsequences, libp, substitutions, d_idx.as<int32_t>(),
                                                            d_mm.as<int32_t>());
            }
        });
        SCG_CUDA_CHECK(cudaGetLastError());
        ++c.launches;
        SCG_CUDA_CHECK(cudaMemcpyAsync(index, d_idx.ptr, (size_t)nsequences * sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
        SCG_CUDA_CHECK(cudaMemcpyAsync(mismatches, d_mm.ptr, (size_t)nsequences * sizeof(int32_t), cudaMemcpyDeviceToHost, c.stream));
        SCG_CUDA_CHECK(cudaStreamSynchronize(c.stream));
    });
}

// ---- resident reads ----------------------------------------------------------------------------
int scg_reads_from_source(scg_ctx* ctx, const scg_source* src, int nthreads, scg_reads** out) {
    return guarded(ctx, [&] {
        Context& c = ctx->impl;
        Source source(src);
        c.ensure_ready();
        std::unique_ptr<scg_reads> reads(new scg_reads);
        reads->owner = ctx;
        ReadPipeline pipe(c, source.reader.get(), nullptr, nthreads, false);
        ReadPipeline::Batch b;
        while (pipe.next(b)) {
            // keep a private copy of the staged batch
            DeviceBatch keep;
            const size_t words = (size_t)((b.n + TILE - 1) / TILE) * tile_words(b.reads1.W);
            keep.data.alloc(words * sizeof(uint32_t) + READ_GUARD_BYTES, false);
            SCG_CUDA_CHECK(cudaMemcpyAsync(keep.data.ptr, b.reads1.data, words * sizeof(uint32_t), cudaMemcpyDeviceToDevice, c.stream));
            keep.view = b.reads1;
            keep.view.data = keep.data.as<uint32_t>();
            reads->device_bytes += (long long)(words * sizeof(uint32_t));
            if (b.reads1.lens) {
                const size_t padded = (size_t)((b.n + TILE - 1) / TILE) * TILE;
                keep.lens.alloc(padded * sizeof(uint16_t), false);
                SCG_CUDA_CHECK(cudaMemcpyAsync(keep.lens.ptr, b.reads1.lens, padded * sizeof(uint16_t), cudaMemcpyDeviceToDevice, c.stream));
                keep.view.lens = keep.lens.as<uint16_t>();
                reads->device_bytes += (long long)(padded * sizeof(uint16_t));
            }
            pipe.submitted(b);
            reads->n += b.n;
            reads->batches.push_back(std::move(keep));
        }
        SCG_CUDA_CHECK(cudaStreamSynchronize(c.stream));
        *out = reads.release();
    });
}

long long scg_reads_count(const scg_reads* r) { return r ? r->n : 0; }
long long scg_reads_device_bytes(const scg_reads* r) { return r ? r->device_bytes : 0; }
void scg_reads_free(scg_reads* r) { delete r; }

// ---- resident single-barcode plan ----------------------------------------------------------------
int scg_single_plan_create(scg_ctx* ctx, const char* constant, int strand, const char* const* pool, int npool, int mismatches,
                           int use_first, scg_plan** out) {
    return guarded(ctx, [&] {
        Context& c = ctx->impl;
        Pool p(pool, npool);
        std::unique_ptr<scg_plan> plan(new scg_plan);
        plan->owner = ctx;
        plan->npool = npool;
        plan->matcher.prepare(constant, strand, p, mismatches, use_first != 0, Duplicates::ERROR);
        c.ensure_ready();
        plan->matcher.upload(c);
        *out = plan.release();
    });
}

int scg_single_plan_run(scg_plan* plan, const scg_reads* reads, int32_t* d_counts, int32_t* d_index, void* cuda_stream) {
    if (!plan || !reads) return 1;
    return guarded(plan->owner, [&] {
        Context& c = plan->owner->impl;
        if (plan->kind != scg_plan::SINGLE) throw Error("not a single-barcode plan");
        SCG_CUDA_CHECK(cudaSetDevice(c.device));
        cudaStream_t st = cuda_stream == SCG_STREAM_OWN ? c.stream : static_cast<cudaStream_t>(cuda_stream);
        long long at = 0;
        for (const auto& b : reads->batches) {
            launch_single(c, b.view, plan->matcher, d_counts, d_index ? d_index + at : nullptr, nullptr, st);
            at += b.view.n;
        }
    });
}

void scg_plan_free(scg_plan* plan) { delete plan; }

const char* scg_plan_kernel(const scg_plan* plan) {
    if (!plan) return "";
    return plan->kind == scg_plan::SINGLE ? plan->matcher.kernel_note.c_str() : plan->kernel_note.c_str();
}

// ---- run-time compiler check (no device needed for the compile step) --------------------------------------
static int jit_selftest(const char* constant, int strand, int mismatches, int words_per_plane, int uniform_len, char* message, size_t capacity);

int scg_jit_selftest(const char* constant, int strand, int mismatches, int words_per_plane, char* message, size_t capacity) {
    return jit_selftest(constant, strand, mismatches, words_per_plane, 0, message, capacity);
}

int scg_jit_selftest_uniform(const char* constant, int strand, int mismatches, int read_len, char* message, size_t capacity) {
    return jit_selftest(constant, strand, mismatches, std::max(1, (read_len + 31) / 32), read_len, message, capacity);
}

static int jit_selftest(const char* constant, int strand, int mismatches, int words_per_plane, int uniform_len, char* message, size_t capacity) {
    std::string msg;
    int status = 1;
    try {
        TemplateSpec t(constant, strand);
        if (t.fwd_regions.size() != 1) throw Error("expected one variable region in the constant template");
        const ScanSpec s = t.scan_spec(mismatches);
        SpecSingleConfig cfg;
        cfg.fbases = t.fwd_seq;
        cfg.rbases = t.rev ? t.rev_seq : std::string(t.length, '-');
        cfg.T = t.length;
        cfg.fwd = t.fwd;
        cfg.rev = t.rev;
        cfg.W = words_per_plane;
        cfg.nb = std::max(1, (32 * words_per_plane - t.length + 1 + 31) / 32);
        cfg.cb = s.cbits;
        cfg.mm = s.mm;
        cfg.maxmm = mismatches;
        cfg.use_first = 1;
        cfg.fstart = s.fstart[0];
        cfg.rstart = s.rstart[0];
        cfg.keylen = s.rlen_f[0];
        // the seeds library.cpp would build for this budget: cap + 1 contiguous parts of the variable region
        const int cap = std::min(std::max(mismatches, 0), cfg.keylen);
        if (cap >= 1 && cap + 1 <= 4 && cfg.keylen <= 32) {
            for (int p = 0; p < cap + 1; ++p) {
                const int from = (int)((long long)cfg.keylen * p / (cap + 1)), to = (int)((long long)cfg.keylen * (p + 1) / (cap + 1));
                uint32_t mask = 0;
                for (int b = from; b < to; ++b) mask |= 1u << b;
                cfg.seed_masks.push_back(mask);
            }
        }
        if (uniform_len > 0) {
            const int nwin = uniform_len - t.length + 1;
            if (nwin < 1) throw Error("the uniform-length kernel needs reads at least as long as the template");
            cfg.ulen = uniform_len;
            cfg.W = std::max(cfg.W, (uniform_len + 31) / 32);
            cfg.nb = 1;
        }
        std::string why;
        cudaKernel_t k = specialised_single_kernel(cfg, 0, &why);
        if (k) {
            msg = "ok: " + jit_status();
            status = 0;
        } else {
            msg = why + " [" + jit_status() + "]";
            // compiling worked if the only failure is loading the cubin onto a (missing) device
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

// ---- host-only reader/packer check ---------------------------------------------------------------------
int scg_host_pack_roundtrip(const scg_source* src, int nthreads, char* bases, long long* offsets, long long* n_reads,
                            long long* n_bases) {
    try {
        Source source(src);
        source.reader->set_threads(nthreads);
        long long nr = 0, nb = 0;
        if (offsets) offsets[0] = 0;
        std::vector<uint32_t> packed;
        std::vector<uint16_t> lens;
        for (;;) {
            const auto& recs = source.reader->next(1u << 16);
            if (recs.empty()) break;
            uint32_t maxlen = 0;
            for (const auto& r : recs) maxlen = std::max(maxlen, r.len);
            const int W = std::max(1, ceil_div((int)maxlen, 32));
            const size_t padded = (recs.size() + TILE - 1) / TILE * TILE;
            packed.assign(padded / TILE * tile_words(W), 0xDEADBEEFu);
            lens.assign(padded, 0);
            pack_records(recs.data(), recs.size(), W, packed.data(), lens.data(), nullptr, nthreads);
            for (size_t i = 0; i < recs.size(); ++i) {
                const uint32_t* base = packed.data() + (i / TILE) * tile_words(W) + (i % TILE);
                if (bases) {
                    for (uint32_t k = 0; k < lens[i]; ++k) {
                        const uint32_t h = (base[(size_t)(PLANE_H * W + (k >> 5)) * TILE] >> (k & 31)) & 1u;
                        const uint32_t l = (base[(size_t)(PLANE_L * W + (k >> 5)) * TILE] >> (k & 31)) & 1u;
                        const uint32_t n = (base[(size_t)(PLANE_N * W + (k >> 5)) * TILE] >> (k & 31)) & 1u;
                        bases[nb + k] = n ? 'N' : "ACGT"[(h << 1) | l];
                    }
                }
                nb += lens[i];
                ++nr;
                if (offsets) offsets[nr] = nb;
            }
        }
        if (n_reads) *n_reads = nr;
        if (n_bases) *n_bases = nb;
        return 0;
    } catch (const std::exception& e) {
        creation_error() = e.what();
        return 1;
    }
}

// ---- plain device helpers ---------------------------------------------------------------------------
int scg_device_alloc(scg_ctx* ctx, size_t bytes, void** out) {
    return guarded(ctx, [&] {
        ctx->impl.ensure_ready();
        void* p = nullptr;
        SCG_CUDA_CHECK(cudaMalloc(&p, std::max<size_t>(bytes, 16)));
        // zeroed on the context's stream and waited for: the context's stream is non-blocking, so a memset on the legacy
        // stream would not be ordered before a following scg_*_plan_run on SCG_STREAM_OWN
        SCG_CUDA_CHECK(cudaMemsetAsync(p, 0, std::max<size_t>(bytes, 16), ctx->impl.stream));
        SCG_CUDA_CHECK(cudaStreamSynchronize(ctx->impl.stream));
        *out = p;
    });
}

int scg_host_alloc(scg_ctx* ctx, size_t bytes, void** out) {
    return guarded(ctx, [&] {
        ctx->impl.ensure_ready();
        void* p = nullptr;
        SCG_CUDA_CHECK(cudaHostAlloc(&p, std::max<size_t>(bytes, 16), cudaHostAllocPortable));
        *out = p;
    });
}

int scg_host_free(scg_ctx* ctx, void* ptr) {
    return guarded(ctx, [&] {
        ctx->impl.ensure_ready();
        if (ptr) SCG_CUDA_CHECK(cudaFreeHost(ptr));
    });
}

int scg_device_free(scg_ctx* ctx, void* ptr) {
    return guarded(ctx, [&] {
        ctx->impl.ensure_ready();
        SCG_CUDA_CHECK(cudaFree(ptr));
    });
}

int scg_device_zero(scg_ctx* ctx, void* ptr, size_t bytes, void* cuda_stream) {
    return guarded(ctx, [&] {
        ctx->impl.ensure_ready();
        cudaStream_t st = cuda_stream == SCG_STREAM_OWN ? ctx->impl.stream : static_cast<cudaStream_t>(cuda_stream);
        SCG_CUDA_CHECK(cudaMemsetAsync(ptr, 0, bytes, st));
    });
}

int scg_device_to_host(scg_ctx* ctx, void* host, const void* dev, size_t bytes) {
    return guarded(ctx, [&] {
        ctx->impl.ensure_ready();
        SCG_CUDA_CHECK(cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, ctx->impl.stream));
        SCG_CUDA_CHECK(cudaStreamSynchronize(ctx->impl.stream));
    });
}

int scg_synchronize(scg_ctx* ctx) {
    return guarded(ctx, [&] {
        ctx->impl.ensure_ready();
        SCG_CUDA_CHECK(cudaDeviceSynchronize());
    });
}

} // extern "C"
