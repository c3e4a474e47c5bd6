#include "engine.hpp"

#include <algorithm>
#include <chrono>
#include <cstring>
#include <mutex>
#include <vector>

#include "ingest.hpp"
#include "pipeline.hpp"

namespace scg {

namespace {
double now_s() {
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
} // namespace

// ---------------------------------------------------------------------------------------
// buffers
// ---------------------------------------------------------------------------------------
// Device allocations are recycled through a small per-device cache: on the target boxes a cudaMalloc / cudaFree
// pair costs anywhere between 0.3 and 20 ms, which is more than a whole counting call.  A released block goes to the
// cache after a device-wide synchronise (what cudaFree would have implied); a request takes the smallest cached block
// of at least its size and at most twice its size.
namespace {
struct BlockCache {
    struct Block {
        void* ptr;
        size_t bytes;
        int device;
    };
    std::mutex mutex;
    std::vector<Block> blocks;
    size_t held = 0;
    static constexpr size_t kMaxHeld = 24ull << 30;
    static constexpr size_t kMaxBlocks = 256;
    ~BlockCache() {
        // process exit: the driver reclaims device memory; calling into a torn-down runtime is not safe
    }
    void* take(size_t n, int device, size_t* got) {
        std::lock_guard<std::mutex> lock(mutex);
        size_t best = blocks.size();
        const size_t limit = std::max<size_t>(2 * n, 1u << 16);
        for (size_t k = 0; k < blocks.size(); ++k) {
            const Block& b = blocks[k];
            if (b.device != device || b.bytes < n || b.bytes > limit) continue;
            if (best == blocks.size() || b.bytes < blocks[best].bytes) best = k;
        }
        if (best == blocks.size()) return nullptr;
        void* p = blocks[best].ptr;
        *got = blocks[best].bytes;
        held -= blocks[best].bytes;
        blocks.erase(blocks.begin() + (long)best);
        return p;
    }
    // frees every cached block of `device` (called on out-of-memory)
    void trim(int device) {
        std::vector<void*> doomed;
        {
            std::lock_guard<std::mutex> lock(mutex);
            for (size_t k = 0; k < blocks.size();) {
                if (blocks[k].device == device) {
                    doomed.push_back(blocks[k].ptr);
                    held -= blocks[k].bytes;
                    blocks.erase(blocks.begin() + (long)k);
                } else {
                    ++k;
                }
            }
        }
        if (!doomed.empty()) cudaDeviceSynchronize();
        for (void* p : doomed) cudaFree(p);
    }
    bool give(void* p, size_t n, int device) {
        std::lock_guard<std::mutex> lock(mutex);
        if (blocks.size() >= kMaxBlocks || held + n > kMaxHeld) return false;
        blocks.push_back(Block{ p, n, device });
        held += n;
        return true;
    }
};
BlockCache& block_cache() {
    static BlockCache* c = new BlockCache;   // intentionally leaked, see ~BlockCache
    return *c;
}
} // namespace

void DeviceBuffer::alloc(size_t n, bool zero) {
    release();
    if (n == 0) n = 16;
    int current = 0;
    SCG_CUDA_CHECK(cudaGetDevice(&current));
    size_t got = 0;
    ptr = block_cache().take(n, current, &got);
    if (ptr) {
        bytes = got;
    } else {
        cudaError_t st = cudaMalloc(&ptr, n);
        if (st == cudaErrorMemoryAllocation) {
            // the cache may be sitting on the memory that is asked for (it holds up to 24 GB): give this device's cached
            // blocks back and try once more before reporting out-of-memory
            cudaGetLastError();
            block_cache().trim(current);
            st = cudaMalloc(&ptr, n);
        }
        if (st != cudaSuccess) {
            ptr = nullptr;
            SCG_CUDA_CHECK(st);
        }
        bytes = n;
    }
    device = current;
    if (zero) {
        // the memset runs on the legacy stream, which the context's non-blocking stream does not wait for
        SCG_CUDA_CHECK(cudaMemset(ptr, 0, n));
        SCG_CUDA_CHECK(cudaStreamSynchronize(cudaStreamLegacy));
    }
}

void DeviceBuffer::reserve(size_t n) {
    if (n > bytes) alloc(n, false);
}

void DeviceBuffer::upload(const void* host, size_t n, cudaStream_t stream) {
    reserve(std::max<size_t>(n, 16));
    if (n) SCG_CUDA_CHECK(cudaMemcpyAsync(ptr, host, n, cudaMemcpyHostToDevice, stream));
}

void DeviceBuffer::release() {
    if (ptr) {
        // The block goes back to the cache of the device it was allocated on, whatever device is current now (handles are
        // freed from Python's garbage collector, R finalisers, other contexts' calls).  Whatever still uses the block on
        // THAT device must be done before somebody else gets it (cudaFree's implicit guarantee).
        int current = -1;
        const bool have_current = cudaGetDevice(&current) == cudaSuccess;
        bool cached = false;
        if (cudaSetDevice(device) == cudaSuccess) {
            cached = cudaDeviceSynchronize() == cudaSuccess && block_cache().give(ptr, bytes, device);
            if (!cached) cudaFree(ptr);
        } else {
            cudaGetLastError();
            cudaFree(ptr);
        }
        if (have_current && current != device) cudaSetDevice(current);
    }
    ptr = nullptr;
    bytes = 0;
}

PinnedBuffer::~PinnedBuffer() {
    if (ptr) cudaFreeHost(ptr);
}

void PinnedBuffer::reserve(size_t n) {
    if (n <= bytes) return;
    if (ptr) cudaFreeHost(ptr);
    ptr = nullptr;
    bytes = 0;
    SCG_CUDA_CHECK(cudaMallocHost(&ptr, n));
    bytes = n;
}

// ---------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------
Context::~Context() {
    if (ready) cudaSetDevice(device);
    for (auto& slot : staging) {
        if (slot.done) cudaEventDestroy(slot.done);
    }
    single_cache.clear();
    matcher_cache.clear();
    ingest[0].reset();
    ingest[1].reset();
    if (stream) cudaStreamDestroy(stream);
}

void Context::ensure_ready() {
    if (ready) {
        SCG_CUDA_CHECK(cudaSetDevice(device));
        return;
    }
    int count = 0;
    cudaError_t st = cudaGetDeviceCount(&count);
    if (st != cudaSuccess || count == 0) {
        throw Error(std::string("no usable CUDA device: this engine has no CPU fallback (") +
                    (st != cudaSuccess ? cudaGetErrorString(st) : "device count is 0") + ")");
    }
    if (device < 0 || device >= count) {
        throw Error("CUDA device " + std::to_string(device) + " does not exist (" + std::to_string(count) + " visible)");
    }
    SCG_CUDA_CHECK(cudaSetDevice(device));
    cudaDeviceProp prop;
    SCG_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        throw Error(std::string("device '") + prop.name + "' is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                    "; this library carries sm_100a code only");
    }
    sm_count = prop.multiProcessorCount;
    // The tables of this engine are probed at random, 16 or 32 bytes at a time: let L2 fetch single 32-byte sectors from DRAM
    // instead of pairs (the streams of packed reads arrive as whole lines by TMA either way).  SCG_L2_FETCH=64/128 restores more.
    {
        size_t granularity = 32;
        if (const char* env = std::getenv("SCG_L2_FETCH")) granularity = (size_t)std::max(32, std::atoi(env));
        cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, granularity);
        cudaGetLastError();
    }
    SCG_CUDA_CHECK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    ready = true;
}

int Context::grid_for(long long ntiles) const {
    // persistent warps: 4 warps per block, up to 16 blocks per SM resident; never more blocks than work
    long long blocks = (ntiles + 3) / 4;
    long long cap = (long long)sm_count * 16;
    return (int)std::max<long long>(1, std::min(blocks, cap));
}

void Context::finish_timing() {
    char buf[512];
    std::snprintf(buf, sizeof buf,
                  "{\"parse_s\": %.6f, \"pack_s\": %.6f, \"h2d_s\": %.6f, \"device_s\": %.6f, \"setup_s\": %.6f, \"harvest_s\": %.6f, \"merge_s\": %.6f, "
                  "\"total_s\": %.6f, \"reads\": %lld, \"bytes_h2d\": %lld, \"launches\": %lld, \"reader\": \"%s\", \"kernel\": \"",
                  timing.parse_s, timing.pack_s, timing.h2d_s, timing.device_s, timing.setup_s, timing.harvest_s, timing.merge_s, timing.total_s,
                  timing.reads, timing.bytes_h2d, timing.launches, timing.reader.c_str());
    timing_json = buf;
    for (char ch : kernel_note) {
        if (ch == '"' || ch == '\\' || (unsigned char)ch < 0x20) ch = ' ';
        timing_json.push_back(ch);
    }
    timing_json += "\"}";
}

// ---------------------------------------------------------------------------------------
// library upload
// ---------------------------------------------------------------------------------------
void DeviceLibrary::upload(Context& ctx) {
    cudaStream_t st = ctx.stream;
    slots.upload(host.slots.data(), host.slots.size() * sizeof(uint32_t), st);
    ent_keys.upload(host.ent_keys.data(), host.ent_keys.size() * sizeof(uint32_t), st);
    ent_idx.upload(host.ent_idx.data(), host.ent_idx.size() * sizeof(int32_t), st);
    seed_masks.upload(host.seed_masks.data(), host.seed_masks.size() * sizeof(uint32_t), st);
    buckets.upload(host.buckets.data(), host.buckets.size() * sizeof(uint2), st);
    cands.upload(host.cands.data(), host.cands.size() * sizeof(int32_t), st);
    cand_rows.upload(host.cand_rows.data(), host.cand_rows.size() * sizeof(uint32_t), st);
    prefix_slots.upload(host.prefix_slots.data(), host.prefix_slots.size() * sizeof(uint32_t), st);
    trie.upload(host.trie.data(), host.trie.size() * sizeof(int32_t), st);
    // seed buckets with their first candidate inline (libdev.hpp LibDev::ibuckets)
    bool inline_buckets = host.KW == 1 && host.nseeds >= 1 && !host.cand_rows.empty() && host.nentries() < (1u << 24);
    if (inline_buckets) {
        for (const uint2& b : host.buckets) inline_buckets = inline_buckets && b.y < 255;
    }
    std::vector<uint32_t> inline_rows;
    if (inline_buckets) {
        inline_rows.assign(host.buckets.size() * 4, 0);
        const size_t per_seed = host.nbuckets, E = host.nentries();
        for (size_t b = 0; b < host.buckets.size(); ++b) {
            const uint2 bk = host.buckets[b];
            if (bk.y == 0) continue;
            const uint32_t* first = &host.cand_rows[4 * ((b / per_seed) * E + bk.x)];
            inline_rows[4 * b + 0] = first[0];
            inline_rows[4 * b + 1] = first[1];
            inline_rows[4 * b + 2] = first[2];
            inline_rows[4 * b + 3] = bk.x | (bk.y << 24);
        }
        ibuckets.upload(inline_rows.data(), inline_rows.size() * sizeof(uint32_t), st);
    } else {
        ibuckets.release();
    }
    SCG_CUDA_CHECK(cudaStreamSynchronize(st));
    std::memset(&dev, 0, sizeof dev);
    dev.L = host.L;
    dev.KW = host.KW;
    dev.nentries = (int)host.nentries();
    dev.dup_first = host.opt.duplicates == Duplicates::FIRST;
    dev.slots = slots.as<uint32_t>();
    dev.slot_words = host.slot_words;
    dev.slot_mask = host.slot_mask;
    dev.ent_keys = ent_keys.as<uint32_t>();
    dev.ent_idx = ent_idx.as<int32_t>();
    dev.nseeds = host.nseeds;
    dev.seed_masks = seed_masks.as<uint32_t>();
    dev.buckets = buckets.as<uint2>();
    dev.bucket_mask = host.nbuckets ? host.nbuckets - 1 : 0;
    dev.cands = cands.as<int32_t>();
    dev.cand_rows = host.cand_rows.empty() ? nullptr : cand_rows.as<uint4>();
    dev.ibuckets = inline_buckets ? ibuckets.as<uint4>() : nullptr;
    dev.seg1 = host.opt.segmented ? host.opt.seg1 : 0;
    dev.prefix_slots = prefix_slots.as<uint32_t>();
    dev.prefix_mask = host.prefix_mask;
    dev.trie = host.trie.empty() ? nullptr : trie.as<int32_t>();
}

// ---------------------------------------------------------------------------------------
// FASTQ -> pinned -> device pipeline
// ---------------------------------------------------------------------------------------
ReadPipeline::ReadPipeline(Context& ctx, FastqReader* r1, FastqReader* r2, int nthreads, bool want_odd)
    : ctx_(ctx), r1_(r1), r2_(r2), nthreads_(std::max(1, nthreads)), want_odd_(want_odd) {
    if (r1_) r1_->set_threads(nthreads_);
    if (r2_) r2_->set_threads(nthreads_);
    slots_ = ctx_.staging;
    for (int k = 0; k < kSlots; ++k) {
        if (!slots_[k].done) SCG_CUDA_CHECK(cudaEventCreateWithFlags(&slots_[k].done, cudaEventDisableTiming));
        slots_[k].in_flight = false;
    }
    // Text that is entirely in host memory (caller's buffer, mmap'd raw file) is read on the device (ingest.hpp); gzip
    // streams keep the host reader.  Paired input needs both files in memory.
    // A block-gzip file (or image in memory) is read there too: its members cross PCIe compressed and are inflated on the device.
    if (device_ingest_enabled() && r1_) {
        auto readable = [&](FastqReader* r) {
            const char* t = nullptr;
            size_t n = 0;
            const BgzfIndex* image = nullptr;
            if (r->memory_text(&t, &n)) return n > 0;
            size_t begin = 0, end = 0;
            return device_inflate_enabled() && r->bgzf_image(&image, &begin, &end) && end > begin;
        };
        auto open = [&](FastqReader* r, int mate, bool odd) {
            const char* t = nullptr;
            size_t n = 0;
            const BgzfIndex* image = nullptr;
            if (r->memory_text(&t, &n)) return new DeviceIngest(ctx_, t, n, nthreads_, mate, odd);
            size_t begin = 0, end = 0;
            r->bgzf_image(&image, &begin, &end);
            return new DeviceIngest(ctx_, image, nthreads_, mate, odd, begin, end);
        };
        if (readable(r1_) && (!r2_ || readable(r2_))) {
            ingest_[0].reset(open(r1_, 0, want_odd_));
            if (r2_) ingest_[1].reset(open(r2_, 1, false));
        }
    }
}

ReadPipeline::~ReadPipeline() {
    // whatever still reads the staging buffers must finish before the next call reuses them
    for (int k = 0; k < kSlots; ++k) {
        if (slots_[k].in_flight) cudaEventSynchronize(slots_[k].done);
        slots_[k].in_flight = false;
    }
}

void ReadPipeline::stage(Slot& slot, int mate, const Record* recs, size_t count, uint32_t minlen, uint32_t maxlen) {
    Staged& s = slot.mate[mate];
    const int W = std::max(1, ceil_div((int)maxlen, 32));
    const size_t padded = (count + TILE - 1) / TILE * TILE;
    const size_t data_bytes = padded / TILE * tile_words(W) * sizeof(uint32_t);
    const bool uniform = (minlen == maxlen);
    s.pinned_data.reserve(data_bytes);
    if (!uniform) s.pinned_lens.reserve(padded * sizeof(uint16_t));
    if (want_odd_) {
        s.odd_host.resize(padded);
    }
    double t0 = now_s();
    pack_records(recs, count, W, s.pinned_data.as<uint32_t>(), uniform ? nullptr : s.pinned_lens.as<uint16_t>(),
                 want_odd_ ? s.odd_host.data() : nullptr, nthreads_);
    ctx_.timing.pack_s += now_s() - t0;

    s.dev.data.reserve(data_bytes + READ_GUARD_BYTES);
    SCG_CUDA_CHECK(cudaMemcpyAsync(s.dev.data.ptr, s.pinned_data.ptr, data_bytes, cudaMemcpyHostToDevice, ctx_.stream));
    ctx_.timing.bytes_h2d += (long long)data_bytes;
    s.dev.view.data = s.dev.data.as<uint32_t>();
    s.dev.view.W = W;
    s.dev.view.n = (long long)count;
    s.dev.view.uniform_len = (int)maxlen;
    s.dev.view.lens = nullptr;
    if (!uniform) {
        s.dev.lens.reserve(padded * sizeof(uint16_t));
        SCG_CUDA_CHECK(cudaMemcpyAsync(s.dev.lens.ptr, s.pinned_lens.ptr, padded * sizeof(uint16_t), cudaMemcpyHostToDevice, ctx_.stream));
        ctx_.timing.bytes_h2d += (long long)(padded * sizeof(uint16_t));
        s.dev.view.lens = s.dev.lens.as<uint16_t>();
    }
    if (want_odd_) {
        // pageable source: the copy is staged by the runtime before the call returns
        s.dev.odd.reserve(padded);
        SCG_CUDA_CHECK(cudaMemcpyAsync(s.dev.odd.ptr, s.odd_host.data(), padded, cudaMemcpyHostToDevice, ctx_.stream));
        ctx_.timing.bytes_h2d += (long long)padded;
    }
}

long long ReadPipeline::count_odd(const Batch& b) const {
    if (!b.slot) return -1;
    const auto& flags = static_cast<StagingSlot*>(b.slot)->mate[0].odd_host;
    long long n = 0;
    for (long long i = 0; i < b.n; ++i) n += flags[(size_t)i];
    return n;
}

void ReadPipeline::raw_read(const Batch& b, long long index, std::string& seq) {
    seq.clear();
    if (!b.slot) {
        ingest_[0]->raw_read(index, seq);
        return;
    }
    const Record& r = b.recs1[index];
    seq.reserve(r.len);
    for (uint32_t k = 0; k < r.span; ++k) {
        if (r.seq[k] != '\n') seq.push_back(r.seq[k]);
    }
}

// One round of the device-side reader(s).  Returns true with a batch in `out`, or true with `ended` set at the clean end
// of the input, or false once the host readers have been positioned to take over.
bool ReadPipeline::next_device(Batch& out, bool& ended) {
    ended = false;
    const bool paired = ingest_[1] != nullptr;
    for (;;) {
        if (handover_pending_) {
            // something that is not a four-line record (or a carry area that ran over): the host reader(s) take over at
            // the byte where the device stopped, both mates having consumed the same number of records
            r1_->resume_at(ingest_[0]->consumed(), ingest_[0]->records());
            ctx_.timing.reader += ", then host from byte " + std::to_string(ingest_[0]->consumed());
            if (paired) r2_->resume_at(ingest_[1]->consumed(), ingest_[1]->records());
            ingest_[0].reset();
            ingest_[1].reset();
            handover_pending_ = false;
            return false;
        }
        DeviceIngest::Result res1, res2;
        bool more = false;
        if (!paired) {
            more = ingest_[0]->next(res1);
        } else {
            const bool s1 = ingest_[0]->stage(), s2 = ingest_[1]->stage();
            if (!s1 && !s2) {
                ended = true;   // both texts consumed to the last byte in the same round
                return true;
            }
            if (!s1 || !s2) {
                // one text has run out of chunks while the other has not: the host readers decide what that means
                // (process_data.hpp:284-285 raises "different number of reads" unless the rest is empty)
                handover_pending_ = true;
                continue;
            }
            DeviceIngest::pair(ctx_, *ingest_[0], *ingest_[1]);
            const bool m1 = ingest_[0]->complete(res1), m2 = ingest_[1]->complete(res2);
            more = m1 || m2;
            if (res1.n != res2.n) throw Error("internal error: the paired device readers disagree on the number of records");
            if (res2.handover) res1.handover = true;
        }
        if (res1.handover) handover_pending_ = true;
        if (res1.n > 0) {
            out = Batch();
            out.first_read = consumed_;
            out.n = res1.n;
            out.reads1 = res1.reads;
            out.odd1 = res1.odd;
            if (paired) out.reads2 = res2.reads;
            out.slot = nullptr;
            consumed_ += res1.n;
            ctx_.timing.reads += res1.n;
            return true;
        }
        if (!more && !handover_pending_) {
            ended = true;
            return true;
        }
    }
}

bool ReadPipeline::next(Batch& out) {
    if (ingest_[0]) {
        bool ended = false;
        if (next_device(out, ended)) return !ended;
    }
    // refill the record windows
    if (cur1_ >= n1_) {
        const auto& b = r1_->next(kMaxBatchReads);
        recs1_ = b.data();
        n1_ = b.size();
        cur1_ = 0;
    }
    if (r2_ && cur2_ >= n2_) {
        const auto& b = r2_->next(kMaxBatchReads);
        recs2_ = b.data();
        n2_ = b.size();
        cur2_ = 0;
    }
    size_t avail = n1_ - cur1_;
    if (r2_) {
        const size_t avail2 = n2_ - cur2_;
        // process_data.hpp:284-285: both files must run out together
        if ((avail == 0) != (avail2 == 0)) throw Error("different number of reads in paired FASTQ files");
        avail = std::min(avail, avail2);
    }
    if (avail == 0) return false;

    // bound the staging buffers: at most kMaxBatchBytes of packed data per mate
    size_t count = avail;
    {
        // the reader already knows the longest read of what it handed out
        uint32_t maxlen = std::max<uint32_t>(1, r1_->batch_max_len());
        if (r2_) maxlen = std::max(maxlen, r2_->batch_max_len());
        const size_t probe = std::min<size_t>(avail, kMaxBatchReads);
        const size_t per_read = (size_t)12 * ceil_div((int)maxlen, 32);
        count = std::max<size_t>(TILE, std::min(probe, kMaxBatchBytes / per_read / TILE * TILE));
        count = std::min(count, avail);
    }
    // exact shortest / longest read of this batch: the reader's figures when the batch is everything it returned
    auto extent = [&](FastqReader* r, const Record* recs, size_t cur, size_t n_all, uint32_t& lo, uint32_t& hi) {
        if (cur == 0 && count == n_all) {
            lo = r->batch_min_len();
            hi = r->batch_max_len();
            return;
        }
        lo = 0xFFFFFFFFu;
        hi = 0;
        for (size_t i = 0; i < count; ++i) {
            lo = std::min(lo, recs[cur + i].len);
            hi = std::max(hi, recs[cur + i].len);
        }
    };
    uint32_t lo1 = 0, hi1 = 0, lo2 = 0, hi2 = 0;
    extent(r1_, recs1_, cur1_, n1_, lo1, hi1);
    if (r2_) extent(r2_, recs2_, cur2_, n2_, lo2, hi2);

    Slot& slot = slots_[next_slot_];
    next_slot_ = (next_slot_ + 1) % kSlots;
    if (slot.in_flight) {
        double t0 = now_s();
        SCG_CUDA_CHECK(cudaEventSynchronize(slot.done));  // the kernel that read this slot has finished
        ctx_.timing.device_s += now_s() - t0;
        slot.in_flight = false;
    }
    stage(slot, 0, recs1_ + cur1_, count, lo1, hi1);
    if (r2_) stage(slot, 1, recs2_ + cur2_, count, lo2, hi2);
    out.first_read = consumed_;
    out.n = (long long)count;
    out.reads1 = slot.mate[0].dev.view;
    out.odd1 = want_odd_ ? slot.mate[0].dev.odd.as<uint8_t>() : nullptr;
    out.recs1 = recs1_ + cur1_;
    if (r2_) out.reads2 = slot.mate[1].dev.view;
    out.slot = &slot;
    cur1_ += count;
    if (r2_) cur2_ += count;
    consumed_ += (long long)count;
    ctx_.timing.reads += (long long)count;
    return true;
}

void ReadPipeline::submitted(Batch& b) {
    if (!b.slot) return;   // device reader: its buffers are recycled in stream order
    Slot* slot = static_cast<Slot*>(b.slot);
    SCG_CUDA_CHECK(cudaEventRecord(slot->done, ctx_.stream));
    slot->in_flight = true;
}

} // namespace scg
