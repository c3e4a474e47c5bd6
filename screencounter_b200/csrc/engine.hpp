// Host-side runtime: context (device, stream, pinned staging), device images of libraries and
// reads, and the FASTQ -> pinned -> HBM -> kernel pipeline.  This is what replaces the
// reference's block driver and thread pool (inst/include/kaori/process_data.hpp:105-340).
#pragma once

#include <cuda_runtime.h>

#include <memory>
#include <string>
#include <vector>

#include "common.hpp"
#include "fastq.hpp"
#include "handlers_params.hpp"
#include "library.hpp"
#include "template_spec.hpp"

namespace scg {

struct DeviceBuffer {
    void* ptr = nullptr;
    size_t bytes = 0;
    int device = 0;   // the CUDA device the block was allocated on (release() returns it there)
    DeviceBuffer() {}
    DeviceBuffer(const DeviceBuffer&) = delete;
    DeviceBuffer& operator=(const DeviceBuffer&) = delete;
    DeviceBuffer(DeviceBuffer&& o) noexcept : ptr(o.ptr), bytes(o.bytes), device(o.device) { o.ptr = nullptr; o.bytes = 0; }
    DeviceBuffer& operator=(DeviceBuffer&& o) noexcept {
        if (this != &o) {
            release();
            ptr = o.ptr;
            bytes = o.bytes;
            device = o.device;
            o.ptr = nullptr;
            o.bytes = 0;
        }
        return *this;
    }
    ~DeviceBuffer() { release(); }
    void alloc(size_t n, bool zero);
    void reserve(size_t n);  // grow-only, contents not preserved
    void upload(const void* host, size_t n, cudaStream_t stream);
    void release();
    template <class T> T* as() const { return static_cast<T*>(ptr); }
};

struct PinnedBuffer {
    void* ptr = nullptr;
    size_t bytes = 0;
    ~PinnedBuffer();
    void reserve(size_t n);
    template <class T> T* as() const { return static_cast<T*>(ptr); }
};

struct Timing {
    double parse_s = 0, pack_s = 0, h2d_s = 0, device_s = 0, total_s = 0;
    double harvest_s = 0; // variable-size results (combination / random-barcode tables) sorted, downloaded and rendered
    double setup_s = 0;   // library tables built + uploaded, kernels specialised (zero when the context had them cached)
    double merge_s = 0;   // a call cut over several devices: the parts' results merged on the first device
    long long reads = 0, bytes_h2d = 0, launches = 0;
    std::string reader = "host";   // which FASTQ reader fed the call: the host parser/packer or the device one (ingest.hpp)
};

// A library resident on the device.
struct DeviceLibrary {
    Library host;
    DeviceBuffer slots, ent_keys, ent_idx, seed_masks, buckets, cands, cand_rows, prefix_slots, trie, ibuckets;
    LibDev dev;
    void upload(struct Context& ctx);
};

// Packed reads of one batch resident on the device.
struct DeviceBatch {
    DeviceBuffer data, lens, odd;
    ReadsDev view;
};

// One slot of the FASTQ -> pinned -> HBM double buffer (pipeline.hpp).  The slots belong to the context so that
// consecutive calls (one per file in matrixOf*-style loops) reuse the pinned and device allocations.
struct Staged {
    PinnedBuffer pinned_data, pinned_lens;
    std::vector<uint8_t> odd_host;
    DeviceBatch dev;
};
struct StagingSlot {
    Staged mate[2];
    cudaEvent_t done = nullptr;
    bool in_flight = false;
};

struct SingleMatcher;
struct IngestBuffers;   // ingest.hpp

struct Context {
    static constexpr int kStagingSlots = 2;
    StagingSlot staging[kStagingSlots];
    // single-barcode matchers (template + both strands' tables on the device) of recent calls, keyed by a
    // 128-bit hash of everything that defines them
    struct CachedMatcher {
        unsigned long long key1 = 0, key2 = 0;
        int npool = 0;                               // secondary check of a cache hit, beside the 128-bit hash
        std::string constant, first_seq, last_seq;
        std::shared_ptr<SingleMatcher> matcher;
    };
    std::vector<CachedMatcher> single_cache;
    // matchers of the other handlers (any type behind the pointer; the key's first word names it), most recent last
    struct CachedObject {
        unsigned long long key1 = 0, key2 = 0;
        unsigned long long fed_bytes = 0;            // secondary check: total bytes hashed into the key
        std::shared_ptr<void> object;
    };
    std::vector<CachedObject> matcher_cache;
    // Scratch of the specialised kernels, shared by every launch on this context: a context serves ONE stream at a time.
    DeviceBuffer slow_list, slow_count;      // reads a specialised kernel hands to its full-search follow-up (spec_single.cuh, spec_handlers.cuh)
    DeviceBuffer defer_words, defer_counts;  // per-warp regions of deferred lookups (libdev.hpp DeferredList)
    DeviceBuffer part_counts;                // keys per (table part, warp) of a partitioned random-barcode launch (libdev.hpp PartitionedKeys)
    DeviceBuffer part_keys;                  // ... and the lists themselves
    std::shared_ptr<IngestBuffers> ingest[2];   // text ring, line tables and streams of the device-side FASTQ reader, per mate
    int device = 0;
    bool ready = false;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    std::string last_error;
    std::string timing_json;
    std::string kernel_note;   // which kernel variant the last launch used
    Timing timing;
    long long launches = 0;

    explicit Context(int dev) : device(dev) {}
    ~Context();
    void ensure_ready();   // lazy CUDA initialisation; throws when no usable device exists
    int grid_for(long long ntiles) const;
    void finish_timing();
};

} // namespace scg

// Opaque C-ABI types.
struct scg_ctx {
    scg::Context impl;
    // scg_ctx_create_multi: the contexts of the other devices.  `impl` is the first device's; file-level calls split a file
    // (or deal the files of a many-files call) over impl and these, one host thread per device.
    std::vector<std::unique_ptr<scg_ctx>> peers;
    explicit scg_ctx(int dev) : impl(dev) {}
};

struct scg_reads {
    scg_ctx* owner = nullptr;
    std::vector<scg::DeviceBatch> batches;
    long long n = 0;
    long long device_bytes = 0;
};

struct scg_result {
    int width = 0;
    std::vector<int32_t> keys;
    std::vector<char> strings;
    std::vector<int32_t> freq;
    int trace_width = 0;
    std::vector<int32_t> trace_index;
    std::vector<uint32_t> trace_info;
    // A table may instead stay ON THE DEVICE, sorted and rendered in its final form, until scg_result_copy_table copies it
    // straight into the caller's arrays: one device-to-host copy, no intermediate host image.
    bool on_device = false;
    int device = 0;
    size_t d_rows = 0;
    scg::DeviceBuffer d_keys, d_strings, d_freq;
    // many-files calls: one column of counts per file over the rows of the table (column-major, like an R matrix)
    int columns = 0;
    std::vector<int32_t> matrix;
    scg::DeviceBuffer d_matrix;
    size_t rows() const { return on_device ? d_rows : freq.size(); }
};
