// FASTQ ingestion on the device (SURVEY 8 row f2): the raw text goes to HBM in fixed chunks over the copy engine
// (straight from the caller's buffer when it is page-locked, through a ring of pinned bounce buffers otherwise) and
// kernels find the newlines, check the records and pack the bases -- the work kaori::FastqReader does one byte at a
// time on the main thread (inst/include/kaori/FastqReader.hpp:42-110).
//
// The kernels accept exactly the FOUR-LINE records for which a line-oriented split provably equals the reference's
// character-by-character parse (the proof is in ingest.cu); anything else -- wrapped sequences or qualities, a '+'
// inside a sequence line, a malformed or truncated record, a record longer than the carry area -- stops the device
// reader at the last record boundary it is sure of, and the host reader (fastq.cpp: the full grammar, the
// reference's error texts and line numbers) resumes from that byte.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>
#include <string>
#include <vector>

#include "bgzf.hpp"
#include "engine.hpp"

namespace scg {

struct IngestState;   // device-side cursor shared by the kernels of consecutive chunks

struct IngestBuffers;

class DeviceIngest {
public:
    static constexpr size_t kChunk = 32u << 20;     // text bytes per H2D copy (SCG_INGEST_CHUNK overrides, for tests)
    static constexpr size_t kBgzfChunk = 128u << 20; // text bytes per chunk of a block-gzip input (2056 members of 64 KiB: one warp each)
    static constexpr size_t kCarry = 1u << 20;      // room in front of every chunk for the unfinished tail of the previous one (SCG_INGEST_CARRY)
    static constexpr int kSlots = 3;                // chunks in flight (copying, being parsed, being consumed)
    // Block-gzip input: a chunk's members are inflated by one warp each and a warp is slow (Huffman decoding is serial), so the
    // inflater needs thousands of members in flight: chunks are issued further ahead (SCG_BGZF_SLOTS) and their kernels run
    // side by side on several streams.
    static constexpr int kBgzfSlots = 12;
    static constexpr int kMaxSlots = 12;
    static constexpr int kCopyStreams = 12;

    struct Result {
        bool handover = false;      // the device reader stops here: resume the host reader at `resume_offset`
        size_t resume_offset = 0;   // byte offset into the text of the first record not consumed
        long long n = 0;            // records of this batch (0 with handover or at the end of the input)
        ReadsDev reads;             // packed batch, valid until the next call's kernels are enqueued
        const uint8_t* odd = nullptr;   // device flags (when asked for): the read holds characters other than ACGTN
    };

    // `mate` selects the context's buffer set (0, or 1 for the second file of paired input); `want_odd` makes the pack
    // kernel flag reads that hold anything but upper-case A, C, G, T, N.
    DeviceIngest(Context& ctx, const char* text, size_t size, int nthreads, int mate, bool want_odd);
    // The same over a block-gzip image (bgzf.hpp): the COMPRESSED members cross PCIe, chunk by chunk (a chunk = a run of whole
    // members), and are inflated on the device (inflate.cuh) straight into the text ring; everything after that is the same.
    // A member the device cannot inflate (or whose CRC does not match) stops the device reader before that chunk and the
    // host reader, which raises the error, takes over.
    // [text_begin, text_end): the part of the text to read (both ends record boundaries; (size_t)-1 = up to the end of the text) --
    // one device's share of a file that several devices read.
    DeviceIngest(Context& ctx, const BgzfIndex* image, int nthreads, int mate, bool want_odd, size_t text_begin = 0,
                 size_t text_end = (size_t)-1);
    ~DeviceIngest();

    // Parses the next chunk.  false = the text is exhausted (and `out.n` is 0).  Same as stage() + complete().
    bool next(Result& out);
    // The two halves, for paired input: stage() enqueues the line and record kernels of the next chunk (false = no chunk
    // left), pair() makes two staged mates agree on the number of records of the round, complete() settles the chunk.
    bool stage();
    static void pair(Context& ctx, DeviceIngest& a, DeviceIngest& b);
    bool complete(Result& out);

    long long records() const { return records_; }
    size_t consumed() const { return consumed_; }
    bool exhausted() const { return stopped_ || parsed_ >= nchunks(); }

    // Raw text of read `index` of the batch handed out last (single-line records).
    void raw_read(long long index, std::string& seq);

private:
    void setup(bool source_pinned);
    void issue_copy(size_t chunk);
    void issue_inflate(size_t chunk);
    void fetch_text(size_t offset, size_t len, std::string& out);
    size_t nchunks() const { return chunk_begin_.size() - 1; }
    size_t chunk_bytes(size_t k) const { return chunk_begin_[k + 1] - chunk_begin_[k]; }
    size_t slot_base(size_t chunk) const { return (chunk % (size_t)slots_) * stride_; }
    IngestBuffers& buffers() const;

    int slots_ = kSlots;
    size_t chunk_ = kChunk, carry_ = kCarry;
    size_t stride_ = 0;      // carry + chunk + 256 (room for an appended newline; keeps slot bases 16-byte aligned)
    size_t line_cap_ = 0;    // newline positions kept per chunk

    std::vector<size_t> chunk_begin_;   // text offset where each chunk starts, and the text's size at the end

    // block-gzip input
    const BgzfIndex* bgzf_ = nullptr;
    std::vector<size_t> chunk_block_;   // first member of each chunk, and the number of members at the end
    size_t skip_front_ = 0;             // text bytes of the first member that precede the part being read
    size_t max_comp_ = 0;               // most compressed bytes any chunk holds
    size_t max_members_ = 0;
    std::vector<char> block_cache_;     // host-inflated member for raw_read()
    size_t block_cached_ = (size_t)-1;

    Context& ctx_;
    const char* text_;
    size_t size_;
    int nthreads_;
    int mate_ = 0;
    bool want_odd_ = false;
    bool pinned_source_ = false;
    bool virtual_newline_ = false;   // the text does not end with '\n': one is appended on the device
    size_t issued_ = 0;              // chunks whose copy has been enqueued
    size_t parsed_ = 0;              // chunks handed out
    size_t consumed_ = 0;            // text bytes consumed as complete records so far
    long long records_ = 0;
    bool stopped_ = false;
    bool staged_ = false;
    int out_slot_ = 0;
    // the batch handed out last, for raw_read()
    long long last_n_ = 0;
    long long last_text_base_ = 0;   // text offset of ring position 0 of the batch's slot
    std::vector<uint32_t> last_off_;
    std::vector<uint16_t> last_len_;
    int last_out_slot_ = 0;
};

// Device-ingest resources owned by the context (kept across calls).
struct IngestBuffers {
    DeviceBuffer text;         // kSlots x (kCarry + kChunk) bytes
    DeviceBuffer lines;        // newline positions of the chunk being parsed
    DeviceBuffer block_counts; // newlines per block
    DeviceBuffer seq_off, seq_len;
    DeviceBuffer state;        // IngestState
    DeviceBuffer packed[2], lens[2], odd[2];
    PinnedBuffer bounce[DeviceIngest::kMaxSlots];
    PinnedBuffer meta;
    // block-gzip input: the compressed members of the chunk in each slot, their table, the inflate kernels' error word
    DeviceBuffer comp[DeviceIngest::kMaxSlots], members[DeviceIngest::kMaxSlots], inflate_errors;
    PinnedBuffer members_host[DeviceIngest::kMaxSlots];
    cudaStream_t copy_stream = nullptr;                                  // = copy_streams[0]
    cudaStream_t copy_streams[DeviceIngest::kCopyStreams] = {};          // block-gzip chunks take them in turn
    cudaEvent_t copied[DeviceIngest::kMaxSlots] = {};     // chunk text is in HBM
    cudaEvent_t bounced[DeviceIngest::kMaxSlots] = {};    // bounce buffer may be refilled
    cudaEvent_t released[DeviceIngest::kMaxSlots] = {};   // the parse no longer needs the slot's text
    cudaEvent_t meta_ready = nullptr;
    bool released_valid[DeviceIngest::kMaxSlots] = {};
    bool bounced_valid[DeviceIngest::kMaxSlots] = {};
    ~IngestBuffers();
    void ensure(size_t chunk, size_t carry, size_t bounce_bytes, int slots);
    void ensure_bgzf(size_t comp_bytes, size_t nmembers, int slots);
};

// false when the device reader is switched off (environment SCG_HOST_PARSE=1): every input then takes the host parser.
bool device_ingest_enabled();
// false when block-gzip members are to be inflated by host threads (environment SCG_BGZF_HOST=1) and parsed there.
bool device_inflate_enabled();

} // namespace scg
