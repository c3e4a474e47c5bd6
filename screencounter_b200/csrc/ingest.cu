// Device-side FASTQ reader: see ingest.hpp.
//
// WHY A LINE SPLIT IS ENOUGH FOR FOUR-LINE RECORDS.  kaori::FastqReader::operator() (FastqReader.hpp:42-110) reads,
// from a record start: '@' (else it throws), the rest of that line; then every character up to the first '+'
// ANYWHERE, dropping newlines, as the sequence (:70-78); the rest of the '+' line (:81-85); then characters until a
// newline at which at least as many quality characters as bases have been seen (:91-105), the two counts having to be
// equal.  Number the lines of the text from a record start as L0 L1 L2 L3.  If (a) L0 starts with '@', (b) L1 holds no
// '+', (c) L2 starts with '+' and (d) |L3| = |L1|, the reference's walk consumes exactly L0, takes L1 as the sequence
// (its first '+' is L2's first character), consumes L2, and stops at the newline that ends L3 because |L3| >= |L1|
// there and not before (there is no earlier newline): the next record starts at the next line.  By induction a text
// whose every group of four lines satisfies (a)-(d) is parsed by the reference into exactly those groups -- including
// '\r' before the newlines (kept as a base, SURVEY 8.1 T13), empty sequences, and a last line without newline.
// `validate_records` checks (a)-(d) per group; the first group that fails ends the device reader's part of the text.
#include "ingest.hpp"

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>

#include "hostpool.hpp"
#include "inflate.cuh"
#include "layout.hpp"

namespace scg {

namespace {

double now_s() {
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

constexpr int kBlockThreads = 256;
constexpr int kBytesPerThread = 16;
constexpr uint32_t kBlockBytes = kBlockThreads * kBytesPerThread;   // 4096

enum : uint32_t {
    ST_LINECAP = 1u,    // more lines than the position buffer holds
    ST_BADREC = 2u,     // a group of four lines is not a four-line record
    ST_REMAINDER = 4u,  // the last chunk does not end on a record boundary
    ST_CARRY = 8u,      // the unfinished tail does not fit the carry area
};

} // namespace

struct IngestState {
    uint32_t begin;      // ring position of the first unconsumed text byte of the chunk about to be parsed
    uint32_t nlines;     // complete lines in [begin, end), capped at the position buffer's size
    uint32_t nrec;       // records accepted from this chunk
    uint32_t bad_rec;    // lowest group of four lines that failed the record checks (>= nrec: none)
    uint32_t min_len, max_len;
    uint32_t status;     // ST_* flags: the device reader stops after this chunk
    uint32_t tail;       // ring position just past the last accepted record
    uint32_t limit;      // paired input: records the other mate can match in this round (0xFFFFFFFF = no limit)
};

namespace {

// ---- kernels ---------------------------------------------------------------------------------------------------

__global__ void ingest_init(IngestState* st, uint32_t begin) {
    st->begin = begin;
    st->nlines = st->nrec = st->bad_rec = 0;
    st->min_len = 0xFFFFFFFFu;
    st->max_len = 0;
    st->status = 0;
    st->tail = begin;
    st->limit = 0xFFFFFFFFu;
}

// newlines among the 16 bytes at ring position p that lie in [begin, end): bit j of the result = byte j is one
__device__ __forceinline__ uint32_t newline_mask(const uint4 v, uint32_t p, uint32_t begin, uint32_t end) {
    const uint32_t w[4] = { v.x, v.y, v.z, v.w };
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t x = w[k] ^ 0x0A0A0A0Au;
        // exact zero-byte detector: 0x80 in every byte of x that is zero
        const uint32_t z = ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x | 0x7F7F7F7Fu);
        m |= (((z >> 7) & 1u) | ((z >> 14) & 2u) | ((z >> 21) & 4u) | ((z >> 28) & 8u)) << (4 * k);
    }
    // clip to [begin, end)
    if (p < begin) m &= (begin - p >= 16) ? 0u : (0xFFFFu << (begin - p));
    if (p + 16 > end) m &= (p >= end) ? 0u : ((1u << (end - p)) - 1u);
    return m & 0xFFFFu;
}

// pass 1: newlines per 4 KiB block of the slot
__global__ void __launch_bounds__(kBlockThreads) count_newlines(const uint8_t* __restrict__ ring, uint32_t slot0, uint32_t end,
                                                                const IngestState* __restrict__ st, uint32_t* __restrict__ block_counts) {
    const uint32_t begin = st->begin;
    const uint32_t bpos = slot0 + blockIdx.x * kBlockBytes;
    __shared__ uint32_t warp_sums[kBlockThreads / 32];
    uint32_t c = 0;
    if (bpos + kBlockBytes > begin && bpos < end) {
        const uint32_t p = bpos + threadIdx.x * kBytesPerThread;
        const uint4 v = *reinterpret_cast<const uint4*>(ring + p);
        c = __popc(newline_mask(v, p, begin, end));
    }
    c = __reduce_add_sync(0xFFFFFFFFu, c);
    if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
#pragma unroll
        for (int k = 0; k < kBlockThreads / 32; ++k) t += warp_sums[k];
        block_counts[blockIdx.x] = t;
    }
}

// pass 2: exclusive scan of the block counts (one block), number of lines and of candidate records
__global__ void __launch_bounds__(1024) scan_blocks(uint32_t* __restrict__ block_counts, int nblocks, IngestState* st, uint32_t line_cap) {
    __shared__ uint32_t warp_tot[32];
    __shared__ uint32_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int base = 0; base < nblocks; base += 1024) {
        const int i = base + threadIdx.x;
        const uint32_t v = i < nblocks ? block_counts[i] : 0u;
        uint32_t x = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, d);
            if (lane >= d) x += y;
        }
        if (lane == 31) warp_tot[wid] = x;
        __syncthreads();
        if (wid == 0) {
            uint32_t t = warp_tot[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, t, d);
                if (lane >= d) t += y;
            }
            warp_tot[lane] = t;   // inclusive totals of the warps
        }
        __syncthreads();
        const uint32_t before = carry + (wid ? warp_tot[wid - 1] : 0u) + (x - v);
        if (i < nblocks) block_counts[i] = before;
        __syncthreads();
        if (threadIdx.x == 0) carry += warp_tot[31];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        uint32_t lines = carry, status = 0;
        if (lines > line_cap) {
            lines = line_cap;
            status |= ST_LINECAP;
        }
        st->nlines = lines;
        st->nrec = lines / 4;
        st->bad_rec = lines / 4;
        st->min_len = 0xFFFFFFFFu;
        st->max_len = 0;
        st->status = status;
        st->limit = 0xFFFFFFFFu;
    }
}

// pass 3: positions of the newlines, in text order
__global__ void __launch_bounds__(kBlockThreads) scatter_newlines(const uint8_t* __restrict__ ring, uint32_t slot0, uint32_t end,
                                                                  const IngestState* __restrict__ st, const uint32_t* __restrict__ block_offsets,
                                                                  uint32_t* __restrict__ lines, uint32_t line_cap) {
    const uint32_t begin = st->begin;
    const uint32_t bpos = slot0 + blockIdx.x * kBlockBytes;
    if (!(bpos + kBlockBytes > begin && bpos < end)) return;   // block-uniform
    __shared__ uint32_t warp_sums[kBlockThreads / 32];
    const uint32_t p = bpos + threadIdx.x * kBytesPerThread;
    const uint4 v = *reinterpret_cast<const uint4*>(ring + p);
    uint32_t m = newline_mask(v, p, begin, end);
    const uint32_t c = __popc(m);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t x = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    uint32_t at = block_offsets[blockIdx.x] + (x - c);
    for (int k = 0; k < wid; ++k) at += warp_sums[k];
    while (m) {
        const int j = __ffs(m) - 1;
        m &= m - 1;
        if (at < line_cap) lines[at] = p + j;
        ++at;
    }
}

// pass 4: conditions (a)-(d) for every group of four lines; sequence offsets and lengths; shortest and longest sequence among
// the groups that are records (a superset of the records finish_chunk accepts when one of them fails: the batch is then
// treated as ragged at worst, never wrongly as uniform)
__global__ void __launch_bounds__(256) validate_records(const uint8_t* __restrict__ ring, const uint32_t* __restrict__ lines, IngestState* st,
                                                        uint32_t* __restrict__ seq_off, uint16_t* __restrict__ seq_len) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = r < st->nrec;
    bool ok = false;
    uint32_t len = 0;
    if (active) {
        const uint32_t e0 = lines[4 * r], e1 = lines[4 * r + 1], e2 = lines[4 * r + 2], e3 = lines[4 * r + 3];
        const uint32_t start = r ? lines[4 * r - 1] + 1 : st->begin;
        const uint32_t s = e0 + 1, qlen = e3 - (e2 + 1);
        len = e1 - s;
        ok = ring[start] == '@' && ring[e1 + 1] == '+' && qlen == len && len <= (uint32_t)MAX_READ_LEN;
        if (ok && len) {
            // a '+' anywhere in the sequence line: four bytes at a time over the aligned words that hold it, the bytes in front of
            // and behind the line made harmless first (the zero-byte test is exact for "does any byte match")
            const uint32_t lead = s & 3u, nwords = (lead + len + 3u) / 4u;
            const uint32_t* __restrict__ w = reinterpret_cast<const uint32_t*>(ring + (s - lead));
            uint32_t found = 0;
            for (uint32_t k = 0; k < nwords; ++k) {
                uint32_t v = w[k];
                if (k == 0 && lead) v |= (1u << (8u * lead)) - 1u;
                const uint32_t upto = lead + len - 4u * k;   // bytes of this word that belong to the line (>= 1)
                if (upto < 4u) v |= 0xFFFFFFFFu << (8u * upto);
                const uint32_t t = v ^ 0x2B2B2B2Bu;
                found |= (t - 0x01010101u) & ~t & 0x80808080u;
            }
            ok = found == 0;
        }
        seq_off[r] = s;
        seq_len[r] = (uint16_t)(ok ? len : 0u);
        if (!ok) atomicMin(&st->bad_rec, r);
    }
    const uint32_t lo = __reduce_min_sync(0xFFFFFFFFu, ok ? len : 0xFFFFFFFFu);
    const uint32_t hi = __reduce_max_sync(0xFFFFFFFFu, ok ? len : 0u);
    if ((threadIdx.x & 31) == 0 && lo != 0xFFFFFFFFu) {
        atomicMin(&st->min_len, lo);
        atomicMax(&st->max_len, hi);
    }
}

// paired input: both mates accept the same number of records in a round; what one has in excess stays in its carry
__global__ void pair_limit(IngestState* a, IngestState* b) {
    const uint32_t n = min(min(a->nrec, a->bad_rec), min(b->nrec, b->bad_rec));
    a->limit = n;
    b->limit = n;
}

// pass 6 (one block): settles what this chunk contributes, moves the unfinished tail in front of the next slot
__global__ void __launch_bounds__(1024) finish_chunk(uint8_t* __restrict__ ring, const uint32_t* __restrict__ lines, IngestState* st, uint32_t end,
                                                     int final_chunk, uint32_t next_data0, uint32_t carry_room) {
    __shared__ uint32_t s_tail, s_len, s_copy;
    if (threadIdx.x == 0) {
        uint32_t status = st->status;
        uint32_t n = st->nrec;
        if (st->bad_rec < n) {
            n = st->bad_rec;
            status |= ST_BADREC;
        }
        if (st->limit < n) {
            // the other mate has fewer records this round: the rest waits in the carry (not an irregularity, and a bad
            // record beyond the limit is next round's business)
            n = st->limit;
            status &= ~(ST_BADREC | ST_LINECAP);
        }
        const uint32_t tail = n ? lines[4 * n - 1] + 1 : st->begin;
        const uint32_t left = end - tail;
        if (final_chunk) {
            // paired input may leave records for a round that will not come: the host readers sort that out
            if (left) status |= ST_REMAINDER;
        } else if (left > carry_room) {
            status |= ST_CARRY;
        }
        st->nrec = n;
        st->tail = tail;
        st->status = status;
        s_tail = tail;
        s_len = left;
        s_copy = (!final_chunk && status == 0) ? 1u : 0u;
        if (s_copy) st->begin = next_data0 - left;
    }
    __syncthreads();
    if (!s_copy) return;
    const uint32_t tail = s_tail, left = s_len, dst = next_data0 - left;
    for (uint32_t k = threadIdx.x; k < left; k += blockDim.x) ring[dst + k] = ring[tail + k];
}

// pass 7: bases -> tile-planar bit planes (layout.hpp); one warp per tile, one lane per record
__global__ void __launch_bounds__(128) pack_records_dev(const uint8_t* __restrict__ ring, const uint32_t* __restrict__ seq_off,
                                                        uint16_t* __restrict__ seq_len, uint32_t nrec, int W, uint32_t* __restrict__ out,
                                                        uint8_t* __restrict__ odd) {
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t ntiles = (nrec + TILE - 1) / TILE;
    if (warp >= ntiles) return;
    const uint32_t r = warp * TILE + lane;
    uint32_t len = 0;
    const uint8_t* s = ring;
    if (r < nrec) {
        len = seq_len[r];
        s = ring + seq_off[r];
    } else {
        seq_len[r] = 0;   // the length array is padded to whole tiles like the host packer's
    }
    uint32_t* base = out + (size_t)warp * 3 * W * TILE + lane;
    // Four bases per step: the sequence is read as the aligned 32-bit words that hold it (funnel-shifted into place), the
    // per-byte tests run on all four bytes of a word at once, and a multiply gathers one bit per byte into four adjacent bits.
    const uint32_t lead = (uint32_t)(reinterpret_cast<size_t>(s) & 3u);
    const uint32_t* __restrict__ aligned = reinterpret_cast<const uint32_t*>(s - lead);
    const uint32_t shift = 8u * lead;
    uint32_t not_plain = 0;   // bytes that are not upper-case A, C, G, T or N (what the random-barcode handler cannot render)
    uint32_t lo = aligned[0];
    for (int w = 0; w < W; ++w) {
        uint32_t hh = 0, ll = 0, nn = 0;
        const int first = 32 * w;
        const int cnt = (int)len > first ? min(32, (int)len - first) : 0;
        for (int j = 0; j < cnt; j += 4) {
            const uint32_t hi = aligned[(first + j) / 4 + 1];
            const uint32_t v = shift ? __funnelshift_r(lo, hi, shift) : lo;   // bases first + j .. first + j + 3
            lo = hi;
            const uint32_t keep = cnt - j >= 4 ? 0xFFFFFFFFu : ((1u << (8u * (uint32_t)(cnt - j))) - 1u);
            const uint32_t u = v & 0xDFDFDFDFu;   // fold case
            // byte == K, exactly, for all four bytes: high bit of (((t & 0x7f..) + 0x7f..) | t) is set iff the byte of t is non-zero
            auto equals = [](uint32_t x, uint32_t k) {
                const uint32_t t = x ^ (k * 0x01010101u);
                return ~(((t & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | t) & 0x80808080u;
            };
            const uint32_t acgt = equals(u, 'A') | equals(u, 'C') | equals(u, 'G') | equals(u, 'T');   // 0x80 per valid byte
            const uint32_t valid = (acgt >> 7) & keep;                                                 // 0x01 per valid byte
            if (odd) {
                const uint32_t upper = equals(v, 'A') | equals(v, 'C') | equals(v, 'G') | equals(v, 'T') | equals(v, 'N');
                not_plain |= ~(upper >> 7) & 0x01010101u & keep;
            }
            // ASCII: bit 2 of A/C/G/T (either case) is 0/0/1/1 = plane H, bit 1 is 0/1/1/0, so L = bit 1 ^ bit 2
            const uint32_t hb = (v >> 2) & valid, lb = ((v >> 1) ^ (v >> 2)) & valid, nb = ~valid & 0x01010101u & keep;
            hh |= ((hb * 0x01020408u) >> 24) << j;
            ll |= ((lb * 0x01020408u) >> 24) << j;
            nn |= ((nb * 0x01020408u) >> 24) << j;
        }
        base[(size_t)(PLANE_H * W + w) * TILE] = hh;
        base[(size_t)(PLANE_L * W + w) * TILE] = ll;
        base[(size_t)(PLANE_N * W + w) * TILE] = nn;
    }
    const bool plain = not_plain == 0;
    if (odd) odd[r] = plain ? 0 : 1;
}

} // namespace

// ---- host side -------------------------------------------------------------------------------------------------

bool device_ingest_enabled() {
    const char* v = std::getenv("SCG_HOST_PARSE");
    return !(v && *v && *v != '0');
}

IngestBuffers::~IngestBuffers() {
    for (int k = 0; k < DeviceIngest::kMaxSlots; ++k) {
        if (copied[k]) cudaEventDestroy(copied[k]);
        if (bounced[k]) cudaEventDestroy(bounced[k]);
        if (released[k]) cudaEventDestroy(released[k]);
    }
    if (meta_ready) cudaEventDestroy(meta_ready);
    for (cudaStream_t st : copy_streams) {
        if (st) cudaStreamDestroy(st);
    }
}

bool device_inflate_enabled() {
    const char* v = std::getenv("SCG_BGZF_HOST");
    return !(v && *v && *v != '0');
}

void IngestBuffers::ensure_bgzf(size_t comp_bytes, size_t nmembers, int slots) {
    for (int k = 0; k < slots; ++k) {
        comp[k].reserve(comp_bytes + 1024);   // the inflate kernel's readers fetch whole lines ahead
        members[k].reserve(std::max<size_t>(nmembers, 1) * sizeof(InflateMember));
        members_host[k].reserve(std::max<size_t>(nmembers, 1) * sizeof(InflateMember));
    }
    inflate_errors.reserve(16);
}

void IngestBuffers::ensure(size_t chunk, size_t carry, size_t bounce_bytes, int slots) {
    const size_t stride = carry + chunk + 256, line_cap = (carry + chunk) / 4;
    if (!copy_stream) {
        for (cudaStream_t& st : copy_streams) SCG_CUDA_CHECK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        copy_stream = copy_streams[0];
        for (int k = 0; k < DeviceIngest::kMaxSlots; ++k) {
            SCG_CUDA_CHECK(cudaEventCreateWithFlags(&copied[k], cudaEventDisableTiming));
            SCG_CUDA_CHECK(cudaEventCreateWithFlags(&bounced[k], cudaEventDisableTiming));
            SCG_CUDA_CHECK(cudaEventCreateWithFlags(&released[k], cudaEventDisableTiming));
        }
        SCG_CUDA_CHECK(cudaEventCreateWithFlags(&meta_ready, cudaEventDisableTiming));
    }
    text.reserve((size_t)slots * stride + 2 * kBlockBytes);
    lines.reserve((line_cap + 4) * sizeof(uint32_t));
    block_counts.reserve((stride / kBlockBytes + 2) * sizeof(uint32_t));
    seq_off.reserve((line_cap / 4 + 1) * sizeof(uint32_t));
    state.reserve(sizeof(IngestState));
    meta.reserve(sizeof(IngestState) + 16);
    for (int k = 0; k < 2; ++k) {
        lens[k].reserve((line_cap / 4 + TILE) * sizeof(uint16_t));
        odd[k].reserve(line_cap / 4 + TILE);
    }
    if (bounce_bytes) {
        for (int k = 0; k < slots; ++k) bounce[k].reserve(bounce_bytes);
    }
    for (int k = 0; k < DeviceIngest::kMaxSlots; ++k) released_valid[k] = bounced_valid[k] = false;
}

IngestBuffers& DeviceIngest::buffers() const { return *ctx_.ingest[mate_]; }

namespace {

bool page_locked(const void* first, const void* last) {
    // a page-locked source (scg_host_alloc, cudaHostRegister) feeds the copy engine directly
    cudaPointerAttributes a0, a1;
    const bool ok0 = cudaPointerGetAttributes(&a0, first) == cudaSuccess && a0.type == cudaMemoryTypeHost;
    const bool ok1 = ok0 && cudaPointerGetAttributes(&a1, last) == cudaSuccess && a1.type == cudaMemoryTypeHost;
    cudaGetLastError();   // an unregistered pointer may leave a sticky-free error behind on old drivers
    return ok0 && ok1;
}

size_t env_size(const char* name, size_t fallback, size_t lo, size_t hi) {
    const char* v = std::getenv(name);
    if (!v || !*v) return fallback;
    const long long x = std::atoll(v);
    return (size_t)std::min<long long>((long long)hi, std::max<long long>((long long)lo, x));
}

} // namespace

DeviceIngest::DeviceIngest(Context& ctx, const char* text, size_t size, int nthreads, int mate, bool want_odd)
    : ctx_(ctx), text_(text), size_(size), nthreads_(std::max(1, nthreads)), mate_(mate ? 1 : 0), want_odd_(want_odd) {
    ctx_.ensure_ready();
    virtual_newline_ = text_[size_ - 1] != '\n';
    // multiples of 16 keep the slots' data areas aligned for the 16-byte loads of the line kernels
    chunk_ = env_size("SCG_INGEST_CHUNK", kChunk, 64, 1u << 30) / 16 * 16;
    for (size_t at = 0; at < size_; at += chunk_) chunk_begin_.push_back(at);
    chunk_begin_.push_back(size_);
    setup(page_locked(text_, text_ + size_ - 1));
}

DeviceIngest::DeviceIngest(Context& ctx, const BgzfIndex* image, int nthreads, int mate, bool want_odd, size_t text_begin, size_t text_end)
    : bgzf_(image), ctx_(ctx), text_(nullptr), size_(std::min(text_end, image->text_size())), nthreads_(std::max(1, nthreads)),
      mate_(mate ? 1 : 0), want_odd_(want_odd) {
    ctx_.ensure_ready();
    text_begin = std::min(text_begin, size_);
    if (text_begin >= size_) throw Error("empty part of a block-gzip text");
    consumed_ = text_begin;
    // the part's last byte decides whether a newline has to be appended: the member that holds it, inflated here
    {
        std::string last;
        fetch_text(size_ - 1, 1, last);
        virtual_newline_ = last.empty() || last[0] != '\n';
    }
    // a chunk = a run of whole members holding at most chunk_ bytes of text (never less than one member can hold)
    // (cutting a small file into several chunks so that its parse starts while members still inflate was measured: slower, 6.4
    // against 4.5 ms for 157 MB of text -- a member takes 1.7 ms however few there are, and every chunk costs a host round trip)
    chunk_ = std::max<size_t>(env_size("SCG_INGEST_CHUNK", kBgzfChunk, 64, 1u << 30), 1u << 16) / 16 * 16;
    // the members that hold the part: from the one with its first byte to the one with its last
    size_t b = bgzf_->block_of(text_begin);
    const size_t nb = bgzf_->block_of(size_ - 1) + 1;
    skip_front_ = text_begin - bgzf_->text_off[b];
    while (b < nb) {
        const size_t first = b;
        size_t bytes = 0;
        while (b < nb && bytes + bgzf_->blocks[b].isize <= chunk_) bytes += bgzf_->blocks[b++].isize;
        chunk_begin_.push_back(bgzf_->text_off[first]);
        chunk_block_.push_back(first);
        const BgzfBlock& lastb = bgzf_->blocks[b - 1];
        max_comp_ = std::max(max_comp_, lastb.data + lastb.csize - bgzf_->blocks[first].data);
        max_members_ = std::max(max_members_, b - first);
    }
    chunk_begin_.push_back(size_);
    chunk_block_.push_back(nb);
    setup(page_locked(bgzf_->image, bgzf_->image + bgzf_->image_size - 1));
}

void DeviceIngest::setup(bool source_pinned) {
    pinned_source_ = source_pinned;
    carry_ = env_size("SCG_INGEST_CARRY", kCarry, 16, 64u << 20) / 16 * 16;
    stride_ = carry_ + chunk_ + 256;
    line_cap_ = (carry_ + chunk_) / 4;
    if (!ctx_.ingest[mate_]) ctx_.ingest[mate_].reset(new IngestBuffers);
    IngestBuffers& B = buffers();
    slots_ = bgzf_ ? (int)env_size("SCG_BGZF_SLOTS", kBgzfSlots, 2, kMaxSlots) : kSlots;
    if (bgzf_) slots_ = (int)std::max<size_t>(2, std::min<size_t>((size_t)slots_, nchunks() + 1));   // a small file does not need the whole ring
    B.ensure(chunk_, carry_, pinned_source_ ? 0 : (bgzf_ ? max_comp_ : chunk_), slots_);
    if (bgzf_) {
        B.ensure_bgzf(max_comp_, max_members_, slots_);
        SCG_CUDA_CHECK(cudaMemsetAsync(B.inflate_errors.ptr, 0, 16, B.copy_stream));
        SCG_CUDA_CHECK(cudaStreamSynchronize(B.copy_stream));   // (the chunks' kernels run on several streams)
    }
    ingest_init<<<1, 1, 0, ctx_.stream>>>(B.state.as<IngestState>(), (uint32_t)(slot_base(0) + carry_ + skip_front_));
    SCG_CUDA_CHECK(cudaGetLastError());
    ++ctx_.launches;
    ctx_.timing.reader = bgzf_ ? (pinned_source_ ? "device (block-gzip members copied from page-locked memory, inflated on the device)"
                                                 : "device (block-gzip members staged through pinned bounce buffers, inflated on the device)")
                               : (pinned_source_ ? "device (text copied from page-locked memory)" : "device (text staged through pinned bounce buffers)");
}

// text [offset, offset + len) of a block-gzip input, inflated on the host member by member (raw_read and the constructor)
void DeviceIngest::fetch_text(size_t offset, size_t len, std::string& out) {
    out.clear();
    while (len > 0) {
        const size_t b = bgzf_->block_of(offset);
        if (b >= bgzf_->blocks.size()) throw Error("raw_read: offset beyond the text");
        if (block_cached_ != b) {
            block_cache_.resize(std::max<size_t>(bgzf_->blocks[b].isize, 1));
            if (!bgzf_inflate_block(*bgzf_, b, block_cache_.data())) throw Error("failed to inflate the block-gzip file (corrupt member)");
            block_cached_ = b;
        }
        const size_t in_block = offset - bgzf_->text_off[b];
        const size_t take = std::min(len, (size_t)bgzf_->blocks[b].isize - in_block);
        if (take == 0) throw Error("raw_read: empty member");
        out.append(block_cache_.data() + in_block, take);
        offset += take;
        len -= take;
    }
}

DeviceIngest::~DeviceIngest() {
    // copies still in flight read the caller's text (or the bounce buffers): let them finish
    if (ctx_.ingest[mate_]) {
        for (cudaStream_t st : ctx_.ingest[mate_]->copy_streams) {
            if (st) cudaStreamSynchronize(st);
        }
    }
}

// block-gzip input: the chunk's members cross PCIe compressed and are inflated into the slot's data area
void DeviceIngest::issue_inflate(size_t chunk) {
    IngestBuffers& B = buffers();
    const int s = (int)(chunk % (size_t)slots_);
    cudaStream_t cs = B.copy_streams[chunk % kCopyStreams];
    const size_t fb = chunk_block_[chunk], lb = chunk_block_[chunk + 1];
    const size_t from = bgzf_->blocks[fb].data, bytes = bgzf_->blocks[lb - 1].data + bgzf_->blocks[lb - 1].csize - from;
    uint8_t* dst = B.text.as<uint8_t>() + slot_base(chunk) + carry_;
    if (B.released_valid[s]) SCG_CUDA_CHECK(cudaStreamWaitEvent(cs, B.released[s], 0));
    // the slot's host staging (member table, bounce buffer) is free once the copies of its previous chunk are done
    if (B.bounced_valid[s]) SCG_CUDA_CHECK(cudaEventSynchronize(B.bounced[s]));
    InflateMember* table = B.members_host[s].as<InflateMember>();
    for (size_t b = fb; b < lb; ++b) {
        const BgzfBlock& blk = bgzf_->blocks[b];
        table[b - fb] = InflateMember{ (uint32_t)(blk.data - from), blk.csize, (uint32_t)(bgzf_->text_off[b] - bgzf_->text_off[fb]), blk.isize, blk.crc };
    }
    const void* src = bgzf_->image + from;
    if (!pinned_source_) {
        const double t0 = now_s();
        char* bb = B.bounce[s].as<char>();
        const int pieces = (int)std::max<size_t>(1, std::min<size_t>((size_t)nthreads_, bytes >> 20));
        const size_t per = (bytes + pieces - 1) / pieces;
        const unsigned char* image = bgzf_->image;
        HostPool::instance().parallel_for(pieces, pieces, [&](int k) {
            const size_t b = (size_t)k * per, e = std::min(bytes, b + per);
            if (b < e) std::memcpy(bb + b, image + from + b, e - b);
        });
        ctx_.timing.pack_s += now_s() - t0;
        src = bb;
    }
    SCG_CUDA_CHECK(cudaMemcpyAsync(B.comp[s].ptr, src, bytes, cudaMemcpyHostToDevice, cs));
    SCG_CUDA_CHECK(cudaMemcpyAsync(B.members[s].ptr, table, (lb - fb) * sizeof(InflateMember), cudaMemcpyHostToDevice, cs));
    SCG_CUDA_CHECK(cudaEventRecord(B.bounced[s], cs));
    B.bounced_valid[s] = true;
    const int launched = launch_inflate(B.comp[s].as<uint8_t>(), B.members[s].as<InflateMember>(), (int)(lb - fb), dst,
                                        B.inflate_errors.as<uint32_t>(), ctx_.sm_count, cs);
    SCG_CUDA_CHECK(cudaGetLastError());
    ctx_.launches += launched;
    ctx_.timing.launches += launched;
    if (chunk + 1 == nchunks() && virtual_newline_) SCG_CUDA_CHECK(cudaMemsetAsync(dst + chunk_bytes(chunk), '\n', 1, cs));
    SCG_CUDA_CHECK(cudaEventRecord(B.copied[s], cs));
    ctx_.timing.bytes_h2d += (long long)(bytes + (lb - fb) * sizeof(InflateMember));
}

void DeviceIngest::issue_copy(size_t chunk) {
    if (bgzf_) {
        issue_inflate(chunk);
        return;
    }
    IngestBuffers& B = buffers();
    const int s = (int)(chunk % (size_t)slots_);
    const size_t off = chunk_begin_[chunk];
    const size_t bytes = chunk_bytes(chunk);
    uint8_t* dst = B.text.as<uint8_t>() + slot_base(chunk) + carry_;
    // the slot's previous text must have been parsed and packed
    if (B.released_valid[s]) SCG_CUDA_CHECK(cudaStreamWaitEvent(B.copy_stream, B.released[s], 0));
    const void* src = text_ + off;
    if (!pinned_source_) {
        if (B.bounced_valid[s]) SCG_CUDA_CHECK(cudaEventSynchronize(B.bounced[s]));
        const double t0 = now_s();
        char* bb = B.bounce[s].as<char>();
        const int pieces = (int)std::max<size_t>(1, std::min<size_t>((size_t)nthreads_, bytes >> 20));
        const size_t per = (bytes + pieces - 1) / pieces;
        HostPool::instance().parallel_for(pieces, pieces, [&](int k) {
            const size_t b = (size_t)k * per, e = std::min(bytes, b + per);
            if (b < e) std::memcpy(bb + b, text_ + off + b, e - b);
        });
        ctx_.timing.pack_s += now_s() - t0;
        src = bb;
    }
    SCG_CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, B.copy_stream));
    if (chunk + 1 == nchunks() && virtual_newline_) SCG_CUDA_CHECK(cudaMemsetAsync(dst + bytes, '\n', 1, B.copy_stream));
    if (!pinned_source_) {
        SCG_CUDA_CHECK(cudaEventRecord(B.bounced[s], B.copy_stream));
        B.bounced_valid[s] = true;
    }
    SCG_CUDA_CHECK(cudaEventRecord(B.copied[s], B.copy_stream));
    ctx_.timing.bytes_h2d += (long long)bytes;
}

bool DeviceIngest::next(Result& out) {
    out = Result();
    if (!stage()) return false;
    return complete(out);
}

bool DeviceIngest::stage() {
    if (exhausted()) return false;
    IngestBuffers& B = buffers();
    const size_t k = parsed_;
    // chunk k + slots - 1 reuses the slot of chunk k - 1, whose kernels (and `released` event) are already enqueued;
    // one further would need the slot this call is about to parse
    while (issued_ < nchunks() && issued_ <= k + (size_t)slots_ - 1) {
        issue_copy(issued_);
        ++issued_;
    }
    const int s = (int)(k % (size_t)slots_);
    const bool final_chunk = k + 1 == nchunks();
    const size_t bytes = chunk_bytes(k) + ((final_chunk && virtual_newline_) ? 1 : 0);
    const uint32_t slot0 = (uint32_t)slot_base(k);
    const uint32_t end = slot0 + (uint32_t)carry_ + (uint32_t)bytes;
    cudaStream_t st = ctx_.stream;
    IngestState* state = B.state.as<IngestState>();
    const uint8_t* ring = B.text.as<uint8_t>();
    uint32_t* lines = B.lines.as<uint32_t>();
    const int nblocks = (int)((end - slot0 + kBlockBytes - 1) / kBlockBytes);
    uint16_t* lens = B.lens[out_slot_].as<uint16_t>();

    SCG_CUDA_CHECK(cudaStreamWaitEvent(st, B.copied[s], 0));
    count_newlines<<<nblocks, kBlockThreads, 0, st>>>(ring, slot0, end, state, B.block_counts.as<uint32_t>());
    scan_blocks<<<1, 1024, 0, st>>>(B.block_counts.as<uint32_t>(), nblocks, state, (uint32_t)line_cap_);
    scatter_newlines<<<nblocks, kBlockThreads, 0, st>>>(ring, slot0, end, state, B.block_counts.as<uint32_t>(), lines, (uint32_t)line_cap_);
    // every group of four lines is looked at, also the ones that are no records (four newlines are four bytes); never more
    // groups than the position buffer describes
    const uint32_t max_rec = (uint32_t)std::min<size_t>(line_cap_ / 4, (end - slot0) / 4 + 1);
    const int rec_blocks = (int)((max_rec + 255) / 256);
    validate_records<<<rec_blocks, 256, 0, st>>>(ring, lines, state, B.seq_off.as<uint32_t>(), lens);
    SCG_CUDA_CHECK(cudaGetLastError());
    ctx_.launches += 4;
    staged_ = true;
    return true;
}

void DeviceIngest::pair(Context& ctx, DeviceIngest& a, DeviceIngest& b) {
    pair_limit<<<1, 1, 0, ctx.stream>>>(a.buffers().state.as<IngestState>(), b.buffers().state.as<IngestState>());
    SCG_CUDA_CHECK(cudaGetLastError());
    ++ctx.launches;
}

bool DeviceIngest::complete(Result& out) {
    out = Result();
    if (!staged_) return false;
    staged_ = false;
    IngestBuffers& B = buffers();
    const size_t k = parsed_;
    const int s = (int)(k % (size_t)slots_);
    const bool final_chunk = k + 1 == nchunks();
    const size_t bytes = chunk_bytes(k) + ((final_chunk && virtual_newline_) ? 1 : 0);
    const uint32_t slot0 = (uint32_t)slot_base(k);
    const uint32_t data0 = slot0 + (uint32_t)carry_;
    const uint32_t end = data0 + (uint32_t)bytes;
    const uint32_t next_data0 = (uint32_t)slot_base(k + 1) + (uint32_t)carry_;
    cudaStream_t st = ctx_.stream;
    IngestState* state = B.state.as<IngestState>();
    const uint8_t* ring = B.text.as<uint8_t>();
    const int out_slot = out_slot_;
    out_slot_ ^= 1;
    uint16_t* lens = B.lens[out_slot].as<uint16_t>();

    finish_chunk<<<1, 1024, 0, st>>>(B.text.as<uint8_t>(), B.lines.as<uint32_t>(), state, end, final_chunk ? 1 : 0, next_data0, (uint32_t)carry_);
    SCG_CUDA_CHECK(cudaGetLastError());
    ++ctx_.launches;
    SCG_CUDA_CHECK(cudaMemcpyAsync(B.meta.ptr, state, sizeof(IngestState), cudaMemcpyDeviceToHost, st));
    uint32_t* inflate_flag = reinterpret_cast<uint32_t*>(B.meta.as<char>() + sizeof(IngestState));
    if (bgzf_) SCG_CUDA_CHECK(cudaMemcpyAsync(inflate_flag, B.inflate_errors.ptr, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    SCG_CUDA_CHECK(cudaEventRecord(B.meta_ready, st));
    {
        const double t0 = now_s();
        SCG_CUDA_CHECK(cudaEventSynchronize(B.meta_ready));
        ctx_.timing.device_s += now_s() - t0;
    }
    if (bgzf_ && *inflate_flag != 0) {
        // a member of this chunk (or of one inflated ahead of it) did not inflate or failed its CRC: nothing of the chunk is
        // used; the host reader resumes where the previous chunk ended, inflates with zlib and raises the error
        SCG_CUDA_CHECK(cudaEventRecord(B.released[s], st));
        B.released_valid[s] = true;
        stopped_ = true;
        out.handover = true;
        out.resume_offset = consumed_;
        last_n_ = 0;
        return true;
    }
    const IngestState m = *B.meta.as<IngestState>();
    ++parsed_;

    const long long tail_off = (long long)chunk_begin_[k] + ((long long)m.tail - (long long)data0);
    consumed_ = (size_t)std::min<long long>(std::max<long long>(tail_off, 0), (long long)size_);
    last_n_ = 0;
    if (m.nrec > 0) {
        const int W = std::max(1, ceil_div((int)m.max_len, 32));
        const size_t ntiles = ((size_t)m.nrec + TILE - 1) / TILE;
        const size_t data_bytes = ntiles * tile_words(W) * sizeof(uint32_t);
        B.packed[out_slot].reserve(data_bytes + READ_GUARD_BYTES);
        uint8_t* odd = want_odd_ ? B.odd[out_slot].as<uint8_t>() : nullptr;
        pack_records_dev<<<(unsigned)((ntiles + 3) / 4), 128, 0, st>>>(ring, B.seq_off.as<uint32_t>(), lens, m.nrec, W,
                                                                       B.packed[out_slot].as<uint32_t>(), odd);
        SCG_CUDA_CHECK(cudaGetLastError());
        ++ctx_.launches;
        out.n = m.nrec;
        out.reads.data = B.packed[out_slot].as<uint32_t>();
        out.reads.W = W;
        out.reads.n = m.nrec;
        out.reads.uniform_len = (int)m.max_len;
        out.reads.lens = (m.min_len == m.max_len) ? nullptr : lens;
        out.odd = odd;
        records_ += m.nrec;
        last_n_ = m.nrec;
        last_text_base_ = (long long)chunk_begin_[k] - (long long)data0;
        last_out_slot_ = out_slot;
        last_off_.clear();
    }
    SCG_CUDA_CHECK(cudaEventRecord(B.released[s], st));
    B.released_valid[s] = true;
    if (m.status != 0) {
        // on the last chunk a clean end (nothing left) has status 0; everything else goes to the host reader
        stopped_ = true;
        out.handover = true;
        out.resume_offset = consumed_;
        return true;
    }
    return parsed_ < nchunks() || out.n > 0;
}

void DeviceIngest::raw_read(long long index, std::string& seq) {
    if (index < 0 || index >= last_n_) throw Error("raw_read: no such read in the current batch");
    if (last_off_.empty()) {
        // sequence offsets (ring positions) and lengths of the batch: still in place until the next chunk is staged
        IngestBuffers& B = buffers();
        last_off_.resize((size_t)last_n_);
        last_len_.resize((size_t)last_n_);
        SCG_CUDA_CHECK(cudaMemcpyAsync(last_off_.data(), B.seq_off.ptr, (size_t)last_n_ * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx_.stream));
        SCG_CUDA_CHECK(cudaMemcpyAsync(last_len_.data(), B.lens[last_out_slot_].ptr, (size_t)last_n_ * sizeof(uint16_t), cudaMemcpyDeviceToHost,
                                       ctx_.stream));
        SCG_CUDA_CHECK(cudaStreamSynchronize(ctx_.stream));
    }
    const size_t at = (size_t)(last_text_base_ + (long long)last_off_[(size_t)index]);
    const size_t len = last_len_[(size_t)index];
    if (bgzf_) {
        fetch_text(at, len, seq);
    } else {
        seq.assign(text_ + at, len);
    }
}

} // namespace scg
