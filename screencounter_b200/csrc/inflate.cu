// DEFLATE on the device, one warp per gzip member (inflate.cuh).
//
// A BGZF member holds at most 64 KiB of text and is a DEFLATE stream of its own (no preset dictionary), so members inflate
// independently: one WARP takes one member.  Huffman decoding is sequential by nature; the warp runs it UNIFORMLY (every lane
// holds the same bit buffer and decodes the same symbol, table lookups are shared-memory broadcasts) and uses its width where
// the format allows it:
//   * the compressed bytes arrive as coalesced 128-byte lines, one 32-bit word per lane, two lines ahead of the bit buffer;
//     a refill takes its word from the owning lane with a shuffle -- no global-memory latency on the decoding chain;
//   * code tables are built by all lanes (counting by shared atomics, canonical codes by __match_any ranks, table fill
//     per symbol);
//   * symbols are decoded in batches of up to 32 (about 2 KiB of text at most), parked in shared memory; the batch's output
//     offsets are one warp scan; the batch's text is ASSEMBLED IN SHARED MEMORY: literals are stored by their lanes, matches
//     whose source lies wholly before the batch are fetched from global memory without any ordering between them (their loads
//     overlap), matches that read bytes of their own batch -- the rule in FASTQ, where a record repeats most of the one before
//     it -- are copied in order at shared-memory latency; the finished batch goes out to global memory as aligned words.
// Tables: 10-bit literal/length and 8-bit distance lookup (2-byte entries: value or base, extra bits, code length), longer codes go
// through the canonical count/symbol arrays bit by bit (rare by construction: a code longer than 10 bits has probability
// < 2^-10).  Text is written to global memory (the FASTQ reader's ring), source bytes of a match are read back from there.
// A second kernel checks the members' CRC-32 (gzip trailer), one warp per member, 2 KiB per lane, slice-by-4 tables in shared
// memory, the lanes' partial CRCs combined with the "2 KiB of zeros" operator.
#include "inflate.cuh"

#include <algorithm>
#include <cstdlib>

namespace scg {

namespace {

constexpr int LIT_BITS = 10, DIST_BITS = 8;
constexpr int INFL_WARPS = 4;   // warps per block
constexpr uint32_t FULL = 0xFFFFFFFFu;
constexpr uint32_t STAGE_BYTES = 2048;   // text assembled per batch at most; a batch closes once it could not take another 258-byte match

// table entry (16 bits, so that a warp's tables stay under 3 KiB and 32 warps fit an SM); bits 0-3 = code length, 0 for
// everything off the hot path (E_INVALID no such code, E_LONG a code longer than the table: bit-by-bit walk, E_EOB end of block).
//   literal/length table: literal  = byte << 8 | code length
//                         length   = (base - 3) << 8 | extra bits << 5 | 1 << 4 | code length      (RFC 1951 3.2.5: base 3 .. 258)
//   distance table:       distance = m << 8 | extra bits << 4 | code length, base = (m << extra bits) + 1  (m = 0 .. 3)
// so a match costs no further table: the symbol's base and its number of extra bits travel in the entry.
constexpr uint32_t E_INVALID = 0, E_LONG = 1u << 8, E_EOB = 2u << 8;
constexpr uint32_t E_MATCH = 1u << 4;
using Entry = uint16_t;

// what a batch of symbols needs in shared memory
struct BatchArea {
    uint32_t syms[32], sym_off[32];           // the batch's symbols (see the kernel) and where their text starts in the batch
    uint32_t stage[STAGE_BYTES / 4 + 2];      // the text of the batch being assembled (+ alignment slack)
};

struct WarpTables {
    Entry lit[1 << LIT_BITS];
    Entry dist[1 << DIST_BITS];
    uint32_t lit_count[16], dist_count[16];   // codes per length (kept for the bit-by-bit path)
    uint32_t next[16], offs[16];              // scratch of the table build
    uint16_t lit_sorted[288 + 32];            // symbols in canonical order (per length, ascending)
    uint16_t dist_sorted[32 + 32];
    uint8_t lens[288 + 32 + 32];              // code lengths of the block being set up
    BatchArea batch;
};

// base value | extra bits << 16 of the length symbols 257 .. 285 (RFC 1951 3.2.5); only the table build reads it
#define SCG_BE(base, extra) ((uint32_t)(base) | ((uint32_t)(extra) << 16))
__constant__ uint32_t c_len_sym[29] = { SCG_BE(3, 0),  SCG_BE(4, 0),  SCG_BE(5, 0),  SCG_BE(6, 0),   SCG_BE(7, 0),   SCG_BE(8, 0),   SCG_BE(9, 0),   SCG_BE(10, 0),
                                        SCG_BE(11, 1), SCG_BE(13, 1), SCG_BE(15, 1), SCG_BE(17, 1),  SCG_BE(19, 2),  SCG_BE(23, 2),  SCG_BE(27, 2),  SCG_BE(31, 2),
                                        SCG_BE(35, 3), SCG_BE(43, 3), SCG_BE(51, 3), SCG_BE(59, 3),  SCG_BE(67, 4),  SCG_BE(83, 4),  SCG_BE(99, 4),  SCG_BE(115, 4),
                                        SCG_BE(131, 5), SCG_BE(163, 5), SCG_BE(195, 5), SCG_BE(227, 5), SCG_BE(258, 0) };
__constant__ uint8_t c_clen_order[19] = { 16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15 };

// what a code of `len` bits for `sym` stands for, as a table entry (E_INVALID = a symbol the format does not define)
__device__ __forceinline__ uint32_t lit_entry(int sym, int len) {
    if (sym < 256) return ((uint32_t)sym << 8) | (uint32_t)len;
    if (sym == 256) return E_EOB;   // its code length is looked up where the block ends
    if (sym > 285) return E_INVALID;
    const uint32_t be = c_len_sym[sym - 257];
    return (((be & 0xFFFFu) - 3u) << 8) | ((be >> 16) << 5) | E_MATCH | (uint32_t)len;
}
// distance symbol s >= 2 has s / 2 - 1 extra bits and base ((2 | s & 1) << extra bits) + 1; symbols 0 and 1 are distances 1 and 2
__device__ __forceinline__ uint32_t dist_entry(int sym, int len) {
    if (sym > 29) return E_INVALID;
    const uint32_t extra = sym < 2 ? 0u : (uint32_t)(sym / 2 - 1);
    const uint32_t m = sym < 2 ? (uint32_t)sym : (2u | ((uint32_t)sym & 1u));
    return (m << 8) | (extra << 4) | (uint32_t)len;
}
// code-length alphabet: the symbol itself is the value
__device__ __forceinline__ uint32_t clen_entry(int sym, int len) { return ((uint32_t)sym << 6) | (uint32_t)len; }

// Builds the lookup table of a canonical Huffman code from the code lengths lens[0 .. n).  KIND 0 literal/length, 1 distance,
// 2 code lengths.  All lanes of the warp take part.  false = over-subscribed set of lengths.
template <int KIND, int TBITS>
__device__ bool build_table(const uint8_t* lens, int n, Entry* table, uint16_t* sorted, uint32_t* count, uint32_t* next, uint32_t* offs,
                            int lane) {
    const uint32_t below = (1u << (threadIdx.x & 31)) - 1u;   // the lanes in front of this one
    for (int i = lane; i < (1 << TBITS); i += 32) table[i] = (Entry)E_INVALID;
    for (int i = lane; i < 16; i += 32) count[i] = 0;
    __syncwarp();
    for (int s = lane; s < n; s += 32) {
        const int l = lens[s];
        if (l) atomicAdd(&count[l], 1u);
    }
    __syncwarp();
    bool ok = true;
    if (lane == 0) {
        uint32_t code = 0, off = 0;
        int left = 1;
        for (int l = 1; l <= 15; ++l) {
            next[l] = code;
            offs[l] = off;
            left = (left << 1) - (int)count[l];
            if (left < 0) ok = false;
            code = (code + count[l]) << 1;
            off += count[l];
        }
    }
    ok = __shfl_sync(FULL, ok ? 1 : 0, 0) != 0;
    if (!ok) return false;
    __syncwarp();
    for (int base = 0; base < n; base += 32) {
        const int s = base + lane;
        const int l = s < n ? lens[s] : 0;
        const uint32_t peers = __match_any_sync(FULL, l);
        const int rank = __popc(peers & below);
        if (l) {
            const uint32_t code = next[l] + (uint32_t)rank;
            sorted[offs[l] + (uint32_t)rank] = (uint16_t)s;
            const uint32_t r = __brev(code) >> (32 - l);   // the code as it appears in the bit stream (first bit = bit 0)
            if (l <= TBITS) {
                const uint32_t e = KIND == 0 ? lit_entry(s, l) : (KIND == 1 ? dist_entry(s, l) : clen_entry(s, l));
                for (uint32_t k = r; k < (1u << TBITS); k += (1u << l)) table[k] = (Entry)e;
            } else {
                table[r & ((1u << TBITS) - 1u)] = (Entry)E_LONG;
            }
        }
        __syncwarp();
        if (l && rank == 0) {
            next[l] += (uint32_t)__popc(peers);
            offs[l] += (uint32_t)__popc(peers);
        }
        __syncwarp();
    }
    return true;
}

// a code longer than the lookup table: bit by bit over the canonical counts (the first TBITS bits cannot end a code either,
// so the walk starts from the top)
__device__ __forceinline__ bool slow_symbol(unsigned long long bits, const uint32_t* count, const uint16_t* sorted, int& sym, int& len) {
    uint32_t code = 0, first = 0, index = 0;
    for (int l = 1; l <= 15; ++l) {
        code |= (uint32_t)(bits & 1ull);
        bits >>= 1;
        const uint32_t c = count[l];
        if (code < first + c) {
            sym = sorted[index + (code - first)];
            len = l;
            return true;
        }
        index += c;
        first = (first + c) << 1;
        code <<= 1;
    }
    return false;
}

// The compressed stream as seen by the warp: a window of 64 bits of the stream that stays put between refills, and the
// number of its bits already consumed -- taking bits moves the position (one add), looking at bits is one 64-bit shift.  The
// window is refilled, 32 bits at a time, from two register-resident lines of 32 words.
struct BitReader {
    const uint32_t* words;      // 4-byte aligned base of the stream
    uint32_t line_cur, line_next;
    uint32_t widx;              // words taken into the window so far (uniform in the warp)
    unsigned long long bits;    // stream bits [32 * (widx - 2), 32 * widx)
    int bp;                     // bits of the window consumed
    int lane;

    __device__ __forceinline__ void open(const uint8_t* comp, size_t byte_off, int lane_) {
        lane = lane_;
        words = reinterpret_cast<const uint32_t*>(comp + (byte_off & ~(size_t)3));
        line_cur = words[lane];
        line_next = words[32 + lane];
        widx = 0;
        const uint32_t lo = next_word();
        bits = (unsigned long long)lo | ((unsigned long long)next_word() << 32);
        bp = (int)(byte_off & 3) * 8;
    }
    __device__ __forceinline__ uint32_t next_word() {
        const uint32_t w = __shfl_sync(FULL, line_cur, (int)(widx & 31u));
        ++widx;
        if ((widx & 31u) == 0) {
            line_cur = line_next;
            line_next = words[widx + 32 + lane];
        }
        return w;
    }
    // at least 33 unconsumed bits afterwards
    __device__ __forceinline__ void refill() {
        if (bp >= 32) {
            bits = (bits >> 32) | ((unsigned long long)next_word() << 32);
            bp -= 32;
        }
    }
    // the next 32 bits of the stream (all of them valid right after a refill; 64 - bp of them in general)
    __device__ __forceinline__ uint32_t window() const { return (uint32_t)(bits >> bp); }
    __device__ __forceinline__ unsigned long long window64() const { return bits >> bp; }
    __device__ __forceinline__ uint32_t peek(int n) const { return window() & ((1u << n) - 1u); }
    __device__ __forceinline__ void drop(int n) { bp += n; }
    __device__ __forceinline__ uint32_t take(int n) {
        const uint32_t v = peek(n);
        drop(n);
        return v;
    }
    __device__ __forceinline__ void to_byte_boundary() { bp = (bp + 7) & ~7; }
    // bits / bytes of the stream consumed, counted from the aligned base
    __device__ __forceinline__ size_t bit_pos() const { return (size_t)widx * 32 - 64 + (size_t)bp; }
    __device__ __forceinline__ size_t byte_pos() const { return (size_t)widx * 4 - 8 + (size_t)(bp >> 3); }
};

// A match of the batch, copied into the stage: byte j comes from batch-relative position off - dist + j (the repeating
// pattern of the last `dist` bytes when the match overlaps itself); positions before the batch are text already in global
// memory (`done` = the batch's first byte there), the others are bytes of the stage written by earlier symbols.
__device__ __forceinline__ void copy_match(uint8_t* stage, const uint8_t* done, uint32_t off, uint32_t len, uint32_t dist, int lane) {
    for (uint32_t j = lane; j < len; j += 32) {
        const int src = (int)off - (int)dist + (int)(dist >= len ? j : j % dist);
        stage[off + j] = src < 0 ? done[src] : stage[src];
    }
}

// The text of a batch of nsym symbols (A.syms, `total` bytes of text in all) assembled in shared memory and written to
// out[pos, pos + total).  All lanes of the warp take part; false = a symbol reaches before the start of the text or the
// batch beyond its end.
__device__ __forceinline__ bool put_batch(BatchArea& A, int nsym, uint32_t staged, uint8_t* out, uint32_t pos, uint32_t out_len, int lane) {
    constexpr uint32_t SHORT_MATCH = 12;
    __syncwarp();
    // ---- where the batch's symbols go: lane l looks after symbol l ----
    const uint32_t my = lane < nsym ? A.syms[lane] : 0u;
    const uint32_t mylen = (my >> 16) & 0x1FFu;
    uint32_t incl = mylen;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t v = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += v;
    }
    const uint32_t total = staged;
    const uint32_t off = incl - mylen;   // relative to the batch's first byte
    A.sym_off[lane] = off;
    const bool is_match = mylen != 0 && !(my >> 31);
    const uint32_t dist = my & 0xFFFFu;
    const bool too_far = is_match && dist > pos + off;
    // matches whose source ends before the batch begins: no ordering among them, their loads overlap
    const bool indep = is_match && off + mylen <= dist;
    const bool indep_short = indep && mylen <= SHORT_MATCH;
    // this lane's symbol among the batch's 32, by what copies it
    const uint32_t long_bits = indep && mylen > SHORT_MATCH ? 1u << lane : 0u;
    const uint32_t dep_bits = is_match && !indep ? 1u << lane : 0u;
    if (pos + total > out_len || __any_sync(FULL, too_far)) {
        return false;
    }
    // the stage mirrors the alignment of the text in global memory, so that it can be flushed as aligned words
    uint8_t* const done = out + pos;
    const uint32_t skew = (uint32_t)(reinterpret_cast<size_t>(done) & 3);
    uint8_t* const stage = reinterpret_cast<uint8_t*>(A.stage) + skew;
    if (my >> 31) stage[off] = (uint8_t)my;
    // Short independent matches (the rule for the bases of a FASTQ record) are copied by the lanes that hold them, all
    // at once: the warp runs as many byte steps as the longest of them has bytes, instead of a round per match.
    if (indep_short) {
        const uint8_t* src = done + ((int)off - (int)dist);
        for (uint32_t i = 0; i < mylen; ++i) stage[off + i] = src[i];
    }
    __syncwarp();   // A.sym_off is read below
    // the longer ones by all lanes together, four matches at a time: a warp issues in order, so the loads of four
    // matches go out before the first store waits
    uint32_t todo = __reduce_or_sync(FULL, long_bits);
    while (todo) {
        uint32_t sy[4], o[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            sy[u] = 0;
            o[u] = 0;
            if (todo) {
                const int k = __ffs(todo) - 1;
                todo &= todo - 1;
                sy[u] = A.syms[k];
                o[u] = A.sym_off[k];
            }
        }
        uint8_t v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            v[u] = 0;
            if ((uint32_t)lane < ((sy[u] >> 16) & 0x1FFu)) v[u] = done[(int)o[u] - (int)(sy[u] & 0xFFFFu) + lane];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if ((uint32_t)lane < ((sy[u] >> 16) & 0x1FFu)) stage[o[u] + lane] = v[u];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const uint32_t len = (sy[u] >> 16) & 0x1FFu;
            for (uint32_t j = lane + 32; j < len; j += 32) stage[o[u] + j] = done[(int)o[u] - (int)(sy[u] & 0xFFFFu) + (int)j];
        }
    }
    // the others read bytes of this batch: in order, each after what precedes it has landed in the stage
    todo = __reduce_or_sync(FULL, dep_bits);
    while (todo) {
        __syncwarp();
        const int k = __ffs(todo) - 1;
        todo &= todo - 1;
        const uint32_t sy = A.syms[k], o = A.sym_off[k];
        copy_match(stage, done, o, (sy >> 16) & 0x1FFu, sy & 0xFFFFu, lane);
    }
    __syncwarp();
    // ---- the finished batch goes out: whole aligned words, the ragged ends byte by byte ----
    {
        const uint32_t span = skew + total;                 // bytes of the stage in use, from its aligned base
        const uint32_t first_word = skew ? 1u : 0u;         // word 0 is partial when the text does not start aligned
        const uint32_t full_words = span / 4;               // words [first_word, full_words) are complete
        uint32_t* gw = reinterpret_cast<uint32_t*>(done - skew);
        for (uint32_t w = first_word + lane; w < full_words; w += 32) gw[w] = A.stage[w];
        const uint8_t* sb = reinterpret_cast<const uint8_t*>(A.stage);
        uint8_t* gb = done - skew;
        if (skew && (uint32_t)lane >= skew && (uint32_t)lane < min(4u, span)) gb[lane] = sb[lane];
        const uint32_t tail = full_words * 4;               // bytes [tail, span) of a last partial word
        if (full_words >= first_word && tail + lane < span && tail + lane >= skew) gb[tail + lane] = sb[tail + lane];
    }
    __syncwarp();
    return true;
}

// one warp per member, INFL_WARPS warps per block
__global__ void __launch_bounds__(INFL_WARPS * 32) inflate_kernel(const uint8_t* __restrict__ comp, const InflateMember* __restrict__ members, int n,
                                                                  uint8_t* out_base, uint32_t* __restrict__ errors) {
    __shared__ WarpTables tables[INFL_WARPS];
    const int lane = threadIdx.x & 31;
    WarpTables& T = tables[threadIdx.x >> 5];
    const int first_member = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int member_stride = (int)((gridDim.x * blockDim.x) >> 5);

    for (int mi = first_member; mi < n; mi += member_stride) {
        const InflateMember M = members[mi];
        uint8_t* out = out_base + M.out_off;
        uint32_t pos = 0;
        bool bad = false;
        if (M.out_len == 0 && M.in_len <= 2) continue;   // the empty member that closes a BGZF file
        BitReader br;
        br.open(comp, M.in_off, lane);
        bool last = false;
        while (!last && !bad) {
            // a block header beyond the member's bytes: a damaged stream running away (it must not leave the image)
            if ((size_t)(reinterpret_cast<const uint8_t*>(br.words) - comp) * 8 + br.bit_pos() >
                ((size_t)M.in_off + M.in_len) * 8) {
                bad = true;
                break;
            }
            br.refill();
            last = br.take(1) != 0;
            const uint32_t type = br.take(2);
            if (type == 0) {
                // ---- stored block: to the byte boundary, LEN, NLEN, LEN raw bytes ----
                br.to_byte_boundary();
                br.refill();
                const uint32_t len = br.take(16);
                br.refill();
                const uint32_t nlen = br.take(16);
                if ((len ^ nlen) != 0xFFFFu || pos + len > M.out_len) {
                    bad = true;
                    break;
                }
                const size_t from = (size_t)(reinterpret_cast<const uint8_t*>(br.words) - comp) + br.byte_pos();
                for (uint32_t j = lane; j < len; j += 32) out[pos + j] = comp[from + j];
                pos += len;
                __syncwarp();
                br.open(comp, from + len, lane);
                continue;
            }
            if (type == 3) {
                bad = true;
                break;
            }
            int nlit = 288, ndist = 30;
            if (type == 1) {
                // ---- fixed codes (RFC 1951 3.2.6) ----
                for (int s = lane; s < 288; s += 32) T.lens[s] = s < 144 ? 8 : (s < 256 ? 9 : (s < 280 ? 7 : 8));
                for (int s = lane; s < 30; s += 32) T.lens[288 + s] = 5;
            } else {
                // ---- dynamic codes: the code-length code first, then the two alphabets' lengths through it ----
                br.refill();
                nlit = (int)br.take(5) + 257;
                ndist = (int)br.take(5) + 1;
                const int nclen = (int)br.take(4) + 4;
                if (nlit > 286 || ndist > 30) {
                    bad = true;
                    break;
                }
                for (int s = lane; s < 19; s += 32) T.lens[320 + s] = 0;
                __syncwarp();
                for (int k = 0; k < nclen; ++k) {
                    br.refill();
                    const uint32_t v = br.take(3);
                    if (lane == 0) T.lens[320 + c_clen_order[k]] = (uint8_t)v;
                }
                __syncwarp();
                if (!build_table<2, 7>(T.lens + 320, 19, T.dist, T.dist_sorted, T.dist_count, T.next, T.offs, lane)) {
                    bad = true;
                    break;
                }
                __syncwarp();
                int i = 0;
                uint32_t prev = 0;
                while (i < nlit + ndist) {
                    br.refill();
                    const uint32_t e = T.dist[br.peek(7)];
                    if ((e & 0xFu) == 0) {
                        bad = true;
                        break;
                    }
                    br.drop((int)(e & 0xFu));
                    const uint32_t sym = e >> 6;
                    uint32_t rep = 1, val = sym;
                    if (sym == 16) {
                        if (i == 0) {
                            bad = true;
                            break;
                        }
                        val = prev;
                        rep = 3 + br.take(2);
                    } else if (sym == 17) {
                        val = 0;
                        rep = 3 + br.take(3);
                    } else if (sym == 18) {
                        val = 0;
                        rep = 11 + br.take(7);
                    }
                    if (i + (int)rep > nlit + ndist) {
                        bad = true;
                        break;
                    }
                    // lengths of the distance alphabet are kept from offset 288 on
                    for (uint32_t k = lane; k < rep; k += 32) {
                        const int at = i + (int)k;
                        T.lens[at < nlit ? at : 288 + (at - nlit)] = (uint8_t)val;
                    }
                    i += (int)rep;
                    prev = val;
                }
                if (bad) break;
                __syncwarp();
                if (T.lens[256] == 0) {   // no end-of-block code
                    bad = true;
                    break;
                }
            }
            __syncwarp();
            if (!build_table<0, LIT_BITS>(T.lens, nlit, T.lit, T.lit_sorted, T.lit_count, T.next, T.offs, lane) ||
                !build_table<1, DIST_BITS>(T.lens + 288, ndist, T.dist, T.dist_sorted, T.dist_count, T.next, T.offs, lane)) {
                bad = true;
                break;
            }
            __syncwarp();

            // ---- the block's symbols, a batch at a time ----
            bool end_of_block = false;
            while (!end_of_block && !bad) {
                // a damaged stream must not read its way out of the image: no batch starts beyond the member's own bytes
                if ((size_t)(reinterpret_cast<const uint8_t*>(br.words) - comp) * 8 + br.bit_pos() >
                    ((size_t)M.in_off + M.in_len) * 8) {
                    bad = true;
                    break;
                }
                // symbols are parked in shared memory: literal = 1 << 31 | 1 << 16 | byte; match = len << 16 | dist
                int nsym = 0;
                uint32_t staged = 0;   // bytes the batch produces so far (uniform in the warp)
#pragma unroll 1
                for (; nsym < 32 && staged <= STAGE_BYTES - 258; ++nsym) {
                    br.refill();
                    const uint32_t w = br.window();   // 32 valid bits: the code (15 at most) and a length's extra bits (5)
                    uint32_t e = T.lit[w & ((1u << LIT_BITS) - 1u)];
                    if ((e & 0xFu) == 0) {
                        // off the hot path: a code longer than the table, the end of the block, or no code at all
                        int sym = 256, len = T.lens[256];
                        if (e == E_LONG) e = slow_symbol(br.window64(), T.lit_count, T.lit_sorted, sym, len) ? lit_entry(sym, len) : E_INVALID;
                        if ((e & 0xFu) == 0) {
                            if (e == E_EOB) {
                                br.drop(len);
                                end_of_block = true;
                            } else {
                                bad = true;
                            }
                            break;
                        }
                    }
                    const uint32_t elen = e & 0xFu;
                    uint32_t sym;
                    if (!(e & E_MATCH)) {
                        br.drop((int)elen);
                        sym = 0x80010000u | (e >> 8);
                        staged += 1;
                    } else {
                        const uint32_t xl = (e >> 5) & 7u;
                        const uint32_t len = (e >> 8) + 3u + ((w >> elen) & ((1u << xl) - 1u));
                        br.drop((int)(elen + xl));
                        br.refill();
                        const uint32_t w2 = br.window();   // the distance code (15 bits at most) and its extra bits (13)
                        uint32_t d = T.dist[w2 & ((1u << DIST_BITS) - 1u)];
                        if ((d & 0xFu) == 0) {
                            int dsym = 0, dlen = 0;
                            if (d == E_LONG) d = slow_symbol(br.window64(), T.dist_count, T.dist_sorted, dsym, dlen) ? dist_entry(dsym, dlen) : E_INVALID;
                            if ((d & 0xFu) == 0) {
                                bad = true;
                                break;
                            }
                        }
                        const uint32_t dl = d & 0xFu, xd = (d >> 4) & 0xFu;
                        const uint32_t dist = ((d >> 8) << xd) + 1u + ((w2 >> dl) & ((1u << xd) - 1u));
                        br.drop((int)(dl + xd));
                        sym = (len << 16) | dist;
                        staged += len;
                    }
                    T.batch.syms[nsym] = sym;   // every lane stores the same word
                }
                if (bad) break;
                if (!put_batch(T.batch, nsym, staged, out, pos, M.out_len, lane)) {
                    bad = true;
                    break;
                }
                pos += staged;
            }
        }
        // the stream must end inside the member and produce exactly its text
        if (!bad) {
            const size_t end_bit = (size_t)(reinterpret_cast<const uint8_t*>(br.words) - comp) * 8 + br.bit_pos();
            bad = pos != M.out_len || end_bit > ((size_t)M.in_off + M.in_len) * 8;
        }
        if (bad && lane == 0) atomicOr(errors, 1u);
        __syncwarp();
    }
}

// ---- CRC-32 of the inflated members -------------------------------------------------------------------------------------------
// bytes per lane in the staging rows of crc_kernel: 256 of text + 16, so that the 16-byte accesses of eight neighbouring lanes fall
// into different banks
constexpr int CRC_ROW = 272;

struct CrcOperator {
    uint32_t zeros2k[32];   // register after 2 KiB of zero bytes, per start bit
};

__global__ void __launch_bounds__(INFL_WARPS * 32) crc_kernel(const InflateMember* __restrict__ members, int n, const uint8_t* __restrict__ out_base,
                                                              CrcOperator op, uint32_t* __restrict__ errors) {
    __shared__ uint32_t tab[4][256];
    __shared__ __align__(16) uint8_t crc_rows[INFL_WARPS][32 * CRC_ROW];
    {
        // slice-by-4 tables of the reflected polynomial 0xEDB88320
        const int t = threadIdx.x;
        for (int v = t; v < 256; v += blockDim.x) {
            uint32_t c = (uint32_t)v;
            for (int k = 0; k < 8; ++k) c = (c & 1u) ? (c >> 1) ^ 0xEDB88320u : c >> 1;
            tab[0][v] = c;
        }
        __syncthreads();
        for (int s = 1; s < 4; ++s) {
            for (int v = t; v < 256; v += blockDim.x) tab[s][v] = (tab[s - 1][v] >> 8) ^ tab[0][tab[s - 1][v] & 0xFFu];
            __syncthreads();
        }
    }
    const int lane = threadIdx.x & 31;
    const int warp = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int nwarps = (int)((gridDim.x * blockDim.x) >> 5);
    for (int mi = warp; mi < n; mi += nwarps) {
        const InflateMember M = members[mi];
        if (M.out_len == 0) continue;
        // segment 0 = the first (len - 2048 * nfull) bytes, 1 .. 2048 of them; segments 1 .. nfull are 2 KiB each
        const uint32_t nfull = (M.out_len - 1) / 2048;
        const uint32_t head = M.out_len - 2048 * nfull;
        uint32_t crc = 0;
        const uint8_t* const text = out_base + M.out_off;
        if (nfull >= 1 && (reinterpret_cast<size_t>(text) & 15) == 0 && (head & 15u) == 0) {
            // Every segment starts on a 16-byte boundary (the rule: BGZF members hold 65 280 bytes).  A lane reading its own 2 KiB
            // word by word costs the L1 a tag look-up per lane and load (32 sectors per request: the kernel sat at 93 % of the
            // L1/TEX pipe and 16 % of issue); so the warp fetches 256 bytes of every segment with coalesced 16-byte loads -- 16
            // lanes per segment, two segments per instruction -- into rows of shared memory, and each lane reads its row.
            uint8_t* const rows = crc_rows[threadIdx.x >> 5];
            const uint32_t mylen = lane == 0 ? head : ((uint32_t)lane <= nfull ? 2048u : 0u);
            crc = lane == 0 ? 0xFFFFFFFFu : 0u;
            const int sub = lane & 15, half = lane >> 4;
            for (uint32_t r = 0; r < 2048u; r += 256u) {
                for (uint32_t row = (uint32_t)half; row <= nfull; row += 2) {
                    const uint32_t seg_begin = row == 0 ? 0u : head + 2048u * (row - 1), seg_len = row == 0 ? head : 2048u;
                    const uint32_t off = r + 16u * (uint32_t)sub;
                    if (off < seg_len)
                        *reinterpret_cast<uint4*>(rows + row * CRC_ROW + 16 * sub) = *reinterpret_cast<const uint4*>(text + seg_begin + off);
                }
                __syncwarp();
                if (r < mylen) {
                    const uint32_t n16 = min(256u, mylen - r) / 16u;
                    for (uint32_t c = 0; c < n16; ++c) {
                        const uint4 q = *reinterpret_cast<const uint4*>(rows + lane * CRC_ROW + 16 * c);
                        const uint32_t v[4] = { q.x, q.y, q.z, q.w };
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            crc ^= v[k];
                            crc = tab[3][crc & 0xFFu] ^ tab[2][(crc >> 8) & 0xFFu] ^ tab[1][(crc >> 16) & 0xFFu] ^ tab[0][crc >> 24];
                        }
                    }
                }
                __syncwarp();
            }
        } else if ((uint32_t)lane <= nfull) {
            const uint32_t begin = lane == 0 ? 0u : head + 2048u * (uint32_t)(lane - 1);
            const uint32_t len = lane == 0 ? head : 2048u;
            const uint8_t* p = out_base + M.out_off + begin;
            crc = lane == 0 ? 0xFFFFFFFFu : 0u;
            const uint32_t* w = reinterpret_cast<const uint32_t*>(reinterpret_cast<size_t>(p) & ~(size_t)3);
            const uint32_t sh = (uint32_t)(reinterpret_cast<size_t>(p) & 3) * 8;
            uint32_t lo = *w;
            const uint32_t nwords = len / 4;
            for (uint32_t k = 0; k < nwords; ++k) {
                const uint32_t hi = sh ? w[k + 1] : 0u;
                const uint32_t v = sh ? __funnelshift_r(lo, hi, sh) : w[k];
                lo = hi;
                crc ^= v;
                crc = tab[3][crc & 0xFFu] ^ tab[2][(crc >> 8) & 0xFFu] ^ tab[1][(crc >> 16) & 0xFFu] ^ tab[0][crc >> 24];
            }
            for (uint32_t k = nwords * 4; k < len; ++k) crc = tab[0][(crc ^ p[k]) & 0xFFu] ^ (crc >> 8);
        }
        // state after segment k = zeros2k(state after segment k - 1) ^ raw CRC of segment k
        uint32_t acc = __shfl_sync(FULL, crc, 0);
        for (uint32_t k = 1; k <= nfull; ++k) {
            const uint32_t part = __shfl_sync(FULL, crc, (int)k);
            uint32_t moved = 0;
#pragma unroll
            for (int b = 0; b < 32; ++b) moved ^= ((acc >> b) & 1u) ? op.zeros2k[b] : 0u;
            acc = moved ^ part;
        }
        if (lane == 0 && ~acc != M.crc) atomicOr(errors, 2u);
    }
}

// host: the "2 KiB of zero bytes" operator of CRC-32
CrcOperator make_crc_operator() {
    uint32_t table[256];
    for (uint32_t v = 0; v < 256; ++v) {
        uint32_t c = v;
        for (int k = 0; k < 8; ++k) c = (c & 1u) ? (c >> 1) ^ 0xEDB88320u : c >> 1;
        table[v] = c;
    }
    CrcOperator op;
    for (int b = 0; b < 32; ++b) {
        uint32_t c = 1u << b;
        for (int k = 0; k < 2048; ++k) c = table[c & 0xFFu] ^ (c >> 8);
        op.zeros2k[b] = c;
    }
    return op;
}

} // namespace

int launch_inflate(const uint8_t* comp, const InflateMember* members, int n, uint8_t* out, uint32_t* errors, int sm_count, cudaStream_t stream) {
    if (n <= 0) return 0;
    static const CrcOperator op = make_crc_operator();
    static const bool check_crc = !std::getenv("SCG_BGZF_NO_CRC");
    const int blocks = std::max(1, std::min((n + INFL_WARPS - 1) / INFL_WARPS, sm_count * 8));
    inflate_kernel<<<blocks, INFL_WARPS * 32, 0, stream>>>(comp, members, n, out, errors);
    if (!check_crc) return 1;
    crc_kernel<<<blocks, INFL_WARPS * 32, 0, stream>>>(members, n, out, op, errors);
    return 2;
}

} // namespace scg
