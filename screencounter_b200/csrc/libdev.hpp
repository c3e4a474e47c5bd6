// Plain-old-data views of device-resident objects, readable by nvcc-built kernels and by the
// run-time specialised kernels (NVRTC) alike: no standard headers.
#pragma once

#include "layout.hpp"

namespace scg {

// Device view of a library (library.hpp builds it): plain pointers into device memory.
struct LibDev {
    int L;              // key length in bases
    int KW;             // words per plane
    int nentries;       // expanded (concrete) entries
    int dup_first;      // ties between different indices resolve to the lowest index
    // exact table, two-table cuckoo: T1 then T2, slot_mask + 1 slots of slot_words words each:
    // h[KW], l[KW], value (-1 = empty), padding; a key is at T1[hash & mask] or T2[hash_second(hash) & mask]
    const uint32_t* slots;
    uint32_t slot_mask;
    int slot_words;
    // expanded entries for verification: ent_keys[e*2KW ..] = h[KW], l[KW]; ent_idx[e] = pool index
    const uint32_t* ent_keys;
    const int32_t* ent_idx;
    // pigeonhole seeds
    int nseeds;
    const uint32_t* seed_masks;  // nseeds * KW words: base positions of each seed (same mask for H and L)
    const uint2* buckets;     // nseeds * (bucket_mask + 1) entries of (start, count) into cands
    uint32_t bucket_mask;
    const int32_t* cands;     // nseeds * nentries entry ids, grouped by bucket
    // KW == 1 only: the same candidates as rows (h, l, pool index, 0), so that a candidate costs one 16-byte load
    const uint4* cand_rows;
    // KW == 1 only (nullptr when not built): the seed buckets with their first candidate inline -- (H word, L word, pool index,
    // start | count << 24) per bucket, indexed like `buckets` -- so that a seed costs ONE 16-byte load in nine cases out of ten
    const uint4* ibuckets;
    // segmented search (dual paired-end): first segment = bases [0, seg1), second = [seg1, L)
    int seg1;
    // table of library rows with their last base dropped (SURVEY 8.1 T8 root rule)
    const uint32_t* prefix_slots;
    uint32_t prefix_mask;
    // the reference's flat trie (library.hpp), nullptr unless the first segment may take 2 or more mismatches
    const int32_t* trie;
};

// What the specialised single-barcode kernel (spec_single.cuh) needs of the two strands' libraries, passed by
// value as a kernel argument so that the table pointers sit in the constant bank.  [0] forward, [1] reverse.
struct SpecTables {
    const uint4* slots[2];      // exact cuckoo tables (16-byte slots)
    const uint2* buckets[2];    // pigeonhole seed buckets
    const uint4* cand_rows[2];  // candidates as rows
    uint32_t slot_mask[2];
    uint32_t bucket_mask[2];
    int nentries[2];
    const LibDev* libs;         // the full descriptors, for the generic search of the rare complicated reads
    // Exact table of BOTH strands for keys of up to 31 bases (uniform-length kernel): a two-table cuckoo hash like the
    // per-strand ones (16-byte slots: H word, L word, pool index, 0; empty = index -1) with the strand as bit 31 of the H
    // word, so that the table's address and size are the same for every lane, and with a hash of three multiply-adds.
    // Table 1 holds n = 1 << (32 - joint_shift) slots, table 2 the next n.
    const uint4* joint;
    uint32_t joint_shift;
    // Seed buckets with their first candidate inline: (H word, L word, pool index, start | count << 24) per bucket, same
    // indexing as `buckets`.  Nine in ten non-empty buckets hold one candidate: one load instead of bucket -> row.
    const uint4* ibuckets[2];
};

// the two homes of a key in the joint table (host builder and kernel alike): top bits of a multiplicative hash
SCG_HD uint32_t joint_hash(uint32_t kh_tagged, uint32_t kl) { return kh_tagged * 0x9E3779B1u + kl * 0x85EBCA6Bu; }
SCG_HD uint32_t joint_hash2(uint32_t x) { return x * 0xC2B2AE35u; }
constexpr int JOINT_MAX_KEYLEN = 31;

// Device count table of 64-bit keys (random barcodes of up to 21 bases, sparse combinations): open addressing with linear
// probing over 16-byte slots (key, count, padding), so that finding or inserting a key touches ONE 32-byte sector -- the
// device-side counterpart of the reference's unordered_map<string, int> (handlers/RandomBarcodeSingleEnd.hpp:93-104).
struct CountSlot {
    unsigned long long key;   // ~0 = empty
    uint32_t count;
    uint32_t pad;
};
struct CountTable64 {
    CountSlot* slots;
    unsigned long long mask;       // capacity - 1
    unsigned long long* live;      // [0] distinct keys inserted so far, [1] != 0: the table overflowed and inserts were dropped
};
// 128-bit keys (random barcodes of 22 to 42 bases): keys and counts in separate arrays
struct CountTable128 {
    ulonglong2* keys;  // EMPTY = (~0, ~0); 16-byte aligned
    uint32_t* counts;
    unsigned long long mask;
    unsigned long long* live;
};
// Keys of more than two words (random barcodes of 43 bases or more, `words` text-order words: SortedTable's layout): a tag
// word per slot (0 = empty; else fingerprint | LONG_OCCUPIED, and while the key is FRESH also LONG_FRESH | its staging row),
// a count per slot and a key store of `words` words per slot.  A counting kernel writes every key to its own staging row
// before it probes, so a slot is claimed with ONE compare-and-swap of its tag and nobody ever waits for another thread's key
// to appear: a FRESH slot is compared against the staging row its tag names, a RESIDENT one against the key store.  A
// follow-up kernel moves the fresh rows (their slots listed in `fresh`) to the key store before the staging rows are reused.
struct CountTableLong {
    unsigned long long* tags;
    uint32_t* counts;
    unsigned long long* keys;          // words per slot
    unsigned long long* staging;       // words per read of the launch, indexed by read
    unsigned long long* fresh;         // slots claimed by the launch
    unsigned long long* fresh_count;
    unsigned long long mask;
    unsigned long long* live;
    int words;
};
// slot of a key: one 64-bit multiply, the halves folded (the low half alone only mixes upwards)
SCG_HD unsigned long long count_hash(unsigned long long key) {
    const unsigned long long x = key * 0x9E3779B97F4A7C15ull;
    return x ^ (x >> 32);
}

// Outcome for reads the packed representation cannot render as text (lower case, symbols other
// than N): the host formats those keys from the raw read (handlers/RandomBarcodeSingleEnd.hpp:93-120).
struct OddOutcome {
    long long read;
    int position;
    int reverse;
};

// Where combinations are tallied: a dense n1 x n2 matrix when it is small, else the 64-bit hash.
struct ComboSink {
    int32_t* dense;        // n1 * n2 counters or nullptr
    CountTable64 sparse;
    int n2;
};

// ---- arguments of the run-time compiled handler kernels (spec_handlers.cuh) ----

// Reads a specialised kernel cannot settle on the spot wait, with everything the search behind them needs, in regions of a
// global list -- ONE REGION PER WARP of the kernel that fills it (a persistent warp visits at most `per_warp / 32` tiles), so
// that appending costs no atomic.  Entries are structures of arrays: word k of entry e is words[k * stride + e]; region w
// holds entries [w * per_warp, w * per_warp + warp_counts[w]).  A follow-up kernel works the regions off.
struct DeferredList {
    uint32_t* words;
    unsigned long long stride;   // entries per word plane (= regions * per_warp)
    uint32_t per_warp;
    uint32_t regions;
    uint32_t* warp_counts;
};
// Reads that need the full per-read search (several candidate windows): their indices, appended with one atomic per warp
// batch; the generic kernel of the handler visits them (handlers.cuh ReadList).
struct SlowList {
    uint32_t* list;
    uint32_t* count;
};
// Random barcodes of one launch sorted by the PART of the count table they live in (part = the top bits of the home slot): the
// main kernel appends every barcode to the list of (part, warp) -- no atomics, one cursor per part in shared memory -- and a
// second kernel counts the lists part by part, so that the slice of the table it works on (a few megabytes) stays in L2 and
// HBM sees the table once per launch, sequentially, instead of one random 32-byte read-modify-write per read.
struct PartitionedKeys {
    unsigned long long* keys;   // region r = part * nwarps + warp holds keys[r * cap .. r * cap + counts[r])
    uint32_t* counts;           // [nparts * nwarps]
    uint32_t cap;               // keys per region (a region that runs over sends its keys straight to the table)
    uint32_t nwarps;
    uint32_t shift;             // part of a key = home slot >> shift
    uint32_t nparts;            // <= 32
};
// Exact table of the dual paired-end design for keys of up to 48 bases (both variable regions concatenated): a two-table
// cuckoo hash of 16-byte slots (H bits 0..31, L bits 0..31, H bits 32..47 | L bits 32..47 << 16, pool row; empty = row -1).
// Table 1 holds 1 << (32 - shift) slots, table 2 the next as many.
struct DualTables {
    const uint4* exact;
    uint32_t shift;
};
SCG_HD uint32_t dual_hash(uint32_t x, uint32_t y, uint32_t z) { return x * 0x9E3779B1u + y * 0x85EBCA6Bu + z * 0xC2B2AE35u; }
SCG_HD uint32_t dual_hash2(uint32_t h) { return h * 0x27D4EB2Fu + 0x165667B1u; }
constexpr int DUAL_MAX_KEYLEN = 48;
// The mismatch-tolerant side of the dual paired-end library for keys of up to 48 bases and budgets of at most one mismatch per
// read (four seeds at most), flattened for the follow-up kernel: candidates as 16-byte rows in the layout of DualTables (H lo, L lo,
// H hi | L hi << 16, pool row), and seed buckets of 32 bytes that carry their first candidate -- (row)(start, count, -, -) -- so
// that a seed costs one aligned 32-byte fetch where the generic search walks bucket -> candidate list -> entry keys -> entry index.
struct DualFlat {
    const uint4* ibuckets;      // nseeds * (bucket_mask + 1) * 2
    const uint4* rows;          // nseeds * nentries
    uint32_t bucket_mask;
    int nentries;
    int nseeds;                 // 1 .. 4
    uint32_t seed_lo[4], seed_hi[4];   // base positions of each seed, words 0 and 1 of the key
    uint32_t seg1_lo, seg1_hi;         // base positions of the first segment
    int kw, seg1, L;
    int dup_first;
    const uint32_t* prefix_slots;      // rows with their last base dropped (root rule), the library's own table
    uint32_t prefix_mask;
    int slot_words;
};
// Exact tables of the four libraries of the single-end combinatorial design, [2 * reverse + region in read order]: the
// libraries' own cuckoo tables (library.cpp CuckooTable, keys of one word per plane, 16-byte slots).
struct ComboTables {
    const uint4* slots[4];
    uint32_t mask[4];
};
// words per deferred entry
constexpr int DUAL_DEFER_WORDS = 6;    // pair index, H lo, L lo, H hi | L hi << 16, N lo, N hi | cap1 << 16 | cap2 << 24
constexpr int COMBO_DEFER_WORDS = 8;   // read index, reverse << 8 | constant mismatches, (H, L, N) of region 0, (H, L, N) of region 1

// Packed reads of one batch on the device.
struct ReadsDev {
    const uint32_t* data;   // tile-planar words
    const uint16_t* lens;   // nullptr when every read has length uniform_len
    int uniform_len;
    int W;
    long long n;
};

} // namespace scg
