/*
 * scg.h -- C ABI of the B200-native barcode-counting engine.
 *
 * Drop-in boundary for the hot path of crisprVerse/screenCounter (FASTQ reads ->
 * template scan -> barcode lookup -> counts).  Each scg_count_* / scg_match_barcodes
 * entry point replaces one Rcpp-exported function of the reference; argument order and
 * meaning follow the reference (R/RcppExports.R:4-30, src/RcppExports.cpp:13-150), with
 * R containers flattened to plain pointers and sizes.  The reference-side binding a
 * maintainer adds (the Rcpp shim) is shown in INTEGRATION.md.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error; the message (kaori's own
 *     wording where the reference has one) is read with scg_last_error().  No C++
 *     exception crosses this boundary.
 *   - a FASTQ input is an scg_source: a file path (raw or gzip, sniffed from the magic
 *     bytes like byteme::SomeFileReader, inst/include/byteme/SomeFileReader.hpp:25-66)
 *     or a host memory buffer holding FASTQ text (like byteme::RawBufferReader).
 *   - fixed-size outputs (count vectors, totals) are caller-owned; variable-size outputs
 *     (combination tables, random-barcode tables, per-read traces) come back as an
 *     scg_result handle that the caller reads with scg_result_* and frees.
 *   - `nthreads` is the reference's num.threads; here it sizes the host FASTQ packer.
 *   - CUDA is initialised lazily by the first call that needs the device (fork safety
 *     under BiocParallel::MulticoreParam), never at library load.
 *   - there is no CPU fallback: without a usable CUDA device every counting call fails.
 */
#ifndef SCG_H
#define SCG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct scg_ctx scg_ctx;
typedef struct scg_result scg_result;
typedef struct scg_reads scg_reads;   /* packed reads resident in device memory */
typedef struct scg_plan scg_plan;     /* a compiled handler: template + libraries on the device */
typedef struct scg_table scg_table;   /* a sparse result as a sorted (key, count) table on the device */

/* FASTQ input: path != NULL -> file (raw or .gz); else `data`/`size` hold FASTQ text. */
typedef struct {
    const char* path;
    const char* data;
    size_t size;
} scg_source;

/* strand codes: src/utils.cpp:33-41 (to_strand(int)) */
enum { SCG_STRAND_ORIGINAL = 0, SCG_STRAND_REVERSE = 1, SCG_STRAND_BOTH = 2 };

/* ---- context ------------------------------------------------------------------------ */
int scg_ctx_create(scg_ctx** out, int device);       /* device = CUDA ordinal; lazy init */
/* One context over SEVERAL devices (the reference runs its threads inside one call, inst/include/kaori/process_data.hpp:131-177;
 * this is the same for GPUs): the single-end entry points scg_count_single, scg_count_combo_single, scg_count_dual_single_end and
 * scg_count_random cut the text of a raw or block-gzip file (or of a memory buffer) at record boundaries into one part per
 * device, and merge the parts' results into exactly what a context of one device returns; the scg_count_*_many calls deal
 * their files to the devices.  Inputs that cannot be cut (plain gzip streams, small files) are read by one device alone.
 * The paired-input entry points (scg_count_dual, scg_count_combo_paired, scg_count_single_paired) run on the first device. */
int scg_ctx_create_multi(scg_ctx** out, const int* devices, int n_devices);
int scg_ctx_devices(const scg_ctx* ctx);
void scg_ctx_destroy(scg_ctx* ctx);
const char* scg_last_error(const scg_ctx* ctx);       /* ctx may be NULL for creation errors */
const char* scg_version(void);
/* JSON with the stage timings of the most recent counting call on this context:
 * parse_s, pack_s, h2d_s, device_s, reads, bytes_h2d, kernel launches. */
const char* scg_timing_json(const scg_ctx* ctx);
/* number of kernels this library has launched on behalf of the context so far */
long long scg_kernel_launches(const scg_ctx* ctx);

/* ---- results ------------------------------------------------------------------------ */
size_t scg_result_rows(const scg_result* r);          /* table rows (combinations / barcodes) */
int scg_result_width(const scg_result* r);            /* ints per key row, or chars per barcode */
size_t scg_result_reads(const scg_result* r);         /* reads (pairs) in the per-read trace */
/* Any pointer may be NULL.  keys: rows*width int32 (0-based pool indices, sorted ascending,
 * one combination per row = one column of the reference's IntegerMatrix, src/utils.h:28-34);
 * strings: rows*width chars, no terminators, sorted A<C<G<N<T (R/countRandomBarcodes.R:73);
 * freq: rows int32. */
int scg_result_copy_table(const scg_result* r, int32_t* keys, char* strings, int32_t* freq);
/* Per-read trace (only filled when the call was made with want_trace != 0):
 * index: reads*trace_width int32, -1 = no match; info: reads uint32,
 * bit 31 found, bit 30 reverse strand, bits 20-24 mismatches, bits 25-29 variable mismatches,
 * bits 0-19 position (meaningful for the single-barcode design only). */
int scg_result_trace_width(const scg_result* r);
int scg_result_copy_trace(const scg_result* r, int32_t* index, uint32_t* info);
void scg_result_free(scg_result* r);

/* ---- the seven entry points of the reference ---------------------------------------- */

/* replaces count_single_barcodes, src/count_single_barcodes.cpp:29-50.
 * counts: npool int32; total: reads seen.  trace (nullable out) receives per-read outcomes. */
int scg_count_single(scg_ctx* ctx, const scg_source* src, const char* constant, int strand,
                     const char* const* pool, int npool, int mismatches, int use_first, int nthreads,
                     int32_t* counts, int32_t* total, scg_result** trace);

/* replaces count_random_barcodes, src/count_random_barcodes.cpp:41-60.
 * table: distinct barcodes (strings) + frequencies. */
int scg_count_random(scg_ctx* ctx, const scg_source* src, const char* constant, int strand,
                     int mismatches, int use_first, int nthreads,
                     scg_result** table, int32_t* total);

/* replaces count_combo_barcodes_single, src/count_combo_barcodes_single.cpp:40-70 (two pools). */
int scg_count_combo_single(scg_ctx* ctx, const scg_source* src, const char* constant, int strand,
                           const char* const* pool1, int npool1, const char* const* pool2, int npool2,
                           int mismatches, int use_first, int nthreads, int want_trace,
                           scg_result** table, int32_t* total);

/* replaces count_dual_barcodes_single_end, src/count_dual_barcodes_single_end.cpp:51-88.
 * pools_flat: npools*nchoices strings, pool-major.  With diagnostics != 0, *table receives the
 * invalid combinations (two pools only, as in the reference glue). */
int scg_count_dual_single_end(scg_ctx* ctx, const scg_source* src, const char* constant,
                              const char* const* pools_flat, int npools, int nchoices, int strand,
                              int mismatches, int use_first, int diagnostics, int nthreads, int want_trace,
                              int32_t* counts, int32_t* total, scg_result** table);

/* replaces count_dual_barcodes, src/count_dual_barcodes.cpp:75-116. */
int scg_count_dual(scg_ctx* ctx,
                   const scg_source* src1, const char* constant1, int reverse1, int mismatches1,
                   const char* const* pool1, int npool1,
                   const scg_source* src2, const char* constant2, int reverse2, int mismatches2,
                   const char* const* pool2, int npool2,
                   int randomized, int use_first, int diagnostics, int nthreads, int want_trace,
                   int32_t* counts, int32_t* total, scg_result** table, int32_t* barcode1_only, int32_t* barcode2_only);

/* replaces count_combo_barcodes_paired, src/count_combo_barcodes_paired.cpp:55-95. */
int scg_count_combo_paired(scg_ctx* ctx,
                           const scg_source* src1, const char* constant1, int reverse1, int mismatches1,
                           const char* const* pool1, int npool1,
                           const scg_source* src2, const char* constant2, int reverse2, int mismatches2,
                           const char* const* pool2, int npool2,
                           int randomized, int use_first, int nthreads, int want_trace,
                           scg_result** table, int32_t* total, int32_t* barcode1_only, int32_t* barcode2_only);

/* kaori's SingleBarcodePairedEnd handler (inst/include/kaori/handlers/SingleBarcodePairedEnd.hpp:27-170): one barcode per
 * read PAIR, searched on read 1 and on read 2 with the same template, pool and options.  screenCounter exports no R
 * function for this handler; the entry point is here for callers of kaori that use it.  trace: per-pair pool index. */
int scg_count_single_paired(scg_ctx* ctx, const scg_source* src1, const scg_source* src2, const char* constant, int strand,
                            const char* const* pool, int npool, int mismatches, int use_first, int nthreads,
                            int32_t* counts, int32_t* total, scg_result** trace);

/* replaces match_barcodes, src/match_barcodes.cpp:7-37.  index is 0-based with -1 where the
 * reference returns NA_INTEGER (the shim adds 1); mismatches is -1 for NA. */
int scg_match_barcodes(scg_ctx* ctx, const char* const* sequences, int nsequences,
                       const char* const* choices, int nchoices, int substitutions, int reverse,
                       int32_t* index, int32_t* mismatches);

/* ---- many files, one call (the matrixOf* wrappers of the reference) ------------------------- */

/* matrixOfSingleBarcodes (R/countSingleBarcodes.R:112-126): count_single_barcodes per file, columns bound.  matrix: npool x
 * nfiles int32, column-major (column f = the counts of sources[f]); totals: nfiles.  The library is built and uploaded once per
 * device; files are dealt to the context's devices (fewer files than devices: each file is cut over all of them). */
int scg_count_single_many(scg_ctx* ctx, const scg_source* sources, int nfiles, const char* constant, int strand,
                          const char* const* pool, int npool, int mismatches, int use_first, int nthreads,
                          int32_t* matrix, int32_t* totals);
/* countComboBarcodes per file + combineComboCounts (R/combineComboCounts.R:31-57): *table holds the sorted union of the files'
 * combinations (scg_result_copy_table: keys, freq = row sums) and one column of counts per file (scg_result_copy_matrix).  The
 * union is made on the device from the files' sorted tables. */
int scg_count_combo_many(scg_ctx* ctx, const scg_source* sources, int nfiles, const char* constant, int strand,
                         const char* const* pool1, int npool1, const char* const* pool2, int npool2,
                         int mismatches, int use_first, int nthreads, scg_result** table, int32_t* totals);
/* matrixOfRandomBarcodes (R/countRandomBarcodes.R:84-105): sort(union of the files' barcodes) and one column per file. */
int scg_count_random_many(scg_ctx* ctx, const scg_source* sources, int nfiles, const char* constant, int strand,
                          int mismatches, int use_first, int nthreads, scg_result** table, int32_t* totals);
/* columns of a many-files result, and its matrix: rows x columns int32, column-major */
int scg_result_columns(const scg_result* r);
int scg_result_copy_matrix(const scg_result* r, int32_t* matrix);

/* ---- block gzip (BGZF: bgzip, bcl-convert) -------------------------------------------------- */
/* A FASTQ source that is a block-gzip file -- or a block-gzip image in memory (scg_source.data) -- is read like raw text by
 * the device-side reader: its members cross PCIe compressed and are inflated (and CRC-checked) on the device.  Plain gzip
 * streams are inflated by zlib on the host like the reference does (inst/include/byteme/GzipFileReader.hpp:39-51).
 *   scg_bgzf_compress   text -> block-gzip image on `nthreads` host threads (zlib `level`, members of `block_text` bytes of
 *                       text, 0 = bgzip's 65280); call with out == NULL to get the capacity needed in *used.
 *   scg_bgzf_inflate    the device inflater on its own: image (host) -> text (host); *device_ms = time of the kernels.
 *                       Call with text == NULL to get the text's size. */
int scg_bgzf_compress(const char* text, size_t size, int level, int block_text, int nthreads, void* out, size_t capacity, size_t* used);
int scg_bgzf_inflate(scg_ctx* ctx, const void* image, size_t size, char* text, size_t capacity, size_t* text_size, double* device_ms);

/* ---- resident objects (for callers that keep reads / libraries on the device) ---------- */

/* Parse + pack a FASTQ into device memory (tile-planar 2-bit bases + N mask; DESIGN.md). */
int scg_reads_from_source(scg_ctx* ctx, const scg_source* src, int nthreads, scg_reads** out);
long long scg_reads_count(const scg_reads* r);
long long scg_reads_device_bytes(const scg_reads* r);
void scg_reads_free(scg_reads* r);

/* Synthetic workload of BASELINE.json / SURVEY.md 8(d): counter-based generator, identical on
 * the host (FASTQ text) and on the device (packed reads), any shard reproducible from
 * (seed, first_read). */
typedef struct {
    uint64_t seed;
    long long first_read;      /* global index of this shard's first read */
    long long n_reads;
    int read_len;              /* 75 */
    const char* constant;      /* template with '-' runs, e.g. 12 + 20 + 12 */
    int n_pools;               /* variable regions filled from pools (<= 2); 0 = random barcodes */
    const char* const* pools[2];
    int n_choices[2];
    int paired_rows;           /* != 0: one row index picks (pools[0][i], pools[1][i]) */
    int strand;                /* SCG_STRAND_*: BOTH = half the constructs reverse-complemented */
    int construct_permille;    /* reads carrying a construct, e.g. 900 */
    int sub_per_10k;           /* per-base substitution rate inside the construct, e.g. 100 = 1 % */
    int n_per_10k;             /* per-base N rate anywhere, e.g. 10 = 0.1 % */
    long long random_space;    /* n_pools == 0: number of distinct "true" random barcodes */
} scg_synth_spec;

int scg_reads_synthesize(scg_ctx* ctx, const scg_synth_spec* spec, scg_reads** out);
/* FASTQ text of the same reads on the host.  Returns bytes needed in *used (call with out=NULL to size). */
int scg_synth_fastq(const scg_synth_spec* spec, char* out, size_t capacity, size_t* used);

/* Compiled single-barcode handler (template + library resident on the device). */
int scg_single_plan_create(scg_ctx* ctx, const char* constant, int strand,
                           const char* const* pool, int npool, int mismatches, int use_first,
                           scg_plan** out);
/* One pass of the hot path over resident reads.  d_counts (device, npool int32) is ACCUMULATED
 * into; d_index (device, nullable) receives the per-read pool index.  Runs on `cuda_stream`, a
 * cudaStream_t used as given (NULL is CUDA's legacy default stream, e.g. torch's default stream);
 * SCG_STREAM_OWN selects the context's own stream.  Does not synchronise. */
#define SCG_STREAM_OWN ((void*)(intptr_t)-1)
int scg_single_plan_run(scg_plan* plan, const scg_reads* reads, int32_t* d_counts, int32_t* d_index,
                        void* cuda_stream);
void scg_plan_free(scg_plan* plan);
/* Which kernel variant the plan's last run used: "specialised (NVRTC) ..." = the template compiled into the
 * kernel at run time, or "generic ... (<why>)". */
const char* scg_plan_kernel(const scg_plan* plan);

/* Compiled handlers of the other designs over resident reads: the kernels behind scg_count_dual (not randomized designs take
 * the run-time specialised kernel), scg_count_combo_single and scg_count_random, without the FASTQ reader in front.  A
 * context serves one stream at a time (the kernels share per-context scratch).
 *   dual    d_counts (device, npool int32) is ACCUMULATED into; d_index (device, nullable) receives the pool row per pair.
 *   combo   the plan owns the tally of combinations; d_pairs (device, nullable, 2 int32 per read) receives (first, second).
 *   random  the plan owns the count table.  expected_distinct > 0 sizes it once for that many distinct barcodes (a run never
 *           synchronises; a table that overflows is reported by scg_plan_harvest); 0 lets it grow like the reference's map.
 *           d_index (device, nullable): 2 * window position + strand of the counted window, or -1.
 * scg_plan_reset empties the plan's tally (asynchronously, on the stream); scg_plan_harvest synchronises the device and
 * returns the table exactly as the file-level call would (sorted; rows stay on the device until scg_result_copy_table). */
int scg_dual_plan_create(scg_ctx* ctx, const char* constant1, int reverse1, int mismatches1, const char* const* pool1, int npool1,
                         const char* constant2, int reverse2, int mismatches2, const char* const* pool2, int npool2,
                         int randomized, int use_first, scg_plan** out);
int scg_dual_plan_run(scg_plan* plan, const scg_reads* reads1, const scg_reads* reads2, int32_t* d_counts, int32_t* d_index,
                      void* cuda_stream);
int scg_combo_plan_create(scg_ctx* ctx, const char* constant, int strand, const char* const* pool1, int npool1,
                          const char* const* pool2, int npool2, int mismatches, int use_first, scg_plan** out);
int scg_combo_plan_run(scg_plan* plan, const scg_reads* reads, int32_t* d_pairs, void* cuda_stream);
int scg_random_plan_create(scg_ctx* ctx, const char* constant, int strand, int mismatches, int use_first,
                           long long expected_distinct, scg_plan** out);
int scg_random_plan_run(scg_plan* plan, const scg_reads* reads, int32_t* d_index, void* cuda_stream);
int scg_plan_reset(scg_plan* plan, void* cuda_stream);
int scg_plan_harvest(scg_plan* plan, scg_result** table);

/* Sparse results as sorted tables ON THE DEVICE: what GPUs exchange when the table of one file (or of several files) is
 * merged across them -- the device-side counterpart of the reference's reduce() for random barcodes
 * (inst/include/kaori/handlers/RandomBarcodeSingleEnd.hpp:197-207) and of the append + sort of combinations
 * (handlers/CombinatorialBarcodesSingleEnd.hpp:268-305, R/combineComboCounts.R:31-57).  keys: unsigned 64-bit, ascending,
 * unique -- combinations as first << 32 | second, random barcodes as three bits per base in text order (A < C < G < N < T),
 * first base most significant; counts: unsigned 32-bit.  key_len > 0 marks random barcodes of that length.
 *   scg_plan_sorted_table   the plan's tally, sorted (synchronises the device)
 *   scg_plan_dense_tally    combinations tallied in a dense n1 x n2 matrix: its device address (else *d_matrix = NULL)
 *   scg_table_from_device   a table from device arrays the caller owns (copied), e.g. rows received from another GPU
 *   scg_table_merge         sorted union of two tables, counts of equal keys added
 *   scg_table_render        the table as the file-level calls return it (rows stay on the device until copied) */
int scg_plan_sorted_table(scg_plan* plan, scg_table** out);
int scg_plan_dense_tally(scg_plan* plan, void** d_matrix, long long* cells);
long long scg_table_rows(const scg_table* t);
int scg_table_key_len(const scg_table* t);
void* scg_table_keys(const scg_table* t);
void* scg_table_counts(const scg_table* t);
int scg_table_from_device(scg_ctx* ctx, const void* d_keys, const void* d_counts, long long rows, int key_len, scg_table** out);
int scg_table_merge(scg_ctx* ctx, const scg_table* a, const scg_table* b, scg_table** out);
int scg_table_render(scg_ctx* ctx, const scg_table* t, scg_result** out);
void scg_table_free(scg_table* t);

/* Host-only check of the FASTQ reader + packer (no device needed): parses `src`, packs every read into
 * the tile-planar 2-bit + N-mask layout and unpacks it again.  bases receives the concatenated
 * sequences as upper-case A/C/G/T with N for every other character; offsets (n_reads + 1 entries)
 * delimit them.  Call with bases == NULL to size the outputs (*n_reads, *n_bases). */
int scg_host_pack_roundtrip(const scg_source* src, int nthreads, char* bases, long long* offsets,
                            long long* n_reads, long long* n_bases);

/* Compiles the run-time specialised single-barcode kernel for a template (NVRTC) and, when a device is
 * present, loads it.  Returns 0 = compiled and loaded, 2 = compiled but no device to load it on,
 * 1 = failed; `message` receives the details.  Diagnostic only. */
int scg_jit_selftest(const char* constant, int strand, int mismatches, int words_per_plane, char* message, size_t capacity);
/* The same for the uniform-length variant of that kernel (every read `read_len` bases, 1 to 32 windows). */
int scg_jit_selftest_uniform(const char* constant, int strand, int mismatches, int read_len, char* message, size_t capacity);

/* The same for the specialised kernels of the other handlers (spec_handlers.cuh): kind 1 = dual paired-end (templates a and
 * b, `strand_*` = 0 original / 1 reverse), 2 = combinatorial single-end, 3 = random barcodes (template a only). */
int scg_jit_selftest_handler(int kind, const char* constant_a, int strand_a, int mismatches_a, const char* constant_b, int strand_b,
                             int mismatches_b, int read_len, int use_first, char* message, size_t capacity);

/* The segmented search behind countDualBarcodes on its own (SegmentedBarcodeSearch<2>::search,
 * inst/include/kaori/BarcodeSearch.hpp:478-487, without its result cache): `caps` holds two budgets per
 * query (first, second segment); index is 0-based, -1 = no match.  Diagnostic, used by the tests. */
int scg_search_segmented(scg_ctx* ctx, const char* const* sequences, int nsequences, const int32_t* caps,
                         const char* const* choices, int nchoices, int len1, int len2, int max1, int max2,
                         int32_t* index, int32_t* mismatches);

/* Plain device-memory helpers so that a caller without a CUDA runtime of its own (R, ctypes)
 * can own buffers for scg_single_plan_run. */
int scg_device_alloc(scg_ctx* ctx, size_t bytes, void** out);   /* zero-initialised */
int scg_device_free(scg_ctx* ctx, void* ptr);
int scg_device_zero(scg_ctx* ctx, void* ptr, size_t bytes, void* cuda_stream);  /* stream as above */
int scg_device_to_host(scg_ctx* ctx, void* host, const void* dev, size_t bytes);
int scg_synchronize(scg_ctx* ctx);

/* Page-locked host memory.  FASTQ text handed over in such a buffer (scg_source.data) goes to the device
 * by DMA straight from it; text in ordinary memory is first copied through the library's own pinned
 * bounce buffers.  Either way the records are split and packed on the device (the device-side
 * counterpart of kaori::FastqReader, inst/include/kaori/FastqReader.hpp:42-110). */
int scg_host_alloc(scg_ctx* ctx, size_t bytes, void** out);
int scg_host_free(scg_ctx* ctx, void* ptr);

#ifdef __cplusplus
}
#endif

#endif /* SCG_H */
