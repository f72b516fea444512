/* gavisunk_b200.h -- C ABI of libgavisunk_b200.so
 *
 * B200-native (sm_100a) engine for GAVISUNK's data-parallel core: SUNK database build, SUNK
 * matching of ONT reads, best-contig (diagonal band) filter, bad-SUNK histogram, inter-SUNK
 * distance validation, validated intervals / gaps and the gap-spanning probability table.
 *
 * The reference (pdishuck/GAVISUNK) has no FFI: its seam is "one OS process per Snakemake rule,
 * argv + TSV/BED files" (SURVEY.md section 8b).  Each entry point below names the reference
 * program / function it replaces (file:line relative to the reference repository).  The Python
 * package `gavisunk_b200` binds these with ctypes and re-creates the reference CLIs on top.
 *
 * Conventions
 *   - every function returns 0 on success, a negative GVS_E_* code on failure;
 *     gvs_last_error(ctx) returns a NUL-terminated message owned by the context.
 *   - one gvs_ctx per GPU; a context is not thread-safe; independent contexts may be driven from
 *     different host threads.  There is NO CPU fallback: without a CUDA device gvs_create fails.
 *   - "host" pointers are ordinary (ideally pinned) host memory; "dev" pointers are device
 *     memory of the context's GPU (e.g. torch tensors' data_ptr()).
 *   - all results live in device memory owned by the context until the next call of the same
 *     stage; the *_get functions copy them to caller-provided host buffers.
 *   - contig ids are indices into the contig list given at database build/load time (ref.fa
 *     order: hap1 contigs then hap2 contigs, workflow/rules/defineSUNKs.smk:17).
 */
#ifndef GAVISUNK_B200_H
#define GAVISUNK_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gvs_ctx gvs_ctx;

enum {
  GVS_OK = 0,
  GVS_E_CUDA = -1,      /* CUDA runtime error (message has the detail)                            */
  GVS_E_ARG = -2,       /* bad argument / call order                                              */
  GVS_E_KEYERROR = -3,  /* a read hit a db k-mer that has no .loc row: the reference raises
                           KeyError here (workflow/src/kmerpos_annot3.nim:90)                     */
  GVS_E_NOMEM = -4,
  GVS_E_OVERFLOW = -5,  /* an internal capacity was exceeded (message says which)                 */
  GVS_E_STATE = -6      /* stage called before its inputs exist                                   */
};

/* stage ids for gvs_stage_ms() */
enum {
  GVS_ST_PROBE = 0,     /* read scan / probe kernel (kmerpos_annot3.nim:85-96 inner loop)         */
  GVS_ST_EMIT = 1,      /* hit ordering + consecutive-group suppression                           */
  GVS_ST_DIAG = 2,      /* diag_filter_v3 + diag_filter_step2                                     */
  GVS_ST_HIST = 3,      /* badsunks_AR.py histogram (gvs_group_hist)                              */
  GVS_ST_VALIDATE = 4,  /* process-by-contig per-read validation                                  */
  GVS_ST_INTERVALS = 5, /* components -> intervals (gvs_intervals), gaps (gvs_gaps): the last call */
  GVS_ST_DBBUILD = 6,
  GVS_ST_COMPONENTS = 7, /* local forest of the validated pairs (gvs_components_local)             */
  GVS_ST_MODE = 8,      /* badsunks_AR.py mode per haplotype (gvs_hist_mode)                      */
  GVS_ST_BAD = 9,       /* bad SUNK groups (gvs_bad_groups)                                       */
  GVS_ST_MERGE = 10,    /* union with the peers' forests (gvs_components_merge_all)               */
  GVS_ST_SUPPORT = 11,  /* support tracks (gvs_placements, gvs_support): no reference counterpart  */
  GVS_ST_EVIDENCE = 12, /* gap evidence (gvs_gap_evidence): no reference counterpart                */
  GVS_ST_SCREEN = 13,   /* junction screen of one batch (gvs_junction_screen)                     */
  GVS_ST_JUNCTIONS = 14, /* junction records (gvs_junctions): no reference counterpart            */
  GVS_ST_DISCORDANCE = 15, /* distance discordance (gvs_spans, gvs_discordance): no reference counterpart */
  GVS_ST_READHAPS = 16, /* haplotype mode of the diag filter (gvs_diag_filter_haps): votes per haplotype, records */
  GVS_ST_SWITCHES = 17, /* strand switches inside a contig (gvs_strand_switches): no reference counterpart       */
  GVS_ST_DEPTH = 18,    /* SUNK hit depth (gvs_sunk_depth, gvs_depth_runs): no reference counterpart                */
  GVS_ST_ALLELES = 19,  /* allele support (gvs_allele_support, gvs_allele_runs): no reference counterpart          */
  GVS_ST_COUNT = 20
};

/* ------------------------------------------------------------------------------------------ */
/* context                                                                                     */
/* ------------------------------------------------------------------------------------------ */
/* k = SUNK_len (config/config.yaml:2).  1 <= k <= 32.  At k = 32 the reference's k-mer iterator is broken
 * (nim-kmer 0.2.6: the forward mask (1 shl 2k) - 1 is 0) but deterministic: window 0 yields min(fwd, rc | 3),
 * window w >= 1 yields min(code(seq[w+31]), rc) -- pinned through the executable by tests/golden/kat_k32,
 * kat_k32b, ksweep -- and gvs_match reproduces exactly that (one plain kernel, no filters: of no practical use). */
gvs_ctx* gvs_create(int device, int k);
void gvs_destroy(gvs_ctx* ctx);
const char* gvs_last_error(gvs_ctx* ctx);
const char* gvs_version(void);
/* Launch all work of this context on `cuda_stream` (a cudaStream_t; NULL = legacy default). */
int gvs_set_stream(gvs_ctx* ctx, void* cuda_stream);
int gvs_sync(gvs_ctx* ctx);
/* Enable per-stage CUDA-event timing; gvs_stage_ms returns the device time of the last run of
 * that stage (sum of its kernels), measured with events on the context's stream. */
int gvs_set_profiling(gvs_ctx* ctx, int on);
int gvs_stage_ms(gvs_ctx* ctx, int stage, float* ms);
/* Page-locked host memory for inputs / results (a *_get into pageable memory is staged by the driver and
 * several times slower; gvs_reads_set only overlaps the copy with the probe from page-locked memory). */
int gvs_host_alloc(uint64_t bytes, void** p);
void gvs_host_free(void* p);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
uint64_t gvs_launch_count(gvs_ctx* ctx);

/* ------------------------------------------------------------------------------------------ */
/* SUNK database                                                                               */
/* ------------------------------------------------------------------------------------------ */
/* Replaces the table load of kmerpos_annot3 (workflow/src/kmerpos_annot3.nim:20-26 db set,
 * :57-69 loc table): db_kmer = kmer.encode() of every jellyfish.db line, loc_* = the four
 * columns of mrsfast/kmer.loc in file order (later duplicates of a k-mer overwrite earlier ones,
 * nim:68).  contig ids index the caller's contig-name list.  All pointers are host memory. */
int gvs_db_load_loc(gvs_ctx* ctx, const uint64_t* db_kmer, uint64_t n_db,
                    const uint64_t* loc_kmer, const uint32_t* loc_contig,
                    const uint32_t* loc_start, const uint32_t* loc_group, uint64_t n_loc,
                    uint32_t n_contigs);

/* Replaces workflow/rules/defineSUNKs.smk:1-127 (combine_asm_haps, jellyfish count -C -U 1,
 * define_SUNKs, mrsfast index/search -e 0, bed_convert): canonical k-mers of the concatenated
 * assembly that occur exactly once, their location and the start of their merged
 * (overlapping-or-book-ended) run.  seq = concatenated contig sequences (ASCII, any case, non-ACGT
 * breaks windows), contig_off[n_contigs+1] = offsets into seq.  `seq_on_device` != 0: both
 * pointers are device memory.  Any k from 1 to 32; contigs that are empty or shorter than k contribute no
 * window, and an assembly without a SUNK gives an empty database (gvs_db_size 0, 0). */
int gvs_db_build(gvs_ctx* ctx, const uint8_t* seq, const uint64_t* contig_off, uint32_t n_contigs,
                 int seq_on_device);

/* The probe kernel has two instantiations, chosen by the size of the database when it is loaded / built: one for
 * databases whose blocked filter stays L2-resident (<= 32 MiB) and one for larger ones (sub-mer fingerprint in
 * every filter block, grouped block loads).  variant = 0: by size (default), 1: small-database, 2: large-database
 * -- results are identical; tests force either one on the golden cases.  Takes effect at the next
 * gvs_db_load_loc / gvs_db_build (the filter layout is part of the database). */
int gvs_set_probe_variant(gvs_ctx* ctx, int variant);

/* gvs_db_build hash-partitions the canonical k-mers into n passes over the assembly, each with its own count table
 * of (total / n) * 3/2 + 1024 slots.  n = 0 (default): the fewest passes whose table fits 70 % of the free device
 * memory (by that formula two for a 2 x 3.1 Gbp diploid assembly on a 180 GB GPU); n = 1..64: exactly n passes,
 * whatever the memory (GVS_E_NOMEM if the table does not fit).  The database does not depend on n; tests force it
 * to reach the multi-pass build on small assemblies.  Takes effect at the next gvs_db_build. */
int gvs_set_db_passes(gvs_ctx* ctx, int n);

int gvs_db_size(gvs_ctx* ctx, uint64_t* n_sunks, uint64_t* n_groups);
/* kmer.loc rows in file order ((contig, start) order for a built database): host buffers of
 * n_sunks entries each; any pointer may be NULL. */
int gvs_db_export(gvs_ctx* ctx, uint64_t* kmer, uint32_t* contig, uint32_t* start,
                  uint32_t* group, uint32_t* group_index);

/* ------------------------------------------------------------------------------------------ */
/* reads                                                                                       */
/* Host ingest of FASTA/FASTQ(.gz) read files (the `readfq` loop of workflow/src/kmerpos_annot3.nim:85 and
 * workflow/src/rlen.nim:13-14; chunk files of workflow/rules/tagONT.smk:17): every file is one chunk, files
 * are decompressed and parsed on `threads` host threads and laid out back to back in one host buffer
 * (page-locked when pin != 0 and a CUDA device exists, so that gvs_reads_set can overlap the copy with
 * the probe).  All arrays are owned by the library until gvs_fastx_free.  No context needed. */
typedef struct gvs_fastx {
  void* impl;
  const uint8_t* seq;          /* total_bases ASCII bytes (+ 64 zero bytes of slack)               */
  const uint64_t* read_off;    /* n_reads + 1                                                     */
  const char* names;           /* read names back to back (no terminators)                        */
  const uint64_t* name_off;    /* n_reads + 1 offsets into names                                  */
  const uint64_t* chunk_first; /* n_files + 1 read indices: file i = reads [chunk_first[i], [i+1]) */
  uint64_t n_reads, total_bases;
  uint32_t n_files;
  int pinned;
  const uint32_t* words;       /* after gvs_fastx_pack: the same bases as 2-bit words (see gvs_reads_set_packed) */
  uint64_t n_words;
} gvs_fastx;
int gvs_fastx_read(const char* const* paths, uint32_t n_files, int threads, int pin, gvs_fastx* out,
                   char* err, uint64_t err_len);
void gvs_fastx_free(gvs_fastx* fx);
/* kmer.encode's byte map (nim-kmer 0.2.6: A/a 0, C/c 1, G/g 2, T/t/U/u 3, bytes 1..3 themselves, everything
 * else 0 -- workflow/src/kmerpos_annot3.nim:88 `slide`) applied on the host: n ASCII bases -> ceil(n/16)
 * big-endian words of 16 bases (first base in the top two bits, tail zero-padded).  Lossless for this path
 * and a quarter of the bytes to move over PCIe.  gvs_fastx_pack does it for a parsed batch (page-locked). */
int gvs_pack_2bit(const uint8_t* ascii, uint64_t n, uint32_t* words, int threads);
int gvs_fastx_pack(gvs_fastx* fx, int threads, int pin);
/* The ingest's native path: parse and 2-bit pack fused.  Same record semantics and chunk layout as gvs_fastx_read,
 * but the ASCII bases never land in memory as a batch: files are streamed in blocks of `block_bytes` (0 = 1 MiB;
 * plain files out of the page cache through mmap, gzip files through an inflate window of that size), packed with
 * kmer.encode's byte map as they are parsed and laid out as ONE (page-locked) array of 16-base words --
 * out->words / n_words, ready for gvs_reads_set_packed; out->seq stays NULL.  Free with gvs_fastx_free. */
int gvs_fastx_read_packed(const char* const* paths, uint32_t n_files, int threads, int pin, uint64_t block_bytes,
                          gvs_fastx* out, char* err, uint64_t err_len);

/* ------------------------------------------------------------------------------------------ */
/* Text egress at the reference's file boundary (SURVEY.md Appendix C): rows of .sunkpos (kmerpos_annot3.nim:93), */
/* .rlen (rlen.nim:14), kmer.loc / jellyfish.db / jellyfish.fa (defineSUNKs.smk:59-60,126), inter_outs / BED files  */
/* (process-by-contig_lowmem_AR.py:203-207,260) formatted from column arrays on host threads.  Host memory only.  */
/* ------------------------------------------------------------------------------------------ */
enum { GVS_COL_U32 = 0, GVS_COL_U64 = 1, GVS_COL_I64 = 2, GVS_COL_NAME = 3, GVS_COL_KMER = 4 };
typedef struct gvs_col {
  int32_t kind;              /* GVS_COL_*                                                                  */
  int32_t k;                 /* GVS_COL_KMER: letters per k-mer (2-bit big-endian value, A C G T)         */
  const void* data;          /* per row: the u32 / u64 / i64 value, the u32 index into the name table, the u64 k-mer */
  const char* names;         /* GVS_COL_NAME: names back to back ...                                       */
  const uint64_t* name_off;  /* ... and their offsets (entries + 1)                                        */
  char prefix;               /* written before the cell when non-zero ('>' of jellyfish.fa)                */
  char sep;                  /* written after the cell: '\t', or '\n' for the last column                  */
} gvs_col;
/* Formats rows [0, n_rows) -- or, with sel != NULL, the n_sel rows sel[i] in that order (one contig's rows of a
 * batch) -- as n_cols cells each.  out == NULL: returns the number of bytes needed; otherwise writes them (no
 * terminator) and returns the count, GVS_E_OVERFLOW when cap is too small. */
int64_t gvs_format_rows(const gvs_col* cols, uint32_t n_cols, uint64_t n_rows, const uint64_t* sel, uint64_t n_sel, char* out,
                        uint64_t cap, int threads);

/* ------------------------------------------------------------------------------------------ */
/* A batch = the reads of one or more chunk files (temp/{sample}/reads/{hap}_{i-of-N}.fq.gz,
 * workflow/rules/tagONT.smk:17), concatenated in file order.
 *   seq            ASCII bases of all reads back to back (no separators)
 *   read_off       n_reads+1 offsets into seq
 *   chunk_first    n_chunks+1 read indices: chunk c = reads [chunk_first[c], chunk_first[c+1]);
 *                  the kmerpos_annot3 `prevLoc` carry (nim:82-84, SURVEY Q4) restarts per chunk
 *   chunk_hap      n_chunks entries, the haplotype (0/1) whose .fai the chunk's reads are
 *                  filtered against (workflow/rules/tagONT.smk:79,92), or GVS_HAP_ANY: unbinned reads,
 *                  whose haplotype the diag filter assigns from their SUNK votes (gvs_diag_filter_haps)
 * on_device != 0: seq and read_off are device pointers that stay valid until the next
 * gvs_reads_* call (no copy is made); chunk arrays are always host memory.
 * With on_device == 0 the arrays are copied host->device on the context's stream. */
enum { GVS_HAP_ANY = 2 };
int gvs_reads_set(gvs_ctx* ctx, const uint8_t* seq, const uint64_t* read_off, uint64_t n_reads,
                  const uint64_t* chunk_first, const uint8_t* chunk_hap, uint32_t n_chunks,
                  int on_device);

/* The same batch with the bases already packed by gvs_pack_2bit / gvs_fastx_pack (words: ceil(total/16)
 * uint32; read_off still counts bases).  The probe then skips its own ASCII -> 2-bit step. */
int gvs_reads_set_packed(gvs_ctx* ctx, const uint32_t* words, const uint64_t* read_off, uint64_t n_reads,
                         const uint64_t* chunk_first, const uint8_t* chunk_hap, uint32_t n_chunks,
                         int on_device);

/* Host batches of at least `min_bytes` are copied in `segments` pieces on a second stream and the
 * probe of each piece starts as soon as it has landed (PCIe transfer overlapped with the match).
 * Defaults: 256 MiB, 16.  segments <= 1 disables the pipeline. */
int gvs_set_copy_pipeline(gvs_ctx* ctx, uint64_t min_bytes, uint32_t segments);

/* How the segments of a pipelined ASCII host batch (gvs_reads_set, on_device == 0) reach the GPU.  The
 * reference reads one ASCII byte per base (readfq, workflow/src/kmerpos_annot3.nim:85); the PCIe link moves
 * those at ~55 GB/s, so a segment may instead be packed to 2 bits per base on `threads` host threads
 * (kmer.encode's byte map, as gvs_pack_2bit) into page-locked staging memory and copied at a quarter of the
 * bytes, after which the PACKED probe variant scans it.  Results are identical either way.
 *   GVS_PACK_OFF       every segment as ASCII (the host cores stay idle)
 *   GVS_PACK_ADAPTIVE  (default) a segment goes out as ASCII while the link has less queued than one
 *                      segment takes to pack, and is packed otherwise: link and cores work side by side;
 *                      a buffer that is not page-locked is always packed
 *   GVS_PACK_ALL       every segment packed
 *   GVS_PACK_ALTERNATE odd segments packed (tests: both kinds in one batch, deterministic)
 * threads = 0: the cores this process may run on, at most 16.  Processes that share one host should split its
 * cores (threads = cores / processes) and switch the packing off below ~12 threads each: packers and DMA reads
 * share the host's memory bandwidth (8 x 4 threads measured 8 % slower than ASCII copies, profiles/README.md).
 * With packing enabled a background thread of
 * the library reads `seq` until gvs_match has returned: the buffer must stay unchanged until then (the same
 * holds for the asynchronous copies of GVS_PACK_OFF). */
enum { GVS_PACK_OFF = 0, GVS_PACK_ADAPTIVE = 1, GVS_PACK_ALL = 2, GVS_PACK_ALTERNATE = 3 };
int gvs_set_host_pack(gvs_ctx* ctx, int mode, int threads);
/* What the last host batch put on the link: sequence bytes copied, segments, segments sent packed (valid
 * once gvs_match has returned). */
int gvs_copy_stats(gvs_ctx* ctx, uint64_t* h2d_bytes, uint32_t* segments, uint32_t* segments_packed);

/* Read table without sequences (the CLI shims that start from .sunkpos / .rlen files):
 * read_len[n_reads] = column 2 of {hap}.rlen (workflow/src/rlen.nim:13-14), chunk layout as above. */
int gvs_reads_meta(gvs_ctx* ctx, const uint32_t* read_len, uint64_t n_reads, const uint64_t* chunk_first,
                   const uint8_t* chunk_hap, uint32_t n_chunks);
/* Rows parsed from a .sunkpos file instead of produced by the previous stage: which = 0 replaces
 * the output of gvs_match (input of gvs_diag_filter: workflow/src/diag_filter_v3.nim:63), which = 1
 * replaces the output of gvs_diag_filter (input of gvs_group_hist / gvs_validate:
 * badsunks_AR.py:20, process-by-contig_lowmem_AR.py:60).  Rows of one read must be contiguous.
 * With a database loaded every (contig, group) must exist in it; without one the group index is
 * derived from the rows (first appearance order) and n_contigs sizes the contig tables. */
int gvs_rows_set(gvs_ctx* ctx, int which, const uint32_t* read_idx, const uint32_t* pos, const uint32_t* contig,
                 const uint32_t* start, const uint32_t* group, uint64_t n_rows, uint32_t n_contigs);

/* ------------------------------------------------------------------------------------------ */
/* stages (must be called in this order; each consumes the previous stage's device results)    */
/* ------------------------------------------------------------------------------------------ */
/* kmerpos_annot3 main loop (workflow/src/kmerpos_annot3.nim:81-97): sunkpos rows
 * (read, pos, contig, start, group) with the consecutive-(contig,group) suppression and the
 * position drift it causes (SURVEY Q3-Q6). */
int gvs_match(gvs_ctx* ctx, uint64_t* n_rows);
/* which: 0 = rows of gvs_match ({hap}_{i}.sunkpos), 1 = rows kept by gvs_diag_filter
 * ({hap}_{i}_diag2.sunkpos).  Host buffers of n_rows entries; any may be NULL. */
int gvs_rows_get(gvs_ctx* ctx, int which, uint32_t* read_idx, uint32_t* pos, uint32_t* contig,
                 uint32_t* start, uint32_t* group);

/* diag_filter_v3 (workflow/src/diag_filter_v3.nim:18-229) + diag_filter_step2
 * (workflow/src/diag_filter_step2.nim:13-66).
 *   contig_hap[n_contigs]   haplotype (0/1) whose .fai lists the contig, 255 = in neither
 *                           (gvs_bad_groups also knows 2/3 = "contig of the other assembly, thresholded
 *                           with haplotype 0/1's limit", badsunks_AR.py:51)
 *   contig_hash[n_contigs]  Nim `hash(name)` of the contig name (MurmurHash3_x86_32, seed 0,
 *                           0 remapped) -- decides ties through Table iteration order (SURVEY Q9)
 * n_best = reads that got a best contig, n_kept = rows that survive. */
int gvs_diag_filter(gvs_ctx* ctx, const uint8_t* contig_hap, const uint32_t* contig_hash,
                    uint64_t* n_best, uint64_t* n_kept);
/* Read haplotypes: the diag filter's vote taken once per haplotype.  No reference counterpart.  For a read r and a
 * haplotype h:
 *   vote_h(r)    the (contig, n, dir) diag_filter_v3 prints for r when it runs over r's chunk with haplotype h's .fai
 *                (candidates limited to the contigs of h; the Table replay of ties still holds every contig of the
 *                read, so slot order and the capacity carried through the chunk do not depend on h); no vote when
 *                maxgood <= 1.  n_h = n, or 0 without a vote;
 *   assigned(r)  h when n_h > n_(1-h), tie when n_0 == n_1 >= 2, none when both are 0.
 * Reads of a binned chunk (haplotype 0/1) keep their rows exactly as gvs_diag_filter keeps them, from the vote of
 * the chunk's haplotype; the other vote is only reported.  Reads of a GVS_HAP_ANY chunk keep their rows on
 * vote_assigned(r)'s contig; a tie or none read keeps no rows and has no best row.
 * Haplotype mode is on when read_haps != 0 or a chunk of the batch is GVS_HAP_ANY; with it off gvs_diag_filter_haps
 * is gvs_diag_filter.  With it on, the filter also writes one record per read with n_0 >= 2 or n_1 >= 2, in read
 * order: read, contig1, n1, strand1, contig2, n2, strand2, hap (contig 0xFFFFFFFF and n 0 without a vote; strand 0
 * '+', 1 '-'; hap 0 / 1 / 2 = tie).  gvs_batch_stash appends them to the run's records with run-wide read indices,
 * which gvs_batches_bind makes current.  gvs_read_haps: *n_records of the last filter in haplotype mode (or of the
 * run after gvs_batches_bind); gvs_read_haps_get: host buffers of *n_records entries, any pointer may be NULL. */
int gvs_diag_filter_haps(gvs_ctx* ctx, const uint8_t* contig_hap, const uint32_t* contig_hash, int read_haps,
                         uint64_t* n_best, uint64_t* n_kept);
int gvs_read_haps(gvs_ctx* ctx, uint64_t* n_records);
int gvs_read_haps_get(gvs_ctx* ctx, uint32_t* read, uint32_t* contig1, uint32_t* n1, uint32_t* strand1, uint32_t* contig2,
                      uint32_t* n2, uint32_t* strand2, uint32_t* hap);
/* rows of {hap}_{i}_diag.sunkpos: read, contig, n, dir (0 = '-', 1 = '+') */
int gvs_best_get(gvs_ctx* ctx, uint32_t* read_idx, uint32_t* contig, uint32_t* ngood,
                 uint8_t* dir);

/* diag_filter_step2 on its own (workflow/src/diag_filter_step2.nim:13-66): best_contig_of_read[n_reads]
 * parsed from a {hap}_{i}_diag.sunkpos file (0xFFFFFFFF = read has no best contig); keeps the rows of
 * gvs_match / gvs_rows_set(0) whose contig equals it -> gvs_rows_get(1). */
int gvs_filter_best(gvs_ctx* ctx, const uint32_t* best_contig_of_read, uint64_t* n_kept);

/* Contig tables for callers that skip gvs_diag_filter (which sets them itself): contig_hap as
 * above (badsunks_AR.py:28-33 "correct" = contig listed in the haplotype's .fai), contig_hash may
 * be NULL. */
int gvs_contigs_set(gvs_ctx* ctx, const uint8_t* contig_hap, const uint32_t* contig_hash,
                    uint32_t n_contigs);

/* badsunks_AR.py:20-52 histogram: rows per (contig, group) over the kept rows, accumulated into a
 * device array of n_groups int32 (index = group_index of gvs_db_export).  *hist_dev receives the
 * device pointer so that the caller can all-reduce it across GPUs (NCCL) before
 * gvs_bad_groups.  accumulate != 0 adds to the previous histogram (several batches). */
int gvs_group_hist(gvs_ctx* ctx, int accumulate, int32_t** hist_dev);
/* mode of the non-zero counts per haplotype (badsunks_AR.py:43, smallest mode) */
int gvs_hist_mode(gvs_ctx* ctx, int64_t mode[2]);
/* bad group <=> count > limit[hap] or count < 2 (badsunks_AR.py:46-52); limit is computed by the
 * caller exactly as the reference does (m + 4*sqrt(m) in float64) and passed as floor(limit). */
int gvs_bad_groups(gvs_ctx* ctx, const int64_t limit_floor[2], uint64_t* n_bad);
int gvs_bad_get(gvs_ctx* ctx, uint32_t* group_index /* n_bad entries */);
/* Bad groups read from a bad_sunks.txt instead of computed here (process-by-contig_lowmem_AR.py:66-72,
 * `ID2 not in @badsunkin`): n (contig, group) pairs in host memory; pairs that name no known group are
 * ignored like the reference's string set does.  *n_bad = groups flagged. */
int gvs_bad_set(gvs_ctx* ctx, const uint32_t* contig, const uint32_t* group, uint64_t n, uint64_t* n_bad);
/* The group table behind every group_index: (contig, group start) and, when hist != NULL, the row
 * count of gvs_group_hist (badsunks_AR.py:24-27 `counts`).  Host buffers of gvs_groups_count entries. */
int gvs_groups_count(gvs_ctx* ctx, uint64_t* n_groups);
int gvs_groups_get(gvs_ctx* ctx, uint32_t* contig, uint32_t* group, int32_t* hist);

/* ------------------------------------------------------------------------------------------ */
/* Several batches of ONE run.  The reference scatters a sample's reads into chunk files, matches and
 * filters per chunk and gathers per haplotype before anything global happens (workflow/Snakefile:23-24
 * scattergather, workflow/rules/tagONT.smk:112-131 combine_ont): badsunks_AR.py:20-27 counts the rows of ALL
 * chunks, process-by-contig_lowmem_AR.py sees every read of a contig.  A run whose reads do not fit one batch
 * has two phases:
 *   gvs_batches_begin
 *   per batch:  gvs_reads_set* -> gvs_match -> gvs_diag_filter -> gvs_group_hist(accumulate = 1) -> gvs_batch_stash
 *   (several GPUs: ONE all-reduce of the histogram)  gvs_hist_mode -> gvs_bad_groups
 *   gvs_batches_bind -> gvs_validate -> gvs_components_local
 *   (several GPUs: ONE all-gather of the forests, gvs_components_merge_all)  gvs_intervals -> gvs_gaps
 * gvs_batch_stash keeps the batch's kept rows (24 B each) and read lengths resident and returns the index its
 * first read has in the run (*read_base); gvs_batches_bind makes the stashed rows of all batches the input of
 * gvs_validate (as if one gvs_diag_filter had kept them; gvs_rows_get(1) / gvs_pairs_get then report run-wide
 * read indices) and ends the run's phase 1. */
int gvs_batches_begin(gvs_ctx* ctx);
int gvs_batch_stash(gvs_ctx* ctx, uint64_t* read_base);
int gvs_batches_bind(gvs_ctx* ctx, uint64_t* n_rows, uint64_t* n_reads);

/* process-by-contig_lowmem_AR.py:50-207 per-read part: validated (group, read) pairs = rows of
 * inter_outs/{contig}_{hap}.tsv.  min_read_len is the reference's hard-coded 10000 (:106). */
int gvs_validate(gvs_ctx* ctx, uint32_t min_read_len, uint64_t* n_pairs);
int gvs_pairs_get(gvs_ctx* ctx, uint32_t* read_idx, uint32_t* contig, uint32_t* group,
                  uint32_t* group_index);
/* after gvs_validate: *n_empty = reads of the last validation whose multipos clean-up dropped every oriented edge
 * (the reference would build an empty graph and raise there; such a read validates nothing). */
int gvs_validate_stats(gvs_ctx* ctx, uint64_t* n_empty);

/* process-by-contig_lowmem_AR.py:215-260 contig-wide components.  The union-find parent array
 * (n_groups uint32, index = group_index) is exposed so that several GPUs can merge their
 * forests: gvs_components_local builds this GPU's forest from singletons, gvs_components_merge_all
 * unions in every peer's forest in one pass, gvs_intervals finalises.  gathered_dev = the all-gathered
 * parent arrays on this GPU, rank r's at gathered_dev + r * n_groups (own_rank's slice is skipped and
 * may be left unwritten). */
int gvs_components_local(gvs_ctx* ctx, uint32_t** parent_dev);
int gvs_components_merge_all(gvs_ctx* ctx, const uint32_t* gathered_dev, uint32_t n_ranks, uint32_t own_rank);
/* validated intervals (contig, min group, max group) of components with >= 3 groups, sorted by
 * (contig, start) = rows of bed_files/{contig}_{hap}.bed */
int gvs_intervals(gvs_ctx* ctx, uint64_t* n_intervals);
int gvs_intervals_get(gvs_ctx* ctx, uint32_t* contig, uint32_t* start, uint32_t* end);

/* Support tracks of the validated reads.  No reference counterpart: the reference only draws pile-up plots
 * (viz.py, viz_detailed.py); these are text tracks for genome browsers and assembly QC.
 * A placement is a read with >= 2 validated IDs (the reads that join groups in gvs_components_local):
 * start / end = its smallest / largest validated ID (group starts, the convention of the intervals), n_ids = its
 * validated IDs, strand = 0 when its orientation majority is 0 (read positions rise with assembly starts), else 1.
 * gvs_placements runs after gvs_validate.  *diff_dev receives an int32 array of n_groups entries indexed by the
 * group's rank in (contig, start) order (+1 at a placement's first group, -1 at its last), zero without
 * placements: several GPUs sum it (like the histogram of gvs_group_hist) before gvs_support.
 * gvs_placements_get: host buffers of *n entries, any pointer may be NULL; read_idx is run-wide as in
 * gvs_pairs_get; placements come in segment (read) order. */
int gvs_placements(gvs_ctx* ctx, uint64_t* n, int32_t** diff_dev);
int gvs_placements_get(gvs_ctx* ctx, uint32_t* read_idx, uint32_t* contig, uint32_t* start, uint32_t* end, uint32_t* n_ids,
                       uint8_t* strand);
/* Support depth from the (summed) difference array: the number of placements with start <= x < end at every
 * base x, as runs (contig, start, end, depth) that tile [0, contig_len[c]) of every contig c (n_contigs
 * entries, host memory) in (contig, start) order, maximal (adjacent runs of a contig differ in depth). */
int gvs_support(gvs_ctx* ctx, const uint32_t* contig_len, uint64_t* n_runs);
int gvs_support_get(gvs_ctx* ctx, uint32_t* contig, uint32_t* start, uint32_t* end, uint32_t* depth);

/* Distance discordance: collapses and expansions inside validated intervals.  No reference counterpart.  The validation's
 * ratio test passes a SUNK pair whose distances agree within 10 %, so a read validates across an event smaller than about a
 * tenth of its reach; the spacing of its SUNKs still shows the event.
 * Inputs: the kept rows (read, pos, contig, start, ID = group) of gvs_diag_filter / gvs_batches_bind / gvs_rows_set(1) minus
 * the rows of bad groups (when set), and the validated IDs of each read from gvs_validate (which must have run; its
 * min_read_len applies).  Per read (validation segment), on its rows of the contig of its first row:
 *   usable row  a non-bad row whose ID is one of the read's validated IDs and which is the read's only non-bad row with
 *               that ID (repeated IDs are ambiguous and skipped);
 *   order       usable rows by (start, ID) -- distinct starts, as different groups cover disjoint start ranges;
 *   span        each pair (a, b) of consecutive usable rows: dstart = start_b - start_a, dpos = |pos_b - pos_a|,
 *               delta = dpos - dstart (signed, as gap evidence);
 *   covers      segment r = [ID_r, ID_r+1) of a contig, r the group's rank in (contig, start) order, for
 *               rank(ID_a) <= r < rank(ID_b): every span that covers a segment contains all of it;
 *   class       longer when 1000*delta >= 1000*min_delta + rel_permille*dstart (the read has more sequence: collapse in
 *               the assembly), else shorter when -1000*delta meets the same bound (expansion), else concordant.
 * gvs_spans: *diff_dev receives int32[3][n_groups] by rank -- spans, longer, shorter -- with +1 at rank(ID_a) and -1 at
 * rank(ID_b) of every span of its kind (zero without spans): several GPUs sum its 3*n_groups entries (as the histogram of
 * gvs_group_hist) before gvs_discordance.  Records: one per non-concordant span, in (segment, span) order: read (run-wide,
 * as in gvs_pairs_get), contig, (id1, start1, pos1) of a, (id2, start2, pos2) of b; longer iff delta >= 0.
 * rel_permille <= 1000000.  gvs_spans_get: host buffers of *n_records entries, any pointer may be NULL.
 * gvs_discordance: per base x, the spans covering x's segment, as runs (contig, start, end, spans, longer, shorter) that
 * tile [0, contig_len[c]) of every contig in (contig, start) order, maximal (adjacent runs of a contig differ in one of
 * the three), with a zero head run before a contig's first group as gvs_support tiles the depth. */
int gvs_spans(gvs_ctx* ctx, uint32_t min_delta, uint32_t rel_permille, uint64_t* n_records, int32_t** diff_dev);
int gvs_spans_get(gvs_ctx* ctx, uint32_t* read, uint32_t* contig, uint32_t* id1, uint32_t* start1, uint32_t* pos1, uint32_t* id2,
                  uint32_t* start2, uint32_t* pos2);
int gvs_discordance(gvs_ctx* ctx, const uint32_t* contig_len, uint64_t* n_runs);
int gvs_discordance_get(gvs_ctx* ctx, uint32_t* contig, uint32_t* start, uint32_t* end, uint32_t* spans, uint32_t* longer,
                        uint32_t* shorter);

/* Intervals parsed from bed_files/{contig}_{hap}.bed instead of produced by gvs_intervals (the input
 * of get_gaps.py:30); any order, host memory. */
int gvs_intervals_set(gvs_ctx* ctx, const uint32_t* contig, const uint32_t* start, const uint32_t* end,
                      uint64_t n, uint32_t n_contigs);

/* get_gaps.py:17-123: per contig merge intervals, gaps (prev_end, next_start-1); contigs without
 * intervals are "nodata".  contig_len[n_contigs]. */
int gvs_gaps(gvs_ctx* ctx, const uint32_t* contig_len, uint64_t* n_gaps, uint64_t* n_nodata);
int gvs_gaps_get(gvs_ctx* ctx, uint32_t* contig, uint32_t* start, uint32_t* end,
                 uint32_t* nodata_contig);

/* Gap evidence: the reads that cross each gap without validating it.  No reference counterpart: the reference only
 * draws pile-up plots (viz.py); this tells a gap without data from a gap the reads disagree with.
 * Inputs: the kept rows (read, pos, contig, start, ID = group) of gvs_diag_filter / gvs_batches_bind / gvs_rows_set(1)
 * minus the bad groups (when set), reads of length >= min_read_len, and the gaps of gvs_gaps (which must have run;
 * gvs_validate need not).  A read's rows are those of its segment on the contig of its first row (gvs_diag_filter
 * keeps one contig per read; callers of gvs_rows_set key reads by (contig, name)).  Per gap (contig, gs, ge) and read:
 *   left row  ID <= gs, right row ID >= ge + 1 (sides by ID, as intervals are built from IDs);
 *   anchored  another row of the same side with a different ID passes 9*|dstart| < 10*|dpos| < 11*|dstart| with it
 *             (the validation's ratio test, process-by-contig_lowmem_AR.py:145-147, Q12);
 *   bridging  at least one anchored left row and one anchored right row;
 *   flanks    the anchored left row with the largest start (ties: smallest pos, then smallest ID) and the anchored
 *             right row with the smallest start (ties: smallest pos, then smallest ID).
 * One record per bridging (read, gap), in (read segment, gap) order.  gvs_gap_evidence_get: host buffers of
 * *n_records entries, any pointer may be NULL; read is run-wide as in gvs_pairs_get, gap indexes the arrays of
 * gvs_gaps_get.  The size change is the caller's: delta = |right_pos - left_pos| - (right_start - left_start). */
int gvs_gap_evidence(gvs_ctx* ctx, uint32_t min_read_len, uint64_t* n_records);
int gvs_gap_evidence_get(gvs_ctx* ctx, uint32_t* read, uint32_t* gap, uint32_t* left_id, uint32_t* left_start,
                         uint32_t* left_pos, uint32_t* right_id, uint32_t* right_start, uint32_t* right_pos);

/* Junctions: reads whose SUNKs jump from one contig to another (contig-end links, misjoins, haplotype switches).  No
 * reference counterpart: the diag filter keeps each read's rows on one best contig, and every later stage sees only those.
 * Inputs: the rows (read, pos, contig, start, ID = group) of gvs_match / gvs_rows_set(0), in row order (gvs_match: pos
 * ascending within a read), minus the rows of bad groups when bad groups are set, reads of length >= min_read_len.
 * Every contig counts, both haplotypes included; the diag filter's choice plays no part.  Per read:
 *   anchored     a row is anchored when another row of the read on the same contig with a different ID passes
 *                9*|dstart| < 10*|dpos| < 11*|dstart| with it (the validation's ratio test, process-by-contig_lowmem_AR.py:145-147, Q12);
 *   qualifying   a contig on which the read has >= 3 distinct anchored IDs;
 *   blocks       the anchored rows of qualifying contigs, in row order, cut into maximal runs on one contig; runs of fewer
 *                than 3 distinct IDs are dropped, then runs left adjacent on the same contig are merged (one pass);
 *   strand       of a block: over the pairs of its rows with different IDs that pass the ratio test, 0 ('+') when at least
 *                half have positions rising with starts, else 1 ('-');
 *   records      one per consecutive block pair (B_i, B_i+1): read (run-wide, as in gvs_pairs_get), contig1, strand1,
 *                ids1 (distinct IDs of B_i), (id1, start1, pos1) of B_i's last row, contig2, strand2, ids2,
 *                (id2, start2, pos2) of B_i+1's first row; in (read, block) order.  Consecutive blocks lie on different
 *                contigs: two clusters on one contig with no other contig between them give no record.
 * gvs_junction_screen runs per batch between gvs_match (or gvs_rows_set(0)) and gvs_batch_stash: without bad groups
 * it keeps the anchored rows of qualifying contigs of the reads with >= 2 qualifying contigs, with the read indices
 * gvs_batch_stash gives the batch (exact: removing bad rows only removes anchors, and an anchor's partner is itself
 * anchored).  gvs_batches_begin empties that stash and the screens of the run append to it; outside a batches run a
 * screen replaces it.  *stash_rows / *stash_reads (may be NULL) = its size afterwards.  The screen writes no buffer of
 * the other stages (rows(0), rows(1), gvs_best_get and the diag filter's segments stay as they were).
 * gvs_junctions resolves the stash with the bad groups of gvs_bad_groups / gvs_bad_set (or none).
 * gvs_junctions_get: host buffers of *n_records entries, any pointer may be NULL. */
int gvs_junction_screen(gvs_ctx* ctx, uint32_t min_read_len, uint64_t* stash_rows, uint64_t* stash_reads);
int gvs_junctions(gvs_ctx* ctx, uint64_t* n_records);
int gvs_junctions_get(gvs_ctx* ctx, uint32_t* read, uint32_t* contig1, uint32_t* strand1, uint32_t* ids1, uint32_t* id1,
                      uint32_t* start1, uint32_t* pos1, uint32_t* contig2, uint32_t* strand2, uint32_t* ids2, uint32_t* id2,
                      uint32_t* start2, uint32_t* pos2);

/* Strand switches: reads whose SUNKs switch strand inside one contig (inversions, fold-back chimeras).  No reference
 * counterpart: the validation takes each read's orientation majority (process-by-contig_lowmem_AR.py:151-152) and an
 * inversion keeps its length, so a read validates straight across it.
 * Inputs: the kept rows (read, pos, contig, start, ID = group) of gvs_diag_filter / gvs_batches_bind / gvs_rows_set(1)
 * minus the rows of bad groups (when set), reads of length >= min_read_len; a read's rows are those of its segment on
 * the contig of its first row (as gvs_gap_evidence takes them).  Per read:
 *   order    rows by ascending pos, ties in row order (gvs_match rows already are: positions rise within a read);
 *   strand   of row i: over the read's rows j with a different ID that pass 9*|dstart| < 10*|dpos| < 11*|dstart| with
 *            it, up_i = pairs with (pos_j > pos_i) == (start_j > start_i), down_i = the others; 0 ('+') when up_i >
 *            down_i, 1 ('-') when down_i > up_i, else unoriented (also a row without a partner);
 *   blocks   the oriented rows, in order, cut into maximal runs of one strand; runs of fewer than 3 distinct IDs are
 *            dropped, then runs left adjacent with one strand are merged (one pass: the junction rule with strand in
 *            place of contig);
 *   records  one per consecutive block pair (B_i, B_i+1), whose strands differ: read (run-wide, as in gvs_pairs_get),
 *            contig, strand1, ids1 (distinct IDs of B_i), lo1 / hi1 (smallest / largest start of B_i), (id1, start1,
 *            pos1) of B_i's last row, strand2, ids2, lo2, hi2, (id2, start2, pos2) of B_i+1's first row; in (read,
 *            block) order.
 * An inversion [x, y) makes every read across a breakpoint give a record with {start1, start2} near {x, y}; a fold-back
 * chimera (a read followed by its reverse complement) gives one whose blocks overlap on the assembly.
 * gvs_strand_switches_get: host buffers of *n_records entries, any pointer may be NULL. */
int gvs_strand_switches(gvs_ctx* ctx, uint32_t min_read_len, uint64_t* n_records);
int gvs_strand_switches_get(gvs_ctx* ctx, uint32_t* read, uint32_t* contig, uint32_t* strand1, uint32_t* ids1, uint32_t* lo1,
                            uint32_t* hi1, uint32_t* id1, uint32_t* start1, uint32_t* pos1, uint32_t* strand2, uint32_t* ids2,
                            uint32_t* lo2, uint32_t* hi2, uint32_t* id2, uint32_t* start2, uint32_t* pos2);

/* SUNK hit depth: how many copies the reads say each SUNK group has.  No reference counterpart: badsunks_AR.py removes the
 * groups with too many kept rows (a collapse of c genomic copies gives its SUNKs about c times the hits) and validation
 * then reports a gap there.  Per group index g (the group table of gvs_db_export / gvs_groups_get):
 *   hits[g]   the match rows of gvs_match / gvs_rows_set(0) with group g: every contig of both haplotypes, every read, no
 *             read-length minimum, no bad-group filter (the rows of combine_ont_nofilt, before the diag filter keeps one
 *             contig per read: reads from a collapsed copy elsewhere often have their best contig elsewhere);
 *   reads[g]  the distinct read records among those rows: a read counts once per group however often it re-enters it;
 *   kept[g]   the histogram of gvs_group_hist (kept rows per group, summed over ranks);
 *   sunks[g]  the .loc rows of group g.
 * An interspersed collapse (copies at other loci) raises hits and reads; a tandem collapse raises hits only (each read
 * crosses the one assembled copy several times).
 * gvs_sunk_depth adds the current match rows (none after gvs_batches_bind or before any gvs_match) to an int32[2][n_groups]
 * array -- hits at [g], reads at [n_groups + g] -- whose device pointer *depth_dev receives.  Inside a batches run it
 * accumulates from gvs_batches_begin on (accumulate != 0); accumulate = 0 replaces.  It writes no buffer of the other
 * stages.  Several GPUs sum the 2*n_groups entries (as the histogram of gvs_group_hist; a read lives on one GPU, so the
 * sums are exact) before gvs_sunk_depth_get / gvs_depth_runs.
 * gvs_sunk_depth_get: host buffers of n_groups entries, any pointer may be NULL.
 * gvs_depth_runs: per base x, the (hits, reads, kept) of x's segment [ID_r, ID_r+1) as runs (contig, start, end, hits, reads,
 * kept) that tile [0, contig_len[c]) of every contig in (contig, start) order, maximal, with a zero head run before a
 * contig's first group (as gvs_discordance tiles its counts).  GVS_E_STATE before gvs_group_hist or gvs_sunk_depth.
 * The calls (collapsed and depleted stretches) are the caller's: DESIGN.md section 5.5g. */
int gvs_sunk_depth(gvs_ctx* ctx, int accumulate, int32_t** depth_dev);
int gvs_sunk_depth_get(gvs_ctx* ctx, int32_t* hits, int32_t* reads, uint32_t* sunks);
int gvs_depth_runs(gvs_ctx* ctx, const uint32_t* contig_len, uint64_t* n_runs);
int gvs_depth_runs_get(gvs_ctx* ctx, uint32_t* contig, uint32_t* start, uint32_t* end, uint32_t* hits, uint32_t* reads,
                       uint32_t* kept);

/* Allele support: whether the reads of each SUNK group's own haplotype carry it, the other haplotype's reads carry it,
 * or no read does.  No reference counterpart.  At a heterozygous site the haplotypes' k-mers differ, so each haplotype
 * has a group of its own there that only its reads should carry.
 * Read haplotype hap(r): the file haplotype of read r (the haplotype whose sunkpos/ files hold it, cli.file_haps): the
 * chunk's haplotype for a binned chunk; for a GVS_HAP_ANY chunk the haplotype its votes assign (the records of the
 * batch's diag filter in haplotype mode), and for a tie or a read without a vote the parity of its run-wide read index
 * (even: haplotype 0), as gvs_batch_stash numbers the batch's reads.
 * Per group index g (the group table of gvs_db_export / gvs_groups_get), with H = contig_hap[grp_contig[g]]:
 *   own[g]    the distinct reads r with a match row of group g and hap(r) == H;
 *   other[g]  the same with hap(r) == 1 - H;
 * over the match rows of gvs_match / gvs_rows_set(0): every contig of both haplotypes, before the diag filter, no
 * read-length minimum, no bad-group filter (the rows gvs_sunk_depth counts).  A group on a contig of neither haplotype
 * counts nothing; for the others own + other equals reads of gvs_sunk_depth.
 *   sunks[g]  the .loc rows of group g;  end[g]  its last SUNK's start + k (group start + k without .loc rows).
 * gvs_allele_support adds the current match rows (none after gvs_batches_bind or before any gvs_match) to an
 * int32[2][n_groups] array -- own at [g], other at [n_groups + g] -- whose device pointer *support_dev receives.  Inside
 * a batches run it accumulates from gvs_batches_begin on (accumulate != 0); accumulate = 0 replaces.  Call it between a
 * batch's diag filter and its gvs_batch_stash (the parity uses the index the stash will give).  GVS_E_STATE before a
 * group table or contig haplotypes, and on match rows of a batch with GVS_HAP_ANY chunks whose diag filter has not run.
 * Several GPUs sum the 2*n_groups entries (as the histogram of gvs_group_hist; a read lives on one GPU, so the sums are
 * exact) before gvs_allele_support_get / gvs_allele_runs.
 * gvs_allele_support_get: host buffers of n_groups entries, any pointer may be NULL.
 * gvs_allele_runs: per base x, the (own, other) of x's segment [ID_r, ID_r+1) as runs (contig, start, end, own, other)
 * that tile [0, contig_len[c]) of every contig in (contig, start) order, maximal, with a zero head run before a contig's
 * first group.  GVS_E_STATE before gvs_allele_support or after the group table changed.
 * The calls (phase flips, switched blocks, consensus errors) are the caller's: DESIGN.md section 5.5h. */
int gvs_allele_support(gvs_ctx* ctx, int accumulate, int32_t** support_dev);
int gvs_allele_support_get(gvs_ctx* ctx, int32_t* own, int32_t* other, uint32_t* sunks, uint32_t* end);
int gvs_allele_runs(gvs_ctx* ctx, const uint32_t* contig_len, uint64_t* n_runs);
int gvs_allele_runs_get(gvs_ctx* ctx, uint32_t* contig, uint32_t* start, uint32_t* end, uint32_t* own, uint32_t* other);

/* covprob.py:56-100: table[0..3499] of gap-spanning probabilities from the read-length
 * histogram.  kbp[n_bins], cnt[n_bins] = distinct int(len/1000) values and their multiplicities
 * in the reference's iteration order, pn = run-of-k survival probability (covprob.py:79-81, host
 * root solve), genome_kbp = sum(fai.len)/1000. */
int gvs_covprob_table(gvs_ctx* ctx, const int64_t* kbp, const int64_t* cnt, uint32_t n_bins,
                      double genome_kbp, double pn, double* table3500);

/* covprob.py:35-40,109-131: per gap the largest inter-group distance `dist` among the SUNK groups with
 * chrom == contig and start-2 < ID < end+2, and covprob = table[int(max_gap/1000)].  grp_contig/grp_id =
 * the first row of every (contig, group) of kmer.loc in file order, which must be (contig, start)
 * order as defineSUNKs.smk:101-126 writes it (dist is the file-order diff, across contig boundaries,
 * clamped at 0, first row = its own ID).  Errors mirror the reference: GVS_E_KEYERROR when a gap has
 * no group in range or max_gap >= 3500 kbp.  All pointers are host memory. */
int gvs_covprob_gaps(gvs_ctx* ctx, const uint32_t* grp_contig, const uint32_t* grp_id, uint64_t n_groups,
                     const uint32_t* gap_contig, const int64_t* gap_start, const int64_t* gap_end,
                     uint64_t n_gaps, const double* table3500, int64_t* max_gap, double* covprob);
/* slop_gaps (workflow/rules/tagONT.smk:249, `bedtools slop -b 200000`): start/end are widened by b in
 * place and clipped to [0, contig_len[contig]]. */
int gvs_slop(gvs_ctx* ctx, const uint32_t* contig, int64_t* start, int64_t* end, uint64_t n,
             const uint32_t* contig_len, uint32_t n_contigs, int64_t b);

/* ------------------------------------------------------------------------------------------ */
/* synthetic workloads (bench.py / tests only; SURVEY.md 8d)                                   */
/* ------------------------------------------------------------------------------------------ */
/* Deterministic diploid assembly on the device: hap1 = i.i.d. ACGT with segmental duplications
 * and N runs, hap2 = hap1 with SNPs at rate snp_rate.  contig_len[n_contigs_per_hap].  Writes
 * 2*sum(len) bytes to seq_dev (hap1 contigs then hap2 contigs). */
int gvs_synth_assembly(gvs_ctx* ctx, uint8_t* seq_dev, const uint64_t* contig_len,
                       uint32_t n_contigs_per_hap, double snp_rate, double dup_frac,
                       uint64_t seed);
/* ONT-like reads sampled from an assembly on the device (log-normal lengths, both strands,
 * substitution/deletion/insertion errors, occasional N runs).  Two-step: _plan computes the
 * read offsets (device array of n_reads+1, returned total in *total_bases), _fill writes bases. */
int gvs_synth_reads_plan(gvs_ctx* ctx, const uint64_t* contig_off_dev, uint32_t contig_lo,
                         uint32_t contig_hi, uint64_t n_reads, double len_mu, double len_sigma,
                         uint32_t len_min, uint32_t len_max, uint64_t seed, uint64_t* read_off_dev,
                         uint64_t* total_bases);
int gvs_synth_reads_fill(gvs_ctx* ctx, const uint8_t* asm_seq_dev, uint8_t* reads_dev,
                         const uint64_t* read_off_dev, uint64_t n_reads);

#ifdef __cplusplus
}
#endif
#endif /* GAVISUNK_B200_H */
