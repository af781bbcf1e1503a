/*
 * nohuman_gpu.h — C ABI of libnohuman_gpu.so, the B200 (sm_100a) replacement
 * for the one hot path of mbhall88/nohuman: the kraken2 classification that
 * the reference runs as a child process.
 *
 * What each entry point replaces in the reference (/root/reference):
 *   - the whole group stands where `CommandRunner::run` spawns kraken2:
 *       src/lib.rs:22-23    Command::new("kraken2").args(args).output()
 *       src/main.rs:270     kraken.run(&kraken_cmd)
 *   - nh_db_open            <- `--db <dir>` (src/main.rs:212-219) after
 *                              validate_db_directory (src/lib.rs:119-141): the
 *                              three files hash.k2d / opts.k2d / taxo.k2d are
 *                              read unchanged
 *   - nh_params_t           <- `--confidence` (src/main.rs:213,222-223; parsed
 *                              by parse_confidence_score, src/lib.rs:145-151),
 *                              `--paired` (src/main.rs:230-235),
 *                              `--classified-out|--unclassified-out`
 *                              (src/main.rs:259-265), `--threads`
 *                              (src/main.rs:212,216-217); minimum_hit_groups is
 *                              the kraken2 wrapper default (2) that nohuman
 *                              never overrides
 *   - nh_run_stats_t        <- the three stderr counts parsed by
 *                              parse_kraken_stderr (src/lib.rs:61-97)
 *   - nh_classify_batch*    <- kraken2's per-read work (upstream classify.cc
 *                              ClassifySequence/ResolveTree; SURVEY.md A.3-A.5)
 *
 * Conventions: C linkage, plain pointers and sizes, no C++/torch types, no
 * exceptions across the boundary.  Every function returns 0 on success or a
 * negative nh_status; nh_last_error() gives the message for the calling
 * thread.  nh_db is immutable after open and may be shared; one nh_session
 * per calling thread.  There is no CPU fallback: without a CUDA device every
 * compute entry point fails with NH_ERR_CUDA.
 */
#ifndef NOHUMAN_GPU_H
#define NOHUMAN_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NH_ABI_VERSION 3

typedef enum {
  NH_OK = 0,
  NH_ERR_INVALID = -1,     /* bad argument */
  NH_ERR_IO = -2,          /* cannot read / malformed k2d file */
  NH_ERR_CUDA = -3,        /* CUDA runtime error or no device */
  NH_ERR_UNSUPPORTED = -4, /* database parameters outside the kernels' range */
  NH_ERR_CAPACITY = -5,    /* batch larger than the session was created for */
  NH_ERR_NOMEM = -6
} nh_status;

typedef struct nh_db nh_db;
typedef struct nh_session nh_session;

/* Parameters read from opts.k2d / hash.k2d / taxo.k2d (SURVEY.md Appendix B). */
typedef struct {
  uint64_t k, l, spaced_seed_mask, toggle_mask, minimum_acceptable_hash_value;
  int32_t dna_db, revcom_version;
  uint64_t capacity, size, key_bits, value_bits;
  uint64_t node_count;
  int32_t device;
  int32_t replicated_by; /* 0: read from disk / memory, 1: NCCL broadcast, 2: peer-copy tree (nh_db_open_multi) */
  uint64_t filter_bytes; /* size of the miss filter built next to the table on the device (capacity / 32 records of 32
                          * bytes; 0: none — NH_FILTER=0, or no memory for it) */
} nh_db_info_t;

typedef struct {
  double confidence;          /* --confidence as kraken2 parses it (a double) */
  int32_t minimum_hit_groups; /* kraken2 default 2; <0 selects the default */
  int32_t paired;             /* sequences 2i, 2i+1 are the mates of unit i */
  int32_t keep_human;         /* 0: keep unclassified (default nohuman), 1: keep classified (-H) */
  int32_t threads;            /* host threads for the file API; <=0: 1 */
  uint64_t max_batch_bases;   /* session capacity; 0 selects 256 MiB */
  uint64_t max_batch_seqs;    /* session capacity; 0 selects max_batch_bases/64 */
  int32_t emit_runs;          /* 1: keep per-sequence (taxid, k-mer count) runs for nh_last_batch_runs
                                 (kraken2's per-read output, --output; costs 5 B per lookup of D2H) */
  int32_t gpu_gzip;           /* 1: gzip output ('g') of nh_run_files / nh_run_files_multi is deflated on the
                                 sessions' GPUs (nh_bgzf_compress's members); 0: zlib level 6 on -t host threads.
                                 Other formats ignore it. */
} nh_params_t;

typedef struct {
  uint64_t n_units;        /* reads (single) or pairs (paired) */
  uint64_t n_classified;   /* kraken2 "sequences classified" */
  uint64_t n_unclassified; /* kraken2 "sequences unclassified" */
  uint64_t n_kept;
  uint64_t n_bases;
  uint64_t n_tiles;        /* minimizer-kernel work items */
  uint64_t n_lookups;      /* hash-table probes issued */
  /* device time per stage (CUDA events).  With fused_kernel = 1 the scan, the
   * probe and the scoring of short units are ONE kernel timed as ms_minimizer
   * (ms_probe = 0) and ms_score covers only the units left to k_score. */
  float ms_plan, ms_minimizer, ms_probe, ms_score;
  float ms_h2d, ms_d2h;
  uint32_t gpu_launches;   /* kernels launched for this batch */
  uint32_t fused_kernel;   /* 0: warp-per-tile kernels, 2: k_stream_classify */
  uint64_t n_sector_reads; /* k_stream_classify: 32-byte table sectors requested (lookups + chain continuations) */
} nh_batch_stats_t;

typedef struct {
  uint64_t total;        /* "N sequences ... processed" */
  uint64_t classified;   /* "N sequences classified" */
  uint64_t unclassified; /* "N sequences unclassified" */
  uint64_t bases;
  double seconds;
  /* where the host threads spent their time: busy seconds per stage, summed over the stage's
   * threads (waiting for another stage is not counted); seconds above is the wall clock */
  double busy_inflate_s;   /* decompressing the inputs (1 thread per plain-gzip / bzip2 file, a pool for blocked gzip) */
  double busy_parse_s;     /* FASTQ / FASTA parsing (1 thread per input file) */
  double busy_stage_s;     /* interleaving mates into the pinned transfer buffers (2 threads per GPU) */
  double busy_classify_s;  /* inside nh_classify_batch: H2D, kernels, D2H (same threads) */
  double busy_serialise_s; /* re-serialising kept records, per-read output lines (same threads) */
  double busy_compress_s;  /* output compression (-t threads; with gpu_gzip, the GPU deflater threads) */
  double busy_write_s;     /* ordered writes to the output files (1 thread) */
  int32_t threads_inflate, threads_compress; /* threads_compress: -t, or one GPU deflater thread per GPU */
} nh_run_stats_t;

/* ------------------------------------------------------------------ */
int nh_abi_version(void);
const char *nh_last_error(void);
/* Number of CUDA devices visible (0 if none / no driver). */
int nh_device_count(void);

/* Open <db_dir>/{hash,opts,taxo}.k2d (or <db_dir>/db/..., as
 * validate_db_directory does, src/lib.rs:119-141) and make the table
 * resident in HBM of `device`. */
int nh_db_open(const char *db_dir, int device, nh_db **out);
/* Same, from memory images of the three files.  `cells` points at the
 * capacity x uint32 cell array (hash.k2d after its 32-byte header); if
 * cells_on_device != 0 it is a device pointer on `device` that the library
 * adopts WITHOUT copying or freeing (used when one rank loads the table and
 * NCCL-broadcasts it to the others); it must be 128-byte aligned and readable,
 * with zero cells, up to the next multiple of 32 cells past `capacity`
 * (nh_db_device_cells of another nh_db satisfies this). */
int nh_db_open_memory(const void *opts, size_t opts_len, const void *taxo, size_t taxo_len,
                      const uint64_t hash_header[4], const uint32_t *cells, int cells_on_device,
                      int device, nh_db **out);
/* The boundary SURVEY.md §8(b) promised: ONE read of <db_dir> from disk, then the table is
 * replicated onto every listed device — by an NCCL broadcast over NVLink / NVSwitch (libnccl.so.2
 * bound at run time), or by a binomial tree of peer copies when NCCL is not available
 * (NH_DB_REPLICATE=p2p forces the tree).  out[n_devices] receives one independent nh_db per
 * device, out[0] on device_ids[0]; nh_db_info().replicated_by says how each one arrived.
 * This is what replaces kraken2 loading the database once per process (reference src/main.rs:270). */
int nh_db_open_multi(const char *db_dir, const int *device_ids, int n_devices, nh_db **out);
/* Replicate an open database onto another device of this process (peer copy,
 * NVLink when the devices are connected); the clone is independent of `src`. */
int nh_db_clone(const nh_db *src, int device, nh_db **out);
int nh_db_info(const nh_db *db, nh_db_info_t *out);
/* Device pointer of the resident cell array (for NCCL broadcast by the host). */
const uint32_t *nh_db_device_cells(const nh_db *db);
void nh_db_close(nh_db *db);

int nh_session_create(nh_db *db, const nh_params_t *params, nh_session **out);
void nh_session_destroy(nh_session *s);

/* Classify one batch held in HOST memory.  bases: concatenated ASCII
 * sequences; offsets[n_seqs+1] byte offsets.  Outputs are per unit and may be
 * NULL: out_call = external taxid of the call (0 = unclassified, i.e.
 * non-human for nohuman), out_keep = 1 if the unit is written to the output
 * under params.keep_human.  H2D and D2H copies happen inside the call. */
int nh_classify_batch(nh_session *s, const uint8_t *bases, const uint64_t *offsets,
                      uint64_t n_seqs, uint32_t *out_call, uint8_t *out_keep,
                      nh_batch_stats_t *stats);

/* ---- packed transfer format: 0.4 bytes per base over PCIe instead of 1 ----
 * Every sequence starts on a UNIT of 32 bases.  codes: 8 bytes per unit, 2 bits per base (A 0, C 1,
 * G 2, T 3, either case), 4 bases per byte, first base in the top bits; valid: one 32-bit word per
 * unit, bit j = base j of the unit is an unambiguous base of the sequence (LSB first; padding and
 * every other byte value: 0); poff[n_seqs+1]: first unit of each sequence.
 * nh_packed_units gives the number of units a batch needs; nh_pack_reads fills the three arrays
 * (codes: units*8 bytes, valid: units words, poff: n_seqs+1) from ASCII with `threads` host
 * threads (AVX2 when the CPU has it).  nh_classify_batch_packed is nh_classify_batch for such input
 * (sessions without emit_runs, databases the streaming kernel covers); offsets still gives the
 * sequence lengths.  Same per-unit results as the ASCII entry point. */
int nh_packed_units(const uint64_t *offsets, uint64_t n_seqs, uint64_t *out_units);
int nh_pack_reads(const uint8_t *bases, const uint64_t *offsets, uint64_t n_seqs, uint8_t *codes, uint32_t *valid,
                  uint32_t *poff, int threads);
int nh_classify_batch_packed(nh_session *s, const uint8_t *codes, const uint32_t *valid, const uint32_t *poff,
                             const uint64_t *offsets, uint64_t n_seqs, uint32_t *out_call, uint8_t *out_keep,
                             nh_batch_stats_t *stats);
/* nh_classify_batch (same arguments, same results: ASCII bases in host memory) with the transfer done in the
 * packed format: nh_pack_reads + nh_classify_batch_packed in one call.  A pool of `pack_threads` threads owned by
 * the session packs into the session's pinned planes; the calling thread sleeps (it does not spin) until the
 * results are back, so that several sessions on several host threads keep every core packing while the other
 * sessions' copies and kernels run — how bench.py's `e2e` gets 76-84 Gbp/s out of a PCIe link that moves 52 GB/s. */
int nh_classify_batch_pack(nh_session *s, const uint8_t *bases, const uint64_t *offsets, uint64_t n_seqs,
                           int pack_threads, uint32_t *out_call, uint8_t *out_keep, nh_batch_stats_t *stats);

/* Same with DEVICE-resident input and output (all pointers are device
 * pointers on the session's device; d_bases must be 16-byte aligned, as any
 * cudaMalloc pointer is).  Asynchronous on the session stream;
 * call nh_session_sync before reading outputs or stats. */
int nh_classify_batch_device(nh_session *s, const uint8_t *d_bases, const uint64_t *d_offsets,
                             uint64_t n_seqs, uint64_t total_bases, uint32_t *d_out_call,
                             uint8_t *d_out_keep);
int nh_session_sync(nh_session *s, nh_batch_stats_t *stats);
/* Per-sequence hit runs of the batch just classified (session created with
 * emit_runs = 1): sequence i owns runs [seq_first_run[i], seq_first_run[i+1]),
 * each an external taxid (0 = minimizer not in the table) and the number of
 * consecutive unambiguous k-mer positions that carry it — kraken2's `taxa`
 * vector (classify.cc) without its ambiguous entries, which the host derives
 * from the sequence itself.  Host pointers; *n_runs gets the total. */
int nh_last_batch_runs(nh_session *s, uint64_t n_seqs, uint32_t *seq_first_run, uint32_t *run_taxon_ext,
                       uint16_t *run_len, uint64_t run_capacity, uint64_t *n_runs);
/* The CUDA stream (cudaStream_t) the session launches on. */
void *nh_session_stream(nh_session *s);

/* ---- file API: the exact stand-in for `kraken.run(&kraken_cmd)` ----
 * (src/main.rs:270).  One call does what the child process did for the argv
 * nohuman assembles at src/main.rs:210-267: read 1-2 FASTQ/FASTA inputs
 * (plain, gzip or bzip2, auto-detected like kraken2 does), classify every
 * read / pair against the session's database, and write the kept records
 * (--unclassified-out, or --classified-out when params.keep_human) in input
 * order.  Unlike kraken2 it writes the FINAL, already compressed outputs, so
 * the temp-file round trip of src/main.rs:248-257,340-368 disappears.
 * `stats` carries the three counts parse_kraken_stderr (src/lib.rs:61-97)
 * extracts from kraken2's stderr; paired counts are pairs. */
typedef struct {
  const char *in1;            /* first (or only) input file */
  const char *in2;            /* second mate file, or NULL for single-end */
  const char *out1;           /* where kept records of in1 go */
  const char *out2;           /* ... of in2 (paired only) */
  int32_t out_format;         /* nohuman -F letter: 'u' none, 'g' gzip (written as BGZF members), 'b' bzip2,
                                 'x' xz, 'z' zstd; 0 = 'u' */
  int32_t tag_classified;     /* 1: append " kraken:taxid|<id>" to classified-out headers as kraken2 does */
  const char *kraken_output;  /* --output: per-read lines; NULL or "/dev/null": not produced */
  const char *kraken_report;  /* --report; NULL: not produced */
} nh_files_t;
int nh_run_files(nh_session *s, const nh_files_t *files, nh_run_stats_t *stats);
/* Same over several sessions, one per GPU with the database replicated
 * (nh_db_clone): read batches are dealt to the GPUs as they free up, nothing is
 * exchanged between them, and the writer restores input order.  Parameters
 * are taken from sessions[0]. */
int nh_run_files_multi(nh_session *const *sessions, int n_sessions, const nh_files_t *files,
                       nh_run_stats_t *stats);
/* Host-logic test hook (no GPU): the same reader -> ordered writer -> block
 * compressor pipeline with the per-unit decisions (keep[], external call[])
 * supplied by the caller. */
int nh_debug_rewrite_files(const nh_files_t *files, const uint8_t *keep, const uint32_t *call_ext,
                           uint64_t n_units, int threads, nh_run_stats_t *stats);

/* BGZF compression on the GPU: in[0..n) becomes gzip members of 0xff00 input bytes each (byte i goes into
 * member i / 0xff00), as the gzip output of nh_run_files is cut, without bgzip's empty end-of-file member.
 * Every member carries the 'BC' subfield with its size and holds one deflate block (dynamic Huffman codes,
 * or stored when that is not smaller), so no member exceeds 65 311 bytes.  The same input gives the same
 * bytes on every call and every GPU.  out_cap must be at least ceil(n / 0xff00) * 65536
 * (NH_ERR_CAPACITY otherwise); *out_len gets the bytes written. */
int nh_bgzf_compress(int device, const uint8_t *in, size_t n, uint8_t *out, size_t out_cap, size_t *out_len);
/* Device time of nh_bgzf_compress's kernels for one batch of n bytes (1 byte to 1 GiB) already on the device:
 * mean over `iters` launches after one warm-up, in seconds. */
int nh_bench_bgzf(int device, const uint8_t *in, size_t n, int iters, double *out_seconds);

/* gzip decompression on the GPU: in[0..n) is a whole gzip file (one member or many, any deflate block types)
 * and out gets what `gzip -dc` writes: bytes after the last member that do not start with 0x1f are ignored,
 * as zlib's gzread ignores them.  NH_ERR_IO for a stream that is not gzip, corrupt or truncated (including a
 * wrong CRC-32 or ISIZE and a distance too far back); NH_ERR_CAPACITY when out_cap is too small, with
 * *out_len set to the size needed. */
int nh_gunzip(int device, const uint8_t *in, size_t n, uint8_t *out, size_t out_cap, size_t *out_len);
/* nh_gunzip with an explicit chunk and window size in compressed bytes (0: the defaults) and test flags;
 * counts[NH_GUNZIP_NCOUNTS] (may be NULL) receives what ran, indexed by NH_GUNZIP_COUNT_*. */
#define NH_GUNZIP_SHIFT_CANDIDATES 1 /* every other chunk's candidate start moved by one bit: forces repairs */
#define NH_GUNZIP_COUNT_WINDOWS 0
#define NH_GUNZIP_COUNT_CHUNKS 1
#define NH_GUNZIP_COUNT_REPAIRED 2   /* chunks decoded again from their predecessor's stop */
#define NH_GUNZIP_COUNT_OVERFLOWED 3 /* chunks whose output outgrew their slot */
#define NH_GUNZIP_COUNT_MEMBERS 4
#define NH_GUNZIP_COUNT_CARRIED 5    /* compressed bytes carried from one window into the next */
/* device time, in nanoseconds (CUDA events), of each phase: finding block starts, the first decode of every
 * chunk, repairs and spills, carrying the 32 KiB history through the chunks, resolving markers + CRC32 */
#define NH_GUNZIP_COUNT_NS_FIND 6
#define NH_GUNZIP_COUNT_NS_DECODE 7
#define NH_GUNZIP_COUNT_NS_REDECODE 8
#define NH_GUNZIP_COUNT_NS_WINDOW 9
#define NH_GUNZIP_COUNT_NS_RESOLVE 10
#define NH_GUNZIP_NCOUNTS 11
int nh_debug_gunzip(int device, const uint8_t *in, size_t n, uint8_t *out, size_t out_cap, size_t *out_len,
                    size_t chunk_bytes, size_t window_bytes, int flags, uint64_t *counts);
/* Device time of nh_gunzip's kernels for in[0..n) (no copies of the input or the output): mean over `iters`
 * runs after one warm-up, in seconds. */
int nh_bench_gunzip(int device, const uint8_t *in, size_t n, int iters, double *out_seconds);

/* ---- database build: kraken2-build --build on the GPU ----
 * nh_build_taxonomy converts an NCBI taxonomy dump to taxo.k2d (host only, no GPU).  Every taxid that
 * seqid2taxid assigns is marked with all its ancestors; the marked nodes are numbered breadth-first from
 * taxid 1 (internal id 1, so every parent id is below its children's), with the children of a node taken in
 * ascending external taxid (a choice made so that the image is deterministic); node 0 is the zeroed
 * "unclassified" node.  Names are the `scientific name` rows of names.dmp, ranks column 3 of nodes.dmp.
 * NH_ERR_IO with the file and line in nh_last_error() for a map taxid missing from nodes.dmp, a parent
 * cycle, a node that does not reach taxid 1, or a malformed line.  *node_count (may be NULL) includes node 0. */
int nh_build_taxonomy(const char *nodes_dmp, const char *names_dmp, const char *seqid2taxid, const char *out_taxo_k2d,
                      uint64_t *node_count);

typedef struct {
  const char *const *fasta; /* library files: FASTA, plain / gzip / bzip2 */
  int32_t n_fasta;
  const char *nodes_dmp, *names_dmp, *seqid2taxid;
  const char *out_dir;      /* receives hash.k2d, opts.k2d, taxo.k2d (created if missing) */
  uint32_t k, l, spaces;    /* 0: kraken2-build's defaults 35 / 31 / 7 */
  uint64_t capacity;        /* table cells; 0: estimated from the library (an extra pass over it) */
  double load_factor;       /* of the estimated capacity; 0: 0.7 */
  uint64_t batch_bases;     /* bases per device batch; 0: 256 MiB.  Longer sequences are cut into pieces */
  int32_t threads;          /* host threads for reading blocked gzip (BGZF) input; <= 0: 1 */
  int32_t device;
} nh_build_params_t;

typedef struct {
  uint64_t sequences;  /* library records inserted */
  uint64_t skipped;    /* records whose ID has no seqid2taxid entry (kraken2 warns and skips them too) */
  uint64_t bases;      /* bases of the inserted records */
  uint64_t minimizers; /* minimizer insertions (runs of equal consecutive non-ambiguous minimizers count once) */
  uint64_t estimate;   /* distinct minimizers estimated by the capacity pass (0 when capacity was given) */
  uint64_t estimate_slots;   /* size of the capacity pass's device set of sampled hashes when it ended */
  uint64_t estimate_rescans; /* batches the capacity pass scanned again after they overfilled the set */
  uint64_t capacity, size, node_count; /* of the written table / taxonomy */
  double s_taxonomy, s_estimate, s_insert, s_write; /* wall seconds per phase */
} nh_build_stats_t;

/* Builds a kraken2 database from FASTA files and an NCBI taxonomy, as `kraken2-build --build` does for a
 * nucleotide library.  A record's ID is the first word of its header, looked up in seqid2taxid; records
 * without an entry are skipped and counted.  Bases other than ACGT / acgt are ambiguous (N, and dustmasker's
 * x).  Every non-ambiguous minimizer is inserted with CompactHashTable::CompareAndSet and the LCA merge on
 * the GPU.  Every lookup on the result returns what a sequential build returns for the same library, except
 * where two distinct minimizers share a compacted key on one probe path (kraken2 merges those by design, and
 * which one survives depends on insertion order): the cell layout is NOT byte-reproducible between runs, as
 * with any concurrent CompareAndSet build.  The files are written as *.tmp and renamed only once all three
 * are complete; if a rename fails, the ones already renamed are removed, so a failed build leaves none of its
 * .k2d files behind (a file of an earlier build in out_dir that a completed rename replaced is gone too).
 * NH_ERR_CAPACITY ("table full") once the load passes 0.95: the inserts stop soon after, the overshoot being at
 * most the claims of the tiles already running (up to 256 cells per running warp).  stats may be NULL. */
int nh_build_db(const nh_build_params_t *p, nh_build_stats_t *stats);

/* ---- low-complexity masking: dustmasker's symmetric DUST on the GPU ----
 * The mask (DESIGN.md §4f): over every run of A/C/G/T in either case (every other byte ends a run), the union
 * of the bases of every "perfect" triplet interval that fits in `window` bases, at score threshold `level`.
 * window 4..64 and level 1..255 (dustmasker's defaults: 64, 20); anything else is NH_ERR_INVALID.
 * nh_dust_mask: records concatenated in host memory, offsets[n_seqs+1] (offsets[0] = 0); out[i] is seq[i]
 * lower-cased where masked and upper-cased everywhere else, which is dustmasker's FASTA form. */
int nh_dust_mask(int device, const uint8_t *seq, const uint64_t *offsets, uint64_t n_seqs, int window, int level,
                 uint8_t *out);

#define NH_DUST_FASTA 0    /* dustmasker -outfmt fasta: headers as read, masked bases lower-case, 60 a line */
#define NH_DUST_INTERVAL 1 /* dustmasker -outfmt interval: each header, then "start - end" lines, 0-based inclusive */
typedef struct {
  const char *in_path;  /* FASTA (or FASTQ): plain, gzip, BGZF or bzip2 */
  const char *out_path; /* NULL or "-": stdout */
  int32_t format;       /* NH_DUST_FASTA or NH_DUST_INTERVAL */
  int32_t window;       /* 0: 64 */
  int32_t level;        /* 0: 20 */
  int32_t threads;      /* host threads for reading blocked gzip (BGZF) input; <= 0: 1 */
  int32_t device;
  uint64_t batch_bases; /* bases per device batch, 8192..2^31; 0: 256 MiB.  Longer records are cut into pieces */
} nh_dust_params_t;

typedef struct {
  uint64_t sequences, bases, masked; /* records, their bases, masked bases */
  uint64_t intervals;                /* maximal runs of masked bases */
  double seconds;                    /* wall clock */
} nh_dust_stats_t;

/* File to file: every record of in_path masked and written as dustmasker writes it.  Headers are copied byte
 * for byte.  An unreadable, corrupt or truncated input is NH_ERR_IO, and a failed run removes out_path.
 * stats may be NULL. */
int nh_dust_fasta(const nh_dust_params_t *p, nh_dust_stats_t *stats);
/* Device time of nh_dust_mask's kernels at window 64, level 20 for records already on the device: mean over
 * `iters` runs after one warm-up, in seconds. */
int nh_bench_dust(int device, const uint8_t *seq, const uint64_t *offsets, uint64_t n_seqs, int iters,
                  double *out_seconds);

/* Pinned host memory for callers that want true async copies. */
void *nh_host_alloc(size_t bytes);
void nh_host_free(void *p);

/* ---- per-stage entry points (parity tests call these through the ABI) ---- */
/* Every k-mer position of every sequence: out_min[pos_offsets[i]+p] and
 * out_ambig[...] as MinimizerScanner::NextMinimizer/is_ambiguous return them.
 * pos_offsets[n_seqs+1] = exclusive scan of max(0, len-k+1). Host pointers. */
int nh_debug_minimizers(nh_session *s, const uint8_t *bases, const uint64_t *offsets,
                        uint64_t n_seqs, const uint64_t *pos_offsets, uint64_t *out_min,
                        uint8_t *out_ambig);
/* CompactHashTable::Get for n host keys -> internal taxids. */
int nh_debug_probe(nh_session *s, const uint64_t *keys, uint64_t n, uint32_t *out_taxon);
/* After nh_classify_batch: per-unit internal call, total_kmers, hit_groups. */
int nh_debug_last_batch(nh_session *s, uint32_t *out_call_internal, uint32_t *out_total_kmers,
                        uint32_t *out_hit_groups, uint64_t n_units);

/* ---- roofline helper ---- */
/* Uniformly random aligned 32-byte sector reads over the resident table:
 * n_reads sectors per launch, `iters` launches; returns the best launch in
 * GB/s of sectors (the random-access HBM roofline the probe is held to). */
int nh_bench_random_gather(nh_db *db, uint64_t n_reads, int iters, double *out_gbs);
/* The probe's own access pattern over the resident table, nothing else: every chain reads a random
 * sector and, with probability p_continue, the adjacent one once the first has arrived; `lanes`
 * (1, 2, 4) lanes share an item and read an aligned block of that many sectors in one instruction
 * (lanes = 0: one sector per lane fetched the way k_stream_classify does it, by lane pairs with
 * cp.async into shared memory; depth 1 or 2 rounds in flight per warp, no SM windows);
 * every thread keeps `depth` (1, 2, 4) chains going and every SM runs `blocks_per_sm` (1..8) blocks
 * of 256 threads, so callers can look for the best number of requests in flight;
 * sm_window_bytes > 0 confines each SM to its own window.  Returns the best of `iters` launches as
 * items (lookups) per second and table requests per second. */
int nh_bench_probe_pattern(nh_db *db, int lanes, int depth, int blocks_per_sm, double p_continue,
                           uint64_t sm_window_bytes, uint32_t items_per_chain, int iters,
                           double *out_items_per_s, double *out_requests_per_s);

#ifdef __cplusplus
}
#endif
#endif
