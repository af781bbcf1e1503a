/* nh_internal.h — host-side objects behind the opaque C-ABI handles. */
#ifndef NH_INTERNAL_H
#define NH_INTERNAL_H

#include <cuda_runtime.h>
#include <stdint.h>

#include <functional>
#include <string>
#include <vector>

#include "../../include/nohuman_gpu.h"
#include "nh_kernels.cuh"

enum {
  EV_H2D0 = 0,
  EV_PLAN0,
  EV_MIN0,
  EV_PROBE0,
  EV_SCORE0,
  EV_SCORE1,
  EV_D2H1,
  NH_NUM_EVENTS
};

struct NhPackPool;
void nh_pack_pool_destroy(NhPackPool *p); /* defined next to the pool (nh_capi.cu) */

struct nh_db {
  nh_db_info_t info{};
  NhDbParams params{};
  uint32_t *d_cells = nullptr;
  bool owns_cells = false;
  uint32_t *d_parent = nullptr;
  uint32_t *d_ext = nullptr;
  uint32_t *d_filter = nullptr; /* miss filter: one 32-byte record per block of 32 cells (k_filter_build) */
  uint32_t n_filter_blocks = 0; /* 0 until the filter is built */
  uint32_t *d_huge = nullptr; /* global-memory taxon table for units with more distinct taxa than shared memory holds */
  std::vector<uint32_t> h_parent, h_ext;
  std::vector<std::string> h_name, h_rank; /* taxo.k2d name / rank strings per node (reports) */
  int sm_count = 0;
};

struct nh_session {
  nh_db *db = nullptr;
  NhDbParams P{}; /* db->params with this session's tile size */
  nh_params_t params{};
  uint64_t cap_bases = 0, cap_seqs = 0, cap_tiles = 0, cap_lookups = 0;
  size_t device_bytes = 0;
  uint8_t *d_bases = nullptr;
  uint64_t *d_offsets = nullptr;
  uint32_t *d_tile_base = nullptr;
  uint2 *d_seq_info = nullptr;
  uint64_t *d_block_sums = nullptr;
  NhTile *d_tiles = nullptr;
  NhTileOut *d_tile_out = nullptr;
  uint64_t *d_lk_min = nullptr;
  uint16_t *d_lk_cnt = nullptr;
  uint32_t *d_lk_taxon = nullptr;
  uint32_t *d_out_call = nullptr;
  uint8_t *d_out_keep = nullptr;
  uint32_t *d_dbg_call = nullptr, *d_dbg_total = nullptr, *d_dbg_groups = nullptr;
  uint32_t *d_overflow = nullptr;
  uint32_t *d_deferred = nullptr;
  uint32_t *d_run_ext = nullptr, *d_tile_run_off = nullptr, *d_run_cursor = nullptr;
  uint16_t *d_run_len = nullptr;
  uint8_t *d_codes = nullptr;  /* packed input planes (nh_classify_batch_packed), allocated on first use */
  uint32_t *d_valid = nullptr, *d_poff = nullptr;
  bool packed_next = false;    /* the batch being enqueued came packed */
  /* nh_classify_batch_pack: the packer threads and the pinned planes they fill */
  NhPackPool *pack_pool = nullptr;
  int pack_threads = 0;
  uint8_t *h_codes = nullptr;
  uint32_t *h_valid = nullptr, *h_poff = nullptr, *h_len32 = nullptr;
  uint32_t *d_len32 = nullptr; /* sequence lengths as sent; k_len_* rebuild d_offsets and d_poff from them */
  uint64_t *d_len_sums = nullptr;
  cudaEvent_t ev_block = nullptr; /* blocking-sync event: the calling thread sleeps instead of spinning */
  uint64_t last_seqs = 0;
  bool use_fused = false, last_fused = false;
  int lane_taxa = NH_LANE_TAXA;
  int filter_mode = 3;
  int last_form = 0;       /* 0: warp-per-tile kernels, 2: k_stream_classify */
  int forced_tile_pos = 0; /* NH_FUSED_TILE_POS */
  NhTileTab *d_tile_tab = nullptr;
  NhTileSum *d_tile_sum = nullptr;
  NhCounters *d_counters = nullptr;
  NhCounters *h_counters = nullptr; /* pinned */
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[NH_NUM_EVENTS] = {};
  bool pending = false;
  bool timed_copies = false;
  uint32_t last_launches = 0;
  uint64_t last_units = 0, last_bases = 0;
};

/* nh_pack.cc: sequences [s0, s1) of a batch into the planes (poff already holds their first units); AVX2 with
 * non-temporal stores when the CPU has it */
void nh_pack_range(const uint8_t *bases, const uint64_t *offsets, uint64_t total_bases, uint64_t s0, uint64_t s1, uint8_t *codes,
                   uint32_t *valid, const uint32_t *poff);

/* BGZF framing, shared by the zlib path (nh_pipeline.cc) and the GPU deflater (nh_deflate.cu), which must
 * cut and frame members byte for byte alike.  Every member is a gzip member whose header carries one extra
 * subfield, 'BC', holding the member's total size - 1 (the two bytes after these 16); output ends in
 * bgzip's empty end-of-file member. */
#define NH_BGZF_HEADER_BYTES 0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0
constexpr uint32_t BGZF_INPUT = 0xff00; /* input bytes per member (the last member of a block may be shorter) */
constexpr unsigned char BGZF_HEADER[16] = {NH_BGZF_HEADER_BYTES};
constexpr unsigned char BGZF_EOF[28] = {NH_BGZF_HEADER_BYTES, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};

/* nh_deflate.cu: BGZF compression on one GPU with its own stream, device buffers and pinned staging for a
 * batch of up to batch_bytes of input.  compress() cuts every block into BGZF_INPUT-byte members as the zlib
 * path does and returns each block's members, one string per block, or hands them in order to a sink; larger
 * inputs go in several rounds.
 * Not thread-safe: one per thread. */
class GpuDeflater {
 public:
  typedef std::pair<const uint8_t *, size_t> Span;
  /* receives the members in order: (block index, bytes, length), one call per member */
  typedef std::function<void(size_t, const uint8_t *, size_t)> Sink;
  static constexpr size_t kBatchBytes = size_t(32) << 20;
  GpuDeflater() = default;
  GpuDeflater(const GpuDeflater &) = delete;
  GpuDeflater &operator=(const GpuDeflater &) = delete;
  ~GpuDeflater();
  int open(int device, size_t batch_bytes = kBatchBytes); /* NH_OK or an nh_status with nh_last_error() set */
  int compress(const std::vector<Span> &blocks, std::vector<std::string> &out);
  int compress(const std::vector<Span> &blocks, const Sink &sink);
  /* device time of the kernels for one batch of `n` bytes (already cut into members), mean of `iters` */
  int time_kernels(const uint8_t *in, size_t n, int iters, double *seconds);

 private:
  int launch(size_t n_members);
  int run(size_t bytes, size_t n_members);
  int device_ = -1;
  size_t batch_ = 0, max_members_ = 0;
  cudaStream_t stream_ = nullptr;
  uint8_t *d_in_ = nullptr, *d_slots_ = nullptr, *d_out_ = nullptr;
  uint8_t *h_in_ = nullptr, *h_out_ = nullptr;
  uint2 *d_members_ = nullptr, *h_members_ = nullptr;
  uint32_t *d_scratch_ = nullptr, *d_sizes_ = nullptr;
  uint64_t *d_offs_ = nullptr, *h_offs_ = nullptr;
};

/* nh_inflate.cu: gzip decompression on one GPU with its own stream, device buffers and pinned staging.
 * inflate() reads the compressed stream from `src` a window at a time and hands the inflated bytes, in
 * order, to `sink` — exactly the bytes zlib's gzread gives, or an error (NH_ERR_IO: truncated or corrupt).
 * Not thread-safe: one per thread. */
struct NhGzMember;
struct NhGzChunk;
struct NhGzEmit;
struct NhGzJob;
class GpuInflater {
 public:
  /* fills dst with up to `want` bytes; 0 at the end of the input, -1 on a read error */
  typedef std::function<long(uint8_t *dst, size_t want)> Source;
  /* receives the next run of inflated bytes; a nonzero return ends inflate() with that code */
  typedef std::function<int(const uint8_t *, size_t)> Sink;
  static constexpr size_t kChunkBytes = size_t(32) << 10;  /* compressed bytes per chunk */
  static constexpr size_t kWindowBytes = size_t(16) << 20; /* new compressed bytes per window */
  GpuInflater() = default;
  GpuInflater(const GpuInflater &) = delete;
  GpuInflater &operator=(const GpuInflater &) = delete;
  ~GpuInflater();
  /* NH_OK or an nh_status with nh_last_error() set; flags: NH_GUNZIP_SHIFT_CANDIDATES */
  int open(int device, size_t chunk_bytes = 0, size_t window_bytes = 0, int flags = 0);
  int inflate(const Source &src, const Sink &sink);
  /* device time of the kernels for inflating in[0..n) (no input or output copies), mean of `iters` after one
   * warm-up */
  int time_kernels(const uint8_t *in, size_t n, int iters, double *seconds);
  size_t device_bytes() const;
  uint64_t counts[NH_GUNZIP_NCOUNTS] = {}; /* of the last inflate(): see nh_debug_gunzip */

 private:
  void lap(int a, int b, int count);
  int device_ = -1, flags_ = 0;
  size_t chunk_ = 0, window_ = 0, cap_ = 0;
  uint32_t max_chunks_ = 0;
  uint64_t slot_cap_ = 0, out_cap_ = 0, max_pieces_ = 0;
  bool timing_ = false;
  double kernel_s_ = 0;
  cudaStream_t stream_ = nullptr;
  cudaEvent_t ev_[8] = {};
  uint8_t *d_win_[2] = {nullptr, nullptr}, *d_dicts_ = nullptr, *d_out_ = nullptr;
  uint64_t *d_cand_ = nullptr, *d_piece_off_ = nullptr;
  NhGzChunk *d_recs_ = nullptr;
  uint16_t *d_slots_ = nullptr, *d_spill_ = nullptr;
  NhGzMember *d_mrec_ = nullptr, *d_spill_mrec_ = nullptr;
  NhGzEmit *d_emit_ = nullptr;
  NhGzJob *d_jobs_ = nullptr, *h_jobs_ = nullptr;
  uint32_t *d_piece_len_ = nullptr, *d_crcs_ = nullptr, *d_bad_ = nullptr;
  uint8_t *h_in_ = nullptr, *h_out_ = nullptr;
  NhGzChunk *h_recs_ = nullptr;
  NhGzMember *h_mrec_ = nullptr;
  NhGzEmit *h_emit_ = nullptr;
  uint64_t *h_piece_off_ = nullptr;
  uint32_t *h_piece_len_ = nullptr, *h_crcs_ = nullptr, *h_bad_ = nullptr;
};

/* nh_pipeline.cc: the records of one FASTA or FASTQ file (plain, gzip, BGZF with `threads` inflaters, bzip2),
 * read by the file pipeline's reader; inflating runs ahead on a thread of its own. */
class NhSeqReader {
 public:
  NhSeqReader();
  NhSeqReader(const NhSeqReader &) = delete;
  NhSeqReader &operator=(const NhSeqReader &) = delete;
  ~NhSeqReader();
  int open(const char *path, int threads); /* NH_OK, or NH_ERR_IO with nh_last_error() set */
  /* The next record: its header line (with the '>') and its sequence lines joined, valid until the next call.
   * 1: a record, 0: end of file, NH_ERR_IO: a read error (truncated or corrupt input) or malformed record. */
  int next(const char **hdr, size_t *hdr_len, const char **seq, size_t *seq_len);

 private:
  struct Impl;
  Impl *impl_;
};

int nh_set_error(int code, const char *fmt, ...);
int nh_db_build_filter(nh_db *db); /* after the cells are on the device (every open path; the synthetic builder calls it itself) */
/* zeroed table of `capacity` cells for the synthetic builder (nh_synth.cu), which fills it and builds the filter */
int nh_db_create_empty(const void *opts, size_t opts_len, const void *taxo, size_t taxo_len, uint64_t capacity, int device,
                       nh_db **out);
int nh_session_create_ex(nh_db *db, const nh_params_t *params, bool need_lookups, nh_session **out);
int nh_resolve_db_dir(const char *db_dir, std::string &out);

#endif
