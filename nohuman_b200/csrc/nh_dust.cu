/*
 * nh_dust.cu — dustmasker's symmetric DUST on the GPU (include/nohuman_gpu.h: nh_dust_mask, nh_dust_fasta,
 * nh_bench_dust).  The mask is defined in DESIGN.md §4f: over every run of A/C/G/T, the union of the bases of
 * the "perfect" triplet intervals that fit in one window.
 *
 *   chunks     the bases are cut into chunks (DUST_CHUNK bases, never across a record or piece); a chunk emits
 *              the perfect intervals whose LAST base lies in it, after replaying the window - 1 bases before it,
 *              which is all such an interval can depend on.  Bits go into a one-bit-per-base mask with atomicOr,
 *              so the mask is the same union for any chunking (NH_TEST_DUST_CHUNK=<bases> forces small chunks).
 *   k_dust_chunks   one warp per chunk, one step per base.  The window's <= 62 interval starts live in
 *              registers, two per lane (ring slot s = start & 63 in lane s & 31): r(a, e) and B[a], the best
 *              perfect interval found so far that starts at a, as an exact (r, l) pair.  Two ballots over the
 *              triplet ring give where the new triplet occurred, so r(a, e) = r(a, e - 1) + popc(those in
 *              [a, e - 1]); a ballot of suspicious starts skips the rest in the common case, else a warp
 *              prefix-max over younger starts decides which [a, e] are perfect.
 *   k_dust_apply    masked bases lower-cased, every other byte upper-cased (dustmasker's FASTA form).
 *
 * nh_dust_fasta reads records with NhSeqReader, cuts them into pieces overlapping by window - 1 bases, and runs
 * batches double-buffered in pinned memory: the host writes batch n and reads batch n + 2 while the GPU masks
 * batch n + 1.  A piece's intervals can mask bases in the overlap with the piece before it, so the last
 * window - 1 bases of a piece are written only after the next piece has been masked (DustWriter::pending_).
 */
#include <cuda_runtime.h>
#include <errno.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <memory>
#include <string>
#include <vector>

#include "../../include/nohuman_gpu.h"
#include "nh_internal.h"

#define CUDA_TRY(expr)                                                                       \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess)                                                                   \
      return nh_set_error(NH_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                          __FILE__, __LINE__);                                               \
  } while (0)

namespace {

constexpr uint32_t DUST_CHUNK = 4096; /* bases a chunk emits for; it reads up to window - 1 more */
constexpr uint32_t FULL = 0xFFFFFFFFu;

/* a warp's work: read bases [from, end) of the batch, emit the intervals whose last base is in [own, end) */
struct DustChunk {
  uint64_t from, own, end;
};

__device__ __forceinline__ uint64_t rotr64(uint64_t x, uint32_t s) { return s ? (x >> s) | (x << (64u - s)) : x; }

/* a score r / l packed as r << 8 | l (r <= 61 * 62 / 2, l <= 61); 1 (0 / 1) stands for "none" */
__device__ __forceinline__ bool score_gt(uint32_t x, uint32_t y) { return (x >> 8) * (y & 255u) > (y >> 8) * (x & 255u); }
__device__ __forceinline__ uint32_t score_max(uint32_t x, uint32_t y) { return score_gt(y, x) ? y : x; }

/* bits [x, y] of the mask, the warp's lanes taking a word each */
__device__ __forceinline__ void mark(uint32_t *mask, uint64_t x, uint64_t y, uint32_t lane) {
  for (uint64_t w = (x >> 5) + lane; w <= (y >> 5); w += 32) {
    uint32_t bits = FULL;
    if (w == (x >> 5)) bits &= FULL << (x & 31);
    if (w == (y >> 5)) bits &= FULL >> (31 - (y & 31));
    atomicOr(&mask[w], bits);
  }
}

__global__ void __launch_bounds__(256) k_dust_chunks(const uint8_t *__restrict__ bases, const DustChunk *__restrict__ chunks,
                                                     uint32_t n_chunks, uint32_t window, uint32_t level,
                                                     uint32_t *__restrict__ mask) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (warp >= n_chunks) return;
  const DustChunk ch = chunks[warp];
  const uint32_t max_d = window - 3; /* an interval [a, e] fits in the window when e - a <= window - 3 */
  /* ring slots lane and lane + 32: the triplet at that position (64: none yet), r(a, e) and B[a] of the start */
  uint32_t t0 = 64, t1 = 64, r0 = 0, r1 = 0, b0 = 1, b1 = 1;
  uint32_t tri = 0, run = 0, ntrip = 0; /* the current run: its last triplet, bases, triplets */
  bool pending = false;                 /* masked bases [ms, me] not yet marked */
  uint64_t ms = 0, me = 0;
  for (uint64_t g = ch.from; g < ch.end; g += 32) {
    const uint32_t nb = ch.end - g < 32 ? (uint32_t)(ch.end - g) : 32u;
    const uint32_t v = lane < nb ? bases[g + lane] : 0u;
    for (uint32_t k = 0; k < nb; k++) {
      const uint32_t c = __shfl_sync(FULL, v, k) | 0x20u;
      const uint32_t code = c == 'a' ? 0u : c == 'c' ? 1u : c == 'g' ? 2u : c == 't' ? 3u : 4u;
      if (code == 4u) { /* every other byte ends the run; stale slots are never live again */
        run = ntrip = 0;
        continue;
      }
      tri = ((tri << 2) | code) & 63u;
      if (++run < 3) continue;
      const uint32_t e = ntrip++, slot = e & 63u;
      if (lane == (slot & 31u)) { /* the new start a = e enters the slot of start e - 64 */
        if (slot >> 5) t1 = tri, r1 = 0, b1 = 1;
        else t0 = tri, r0 = 0, b0 = 1;
      }
      const uint64_t hit = (uint64_t)__ballot_sync(FULL, t0 == tri) | ((uint64_t)__ballot_sync(FULL, t1 == tri) << 32);
      const uint32_t d0 = (e - lane) & 63u, d1 = (e - lane - 32u) & 63u; /* l = e - a of the slots' starts */
      const bool live0 = d0 < ntrip && d0 <= max_d, live1 = d1 < ntrip && d1 <= max_d;
      if (live0) r0 += __popcll(rotr64(hit, lane) & ((1ull << d0) - 1));
      if (live1) r1 += __popcll(rotr64(hit, lane + 32u) & ((1ull << d1) - 1));
      const bool s0 = live0 && 10u * r0 > level * d0, s1 = live1 && 10u * r1 > level * d1;
      if (!__any_sync(FULL, s0 || s1)) continue;
      /* [a, e] is perfect iff suspicious and its score >= B[a], and >= max(B[s], score(s, e)) of every s > a */
      const uint32_t f0 = r0 << 8 | d0, f1 = r1 << 8 | d1;
      const uint32_t v0 = live0 ? (s0 ? score_max(b0, f0) : b0) : 1u, v1 = live1 ? (s1 ? score_max(b1, f1) : b1) : 1u;
      const uint32_t sa = (e - 2u * lane) & 63u, sb = (e - 2u * lane - 1u) & 63u; /* lane k: l = 2k, 2k + 1 */
      uint32_t x = __shfl_sync(FULL, v0, sa & 31u), y = __shfl_sync(FULL, v1, sa & 31u);
      const uint32_t va = (sa >> 5) ? y : x;
      x = __shfl_sync(FULL, v0, sb & 31u);
      y = __shfl_sync(FULL, v1, sb & 31u);
      const uint32_t vb = (sb >> 5) ? y : x;
      uint32_t acc = score_max(va, vb);
#pragma unroll
      for (uint32_t off = 1; off < 32; off <<= 1) {
        const uint32_t o = __shfl_up_sync(FULL, acc, off);
        if (lane >= off) acc = score_max(acc, o);
      }
      uint32_t ex = __shfl_up_sync(FULL, acc, 1);
      if (lane == 0) ex = 1u;
      const uint32_t xa = ex, xb = score_max(ex, va); /* best over l < 2k, l < 2k + 1 */
      x = __shfl_sync(FULL, xa, d0 >> 1);
      y = __shfl_sync(FULL, xb, d0 >> 1);
      const uint32_t younger0 = (d0 & 1u) ? y : x;
      x = __shfl_sync(FULL, xa, d1 >> 1);
      y = __shfl_sync(FULL, xb, d1 >> 1);
      const uint32_t younger1 = (d1 & 1u) ? y : x;
      const bool p0 = s0 && !score_gt(younger0, f0) && !score_gt(b0, f0);
      const bool p1 = s1 && !score_gt(younger1, f1) && !score_gt(b1, f1);
      if (p0) b0 = f0;
      if (p1) b1 = f1;
      /* the union of this step's perfect intervals: bases from the oldest start to the triplet's last base */
      const uint32_t oldest = __reduce_max_sync(FULL, max(p0 ? d0 + 1u : 0u, p1 ? d1 + 1u : 0u));
      const uint64_t i = g + k;
      if (!oldest || i < ch.own) continue;
      const uint64_t lo = i - 1u - oldest;
      if (pending && lo <= me + 1) {
        ms = lo < ms ? lo : ms;
        me = i;
      } else {
        if (pending) mark(mask, ms, me, lane);
        ms = lo, me = i, pending = true;
      }
    }
  }
  if (pending) mark(mask, ms, me, lane);
}

__global__ void __launch_bounds__(256) k_dust_apply(uint8_t *__restrict__ bases, const uint32_t *__restrict__ mask, uint64_t n) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t c = bases[i];
    const bool m = (mask[i >> 5] >> (i & 31)) & 1u;
    bases[i] = (uint8_t)(m ? (c | 0x20u) : (c >= 'a' && c <= 'z' ? c - 32u : c));
  }
}

uint32_t chunk_bases() {
  /* NH_TEST_DUST_CHUNK=<bases>: tests force small chunks so that intervals straddle chunk borders */
  if (const char *e = getenv("NH_TEST_DUST_CHUNK")) {
    const unsigned long v = strtoul(e, nullptr, 10);
    if (v >= 1 && v <= (1ul << 24)) return (uint32_t)v;
  }
  return DUST_CHUNK;
}

/* the chunks of the piece [start, end) of the batch that emit for bases [own, end) */
void add_chunks(std::vector<DustChunk> &out, uint64_t start, uint64_t own, uint64_t end, uint32_t window, uint32_t ch) {
  for (uint64_t c = own; c < end; c += ch) {
    const uint64_t from = c - start > window - 1 ? c - (window - 1) : start;
    out.push_back(DustChunk{from, c, std::min<uint64_t>(end, c + ch)});
  }
}

int check_params(int window, int level) {
  if (window < 4 || window > 64) return nh_set_error(NH_ERR_INVALID, "DUST window %d is out of range (4..64)", window);
  if (level < 1 || level > 255) return nh_set_error(NH_ERR_INVALID, "DUST level %d is out of range (1..255)", level);
  return NH_OK;
}

int device_check(int device) {
  int nd = 0;
  if (cudaGetDeviceCount(&nd) != cudaSuccess || nd < 1) {
    cudaGetLastError();
    return nh_set_error(NH_ERR_CUDA, "no CUDA device (no CPU path)");
  }
  if (device < 0 || device >= nd) return nh_set_error(NH_ERR_INVALID, "no CUDA device %d", device);
  return NH_OK;
}

/* The device side of one batch: bases, chunks and the mask, on a stream of its own. */
class DustMasker {
 public:
  ~DustMasker() {
    if (stream_) cudaStreamSynchronize(stream_);
    cudaFree(d_bases_);
    cudaFree(d_chunks_);
    cudaFree(d_mask_);
    for (auto ev : ev_)
      if (ev) cudaEventDestroy(ev);
    if (stream_) cudaStreamDestroy(stream_);
  }
  int open(int device, uint64_t max_bases, uint64_t max_chunks, int window, int level) {
    if (int rc = device_check(device)) return rc;
    CUDA_TRY(cudaSetDevice(device));
    window_ = (uint32_t)window;
    level_ = (uint32_t)level;
    max_bases_ = max_bases;
    max_chunks_ = max_chunks;
    CUDA_TRY(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
    for (auto &ev : ev_) CUDA_TRY(cudaEventCreate(&ev));
    CUDA_TRY(cudaMalloc(&d_bases_, max_bases + 32));
    CUDA_TRY(cudaMalloc(&d_chunks_, std::max<uint64_t>(max_chunks, 1) * sizeof(DustChunk)));
    CUDA_TRY(cudaMalloc(&d_mask_, (max_bases / 32 + 2) * 4));
    return NH_OK;
  }
  /* the kernels over the nb bases and n chunks already on the device */
  void kernels(uint64_t nb, uint64_t n) {
    cudaMemsetAsync(d_mask_, 0, (nb / 32 + 1) * 4, stream_);
    if (n) k_dust_chunks<<<(unsigned)((n + 7) / 8), 256, 0, stream_>>>(d_bases_, d_chunks_, (uint32_t)n, window_, level_, d_mask_);
    if (nb) k_dust_apply<<<(unsigned)std::min<uint64_t>((nb + 255) / 256, 1u << 16), 256, 0, stream_>>>(d_bases_, d_mask_, nb);
  }
  /* bases[0..nb) masked in place, asynchronously (bases and chunks should be pinned for the copies to overlap) */
  int launch(uint8_t *bases, uint64_t nb, const DustChunk *chunks, uint64_t n) {
    if (nb > max_bases_ || n > max_chunks_ || n >= (1ull << 32)) return nh_set_error(NH_ERR_CAPACITY, "DUST batch too large");
    CUDA_TRY(cudaMemcpyAsync(d_bases_, bases, nb, cudaMemcpyHostToDevice, stream_));
    CUDA_TRY(cudaMemcpyAsync(d_chunks_, chunks, n * sizeof(DustChunk), cudaMemcpyHostToDevice, stream_));
    kernels(nb, n);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(bases, d_bases_, nb, cudaMemcpyDeviceToHost, stream_));
    return NH_OK;
  }
  int sync() {
    const cudaError_t e = cudaStreamSynchronize(stream_);
    return e == cudaSuccess ? NH_OK : nh_set_error(NH_ERR_CUDA, "DUST batch failed: %s", cudaGetErrorString(e));
  }
  /* mean device time of the kernels over `iters` runs after one warm-up, bases and chunks copied once */
  int time_kernels(const uint8_t *bases, uint64_t nb, const DustChunk *chunks, uint64_t n, int iters, double *seconds) {
    if (nb > max_bases_ || n > max_chunks_) return nh_set_error(NH_ERR_CAPACITY, "DUST batch too large");
    CUDA_TRY(cudaMemcpyAsync(d_bases_, bases, nb, cudaMemcpyHostToDevice, stream_));
    CUDA_TRY(cudaMemcpyAsync(d_chunks_, chunks, n * sizeof(DustChunk), cudaMemcpyHostToDevice, stream_));
    kernels(nb, n);
    CUDA_TRY(cudaEventRecord(ev_[0], stream_));
    for (int i = 0; i < iters; i++) kernels(nb, n);
    CUDA_TRY(cudaEventRecord(ev_[1], stream_));
    CUDA_TRY(cudaGetLastError());
    if (int rc = sync()) return rc;
    float ms = 0;
    CUDA_TRY(cudaEventElapsedTime(&ms, ev_[0], ev_[1]));
    *seconds = ms / 1e3 / iters;
    return NH_OK;
  }

 private:
  uint32_t window_ = 64, level_ = 20;
  uint64_t max_bases_ = 0, max_chunks_ = 0;
  cudaStream_t stream_ = nullptr;
  cudaEvent_t ev_[2] = {nullptr, nullptr};
  uint8_t *d_bases_ = nullptr;
  DustChunk *d_chunks_ = nullptr;
  uint32_t *d_mask_ = nullptr;
};

/* records concatenated in host memory: every record one piece */
int records_chunks(const uint64_t *offsets, uint64_t n_seqs, uint32_t window, std::vector<DustChunk> &out) {
  const uint32_t ch = chunk_bases();
  for (uint64_t s = 0; s < n_seqs; s++) {
    if (offsets[s + 1] < offsets[s]) return nh_set_error(NH_ERR_INVALID, "offsets are not ascending at %llu", (unsigned long long)s);
    add_chunks(out, offsets[s], offsets[s], offsets[s + 1], window, ch);
  }
  return NH_OK;
}

int records_check(const uint8_t *seq, const uint64_t *offsets, uint64_t n_seqs, const void *out) {
  if (!offsets || (n_seqs && !seq) || !out) return nh_set_error(NH_ERR_INVALID, "null argument");
  if (offsets[0] != 0) return nh_set_error(NH_ERR_INVALID, "offsets[0] must be 0");
  return NH_OK;
}

/* ------------------------------------------------------------------ */
/* file to file                                                        */

using Clock = std::chrono::steady_clock;

/* a piece of a record in a batch: bases [off, off + len); the header (for the record's first piece) */
struct DustPiece {
  uint64_t off, len;
  size_t hdr_off, hdr_len;
  bool first, last;
};

/* one batch: bases and chunks in pinned memory, pieces and headers in ordinary memory */
struct DustBatch {
  uint8_t *bases = nullptr;
  DustChunk *chunks = nullptr;
  uint64_t nb = 0, n_chunks = 0;
  std::vector<DustPiece> pieces;
  std::string headers;
  ~DustBatch() {
    if (bases) cudaFreeHost(bases);
    if (chunks) cudaFreeHost(chunks);
  }
};

/* reads one file's records and cuts them into batches of pieces that overlap by window - 1 bases */
class DustReader {
 public:
  DustReader(uint32_t window, uint64_t max_bases, uint32_t max_pieces)
      : window_(window), max_bases_(max_bases), max_pieces_(max_pieces), chunk_(chunk_bases()) {}
  int open(const char *path, int threads) { return reader_.open(path, threads); }
  /* fills b; false when the file is exhausted and b is empty, or on error (rc set) */
  bool fill(DustBatch &b, int &rc) {
    b.nb = b.n_chunks = 0;
    b.pieces.clear();
    b.headers.clear();
    std::vector<DustChunk> &ch = chunks_;
    ch.clear();
    while (b.pieces.size() < max_pieces_) {
      if (!have_) {
        const char *h, *s;
        size_t hl, sl;
        const int r = reader_.next(&h, &hl, &s, &sl);
        if (r < 0) {
          rc = r;
          return false;
        }
        if (r == 0) break;
        hdr_ = h;
        hdr_len_ = hl;
        seq_ = (const uint8_t *)s;
        len_ = sl;
        pos_ = 0;
        have_ = true;
      }
      const uint64_t room = max_bases_ - b.nb, left = len_ - pos_;
      const uint64_t take = std::min(left, room);
      if (take < left && take < window_ + 4096u) break; /* too little room for a useful piece: next batch */
      DustPiece p{b.nb, take, b.headers.size(), 0, pos_ == 0, take == left};
      if (p.first) {
        b.headers.append(hdr_, hdr_len_);
        p.hdr_len = hdr_len_;
      }
      memcpy(b.bases + b.nb, seq_ + pos_, take);
      add_chunks(ch, b.nb, p.first ? b.nb : b.nb + window_ - 1, b.nb + take, window_, chunk_);
      b.nb += take;
      b.pieces.push_back(p);
      if (p.last)
        have_ = false;
      else
        pos_ += take - (window_ - 1); /* the next piece replays the window - 1 bases before its own */
    }
    memcpy(b.chunks, ch.data(), ch.size() * sizeof(DustChunk));
    b.n_chunks = ch.size();
    return !b.pieces.empty();
  }
  uint64_t max_chunks() const { return max_bases_ / chunk_ + max_pieces_ + 1; }

 private:
  uint32_t window_;
  uint64_t max_bases_;
  uint32_t max_pieces_, chunk_;
  NhSeqReader reader_;
  std::vector<DustChunk> chunks_;
  bool have_ = false;
  const char *hdr_ = nullptr;
  size_t hdr_len_ = 0;
  const uint8_t *seq_ = nullptr;
  uint64_t len_ = 0, pos_ = 0;
};

/* writes masked pieces as FASTA (60 bases a line) or intervals, and counts */
class DustWriter {
 public:
  DustWriter(FILE *f, int format, uint32_t window) : f_(f), format_(format), window_(window) {}
  int write(DustBatch &b) {
    out_.clear();
    for (const DustPiece &p : b.pieces) {
      uint8_t *s = b.bases + p.off;
      if (p.first) {
        out_.append(b.headers, p.hdr_off, p.hdr_len);
        out_.push_back('\n');
        col_ = rec_pos_ = 0;
        open_ = false;
      } else { /* the overlap: masked where either piece masked it */
        for (size_t k = 0; k < pending_.size(); k++)
          if (pending_[k] >= 'a') s[k] |= 0x20;
      }
      const uint64_t n = p.last ? p.len : p.len - (window_ - 1);
      if (!p.last) pending_.assign((const char *)s + n, window_ - 1);
      emit(s, n);
      if (p.last) {
        if (open_) close_interval(rec_pos_ - 1);
        if (format_ == NH_DUST_FASTA && col_) out_.push_back('\n');
        stats.sequences++;
      }
    }
    if (!out_.empty() && fwrite(out_.data(), 1, out_.size(), f_) != out_.size())
      return nh_set_error(NH_ERR_IO, "writing the DUST output failed: %s", strerror(errno));
    return NH_OK;
  }
  nh_dust_stats_t stats{};

 private:
  void close_interval(uint64_t end) {
    open_ = false;
    stats.intervals++;
    if (format_ == NH_DUST_INTERVAL) {
      char line[64];
      out_.append(line, (size_t)snprintf(line, sizeof line, "%llu - %llu\n", (unsigned long long)start_, (unsigned long long)end));
    }
  }
  void emit(const uint8_t *s, uint64_t n) {
    for (uint64_t i = 0; i < n; i++) {
      const bool m = s[i] >= 'a';
      if (m && !open_) open_ = true, start_ = rec_pos_ + i;
      if (!m && open_) close_interval(rec_pos_ + i - 1);
      stats.masked += m;
    }
    rec_pos_ += n;
    stats.bases += n;
    if (format_ != NH_DUST_FASTA) return;
    for (uint64_t i = 0; i < n;) {
      const uint64_t k = std::min<uint64_t>(60 - col_, n - i);
      out_.append((const char *)s + i, k);
      i += k;
      col_ += k;
      if (col_ == 60) out_.push_back('\n'), col_ = 0;
    }
  }
  FILE *f_;
  int format_;
  uint32_t window_;
  std::string out_, pending_;
  uint64_t col_ = 0, rec_pos_ = 0, start_ = 0;
  bool open_ = false;
};

int dust_file(const nh_dust_params_t &p, FILE *f, nh_dust_stats_t *stats) {
  const uint32_t max_pieces = (uint32_t)(p.batch_bases / 64 + 1024);
  DustReader reader((uint32_t)p.window, p.batch_bases, max_pieces);
  if (int rc = reader.open(p.in_path, p.threads)) return rc;
  DustBatch hb[2]; /* declared before the masker, whose destructor waits for copies into them */
  DustMasker M;
  if (int rc = M.open(p.device, p.batch_bases, reader.max_chunks(), p.window, p.level)) return rc;
  for (auto &b : hb) {
    CUDA_TRY(cudaHostAlloc(&b.bases, p.batch_bases + 32, cudaHostAllocDefault));
    CUDA_TRY(cudaHostAlloc(&b.chunks, reader.max_chunks() * sizeof(DustChunk), cudaHostAllocDefault));
  }
  DustWriter W(f, p.format, (uint32_t)p.window);
  int rc = NH_OK;
  bool have[2] = {false, false};
  have[0] = reader.fill(hb[0], rc);
  if (have[0] && !rc) rc = M.launch(hb[0].bases, hb[0].nb, hb[0].chunks, hb[0].n_chunks);
  if (have[0] && !rc) have[1] = reader.fill(hb[1], rc);
  for (int cur = 0; have[cur] && !rc; cur ^= 1) {
    if ((rc = M.sync())) break;
    DustBatch &nx = hb[cur ^ 1];
    if (have[cur ^ 1] && (rc = M.launch(nx.bases, nx.nb, nx.chunks, nx.n_chunks))) break;
    if ((rc = W.write(hb[cur]))) break;
    have[cur] = reader.fill(hb[cur], rc); /* two batches on: the GPU is masking the next one meanwhile */
  }
  if (!rc && fflush(f) != 0) rc = nh_set_error(NH_ERR_IO, "writing the DUST output failed: %s", strerror(errno));
  *stats = W.stats;
  return rc;
}

}  // namespace

extern "C" int nh_dust_mask(int device, const uint8_t *seq, const uint64_t *offsets, uint64_t n_seqs, int window,
                            int level, uint8_t *out) {
  if (int rc = records_check(seq, offsets, n_seqs, out)) return rc;
  if (int rc = check_params(window, level)) return rc;
  std::vector<DustChunk> chunks;
  if (int rc = records_chunks(offsets, n_seqs, (uint32_t)window, chunks)) return rc;
  const uint64_t nb = offsets[n_seqs];
  DustMasker M;
  if (int rc = M.open(device, nb, chunks.size(), window, level)) return rc;
  if (nb) memcpy(out, seq, nb);
  if (int rc = M.launch(out, nb, chunks.data(), chunks.size())) return rc;
  return M.sync();
}

extern "C" int nh_bench_dust(int device, const uint8_t *seq, const uint64_t *offsets, uint64_t n_seqs, int iters,
                             double *out_seconds) {
  if (int rc = records_check(seq, offsets, n_seqs, out_seconds)) return rc;
  if (iters < 1) return nh_set_error(NH_ERR_INVALID, "iters must be positive");
  std::vector<DustChunk> chunks;
  if (int rc = records_chunks(offsets, n_seqs, 64, chunks)) return rc;
  DustMasker M;
  if (int rc = M.open(device, offsets[n_seqs], chunks.size(), 64, 20)) return rc;
  return M.time_kernels(seq, offsets[n_seqs], chunks.data(), chunks.size(), iters, out_seconds);
}

extern "C" int nh_dust_fasta(const nh_dust_params_t *pin, nh_dust_stats_t *stats) {
  if (!pin || !pin->in_path) return nh_set_error(NH_ERR_INVALID, "bad argument");
  nh_dust_params_t p = *pin;
  if (!p.window) p.window = 64;
  if (!p.level) p.level = 20;
  if (!p.batch_bases) p.batch_bases = 256ull << 20;
  if (int rc = check_params(p.window, p.level)) return rc;
  if (p.format != NH_DUST_FASTA && p.format != NH_DUST_INTERVAL)
    return nh_set_error(NH_ERR_INVALID, "unknown DUST output format %d", p.format);
  if (p.batch_bases < 8192 || p.batch_bases > (1ull << 31))
    return nh_set_error(NH_ERR_INVALID, "batch_bases must be in [8192, 2^31]");
  if (int rc = device_check(p.device)) return rc; /* before the output file is created */
  const auto t0 = Clock::now();
  const bool to_stdout = !p.out_path || !strcmp(p.out_path, "-");
  FILE *f = to_stdout ? stdout : fopen(p.out_path, "wb");
  if (!f) return nh_set_error(NH_ERR_IO, "cannot create %s: %s", p.out_path, strerror(errno));
  nh_dust_stats_t S;
  memset(&S, 0, sizeof S);
  int rc = dust_file(p, f, &S);
  if (!to_stdout && fclose(f) != 0 && !rc) rc = nh_set_error(NH_ERR_IO, "writing %s failed: %s", p.out_path, strerror(errno));
  if (rc) {
    if (!to_stdout) unlink(p.out_path); /* a failed run leaves no partial output behind */
    return rc;
  }
  S.seconds = std::chrono::duration<double>(Clock::now() - t0).count();
  if (stats) *stats = S;
  return NH_OK;
}
