/*
 * nh_pipeline.cc — the file API of libnohuman_gpu.so: nh_run_files() is the
 * in-process stand-in for `kraken.run(&kraken_cmd)` (reference
 * src/main.rs:270, argv built at src/main.rs:210-267) plus the compression
 * pass that follows it (src/main.rs:340-368, src/compression.rs:182-268).
 *
 *   reader thread per input file   inflate (zlib; bzip2 through a pipe) + FASTQ/FASTA parse
 *        |  chunks of NH_CHUNK_RECORDS records
 *   classifier threads (2 per GPU) mates interleaved into PINNED bases/offsets,
 *        |                         nh_classify_batch (H2D, kernels, D2H) on their own session,
 *        |                         kept records re-serialised the way kraken2 prints them
 *   writer thread                  batches back in input order, cut into blocks
 *   compressor pool (-t threads)   every block an independent gzip member / zstd frame
 *        |                         (what gzp does for the reference), written in order
 *   final out1 / out2              no temporary FASTQ, no second pass
 *
 * With --kraken-output the sessions keep per-sequence hit runs
 * (nh_last_batch_runs) and the writer prints kraken2's per-read line
 * "C|U <id> <taxid> <len[|len2]> <hitlist>" (classify.cc, AddHitlistString);
 * with --kraken-report it prints the clade-aggregated report at the end
 * (reports.cc ReportKrakenStyle / KrakenReportDFS).
 *
 * What kraken2 does on this path and is restated here (upstream seqreader.cc /
 * classify.cc, SURVEY.md A.6): format auto-detected from the first byte ('@'
 * FASTQ, '>' FASTA); header/sequence/quality lines stripped of trailing
 * whitespace; FASTA sequences joined to one line; records written as
 * header\nseq\n+\nquals\n (or header\nseq\n); classified records get
 * " kraken:taxid|<external id>" appended to the header; paired input is read
 * in lock step and stops at the shorter file; output order == input order.
 */
#include <dlfcn.h>
#include <fcntl.h>
#include <spawn.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <errno.h>
#include <sys/socket.h>
#include <sys/stat.h>
#include <sys/wait.h>
#include <unistd.h>
#include <zlib.h>

#include <chrono>
#include <condition_variable>
#include <deque>
#include <algorithm>
#include <atomic>
#include <memory>
#include <unordered_map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/nohuman_gpu.h"
#include "nh_internal.h"
#include "nh_ordered.h"

extern char **environ;

namespace {

constexpr size_t NH_CHUNK_RECORDS = 1u << 16; /* records per reader chunk (per file) */
constexpr uint64_t NH_CHUNK_BASES = 48u << 20;  /* ... or this many bases in the first file's chunk, whichever comes first */
constexpr size_t NH_CHUNK_TEXT = 1u << 30;      /* ... or this much header + sequence + quality text */
constexpr uint64_t NH_BATCH_BASES = 64u << 20;  /* bases per nh_classify_batch call (session capacity; grows for a longer single unit) */
constexpr size_t NH_OUT_BLOCK = 1u << 20;     /* uncompressed bytes per compression block */

/* ------------------------------------------------------------------ */
/* busy time per pipeline stage (nh_run_stats_t.busy_*): what limits the file path is a host
 * question, so every stage accounts for the time it actually works */
enum Stage { ST_INFLATE = 0, ST_PARSE, ST_STAGE, ST_CLASSIFY, ST_SERIALISE, ST_COMPRESS, ST_WRITE, ST_COUNT };
struct StageClock {
  std::atomic<uint64_t> ns[ST_COUNT];
  StageClock() {
    for (auto &x : ns) x = 0;
  }
};
struct Busy {
  StageClock *c;
  int st;
  std::chrono::steady_clock::time_point t0;
  Busy(StageClock *clk, int stage) : c(clk), st(stage), t0(std::chrono::steady_clock::now()) {}
  ~Busy() {
    if (c) c->ns[st] += (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count();
  }
};

/* ------------------------------------------------------------------ */
/* small blocking queue                                                */

template <typename T>
class Channel {
 public:
  explicit Channel(size_t cap) : cap_(cap) {}
  bool push(T &&v) {
    std::unique_lock<std::mutex> lk(m_);
    not_full_.wait(lk, [&] { return q_.size() < cap_ || closed_; });
    if (closed_) return false;
    q_.push_back(std::move(v));
    not_empty_.notify_one();
    return true;
  }
  bool pop(T &out) {
    std::unique_lock<std::mutex> lk(m_);
    not_empty_.wait(lk, [&] { return !q_.empty() || closed_; });
    if (q_.empty()) return false;
    out = std::move(q_.front());
    q_.pop_front();
    not_full_.notify_one();
    return true;
  }
  void close() {
    std::lock_guard<std::mutex> lk(m_);
    closed_ = true;
    not_empty_.notify_all();
    not_full_.notify_all();
  }

 private:
  std::mutex m_;
  std::condition_variable not_full_, not_empty_;
  std::deque<T> q_;
  size_t cap_;
  bool closed_ = false;
};

/* ------------------------------------------------------------------ */
/* input: plain / gzip through zlib, bzip2 through `bzip2 -dc`          */

static int spawn_filter(const std::vector<std::string> &argv, int stdin_fd, int stdout_fd, pid_t *pid) {
  posix_spawn_file_actions_t fa;
  posix_spawn_file_actions_init(&fa);
  if (stdin_fd >= 0) posix_spawn_file_actions_adddup2(&fa, stdin_fd, 0);
  if (stdout_fd >= 0) posix_spawn_file_actions_adddup2(&fa, stdout_fd, 1);
  std::vector<char *> av;
  for (auto &a : argv) av.push_back(const_cast<char *>(a.c_str()));
  av.push_back(nullptr);
  int rc = posix_spawnp(pid, av[0], &fa, nullptr, av.data(), environ);
  posix_spawn_file_actions_destroy(&fa);
  return rc;
}

/* ------------------------------------------------------------------ */
/* blocked gzip (BGZF: what bgzip, bcl2fastq and this library write): every member carries its
 * compressed size in a 'BC' extra subfield, so members can be inflated in parallel */

static bool bgzf_block_size(const unsigned char *hdr, size_t n, size_t *xlen, size_t *bsize) {
  /* gzip magic and deflate (BGZF_HEADER[0..2]) with FEXTRA set */
  if (n < 12 || memcmp(hdr, BGZF_HEADER, 3) != 0 || !(hdr[3] & 4)) return false;
  *xlen = hdr[10] | (size_t)hdr[11] << 8;
  if (n < 12 + *xlen) return false;
  for (size_t o = 12; o + 4 <= 12 + *xlen;) {
    const size_t slen = hdr[o + 2] | (size_t)hdr[o + 3] << 8;
    /* 'B', 'C' and a 2-byte length: BGZF_HEADER[12..15] */
    if (memcmp(hdr + o, BGZF_HEADER + 12, 4) == 0 && o + 6 <= 12 + *xlen) {
      *bsize = (hdr[o + 4] | (size_t)hdr[o + 5] << 8) + 1;
      return true;
    }
    o += 4 + slen;
  }
  return false;
}

/* Streaming inflate of ordinary gzip (any number of concatenated members), restating what zlib's
 * gzread does for kraken2's reader — except that a stream that ends inside a member is an ERROR
 * here, where gzread hands back the bytes it has and only flags Z_BUF_ERROR in gzerror(). */
class GzipStream {
 public:
  ~GzipStream() {
    if (init_) inflateEnd(&zs_);
  }
  /* `f` is positioned at the first byte of a gzip member; `pre` = bytes already consumed from it */
  bool begin(FILE *f, const unsigned char *pre, size_t n_pre) {
    f_ = f;
    in_.resize(1u << 20);
    memcpy(&in_[0], pre, n_pre);
    zs_ = z_stream{};
    if (inflateInit2(&zs_, 15 + 16) != Z_OK) return false;
    init_ = true;
    zs_.next_in = (Bytef *)&in_[0];
    zs_.avail_in = (uInt)n_pre;
    return true;
  }
  /* fills `out` (capacity bytes); returns bytes produced, 0 at the clean end, -1 on a corrupt or truncated stream */
  long read(char *out, size_t cap) {
    if (done_) return 0;
    zs_.next_out = (Bytef *)out;
    zs_.avail_out = (uInt)cap;
    while (zs_.avail_out > 0) {
      if (zs_.avail_in == 0) {
        const size_t n = fread(&in_[0], 1, in_.size(), f_);
        if (n == 0) {
          if (ferror(f_) || in_member_) return -1; /* the file ends inside a member: truncated */
          done_ = true;
          break;
        }
        zs_.next_in = (Bytef *)&in_[0];
        zs_.avail_in = (uInt)n;
      }
      if (!in_member_) {
        /* between members: another gzip header continues the stream, anything else is trailing
         * garbage, which gzread ignores */
        if (zs_.next_in[0] != 0x1f) {
          done_ = true;
          break;
        }
        inflateReset(&zs_);
        in_member_ = true;
      }
      const int rc = inflate(&zs_, Z_NO_FLUSH);
      if (rc == Z_STREAM_END) {
        in_member_ = false;
      } else if (rc != Z_OK && rc != Z_BUF_ERROR) {
        return -1;
      }
    }
    return (long)(cap - zs_.avail_out);
  }

 private:
  FILE *f_ = nullptr;
  z_stream zs_{};
  std::string in_;
  bool init_ = false, in_member_ = true, done_ = false;
};

class BgzfReader {
 public:
  ~BgzfReader() { close(); }
  bool open(const std::string &path, int threads, StageClock *clk) {
    clk_ = clk;
    f_ = fopen(path.c_str(), "rb");
    if (!f_) return false;
    setvbuf(f_, nullptr, _IOFBF, 4u << 20);
    producer_ = std::thread([this] { produce(); });
    for (int i = 0; i < threads; i++) workers_.emplace_back([this] { work(); });
    return true;
  }
  /* next run of inflated bytes, in file order; 0 at the end, -1 on error */
  long next(std::string &out) {
    std::shared_ptr<Blk> b = q_.pop();
    if (!b) return failed_ ? -1 : 0;
    if (!b->ok) {
      fail();
      return -1;
    }
    out.swap(b->raw);
    return (long)out.size();
  }
  void close() {
    q_.stop();
    if (producer_.joinable()) producer_.join();
    for (auto &t : workers_)
      if (t.joinable()) t.join();
    workers_.clear();
    if (f_) fclose(f_), f_ = nullptr;
  }

 private:
  /* one task = up to NH_BGZF_BATCH consecutive members (fewer wake-ups than one per 64 KiB member) */
  static constexpr int NH_BGZF_BATCH = 16;
  struct Blk {
    std::string comp, raw;
    std::vector<uint32_t> clen; /* deflate bytes + 8-byte trailer of each member in comp */
    bool ok = true;
  };
  typedef OrderedQueue<Blk> Queue;
  /* a bad member or stream fails the whole reader at once: next() returns -1 from then on */
  void fail() {
    failed_ = true;
    q_.stop();
  }
  /* A member without the BC subfield (e.g. `cat blocked.gz plain.gz`): zlib and kraken2 read such a
   * file, so the rest of it is inflated as an ordinary gzip stream on this thread. */
  void serial_tail(const unsigned char *pre, size_t n_pre) {
    GzipStream gs;
    if (!gs.begin(f_, pre, n_pre)) return fail();
    for (;;) {
      auto b = std::make_shared<Blk>();
      b->raw.resize(1u << 20);
      long n;
      {
        Busy busy(clk_, ST_INFLATE);
        n = gs.read(&b->raw[0], b->raw.size());
      }
      if (n < 0) return fail();
      if (n == 0) break;
      b->raw.resize((size_t)n);
      if (!q_.push(b, Queue::DONE)) return;
    }
    q_.close();
  }
  void produce() {
    bool at_end = false;
    while (!at_end) {
      auto b = std::make_shared<Blk>();
      bool bad = false, plain_member = false;
      unsigned char hdr[12 + 65536];
      size_t n_hdr = 0;
      for (int k = 0; k < NH_BGZF_BATCH; k++) {
        size_t n = fread(hdr, 1, 12, f_);
        n_hdr = n;
        if (n == 0) { /* clean end of file */
          at_end = true;
          break;
        }
        if (n == 12 && hdr[0] == 0x1f && hdr[1] == 0x8b && !(hdr[3] & 4)) { /* gzip, but no extra field */
          plain_member = true;
          break;
        }
        size_t xlen = n == 12 ? (hdr[10] | (size_t)hdr[11] << 8) : 0, bsize = 0;
        if (n != 12 || fread(hdr + 12, 1, xlen, f_) != xlen) {
          bad = true;
          break;
        }
        n_hdr = 12 + xlen;
        if (!bgzf_block_size(hdr, 12 + xlen, &xlen, &bsize)) {
          if (hdr[0] == 0x1f && hdr[1] == 0x8b)
            plain_member = true; /* extra field without BC */
          else
            bad = true; /* not gzip at all: gzread would stop here; a blocked file never has trailing garbage */
          break;
        }
        if (bsize < 12 + xlen + 8) {
          bad = true;
          break;
        }
        const size_t len = bsize - 12 - xlen, at = b->comp.size();
        b->comp.resize(at + len);
        if (fread(&b->comp[at], 1, len, f_) != len) {
          bad = true;
          break;
        }
        b->clen.push_back((uint32_t)len);
      }
      if (bad) return fail();
      if (!b->clen.empty() && !q_.push(b, Queue::QUEUED)) return;
      if (plain_member) return serial_tail(hdr, n_hdr);
    }
    q_.close();
  }
  void work() {
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    if (inflateInit2(&zs, -15) != Z_OK) return;
    while (std::shared_ptr<Blk> b = q_.take()) {
      Busy busy(clk_, ST_INFLATE);
      bool ok = true;
      size_t total = 0, at = 0;
      for (uint32_t len : b->clen) {
        const unsigned char *tr = (const unsigned char *)b->comp.data() + at + len - 8;
        const size_t isize = tr[4] | tr[5] << 8 | tr[6] << 16 | (size_t)tr[7] << 24;
        if (isize > 65536) ok = false; /* the BGZF limit; also bounds the allocation below */
        total += isize;
        at += len;
      }
      if (ok) b->raw.resize(total);
      size_t out_at = 0;
      at = 0;
      for (uint32_t len : b->clen) {
        if (!ok) break;
        const size_t clen = len - 8;
        const unsigned char *tr = (const unsigned char *)b->comp.data() + at + clen;
        const uint32_t crc = tr[0] | tr[1] << 8 | tr[2] << 16 | (uint32_t)tr[3] << 24;
        const uint32_t isize = tr[4] | tr[5] << 8 | tr[6] << 16 | (uint32_t)tr[7] << 24;
        inflateReset(&zs);
        zs.next_in = (Bytef *)b->comp.data() + at;
        zs.avail_in = (uInt)clen;
        zs.next_out = (Bytef *)(isize ? &b->raw[out_at] : nullptr);
        zs.avail_out = isize;
        const int rc = isize ? inflate(&zs, Z_FINISH) : Z_STREAM_END;
        ok = ok && rc == Z_STREAM_END && zs.total_out == isize &&
             (uint32_t)crc32(crc32(0L, Z_NULL, 0), (const Bytef *)b->raw.data() + out_at, isize) == crc;
        out_at += isize;
        at += len;
      }
      std::string().swap(b->comp);
      b->ok = ok;
      q_.done(b);
    }
    inflateEnd(&zs);
  }
  FILE *f_ = nullptr;
  StageClock *clk_ = nullptr;
  std::thread producer_;
  std::vector<std::thread> workers_;
  Queue q_{64};
  std::atomic<bool> failed_{false};
};

/* Decompressed bytes of one input file, produced ahead of the parser by a thread of its own
 * (blocked gzip: by the BgzfReader's pool), so that inflate and FASTQ parsing overlap.  The reference
 * leaves this to kraken2, which inflates inline in its reader (src/main.rs:267 hands it the paths). */
class InputStream {
 public:
  ~InputStream() { close(); }
  int inflate_threads() const { return bgzf_ ? bgzf_threads_ : 1; }
  bool open(const std::string &path, int threads, std::string &err, StageClock *clk) {
    clk_ = clk;
    FILE *f = fopen(path.c_str(), "rb");
    if (!f) {
      err = "cannot open " + path;
      return false;
    }
    unsigned char magic[64] = {0};
    size_t n = fread(magic, 1, sizeof magic, f);
    size_t xlen = 0, bsize = 0;
    if (threads > 1 && bgzf_block_size(magic, n, &xlen, &bsize)) {
      /* blocked gzip: members inflated in parallel */
      fclose(f);
      bgzf_.reset(new BgzfReader());
      bgzf_threads_ = threads;
      if (!bgzf_->open(path, threads, clk)) {
        err = "cannot open " + path;
        return false;
      }
      return true;
    }
    if (n >= 6 && magic[0] == 0xFD && !memcmp(magic + 1, "7zXZ", 4)) {
      fclose(f);
      err = path + ": xz-compressed input is not supported (kraken2 reads plain, gzip and bzip2)";
      return false;
    }
    if (n >= 4 && magic[0] == 0x28 && magic[1] == 0xB5 && magic[2] == 0x2F && magic[3] == 0xFD) {
      fclose(f);
      err = path + ": zstd-compressed input is not supported (kraken2 reads plain, gzip and bzip2)";
      return false;
    }
    if (n >= 3 && magic[0] == 'B' && magic[1] == 'Z' && magic[2] == 'h') {
      fclose(f);
      int fds[2];
      if (pipe2(fds, O_CLOEXEC)) {
        err = "pipe failed";
        return false;
      }
      int in = ::open(path.c_str(), O_RDONLY | O_CLOEXEC);
      if (in < 0 || spawn_filter({"bzip2", "-dc"}, in, fds[1], &pid_) != 0) {
        err = "cannot run bzip2 to read " + path;
        if (in >= 0) ::close(in);
        ::close(fds[0]);
        ::close(fds[1]);
        return false;
      }
      ::close(in);
      ::close(fds[1]);
      file_ = fdopen(fds[0], "rb");
      if (!file_) {
        ::close(fds[0]);
        err = "cannot read from bzip2";
        return false;
      }
      kind_ = 'b';
    } else if (n >= 2 && magic[0] == 0x1f && magic[1] == 0x8b) {
      file_ = f;
      setvbuf(file_, nullptr, _IONBF, 0);
      if (!gz_.begin(file_, magic, n)) {
        err = "zlib initialisation failed";
        return false;
      }
      kind_ = 'g';
    } else {
      file_ = f;
      rewind(file_);
      setvbuf(file_, nullptr, _IONBF, 0);
      kind_ = 'u';
    }
    producer_ = std::thread([this] { produce(); });
    return true;
  }
  /* next run of decompressed bytes; returns its size, 0 at EOF, -1 on error */
  long next(std::string &out) {
    if (bgzf_) return bgzf_->next(out);
    std::string *b = nullptr;
    if (!ready_.pop(b)) return failed_ ? -1 : 0;
    out.swap(*b);
    free_.push(std::move(b));
    return (long)out.size();
  }
  void close() {
    ready_.close();
    free_.close();
    if (producer_.joinable()) producer_.join();
    bgzf_.reset();
    if (file_) fclose(file_), file_ = nullptr;
    reap();
  }

 private:
  static constexpr size_t BUF = 4u << 20;
  static constexpr int NBUF = 4;
  void reap() {
    if (pid_ > 0) {
      int st = 0;
      waitpid(pid_, &st, 0);
      pid_ = -1;
      if (!(WIFEXITED(st) && WEXITSTATUS(st) == 0)) child_failed_ = true;
    }
  }
  /* fills the NBUF buffers in turn: a buffer goes back on free_ once next() has swapped its bytes out */
  void produce() {
    for (int i = 0; i < NBUF; i++) free_.push(&bufs_[i]);
    std::string *b = nullptr;
    while (free_.pop(b)) {
      b->resize(BUF);
      long n;
      {
        Busy busy(clk_, ST_INFLATE);
        if (kind_ == 'g') {
          n = gz_.read(&(*b)[0], BUF);
        } else {
          const size_t r = fread(&(*b)[0], 1, BUF, file_);
          n = (r == 0 && ferror(file_)) ? -1 : (long)r;
        }
      }
      if (n == 0 && kind_ == 'b') {
        /* a truncated or corrupt .bz2 shows only in the exit status of the child */
        fclose(file_), file_ = nullptr;
        reap();
        if (child_failed_) n = -1;
      }
      if (n <= 0) {
        failed_ = n < 0;
        break;
      }
      b->resize((size_t)n);
      if (!ready_.push(std::move(b))) break;
    }
    ready_.close();
  }

  std::unique_ptr<BgzfReader> bgzf_;
  int bgzf_threads_ = 0;
  StageClock *clk_ = nullptr;
  GzipStream gz_;
  FILE *file_ = nullptr;
  int kind_ = 'u';
  pid_t pid_ = -1;
  bool child_failed_ = false;
  std::thread producer_;
  std::string bufs_[NBUF];
  Channel<std::string *> ready_{NBUF}, free_{NBUF};
  bool failed_ = false; /* set by the producer before it closes ready_ */
};

/* ------------------------------------------------------------------ */
/* records                                                             */

struct Rec {
  size_t hdr_off, seq_off, qual_off; /* into Chunk::text; header = full line incl. '@' / '>'; quality FASTQ only */
  uint32_t hdr_len, seq_len, qual_len;
};

struct Chunk {
  std::string text; /* arena the records point into */
  std::vector<Rec> recs;
  uint64_t bases = 0;
  bool fastq = true;
  bool last = false;
  std::string error;
};

class RecordReader {
 public:
  bool open(const std::string &path, int threads, std::string &err, StageClock *clk) {
    path_ = path;
    clk_ = clk;
    return in_.open(path, threads, err, clk);
  }
  int inflate_threads() const { return in_.inflate_threads(); }
  /* Fills `c`; c.last set at EOF.  With want_records == 0 the reader cuts the chunk itself (records,
   * bases or text bound); otherwise it reads exactly that many records (the second mate file follows
   * the cuts of the first, so mates always sit in the same Work). */
  void next_chunk(Chunk &c, size_t want_records = 0) {
    const auto t_begin = std::chrono::steady_clock::now();
    wait_ns_ = 0;
    struct Account { /* parse time = time in here minus the time spent waiting for inflated bytes */
      RecordReader *r;
      std::chrono::steady_clock::time_point t0;
      ~Account() {
        const uint64_t all = (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count();
        if (r->clk_) r->clk_->ns[ST_PARSE] += all > r->wait_ns_ ? all - r->wait_ns_ : 0;
      }
    } account{this, t_begin};
    c.text.clear();
    c.recs.clear();
    c.bases = 0;
    c.error.clear();
    c.last = false;
    c.text.reserve(24u << 20);
    c.recs.reserve(want_records ? want_records : NH_CHUNK_RECORDS);
    const size_t max_records = want_records ? want_records : NH_CHUNK_RECORDS;
    while (c.recs.size() < max_records) {
      if (format_ == 0) {
        int ch = peek();
        if (ch < 0) {
          c.last = true;
          break;
        }
        if (ch == '@')
          format_ = 'q';
        else if (ch == '>')
          format_ = 'a';
        else {
          c.error = path_ + ": sequence format not recognised (first byte is neither '@' nor '>')";
          c.last = true;
          break;
        }
      }
      c.fastq = format_ == 'q';
      Rec r{};
      if (format_ == 'q' && fast_fastq(c, r)) {
        /* whole record inside the current buffer: taken with four memchr calls */
      } else if (format_ == 'q') {
        std::string *t = &c.text;
        size_t h0 = t->size();
        if (!getline_strip(*t)) {
          c.last = true;
          break;
        }
        r.hdr_off = h0;
        r.hdr_len = (uint32_t)(t->size() - h0);
        if (r.hdr_len == 0) { /* kraken2 stops at an empty header line */
          t->resize(h0);
          c.last = true;
          break;
        }
        if ((*t)[h0] != '@') {
          c.error = path_ + ": malformed FASTQ file (exp. '@', saw \"" + t->substr(h0, 20) + "\")";
          c.last = true;
          break;
        }
        size_t s0 = t->size();
        getline_strip(*t);
        r.seq_off = s0;
        r.seq_len = (uint32_t)(t->size() - s0);
        size_t p0 = t->size();
        getline_strip(*t); /* '+' line: dropped, kraken2 prints a bare '+' */
        t->resize(p0);
        size_t q0 = t->size();
        getline_strip(*t);
        r.qual_off = q0;
        r.qual_len = (uint32_t)(t->size() - q0);
      } else {
        std::string *t = &c.text;
        size_t h0 = t->size();
        if (!getline_strip(*t)) {
          c.last = true;
          break;
        }
        r.hdr_off = h0;
        r.hdr_len = (uint32_t)(t->size() - h0);
        if (r.hdr_len == 0) {
          t->resize(h0);
          c.last = true;
          break;
        }
        if ((*t)[h0] != '>') {
          c.error = path_ + ": malformed FASTA file (exp. '>', saw \"" + t->substr(h0, 20) + "\")";
          c.last = true;
          break;
        }
        size_t s0 = t->size();
        for (;;) { /* sequence lines up to the next '>' or EOF, joined */
          int ch = peek();
          if (ch < 0 || ch == '>') break;
          getline_strip(*t);
        }
        r.seq_off = s0;
        if (t->size() - s0 > 0x7FFFFFFFu) {
          c.error = path_ + ": a sequence longer than 2^31 bases is not supported";
          c.last = true;
          break;
        }
        r.seq_len = (uint32_t)(t->size() - s0);
      }
      c.bases += r.seq_len;
      c.recs.push_back(r);
      if (!want_records && (c.bases >= NH_CHUNK_BASES || c.text.size() >= NH_CHUNK_TEXT)) break;
    }
    if (io_error_) c.error = path_ + ": read error (truncated or corrupt compressed stream?)";
  }

 private:
  bool fill() {
    if (eof_) return false;
    const auto w0 = std::chrono::steady_clock::now();
    long n = in_.next(buf_);
    wait_ns_ += (uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - w0).count();
    if (n < 0) {
      io_error_ = true;
      eof_ = true;
      return false;
    }
    if (n == 0) {
      eof_ = true;
      return false;
    }
    pos_ = 0;
    end_ = (size_t)n;
    return true;
  }
  int peek() {
    if (pos_ >= end_ && !fill()) return -1;
    return (unsigned char)buf_[pos_];
  }
  /* FASTQ fast path: the four lines of the next record lie completely inside buf_ and the header
   * starts with '@'.  Same result as the general path below (trailing whitespace stripped, '+' line
   * dropped); anything unusual - a buffer border, an empty or malformed header - returns false with
   * nothing consumed and the general path decides. */
  bool fast_fastq(Chunk &c, Rec &r) {
    if (pos_ >= end_) return false;
    const char *p = &buf_[pos_], *e = &buf_[0] + end_;
    if (*p != '@') return false;
    const char *l1 = (const char *)memchr(p, '\n', (size_t)(e - p));
    if (!l1) return false;
    const char *l2 = (const char *)memchr(l1 + 1, '\n', (size_t)(e - l1 - 1));
    if (!l2) return false;
    const char *l3 = (const char *)memchr(l2 + 1, '\n', (size_t)(e - l2 - 1));
    if (!l3) return false;
    const char *l4 = (const char *)memchr(l3 + 1, '\n', (size_t)(e - l3 - 1));
    if (!l4) return false;
    auto rstrip = [](const char *b, const char *en) {
      while (en > b && isspace((unsigned char)en[-1])) en--;
      return en;
    };
    const char *he = rstrip(p, l1), *se = rstrip(l1 + 1, l2), *qe = rstrip(l3 + 1, l4);
    if (he == p) return false;
    std::string &t = c.text;
    r.hdr_off = t.size();
    r.hdr_len = (uint32_t)(he - p);
    t.append(p, (size_t)(he - p));
    r.seq_off = t.size();
    r.seq_len = (uint32_t)(se - (l1 + 1));
    t.append(l1 + 1, (size_t)(se - (l1 + 1)));
    r.qual_off = t.size();
    r.qual_len = (uint32_t)(qe - (l3 + 1));
    t.append(l3 + 1, (size_t)(qe - (l3 + 1)));
    pos_ = (size_t)(l4 + 1 - &buf_[0]);
    return true;
  }
  /* appends the next line without its terminator and trailing whitespace; false at EOF with nothing read */
  bool getline_strip(std::string &out) {
    size_t start = out.size();
    bool any = false;
    for (;;) {
      if (pos_ >= end_ && !fill()) break;
      any = true;
      const char *p = &buf_[pos_];
      const char *nl = (const char *)memchr(p, '\n', end_ - pos_);
      if (nl) {
        out.append(p, nl - p);
        pos_ += (size_t)(nl - p) + 1;
        break;
      }
      out.append(p, end_ - pos_);
      pos_ = end_;
    }
    size_t e = out.size();
    while (e > start && isspace((unsigned char)out[e - 1])) e--;
    out.resize(e);
    return any;
  }

  InputStream in_;
  StageClock *clk_ = nullptr;
  uint64_t wait_ns_ = 0;
  std::string path_;
  std::string buf_;
  size_t pos_ = 0, end_ = 0;
  bool eof_ = false, io_error_ = false;
  int format_ = 0;
};

/* ------------------------------------------------------------------ */
/* output: ordered block compression                                    */

typedef size_t (*zstd_bound_fn)(size_t);
typedef unsigned (*zstd_iserror_fn)(size_t);
typedef void *(*zstd_create_fn)(void);
typedef size_t (*zstd_free_fn)(void *);
typedef size_t (*zstd_setparam_fn)(void *, int, int);
typedef size_t (*zstd_compress2_fn)(void *, void *, size_t, const void *, size_t);

/* libzstd has no header in this image: the stable API is bound by hand (zstd.h, v1.4+) */
struct ZstdLib {
  static constexpr int C_COMPRESSION_LEVEL = 100, C_CHECKSUM_FLAG = 201; /* ZSTD_cParameter */
  void *h = nullptr;
  zstd_bound_fn bound = nullptr;
  zstd_iserror_fn is_error = nullptr;
  zstd_create_fn create = nullptr;
  zstd_free_fn free_ctx = nullptr;
  zstd_setparam_fn set_param = nullptr;
  zstd_compress2_fn compress2 = nullptr;
  bool load() {
    if (h) return true;
    h = dlopen("libzstd.so.1", RTLD_NOW);
    if (!h) return false;
    bound = (zstd_bound_fn)dlsym(h, "ZSTD_compressBound");
    is_error = (zstd_iserror_fn)dlsym(h, "ZSTD_isError");
    create = (zstd_create_fn)dlsym(h, "ZSTD_createCCtx");
    free_ctx = (zstd_free_fn)dlsym(h, "ZSTD_freeCCtx");
    set_param = (zstd_setparam_fn)dlsym(h, "ZSTD_CCtx_setParameter");
    compress2 = (zstd_compress2_fn)dlsym(h, "ZSTD_compress2");
    return bound && is_error && create && free_ctx && set_param && compress2;
  }
  /* one frame per block, zstd's default level (3) with the content checksum the reference turns on
   * (src/compression.rs:256-268: Encoder::new(out, 0) + include_checksum(true)) */
  bool frame(const std::string &in, std::string &out) const {
    void *cctx = create();
    if (!cctx) return false;
    bool ok = !is_error(set_param(cctx, C_COMPRESSION_LEVEL, 3)) && !is_error(set_param(cctx, C_CHECKSUM_FLAG, 1));
    if (ok) {
      out.resize(bound(in.size()));
      const size_t n = compress2(cctx, &out[0], out.size(), in.data(), in.size());
      ok = !is_error(n);
      if (ok) out.resize(n);
    }
    free_ctx(cctx);
    return ok;
  }
};

/* gzip output is written as BGZF: a series of gzip members of at most 64 KiB, each announcing its
 * compressed size in a 'BC' extra subfield.  Any gunzip reads it as ordinary multi-member gzip (which
 * is also what gzp writes for the reference, src/compression.rs:214-234); bgzip-aware tools and this
 * library's own reader can inflate the members in parallel. */
static bool bgzf_members(const std::string &in, std::string &out) {
  z_stream zs;
  memset(&zs, 0, sizeof zs);
  /* level 6 = the default level flate2/gzp use in the reference */
  if (deflateInit2(&zs, 6, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) return false;
  out.clear();
  out.reserve(in.size() / 3 + 1024);
  unsigned char buf[65536];
  bool ok = true;
  for (size_t pos = 0; pos < in.size() && ok; pos += BGZF_INPUT) {
    const size_t n = std::min<size_t>(BGZF_INPUT, in.size() - pos);
    deflateReset(&zs);
    zs.next_in = (Bytef *)in.data() + pos;
    zs.avail_in = (uInt)n;
    zs.next_out = buf + 18;
    zs.avail_out = sizeof buf - 18 - 8;
    if (deflate(&zs, Z_FINISH) != Z_STREAM_END) {
      ok = false;
      break;
    }
    const size_t clen = zs.total_out, bsize = 18 + clen + 8;
    memcpy(buf, BGZF_HEADER, 16);
    buf[16] = (unsigned char)((bsize - 1) & 0xff);
    buf[17] = (unsigned char)((bsize - 1) >> 8);
    const uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), (const Bytef *)in.data() + pos, (uInt)n);
    unsigned char *tr = buf + 18 + clen;
    for (int i = 0; i < 4; i++) tr[i] = (unsigned char)(crc >> (8 * i)), tr[4 + i] = (unsigned char)((uint32_t)n >> (8 * i));
    out.append((const char *)buf, bsize);
  }
  deflateEnd(&zs);
  return ok;
}

/* One output file.  Blocks are compressed by a shared pool and written in
 * submission order.  'u': straight write; 'g': gzip members; 'z': zstd frames;
 * 'b' / 'x': piped through bzip2 / xz (their libraries have no headers here). */
class OutputFile {
 public:
  ~OutputFile() { close(); }
  bool open(const std::string &path, int format, int threads, std::string &err) {
    path_ = path;
    format_ = format;
    if (format == 'b' || format == 'x') {
      /* the filter reads its stdin from a socket, not a pipe: send(MSG_NOSIGNAL) turns a filter that
       * died early into an error return instead of a SIGPIPE that would kill the calling process */
      int out = ::open(path.c_str(), O_WRONLY | O_CREAT | O_TRUNC | O_CLOEXEC, 0644);
      int fds[2] = {-1, -1};
      if (out < 0 || socketpair(AF_UNIX, SOCK_STREAM | SOCK_CLOEXEC, 0, fds)) {
        if (out >= 0) ::close(out);
        err = "cannot create " + path;
        return false;
      }
      /* bzip2 level 6 = bzip2::Compression::default() (src/compression.rs:203-212); xz preset 6 with
       * the CLI's default CRC64 check, multi-threaded (src/compression.rs:236-254) */
      std::vector<std::string> av = format == 'b' ? std::vector<std::string>{"bzip2", "-6", "-c"}
                                                  : std::vector<std::string>{"xz", "-c", "-6", "--check=crc64", "-T",
                                                                             std::to_string(threads < 1 ? 1 : threads)};
      const int rc = spawn_filter(av, fds[0], out, &pid_);
      ::close(out);
      ::close(fds[0]);
      if (rc != 0) {
        ::close(fds[1]);
        pid_ = -1;
        err = "cannot run " + av[0];
        return false;
      }
      sock_ = fds[1];
      return true;
    }
    if (format == 'z' && !zstd_.load()) {
      err = "zstd output requested but libzstd.so.1 could not be loaded";
      return false;
    }
    f_ = fopen(path.c_str(), "wb");
    if (!f_) {
      err = "cannot create " + path;
      return false;
    }
    setvbuf(f_, nullptr, _IOFBF, 1u << 20);
    return true;
  }
  bool parallel() const { return format_ == 'g' || format_ == 'z'; }
  bool compress_block(const std::string &in, std::string &out) {
    if (format_ == 'g') return bgzf_members(in, out);
    if (format_ == 'z') return zstd_.frame(in, out);
    return false;
  }
  bool write(const std::string &s) {
    if (s.empty()) return true;
    if (sock_ >= 0) {
      size_t at = 0;
      while (at < s.size()) {
        const ssize_t n = send(sock_, s.data() + at, s.size() - at, MSG_NOSIGNAL);
        if (n < 0) {
          if (errno == EINTR) continue;
          return false; /* EPIPE: the filter is gone */
        }
        at += (size_t)n;
      }
      return true;
    }
    return f_ && fwrite(s.data(), 1, s.size(), f_) == s.size();
  }
  bool close() {
    bool ok = true;
    if (f_ && format_ == 'g') ok = fwrite(BGZF_EOF, 1, sizeof BGZF_EOF, f_) == sizeof BGZF_EOF; /* bgzip's end marker */
    if (f_) ok = (fclose(f_) == 0) && ok, f_ = nullptr;
    if (sock_ >= 0) ::close(sock_), sock_ = -1; /* end of input for the filter */
    if (pid_ > 0) {
      int st = 0;
      waitpid(pid_, &st, 0);
      ok = ok && WIFEXITED(st) && WEXITSTATUS(st) == 0;
      pid_ = -1;
    }
    return ok;
  }
  const std::string &path() const { return path_; }

 private:
  std::string path_;
  int format_ = 'u';
  FILE *f_ = nullptr;
  int sock_ = -1;
  pid_t pid_ = -1;
  ZstdLib zstd_;
};

struct Block {
  int file = 0;
  std::string raw, packed;
  bool ok = true;     /* false when compressing it failed */
  int gpu_rc = NH_OK; /* a GPU deflater's failure and its message */
  std::string gpu_msg;
};

/* Compresses blocks on `threads` host threads, or, given GPUs, on one deflater thread per GPU that takes
 * every waiting block up to GpuDeflater::kBatchBytes at a time; the flusher writes them in order. */
class BlockWriter {
 public:
  BlockWriter(OutputFile *files, int threads, const std::vector<int> &gpus, StageClock *clk) : files_(files), clk_(clk) {
    for (int dev : gpus) workers_.emplace_back([this, dev] { gpu_work(dev); });
    const int n = gpus.empty() ? (threads < 1 ? 1 : threads) : 0;
    for (int i = 0; i < n; i++) workers_.emplace_back([this] { work(); });
    flusher_ = std::thread([this] { flush(); });
  }
  void submit(int file, std::string &&raw) {
    if (raw.empty()) return;
    auto b = std::make_shared<Block>();
    b->file = file;
    b->raw = std::move(raw);
    q_.push(b, files_[file].parallel() ? Queue::QUEUED : Queue::DONE);
  }
  bool finish() {
    q_.close();
    for (auto &t : workers_) t.join();
    flusher_.join();
    return ok_;
  }
  /* the first GPU deflater failure in output order (NH_OK if none) and its message */
  int error(std::string &msg) const {
    msg = err_msg_;
    return err_code_;
  }

 private:
  typedef OrderedQueue<Block> Queue;
  void gpu_work(int device) {
    GpuDeflater gd;
    int rc = gd.open(device);
    std::string msg = rc ? nh_last_error() : "";
    for (;;) {
      std::vector<std::shared_ptr<Block>> batch = q_.take(GpuDeflater::kBatchBytes, [](const Block &b) { return b.raw.size(); });
      if (batch.empty()) return;
      if (rc == NH_OK) {
        Busy busy(clk_, ST_COMPRESS);
        std::vector<GpuDeflater::Span> spans;
        for (auto &b : batch) spans.emplace_back((const uint8_t *)b->raw.data(), b->raw.size());
        std::vector<std::string> packed;
        rc = gd.compress(spans, packed);
        if (rc != NH_OK)
          msg = nh_last_error();
        else
          for (size_t i = 0; i < batch.size(); i++) batch[i]->packed = std::move(packed[i]);
      }
      for (auto &b : batch) {
        if (rc != NH_OK) b->ok = false, b->gpu_rc = rc, b->gpu_msg = msg;
        b->raw.clear();
        b->raw.shrink_to_fit();
      }
      q_.done(batch);
    }
  }
  void work() {
    while (std::shared_ptr<Block> b = q_.take()) {
      {
        Busy busy(clk_, ST_COMPRESS);
        b->ok = files_[b->file].compress_block(b->raw, b->packed);
      }
      b->raw.clear();
      b->raw.shrink_to_fit();
      q_.done(b);
    }
  }
  /* the only thread that writes ok_ and the error, so they need no lock */
  void flush() {
    while (std::shared_ptr<Block> b = q_.pop()) {
      if (!b->ok) ok_ = false;
      if (b->gpu_rc != NH_OK && err_code_ == NH_OK) err_code_ = b->gpu_rc, err_msg_ = b->gpu_msg;
      const std::string &s = files_[b->file].parallel() ? b->packed : b->raw;
      Busy busy(clk_, ST_WRITE);
      if (!files_[b->file].write(s)) ok_ = false;
    }
  }
  OutputFile *files_;
  StageClock *clk_;
  Queue q_{64};
  std::vector<std::thread> workers_;
  std::thread flusher_;
  bool ok_ = true;
  int err_code_ = NH_OK;
  std::string err_msg_;
};

/* ------------------------------------------------------------------ */
/* the pipeline                                                        */

struct Work {
  Chunk c[2];
  uint64_t n_units = 0;
  std::vector<uint32_t> call;
  std::vector<uint8_t> keep;
  std::vector<uint32_t> first_run, run_ext; /* per-sequence hit runs (kraken output only) */
  std::vector<uint16_t> run_len;
  std::string out[2];  /* kept records of this batch, serialised by the classifier thread */
  std::string klines;  /* kraken2 --output lines of this batch */
  uint64_t n_classified = 0, bases = 0;
  std::string error;
};

/* source of classification decisions: the GPU session, or (host-logic tests) fixed arrays */
struct Decider {
  std::vector<nh_db *> dbs; /* one replica per GPU */
  nh_params_t params{};
  const uint8_t *fixed_keep = nullptr;
  const uint32_t *fixed_call = nullptr;
  uint64_t fixed_n = 0;
};

/* A classifier thread's GPU session and the pinned buffers it stages sub-batches in, freed with it. */
struct GpuStaging {
  nh_session *sess = nullptr;
  uint8_t *h_bases = nullptr; /* cap_bases bases */
  uint64_t *h_off = nullptr;  /* offsets of up to max_batch_seqs sequences, and the end */
  uint64_t cap_bases = 0;
  GpuStaging() = default;
  GpuStaging(const GpuStaging &) = delete;
  GpuStaging &operator=(const GpuStaging &) = delete;
  ~GpuStaging() { release(); }
  void release() {
    if (sess) nh_session_destroy(sess), sess = nullptr;
    if (h_bases) nh_host_free(h_bases), h_bases = nullptr;
    if (h_off) nh_host_free(h_off), h_off = nullptr;
    cap_bases = 0;
  }
  /* a session on `db` for sub-batches of up to `bases` bases and `seqs` sequences, made anew only when there
   * is none yet or `bases` is more than the current one holds; "" or the reason it failed */
  std::string fit(nh_db *db, nh_params_t p, uint64_t bases, size_t seqs) {
    if (sess && bases <= cap_bases) return "";
    release();
    if (bases > (1ull << 31)) return "a single read (pair) of more than 2^31 bases is not supported";
    p.max_batch_bases = bases;
    p.max_batch_seqs = seqs;
    h_bases = (uint8_t *)nh_host_alloc(bases);
    h_off = (uint64_t *)nh_host_alloc(seqs * 8);
    if (!h_bases || !h_off || nh_session_create(db, &p, &sess) != NH_OK) {
      const std::string err = std::string("cannot set up a GPU session: ") + nh_last_error();
      release();
      return err;
    }
    cap_bases = bases;
    return "";
  }
};

static void append_record(std::string &out, const Chunk &c, const Rec &r, bool tagged, uint32_t ext) {
  out.append(c.text, r.hdr_off, r.hdr_len);
  if (tagged) {
    char tag[48];
    int n = snprintf(tag, sizeof tag, " kraken:taxid|%u", ext);
    out.append(tag, (size_t)n);
  }
  out.push_back('\n');
  out.append(c.text, r.seq_off, r.seq_len);
  out.push_back('\n');
  if (c.fastq) {
    out.append("+\n", 2);
    out.append(c.text, r.qual_off, r.qual_len);
    out.push_back('\n');
  }
}

static inline bool is_acgt(unsigned char c) {
  c &= 0xDF;
  return c == 'A' || c == 'C' || c == 'G' || c == 'T';
}

/* run-length printer of kraken2's `taxa` vector (classify.cc AddHitlistString) */
struct Hitlist {
  static constexpr int64_t NONE = -1, AMBIG = -2, BORDER = -3;
  std::string &out;
  int64_t last = NONE;
  uint64_t count = 0;
  bool any = false;
  explicit Hitlist(std::string &o) : out(o) {}
  void flush() {
    if (last == NONE) return;
    if (any) out.push_back(' ');
    any = true;
    char buf[48];
    int n;
    if (last == BORDER)
      n = snprintf(buf, sizeof buf, "|:|");
    else if (last == AMBIG)
      n = snprintf(buf, sizeof buf, "A:%llu", (unsigned long long)count);
    else
      n = snprintf(buf, sizeof buf, "%lld:%llu", (long long)last, (unsigned long long)count);
    out.append(buf, (size_t)n);
  }
  void push(int64_t code) {
    if (code == last) {
      count++;
      return;
    }
    flush();
    last = code;
    count = 1;
  }
  void finish() {
    flush();
    if (!any) out.append("0:0");
  }
};

/* one line of kraken2's --output for unit i of w */
static void append_kraken_line(std::string &out, const Work &w, uint64_t i, int nf, int k, int amb_span) {
  out.push_back(w.call[i] ? 'C' : 'U');
  out.push_back('\t');
  {
    const Rec &r = w.c[0].recs[i];
    const char *h = w.c[0].text.data() + r.hdr_off + 1;
    size_t n = 0;
    while (n + 1 < r.hdr_len && !isspace((unsigned char)h[n])) n++;
    if (nf == 2 && n > 2 && h[n - 2] == '/' && (h[n - 1] == '1' || h[n - 1] == '2')) n -= 2; /* TrimPairInfo */
    out.append(h, n);
  }
  char buf[64];
  int n = snprintf(buf, sizeof buf, "\t%u\t", w.call[i]);
  out.append(buf, (size_t)n);
  for (int f = 0; f < nf; f++) {
    n = snprintf(buf, sizeof buf, f ? "|%u" : "%u", w.c[f].recs[i].seq_len);
    out.append(buf, (size_t)n);
  }
  out.push_back('\t');
  Hitlist hl(out);
  for (int f = 0; f < nf; f++) {
    const Rec &r = w.c[f].recs[i];
    const unsigned char *s = (const unsigned char *)w.c[f].text.data() + r.seq_off;
    const uint64_t seq = i * nf + f;
    uint32_t ri = w.first_run[seq];
    const uint32_t rend = w.first_run[seq + 1];
    uint32_t left = ri < rend ? w.run_len[ri] : 0;
    uint32_t c_run = 0;
    for (uint32_t b = 0; b < r.seq_len; b++) {
      c_run = is_acgt(s[b]) ? c_run + 1 : 0;
      if (b + 1 < (uint32_t)k) continue;
      if (c_run >= (uint32_t)amb_span && ri < rend) {
        hl.push((int64_t)w.run_ext[ri]);
        if (--left == 0 && ++ri < rend) left = w.run_len[ri];
      } else {
        hl.push(Hitlist::AMBIG);
      }
    }
    if (nf == 2 && f == 0) hl.push(Hitlist::BORDER);
  }
  hl.finish();
  out.push_back('\n');
}

}  // namespace

/* kraken2 report (reports.cc ReportKrakenStyle): percentage, clade count, direct count, rank code, taxid, indented name */
bool write_report(FILE *f, const nh_db *db, const std::vector<uint64_t> &call_counts, uint64_t total, uint64_t unclassified,
                  bool zero_counts) {
  const size_t n = db->h_parent.size();
  std::vector<uint64_t> clade(call_counts);
  for (size_t i = n; i-- > 2;) clade[db->h_parent[i]] += clade[i]; /* parent id < child id */
  std::vector<std::vector<uint32_t>> kids(n);
  for (size_t i = 2; i < n; i++) kids[db->h_parent[i]].push_back((uint32_t)i);
  auto line = [&](uint64_t cl, uint64_t direct, const std::string &rank, uint64_t taxid, const std::string &name, int depth) {
    fprintf(f, "%6.2f\t%llu\t%llu\t%s\t%llu\t%*s%s\n", total ? 100.0 * (double)cl / (double)total : 0.0,
            (unsigned long long)cl, (unsigned long long)direct, rank.c_str(), (unsigned long long)taxid, 2 * depth, "",
            name.c_str());
  };
  if (unclassified || zero_counts) line(unclassified, unclassified, "U", 0, "unclassified", 0);
  struct Frame {
    uint32_t id;
    char code;
    int rank_depth, depth;
  };
  std::vector<Frame> stack;
  if (n > 1) stack.push_back({1, 'R', -1, 0});
  while (!stack.empty()) {
    Frame fr = stack.back();
    stack.pop_back();
    if (clade[fr.id] == 0 && !zero_counts) continue;
    const std::string &rank = db->h_rank[fr.id];
    static const std::pair<const char *, char> codes[] = {{"superkingdom", 'D'}, {"kingdom", 'K'}, {"phylum", 'P'}, {"class", 'C'},
                                                          {"order", 'O'},        {"family", 'F'},  {"genus", 'G'},  {"species", 'S'}};
    bool named = false;
    for (auto &c : codes)
      if (rank == c.first) {
        fr.code = c.second;
        fr.rank_depth = 0;
        named = true;
      }
    if (!named) fr.rank_depth++;
    std::string rs(1, fr.code);
    if (fr.rank_depth != 0) rs += std::to_string(fr.rank_depth);
    line(clade[fr.id], call_counts[fr.id], rs, db->h_ext[fr.id], db->h_name[fr.id], fr.depth);
    std::vector<uint32_t> ch = kids[fr.id];
    std::stable_sort(ch.begin(), ch.end(), [&](uint32_t a, uint32_t b) { return clade[a] > clade[b]; });
    for (auto it = ch.rbegin(); it != ch.rend(); ++it) stack.push_back({*it, fr.code, fr.rank_depth, fr.depth + 1});
  }
  return !ferror(f);
}

namespace {

static int run_pipeline(const Decider &dec, const nh_files_t *files, nh_run_stats_t *stats) {
  const auto t0 = std::chrono::steady_clock::now();
  const bool paired = files->in2 != nullptr;
  const int nf = paired ? 2 : 1;
  if (!files->in1 || !files->out1 || (paired && !files->out2))
    return nh_set_error(NH_ERR_INVALID, "nh_run_files: in1/out1 (and out2 for paired input) are required");
  const bool want_lines = files->kraken_output && strcmp(files->kraken_output, "/dev/null") != 0;
  const bool want_report = files->kraken_report != nullptr;
  if ((want_lines || want_report) && dec.dbs.empty())
    return nh_set_error(NH_ERR_UNSUPPORTED, "kraken output / report need the database (not available to the rewrite hook)");
  int fmt = files->out_format ? files->out_format : 'u';
  if (!strchr("ugbxz", fmt)) return nh_set_error(NH_ERR_INVALID, "unknown output format '%c'", fmt);
  FILE *kout = nullptr;
  struct Closer { /* every early return below closes the per-read output */
    FILE *&f;
    ~Closer() {
      if (f) fclose(f);
    }
  } kout_closer{kout};
  if (want_lines) {
    kout = fopen(files->kraken_output, "w");
    if (!kout) return nh_set_error(NH_ERR_IO, "cannot create %s", files->kraken_output);
    setvbuf(kout, nullptr, _IOFBF, 1u << 20);
  }
  std::unordered_map<uint32_t, uint32_t> ext_to_internal;
  std::vector<uint64_t> call_counts;
  if (want_report) {
    const nh_db *d0 = dec.dbs[0];
    call_counts.assign(d0->h_ext.size(), 0);
    for (size_t i = 1; i < d0->h_ext.size(); i++) ext_to_internal[d0->h_ext[i]] = (uint32_t)i;
  }
  const int db_k = dec.dbs.empty() ? 0 : (int)dec.dbs[0]->info.k;
  const int db_amb_span = dec.dbs.empty() ? 0 : dec.dbs[0]->params.amb_span;
  const int threads = dec.params.threads < 1 ? 1 : dec.params.threads;

  std::string err;
  StageClock clock;
  RecordReader readers[2];
  /* inflate threads per input file (only blocked gzip can use more than one) */
  const int in_threads = std::max(1, std::min(8, threads / nf));
  if (!readers[0].open(files->in1, in_threads, err, &clock) || (paired && !readers[1].open(files->in2, in_threads, err, &clock)))
    return nh_set_error(NH_ERR_IO, "%s", err.c_str());
  OutputFile outs[2];
  /* like src/main.rs:342-346: one output gets all the threads, two share them */
  const int per_file_threads = paired ? (threads / 2 < 1 ? 1 : threads / 2) : threads;
  if (!outs[0].open(files->out1, fmt, per_file_threads, err) ||
      (paired && !outs[1].open(files->out2, fmt, per_file_threads, err)))
    return nh_set_error(NH_ERR_IO, "%s", err.c_str());

  /* readers */
  Channel<std::unique_ptr<Chunk>> chunks[2] = {Channel<std::unique_ptr<Chunk>>(3), Channel<std::unique_ptr<Chunk>>(3)};
  std::vector<std::thread> reader_threads;
  /* the first file's reader decides where chunks end; the second mate file reads the same number of
   * records, so a pair never straddles two Works whatever the read lengths are */
  struct Cut {
    size_t records;
    bool last;
  };
  Channel<Cut> cuts(64);
  for (int f = 0; f < nf; f++)
    reader_threads.emplace_back([&, f] {
      for (;;) {
        auto c = std::make_unique<Chunk>();
        if (f == 0) {
          readers[0].next_chunk(*c);
          if (paired && !cuts.push(Cut{c->recs.size(), c->last})) c->last = true;
        } else {
          Cut cut{0, true};
          if (!cuts.pop(cut)) cut = Cut{0, true};
          if (cut.records)
            readers[1].next_chunk(*c, cut.records);
          else
            c->fastq = true;
          if (cut.last) c->last = true; /* nothing of this file is needed beyond the end of the first */
        }
        bool last = c->last;
        if (!chunks[f].push(std::move(c)) || last) break;
      }
      chunks[f].close();
      if (f == 0) cuts.close();
    });

  /* classifiers: a Work enters `handoff` when it is taken and leaves to the writer in that order.
   * Back-pressure: the GPU outruns the output compressor by orders of magnitude, so batches are only
   * handed out while fewer than NH_MAX_AHEAD are inside. */
  constexpr size_t NH_MAX_AHEAD = 8;
  typedef OrderedQueue<Work> Handoff;
  Handoff handoff(NH_MAX_AHEAD);
  std::mutex pair_m; /* both files' chunks and the Work's place in `handoff` are taken as one step */
  bool input_done = false;

  auto take = [&]() -> std::shared_ptr<Work> {
    std::lock_guard<std::mutex> lk(pair_m);
    if (input_done) return nullptr;
    /* the Work enters before its chunks leave the readers' channels, so that a full window holds the
     * chunks back in the channels; it enters empty if there turn out to be none */
    auto w = std::make_shared<Work>();
    if (!handoff.push(w, Handoff::CLAIMED)) return nullptr;
    std::unique_ptr<Chunk> c[2];
    for (int f = 0; f < nf; f++)
      if (!chunks[f].pop(c[f])) {
        input_done = true;
        handoff.done(w);
        return nullptr;
      }
    for (int f = 0; f < nf; f++) {
      w->c[f] = std::move(*c[f]);
      if (!w->c[f].error.empty()) w->error = w->c[f].error;
      if (w->c[f].last) input_done = true;
    }
    w->n_units = w->c[0].recs.size();
    if (paired && w->c[1].recs.size() != w->n_units) {
      /* kraken2 stops at the end of the shorter file */
      if (w->c[1].recs.size() < w->n_units) w->n_units = w->c[1].recs.size();
      input_done = true;
    }
    if (input_done) {
      for (int f = 0; f < nf; f++) chunks[f].close();
      cuts.close();
    }
    return w;
  };

  /* at least two classifier threads per GPU, so that one batch's copies overlap the other's kernel;
   * up to four when -t allows it, because the same threads re-serialise the kept records */
  const int per_gpu = std::max(2, std::min(4, threads / 4));
  const int n_classifiers = dec.fixed_keep ? 1 : per_gpu * (int)dec.dbs.size();
  std::atomic<int> running_classifiers{n_classifiers};
  nh_params_t sess_params = dec.params;
  sess_params.emit_runs = want_lines ? 1 : 0;
  uint64_t fixed_cursor = 0;
  std::vector<std::thread> classifier_threads;
  for (int ci = 0; ci < n_classifiers; ci++)
    classifier_threads.emplace_back([&, ci] {
      GpuStaging gpu;
      while (std::shared_ptr<Work> w = take()) {
        if (w->error.empty() && w->n_units) {
          const uint64_t n_seqs = w->n_units * nf;
          uint64_t total = 0;
          for (int f = 0; f < nf; f++)
            for (uint64_t i = 0; i < w->n_units; i++) total += w->c[f].recs[i].seq_len;
          w->call.assign(w->n_units, 0);
          w->keep.assign(w->n_units, 0);
          if (dec.fixed_keep) {
            if (fixed_cursor + w->n_units > dec.fixed_n) {
              w->error = "fewer decisions than records";
            } else {
              memcpy(w->keep.data(), dec.fixed_keep + fixed_cursor, w->n_units);
              memcpy(w->call.data(), dec.fixed_call + fixed_cursor, w->n_units * 4);
              fixed_cursor += w->n_units;
            }
          } else {
            /* A Work goes to the GPU in sub-batches of at most cap_bases bases: the session keeps one
             * size whatever the read lengths are (ultra-long ONT, FASTA contigs) and only grows when a
             * single unit is longer than it. */
            uint64_t longest = 0;
            for (uint64_t i = 0; i < w->n_units; i++) {
              uint64_t ub = 0;
              for (int f = 0; f < nf; f++) ub += w->c[f].recs[i].seq_len;
              longest = std::max(longest, ub);
            }
            w->error = gpu.fit(dec.dbs[(size_t)ci % dec.dbs.size()], sess_params,
                               std::max<uint64_t>(NH_BATCH_BASES, longest + 64), (size_t)NH_CHUNK_RECORDS * nf + 2);
            if (want_lines && w->error.empty()) {
              w->first_run.assign(n_seqs + 1, 0);
              w->run_ext.resize(total + 1);
              w->run_len.resize(total + 1);
            }
            uint64_t u0 = 0, runs_at = 0;
            while (w->error.empty() && u0 < w->n_units) {
              uint64_t o = 0, s = 0, u1 = u0;
              {
              Busy staging(&clock, ST_STAGE);
              for (; u1 < w->n_units; u1++) {
                uint64_t ub = 0;
                for (int f = 0; f < nf; f++) ub += w->c[f].recs[u1].seq_len;
                if (u1 > u0 && o + ub + 64 > gpu.cap_bases) break;
                for (int f = 0; f < nf; f++) { /* mates interleaved: sequences 2i, 2i+1 */
                  const Rec &r = w->c[f].recs[u1];
                  gpu.h_off[s++] = o;
                  memcpy(gpu.h_bases + o, w->c[f].text.data() + r.seq_off, r.seq_len);
                  o += r.seq_len;
                }
              }
              gpu.h_off[s] = o;
              }
              Busy classifying(&clock, ST_CLASSIFY);
              if (nh_classify_batch(gpu.sess, gpu.h_bases, gpu.h_off, s, w->call.data() + u0, w->keep.data() + u0, nullptr) != NH_OK)
                w->error = std::string("classification failed: ") + nh_last_error();
              if (want_lines && w->error.empty()) {
                uint64_t nr = 0;
                uint32_t *fr = w->first_run.data() + u0 * nf;
                if (nh_last_batch_runs(gpu.sess, s, fr, w->run_ext.data() + runs_at, w->run_len.data() + runs_at,
                                       total + 1 - runs_at, &nr) != NH_OK)
                  w->error = std::string("reading the hit runs failed: ") + nh_last_error();
                else {
                  for (uint64_t j = 0; j <= s; j++) fr[j] += (uint32_t)runs_at; /* fr[s] is the next sub-batch's first entry */
                  runs_at += nr;
                }
              }
              u0 = u1;
            }
          }
        }
        if (w->error.empty() && w->n_units) {
          Busy serialising(&clock, ST_SERIALISE);
          /* serialise here, in parallel across batches; the writer only restores the order */
          if (want_lines) {
            w->klines.reserve(w->n_units * 96);
            for (uint64_t i = 0; i < w->n_units; i++) append_kraken_line(w->klines, *w, i, nf, db_k, db_amb_span);
          }
          for (int f = 0; f < nf; f++) {
            uint64_t kept_bytes = 0;
            for (uint64_t i = 0; i < w->n_units; i++) {
              const Rec &r = w->c[f].recs[i];
              w->bases += r.seq_len;
              if (w->keep[i]) kept_bytes += r.hdr_len + 2ull * r.seq_len + 32;
            }
            w->out[f].reserve(kept_bytes);
          }
          for (uint64_t i = 0; i < w->n_units; i++) {
            const bool classified = w->call[i] != 0;
            w->n_classified += classified;
            if (!w->keep[i]) continue;
            for (int f = 0; f < nf; f++)
              append_record(w->out[f], w->c[f], w->c[f].recs[i], classified && files->tag_classified, w->call[i]);
          }
          for (int f = 0; f < nf; f++) { /* the text arena is no longer needed */
            std::string().swap(w->c[f].text);
            if (!want_report) std::vector<Rec>().swap(w->c[f].recs);
          }
        }
        handoff.done(w);
      }
      if (--running_classifiers == 0) handoff.close(); /* no Work will enter any more */
    });

  /* writer (this thread): batches in input order; gzip output is deflated on the sessions' GPUs on request */
  std::vector<int> deflate_gpus;
  if (dec.params.gpu_gzip && fmt == 'g')
    for (const nh_db *db : dec.dbs)
      if (std::find(deflate_gpus.begin(), deflate_gpus.end(), db->info.device) == deflate_gpus.end())
        deflate_gpus.push_back(db->info.device);
  BlockWriter bw(outs, threads, deflate_gpus, &clock);
  uint64_t total_units = 0, n_classified = 0, total_bases = 0;
  bool failed = false;
  std::string fail_msg;
  std::string pend[2];
  while (std::shared_ptr<Work> w = handoff.pop()) {
    if (!w->error.empty()) {
      if (!failed) fail_msg = w->error;
      failed = true;
    }
    if (failed) continue; /* drain */
    if (kout && fwrite(w->klines.data(), 1, w->klines.size(), kout) != w->klines.size()) {
      failed = true;
      fail_msg = std::string("writing ") + files->kraken_output + " failed";
    }
    if (want_report)
      for (uint64_t i = 0; i < w->n_units; i++)
        if (w->call[i]) call_counts[ext_to_internal[w->call[i]]]++;
    n_classified += w->n_classified;
    total_units += w->n_units;
    total_bases += w->bases;
    for (int f = 0; f < nf; f++) {
      /* cut into compression blocks; a few bytes of one batch may ride along with the next */
      const std::string &o = w->out[f];
      size_t pos = 0;
      while (pos < o.size()) {
        const size_t take_n = std::min(o.size() - pos, NH_OUT_BLOCK - pend[f].size());
        pend[f].append(o, pos, take_n);
        pos += take_n;
        if (pend[f].size() >= NH_OUT_BLOCK) {
          bw.submit(f, std::move(pend[f]));
          pend[f].clear();
        }
      }
    }
  }
  for (int f = 0; f < nf; f++) bw.submit(f, std::move(pend[f]));
  for (int f = 0; f < nf; f++) chunks[f].close();
  cuts.close();
  for (auto &t : classifier_threads) t.join();
  for (auto &t : reader_threads) t.join();
  bool wrote = bw.finish();
  for (int f = 0; f < nf; f++) wrote = outs[f].close() && wrote;
  if (kout) {
    const bool closed_ok = fclose(kout) == 0;
    kout = nullptr;
    if (!closed_ok && !failed) {
      failed = true;
      fail_msg = std::string("writing ") + files->kraken_output + " failed";
    }
  }
  if (want_report && !failed) {
    FILE *rf = fopen(files->kraken_report, "w");
    bool ok = rf && write_report(rf, dec.dbs[0], call_counts, total_units, total_units - n_classified, false);
    if (rf) ok = fclose(rf) == 0 && ok;
    if (!ok) {
      failed = true;
      fail_msg = std::string("writing ") + files->kraken_report + " failed";
    }
  }
  if (failed) return nh_set_error(NH_ERR_IO, "%s", fail_msg.c_str());
  std::string deflate_msg;
  if (const int rc = bw.error(deflate_msg)) return nh_set_error(rc, "%s", deflate_msg.c_str());
  if (!wrote) return nh_set_error(NH_ERR_IO, "writing %s failed", outs[0].path().c_str());
  if (stats) {
    stats->total = total_units;
    stats->classified = n_classified;
    stats->unclassified = total_units - n_classified;
    stats->bases = total_bases;
    stats->seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    stats->busy_inflate_s = 1e-9 * (double)clock.ns[ST_INFLATE];
    stats->busy_parse_s = 1e-9 * (double)clock.ns[ST_PARSE];
    stats->busy_stage_s = 1e-9 * (double)clock.ns[ST_STAGE];
    stats->busy_classify_s = 1e-9 * (double)clock.ns[ST_CLASSIFY];
    stats->busy_serialise_s = 1e-9 * (double)clock.ns[ST_SERIALISE];
    stats->busy_compress_s = 1e-9 * (double)clock.ns[ST_COMPRESS];
    stats->busy_write_s = 1e-9 * (double)clock.ns[ST_WRITE];
    stats->threads_inflate = readers[0].inflate_threads() + (paired ? readers[1].inflate_threads() : 0);
    stats->threads_compress = !outs[0].parallel() ? 0 : deflate_gpus.empty() ? threads : (int)deflate_gpus.size();
  }
  return NH_OK;
}

}  // namespace

extern "C" int nh_run_files(nh_session *s, const nh_files_t *files, nh_run_stats_t *stats) {
  if (!s || !files) return nh_set_error(NH_ERR_INVALID, "null argument");
  Decider d;
  d.dbs.push_back(s->db);
  d.params = s->params;
  d.params.paired = files->in2 != nullptr;
  return run_pipeline(d, files, stats);
}

extern "C" int nh_run_files_multi(nh_session *const *sessions, int n_sessions, const nh_files_t *files,
                                  nh_run_stats_t *stats) {
  if (!sessions || n_sessions < 1 || !files) return nh_set_error(NH_ERR_INVALID, "bad argument");
  Decider d;
  for (int i = 0; i < n_sessions; i++) {
    if (!sessions[i]) return nh_set_error(NH_ERR_INVALID, "null session");
    d.dbs.push_back(sessions[i]->db);
  }
  d.params = sessions[0]->params;
  d.params.paired = files->in2 != nullptr;
  return run_pipeline(d, files, stats);
}

/* Host-logic test hook: the same reader -> writer -> compressor pipeline with
 * the per-unit decisions supplied by the caller instead of the GPU. */
extern "C" int nh_debug_rewrite_files(const nh_files_t *files, const uint8_t *keep, const uint32_t *call_ext,
                                      uint64_t n_units, int threads, nh_run_stats_t *stats) {
  if (!files || !keep || !call_ext) return nh_set_error(NH_ERR_INVALID, "null argument");
  Decider d;
  d.params.threads = threads;
  d.params.paired = files->in2 != nullptr;
  d.fixed_keep = keep;
  d.fixed_call = call_ext;
  d.fixed_n = n_units;
  return run_pipeline(d, files, stats);
}

/* ------------------------------------------------------------------ */
/* NhSeqReader: the reader above, a record at a time (nh_build.cu)     */

struct NhSeqReader::Impl {
  RecordReader reader;
  Chunk chunk;
  size_t next = 0;
};

NhSeqReader::NhSeqReader() : impl_(new Impl()) {}
NhSeqReader::~NhSeqReader() { delete impl_; }

int NhSeqReader::open(const char *path, int threads) {
  std::string err;
  if (!impl_->reader.open(path, threads < 1 ? 1 : threads, err, nullptr)) return nh_set_error(NH_ERR_IO, "%s", err.c_str());
  return NH_OK;
}

int NhSeqReader::next(const char **hdr, size_t *hdr_len, const char **seq, size_t *seq_len) {
  Impl &m = *impl_;
  while (m.next >= m.chunk.recs.size()) {
    if (m.chunk.last) return 0;
    m.reader.next_chunk(m.chunk);
    m.next = 0;
    if (!m.chunk.error.empty()) {
      m.chunk.recs.clear();
      m.chunk.last = true;
      return nh_set_error(NH_ERR_IO, "%s", m.chunk.error.c_str());
    }
  }
  const Rec &r = m.chunk.recs[m.next++];
  *hdr = m.chunk.text.data() + r.hdr_off;
  *hdr_len = r.hdr_len;
  *seq = m.chunk.text.data() + r.seq_off;
  *seq_len = r.seq_len;
  return 1;
}
