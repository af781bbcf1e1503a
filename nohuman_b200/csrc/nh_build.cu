/*
 * nh_build.cu — kraken2-build --build on the GPU (include/nohuman_gpu.h: nh_build_taxonomy, nh_build_db).
 *
 *   taxonomy   host: nodes.dmp / names.dmp / seqid2taxid.map -> taxo.k2d image (taxonomy.cc's layout,
 *              SURVEY.md Appendix B) and the internal taxon of every sequence ID
 *   estimate   only without a given capacity: every library minimizer whose hash falls in 4 of 1024 ranges
 *              goes into an exact device set (k_estimate_tiles); capacity from its size (kraken2's
 *              estimate_capacity + build_kraken2_db.sh, as recalled: see estimate_capacity below)
 *   insert     records cut into batches of pieces overlapping by k-1 bases, each piece with its taxon;
 *              plan -> warp-per-tile minimizers -> k_insert_tiles (nh_insert.cuh), the host reading and
 *              parsing the next batch into the other pinned buffer while the GPU works
 *   write      cells copied back in pieces, hash.k2d / opts.k2d / taxo.k2d written as *.tmp, then renamed
 *
 * The cell layout depends on the order in which concurrent inserts meet, so it is not byte-reproducible
 * between runs; every lookup is (see nh_build_db in the header).
 */
#include <cuda_runtime.h>
#include <ctype.h>
#include <errno.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <memory>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/nohuman_gpu.h"
#include "nh_insert.cuh"
#include "nh_internal.h"
#include "nh_kernels.cuh"

/* ------------------------------------------------------------------ */
/* taxonomy (host)                                                     */

namespace {

struct LineFile {
  FILE *f = nullptr;
  char *buf = nullptr;
  size_t cap = 0;
  uint64_t line = 0;
  std::string path;
  ~LineFile() {
    free(buf);
    if (f) fclose(f);
  }
  int open(const char *p) {
    path = p ? p : "";
    f = p ? fopen(p, "rb") : nullptr;
    return f ? NH_OK : nh_set_error(NH_ERR_IO, "cannot open %s", path.c_str());
  }
  /* the next line without its terminator; false at the end */
  bool next(std::string &out) {
    const ssize_t n = getline(&buf, &cap, f);
    if (n < 0) return false;
    line++;
    size_t e = (size_t)n;
    while (e && (buf[e - 1] == '\n' || buf[e - 1] == '\r')) e--;
    out.assign(buf, e);
    return true;
  }
  int bad(const char *what) const {
    return nh_set_error(NH_ERR_IO, "%s:%llu: %s", path.c_str(), (unsigned long long)line, what);
  }
};

std::string trim(const std::string &s, size_t b, size_t e) {
  while (b < e && (s[b] == ' ' || s[b] == '\t')) b++;
  while (e > b && (s[e - 1] == ' ' || s[e - 1] == '\t')) e--;
  return s.substr(b, e - b);
}

/* NCBI dump line "f0\t|\tf1\t|\t...\t|": the fields between the bars, trimmed */
bool dmp_fields(const std::string &s, std::vector<std::string> &out) {
  out.clear();
  size_t b = 0;
  for (;;) {
    const size_t bar = s.find('|', b);
    if (bar == std::string::npos) {
      if (!trim(s, b, s.size()).empty()) out.push_back(trim(s, b, s.size()));
      break;
    }
    out.push_back(trim(s, b, bar));
    b = bar + 1;
  }
  return !out.empty() && s.find('|') != std::string::npos;
}

bool parse_u64(const std::string &s, uint64_t &v) {
  if (s.empty() || s.size() > 19) return false;
  v = 0;
  for (char c : s) {
    if (c < '0' || c > '9') return false;
    v = v * 10 + (uint64_t)(c - '0');
  }
  return true;
}

struct TaxNodeIn {
  uint64_t parent;
  std::string rank;
  uint64_t line; /* in nodes.dmp */
  int state = 0; /* 0: not visited, 1: on the walk being checked, 2: marked (reaches taxid 1) */
};

struct Taxonomy {
  std::vector<uint8_t> image;                       /* taxo.k2d */
  std::unordered_map<std::string, uint32_t> seq_taxon; /* sequence ID -> internal taxon */
  uint64_t node_count = 0;
};

void put_u64(std::vector<uint8_t> &v, size_t at, uint64_t x) { memcpy(v.data() + at, &x, 8); }

int load_taxonomy(const char *nodes_dmp, const char *names_dmp, const char *seqid2taxid, Taxonomy &T) {
  std::unordered_map<uint64_t, TaxNodeIn> nodes;
  std::vector<std::string> fld;
  std::string s;
  {
    LineFile lf;
    if (int rc = lf.open(nodes_dmp)) return rc;
    while (lf.next(s)) {
      if (s.empty()) continue;
      uint64_t id, parent;
      if (!dmp_fields(s, fld) || fld.size() < 3 || !parse_u64(fld[0], id) || !parse_u64(fld[1], parent))
        return lf.bad("malformed nodes.dmp line (expected taxid | parent | rank | ...)");
      TaxNodeIn &n = nodes[id];
      if (n.line) return lf.bad("taxid listed twice");
      n.parent = parent;
      n.rank = fld[2];
      n.line = lf.line;
    }
  }
  /* seqid2taxid: every assigned taxid and its ancestors are marked */
  {
    LineFile lf;
    if (int rc = lf.open(seqid2taxid)) return rc;
    std::vector<TaxNodeIn *> walk;
    while (lf.next(s)) {
      size_t a = 0;
      while (a < s.size() && isspace((unsigned char)s[a])) a++;
      if (a == s.size()) continue;
      size_t b = a;
      while (b < s.size() && !isspace((unsigned char)s[b])) b++;
      const std::string seqid = s.substr(a, b - a);
      const std::string tax = trim(s, b, s.size());
      uint64_t id;
      if (!parse_u64(tax, id)) return lf.bad("malformed seqid2taxid line (expected <sequence ID> <taxid>)");
      auto it = nodes.find(id);
      if (it == nodes.end()) {
        char m[96];
        snprintf(m, sizeof m, "taxid %llu is not in nodes.dmp", (unsigned long long)id);
        return lf.bad(m);
      }
      T.seq_taxon.emplace(seqid, (uint32_t)id); /* external id for now; the first entry of an ID wins */
      walk.clear();
      uint64_t cur = id;
      for (;;) {
        TaxNodeIn &n = nodes[cur];
        if (n.state == 2) break;
        if (n.state == 1)
          return nh_set_error(NH_ERR_IO, "%s:%llu: taxid %llu is on a parent cycle", nodes_dmp,
                              (unsigned long long)n.line, (unsigned long long)cur);
        n.state = 1;
        walk.push_back(&n);
        if (cur == 1) break;
        auto p = nodes.find(n.parent);
        if (n.parent == cur || p == nodes.end())
          return nh_set_error(NH_ERR_IO, "%s:%llu: taxid %llu does not reach taxid 1 (parent %llu %s)", nodes_dmp,
                              (unsigned long long)n.line, (unsigned long long)cur, (unsigned long long)n.parent,
                              n.parent == cur ? "is itself" : "is not in nodes.dmp");
        cur = n.parent;
      }
      for (TaxNodeIn *n : walk) n->state = 2;
    }
  }
  /* breadth-first numbering from taxid 1 over the marked nodes, children in ascending taxid */
  std::unordered_map<uint64_t, std::vector<uint64_t>> children;
  for (auto &kv : nodes)
    if (kv.second.state == 2 && kv.first != 1) children[kv.second.parent].push_back(kv.first);
  for (auto &kv : children) std::sort(kv.second.begin(), kv.second.end());
  std::vector<uint64_t> order;
  std::unordered_map<uint64_t, uint32_t> internal;
  if (nodes.count(1) && nodes[1].state == 2) {
    order.push_back(1);
    internal[1] = 1;
  }
  for (size_t i = 0; i < order.size(); i++) {
    auto c = children.find(order[i]);
    if (c == children.end()) continue;
    for (uint64_t ch : c->second) {
      internal[ch] = (uint32_t)(order.size() + 1);
      order.push_back(ch);
    }
  }
  /* names: the scientific names of the marked nodes */
  std::unordered_map<uint64_t, std::string> names;
  {
    LineFile lf;
    if (int rc = lf.open(names_dmp)) return rc;
    while (lf.next(s)) {
      if (s.empty()) continue;
      uint64_t id;
      if (!dmp_fields(s, fld) || fld.size() < 4 || !parse_u64(fld[0], id))
        return lf.bad("malformed names.dmp line (expected taxid | name | unique name | name class | ...)");
      if (fld[3] == "scientific name" && internal.count(id)) names.emplace(id, fld[1]);
    }
  }
  /* the image: header, node 0 zeroed, one 56-byte TaxonomyNode per marked node, names, ranks */
  const uint64_t n = order.size() + 1;
  std::string name_data, rank_data;
  std::vector<uint8_t> &img = T.image;
  img.assign(32 + n * 56, 0);
  memcpy(img.data(), "K2TAXDAT", 8);
  for (size_t i = 0; i < order.size(); i++) {
    const uint64_t ext = order[i], id = i + 1;
    const TaxNodeIn &nd = nodes[ext];
    const size_t at = 32 + id * 56;
    auto c = children.find(ext);
    const uint64_t nch = c == children.end() ? 0 : c->second.size();
    put_u64(img, at + 0, ext == 1 ? 0 : internal[nd.parent]);
    put_u64(img, at + 8, nch ? internal[c->second[0]] : 0);
    put_u64(img, at + 16, nch);
    put_u64(img, at + 24, name_data.size());
    put_u64(img, at + 32, rank_data.size());
    put_u64(img, at + 40, ext);
    auto nm = names.find(ext);
    if (nm != names.end()) name_data += nm->second;
    name_data.push_back('\0');
    rank_data += nd.rank;
    rank_data.push_back('\0');
  }
  put_u64(img, 8, n);
  put_u64(img, 16, name_data.size());
  put_u64(img, 24, rank_data.size());
  img.insert(img.end(), name_data.begin(), name_data.end());
  img.insert(img.end(), rank_data.begin(), rank_data.end());
  for (auto &kv : T.seq_taxon) kv.second = internal[kv.second];
  T.node_count = n;
  return NH_OK;
}

int write_file(const std::string &path, const void *data, size_t n) {
  FILE *f = fopen(path.c_str(), "wb");
  if (!f) return nh_set_error(NH_ERR_IO, "cannot create %s: %s", path.c_str(), strerror(errno));
  const bool ok = fwrite(data, 1, n, f) == n;
  if (fclose(f) != 0 || !ok) return nh_set_error(NH_ERR_IO, "writing %s failed", path.c_str());
  return NH_OK;
}

}  // namespace

extern "C" int nh_build_taxonomy(const char *nodes_dmp, const char *names_dmp, const char *seqid2taxid,
                                 const char *out_taxo_k2d, uint64_t *node_count) {
  if (!nodes_dmp || !names_dmp || !seqid2taxid || !out_taxo_k2d) return nh_set_error(NH_ERR_INVALID, "null argument");
  Taxonomy T;
  int rc = load_taxonomy(nodes_dmp, names_dmp, seqid2taxid, T);
  if (!rc) rc = write_file(out_taxo_k2d, T.image.data(), T.image.size());
  if (!rc && node_count) *node_count = T.node_count;
  return rc;
}

/* ------------------------------------------------------------------ */
/* pass 1: capacity estimate                                           */

#define CUDA_TRY(expr)                                                                       \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess)                                                                   \
      return nh_set_error(NH_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                          __FILE__, __LINE__);                                               \
  } while (0)

constexpr uint64_t EST_EMPTY = ~0ull; /* its low bits (1023) are never sampled */
constexpr uint32_t EST_RANGES = 1024, EST_SAMPLED = 4;

/* counters: [0] keys in the set, [1] set when a claim passed `limit` or a walk found no empty slot */
__global__ void __launch_bounds__(NH_BLOCK_THREADS)
k_estimate_tiles(const NhBatchPtrs b, unsigned long long *set, uint64_t mask, unsigned long long limit,
                 unsigned long long *counters) {
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t n_tiles = b.counters->n_tiles;
  for (uint32_t tile = blockIdx.x * NH_WARPS_PER_BLOCK + warp; tile < n_tiles; tile += gridDim.x * NH_WARPS_PER_BLOCK) {
    const unsigned long long over = __shfl_sync(0xFFFFFFFFu, lane == 0 ? *((volatile unsigned long long *)&counters[1]) : 0ull, 0);
    if (over) break;
    const NhTileOut to = b.tile_out[tile];
    for (uint32_t j = lane; j < to.lk_cnt; j += 32u) {
      const uint64_t h = nh_fmix64(b.lk_min[to.lk_off + j]);
      if ((h & (EST_RANGES - 1)) >= EST_SAMPLED) continue;
      uint64_t i = (h >> 10) & mask;
      for (uint64_t probes = 0;; probes++) {
        if (probes > mask) {
          atomicExch(&counters[1], 1ull);
          break;
        }
        const unsigned long long old = atomicCAS(&set[i], EST_EMPTY, (unsigned long long)h);
        if (old == EST_EMPTY) {
          if (atomicAdd(&counters[0], 1ull) + 1 > limit) atomicExch(&counters[1], 1ull);
          break;
        }
        if (old == h) break;
        i = (i + 1) & mask;
      }
    }
  }
}

/* the keys of a set into one twice its size (same walk as above; every key is new there) */
__global__ void __launch_bounds__(256) k_estimate_rehash(const unsigned long long *from, uint64_t n_from,
                                                         unsigned long long *to, uint64_t mask) {
  for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < n_from; s += (uint64_t)gridDim.x * blockDim.x) {
    const unsigned long long h = from[s];
    if (h == EST_EMPTY) continue;
    uint64_t i = (h >> 10) & mask;
    while (atomicCAS(&to[i], EST_EMPTY, h) != EST_EMPTY) i = (i + 1) & mask;
  }
}

/* insert: a piece's taxon, from the batch's per-piece array */
struct PieceTaxa {
  const uint32_t *taxa;
  __device__ uint2 operator()(const NhTile &t) const { return make_uint2(taxa[t.seq], 0u); }
};

namespace {

using Clock = std::chrono::steady_clock;
double since(Clock::time_point t0) { return std::chrono::duration<double>(Clock::now() - t0).count(); }

uint64_t spaced_seed_mask(uint32_t l, uint32_t spaces) {
  /* kraken2-build's template '1' * (l - 2s) + '01' * s, every bit doubled (SURVEY A.1) */
  uint64_t m = 0;
  for (uint32_t i = 0; i < l; i++) {
    const bool one = i < l - 2 * spaces || ((i - (l - 2 * spaces)) & 1u);
    m = (m << 2) | (one ? 3u : 0u);
  }
  return m;
}

/* One host batch in pinned memory: concatenated pieces, their offsets and internal taxa. */
struct HostBatch {
  uint8_t *bases = nullptr;
  uint64_t *offs = nullptr;
  uint32_t *taxa = nullptr;
  uint32_t n = 0;
  uint64_t nb = 0;
};

/* Reads the library files in order and cuts their records into batches (the same cut for both passes). */
class Library {
 public:
  Library(const nh_build_params_t &p, const Taxonomy &T, uint64_t k, uint64_t max_bases, uint32_t max_pieces)
      : p_(p), T_(T), k_(k), max_bases_(max_bases), max_pieces_(max_pieces) {}
  void rewind() {
    file_ = -1;
    have_ = false;
    reader_.reset();
    sequences = skipped = bases = 0;
  }
  /* fills b; false when the library is exhausted and b is empty, or on error (rc set) */
  bool fill(HostBatch &b, int &rc) {
    b.n = 0;
    b.nb = 0;
    b.offs[0] = 0;
    while (b.n < max_pieces_) {
      if (!have_) {
        if ((rc = next_record())) return false;
        if (!have_) break; /* end of the library */
      }
      const uint64_t room = max_bases_ - b.nb, left = len_ - pos_;
      uint64_t take = left < room ? left : room;
      if (take < left && take < k_ + 256) break; /* too little room for a useful piece: next batch */
      memcpy(b.bases + b.nb, seq_ + pos_, take);
      b.nb += take;
      b.taxa[b.n] = taxon_;
      b.offs[++b.n] = b.nb;
      if (take == left)
        have_ = false;
      else
        pos_ += take - (k_ - 1); /* pieces overlap by k-1 bases so every k-mer is seen once */
    }
    return b.n > 0;
  }
  uint64_t sequences = 0, skipped = 0, bases = 0;

 private:
  int next_record() {
    for (;;) {
      if (!reader_) {
        if (++file_ >= p_.n_fasta) return NH_OK;
        reader_.reset(new NhSeqReader());
        if (int rc = reader_->open(p_.fasta[file_], p_.threads)) return rc;
      }
      const char *h, *s;
      size_t hl, sl;
      const int r = reader_->next(&h, &hl, &s, &sl);
      if (r < 0) return r;
      if (r == 0) {
        reader_.reset();
        continue;
      }
      size_t e = 1;
      while (e < hl && !isspace((unsigned char)h[e])) e++;
      auto it = T_.seq_taxon.find(std::string(h + 1, e - 1));
      if (it == T_.seq_taxon.end()) {
        skipped++;
        continue;
      }
      sequences++;
      bases += sl;
      if (sl < k_) continue; /* no k-mer */
      seq_ = (const uint8_t *)s;
      len_ = sl;
      pos_ = 0;
      taxon_ = it->second;
      have_ = true;
      return NH_OK;
    }
  }
  const nh_build_params_t &p_;
  const Taxonomy &T_;
  uint64_t k_, max_bases_;
  uint32_t max_pieces_;
  int file_ = -1;
  std::unique_ptr<NhSeqReader> reader_;
  bool have_ = false;
  const uint8_t *seq_ = nullptr;
  uint64_t len_ = 0, pos_ = 0;
  uint32_t taxon_ = 0;
};

struct SessionCloser {
  void operator()(nh_session *s) const { nh_session_destroy(s); }
};
struct DbCloser {
  void operator()(nh_db *d) const { nh_db_close(d); }
};

/* Everything one pass owns on the device and in pinned memory; freed on every path. */
struct Pass {
  std::unique_ptr<nh_db, DbCloser> db;
  std::unique_ptr<nh_session, SessionCloser> s;
  HostBatch hb[2];
  uint32_t *d_taxa = nullptr;
  unsigned long long *d_ctr = nullptr, *h_ctr = nullptr; /* [0] size / set keys, [1] full flag, [2] lookups */
  ~Pass() {
    if (s) cudaStreamSynchronize(s->stream);
    for (auto &b : hb) {
      if (b.bases) cudaFreeHost(b.bases);
      if (b.offs) cudaFreeHost(b.offs);
      if (b.taxa) cudaFreeHost(b.taxa);
    }
    if (h_ctr) cudaFreeHost(h_ctr);
    cudaFree(d_taxa);
    cudaFree(d_ctr);
  }
  int open(const std::vector<uint8_t> &opts, const std::vector<uint8_t> &taxo, uint64_t capacity, int device,
           uint64_t max_bases, uint32_t max_pieces) {
    nh_db *d = nullptr;
    if (int rc = nh_db_create_empty(opts.data(), opts.size(), taxo.data(), taxo.size(), capacity, device, &d)) return rc;
    db.reset(d);
    nh_params_t sp;
    memset(&sp, 0, sizeof sp);
    sp.minimum_hit_groups = 2;
    sp.max_batch_bases = max_bases;
    sp.max_batch_seqs = max_pieces;
    nh_session *ss = nullptr;
    if (int rc = nh_session_create_ex(d, &sp, true, &ss)) return rc; /* with the warp-per-tile kernel's lookup arrays */
    s.reset(ss);
    for (auto &b : hb) {
      CUDA_TRY(cudaHostAlloc(&b.bases, max_bases + 64, cudaHostAllocDefault));
      CUDA_TRY(cudaHostAlloc(&b.offs, (max_pieces + 1) * 8, cudaHostAllocDefault));
      CUDA_TRY(cudaHostAlloc(&b.taxa, max_pieces * 4, cudaHostAllocDefault));
    }
    CUDA_TRY(cudaHostAlloc(&h_ctr, 32, cudaHostAllocDefault));
    CUDA_TRY(cudaMalloc(&d_taxa, max_pieces * 4));
    CUDA_TRY(cudaMalloc(&d_ctr, 16));
    CUDA_TRY(cudaMemset(d_ctr, 0, 16));
    return NH_OK;
  }
  /* copies b and runs plan + minimizers on the session stream */
  NhBatchPtrs scan(const HostBatch &b) {
    nh_session *S = s.get();
    cudaStream_t st = S->stream;
    cudaMemcpyAsync(S->d_bases, b.bases, b.nb, cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(S->d_offsets, b.offs, (b.n + 1) * 8, cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(d_taxa, b.taxa, b.n * 4, cudaMemcpyHostToDevice, st);
    NhBatchPtrs B;
    memset(&B, 0, sizeof B);
    B.bases = S->d_bases;
    B.offsets = S->d_offsets;
    B.n_seqs = b.n;
    B.n_units = b.n;
    B.tile_base = S->d_tile_base;
    B.seq_info = S->d_seq_info; /* tiles written one thread per tile: pieces are long */
    B.tiles_upper = (uint32_t)(b.nb / (uint64_t)db->params.tile_pos + b.n + 1);
    B.block_sums = S->d_block_sums;
    B.tiles = S->d_tiles;
    B.tile_out = S->d_tile_out;
    B.lk_min = S->d_lk_min;
    B.lk_cnt = S->d_lk_cnt;
    B.lk_taxon = S->d_lk_taxon;
    B.counters = S->d_counters;
    nh_launch_plan(db->params, B, st);
    nh_launch_minimizers(db->params, B, B.tiles_upper, db->sm_count, st);
    return B;
  }
  /* the batch's counters back to the host; waits for the stream */
  int finish() {
    cudaStream_t st = s->stream;
    cudaMemcpyAsync(h_ctr, d_ctr, 16, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(h_ctr + 2, &s->d_counters->n_lookups, 4, cudaMemcpyDeviceToHost, st);
    const cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return nh_set_error(NH_ERR_CUDA, "build batch failed: %s", cudaGetErrorString(e));
    h_ctr[2] &= 0xFFFFFFFFull;
    return NH_OK;
  }
};

/* Pass 1: kraken2's estimate_capacity as recalled, not verified against its source: the minimizers whose
 * MurmurHash3 finaliser falls in the first EST_SAMPLED of EST_RANGES hash ranges (low bits) are collected
 * exactly, and estimate = |set| * EST_RANGES / EST_SAMPLED.  The set is exact for its sample, so the estimate
 * does not depend on scheduling. */
int estimate_capacity(Library &lib, Pass &P, uint64_t *estimate, uint64_t *final_slots, uint64_t *rescans) {
  /* NH_TEST_ESTIMATE_SLOTS=n (a power of two >= 64) starts the set that small, so that tests reach its growth */
  uint64_t slots = 1ull << 20;
  if (const char *e = getenv("NH_TEST_ESTIMATE_SLOTS")) {
    const uint64_t v = strtoull(e, nullptr, 10);
    if (v >= 64 && !(v & (v - 1))) slots = v;
  }
  typedef std::unique_ptr<unsigned long long, void (*)(unsigned long long *)> DevSet;
  auto dev_set = [](uint64_t n, DevSet &out) -> int {
    unsigned long long *p = nullptr;
    CUDA_TRY(cudaMalloc(&p, n * 8));
    out.reset(p);
    return NH_OK;
  };
  DevSet own(nullptr, [](unsigned long long *q) { cudaFree(q); }); /* frees the set on every return */
  if (int r = dev_set(slots, own)) return r;
  CUDA_TRY(cudaMemset(own.get(), 0xFF, slots * 8));
  const int sm = P.db->sm_count;
  cudaStream_t st = P.s->stream;
  /* doubles the set (k_estimate_rehash) and clears the overflow flag; the old set is freed only after the
   * rehash that reads it has finished */
  auto grow = [&]() -> int {
    DevSet bigger(nullptr, [](unsigned long long *q) { cudaFree(q); });
    if (int r = dev_set(2 * slots, bigger)) return r;
    CUDA_TRY(cudaMemsetAsync(bigger.get(), 0xFF, slots * 16, st));
    k_estimate_rehash<<<sm * 8, 256, 0, st>>>(own.get(), slots, bigger.get(), 2 * slots - 1);
    CUDA_TRY(cudaMemsetAsync(P.d_ctr + 1, 0, 8, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    own = std::move(bigger); /* frees the old set */
    slots *= 2;
    return NH_OK;
  };
  int rc = NH_OK, cur = 0;
  bool more = lib.fill(P.hb[cur], rc);
  while (more && rc == NH_OK) {
    const NhBatchPtrs B = P.scan(P.hb[cur]);
    k_estimate_tiles<<<sm * 8, NH_BLOCK_THREADS, 0, st>>>(B, own.get(), slots - 1, slots * 3 / 4, P.d_ctr);
    more = lib.fill(P.hb[cur ^ 1], rc); /* the host reads the next batch while the GPU works */
    cur ^= 1;
    if (int r = P.finish()) return r;
    while (P.h_ctr[1]) { /* the set filled up during the batch: double it and scan the batch again (idempotent) */
      if (int r = grow()) return r;
      k_estimate_tiles<<<sm * 8, NH_BLOCK_THREADS, 0, st>>>(B, own.get(), slots - 1, slots * 3 / 4, P.d_ctr);
      if (int r = P.finish()) return r;
      ++*rescans;
    }
    if (P.h_ctr[0] > slots / 2)
      if (int r = grow()) return r;
  }
  if (rc) return rc;
  *estimate = (uint64_t)P.h_ctr[0] * EST_RANGES / EST_SAMPLED;
  *final_slots = slots;
  return NH_OK;
}

/* Pass 2: every library minimizer into the table. */
int insert_library(Library &lib, Pass &P, uint64_t *minimizers) {
  const int sm = P.db->sm_count;
  cudaStream_t st = P.s->stream;
  const uint64_t capacity = P.db->info.capacity;
  const unsigned long long limit = (unsigned long long)(0.95 * (double)capacity);
  int rc = NH_OK, cur = 0;
  bool more = lib.fill(P.hb[cur], rc);
  *minimizers = 0;
  while (more && rc == NH_OK) {
    const NhBatchPtrs B = P.scan(P.hb[cur]);
    k_insert_tiles<<<sm * 8, NH_BLOCK_THREADS, 0, st>>>(P.db->params, P.db->d_cells, B, PieceTaxa{P.d_taxa}, limit,
                                                         P.d_ctr);
    more = lib.fill(P.hb[cur ^ 1], rc);
    cur ^= 1;
    if (int r = P.finish()) return r;
    *minimizers += P.h_ctr[2];
    if (P.h_ctr[1] || P.h_ctr[0] > limit)
      return nh_set_error(NH_ERR_CAPACITY, "table full: capacity %llu, size %llu (the load may not pass 0.95)",
                          (unsigned long long)capacity, (unsigned long long)P.h_ctr[0]);
  }
  return rc;
}

/* hash.k2d: the header, then the cells, copied back through two pinned buffers */
int write_hash(const std::string &path, Pass &P, uint64_t size) {
  const nh_db_info_t &I = P.db->info;
  FILE *f = fopen(path.c_str(), "wb");
  if (!f) return nh_set_error(NH_ERR_IO, "cannot create %s: %s", path.c_str(), strerror(errno));
  std::unique_ptr<FILE, int (*)(FILE *)> own(f, fclose);
  const uint64_t hdr[4] = {I.capacity, size, I.key_bits, I.value_bits};
  if (fwrite(hdr, 8, 4, f) != 4) return nh_set_error(NH_ERR_IO, "writing %s failed", path.c_str());
  const size_t total = I.capacity * 4;
  const size_t CH = std::min<size_t>(total, 64u << 20);
  uint8_t *stage[2] = {nullptr, nullptr};
  cudaEvent_t ev[2] = {nullptr, nullptr};
  int rc = NH_OK;
  cudaStream_t st = P.s->stream;
  cudaError_t e = cudaSuccess;
  for (int i = 0; i < 2 && e == cudaSuccess; i++) {
    e = cudaHostAlloc(&stage[i], CH, cudaHostAllocDefault);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming);
  }
  /* piece j is copied into stage[j & 1] while piece j - 1 is written */
  const size_t n_pieces = (total + CH - 1) / CH;
  for (size_t j = 0; e == cudaSuccess && j <= n_pieces && rc == NH_OK; j++) {
    if (j < n_pieces) {
      const size_t n = std::min(CH, total - j * CH);
      e = cudaMemcpyAsync(stage[j & 1], (const uint8_t *)P.db->d_cells + j * CH, n, cudaMemcpyDeviceToHost, st);
      if (e == cudaSuccess) e = cudaEventRecord(ev[j & 1], st);
    }
    if (j > 0 && e == cudaSuccess) {
      const size_t w = j - 1, n = std::min(CH, total - w * CH);
      e = cudaEventSynchronize(ev[w & 1]);
      if (e == cudaSuccess && fwrite(stage[w & 1], 1, n, f) != n) rc = nh_set_error(NH_ERR_IO, "writing %s failed", path.c_str());
    }
  }
  cudaStreamSynchronize(st);
  for (int i = 0; i < 2; i++) {
    if (stage[i]) cudaFreeHost(stage[i]);
    if (ev[i]) cudaEventDestroy(ev[i]);
  }
  if (rc == NH_OK && e != cudaSuccess) rc = nh_set_error(NH_ERR_CUDA, "copying the table back failed: %s", cudaGetErrorString(e));
  if (fclose(own.release()) != 0 && rc == NH_OK) rc = nh_set_error(NH_ERR_IO, "writing %s failed", path.c_str());
  return rc;
}

}  // namespace

extern "C" int nh_build_db(const nh_build_params_t *pin, nh_build_stats_t *stats) {
  if (!pin || !pin->out_dir || !pin->nodes_dmp || !pin->names_dmp || !pin->seqid2taxid || pin->n_fasta < 0 ||
      (pin->n_fasta && !pin->fasta))
    return nh_set_error(NH_ERR_INVALID, "bad argument");
  nh_build_params_t p = *pin;
  if (!p.k) p.k = 35;
  if (!p.l) p.l = 31;
  if (!p.spaces) p.spaces = 7;
  if (!(p.load_factor > 0)) p.load_factor = 0.7;
  if (!p.batch_bases) p.batch_bases = 256ull << 20;
  if (p.l > 31 || p.l < 1 || p.k < p.l || p.k - p.l + 1 > NH_MAX_WINDOW || 2 * p.spaces > p.l)
    return nh_set_error(NH_ERR_INVALID, "unsupported k=%u l=%u spaces=%u", p.k, p.l, p.spaces);
  if (p.load_factor > 0.95) return nh_set_error(NH_ERR_INVALID, "load factor %g above 0.95", p.load_factor);
  if (p.batch_bases < 4096 + 2ull * p.k || p.batch_bases > (1ull << 31))
    return nh_set_error(NH_ERR_INVALID, "batch_bases must be in [4096 + 2k, 2^31]");
  for (int i = 0; i < p.n_fasta; i++)
    if (!p.fasta[i]) return nh_set_error(NH_ERR_INVALID, "null library file name");
  nh_build_stats_t S;
  memset(&S, 0, sizeof S);
  auto t0 = Clock::now();
  Taxonomy T;
  if (int rc = load_taxonomy(p.nodes_dmp, p.names_dmp, p.seqid2taxid, T)) return rc;
  S.node_count = T.node_count;
  S.s_taxonomy = since(t0);

  /* opts.k2d: IndexOptions as kraken2-build writes it for a nucleotide library (SURVEY Appendix B) */
  std::vector<uint8_t> opts(64, 0);
  const uint64_t ok = p.k, ol = p.l, ssm = spaced_seed_mask(p.l, p.spaces), toggle = 0xE37E28C4271B5A2DULL;
  const int32_t revcom_version = 1;
  memcpy(&opts[0], &ok, 8);
  memcpy(&opts[8], &ol, 8);
  memcpy(&opts[16], &ssm, 8);
  memcpy(&opts[24], &toggle, 8);
  opts[32] = 1; /* dna_db */
  memcpy(&opts[48], &revcom_version, 4);

  const uint32_t max_pieces = (uint32_t)(p.batch_bases / 64 + 1024);
  Library lib(p, T, p.k, p.batch_bases, max_pieces);
  uint64_t capacity = p.capacity;
  if (!capacity) {
    t0 = Clock::now();
    Pass P1;
    if (int rc = P1.open(opts, T.image, 1024, p.device, p.batch_bases, max_pieces)) return rc;
    lib.rewind();
    if (int rc = estimate_capacity(lib, P1, &S.estimate, &S.estimate_slots, &S.estimate_rescans)) return rc;
    /* build_kraken2_db.sh, as recalled: capacity = (estimate + 8192) / load factor (rounded up here) */
    capacity = (uint64_t)ceil((double)(S.estimate + 8192) / p.load_factor);
    S.s_estimate = since(t0);
  }
  t0 = Clock::now();
  Pass P2;
  if (int rc = P2.open(opts, T.image, capacity, p.device, p.batch_bases, max_pieces)) return rc;
  lib.rewind();
  if (int rc = insert_library(lib, P2, &S.minimizers)) return rc;
  S.sequences = lib.sequences;
  S.skipped = lib.skipped;
  S.bases = lib.bases;
  S.capacity = capacity;
  S.size = P2.h_ctr[0];
  S.s_insert = since(t0);

  t0 = Clock::now();
  const std::string dir(p.out_dir);
  mkdir(dir.c_str(), 0777); /* an existing directory is fine; a failure shows when the files are created */
  const char *names[3] = {"hash.k2d", "opts.k2d", "taxo.k2d"};
  int rc = write_hash(dir + "/hash.k2d.tmp", P2, S.size);
  if (!rc) rc = write_file(dir + "/opts.k2d.tmp", opts.data(), opts.size());
  if (!rc) rc = write_file(dir + "/taxo.k2d.tmp", T.image.data(), T.image.size());
  int renamed = 0;
  for (; renamed < 3 && !rc; renamed++) {
    const std::string f = dir + "/" + names[renamed];
    if (rename((f + ".tmp").c_str(), f.c_str()) != 0) {
      rc = nh_set_error(NH_ERR_IO, "cannot rename %s.tmp: %s", f.c_str(), strerror(errno));
      break;
    }
  }
  if (rc) {
    /* the files already renamed go too: the directory never holds a partial set of this build's files */
    for (int i = 0; i < renamed; i++) unlink((dir + "/" + names[i]).c_str());
    for (auto n : names) unlink((dir + "/" + n + ".tmp").c_str());
    return rc;
  }
  S.s_write = since(t0);
  if (stats) *stats = S;
  return NH_OK;
}
