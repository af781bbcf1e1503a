/*
 * nh_inspect.cu — kraken2-inspect on the GPU (include/nohuman_gpu.h: nh_db_taxon_counts, nh_db_inspect,
 * nh_bench_taxon_counts; DESIGN.md §4g).
 *
 *   k_taxon_counts  one streaming pass over the resident cell array in 16-byte loads: every cell whose value
 *              (cell & value_mask) is non-zero is occupied; a value below node_count adds 1 to its taxon's
 *              count, one at or above it to out_of_range.  Value 0 is skipped as CompactHashTable::GetValueCounts
 *              skips it, whatever the key bits hold.  A lane holding its warp's hot taxon (in a human database
 *              nearly every cell) counts it in a register; other values are aggregated over the warp by a ballot
 *              and __match_any_sync, and one lane per distinct value adds the group (add_cell).
 *                SHARED    the groups go into a per-CTA histogram of uint32 bins in shared memory, whose non-zero
 *                          bins are added to the global uint64 counters at the end: taxonomies up to the opt-in
 *                          shared-memory size / 4 nodes (NH_TEST_INSPECT_SHARED_BINS=<n> lowers the bound so that
 *                          tests reach the other path).
 *                global    larger taxonomies add the groups to the global uint64 counters directly.
 *
 * nh_db_inspect counts first and writes afterwards, so a table with values that are not taxo.k2d nodes, or whose
 * occupied cells differ from the header's size, fails before any output exists.  The report body is the file
 * pipeline's --kraken-report writer (write_report, nh_pipeline.cc) over the per-taxon cell counts.
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include <algorithm>
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

constexpr uint32_t FULL = 0xFFFFFFFFu;
constexpr int COUNT_THREADS = 1024;
constexpr int COUNT_UNROLL = 4;                        /* 16-byte loads a lane has in flight per tile */
constexpr uint64_t TILE_VECS = 32 * COUNT_UNROLL;      /* a warp's tile: 128 loads of 4 cells */
constexpr uint64_t MAX_TILES_PER_WARP = (1ull << 18) - 1; /* keeps a CTA's cells below 2^32 (CountRun::open) */

typedef unsigned long long ull;

constexpr uint32_t NO_KEY = 0xFFFFFFFFu; /* no taxon id: node_count <= 2^31 */

/* Adds one cell per lane, `key` (a taxon id; 0: nothing), to its counter.  A lane holding the warp's `hot` key only
 * bumps its register hot_n, so a table that is nearly one taxon costs a compare and a ballot per cell.  Any other
 * key is aggregated over the warp (one atomic per distinct key): the lanes equal to the first such lane's key by a
 * ballot, the rest by __match_any_sync.  The first key aggregated that way becomes the warp's hot key (warp-uniform,
 * from a shuffle); in a human database that is nearly always the one taxon that holds most cells. */
template <bool SHARED>
__device__ __forceinline__ void add_cell(uint32_t key, uint32_t lane, uint32_t &hot, uint32_t &hot_n, uint32_t *bins,
                                         ull *counts) {
  hot_n += key == hot;
  const uint32_t rest = __ballot_sync(FULL, key != 0 && key != hot);
  if (rest == 0) return;
  const uint32_t src = __ffs(rest) - 1;
  const uint32_t first = __shfl_sync(FULL, key, src);
  const uint32_t same = __ballot_sync(FULL, key == first) & rest;
  uint32_t n = lane == src ? __popc(same) : 0;
  if ((rest & ~same) >> lane & 1u) { /* exactly the lanes of rest & ~same reach this call */
    const uint32_t peers = __match_any_sync(rest & ~same, key);
    n = lane == __ffs(peers) - 1 ? __popc(peers) : 0;
  }
  if (n) {
    if (SHARED)
      atomicAdd(&bins[key], n);
    else
      atomicAdd(&counts[key], (ull)n);
  }
  if (hot == NO_KEY) hot = first;
}

/* counts[node_count] += cells per value, totals[0] += occupied cells, totals[1] += values >= node_count.
 * cells: n_vec 16-byte groups (the array is zero-padded to a multiple of 32 cells).  Warp w reads tiles w, w + W,
 * ... of TILE_VECS groups; the tile loop is warp-uniform, so every lane takes part in every warp collective. */
template <bool SHARED>
__global__ void __launch_bounds__(COUNT_THREADS, 1) k_taxon_counts(const uint4 *__restrict__ cells, uint64_t n_vec,
                                                                uint32_t value_mask, uint32_t node_count,
                                                                ull *__restrict__ counts, ull *__restrict__ totals) {
  extern __shared__ uint32_t bins[];
  const uint32_t lane = threadIdx.x & 31u;
  if (SHARED) {
    for (uint32_t i = threadIdx.x; i < node_count; i += blockDim.x) bins[i] = 0;
    __syncthreads();
  }
  const uint64_t n_warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
  /* per-lane totals fit 32 bits: a lane reads at most 16 cells of each of < 2^18 tiles */
  uint32_t occupied = 0, out_of_range = 0, hot = NO_KEY, hot_n = 0;
  for (uint64_t t = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); t * TILE_VECS < n_vec; t += n_warps) {
    uint4 v[COUNT_UNROLL];
#pragma unroll
    for (int j = 0; j < COUNT_UNROLL; j++) {
      const uint64_t i = t * TILE_VECS + j * 32 + lane;
      v[j] = i < n_vec ? __ldcs(cells + i) : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int j = 0; j < COUNT_UNROLL; j++) {
      const uint32_t c[4] = {v[j].x & value_mask, v[j].y & value_mask, v[j].z & value_mask, v[j].w & value_mask};
#pragma unroll
      for (int q = 0; q < 4; q++) {
        occupied += c[q] != 0;
        out_of_range += c[q] >= node_count; /* node_count >= 1, so value 0 is never out of range */
        add_cell<SHARED>(c[q] < node_count ? c[q] : 0, lane, hot, hot_n, bins, counts);
      }
    }
  }
  occupied = __reduce_add_sync(FULL, occupied);
  out_of_range = __reduce_add_sync(FULL, out_of_range);
  hot_n = __reduce_add_sync(FULL, hot_n); /* a warp's cells, like its CTA's, are fewer than 2^32 */
  if (lane == 0) {
    if (occupied) atomicAdd(&totals[0], (ull)occupied);
    if (out_of_range) atomicAdd(&totals[1], (ull)out_of_range);
    if (hot_n) {
      if (SHARED)
        atomicAdd(&bins[hot], hot_n);
      else
        atomicAdd(&counts[hot], (ull)hot_n);
    }
  }
  if (SHARED) {
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < node_count; i += blockDim.x)
      if (bins[i]) atomicAdd(&counts[i], (ull)bins[i]);
  }
}

int device_check() {
  int nd = 0;
  if (cudaGetDeviceCount(&nd) != cudaSuccess || nd < 1) {
    cudaGetLastError();
    return nh_set_error(NH_ERR_CUDA, "no CUDA device (no CPU path)");
  }
  return NH_OK;
}

/* taxonomies up to this many nodes are counted in shared memory */
uint64_t shared_bins_bound(int device) {
  int optin = 0;
  if (cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device) != cudaSuccess) {
    cudaGetLastError();
    optin = 48 << 10;
  }
  uint64_t bound = (uint64_t)optin / 4;
  /* NH_TEST_INSPECT_SHARED_BINS=<n>: tests force the global path on a small taxonomy */
  if (const char *e = getenv("NH_TEST_INSPECT_SHARED_BINS")) bound = std::min<uint64_t>(bound, strtoull(e, nullptr, 10));
  return bound;
}

/* One run of k_taxon_counts over db's table on db's device: its own stream, events and scratch (node_count
 * counters, then occupied and out_of_range), released when it goes out of scope. */
class CountRun {
 public:
  ~CountRun() {
    if (stream_) cudaStreamSynchronize(stream_);
    cudaFree(d_scratch_);
    for (auto ev : ev_)
      if (ev) cudaEventDestroy(ev);
    if (stream_) cudaStreamDestroy(stream_);
  }
  int open(const nh_db *db) {
    if (int rc = device_check()) return rc;
    if (!db) return nh_set_error(NH_ERR_INVALID, "null database");
    db_ = db;
    const int dev = db->info.device;
    CUDA_TRY(cudaSetDevice(dev));
    CUDA_TRY(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
    for (auto &ev : ev_) CUDA_TRY(cudaEventCreate(&ev));
    n_nodes_ = db->info.node_count;
    CUDA_TRY(cudaMalloc(&d_scratch_, (n_nodes_ + 2) * sizeof(ull)));
    n_vec_ = (db->info.capacity + 31) / 32 * 8;
    shared_ = n_nodes_ <= shared_bins_bound(dev);
    smem_ = shared_ ? n_nodes_ * 4 : 0;
    int optin = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    int per_sm = 0;
    if (shared_) {
      /* always the same value, so concurrent callers cannot undo each other's setting */
      CUDA_TRY(cudaFuncSetAttribute(k_taxon_counts<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
      CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_taxon_counts<true>, COUNT_THREADS, smem_));
    } else {
      CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_taxon_counts<false>, COUNT_THREADS, 0));
    }
    /* A CTA's shared bins must not wrap: its 32 warps read at most ceil(tiles / warps) tiles each, 4 * TILE_VECS
     * cells a tile, so with at most MAX_TILES_PER_WARP tiles a warp a CTA reads fewer than 32 * 2^18 * 512 = 2^32
     * cells.  The grid is one wave of resident CTAs, or more when the table needs more to keep that bound. */
    const uint64_t tiles = (n_vec_ + TILE_VECS - 1) / TILE_VECS;
    const uint64_t min_grid = (tiles + 32 * MAX_TILES_PER_WARP - 1) / (32 * MAX_TILES_PER_WARP);
    grid_ = (uint64_t)std::max(per_sm, 1) * std::max(db->sm_count, 1);
    grid_ = std::max(std::min(grid_, tiles), min_grid);
    if (grid_ > 0x7FFFFFFFull) return nh_set_error(NH_ERR_UNSUPPORTED, "table too large to count");
    return NH_OK;
  }
  void launch() {
    cudaMemsetAsync(d_scratch_, 0, (n_nodes_ + 2) * sizeof(ull), stream_);
    const uint4 *cells = (const uint4 *)db_->d_cells;
    const uint32_t mask = db_->params.value_mask, nc = (uint32_t)n_nodes_;
    ull *totals = d_scratch_ + n_nodes_;
    if (shared_)
      k_taxon_counts<true><<<(unsigned)grid_, COUNT_THREADS, smem_, stream_>>>(cells, n_vec_, mask, nc, d_scratch_, totals);
    else
      k_taxon_counts<false><<<(unsigned)grid_, COUNT_THREADS, 0, stream_>>>(cells, n_vec_, mask, nc, d_scratch_, totals);
  }
  /* counts[node_count], *occupied, *out_of_range of one run */
  int run(std::vector<uint64_t> &counts, uint64_t *occupied, uint64_t *out_of_range) {
    counts.assign(n_nodes_ + 2, 0);
    launch();
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(counts.data(), d_scratch_, (n_nodes_ + 2) * sizeof(ull), cudaMemcpyDeviceToHost, stream_));
    if (int rc = sync()) return rc;
    *occupied = counts[n_nodes_];
    *out_of_range = counts[n_nodes_ + 1];
    counts.resize(n_nodes_);
    return NH_OK;
  }
  /* mean device time of a run (counter reset and kernel) over `iters` runs after one warm-up */
  int time(int iters, double *seconds) {
    launch();
    CUDA_TRY(cudaEventRecord(ev_[0], stream_));
    for (int i = 0; i < iters; i++) launch();
    CUDA_TRY(cudaEventRecord(ev_[1], stream_));
    CUDA_TRY(cudaGetLastError());
    if (int rc = sync()) return rc;
    float ms = 0;
    CUDA_TRY(cudaEventElapsedTime(&ms, ev_[0], ev_[1]));
    *seconds = ms / 1e3 / iters;
    return NH_OK;
  }

 private:
  int sync() {
    const cudaError_t e = cudaStreamSynchronize(stream_);
    return e == cudaSuccess ? NH_OK : nh_set_error(NH_ERR_CUDA, "counting the table's taxa failed: %s", cudaGetErrorString(e));
  }
  const nh_db *db_ = nullptr;
  uint64_t n_nodes_ = 0, n_vec_ = 0, grid_ = 0;
  size_t smem_ = 0;
  bool shared_ = false;
  cudaStream_t stream_ = nullptr;
  cudaEvent_t ev_[2] = {nullptr, nullptr};
  ull *d_scratch_ = nullptr;
};

/* the n low bits of mask, most significant first (dump_table.cc's mask2str) */
std::string mask_bits(uint64_t mask, int n) {
  std::string s;
  for (int i = n - 1; i >= 0; i--) s.push_back((mask >> i) & 1 ? '1' : '0');
  return s;
}

}  // namespace

extern "C" int nh_db_taxon_counts(const nh_db *db, uint64_t *counts, uint64_t n_counts, uint64_t *occupied,
                                  uint64_t *out_of_range) {
  if (int rc = device_check()) return rc;
  if (!db || !counts) return nh_set_error(NH_ERR_INVALID, "null argument");
  if (n_counts < db->info.node_count)
    return nh_set_error(NH_ERR_INVALID, "counts holds %llu entries, the taxonomy has %llu nodes",
                        (unsigned long long)n_counts, (unsigned long long)db->info.node_count);
  CountRun run;
  std::vector<uint64_t> c;
  uint64_t occ = 0, oor = 0;
  if (int rc = run.open(db)) return rc;
  if (int rc = run.run(c, &occ, &oor)) return rc;
  std::copy(c.begin(), c.end(), counts);
  std::fill(counts + c.size(), counts + n_counts, 0);
  if (occupied) *occupied = occ;
  if (out_of_range) *out_of_range = oor;
  return NH_OK;
}

extern "C" int nh_db_inspect(const nh_db *db, const char *out_path, int32_t flags) {
  if (int rc = device_check()) return rc;
  if (!db) return nh_set_error(NH_ERR_INVALID, "null database");
  if (flags & ~(NH_INSPECT_SKIP_COUNTS | NH_INSPECT_ZERO_COUNTS)) return nh_set_error(NH_ERR_INVALID, "unknown flags %d", flags);
  const nh_db_info_t &I = db->info;
  CountRun run;
  std::vector<uint64_t> counts;
  uint64_t occupied = 0, out_of_range = 0;
  if (int rc = run.open(db)) return rc;
  if (int rc = run.run(counts, &occupied, &out_of_range)) return rc;
  if (out_of_range)
    return nh_set_error(NH_ERR_IO, "hash.k2d: %llu cells hold taxon ids >= node_count %llu", (unsigned long long)out_of_range,
                        (unsigned long long)I.node_count);
  if (occupied != I.size)
    return nh_set_error(NH_ERR_IO, "hash.k2d: occupied cells %llu != header size %llu", (unsigned long long)occupied,
                        (unsigned long long)I.size);
  const bool to_stdout = !out_path || !strcmp(out_path, "-");
  FILE *f = to_stdout ? stdout : fopen(out_path, "w");
  if (!f) return nh_set_error(NH_ERR_IO, "cannot open %s for writing", out_path);
  fprintf(f, "# Database options: %s db, k = %llu, l = %llu\n", I.dna_db ? "nucleotide" : "protein",
          (unsigned long long)I.k, (unsigned long long)I.l);
  fprintf(f, "# Spaced mask = %s\n", mask_bits(I.spaced_seed_mask, (int)I.l * 2).c_str());
  fprintf(f, "# Toggle mask = %s\n", mask_bits(I.toggle_mask, 64).c_str());
  fprintf(f, "# Total taxonomy nodes: %llu\n", (unsigned long long)I.node_count);
  fprintf(f, "# Table size: %llu\n", (unsigned long long)I.size);
  fprintf(f, "# Table capacity: %llu\n", (unsigned long long)I.capacity);
  if (I.minimum_acceptable_hash_value)
    fprintf(f, "# Min clear hash value = %llu\n", (unsigned long long)I.minimum_acceptable_hash_value);
  bool ok = true;
  if (!(flags & NH_INSPECT_SKIP_COUNTS)) {
    uint64_t total = 0;
    for (uint64_t c : counts) total += c;
    ok = write_report(f, db, counts, total, 0, (flags & NH_INSPECT_ZERO_COUNTS) != 0);
  }
  ok = fflush(f) == 0 && !ferror(f) && ok;
  if (!to_stdout) {
    ok = fclose(f) == 0 && ok;
    if (!ok) unlink(out_path);
  }
  return ok ? NH_OK : nh_set_error(NH_ERR_IO, "writing %s failed", to_stdout ? "stdout" : out_path);
}

extern "C" int nh_bench_taxon_counts(const nh_db *db, int iters, double *out_seconds) {
  if (int rc = device_check()) return rc;
  if (!db || !out_seconds || iters < 1) return nh_set_error(NH_ERR_INVALID, "bad argument");
  CountRun run;
  if (int rc = run.open(db)) return rc;
  return run.time(iters, out_seconds);
}
