/*
 * nh_synth.cu — synthetic workload tooling (include/nohuman_synth.h): a
 * deterministic synthetic pangenome, a GPU kraken2-build (minimizer kernel +
 * atomicCAS insert with LCA merge, restating build_db.cc ProcessSequence /
 * CompactHashTable::CompareAndSet; SURVEY.md A.7) and a read sampler.
 * Not part of the classification path and never timed by bench.py.
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../../include/nohuman_synth.h"
#include "nh_internal.h"
#include "nh_kernels.cuh"

#define CUDA_TRY(expr)                                                                       \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess)                                                                   \
      return nh_set_error(NH_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                          __FILE__, __LINE__);                                               \
  } while (0)

/* ------------------------------------------------------------------ */
__device__ __forceinline__ uint32_t genome_code(uint64_t seed, uint64_t i) {
  const uint64_t w = nh_fmix64(seed + ((i >> 5) + 1ULL) * 0x9E3779B97F4A7C15ULL);
  return (uint32_t)(w >> (2u * (uint32_t)(i & 31ULL))) & 3u;
}

__device__ __forceinline__ uint8_t code_to_ascii(uint32_t c) {
  return (uint8_t)((0x54474341u >> (8u * c)) & 0xFFu); /* "ACGT" */
}

__global__ void __launch_bounds__(256)
k_synth_genome(uint8_t *__restrict__ out, uint64_t start, uint64_t n, uint64_t seed) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride)
    out[j] = code_to_ascii(genome_code(seed, start + j));
}

/* ------------------------------------------------------------------ */
/* build: CompareAndSet loop of build_db.cc collapsed to value := LCA(old, taxon) */

__device__ __forceinline__ uint32_t d_lca(const uint32_t *parent, uint32_t a, uint32_t b) {
  if (!a || !b) return a ? a : b;
  while (a != b) {
    if (a > b)
      a = parent[a];
    else
      b = parent[b];
  }
  return a;
}

/* returns 1 if a previously empty cell was claimed */
__device__ uint32_t cht_insert_lca(const NhDbParams &db, uint32_t *cells, uint64_t key,
                                   uint32_t taxon) {
  const uint64_t h = nh_fmix64(key);
  if (db.min_hash && h < db.min_hash) return 0;
  const uint32_t ckey = (uint32_t)(h >> (32u + db.value_bits));
  uint64_t idx = nh_fastmod(h, db.capacity, db.mod_m, db.mod_sh1, db.mod_sh2);
  for (uint64_t probes = 0; probes < db.capacity;) {
    uint32_t cell = *((volatile uint32_t *)&cells[idx]);
    if ((cell & db.value_mask) == 0u) {
      const uint32_t want = (ckey << db.value_bits) | taxon;
      const uint32_t old = atomicCAS(&cells[idx], 0u, want);
      if (old == 0u) return 1;
      cell = old; /* somebody else claimed it: examine what they wrote */
    }
    if ((cell >> db.value_bits) == ckey) {
      for (;;) {
        const uint32_t cur = cell & db.value_mask;
        const uint32_t nv = d_lca(db.parent, cur, taxon);
        if (nv == cur) return 0;
        const uint32_t want = (ckey << db.value_bits) | nv;
        const uint32_t old = atomicCAS(&cells[idx], cell, want);
        if (old == cell) return 0;
        cell = old;
      }
    }
    idx++;
    if (idx >= db.capacity) idx = 0;
    probes++;
  }
  return 0; /* table full: caller sees the load factor stall */
}

__global__ void __launch_bounds__(NH_BLOCK_THREADS)
k_insert_tiles(const NhDbParams db, uint32_t *cells, const NhBatchPtrs b, uint64_t chunk_start,
               const uint32_t *__restrict__ leaf_taxa, uint32_t n_leaves, uint64_t block_bases,
               uint64_t overlap_start, unsigned long long *size_counter) {
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t n_tiles = b.counters->n_tiles;
  uint32_t claimed = 0;
  for (uint32_t tile = blockIdx.x * NH_WARPS_PER_BLOCK + warp; tile < n_tiles;
       tile += gridDim.x * NH_WARPS_PER_BLOCK) {
    const NhTile t = b.tiles[tile];
    const NhTileOut to = b.tile_out[tile];
    const uint64_t g = chunk_start + t.pos_begin;
    const uint64_t blk = g / block_bases, r = g % block_bases;
    const uint32_t ta = leaf_taxa[blk % n_leaves];
    const uint32_t tb = r >= overlap_start ? leaf_taxa[(blk + 1) % n_leaves] : 0u;
    for (uint32_t j = lane; j < to.lk_cnt; j += 32u) {
      const uint64_t key = b.lk_min[to.lk_off + j];
      claimed += cht_insert_lca(db, cells, key, ta);
      if (tb) claimed += cht_insert_lca(db, cells, key, tb);
    }
  }
  claimed = __reduce_add_sync(0xFFFFFFFFu, claimed);
  if (lane == 0 && claimed) atomicAdd(size_counter, (unsigned long long)claimed);
}

extern "C" int nh_synth_build_db(const void *opts, size_t opts_len, const void *taxo,
                                 size_t taxo_len, const uint32_t *leaf_taxa, int n_leaves,
                                 const nh_synth_db_params_t *p, int device, nh_db **out,
                                 uint64_t *genome_bases) {
  if (!opts || !taxo || !leaf_taxa || n_leaves < 1 || !p || !out)
    return nh_set_error(NH_ERR_INVALID, "bad argument");
  if (p->capacity < 1024 || !(p->target_load > 0 && p->target_load < 0.95) || p->block_bases < 1024)
    return nh_set_error(NH_ERR_INVALID, "bad synthetic database parameters");
  nh_db *db = nullptr;
  int rc = nh_db_create_empty(opts, opts_len, taxo, taxo_len, p->capacity, device, &db);
  if (rc) return rc;
  for (int i = 0; i < n_leaves; i++)
    if (leaf_taxa[i] == 0 || leaf_taxa[i] >= db->info.node_count) {
      nh_db_close(db);
      return nh_set_error(NH_ERR_INVALID, "leaf taxon %u out of range", leaf_taxa[i]);
    }
  const uint64_t k = db->info.k;
  uint64_t chunk_max = p->capacity / 8;
  if (chunk_max > (128ULL << 20)) chunk_max = 128ULL << 20;
  if (chunk_max < (1ULL << 16)) chunk_max = 1ULL << 16;
  nh_params_t sp;
  memset(&sp, 0, sizeof sp);
  sp.minimum_hit_groups = 2;
  sp.max_batch_bases = chunk_max;
  sp.max_batch_seqs = 16;
  nh_session *s = nullptr;
  rc = nh_session_create_ex(db, &sp, true, &s); /* the builder runs the warp-per-tile minimizer kernel */
  if (rc) {
    nh_db_close(db);
    return rc;
  }
  uint32_t *d_leaf = nullptr;
  unsigned long long *d_size = nullptr;
  cudaError_t e = cudaMalloc(&d_leaf, n_leaves * 4);
  if (e == cudaSuccess) e = cudaMalloc(&d_size, 8);
  if (e == cudaSuccess) e = cudaMemcpy(d_leaf, leaf_taxa, n_leaves * 4, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemset(d_size, 0, 8);
  const uint64_t target = (uint64_t)(p->target_load * (double)p->capacity);
  const uint64_t overlap_start =
      (uint64_t)((1.0 - (p->overlap_frac < 0 ? 0 : p->overlap_frac)) * (double)p->block_bases);
  uint64_t gpos = 0; /* genome coordinate of the next chunk's first base */
  unsigned long long size = 0;
  cudaStream_t st = s->stream;
  const int sm = db->sm_count;
  int stalls = 0;
  while (e == cudaSuccess && size < target) {
    uint64_t need = target - size;
    uint64_t n = need * 3 + 4096; /* ~1 new cell per 3 bases (w = 5) */
    if (n > chunk_max) n = chunk_max;
    if (p->max_genome_bases && gpos + n > p->max_genome_bases) {
      if (gpos + k >= p->max_genome_bases) break;
      n = p->max_genome_bases - gpos;
    }
    const uint64_t offs[2] = {0, n};
    k_synth_genome<<<sm * 8, 256, 0, st>>>(s->d_bases, gpos, n, p->genome_seed);
    cudaMemcpyAsync(s->d_offsets, offs, 16, cudaMemcpyHostToDevice, st);
    NhBatchPtrs B;
    memset(&B, 0, sizeof B);
    B.bases = s->d_bases;
    B.offsets = s->d_offsets;
    B.n_seqs = 1;
    B.n_units = 1;
    B.tile_base = s->d_tile_base;
    B.block_sums = s->d_block_sums;
    B.tiles = s->d_tiles;
    B.tile_out = s->d_tile_out;
    B.lk_min = s->d_lk_min;
    B.lk_cnt = s->d_lk_cnt;
    B.lk_taxon = s->d_lk_taxon;
    B.counters = s->d_counters;
    nh_launch_plan(db->params, B, st);
    nh_launch_minimizers(db->params, B, (uint32_t)(n / (uint64_t)db->params.tile_pos + 2), sm, st);
    k_insert_tiles<<<sm * 8, NH_BLOCK_THREADS, 0, st>>>(db->params, db->d_cells, B, gpos, d_leaf,
                                                        (uint32_t)n_leaves, p->block_bases,
                                                        overlap_start, d_size);
    unsigned long long prev = size;
    e = cudaMemcpyAsync(&size, d_size, 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    gpos += n - (k - 1); /* chunks overlap by k-1 bases so every k-mer is seen once */
    if (size == prev && ++stalls > 8) break;
  }
  cudaFree(d_leaf);
  cudaFree(d_size);
  nh_session_destroy(s);
  if (e != cudaSuccess) {
    nh_db_close(db);
    return nh_set_error(NH_ERR_CUDA, "synthetic build failed: %s", cudaGetErrorString(e));
  }
  db->info.size = size;
  if (genome_bases) *genome_bases = gpos + (k - 1);
  rc = nh_db_build_filter(db);
  if (rc) {
    nh_db_close(db);
    return rc;
  }
  *out = db;
  return NH_OK;
}

extern "C" int nh_db_download_cells(const nh_db *db, uint32_t *out_cells) {
  if (!db || !out_cells) return nh_set_error(NH_ERR_INVALID, "null argument");
  CUDA_TRY(cudaSetDevice(db->info.device));
  CUDA_TRY(cudaMemcpy(out_cells, db->d_cells, db->info.capacity * 4, cudaMemcpyDeviceToHost));
  return NH_OK;
}

extern "C" int nh_synth_genome(int device, uint64_t genome_seed, uint64_t start, uint64_t n,
                               uint8_t *out_host) {
  if (!out_host) return nh_set_error(NH_ERR_INVALID, "null argument");
  if (n == 0) return NH_OK;
  CUDA_TRY(cudaSetDevice(device));
  uint8_t *d = nullptr;
  CUDA_TRY(cudaMalloc(&d, n));
  k_synth_genome<<<1024, 256>>>(d, start, n, genome_seed);
  cudaError_t e = cudaMemcpy(out_host, d, n, cudaMemcpyDeviceToHost);
  cudaFree(d);
  CUDA_TRY(e);
  return NH_OK;
}

/* ------------------------------------------------------------------ */
/* reads                                                               */

struct SynthReadsDev {
  uint64_t seed, genome_seed, genome_bases;
  uint32_t human_thr;  /* of 2^24 */
  uint32_t sub_thr, ins_thr, del_thr; /* cumulative, of 2^16 */
  uint32_t n_thr;      /* of 2^24 */
  int32_t paired;
  float insert_mean, insert_sd;
};

__global__ void __launch_bounds__(256)
k_synth_reads(uint8_t *__restrict__ bases, const uint64_t *__restrict__ off, uint64_t n_seqs,
              const SynthReadsDev P) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint64_t wstride = ((uint64_t)gridDim.x * blockDim.x) >> 5;
  for (uint64_t s = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; s < n_seqs;
       s += wstride) {
    const uint64_t o = off[s];
    const uint64_t len = off[s + 1] - o;
    if (len == 0) continue;
    const uint64_t u = P.paired ? (s >> 1) : s;
    const uint32_t mate = P.paired ? (uint32_t)(s & 1ULL) : 0u;
    const uint64_t hu = nh_fmix64(P.seed ^ nh_fmix64(u + 0x51ED27ULL));
    const bool human = (uint32_t)(hu & 0xFFFFFFu) < P.human_thr;
    /* fragment geometry (shared by both mates) */
    uint64_t frag_len = len + len / 8 + 64; /* slack for deletions */
    if (P.paired) {
      const uint64_t h2 = nh_fmix64(hu + 1);
      /* ~normal from 4 uniforms */
      float z = 0.f;
      /* explicit fused multiply-adds: oracle/k2_synth.c computes the same bits with fmaf() */
      for (int i = 0; i < 4; i++) z = __fmaf_rn((float)((h2 >> (16 * i)) & 0xFFFFu), 1.0f / 65536.0f, z);
      z = __fmul_rn(__fsub_rn(z, 2.0f), 1.7320508f);
      long long fl = (long long)__fmaf_rn(P.insert_sd, z, P.insert_mean);
      const uint64_t other = s ^ 1ULL;
      const uint64_t len_other = off[other + 1] - off[other];
      const uint64_t lmax = len > len_other ? len : len_other;
      if (fl < (long long)lmax) fl = (long long)lmax;
      frag_len = (uint64_t)fl + lmax / 8 + 64;
    }
    const uint64_t h3 = nh_fmix64(hu + 2);
    const uint64_t span = P.genome_bases > frag_len + 1 ? P.genome_bases - frag_len - 1 : 1;
    const uint64_t start = __umul64hi(h3, span);
    const uint32_t strand = (uint32_t)(nh_fmix64(hu + 3) & 1ULL);
    const bool forward = (mate ^ strand) == 0u;
    const uint64_t hs = nh_fmix64(hu ^ (0xA5A5ULL + mate));
    const bool has_n = (uint32_t)(hs & 0xFFFFFFu) < P.n_thr;
    const uint64_t n_pos = __umul64hi(nh_fmix64(hs + 7), len);
    for (uint64_t c = lane; c * 32ULL < len; c += 32ULL) {
      uint64_t rng = nh_fmix64(hs + 0x1000ULL + c);
      uint64_t sp = c * 32ULL; /* source offset inside the fragment */
      const uint64_t jend = (c * 32ULL + 32ULL < len) ? c * 32ULL + 32ULL : len;
      for (uint64_t j = c * 32ULL; j < jend; j++) {
        rng = rng * 6364136223846793005ULL + 1442695040888963407ULL;
        const uint32_t x = (uint32_t)(rng >> 48);
        const uint32_t rb = (uint32_t)(rng >> 40) & 3u;
        uint32_t code;
        if (!human) {
          code = rb;
        } else {
          bool take_src = true;
          if (x < P.sub_thr) {
            code = rb;
            sp++;
            take_src = false;
          } else if (x < P.ins_thr) {
            code = rb;
            take_src = false;
          } else if (x < P.del_thr) {
            sp++;
          }
          if (take_src) {
            const uint64_t fo = sp < frag_len ? sp : frag_len - 1;
            code = forward ? genome_code(P.genome_seed, start + fo)
                           : 3u - genome_code(P.genome_seed, start + frag_len - 1 - fo);
            sp++;
          }
        }
        uint8_t ch = code_to_ascii(code);
        if (has_n && j == n_pos) ch = 'N';
        bases[o + j] = ch;
      }
    }
  }
}

extern "C" int nh_synth_reads(int device, uint8_t *d_bases, const uint64_t *d_offsets,
                              uint64_t n_seqs, const nh_synth_reads_params_t *p,
                              void *cuda_stream) {
  if (!d_bases || !d_offsets || !p) return nh_set_error(NH_ERR_INVALID, "null argument");
  if (n_seqs == 0) return NH_OK;
  CUDA_TRY(cudaSetDevice(device));
  SynthReadsDev P;
  P.seed = p->seed;
  P.genome_seed = p->genome_seed;
  P.genome_bases = p->genome_bases;
  P.human_thr = (uint32_t)(p->human_frac * 16777216.0);
  const double s1 = p->sub_rate, s2 = s1 + p->ins_rate, s3 = s2 + p->del_rate;
  P.sub_thr = (uint32_t)(s1 * 65536.0);
  P.ins_thr = (uint32_t)(s2 * 65536.0);
  P.del_thr = (uint32_t)(s3 * 65536.0);
  P.n_thr = (uint32_t)(p->n_rate * 16777216.0);
  P.paired = p->paired;
  P.insert_mean = (float)p->insert_mean;
  P.insert_sd = (float)p->insert_sd;
  uint64_t blocks = (n_seqs + 7) / 8;
  if (blocks > 148 * 16) blocks = 148 * 16;
  k_synth_reads<<<(unsigned)blocks, 256, 0, (cudaStream_t)cuda_stream>>>(d_bases, d_offsets, n_seqs, P);
  CUDA_TRY(cudaGetLastError());
  return NH_OK;
}
