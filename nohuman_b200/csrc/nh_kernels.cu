/*
 * nh_kernels.cu — the classification path as hand-written sm_100a kernels.
 * Integer/byte work bound by issue slots (minimizer scan) and by random
 * 32-byte reads of the hash table, which on B200 are limited by address
 * translation (DESIGN.md §3); no tensor-core work exists on this path.
 *
 * Upstream units each kernel stands for (kraken2 @ reference Dockerfile:15,
 * 35-38; behavioural spec SURVEY.md Appendix A):
 *   k_plan_*             (none: tiles, lookup slots, tile roles, deferred units)
 *   k_stream_classify    mmscanner.cc MinimizerScanner::NextMinimizer/is_ambiguous,
 *                        the last_minimizer de-duplication of classify.cc
 *                        ClassifySequence, kv_store.h MurmurHash3, compact_hash.cc
 *                        CompactHashTable::Get (LINEAR_PROBING build), classify.cc
 *                        ResolveTree + taxonomy.cc IsAAncestorOfB /
 *                        LowestCommonAncestor — one kernel, the default path (A.3-A.5)
 *   k_score              ClassifySequence tail + ResolveTree for units whose tiles span
 *                        several warps (long reads)                              (A.5)
 *   k_score_big          a whole unit again, warp-per-unit with a 16K-slot table: units
 *                        that hit more distinct taxa than the in-warp tables hold  (A.3-A.5)
 *   k_minimizers, k_probe  warp-per-tile scan and thread-per-lookup probe: any window
 *                        width k-l+1 <= 32, the synthetic builder, A/B runs     (A.3, A.4)
 *   k_gather_runs        per-read hit runs for kraken2's --output lines          (A.6)
 * and, in the reference itself, the keep/drop polarity of
 * src/main.rs:259-265 (--classified-out vs --unclassified-out).
 */
#include <stdlib.h>
#include <string.h>

#include "nh_kernels.cuh"

#define FULL_MASK 0xFFFFFFFFu

/* ------------------------------------------------------------------ */
/* small helpers                                                       */

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

__device__ __forceinline__ uint32_t warp_sum_u32(uint32_t v) {
  return __reduce_add_sync(FULL_MASK, v);
}

/* exclusive scan over a block of up to 1024 threads; *total gets the sum.
 * The plan scans (tiles << 32 | k-mer positions) in one pass. */
__device__ __forceinline__ uint64_t block_excl_scan(uint64_t v, uint64_t *total,
                                                    uint64_t *s_warp /* [33] */) {
  uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
  uint64_t inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint64_t o = __shfl_up_sync(FULL_MASK, inc, d);
    if (lane >= (uint32_t)d) inc += o;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    uint32_t nw = (blockDim.x + 31) >> 5;
    uint64_t ws = lane < nw ? s_warp[lane] : 0;
    uint64_t winc = ws;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint64_t o = __shfl_up_sync(FULL_MASK, winc, d);
      if (lane >= (uint32_t)d) winc += o;
    }
    s_warp[lane] = winc - ws; /* exclusive warp base */
    if (lane == 31) s_warp[32] = winc;
  }
  __syncthreads();
  uint64_t r = s_warp[warp] + inc - v;
  *total = s_warp[32];
  __syncthreads();
  return r;
}

/* ------------------------------------------------------------------ */
/* stage 0: plan — cut every sequence into tiles of <= tile_pos k-mers  */

#define PLAN_THREADS 1024

__device__ __forceinline__ uint32_t seq_npos(const uint64_t *__restrict__ off, uint32_t s, int k) {
  uint64_t len = off[s + 1] - off[s];
  return len < (uint64_t)k ? 0u : (uint32_t)(len - (uint64_t)k + 1);
}

__device__ __forceinline__ uint32_t npos_ntiles(uint32_t npos, int tile_pos) {
  return (npos + (uint32_t)tile_pos - 1u) / (uint32_t)tile_pos;
}

/* (tiles << 32) | positions of sequence s */
__device__ __forceinline__ uint64_t seq_work(const uint64_t *__restrict__ off, uint32_t s, int k,
                                             int tile_pos) {
  const uint32_t np = seq_npos(off, s, k);
  return ((uint64_t)npos_ntiles(np, tile_pos) << 32) | np;
}

__global__ void __launch_bounds__(PLAN_THREADS)
k_plan_count(const uint64_t *__restrict__ off, uint32_t n_seqs, int k, int tile_pos,
             uint64_t *__restrict__ block_sums) {
  __shared__ uint64_t s_warp[33];
  uint32_t s = blockIdx.x * PLAN_THREADS + threadIdx.x;
  uint64_t v = s < n_seqs ? seq_work(off, s, k, tile_pos) : 0;
  uint64_t total;
  block_excl_scan(v, &total, s_warp);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

/* single block: exclusive scan of the per-block sums, reset of the batch counters */
__global__ void __launch_bounds__(PLAN_THREADS)
k_plan_scan(uint64_t *__restrict__ block_sums, uint32_t nb, NhCounters *__restrict__ counters) {
  __shared__ uint64_t s_warp[33];
  __shared__ uint64_t s_running;
  if (threadIdx.x == 0) s_running = 0;
  __syncthreads();
  for (uint32_t base = 0; base < nb; base += PLAN_THREADS) {
    uint32_t i = base + threadIdx.x;
    uint64_t v = i < nb ? block_sums[i] : 0;
    uint64_t total;
    uint64_t ex = block_excl_scan(v, &total, s_warp);
    uint64_t run = s_running;
    if (i < nb) block_sums[i] = run + ex;
    __syncthreads();
    if (threadIdx.x == 0) s_running = run + total;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    counters->n_tiles = (uint32_t)(s_running >> 32);
    counters->n_lookups = 0;
    counters->n_classified = 0;
    counters->n_kept = 0;
    counters->n_overflow = 0;
    counters->error = 0;
    counters->n_deferred = 0;
    counters->next_group = 0;
    counters->n_sector_reads = 0;
  }
}

/* Writes the tile descriptors.  With `fused` set it also decides, per unit,
 * whether the streaming kernel can score it inside one warp (all its tiles in
 * one group of 32) and queues the other units for k_score. */
__global__ void __launch_bounds__(PLAN_THREADS)
k_plan_fill(const uint64_t *__restrict__ off, uint32_t n_seqs, int k, int tile_pos, int paired,
            int fused, const uint64_t *__restrict__ block_sums, uint32_t *__restrict__ tile_base,
            NhTile *__restrict__ tiles, uint32_t *__restrict__ deferred_units,
            NhCounters *__restrict__ counters, uint2 *__restrict__ seq_info) {
  __shared__ uint64_t s_warp[33];
  uint32_t s = blockIdx.x * PLAN_THREADS + threadIdx.x;
  uint64_t w = s < n_seqs ? seq_work(off, s, k, tile_pos) : 0;
  uint64_t total;
  uint64_t ex = block_excl_scan(w, &total, s_warp);
  if (s < n_seqs) {
    const uint64_t before = block_sums[blockIdx.x] + ex;
    const uint32_t tb = (uint32_t)(before >> 32), pb = (uint32_t)before;
    const uint32_t v = (uint32_t)(w >> 32);
    tile_base[s] = tb;
    uint32_t first_tile = tb;
    bool in_warp = false;
    if (fused) {
      const uint32_t mate = paired ? (s & 1u) : 0u;
      const uint32_t v_other = paired ? npos_ntiles(seq_npos(off, s ^ 1u, k), tile_pos) : 0u;
      /* mates are consecutive sequences, so a pair's tiles are consecutive too */
      first_tile = mate == 0u ? tb : tb - v_other;
      const uint32_t vt = v + v_other;
      in_warp = vt >= 1u && vt <= 32u && (first_tile >> 5) == ((first_tile + vt - 1u) >> 5);
      if (mate == 0u && !in_warp) /* also units without any k-mer: k_score calls them unclassified */
        deferred_units[atomicAdd(&counters->n_deferred, 1u)] = paired ? (s >> 1) : s;
    }
    if (seq_info != nullptr) {
      /* long reads: k_plan_tiles writes the descriptors, one thread per tile */
      seq_info[s] = make_uint2(pb, in_warp ? first_tile : 0xFFFFFFFFu);
    } else {
      for (uint32_t t = 0; t < v; t++) {
        NhTile d;
        d.seq = s;
        d.pos_begin = t * (uint32_t)tile_pos;
        d.slot = pb + d.pos_begin;
        d.role = !in_warp ? NH_ROLE_DEFERRED
                          : (tb + t == first_tile ? NH_ROLE_LEADER : (NH_ROLE_MEMBER | ((tb + t - first_tile) << 8)));
        tiles[tb + t] = d;
      }
    }
  }
  if (s == 0) tile_base[n_seqs] = counters->n_tiles;
}

/* Sequence lengths -> what the kernels read: base offsets (u64) and, for packed input, every sequence's
 * first unit of 32 bases (u32).  nh_classify_batch_pack sends 4 bytes per sequence instead of 12. */
__global__ void __launch_bounds__(PLAN_THREADS)
k_len_count(const uint32_t *__restrict__ len, uint32_t n_seqs, uint64_t *__restrict__ sums /* [2 * blocks] */) {
  __shared__ uint64_t s_warp[33];
  const uint32_t s = blockIdx.x * PLAN_THREADS + threadIdx.x;
  const uint64_t l = s < n_seqs ? len[s] : 0;
  uint64_t total_l, total_u;
  block_excl_scan(l, &total_l, s_warp);
  block_excl_scan((l + 31) >> 5, &total_u, s_warp);
  if (threadIdx.x == 0) {
    sums[2u * blockIdx.x] = total_l;
    sums[2u * blockIdx.x + 1u] = total_u;
  }
}

__global__ void __launch_bounds__(PLAN_THREADS)
k_len_scan(uint64_t *__restrict__ sums, uint32_t nb) {
  __shared__ uint64_t s_warp[33];
  __shared__ uint64_t s_run[2];
  if (threadIdx.x < 2) s_run[threadIdx.x] = 0;
  __syncthreads();
  for (uint32_t base = 0; base < nb; base += PLAN_THREADS) {
    const uint32_t i = base + threadIdx.x;
#pragma unroll
    for (uint32_t q = 0; q < 2; q++) {
      const uint64_t v = i < nb ? sums[2u * i + q] : 0;
      uint64_t total;
      const uint64_t ex = block_excl_scan(v, &total, s_warp);
      const uint64_t run = s_run[q];
      if (i < nb) sums[2u * i + q] = run + ex;
      __syncthreads();
      if (threadIdx.x == 0) s_run[q] = run + total;
      __syncthreads();
    }
  }
}

__global__ void __launch_bounds__(PLAN_THREADS)
k_len_fill(const uint32_t *__restrict__ len, uint32_t n_seqs, const uint64_t *__restrict__ sums,
           uint64_t *__restrict__ off /* [n_seqs + 1] */, uint32_t *__restrict__ poff /* [n_seqs + 1] */) {
  __shared__ uint64_t s_warp[33];
  const uint32_t s = blockIdx.x * PLAN_THREADS + threadIdx.x;
  const uint64_t l = s < n_seqs ? len[s] : 0;
  uint64_t total;
  const uint64_t ex_l = block_excl_scan(l, &total, s_warp);
  const uint64_t ex_u = block_excl_scan((l + 31) >> 5, &total, s_warp);
  if (s < n_seqs) {
    const uint64_t o = sums[2u * blockIdx.x] + ex_l, u = sums[2u * blockIdx.x + 1u] + ex_u;
    off[s] = o;
    poff[s] = (uint32_t)u;
    if (s == n_seqs - 1u) {
      off[n_seqs] = o + l;
      poff[n_seqs] = (uint32_t)(u + ((l + 31) >> 5));
    }
  }
}

/* The tile descriptors of a batch of long reads, one thread per tile (a 100 kb read has 400 tiles:
 * one thread writing them all was 7 % of a step of 50 kb reads).  The sequence of a tile is found
 * by bisection over tile_base. */
__global__ void __launch_bounds__(256)
k_plan_tiles(const uint32_t *__restrict__ tile_base, const uint2 *__restrict__ seq_info, uint32_t n_seqs, int tile_pos,
             NhTile *__restrict__ tiles, const NhCounters *__restrict__ counters) {
  const uint32_t n_tiles = counters->n_tiles;
  for (uint32_t tile = blockIdx.x * blockDim.x + threadIdx.x; tile < n_tiles; tile += gridDim.x * blockDim.x) {
    uint32_t lo = 0, hi = n_seqs; /* last s with tile_base[s] <= tile (sequences without tiles share their successor's base) */
    while (hi - lo > 1u) {
      const uint32_t mid = (lo + hi) >> 1;
      if (tile_base[mid] <= tile) lo = mid; else hi = mid;
    }
    const uint2 si = seq_info[lo];
    NhTile d;
    d.seq = lo;
    d.pos_begin = (tile - tile_base[lo]) * (uint32_t)tile_pos;
    d.slot = si.x + d.pos_begin;
    d.role = si.y == 0xFFFFFFFFu ? NH_ROLE_DEFERRED : (tile == si.y ? NH_ROLE_LEADER : (NH_ROLE_MEMBER | ((tile - si.y) << 8)));
    tiles[tile] = d;
  }
}

/* ------------------------------------------------------------------ */
/* stage 1: minimizers — one warp per tile                             */

struct __align__(16) MinWarpSmem {
  uint64_t st_min[NH_TILE_LMERS];      /* staged distinct-consecutive minimizers */
  uint32_t packed[16];                 /* 2-bit bases, 16 per word, first base in the MSBs */
  uint32_t ambits[8];                  /* 1 bit per base, LSB first */
  uint8_t st_start[NH_TILE_LMERS + 8]; /* ordinal (among non-ambiguous positions) of each run start */
};

__device__ __forceinline__ bool any_bits(const uint32_t *bits, uint32_t start, uint32_t n) {
  uint32_t j = start >> 5, o = start & 31u;
  uint32_t lo = __funnelshift_r(bits[j], bits[j + 1], o);
  if (n <= 32) return (lo & (n == 32 ? 0xFFFFFFFFu : ((1u << n) - 1u))) != 0;
  uint32_t hi = __funnelshift_r(bits[j + 1], bits[j + 2], o);
  n -= 32;
  return lo != 0 || (hi & (n >= 32 ? 0xFFFFFFFFu : ((1u << n) - 1u))) != 0;
}

__device__ __forceinline__ uint64_t shfl_carry(uint64_t cur, uint64_t prev, uint32_t d,
                                               uint32_t lane) {
  /* value of lane (lane - d); lanes that wrap take the previous iteration's value */
  uint64_t send = (lane >= 32u - d) ? prev : cur;
  return __shfl_sync(FULL_MASK, send, (lane - d) & 31u);
}

__device__ __forceinline__ uint64_t min_u64(uint64_t a, uint64_t b) { return a < b ? a : b; }

/* Returns the number of runs staged in sm (warp-uniform). */
template <int WT>
__device__ __forceinline__ uint32_t minimizer_tile(const NhDbParams &db, const NhBatchPtrs &b,
                                                   const NhTile t, MinWarpSmem &sm,
                                                   uint32_t lane) {
  const int k = db.k, l = db.l;
  const int w = WT ? WT : db.w;
  const uint64_t so = b.offsets[t.seq];
  const uint32_t len = (uint32_t)(b.offsets[t.seq + 1] - so);
  const uint32_t npos_total = len - (uint32_t)k + 1u;
  uint32_t npos = npos_total - t.pos_begin;
  if (npos > (uint32_t)db.legacy_tile_pos) npos = (uint32_t)db.legacy_tile_pos;
  const uint32_t nb = npos + (uint32_t)k - 1u; /* bases of this tile */
  const uint32_t nq = npos + (uint32_t)w - 1u; /* l-mers of this tile */

  /* -- load + 2-bit pack: 8 bases per lane, 8-byte aligned loads (or 2 code bytes + 1 validity byte of packed input) -- */
  const uint8_t *g = b.bases + so + t.pos_begin;
  const uint64_t pbase = b.codes ? (uint64_t)b.poff[t.seq] * 32ULL + t.pos_begin : 0ULL; /* base index in the packed planes */
  const uint32_t shift = b.codes ? (uint32_t)(pbase & 7ULL) : (uint32_t)((uintptr_t)g & 7u);
  const uint8_t *ga = g - shift;
  const uint32_t nchunks = (shift + nb + 7u) >> 3;
  uint32_t half = 0, amb8 = 0;
  if (lane < nchunks) {
    if (b.codes) {
      const uint64_t first = (pbase - shift) + 8ULL * lane; /* a multiple of 8 */
      const uint32_t c2 = *reinterpret_cast<const uint16_t *>(b.codes + (first >> 2));
      half = ((c2 & 0xFFu) << 8) | (c2 >> 8);
      amb8 = (~(uint32_t)reinterpret_cast<const uint8_t *>(b.valid)[first >> 3]) & 0xFFu;
    } else {
      uint2 v = __ldg(reinterpret_cast<const uint2 *>(ga) + lane);
      uint32_t a0, a1;
      uint32_t p0 = nh_pack4(v.x, &a0);
      uint32_t p1 = nh_pack4(v.y, &a1);
      half = (p0 << 8) | p1;
      amb8 = a0 | (a1 << 4);
    }
    /* keep only ambiguity bits of bases inside [shift, shift + nb) */
    int lo = (int)shift - (int)(lane * 8u);
    int hi = (int)(shift + nb) - (int)(lane * 8u);
    lo = lo < 0 ? 0 : lo;
    hi = hi > 8 ? 8 : hi;
    uint32_t keep = (lo < 8 && hi > lo) ? (((1u << hi) - 1u) & ~((1u << lo) - 1u)) : 0u;
    amb8 &= keep;
  }
  reinterpret_cast<uint16_t *>(sm.packed)[lane ^ 1u] = (uint16_t)half;
  reinterpret_cast<uint8_t *>(sm.ambits)[lane] = (uint8_t)amb8;
  const bool any_amb = __ballot_sync(FULL_MASK, amb8 != 0) != 0;
  __syncwarp();

  uint64_t prev_lvl[6];
#pragma unroll
  for (int i = 0; i < 6; i++) prev_lvl[i] = NH_NONE64;
  uint64_t carry_last = NH_NONE64; /* last non-ambiguous minimizer seen in this tile */
  uint32_t nonamb_sofar = 0, n_runs = 0;
  const uint32_t lane_lt = (1u << lane) - 1u;
  const uint32_t iters = (nq + 31u) >> 5;

  for (uint32_t it = 0; it < iters; it++) {
    const uint32_t qi = it * 32u + lane; /* l-mer index in the tile */
    const uint32_t tb = shift + qi;      /* its first base in the packed stream */
    bool lmer_ok = qi < nq;
    if (any_amb && lmer_ok) lmer_ok = !any_bits(sm.ambits, tb, (uint32_t)l);
    uint64_t cand = NH_NONE64;
    {
      uint64_t x = nh_extract_lmer(sm.packed, tb, l);
      uint64_t rc = nh_revcomp(x, l, db.revcom_version);
      uint64_t c = min_u64(x, rc) & db.seed_mask;
      c ^= db.toggle;
      if (lmer_ok) cand = c;
    }
    /* sliding-window minimum over the last w l-mers (prefix doubling) */
    uint64_t m = cand;
    uint32_t span = 1;
#pragma unroll
    for (int lev = 0; lev < 5; lev++) {
      if ((int)(span * 2u) <= w) {
        uint64_t o = shfl_carry(m, prev_lvl[lev], span, lane);
        prev_lvl[lev] = m;
        m = min_u64(m, o);
        span *= 2u;
      }
    }
    if ((int)span < w) {
      uint64_t o = shfl_carry(m, prev_lvl[5], (uint32_t)w - span, lane);
      prev_lvl[5] = m;
      m = min_u64(m, o);
    }
    const uint64_t mz = m ^ db.toggle;

    const bool valid = qi >= (uint32_t)(w - 1) && qi < nq;
    const uint32_t pp = qi - (uint32_t)(w - 1); /* k-mer position within the tile */
    bool pos_amb = false;
    if (any_amb && valid)
      pos_amb = any_bits(sm.ambits, tb + (uint32_t)l - (uint32_t)db.amb_span,
                         (uint32_t)db.amb_span);
    const bool nonamb = valid && !pos_amb;

    /* de-duplicate against the previous non-ambiguous position */
    const uint32_t nb_mask = __ballot_sync(FULL_MASK, nonamb);
    const uint32_t lower = nb_mask & lane_lt;
    const uint32_t src = lower ? 31u - (uint32_t)__clz(lower) : lane;
    const uint64_t pm = __shfl_sync(FULL_MASK, mz, src);
    const uint64_t prev_m = lower ? pm : carry_last;
    const bool is_new = nonamb && (mz != prev_m);
    const uint32_t ordinal = nonamb_sofar + __popc(lower);
    const uint32_t new_mask = __ballot_sync(FULL_MASK, is_new);
    if (is_new) {
      uint32_t slot = n_runs + __popc(new_mask & lane_lt);
      sm.st_min[slot] = mz;
      sm.st_start[slot] = (uint8_t)ordinal;
    }
    n_runs += __popc(new_mask);
    if (nb_mask) carry_last = __shfl_sync(FULL_MASK, mz, 31u - (uint32_t)__clz(nb_mask));
    nonamb_sofar += __popc(nb_mask);

    if (b.dbg_pos_min != nullptr && valid) {
      uint64_t o = b.dbg_pos_offsets[t.seq] + t.pos_begin + pp;
      b.dbg_pos_min[o] = mz;
      b.dbg_pos_ambig[o] = pos_amb ? 1 : 0;
    }
  }
  if (lane == 0) sm.st_start[n_runs] = (uint8_t)nonamb_sofar;
  __syncwarp();
  return n_runs;
}

template <int WT>
__global__ void __launch_bounds__(NH_BLOCK_THREADS)
k_minimizers(const NhDbParams db, const NhBatchPtrs b) {
  __shared__ MinWarpSmem s_warp[NH_WARPS_PER_BLOCK];
  __shared__ uint32_t s_runs[2][NH_WARPS_PER_BLOCK];
  __shared__ uint32_t s_base[2];
  const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
  const uint32_t n_tiles = b.counters->n_tiles;
  uint32_t par = 0;
  for (uint32_t group = blockIdx.x; group * NH_WARPS_PER_BLOCK < n_tiles;
       group += gridDim.x, par ^= 1u) {
    const uint32_t tile = group * NH_WARPS_PER_BLOCK + warp;
    uint32_t n_runs = 0;
    if (tile < n_tiles) n_runs = minimizer_tile<WT>(db, b, b.tiles[tile], s_warp[warp], lane);
    if (lane == 0) s_runs[par][warp] = n_runs;
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t tot = 0;
#pragma unroll
      for (int i = 0; i < NH_WARPS_PER_BLOCK; i++) tot += s_runs[par][i];
      s_base[par] = tot ? atomicAdd(&b.counters->n_lookups, tot) : 0u;
    }
    __syncthreads();
    if (tile < n_tiles) {
      uint32_t base = s_base[par];
      for (uint32_t i = 0; i < warp; i++) base += s_runs[par][i];
      const MinWarpSmem &sm = s_warp[warp];
      for (uint32_t r = lane; r < n_runs; r += 32u) {
        b.lk_min[base + r] = sm.st_min[r];
        b.lk_cnt[base + r] = (uint16_t)(sm.st_start[r + 1] - sm.st_start[r]);
      }
      if (lane == 0) {
        NhTileOut o;
        o.lk_off = base;
        o.lk_cnt = n_runs;
        b.tile_out[tile] = o;
      }
    }
    __syncwarp();
  }
}

/* ------------------------------------------------------------------ */
/* stage 2: compact hash table probe — one thread per lookup            */

__device__ __forceinline__ void ld_sector(const uint32_t *p, uint32_t (&c)[8]) {
  /* one 32-byte sector in one request (256-bit global load, sm_100+) */
#ifndef NH_LD_SECTOR_OP
#define NH_LD_SECTOR_OP "ld.global.nc.L1::no_allocate.L2::64B.v8.u32"
#endif
  asm volatile(NH_LD_SECTOR_OP " {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(c[0]), "=r"(c[1]), "=r"(c[2]), "=r"(c[3]), "=r"(c[4]), "=r"(c[5]),
                 "=r"(c[6]), "=r"(c[7])
               : "l"(p));
}

/* the probe chain of compacted key ckey from cell idx on: the value of the first cell that is empty or holds ckey,
 * 0 after a whole table without either.  64-bit throughout, so it walks any distance. */
__device__ __forceinline__ uint32_t cht_walk(const NhDbParams &db, uint64_t idx, uint32_t ckey) {
  uint64_t inspected = 0;
  for (;;) {
    const uint64_t sbase = idx & ~7ULL;
    uint32_t c[8];
    ld_sector(db.cells + sbase, c);
    const int start = (int)(idx & 7ULL);
    const uint64_t rem = db.capacity - sbase;
    const int limit = rem < 8 ? (int)rem : 8;
    int state = -1;
#pragma unroll
    for (int j = 7; j >= 0; j--) {
      const uint32_t val = c[j] & db.value_mask;
      const bool term = (val == 0) || ((c[j] >> db.value_bits) == ckey);
      if (j >= start && j < limit && term) state = (int)val;
    }
    if (state >= 0) return (uint32_t)state;
    inspected += (uint64_t)(limit - start);
    if (inspected >= db.capacity) return 0; /* table without an empty cell */
    idx = sbase + 8;
    if (idx >= db.capacity) idx = 0;
  }
}

__device__ __forceinline__ uint32_t cht_get(const NhDbParams &db, uint64_t key) {
  const uint64_t h = nh_fmix64(key);
  if (db.min_hash && h < db.min_hash) return 0;
  return cht_walk(db, nh_fastmod(h, db.capacity, db.mod_m, db.mod_sh1, db.mod_sh2),
                  (uint32_t)(h >> (32u + db.value_bits)));
}

__global__ void __launch_bounds__(256)
k_probe(const NhDbParams db, const uint64_t *__restrict__ keys, uint32_t *__restrict__ taxa,
        const uint32_t *__restrict__ n_dev, uint32_t n_fixed) {
  const uint32_t n = n_dev ? *n_dev : n_fixed;
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    taxa[i] = cht_get(db, keys[i]);
}

/* ------------------------------------------------------------------ */
/* stage 3: per-unit scoring, confidence walk-up, keep/drop             */

__device__ __forceinline__ uint32_t hash_slot(uint32_t taxon, uint32_t cap_mask) {
  return (taxon * 2654435761u >> 7) & cap_mask;
}

__device__ __forceinline__ bool hc_add(uint32_t *keys, uint32_t *cnts, uint32_t cap_mask,
                                       uint32_t taxon, uint32_t n) {
  uint32_t s = hash_slot(taxon, cap_mask);
  for (uint32_t p = 0; p <= cap_mask; p++) {
    uint32_t old = atomicCAS(&keys[s], 0u, taxon);
    if (old == 0u || old == taxon) {
      atomicAdd(&cnts[s], n);
      return true;
    }
    s = (s + 1u) & cap_mask;
  }
  return false;
}

__device__ __forceinline__ uint32_t hc_get(const uint32_t *keys, const uint32_t *cnts,
                                           uint32_t cap_mask, uint32_t taxon) {
  if (!taxon) return 0;
  uint32_t s = hash_slot(taxon, cap_mask);
  for (uint32_t p = 0; p <= cap_mask; p++) {
    uint32_t kx = keys[s];
    if (kx == taxon) return cnts[s];
    if (kx == 0u) return 0;
    s = (s + 1u) & cap_mask;
  }
  return 0;
}

__device__ __forceinline__ bool is_a_ancestor_of_b(const uint32_t *parent, uint32_t a,
                                                   uint32_t b) {
  if (!a || !b) return false;
  while (b > a) b = parent[b];
  return b == a;
}

__device__ __forceinline__ uint32_t lca(const uint32_t *parent, uint32_t a, uint32_t b) {
  if (!a || !b) return a ? a : b;
  while (a != b) {
    if (a > b)
      a = parent[a];
    else
      b = parent[b];
  }
  return a;
}

/* ---- a unit's taxon -> k-mer count table (shared memory, one warp), filled one of three ways ---- */

struct UnitAcc {
  uint32_t total_kmers;
  int groups; /* per lane; summed over the warp by resolve_unit */
  bool ok;    /* false: the table overflowed */
};

__device__ __forceinline__ void acc_begin(uint32_t *keys, uint32_t *cnts, uint32_t cap_mask, uint32_t lane) {
  for (uint32_t s = lane; s <= cap_mask; s += 32u) {
    keys[s] = 0;
    cnts[s] = 0;
  }
  __syncwarp();
}

__device__ __forceinline__ uint32_t unit_total_kmers(const NhDbParams &db, const NhBatchPtrs &b, uint32_t u) {
  const uint32_t nm = b.paired ? 2u : 1u;
  uint32_t total = 0;
  for (uint32_t mate = 0; mate < nm; mate++) {
    const uint32_t s = u * nm + mate;
    const uint64_t len = b.offsets[s + 1] - b.offsets[s];
    if (len >= (uint64_t)db.k) total += (uint32_t)(len - (uint64_t)db.k + 1);
  }
  return total;
}

/* streaming kernel, unit spread over several warps: every tile left its own small table and a
 * summary; lanes take tiles in parallel */
__device__ UnitAcc acc_from_tile_tables(const NhDbParams &db, const NhBatchPtrs &b, uint32_t *keys, uint32_t *cnts,
                                        uint32_t cap_mask, uint32_t u, uint32_t lane) {
  UnitAcc a;
  a.total_kmers = unit_total_kmers(db, b, u);
  a.groups = 0;
  a.ok = true;
  const uint32_t nm = b.paired ? 2u : 1u;
  for (uint32_t mate = 0; mate < nm; mate++) {
    const uint32_t s = u * nm + mate;
    const uint32_t t0 = b.tile_base[s], t1 = b.tile_base[s + 1];
    for (uint32_t tile = t0 + lane; tile < t1; tile += 32u) {
      const NhTileSum ts = b.tile_sum[tile];
      a.groups += (int)ts.groups;
      if (ts.flags & NH_TILE_OVERFLOW) {
        a.ok = false; /* k_score_big scans the unit again */
      } else {
        const NhTileTab tt = b.tile_tab[tile];
#pragma unroll
        for (int j = 0; j < NH_LANE_TAXA; j++)
          if (tt.keys[j]) a.ok &= hc_add(keys, cnts, cap_mask, tt.keys[j], tt.cnts[j]);
      }
      /* a tile starts with a fresh lookup even when its first minimizer equals the last one of
       * the tile before: upstream counts that as one group (last_minimizer lives per mate) */
      if (tile > t0 && (ts.flags & NH_TILE_HAS) && (ts.flags & NH_TILE_FIRST_HIT)) {
        uint32_t p = tile;
        while (p > t0 && !(b.tile_sum[p - 1u].flags & NH_TILE_HAS)) p--;
        if (p > t0 && b.tile_sum[p - 1u].last_min == ts.first_min) a.groups--;
      }
    }
  }
  return a;
}

/* warp-per-tile kernels: every lookup sits in lk_min / lk_cnt / lk_taxon */
__device__ UnitAcc acc_from_lookups(const NhDbParams &db, const NhBatchPtrs &b, uint32_t *keys, uint32_t *cnts,
                                    uint32_t cap_mask, uint32_t u, uint32_t lane) {
  UnitAcc a;
  a.total_kmers = unit_total_kmers(db, b, u);
  a.groups = 0;
  a.ok = true;
  const uint32_t nm = b.paired ? 2u : 1u;
  for (uint32_t mate = 0; mate < nm; mate++) {
    const uint32_t s = u * nm + mate;
    const uint32_t t0 = b.tile_base[s], t1 = b.tile_base[s + 1];
    uint64_t prev_last = NH_NONE64; /* ClassifySequence resets last_minimizer per mate */
    for (uint32_t tile = t0; tile < t1; tile++) {
      const NhTileOut to = b.tile_out[tile];
      for (uint32_t j = lane; j < to.lk_cnt; j += 32u) {
        const uint32_t tx = b.lk_taxon[to.lk_off + j];
        if (tx) {
          a.groups++;
          a.ok &= hc_add(keys, cnts, cap_mask, tx, b.lk_cnt[to.lk_off + j]);
        }
      }
      if (to.lk_cnt && t1 - t0 > 1u) {
        if (lane == 0 && tile > t0 && b.lk_min[to.lk_off] == prev_last && b.lk_taxon[to.lk_off] != 0u) a.groups--;
        prev_last = b.lk_min[to.lk_off + to.lk_cnt - 1u];
      }
    }
  }
  return a;
}

/* the unit again, from its bases: warp-per-tile minimizers + one table walk per lookup.  Needs no
 * scratch of the batch, so the streaming kernel never has to park lookups in global memory for
 * the rare unit that overflows its in-warp table. */
__device__ UnitAcc acc_rescan(const NhDbParams &db, const NhBatchPtrs &b, uint32_t *keys, uint32_t *cnts,
                              uint32_t cap_mask, uint32_t u, uint32_t lane, MinWarpSmem &msm) {
  UnitAcc a;
  a.total_kmers = unit_total_kmers(db, b, u);
  a.groups = 0;
  a.ok = true;
  const uint32_t nm = b.paired ? 2u : 1u;
  for (uint32_t mate = 0; mate < nm; mate++) {
    const uint32_t s = u * nm + mate;
    const uint64_t len = b.offsets[s + 1] - b.offsets[s];
    if (len < (uint64_t)db.k) continue;
    const uint32_t npos = (uint32_t)(len - (uint64_t)db.k + 1);
    uint64_t prev_last = NH_NONE64;
    for (uint32_t pos0 = 0; pos0 < npos; pos0 += (uint32_t)db.legacy_tile_pos) {
      NhTile t;
      t.seq = s;
      t.pos_begin = pos0;
      t.slot = 0;
      t.role = 0;
      const uint32_t n_runs = db.w == 5 ? minimizer_tile<5>(db, b, t, msm, lane) : minimizer_tile<0>(db, b, t, msm, lane);
      for (uint32_t j = lane; j < n_runs; j += 32u) {
        const uint32_t tx = cht_get(db, msm.st_min[j]);
        if (tx) {
          a.groups++;
          a.ok &= hc_add(keys, cnts, cap_mask, tx, (uint32_t)(msm.st_start[j + 1] - msm.st_start[j]));
        }
      }
      if (n_runs) {
        if (lane == 0 && pos0 > 0 && msm.st_min[0] == prev_last && cht_get(db, msm.st_min[0]) != 0u) a.groups--;
        prev_last = msm.st_min[n_runs - 1u];
      }
      __syncwarp(); /* the staging area is reused by the next tile */
    }
  }
  return a;
}

/* ResolveTree + min-hit-groups + keep/drop for the unit whose table is in keys/cnts.
 * Returns false (and writes nothing) if the table had overflowed. */
__device__ bool resolve_unit(const NhDbParams &db, const NhBatchPtrs &b, const NhScoreParams &sp,
                             const uint32_t *parent, const uint32_t *keys, const uint32_t *cnts,
                             uint32_t cap_mask, uint32_t u, uint32_t lane, UnitAcc a, uint32_t *classified,
                             uint32_t *kept) {
  __syncwarp();
  const int groups = (int)__reduce_add_sync(FULL_MASK, (uint32_t)a.groups);
  if (!__all_sync(FULL_MASK, a.ok)) return false;
  const uint32_t total_kmers = a.total_kmers;

  /* root-to-leaf score of every hit taxon, ties fold to the LCA */
  uint32_t best_s = 0, best_t = 0;
  for (uint32_t s = lane; s <= cap_mask; s += 32u) {
    const uint32_t tx = keys[s];
    if (!tx) continue;
    uint32_t score = 0;
    for (uint32_t an = tx; an; an = parent[an]) score += hc_get(keys, cnts, cap_mask, an);
    if (score > best_s) {
      best_s = score;
      best_t = tx;
    } else if (score == best_s) {
      best_t = lca(parent, best_t, tx);
    }
  }
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) {
    const uint32_t os = __shfl_xor_sync(FULL_MASK, best_s, d);
    const uint32_t ot = __shfl_xor_sync(FULL_MASK, best_t, d);
    if (os > best_s) {
      best_s = os;
      best_t = ot;
    } else if (os == best_s) {
      best_t = lca(parent, best_t, ot);
    }
  }
  uint32_t max_taxon = best_t;
  uint32_t max_score = hc_get(keys, cnts, cap_mask, max_taxon);
  const uint32_t required = (uint32_t)ceil(__dmul_rn(sp.confidence, (double)total_kmers));
  while (max_taxon && max_score < required) {
    uint32_t part = 0;
    for (uint32_t s = lane; s <= cap_mask; s += 32u) {
      const uint32_t tx = keys[s];
      if (tx && is_a_ancestor_of_b(parent, max_taxon, tx)) part += cnts[s];
    }
    max_score = warp_sum_u32(part);
    if (max_score >= required) break;
    max_taxon = parent[max_taxon];
  }
  uint32_t call = max_taxon;
  if (call && groups < sp.min_hit_groups) call = 0;
  if (lane == 0) {
    const uint32_t is_cls = call != 0u;
    const uint32_t keep = sp.keep_human ? is_cls : !is_cls;
    if (b.out_call) b.out_call[u] = call ? db.ext_id[call] : 0u;
    if (b.out_keep) b.out_keep[u] = (uint8_t)keep;
    if (b.dbg_call) b.dbg_call[u] = call;
    if (b.dbg_total_kmers) b.dbg_total_kmers[u] = total_kmers;
    if (b.dbg_hit_groups) b.dbg_hit_groups[u] = (uint32_t)groups;
    *classified += is_cls;
    *kept += keep;
  }
  __syncwarp();
  return true;
}

template <bool SMEM_PARENT>
__global__ void __launch_bounds__(NH_BLOCK_THREADS)
k_score(const NhDbParams db, const NhBatchPtrs b, const NhScoreParams sp) {
  extern __shared__ uint32_t s_dyn[];
  uint32_t *s_parent = s_dyn;
  const uint32_t parent_words = SMEM_PARENT ? db.node_count : 0u;
  uint32_t *s_hash = s_dyn + parent_words;
  if (SMEM_PARENT) {
    for (uint32_t i = threadIdx.x; i < db.node_count; i += blockDim.x) s_parent[i] = db.parent[i];
    __syncthreads();
  }
  const uint32_t *parent = SMEM_PARENT ? s_parent : db.parent;
  const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
  uint32_t *keys = s_hash + warp * 2u * NH_WARP_HASH_SLOTS;
  uint32_t *cnts = keys + NH_WARP_HASH_SLOTS;
  uint32_t classified = 0, kept = 0;
  const uint32_t wstride = gridDim.x * NH_WARPS_PER_BLOCK;
  /* streaming path: only the units k_plan_fill deferred; warp-per-tile path: every unit */
  const uint32_t n_todo = b.deferred_units ? b.counters->n_deferred : b.n_units;
  for (uint32_t i = blockIdx.x * NH_WARPS_PER_BLOCK + warp; i < n_todo; i += wstride) {
    const uint32_t u = b.deferred_units ? b.deferred_units[i] : i;
    acc_begin(keys, cnts, NH_WARP_HASH_SLOTS - 1u, lane);
    const UnitAcc a = b.tile_tab != nullptr ? acc_from_tile_tables(db, b, keys, cnts, NH_WARP_HASH_SLOTS - 1u, u, lane)
                                            : acc_from_lookups(db, b, keys, cnts, NH_WARP_HASH_SLOTS - 1u, u, lane);
    if (!resolve_unit(db, b, sp, parent, keys, cnts, NH_WARP_HASH_SLOTS - 1u, u, lane, a, &classified, &kept)) {
      if (lane == 0) b.overflow_units[atomicAdd(&b.counters->n_overflow, 1u)] = u;
    }
  }
  if (lane == 0) {
    if (classified) atomicAdd(&b.counters->n_classified, classified);
    if (kept) atomicAdd(&b.counters->n_kept, kept);
  }
}

/* overflow pass: units with more distinct taxa than the in-warp tables hold are classified again
 * from their bases, one warp per block with a 16K-slot table */
__global__ void __launch_bounds__(32)
k_score_big(const NhDbParams db, const NhBatchPtrs b, const NhScoreParams sp) {
  extern __shared__ uint32_t s_dyn[];
  __shared__ MinWarpSmem s_min;
  uint32_t *keys = s_dyn;
  uint32_t *cnts = s_dyn + NH_BIG_HASH_SLOTS;
  const uint32_t lane = lane_id();
  const uint32_t n = b.counters->n_overflow;
  uint32_t classified = 0, kept = 0;
  for (uint32_t i = blockIdx.x; i < n; i += gridDim.x) {
    const uint32_t u = b.overflow_units[i];
    acc_begin(keys, cnts, NH_BIG_HASH_SLOTS - 1u, lane);
    const UnitAcc a = acc_rescan(db, b, keys, cnts, NH_BIG_HASH_SLOTS - 1u, u, lane, s_min);
    if (!resolve_unit(db, b, sp, db.parent, keys, cnts, NH_BIG_HASH_SLOTS - 1u, u, lane, a, &classified, &kept)) {
      /* more than 16K distinct taxa in ONE read: the device's table in global memory can hold every
       * node of the taxonomy; units this extreme take turns on it */
      if (db.huge_slots == 0u) {
        if (lane == 0) atomicExch(&b.counters->error, 1u); /* cannot happen: node_count fits the shared table */
        continue;
      }
      uint32_t *gkeys = db.huge_table, *gcnts = db.huge_table + db.huge_slots, *lock = db.huge_table + 2u * db.huge_slots;
      if (lane == 0)
        while (atomicCAS(lock, 0u, 1u) != 0u) __nanosleep(200);
      __syncwarp();
      __threadfence();
      acc_begin(gkeys, gcnts, db.huge_slots - 1u, lane);
      const UnitAcc ga = acc_rescan(db, b, gkeys, gcnts, db.huge_slots - 1u, u, lane, s_min);
      const bool ok = resolve_unit(db, b, sp, db.parent, gkeys, gcnts, db.huge_slots - 1u, u, lane, ga, &classified, &kept);
      __threadfence();
      __syncwarp();
      if (lane == 0) {
        atomicExch(lock, 0u);
        if (!ok) atomicExch(&b.counters->error, 1u);
      }
    }
  }
  if (lane == 0) {
    if (classified) atomicAdd(&b.counters->n_classified, classified);
    if (kept) atomicAdd(&b.counters->n_kept, kept);
  }
}

/* ------------------------------------------------------------------ */
/* the streaming kernel: scan -> probe -> score, one warp per group of 32 tiles */
/*
 * Every lane scans ITS OWN tile base by base: rolling forward and reverse-
 * complement l-mers, canonical / spaced seed / toggle, window minimum over a
 * register ring, run-length de-duplication (about a third of the instructions
 * of the warp-per-tile kernel, which recomputes every l-mer).  A closed run
 * goes straight into a small queue in shared memory; whenever 32 lookups are
 * waiting the warp runs a PROBE ROUND: it finishes the 32 lookups whose table
 * sectors were requested in the previous round (scan the sector, fold the hit
 * into the owning unit's taxon table, or queue the chain's continuation into
 * the next sector), hashes the next 32 and requests their sectors, and goes
 * back to scanning.  Nothing the warp waits for sits on a load scoreboard:
 * bases and sectors arrive by cp.async into shared memory and complete on
 * mbarriers, because ptxas drains every scoreboard at the first potentially
 * divergent branch after a load (measured: profiles/r02_summary.md), which
 * had turned "look at the sector one round later" into "wait for it now".
 * Units whose tiles all sit in this group are scored here (ResolveTree on the
 * leader lane); tiles of other units leave their table and a summary for
 * k_score.  Only the window width W is a template parameter (kraken2's
 * default k=35, l=31 gives W=5); other databases take the warp-per-tile kernels.
 */

#ifndef NH_BCHUNK_WORDS
#define NH_BCHUNK_WORDS 8u                            /* base words (4 bases each) per lane and chunk */
#endif
#define NH_BCHUNK_STRIDE (NH_BCHUNK_WORDS * 4u + 16u) /* + up to 12 bytes of 16-byte misalignment */
#ifndef NH_PQ_SLOTS
#define NH_PQ_SLOTS 128u
#endif
#define NH_META_FIRST 0x8000u /* the first lookup of its tile */
#define NH_AUX_NONE 0xFFFFFFFFu
#ifndef NH_FILTER_RECENT
#define NH_FILTER_RECENT 4u
#endif
#define NH_AUX_FILTER 0x80000000u /* FILTER kernels: the request in flight is a filter record, not a table sector */

template <bool EMIT>
struct __align__(16) StreamWarpSmem {
  uint4 pq[NH_PQ_SLOTS];                 /* closed runs waiting to be probed (ring): key lo, key hi, meta, lookup slot;
                                          * meta = tile's lane | k-mer count << 5 | NH_META_FIRST */
  uint32_t q_unit[32];                   /* probe chains that continue into the next sector (at most one per lane) */
  uint32_t q_ckey[32];
  uint32_t q_aux[32];                    /* pq_meta | sectors visited << 16 */
  uint64_t first_min[32], last_min[32];  /* first / last distinct minimizer of each lane's tile */
  uint32_t keys[NH_LANE_TAXA * 32];      /* taxon tables, [slot][owner lane] */
  uint32_t cnts[NH_LANE_TAXA * 32];
  uint32_t groups[32];                   /* minimizer_hit_groups per owner lane */
  uint8_t owner[32];                     /* per tile: the lane whose table takes its hits */
  uint32_t overflow;                     /* bit per owner lane: table overflowed */
  uint32_t first_hit;                    /* bit per lane: the tile's first lookup hit */
  /* staging: every lane's next NH_BCHUNK_WORDS base words arrive by 16-byte cp.async copies into its
   * own 48-byte window (double-buffered), every lane's table sector into sect[] */
  uint64_t bbar[2], sbar;
  __align__(16) uint8_t bchunk[2][32 * NH_BCHUNK_STRIDE];
  __align__(16) uint32_t sect[32 * 8];
  uint32_t q_slot[EMIT ? 32 : 1]; /* per-read output only: where the lookup's taxon goes */
  uint8_t recent[32];             /* FILTER kernels, per tile: lookups still to send straight to the table after a hit */
};

/* 3 blocks of 8 warps per SM (up to 85 registers): the overlap of table latency and scan happens
 * inside the warp, so registers are worth more than resident warps */
#ifndef NH_STREAM_MIN_BLOCKS
#define NH_STREAM_MIN_BLOCKS 3
#endif
/* NH_STREAM_MIN_BLOCKS blocks of NH_WARPS_PER_BLOCK warps must fit the SM's 227 KB next to the staged
 * parent array of a small taxonomy and the 1 KB the system reserves per block */
static_assert((sizeof(StreamWarpSmem<false>) * NH_WARPS_PER_BLOCK + 1024 + 512) * NH_STREAM_MIN_BLOCKS <= 227 * 1024,
              "k_stream_classify would no longer fit its blocks per SM");

template <typename SM>
__device__ __forceinline__ uint32_t lane_tab_get(const SM &sm, uint32_t lane, uint32_t n, uint32_t taxon) {
  for (uint32_t i = 0; i < n; i++)
    if (sm.keys[i * 32u + lane] == taxon) return sm.cnts[i * 32u + lane];
  return 0;
}

__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
/* 16 bytes global -> shared without a register or a load scoreboard in between (LDGSTS, L2 only) */
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
/* 8 and 4 bytes (packed input: one unit's codes and validity word) */
__device__ __forceinline__ void cp_async8(uint32_t dst, const void *src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(uint32_t dst, const void *src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
/* the same with only the first n_src bytes taken from global memory and the rest zero-filled */
__device__ __forceinline__ void cp_async16_zfill(uint32_t dst, const void *src, uint32_t n_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(n_src) : "memory");
}
/* the same for a table sector half: a miss fills 64 bytes of L2, not the default 128 */
__device__ __forceinline__ void cp_async16_l2_64(uint32_t dst, const void *src) {
  asm volatile("cp.async.cg.shared.global.L2::64B [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
/* the mbarrier gets this thread's arrival once all its earlier cp.async copies have landed */
__device__ __forceinline__ void cp_async_arrive(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "NH_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra NH_DONE;\n"
      "bra NH_WAIT;\n"
      "NH_DONE:\n"
      "}" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}


/* ------------------------------------------------------------------ */
/* The miss filter: one 32-byte record per block of 32 table cells, built when the database is opened.
 * word 0: occupancy of the block's cells (cells past the table's end count as occupied);
 * words 1-7: a partitioned Bloom filter of the compacted keys stored IN the block — one bit in words 1-2,
 * one in 3-4, one in 5-6, one in word 7 (22 keys per block at load 0.7: about 1.3 % false positives).
 * A probe chain that starts at cell `off` of the block and whose key is in none of the block's cells ends at
 * the block's first free cell at or after `off`: if there is one, the lookup is a MISS after one 32-byte
 * request instead of the 1.65 sectors a missing key walks in the table; if there is none the chain runs
 * into the next block, whose record is asked next.  A positive answer sends the lookup to the table at the
 * cell it had reached.  The filter never changes a result; who asks it is decided per unit (NhScoreParams). */
__device__ __forceinline__ uint32_t nh_filter_hash(uint32_t ckey) {
  uint32_t h = ckey * 0x9E3779B1u;
  h ^= h >> 15;
  h *= 0x85EBCA77u;
  h ^= h >> 13;
  return h;
}

__global__ void __launch_bounds__(256)
k_filter_build(const uint32_t *__restrict__ cells, uint64_t capacity, uint32_t value_bits, uint32_t value_mask,
               uint32_t *__restrict__ filter, uint32_t n_blocks) {
  const uint32_t blk = blockIdx.x * blockDim.x + threadIdx.x;
  if (blk >= n_blocks) return;
  uint32_t rec[8];
#pragma unroll
  for (int i = 0; i < 8; i++) rec[i] = 0;
  const uint64_t base = (uint64_t)blk * 32ULL;
#pragma unroll 1
  for (uint32_t q = 0; q < 8; q++) {
    uint32_t c[4] = {0u, 0u, 0u, 0u};
    if (base + q * 4u + 4u <= capacity) {
      const uint4 v = __ldg(reinterpret_cast<const uint4 *>(cells + base) + q);
      c[0] = v.x; c[1] = v.y; c[2] = v.z; c[3] = v.w;
    } else { /* the table's last cells: an adopted array need not be padded */
      for (uint32_t j = 0; j < 4; j++)
        if (base + q * 4u + j < capacity) c[j] = __ldg(cells + base + q * 4u + j);
    }
#pragma unroll
    for (uint32_t j = 0; j < 4; j++) {
      const uint32_t cell = q * 4u + j;
      if (base + cell >= capacity) {
        rec[0] |= 1u << cell;
      } else if (c[j] & value_mask) {
        rec[0] |= 1u << cell;
        const uint32_t h = nh_filter_hash(c[j] >> value_bits);
        const uint32_t i0 = h & 63u, i1 = (h >> 6) & 63u, i2 = (h >> 12) & 63u, i3 = (h >> 18) & 31u;
        rec[1 + (i0 >> 5)] |= 1u << (i0 & 31u);
        rec[3 + (i1 >> 5)] |= 1u << (i1 & 31u);
        rec[5 + (i2 >> 5)] |= 1u << (i2 & 31u);
        rec[7] |= 1u << i3;
      }
    }
  }
  uint4 *out = reinterpret_cast<uint4 *>(filter + (uint64_t)blk * 8ULL);
  out[0] = make_uint4(rec[0], rec[1], rec[2], rec[3]);
  out[1] = make_uint4(rec[4], rec[5], rec[6], rec[7]);
}

#ifndef NH_STREAM_CHECK_MASK
#define NH_STREAM_CHECK_MASK 1 /* probe check after bases with (j & mask) == mask: 1 -> every 2nd base */
#endif

/* KL = 1: kraken2's default k = 35, l = 31 compiled in (shift counts and thresholds become
 * immediates); KL = 0: any k, l with k - l + 1 = W, read from the database.
 * PACKED: the batch came as 2-bit codes + validity bits (nh_classify_batch_packed), every sequence
 * starting on a unit of 32 bases; tiles then start on units too (tile_pos is a multiple of 32). */
/* FILTER: 0 no miss filter, 1 / 2 / 3 the policy of NhScoreParams::filter_mode compiled in */
template <int W, int KL, bool DBG, bool REV0, bool EMIT, bool PACKED, int FILTER>
__global__ void __launch_bounds__(NH_BLOCK_THREADS, NH_STREAM_MIN_BLOCKS)
k_stream_classify(const NhDbParams db, const NhBatchPtrs b, const NhScoreParams sp) {
  static_assert(W == 5, "the scan consumes one 4-byte word per ring rotation");
  static_assert(NH_PQ_SLOTS >= 31u + 32u * (NH_STREAM_CHECK_MASK + 1u), "runs closed between two probe checks must fit the ring");
  static_assert((NH_PQ_SLOTS & (NH_PQ_SLOTS - 1u)) == 0 && (NH_BCHUNK_WORDS & (NH_BCHUNK_WORDS - 1u)) == 0, "powers of two");
  typedef StreamWarpSmem<EMIT> Smem;
  extern __shared__ __align__(16) uint32_t s_dyn[];
  uint32_t *s_parent = s_dyn;
  const bool smem_parent = db.node_count <= NH_SMEM_PARENT_MAX;
  const uint32_t parent_words = smem_parent ? db.node_count : 0u;
  Smem *s_warps = reinterpret_cast<Smem *>(s_dyn + ((parent_words + 3u) & ~3u));
  if (smem_parent) {
    for (uint32_t i = threadIdx.x; i < db.node_count; i += blockDim.x) s_parent[i] = db.parent[i];
    __syncthreads();
  }
  const uint32_t *parent = smem_parent ? s_parent : db.parent;
  const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
  const uint32_t lane_lt = (1u << lane) - 1u;
  Smem &sm = s_warps[warp];
  const uint32_t n_tiles = b.counters->n_tiles;
  const int k = KL ? 35 : db.k, l = KL ? 31 : db.l;
  const uint32_t amb_span = KL ? 34u : (uint32_t)db.amb_span;
  const uint64_t lmask = (1ULL << (2 * l)) - 1ULL;
  const uint32_t rc_shift = 2u * (uint32_t)(l - 1);
  const uint32_t n_sectors = (uint32_t)((db.capacity + 7ULL) >> 3); /* nh_fused_supported: capacity < 2^35 */
  const uint32_t last_sector = n_sectors - 1u;
  /* cells of the last sector that exist (the allocation is zero-padded past the table's end) */
  const uint32_t last_range = (db.capacity & 7ULL) ? (1u << (uint32_t)(db.capacity & 7ULL)) - 1u : 0xFFu;
  /* The visit count of a chain lives in 16 bits of its state (15 in the FILTER kernels, which keep bit 31 for
   * NH_AUX_FILTER and the cell a continuation starts at in the top value_bits (>= 5, nh_db_build_filter) bits of
   * its compacted key).  A chain that reaches max_visits is not a miss: every unit of the group is marked
   * overflowed, like a unit with more taxa than a lane table holds, and k_score_big classifies them again with
   * cht_get, which walks any distance and still ends on a table without any empty cell (one constant store keeps
   * the probe round's code as it was).  EMIT kernels also need the lookup's own taxon for
   * the per-read output, so there the lane walks the rest of the chain itself with cht_walk.  Only tables built at a
   * load close to 1 have runs that long (about 262 K cells when walking sectors in the FILTER kernels, 524 K
   * otherwise), and the common branch gains nothing. */
  const uint32_t max_visits = FILTER ? (n_sectors + 1u < 0x7FFEu ? n_sectors + 1u : 0x7FFEu) : (n_sectors + 1u < 0xFFFFu ? n_sectors + 1u : 0xFFFFu);
  const uint32_t last_block = FILTER ? sp.n_filter_blocks - 1u : 0u;
  const uint32_t ck_bits = 32u - db.value_bits;
  uint32_t tot_lookups = 0, tot_sectors = 0, tot_classified = 0, tot_kept = 0;

  const uint32_t bar0 = smem_addr(&sm.bbar[0]);
  const uint32_t win0 = smem_addr(&sm.bchunk[0][lane * NH_BCHUNK_STRIDE]);
  const uint32_t sbar = smem_addr(&sm.sbar);
  const uint32_t sect0 = smem_addr(&sm.sect[0]);
  uint32_t bar_par = 0;  /* bit per base buffer: parity of the phase its next chunk completes (warp-uniform) */
  uint32_t sect_par = 0; /* parity of the phase the sectors in flight complete */
  if (lane == 0) {
    mbar_init(bar0, 32u); /* every lane arrives once per chunk / round, when its copies have landed */
    mbar_init(bar0 + 8u, 32u);
    mbar_init(sbar, 32u);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncwarp();

  /* groups of 32 tiles are handed out through a counter: warps that draw short tiles take more */
  for (;;) {
    uint32_t group = 0;
    if (lane == 0) group = atomicAdd(&b.counters->next_group, 1u);
    group = __shfl_sync(FULL_MASK, group, 0);
    if ((uint64_t)group * 32ULL >= n_tiles) break;
    const uint32_t tile = group * 32u + lane;
    const bool have = tile < n_tiles;
    NhTile t;
    t.seq = 0; t.pos_begin = 0; t.slot = 0; t.role = NH_ROLE_DEFERRED;
    if (have) t = b.tiles[tile];
    const uint32_t kind = NH_ROLE_KIND(t.role);
    /* a MEMBER tile folds its hits into its unit's LEADER lane; every other tile into its own table
     * (tiles of deferred units hand theirs to k_score through tile_tab) */
    const uint32_t owner = kind == NH_ROLE_MEMBER ? lane - NH_ROLE_DELTA(t.role) : lane;
#pragma unroll
    for (int i = 0; i < NH_LANE_TAXA; i++) {
      sm.keys[i * 32 + lane] = 0;
      sm.cnts[i * 32 + lane] = 0;
    }
    sm.groups[lane] = 0;
    if (FILTER == 3) sm.recent[lane] = 0;
    sm.owner[lane] = (uint8_t)owner;
    if (lane == 0) {
      sm.overflow = 0;
      sm.first_hit = 0;
    }
    __syncwarp();

    /* warp-uniform queue state */
    uint32_t pq_head = 0, pq_n = 0, cq_n = 0;
    uint32_t n_popped = 0; /* fresh lookups handed to the probe = distinct-consecutive minimizers of the group */
    uint32_t n_conts = 0;  /* chain continuations: a second, third ... sector of a lookup */
    /* the lookup this lane has in flight: its sector lands in sm.sect, looked at in the next round */
    uint32_t f_unit = 0, f_ckey = 0, f_slot = 0, f_aux = NH_AUX_NONE, f_start = 0;
    bool any_inflight = false; /* warp-uniform */

    /* one probe round: finish the lookups in flight, then put up to 32 waiting ones in flight */
    auto probe_round = [&]() {
      /* ---- 1. look at the sectors requested last round ---- */
      if (any_inflight) {
        const bool active = f_aux != NH_AUX_NONE;
        bool done = false;
        uint32_t result = 0;
        mbar_wait(sbar, sect_par);
        sect_par ^= 1u;
        if (active) {
          uint32_t c[8];
          {
            const uint4 lo = *reinterpret_cast<const uint4 *>(&sm.sect[lane * 8u]);
            const uint4 hi = *reinterpret_cast<const uint4 *>(&sm.sect[lane * 8u + 4u]);
            c[0] = lo.x; c[1] = lo.y; c[2] = lo.z; c[3] = lo.w;
            c[4] = hi.x; c[5] = hi.y; c[6] = hi.z; c[7] = hi.w;
          }
          if (FILTER) {
            const uint32_t ck = f_ckey & ((1u << ck_bits) - 1u);
            const uint32_t st = f_ckey >> ck_bits; /* cell of the block / sector the chain enters at */
            const uint32_t visits = ((f_aux >> 16) & 0x7FFFu) + 1u;
            f_ckey = ck;
            if (f_aux & NH_AUX_FILTER) {
              /* the record of block f_unit */
              const uint32_t h = nh_filter_hash(ck);
              const uint32_t w0 = (h & 32u) ? c[2] : c[1], w1 = (h & (32u << 6)) ? c[4] : c[3], w2 = (h & (32u << 12)) ? c[6] : c[5];
              const bool maybe = (((w0 >> (h & 31u)) & (w1 >> ((h >> 6) & 31u)) & (w2 >> ((h >> 12) & 31u)) & (c[7] >> ((h >> 18) & 31u))) & 1u) != 0u;
              const uint32_t free_cells = ~c[0] & (0xFFFFFFFFu << st);
              if (!maybe && free_cells != 0u) {
                done = true; /* the key is not in the block and the chain ends in it: a miss */
              } else if (visits >= max_visits) {
                done = true;
                atomicOr(&sm.overflow, FULL_MASK); /* every unit of the group: k_score_big walks the rest */
              } else if (maybe) { /* to the table, at the cell the chain has reached */
                f_aux = (f_aux & 0xFFFFu) | (visits << 16);
                f_unit = f_unit * 4u + (st >> 3);
                f_ckey = ck | ((st & 7u) << ck_bits);
              } else { /* every cell from st on is taken by other keys: the next block */
                f_aux = (f_aux & (NH_AUX_FILTER | 0xFFFFu)) | (visits << 16);
                f_unit = f_unit == last_block ? 0u : f_unit + 1u;
              }
            } else {
              uint32_t range = 0xFFu << st;
              if (f_unit == last_sector) range &= last_range;
              int state = -1;
#pragma unroll
              for (int j = 7; j >= 0; j--) {
                const uint32_t val = c[j] & db.value_mask;
                const bool term = (val == 0u) || ((c[j] >> db.value_bits) == ck);
                if (term && ((range >> j) & 1u)) state = (int)val;
              }
              if (state >= 0) {
                done = true;
                result = (uint32_t)state;
              } else if (visits >= max_visits) {
                done = true;
                atomicOr(&sm.overflow, FULL_MASK); /* every unit of the group: k_score_big walks the rest */
              } else {
                f_aux = (f_aux & 0xFFFFu) | (visits << 16);
                f_unit = f_unit == last_sector ? 0u : f_unit + 1u;
              }
            }
          } else {
          uint32_t range = 0xFFu << f_start;
          if (f_unit == last_sector) range &= last_range;
          int state = -1;
#pragma unroll
          for (int j = 7; j >= 0; j--) {
            const uint32_t val = c[j] & db.value_mask;
            const bool term = (val == 0u) || ((c[j] >> db.value_bits) == f_ckey);
            if (term && ((range >> j) & 1u)) state = (int)val;
          }
          if (state >= 0) {
            done = true;
            result = (uint32_t)state;
          } else {
            const uint32_t visits = (f_aux >> 16) + 1u;
            if (visits >= max_visits) {
              done = true;
              if (EMIT) result = cht_walk(db, (uint64_t)f_unit * 8ULL + f_start, f_ckey);
              else atomicOr(&sm.overflow, FULL_MASK); /* every unit of the group: k_score_big walks the rest */
            } else {
              f_aux = (f_aux & 0xFFFFu) | (visits << 16);
              f_unit = f_unit == last_sector ? 0u : f_unit + 1u;
            }
          }
          }
        }
        const bool cont = active && !done;
        const uint32_t cmask = __ballot_sync(FULL_MASK, cont);
        if (cont) {
          const uint32_t pos = cq_n + __popc(cmask & lane_lt);
          sm.q_unit[pos] = f_unit;
          sm.q_ckey[pos] = f_ckey;
          sm.q_aux[pos] = f_aux;
          if (EMIT) sm.q_slot[pos] = f_slot;
        }
        cq_n += __popc(cmask);
        if (active && done) {
          const uint32_t tile_lane = f_aux & 31u;
          if (EMIT) b.lk_taxon[f_slot] = result;
          if (FILTER == 3) {
            /* hits come in bursts (an error-free stretch of a read): after a hit the tile's next NH_FILTER_RECENT
             * lookups go straight to the table, after that many misses in a row it asks the filter again.
             * Plain loads and stores: a lost update only changes who asks, never a result */
            const uint32_t r = sm.recent[tile_lane];
            if (result) sm.recent[tile_lane] = NH_FILTER_RECENT;
            else if (r) sm.recent[tile_lane] = (uint8_t)(r - 1u);
          }
          if (result) {
            const uint32_t own = sm.owner[tile_lane];
            const uint32_t n = (f_aux >> 5) & 0x3FFu;
            if (f_aux & NH_META_FIRST) atomicOr(&sm.first_hit, 1u << tile_lane);
            atomicAdd(&sm.groups[own], 1u);
            int i = 0;
            for (; i < sp.lane_taxa; i++) {
              const uint32_t old = atomicCAS(&sm.keys[i * 32 + own], 0u, result);
              if (old == 0u || old == result) {
                atomicAdd(&sm.cnts[i * 32 + own], n);
                break;
              }
            }
            if (i == sp.lane_taxa) atomicOr(&sm.overflow, 1u << own);
          }
        }
      }
      __syncwarp(); /* continuation queue and the runs queued by emit() are written before other lanes read them below */
      /* ---- 2. next 32 lookups: continuations first, then fresh runs ---- */
      const uint32_t n_cq = cq_n; /* <= 32: one per lane in flight at most */
      const uint32_t room = 32u - n_cq;
      const uint32_t n_pq = pq_n < room ? pq_n : room;
      f_aux = NH_AUX_NONE;
      f_start = 0;
      if (lane < n_cq) {
        f_unit = sm.q_unit[lane];
        f_ckey = sm.q_ckey[lane];
        f_aux = sm.q_aux[lane];
        if (EMIT) f_slot = sm.q_slot[lane];
      } else if (lane - n_cq < n_pq) {
        const uint4 e = sm.pq[(pq_head + (lane - n_cq)) & (NH_PQ_SLOTS - 1u)];
        const uint64_t h = nh_fmix64(((uint64_t)e.y << 32) | e.x);
        if (EMIT) f_slot = e.w;
        const uint32_t meta = e.z;
        if (db.min_hash && h < db.min_hash) {
          /* below minimum_acceptable_hash_value: kraken2 skips the lookup, taxon 0 */
          if (EMIT) b.lk_taxon[f_slot] = 0u;
        } else {
          const uint64_t idx = nh_fastmod(h, db.capacity, db.mod_m, db.mod_sh1, db.mod_sh2);
          if (FILTER) {
            /* who asks the filter first: units whose last few lookups all missed (sp.filter_mode 3), units none of
             * whose lookups has hit so far (1), or everybody (2).  A unit of human reads goes straight to the table
             * while its hits keep coming; a unit that keeps missing pays one request per lookup instead of 1.65 */
            const bool ask = FILTER == 2 || (FILTER == 3 ? sm.recent[meta & 31u] == 0u : sm.groups[sm.owner[meta & 31u]] == 0u);
            const uint32_t st = (uint32_t)idx & (ask ? 31u : 7u);
            f_unit = (uint32_t)(idx >> (ask ? 5 : 3));
            f_ckey = (uint32_t)(h >> (32u + db.value_bits)) | (st << ck_bits);
            f_aux = ask ? (meta | NH_AUX_FILTER) : meta;
          } else {
            f_unit = (uint32_t)(idx >> 3);
            f_start = (uint32_t)idx & 7u;
            f_ckey = (uint32_t)(h >> (32u + db.value_bits));
            f_aux = meta; /* zero sectors visited */
          }
        }
      }
      cq_n = 0;
      pq_head = (pq_head + n_pq) & (NH_PQ_SLOTS - 1u);
      pq_n -= n_pq;
      n_popped += n_pq;
      n_conts += n_cq;
      any_inflight = (n_cq + n_pq) != 0u;
      if (any_inflight) {
        /* lane pairs fetch the two 16-byte halves of one sector with ONE instruction, so a sector
         * stays one request (request = warp instruction x 128-byte line, DESIGN.md §3): the first
         * instruction covers the sectors of lanes 0-15, the second those of lanes 16-31 */
        const uint32_t mine = f_aux != NH_AUX_NONE ? f_unit : 0xFFFFFFFFu;
        const uint32_t half = lane & 1u, src_lane = lane >> 1;
        const uint32_t u0 = __shfl_sync(FULL_MASK, mine, src_lane);
        const uint32_t u1 = __shfl_sync(FULL_MASK, mine, 16u + src_lane);
        const uint32_t dst = sect0 + src_lane * 32u + half * 16u;
        const uint32_t *src0 = db.cells, *src1 = db.cells;
        if (FILTER) { /* filter records and table sectors are both 32 bytes, indexed alike */
          const uint32_t fmask = __ballot_sync(FULL_MASK, f_aux != NH_AUX_NONE && (f_aux & NH_AUX_FILTER));
          if ((fmask >> src_lane) & 1u) src0 = sp.filter;
          if ((fmask >> (16u + src_lane)) & 1u) src1 = sp.filter;
        }
        if (u0 != 0xFFFFFFFFu) cp_async16_l2_64(dst, src0 + (uint64_t)u0 * 8ULL + half * 4u);
        if (u1 != 0xFFFFFFFFu) cp_async16_l2_64(dst + 512u, src1 + (uint64_t)u1 * 8ULL + half * 4u);
        cp_async_arrive(sbar);
      }
      __syncwarp(); /* queue slots just read may be overwritten by the next pushes */
    };

    /* ---------------- scan, feeding the probe ---------------- */
    uint32_t n_runs = 0;           /* EMIT and DBG only: runs this lane has closed */
    uint32_t first_flag = NH_META_FIRST; /* cleared by the lane's first run */
    uint64_t last = NH_NONE64;     /* minimizer of the open run */
    {
      uint64_t so = 0;
      uint32_t nb = 0; /* bases of this lane's tile */
      if (have) {
        so = b.offsets[t.seq];
        const uint32_t len = (uint32_t)(b.offsets[t.seq + 1] - so);
        uint32_t npos = len - (uint32_t)k + 1u - t.pos_begin;
        if (npos > (uint32_t)db.tile_pos) npos = (uint32_t)db.tile_pos;
        nb = npos + (uint32_t)k - 1u;
      }
      const uint8_t *g = PACKED ? nullptr : b.bases + so + t.pos_begin;
      const uint32_t mis = PACKED ? 0u : (uint32_t)((uintptr_t)g & 3u);
      const uint32_t my_words = have ? (mis + nb + 3u) >> 2 : 0u; /* groups of four bases */
      const uint32_t max_words = __reduce_max_sync(FULL_MASK, my_words);

      uint64_t fwd = 0, rc = 0;
      /* window of 5 candidates c_i..c_{i-4}: a_i = min(c_i, c_{i-1}), m_i = min(a_i, a_{i-2}, c_{i-4});
       * ring[] holds c_{i-1}..c_{i-4}, pair[] holds a_{i-1}, a_{i-2} */
      uint64_t ring[4], pair[2];
#pragma unroll
      for (int i = 0; i < 4; i++) ring[i] = NH_NONE64;
      pair[0] = pair[1] = NH_NONE64;
      uint32_t c_run = 0; /* consecutive unambiguous bases ending here */
      uint32_t cnt = 0;   /* k-mer positions in the open run */
      const uint64_t dbg_base = DBG && have ? b.dbg_pos_offsets[t.seq] + t.pos_begin : 0;
      const uint32_t first_pos = mis + (uint32_t)(k - 1);
      const uint32_t end_idx = mis + nb;

      /* a closed run goes to the shared queue as one 16-byte entry */
      auto emit = [&](bool pred, uint64_t key, uint32_t count) {
        const uint32_t emask = __ballot_sync(FULL_MASK, pred);
        if (pred) {
          uint4 e;
          e.x = (uint32_t)key;
          e.y = (uint32_t)(key >> 32);
          e.z = lane | (count << 5) | first_flag;
          e.w = 0;
          if (EMIT) {
            e.w = t.slot + n_runs;
            b.lk_cnt[e.w] = (uint16_t)count;
          }
          sm.pq[(pq_head + pq_n + __popc(emask & lane_lt)) & (NH_PQ_SLOTS - 1u)] = e;
          if (first_flag) sm.first_min[lane] = key;
          first_flag = 0;
          if (EMIT || DBG) n_runs++;
        }
        pq_n += __popc(emask);
      };

      /* Four bases (one 4-byte word of the word-aligned stream, first base at stream index base_i).
       * Bytes outside the tile never get here as bases: the staging zero-fills what lies past the
       * tile's end and the head of the first word is cleared below, and a zero byte is an ambiguous
       * base - it resets the l-mer and cannot end a k-mer. */
      auto scan_quad = [&](const uint32_t codes /* first base in bits 7..6 */, const uint32_t ambs, const uint32_t base_i) {
#pragma unroll
        for (int j = 0; j < 4; j++) {
          const uint32_t i = base_i + (uint32_t)j; /* index in the word-aligned stream */
          const uint32_t cc = (codes >> (6u - 2u * (uint32_t)j)) & 3u;
          const bool amb = (ambs >> j) & 1u;
          fwd = ((fwd << 2) | cc) & lmask;
          rc = (rc >> 2) | ((uint64_t)(3u - cc) << rc_shift);
          c_run = amb ? 0u : c_run + 1u;
          uint64_t cand = NH_NONE64;
          if (c_run >= (uint32_t)l) {
            /* revcom_version 0 (databases built before kraken2 2.0.8) keeps the un-shifted low bits */
            const bool rev0 = REV0 || (DBG && db.revcom_version == 0); /* the debug instantiation decides at run time */
            const uint64_t rcv = rev0 ? (((rc << (64 - 2 * l)) | ((1ULL << (64 - 2 * l)) - 1ULL)) & lmask) : rc;
            cand = ((fwd < rcv ? fwd : rcv) & db.seed_mask) ^ db.toggle;
          }
          const uint64_t a_i = min_u64(cand, ring[0]);
          const uint64_t m = min_u64(min_u64(a_i, pair[1]), ring[3]);
          pair[1] = pair[0];
          pair[0] = a_i;
#pragma unroll
          for (int r = 3; r > 0; r--) ring[r] = ring[r - 1];
          ring[0] = cand;
          /* c_run counts from the tile's first base, so before first_pos a k-mer cannot have ended */
          const bool nonamb = i >= first_pos && c_run >= amb_span;
          const uint64_t mz = m ^ db.toggle;
          if (DBG && i >= first_pos && i < end_idx) { /* per-position output for nh_debug_minimizers */
            const uint64_t o = dbg_base + (i - first_pos);
            b.dbg_pos_min[o] = mz;
            b.dbg_pos_ambig[o] = nonamb ? 0 : 1;
          }
          const bool newrun = nonamb && mz != last;
          emit(newrun && cnt != 0u, last, cnt);
          cnt = newrun ? 1u : cnt + (nonamb ? 1u : 0u);
          last = newrun ? mz : last;
          if ((j & NH_STREAM_CHECK_MASK) == NH_STREAM_CHECK_MASK) {
            while (pq_n >= 32u) probe_round(); /* cq_n is 0 between rounds */
          }
        }
      };

      auto scan_word = [&](const uint32_t word, const uint32_t base_i) {
        uint32_t ambs;
        const uint32_t codes = nh_pack4(word, &ambs);
        scan_quad(codes, ambs, base_i);
      };

      if (PACKED) {
        /* one chunk = one unit of 32 bases: 8 code bytes + 1 validity word per lane, double-buffered */
        const uint64_t unit0 = have ? (uint64_t)b.poff[t.seq] + (t.pos_begin >> 5) : 0ULL;
        const uint32_t my_units = have ? (nb + 31u) >> 5 : 0u;
        const uint32_t n_chunks = (max_words + 7u) >> 3;
        auto stage = [&](const uint32_t ch) {
          const uint32_t buf = ch & 1u;
          const uint32_t dst = win0 + buf * (32u * NH_BCHUNK_STRIDE);
          if (ch < my_units) {
            cp_async8(dst, b.codes + (unit0 + ch) * 8ULL);
            cp_async4(dst + 8u, b.valid + unit0 + ch);
          }
          cp_async_arrive(bar0 + buf * 8u);
        };
        if (n_chunks) stage(0u);
        for (uint32_t ch = 0; ch < n_chunks; ch++) {
          if (ch + 1u < n_chunks) stage(ch + 1u);
          const uint32_t buf = ch & 1u;
          mbar_wait(bar0 + buf * 8u, (bar_par >> buf) & 1u);
          bar_par ^= 1u << buf;
          const uint32_t wbase = win0 + buf * (32u * NH_BCHUNK_STRIDE);
          const uint32_t c_lo = lds_u32(wbase), c_hi = lds_u32(wbase + 4u);
          uint32_t vw = lds_u32(wbase + 8u);
          /* bases past the tile's end (the next tile's, or stale bytes of a lane that is done) are ambiguous */
          const int rem = (int)nb - (int)(ch * 32u);
          vw = rem <= 0 ? 0u : (rem >= 32 ? vw : vw & ((1u << rem) - 1u));
          const uint32_t amb_w = ~vw;
          const uint32_t q0 = ch * 8u;
          const uint32_t qn = max_words - q0 < 8u ? max_words - q0 : 8u;
#pragma unroll 1
          for (uint32_t qd = 0; qd < qn; qd++) {
            const uint32_t cw = qd < 4u ? c_lo : c_hi;
            scan_quad((cw >> ((qd & 3u) * 8u)) & 0xFFu, (amb_w >> (qd * 4u)) & 0xFu, (q0 + qd) * 4u);
          }
          __syncwarp();
        }
        emit(cnt != 0u, last, cnt);
      } else {
      /* the lane's window for chunk c: bytes [32c, 32c + 48) from src0, the 16-byte block holding word 0 */
      const uint8_t *q = g - mis;
      const uint32_t a16 = (uint32_t)((uintptr_t)q & 15u);
      const uint8_t *src0 = q - a16;
      const uint32_t my_bytes = have ? a16 + mis + nb : 0u; /* from src0 to the tile's last base */
      const uint32_t n_chunks = (max_words + NH_BCHUNK_WORDS - 1u) / NH_BCHUNK_WORDS;
      auto stage = [&](const uint32_t ch) {
        const uint32_t buf = ch & 1u;
        const uint32_t lo = ch * (NH_BCHUNK_WORDS * 4u);
        const uint32_t dst = win0 + buf * (32u * NH_BCHUNK_STRIDE);
#pragma unroll
        for (uint32_t pc = 0; pc < NH_BCHUNK_STRIDE; pc += 16u) {
          /* bytes past the tile's end arrive as zeros (ambiguous bases); a lane whose tile is over keeps
           * clearing its window, so what it scans while longer tiles finish can never close a run */
          const uint32_t at = lo + pc;
          const uint32_t n_src = at < my_bytes ? (my_bytes - at < 16u ? my_bytes - at : 16u) : 0u;
          cp_async16_zfill(dst + pc, n_src ? src0 + at : src0, n_src);
        }
        cp_async_arrive(bar0 + buf * 8u);
      };
      if (n_chunks) stage(0u);
      for (uint32_t ch = 0; ch < n_chunks; ch++) {
        if (ch + 1u < n_chunks) stage(ch + 1u); /* its buffer was read two chunks ago (syncwarp below) */
        const uint32_t buf = ch & 1u;
        mbar_wait(bar0 + buf * 8u, (bar_par >> buf) & 1u);
        bar_par ^= 1u << buf;
        const uint32_t wbase = win0 + buf * (32u * NH_BCHUNK_STRIDE) + a16;
        const uint32_t w0 = ch * NH_BCHUNK_WORDS;
        const uint32_t wn = max_words - w0 < NH_BCHUNK_WORDS ? max_words - w0 : NH_BCHUNK_WORDS;
        uint32_t w_next = lds_u32(wbase);
        if (ch == 0u) w_next &= 0xFFFFFFFFu << (8u * mis); /* the bytes before the tile's first base */
#pragma unroll 1
        for (uint32_t w = 0; w < wn; w++) {
          const uint32_t word = w_next;
          w_next = lds_u32(wbase + (((w + 1u) & (NH_BCHUNK_WORDS - 1u)) << 2)); /* one word ahead; the wrap is a harmless re-read */
          scan_word(word, (w0 + w) * 4u);
        }
        __syncwarp(); /* every lane is done with this buffer before chunk ch + 2 lands in it */
      }
      emit(cnt != 0u, last, cnt);
      } /* !PACKED */
    }
    const bool has_runs = first_flag == 0u;
    if (EMIT && have) {
      NhTileOut o;
      o.lk_off = t.slot;
      o.lk_cnt = n_runs;
      b.tile_out[tile] = o;
    }
    if (has_runs) sm.last_min[lane] = last; /* the run closed last carried `last` */
    /* drain: whatever is waiting or in flight */
    while (pq_n + cq_n != 0u || any_inflight) probe_round();
    tot_lookups += n_popped; /* warp-uniform; added once per warp below */
    tot_sectors += n_popped + n_conts;

    /* ---------------- tile borders inside a unit scored here ---------------- */
    /* A tile starts with a fresh lookup even when its first minimizer equals the last one of the
     * tile before it in the same sequence; upstream counts that as ONE hit group (its
     * last_minimizer lives per mate, ambiguous stretches included). */
    {
      __syncwarp(); /* last_min / first_min / groups of the other lanes are final */
      const uint32_t has_mask = __ballot_sync(FULL_MASK, has_runs);
      if (have && kind != NH_ROLE_DEFERRED && t.pos_begin != 0u && has_runs && ((sm.first_hit >> lane) & 1u)) {
        const uint32_t seq_lane = lane - t.pos_begin / (uint32_t)db.tile_pos; /* lane of the sequence's first tile */
        const uint32_t cand = has_mask & lane_lt & ~((1u << seq_lane) - 1u);
        if (cand) {
          const uint32_t pl = 31u - (uint32_t)__clz(cand);
          if (sm.last_min[pl] == sm.first_min[lane]) atomicSub(&sm.groups[owner], 1u);
        }
      }
      __syncwarp();
    }

    /* ---------------- tiles of deferred units: hand the tile's table to k_score ---------------- */
    if (have && kind == NH_ROLE_DEFERRED) {
      const bool ovf = (sm.overflow >> lane) & 1u;
      NhTileSum ts;
      ts.first_min = has_runs ? sm.first_min[lane] : NH_NONE64;
      ts.last_min = has_runs ? last : NH_NONE64;
      ts.groups = sm.groups[lane];
      ts.flags = (has_runs ? NH_TILE_HAS : 0u) | (((sm.first_hit >> lane) & 1u) ? NH_TILE_FIRST_HIT : 0u) |
                 (ovf ? NH_TILE_OVERFLOW : 0u);
      b.tile_sum[tile] = ts;
      if (!ovf) {
        NhTileTab tt;
#pragma unroll
        for (int i = 0; i < NH_LANE_TAXA; i++) {
          tt.keys[i] = sm.keys[i * 32 + lane];
          tt.cnts[i] = sm.cnts[i * 32 + lane];
        }
        b.tile_tab[tile] = tt;
      }
    }

    /* ---------------- score the units that live in this warp ---------------- */
    if (have && kind == NH_ROLE_LEADER) {
      const uint32_t u = b.paired ? (t.seq >> 1) : t.seq;
      if ((sm.overflow >> lane) & 1u) {
        /* more distinct taxa than a lane table holds: k_score_big classifies the unit again */
        b.overflow_units[atomicAdd(&b.counters->n_overflow, 1u)] = u;
      } else {
        uint32_t ntab = 0;
        while (ntab < (uint32_t)sp.lane_taxa && sm.keys[ntab * 32u + lane] != 0u) ntab++;
        const int groups = (int)sm.groups[lane];
        const uint32_t total_kmers = unit_total_kmers(db, b, u);
        uint32_t best_s = 0, best_t = 0;
        for (uint32_t i = 0; i < ntab; i++) {
          const uint32_t tx = sm.keys[i * 32u + lane];
          uint32_t score = 0;
          for (uint32_t a = tx; a; a = parent[a]) score += lane_tab_get(sm, lane, ntab, a);
          if (score > best_s) {
            best_s = score;
            best_t = tx;
          } else if (score == best_s) {
            best_t = lca(parent, best_t, tx);
          }
        }
        uint32_t max_taxon = best_t;
        uint32_t max_score = max_taxon ? lane_tab_get(sm, lane, ntab, max_taxon) : 0u;
        const uint32_t required = (uint32_t)ceil(__dmul_rn(sp.confidence, (double)total_kmers));
        while (max_taxon && max_score < required) {
          uint32_t sum = 0;
          for (uint32_t i = 0; i < ntab; i++)
            if (is_a_ancestor_of_b(parent, max_taxon, sm.keys[i * 32u + lane]))
              sum += sm.cnts[i * 32u + lane];
          max_score = sum;
          if (max_score >= required) break;
          max_taxon = parent[max_taxon];
        }
        uint32_t call = max_taxon;
        if (call && groups < sp.min_hit_groups) call = 0;
        const uint32_t is_cls = call != 0u;
        const uint32_t keep = sp.keep_human ? is_cls : !is_cls;
        if (b.out_call) b.out_call[u] = call ? db.ext_id[call] : 0u;
        if (b.out_keep) b.out_keep[u] = (uint8_t)keep;
        if (b.dbg_call) b.dbg_call[u] = call;
        if (b.dbg_total_kmers) b.dbg_total_kmers[u] = total_kmers;
        if (b.dbg_hit_groups) b.dbg_hit_groups[u] = (uint32_t)groups;
        tot_classified += is_cls;
        tot_kept += keep;
      }
    }
    __syncwarp();
  }
  tot_classified = warp_sum_u32(tot_classified);
  tot_kept = warp_sum_u32(tot_kept);
  if (lane == 0) {
    if (tot_lookups) atomicAdd(&b.counters->n_lookups, tot_lookups);
    if (tot_sectors) atomicAdd(&b.counters->n_sector_reads, tot_sectors);
    if (tot_classified) atomicAdd(&b.counters->n_classified, tot_classified);
    if (tot_kept) atomicAdd(&b.counters->n_kept, tot_kept);
  }
}

/* ------------------------------------------------------------------ */
/* per-read output support: pack every tile's (external taxid, run length) */

__global__ void __launch_bounds__(NH_BLOCK_THREADS)
k_gather_runs(const NhDbParams db, const NhBatchPtrs b, uint32_t *__restrict__ run_ext,
              uint16_t *__restrict__ run_len, uint32_t *__restrict__ tile_run_off,
              uint32_t *__restrict__ cursor) {
  const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
  const uint32_t n_tiles = b.counters->n_tiles;
  for (uint32_t tile = blockIdx.x * NH_WARPS_PER_BLOCK + warp; tile < n_tiles;
       tile += gridDim.x * NH_WARPS_PER_BLOCK) {
    const NhTileOut to = b.tile_out[tile];
    uint32_t base = 0;
    if (lane == 0) base = to.lk_cnt ? atomicAdd(cursor, to.lk_cnt) : 0u;
    base = __shfl_sync(FULL_MASK, base, 0);
    if (lane == 0) tile_run_off[tile] = base;
    for (uint32_t j = lane; j < to.lk_cnt; j += 32u) {
      run_ext[base + j] = db.ext_id[b.lk_taxon[to.lk_off + j]];
      run_len[base + j] = b.lk_cnt[to.lk_off + j];
    }
  }
}

/* ------------------------------------------------------------------ */
/* roofline helper: the probe's access pattern and nothing else             */
/*
 * What bounds the hash probe on B200 is the rate of random table requests
 * (address translation, DESIGN.md §3), so the ceiling the streaming kernel is
 * held to is measured with its own access pattern: every lane keeps DEPTH
 * independent probe chains going; a chain reads a random 32-byte sector and,
 * with probability p (the table's chain-spill rate, 0.41 at load 0.7), the
 * ADJACENT sector - but only after the first one has arrived, exactly like a
 * continuation that waits one probe round in k_stream_classify.  G lanes can
 * share one item and read G adjacent sectors of an aligned 32*G-byte block
 * with one instruction (a request is a warp instruction x 128-byte line).
 * SMWIN > 0 confines every SM to its own window of that many bytes (perfect
 * page locality: not reachable by a hash table, reported as a curiosity).
 * No hashing of k-mers, no scan, no scoring: whatever this reaches is an upper
 * bound for any kernel that makes the same table requests.
 */
/* the streaming kernel's own fetch: lane pairs copy the two halves of a sector with cp.async */
__device__ __forceinline__ void fetch_sector_async(const uint32_t *cells, uint64_t sector, uint32_t smem_slot0, uint32_t lane) {
  const uint32_t half = lane & 1u, src_lane = lane >> 1;
  const uint64_t u0 = __shfl_sync(FULL_MASK, sector, src_lane);
  const uint64_t u1 = __shfl_sync(FULL_MASK, sector, 16u + src_lane);
  const uint32_t dst = smem_slot0 + src_lane * 32u + half * 16u;
  cp_async16_l2_64(dst, cells + u0 * 8ULL + half * 4u);
  cp_async16_l2_64(dst + 512u, cells + u1 * 8ULL + half * 4u);
}

/* DEPTH rounds in flight per warp, every round one sector per lane through cp.async + commit/wait groups */
template <int DEPTH>
__global__ void __launch_bounds__(256)
k_probe_pattern_async(const uint32_t *__restrict__ cells, uint64_t n_sectors, uint32_t items_per_chain,
                      uint32_t p_thresh, uint64_t seed, unsigned long long *__restrict__ counters,
                      uint32_t *__restrict__ sink) {
  __shared__ __align__(16) uint32_t s_sect[8][DEPTH][32 * 8];
  const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
  const uint64_t chain0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * DEPTH;
  uint64_t blk[DEPTH];
  uint32_t left[DEPTH], cont[DEPTH];
  uint32_t acc = 0;
  unsigned long long items = 0, requests = 0;
#pragma unroll
  for (int d = 0; d < DEPTH; d++) {
    blk[d] = __umul64hi(nh_fmix64(seed + (chain0 + d) * 0x9E3779B97F4A7C15ULL), n_sectors);
    left[d] = items_per_chain;
    cont[d] = 0;
    fetch_sector_async(cells, blk[d], smem_addr(&s_sect[warp][d][0]), lane);
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  for (uint32_t it = 1; it <= 2u * items_per_chain + 2u; it++) { /* warp-uniform trip count: lanes that are done idle along */
#pragma unroll
    for (int d = 0; d < DEPTH; d++) {
      asm volatile("cp.async.wait_group %0;" ::"n"(DEPTH - 1) : "memory");
      __syncwarp();
      const uint4 lo = *reinterpret_cast<const uint4 *>(&s_sect[warp][d][lane * 8u]);
      const uint4 hi = *reinterpret_cast<const uint4 *>(&s_sect[warp][d][lane * 8u + 4u]);
      const uint32_t x = lo.x ^ lo.y ^ lo.z ^ lo.w ^ hi.x ^ hi.y ^ hi.z ^ hi.w;
      __syncwarp();
      if (left[d] != 0u) {
        acc ^= x;
        requests++;
        const uint64_t h = nh_fmix64(seed ^ ((chain0 + d) << 20) ^ it ^ (uint64_t)(x & 1u) << 63);
        if (!cont[d] && (uint32_t)h < p_thresh) {
          cont[d] = 1;
          blk[d] = blk[d] + 1 < n_sectors ? blk[d] + 1 : 0;
        } else {
          cont[d] = 0;
          items++;
          left[d]--;
          blk[d] = __umul64hi(h, n_sectors);
        }
      }
      fetch_sector_async(cells, blk[d], smem_addr(&s_sect[warp][d][0]), lane);
      asm volatile("cp.async.commit_group;" ::: "memory");
    }
    if (!__any_sync(FULL_MASK, left[0] != 0u || left[DEPTH - 1] != 0u)) break;
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  if (acc == 0x9E3779B9u) sink[0] = acc;
  items = __reduce_add_sync(FULL_MASK, (uint32_t)items);
  requests = __reduce_add_sync(FULL_MASK, (uint32_t)requests);
  if (lane == 0) {
    atomicAdd(&counters[0], items);
    atomicAdd(&counters[1], requests);
  }
}

template <int G, int DEPTH>
__global__ void __launch_bounds__(256)
k_probe_pattern(const uint32_t *__restrict__ cells, uint64_t n_sectors, uint32_t items_per_chain,
                uint32_t p_thresh /* of 2^32 */, uint64_t seed, uint64_t sm_window_sectors,
                unsigned long long *__restrict__ counters /* [0] items, [1] requests */, uint32_t *__restrict__ sink) {
  const uint32_t lane = lane_id();
  const uint32_t sub = lane % G;
  const uint64_t chain0 = (((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) / G) * DEPTH;
  uint64_t win_base = 0, win_size = n_sectors / G; /* in blocks of G sectors */
  if (sm_window_sectors) {
    uint32_t smid;
    asm("mov.u32 %0, %%smid;" : "=r"(smid));
    win_size = sm_window_sectors / G;
    const uint64_t n_win = (n_sectors / G) / win_size;
    win_base = (uint64_t)(smid % (uint32_t)(n_win ? n_win : 1)) * win_size;
  }
  uint32_t acc = 0;
  uint32_t c[DEPTH][8];
  uint64_t blk[DEPTH];    /* block of G sectors the chain reads next / has in flight */
  uint32_t left[DEPTH];   /* items the chain still has to start */
  uint32_t cont[DEPTH];   /* the request in flight is a continuation */
  unsigned long long items = 0, requests = 0;
#pragma unroll
  for (int d = 0; d < DEPTH; d++) {
    const uint64_t h = nh_fmix64(seed + (chain0 + d) * 0x9E3779B97F4A7C15ULL);
    blk[d] = win_base + __umul64hi(h, win_size);
    left[d] = items_per_chain;
    cont[d] = 0;
    ld_sector(cells + (blk[d] * G + sub) * 8ULL, c[d]);
  }
  bool busy = true;
  for (uint32_t it = 1; busy; it++) {
    busy = false;
#pragma unroll
    for (int d = 0; d < DEPTH; d++) {
      if (left[d] == 0u) continue;
      busy = true;
      /* the data in flight decides what the chain does next, as a probe's sector does */
      const uint32_t x = c[d][0] ^ c[d][1] ^ c[d][2] ^ c[d][3] ^ c[d][4] ^ c[d][5] ^ c[d][6] ^ c[d][7];
      acc ^= x;
      requests++;
      const uint64_t h = nh_fmix64(seed ^ ((chain0 + d) << 20) ^ it ^ (uint64_t)(x & 1u) << 63);
      if (!cont[d] && (uint32_t)h < p_thresh) {
        cont[d] = 1;
        blk[d] = blk[d] + 1 < win_base + win_size ? blk[d] + 1 : win_base;
      } else {
        cont[d] = 0;
        items++;
        if (--left[d] == 0u) continue;
        blk[d] = win_base + __umul64hi(h, win_size);
      }
      ld_sector(cells + (blk[d] * G + sub) * 8ULL, c[d]);
    }
  }
  if (acc == 0x9E3779B9u) sink[0] = acc; /* keeps the loads alive */
  if (sub == 0) {
    items = __reduce_add_sync(__activemask(), (uint32_t)items);
    requests = __reduce_add_sync(__activemask(), (uint32_t)requests);
    if (lane == 0) {
      atomicAdd(&counters[0], items);
      atomicAdd(&counters[1], requests);
    }
  }
}

/* ------------------------------------------------------------------ */
/* launchers                                                            */

template <bool EMIT>
static size_t stream_smem_bytes(uint32_t node_count) {
  const uint32_t parent_words = node_count <= NH_SMEM_PARENT_MAX ? node_count : 0u;
  return (size_t)((parent_words + 3u) & ~3u) * 4 + NH_WARPS_PER_BLOCK * sizeof(StreamWarpSmem<EMIT>);
}

cudaError_t nh_kernels_init(void) {
  cudaError_t e = cudaFuncSetAttribute(k_score_big, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       NH_BIG_HASH_SLOTS * 8);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(k_score<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           NH_SMEM_PARENT_MAX * 4 + NH_WARPS_PER_BLOCK * NH_WARP_HASH_SLOTS * 8);
  if (e != cudaSuccess) return e;
  const int smax = (int)stream_smem_bytes<false>(NH_SMEM_PARENT_MAX), smax_emit = (int)stream_smem_bytes<true>(NH_SMEM_PARENT_MAX);
#define NH_SET_SMEM(kern, bytes)                                                             \
  e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);       \
  if (e != cudaSuccess) return e;
  NH_SET_SMEM((k_stream_classify<5, 1, false, false, false, false, 0>), smax)
  NH_SET_SMEM((k_stream_classify<5, 1, false, false, true, false, 0>), smax_emit)
  NH_SET_SMEM((k_stream_classify<5, 0, false, false, false, false, 0>), smax)
  NH_SET_SMEM((k_stream_classify<5, 0, false, true, false, false, 0>), smax)
  NH_SET_SMEM((k_stream_classify<5, 0, true, false, false, false, 0>), smax)
  NH_SET_SMEM((k_stream_classify<5, 0, false, false, true, false, 0>), smax_emit)
  NH_SET_SMEM((k_stream_classify<5, 0, false, true, true, false, 0>), smax_emit)
  NH_SET_SMEM((k_stream_classify<5, 1, false, false, false, true, 0>), smax)
  NH_SET_SMEM((k_stream_classify<5, 0, false, false, false, true, 0>), smax)
  NH_SET_SMEM((k_stream_classify<5, 0, false, true, false, true, 0>), smax)
  NH_SET_SMEM((k_stream_classify<5, 1, false, false, false, false, 1>), smax)
  NH_SET_SMEM((k_stream_classify<5, 1, false, false, false, false, 2>), smax)
  NH_SET_SMEM((k_stream_classify<5, 1, false, false, false, false, 3>), smax)
  NH_SET_SMEM((k_stream_classify<5, 1, false, false, false, true, 1>), smax)
  NH_SET_SMEM((k_stream_classify<5, 1, false, false, false, true, 2>), smax)
  NH_SET_SMEM((k_stream_classify<5, 1, false, false, false, true, 3>), smax)
#undef NH_SET_SMEM
  return cudaSuccess;
}

void nh_launch_filter_build(const NhDbParams &db, uint32_t *filter, uint32_t n_blocks, cudaStream_t st) {
  k_filter_build<<<(n_blocks + 255u) / 256u, 256, 0, st>>>(db.cells, db.capacity, db.value_bits, db.value_mask, filter, n_blocks);
}

int nh_launch_len_scan(const uint32_t *len, uint32_t n_seqs, uint64_t *sums, uint64_t *off, uint32_t *poff, cudaStream_t st) {
  const uint32_t nb = (n_seqs + PLAN_THREADS - 1) / PLAN_THREADS;
  if (nb == 0) return 0;
  k_len_count<<<nb, PLAN_THREADS, 0, st>>>(len, n_seqs, sums);
  k_len_scan<<<1, PLAN_THREADS, 0, st>>>(sums, nb);
  k_len_fill<<<nb, PLAN_THREADS, 0, st>>>(len, n_seqs, sums, off, poff);
  return 3;
}

int nh_launch_plan(const NhDbParams &db, const NhBatchPtrs &b, cudaStream_t st) {
  const uint32_t nb = (b.n_seqs + PLAN_THREADS - 1) / PLAN_THREADS;
  k_plan_count<<<nb, PLAN_THREADS, 0, st>>>(b.offsets, b.n_seqs, db.k, db.tile_pos, b.block_sums);
  k_plan_scan<<<1, PLAN_THREADS, 0, st>>>(b.block_sums, nb, b.counters);
  k_plan_fill<<<nb, PLAN_THREADS, 0, st>>>(b.offsets, b.n_seqs, db.k, db.tile_pos, b.paired,
                                           b.deferred_units != nullptr, b.block_sums, b.tile_base,
                                           b.tiles, b.deferred_units, b.counters, b.seq_info);
  if (b.seq_info == nullptr) return 3;
  uint32_t blocks = (b.tiles_upper + 255u) / 256u;
  if (blocks > 148u * 16u) blocks = 148u * 16u;
  k_plan_tiles<<<blocks ? blocks : 1u, 256, 0, st>>>(b.tile_base, b.seq_info, b.n_seqs, db.tile_pos, b.tiles, b.counters);
  return 4;
}

bool nh_fused_supported(const NhDbParams &db) {
  /* window of 5 l-mers, 10-bit run lengths, u32 sector indices with 0xFFFFFFFF meaning "none" */
  return db.w == 5 && db.tile_pos <= NH_FUSED_TILE_POS_MAX && db.capacity < (1ULL << 35) - 8ULL;
}

int nh_launch_stream(const NhDbParams &db, const NhBatchPtrs &b, const NhScoreParams &sp,
                     uint32_t tiles_upper, int sm_count, cudaStream_t st) {
  const uint32_t groups = (tiles_upper + 31u) / 32u;
  const uint32_t blocks = (groups + NH_WARPS_PER_BLOCK - 1) / NH_WARPS_PER_BLOCK;
  const uint32_t smax = (uint32_t)sm_count * NH_STREAM_MIN_BLOCKS; /* persistent: groups come from a counter */
  uint32_t grid = blocks < smax ? blocks : smax;
  if (grid == 0) grid = 1;
  const bool emit = b.emit_all_taxa != 0;
  const size_t smem = emit ? stream_smem_bytes<true>(db.node_count) : stream_smem_bytes<false>(db.node_count);
  /* kraken2's defaults (k 35, l 31, current reverse-complement) get the instantiation with the
   * constants compiled in; anything else with a window of 5 takes the generic one */
  const bool kl_default = db.k == 35 && db.l == 31 && db.revcom_version != 0;
#define NH_LAUNCH(KLv, DBGv, REVv, EMITv, PACKv) \
  k_stream_classify<5, KLv, DBGv, REVv, EMITv, PACKv, 0><<<grid, NH_BLOCK_THREADS, smem, st>>>(db, b, sp)
#define NH_LAUNCH_FILTER(PACKv, POLv) \
  k_stream_classify<5, 1, false, false, false, PACKv, POLv><<<grid, NH_BLOCK_THREADS, smem, st>>>(db, b, sp)
  /* the miss filter goes with the default instantiations (k 35, l 31, no per-read output) */
  const bool filter = sp.filter != nullptr && sp.filter_mode != 0 && kl_default && !emit && b.dbg_pos_min == nullptr;
  if (filter && b.codes != nullptr) {
    if (sp.filter_mode == 1) NH_LAUNCH_FILTER(true, 1);
    else if (sp.filter_mode == 2) NH_LAUNCH_FILTER(true, 2);
    else NH_LAUNCH_FILTER(true, 3);
  } else if (filter) {
    if (sp.filter_mode == 1) NH_LAUNCH_FILTER(false, 1);
    else if (sp.filter_mode == 2) NH_LAUNCH_FILTER(false, 2);
    else NH_LAUNCH_FILTER(false, 3);
  }
  else if (b.codes != nullptr) { /* packed input: never with the per-position debug output or per-read runs */
    if (kl_default) NH_LAUNCH(1, false, false, false, true);
    else if (db.revcom_version == 0) NH_LAUNCH(0, false, true, false, true);
    else NH_LAUNCH(0, false, false, false, true);
  } else if (b.dbg_pos_min != nullptr) /* nh_debug_minimizers (never with emit_runs) */
    NH_LAUNCH(0, true, false, false, false);
  else if (kl_default && emit) NH_LAUNCH(1, false, false, true, false);
  else if (kl_default) NH_LAUNCH(1, false, false, false, false);
  else if (db.revcom_version == 0 && emit) NH_LAUNCH(0, false, true, true, false);
  else if (db.revcom_version == 0) NH_LAUNCH(0, false, true, false, false);
  else if (emit) NH_LAUNCH(0, false, false, true, false);
  else NH_LAUNCH(0, false, false, false, false);
#undef NH_LAUNCH
#undef NH_LAUNCH_FILTER
  return 1;
}

int nh_launch_minimizers(const NhDbParams &db, const NhBatchPtrs &b, uint32_t tiles_upper,
                         int sm_count, cudaStream_t st) {
  uint32_t groups = (tiles_upper + NH_WARPS_PER_BLOCK - 1) / NH_WARPS_PER_BLOCK;
  uint32_t max_grid = (uint32_t)sm_count * 8u;
  uint32_t grid = groups < max_grid ? groups : max_grid;
  if (grid == 0) grid = 1;
  if (db.w == 5)
    k_minimizers<5><<<grid, NH_BLOCK_THREADS, 0, st>>>(db, b);
  else
    k_minimizers<0><<<grid, NH_BLOCK_THREADS, 0, st>>>(db, b);
  return 1;
}

int nh_launch_probe(const NhDbParams &db, const uint64_t *keys, uint32_t *taxa,
                    const uint32_t *n_dev, uint32_t n_upper, int sm_count, cudaStream_t st) {
  uint32_t blocks = (n_upper + 255u) / 256u;
  uint32_t max_grid = (uint32_t)sm_count * 8u;
  uint32_t grid = blocks < max_grid ? blocks : max_grid;
  if (grid == 0) grid = 1;
  k_probe<<<grid, 256, 0, st>>>(db, keys, taxa, n_dev, n_upper);
  return 1;
}

int nh_launch_score(const NhDbParams &db, const NhBatchPtrs &b, const NhScoreParams &sp,
                    int sm_count, cudaStream_t st) {
  uint32_t blocks = (b.n_units + NH_WARPS_PER_BLOCK - 1) / NH_WARPS_PER_BLOCK;
  uint32_t max_grid = (uint32_t)sm_count * 8u;
  uint32_t grid = blocks < max_grid ? blocks : max_grid;
  if (grid == 0) grid = 1;
  const size_t hash_bytes = NH_WARPS_PER_BLOCK * NH_WARP_HASH_SLOTS * 8;
  if (db.node_count <= NH_SMEM_PARENT_MAX)
    k_score<true><<<grid, NH_BLOCK_THREADS, db.node_count * 4 + hash_bytes, st>>>(db, b, sp);
  else
    k_score<false><<<grid, NH_BLOCK_THREADS, hash_bytes, st>>>(db, b, sp);
  k_score_big<<<sm_count, 32, NH_BIG_HASH_SLOTS * 8, st>>>(db, b, sp);
  return 2;
}

int nh_launch_gather_runs(const NhDbParams &db, const NhBatchPtrs &b, uint32_t tiles_upper,
                          uint32_t *run_ext, uint16_t *run_len, uint32_t *tile_run_off,
                          uint32_t *cursor, int sm_count, cudaStream_t st) {
  uint32_t blocks = (tiles_upper + NH_WARPS_PER_BLOCK - 1) / NH_WARPS_PER_BLOCK;
  uint32_t max_grid = (uint32_t)sm_count * 8u;
  uint32_t grid = blocks < max_grid ? blocks : max_grid;
  if (grid == 0) grid = 1;
  cudaMemsetAsync(cursor, 0, 4, st);
  k_gather_runs<<<grid, NH_BLOCK_THREADS, 0, st>>>(db, b, run_ext, run_len, tile_run_off, cursor);
  return 1;
}

int nh_launch_probe_pattern(const uint32_t *cells, uint64_t n_sectors, int lanes, int depth, int blocks_per_sm,
                            uint32_t items_per_chain, uint32_t p_thresh, uint64_t seed, uint64_t sm_window_sectors,
                            unsigned long long *counters, uint32_t *sink, int sm_count, cudaStream_t st) {
  const int grid = sm_count * blocks_per_sm; /* 256 threads per block: 1..8 blocks per SM */
  if (lanes == 0) { /* the streaming kernel's fetch (cp.async, lane pairs) */
    if (depth == 1)
      k_probe_pattern_async<1><<<grid, 256, 0, st>>>(cells, n_sectors, items_per_chain, p_thresh, seed, counters, sink);
    else
      k_probe_pattern_async<2><<<grid, 256, 0, st>>>(cells, n_sectors, items_per_chain, p_thresh, seed, counters, sink);
    return 1;
  }
#define NH_PP(G, D)                                                                                                  \
  k_probe_pattern<G, D><<<grid, 256, 0, st>>>(cells, n_sectors, items_per_chain, p_thresh, seed, sm_window_sectors, \
                                              counters, sink)
  if (lanes == 4) {
    if (depth == 1) NH_PP(4, 1); else if (depth == 2) NH_PP(4, 2); else NH_PP(4, 4);
  } else if (lanes == 2) {
    if (depth == 1) NH_PP(2, 1); else if (depth == 2) NH_PP(2, 2); else NH_PP(2, 4);
  } else {
    if (depth == 1) NH_PP(1, 1); else if (depth == 2) NH_PP(1, 2); else NH_PP(1, 4);
  }
#undef NH_PP
  return 1;
}
