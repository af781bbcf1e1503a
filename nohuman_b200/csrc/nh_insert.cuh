/*
 * nh_insert.cuh — the build side of the table: build_db.cc's ProcessSequence / CompactHashTable::CompareAndSet
 * loop (SURVEY.md A.7) as an atomicCAS insert with the LCA merge, and the kernel that inserts the minimizers the
 * warp-per-tile kernel left in a batch's lookup arrays.  Shared by the synthetic builder (nh_synth.cu) and the
 * library builder (nh_build.cu), which differ only in where a tile's taxon comes from.
 */
#ifndef NH_INSERT_CUH
#define NH_INSERT_CUH

#include <stdint.h>

#include "nh_kernels.cuh"

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

/* The CompareAndSet loop of build_db.cc collapsed to value := LCA(old, taxon).  Returns 1 if a previously
 * empty cell was claimed.  A walk that has gone past 64 cells gives up once *stop is nonzero (the table is too
 * full and the build fails anyway), so that a full table cannot hold every lane to a walk over all of it. */
__device__ __forceinline__ uint32_t cht_insert_lca(const NhDbParams &db, uint32_t *cells, uint64_t key, uint32_t taxon,
                                                   const unsigned long long *stop) {
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
    if ((probes & 63u) == 0 && *((volatile const unsigned long long *)stop)) return 0;
  }
  return 0; /* table full: the caller sees the load stall */
}

/* One warp per tile of the batch: every lookup of the tile (b.lk_min) is inserted under the taxa that
 * `taxa(tile)` gives (.x, and .y too when it is not 0).  counters[0] counts the claimed cells, added once per
 * tile; once it passes size_limit, counters[1] becomes 1, the tiles not yet started are left alone and walks
 * longer than 64 cells give up, so that a table that is too small fails fast instead of walking ever longer
 * probe chains.  The tiles already running when the flag is set still claim cells: the load can pass
 * size_limit by at most their claims (up to 128 lookups, 256 inserts, per running warp). */
template <typename TaxonSource>
__global__ void __launch_bounds__(NH_BLOCK_THREADS)
k_insert_tiles(const NhDbParams db, uint32_t *cells, const NhBatchPtrs b, const TaxonSource taxa,
               unsigned long long size_limit, unsigned long long *counters) {
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t n_tiles = b.counters->n_tiles;
  for (uint32_t tile = blockIdx.x * NH_WARPS_PER_BLOCK + warp; tile < n_tiles;
       tile += gridDim.x * NH_WARPS_PER_BLOCK) {
    const unsigned long long full = __shfl_sync(0xFFFFFFFFu, lane == 0 ? *((volatile unsigned long long *)&counters[1]) : 0ull, 0);
    if (full) break;
    const NhTile t = b.tiles[tile];
    const NhTileOut to = b.tile_out[tile];
    const uint2 tx = taxa(t);
    uint32_t claimed = 0;
    for (uint32_t j = lane; j < to.lk_cnt; j += 32u) {
      const uint64_t key = b.lk_min[to.lk_off + j];
      claimed += cht_insert_lca(db, cells, key, tx.x, counters + 1);
      if (tx.y) claimed += cht_insert_lca(db, cells, key, tx.y, counters + 1);
    }
    claimed = __reduce_add_sync(0xFFFFFFFFu, claimed);
    if (lane == 0 && claimed) {
      const unsigned long long before = atomicAdd(&counters[0], (unsigned long long)claimed);
      if (before + claimed > size_limit) atomicExch(&counters[1], 1ull);
    }
  }
}

#endif
