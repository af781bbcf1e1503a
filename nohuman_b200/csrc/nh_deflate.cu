/*
 * nh_deflate.cu — BGZF (blocked gzip) compression on the GPU.
 *
 * The input is a list of host blocks, each cut into members of BGZF_INPUT (0xff00) bytes and a shorter
 * last member, exactly as the pipeline's zlib path (bgzf_members in nh_pipeline.cc) cuts them.  Every
 * member becomes one complete gzip member: the 18-byte header with the 'BC' subfield holding BSIZE - 1,
 * one raw deflate block (dynamic Huffman, or stored when that is not smaller), CRC32 and ISIZE.
 *
 * k_bgzf_deflate: one CTA of NT threads per member, the member staged in shared memory.
 *   1. CRC32: every thread takes a slice, computes its raw CRC and shifts it by the bytes after the
 *      slice (multiplication by x^(8n) mod P, the crc32_combine algebra); the shifted CRCs XOR together.
 *   2. Hash chains: the hash of the 4 bytes at each position is computed in parallel; warp 0 then links
 *      every position to the previous one with the same hash, 32 positions a step: __match_any_sync
 *      finds the predecessors inside the step, a head table (written only by each group's last lane)
 *      those before it.  No result depends on thread scheduling.
 *   3. Matches: every position walks its chain (CHAIN candidates, distance <= 32768) for the longest
 *      match of 4..258 bytes, in parallel across positions.
 *   4. Parse: the member is cut into NSEG segments; one thread per segment parses its segment lazily
 *      (a match shorter than LAZY yields to a longer one at the next position), matches clipped at
 *      the segment's end, and counts literal/length and distance symbols with shared-memory atomics.
 *   5. Codes: length-limited canonical Huffman codes (15 bits; 7 for the code-length code) from a
 *      two-queue Huffman tree and the JPEG Annex K.3 depth adjustment; code lengths RLE-coded with
 *      symbols 16, 17 and 18.
 *   6. Bits: every segment's bit count, a scan over segments, and each segment thread ORs its tokens'
 *      codes into shared-memory words.  When the coded block is not smaller than a stored block, the
 *      member is stored (BTYPE 0), which bounds BSIZE at 65 311 bytes.
 * k_bgzf_scan and k_bgzf_compact then pack the members back to back so that only compressed bytes are
 * copied to the host.
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "nh_crc.cuh"
#include "nh_internal.h"

namespace {

constexpr uint32_t BGZF_SLOT = 65536;     /* device bytes reserved per member before compaction */
constexpr int NT = 512;                   /* threads per member */
constexpr int NSEG = 128;                 /* parse segments per member */
constexpr int HBITS = 14;                 /* hash table of 2^14 heads */
constexpr int CHAIN = 48;                 /* candidates tried per position */
constexpr uint32_t NICE = 128;            /* a match this long ends the search */
constexpr uint32_t LAZY = 16;             /* a shorter match is checked against the next position's */
constexpr uint32_t NO_HASH = 0xffff;      /* positions with fewer than 4 bytes left */
constexpr uint32_t MATCH_FLAG = 0x80000000u;

constexpr size_t SMEM_IN = 65536;                    /* member bytes as words, zero padded */
constexpr size_t SMEM_PREV = BGZF_INPUT * 2;         /* chain links (u16); later the output bit buffer */
constexpr size_t SMEM_HEAD = (size_t(1) << HBITS) * 2; /* hash heads (u16); later the Huffman workspace */
constexpr size_t SMEM_BYTES = SMEM_IN + SMEM_PREV + SMEM_HEAD;

/* gzip member header up to the BC subfield's value: BGZF's fixed fields (BGZF_HEADER) */
__constant__ uint8_t c_gz_header[16] = {NH_BGZF_HEADER_BYTES};

__constant__ uint8_t c_cl_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

__device__ __forceinline__ uint32_t byte_at(const uint32_t *w, uint32_t i) { return (w[i >> 2] >> ((i & 3) * 8)) & 0xff; }

__device__ __forceinline__ uint32_t load32(const uint32_t *w, uint32_t i) {
  return __funnelshift_r(w[i >> 2], w[(i >> 2) + 1], (i & 3) * 8);
}

__device__ __forceinline__ uint32_t hash4(uint32_t v) { return (v * 2654435761u) >> (32 - HBITS); }

/* deflate length code (257..285), its extra bits and their value */
__device__ __forceinline__ void len_code(uint32_t len, uint32_t &code, uint32_t &nx, uint32_t &xv) {
  const uint32_t x = len - 3;
  if (len == 258) {
    code = 285, nx = 0, xv = 0;
  } else if (x < 8) {
    code = 257 + x, nx = 0, xv = 0;
  } else {
    const uint32_t nb = 31 - __clz(x);
    code = 257 + 4 * (nb - 1) + ((x >> (nb - 2)) & 3);
    nx = nb - 2;
    xv = x & ((1u << nx) - 1);
  }
}

/* deflate distance code (0..29), its extra bits and their value */
__device__ __forceinline__ void dist_code(uint32_t dist, uint32_t &code, uint32_t &nx, uint32_t &xv) {
  const uint32_t x = dist - 1;
  if (x < 4) {
    code = x, nx = 0, xv = 0;
  } else {
    const uint32_t nb = 31 - __clz(x);
    code = 2 * nb + ((x >> (nb - 1)) & 1);
    nx = nb - 1;
    xv = x & ((1u << nx) - 1);
  }
}

struct HuffScratch {
  uint32_t w[576];
  uint16_t sorted[288];
  uint16_t parent[576];
  uint16_t depth[576];
  uint16_t count[296];
  uint32_t next[16], cnt[16];
};

/* Huffman workspace, in the head table's space once the chains are built */
struct CodeWork {
  uint32_t hist_ll[288], hist_d[32], hist_cl[20];
  uint16_t code_ll[288], code_d[32], code_cl[20];
  uint8_t len_ll[288], len_d[32], len_cl[20];
  uint16_t rle[320]; /* code-length symbol | extra value << 5 */
  uint32_t n_rle, hlit, hdist, hclen, header_bits;
  HuffScratch hs[2];
};
static_assert(sizeof(CodeWork) <= SMEM_HEAD, "Huffman workspace exceeds the head table");

/* Length-limited canonical Huffman code over freq[0..n) (warp-collective; lane 0 does the serial
 * part).  Symbols are ordered by (frequency, symbol), so the result does not depend on scheduling.
 * At least two symbols get codes: inflate rejects a one-symbol code other than a distance code. */
__device__ void build_code(uint32_t *freq, int n, int limit, uint8_t *len, uint16_t *code, HuffScratch &hs) {
  const int lane = threadIdx.x & 31;
  if (lane == 0) {
    int m = 0;
    for (int i = 0; i < n; i++) m += freq[i] != 0;
    for (int i = 0; m < 2 && i < n; i++)
      if (!freq[i]) freq[i] = 1, m++;
  }
  __syncwarp();
  for (int i = lane; i < n; i += 32) {
    const uint32_t f = freq[i];
    len[i] = 0;
    if (!f) continue;
    int r = 0;
    for (int j = 0; j < n; j++) {
      const uint32_t g = freq[j];
      r += g && (g < f || (g == f && j < i));
    }
    hs.sorted[r] = (uint16_t)i;
  }
  __syncwarp();
  if (lane == 0) {
    int m = 0;
    for (int i = 0; i < n; i++) m += freq[i] != 0;
    for (int k = 0; k < m; k++) hs.w[k] = freq[hs.sorted[k]];
    /* two queues: leaves in frequency order, internal nodes in the order they are made */
    int li = 0, ii = m, nx = m;
    while (nx < 2 * m - 1) {
      int pick[2];
      for (int t = 0; t < 2; t++) pick[t] = (li < m && (ii >= nx || hs.w[li] <= hs.w[ii])) ? li++ : ii++;
      hs.w[nx] = hs.w[pick[0]] + hs.w[pick[1]];
      hs.parent[pick[0]] = hs.parent[pick[1]] = (uint16_t)nx;
      nx++;
    }
    const int root = 2 * m - 2;
    hs.depth[root] = 0;
    for (int k = root - 1; k >= 0; k--) hs.depth[k] = hs.depth[hs.parent[k]] + 1;
    int maxd = 0;
    for (int d = 0; d <= m; d++) hs.count[d] = 0;
    for (int k = 0; k < m; k++) hs.count[hs.depth[k]]++, maxd = max(maxd, (int)hs.depth[k]);
    /* JPEG Annex K.3: move leaves up until no code is longer than the limit; the code stays complete */
    for (int i = maxd; i > limit; i--)
      while (hs.count[i] > 0) {
        int j = i - 2;
        while (hs.count[j] == 0) j--;
        hs.count[i] -= 2;
        hs.count[i - 1]++;
        hs.count[j + 1] += 2;
        hs.count[j]--;
      }
    /* the most frequent symbols take the shortest lengths */
    int k = m - 1;
    for (int l = 1; l <= limit; l++)
      for (int c = 0; c < hs.count[l]; c++) len[hs.sorted[k--]] = (uint8_t)l;
    /* canonical codes (RFC 1951 3.2.2), bit-reversed for LSB-first output */
    for (int b = 0; b < 16; b++) hs.cnt[b] = 0;
    for (int i = 0; i < n; i++) hs.cnt[len[i]]++;
    hs.cnt[0] = 0;
    uint32_t c = 0;
    for (int b = 1; b <= limit; b++) c = (c + hs.cnt[b - 1]) << 1, hs.next[b] = c;
    for (int i = 0; i < n; i++)
      if (len[i]) code[i] = (uint16_t)(__brev(hs.next[len[i]]++) >> (32 - len[i]));
  }
  __syncwarp();
}

__device__ __forceinline__ void put_bits(uint32_t *buf, uint32_t pos, uint32_t v, uint32_t nb) {
  if (!nb) return;
  const uint32_t w = pos >> 5, o = pos & 31;
  atomicOr(&buf[w], v << o);
  if (o + nb > 32) atomicOr(&buf[w + 1], v >> (32 - o));
}

/* bits of one token under the block's codes */
__device__ __forceinline__ uint32_t token_bits(uint32_t t, const CodeWork &cw) {
  if (!(t & MATCH_FLAG)) return cw.len_ll[t];
  uint32_t lc, lx, lv, dc, dx, dv;
  len_code((t >> 16) & 0x1ff, lc, lx, lv);
  dist_code(t & 0xffff, dc, dx, dv);
  return cw.len_ll[lc] + lx + cw.len_d[dc] + dx;
}

__device__ __forceinline__ uint32_t put_token(uint32_t *buf, uint32_t pos, uint32_t t, const CodeWork &cw) {
  if (!(t & MATCH_FLAG)) {
    put_bits(buf, pos, cw.code_ll[t], cw.len_ll[t]);
    return pos + cw.len_ll[t];
  }
  uint32_t lc, lx, lv, dc, dx, dv;
  len_code((t >> 16) & 0x1ff, lc, lx, lv);
  dist_code(t & 0xffff, dc, dx, dv);
  put_bits(buf, pos, cw.code_ll[lc] | (lv << cw.len_ll[lc]), cw.len_ll[lc] + lx);
  pos += cw.len_ll[lc] + lx;
  put_bits(buf, pos, cw.code_d[dc] | (dv << cw.len_d[dc]), cw.len_d[dc] + dx);
  return pos + cw.len_d[dc] + dx;
}

/* members: (offset in `in`, length) per member; scratch: BGZF_INPUT words per member (matches, then
 * tokens); slots: BGZF_SLOT bytes per member; sizes: BSIZE per member */
__global__ void __launch_bounds__(NT, 1)
k_bgzf_deflate(const uint8_t *__restrict__ in, const uint2 *__restrict__ members, uint32_t *__restrict__ scratch,
               uint8_t *__restrict__ slots, uint32_t *__restrict__ sizes) {
  extern __shared__ __align__(16) uint8_t smem[];
  uint32_t *s_in = (uint32_t *)smem;
  uint16_t *s_prev = (uint16_t *)(smem + SMEM_IN);
  uint32_t *s_bits = (uint32_t *)(smem + SMEM_IN); /* over the chain links once they are dead */
  uint16_t *s_head = (uint16_t *)(smem + SMEM_IN + SMEM_PREV);
  CodeWork &cw = *(CodeWork *)(smem + SMEM_IN + SMEM_PREV);
  __shared__ uint32_t s_crc_table[256];
  __shared__ uint32_t s_ntok[NSEG], s_segbits[NSEG];
  __shared__ uint32_t s_crc_part[NT / 32];
  __shared__ uint32_t s_total_bits, s_stored;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint2 mem = members[blockIdx.x];
  const uint8_t *src = in + mem.x;
  const uint32_t n = mem.y;
  uint32_t *match = scratch + (size_t)blockIdx.x * BGZF_INPUT;

  /* stage the member as little-endian words, zero padded */
  for (uint32_t w = tid; w < SMEM_IN / 4; w += NT) {
    uint32_t v = 0;
    for (uint32_t b = 0; b < 4; b++)
      if (4 * w + b < n) v |= (uint32_t)src[4 * w + b] << (8 * b);
    s_in[w] = v;
  }
  for (uint32_t i = tid; i < (1u << HBITS); i += NT) s_head[i] = 0;
  for (uint32_t i = tid; i < 256; i += NT) {
    uint32_t c = i;
    for (int k = 0; k < 8; k++) c = c & 1 ? (c >> 1) ^ 0xedb88320u : c >> 1;
    s_crc_table[i] = c;
  }
  __syncthreads();
  for (uint32_t p = tid; p < n; p += NT) s_prev[p] = p + 4 <= n ? (uint16_t)hash4(load32(s_in, p)) : (uint16_t)NO_HASH;
  __syncthreads();

  if (warp == 0) {
    /* chain links: s_prev[p] = distance to the previous position with the same hash (0: none) */
    for (uint32_t base = 0; base < n; base += 32) {
      const uint32_t p = base + lane;
      const uint32_t h = p < n ? s_prev[p] : NO_HASH;
      const uint32_t group = __match_any_sync(0xffffffffu, h);
      const uint32_t lower = group & ((1u << lane) - 1);
      uint32_t dist = 0;
      if (h != NO_HASH) {
        if (lower)
          dist = lane - (31 - __clz(lower));
        else if (const uint32_t hd = s_head[h])
          dist = p - (hd - 1);
      }
      __syncwarp();
      if (h != NO_HASH && (group >> lane) == 1) s_head[h] = (uint16_t)(p + 1);
      if (p < n) s_prev[p] = (uint16_t)dist;
      __syncwarp();
    }
  } else {
    /* CRC32 of the member by the other warps, one slice each */
    const uint32_t nw = NT - 32, t = tid - 32;
    const uint32_t slice = (n + nw - 1) / nw;
    const uint32_t a = min(n, t * slice), b = min(n, a + slice);
    uint32_t c = 0;
    for (uint32_t i = a; i < b; i++) c = s_crc_table[(c ^ byte_at(s_in, i)) & 0xff] ^ (c >> 8);
    if (b > a) c = crc_mulmod(crc_x8n(n - b), c);
    for (int o = 16; o; o >>= 1) c ^= __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0) s_crc_part[warp] = c;
  }
  __syncthreads();

  /* longest match at every position */
  for (uint32_t p = tid; p < n; p += NT) {
    uint32_t best = 3, bestd = 0;
    if (p + 4 <= n) {
      const uint32_t maxlen = min(258u, n - p);
      uint32_t cand = p, d = s_prev[p];
      for (int depth = 0; d && depth < CHAIN; depth++) {
        cand -= d;
        if (p - cand > 32768) break;
        if (byte_at(s_in, cand + best) == byte_at(s_in, p + best)) {
          uint32_t l = 0;
          while (l < maxlen) {
            const uint32_t x = load32(s_in, cand + l) ^ load32(s_in, p + l);
            if (x) {
              l += (__ffs(x) - 1) >> 3;
              break;
            }
            l += 4;
          }
          l = min(l, maxlen);
          if (l > best) {
            best = l, bestd = p - cand;
            if (l >= NICE || l == maxlen) break;
          }
        }
        d = s_prev[cand];
      }
    }
    match[p] = bestd ? (best << 16) | bestd : 0;
  }
  __syncthreads();

  /* the chain links and head table are dead: clear the histograms and the bit buffer */
  for (uint32_t i = tid; i < sizeof(CodeWork) / 4; i += NT) ((uint32_t *)&cw)[i] = 0;
  const uint32_t bit_words = (n + 5) / 4 + 2;
  for (uint32_t i = tid; i < bit_words; i += NT) s_bits[i] = 0;
  __syncthreads();

  /* lazy parse of each segment into tokens, written over its own matches */
  const uint32_t seg = (n + NSEG - 1) / NSEG;
  if (tid < NSEG) {
    const uint32_t s0 = min(n, tid * seg), s1 = min(n, s0 + seg);
    uint32_t p = s0, k = 0;
    while (p < s1) {
      const uint32_t m = match[p];
      uint32_t L = min(m >> 16, s1 - p);
      if (L >= 4 && L < LAZY && p + 1 < s1 && min(match[p + 1] >> 16, s1 - p - 1) > L) L = 0;
      uint32_t t;
      if (L >= 4) {
        uint32_t lc, lx, lv, dc, dx, dv;
        len_code(L, lc, lx, lv);
        dist_code(m & 0xffff, dc, dx, dv);
        atomicAdd(&cw.hist_ll[lc], 1u);
        atomicAdd(&cw.hist_d[dc], 1u);
        t = MATCH_FLAG | (L << 16) | (m & 0xffff);
        p += L;
      } else {
        t = byte_at(s_in, p);
        atomicAdd(&cw.hist_ll[t], 1u);
        p++;
      }
      match[s0 + k++] = t;
    }
    s_ntok[tid] = k;
  }
  if (tid == 0) atomicAdd(&cw.hist_ll[256], 1u);
  __syncthreads();

  if (warp == 0) build_code(cw.hist_ll, 286, 15, cw.len_ll, cw.code_ll, cw.hs[0]);
  if (warp == 1) build_code(cw.hist_d, 30, 15, cw.len_d, cw.code_d, cw.hs[1]);
  __syncthreads();
  if (warp == 0) {
    if (lane == 0) {
      int hlit = 286, hdist = 30;
      while (hlit > 257 && !cw.len_ll[hlit - 1]) hlit--;
      while (hdist > 1 && !cw.len_d[hdist - 1]) hdist--;
      const int total = hlit + hdist;
      uint32_t nr = 0;
      for (int i = 0; i < total;) {
        const uint32_t v = i < hlit ? cw.len_ll[i] : cw.len_d[i - hlit];
        int run = 1;
        while (i + run < total && (i + run < hlit ? cw.len_ll[i + run] : cw.len_d[i + run - hlit]) == v) run++;
        int r = run;
        if (v == 0) {
          while (r >= 11) {
            const int t = min(r, 138);
            cw.rle[nr++] = (uint16_t)(18 | (t - 11) << 5);
            r -= t;
          }
          if (r >= 3) cw.rle[nr++] = (uint16_t)(17 | (r - 3) << 5), r = 0;
        } else {
          cw.rle[nr++] = (uint16_t)v;
          r--;
          while (r >= 3) {
            const int t = min(r, 6);
            cw.rle[nr++] = (uint16_t)(16 | (t - 3) << 5);
            r -= t;
          }
        }
        while (r-- > 0) cw.rle[nr++] = (uint16_t)v;
        i += run;
      }
      for (uint32_t i = 0; i < nr; i++) cw.hist_cl[cw.rle[i] & 31]++;
      cw.n_rle = nr, cw.hlit = hlit, cw.hdist = hdist;
    }
    __syncwarp();
    build_code(cw.hist_cl, 19, 7, cw.len_cl, cw.code_cl, cw.hs[0]);
    if (lane == 0) {
      int hclen = 19;
      while (hclen > 4 && !cw.len_cl[c_cl_order[hclen - 1]]) hclen--;
      uint32_t bits = 3 + 5 + 5 + 4 + 3 * hclen;
      for (uint32_t i = 0; i < cw.n_rle; i++) {
        const uint32_t s = cw.rle[i] & 31;
        bits += cw.len_cl[s] + (s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0);
      }
      cw.hclen = hclen, cw.header_bits = bits;
    }
  }
  __syncthreads();

  if (tid < NSEG) {
    const uint32_t s0 = min(n, tid * seg);
    uint32_t bits = 0;
    for (uint32_t k = 0; k < s_ntok[tid]; k++) bits += token_bits(match[s0 + k], cw);
    s_segbits[tid] = bits;
  }
  __syncthreads();
  if (tid == 0) {
    uint32_t off = cw.header_bits;
    for (int s = 0; s < NSEG; s++) {
      const uint32_t b = s_segbits[s];
      s_segbits[s] = off;
      off += b;
    }
    off += cw.len_ll[256];
    s_total_bits = off;
    s_stored = (off + 7) / 8 >= n + 5;
  }
  __syncthreads();

  uint32_t *bits = s_bits;
  const bool stored = s_stored;
  if (!stored) {
    if (tid == 0) {
      uint32_t pos = 0;
      put_bits(bits, pos, 1, 1), pos += 1; /* BFINAL */
      put_bits(bits, pos, 2, 2), pos += 2; /* BTYPE 2: dynamic Huffman codes */
      put_bits(bits, pos, cw.hlit - 257, 5), pos += 5;
      put_bits(bits, pos, cw.hdist - 1, 5), pos += 5;
      put_bits(bits, pos, cw.hclen - 4, 4), pos += 4;
      for (uint32_t i = 0; i < cw.hclen; i++) put_bits(bits, pos, cw.len_cl[c_cl_order[i]], 3), pos += 3;
      for (uint32_t i = 0; i < cw.n_rle; i++) {
        const uint32_t s = cw.rle[i] & 31, x = cw.rle[i] >> 5;
        put_bits(bits, pos, cw.code_cl[s], cw.len_cl[s]), pos += cw.len_cl[s];
        const uint32_t nx = s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0;
        put_bits(bits, pos, x, nx), pos += nx;
      }
      put_bits(bits, s_total_bits - cw.len_ll[256], cw.code_ll[256], cw.len_ll[256]); /* end of block */
    }
    if (tid < NSEG) {
      const uint32_t s0 = min(n, tid * seg);
      uint32_t pos = s_segbits[tid];
      for (uint32_t k = 0; k < s_ntok[tid]; k++) pos = put_token(bits, pos, match[s0 + k], cw);
    }
  }
  __syncthreads();

  uint32_t crc = 0;
  for (int w = 1; w < NT / 32; w++) crc ^= s_crc_part[w];
  crc ^= crc_mulmod(crc_x8n(n), 0xffffffffu) ^ 0xffffffffu;
  const uint32_t dlen = stored ? n + 5 : (s_total_bits + 7) / 8;
  const uint32_t bsize = 18 + dlen + 8;
  uint8_t *out = slots + (size_t)blockIdx.x * BGZF_SLOT;
  for (uint32_t i = tid; i < bsize; i += NT) {
    uint32_t v;
    if (i < 18) {
      v = i < 16 ? c_gz_header[i] : i == 16 ? (bsize - 1) & 0xff : (bsize - 1) >> 8;
    } else if (i < 18 + dlen) {
      const uint32_t j = i - 18;
      if (!stored)
        v = byte_at(bits, j);
      else if (j >= 5)
        v = byte_at(s_in, j - 5);
      else
        v = j == 0 ? 1 : j == 1 ? n & 0xff : j == 2 ? n >> 8 : j == 3 ? ~n & 0xff : (~n >> 8) & 0xff;
    } else {
      const uint32_t j = i - 18 - dlen;
      v = ((j < 4 ? crc : n) >> (8 * (j & 3))) & 0xff;
    }
    out[i] = (uint8_t)v;
  }
  if (tid == 0) sizes[blockIdx.x] = bsize;
}

/* offs[0..nm] = exclusive scan of sizes (one CTA of 1024 threads) */
__global__ void __launch_bounds__(1024) k_bgzf_scan(const uint32_t *__restrict__ sizes, uint32_t nm, uint64_t *__restrict__ offs) {
  __shared__ uint64_t s[1024];
  const uint32_t tid = threadIdx.x, per = (nm + 1023) / 1024;
  const uint32_t a = min(nm, tid * per), b = min(nm, a + per);
  uint64_t sum = 0;
  for (uint32_t i = a; i < b; i++) sum += sizes[i];
  s[tid] = sum;
  __syncthreads();
  for (uint32_t o = 1; o < 1024; o <<= 1) {
    const uint64_t v = tid >= o ? s[tid - o] : 0;
    __syncthreads();
    s[tid] += v;
    __syncthreads();
  }
  uint64_t off = s[tid] - sum;
  for (uint32_t i = a; i < b; i++) offs[i] = off, off += sizes[i];
  if (tid == 1023) offs[nm] = s[1023];
}

/* members back to back: one CTA per member */
__global__ void __launch_bounds__(256) k_bgzf_compact(const uint8_t *__restrict__ slots, const uint64_t *__restrict__ offs,
                                                     uint8_t *__restrict__ out) {
  const uint8_t *src = slots + (size_t)blockIdx.x * BGZF_SLOT;
  uint8_t *dst = out + offs[blockIdx.x];
  const uint32_t n = (uint32_t)(offs[blockIdx.x + 1] - offs[blockIdx.x]);
  for (uint32_t i = threadIdx.x; i < n; i += 256) dst[i] = src[i];
}

}  // namespace

#define DEFLATE_TRY(expr)                                                                                    \
  do {                                                                                                       \
    cudaError_t _e = (expr);                                                                                 \
    if (_e != cudaSuccess)                                                                                   \
      return nh_set_error(_e == cudaErrorMemoryAllocation ? NH_ERR_NOMEM : NH_ERR_CUDA, "GPU deflate: %s failed: %s", #expr, \
                          cudaGetErrorString(_e));                                                           \
  } while (0)

GpuDeflater::~GpuDeflater() {
  if (device_ < 0) return;
  cudaSetDevice(device_);
  if (stream_) cudaStreamSynchronize(stream_);
  cudaFree(d_in_), cudaFree(d_members_), cudaFree(d_scratch_), cudaFree(d_slots_), cudaFree(d_sizes_), cudaFree(d_offs_),
      cudaFree(d_out_);
  cudaFreeHost(h_in_), cudaFreeHost(h_members_), cudaFreeHost(h_offs_), cudaFreeHost(h_out_);
  if (stream_) cudaStreamDestroy(stream_);
}

int GpuDeflater::open(int device, size_t batch_bytes) {
  int nd = 0;
  if (cudaGetDeviceCount(&nd) != cudaSuccess || nd < 1) {
    cudaGetLastError();
    return nh_set_error(NH_ERR_CUDA, "GPU deflate: no CUDA device (no CPU path)");
  }
  if (device < 0 || device >= nd) return nh_set_error(NH_ERR_INVALID, "GPU deflate: no CUDA device %d", device);
  device_ = device;
  batch_ = std::max<size_t>(BGZF_INPUT, (batch_bytes + BGZF_INPUT - 1) / BGZF_INPUT * BGZF_INPUT);
  /* blocks that are not multiples of 0xff00 end in short members: allow one per MiB of input besides */
  max_members_ = batch_ / BGZF_INPUT + (batch_ >> 20) + 1;
  const size_t out_cap = max_members_ * (size_t)BGZF_SLOT;
  DEFLATE_TRY(cudaSetDevice(device));
  DEFLATE_TRY(cudaFuncSetAttribute(k_bgzf_deflate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
  DEFLATE_TRY(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
  DEFLATE_TRY(cudaMalloc(&d_in_, batch_ + 16));
  DEFLATE_TRY(cudaMalloc(&d_members_, max_members_ * sizeof(uint2)));
  DEFLATE_TRY(cudaMalloc(&d_scratch_, max_members_ * (size_t)BGZF_INPUT * 4));
  DEFLATE_TRY(cudaMalloc(&d_slots_, out_cap));
  DEFLATE_TRY(cudaMalloc(&d_sizes_, max_members_ * 4));
  DEFLATE_TRY(cudaMalloc(&d_offs_, (max_members_ + 1) * 8));
  DEFLATE_TRY(cudaMalloc(&d_out_, out_cap));
  DEFLATE_TRY(cudaHostAlloc(&h_in_, batch_ + 16, cudaHostAllocDefault));
  DEFLATE_TRY(cudaHostAlloc(&h_members_, max_members_ * sizeof(uint2), cudaHostAllocDefault));
  DEFLATE_TRY(cudaHostAlloc(&h_offs_, (max_members_ + 1) * 8, cudaHostAllocDefault));
  DEFLATE_TRY(cudaHostAlloc(&h_out_, out_cap, cudaHostAllocDefault));
  return NH_OK;
}

int GpuDeflater::launch(size_t n_members) {
  const uint32_t nm = (uint32_t)n_members;
  k_bgzf_deflate<<<nm, NT, SMEM_BYTES, stream_>>>(d_in_, (const uint2 *)d_members_, d_scratch_, d_slots_, d_sizes_);
  k_bgzf_scan<<<1, 1024, 0, stream_>>>(d_sizes_, nm, d_offs_);
  k_bgzf_compact<<<nm, 256, 0, stream_>>>(d_slots_, d_offs_, d_out_);
  DEFLATE_TRY(cudaGetLastError());
  return NH_OK;
}

int GpuDeflater::run(size_t bytes, size_t n_members) {
  DEFLATE_TRY(cudaSetDevice(device_));
  DEFLATE_TRY(cudaMemcpyAsync(d_in_, h_in_, bytes, cudaMemcpyHostToDevice, stream_));
  DEFLATE_TRY(cudaMemcpyAsync(d_members_, h_members_, n_members * sizeof(uint2), cudaMemcpyHostToDevice, stream_));
  if (int rc = launch(n_members)) return rc;
  DEFLATE_TRY(cudaMemcpyAsync(h_offs_, d_offs_, (n_members + 1) * 8, cudaMemcpyDeviceToHost, stream_));
  DEFLATE_TRY(cudaStreamSynchronize(stream_));
  DEFLATE_TRY(cudaMemcpyAsync(h_out_, d_out_, h_offs_[n_members], cudaMemcpyDeviceToHost, stream_));
  DEFLATE_TRY(cudaStreamSynchronize(stream_));
  return NH_OK;
}

int GpuDeflater::compress(const std::vector<Span> &blocks, std::vector<std::string> &out) {
  out.assign(blocks.size(), std::string());
  return compress(blocks, [&](size_t b, const uint8_t *p, size_t n) { out[b].append((const char *)p, n); });
}

int GpuDeflater::compress(const std::vector<Span> &blocks, const Sink &sink) {
  std::vector<uint32_t> owner; /* block of each member of the round */
  size_t bytes = 0;
  auto flush = [&]() -> int {
    if (owner.empty()) return NH_OK;
    if (int rc = run(bytes, owner.size())) return rc;
    for (size_t m = 0; m < owner.size(); m++) sink(owner[m], h_out_ + h_offs_[m], (size_t)(h_offs_[m + 1] - h_offs_[m]));
    owner.clear();
    bytes = 0;
    return NH_OK;
  };
  for (size_t b = 0; b < blocks.size(); b++)
    for (size_t pos = 0; pos < blocks[b].second; pos += BGZF_INPUT) {
      const size_t len = std::min<size_t>(BGZF_INPUT, blocks[b].second - pos);
      if (bytes + len > batch_ || owner.size() == max_members_)
        if (int rc = flush()) return rc;
      memcpy(h_in_ + bytes, blocks[b].first + pos, len);
      h_members_[owner.size()] = make_uint2((uint32_t)bytes, (uint32_t)len);
      owner.push_back((uint32_t)b);
      bytes += len;
    }
  return flush();
}

int GpuDeflater::time_kernels(const uint8_t *in, size_t n, int iters, double *seconds) {
  if (n > batch_) return nh_set_error(NH_ERR_CAPACITY, "GPU deflate: %zu bytes exceed the batch of %zu", n, batch_);
  size_t nm = 0;
  for (size_t pos = 0; pos < n; pos += BGZF_INPUT, nm++)
    h_members_[nm] = make_uint2((uint32_t)pos, (uint32_t)std::min<size_t>(BGZF_INPUT, n - pos));
  if (!nm) return nh_set_error(NH_ERR_INVALID, "GPU deflate: nothing to time");
  memcpy(h_in_, in, n);
  DEFLATE_TRY(cudaSetDevice(device_));
  DEFLATE_TRY(cudaMemcpyAsync(d_in_, h_in_, n, cudaMemcpyHostToDevice, stream_));
  DEFLATE_TRY(cudaMemcpyAsync(d_members_, h_members_, nm * sizeof(uint2), cudaMemcpyHostToDevice, stream_));
  if (int rc = launch(nm)) return rc; /* warm-up */
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  DEFLATE_TRY(cudaEventCreate(&e0));
  DEFLATE_TRY(cudaEventCreate(&e1));
  int rc = NH_OK;
  cudaEventRecord(e0, stream_);
  for (int i = 0; i < iters && rc == NH_OK; i++) rc = launch(nm);
  cudaEventRecord(e1, stream_);
  float ms = 0;
  const cudaError_t e = cudaEventSynchronize(e1);
  if (rc == NH_OK && e == cudaSuccess) cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (rc) return rc;
  DEFLATE_TRY(e);
  *seconds = 1e-3 * ms / iters;
  return NH_OK;
}

static int bgzf_device_check(int device) {
  int nd = 0;
  if (cudaGetDeviceCount(&nd) != cudaSuccess || nd < 1) {
    cudaGetLastError();
    return nh_set_error(NH_ERR_CUDA, "no CUDA device (no CPU path)");
  }
  if (device < 0 || device >= nd) return nh_set_error(NH_ERR_INVALID, "no CUDA device %d", device);
  return NH_OK;
}

extern "C" int nh_bgzf_compress(int device, const uint8_t *in, size_t n, uint8_t *out, size_t out_cap, size_t *out_len) {
  if ((n && (!in || !out)) || !out_len) return nh_set_error(NH_ERR_INVALID, "nh_bgzf_compress: null argument");
  const size_t need = (n + BGZF_INPUT - 1) / BGZF_INPUT * (size_t)BGZF_SLOT;
  if (out_cap < need)
    return nh_set_error(NH_ERR_CAPACITY, "nh_bgzf_compress: %zu input bytes need %zu output bytes, %zu given", n, need, out_cap);
  if (int rc = bgzf_device_check(device)) return rc;
  *out_len = 0;
  if (!n) return NH_OK;
  GpuDeflater gd;
  if (int rc = gd.open(device, std::min(n, GpuDeflater::kBatchBytes))) return rc;
  size_t at = 0; /* members go straight into the caller's buffer, which holds 65536 bytes per member */
  const int rc = gd.compress({{in, n}}, [&](size_t, const uint8_t *p, size_t len) {
    memcpy(out + at, p, len);
    at += len;
  });
  if (rc == NH_OK) *out_len = at;
  return rc;
}

extern "C" int nh_bench_bgzf(int device, const uint8_t *in, size_t n, int iters, double *out_seconds) {
  if (!in || !n || n > (size_t(1) << 30) || iters < 1 || !out_seconds)
    return nh_set_error(NH_ERR_INVALID, "nh_bench_bgzf: bad argument (1 byte to 1 GiB of input, iters >= 1)");
  if (int rc = bgzf_device_check(device)) return rc;
  GpuDeflater gd;
  if (int rc = gd.open(device, n)) return rc;
  return gd.time_kernels(in, n, iters, out_seconds);
}
