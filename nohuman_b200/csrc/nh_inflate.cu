/*
 * nh_inflate.cu — gzip decompression on the GPU for ordinary single-stream gzip (one member or many,
 * every deflate block type), with no index and no cooperation from the writer: two-stage speculative
 * decoding as in pugz and rapidgzip.
 *
 * The compressed stream goes through in WINDOWS: up to `window` new bytes per window plus the bytes
 * carried from the previous one.  A window is cut into CHUNKS of `chunk` bytes.
 *   k_gunzip_find    one warp per chunk after the first finds the first bit offset at or after the
 *                    chunk's start where a deflate block can begin: a stored block (LEN == ~NLEN, zero
 *                    padding) or a dynamic-Huffman block whose header passes zlib's inflate_table rules
 *                    and whose first NTEST symbols decode without an invalid code.  Lanes test 32 bit
 *                    offsets at a time; fixed-Huffman blocks are not searched for.
 *   k_gunzip_decode  one warp per chunk decodes from its candidate (chunk 0: from the window's known
 *                    start) to the first block boundary at or beyond the start of the next chunk that
 *                    has a candidate.  All lanes decode the same symbol, so control flow is warp-uniform;
 *                    stored runs and match copies are written by the lanes in parallel.  The output is
 *                    16-bit symbols: 0-255 a byte, 256 + i byte i of the unknown 32 KiB before the chunk
 *                    (a marker).  Member ends record CRC32 and ISIZE and the next gzip header is parsed.
 * The host chains the chunks: a chunk's output is accepted only when its confirmed predecessor stopped
 * exactly on its start bit; otherwise it is decoded again from that stop (a repair; all of a round in one
 * launch).  By induction the result is what zlib gives, however wrong the finder is.
 *   k_gunzip_window  one CTA carries the last 32 KiB of resolved output through the accepted chunks.
 *   k_gunzip_resolve replaces every marker from its chunk's window and writes bytes at prefix offsets;
 *                    a marker before the start of its member is zlib's "invalid distance too far back".
 *   k_gunzip_crc     CRC32 per piece of output; the host joins the pieces of a member (crc32_combine)
 *                    and checks every member's CRC32 and ISIZE.
 * A chunk whose output outgrows its slot keeps decoding without storing (to find its stop and size) and
 * is then decoded again into a spill buffer at that size, which bounds device memory at any compression
 * ratio.
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>
#include <zlib.h>

#include <algorithm>
#include <chrono>
#include <string>
#include <vector>

#include "nh_crc.cuh"
#include "nh_internal.h"

/* shared with GpuInflater (nh_internal.h) */
struct NhGzMember {
  uint64_t out;  /* output symbols of the chunk before the member's end */
  uint32_t crc, isize;
};

/* One decode of one chunk.  stop/out_len/members/stop_mode describe where it stopped: the block start
 * past the threshold (ST_STOPPED), the end of the stream (ST_END), or, for ST_NEED, the last block start
 * or member end it passed before the input ran out. */
struct NhGzChunk {
  uint64_t start, stop, out_len, total_out; /* total_out: symbols decoded up to where decoding ended */
  uint32_t status, members, total_members, stop_mode, start_mode, pad;
};

struct NhGzEmit {
  const uint16_t *sym;
  uint64_t len, out; /* symbols, output offset */
  uint32_t hist;     /* bytes of the chunk's member before the chunk (at most 32 KiB) */
  uint32_t pad;
};

/* one decode: a chunk from a start, into an output buffer */
struct NhGzJob {
  uint64_t start;       /* NONE: the chunk's candidate (chunk 0: start0) */
  uint32_t mode;
  int32_t chunk;
  uint16_t *out;
  uint64_t cap;         /* symbols that fit in out */
  NhGzMember *mrec;
  uint32_t mcap;
  uint32_t soft_mem;    /* stop at the first boundary with this many member ends (spill) */
  uint64_t soft_out;    /* ... or this many symbols */
  NhGzChunk *rec;
};

namespace {

using MemberEnd = NhGzMember;
using Job = NhGzJob;
using ChunkRec = NhGzChunk;
using Emit = NhGzEmit;

constexpr uint64_t NONE = ~0ull;
constexpr int LB = 10;            /* litlen fast-table bits */
constexpr int DB = 8;             /* distance fast-table bits */
constexpr int NTEST = 256;        /* symbols a dynamic-block candidate must decode */
constexpr int WARPS = 4;          /* warps per CTA of find / decode */
constexpr uint32_t HIST = 32768;  /* deflate window */
constexpr uint32_t SEG = 65536;   /* output bytes per CRC piece */

enum { ST_STOPPED = 0, ST_END, ST_CORRUPT, ST_NEED };
enum { MODE_BLOCK = 0, MODE_HEADER = 1 };




struct Win {
  const uint32_t *in; /* window bytes as words, zero padded */
  uint64_t nbits;
  uint64_t chunk_bits;
  uint32_t n_chunks, eof;
};

template <int B, int N>
struct HT {
  uint16_t fast[1 << B]; /* sym << 4 | len; 0: longer than B bits or no code */
  uint16_t cnt[16], first[16], off[16], cur[16];
  uint16_t sym[N]; /* symbols by (length, value): puff's canonical order */
};

struct WarpTabs {
  HT<LB, 288> ll; /* also the code-length code while the lengths are read */
  HT<DB, 32> d;
  uint8_t lens[320];
};

__constant__ uint16_t c_lbase[29] = {3,  4,  5,  6,  7,  8,  9,  10, 11,  13,  15,  17,  19,  23, 27,
                                     31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t c_lext[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint16_t c_dbase[30] = {1,   2,   3,   4,   5,   7,    9,    13,   17,   25,   33,   49,    65,    97,    129,
                                     193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t c_dext[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__constant__ uint8_t c_cl_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

constexpr unsigned FULL = 0xffffffffu;

/* at least 64 bits of the stream from bit `pos` (the window is padded with zero words) */
__device__ __forceinline__ uint64_t peek(const uint32_t *in, uint64_t pos) {
  const uint64_t w = pos >> 5;
  const uint32_t sh = pos & 31;
  uint64_t v = ((uint64_t)__ldg(in + w) | (uint64_t)__ldg(in + w + 1) << 32) >> sh;
  if (sh) v |= (uint64_t)__ldg(in + w + 2) << (64 - sh);
  return v;
}

__device__ __forceinline__ uint32_t byte_at(const uint32_t *in, uint64_t i) { return (__ldg(in + (i >> 2)) >> ((i & 3) * 8)) & 0xff; }

/* Canonical code from lens[0..n) (warp-collective).  Returns zlib's verdict: no oversubscribed code;
 * an incomplete code only with max length 1, never for the code-length code; an empty code is allowed
 * for distances only (litlen always needs code 256; an empty code-length code decodes nothing). */
template <int B, int N>
__device__ bool build(HT<B, N> &t, const uint8_t *lens, int n, bool codes) {
  const int lane = threadIdx.x & 31;
  if (lane < 16) t.cnt[lane] = 0, t.cur[lane] = 0;
  for (int e = lane; e < (1 << B); e += 32) t.fast[e] = 0;
  __syncwarp();
  for (int base = 0; base < n; base += 32) {
    const int i = base + lane;
    const uint32_t l = i < n ? lens[i] : 0;
    const uint32_t m = __match_any_sync(FULL, l);
    if (l && lane == __ffs(m) - 1) t.cnt[l] += __popc(m);
    __syncwarp();
  }
  bool ok = true;
  if (lane == 0) {
    int left = 1, max = 0;
    for (int l = 1; l <= 15; l++) {
      left = (left << 1) - t.cnt[l];
      if (left < 0) ok = false;
      if (t.cnt[l]) max = l;
    }
    if (ok && left > 0 && (codes || max != 1) && max != 0) ok = false;
    if (codes && max == 0) ok = false;
    uint32_t code = 0, off = 0;
    t.cnt[0] = 0;
    for (int l = 1; l <= 15; l++) {
      code = (code + t.cnt[l - 1]) << 1;
      t.first[l] = (uint16_t)code;
      t.off[l] = (uint16_t)off;
      off += t.cnt[l];
    }
  }
  ok = __shfl_sync(FULL, ok, 0);
  __syncwarp();
  if (!ok) return false;
  for (int base = 0; base < n; base += 32) {
    const int i = base + lane;
    const uint32_t l = i < n ? lens[i] : 0;
    const uint32_t m = __match_any_sync(FULL, l);
    if (l) {
      const uint32_t r = t.cur[l] + __popc(m & ((1u << lane) - 1));
      t.sym[t.off[l] + r] = (uint16_t)i;
      if (l <= B) {
        const uint32_t rc = __brev(t.first[l] + r) >> (32 - l);
        for (uint32_t k = 0; k < (1u << (B - l)); k++) t.fast[rc | k << l] = (uint16_t)(i << 4 | l);
      }
    }
    __syncwarp();
    if (l && lane == __ffs(m) - 1) t.cur[l] += __popc(m);
    __syncwarp();
  }
  return true;
}

/* symbol at the front of v, its length in `len`; -1 for a code the table does not have */
template <int B, int N>
__device__ __forceinline__ int hdecode(const HT<B, N> &t, uint64_t v, uint32_t &len) {
  const uint32_t e = t.fast[v & ((1u << B) - 1)];
  if (e) {
    len = e & 15;
    return (int)(e >> 4);
  }
  int code = 0, first = 0, index = 0;
  for (int l = 1; l <= 15; l++) {
    code |= (int)((v >> (l - 1)) & 1);
    const int c = t.cnt[l];
    if (code - first < c) {
      len = l;
      return t.sym[index + code - first];
    }
    index += c;
    first = (first + c) << 1;
    code <<= 1;
  }
  return -1;
}

/* the dynamic block header at `pos` (after BFINAL/BTYPE): tables in tb and pos advanced (ST_STOPPED);
 * ST_NEED when the window ends inside it; ST_CORRUPT when zlib rejects it.  Nothing past the window's
 * end is acted on: bits beyond w.nbits are only ever read as a reason to wait for more input. */
__device__ int read_dynamic(const Win &w, uint64_t &pos, WarpTabs &tb) {
  const int lane = threadIdx.x & 31;
  if (pos + 14 > w.nbits) return ST_NEED;
  const uint64_t v = peek(w.in, pos);
  const uint32_t nlen = 257 + (v & 31), ndist = 1 + ((v >> 5) & 31), ncl = 4 + ((v >> 10) & 15);
  if (nlen > 286 || ndist > 30) return ST_CORRUPT;
  pos += 14;
  if (pos + 3 * ncl > w.nbits) return ST_NEED;
  if (lane < 19) tb.lens[c_cl_order[lane]] = lane < (int)ncl ? (uint8_t)((peek(w.in, pos + 3 * lane) & 7)) : 0;
  pos += 3 * ncl;
  __syncwarp();
  if (!build(tb.ll, tb.lens, 19, true)) return ST_CORRUPT;
  /* the code lengths, warp-uniform */
  uint32_t i = 0, prev = 0;
  const uint32_t total = nlen + ndist;
  uint8_t *L = tb.lens;
  __syncwarp();
  while (i < total) {
    if (pos >= w.nbits) return ST_NEED;
    uint64_t b = peek(w.in, pos);
    uint32_t len;
    const int s = hdecode(tb.ll, b, len); /* the code-length code is complete: every 7 bits decode */
    const uint32_t nx = s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0;
    if (s < 0 || pos + len + nx > w.nbits) return s < 0 && pos + 7 <= w.nbits ? ST_CORRUPT : ST_NEED;
    pos += len;
    b >>= len;
    uint32_t val, rep;
    if (s < 16) {
      val = s, rep = 1;
    } else if (s == 16) {
      if (i == 0) return ST_CORRUPT;
      val = prev, rep = 3 + (b & 3);
    } else if (s == 17) {
      val = 0, rep = 3 + (b & 7);
    } else {
      val = 0, rep = 11 + (b & 127);
    }
    pos += nx;
    if (i + rep > total) return ST_CORRUPT;
    for (uint32_t j = lane; j < rep; j += 32) L[i + j] = (uint8_t)val;
    i += rep;
    prev = val;
  }
  __syncwarp();
  if (L[256] == 0) return ST_CORRUPT;
  if (!build(tb.ll, L, nlen, false)) return ST_CORRUPT;
  return build(tb.d, L + nlen, ndist, false) ? ST_STOPPED : ST_CORRUPT;
}

__device__ void load_fixed(WarpTabs &tb) {
  const int lane = threadIdx.x & 31;
  for (int i = lane; i < 288; i += 32) tb.lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : 8;
  __syncwarp();
  build(tb.ll, tb.lens, 288, false);
  __syncwarp();
  for (int i = lane; i < 32; i += 32) tb.lens[i] = 5;
  __syncwarp();
  build(tb.d, tb.lens, 32, false);
}

__device__ uint32_t crc_bytes(const uint32_t *in, uint64_t a, uint64_t b) {
  uint32_t c = 0xffffffffu;
  for (uint64_t i = a; i < b; i++) {
    c ^= byte_at(in, i);
    for (int k = 0; k < 8; k++) c = c & 1 ? (c >> 1) ^ 0xedb88320u : c >> 1;
  }
  return ~c;
}

/* first zero byte at or after byte p (warp-collective); NONE if the window ends first */
__device__ uint64_t find_zero(const Win &w, uint64_t p) {
  const int lane = threadIdx.x & 31;
  const uint64_t nbytes = w.nbits >> 3;
  for (;; p += 32) {
    if (p >= nbytes) return NONE;
    const uint64_t q = p + lane;
    const uint32_t z = __ballot_sync(FULL, q < nbytes && byte_at(w.in, q) == 0);
    if (z) return p + __ffs(z) - 1;
  }
}

/* gzip header at byte-aligned pos: ST_STOPPED with pos past it, ST_NEED, or ST_CORRUPT */
__device__ int read_header(const Win &w, uint64_t &pos) {
  const uint64_t h0 = pos >> 3, nbytes = w.nbits >> 3;
  if (h0 + 10 > nbytes) return ST_NEED;
  if (byte_at(w.in, h0) != 0x1f || byte_at(w.in, h0 + 1) != 0x8b || byte_at(w.in, h0 + 2) != 8) return ST_CORRUPT;
  const uint32_t flg = byte_at(w.in, h0 + 3);
  if (flg & 0xe0) return ST_CORRUPT;
  uint64_t p = h0 + 10;
  if (flg & 4) {
    if (p + 2 > nbytes) return ST_NEED;
    p += 2 + (byte_at(w.in, p) | byte_at(w.in, p + 1) << 8);
    if (p > nbytes) return ST_NEED;
  }
  for (uint32_t f = 8; f <= 16; f <<= 1)
    if (flg & f) {
      const uint64_t z = find_zero(w, p);
      if (z == NONE) return ST_NEED;
      p = z + 1;
    }
  if (flg & 2) {
    if (p + 2 > nbytes) return ST_NEED;
    const uint32_t want = byte_at(w.in, p) | byte_at(w.in, p + 1) << 8;
    if ((crc_bytes(w.in, h0, p) & 0xffff) != want) return ST_CORRUPT;
    p += 2;
  }
  pos = p << 3;
  return ST_STOPPED;
}

/*
 * Decodes from job.start (warp-uniform) and fills *rec.  stop_at: the first block start at or past it
 * ends the decode.  max_syms > 0 is the finder's test decode: it returns ST_STOPPED after that many
 * symbols or at the block's end, storing nothing.  mstart is the output position where the current
 * member's data begins (negative: before the chunk, which only the host can check).
 */
__device__ __forceinline__ void decode(const Win &w, const Job &job, uint64_t start, uint32_t mode, uint64_t stop_at, int max_syms, WarpTabs &tb,
                       ChunkRec &r) {
  const int lane = threadIdx.x & 31;
  uint64_t pos = start, o = 0;
  int64_t mstart = -(int64_t)HIST;
  uint32_t members = 0;
  bool fixed = false;
  int status;
  r.start = start, r.start_mode = mode;
  r.stop = start, r.stop_mode = mode, r.out_len = 0, r.members = 0;
#define BOUNDARY(m) (r.stop = pos, r.stop_mode = (m), r.out_len = o, r.members = members)
  if (mode == MODE_HEADER) goto member_gap;
  for (;;) {
    /* a block start */
    BOUNDARY(MODE_BLOCK);
    if (max_syms == 0 && (pos >= stop_at || o >= job.soft_out || members >= job.soft_mem)) {
      status = ST_STOPPED;
      goto done;
    }
    {
      if (pos + 3 > w.nbits) {
        status = ST_NEED;
        goto done;
      }
      const uint32_t h = (uint32_t)peek(w.in, pos) & 7;
      const bool final = h & 1;
      const uint32_t type = h >> 1;
      pos += 3;
      if (type == 0) {
        pos = (pos + 7) & ~7ull;
        if (pos + 32 > w.nbits) {
          status = ST_NEED;
          goto done;
        }
        const uint32_t v = (uint32_t)peek(w.in, pos);
        const uint32_t len = v & 0xffff;
        if (len != (~v >> 16)) {
          status = ST_CORRUPT;
          goto done;
        }
        pos += 32;
        if (pos + 8ull * len > w.nbits) {
          status = ST_NEED;
          goto done;
        }
        if (max_syms) {
          status = ST_STOPPED;
          goto done;
        }
        const uint64_t b0 = pos >> 3;
        for (uint32_t j = lane; j < len; j += 32)
          if (o + j < job.cap) job.out[o + j] = (uint16_t)byte_at(w.in, b0 + j);
        o += len;
        pos += 8ull * len;
      } else if (type == 3) {
        status = ST_CORRUPT;
        goto done;
      } else {
        if (type == 1) {
          if (!fixed) load_fixed(tb);
          fixed = true;
        } else {
          fixed = false;
          status = read_dynamic(w, pos, tb);
          if (status != ST_STOPPED) goto done;
        }
        __syncwarp();
        /* a symbol is acted on only when all of its bits lie inside the window; a code that the window
         * cuts off is a reason to wait for more input, not corruption */
        for (int ns = 0;; ns++) {
          if (pos >= w.nbits) {
            status = ST_NEED;
            goto done;
          }
          if (max_syms && ns >= max_syms) {
            status = ST_STOPPED;
            goto done;
          }
          uint64_t v = peek(w.in, pos);
          uint32_t len;
          const int s = hdecode(tb.ll, v, len);
          if (s < 0 || pos + len > w.nbits) {
            status = s < 0 && pos + 15 <= w.nbits ? ST_CORRUPT : ST_NEED;
            goto done;
          }
          if (s >= 286) {
            status = ST_CORRUPT;
            goto done;
          }
          v >>= len;
          if (s < 256) {
            pos += len;
            if (lane == 0 && o < job.cap) job.out[o] = (uint16_t)s;
            o++;
            continue;
          }
          if (s == 256) {
            pos += len;
            break;
          }
          const uint32_t li = s - 257, lx = c_lext[li];
          const uint32_t L = c_lbase[li] + (uint32_t)(v & ((1u << lx) - 1));
          v >>= lx;
          uint32_t dlen;
          const int ds = hdecode(tb.d, v, dlen);
          const uint64_t at = pos + len + lx; /* the distance code */
          if (ds < 0 || at + dlen > w.nbits) {
            status = ds < 0 && at + 15 <= w.nbits ? ST_CORRUPT : ST_NEED;
            goto done;
          }
          if (ds >= 30) {
            status = ST_CORRUPT;
            goto done;
          }
          v >>= dlen;
          const uint32_t dx = c_dext[ds];
          if (at + dlen + dx > w.nbits) {
            status = ST_NEED;
            goto done;
          }
          const uint32_t D = c_dbase[ds] + (uint32_t)(v & ((1u << dx) - 1));
          pos = at + dlen + dx;
          const int64_t src = (int64_t)o - D;
          if (src < mstart) {
            status = ST_CORRUPT; /* invalid distance too far back */
            goto done;
          }
          if (o < job.cap) {
            __syncwarp();
            for (uint32_t j = lane; j < L; j += 32) {
              const int64_t q = src + (D >= L ? j : j % D);
              if (o + j < job.cap) job.out[o + j] = q >= 0 ? job.out[q] : (uint16_t)(256 + HIST + q);
            }
            __syncwarp();
          }
          o += L;
        }
      }
      if (max_syms) {
        status = ST_STOPPED;
        goto done;
      }
      if (!final) continue;
      /* member trailer */
      pos = (pos + 7) & ~7ull;
      if (pos + 64 > w.nbits) {
        status = ST_NEED;
        goto done;
      }
      const uint64_t t = peek(w.in, pos);
      if (members < job.mcap && lane == 0) job.mrec[members] = MemberEnd{o, (uint32_t)t, (uint32_t)(t >> 32)};
      members++;
      pos += 64;
    }
  member_gap:
    BOUNDARY(MODE_HEADER);
    if (max_syms == 0 && (o >= job.soft_out || members >= job.soft_mem)) {
      status = ST_STOPPED;
      goto done;
    }
    if (pos >= w.nbits) {
      status = w.eof ? ST_END : ST_NEED;
      goto done;
    }
    if (byte_at(w.in, pos >> 3) != 0x1f) { /* trailing garbage, which gzread ignores */
      status = ST_END;
      goto done;
    }
    status = read_header(w, pos);
    if (status != ST_STOPPED) goto done;
    mstart = (int64_t)o;
  }
done:
  r.status = status;
  r.total_out = o;
  r.total_members = members;
#undef BOUNDARY
}

/* ------------------------------------------------------------------ */

struct FindTabs {
  WarpTabs tb;
  uint8_t clen[19][32];
  uint8_t ctab[128][32];
};

/* a stored block at bit b: zero padding, LEN == ~NLEN */
__device__ __forceinline__ bool stored_ok(const Win &w, uint64_t b, uint32_t hdr) {
  const uint64_t p = (b + 3 + 7) & ~7ull;
  if (p + 32 > w.nbits) return false;
  const uint32_t pad = (uint32_t)(p - b - 3);
  if (pad && ((hdr >> 3) & ((1u << pad) - 1))) return false;
  const uint32_t v = (uint32_t)peek(w.in, p);
  return (v & 0xffff) == (~v >> 16);
}

/* zlib's checks of a dynamic header at bit b, per lane (no test decode) */
__device__ bool dynamic_ok(const Win &w, uint64_t b, FindTabs &ft) {
  const int lane = threadIdx.x & 31;
  uint64_t v = peek(w.in, b) >> 3;
  const uint32_t nlen = 257 + (v & 31), ndist = 1 + ((v >> 5) & 31), ncl = 4 + ((v >> 10) & 15);
  if (nlen > 286 || ndist > 30) return false;
  uint64_t pos = b + 17;
  const uint64_t c = peek(w.in, pos);
  uint64_t cnt = 0; /* 8-bit count per length */
  for (int i = 0; i < 19; i++) {
    const uint32_t l = i < (int)ncl ? (uint32_t)(c >> (3 * i)) & 7 : 0;
    ft.clen[c_cl_order[i]][lane] = (uint8_t)l;
    cnt += (uint64_t)(l != 0) << (8 * l);
  }
  int left = 1;
  for (int l = 1; l <= 7; l++) left = (left << 1) - (int)((cnt >> (8 * l)) & 0xff);
  if (left != 0) return false; /* the code-length code must be complete */
  pos += 3 * ncl;
  /* next code of each length (8 bits per length), canonical order; the per-lane table is complete */
  uint64_t next = 0;
  for (uint32_t l = 1, code = 0, prevc = 0; l <= 7; l++) {
    code = (code + prevc) << 1;
    prevc = (uint32_t)((cnt >> (8 * l)) & 0xff);
    next |= (uint64_t)code << (8 * l);
  }
  for (int s = 0; s < 19; s++) {
    const uint32_t l = ft.clen[s][lane];
    if (!l) continue;
    const uint32_t code = (uint32_t)(next >> (8 * l)) & 0xff;
    next += 1ull << (8 * l);
    const uint32_t rc = __brev(code) >> (32 - l);
    for (uint32_t k = 0; k < (1u << (7 - l)); k++) ft.ctab[rc | k << l][lane] = (uint8_t)(s << 3 | l);
  }
  uint32_t i = 0, prev = 0, kll = 0, kd = 0, maxll = 0, maxd = 0;
  bool eob = false;
  const uint32_t total = nlen + ndist;
  while (i < total) {
    if (pos > w.nbits) return false;
    uint64_t x = peek(w.in, pos);
    const uint32_t e = ft.ctab[x & 127][lane];
    const uint32_t s = e >> 3, len = e & 7;
    pos += len;
    x >>= len;
    uint32_t val, rep;
    if (s < 16) {
      val = s, rep = 1;
    } else if (s == 16) {
      if (i == 0) return false;
      val = prev, rep = 3 + (x & 3), pos += 2;
    } else if (s == 17) {
      val = 0, rep = 3 + (x & 7), pos += 3;
    } else {
      val = 0, rep = 11 + (x & 127), pos += 7;
    }
    if (i + rep > total) return false;
    const uint32_t in_ll = i < nlen ? min(rep, nlen - i) : 0, in_d = rep - in_ll;
    if (val) {
      kll += in_ll << (15 - val);
      kd += in_d << (15 - val);
      if (in_ll) maxll = max(maxll, val);
      if (in_d) maxd = max(maxd, val);
      if (i <= 256 && 256 < i + in_ll) eob = true;
    }
    i += rep;
    prev = val;
  }
  if (!eob) return false;
  if (kll > 32768 || (kll < 32768 && maxll != 1)) return false;
  if (kd > 32768 || (kd < 32768 && maxd > 1)) return false;
  return true;
}

__global__ void __launch_bounds__(WARPS * 32) k_gunzip_find(Win w, int shift_odd, uint64_t *__restrict__ cand) {
  __shared__ FindTabs s_ft[WARPS];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const uint32_t chunk = blockIdx.x * WARPS + wid + 1;
  if (chunk >= w.n_chunks) return;
  FindTabs &ft = s_ft[wid];
  const uint64_t b0 = chunk * w.chunk_bits, b1 = min(b0 + w.chunk_bits, w.nbits);
  uint64_t found = NONE;
  for (uint64_t base = b0; base < b1 && found == NONE; base += 32) {
    const uint64_t b = base + lane;
    bool ok = false, stored = false;
    if (b < b1) {
      const uint32_t h = (uint32_t)peek(w.in, b);
      const uint32_t type = (h >> 1) & 3;
      if (type == 0)
        ok = stored = stored_ok(w, b, h);
      else if (type == 2)
        ok = dynamic_ok(w, b, ft);
    }
    uint32_t pass = __ballot_sync(FULL, ok);
    const uint32_t st = __ballot_sync(FULL, stored);
    while (pass) {
      const int l = __ffs(pass) - 1;
      pass &= pass - 1;
      const uint64_t cb = base + l;
      if (st >> l & 1) {
        found = cb;
        break;
      }
      Job job{};
      ChunkRec r;
      decode(w, job, cb, MODE_BLOCK, NONE, NTEST, ft.tb, r);
      if (r.status == ST_STOPPED || r.status == ST_NEED) {
        found = cb;
        break;
      }
    }
  }
  if (lane == 0) cand[chunk] = found != NONE && shift_odd && (chunk & 1) ? found + 1 : found;
}

/* one warp per chunk, or (jobs != nullptr) one warp per job: repairs and spills */
__global__ void __launch_bounds__(WARPS * 32, 1) k_gunzip_decode(Win w, const uint64_t *__restrict__ cand, uint64_t start0, uint32_t mode0,
                                                             const Job *__restrict__ jobs, uint32_t n_jobs, ChunkRec *__restrict__ recs, uint16_t *__restrict__ slots,
                                                             uint64_t slot_cap, MemberEnd *__restrict__ mrecs, uint32_t mcap) {
  __shared__ WarpTabs s_tb[WARPS];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t chunk;
  uint64_t start;
  uint32_t mode = MODE_BLOCK;
  Job j;
  if (jobs) {
    const uint32_t g = blockIdx.x * WARPS + wid;
    if (g >= n_jobs) return;
    j = jobs[g];
    chunk = j.chunk;
    start = j.start;
    mode = j.mode;
  } else {
    chunk = blockIdx.x * WARPS + wid;
    if (chunk >= w.n_chunks) return;
    start = chunk ? cand[chunk] : start0;
    if (!chunk) mode = mode0;
    j.out = slots + chunk * slot_cap;
    j.cap = slot_cap;
    j.mrec = mrecs + (size_t)chunk * mcap;
    j.mcap = mcap;
    j.soft_out = NONE;
    j.soft_mem = ~0u;
    j.rec = recs + chunk;
  }
  /* the next chunk with a candidate */
  uint64_t stop_at = NONE;
  for (uint32_t k = chunk + 1; k < w.n_chunks; k++)
    if (cand[k] != NONE) {
      stop_at = k * w.chunk_bits;
      break;
    }
  ChunkRec r{};
  if (start == NONE) {
    r.start = NONE, r.status = ST_CORRUPT;
  } else {
    decode(w, j, start, mode, stop_at, 0, s_tb[wid], r);
  }
  if (lane == 0) *j.rec = r;
}


/* dicts[k] = the 32 KiB before chunk k, dicts[m] the 32 KiB after the last (one CTA) */
__global__ void __launch_bounds__(1024) k_gunzip_window(const Emit *__restrict__ emit, uint32_t m, uint8_t *__restrict__ dicts) {
  extern __shared__ uint8_t s_dict[]; /* two buffers of HIST bytes */
  uint8_t *cur = s_dict, *nxt = s_dict + HIST;
  for (uint32_t j = threadIdx.x; j < HIST; j += 1024) cur[j] = dicts[j];
  __syncthreads();
  for (uint32_t k = 0; k < m; k++) {
    const uint16_t *sym = emit[k].sym;
    const uint64_t len = emit[k].len;
    for (uint32_t j = threadIdx.x; j < HIST; j += 1024) {
      if (k) dicts[(size_t)k * HIST + j] = cur[j];
      const int64_t p = (int64_t)len - HIST + j;
      uint8_t v;
      if (p >= 0) {
        const uint32_t s = sym[p];
        v = s < 256 ? (uint8_t)s : cur[s - 256];
      } else {
        v = cur[j + len];
      }
      nxt[j] = v;
    }
    __syncthreads();
    uint8_t *t = cur;
    cur = nxt, nxt = t;
  }
  for (uint32_t j = threadIdx.x; j < HIST; j += 1024) dicts[(size_t)m * HIST + j] = cur[j];
}

/* bytes of every accepted chunk at its output offset; grid (chunks, RY) */
__global__ void __launch_bounds__(256) k_gunzip_resolve(const Emit *__restrict__ emit, const uint8_t *__restrict__ dicts, uint8_t *__restrict__ out,
                                                       uint32_t *__restrict__ bad) {
  const Emit e = emit[blockIdx.x];
  const uint8_t *dict = dicts + (size_t)blockIdx.x * HIST;
  uint8_t *dst = out + e.out;
  bool far = false;
  for (uint64_t i = blockIdx.y * 256 + threadIdx.x; i < e.len; i += (uint64_t)gridDim.y * 256) {
    const uint32_t s = e.sym[i];
    if (s < 256) {
      dst[i] = (uint8_t)s;
    } else {
      far |= HIST - (s - 256) > e.hist;
      dst[i] = dict[s - 256];
    }
  }
  if (__syncthreads_or(far) && threadIdx.x == 0) atomicOr(bad, 1u);
}

/* standard CRC-32 of each piece of out (offset, length <= SEG); one CTA per piece */
__global__ void __launch_bounds__(256) k_gunzip_crc(const uint8_t *__restrict__ out, const uint64_t *__restrict__ off,
                                                   const uint32_t *__restrict__ len, uint32_t *__restrict__ crcs) {
  __shared__ uint32_t s_tab[256], s_part[8];
  uint32_t c = threadIdx.x;
  for (int k = 0; k < 8; k++) c = c & 1 ? (c >> 1) ^ 0xedb88320u : c >> 1;
  s_tab[threadIdx.x] = c;
  __syncthreads();
  const uint8_t *src = out + off[blockIdx.x];
  const uint32_t n = len[blockIdx.x], slice = (n + 255) / 256;
  const uint32_t a = min(n, threadIdx.x * slice), b = min(n, a + slice);
  c = 0;
  for (uint32_t i = a; i < b; i++) c = s_tab[(c ^ src[i]) & 0xff] ^ (c >> 8);
  if (b > a) c = crc_mulmod(crc_x8n(n - b), c);
  for (int o = 16; o; o >>= 1) c ^= __shfl_xor_sync(FULL, c, o);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t x = 0;
    for (int w = 0; w < 8; w++) x ^= s_part[w];
    crcs[blockIdx.x] = x ^ crc_mulmod(crc_x8n(n), 0xffffffffu) ^ 0xffffffffu;
  }
}

}  // namespace

/* ------------------------------------------------------------------ */
/* host side                                                           */

#define INFLATE_TRY(expr)                                                                                            \
  do {                                                                                                               \
    cudaError_t _e = (expr);                                                                                         \
    if (_e != cudaSuccess)                                                                                           \
      return nh_set_error(_e == cudaErrorMemoryAllocation ? NH_ERR_NOMEM : NH_ERR_CUDA, "GPU gunzip: %s failed: %s", \
                          #expr, cudaGetErrorString(_e));                                                            \
  } while (0)

namespace {
constexpr uint32_t SLOT_MULT = 8;      /* output symbols per compressed byte a chunk's slot holds */
constexpr uint32_t MREC = 16;          /* member ends a chunk's slot records */
constexpr uint64_t SPILL = 32u << 20;  /* symbols of the spill buffer; a spilled chunk stops past half of it */
constexpr uint32_t SPILL_MREC = 1u << 16;
constexpr int RY = 16;                 /* resolve CTAs per chunk */
constexpr size_t PAD = 64;             /* zero bytes after a window's last: peek() near the end reads them */
}  // namespace

GpuInflater::~GpuInflater() {
  if (device_ < 0) return;
  cudaSetDevice(device_);
  if (stream_) cudaStreamSynchronize(stream_);
  for (void *p : {(void *)d_win_[0], (void *)d_win_[1], (void *)d_cand_, (void *)d_recs_, (void *)d_slots_, (void *)d_mrec_,
                  (void *)d_spill_, (void *)d_spill_mrec_, (void *)d_dicts_, (void *)d_out_, (void *)d_emit_, (void *)d_piece_len_,
                  (void *)d_piece_off_, (void *)d_crcs_, (void *)d_bad_, (void *)d_jobs_})
    cudaFree(p);
  for (void *p : {(void *)h_in_, (void *)h_recs_, (void *)h_mrec_, (void *)h_out_, (void *)h_emit_, (void *)h_piece_len_,
                  (void *)h_piece_off_, (void *)h_crcs_, (void *)h_bad_, (void *)h_jobs_})
    cudaFreeHost(p);
  for (cudaEvent_t e : ev_)
    if (e) cudaEventDestroy(e);
  if (stream_) cudaStreamDestroy(stream_);
}

int GpuInflater::open(int device, size_t chunk, size_t window, int flags) {
  int nd = 0;
  if (cudaGetDeviceCount(&nd) != cudaSuccess || nd < 1) {
    cudaGetLastError();
    return nh_set_error(NH_ERR_CUDA, "GPU gunzip: no CUDA device (no CPU path)");
  }
  if (device < 0 || device >= nd) return nh_set_error(NH_ERR_INVALID, "GPU gunzip: no CUDA device %d", device);
  chunk_ = chunk ? chunk : kChunkBytes;
  window_ = window ? window : kWindowBytes;
  if (chunk_ < 1024 || chunk_ > (size_t(1) << 24) || window_ < chunk_ || window_ > (size_t(1) << 30))
    return nh_set_error(NH_ERR_INVALID, "GPU gunzip: chunk of %zu and window of %zu bytes are out of range", chunk_, window_);
  flags_ = flags;
  device_ = device;
  cap_ = 2 * window_; /* carried bytes + new bytes */
  max_chunks_ = (uint32_t)((cap_ + chunk_ - 1) / chunk_);
  slot_cap_ = SLOT_MULT * chunk_;
  out_cap_ = std::max<uint64_t>(SLOT_MULT * cap_ / 2, SPILL);
  max_pieces_ = out_cap_ / SEG + 2 * (uint64_t)max_chunks_ * MREC + SPILL_MREC + 16;
  INFLATE_TRY(cudaSetDevice(device));
  INFLATE_TRY(cudaFuncSetAttribute(k_gunzip_window, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * HIST));
  INFLATE_TRY(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
  for (cudaEvent_t &e : ev_) INFLATE_TRY(cudaEventCreate(&e));
  for (int i = 0; i < 2; i++) {
    INFLATE_TRY(cudaMalloc(&d_win_[i], cap_ + PAD));
    INFLATE_TRY(cudaMemsetAsync(d_win_[i], 0, cap_ + PAD, stream_));
  }
  INFLATE_TRY(cudaMalloc(&d_cand_, max_chunks_ * 8));
  INFLATE_TRY(cudaMalloc(&d_recs_, (2 * max_chunks_ + 2) * sizeof(ChunkRec))); /* chunks, a lone spill, batched spills */
  INFLATE_TRY(cudaMalloc(&d_jobs_, (max_chunks_ + 1) * sizeof(Job)));
  INFLATE_TRY(cudaMalloc(&d_slots_, (size_t)max_chunks_ * slot_cap_ * 2));
  INFLATE_TRY(cudaMalloc(&d_mrec_, (size_t)max_chunks_ * MREC * sizeof(MemberEnd)));
  INFLATE_TRY(cudaMalloc(&d_spill_, SPILL * 2));
  INFLATE_TRY(cudaMalloc(&d_spill_mrec_, SPILL_MREC * sizeof(MemberEnd)));
  INFLATE_TRY(cudaMalloc(&d_dicts_, (size_t)(max_chunks_ + 1) * HIST));
  INFLATE_TRY(cudaMemsetAsync(d_dicts_, 0, HIST, stream_));
  INFLATE_TRY(cudaMalloc(&d_out_, out_cap_));
  INFLATE_TRY(cudaMalloc(&d_emit_, max_chunks_ * sizeof(Emit)));
  INFLATE_TRY(cudaMalloc(&d_piece_len_, max_pieces_ * 4));
  INFLATE_TRY(cudaMalloc(&d_piece_off_, max_pieces_ * 8));
  INFLATE_TRY(cudaMalloc(&d_crcs_, max_pieces_ * 4));
  INFLATE_TRY(cudaMalloc(&d_bad_, 4));
  INFLATE_TRY(cudaHostAlloc(&h_in_, window_ + 16, cudaHostAllocDefault));
  INFLATE_TRY(cudaHostAlloc(&h_recs_, (max_chunks_ + 1) * sizeof(ChunkRec), cudaHostAllocDefault));
  INFLATE_TRY(cudaHostAlloc(&h_mrec_, ((size_t)max_chunks_ * MREC + SPILL_MREC) * sizeof(MemberEnd), cudaHostAllocDefault));
  INFLATE_TRY(cudaHostAlloc(&h_jobs_, (max_chunks_ + 1) * sizeof(Job), cudaHostAllocDefault));
  INFLATE_TRY(cudaHostAlloc(&h_out_, out_cap_, cudaHostAllocDefault));
  INFLATE_TRY(cudaHostAlloc(&h_emit_, max_chunks_ * sizeof(Emit), cudaHostAllocDefault));
  INFLATE_TRY(cudaHostAlloc(&h_piece_len_, max_pieces_ * 4, cudaHostAllocDefault));
  INFLATE_TRY(cudaHostAlloc(&h_piece_off_, max_pieces_ * 8, cudaHostAllocDefault));
  INFLATE_TRY(cudaHostAlloc(&h_crcs_, max_pieces_ * 4, cudaHostAllocDefault));
  INFLATE_TRY(cudaHostAlloc(&h_bad_, 4, cudaHostAllocDefault));
  INFLATE_TRY(cudaStreamSynchronize(stream_));
  return NH_OK;
}

size_t GpuInflater::device_bytes() const {
  return 2 * (cap_ + PAD) + max_chunks_ * 8 + (2 * max_chunks_ + 2) * sizeof(ChunkRec) + (max_chunks_ + 1) * sizeof(Job) + (size_t)max_chunks_ * slot_cap_ * 2 +
         (size_t)max_chunks_ * MREC * sizeof(MemberEnd) + SPILL * 2 + SPILL_MREC * sizeof(MemberEnd) +
         (size_t)(max_chunks_ + 1) * HIST + out_cap_ + max_chunks_ * sizeof(Emit) + max_pieces_ * 16;
}

/* device time between two recorded events (the stream has been synchronised) into counts[c] */
void GpuInflater::lap(int a, int b, int c) {
  float ms = 0;
  if (cudaEventElapsedTime(&ms, ev_[a], ev_[b]) != cudaSuccess) return (void)cudaGetLastError();
  counts[c] += (uint64_t)(1e6 * ms);
  kernel_s_ += 1e-3 * ms;
}

int GpuInflater::inflate(const Source &src, const Sink &sink) {
  for (auto &c : counts) c = 0;
  kernel_s_ = 0;
  INFLATE_TRY(cudaSetDevice(device_));
  const uint64_t chunk_bits = 8ull * chunk_;
  /* the stream: the carried bytes sit at the front of d_win_[cur] */
  int cur = 0;
  uint64_t carry = 0, start_bit = 0; /* bytes carried; bit of the first chunk within them */
  uint32_t start_mode = MODE_HEADER;
  uint64_t member_len = 0;           /* bytes of the current member emitted so far */
  uint32_t member_crc = 0;           /* their CRC-32 */
  bool eof = false;
  size_t pending = 0;                /* bytes read ahead in h_in_ */
  auto read_more = [&](size_t want) -> int {
    while (!eof && pending < want) {
      const long n = src(h_in_ + pending, want - pending);
      if (n < 0) return nh_set_error(NH_ERR_IO, "GPU gunzip: read error");
      if (n == 0) eof = true;
      pending += (size_t)n;
    }
    return NH_OK;
  };
  if (int rc = read_more(window_)) return rc;
  if (pending < 2 || h_in_[0] != 0x1f || h_in_[1] != 0x8b) return nh_set_error(NH_ERR_IO, "GPU gunzip: not in gzip format");
  ChunkRec *recs = (ChunkRec *)h_recs_;
  MemberEnd *mrecs = (MemberEnd *)h_mrec_;
  Emit *emit = (Emit *)h_emit_;
  for (;;) {
    /* the window: carried bytes + what was read ahead */
    const size_t take = std::min<size_t>(pending, cap_ - carry);
    uint8_t *d_w = d_win_[cur];
    if (take) INFLATE_TRY(cudaMemcpyAsync(d_w + carry, h_in_, take, cudaMemcpyHostToDevice, stream_));
    const uint64_t nbytes = carry + take;
    /* zero words past the end, so that peek() reads zeros there */
    INFLATE_TRY(cudaMemsetAsync(d_w + nbytes, 0, PAD, stream_));
    INFLATE_TRY(cudaStreamSynchronize(stream_)); /* h_in_ is reused below */
    memmove(h_in_, h_in_ + take, pending - take);
    pending -= take;
    const bool win_eof = eof && pending == 0;
    Win w{(const uint32_t *)d_w, 8 * nbytes, chunk_bits, (uint32_t)((nbytes + chunk_ - 1) / chunk_), win_eof};
    if (w.n_chunks == 0) w.n_chunks = 1;
    counts[0]++;
    counts[1] += w.n_chunks;
    INFLATE_TRY(cudaEventRecord(ev_[0], stream_));
    const uint32_t fb = (w.n_chunks - 1 + WARPS - 1) / WARPS;
    if (fb) k_gunzip_find<<<fb, WARPS * 32, 0, stream_>>>(w, flags_ & NH_GUNZIP_SHIFT_CANDIDATES, d_cand_);
    INFLATE_TRY(cudaEventRecord(ev_[1], stream_));
    k_gunzip_decode<<<(w.n_chunks + WARPS - 1) / WARPS, WARPS * 32, 0, stream_>>>(w, d_cand_, start_bit, start_mode, nullptr, 0, d_recs_, d_slots_,
                                                                                   slot_cap_, d_mrec_, MREC);
    INFLATE_TRY(cudaGetLastError());
    INFLATE_TRY(cudaEventRecord(ev_[2], stream_));
    INFLATE_TRY(cudaMemcpyAsync(recs, d_recs_, w.n_chunks * sizeof(ChunkRec), cudaMemcpyDeviceToHost, stream_));
    /* read the next window's bytes while the kernels run */
    if (int rc = read_more(window_)) return rc;
    INFLATE_TRY(cudaStreamSynchronize(stream_));
    lap(0, 1, NH_GUNZIP_COUNT_NS_FIND);
    lap(1, 2, NH_GUNZIP_COUNT_NS_DECODE);

    Job *jobs = h_jobs_;
    auto slot_job = [&](uint32_t c, uint64_t start, uint32_t mode) {
      Job j{};
      j.chunk = (int32_t)c, j.start = start, j.mode = mode;
      j.out = d_slots_ + c * slot_cap_, j.cap = slot_cap_, j.mrec = d_mrec_ + (size_t)c * MREC, j.mcap = MREC;
      j.soft_out = NONE, j.soft_mem = ~0u, j.rec = d_recs_ + c;
      return j;
    };
    auto run_jobs = [&](uint32_t nj) -> int {
      INFLATE_TRY(cudaMemcpyAsync(d_jobs_, jobs, nj * sizeof(Job), cudaMemcpyHostToDevice, stream_));
      INFLATE_TRY(cudaEventRecord(ev_[3], stream_));
      k_gunzip_decode<<<(nj + WARPS - 1) / WARPS, WARPS * 32, 0, stream_>>>(w, d_cand_, 0, 0, d_jobs_, nj, d_recs_, d_slots_, slot_cap_,
                                                                          d_mrec_, MREC);
      INFLATE_TRY(cudaGetLastError());
      INFLATE_TRY(cudaEventRecord(ev_[4], stream_));
      INFLATE_TRY(cudaMemcpyAsync(recs, d_recs_, (max_chunks_ + 1) * sizeof(ChunkRec), cudaMemcpyDeviceToHost, stream_));
      INFLATE_TRY(cudaStreamSynchronize(stream_));
      lap(3, 4, NH_GUNZIP_COUNT_NS_REDECODE);
      return NH_OK;
    };
    auto corrupt = [] { return nh_set_error(NH_ERR_IO, "GPU gunzip: corrupt deflate data or gzip header"); };

    /* repair rounds: every chunk that does not start where its predecessor stopped is decoded again from
     * there, all in one launch; the first such chunk of a round has a confirmed predecessor, so every
     * round confirms at least one more link */
    for (;;) {
      uint32_t nj = 0;
      bool confirmed = true;
      const ChunkRec *prev = nullptr;
      for (uint32_t c = 0; c < w.n_chunks; c++) {
        if (c && recs[c].start == NONE) continue; /* no candidate: its bytes belong to the predecessor */
        if (prev) {
          if (prev->status != ST_STOPPED) break;
          if (recs[c].start != prev->stop) jobs[nj++] = slot_job(c, prev->stop, MODE_BLOCK), confirmed = false;
        }
        if (confirmed && recs[c].status == ST_CORRUPT) return corrupt();
        prev = &recs[c];
      }
      if (!nj) break;
      counts[2] += nj;
      if (int rc = run_jobs(nj)) return rc;
    }

    /* the chain: chunk 0 and every chunk up to the stream's end or the window's */
    struct Acc {
      uint32_t chunk;
      ChunkRec r;
      const uint16_t *sym;
      const MemberEnd *mrec; /* host copy of its member ends */
    };
    std::vector<Acc> acc;
    for (uint32_t c = 0; c < w.n_chunks; c++) {
      if (c && recs[c].start == NONE) continue;
      acc.push_back({c, recs[c], d_slots_ + c * slot_cap_, mrecs + (size_t)c * MREC});
      if (recs[c].status != ST_STOPPED) break;
    }
    /* chunks that outgrew their slots: decoded again into the spill buffer at prefix offsets of their
     * (now known) sizes, all in one launch; one larger than the whole spill buffer goes alone and stops
     * at the first boundary past half of it */
    uint32_t nj = 0;
    uint64_t spill_used = 0, spill_m = 0;
    MemberEnd *h_spill_m = mrecs + (size_t)max_chunks_ * MREC;
    for (size_t k = 0; k < acc.size(); k++) {
      ChunkRec &r = acc[k].r;
      if (r.out_len <= slot_cap_ && r.members <= MREC) continue;
      counts[3]++;
      Job j = slot_job(acc[k].chunk, r.start, r.start_mode);
      if (spill_used + r.out_len <= SPILL && spill_m + r.members <= SPILL_MREC) {
        j.out = d_spill_ + spill_used, j.cap = r.out_len, j.mrec = d_spill_mrec_ + spill_m, j.mcap = r.members;
        j.rec = d_recs_ + max_chunks_ + 1 + nj;
        acc[k].sym = d_spill_ + spill_used, acc[k].mrec = h_spill_m + spill_m;
        jobs[nj++] = j;
        spill_used += r.out_len, spill_m += r.members;
        continue;
      }
      acc.resize(k + (nj == 0)); /* the rest is carried */
      if (nj) break;
      j.out = d_spill_, j.cap = SPILL, j.mrec = d_spill_mrec_, j.mcap = SPILL_MREC;
      j.soft_out = SPILL / 2, j.soft_mem = SPILL_MREC / 2, j.rec = d_recs_ + max_chunks_;
      jobs[nj++] = j;
      if (int rc = run_jobs(nj)) return rc;
      nj = 0;
      const ChunkRec &sr = recs[max_chunks_];
      if (sr.status == ST_CORRUPT) return corrupt();
      if (sr.out_len > SPILL || sr.members > SPILL_MREC)
        return nh_set_error(NH_ERR_CAPACITY, "GPU gunzip: a deflate block inflates to more than %llu bytes", (unsigned long long)(SPILL / 2));
      const bool partial = sr.stop != r.stop || sr.status != r.status;
      r = sr;
      if (partial) r.status = ST_NEED; /* carry the rest of the chunk */
      acc[k].sym = d_spill_, acc[k].mrec = h_spill_m;
      spill_m = r.members;
      break;
    }
    if (nj)
      if (int rc = run_jobs(nj)) return rc;
    /* no more output than the output buffer holds */
    uint64_t emitted = 0;
    for (size_t k = 0; k < acc.size(); k++) {
      if (emitted + acc[k].r.out_len > out_cap_) {
        acc.resize(k);
        break;
      }
      emitted += acc[k].r.out_len;
    }
    bool done = !acc.empty() && acc.back().r.status == ST_END;
    uint64_t next_bit = acc.empty() ? start_bit : acc.back().r.stop;
    uint32_t next_mode = acc.empty() ? start_mode : acc.back().r.stop_mode;
    if (!done && next_bit == start_bit && next_mode == start_mode) {
      /* no block boundary reached: more input, or a bigger window, is needed */
      if (win_eof) return nh_set_error(NH_ERR_IO, "GPU gunzip: truncated gzip stream");
      if (nbytes >= cap_)
        return nh_set_error(NH_ERR_CAPACITY, "GPU gunzip: a deflate block is longer than the window of %zu bytes", cap_);
      acc.clear();
    }

    /* accepted output: offsets, member checks, dictionaries, bytes */
    const uint32_t m = (uint32_t)acc.size();
    if (m) {
      /* member ends of the accepted chunks */
      bool any_members = false;
      for (auto &a : acc) any_members |= a.r.members != 0;
      if (any_members) {
        INFLATE_TRY(cudaMemcpyAsync(mrecs, d_mrec_, (size_t)(acc.back().chunk + 1) * MREC * sizeof(MemberEnd), cudaMemcpyDeviceToHost,
                                    stream_));
        if (spill_m) INFLATE_TRY(cudaMemcpyAsync(h_spill_m, d_spill_mrec_, spill_m * sizeof(MemberEnd), cudaMemcpyDeviceToHost, stream_));
        INFLATE_TRY(cudaStreamSynchronize(stream_));
      }
      /* CRC pieces, cut at member ends and every SEG bytes; checks[i]: pieces before member end i */
      struct MemberCheck {
        uint64_t pieces;
        uint32_t crc, isize;
      };
      std::vector<MemberCheck> checks;
      uint64_t np = 0, out = 0, piece_from = 0, hist_member = member_len;
      auto add_pieces = [&](uint64_t a, uint64_t b) {
        for (uint64_t p = a; p < b; p += SEG, np++) h_piece_off_[np] = p, h_piece_len_[np] = (uint32_t)std::min<uint64_t>(SEG, b - p);
      };
      for (uint32_t k = 0; k < m; k++) {
        const ChunkRec &r = acc[k].r;
        emit[k].sym = acc[k].sym;
        emit[k].len = r.out_len;
        emit[k].out = out;
        emit[k].hist = (uint32_t)std::min<uint64_t>(HIST, hist_member);
        const MemberEnd *me = acc[k].mrec;
        for (uint32_t i = 0; i < r.members; i++) {
          add_pieces(piece_from, out + me[i].out);
          checks.push_back({np, me[i].crc, me[i].isize});
          piece_from = out + me[i].out;
        }
        hist_member = r.members ? r.out_len - me[r.members - 1].out : hist_member + r.out_len;
        out += r.out_len;
      }
      add_pieces(piece_from, out);
      INFLATE_TRY(cudaMemcpyAsync(d_emit_, emit, m * sizeof(Emit), cudaMemcpyHostToDevice, stream_));
      INFLATE_TRY(cudaMemsetAsync(d_bad_, 0, 4, stream_));
      if (np) {
        INFLATE_TRY(cudaMemcpyAsync(d_piece_len_, h_piece_len_, np * 4, cudaMemcpyHostToDevice, stream_));
        INFLATE_TRY(cudaMemcpyAsync(d_piece_off_, h_piece_off_, np * 8, cudaMemcpyHostToDevice, stream_));
      }
      INFLATE_TRY(cudaEventRecord(ev_[5], stream_));
      k_gunzip_window<<<1, 1024, 2 * HIST, stream_>>>(d_emit_, m, d_dicts_);
      INFLATE_TRY(cudaEventRecord(ev_[6], stream_));
      k_gunzip_resolve<<<dim3(m, RY), 256, 0, stream_>>>(d_emit_, d_dicts_, d_out_, d_bad_);
      if (np) k_gunzip_crc<<<(uint32_t)np, 256, 0, stream_>>>(d_out_, d_piece_off_, d_piece_len_, d_crcs_);
      INFLATE_TRY(cudaGetLastError());
      INFLATE_TRY(cudaEventRecord(ev_[7], stream_));
      /* the window after the last accepted chunk is the next window's first */
      INFLATE_TRY(cudaMemcpyAsync(d_dicts_, d_dicts_ + (size_t)m * HIST, HIST, cudaMemcpyDeviceToDevice, stream_));
      INFLATE_TRY(cudaMemcpyAsync(h_bad_, d_bad_, 4, cudaMemcpyDeviceToHost, stream_));
      if (np) INFLATE_TRY(cudaMemcpyAsync(h_crcs_, d_crcs_, np * 4, cudaMemcpyDeviceToHost, stream_));
      if (!timing_ && out) INFLATE_TRY(cudaMemcpyAsync(h_out_, d_out_, out, cudaMemcpyDeviceToHost, stream_));
      INFLATE_TRY(cudaStreamSynchronize(stream_));
      lap(5, 6, NH_GUNZIP_COUNT_NS_WINDOW);
      lap(6, 7, NH_GUNZIP_COUNT_NS_RESOLVE);
      if (*h_bad_) return nh_set_error(NH_ERR_IO, "GPU gunzip: invalid distance too far back");
      /* every member's CRC-32 and ISIZE */
      uint64_t p = 0;
      auto take_pieces = [&](uint64_t upto) {
        for (; p < upto; p++) {
          member_crc = (uint32_t)crc32_combine(member_crc, h_crcs_[p], (z_off_t)h_piece_len_[p]);
          member_len += h_piece_len_[p];
        }
      };
      for (const MemberCheck &mc : checks) {
        take_pieces(mc.pieces);
        if (member_crc != mc.crc) return nh_set_error(NH_ERR_IO, "GPU gunzip: incorrect data check (CRC-32) in a member trailer");
        if ((uint32_t)member_len != mc.isize) return nh_set_error(NH_ERR_IO, "GPU gunzip: incorrect length check in a member trailer");
        member_crc = 0, member_len = 0;
        counts[4]++;
      }
      take_pieces(np);
      if (!timing_ && out)
        if (int rc = sink(h_out_, out)) return rc;
    }
    if (done) return NH_OK;
    /* carry everything from the stop of the last accepted chunk */
    const uint64_t stop_byte = next_bit >> 3;
    if (stop_byte > nbytes) return nh_set_error(NH_ERR_IO, "GPU gunzip: internal error: a stop past the window's end");
    carry = nbytes - stop_byte;
    counts[5] += carry;
    start_bit = next_bit & 7;
    start_mode = next_mode;
    if (carry) INFLATE_TRY(cudaMemcpyAsync(d_win_[cur ^ 1], d_w + stop_byte, carry, cudaMemcpyDeviceToDevice, stream_));
    cur ^= 1;
  }
}

int GpuInflater::time_kernels(const uint8_t *in, size_t n, int iters, double *seconds) {
  timing_ = true;
  double total = 0;
  int rc = NH_OK;
  for (int i = 0; i < iters + 1 && rc == NH_OK; i++) { /* the first pass warms up */
    size_t at = 0;
    rc = inflate([&](uint8_t *dst, size_t want) -> long {
                   const size_t k = std::min(want, n - at);
                   memcpy(dst, in + at, k);
                   at += k;
                   return (long)k;
                 },
                 [](const uint8_t *, size_t) { return NH_OK; });
    if (i) total += kernel_s_;
  }
  timing_ = false;
  if (rc == NH_OK) *seconds = total / iters;
  return rc;
}

static int gunzip_device_check(int device) {
  int nd = 0;
  if (cudaGetDeviceCount(&nd) != cudaSuccess || nd < 1) {
    cudaGetLastError();
    return nh_set_error(NH_ERR_CUDA, "no CUDA device (no CPU path)");
  }
  if (device < 0 || device >= nd) return nh_set_error(NH_ERR_INVALID, "no CUDA device %d", device);
  return NH_OK;
}

extern "C" int nh_debug_gunzip(int device, const uint8_t *in, size_t n, uint8_t *out, size_t out_cap, size_t *out_len, size_t chunk_bytes,
                               size_t window_bytes, int flags, uint64_t *counts) {
  if ((n && !in) || (out_cap && !out) || !out_len || (flags & ~NH_GUNZIP_SHIFT_CANDIDATES))
    return nh_set_error(NH_ERR_INVALID, "nh_gunzip: bad argument");
  *out_len = 0;
  if (int rc = gunzip_device_check(device)) return rc;
  GpuInflater gi;
  const size_t window = window_bytes ? window_bytes : std::min<size_t>(GpuInflater::kWindowBytes, std::max<size_t>(n, 1));
  const size_t chunk = chunk_bytes ? chunk_bytes : GpuInflater::kChunkBytes;
  if (int rc = gi.open(device, chunk, std::max(window, chunk), flags)) return rc;
  size_t at = 0, total = 0;
  const int rc = gi.inflate(
      [&](uint8_t *dst, size_t want) -> long {
        const size_t k = std::min(want, n - at);
        memcpy(dst, in + at, k);
        at += k;
        return (long)k;
      },
      [&](const uint8_t *p, size_t len) {
        if (total + len <= out_cap) memcpy(out + total, p, len);
        total += len;
        return NH_OK;
      });
  if (counts)
    for (int i = 0; i < NH_GUNZIP_NCOUNTS; i++) counts[i] = gi.counts[i];
  if (rc) return rc;
  *out_len = total;
  if (total > out_cap)
    return nh_set_error(NH_ERR_CAPACITY, "nh_gunzip: the stream inflates to %zu bytes, %zu given", total, out_cap);
  return NH_OK;
}

extern "C" int nh_gunzip(int device, const uint8_t *in, size_t n, uint8_t *out, size_t out_cap, size_t *out_len) {
  return nh_debug_gunzip(device, in, n, out, out_cap, out_len, 0, 0, 0, nullptr);
}

extern "C" int nh_bench_gunzip(int device, const uint8_t *in, size_t n, int iters, double *out_seconds) {
  if (!in || !n || iters < 1 || !out_seconds) return nh_set_error(NH_ERR_INVALID, "nh_bench_gunzip: bad argument");
  if (int rc = gunzip_device_check(device)) return rc;
  GpuInflater gi;
  if (int rc = gi.open(device)) return rc;
  return gi.time_kernels(in, n, iters, out_seconds);
}
