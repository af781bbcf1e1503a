/*
 * dust_oracle.c — CPU restatement of dustmasker's symmetric DUST (Morgulis et al. 2006): the sequential loop of
 * minimap2's sdust.c (shift_window, find_perfect, save_masked_regions) as recalled, not verified against it.
 * TEST INFRASTRUCTURE ONLY: tests/dust_oracle.py builds it, and the GPU masking (nohuman_b200/csrc/nh_dust.cu)
 * is checked byte for byte against it; tests/test_dust_host.py checks it against a brute-force enumeration of
 * the definition in DESIGN.md §4f.  The product never links it.
 */
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#ifdef _OPENMP
#include <omp.h>
#endif
typedef struct {
  int32_t start, finish, r, l; /* bases [start, finish) of the record */
} dust_perf;

typedef struct {
  int W, T;
  int w[64], wh, wn; /* triplet window: w[(wh + k) & 63] is the k-th oldest of wn */
  int cv[64], cw[64];
  int rv, rw, L;
  dust_perf *P; /* perfect intervals, start descending */
  size_t pn, pcap;
  uint8_t *out; /* the record's output bytes */
} dust_state;

static int dust_at(const dust_state *d, int k) { return d->w[(d->wh + k) & 63]; }

/* the perfect interval with the smallest start joins the mask once the window has passed its start; every
 * interval that starts before the window leaves the list */
static void dust_save(dust_state *d, int start) {
  if (d->pn == 0 || d->P[d->pn - 1].start >= start) return;
  const dust_perf *p = &d->P[d->pn - 1];
  for (int32_t i = p->start; i < p->finish; i++) d->out[i] |= 0x20;
  ptrdiff_t i = (ptrdiff_t)d->pn - 1;
  while (i >= 0 && d->P[i].start < start) i--;
  d->pn = (size_t)(i + 1);
}

static void dust_shift(dust_state *d, int t) {
  if (d->wn >= d->W - 2) {
    const int s = dust_at(d, 0);
    d->wh = (d->wh + 1) & 63;
    d->wn--;
    d->rw -= --d->cw[s];
    if (d->L > d->wn) {
      d->L--;
      d->rv -= --d->cv[s];
    }
  }
  d->w[(d->wh + d->wn) & 63] = t;
  d->wn++;
  d->L++;
  d->rw += d->cw[t]++;
  d->rv += d->cv[t]++;
  if (d->cv[t] * 10 > d->T * 2) { /* drop the suffix's head up to the previous t: no count there exceeds 2T/10 */
    int s;
    do {
      s = dust_at(d, d->wn - d->L);
      d->rv -= --d->cv[s];
      d->L--;
    } while (s != t);
  }
}

static int dust_find_perfect(dust_state *d, int start) {
  int c[64];
  memcpy(c, d->cv, sizeof c);
  int r = d->rv, max_r = 0, max_l = 0;
  for (int i = d->wn - d->L - 1; i >= 0; i--) {
    const int t = dust_at(d, i);
    r += c[t]++;
    const int new_r = r, new_l = d->wn - i - 1;
    if (new_r * 10 <= d->T * new_l) continue;
    size_t j = 0;
    for (; j < d->pn && d->P[j].start >= i + start; j++) {
      const dust_perf *p = &d->P[j];
      if (max_r == 0 || p->r * max_l > max_r * p->l) max_r = p->r, max_l = p->l;
    }
    if (max_r == 0 || new_r * max_l >= max_r * new_l) {
      max_r = new_r, max_l = new_l;
      if (d->pn == d->pcap) {
        const size_t cap = d->pcap ? 2 * d->pcap : 256;
        dust_perf *np = (dust_perf *)realloc(d->P, cap * sizeof *np);
        if (!np) return -1;
        d->P = np, d->pcap = cap;
      }
      memmove(d->P + j + 1, d->P + j, (d->pn - j) * sizeof *d->P);
      d->P[j].start = i + start;
      d->P[j].finish = d->wn + 2 + start;
      d->P[j].r = new_r;
      d->P[j].l = new_l;
      d->pn++;
    }
  }
  return 0;
}

static void dust_reset(dust_state *d) {
  d->wh = d->wn = 0;
  memset(d->cv, 0, sizeof d->cv);
  memset(d->cw, 0, sizeof d->cw);
  d->rv = d->rw = d->L = 0;
}

static int dust_record(dust_state *d, const uint8_t *seq, size_t len) {
  for (size_t i = 0; i < len; i++) {
    const uint8_t ch = seq[i];
    d->out[i] = ch >= 'a' && ch <= 'z' ? (uint8_t)(ch - 32) : ch;
  }
  dust_reset(d);
  d->pn = 0;
  int l = 0, t = 0;
  for (size_t i = 0; i <= len; i++) {
    int b = 4;
    if (i < len) switch (seq[i] | 0x20) {
        case 'a': b = 0; break;
        case 'c': b = 1; break;
        case 'g': b = 2; break;
        case 't': b = 3; break;
      }
    if (b < 4) {
      l++;
      t = ((t << 2) | b) & 63;
      if (l >= 3) {
        const int start = (l - d->W > 0 ? l - d->W : 0) + (int)(i + 1) - l;
        dust_save(d, start);
        dust_shift(d, t);
        if (d->rw * 10 > d->L * d->T && dust_find_perfect(d, start)) return -1;
      }
    } else {
      /* the flush starts at the window start after the last step's.  The loop as recalled starts one later,
       * (l - W + 1) + (i + 1 - l), which for runs of at least W bases drops the intervals that start at the
       * skipped position unsaved: the mask then misses bases of the definition (DESIGN.md §4f) */
      int start = (l - d->W > 0 ? l - d->W : 0) + (int)i - l + 1;
      while (d->pn) dust_save(d, start++);
      l = t = 0;
      dust_reset(d);
    }
  }
  return 0;
}

/* Sequences concatenated in `bases`, offsets[n_seqs+1]; out[i] is bases[i] lower-cased where masked (only
 * A/C/G/T in either case can be) and upper-cased elsewhere.  window 4..64 bases, level 1..255 (dustmasker's
 * defaults: 64, 20).  OpenMP over records with `threads` threads (<=0: all).  0, or -1 for parameters out of
 * range or records over 2^31 bases. */
int dust_oracle_mask(const uint8_t *bases, const uint64_t *offsets, uint64_t n_seqs, int window, int level,
                     int threads, uint8_t *out) {
  if (window < 4 || window > 64 || level < 1 || level > 255) return -1;
  int failed = 0;
#ifdef _OPENMP
  if (threads <= 0) threads = omp_get_max_threads();
#else
  (void)threads;
#endif
#pragma omp parallel num_threads(threads)
  {
    dust_state d;
    memset(&d, 0, sizeof d);
    d.W = window;
    d.T = level;
    int64_t s;
#pragma omp for schedule(dynamic, 16)
    for (s = 0; s < (int64_t)n_seqs; s++) {
      const uint64_t o = offsets[s], n = offsets[s + 1] - o;
      d.out = out + o;
      if (n > 0x7fffffff || dust_record(&d, bases + o, (size_t)n)) {
#pragma omp atomic write
        failed = 1;
      }
    }
    free(d.P);
  }
  return failed ? -1 : 0;
}
