/* oracle/kslam_oracle.c — TEST INFRASTRUCTURE ONLY (see kslam_oracle.h).
 *
 * CPU restatement of k-SLAM's matching path; each function cites the reference file:line
 * it follows. Pinned against the compiled reference (oracle/_ref) — "parity pinned".
 * Never used, linked or loaded by the product path.
 */
#include "kslam_oracle.h"
#include <stdlib.h>
#include <string.h>
#include <omp.h>

/* ------------------------------------------------------------------ k-mers */

/* KMer.h:246-266 — A=0 C=1 T=2 G=3, everything else (N, lower case, IUPAC) = 0 */
static inline uint64_t two_bits(char c) {
  switch (c) { case 'A': return 0; case 'C': return 1; case 'T': return 2; case 'G': return 3; default: return 0; }
}

/* KMer.h:160-181 (splitIntoKMersAndAddToVector) + KMer.h:272-280 (addBaseToKMers) */
uint64_t ko_extract_kmers(uint64_t n, const char *bases, const uint64_t *offs, int is_gb,
                          uint32_t gap, ko_kmer *out) {
  uint64_t cnt = 0;
  for (uint64_t id = 0; id < n; id++) {
    const char *s = bases + offs[id];
    uint64_t len = offs[id + 1] - offs[id];
    if (len < KO_K) continue; /* KMer.h:167 */
    uint64_t f = 0, rc = 0;
    for (uint64_t i = 0; i < len; i++) {
      uint64_t b = two_bits(s[i]);
      f = (f << 2) | b;                       /* K==32: the mask is all ones (KMer.h:42-44) */
      rc = (rc >> 2) | ((b ^ 2) << 62);       /* complement = flip bit 1 (KMer.h:279) */
      if (i < KO_K - 1) continue;
      if ((i - (KO_K - 1)) % gap) continue;
      if (out) {
        ko_kmer *o = &out[cnt];
        if (f < rc) {                         /* forward wins only if strictly smaller (KMer.h:173) */
          o->kmer = f; o->offset = (uint32_t)(i - (KO_K - 1));
          o->id_flags = ((uint32_t)id & 0x3FFFFFFFu) | ((uint32_t)(is_gb != 0) << 31);
        } else {
          o->kmer = rc; o->offset = (uint32_t)(is_gb ? i - (KO_K - 1) : len - 1 - i); /* KMer.h:176 */
          o->id_flags = ((uint32_t)id & 0x3FFFFFFFu) | ((uint32_t)(is_gb != 0) << 31) | (1u << 30);
        }
      }
      cnt++;
    }
  }
  return cnt;
}

/* KMer.h:392-396 */
static int cmp_kmer(const void *a, const void *b) {
  const ko_kmer *x = (const ko_kmer *)a, *y = (const ko_kmer *)b;
  if (x->kmer != y->kmer) return x->kmer < y->kmer ? -1 : 1;
  if (x->id_flags != y->id_flags) return x->id_flags > y->id_flags ? -1 : 1; /* descending */
  if (x->offset != y->offset) return x->offset < y->offset ? -1 : 1;         /* our tie-break (H1) */
  return 0;
}
void ko_sort_kmers(ko_kmer *recs, uint64_t n) { qsort(recs, n, sizeof(ko_kmer), cmp_kmer); }

/* Overlap.h:230-246 (findOverlaps) + Overlap.h:153-199 (processPileUp) */
uint64_t ko_find_seeds_raw(const ko_kmer *recs, uint64_t n, const uint32_t *read_lens, ko_seed *out) {
  uint64_t cnt = 0, i = 0;
  while (i < n) {
    if (recs[i].kmer == 0) { i++; continue; }                 /* Overlap.h:236-239 */
    uint64_t j = i + 1;
    while (j < n && recs[j].kmer == recs[i].kmer) j++;
    if (j - i >= 2 && (recs[i].id_flags >> 31)) {             /* adjacent_find + Overlap.h:157 */
      uint64_t g_end = i;
      while (g_end < j && (recs[g_end].id_flags >> 31)) g_end++;
      for (uint64_t r = i; r < j; r++) {
        if (recs[r].id_flags >> 31) continue;                 /* Overlap.h:177 */
        uint32_t rid = recs[r].id_flags & 0x3FFFFFFFu, r_rc = (recs[r].id_flags >> 30) & 1;
        for (uint64_t g = i; g < r && g < g_end; g++) {       /* Overlap.h:179-181 */
          if (!(recs[g].id_flags >> 31)) break;
          uint32_t g_rc = (recs[g].id_flags >> 30) & 1;
          uint32_t off = !g_rc ? recs[r].offset : read_lens[rid] - recs[r].offset - KO_K; /* :185-189 */
          if (out) {
            out[cnt].read = rid; out[cnt].entry = recs[g].id_flags & 0x3FFFFFFFu;
            out[cnt].rel = (int32_t)(recs[g].offset - off);   /* u32 wrap then i32 (Overlap.h:36-41) */
            out[cnt].rev_comp = g_rc != r_rc;                 /* !sameComp */
          }
          cnt++;
        }
      }
    }
    i = j;
  }
  return cnt;
}

/* Overlap.h:87-98; rev_comp appended so exact ties have one canonical order (SURVEY App. C H2) */
static int cmp_seed(const void *a, const void *b) {
  const ko_seed *x = (const ko_seed *)a, *y = (const ko_seed *)b;
  if (x->read != y->read) return x->read < y->read ? -1 : 1;
  if (x->entry != y->entry) return x->entry < y->entry ? -1 : 1;
  if (x->rel != y->rel) return x->rel < y->rel ? -1 : 1;
  if (x->rev_comp != y->rev_comp) return x->rev_comp < y->rev_comp ? -1 : 1;
  return 0;
}
/* Overlap.h:289-291 with overlapEqual :79-85 — std::unique compares with the last KEPT element */
uint64_t ko_sort_unique_seeds(ko_seed *s, uint64_t n) {
  if (!n) return 0;
  qsort(s, n, sizeof(ko_seed), cmp_seed);
  uint64_t w = 0;
  for (uint64_t i = 1; i < n; i++) {
    int64_t d = (int64_t)s[i].rel - (int64_t)s[w].rel;
    /* abs() on int: |d| < 3 (differences here never overflow int in practice) */
    int eq = s[i].read == s[w].read && s[i].entry == s[w].entry && (d < 0 ? -d : d) < 3;
    if (!eq) s[++w] = s[i];
  }
  return w + 1;
}

/* ------------------------------------------------------------- Smith-Waterman */

/* ssw_cpp.cpp:11-23 (kBaseTranslation): A/a 0, C/c 1, G/g 2, T/t 3, U/u 0, else 4 */
static inline int8_t ssw_code(char c) {
  switch (c) {
    case 'A': case 'a': case 'U': case 'u': return 0;
    case 'C': case 'c': return 1;
    case 'G': case 'g': return 2;
    case 'T': case 't': return 3;
    default: return 4;
  }
}
/* ssw_cpp.cpp:25-49 (BuildSwScoreMatrix): any pair involving code 4 scores 0. match / mismatch arrive as uint8_t
 * (ssw_cpp.cpp:114-117) and are stored in an int8_t matrix: match as is, mismatch as static_cast<int8_t>(-mismatch). */
static inline int32_t sc(const ko_params *p, int8_t a, int8_t b) {
  if (a == 4 || b == 4) return 0;
  return a == b ? (int32_t)(int8_t)(uint8_t)p->match : (int32_t)(int8_t)(-(int32_t)(uint8_t)p->mismatch);
}

typedef struct { int32_t score, ref, read; } sw_end;

/* ssw.c:143-383 / 408-592 restated without striping (SURVEY App. A.6/A.7): plain Gotoh with SSW's tie rules.
 * Equal to the striped kernels when gap_extend < gap_open and mismatch <= 2 * gap_extend (checked by
 * tests/test_oracle_vs_ref.py); kept as the cross-check of sw_striped below, which is what ko_ssw_align uses.
 * Columns are scanned from `begin` in direction `step`; q[0..m) are query rows.
 * Returns the max score, the first column (scan order) attaining it, and the smallest row holding it
 * in that column. If terminate >= 0, stop after the first column whose max equals it (ssw.c:330,545). */
static sw_end sw_scan(const int8_t *ref, int32_t ref_len, int dir, const int8_t *q, int32_t m,
                      const ko_params *p, int32_t terminate, int32_t *H, int32_t *E) {
  const int32_t go = (uint8_t)p->gap_open, ge = (uint8_t)p->gap_extend;
  sw_end best = {0, -1, 0};
  for (int32_t i = 0; i < m; i++) H[i] = E[i] = 0;
  int32_t begin = dir ? ref_len - 1 : 0, end = dir ? -1 : ref_len, step = dir ? -1 : 1;
  for (int32_t j = begin; j != end; j += step) {
    int32_t F = 0, diag = 0, colmax = 0, colrow = 0;
    for (int32_t i = 0; i < m; i++) {
      int32_t h = diag + sc(p, ref[j], q[i]);
      int32_t e = E[i];
      if (h < e) h = e;
      if (h < F) h = F;
      if (h < 0) h = 0;
      diag = H[i];
      H[i] = h;
      if (h > colmax) { colmax = h; colrow = i; }          /* smallest row with the column max */
      int32_t hg = h - go; if (hg < 0) hg = 0;             /* _mm_subs_epu* saturates at 0 */
      e -= ge; if (e < 0) e = 0; E[i] = e > hg ? e : hg;
      F -= ge; if (F < 0) F = 0; if (F < hg) F = hg;
    }
    if (colmax > best.score) { best.score = colmax; best.ref = j; best.read = colrow; } /* ssw.c:316-319 */
    if (terminate >= 0 && colmax == terminate) break;
  }
  return best;
}

/* sw_sse2_byte (ssw.c:143-383, word == 0) and sw_sse2_word (ssw.c:408-592, word == 1) LITERALLY, lane by lane: the
 * striped layout (vector j, lane l <-> query row j + l * segLen, ssw.c:105-133,385-406), the saturating byte arithmetic
 * with its bias, E updated from the H value BEFORE the lazy-F correction (:257-264), the two different lazy-F loops
 * (byte: until no lane's F exceeds H - gapO, vMaxColumn updated inside, :289-305; word: at most 8 rounds, early exit on
 * the first vector where no lane's F exceeds H - gapO, vMaxColumn NOT updated, :514-524) and the end-position rules
 * (:307-343,526-558). For scoring parameters outside the "plain Gotoh" domain those details decide the result.
 * buf: 9 * segLen * lanes int32 of scratch. Values are held in int32 but clamped exactly like the 8 / 16-bit lanes. */
static sw_end sw_striped(const int8_t *ref, int dir, int32_t refLen, const int8_t *read, int32_t readLen, const int8_t *mat,
                         int32_t go, int32_t ge, int32_t terminate, int word, int32_t bias, int32_t *buf) {
  const int L = word ? 8 : 16;
  const int32_t segLen = (readLen + L - 1) / L, N = segLen * L;
  int32_t *Hs = buf, *Hl = buf + N, *E = buf + 2 * N, *Hm = buf + 3 * N, *P = buf + 4 * N;   /* P: 5 * N */
  for (int32_t nt = 0; nt < 5; nt++)
    for (int32_t i = 0; i < segLen; i++)
      for (int l = 0; l < L; l++) {
        const int32_t j = i + l * segLen;
        if (word) P[nt * N + i * L + l] = j >= readLen ? 0 : mat[nt * 5 + read[j]];
        else P[nt * N + i * L + l] = j >= readLen ? (uint8_t)bias : (uint8_t)(mat[nt * 5 + read[j]] + bias);
      }
  for (int32_t k = 0; k < 4 * N; k++) buf[k] = 0;
  int32_t max = 0, end_read = readLen - 1, end_ref = word ? 0 : -1;
  int32_t vMaxScore[16] = {0}, vMaxMark[16] = {0}, vF[16], vH[16], vMaxColumn[16];
  const int32_t begin = dir ? refLen - 1 : 0, end = dir ? -1 : refLen, step = dir ? -1 : 1;
  for (int32_t i = begin; i != end; i += step) {
    for (int l = 0; l < L; l++) { vF[l] = 0; vMaxColumn[l] = 0; }
    for (int l = L - 1; l > 0; l--) vH[l] = Hs[(segLen - 1) * L + l - 1];     /* _mm_slli_si128 by one lane */
    vH[0] = 0;
    const int32_t *vP = P + ref[i] * N;
    { int32_t *t = Hl; Hl = Hs; Hs = t; }
    for (int32_t j = 0; j < segLen; j++)
      for (int l = 0; l < L; l++) {
        int32_t h = vH[l] + vP[j * L + l];
        if (word) { if (h > 32767) h = 32767; if (h < -32768) h = -32768; }   /* _mm_adds_epi16 */
        else { if (h > 255) h = 255; h -= bias; if (h < 0) h = 0; }             /* _mm_adds_epu8, _mm_subs_epu8 */
        int32_t e = E[j * L + l];
        if (h < e) h = e;
        if (h < vF[l]) h = vF[l];
        if (vMaxColumn[l] < h) vMaxColumn[l] = h;
        Hs[j * L + l] = h;
        h -= go; if (h < 0) h = 0;
        e -= ge; if (e < 0) e = 0;
        if (e < h) e = h;
        E[j * L + l] = e;
        int32_t f = vF[l] - ge; if (f < 0) f = 0;
        vF[l] = f > h ? f : h;
        vH[l] = Hl[j * L + l];
      }
    if (!word) {                                                              /* ssw.c:276-305 */
      int32_t j = 0;
      for (int l = L - 1; l > 0; l--) vF[l] = vF[l - 1];
      vF[0] = 0;
      for (;;) {
        int any = 0;
        for (int l = 0; l < L; l++) { int32_t t = Hs[j * L + l] - go; if (t < 0) t = 0; any |= vF[l] > t; }
        if (!any) break;
        for (int l = 0; l < L; l++) {
          int32_t h = Hs[j * L + l];
          if (h < vF[l]) h = vF[l];
          if (vMaxColumn[l] < h) vMaxColumn[l] = h;
          Hs[j * L + l] = h;
          vF[l] -= ge; if (vF[l] < 0) vF[l] = 0;
        }
        if (++j >= segLen) { j = 0; for (int l = L - 1; l > 0; l--) vF[l] = vF[l - 1]; vF[0] = 0; }
      }
    } else {                                                                  /* ssw.c:512-524 */
      int done = 0;
      for (int k = 0; k < 8 && !done; k++) {
        for (int l = L - 1; l > 0; l--) vF[l] = vF[l - 1];
        vF[0] = 0;
        for (int32_t j = 0; j < segLen && !done; j++) {
          int any = 0;
          for (int l = 0; l < L; l++) {
            int32_t h = Hs[j * L + l];
            if (h < vF[l]) h = vF[l];
            Hs[j * L + l] = h;
            h -= go; if (h < 0) h = 0;
            vF[l] -= ge; if (vF[l] < 0) vF[l] = 0;
            any |= vF[l] > h;
          }
          if (!any) done = 1;
        }
      }
    }
    int differs = 0;
    for (int l = 0; l < L; l++) { if (vMaxScore[l] < vMaxColumn[l]) vMaxScore[l] = vMaxColumn[l]; differs |= vMaxMark[l] != vMaxScore[l]; }
    if (differs) {
      int32_t temp = 0;
      for (int l = 0; l < L; l++) { vMaxMark[l] = vMaxScore[l]; if (temp < vMaxScore[l]) temp = vMaxScore[l]; }
      if (temp > max) {
        max = temp;
        if (!word && max + bias >= 255) break;                                /* overflow, ssw.c:318 */
        end_ref = i;
        for (int32_t k = 0; k < N; k++) Hm[k] = Hs[k];
      }
    }
    int32_t colmax = 0;
    for (int l = 0; l < L; l++) if (colmax < vMaxColumn[l]) colmax = vMaxColumn[l];
    if (colmax == terminate) break;
  }
  for (int32_t k = 0; k < N; k++)                                             /* ssw.c:334-342,549-557 */
    if (Hm[k] == max) { const int32_t row = k / L + k % L * segLen; if (row < end_read) end_read = row; }
  sw_end r;
  r.score = (!word && max + bias >= 255) ? 255 : max; r.ref = end_ref; r.read = end_read;
  return r;
}

/* ssw.c:56-71 */
#define SET_U(u, w, i, j) { int x_ = (i) - (w); x_ = x_ > 0 ? x_ : 0; (u) = (j) - x_ + 1; }
#define SET_D(u, w, i, j, p) { int x_ = (i) - (w); x_ = x_ > 0 ? x_ : 0; x_ = (j) - x_; (u) = x_ * 3 + (p); }

/* ssw.c:594-792 (banded_sw), emulating its rolling arrays literally (SURVEY App. A.8).
 * Returns cigar length, or -1 when the reference's behaviour is undefined (traceback reads a
 * direction byte that was never written / left the matrix). */
static int32_t banded_cigar(const int8_t *ref, const int8_t *read, int32_t refLen, int32_t readLen,
                            int32_t score, const ko_params *p, uint32_t *cig, uint32_t cap, int *overflow) {
  const int32_t go = (uint8_t)p->gap_open, ge = (uint8_t)p->gap_extend;
  int32_t band_width = abs(refLen - readLen) + 1; /* ssw.c:932 */
  int32_t width = 0, width_d = 0, max = 0;
  int32_t *h_b = NULL, *e_b = NULL, *h_c = NULL;
  int8_t *direction = NULL;
  do {
    width = band_width * 2 + 3; width_d = band_width * 2 + 1;
    if ((int64_t)width_d * readLen * 3 >= (1LL << 30)) { /* ssw.c:626-641: s2 would overflow int32 */
      free(h_b); free(e_b); free(h_c); free(direction);
      return -2;
    }
    h_b = (int32_t *)realloc(h_b, (size_t)width * 4); e_b = (int32_t *)realloc(e_b, (size_t)width * 4);
    h_c = (int32_t *)realloc(h_c, (size_t)width * 4);
    free(direction);
    direction = (int8_t *)calloc((size_t)width_d * readLen * 3 + 8, 1); /* 0 = never written */
    for (int32_t j = 1; j < width - 1; j++) h_b[j] = 0; /* ssw.c:645 */
    /* e_b is uninitialised in the reference; every slot is written (or zeroed at [0]/[edge]) before it
       is read — see DESIGN.md "banded_sw emulation". h_c likewise. */
    for (int32_t j = 0; j < width; j++) { e_b[j] = 0; h_c[j] = 0; }
    for (int32_t i = 0; i < readLen; i++) {
      int32_t beg = 0, end = refLen - 1, u = 0, edge, f;
      int32_t j = i - band_width; beg = beg > j ? beg : j;
      j = i + band_width; end = end < j ? end : j;
      edge = end + 1 < width - 1 ? end + 1 : width - 1;
      f = h_b[0] = e_b[0] = h_b[edge] = e_b[edge] = h_c[0] = 0; /* ssw.c:653-654 */
      int8_t *dl = direction + (size_t)width_d * i * 3;
      for (j = beg; j <= end; j++) {
        int32_t b, e1, f1, d, de, df, dh, e, t1, t2;
        SET_U(u, band_width, i, j); SET_U(e, band_width, i - 1, j);
        SET_U(b, band_width, i, j - 1); SET_U(d, band_width, i - 1, j - 1);
        SET_D(de, band_width, i, j, 0); SET_D(df, band_width, i, j, 1); SET_D(dh, band_width, i, j, 2);
        t1 = i == 0 ? -go : h_b[e] - go;
        t2 = i == 0 ? -ge : e_b[e] - ge;
        e_b[u] = t1 > t2 ? t1 : t2;
        dl[de] = t1 > t2 ? 3 : 2;
        t1 = h_c[b] - go; t2 = f - ge;
        f = t1 > t2 ? t1 : t2;
        dl[df] = t1 > t2 ? 5 : 4;
        e1 = e_b[u] > 0 ? e_b[u] : 0; f1 = f > 0 ? f : 0;
        t1 = e1 > f1 ? e1 : f1;
        t2 = h_b[d] + sc(p, ref[j], read[i]);
        h_c[u] = t1 > t2 ? t1 : t2;
        if (h_c[u] > max) max = h_c[u];
        if (t1 <= t2) dl[dh] = 1; else dl[dh] = e1 > f1 ? dl[de] : dl[df];
      }
      for (j = 1; j <= u; j++) h_b[j] = h_c[j]; /* ssw.c:691 */
    }
    band_width *= 2;
  } while (max < score);
  band_width /= 2;

  /* trace back, ssw.c:698-771 */
  int32_t i = readLen - 1, j = refLen - 1, e = 0, l = 0, f = 0, cur = 0, t2 = 2, undefined = 0;
  uint32_t *c = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)(readLen + refLen + 4));
  while (i > 0) {
    int32_t lo = i - band_width > 0 ? i - band_width : 0;
    int32_t hi = i + band_width < refLen - 1 ? i + band_width : refLen - 1;
    if (j < lo || j > hi) { undefined = 1; break; }
    int32_t t1; SET_D(t1, band_width, i, j, t2);
    int8_t code = direction[(size_t)width_d * i * 3 + t1];
    switch (code) {
      case 1: --i; --j; t2 = 2; f = 0; break;
      case 2: --i; t2 = 0; f = 1; break;
      case 3: --i; t2 = 2; f = 1; break;
      case 4: --j; t2 = 1; f = 2; break;
      case 5: --j; t2 = 2; f = 2; break;
      default: undefined = 1; break;
    }
    if (undefined) break;
    if (f == cur) ++e;
    else { ++l; c[l - 1] = (uint32_t)e << 4 | (uint32_t)cur; cur = f; e = 1; }
  }
  int32_t n = -1;
  if (!undefined) {
    if (f == 0) { ++l; c[l - 1] = (uint32_t)(e + 1) << 4; }
    else { l += 2; c[l - 2] = (uint32_t)e << 4 | (uint32_t)f; c[l - 1] = 16; }
    n = l;
    if ((uint32_t)l > cap) *overflow = 1;
    for (int32_t s = 0; s < l && (uint32_t)s < cap; s++) cig[s] = c[l - 1 - s]; /* reverse, ssw.c:773-783 */
  }
  free(c); free(h_b); free(e_b); free(h_c); free(direction);
  return n;
}

/* ssw_cpp.cpp:234-283 (Aligner::Align) -> ssw.c:808-833 (ssw_init) + ssw.c:841-951 (ssw_align) */
void ko_ssw_align(const char *qs, int32_t qlen, const char *rs, int32_t rlen, const ko_params *p,
                  ko_overlap *out, uint32_t *cigar, uint32_t cigar_cap) {
  int8_t *q = (int8_t *)malloc((size_t)qlen + 1), *r = (int8_t *)malloc((size_t)rlen + 1);
  int8_t *qr = (int8_t *)malloc((size_t)qlen + 1);
  int32_t *buf = (int32_t *)malloc(sizeof(int32_t) * 9 * (size_t)(qlen + 16));
  for (int32_t i = 0; i < qlen; i++) q[i] = ssw_code(qs[i]);
  for (int32_t i = 0; i < rlen; i++) r[i] = ssw_code(rs[i]);
  int8_t mat[25];
  int32_t bias = 0;
  for (int a = 0; a < 5; a++) for (int b = 0; b < 5; b++) { mat[a * 5 + b] = (int8_t)sc(p, (int8_t)a, (int8_t)b); if (mat[a * 5 + b] < bias) bias = mat[a * 5 + b]; }
  bias = abs(bias);                                                            /* ssw.c:817-822 */
  const int32_t go = (uint8_t)p->gap_open, ge = (uint8_t)p->gap_extend;
  out->cigar_len = 0; out->flags = 0;
  /* forward: byte pass, word pass when the byte pass overflowed (ssw.c:868-877) */
  int word = 0;
  sw_end fw = sw_striped(r, 0, rlen, q, qlen, mat, go, ge, 255, 0, bias, buf);
  if (fw.score == 255) { fw = sw_striped(r, 0, rlen, q, qlen, mat, go, ge, 65535, 1, bias, buf); word = 1; }
  out->sw_score = (uint16_t)fw.score; out->ref_end = fw.ref; out->query_end = fw.read;
  if (fw.score == 0) {
    /* degenerate (ssw.c:169 end_ref=-1; reverse pass over an empty range): begins -1 / 0;
       with cigar requested the reference reads ref[-1] — undefined, flagged */
    out->ref_end = -1; out->query_end = 0; out->ref_begin = -1; out->query_begin = 0;
    if (p->report_cigar && 0 >= (int32_t)(uint16_t)p->score_threshold) out->flags |= KO_FLAG_UNDEFINED;
    goto done;
  }
  /* reverse pass, ssw.c:905-923 */
  for (int32_t i = 0; i <= fw.read; i++) qr[i] = q[fw.read - i]; /* seq_reverse ssw.c:794-806 */
  {
    const sw_end rv = sw_striped(r, 1, fw.ref + 1, qr, fw.read + 1, mat, go, ge, word ? fw.score : (int32_t)(uint8_t)fw.score, word, bias, buf);
    out->ref_begin = rv.ref; out->query_begin = fw.read - rv.read;
  }
  /* cigar, ssw.c:924-946; flag = 0x0f iff report_cigar (ssw_cpp.cpp:90-93), filters = score_filter */
  if (p->report_cigar && fw.score >= (int32_t)(uint16_t)p->score_threshold) {
    int overflow = 0;
    int32_t refLen = out->ref_end - out->ref_begin + 1, readLen = out->query_end - out->query_begin + 1;
    if (out->ref_begin < 0 || refLen <= 0 || readLen <= 0) { out->flags |= KO_FLAG_UNDEFINED; goto done; }   /* banded_sw would read outside ref / read */
    int32_t n = banded_cigar(r + out->ref_begin, q + out->query_begin, refLen, readLen, fw.score, p,
                             cigar, cigar_cap, &overflow);
    if (n == -2) { out->cigar_len = 0; out->sw_score = 0; }   /* ssw.c:941-944 */
    else if (n < 0) out->flags |= KO_FLAG_UNDEFINED;
    else { out->cigar_len = (uint32_t)n; if (overflow) out->flags |= KO_FLAG_CIGAR_OVERFLOW; }
  }
done:
  free(q); free(r); free(qr); free(buf);
}

/* The same alignment through the un-striped scan (plain Gotoh): the cross-check of the striped restatement inside the
 * domain where the two are equal. Fills score and the four coordinates only. */
void ko_ssw_align_gotoh(const char *qs, int32_t qlen, const char *rs, int32_t rlen, const ko_params *p, ko_overlap *out) {
  int8_t *q = (int8_t *)malloc((size_t)qlen + 1), *r = (int8_t *)malloc((size_t)rlen + 1), *qr = (int8_t *)malloc((size_t)qlen + 1);
  int32_t *H = (int32_t *)malloc(sizeof(int32_t) * 2 * (size_t)(qlen + 1)), *E = H + qlen + 1;
  for (int32_t i = 0; i < qlen; i++) q[i] = ssw_code(qs[i]);
  for (int32_t i = 0; i < rlen; i++) r[i] = ssw_code(rs[i]);
  memset(out, 0, sizeof *out);
  sw_end fw = sw_scan(r, rlen, 0, q, qlen, p, -1, H, E);
  out->sw_score = (uint16_t)fw.score; out->ref_end = fw.ref; out->query_end = fw.read;
  if (fw.score == 0) { out->ref_end = -1; out->query_end = 0; out->ref_begin = -1; out->query_begin = 0; }
  else {
    for (int32_t i = 0; i <= fw.read; i++) qr[i] = q[fw.read - i];
    sw_end rv = sw_scan(r, fw.ref + 1, 1, qr, fw.read + 1, p, fw.score, H, E);
    out->ref_begin = rv.ref; out->query_begin = fw.read - rv.read;
  }
  free(q); free(r); free(qr); free(H);
}

void ko_ssw_batch(uint64_t n, const char *q, const uint64_t *qoffs, const char *r,
                  const uint64_t *roffs, const ko_params *p, ko_overlap *out, uint32_t *cigar_pool,
                  uint32_t cigar_cap, int threads) {
  if (threads <= 0) threads = 1;
#pragma omp parallel for schedule(dynamic, 64) num_threads(threads)
  for (int64_t i = 0; i < (int64_t)n; i++) {
    memset(&out[i], 0, sizeof(ko_overlap));
    out[i].cigar_off = (uint32_t)(i * cigar_cap);
    ko_ssw_align(q + qoffs[i], (int32_t)(qoffs[i + 1] - qoffs[i]), r + roffs[i],
                 (int32_t)(roffs[i + 1] - roffs[i]), p, &out[i],
                 cigar_pool ? cigar_pool + (uint64_t)i * cigar_cap : NULL, cigar_cap);
  }
}

/* sequenceTools.h:77-116 (inPlaceReverseComplement): swaps upper-case ACGT only */
static inline char comp_char(char c) {
  switch (c) { case 'A': return 'T'; case 'T': return 'A'; case 'C': return 'G'; case 'G': return 'C'; default: return c; }
}

/* SmithWaterman.h:184-233 (performSmithWatermanOnRange2) */
void ko_align_seeds(uint64_t n_seeds, ko_overlap *ov, const char *read_bases, const uint64_t *read_offs,
                    const char *gen_bases, const uint64_t *gen_offs, const ko_params *p,
                    uint32_t *cigar_pool, uint32_t cigar_cap, int threads) {
  if (threads <= 0) threads = 1;
#pragma omp parallel for schedule(dynamic, 64) num_threads(threads)
  for (int64_t s = 0; s < (int64_t)n_seeds; s++) {
    ko_overlap *o = &ov[s];
    const char *q = read_bases + read_offs[o->read];
    int64_t qlen = (int64_t)(read_offs[o->read + 1] - read_offs[o->read]);
    int64_t glen = (int64_t)(gen_offs[o->entry + 1] - gen_offs[o->entry]);
    int64_t start = o->rel > 0 ? o->rel : 0;                   /* SmithWaterman.h:205 */
    int64_t wlen = start >= glen ? 0 : (glen - start < qlen ? glen - start : qlen); /* substr clamps, :206-207 */
    char *w = (char *)malloc((size_t)wlen + 1);
    const char *g = gen_bases + gen_offs[o->entry] + start;
    if (o->rev_comp) for (int64_t i = 0; i < wlen; i++) w[i] = comp_char(g[wlen - 1 - i]); /* :208 */
    else memcpy(w, g, (size_t)wlen);
    uint32_t *cig = cigar_pool ? cigar_pool + (uint64_t)s * cigar_cap : NULL;
    o->cigar_off = (uint32_t)(s * cigar_cap);
    ko_ssw_align(q, (int32_t)qlen, w, (int32_t)wlen, p, o, cig, cigar_cap);
    if (o->rev_comp) {                                         /* :212-227 */
      if (p->report_cigar && o->cigar_len && cig) {
        uint32_t n = o->cigar_len < cigar_cap ? o->cigar_len : cigar_cap;
        for (uint32_t a = 0, b = n - 1; a < b; a++, b--) { uint32_t t = cig[a]; cig[a] = cig[b]; cig[b] = t; }
      }
      int32_t t = o->ref_begin;
      o->ref_begin = (int32_t)wlen - (o->ref_end + 1); o->ref_end = (int32_t)wlen - (t + 1);
      t = o->query_begin;
      o->query_begin = (int32_t)qlen - (o->query_end + 1); o->query_end = (int32_t)qlen - (t + 1);
    }
    o->ref_begin += (int32_t)start; o->ref_end += (int32_t)start; /* :228-229 */
    free(w);
  }
}

/* ------------------------------------------------------------------ pairing */

static uint32_t g_mid; /* qsort has no context argument; ko_sort_for_pairing is not re-entrant */
/* PairedOverlap.h:248-257; ties (H3) broken by read index then rev_comp for a canonical order */
static int cmp_pairsort(const void *a, const void *b) {
  const ko_overlap *x = (const ko_overlap *)a, *y = (const ko_overlap *)b;
  uint32_t px = x->read % g_mid, py = y->read % g_mid;
  if (px != py) return px < py ? -1 : 1;
  if (x->entry != y->entry) return x->entry < y->entry ? -1 : 1;
  if (x->rel != y->rel) return x->rel < y->rel ? -1 : 1;
  if (x->read != y->read) return x->read < y->read ? -1 : 1;
  if (x->rev_comp != y->rev_comp) return x->rev_comp < y->rev_comp ? -1 : 1;
  return 0;
}
void ko_sort_for_pairing(ko_overlap *ov, uint64_t n, uint32_t mid) {
  g_mid = mid;
  qsort(ov, n, sizeof(ko_overlap), cmp_pairsort);
}

static void emit_single(ko_pair *out, uint64_t *cnt, const ko_overlap *ov, int64_t idx, int is_r1) {
  if (out) {
    ko_pair *p = &out[*cnt];
    p->combined_score = (uint16_t)ov[idx].sw_score; p->entry = ov[idx].entry;
    p->ref_start = ov[idx].ref_begin; p->ref_end = ov[idx].ref_end; p->insert_size = 0;
    p->r1_idx = is_r1 ? (int32_t)idx : -1; p->r2_idx = is_r1 ? -1 : (int32_t)idx; p->pad = 0;
  }
  (*cnt)++;
}
/* PairedOverlap.h:107-123 (makePair) */
static void emit_pair(ko_pair *out, uint64_t *cnt, const ko_overlap *ov, int64_t r1, int64_t r2,
                      int orientation, const uint32_t *read_lens) {
  if (out) {
    ko_pair *p = &out[*cnt];
    p->combined_score = (uint16_t)(ov[r1].sw_score + ov[r2].sw_score); /* u16 ctor parameter */
    p->entry = ov[r2].entry;
    p->ref_start = ov[r1].ref_begin < ov[r2].ref_begin ? ov[r1].ref_begin : ov[r2].ref_begin;
    p->ref_end = ov[r1].ref_end > ov[r2].ref_end ? ov[r1].ref_end : ov[r2].ref_end;
    p->insert_size = orientation ? (uint32_t)(ov[r2].rel - ov[r1].rel) + read_lens[ov[r2].read]
                                 : (uint32_t)(ov[r1].rel - ov[r2].rel) + read_lens[ov[r1].read];
    p->r1_idx = (int32_t)r1; p->r2_idx = (int32_t)r2; p->pad = 0;
  }
  (*cnt)++;
}

/* PairedOverlap.h:132-242 (getPairsFromRead) driven by :258-262 */
uint64_t ko_pair_overlaps(const ko_overlap *ov, uint64_t n, uint32_t mid, const uint32_t *read_lens, ko_pair *out) {
  uint64_t cnt = 0, cur = 0;
  while (cur < n) {
    uint32_t pid = ov[cur].read % mid, entry = ov[cur].entry;
    int64_t l1 = -1, l2 = -1, l1rc = -1, l2rc = -1;
    int u1 = 0, u2 = 0, u1rc = 0, u2rc = 0;
    while (cur < n && ov[cur].read % mid == pid && ov[cur].entry == entry) {
      if (ov[cur].read < mid) {
        if (ov[cur].rev_comp) {
          if (!u1rc && l1rc >= 0) emit_single(out, &cnt, ov, l1rc, 1);
          l1rc = (int64_t)cur; u1rc = 0;
          if (l2 >= 0) { emit_pair(out, &cnt, ov, (int64_t)cur, l2, 0, read_lens); u1rc = 1; u2 = 1; }
        } else {
          if (!u1 && l1 >= 0) emit_single(out, &cnt, ov, l1, 1);
          l1 = (int64_t)cur; u1 = 0;
          if (l2rc >= 0) { emit_pair(out, &cnt, ov, (int64_t)cur, l2rc, 0, read_lens); u1 = 1; u2rc = 1; }
        }
      } else {
        if (ov[cur].rev_comp) {
          if (!u2rc && l2rc >= 0) emit_single(out, &cnt, ov, l2rc, 0);
          l2rc = (int64_t)cur; u2rc = 0;
          if (l1 >= 0) { emit_pair(out, &cnt, ov, l1, (int64_t)cur, 1, read_lens); u1 = 1; u2rc = 1; }
        } else {
          if (!u2 && l2 >= 0) emit_single(out, &cnt, ov, l2, 0);
          l2 = (int64_t)cur; u2 = 0;
          if (l1rc >= 0) { emit_pair(out, &cnt, ov, l1rc, (int64_t)cur, 1, read_lens); u1rc = 1; u2 = 1; }
        }
      }
      cur++;
    }
    if (!u2 && l2 >= 0) emit_single(out, &cnt, ov, l2, 0);       /* PairedOverlap.h:217-240 */
    if (!u2rc && l2rc >= 0) emit_single(out, &cnt, ov, l2rc, 0);
    if (!u1 && l1 >= 0) emit_single(out, &cnt, ov, l1, 1);
    if (!u1rc && l1rc >= 0) emit_single(out, &cnt, ov, l1rc, 1);
  }
  return cnt;
}
