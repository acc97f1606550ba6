// sw_band.cuh — banded forward / reverse Smith-Waterman sweep, exact by construction (included by sw.cu).
//
// Why a band can be EXACT here. An alignment that scores S needs at least a = ceil(S / match) diagonal steps.
// A path that touches matrix offset d = j - i consumes d extra columns (d >= 0) or -d extra rows, so inside an
// m x n matrix it has at most n - d (resp. m + d) diagonal steps. Hence EVERY alignment scoring >= S lies inside
// the offsets [-(m - a), n - a].
//   MODE 0 (forward, nothing known): sweep a W-diagonal band placed on that interval's centre, take the best score
//     S' found in it (a true alignment score, so S' <= S); if [-(m - a'), n - a'] fits in the band then all
//     alignments scoring >= S' — every optimal one, hence every cell SSW's tie rules (ssw.c:316-342) look at — are
//     inside the band and were computed with their true H: exact. Otherwise S' is kept as a lower bound and the
//     alignment moves to the next tier (a 64-wide band placed exactly on [-(m - a'), ...] if that is <= 64 wide,
//     else the full-matrix kernel k_sw_fast).
//   MODE 2 (forward, lower bound S' known): band placed at c0 = -(m - a'); it contains every alignment scoring
//     >= S', so the sweep is exact without a further check (the check is still evaluated; a failure would fall back).
//   MODE 1 (reverse pass, ssw.c:905-923): S is known and every alignment scoring S starts at the reversed origin, so
//     the band is the interval an anchored path can reach (reverse_band below), about half of [-(rows - a), cols - a].
//
// Mapping: ONE THREAD owns two alignments (halves of s16x2 registers) and keeps the band's previous row (H), the
// vertical-gap state (V) and W PRMT column selectors in registers; it walks the rows, W cells per row fully
// unrolled, 7 DPX/PRMT ops per cell pair, no shuffles and no shared memory. Column selectors slide by one
// register per row (moves go to the FMA pipe; the ALU pipe only sees the recurrences). Band cells that fall
// outside the matrix use "replicate-sign" selectors that can only produce 0 or -1, so they stay at H = 0 on the
// left and can never reach a maximum on the right. Per-alignment inputs (column selectors and query codes) come
// from two planes written by k_band_bytes as ready-made PRMT selectors, one coalesced load each per row and pair, so
// the per-row overhead next to the W x 7 cell ops is two PRMTs, the row-winner compare and the selector slide.
#pragma once
#include <type_traits>

#define SWB_MAXROWS 160
#define SWB_BLOCK 64
#define SWB_MAXW 128

// shared-memory selector streams of one CTA, word w of thread t at [w * SWB_BLOCK + t] (conflict-free): per alignment
// (SWB_MAXROWS + W + 4) column-selector bytes, plus one byte per query row holding both alignments' row codes
template <int W> struct BandSmem {      // W = slots per lane; + 4: the lanes of a multi-lane band lag up to 3 rows
  static constexpr int COLW = (SWB_MAXROWS + 4 + W + 4 + 7) / 8;        // column stream: one NIBBLE per column, eight per word
  static constexpr int QW = (SWB_MAXROWS + 4 + 4 + 3) / 4;
  static constexpr int WORDS = 2 * COLW + QW;
  static constexpr size_t BYTES = (size_t)WORDS * SWB_BLOCK * 4;
};

__device__ __forceinline__ int32_t ceil_div_pos(int32_t a, int32_t b) { return (a + b - 1) / b; }

// Slot reservation in an append-only work list from divergent code: the lanes that are here together take one atomic
// (millions of single-lane atomics on ONE counter serialise in L2: 12 ms for the 25 M full-matrix fallbacks of config 2).
__device__ __forceinline__ uint32_t list_slot(uint32_t *counter) {
  const uint32_t peers = __activemask(), lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
  uint32_t base = 0;
  if (lane == leader) base = atomicAdd(counter, (uint32_t)__popc(peers));
  base = __shfl_sync(peers, base, leader);
  return base + __popc(peers & ((1u << lane) - 1u));
}

// the same with one counter per key: the lanes here together are grouped by key first
__device__ __forceinline__ uint32_t list_slot_keyed(uint32_t *counters, uint32_t key) {
  const uint32_t peers = __match_any_sync(__activemask(), key), lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
  uint32_t base = 0;
  if (lane == leader) base = atomicAdd(counters + key, (uint32_t)__popc(peers));
  base = __shfl_sync(peers, base, leader);
  return base + __popc(peers & ((1u << lane) - 1u));
}

// 32 two-bit codes of `plane` starting at base p of the sequence that begins at word w_word (p may be negative or run
// past the window: those lanes are masked by the caller; guard words keep the reads inside the allocation)
__device__ __forceinline__ uint64_t bits_at(const uint64_t *__restrict__ plane, uint64_t w_word, int32_t p) {
  const int32_t wi = p >> 5; const uint32_t sh = (uint32_t)p & 31u;
  const uint64_t lo = wi >= 0 ? __ldg(&plane[w_word + wi]) : 0ull;
  if (sh == 0) return lo;
  const uint64_t hi = wi + 1 >= 0 ? __ldg(&plane[w_word + wi + 1]) : 0ull;
  return (lo >> (2 * sh)) | (hi << (64 - 2 * sh));
}
__device__ __forceinline__ uint32_t mask_at(const uint32_t *__restrict__ plane, uint64_t w_word, int32_t p) {
  const int32_t wi = p >> 5; const uint32_t sh = (uint32_t)p & 31u;
  const uint32_t lo = wi >= 0 ? __ldg(&plane[w_word + wi]) : 0u, hi = wi + 1 >= 0 ? __ldg(&plane[w_word + wi + 1]) : 0u;
  return __funnelshift_r(lo, hi, sh);
}
__device__ __forceinline__ uint64_t pair_mask(uint32_t m) {     // bit b -> bits 2b and 2b+1
  uint64_t x = m;
  x = (x | (x << 16)) & 0x0000FFFF0000FFFFull; x = (x | (x << 8)) & 0x00FF00FF00FF00FFull;
  x = (x | (x << 4)) & 0x0F0F0F0F0F0F0F0Full; x = (x | (x << 2)) & 0x3333333333333333ull;
  x = (x | (x << 1)) & 0x5555555555555555ull;
  return x * 3ull;
}
__device__ __forceinline__ uint64_t reverse_pairs(uint64_t e) {     // 2-bit group g -> group 31 - g
  e = __brevll(e);
  return ((e >> 1) & 0x5555555555555555ull) | ((e & 0x5555555555555555ull) << 1);
}

// ---- reverse pass: the band an ANCHORED alignment can reach -------------------------------------------------
// The reverse sweep (ssw.c:905-923) runs over the reversed prefixes read[0..read_end], ref[0..ref_end] and looks for the
// first column holding a cell with H == S, S the forward score. Every alignment scoring S inside that prefix rectangle
// ends exactly at (read_end, ref_end): the forward pass took the FIRST column attaining S and the SMALLEST row in it
// (ssw.c:316-342), so none can end in an earlier column or row. In the reversed matrix all of them therefore start at the
// origin, offset 0, and one that touches offset d > 0 holds at least d horizontal gap bases — cost >= gapOpen +
// (d - 1) gapExtend, one gap being the cheapest way to get there while gapExtend <= gapOpen (always true where these
// kernels run, kslam_params_fast) — and has at most min(rows, cols - d) diagonal steps. It can only score S if
//     match * min(rows, cols - d) - gapOpen - (d - 1) gapExtend >= S.
// anchored_reach() is the largest such d (0: the path stays on the main diagonal); the same with rows and columns swapped
// bounds the negative offsets. The interval is about half of [-(rows - a), cols - a], which ignores both the anchor and
// the gap costs, so most reverse sweeps drop one tier. The in-band cells are a lower bound of the true H (paths leaving
// the band are cut) and never exceed S, so a cell equals S iff an S-path reaches it: the set SSW's rule looks at.
__host__ __device__ __forceinline__ int32_t anchored_reach(int32_t other, int32_t shrinking, int32_t S, int32_t match, int32_t go, int32_t ge) {
  const int32_t nb = match * shrinking - go + ge - S;      // match (shrinking - d) - go - (d - 1) ge >= S
  const int32_t na = match * other - go - S;               // match other - go - (d - 1) ge >= S
  if (nb < 0 || na < 0) return 0;
  int32_t d = nb / (match + ge);
  if (ge > 0) { const int32_t da = 1 + na / ge; d = d < da ? d : da; }
  if (d > shrinking - 1) d = shrinking - 1;
  return d > 0 ? d : 0;
}
// offsets [lo, hi] of the reverse band of an alignment scoring S whose reversed prefixes are rows x cols
__host__ __device__ __forceinline__ void reverse_band(int32_t rows, int32_t cols, int32_t S, const SwScore &sc, int32_t *lo, int32_t *hi) {
  *hi = anchored_reach(rows, cols, S, sc.match, sc.gap_open, sc.gap_extend);
  *lo = -anchored_reach(cols, rows, S, sc.match, sc.gap_open, sc.gap_extend);
}

// geometry of one alignment inside the band sweep
struct BandGeo { int32_t rows, cols, c0; };

template <int MODE, int W>
__device__ __forceinline__ BandGeo band_geo(const SwTask &t, const SwRes &r, const SwScore &sc) {
  BandGeo g;
  if (MODE == 1) {
    g.rows = r.read_end + 1; g.cols = r.ref_end + 1;
    int32_t hi;
    reverse_band(g.rows, g.cols, r.score, sc, &g.c0, &hi);
  } else {
    g.rows = (int32_t)t.m; g.cols = (int32_t)t.n;
    if (MODE == 0) g.c0 = ((g.cols - g.rows) >> 1) - W / 2;   // centre of [-(m - a), n - a] is (n - m) / 2 whatever a is
    else g.c0 = -(g.rows - ceil_div_pos(r.score, sc.match));   // r.score = proven lower bound from the 32-wide sweep
  }
  return g;
}

// ---- selector streams ------------------------------------------------------------------------------------
// Column stream of one alignment: nibble k = 2-bit code of matrix column j = k + c0 in the sweep's orientation, 4 =
// outside the matrix, eight columns per word; col_selectors() turns four nibbles into PRMT selector bytes for
// alignment A or B. 32 columns are fetched as one oriented 2-bit word.
// NCOL: the window may hold code-4 bases; their columns get nibble 5 (the selector LUTs answer it with a byte whose bit 7
// is clear, which make_selector turns into a masking second selector).
template <int MODE, bool NCOL>
__device__ __forceinline__ void fill_col_stream(const SwPlanes &pl, const SwTask &t, const SwRes &r, const BandGeo &g,
                                                int32_t kmax, uint32_t *__restrict__ col) {
  constexpr bool REVERSE = MODE == 1;
  const bool rev = (t.flags & SWT_REV) != 0;
  // genome position of matrix column j is P0 + sg * j (window reversal and the reverse sweep both flip the sign)
  int32_t P0, sg;
  if (!REVERSE) { P0 = rev ? (int32_t)(t.w_start + t.n - 1) : (int32_t)t.w_start; sg = rev ? -1 : 1; }
  else { P0 = rev ? (int32_t)(t.w_start + t.n - 1) - r.ref_end : (int32_t)t.w_start + r.ref_end; sg = rev ? 1 : -1; }
  for (int32_t k0 = 0; k0 < kmax; k0 += 32) {
    const int32_t j0 = g.c0 + k0;
    const int32_t lo = j0 < 0 ? -j0 : 0, hi = g.cols - j0 < 32 ? g.cols - j0 : 32;
    uint32_t valid = 0, ncols = 0;
    uint64_t codes = 0;
    if (hi > lo) {
      valid = (hi - lo >= 32 ? 0xffffffffu : ((1u << (hi - lo)) - 1u) << lo);
      if (sg > 0) {
        const int32_t p = P0 + j0;
        codes = bits_at(pl.w_sbits, t.w_word, p);
        if (rev) codes ^= pair_mask(~mask_at(pl.w_xmask, t.w_word, p));          // complement unless a/c/g/t/U/u
        if (NCOL) ncols = mask_at(pl.w_nmask, t.w_word, p) & valid;
      } else {
        const int32_t p = P0 - j0 - 31;                                            // column j0 + b <-> base p + 31 - b
        codes = reverse_pairs(bits_at(pl.w_sbits, t.w_word, p));
        if (rev) codes ^= pair_mask(~__brev(mask_at(pl.w_xmask, t.w_word, p)));
        if (NCOL) ncols = __brev(mask_at(pl.w_nmask, t.w_word, p)) & valid;
      }
    }
#pragma unroll
    for (int grp = 0; grp < 4; grp++) {                      // eight columns per word: nibble = 2-bit code, 4 = outside the matrix
      if (k0 + 8 * grp >= kmax) break;
      uint32_t n = (uint32_t)(codes >> (16 * grp)) & 0xffffu;
      n = (n | (n << 8)) & 0x00ff00ffu; n = (n | (n << 4)) & 0x0f0f0f0fu; n = (n | (n << 2)) & 0x33333333u;
      const uint32_t inv = ~(valid >> (8 * grp)) & 0xffu;
      if (inv) {
        uint32_t m = (inv | (inv << 12)) & 0x000f000fu; m = (m | (m << 6)) & 0x03030303u; m = (m | (m << 3)) & 0x11111111u;   // bit 0 of nibble b
        n = (n & ~(m * 3u)) | (m << 2);
      }
      if (NCOL) {
        const uint32_t nc = (ncols >> (8 * grp)) & 0xffu;
        if (nc) {
          uint32_t m = (nc | (nc << 12)) & 0x000f000fu; m = (m | (m << 6)) & 0x03030303u; m = (m | (m << 3)) & 0x11111111u;
          n = (n & ~(m * 15u)) | (m * 5u);
        }
      }
      col[(size_t)(k0 / 8 + grp) * SWB_BLOCK] = n;
    }
  }
}
// four selector bytes (columns k .. k + 3 of a nibble stream, k a multiple of 4) for alignment A (nibbles {w, 8|w} on
// profile A) or B ({4|w, 12|w} on profile B); outside the matrix: replicate the sign of byte 0. PRMT reads the low 16
// bits of its selector only, so the four nibbles need no masking.
__device__ __forceinline__ uint32_t col_selectors(const uint32_t *__restrict__ col, int32_t k, bool is_b) {
  const uint32_t w = col[(size_t)(k >> 3) * SWB_BLOCK] >> (4 * (k & 7));
  return is_b ? prmt(0xF7E6D5C4u, 0x000044CCu, w) : prmt(0xB3A29180u, 0x00000088u, w);     // nibble 5 (code-4 column): 0x44 / 0x00, bit 7 clear
}
// One selector register from byte r of both alignments' selector words. NCOL: its upper half carries a SECOND selector for
// a PRMT over (score, 0) that passes the score of an alignment through (bytes 0-1 / 2-3) or replaces it by zero where that
// alignment's column is a code-4 base (selector byte with bit 7 clear): 0x3210 -> 0x..44 / 0x44...
template <bool NCOL>
__device__ __forceinline__ uint32_t make_selector(uint32_t wa, uint32_t wb, int r) {
  const uint32_t x = prmt(wa, wb, (uint32_t)(((4 + r) << 4) | r));
  if (!NCOL) return x;
  const uint32_t ma = ((x >> 7) & 1u) - 1u, mb = ((x >> 15) & 1u) - 1u;                      // all ones where the column is a code-4 base
  return (x & 0xffffu) | ((0x3210u ^ (ma & 0x0054u) ^ (mb & 0x7600u)) << 16);
}

// row codes of one alignment for rows 32g .. 32g+31 of the sweep as bytes in four-row words: 0-3 = base, 4 = code-4
// base (scores 0 against everything, ssw_cpp.cpp:43-48), 5 = past the query end (mismatches everything)
template <int MODE>
__device__ __forceinline__ void q_group(const SwPlanes &pl, const SwTask &t, int32_t rows, int32_t g, uint32_t out[8]) {
  uint64_t codes; uint32_t nm;
  if (MODE != 1) {
    const bool in = 32 * g < rows;
    codes = in ? __ldg(&pl.q_sbits[t.q_word + g]) : 0ull; nm = in ? __ldg(&pl.q_nmask[t.q_word + g]) : 0u;
  } else {
    const int32_t p = rows - 1 - 32 * g - 31;                                       // sweep row 32g + b <-> query base p + 31 - b
    codes = reverse_pairs(bits_at(pl.q_sbits, t.q_word, p)); nm = __brev(mask_at(pl.q_nmask, t.q_word, p));
  }
  const int32_t nv = rows - 32 * g;                                                // rows of this group inside the query
#pragma unroll
  for (int grp = 0; grp < 8; grp++) {
    const uint32_t x8 = (uint32_t)(codes >> (8 * grp)) & 0xffu;
    uint32_t y = (x8 | (x8 << 12)) & 0x000f000fu; y = (y | (y << 6)) & 0x03030303u;  // byte b = code of row 4 grp + b
    const uint32_t n4 = (nm >> (4 * grp)) & 15u;
    if (n4 | (uint32_t)(nv < 4 * grp + 4)) {
#pragma unroll
      for (int b = 0; b < 4; b++) {
        if ((n4 >> b) & 1u) y = (y & ~(0xffu << (8 * b))) | (4u << (8 * b));
        if (4 * grp + b >= nv) y = (y & ~(0xffu << (8 * b))) | (5u << (8 * b));
      }
    }
    out[grp] = y;
  }
}

// Slot pairs (2p, 2p+1) of `list` share a thread group. Failures of the sweep-and-verify tier go to next_list (second
// round: tier_f[] gets the direct tier the interval they need fits, marked SWT_SWEPT and counted in tier2_count[]; the
// score lower bound is left in res[].score), else to fb_keys (full-matrix kernel, key = columns).
//
// PARTS > 1: the band is PARTS x WP diagonals wide and PARTS neighbouring lanes share it, lane `part` owning slots
// [part * WP, (part + 1) * WP). A cell needs its left neighbour of the same row (horizontal gap), the cell above-right
// in band coordinates (vertical gap) and its own slot of the row above (diagonal), so lane `part` runs `part` rows
// behind lane 0: at step s it works on row s - part, takes the horizontal-gap state its left neighbour left at the end of
// step s - 1 (same row) and, after its FIRST cell, hands that cell's vertical-gap output to its left neighbour, whose
// LAST cell of this step (one row further down, one column to the left in band terms = the same matrix column) is the
// one that needs it. Two shuffles per row and lane; everything else is the one-lane sweep with c0 advanced by
// part * (WP - 1) and the query rows delayed by `part`.
// resident CTAs per SM a tier is compiled for: narrow single-lane tiers need few registers and, with nibble streams, 22 KB
// of shared memory per CTA — their stalls are the plane loads of the stream fill, which more warps hide
template <int WP, int PARTS> struct BandOcc { static constexpr int CTAS = PARTS > 1 ? 6 : (WP <= 8 ? 10 : (WP <= 16 ? 9 : (WP <= 24 ? 7 : 6))); };
template <int MODE, int WP, int PARTS, bool NCOL>
__global__ void __launch_bounds__(SWB_BLOCK, (BandOcc<WP, PARTS>::CTAS))
k_sw_band(const SwTask *__restrict__ tasks, const uint32_t *__restrict__ list, uint32_t n_list, SwPlanes pl, SwScore sc,
          SwRes *__restrict__ res, Rec16 *__restrict__ fb_keys, uint32_t *__restrict__ fb_count,
          uint32_t *__restrict__ next_list, uint32_t *__restrict__ next_count, uint8_t *__restrict__ tier_f,
          uint32_t *__restrict__ tier2_count, uint32_t level, uint32_t one /* == 1, opaque to ptxas */) {
  constexpr bool REVERSE = MODE == 1;
  constexpr int W = WP * PARTS;                // diagonals of the whole band
  constexpr int NH = (WP + 31) / 32;           // tracking keys per 32-slot half
  constexpr int COLW = BandSmem<WP>::COLW;
  constexpr int GPW = 32 / PARTS;              // lane groups per warp (PARTS = 3 leaves two lanes idle)
  extern __shared__ uint32_t smem[];
  uint32_t *colA = smem + threadIdx.x, *colB = colA + COLW * SWB_BLOCK, *qAB = colB + COLW * SWB_BLOCK;
  const uint32_t lane = threadIdx.x & 31, part = PARTS == 1 ? 0u : lane % PARTS;
  uint32_t p;
  if (PARTS == 1) p = blockIdx.x * SWB_BLOCK + threadIdx.x;
  else {
    if (lane >= GPW * PARTS) return;
    p = (blockIdx.x * (SWB_BLOCK / 32) + (threadIdx.x >> 5)) * GPW + lane / PARTS;
  }
  if (2 * p >= n_list) return;                 // a whole group leaves together
  const uint32_t gmask = PARTS == 1 ? 0u : (((1u << PARTS) - 1u) << (lane - part));
  const bool single = 2 * p + 1 >= n_list;
  const uint32_t ia = list[2 * p], ib = single ? ia : list[2 * p + 1];
  const SwTask ta = tasks[ia], tb = tasks[ib];
  SwRes ra, rb;
  if (MODE != 0) { ra = res[ia]; rb = res[ib]; }
  BandGeo ga = band_geo<MODE, W>(ta, ra, sc), gb = band_geo<MODE, W>(tb, rb, sc);
  const int32_t rows[2] = {ga.rows, gb.rows}, cols[2] = {ga.cols, gb.cols}, c0[2] = {ga.c0, gb.c0};
  const int32_t rows_max = rows[0] > rows[1] ? rows[0] : rows[1];
  const int32_t rows4 = (rows_max + (PARTS - 1) + 3) & ~3;     // steps of the sweep, whole groups of four (lane `part` lags `part` rows)
  const int32_t slot0 = (int32_t)part * WP;                    // first band slot of this lane
  ga.c0 += (int32_t)part * (WP - 1); gb.c0 += (int32_t)part * (WP - 1);   // step s, local slot t <-> column s + t + c0

  // ---- unpack this thread's selector streams (low half = alignment A, high half = B; an unpaired last slot runs the
  // same alignment in both halves and drops the second result)
  fill_col_stream<MODE, NCOL>(pl, ta, ra, ga, rows4 + WP, colA);
  fill_col_stream<MODE, NCOL>(pl, tb, rb, gb, rows4 + WP, colB);
  for (int32_t g = 0; 32 * g < rows4 + 4; g++) {
    uint32_t qa[8], qb[8];
    q_group<MODE>(pl, ta, rows[0], g, qa);
    q_group<MODE>(pl, tb, rows[1], g, qb);
#pragma unroll
    for (int grp = 0; grp < 8; grp++)
      if (32 * g + 4 * grp < rows4 + 4) qAB[(size_t)(8 * g + grp) * SWB_BLOCK] = qa[grp] | (qb[grp] << 4);
  }

  const uint32_t mis_b = (uint32_t)(-(sc.mismatch * 32)) & 0xffu, mat_b = (uint32_t)(sc.match * 32) & 0xffu;
  const uint32_t PSRC = mis_b | (mat_b << 8);                 // bytes {mismatch, match, 0, 0}: source of every row profile
  const uint32_t QLUT0 = 0x20100201u, QLUT1 = 0x00000033u;    // row code 0-5 -> the byte naming its profile selector ...
  const uint32_t QSRC = 0x22100100u;                          // ... whose nibbles pick the selector's two bytes here
  const uint32_t NEG_GE = pack2(-sc.gap_extend * 32);
  // Biased cells: every H / gap value is stored + KB (sw_bias), so nothing the recurrences produce is ever negative: the
  // floor of a cell is KB instead of 0, gap states are bounded below by KB - gapOpen > 0 by their own recurrence (no
  // clamp needed), and "H - gapOpen" for both halves is ONE plain 32-bit add of -gapOpen * 0x10001 (no borrow can cross
  // the halves) — issued as an IMAD on the FMA pipe (mad_add), which leaves 6 ALU-pipe ops per cell pair instead of 7.
  const uint32_t KB = sw_bias(sc), K2 = KB * 0x10001u;
  const uint32_t NEG_GO32 = (uint32_t)(-(int32_t)(sc.gap_open * 32) * 0x10001);

  uint32_t H[WP], V[WP], sel[WP];
#pragma unroll
  for (int t = 0; t < WP; t += 4) {
    const uint32_t wa = col_selectors(colA, t, false), wb = col_selectors(colB, t, true);
#pragma unroll
    for (int r = 0; r < 4; r++) { H[t + r] = K2; V[t + r] = K2; sel[t + r] = make_selector<NCOL>(wa, wb, r); }
  }
  // forward: key = score * 32 | 31 of the best cell so far, info = row << 8 | band slot of that cell;
  // reverse: (rcol, info) = first (smallest scan column, then smallest row) cell reaching the forward score
  uint32_t keyA = KB + 31u, keyB = KB + 31u, infoA = 0, infoB = 0;
  uint32_t rcolA = 0xffffffffu, rcolB = 0xffffffffu;
  const uint32_t thrA = REVERSE ? (uint32_t)ra.score * 32u + KB : 0u, thrB = REVERSE ? (uint32_t)rb.score * 32u + KB : 0u;
  uint32_t e_end = K2, qprev = 0x55555555u;                   // (row code 5 for both alignments: the rows before row 0)
  const uint32_t qshift = 0x7654u - 0x1111u * part;           // bytes of {qprev, qcur} holding rows s - part .. s - part + 3
  // A cell of row i ends at most i + 1 diagonal steps, so it can reach the known bound B (MODE 2: the lower bound the
  // band was placed with; MODE 1: the forward score) only from row ceil(B / match) - 1 on: the rows before it run without
  // the tracking op (5 ALU ops per cell pair instead of 6) and without the row-winner code. The switch row is the
  // smallest one among the lanes that are here together, so a warp changes loops once.
  int32_t n_quiet = 0;
  if (MODE != 0) {
    const int32_t qa = ceil_div_pos(ra.score, sc.match) - 1, qb = ceil_div_pos(rb.score, sc.match) - 1;
    n_quiet = __reduce_min_sync(__activemask(), (qa < qb ? qa : qb)) & ~3;
    if (n_quiet < 0) n_quiet = 0;
    if (n_quiet > rows4) n_quiet = rows4;
  }
  auto sweep = [&](auto track_c, const int32_t i_begin, const int32_t i_end) {
  constexpr bool TRACK = decltype(track_c)::value;
  for (int32_t i0 = i_begin; i0 < i_end; i0 += 4) {
    uint32_t qword = qAB[(size_t)(i0 / 4) * SWB_BLOCK];
    if (PARTS > 1) { const uint32_t qcur = qword; qword = __byte_perm(qprev, qcur, qshift); qprev = qcur; }
    const uint32_t ewa = col_selectors(colA, i0 + WP, false), ewb = col_selectors(colB, i0 + WP, true);
#pragma unroll
    for (int r = 0; r < 4; r++) {
      const int32_t i = i0 + r - (int32_t)part;               // the matrix row this lane works on (negative: not started)
      // row profiles [s(q,A) s(q,C) s(q,G) s(q,T)] x 32 of both alignments from the row's code byte, PRMTs only
      const uint32_t codes = prmt(qword, 0u, 0x4440u | (uint32_t)r);
      const uint32_t q32 = prmt(QSRC, 0u, prmt(QLUT0, QLUT1, codes));
      const uint32_t PA = prmt(PSRC, 0u, q32), PB = prmt(PSRC, 0u, q32 >> 16);
      uint32_t e = K2, acc[NH];
      if (PARTS > 1) { const uint32_t left = __shfl_sync(gmask, e_end, part ? lane - 1 : lane); if (part) e = left; }
#pragma unroll
      for (int h = 0; h < NH; h++) acc[h] = 0;
#pragma unroll
      for (int t = 0; t < WP; t++) {
        uint32_t s = prmt(PA, PB, sel[t]);
        if (NCOL) s = prmt(s, 0u, sel[t] >> 16);                   // code-4 columns score 0 against every row
        const uint32_t v = V[t];
        uint32_t h = __viaddmax_s16x2(H[t], s, v);                // max(H[i-1][j-1] + s, vertical gap)
        h = __vimax3_s16x2(h, e, K2);                               // ... the horizontal gap and the floor (0, biased)
        H[t] = h;
        const uint32_t hgo = mad_add(h, one, NEG_GO32);             // H - gapOpen in both halves, on the FMA pipe
        e = __viaddmax_s16x2(e, NEG_GE, hgo);                      // horizontal gap into (i, j+1)
        if (t > 0) V[t - 1] = __viaddmax_s16x2(v, NEG_GE, hgo);    // vertical gap into (i+1, j): band slot t-1 next row
        else if (PARTS > 1) {                                      // ... which for slot 0 is the left neighbour's last slot, this step
          const uint32_t down = __shfl_sync(gmask, __viaddmax_s16x2(v, NEG_GE, hgo), part + 1 < PARTS ? lane + 1 : lane);
          V[WP - 1] = part + 1 < PARTS ? down : K2;
        }
        if (TRACK) acc[t / 32] = __viaddmax_s16x2(h, (uint32_t)(31 - (t & 31)) * 0x10001u, acc[t / 32]);   // H*32 + (31 - slot): smallest column wins ties
      }
      e_end = e;
      // slide the column selectors: next row's slot t is this row's slot t+1; the last slot takes the entering column
#pragma unroll
      for (int t = 0; t < WP - 1; t++) sel[t] = sel[t + 1];
      sel[WP - 1] = make_selector<NCOL>(ewa, ewb, r);
      // row winners -> running best. SSW's rule: first column attaining the maximum, then the smallest row
      // (ssw.c:316-342). Rows only grow, so a strictly larger score always wins (the common, branch-free path) and an
      // equal score wins only with a strictly smaller column.
      if (TRACK) {
#pragma unroll
      for (int h = 0; h < NH; h++) {
        const uint32_t aA = acc[h] & 0xffffu, aB = acc[h] >> 16;
        if (REVERSE) {
          if (aA >= thrA) { const uint32_t j = (uint32_t)(i + slot0 + 32 * h + (int32_t)(31u - (aA & 31u)) + c0[0]);
                            if (j < rcolA && j < 4096u) { rcolA = j; infoA = (uint32_t)i; } }
          if (aB >= thrB) { const uint32_t j = (uint32_t)(i + slot0 + 32 * h + (int32_t)(31u - (aB & 31u)) + c0[1]);
                            if (j < rcolB && j < 4096u) { rcolB = j; infoB = (uint32_t)i; } }
        } else {
          const uint32_t nA = ((uint32_t)i << 8) | ((uint32_t)(slot0 + 32 * h + 31) - (aA & 31u)), nB = ((uint32_t)i << 8) | ((uint32_t)(slot0 + 32 * h + 31) - (aB & 31u));
          if (aA > keyA) { keyA = aA | 31u; infoA = nA; }
          else if ((aA | 31u) == keyA && aA > KB + 31u && (nA >> 8) + (nA & 255u) < (infoA >> 8) + (infoA & 255u)) infoA = nA;
          if (aB > keyB) { keyB = aB | 31u; infoB = nB; }
          else if ((aB | 31u) == keyB && aB > KB + 31u && (nB >> 8) + (nB & 255u) < (infoB >> 8) + (infoB & 255u)) infoB = nB;
        }
      }
      }
    }
  }
  };
  sweep(std::false_type{}, 0, n_quiet);
  sweep(std::true_type{}, n_quiet, rows4);

  // ---- per-lane winners as one comparable word: forward score << 20 | (1023 - column) << 10 | (1023 - row), reverse
  // 1 << 31 | (4095 - column) << 12 | (4095 - row); 0 = nothing. The lanes of a group keep the largest.
  uint32_t win[2];
#pragma unroll
  for (int al = 0; al < 2; al++) {
    if (REVERSE) {
      const uint32_t rcol = al ? rcolB : rcolA, rrow = al ? infoB : infoA;
      win[al] = rcol != 0xffffffffu ? (0x80000000u | ((4095u - rcol) << 12) | (4095u - rrow)) : 0u;
    } else {
      const uint32_t key = al ? keyB : keyA, info = al ? infoB : infoA;
      const uint32_t S = (key - KB) >> 5, brow = info >> 8, bcol = (uint32_t)((int32_t)brow + (int32_t)(info & 255u) + c0[al]);
      win[al] = S > 0 ? ((S << 20) | ((1023u - bcol) << 10) | (1023u - brow)) : 0u;
    }
    if (PARTS > 1) {
#pragma unroll
      for (int k = 1; k < PARTS; k++) {
        const uint32_t o = __shfl_sync(gmask, win[al], lane - part + (part + k) % PARTS);
        win[al] = win[al] > o ? win[al] : o;
      }
    }
  }
  if (part != 0) return;

#pragma unroll
  for (int al = 0; al < 2; al++) {
    if (al == 1 && single) break;
    const uint32_t idx = al ? ib : ia;
    if (REVERSE) {
      const SwRes &r0 = al ? rb : ra;
      if (win[al]) {
        res[idx].ref_begin = r0.ref_end - (int32_t)(4095u - ((win[al] >> 12) & 4095u));
        res[idx].read_begin = r0.read_end - (int32_t)(4095u - (win[al] & 4095u));
        res[idx].flags = r0.flags | SWR_REV_TIER(SWR_TIER_OF_W(W));
      } else {                      // cannot happen when the bound holds; never guess: hand over to the full kernel
        const uint32_t k = list_slot(fb_count);
        fb_keys[k].key = (uint64_t)(r0.ref_end + 1); fb_keys[k].val = idx;
      }
    } else {
      const int32_t S = (int32_t)(win[al] >> 20);
      const int32_t bcol = (int32_t)(1023u - ((win[al] >> 10) & 1023u)), brow = (int32_t)(1023u - (win[al] & 1023u));
      const int32_t a = ceil_div_pos(S, sc.match);
      const bool proven = S > 0 && c0[al] <= -(rows[al] - a) && (cols[al] - a) <= c0[al] + (W - 1);
      const int32_t need = rows[al] + cols[al] - 2 * a + 1;      // width of the interval every alignment scoring >= S lies in
      if (proven) {
        SwRes o;
        o.flags = SWR_FWD_TIER(SWR_TIER_OF_W(W)); o.pad0 = o.pad1 = 0; o.ref_begin = -1; o.read_begin = 0;
        o.score = S; o.ref_end = bcol; o.read_end = brow;
        res[idx] = o;
      } else if (MODE == 0 && next_list && S > 0 && tier_of_interval(need, level) != SWT_TIER_NONE) {
        res[idx].score = S;         // lower bound: every alignment scoring >= S lies in [-(m - a), n - a]
        const uint32_t t2 = NCOL ? ncol_tier(tier_of_interval(need, level)) : tier_of_interval(need, level);
        tier_f[idx] = (uint8_t)(t2 | SWT_SWEPT | (NCOL ? SWT_NCOL : 0u));
        list_slot_keyed(tier2_count, t2 + (NCOL ? SWT_N_DIRECT : 0u));
        next_list[list_slot(next_count)] = idx;
      } else {
        const uint32_t k = list_slot(fb_count);
        fb_keys[k].key = (uint64_t)(al ? tb.n : ta.n); fb_keys[k].val = idx;
      }
    }
  }
}
