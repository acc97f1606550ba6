// sw.cu — Smith-Waterman validation of seeds (kernels K5-K8).
//
// Reference: performSmithWatermanOnRange2 (/root/reference/src/SmithWaterman.h:184-233) builds the window,
// calls StripedSmithWaterman::Aligner::Align (/root/reference/src/ssw_cpp.cpp:234-283) which runs SSW's
// striped forward pass, reverse pass and banded traceback (/root/reference/src/ssw.c:841-951, :143-592,
// :594-792), then un-flips coordinates for reverse-complement seeds.
//
// Here (DESIGN.md §3.4):
//  * k_sw_band<MODE, WP, PARTS> (sw_band.cuh): one THREAD (or 2-4 neighbouring lanes) owns two alignments packed in the
//    halves of s16x2 registers and sweeps a band of one of twelve tiers of 8-128 diagonals that provably contains every
//    optimal alignment (the bound comes from diag_lower_bound, from a first 32-wide sweep, or — reverse pass — from the
//    forward score). Most alignments.
//  * k_sw_fast<LANES, REVERSE>: a group of LANES threads owns two alignments; each lane keeps SW_R=20 query rows (H, E and a
//    4-byte score profile per row) in registers and the group sweeps the columns as an anti-diagonal wavefront (lane g works
//    on column t-g at step t, boundary H/F handed down with shuffles). The full matrix, for what no band can hold.
//    Both kernels: one PRMT builds the packed substitution score from the two profiles, the recurrences are DPX
//    VIADDMNMX/VIMNMX3 ops on BIASED cells (H - gapOpen is then a plain 32-bit add issued as an IMAD on the FMA pipe: six
//    ALU-pipe ops per cell pair). Scores are scaled by 32 so the free low 5 bits of a tracking key carry (31 - row-in-lane)
//    or (31 - band slot): one viaddmax per cell tracks "max score, then smallest row / column", which together with the
//    step / row counter reproduces SSW's tie rules exactly (first column, then smallest row). REVERSE runs the same sweep
//    over the reversed prefixes and records the first column reaching the forward score (ssw.c:905-923). No tensor cores:
//    nothing here is a dense contraction.
//  * k_sw_striped: SSW's striped byte / word kernels restated lane for lane (16 threads per alignment), for every
//    alignment the packed kernels cannot take: parameters outside the plain-Gotoh domain or the packed cells' range,
//    reads or windows over 640 bases, scores the 16-bit cells cannot hold.
//  * k_sw_traceback: pass 0 emits "len M" when the sub-rectangle's main diagonal already scores the alignment score
//    (word-parallel XOR + popcount); the rest runs a literal restatement of banded_sw (ssw.c:594-792) — rolling h_b/e_b/h_c
//    arrays with the reference's index maps (set_u/set_d), direction bytes, band doubling, traceback quirks — one thread
//    per alignment; then the reverse-complement un-flip and refStart offset (SmithWaterman.h:212-229) and the compaction
//    of the CIGAR pool.
// Roofline: integer (ALU) pipe; cells/s reported as GCUPS next to the counted ops/cell.
#include "common.cuh"

#define SW_R 20
#define SW_MAXCOLS 640
#define SW_BLOCK 128
#define SW_INVALID 0xFFFFFFFFu
#define SW_TB_MAXBAND 7
#define SW_TB_MAXROWS 160

struct __align__(16) SwTask {
  uint64_t q_word;   // first 32-base word of the query in the query planes
  uint64_t w_word;   // first word of the sequence holding the window
  uint32_t m;        // query length
  uint32_t n;        // window length (== ref_len passed to Align)
  uint32_t w_start;  // window start (bases) inside its sequence
  uint32_t flags;    // bit0: window is reverse-complemented; bits 8-15: class
};
#define SWT_REV 1u
#define SWT_BAND 2u   // shape allows the banded kernel (rows <= 160)
#define SWT_CLEAN 4u  // no code-4 base in the window (SWT_BAND without it: the masked variants of the band tiers)
#define SWC_FAST8 0u    // full-matrix kernel classes: 8 / 16 / 32 lanes x SW_R rows = reads up to 160 / 320 / 640 bases
#define SWC_FAST16 1u
#define SWC_FAST32 2u
#define SWC_SLOW 3u
#define SWC_NONE 4u   // empty query or window: score 0, nothing to run

struct __align__(16) SwRes {
  int32_t score, ref_end, read_end, ref_begin, read_begin;
  uint32_t flags, pad0, pad1;   // flags: low byte = KSLAM_FLAG_*, bits 8-11 forward tier code, bits 12-15 reverse tier code
};
// Work-list tier of an alignment (byte arrays tier_f / tier_r): a band of tier_width(t) diagonals placed exactly on the
// interval a known score bound allows (no verification needed):
//   t         0   1   2   3   4     5     6     7     8     9     10    11
//   diagonals 8   16  24  32  40    48    56    64    72    80    96    128
//   lanes     1   1   1   1   2x20  2x24  2x28  2x32  3x24  4x20  3x32  4x32      (k_sw_band<MODE, slots per lane, lanes>)
// 12 = 32 diagonals centred, sweep-and-verify; 255 = not in a band list. A forward tier byte with SWT_SWEPT set: the
// alignment went through the 32-wide trial sweep first and then into that tier with the score the sweep found as its bound.
// Tier code in SwRes.flags: tier + 1, 0 = full-matrix / striped kernel.
// A tier byte with SWT_NCOL set: the window has code-4 columns (score 0 against every row, ssw_cpp.cpp:43-48), which a
// PRMT column selector cannot express; such alignments run the NCOL instances of the kernel (a second PRMT per cell masks
// the score), which exist for the tiers of 16, 32, 64 and 128 diagonals and the trial sweep, and have lists of their own
// (list index = tier, + SWT_N_TIERS for NCOL).
#define SWT_N_DIRECT 12u
#define SWT_TIER_SWEEP 12u
#define SWT_N_TIERS 13u
#define SWT_N_LISTS 26u
#define SWT_NCOL 0x20u
#define SWT_SWEPT 0x40u
#define SWT_TIER_NONE 255u
__host__ __device__ __forceinline__ uint32_t tier_list(uint32_t t) { return (t & SWT_NCOL) ? SWT_N_TIERS + (t & 0x1fu) : (t & 0x1fu); }   // t != SWT_TIER_NONE
__host__ __device__ __forceinline__ uint32_t ncol_tier(uint32_t t) { return t <= 1 ? 1u : t <= 3 ? 3u : t <= 7 ? 7u : 11u; }             // direct tier -> the NCOL tier that holds it
#define SWR_FWD_TIER(code) ((uint32_t)(code) << 8)
#define SWR_REV_TIER(code) ((uint32_t)(code) << 12)
__host__ __device__ __forceinline__ constexpr uint32_t tier_width(uint32_t t) { return t < 8 ? 8u * (t + 1) : t == 8 ? 72u : t == 9 ? 80u : t == 10 ? 96u : 128u; }
__host__ __device__ __forceinline__ constexpr uint32_t tier_of_band_width(uint32_t w) { return w <= 64 ? (w + 7) / 8 - 1 : w <= 72 ? 8u : w <= 80 ? 9u : w <= 96 ? 10u : 11u; }
#define SWR_TIER_OF_W(W) (tier_of_band_width(W) + 1u)

struct SwPlanes {
  const uint64_t *q_sbits; const uint32_t *q_nmask;
  const uint64_t *w_sbits; const uint32_t *w_nmask; const uint32_t *w_xmask;
};

struct SwScore {
  int32_t match, mismatch, gap_open, gap_extend;   // positive magnitudes, as given
  uint32_t score_threshold; uint32_t report_cigar; uint32_t cigar_cap;
  uint32_t literal;   // 1: scoring parameters outside the plain-Gotoh domain -> every alignment runs k_sw_striped
};

struct SwWorkspace {
  DevBuf tasks, res, keys, keys2, items, lists, tb_scratch, tier;
  uint64_t n = 0;
};

// ---------------------------------------------------------------- sequence accessors
__device__ __forceinline__ uint32_t q_code(const SwPlanes &p, const SwTask &t, uint32_t i) {
  uint64_t w = t.q_word + (i >> 5); uint32_t b = i & 31;
  if ((__ldg(&p.q_nmask[w]) >> b) & 1) return 4;
  return (uint32_t)(__ldg(&p.q_sbits[w]) >> (2 * b)) & 3;
}
// window base x (0..n-1) in the orientation Align sees (SmithWaterman.h:206-208): reversed + complemented
// when the seed is reverse-complement; only upper-case ACGT are complemented (sequenceTools.h:98-116)
__device__ __forceinline__ uint32_t w_code(const SwPlanes &p, const SwTask &t, uint32_t x) {
  uint32_t pos = (t.flags & SWT_REV) ? t.w_start + t.n - 1 - x : t.w_start + x;
  uint64_t w = t.w_word + (pos >> 5); uint32_t b = pos & 31;
  if ((__ldg(&p.w_nmask[w]) >> b) & 1) return 4;
  uint32_t c = (uint32_t)(__ldg(&p.w_sbits[w]) >> (2 * b)) & 3;
  if ((t.flags & SWT_REV) && !((__ldg(&p.w_xmask[w]) >> b) & 1)) c = 3 - c;
  return c;
}

__device__ __forceinline__ uint32_t pack2(int v) { return ((uint32_t)v & 0xffffu) * 0x10001u; }

// prmt.b32 in its generic form: selector nibble bit 3 replicates the sign of the chosen byte over the target
// byte (the __byte_perm intrinsic masks that bit away, so the PTX instruction is used directly)
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}

// bias added to every stored cell / gap value of the packed sweeps (see k_sw_band): a multiple of 32 larger than
// (gapOpen + gapExtend) * 32, so that H - gapOpen and the gap recurrences stay positive in both 16-bit halves
__host__ __device__ __forceinline__ uint32_t sw_bias(const SwScore &sc) { return 32u * (uint32_t)(sc.gap_open + sc.gap_extend + 2); }
// a * one + c with `one` == 1 passed as a kernel argument: ptxas cannot fold the multiply away, so this is an IMAD and
// issues on the FMA pipe, not on the ALU pipe that the DPX recurrences saturate
__device__ __forceinline__ uint32_t mad_add(uint32_t a, uint32_t one, uint32_t c) {
  uint32_t d;
  asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(one), "r"(c));
  return d;
}

// smallest tier whose band holds an interval of `width` diagonals; SWT_TIER_NONE when nothing allowed does (the widest
// tier is 128 diagonals). level: 1 = 32 only, 2 = 32 and 64, 3 = every width.
__host__ __device__ __forceinline__ uint32_t tier_of_interval(int32_t width, uint32_t level) {
  if (width > 128) return SWT_TIER_NONE;
  if (level >= 3) return tier_of_band_width((uint32_t)(width > 0 ? width : 1));
  if (width <= 32) return 3u;
  return (level >= 2 && width <= 64) ? 7u : SWT_TIER_NONE;
}

// counters (u32) in c->counters + 32
#define CNT_FULL 1
#define CNT_SLOW 2
#define CNT_RETRY 4
#define CNT_EXTRA 5
#define CNT_OVERFLOW 7   // alignments whose CIGAR has more ops than the pool stride (KSLAM_FLAG_CIGAR_OVERFLOW)
#define CNT_NEXT 8       // failures of the sweep tier that go on to a direct tier (second round)
#define CNT_TIER 16      // SWT_N_LISTS counters: alignments per work list
#define CNT_CUR 42       // SWT_N_LISTS cursors of k_tier_scatter
#define CNT_TIER2 68     // 2 * SWT_N_DIRECT counters: second-round alignments per direct tier (clean, NCOL)
#define CNT_WORDS 92

#include "sw_band.cuh"

// ---------------------------------------------------------------- fast (full-matrix) kernel
template <int LANES, bool REVERSE>
__global__ void __launch_bounds__(SW_BLOCK, 4)
k_sw_fast(const SwTask *__restrict__ tasks, const uint2 *__restrict__ items, uint32_t n_items, SwPlanes pl,
          SwScore sc, SwRes *__restrict__ res, uint32_t one /* == 1, opaque to ptxas */) {
  constexpr int GROUPS = SW_BLOCK / LANES;
  __shared__ uint32_t s_sel[GROUPS][SW_MAXCOLS];
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t g = lane % LANES;
  const uint32_t grp = threadIdx.x / LANES;
  const uint32_t gmask = LANES == 32 ? 0xffffffffu : (((1u << LANES) - 1u) << (lane - g));
  const uint32_t item = blockIdx.x * GROUPS + grp;
  uint2 it = make_uint2(SW_INVALID, SW_INVALID);
  if (item < n_items) it = items[item];
  if (it.x == SW_INVALID) return;            // whole group leaves together (shuffles below use gmask only)
  const SwTask ta = tasks[it.x], tb = tasks[it.y];
  if (((ta.flags >> 8) & 0xffu) != (LANES == 8 ? SWC_FAST8 : LANES == 16 ? SWC_FAST16 : SWC_FAST32)) return;   // another instance's item
  SwRes ra, rb;
  uint32_t ncols, rowsA, rowsB;
  if (REVERSE) {
    ra = res[it.x]; rb = res[it.y];
    ncols = (uint32_t)ra.ref_end + 1; rowsA = (uint32_t)ra.read_end + 1; rowsB = (uint32_t)rb.read_end + 1;
  } else { ncols = ta.n; rowsA = ta.m; rowsB = tb.m; }

  // column selectors: PRMT nibbles picking byte w of profile A (-> low half, sign-extended) and byte w of
  // profile B (-> high half); flag bits 16/17 mark code-4 columns (score 0 against everything)
  for (uint32_t j = g; j < ncols; j += LANES) {
    uint32_t xa = REVERSE ? (uint32_t)ra.ref_end - j : j, xb = REVERSE ? (uint32_t)rb.ref_end - j : j;
    uint32_t wa = w_code(pl, ta, xa), wb = w_code(pl, tb, xb);
    uint32_t fl = (wa == 4 ? 0x10000u : 0u) | (wb == 4 ? 0x20000u : 0u);
    wa &= 3; wb &= 3;
    s_sel[grp][j] = wa | ((8u | wa) << 4) | ((4u + wb) << 8) | ((12u + wb) << 12) | fl;
  }
  // row profiles: bytes [s(q,A) s(q,C) s(q,G) s(q,T)] scaled by 32; code-4 query rows score 0; padding rows
  // (beyond the query) mismatch everything so they can never create or extend a maximum
  const uint32_t mis_b = (uint32_t)(-(sc.mismatch * 32)) & 0xffu, mat_b = (uint32_t)(sc.match * 32) & 0xffu;
  uint32_t PA[SW_R], PB[SW_R];
#pragma unroll
  for (int r = 0; r < SW_R; r++) {
    uint32_t i = g * SW_R + r;
    uint32_t pa = mis_b * 0x01010101u, pb = pa;
    if (i < rowsA) { uint32_t c = q_code(pl, ta, REVERSE ? rowsA - 1 - i : i);
                     pa = c == 4 ? 0u : (pa ^ ((mis_b ^ mat_b) << (8 * c))); }
    if (i < rowsB) { uint32_t c = q_code(pl, tb, REVERSE ? rowsB - 1 - i : i);
                     pb = c == 4 ? 0u : (pb ^ ((mis_b ^ mat_b) << (8 * c))); }
    PA[r] = pa; PB[r] = pb;
  }
  __syncwarp(gmask);

  // biased cells, H - gapOpen as one IMAD on the FMA pipe: see k_sw_band
  const uint32_t NEG_GE = pack2(-sc.gap_extend * 32);
  const uint32_t KB = sw_bias(sc), K2 = KB * 0x10001u;
  const uint32_t NEG_GO32 = (uint32_t)(-(int32_t)(sc.gap_open * 32) * 0x10001);
  uint32_t H[SW_R], E[SW_R];
#pragma unroll
  for (int r = 0; r < SW_R; r++) { H[r] = K2; E[r] = K2; }
  uint32_t lastH = K2, lastF = K2, prevUpH = K2;
  // forward: best = (H*32 | 31) of the running maximum, info = step << 16 | key at the step it was set
  // reverse: thr = forward score * 32, info = first step whose lane maximum reaches it
  uint32_t bestA = KB + 31u, bestB = KB + 31u, infoA = 0, infoB = 0;
  const uint32_t thrA = REVERSE ? (uint32_t)ra.score * 32u + KB : 0u, thrB = REVERSE ? (uint32_t)rb.score * 32u + KB : 0u;
  bool hitA = false, hitB = false;

  const uint32_t steps = ncols + LANES - 1;
  for (uint32_t t = 0; t < steps; t++) {
    uint32_t upH = __shfl_up_sync(gmask, lastH, 1, LANES);
    uint32_t upF = __shfl_up_sync(gmask, lastF, 1, LANES);
    if (g == 0) { upH = K2; upF = K2; }
    const int32_t j = (int32_t)t - (int32_t)g;
    if (j >= 0 && j < (int32_t)ncols) {
      const uint32_t selw = s_sel[grp][j];
      const uint32_t sel = selw & 0xffffu;
      uint32_t hd = prevUpH, f = upF, acc = 0;
      if (selw >> 16) {
        // a code-4 (N) column in one or both alignments: substitution score 0 there (ssw_cpp.cpp:43-48)
        const uint32_t cm = ((selw & 0x10000u) ? 0u : 0xffffu) | ((selw & 0x20000u) ? 0u : 0xffff0000u);
#pragma unroll
        for (int r = 0; r < SW_R; r++) {
          uint32_t s = prmt(PA[r], PB[r], sel) & cm;
          uint32_t h = __viaddmax_s16x2(hd, s, E[r]);
          h = __vimax3_s16x2(h, f, K2);
          hd = H[r]; H[r] = h;
          uint32_t hgo = mad_add(h, one, NEG_GO32);
          E[r] = __viaddmax_s16x2(E[r], NEG_GE, hgo);
          f = __viaddmax_s16x2(f, NEG_GE, hgo);
          acc = __viaddmax_s16x2(h, (uint32_t)(31 - r) * 0x10001u, acc);
        }
      } else {
#pragma unroll
        for (int r = 0; r < SW_R; r++) {
          uint32_t s = prmt(PA[r], PB[r], sel);
          uint32_t h = __viaddmax_s16x2(hd, s, E[r]);            // max(H[i-1][j-1] + s, E)
          h = __vimax3_s16x2(h, f, K2);                           // ... F and the floor (0, biased)
          hd = H[r]; H[r] = h;
          uint32_t hgo = mad_add(h, one, NEG_GO32);               // H - gapOpen, both halves, FMA pipe
          E[r] = __viaddmax_s16x2(E[r], NEG_GE, hgo);             // E for column j+1
          f = __viaddmax_s16x2(f, NEG_GE, hgo);                   // F for row i+1
          acc = __viaddmax_s16x2(h, (uint32_t)(31 - r) * 0x10001u, acc);  // max of H*32 + (31 - r)
        }
      }
      lastH = H[SW_R - 1]; lastF = f; prevUpH = upH;
      const uint32_t aA = acc & 0xffffu, aB = acc >> 16;
      if (REVERSE) {
        if (!hitA && aA >= thrA) { hitA = true; infoA = (t << 16) | aA; }
        if (!hitB && aB >= thrB) { hitB = true; infoB = (t << 16) | aB; }
      } else {
        if (aA > bestA) { bestA = aA | 31u; infoA = (t << 16) | aA; }
        if (aB > bestB) { bestB = aB | 31u; infoB = (t << 16) | aB; }
      }
    }
  }

  // group reduction. forward: max score, then smallest column, then smallest row. reverse: first column
  // (smallest scan index) that reached the score, then smallest row.
  uint32_t keyA, keyB;
  {
    uint32_t colA = (infoA >> 16) - g, rowA = g * SW_R + (31u - (infoA & 31u));
    uint32_t colB = (infoB >> 16) - g, rowB = g * SW_R + (31u - (infoB & 31u));
    if (REVERSE) {
      keyA = hitA ? (((1023u - colA) << 10) | (1023u - rowA)) : 0u;
      keyB = hitB ? (((1023u - colB) << 10) | (1023u - rowB)) : 0u;
    } else {
      keyA = bestA > KB + 31u ? ((((bestA - KB) >> 5) << 20) | ((1023u - colA) << 10) | (1023u - rowA)) : 0u;
      keyB = bestB > KB + 31u ? ((((bestB - KB) >> 5) << 20) | ((1023u - colB) << 10) | (1023u - rowB)) : 0u;
    }
  }
#pragma unroll
  for (int d = 1; d < LANES; d <<= 1) {
    uint32_t oa = __shfl_xor_sync(gmask, keyA, d, LANES), ob = __shfl_xor_sync(gmask, keyB, d, LANES);
    keyA = keyA > oa ? keyA : oa; keyB = keyB > ob ? keyB : ob;
  }
  if (g == 0) {
#pragma unroll
    for (int half = 0; half < 2; half++) {
      if (half == 1 && it.y == it.x) break;
      const uint32_t key = half ? keyB : keyA;
      const uint32_t idx = half ? it.y : it.x;
      const uint32_t col = 1023u - ((key >> 10) & 1023u), row = 1023u - (key & 1023u);
      if (REVERSE) {
        const SwRes &r0 = half ? rb : ra;
        if (key) { res[idx].ref_begin = r0.ref_end - (int32_t)col; res[idx].read_begin = r0.read_end - (int32_t)row; }
        else { res[idx].ref_begin = 0; res[idx].read_begin = 0; res[idx].flags = r0.flags | KSLAM_FLAG_UNDEFINED; }
      } else {
        SwRes o;
        o.flags = 0; o.pad0 = o.pad1 = 0; o.ref_begin = -1; o.read_begin = 0;
        if (key) { o.score = (int32_t)(key >> 20); o.ref_end = (int32_t)col; o.read_end = (int32_t)row; }
        else { o.score = 0; o.ref_end = -1; o.read_end = 0; }        // ssw.c:169 (no positive cell)
        res[idx] = o;
      }
    }
  }
}

// ---------------------------------------------------------------- literal striped SSW (any scoring parameters)
// SSW's striped kernels equal plain Gotoh only when gap_extend < gap_open and mismatch <= 2 * gap_extend (DESIGN.md
// §3.4). Outside that domain the result depends on details of the striping itself: E is updated from the H value BEFORE
// the lazy-F correction (ssw.c:257-264), the byte kernel's lazy-F loop runs until no lane's F exceeds H - gapO and
// raises the column maximum as it goes (ssw.c:289-305), the word kernel's runs at most 8 rounds, leaves at the first
// vector where no lane's F exceeds H - gapO and does NOT raise the column maximum (ssw.c:514-524). k_sw_striped
// restates both kernels lane for lane — a group of 16 threads IS the 16 byte lanes (8 of them the word lanes), vector j
// of lane l holds query row j + l * segLen (ssw.c:105-133,385-406), _mm_slli_si128 is a shuffle-up inside the group,
// movemask tests are ballots — and then ssw_align's control flow: byte pass, word pass on overflow (ssw.c:868-877),
// reverse pass over the reversed prefixes with the forward score as `terminate` (ssw.c:905-923). Inside the domain this
// is plain Gotoh up to the word pass's saturation at 32767, which it keeps as the reference does. Speed is secondary
// here (it runs only for what the packed kernels cannot take: non-default --match-score / --mismatch-penalty / --gap-*
// combinations, reads or windows over 640 bases); exactness is not.
#define STR_GROUPS 8          // 16-lane groups per CTA
#define STR_SMEM_SEGS 24      // state of reads up to 192 bases (word mode) lives in shared memory, longer ones in global scratch

struct StripedEnd { int32_t score, ref, read; };

__device__ __forceinline__ int32_t group_max16(uint32_t gmask, int32_t v) {
#pragma unroll
  for (int d = 8; d; d >>= 1) { const int32_t o = __shfl_xor_sync(gmask, v, d, 16); v = v > o ? v : o; }
  return v;
}
__device__ __forceinline__ int32_t shift_lane(uint32_t gmask, uint32_t l, int32_t v) {   // _mm_slli_si128 by one lane
  const int32_t o = __shfl_up_sync(gmask, v, 1, 16);
  return l == 0 ? 0 : o;
}

// one sw_sse2_byte / sw_sse2_word call. st: 5 arrays of seg_cap * 16 shorts (Hstore, Hload, E, Hmax, row codes).
__device__ StripedEnd striped_pass(const SwPlanes &pl, const SwTask &t, int32_t m8, int32_t x8, int32_t go, int32_t ge, int32_t bias,
                                   bool reverse, int32_t refLen, int32_t readLen, int32_t ref_end, int32_t read_end,
                                   int32_t terminate, bool word, int16_t *st, uint32_t seg_cap, uint32_t l, uint32_t gmask) {
  const int32_t L = word ? 8 : 16;
  const int32_t segLen = (readLen + L - 1) / L;
  const bool act = (int32_t)l < L;
  int16_t *Hs = st + l, *Hl = Hs + seg_cap * 16, *E = Hl + seg_cap * 16, *Hm = E + seg_cap * 16, *QC = Hm + seg_cap * 16;   // values fit 16 bits
  for (int32_t j = 0; j < segLen; j++) {
    const int32_t row = j + (int32_t)l * segLen;
    Hs[j * 16] = 0; Hl[j * 16] = 0; E[j * 16] = 0; Hm[j * 16] = 0;
    QC[j * 16] = (act && row < readLen) ? (int16_t)q_code(pl, t, (uint32_t)(reverse ? read_end - row : row)) : 5;   // 5 = padding row
  }
  int32_t max = 0, end_read = readLen - 1, end_ref = word ? 0 : -1;
  int32_t vMaxScore = 0, vMaxMark = 0;
  bool overflow = false;
  for (int32_t step = 0; step < refLen; step++) {
    const int32_t i = reverse ? refLen - 1 - step : step;
    const int32_t c = (int32_t)w_code(pl, t, (uint32_t)i);
    int32_t vF = 0, vMaxColumn = 0;
    int32_t vH = shift_lane(gmask, l, Hs[(segLen - 1) * 16]);
    { int16_t *tmp = Hl; Hl = Hs; Hs = tmp; }
    for (int32_t j = 0; j < segLen; j++) {
      const int32_t qc = QC[j * 16];
      const int32_t sco = (qc == 5 || qc == 4 || c == 4) ? 0 : (qc == c ? m8 : x8);
      int32_t h;
      if (word) { h = vH + sco; h = h > 32767 ? 32767 : h; }                                // _mm_adds_epi16 (never below -32768 here)
      else { h = vH + ((sco + bias) & 0xff); h = h > 255 ? 255 : h; h -= bias; h = h < 0 ? 0 : h; }   // _mm_adds_epu8, _mm_subs_epu8
      int32_t e = E[j * 16];
      h = h > e ? h : e; h = h > vF ? h : vF;
      if (!act) h = 0;
      vMaxColumn = vMaxColumn > h ? vMaxColumn : h;
      Hs[j * 16] = (int16_t)h;
      h -= go; h = h < 0 ? 0 : h;
      e -= ge; e = e < 0 ? 0 : e; e = e > h ? e : h;
      E[j * 16] = (int16_t)(act ? e : 0);
      vF -= ge; vF = vF < 0 ? 0 : vF; vF = vF > h ? vF : h;
      if (!act) vF = 0;
      vH = Hl[j * 16];
    }
    if (!word) {                                                                             // ssw.c:276-305
      int32_t j = 0;
      vF = shift_lane(gmask, l, vF);
      for (;;) {
        int32_t h = Hs[j * 16];
        int32_t tt = h - go; tt = tt < 0 ? 0 : tt;
        if (!(__ballot_sync(gmask, act && vF > tt) & gmask)) break;
        h = h > vF ? h : vF;
        vMaxColumn = vMaxColumn > h ? vMaxColumn : h;
        Hs[j * 16] = (int16_t)h;
        vF -= ge; vF = vF < 0 ? 0 : vF;
        if (++j >= segLen) { j = 0; vF = shift_lane(gmask, l, vF); }
      }
    } else {                                                                                 // ssw.c:512-524
      bool done = false;
      for (int k = 0; k < 8 && !done; k++) {
        vF = shift_lane(gmask, l, vF);
        if (!act) vF = 0;
        for (int32_t j = 0; j < segLen; j++) {
          int32_t h = Hs[j * 16];
          h = h > vF ? h : vF;
          Hs[j * 16] = (int16_t)h;
          h -= go; h = h < 0 ? 0 : h;
          vF -= ge; vF = vF < 0 ? 0 : vF;
          if (!(__ballot_sync(gmask, act && vF > h) & gmask)) { done = true; break; }
        }
      }
    }
    vMaxScore = vMaxScore > vMaxColumn ? vMaxScore : vMaxColumn;
    if (__ballot_sync(gmask, vMaxMark != vMaxScore) & gmask) {                              // ssw.c:307-327
      vMaxMark = vMaxScore;
      const int32_t temp = group_max16(gmask, vMaxScore);
      if (temp > max) {
        max = temp;
        if (!word && max + bias >= 255) { overflow = true; break; }
        end_ref = i;
        for (int32_t j = 0; j < segLen; j++) Hm[j * 16] = Hs[j * 16];
      }
    }
    if (group_max16(gmask, vMaxColumn) == terminate) break;
  }
  int32_t mine = end_read;                                                                   // ssw.c:334-342: smallest row holding max
  if (act)
    for (int32_t j = 0; j < segLen; j++)
      if (Hm[j * 16] == max) { const int32_t row = j + (int32_t)l * segLen; mine = row < mine ? row : mine; }
  end_read = -group_max16(gmask, -mine);
  StripedEnd r;
  r.score = overflow ? 255 : max; r.ref = end_ref; r.read = end_read;
  return r;
}

__global__ void __launch_bounds__(STR_GROUPS * 16)
k_sw_striped(const SwTask *__restrict__ tasks, const uint32_t *__restrict__ list, uint32_t n_list, SwPlanes pl, SwScore sc,
             SwRes *__restrict__ res, int16_t *__restrict__ scratch, uint32_t seg_cap) {
  __shared__ int16_t s_state[STR_GROUPS][5 * STR_SMEM_SEGS * 16];
  const uint32_t l = threadIdx.x & 15, grp = threadIdx.x >> 4;
  const uint32_t gmask = 0xffffu << (threadIdx.x & 16);
  const uint32_t slot = blockIdx.x * STR_GROUPS + grp, n_slots = gridDim.x * STR_GROUPS;
  int16_t *st = seg_cap <= STR_SMEM_SEGS ? s_state[grp] : scratch + (size_t)slot * 5 * seg_cap * 16;
  // the int8_t score matrix of BuildSwScoreMatrix (ssw_cpp.cpp:25-49) and ssw_init's bias (ssw.c:817-822)
  const int32_t m8 = sc.match, x8 = -sc.mismatch;
  int32_t bias = m8 < x8 ? m8 : x8; bias = bias < 0 ? -bias : 0;
  for (uint32_t k = slot; k < n_list; k += n_slots) {
    const uint32_t idx = list[k];
    const SwTask t = tasks[idx];
    const int32_t m = (int32_t)t.m, n = (int32_t)t.n;
    bool word = false;
    StripedEnd fw = striped_pass(pl, t, m8, x8, sc.gap_open, sc.gap_extend, bias, false, n, m, 0, 0, 255, false, st, seg_cap, l, gmask);
    if (fw.score == 255) { fw = striped_pass(pl, t, m8, x8, sc.gap_open, sc.gap_extend, bias, false, n, m, 0, 0, 65535, true, st, seg_cap, l, gmask); word = true; }
    SwRes o; o.flags = 0; o.pad0 = o.pad1 = 0;
    o.score = fw.score; o.ref_end = fw.ref; o.read_end = fw.read; o.ref_begin = -1; o.read_begin = 0;
    if (fw.score > 0) {
      const StripedEnd rv = striped_pass(pl, t, m8, x8, sc.gap_open, sc.gap_extend, bias, true, fw.ref + 1, fw.read + 1, fw.ref, fw.read,
                                         word ? fw.score : (fw.score & 0xff), word, st, seg_cap, l, gmask);
      o.ref_begin = rv.ref; o.read_begin = fw.read - rv.read;
    } else { o.ref_end = -1; o.read_end = 0; }
    if (l == 0) res[idx] = o;
  }
}

// ---------------------------------------------------------------- banded traceback (ssw.c:594-792)
#define SET_U(u, w, i, j) { int x_ = (i) - (w); x_ = x_ > 0 ? x_ : 0; (u) = (j) - x_ + 1; }

// Returns cigar length (>= 1), -1 = undefined in the reference, -2 = "no cigar" (ssw.c:631-642),
// -3 = scratch too small for the band this alignment needs (caller retries with the big-scratch path).
// dir holds one byte per band cell: bit0 = (E came from H, code 3), bit1 = (F came from H, code 5),
// bits 2-4 = the H direction code 1..5 exactly as banded_sw would store it.
// rowdir (bands up to SW_TB_MAXBAND, i.e. at most 15 cells per row): the same as ONE 64-bit word per row, 4 bits per
// cell — bit0, bit1 as above, bits 2-3 = where H came from (0 diagonal, 1 E, 2 F; the code 2/3 or 4/5 banded_sw stores is
// the cell's own E / F code). The threads of a warp walk the rows together, so the row words of a warp's 32 alignments
// are one coalesced local-memory store per row; the byte-per-cell form scattered 32 single bytes per cell (1.15 GB of
// DRAM traffic for 400 k alignments, profiles/r1_ncu_summaries.txt).
__device__ int32_t banded_traceback(const SwPlanes &pl, const SwTask &t, const SwScore &sc, int32_t ref0,
                                    int32_t read0, int32_t refLen, int32_t readLen, int32_t score, int32_t *h_b,
                                    int32_t *e_b, int32_t *h_c, uint32_t hs /* stride of the three rolling arrays */, uint32_t arr_cap, uint8_t *dir, size_t dir_cap,
                                    size_t dstride, uint64_t *rowdir, uint32_t *cig, uint32_t cig_cap, bool reverse_out,
                                    uint32_t *overflow) {
  const int32_t go = sc.gap_open, ge = sc.gap_extend;
  int32_t band = (refLen > readLen ? refLen - readLen : readLen - refLen) + 1;
  int32_t width = 0, width_d = 0, maxv = 0, ws = 0;
  do {
    width = band * 2 + 3; width_d = band * 2 + 1;
    if ((int64_t)width_d * readLen * 3 >= (1ll << 30)) return -2;
    // A band wider than the reference sequence touches only slots 0..refLen of the rolling arrays and refLen direction
    // cells per row (j stays inside [0, refLen)), so the scratch is sized by what is touched, not by the nominal width:
    // the band may double up to the "no cigar" limit above without leaving the scratch.
    const int32_t aw = width < refLen + 2 ? width : refLen + 2;
    ws = width_d < refLen ? width_d : refLen;
    if ((uint32_t)aw > arr_cap || (rowdir ? (ws > 2 * SW_TB_MAXBAND + 1 || readLen > SW_TB_MAXROWS) : (size_t)ws * (size_t)readLen > dir_cap)) return -3;
    for (int32_t j = 1; j < aw - 1; j++) h_b[(j) * hs] = 0;
    // Window codes of the band cells of a row, one nibble per cell (bands up to 7: 15 cells): nibble k of `wwin` holds the
    // code of column i - band + k. A row needs ONE new code (column i + band); the plane loads of w_code were per cell.
    const bool windowed = band <= SW_TB_MAXBAND;
    uint64_t wwin = 0;
    if (windowed)
      for (int32_t k = band; k <= 2 * band; k++)
        if (k - band < refLen) wwin |= (uint64_t)w_code(pl, t, (uint32_t)(ref0 + k - band)) << (4 * k);
    for (int32_t i = 0; i < readLen; i++) {
      const int32_t beg = i - band > 0 ? i - band : 0, end = i + band < refLen - 1 ? i + band : refLen - 1;
      const int32_t edge = end + 1 < width - 1 ? end + 1 : width - 1;
      int32_t u = 0, f = 0;
      h_b[(0) * hs] = 0; e_b[(0) * hs] = 0; h_b[(edge) * hs] = 0; e_b[(edge) * hs] = 0; h_c[(0) * hs] = 0;
      const uint32_t qc = q_code(pl, t, (uint32_t)(read0 + i));
      uint8_t *dl = rowdir ? nullptr : dir + (size_t)ws * i * dstride;
      uint64_t rowbits = 0;
      // set_u (ssw.c:56-61): u = j - max(i - band, 0) + 1 for row i; the row above is shifted by `up` = 0 or 1 slots
      const int32_t xoff = beg, up = xoff - (i - 1 - band > 0 ? i - 1 - band : 0);
      for (int32_t j = beg; j <= end; j++) {
        u = j - xoff + 1;
        const int32_t e = u + up, b = u - 1, d = e - 1;
        int32_t t1 = i == 0 ? -go : h_b[(e) * hs] - go;
        int32_t t2 = i == 0 ? -ge : e_b[(e) * hs] - ge;
        const int32_t ev = t1 > t2 ? t1 : t2;
        const uint32_t de = t1 > t2 ? 3u : 2u;
        e_b[(u) * hs] = ev;
        t1 = h_c[(b) * hs] - go; t2 = f - ge;
        f = t1 > t2 ? t1 : t2;
        const uint32_t df = t1 > t2 ? 5u : 4u;
        const int32_t e1 = ev > 0 ? ev : 0, f1 = f > 0 ? f : 0;
        t1 = e1 > f1 ? e1 : f1;
        const uint32_t wc = windowed ? (uint32_t)(wwin >> (4 * (j - i + band))) & 7u : w_code(pl, t, (uint32_t)(ref0 + j));
        const int32_t s = (wc == 4 || qc == 4) ? 0 : (wc == qc ? sc.match : -sc.mismatch);
        t2 = h_b[(d) * hs] + s;
        const int32_t hv = t1 > t2 ? t1 : t2;
        h_c[(u) * hs] = hv;
        if (hv > maxv) maxv = hv;
        const uint32_t dh = t1 <= t2 ? 1u : (e1 > f1 ? de : df);
        if (rowdir) rowbits |= (uint64_t)((de == 3u) | ((df == 5u) << 1) | ((dh == 1u ? 0u : (dh <= 3u ? 1u : 2u)) << 2)) << (4 * (j - xoff));
        else dl[(size_t)(j - xoff) * dstride] = (uint8_t)((de == 3u) | ((df == 5u) << 1) | (dh << 2));
      }
      if (rowdir) rowdir[i] = rowbits;
      for (int32_t j = 1; j <= u; j++) h_b[(j) * hs] = h_c[(j) * hs];
      if (windowed) {
        wwin >>= 4;
        const int32_t col = i + 1 + band;
        if (col < refLen) wwin |= (uint64_t)w_code(pl, t, (uint32_t)(ref0 + col)) << (8 * band);
      }
    }
    band *= 2;
  } while (maxv < score);
  band /= 2;

  // trace back from the bottom-right corner while i > 0 (ssw.c:698-753); ops collected in reverse
  int32_t i = readLen - 1, j = refLen - 1, e = 0, l = 0, f = 0, cur = 0, st = 2;
  // pass 1 counts ops so that pass 2 can place them without a temporary list
  for (int pass = 0; pass < 2; pass++) {
    const int32_t total = l;
    i = readLen - 1; j = refLen - 1; e = 0; l = 0; f = 0; cur = 0; st = 2;
    while (i > 0) {
      const int32_t lo = i - band > 0 ? i - band : 0, hi = i + band < refLen - 1 ? i + band : refLen - 1;
      if (j < lo || j > hi) return -1;
      uint32_t cell;
      if (rowdir) {
        cell = (uint32_t)(rowdir[i] >> (4 * (j - lo))) & 15u;
        const uint32_t from = cell >> 2;                    // -> the byte form: H code 1, the cell's E code or its F code
        cell = (cell & 3u) | ((from == 0u ? 1u : from == 1u ? ((cell & 1u) ? 3u : 2u) : ((cell & 2u) ? 5u : 4u)) << 2);
      } else cell = dir[((size_t)ws * i + (size_t)(j - lo)) * dstride];
      uint32_t code = st == 2 ? (cell >> 2) : (st == 0 ? ((cell & 1u) ? 3u : 2u) : ((cell & 2u) ? 5u : 4u));
      switch (code) {
        case 1: --i; --j; st = 2; f = 0; break;
        case 2: --i; st = 0; f = 1; break;
        case 3: --i; st = 2; f = 1; break;
        case 4: --j; st = 1; f = 2; break;
        case 5: --j; st = 2; f = 2; break;
        default: return -1;
      }
      if (f == cur) ++e;
      else {
        ++l;
        if (pass == 1) {      // op number l-1 in trace order; final cigar is the reverse of the trace order
          const int32_t k = reverse_out ? l - 1 : total - l;
          if (k >= 0 && (uint32_t)k < cig_cap) cig[k] = ((uint32_t)e << 4) | (uint32_t)cur;
        }
        cur = f; e = 1;
      }
    }
    if (f == 0) {
      ++l;
      if (pass == 1) { const int32_t k = reverse_out ? l - 1 : total - l; if (k >= 0 && (uint32_t)k < cig_cap) cig[k] = (uint32_t)(e + 1) << 4; }
    } else {
      l += 2;
      if (pass == 1) {
        int32_t k = reverse_out ? l - 2 : total - (l - 1); if (k >= 0 && (uint32_t)k < cig_cap) cig[k] = ((uint32_t)e << 4) | (uint32_t)f;
        k = reverse_out ? l - 1 : total - l; if (k >= 0 && (uint32_t)k < cig_cap) cig[k] = 16u;
      }
    }
  }
  if ((uint32_t)l > cig_cap) *overflow = 1;
  return l;
}

__device__ __forceinline__ int32_t diagonal_score_slow(const SwPlanes &pl, const SwTask &t, const SwScore &sc, int32_t ref0,
                                                       int32_t read0, int32_t len);
// 2-bit codes of the 32 window columns j = 32 qw + d0 + b (b = 0..31) in the orientation Align sees; windows without
// code-4 bases only (the caller checks SWT_CLEAN)
__device__ __forceinline__ uint64_t window_word_on_diagonal(const SwPlanes &pl, const SwTask &t, int32_t qw, int32_t d0) {
  if (!(t.flags & SWT_REV)) return bits_at(pl.w_sbits, t.w_word, (int32_t)t.w_start + 32 * qw + d0);
  const int32_t p0 = (int32_t)t.w_start + (int32_t)t.n - 1 - 32 * qw - d0 - 31;   // column 32qw + d0 + b <-> base p0 + 31 - b
  return reverse_pairs(bits_at(pl.w_sbits, t.w_word, p0)) ^ pair_mask(~__brev(mask_at(pl.w_xmask, t.w_word, p0)));   // complement unless a/c/g/t/U/u
}

// Score of the gap-free alignment of read'[0..len) against ref'[0..len) (the sub-rectangle's main diagonal).
// Word-parallel when the window has no code-4 base: XOR of the 2-bit planes, population counts.
__device__ __forceinline__ int32_t diagonal_score(const SwPlanes &pl, const SwTask &t, const SwScore &sc, int32_t ref0,
                                                  int32_t read0, int32_t len) {
  if (!(t.flags & SWT_CLEAN)) return diagonal_score_slow(pl, t, sc, ref0, read0, len);
  const int32_t d0 = ref0 - read0, i_lo = read0, i_hi = read0 + len;
  int32_t matches = 0, mism = 0;
  for (int32_t qw = i_lo >> 5; qw <= (i_hi - 1) >> 5; qw++) {
    const uint64_t x = __ldg(&pl.q_sbits[t.q_word + qw]) ^ window_word_on_diagonal(pl, t, qw, d0);
    const uint64_t mm = (x | (x >> 1)) & 0x5555555555555555ull;
    const int32_t b_lo = i_lo - 32 * qw > 0 ? i_lo - 32 * qw : 0, b_hi = i_hi - 32 * qw < 32 ? i_hi - 32 * qw : 32;
    const uint32_t span = (b_hi - b_lo >= 32 ? 0xffffffffu : ((1u << (b_hi - b_lo)) - 1u) << b_lo);
    const uint64_t live = pair_mask(span & ~__ldg(&pl.q_nmask[t.q_word + qw])) & 0x5555555555555555ull;   // code-4 query bases score 0
    mism += __popcll(mm & live); matches += __popcll(~mm & live);
  }
  return sc.match * matches - sc.mismatch * mism;
}

__device__ __forceinline__ int32_t diagonal_score_slow(const SwPlanes &pl, const SwTask &t, const SwScore &sc, int32_t ref0,
                                                  int32_t read0, int32_t len) {
  int32_t d = 0;
  for (int32_t i = 0; i < len; i++) {
    const uint32_t qc = q_code(pl, t, (uint32_t)(read0 + i)), wc = w_code(pl, t, (uint32_t)(ref0 + i));
    d += (wc == 4 || qc == 4) ? 0 : (wc == qc ? sc.match : -sc.mismatch);
  }
  return d;
}

// Finishes every alignment: cigar (if requested and score >= threshold, ssw.c:924-927), un-flip for
// reverse-complement seeds and + refStart (SmithWaterman.h:212-229), and writes the kslam_overlap fields.
//  mode 0 (all alignments, no DP): when the sub-rectangle is square and its main diagonal already scores `score`,
//         banded_sw's first band (width 1) reaches the score, every diagonal cell has direction 1 (a gap path into
//         a diagonal cell scoring more than the diagonal prefix would lift the corner above the global maximum; all
//         prefix sums are positive or the reverse pass would have started later) and the traceback yields exactly
//         `len M` — emitted directly. Everything else is appended to retry_list.
//  mode 1 (retry_list): literal banded_sw with per-thread local arrays (band <= SW_TB_MAXBAND, rows <= SW_TB_MAXROWS);
//         larger cases are appended to the next retry list.
//  mode 2: same with a big global scratch per thread.
__global__ void __launch_bounds__(128)
k_sw_traceback(const SwTask *__restrict__ tasks, const SwRes *__restrict__ res, uint32_t n, const uint32_t *list,
               SwPlanes pl, SwScore sc, kslam_overlap *__restrict__ ov, uint32_t *__restrict__ cigs, int unflip,
               int mode, uint32_t *__restrict__ retry_list, uint32_t *__restrict__ retry_count,
               uint32_t *__restrict__ overflow_count, uint8_t *__restrict__ big, size_t big_per_thread) {
  const uint32_t gtid = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t nthreads = gridDim.x * blockDim.x;
  // the three rolling arrays of banded_sw, touched for every cell: shared memory, [slot][thread] (conflict-free). In local
  // memory they (and the direction words) took 1.5 KB per thread — 3 MB per SM at full occupancy, far beyond L1 — and every
  // cell waited on L2. The direction words stay in local memory: one coalesced store per row, read once by the trace.
  __shared__ int32_t s_roll[3 * (SW_TB_MAXBAND * 2 + 3) * 128];
  int32_t *l_hb = s_roll + threadIdx.x, *l_eb = l_hb + (SW_TB_MAXBAND * 2 + 3) * 128, *l_hc = l_eb + (SW_TB_MAXBAND * 2 + 3) * 128;
  uint64_t l_rowdir[SW_TB_MAXROWS];
  for (uint32_t k = gtid; k < n; k += nthreads) {
    const uint32_t idx = list ? list[k] : k;
    const SwTask t = tasks[idx];
    const SwRes r = res[idx];
    kslam_overlap o = ov[idx];
    o.sw_score = (uint32_t)r.score & 0xffffu;
    o.ref_begin = r.ref_begin; o.ref_end = r.ref_end; o.query_begin = r.read_begin; o.query_end = r.read_end;
    o.cigar_len = 0; o.cigar_off = idx * sc.cigar_cap; o.flags = r.flags & 0xffu;
    const bool rev = (t.flags & SWT_REV) != 0;
    uint32_t *cig = cigs ? cigs + (size_t)idx * sc.cigar_cap : nullptr;
    bool deferred = false;
    if (sc.report_cigar && cig && (uint32_t)r.score >= sc.score_threshold && !(r.flags & KSLAM_FLAG_UNDEFINED)) {
      if (r.score == 0) o.flags |= KSLAM_FLAG_UNDEFINED;      // the reference reads ref[-1] here
      else {
        const int32_t refLen = r.ref_end - r.ref_begin + 1, readLen = r.read_end - r.read_begin + 1;
        uint32_t overflow = 0; int32_t len;
        if (mode == 0) {
          if (!sc.literal && refLen == readLen && sc.cigar_cap >= 1 && diagonal_score(pl, t, sc, r.ref_begin, r.read_begin, readLen) == r.score) {
            cig[0] = (uint32_t)readLen << 4; len = 1;
          } else len = -3;
        } else if (mode == 1)
          len = banded_traceback(pl, t, sc, r.ref_begin, r.read_begin, refLen, readLen, r.score, l_hb, l_eb, l_hc, 128,
                                 SW_TB_MAXBAND * 2 + 3, nullptr, 0, 1, l_rowdir, cig, sc.cigar_cap, rev && unflip, &overflow);
        else {
          uint8_t *base = big + (size_t)gtid * big_per_thread;
          const uint32_t arr_cap = (uint32_t)(big_per_thread / 64);   // ints per rolling array
          int32_t *hb = reinterpret_cast<int32_t *>(base), *eb = hb + arr_cap, *hc = eb + arr_cap;
          uint8_t *d = base + (size_t)arr_cap * 12;
          len = banded_traceback(pl, t, sc, r.ref_begin, r.read_begin, refLen, readLen, r.score, hb, eb, hc, 1, arr_cap, d,
                                 big_per_thread - (size_t)arr_cap * 12, 1, nullptr, cig, sc.cigar_cap, rev && unflip, &overflow);
        }
        if (len == -3) {
          if (mode < 2) { deferred = true; retry_list[list_slot(retry_count)] = idx; }
          else o.flags |= KSLAM_FLAG_UNDEFINED;   // beyond even the big scratch: report, never guess
        } else if (len == -2) { o.cigar_len = 0; o.sw_score = 0; }           // ssw.c:941-944
        else if (len == -1) o.flags |= KSLAM_FLAG_UNDEFINED;
        else {
          o.cigar_len = (uint32_t)len < sc.cigar_cap ? (uint32_t)len : sc.cigar_cap;
          if (overflow) { o.flags |= KSLAM_FLAG_CIGAR_OVERFLOW; atomicAdd(overflow_count, 1u); }
        }
      }
    }
    if (deferred) continue;
    if (unflip) {
      if (rev) {     // SmithWaterman.h:212-227
        const int32_t wl = (int32_t)t.n, ql = (int32_t)t.m;
        int32_t tmp = o.ref_begin; o.ref_begin = wl - (o.ref_end + 1); o.ref_end = wl - (tmp + 1);
        tmp = o.query_begin; o.query_begin = ql - (o.query_end + 1); o.query_end = ql - (tmp + 1);
      }
      o.ref_begin += (int32_t)t.w_start; o.ref_end += (int32_t)t.w_start;   // :228-229
    }
    ov[idx] = o;
  }
}

// ---------------------------------------------------------------- task preparation and work lists

// ---- lower bound of the optimal score from the seed's own diagonal ------------------------------------------
// Best ungapped local segment (Kadane) along matrix diagonal j = i + d0, in the orientation Align sees. It is the score
// of a real local alignment, hence a LOWER BOUND L of the optimum: every alignment scoring >= L lies inside the offsets
// [-(m - a), n - a] with a = ceil(L / match) (sw_band.cuh), which picks the band tier without a trial sweep. Only
// called for windows without code-4 bases; code-4 query bases score 0 (ssw_cpp.cpp:43-48).
__device__ int32_t diag_lower_bound(const SwPlanes &pl, const SwTask &t, int32_t d0, const SwScore &sc) {
  const int32_t m = (int32_t)t.m, n = (int32_t)t.n;
  const int32_t i_lo = d0 < 0 ? -d0 : 0, i_hi = (n - d0) < m ? (n - d0) : m;
  if (i_lo >= i_hi) return 0;
  int32_t run = 0, best = 0;
  for (int32_t qw = i_lo >> 5; qw <= (i_hi - 1) >> 5; qw++) {
    const uint64_t Q = __ldg(&pl.q_sbits[t.q_word + qw]);
    const uint32_t qn = __ldg(&pl.q_nmask[t.q_word + qw]);
    const uint64_t W = window_word_on_diagonal(pl, t, qw, d0);
    const uint64_t x = Q ^ W;
    const uint64_t mm = (x | (x >> 1)) & 0x5555555555555555ull;              // bit 2b set: base b mismatches
    const int32_t b_lo = i_lo - 32 * qw > 0 ? i_lo - 32 * qw : 0, b_hi = i_hi - 32 * qw < 32 ? i_hi - 32 * qw : 32;
    if (qn == 0) {
      int32_t b = b_lo;
      while (b < b_hi) {
        const uint64_t rest = mm >> (2 * b);
        int32_t z = rest ? (__ffsll((long long)rest) - 1) >> 1 : 32;         // matches before the next mismatch
        if (b + z > b_hi) z = b_hi - b;
        run += sc.match * z; if (run > best) best = run;
        b += z;
        if (b < b_hi) { run -= sc.mismatch; if (run < 0) run = 0; b++; }
      }
    } else {
      for (int32_t b = b_lo; b < b_hi; b++) {
        const int32_t sco = ((qn >> b) & 1u) ? 0 : (((mm >> (2 * b)) & 1ull) ? -sc.mismatch : sc.match);
        run += sco; if (run < 0) run = 0; if (run > best) best = run;
      }
    }
  }
  return best;
}
// smallest direct tier (0..11 = 8-128 diagonals, table at the top of this file) whose band holds [-(rows - a), cols - a],
// a = ceil(score / match); SWT_TIER_NONE when the interval is wider than the widest tier allowed or the score says
// nothing. level: 1 = 32 only, 2 = 32 and 64, 3 = all twelve widths.
__device__ __forceinline__ uint32_t tier_of_width(int32_t rows, int32_t cols, int32_t score, const SwScore &sc, uint32_t level) {
  if (score <= 0) return SWT_TIER_NONE;
  return tier_of_interval(rows + cols - 2 * ceil_div_pos(score, sc.match) + 1, level);
}
// One counter per tier, one GLOBAL atomic per (CTA, tier): every thread of the CTA calls this once at the end of its kernel
// (dead threads with SWT_TIER_NONE). Per-warp global atomics — 5 M warps x up to 6 tiers on six addresses — serialised in
// L2: k_sw_rev_lists took 14.5 ms for 167 M alignments (profiles/r2_launches_bench_config2.txt), 10 ms of it these atomics.
__device__ __forceinline__ void count_tier_block(uint32_t tier, uint32_t *__restrict__ counts) {
  __shared__ uint32_t s_cnt[SWT_N_LISTS];
  if (threadIdx.x < SWT_N_LISTS) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t peers = __match_any_sync(0xffffffffu, tier);
  if (tier != SWT_TIER_NONE && (threadIdx.x & 31) == (uint32_t)(__ffs(peers) - 1)) atomicAdd(&s_cnt[tier_list(tier)], (uint32_t)__popc(peers));
  __syncthreads();
  if (threadIdx.x < SWT_N_LISTS && s_cnt[threadIdx.x]) atomicAdd(&counts[CNT_TIER + threadIdx.x], s_cnt[threadIdx.x]);
}

// Kernel class of an alignment. SWC_SLOW (the slow list, run by k_sw_striped): parameters outside the plain-Gotoh domain,
// and shapes or scores the packed full-matrix kernels cannot hold.
__device__ __forceinline__ uint32_t classify(uint32_t m, uint32_t n, const SwScore &sc) {
  if (m == 0 || n == 0) return SWC_NONE;
  if (sc.literal) return SWC_SLOW;
  const uint32_t mn = m < n ? m : n;
  // 16-bit cells: the largest possible score, scaled by 32 and biased (sw_bias), must stay below 2^15
  const bool score_ok = sc.match >= 1 && sc.match * 32 <= 127 && sc.mismatch * 32 <= 128 && sc.gap_open <= 100 && sc.gap_extend <= 100 &&
                        (uint32_t)sc.match * mn * 32u + sw_bias(sc) + 64u <= 32767u;
  if (score_ok && n <= SW_MAXCOLS) {
    if (m <= 8 * SW_R) return SWC_FAST8;
    if (m <= 16 * SW_R) return SWC_FAST16;
    if (m <= 32 * SW_R) return SWC_FAST32;
  }
  return SWC_SLOW;
}

// A band can only ever hold [-(m - a), n - a] (sw_band.cuh) when that interval's minimum width |n - m| + 1 (reached at
// a = min(m, n)) fits the widest tier (128); wider shapes (e.g. a 150-base read in a 300-base window) go straight to the
// full-matrix kernel instead of paying for a sweep that cannot prove anything.
__device__ __forceinline__ bool band_shape_ok(uint32_t m, uint32_t n) {
  const uint32_t d = m > n ? m - n : n - m;
  return m <= SWB_MAXROWS && d + 1 <= SWB_MAXW;
}

// true when no base of the window [w_start, w_start + n) has SSW code 4
__device__ __forceinline__ bool window_clean(const uint32_t *__restrict__ nmask, uint64_t w_word, uint32_t w_start, uint32_t n) {
  const uint32_t first = w_start >> 5, last = (w_start + n - 1) >> 5;
  for (uint32_t w = first; w <= last; w++) {
    uint32_t m = __ldg(&nmask[w_word + w]);
    if (w == first) m &= 0xffffffffu << (w_start & 31);
    if (w == last) { const uint32_t e = (w_start + n - 1) & 31; if (e < 31) m &= (2u << e) - 1u; }
    if (m) return false;
  }
  return true;
}

// Forward work lists. Band-eligible alignments get a tier (written to tier_f, listed later by k_tier_scatter): with
// `tiers` on, the seed-diagonal lower bound L picks the narrowest band that provably holds every optimal alignment
// (res[].score = L is what MODE 2 of k_sw_band places the band with); otherwise, or when L allows nothing <= 64
// diagonals (e.g. an indel splits the read over two diagonals), the 32-wide sweep-and-verify tier.
__device__ __forceinline__ uint32_t enlist(const SwPlanes &pl, const SwTask &t, uint32_t i, uint32_t cls, int32_t d0, uint32_t level,
                                       const SwScore &sc, SwRes *__restrict__ res, uint8_t *__restrict__ tier_f,
                                       Rec16 *__restrict__ full_keys, uint32_t *__restrict__ slow_list, uint32_t *__restrict__ counts) {
  uint32_t tier = SWT_TIER_NONE;
  if (cls == SWC_NONE) {
    SwRes o; o.score = 0; o.ref_end = -1; o.read_end = 0; o.ref_begin = -1; o.read_begin = 0; o.flags = 0; o.pad0 = o.pad1 = 0;
    res[i] = o;
  } else if (cls == SWC_SLOW) slow_list[list_slot(&counts[CNT_SLOW])] = i;
  else if ((t.flags & SWT_BAND) && !(t.flags & SWT_CLEAN)) tier = SWT_TIER_SWEEP | SWT_NCOL;   // code-4 columns: trial sweep of the masked variant
  else if (t.flags & SWT_BAND) {
    tier = SWT_TIER_SWEEP;
    if (level >= 3) {
      const int32_t L = diag_lower_bound(pl, t, d0, sc);
      const uint32_t tt = tier_of_width((int32_t)t.m, (int32_t)t.n, L, sc, level);
      if (tt != SWT_TIER_NONE) { tier = tt; res[i].score = L; }
    }
  } else { const uint32_t k = list_slot(&counts[CNT_FULL]); full_keys[k].key = t.n | ((uint64_t)cls << 16); full_keys[k].val = i; }   // same class + columns share a group
  tier_f[i] = (uint8_t)tier;
  return tier;
}

// tier byte array -> one list per tier inside `list` (tier t starts at offs[t]); order inside a list is arbitrary
// (src: the alignments to list, nullptr = all of 0..n-1; counts: the per-tier totals the lists are laid out by)
__global__ void __launch_bounds__(256)
k_tier_scatter(const uint8_t *__restrict__ tier, const uint32_t *__restrict__ src, uint32_t n, const uint32_t *__restrict__ counts,
               uint32_t *__restrict__ cursors, uint32_t *__restrict__ list, uint32_t ncol_base /* first list of the NCOL tiers */) {
  __shared__ uint32_t s_wcnt[8][SWT_N_LISTS];          // per warp and list: members, then the warp's offset inside the CTA's run
  __shared__ uint32_t s_base[SWT_N_LISTS];             // where the CTA's run of a list starts in that list
  const uint32_t k0 = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t i = k0 < n ? (src ? src[k0] : k0) : 0u;
  uint32_t t = k0 < n ? tier[i] : SWT_TIER_NONE;
  if (t != SWT_TIER_NONE) t = (t & SWT_NCOL) ? ncol_base + (t & 0x1fu) : (t & 0x1fu);
  if (threadIdx.x < 8 * SWT_N_LISTS) (&s_wcnt[0][0])[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t peers = __match_any_sync(0xffffffffu, t);
  if (t != SWT_TIER_NONE && lane == (uint32_t)(__ffs(peers) - 1)) s_wcnt[warp][t] = (uint32_t)__popc(peers);
  __syncthreads();
  if (threadIdx.x < SWT_N_LISTS) {                       // one global atomic per (CTA, list)
    uint32_t run = 0;
    for (int w = 0; w < 8; w++) { const uint32_t c = s_wcnt[w][threadIdx.x]; s_wcnt[w][threadIdx.x] = run; run += c; }
    uint32_t off = 0;
    for (uint32_t k = 0; k < threadIdx.x; k++) off += counts[k];
    s_base[threadIdx.x] = off + (run ? atomicAdd(&cursors[threadIdx.x], run) : 0u);
  }
  __syncthreads();
  if (t != SWT_TIER_NONE) list[s_base[t] + s_wcnt[warp][t] + __popc(peers & ((1u << lane) - 1u))] = i;
}

// pipeline mode: one task per seed (SmithWaterman.h:199-211)
__device__ __forceinline__ uint32_t
prepare_seed(uint32_t i, const kslam_seed *__restrict__ seeds, const uint64_t *__restrict__ r_offs,
             const uint64_t *__restrict__ r_word, const uint64_t *__restrict__ g_offs,
             const uint64_t *__restrict__ g_word, const uint32_t *__restrict__ g_nmask, const uint8_t *__restrict__ g_has_n, const SwScore &sc, uint32_t use_band,
             const SwPlanes &pl, SwTask *__restrict__ tasks, SwRes *__restrict__ res, uint8_t *__restrict__ tier_f,
             Rec16 *__restrict__ full_keys, uint32_t *__restrict__ slow_list, uint32_t *__restrict__ counts) {
  const kslam_seed s = seeds[i];
  const uint64_t qlen = r_offs[s.read + 1] - r_offs[s.read], glen = g_offs[s.entry + 1] - g_offs[s.entry];
  const uint64_t start = s.rel > 0 ? (uint64_t)s.rel : 0;                     // :205
  const uint64_t wlen = start >= glen ? 0 : (glen - start < qlen ? glen - start : qlen);   // substr clamp :206-207
  SwTask t;
  t.q_word = r_word[s.read]; t.w_word = g_word[s.entry];
  t.m = (uint32_t)qlen; t.n = (uint32_t)wlen; t.w_start = (uint32_t)start;
  const uint32_t cls = classify(t.m, t.n, sc);
  t.flags = (s.rev_comp ? SWT_REV : 0u) | (cls << 8);
  if (cls != SWC_NONE && ((g_has_n && !__ldg(&g_has_n[s.entry])) || window_clean(g_nmask, t.w_word, t.w_start, t.n))) t.flags |= SWT_CLEAN;   // (a genome without any code-4 base: no scan)
  if (use_band && cls == SWC_FAST8 && band_shape_ok(t.m, t.n) && ((t.flags & SWT_CLEAN) || use_band >= 3)) t.flags |= SWT_BAND;
  tasks[i] = t;
  // matrix diagonal of the seed's exact 32-mer match: forward seeds put read base i on genome base rel + i; reverse-
  // complement seeds put rc(read) base i there and Align sees the window reversed (SmithWaterman.h:205-208)
  const int32_t d0 = s.rev_comp ? (int32_t)t.w_start + (int32_t)t.n - s.rel - (int32_t)t.m : s.rel - (int32_t)t.w_start;
  return enlist(pl, t, i, cls, d0, use_band, sc, res, tier_f, full_keys, slow_list, counts);
}
__global__ void __launch_bounds__(256)
k_sw_prepare_seeds(const kslam_seed *__restrict__ seeds, uint32_t n, const uint64_t *__restrict__ r_offs,
                   const uint64_t *__restrict__ r_word, const uint64_t *__restrict__ g_offs,
                   const uint64_t *__restrict__ g_word, const uint32_t *__restrict__ g_nmask, const uint8_t *__restrict__ g_has_n, SwScore sc, uint32_t use_band,
                   SwPlanes pl, SwTask *__restrict__ tasks, SwRes *__restrict__ res, uint8_t *__restrict__ tier_f,
                   Rec16 *__restrict__ full_keys, uint32_t *__restrict__ slow_list, uint32_t *__restrict__ counts) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t tier = SWT_TIER_NONE;
  if (i < n) tier = prepare_seed(i, seeds, r_offs, r_word, g_offs, g_word, g_nmask, g_has_n, sc, use_band, pl, tasks, res, tier_f, full_keys, slow_list, counts);
  count_tier_block(tier, counts);       // every thread of the CTA, from this one place (it holds barriers and a full-warp match)
}

// Aligner::Align batch mode: query i against ref i, whole sequences
__global__ void __launch_bounds__(256)
k_sw_prepare_pairs(uint32_t n, const uint64_t *__restrict__ q_offs, const uint64_t *__restrict__ q_word,
                   const uint64_t *__restrict__ r_offs, const uint64_t *__restrict__ r_word,
                   const uint32_t *__restrict__ r_nmask, SwScore sc, uint32_t use_band, SwPlanes pl, SwTask *__restrict__ tasks,
                   SwRes *__restrict__ res,
                   uint8_t *__restrict__ tier_f, Rec16 *__restrict__ full_keys, uint32_t *__restrict__ slow_list,
                   uint32_t *__restrict__ counts) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t tier = SWT_TIER_NONE;
  if (i < n) {
    SwTask t;
    t.q_word = q_word[i]; t.w_word = r_word[i];
    t.m = (uint32_t)(q_offs[i + 1] - q_offs[i]); t.n = (uint32_t)(r_offs[i + 1] - r_offs[i]); t.w_start = 0;
    const uint32_t cls = classify(t.m, t.n, sc);
    t.flags = cls << 8;
    if (cls != SWC_NONE && window_clean(r_nmask, t.w_word, 0, t.n)) t.flags |= SWT_CLEAN;
    if (use_band && cls == SWC_FAST8 && band_shape_ok(t.m, t.n) && ((t.flags & SWT_CLEAN) || use_band >= 3)) t.flags |= SWT_BAND;
    tasks[i] = t;
    tier = enlist(pl, t, i, cls, 0, use_band, sc, res, tier_f, full_keys, slow_list, counts);   // no seed: try the main diagonal
  }
  count_tier_block(tier, counts);
}

// reverse pass work lists: score 0 has no reverse pass (ssw.c:903 is reached with an empty range). The forward score S
// is known, so the interval an anchored path can reach (reverse_band, sw_band.cuh) is exact and its width picks the tier.
// A band that is ONE diagonal wide (score within a mismatch or so of the perfect one) leaves only gap-free alignments
// on the main diagonal of the reversed matrix: k steps back from the end score match * k - (match + mismatch) * x with x
// mismatches, the first column holding S is the smallest such k, i.e. the smallest x — x = 0, then x = 1 are tried with
// one word-parallel diagonal score each (the rows on the way stay below S: they have fewer steps). Found: the begin
// coordinates are written here and the alignment needs no reverse sweep at all (tier code 15); not found (more
// mismatches, code-4 bases): the 8-diagonal tier as before.
#define SWR_CODE_DIAGONAL 15u
__global__ void __launch_bounds__(256)
k_sw_rev_lists(const SwTask *__restrict__ tasks, SwRes *__restrict__ res, uint32_t n, SwScore sc, SwPlanes pl,
               uint8_t *__restrict__ tier_r, uint32_t level,
               Rec16 *__restrict__ full_keys, uint32_t *__restrict__ counts) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t tier = SWT_TIER_NONE;
  if (i < n) {
    const SwTask t = tasks[i];
    const SwRes r = res[i];
    const uint32_t cls = (t.flags >> 8) & 0xffu;
    if (cls <= SWC_FAST32 && r.score > 0) {
      const int32_t rows = r.read_end + 1, cols = r.ref_end + 1;
      if (t.flags & SWT_BAND) {
        int32_t lo, hi;
        reverse_band(rows, cols, r.score, sc, &lo, &hi);
        tier = tier_of_interval(hi - lo + 1, level);
        if (!(t.flags & SWT_CLEAN)) { if (tier != SWT_TIER_NONE) tier = ncol_tier(tier) | SWT_NCOL; }
        else if (lo == 0 && hi == 0 && level >= 3) tier = SWT_TIER_SWEEP;     // (the reverse pass has no trial sweep: this list is k_sw_rev_diagonal's)
      }
      if (tier == SWT_TIER_NONE) { const uint32_t k = list_slot(&counts[CNT_FULL]); full_keys[k].key = (uint64_t)cols | ((uint64_t)cls << 16); full_keys[k].val = i; }
    }
    tier_r[i] = (uint8_t)tier;
  }
  count_tier_block(tier, counts);
}

// the diagonal shortcut over its own dense list (inside k_sw_rev_lists one alignment in eight took it and every warp paid)
__global__ void __launch_bounds__(256)
k_sw_rev_diagonal(const SwTask *__restrict__ tasks, SwRes *__restrict__ res, const uint32_t *__restrict__ list, uint32_t n_list, SwScore sc,
                  SwPlanes pl, uint8_t *__restrict__ tier_r, uint32_t *__restrict__ next_list, uint32_t *__restrict__ next_count) {
  const uint32_t k0 = blockIdx.x * blockDim.x + threadIdx.x;
  if (k0 >= n_list) return;
  const uint32_t i = list[k0];
  const SwTask t = tasks[i];
  const SwRes r = res[i];
  const int32_t rows = r.read_end + 1, cols = r.ref_end + 1;
  for (int32_t x = 0; x < 2; x++) {
    const int32_t num = r.score + (sc.match + sc.mismatch) * x;
    if (num % sc.match) continue;
    const int32_t k = num / sc.match;
    if (k < 1 || k > rows || k > cols) continue;
    if (diagonal_score(pl, t, sc, r.ref_end - k + 1, r.read_end - k + 1, k) != r.score) continue;
    res[i].ref_begin = r.ref_end - k + 1; res[i].read_begin = r.read_end - k + 1;
    res[i].flags = r.flags | SWR_REV_TIER(SWR_CODE_DIAGONAL);
    tier_r[i] = (uint8_t)SWT_TIER_NONE;
    return;
  }
  tier_r[i] = 0;                                      // the 8-diagonal tier after all
  next_list[list_slot(next_count)] = i;
}

// sorted (by columns) task ids -> work items of the full-matrix kernel: two alignments with the same column count
// share a group. Item w < W = ceil(n/2) is dense; the second member of an unequal neighbour pair becomes a single
// item appended after W through an atomic counter (slots [W, 2W) are pre-filled with SW_INVALID and exit at once).
__global__ void __launch_bounds__(256)
k_sw_make_items(const Rec16 *__restrict__ sorted, uint32_t n_fast, uint2 *__restrict__ items, uint32_t *__restrict__ extra) {
  const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
  if (2 * w >= n_fast) return;
  const uint32_t W = (n_fast + 1) / 2;
  const Rec16 a = sorted[2 * w];
  uint2 i0 = make_uint2((uint32_t)a.val, (uint32_t)a.val);
  if (2 * w + 1 < n_fast) {
    const Rec16 b = sorted[2 * w + 1];
    if (b.key == a.key) i0.y = (uint32_t)b.val;
    else items[W + list_slot(extra)] = make_uint2((uint32_t)b.val, (uint32_t)b.val);
  }
  items[w] = i0;
}

// out[0..1]: matrix cells (readLen x windowLen) of the forward / reverse sweeps — the GCUPS numerator.
// out[2]: cells actually computed by the sweep kernels (band cells of every tier an alignment went through, the whole
// matrix for the full-matrix kernel). out[3]: ALU-pipe thread-ops those cells need, the numerator of the integer-pipe
// roofline: 3 per cell (6 per s16x2 cell pair: PRMT + 5 DPX), 2.5 in the rows a direct-tier sweep runs without the
// tracking op (estimated from the final score, which can only under-count: the kernel switches at the smallest bound of
// its warp and, forward, with the lower bound it was given). Stored as twice the count to stay integral.
__global__ void __launch_bounds__(256)
k_sw_cells(const SwTask *__restrict__ tasks, const SwRes *__restrict__ res, const uint8_t *__restrict__ tier_f,
           const uint8_t *__restrict__ tier_r, uint32_t n, int32_t sc_match, unsigned long long *out) {
  unsigned long long fw = 0, rv = 0, comp = 0, ops2 = 0;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const SwTask t = tasks[i]; const SwRes r = res[i];
    if (((t.flags >> 8) & 0xffu) > SWC_FAST32) continue;
    fw += (unsigned long long)t.m * t.n;
    const uint32_t tf = tier_f[i], tr = tier_r[i], ft = (r.flags >> 8) & 15u;
    unsigned long long quiet = r.score > 0 ? (unsigned long long)(((r.score + sc_match - 1) / sc_match - 1) & ~3) : 0ull;
    if (tf != SWT_TIER_NONE && ((tf & 0x1fu) == SWT_TIER_SWEEP || (tf & SWT_SWEPT))) { comp += 32ull * t.m; ops2 += 6ull * 32ull * t.m; }      // the trial sweep
    if (tf != SWT_TIER_NONE && (tf & 0x1fu) < SWT_N_DIRECT) {
      const unsigned long long w = tier_width(tf & 0x1fu), q = quiet < t.m ? quiet : t.m;
      comp += w * t.m; ops2 += w * (5ull * q + 6ull * (t.m - q));
    }
    if (ft == 0u) { comp += (unsigned long long)t.m * t.n; ops2 += 6ull * t.m * t.n; }
    if (r.score > 0) {
      const unsigned long long rows = (unsigned long long)(r.read_end + 1), cols = (unsigned long long)(r.ref_end + 1);
      rv += rows * cols;
      if (tr != SWT_TIER_NONE && (tr & 0x1fu) < SWT_N_DIRECT) { const unsigned long long w = tier_width(tr & 0x1fu), q = quiet < rows ? quiet : rows; comp += w * rows; ops2 += w * (5ull * q + 6ull * (rows - q)); }
      else if (((r.flags >> 12) & 15u) != SWR_CODE_DIAGONAL) { comp += rows * cols; ops2 += 6ull * rows * cols; }      // (the diagonal shortcut sweeps nothing)
    }
  }
  for (int d = 16; d; d >>= 1) {
    fw += __shfl_xor_sync(0xffffffffu, fw, d); rv += __shfl_xor_sync(0xffffffffu, rv, d); comp += __shfl_xor_sync(0xffffffffu, comp, d);
    ops2 += __shfl_xor_sync(0xffffffffu, ops2, d);
  }
  if ((threadIdx.x & 31) == 0) { atomicAdd(out, fw); atomicAdd(out + 1, rv); atomicAdd(out + 2, comp); atomicAdd(out + 3, ops2); }
}

// Integer-pipe issue-rate microbenchmark: dependency-free streams of the DPX op the sweeps are made of
// (VIADDMNMX.S16x2). 8 independent chains per thread; the result is thread-ops per second.
__global__ void __launch_bounds__(256)
k_int_peak(uint32_t *__restrict__ out, uint32_t iters, uint32_t b, uint32_t c) {
  uint32_t a[8];
#pragma unroll
  for (int k = 0; k < 8; k++) a[k] = threadIdx.x * 0x10001u + k;
  for (uint32_t i = 0; i < iters; i++) {
#pragma unroll
    for (int k = 0; k < 8; k++) a[k] = __viaddmax_s16x2(a[k], b, c);
  }
  uint32_t x = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) x ^= a[k];
  out[blockIdx.x * blockDim.x + threadIdx.x] = x;
}

double sw_measure_int_peak(kslam_ctx *c) {
  const uint32_t blocks = (uint32_t)c->num_sms * 8, iters = 4096;
  DevBuf buf; buf.reserve((size_t)blocks * 256 * 4);
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
  float best = 1e30f;
  for (int rep = 0; rep < 5; rep++) {
    CUDA_TRY(cudaEventRecord(e0, c->stream));
    k_int_peak<<<blocks, 256, 0, c->stream>>>(buf.as<uint32_t>(), iters, 0x00010001u, 0x00020002u);
    CUDA_TRY(cudaEventRecord(e1, c->stream));
    CUDA_TRY(cudaEventSynchronize(e1));
    float ms; CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    if (rep && ms < best) best = ms;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  buf.release();
  return (double)blocks * 256.0 * iters * 8.0 / (best * 1e-3);
}

// ---------------------------------------------------------------- host orchestration
static SwScore make_score(const kslam_ctx *c) {
  SwScore s;
  // the reference stores the scores in an int8_t matrix: match as is, mismatch as static_cast<int8_t>(-mismatch) (ssw_cpp.cpp:25-49)
  s.match = (int8_t)c->prm.match; s.mismatch = -(int32_t)(int8_t)(-(int32_t)c->prm.mismatch);
  s.gap_open = c->prm.gap_open; s.gap_extend = c->prm.gap_extend;
  s.literal = kslam_params_fast(&c->prm) ? 0u : 1u;
  s.score_threshold = c->prm.score_threshold; s.report_cigar = c->prm.report_cigar; s.cigar_cap = c->prm.max_cigar_ops;
  return s;
}

static uint32_t read_count(kslam_ctx *c, uint32_t *d_counts, uint32_t *h_counts, int which) {
  read_small(c, h_counts + which, d_counts + which, 4);
  CUDA_TRY(cudaStreamSynchronize(c->stream));
  return h_counts[which];
}

// one banded tier over a list: the sweep kernel unpacks its own selector streams into shared memory
static uint32_t sw_level(const kslam_ctx *c);
template <int MODE, int WP, int PARTS = 1, bool NCOL = false>
static void run_band(kslam_ctx *c, const SwPlanes &pl, const SwScore &sc, const uint32_t *list, uint32_t n_list,
                     uint32_t *d_counts, uint32_t *next_list) {
  if (!n_list) return;
  SwWorkspace *w = c->sw;
  const uint32_t pairs = (n_list + 1) / 2, per_block = PARTS == 1 ? SWB_BLOCK : (SWB_BLOCK / 32) * (32 / PARTS);
  const uint32_t blocks = (pairs + per_block - 1) / per_block;
  k_sw_band<MODE, WP, PARTS, NCOL><<<blocks, SWB_BLOCK, BandSmem<WP>::BYTES, c->stream>>>(w->tasks.as<SwTask>(), list, n_list, pl, sc, w->res.as<SwRes>(),
      w->keys.as<Rec16>(), d_counts + CNT_FULL, next_list, d_counts + CNT_NEXT, w->tier.as<uint8_t>(), d_counts + CNT_TIER2, sw_level(c), 1u);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
}

// 0 = full-matrix only, 1 = 32-wide sweep tier, 2 = + 64-wide tier, 3 = + direct tiers from the seed-diagonal bound
static uint32_t sw_level(const kslam_ctx *c) { return !c->sw_band ? 0u : (!c->sw_band64 ? 1u : (c->sw_tiers ? 3u : 2u)); }

// one direct tier over its list (tier table: top of this file)
template <int MODE>
static void run_tier(kslam_ctx *c, const SwPlanes &pl, const SwScore &sc, uint32_t t, const uint32_t *list, uint32_t n_list, uint32_t *d_counts) {
  switch (t) {
    case 0: run_band<MODE, 8>(c, pl, sc, list, n_list, d_counts, nullptr); break;
    case 1: run_band<MODE, 16>(c, pl, sc, list, n_list, d_counts, nullptr); break;
    case 2: run_band<MODE, 24>(c, pl, sc, list, n_list, d_counts, nullptr); break;
    case 3: run_band<MODE, 32>(c, pl, sc, list, n_list, d_counts, nullptr); break;
    case 4: run_band<MODE, 20, 2>(c, pl, sc, list, n_list, d_counts, nullptr); break;
    case 5: run_band<MODE, 24, 2>(c, pl, sc, list, n_list, d_counts, nullptr); break;
    case 6: run_band<MODE, 28, 2>(c, pl, sc, list, n_list, d_counts, nullptr); break;
    case 7: run_band<MODE, 32, 2>(c, pl, sc, list, n_list, d_counts, nullptr); break;
    case 8: run_band<MODE, 24, 3>(c, pl, sc, list, n_list, d_counts, nullptr); break;
    case 9: run_band<MODE, 20, 4>(c, pl, sc, list, n_list, d_counts, nullptr); break;
    case 10: run_band<MODE, 32, 3>(c, pl, sc, list, n_list, d_counts, nullptr); break;
    default: run_band<MODE, 32, 4>(c, pl, sc, list, n_list, d_counts, nullptr); break;
  }
}
// ... and its masked variant for windows with code-4 columns (tiers of 16, 32, 64 and 128 diagonals only: ncol_tier())
template <int MODE>
static void run_tier_ncol(kslam_ctx *c, const SwPlanes &pl, const SwScore &sc, uint32_t t, const uint32_t *list, uint32_t n_list, uint32_t *d_counts) {
  if (!n_list) return;
  switch (t) {
    case 1: run_band<MODE, 16, 1, true>(c, pl, sc, list, n_list, d_counts, nullptr); break;
    case 3: run_band<MODE, 32, 1, true>(c, pl, sc, list, n_list, d_counts, nullptr); break;
    case 7: run_band<MODE, 32, 2, true>(c, pl, sc, list, n_list, d_counts, nullptr); break;
    case 11: run_band<MODE, 32, 4, true>(c, pl, sc, list, n_list, d_counts, nullptr); break;
    default: throw ArgError{"internal: no masked band kernel for this tier"};
  }
}

// tier byte array -> per-tier lists in `out` (of the alignments in src, nullptr = all n); d_cnt: the per-tier totals
static void make_tier_lists(kslam_ctx *c, uint32_t n, const uint8_t *tier, const uint32_t *src, uint32_t *d_counts, uint32_t *h_counts,
                            uint32_t cnt_at, uint32_t n_tiers, uint32_t *out, uint32_t *cnt) {
  cudaStream_t st = c->stream;
  CUDA_TRY(cudaMemsetAsync(d_counts + CNT_CUR, 0, SWT_N_LISTS * 4, st));
  if (n) {
    k_tier_scatter<<<(n + 255) / 256, 256, 0, st>>>(tier, src, n, d_counts + cnt_at, d_counts + CNT_CUR, out, n_tiers / 2);   // (lists: clean tiers, then NCOL tiers)
    c->launches++;
    CUDA_TRY(cudaGetLastError());
  }
  read_small(c, h_counts + cnt_at, d_counts + cnt_at, n_tiers * 4);
  CUDA_TRY(cudaStreamSynchronize(st));
  for (uint32_t t = 0; t < n_tiers; t++) cnt[t] = h_counts[cnt_at + t];
}

// one direction (forward or reverse) over the tier lists: the direct tiers (band placed exactly, 8-128 diagonals) and
// their NCOL instances; reverse only: the one-diagonal list through k_sw_rev_diagonal, what it cannot settle in the
// 8-diagonal tier; forward only: the 32-wide trial sweep, and what it bounds but cannot prove through the direct tiers
// in a second round; then every remaining alignment through the full-matrix kernel, bucketed by column count
template <bool REVERSE>
static void sw_pass(kslam_ctx *c, uint32_t n, const SwPlanes &pl, const SwScore &sc, const uint32_t cnt[SWT_N_LISTS], uint32_t *d_counts,
                    uint32_t *h_counts, uint64_t *n_band64_via_sweep, uint64_t *n_full_done) {
  SwWorkspace *w = c->sw;
  cudaStream_t st = c->stream;
  SwTask *tasks = w->tasks.as<SwTask>();
  SwRes *res = w->res.as<SwRes>();
  uint32_t *lists = w->lists.as<uint32_t>(), *next = lists + 2 * (size_t)n, *lists2 = lists + 3 * (size_t)n;
  Rec16 *keys = w->keys.as<Rec16>(), *keys2 = w->keys2.as<Rec16>();
  uint32_t off[SWT_N_LISTS + 1] = {0};
  for (uint32_t t = 1; t <= SWT_N_LISTS; t++) off[t] = off[t - 1] + cnt[t - 1];
  constexpr int DM = REVERSE ? 1 : 2;
  for (uint32_t t = 0; t < SWT_N_DIRECT; t++) run_tier<DM>(c, pl, sc, t, lists + off[t], cnt[t], d_counts);
  for (uint32_t t = 0; t < SWT_N_DIRECT; t++) run_tier_ncol<DM>(c, pl, sc, t, lists + off[SWT_N_TIERS + t], cnt[SWT_N_TIERS + t], d_counts);
  if (REVERSE && cnt[SWT_TIER_SWEEP]) {
    // one-diagonal bands: begin coordinates from a word-parallel diagonal score, no sweep; what it cannot settle runs 8 diagonals
    CUDA_TRY(cudaMemsetAsync(d_counts + CNT_NEXT, 0, 4, st));
    k_sw_rev_diagonal<<<(cnt[SWT_TIER_SWEEP] + 255) / 256, 256, 0, st>>>(tasks, res, lists + off[SWT_TIER_SWEEP], cnt[SWT_TIER_SWEEP], sc, pl,
                                                                       w->tier.as<uint8_t>() + n, next, d_counts + CNT_NEXT);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    const uint32_t n_next = read_count(c, d_counts, h_counts, CNT_NEXT);
    run_band<1, 8>(c, pl, sc, next, n_next, d_counts, nullptr);
    c->tm.n_sw_rev_diagonal = cnt[SWT_TIER_SWEEP] - n_next;
  }
  if (!REVERSE && cnt[SWT_TIER_SWEEP] + cnt[SWT_N_TIERS + SWT_TIER_SWEEP]) {
    // trial sweep; what it bounds but cannot prove goes through the direct tiers once more (second round)
    run_band<0, 32>(c, pl, sc, lists + off[SWT_TIER_SWEEP], cnt[SWT_TIER_SWEEP], d_counts, c->sw_band64 ? next : nullptr);
    run_band<0, 32, 1, true>(c, pl, sc, lists + off[SWT_N_TIERS + SWT_TIER_SWEEP], cnt[SWT_N_TIERS + SWT_TIER_SWEEP], d_counts, c->sw_band64 ? next : nullptr);
    const uint32_t n_next = read_count(c, d_counts, h_counts, CNT_NEXT);
    uint32_t cnt2[2 * SWT_N_DIRECT], off2 = 0;
    make_tier_lists(c, n_next, w->tier.as<uint8_t>(), next, d_counts, h_counts, CNT_TIER2, 2 * SWT_N_DIRECT, lists2, cnt2);
    for (uint32_t t = 0; t < SWT_N_DIRECT; t++) { run_tier<2>(c, pl, sc, t, lists2 + off2, cnt2[t], d_counts); off2 += cnt2[t]; c->tm.n_sw_fwd_tier[t] += cnt2[t]; }
    for (uint32_t t = 0; t < SWT_N_DIRECT; t++) {
      run_tier_ncol<2>(c, pl, sc, t, lists2 + off2, cnt2[SWT_N_DIRECT + t], d_counts); off2 += cnt2[SWT_N_DIRECT + t]; c->tm.n_sw_fwd_tier[t] += cnt2[SWT_N_DIRECT + t];
    }
    *n_band64_via_sweep += n_next;
  }
  const uint32_t n_full = read_count(c, d_counts, h_counts, CNT_FULL);
  *n_full_done += n_full;
  if (n_full) {
    uint64_t passes = 0;
    Rec16 *sorted = radix_sort(c, keys, keys2, n_full, 0, 0, 18, &passes);    // columns | class << 16
    uint2 *items = w->items.as<uint2>();
    const uint32_t n_items = 2 * ((n_full + 1) / 2);
    CUDA_TRY(cudaMemsetAsync(items, 0xff, (size_t)n_items * sizeof(uint2), st));
    CUDA_TRY(cudaMemsetAsync(d_counts + CNT_EXTRA, 0, 4, st));
    k_sw_make_items<<<(n_items / 2 + 255) / 256, 256, 0, st>>>(sorted, n_full, items, d_counts + CNT_EXTRA);
    constexpr int GROUPS = SW_BLOCK / 8;
    k_sw_fast<8, REVERSE><<<(n_items + GROUPS - 1) / GROUPS, SW_BLOCK, 0, st>>>(tasks, items, n_items, pl, sc, res, 1u);
    // reads of 161-320 / 321-640 bases: the same wavefront with 16 / 32 lanes per group; each instance skips the others' items
    uint32_t longest = c->reads_loaded ? c->reads.max_len : 0;
    if (c->sw_loaded && c->swq.max_len > longest) longest = c->swq.max_len;
    if (longest > 8 * SW_R) { k_sw_fast<16, REVERSE><<<(n_items + SW_BLOCK / 16 - 1) / (SW_BLOCK / 16), SW_BLOCK, 0, st>>>(tasks, items, n_items, pl, sc, res, 1u); c->launches++; }
    if (longest > 16 * SW_R) { k_sw_fast<32, REVERSE><<<(n_items + SW_BLOCK / 32 - 1) / (SW_BLOCK / 32), SW_BLOCK, 0, st>>>(tasks, items, n_items, pl, sc, res, 1u); c->launches++; }
    c->launches += 2;
    CUDA_TRY(cudaGetLastError());
  }
}

// finalize every alignment (+ the diagonal fast path), then the literal banded_sw on what is left, then the big-scratch retry
static void sw_traceback_stage(kslam_ctx *c, uint32_t n, const SwPlanes &pl, const SwScore &sc, kslam_overlap *ov, uint32_t *cig, int unflip) {
  SwWorkspace *w = c->sw;
  cudaStream_t st = c->stream;
  SwTask *tasks = w->tasks.as<SwTask>();
  SwRes *res = w->res.as<SwRes>();
  uint32_t *d_counts = c->counters.as<uint32_t>() + 32, *h_counts = c->h_counters.as<uint32_t>() + 32;
  uint32_t *retry_count = d_counts + CNT_RETRY, *overflow_count = d_counts + CNT_OVERFLOW;
  uint32_t *list1 = reinterpret_cast<uint32_t *>(w->keys.p), *list2 = reinterpret_cast<uint32_t *>(w->keys2.p);   // keys are dead by now
  CUDA_TRY(cudaMemsetAsync(retry_count, 0, 4, st));
  CUDA_TRY(cudaMemsetAsync(overflow_count, 0, 4, st));
  k_sw_traceback<<<(n + 127) / 128, 128, 0, st>>>(tasks, res, n, nullptr, pl, sc, ov, cig, unflip, 0, list1, retry_count, overflow_count, nullptr, 0);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
  const uint32_t n_dp = read_count(c, d_counts, h_counts, CNT_RETRY);
  c->tm.n_traceback_dp = n_dp;
  if (!n_dp) return;
  CUDA_TRY(cudaMemsetAsync(retry_count, 0, 4, st));
  k_sw_traceback<<<(n_dp + 127) / 128, 128, 0, st>>>(tasks, res, n_dp, list1, pl, sc, ov, cig, unflip, 1, list2, retry_count, overflow_count, nullptr, 0);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
  const uint32_t n_big = read_count(c, d_counts, h_counts, CNT_RETRY);
  if (!n_big) return;
  // up to 1 MiB per thread covers band 512 x 640 rows; few threads
  const size_t per_thread = 1u << 20;
  const uint32_t threads = n_big < 2048 ? n_big : 2048, rblocks = (threads + 127) / 128;
  w->tb_scratch.reserve((size_t)rblocks * 128 * per_thread);
  k_sw_traceback<<<rblocks, 128, 0, st>>>(tasks, res, n_big, list2, pl, sc, ov, cig, unflip, 2, nullptr, nullptr, overflow_count,
                                           w->tb_scratch.as<uint8_t>(), per_thread);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
}

static void sw_run(kslam_ctx *c, uint32_t n, const SwPlanes &pl, kslam_overlap *ov, uint32_t *cig, int unflip, DevBuf *grow_cig) {
  SwWorkspace *w = c->sw;
  cudaStream_t st = c->stream;
  const SwScore sc = make_score(c);
  SwTask *tasks = w->tasks.as<SwTask>();
  SwRes *res = w->res.as<SwRes>();
  uint32_t *d_counts = c->counters.as<uint32_t>() + 32;      // CNT_WORDS u32 counters
  uint32_t *h_counts = c->h_counters.as<uint32_t>() + 32;
  const unsigned nb = (n + 255) / 256;
  uint32_t *slow_list = w->lists.as<uint32_t>() + n;
  uint8_t *tier_f = w->tier.as<uint8_t>(), *tier_r = tier_f + n;

  // ---- forward
  cudaEvent_t e1 = tm_mark(c);
  uint32_t cnt[SWT_N_LISTS];
  make_tier_lists(c, n, tier_f, nullptr, d_counts, h_counts, CNT_TIER, SWT_N_LISTS, w->lists.as<uint32_t>(), cnt);
  const uint32_t n_slow = read_count(c, d_counts, h_counts, CNT_SLOW);
  for (uint32_t t = 0; t < SWT_N_DIRECT; t++) c->tm.n_sw_fwd_tier[t] = cnt[t] + cnt[SWT_N_TIERS + t];
  uint64_t band64_sweep = 0, full_done = 0;
  sw_pass<false>(c, n, pl, sc, cnt, d_counts, h_counts, &band64_sweep, &full_done);
  c->tm.n_sw_fast = full_done; c->tm.n_sw_slow = n_slow;
  c->tm.n_sw_band = 0;
  for (uint32_t t = 0; t < SWT_N_LISTS; t++) c->tm.n_sw_band += cnt[t];
  c->tm.n_sw_band64 = cnt[7] + band64_sweep;        // the 64-wide tier + everything that ran a direct tier after the trial sweep
  c->tm.n_sw_tier96 = cnt[10]; c->tm.n_sw_tier128 = cnt[11];
  c->tm.n_sw_tier8 = cnt[0]; c->tm.n_sw_tier16 = cnt[1]; c->tm.n_sw_tier32 = cnt[3]; c->tm.n_sw_tier48 = cnt[5]; c->tm.n_sw_tier64 = cnt[7];
  c->tm.n_sw_sweep32 = cnt[SWT_TIER_SWEEP] + cnt[SWT_N_TIERS + SWT_TIER_SWEEP];
  cudaEvent_t e2 = tm_mark(c);

  // ---- reverse
  CUDA_TRY(cudaMemsetAsync(d_counts + CNT_FULL, 0, 4, st));
  CUDA_TRY(cudaMemsetAsync(d_counts + CNT_TIER, 0, SWT_N_LISTS * 4, st));
  k_sw_rev_lists<<<nb, 256, 0, st>>>(tasks, res, n, sc, pl, tier_r, sw_level(c), w->keys.as<Rec16>(), d_counts);
  c->launches++;
  make_tier_lists(c, n, tier_r, nullptr, d_counts, h_counts, CNT_TIER, SWT_N_LISTS, w->lists.as<uint32_t>(), cnt);
  uint64_t dummy = 0, full_rev = 0;
  sw_pass<true>(c, n, pl, sc, cnt, d_counts, h_counts, &dummy, &full_rev);
  c->tm.n_sw_band_rev = 0;
  for (uint32_t t = 0; t < SWT_N_DIRECT; t++) { c->tm.n_sw_rev_tier[t] = cnt[t] + cnt[SWT_N_TIERS + t]; c->tm.n_sw_band_rev += cnt[t] + cnt[SWT_N_TIERS + t]; }
  cudaEvent_t e3 = tm_mark(c);

  // ---- the slow list (classify): k_sw_striped gives SSW's result for every parameter set
  if (n_slow) {
    uint32_t max_rows = c->reads_loaded ? c->reads.max_len : 0;
    if (c->sw_loaded && c->swq.max_len > max_rows) max_rows = c->swq.max_len;
    const uint32_t seg_cap = (max_rows + 7) / 8 + 1;
    uint32_t blocks = (n_slow + STR_GROUPS - 1) / STR_GROUPS; if (blocks > (uint32_t)c->num_sms * 8) blocks = c->num_sms * 8;
    if (seg_cap > STR_SMEM_SEGS) w->tb_scratch.reserve((size_t)blocks * STR_GROUPS * 5 * seg_cap * 16 * 2 + 64);
    else w->tb_scratch.reserve(64);
    k_sw_striped<<<blocks, STR_GROUPS * 16, 0, st>>>(tasks, slow_list, n_slow, pl, sc, res, w->tb_scratch.as<int16_t>(), seg_cap);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
  }
  cudaEvent_t e4 = tm_mark(c);
  sw_traceback_stage(c, n, pl, make_score(c), ov, cig, unflip);
  if (grow_cig) {
    // A CIGAR longer than the pool stride was truncated and flagged. The reference has no such limit (ssw.c:760-790 grows
    // its array), so the stride is raised and the stage re-run until nothing overflows; the larger stride stays with the ctx.
    while (read_count(c, d_counts, h_counts, CNT_OVERFLOW) && c->prm.max_cigar_ops < (1u << 14)) {
      c->prm.max_cigar_ops *= 4;
      grow_cig->reserve((size_t)n * c->prm.max_cigar_ops * 4 + 64);
      cig = grow_cig->as<uint32_t>();
      sw_traceback_stage(c, n, pl, make_score(c), ov, cig, unflip);
    }
  }
  cudaEvent_t e5 = tm_mark(c);
  unsigned long long *d_cells = c->counters.as<unsigned long long>() + 8;
  CUDA_TRY(cudaMemsetAsync(d_cells, 0, 32, st));
  k_sw_cells<<<c->num_sms * 2, 256, 0, st>>>(tasks, res, tier_f, tier_r, n, sc.match, d_cells);
  c->launches++;
  unsigned long long *h_cells = c->h_counters.as<unsigned long long>() + 8;
  read_small(c, h_cells, d_cells, 32);
  CUDA_TRY(cudaStreamSynchronize(st));
  c->tm.sw_cells_forward = h_cells[0]; c->tm.sw_cells_reverse = h_cells[1]; c->tm.sw_cells_computed = h_cells[2]; c->tm.sw_alu_ops = h_cells[3] / 2;
  c->tm.ms_sw_forward = tm_ms(e1, e2);
  c->tm.ms_sw_reverse = tm_ms(e2, e3);
  c->tm.ms_sw_slow = tm_ms(e3, e4);
  c->tm.ms_sw_traceback = tm_ms(e4, e5);
}


static void sw_reserve(kslam_ctx *c, uint32_t n) {
  if (!c->sw) c->sw = new SwWorkspace();
  SwWorkspace *w = c->sw;
  w->tasks.reserve((size_t)n * sizeof(SwTask) + 64);
  w->res.reserve((size_t)n * sizeof(SwRes) + 64);
  w->keys.reserve((size_t)n * sizeof(Rec16) + 64);
  w->keys2.reserve((size_t)n * sizeof(Rec16) + 64);
  w->items.reserve((size_t)(2 * ((n + 1) / 2)) * sizeof(uint2) + 64);
  w->lists.reserve((size_t)n * 16 + 64);      // tier lists | slow list | second-round alignments (sweep tier's failures) | their tier lists
  w->tier.reserve((size_t)n * 2 + 64);        // work-list tier of every alignment: forward | reverse
  c->counters.reserve(64 * 8); c->h_counters.reserve(64 * 8);
  w->n = n;
}

static void sw_reset_timers(kslam_ctx *c) {
  c->tm.ms_sw_prepare = c->tm.ms_sw_forward = c->tm.ms_sw_reverse = c->tm.ms_sw_slow = c->tm.ms_sw_traceback = 0;
  c->tm.sw_cells_forward = c->tm.sw_cells_reverse = 0;
  c->tm.n_sw_fast = c->tm.n_sw_slow = c->tm.n_sw_band = c->tm.n_sw_band64 = c->tm.n_sw_band_rev = 0; c->tm.n_traceback_dp = 0;
  c->tm.n_sw_tier8 = c->tm.n_sw_tier16 = c->tm.n_sw_tier32 = c->tm.n_sw_tier48 = c->tm.n_sw_tier64 = c->tm.n_sw_sweep32 = 0; c->tm.sw_cells_computed = 0;
  c->tm.n_sw_tier96 = c->tm.n_sw_tier128 = 0; c->tm.sw_alu_ops = 0;
  for (uint32_t t = 0; t < 12; t++) c->tm.n_sw_rev_tier[t] = c->tm.n_sw_fwd_tier[t] = 0;
  c->tm.n_sw_rev_diagonal = 0;
}

// ---- CIGAR pool compaction: the traceback writes alignment i's ops at the fixed stride i * cigar_cap; almost every
// CIGAR is one or three ops, so the pool that leaves the GPU is the dense concatenation and cigar_off indexes into it
__global__ void __launch_bounds__(256) k_cigar_lens(const kslam_overlap *__restrict__ ov, uint32_t n, uint32_t *__restrict__ lens) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) lens[i] = ov[i].cigar_len;
}
// (the strided offset is recomputed in 64 bits: i * stride passes 2^32 words from 134 M alignments on at stride 32, and
// ov[i].cigar_off, a u32, holds only its low half by then)
__global__ void __launch_bounds__(256) k_cigar_compact(kslam_overlap *__restrict__ ov, uint32_t n, const uint32_t *__restrict__ offs,
                                                       const uint32_t *__restrict__ strided, uint32_t stride, uint32_t *__restrict__ dense) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t len = ov[i].cigar_len, dst = offs[i];
  const uint32_t *src = strided + (size_t)i * stride;
  for (uint32_t j = 0; j < len; j++) dense[dst + j] = src[j];
  ov[i].cigar_off = dst;
}

static void compact_cigars(kslam_ctx *c, uint32_t n) {
  cudaStream_t st = c->stream;
  c->n_cig_words = 0;
  if (!n || !c->prm.report_cigar) return;
  c->seed_keep.reserve((size_t)n * 8 + 64);                 // free again by now: lens | offsets
  uint32_t *lens = c->seed_keep.as<uint32_t>(), *offs = lens + n;
  unsigned long long *d_cnt = c->counters.as<unsigned long long>() + 3, *h_cnt = c->h_counters.as<unsigned long long>() + 3;
  k_cigar_lens<<<(n + 255) / 256, 256, 0, st>>>(c->ov.as<kslam_overlap>(), n, lens);
  exclusive_scan_u32(c, lens, offs, n, (uint64_t *)d_cnt);
  read_small(c, h_cnt, d_cnt, 8);
  CUDA_TRY(cudaStreamSynchronize(st));
  c->n_cig_words = h_cnt[0];
  if (c->n_cig_words >> 32) throw ArgError{"the batch's CIGAR pool exceeds 2^32 words (kslam_overlap.cigar_off is 32 bits): use smaller batches"};
  c->cig_dense.reserve((size_t)c->n_cig_words * 4 + 64);
  k_cigar_compact<<<(n + 255) / 256, 256, 0, st>>>(c->ov.as<kslam_overlap>(), n, offs, c->cig.as<uint32_t>(), c->prm.max_cigar_ops, c->cig_dense.as<uint32_t>());
  c->launches += 2;
  CUDA_TRY(cudaGetLastError());
}

void sw_align_seeds(kslam_ctx *c) {
  if (c->n_seeds >> 32) throw ArgError{"more than 2^32 seeds in one batch: use smaller batches (--num-reads-at-once)"};
  const uint32_t n = (uint32_t)c->n_seeds;
  sw_reset_timers(c);
  if (!n) return;
  sw_reserve(c, n);
  cudaStream_t st = c->stream;
  const uint32_t cap = c->prm.max_cigar_ops;
  if (c->prm.report_cigar) c->cig.reserve((size_t)n * cap * 4 + 64);
  uint32_t *d_counts = c->counters.as<uint32_t>() + 32;
  SwWorkspace *w = c->sw;
  cudaEvent_t e0 = tm_mark(c);
  CUDA_TRY(cudaMemsetAsync(d_counts, 0, CNT_WORDS * 4, st));
  SwPlanes pl{c->reads.sbits.as<uint64_t>(), c->reads.nmask.as<uint32_t>(), c->genomes.sbits.as<uint64_t>(),
              c->genomes.nmask.as<uint32_t>(), c->genomes.xmask.as<uint32_t>()};
  k_sw_prepare_seeds<<<(n + 255) / 256, 256, 0, st>>>(c->seeds.as<kslam_seed>(), n, c->reads.offs.as<uint64_t>(),
      c->reads.word_off.as<uint64_t>(), c->genomes.offs.as<uint64_t>(), c->genomes.word_off.as<uint64_t>(),
      c->genomes.nmask.as<uint32_t>(), c->genomes.has_n.p ? c->genomes.has_n.as<uint8_t>() : nullptr, make_score(c), sw_level(c), pl, w->tasks.as<SwTask>(), w->res.as<SwRes>(), w->tier.as<uint8_t>(),
      w->keys.as<Rec16>(), w->lists.as<uint32_t>() + n, d_counts);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
  cudaEvent_t e1 = tm_mark(c);
  sw_run(c, n, pl, c->ov.as<kslam_overlap>(), c->prm.report_cigar ? c->cig.as<uint32_t>() : nullptr, 1, c->prm.report_cigar ? &c->cig : nullptr);
  cudaEvent_t e2 = tm_mark(c);
  compact_cigars(c, n);
  cudaEvent_t e3 = tm_mark(c);
  CUDA_TRY(cudaStreamSynchronize(st));
  c->tm.ms_sw_traceback += tm_ms(e2, e3);
  c->tm.ms_sw_prepare = tm_ms(e0, e1);
}

void sw_align_pairs(kslam_ctx *c, uint64_t n64, kslam_overlap *out_dev, uint32_t *cig_dev) {
  // the caller's pool is strided: alignment i owns words [i * max_cigar_ops, (i + 1) * max_cigar_ops), a 32-bit offset
  if (cig_dev && (n64 * c->prm.max_cigar_ops) >> 32) throw ArgError{"n * max_cigar_ops exceeds 2^32 words: split the batch"};
  const uint32_t n = (uint32_t)n64;
  sw_reset_timers(c);
  if (!n) return;
  sw_reserve(c, n);
  cudaStream_t st = c->stream;
  uint32_t *d_counts = c->counters.as<uint32_t>() + 32;
  SwWorkspace *w = c->sw;
  cudaEvent_t e0 = tm_mark(c);
  CUDA_TRY(cudaMemsetAsync(d_counts, 0, CNT_WORDS * 4, st));
  CUDA_TRY(cudaMemsetAsync(out_dev, 0, (size_t)n * sizeof(kslam_overlap), st));
  SwPlanes pl{c->swq.sbits.as<uint64_t>(), c->swq.nmask.as<uint32_t>(), c->swr.sbits.as<uint64_t>(),
              c->swr.nmask.as<uint32_t>(), c->swr.xmask.as<uint32_t>()};
  k_sw_prepare_pairs<<<(n + 255) / 256, 256, 0, st>>>(n, c->swq.offs.as<uint64_t>(), c->swq.word_off.as<uint64_t>(),
      c->swr.offs.as<uint64_t>(), c->swr.word_off.as<uint64_t>(), c->swr.nmask.as<uint32_t>(), make_score(c), sw_level(c), pl,
      w->tasks.as<SwTask>(), w->res.as<SwRes>(), w->tier.as<uint8_t>(), w->keys.as<Rec16>(), w->lists.as<uint32_t>() + n, d_counts);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
  cudaEvent_t e1 = tm_mark(c);
  sw_run(c, n, pl, out_dev, cig_dev, 0, nullptr);
  c->tm.ms_sw_prepare = tm_ms(e0, e1);
}

// the band of the reverse sweeps as a host function (pure arithmetic: tests/test_reverse_band.py checks it against a
// brute-force scan of the full reversed matrix without a GPU)
extern "C" int kslam_reverse_band(int32_t rows, int32_t cols, int32_t score, const kslam_params *p, int32_t *lo, int32_t *hi) {
  if (!p || !lo || !hi || rows < 1 || cols < 1 || score < 1 || !kslam_params_fast(p)) return KSLAM_ERR_ARG;
  SwScore sc{};
  sc.match = (int8_t)p->match; sc.mismatch = p->mismatch; sc.gap_open = p->gap_open; sc.gap_extend = p->gap_extend;
  reverse_band(rows, cols, score, sc, lo, hi);
  return KSLAM_OK;
}

void sw_workspace_free(kslam_ctx *c) {
  if (!c->sw) return;
  c->sw->tasks.release(); c->sw->res.release(); c->sw->keys.release(); c->sw->keys2.release();
  c->sw->items.release(); c->sw->lists.release(); c->sw->tb_scratch.release(); c->sw->tier.release();
  delete c->sw; c->sw = nullptr;
}
