// pair.cu — score screen + R1/R2 pairing (kernel K9).
//
// Reference: screenOverlapsByScoreThreshold (/root/reference/src/Overlap.h:329-341) then getPairedOverlaps
// (/root/reference/src/PairedOverlap.h:243-272): sort by (read % mid, entry, rel) and run the four-slot state
// machine getPairsFromRead (:132-242, makePair :107-123) over every (pair, entry) run.
//
// The alignment array is already ordered by (read, entry, rel) with all R1 reads before all R2 reads, so a
// STABLE radix sort on (pair id, entry, rel) yields the reference's order with R1 first on exact ties
// (SURVEY.md App. C H3). One thread walks one (pair, entry) run twice (count, then emit after a prefix sum).
#include "common.cuh"

// ---- pair order by MERGE ------------------------------------------------------------------------------------------
// alignToDatabase's vector is ordered by (read, entry, rel) with every R1 read before every R2 read, so its R1 part and
// its R2 part are each already ordered by (pair id, entry, rel): getPairedOverlaps' order is the stable merge of the two
// (R1 first on exact ties, SURVEY.md App. C H3) — one pass over the data instead of an 8-pass radix sort.
//   k_pair_flags   pass[i] = sw_score >= threshold (Overlap.h:335)                -> exclusive scan -> compact index list
//   k_pair_compact idx[pos[i]] = i for passing overlaps; the list keeps input order, its first n_a entries are R1
//   k_pair_split   merge-path partition: for every tile of PM_TILE outputs, how many come from the R1 list
//   k_pair_merge   one CTA per tile: keys of both sub-ranges staged in shared memory, every thread finds its own
//                  diagonal by binary search and merges PM_IPT outputs, writing the merged overlap records
#define PM_THREADS 128
#define PM_IPT 8
#define PM_TILE (PM_THREADS * PM_IPT)

struct PairKey { uint64_t hi; uint32_t lo; };            // (pair id << 32 | entry, rel + bias)
__device__ __forceinline__ PairKey pair_key(const kslam_overlap *__restrict__ ov, uint32_t i, uint32_t mid, uint32_t bias) {
  const uint4 w = __ldg(reinterpret_cast<const uint4 *>(ov + i));     // read, entry, rel, rev_comp
  PairKey k; k.hi = ((uint64_t)(w.x % mid) << 32) | w.y; k.lo = (uint32_t)((int32_t)w.z + (int32_t)bias);
  return k;
}
// a strictly before b? (ties: the R1 list wins, which is what the callers' "<= / <" choice encodes)
__device__ __forceinline__ bool key_less(const PairKey &a, const PairKey &b) { return a.hi < b.hi || (a.hi == b.hi && a.lo < b.lo); }

__global__ void __launch_bounds__(256)
k_pair_flags(const kslam_overlap *__restrict__ ov, uint32_t n, uint32_t mid, uint32_t thr, uint32_t *__restrict__ pass,
             uint32_t *__restrict__ n_r1_pass) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  bool p = false, r1 = false;
  if (i < n) { p = ov[i].sw_score >= thr; r1 = p && ov[i].read < mid; pass[i] = p ? 1u : 0u; }
  const uint32_t m = __ballot_sync(0xffffffffu, r1);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd(n_r1_pass, (uint32_t)__popc(m));
}

__global__ void __launch_bounds__(256)
k_pair_compact(const uint32_t *__restrict__ pass, const uint32_t *__restrict__ pos, uint32_t n, uint32_t *__restrict__ idx) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && pass[i]) idx[pos[i]] = i;
}

// the index list of the passing overlaps; nullptr = every overlap passed (threshold 0: the list would be the identity)
__device__ __forceinline__ uint32_t idx_at(const uint32_t *__restrict__ idx, uint32_t i) { return idx ? idx[i] : i; }
// threshold 0: n_r1[0] = number of overlaps of R1 reads = first position whose read is >= mid (the array is ordered by read)
__global__ void k_pair_first_r2(const kslam_overlap *__restrict__ ov, uint32_t n, uint32_t mid, uint32_t *__restrict__ n_r1) {
  uint32_t lo = 0, hi = n;
  while (lo < hi) { const uint32_t m = (lo + hi) >> 1; if (ov[m].read < mid) lo = m + 1; else hi = m; }
  *n_r1 = lo;
}

// number of R1-list elements among the first `diag` outputs of the merge of A = idx[0..na) and B = idx[na..na+nb)
__device__ __forceinline__ uint32_t merge_split(const kslam_overlap *__restrict__ ov, const uint32_t *__restrict__ idx, uint32_t na,
                                                uint32_t nb, uint32_t diag, uint32_t mid, uint32_t bias) {
  uint32_t lo = diag > nb ? diag - nb : 0u, hi = diag < na ? diag : na;       // a in [lo, hi]
  while (lo < hi) {
    const uint32_t a = (lo + hi) >> 1, b = diag - 1 - a;                        // compare A[a] with B[b]
    // A[a] goes before B[b] unless B[b] is strictly smaller (ties: A first)
    if (!key_less(pair_key(ov, idx_at(idx, na + b), mid, bias), pair_key(ov, idx_at(idx, a), mid, bias))) lo = a + 1; else hi = a;
  }
  return lo;
}

__global__ void __launch_bounds__(256)
k_pair_split(const kslam_overlap *__restrict__ ov, const uint32_t *__restrict__ idx, uint32_t na, uint32_t nb, uint32_t mid,
             uint32_t bias, uint32_t n_tiles, uint32_t *__restrict__ tile_a) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t > n_tiles) return;
  const uint64_t d = (uint64_t)t * PM_TILE;
  const uint32_t diag = d < (uint64_t)na + nb ? (uint32_t)d : na + nb;
  tile_a[t] = merge_split(ov, idx, na, nb, diag, mid, bias);
}

__global__ void __launch_bounds__(PM_THREADS)
k_pair_merge(const kslam_overlap *__restrict__ ov, const uint32_t *__restrict__ idx, uint32_t na, uint32_t nb, uint32_t mid,
             uint32_t bias, const uint32_t *__restrict__ tile_a, kslam_overlap *__restrict__ out) {
  __shared__ uint64_t s_hi[PM_TILE + 2];
  __shared__ uint32_t s_lo[PM_TILE + 2];
  __shared__ uint32_t s_src[PM_TILE + 2];
  const uint32_t tile = blockIdx.x, n = na + nb;
  const uint32_t d0 = tile * PM_TILE, d1 = d0 + PM_TILE < n ? d0 + PM_TILE : n;
  const uint32_t a0 = tile_a[tile], a1 = tile_a[tile + 1], b0 = d0 - a0, b1 = d1 - a1;
  const uint32_t ca = a1 - a0, cb = b1 - b0;                     // ca + cb == d1 - d0; A keys at [0, ca), B keys at [ca, ca + cb)
  for (uint32_t i = threadIdx.x; i < ca + cb; i += PM_THREADS) {
    const uint32_t src = i < ca ? idx_at(idx, a0 + i) : idx_at(idx, na + b0 + (i - ca));
    const PairKey k = pair_key(ov, src, mid, bias);
    s_hi[i] = k.hi; s_lo[i] = k.lo; s_src[i] = src;
  }
  __syncthreads();
  auto less_ba = [&](uint32_t b, uint32_t a) {                   // B[b] strictly before A[a]?
    return s_hi[ca + b] < s_hi[a] || (s_hi[ca + b] == s_hi[a] && s_lo[ca + b] < s_lo[a]);
  };
  const uint32_t diag = threadIdx.x * PM_IPT < ca + cb ? threadIdx.x * PM_IPT : ca + cb;
  uint32_t lo = diag > cb ? diag - cb : 0u, hi = diag < ca ? diag : ca;
  while (lo < hi) {
    const uint32_t a = (lo + hi) >> 1, b = diag - 1 - a;
    if (!less_ba(b, a)) lo = a + 1; else hi = a;
  }
  uint32_t a = lo, b = diag - lo;
  __shared__ uint32_t s_out[PM_TILE];                             // source record of every output of the tile
#pragma unroll
  for (int k = 0; k < PM_IPT; k++) {
    const uint32_t o = diag + k;
    if (o >= ca + cb) break;
    const bool take_b = a >= ca || (b < cb && less_ba(b, a));
    s_out[o] = take_b ? s_src[ca + b] : s_src[a];
    if (take_b) b++; else a++;
  }
  __syncthreads();
  // The records move as 16-byte thirds, consecutive threads on consecutive thirds: coalesced stores, and loads that are
  // sequential inside each source list (one thread copying its eight 48-byte records wrote 384-byte strides per lane:
  // 19 ms for 167 M records in profiles/r2_launches_bench_config2.txt against ~3 ms of bandwidth).
  static_assert(sizeof(kslam_overlap) == 48, "three 16-byte thirds per record");
  const uint4 *src16 = reinterpret_cast<const uint4 *>(ov);
  uint4 *dst16 = reinterpret_cast<uint4 *>(out + d0);
  for (uint32_t c = threadIdx.x; c < 3 * (ca + cb); c += PM_THREADS) {
    const uint32_t o = c / 3, part = c - 3 * o;
    dst16[c] = __ldg(src16 + (size_t)s_out[o] * 3 + part);        // cigar_off keeps pointing into the batch's dense CIGAR pool
  }
}

// getPairsFromRead over the run starting at `first`; emits into out (or only counts when out == nullptr)
__device__ uint32_t pair_run(const kslam_overlap *__restrict__ ov, uint32_t first, uint32_t n, uint32_t mid,
                             const uint64_t *__restrict__ read_offs, kslam_pair *out) {
  const uint32_t pid = ov[first].read % mid, entry = ov[first].entry;
  int32_t l1 = -1, l2 = -1, l1rc = -1, l2rc = -1;
  bool u1 = false, u2 = false, u1rc = false, u2rc = false;
  uint32_t cnt = 0;
  auto single = [&](int32_t idx, bool is_r1) {
    if (out) {
      kslam_pair p;
      p.combined_score = ov[idx].sw_score & 0xffffu; p.entry = ov[idx].entry;
      p.ref_start = ov[idx].ref_begin; p.ref_end = ov[idx].ref_end; p.insert_size = 0;
      p.r1_idx = is_r1 ? idx : -1; p.r2_idx = is_r1 ? -1 : idx; p.pad = 0;
      out[cnt] = p;
    }
    cnt++;
  };
  auto both = [&](int32_t r1, int32_t r2, bool orientation) {   // makePair, PairedOverlap.h:107-123
    if (out) {
      kslam_pair p;
      p.combined_score = (ov[r1].sw_score + ov[r2].sw_score) & 0xffffu;   // u16 ctor parameter
      p.entry = ov[r2].entry;
      p.ref_start = ov[r1].ref_begin < ov[r2].ref_begin ? ov[r1].ref_begin : ov[r2].ref_begin;
      p.ref_end = ov[r1].ref_end > ov[r2].ref_end ? ov[r1].ref_end : ov[r2].ref_end;
      const uint32_t ra = orientation ? ov[r2].read : ov[r1].read;
      const uint32_t len = (uint32_t)(read_offs[ra + 1] - read_offs[ra]);
      p.insert_size = orientation ? (uint32_t)(ov[r2].rel - ov[r1].rel) + len : (uint32_t)(ov[r1].rel - ov[r2].rel) + len;
      p.r1_idx = r1; p.r2_idx = r2; p.pad = 0;
      out[cnt] = p;
    }
    cnt++;
  };
  uint32_t cur = first;
  while (cur < n && ov[cur].read % mid == pid && ov[cur].entry == entry) {
    const int32_t c = (int32_t)cur;
    if (ov[cur].read < mid) {
      if (ov[cur].rev_comp) {
        if (!u1rc && l1rc >= 0) single(l1rc, true);
        l1rc = c; u1rc = false;
        if (l2 >= 0) { both(c, l2, false); u1rc = true; u2 = true; }
      } else {
        if (!u1 && l1 >= 0) single(l1, true);
        l1 = c; u1 = false;
        if (l2rc >= 0) { both(c, l2rc, false); u1 = true; u2rc = true; }
      }
    } else {
      if (ov[cur].rev_comp) {
        if (!u2rc && l2rc >= 0) single(l2rc, false);
        l2rc = c; u2rc = false;
        if (l1 >= 0) { both(l1, c, true); u1 = true; u2rc = true; }
      } else {
        if (!u2 && l2 >= 0) single(l2, false);
        l2 = c; u2 = false;
        if (l1rc >= 0) { both(l1rc, c, true); u1rc = true; u2 = true; }
      }
    }
    cur++;
  }
  if (!u2 && l2 >= 0) single(l2, false);          // flush order: PairedOverlap.h:217-240
  if (!u2rc && l2rc >= 0) single(l2rc, false);
  if (!u1 && l1 >= 0) single(l1, true);
  if (!u1rc && l1rc >= 0) single(l1rc, true);
  return cnt;
}

__global__ void __launch_bounds__(256)
k_pair_count(const kslam_overlap *__restrict__ ov, uint32_t n, uint32_t mid, const uint64_t *__restrict__ read_offs,
             uint32_t *__restrict__ cnt) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const bool head = k == 0 || ov[k - 1].read % mid != ov[k].read % mid || ov[k - 1].entry != ov[k].entry;
  cnt[k] = head ? pair_run(ov, k, n, mid, read_offs, nullptr) : 0u;
}

__global__ void __launch_bounds__(256)
k_pair_emit(const kslam_overlap *__restrict__ ov, uint32_t n, uint32_t mid, const uint64_t *__restrict__ read_offs,
            const uint32_t *__restrict__ cnt, const uint32_t *__restrict__ pos, kslam_pair *__restrict__ out) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n || cnt[k] == 0) return;
  pair_run(ov, k, n, mid, read_offs, out + pos[k]);
}

void pair_overlaps(kslam_ctx *c) {
  cudaStream_t st = c->stream;
  const uint32_t n = (uint32_t)c->n_seeds;
  c->n_sorted = 0; c->n_pairs = 0;
  if (!n) return;
  const uint32_t mid = (uint32_t)(c->reads.n / 2);
  if (mid == 0) return;
  uint32_t *d_cnt = c->counters.as<uint32_t>() + 48;
  uint32_t *h_cnt = c->h_counters.as<uint32_t>() + 48;
  // pass flags | positions | compact index list | tile splits, all u32
  const uint32_t max_tiles = n / PM_TILE + 2;
  c->pair_keys.reserve(((size_t)n * 3 + max_tiles + 8) * 4 + 64);
  uint32_t *pass = c->pair_keys.as<uint32_t>(), *ppos = pass + n, *idx = ppos + n, *tile_a = idx + n;
  CUDA_TRY(cudaMemsetAsync(d_cnt, 0, 16, st));
  const unsigned nb = (n + 255) / 256;
  uint32_t ns, na;
  if (c->prm.score_threshold == 0) {
    // every score passes (Overlap.h:335 compares >= 0): no flags, no scan, no index list — only where the R2 part starts
    k_pair_first_r2<<<1, 1, 0, st>>>(c->ov.as<kslam_overlap>(), n, mid, d_cnt);
    c->launches++;
    read_small(c, h_cnt, d_cnt, 4);
    CUDA_TRY(cudaStreamSynchronize(st));
    ns = n; na = h_cnt[0]; idx = nullptr;
  } else {
    k_pair_flags<<<nb, 256, 0, st>>>(c->ov.as<kslam_overlap>(), n, mid, c->prm.score_threshold, pass, d_cnt);
    unsigned long long *d_ns = c->counters.as<unsigned long long>() + 31;
    exclusive_scan_u32(c, pass, ppos, n, (uint64_t *)d_ns);
    k_pair_compact<<<nb, 256, 0, st>>>(pass, ppos, n, idx);
    c->launches += 2;
    unsigned long long *h_ns = c->h_counters.as<unsigned long long>() + 31;
    read_small(c, h_cnt, d_cnt, 4);
    read_small(c, h_ns, d_ns, 8);
    CUDA_TRY(cudaStreamSynchronize(st));
    ns = (uint32_t)h_ns[0]; na = h_cnt[0];
  }
  c->n_sorted = ns;
  if (!ns) return;
  c->ov_sorted.reserve((size_t)ns * sizeof(kslam_overlap) + 64);
  const uint32_t bias = c->reads.max_len;
  // the stable merge of the lists idx[0..la) and idx[la..la+lb) of `src` into dst[0..la+lb)
  auto merge = [&](const kslam_overlap *src, const uint32_t *ix, uint32_t la, uint32_t lb, kslam_overlap *dst) {
    const uint32_t tiles = (la + lb + PM_TILE - 1) / PM_TILE;
    if (!tiles) return;
    k_pair_split<<<(tiles + 1 + 255) / 256, 256, 0, st>>>(src, ix, la, lb, mid, bias, tiles, tile_a);
    k_pair_merge<<<tiles, PM_THREADS, 0, st>>>(src, ix, la, lb, mid, bias, tile_a, dst);
    c->launches += 2;
  };
  // An odd read count 2 mid + 1 (FASTQsequence.h:117-122 lets n2 = n1 + 1 through) gives the last read, 2 mid, pair id 0.
  // Its passing overlaps are the tail [tail, ns) of the R2 list (the input is ordered by read), out of pair-id order, so the
  // R2 list without that tail is merged with the R1 list first and the result then with the tail. The tail goes second:
  // on equal keys the reference's order is by read index, and 2 mid is the largest.
  uint32_t tail = ns;
  if (c->reads.n & 1) {
    k_pair_first_r2<<<1, 1, 0, st>>>(c->ov.as<kslam_overlap>(), n, 2 * mid, d_cnt + 1);   // first overlap of read 2 mid
    c->launches++;
    read_small(c, h_cnt + 1, d_cnt + 1, 4);
    CUDA_TRY(cudaStreamSynchronize(st));
    const uint32_t first = h_cnt[1];
    if (idx == nullptr) tail = first;
    else if (first < n) {                                  // passing overlaps before it: the exclusive scan's value there
      read_small(c, h_cnt + 1, ppos + first, 4);
      CUDA_TRY(cudaStreamSynchronize(st));
      tail = h_cnt[1];
    }
  }
  if (tail == ns) {
    merge(c->ov.as<kslam_overlap>(), idx, na, ns - na, c->ov_sorted.as<kslam_overlap>());
  } else {
    c->pair_keys2.reserve((size_t)ns * sizeof(kslam_overlap) + 64);   // (used by nothing else)
    kslam_overlap *tmp = c->pair_keys2.as<kslam_overlap>();
    merge(c->ov.as<kslam_overlap>(), idx, na, tail - na, tmp);
    // a one-list merge is a gather in list order: the tail's records follow the merged part in tmp
    merge(idx ? c->ov.as<kslam_overlap>() : c->ov.as<kslam_overlap>() + tail, idx ? idx + tail : nullptr, ns - tail, 0, tmp + tail);
    merge(tmp, nullptr, tail, ns - tail, c->ov_sorted.as<kslam_overlap>());
  }
  const unsigned nbs = (ns + 255) / 256;
  c->pair_cnt.reserve((size_t)ns * 8 + 64);
  uint32_t *cnt = c->pair_cnt.as<uint32_t>(), *pos = cnt + ns;
  k_pair_count<<<nbs, 256, 0, st>>>(c->ov_sorted.as<kslam_overlap>(), ns, mid, c->reads.offs.as<uint64_t>(), cnt);
  c->launches++;
  unsigned long long *d_tot = c->counters.as<unsigned long long>() + 30;
  exclusive_scan_u32(c, cnt, pos, ns, (uint64_t *)d_tot);
  unsigned long long *h_tot = c->h_counters.as<unsigned long long>() + 30;
  read_small(c, h_tot, d_tot, 8);
  CUDA_TRY(cudaStreamSynchronize(st));
  if (h_tot[0] >> 32) throw ArgError{"more than 2^32 pair records in one batch: use smaller batches (--num-reads-at-once)"};   // (pos[] is 32-bit)
  c->n_pairs = h_tot[0];
  if (c->n_pairs) {
    c->pairs.reserve((size_t)c->n_pairs * sizeof(kslam_pair) + 64);
    k_pair_emit<<<nbs, 256, 0, st>>>(c->ov_sorted.as<kslam_overlap>(), ns, mid, c->reads.offs.as<uint64_t>(), cnt, pos,
                                     c->pairs.as<kslam_pair>());
    c->launches++;
  }
  CUDA_TRY(cudaGetLastError());
}

// ---- compact results for runs without --sam-file (SURVEY.md §8f-3) ----------------------------------------------------------
// After pairing, a run that writes XML only needs per pair: which read pair it belongs to, entry, reference span, insert
// size, score and which mates it has (PairedOverlap.h:32-58; MetagenomicResults.h:88-111 reads nothing else) — 24 bytes
// instead of the 32-byte pair record plus the 48-byte alignment records it indexes. The one place the host stages look
// at the mates of a pair is screenPairedAlignmentsByInsertSize(replace = true) (PairedOverlap.h:396-436), which splits a
// pair whose insert size exceeds the batch's limit into its two single-ended records: those few pairs' mates are fetched
// separately once the limit is known (k_far_flags / k_far_emit keep them in pair order).
__global__ void __launch_bounds__(256)
k_pairs_compact(const kslam_pair *__restrict__ pairs, const kslam_overlap *__restrict__ ov, uint64_t n, uint32_t mid,
                kslam_pair_compact *__restrict__ out) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const kslam_pair p = pairs[i];
    kslam_pair_compact r;
    r.pair_id = p.r1_idx >= 0 ? ov[p.r1_idx].read : ov[p.r2_idx].read - mid;     // getPerReadOverlaps' thisReadPos, PairedOverlap.h:446-450
    r.entry = p.entry; r.ref_start = p.ref_start; r.ref_end = p.ref_end; r.insert_size = p.insert_size;
    r.score_flags = (p.combined_score & 0x3FFFFFFFu) | (p.r1_idx >= 0 ? 0x40000000u : 0u) | (p.r2_idx >= 0 ? 0x80000000u : 0u);
    out[i] = r;
  }
}

__global__ void __launch_bounds__(256)
k_far_flags(const kslam_pair *__restrict__ pairs, uint32_t n, uint32_t limit, uint32_t *__restrict__ flags) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flags[i] = pairs[i].insert_size > limit ? 1u : 0u;       // (a single-ended record has insert size 0)
}

__global__ void __launch_bounds__(256)
k_far_emit(const kslam_pair *__restrict__ pairs, const kslam_overlap *__restrict__ ov, uint32_t n, const uint32_t *__restrict__ flags,
           const uint32_t *__restrict__ pos, kslam_far_mates *__restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !flags[i]) return;
  const kslam_pair p = pairs[i];
  kslam_far_mates f;
  f.pair_index = i; f.pad = 0;
  const kslam_overlap a = ov[p.r1_idx], b = ov[p.r2_idx];
  f.score1 = a.sw_score; f.ref_begin1 = a.ref_begin; f.ref_end1 = a.ref_end;
  f.score2 = b.sw_score; f.ref_begin2 = b.ref_begin; f.ref_end2 = b.ref_end;
  out[pos[i]] = f;
}

// Insert-size histogram of the batch's pair records: getMaxAllowedInsertSize (PairedOverlap.h:314-360) is a function of the
// value counts only (sam.cu: InsertRuns), so the host needs the counts, not a pass over 100 M records. Fragment lengths
// crowd a few hundred values: the low range is counted in shared memory per CTA; what falls outside (0, span) is only
// counted (the caller then takes the host path over the records).
#define IH_LOW 4096u
__global__ void __launch_bounds__(256)
k_insert_hist(const kslam_pair *__restrict__ pairs, uint64_t n, uint32_t span, unsigned long long *__restrict__ hist,
              unsigned long long *__restrict__ misc /* [0] values outside (0, span), [1] largest value inside */) {
  __shared__ uint32_t s_low[IH_LOW];
  for (uint32_t i = threadIdx.x; i < IH_LOW; i += blockDim.x) s_low[i] = 0;
  __syncthreads();
  uint32_t outside = 0, top = 0;
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t v = pairs[i].insert_size;
    if (v == 0) continue;                                   // single-ended records (PairedOverlap.h:321)
    if (v >= span) { outside++; continue; }                 // (also every value that is negative as an int32)
    top = v > top ? v : top;
    if (v < IH_LOW) atomicAdd(&s_low[v], 1u); else atomicAdd(&hist[v], 1ull);
  }
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < IH_LOW; i += blockDim.x) if (s_low[i]) atomicAdd(&hist[i], (unsigned long long)s_low[i]);
  for (int d = 16; d; d >>= 1) { outside += __shfl_xor_sync(0xffffffffu, outside, d); const uint32_t o = __shfl_xor_sync(0xffffffffu, top, d); top = o > top ? o : top; }
  if ((threadIdx.x & 31) == 0) { if (outside) atomicAdd(&misc[0], (unsigned long long)outside); if (top) atomicMax(&misc[1], (unsigned long long)top); }
}

// counts of the insert sizes 0 .. *top of the batch into the ctx's pinned buffer; false when some value lies outside
// (0, 2^22) — the caller falls back to the records
bool insert_hist_device(kslam_ctx *c, const unsigned long long **h_hist, uint32_t *top) {
  constexpr uint32_t SPAN = 1u << 22;
  cudaStream_t st = c->stream;
  c->insert_hist.reserve((size_t)(SPAN + 2) * 8);
  unsigned long long *d = c->insert_hist.as<unsigned long long>(), *misc = d + SPAN;
  CUDA_TRY(cudaMemsetAsync(d, 0, (size_t)(SPAN + 2) * 8, st));
  if (c->n_pairs) {
    uint64_t blocks = (c->n_pairs + 256 * 16 - 1) / (256 * 16), maxb = (uint64_t)c->num_sms * 8;
    if (blocks > maxb) blocks = maxb;
    k_insert_hist<<<(unsigned)blocks, 256, 0, st>>>(c->pairs.as<kslam_pair>(), c->n_pairs, SPAN, d, misc);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
  }
  unsigned long long *h_misc = c->h_counters.as<unsigned long long>() + 60;   // (bytes 480-495 of the 512-byte block: nobody else's)
  read_small(c, h_misc, misc, 16);
  CUDA_TRY(cudaStreamSynchronize(st));
  if (h_misc[0]) return false;
  *top = (uint32_t)h_misc[1];
  c->h_insert_hist.reserve((size_t)(*top + 1) * 8 + 64);
  CUDA_TRY(cudaMemcpyAsync(c->h_insert_hist.p, d, (size_t)(*top + 1) * 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  *h_hist = c->h_insert_hist.as<unsigned long long>();
  return true;
}

void pairs_compact_device(kslam_ctx *c, kslam_pair_compact *out_dev) {
  if (!c->n_pairs) return;
  uint64_t blocks = (c->n_pairs + 255) / 256, maxb = (uint64_t)c->num_sms * 16;
  if (blocks > maxb) blocks = maxb;
  k_pairs_compact<<<(unsigned)blocks, 256, 0, c->stream>>>(c->pairs.as<kslam_pair>(), c->ov_sorted.as<kslam_overlap>(), c->n_pairs,
                                                           (uint32_t)(c->reads.n / 2), out_dev);
  c->launches++;
  CUDA_TRY(cudaGetLastError());
}

// the mates of every pair whose insert size exceeds `limit`, in pair order, into out_buf (device); returns their number
uint64_t far_mates_device(kslam_ctx *c, uint32_t limit, DevBuf &out_buf) {
  const uint32_t n = (uint32_t)c->n_pairs;
  if (!n) return 0;
  cudaStream_t st = c->stream;
  c->pair_cnt.reserve((size_t)n * 8 + 64);                  // free again after pairing: flags | positions
  uint32_t *flags = c->pair_cnt.as<uint32_t>(), *pos = flags + n;
  k_far_flags<<<(n + 255) / 256, 256, 0, st>>>(c->pairs.as<kslam_pair>(), n, limit, flags);
  unsigned long long *d_tot = c->counters.as<unsigned long long>() + 30, *h_tot = c->h_counters.as<unsigned long long>() + 30;
  exclusive_scan_u32(c, flags, pos, n, (uint64_t *)d_tot);
  read_small(c, h_tot, d_tot, 8);
  CUDA_TRY(cudaStreamSynchronize(st));
  const uint64_t n_far = h_tot[0];
  if (n_far) {
    out_buf.reserve((size_t)n_far * sizeof(kslam_far_mates) + 64);
    k_far_emit<<<(n + 255) / 256, 256, 0, st>>>(c->pairs.as<kslam_pair>(), c->ov_sorted.as<kslam_overlap>(), n, flags, pos,
                                                 out_buf.as<kslam_far_mates>());
    CUDA_TRY(cudaGetLastError());
  }
  c->launches += 2;
  return n_far;
}
