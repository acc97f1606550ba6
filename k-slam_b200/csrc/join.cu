// join.cu — merge-join of the sorted read k-mer list against the resident sorted genome k-mer list
// (kernel K3), then seed sort + fuzzy unique (kernel K4).
//
// Reference: findOverlaps / processPileUp, /root/reference/src/Overlap.h:153-246 — for every pile of
// equal k-mers that starts with genome records, every read record r is crossed with every genome record
// g: seed = {r.id, g.id, (int32)(g.offset - (g.rc ? len(read) - r.offset - 32 : r.offset)), g.rc != r.rc};
// piles with kMerInt == 0 are ignored (:236-239). The reference re-extracts and re-sorts the genome
// k-mers with every batch (SLAM.h:65-66); the seed multiset only depends on which read k-mers equal which
// genome k-mers, so here the genome list is sorted once at load time and each batch sorts read records only.
// Then findOverlaps_parallel (:277-295): sort by (read, entry, rel) and std::unique with the non-transitive
// predicate overlapEqual (:79-85) — an element is dropped iff it has the same read and entry as the last
// KEPT element and |rel - rel_kept| < 3.
//
// Join: one CTA per tile of 2048 sorted read records. Two warps find the genome sub-range covered by the
// tile's [min key, max key] with a 32-ary search (one coalesced probe vector per step), the sub-range is
// staged in shared memory, every thread binary-searches its keys there, matches are counted, a CTA-wide
// scan + one global atomic reserves the output range, and seeds are emitted. HBM-bound: 16 B read per
// read record + 16 B written per seed.
#include "common.cuh"

#define JN_THREADS 256
#define JN_IPT 8
#define JN_TILE (JN_THREADS * JN_IPT)
#define JN_GCAP 3072   // genome keys staged per tile (24 KB)

// seed packing: key = read << 32 | entry ; val = (rel + bias) << 1 | rev_comp
__device__ __forceinline__ Rec16 pack_seed(uint32_t read, uint32_t entry, int32_t rel, uint32_t rc, uint32_t bias) {
  Rec16 s;
  s.key = ((uint64_t)read << 32) | entry;
  s.val = ((uint64_t)(uint32_t)(rel + (int32_t)bias) << 1) | rc;
  return s;
}

// Compact seeds: when read id, entry, rel + bias and the strand bit fit 64 bits together (every workload of BASELINE.json:
// 25 + 9 + 23 bits for config 2) a seed is ONE word, read | entry | (rel + bias) << 1 | rev_comp from the top down, whose
// plain integer order is the seed order (read, entry, rel, rev_comp). The join writes 8 bytes per seed instead of 16 and
// the seed sort is a sort of bare keys over the bits in use (radix_sort_u64): 16 B per seed and pass instead of 32 B, 7
// passes instead of 9 for config 2.
struct SeedBits { uint32_t rel_bits, ebits, rbits, compact; };
static SeedBits seed_bits(const kslam_ctx *c) {
  SeedBits b;
  b.rel_bits = ceil_log2_u64((uint64_t)c->max_genome_len + 2ull * c->reads.max_len + 2) + 1;   // (rel + bias) << 1 | rev_comp
  if (b.rel_bits > 33) b.rel_bits = 33;
  b.ebits = ceil_log2_u64(c->genomes.n > 1 ? c->genomes.n : 2);
  b.rbits = ceil_log2_u64(c->reads.n > 1 ? c->reads.n : 2);
  b.compact = b.rel_bits + b.ebits + b.rbits <= 64 ? 1u : 0u;
  return b;
}
__device__ __forceinline__ uint64_t pack_seed64(uint32_t read, uint32_t entry, int32_t rel, uint32_t rc, uint32_t bias, uint32_t rel_bits, uint32_t ebits) {
  return ((((uint64_t)read << ebits) | entry) << rel_bits) | ((uint64_t)(uint32_t)(rel + (int32_t)bias) << 1) | rc;
}
__device__ __forceinline__ Rec16 unpack_seed64(uint64_t k, uint32_t rel_bits, uint32_t ebits) {
  Rec16 s;
  const uint64_t re = k >> rel_bits;
  s.key = ((re >> ebits) << 32) | (re & ((1ull << ebits) - 1ull));
  s.val = k & ((1ull << rel_bits) - 1ull);
  return s;
}
__global__ void __launch_bounds__(256)
k_seeds_expand(const uint64_t *__restrict__ in, uint64_t n, uint32_t rel_bits, uint32_t ebits, Rec16 *__restrict__ out) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const Rec16 s = unpack_seed64(in[i], rel_bits, ebits);
    *reinterpret_cast<ulonglong2 *>(out + i) = make_ulonglong2(s.key, s.val);
  }
}

// first index in keys[0..n) with keys[idx] >= target (upper=false) or > target (upper=true); whole warp cooperates
__device__ __forceinline__ uint64_t warp_bound(const uint64_t *__restrict__ keys, uint64_t n, uint64_t target, bool upper) {
  const uint32_t lane = threadIdx.x & 31;
  uint64_t lo = 0, hi = n;   // answer in [lo, hi]
  while (hi - lo > 32) {
    uint64_t step = (hi - lo) / 33 + 1;
    uint64_t pos = lo + step * (lane + 1) - 1;        // probe positions, ascending with lane
    bool below = false;                               // true when keys[pos] is left of the answer
    if (pos < hi) { uint64_t k = __ldg(&keys[pos]); below = upper ? (k <= target) : (k < target); }
    uint32_t m = __ballot_sync(0xffffffffu, below);   // a prefix of lanes
    uint32_t nb = __popc(m);
    uint64_t nlo = nb ? lo + step * nb : lo;          // keys[lo + step*nb - 1] is below -> answer >= that + 1
    uint64_t nhi = hi;
    if (nb < 32) { uint64_t p2 = lo + step * (nb + 1) - 1; if (p2 < hi) nhi = p2; }
    lo = nlo; hi = nhi;
  }
  uint64_t pos = lo + lane;
  bool below = false;
  if (pos < hi) { uint64_t k = __ldg(&keys[pos]); below = upper ? (k <= target) : (k < target); }
  uint32_t m = __ballot_sync(0xffffffffu, below);
  return lo + __popc(m);
}

// MATCH = false: emit one-word seeds (see SeedBits) into out64 (needs the read lengths, i.e. the reads live on this GPU).
// MATCH = true: emit the raw match {read record val, genome record val}; k_matches_to_seeds turns it into a 16-byte seed
// on the GPU that owns the read, because only it knows the read length (k-mer-range partitioned database, dist.cu), or on
// this GPU when a seed does not fit one word.
template <bool MATCH>
__global__ void __launch_bounds__(JN_THREADS)
k_join(const Rec16 *__restrict__ R, uint64_t n_r, const uint64_t *__restrict__ gkeys,
       const uint64_t *__restrict__ gvals, uint64_t n_g, const uint64_t *__restrict__ read_offs,
       Rec16 *__restrict__ out, uint64_t cap, unsigned long long *__restrict__ counter, uint32_t bias, uint64_t low_mask,
       uint32_t rel_bits, uint32_t ebits) {
  uint64_t *out64 = reinterpret_cast<uint64_t *>(out);
  // R is ordered on the key bits above low_mask only (the radix sort stops there: the binary search below does not
  // need more), so the tile's key range is widened by the unsorted low bits
  __shared__ uint64_t s_g[JN_GCAP];
  __shared__ uint64_t s_range[2];
  __shared__ uint32_t s_warp[32];
  __shared__ uint32_t s_total;
  __shared__ unsigned long long s_base;
  const uint32_t tid = threadIdx.x, warp = tid >> 5;
  const uint64_t t0 = (uint64_t)blockIdx.x * JN_TILE;
  const uint64_t t1 = t0 + JN_TILE < n_r ? t0 + JN_TILE : n_r;
  if (warp == 0) { uint64_t v = warp_bound(gkeys, n_g, R[t0].key & ~low_mask, false); if (tid == 0) s_range[0] = v; }
  if (warp == 1) { uint64_t v = warp_bound(gkeys, n_g, R[t1 - 1].key | low_mask, true); if ((tid & 31) == 0) s_range[1] = v; }
  __syncthreads();
  const uint64_t g_lo = s_range[0], g_hi = s_range[1];
  const uint64_t ng = g_hi - g_lo;
  if (ng == 0) return;                               // no genome k-mer inside this tile's key range
  const bool staged = ng <= JN_GCAP;
  if (staged) for (uint32_t i = tid; i < ng; i += JN_THREADS) s_g[i] = __ldg(&gkeys[g_lo + i]);
  __syncthreads();

  uint32_t first[JN_IPT], cnt[JN_IPT];
  uint64_t rkey[JN_IPT], rval[JN_IPT];
  uint32_t my_total = 0;
#pragma unroll
  for (int i = 0; i < JN_IPT; i++) {
    uint64_t idx = t0 + (uint64_t)i * JN_THREADS + tid;
    first[i] = 0; cnt[i] = 0;
    if (idx < t1) {
      ulonglong2 r = __ldg(reinterpret_cast<const ulonglong2 *>(R + idx));
      rkey[i] = r.x; rval[i] = r.y;
      if (r.x != 0) {                                 // Overlap.h:236-239: zero k-mers never seed
        uint64_t lo = 0, hi = ng;                     // lower_bound within the tile's genome range
        if (staged) { while (lo < hi) { uint64_t mid = (lo + hi) >> 1; if (s_g[mid] < r.x) lo = mid + 1; else hi = mid; } }
        else { while (lo < hi) { uint64_t mid = (lo + hi) >> 1; if (__ldg(&gkeys[g_lo + mid]) < r.x) lo = mid + 1; else hi = mid; } }
        uint64_t e = lo;
        if (staged) { while (e < ng && s_g[e] == r.x) e++; }
        else { while (e < ng && __ldg(&gkeys[g_lo + e]) == r.x) e++; }
        first[i] = (uint32_t)lo; cnt[i] = (uint32_t)(e - lo);
        my_total += cnt[i];
      }
    }
  }
  // CTA-wide exclusive scan of per-thread seed counts, one atomic reserves the output range
  uint32_t lane = tid & 31, inc = my_total;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = lane < (JN_THREADS / 32) ? s_warp[lane] : 0, winc = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, winc, d); if (lane >= d) winc += t; }
    s_warp[lane] = winc - w;
    if (lane == 31) { s_total = winc; s_base = winc ? atomicAdd(counter, (unsigned long long)winc) : 0ull; }
  }
  __syncthreads();
  if (s_total == 0) return;
  uint64_t o = s_base + s_warp[warp] + inc - my_total;
  if (s_base + s_total > cap) return;                 // overflow: host re-runs with a larger buffer
#pragma unroll
  for (int i = 0; i < JN_IPT; i++) {
    if (cnt[i]) {
      uint32_t idf = (uint32_t)rval[i], r_off = (uint32_t)(rval[i] >> 32);
      uint32_t rid = idf & 0x3FFFFFFFu, r_rc = (idf >> 30) & 1;
      uint32_t rlen = MATCH ? 0u : (uint32_t)(__ldg(&read_offs[rid + 1]) - __ldg(&read_offs[rid]));
      for (uint32_t j = 0; j < cnt[i]; j++) {
        uint64_t gv = __ldg(&gvals[g_lo + first[i] + j]);
        if (MATCH) { *reinterpret_cast<ulonglong2 *>(out + o) = make_ulonglong2(rval[i], gv); o++; continue; }
        uint32_t gf = (uint32_t)gv, g_off = (uint32_t)(gv >> 32);
        uint32_t g_rc = (gf >> 30) & 1;
        uint32_t off = g_rc ? rlen - r_off - KSLAM_K : r_off;           // Overlap.h:185-189
        out64[o] = pack_seed64(rid, gf & 0x3FFFFFFFu, (int32_t)(g_off - off), g_rc != r_rc, bias, rel_bits, ebits);
        o++;
      }
    }
  }
}

// ---- fuzzy unique over sorted packed seeds ------------------------------------------------------
// keep[i] = 1 iff std::unique with overlapEqual (Overlap.h:79-85,290) keeps element i. The dependency on the
// last KEPT element is sequential inside a (read, entry) run, so the thread that owns a run head walks it.
__global__ void __launch_bounds__(256)
k_unique_flags(const Rec16 *__restrict__ s, uint64_t n, uint32_t *__restrict__ keep) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t k = s[i].key;
    if (i > 0 && s[i - 1].key == k) continue;       // not a run head
    int64_t last = (int64_t)(s[i].val >> 1);
    keep[i] = 1;
    for (uint64_t j = i + 1; j < n && s[j].key == k; j++) {
      int64_t rel = (int64_t)(s[j].val >> 1);
      int64_t d = rel - last; if (d < 0) d = -d;
      if (d < 3) keep[j] = 0; else { keep[j] = 1; last = rel; }
    }
  }
}

// kept seed i (packed form r) -> seeds[pos[i]], and ov[pos[i]] = the seed with every alignment field zero
__device__ __forceinline__ void emit_seed(const Rec16 r, uint32_t bias, const uint32_t *__restrict__ pos, uint64_t i,
                                          kslam_seed *__restrict__ seeds, kslam_overlap *__restrict__ ov) {
  kslam_seed o;
  o.read = (uint32_t)(r.key >> 32); o.entry = (uint32_t)r.key;
  o.rel = (int32_t)((uint32_t)(r.val >> 1) - bias); o.rev_comp = (uint32_t)(r.val & 1);
  const uint32_t p = pos[i];
  seeds[p] = o;
  kslam_overlap v;
  v.read = o.read; v.entry = o.entry; v.rel = o.rel; v.rev_comp = o.rev_comp;
  v.ref_begin = v.ref_end = v.query_begin = v.query_end = 0;
  v.sw_score = 0; v.cigar_off = 0; v.cigar_len = 0; v.flags = 0;
  ov[p] = v;
}

// the same over one-word seeds: a run is the seeds sharing the bits above rel_bits
__global__ void __launch_bounds__(256)
k_unique_flags64(const uint64_t *__restrict__ s, uint64_t n, uint32_t rel_bits, uint32_t *__restrict__ keep) {
  const uint64_t rmask = (1ull << rel_bits) - 1ull;
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t v = s[i], k = v >> rel_bits;
    if (i > 0 && (s[i - 1] >> rel_bits) == k) continue;       // not a run head
    int64_t last = (int64_t)((v & rmask) >> 1);
    keep[i] = 1;
    for (uint64_t j = i + 1; j < n; j++) {
      const uint64_t w = s[j];
      if ((w >> rel_bits) != k) break;
      const int64_t rel = (int64_t)((w & rmask) >> 1);
      int64_t d = rel - last; if (d < 0) d = -d;
      if (d < 3) keep[j] = 0; else { keep[j] = 1; last = rel; }
    }
  }
}
__global__ void __launch_bounds__(256)
k_unique_compact64(const uint64_t *__restrict__ s, uint64_t n, const uint32_t *__restrict__ keep, const uint32_t *__restrict__ pos,
                   uint32_t bias, uint32_t rel_bits, uint32_t ebits, kslam_seed *__restrict__ seeds, kslam_overlap *__restrict__ ov) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    if (!keep[i]) continue;
    emit_seed(unpack_seed64(s[i], rel_bits, ebits), bias, pos, i, seeds, ov);
  }
}

__global__ void __launch_bounds__(256)
k_unique_compact(const Rec16 *__restrict__ s, uint64_t n, const uint32_t *__restrict__ keep,
                 const uint32_t *__restrict__ pos, uint32_t bias, kslam_seed *__restrict__ seeds,
                 kslam_overlap *__restrict__ ov) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    if (!keep[i]) continue;
    emit_seed(s[i], bias, pos, i, seeds, ov);
  }
}

// Owner side of the partitioned path: raw matches {read record val, genome record val} -> packed seeds, with the
// batch-local read id (global id - id_base) and the read length only this GPU knows (Overlap.h:185-193).
__global__ void __launch_bounds__(256)
k_matches_to_seeds(const Rec16 *__restrict__ m, uint64_t n, uint32_t id_base, const uint64_t *__restrict__ read_offs,
                   uint32_t bias, Rec16 *__restrict__ out) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const ulonglong2 r = __ldg(reinterpret_cast<const ulonglong2 *>(m + i));
    const uint32_t idf = (uint32_t)r.x, r_off = (uint32_t)(r.x >> 32);
    const uint32_t rid = (idf & 0x3FFFFFFFu) - id_base, r_rc = (idf >> 30) & 1;
    const uint32_t gf = (uint32_t)r.y, g_off = (uint32_t)(r.y >> 32), g_rc = (gf >> 30) & 1;
    const uint32_t rlen = (uint32_t)(__ldg(&read_offs[rid + 1]) - __ldg(&read_offs[rid]));
    const uint32_t off = g_rc ? rlen - r_off - KSLAM_K : r_off;
    const Rec16 s = pack_seed(rid, gf & 0x3FFFFFFFu, (int32_t)(g_off - off), g_rc != r_rc, bias);
    *reinterpret_cast<ulonglong2 *>(out + i) = make_ulonglong2(s.key, s.val);
  }
}

void matches_to_seeds(kslam_ctx *c, const Rec16 *m, uint64_t n, uint32_t id_base) {
  c->n_raw = n;
  c->seeds_compact = false;
  if (!n) return;
  c->seedA.reserve((size_t)n * sizeof(Rec16));
  uint64_t blocks = (n + 255) / 256, maxb = (uint64_t)c->num_sms * 16;
  if (blocks > maxb) blocks = maxb;
  k_matches_to_seeds<<<(unsigned)blocks, 256, 0, c->stream>>>(m, n, id_base, c->reads.offs.as<uint64_t>(), c->reads.max_len,
                                                              c->seedA.as<Rec16>());
  c->launches++;
  CUDA_TRY(cudaGetLastError());
}

// merge-join of n_r sorted read records against the resident genome list; returns the number of records emitted
// into `outbuf` (one-word seeds, or raw matches when `match` is set). The buffer is regrown once on overflow.
uint64_t run_join(kslam_ctx *c, const Rec16 *R, uint64_t n_r, bool match, DevBuf &outbuf) {
  cudaStream_t st = c->stream;
  unsigned long long *d_cnt = c->counters.as<unsigned long long>();
  unsigned long long *h_cnt = c->h_counters.as<unsigned long long>();
  const uint32_t bias = c->reads.max_len;
  const uint32_t sb = kmer_sort_bits(c);
  const uint64_t low_mask = sb >= 64 ? 0ull : (~0ull >> sb);
  if (!n_r || !c->n_gk) return 0;
  const SeedBits sb64 = seed_bits(c);
  const size_t rec = match ? sizeof(Rec16) : 8;
  uint64_t cap = outbuf.cap > 64 ? (outbuf.cap - 64) / rec : 0;                  // (64 bytes of slack: the radix sort's bulk copies)
  if (cap < (1u << 20)) { outbuf.reserve((size_t)(n_r / 8 + (1u << 20)) * rec + 64); cap = (outbuf.cap - 64) / rec; }
  const uint64_t tiles = (n_r + JN_TILE - 1) / JN_TILE;
  for (int attempt = 0; attempt < 2; attempt++) {
    CUDA_TRY(cudaMemsetAsync(d_cnt, 0, 8, st));
    if (match)
      k_join<true><<<(unsigned)tiles, JN_THREADS, 0, st>>>(R, n_r, c->g_keys.as<uint64_t>(), c->g_vals.as<uint64_t>(), c->n_gk,
                                                           nullptr, outbuf.as<Rec16>(), cap, d_cnt, bias, low_mask, 0, 0);
    else
      k_join<false><<<(unsigned)tiles, JN_THREADS, 0, st>>>(R, n_r, c->g_keys.as<uint64_t>(), c->g_vals.as<uint64_t>(), c->n_gk,
                                                            c->reads.offs.as<uint64_t>(), outbuf.as<Rec16>(), cap, d_cnt, bias, low_mask, sb64.rel_bits, sb64.ebits);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    read_small(c, h_cnt, d_cnt, 8);
    CUDA_TRY(cudaStreamSynchronize(st));
    if (h_cnt[0] <= cap) break;
    if (attempt == 1) throw CudaError{cudaErrorMemoryAllocation, "seed buffer overflow after regrow", __FILE__, __LINE__};
    outbuf.reserve((size_t)h_cnt[0] * rec + 64);   // exact size is now known: grow once and redo
    cap = (outbuf.cap - 64) / rec;
  }
  return h_cnt[0];
}

void join_and_unique(kslam_ctx *c) {
  c->counters.reserve(64 * 8);
  c->h_counters.reserve(64 * 8);
  c->n_raw = 0; c->n_seeds = 0;
  cudaEvent_t e0 = tm_mark(c);
  c->seeds_compact = seed_bits(c).compact != 0;
  if (c->seeds_compact) {
    c->n_raw = run_join(c, c->sorted_rk, c->n_rk, false, c->seedA);
  } else {   // 16-byte seeds: raw matches, then the partitioned path's conversion (read ids here are batch-local)
    const uint64_t n_m = run_join(c, c->sorted_rk, c->n_rk, true, c->seedB);
    matches_to_seeds(c, c->seedB.as<Rec16>(), n_m, 0);
  }
  cudaEvent_t e1 = tm_mark(c);
  seed_sort_unique(c);
  c->tm.ms_join = tm_ms(e0, e1);
}

// seed sort + fuzzy unique (Overlap.h:277-295) over the c->n_raw packed seeds in c->seedA
void seed_sort_unique(kslam_ctx *c) {
  cudaStream_t st = c->stream;
  c->counters.reserve(64 * 8);
  c->h_counters.reserve(64 * 8);
  unsigned long long *d_cnt = c->counters.as<unsigned long long>();
  unsigned long long *h_cnt = c->h_counters.as<unsigned long long>();
  const uint32_t bias = c->reads.max_len;
  c->n_seeds = 0;
  cudaEvent_t e1 = tm_mark(c);
  c->tm.n_raw_seeds = c->n_raw;
  cudaEvent_t e2 = e1, e3 = e1;
  const SeedBits sb = seed_bits(c);
  uint64_t blocks = (c->n_raw + 255) / 256;
  if (blocks > (uint64_t)c->num_sms * 16) blocks = (uint64_t)c->num_sms * 16;
  if (c->n_raw && c->seeds_compact) {
    c->seedB.reserve((size_t)c->n_raw * 8 + 64);
    if (c->keep_taps) {   // tap: raw seeds before sorting (order is not contractual), in the 16-byte form the getter unpacks
      c->raw_seeds.reserve((size_t)c->n_raw * sizeof(Rec16));
      k_seeds_expand<<<(unsigned)blocks, 256, 0, st>>>(c->seedA.as<uint64_t>(), c->n_raw, sb.rel_bits, sb.ebits, c->raw_seeds.as<Rec16>());
      c->launches++;
    }
    uint64_t passes = 0;
    uint64_t *cur = radix_sort_u64(c, c->seedA.as<uint64_t>(), c->seedB.as<uint64_t>(), c->n_raw, 0, sb.rel_bits + sb.ebits + sb.rbits, &passes);
    c->tm.n_sort_passes += passes;
    e2 = tm_mark(c);
    c->seed_keep.reserve((size_t)c->n_raw * 8 + 64);
    uint32_t *keep = c->seed_keep.as<uint32_t>();
    uint32_t *pos = keep + c->n_raw;
    k_unique_flags64<<<(unsigned)blocks, 256, 0, st>>>(cur, c->n_raw, sb.rel_bits, keep);
    c->launches++;
    exclusive_scan_u32(c, keep, pos, c->n_raw, (uint64_t *)(d_cnt + 1));
    read_small(c, h_cnt + 1, d_cnt + 1, 8);
    CUDA_TRY(cudaStreamSynchronize(st));
    c->n_seeds = h_cnt[1];
    c->seeds.reserve((size_t)c->n_seeds * sizeof(kslam_seed) + 64);
    c->ov.reserve((size_t)c->n_seeds * sizeof(kslam_overlap) + 64);
    k_unique_compact64<<<(unsigned)blocks, 256, 0, st>>>(cur, c->n_raw, keep, pos, bias, sb.rel_bits, sb.ebits, c->seeds.as<kslam_seed>(),
                                                         c->ov.as<kslam_overlap>());
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    e3 = tm_mark(c);
  } else if (c->n_raw) {
    c->seedB.reserve((size_t)c->n_raw * sizeof(Rec16));
    if (c->keep_taps) {   // tap: raw seeds before sorting (order is not contractual)
      c->raw_seeds.reserve((size_t)c->n_raw * sizeof(Rec16));
      CUDA_TRY(cudaMemcpyAsync(c->raw_seeds.p, c->seedA.p, (size_t)c->n_raw * sizeof(Rec16), cudaMemcpyDeviceToDevice, st));
    }
    // LSD over the 128-bit composite (read, entry, rel, rev_comp): low word first, then the high word
    uint64_t passes = 0;
    Rec16 *a = c->seedA.as<Rec16>(), *b = c->seedB.as<Rec16>();
    Rec16 *cur = radix_sort(c, a, b, c->n_raw, 1, 0, sb.rel_bits, &passes);
    Rec16 *alt = cur == a ? b : a;
    cur = radix_sort(c, cur, alt, c->n_raw, 0, 0, sb.ebits, &passes);
    alt = cur == a ? b : a;
    cur = radix_sort(c, cur, alt, c->n_raw, 0, 32, 32 + sb.rbits, &passes);
    c->tm.n_sort_passes += passes;
    e2 = tm_mark(c);
    // unique
    c->seed_keep.reserve((size_t)c->n_raw * 8 + 64);
    uint32_t *keep = c->seed_keep.as<uint32_t>();
    uint32_t *pos = keep + c->n_raw;
    k_unique_flags<<<(unsigned)blocks, 256, 0, st>>>(cur, c->n_raw, keep);
    c->launches++;
    exclusive_scan_u32(c, keep, pos, c->n_raw, (uint64_t *)(d_cnt + 1));
    read_small(c, h_cnt + 1, d_cnt + 1, 8);
    CUDA_TRY(cudaStreamSynchronize(st));
    c->n_seeds = h_cnt[1];
    c->seeds.reserve((size_t)c->n_seeds * sizeof(kslam_seed) + 64);
    c->ov.reserve((size_t)c->n_seeds * sizeof(kslam_overlap) + 64);
    k_unique_compact<<<(unsigned)blocks, 256, 0, st>>>(cur, c->n_raw, keep, pos, bias, c->seeds.as<kslam_seed>(),
                                                       c->ov.as<kslam_overlap>());
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    e3 = tm_mark(c);
  }
  CUDA_TRY(cudaStreamSynchronize(st));
  c->tm.ms_seed_sort = tm_ms(e1, e2);
  c->tm.ms_unique = tm_ms(e2, e3);
  c->tm.n_seeds = c->n_seeds;
}
