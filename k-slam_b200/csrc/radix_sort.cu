// radix_sort.cu — hand-written LSD radix sort by a 64-bit key (kernel K2): 16-byte records (Rec16, by .key or .val) or
// bare 8-byte keys (the one-word seeds of join.cu).
//
// Replaces __gnu_parallel::sort in sortKMers (/root/reference/src/KMer.h:388-398) and the seed / pairing
// sorts (/root/reference/src/Overlap.h:289, /root/reference/src/PairedOverlap.h:248-257). ONE histogram launch counts
// every 8-bit digit of every pass in shared memory; then each pass is ONE launch of k_rs_pass2, in which a CTA loads a tile
// (4096 records, or 8192 bare keys) with one bulk copy, ranks it with per-warp digit histograms, learns its global digit
// offsets by decoupled look-back over the previous tiles' published counts, stages the tile in shared memory in digit order
// and writes it out in contiguous runs. Per pass every record is read once and written once (32 B; 16 B per bare key);
// passes whose digit is constant over the whole input are skipped. Stable, so LSD order holds.
//
// Roofline: HBM. Algorithmic bytes per record = 32 B x passes (+16 B for the histogram read).
// Why the pass looks the way it does (ncu on an earlier form, profiles/r2_ncu_sort_passes.txt: traffic was exactly the
// algorithmic 32 B per record, but the ALU pipe was 48 % busy, 26 % of all executed instructions sat in the look-back and
// 48 % in the ranking — issue-bound as much as latency-bound):
//  * the tile arrives by ONE bulk copy (cp.async.bulk -> mbarrier; SASS UBLKCP) straight into the staging buffer. Sixteen
//    LDG.128 per thread were interleaved by ptxas with the ranking to save registers, so every item waited out a full
//    memory latency on its own (ncu: ~900 stall samples on the first use of each of the 16 loads);
//  * ranking: per digit bit one bit-test into a predicate, VOTE, SELP, LOP3 — written in PTX because the compiler spends
//    six instructions per bit on the C form; the key word is a template parameter. Eight ballots cost the same for any
//    digit distribution; MATCH.ANY walks the distinct digits of the warp one by one (32 of them for random digits: the ADU
//    pipe was the limiter of those passes, profiles/r1k);
//  * look-back with a fast path for eight published aggregates in a row (the common case deep in the window): two
//    reductions and eight adds instead of eight flag tests. Tile states are 32-bit words below 2^30 records, which halves
//    the words the look-back polls, and 64-bit words from 2^30 on, where a per-digit prefix no longer fits 30 bits. (A
//    transposed layout, agg[digit][tile] as 16-bit counts fetched eight tiles per 16-byte load, was 3.5x SLOWER — 256
//    scattered 2-byte publications per tile, and eight tiles share every sector that successors poll.)
//  * scatter and write-out read ONE precomputed value per digit (warp offset + tile offset; global base - tile offset).
#include "common.cuh"

#define RS_MAX_PASSES 8

struct PassPlan {
  uint32_t n_passes;
  uint32_t shift[RS_MAX_PASSES];
  uint32_t mask[RS_MAX_PASSES];
};

// ---- histogram of all digits in one read of the keys ----------------------------------------
template <typename REC>
__global__ void __launch_bounds__(512)
k_rs_hist(const REC *__restrict__ in, uint64_t n, PassPlan plan, uint32_t word,
          unsigned long long *__restrict__ ghist) {
  __shared__ uint32_t s_hist[RS_MAX_PASSES * 256];
  for (uint32_t i = threadIdx.x; i < plan.n_passes * 256; i += blockDim.x) s_hist[i] = 0;
  __syncthreads();
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n;
       i += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t key;
    if constexpr (sizeof(REC) == 8) key = __ldg(&in[i]);
    else key = word ? __ldg(&in[i].val) : __ldg(&in[i].key);
#pragma unroll
    for (uint32_t p = 0; p < RS_MAX_PASSES; p++)
      if (p < plan.n_passes) atomicAdd(&s_hist[p * 256 + ((uint32_t)(key >> plan.shift[p]) & plan.mask[p])], 1u);
  }
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < plan.n_passes * 256; i += blockDim.x) {
    uint32_t v = s_hist[i];
    if (v) atomicAdd(&ghist[i], (unsigned long long)v);
  }
}

// exclusive scan of each pass' 256 counts; trivial[p] = 1 when one digit holds every record
__global__ void __launch_bounds__(256)
k_rs_scan_hist(unsigned long long *__restrict__ ghist, uint32_t n_passes, uint64_t n, uint32_t *__restrict__ trivial) {
  __shared__ unsigned long long s[256];
  for (uint32_t p = 0; p < n_passes; p++) {
    unsigned long long v = ghist[p * 256 + threadIdx.x];
    s[threadIdx.x] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned long long run = 0; uint32_t triv = 0;
      for (int d = 0; d < 256; d++) { unsigned long long t = s[d]; if (t == n) triv = 1; s[d] = run; run += t; }
      trivial[p] = triv;
    }
    __syncthreads();
    ghist[p * 256 + threadIdx.x] = s[threadIdx.x];
    __syncthreads();
  }
}

// mbarrier + bulk copy (cp.async.bulk, SASS UBLKCP) helpers: k_rs_pass2 loads its tile with one bulk copy
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  } while (!done);
}

template <int B> __device__ __forceinline__ void rs2_peer_bit(uint32_t &peers, uint32_t d) {
  asm volatile("{\n\t.reg .pred p;\n\t.reg .b32 t, v, m;\n\t"
               "and.b32 t, %1, %2;\n\tsetp.ne.u32 p, t, 0;\n\tvote.sync.ballot.b32 v, p, 0xffffffff;\n\t"
               "selp.b32 m, -1, 0, p;\n\tlop3.b32 %0, %0, v, m, 0x90;\n\t}"      // peers & ~(v ^ m)
               : "+r"(peers) : "r"(d), "n"(1 << B));
}
// lanes of the (full) warp holding the same 8-bit digit
__device__ __forceinline__ uint32_t rs2_digit_peers(uint32_t d) {
  uint32_t peers = 0xffffffffu;
  rs2_peer_bit<0>(peers, d); rs2_peer_bit<1>(peers, d); rs2_peer_bit<2>(peers, d); rs2_peer_bit<3>(peers, d);
  rs2_peer_bit<4>(peers, d); rs2_peer_bit<5>(peers, d); rs2_peer_bit<6>(peers, d); rs2_peer_bit<7>(peers, d);
  return peers;
}

// Tile states are words S (uint32_t or unsigned long long), state[tile][digit]: the highest bit = this is the inclusive
// prefix over all tiles up to and including this one, the second-highest = this is the tile's own count (aggregate); the
// value sits below both, so 32-bit states serve sorts of fewer than 2^30 records.
template <typename S> struct RsState {
  static constexpr S INCL = S(1) << (8 * sizeof(S) - 1);
  static constexpr S AGG = INCL >> 1;
  static constexpr S VAL = AGG - 1;
};

// The caller has published the aggregate of (tile, d). Sum the predecessors back to the nearest one that already carries
// an inclusive prefix, eight at a time; publish the inclusive prefix of this tile, return the exclusive one. Fast path:
// eight published aggregates and no inclusive prefix among them add up as raw words — their eight AGG bits sum to twice
// the word's range and fall off.
template <typename S>
__device__ __forceinline__ S rs2_look_back(volatile S *state, uint32_t tile, uint32_t d, uint32_t count) {
  constexpr S INCL = RsState<S>::INCL, AGG = RsState<S>::AGG, VAL = RsState<S>::VAL;
  volatile S *mine = state + (size_t)tile * 256 + d;
  S excl = 0;
  int32_t t = (int32_t)tile - 1;
  while (t >= 0) {
    S s[8];
#pragma unroll
    for (int k = 0; k < 8; k++) s[k] = (t - k >= 0) ? state[(size_t)(t - k) * 256 + d] : INCL;   // before tile 0: prefix 0
    const S all = s[0] & s[1] & s[2] & s[3] & s[4] & s[5] & s[6] & s[7];
    const S any = s[0] | s[1] | s[2] | s[3] | s[4] | s[5] | s[6] | s[7];
    if ((all & AGG) && !(any & INCL)) {
      excl += s[0] + s[1] + s[2] + s[3] + s[4] + s[5] + s[6] + s[7];
      t -= 8;
      continue;
    }
    bool done = false;
    int used = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      if (!done && used == k && (s[k] & (AGG | INCL))) {
        excl += s[k] & VAL; used = k + 1;
        if (s[k] & INCL) done = true;
      }
    }
    if (done) break;
    t -= used;                                             // an unpublished predecessor: fetch again from there
  }
  *mine = INCL | (excl + count);
  return excl;
}

// ---- one LSD pass ------------------------------------------------------------------------------
// REC = Rec16: 16-byte records sorted by .key (WORD 0) or .val (WORD 1); REC = uint64_t: bare 8-byte keys (half the bytes
// per record and pass: the packed seeds of join.cu, WORD ignored). S: tile-state word (RsState).
template <int RS_THREADS, int RS_IPT, int WORD, typename REC, typename S>
__global__ void __launch_bounds__(RS_THREADS, 2)
k_rs_pass2(const REC *__restrict__ in, REC *__restrict__ out, uint64_t n, uint32_t shift, uint32_t mask,
           const unsigned long long *__restrict__ digit_base,  // [256] exclusive global offsets
           volatile S *state,                                  // [tiles][256], zero-initialised
           uint32_t *__restrict__ ticket) {
  constexpr int RS_WARPS = RS_THREADS / 32;
  constexpr uint32_t RS_TILE = RS_THREADS * RS_IPT;
  static_assert(RS_THREADS >= 256 && RS_THREADS % 256 == 0, "threads 0..255 own one digit each");
  extern __shared__ __align__(128) unsigned char smem_raw[];   // (the alignment sets where the staging buffer starts)
  constexpr bool BARE = sizeof(REC) == 8;
  REC *stage = reinterpret_cast<REC *>(smem_raw);                                   // RS_TILE records
  uint32_t *whist = reinterpret_cast<uint32_t *>(smem_raw + RS_TILE * sizeof(REC)); // [RS_WARPS][256]
  __shared__ unsigned long long s_delta[256];
  __shared__ uint32_t s_scan[8];
  __shared__ uint32_t s_tile;

  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // 1. the tile arrives by ONE bulk copy straight into the staging buffer
  __shared__ __align__(8) uint64_t s_bar;
  if (tid == 0) {
    const uint32_t t = atomicAdd(ticket, 1u);
    s_tile = t;
    const uint64_t base = (uint64_t)t * RS_TILE;
    const uint32_t cnt = (uint32_t)((n - base) < RS_TILE ? (n - base) : RS_TILE);
    mbar_init(&s_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const uint32_t bytes = (cnt * (uint32_t)sizeof(REC) + 15u) & ~15u;      // bulk copies move multiples of 16 bytes: the buffers of
    mbar_expect_tx(&s_bar, bytes);                                          // bare 8-byte keys carry 16 bytes of slack behind the last one
    bulk_load(stage, in + base, bytes, &s_bar);
  }
#pragma unroll
  for (uint32_t i = tid; i < RS_WARPS * 256; i += RS_THREADS) whist[i] = 0;
  __syncthreads();
  const uint32_t tile = s_tile;
  const uint64_t tile_base = (uint64_t)tile * RS_TILE;
  const uint32_t count = (uint32_t)((n - tile_base) < RS_TILE ? (n - tile_base) : RS_TILE);
  mbar_wait(&s_bar, 0);

  // records to registers, warp-striped so that (warp, item, lane) order == input order (stability)
  uint64_t key[RS_IPT], val[BARE ? 1 : RS_IPT];
  const uint32_t wbase = warp * 32 * RS_IPT;
#pragma unroll
  for (int i = 0; i < RS_IPT; i++) {
    const uint32_t idx = wbase + i * 32 + lane;
    if (BARE) key[i] = idx < count ? *reinterpret_cast<const uint64_t *>(stage + idx) : ~0ull;
    else if (idx < count) {
      const ulonglong2 r = *reinterpret_cast<const ulonglong2 *>(stage + idx);
      key[i] = r.x; val[BARE ? 0 : i] = r.y;
    } else { key[i] = ~0ull; val[BARE ? 0 : i] = ~0ull; }   // padding: digit 255 whatever the shift, sorts to the very end of the tile
  }

  // 2. per-warp digit ranks: rank = earlier peers in this row + the warp's running count of the digit
  uint32_t *myhist = whist + warp * 256;
  const uint32_t lt_mask = (1u << lane) - 1;
  uint32_t dr[RS_IPT];                                    // digit << 16 | rank inside (warp, digit)
#pragma unroll
  for (int i = 0; i < RS_IPT; i++) {
    const uint32_t d = (uint32_t)(((WORD && !BARE) ? val[BARE ? 0 : i] : key[i]) >> shift) & mask & 255u;   // (padding stays 255: mask may be narrower)
    const uint32_t dd = (wbase + i * 32 + lane < count) ? d : 255u;
    const uint32_t peers = rs2_digit_peers(dd);
    const uint32_t old = myhist[dd];
    __syncwarp();
    if ((peers & lt_mask) == 0) myhist[dd] = old + __popc(peers);
    __syncwarp();
    dr[i] = (dd << 16) | (old + __popc(peers & lt_mask));
  }
  __syncthreads();

  // 3. thread d (< 256) owns digit d: exclusive offsets over warps, tile count -> publish, scan over digits, look back
  uint32_t cnt_d = 0, real_d = 0, inc = 0;
  if (tid < 256) {
#pragma unroll
    for (int w = 0; w < RS_WARPS; w++) { const uint32_t t = whist[w * 256 + tid]; whist[w * 256 + tid] = cnt_d; cnt_d += t; }
    real_d = cnt_d;
    if (tid == 255) real_d -= (RS_TILE - count);          // padding records were counted in digit 255
    state[(size_t)tile * 256 + tid] = (tile == 0 ? RsState<S>::INCL : RsState<S>::AGG) | real_d;   // successors can start summing while this tile scans
    inc = cnt_d;
#pragma unroll
    for (int dlt = 1; dlt < 32; dlt <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, inc, dlt); if (lane >= dlt) inc += t; }
    if (lane == 31) s_scan[warp] = inc;
  }
  __syncthreads();
  if (tid < 256) {
    uint32_t wexcl = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) if (w < (int)warp) wexcl += s_scan[w];
    const uint32_t dexcl = wexcl + inc - cnt_d;           // first position of digit `tid` in the staged tile
    const S excl = tile ? rs2_look_back(state, tile, tid, real_d) : S(0);
    s_delta[tid] = digit_base[tid] + excl - dexcl;        // staged position j of this digit -> global position s_delta + j
#pragma unroll
    for (int w = 0; w < RS_WARPS; w++) whist[w * 256 + tid] += dexcl;
  }
  __syncthreads();

  // 4. stage in digit order
#pragma unroll
  for (int i = 0; i < RS_IPT; i++) {
    const uint32_t pos = myhist[dr[i] >> 16] + (dr[i] & 0xffffu);
    if (BARE) *reinterpret_cast<uint64_t *>(stage + pos) = key[i];
    else *reinterpret_cast<ulonglong2 *>(stage + pos) = make_ulonglong2(key[i], val[BARE ? 0 : i]);
  }
  __syncthreads();

  // 5. write out: staged position j belongs to digit d at global s_delta[d] + j. Full tiles take the unrolled form: the
  // shared-memory loads of all items are in flight together instead of one dependent LDS -> LDS -> STG chain per item.
  if (BARE) {
    if (count == RS_TILE) {
      uint64_t r[RS_IPT];
#pragma unroll
      for (int i = 0; i < RS_IPT; i++) r[i] = *reinterpret_cast<const uint64_t *>(stage + tid + i * RS_THREADS);
#pragma unroll
      for (int i = 0; i < RS_IPT; i++) {
        const uint32_t d = (uint32_t)(r[i] >> shift) & mask;
        *reinterpret_cast<uint64_t *>(out + s_delta[d] + (tid + i * RS_THREADS)) = r[i];
      }
    } else {
      for (uint32_t j = tid; j < count; j += RS_THREADS) {
        const uint64_t r = *reinterpret_cast<const uint64_t *>(stage + j);
        *reinterpret_cast<uint64_t *>(out + s_delta[(uint32_t)(r >> shift) & mask] + j) = r;
      }
    }
  } else if (count == RS_TILE) {
    ulonglong2 r[RS_IPT];
#pragma unroll
    for (int i = 0; i < RS_IPT; i++) r[i] = *reinterpret_cast<const ulonglong2 *>(stage + tid + i * RS_THREADS);
#pragma unroll
    for (int i = 0; i < RS_IPT; i++) {
      const uint32_t d = (uint32_t)((WORD ? r[i].y : r[i].x) >> shift) & mask;
      *reinterpret_cast<ulonglong2 *>(out + s_delta[d] + (tid + i * RS_THREADS)) = r[i];
    }
  } else {
    for (uint32_t j = tid; j < count; j += RS_THREADS) {
      const ulonglong2 r = *reinterpret_cast<const ulonglong2 *>(stage + j);
      const uint32_t d = (uint32_t)((WORD ? r.y : r.x) >> shift) & mask;
      *reinterpret_cast<ulonglong2 *>(out + s_delta[d] + j) = r;
    }
  }
}

// 256 threads x 16 records (4096-record tiles) for Rec16, x 32 keys (8192-key tiles) for bare keys: 64 KB of staging
// either way (4096-key tiles of bare keys: 22.7 instead of 17.4 ms for config 2's seed sort, DESIGN.md §3.2)
template <typename REC> constexpr int rs_ipt() { return sizeof(REC) == 8 ? 32 : 16; }

template <typename REC, typename S>
static void launch_pass2(kslam_ctx *c, const REC *in, REC *out, uint64_t n, uint32_t word, uint32_t shift, uint32_t mask,
                         const unsigned long long *base, void *state, uint32_t *ticket) {
  constexpr int T = 256, I = rs_ipt<REC>();
  constexpr size_t smem = (size_t)T * I * sizeof(REC) + (T / 32) * 256 * sizeof(uint32_t);
  const uint64_t tiles = (n + (uint64_t)T * I - 1) / ((uint64_t)T * I);
  auto kern = k_rs_pass2<T, I, 0, REC, S>;
  if constexpr (sizeof(REC) == 16)
    if (word) kern = k_rs_pass2<T, I, 1, REC, S>;
  static bool attr_set[2][64] = {};   // per kernel and device
  bool *set = attr_set[word ? 1 : 0];
  if (!(c->device < 64 && set[c->device])) {
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (c->device < 64) set[c->device] = true;
  }
  kern<<<(unsigned)tiles, T, smem, c->stream>>>(in, out, n, shift, mask, base, static_cast<S *>(state), ticket);
}

// Sorts n records by bits [lo_bit, hi_bit) of the key word `word` (Rec16) or of the bare key, in groups of <= 8 passes.
template <typename REC>
static REC *sort_records(kslam_ctx *c, REC *a, REC *b, uint64_t n, uint32_t word, uint32_t lo_bit, uint32_t hi_bit,
                         uint64_t *passes_done) {
  if (n < 2 || hi_bit <= lo_bit) return a;
  if (hi_bit > 64) hi_bit = 64;
  cudaStream_t st = c->stream;
  REC *cur = a, *alt = b;
  PassPlan plan;
  plan.n_passes = 0;
  for (uint32_t s = lo_bit; s < hi_bit && plan.n_passes < RS_MAX_PASSES; s += 8) {
    uint32_t bits = hi_bit - s < 8 ? hi_bit - s : 8;
    plan.shift[plan.n_passes] = s; plan.mask[plan.n_passes] = (1u << bits) - 1; plan.n_passes++;
  }
  const uint64_t tile_recs = 256 * rs_ipt<REC>();
  const uint64_t tiles = (n + tile_recs - 1) / tile_recs;
  const bool wide = n >= (1ull << 30);                     // 32-bit tile states hold per-digit prefixes below 2^30
  // layout of sort_hist: [8*256 u64 hist][8 u32 trivial][8 u32 tickets][pad][tiles*256 tile states]
  const size_t hist_bytes = RS_MAX_PASSES * 256 * 8, misc_bytes = 128;
  const size_t state_bytes = tiles * 256 * (wide ? sizeof(unsigned long long) : sizeof(uint32_t));
  c->sort_hist.reserve(hist_bytes + misc_bytes + state_bytes);
  unsigned long long *ghist = c->sort_hist.as<unsigned long long>();
  uint32_t *trivial = reinterpret_cast<uint32_t *>((char *)c->sort_hist.p + hist_bytes);
  uint32_t *tickets = trivial + 8;
  void *state = (char *)c->sort_hist.p + hist_bytes + misc_bytes;
  CUDA_TRY(cudaMemsetAsync(c->sort_hist.p, 0, hist_bytes + misc_bytes, st));
  {
    uint64_t blocks = (n + 512 * 16 - 1) / (512 * 16);
    uint64_t maxb = (uint64_t)c->num_sms * 4;
    if (blocks > maxb) blocks = maxb;
    k_rs_hist<REC><<<(unsigned)blocks, 512, 0, st>>>(cur, n, plan, word, ghist);
    k_rs_scan_hist<<<1, 256, 0, st>>>(ghist, plan.n_passes, n, trivial);
    c->launches += 2;
  }
  c->h_counters.reserve(64 * 8);
  uint32_t *h_trivial = c->h_counters.as<uint32_t>() + 112;     // 8 words of the ctx's pinned block
  read_small(c, h_trivial, trivial, 8 * sizeof(uint32_t));
  CUDA_TRY(cudaStreamSynchronize(st));
  for (uint32_t p = 0; p < plan.n_passes; p++) {
    if (h_trivial[p]) continue;   // every record has the same digit: the pass would be the identity
    CUDA_TRY(cudaMemsetAsync(state, 0, state_bytes, st));
    if (wide) launch_pass2<REC, unsigned long long>(c, cur, alt, n, word, plan.shift[p], plan.mask[p], ghist + p * 256, state, tickets + p);
    else launch_pass2<REC, uint32_t>(c, cur, alt, n, word, plan.shift[p], plan.mask[p], ghist + p * 256, state, tickets + p);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    REC *t = cur; cur = alt; alt = t;
    if (passes_done) (*passes_done)++;
  }
  return cur;
}

Rec16 *radix_sort(kslam_ctx *c, Rec16 *a, Rec16 *b, uint64_t n, uint32_t word, uint32_t lo_bit, uint32_t hi_bit,
                  uint64_t *passes_done) {
  return sort_records(c, a, b, n, word, lo_bit, hi_bit, passes_done);
}

uint64_t *radix_sort_u64(kslam_ctx *c, uint64_t *a, uint64_t *b, uint64_t n, uint32_t lo_bit, uint32_t hi_bit, uint64_t *passes_done) {
  return sort_records(c, a, b, n, 0, lo_bit, hi_bit, passes_done);
}
