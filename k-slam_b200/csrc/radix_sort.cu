// radix_sort.cu — hand-written LSD radix sort of 16-byte records by a 64-bit key (kernel K2).
//
// Replaces __gnu_parallel::sort in sortKMers (/root/reference/src/KMer.h:388-398) and the seed / pairing
// sorts (/root/reference/src/Overlap.h:289, /root/reference/src/PairedOverlap.h:248-257). Design
// ("onesweep"): ONE histogram launch counts every 8-bit digit of every pass in shared memory; then each
// pass is ONE launch in which a CTA ranks a 4096-record tile with warp-wide digit matching
// (eight ballots per digit + popc, per-warp shared-memory histograms), learns its global digit offsets
// by decoupled look-back over the previous tiles' published counts, stages the tile in shared memory in
// digit order and writes it out in contiguous runs. Per pass every record is read once and written once
// (32 B); passes whose digit is constant over the whole input are skipped. Stable, so LSD order holds.
//
// Roofline: HBM. Algorithmic bytes per record = 32 B x passes (+16 B for the histogram read).
#include "common.cuh"

#define RS_MAX_PASSES 8

#define RS_FLAG_AGG (1ull << 62)
#define RS_FLAG_INCL (2ull << 62)
#define RS_VAL_MASK ((1ull << 62) - 1)

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

// lanes of the warp holding the same 8-bit digit. MATCH.ANY walks the distinct values of the warp one by one (32 of them
// for random digits: the ADU pipe was the limiter of those passes, profiles/r1k); eight ballots cost the same for any
// distribution.
__device__ __forceinline__ uint32_t digit_peers(uint32_t d) {
  uint32_t peers = 0xffffffffu;
#pragma unroll
  for (int b = 0; b < 8; b++) {
    const bool bit = (d >> b) & 1u;
    const uint32_t v = __ballot_sync(0xffffffffu, bit);
    peers &= bit ? v : ~v;
  }
  return peers;
}

// Decoupled look-back for digit `tid` of tile `tile`: publish this tile's count, sum the predecessors' published counts
// back to the nearest one that already carries an inclusive prefix, publish the inclusive prefix, return the exclusive one.
// The states of RS_LB predecessors are fetched together (independent loads in flight) and consumed in order; an
// unpublished one restarts the batch at that tile.
__device__ __forceinline__ unsigned long long publish_and_look_back(volatile unsigned long long *tile_state, uint64_t tile, uint32_t tid,
                                                                    uint32_t real_d) {
  volatile unsigned long long *my_state = tile_state + tile * 256 + tid;
  if (tile == 0) { *my_state = RS_FLAG_INCL | real_d; return 0; }
  *my_state = RS_FLAG_AGG | real_d;
  unsigned long long excl = 0;
  constexpr int RS_LB = 8;
  int64_t t = (int64_t)tile - 1;
  bool done = false;
  while (!done) {
    unsigned long long s[RS_LB];
#pragma unroll
    for (int k = 0; k < RS_LB; k++)
      s[k] = (t - k >= 0) ? tile_state[(uint64_t)(t - k) * 256 + tid] : RS_FLAG_INCL;   // before tile 0: prefix 0
    int used = 0;
#pragma unroll
    for (int k = 0; k < RS_LB; k++) {
      if (!done && used == k) {
        const unsigned long long f = s[k] >> 62;
        if (f != 0) { excl += s[k] & RS_VAL_MASK; used = k + 1; if (f == 2) done = true; }
      }
    }
    t -= used;
  }
  *my_state = RS_FLAG_INCL | (excl + real_d);
  return excl;
}

// ---- one LSD pass ------------------------------------------------------------------------------
template <int RS_THREADS, int RS_IPT>
__global__ void __launch_bounds__(RS_THREADS, (RS_THREADS * RS_IPT > 4096 ? 1 : (RS_THREADS * RS_IPT > 3072 ? 2 : (RS_THREADS * RS_IPT > 2048 ? 3 : 4))))
k_rs_onesweep(const Rec16 *__restrict__ in, Rec16 *__restrict__ out, uint64_t n, uint32_t shift, uint32_t mask,
              uint32_t word,                                       // 0: sort by .key, 1: sort by .val
              const unsigned long long *__restrict__ digit_base,  // [256] exclusive global offsets
              volatile unsigned long long *tile_state,            // [tiles][256], zero-initialised
              uint32_t *__restrict__ ticket) {
  constexpr int RS_WARPS = RS_THREADS / 32;
  constexpr uint32_t RS_TILE = RS_THREADS * RS_IPT;     // records per tile, staged in shared memory
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Rec16 *stage = reinterpret_cast<Rec16 *>(smem_raw);                               // RS_TILE records
  uint32_t *whist = reinterpret_cast<uint32_t *>(smem_raw + RS_TILE * sizeof(Rec16)); // [RS_WARPS][256]
  __shared__ uint32_t s_dexcl[256];
  __shared__ unsigned long long s_gbase[256];
  __shared__ uint32_t s_scan[32];
  __shared__ uint32_t s_tile;

  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);
#pragma unroll
  for (uint32_t i = tid; i < RS_WARPS * 256; i += RS_THREADS) whist[i] = 0;
  __syncthreads();
  const uint64_t tile = s_tile;
  const uint64_t tile_base = tile * RS_TILE;
  const uint32_t count = (uint32_t)((n - tile_base) < RS_TILE ? (n - tile_base) : RS_TILE);

  // 1. load, warp-striped so that (warp, item, lane) order == input order (stability)
  uint64_t key[RS_IPT], val[RS_IPT];
  uint32_t rank[RS_IPT];
  const uint32_t wbase = warp * 32 * RS_IPT;
#pragma unroll
  for (int i = 0; i < RS_IPT; i++) {
    uint32_t idx = wbase + i * 32 + lane;
    if (idx < count) {
      ulonglong2 r = __ldg(reinterpret_cast<const ulonglong2 *>(in + tile_base + idx));
      key[i] = r.x; val[i] = r.y;
    } else { key[i] = ~0ull; val[i] = 0; }   // padding sorts to the very end of the tile
  }

  // 2. per-warp digit ranks: peers with my digit (digit_peers), rank = earlier peers + warp running count
  uint32_t *myhist = whist + warp * 256;
  const uint32_t lt_mask = (1u << lane) - 1;
#pragma unroll
  for (int i = 0; i < RS_IPT; i++) {
    const uint32_t idx = wbase + i * 32 + lane;
    const uint32_t d = idx < count ? ((uint32_t)((word ? val[i] : key[i]) >> shift) & mask) : 255u;
    const uint32_t peers = digit_peers(d);
    const uint32_t old = myhist[d];              // every peer reads the warp's running count (broadcast)
    __syncwarp();
    if ((peers & lt_mask) == 0) myhist[d] = old + __popc(peers);   // lowest peer publishes the new count
    __syncwarp();
    rank[i] = old + __popc(peers & lt_mask);
  }
  // (a software-pipelined variant — all MATCH ops, then shared-memory atomics, then shuffles — measured 5 % slower)
  __syncthreads();

  // 3. thread d (< 256) owns digit d: exclusive offsets over warps, tile count
  uint32_t cnt_d = 0;
  if (tid < 256) {
#pragma unroll
    for (int w = 0; w < RS_WARPS; w++) { uint32_t t = whist[w * 256 + tid]; whist[w * 256 + tid] = cnt_d; cnt_d += t; }
    uint32_t real_d = cnt_d;
    if (tid == 255) real_d -= (RS_TILE - count);   // padding records were counted in digit 255

    // 4. publish, then look back for the exclusive prefix over earlier tiles
    s_gbase[tid] = digit_base[tid] + publish_and_look_back(tile_state, tile, tid, real_d);
  }

  // 5. tile-local exclusive scan over digits (counts include padding so positions cover the tile)
  if (tid < 256) {
    uint32_t inc = cnt_d;
#pragma unroll
    for (int dlt = 1; dlt < 32; dlt <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, inc, dlt); if (lane >= dlt) inc += t; }
    if (lane == 31) s_scan[warp] = inc;
    s_dexcl[tid] = inc - cnt_d;                  // exclusive within the owning warp (8 warps x 32 digits)
  }
  __syncthreads();
  if (warp == 0) {
    uint32_t w = lane < 8 ? s_scan[lane] : 0, winc = w;
#pragma unroll
    for (int dlt = 1; dlt < 8; dlt <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, winc, dlt); if (lane >= dlt) winc += t; }
    if (lane < 8) s_scan[lane] = winc - w;
  }
  __syncthreads();
  if (tid < 256) s_dexcl[tid] += s_scan[warp];
  __syncthreads();

  // 6. stage in digit order
#pragma unroll
  for (int i = 0; i < RS_IPT; i++) {
    uint32_t idx = wbase + i * 32 + lane;
    uint32_t d = idx < count ? ((uint32_t)((word ? val[i] : key[i]) >> shift) & mask) : 255u;
    uint32_t pos = s_dexcl[d] + myhist[d] + rank[i];
    *reinterpret_cast<ulonglong2 *>(stage + pos) = make_ulonglong2(key[i], val[i]);
  }
  __syncthreads();

  // 7. write out: position j of the staged tile belongs to digit d at global gbase[d] + (j - dexcl[d])
  for (uint32_t j = tid; j < count; j += RS_THREADS) {
    ulonglong2 r = *reinterpret_cast<const ulonglong2 *>(stage + j);
    uint32_t d = (uint32_t)((word ? r.y : r.x) >> shift) & mask;
    *reinterpret_cast<ulonglong2 *>(out + s_gbase[d] + (j - s_dexcl[d])) = r;
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

#include "radix_pass2.cuh"

template <int T, int I, int WORD, typename REC = Rec16>
static void launch_pass2(kslam_ctx *c, const REC *in, REC *out, uint64_t n, uint32_t shift, uint32_t mask,
                         const unsigned long long *base, uint32_t *state, uint32_t *ticket) {
  constexpr size_t smem = (size_t)T * I * sizeof(REC) + (T / 32) * 256 * sizeof(uint32_t);
  const uint64_t tiles = (n + (uint64_t)T * I - 1) / ((uint64_t)T * I);
  static bool attr_set[64] = {false};   // per instantiation
  if (!(c->device < 64 && attr_set[c->device])) {
    CUDA_TRY(cudaFuncSetAttribute(k_rs_pass2<T, I, WORD, REC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (c->device < 64) attr_set[c->device] = true;
  }
  k_rs_pass2<T, I, WORD, REC><<<(unsigned)tiles, T, smem, c->stream>>>(in, out, n, shift, mask, base, state, ticket);
}

template <int T, int I>
static void launch_onesweep(kslam_ctx *c, const Rec16 *in, Rec16 *out, uint64_t n, uint32_t shift, uint32_t mask,
                            uint32_t word, const unsigned long long *base, unsigned long long *state, uint32_t *ticket) {
  constexpr size_t smem = (size_t)T * I * sizeof(Rec16) + (T / 32) * 256 * sizeof(uint32_t);
  const uint64_t tiles = (n + (uint64_t)T * I - 1) / ((uint64_t)T * I);
  static bool attr_set[64] = {false};   // per instantiation
  if (!(c->device < 64 && attr_set[c->device])) {
    CUDA_TRY(cudaFuncSetAttribute(k_rs_onesweep<T, I>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (c->device < 64) attr_set[c->device] = true;
  }
  k_rs_onesweep<T, I><<<(unsigned)tiles, T, smem, c->stream>>>(in, out, n, shift, mask, word, base, state, ticket);
}

Rec16 *radix_sort(kslam_ctx *c, Rec16 *a, Rec16 *b, uint64_t n, uint32_t word, uint32_t lo_bit, uint32_t hi_bit,
                  uint64_t *passes_done) {
  if (n < 2 || hi_bit <= lo_bit) return a;
  if (hi_bit > 64) hi_bit = 64;
  cudaStream_t st = c->stream;
  // a wide key range is sorted in groups of <= 8 passes
  Rec16 *cur = a, *alt = b;
  PassPlan plan;
  plan.n_passes = 0;
  for (uint32_t s = lo_bit; s < hi_bit && plan.n_passes < RS_MAX_PASSES; s += 8) {
    uint32_t bits = hi_bit - s < 8 ? hi_bit - s : 8;
    plan.shift[plan.n_passes] = s; plan.mask[plan.n_passes] = (1u << bits) - 1; plan.n_passes++;
  }
  const uint64_t tile_recs = 4096;
  const uint64_t tiles = (n + tile_recs - 1) / tile_recs;
  // layout of sort_hist: [8*256 u64 hist][8 u32 trivial][8 u32 tickets][pad][tiles*256 u64 state / inclusive prefixes]
  // (k_rs_pass2: tiles*256 u32)
  const size_t hist_bytes = RS_MAX_PASSES * 256 * 8, misc_bytes = 128;
  const bool pass2 = n < (1ull << 30);                     // its 32-bit tile states hold prefixes below 2^30
  const size_t state_bytes = tiles * 256 * (pass2 ? 4 : 8);
  c->sort_hist.reserve(hist_bytes + misc_bytes + state_bytes);
  unsigned long long *ghist = c->sort_hist.as<unsigned long long>();
  uint32_t *trivial = reinterpret_cast<uint32_t *>((char *)c->sort_hist.p + hist_bytes);
  uint32_t *tickets = trivial + 8;
  unsigned long long *state = reinterpret_cast<unsigned long long *>((char *)c->sort_hist.p + hist_bytes + misc_bytes);
  CUDA_TRY(cudaMemsetAsync(c->sort_hist.p, 0, hist_bytes + misc_bytes, st));
  {
    uint64_t blocks = (n + 512 * 16 - 1) / (512 * 16);
    uint64_t maxb = (uint64_t)c->num_sms * 4;
    if (blocks > maxb) blocks = maxb;
    k_rs_hist<Rec16><<<(unsigned)blocks, 512, 0, st>>>(cur, n, plan, word, ghist);
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
    if (!pass2) launch_onesweep<256, 16>(c, cur, alt, n, plan.shift[p], plan.mask[p], word, ghist + p * 256, state, tickets + p);
    else if (word) launch_pass2<256, 16, 1>(c, cur, alt, n, plan.shift[p], plan.mask[p], ghist + p * 256, reinterpret_cast<uint32_t *>(state), tickets + p);
    else launch_pass2<256, 16, 0>(c, cur, alt, n, plan.shift[p], plan.mask[p], ghist + p * 256, reinterpret_cast<uint32_t *>(state), tickets + p);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    Rec16 *t = cur; cur = alt; alt = t;
    if (passes_done) (*passes_done)++;
  }
  return cur;
}


// Bare 8-byte keys (n < 2^30), bits [lo_bit, hi_bit): the same histogram + k_rs_pass2 passes at 16 B per key and pass,
// 8192-key tiles.
uint64_t *radix_sort_u64(kslam_ctx *c, uint64_t *a, uint64_t *b, uint64_t n, uint32_t lo_bit, uint32_t hi_bit, uint64_t *passes_done) {
  if (n < 2 || hi_bit <= lo_bit) return a;
  if (hi_bit > 64) hi_bit = 64;
  if (n >= (1ull << 30)) throw ArgError{"radix_sort_u64: more than 2^30 keys"};
  cudaStream_t st = c->stream;
  uint64_t *cur = a, *alt = b;
  PassPlan plan;
  plan.n_passes = 0;
  for (uint32_t s = lo_bit; s < hi_bit && plan.n_passes < RS_MAX_PASSES; s += 8) {
    uint32_t bits = hi_bit - s < 8 ? hi_bit - s : 8;
    plan.shift[plan.n_passes] = s; plan.mask[plan.n_passes] = (1u << bits) - 1; plan.n_passes++;
  }
  const uint64_t tile_recs = 8192;
  const uint64_t tiles = (n + tile_recs - 1) / tile_recs;
  const size_t hist_bytes = RS_MAX_PASSES * 256 * 8, misc_bytes = 128;
  const size_t state_bytes = tiles * 256 * 4;
  c->sort_hist.reserve(hist_bytes + misc_bytes + state_bytes);
  unsigned long long *ghist = c->sort_hist.as<unsigned long long>();
  uint32_t *trivial = reinterpret_cast<uint32_t *>((char *)c->sort_hist.p + hist_bytes);
  uint32_t *tickets = trivial + 8;
  uint32_t *state = reinterpret_cast<uint32_t *>((char *)c->sort_hist.p + hist_bytes + misc_bytes);
  CUDA_TRY(cudaMemsetAsync(c->sort_hist.p, 0, hist_bytes + misc_bytes, st));
  {
    uint64_t blocks = (n + 512 * 16 - 1) / (512 * 16);
    uint64_t maxb = (uint64_t)c->num_sms * 4;
    if (blocks > maxb) blocks = maxb;
    k_rs_hist<uint64_t><<<(unsigned)blocks, 512, 0, st>>>(cur, n, plan, 0, ghist);
    k_rs_scan_hist<<<1, 256, 0, st>>>(ghist, plan.n_passes, n, trivial);
    c->launches += 2;
  }
  c->h_counters.reserve(64 * 8);
  uint32_t *h_trivial = c->h_counters.as<uint32_t>() + 112;
  read_small(c, h_trivial, trivial, 8 * sizeof(uint32_t));
  CUDA_TRY(cudaStreamSynchronize(st));
  for (uint32_t p = 0; p < plan.n_passes; p++) {
    if (h_trivial[p]) continue;
    CUDA_TRY(cudaMemsetAsync(state, 0, state_bytes, st));
    launch_pass2<256, 32, 0, uint64_t>(c, cur, alt, n, plan.shift[p], plan.mask[p], ghist + p * 256, state, tickets + p);
    c->launches++;
    CUDA_TRY(cudaGetLastError());
    uint64_t *t = cur; cur = alt; alt = t;
    if (passes_done) (*passes_done)++;
  }
  return cur;
}
