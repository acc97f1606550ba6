// radix_pass2.cuh — one LSD pass of the radix sort, second form (included by radix_sort.cu; the default).
//
// ncu on the first form, k_rs_onesweep (profiles/r2d_sort_passes.txt): traffic is exactly the algorithmic 32 B per record,
// but the ALU pipe is 48 % busy, 26 % of all executed instructions (33 % of the stall samples) sit in the look-back and
// another 48 % in the ranking — the pass is issue-bound as much as latency-bound. Same tile pipeline here (4096 records
// per CTA: load, rank, look back, stage in shared memory in digit order, write out in contiguous runs), a third fewer
// instructions:
//  * look-back over 32-bit states with a fast path for eight published aggregates in a row (the common case deep in the
//    window): two reductions and eight adds instead of eight flag tests. (A transposed layout, agg[digit][tile] as 16-bit
//    counts fetched eight tiles per 16-byte load, was tried first: 3.5x SLOWER — 256 scattered 2-byte publications per
//    tile, and eight tiles share every sector that successors poll.)
//  * ranking: per digit bit one bit-test into a predicate, VOTE, SELP, LOP3 — written in PTX because the compiler spends
//    six instructions per bit on the C form; the key word is a template parameter;
//  * scatter and write-out read ONE precomputed value per digit (warp offset + tile offset; global base - tile offset).
#pragma once


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

// Tile states are 32-bit words, state[tile][digit]: bit 30 = this is the tile's own count (aggregate), bit 31 = this is the
// inclusive prefix over all tiles up to and including this one; the value sits in the low 30 bits (the pass is used for
// sorts of fewer than 2^30 records). The caller has published the aggregate of (tile, d). Sum the predecessors back to the
// nearest one that already carries an inclusive prefix, eight at a time; publish the inclusive prefix of this tile, return
// the exclusive one. Fast path: eight published aggregates and no inclusive prefix among them add up as raw words — their
// eight flag bits sum to 2^33 and fall off the 32-bit word.
#define RS2_AGG (1u << 30)
#define RS2_INCL (1u << 31)
#define RS2_VAL (RS2_AGG - 1u)
__device__ __forceinline__ uint32_t rs2_look_back(volatile uint32_t *state, uint32_t tile, uint32_t d, uint32_t count) {
  volatile uint32_t *mine = state + (size_t)tile * 256 + d;
  uint32_t excl = 0;
  int32_t t = (int32_t)tile - 1;
  while (t >= 0) {
    uint32_t s[8];
#pragma unroll
    for (int k = 0; k < 8; k++) s[k] = (t - k >= 0) ? state[(size_t)(t - k) * 256 + d] : RS2_INCL;   // before tile 0: prefix 0
    const uint32_t all = s[0] & s[1] & s[2] & s[3] & s[4] & s[5] & s[6] & s[7];
    const uint32_t any = s[0] | s[1] | s[2] | s[3] | s[4] | s[5] | s[6] | s[7];
    if ((all & RS2_AGG) && !(any & RS2_INCL)) {
      excl += s[0] + s[1] + s[2] + s[3] + s[4] + s[5] + s[6] + s[7];
      t -= 8;
      continue;
    }
    bool done = false;
    int used = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      if (!done && used == k && (s[k] & (RS2_AGG | RS2_INCL))) {
        excl += s[k] & RS2_VAL; used = k + 1;
        if (s[k] & RS2_INCL) done = true;
      }
    }
    if (done) break;
    t -= used;                                             // an unpublished predecessor: fetch again from there
  }
  *mine = RS2_INCL | (excl + count);
  return excl;
}

// REC = Rec16: 16-byte records sorted by .key (WORD 0) or .val (WORD 1); REC = uint64_t: bare 8-byte keys (half the bytes
// per record and pass: the packed seeds of join.cu, WORD ignored).
template <int RS_THREADS, int RS_IPT, int WORD, typename REC>
__global__ void __launch_bounds__(RS_THREADS, 2)
k_rs_pass2(const REC *__restrict__ in, REC *__restrict__ out, uint64_t n, uint32_t shift, uint32_t mask,
           const unsigned long long *__restrict__ digit_base,  // [256] exclusive global offsets
           volatile uint32_t *state,                           // [tiles][256], zero-initialised
           uint32_t *__restrict__ ticket) {
  constexpr int RS_WARPS = RS_THREADS / 32;
  constexpr uint32_t RS_TILE = RS_THREADS * RS_IPT;
  static_assert(RS_THREADS >= 256 && RS_THREADS % 256 == 0, "threads 0..255 own one digit each");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr bool BARE = sizeof(REC) == 8;
  REC *stage = reinterpret_cast<REC *>(smem_raw);                                   // RS_TILE records
  uint32_t *whist = reinterpret_cast<uint32_t *>(smem_raw + RS_TILE * sizeof(REC)); // [RS_WARPS][256]
  __shared__ unsigned long long s_delta[256];
  __shared__ uint32_t s_scan[8];
  __shared__ uint32_t s_tile;

  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // 1. the tile arrives by ONE bulk copy (cp.async.bulk -> mbarrier; SASS UBLKCP) straight into the staging buffer. The
  // first form issued 16 LDG.128 per thread; ptxas interleaved them with the ranking to save registers, so every item
  // waited out a full memory latency on its own (ncu: ~900 stall samples on the first use of each of the 16 loads).
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
    state[(size_t)tile * 256 + tid] = (tile == 0 ? RS2_INCL : RS2_AGG) | real_d;   // successors can start summing while this tile scans
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
    const uint32_t excl = tile ? rs2_look_back(state, tile, tid, real_d) : 0u;
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
