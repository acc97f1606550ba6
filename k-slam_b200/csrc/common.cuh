// common.cuh — internal declarations shared by the CUDA translation units of libkslam.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <exception>
#include <vector>
#include "../../include/kslam.h"

#define KSLAM_NUM_SMS_DEFAULT 148

struct CudaError {
  cudaError_t e; const char *what; const char *file; int line;
};

// thrown by internal stages for inputs the ABI cannot represent; API_END turns it into KSLAM_ERR_ARG
struct ArgError { const char *what; };

#define CUDA_TRY(x)                                                        \
  do {                                                                     \
    cudaError_t e_ = (x);                                                  \
    if (e_ != cudaSuccess) throw CudaError{e_, #x, __FILE__, __LINE__};    \
  } while (0)

// Growable device buffer owned by a ctx; never shrinks (batches have similar sizes).
struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  void reserve(size_t bytes) {
    if (bytes <= cap) return;
    if (p) CUDA_TRY(cudaFree(p));
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    CUDA_TRY(cudaMalloc(&p, want));
    cap = want;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T *as() const { return (T *)p; }
};

// Growable pinned host buffer.
struct HostBuf {
  void *p = nullptr;
  size_t cap = 0;
  void reserve(size_t bytes) {
    if (bytes <= cap) return;
    if (p) CUDA_TRY(cudaFreeHost(p));
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    CUDA_TRY(cudaMallocHost(&p, want));
    cap = want;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
  template <class T> T *as() const { return (T *)p; }
};

// 16-byte record moved by the radix sort: the sort key is `key`, `val` rides along.
// A k-mer record is {key = kMerInt, val = id_flags | offset << 32} == kslam_kmer's memory layout.
struct __align__(16) Rec16 { uint64_t key; uint64_t val; };

// A packed sequence set in HBM (reads of a batch, or the genomes). Sequence i occupies 32-base
// words [word_off[i], word_off[i+1]) of every plane; base b of the word sits at bits 2b..2b+1
// (2-bit planes) / bit b (mask plane).
struct PackedSeqs {
  uint64_t n = 0;          // sequences
  uint64_t n_bases = 0;    // raw bytes
  uint64_t n_words = 0;    // 32-base words
  DevBuf raw;              // u8  raw bytes (transient for reads; dropped for genomes after packing)
  DevBuf offs;             // u64 n+1 raw offsets
  DevBuf word_off;         // u64 n+1 word offsets
  DevBuf kbits;            // u64 per word: k-mer alphabet A0 C1 T2 G3, everything else 0 (KMer.h:246-266)
  DevBuf sbits;            // u64 per word: SSW alphabet A0 C1 G2 T3 (U->0), code-4 bases 0 (ssw_cpp.cpp:11-23)
  DevBuf nmask;            // u32 per word: bit set where the SSW code is 4
  DevBuf xmask;            // u32 per word: bit set for a c g t U u (SSW code < 4 but never complemented)
  DevBuf kmer_off;         // u64 n+1: first k-mer record index of each sequence
  DevBuf has_n;            // u8 per sequence: 1 when it holds a code-4 base anywhere (genomes only; empty otherwise)
  uint64_t n_kmers = 0;
  uint32_t max_len = 0;
  void release() { raw.release(); offs.release(); word_off.release(); kbits.release(); sbits.release();
                   nmask.release(); xmask.release(); kmer_off.release(); has_n.release(); }
};

struct SwWorkspace;

struct kslam_ctx {
  kslam_params prm;
  int device = 0;
  int num_sms = KSLAM_NUM_SMS_DEFAULT;
  cudaStream_t stream = nullptr;
  std::string err;
  bool keep_taps = true;

  PackedSeqs genomes, reads;
  bool genomes_loaded = false, reads_loaded = false, aligned = false, paired = false;
  DevBuf g_keys;   // u64 sorted genome k-mers
  DevBuf g_vals;   // u64 id_flags | offset<<32, same order
  uint64_t n_gk = 0;
  DevBuf bitmap;   // prefilter: 2^filter_bits bits over hashed genome k-mers (kmer.cu)
  uint32_t filter_bits = 0;
  bool prefilter = true;
  bool sw_band64 = true;   // second banded tier (64 diagonals) for what the 32-wide sweep cannot prove
  uint32_t sort_bits = 0;  // leading k-mer bits the read records are sorted on before the join; 0 = auto
  bool sw_tiers = true;    // direct tiers (8 / 16 / 32 / 64 diagonals) picked from the seed-diagonal lower bound
  bool sw_band = true;     // banded SW kernel with exactness proof + full-matrix fallback (sw_band.cuh)
  uint32_t max_genome_len = 0;

  DevBuf recA, recB;        // Rec16 ping-pong (read k-mers, then seeds)
  DevBuf sort_hist;         // radix-sort histograms + look-back state
  DevBuf scan_tmp;
  DevBuf counters;          // small u64 counter block
  HostBuf h_counters;
  HostBuf h_stage;          // pinned staging for ragged-batch offset tables
  bool keep_raw_reads = true;  // keep the raw-byte device buffer between batches (avoids a cudaMalloc per batch)
  uint64_t n_rk = 0;        // read k-mer records
  Rec16 *sorted_rk = nullptr;  // points into recA/recB

  DevBuf raw_seeds;         // kslam_seed (tap) / Rec16 packed seeds
  DevBuf seedA, seedB;      // Rec16 packed seeds ping-pong
  DevBuf seed_keep;         // u8
  DevBuf seeds;             // kslam_seed, de-duplicated, final order
  uint64_t n_raw = 0, n_seeds = 0;
  bool seeds_compact = false;   // seedA holds one-word seeds (join.cu: SeedBits)

  DevBuf ov;                // kslam_overlap[n_seeds]
  DevBuf cig;               // u32[n_seeds * max_cigar_ops]: traceback scratch, fixed stride
  DevBuf cig_dense;         // u32[n_cig_words]: the CIGAR pool that leaves the GPU (dense; cigar_off indexes it)
  uint64_t n_cig_words = 0;
  SwWorkspace *sw = nullptr;
  HostBuf h_ov, h_cig;

  DevBuf pair_keys, pair_keys2, ov_sorted, cig_sorted, pair_cnt, pairs, pairs_compact, far_mates, insert_hist;
  HostBuf h_ov_sorted, h_cig_sorted, h_pairs, h_pairs_compact, h_far_mates, h_insert_hist;
  uint64_t n_sorted = 0, n_pairs = 0;

  // k-mer-range partitioned database (dist.cu, SURVEY.md §8e config 4)
  uint32_t part = 0, n_parts = 1;
  std::vector<uint64_t> splitters;   // n_parts + 1 lower bounds; part p owns keys in [splitters[p], splitters[p+1])
  DevBuf d_bounds;                   // u64[64] bucket bounds on the device (key splitters or read-id bases)
  DevBuf part_send, part_recv, part_tmp, part_m, part_msend, part_mrecv;
  uint64_t n_gk_total = 0;
  float part_ms_bucket = 0, part_ms_bucket_matches = 0;   // device time of the two bucketing steps of the last partitioned batch

  // microbench / Aligner::Align batch
  PackedSeqs swq, swr;
  bool sw_loaded = false;

  kslam_timings tm;
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  uint64_t launches = 0;
};

// ---- helpers implemented across the .cu files ---------------------------------------------
// pack.cu
void pack_sequences(kslam_ctx *c, PackedSeqs &s, uint64_t n, const char *bases, const uint64_t *offs,
                    uint32_t kmer_gap, bool keep_raw);
// kmer.cu
void extract_kmers(kslam_ctx *c, const PackedSeqs &s, bool is_gb, uint32_t gap, Rec16 *out);
void build_prefilter(kslam_ctx *c);
uint64_t extract_read_kmers_filtered(kslam_ctx *c, const PackedSeqs &s, DevBuf &outbuf, uint32_t id_base = 0);
void extract_genome_kmers_range(kslam_ctx *c, const PackedSeqs &s, uint32_t gap, uint64_t i_begin, uint64_t i_stride,
                                uint64_t n_out, Rec16 *out);
// radix_sort.cu
// Sorts n records by bits [lo_bit, hi_bit) of their .key (word 0) or .val (word 1); stable.
// Returns the buffer (a or b) holding the result; *passes_done is incremented per executed pass.
uint64_t *radix_sort_u64(kslam_ctx *c, uint64_t *a, uint64_t *b, uint64_t n, uint32_t lo_bit, uint32_t hi_bit, uint64_t *passes_done);
Rec16 *radix_sort(kslam_ctx *c, Rec16 *a, Rec16 *b, uint64_t n, uint32_t word, uint32_t lo_bit, uint32_t hi_bit,
                  uint64_t *passes_done);
// scan.cu
void exclusive_scan_u32(kslam_ctx *c, const uint32_t *in, uint32_t *out, uint64_t n, uint64_t *total_dev);
// join.cu
void join_and_unique(kslam_ctx *c);
void seed_sort_unique(kslam_ctx *c);
uint64_t run_join(kslam_ctx *c, const Rec16 *R, uint64_t n_r, bool match, DevBuf &outbuf);
void matches_to_seeds(kslam_ctx *c, const Rec16 *m, uint64_t n, uint32_t id_base);
// api.cu: sort an extracted genome k-mer list into the reference's order and split it into g_keys / g_vals
void finish_genome_index(kslam_ctx *c, DevBuf &a, DevBuf &b, uint64_t n);
// sw.cu
void sw_align_seeds(kslam_ctx *c);
void sw_align_pairs(kslam_ctx *c, uint64_t n, kslam_overlap *out_dev, uint32_t *cig_dev);
void sw_workspace_free(kslam_ctx *c);
double sw_measure_int_peak(kslam_ctx *c);
// dist.cu
void part_matches_to_seeds(kslam_ctx *c, uint64_t n_matches, uint32_t read_id_base);
// pair.cu
void pair_overlaps(kslam_ctx *c);
void pairs_compact_device(kslam_ctx *c, kslam_pair_compact *out_dev);
uint64_t far_mates_device(kslam_ctx *c, uint32_t limit, DevBuf &out_buf);
bool insert_hist_device(kslam_ctx *c, const unsigned long long **h_hist, uint32_t *top);

// api.cu: error plumbing of the C ABI (no exception crosses the boundary)
int api_fail(kslam_ctx *c, int code, const std::string &msg);
#define API_BEGIN(ctx)                                                                          \
  if (!(ctx)) return KSLAM_ERR_ARG;                                                            \
  try {                                                                                         \
    if (cudaSetDevice((ctx)->device) != cudaSuccess) return api_fail((ctx), KSLAM_ERR_CUDA, "cudaSetDevice failed");
#define API_END(ctx)                                                                            \
  } catch (const CudaError &e) {                                                                \
    char buf[512];                                                                              \
    snprintf(buf, sizeof buf, "%s:%d: %s: %s", e.file, e.line, e.what, cudaGetErrorString(e.e)); \
    cudaGetLastError();                                                                         \
    return api_fail((ctx), e.e == cudaErrorMemoryAllocation ? KSLAM_ERR_NOMEM : KSLAM_ERR_CUDA, buf); \
  } catch (const ArgError &e) { return api_fail((ctx), KSLAM_ERR_ARG, e.what);                      \
  } catch (const std::exception &e) { return api_fail((ctx), KSLAM_ERR_NOMEM, e.what()); }

// api.cu: read a few words of device memory into PINNED host memory without the copy engine — a one-warp kernel
// stores them through the PCIe mapping of the pinned allocation (UVA). The D2H copy engine is a FIFO: while another
// context on the same GPU drains an 8 GB result buffer, a 4-byte cudaMemcpyAsync counter read waits behind it (measured:
// +0.2 s per config-2 batch when two contexts double-buffer). Enqueues only; the caller synchronises the stream.
void read_small(kslam_ctx *c, void *host_pinned, const void *dev, size_t bytes);

// event-based stage timing
cudaEvent_t tm_mark(kslam_ctx *c);
float tm_ms(cudaEvent_t a, cudaEvent_t b);

// prefilter hash (kmer.cu): position of a k-mer in the 2^bits-bit bitmap of genome k-mers
__device__ __forceinline__ uint64_t kmer_hash(uint64_t k, uint32_t bits) {
  return (k * 0x9E3779B97F4A7C15ull) >> (64 - bits);
}
static inline uint32_t prefilter_bits(uint64_t n_genome_kmers) {
  uint32_t b = 0;
  while (b < 64 && (1ull << b) < n_genome_kmers * 16) b++;
  return b < 26 ? 26 : (b > 34 ? 34 : b);
}

static inline uint32_t ceil_log2_u64_(uint64_t x) { uint32_t b = 0; while (b < 64 && (1ull << b) < x) b++; return b; }
// The merge-join binary-searches every read record inside the genome sub-range its tile covers, so read records only
// have to be GROUPED finely enough for that sub-range to stay small: sorting on the leading log2(genome k-mers) + 2
// bits (rounded up to whole 8-bit digits) leaves < 1 genome key per bucket and halves the radix passes.
static inline uint32_t kmer_sort_bits(const kslam_ctx *c) {
  if (c->sort_bits) return c->sort_bits > 64 ? 64 : c->sort_bits;
  uint32_t b = (ceil_log2_u64_(c->n_gk_total ? c->n_gk_total : 1) + 2 + 7) & ~7u;
  return b < 16 ? 16 : (b > 64 ? 64 : b);
}

static inline uint32_t ceil_log2_u64(uint64_t x) {
  uint32_t b = 0;
  while (b < 64 && (1ull << b) < x) b++;
  return b;
}
