// sam.cu — host stages after pairing, up to the SAM text (host code; SURVEY.md §8f ranks 2-3).
//
// north_star keeps these stages on the host; they are restated here so that the library is a drop-in from FASTQ to SAM
// for the --sam-file run. Every step follows the reference literally, including the order of its (unstable) std::sort
// calls — the same libstdc++ std::sort over the same sequence with the same comparator yields the same permutation,
// which is what makes ties come out as in the reference:
//   getPerReadOverlaps                   /root/reference/src/PairedOverlap.h:437-471
//   getMaxAllowedInsertSize              PairedOverlap.h:314-360   (double arithmetic, same expressions)
//   screenPairedAlignmentsByInsertSize   PairedOverlap.h:396-436   (replace = true: a far pair splits into two singles)
//   screenPairedAlignmentsByScore        PairedOverlap.h:361-390
//   pseudoAssembly                       PairedOverlap.h:480-576   (optional, on by default as in Globals.h:36)
//   getCigarAndMD / SAMEntry / getSAMFromPair / writeSAMOutputPairs / getHeader    SAM.h:101-237,240-534
// Input is exactly what kslam_pair_batch returns plus the batch's reads (ids, bases, qualities: kslam_read_batch) and
// the database entries' bases / locus tags / taxonomy ids / gene tables (XG / XP / XR of GenBank databases).
// kslam_batch_outputs runs the same chain and then hands the per-read records to taxon.cu (LCA, genes; SLAM.h:243-249).
#include "common.cuh"
#include "host_stages.h"
#include <algorithm>
#include <stdexcept>
#include <atomic>
#include <cmath>
#include <climits>
#include <numeric>
#include <string.h>
#include <chrono>
#include <stdlib.h>
#include <malloc.h>
#include <mutex>
#include <thread>
#include <unordered_map>

using namespace kslam_host;

namespace {

// batches smaller than this take the single-threaded form of the stages below (KSLAM_HOST_PAR_MIN: test hook)
size_t par_min() { const char *e = getenv("KSLAM_HOST_PAR_MIN"); return e ? (size_t)strtoull(e, nullptr, 10) : 65536; }

// getPerReadOverlaps, PairedOverlap.h:437-471: consecutive records of one read pair become one ReadPair. The reference walks
// the vector once; here every thread walks a range that starts and ends on a read boundary, the pieces are joined in order.
void per_read_range(const kslam_pairs *in, uint32_t midpoint, uint64_t lo, uint64_t hi, std::vector<ReadPair> &out) {
  ReadPair cur;
  uint32_t readPos = 0;
  for (uint64_t i = lo; i < hi; i++) {
    const kslam_pair &k = in->pairs[i];
    POv p;
    p.combinedScore = k.combined_score; p.entry = k.entry; p.refStart = k.ref_start; p.refEnd = k.ref_end;
    p.insertSize = k.insert_size; p.hasR1 = k.r1_idx >= 0; p.hasR2 = k.r2_idx >= 0; p.r1 = k.r1_idx; p.r2 = k.r2_idx;
    const uint32_t thisReadPos = p.hasR1 ? in->sorted_overlaps[p.r1].read : in->sorted_overlaps[p.r2].read - midpoint;
    if (thisReadPos != readPos) {
      if (cur.pairs.size()) { out.push_back(std::move(cur)); cur.pairs.clear(); }
      readPos = thisReadPos;
    }
    cur.pairs.push_back(p);
    cur.r1Pos = thisReadPos; cur.r2Pos = thisReadPos + midpoint;
  }
  if (cur.pairs.size()) out.push_back(cur);
}
std::vector<ReadPair> per_read(const kslam_pairs *in, uint32_t midpoint, uint32_t threads) {
  std::vector<ReadPair> out;
  const uint64_t n = in->n_pairs;
  if (threads <= 1 || n < par_min() || n < threads) { per_read_range(in, midpoint, 0, n, out); return out; }
  auto read_of = [&](uint64_t i) {
    const kslam_pair &k = in->pairs[i];
    return k.r1_idx >= 0 ? in->sorted_overlaps[k.r1_idx].read : in->sorted_overlaps[k.r2_idx].read - midpoint;
  };
  std::vector<uint64_t> cut(threads + 1, n);
  cut[0] = 0;
  for (uint32_t t = 1; t < threads; t++) {
    uint64_t b = std::max(cut[t - 1], n * t / threads);
    while (b > 0 && b < n && read_of(b) == read_of(b - 1)) b++;      // move to the next read boundary
    cut[t] = b;
  }
  std::vector<std::vector<ReadPair>> parts(threads);
  parallel_threads(threads, [&](uint32_t t) { per_read_range(in, midpoint, cut[t], cut[t + 1], parts[t]); });
  size_t total = 0;
  for (auto &p : parts) total += p.size();
  out.reserve(total);
  for (auto &p : parts) for (auto &r : p) out.push_back(std::move(r));
  return out;
}

// ---- getMaxAllowedInsertSize, PairedOverlap.h:314-360 -------------------------------------------------------------
// The reference sorts every non-zero insert size of the batch and reads order statistics off the sorted vector. What it
// computes is a function of the value COUNTS only, so the batch is kept as a run-length list (value ascending, count,
// cumulative count): order statistics are a binary search, the filtered moments a walk over the runs. The same structure
// can be filled from a histogram computed elsewhere (insert_size_limit_from_runs).
struct InsertRuns {
  std::vector<int32_t> value;      // ascending, distinct
  std::vector<uint64_t> upto;      // upto[k] = number of elements <= value[k]
  uint64_t total() const { return upto.empty() ? 0 : upto.back(); }
  int32_t at(uint64_t rank) const { return value[(size_t)(std::upper_bound(upto.begin(), upto.end(), rank) - upto.begin())]; }
  void push(int32_t v, uint64_t count) { if (count) { value.push_back(v); upto.push_back(total() + count); } }
};

InsertRuns insert_size_runs(const std::vector<ReadPair> &reads) {
  InsertRuns runs;
  int64_t lo = INT64_MAX, hi = INT64_MIN;
  uint64_t n = 0;
  for (auto &read : reads)
    for (auto &p : read.pairs)
      if (p.insertSize != 0) { const int32_t v = (int32_t)p.insertSize; lo = std::min<int64_t>(lo, v); hi = std::max<int64_t>(hi, v); n++; }
  if (!n) return runs;
  if (hi - lo < (1 << 22)) {                               // the normal case (fragment lengths): one counter per value
    std::vector<uint64_t> count((size_t)(hi - lo + 1), 0);
    for (auto &read : reads)
      for (auto &p : read.pairs)
        if (p.insertSize != 0) count[(size_t)((int32_t)p.insertSize - lo)]++;
    for (int64_t v = lo; v <= hi; v++) runs.push((int32_t)v, count[(size_t)(v - lo)]);
  } else {
    std::vector<int32_t> all; all.reserve(n);
    for (auto &read : reads)
      for (auto &p : read.pairs)
        if (p.insertSize != 0) all.push_back((int32_t)p.insertSize);
    std::sort(all.begin(), all.end());
    for (size_t i = 0; i < all.size();) { size_t j = i; while (j < all.size() && all[j] == all[i]) j++; runs.push(all[i], j - i); i = j; }
  }
  return runs;
}

// acc + v + v + ... (count times) exactly as a chain of double additions would give it: while every partial sum is an
// integer below 2^53 the chain is exact, so it collapses into one addition; beyond that the additions are issued one by one
inline double add_repeated(double acc, double v, uint64_t count) {
  const double block = v * (double)count, lim = 9007199254740992.0;
  if (std::fabs(acc) + std::fabs(block) < lim && count < (1ull << 52)) return acc + block;
  while (count--) acc += v;
  return acc;
}

uint32_t insert_size_limit_from_runs(const InsertRuns &runs) {
  const uint64_t n = runs.total();
  if (n == 0) return UINT32_MAX;
  // first percentile step wider than 1000 (:327-333): the percentile positions are floor(n * i / 100.0)
  int32_t spike = 0;
  for (int pc = 0; pc < 99 && !spike; pc++) {
    const int32_t here = runs.at((uint64_t)floor(n * pc / 100.0)), next = runs.at((uint64_t)floor(n * (pc + 1) / 100.0));
    if (next - here > 1000) { spike = runs.at((uint64_t)(n * (uint64_t)pc / 100)); break; }
  }
  const int32_t q1 = runs.at((uint64_t)floor(n * 0.25)), q3 = runs.at((uint64_t)floor(n * 0.75));
  int32_t ceiling = spike ? spike : q3 + 2 * (q3 - q1);
  if (ceiling == 0) ceiling = INT32_MAX;
  // mean and deviation of the values in [0, ceiling], accumulated in ascending order like the reference's accumulate /
  // inner_product over the sorted vector (the square is an int product there, converted afterwards)
  uint64_t kept = 0;
  double sum = 0.0, squares = 0.0;
  for (size_t k = 0; k < runs.value.size(); k++) {
    const int32_t v = runs.value[k];
    if (v < 0 || v > ceiling) continue;
    const uint64_t count = runs.upto[k] - (k ? runs.upto[k - 1] : 0);
    kept += count;
    sum = add_repeated(sum, (double)v, count);
    squares = add_repeated(squares, (double)(int32_t)((uint32_t)v * (uint32_t)v), count);
  }
  const double mean = sum / kept;
  const double sigma = std::sqrt(squares / kept - mean * mean);
  const double bound = floor(mean + 6 * sigma);
  return std::isnan(bound) ? UINT_MAX : (uint32_t)bound;
}

uint32_t max_allowed_insert_size(const std::vector<ReadPair> &reads) { return insert_size_limit_from_runs(insert_size_runs(reads)); }

// the same statistic straight from compact pair records (kslam_pairs_compact): per-thread counters over value ranges
InsertRuns insert_size_runs_compact(const kslam_pair_compact *p, uint64_t n, uint32_t threads) {
  InsertRuns runs;
  constexpr int64_t SPAN = 1 << 22;
  if (threads < 1) threads = 1;
  std::vector<std::vector<uint64_t>> cnt(threads);
  std::vector<std::vector<int32_t>> rest(threads);          // values outside [0, SPAN)
  parallel_ranges(threads, n, [&](uint32_t t, size_t lo, size_t hi) {
    cnt[t].assign(SPAN, 0);
    for (size_t i = lo; i < hi; i++) {
      const int32_t v = (int32_t)p[i].insert_size;
      if (v == 0) continue;
      if (v > 0 && v < SPAN) cnt[t][v]++; else rest[t].push_back(v);
    }
  });
  std::vector<int32_t> other;
  for (auto &r : rest) other.insert(other.end(), r.begin(), r.end());
  std::sort(other.begin(), other.end());
  size_t k = 0;
  auto flush_other = [&](int64_t below) {                   // runs of the sorted out-of-range values smaller than `below`
    while (k < other.size() && other[k] < below) { size_t j = k; while (j < other.size() && other[j] == other[k]) j++; runs.push(other[k], j - k); k = j; }
  };
  flush_other(0);
  for (int64_t v = 1; v < SPAN; v++) {
    uint64_t c = 0;
    for (uint32_t t = 0; t < threads; t++) if (!cnt[t].empty()) c += cnt[t][v];
    runs.push((int32_t)v, c);
  }
  flush_other(INT64_MAX);
  return runs;
}

std::vector<ReadPair> per_read_compact(const kslam_pairs_compact *in, uint32_t midpoint, uint32_t threads) {
  const uint64_t n = in->n_pairs;
  const kslam_pair_compact *rec = in->pairs;
  auto range = [&](uint64_t lo, uint64_t hi, std::vector<ReadPair> &out) {
    ReadPair cur;
    uint32_t readPos = 0;
    for (uint64_t i = lo; i < hi; i++) {
      const kslam_pair_compact &k = rec[i];
      POv p;
      p.combinedScore = k.score_flags & 0x3FFFFFFFu; p.entry = k.entry; p.refStart = k.ref_start; p.refEnd = k.ref_end;
      p.insertSize = k.insert_size; p.hasR1 = (k.score_flags >> 30) & 1u; p.hasR2 = (k.score_flags >> 31) & 1u;
      p.r1 = p.hasR1 ? (int32_t)i : -1; p.r2 = p.hasR2 ? (int32_t)i : -1;           // the PAIR index (Ctx::far is keyed by it)
      if (k.pair_id != readPos) {
        if (cur.pairs.size()) { out.push_back(std::move(cur)); cur.pairs.clear(); }
        readPos = k.pair_id;
      }
      cur.pairs.push_back(p);
      cur.r1Pos = k.pair_id; cur.r2Pos = k.pair_id + midpoint;
    }
    if (cur.pairs.size()) out.push_back(cur);
  };
  std::vector<ReadPair> out;
  if (threads <= 1 || n < par_min() || n < threads) { range(0, n, out); return out; }
  std::vector<uint64_t> cut(threads + 1, n);
  cut[0] = 0;
  for (uint32_t t = 1; t < threads; t++) {
    uint64_t b = std::max(cut[t - 1], n * t / threads);
    while (b > 0 && b < n && rec[b].pair_id == rec[b - 1].pair_id) b++;
    cut[t] = b;
  }
  std::vector<std::vector<ReadPair>> parts(threads);
  parallel_threads(threads, [&](uint32_t t) { range(cut[t], cut[t + 1], parts[t]); });
  size_t total = 0;
  for (auto &pt : parts) total += pt.size();
  out.reserve(total);
  for (auto &pt : parts) for (auto &r : pt) out.push_back(std::move(r));
  return out;
}

// score and reference span of the two alignments of a pair record: from the alignment vector, or (compact input) from the
// far-mates table, which holds every pair the insert-size screen can ask about
struct MatePair { uint32_t s1; int32_t b1, e1; uint32_t s2; int32_t b2, e2; };
inline MatePair mates_of(const Ctx &c, const POv &p) {
  if (c.in) {
    const kslam_overlap &o1 = c.in->sorted_overlaps[p.r1], &o2 = c.in->sorted_overlaps[p.r2];
    return MatePair{o1.sw_score, o1.ref_begin, o1.ref_end, o2.sw_score, o2.ref_begin, o2.ref_end};
  }
  const kslam_far_mates *f = std::lower_bound(c.far, c.far + c.n_far, (uint32_t)p.r1,
                                              [](const kslam_far_mates &x, uint32_t idx) { return x.pair_index < idx; });
  if (f == c.far + c.n_far || f->pair_index != (uint32_t)p.r1) throw std::runtime_error("pair beyond the insert-size limit without its mates");
  return MatePair{f->score1, f->ref_begin1, f->ref_end1, f->score2, f->ref_begin2, f->ref_end2};
}

void screen_by_insert_size(std::vector<ReadPair> &reads, const Ctx &ctx, const uint32_t insertSize, uint32_t threads) {   // :396-436, replace = true
  std::atomic<bool> failed{false};
  parallel_ranges(threads, reads.size(), [&](uint32_t, size_t lo, size_t hi) {
  try {
  for (size_t ri = lo; ri < hi; ri++) {
    ReadPair &read = reads[ri];
    std::sort(read.pairs.begin(), read.pairs.end(), [](const POv &i, const POv &j) { return i.insertSize < j.insertSize; });
    auto cutoff = std::find_if(read.pairs.begin(), read.pairs.end(), [&](const POv &i) { return i.insertSize > insertSize; });
    auto cutoffPos = std::distance(read.pairs.begin(), cutoff);
    read.pairs.reserve(read.pairs.size() + std::distance(cutoff, read.pairs.end()));
    const size_t oldEnd = read.pairs.size();
    for (size_t cur = (size_t)cutoffPos; cur < oldEnd; cur++) {
      const MatePair m = mates_of(ctx, read.pairs[cur]);
      POv single;                                            // the R1 half becomes a pair record of its own
      single.combinedScore = (uint16_t)m.s1; single.entry = read.pairs[cur].entry;
      single.refStart = m.b1; single.refEnd = m.e1; single.insertSize = 0;
      single.hasR1 = true; single.hasR2 = false; single.r1 = read.pairs[cur].r1; single.r2 = -1;
      read.pairs.push_back(single);
      POv &c = read.pairs[cur];                              // ... and the record itself keeps R2 only
      c.combinedScore = (uint16_t)m.s2; c.hasR1 = false; c.insertSize = 0; c.r1 = -1;
      c.refStart = m.b2; c.refEnd = m.e2;
    }
  }
  } catch (const std::exception &) { failed = true; }
  });
  if (failed) throw std::runtime_error("insert-size screen: mates missing");
}

void screen_by_score(std::vector<ReadPair> &reads, double fraction, uint32_t threads) {   // PairedOverlap.h:361-390
  parallel_ranges(threads, reads.size(), [&](uint32_t, size_t lo, size_t hi) {
  for (size_t ri = lo; ri < hi; ri++) {
    ReadPair &read = reads[ri];
    if (read.pairs.size() == 0) continue;
    std::sort(read.pairs.begin(), read.pairs.end(), [](const POv &i, const POv &j) { return i.combinedScore > j.combinedScore; });
    unsigned topScore = read.pairs[0].combinedScore;
    auto cutoff = std::find_if(read.pairs.begin(), read.pairs.end(), [&](const POv &i) { return i.combinedScore < topScore * fraction; });
    read.pairs.erase(cutoff, read.pairs.end());
  }
  });
}

void pseudo_assembly(std::vector<ReadPair> &pairedAlignments, uint32_t threads, uint64_t n_entries) {     // PairedOverlap.h:480-576
  struct coverage { int start = 0; int stop = 0; };
  struct entryAndOverlaps { uint32_t entryPos = 0; std::vector<std::pair<coverage, POv *>> reads; };
  // The reference appends every record to its entry's list while walking the reads in order (an unordered_map keyed by
  // entry). The same lists, in the same order, are built here by all threads: count per (thread range, entry), prefix,
  // fill. Chains never cross entries, so the map's iteration order does not matter.
  std::vector<entryAndOverlaps> lists;
  std::vector<entryAndOverlaps *> entries;
  std::unordered_map<uint32_t, entryAndOverlaps> entriesAndOverlaps;
  const size_t n_reads = pairedAlignments.size();
  if (threads > 1 && n_reads >= par_min() && n_entries * threads <= (16u << 20)) {
    std::vector<std::vector<uint32_t>> cnt(threads, std::vector<uint32_t>(n_entries, 0));
    parallel_threads(threads, [&](uint32_t t) {
      for (size_t r = n_reads * t / threads; r < n_reads * (t + 1) / threads; r++)
        for (auto &overlap : pairedAlignments[r].pairs) cnt[t][overlap.entry]++;
    });
    lists.resize(n_entries);
    for (uint64_t e = 0; e < n_entries; e++) {
      uint32_t total = 0;
      for (uint32_t t = 0; t < threads; t++) { const uint32_t c = cnt[t][e]; cnt[t][e] = total; total += c; }
      lists[e].entryPos = (uint32_t)e;
      lists[e].reads.resize(total);
    }
    parallel_threads(threads, [&](uint32_t t) {
      for (size_t r = n_reads * t / threads; r < n_reads * (t + 1) / threads; r++)
        for (auto &overlap : pairedAlignments[r].pairs) {
          coverage c; c.start = overlap.refStart; c.stop = overlap.refEnd;
          lists[overlap.entry].reads[cnt[t][overlap.entry]++] = {c, &overlap};
        }
    });
    for (auto &l : lists) if (l.reads.size()) entries.push_back(&l);
  } else {
    for (auto &read : pairedAlignments)
      for (auto &overlap : read.pairs) {
        coverage c; c.start = overlap.refStart; c.stop = overlap.refEnd;
        auto &e = entriesAndOverlaps[overlap.entry];
        e.entryPos = overlap.entry;
        e.reads.push_back({c, &overlap});
      }
    for (auto &entry : entriesAndOverlaps) entries.push_back(&entry.second);
  }
  // One entry at a time (they differ a lot in size, so threads take them from a shared counter). Records ordered by start
  // are cut into chains: a record opens a new chain when it starts more than 20 bases before the furthest stop seen so
  // far is reached ... i.e. when start > reach - 20 (PairedOverlap.h:521-573). A chain of two or more records gives all its
  // members the score  (bases / span) * (sum of per-base scores / members) * span,  evaluated in that order in double and
  // truncated on assignment, as the reference does.
  struct Chain {
    size_t first = 0; int reach = -1000000; uint32_t bases = 0; double per_base_sum = 0;
    void open(size_t at, const POv &r, int stop) {
      first = at; reach = stop;
      const int extent = abs(r.refEnd - r.refStart);
      per_base_sum = r.combinedScore * 1.0 / extent; bases = (uint32_t)extent;
    }
    void extend(const POv &r, int stop) {
      if (stop > reach) reach = stop;
      const int extent = abs(r.refEnd - r.refStart);
      per_base_sum += r.combinedScore * 1.0 / extent; bases += (uint32_t)extent;
    }
  };
  std::atomic<size_t> next{0};
  parallel_threads(entries.size() < 2 ? 1u : threads, [&](uint32_t) {
    for (size_t ei = next++; ei < entries.size(); ei = next++) {
      auto &recs = entries[ei]->reads;
      std::sort(recs.begin(), recs.end(),
                [](const std::pair<coverage, POv *> &a, const std::pair<coverage, POv *> &b) { return a.first.start < b.first.start; });
      Chain chain;
      auto close = [&](size_t end) {
        const ptrdiff_t members = (ptrdiff_t)(end - chain.first);
        if (members < 2) return;
        const double span = chain.reach - recs[chain.first].first.start;
        const double depth = chain.bases / span;
        const double mean_per_base = chain.per_base_sum / members;
        const double rescored = depth * mean_per_base * span;
        for (size_t k = chain.first; k < end; k++) recs[k].second->combinedScore = rescored;
      };
      for (size_t k = 0; k < recs.size(); k++) {
        if (recs[k].first.start > chain.reach - 20) { close(k); chain.open(k, *recs[k].second, recs[k].first.stop); }
        else chain.extend(*recs[k].second, recs[k].first.stop);
      }
      close(recs.size());
    }
  });
}

// ---- SAM.h ---------------------------------------------------------------------------------------------------
struct SequenceDifference { std::string cigar, MD; uint32_t NM = 0; double logProbability = 0; };

const std::vector<double> &log_match_table() {           // SAM.h:33-40
  static std::vector<double> table = [] {
    std::vector<double> t;
    t.push_back(std::log10(1.0 - std::pow(10.0, 1.0 / -10.0)));
    for (int i = 1; i < 100; i++) t.push_back(std::log10(1.0 - std::pow(10.0, i / -10.0)));
    return t;
  }();
  return table;
}
const std::vector<double> &log_mismatch_table() {        // SAM.h:41-48
  static std::vector<double> table = [] {
    std::vector<double> t;
    t.push_back(1 / -10.0);
    for (int i = 1; i < 100; i++) t.push_back(i / -10.0);
    return t;
  }();
  return table;
}

// decimal digits of v appended to out (std::to_string without the temporary)
inline void put_uint(std::string &out, uint64_t v) {
  char buf[24]; int n = 0;
  do { buf[n++] = (char)('0' + v % 10); v /= 10; } while (v);
  while (n) out.push_back(buf[--n]);
}
inline void put_int(std::string &out, int64_t v) {
  if (v < 0) { out.push_back('-'); put_uint(out, (uint64_t)(-v)); } else put_uint(out, (uint64_t)v);
}

// getCigarAndMD, SAM.h:101-237. Same walk, same order of the floating-point additions; the reference's temporaries
// (reverse-complemented copy of the read, reversed copy of the qualities, the vector of MD components that is
// concatenated afterwards) are replaced by index arithmetic and a streaming MD writer with the same merging rules:
// consecutive numeric components are summed, a deleted block is "^" + bases, and a mismatch base directly after a
// deleted block is preceded by "0".
// reverseComplement(bases)[p] (sequenceTools.h:83-116: only upper-case A/C/G/T are complemented) as a table walk from the
// read's end — no data-dependent branch on the base
static const struct CompTable { unsigned char t[256]; CompTable() { for (int i = 0; i < 256; i++) t[i] = (unsigned char)i; t['A'] = 'T'; t['T'] = 'A'; t['C'] = 'G'; t['G'] = 'C'; } } kComp;

// The run of matching bases from the current position: how long it is, and the running sum of the per-base log-probabilities
// continued over it. A function of its own (never inlined) so that the sum lives in a register: inside the walk below the
// compiler keeps it in a stack slot because of the calls on the mismatch path, and the chain of dependent additions then
// goes through memory on every base (measured 3.2 instead of 1.5 ns per base).
template <bool RC>
__attribute__((noinline)) double match_run(const char *ref, const unsigned char *qp, const unsigned char *qqp, int left, double acc,
                                           const double *matchTable, int *run_out) {
  constexpr int STEP = RC ? -1 : 1;
  int run = 0;
  while (run < left && ref[run] == (RC ? (char)kComp.t[qp[STEP * run]] : (char)qp[STEP * run])) {
    acc += matchTable[(int)qqp[STEP * run] - 33];
    run++;
  }
  *run_out = run;
  return acc;
}

// The walk for one strand. RC: query[p] = complement(read[len - 1 - p]), quality[p] = qualities[len - 1 - p] — the pointers
// start at the read's end and step backwards.
template <bool RC>
void cigar_and_md_walk(const char *ref, const unsigned char *qp, const unsigned char *qqp, int qlen, const uint32_t *cig,
                       const kslam_overlap &overlap, SequenceDifference &sd) {
  constexpr int STEP = RC ? -1 : 1;
  const double *matchTable = log_match_table().data(), *misMatchTable = log_mismatch_table().data();
  double logp = 0;
  uint32_t nm = 0;
  int refPos = overlap.ref_begin;
  if (overlap.query_begin > 0) {
    put_int(sd.cigar, overlap.query_begin); sd.cigar.push_back('S');
    qp += STEP * overlap.query_begin; qqp += STEP * overlap.query_begin;
  }
  long pending = -1;               // sum of the numeric MD components not yet written
  bool ambiguous = false;
  auto md_number = [&](int v) { pending = pending < 0 ? v : pending + v; };
  auto md_flush = [&]() { if (pending >= 0) { put_uint(sd.MD, (uint64_t)pending); pending = -1; ambiguous = false; } };
  for (uint32_t e = 0; e < overlap.cigar_len; e++) {
    int numMatch = 0;
    const uint32_t length = cig[e] >> 4, operation = cig[e] & 0xf;
    put_uint(sd.cigar, length);
    switch (operation) {
      case 0:
        sd.cigar.push_back('M');
        for (int i = 0; i < (int)length;) {
          int run = 0;
          logp = match_run<RC>(ref + refPos, qp, qqp, (int)length - i, logp, matchTable, &run);
          numMatch += run; refPos += run; qp += STEP * run; qqp += STEP * run; i += run;
          if (i < (int)length) {                           // the base that ended the run is a mismatch
            nm++;
            if (numMatch) md_number(numMatch);
            md_flush();
            if (ambiguous) { sd.MD.push_back('0'); ambiguous = false; }
            sd.MD.push_back(ref[refPos]);
            logp += misMatchTable[(int)*qqp - 33];
            numMatch = 0;
            refPos++; qp += STEP; qqp += STEP; i++;
          }
        }
        if (numMatch) md_number(numMatch);
        break;
      case 1:
        sd.cigar.push_back('I'); nm += length; qp += STEP * (int)length; qqp += STEP * (int)length;
        break;
      case 2:
        sd.cigar.push_back('D');
        md_flush();
        sd.MD.push_back('^');
        for (int i = 0; i < (int)length; i++) { sd.MD.push_back(ref[refPos]); nm++; refPos++; }
        ambiguous = true;
        break;
      default: break;
    }
  }
  md_flush();
  const int end = qlen - overlap.query_end - 1;
  if (end > 0) { put_int(sd.cigar, end); sd.cigar.push_back('S'); }
  sd.NM = nm; sd.logProbability = logp;
}


// (sd is the caller's, reused from alignment to alignment so that its strings keep their capacity)
void cigar_and_md(const Ctx &c, const kslam_overlap &overlap, SequenceDifference &sd) {
  sd.cigar.clear(); sd.MD.clear(); sd.NM = 0; sd.logProbability = 0;
  if (!overlap.cigar_len || !c.in->cigar_pool) return;                                  // Alignment::cigar == nullptr
  const char *ref = c.db->bases + c.db->offs[overlap.entry];
  const unsigned char *rb = (const unsigned char *)c.reads->bases + c.reads->offs[overlap.read];
  const int qlen = (int)(c.reads->offs[overlap.read + 1] - c.reads->offs[overlap.read]);
  const unsigned char *qq = (const unsigned char *)c.reads->quals + c.reads->qual_offs[overlap.read];
  const int qqlen = (int)(c.reads->qual_offs[overlap.read + 1] - c.reads->qual_offs[overlap.read]);
  const uint32_t *cig = c.in->cigar_pool + overlap.cigar_off;
  if (overlap.rev_comp) cigar_and_md_walk<true>(ref, rb + qlen - 1, qq + qqlen - 1, qlen, cig, overlap, sd);
  else cigar_and_md_walk<false>(ref, rb, qq, qlen, cig, overlap, sd);
}

// ---- SAM lines of one read (getSAMFromPair + writeSAMOutputPairs + SAMEntry::getEntry / getFlag, SAM.h:240-517) ------------
// The reference fills two SAMEntry objects per pair record, copies them into a vector and prints them. Here a pair record
// becomes two `Mate`s — what differs between its two lines — in a per-thread scratch that is reused from read to read,
// and each line is composed from those values directly. The rules, restated:
//   * the read's records are taken best combined score first, at most --num-alignments of them (at least one); X0 of a
//     line is the number of TAKEN records that have this mate (:455-466);
//   * an unmapped mate shows its partner's RNAME and POS; with one mapped mate every PNEXT of the record is that mate's
//     POS, with both it is the partner's (:402-417);
//   * FLAG: 0x1 paired data; 0x2 both mates mapped; 0x4 this mate unmapped and its partner mapped; 0x8 the reverse;
//     0x10 this mate reverse-complemented; 0x20 its partner is (only when both are mapped); 0x40 / 0x80 first / second
//     line of paired data; 0x100 every record but the read's first (:373-401, 309-326);
//   * TLEN is the record's refEnd - refStart + 1, with a minus sign on the first line when both mates are mapped and R1
//     does not start before R2, on the second line otherwise (:419-424);
//   * MAPQ = ceil(-10 log10(max(1 - p / sum of p over the read's taken records of that mate, 1e-5))), p = 10 ^ (sum of the
//     per-base log-probabilities of the alignment) (:488-498); an unmapped mate has p = 0;
//   * single-end data: one line per record, RNEXT "*", PNEXT 0, never 0x8 (:425-429);
//   * the line of a mate flagged 0x4 ends after QUAL; SEQ and QUAL are "*" (:282-297).
struct Mate {
  bool mapped = false, rev = false;
  int32_t ref_begin = 0;            // POS - 1
  uint32_t score = 0;               // AS
  std::string_view rname;
  SequenceDifference diff;          // CIGAR, MD, NM and the log-probability (getCigarAndMD)
  double prob = 0;
};
struct RecordLines { Mate mate[2]; const POv *rec = nullptr; const kslam_gene *gene = nullptr; };

static const struct Digits2 { char t[200]; Digits2() { for (int i = 0; i < 100; i++) { t[2 * i] = (char)('0' + i / 10); t[2 * i + 1] = (char)('0' + i % 10); } } } kDigits2;

// raw-pointer writers: a line is composed in place at the end of the output string (the caller has made room)
inline char *w_bytes(char *p, const char *s, size_t n) { memcpy(p, s, n); return p + n; }
inline char *w_view(char *p, std::string_view v) { return w_bytes(p, v.data(), v.size()); }
template <size_t N> inline char *w_lit(char *p, const char (&lit)[N]) { memcpy(p, lit, N - 1); return p + (N - 1); }
inline char *w_uint(char *p, uint64_t v) {                 // two digits per division; most fields have one to four digits
  if (v < 10) { *p = (char)('0' + v); return p + 1; }
  if (v < 100) { memcpy(p, kDigits2.t + 2 * v, 2); return p + 2; }
  char buf[20], *q = buf + 20;
  if (v <= 0xffffffffull) {
    uint32_t w = (uint32_t)v;
    while (w >= 100) { q -= 2; memcpy(q, kDigits2.t + 2 * (w % 100), 2); w /= 100; }
    if (w >= 10) { q -= 2; memcpy(q, kDigits2.t + 2 * w, 2); } else *--q = (char)('0' + w);
  } else {
    while (v >= 100) { q -= 2; memcpy(q, kDigits2.t + 2 * (v % 100), 2); v /= 100; }
    if (v >= 10) { q -= 2; memcpy(q, kDigits2.t + 2 * v, 2); } else *--q = (char)('0' + v);
  }
  const size_t n = (size_t)(buf + 20 - q);
  memcpy(p, q, n);
  return p + n;
}
inline char *w_int(char *p, int64_t v) { if (v < 0) { *p++ = '-'; return w_uint(p, (uint64_t)(-v)); } return w_uint(p, (uint64_t)v); }

// line of mate m of one record; k = the record's rank among the read's taken records
void sam_line(std::string &out, const Ctx &c, const RecordLines &L, int m, size_t k, std::string_view qname, uint32_t hits, uint8_t mapq) {
  const Mate &me = L.mate[m], &partner = L.mate[1 - m];
  const bool paired = c.paired, report_cigar = c.prm->report_cigar != 0;
  const bool both = me.mapped && partner.mapped, ends_early = !me.mapped && partner.mapped;
  const Mate &shown = me.mapped || !partner.mapped ? me : partner;       // whose RNAME / POS this line carries
  unsigned flag = (paired ? 0x1u : 0u) | (both ? 0x2u : 0u) | (ends_early ? 0x4u : 0u) | (me.mapped && me.rev ? 0x10u : 0u) |
                  (both && partner.rev ? 0x20u : 0u) | (paired ? (m == 0 ? 0x40u : 0x80u) : 0u) | (k != 0 ? 0x100u : 0u);
  if (me.mapped && !partner.mapped && (paired || m != 0)) flag |= 0x8u;
  const uint32_t pos = (uint32_t)(shown.ref_begin + 1);
  uint32_t pnext = both ? (uint32_t)(partner.ref_begin + 1) : pos;
  int32_t tlen = me.mapped || partner.mapped ? L.rec->refEnd - L.rec->refStart + 1 : 0;
  if (both && !(L.mate[0].ref_begin < L.mate[1].ref_begin)) tlen *= -1;
  if (m == 1) tlen *= -1;
  const bool star_next = !paired && m == 0;
  if (star_next) pnext = 0;
  std::string_view xg, xp, xr;
  if (L.gene) { xg = gene_str(c.db, L.gene, GENE_NAME); xp = gene_str(c.db, L.gene, GENE_PROTEIN); xr = gene_str(c.db, L.gene, GENE_PRODUCT); }
  // one bounds check per line instead of one per field: 13 numbers of at most 20 digits + ~70 bytes of literals + the strings
  const size_t bound = qname.size() + shown.rname.size() + me.diff.cigar.size() + me.diff.MD.size() + xg.size() + xp.size() + xr.size() + 400;
  const size_t old = out.size();
  if (out.capacity() < old + bound) out.reserve(std::max(out.capacity() * 2, old + bound));
  out.resize(old + bound);
  char *p = &out[old];
  p = w_view(p, qname); *p++ = '\t'; p = w_uint(p, flag); *p++ = '\t';
  p = w_view(p, shown.rname); *p++ = '\t'; p = w_uint(p, pos); *p++ = '\t'; p = w_uint(p, mapq); *p++ = '\t';
  if (report_cigar && me.mapped) p = w_view(p, me.diff.cigar); else *p++ = '*';
  *p++ = '\t'; *p++ = star_next ? '*' : '='; *p++ = '\t'; p = w_uint(p, pnext); *p++ = '\t'; p = w_int(p, tlen);
  p = w_lit(p, "\t*\t*");
  if (!ends_early) {
    if (report_cigar) { p = w_lit(p, "\tMD:Z:"); if (me.mapped) p = w_view(p, me.diff.MD); }
    p = w_lit(p, "\tAS:i:"); p = w_uint(p, me.mapped ? (uint16_t)me.score : 0u);
    p = w_lit(p, "\tXS:i:"); p = w_uint(p, (uint16_t)L.rec->combinedScore);
    p = w_lit(p, "\tNM:i:"); p = w_uint(p, me.mapped ? me.diff.NM : 0u);
    p = w_lit(p, "\tX0:i:"); p = w_uint(p, hits);
    const uint32_t tax = c.db->taxonomy_ids ? c.db->taxonomy_ids[L.rec->entry] : 0;
    if (tax != 0) { p = w_lit(p, "\tXT:i:"); p = w_uint(p, tax); }
    if (xg.size()) { p = w_lit(p, "\tXG:Z:"); p = w_view(p, xg); }
    if (xp.size()) { p = w_lit(p, "\tXP:Z:"); p = w_view(p, xp); }
    if (xr.size()) { p = w_lit(p, "\tXR:Z:\""); p = w_view(p, xr); *p++ = '"'; }
  }
  *p++ = '\n';
  out.resize((size_t)(p - out.data()));
}

void write_pairs(std::string &out, const Ctx &c, ReadPair &read) {
  // best combined score first, IN PLACE as in the reference: the taxonomy stage that follows sees the records in this order
  // (SLAM.h:235-246), and where std::sort leaves equal scores is part of the output
  std::sort(read.pairs.begin(), read.pairs.end(), [](const POv &i, const POv &j) { return i.combinedScore > j.combinedScore; });
  const size_t n = std::min<size_t>(read.pairs.size(), std::max<uint32_t>(1u, c.prm->num_alignments));
  if (n == 0) return;                                      // (the reference would dereference begin() of an empty vector here)
  static thread_local std::vector<RecordLines> scratch;
  if (scratch.size() < n) scratch.resize(n);
  const kslam_overlap *ov = c.in->sorted_overlaps;
  uint32_t hits[2] = {0, 0};
  double prob_sum[2] = {0, 0};
  for (size_t k = 0; k < n; k++) {
    const POv &rec = read.pairs[k];
    RecordLines &L = scratch[k];
    L.rec = &rec;
    L.gene = best_gene(c.db, rec.entry, rec.refStart, rec.refEnd);                       // SAM.h:361-370
    for (int m = 0; m < 2; m++) {
      Mate &mate = L.mate[m];
      mate.mapped = m == 0 ? rec.hasR1 : rec.hasR2;
      if (!mate.mapped) { mate.rev = false; mate.ref_begin = -1; mate.score = 0; mate.rname = std::string_view(); mate.prob = 0; continue; }
      const kslam_overlap &o = ov[m == 0 ? rec.r1 : rec.r2];
      hits[m]++;
      cigar_and_md(c, o, mate.diff);
      mate.prob = std::pow(10, mate.diff.logProbability);
      mate.rev = o.rev_comp != 0; mate.ref_begin = o.ref_begin; mate.score = o.sw_score;
      mate.rname = std::string_view(c.db->locus_tags + c.db->locus_offs[o.entry], (size_t)(c.db->locus_offs[o.entry + 1] - c.db->locus_offs[o.entry]));
    }
    prob_sum[0] += L.mate[0].prob; prob_sum[1] += L.mate[1].prob;                        // in record order (:474-475)
  }
  auto id_view = [&](uint32_t i) { return std::string_view(c.reads->ids + c.reads->id_offs[i], (size_t)(c.reads->id_offs[i + 1] - c.reads->id_offs[i])); };
  const std::string_view qname[2] = {id_view(read.r1Pos), c.paired ? id_view(read.r2Pos) : std::string_view()};
  const int lines_per_record = c.paired ? 2 : 1;
  for (size_t k = 0; k < n; k++) {
    for (int m = 0; m < lines_per_record; m++) {
      double miss = 1.0 - scratch[k].mate[m].prob / prob_sum[m];
      if (miss <= 0.00001) miss = 0.00001;
      const uint8_t mapq = ceil(-10.0 * std::log10(miss));
      sam_line(out, c, scratch[k], m, k, qname[m], hits[m], mapq);
    }
    if (c.prm->sam_xa) break;
  }
}

}  // namespace

char *kslam_host::dup_text(const std::string &s) {
  char *p = (char *)malloc(s.size() + 1);
  if (!p) return nullptr;
  memcpy(p, s.data(), s.size()); p[s.size()] = 0;
  return p;
}

extern "C" {

int kslam_sam_header(const kslam_sam_db *db, const char *command_line, char **text, uint64_t *len) {   // SAM.h:518-531
  if (!db || !text) return KSLAM_ERR_ARG;
  std::string h = "@HD\tVN:1.0\tSO:unsorted\n";
  for (uint64_t e = 0; e < db->n_entries; e++) {
    h += "@SQ\tSN:";
    h.append(db->locus_tags + db->locus_offs[e], db->locus_tags + db->locus_offs[e + 1]);
    h += "\tLN:";
    h += std::to_string(db->offs[e + 1] - db->offs[e]);
    if (db->taxonomy_ids && db->taxonomy_ids[e]) { h += "\tSP:"; h += std::to_string(db->taxonomy_ids[e]); }
    h += "\n";
  }
  h += "@PG\tID:SLAM\tPN:SLAM\tVN:1.0\tCL:\"";
  h += command_line ? command_line : "";
  h += "\"\n";
  *text = dup_text(h);
  if (len) *len = h.size();
  return *text ? KSLAM_OK : KSLAM_ERR_NOMEM;
}

// Text buffers are recycled from batch to batch. A 10 M-pair batch writes ~2 GB of SAM text, first into one string per
// thread, then into the buffer handed to the caller; taken fresh from malloc every batch, each of those pages is faulted in
// (and zeroed) again, which costs more than writing the text. The pool keeps the per-thread strings (emptied, capacity
// kept) and the one largest buffer given back through kslam_sam_free; a second writer running at the same time simply
// allocates.
struct TextPool {
  std::mutex m;
  std::vector<std::string> parts;
  char *buf = nullptr; size_t cap = 0;
  ~TextPool() { free(buf); }
  std::vector<std::string> take_parts(uint32_t threads) {
    std::vector<std::string> p;
    { std::lock_guard<std::mutex> l(m); p.swap(parts); }
    p.resize(threads);                                       // (a different thread count keeps what fits)
    return p;
  }
  void give_parts(std::vector<std::string> &p) {
    for (std::string &x : p) x.clear();
    std::lock_guard<std::mutex> l(m);
    if (parts.empty()) parts.swap(p);
  }
  char *take_buf(size_t bytes) {
    {
      std::lock_guard<std::mutex> l(m);
      if (buf && cap >= bytes) { char *b = buf; buf = nullptr; cap = 0; return b; }
    }
    return (char *)malloc(bytes);
  }
  void give_buf(char *b) {
    if (!b) return;
    const size_t have = malloc_usable_size(b);
    if (have >= (1u << 20)) {                                // small texts (headers) are not worth keeping
      std::lock_guard<std::mutex> l(m);
      if (have > cap) { std::swap(b, buf); cap = have; }
    }
    free(b);
  }
};
static TextPool &text_pool() { static TextPool p; return p; }

// everything after the per-read grouping: screens, pseudo-assembly, records, text (shared by paired and single-end input);
// with a taxonomy database the per-read records then go to taxon.cu, after the SAM records exactly as in the batch loop
// (writeSAMOutputPairs re-sorts every read's records in place before the taxonomy step sees them, SLAM.h:235-246)
static int sam_finish(Ctx &c, std::vector<ReadPair> &rp, bool insert_screen, bool want_sam, char **text, uint64_t *len, uint32_t *max_insert_size,
                      const kslam_taxdb *taxdb, kslam_taxa *taxa) {
  const kslam_sam_params *prm = c.prm;
  const bool trace = getenv("KSLAM_SAM_TRACE") != nullptr;
  auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  double t1 = now();
  uint32_t threads = prm->threads ? prm->threads : std::max(1u, std::thread::hardware_concurrency());
  if (threads > 64) threads = 64;
  if (insert_screen) {
    const uint32_t maxInsert = max_allowed_insert_size(rp);
    if (max_insert_size) *max_insert_size = maxInsert;
    screen_by_insert_size(rp, c, maxInsert, threads);
  } else if (max_insert_size) *max_insert_size = UINT32_MAX;
  double t2 = now();
  screen_by_score(rp, prm->score_fraction_threshold, threads);
  if (prm->pseudo_assembly) { pseudo_assembly(rp, threads, c.db->n_entries); screen_by_score(rp, prm->score_fraction_threshold, threads); }
  double t3 = now();
  int rc = KSLAM_OK;
  if (want_sam) {
    std::vector<std::string> parts = text_pool().take_parts(threads);
    // Every alignment reads ~150 reference bases at an unrelated place of the database: three cache lines that are never
    // in cache. They are requested a few read pairs ahead of their use.
    auto prefetch_windows = [&](const ReadPair &read) {
      size_t k = 0;
      for (const POv &ap : read.pairs) {
        for (int32_t idx : {ap.r1, ap.r2}) {
          if (idx < 0) continue;
          const kslam_overlap &o = c.in->sorted_overlaps[idx];
          const char *w = c.db->bases + c.db->offs[o.entry] + o.ref_begin;
          __builtin_prefetch(w); __builtin_prefetch(w + 64); __builtin_prefetch(w + 128);
        }
        if (++k >= prm->num_alignments) break;
      }
    };
    parallel_ranges(threads, rp.size(), [&](uint32_t t, size_t lo, size_t hi) {
      constexpr size_t AHEAD = 4;
      parts[t].reserve((hi - lo) * 2 * 128);             // about two short lines per read pair: most of the growth (and its page faults) up front
      for (size_t i = lo; i < std::min(hi, lo + AHEAD); i++) prefetch_windows(rp[i]);
      for (size_t i = lo; i < hi; i++) {
        if (i + AHEAD < hi) prefetch_windows(rp[i + AHEAD]);
        write_pairs(parts[t], c, rp[i]);
      }
    });
    const double t_lines = now();
    size_t total = 0;
    std::vector<size_t> at(threads + 1, 0);
    for (uint32_t t = 0; t < threads; t++) { at[t] = total; total += parts[t].size(); }
    char *buf = text_pool().take_buf(total + 1);                // the threads' pieces go straight into the result buffer
    if (buf) {
      parallel_threads(threads, [&](uint32_t t) { memcpy(buf + at[t], parts[t].data(), parts[t].size()); });
      buf[total] = 0;
    }
    *text = buf;
    if (len) *len = total;
    if (!buf) rc = KSLAM_ERR_NOMEM;
    text_pool().give_parts(parts);
    if (trace) fprintf(stderr, "[kslam_sam] lines %.1f ms, joined into one buffer %.1f ms\n", (t_lines - t3) * 1e3, (now() - t_lines) * 1e3);
  } else {
    if (text) *text = nullptr;
    if (len) *len = 0;
  }
  double t4 = now();
  if (rc == KSLAM_OK && taxdb && taxa) rc = taxa_add_batch(taxa, taxdb, c, rp, threads);
  if (trace) fprintf(stderr, "[kslam_sam] insert limit + screen %.1f ms, score screens + assembly %.1f ms, records %.1f ms (incl. concat), taxonomy %.1f ms, %u threads\n",
                     (t2 - t1) * 1e3, (t3 - t2) * 1e3, (t4 - t3) * 1e3, (now() - t4) * 1e3, threads);
  return rc;
}

static int check_overlaps(const kslam_sam_db *db, const kslam_read_batch *reads, const kslam_overlap *ov, uint64_t n, const uint32_t *pool,
                          uint64_t n_pool) {
  // the records index each other and the read / entry arrays: refuse anything out of range instead of reading past a buffer
  uint64_t undefined = 0;
  for (uint64_t i = 0; i < n; i++) {
    const kslam_overlap &o = ov[i];
    if (o.read >= reads->n_reads || o.entry >= db->n_entries) return KSLAM_ERR_ARG;
    if (o.cigar_len && pool && (uint64_t)o.cigar_off + o.cigar_len > n_pool) return KSLAM_ERR_ARG;
    // A truncated CIGAR would give a wrong CIGAR / MD / NM without any sign of it. kslam_align_batch raises the pool stride
    // until nothing overflows, so this only fires for records a caller built with a fixed pool (kslam_ssw_batch).
    if (pool && (o.flags & KSLAM_FLAG_CIGAR_OVERFLOW)) {
      fprintf(stderr, "kslam: alignment %llu carries a truncated CIGAR (KSLAM_FLAG_CIGAR_OVERFLOW): raise max_cigar_ops\n", (unsigned long long)i);
      return KSLAM_ERR_STATE;
    }
    undefined += (o.flags & KSLAM_FLAG_UNDEFINED) != 0;
  }
  if (undefined)
    fprintf(stderr, "kslam: warning: %llu alignments are outside the reference's defined behaviour (score 0 with a CIGAR requested, or a "
                    "traceback leaving its band); their records carry no CIGAR\n", (unsigned long long)undefined);
  return KSLAM_OK;
}

int kslam_sam_batch(const kslam_sam_params *prm, const kslam_sam_db *db, const kslam_read_batch *reads, const kslam_pairs *pairs,
                    char **text, uint64_t *len, uint32_t *max_insert_size) {
  return kslam_batch_outputs(prm, db, reads, pairs, 1, text, len, max_insert_size, nullptr, nullptr);
}

int kslam_batch_outputs(const kslam_sam_params *prm, const kslam_sam_db *db, const kslam_read_batch *reads, const kslam_pairs *pairs,
                        int want_sam, char **text, uint64_t *len, uint32_t *max_insert_size, const kslam_taxdb *taxdb, kslam_taxa *taxa) {
  if (!prm || !db || !reads || !pairs || (want_sam && !text) || ((taxdb != nullptr) != (taxa != nullptr))) return KSLAM_ERR_ARG;
  if ((db->genes != nullptr) != (db->gene_offs != nullptr) || (db->genes && !db->gene_strings)) return KSLAM_ERR_ARG;
  if (pairs->n_pairs && (!pairs->pairs || !pairs->sorted_overlaps)) return KSLAM_ERR_ARG;
  if (int rc = check_overlaps(db, reads, pairs->sorted_overlaps, pairs->n_sorted, pairs->cigar_pool, pairs->n_cigar_words)) return rc;
  for (uint64_t i = 0; i < pairs->n_pairs; i++) {
    const kslam_pair &k = pairs->pairs[i];
    if ((k.r1_idx < 0 && k.r2_idx < 0) || k.r1_idx >= (int64_t)pairs->n_sorted || k.r2_idx >= (int64_t)pairs->n_sorted ||
        k.entry >= db->n_entries) return KSLAM_ERR_ARG;
  }
  try {
    Ctx c{prm, db, reads, pairs, true};
    uint32_t threads = prm->threads ? prm->threads : std::max(1u, std::thread::hardware_concurrency());
    const bool trace = getenv("KSLAM_SAM_TRACE") != nullptr;
    auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t0 = now();
    int rc;
    double t1, t2;
    {
      auto rp = per_read(pairs, (uint32_t)(reads->n_reads / 2), std::min(threads, 64u));
      t1 = now();
      rc = sam_finish(c, rp, true, want_sam != 0, text, len, max_insert_size, taxdb, taxa);
      t2 = now();
      // one small heap block per read pair: give them back on all threads instead of in the vector's destructor
      parallel_ranges(std::min(threads, 64u), rp.size(), [&](uint32_t, size_t lo, size_t hi) {
        for (size_t i = lo; i < hi; i++) std::vector<POv>().swap(rp[i].pairs);
      });
    }
    if (trace) fprintf(stderr, "[kslam_sam] grouping %.1f ms, stages %.1f ms, release %.1f ms\n", (t1 - t0) * 1e3, (t2 - t1) * 1e3, (now() - t2) * 1e3);
    return rc;
  } catch (const std::exception &) { return KSLAM_ERR_NOMEM; }
}

// the same from value counts: counts[v] = number of pair records with insert size v, v = 0 .. top (counts[0] is ignored:
// single-ended records carry insert size 0 and never enter the statistic, PairedOverlap.h:321)
uint32_t kslam_insert_size_limit_counts(const uint64_t *counts, uint32_t top) {
  if (!counts) return UINT32_MAX;
  try {
    InsertRuns runs;
    for (uint32_t v = 1; v <= top; v++) runs.push((int32_t)v, counts[v]);
    return insert_size_limit_from_runs(runs);
  } catch (const std::exception &) { return UINT32_MAX; }
}

uint32_t kslam_insert_size_limit_compact(const kslam_pair_compact *pairs, uint64_t n, uint32_t host_threads) {
  if (!pairs || !n) return UINT32_MAX;
  uint32_t threads = host_threads ? host_threads : std::max(1u, std::thread::hardware_concurrency());
  if (threads > 16) threads = 16;                           // 32 MB of counters per thread
  if (n < (1u << 20)) threads = 1;
  try { return insert_size_limit_from_runs(insert_size_runs_compact(pairs, n, threads)); } catch (const std::exception &) { return UINT32_MAX; }
}

int kslam_batch_outputs_compact(const kslam_sam_params *prm, const kslam_sam_db *db, const kslam_read_batch *reads, const kslam_pairs_compact *in,
                                uint32_t *max_insert_size, const kslam_taxdb *taxdb, kslam_taxa *taxa) {
  if (!prm || !db || !reads || !in || ((taxdb != nullptr) != (taxa != nullptr))) return KSLAM_ERR_ARG;
  if ((db->genes != nullptr) != (db->gene_offs != nullptr) || (db->genes && !db->gene_strings)) return KSLAM_ERR_ARG;
  if ((in->n_pairs && !in->pairs) || (in->n_far && !in->far)) return KSLAM_ERR_ARG;
  const uint32_t mid = (uint32_t)(reads->n_reads / 2);
  for (uint64_t i = 0; i < in->n_pairs; i++)
    if (in->pairs[i].entry >= db->n_entries || in->pairs[i].pair_id >= mid) return KSLAM_ERR_ARG;
  try {
    Ctx c{prm, db, reads, nullptr, true};
    c.far = in->far; c.n_far = in->n_far;
    const uint32_t threads = std::min(prm->threads ? (uint32_t)prm->threads : std::max(1u, std::thread::hardware_concurrency()), 64u);
    auto rp = per_read_compact(in, mid, threads);
    uint32_t limit = 0;
    int rc = sam_finish(c, rp, true, false, nullptr, nullptr, &limit, taxdb, taxa);
    if (rc == KSLAM_OK && limit != in->insert_size_limit) rc = KSLAM_ERR_STATE;   // the far-mates table was fetched for another limit
    if (max_insert_size) *max_insert_size = limit;
    parallel_ranges(threads, rp.size(), [&](uint32_t, size_t lo, size_t hi) {
      for (size_t i = lo; i < hi; i++) std::vector<POv>().swap(rp[i].pairs);
    });
    return rc;
  } catch (const std::exception &) { return KSLAM_ERR_STATE; }
}

// Single-end reads (SLAM.h:223-228): alignToDatabase's vector, score screen (Overlap.h:329-341), getPerReadOverlaps
// (Overlap.h:302-327), one R1-only dummy pair per overlap (getDummyAlignmentPairsFromSingleEndReads, PairedOverlap.h:280-298),
// then the same screens / pseudo-assembly / records with pairedData = false (one line per alignment, no mate fields).
int kslam_sam_batch_single(const kslam_sam_params *prm, const kslam_sam_db *db, const kslam_read_batch *reads,
                           const kslam_alignments *al, uint32_t score_threshold, char **text, uint64_t *len) {
  return kslam_batch_outputs_single(prm, db, reads, al, score_threshold, 1, text, len, nullptr, nullptr);
}

int kslam_batch_outputs_single(const kslam_sam_params *prm, const kslam_sam_db *db, const kslam_read_batch *reads, const kslam_alignments *al,
                               uint32_t score_threshold, int want_sam, char **text, uint64_t *len, const kslam_taxdb *taxdb, kslam_taxa *taxa) {
  if (!prm || !db || !reads || !al || (want_sam && !text) || ((taxdb != nullptr) != (taxa != nullptr))) return KSLAM_ERR_ARG;
  if ((db->genes != nullptr) != (db->gene_offs != nullptr) || (db->genes && !db->gene_strings)) return KSLAM_ERR_ARG;
  if (al->n_overlaps && !al->overlaps) return KSLAM_ERR_ARG;
  if (int rc = check_overlaps(db, reads, al->overlaps, al->n_overlaps, al->cigar_pool, al->n_cigar_words)) return rc;
  try {
    kslam_pairs view;
    memset(&view, 0, sizeof view);
    view.sorted_overlaps = al->overlaps; view.n_sorted = al->n_overlaps;
    view.cigar_pool = al->cigar_pool; view.n_cigar_words = al->n_cigar_words;
    Ctx c{prm, db, reads, &view, false};
    std::vector<ReadPair> rp;
    ReadPair cur;
    uint32_t readPos = 0;
    for (uint64_t i = 0; i < al->n_overlaps; i++) {
      const kslam_overlap &o = al->overlaps[i];
      if (o.sw_score < score_threshold) continue;             // screenOverlapsByScoreThreshold
      if (o.read != readPos) {
        if (cur.pairs.size()) { rp.push_back(std::move(cur)); cur.pairs.clear(); }
        readPos = o.read;
      }
      POv p;
      p.combinedScore = (uint16_t)o.sw_score; p.entry = o.entry; p.refStart = o.ref_begin; p.refEnd = o.ref_end;
      p.insertSize = 0; p.hasR1 = true; p.hasR2 = false; p.r1 = (int32_t)i; p.r2 = -1;
      cur.pairs.push_back(p);
      cur.r1Pos = o.read; cur.r2Pos = 0;
    }
    if (cur.pairs.size()) rp.push_back(cur);
    return sam_finish(c, rp, false, want_sam != 0, text, len, nullptr, taxdb, taxa);
  } catch (const std::exception &) { return KSLAM_ERR_NOMEM; }
}

void kslam_sam_free(char *text) { text_pool().give_buf(text); }

}  // extern "C"
