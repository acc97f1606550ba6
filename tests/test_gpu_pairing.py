"""The pairing stage (K9, csrc/pair.cu) and the compact pair results where their code paths switch.

The reference for K9 alone takes the GPU's own unsorted alignments (other tests pin those to the oracle), orders the ones
that pass the score threshold by (read % mid, entry, rel, read) with a stable sort, so equal keys keep input order, and runs
the oracle's getPairsFromRead restatement (ko_pair_overlaps) on that order. That lets it check batches of millions of
alignments; T.ko_pipeline checks the small batches end to end. Every case asserts that its data reaches the switch it is
meant for: the merge-path split over several CTAs and the tile edges (PM_TILE = 1024 outputs per tile), empty R1 or R2
lists, ties between the lists, the scan's carry loop (more than 2^21 inputs), odd read counts, the insert-size histogram's
global-memory counts (values in [4096, 2^22)) and its host fallback (values >= 2^22)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PM_TILE = 1024
SCAN_ONE_PASS = 1024 * 2048          # k_scan_tiles carries across passes beyond this many inputs
HIST_LOW, HIST_SPAN = 4096, 1 << 22
NO_LIMIT = 0xFFFFFFFF
FIELDS = ("read", "entry", "rel", "rev_comp", "ref_begin", "ref_end", "query_begin", "query_end", "sw_score", "cigar_len", "flags")
ACGT = np.frombuffer(b"ACGT", np.uint8)
COMP = np.arange(256, dtype=np.uint8)
COMP[list(b"ACGT")] = list(b"TGCA")


# ---------------------------------------------------------------- references and comparisons

def k9_reference(T, ov, read_offs, thr):
    """screen + getPairedOverlaps on the alignment vector `ov` -> (pair-sorted overlaps, pair records)"""
    mid = (len(read_offs) - 1) // 2
    kept = ov[ov["sw_score"] >= thr]
    srt = np.ascontiguousarray(kept[np.lexsort((kept["read"], kept["rel"], kept["entry"], kept["read"] % np.uint32(mid)))])
    lens = np.ascontiguousarray(np.diff(read_offs), dtype=np.uint32)
    L = T.oracle()
    cnt = L.ko_pair_overlaps(srt.ctypes.data, len(srt), mid, lens.ctypes.data, None)
    pairs = np.zeros(cnt, dtype=T.PAIR_DT)
    L.ko_pair_overlaps(srt.ctypes.data, len(srt), mid, lens.ctypes.data, pairs.ctypes.data)
    return srt, pairs


def first_diff(got, want, fields):
    for f in fields:
        if not np.array_equal(got[f], want[f]):
            i = int(np.flatnonzero(got[f] != want[f])[0])
            return f"record {i} differs in {f}: got {got[i]}, want {want[i]}"
    return None


def assert_pairs(T, got, want_sorted, want_pool, want_pairs, cigars=False):
    assert len(got.sorted_overlaps) == len(want_sorted), f"n_sorted {len(got.sorted_overlaps)} != {len(want_sorted)}"
    msg = first_diff(got.sorted_overlaps, want_sorted, FIELDS)
    assert msg is None, "sorted_overlaps: " + msg
    if cigars:
        assert T.cigars_of(got.sorted_overlaps, got.cigar_pool) == T.cigars_of(want_sorted, want_pool)
    assert len(got.pairs) == len(want_pairs), f"n_pairs {len(got.pairs)} != {len(want_pairs)}"
    msg = first_diff(got.pairs, want_pairs, want_pairs.dtype.names)
    assert msg is None, "pairs: " + msg


def align_and_pair(T, al, rb, ro, thr, cigars=False):
    """align_batch + pair_batch on `al` (created with score_threshold=thr), checked against the K9 reference"""
    a = al.align_batch(rb, ro)
    got = al.pair_batch(fetch=True)
    srt, pairs = k9_reference(T, a.overlaps, ro, thr)
    assert_pairs(T, got, srt, a.cigar_pool, pairs, cigars)
    return a, got


def far_host(pkg, full, limit):
    """the mates of the pair records with insert_size > limit, in pair order (what kslam_fetch_far_mates returns)"""
    pr, ov = full.pairs, full.sorted_overlaps
    sel = np.flatnonzero(pr["insert_size"] > np.uint32(limit))
    far = np.zeros(len(sel), dtype=pkg.FAR_MATES_DT)
    far["pair_index"] = sel
    a, b = ov[pr["r1_idx"][sel]], ov[pr["r2_idx"][sel]]
    far["score1"], far["ref_begin1"], far["ref_end1"] = a["sw_score"], a["ref_begin"], a["ref_end"]
    far["score2"], far["ref_begin2"], far["ref_end2"] = b["sw_score"], b["ref_begin"], b["ref_end"]
    return far


def threshold_dropping(ov, frac):
    """a score threshold that drops about `frac` of the alignments (and at least one)"""
    sc = np.sort(ov["sw_score"])
    return int(sc[int(len(sc) * frac)]) or 1


# ---------------------------------------------------------------- read builders

def mutate(rng, s, rate=0.01):
    s = s.copy()
    m = rng.random(len(s)) < rate
    s[m] = ACGT[(np.searchsorted(ACGT, s[m]) + rng.integers(1, 4, int(m.sum()))) % 4]
    return s


def rc(s):
    return COMP[s[::-1]]


def fragment_pair(rng, g, p, l1, l2, frag, swap):
    """R1 = g[p:p+l1], R2 = revcomp(g[p+frag-l2:p+frag]) (lightly mutated), mates swapped when `swap`"""
    a = mutate(rng, g[p:p + l1]); b = rc(mutate(rng, g[p + frag - l2:p + frag]))
    return (b, a) if swap else (a, b)


def reads_of(r1, r2, extra=()):
    seqs = list(r1) + list(r2) + list(extra)
    offs = np.zeros(len(seqs) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(s) for s in seqs])
    return np.concatenate(seqs), offs


def shorten(rb, ro, cut, keep_len=20):
    """reads with cut[i] keep their first `keep_len` bases: no k-mer, so no alignment; every other read is unchanged"""
    lens = np.diff(ro).astype(np.int64)
    new = np.where(cut, np.minimum(lens, keep_len), lens)
    offs = np.zeros(len(ro), dtype=np.int64)
    offs[1:] = np.cumsum(new)
    idx = np.arange(offs[-1]) + np.repeat(ro[:-1].astype(np.int64) - offs[:-1], new)
    return rb[idx], offs.astype(np.uint64)


def reads_for_count(rng, cnt, target):
    """which reads to keep at full length so that exactly `target` passing alignments remain (alignments are per read);
    reads without passing alignments are always kept"""
    multi, ones = rng.permutation(np.flatnonzero(cnt > 1)), rng.permutation(np.flatnonzero(cnt == 1))
    cs = np.cumsum(cnt[multi])
    k = int(np.searchsorted(cs, target, side="right"))
    rest = target - (int(cs[k - 1]) if k else 0)
    assert rest <= len(ones)
    keep = cnt == 0
    keep[multi[:k]] = True
    keep[ones[:rest]] = True
    return keep


# ---------------------------------------------------------------- 1. tile edges

def test_tile_edges(pkg, T):
    """n_sorted exactly 1, 1023, 1024, 1025, 262144 and 262145, at threshold 0 and above: the merge's first and last tiles,
    and a k_pair_split grid of more than one CTA (257 tile boundaries from 262144 on)"""
    gb, go = pkg.synth.random_genomes(4, 250_000, seed=101)
    rb, ro, _ = pkg.synth.paired_reads(gb, go, 200_000, seed=102)
    with pkg.Aligner() as al:
        al.load_genomes(gb, go)
        ov = al.align_batch(rb, ro).overlaps
    thr1 = threshold_dropping(ov, 0.2)
    rng = np.random.default_rng(103)
    for thr in (0, thr1):
        cnt = np.bincount(ov["read"][ov["sw_score"] >= thr], minlength=len(ro) - 1)
        assert cnt.sum() > 262_145 and (thr == 0 or (ov["sw_score"] < thr).sum() > 10_000)
        with pkg.Aligner(score_threshold=thr) as al:
            al.load_genomes(gb, go)
            for target in (1, 1023, 1024, 1025, 262_144, 262_145):
                keep = reads_for_count(rng, cnt, target)
                sb, so = shorten(rb, ro, ~keep)
                a, got = align_and_pair(T, al, sb, so, thr)
                assert len(got.sorted_overlaps) == target
                assert len(a.overlaps) > target or thr == 0
                n_tiles = (target + PM_TILE - 1) // PM_TILE
                assert (n_tiles + 1 > 256) == (target > 261_120)


# ---------------------------------------------------------------- 2. volume (and 6c: an odd read count at that volume)

@pytest.fixture(scope="module")
def volume(pkg):
    gb, go = pkg.synth.related_genomes(24, 150_000, seed=201, n_roots=1, divergence=0.015)
    rb, ro, _ = pkg.synth.paired_reads(gb, go, 82_000, seed=202)
    return gb, go, rb, ro


@pytest.mark.parametrize("odd", [False, True])
def test_volume(pkg, T, volume, odd):
    """more than 2^21 passing alignments at threshold 0 and at a threshold that drops a third: k_pair_split over many CTAs
    and the carry loop of k_scan_tiles in the scan of the pass flags and in the scan of the pair counts"""
    gb, go, rb, ro = volume
    if odd:                                  # read 2m: a lightly mutated copy of read m, pair 0's R2
        m = (len(ro) - 1) // 2
        rng = np.random.default_rng(203)
        extra = mutate(rng, rb[int(ro[m]):int(ro[m + 1])], 0.02)
        rb, ro = np.concatenate([rb, extra]), np.append(ro, ro[-1] + np.uint64(len(extra)))
    with pkg.Aligner() as al:
        al.load_genomes(gb, go)
        a, got = align_and_pair(T, al, rb, ro, 0)
    n = len(a.overlaps)
    assert n > 1.5 * SCAN_ONE_PASS
    thr = threshold_dropping(a.overlaps, 1 / 3)
    with pkg.Aligner(score_threshold=thr) as al:
        al.load_genomes(gb, go)
        _, got = align_and_pair(T, al, rb, ro, thr)
    ns = len(got.sorted_overlaps)
    assert SCAN_ONE_PASS < ns < 0.85 * n
    if odd:
        assert (a.overlaps["read"] == len(ro) - 2).sum() > 0


# ---------------------------------------------------------------- 3. an empty R1 list or an empty R2 list

@pytest.mark.parametrize("empty", ["r1", "r2"])
def test_empty_half(pkg, T, empty):
    gb, go = pkg.synth.random_genomes(4, 100_000, seed=301)
    rb, ro, _ = pkg.synth.paired_reads(gb, go, 3000, seed=302)
    n = len(ro) - 1
    cut = np.arange(n) < n // 2 if empty == "r1" else np.arange(n) >= n // 2
    sb, so = shorten(rb, ro, cut)
    with pkg.Aligner() as al:
        al.load_genomes(gb, go)
        a, got = align_and_pair(T, al, sb, so, 0)
    reads = a.overlaps["read"]
    assert len(reads) > 2 * PM_TILE and ((reads < n // 2).all() if empty == "r2" else (reads >= n // 2).all())
    thr = threshold_dropping(a.overlaps, 0.3)
    with pkg.Aligner(score_threshold=thr) as al:
        al.load_genomes(gb, go)
        _, got = align_and_pair(T, al, sb, so, thr)
    assert 0 < len(got.sorted_overlaps) < len(a.overlaps)
    assert ((got.pairs["r1_idx"] < 0) if empty == "r1" else (got.pairs["r2_idx"] < 0)).all()
    with pkg.Aligner(score_threshold=60_000) as al:          # above every score: nothing passes
        al.load_genomes(gb, go)
        al.align_batch(sb, so)
        got = al.pair_batch(fetch=True)
        assert len(got.sorted_overlaps) == 0 and len(got.pairs) == 0
        compact, limit, far = al.fetch_pairs_compact()
        assert len(compact) == 0 and limit == NO_LIMIT and len(far) == 0
        assert len(al.fetch_far_mates(0)) == 0


# ---------------------------------------------------------------- 4. ties between the R1 and the R2 list

def test_ties(pkg, T):
    """fragment == read length: R1 = g[p:p+L1] and R2 = revcomp(g[p:p+L2]) share (pair, entry, rel). With L1 != L2 the
    order of the tie decides which makePair formula sets insert_size (L1 or L2); R1 goes first."""
    gb, go = pkg.synth.random_genomes(4, 100_000, seed=401)
    rng = np.random.default_rng(402)
    r1, r2, n_tie, n_uneq = [], [], 0, 0
    for i in range(4000):
        e = int(rng.integers(0, 4)); g = gb[int(go[e]):int(go[e + 1])]
        if i % 3:                            # a tie pair
            l1 = int(rng.integers(100, 160)); l2 = l1 if rng.random() < 0.5 else int(rng.integers(100, 160))
            p = int(rng.integers(0, len(g) - 200))
            a, b = mutate(rng, g[p:p + l1], 0.005), rc(mutate(rng, g[p:p + l2], 0.005))
            if rng.random() < 0.5:
                a, b = b, a
            n_tie += 1; n_uneq += l1 != l2
        else:
            frag = int(rng.integers(200, 500)); p = int(rng.integers(0, len(g) - frag))
            a, b = fragment_pair(rng, g, p, 150, 150, frag, rng.random() < 0.5)
        r1.append(a); r2.append(b)
    rb, ro = reads_of(r1, r2)
    mid = len(r1)
    with pkg.Aligner(report_cigar=True) as al:
        al.load_genomes(gb, go)
        a, got = align_and_pair(T, al, rb, ro, 0, cigars=True)
    want = T.ko_pipeline(gb, go, rb, ro, T.default_params(report_cigar=1))
    assert_pairs(T, got, want["pair_sorted_overlaps"], want["cigar_pool"], want["pairs"], cigars=True)
    so = got.sorted_overlaps
    key = np.stack([so["read"] % mid, so["entry"], so["rel"].view(np.uint32)], axis=1)
    same = (key[1:] == key[:-1]).all(axis=1) & (so["read"][:-1] < mid) & (so["read"][1:] >= mid)
    tied = np.flatnonzero(same)
    assert len(tied) > 1500 and n_uneq > 1000 and len(so) > 4 * PM_TILE
    lens = np.diff(ro).astype(np.int64)
    uneq = tied[lens[so["read"][tied]] != lens[so["read"][tied + 1]]]
    assert len(uneq) > 500                  # ties whose insert size depends on the order
    assert len(np.unique(tied // PM_TILE)) > 3


# ---------------------------------------------------------------- 5. ragged reads and long runs

def test_ragged_reads_and_long_runs(pkg, T):
    """reads of 32-400 bases in one batch (insert_size takes the length of the specific read; the key bias is the longest
    read), and pairs from a tandem repeat, whose (pair, entry) runs hold dozens of alignments"""
    gb, go = pkg.synth.random_genomes(3, 150_000, seed=501)
    rng = np.random.default_rng(502)
    unit = ACGT[rng.integers(0, 4, 37)]
    rep0 = 60_000
    gb = gb.copy()
    gb[rep0:rep0 + 37 * 60] = np.tile(unit, 60)
    r1, r2 = [], []
    for i in range(5000):
        l1, l2 = int(rng.integers(32, 401)), int(rng.integers(32, 401))
        frag = max(l1, l2) + int(rng.integers(0, 300))
        if i % 25 == 0:                      # inside the repeat
            e, p = 0, rep0 + int(rng.integers(0, 37 * 60 - frag)) if frag < 37 * 60 else rep0
            frag = min(frag, 37 * 60)
        else:
            e = int(rng.integers(0, 3)); p = int(rng.integers(0, 150_000 - frag))
        g = gb[int(go[e]):int(go[e + 1])]
        a, b = fragment_pair(rng, g, p, min(l1, frag), min(l2, frag), frag, rng.random() < 0.5)
        r1.append(a); r2.append(b)
    rb, ro = reads_of(r1, r2)
    lens = np.diff(ro)
    assert lens.min() == 32 and lens.max() >= 395
    with pkg.Aligner() as al:
        al.load_genomes(gb, go)
        a, got = align_and_pair(T, al, rb, ro, 0)
        so = got.sorted_overlaps
        key = (so["read"] % np.uint32(len(r1))).astype(np.uint64) << np.uint64(32) | so["entry"].astype(np.uint64)
        starts = np.flatnonzero(np.r_[True, key[1:] != key[:-1]])
        assert np.diff(np.r_[starts, len(so)]).max() >= 24
        paired = got.pairs[(got.pairs["r1_idx"] >= 0) & (got.pairs["r2_idx"] >= 0)]
        assert len(np.unique(paired["insert_size"])) > 300
    thr = threshold_dropping(a.overlaps, 0.25)
    with pkg.Aligner(score_threshold=thr) as al:
        al.load_genomes(gb, go)
        align_and_pair(T, al, rb, ro, thr)


# ---------------------------------------------------------------- 6. odd read counts

def odd_batch(pkg, m, seed, extra_len=None):
    """m read pairs and one more read, 2m: a lightly mutated copy of read m (pair 0's R2), which pairs with pair 0"""
    gb, go = pkg.synth.random_genomes(3, 60_000, seed=seed)
    rb, ro, _ = pkg.synth.paired_reads(gb, go, m, seed=seed + 1)
    rng = np.random.default_rng(seed + 2)
    extra = mutate(rng, rb[int(ro[m]):int(ro[m + 1])], 0.02)[:extra_len]
    return gb, go, np.concatenate([rb, extra]), np.append(ro, ro[-1] + np.uint64(len(extra)))


@pytest.mark.parametrize("m,extra_len", [(1, None), (3000, None), (3000, 20)])
def test_odd_read_count(pkg, T, m, extra_len):
    """n = 2m + 1: the last read has pair id 2m % m = 0, so its alignments belong in pair 0's run, not at the end of the R2
    list (extra_len 20: it has no alignment at all)"""
    gb, go, rb, ro = odd_batch(pkg, m, 600 + m, extra_len)
    n = len(ro) - 1
    assert n == 2 * m + 1
    want = T.ko_pipeline(gb, go, rb, ro, T.default_params(report_cigar=1))
    with pkg.Aligner(report_cigar=True) as al:
        al.load_genomes(gb, go)
        a, got = align_and_pair(T, al, rb, ro, 0, cigars=True)
        assert_pairs(T, got, want["pair_sorted_overlaps"], want["cigar_pool"], want["pairs"], cigars=True)
    last = a.overlaps["read"] == n - 1
    assert last.any() == (extra_len is None)
    if extra_len is None:                    # read 2m joins pair 0's run
        so = got.sorted_overlaps
        pos = np.flatnonzero(so["read"] == n - 1)
        assert len(pos) and (so["read"][pos - 1] % m == 0).all()
        assert (pos < len(so) - 1).any() or m == 1
    thr = threshold_dropping(a.overlaps, 0.3)
    with pkg.Aligner(score_threshold=thr, report_cigar=True) as al:
        al.load_genomes(gb, go)
        align_and_pair(T, al, rb, ro, thr, cigars=True)


# ---------------------------------------------------------------- 7. insert-size histogram and far mates

@pytest.fixture(scope="module")
def chimeric(pkg):
    """one entry of 4.5 Mbp and two of 300 kbp; three batches of pairs whose R2 is the reverse complement of the span
    ending D bases after R1's start (insert size D): (a) every D < 4096, (b) 20 % of D in [4096, 200000], (c) a few D >= 2^22"""
    gl, go = pkg.synth.random_genomes(1, 4_500_000, seed=701)
    gs, _ = pkg.synth.random_genomes(2, 300_000, seed=702)
    gb = np.concatenate([gl, gs])
    go = np.array([0, 4_500_000, 4_800_000, 5_100_000], dtype=np.uint64)
    rng = np.random.default_rng(703)

    def batch(n, far_frac, far_lo, far_hi, on_long=False):
        r1, r2 = [], []
        for i in range(n):
            far = rng.random() < far_frac
            d = int(rng.integers(far_lo, far_hi)) if far else int(np.clip(np.rint(rng.normal(350, 35)), 151, 600))
            if not far and rng.random() < 0.03:
                d = int(rng.integers(600, 4000))
            e = 0 if (far and on_long) else int(rng.integers(0, 3))
            g = gb[int(go[e]):int(go[e + 1])]
            p = int(rng.integers(0, len(g) - d))
            a, b = fragment_pair(rng, g, p, 150, 150, d, rng.random() < 0.5)
            r1.append(a); r2.append(b)
        return reads_of(r1, r2)

    return gb, go, {"a": batch(6000, 0.0, 0, 1), "b": batch(6000, 0.2, HIST_LOW, 200_000),
                    "c": batch(6000, 0.004, HIST_SPAN + 1000, 4_400_000, on_long=True)}


@pytest.mark.parametrize("which", ["a", "b", "c"])
def test_insert_sizes_and_far_mates(pkg, T, chimeric, which):
    gb, go, batches = chimeric
    rb, ro = batches[which]
    mid = (len(ro) - 1) // 2
    with pkg.Aligner() as al:
        al.load_genomes(gb, go)
        _, full = align_and_pair(T, al, rb, ro, 0)
        compact, limit, far = al.fetch_pairs_compact()
        want_c, want_limit, want_far = pkg.compact_pairs_host(full.sorted_overlaps, full.pairs, mid)
        assert np.array_equal(compact, want_c) and limit == want_limit
        assert np.array_equal(far, want_far)
        for lim in (0, 1000, limit, NO_LIMIT):
            assert np.array_equal(al.fetch_far_mates(lim), far_host(pkg, full, lim)), lim
    ins = full.pairs["insert_size"]
    big = ins[ins >= HIST_LOW]
    if which == "a":
        assert 0 < ins.max() < HIST_LOW
    elif which == "b":
        assert len(big) > 500 and big.max() < HIST_SPAN
        v = np.sort(ins[ins > 0]).astype(np.int64)
        k = len(v)
        steps = [v[int(k * (pc + 1) / 100.0)] - v[int(k * pc / 100.0)] for pc in range(99)]
        assert max(steps) > 1000                                  # the spike branch of the limit
        assert len(far) > 500
    else:
        assert (ins >= HIST_SPAN).sum() >= 5                       # the host fallback
    assert 0 < len(far) or which == "a"


# ---------------------------------------------------------------- 8. buffer reuse

def test_buffer_reuse(pkg, T, chimeric):
    """pair_batch, fetch_pairs_compact, fetch_far_mates at two limits (they reuse the pair-count buffer), fetch_pairs again,
    then a smaller batch: every result equals the first fetch or a fresh context's"""
    gb, go, batches = chimeric
    rb, ro = batches["b"]
    n_small = 1000
    n = len(ro) - 1
    keep = np.r_[np.arange(n_small), n // 2 + np.arange(n_small)]
    sb = np.concatenate([rb[int(ro[i]):int(ro[i + 1])] for i in keep])
    so = np.zeros(len(keep) + 1, np.uint64); so[1:] = np.cumsum(np.diff(ro)[keep])
    with pkg.Aligner(report_cigar=True) as fresh:
        fresh.load_genomes(gb, go)
        fresh.align_batch(sb, so)
        want_small = fresh.pair_batch(fetch=True)
        want_small_c = fresh.fetch_pairs_compact()
    with pkg.Aligner(report_cigar=True) as al:
        al.load_genomes(gb, go)
        al.upload_reads(rb, ro)
        al.align_resident(fetch=False)
        first = al.pair_batch(fetch=True)
        compact, limit, far = al.fetch_pairs_compact()
        assert len(far) > 0
        for lim in (1000, 50_000):
            assert np.array_equal(al.fetch_far_mates(lim), far_host(pkg, first, lim))
        again = al.fetch_pairs()
        assert np.array_equal(again.sorted_overlaps, first.sorted_overlaps) and np.array_equal(again.pairs, first.pairs)
        assert np.array_equal(again.cigar_pool, first.cigar_pool)
        al.align_batch(sb, so)
        small = al.pair_batch(fetch=True)
        small_c = al.fetch_pairs_compact()
    assert np.array_equal(small.sorted_overlaps, want_small.sorted_overlaps) and np.array_equal(small.pairs, want_small.pairs)
    assert np.array_equal(small.cigar_pool, want_small.cigar_pool)
    for x, y in zip(small_c, want_small_c):
        assert np.array_equal(np.asarray(x), np.asarray(y))
