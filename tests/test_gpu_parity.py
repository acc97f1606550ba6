"""GPU tier: the CUDA path (through the C ABI) against the oracle and the committed golden vectors."""
import numpy as np
import pytest

import _lib as T

pytestmark = pytest.mark.gpu

FIELDS = ["read", "entry", "rel", "rev_comp", "ref_begin", "ref_end", "query_begin", "query_end", "sw_score", "cigar_len"]


def canon(a):
    return np.sort(a, order=list(a.dtype.names))


def rec_hash(r):
    """64-bit fingerprint of a 16-byte k-mer record (set algebra on millions of records with np.isin)."""
    with np.errstate(over="ignore"):
        lo = r["id_flags"].astype(np.uint64) | (r["offset"].astype(np.uint64) << np.uint64(32))
        return r["kmer"] * np.uint64(0x9E3779B97F4A7C15) ^ (lo + np.uint64(0x632BE59BD9B4E019)) * np.uint64(0xC2B2AE3D27D4EB4F)


def check_overlaps(got, gpool, want, wpool, fields=FIELDS, cigars=True):
    assert len(got) == len(want)
    undefined = (want["flags"] & 1) != 0      # only where the ORACLE says the reference is undefined
    assert np.array_equal(got["flags"] & 1, want["flags"] & 1), "undefined flags differ"
    for f in fields:
        bad = (got[f] != want[f]) & ~undefined
        assert not bad.any(), (f, int(bad.sum()), got[bad][:3], want[bad][:3])
    if cigars:
        a, b = T.cigars_of(got, gpool), T.cigars_of(want, wpool)
        bad = [i for i in range(len(a)) if a[i] != b[i] and not undefined[i]]
        assert not bad, (len(bad), [(a[i], b[i]) for i in bad[:3]])


def run_pipeline(pkg, gb, go, rb, ro, P, prefilter=True, band=3, sort_bits=0):
    with pkg.Aligner(match=P.match, mismatch=P.mismatch, gap_open=P.gap_open, gap_extend=P.gap_extend,
                     score_threshold=P.score_threshold, report_cigar=bool(P.report_cigar)) as al:
        al.set_prefilter(prefilter)
        al.set_sw_band(band)
        al.set_kmer_sort_bits(sort_bits)
        al.load_genomes(gb, go)
        res = al.align_batch(rb, ro)
        taps = dict(genome_kmers=al.genome_kmers(), read_kmers=al.read_kmers(), raw_seeds=al.raw_seeds(), seeds=al.seeds())
        pairs = al.pair_batch()
        tm = al.timings()
        tm["kmer_sort_bits"] = al.kmer_sort_bits()
    return res, taps, pairs, tm


def check_pipeline(pkg, gb, go, rb, ro, P, want=None):
    """Runs the CUDA path twice — prefilter off (every k-mer record is materialised, so K1/K2 can be compared
    record for record) and on (the production setting) — and checks every stage of both against `want`."""
    want = want or T.ko_pipeline(gb, go, rb, ro, P)
    for prefilter, band in ((False, 0), (True, 2), (True, 3)):
        out = check_pipeline_mode(pkg, gb, go, rb, ro, P, want, prefilter, band)
    return out


def check_pipeline_mode(pkg, gb, go, rb, ro, P, want, prefilter, band):
    # without the prefilter the read list is also sorted in full (KMer.h:388-398); with it, on the leading bits only
    res, taps, pairs, tm = run_pipeline(pkg, gb, go, rb, ro, P, prefilter, band, sort_bits=0 if prefilter else 64)
    assert tm["kmer_sort_bits"] == (64 if not prefilter else tm["kmer_sort_bits"]) and 16 <= tm["kmer_sort_bits"] <= 64
    if not band:
        assert tm["n_sw_band"] == 0 and tm["n_sw_band_rev"] == 0
    # K1/K2: genome list in the reference's order (kmer asc, id_flags desc); read list sorted by k-mer
    wg = T.ko_sort_kmers(want["genome_kmers"])
    assert np.array_equal(taps["genome_kmers"]["kmer"], wg["kmer"])
    assert np.array_equal(taps["genome_kmers"]["id_flags"], wg["id_flags"])
    assert np.array_equal(canon(taps["genome_kmers"]), canon(wg))
    rk = taps["read_kmers"]
    top = rk["kmer"].astype(np.uint64) >> np.uint64(64 - tm["kmer_sort_bits"])
    assert (top[1:] >= top[:-1]).all()
    wr = want["read_kmers"]
    if not prefilter:
        assert np.array_equal(canon(rk), canon(wr))           # same multiset as KMer.h:160-181 produces
    else:
        # survivors: a subset of the reference's records that still holds every record able to seed
        gset = np.unique(wg["kmer"][wg["kmer"] != 0])
        must = wr[np.isin(wr["kmer"], gset)]
        assert np.isin(rec_hash(rk), rec_hash(wr)).all()
        assert np.isin(rec_hash(must), rec_hash(rk)).all()
        assert len(np.unique(rec_hash(rk))) == len(rk)
        assert tm["n_sorted_kmers"] == len(rk) <= tm["n_read_kmers"] == len(wr)
    # K3: raw seed multiset; K4: exact de-duplicated sequence
    assert np.array_equal(canon(taps["raw_seeds"]), canon(want["raw_seeds"]))
    assert np.array_equal(taps["seeds"], want["seeds"])
    # K5-K8
    check_overlaps(res.overlaps, res.cigar_pool, want["overlaps"], want["cigar_pool"], cigars=bool(P.report_cigar))
    # K9
    check_overlaps(pairs.sorted_overlaps, pairs.cigar_pool, want["pair_sorted_overlaps"],
                   want.get("pair_cigar_pool", want["cigar_pool"]), cigars=bool(P.report_cigar))
    assert np.array_equal(pairs.pairs, want["pairs"])
    assert tm["kernel_launches"] > 10
    return res, tm


def params_of(g):
    p = g["params"]
    return T.default_params(match=int(p[0]), mismatch=int(p[1]), gap_open=int(p[2]), gap_extend=int(p[3]),
                            score_threshold=int(p[4]), report_cigar=int(p[5]))


@pytest.mark.parametrize("name", ["pipeline_adversarial_cigar.npz", "pipeline_adversarial_thr60.npz",
                                  "pipeline_config1_mini.npz"])
def test_pipeline_golden(pkg, golden, name):
    """Against the reference's own outputs (fixtures made by tests/golden/make_golden.py)."""
    g = golden(name)
    want = dict(read_kmers=g["read_kmers"], genome_kmers=g["genome_kmers"], raw_seeds=g["raw_seeds_sorted"],
                seeds=g["seeds"], overlaps=g["overlaps"], cigar_pool=g["cigar_pool"],
                pair_sorted_overlaps=g["pair_sorted_overlaps"], pair_cigar_pool=g["pair_sorted_cigar_pool"],
                pairs=g["pairs"])
    want["overlaps"] = want["overlaps"].copy()
    check_pipeline(pkg, g["gen_bases"], g["gen_offs"], g["read_bases"], g["read_offs"], params_of(g), want)


@pytest.mark.parametrize("seed,cigar,thr", [(11, 1, 0), (12, 0, 0), (13, 1, 80)])
def test_pipeline_adversarial(pkg, seed, cigar, thr):
    gb, go, rb, ro = pkg.synth.adversarial_set(seed=seed, n_genomes=10, glen=15_000, n_pairs=2500)
    check_pipeline(pkg, gb, go, rb, ro, T.default_params(report_cigar=cigar, score_threshold=thr))


def test_pipeline_config1_shape(pkg):
    """Config 1 shape, scaled to what the oracle finishes in seconds: 8 x 250 kbp genomes, 20 k pairs."""
    gb, go = pkg.synth.random_genomes(8, 250_000, seed=1)
    rb, ro, truth = pkg.synth.paired_reads(gb, go, 20_000, seed=2)
    res, tm = check_pipeline(pkg, gb, go, rb, ro, T.default_params(report_cigar=1))
    assert tm["n_read_kmers"] == 2 * 20_000 * 119
    assert tm["n_sw_slow"] == 0


def test_pipeline_related_genomes_multi_hit(pkg):
    """Config 2 shape in small: related genomes -> multi-genome piles and several seeds per read."""
    gb, go = pkg.synth.related_genomes(12, 60_000, seed=3, n_roots=3, divergence=0.02)
    rb, ro, _ = pkg.synth.paired_reads(gb, go, 5000, seed=4)
    check_pipeline(pkg, gb, go, rb, ro, T.default_params(report_cigar=1))


def test_empty_and_ragged_inputs(pkg):
    P = T.default_params(report_cigar=1)
    gb, go = pkg.synth.random_genomes(2, 5000, seed=5)
    with pkg.Aligner(report_cigar=True) as al:
        al.load_genomes(gb, go)
        # no reads at all
        res = al.align_batch(np.zeros(0, np.uint8), np.zeros(1, np.uint64))
        assert len(res.overlaps) == 0
        assert len(al.pair_batch().pairs) == 0
        # reads all shorter than k, plus empty reads
        seqs = [b"ACGT" * 5, b"", b"ACGTT" * 6, b""]
        rb, ro = T.concat([np.frombuffer(s, np.uint8) for s in seqs])
        res = al.align_batch(rb, ro)
        assert len(res.overlaps) == 0 and len(al.read_kmers()) == 0
    # a genome set with no k-mers
    with pkg.Aligner(report_cigar=True) as al:
        al.load_genomes(np.frombuffer(b"ACGT" * 5, np.uint8), np.array([0, 20], np.uint64))
        rb, ro, _ = pkg.synth.paired_reads(gb, go, 10, seed=1)
        assert len(al.align_batch(rb, ro).overlaps) == 0


@pytest.mark.parametrize("read_len,frag,kernel", [(251, 500, "fast"), (301, 560, "fast"), (500, 590, "fast"), (700, 900, "slow")])
def test_long_reads(pkg, read_len, frag, kernel):
    """Reads beyond the 160 rows of the 8-lane full-matrix kernel: 161-320 bases run the 16-lane instance (250 / 300-bp
    MiSeq reads), 321-640 the 32-lane one, longer ones the striped kernel (k_sw_striped) — bit-exact either way."""
    gb, go = pkg.synth.random_genomes(3, 40_000, seed=8)
    rb, ro, _ = pkg.synth.paired_reads(gb, go, 300, read_len=read_len, seed=9, frag_mean=frag, frag_sd=30)
    res, tm = check_pipeline(pkg, gb, go, rb, ro, T.default_params(report_cigar=1))
    if kernel == "fast":
        assert tm["n_sw_slow"] == 0 and tm["n_sw_fast"] > 0
    else:
        assert tm["n_sw_slow"] > 0


def test_ssw_long_and_mixed_lengths(pkg):
    """Aligner::Align batches mixing the three full-matrix classes (queries of 20-500 bases — 16-bit cells hold scores up to 2 x 507 —, windows up to 640)."""
    rng = np.random.default_rng(17)
    ACGT = pkg.synth.ACGT
    qs, rs = [], []
    for _ in range(3000):
        L = int(rng.integers(30, 641)); w = ACGT[rng.integers(0, 4, size=L)]
        ql = int(rng.integers(20, min(L, 500) + 1)); st = int(rng.integers(0, L - ql + 1)); qq = w[st:st + ql].copy()
        mm = rng.random(ql) < 0.04; qq[mm] = ACGT[rng.integers(0, 4, size=int(mm.sum()))]
        if rng.random() < 0.3 and ql > 40:
            p = int(rng.integers(10, ql - 10)); k = int(rng.integers(1, 6)); qq = np.concatenate([qq[:p], qq[p + k:]])
        qs.append(qq); rs.append(w)
    q, qo = T.concat(qs); r, ro = T.concat(rs)
    for cigar in (1, 0):
        P = T.default_params(report_cigar=cigar)
        want, wpool = T.ko_ssw_batch(q, qo, r, ro, P, cigar_cap=64)
        with pkg.Aligner(report_cigar=bool(cigar), max_cigar_ops=64) as al:
            out, pool = al.ssw_batch(q, qo, r, ro)
            tm = al.timings()
        check_overlaps(out, pool, want, wpool, fields=FIELDS[4:], cigars=bool(cigar))
        assert tm["n_sw_slow"] == 0


def test_cigar_pool_stride_grows_instead_of_truncating(pkg):
    """max_cigar_ops = 1 cannot hold a gapped CIGAR: kslam_align_batch raises the stride and re-runs the traceback until
    nothing is flagged KSLAM_FLAG_CIGAR_OVERFLOW (the reference has no cap, ssw.c:760-790), so CIGARs equal the oracle's."""
    gb, go = pkg.synth.random_genomes(3, 40_000, seed=5)
    rb, ro, _ = pkg.synth.paired_reads(gb, go, 3000, seed=6, indel_frac=0.5)
    P = T.default_params(report_cigar=1)
    want = T.ko_pipeline(gb, go, rb, ro, P)
    with pkg.Aligner(report_cigar=True, max_cigar_ops=1) as al:
        al.load_genomes(gb, go)
        got = al.align_batch(rb, ro)
    assert (got.overlaps["cigar_len"] > 1).any() and not (got.overlaps["flags"] & 2).any()
    check_overlaps(got.overlaps, got.cigar_pool, want["overlaps"], want["cigar_pool"])


@pytest.mark.parametrize("name", ["ssw_150x150.npz", "ssw_150x300.npz", "ssw_101x140_nocigar.npz"])
def test_ssw_golden(pkg, golden, name):
    g = golden(name)
    P = params_of(g)
    with pkg.Aligner(report_cigar=bool(P.report_cigar)) as al:
        out, pool = al.ssw_batch(g["q"], g["qoffs"], g["r"], g["roffs"])
    want = g["expect"].copy()
    check_overlaps(out, pool, want, g["cigar_pool"], fields=FIELDS[4:], cigars=bool(P.report_cigar))


@pytest.mark.parametrize("shape", [(150, 150), (150, 300), (100, 130), (40, 64), (160, 160)])
@pytest.mark.parametrize("cigar", [0, 1])
@pytest.mark.parametrize("band", [0, 1, 2, 3])
def test_ssw_vs_oracle(pkg, shape, cigar, band):
    q, qo, r, ro = pkg.synth.sw_pairs(20_000, shape[0], shape[1], seed=100 + shape[0] + cigar)
    P = T.default_params(report_cigar=cigar)
    want, wpool = T.ko_ssw_batch(q, qo, r, ro, P, cigar_cap=32)
    with pkg.Aligner(report_cigar=bool(cigar)) as al:
        al.set_sw_band(band)
        out, pool = al.ssw_batch(q, qo, r, ro)
        tm = al.timings()
    check_overlaps(out, pool, want, wpool, fields=FIELDS[4:], cigars=bool(cigar))
    assert tm["n_sw_slow"] == 0
    if band and shape[1] - shape[0] + 1 > 64:
        assert tm["n_sw_band"] == 0 and tm["n_sw_fast"] == 20_000     # no band can hold [-(m - a), n - a]: full matrix at once
    elif band:
        assert tm["n_sw_band"] > 15_000                    # every clean window tries the band first ...
        if shape[1] - shape[0] < 16:
            assert tm["n_sw_fast"] < 10_000                # ... and most are proven there; the rest fall back
    else:
        assert tm["n_sw_band"] == 0 and tm["n_sw_fast"] == 20_000


OUTSIDE = [(5, 4, 10, 10), (1, 1, 1, 1), (2, 8, 3, 3), (3, 1, 1, 4), (2, 9, 2, 1), (4, 6, 4, 4), (10, 2, 3, 3), (2, 3, 2, 5), (3, 0, 0, 0)]


@pytest.mark.parametrize("prm", OUTSIDE)
def test_ssw_scoring_outside_the_gotoh_domain(pkg, prm):
    """gap_extend >= gap_open or mismatch > 2 * gap_extend (main.cpp:45-52 accepts anything): SSW's result depends on its
    striping and k_sw_striped restates the striped byte / word kernels lane for lane (ssw.c:143-592). Score, coordinates and
    CIGAR against the oracle, which tests/test_oracle_vs_ref.py pins to the compiled reference for these parameters."""
    m, x, go, ge = prm
    for shape, n, thr in (((150, 150), 4000, 0), ((120, 160), 3000, 90), ((40, 64), 1500, 0)):
        q, qo, r, ro = pkg.synth.sw_pairs(n, shape[0], shape[1], seed=500 + shape[0] + m)
        for cigar in (1, 0):
            P = T.default_params(report_cigar=cigar, match=m, mismatch=x, gap_open=go, gap_extend=ge, score_threshold=thr)
            want, wpool = T.ko_ssw_batch(q, qo, r, ro, P, cigar_cap=512)
            with pkg.Aligner(match=m, mismatch=x, gap_open=go, gap_extend=ge, score_threshold=thr, report_cigar=bool(cigar), max_cigar_ops=512) as al:
                assert al.exact and not al.fast
                out, pool = al.ssw_batch(q, qo, r, ro)
                tm = al.timings()
            assert tm["n_sw_slow"] == n and tm["n_sw_fast"] == 0 and tm["n_sw_band"] == 0
            check_overlaps(out, pool, want, wpool, fields=FIELDS[4:], cigars=bool(cigar))


@pytest.mark.parametrize("name", ["ssw_params_5_4_10_10.npz", "ssw_params_2_8_3_3.npz", "ssw_params_1_1_1_1.npz"])
def test_ssw_outside_domain_golden(pkg, golden, name):
    """The same against vectors the UNMODIFIED reference produced here (tests/golden/make_golden.py)."""
    g = golden(name)
    P = params_of(g)
    with pkg.Aligner(match=P.match, mismatch=P.mismatch, gap_open=P.gap_open, gap_extend=P.gap_extend, report_cigar=True, max_cigar_ops=256) as al:
        out, pool = al.ssw_batch(g["q"], g["qoffs"], g["r"], g["roffs"])
    check_overlaps(out, pool, g["expect"].copy(), g["cigar_pool"], fields=FIELDS[4:], cigars=True)


def test_ssw_outside_domain_long_and_ragged_reads(pkg):
    """Reads of 1-400 bases (the striped state of the long ones lives in global scratch), repeats, N's."""
    rng = np.random.default_rng(9)
    ACGT = pkg.synth.ACGT
    qs, rs = [], []
    for _ in range(1500):
        per = int(rng.integers(2, 40)); unit = ACGT[rng.integers(0, 4, size=per)]
        L = int(rng.integers(20, 420)); w = np.tile(unit, L // per + 2)[:L].copy()
        mm = rng.random(L) < 0.05; w[mm] = ACGT[rng.integers(0, 4, size=int(mm.sum()))]
        ql = int(rng.integers(1, 401)); st = int(rng.integers(0, max(1, L - ql))); qq = w[st:st + ql].copy()
        if len(qq) == 0:
            qq = ACGT[rng.integers(0, 4, size=5)]
        mm = rng.random(len(qq)) < 0.05; qq[mm] = ACGT[rng.integers(0, 4, size=int(mm.sum()))]
        if rng.random() < 0.1:
            qq[rng.integers(0, len(qq))] = ord("N")
        qs.append(qq); rs.append(w)
    q, qo = T.concat(qs); r, ro = T.concat(rs)
    for (m, x, go, ge) in [(5, 4, 10, 10), (2, 8, 3, 3)]:
        P = T.default_params(report_cigar=1, match=m, mismatch=x, gap_open=go, gap_extend=ge)
        want, wpool = T.ko_ssw_batch(q, qo, r, ro, P, cigar_cap=1024)
        with pkg.Aligner(match=m, mismatch=x, gap_open=go, gap_extend=ge, report_cigar=True, max_cigar_ops=1024) as al:
            out, pool = al.ssw_batch(q, qo, r, ro)
        check_overlaps(out, pool, want, wpool, fields=FIELDS[4:], cigars=True)


@pytest.mark.parametrize("prm", [(5, 4, 10, 10), (2, 8, 3, 3)])
def test_pipeline_scoring_outside_the_gotoh_domain(pkg, prm):
    """The whole path (seeds, windows, un-flip, CIGAR pool, pairing) with such parameters."""
    m, x, go, ge = prm
    gb, go_, rb, ro = pkg.synth.adversarial_set(seed=21, n_genomes=8, glen=10_000, n_pairs=1200)
    P = T.default_params(report_cigar=1, match=m, mismatch=x, gap_open=go, gap_extend=ge)
    want = T.ko_pipeline(gb, go_, rb, ro, P, cigar_cap=256)
    with pkg.Aligner(match=m, mismatch=x, gap_open=go, gap_extend=ge, report_cigar=True) as al:
        al.load_genomes(gb, go_)
        got = al.align_batch(rb, ro)
        pairs = al.pair_batch()
    check_overlaps(got.overlaps, got.cigar_pool, want["overlaps"], want["cigar_pool"])
    assert np.array_equal(pairs.pairs, want["pairs"])


def test_ssw_ragged_lengths_and_repeats(pkg):
    rng = np.random.default_rng(5)
    ACGT = pkg.synth.ACGT
    qs, rs = [], []
    for _ in range(6000):
        per = int(rng.integers(2, 25)); unit = ACGT[rng.integers(0, 4, size=per)]
        L = int(rng.integers(20, 181)); w = np.tile(unit, L // per + 2)[:L].copy()
        m = rng.random(L) < 0.03; w[m] = ACGT[rng.integers(0, 4, size=int(m.sum()))]
        ql = int(rng.integers(1, 161)); st = int(rng.integers(0, max(1, L - ql))); qq = w[st:st + ql].copy()
        if len(qq) == 0:
            qq = ACGT[rng.integers(0, 4, size=5)]
        m = rng.random(len(qq)) < 0.03; qq[m] = ACGT[rng.integers(0, 4, size=int(m.sum()))]
        if rng.random() < 0.1:
            qq[rng.integers(0, len(qq))] = ord("N")
        if rng.random() < 0.1:
            w[rng.integers(0, len(w))] = ord("n")
        qs.append(qq); rs.append(w)
    q, qo = T.concat(qs); r, ro = T.concat(rs)
    P = T.default_params(report_cigar=1)
    want, wpool = T.ko_ssw_batch(q, qo, r, ro, P, cigar_cap=32)
    assert ((want["flags"] & 1) != 0).mean() < 0.01
    for band in (0, 1, 2, 3):
        with pkg.Aligner(report_cigar=True) as al:
            al.set_sw_band(band)
            out, pool = al.ssw_batch(q, qo, r, ro)
        check_overlaps(out, pool, want, wpool, fields=FIELDS[4:])


def diverged_pairs(pkg, n, read_len, window_len, seed):
    """(read, window) pairs whose optimal alignments need every band tier: per-pair substitution rate 0-30 %, 0-4 indels
    of 1-12 bases, a quarter of the reads keep only a prefix / suffix of the planted copy (partial hits), some windows
    carry a tandem repeat (ties between begin positions)."""
    rng = np.random.default_rng(seed)
    ACGT = pkg.synth.ACGT
    qs, rs = [], []
    for _ in range(n):
        w = ACGT[rng.integers(0, 4, size=window_len)]
        if rng.random() < 0.1:
            per = int(rng.integers(1, 9)); st = int(rng.integers(0, window_len - 40)); ln = int(rng.integers(20, 80))
            w[st:st + ln] = np.tile(w[st:st + per], ln // per + 1)[:len(w[st:st + ln])]
        off = int(rng.integers(0, max(1, window_len - read_len + 1)))     # a window shorter than the read: the read is padded below
        src = list(w[off:off + read_len])
        for _k in range(int(rng.integers(0, 5))):
            pos = int(rng.integers(5, max(6, len(src) - 5))); ln = int(rng.integers(1, 13))
            if rng.random() < 0.5:
                del src[pos:pos + ln]
            else:
                src[pos:pos] = list(ACGT[rng.integers(0, 4, size=ln)])
        q = np.array(src[:read_len], dtype=np.uint8)
        if len(q) < read_len:
            q = np.concatenate([q, ACGT[rng.integers(0, 4, size=read_len - len(q))]])
        rate = rng.random() * 0.3
        m = rng.random(read_len) < rate
        q[m] = ACGT[rng.integers(0, 4, size=int(m.sum()))]
        u = rng.random()
        if u < 0.125:
            k = int(rng.integers(20, read_len - 20)); q[k:] = ACGT[rng.integers(0, 4, size=read_len - k)]
        elif u < 0.25:
            k = int(rng.integers(20, read_len - 20)); q[:k] = ACGT[rng.integers(0, 4, size=k)]
        qs.append(q); rs.append(w)
    q, qo = T.concat(qs); r, ro = T.concat(rs)
    return q, qo, r, ro


@pytest.mark.parametrize("shape", [(150, 150), (150, 190), (120, 160), (160, 100)])
@pytest.mark.parametrize("cigar", [0, 1])
def test_ssw_diverged_reads_use_every_band_tier(pkg, shape, cigar):
    """Diverged, gapped and partial hits against the oracle: the forward intervals [-(m - a), n - a] of such alignments are
    65-128 diagonals wide (the multi-lane tiers) and their reverse sweeps run in the anchored band (sw_band.cuh), which must
    find the same begin coordinates as SSW's full reverse pass."""
    q, qo, r, ro = diverged_pairs(pkg, 12_000, shape[0], shape[1], seed=500 + shape[0] + shape[1] + cigar)
    P = T.default_params(report_cigar=cigar)
    want, wpool = T.ko_ssw_batch(q, qo, r, ro, P, cigar_cap=64)
    res = {}
    for band in (0, 3):
        with pkg.Aligner(report_cigar=bool(cigar), max_cigar_ops=64) as al:
            al.set_sw_band(band)
            out, pool = al.ssw_batch(q, qo, r, ro)
            res[band] = al.timings()
        check_overlaps(out, pool, want, wpool, fields=FIELDS[4:], cigars=bool(cigar))
    tm = res[3]
    assert tm["n_sw_slow"] == 0
    if shape == (150, 150):
        assert tm["n_sw_tier96"] > 100 and tm["n_sw_tier128"] > 100, tm        # direct, from the seed-diagonal bound
    assert tm["n_sw_tier96"] + tm["n_sw_tier128"] + tm["n_sw_band64"] > 100, tm  # ... or after the 32-wide trial sweep
    rev = tm["n_sw_rev_tier"]
    assert sum(rev) > 8_000 and rev[0] > 100 and rev[4] + rev[5] + rev[6] > 100, rev
    if shape == (150, 150):
        assert tm["sw_cells_computed"] < res[0]["sw_cells_computed"]


INSIDE = [(1, 2, 3, 1), (3, 4, 9, 2), (2, 0, 2, 1), (1, 1, 2, 1), (2, 4, 12, 7), (2, 4, 3, 2), (1, 0, 1, 0)]       # (the packed cells hold match <= 3, mismatch <= 4)


@pytest.mark.parametrize("prm", INSIDE)
def test_ssw_fast_domain_other_parameters(pkg, prm):
    """Scoring parameters other than 2/3/5/2 INSIDE the plain-Gotoh domain (gap_extend < gap_open, mismatch <= 2 gap_extend):
    the packed band kernels run, and every bound they are placed with depends on the parameters — the forward interval on
    match, the anchored reverse band on match and both gap costs, the untracked rows on match, the diagonal shortcut on
    match + mismatch. Diverged / gapped / partial pairs against the oracle (pinned to the reference for such sets in
    tests/test_oracle_vs_ref.py)."""
    m, x, go, ge = prm
    q, qo, r, ro = diverged_pairs(pkg, 6_000, 150, 150, seed=900 + 7 * m + x + go)
    P = T.default_params(report_cigar=1, match=m, mismatch=x, gap_open=go, gap_extend=ge)
    want, wpool = T.ko_ssw_batch(q, qo, r, ro, P, cigar_cap=64)
    with pkg.Aligner(report_cigar=True, max_cigar_ops=64, match=m, mismatch=x, gap_open=go, gap_extend=ge) as al:
        assert al.fast
        out, pool = al.ssw_batch(q, qo, r, ro)
        tm = al.timings()
    check_overlaps(out, pool, want, wpool, fields=FIELDS[4:])
    assert tm["n_sw_slow"] == 0 and tm["n_sw_band"] > 3_000


@pytest.mark.parametrize("prm", [(4, 4, 6, 2), (3, 5, 9, 3), (5, 6, 12, 3), (8, 9, 20, 5), (100, 100, 120, 60)])
def test_ssw_fast_domain_beyond_the_packed_cells(pkg, prm):
    """Parameters inside the plain-Gotoh domain that the packed kernels cannot hold (match > 3, mismatch > 4, or scores
    beyond the 16-bit cells): every alignment runs the slow list (k_sw_striped). With match 100, 700-base reads score above
    32767, where SSW's word pass saturates; the result is the saturated one, as the oracle computes it."""
    m, x, go, ge = prm
    if m == 100:
        rng = np.random.default_rng(41)
        ws = [pkg.synth.ACGT[rng.integers(0, 4, size=700)] for _ in range(300)]       # reads: the windows with 1 % substitutions
        qs = [np.where(rng.random(700) < 0.01, pkg.synth.ACGT[rng.integers(0, 4, size=700)], w) for w in ws]
        sets = [T.concat(qs) + T.concat(ws)]
    else:
        sets = [diverged_pairs(pkg, 3000, a, b, seed=950 + 7 * m + x + a) for a, b in ((150, 150), (120, 160))]
    for q, qo, r, ro in sets:
        n = len(qo) - 1
        for cigar in (1, 0):
            P = T.default_params(report_cigar=cigar, match=m, mismatch=x, gap_open=go, gap_extend=ge)
            want, wpool = T.ko_ssw_batch(q, qo, r, ro, P, cigar_cap=64)
            with pkg.Aligner(report_cigar=bool(cigar), max_cigar_ops=64, match=m, mismatch=x, gap_open=go, gap_extend=ge) as al:
                assert al.fast
                out, pool = al.ssw_batch(q, qo, r, ro)
                tm = al.timings()
            assert tm["n_sw_slow"] == n and tm["n_sw_fast"] == 0 and tm["n_sw_band"] == 0
            if m == 100:
                assert (want["sw_score"] == 32767).all() and not (want["flags"] & 1).any()
            check_overlaps(out, pool, want, wpool, fields=FIELDS[4:], cigars=bool(cigar))


@pytest.mark.parametrize("shape", [(150, 150), (120, 160)])
@pytest.mark.parametrize("cigar", [0, 1])
def test_ssw_windows_with_code4_columns(pkg, shape, cigar):
    """Windows holding code-4 bases (N runs, lower-case n, IUPAC letters: score 0 against every row, ssw_cpp.cpp:43-48) run
    the masked variants of the band tiers instead of the full-matrix kernel; same results as the oracle on diverged, gapped
    and partial pairs, forward and reverse, with N runs in most windows and some reads."""
    q, qo, r, ro = diverged_pairs(pkg, 10_000, shape[0], shape[1], seed=700 + shape[0] + cigar)
    rng = np.random.default_rng(71)
    q = q.copy(); r = r.copy()
    for i in range(10_000):
        if rng.random() < 0.7:
            for _k in range(int(rng.integers(1, 4))):
                st = int(rng.integers(0, shape[1] - 1)); ln = int(rng.integers(1, 13))
                r[int(ro[i]) + st:min(int(ro[i]) + st + ln, int(ro[i + 1]))] = rng.choice(np.frombuffer(b"NnRYK", dtype=np.uint8))
        if rng.random() < 0.1:
            st = int(rng.integers(0, shape[0] - 1)); ln = int(rng.integers(1, 9))
            q[int(qo[i]) + st:min(int(qo[i]) + st + ln, int(qo[i + 1]))] = ord("N")
    P = T.default_params(report_cigar=cigar)
    want, wpool = T.ko_ssw_batch(q, qo, r, ro, P, cigar_cap=64)
    with pkg.Aligner(report_cigar=bool(cigar), max_cigar_ops=64) as al:
        out, pool = al.ssw_batch(q, qo, r, ro)
        tm = al.timings()
    check_overlaps(out, pool, want, wpool, fields=FIELDS[4:], cigars=bool(cigar))
    assert tm["n_sw_slow"] == 0
    assert tm["n_sw_band"] == 10_000, tm["n_sw_band"]          # every window is band-eligible, clean or not
    assert tm["n_sw_fast"] < 9_000, tm["n_sw_fast"]            # (what is left: trial sweeps that bound nothing <= 128 diagonals)


def test_radix_sort_matches_numpy(pkg):
    rng = np.random.default_rng(3)
    with pkg.Aligner() as al:
        for n, lo, hi in [(1, 0, 64), (5000, 0, 64), (300_000, 0, 64), (100_000, 8, 40), (70_000, 0, 13)]:
            recs = np.zeros(n, dtype=pkg.KMER_DT)
            recs["kmer"] = rng.integers(0, 2**63, size=n, dtype=np.uint64) * 2 + rng.integers(0, 2, size=n, dtype=np.uint64)
            recs["id_flags"] = np.arange(n, dtype=np.uint32)       # arrival order: checks stability
            recs["offset"] = rng.integers(0, 2**32, size=n, dtype=np.uint64).astype(np.uint32)
            got, ms = al.sort_records(recs, lo, hi)
            mask = np.uint64(((1 << (hi - lo)) - 1) if hi - lo < 64 else 0xFFFFFFFFFFFFFFFF)
            key = (recs["kmer"] >> np.uint64(lo)) & mask
            order = np.argsort(key, kind="stable")
            assert np.array_equal(got, recs[order]), (n, lo, hi)


def test_full_size_properties_config1_slice(pkg):
    """Size-independent properties at a larger scale than the oracle can check quickly: planted position is
    recovered (Tests.h:161-264), perfect reads score 2 x length (Tests.h:136,323), results are identical when
    the same batch is split in two (seeds are per-read), and the record counts obey KMer.h:202."""
    gb, go = pkg.synth.random_genomes(20, 1_000_000, seed=1)
    n_pairs = 200_000
    rb, ro, truth = pkg.synth.paired_reads(gb, go, n_pairs, seed=2, sub_rate=0.0, indel_frac=0.0)
    with pkg.Aligner(report_cigar=False) as al:
        al.load_genomes(gb, go)
        res = al.align_batch(rb, ro)
        tm = al.timings()
        ov = res.overlaps
        assert tm["n_read_kmers"] == 2 * n_pairs * 119
        assert tm["n_genome_kmers"] == 20 * ((1_000_000 - 32) // 16 + 1)
        # error-free reads: every read has a seed on its own genome scoring exactly 300
        best = np.zeros(2 * n_pairs, dtype=np.uint32)
        np.maximum.at(best, ov["read"], ov["sw_score"])
        assert (best == 300).mean() > 0.999
        # planted genome and position are recovered for the left mate (forward strand, rel == pos)
        r1_is_left = truth["swapped"] == 0
        left_read = np.where(r1_is_left, np.arange(n_pairs), np.arange(n_pairs) + n_pairs)
        sel = (ov["sw_score"] == 300) & (ov["rev_comp"] == 0)
        hit = {}
        for rd, en, rel in zip(ov["read"][sel], ov["entry"][sel], ov["rel"][sel]):
            hit[int(rd)] = (int(en), int(rel))
        ok = sum(1 for i in range(0, n_pairs, 97) if hit.get(int(left_read[i])) == (int(truth["genome"][i]), int(truth["pos"][i])))
        assert ok >= 0.99 * len(range(0, n_pairs, 97))
        # sorted, de-duplicated order
        key = (ov["read"].astype(np.int64) << 32) | ov["entry"].astype(np.int64)
        assert (np.diff(key) >= 0).all()
        # splitting the batch changes nothing for the reads of the first half
        half = n_pairs // 2
        sub = np.concatenate([np.arange(half), np.arange(n_pairs, n_pairs + half)])
        L = 150
        rb2 = rb.reshape(-1, L)[sub].reshape(-1)
        ro2 = np.arange(len(sub) + 1, dtype=np.uint64) * np.uint64(L)
        res2 = al.align_batch(rb2, ro2)
        a = ov[ov["read"] < half]
        b = res2.overlaps[res2.overlaps["read"] < half]
        for f in FIELDS[1:9]:
            assert np.array_equal(a[f], b[f]), f


def test_direct_tiers_match_full_matrix_at_volume(pkg):
    """The tier an alignment runs in never changes its result: 60k config-1-like pairs (1 % substitutions, 5 % reads with
    an indel) and 40k pairs against a diverged phylogeny give identical alignments at level 3 (direct tiers from the
    seed-diagonal bound) and level 0 (full matrix only); the narrow tiers must actually carry the bulk of the work."""
    cases = [(pkg.synth.random_genomes(20, 500_000, seed=3), 60_000, 0.8),
             (pkg.synth.tree_genomes(40, 300_000, seed=4), 40_000, 0.2)]
    for (gb, go), n_pairs, min_narrow in cases:
        rb, ro, _ = pkg.synth.paired_reads(gb, go, n_pairs, seed=9)
        outs = {}
        for level in (0, 3):
            with pkg.Aligner(report_cigar=True) as al:
                al.set_sw_band(level)
                al.load_genomes(gb, go)
                outs[level] = (al.align_batch(rb, ro), al.timings())
        (a, ta), (b, tb) = outs[0], outs[3]
        assert len(a.overlaps) > n_pairs
        for f in FIELDS:
            assert np.array_equal(a.overlaps[f], b.overlaps[f]), f
        assert T.cigars_of(a.overlaps[:5000], a.cigar_pool) == T.cigars_of(b.overlaps[:5000], b.cigar_pool)
        assert ta["n_sw_band"] == 0
        narrow = tb["n_sw_tier8"] + tb["n_sw_tier16"]
        assert narrow >= min_narrow * tb["n_seeds"], (narrow, tb["n_seeds"])
        assert tb["sw_cells_computed"] < ta["sw_cells_computed"]


def test_align_pair_batch_equals_two_calls(pkg):
    """kslam_align_pair_batch (the batch-loop body in one call, no copy of the unsorted vector) returns exactly what
    kslam_align_batch + kslam_pair_batch return; two contexts on one GPU driven from two threads do not disturb each other."""
    import threading
    gb, go, rb, ro = pkg.synth.adversarial_set(seed=51, n_genomes=8, glen=8000, n_pairs=700)
    with pkg.Aligner(report_cigar=True) as al:
        al.load_genomes(gb, go)
        al.align_batch(rb, ro)
        want = al.pair_batch()
    got = [None, None]

    def run(k):
        with pkg.Aligner(report_cigar=True) as a2:
            a2.load_genomes(gb, go)
            for _ in range(3):
                got[k] = a2.align_pair_batch(rb, ro)
    th = [threading.Thread(target=run, args=(k,)) for k in range(2)]
    [t.start() for t in th]; [t.join() for t in th]
    for g in got:
        assert np.array_equal(g.sorted_overlaps, want.sorted_overlaps)
        assert np.array_equal(g.pairs, want.pairs)
        assert T.cigars_of(g.sorted_overlaps, g.cigar_pool) == T.cigars_of(want.sorted_overlaps, want.cigar_pool)


def test_compact_pair_records(pkg):
    """kslam_fetch_pairs_compact (SURVEY.md §8f-3): the 24-byte records, the batch's insert-size limit and the mates of the
    pairs beyond it equal what the full records give (built on the host), on data with far pairs."""
    gb, go = pkg.synth.random_genomes(6, 120_000, seed=31)
    rb, ro, _ = pkg.synth.paired_reads(gb, go, 8000, seed=32)
    rb2, ro2, _ = pkg.synth.paired_reads(gb, go, 1500, seed=33, frag_mean=560.0, frag_sd=10.0)     # a second library far out
    mid = 8000
    rows = rb.reshape(2, mid, 150).copy(); far_rows = rb2.reshape(2, 1500, 150)
    rows[:, :1500] = far_rows
    rb = rows.reshape(-1)
    with pkg.Aligner(report_cigar=False) as al:
        al.load_genomes(gb, go)
        al.upload_reads(rb, ro)
        al.align_resident(fetch=False)
        full = al.pair_batch(fetch=True)
        compact, limit, far = al.fetch_pairs_compact()
    want_c, want_limit, want_far = pkg.compact_pairs_host(full.sorted_overlaps, full.pairs, mid)
    assert np.array_equal(compact, want_c) and limit == want_limit and len(compact) > 8_000
    assert np.array_equal(far, want_far)
    assert 0 < len(far) < len(compact) // 4 and limit < 620


def test_fastq_to_alignments(pkg, tmp_path):
    """FASTQ files -> kslam_fastq_next (pinned batch, R1 block then R2 block) -> kslam_align_pair_batch: same pairs as
    handing the arrays over directly, batch by batch (--num-reads-at-once)."""
    gb, go, rb, ro = pkg.synth.adversarial_set(seed=61, n_genomes=8, glen=8000, n_pairs=500)
    n = len(ro) - 1; mid = n // 2
    seqs = [bytes(rb[int(ro[i]):int(ro[i + 1])]) for i in range(n)]
    for k, (lo, hi) in enumerate(((0, mid), (mid, n))):
        with open(tmp_path / f"R{k + 1}.fq", "wb") as f:
            for i in range(lo, hi):
                f.write(b"@r%d/%d\n" % (i - lo, k + 1) + seqs[i] + b"\n+\n" + b"I" * len(seqs[i]) + b"\n")
    with pkg.Aligner(report_cigar=True) as al, pkg.FastqReader(str(tmp_path / "R1.fq"), str(tmp_path / "R2.fq")) as rd:
        al.load_genomes(gb, go)
        done = 0
        while True:
            b = rd.next(200, copy=False)
            if b is None:
                break
            cnt = b.n_r1
            got = al.align_pair_batch(b.bases, b.offs)
            sub = [seqs[done + i] for i in range(cnt)] + [seqs[mid + done + i] for i in range(cnt)]
            sb, so = T.concat([np.frombuffer(s, np.uint8) for s in sub])
            want = al.align_pair_batch(sb, so)
            assert len(want.pairs) > 0 and np.array_equal(got.pairs, want.pairs)
            assert np.array_equal(got.sorted_overlaps, want.sorted_overlaps)
            done += cnt
        assert done == mid


@pytest.mark.skipif(not T.have_ref(), reason="needs the prebuilt oracle/_ref")
@pytest.mark.parametrize("kind,seed", [("related", 81), ("config1", 82)])
def test_fastq_to_sam_equals_reference(pkg, tmp_path, kind, seed):
    """The whole --sam-file run — FASTQ files -> reader -> GPU matching path -> host stages -> SAM text — against the
    reference's own chain (alignToDatabase ... writeSAMOutputPairs, oracle/_ref) on the same reads, byte for byte, in one
    batch and in three (--num-reads-at-once)."""
    from kslam_b200 import slam
    from test_sam_host import make_inputs
    gb, go, rb, ro, quals, idb, ido = make_inputs(pkg, seed, n_pairs=600, kind=kind)
    n = len(ro) - 1; mid = n // 2
    fa = tmp_path / "db.fa"
    with open(fa, "wb") as f:
        for i in range(len(go) - 1):
            f.write(b">g%d synthetic entry\n" % i + bytes(gb[int(go[i]):int(go[i + 1])]) + b"\n")
    for k, (lo, hi) in enumerate(((0, mid), (mid, n))):
        with open(tmp_path / f"R{k + 1}.fq", "wb") as f:
            for i in range(lo, hi):
                f.write(b"@r%d\n" % i + bytes(rb[int(ro[i]):int(ro[i + 1])]) + b"\n+\n" + bytes(quals[int(ro[i]):int(ro[i + 1])]) + b"\n")

    def reference(lo, hi):
        sel = list(range(lo, hi)) + list(range(mid + lo, mid + hi))
        sb, so = T.concat([rb[int(ro[i]):int(ro[i + 1])] for i in sel])
        sq, _ = T.concat([quals[int(ro[i]):int(ro[i + 1])] for i in sel])
        R = T.Ref(gb, go, sb, so, T.default_params(report_cigar=1))
        R.align_to_database(); R.screen_and_pair()
        text, _ = T.ref_sam(R, sq, so)
        R.close()
        # the harness names reads r<local index>; the files name them r<global index>
        for j in sorted(range(len(sel)), reverse=True):
            text = text.replace(b"r%d\t" % j, b"R%d\t" % sel[j])
        return text.replace(b"R", b"r")

    for at_once in (mid, 200):
        sam = tmp_path / f"out_{at_once}.sam"
        st = slam.align_to_sam(pkg, [str(fa)], str(tmp_path / "R1.fq"), str(tmp_path / "R2.fq"), str(sam), reads_at_once=at_once, command_line="x")
        body = b"".join(l for l in open(sam, "rb").read().splitlines(keepends=True) if not l.startswith(b"@"))
        want = b"".join(reference(lo, min(lo + at_once, mid)) for lo in range(0, mid, at_once))
        assert st["pairs"] == mid and len(want) > 10_000
        assert body == want


@pytest.mark.skipif(not T.have_ref(), reason="needs the prebuilt oracle/_ref")
def test_single_end_gpu_to_sam_equals_reference(pkg):
    """Single-end reads: kslam_align_batch on the GPU -> kslam_sam_batch_single, against the reference's single-end chain."""
    from test_sam_host import make_inputs
    gb, go, rb, ro, quals, idb, ido = make_inputs(pkg, 95, n_pairs=500, kind="related")
    R = T.Ref(gb, go, rb, ro, T.default_params(report_cigar=1))
    R.align_to_database(); R.L.kref_screen(R.h)
    want = T.ref_sam_single(R, quals, ro)
    R.close()
    with pkg.Aligner(report_cigar=True) as al:
        al.load_genomes(gb, go)
        res = al.align_batch(rb, ro)
    w = pkg.SamWriter(gb, go, [f"g{i}" for i in range(len(go) - 1)], report_cigar=True)
    assert w.batch_single(rb, ro, quals, ro, idb, ido, res.overlaps, res.cigar_pool) == want and len(want) > 10_000
