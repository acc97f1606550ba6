"""CPU tier: the host stages after pairing (kslam_sam_batch: per-read grouping, insert-size limit, both screens,
pseudo-assembly, SAM records with CIGAR / MD / NM / MAPQ) against the reference's OWN functions run here
(oracle/_ref: SLAM.h:215-239 chain, PairedOverlap.h:314-576, SAM.h), byte for byte, and against a golden SAM file."""
import hashlib
import zlib

import numpy as np
import pytest

import _lib as T


def make_inputs(pkg, seed, n_pairs=400, kind="adversarial"):
    if kind == "adversarial":
        gb, go, rb, ro = pkg.synth.adversarial_set(seed=seed, n_genomes=8, glen=6000, n_pairs=n_pairs)
    elif kind == "related":
        gb, go = pkg.synth.related_genomes(12, 20_000, seed=seed)          # multi-genome hits: ties, chains, far pairs
        rb, ro, _ = pkg.synth.paired_reads(gb, go, n_pairs, seed=seed + 1)
    else:
        gb, go = pkg.synth.random_genomes(4, 30_000, seed=seed)
        rb, ro, _ = pkg.synth.paired_reads(gb, go, n_pairs, seed=seed + 1)
    rng = np.random.default_rng(seed)
    quals = rng.integers(35, 75, size=len(rb), dtype=np.uint8)
    n = len(ro) - 1
    ids = [b"r%d" % i for i in range(n)]            # what "@r<i>" becomes (FASTQsequence.h:61-71)
    idb = np.frombuffer(b"".join(ids), np.uint8); ido = np.zeros(n + 1, np.uint64); ido[1:] = np.cumsum([len(x) for x in ids])
    return gb, go, rb, ro, quals, idb, ido


def reference_side(gb, go, rb, ro, quals, cigar, **kw):
    R = T.Ref(gb, go, rb, ro, T.default_params(report_cigar=int(cigar)))
    R.align_to_database()
    ov, pool, pairs = R.screen_and_pair()
    hdr = T.ref_sam_header(R, "SLAM --db x")
    text, mi = T.ref_sam(R, quals, ro, **kw)
    R.close()
    return ov, pool, pairs, text, mi, hdr


@pytest.mark.skipif(not T.have_ref(), reason="needs oracle/_ref (built where /root/reference exists)")
@pytest.mark.parametrize("kind,seed", [("adversarial", 71), ("related", 72), ("config1", 73)])
@pytest.mark.parametrize("cigar", [1, 0])
def test_sam_text_equals_reference(pkg, kind, seed, cigar):
    gb, go, rb, ro, quals, idb, ido = make_inputs(pkg, seed, kind=kind)
    tags = [f"g{i}" for i in range(len(go) - 1)]
    for kw in (dict(), dict(pseudo=False), dict(num_alignments=1), dict(sam_xa=True, fraction=0.5), dict(num_alignments=3, fraction=0.0)):
        ov, pool, pairs, want, want_mi, want_hdr = reference_side(gb, go, rb, ro, quals, cigar, **kw)
        assert len(pairs) > 50 and len(want) > 1000
        w = pkg.SamWriter(gb, go, tags, num_alignments=kw.get("num_alignments", 10), score_fraction_threshold=kw.get("fraction", 0.95),
                          pseudo_assembly=kw.get("pseudo", True), report_cigar=bool(cigar), sam_xa=kw.get("sam_xa", False))
        got, mi = w.batch(rb, ro, quals, ro, idb, ido, ov, pool, pairs)
        assert mi == want_mi
        if got != want:
            a, b = got.split(b"\n"), want.split(b"\n")
            bad = [(i, x, y) for i, (x, y) in enumerate(zip(a, b)) if x != y][:3]
            raise AssertionError((kw, len(a), len(b), bad))
        assert w.header("SLAM --db x") == want_hdr


@pytest.mark.skipif(not T.have_ref(), reason="needs oracle/_ref")
@pytest.mark.parametrize("kind,seed,threads", [("related", 81, 5), ("config1", 82, 3), ("adversarial", 83, 8)])
def test_sam_parallel_host_stages_equal_reference(pkg, kind, seed, threads, monkeypatch):
    """Large batches group the reads, sort the insert sizes and build the pseudo-assembly lists on all host threads
    (ranges cut at read boundaries, counting sort, count / prefix / fill); forced on here for a small batch."""
    monkeypatch.setenv("KSLAM_HOST_PAR_MIN", "1")
    gb, go, rb, ro, quals, idb, ido = make_inputs(pkg, seed, n_pairs=700, kind=kind)
    tags = [f"g{i}" for i in range(len(go) - 1)]
    ov, pool, pairs, want, want_mi, _ = reference_side(gb, go, rb, ro, quals, 1)
    w = pkg.SamWriter(gb, go, tags, report_cigar=True, threads=threads)
    got, mi = w.batch(rb, ro, quals, ro, idb, ido, ov, pool, pairs)
    assert mi == want_mi and got == want and len(want) > 10_000


def test_sam_golden(pkg, golden):
    """Inputs and the reference's SAM text from tests/golden/make_golden.py: travels to boxes without /root/reference."""
    g = golden("sam_config1_mini.npz")
    tags = [f"g{i}" for i in range(len(g["go"]) - 1)]
    w = pkg.SamWriter(g["gb"], g["go"], tags, report_cigar=True)
    got, mi = w.batch(g["rb"], g["ro"], g["quals"], g["ro"], g["ids"], g["id_offs"], g["ov"], g["pool"], g["pairs"])
    assert got == g["sam"].tobytes() and mi == int(g["max_insert"])
    assert w.header("SLAM golden") == g["header"].tobytes()


def oracle_side(gb, go, rb, ro):
    """Pair-sorted alignments, CIGAR pool and pair records from the oracle's restatement of alignToDatabase + screen +
    getPairedOverlaps, which tests/test_oracle_golden.py pins to the reference's on the stored batches."""
    w = T.ko_pipeline(gb, go, rb, ro, T.default_params(report_cigar=1))
    return w["pair_sorted_overlaps"], w["cigar_pool"], w["pairs"]


def crc32_of(*arrays):
    return zlib.crc32(b"".join(np.ascontiguousarray(a).tobytes() for a in arrays))


def sam_digest(text):
    """What tests/golden/sam_random_6000_digest.npz keeps of a SAM text too large to store: its SHA-256, its length and
    one CRC-32 per line (to name the first line that differs)."""
    return dict(sha256=np.frombuffer(hashlib.sha256(text).digest(), np.uint8), length=len(text),
                line_crc32=np.array([zlib.crc32(x) for x in text.split(b"\n")], np.uint32))


def test_sam_text_buffers_are_recycled_between_batches(pkg, golden):
    """The library keeps the per-thread strings and the largest buffer given back through kslam_sam_free for the next batch
    (page faults cost more than the text): a long batch, a short one and the long one again, with different thread counts,
    must give the recorded texts (> 1 MB so that the buffer is actually kept). The short one is the reference's, stored
    whole; the long one is known by its digest, whose origin tests/golden/make_golden.py sam_digest_fixture states."""
    gb, go, rb, ro, quals, idb, ido = make_inputs(pkg, 5, n_pairs=6000, kind="random")
    tags = [f"g{i}" for i in range(len(go) - 1)]
    ov, pool, pairs = oracle_side(gb, go, rb, ro)
    d = golden("sam_random_6000_digest.npz")
    assert crc32_of(gb, go, rb, ro, quals, idb, ido) == int(d["inputs_crc32"]), "synth.py no longer makes the recorded reads"
    assert crc32_of(ov, pool, pairs) == int(d["alignments_crc32"]), "the oracle no longer gives the recorded alignments"
    assert int(d["length"]) > (1 << 20)
    g = golden("sam_config1_mini.npz")
    gtags = [f"g{i}" for i in range(len(g["go"]) - 1)]
    for threads in (4, 2, 7):
        w = pkg.SamWriter(gb, go, tags, report_cigar=True, threads=threads)
        got, mi = w.batch(rb, ro, quals, ro, idb, ido, ov, pool, pairs)
        have = sam_digest(got)
        if not np.array_equal(have["sha256"], d["sha256"]):
            a, b = have["line_crc32"], d["line_crc32"]
            i = next((i for i, (x, y) in enumerate(zip(a, b)) if x != y), min(len(a), len(b)))
            raise AssertionError((threads, len(got), int(d["length"]), len(a), len(b), i, got.split(b"\n")[i:i + 1]))
        assert mi == int(d["max_insert"])
        ws = pkg.SamWriter(g["gb"], g["go"], gtags, report_cigar=True, threads=threads)
        got, _ = ws.batch(g["rb"], g["ro"], g["quals"], g["ro"], g["ids"], g["id_offs"], g["ov"], g["pool"], g["pairs"])
        assert got == g["sam"].tobytes()


def test_sam_empty_batch(pkg):
    gb, go = pkg.synth.random_genomes(2, 1000, seed=1)
    w = pkg.SamWriter(gb, go, ["a", "b"])
    z8, z1 = np.zeros(0, np.uint8), np.zeros(1, np.uint64)
    got, mi = w.batch(z8, z1, z8, z1, z8, z1, np.zeros(0, pkg.OVERLAP_DT), np.zeros(0, np.uint32), np.zeros(0, pkg.PAIR_DT))
    assert got == b"" and mi == 2**32 - 1


def test_sam_rejects_out_of_range_records(pkg, golden):
    g = golden("sam_config1_mini.npz")
    tags = [f"g{i}" for i in range(len(g["go"]) - 1)]
    w = pkg.SamWriter(g["gb"], g["go"], tags)
    args = [g["rb"], g["ro"], g["quals"], g["ro"], g["ids"], g["id_offs"]]
    for field, arr, bad in (("read", "ov", 10**9), ("entry", "ov", 10**6), ("r1_idx", "pairs", 10**9)):
        ov, pairs = g["ov"].copy(), g["pairs"].copy()
        (ov if arr == "ov" else pairs)[field][0] = bad
        with pytest.raises(pkg.KslamError):
            w.batch(*args, ov, g["pool"], pairs)


@pytest.mark.skipif(not T.have_ref(), reason="needs oracle/_ref")
@pytest.mark.parametrize("kind,seed,thr", [("adversarial", 91, 0), ("related", 92, 0), ("config1", 93, 120)])
def test_single_end_sam_equals_reference(pkg, kind, seed, thr):
    """Single-end reads (SLAM.h:223-228): the same reads treated as one unpaired set."""
    gb, go, rb, ro, quals, idb, ido = make_inputs(pkg, seed, kind=kind)
    tags = [f"g{i}" for i in range(len(go) - 1)]
    for kw in (dict(), dict(pseudo=False, num_alignments=2), dict(sam_xa=True)):
        R = T.Ref(gb, go, rb, ro, T.default_params(report_cigar=1, score_threshold=thr))
        ov_all, pool_all = R.align_to_database()
        R.L.kref_screen(R.h)
        want = T.ref_sam_single(R, quals, ro, **kw)
        R.close()
        assert len(want) > 1000
        w = pkg.SamWriter(gb, go, tags, num_alignments=kw.get("num_alignments", 10), pseudo_assembly=kw.get("pseudo", True),
                          report_cigar=True, sam_xa=kw.get("sam_xa", False))
        got = w.batch_single(rb, ro, quals, ro, idb, ido, ov_all, pool_all, score_threshold=thr)
        if got != want:
            a, b = got.split(b"\n"), want.split(b"\n")
            bad = [(i, x, y) for i, (x, y) in enumerate(zip(a, b)) if x != y][:3]
            raise AssertionError((kw, len(a), len(b), bad))
