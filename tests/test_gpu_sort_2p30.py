"""GPU tier: sorts of 2^30 records or more, where the radix pass switches from 32-bit to 64-bit tile states (a per-digit
prefix no longer fits the 30 value bits of a 32-bit state)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CHUNK = 1 << 26


def test_sort_records_beyond_2p30(pkg):
    """2^30 + 2^20 16-byte records sorted on bits [0, 16) through Aligner.sort_records. All but about 2^19 records have low
    byte 0, so the prefixes of that digit pass 2^30 in the first pass; the second byte is random. Keys non-decreasing,
    input indices (in id_flags) strictly rising within equal keys, and every output record equal to the input record its
    index names: together a stable permutation. Needs about 50 GB of host memory (input, sorted copy, checks in chunks)."""
    n = (1 << 30) + (1 << 20)
    rng = np.random.default_rng(11)
    recs = np.zeros(n, dtype=pkg.KMER_DT)
    k = rng.integers(0, 2**63, size=n, dtype=np.uint64)
    k &= ~np.uint64(0xFF)
    k[::2048] |= rng.integers(0, 256, size=len(k[::2048]), dtype=np.uint64)
    recs["kmer"] = k
    recs["offset"] = (k >> np.uint64(32)).astype(np.uint32)
    del k
    recs["id_flags"] = np.arange(n, dtype=np.uint32)
    zeros = n - int(np.count_nonzero(recs["kmer"][::2048] & np.uint64(0xFF)))
    assert zeros > 1 << 30
    with pkg.Aligner() as al:
        got, _ms = al.sort_records(recs, 0, 16)
    m16 = np.uint64(0xFFFF)
    for a in range(0, n, CHUNK):
        b = min(n, a + CHUNK + 1)                      # one record of overlap with the next chunk
        key = got["kmer"][a:b] & m16
        idx = got["id_flags"][a:b]
        assert (key[1:] >= key[:-1]).all(), a
        tie = key[1:] == key[:-1]
        assert (idx[1:][tie] > idx[:-1][tie]).all(), a
        src = recs[idx]
        for f in ("kmer", "id_flags", "offset"):
            assert np.array_equal(src[f], got[f][a:b]), (a, f)


def test_one_word_seeds_beyond_2p30(pkg):
    """One batch with at least 2^30 raw seeds, sorted as one-word seeds. The genome is AC repeated over 64 kbp; genome
    k-mers are taken every 16 bases, so all 4095 of them are the same k-mer, and half the positions of every read cut from
    it match each of them: 880 reads of 640 bases give about 1.1 G raw seeds and 14.5 M unique ones. The seeds equal those
    of the same reads aligned as two batches of 440 (below 2^30 raw seeds each), read ids mapped back."""
    glen, rlen, n_reads = 1 << 16, 640, 880
    gb = np.frombuffer(b"AC" * (glen // 2), dtype=np.uint8)
    go = np.array([0, glen], dtype=np.uint64)
    starts = (np.arange(n_reads, dtype=np.int64) * 37) % (glen - rlen + 1)
    rb = np.concatenate([gb[s:s + rlen] for s in starts])
    ro = np.arange(n_reads + 1, dtype=np.uint64) * np.uint64(rlen)
    half = n_reads // 2
    with pkg.Aligner(report_cigar=False) as al:
        al.load_genomes(gb, go)
        al.align_batch(rb, ro, copy=False)
        assert al.timings()["n_raw_seeds"] >= 1 << 30
        whole = al.seeds()
        parts = []
        for lo, hi in ((0, half), (half, n_reads)):
            al.align_batch(rb[lo * rlen:hi * rlen], ro[lo:hi + 1] - ro[lo], copy=False)
            assert al.timings()["n_raw_seeds"] < 1 << 30
            s = al.seeds()
            s["read"] += lo
            parts.append(s)
    assert np.array_equal(whole, np.concatenate(parts))
