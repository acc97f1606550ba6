"""The batch's insert-size limit (getMaxAllowedInsertSize, PairedOverlap.h:314-360) from its two inputs: the value counts that
the device histogram feeds (kslam_insert_size_limit_counts) and the compact pair records (kslam_insert_size_limit_compact).
Host code; no GPU involved."""
import ctypes as C
import math

import numpy as np
import pytest

from _lib import load_pkg

pkg = load_pkg()


def limit_compact(values, threads=0):
    rec = np.zeros(len(values), dtype=pkg.PAIR_COMPACT_DT)
    rec["insert_size"] = np.asarray(values, dtype=np.uint32)
    return int(pkg.lib().kslam_insert_size_limit_compact(rec.ctypes.data if len(rec) else None, len(rec), threads))


def limit_counts(values):
    v = np.asarray(values, dtype=np.uint32)
    top = int(v.max()) if len(v) else 0
    counts = np.bincount(v, minlength=top + 1).astype(np.uint64)
    return int(pkg.lib().kslam_insert_size_limit_counts(counts.ctypes.data_as(C.c_void_p), top))


def limit_numpy(values):
    """insert_size_limit_from_runs (sam.cu) over the non-zero values taken as int32, restated from the reference's text."""
    v = np.sort(np.asarray(values, dtype=np.uint32).view(np.int32))
    v = v[v != 0].astype(np.int64)
    n = len(v)
    if n == 0:
        return 0xFFFFFFFF
    spike = 0
    for pc in range(99):
        here, nxt = v[math.floor(n * pc / 100.0)], v[math.floor(n * (pc + 1) / 100.0)]
        if nxt - here > 1000:
            spike = int(v[n * pc // 100])
            break
    q1, q3 = int(v[math.floor(n * 0.25)]), int(v[math.floor(n * 0.75)])
    ceiling = spike if spike else q3 + 2 * (q3 - q1)
    if ceiling == 0:
        ceiling = 2**31 - 1
    kept = v[(v >= 0) & (v <= ceiling)]
    if len(kept) == 0:
        return 0xFFFFFFFF
    sq = (kept.astype(np.uint64) * kept.astype(np.uint64)).astype(np.uint32).view(np.int32).astype(np.int64)   # int square
    mean = float(int(kept.sum())) / len(kept)      # every partial sum is an integer below 2^53: the sum is exact
    sigma = math.sqrt(float(int(sq.sum())) / len(kept) - mean * mean)
    return int(math.floor(mean + 6 * sigma))


def proper(rng, n, mean=350, sd=35):
    return np.clip(np.rint(rng.normal(mean, sd, n)), 151, 600).astype(np.uint32)


def with_singles(rng, v, frac=0.3):
    """interleave single-ended records (insert size 0), which never enter the statistic"""
    out = np.zeros(len(v) + int(len(v) * frac), dtype=np.uint32)
    pos = np.sort(rng.choice(len(out), len(v), replace=False))
    out[pos] = v
    return out


def distributions():
    rng = np.random.default_rng(5)
    far = np.concatenate([proper(rng, 9000), rng.integers(3000, 3600, 1000).astype(np.uint32)])
    wide = np.concatenate([proper(rng, 5000), rng.integers(4096, 200_000, 1500).astype(np.uint32)])
    return {
        "proper": with_singles(rng, proper(rng, 20_000)),
        "far_cluster": with_singles(rng, rng.permutation(far)),       # 10 % far out: a percentile step > 1000 (spike)
        "above_4096": with_singles(rng, rng.permutation(wide)),
        "above_4096_only": rng.integers(4096, 1 << 21, 3000).astype(np.uint32),
        "one_value": np.full(7, 333, np.uint32),
    }


@pytest.mark.parametrize("name", list(distributions()))
def test_counts_equal_compact(name):
    v = distributions()[name]
    want = limit_numpy(v)
    assert limit_compact(v, 1) == want
    assert limit_counts(v) == want


def test_far_cluster_takes_the_spike_branch():
    v = distributions()["far_cluster"]
    nz = np.sort(v[v > 0]).astype(np.int64)
    n = len(nz)
    steps = [nz[math.floor(n * (pc + 1) / 100.0)] - nz[math.floor(n * pc / 100.0)] for pc in range(99)]
    assert max(steps) > 1000
    assert limit_counts(v) < 3000 < int(nz.max())        # the spike cuts the far cluster off


def test_only_single_ended_records():
    v = np.zeros(5000, np.uint32)
    assert limit_compact(v, 1) == 0xFFFFFFFF
    assert limit_counts(v) == 0xFFFFFFFF
    assert limit_compact(np.zeros(0, np.uint32)) == 0xFFFFFFFF


@pytest.mark.parametrize("threads", [1, 16])
def test_threaded_counts(threads):
    """n >= 2^20 records: the compact function splits them over host threads"""
    rng = np.random.default_rng(6)
    v = with_singles(rng, np.concatenate([proper(rng, 1_200_000), rng.integers(4096, 300_000, 60_000).astype(np.uint32)]), 0.1)
    assert len(v) >= 1 << 20
    want = limit_numpy(v)
    assert limit_compact(v, threads) == want
    assert limit_counts(v) == want


@pytest.mark.parametrize("name,extra", [
    ("beyond_2p22", lambda rng: rng.integers(1 << 22, 1 << 26, 40)),
    ("mostly_beyond_2p22", lambda rng: rng.integers(1 << 22, 1 << 28, 30_000)),
    ("beyond_2p31", lambda rng: (2**32 - rng.integers(1, 5000, 60)).astype(np.uint64)),   # negative as int32
    ("both", lambda rng: np.concatenate([rng.integers(1 << 22, 1 << 25, 50), 2**32 - rng.integers(1, 900, 500)])),
])
def test_compact_beyond_the_histogram(name, extra):
    """values >= 2^22 (and >= 2^31, i.e. negative int32) never reach the device histogram: the host path sorts them"""
    rng = np.random.default_rng(7)
    v = np.concatenate([proper(rng, 20_000), np.asarray(extra(rng), dtype=np.uint64).astype(np.uint32)])
    v = with_singles(rng, rng.permutation(v), 0.05)
    assert int(v.max()) >= 1 << 22
    assert limit_compact(v, 1) == limit_numpy(v)
    assert limit_compact(v, 4) == limit_numpy(v)
