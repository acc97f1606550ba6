"""Worker for tests/test_gpu_parity.py::test_switches_give_the_same_results: the library reads its fall-back switches
(KSLAM_SEEDS_EXPAND_AT, KSLAM_SEEDS_16B) once per process, so every setting runs in a process of its own: whole pipeline
on adversarial + related-genome data and the SW stage on diverged pairs with code-4 windows, each against the oracle."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import _lib as T  # noqa: E402
import test_gpu_parity as G  # noqa: E402


def main():
    pkg = T.load_pkg()
    P = T.default_params(report_cigar=1)
    gb, go, rb, ro = pkg.synth.adversarial_set(seed=31, n_genomes=10, glen=15_000, n_pairs=2000)
    G.check_pipeline(pkg, gb, go, rb, ro, P)
    gb, go = pkg.synth.tree_genomes(20, 60_000, seed=5)
    rb, ro, _ = pkg.synth.paired_reads(gb, go, 3000, seed=6)
    G.check_pipeline(pkg, gb, go, rb, ro, P)
    q, qo, r, ro2 = G.diverged_pairs(pkg, 4000, 150, 150, seed=77)
    r = r.copy()
    rng = np.random.default_rng(3)
    for i in range(0, 4000, 2):
        st = int(rng.integers(0, 140))
        r[int(ro2[i]) + st:int(ro2[i]) + st + int(rng.integers(1, 9))] = ord("N")
    want, wpool = T.ko_ssw_batch(q, qo, r, ro2, P, cigar_cap=64)
    with pkg.Aligner(report_cigar=True, max_cigar_ops=64) as al:
        out, pool = al.ssw_batch(q, qo, r, ro2)
    G.check_overlaps(out, pool, want, wpool, fields=G.FIELDS[4:])
    print("SWITCHES-OK")


if __name__ == "__main__":
    main()
