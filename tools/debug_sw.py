"""GPU debugging aid: the SW stage against the oracle on diverged pairs, with per-tier counts and the first mismatches."""
import os, sys, numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, ROOT)
import _lib as T
import importlib.util
pkg = T.load_pkg()
spec = importlib.util.spec_from_file_location("tgp", os.path.join(ROOT, "tests", "test_gpu_parity.py"))
tgp = importlib.util.module_from_spec(spec); spec.loader.exec_module(tgp)
F = ("ref_begin", "ref_end", "query_begin", "query_end", "sw_score")
for shape in [(150, 150), (120, 160), (160, 100)]:
    q, qo, r, ro = tgp.diverged_pairs(pkg, 8000, shape[0], shape[1], seed=3)
    want, _ = T.ko_ssw_batch(q, qo, r, ro, T.default_params(report_cigar=0))
    with pkg.Aligner(report_cigar=False) as al:
        al.set_sw_band(3)
        out, _ = al.ssw_batch(q, qo, r, ro)
        tm = al.timings()
    bad = np.zeros(len(out), bool)
    for f in F:
        bad |= out[f] != want[f]
    print(shape, "mismatch", int(bad.sum()), "of", len(out), "fwd tiers", [tm[k] for k in ("n_sw_tier8", "n_sw_tier16", "n_sw_tier32", "n_sw_tier48", "n_sw_tier64", "n_sw_tier96", "n_sw_tier128", "n_sw_sweep32", "n_sw_fast")], "rev", tm["n_sw_rev_tier"])
    for i in np.flatnonzero(bad)[:6]:
        w, g = want[i], out[i]
        rows, cols, S = int(w["query_end"]) + 1, int(w["ref_end"]) + 1, int(w["sw_score"])
        print("  i", i, "want", [int(w[f]) for f in F], "got", [int(g[f]) for f in F], "flags", int(g["flags"]), "fwd width", shape[0] + shape[1] - 2 * ((S + 1) // 2) + 1)
