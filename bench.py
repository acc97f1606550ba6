#!/usr/bin/env python
"""bench.py — the matching path's headline metric on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload config2|config1|config3] [--pairs P]
  python bench.py --impl reference ...      # the reference's own CPU implementation (oracle/_ref), rank 0 only

A step = one pass of the hot path (alignToDatabase + score screen + getPairedOverlaps, SLAM.h:209-214) over
one batch of synthetic read pairs. `value` is measured with the batch already packed-resident in HBM
(kslam_align_resident + kslam_pair_batch, no result copy); `e2e` goes through the reference-facing C-ABI call
with HOST buffers (kslam_align_batch + kslam_pair_batch with results copied back), host<->device copies inside
the timed region. Ranks shard read pairs (weak scaling: every rank owns a full batch, the genome index is
replicated, no collective on the data path); the timed region is bracketed by barrier + synchronize and the
MAX over ranks is taken. One JSON line on stdout from rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
T_START = time.time()
EXTRAS_BUDGET_S = float(os.environ.get("KSLAM_BENCH_EXTRAS_BUDGET_S", "480"))   # no further secondary block is started after this many seconds
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

METRIC = "M read-pairs/min end-to-end at 1/2/4/8 B200; SW GCUPS; k-mer join GB/s"
UNIT = "M read-pairs/min"


# stdout carries exactly ONE JSON line: libraries that print there (NCCL's version banner ...) are sent to stderr
_REAL_STDOUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(obj):
    _REAL_STDOUT.write(json.dumps(obj) + "\n")
    _REAL_STDOUT.flush()


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t_begin=None, t_end=None):
        """Summarise the samples that arrived inside [t_begin, t_end] (the timed region)."""
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for t, r in self.rows if (t_begin is None or t >= t_begin) and (t_end is None or t <= t_end + 0.05)]
        if not rows:   # region shorter than one sampling period: fall back to the samples taken under warm-up load
            rows = [r for _, r in self.rows[-5:]]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_workload(pkg, name, pairs, seed_shift=0, pin=False, reads=True):
    """Synthetic workload of a named shape, generated with torch on the GPU when there is one (k-slam_b200/synth_torch.py:
    same distributions as synth.py; 10 M pairs + 1 Gbp of genomes in seconds instead of ~90 s of numpy)."""
    import torch
    from kslam_b200 import synth_torch as st
    t0 = time.time()
    if name in ("config1", "config5"):
        gdev, go = st.random_genomes(50, 3_000_000, seed=1, keep_device=True)
        desc = f"config1-shape: {pairs} x 150bp FR pairs from 50 x 3 Mbp random genomes"
    elif name == "config2":
        gdev, go = st.tree_genomes(500, 2_000_000, seed=1, keep_device=True)
        desc = (f"config2-shape (metagenomic): {pairs} x 150bp FR pairs vs 500 x 2 Mbp genomes in a 5/25/100/500 "
                "phylogeny (multi-genome piles)")
    elif name == "config4":
        ng = int(os.environ.get("KSLAM_CONFIG4_GENOMES", "500"))
        gdev, go = st.random_genomes(ng, 4_000_000, seed=1, keep_device=True)
        desc = (f"config4-shape (k-mer-range partitioned DB): {pairs} x 150bp FR pairs per GPU vs {ng} x 4 Mbp genomes "
                f"({ng * 250_000 / 1e6:.0f} M genome k-mer records range-partitioned across the GPUs, NCCL all-to-all both ways)")
    else:
        raise SystemExit(f"unknown workload {name}")
    rb = ro = None
    if reads:
        rb, ro = st.paired_reads(gdev, go, pairs, seed=2 + seed_shift, pin=pin)
    gb = st._host(gdev)
    del gdev
    if torch.cuda.is_available():
        torch.cuda.empty_cache()
    log(f"[bench] generated {desc} in {time.time() - t0:.1f}s")
    return gb, go, rb, ro, desc


def make_comm(pkg, al, rank, world, local):
    """kslam_comm for this rank: rank 0 draws the NCCL unique id, torch.distributed (the launcher's rendezvous) hands it out;
    from then on the exchanges are the library's own ncclSend / ncclRecv (csrc/comm.cu)."""
    import torch
    if world == 1:
        return pkg.Comm.init_rank(al, 0, 1, pkg.Comm.unique_id())
    import torch.distributed as dist
    uid = torch.frombuffer(bytearray(pkg.Comm.unique_id() if rank == 0 else bytes(128)), dtype=torch.uint8).to(f"cuda:{local}")
    dist.broadcast(uid, src=0)
    return pkg.Comm.init_rank(al, rank, world, bytes(uid.cpu().numpy().tobytes()))


def config4_block(args, pkg, rank, world, local, barrier):
    """Config 4: the genome k-mer list range-partitioned by k-mer prefix over the GPUs of the job, read k-mers routed to their
    key owner and raw matches routed back with NCCL all-to-alls issued by the C++ host (kslam_comm, csrc/comm.cu). The
    database grows with the job: 625 x 4 Mbp genomes per GPU (8 GPUs: the named 5,000 genomes, 20 Gbp, 1.25 G k-mer
    records); it is generated ON each GPU and handed to the library as a device pointer. COLLECTIVE: every rank calls this."""
    import torch
    from kslam_b200 import synth_torch as st
    ng = int(os.environ.get("KSLAM_CONFIG4_GENOMES_PER_GPU", "625")) * world
    L, pairs = 4_000_000, args.pairs or 2_000_000
    dev = torch.device("cuda", local)
    g = st._gen(1, dev)
    gdev = torch.empty(ng * L, dtype=torch.uint8, device=dev)
    for lo in range(0, ng * L, 1 << 30):                    # the same seed on every rank: identical databases
        hi = min(ng * L, lo + (1 << 30))
        gdev[lo:hi] = st._acgt((hi - lo,), g, dev)
    go = np.arange(ng + 1, dtype=np.uint64) * np.uint64(L)
    al = pkg.Aligner(report_cigar=False, device=local)
    al.set_debug_taps(False)
    t0 = time.time()
    al.load_genomes_part(gdev, go, rank, world)
    t_load = time.time() - t0
    rb, ro = st.paired_reads(gdev, go, pairs, seed=2 + rank, pin=True)
    del gdev
    torch.cuda.empty_cache()
    comm = make_comm(pkg, al, rank, world, local)
    al.upload_reads(rb, ro)
    for _ in range(2):
        comm.align_resident(fetch=False); al.pair_batch(fetch=False)
    steps = 5
    acc = {}
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        comm.align_resident(fetch=False); al.pair_batch(fetch=False)
        for k, v in comm.stats().items():
            acc[k] = acc.get(k, 0) + v / steps
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    dt = float(dt[0])
    part = al.partition()
    tm = al.timings()
    comm.close(); al.close()
    xk = acc["bytes_sent_kmers"] / (acc["ms_exchange_kmers"] / 1e3) / 1e9 if acc["ms_exchange_kmers"] > 0 else 0.0
    xm = acc["bytes_sent_matches"] / (acc["ms_exchange_matches"] / 1e3) / 1e9 if acc["ms_exchange_matches"] > 0 else 0.0
    step_ms = dt / steps * 1e3
    return {"workload": f"config4: {ng} x 4 Mbp genomes ({part['n_genome_kmers_total'] / 1e6:.0f} M genome k-mer records, {16 * part['n_genome_kmers_total'] / 1e9:.1f} GB) "
                        f"range-partitioned by k-mer prefix over {world} GPUs; {pairs} x 150bp pairs per GPU per step; exchanges = ncclSend/ncclRecv groups issued by libkslam (kslam_comm)",
            "value": pairs * world * steps / dt * 60 / 1e6, "unit": UNIT, "n_gpus": world, "ms_per_step": step_ms, "scaling": "weak (reads and database grow with the job)",
            "index_build_s": t_load, "rank0_stage_ms": {k: acc[k] for k in acc if k.startswith("ms_")} | {"ms_pair": tm["ms_pair"]},
            "exchange": {"rank0_bytes_sent_per_step": {"kmers": acc["bytes_sent_kmers"], "matches": acc["bytes_sent_matches"]},
                         "nvlink_gbs_out_of_rank0": {"kmers": xk, "matches": xm}, "peak_gbs_per_direction": 770.0,
                         "share_of_step": (acc["ms_exchange_kmers"] + acc["ms_exchange_matches"]) / step_ms,
                         "routing_share_of_step": (acc["ms_bucket_kmers"] + acc["ms_bucket_matches"]) / step_ms,
                         "extract_prefilter_share_of_step": (acc["ms_route"] - acc["ms_bucket_kmers"]) / step_ms,
                         "note": "exchange = device time of the two ncclSend/ncclRecv groups (CUDA events on the ctx stream); routing = the two bucketing steps the partition adds "
                                 "(count + scatter by destination); extract + prefilter is the same work the replicated path does; "
                                 "peak = the measured 770 GB/s peer copy per direction (B200_PROFILING.md)"}}


def reference_run(pkg, gb, go, rb, ro, report_cigar, threshold=0, keep=False, threads=0):
    """The reference's own alignToDatabase + screen + getPairedOverlaps (oracle/_ref, all host threads; the oracle port where
    _ref is absent) on the given reads. -> (seconds, cores, kind, outputs or None)"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _lib as T
    P = T.default_params(report_cigar=int(report_cigar), score_threshold=threshold)
    out = None
    if T.have_ref():
        T.ref().kref_set_threads(threads or os.cpu_count() or 1)     # torchrun exports OMP_NUM_THREADS=1: ask for every core
        R = T.Ref(gb, go, rb, ro, P)
        cores = T.ref().kref_num_threads()
        t0 = time.time()
        R.align_to_database()
        ovs, pools, pairs = R.screen_and_pair()
        dt = time.time() - t0
        if keep:
            out = dict(overlaps=ovs, cigar_pool=pools, pairs=pairs)
        R.close()
        kind = "reference"
    else:
        cores = threads or os.cpu_count() or 1
        t0 = time.time()
        w = T.ko_pipeline(gb, go, rb, ro, P, threads=cores)
        dt = time.time() - t0
        if keep:
            out = dict(overlaps=w["pair_sorted_overlaps"], cigar_pool=w["cigar_pool"], pairs=w["pairs"])
        kind = "port"
    return dt, cores, kind, out


PARITY_FIELDS = ("read", "entry", "rel", "rev_comp", "ref_begin", "ref_end", "query_begin", "query_end", "sw_score", "cigar_len")


def parity_against(al, rb, ro, want, with_cigar):
    """The same reads through the GPU path (C ABI, host buffers), results compared with the reference's field for field:
    the pair-sorted alignment vector (the order getPairedOverlaps leaves it in), the CIGARs and the pair records."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _lib as T
    got = al.align_pair_batch(rb, ro)
    ov, wv = got.sorted_overlaps, want["overlaps"]
    res = {"parity_checked": True, "n_compared": int(len(wv)), "n_pairs_compared": int(len(want["pairs"])),
           "undefined_flagged": int((ov["flags"] & 1).sum()), "cigar_overflow_flagged": int((ov["flags"] & 2).sum())}
    bad = []
    if len(ov) != len(wv):
        bad.append(f"overlap count {len(ov)} != {len(wv)}")
    else:
        bad += [f for f in PARITY_FIELDS if not np.array_equal(ov[f], wv[f])]
        if with_cigar and T.cigars_of(ov, got.cigar_pool) != T.cigars_of(wv, want["cigar_pool"]):
            bad.append("cigars")
    if not np.array_equal(got.pairs, want["pairs"]):
        bad.append("pairs")
    res["identical"] = not bad and res["undefined_flagged"] == 0
    if bad:
        res["differing"] = bad
    return res


def cpu_baseline_block(pkg, al, gb, go, workload, sample, full_pairs, report_cigar, seed=99):
    """cpu_baseline: the reference on `sample` pairs of the workload (bounded), the SAME pairs through the GPU path with
    the outputs compared, and — because the reference re-extracts and re-sorts the genome k-mers with every batch
    (SLAM.h:65-66), a fixed cost a small sample over-weights — a second run on half the sample: the two-point fit
    t = a + b * pairs gives the rate the reference would reach on the full batch."""
    from kslam_b200 import synth_torch as st
    rb, ro = st.paired_reads(gb, go, sample, seed=seed)
    dt, cores, kind, out = reference_run(pkg, gb, go, rb, ro, report_cigar, keep=True)
    block = {"value": sample / dt * 60 / 1e6, "unit": UNIT, "cores": cores, "kind": kind,
             "sample": f"{sample} pairs of the same workload in {dt:.1f}s (alignToDatabase+screen+getPairedOverlaps; the genome k-mers are "
                       "re-extracted and re-sorted per batch as the reference does, so a small sample understates its full-batch rate: see amortised)"}
    block["parity"] = parity_against(al, rb, ro, out, report_cigar)
    half = sample // 2
    rb2 = np.concatenate([rb[:half * 150], rb[sample * 150:(sample + half) * 150]])
    ro2 = np.arange(2 * half + 1, dtype=np.uint64) * np.uint64(150)
    dt2, _, _, _ = reference_run(pkg, gb, go, rb2, ro2, report_cigar)
    b = max(1e-12, (dt - dt2) / (sample - half)); a = max(0.0, dt - b * sample)
    block["amortised"] = {"value": full_pairs / (a + b * full_pairs) * 60 / 1e6, "unit": UNIT, "at_pairs": full_pairs,
                          "fit": {"fixed_s": a, "s_per_pair": b, "points": [[half, dt2], [sample, dt]]},
                          "note": "t = fixed + per_pair * pairs fitted on two sample sizes; value = the reference's projected rate on the full batch"}
    # one host thread (SURVEY.md §8d), on a sixteenth of the sample; one run only, so the per-batch genome work (which a
    # single thread pays in full) stays inside the figure
    try:
        n1 = max(1000, sample // 16)
        rb1 = np.concatenate([rb[:n1 * 150], rb[sample * 150:(sample + n1) * 150]])
        ro1 = np.arange(2 * n1 + 1, dtype=np.uint64) * np.uint64(150)
        t1, c1, _, _ = reference_run(pkg, gb, go, rb1, ro1, report_cigar, threads=1)
        block["one_thread"] = {"value": n1 / t1 * 60 / 1e6, "unit": UNIT, "cores": c1,
                               "sample": f"{n1} pairs in {t1:.1f}s, per-batch genome k-mer extraction + sort included (not amortised)"}
    except Exception as e:   # noqa: BLE001  (a reported extra: never costs the line)
        block["one_thread"] = {"error": str(e)[:200]}
    T_ = sys.modules.get("_lib")
    if T_ is not None and T_.have_ref():
        T_.ref().kref_set_threads(os.cpu_count() or 1)
    log(f"[bench/{workload}] cpu_baseline {block['value']:.3f} M pairs/min on the sample, {block['amortised']['value']:.3f} amortised; one thread {block['one_thread']}; parity {block['parity']}")
    return block


def sw_pairs_chunk(n, read_len, window_len, seed, qbuf, rbuf):
    """One chunk of the config-3 mix, generated on the GPU (sub-chunks of 2 M pairs keep the index tensors small) straight
    into the page-locked host buffers qbuf / rbuf (torch uint8 tensors, reused from chunk to chunk)."""
    from kslam_b200 import synth_torch as st
    import torch
    for k, lo in enumerate(range(0, n, 2_000_000)):
        m = min(2_000_000, n - lo)
        a, _, b, _ = st.sw_pairs(m, read_len, window_len, seed=seed + k, keep_device=True)
        qbuf[lo * read_len:(lo + m) * read_len].copy_(a, non_blocking=True); rbuf[lo * window_len:(lo + m) * window_len].copy_(b, non_blocking=True)
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    return (qbuf.numpy()[:n * read_len], np.arange(n + 1, dtype=np.uint64) * np.uint64(read_len),
            rbuf.numpy()[:n * window_len], np.arange(n + 1, dtype=np.uint64) * np.uint64(window_len))


def config3_block(args, pkg, total_pairs, chunk_pairs, steps=1):
    """Config 3, the Smith-Waterman microbenchmark at its named size: `total_pairs` (read 150, window) pairs per shape,
    streamed in chunks through the batched Aligner::Align entry point (kslam_ssw_upload + kslam_ssw_resident), both shapes
    SURVEY.md §8d names (the live reference window of 150 and the 300-wide one), with and without CIGAR, next to ssw.c
    (oracle/_ref) on the host cores. GCUPS = read x window cells / all SW device time (forward + reverse + traceback)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _lib as T
    shapes = []
    int_peak = None
    for window in (150, 300):
        row = {"read_len": 150, "window_len": window, "pairs": total_pairs, "chunk_pairs": chunk_pairs}
        acc = {False: dict(ms=0.0, cells=0, fwd_rev_ms=0.0, tiers={}), True: dict(ms=0.0, cells=0, fwd_rev_ms=0.0, tiers={})}
        import torch
        qbuf = torch.empty(chunk_pairs * 150, dtype=torch.uint8, pin_memory=True)
        rbuf = torch.empty(chunk_pairs * window, dtype=torch.uint8, pin_memory=True)
        al = pkg.Aligner(report_cigar=False)
        sample = None
        for k, lo in enumerate(range(0, total_pairs, chunk_pairs)):
            n = min(chunk_pairs, total_pairs - lo)
            q, qo, r, ro = sw_pairs_chunk(n, 150, window, 300 + window + 64 * k, qbuf, rbuf)
            if sample is None:
                cs = min(n, args.cpu_sample or 200_000)
                sample = (q[:cs * 150].copy(), qo[:cs + 1], r[:cs * window].copy(), ro[:cs + 1], cs)
            al.ssw_upload(q, qo, r, ro)                            # one upload per chunk, both modes run on it
            for cigar in (False, True):
                al.set_report_cigar(cigar)
                if k == 0:
                    al.ssw_resident()                              # warm-up (allocations)
                for _ in range(steps):
                    al.ssw_resident()
                    tm = al.timings()
                    a = acc[cigar]
                    a["ms"] += tm["ms_total"]; a["cells"] += tm["sw_alu_ops"]; a["fwd_rev_ms"] += tm["ms_sw_forward"] + tm["ms_sw_reverse"]
                    for t in ("n_sw_tier8", "n_sw_tier16", "n_sw_tier32", "n_sw_tier48", "n_sw_tier64", "n_sw_tier96", "n_sw_tier128", "n_sw_sweep32", "n_sw_fast", "n_sw_slow", "n_traceback_dp"):
                        a["tiers"][t] = a["tiers"].get(t, 0) + tm[t]
        if int_peak is None:
            int_peak = al.measure_int_peak()
        for cigar in (False, True):
            a = acc[cigar]
            t = a["ms"] / 1e3 / steps
            row["cigar" if cigar else "score_only"] = {
                "gcups": 150.0 * window * total_pairs / t / 1e9, "ms": t * 1e3, "M_pairs_per_min": total_pairs / t * 60 / 1e6,
                "tiers": {k2: v // steps for k2, v in a["tiers"].items()},
                "int_pipe_frac": (a["cells"] / steps) / (a["fwd_rev_ms"] / steps / 1e3) / int_peak}      # ALU thread-ops of the computed cells / peak
        al.close()
        del qbuf, rbuf
        if not args.no_cpu_baseline and T.have_ref():
            q, qo, r, ro, cs = sample
            P = T.default_params(report_cigar=1)
            t0 = time.time(); want, wpool = T.ref_ssw_batch(q, qo, r, ro, P, cigar_cap=32, threads=os.cpu_count() or 1)
            dt = time.time() - t0
            with pkg.Aligner(report_cigar=True) as al:
                got, gpool = al.ssw_batch(q, qo, r, ro)
            same = all(np.array_equal(got[f], want[f]) for f in PARITY_FIELDS[4:]) and T.cigars_of(got, gpool) == T.cigars_of(want, wpool)
            row["ssw_c_reference"] = {"gcups": 150.0 * window * cs / dt / 1e9, "cores": os.cpu_count() or 1, "sample_pairs": cs, "with_cigar": True,
                                      "parity": {"parity_checked": True, "n_compared": cs, "identical": bool(same)}}
        shapes.append(row)
        log(f"[bench/config3] {row}")
    return {"workload": f"config3 (SW microbench): {total_pairs} read/window pairs per shape in chunks of {chunk_pairs}, scoring 2/3/5/2; mix 70 % 1 % subs, "
                        "20 % one 1-5 bp indel, 5 % unrelated, 5 % with N runs; inputs larger than L2",
            "sw_gcups": shapes[0]["score_only"]["gcups"], "shapes": shapes, "int_peak_thread_ops_per_s": int_peak,
            "roofline": {"bound": "int-pipe", "kernel": "k_sw_band / k_sw_fast", "frac": shapes[0]["score_only"]["int_pipe_frac"],
                         "note": "3 ALU thread-ops per computed cell over the forward + reverse sweep time; peak = VIADDMNMX.S16x2 issue rate measured live"}}


def run_config3(args, pkg):
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the matching path has no CPU fallback")
    total = args.pairs or 100_000_000
    blk = config3_block(args, pkg, total, min(total, 10_000_000), steps=args.steps)
    live = blk["shapes"][0]["score_only"]
    emit({"metric": METRIC, "value": live["M_pairs_per_min"], "unit": "M read/window pairs per min (SW microbench, 150 x 150, score + coordinates)",
          "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": live["ms"], "higher_is_better": True, "scaling": "weak",
          "vs_baseline": None, "dtype": "int16x2", "data": "synthetic", "config": {"workload": blk["workload"], "l2": "inputs larger than L2"},
          "sw_gcups": blk["sw_gcups"], "shapes": blk["shapes"], "int_peak_thread_ops_per_s": blk["int_peak_thread_ops_per_s"], "roofline": blk["roofline"]})


def fixed_ids(n, prefix=b"r"):
    """n read ids of one width ("r00000042"): byte array + offsets without a Python loop"""
    w = 8
    digits = (np.arange(n, dtype=np.int64)[:, None] // (10 ** np.arange(w - 1, -1, -1, dtype=np.int64))[None, :]) % 10
    ids = np.empty((n, w + len(prefix)), dtype=np.uint8)
    ids[:, :len(prefix)] = np.frombuffer(prefix, np.uint8)
    ids[:, len(prefix):] = digits + 48
    return ids.reshape(-1), np.arange(n + 1, dtype=np.uint64) * np.uint64(w + len(prefix))


def config5_block(args, pkg, n_batches, batch_pairs, device=0):
    """Config 5: `n_batches` x `batch_pairs` read pairs streamed through the batch loop (SLAM.h:194-251) — the GPU path with
    CIGARs, then the host stages of a --sam-file run with pseudo-assembly and --num-alignments 10 (insert-size limit PER
    BATCH, screens, pseudo-assembly, SAM text) — GPU and host stages of consecutive batches overlapped as the executable
    does. The per-batch insert-size limits and SAM text are checked against the reference's own chain on sub-sampled
    batches (it needs ~100 s per 10 M pairs on these host cores)."""
    import queue
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _lib as T
    from kslam_b200 import synth_torch as st
    gdev, go = st.random_genomes(50, 3_000_000, seed=1, keep_device=True)
    gb = st._host(gdev)
    tags = [b"g%d" % i for i in range(len(go) - 1)]
    al = pkg.Aligner(report_cigar=True, device=device)
    al.set_debug_taps(False)
    al.load_genomes(gb, go)
    sw = pkg.SamWriter(gb, go, tags, num_alignments=10, pseudo_assembly=True, report_cigar=True)
    n_reads = 2 * batch_pairs
    quals = np.full(n_reads * 150, ord("I"), dtype=np.uint8)
    qo = np.arange(n_reads + 1, dtype=np.uint64) * np.uint64(150)
    idp, _ = fixed_ids(batch_pairs)
    ids = np.concatenate([idp, idp]); ido = np.arange(n_reads + 1, dtype=np.uint64) * np.uint64(9)
    work = queue.Queue(maxsize=1)
    stats = {"sam_bytes": 0, "limits": [], "host_s": 0.0, "gpu_s": 0.0, "gen_s": 0.0}
    import torch
    ring = [torch.empty((2, batch_pairs, 150), dtype=torch.uint8, pin_memory=True) for _ in range(3)]   # being generated | queued | in the host stage

    def host_stage():
        while True:
            item = work.get()
            if item is None:
                return
            rb, ro, so, cg, pr = item
            t0 = time.perf_counter()
            with open(os.devnull, "wb") as sink:
                nbytes, limit = sw.batch(rb, ro, quals, qo, ids, ido, so, cg, pr, out_file=sink)
            stats["host_s"] += time.perf_counter() - t0
            stats["sam_bytes"] += nbytes; stats["limits"].append(int(limit))
    th = threading.Thread(target=host_stage); th.start()
    t_all = time.perf_counter()
    for b in range(n_batches):
        t0 = time.perf_counter()
        rb, ro = st.paired_reads(gdev, go, batch_pairs, seed=500 + b, out=ring[b % 3])
        t1 = time.perf_counter()
        p = al.align_pair_batch(rb, ro)                              # copies out of the ctx's pinned buffers: the next batch reuses them
        stats["gen_s"] += t1 - t0; stats["gpu_s"] += time.perf_counter() - t1
        work.put((rb, ro, p.sorted_overlaps, p.cigar_pool, p.pairs))
    work.put(None); th.join()
    dt = time.perf_counter() - t_all
    pairs = n_batches * batch_pairs
    blk = {"workload": f"config5: {n_batches} batches x {batch_pairs} x 150bp pairs streamed (--num-reads-at-once {batch_pairs}) vs 50 x 3 Mbp genomes, "
                       "pseudo-assembly on, --num-alignments 10, SAM text produced per batch (written to /dev/null)",
           "value": pairs / dt * 60 / 1e6, "unit": UNIT, "wall_s": dt, "includes": "read generation on the GPU (stands in for FASTQ ingest), H2D, matching path with CIGARs, "
           "D2H, per-batch insert-size statistics, screens, pseudo-assembly, SAM text", "stage_busy_s": {k: stats[k] for k in ("gen_s", "gpu_s", "host_s")},
           "sam_bytes": stats["sam_bytes"], "insert_size_limit_per_batch": stats["limits"]}
    # per-batch check against the reference's own chain on sub-sampled batches
    if not args.no_cpu_baseline and T.have_ref():
        cs = 60_000
        checks = []
        q1 = np.full(2 * cs * 150, ord("I"), dtype=np.uint8); qo1 = np.arange(2 * cs + 1, dtype=np.uint64) * np.uint64(150)
        i1, _ = fixed_ids(cs); ids1 = np.concatenate([i1, i1]); ido1 = np.arange(2 * cs + 1, dtype=np.uint64) * np.uint64(9)
        T.ref().kref_set_threads(os.cpu_count() or 1)
        R = None
        t_ref = 0.0
        for b in range(2):
            rb, ro = st.paired_reads(gdev, go, cs, seed=900 + b, frag_mean=350.0 + 40 * b)     # different libraries: different limits
            t0 = time.time()
            if R is None:
                R = T.Ref(gb, go, rb, ro, T.default_params(report_cigar=1))
            else:
                R.L.kref_set_reads(R.h, len(ro) - 1, T._p(T.u8(rb)), T._p(ro))
            R.L.kref_set_read_ids(R.h, T._p(T.u8(ids1)), T._p(ido1))
            R.align_to_database(); R.screen_and_pair()
            want_text, want_limit = T.ref_sam(R, q1, qo1, num_alignments=10)
            t_ref += time.time() - t0
            p = al.align_pair_batch(rb, ro)
            got_text, got_limit = sw.batch(rb, ro, q1, qo1, ids1, ido1, p.sorted_overlaps, p.cigar_pool, p.pairs)
            checks.append({"pairs": cs, "limit_ref": int(want_limit), "limit_ours": int(got_limit), "sam_lines": want_text.count(b"\n"),
                           "sam_identical": want_text == got_text})
        R.close()
        blk["per_batch_check"] = {"batches": checks, "all_identical": all(c["limit_ref"] == c["limit_ours"] and c["sam_identical"] for c in checks),
                                  "reference_s": t_ref}
        blk["cpu_baseline"] = {"value": 2 * cs / t_ref * 60 / 1e6, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "reference",
                               "sample": f"2 x {cs} pairs through the reference's alignToDatabase + pairing + host stages + SAM (its SAM loop is serial)"}
    al.close()
    log(f"[bench/config5] {blk}")
    return blk


def run_fastq_to_sam(args, pkg):
    """--workload sam: the --just-align --sam-file run end to end, FASTQ text + FASTA in, SAM text out (config-1 data),
    through slam.align_to_sam (reader | GPU | host stages + SAM writer pipeline). Wall clock of the whole call, including
    FASTA parsing, index build and pipeline fill; per-stage busy times alongside."""
    import tempfile
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the matching path has no CPU fallback")
    from kslam_b200 import slam
    pairs = args.pairs or 4_000_000
    at_once = 1_000_000
    gb, go = pkg.synth.random_genomes(50, 3_000_000, seed=1)
    rb, ro, _ = pkg.synth.paired_reads(gb, go, pairs, seed=2)
    d = tempfile.mkdtemp(prefix="kslam_bench_")
    fa = os.path.join(d, "db.fa")
    with open(fa, "wb") as f:
        for i in range(len(go) - 1):
            f.write(b">g%02d synthetic\n" % i + gb[int(go[i]):int(go[i + 1])].tobytes() + b"\n")
    paths = []
    for k in range(2):
        rows = rb.reshape(-1, 150)[k * pairs:(k + 1) * pairs]
        p = os.path.join(d, f"R{k + 1}.fq"); paths.append(p)
        with open(p, "wb") as f:
            for lo in range(0, pairs, 100_000):
                blk = rows[lo:lo + 100_000]
                f.write(b"".join(b"@r%d/%d\n" % (lo + i, k + 1) + blk[i].tobytes() + b"\n+\n" + b"I" * 150 + b"\n" for i in range(len(blk))))
    in_bytes = sum(os.path.getsize(p) for p in paths)
    runs = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        st = slam.align_to_sam(pkg, [fa], paths[0], paths[1], os.path.join(d, "out.sam"), reads_at_once=at_once)
        dt = time.perf_counter() - t0
        log(f"[bench/sam] run {i}: {pairs} pairs in {dt:.2f}s, stage busy {st['seconds']}")
        if i >= args.warmup:
            runs.append((dt, st))
    dt = float(np.mean([r[0] for r in runs])); st = runs[-1][1]
    for p in paths + [fa, os.path.join(d, "out.sam")]:
        os.unlink(p)
    os.rmdir(d)
    emit({"metric": METRIC, "value": pairs / dt * 60 / 1e6, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
          "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16x2 (SW) / u64 (k-mers) / f64 (MAPQ)",
          "data": "synthetic",
          "config": {"workload": f"FASTQ -> SAM whole process: {pairs} x 150bp FR pairs (FASTQ text, {in_bytes / 1e9:.2f} GB) vs 50 x 3 Mbp genomes (FASTA), "
                                 f"--num-reads-at-once {at_once}, pseudo-assembly on, 10 alignments per read, CIGAR/MD/NM/MAPQ",
                     "includes": "FASTA parse, index build, FASTQ ingest, GPU matching path, host screens + pseudo-assembly + SAM text, file write"},
          "stage_busy_s": st["seconds"], "sam_bytes": st["sam_bytes"], "batches": st["batches"]})


def cli_block(args, pkg, meta, pairs, runs_timed=1, runs_warm=0):
    """--workload cli / cli-meta: the `SLAM` executable (k-slam_b200/csrc/slam_main.cpp, C++ host over the C ABI) as a user
    runs it, wall clock of the whole process: database load, index build, FASTQ ingest, GPU matching path, host stages, output.
    cli      = config-1 data, FASTA database (built with SLAM --parse-fasta), --just-align --sam-file   (configs 1 / 5)
    cli-meta = config-2 data scaled down (strains in a phylogeny as GenBank flat files with genes + names.dmp / nodes.dmp,
               built with SLAM --parse-genbank / --parse-taxonomy), SAM + LCA XML + _PerRead + _abbreviated   (config 2)."""
    import shutil
    from kslam_b200 import synth_torch as st
    import tempfile
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the matching path has no CPU fallback")
    exe = os.environ.get("KSLAM_BENCH_EXE") or os.path.join(ROOT, "k-slam_b200", "SLAM")   # (the override times another build of the CLI)
    at_once = 1_000_000
    d = tempfile.mkdtemp(prefix="kslam_cli_")
    db = os.path.join(d, "db"); os.mkdir(db)
    t_build = time.perf_counter()
    if meta:
        n_strains, length = 100, 1_000_000
        gb, go = st.tree_genomes(n_strains, length, seed=1)
        nodes, strain_tax = pkg.synth.tree_taxonomy(n_strains)
        pkg.synth.write_taxonomy_dumps(nodes, os.path.join(d, "names.dmp"), os.path.join(d, "nodes.dmp"))
        gbff = os.path.join(d, "all.gbff")
        with open(gbff, "wb") as f:
            for i in range(n_strains):
                f.write(pkg.synth.genbank_text(gb[int(go[i]):int(go[i + 1])].tobytes(), f"NC_{i:06d}", 7_000_000 + i, int(strain_tax[i]),
                                               f"Synthetic strain {i}", i, i % (n_strains // 5), seed=i % (n_strains // 5)))
        subprocess.run([exe, "--parse-genbank", "--output-file", os.path.join(db, "database"), gbff], check=True, cwd=d)
        subprocess.run([exe, "--parse-taxonomy", "--output-file", os.path.join(db, "taxDB"), os.path.join(d, "names.dmp"), os.path.join(d, "nodes.dmp")],
                       check=True, cwd=d)
        what = f"{n_strains} strains x {length} bp in a phylogeny (GenBank flat files, ~1 gene / kb)"
    else:
        gb, go = st.random_genomes(50, 3_000_000, seed=1)
        fa = os.path.join(d, "db.fa")
        with open(fa, "wb") as f:
            for i in range(len(go) - 1):
                f.write(b">g%02d synthetic\n" % i + gb[int(go[i]):int(go[i + 1])].tobytes() + b"\n")
        subprocess.run([exe, "--parse-fasta", "--output-file", os.path.join(db, "database"), fa], check=True, cwd=d)
        what = "50 x 3 Mbp genomes (FASTA)"
    t_build = time.perf_counter() - t_build
    rb, ro = st.paired_reads(gb, go, pairs, seed=2)
    paths = []
    for k in range(2):
        rows = rb.reshape(-1, 150)[k * pairs:(k + 1) * pairs]
        p = os.path.join(d, f"R{k + 1}.fq"); paths.append(p)
        with open(p, "wb") as f:
            for lo in range(0, pairs, 100_000):
                blk = rows[lo:lo + 100_000]
                f.write(b"".join(b"@r%d/%d\n" % (lo + i, k + 1) + blk[i].tobytes() + b"\n+\n" + b"I" * 150 + b"\n" for i in range(len(blk))))
    in_bytes = sum(os.path.getsize(p) for p in paths)
    cmd = [exe, "--db", db, "--sam-file", os.path.join(d, "out.sam"), "--num-reads-at-once", str(at_once)]
    cmd += ["--output-file", os.path.join(d, "out.xml")] if meta else ["--just-align"]
    cmd += paths
    runs = []
    for i in range(runs_warm + runs_timed):
        t0 = time.perf_counter()
        r = subprocess.run(cmd, cwd=d, capture_output=True)
        dt = time.perf_counter() - t0
        if r.returncode != 0:
            raise SystemExit(f"SLAM failed ({r.returncode}): {r.stderr.decode()[-500:]}")
        stages = open(os.path.join(d, "log.txt")).read().strip().splitlines()
        log(f"[bench/cli] run {i}: {pairs} pairs in {dt:.2f}s; last log line: {stages[-1] if stages else ''}")
        if i == runs_warm + runs_timed - 1:
            log("[bench/cli] log.txt of the last run (first / last lines):\n  " + "\n  ".join(stages[:8] + ["..."] + stages[-6:]))
        if i >= runs_warm:
            runs.append(dt)
    dt = float(np.mean(runs))
    out_bytes = {n: os.path.getsize(os.path.join(d, n)) for n in os.listdir(d) if n.startswith("out.")}
    # the reference's OWN executable (oracle/_ref/SLAM_ref, its unmodified main.cpp) on the same files and database directory,
    # bounded by --num-reads; our executable on the same prefix must write the same files
    cpu_baseline = None
    ref_exe = os.path.join(ROOT, "oracle", "_ref", "SLAM_ref")
    try:
        if not args.no_cpu_baseline and subprocess.run([ref_exe, "--version"], capture_output=True, timeout=60).stdout == b"1.0\n":
            sample = args.cpu_sample or (50_000 if meta else 200_000)
            cores = os.cpu_count() or 1
            both = {}
            for tag, exe in (("ref", ref_exe), ("ours", exe)):
                wd = os.path.join(d, "cmp_" + tag); os.mkdir(wd)
                cmd2 = [exe, "--db", db, "--sam-file", "o.sam", "--num-reads", str(sample), "--num-reads-at-once", str(at_once)]
                cmd2 += ["--output-file", "o.xml"] if meta else ["--just-align"]
                t0 = time.perf_counter()
                r = subprocess.run(cmd2 + paths, cwd=wd, capture_output=True, env=dict(os.environ, OMP_NUM_THREADS=str(cores)))
                both[tag] = (time.perf_counter() - t0, r.returncode, wd)
            same = None
            if both["ref"][1] == 0 and both["ours"][1] == 0:
                def body(path):
                    t = open(path, "rb").read()
                    return t[t.index(b"@PG"):].split(b"\n", 1)[1] if path.endswith(".sam") else t
                names = ["o.sam"] + (["o.xml_PerRead"] if meta else [])   # (the XML's gene representatives depend on the reference's thread count)
                same = all(body(os.path.join(both["ref"][2], n)) == body(os.path.join(both["ours"][2], n)) for n in names)
            cpu_baseline = {"value": sample / both["ref"][0] * 60 / 1e6, "unit": UNIT, "cores": cores, "kind": "reference",
                            "sample": f"the reference's own executable (unmodified main.cpp) on the first {sample} pairs of the same files, "
                                      f"whole process, {both['ref'][0]:.1f}s", "same_output_as_ours": same,
                            "ours_on_the_same_sample_s": both["ours"][0]}
            log(f"[bench/cli] reference executable: {sample} pairs in {both['ref'][0]:.1f}s; ours {both['ours'][0]:.2f}s; same output: {same}")
    except Exception as e:   # noqa: BLE001
        log(f"[bench/cli] reference executable leg skipped: {e}")
    shutil.rmtree(d, ignore_errors=True)
    return {"value": pairs / dt * 60 / 1e6, "unit": UNIT, "wall_s": dt,
            "workload": f"SLAM executable, whole process: {pairs} x 150bp FR pairs (FASTQ text, {in_bytes / 1e9:.2f} GB) vs {what}, "
                        f"--num-reads-at-once {at_once}, pseudo-assembly on, 10 alignments per read, "
                        + ("SAM + LCA XML + _PerRead + _abbreviated" if meta else "--just-align SAM"),
            "includes": "process start, CUDA context, DIR/database parse, index build, FASTQ ingest, GPU matching path, host stages, output files",
            "command": " ".join(os.path.basename(c) if os.sep in c else c for c in cmd),
            "output_bytes": out_bytes, "database_build_s": t_build, "cpu_baseline": cpu_baseline}


def run_cli(args, pkg, meta):
    blk = cli_block(args, pkg, meta, args.pairs or (2_000_000 if meta else 4_000_000), runs_timed=args.steps, runs_warm=args.warmup)
    emit({"metric": METRIC, "value": blk["value"], "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
          "ms_per_step": blk["wall_s"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
          "dtype": "int16x2 (SW) / u64 (k-mers) / f64 (MAPQ)", "data": "synthetic",
          "config": {"workload": blk["workload"], "includes": blk["includes"], "command": blk["command"]},
          "output_bytes": blk["output_bytes"], "database_build_s": blk["database_build_s"], "cpu_baseline": blk["cpu_baseline"]})


def run_reference_arm(args, pkg):
    """--impl reference: the reference's CPU path on this box's host cores, same config/metric/unit."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    pairs = args.pairs or DEFAULT_PAIRS[args.workload]
    sample = args.ref_sample or CPU_SAMPLE[args.workload]
    from kslam_b200 import synth_torch as st
    gb, go, _, _, desc = make_workload(pkg, args.workload, pairs, reads=False)
    rb, ro = st.paired_reads(gb, go, sample, seed=99)
    vals = []
    for i in range(args.warmup + args.steps):
        dt, cores, kind, _ = reference_run(pkg, gb, go, rb, ro, args.workload == "config1")
        v = sample / dt * 60 / 1e6
        log(f"[bench/reference] step {i}: {sample} pairs in {dt:.2f}s -> {v:.3f} M pairs/min on {cores} threads")
        if i >= args.warmup:
            vals.append((v, dt))
    v = float(np.mean([x[0] for x in vals])); dt = float(np.mean([x[1] for x in vals]))
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "int16/int32/u64", "data": "synthetic",
           "config": {"workload": desc, "batch_pairs_per_gpu": pairs},
           "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
                            "sample": f"{sample} pairs of the workload per step (same genomes), alignToDatabase+screen+getPairedOverlaps; the genome k-mers "
                                      "are re-extracted and re-sorted with every batch (SLAM.h:65-66), a fixed cost that a sample this small over-weights by "
                                      "about 2x against the full 10 M-pair batch (bench.py's own arm reports the two-point fit as cpu_baseline.amortised)"},
           "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


DEFAULT_PAIRS = {"config1": 1_000_000, "config2": 10_000_000, "config4": 2_000_000}
# bounded CPU samples (pairs): sized for roughly 10-20 s of host work per step on a 16-core box
CPU_SAMPLE = {"config1": 400_000, "config2": 150_000, "config4": 100_000}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="kslam", choices=["kslam", "reference"])
    ap.add_argument("--workload", default=os.environ.get("KSLAM_BENCH_WORKLOAD", "config2"), choices=["config1", "config2", "config3", "config4", "config5", "sam", "cli", "cli-meta"])
    ap.add_argument("--pairs", type=int, default=0, help="read pairs per batch per GPU (default: the config's)")
    ap.add_argument("--ref-sample", type=int, default=0, help="pairs per step for the CPU reference arm (0 = per workload)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="pairs for the cpu_baseline leg (rank 0, N=1; 0 = per workload)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="default workload only: skip the config1 / config3 / config5 / cli blocks")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy (config1 / config2 / config4)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "kslam" or args.workload not in DEFAULT_PAIRS):
        raise SystemExit("--dump-outputs: only the matching-path workloads (config1, config2, config4) write their outputs")

    pkg = ge.load_pkg()
    if args.workload == "config3":
        return run_config3(args, pkg)
    if args.workload == "config5":
        blk = config5_block(args, pkg, args.steps, args.pairs or 10_000_000)
        return emit({"metric": METRIC, "value": blk["value"], "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": 0,
                     "ms_per_step": blk["wall_s"] / args.steps * 1e3,
                     "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16x2 (SW) / u64 (k-mers) / f64 (MAPQ)", "data": "synthetic",
                     "config": {"workload": blk["workload"]}, **{k: v for k, v in blk.items() if k not in ("value", "unit", "workload")}})
    if args.workload == "sam":
        return run_fastq_to_sam(args, pkg)
    if args.workload in ("cli", "cli-meta"):
        return run_cli(args, pkg, args.workload == "cli-meta")
    if args.impl == "reference":
        return run_reference_arm(args, pkg)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the matching path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    pairs = args.pairs or DEFAULT_PAIRS[args.workload]
    # reads land in pinned host memory: the e2e leg hands plain host pointers to the C ABI
    gb, go, rb_host, ro, desc = make_workload(pkg, args.workload, pairs, seed_shift=rank, pin=True)
    # config 1 is the --just-align / --sam-file run: reportCigar is on there (SLAM.h:169); configs 2 and 4 write XML only
    want_cigar = args.workload == "config1"
    al = pkg.Aligner(report_cigar=want_cigar, device=local)
    al.set_debug_taps(False)
    partitioned = args.workload == "config4"
    t0 = time.time()
    if partitioned:
        al.load_genomes_part(gb, go, rank, world)
        comm = make_comm(pkg, al, rank, world, local)
        xstats = {}

        def step_resident():
            comm.align_resident(fetch=False)
            xstats.update(comm.stats())
            al.pair_batch(fetch=False)

        def step_e2e():
            al.upload_reads(rb_host, ro)
            comm.align_resident(fetch=False)
            return None, al.pair_batch(fetch=True, copy=False)
    else:
        al.load_genomes(gb, go)

        def step_resident():
            al.align_resident(fetch=False); al.pair_batch(fetch=False)

        def step_e2e():
            return None, al.align_pair_batch(rb_host, ro, copy=False)
    t_load = time.time() - t0
    log(f"[bench r{rank}] genome index built in {t_load:.2f}s")

    # ---- value: inputs resident in HBM -------------------------------------------------------
    al.upload_reads(rb_host, ro)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step_resident()
    launches0 = al.timings()["kernel_launches"]
    barrier()
    tw0 = time.perf_counter()
    tw_first = tw0
    stage = {}
    for _ in range(args.steps):
        step_resident()
        tm = al.timings()
        for k, v in tm.items():
            if k.startswith("ms_"):
                stage[k] = stage.get(k, 0.0) + v
    barrier()
    tw1 = time.perf_counter()
    t_res = tw1 - tw0                           # library calls are synchronous: wall == device time of the chain
    tm = al.timings()
    launches = (tm["kernel_launches"] - launches0) // max(1, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, al.fetch_pairs(copy=False))

    # ---- e2e: host buffers in, results back on the host ------------------------------------------
    # The reference-facing call with HOST buffers: kslam_align_pair_batch = the body of the batch loop (SLAM.h:209-214),
    # H2D of the reads and D2H of everything the loop keeps inside the timed region. Batches are streamed through TWO
    # contexts on the same GPU (include/kslam.h: "two per GPU to double-buffer"), each driven by its own host thread. A
    # batch is kslam_upload_reads (H2D) | kslam_align_resident + kslam_pair_batch (kernels) | kslam_fetch_pairs (D2H), and
    # a host mutex around the kernel phase hands the GPU from one context to the other, so the copies of one batch always
    # run under the kernels of the other. The partitioned workload runs one context (its NCCL collectives are issued in
    # program order).
    depth = 1 if partitioned else 2
    ctxs = [al]
    if depth == 2:
        al2 = pkg.Aligner(report_cigar=want_cigar, device=local, )
        al2.set_debug_taps(False)
        al2.load_genomes(gb, go)
        ctxs.append(al2)
    last = [None] * depth

    compact = not want_cigar                  # a run without --sam-file keeps only the compact pair records (SURVEY.md §8f-3)

    def run_e2e(n_batches):
        if depth == 1:
            for _ in range(n_batches):
                last[0] = step_e2e()[1]
            return
        e2e_pipeline(ctxs, rb_host, ro, n_batches, local, compact, last)

    run_e2e(max(2, args.warmup - 1))
    barrier()
    tw0 = time.perf_counter()
    run_e2e(args.steps)
    barrier()
    tw3 = time.perf_counter()
    t_e2e = tw3 - tw0
    clocks = sampler.stop(tw_first, tw3) if rank == 0 else None
    h2d = int(rb_host.nbytes + 3 * ro.nbytes)
    d2h = d2h_bytes(last[0], compact and depth == 2)
    if depth == 2:
        al2.close()

    t_max = torch.tensor([t_res, t_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_max, op=dist.ReduceOp.MAX)
    t_res, t_e2e = float(t_max[0]), float(t_max[1])
    total_pairs = pairs * world * args.steps
    value = total_pairs / t_res * 60 / 1e6
    e2e = total_pairs / t_e2e * 60 / 1e6

    int_peak = al.measure_int_peak() if rank == 0 else 0.0
    if rank == 0:
        peak, peak_src = measured_peaks()
        ms = {k: v / args.steps for k, v in stage.items()}
        n_rk, n_raw = tm["n_sorted_kmers"], tm["n_raw_seeds"]     # records actually sorted (after the prefilter)
        passes_kmer = max(1, al.kmer_sort_bits() // 8)     # 8-bit digits over the leading bits the join needs (DESIGN.md §3.2)
        sort_s = ms["ms_sort"] / 1e3
        # dominant HBM-bound kernel: k_rs_onesweep of the read k-mer sort. algorithmic bytes per launch = 32 B x records
        # (one read + one write of every 16 B record per pass); duration = sort time / passes (histogram charged too)
        per_launch_s = sort_s / passes_kmer if sort_s > 0 else float("nan")
        achieved = 32.0 * n_rk / per_launch_s / 1e9 if sort_s > 0 else 0.0
        join_gbs = (32.0 * n_rk + 16.0 * n_rk + 16.0 * n_raw) / ((ms["ms_sort"] + ms["ms_join"]) / 1e3) / 1e9
        sw_s = (ms["ms_sw_forward"] + ms["ms_sw_reverse"] + ms["ms_sw_traceback"] + ms["ms_sw_slow"] + ms["ms_sw_prepare"]) / 1e3
        gcups = tm["sw_cells_forward"] / sw_s / 1e9 if sw_s > 0 else 0.0
        gcups_kernel = (tm["sw_cells_forward"] + tm["sw_cells_reverse"]) / ((ms["ms_sw_forward"] + ms["ms_sw_reverse"]) / 1e3) / 1e9 \
            if ms["ms_sw_forward"] + ms["ms_sw_reverse"] > 0 else 0.0
        hbm_roof = {"bound": "hbm", "kernel": "k_rs_pass2 (read k-mer LSD pass)", "achieved": achieved, "peak": peak,
                    "unit": "GB/s", "frac": achieved / peak,
                    # ncu --set full of this kernel on 32 M records (profiles/r2_ncu_sort_passes.txt): dram read 516.8 MB + write
                    # 471.7 MB per launch = 30.9 B per record (part of the previous pass' output is still in L2): no re-reads
                    "traffic": 30.9 * n_rk, "traffic_source": "ncu dram__bytes_read+write per record (32 M-record capture) x records per launch",
                    "peak_source": peak_src,
                    "share_of_step": ms["ms_sort"] / (t_res / args.steps * 1e3),
                    "note": f"algorithmic 32 B/record/pass; duration = (sort stage incl. histogram)/{passes_kmer} passes, CUDA events on the ctx stream"}
        # SW sweeps (k_sw_band / k_sw_fast): integer-pipe bound. 6 ALU thread-ops (1 PRMT + 5 s16x2 DPX) per two cells
        # (the seventh op of the recurrence, H - gapOpen, is an IMAD on the FMA pipe thanks to the biased cells);
        # numerator = cells the sweep kernels actually computed (band cells, not matrix cells), denominator = the
        # issue rate of VIADDMNMX.S16x2 measured on this GPU right now (kslam_measure_int_peak).
        sweep_s = (ms["ms_sw_forward"] + ms["ms_sw_reverse"]) / 1e3
        int_ops = float(tm["sw_alu_ops"])
        int_ach = int_ops / sweep_s / 1e12 if sweep_s > 0 else 0.0
        int_roof = {"bound": "int-pipe", "kernel": "k_sw_band / k_sw_fast (SW forward + reverse sweeps)", "achieved": int_ach,
                    "peak": int_peak / 1e12, "unit": "T int16x2 thread-ops/s", "frac": int_ach / (int_peak / 1e12) if int_peak else None,
                    "traffic": None, "peak_source": "measured live: dependency-free VIADDMNMX.S16x2 issue-rate microbenchmark (kslam_measure_int_peak)",
                    "share_of_step": sweep_s * 1e3 / (t_res / args.steps * 1e3),
                    "note": "ALU thread-ops the computed cells need: 3 per cell (1 PRMT + 5 DPX per s16x2 cell pair; H - gapOpen is an IMAD on the FMA pipe), 2.5 in the rows a band "
                            "sweep runs without the tracking op (they cannot reach the score bound yet); cells computed = band cells (tier width x rows; n_sw_fwd_tier / n_sw_rev_tier "
                            "count the tiers of 8 16 24 32 40 48 56 64 72 80 96 128 diagonals) or the full matrix for fallback alignments; CUDA events on the ctx stream"}
        dominant = int_roof if sweep_s * 1e3 >= ms["ms_sort"] else hbm_roof
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": t_res / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "int16x2 (SW) / u64 (k-mers)", "data": "synthetic",
               "config": {"workload": desc, "batch_pairs_per_gpu": pairs, "sharding": (f"genome k-mer list range-partitioned over {world} ranks + read pairs per rank; all-to-all of k-mer records "
                                       f"and of raw matches (NCCL)" if partitioned else f"read pairs, {world} ranks, no collective"),
                          "l2": "inputs larger than L2 (3.8 GB+ of k-mer records per step)", "report_cigar": want_cigar},
               "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                       "call": ("kslam_upload_reads + kslam_align_resident + kslam_pair_batch + kslam_fetch_pairs_compact (host buffers in; back on the host: what the batch loop of a run "
                                "without --sam-file keeps — 24-byte pair records, the batch's insert-size limit computed from them, the mates of the pairs beyond it)"
                                if compact and depth == 2 else
                                "kslam_upload_reads + kslam_align_resident + kslam_pair_batch + kslam_fetch_pairs (host buffers in, pair-sorted overlaps + CIGAR pool + pairs back on the host)"),
                       "contexts_per_gpu": depth},
               "gpu_launches": int(launches),
               "clocks": clocks,
               "roofline": dominant, "roofline_hbm": hbm_roof, "roofline_int": int_roof,
               "kmer_join_gbs": join_gbs, "sw_gcups": gcups, "sw_kernel_gcups_fwd_plus_rev": gcups_kernel,
               "stage_ms": ms,
               "counts": {k: tm[k] for k in ("n_read_kmers", "n_sorted_kmers", "n_genome_kmers", "n_raw_seeds", "n_seeds", "n_pairs",
                                             "n_sw_band", "n_sw_band64", "n_sw_fast", "n_sw_slow", "n_sw_band_rev",
                                             "n_sw_tier8", "n_sw_tier16", "n_sw_tier32", "n_sw_tier48", "n_sw_tier64", "n_sw_sweep32",
                                             "n_sw_tier96", "n_sw_tier128", "n_sw_fwd_tier", "n_sw_rev_tier", "n_sw_rev_diagonal",
                                             "sw_cells_forward", "sw_cells_reverse", "sw_cells_computed", "n_sort_passes")},
               "genome_index_build_s": t_load}
        if partitioned:
            out["exchange"] = {"rank0_per_step": xstats, "record_bytes": 16, "issued_by": "libkslam (kslam_comm: ncclSend / ncclRecv groups on the ctx stream)",
                               "partition": {k: (v.tolist() if hasattr(v, "tolist") else v) for k, v in al.partition().items() if k != "splitters"}}
        if world == 1 and not args.no_cpu_baseline:
            cs = args.cpu_sample or CPU_SAMPLE[args.workload]
            out["cpu_baseline"] = cpu_baseline_block(pkg, al, gb, go, args.workload, cs, pairs, want_cigar)
    al.close()
    extras_on = args.workload == "config2" and not args.no_extras and not partitioned
    del gb, rb_host
    # ---- config 4 next to the headline workload whenever the job has more than one GPU (all ranks take part)
    if extras_on and world > 1 and time.time() - T_START < EXTRAS_BUDGET_S:
        try:
            blk = config4_block(args, pkg, rank, world, local, barrier)
        except Exception as e:   # noqa: BLE001
            blk = {"error": f"{type(e).__name__}: {e}"}
        if rank == 0:
            out["configs"] = {"config4": blk}
    if rank == 0:
        # ---- the other named configurations (BASELINE.json configs 1, 3, 5 and the process interface), N = 1 only: bounded
        # blocks of their own next to the headline workload, each with its roofline / cpu_baseline / parity figures
        if extras_on and world == 1:
            extras = {}
            for name, fn in (("config1", lambda: config1_block(args, pkg, local)),
                             ("config3", lambda: config3_block(args, pkg, 100_000_000, 10_000_000)),
                             ("config5", lambda: config5_block(args, pkg, 10, 10_000_000, device=local)),
                             ("cli", lambda: cli_block(args, pkg, False, 1_000_000))):
                t0 = time.time()
                if t0 - T_START > EXTRAS_BUDGET_S:
                    extras[name] = {"skipped": f"time budget ({EXTRAS_BUDGET_S:.0f}s of bench.py run time) spent before this block"}
                    continue
                try:
                    extras[name] = fn()
                except Exception as e:   # noqa: BLE001  (a failing block must not take the headline line with it)
                    extras[name] = {"error": f"{type(e).__name__}: {e}"}
                extras[name]["block_wall_s"] = time.time() - t0
                log(f"[bench] block {name} took {extras[name]['block_wall_s']:.1f}s")
            out["configs"] = extras
        emit(out)
    if world > 1:
        dist.destroy_process_group()


def e2e_pipeline(ctxs, rb, ro, n_batches, device, compact, last):
    """Batches streamed through the contexts of one GPU (include/kslam.h: "two per GPU to double-buffer"), one host thread
    each: kslam_upload_reads (H2D) | kslam_align_resident + kslam_pair_batch (kernels) | fetch (D2H). A host mutex around
    the kernel phase hands the GPU from one context to the other, so the copies of one batch run under the kernels of the
    other. compact: fetch = kslam_fetch_pairs_compact (runs without --sam-file), else kslam_fetch_pairs."""
    import torch
    depth = len(ctxs)
    errs = []
    gpu_turn = threading.Lock()
    trace = bool(os.environ.get("KSLAM_BENCH_TRACE"))

    def worker(k):
        try:
            torch.cuda.set_device(device)
            for _b in range(k, n_batches, depth):
                t0 = time.perf_counter()
                ctxs[k].upload_reads(rb, ro)
                t1 = time.perf_counter()
                with gpu_turn:
                    t2 = time.perf_counter()
                    ctxs[k].align_resident(fetch=False); ctxs[k].pair_batch(fetch=False)
                    t3 = time.perf_counter()
                last[k] = ctxs[k].fetch_pairs_compact(copy=False) if compact else ctxs[k].fetch_pairs(copy=False)
                if trace:
                    log(f"[e2e ctx{k} batch{_b}] upload {t1 - t0:.3f}s wait {t2 - t1:.3f}s kernels {t3 - t2:.3f}s fetch {time.perf_counter() - t3:.3f}s")
        except Exception as e:   # noqa: BLE001
            errs.append(e)
    th = [threading.Thread(target=worker, args=(k,)) for k in range(depth)]
    [t.start() for t in th]; [t.join() for t in th]
    if errs:
        raise errs[0]


def dump_outputs(out_dir, res, seed=0, limit=60 << 20):
    """--dump-outputs DIR: what kslam_fetch_pairs hands the caller after the last timed step (pair-sorted overlaps, their
    CIGARs, pair records), one float64 .npy per field (all are 32-bit integers, exact in float64), so that two builds can
    be compared output for output on the same seeded workload. Larger outputs are cut to a seeded sample of rows, the
    same rows for the same record counts: 2^17 overlaps and 2^18 pairs. cigar_off, a position in this build's CIGAR pool,
    is given as the words it points to: cigar_words holds the whole CIGARs (cigar_len words each) of the sampled overlaps
    in order, as many as fit in `limit` bytes of arrays in all (every one of them unless the sample averages more than
    ~35 words per CIGAR). A workload without CIGARs (config2, config4) has no cigar_words."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(seed)

    def sample(a, k):
        return a if len(a) <= k else a[np.sort(rng.choice(len(a), k, replace=False))]
    ov, pr = sample(res.sorted_overlaps, 1 << 17), sample(res.pairs, 1 << 18)
    arrays = {"counts": [len(res.sorted_overlaps), len(res.pairs)]}
    arrays.update({"sorted_overlaps_" + f: ov[f] for f in ov.dtype.names if f != "cigar_off"})
    arrays.update({"pairs_" + f: pr[f] for f in pr.dtype.names if f != "pad"})
    if len(res.cigar_pool):
        room = (limit - 8 * sum(np.size(a) for a in arrays.values())) // 8          # float64 words left
        k = int(np.searchsorted(np.cumsum(ov["cigar_len"], dtype=np.int64), room, side="right"))
        arrays["cigar_words"] = np.concatenate([res.cigar_pool[o:o + n] for o, n in zip(ov["cigar_off"][:k], ov["cigar_len"][:k])])
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))
    n_cig = f", CIGARs of the first {k}" if "cigar_words" in arrays else ""
    log(f"[bench] wrote {len(arrays)} arrays ({len(ov)} of {len(res.sorted_overlaps)} overlaps{n_cig}, {len(pr)} of {len(res.pairs)} pairs) to {out_dir}")


def d2h_bytes(res, compact):
    if compact:
        return int(res[0].nbytes + res[2].nbytes)
    return int(res.sorted_overlaps.nbytes + res.cigar_pool.nbytes + res.pairs.nbytes)


def config1_block(args, pkg, device):
    """Config 1 (the --just-align --sam-file run, reportCigar on): 1 M pairs vs 50 x 3 Mbp, resident value, e2e through the
    C ABI with pinned host buffers, stage times, the sort's HBM figure, and the reference on a sample with outputs compared."""
    pairs = 1_000_000
    gb, go, rb, ro, desc = make_workload(pkg, "config1", pairs, pin=True)
    al = pkg.Aligner(report_cigar=True, device=device)
    al.set_debug_taps(False)
    al.load_genomes(gb, go)
    al.upload_reads(rb, ro)
    for _ in range(3):
        al.align_resident(fetch=False); al.pair_batch(fetch=False)
    steps = 10
    stage = {}
    t0 = time.perf_counter()
    for _ in range(steps):
        al.align_resident(fetch=False); al.pair_batch(fetch=False)
        tm = al.timings()
        for k, v in tm.items():
            if k.startswith("ms_"):
                stage[k] = stage.get(k, 0.0) + v / steps
    t_res = (time.perf_counter() - t0) / steps
    al2 = pkg.Aligner(report_cigar=True, device=device)
    al2.set_debug_taps(False)
    al2.load_genomes(gb, go)
    last = [None, None]
    e2e_pipeline([al, al2], rb, ro, 4, device, False, last)
    t0 = time.perf_counter()
    e2e_pipeline([al, al2], rb, ro, 2 * steps, device, False, last)
    t_e2e = (time.perf_counter() - t0) / (2 * steps)
    pr = last[0]
    al2.close()
    peak, peak_src = measured_peaks()
    passes = max(1, al.kmer_sort_bits() // 8)
    n_rk = tm["n_sorted_kmers"]
    ach = 32.0 * n_rk / (stage["ms_sort"] / 1e3 / passes) / 1e9
    blk = {"workload": desc + ", CIGARs on", "value": pairs / t_res * 60 / 1e6, "unit": UNIT, "ms_per_step": t_res * 1e3,
           "e2e": {"value": pairs / t_e2e * 60 / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(rb.nbytes + 3 * ro.nbytes),
                   "d2h_bytes_per_step": d2h_bytes(pr, False), "contexts_per_gpu": 2},
           "stage_ms": stage, "roofline_hbm": {"kernel": "k_rs_pass2 (read k-mer LSD pass)", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                               "peak_source": peak_src, "note": f"32 B x {n_rk} records per pass / (sort stage incl. histogram / {passes} passes)"},
           "counts": {k: tm[k] for k in ("n_sorted_kmers", "n_raw_seeds", "n_seeds", "n_pairs", "n_sw_tier8", "n_sw_tier16", "n_sw_tier32", "n_sw_fast", "n_traceback_dp")}}
    if not args.no_cpu_baseline:
        blk["cpu_baseline"] = cpu_baseline_block(pkg, al, gb, go, "config1", 200_000, pairs, True, seed=98)
    al.close()
    return blk


if __name__ == "__main__":
    main()
