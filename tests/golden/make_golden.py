"""Generate tests/golden/*.npz from the reference's own code (oracle/_ref/libkslam_ref.so).

Run here (the container that has /root/reference): `python tests/golden/make_golden.py`.
The reference ships no golden vectors for this path (SURVEY.md §4), so these fixtures — inputs plus
the outputs of the UNMODIFIED reference functions — are what pins the oracle and the CUDA path on
machines where the reference sources are absent. Inputs are seeded (k-slam_b200/synth.py).
"""
import os
import sys
import zipfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import _lib as T  # noqa: E402

synth = T.load_pkg().synth


def savez_lzma(path, **arrays):
    """np.savez_compressed with LZMA members instead of deflate (np.load reads both): the k-mer lists of the pipeline
    fixtures compress to well under the 1 MB a stored file may take."""
    with zipfile.ZipFile(path, "w", zipfile.ZIP_LZMA) as z:
        for k, a in arrays.items():
            with z.open(k + ".npy", "w", force_zip64=True) as f:
                np.lib.format.write_array(f, np.asanyarray(a), allow_pickle=False)


def pipeline_fixture(name, gb, go, rb, ro, params):
    R = T.Ref(gb, go, rb, ro, params)
    read_k = R.kmers(1)
    gen_k = R.kmers(2)
    R.kmers(3, sort=True)
    raw = R.seeds(raw=True)
    raw = np.sort(raw, order=["read", "entry", "rel", "rev_comp"])  # multiset: order is not contractual
    seeds = R.seeds(raw=False)
    ov, pool = R.align_to_database()
    ovs, pools, pairs = R.screen_and_pair()
    savez_lzma(
        os.path.join(HERE, name), gen_bases=gb, gen_offs=go, read_bases=rb, read_offs=ro,
        params=np.array([params.match, params.mismatch, params.gap_open, params.gap_extend,
                         params.score_threshold, params.report_cigar], dtype=np.int64),
        read_kmers=read_k, genome_kmers=gen_k, raw_seeds_sorted=raw, seeds=seeds, overlaps=ov,
        cigar_pool=pool, pair_sorted_overlaps=ovs, pair_sorted_cigar_pool=pools, pairs=pairs)
    print(name, "reads", len(ro) - 1, "kmers", len(read_k), len(gen_k), "raw", len(raw), "seeds", len(seeds),
          "pairs", len(pairs))


def ssw_fixture(name, q, qo, r, ro, params, cigar_cap=32):
    a, pool = T.ref_ssw_batch(q, qo, r, ro, params, cigar_cap=cigar_cap)
    assert (a["cigar_len"] <= cigar_cap).all()
    np.savez_compressed(os.path.join(HERE, name), q=q, qoffs=qo, r=r, roffs=ro,
                        params=np.array([params.match, params.mismatch, params.gap_open, params.gap_extend,
                                         params.score_threshold, params.report_cigar], dtype=np.int64),
                        expect=a, cigar_pool=pool)
    print(name, len(a), "alignments; score range", a["sw_score"].min(), a["sw_score"].max())


def fastq_fixture(name):
    """A small paired FASTQ (CRLF and LF mixed, tricky ids, '@' quality lines, no final newline) and what the
    reference's own reader (FASTQsequence.h:110-165) returns for it in batches of 11."""
    import tempfile
    from test_fastq_ingest import fastq_bytes
    r1 = fastq_bytes(40, 5, b"\n", final_newline=False); r2 = fastq_bytes(40, 6, b"\r\n")
    d = tempfile.mkdtemp()
    p1, p2 = os.path.join(d, "R1.fq"), os.path.join(d, "R2.fq")
    open(p1, "wb").write(r1); open(p2, "wb").write(r2)
    batches = T.ref_read_fastq(p1, p2, 11)
    fields = [f for b in batches for rec in b for f in rec]
    np.savez_compressed(os.path.join(HERE, name), r1=np.frombuffer(r1, np.uint8), r2=np.frombuffer(r2, np.uint8), max_reads=11,
                        fields=np.frombuffer(b"".join(fields), np.uint8), field_lens=np.array([len(f) for f in fields], np.int64),
                        batch_sizes=np.array([len(b) for b in batches], np.int64))


def sam_fixture(name):
    """Reference SAM text (SLAM.h:215-239 chain + SAM.h) for a small config-1-like batch, with its inputs."""
    from test_sam_host import make_inputs, reference_side
    gb, go, rb, ro, quals, idb, ido = make_inputs(T.load_pkg(), 5, n_pairs=300, kind="config1")
    ov, pool, pairs, text, mi, _ = reference_side(gb, go, rb, ro, quals, 1)
    R = T.Ref(gb, go, rb[:0], ro[:1], T.default_params()); hdr = T.ref_sam_header(R, "SLAM golden"); R.close()
    np.savez_compressed(os.path.join(HERE, name), gb=gb, go=go, rb=rb, ro=ro, quals=quals, ids=idb, id_offs=ido, ov=ov, pool=pool, pairs=pairs,
                        sam=np.frombuffer(text, np.uint8), max_insert=mi, header=np.frombuffer(hdr, np.uint8))


def sam_digest_fixture(name):
    """Digest of the reference's SAM text (SLAM.h:215-239 chain + SAM.h) for a 6000-pair batch, too large to store at
    > 1 MB. test_sam_host.py feeds the library the oracle's alignments for this batch, so they are checked here against
    the reference's (every overlap field but cigar_off, the CIGARs, the pairs) before the text is digested.
    The file in the repository was NOT made by this function: it was recorded where the reference sources were absent,
    from the library's SAM writer on the oracle's alignments, with sam.cu as it stood when test_sam_host.py last compared
    this batch (on the reference's alignments) with the reference's text. Nothing in the repository shows that the two
    agree on this batch; on the 300-pair batch of the same genomes they do (sam_config1_mini.npz). Running this function
    where the reference exists settles it: the same arrays mean the digest is the reference's."""
    from test_sam_host import crc32_of, make_inputs, oracle_side, reference_side, sam_digest
    gb, go, rb, ro, quals, idb, ido = make_inputs(T.load_pkg(), 5, n_pairs=6000, kind="random")
    ov, pool, pairs = oracle_side(gb, go, rb, ro)
    rov, rpool, rpairs, text, mi, _ = reference_side(gb, go, rb, ro, quals, 1)
    assert len(ov) == len(rov) and all(np.array_equal(ov[f], rov[f]) for f in ov.dtype.names if f != "cigar_off"), "overlaps"
    assert T.cigars_of(ov, pool) == T.cigars_of(rov, rpool), "cigars"
    assert np.array_equal(pairs, rpairs), "pairs"
    np.savez_compressed(os.path.join(HERE, name), max_insert=mi, inputs_crc32=crc32_of(gb, go, rb, ro, quals, idb, ido),
                        alignments_crc32=crc32_of(ov, pool, pairs), **sam_digest(text))
    print(name, "sam bytes", len(text), "lines", text.count(b"\n"))


def meta_fixture(name):
    """Metagenomic run of the reference on a small GenBank database (its own createIndexFromGBFF, SLAM.h:209-265 with one
    OpenMP thread): the GenBank text, the taxDB file, the batch's alignments and the four output texts."""
    import pathlib
    import tempfile
    from test_taxon_host import make_db, make_reads
    pkg = T.load_pkg()
    tmp = pathlib.Path(tempfile.mkdtemp())
    gb, go, _, _, _, _, taxdb, paths = make_db(pkg, tmp, n_strains=10, length=6000, files=1)
    L = T.ref()
    assert T.ref_parse_index(0, paths, taxdb) is not None
    rt = L.kref_taxdb_open(taxdb.encode())
    L.kref_set_threads(1)
    rb, ro, quals, idb, ido = make_reads(pkg, gb, go, 200, seed=31)
    R = T.Ref(gb, go, rb, ro, T.default_params(report_cigar=1))
    L.kref_use_parsed_index(R.h)
    R.align_to_database()
    ov, pool, pairs = R.screen_and_pair()
    sam = T.ref_meta_batch(R, rt, quals, ro, idb, ido)
    per_read, xml, abbreviated = T.ref_meta_finish(R, rt, (len(ro) - 1) // 2)
    R.close(); L.kref_taxdb_close(rt); L.kref_set_threads(os.cpu_count() or 1)
    u = lambda b: np.frombuffer(b, np.uint8)   # noqa: E731
    np.savez_compressed(os.path.join(HERE, name), gbff=u(open(paths[0], "rb").read()), taxdb=u(open(taxdb, "rb").read()), rb=rb, ro=ro,
                        quals=quals, ids=idb, id_offs=ido, ov=ov, pool=pool, pairs=pairs, sam=u(sam), per_read=u(per_read), xml=u(xml),
                        abbreviated=u(abbreviated))
    print(name, "pairs", len(pairs), "sam", len(sam), "xml", len(xml), "taxa", xml.count(b"<taxon>"))


def boost_archive_fixture(name):
    """A small GenBank index written by the REAL Boost.Serialization library (oracle/_ref/boost_archive_probe): the GenBank text
    and the archive bytes."""
    import pathlib
    import subprocess
    import tempfile
    from test_taxon_host import make_db
    from test_database_format import _dump, _probe
    pkg = T.load_pkg()
    from kslam_b200 import database
    tmp = pathlib.Path(tempfile.mkdtemp())
    *_, paths = make_db(pkg, tmp, n_strains=3, length=2500, files=1)
    ix = pkg.Index.parse_genbank(paths)
    ix.write(str(tmp / "ours"))
    (tmp / "dump").write_bytes(_dump(database.read_database(str(tmp / "ours"))))
    subprocess.run([_probe(), str(tmp / "dump"), str(tmp / "real")], check=True)
    u = lambda b: np.frombuffer(b, np.uint8)   # noqa: E731
    np.savez_compressed(os.path.join(HERE, name), gbff=u(open(paths[0], "rb").read()), archive=u((tmp / "real").read_bytes()))
    print(name, "archive bytes", len((tmp / "real").read_bytes()))


def ssw_params_fixtures():
    """Scoring parameters outside the plain-Gotoh domain (SSW's result depends on its striping there)."""
    q, qo, r, ro2 = synth.sw_pairs(800, 130, 150, seed=24)
    for prm in ((5, 4, 10, 10), (2, 8, 3, 3), (1, 1, 1, 1)):
        P = T.default_params(report_cigar=1, match=prm[0], mismatch=prm[1], gap_open=prm[2], gap_extend=prm[3])
        ssw_fixture("ssw_params_%d_%d_%d_%d.npz" % prm, q, qo, r, ro2, P, cigar_cap=256)


def main():
    sys.path.insert(0, os.path.dirname(HERE))
    if len(sys.argv) > 1 and sys.argv[1] == "ssw-params":
        return ssw_params_fixtures()
    if len(sys.argv) > 1 and sys.argv[1] == "meta":
        return meta_fixture("meta_mini.npz")
    if len(sys.argv) > 1 and sys.argv[1] == "boost":
        return boost_archive_fixture("database_boost178.npz")
    if len(sys.argv) > 1 and sys.argv[1] == "sam-digest":
        return sam_digest_fixture("sam_random_6000_digest.npz")
    boost_archive_fixture("database_boost178.npz")
    meta_fixture("meta_mini.npz")
    fastq_fixture("fastq_reader.npz")
    sam_fixture("sam_config1_mini.npz")
    gb, go, rb, ro = synth.adversarial_set(seed=7, n_genomes=8, glen=6000, n_pairs=400)
    pipeline_fixture("pipeline_adversarial_cigar.npz", gb, go, rb, ro, T.default_params(report_cigar=1))
    pipeline_fixture("pipeline_adversarial_thr60.npz", gb, go, rb, ro,
                     T.default_params(report_cigar=0, score_threshold=60))
    gb, go = synth.random_genomes(4, 30_000, seed=1)
    rb, ro, _ = synth.paired_reads(gb, go, 600, seed=2)
    pipeline_fixture("pipeline_config1_mini.npz", gb, go, rb, ro, T.default_params(report_cigar=1))
    q, qo, r, ro2 = synth.sw_pairs(1500, 150, 150, seed=21)
    ssw_fixture("ssw_150x150.npz", q, qo, r, ro2, T.default_params(report_cigar=1))
    q, qo, r, ro2 = synth.sw_pairs(1000, 150, 300, seed=22)
    ssw_fixture("ssw_150x300.npz", q, qo, r, ro2, T.default_params(report_cigar=1))
    q, qo, r, ro2 = synth.sw_pairs(800, 101, 140, seed=23)
    ssw_fixture("ssw_101x140_nocigar.npz", q, qo, r, ro2, T.default_params(report_cigar=0))
    ssw_params_fixtures()


if __name__ == "__main__":
    main()
