"""kslam_b200 — host-side mirror of the reference's matching-path interface over libkslam.so.

The product is the CUDA library behind the C ABI in include/kslam.h; this module is the thin
Python host layer used by the tests, bench.py and the multi-GPU driver. It mirrors the reference's
operator names for this path:

    Aligner.load_genomes   <- GenbankIndex (GenbankTools.h:189-219) handed to alignToDatabase
    Aligner.align_batch    <- alignToDatabase            (/root/reference/src/SLAM.h:60-79)
    Aligner.pair_batch     <- screenOverlapsByScoreThreshold + getPairedOverlaps
                              (/root/reference/src/Overlap.h:329-341, PairedOverlap.h:243-272)
    Aligner.ssw_batch      <- StripedSmithWaterman::Aligner::Align (/root/reference/src/ssw_cpp.cpp:234-283)

There is no CPU fallback: importing works anywhere (so the CPU test tier can check symbols), but every
compute call needs libkslam.so and an sm_100 GPU and raises KslamError otherwise. Nothing here imports
or loads oracle/.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from dataclasses import dataclass

import numpy as np

from . import synth  # noqa: F401  (seeded workload generators)

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
LIB_PATH = os.path.join(PKG_DIR, "libkslam.so")
HEADER = os.path.join(ROOT, "include", "kslam.h")

KMER_DT = np.dtype([("kmer", "<u8"), ("id_flags", "<u4"), ("offset", "<u4")])
SEED_DT = np.dtype([("read", "<u4"), ("entry", "<u4"), ("rel", "<i4"), ("rev_comp", "<u4")])
OVERLAP_DT = np.dtype([("read", "<u4"), ("entry", "<u4"), ("rel", "<i4"), ("rev_comp", "<u4"),
                       ("ref_begin", "<i4"), ("ref_end", "<i4"), ("query_begin", "<i4"), ("query_end", "<i4"),
                       ("sw_score", "<u4"), ("cigar_off", "<u4"), ("cigar_len", "<u4"), ("flags", "<u4")])
PAIR_DT = np.dtype([("combined_score", "<u4"), ("entry", "<u4"), ("ref_start", "<i4"), ("ref_end", "<i4"),
                    ("insert_size", "<u4"), ("r1_idx", "<i4"), ("r2_idx", "<i4"), ("pad", "<u4")])
PAIR_COMPACT_DT = np.dtype([("pair_id", "<u4"), ("entry", "<u4"), ("ref_start", "<i4"), ("ref_end", "<i4"), ("insert_size", "<u4"), ("score_flags", "<u4")])
FAR_MATES_DT = np.dtype([("pair_index", "<u4"), ("score1", "<u4"), ("ref_begin1", "<i4"), ("ref_end1", "<i4"),
                         ("score2", "<u4"), ("ref_begin2", "<i4"), ("ref_end2", "<i4"), ("pad", "<u4")])
GENE_DT = np.dtype([("cds_start", "<u4"), ("cds_stop", "<u4"), ("gene_id", "<u4"), ("complement", "<u4"), ("str_offs", "<u8", (6,))])
GENE_STRINGS = ("gene_name", "locus_tag", "protein_id", "product", "reference_sequence")
FLAG_UNDEFINED = 1
FLAG_CIGAR_OVERFLOW = 2


class KslamError(RuntimeError):
    pass


class Params(C.Structure):
    _fields_ = [("match", C.c_uint8), ("mismatch", C.c_uint8), ("gap_open", C.c_uint8), ("gap_extend", C.c_uint8),
                ("score_threshold", C.c_uint16), ("report_cigar", C.c_uint8), ("reserved0", C.c_uint8),
                ("device", C.c_int32), ("genome_gap", C.c_uint32), ("max_cigar_ops", C.c_uint32),
                ("stream_priority", C.c_uint32)]


class _Alignments(C.Structure):
    _fields_ = [("n_overlaps", C.c_uint64), ("overlaps", C.c_void_p), ("n_cigar_words", C.c_uint64),
                ("cigar_pool", C.c_void_p)]


class _Pairs(C.Structure):
    _fields_ = [("n_sorted", C.c_uint64), ("sorted_overlaps", C.c_void_p), ("n_cigar_words", C.c_uint64),
                ("cigar_pool", C.c_void_p), ("n_pairs", C.c_uint64), ("pairs", C.c_void_p)]


class _PairsCompact(C.Structure):
    _fields_ = [("n_pairs", C.c_uint64), ("pairs", C.c_void_p), ("insert_size_limit", C.c_uint32), ("n_far", C.c_uint64), ("far", C.c_void_p)]


class Timings(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("ms_h2d", "ms_pack", "ms_extract", "ms_sort", "ms_join", "ms_seed_sort",
                                         "ms_unique", "ms_sw_prepare", "ms_sw_forward", "ms_sw_reverse",
                                         "ms_sw_traceback", "ms_sw_slow", "ms_d2h", "ms_pair", "ms_total")] + \
               [("_pad", C.c_float)] + \
               [(n, C.c_uint64) for n in ("n_read_kmers", "n_sorted_kmers", "n_genome_kmers", "n_raw_seeds", "n_seeds", "n_sort_passes",
                                          "sw_cells_forward", "sw_cells_reverse", "sw_cells_computed", "n_sw_fast", "n_sw_slow", "n_sw_band", "n_sw_band64", "n_sw_band_rev", "n_traceback_dp", "n_pairs",
                                          "n_sw_tier8", "n_sw_tier16", "n_sw_tier32", "n_sw_tier48", "n_sw_tier64", "n_sw_sweep32",
                                          "n_sw_tier96", "n_sw_tier128")] + \
               [("n_sw_fwd_tier", C.c_uint64 * 12), ("n_sw_rev_tier", C.c_uint64 * 12), ("n_sw_rev_diagonal", C.c_uint64), ("sw_alu_ops", C.c_uint64), ("kernel_launches", C.c_uint64)]

    def as_dict(self):
        return {n: (list(getattr(self, n)) if n in ("n_sw_rev_tier", "n_sw_fwd_tier") else getattr(self, n)) for n, _ in self._fields_ if n != "_pad"}


class CommStats(C.Structure):
    """kslam_comm_stats (include/kslam.h)"""
    _fields_ = [(n, C.c_float) for n in ("ms_route", "ms_exchange_kmers", "ms_sort", "ms_join", "ms_exchange_matches", "ms_finish")] + \
               [(n, C.c_uint64) for n in ("kmers_sent", "kmers_received", "matches_sent", "matches_received", "bytes_sent_kmers", "bytes_sent_matches")] + \
               [(n, C.c_float) for n in ("ms_bucket_kmers", "ms_bucket_matches")]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class _ReadBatch(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("n_r1", C.c_uint64), ("bases", C.c_void_p), ("offs", C.c_void_p),
                ("quals", C.c_void_p), ("qual_offs", C.c_void_p), ("ids", C.c_void_p), ("id_offs", C.c_void_p)]


class SamParams(C.Structure):
    _fields_ = [("num_alignments", C.c_uint32), ("pseudo_assembly", C.c_uint8), ("report_cigar", C.c_uint8),
                ("sam_xa", C.c_uint8), ("threads", C.c_uint8), ("score_fraction_threshold", C.c_double)]


class _SamDb(C.Structure):
    _fields_ = [("n_entries", C.c_uint64), ("bases", C.c_void_p), ("offs", C.c_void_p), ("locus_tags", C.c_void_p),
                ("locus_offs", C.c_void_p), ("taxonomy_ids", C.c_void_p),
                ("genes", C.c_void_p), ("gene_offs", C.c_void_p), ("gene_strings", C.c_void_p), ("gene_index", C.c_void_p)]


def declared_symbols():
    """Every function the public header declares (used by the CPU-tier symbol test)."""
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(kslam_[a-z_0-9]+)\s*\(", text)))


_lib = None


def lib():
    """dlopen libkslam.so and bind every entry point; raises KslamError (never falls back) if missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise KslamError(f"{LIB_PATH} not built: run `python __graft_entry__.py` (nvcc, sm_100a). "
                         "There is no CPU fallback for the matching path.")
    L = C.CDLL(LIB_PATH)
    missing = [s for s in declared_symbols() if not hasattr(L, s)]
    if missing:
        raise KslamError(f"libkslam.so lacks symbols declared in include/kslam.h: {missing}")
    vp, u64, i32 = C.c_void_p, C.c_uint64, C.c_int
    L.kslam_create.argtypes = [C.POINTER(Params), C.POINTER(vp)]
    L.kslam_destroy.argtypes = [vp]
    L.kslam_destroy.restype = None
    L.kslam_last_error.argtypes = [vp]
    L.kslam_last_error.restype = C.c_char_p
    L.kslam_version.restype = C.c_char_p
    L.kslam_params_exact.argtypes = [C.POINTER(Params)]
    L.kslam_params_fast.argtypes = [C.POINTER(Params)]
    L.kslam_load_genomes.argtypes = [vp, u64, vp, vp]
    L.kslam_align_batch.argtypes = [vp, u64, vp, vp, C.POINTER(_Alignments)]
    L.kslam_upload_reads.argtypes = [vp, u64, vp, vp]
    L.kslam_align_pair_batch.argtypes = [vp, u64, vp, vp, C.POINTER(_Pairs)]
    L.kslam_align_resident.argtypes = [vp, i32, C.POINTER(_Alignments)]
    L.kslam_pair_batch.argtypes = [vp, i32, C.POINTER(_Pairs)]
    L.kslam_fetch_pairs.argtypes = [vp, C.POINTER(_Pairs)]
    L.kslam_ssw_batch.argtypes = [vp, u64, vp, vp, vp, vp, vp, vp]
    L.kslam_ssw_upload.argtypes = [vp, u64, vp, vp, vp, vp]
    L.kslam_ssw_resident.argtypes = [vp, vp, vp]
    for name in ("kslam_get_genome_kmers", "kslam_get_read_kmers", "kslam_get_raw_seeds", "kslam_get_seeds"):
        getattr(L, name).argtypes = [vp, vp, u64]
        getattr(L, name).restype = C.c_int64
    L.kslam_sort_records.argtypes = [vp, vp, u64, C.c_uint32, C.c_uint32, C.POINTER(C.c_float)]
    L.kslam_get_timings.argtypes = [vp, C.POINTER(Timings)]
    L.kslam_set_debug_taps.argtypes = [vp, i32]
    L.kslam_measure_int_peak.argtypes = [vp, C.POINTER(C.c_double)]
    L.kslam_set_prefilter.argtypes = [vp, i32]
    L.kslam_set_report_cigar.argtypes = [vp, i32]
    L.kslam_fetch_pairs_compact.argtypes = [vp, C.c_uint32, C.POINTER(_PairsCompact)]
    L.kslam_insert_size_limit_compact.argtypes = [vp, u64, C.c_uint32]
    L.kslam_insert_size_limit_compact.restype = C.c_uint32
    L.kslam_insert_size_limit_counts.argtypes = [vp, C.c_uint32]
    L.kslam_insert_size_limit_counts.restype = C.c_uint32
    L.kslam_fetch_far_mates.argtypes = [vp, C.c_uint32, C.POINTER(u64), C.POINTER(vp)]
    L.kslam_batch_outputs_compact.argtypes = [C.POINTER(SamParams), C.POINTER(_SamDb), C.POINTER(_ReadBatch), C.POINTER(_PairsCompact), C.POINTER(C.c_uint32), vp, vp]
    L.kslam_comm_unique_id.argtypes = [vp]
    L.kslam_comm_init_rank.argtypes = [vp, C.c_uint32, C.c_uint32, vp, C.POINTER(vp)]
    L.kslam_comm_init_all.argtypes = [C.c_uint32, C.POINTER(vp), C.POINTER(vp)]
    L.kslam_comm_destroy.argtypes = [vp]
    L.kslam_comm_destroy.restype = None
    L.kslam_comm_rank.argtypes = [vp, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    L.kslam_comm_align_resident.argtypes = [vp, i32, C.POINTER(_Alignments)]
    L.kslam_comm_get_stats.argtypes = [vp, C.POINTER(CommStats)]
    L.kslam_comm_abort_batch.argtypes = [vp]
    L.kslam_set_sw_band.argtypes = [vp, i32]
    u32 = C.c_uint32
    L.kslam_fastq_open.argtypes = [C.c_char_p, C.c_char_p, u32, C.POINTER(vp)]
    L.kslam_fastq_next.argtypes = [vp, u64, C.POINTER(_ReadBatch)]
    L.kslam_fastq_set_ring.argtypes = [vp, u32]
    L.kslam_fastq_error.argtypes = [vp]
    L.kslam_fastq_error.restype = C.c_char_p
    L.kslam_fastq_close.argtypes = [vp]
    L.kslam_fastq_close.restype = None
    L.kslam_sam_header.argtypes = [C.POINTER(_SamDb), C.c_char_p, C.POINTER(vp), C.POINTER(u64)]
    L.kslam_sam_batch.argtypes = [C.POINTER(SamParams), C.POINTER(_SamDb), C.POINTER(_ReadBatch), C.POINTER(_Pairs), C.POINTER(vp),
                                  C.POINTER(u64), C.POINTER(u32)]
    L.kslam_sam_batch_single.argtypes = [C.POINTER(SamParams), C.POINTER(_SamDb), C.POINTER(_ReadBatch), C.POINTER(_Alignments), u32,
                                         C.POINTER(vp), C.POINTER(u64)]
    L.kslam_sam_free.argtypes = [vp]
    L.kslam_sam_free.restype = None
    L.kslam_taxdb_open.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.kslam_taxdb_build.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p]
    L.kslam_taxdb_size.argtypes = [vp]
    L.kslam_taxdb_size.restype = u64
    L.kslam_taxdb_lca.argtypes = [vp, vp, u64]
    L.kslam_taxdb_lca.restype = u32
    L.kslam_taxdb_lineage.argtypes = [vp, u32, C.POINTER(vp), C.POINTER(u64)]
    L.kslam_taxdb_name.argtypes = [vp, u32, C.POINTER(vp), C.POINTER(u64)]
    L.kslam_taxdb_close.argtypes = [vp]
    L.kslam_taxdb_close.restype = None
    L.kslam_taxa_create.argtypes = [C.POINTER(vp)]
    L.kslam_taxa_destroy.argtypes = [vp]
    L.kslam_taxa_destroy.restype = None
    L.kslam_batch_outputs.argtypes = [C.POINTER(SamParams), C.POINTER(_SamDb), C.POINTER(_ReadBatch), C.POINTER(_Pairs), i32, C.POINTER(vp),
                                      C.POINTER(u64), C.POINTER(u32), vp, vp]
    L.kslam_batch_outputs_single.argtypes = [C.POINTER(SamParams), C.POINTER(_SamDb), C.POINTER(_ReadBatch), C.POINTER(_Alignments), u32, i32,
                                             C.POINTER(vp), C.POINTER(u64), vp, vp]
    L.kslam_taxa_results.argtypes = [vp, vp, u32] + [C.POINTER(vp), C.POINTER(u64)] * 3
    L.kslam_index_parse_genbank.argtypes = [C.POINTER(C.c_char_p), u64, C.POINTER(vp)]
    L.kslam_index_parse_fasta.argtypes = [C.POINTER(C.c_char_p), u64, C.POINTER(vp)]
    L.kslam_index_read.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.kslam_index_write.argtypes = [vp, C.c_char_p]
    L.kslam_index_db.argtypes = [vp, C.POINTER(_SamDb)]
    L.kslam_gene_index_build.argtypes = [C.POINTER(_SamDb), C.POINTER(vp)]
    L.kslam_gene_index_free.argtypes = [vp]
    L.kslam_gene_index_free.restype = None
    L.kslam_index_error.restype = C.c_char_p
    L.kslam_index_free.argtypes = [vp]
    L.kslam_index_free.restype = None
    L.kslam_set_kmer_sort_bits.argtypes = [vp, u32]
    L.kslam_get_kmer_sort_bits.argtypes = [vp]
    L.kslam_load_genomes_part.argtypes = [vp, u64, vp, vp, u32, u32]
    L.kslam_get_partition.argtypes = [vp, C.POINTER(u32), C.POINTER(u32), vp, C.POINTER(u64)]
    L.kslam_part_route_kmers.argtypes = [vp, u32, C.POINTER(vp), vp]
    L.kslam_part_recv_buffer.argtypes = [vp, u64, C.POINTER(vp)]
    L.kslam_part_join.argtypes = [vp, u64, vp, C.POINTER(vp), vp]
    L.kslam_part_match_buffer.argtypes = [vp, u64, C.POINTER(vp)]
    L.kslam_part_finish.argtypes = [vp, u64, u32, i32, C.POINTER(_Alignments)]
    _lib = L
    return L


def _u8(a):
    if isinstance(a, (bytes, bytearray)):
        a = np.frombuffer(a, dtype=np.uint8)
    return np.ascontiguousarray(a, dtype=np.uint8)


def _u64(a):
    return np.ascontiguousarray(a, dtype=np.uint64)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _view(ptr, n, dtype):
    if not n or not ptr:
        return np.zeros(0, dtype=dtype)
    buf = (C.c_char * (n * dtype.itemsize)).from_address(ptr)
    return np.frombuffer(buf, dtype=dtype, count=n)


@dataclass
class Alignments:
    """alignToDatabase's std::vector<Overlap>, same order; cigar i = cigar_pool[cigar_off:cigar_off+cigar_len]."""
    overlaps: np.ndarray
    cigar_pool: np.ndarray


@dataclass
class Pairs:
    """getPairedOverlaps' std::vector<PairedOverlap> plus the pair-sorted overlap array r1_idx/r2_idx point into."""
    sorted_overlaps: np.ndarray
    cigar_pool: np.ndarray
    pairs: np.ndarray


class Aligner:
    """One matching context on one GPU (one kslam_ctx)."""

    def __init__(self, match=2, mismatch=3, gap_open=5, gap_extend=2, score_threshold=0, report_cigar=False,
                 device=0, genome_gap=16, max_cigar_ops=32, stream_priority=0):
        self.L = lib()
        self.params = Params(match, mismatch, gap_open, gap_extend, score_threshold, int(bool(report_cigar)), 0,
                             device, genome_gap, max_cigar_ops, stream_priority)
        h = C.c_void_p()
        rc = self.L.kslam_create(C.byref(self.params), C.byref(h))
        if rc != 0:
            raise KslamError(f"kslam_create failed ({rc}): {self.L.kslam_last_error(None).decode()}")
        self.h = h
        self._keep = []
        self.n_parts = 1

    # -- lifecycle
    def close(self):
        if getattr(self, "h", None):
            self.L.kslam_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc < 0:
            raise KslamError(f"{what} failed ({rc}): {self.L.kslam_last_error(self.h).decode()}")
        return rc

    @property
    def exact(self):
        return bool(self.L.kslam_params_exact(C.byref(self.params)))

    @property
    def fast(self):
        """True: packed band / wavefront kernels; False: the literal restatement of SSW's striped kernels (same results)."""
        return bool(self.L.kslam_params_fast(C.byref(self.params)))

    # -- the path
    def load_genomes(self, bases, offs):
        bases, offs = _u8(bases), _u64(offs)
        self._check(self.L.kslam_load_genomes(self.h, len(offs) - 1, _ptr(bases), _ptr(offs)), "kslam_load_genomes")
        self.n_parts = 1

    # -- k-mer-range partitioned database (include/kslam.h "partitioned"; protocol in dist.py)
    def load_genomes_part(self, bases, offs, part, n_parts):
        """bases: host bytes, or a torch uint8 tensor on the ctx's GPU (include/kslam.h: the copy is cudaMemcpyDefault)"""
        offs = _u64(offs)
        if hasattr(bases, "data_ptr"):
            if getattr(bases, "is_cuda", False):
                import torch
                torch.cuda.synchronize(bases.device)       # the library copies on its own stream: the producer must be done
            ptr = C.c_void_p(bases.data_ptr())
        else:
            bases = _u8(bases); ptr = _ptr(bases)
        self._check(self.L.kslam_load_genomes_part(self.h, len(offs) - 1, ptr, _ptr(offs), part, n_parts),
                    "kslam_load_genomes_part")
        self.n_parts = n_parts

    def partition(self):
        part, n_parts, total = C.c_uint32(), C.c_uint32(), C.c_uint64()
        self._check(self.L.kslam_get_partition(self.h, C.byref(part), C.byref(n_parts), None, C.byref(total)), "kslam_get_partition")
        spl = np.zeros(n_parts.value + 1, dtype=np.uint64)
        self._check(self.L.kslam_get_partition(self.h, None, None, _ptr(spl), None), "kslam_get_partition")
        return dict(part=part.value, n_parts=n_parts.value, splitters=spl, n_genome_kmers_total=total.value)

    def part_route_kmers(self, read_id_base):
        """-> (device pointer of the k-mer records grouped by key owner, counts per owner)"""
        ptr = C.c_void_p()
        counts = np.zeros(self.n_parts, dtype=np.uint64)
        self._check(self.L.kslam_part_route_kmers(self.h, read_id_base, C.byref(ptr), _ptr(counts)), "kslam_part_route_kmers")
        return ptr.value or 0, counts

    def part_recv_buffer(self, n_records):
        ptr = C.c_void_p()
        self._check(self.L.kslam_part_recv_buffer(self.h, n_records, C.byref(ptr)), "kslam_part_recv_buffer")
        return ptr.value or 0

    def part_join(self, n_records, id_bases):
        """-> (device pointer of the raw matches grouped by read owner, counts per owner)"""
        ptr = C.c_void_p()
        idb = np.ascontiguousarray(id_bases, dtype=np.uint32)
        assert len(idb) == self.n_parts + 1
        counts = np.zeros(self.n_parts, dtype=np.uint64)
        self._check(self.L.kslam_part_join(self.h, n_records, _ptr(idb), C.byref(ptr), _ptr(counts)), "kslam_part_join")
        return ptr.value or 0, counts

    def part_match_buffer(self, n_matches):
        ptr = C.c_void_p()
        self._check(self.L.kslam_part_match_buffer(self.h, n_matches, C.byref(ptr)), "kslam_part_match_buffer")
        return ptr.value or 0

    def part_finish(self, n_matches, read_id_base, fetch=True, copy=True):
        out = _Alignments()
        self._check(self.L.kslam_part_finish(self.h, n_matches, read_id_base, int(fetch), C.byref(out)), "kslam_part_finish")
        return self._alignments(out, copy) if fetch else int(out.n_overlaps)

    def align_batch(self, bases, offs, copy=True) -> Alignments:
        bases, offs = _u8(bases), _u64(offs)
        out = _Alignments()
        self._check(self.L.kslam_align_batch(self.h, len(offs) - 1, _ptr(bases), _ptr(offs), C.byref(out)),
                    "kslam_align_batch")
        return self._alignments(out, copy)

    def upload_reads(self, bases, offs):
        bases, offs = _u8(bases), _u64(offs)
        self._check(self.L.kslam_upload_reads(self.h, len(offs) - 1, _ptr(bases), _ptr(offs)), "kslam_upload_reads")

    def align_resident(self, fetch=False, copy=True):
        out = _Alignments()
        self._check(self.L.kslam_align_resident(self.h, int(fetch), C.byref(out)), "kslam_align_resident")
        return self._alignments(out, copy) if fetch else int(out.n_overlaps)

    def _alignments(self, out, copy):
        ov = _view(out.overlaps, out.n_overlaps, OVERLAP_DT)
        cg = _view(out.cigar_pool, out.n_cigar_words, np.dtype("<u4"))
        return Alignments(ov.copy() if copy else ov, cg.copy() if copy else cg)

    def align_pair_batch(self, bases, offs, copy=True) -> "Pairs":
        """alignToDatabase + screen + getPairedOverlaps (SLAM.h:209-214) in one call; only the pair-stage results
        (what the reference's loop keeps) are copied back."""
        bases, offs = _u8(bases), _u64(offs)
        out = _Pairs()
        self._check(self.L.kslam_align_pair_batch(self.h, len(offs) - 1, _ptr(bases), _ptr(offs), C.byref(out)),
                    "kslam_align_pair_batch")
        return self._pairs(out, copy)

    def pair_batch(self, fetch=True, copy=True):
        out = _Pairs()
        self._check(self.L.kslam_pair_batch(self.h, int(fetch), C.byref(out)), "kslam_pair_batch")
        if not fetch:
            return int(out.n_pairs)
        return self._pairs(out, copy)

    def fetch_pairs_compact(self, copy=True, threads=0):
        """After pair_batch(fetch=False): -> (compact pair records, insert-size limit of the batch, mates of the pairs beyond it)
        (kslam_fetch_pairs_compact: 24 B per pair instead of the pair + alignment records; runs without --sam-file)."""
        out = _PairsCompact()
        self._check(self.L.kslam_fetch_pairs_compact(self.h, threads, C.byref(out)), "kslam_fetch_pairs_compact")
        f = (lambda a: a.copy()) if copy else (lambda a: a)
        return f(_view(out.pairs, out.n_pairs, PAIR_COMPACT_DT)), int(out.insert_size_limit), f(_view(out.far, out.n_far, FAR_MATES_DT))

    def fetch_far_mates(self, limit, copy=True):
        """After pair_batch: the mates of every pair record with insert_size > limit, in pair order (kslam_fetch_far_mates;
        what a caller needs once the insert-size limit of a run is known, e.g. after merging the batches of several GPUs)."""
        n, ptr = C.c_uint64(), C.c_void_p()
        self._check(self.L.kslam_fetch_far_mates(self.h, int(limit), C.byref(n), C.byref(ptr)), "kslam_fetch_far_mates")
        far = _view(ptr.value, n.value, FAR_MATES_DT)
        return far.copy() if copy else far

    def fetch_pairs(self, copy=True) -> "Pairs":
        """D2H of the last pair_batch(fetch=False)."""
        out = _Pairs()
        self._check(self.L.kslam_fetch_pairs(self.h, C.byref(out)), "kslam_fetch_pairs")
        return self._pairs(out, copy)

    def _pairs(self, out, copy):
        so = _view(out.sorted_overlaps, out.n_sorted, OVERLAP_DT)
        cg = _view(out.cigar_pool, out.n_cigar_words, np.dtype("<u4"))
        pr = _view(out.pairs, out.n_pairs, PAIR_DT)
        return Pairs(so.copy() if copy else so, cg.copy() if copy else cg, pr.copy() if copy else pr)

    def ssw_batch(self, q, qoffs, r, roffs):
        """Batched Aligner::Align; returns (overlap records in SSW coordinates, cigar pool)."""
        q, r, qoffs, roffs = _u8(q), _u8(r), _u64(qoffs), _u64(roffs)
        n = len(qoffs) - 1
        out = np.zeros(n, dtype=OVERLAP_DT)
        pool = np.zeros(max(1, n * self.params.max_cigar_ops), dtype=np.uint32)
        self._check(self.L.kslam_ssw_batch(self.h, n, _ptr(q), _ptr(qoffs), _ptr(r), _ptr(roffs), _ptr(out), _ptr(pool)),
                    "kslam_ssw_batch")
        return out, pool

    def ssw_upload(self, q, qoffs, r, roffs):
        q, r, qoffs, roffs = _u8(q), _u8(r), _u64(qoffs), _u64(roffs)
        self._check(self.L.kslam_ssw_upload(self.h, len(qoffs) - 1, _ptr(q), _ptr(qoffs), _ptr(r), _ptr(roffs)),
                    "kslam_ssw_upload")

    def ssw_resident(self):
        self._check(self.L.kslam_ssw_resident(self.h, None, None), "kslam_ssw_resident")

    # -- taps
    def _tap(self, fn, dtype):
        n = self._check(fn(self.h, None, 0), fn.__name__)
        out = np.zeros(n, dtype=dtype)
        if n:
            self._check(fn(self.h, _ptr(out), n), fn.__name__)
        return out

    def genome_kmers(self):
        return self._tap(self.L.kslam_get_genome_kmers, KMER_DT)

    def read_kmers(self):
        return self._tap(self.L.kslam_get_read_kmers, KMER_DT)

    def raw_seeds(self):
        return self._tap(self.L.kslam_get_raw_seeds, SEED_DT)

    def seeds(self):
        return self._tap(self.L.kslam_get_seeds, SEED_DT)

    def sort_records(self, recs, lo_bit=0, hi_bit=64):
        recs = np.ascontiguousarray(recs, dtype=KMER_DT).copy()
        ms = C.c_float()
        self._check(self.L.kslam_sort_records(self.h, _ptr(recs), len(recs), lo_bit, hi_bit, C.byref(ms)), "kslam_sort_records")
        return recs, ms.value

    def timings(self) -> dict:
        t = Timings()
        self._check(self.L.kslam_get_timings(self.h, C.byref(t)), "kslam_get_timings")
        return t.as_dict()

    def measure_int_peak(self) -> float:
        v = C.c_double()
        self._check(self.L.kslam_measure_int_peak(self.h, C.byref(v)), "kslam_measure_int_peak")
        return v.value

    def set_report_cigar(self, on: bool):
        self._check(self.L.kslam_set_report_cigar(self.h, int(on)), "kslam_set_report_cigar")
        self.params.report_cigar = int(on)

    def set_prefilter(self, on: bool):
        self._check(self.L.kslam_set_prefilter(self.h, int(on)), "kslam_set_prefilter")

    def set_sw_band(self, level: int):
        """0 = full-matrix kernel only, 1 = 32-diagonal sweep tier, 2 = + 64-diagonal tier, 3 (default) = + direct tiers."""
        self._check(self.L.kslam_set_sw_band(self.h, int(level)), "kslam_set_sw_band")

    def set_kmer_sort_bits(self, bits: int):
        """Leading k-mer bits the read records are sorted on before the join (0 = auto, 64 = total order)."""
        self._check(self.L.kslam_set_kmer_sort_bits(self.h, int(bits)), "kslam_set_kmer_sort_bits")

    def kmer_sort_bits(self) -> int:
        return self._check(self.L.kslam_get_kmer_sort_bits(self.h), "kslam_get_kmer_sort_bits")

    def set_debug_taps(self, keep: bool):
        self._check(self.L.kslam_set_debug_taps(self.h, int(keep)), "kslam_set_debug_taps")


class Comm:
    """kslam_comm: one rank of the k-mer-range partitioned path with the exchanges issued by the library over NCCL
    (csrc/comm.cu). The Aligner must hold this rank's key range: load_genomes_part(bases, offs, rank, n_ranks)."""

    def __init__(self, aligner, handle):
        self.al, self.h, self.L = aligner, handle, aligner.L

    @staticmethod
    def unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        if lib().kslam_comm_unique_id(buf) != 0:
            raise KslamError("kslam_comm_unique_id failed: " + lib().kslam_last_error(None).decode())
        return buf.raw

    @classmethod
    def init_rank(cls, aligner, rank, n_ranks, uid: bytes):
        h = C.c_void_p()
        aligner._check(aligner.L.kslam_comm_init_rank(aligner.h, rank, n_ranks, C.create_string_buffer(uid, 128), C.byref(h)), "kslam_comm_init_rank")
        return cls(aligner, h)

    @classmethod
    def init_all(cls, aligners):
        """One process, one Aligner per DISTINCT device; drive every returned Comm from its own host thread."""
        n = len(aligners)
        ctxs = (C.c_void_p * n)(*[a.h for a in aligners])
        out = (C.c_void_p * n)()
        aligners[0]._check(aligners[0].L.kslam_comm_init_all(n, ctxs, out), "kslam_comm_init_all")
        return [cls(a, C.c_void_p(out[i])) for i, a in enumerate(aligners)]

    def align_resident(self, fetch=True, copy=True):
        """Collective: alignToDatabase over the partitioned index for the reads this rank uploaded (Aligner.upload_reads)."""
        out = _Alignments()
        self.al._check(self.L.kslam_comm_align_resident(self.h, int(fetch), C.byref(out)), "kslam_comm_align_resident")
        return self.al._alignments(out, copy) if fetch else int(out.n_overlaps)

    def abort_batch(self):
        """Collective stand-in for align_resident on a rank that cannot take part: the other ranks' calls fail instead of waiting."""
        self.al._check(self.L.kslam_comm_abort_batch(self.h), "kslam_comm_abort_batch")

    def stats(self) -> dict:
        st = CommStats()
        self.L.kslam_comm_get_stats(self.h, C.byref(st))
        return st.as_dict()

    def close(self):
        if self.h:
            self.L.kslam_comm_destroy(self.h)
            self.h = None


@dataclass
class ReadBatch:
    """One batch of the FASTQ reader: R1 block then R2 block, the layout Aligner.align_batch takes."""
    n_r1: int
    bases: np.ndarray
    offs: np.ndarray
    quals: np.ndarray
    qual_offs: np.ndarray
    ids: np.ndarray
    id_offs: np.ndarray

    def __len__(self):
        return len(self.offs) - 1

    def records(self):
        b, q, i = self.bases.tobytes(), self.quals.tobytes(), self.ids.tobytes()
        return [(i[int(self.id_offs[k]):int(self.id_offs[k + 1])], b[int(self.offs[k]):int(self.offs[k + 1])],
                 q[int(self.qual_offs[k]):int(self.qual_offs[k + 1])]) for k in range(len(self))]


class FastqReader:
    """kslam_fastq_*: chunk-parallel FASTQ ingest with the reference reader's exact semantics (FASTQsequence.h:110-165)."""

    def __init__(self, r1, r2=None, threads=0, ring=1):
        self.L = lib()
        h = C.c_void_p()
        rc = self.L.kslam_fastq_open(os.fsencode(r1), os.fsencode(r2) if r2 else None, threads, C.byref(h))
        if rc != 0:
            raise KslamError(f"kslam_fastq_open failed ({rc}): {self.L.kslam_last_error(None).decode()}")
        self.h = h
        if ring != 1 and self.L.kslam_fastq_set_ring(self.h, ring) != 0:
            raise KslamError("kslam_fastq_set_ring failed")

    def next(self, max_reads, copy=True):
        """Next batch (None at end of input). Raises KslamError on the reference's R1/R2 size mismatch."""
        out = _ReadBatch()
        rc = self.L.kslam_fastq_next(self.h, max_reads, C.byref(out))
        if rc != 0:
            raise KslamError(f"kslam_fastq_next failed ({rc}): {self.L.kslam_fastq_error(self.h).decode()}")
        n = out.n_reads
        if n == 0:
            return None
        offs = _view(out.offs, n + 1, np.dtype("<u8")); qo = _view(out.qual_offs, n + 1, np.dtype("<u8"))
        io = _view(out.id_offs, n + 1, np.dtype("<u8"))
        f = (lambda a: a.copy()) if copy else (lambda a: a)
        return ReadBatch(int(out.n_r1), f(_view(out.bases, int(offs[-1]), np.dtype("u1"))), f(offs),
                         f(_view(out.quals, int(qo[-1]), np.dtype("u1"))), f(qo), f(_view(out.ids, int(io[-1]), np.dtype("u1"))), f(io))

    def close(self):
        if getattr(self, "h", None):
            self.L.kslam_fastq_close(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def _cat(strings):
    offs = np.zeros(len(strings) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(x) for x in strings])
    buf = np.frombuffer(b"".join(strings), dtype=np.uint8).copy() if offs[-1] else np.zeros(1, np.uint8)
    return buf, offs


class SamWriter:
    """kslam_sam_header / kslam_sam_batch: the reference's host stages after pairing up to the SAM text
    (PairedOverlap.h:314-576, SAM.h). Host code: works without a GPU on any (sorted_overlaps, cigar_pool, pairs)."""

    def __init__(self, gen_bases=None, gen_offs=None, locus_tags=None, taxonomy_ids=None, num_alignments=10, score_fraction_threshold=0.95,
                 pseudo_assembly=True, report_cigar=True, sam_xa=False, threads=0, genes=None, index=None, gene_index=True):
        """The database either as arrays (genes = (GENE_DT records, gene_offs u64[n+1], gene string bytes) or None) or as an
        Index (kslam_index_*), whose buffers are used in place."""
        self.L = lib()
        if index is not None:
            self.index = index                              # keeps the buffers alive
            self.db = index.db
        else:
            self.gb, self.go = _u8(gen_bases), _u64(gen_offs)
            self.lt, self.lo = _cat([t if isinstance(t, bytes) else t.encode() for t in locus_tags])
            self.tax = None if taxonomy_ids is None else np.ascontiguousarray(taxonomy_ids, dtype=np.uint32)
            self.db = _SamDb(len(self.go) - 1, self.gb.ctypes.data, self.go.ctypes.data, self.lt.ctypes.data, self.lo.ctypes.data,
                             None if self.tax is None else self.tax.ctypes.data)
            if genes is not None:
                self.genes = np.ascontiguousarray(genes[0], dtype=GENE_DT); self.gene_offs = _u64(genes[1])
                self.gene_strings = _u8(genes[2]) if len(genes[2]) else np.zeros(1, np.uint8)
                self.db.genes, self.db.gene_offs, self.db.gene_strings = self.genes.ctypes.data, self.gene_offs.ctypes.data, self.gene_strings.ctypes.data
                if gene_index:                              # binary-search lookup of the best gene (same answers as the full scan)
                    gi = C.c_void_p()
                    if self.L.kslam_gene_index_build(C.byref(self.db), C.byref(gi)) != 0:
                        raise KslamError("kslam_gene_index_build failed")
                    self.db.gene_index = self._gene_index = gi
        self.prm = SamParams(num_alignments, int(pseudo_assembly), int(report_cigar), int(sam_xa), threads, score_fraction_threshold)

    def __del__(self):
        gi = getattr(self, "_gene_index", None)
        if gi:
            self.L.kslam_gene_index_free(gi)
            self._gene_index = None

    def _take(self, ptr, n):
        try:
            return C.string_at(ptr, n.value)
        finally:
            self.L.kslam_sam_free(ptr)

    def header(self, command_line=""):
        ptr, n = C.c_void_p(), C.c_uint64()
        rc = self.L.kslam_sam_header(C.byref(self.db), command_line.encode(), C.byref(ptr), C.byref(n))
        if rc != 0:
            raise KslamError(f"kslam_sam_header failed ({rc})")
        return self._take(ptr, n)

    def batch_single(self, read_bases, read_offs, quals, qual_offs, ids, id_offs, overlaps, cigar_pool, score_threshold=0,
                     want_sam=True, taxdb=None, taxa=None):
        """Single-end reads: SAM text (and taxon assignments) from align_batch's output (kslam_batch_outputs_single)."""
        rb, ro, q, qo, i, io = _u8(read_bases), _u64(read_offs), _u8(quals), _u64(qual_offs), _u8(ids), _u64(id_offs)
        n = len(ro) - 1
        reads = _ReadBatch(n, n, rb.ctypes.data, ro.ctypes.data, q.ctypes.data, qo.ctypes.data, i.ctypes.data, io.ctypes.data)
        ov = np.ascontiguousarray(overlaps, dtype=OVERLAP_DT); cg = np.ascontiguousarray(cigar_pool, dtype=np.uint32)
        a = _Alignments()
        a.n_overlaps = len(ov); a.overlaps = ov.ctypes.data if len(ov) else None
        a.n_cigar_words = len(cg); a.cigar_pool = cg.ctypes.data if len(cg) else None
        ptr, ln = C.c_void_p(), C.c_uint64()
        rc = self.L.kslam_batch_outputs_single(C.byref(self.prm), C.byref(self.db), C.byref(reads), C.byref(a), score_threshold, int(want_sam),
                                               C.byref(ptr), C.byref(ln), taxdb.h if taxdb is not None else None, taxa.h if taxa is not None else None)
        if rc != 0:
            raise KslamError(f"kslam_batch_outputs_single failed ({rc})")
        if not want_sam:
            return b""
        return self._take(ptr, ln)

    def batch_compact(self, read_offs, ids, id_offs, compact, limit, far, taxdb=None, taxa=None):
        """kslam_batch_outputs_compact: the host stages of a run without --sam-file on compact pair records. -> insert-size limit"""
        ro, i, io = _u64(read_offs), _u8(ids), _u64(id_offs)
        n = len(ro) - 1
        reads = _ReadBatch(n, n // 2, None, ro.ctypes.data, None, None, i.ctypes.data, io.ctypes.data)
        cp = np.ascontiguousarray(compact, dtype=PAIR_COMPACT_DT); fm = np.ascontiguousarray(far, dtype=FAR_MATES_DT)
        p = _PairsCompact(len(cp), cp.ctypes.data if len(cp) else None, int(limit), len(fm), fm.ctypes.data if len(fm) else None)
        mi = C.c_uint32()
        rc = self.L.kslam_batch_outputs_compact(C.byref(self.prm), C.byref(self.db), C.byref(reads), C.byref(p), C.byref(mi),
                                                taxdb.h if taxdb is not None else None, taxa.h if taxa is not None else None)
        if rc != 0:
            raise KslamError(f"kslam_batch_outputs_compact failed ({rc})")
        return mi.value

    def batch(self, read_bases, read_offs, quals, qual_offs, ids, id_offs, sorted_overlaps, cigar_pool, pairs, out_file=None,
              want_sam=True, taxdb=None, taxa=None):
        """-> (SAM text of the batch, max allowed insert size); with out_file the text is written to it straight from the
        library's buffer and its length is returned instead. With taxdb + taxa (TaxDb, Taxa) the batch's per-read taxon
        assignments are appended to taxa (kslam_batch_outputs); want_sam=False skips the SAM records like a run without
        --sam-file."""
        rb, ro, q, qo, i, io = _u8(read_bases), _u64(read_offs), _u8(quals), _u64(qual_offs), _u8(ids), _u64(id_offs)
        n = len(ro) - 1
        reads = _ReadBatch(n, n // 2, rb.ctypes.data, ro.ctypes.data, q.ctypes.data, qo.ctypes.data, i.ctypes.data, io.ctypes.data)
        so = np.ascontiguousarray(sorted_overlaps, dtype=OVERLAP_DT); pr = np.ascontiguousarray(pairs, dtype=PAIR_DT)
        cg = np.ascontiguousarray(cigar_pool, dtype=np.uint32)
        p = _Pairs()
        p.n_sorted = len(so); p.sorted_overlaps = so.ctypes.data if len(so) else None
        p.n_cigar_words = len(cg); p.cigar_pool = cg.ctypes.data if len(cg) else None
        p.n_pairs = len(pr); p.pairs = pr.ctypes.data if len(pr) else None
        ptr, ln, mi = C.c_void_p(), C.c_uint64(), C.c_uint32()
        rc = self.L.kslam_batch_outputs(C.byref(self.prm), C.byref(self.db), C.byref(reads), C.byref(p), int(want_sam), C.byref(ptr), C.byref(ln),
                                        C.byref(mi), taxdb.h if taxdb is not None else None, taxa.h if taxa is not None else None)
        if rc != 0:
            raise KslamError(f"kslam_batch_outputs failed ({rc})")
        if not want_sam:
            return (0 if out_file is not None else b""), mi.value
        if out_file is not None:
            try:
                if ln.value:
                    out_file.write(memoryview((C.c_char * ln.value).from_address(ptr.value)))
            finally:
                self.L.kslam_sam_free(ptr)
            return ln.value, mi.value
        return self._take(ptr, ln), mi.value


def compact_pairs_host(sorted_overlaps, pairs, midpoint):
    """What kslam_fetch_pairs_compact ships, built on the host from full records (tests; a caller that already has them)."""
    pr = np.ascontiguousarray(pairs, dtype=PAIR_DT); ov = np.ascontiguousarray(sorted_overlaps, dtype=OVERLAP_DT)
    out = np.zeros(len(pr), dtype=PAIR_COMPACT_DT)
    has1, has2 = pr["r1_idx"] >= 0, pr["r2_idx"] >= 0
    rd = np.where(has1, ov["read"][np.maximum(pr["r1_idx"], 0)], ov["read"][np.maximum(pr["r2_idx"], 0)] - np.uint32(midpoint)) if len(pr) else np.zeros(0, np.uint32)
    out["pair_id"] = rd
    for f in ("entry", "ref_start", "ref_end", "insert_size"):
        out[f] = pr[f]
    out["score_flags"] = (pr["combined_score"] & np.uint32(0x3FFFFFFF)) | (has1.astype(np.uint32) << np.uint32(30)) | (has2.astype(np.uint32) << np.uint32(31))
    limit = int(lib().kslam_insert_size_limit_compact(out.ctypes.data, len(out), 0)) if len(out) else 0xFFFFFFFF
    sel = np.flatnonzero(pr["insert_size"] > np.uint32(limit))
    far = np.zeros(len(sel), dtype=FAR_MATES_DT)
    far["pair_index"] = sel
    a, b = ov[pr["r1_idx"][sel]], ov[pr["r2_idx"][sel]]
    far["score1"], far["ref_begin1"], far["ref_end1"] = a["sw_score"], a["ref_begin"], a["ref_end"]
    far["score2"], far["ref_begin2"], far["ref_end2"] = b["sw_score"], b["ref_begin"], b["ref_end"]
    return out, limit, far


def _take_text(L, ptr, n):
    try:
        return C.string_at(ptr, n.value) if ptr.value else b""
    finally:
        L.kslam_sam_free(ptr)


class TaxDb:
    """kslam_taxdb_*: the reference's TaxonomyDB (TaxonomyDatabase.h) — DIR/taxDB, LCA, lineage."""

    def __init__(self, path):
        self.L = lib()
        h = C.c_void_p()
        rc = self.L.kslam_taxdb_open(os.fsencode(path), C.byref(h))
        if rc != 0:
            raise KslamError(f"kslam_taxdb_open({path}) failed ({rc})")
        self.h = h

    @staticmethod
    def build(names_dmp, nodes_dmp, out_path):
        """--parse-taxonomy: names.dmp + nodes.dmp -> the taxDB file."""
        rc = lib().kslam_taxdb_build(os.fsencode(names_dmp), os.fsencode(nodes_dmp), os.fsencode(out_path))
        if rc != 0:
            raise KslamError(f"kslam_taxdb_build failed ({rc})")

    def __len__(self):
        return int(self.L.kslam_taxdb_size(self.h))

    def lca(self, tax_ids):
        a = np.ascontiguousarray(tax_ids, dtype=np.uint32)
        return int(self.L.kslam_taxdb_lca(self.h, a.ctypes.data if len(a) else None, len(a)))

    def _text(self, fn, tax_id):
        ptr, n = C.c_void_p(), C.c_uint64()
        if fn(self.h, tax_id, C.byref(ptr), C.byref(n)) != 0:
            raise KslamError("taxonomy query failed")
        return _take_text(self.L, ptr, n)

    def lineage(self, tax_id):
        return self._text(self.L.kslam_taxdb_lineage, tax_id)

    def name(self, tax_id):
        return self._text(self.L.kslam_taxdb_name, tax_id)

    def close(self):
        if getattr(self, "h", None):
            self.L.kslam_taxdb_close(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:   # noqa: BLE001
            pass


class Taxa:
    """kslam_taxa_*: the run's per-read taxon assignments (std::vector<IdentifiedTaxonomy>), filled by SamWriter.batch."""

    def __init__(self):
        self.L = lib()
        h = C.c_void_p()
        if self.L.kslam_taxa_create(C.byref(h)) != 0:
            raise KslamError("kslam_taxa_create failed")
        self.h = h

    def results(self, taxdb, num_reads):
        """-> (text of <out>_PerRead, XML text of <out>, text of <out>_abbreviated), SLAM.h:256-265."""
        p = [C.c_void_p() for _ in range(3)]; n = [C.c_uint64() for _ in range(3)]
        rc = self.L.kslam_taxa_results(self.h, taxdb.h, num_reads, C.byref(p[0]), C.byref(n[0]), C.byref(p[1]), C.byref(n[1]), C.byref(p[2]), C.byref(n[2]))
        if rc != 0:
            raise KslamError(f"kslam_taxa_results failed ({rc})")
        return tuple(_take_text(self.L, p[i], n[i]) for i in range(3))

    def close(self):
        if getattr(self, "h", None):
            self.L.kslam_taxa_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:   # noqa: BLE001
            pass


class Index:
    """kslam_index_*: GenbankIndex built from GenBank flat files / FASTA files or read from DIR/database, held flat."""

    def __init__(self, h):
        self.L = lib()
        self.h = h
        self.db = _SamDb()
        if self.L.kslam_index_db(self.h, C.byref(self.db)) != 0:
            raise KslamError("kslam_index_db failed")
        n = self.n_entries = int(self.db.n_entries)
        self.offs = _view(self.db.offs, n + 1, np.dtype("<u8"))
        self.bases = _view(self.db.bases, int(self.offs[-1]), np.dtype("u1"))
        lo = _view(self.db.locus_offs, n + 1, np.dtype("<u8"))
        lt = _view(self.db.locus_tags, int(lo[-1]), np.dtype("u1")).tobytes()
        self.locus_tags = [lt[int(lo[i]):int(lo[i + 1])] for i in range(n)]
        self.taxonomy_ids = _view(self.db.taxonomy_ids, n, np.dtype("<u4"))
        if self.db.genes:
            self.gene_offs = _view(self.db.gene_offs, n + 1, np.dtype("<u8"))
            self.genes = _view(self.db.genes, int(self.gene_offs[-1]), GENE_DT)
            self.gene_strings = _view(self.db.gene_strings, int(self.genes["str_offs"][-1][5]) if len(self.genes) else 0, np.dtype("u1"))
        else:
            self.gene_offs, self.genes, self.gene_strings = np.zeros(n + 1, np.uint64), np.zeros(0, GENE_DT), np.zeros(0, np.uint8)

    @classmethod
    def _make(cls, fn, *args):
        L = lib()
        h = C.c_void_p()
        rc = fn(*args, C.byref(h))
        if rc != 0:
            raise KslamError(f"building the index failed ({rc}): {L.kslam_index_error().decode()}")
        return cls(h)

    @classmethod
    def parse_genbank(cls, paths):
        arr = (C.c_char_p * len(paths))(*[os.fsencode(p) for p in paths])
        return cls._make(lib().kslam_index_parse_genbank, arr, len(paths))

    @classmethod
    def parse_fasta(cls, paths):
        arr = (C.c_char_p * len(paths))(*[os.fsencode(p) for p in paths])
        return cls._make(lib().kslam_index_parse_fasta, arr, len(paths))

    @classmethod
    def read(cls, database_path):
        return cls._make(lib().kslam_index_read, os.fsencode(database_path))

    def write(self, database_path):
        rc = self.L.kslam_index_write(self.h, os.fsencode(database_path))
        if rc != 0:
            raise KslamError(f"kslam_index_write failed ({rc}): {self.L.kslam_index_error().decode()}")

    def gene_records(self, entry):
        """[(dict of the five strings + gene_id, start, stop)] of one entry."""
        gs = self.gene_strings.tobytes()
        out = []
        for g in self.genes[int(self.gene_offs[entry]):int(self.gene_offs[entry + 1])]:
            so = g["str_offs"]
            d = {k: gs[int(so[i]):int(so[i + 1])] for i, k in enumerate(GENE_STRINGS)}
            d.update(gene_id=int(g["gene_id"]), start=int(g["cds_start"]), stop=int(g["cds_stop"]), complement=int(g["complement"]))
            out.append(d)
        return out

    def close(self):
        if getattr(self, "h", None):
            self.L.kslam_index_free(self.h)
            self.h = None
