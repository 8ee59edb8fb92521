"""nimble_aligner_b200 — B200-native replacement for nimble-aligner's read-alignment hot path.

Python is only the test / bench harness here: everything below is a thin ctypes binding of the C ABI declared in
``include/nimble_b200.h`` (built by ``nimble_aligner_b200/build.py`` into ``libnimble_b200.so``).  Names mirror the
reference's library entry points (paths under /root/reference):

  get_reference_library        src/reference_library.rs:20
  get_reference_sequence_data  src/utils.rs:7
  build_index                  debruijn_mapping::build_index::build_index::<Kmer30>  (src/bin/main.rs:121-128)
  get_calls / call             src/align.rs:392 / src/score.rs:14
  process_fastq                src/process/fastq.rs:7
  process_samples              many FASTQ or bulk BAM samples in one run (nb_process_samples)

There is no CPU fallback: if the shared library is missing or no sm_100 device is present, calls raise NbError.
"""
import ctypes as C
import os
import re

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("NIMBLE_B200_SO") or os.path.join(_HERE, "libnimble_b200.so")   # the override selects a tuning build (scripts/build_variant.sh)

CHEM = {"unstranded": 0, "fiveprime": 1, "threeprime": 2, "none": 3}
REASONS = ["ScoreBelowThreshold", "DiscardedMultipleMatch", "DiscardedNonzeroMismatch", "NoMatch", "NoMatchAndScoreBelowThreshold",
           "DifferentFilterReasons", "NotMatchingPair", "ForceIntersectFailure", "ShortRead", "MaxHitsExceeded", "HighEntropy",
           "SuccessfulMatch", "StrandWasWrong", "TriageEmptyEquivalenceClass", "AboveMismatchThreshold",
           "SkippedAlignDueToUnpairedDummy", "None"]
R = {n: i for i, n in enumerate(REASONS)}
NB_MEM_HOST, NB_MEM_DEVICE = 0, 1
NB_SEQ_ASCII, NB_SEQ_2BIT, NB_SEQ_BAM4 = 0, 1, 2
FLAG_SKIP_ALIGN, FLAG_REVCOMP = 1, 2


class NbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("nimble_b200 error %d: %s" % (code, msg))
        self.code = code


class Config(C.Structure):  # nb_config == AlignFilterConfig (src/align.rs:80-95)
    _fields_ = [("reference_genome_size", C.c_uint64), ("score_percent", C.c_double), ("score_threshold", C.c_uint64),
                ("num_mismatches", C.c_uint64), ("discard_nonzero_mismatch", C.c_int32), ("discard_multiple_matches", C.c_int32),
                ("score_filter", C.c_int32), ("intersect_level", C.c_int32), ("require_valid_pair", C.c_int32),
                ("strand_filter", C.c_int32), ("discard_multi_hits", C.c_uint64), ("max_hits_to_report", C.c_uint64),
                ("trim_strictness", C.c_double), ("trim_target_length", C.c_uint64)]

    def copy(self, **kw):
        c = Config.from_buffer_copy(bytes(self))
        for k, v in kw.items():
            if k == "strand_filter" and isinstance(v, str):
                v = CHEM[v]
            setattr(c, k, v)
        return c


class Batch(C.Structure):
    _fields_ = [("n_pairs", C.c_uint64), ("location", C.c_int32), ("max_read_len", C.c_uint32),
                ("r1", C.c_void_p), ("r1_off", C.c_void_p), ("r2", C.c_void_p), ("r2_off", C.c_void_p),
                ("q1", C.c_void_p), ("q2", C.c_void_p), ("flags1", C.c_void_p), ("flags2", C.c_void_p),
                ("scope_id", C.c_void_p), ("cell_id", C.c_void_p),
                ("encoding", C.c_int32), ("reserved", C.c_int32), ("r1_len", C.c_void_p), ("r2_len", C.c_void_p)]


class Counts(C.Structure):
    _fields_ = [("n_rows", C.c_uint64), ("row_scope", C.POINTER(C.c_uint32)), ("row_callset", C.POINTER(C.c_uint32)),
                ("row_count", C.POINTER(C.c_int64)), ("n_callsets", C.c_uint64), ("callset_off", C.POINTER(C.c_uint64)),
                ("callset_items", C.POINTER(C.c_uint32)), ("n_pairs_seen", C.c_uint64), ("n_unique_keys", C.c_uint64),
                ("n_slots", C.c_uint64), ("slot_to_callset", C.POINTER(C.c_uint32))]


class CellCounts(C.Structure):  # nb_cell_counts
    _fields_ = [("n_rows", C.c_uint64), ("row_cell", C.POINTER(C.c_uint32)), ("row_callset", C.POINTER(C.c_uint32)),
                ("row_umis", C.POINTER(C.c_int64)), ("row_reads", C.POINTER(C.c_int64)), ("n_callsets", C.c_uint64),
                ("callset_off", C.POINTER(C.c_uint64)), ("callset_items", C.POINTER(C.c_uint32)), ("n_scopes", C.c_uint64)]


READ_DT = np.dtype([("reason", "u1"), ("pass", "u1"), ("score", "<u2"), ("mismatches", "<u2"), ("trimmed_len", "<u2"),
                    ("ec_len", "<u4"), ("ec_hash", "<u4")])
PAIR_DT = np.dtype([("callset", "<u4"), ("triage", "u1"), ("fr1", "u1"), ("fr2", "u1"), ("insertable", "u1"),
                    ("key_lo", "<u8"), ("key_hi", "<u8")])

_lib = None

_SIGS = {
    "nb_last_error": (C.c_char_p, []), "nb_reason_str": (C.c_char_p, [C.c_int]), "nb_version": (C.c_char_p, []),
    "nb_library_load_json": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(C.c_void_p)]),
    "nb_library_parse_json": (C.c_int, [C.c_char_p, C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]),
    "nb_library_from_columns": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "nb_library_free": (None, [C.c_void_p]),
    "nb_library_get_config": (C.c_int, [C.c_void_p, C.POINTER(Config)]), "nb_library_set_config": (C.c_int, [C.c_void_p, C.POINTER(Config)]),
    "nb_library_n_rows": (C.c_uint32, [C.c_void_p]), "nb_library_n_headers": (C.c_uint32, [C.c_void_p]),
    "nb_library_header": (C.c_char_p, [C.c_void_p, C.c_uint32]), "nb_library_value": (C.c_char_p, [C.c_void_p, C.c_uint32, C.c_uint32]),
    "nb_library_group_on": (C.c_uint32, [C.c_void_p]), "nb_library_sequence_name_idx": (C.c_uint32, [C.c_void_p]),
    "nb_library_sequence_idx": (C.c_uint32, [C.c_void_p]),
    "nb_library_push_column": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_uint32, C.c_int]),
    "nb_library_n_groups": (C.c_uint32, [C.c_void_p]), "nb_library_group_name": (C.c_char_p, [C.c_void_p, C.c_uint32]),
    "nb_index_build": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "nb_index_build_from_sequences": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.POINTER(C.c_void_p)]),
    "nb_index_build_gpu": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "nb_index_build_gpu_from_sequences": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "nb_index_compare": (C.c_int, [C.c_void_p, C.c_void_p]),
    "nb_index_free": (None, [C.c_void_p]),
    "nb_index_save": (C.c_int, [C.c_void_p, C.c_char_p]), "nb_index_load": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]), "nb_index_stats": (C.c_int, [C.c_void_p, C.c_void_p]),
    "nb_index_dump": (C.c_uint64, [C.c_void_p, C.c_char_p, C.c_uint64]),
    "nb_device_count": (C.c_int, []),
    "nb_ctx_create": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "nb_ctx_free": (None, [C.c_void_p]), "nb_ctx_set_config": (C.c_int, [C.c_void_p, C.POINTER(Config)]),
    "nb_ctx_sync": (C.c_int, [C.c_void_p]), "nb_ctx_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_uint64]),
    "nb_host_alloc": (C.c_void_p, [C.c_size_t]), "nb_host_free": (None, [C.c_void_p]),
    "nb_align_batch": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_void_p, C.c_void_p]),
    "nb_last_batch_ecs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "nb_counts_finalize": (C.c_int, [C.c_void_p, C.POINTER(Counts)]),
    "nb_counts_device_rows": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]), "nb_counts_reset": (C.c_int, [C.c_void_p]),
    "nb_keys_export_count": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "nb_keys_export": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]),
    "nb_keys_import": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64]),
    "nb_keys_export_partitioned": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p]),
    "nb_callsets_export": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]),
    "nb_callsets_import": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64]),
    "nb_callsets_import_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64]),
    "nb_route_create": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p]),
    "nb_route_attach_ipc": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint64]),
    "nb_route_sent": (C.c_int, [C.c_void_p, C.c_void_p]),
    "nb_route_attach_ctx": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint64]),
    "nb_route_set_pair_base": (C.c_int, [C.c_void_p, C.c_uint64]),
    "nb_route_import": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]),
    "nb_route_detach": (C.c_int, [C.c_void_p]),
    "nb_ctx_kernel_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "nb_ctx_work_counters": (C.c_int, [C.c_void_p, C.c_void_p]),
    "nb_comm_unique_id": (C.c_int, [C.c_void_p]),
    "nb_comm_init_rank": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32]),
    "nb_comm_attach": (C.c_int, [C.c_void_p, C.c_void_p]),
    "nb_comm_init_all": (C.c_int, [C.c_void_p, C.c_uint32]),
    "nb_comm_free": (C.c_int, [C.c_void_p]),
    "nb_comm_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "nb_route_setup": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64]),
    "nb_merge_whole_run": (C.c_int, [C.c_void_p, C.POINTER(Counts)]),
    "nb_merge_scoped": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(Counts)]),
    "nb_merge_scoped_sharded": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(Counts)]),
    "nb_measure_gather": (C.c_int, [C.c_int, C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(C.c_double)]),
    "nb_measure_h2d": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint32, C.c_void_p, C.POINTER(C.c_double)]),
    "nb_write_fastq_tsv": (C.c_int, [C.c_char_p, C.c_void_p, C.POINTER(Counts)]),
    "nb_bam_dump_groups": (C.c_int, [C.c_char_p, C.c_int, C.c_int, C.c_char_p]),
    "nb_fastq_dump": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, C.c_uint64, C.c_char_p]),
    "nb_gunzip_parallel": (C.c_int, [C.c_char_p, C.c_uint64, C.c_int, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "nb_gzip_fast": (C.c_int, [C.c_char_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "nb_index_cache_key": (C.c_int, [C.c_void_p, C.c_char_p]),
    "nb_index_build_cached": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "nb_inflate": (C.c_int, [C.c_char_p, C.c_uint64, C.c_int, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "nb_process_fastq_devices": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_void_p, C.c_uint32]),
    "nb_process_bam": (C.c_int, [C.c_char_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_int]),
    "nb_process_bam_cells": (C.c_int, [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_int]),
    "nb_process_bam_cells_any_order": (C.c_int, [C.c_char_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_char_p, C.c_int, C.c_int]),
    "nb_bam_dump_scopes_any_order": (C.c_int, [C.c_char_p, C.c_int, C.c_int, C.c_char_p]),
    "nb_process_bam_cells_any_order_budget": (C.c_int, [C.c_char_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_uint64]),
    "nb_bam_dump_scopes_any_order_budget": (C.c_int, [C.c_char_p, C.c_int, C.c_int, C.c_uint64, C.c_char_p]),
    "nb_any_order_umi_bucket": (C.c_int, [C.c_char_p, C.c_uint32, C.POINTER(C.c_uint32)]),
    "nb_process_bam_rows_any_order": (C.c_int, [C.c_char_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_uint64]),
    "nb_process_bam_bulk": (C.c_int, [C.c_char_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_int]),
    "nb_bam_dump_pairs_bulk": (C.c_int, [C.c_char_p, C.c_int, C.c_int, C.c_char_p]),
    "nb_process_samples": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_int]),
    "nb_cells_roll": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64]),
    "nb_cells_finalize": (C.c_int, [C.c_void_p, C.POINTER(CellCounts)]),
    "nb_cells_reset": (C.c_int, [C.c_void_p]),
    "nb_write_cell_matrix": (C.c_int, [C.c_char_p, C.c_void_p, C.POINTER(CellCounts), C.c_void_p, C.c_uint64]),
    "nb_process_fastq": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_int]),
}


def lib():
    """Loads libnimble_b200.so.  Fails loudly when it has not been built: there is no other implementation."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise NbError(-6, "libnimble_b200.so is missing (run `python nimble_aligner_b200/build.py`); there is no CPU fallback")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in _SIGS.items():
            f = getattr(L, name)
            f.restype, f.argtypes = res, args
        _lib = L
    return _lib


def _ck(rc):
    if rc != 0:
        raise NbError(rc, lib().nb_last_error().decode("utf-8", "replace"))


def _strs(strs):
    arr = (C.c_char_p * len(strs))(*[str(s).encode("utf-8") for s in strs])
    return arr


class Library:
    """Reference + AlignFilterConfig (src/reference_library.rs:11-17, src/align.rs:80-95)."""

    def __init__(self, handle):
        self.h = handle

    @classmethod
    def from_json(cls, path, strand_filter="unstranded"):
        h = C.c_void_p()
        _ck(lib().nb_library_load_json(str(path).encode(), CHEM[strand_filter] if isinstance(strand_filter, str) else strand_filter, C.byref(h)))
        return cls(h)

    @classmethod
    def from_text(cls, text, strand_filter="unstranded"):
        h = C.c_void_p()
        b = text.encode() if isinstance(text, str) else text
        _ck(lib().nb_library_parse_json(b, len(b), CHEM[strand_filter], C.byref(h)))
        return cls(h)

    @classmethod
    def from_columns(cls, headers, columns, group_on, sequence_name_idx, sequence_idx, cfg):
        hs = _strs(headers)
        cols = [_strs(c) for c in columns]
        colptr = (C.c_void_p * len(cols))(*[C.cast(c, C.c_void_p) for c in cols])
        h = C.c_void_p()
        _ck(lib().nb_library_from_columns(hs, len(headers), colptr, len(columns[0]), group_on, sequence_name_idx, sequence_idx, C.byref(cfg), C.byref(h)))
        return cls(h)

    def __del__(self):
        if getattr(self, "h", None):
            lib().nb_library_free(self.h)
            self.h = None

    @property
    def config(self):
        c = Config()
        _ck(lib().nb_library_get_config(self.h, C.byref(c)))
        return c

    def set_config(self, cfg):
        _ck(lib().nb_library_set_config(self.h, C.byref(cfg)))

    @property
    def n_rows(self):
        return lib().nb_library_n_rows(self.h)

    @property
    def headers(self):
        return [lib().nb_library_header(self.h, i).decode() for i in range(lib().nb_library_n_headers(self.h))]

    def column(self, c):
        return [lib().nb_library_value(self.h, c, r).decode() for r in range(self.n_rows)]

    @property
    def group_on(self):
        return lib().nb_library_group_on(self.h)

    @property
    def sequence_name_idx(self):
        return lib().nb_library_sequence_name_idx(self.h)

    @property
    def sequence_idx(self):
        return lib().nb_library_sequence_idx(self.h)

    def push_column(self, header, values, set_group_on=True):
        _ck(lib().nb_library_push_column(self.h, header.encode(), _strs(values), len(values), int(set_group_on)))

    def group_names(self):
        return [lib().nb_library_group_name(self.h, g).decode() for g in range(lib().nb_library_n_groups(self.h))]


def get_reference_library(path, strand_filter="unstranded"):
    """reference_library::get_reference_library -> (AlignFilterConfig, Reference)."""
    l = Library.from_json(path, strand_filter)
    return l.config, l


def get_reference_sequence_data(reference):
    """utils::get_reference_sequence_data -> (sequences, names) (src/utils.rs:7-24)."""
    return reference.column(reference.sequence_idx), reference.column(reference.sequence_name_idx)


class Index:
    """PseudoAligner (src/align.rs:21): coloured compacted de Bruijn index in the flat GPU layout."""

    def __init__(self, handle):
        self.h = handle

    @classmethod
    def build(cls, library, threads=1, device=None):
        """device=None: host builder; device=i: the CUDA builder on GPU i (same artefact)."""
        h = C.c_void_p()
        if device is None:
            _ck(lib().nb_index_build(library.h, threads, C.byref(h)))
        else:
            _ck(lib().nb_index_build_gpu(library.h, device, threads, C.byref(h)))
        return cls(h)

    @classmethod
    def from_sequences(cls, seqs, threads=1, device=None):
        data, off = pack_reads(seqs)
        h = C.c_void_p()
        if device is None:
            _ck(lib().nb_index_build_from_sequences(data.ctypes.data, off.ctypes.data, len(seqs), threads, C.byref(h)))
        else:
            _ck(lib().nb_index_build_gpu_from_sequences(data.ctypes.data, off.ctypes.data, len(seqs), device, threads, C.byref(h)))
        return cls(h)

    def compare(self, other):
        """0 when both artefacts describe the same index (nb_index_compare)."""
        return lib().nb_index_compare(self.h, other.h)

    def __del__(self):
        if getattr(self, "h", None):
            lib().nb_index_free(self.h)
            self.h = None

    def save(self, path):
        _ck(lib().nb_index_save(self.h, str(path).encode()))

    @classmethod
    def build_cached(cls, library, cache_dir, device=0, threads=1):
        """<cache_dir>/<key of the library>.nbix when it is there, else the CUDA builder + that file (nb_index_build_cached)."""
        h = C.c_void_p()
        _ck(lib().nb_index_build_cached(library.h, str(cache_dir).encode() if cache_dir is not None else None, device, threads, C.byref(h)))
        return cls(h)

    @staticmethod
    def cache_key(library):
        buf = C.create_string_buffer(33)
        _ck(lib().nb_index_cache_key(library.h, buf))
        return buf.value.decode()

    @classmethod
    def load(cls, path):
        h = C.c_void_p()
        _ck(lib().nb_index_load(str(path).encode(), C.byref(h)))
        return cls(h)

    def stats(self):
        o = np.zeros(8, dtype=np.uint64)
        _ck(lib().nb_index_stats(self.h, o.ctypes.data))
        return dict(zip(["n_kmers", "n_nodes", "n_colours", "colour_elems", "unitig_bases", "table_slots", "device_bytes", "n_sequences"], o.tolist()))

    def dump(self):
        n = lib().nb_index_dump(self.h, None, 0)
        buf = C.create_string_buffer(max(n, 1))
        lib().nb_index_dump(self.h, buf, n)
        return buf.raw[:n].decode()


def build_index(library, threads=1, device=None):
    return Index.build(library, threads, device)


def encode_2bit(ascii_bases, off):
    """ASCII reads (uint8 array + uint64 offsets) -> NB_SEQ_2BIT stream with the same base offsets (host-side packer of the
    harness; a real producer holds packed reads already).  Non-ACGT -> A like DnaString::from_acgt_bytes."""
    n = int(off[-1])
    lut = np.zeros(256, dtype=np.uint8)
    for ch, code in ((b"C", 1), (b"c", 1), (b"G", 2), (b"g", 2), (b"T", 3), (b"t", 3)):
        lut[ch[0]] = code
    codes = lut[np.asarray(ascii_bases[:n])]
    pad = (-n) % 4
    if pad:
        codes = np.concatenate([codes, np.zeros(pad, dtype=np.uint8)])
    q = codes.reshape(-1, 4)
    out = (q[:, 0] | (q[:, 1] << 2) | (q[:, 2] << 4) | (q[:, 3] << 6)).astype(np.uint8)
    return np.concatenate([out, np.zeros(64, dtype=np.uint8)])


def encode_bam4(ascii_bases, off):
    """ASCII reads -> NB_SEQ_BAM4 nibble stream with the same base offsets (high nibble first, "=ACMGRSVTWYHKDBN")."""
    n = int(off[-1])
    lut = np.full(256, 15, dtype=np.uint8)   # anything unknown -> N
    for i, ch in enumerate("=ACMGRSVTWYHKDBN"):
        lut[ord(ch)] = i
        lut[ord(ch.lower())] = i
    codes = lut[np.asarray(ascii_bases[:n])]
    if n % 2:
        codes = np.concatenate([codes, np.zeros(1, dtype=np.uint8)])
    q = codes.reshape(-1, 2)
    out = ((q[:, 0] << 4) | q[:, 1]).astype(np.uint8)
    return np.concatenate([out, np.zeros(64, dtype=np.uint8)])


def pack_reads(reads):
    """list of str/bytes -> (uint8 array, uint64 offsets[n+1])."""
    bs = [r.encode() if isinstance(r, str) else bytes(r) for r in reads]
    off = np.zeros(len(bs) + 1, dtype=np.uint64)
    if bs:
        off[1:] = np.cumsum([len(b) for b in bs], dtype=np.uint64)
    data = np.frombuffer(b"".join(bs), dtype=np.uint8).copy() if bs and off[-1] else np.zeros(1, dtype=np.uint8)
    return data, off


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):  # torch tensor
        return a.data_ptr()
    return int(a)


class Context:
    """One (GPU, stream) execution context: device index copy + aggregation state."""

    def __init__(self, index, library, device=0, stream=None, **options):
        self.index, self.library = index, library
        h = C.c_void_p()
        _ck(lib().nb_ctx_create(index.h, library.h, device, stream, C.byref(h)))
        self.h = h
        for k, v in options.items():
            self.set_option(k, v)

    def __del__(self):
        self.close()

    def close(self):
        if getattr(self, "h", None):
            lib().nb_ctx_free(self.h)
            self.h = None

    def set_config(self, cfg):
        _ck(lib().nb_ctx_set_config(self.h, C.byref(cfg)))

    def set_option(self, name, value):
        _ck(lib().nb_ctx_set_option(self.h, name.encode(), int(value)))

    def sync(self):
        _ck(lib().nb_ctx_sync(self.h))

    def align_batch(self, r1, r1_off, r2=None, r2_off=None, q1=None, q2=None, flags1=None, flags2=None, scope_id=None, cell_id=None,
                    n_pairs=None, max_read_len=0, location=NB_MEM_HOST, reads_out=None, pairs_out=None, want_reads=False, want_pairs=False,
                    encoding=NB_SEQ_ASCII, r1_len=None, r2_len=None):
        """nb_align_batch.  Host arrays are numpy; device arrays may be torch tensors or raw pointers (then pass n_pairs)."""
        keep = [np.ascontiguousarray(a) if isinstance(a, np.ndarray) else a for a in (r1, r1_off, r2, r2_off, q1, q2, flags1, flags2, scope_id, cell_id)]
        lens = [np.ascontiguousarray(a, dtype=np.uint32) if isinstance(a, np.ndarray) else a for a in (r1_len, r2_len)]
        if n_pairs is None:
            n_pairs = len(keep[1]) - 1
        b = Batch(n_pairs, location, max_read_len, *[_ptr(a) for a in keep], encoding, 0, _ptr(lens[0]), _ptr(lens[1]))
        sides = 2 if r2 is not None else 1
        if want_reads and reads_out is None:
            reads_out = np.zeros(n_pairs * sides, dtype=READ_DT)
        if want_pairs and pairs_out is None:
            pairs_out = np.zeros(n_pairs, dtype=PAIR_DT)
        _ck(lib().nb_align_batch(self.h, C.byref(b), _ptr(reads_out), _ptr(pairs_out)))
        if location == NB_MEM_HOST:
            self.sync()   # keeps the numpy temporaries alive until the copies have run
        return reads_out, pairs_out

    def last_batch_ecs(self, n_reads):
        off = np.zeros(n_reads + 1, dtype=np.uint64)
        tot = C.c_uint64(0)
        _ck(lib().nb_last_batch_ecs(self.h, off.ctypes.data, None, 0, C.byref(tot)))
        ids = np.zeros(max(tot.value, 1), dtype=np.uint32)
        _ck(lib().nb_last_batch_ecs(self.h, off.ctypes.data, ids.ctypes.data, len(ids), C.byref(tot)))
        return off, ids[:tot.value]

    def counts(self):
        """nb_counts_finalize -> dict(rows=[(scope, [group names], count)], callsets=[[names]], n_pairs_seen, n_unique_keys)."""
        raw = self.counts_raw()
        return self.decode_counts(raw)

    def counts_raw(self, rows=True, copy=True):
        """nb_counts_finalize -> numpy copies of the C arrays (group indices, no strings).  rows=False leaves the row
        columns out (a multi-GPU host that reduces them on the device, counts_device_rows, has no use for host copies).
        copy=False returns views of the library's buffers instead: valid until the next finalize / reset / close, as the C ABI
        says (a scoped job has millions of rows: copying them in numpy costs more than the library's whole finalize)."""
        c = Counts()
        _ck(lib().nb_counts_finalize(self.h, C.byref(c)))
        return self._raw(c, rows, copy)

    @staticmethod
    def _raw(c, rows=True, copy=True):
        def arr(p, n, dt):
            if not n:
                return np.zeros(0, dt)
            a = np.ctypeslib.as_array(p, (n,))
            return a.copy() if copy else a
        n_items = int(c.callset_off[c.n_callsets]) if c.n_callsets else 0
        nr = c.n_rows if rows else 0
        return dict(row_scope=arr(c.row_scope, nr, np.uint32), row_callset=arr(c.row_callset, nr, np.uint32),
                    row_count=arr(c.row_count, nr, np.int64), callset_off=arr(c.callset_off, c.n_callsets + 1, np.uint64),
                    callset_items=arr(c.callset_items, n_items, np.uint32), n_pairs_seen=c.n_pairs_seen, n_unique_keys=c.n_unique_keys,
                    slot_to_callset=arr(c.slot_to_callset, c.n_slots, np.uint32))

    # ---- multi-GPU merge inside the library (nb_comm_*, nb_merge_*)
    def comm_init_rank(self, unique_id, world, rank):
        uid = np.ascontiguousarray(unique_id, dtype=np.uint8)
        assert uid.size == 128
        _ck(lib().nb_comm_init_rank(self.h, uid.ctypes.data, int(world), int(rank)))
        self._route_world = int(world)

    def comm_free(self):
        _ck(lib().nb_comm_free(self.h))

    def route_setup(self, records_per_peer, pair_index_base):
        """nb_route_create + IPC handle all-gather + attach, over the context's communicator; raises on every rank when any
        rank cannot open its peers."""
        _ck(lib().nb_route_setup(self.h, int(records_per_peer), int(pair_index_base)))

    def merge_whole_run(self):
        """nb_merge_whole_run -> the whole job's counts (same dict as counts_raw), identical on every rank."""
        c = Counts()
        _ck(lib().nb_merge_whole_run(self.h, C.byref(c)))
        return self._raw(c)

    def merge_scoped(self, n_cells, copy=True, sharded=False):
        """nb_merge_scoped -> per-cell rows of the whole job (row_scope = cell id), identical on every rank;
        sharded=True (nb_merge_scoped_sharded): this rank's range of cells only."""
        c = Counts()
        _ck((lib().nb_merge_scoped_sharded if sharded else lib().nb_merge_scoped)(self.h, int(n_cells), C.byref(c)))
        return self._raw(c, True, copy)

    def counts_device_rows(self):
        """(row_scope, row_callset, row_count) of the last finalize as objects with __cuda_array_interface__ (zero copy)."""
        a, b, c, n = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_uint64(0)
        _ck(lib().nb_counts_device_rows(self.h, C.byref(a), C.byref(b), C.byref(c), C.byref(n)))

        class _Dev:
            def __init__(self, ptr, n, typestr):
                self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr or 0, False), "version": 2}
        n = n.value
        return _Dev(a.value, n, "<u4"), _Dev(b.value, n, "<u4"), _Dev(c.value, n, "<i8"), n

    def decode_counts(self, raw):
        if getattr(self, "_group_names", None) is None:
            self._group_names = self.library.group_names()
        names = self._group_names
        off, items = raw["callset_off"].tolist(), raw["callset_items"].tolist()
        callsets = [[names[g] for g in items[off[i]:off[i + 1]]] for i in range(len(off) - 1)]
        rows = [(sc, callsets[cs], n) for sc, cs, n in zip(raw["row_scope"].tolist(), raw["row_callset"].tolist(), raw["row_count"].tolist())]
        out = dict(raw)
        out.update(rows=rows, callsets=callsets)
        return out

    def write_tsv(self, path):
        c = Counts()
        _ck(lib().nb_counts_finalize(self.h, C.byref(c)))
        _ck(lib().nb_write_fastq_tsv(str(path).encode(), self.library.h, C.byref(c)))

    def reset(self):
        _ck(lib().nb_counts_reset(self.h))

    # ---- per-cell table (nb_cells_*): survives reset()
    def cells_roll(self, cell_of_scope):
        """nb_cells_roll: after counts_raw()/counts() of a scoped batch, cell_of_scope[scope_id] = cell id of each of its scopes."""
        a = np.ascontiguousarray(cell_of_scope, dtype=np.uint32)
        _ck(lib().nb_cells_roll(self.h, a.ctypes.data if a.size else None, a.size))

    def cells_finalize(self):
        """nb_cells_finalize -> dict(row_cell, row_callset, row_umis, row_reads, callset_off, callset_items, n_scopes) (numpy copies);
        rows sorted by (cell, callset), callsets numbered in Vec<String> Ord."""
        c = CellCounts()
        _ck(lib().nb_cells_finalize(self.h, C.byref(c)))
        return cell_counts_dict(c)

    def cells_reset(self):
        _ck(lib().nb_cells_reset(self.h))

    # ---- peer routing of the whole-run scope (nb_route_*)
    def route_create(self, world, records_per_peer):
        """Allocates the inbox (one region per source rank); returns its 64-byte CUDA IPC handle (np.uint8[64])."""
        h = np.zeros(64, dtype=np.uint8)
        _ck(lib().nb_route_create(self.h, int(world), int(records_per_peer), h.ctypes.data))
        self._route_world = int(world)
        return h

    def route_attach_ipc(self, world, rank, handles, pair_index_base):
        handles = np.ascontiguousarray(handles, dtype=np.uint8)
        assert handles.size == 64 * world
        _ck(lib().nb_route_attach_ipc(self.h, world, rank, handles.ctypes.data, int(pair_index_base)))

    def route_attach_ctx(self, world, rank, peers, pair_index_base):
        arr = (C.c_void_p * world)(*[p.h for p in peers])
        _ck(lib().nb_route_attach_ctx(self.h, world, rank, arr, int(pair_index_base)))

    def route_set_pair_base(self, pair_index_base):
        _ck(lib().nb_route_set_pair_base(self.h, int(pair_index_base)))

    def route_sent(self):
        """Records stored per destination rank since the last call (waits for the submitted batches)."""
        o = np.zeros(16, dtype=np.uint64)
        _ck(lib().nb_route_sent(self.h, o.ctypes.data))
        return o[: self._route_world].copy()

    def route_import(self, counts):
        counts = np.ascontiguousarray(counts, dtype=np.uint64)
        n = C.c_uint64(0)
        _ck(lib().nb_route_import(self.h, counts.ctypes.data, C.byref(n)))
        return n.value

    def route_detach(self):
        _ck(lib().nb_route_detach(self.h))

    def kernel_stats(self, reset=False):
        o = np.zeros(4, dtype=np.float64)
        _ck(lib().nb_ctx_kernel_stats(self.h, o.ctypes.data, int(reset)))
        return dict(map_launches=int(o[0]), map_ms=float(o[1]), map_reads=int(o[2]), launches=int(o[3]))

    def work_counters(self):
        o = np.zeros(4, dtype=np.uint64)
        _ck(lib().nb_ctx_work_counters(self.h, o.ctypes.data))
        return dict(zip(["probes", "nodes", "bases", "colour_elems"], o.tolist()))


def measure_gather(table_bytes, record_bytes=32, device=0, reps=3):
    """Random-record gather bandwidth (GB/s) over a table of `table_bytes`: the L2 roof when it fits L2, else the HBM gather roof."""
    g = C.c_double(0)
    _ck(lib().nb_measure_gather(device, int(table_bytes), record_bytes, reps, C.byref(g)))
    return g.value


def measure_h2d(devices=(0,), nbytes=256 << 20, reps=8):
    """Pinned host -> device bandwidth with all `devices` copying at once -> (per-device GB/s list, aggregate GB/s)."""
    d = np.asarray(devices, dtype=np.int32)
    per = np.zeros(len(d), dtype=np.float64)
    agg = C.c_double(0)
    _ck(lib().nb_measure_h2d(d.ctypes.data, len(d), int(nbytes), reps, per.ctypes.data, C.byref(agg)))
    return per.tolist(), agg.value


def comm_unique_id():
    """ncclGetUniqueId through the library (128 bytes): rank 0 creates it, the host hands it to every rank."""
    uid = np.zeros(128, dtype=np.uint8)
    _ck(lib().nb_comm_unique_id(uid.ctypes.data))
    return uid


def comm_init_all(contexts):
    """One process driving several GPUs: ncclCommInitAll over the contexts' devices (rank i = contexts[i])."""
    arr = (C.c_void_p * len(contexts))(*[c.h for c in contexts])
    _ck(lib().nb_comm_init_all(arr, len(contexts)))
    for c in contexts:
        c._route_world = len(contexts)


def get_calls(sequences, mate_sequences, sequence_metadata, index, reference, aligner_config, device=0):
    """align::get_calls (src/align.rs:392-467) for one aggregation scope.  `sequences` / `mate_sequences`: lists of
    strings; `sequence_metadata`: None/[] (FASTQ mode) or per-pair dict(q1, q2, skip1, skip2) arrays.
    Returns (sorted [(callset, count)], per-read records, per-pair records)."""
    ctx = Context(index, reference, device)
    try:
        ctx.set_config(aligner_config)
        r1, o1 = pack_reads(sequences)
        r2 = o2 = None
        if mate_sequences is not None:
            r2, o2 = pack_reads(mate_sequences)
        md = sequence_metadata or {}
        reads, pairs = ctx.align_batch(r1, o1, r2, o2, q1=md.get("q1"), q2=md.get("q2"), flags1=md.get("flags1"), flags2=md.get("flags2"),
                                       want_reads=True, want_pairs=True)
        res = ctx.counts()
        return [(cs, n) for _, cs, n in res["rows"]], reads, pairs
    finally:
        ctx.close()


def call(sequences, mate_sequences, per_sequence_metadata, reference_index, reference, aligner_config, device=0):
    """score::call (src/score.rs:14-46): get_calls + sort_score_vector (rows already come back sorted)."""
    return get_calls(sequences, mate_sequences, per_sequence_metadata, reference_index, reference, aligner_config, device)


def process_fastq(input_files, reference_json_paths, output_paths, strand_filter="unstranded", num_cores=1, device=0, devices=None):
    """process::fastq::process behind main.rs's library loop (src/process/fastq.rs:7-30, src/bin/main.rs:95-147).
    devices=[...]: one context per listed GPU (nb_process_fastq_devices)."""
    if devices is not None:
        dv = (C.c_int * len(devices))(*devices)
        _ck(lib().nb_process_fastq_devices(_strs(input_files), len(input_files), _strs(reference_json_paths), _strs(output_paths),
                                           len(reference_json_paths), CHEM[strand_filter], num_cores, dv, len(devices)))
        return
    _ck(lib().nb_process_fastq(_strs(input_files), len(input_files), _strs(reference_json_paths), _strs(output_paths),
                               len(reference_json_paths), CHEM[strand_filter], num_cores, device))


def fastq_dump(input_files, out_path, num_cores=1, chunk_bytes=0):
    """host-only: what the FASTQ feeder would hand to the device (one line per record, mates TAB-separated)."""
    _ck(lib().nb_fastq_dump(_strs(input_files), len(input_files), num_cores, chunk_bytes, str(out_path).encode()))


def process_bam(input_file, reference_json_paths, output_paths, strand_filter="unstranded", trim=None, num_cores=1, force_bam_paired=False, device=0,
                matrix_dirs=None, any_order=False, device_budget=None, bulk=False):
    """process::bam::process behind main.rs's library loop (src/process/bam.rs:45-243, src/bin/main.rs:95-156).
    matrix_dirs=[dir per library]: also a cell x feature matrix per library (nb_process_bam_cells); output_paths=None with
    matrix_dirs: no TSV rows at all.  any_order=True: from a BAM in any record order, scopes formed on the GPU, no
    force_bam_paired; either the TSV rows (output_paths, matrix_dirs=None: nb_process_bam_rows_any_order, the grouped
    driver's rows on the (UMI, CB)-sorted file) or the matrices (output_paths=None, matrix_dirs: nb_process_bam_cells_any_order).
    device_budget=bytes (any_order only): the device memory that path may allocate; it takes passes over the file by UMI
    bucket when the records do not fit (nb_process_bam_cells_any_order_budget), and writes the same bytes (the rows: the
    same lines, pass by pass).  bulk=True: a BAM without cell barcodes in any record order, counted as FASTQ mode counts the
    reads it stands for (nb_process_bam_bulk): output_paths get exactly what process_fastq writes; trim is ignored, as FASTQ
    mode ignores it; no matrix_dirs, any_order, force_bam_paired or device_budget."""
    if bulk:
        if matrix_dirs is not None or any_order or force_bam_paired or device_budget is not None:
            raise NbError(-1, "bulk counts a BAM as FASTQ mode counts reads: it takes no matrix_dirs, any_order, force_bam_paired or device_budget")
        if output_paths is None or len(output_paths) != len(reference_json_paths):
            raise NbError(-1, "bulk needs one output path per reference library")
        _ck(lib().nb_process_bam_bulk(str(input_file).encode(), _strs(reference_json_paths), _strs(output_paths), len(reference_json_paths),
                                      CHEM[strand_filter], num_cores, device))
        return
    if device_budget is not None:
        _check_budget(device_budget, any_order)
    if any_order:
        if output_paths is not None and matrix_dirs is not None:
            raise NbError(-1, "any_order writes either TSV rows (output_paths) or matrices (matrix_dirs), not both: run the two modes separately")
        if output_paths is None and matrix_dirs is None:
            raise NbError(-1, "any_order needs output_paths or matrix_dirs")
        if force_bam_paired:
            raise NbError(-1, "any_order cannot pair mates (force_bam_paired): the mates of a position-sorted file are not neighbours")
        if output_paths is not None:
            if len(output_paths) != len(reference_json_paths):
                raise NbError(-1, "any_order needs one output path per reference library")
            _ck(lib().nb_process_bam_rows_any_order(str(input_file).encode(), _strs(reference_json_paths), _strs(output_paths), len(reference_json_paths),
                                                    CHEM[strand_filter], trim.encode() if trim else None, num_cores, device,
                                                    int(device_budget) if device_budget is not None else 0))
            return
        if device_budget is not None:
            _ck(lib().nb_process_bam_cells_any_order_budget(str(input_file).encode(), _strs(reference_json_paths), _strs(matrix_dirs), len(reference_json_paths),
                                                            CHEM[strand_filter], trim.encode() if trim else None, num_cores, device, int(device_budget)))
            return
        _ck(lib().nb_process_bam_cells_any_order(str(input_file).encode(), _strs(reference_json_paths), _strs(matrix_dirs), len(reference_json_paths),
                                                 CHEM[strand_filter], trim.encode() if trim else None, num_cores, device))
        return
    if matrix_dirs is not None or output_paths is None:
        _ck(lib().nb_process_bam_cells(str(input_file).encode(), _strs(reference_json_paths), _strs(output_paths) if output_paths is not None else None,
                                       _strs(matrix_dirs) if matrix_dirs is not None else None, len(reference_json_paths),
                                       CHEM[strand_filter], trim.encode() if trim else None, num_cores, int(force_bam_paired), device))
        return
    _ck(lib().nb_process_bam(str(input_file).encode(), _strs(reference_json_paths), _strs(output_paths), len(reference_json_paths),
                             CHEM[strand_filter], trim.encode() if trim else None, num_cores, int(force_bam_paired), device))


_SAMPLE_NAME = re.compile(r"[A-Za-z0-9._-]+")


def read_manifest(path):
    """The samples of a manifest file as [(name, [inputs], line)]: one sample per line, name<TAB>input1[<TAB>input2]; blank
    lines and lines starting with '#' are skipped.  NbError(-1) naming the line on a syntax error, an illegal or repeated
    name, or a manifest without samples."""
    try:
        with open(path, "rb") as f:
            text = f.read().decode("utf-8")
    except (OSError, UnicodeDecodeError) as e:
        raise NbError(-1, "could not read the sample manifest %s: %s" % (path, e))
    out, seen = [], {}
    for k, line in enumerate(text.split("\n"), 1):
        if line.endswith("\r"):
            line = line[:-1]
        if not line.strip(" \t") or line.startswith("#"):
            continue
        at = "%s line %d: " % (path, k)
        col = line.split("\t")
        if not 2 <= len(col) <= 3:
            raise NbError(-1, at + "expected name<TAB>input1[<TAB>input2], found %d column(s)" % len(col))
        if not all(col):
            raise NbError(-1, at + "empty column")
        if not _SAMPLE_NAME.fullmatch(col[0]) or col[0] in (".", ".."):
            raise NbError(-1, at + "sample name '%s' must match [A-Za-z0-9._-]+ and not be '.' or '..'" % col[0])
        if col[0] in seen:
            raise NbError(-1, at + "sample name '%s' is already used on line %d" % (col[0], seen[col[0]]))
        seen[col[0]] = k
        out.append((col[0], col[1:], k))
    if not out:
        raise NbError(-1, "the sample manifest %s has no samples" % path)
    return out


def process_samples(samples, reference_json_paths, output_dirs, strand_filter="unstranded", num_cores=1, device=0, bulk=False):
    """Many samples in one run on one GPU, the libraries set up once (nb_process_samples).  samples: a manifest path (see
    read_manifest) or a list of (name, [inputs]): one or two FASTQs each, or with bulk=True one BAM each.  output_dirs: one
    directory per library; library i's TSV of sample s is <output_dirs[i]>/<s>.tsv, exactly what process_fastq (or
    process_bam(..., bulk=True)) writes for that sample alone.  Bad arguments raise NbError(-1) before the call; a failing
    sample raises the single run's code with the message behind "sample <name> (line N): " (a list: "sample <name>: ")."""
    if isinstance(samples, (str, os.PathLike)):
        entries = read_manifest(os.fspath(samples))
    else:
        if not isinstance(samples, (list, tuple)) or not samples:
            raise NbError(-1, "samples must be a manifest path or a non-empty list of (name, [inputs])")
        entries = []
        for k, smp in enumerate(samples):   # (names, duplicates and input kinds: nb_process_samples, before any device work)
            if not isinstance(smp, (list, tuple)) or len(smp) != 2 or not isinstance(smp[0], str) or not isinstance(smp[1], (list, tuple)) \
                    or not 1 <= len(smp[1]) <= 2 or not all(isinstance(x, (str, os.PathLike)) for x in smp[1]):
                raise NbError(-1, "samples[%d]: expected (name, [one or two input paths])" % k)
            entries.append((smp[0], [os.fspath(x) for x in smp[1]], None))
    if isinstance(reference_json_paths, (str, os.PathLike)) or not reference_json_paths:
        raise NbError(-1, "reference_json_paths must be a non-empty list")
    if isinstance(output_dirs, (str, os.PathLike)) or output_dirs is None or len(output_dirs) != len(reference_json_paths):
        raise NbError(-1, "process_samples needs one output directory per reference library")
    if strand_filter not in CHEM:
        raise NbError(-1, "unknown strand_filter %r" % (strand_filter,))
    names = (C.c_char_p * len(entries))(*[e[0].encode("utf-8") for e in entries])
    inputs = (C.c_char_p * (2 * len(entries)))(*[x for e in entries for x in (e[1][0].encode("utf-8"), e[1][1].encode("utf-8") if len(e[1]) > 1 else None)])
    rc = lib().nb_process_samples(names, inputs, len(entries), _strs(reference_json_paths), _strs(output_dirs), len(reference_json_paths),
                                  CHEM[strand_filter], int(num_cores), int(device), 1 if bulk else 0)
    if rc != 0:
        msg = lib().nb_last_error().decode("utf-8", "replace")
        m = re.match(r"sample ([A-Za-z0-9._-]+): ", msg)
        line = {e[0]: e[2] for e in entries}.get(m.group(1)) if m else None
        if line is not None:
            msg = msg[:m.end(1)] + " (line %d)" % line + msg[m.end(1):]
        raise NbError(rc, msg)


def cell_counts_dict(c):
    def arr(p, n, dt):
        return np.ctypeslib.as_array(p, (n,)).copy() if n else np.zeros(0, dt)
    n_items = int(c.callset_off[c.n_callsets]) if c.n_callsets else 0
    return dict(row_cell=arr(c.row_cell, c.n_rows, np.uint32), row_callset=arr(c.row_callset, c.n_rows, np.uint32),
                row_umis=arr(c.row_umis, c.n_rows, np.int64), row_reads=arr(c.row_reads, c.n_rows, np.int64),
                callset_off=arr(c.callset_off, c.n_callsets + 1, np.uint64) if c.n_callsets else np.zeros(1, np.uint64),
                callset_items=arr(c.callset_items, n_items, np.uint32), n_scopes=c.n_scopes)


def write_cell_matrix(out_dir, library, counts, barcodes):
    """nb_write_cell_matrix (host-only): `counts` is a cells_finalize() dict, `barcodes` the cell ids' CB strings."""
    keep = {k: np.ascontiguousarray(counts[k], dtype=dt) for k, dt in (("row_cell", np.uint32), ("row_callset", np.uint32), ("row_umis", np.int64),
                                                                      ("row_reads", np.int64), ("callset_off", np.uint64), ("callset_items", np.uint32))}
    p = lambda k, t: keep[k].ctypes.data_as(C.POINTER(t))
    c = CellCounts(len(keep["row_cell"]), p("row_cell", C.c_uint32), p("row_callset", C.c_uint32), p("row_umis", C.c_int64), p("row_reads", C.c_int64),
                   len(keep["callset_off"]) - 1, p("callset_off", C.c_uint64), p("callset_items", C.c_uint32), int(counts.get("n_scopes", 0)))
    bc = _strs(barcodes)
    _ck(lib().nb_write_cell_matrix(str(out_dir).encode(), library.h, C.byref(c), bc if len(barcodes) else None, len(barcodes)))


def inflate(data, raw=False, window=0, out_cap=None):
    """The file drivers' own inflate on a buffer (tests against zlib): raw deflate in one piece, or gzip members through
    windows of `window` bytes.  Returns the bytes; NbError on a damaged stream."""
    cap = int(out_cap) if out_cap is not None else max(1 << 16, 1100 * len(data))
    out = C.create_string_buffer(max(cap, 1))
    n = C.c_uint64(0)
    _ck(lib().nb_inflate(bytes(data), len(data), int(raw), int(window), out, cap, C.byref(n)))
    return out.raw[:n.value]


def gunzip_parallel(data, threads=4, chunk_bytes=1 << 20, out_cap=None):
    """A gzip file in memory through the FASTQ feeder's parallel reader (tests against zlib)."""
    cap = int(out_cap) if out_cap is not None else max(1 << 16, 1100 * len(data))
    out = C.create_string_buffer(max(cap, 1))
    n = C.c_uint64(0)
    _ck(lib().nb_gunzip_parallel(bytes(data), len(data), int(threads), int(chunk_bytes), out, cap, C.byref(n)))
    return out.raw[:n.value]


def gzip_fast(data):
    """One gzip member made by the BAM driver's TSV compressor (tests inflate it with zlib)."""
    cap = len(data) + len(data) // 4 + 4096
    out = C.create_string_buffer(cap)
    n = C.c_uint64(0)
    _ck(lib().nb_gzip_fast(bytes(data), len(data), out, cap, C.byref(n)))
    return out.raw[:n.value]


def bam_dump_groups(input_file, out_path, force_bam_paired=False, num_cores=1):
    _ck(lib().nb_bam_dump_groups(str(input_file).encode(), int(force_bam_paired), num_cores, str(out_path).encode()))


def _check_budget(device_budget, any_order=True):
    if not any_order:
        raise NbError(-1, "device_budget applies to any_order=True only")
    if isinstance(device_budget, bool) or not isinstance(device_budget, int) or device_budget <= 0:
        raise NbError(-1, "device_budget must be a positive number of bytes")


def bam_dump_scopes_any_order(input_file, out_path, num_cores=1, device=0, device_budget=None):
    """The device grouping of process_bam(any_order=True), one line per pair (nb_bam_dump_scopes_any_order).  With
    device_budget: the passes of that budget, each line led by its pass index and followed by both slots' bases and quals
    as read back from the store (nb_bam_dump_scopes_any_order_budget)."""
    if device_budget is not None:
        _check_budget(device_budget)
        _ck(lib().nb_bam_dump_scopes_any_order_budget(str(input_file).encode(), num_cores, device, int(device_budget), str(out_path).encode()))
        return
    _ck(lib().nb_bam_dump_scopes_any_order(str(input_file).encode(), num_cores, device, str(out_path).encode()))


def bam_dump_pairs_bulk(input_file, out_path, num_cores=1, device=0):
    """The pairs of process_bam(bulk=True), one line per pair sorted by R1 ordinal (nb_bam_dump_pairs_bulk): R1 ordinal,
    R2 ordinal, both lengths, both NB_FLAG_* bytes; '-' for every R2 field of a single-end file."""
    _ck(lib().nb_bam_dump_pairs_bulk(str(input_file).encode(), num_cores, device, str(out_path).encode()))


def any_order_umi_bucket(umi):
    """The UMI bucket (0..65535) that process_bam(any_order=True, device_budget=...) splits its passes by (host-only)."""
    b = C.c_uint32(0)
    u = umi.encode()
    _ck(lib().nb_any_order_umi_bucket(u, len(u), C.byref(b)))
    return b.value
