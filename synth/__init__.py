"""Deterministic synthetic workloads shaped like BASELINE.json's configs (SURVEY.md §8d).  Test / bench infrastructure
shared by the GPU arm and the CPU oracle arm so that both see byte-identical inputs; not part of the product."""
import ctypes as C
import json
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libsynth.so")
_lib = None


def build(force=False):
    src = os.path.join(_HERE, "synth.cpp")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-pthread", "-shared", "-o", _SO, src, "-lz"])
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        L.synth_library.restype = C.c_uint64
        L.synth_library.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
        L.synth_pair_offsets.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, C.c_double, C.c_void_p, C.c_void_p, C.c_int]
        L.synth_pairs.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_uint32,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.synth_umi_sizes.restype = C.c_uint64
        L.synth_umi_sizes.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p]
        L.synth_umi_reads.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_double, C.c_void_p, C.c_void_p,
                                      C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.synth_write_fastq.restype = C.c_uint64
        L.synth_write_fastq.argtypes = [C.c_char_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.synth_write_bam.restype = C.c_uint64
        L.synth_write_bam.argtypes = [C.c_char_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_int, C.c_void_p]
        L.synth_encode_2bit.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_int]
        _lib = L
    return _lib


BASE_CONFIG = dict(trim_target_length=40, trim_strictness=0.9, score_percent=0.33, score_filter=25, score_threshold=50, num_mismatches=0,
                   discard_multiple_matches=False, max_hits_to_report=10, intersect_level=0, group_on="", discard_multi_hits=0,
                   require_valid_pair=False, data_type="DNA")   # tests/test-sequences/libraries/basic.json object 0


class SynthLibrary:
    """n_fam families x n_all alleles (C2: 200 x 5, seed 1234).  Names are zero-padded so natural order == byte order."""

    def __init__(self, seed=1234, n_fam=200, n_all=5, group_on="", **cfg_overrides):
        self.seed, self.n_fam, self.n_all = seed, n_fam, n_all
        n = n_fam * n_all
        self.off = np.zeros(n + 1, dtype=np.uint64)
        tot = lib().synth_library(seed, n_fam, n_all, None, self.off.ctypes.data)
        self.seqs = np.zeros(tot, dtype=np.uint8)
        lib().synth_library(seed, n_fam, n_all, self.seqs.ctypes.data, self.off.ctypes.data)
        w = max(4, len(str(n_fam - 1)))
        self.names = ["F%0*d_A%02d" % (w, f, a) for f in range(n_fam) for a in range(n_all)]
        self.families = ["F%0*d" % (w, f) for f in range(n_fam) for a in range(n_all)]
        self.config = dict(BASE_CONFIG)
        self.config["group_on"] = group_on
        self.config.update(cfg_overrides)

    def sequences(self):
        b = self.seqs.tobytes()
        return [b[int(self.off[i]):int(self.off[i + 1])].decode() for i in range(len(self.names))]

    def to_json_obj(self):
        seqs = self.sequences()
        return [self.config, {"headers": ["reference_genome", "sequence_name", "family", "nt_length", "sequence"],
                              "columns": [["synth"] * len(seqs), self.names, self.families, [str(len(s)) for s in seqs], seqs]}]

    def write_json(self, path):
        with open(path, "w") as f:
            json.dump(self.to_json_obj(), f)
        return path


def pairs(library, first, n, seed=1234, read_len=150, dup_rate=0.1, err=0.003, paired=True, threads=8, out=None):
    """Read pairs [first, first+n) of the C2-shaped workload -> (r1, r1_off, r2, r2_off) numpy arrays (r2 None if single)."""
    o1 = np.zeros(n + 1, dtype=np.uint64)
    o2 = np.zeros(n + 1, dtype=np.uint64) if paired else None
    lib().synth_pair_offsets(seed, first, n, read_len, dup_rate, o1.ctypes.data, o2.ctypes.data if paired else None, threads)
    r1 = np.empty(int(o1[-1]) + 64, dtype=np.uint8) if out is None else out[0]
    r2 = (np.empty(int(o2[-1]) + 64, dtype=np.uint8) if out is None else out[1]) if paired else None
    lib().synth_pairs(seed, first, n, read_len, dup_rate, err, library.seqs.ctypes.data, library.off.ctypes.data, len(library.names),
                      r1.ctypes.data, o1.ctypes.data, r2.ctypes.data if paired else None, o2.ctypes.data if paired else None, threads)
    return r1, o1, r2, o2


def umi_reads(library, first_group, n_groups, seed=2345, L=91, n_cells=8000, err=0.003, threads=8):
    """10x-style single-end records (C3 shape): returns dict(bases, qual, off, cell, scope, sizes)."""
    sizes = np.zeros(n_groups, dtype=np.uint32)
    tot = lib().synth_umi_sizes(seed, first_group, n_groups, sizes.ctypes.data)
    start = np.zeros(n_groups + 1, dtype=np.uint64)
    start[1:] = np.cumsum(sizes, dtype=np.uint64)
    bases = np.empty(tot * L + 64, dtype=np.uint8)
    qual = np.empty(tot * L + 64, dtype=np.uint8)
    cell = np.zeros(tot, dtype=np.uint32)
    scope = np.zeros(tot, dtype=np.uint32)
    lib().synth_umi_reads(seed, first_group, n_groups, sizes.ctypes.data, start.ctypes.data, L, n_cells, err, library.seqs.ctypes.data,
                          library.off.ctypes.data, len(library.names), bases.ctypes.data, qual.ctypes.data, cell.ctypes.data, scope.ctypes.data, threads)
    off = np.arange(tot + 1, dtype=np.uint64) * L
    return dict(bases=bases, qual=qual, off=off, cell=cell, scope=scope, sizes=sizes, n_reads=int(tot))


def write_umi_bam(path, u, L=91, first_scope=0, level=1, threads=8, name_ids=None):
    """Writes the records of `umi_reads` as a 10x-style unaligned BAM (threaded BGZF).  Record i is named r<i>, or
    r<name_ids[i]> (a uint64 array) so that a reordering of another file's records keeps their names.  Returns the file size."""
    ids = None if name_ids is None else np.ascontiguousarray(name_ids, dtype=np.uint64)
    n = lib().synth_write_bam(str(path).encode(), u["n_reads"], L, u["bases"].ctypes.data, u["qual"].ctypes.data, u["cell"].ctypes.data, u["scope"].ctypes.data,
                              first_scope, level, threads, None if ids is None else ids.ctypes.data)
    if not n:
        raise IOError("could not write %s" % path)
    return int(n)


def write_fastq(path, r, off, mate=1, level=1):
    """FASTQ (gzip when the path ends in .gz) of the reads of `pairs`.  Returns the uncompressed size."""
    n = lib().synth_write_fastq(str(path).encode(), len(off) - 1, r.ctypes.data, off.ctypes.data, mate, level)
    if not n:
        raise IOError("could not write %s" % path)
    return int(n)


def encode_2bit(src, n_bases, dst=None, threads=8):
    """ASCII bases -> NB_SEQ_2BIT byte stream (4 bases per byte, first base in the low bits; non-ACGT -> A)."""
    if dst is None:
        dst = np.zeros((n_bases + 3) // 4 + 64, dtype=np.uint8)
    lib().synth_encode_2bit(src.ctypes.data, int(n_bases), dst.ctypes.data, threads)
    return dst
