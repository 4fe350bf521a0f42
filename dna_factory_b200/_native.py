"""ctypes binding of include/dnaf_b200.h.

There is no CPU fallback: if the CUDA library is missing or no GPU is visible, every entry point
raises.  The library is built in-tree by ``python -m dna_factory_b200.build`` (or __graft_entry__.build()).
"""
import ctypes
import os

import numpy as np

from .build import LIB_PATH

KMAX = 4
CLASS_AUTO, CLASS_X, CLASS_Y, CLASS_MT = 0, 1, 2, 3
E_ARG, E_CUDA, E_NOMEM, E_SPACE, E_SINK, E_INPUT = -1, -2, -3, -4, -5, -6

SINK_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint8), ctypes.c_uint64)


class Stats(ctypes.Structure):
    _fields_ = [("rows", ctypes.c_uint64), ("calls", ctypes.c_uint64), ("text_bytes", ctypes.c_uint64),
                ("bgzf_bytes", ctypes.c_uint64), ("bgzf_blocks", ctypes.c_uint64), ("crc_xor", ctypes.c_uint32),
                ("kernel_launches", ctypes.c_uint32), ("ms_sample", ctypes.c_float), ("ms_format", ctypes.c_float),
                ("ms_deflate", ctypes.c_float), ("ms_fused", ctypes.c_float), ("ms_total", ctypes.c_float),
                ("ms_auto", ctypes.c_float), ("auto_launches", ctypes.c_uint32), ("auto_text_bytes", ctypes.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class DnafError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("dnaf_b200 error %d: %s" % (code, message))
        self.code = code


# every symbol include/dnaf_b200.h declares (tests check the built library exports all of them)
ABI_VERSION = 5   # include/dnaf_b200.h DNAF_ABI_VERSION
EXPORTS = ["dnaf_abi_version", "dnaf_device_count", "dnaf_last_error", "dnaf_create", "dnaf_destroy", "dnaf_set_stream",
           "dnaf_set_chunk_bytes", "dnaf_set_row_base", "dnaf_set_fused", "dnaf_set_samples", "dnaf_set_snps", "dnaf_set_overrides",
           "dnaf_plan", "dnaf_row_offsets", "dnaf_generate", "dnaf_generate_stream", "dnaf_generate_fd", "dnaf_generate_fd_at", "dnaf_generate_device", "dnaf_genotypes",
           "dnaf_text", "dnaf_bgzf_compress", "dnaf_bgzf_bound", "dnaf_bgzf_eof", "dnaf_bgzf_scan", "dnaf_block_log",
           "dnaf_block_log_get", "dnaf_select_snps", "dnaf_parse_snps_jsonl", "dnaf_format_prefixes",
           "dnaf_format_snps_jsonl", "dnaf_debug_lz_block", "dnaf_generate_bed", "dnaf_generate_bed_fd_at",
           "dnaf_generate_bed_device", "dnaf_allele_counts", "dnaf_allele_counts_device", "dnaf_format_assoc",
           "dnaf_genotype_counts", "dnaf_genotype_counts_device", "dnaf_hwe_exact", "dnaf_format_model", "dnaf_format_hardy",
           "dnaf_genotype_tests", "dnaf_genotype_tests_device", "dnaf_fisher_exact", "dnaf_format_assoc_fisher",
           "dnaf_format_model_fisher", "dnaf_perm_case_masks", "dnaf_mperm", "dnaf_mperm_device", "dnaf_format_mperm"]

_lib = None


def load():
    """Load the CUDA library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s is missing: run `python -m dna_factory_b200.build` (needs nvcc). "
                          "dna_factory_b200 has no CPU fallback." % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp, u8p, u32p, u64p = ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint8), ctypes.POINTER(ctypes.c_uint32), \
        ctypes.POINTER(ctypes.c_uint64)
    u64, i32 = ctypes.c_uint64, ctypes.c_int
    f64p = ctypes.POINTER(ctypes.c_double)
    sp = ctypes.POINTER(Stats)
    sig = {
        "dnaf_abi_version": (i32, []),
        "dnaf_device_count": (i32, []),
        "dnaf_last_error": (ctypes.c_char_p, [vp]),
        "dnaf_create": (i32, [i32, ctypes.POINTER(vp)]),
        "dnaf_destroy": (None, [vp]),
        "dnaf_set_stream": (i32, [vp, vp]),
        "dnaf_set_chunk_bytes": (i32, [vp, u64]),
        "dnaf_set_row_base": (i32, [vp, u64]),
        "dnaf_set_fused": (i32, [vp, i32]),
        "dnaf_set_samples": (i32, [vp, ctypes.c_uint32, u8p, u8p]),
        "dnaf_set_snps": (i32, [vp, u64, u8p, u8p, u32p, u8p, u64p]),
        "dnaf_set_overrides": (i32, [vp, u64, u64p, u32p]),
        "dnaf_plan": (i32, [vp, u64, u64, u64p, u64p]),
        "dnaf_row_offsets": (i32, [vp, u64, u64, u64p]),
        "dnaf_generate": (i32, [vp, u64, u64, u64, i32, u8p, u64, sp]),
        "dnaf_generate_stream": (i32, [vp, u64, u64, u64, i32, SINK_FN, vp, sp]),
        "dnaf_generate_fd": (i32, [vp, u64, u64, u64, i32, i32, sp]),
        "dnaf_generate_fd_at": (i32, [vp, u64, u64, u64, i32, i32, u64, sp]),
        "dnaf_generate_device": (i32, [vp, u64, u64, u64, i32, sp]),
        "dnaf_generate_bed": (i32, [vp, u64, u64, u64, u8p, u64, sp]),
        "dnaf_generate_bed_fd_at": (i32, [vp, u64, u64, u64, i32, u64, sp]),
        "dnaf_generate_bed_device": (i32, [vp, u64, u64, u64, sp]),
        "dnaf_allele_counts": (i32, [vp, u64, u64, u64, u32p, sp]),
        "dnaf_allele_counts_device": (i32, [vp, u64, u64, u64, sp]),
        "dnaf_format_assoc": (u64, [u64, ctypes.POINTER(ctypes.c_int32), ctypes.c_char_p, ctypes.POINTER(ctypes.c_int64),
                                    ctypes.POINTER(ctypes.c_int64), u8p, u8p, u32p, u8p]),
        "dnaf_genotype_counts": (i32, [vp, u64, u64, u64, u32p, f64p, sp]),
        "dnaf_genotype_counts_device": (i32, [vp, u64, u64, u64, i32, sp]),
        "dnaf_hwe_exact": (i32, [vp, u64, u32p, f64p]),
        "dnaf_format_model": (u64, [u64, ctypes.POINTER(ctypes.c_int32), ctypes.c_char_p, ctypes.POINTER(ctypes.c_int64),
                                    u8p, u8p, u32p, u8p]),
        "dnaf_format_hardy": (u64, [u64, ctypes.POINTER(ctypes.c_int32), ctypes.c_char_p, ctypes.POINTER(ctypes.c_int64),
                                    u8p, u8p, u32p, f64p, u8p]),
        "dnaf_genotype_tests": (i32, [vp, u64, u64, u64, u32p, f64p, f64p, sp]),
        "dnaf_genotype_tests_device": (i32, [vp, u64, u64, u64, i32, i32, sp]),
        "dnaf_fisher_exact": (i32, [vp, u64, u32p, f64p]),
        "dnaf_format_assoc_fisher": (u64, [u64, ctypes.POINTER(ctypes.c_int32), ctypes.c_char_p, ctypes.POINTER(ctypes.c_int64),
                                           ctypes.POINTER(ctypes.c_int64), u8p, u8p, u32p, f64p, u8p]),
        "dnaf_format_model_fisher": (u64, [u64, ctypes.POINTER(ctypes.c_int32), ctypes.c_char_p, ctypes.POINTER(ctypes.c_int64),
                                           u8p, u8p, u32p, f64p, u8p]),
        "dnaf_perm_case_masks": (i32, [vp, u64, u64, ctypes.c_uint32, u32p, u32p]),
        "dnaf_mperm": (i32, [vp, u64, u64, u64, ctypes.c_uint32, f64p, u32p, f64p, sp]),
        "dnaf_mperm_device": (i32, [vp, u64, u64, u64, ctypes.c_uint32, sp]),
        "dnaf_format_mperm": (u64, [u64, ctypes.POINTER(ctypes.c_int32), ctypes.c_char_p, ctypes.POINTER(ctypes.c_int64), f64p,
                                    u8p]),
        "dnaf_genotypes": (i32, [vp, u64, u64, u64, u8p, u64]),
        "dnaf_text": (i32, [vp, u64, u64, u64, u8p, u64, u64p]),
        "dnaf_bgzf_compress": (i32, [vp, u8p, u64, u8p, u64, sp]),
        "dnaf_bgzf_bound": (u64, [u64]),
        "dnaf_bgzf_eof": (i32, [u8p]),
        "dnaf_bgzf_scan": (i32, [u8p, u64, u32p, u32p, u64, u64p]),
        "dnaf_block_log": (i32, [vp, i32]),
        "dnaf_block_log_get": (i32, [vp, ctypes.POINTER(u32p), ctypes.POINTER(u32p), u64p]),
        "dnaf_parse_snps_jsonl": (ctypes.c_int64, [ctypes.c_char_p, u64, u64, ctypes.POINTER(ctypes.c_int64),
                                                   ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int64), u8p, u8p, f64p,
                                                   ctypes.c_char_p, ctypes.c_uint32, u32p]),
        "dnaf_format_prefixes": (u64, [u64, ctypes.POINTER(ctypes.c_int32), ctypes.c_char_p, ctypes.POINTER(ctypes.c_int64),
                                       ctypes.POINTER(ctypes.c_int64), u8p, u8p, u8p, u64p]),
        "dnaf_format_snps_jsonl": (u64, [u64, ctypes.POINTER(ctypes.c_int32), ctypes.c_char_p, ctypes.POINTER(ctypes.c_int64),
                                         ctypes.POINTER(ctypes.c_int64), u8p, u8p, u32p, ctypes.c_char_p, u32p, u8p]),
        "dnaf_debug_lz_block": (ctypes.c_int64, [ctypes.c_double, i32, u32p, ctypes.c_uint32, u8p, ctypes.c_uint32, i32, u8p, u64]),
        "dnaf_select_snps": (i32, [vp, u64, u64, ctypes.c_uint32, f64p, f64p, u8p, ctypes.c_uint32, f64p, i32, u32p, u8p, u8p,
                                   u32p, u8p, u8p]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    if L.dnaf_abi_version() != ABI_VERSION:
        raise ImportError("%s has ABI %d, this binding needs %d: rebuild with `python -m dna_factory_b200.build --force`"
                          % (LIB_PATH, L.dnaf_abi_version(), ABI_VERSION))
    _lib = L
    return L


def device_count():
    """CUDA devices visible to the process."""
    return int(load().dnaf_device_count())


def _u8(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))


class Engine:
    """One GPU context.  Thin, numpy-in / bytes-out wrapper over the C ABI."""

    def __init__(self, device=0):
        self._lib = load()
        h = ctypes.c_void_p()
        rc = self._lib.dnaf_create(device, ctypes.byref(h))
        if rc:
            raise DnafError(rc, self._lib.dnaf_last_error(None).decode())
        self._h = h
        self.n_samples = 0
        self.n_snps = 0

    def close(self):
        if getattr(self, "_h", None):
            self._lib.dnaf_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc):
        if rc:
            raise DnafError(rc, self._lib.dnaf_last_error(self._h).decode())

    # -- configuration
    def set_stream(self, cuda_stream):
        self._check(self._lib.dnaf_set_stream(self._h, ctypes.c_void_p(cuda_stream)))

    def set_chunk_bytes(self, n):
        self._check(self._lib.dnaf_set_chunk_bytes(self._h, n))

    def set_row_base(self, row_base):
        self._check(self._lib.dnaf_set_row_base(self._h, row_base))

    def set_fused(self, enable):
        self._check(self._lib.dnaf_set_fused(self._h, 1 if enable else 0))

    def set_samples(self, sex, is_control):
        sex = np.ascontiguousarray(sex, dtype=np.uint8)
        ctl = np.ascontiguousarray(is_control, dtype=np.uint8)
        if sex.shape != ctl.shape or sex.ndim != 1:
            raise ValueError("sex and is_control must be 1-D arrays of equal length")
        self._check(self._lib.dnaf_set_samples(self._h, len(sex), _u8(sex), _u8(ctl)))
        self.n_samples = len(sex)

    def set_snps(self, chrom_class, n_alleles, thresholds, prefix_bytes, prefix_off):
        cls = np.ascontiguousarray(chrom_class, dtype=np.uint8)
        k = np.ascontiguousarray(n_alleles, dtype=np.uint8)
        thr = np.ascontiguousarray(thresholds, dtype=np.uint32).reshape(-1)
        pre = np.ascontiguousarray(prefix_bytes, dtype=np.uint8)
        off = np.ascontiguousarray(prefix_off, dtype=np.uint64)
        S = len(cls)
        if len(k) != S or len(thr) != S * KMAX or len(off) != S + 1:
            raise ValueError("inconsistent SNP array lengths")
        if len(pre) < int(off[-1]):
            raise ValueError("prefix_bytes shorter than prefix_off[-1]")
        self._check(self._lib.dnaf_set_snps(self._h, S, _u8(cls), _u8(k), thr.ctypes.data_as(
            ctypes.POINTER(ctypes.c_uint32)), _u8(pre), off.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64))))
        self.n_snps = S

    def set_overrides(self, rows, samples):
        rows = np.ascontiguousarray(rows, dtype=np.uint64)
        samples = np.ascontiguousarray(samples, dtype=np.uint32)
        if len(rows) != len(samples):
            raise ValueError("rows and samples differ in length")
        self._check(self._lib.dnaf_set_overrides(self._h, len(rows), rows.ctypes.data_as(
            ctypes.POINTER(ctypes.c_uint64)), samples.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32))))

    # -- SNP selection (SnpFactory.random_snp_tuples + the sort of pop_factory.py:245, on the GPU)
    def select_snps(self, n, seed, chrom_cdf, chrom_max_pos, chrom_rank, maf_cdf, sort=True):
        """-> dict of columns in final order: order (draw index), chrom_idx, maf_bin, position, ref, alt."""
        ccdf = np.ascontiguousarray(chrom_cdf, dtype=np.float64)
        cmax = np.ascontiguousarray(chrom_max_pos, dtype=np.float64)
        rank = np.ascontiguousarray(chrom_rank, dtype=np.uint8)
        mcdf = np.ascontiguousarray(maf_cdf, dtype=np.float64)
        if not (len(ccdf) == len(cmax) == len(rank)):
            raise ValueError("chromosome arrays differ in length")
        out = dict(order=np.empty(n, np.uint32), chrom_idx=np.empty(n, np.uint8), maf_bin=np.empty(n, np.uint8),
                   position=np.empty(n, np.uint32), ref=np.empty(n, np.uint8), alt=np.empty(n, np.uint8))
        f64p, u32p = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_uint32)
        self._check(self._lib.dnaf_select_snps(
            self._h, n, seed, len(ccdf), ccdf.ctypes.data_as(f64p), cmax.ctypes.data_as(f64p), _u8(rank), len(mcdf),
            mcdf.ctypes.data_as(f64p), 1 if sort else 0, out["order"].ctypes.data_as(u32p), _u8(out["chrom_idx"]),
            _u8(out["maf_bin"]), out["position"].ctypes.data_as(u32p), _u8(out["ref"]), _u8(out["alt"])))
        return out

    # -- sizes
    def plan(self, row_begin, row_end):
        t, b = ctypes.c_uint64(), ctypes.c_uint64()
        self._check(self._lib.dnaf_plan(self._h, row_begin, row_end, ctypes.byref(t), ctypes.byref(b)))
        return t.value, b.value

    # -- the hot path
    def generate(self, row_begin, row_end, seed, level=6):
        """BGZF bytes (whole blocks, no EOF) of rows [row_begin,row_end) -> (bytes, stats dict)."""
        _, bound = self.plan(row_begin, row_end)
        out = np.empty(bound, dtype=np.uint8)
        st = Stats()
        self._check(self._lib.dnaf_generate(self._h, row_begin, row_end, seed, level, _u8(out), bound,
                                            ctypes.byref(st)))
        return out[:st.bgzf_bytes].tobytes(), st.as_dict()

    def generate_into(self, row_begin, row_end, seed, out, level=6):
        """Same, into a caller-owned uint8 numpy buffer; returns stats dict."""
        st = Stats()
        self._check(self._lib.dnaf_generate(self._h, row_begin, row_end, seed, level, _u8(out), out.nbytes,
                                            ctypes.byref(st)))
        return st.as_dict()

    def generate_stream(self, row_begin, row_end, seed, write, level=6):
        """Calls write(bytes) for consecutive pieces of the stream; returns stats dict."""
        err = []

        def cb(user, data, n):
            try:
                write(ctypes.string_at(data, n))
                return 0
            except BaseException as e:  # noqa: surfaced after the call returns
                err.append(e)
                return 1

        st = Stats()
        rc = self._lib.dnaf_generate_stream(self._h, row_begin, row_end, seed, level, SINK_FN(cb), None,
                                            ctypes.byref(st))
        if err:
            raise err[0]
        self._check(rc)
        return st.as_dict()

    def generate_fd(self, row_begin, row_end, seed, fd, level=6):
        """Same stream, written to an open file descriptor by the library itself; returns stats dict."""
        st = Stats()
        self._check(self._lib.dnaf_generate_fd(self._h, row_begin, row_end, seed, level, fd, ctypes.byref(st)))
        return st.as_dict()

    def generate_fd_at(self, row_begin, row_end, seed, fd, file_offset, level=6):
        """Same stream, written with pwrite() at `file_offset` of an open file descriptor; returns stats dict."""
        st = Stats()
        self._check(self._lib.dnaf_generate_fd_at(self._h, row_begin, row_end, seed, level, fd, int(file_offset), ctypes.byref(st)))
        return st.as_dict()

    def row_offsets(self, row_begin, row_end):
        """uint64[row_end-row_begin+1]: text offset of every row of the range (and of its end) from the range's start."""
        out = np.empty(row_end - row_begin + 1, np.uint64)
        self._check(self._lib.dnaf_row_offsets(self._h, row_begin, row_end,
                                               out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64))))
        return out

    def block_log(self, enable=True):
        """Start (and clear) or stop the record of BGZF blocks later generate* calls hand to the host."""
        self._check(self._lib.dnaf_block_log(self._h, 1 if enable else 0))

    def block_log_get(self):
        """(csize, usize) uint32 arrays: compressed and text size of every block logged so far, in order."""
        cs, us = ctypes.POINTER(ctypes.c_uint32)(), ctypes.POINTER(ctypes.c_uint32)()
        n = ctypes.c_uint64()
        self._check(self._lib.dnaf_block_log_get(self._h, ctypes.byref(cs), ctypes.byref(us), ctypes.byref(n)))
        if not n.value:
            return np.zeros(0, np.uint32), np.zeros(0, np.uint32)
        return np.ctypeslib.as_array(cs, (n.value,)).copy(), np.ctypeslib.as_array(us, (n.value,)).copy()

    def generate_device(self, row_begin, row_end, seed, level=6):
        st = Stats()
        self._check(self._lib.dnaf_generate_device(self._h, row_begin, row_end, seed, level,
                                                   ctypes.byref(st)))
        return st.as_dict()

    # -- PLINK 1 .bed rows (payload only: the caller writes the magic bytes, pop_factory.BED_MAGIC, first)
    def bed_pitch(self):
        """Bytes per .bed row: ceil(samples / 4)."""
        return (self.n_samples + 3) // 4

    def generate_bed(self, row_begin, row_end, seed):
        """.bed bytes of rows [row_begin,row_end) -> (bytes, stats dict)."""
        out = np.empty(max((row_end - row_begin) * self.bed_pitch(), 1), dtype=np.uint8)
        st = Stats()
        self._check(self._lib.dnaf_generate_bed(self._h, row_begin, row_end, seed, _u8(out), out.nbytes, ctypes.byref(st)))
        return out[:(row_end - row_begin) * self.bed_pitch()].tobytes(), st.as_dict()

    def generate_bed_into(self, row_begin, row_end, seed, out):
        """Same, into a caller-owned uint8 numpy buffer (page-locked memory is written by DMA); returns stats dict."""
        st = Stats()
        self._check(self._lib.dnaf_generate_bed(self._h, row_begin, row_end, seed, _u8(out), out.nbytes, ctypes.byref(st)))
        return st.as_dict()

    def generate_bed_fd_at(self, row_begin, row_end, seed, fd, file_offset):
        """Same bytes, written with pwrite() at `file_offset` of an open file descriptor; returns stats dict."""
        st = Stats()
        self._check(self._lib.dnaf_generate_bed_fd_at(self._h, row_begin, row_end, seed, fd, int(file_offset), ctypes.byref(st)))
        return st.as_dict()

    def generate_bed_device(self, row_begin, row_end, seed):
        """Same work, output left on the device; returns stats dict."""
        st = Stats()
        self._check(self._lib.dnaf_generate_bed_device(self._h, row_begin, row_end, seed, ctypes.byref(st)))
        return st.as_dict()

    # -- case/control allele counts (the allelic association test, pop_factory --assoc)
    def allele_counts(self, row_begin, row_end, seed):
        """uint32[rows, 4] of rows [row_begin,row_end): ALT in cases, observed in cases, ALT in controls, observed in
        controls (counting rule: include/dnaf_b200.h, dnaf_allele_counts)."""
        return self.allele_counts_stats(row_begin, row_end, seed)[0]

    def allele_counts_stats(self, row_begin, row_end, seed):
        """Same counts -> (counts, stats dict)."""
        out = np.zeros((max(row_end - row_begin, 0), 4), np.uint32)
        st = Stats()
        self._check(self._lib.dnaf_allele_counts(self._h, row_begin, row_end, seed,
                                                 out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)), ctypes.byref(st)))
        return out, st.as_dict()

    def allele_counts_device(self, row_begin, row_end, seed):
        """Same work, counts left on the device; returns stats dict."""
        st = Stats()
        self._check(self._lib.dnaf_allele_counts_device(self._h, row_begin, row_end, seed, ctypes.byref(st)))
        return st.as_dict()

    # -- case/control genotype counts and Hardy-Weinberg exact tests (pop_factory --model / --hardy)
    def genotype_counts(self, row_begin, row_end, seed, hwe=True):
        """(uint32[rows, 10], float64[rows, 3] or None) of rows [row_begin,row_end): per row dip, het, hom, hap, hap_alt
        of the cases, then of the controls, and the Hardy-Weinberg exact P of ALL, AFF, UNAFF (counting rule and test:
        include/dnaf_b200.h, dnaf_genotype_counts)."""
        return self.genotype_counts_stats(row_begin, row_end, seed, hwe)[:2]

    def genotype_counts_stats(self, row_begin, row_end, seed, hwe=True):
        """Same -> (counts, P or None, stats dict)."""
        rows = max(row_end - row_begin, 0)
        out = np.zeros((rows, 10), np.uint32)
        p = np.zeros((rows, 3), np.float64) if hwe else None
        st = Stats()
        self._check(self._lib.dnaf_genotype_counts(
            self._h, row_begin, row_end, seed, out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)),
            p.ctypes.data_as(ctypes.POINTER(ctypes.c_double)) if hwe else None, ctypes.byref(st)))
        return out, p, st.as_dict()

    def genotype_counts_device(self, row_begin, row_end, seed, hwe=True):
        """Same work, results left on the device; returns stats dict."""
        st = Stats()
        self._check(self._lib.dnaf_genotype_counts_device(self._h, row_begin, row_end, seed, int(bool(hwe)), ctypes.byref(st)))
        return st.as_dict()

    def hwe_exact(self, geno):
        """float64[n]: the Hardy-Weinberg exact P of every (n11, n12, n22) row of `geno`, computed by the device kernel
        (dnaf_hwe_exact)."""
        g = np.ascontiguousarray(geno, np.uint32).reshape(-1, 3)
        p = np.zeros(len(g), np.float64)
        self._check(self._lib.dnaf_hwe_exact(self._h, len(g), g.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)),
                                             p.ctypes.data_as(ctypes.POINTER(ctypes.c_double))))
        return p

    # -- counts, Hardy-Weinberg and Fisher exact tests in one pass (pop_factory --fisher / --model / --hardy)
    def genotype_tests(self, row_begin, row_end, seed, hwe=True, fisher=True):
        """(uint32[rows, 10], float64[rows, 3] or None, float64[rows, 4] or None) of rows [row_begin,row_end): the
        genotype counts, the Hardy-Weinberg exact P of ALL, AFF, UNAFF and log10 of the Fisher exact P of GENO, ALLELIC,
        DOM, REC (include/dnaf_b200.h, dnaf_genotype_tests)."""
        return self.genotype_tests_stats(row_begin, row_end, seed, hwe, fisher)[:3]

    def genotype_tests_stats(self, row_begin, row_end, seed, hwe=True, fisher=True):
        """Same -> (counts, P or None, log10 P or None, stats dict)."""
        rows = max(row_end - row_begin, 0)
        out = np.zeros((rows, 10), np.uint32)
        p = np.zeros((rows, 3), np.float64) if hwe else None
        l = np.zeros((rows, 4), np.float64) if fisher else None
        f64p = ctypes.POINTER(ctypes.c_double)
        st = Stats()
        self._check(self._lib.dnaf_genotype_tests(
            self._h, row_begin, row_end, seed, out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)),
            p.ctypes.data_as(f64p) if hwe else None, l.ctypes.data_as(f64p) if fisher else None, ctypes.byref(st)))
        return out, p, l, st.as_dict()

    def genotype_tests_device(self, row_begin, row_end, seed, hwe=True, fisher=True):
        """Same work, results left on the device; returns stats dict."""
        st = Stats()
        self._check(self._lib.dnaf_genotype_tests_device(self._h, row_begin, row_end, seed, int(bool(hwe)), int(bool(fisher)),
                                                         ctypes.byref(st)))
        return st.as_dict()

    def fisher_exact(self, tables):
        """float64[n]: log10 of the two-sided Fisher exact P of every (x1, x2, x3, y1, y2, y3) row of `tables` (case row,
        control row), computed by the device kernel (dnaf_fisher_exact); NaN where there is no test."""
        t = np.ascontiguousarray(tables, np.uint32).reshape(-1, 6)
        l = np.zeros(len(t), np.float64)
        self._check(self._lib.dnaf_fisher_exact(self._h, len(t), t.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)),
                                                l.ctypes.data_as(ctypes.POINTER(ctypes.c_double))))
        return l

    # -- max(T) permutation tests of ALLELIC and REC (pop_factory --mperm)
    def perm_case_masks(self, seed, first_perm, n_perm):
        """(uint32[n_perm, ceil(N/32)], uint32[n_perm, 2]): the case masks of permutations first_perm ..
        first_perm + n_perm - 1 (bit i & 31 of word i >> 5 = sample i is a case) and their (male, female) cases
        (include/dnaf_b200.h, dnaf_perm_case_masks)."""
        masks = np.zeros((n_perm, (self.n_samples + 31) // 32), np.uint32)
        sexc = np.zeros((n_perm, 2), np.uint32)
        u32p = ctypes.POINTER(ctypes.c_uint32)
        self._check(self._lib.dnaf_perm_case_masks(self._h, seed, first_perm, n_perm, masks.ctypes.data_as(u32p),
                                                   sexc.ctypes.data_as(u32p)))
        return masks, sexc

    def mperm(self, row_begin, row_end, seed, n_perm):
        """(float64[rows, 2], uint32[rows, 2], float64[n_perm, 2]) of rows [row_begin,row_end) under n_perm permutations:
        the observed ALLELIC and REC statistics (NaN: no test), how many permutations reach them, and every
        permutation's maximum over the rows (include/dnaf_b200.h, dnaf_mperm)."""
        return self.mperm_stats(row_begin, row_end, seed, n_perm)[:3]

    def mperm_stats(self, row_begin, row_end, seed, n_perm):
        """Same -> (t_obs, exceed, max_t, stats dict)."""
        rows = max(row_end - row_begin, 0)
        t_obs = np.zeros((rows, 2), np.float64)
        exceed = np.zeros((rows, 2), np.uint32)
        max_t = np.zeros((n_perm, 2), np.float64)
        f64p = ctypes.POINTER(ctypes.c_double)
        st = Stats()
        self._check(self._lib.dnaf_mperm(self._h, row_begin, row_end, seed, n_perm, t_obs.ctypes.data_as(f64p),
                                         exceed.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)), max_t.ctypes.data_as(f64p),
                                         ctypes.byref(st)))
        return t_obs, exceed, max_t, st.as_dict()

    def mperm_device(self, row_begin, row_end, seed, n_perm):
        """Same work, results left on the device; returns stats dict."""
        st = Stats()
        self._check(self._lib.dnaf_mperm_device(self._h, row_begin, row_end, seed, n_perm, ctypes.byref(st)))
        return st.as_dict()

    # -- parity gates
    def genotypes(self, row_begin, row_end, seed):
        rows = row_end - row_begin
        out = np.empty(max(rows * self.n_samples * 2, 1), dtype=np.uint8)
        self._check(self._lib.dnaf_genotypes(self._h, row_begin, row_end, seed, _u8(out), out.nbytes))
        return out[:rows * self.n_samples * 2].reshape(rows, self.n_samples, 2)

    def text(self, row_begin, row_end, seed):
        t, _ = self.plan(row_begin, row_end)
        out = np.empty(max(t, 1), dtype=np.uint8)
        n = ctypes.c_uint64()
        self._check(self._lib.dnaf_text(self._h, row_begin, row_end, seed, _u8(out), out.nbytes, ctypes.byref(n)))
        return out[:n.value].tobytes()

    def bgzf_compress(self, data):
        buf = np.frombuffer(bytes(data) + b"\0", dtype=np.uint8)
        n = len(buf) - 1
        bound = int(self._lib.dnaf_bgzf_bound(n))
        out = np.empty(bound, dtype=np.uint8)
        st = Stats()
        self._check(self._lib.dnaf_bgzf_compress(self._h, _u8(buf), n, _u8(out), bound, ctypes.byref(st)))
        return out[:st.bgzf_bytes].tobytes(), st.as_dict()


def bgzf_scan(data):
    """(csize, usize) of every block of a BGZF stream held in memory (host only, no GPU work)."""
    lib = load()
    buf = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data
    n = ctypes.c_uint64()
    rc = lib.dnaf_bgzf_scan(_u8(buf) if len(buf) else None, len(buf), None, None, 0, ctypes.byref(n))
    if rc:
        raise DnafError(rc, "not a whole number of BGZF blocks")
    cs, us = np.empty(n.value, np.uint32), np.empty(n.value, np.uint32)
    if n.value:
        u32p = ctypes.POINTER(ctypes.c_uint32)
        rc = lib.dnaf_bgzf_scan(_u8(buf), len(buf), cs.ctypes.data_as(u32p), us.ctypes.data_as(u32p), n.value, ctypes.byref(n))
        if rc:
            raise DnafError(rc, "not a whole number of BGZF blocks")
    return cs, us


def parse_snps_jsonl(data):
    """Columns of an inflated snps.json (bytes), or None when a record needs the generic json path."""
    lib = load()
    cap = data.count(b"\n") + 1
    ids = np.empty(cap, np.int64)
    ci = np.empty(cap, np.int32)
    pos = np.empty(cap, np.int64)
    k = np.empty(cap, np.uint8)
    nts = np.empty((cap, KMAX), np.uint8)
    cum = np.empty((cap, KMAX), np.float64)
    labels = ctypes.create_string_buffer(8 * 256)
    nl = ctypes.c_uint32()
    n = lib.dnaf_parse_snps_jsonl(data, len(data), cap, ids.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
                                  ci.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                                  pos.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), _u8(k), _u8(nts),
                                  cum.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), labels, 256, ctypes.byref(nl))
    if n < 0:
        return None
    names = [labels.raw[8 * i:8 * i + 8].split(b"\0")[0].decode("latin-1") for i in range(nl.value)]
    return dict(ids=ids[:n], chrom_idx=ci[:n], chrom_labels=names, position=pos[:n], n_alleles=k[:n], nts=nts[:n], cum=cum[:n])


def _label_block(labels):
    buf = bytearray(8 * len(labels))
    for i, name in enumerate(labels):
        b = name.encode("latin-1")
        if not 0 < len(b) <= 7:
            raise ValueError("chromosome label %r does not fit 7 bytes" % name)
        buf[8 * i:8 * i + len(b)] = b
    return bytes(buf)


def format_prefixes(ids, chrom_idx, labels, position, n_alleles, nts):
    """Row prefixes (pop_factory.py:503-507) of a column-form SNP table -> (bytes array incl. one pad byte, offsets)."""
    lib = load()
    n = len(ids)
    ids = np.ascontiguousarray(ids, np.int64)
    pos = np.ascontiguousarray(position, np.int64)
    ci = np.ascontiguousarray(chrom_idx, np.int32)
    k = np.ascontiguousarray(n_alleles, np.uint8)
    nt = np.ascontiguousarray(nts, np.uint8)
    out = np.empty(n * 72 + 16, np.uint8)
    off = np.empty(n + 1, np.uint64)
    i64p = ctypes.POINTER(ctypes.c_int64)
    used = lib.dnaf_format_prefixes(n, ci.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), _label_block(labels),
                                    pos.ctypes.data_as(i64p), ids.ctypes.data_as(i64p), _u8(k), _u8(nt), _u8(out),
                                    off.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)))
    out[used] = 0
    return out[:used + 1], off


def format_snps_jsonl(ids, chrom_idx, labels, position, n_alleles, nts, cum):
    """snps.json text (SNPTuples.__str__ per line, pop_factory.py:118-124) of a column-form SNP table -> bytes."""
    import json
    lib = load()
    n = len(ids)
    ids = np.ascontiguousarray(ids, np.int64)
    pos = np.ascontiguousarray(position, np.int64)
    ci = np.ascontiguousarray(chrom_idx, np.int32)
    k = np.ascontiguousarray(n_alleles, np.uint8)
    nt = np.ascontiguousarray(nts, np.uint8)
    uniq, inv = np.unique(np.ascontiguousarray(cum, np.float64), return_inverse=True)
    strs = [json.dumps(float(v)).encode() + b"\0" for v in uniq]     # Python's float repr, as json.dumps prints it
    roff = np.zeros(len(strs) + 1, np.uint32)
    roff[1:] = np.cumsum([len(x) for x in strs])
    ridx = np.ascontiguousarray(inv.reshape(n, KMAX), np.uint32)
    out = np.empty(n * (96 + KMAX * (8 + max(len(x) for x in strs))) + 16, np.uint8)
    i64p, u32p = ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_uint32)
    used = lib.dnaf_format_snps_jsonl(n, ci.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), _label_block(labels),
                                      pos.ctypes.data_as(i64p), ids.ctypes.data_as(i64p), _u8(k), _u8(nt),
                                      ridx.ctypes.data_as(u32p), b"".join(strs), roff.ctypes.data_as(u32p), _u8(out))
    return out[:used].tobytes()


def format_assoc(ids, chrom_idx, labels, position, n_alleles, nts, counts):
    """.assoc body lines (dnaf_format_assoc: F_A, F_U, CHISQ, P, OR in double, "%.4g", NA rules) of a column-form SNP
    table and its uint32[rows, 4] allele counts -> bytes."""
    lib = load()
    n = len(ids)
    if n == 0:
        return b""
    ids = np.ascontiguousarray(ids, np.int64)
    pos = np.ascontiguousarray(position, np.int64)
    ci = np.ascontiguousarray(chrom_idx, np.int32)
    k = np.ascontiguousarray(n_alleles, np.uint8)
    nt = np.ascontiguousarray(nts, np.uint8).reshape(n, KMAX)
    cnt = np.ascontiguousarray(counts, np.uint32).reshape(n, 4)
    out = np.empty(n * 192 + 16, np.uint8)
    i64p = ctypes.POINTER(ctypes.c_int64)
    used = lib.dnaf_format_assoc(n, ci.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), _label_block(labels),
                                 ids.ctypes.data_as(i64p), pos.ctypes.data_as(i64p), _u8(nt), _u8(k),
                                 cnt.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)), _u8(out))
    return out[:used].tobytes()


def _geno_columns(ids, chrom_idx, labels, n_alleles, nts, counts):
    n = len(ids)
    return (np.ascontiguousarray(ids, np.int64), np.ascontiguousarray(chrom_idx, np.int32), _label_block(labels),
            np.ascontiguousarray(n_alleles, np.uint8), np.ascontiguousarray(nts, np.uint8).reshape(n, KMAX),
            np.ascontiguousarray(counts, np.uint32).reshape(n, 10))


def format_model(ids, chrom_idx, labels, n_alleles, nts, counts):
    """.model body lines (dnaf_format_model: GENO, TREND, ALLELIC, DOM, REC per SNP) of a column-form SNP table and its
    uint32[rows, 10] genotype counts -> bytes."""
    lib = load()
    n = len(ids)
    if n == 0:
        return b""
    ids, ci, lab, k, nt, cnt = _geno_columns(ids, chrom_idx, labels, n_alleles, nts, counts)
    out = np.empty(n * 960 + 16, np.uint8)
    used = lib.dnaf_format_model(n, ci.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), lab,
                                 ids.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), _u8(nt), _u8(k),
                                 cnt.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)), _u8(out))
    return out[:used].tobytes()


def format_hardy(ids, chrom_idx, labels, n_alleles, nts, counts, hwe_p):
    """.hwe body lines (dnaf_format_hardy: ALL, AFF, UNAFF per SNP) of a column-form SNP table, its uint32[rows, 10]
    genotype counts and float64[rows, 3] exact-test P -> bytes."""
    lib = load()
    n = len(ids)
    if n == 0:
        return b""
    ids, ci, lab, k, nt, cnt = _geno_columns(ids, chrom_idx, labels, n_alleles, nts, counts)
    p = np.ascontiguousarray(hwe_p, np.float64).reshape(n, 3)
    out = np.empty(n * 576 + 16, np.uint8)
    used = lib.dnaf_format_hardy(n, ci.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), lab,
                                 ids.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), _u8(nt), _u8(k),
                                 cnt.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)),
                                 p.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), _u8(out))
    return out[:used].tobytes()


def format_assoc_fisher(ids, chrom_idx, labels, position, n_alleles, nts, counts, log10p):
    """.assoc.fisher body lines (dnaf_format_assoc_fisher: F_A, F_U, P of Fisher ALLELIC, OR) of a column-form SNP
    table, its uint32[rows, 10] genotype counts and float64[rows, 4] Fisher log10 P -> bytes."""
    lib = load()
    n = len(ids)
    if n == 0:
        return b""
    ids, ci, lab, k, nt, cnt = _geno_columns(ids, chrom_idx, labels, n_alleles, nts, counts)
    pos = np.ascontiguousarray(position, np.int64)
    l = np.ascontiguousarray(log10p, np.float64).reshape(n, 4)
    out = np.empty(n * 192 + 16, np.uint8)
    i64p = ctypes.POINTER(ctypes.c_int64)
    used = lib.dnaf_format_assoc_fisher(n, ci.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), lab, ids.ctypes.data_as(i64p),
                                        pos.ctypes.data_as(i64p), _u8(nt), _u8(k),
                                        cnt.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)),
                                        l.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), _u8(out))
    return out[:used].tobytes()


def format_model_fisher(ids, chrom_idx, labels, n_alleles, nts, counts, log10p):
    """Fisher .model body lines (dnaf_format_model_fisher: GENO, TREND, ALLELIC, DOM, REC per SNP) of a column-form SNP
    table, its uint32[rows, 10] genotype counts and float64[rows, 4] Fisher log10 P -> bytes."""
    lib = load()
    n = len(ids)
    if n == 0:
        return b""
    ids, ci, lab, k, nt, cnt = _geno_columns(ids, chrom_idx, labels, n_alleles, nts, counts)
    l = np.ascontiguousarray(log10p, np.float64).reshape(n, 4)
    out = np.empty(n * 960 + 16, np.uint8)
    used = lib.dnaf_format_model_fisher(n, ci.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), lab,
                                        ids.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), _u8(nt), _u8(k),
                                        cnt.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)),
                                        l.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), _u8(out))
    return out[:used].tobytes()


def format_mperm(ids, chrom_idx, labels, emp):
    """.mperm body lines (dnaf_format_mperm: CHR SNP EMP1 EMP2, "%.4g", NA for NaN) of a column-form SNP table and its
    float64[rows, 2] (EMP1, EMP2) -> bytes."""
    lib = load()
    n = len(ids)
    if n == 0:
        return b""
    ids = np.ascontiguousarray(ids, np.int64)
    ci = np.ascontiguousarray(chrom_idx, np.int32)
    e = np.ascontiguousarray(emp, np.float64).reshape(n, 2)
    out = np.empty(n * 96 + 16, np.uint8)
    used = lib.dnaf_format_mperm(n, ci.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), _label_block(labels),
                                 ids.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), e.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                 _u8(out))
    return out[:used].tobytes()


def debug_lz_block(p_minor, level, allele_bits, n_cells, prefix=b"", ends_row=False):
    """Raw deflate bytes of one autosome segment under the LZ tier `level` (host self-test hook, see dnaf_b200.h)."""
    L = load()
    bits = np.ascontiguousarray(allele_bits, dtype=np.uint32)
    assert bits.size * 32 >= 2 * n_cells
    pre = np.frombuffer(bytes(prefix) + b"\0", dtype=np.uint8)
    out = np.empty(4 * n_cells + 1024, dtype=np.uint8)
    n = L.dnaf_debug_lz_block(float(p_minor), int(level), bits.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)), int(n_cells),
                              _u8(pre), len(prefix), 1 if ends_row else 0, _u8(out), out.size)
    if n < 0:
        raise DnafError(int(n), "dnaf_debug_lz_block failed")
    return out[:n].tobytes()


def bgzf_eof():
    out = np.empty(28, dtype=np.uint8)
    load().dnaf_bgzf_eof(_u8(out))
    return out.tobytes()
