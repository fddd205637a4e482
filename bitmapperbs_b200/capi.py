"""ctypes binding of include/bmbs.h (same names, same argument meaning, same error behaviour)."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

NONE, EXACT_UNIQUE, MULTI_EXACT, ONE_MISMATCH, VERIFY = 0, 1, 2, 3, 4

# numpy views of the C structs
ReadResult = np.dtype([("site", "<u8"), ("first_cand", "<u4"), ("n_cand", "<u4"), ("one_mismatch_pos", "<i2"),
                       ("state", "u1"), ("is_multiple_map", "u1"), ("reserved", "<u4")])
Cand = np.dtype([("site", "<u8"), ("vote", "<u4"), ("end_site", "<i2"), ("err", "<u2")])
assert ReadResult.itemsize == 24 and Cand.itemsize == 16
# bmbs_final: one finished single-end read (bmbs_batch_finish)
FIN_UNMAPPED, FIN_UNIQUE, FIN_AMBIGUOUS, FIN_DP, FIN_HOST = 0, 1, 2, 3, 4
FINF_REVERSE, FINF_AMBIGUOUS = 1, 2
Final = np.dtype([("site", "<u8"), ("chrom_pos", "<u8"), ("aux_first", "<u4"), ("end_site", "<i2"), ("nm", "u1"), ("sbd", "u1"), ("status", "u1"),
                  ("flags", "u1"), ("mapq_fixed", "u1"), ("k", "u1"), ("n_aux", "<u4")])
assert Final.itemsize == 32


class Params(C.Structure):
    _fields_ = [("e_rate", C.c_double), ("seed_len", C.c_int), ("min_ins", C.c_int), ("max_ins", C.c_int), ("sensitive", C.c_int), ("ambiguous_out", C.c_int)]


class Scoring(C.Structure):
    """bmbs_scoring (include/bmbs.h): --mp_max --mp_min --np --gap_open --gap_extension, quality base"""
    _fields_ = [("mp_max", C.c_int), ("mp_min", C.c_int), ("n_pen", C.c_int), ("gap_open", C.c_int), ("gap_ext", C.c_int), ("q_base", C.c_int)]


RefineItem = np.dtype([("site", "<u8"), ("seq_off", "<u4"), ("len", "<u2"), ("k", "u1"), ("pad", "u1")])
RefineResult = np.dtype([("score", "<i4"), ("qb", "<i4"), ("qe", "<i4"), ("n_ops", "<u4"), ("ops_off", "<u4"), ("nm", "<u4")])


class BmbsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"bmbs error {code}: {msg}")
        self.code = code


def lib_path() -> Path:
    return Path(__file__).resolve().parent / "libbmbs_gpu.so"


_lib = None

EXPORTS = ["bmbs_index_load", "bmbs_index_free", "bmbs_index_genome_length", "bmbs_index_device_bytes", "bmbs_last_error",
           "bmbs_params_default", "bmbs_map_batch_se", "bmbs_map_batch_pe", "bmbs_verify", "bmbs_batch_create", "bmbs_batch_free",
           "bmbs_batch_upload", "bmbs_batch_run", "bmbs_batch_download", "bmbs_batch_sync", "bmbs_batch_timings",
           "bmbs_batch_counters", "bmbs_batch_launches", "bmbs_batch_verify", "bmbs_batch_download_verify", "bmbs_ubench_int_pipe", "bmbs_pinned_alloc", "bmbs_pinned_free", "bmbs_ubench_random_sectors",
           "bmbs_refiner_create", "bmbs_refiner_free", "bmbs_refine", "bmbs_batch_finish", "bmbs_batch_download_final", "bmbs_batch_finish_counters", "bmbs_debug_sort_order", "bmbs_refiner_kernel_ms", "bmbs_batch_output_sizes",
           "bmbs_batch_grid"]


def load_library():
    """dlopen libbmbs_gpu.so; raises (no fallback) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not p.exists():
        raise BmbsError(-1, f"{p} is missing: build it with `python -m bitmapperbs_b200.build` (nvcc, sm_100a); there is no CPU fallback")
    L = C.CDLL(str(p))
    vp, u64p = C.c_void_p, C.POINTER(C.c_uint64)
    L.bmbs_last_error.restype = C.c_char_p
    L.bmbs_index_load.argtypes = [C.c_char_p, C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]
    L.bmbs_index_free.argtypes = [vp]
    L.bmbs_index_genome_length.argtypes = [vp]; L.bmbs_index_genome_length.restype = C.c_uint64
    L.bmbs_index_device_bytes.argtypes = [vp]; L.bmbs_index_device_bytes.restype = C.c_uint64
    L.bmbs_params_default.argtypes = [C.POINTER(Params)]
    for f in (L.bmbs_map_batch_se, L.bmbs_map_batch_pe):
        f.argtypes = [vp, C.c_int, vp, vp, C.c_int, C.POINTER(Params), vp, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    L.bmbs_verify.argtypes = [vp, C.c_int, vp, vp, C.c_int, vp, vp, C.c_size_t, C.c_double, vp, vp]
    L.bmbs_batch_create.argtypes = [vp, C.c_int, C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(vp)]
    L.bmbs_batch_free.argtypes = [vp]
    L.bmbs_batch_upload.argtypes = [vp, vp, vp, C.c_int, C.c_int]
    L.bmbs_batch_run.argtypes = [vp, C.POINTER(Params)]
    L.bmbs_batch_download.argtypes = [vp, vp, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    L.bmbs_batch_sync.argtypes = [vp]
    L.bmbs_batch_output_sizes.argtypes = [vp, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    L.bmbs_batch_timings.argtypes = [vp, C.POINTER(C.c_float)]
    L.bmbs_batch_counters.argtypes = [vp, u64p]
    L.bmbs_batch_launches.argtypes = [vp]
    L.bmbs_batch_grid.argtypes = [vp, C.POINTER(C.c_uint32)]
    L.bmbs_batch_verify.argtypes = [vp, vp, vp, C.c_size_t, C.c_double]
    L.bmbs_batch_download_verify.argtypes = [vp, vp, vp, C.c_size_t]
    L.bmbs_ubench_int_pipe.argtypes = [C.c_int, C.POINTER(C.c_double)]
    L.bmbs_ubench_random_sectors.argtypes = [C.c_int, C.c_size_t, C.POINTER(C.c_double)]
    L.bmbs_batch_finish.argtypes = [vp]
    L.bmbs_batch_download_final.argtypes = [vp, vp, vp, C.c_size_t, C.POINTER(C.c_size_t), vp, C.c_size_t, C.POINTER(C.c_size_t)]
    L.bmbs_batch_finish_counters.argtypes = [vp, u64p]
    L.bmbs_debug_sort_order.argtypes = [C.c_int, vp, vp, C.c_uint32, vp, vp]
    L.bmbs_refiner_create.argtypes = [vp, C.c_int, C.POINTER(vp)]
    L.bmbs_refiner_free.argtypes = [vp]
    L.bmbs_refiner_kernel_ms.argtypes = [vp, C.POINTER(C.c_float)]
    L.bmbs_refine.argtypes = [vp, vp, vp, C.c_size_t, vp, C.c_size_t, C.POINTER(Scoring), vp, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    _lib = L
    return L


def _check(rc):
    if rc != 0:
        raise BmbsError(rc, load_library().bmbs_last_error().decode(errors="replace"))


def int_pipe_peak(dev=0) -> float:
    """measured LOP3+IADD3 throughput of the device, 32-bit integer ops per second"""
    v = C.c_double(0)
    _check(load_library().bmbs_ubench_int_pipe(dev, C.byref(v)))
    return v.value


def random_sector_peak(dev=0, nbytes=8 << 30) -> float:
    """measured rate of independent random 32-byte sector loads, sectors per second"""
    v = C.c_double(0)
    _check(load_library().bmbs_ubench_random_sectors(dev, nbytes, C.byref(v)))
    return v.value


def debug_sort_order(vote_lists, dev=0):
    """the order std::sort by vote (descending) leaves each list in, replayed by the device finishing's warp routine
    -> (list of position arrays, ok flags)"""
    offs = np.zeros(len(vote_lists) + 1, dtype=np.uint32)
    offs[1:] = np.cumsum([len(v) for v in vote_lists], dtype=np.uint32)
    votes = np.concatenate([np.asarray(v, dtype=np.uint32) for v in vote_lists]) if vote_lists else np.zeros(0, np.uint32)
    order = np.zeros(len(votes) + 8, dtype=np.uint16); ok = np.zeros(len(vote_lists) + 4, dtype=np.int32)
    _check(load_library().bmbs_debug_sort_order(dev, votes.ctypes.data, offs.ctypes.data, len(vote_lists), order.ctypes.data, ok.ctypes.data))
    return [order[offs[i]:offs[i + 1]] for i in range(len(vote_lists))], ok[: len(vote_lists)]


def default_params(**kw) -> Params:
    p = Params()
    load_library().bmbs_params_default(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def flatten(reads):
    """list of bytes -> (uint8 array, uint64 offsets)"""
    offs = np.zeros(len(reads) + 1, dtype=np.uint64)
    if reads:
        offs[1:] = np.cumsum([len(r) for r in reads], dtype=np.uint64)
    flat = np.frombuffer(b"".join(reads), dtype=np.uint8).copy() if reads else np.zeros(0, dtype=np.uint8)
    return flat, offs


class Index:
    """bmbs_index_load / bmbs_index_free (replaces Start_Load_Index + Load_Index + load_index)."""

    def __init__(self, index_prefix: str, devices=(0,)):
        self._L = load_library()
        self._h = C.c_void_p()
        devs = (C.c_int * len(devices))(*devices)
        _check(self._L.bmbs_index_load(str(index_prefix).encode(), devs, len(devices), C.byref(self._h)))
        self.devices = tuple(devices)

    @property
    def genome_length(self):
        return int(self._L.bmbs_index_genome_length(self._h))

    @property
    def device_bytes(self):
        return int(self._L.bmbs_index_device_bytes(self._h))

    def close(self):
        if self._h:
            self._L.bmbs_index_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # one-call forms -------------------------------------------------------------------------
    def _map(self, fn, reads, n_units, params, dev, cand_cap):
        flat, offs = reads if isinstance(reads, tuple) else flatten(reads)
        n_reads = len(offs) - 1
        params = params or default_params()
        cand_cap = cand_cap or max(1 << 16, 32 * n_reads)
        while True:
            res = np.zeros(n_reads, dtype=ReadResult)
            cand = np.zeros(cand_cap, dtype=Cand)
            used = C.c_size_t(0)
            rc = fn(self._h, dev, flat.ctypes.data, offs.ctypes.data, n_units, C.byref(params), res.ctypes.data, cand.ctypes.data, cand_cap, C.byref(used))
            if rc == -4 and used.value > cand_cap:
                cand_cap = int(used.value * 1.25) + 1024
                continue
            _check(rc)
            return res, cand[: used.value]

    def map_batch_se(self, reads, params=None, dev=0, cand_cap=None):
        n = (len(reads[1]) - 1) if isinstance(reads, tuple) else len(reads)
        return self._map(self._L.bmbs_map_batch_se, reads, n, params, dev, cand_cap)

    def map_batch_pe(self, mates, params=None, dev=0, cand_cap=None):
        """mates: [mate1_0, mate2_0(revcomp), mate1_1, ...]"""
        n = (len(mates[1]) - 1) if isinstance(mates, tuple) else len(mates)
        return self._map(self._L.bmbs_map_batch_pe, mates, n // 2, params, dev, cand_cap)

    def verify(self, reads, read_idx, sites, e_rate=0.08, dev=0):
        flat, offs = reads if isinstance(reads, tuple) else flatten(reads)
        read_idx = np.ascontiguousarray(read_idx, dtype=np.uint32)
        sites = np.ascontiguousarray(sites, dtype=np.uint64)
        n = len(sites)
        end = np.zeros(n, dtype=np.int32); err = np.zeros(n, dtype=np.uint32)
        _check(self._L.bmbs_verify(self._h, dev, flat.ctypes.data, offs.ctypes.data, len(offs) - 1, read_idx.ctypes.data, sites.ctypes.data, n,
                                   e_rate, end.ctypes.data, err.ctypes.data))
        return end, err


class Batch:
    """Staged form: upload / run / download with device timings and work counters."""

    def __init__(self, index: Index, dev, max_reads, max_bases, cand_cap):
        self._L = load_library(); self._h = C.c_void_p(); self.index = index
        _check(self._L.bmbs_batch_create(index._h, dev, max_reads, max_bases, cand_cap, C.byref(self._h)))
        self.cand_cap = cand_cap; self.n_reads = 0

    def upload(self, flat, offs, pe=False):
        self.n_reads = len(offs) - 1
        _check(self._L.bmbs_batch_upload(self._h, flat.ctypes.data, offs.ctypes.data, self.n_reads, 1 if pe else 0))

    def run(self, params):
        _check(self._L.bmbs_batch_run(self._h, C.byref(params)))

    def sync(self):
        _check(self._L.bmbs_batch_sync(self._h))

    def download(self, res=None, cand=None):
        res = np.zeros(self.n_reads, dtype=ReadResult) if res is None else res
        cand = np.zeros(self.cand_cap, dtype=Cand) if cand is None else cand
        used = C.c_size_t(0)
        _check(self._L.bmbs_batch_download(self._h, res.ctypes.data, cand.ctypes.data, len(cand), C.byref(used)))
        return res, cand, used.value

    def output_sizes(self):
        """waits for the batch -> (entries of cand[], mismatch positions) the download call will write"""
        nc, nm = C.c_size_t(0), C.c_size_t(0)
        _check(self._L.bmbs_batch_output_sizes(self._h, C.byref(nc), C.byref(nm)))
        return nc.value, nm.value

    def finish(self):
        """the finished records on the device, behind run() on the batch's stream: for single-end reads the reduction over the
        window list, for pairs the hit compaction, distance filter and pair pick; then the ungapped CIGAR check and coordinates"""
        _check(self._L.bmbs_batch_finish(self._h))

    def download_final(self, fin=None, mism=None, cand=None):
        """-> (Final[n_reads], mismatch positions u16[], handed-back windows Cand[])"""
        fin = np.zeros(self.n_reads, dtype=Final) if fin is None else fin
        mism = np.zeros(32 * self.n_reads + 64, dtype=np.uint16) if mism is None else mism
        cand = np.zeros(1 << 16, dtype=Cand) if cand is None else cand
        while True:
            nm, nc = C.c_size_t(0), C.c_size_t(0)
            rc = self._L.bmbs_batch_download_final(self._h, fin.ctypes.data, mism.ctypes.data, len(mism), C.byref(nm), cand.ctypes.data, len(cand), C.byref(nc))
            if rc == -4 and (nm.value > len(mism) or nc.value > len(cand)):
                mism = np.zeros(max(len(mism), nm.value + 64), dtype=np.uint16); cand = np.zeros(max(len(cand), nc.value + 64), dtype=Cand)
                continue
            _check(rc)
            return fin, mism[: nm.value], cand[: nc.value]

    def finish_counters(self):
        c = (C.c_uint64 * 8)()
        _check(self._L.bmbs_batch_finish_counters(self._h, c))
        return dict(zip(["mismatch_positions", "handed_back_windows", "reads_sort_replayed", "reads_handed_back", "reads_dp", "order_decides_window", "order_decides_sbd", "device_us"], [int(x) for x in c]))

    def verify(self, read_idx, sites, e_rate=0.08):
        """kernel 3 alone over the uploaded reads (async); results via download_verify"""
        self._vn = len(sites)
        _check(self._L.bmbs_batch_verify(self._h, read_idx.ctypes.data, sites.ctypes.data, self._vn, e_rate))

    def download_verify(self, end=None, err=None):
        end = np.zeros(self._vn, dtype=np.int32) if end is None else end
        err = np.zeros(self._vn, dtype=np.uint32) if err is None else err
        _check(self._L.bmbs_batch_download_verify(self._h, end.ctypes.data, err.ctypes.data, self._vn))
        return end, err

    def timings(self):
        ms = (C.c_float * 8)()
        _check(self._L.bmbs_batch_timings(self._h, ms))
        return dict(zip(["total", "pack", "seed", "locate", "votes", "pair_filter", "verify", "sensitive"], list(ms)[:8]))

    def counters(self):
        c = (C.c_uint64 * 8)()
        _check(self._L.bmbs_batch_counters(self._h, c))
        return dict(zip(["hash_queries", "occ_lookups", "located_rows", "locate_lf_steps", "verified", "cells", "candidates", "window_bytes"], [int(x) for x in c]))

    def launches(self):
        return int(self._L.bmbs_batch_launches(self._h))

    def grid(self):
        """test entry: [SMs the grids are sized for, seed_reads blocks of the last run, verify_windows blocks of its last
        launch, their block size]"""
        g = (C.c_uint32 * 4)()
        _check(self._L.bmbs_batch_grid(self._h, g))
        return [int(x) for x in g]

    def close(self):
        if self._h:
            self._L.bmbs_batch_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Refiner:
    """bmbs_refiner: the banded affine-gap DP with traceback of the CIGAR refinement (SURVEY.md 8f-1) on the device"""

    def __init__(self, index: Index, dev=0):
        self.L = load_library(); self.h = C.c_void_p()
        _check(self.L.bmbs_refiner_create(index._h, dev, C.byref(self.h)))

    def refine(self, seqs: bytes, quals: bytes, items: np.ndarray, scoring=(6, 2, 1, 5, 3, 33)):
        """items: RefineItem array; returns (RefineResult array, ops u32 array)"""
        assert items.dtype == RefineItem and len(seqs) == len(quals)
        n = len(items)
        res = np.zeros(n, dtype=RefineResult)
        cap = int((2 * items["len"].astype(np.int64) + 2 * items["k"].astype(np.int64) + 2).sum()) + 1
        ops = np.zeros(cap, dtype=np.uint32); used = C.c_size_t(0)
        sc = Scoring(*scoring)
        items = np.ascontiguousarray(items)
        _check(self.L.bmbs_refine(self.h, seqs, quals, len(seqs), items.ctypes.data, n, C.byref(sc), res.ctypes.data, ops.ctypes.data, cap, C.byref(used)))
        return res, ops[: used.value]

    def kernel_ms(self) -> float:
        """device time of the last refine() call's kernels"""
        v = C.c_float(0)
        _check(self.L.bmbs_refiner_kernel_ms(self.h, C.byref(v)))
        return v.value

    def close(self):
        if self.h:
            self.L.bmbs_refiner_free(self.h); self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
