"""ctypes binding of libfrogmatch.so (include/frogmatch.h) -- the binding a Python caller such as
the reference's FROG.py / tools/register.py would use instead of spawning `bin/match`.

No CPU fallback: importing works anywhere, but `Matcher()` raises unless the CUDA library loads
and a B200 is present.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfrogmatch.so")

FLAG_SYM = 1
FLAG_FORCE_EXACT = 2
FLAG_DEVICE_ONLY = 4
FLAG_ASYNC = 8
FLAG_MATCH_ALL = 16
FLAG_DISTANCES = 32
FLAG_ROW_TABLE = 64
# one row of a row table (fm_row, include/frogmatch.h)
ROW_DTYPE = np.dtype([("d1", "<f4"), ("d2", "<f4"), ("nearest", "<u4")])

# every symbol include/frogmatch.h declares (checked by tests/test_abi.py)
PUBLIC_SYMBOLS = [
    "fm_device_count", "fm_create", "fm_destroy", "fm_last_error", "fm_set_stream", "fm_synchronize", "fm_upload_image",
    "fm_clear_images", "fm_image_points", "fm_match", "fm_result_wait", "fm_result_num_pairs", "fm_result_total",
    "fm_result_count", "fm_result_pairs", "fm_result_distances", "fm_result_fetch", "fm_result_device_counts",
    "fm_result_device_pairs", "fm_result_free", "fm_get_stats", "fm_result_stats", "fm_version",
    "fm_links_build", "fm_links_total", "fm_links_fetch", "fm_links_offsets", "fm_links_data", "fm_links_device_offsets",
    "fm_links_device_data", "fm_links_build_ms", "fm_links_free",
    "fm_group_create", "fm_group_destroy", "fm_group_last_error", "fm_group_synchronize", "fm_group_clear_images",
    "fm_group_upload_image", "fm_group_match",
    "fm_result_select", "fm_result_rows_device", "fm_result_row_offset", "fm_result_rows_copy",
]
DEBUG_SYMBOLS = ["fm_debug_image", "fm_debug_image_norms", "fm_debug_score_unit", "fm_debug_set_option",
                 "fm_debug_reject_rows", "fm_debug_wide_unit", "fm_debug_compact"]
ERR_INVALID = -1  # FM_ERR_INVALID
ERR_CUDA = -2  # FM_ERR_CUDA
ERR_UNSUPPORTED = -4  # FM_ERR_UNSUPPORTED
# fm_debug_compact paths (include/frogmatch_debug.h)
COMPACT_AUTO, COMPACT_ONE, COMPACT_THREE, COMPACT_LOOKALL = 0, 1, 2, 3


class Stats(C.Structure):
    _fields_ = [
        ("descriptor_pairs", C.c_uint64), ("scored_pairs", C.c_uint64), ("rows", C.c_uint64),
        ("rows_exact", C.c_uint64), ("candidates", C.c_uint64), ("kernel_launches", C.c_uint64),
        ("score_launches", C.c_uint64), ("ms_total", C.c_float), ("ms_score", C.c_float),
        ("ms_rescore", C.c_float), ("ms_exact", C.c_float), ("ms_compact", C.c_float), ("ms_prep", C.c_float),
        ("rows_rejected_early", C.c_uint64), ("two_phase_batches", C.c_uint64),
    ]

    def as_dict(self) -> dict:
        return {n: getattr(self, n) for n, _ in self._fields_}


class FrogMatchError(RuntimeError):
    pass


_lib = None


def load():
    """Load libfrogmatch.so; fails loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FrogMatchError(f"{LIB_PATH} is missing: build it with `python -m frog_b200.build` "
                             "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, u32p, f32p = C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_float)
    L.fm_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.fm_destroy.argtypes = [vp]
    L.fm_destroy.restype = None
    L.fm_last_error.argtypes = [vp]
    L.fm_last_error.restype = C.c_char_p
    L.fm_set_stream.argtypes = [vp, vp]
    L.fm_synchronize.argtypes = [vp]
    L.fm_upload_image.argtypes = [vp, C.c_uint32, vp, vp, vp, C.c_uint32, C.c_uint32]
    L.fm_clear_images.argtypes = [vp]
    L.fm_image_points.argtypes = [vp, C.c_uint32, u32p]
    L.fm_match.argtypes = [vp, vp, vp, C.c_size_t, C.c_float, C.c_float, C.c_uint32, C.POINTER(vp)]
    L.fm_result_num_pairs.argtypes = [vp]
    L.fm_result_num_pairs.restype = C.c_size_t
    L.fm_result_total.argtypes = [vp]
    L.fm_result_total.restype = C.c_uint64
    L.fm_result_count.argtypes = [vp, C.c_size_t]
    L.fm_result_count.restype = C.c_uint32
    L.fm_result_pairs.argtypes = [vp, C.c_size_t]
    L.fm_result_pairs.restype = u32p
    L.fm_result_distances.argtypes = [vp, C.c_size_t]
    L.fm_result_distances.restype = f32p
    L.fm_result_fetch.argtypes = [vp]
    L.fm_result_wait.argtypes = [vp]
    L.fm_result_stats.argtypes = [vp, C.POINTER(Stats)]
    L.fm_result_device_counts.argtypes = [vp]
    L.fm_result_device_counts.restype = vp
    L.fm_result_device_pairs.argtypes = [vp]
    L.fm_result_device_pairs.restype = vp
    L.fm_result_free.argtypes = [vp]
    L.fm_result_free.restype = None
    L.fm_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.fm_version.restype = C.c_char_p
    L.fm_debug_image.argtypes = [vp, C.c_uint32, u32p, u32p, f32p, u32p, f32p, vp, vp, vp, vp]
    L.fm_debug_image_norms.argtypes = [vp, C.c_uint32, f32p, f32p, f32p]
    L.fm_debug_score_unit.argtypes = [vp, C.c_uint32, C.c_uint32, C.c_uint32, vp, C.c_uint32, vp, vp, vp]
    L.fm_debug_set_option.argtypes = [C.c_char_p, C.c_int]
    L.fm_debug_reject_rows.argtypes = [vp, C.c_uint32, C.c_uint32, vp, vp, vp, vp, u32p]
    L.fm_debug_wide_unit.argtypes = [vp, C.c_uint32, C.c_uint32, C.c_uint32, vp, C.c_uint32, vp, vp, vp, f32p, u32p]
    L.fm_debug_compact.argtypes = [vp, vp, vp, C.c_uint32, vp, C.c_uint32, C.c_int, C.c_uint64, vp, vp, C.c_uint64,
                                   vp, C.c_uint32, C.POINTER(C.c_uint64), vp, u32p]
    L.fm_links_build.argtypes = [vp, vp, vp, vp, C.POINTER(vp)]
    L.fm_links_total.argtypes = [vp]
    L.fm_links_total.restype = C.c_uint64
    L.fm_links_fetch.argtypes = [vp]
    L.fm_links_offsets.argtypes = [vp, C.c_uint32, u32p]
    L.fm_links_offsets.restype = C.POINTER(C.c_uint64)
    L.fm_links_data.argtypes = [vp]
    L.fm_links_data.restype = u32p
    L.fm_links_build_ms.argtypes = [vp]
    L.fm_links_build_ms.restype = C.c_float
    L.fm_links_free.argtypes = [vp]
    L.fm_links_free.restype = None
    L.fm_group_create.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]
    L.fm_group_destroy.argtypes = [vp]
    L.fm_group_destroy.restype = None
    L.fm_group_last_error.argtypes = [vp]
    L.fm_group_last_error.restype = C.c_char_p
    L.fm_group_synchronize.argtypes = [vp]
    L.fm_group_clear_images.argtypes = [vp]
    L.fm_group_upload_image.argtypes = [vp, C.c_uint32, vp, vp, vp, C.c_uint32, C.c_uint32]
    L.fm_group_match.argtypes = [vp, vp, vp, C.c_size_t, C.c_float, C.c_float, C.c_uint32, C.POINTER(vp)]
    L.fm_result_select.argtypes = [vp, C.c_float, C.c_float, C.c_uint32, C.POINTER(vp)]
    L.fm_result_rows_device.argtypes = [vp]
    L.fm_result_rows_device.restype = vp
    L.fm_result_row_offset.argtypes = [vp, C.c_size_t]
    L.fm_result_row_offset.restype = C.c_uint64
    L.fm_result_rows_copy.argtypes = [vp, C.c_size_t, vp]
    _lib = L
    return L


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _flags(sym, force_exact, device_only, asynchronous, match_all, distances, row_table=False) -> int:
    return (FLAG_SYM if sym else 0) | (FLAG_FORCE_EXACT if force_exact else 0) | \
        (FLAG_DEVICE_ONLY if device_only else 0) | (FLAG_ASYNC if asynchronous else 0) | \
        (FLAG_MATCH_ALL if match_all else 0) | (FLAG_DISTANCES if distances else 0) | \
        (FLAG_ROW_TABLE if row_table else 0)


class Result:
    """Owns one fm_result (of a Matcher or a Group): per-pair match lists, on the host and/or on the device."""

    def __init__(self, matcher, handle, pending: bool = False):
        self._m, self._h = matcher, handle
        matcher._live.add(self)
        self.n_pairs = matcher._L.fm_result_num_pairs(handle)
        self.total, self.counts = None, None
        if not pending:
            self._read_counts()

    def _read_counts(self) -> None:
        L = self._m._L
        self.total = L.fm_result_total(self._h)
        self.counts = np.array([L.fm_result_count(self._h, p) for p in range(self.n_pairs)], np.uint32)

    def wait(self) -> "Result":
        """Complete an asynchronous (FM_FLAG_ASYNC) result: counts, totals and -- unless device-only -- host lists."""
        self._m._check(self._m._L.fm_result_wait(self._h))
        if self.counts is None:
            self._read_counts()
        return self

    def fetch(self) -> None:
        self._m._check(self._m._L.fm_result_fetch(self._h))
        if self.counts is None:
            self._read_counts()

    def stats(self) -> dict:
        """fm_stats of the call that produced this result (waits for it)."""
        s = Stats()
        self._m._check(self._m._L.fm_result_stats(self._h, C.byref(s)))
        if self.counts is None:
            self._read_counts()
        return s.as_dict()

    def pairs(self, p: int) -> np.ndarray:
        """[count,2] uint32 (first_idx, second_idx) of pair p -- the bytes match.cpp:738 writes."""
        if self.counts is None:
            self.wait()
        n = int(self.counts[p])
        if n == 0:
            return np.zeros((0, 2), np.uint32)
        ptr = self._m._L.fm_result_pairs(self._h, p)
        if not ptr:
            raise FrogMatchError("result not fetched to the host yet (FM_FLAG_DEVICE_ONLY)")
        return np.ctypeslib.as_array(ptr, shape=(n, 2)).copy()

    def distances(self, p: int) -> np.ndarray:
        """[count] float32 squared distances of pair p's matches (FM_FLAG_DISTANCES), in list order."""
        if self.counts is None:
            self.wait()
        n = int(self.counts[p])
        if n == 0:
            return np.zeros(0, np.float32)
        ptr = self._m._L.fm_result_distances(self._h, p)
        if not ptr:
            raise FrogMatchError("no distances: pass distances=True to match() (and fetch device-only results)")
        return np.ctypeslib.as_array(ptr, shape=(n,)).copy()

    def links(self, pair_first, pair_second, block_order=None):
        """The adjacency bin/frog builds from pairs.bin (ImageGroup::readPairs), built on the device from this result's
        lists.  Returns (offsets, links, build_ms): offsets[img] = n_points + 1 uint64 offsets into `links`
        ([total, 2] uint32: (image, point)), every point's links in the reference's push_back order."""
        if self.counts is None:
            self.wait()
        L = self._m._L
        pf = np.ascontiguousarray(pair_first, np.uint32)
        ps = np.ascontiguousarray(pair_second, np.uint32)
        bo = None if block_order is None else np.ascontiguousarray(block_order, np.uint32)
        h = C.c_void_p()
        self._m._check(L.fm_links_build(self._h, _ptr(pf), _ptr(ps), None if bo is None else _ptr(bo), C.byref(h)))
        try:
            self._m._check(L.fm_links_fetch(h))
            total = L.fm_links_total(h)
            data = np.ctypeslib.as_array(L.fm_links_data(h), shape=(max(total, 1), 2))[:total].copy()
            offsets = {}
            for img in sorted(set(pf.tolist()) | set(ps.tolist())):
                n = C.c_uint32()
                ptr = L.fm_links_offsets(h, img, C.byref(n))
                offsets[img] = np.ctypeslib.as_array(ptr, shape=(n.value + 1,)).copy()
            return offsets, data, float(L.fm_links_build_ms(h))
        finally:
            L.fm_links_free(h)

    def all_pairs(self):
        return [self.pairs(p) for p in range(self.n_pairs)]

    def select(self, dist: float, ratio: float, distances: bool = False, device_only: bool = False,
               asynchronous: bool = False) -> "Result":
        """The lists match() would return at (dist, ratio) on the same pairs, from this result's row table
        (match(..., row_table=True)) without scoring again: a new, independent Result."""
        flags = _flags(False, False, device_only, asynchronous, False, distances)
        h = C.c_void_p()
        self._m._check(self._m._L.fm_result_select(self._h, dist, ratio, flags, C.byref(h)))
        return Result(self._m, h, pending=asynchronous)

    def row_offset(self, p: int) -> int:
        """First row of pair p in the row table (p == n_pairs: the number of rows)."""
        return int(self._m._L.fm_result_row_offset(self._h, p))

    def rows(self, p: int) -> np.ndarray:
        """Pair p's rows of the row table: a structured array (d1, d2, nearest) -- N_second rows in keypoint order,
        then, with sym, the reverse direction's N_first rows."""
        n = self.row_offset(p + 1) - self.row_offset(p)
        out = np.zeros(max(n, 0), ROW_DTYPE)
        self._m._check(self._m._L.fm_result_rows_copy(self._h, p, _ptr(out)))
        return out

    def rows_device_pointer(self) -> int:
        """Raw device address of the whole row table (None for a group of several devices or without a table)."""
        return self._m._L.fm_result_rows_device(self._h)

    def device_pointers(self):
        """(counts_ptr, pairs_ptr) raw device addresses, for GPU-to-GPU gathers."""
        L = self._m._L
        return L.fm_result_device_counts(self._h), L.fm_result_device_pairs(self._h)

    def free(self) -> None:
        if self._h:
            if self._m._h:  # a closed Matcher has already released everything its results own (fm_destroy)
                self._m._L.fm_result_free(self._h)
            self._m._live.discard(self)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Matcher:
    """One libfrogmatch context = one GPU.  Mirrors the reference's flow: load keypoints
    (match.cpp:508-570) -> ComputeMatches per image pair (:638-652)."""

    def __init__(self, device: int = 0):
        self._L = load()
        h = C.c_void_p()
        rc = self._L.fm_create(device, C.byref(h))
        if rc != 0:
            raise FrogMatchError(f"fm_create failed ({rc}): {self._L.fm_last_error(None).decode()}")
        self._h = h
        self._keep = []
        self._live = set()  # results that still own native buffers: freed before the context goes away

    def _check(self, rc: int) -> None:
        if rc != 0:
            raise FrogMatchError(f"libfrogmatch error {rc}: {self._L.fm_last_error(self._h).decode()}")

    def close(self) -> None:
        if self._h:
            for r in list(self._live):
                r.free()
            self._L.fm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream: int) -> None:
        self._check(self._L.fm_set_stream(self._h, C.c_void_p(cuda_stream)))

    def synchronize(self) -> None:
        self._check(self._L.fm_synchronize(self._h))

    def clear(self) -> None:
        self._check(self._L.fm_clear_images(self._h))

    def upload(self, img: int, desc, scale, lap) -> None:
        desc = np.ascontiguousarray(desc, np.float32)
        scale = np.ascontiguousarray(scale, np.float32)
        lap = np.ascontiguousarray(lap, np.float32)
        n, d = desc.shape
        self._check(self._L.fm_upload_image(self._h, img, _ptr(desc), _ptr(scale), _ptr(lap), n, d))
        self.synchronize()  # the numpy temporaries above may be freed after return

    def upload_raw(self, img: int, desc_ptr: int, scale_ptr: int, lap_ptr: int, n: int, d: int) -> None:
        """Asynchronous upload from caller-owned (ideally pinned) host memory."""
        self._check(self._L.fm_upload_image(self._h, img, C.c_void_p(desc_ptr), C.c_void_p(scale_ptr),
                                            C.c_void_p(lap_ptr), n, d))

    def match(self, pair_first, pair_second, dist: float = 0.22, ratio: float = 1.0, sym: bool = False,
              force_exact: bool = False, device_only: bool = False, asynchronous: bool = False,
              match_all: bool = False, distances: bool = False, row_table: bool = False) -> Result:
        pf = np.ascontiguousarray(pair_first, np.uint32)
        ps = np.ascontiguousarray(pair_second, np.uint32)
        flags = _flags(sym, force_exact, device_only, asynchronous, match_all, distances, row_table)
        h = C.c_void_p()
        self._check(self._L.fm_match(self._h, _ptr(pf), _ptr(ps), pf.shape[0], dist, ratio, flags, C.byref(h)))
        return Result(self, h, pending=asynchronous)

    def stats(self) -> dict:
        s = Stats()
        self._check(self._L.fm_get_stats(self._h, C.byref(s)))
        return s.as_dict()

    # ---- test hooks (include/frogmatch_debug.h) --------------------------------------------------
    def debug_image(self, img: int, n: int, operands: bool = True) -> dict:
        flags, ncls, mx = C.c_uint32(), C.c_uint32(), C.c_float()
        class_lap = (C.c_float * 8)()
        class_begin = (C.c_uint32 * 9)()
        perm = np.zeros(max(n, 1), np.uint32)
        ss = np.zeros(max(n, 1), np.float32)
        n_pad = (n + 255) & ~255
        rowop = np.zeros((n_pad, 64), np.float16) if operands else None
        colop = np.zeros((n_pad, 64), np.float16) if operands else None
        self._check(self._L.fm_debug_image(self._h, img, C.byref(flags), C.byref(ncls), class_lap, class_begin,
                                           C.byref(mx), _ptr(perm), _ptr(ss),
                                           _ptr(rowop) if operands else None, _ptr(colop) if operands else None))
        return dict(flags=flags.value, n_classes=ncls.value, max_norm2=mx.value,
                    class_lap=np.array(class_lap[:ncls.value], np.float32),
                    class_begin=np.array(class_begin[:ncls.value + 1], np.uint32),
                    perm=perm[:n], scale_sorted=ss[:n], rowop=rowop, colop=colop)

    def debug_image_norms(self, img: int) -> dict:
        mn, mx, md = C.c_float(), C.c_float(), C.c_float()
        self._check(self._L.fm_debug_image_norms(self._h, img, C.byref(mn), C.byref(mx), C.byref(md)))
        return dict(min_norm2=mn.value, max_norm2=mx.value, max_delta2=md.value)

    def debug_score_unit(self, first_img: int, second_img: int, row_block: int, n_first: int, n_second: int) -> dict:
        ld = (n_first + 255) & ~255
        t = np.zeros((256, ld), np.float32)
        nr = min(256, n_second - row_block * 256)
        bands = np.zeros((nr, 2), np.uint32)
        ct = np.zeros((nr, 8), np.float32)
        cc = np.zeros((nr, 8), np.uint32)
        self._check(self._L.fm_debug_score_unit(self._h, first_img, second_img, row_block, _ptr(t), ld,
                                                _ptr(bands), _ptr(ct), _ptr(cc)))
        return dict(t=t, bands=bands, cand_t=ct, cand_col=cc)

    def debug_wide_unit(self, first_img: int, second_img: int, row_block: int, n_first: int, n_second: int) -> dict:
        """One 128-row unit of the wide scoring kernel (d != 48) in dump mode: t [128, n_pad(first)] float32 scores of
        the columns its MMAs computed (NaN elsewhere), bands [rows, 2], the 8-entry candidate lists cand_t / cand_col
        [rows, 8], the task's eps and K_pad."""
        ld = (n_first + 255) & ~255
        t = np.zeros((128, max(ld, 1)), np.float32)
        nr = min(128, n_second - row_block * 128)
        bands = np.zeros((nr, 2), np.uint32)
        ct = np.zeros((nr, 8), np.float32)
        cc = np.zeros((nr, 8), np.uint32)
        eps, kpad = C.c_float(), C.c_uint32()
        self._check(self._L.fm_debug_wide_unit(self._h, first_img, second_img, row_block, _ptr(t), ld, _ptr(bands),
                                               _ptr(ct), _ptr(cc), C.byref(eps), C.byref(kpad)))
        return dict(t=t, bands=bands, cand_t=ct, cand_col=cc, eps=eps.value, k_pad=kpad.value)

    def debug_reject_rows(self, task: int, n_rows: int):
        """What the reject pass computed for task `task` (n_rows sorted rows) of the last match(), run with the
        "reject_dump" option set: args [n,4] float32 (a1, a2, |a|^2, eps; NaN rows have no band), rowstat [n] uint8,
        bands [n,2] uint32 and the ascending survivor list.  None (FM_ERR_INVALID) if the task did not go through
        the reject pass, or n_rows is not its row count."""
        args = np.zeros((max(n_rows, 1), 4), np.float32)
        stat = np.zeros(max(n_rows, 1), np.uint8)
        bands = np.zeros((max(n_rows, 1), 2), np.uint32)
        surv = np.zeros(max(n_rows, 1), np.uint32)
        ns = C.c_uint32()
        rc = self._L.fm_debug_reject_rows(self._h, task, n_rows, _ptr(args), _ptr(stat), _ptr(bands), _ptr(surv), C.byref(ns))
        if rc == ERR_INVALID:
            return None
        self._check(rc)
        return dict(args=args[:n_rows], rowstat=stat[:n_rows], bands=bands[:n_rows], survivors=surv[:ns.value])

    def debug_compact(self, rowres, chunks, path: int, base: int, out_pairs, pair_counts, rowdist=None, out_dist=None,
                      epoch=None, status: bool = False) -> dict:
        """One batch's compaction through the library's launch routine on this context (fm_debug_compact).
        rowres [n] uint32 (0xFFFFFFFF = no match), chunks [k, 4] uint32 records, path COMPACT_*, out_pairs [slots, 2]
        uint32 and pair_counts uint32 are in/out (updated in place), as is out_dist [slots] float32 with rowdist.
        epoch: set the context's launch epoch counter first.  Returns dict(total, epoch, status) -- status the 1536
        look-back words when asked for.  FrogMatchError when the library refuses the arguments."""
        rowres = np.ascontiguousarray(rowres, np.uint32)
        chunks = np.ascontiguousarray(chunks, np.uint32).reshape(-1, 4)
        assert out_pairs.dtype == np.uint32 and out_pairs.flags.c_contiguous and out_pairs.ndim == 2
        assert pair_counts.dtype == np.uint32 and pair_counts.flags.c_contiguous
        rd = None if rowdist is None else np.ascontiguousarray(rowdist, np.float32)
        if out_dist is not None:
            assert out_dist.dtype == np.float32 and out_dist.flags.c_contiguous
        total = C.c_uint64()
        ep = C.c_uint32(0 if epoch is None else epoch)
        st = np.zeros(1536, np.uint64) if status else None
        self._check(self._L.fm_debug_compact(
            self._h, _ptr(rowres), None if rd is None else _ptr(rd), rowres.shape[0], _ptr(chunks), chunks.shape[0], path,
            base, _ptr(out_pairs), None if out_dist is None else _ptr(out_dist), out_pairs.shape[0], _ptr(pair_counts),
            pair_counts.shape[0], C.byref(total), None if st is None else _ptr(st), C.byref(ep) if epoch is not None else None))
        return dict(total=total.value, epoch=ep.value if epoch is not None else None, status=st)


class Group:
    """One libfrogmatch group (fm_group_*): a context per device, used as one.  devices[0] is the lead: match() splits
    the pairs over the devices and returns one Result whose lists are gathered on the lead, in submission order."""

    def __init__(self, devices):
        self._L = load()
        self.devices = [int(d) for d in devices]
        devs = (C.c_int * len(self.devices))(*self.devices)
        h = C.c_void_p()
        rc = self._L.fm_group_create(devs, len(self.devices), C.byref(h))
        if rc != 0:
            self._h = None
            raise FrogMatchError(f"fm_group_create failed ({rc}): {self._L.fm_group_last_error(None).decode()}")
        self._h = h
        self._live = set()  # results that still own native buffers: freed before the group goes away

    def _check(self, rc: int) -> None:
        if rc != 0:
            raise FrogMatchError(f"libfrogmatch error {rc}: {self._L.fm_group_last_error(self._h).decode()}")

    def close(self) -> None:
        if self._h:
            for r in list(self._live):
                r.free()
            self._L.fm_group_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def synchronize(self) -> None:
        self._check(self._L.fm_group_synchronize(self._h))

    def clear(self) -> None:
        self._check(self._L.fm_group_clear_images(self._h))

    def upload(self, img: int, desc, scale, lap) -> None:
        desc = np.ascontiguousarray(desc, np.float32)
        scale = np.ascontiguousarray(scale, np.float32)
        lap = np.ascontiguousarray(lap, np.float32)
        n, d = desc.shape
        self._check(self._L.fm_group_upload_image(self._h, img, _ptr(desc), _ptr(scale), _ptr(lap), n, d))
        self.synchronize()  # the numpy temporaries above may be freed after return

    def upload_raw(self, img: int, desc_ptr: int, scale_ptr: int, lap_ptr: int, n: int, d: int) -> None:
        """Asynchronous upload from caller-owned pinned host memory or device memory of any member's GPU."""
        self._check(self._L.fm_group_upload_image(self._h, img, C.c_void_p(desc_ptr), C.c_void_p(scale_ptr),
                                                  C.c_void_p(lap_ptr), n, d))

    def match(self, pair_first, pair_second, dist: float = 0.22, ratio: float = 1.0, sym: bool = False,
              force_exact: bool = False, device_only: bool = False, asynchronous: bool = False,
              match_all: bool = False, distances: bool = False, row_table: bool = False) -> Result:
        pf = np.ascontiguousarray(pair_first, np.uint32)
        ps = np.ascontiguousarray(pair_second, np.uint32)
        flags = _flags(sym, force_exact, device_only, asynchronous, match_all, distances, row_table)
        h = C.c_void_p()
        self._check(self._L.fm_group_match(self._h, _ptr(pf), _ptr(ps), pf.shape[0], dist, ratio, flags, C.byref(h)))
        return Result(self, h, pending=asynchronous)


def debug_set_option(name: str, value: int) -> None:
    """Experiment switch of the scoring kernel (include/frogmatch_debug.h); not part of the boundary."""
    if load().fm_debug_set_option(name.encode(), int(value)) != 0:
        raise FrogMatchError(f"unknown debug option {name!r}")


def version() -> str:
    return load().fm_version().decode()
