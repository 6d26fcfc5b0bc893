"""Shared test helpers: a Python restatement of bin/match's driver logic (argv quirks, list file,
pair schedule -- match.cpp:340-499, 617-628) on top of the real host C++ (frog_b200.hostio), so a
whole pairs.bin can be produced with any matching engine (oracle port on CPU, libfrogmatch on GPU)
and compared byte-for-byte with the reference binary's output."""
from __future__ import annotations

import os

import numpy as np

from frog_b200 import hostio


def parse_args(argv):
    """match.cpp:365-431: key/value pairs, every key advances by 2 except -sym (1)."""
    o = dict(N=1000000, sp=0.0, np=1000000, dist=np.float32(0.22), ratio=np.float32(1.0), zmin=np.float32(-1e20),
             zmax=np.float32(1e20), sym=False, target=-1, out=None, all=False)
    k = 0
    while k < len(argv):
        key = argv[k]
        val = argv[k + 1] if k + 1 < len(argv) else None
        if val is not None:
            if key == "-n": o["N"] = int(val)
            if key == "-sp": o["sp"] = float(val)
            if key == "-np": o["np"] = int(val)
            if key == "-d": o["dist"] = np.float32(float(val))
            if key == "-d2": o["ratio"] = np.float32(float(val))
            if key == "-zmin": o["zmin"] = np.float32(float(val))
            if key == "-zmax": o["zmax"] = np.float32(float(val))
            if key == "-o": o["out"] = val
            if key == "-targ": o["target"] = int(val)
        if key == "-all":  # a flag, but the parser still skips the token after it (match.cpp:417-418, 430)
            o["all"] = True
        if key == "-sym":
            o["sym"] = True
            k -= 1
        k += 2
    return o


def load_group(list_path: str, opts: dict):
    """-> filenames, rigids (or None), heads, descs after z-filter and pruning."""
    parent = os.path.dirname(os.path.abspath(list_path))
    filenames, rigids = [], []
    for line in open(list_path).read().splitlines():
        cells = line.split(",")
        name = cells[0]
        filenames.append(name if name.startswith("/") else parent + "/" + name + ".csv")
        rg = [0.0, 0.0, 0.0]
        try:
            for c in range(3):
                rg[c] = float(np.float32(float(cells[1 + c])))
        except (IndexError, ValueError):
            pass
        rigids.append(rg)
    filenames = filenames[:opts["N"]]
    heads, descs = [], []
    for it, f in enumerate(filenames):
        head, desc = hostio.read_keypoints(f)
        head, desc = hostio.filter_prune(head, desc, zT=np.float32(rigids[it][2]), zmin=opts["zmin"], zmax=opts["zmax"],
                                         sp=opts["sp"], np_keep=opts["np"])
        heads.append(head)
        descs.append(desc)
    return filenames, rigids, heads, descs


def pair_schedule(nb: int, target: int):
    """match.cpp:617-628."""
    idx = []
    for i in range(nb - 1):
        if target >= 0:
            if i != target:
                idx.append((i, target))
        else:
            idx += [(i, j) for j in range(i + 1, nb)]
    return idx


def images_of(heads, descs):
    return [(d, h[:, 3].copy(), h[:, 4].copy()) for h, d in zip(heads, descs)]


def write_pairs(out_path, filenames, rigids, heads, schedule, lists):
    order = sorted(range(len(schedule)), key=lambda k: schedule[k])
    blocks = [(schedule[k][0], schedule[k][1], lists[k]) for k in order]
    hostio.write_pairs_bin(out_path, filenames, rigids, heads, blocks)


def random_group(kind, n_images, n_points, seed0=0):
    from frog_b200 import synth
    kps = [synth.make(kind, n_points, seed0 + i) for i in range(n_images)]
    return [(k.desc, k.scale, k.lap) for k in kps]


# ---- the gate replayed in the library's sorted order (tensor-core path, fm_score.cuh bands_kernel) ----------------

def sorted_view(img):
    """(scale, laplacian) in the library's sorted order: by the laplacian's top 16 pattern bits, then by scale."""
    _, s, l = img
    l = np.where(l == 0, np.float32(0), l).astype(np.float32)
    order = np.lexsort((s.view(np.uint32), l.view(np.uint32) >> 16))
    return s[order], l[order]


def first_true(pred, lo, hi):
    """Per entry, the first index in [lo, hi) at which the monotone predicate holds (hi if none): binary search."""
    lo, hi = lo.copy(), hi.copy()
    while np.any(lo < hi):
        act = lo < hi
        m = (lo + hi) >> 1
        p = pred(np.where(act, m, 0)) & act
        lo = np.where(act & ~p, m + 1, lo)
        hi = np.where(p, m, hi)
    return lo


def gate_bands(col, row):
    """The reference's gates (match.cpp:270-275) as sorted column intervals [lo, hi) per sorted row."""
    sc, lc = sorted_view(col)
    sr, lr = sorted_view(row)
    lo = np.zeros(sr.shape[0], np.int64)
    hi = np.zeros(sr.shape[0], np.int64)
    for lap in np.unique(lr):
        rows = np.nonzero(lr == lap)[0]
        cls = np.nonzero(lc == lap)[0]
        if cls.size == 0:
            continue
        beg, end = int(cls[0]), int(cls[-1]) + 1
        x = sr[rows]
        b = np.full(rows.size, beg, np.int64)
        e = np.full(rows.size, end, np.int64)
        # float32 quotients compared with 1.3 (the reference's `float / float > 1.3`)
        l0 = first_true(lambda m: ~((x / sc[m]).astype(np.float64) > 1.3), b, e)
        h0 = first_true(lambda m: (sc[m] / x).astype(np.float64) > 1.3, l0, e)
        lo[rows], hi[rows] = l0, np.maximum(h0, l0)
    return lo, hi
