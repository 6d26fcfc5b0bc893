"""GPU: row tables (FM_FLAG_ROW_TABLE) and fm_result_select.  A table-mode call must return the lists a plain call
returns; select at any (dist, ratio) must return byte for byte -- counts, lists, distances, device views, links -- what
a fresh fm_match returns at those thresholds, on every engine and call shape; and every table row must equal a float32
sequential restatement of match.cpp:262-317."""
import ctypes as C

import numpy as np
import pytest
import torch

import test_gpu_wide as W
from frog_b200 import capi, synth
from frog_b200 import dist as fdist

pytestmark = pytest.mark.gpu

# the thresholds FROG's callers use (reference default, run.sh / register.py, FROG.py, desk UI) and more; (1, 1.01)
# accepts rows whose two nearest distances tie
SETTINGS = [(0.22, 1.0), (1.0, 1.0), (1e10, 1.0), (0.5, 0.998), (1.0, 0.8), (0.3, 0.6), (1.0, 1.01)]
FLT_MAX = float(np.finfo(np.float32).max)


@pytest.fixture(scope="module")
def m(built):
    h = capi.Matcher(0)
    yield h
    h.close()


def images_of(kind, n_images, n, seed=0):
    return [(k.desc, k.scale, k.lap) for k in (synth.make(kind, n, seed + i) for i in range(n_images))]


def row_major(n_images):
    return ([i for i in range(n_images) for j in range(i + 1, n_images)],
            [j for i in range(n_images) for j in range(i + 1, n_images)])


def load(h, images):
    h.clear()
    for i, (d, s, l) in enumerate(images):
        h.upload(i, d, s, l)


def snapshot(res, distances, pf=None, ps=None):
    """Everything a caller reads from a result, as bytes (device views before the host copy)."""
    res.wait()
    cptr, pptr = res.device_pointers()
    dev = torch.device("cuda", 0)
    snap = {"total": int(res.total), "counts": res.counts.tobytes(),
            "dev_counts": fdist.as_torch_u32(cptr, res.n_pairs, dev).cpu().numpy().tobytes(),
            "dev_pairs": fdist.as_torch_u32(pptr, 2 * int(res.total), dev).cpu().numpy().tobytes()}
    res.fetch()
    snap["lists"] = b"".join(res.pairs(p).tobytes() for p in range(res.n_pairs))
    if distances:
        snap["dist"] = b"".join(res.distances(p).tobytes() for p in range(res.n_pairs))
    if pf is not None:
        off, data, _ = res.links(pf, ps)
        snap["links"] = b"".join(off[i].tobytes() for i in sorted(off)) + data.tobytes()
    return snap


def assert_snap(got, want, what):
    for k in got:
        assert got[k] == want[k], f"{what}: {k} differs (totals {got['total']} vs {want['total']})"


def fresh(h, pf, ps, thr, rat, two_phase=None, links=False, **kw):
    """A plain fm_match at (thr, rat) with distances, optionally forcing the two-phase choice: (snapshot, stats)."""
    if two_phase is not None:
        capi.debug_set_option("two_phase", two_phase)
    try:
        res = h.match(pf, ps, thr, rat, distances=True, **kw)
    finally:
        capi.debug_set_option("two_phase", -1)
    try:
        return snapshot(res, True, pf if links else None, ps), res.stats()
    finally:
        res.free()


def check_select(h, pf, ps, settings=SETTINGS, own=(1.0, 0.8), two_phase=(None,), links=False, **kw):
    """A table-mode call at `own` against a plain one, then select at each setting against fresh calls (with each
    forced two-phase choice in `two_phase`).  Returns the table-mode result (the caller frees it)."""
    want, _ = fresh(h, pf, ps, *own, **kw)
    capi.debug_set_option("two_phase", 1)  # a table call never scores in two phases, whatever is asked
    try:
        tab = h.match(pf, ps, *own, distances=True, row_table=True, **kw)
    finally:
        capi.debug_set_option("two_phase", -1)
    assert_snap(snapshot(tab, True), want, f"table-mode call at {own}")
    st = tab.stats()
    assert st["rows_rejected_early"] == 0 and st["two_phase_batches"] == 0
    assert tab.row_offset(len(pf)) == st["rows"]
    for thr, rat in settings:
        for tp in two_phase:
            want, _ = fresh(h, pf, ps, thr, rat, two_phase=tp, links=links, **kw)
            sel = tab.select(thr, rat, distances=True)
            assert_snap(snapshot(sel, True, pf if links else None, ps), want, f"select({thr}, {rat}), two_phase={tp}")
            sel.free()
        sel = tab.select(thr, rat)  # without distances
        got = snapshot(sel, False)
        sel.free()
        assert got["lists"] == want["lists"] and got["counts"] == want["counts"]
    return tab


# ---- settings: bank and iid groups, 10 x 20 000 at d = 48 -------------------------------------------------------------
@pytest.mark.parametrize("kind", ["bank", "iid"])
def test_settings(m, kind):
    load(m, images_of(kind, 10, 20000))
    pf, ps = row_major(10)
    tab = check_select(m, pf, ps, two_phase=(None, 0, 1), links=True)
    tab.free()


# ---- engines ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", [24, 192, 1000])
def test_wide_path(m, d):
    load(m, W.bank_group(d, 4, 1500, seed=d))
    pf, ps = row_major(4)
    _, st = fresh(m, pf, ps, 1.0, 0.8)
    assert st["score_launches"] >= 1 and st["rows_exact"] < st["rows"]
    check_select(m, pf, ps).free()


def test_exact_engine_forced(m):
    load(m, images_of("bank", 4, 2000, seed=3))
    pf, ps = row_major(4)
    check_select(m, pf, ps, force_exact=True).free()
    load(m, W.bank_group(192, 3, 800, seed=4))
    check_select(m, [0, 0, 1], [1, 2, 2], force_exact=True).free()


@pytest.mark.parametrize("d", [48, 192])
def test_exact_engine_flagged_images(m, d):
    """NaN, |desc|^2 > 16 and 11 laplacian classes route whole tasks to the exact kernels; the others stay fast."""
    images = W.bank_group(d, 5, 700, seed=6 + d)
    nan = list(images[2]); nan[0] = nan[0].copy(); nan[0][7, 5] = np.nan; images[2] = tuple(nan)
    big = list(images[3]); big[0] = big[0] * np.float32(4.5); images[3] = tuple(big)
    many = list(images[4]); many[2] = (np.arange(700) % 11).astype(np.float32); images[4] = tuple(many)
    load(m, images)
    pf, ps = [0, 0, 0, 0, 1, 2, 3, 4], [1, 2, 3, 4, 0, 1, 1, 1]
    _, st = fresh(m, pf, ps, 1.0, 0.9)
    assert 0 < st["rows_exact"] < st["rows"] and st["scored_pairs"] > 0
    check_select(m, pf, ps).free()


def test_exact_engine_long_descriptors(m):
    load(m, W.bank_group(24 * 6 ** 3, 3, 200, seed=5))  # d = 5184: no tensor-core path
    check_select(m, [0, 0, 1], [1, 2, 2]).free()


def test_exact_engine_raw_haar(m):
    """surf3d -type 1 descriptors as the producer writes them (raw Haar sums, |desc|^2 far above 16)."""
    group = W.haar_group(2)
    raw = [(desc, pts["scale"].copy(), pts["laplacian"].astype(np.float32)) for pts, desc in group]
    load(m, raw)
    pf, ps = [0, 0, 0, 1, 1, 2], [1, 2, 3, 2, 3, 3]
    _, st = fresh(m, pf, ps, 1e10, 1.0)
    assert st["rows_exact"] == st["rows"]
    check_select(m, pf, ps, settings=SETTINGS + [(1e3, 0.9), (300.0, 1.0)]).free()


def test_overflow_route(m):
    """Duplicated columns overflow the candidate lists: those rows go to the exact row kernels (d = 48 and wide)."""
    for d in (48, 192):
        images = W.bank_group(d, 2, 800, seed=8)
        desc, scale, lap = (x.copy() for x in images[0])
        for src in range(0, 240, 12):
            desc[src + 1: src + 12] = desc[src]
            scale[src + 1: src + 12] = scale[src]
            lap[src + 1: src + 12] = lap[src]
        images[0] = (desc, scale, lap)
        images[1] = (np.concatenate([images[1][0][:700], desc[0:240:12].repeat(5, axis=0)]),
                     np.concatenate([images[1][1][:700], scale[0:240:12].repeat(5)]),
                     np.concatenate([images[1][2][:700], lap[0:240:12].repeat(5)]))
        load(m, images)
        _, st = fresh(m, [0, 1], [1, 0], 1e10, 1.0)
        assert st["rows_exact"] > 0
        check_select(m, [0, 1], [1, 0]).free()


# ---- call shapes -----------------------------------------------------------------------------------------------------
def test_call_shapes(m):
    images = images_of("bank", 6, 3000, seed=20)
    images[4] = (np.zeros((0, 48), np.float32), np.zeros(0, np.float32), np.zeros(0, np.float32))  # no keypoints
    load(m, images)
    pf, ps = row_major(6)
    check_select(m, pf, ps, sym=True, links=True).free()
    # unordered and repeated pairs, and pairs with an empty image
    pf, ps = [3, 0, 1, 0, 4, 2, 3], [0, 3, 0, 3, 1, 4, 0]
    check_select(m, pf, ps, sym=True, links=True).free()
    check_select(m, pf, ps).free()
    # -targ-style blocks: one target against every other image, both ways
    pf, ps = [0, 0, 0, 0, 1, 2, 3, 5], [1, 2, 3, 5, 0, 0, 0, 0]
    check_select(m, pf, ps, links=True).free()
    # no pairs
    tab = m.match([], [], 1.0, 1.0, row_table=True)
    sel = tab.select(0.5, 0.9)
    assert sel.total == 0 and sel.n_pairs == 0 and tab.row_offset(0) == 0
    sel.free()
    tab.free()


def test_async_device_only_and_source_freed(m):
    load(m, images_of("iid", 5, 6000, seed=30))
    pf, ps = row_major(5)
    want = {s: fresh(m, pf, ps, *s)[0] for s in SETTINGS[:4]}
    tab = m.match(pf, ps, 1.0, 0.8, asynchronous=True, device_only=True, row_table=True)
    sels = {s: tab.select(*s, distances=True, device_only=True, asynchronous=True) for s in want}
    tab.free()  # the source may go as soon as the selects are queued
    for s, sel in sels.items():
        sel.wait()
        assert sel.counts is not None
        assert_snap(snapshot(sel, True), want[s], f"async device-only select {s}")
        sel.free()


# ---- table values ----------------------------------------------------------------------------------------------------
def reference_rows(col, row):
    """float32 sequential restatement of match.cpp:262-317 for the rows of image `row` against the columns of `col`:
    (d1, d2, nearest) per row, nearest = 0xFFFFFFFF where d1 stays FLT_MAX."""
    (ad, asc, al), (bd, bsc, bl) = col, row
    d = ad.shape[1]
    acc = np.zeros((len(bd), len(ad)), np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        for k in range(d):  # r = fl(r + fl(fl(a - b)^2)), k ascending (match.cpp:243-251)
            e = (bd[:, k][:, None] - ad[:, k][None, :]).astype(np.float32)
            acc = (acc + e * e).astype(np.float32)
        gate = (bl[:, None] == al[None, :]) & ~((bsc[:, None] / asc[None, :]) > np.float32(1.3)) \
            & ~((asc[None, :] / bsc[:, None]) > np.float32(1.3))
    out = np.zeros(len(bd), capi.ROW_DTYPE)
    for i in range(len(bd)):
        d1 = d2 = FLT_MAX
        match = 0
        for j in np.nonzero(gate[i])[0]:  # match.cpp:303-313: strict '<', columns ascending
            v = float(acc[i, j])
            if v < d1:
                d2, d1, match = d1, v, int(j)
            elif v < d2:
                d2 = v
        out[i] = (d1, d2, match if d1 < FLT_MAX else 0xFFFFFFFF)
    return out


def assert_rows(got, want, what):
    assert len(got) == len(want), what
    for f in ("d1", "d2"):
        bad = np.nonzero(got[f].view(np.uint32) != want[f].view(np.uint32))[0]
        assert len(bad) == 0, f"{what}: {f} differs at rows {bad[:5]}: {got[bad[:5]]} vs {want[bad[:5]]}"
    bad = np.nonzero(got["nearest"] != want["nearest"])[0]
    assert len(bad) == 0, f"{what}: nearest differs at rows {bad[:5]}: {got[bad[:5]]} vs {want[bad[:5]]}"


def table_cases():
    nan = W.bank_group(192, 3, 300, seed=41)
    nan[1] = (nan[1][0].copy(), nan[1][1], nan[1][2])
    nan[1][0][5, 3] = np.nan
    dup = images_of("bank", 3, 400, seed=42)
    dup[0] = (dup[0][0].copy(), dup[0][1].copy(), dup[0][2].copy())
    dup[0][0][10:30] = dup[0][0][10]
    dup[0][1][10:30] = dup[0][1][10]
    dup[0][2][10:30] = dup[0][2][10]
    return {"d48": (images_of("bank", 3, 400, seed=40), {}), "d48_exact": (images_of("iid", 3, 400, seed=43), {"force_exact": True}),
            "d192": (W.bank_group(192, 3, 300, seed=44), {}), "d192_nan": (nan, {}), "d48_ties": (dup, {}),
            "d5184": (W.bank_group(5184, 3, 60, seed=45), {})}


@pytest.mark.parametrize("case", ["d48", "d48_exact", "d192", "d192_nan", "d48_ties", "d5184"])
def test_table_values(m, case):
    images, kw = table_cases()[case]
    load(m, images)
    pf, ps = [0, 0, 1, 2], [1, 2, 2, 0]
    for sym in (False, True):
        tab = m.match(pf, ps, 0.5, 0.9, row_table=True, sym=sym, **kw)
        dev = tab.rows_device_pointer()
        assert dev
        for p, (a, b) in enumerate(zip(pf, ps)):
            want = reference_rows(images[a], images[b])
            if sym:
                want = np.concatenate([want, reference_rows(images[b], images[a])])
            got = tab.rows(p)
            assert tab.row_offset(p + 1) - tab.row_offset(p) == len(want)
            assert_rows(got, want, f"{case} sym={sym} pair {p}")
            # the device view holds the same bytes at the pair's offset
            raw = fdist.as_torch_u32(dev + 12 * tab.row_offset(p), 3 * len(want), torch.device("cuda", 0))
            assert raw.cpu().numpy().tobytes() == got.tobytes()
        tab.free()


# ---- groups ----------------------------------------------------------------------------------------------------------
def group_devices():
    n = torch.cuda.device_count()
    return [[0], [0, 0], [0, 0, 0]] + ([[0, 1]] if n >= 2 else []) + ([list(range(n))] if n > 2 else [])


def make_group(devs):
    repeat = len(set(devs)) < len(devs)
    if repeat:
        capi.debug_set_option("group_repeat", 1)
    try:
        return capi.Group(devs)
    finally:
        if repeat:
            capi.debug_set_option("group_repeat", 0)


@pytest.mark.parametrize("devs", group_devices(), ids=lambda d: "-".join(map(str, d)))
def test_groups(m, devs):
    images = images_of("bank", 8, 5000, seed=50)
    pf, ps = row_major(8)
    pf, ps = pf + [3, 3], ps + [0, 0]  # unordered and repeated
    load(m, images)
    want = {s: fresh(m, pf, ps, *s, sym=True, links=True)[0] for s in SETTINGS}
    ref = m.match(pf, ps, 1.0, 0.8, sym=True, row_table=True)
    want_rows = [ref.rows(p).tobytes() for p in range(len(pf))]
    want_off = [ref.row_offset(p) for p in range(len(pf) + 1)]
    ref.free()
    g = make_group(devs)
    try:
        load(g, images)
        tab = g.match(pf, ps, 1.0, 0.8, sym=True, distances=True, row_table=True)
        assert_snap(snapshot(tab, True), want[(1.0, 0.8)], f"group {devs} table-mode call")
        assert [tab.row_offset(p) for p in range(len(pf) + 1)] == want_off
        assert [tab.rows(p).tobytes() for p in range(len(pf))] == want_rows
        assert bool(tab.rows_device_pointer()) == (len(devs) == 1)
        for s in SETTINGS:
            sel = tab.select(*s, distances=True)
            assert_snap(snapshot(sel, True, pf, ps), want[s], f"group {devs} select {s}")
            assert sel.stats()["rows"] == want_off[-1]
            sel.free()
        sels = [tab.select(*s, distances=True, device_only=True, asynchronous=True) for s in SETTINGS[:3]]
        tab.free()
        for s, sel in zip(SETTINGS[:3], sels):
            sel.wait()
            assert_snap(snapshot(sel, True), want[s], f"group {devs} async select {s}")
            sel.free()
        with pytest.raises(capi.FrogMatchError):
            g.match(pf, ps, 1.0, 1.0, match_all=True, row_table=True)
    finally:
        g.close()


# ---- errors ----------------------------------------------------------------------------------------------------------
def test_errors(m):
    L = capi.load()
    load(m, images_of("bank", 3, 2000, seed=60))
    pf, ps = [0, 1], [1, 2]
    a, b = np.array(pf, np.uint32), np.array(ps, np.uint32)
    h = C.c_void_p()
    assert L.fm_match(m._h, capi._ptr(a), capi._ptr(b), 2, 1.3, 1.0, capi.FLAG_ROW_TABLE | capi.FLAG_MATCH_ALL, C.byref(h)) == capi.ERR_INVALID
    plain = m.match(pf, ps, 1.0, 0.8)
    tab = m.match(pf, ps, 1.0, 0.8, row_table=True)
    out = C.c_void_p()
    assert L.fm_result_select(plain._h, 1.0, 1.0, 0, C.byref(out)) == capi.ERR_INVALID  # no table
    assert plain.row_offset(0) == 2 ** 64 - 1 and not plain.rows_device_pointer()
    for flags in (capi.FLAG_SYM, capi.FLAG_FORCE_EXACT, capi.FLAG_MATCH_ALL, capi.FLAG_ROW_TABLE, 128):
        assert L.fm_result_select(tab._h, 1.0, 1.0, flags, C.byref(out)) == capi.ERR_INVALID
    assert L.fm_result_select(tab._h, float("nan"), 1.0, 0, C.byref(out)) == capi.ERR_INVALID
    assert L.fm_result_select(tab._h, 1.0, float("nan"), 0, C.byref(out)) == capi.ERR_INVALID
    assert L.fm_result_select(tab._h, 1.8e19, 1.0, 0, C.byref(out)) == capi.ERR_UNSUPPORTED
    assert L.fm_result_select(tab._h, float("inf"), 1.0, 0, C.byref(out)) == capi.ERR_UNSUPPORTED
    assert L.fm_result_rows_copy(tab._h, 2, None) == capi.ERR_INVALID
    assert tab.row_offset(3) == 2 ** 64 - 1
    sel = tab.select(1.0, 1.0)
    assert L.fm_result_select(sel._h, 1.0, 1.0, 0, C.byref(out)) == capi.ERR_INVALID  # a selected result has no table
    sel.free()
    plain.free()
    tab.free()


def test_table_that_does_not_fit(m):
    """A table larger than the device: FM_ERR_NOMEM before any work, and the context stays usable."""
    L = capi.load()
    n = 50000
    load(m, images_of("iid", 2, n, seed=70))
    total = torch.cuda.get_device_properties(0).total_memory
    n_pairs = total // (12 * n) + 1
    a = np.zeros(n_pairs, np.uint32)
    b = np.ones(n_pairs, np.uint32)
    h = C.c_void_p()
    assert L.fm_match(m._h, capi._ptr(a), capi._ptr(b), n_pairs, 1.0, 1.0, capi.FLAG_ROW_TABLE, C.byref(h)) == -3
    assert "row table" in L.fm_last_error(m._h).decode()
    want, _ = fresh(m, [0, 1], [1, 0], 1.0, 0.8)
    tab = check_select(m, [0, 1], [1, 0], settings=SETTINGS[:2])
    tab.free()
    assert want["total"] > 0
