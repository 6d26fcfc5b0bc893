"""Reject pass of two-phase scoring (fm_reject.cuh), row by row: every row's g1, g2 and rejection decision against a
float64 replay from the FP16 operands and the FP32 descriptors.

The other reject-pass tests compare match lists only, and a wrong g1 or g2 leaves those unchanged unless it flips the
decision of one of the few rows the reference accepts.  Here the library keeps what its reject pass computed
(fm_debug_reject_rows: the arguments of certified_reject per row, rowstat, the bands and the survivor list) and each
row is checked at four levels:
  1. bands    : the gate replayed in numpy;
  2. tight    : a1 and a2 against the largest and second largest 16-column chunk maximum of the FP16-operand scores
                (what the tensor cores should produce, K = 48 or 64 slots as the pass chose), minus the K = 48 norm
                offsets -- to FP32-accumulation accuracy, far below eps;
  3. certified: a1 >= best exact score - eps, a2 <= second exact chunk maximum + eps, both within eps (+ the K = 48
                norm spread) of the exact values; eps and |a|^2 against float64;
  4. decision : rowstat against certified_reject evaluated in float64 on the dumped arguments, the survivor list
                against rowstat, and no rejected row in the fast oracle's match list.
In the deep call the filler gives every persistent CTA more than six units before the edge tasks come, so those run
after the unit ring, the per-unit buffers and the column ring have wrapped."""
import numpy as np
import pytest

import helpers
from frog_b200 import capi, synth
from oracle import oracle as O

pytestmark = pytest.mark.gpu

CHUNK = 16
UNIT = 256
TIGHT_TOL = 2e-5  # FP32 accumulation in the tensor core plus one ulp of directed rounding (test_gpu_stages: 2e-5)
# sorted column positions where one scale level ends and the next begins (as in test_gpu_reject_rounds)
ROUND_EDGES = (0, 5, 127, 129, 200, 255, 257, 266, 383, 384, 385, 511, 513, 640, 700, 767, 769, 1030)
# levels of 1 column, 2 columns inside one chunk, 12, 2 columns across a chunk boundary, 23
NARROW_EDGES = (0, 1, 3, 15, 17, 40)


@pytest.fixture(scope="module")
def oracle_lib(built):
    return O.FastLib()


@pytest.fixture(scope="module")
def sm_count(built):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _image(kind, n, seed):
    k = synth.make(kind, n, seed)
    return (k.desc, k.scale, k.lap)


def _levels(levels, seed):
    """Descriptors of the iid set, laplacian 1, scale 2^level (jittered by < 1 %): a row's band is its level."""
    d, _, _ = _image("iid", len(levels), seed)
    rng = np.random.default_rng(seed)
    s = (2.0 ** np.asarray(levels, np.float64) * rng.uniform(1.0, 1.01, len(levels))).astype(np.float32)
    return (d, s, np.ones(len(levels), np.float32))


def _level_columns(edges, seed):
    sizes = np.diff(edges)
    return _levels(np.repeat(np.arange(sizes.size), sizes), seed)


def _task_eps(col_desc, row_desc):
    """task_eps (fm_score.cuh) in float64 from the descriptors: Cauchy-Schwarz on the FP16 rounding residuals."""
    def stats(d):
        d = d.astype(np.float64)
        r = d.astype(np.float16).astype(np.float64) - d
        return (d ** 2).sum(1).max(), np.sqrt((r ** 2).sum(1).max())
    na2, da = stats(col_desc)
    nb2, db = stats(row_desc)
    na, nb = np.sqrt(na2), np.sqrt(nb2)
    return 1.01 * (na * db + da * nb + da * db) + 3e-5 * max(1.0, na2, nb2)


def _near_eps(base, row, frac):
    """`base` with two descriptors scaled by 1 + delta and 1 - delta, delta chosen so that the column image's norm
    spread (n_max - n_min) / 2 = 2 delta is `frac` x the eps of a task against `row`."""
    d0, s, l = base
    delta = 0.0
    for _ in range(4):  # eps hardly depends on delta: a few fixed-point steps settle it
        d = d0.copy()
        d[10] *= np.float32(1 + delta)
        d[20] *= np.float32(1 - delta)
        delta = frac * _task_eps(d, row[0]) / 2
    d = d0.copy()
    d[10] *= np.float32(1 + delta)
    d[20] *= np.float32(1 - delta)
    return (d, s, l)


def _ties():
    """Columns: 64 keypoints of one class at increasing scales (sorted order = upload order), with duplicate
    descriptors in one chunk (3 and 5) and in two chunks (20 and 40).  Rows: those descriptors again, so the
    duplicates are the rows' best columns (g1 == g2 for the second), among random rows."""
    d, _, _ = _image("iid", 64, 900)
    d = d.copy()
    d[5], d[40] = d[3], d[20]
    cols = (d, np.linspace(2.0, 2.5, 64).astype(np.float32), np.ones(64, np.float32))
    r, _, _ = _image("iid", 8, 901)
    r = r.copy()
    r[2], r[5] = d[3], d[20]
    rows = (r, np.full(8, 2.2, np.float32), np.ones(8, np.float32))
    return cols, rows


class Tally:
    def __init__(self):
        self.tasks = self.exact = self.rows = self.band_rows = self.tight_a2 = self.boundary = 0
        self.tight = self.cert = 0.0
        self.k48 = self.k64 = 0
        self.K = {}  # (column image, row image) -> K of the task's chains

    def report(self, name):
        print(f"[{name}] tasks {self.tasks} (K=48 {self.k48}, K=64 {self.k64}, exact {self.exact}); rows: bands {self.rows}, "
              f"tight/certified/decision {self.band_rows} (a2 finite {self.tight_a2}); "
              f"max tight dev {self.tight:.2e}, max certified dev / eps {self.cert:.3f}; boundary rows {self.boundary}")


def _decisions(na, a1, a2, eps, thr, ratio):
    """certified_reject (fm_score.cuh) in float64 on the dumped arguments.  Returns the decision with every
    comparison within 1e-6 of its operands' magnitude resolved as false, and as true (nvcc contracts the float32
    expression to FMAs, so a bit-exact replay is not promised): rows where they differ are at the boundary."""
    with np.errstate(invalid="ignore", over="ignore"):
        margin = 2.0 * eps + 1e-5 * (na + 4.0)
        d1 = na - 2.0 * a1 - margin
        d2 = na - 2.0 * a2 + margin
        b1 = np.float64(thr) * thr * 1.00001
        c2 = (a2 > -np.inf) & (d2 > 0) & (ratio < 1e4)
        b2 = np.where(c2, np.float64(ratio) * ratio * np.where(c2, d2, 0.0) * 1.0001, np.inf)
        s1 = 1e-6 * (na + 2.0 * np.abs(a1) + margin + b1)
        s2 = s1 + 1e-6 * np.float64(ratio) * ratio * np.where(c2, na + 2.0 * np.abs(a2) + margin, 0.0)
        lo = (d1 > b1 + s1) | (c2 & (d1 > b2 + s2))
        hi = (d1 > b1 - s1) | (c2 & (d1 > b2 - s2))
    return lo, hi


def _top2(x):
    """Largest and second largest along axis 1 (-inf where there are fewer)."""
    if x.shape[1] == 1:
        return x[:, 0], np.full(x.shape[0], -np.inf)
    p = np.partition(x, x.shape[1] - 2, axis=1)
    return p[:, -1], p[:, -2]


class Replay:
    """Reference data of the images of one call, fetched once per image."""

    def __init__(self, m, images):
        self.m, self.images, self.cache = m, images, {}

    def image(self, i):
        if i not in self.cache:
            d, _, _ = self.images[i]
            n = d.shape[0]
            dbg = self.m.debug_image(i, n)
            nm = self.m.debug_image_norms(i)
            perm = dbg["perm"]
            x = np.zeros((dbg["rowop"].shape[0], d.shape[1]), np.float64)
            x[:n] = d[perm]
            self.cache[i] = dict(n=n, perm=perm, x=x, n2=(x ** 2).sum(1), rowop=dbg["rowop"].astype(np.float64),
                                 colop=dbg["colop"].astype(np.float64), min_norm2=nm["min_norm2"],
                                 max_norm2=nm["max_norm2"])
        return self.cache[i]


def _check_task(rp, task, col, row, thr, rat, want, tally, tag):
    C, R = rp.image(col), rp.image(row)
    n = R["n"]
    got = rp.m.debug_reject_rows(task, n)
    assert got is not None, f"{tag}: task went through the reject pass but the hook has nothing"
    tally.tasks += 1
    tally.rows += n
    # 1. bands
    lo, hi = helpers.gate_bands(rp.images[col], rp.images[row])
    assert np.array_equal(got["bands"][:, 0], lo) and np.array_equal(got["bands"][:, 1], hi), f"{tag}: bands"
    has = hi > lo
    args = got["args"].astype(np.float64)
    a1, a2, na, eps = args.T
    stat = got["rowstat"]
    assert np.all(np.isnan(args[~has])), f"{tag}: a row without a band has arguments"
    assert np.all(stat[~has] == 1), f"{tag}: a row without a band survived"
    assert np.all(np.isfinite(a1[has])), f"{tag}: a row with a band has a1 = -inf (no column folded in)"
    assert np.all(np.isin(stat, (0, 1)))
    survivors = np.nonzero(stat == 0)[0]
    assert np.array_equal(got["survivors"], survivors), f"{tag}: survivor list is not the rows with rowstat 0"
    # no rejected row has a match in the reference (want: (column, row) original indices)
    inv = np.empty(n, np.int64)
    inv[R["perm"]] = np.arange(n)
    assert np.all(stat[inv[want[:, 1]]] == 0), f"{tag}: a row the reference matches was rejected"
    if not has.any():
        return
    # eps, |a|^2 and the K choice the pass made (rj_ksteps, replayed in float32)
    e = eps[has]
    assert np.all(e == e[0]), f"{tag}: eps differs between rows"
    eps = float(e[0])
    eps64 = _task_eps(rp.images[col][0], rp.images[row][0])
    assert abs(eps - eps64) <= 1e-5 * eps64, f"{tag}: eps {eps} vs float64 {eps64}"
    assert np.all(np.abs(na[has] - R["n2"][:n][has]) <= 1e-6 * np.maximum(1.0, R["n2"][:n][has])), f"{tag}: |a|^2"
    mn, mx = np.float32(C["min_norm2"]), np.float32(C["max_norm2"])
    k48 = bool(np.float32(0.5) * (mx - mn) <= np.float32(eps))
    K = 48 if k48 else 64
    noff1 = float(np.float32(0.5) * mn) if k48 else 0.0
    noff2 = float(np.float32(0.5) * mx) if k48 else 0.0
    spread = 0.5 * (float(mx) - float(mn)) if k48 else 0.0
    tally.k48 += k48
    tally.k64 += not k48
    tally.K[(col, row)] = K
    # per 256-row unit over its band union: chunk maxima of the FP16-operand scores (G) and of the exact ones (T)
    G1, G2, T1, T2 = (np.full(n, -np.inf) for _ in range(4))
    for s0 in range(0, n, UNIT):
        sl = slice(s0, min(s0 + UNIT, n))
        h = has[sl]
        if not h.any():
            continue
        u0 = int(lo[sl][h].min()) // CHUNK * CHUNK
        u1 = -(-int(hi[sl][h].max()) // CHUNK) * CHUNK
        cols = np.arange(u0, u1)
        out = ~((cols >= lo[sl, None]) & (cols < hi[sl, None]))
        t = R["rowop"][sl, :K] @ C["colop"][u0:u1, :K].T
        x = R["x"][sl] @ C["x"][u0:u1].T - 0.5 * C["n2"][u0:u1]
        t[out] = -np.inf
        x[out] = -np.inf
        G1[sl], G2[sl] = _top2(t.reshape(t.shape[0], -1, CHUNK).max(2))
        T1[sl], T2[sl] = _top2(x.reshape(x.shape[0], -1, CHUNK).max(2))
    # 2. tight tier
    two = has & ((hi + CHUNK - 1) // CHUNK - lo // CHUNK >= 2)
    assert np.all(a2[has & ~two] == -np.inf), f"{tag}: a2 finite for a band inside one chunk"
    assert np.all(np.isfinite(a2[two])), f"{tag}: a2 = -inf for a band over two chunks"
    d1 = np.abs(a1[has] - (G1[has] - noff1))
    d2 = np.abs(a2[two] - (G2[two] - noff2))
    worst = max(d1.max(), d2.max(initial=0.0))
    bad = np.nonzero(has)[0][d1 > TIGHT_TOL]
    assert bad.size == 0, f"{tag} K={K}: a1 off the FP16-operand g1 on {bad.size} rows, e.g. row {bad[0]}: " \
                          f"{a1[bad[0]]!r} vs {G1[bad[0]] - noff1!r}"
    bad = np.nonzero(two)[0][d2 > TIGHT_TOL]
    assert bad.size == 0, f"{tag} K={K}: a2 off the FP16-operand g2 on {bad.size} rows, e.g. row {bad[0]}: " \
                          f"{a2[bad[0]]!r} vs {G2[bad[0]] - noff2!r}"
    tally.tight = max(tally.tight, worst)
    tally.band_rows += int(has.sum())
    tally.tight_a2 += int(two.sum())
    # 3. certified tier
    assert np.all(a1[has] >= T1[has] - eps), f"{tag}: a1 below the best exact score - eps"
    assert np.all(a2[two] <= T2[two] + eps), f"{tag}: a2 above the second exact chunk maximum + eps"
    c1 = np.abs(a1[has] - T1[has])
    c2 = np.abs(a2[two] - T2[two])
    assert np.all(c1 <= eps + spread) and np.all(c2 <= eps + spread), f"{tag}: two-sided bound"
    tally.cert = max(tally.cert, max(c1.max(), c2.max(initial=0.0)) / eps)
    # 4. decision
    rej_lo, rej_hi = _decisions(na[has], a1[has], a2[has], eps, np.float32(thr), np.float32(rat))
    sure = rej_lo == rej_hi
    tally.boundary += int((~sure).sum())
    st = stat[has].astype(bool)
    bad = np.nonzero(has)[0][sure & (st != rej_lo)]
    assert bad.size == 0, f"{tag}: rowstat disagrees with certified_reject on {bad.size} rows, e.g. row {bad[0]}"


def _run(images, pf, ps, thr, rat, sym, oracle_lib, name, expect_units=None):
    """One fm_match with two-phase scoring forced and the reject dump on; every task checked.  Returns the tally."""
    m = capi.Matcher(0)
    try:
        capi.debug_set_option("two_phase", 1)
        capi.debug_set_option("reject_dump", 1)
        for i, (d, s, l) in enumerate(images):
            m.upload(i, d, s, l)
        res = m.match(pf, ps, thr, rat, sym=sym)
        lists, st = res.all_pairs(), m.stats()
        res.free()
        assert st["two_phase_batches"] >= 1
        tasks = [(a, b) for a, b in zip(pf, ps)]
        if sym:
            tasks = [t for a, b in zip(pf, ps) for t in ((a, b), (b, a))]
        rp = Replay(m, images)
        tally = Tally()
        for t, (col, row) in enumerate(tasks):
            want = oracle_lib.compute_matches(images[col], images[row], thr, rat)
            if not sym:  # the match list itself, as the other reject-pass tests check it
                assert np.array_equal(lists[t], want), f"pair {t}: match list"
            flags = [m.debug_image(i, images[i][0].shape[0], operands=False)["flags"] for i in (col, row)]
            if any(flags):  # exact-flagged: the reject pass skips the task
                assert m.debug_reject_rows(t, images[row][0].shape[0]) is None, f"task {t}: exact task has a dump"
                tally.exact += 1
                continue
            _check_task(rp, t, col, row, thr, rat, want, tally, f"task {t} ({col} x {row})")
    finally:
        capi.debug_set_option("reject_dump", 0)
        capi.debug_set_option("two_phase", -1)
        m.close()
    tally.report(name)
    return tally, st


def _units(images, tasks):
    return sum((images[r][0].shape[0] + UNIT - 1) // UNIT for _, r in tasks)


def test_reject_rows_deep(oracle_lib, sm_count):
    """-sym at -d 1 -d2 0.8: iid filler of at least 6 x sm_count units, then every edge family in the same launch."""
    n_fill = 4
    while n_fill * (n_fill - 1) * ((20000 + UNIT - 1) // UNIT) < 6 * sm_count:  # two tasks per pair under -sym
        n_fill += 1
    images = [_image("iid", 20000, i) for i in range(n_fill)]
    pf = [i for i in range(n_fill) for j in range(i + 1, n_fill)]
    ps = [j for i in range(n_fill) for j in range(i + 1, n_fill)]
    filler_pairs = len(pf)

    def new(img):
        images.append(img)
        return len(images) - 1

    def pair(first, second):  # -sym adds the reverse task
        pf.append(first)
        ps.append(second)

    for n in (1, 127, 128, 129, 385):  # row images ending at 1, 127, 128, 129 rows of a unit
        pair(0, new(_image("iid", n, 100 + n)))
    for n in (1, 15, 16, 17, 255, 257, 4097):  # column images
        pair(new(_image("iid", n, 200 + n)), 1)
    lev = new(_level_columns(ROUND_EDGES, 500))  # band edges at round and step boundaries +-1
    n_lev = len(ROUND_EDGES) - 1
    rng = np.random.default_rng(7)
    for lv in (rng.integers(0, n_lev, 3000), np.repeat(np.arange(n_lev), 64), np.full(256, 3), np.full(256, 1),
               np.full(256, 6), rng.integers(0, n_lev, 100), np.full(1, 12)):
        pair(lev, new(_levels(np.sort(lv), 600 + len(images))))
    narrow = new(_level_columns(NARROW_EDGES, 550))  # bands of one column and of two columns in one chunk
    pair(narrow, new(_levels(np.repeat(np.arange(len(NARROW_EDGES) - 1), 40), 560)))
    tie_cols, tie_rows = _ties()
    pair(new(tie_cols), new(tie_rows))
    d, s, _ = _image("iid", 256, 700)  # split-class unit: the halves' bands are disjoint
    pair(0, new((d, s, np.concatenate([np.zeros(128, np.float32), np.ones(128, np.float32)]))))
    d, s, _ = _image("iid", 600, 701)  # laplacian class absent from the other image: every band empty
    pair(0, new((d, s, np.full(600, 5.0, np.float32))))
    d, s, _ = _image("iid", 900, 702)  # nine laplacian classes: exact-flagged
    pair(0, new((d, s, (np.arange(900) % 9 + 1).astype(np.float32))))
    # K choice: per-keypoint scaled descriptors and an all-zero one (K = 64); norm spread just below / above eps
    rs = np.random.default_rng(5)
    d, s, l = _image("iid", 3000, 400)
    d = (d * rs.uniform(0.5, 2.0, size=(d.shape[0], 1))).astype(np.float32)
    d[777] = 0.0
    scaled = new((d, s, l))
    below = new(_near_eps(_image("iid", 2000, 401), images[1], 0.95))
    above = new(_near_eps(_image("iid", 2000, 402), images[1], 1.05))
    for k in (scaled, below, above):
        pair(k, 1)
    tasks = [t for a, b in zip(pf, ps) for t in ((a, b), (b, a))]
    assert _units(images, tasks[:2 * filler_pairs]) >= 6 * sm_count
    tally, st = _run(images, pf, ps, 1.0, 0.8, True, oracle_lib, "deep -sym -d 1 -d2 0.8")
    assert st["rows_exact"] > 0
    assert tally.k48 > 0
    assert [tally.K[(k, 1)] for k in (scaled, below, above)] == [64, 48, 64]


def test_reject_rows_bank_survivors(oracle_lib, sm_count):
    """-d 1 -d2 0.99 on bank: most rows survive, so the survivor lists are long."""
    n_img = 4
    while n_img * (n_img - 1) // 2 * ((16000 + UNIT - 1) // UNIT) < 2 * sm_count:
        n_img += 1
    images = [_image("bank", 16000, i) for i in range(n_img)]
    pf = [i for i in range(n_img) for j in range(i + 1, n_img)]
    ps = [j for i in range(n_img) for j in range(i + 1, n_img)]
    images.append(_image("bank", 129, 129))
    pf.append(0), ps.append(len(images) - 1)
    images.append(_image("bank", 257, 257))
    pf.append(len(images) - 1), ps.append(1)
    tally, st = _run(images, pf, ps, 1.0, 0.99, False, oracle_lib, "bank -d 1 -d2 0.99")
    assert st["rows"] - st["rows_rejected_early"] > 0.5 * st["rows"]


def test_reject_rows_threshold(oracle_lib, sm_count):
    """-d 0.05: the distance test rejects every row."""
    n_img = 4
    while n_img * (n_img - 1) // 2 * ((16000 + UNIT - 1) // UNIT) < 2 * sm_count:
        n_img += 1
    images = [_image("iid", 16000, i) for i in range(n_img)]
    pf = [i for i in range(n_img) for j in range(i + 1, n_img)]
    ps = [j for i in range(n_img) for j in range(i + 1, n_img)]
    images.append(_image("iid", 129, 129))
    pf.append(0), ps.append(len(images) - 1)
    images.append(_image("iid", 17, 17))
    pf.append(len(images) - 1), ps.append(1)
    tally, st = _run(images, pf, ps, 0.05, 0.8, False, oracle_lib, "iid -d 0.05")
    assert st["rows_rejected_early"] == st["rows"]
