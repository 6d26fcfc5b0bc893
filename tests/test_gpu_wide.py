"""GPU: the wide tensor-core path (descriptor lengths d != 48, fm_wide.cuh) -- match lists bit-identical to the oracle
port and to the exact engine, routing, the candidate-list overflow route, real raw Haar descriptors from the producer,
and the certified score bound through the fm_debug_wide_unit dump."""
import functools
import json
import subprocess

import numpy as np
import pytest

from frog_b200 import build, capi, surf, synth
from oracle import oracle as O

pytestmark = pytest.mark.gpu

PARAMS = [(0.22, 1.0), (1.0, 0.8), (1e10, 1.0), (0.5, 0.998)]
LENGTHS = [1, 2, 3, 24, 47, 49, 63, 64, 65, 72, 192, 648, 1000, 1536, 3000, 4096]


@pytest.fixture(scope="module")
def env(built):
    m = capi.Matcher(0)
    yield m, O.PortLib()
    m.close()


def unit_rows(x):
    x = np.asarray(x, np.float64)
    return (x / np.maximum(np.linalg.norm(x, axis=1, keepdims=True), 1e-30)).astype(np.float32)


def bank_group(d, n_images, n, seed, noise=0.1, outliers=0.1):
    """`bank`-style group at length d: images draw from 2n shared prototypes plus noise of norm ~`noise`,
    renormalised, so true matches exist; SURF3D scale and laplacian distributions (synth)."""
    rng = np.random.default_rng(seed)
    proto = unit_rows(rng.standard_normal((2 * n, d)))
    pscale = synth._scales(rng, 2 * n)
    plap = rng.integers(0, 2, 2 * n).astype(np.float32)
    images = []
    for _ in range(n_images):
        pick = rng.permutation(2 * n)[:n]
        desc = unit_rows(proto[pick] + noise / np.sqrt(d) * rng.standard_normal((n, d)))
        scale = pscale[pick] * (1.0 + rng.uniform(-0.03, 0.03, n))
        lap = plap[pick].copy()
        out = rng.uniform(size=n) < outliers
        desc[out] = unit_rows(rng.standard_normal((int(out.sum()), d)))
        images.append((desc, scale.astype(np.float32), lap))
    return images


def upload(m, images):
    m.clear()
    for i, (d, s, l) in enumerate(images):
        m.upload(i, d, s, l)


def match_lists(m, pf, ps, thr, rat, **kw):
    res = m.match(pf, ps, thr, rat, **kw)
    got = res.all_pairs()
    dist = [res.distances(p) for p in range(len(pf))] if kw.get("distances") else None
    st = res.stats()
    res.free()
    return got, dist, st


def assert_same(got, want, what):
    assert len(got) == len(want)
    for p, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g, w), f"{what}: pair {p}: {len(g)} vs {len(w)} matches"


def assert_wide_ran(st, d):
    assert st["score_launches"] >= 1 and st["scored_pairs"] > 0, "the wide scoring kernel did not run"
    if d > 3:  # d <= 3: unit descriptors take few distinct values, most rows tie and go to the exact redo
        assert st["rows_exact"] < 0.02 * st["rows"], st


# ---- 1. lengths ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", LENGTHS)
def test_lengths_against_port(env, d):
    m, port = env
    n = 600 if d <= 1000 else 400
    images = bank_group(d, 3, n, seed=d)
    images[2] = tuple(x[: n - 77] for x in images[2])  # ragged
    upload(m, images)
    pf, ps = [0, 0, 1], [1, 2, 2]
    for thr, rat in PARAMS:
        want = port.match_pairs(images, pf, ps, thr, rat)
        got, _, st = match_lists(m, pf, ps, thr, rat)
        assert_same(got, want, f"d={d} -d {thr} -d2 {rat}")
        assert_wide_ran(st, d)
    # -sym with repeated pairs and a self pair; emitted distances equal the exact engine's bit for bit
    pf, ps = [0, 0, 2, 1, 1], [1, 1, 0, 2, 1]
    want = port.match_pairs(images, pf, ps, 1.0, 0.9, True)
    got, dist, st = match_lists(m, pf, ps, 1.0, 0.9, sym=True, distances=True)
    assert_same(got, want, f"d={d} -sym")
    assert_wide_ran(st, d)
    xgot, xdist, xst = match_lists(m, pf, ps, 1.0, 0.9, sym=True, distances=True, force_exact=True)
    assert_same(xgot, want, f"d={d} -sym exact engine")
    assert xst["rows_exact"] == xst["rows"]
    for a, b in zip(dist, xdist):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


# ---- 2. shapes -----------------------------------------------------------------------------------------------------
def test_shapes(env):
    m, port = env
    d = 192
    rng = np.random.default_rng(11)
    rows = [1, 127, 128, 129, 1100]
    cols = [1, 255, 256, 257, 4097]
    base = bank_group(d, 2, 4097, seed=3)
    images = []
    for k, n in enumerate(rows + cols):
        src = base[k % 2]
        sel = rng.permutation(4097)[:n]
        images.append(tuple(x[sel] for x in src))
    images.append((np.zeros((0, d), np.float32), np.zeros(0, np.float32), np.zeros(0, np.float32)))  # empty image
    upload(m, images)
    nr, empty = len(rows), len(rows) + len(cols)
    pf = [nr + j for j in range(len(cols)) for _ in range(nr)] + [empty, 0]
    ps = [i for _ in range(len(cols)) for i in range(nr)] + [0, empty]
    for thr, rat in [(1.0, 0.9), (1e10, 1.0)]:
        want = port.match_pairs(images, pf, ps, thr, rat)
        got, _, st = match_lists(m, pf, ps, thr, rat)
        assert_same(got, want, f"shapes -d {thr} -d2 {rat}")
        assert_wide_ran(st, d)


def test_one_column_bands_and_step_edges(env):
    """One laplacian class; scales a factor 2 apart give every row a band of exactly one column, and two scale groups
    of 256 columns put a band edge exactly on a 256-column step boundary."""
    m, port = env
    d = 72
    rng = np.random.default_rng(12)
    n1 = 300
    s1 = (2.0 ** rng.integers(0, 20, n1)).astype(np.float32)
    a = unit_rows(rng.standard_normal((n1, d)))
    b = unit_rows(a + 0.05 / np.sqrt(d) * rng.standard_normal((n1, d)))
    one = [(a, s1, np.zeros(n1, np.float32)), (b, s1[rng.permutation(n1)], np.zeros(n1, np.float32))]
    s2 = np.repeat(np.float32([1.0, 2.0]), 256)
    c = unit_rows(rng.standard_normal((512, d)))
    e = unit_rows(c + 0.05 / np.sqrt(d) * rng.standard_normal((512, d)))
    edge = [(c, s2, np.zeros(512, np.float32)), (e, s2.copy(), np.zeros(512, np.float32))]
    for images in (one, edge):
        upload(m, images)
        for thr, rat in [(1.0, 0.9), (1e10, 1.0)]:
            want = port.match_pairs(images, [0, 1], [1, 0], thr, rat)
            got, _, st = match_lists(m, [0, 1], [1, 0], thr, rat)
            assert_same(got, want, "one-column bands / step edge")
            assert st["score_launches"] >= 1 and st["scored_pairs"] > 0


# ---- 3. routing ----------------------------------------------------------------------------------------------------
def test_too_long_stays_exact(env):
    m, port = env
    d = 24 * 6 ** 3  # surf3d -type 1 -r 6
    images = bank_group(d, 3, 200, seed=5)
    upload(m, images)
    want = port.match_pairs(images, [0, 0, 1], [1, 2, 2], 1.0, 0.9)
    got, _, st = match_lists(m, [0, 0, 1], [1, 2, 2], 1.0, 0.9)
    assert_same(got, want, "d = 5184")
    assert st["rows_exact"] == st["rows"] and st["scored_pairs"] == 0


def test_flagged_images_route_to_exact(env):
    m, port = env
    d = 192
    images = bank_group(d, 6, 500, seed=6)
    nan = list(images[2]); nan[0] = nan[0].copy(); nan[0][7, 5] = np.nan; images[2] = tuple(nan)
    big = list(images[3]); big[0] = big[0] * np.float32(4.5); images[3] = tuple(big)  # |desc|^2 = 20.25 > 16
    neg = list(images[4]); neg[1] = neg[1].copy(); neg[1][3] = 0.0; images[4] = tuple(neg)  # scale <= 0
    many = list(images[5]); many[2] = (np.arange(500) % 11).astype(np.float32); images[5] = tuple(many)  # 11 classes
    upload(m, images)
    pf = [0, 0, 0, 0, 0, 1, 2, 3]
    ps = [1, 2, 3, 4, 5, 0, 1, 1]
    n = [len(im[1]) for im in images]
    exact_rows = sum(n[b] for a, b in zip(pf, ps) if a >= 2 or b >= 2)
    for thr, rat in [(1.0, 0.9), (1e10, 1.0)]:
        want = port.match_pairs(images, pf, ps, thr, rat)
        got, _, st = match_lists(m, pf, ps, thr, rat)
        assert_same(got, want, "flagged images")
        assert st["scored_pairs"] > 0
        assert exact_rows <= st["rows_exact"] < exact_rows + 0.02 * (st["rows"] - exact_rows)


def test_force_exact_and_match_all_unchanged(env):
    m, port = env
    d = 648
    images = bank_group(d, 3, 300, seed=7)
    upload(m, images)
    want = port.match_pairs(images, [0, 0, 1], [1, 2, 2], 1.0, 0.9)
    got, _, st = match_lists(m, [0, 0, 1], [1, 2, 2], 1.0, 0.9, force_exact=True)
    assert_same(got, want, "force_exact")
    assert st["rows_exact"] == st["rows"] and st["scored_pairs"] == 0
    want = port.match_pairs_all(images, [0, 1], [1, 2], 1.3, True)
    res = m.match([0, 1], [1, 2], 1.3, 1.0, sym=True, match_all=True)
    assert res.total == sum(len(w) for w in want)
    assert_same(res.all_pairs(), want, "match_all")
    res.free()


# ---- 4. overflow ---------------------------------------------------------------------------------------------------
def test_truncated_lists_go_to_redo(env):
    """Columns duplicated 12 times (and near-duplicates) tie far beyond the 8 kept candidates: those rows' lists are
    truncated with the 8th score inside the band, so they go to the exact redo kernel -- and still come out identical."""
    m, port = env
    d = 192
    images = bank_group(d, 2, 600, seed=8)
    desc, scale, lap = (x.copy() for x in images[0])
    rng = np.random.default_rng(9)
    for src in range(0, 240, 12):  # 20 descriptors, each copied onto the next 11 columns (same scale and class)
        desc[src + 1: src + 12] = desc[src]
        scale[src + 1: src + 12] = scale[src]
        lap[src + 1: src + 12] = lap[src]
        desc[src + 6: src + 12] = unit_rows(desc[src + 6: src + 12] + 1e-7 * rng.standard_normal((6, d)))
    upload(m, images)
    _, _, st0 = match_lists(m, [0], [1], 1e10, 1.0)
    images[0] = (desc, scale, lap)
    upload(m, images)
    want = port.match_pairs(images, [0], [1], 1e10, 1.0)
    got, _, st = match_lists(m, [0], [1], 1e10, 1.0)
    assert_same(got, want, "duplicated columns")
    assert st["rows_exact"] > st0["rows_exact"]


# ---- 5. real raw Haar descriptors ----------------------------------------------------------------------------------
@functools.lru_cache(maxsize=1)
def haar_volumes():
    """Four 160^3 volumes, each assembled from eight independently seeded textured octants (like the producer's
    benchmark volume, at 6 % of its size); volumes 0 and 1 share their structure (1 is a shifted copy of 0)."""
    def volume(seed, size=160):
        h = size // 2
        out = np.empty((size, size, size), np.int16)
        for k, (z, y, x) in enumerate([(z, y, x) for z in (0, h) for y in (0, h) for x in (0, h)]):
            out[z:z + h, y:y + h, x:x + h] = synth.make_volume((h, h, h), seed + k, blobs_per_mvox=1500.0, texture=250.0)
        return out
    vols = [volume(60 + 10 * k) for k in range(3)]
    vols.insert(1, np.roll(vols[0], (2, -3, 4), axis=(0, 1, 2)))
    return vols


def haar_group(radius):
    """surf3d -type 1 -r radius on the four volumes of haar_volumes()."""
    out = []
    for v in haar_volumes():
        pts, desc, _ = surf.run(v, descriptor_type=1, radius=radius, number_of_points=600)
        out.append((pts, desc.reshape(len(pts), -1)))
    return out


def l2_rows(desc):
    """Each descriptor divided by its L2 length (in double, as surf3d normalises -type 0); zero rows stay zero."""
    x = desc.astype(np.float64)
    n = np.linalg.norm(x, axis=1, keepdims=True)
    return np.where(n > 0, x / np.where(n > 0, n, 1.0), x).astype(np.float32)


@pytest.mark.parametrize("radius", [2, 3])
def test_raw_haar_descriptors(env, tmp_path, radius):
    """The producer writes -type 1 descriptors as raw Haar sums, not L2-normalised (its normalisation step is -type 0
    only): |desc|^2 is far above 16, so those images stay on the exact kernel.  The same descriptors L2-normalised, as a
    caller does before matching them, take the wide path -- through the C ABI and through bin/match."""
    m, port = env
    group = haar_group(radius)
    d = 24 * radius ** 3
    assert all(desc.shape[1] == d and len(desc) >= 100 for _, desc in group)
    pf, ps = [0, 0, 0, 1, 1, 2], [1, 2, 3, 2, 3, 3]
    raw = [(desc, pts["scale"].copy(), pts["laplacian"].astype(np.float32)) for pts, desc in group]
    upload(m, raw)
    want = port.match_pairs(raw, pf, ps, 1e10, 1.0)
    got, _, st = match_lists(m, pf, ps, 1e10, 1.0)
    assert_same(got, want, f"raw Haar r={radius}, as written")
    assert st["rows_exact"] == st["rows"]  # kImgBigNorm
    images = [(l2_rows(desc), s, l) for desc, s, l in raw]
    upload(m, images)
    for thr, rat in [(0.22, 1.0), (1.0, 0.8), (1e10, 1.0)]:
        want = port.match_pairs(images, pf, ps, thr, rat)
        got, _, st = match_lists(m, pf, ps, thr, rat)
        assert_same(got, want, f"raw Haar r={radius} -d {thr} -d2 {rat}")
        assert_wide_ran(st, d)
    assert len(got[0]) > 50  # volumes 0 and 1 share structure: real matches
    # bin/match on .csv.gz files written like surf3d writes them: byte-identical to its exact engine
    paths = []
    for k, (pts, _) in enumerate(group):
        p = str(tmp_path / f"haar{k}.csv.gz")
        surf.write_points(p, "csv.gz", pts, images[k][0])
        paths.append(p)
    lst = tmp_path / "list.txt"
    lst.write_text("\n".join(paths) + "\n")
    outs = {}
    for exact in ("0", "1"):
        out, stats = str(tmp_path / f"p{exact}.bin"), str(tmp_path / f"s{exact}.json")
        r = subprocess.run([build.BIN, str(lst), "-o", out, "-d", "1", "-d2", "0.9", "-exact", exact, "-stats", stats],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert f"{d} values per descriptor" in r.stdout
        outs[exact] = (open(out, "rb").read(), json.load(open(stats)))
    assert outs["0"][0] == outs["1"][0]
    assert outs["0"][1]["scored_pairs"] > 0 and outs["1"][1]["scored_pairs"] == 0


# ---- 6. the certified bound ----------------------------------------------------------------------------------------
def f32_norm_rows(x):
    """prep's FP32 |x|^2 per row: fmaf(v, v, acc), k ascending (v*v is exact in float64)."""
    acc = np.zeros(x.shape[0], np.float32)
    for k in range(x.shape[1]):
        v = x[:, k].astype(np.float64)
        acc = (acc.astype(np.float64) + v * v).astype(np.float32)
    return acc


def ref_dist2(at, ia, bt, ib):
    """The reference's norm (match.cpp:243-251) of the pairs (at[:, ia], bt[:, ib]) (descriptors as columns) in
    float32, one separately rounded operation at a time, k ascending."""
    acc = np.zeros(ia.shape[0], np.float32)
    for k in range(at.shape[0]):
        e = at[k][ia] - bt[k][ib]
        acc = acc + e * e
    return acc


@pytest.mark.parametrize("d", [24, 192, 1000, 3000, 4096])
def test_bound_through_unit_dump(env, d):
    m, _ = env
    na, nb = 700, 300
    images = bank_group(d, 2, max(na, nb), seed=100 + d)
    images = [tuple(x[:na] for x in images[0]), tuple(x[:nb] for x in images[1])]
    upload(m, images)
    A, B = images
    pa = m.debug_image(0, na, operands=False)["perm"]
    pb = m.debug_image(1, nb, operands=False)["perm"]
    a16 = A[0].astype(np.float16).astype(np.float64)
    b16 = B[0].astype(np.float16).astype(np.float64)
    nrm_a = f32_norm_rows(A[0]).astype(np.float64)
    worst_tight, worst_cert = 0.0, 0.0
    for rb in range((nb + 127) // 128):
        u = m.debug_wide_unit(0, 1, rb, na, nb)
        eps, kpad = u["eps"], u["k_pad"]
        assert kpad == (d + 63) // 64 * 64 and eps > 0
        nr = u["bands"].shape[0]
        t = u["t"][:nr, :na]
        rows = pb[rb * 128: rb * 128 + nr]
        seen = np.isfinite(t)
        lo, hi = u["bands"][:, 0].astype(np.int64), u["bands"][:, 1].astype(np.int64)
        cols = np.arange(na)
        inband = (cols[None, :] >= lo[:, None]) & (cols[None, :] < hi[:, None])
        assert np.all(seen[inband]), "an in-band column was not scored"
        r_idx, c_idx = np.nonzero(seen)
        ra, cb = rows[r_idx], pa[c_idx]
        got = t[r_idx, c_idx].astype(np.float64)
        # tight: the float64 product of the FP16 operands minus prep's |b|^2 / 2 (packing, k-blocks, TMEM columns)
        prod = b16[rows] @ a16[pa].T
        want = prod[r_idx, c_idx] - 0.5 * nrm_a[cb]
        tol = 2.0 ** -21 * (1 + kpad / 64)
        worst_tight = max(worst_tight, float(np.max(np.abs(got - want))) / tol)
        assert np.all(np.abs(got - want) <= tol), f"d={d}: dumped score off by {np.max(np.abs(got - want))}"
        # certified: |t~ - t_ref| <= eps, t_ref = (|a|^2 - d_ref^2) / 2 with the reference's FP32 distance
        if rb == 0:
            row_n2 = np.einsum("ij,ij->i", B[0].astype(np.float64), B[0].astype(np.float64))
            t_ref = 0.5 * (row_n2[ra] - ref_dist2(np.ascontiguousarray(B[0].T), ra, np.ascontiguousarray(A[0].T), cb).astype(np.float64))
            err = np.abs(got - t_ref)
            worst_cert = max(worst_cert, float(np.max(err)) / eps)
            assert np.all(err <= eps), f"d={d}: |t~ - t_ref| = {np.max(err)} > eps = {eps}"
        # candidates: the row's 8 largest gated scores, truncated bit exactly when more than 8 columns are gated
        for r in range(nr):
            w = int(hi[r] - lo[r])
            ct, cc = u["cand_t"][r], u["cand_col"][r]
            assert bool(cc[0] & 0x80000000) == (w > 8)
            cc = cc & 0x7FFFFFFF
            top = np.sort(t[r, lo[r]:hi[r]])[::-1][:8]
            k = min(w, 8)
            assert np.array_equal(ct[:k], top), f"d={d} row {r}"
            assert np.all(ct[k:] == -np.inf)
            assert np.all((cc[:k] >= lo[r]) & (cc[:k] < hi[r])) and np.array_equal(t[r, cc[:k]], ct[:k])
            assert len(set(cc[:k].tolist())) == k
    print(f"\nwide bound d={d}: K_pad={kpad} eps={eps:.3e} max|t~ - t_ref|/eps={worst_cert:.4f} "
          f"max tight error/tol={worst_tight:.4f}")
