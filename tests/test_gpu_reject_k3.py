"""Reject pass of two-phase scoring (fm_reject.cuh): 3-K-step chains for column images of normalised descriptors, and
MMAs trimmed to each row half's own band union.

Match lists are compared with the fast oracle with two-phase scoring forced, on batches that mix normalised column
images (K = 48) with others (K = 64), and on the shapes the 16-column trim has edges at.  The issued-work count is
checked against the band arithmetic replayed in numpy with the reference's gate predicate."""
import numpy as np
import pytest

import helpers
from frog_b200 import capi, synth
from oracle import oracle as O

FILLER = 4        # large images: 6 pairs of 16 000 rows = 378 units, more than one persistent CTA per SM can hold
FILLER_N = 16000
COL_SIZES = (1, 15, 16, 17, 255, 257, 4097)  # column images: steps of 1, 15, 16, 17 columns, one past a step, ...
ROW_SIZES = (1, 127, 128, 129, 385)          # row images: the last unit ends at 1, 127, 128 and 129 rows


@pytest.fixture(scope="module")
def oracle_lib(built):
    return O.FastLib()


def _image(kind, n, seed):
    k = synth.make(kind, n, seed)
    return (k.desc, k.scale, k.lap)


def _split_classes(kind, seed):
    """256 keypoints, laplacian 0 for the first 128 and 1 for the rest: the unit's two row halves are the two classes,
    whose bands (and so whose trimmed spans) lie in disjoint column ranges."""
    d, s, _ = _image(kind, 256, seed)
    return (d, s, np.concatenate([np.zeros(128, np.float32), np.ones(128, np.float32)]))


def _filler(kind):
    images = [_image(kind, FILLER_N, i) for i in range(FILLER)]
    pf = [i for i in range(FILLER) for j in range(i + 1, FILLER)]
    ps = [j for i in range(FILLER) for j in range(i + 1, FILLER)]
    return images, pf, ps


def _add_edges(kind, images, pf, ps):
    for n in COL_SIZES:  # columns: image `first`, against a filler image's rows
        images.append(_image(kind, n, 200 + n))
        pf.append(len(images) - 1)
        ps.append(1)
    for n in ROW_SIZES:  # rows: image `second`, against a filler image's columns
        images.append(_image(kind, n, 100 + n))
        pf.append(0)
        ps.append(len(images) - 1)
    images.append(_split_classes(kind, 300))
    pf += [0, len(images) - 1]
    ps += [len(images) - 1, 2]


def _match(images, pf, ps, thr, rat):
    m = capi.Matcher(0)
    try:
        capi.debug_set_option("two_phase", 1)
        for i, (d, s, l) in enumerate(images):
            m.upload(i, d, s, l)
        res = m.match(pf, ps, thr, rat)
        got, st = res.all_pairs(), m.stats()
        res.free()
    finally:
        capi.debug_set_option("two_phase", -1)
        m.close()
    assert st["two_phase_batches"] >= 1
    return got, st


def _check(images, pf, ps, thr, rat, oracle_lib):
    got, st = _match(images, pf, ps, thr, rat)
    want = [oracle_lib.compute_matches(images[i], images[j], thr, rat) for i, j in zip(pf, ps)]
    for p, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g, w), f"pair {p} ({pf[p]}, {ps[p]}): {g.shape[0]} vs {w.shape[0]}"
    return st, want


@pytest.mark.gpu
def test_reject_k3_mixed_with_k4(oracle_lib):
    """Column images whose norms vary (descriptors scaled per keypoint by [0.5, 2]; one all-zero descriptor) take
    the K = 64 chain in the same launch as normalised ones, which take K = 48, as columns and as rows."""
    rng = np.random.default_rng(5)
    images, pf, ps = _filler("iid")
    d, s, l = _image("iid", 3000, 400)
    images.append(((d * rng.uniform(0.5, 2.0, size=(d.shape[0], 1))).astype(np.float32), s, l))
    d, s, l = _image("iid", 2000, 401)
    d = d.copy()
    d[777] = 0.0
    images.append((d, s, l))
    for k in (len(images) - 2, len(images) - 1):
        pf += [k, 0]
        ps += [1, k]
    st, want = _check(images, pf, ps, 1.0, 0.8, oracle_lib)
    assert sum(w.shape[0] for w in want[-4:]) > 0


def _task_eps(ma, mb):
    """task_eps (fm_score.cuh) from the two images' norm statistics."""
    na, nb = np.sqrt(ma["max_norm2"]), np.sqrt(mb["max_norm2"])
    da, db = np.sqrt(ma["max_delta2"]), np.sqrt(mb["max_delta2"])
    return 1.01 * (na * db + da * nb + da * db) + 3e-5 * max(1.0, ma["max_norm2"], mb["max_norm2"])


@pytest.mark.gpu
def test_reject_k_choice_inputs(built):
    """The per-image norm range the reject pass chooses K from (rj_ksteps, fm_reject.cuh): min_norm2 and max_norm2
    are the descriptors' FP32 extremes, and the rule (n_max - n_min) / 2 <= eps picks K = 48 for normalised column
    images and K = 64 for the scaled image and the image with an all-zero descriptor."""
    rng = np.random.default_rng(5)
    norm = _image("iid", 3000, 400)
    d, s, l = _image("iid", 3000, 401)
    scaled = ((d * rng.uniform(0.5, 2.0, size=(d.shape[0], 1))).astype(np.float32), s, l)
    d, s, l = _image("iid", 2000, 402)
    d = d.copy()
    d[777] = 0.0
    zero = (d, s, l)
    images = [norm, scaled, zero, _image("bank", 1000, 403)]
    m = capi.Matcher(0)
    try:
        for i, (d, s, l) in enumerate(images):
            m.upload(i, d, s, l)
        st = [m.debug_image_norms(i) for i in range(len(images))]
    finally:
        m.close()
    for (d, _, _), x in zip(images, st):
        n2 = (d.astype(np.float64) ** 2).sum(1)
        assert abs(x["min_norm2"] - n2.min()) < 1e-5 and abs(x["max_norm2"] - n2.max()) < 1e-5
    assert st[2]["min_norm2"] == 0.0
    row = st[0]
    k48 = [0.5 * (x["max_norm2"] - x["min_norm2"]) <= _task_eps(x, row) for x in st]
    assert k48 == [True, False, False, True]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,rat", [("iid", 0.8), ("bank", 0.9), ("dense", 0.8)])
def test_reject_trim_edges(kind, rat, oracle_lib):
    images, pf, ps = _filler(kind)
    _add_edges(kind, images, pf, ps)
    _check(images, pf, ps, 1.0, rat, oracle_lib)


# ---- issued-work accounting ------------------------------------------------------------------------------------

def _issued(col, row):
    """Scores the reject pass issues for one task: per 256-row unit and row half, 128 x N per 256-column step the
    half's band union meets, N = the step's part of the union rounded out to 16 columns."""
    lo, hi = helpers.gate_bands(col, row)
    total = 0
    for s0 in range(0, lo.shape[0], 256):
        for h in range(2):
            a, b = s0 + 128 * h, min(s0 + 128 * h + 128, lo.shape[0])
            if a >= b:
                continue
            ok = hi[a:b] > lo[a:b]
            if not ok.any():
                continue
            x, y = int(lo[a:b][ok].min()), int(hi[a:b][ok].max())
            for c0 in range(x // 256 * 256, y, 256):
                l, r = max(x, c0) - c0, min(y, c0 + 256) - c0
                total += 128 * (((r + 15) // 16 * 16) - (l // 16 * 16))
    return total


@pytest.mark.gpu
def test_reject_issued_work(built):
    """At -d 0.05 every row fails the distance test, so the capture pass has no survivor unit and scored_pairs is
    the reject pass's count alone."""
    images, pf, ps = _filler("iid")
    _add_edges("iid", images, pf, ps)
    _, st = _match(images, pf, ps, 0.05, 0.8)
    assert st["rows_rejected_early"] == st["rows"]
    want = sum(_issued(images[i], images[j]) for i, j in zip(pf, ps))
    assert st["scored_pairs"] == want


@pytest.mark.gpu
def test_reject_power_iid_20k(built):
    images = [_image("iid", 20000, i) for i in range(4)]
    pf = [i for i in range(4) for j in range(i + 1, 4)]
    ps = [j for i in range(4) for j in range(i + 1, 4)]
    _, st = _match(images, pf, ps, 1.0, 0.8)
    assert st["rows_rejected_early"] >= 0.998 * st["rows"]
