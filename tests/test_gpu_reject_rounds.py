"""Reject pass of two-phase scoring (fm_reject.cuh): each epilogue warp drains one 128-column round of every step of
both row halves, and the two warps of a lane quadrant merge their partial (g1, g2) at unit end.

The column images here have scale levels a factor 2 apart (the scale gate accepts 1.3), so a row's band is exactly
the columns of its level, and the level sizes put band edges where the rounds have theirs: at 128- and 256-column
boundaries and one column either side, bands narrower than a 16-column chunk, and bands wholly inside one round of
every step (one warp of the pair then contributes nothing and merges -inf).  Match lists are compared with the fast
oracle with two-phase scoring forced; the large filler images give the batch enough units to take that path."""
import numpy as np
import pytest

from frog_b200 import capi, synth
from oracle import oracle as O

FILLER = 4
FILLER_N = 16000
# sorted column positions where one scale level ends and the next begins
EDGES = (0, 5, 127, 129, 200, 255, 257, 266, 383, 384, 385, 511, 513, 640, 700, 767, 769, 1030)


@pytest.fixture(scope="module")
def oracle_lib(built):
    return O.FastLib()


def _image(kind, n, seed):
    k = synth.make(kind, n, seed)
    return (k.desc, k.scale, k.lap)


def _levels(levels, seed):
    """Descriptors of the iid set, laplacian 1, scale 2^level (jittered by < 1 %) per keypoint."""
    d, _, _ = _image("iid", len(levels), seed)
    rng = np.random.default_rng(seed)
    s = (2.0 ** np.asarray(levels, np.float64) * rng.uniform(1.0, 1.01, len(levels))).astype(np.float32)
    return (d, s, np.ones(len(levels), np.float32))


def _level_columns():
    sizes = np.diff(EDGES)
    return np.repeat(np.arange(sizes.size), sizes)


def _match(images, pf, ps, thr, rat, oracle_lib):
    want = [oracle_lib.compute_matches(images[i], images[j], thr, rat) for i, j in zip(pf, ps)]
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
    for p, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g, w), f"pair {p} ({pf[p]}, {ps[p]}): {g.shape[0]} vs {w.shape[0]}"
    return st, want


@pytest.mark.gpu
@pytest.mark.parametrize("rat", [0.8, 0.99])
def test_reject_rounds_band_edges(rat, oracle_lib):
    images = [_image("iid", FILLER_N, i) for i in range(FILLER)]
    pf = [i for i in range(FILLER) for j in range(i + 1, FILLER)]
    ps = [j for i in range(FILLER) for j in range(i + 1, FILLER)]
    n_lev = len(EDGES) - 1
    cols = len(images)
    images.append(_levels(_level_columns(), 500))
    rng = np.random.default_rng(7)
    rows = [
        rng.integers(0, n_lev, 3000),          # every level mixed in every warp
        np.repeat(np.arange(n_lev), 64),       # levels in 64-row runs: warps see one or two levels
        np.full(256, 3),                       # one unit, one step, band [129, 200) inside round 1 of step 0
        np.full(256, 1),                       # band [5, 127) inside round 0
        np.full(256, 6),                       # band [257, 266): one chunk wide, just past a step boundary
        rng.integers(0, n_lev, 100),           # 100 rows: row half 1 empty
        np.full(1, 12),                        # one row, band [513, 640)
    ]
    for lv in rows:
        images.append(_levels(np.sort(lv), 600 + len(images)))
        pf.append(cols)
        ps.append(len(images) - 1)
        pf.append(len(images) - 1)  # and the other way round: the level image as columns
        ps.append(cols)
    # split-class unit: laplacian 0 for the first 128 keypoints, 1 for the rest (the halves' bands are disjoint)
    d, s, _ = _image("iid", 256, 700)
    images.append((d, s, np.concatenate([np.zeros(128, np.float32), np.ones(128, np.float32)])))
    pf += [0, len(images) - 1]
    ps += [len(images) - 1, 2]
    # exact-flagged tasks in the same batch: nine laplacian classes route the image to the exact kernel
    d, s, _ = _image("iid", 900, 701)
    images.append((d, s, (np.arange(900) % 9 + 1).astype(np.float32)))
    pf += [0, len(images) - 1]
    ps += [len(images) - 1, 1]
    st, want = _match(images, pf, ps, 1.0, rat, oracle_lib)
    assert st["rows_exact"] > 0
    assert sum(w.shape[0] for w in want[6:]) > 0
