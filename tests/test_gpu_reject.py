"""Reject pass of two-phase scoring (fm_reject.cuh) against the fast oracle, on the shapes its tiling has edges at.

Two-phase scoring only runs when a batch has at least 2 x SM-count score units (fewer units split rows into column
segments and take the single pass), so every call here carries a few large image pairs beside the edge cases, and
every test checks that the call really went through the reject pass."""
import numpy as np
import pytest

from frog_b200 import capi, synth
from oracle import oracle as O

FILLER = 4        # large images: 6 pairs of 16 000 rows = 378 units, more than one persistent CTA per SM can hold
FILLER_N = 16000
ROW_SIZES = (1, 127, 128, 129, 255, 256, 257, 7777)  # row images: last unit empty, partial or one row past a half
COL_SIZES = (1, 100, 128, 129, 300)                   # column images: one partial 256-column step


@pytest.fixture(scope="module")
def oracle_lib(built):
    return O.FastLib()


def _image(kind, n, seed):
    k = synth.make(kind, n, seed)
    return (k.desc, k.scale, k.lap)


def _split_classes(kind, seed):
    """256 keypoints, laplacian 0 for the first 128 and 1 for the rest: sorted by (class, scale), the unit's two row
    halves are the two classes, whose bands lie in disjoint column ranges."""
    d, s, l = _image(kind, 256, seed)
    l = np.concatenate([np.zeros(128, np.float32), np.ones(128, np.float32)])
    return (d, s, l)


def _run(kind, thr, rat, oracle_lib):
    images = [_image(kind, FILLER_N, i) for i in range(FILLER)]
    pf = [i for i in range(FILLER) for j in range(i + 1, FILLER)]
    ps = [j for i in range(FILLER) for j in range(i + 1, FILLER)]
    for n in ROW_SIZES:  # rows: image `second`
        images.append(_image(kind, n, 100 + n))
        pf.append(0)
        ps.append(len(images) - 1)
    for n in COL_SIZES:  # columns: image `first`
        images.append(_image(kind, n, 200 + n))
        pf.append(len(images) - 1)
        ps.append(1)
    images.append(_split_classes(kind, 300))
    pf += [0, len(images) - 1]
    ps += [len(images) - 1, 2]
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
def test_reject_pass_edges_iid(oracle_lib):
    st, _ = _run("iid", 1.0, 0.8, oracle_lib)
    assert st["rows_rejected_early"] > 0.98 * st["rows"]


@pytest.mark.gpu
def test_reject_pass_edges_bank(oracle_lib):
    """Most rows survive: the survivor lists and the capture pass carry the matches."""
    _, want = _run("bank", 1.0, 0.9, oracle_lib)
    assert sum(w.shape[0] for w in want) > 1000


@pytest.mark.gpu
def test_reject_pass_edges_dense(oracle_lib):
    """One laplacian class and one scale: every column of every step is gated in (no masked group)."""
    st, _ = _run("dense", 1.0, 0.8, oracle_lib)
    assert st["rows_rejected_early"] > 0.98 * st["rows"]
