"""Reject pass of two-phase scoring (fm_reject.cuh) with 512-row units: four 128-row quarters per unit, filled into
the two accumulator buffers in turn, and per-quarter partial (g1, g2) merged at unit end.

Every row's g1, g2 and rejection decision is checked against the float64 replay of test_gpu_reject_rows (bands, tight,
certified and decision tiers), and each match list against the fast oracle, on what 512-row units newly expose:
  * row images of 255 .. 1025 rows: units with 1, 2, 3 and 4 row-operand tiles and partial last quarters (n_pad is a
    multiple of 256, not 512, and a unit loads only the tiles of quarters that have rows, so the last unit of an image
    may load fewer than four tiles);
  * a laplacian class boundary inside quarter 1, 2 and 3, so the quarters of one unit have disjoint bands;
  * quarters whose span misses whole column steps of their unit (scale levels far apart inside one unit);
  * K = 48 and K = 64 units in the same launch;
  * a filler of at least 6 x sm_count units ahead of them, so every CTA's row buffers, unit slots, column stages and
    accumulator buffers have wrapped several times when the edge tasks run.
"""
import numpy as np
import pytest

from test_gpu_reject_rows import _image, _level_columns, _levels, _run, oracle_lib, sm_count  # noqa: F401

pytestmark = pytest.mark.gpu

RJ_UNIT = 512  # rows per reject-pass unit
# sorted column positions where one scale level ends and the next begins: levels from 1 column to ~1800 columns wide,
# so a unit whose quarters sit on levels far apart covers steps that some quarters' spans miss
LEVEL_EDGES = (0, 300, 700, 1200, 1201, 1500, 2100, 2400, 4000, 4100, 6000)


def _rj_units(images, ps):
    return sum((images[r][0].shape[0] + RJ_UNIT - 1) // RJ_UNIT for r in ps)


def test_reject_units_edges(oracle_lib, sm_count):
    """-d 1 -d2 0.8, two-phase scoring forced: iid filler, then every 512-row unit edge family in the same launch."""
    n_fill = 4
    while n_fill * (n_fill - 1) // 2 * ((20000 + RJ_UNIT - 1) // RJ_UNIT) < 6 * sm_count:
        n_fill += 1
    images = [_image("iid", 20000, i) for i in range(n_fill)]
    pf = [i for i in range(n_fill) for j in range(i + 1, n_fill)]
    ps = [j for i in range(n_fill) for j in range(i + 1, n_fill)]
    assert _rj_units(images, ps) >= 6 * sm_count

    def new(img):
        images.append(img)
        return len(images) - 1

    # units of 1 to 4 tiles, with full and partial last quarters
    sizes = (255, 256, 257, 383, 384, 385, 511, 512, 513, 1025)
    for n in sizes:
        pf.append(0), ps.append(new(_image("iid", n, 300 + n)))
    # a laplacian class boundary inside quarter 1, 2 and 3 of a 512-row unit (sorted order: class 0, then class 1)
    for p in (200, 300, 450, 640):
        d, s, _ = _image("iid", 700, 400 + p)
        pf.append(1), ps.append(new((d, s, (np.arange(700) >= p).astype(np.float32))))
    # quarters far apart in scale: each quarter's span covers a few steps of the unit's range, and misses the rest
    lev = new(_level_columns(LEVEL_EDGES, 500))
    n_lev = len(LEVEL_EDGES) - 1
    for q_levels in ((0, 3, 7, 9), (0, 0, 9, 9), (1, 1, 1, 8), (2, 5, 5, 5)):  # quarter h at q_levels[h]
        pf.append(lev), ps.append(new(_levels(np.repeat(q_levels, 128), 510 + len(images))))
    rng = np.random.default_rng(11)
    pf.append(lev), ps.append(new(_levels(np.sort(rng.integers(0, n_lev, 1500)), 520)))
    # K = 64: a column image whose squared norms vary (per-keypoint scaled descriptors), against 512-row units
    d, s, l = _image("iid", 3000, 600)
    d = (d * np.random.default_rng(12).uniform(0.5, 2.0, size=(d.shape[0], 1))).astype(np.float32)
    scaled = new((d, s, l))
    for n in (513, 1025):
        pf.append(scaled), ps.append(new(_image("iid", n, 610 + n)))
    pf.append(scaled), ps.append(1)

    tally, st = _run(images, pf, ps, 1.0, 0.8, False, oracle_lib, "512-row units -d 1 -d2 0.8")
    assert tally.exact == 0
    assert tally.tasks == len(pf)
    assert tally.k48 > 0 and tally.k64 >= 3
    assert tally.K[(scaled, 1)] == 64 and tally.K[(0, 1)] == 48
