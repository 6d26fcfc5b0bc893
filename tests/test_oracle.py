"""CPU: the three statements of the reference hot path pin each other, and the golden pairs.bin
files written by the unmodified reference binary pin all of them (oracle parity = PINNED)."""
import json
import os
import sys

import numpy as np
import pytest

import helpers
from frog_b200 import pairsbin, synth
from oracle import oracle as O

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import make_ref_golden as rg  # noqa: E402

CASES = sorted(json.load(open(os.path.join(os.path.dirname(__file__), "golden", "manifest.json"))).items())


@pytest.fixture(scope="module")
def libs(built):
    port = O.PortLib()
    ref = O.RefLib() if os.path.exists(O.REF_LIB) else None
    return port, ref


PARAMS = [(0.22, 1.0, False), (1.0, 0.8, False), (1e10, 1.0, False), (0.5, 0.998, True), (1.0, 1.01, False)]


@pytest.mark.parametrize("kind", ["bank", "iid"])
def test_numpy_port_reference_agree(libs, kind):
    port, ref = libs
    a, b = synth.make(kind, 310, 0), synth.make(kind, 257, 1)
    fa, fb = (a.desc, a.scale, a.lap), (b.desc, b.scale, b.lap)
    for thr, rat, sym in PARAMS:
        p = port.compute_matches(fa, fb, thr, rat, sym)
        n = O.compute_matches_numpy(fa, fb, thr, rat, sym)
        assert np.array_equal(p, n)
        if ref is not None:
            assert np.array_equal(ref.compute_matches(fa, fb, thr, rat, sym), p)


def test_norm_is_sequential_fp32(libs):
    port, ref = libs
    rng = np.random.default_rng(3)
    a = rng.standard_normal(48).astype(np.float32)
    b = rng.standard_normal(48).astype(np.float32)
    acc = np.float32(0)
    for k in range(48):
        d = np.float32(a[k] - b[k])
        acc = np.float32(acc + np.float32(d * d))
    assert port.norm(a, b) == acc
    assert O.norm_matrix_numpy(a[None], b[None])[0, 0] == acc
    if ref is not None:
        assert ref.norm(a, b) == acc


def test_known_answers(libs):
    """Edge cases of match.cpp:264-330 (SURVEY.md 8c KAT list)."""
    port, _ = libs
    e = np.eye(48, dtype=np.float32)
    one = np.ones(1, np.float32)

    def cm(first, second, thr=1.0, rat=1.0):
        return port.compute_matches(first, second, thr, rat).tolist()

    row = (0.6 * e[:1] + 0.0, one, one * 0)
    # single surviving column: d2 stays FLT_MAX -> ratio test bypassed (match.cpp:320)
    assert cm((e[:1] * 0.5, one, one * 0), row) == [[0, 0]]
    # laplacian mismatch (match.cpp:270) and scale ratio beyond 1.3 (match.cpp:273-275)
    assert cm((e[:1] * 0.5, one, one * 1), row) == []
    assert cm((e[:1] * 0.5, one * 1.31, one * 0), row) == []
    # scale ratio exactly representable at the boundary: 1.3f/1 == 1.3f is NOT > 1.3 (double)
    assert cm((e[:1] * 0.5, one * np.float32(1.3), one * 0), row) == [[0, 0]]
    assert cm((e[:1] * 0.5, one * np.nextafter(np.float32(1.3), np.float32(2)), one * 0), row) == []
    # exact tie d1 == d2: rejected at -d2 1, accepted at -d2 1.01; lowest column index wins
    two = (np.stack([e[1] * 0.5, e[2] * 0.5]), np.ones(2, np.float32), np.zeros(2, np.float32))
    assert cm(two, row, rat=1.0) == []
    assert cm(two, row, rat=1.01) == [[0, 0]]
    # duplicate of the row itself twice: d1 = d2 = 0 -> sqrt(0/0) is NaN -> rejected even at 1.01
    dup = (np.stack([row[0][0], row[0][0]]), np.ones(2, np.float32), np.zeros(2, np.float32))
    assert cm(dup, row, rat=1.01) == []
    # no surviving column: d1 = FLT_MAX, sqrt(FLT_MAX) = 1.8e19 > 1e10 -> no emit (FROG.py's -d)
    assert cm((e[:1] * 0.5, one, one * 1), row, thr=1e10) == []
    # distance threshold is strict: sqrt(d1) < thr
    d = float(np.sqrt(O.norm_matrix_numpy(row[0], e[:1] * 0.5)[0, 0]))
    assert cm((e[:1] * 0.5, one, one * 0), row, thr=d) == []
    assert cm((e[:1] * 0.5, one, one * 0), row, thr=float(np.nextafter(np.float32(d), np.float32(9)))) == [[0, 0]]


def test_match_all_port_equals_reference(libs):
    """`-all` (matchAll, match.cpp:295-300): the C port against the verbatim reference in-process, including the
    stale `match` carried across rows and the -sym orientation.  Where oracle/_ref is not built, the reference's lists
    as recorded in tests/golden/ref."""
    port, ref = libs
    recorded = rg.load("match_all")[1]
    for key, A, B, thr, sym in rg.match_all_cases():
        want = ref.compute_matches_all(A, B, thr, sym) if ref is not None else recorded[key]
        assert np.array_equal(want, port.compute_matches_all(A, B, thr, sym)), key
    # known answer: rows 0 and 1 both lie within the threshold of column 1 only; column 0 is far.  Row 0 meets the far
    # column first (match = 0), row 1 has its own far column 0 as well -> both emit (0, row); a third row that sees NO
    # far column before its near one inherits the previous row's value.
    e = np.eye(48, dtype=np.float32)
    first = (np.stack([e[0], e[1] * 0.5]), np.ones(2, np.float32), np.zeros(2, np.float32))
    second = (np.stack([e[1] * 0.6, e[1] * 0.55, e[1] * 0.5]), np.ones(3, np.float32), np.zeros(3, np.float32))
    assert port.compute_matches_all(first, second, 0.2).tolist() == [[0, 0], [0, 1], [0, 2]]
    first_r = (first[0][::-1].copy(), first[1], first[2])  # near column first: row 0 emits the initial match = 0
    assert port.compute_matches_all(first_r, second, 0.2).tolist() == [[0, 0], [1, 1], [1, 2]]


@pytest.mark.parametrize("name,case", CASES)
def test_golden_pairs_bin(libs, golden_dir, tmp_path, name, case):
    """host readers/pruning/writer (the C++ bin/match runs) + oracle port == reference bytes."""
    port, _ = libs
    opts = helpers.parse_args(case["args"])
    filenames, rigids, heads, descs = helpers.load_group(os.path.join(golden_dir, case["list"]), opts)
    sched = helpers.pair_schedule(len(filenames), opts["target"])
    if opts["all"]:
        lists = port.match_pairs_all(helpers.images_of(heads, descs), [s[0] for s in sched], [s[1] for s in sched],
                                     opts["dist"], opts["sym"])
    else:
        lists = port.match_pairs(helpers.images_of(heads, descs), [s[0] for s in sched], [s[1] for s in sched],
                                 opts["dist"], opts["ratio"], opts["sym"])
    assert sum(len(l) for l in lists) == case["nb_match"]
    out = str(tmp_path / "pairs.bin")
    helpers.write_pairs(out, filenames, rigids, heads, sched, lists)
    golden = open(os.path.join(golden_dir, name + ".pairs.bin"), "rb").read()
    mine = open(out, "rb").read()
    if mine != golden:
        d = pairsbin.diff(pairsbin.parse(golden), pairsbin.parse(mine))
        pytest.fail(f"pairs.bin differs from the reference: {d}")


def test_reference_binary_regenerates_golden(golden_dir, tmp_path, built):
    """Where the reference binary exists, it must still reproduce a committed fixture."""
    if not os.path.exists(O.REF_BIN):
        pytest.skip("oracle/_ref/match_ref not built here")
    out = str(tmp_path / "o.bin")
    O.run_ref_binary([os.path.join(golden_dir, "list_bin.txt"), "-o", out, "-d", "1", "-d2", "0.8"])
    assert open(out, "rb").read() == open(os.path.join(golden_dir, "bin_ratio.pairs.bin"), "rb").read()


def test_fast_oracle_is_pinned(libs):
    """oracle/fast_oracle.c (vectorised across columns, k sequential) == the plain port == the verbatim reference, on
    the flag sets of the callers, ragged sizes that are no multiple of its 512-column tile, exact ties (strict '<':
    the lowest column wins), duplicated rows (d1 == d2 == 0: NaN ratio), scales sitting exactly on the 1.3f gate,
    a third laplacian value and single-survivor rows (d2 == FLT_MAX)."""
    port, ref = libs
    fast = O.FastLib()
    rng = np.random.default_rng(17)
    cases = []
    for kind, na, nb in (("bank", 1300, 777), ("iid", 513, 1025), ("bank", 1, 40), ("iid", 40, 1), ("iid", 0, 9), ("iid", 9, 0)):
        a, b = synth.make(kind, max(na, 1), 0), synth.make(kind, max(nb, 1), 1)
        cases.append(((a.desc[:na], a.scale[:na], a.lap[:na]), (b.desc[:nb], b.scale[:nb], b.lap[:nb])))
    # adversarial set: ties, duplicates, gate boundaries
    a, b = synth.make("bank", 600, 3), synth.make("bank", 700, 4)
    da, sa, la = a.desc.copy(), a.scale.copy(), a.lap.copy()
    db, sb, lb = b.desc.copy(), b.scale.copy(), b.lap.copy()
    da[100:110] = da[50:60]            # duplicated columns: tie between two columns of image `first`
    db[5] = da[7]; db[6] = da[7]       # rows identical to a column (d1 = 0) ...
    da[8] = da[7]                      # ... and to a second one (d1 = d2 = 0 -> 0/0)
    sb[20:40] = sa[20:40] * np.float32(1.3)   # scale ratio at / next to the float 1.3 boundary
    sb[40:60] = np.nextafter(sa[40:60] * np.float32(1.3), np.float32(10), dtype=np.float32)
    la[300:320] = 2.0; lb[300:330] = 2.0      # a third laplacian value
    la[590:] = 7.0; lb[690] = 7.0             # few columns share the class: some rows have one survivor only
    cases.append(((da, sa, la), (db, sb, lb)))
    n_checked = 0
    for first, second in cases:
        for thr, rat, sym in PARAMS + [(1.0, 1.0, False)]:
            f = fast.compute_matches(first, second, thr, rat, sym)
            assert np.array_equal(f, port.compute_matches(first, second, thr, rat, sym))
            if ref is not None:
                assert np.array_equal(f, ref.compute_matches(first, second, thr, rat, sym))
            n_checked += 1
    assert n_checked == len(cases) * (len(PARAMS) + 1)
    with pytest.raises(ValueError):  # thresholds at which the reference's carried `match` would show: refused
        fast.compute_matches(cases[0][0], cases[0][1], 2e19, 1.0)


def test_links_restatements_agree(libs):
    """readPairs restated literally (push_back loops) == the stable-sort CSR form used at scale."""
    port, _ = libs
    rng = np.random.default_rng(5)
    n_points = {0: 40, 1: 35, 2: 50}
    blocks = []
    for i, j in ((0, 1), (0, 2), (1, 2), (2, 0)):  # the last one: a -targ style block order
        m = np.stack([rng.integers(0, n_points[i], 60), rng.integers(0, n_points[j], 60)], axis=1).astype(np.uint32)
        blocks.append((i, j, m))
    blocks.append((1, 0, np.zeros((0, 2), np.uint32)))
    lists = O.read_pairs_links(blocks, n_points)
    off, data = O.read_pairs_links_csr(blocks, n_points)
    for img, n in n_points.items():
        for p in range(n):
            got = [tuple(x) for x in data[int(off[img][p]): int(off[img][p + 1])].tolist()]
            assert got == lists[img][p]
    assert data.shape[0] == 2 * sum(b[2].shape[0] for b in blocks)
