"""GPU: compaction (fm_compact.cuh), the last device stage of every fm_match, against a numpy replay of its contract.

Compaction turns the per-row results of a batch (`rowres[row]` = matched column or 0xFFFFFFFF) into the dense per-pair
lists, the per-pair counts and the running total.  fm_debug_compact runs one batch's compaction on given data through
the same launch routine fm_match uses, on the context's own scratch and look-back state.  The replay here restates the
contract of the fm_compact.cuh header: chunks in order, rows ascending inside each chunk, (m, row_local + i) -- or
(row_local + i, m) when the chunk's swap bit is set -- distances copied bit for bit, pair_counts += each chunk's total,
total = base + all of them.  Every comparison is exact (integers, float32 bit patterns as uint32), over the whole
output array, so the sentinel slots before `base` and after `base + total` must come back untouched.

Paths: the library's choice, one launch (decoupled look-back), the three launches in versions 3 (default), 2 and 1,
and the look-all study build of the one-launch kernel (every chunk sums all its predecessors, 1024 per round).
"""
import numpy as np
import pytest

from frog_b200 import capi, synth
from oracle import oracle as O

pytestmark = pytest.mark.gpu

NONE = 0xFFFFFFFF
SENTINEL = 0xA5A5A5A5
ONE_PASS_CHUNKS = 1536
# path name -> (fm_debug_compact path, "compact_v" option)
PATHS = {
    "auto": (capi.COMPACT_AUTO, 3),
    "one": (capi.COMPACT_ONE, 3),
    "v3": (capi.COMPACT_THREE, 3),
    "v2": (capi.COMPACT_THREE, 2),
    "v1": (capi.COMPACT_THREE, 1),
    "lookall": (capi.COMPACT_LOOKALL, 3),
}


@pytest.fixture(scope="module")
def m(built):
    matcher = capi.Matcher(0)
    yield matcher
    matcher.close()


@pytest.fixture(scope="module")
def sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- the replay ---------------------------------------------------------------------------------------------------


def replay(rowres, rowdist, chunks, pair_counts):
    """(pairs [T,2] uint32, dists [T] float32 or None, pair_counts after) of one batch, in output order."""
    ch = chunks.astype(np.int64)
    n = ch[:, 1] & 0x7FFFFFFF
    swap = (ch[:, 1] >> 31).astype(bool)
    cid = np.repeat(np.arange(ch.shape[0]), n)
    off = np.arange(int(n.sum())) - np.repeat(np.cumsum(n) - n, n)
    rows = ch[cid, 0] + off
    col = rowres[rows]
    hit = col != NONE
    cid, off, rows, col = cid[hit], off[hit], rows[hit], col[hit].astype(np.int64)
    local = ch[cid, 2] + off
    sw = swap[cid]
    pairs = np.stack([np.where(sw, local, col), np.where(sw, col, local)], 1).astype(np.uint32)
    counts = pair_counts + np.bincount(ch[cid, 3], minlength=pair_counts.shape[0]).astype(np.uint32)
    return pairs, (None if rowdist is None else rowdist[rows]), counts


def run_checked(m, rowres, rowdist, chunks, pair_counts, path, base, epoch=None, status=False):
    """One fm_debug_compact call against the replay; returns the hook's dict (total, epoch, status)."""
    pairs, dists, counts = replay(rowres, rowdist, chunks, pair_counts)
    total = pairs.shape[0]
    slots = base + total + 5
    out = np.full((slots, 2), SENTINEL, np.uint32)
    want = out.copy()
    want[base:base + total] = pairs
    out_dist = want_dist = None
    if rowdist is not None:
        out_dist = np.full(slots, SENTINEL, np.uint32).view(np.float32)
        want_dist = out_dist.copy()
        want_dist[base:base + total] = dists
    pc = pair_counts.copy()
    code, version = PATHS[path]
    if version != 3:
        capi.debug_set_option("compact_v", version)
    try:
        got = m.debug_compact(rowres, chunks, code, base, out, pc, rowdist=rowdist, out_dist=out_dist, epoch=epoch,
                              status=status)
    finally:
        if version != 3:
            capi.debug_set_option("compact_v", 3)
    what = f"path {path}, {chunks.shape[0]} chunks, base {base}, distances {rowdist is not None}"
    assert got["total"] == base + total, what
    bad = np.nonzero(np.any(out != want, axis=1))[0]
    assert bad.size == 0, f"{what}: {bad.size} slots differ, first at {bad[:8]} (matches at [{base}, {base + total}))"
    if rowdist is not None:
        assert np.array_equal(out_dist.view(np.uint32), want_dist.view(np.uint32)), what
    assert np.array_equal(pc, counts), what
    return got


# ---- batches built from chunk specifications ----------------------------------------------------------------------


def assemble(specs, seed, n_pairs=5):
    """rowres / rowdist / chunk records for chunks given as (rows, matched row indices).  Every chunk is preceded by
    rows no chunk covers, holding non-kNone values the kernels must ignore; row_abs alternates odd and even; half the
    chunks carry the swap bit; pair ids cycle through a non-monotone permutation; pair_counts start non-zero."""
    rng = np.random.default_rng(seed)
    perm = rng.permutation(n_pairs)
    parts, recs, pos = [], [], 0
    for k, (n, hits) in enumerate(specs):
        gap = 1 + 2 * int(rng.integers(0, 3))
        if (pos + gap) % 2 != (1 if k % 2 == 0 else 0):
            gap += 1
        parts.append(rng.integers(0, 1 << 20, gap, dtype=np.uint32))  # uncovered rows: not kNone
        pos += gap
        seg = np.full(n, NONE, np.uint32)
        hits = np.asarray(hits, np.int64)
        seg[hits] = rng.integers(0, 1 << 31, hits.shape[0], dtype=np.uint32)
        parts.append(seg)
        row_local = int(rng.integers(0, 1 << 24))
        recs.append((pos, n | (0x80000000 if k % 2 else 0), row_local, int(perm[k % n_pairs])))
        pos += n
    parts.append(np.arange(3, dtype=np.uint32))  # trailing uncovered rows
    rowres = np.concatenate(parts)
    rowdist = (rng.random(rowres.shape[0]) * 4.0).astype(np.float32)
    chunks = np.array(recs, np.uint32)
    pair_counts = rng.integers(1, 1000, n_pairs).astype(np.uint32)
    return rowres, rowdist, chunks, pair_counts


def _family(name, seed):
    rng = np.random.default_rng(seed)

    def some(lo, hi, k):  # k distinct rows in [lo, hi)
        return np.sort(rng.choice(np.arange(lo, hi), size=k, replace=False))

    if name == "lengths":  # partial chunks and full ones, ~30 % of rows matched, first and last row always
        specs = []
        for n in (1, 31, 32, 33, 511, 512, 513, 4095, 4096):
            hits = set(np.nonzero(rng.random(n) < 0.3)[0].tolist()) | {0, n - 1}
            specs.append((n, sorted(hits)))
        return specs
    if name == "totals":  # the parking boundary (<= 64 matches park during the count pass) and dense chunks
        return [(4096, some(0, 4096, t)) for t in (0, 1, 63, 64, 65, 512, 4096)] + [(1000, some(0, 1000, 64)),
                                                                                   (1000, some(0, 1000, 65))]
    if name == "placement":  # warps of the v3 count pass own 512 consecutive rows; the others interleave by 128 rows
        return [
            (4096, [0]),
            (4096, [4095]),
            (4096, some(1536, 2048, 40)),                   # one warp's slice, parked
            (4096, some(1536, 2048, 300)),                  # one warp's slice, dense
            (4096, np.arange(3584, 4096)),                  # all of the last warp
            (4096, some(3584, 4096, 50)),
            (4096, 32 * np.arange(128) + rng.integers(0, 32, 128)),  # one per 32-row slice
            (2048, 32 * np.arange(64) + rng.integers(0, 32, 64)),    # ... 64 of them: parked
            (1000, [0, 511, 999]),
            (513, [512]),
            (4096, sorted(set((512 * np.arange(1, 8) - 1).tolist()) | set((512 * np.arange(1, 8)).tolist()))),
        ]
    raise ValueError(name)


@pytest.mark.parametrize("odd_base", [False, True])
@pytest.mark.parametrize("dist", [False, True])
@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("family", ["lengths", "totals", "placement"])
def test_chunk_families(m, family, path, dist, odd_base):
    seed = {"lengths": 1, "totals": 2, "placement": 3}[family]
    rowres, rowdist, chunks, pc = assemble(_family(family, seed), seed)
    run_checked(m, rowres, rowdist if dist else None, chunks, pc, path, 7 if odd_base else 6)


# ---- chunk counts -------------------------------------------------------------------------------------------------


def small_chunks(k, seed):
    """k chunks of 1..64 rows: a third without matches, a third sparse, a third fully matched."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, 65, k)
    kind = rng.integers(0, 3, k)
    specs = []
    for n, t in zip(lens.tolist(), kind.tolist()):
        hits = [] if t == 0 else (np.nonzero(rng.random(n) < 0.2)[0] if t == 1 else np.arange(n))
        specs.append((n, hits))
    return assemble(specs, seed, n_pairs=37)


@pytest.mark.parametrize("count", [1, 2, 1023, 1024, 1025, 1536, 1537, "3sm+1", "8sm+1", 32768, 32769])
def test_chunk_counts(m, sm_count, count):
    """Both sides of the one-launch limit (1536 chunks) and of a second look-back round (1024 predecessors), a wrap of
    the persistent count pass (3 CTAs per SM) and of the grid-stride scatter pass (8 per SM), and both sides of the
    scan pass's register limit (32 768 chunks).  Batches the library would compact in one launch are also run through
    the three launches and the look-all build."""
    k = {"3sm+1": 3 * sm_count + 1, "8sm+1": 8 * sm_count + 1}.get(count, count)
    rowres, rowdist, chunks, pc = small_chunks(k, seed=k)
    paths = ["auto"] + (["v3", "lookall"] if k <= ONE_PASS_CHUNKS else [])
    for dist in (False, True):
        for path in paths:
            run_checked(m, rowres, rowdist if dist else None, chunks, pc, path, 5)


def test_refuses_bad_arguments(m):
    rowres, rowdist, chunks, pc = small_chunks(4, seed=4)
    out = np.zeros((rowres.shape[0] + 8, 2), np.uint32)

    def refused(rr, ch, path=capi.COMPACT_AUTO, base=0, slots=None, counts=pc):
        o = out if slots is None else np.zeros((slots, 2), np.uint32)
        with pytest.raises(capi.FrogMatchError):
            m.debug_compact(rr, ch, path, base, o, counts.copy())

    big = chunks.copy()
    big[0, 1] = 4097
    refused(np.full(8192, NONE, np.uint32), big)                # more than 4096 rows
    past = chunks.copy()
    past[-1, 0] = rowres.shape[0] - (past[-1, 1] & 0x7FFFFFFF) + 1
    refused(rowres, past)                                       # reaches past n_rows
    refused(rowres, chunks, counts=pc[:int(chunks[:, 3].max())])  # pair >= n_pairs
    many = np.array([(i, 1, 0, 0) for i in range(ONE_PASS_CHUNKS + 1)], np.uint32)
    ones = np.zeros(ONE_PASS_CHUNKS + 1, np.uint32)
    refused(ones, many, path=capi.COMPACT_ONE, slots=2000)      # one launch, > 1536 chunks
    refused(ones, many, path=capi.COMPACT_LOOKALL, slots=2000)
    total = int(replay(rowres, None, chunks, pc)[0].shape[0])
    refused(rowres, chunks, base=3, slots=3 + total - 1)        # base + total > out_slots
    # the boundaries themselves are accepted
    m.debug_compact(ones, many, capi.COMPACT_THREE, 0, np.zeros((ONE_PASS_CHUNKS + 1, 2), np.uint32), pc.copy())
    o = np.zeros((3 + total, 2), np.uint32)
    assert m.debug_compact(rowres, chunks, capi.COMPACT_ONE, 3, o, pc.copy())["total"] == 3 + total


# ---- look-back state across calls ---------------------------------------------------------------------------------


def _small_group():
    kps = [synth.make("bank", 3000, i) for i in range(3)]
    return [(k.desc, k.scale, k.lap) for k in kps], [0, 0, 1], [1, 2, 2]


def _match_lists(m, pf, ps, sym):
    res = m.match(pf, ps, 1.0, 0.9, sym=sym, distances=True)
    out = [(res.pairs(p), res.distances(p).view(np.uint32)) for p in range(len(pf))]
    res.free()
    return out


def test_lookback_state_across_calls(built):
    """One-launch hook calls and fm_match calls on one context share the look-back words and the epoch counter."""
    images, pf, ps = _small_group()
    fresh = capi.Matcher(0)
    try:
        for i, im in enumerate(images):
            fresh.upload(i, *im)
        want = [_match_lists(fresh, pf, ps, sym) for sym in (False, True)]
    finally:
        fresh.close()
    m = capi.Matcher(0)
    try:
        for i, im in enumerate(images):
            m.upload(i, *im)
        got = []
        run_checked(m, *_count_case(ONE_PASS_CHUNKS, 11), "one", 6)
        got.append(_match_lists(m, pf, ps, False))
        run_checked(m, *_count_case(10, 12), "one", 7)
        got.append(_match_lists(m, pf, ps, True))
        run_checked(m, *_count_case(ONE_PASS_CHUNKS, 13), "one", 7)
    finally:
        m.close()
    for g, w in zip(got, want):
        for (gp, gd), (wp, wd) in zip(g, w):
            assert np.array_equal(gp, wp) and np.array_equal(gd, wd)
    assert sum(p.shape[0] for p, _ in want[0]) > 0


def _count_case(k, seed, dist=True):
    rowres, rowdist, chunks, pc = small_chunks(k, seed)
    return rowres, (rowdist if dist else None), chunks, pc


def test_epoch_wrap_clears_status_words(built):
    """The launch epoch cycles 1 .. 2^30 - 2.  Back at epoch 1, the words an earlier epoch-1 launch left must not pass
    for current ones: a later launch would take a stale word of a predecessor that has not published yet as its
    total or prefix.  The counter is set through the hook instead of running 2^30 launches."""
    m = capi.Matcher(0)
    try:
        r = run_checked(m, *_count_case(ONE_PASS_CHUNKS, 21), "one", 4, epoch=0, status=True)
        assert r["epoch"] == 1 and np.all((r["status"] >> np.uint64(34)) == 1)
        r = run_checked(m, *_count_case(3, 22), "one", 4, epoch=(1 << 30) - 3)
        assert r["epoch"] == (1 << 30) - 2
        r = run_checked(m, *_count_case(10, 23), "one", 5, epoch=r["epoch"], status=True)
        assert r["epoch"] == 1
        ep = (r["status"] >> np.uint64(34)).astype(np.int64)
        assert np.all(ep[:10] == 1)
        stale = np.nonzero(ep[10:] == 1)[0] + 10
        assert stale.size == 0, f"{stale.size} status words past the 10 chunks still carry epoch 1 (first {stale[:4]})"
        run_checked(m, *_count_case(ONE_PASS_CHUNKS, 24), "one", 5)
        run_checked(m, *_count_case(ONE_PASS_CHUNKS, 25), "lookall", 6)
    finally:
        m.close()


# ---- distances on the three-launch path, end to end ---------------------------------------------------------------


def _sq_dist(rows_desc, cols_desc):
    """float32 squared distance per (row, column) in the reference's operation order: r += (a_k - b_k)^2, k ascending."""
    r = np.zeros(rows_desc.shape[0], np.float32)
    for k in range(rows_desc.shape[1]):
        d = rows_desc[:, k] - cols_desc[:, k]
        r += d * d
    return r


def test_distances_three_launch_path_end_to_end(built):
    """64 x 20 000 keypoints, a quarter `bank` images (many true matches), the rest `iid`: all 2016 image pairs are
    40 M rows (80 M with -sym) in batches of <= 24 Mi rows, i.e. 1258 tasks x 5 chunks -- well past the one-launch
    limit, so every batch goes through count3 / scan2 / scatter2.  With distances the count pass parks nothing and
    scatter re-ranks every non-empty chunk and routes the distances through its staging area; without them the
    sparse chunks take the parking route.  Both must give the same lists."""
    n_img, n_pts, thr, rat = 64, 20000, 1.0, 0.8
    kps = [synth.make("bank" if i % 4 == 0 else "iid", n_pts, i) for i in range(n_img)]
    pairs = [(i, j) for i in range(n_img) for j in range(i + 1, n_img)]
    pf, ps = [p[0] for p in pairs], [p[1] for p in pairs]
    m = capi.Matcher(0)
    runs = {}
    try:
        for i, k in enumerate(kps):
            m.upload(i, k.desc, k.scale, k.lap)
        for sym in (False, True):
            for dist in (False, True):
                res = m.match(pf, ps, thr, rat, sym=sym, distances=dist)
                lists = res.all_pairs()
                dists = [res.distances(p) for p in range(len(pairs))] if dist else None
                res.free()
                runs[sym, dist] = (lists, dists)
    finally:
        m.close()
    for sym in (False, True):
        for a, b in zip(runs[sym, True][0], runs[sym, False][0]):
            assert np.array_equal(a, b)
    fwd, dist_fwd = runs[False, True]
    both, dist_both = runs[True, True]
    chunk_totals = []
    for p, (i, j) in enumerate(pairs):
        n_fwd = fwd[p].shape[0]
        assert np.array_equal(both[p][:n_fwd], fwd[p])
        a, b = kps[i].desc, kps[j].desc
        # forward: rows of image j scan columns of image i, emitted (first = i's keypoint, second = j's)
        f = fwd[p]
        assert np.array_equal(dist_fwd[p].view(np.uint32), _sq_dist(b[f[:, 1]], a[f[:, 0]]).view(np.uint32)), (i, j)
        assert np.array_equal(dist_both[p][:n_fwd].view(np.uint32), dist_fwd[p].view(np.uint32)), (i, j)
        # -sym half: rows of image i scan columns of image j, emitted (row, match)
        r = both[p][n_fwd:]
        assert np.array_equal(dist_both[p][n_fwd:].view(np.uint32), _sq_dist(a[r[:, 0]], b[r[:, 1]]).view(np.uint32)), (i, j)
        chunk_totals.append(np.bincount(f[:, 1] // 4096, minlength=5))
        chunk_totals.append(np.bincount(r[:, 0] // 4096, minlength=5))
    ct = np.concatenate(chunk_totals)
    assert (ct == 0).any() and ((ct >= 1) & (ct <= 64)).any() and (ct > 64).any(), np.bincount(np.minimum(ct, 65))
    fast = O.FastLib()
    rng = np.random.default_rng(3)
    spread = sorted({0, len(pairs) - 1} | set(rng.choice(len(pairs), 14, replace=False).tolist()))
    for i, j in [pairs[q] for q in spread]:
        p = pairs.index((i, j))
        a, b = (kps[i].desc, kps[i].scale, kps[i].lap), (kps[j].desc, kps[j].scale, kps[j].lap)
        want = fast.compute_matches(a, b, thr, rat)
        assert np.array_equal(fwd[p], want), f"pair ({i},{j}): {fwd[p].shape[0]} vs {want.shape[0]} matches"
        # -sym: the reference's second ComputeMatches call, roles swapped and its pairs pushed as (row, match)
        want = np.concatenate([want, fast.compute_matches(b, a, thr, rat, sym=True)])
        assert np.array_equal(both[p], want), f"pair ({i},{j}) -sym: {both[p].shape[0]} vs {want.shape[0]} matches"
