"""GPU: device groups (fm_group_*).  Every case runs one fm_ctx on the lead and groups with the same uploads and call,
and requires counts, lists, distances, device views and fm_links_build output to be byte-identical.  The groups are one
over 2 GPUs and one over all visible GPUs when there are more (skipped below two devices), and two whose members share
GPU 0 (2 and 3 contexts, debug option "group_repeat"), which run the same sharding, gather and stream ordering on
any box."""
import numpy as np
import pytest
import torch

from frog_b200 import capi, synth
from frog_b200 import dist as fdist

pytestmark = pytest.mark.gpu


def n_gpus():
    return torch.cuda.device_count()


def device_lists(multi_only=False):
    """Member devices of the groups under test (the lead is always GPU 0)."""
    n = n_gpus()
    out = [[0, 1]] + ([list(range(n))] if n > 2 else []) if n >= 2 else []
    if not multi_only:
        out += [[0, 0], [0, 0, 0]]
    if not out:
        pytest.skip("needs two CUDA devices")
    return out


def make_group(devs):
    repeat = len(set(devs)) < len(devs)
    if repeat:
        capi.debug_set_option("group_repeat", 1)
    try:
        return capi.Group(devs)
    finally:
        if repeat:
            capi.debug_set_option("group_repeat", 0)


@pytest.fixture(scope="module")
def ref(built):
    m = capi.Matcher(0)
    yield m
    m.close()


def group(kind, n_images, n, seed=0):
    return [(k.desc, k.scale, k.lap) for k in (synth.make(kind, n, seed + i) for i in range(n_images))]


def wide_group(d, n_images, n, seed):
    """bank-style images at descriptor length d (prototypes + noise, renormalised): true matches exist."""
    rng = np.random.default_rng(seed)

    def unit(x):
        return (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)

    proto = unit(rng.standard_normal((2 * n, d)))
    pscale = synth._scales(rng, 2 * n)
    plap = rng.integers(0, 2, 2 * n).astype(np.float32)
    out = []
    for _ in range(n_images):
        pick = rng.permutation(2 * n)[:n]
        desc = unit(proto[pick] + 0.1 / np.sqrt(d) * rng.standard_normal((n, d)))
        out.append((desc, (pscale[pick] * (1.0 + rng.uniform(-0.03, 0.03, n))).astype(np.float32), plap[pick].copy()))
    return out


def row_major(n_images):
    return [i for i in range(n_images) for j in range(i + 1, n_images)], [j for i in range(n_images) for j in range(i + 1, n_images)]


def load(h, images):
    h.clear()
    for i, (d, s, l) in enumerate(images):
        h.upload(i, d, s, l)


def snapshot(res, pf, ps, device, distances=False, links=True):
    """Everything a caller can read from a result, as bytes: device views first (before any host copy), then counts,
    lists, distances and the links (submission order and pairs.bin order)."""
    res.wait()
    cptr, pptr = res.device_pointers()
    dev = torch.device("cuda", device)
    snap = {"total": int(res.total), "counts": res.counts.tobytes(),
            "dev_counts": fdist.as_torch_u32(cptr, res.n_pairs, dev).cpu().numpy().tobytes(),
            "dev_pairs": fdist.as_torch_u32(pptr, 2 * int(res.total), dev).cpu().numpy().tobytes()}
    res.fetch()
    snap["lists"] = b"".join(res.pairs(p).tobytes() for p in range(res.n_pairs))
    if distances:
        snap["dist"] = b"".join(res.distances(p).tobytes() for p in range(res.n_pairs))
    if links:
        order = sorted(range(len(pf)), key=lambda k: (pf[k], ps[k]))
        for name, bo in (("links", None), ("links_file_order", order)):
            off, data, _ = res.links(pf, ps, bo)
            snap[name] = b"".join(off[i].tobytes() for i in sorted(off)) + data.tobytes()
    return snap


def compare(ref, images, pf, ps, dist, ratio, groups=None, **kw):
    """One context on the lead against groups of each size; returns the single-context snapshot."""
    links = not kw.get("match_all", False)
    load(ref, images)
    res = ref.match(pf, ps, dist, ratio, **kw)
    want = snapshot(res, pf, ps, 0, kw.get("distances", False), links)
    want_stats = res.stats()
    res.free()
    assert want["total"] > 0
    for devs in groups or device_lists():
        G = devs
        g = make_group(devs)
        try:
            load(g, images)
            res = g.match(pf, ps, dist, ratio, **kw)
            got = snapshot(res, pf, ps, 0, kw.get("distances", False), links)
            st = res.stats()
            res.free()
        finally:
            g.close()
        for k in want:
            assert got[k] == want[k], f"G={G}: {k} differs from one context"
        for k in ("descriptor_pairs", "rows"):
            assert st[k] == want_stats[k], (G, k)
    return want


@pytest.mark.parametrize("kind", ["bank", "iid"])
def test_c2_group(ref, kind):
    images = group(kind, 10, 20000, 100)
    pf, ps = row_major(10)
    compare(ref, images, pf, ps, 1.0, 1.0, distances=True)


def test_sym(ref):
    images = group("bank", 6, 8000, 200)
    pf, ps = row_major(6)
    compare(ref, images, pf, ps, 1.0, 1.0, sym=True, distances=True)


def test_targ_pairs(ref):
    images = group("bank", 8, 8000, 300)
    pf = [i for i in range(8) if i != 3]
    compare(ref, images, pf, [3] * len(pf), 1.0, 0.9)


def test_match_all(ref):
    images = group("bank", 5, 3000, 400)
    pf, ps = row_major(5)
    compare(ref, images, pf, ps, 0.3, 1.0, match_all=True)


def test_match_all_row_limit(ref):
    """-all takes at most 2^32 outer-loop rows per call: a group refuses a call one context refuses, even though each
    member's share would be under the limit."""
    n = 1 << 20
    img = group("iid", 1, n, 450)[0]
    pf = ps = [0] * ((0xFFFFFFF0 // n) + 1)
    load(ref, [img])
    with pytest.raises(capi.FrogMatchError, match=r"error -4.*2\^32 outer-loop rows"):
        ref.match(pf, ps, 1e-6, 1.0, match_all=True)
    for devs in device_lists():
        g = make_group(devs)
        try:
            load(g, [img])
            with pytest.raises(capi.FrogMatchError, match=r"error -4.*2\^32 outer-loop rows"):
                g.match(pf, ps, 1e-6, 1.0, match_all=True)
        finally:
            g.close()


def test_unordered_and_repeated_pairs(ref):
    images = group("bank", 6, 6000, 500)
    pf, ps = row_major(6)
    rng = np.random.default_rng(5)
    pf, ps = list(pf) + [4, 0, 2, 4], list(ps) + [1, 1, 3, 1]  # reversed and repeated pairs
    perm = rng.permutation(len(pf))
    compare(ref, images, [pf[k] for k in perm], [ps[k] for k in perm], 1.0, 1.0, distances=True)


def test_wide_d192(ref):
    images = wide_group(192, 5, 4000, 600)
    pf, ps = row_major(5)
    compare(ref, images, pf, ps, 0.3, 0.9, distances=True)


def test_force_exact(ref):
    images = group("bank", 5, 4000, 700)
    pf, ps = row_major(5)
    compare(ref, images, pf, ps, 1.0, 0.9, force_exact=True, distances=True)


def test_two_phase(ref):
    # 28 pairs x 51 row units: every member of a 3-member group still has the 2 x 148 units unsegmented scoring (and so
    # two-phase scoring) needs
    images = group("iid", 8, 13000, 800)
    pf, ps = row_major(8)
    capi.debug_set_option("two_phase", 1)
    try:
        compare(ref, images, pf, ps, 1.0, 0.8, distances=True)
        devs = device_lists()[0]
        g = make_group(devs)
        try:
            load(g, images)
            res = g.match(pf, ps, 1.0, 0.8)
            assert res.stats()["two_phase_batches"] >= len(devs)  # summed over the members
            res.free()
        finally:
            g.close()
    finally:
        capi.debug_set_option("two_phase", -1)


def test_async_two_in_flight(ref):
    images = group("bank", 6, 8000, 900)
    pf, ps = row_major(6)
    pf2, ps2 = ps[::-1], pf[::-1]
    load(ref, images)
    want = []
    for a, b in ((pf, ps), (pf2, ps2)):
        r = ref.match(a, b, 1.0, 1.0, distances=True)
        want.append(snapshot(r, a, b, 0, True))
        r.free()
    for devs in device_lists():
        g = make_group(devs)
        try:
            load(g, images)
            r1 = g.match(pf, ps, 1.0, 1.0, asynchronous=True, distances=True)
            r2 = g.match(pf2, ps2, 1.0, 1.0, asynchronous=True, distances=True)
            assert r1.counts is None and r2.counts is None
            r2.wait()
            r1.wait()
            assert snapshot(r1, pf, ps, 0, True) == want[0]
            assert snapshot(r2, pf2, ps2, 0, True) == want[1]
            r1.free()
            r2.free()
        finally:
            g.close()


def test_device_only_then_fetch(ref):
    images = group("bank", 6, 8000, 1000)
    pf, ps = row_major(6)
    want = compare(ref, images, pf, ps, 1.0, 1.0, device_only=True, distances=True)
    g = make_group(device_lists()[0])
    try:
        load(g, images)
        res = g.match(pf, ps, 1.0, 1.0, device_only=True, distances=True)
        with pytest.raises(capi.FrogMatchError):
            res.pairs(int(np.argmax(res.counts)))  # not on the host before fetch
        res.fetch()
        assert b"".join(res.pairs(p).tobytes() for p in range(res.n_pairs)) == want["lists"]
        res.free()
    finally:
        g.close()


def test_device_pointer_uploads(ref):
    """Images given as device memory of a member's GPU (not the lead's) reach every member directly."""
    images = group("bank", 6, 8000, 1100)
    pf, ps = row_major(6)
    load(ref, images)
    r = ref.match(pf, ps, 1.0, 1.0, distances=True)
    want = snapshot(r, pf, ps, 0, True)
    r.free()
    for devs in device_lists():
        g = make_group(devs)
        try:
            g.clear()
            dev = torch.device("cuda", devs[-1])
            keep = []
            for i, (d, s, l) in enumerate(images):
                t = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in (d, s, l)]
                keep.append(t)
                g.upload_raw(i, t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), d.shape[0], d.shape[1])
            torch.cuda.synchronize(dev)
            res = g.match(pf, ps, 1.0, 1.0, distances=True)
            assert snapshot(res, pf, ps, 0, True) == want
            res.free()
            del keep
        finally:
            g.close()


def test_one_device_group_is_a_context(ref):
    images = group("bank", 5, 6000, 1200)
    pf, ps = row_major(5)
    want = compare(ref, images, pf, ps, 1.0, 0.9, groups=[[0]], distances=True)
    g = capi.Group([0])
    try:
        load(g, images)
        res = g.match(pf, ps, 1.0, 0.9, distances=True)
        st = res.stats()
        assert snapshot(res, pf, ps, 0, True) == want
        res.free()
    finally:
        g.close()
    load(ref, images)
    r = ref.match(pf, ps, 1.0, 0.9, distances=True)
    st_ref = r.stats()
    r.free()
    for k in ("descriptor_pairs", "scored_pairs", "rows", "rows_exact", "candidates", "kernel_launches", "score_launches"):
        assert st[k] == st_ref[k], k


def test_fewer_pairs_than_members(ref):
    images = group("bank", 3, 8000, 1300)
    compare(ref, images, [0], [2], 1.0, 1.0, distances=True)
    compare(ref, images, [1, 0], [2, 1], 1.0, 1.0)


def test_empty_pair_list(ref):
    g = make_group(device_lists()[0])
    try:
        load(g, group("bank", 2, 1000, 1400))
        res = g.match([], [], 1.0, 1.0)
        assert res.total == 0 and res.n_pairs == 0
        res.free()
    finally:
        g.close()


def test_errors(built):
    with pytest.raises(capi.FrogMatchError, match=r"\(-1\).*given twice"):
        capi.Group([0, 0])
    with pytest.raises(capi.FrogMatchError, match=r"\(-1\).*out of range"):
        capi.Group([0, n_gpus()])
    with pytest.raises(capi.FrogMatchError, match=r"\(-1\)"):
        capi.Group([-1])
    g = make_group(device_lists()[0])
    try:
        images = group("bank", 3, 2000, 1500)
        load(g, images)
        with pytest.raises(capi.FrogMatchError, match=r"error -1.*share d"):
            g.upload(3, np.zeros((10, 64), np.float32), np.ones(10, np.float32), np.ones(10, np.float32))
        with pytest.raises(capi.FrogMatchError, match=r"error -1.*not uploaded"):
            g.match([0, 1], [1, 7], 1.0, 1.0)
        with pytest.raises(capi.FrogMatchError, match=r"error -4"):
            g.match([0], [1], 2e19, 1.0)
        res = g.match([0], [1], 1.0, 1.0)  # the group is still usable
        assert res.n_pairs == 1
        res.free()
    finally:
        g.close()


def test_free_after_further_calls(ref):
    images = group("bank", 5, 6000, 1600)
    pf, ps = row_major(5)
    load(ref, images)
    want = []
    for k in range(3):
        r = ref.match(pf[k:], ps[k:], 1.0, 1.0, distances=True)
        want.append(snapshot(r, pf[k:], ps[k:], 0, True))
        r.free()
    g = make_group(device_lists()[0])
    try:
        load(g, images)
        rs = [g.match(pf[k:], ps[k:], 1.0, 1.0, distances=True, asynchronous=k == 1) for k in range(3)]
        rs[0].free()
        assert snapshot(rs[2], pf[2:], ps[2:], 0, True) == want[2]
        rs[2].free()
        r3 = g.match(pf, ps, 1.0, 1.0, distances=True)
        assert snapshot(rs[1], pf[1:], ps[1:], 0, True) == want[1]
        rs[1].free()
        assert snapshot(r3, pf, ps, 0, True) == want[0]
        r3.free()
    finally:
        g.close()
