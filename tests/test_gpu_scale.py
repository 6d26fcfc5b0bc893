"""GPU: parity at BASELINE.json scale (VERDICT r1: "parity at scale, inside pytest -m gpu").

* C2 (10 x 20 000), both synthetic sets, whole group through bin/match: pairs.bin byte-identical to the verbatim
  reference binary run here on the same files (where oracle/_ref is built; elsewhere to its files as recorded in
  tests/golden/ref).
* C3 (50 x 50 000) and C4 (200 x 20 000): 64 image pairs spread over the whole group (not "the first images"), each
  list bit-identical to the fast oracle (oracle/fast_oracle.c, itself pinned to the verbatim build in
  tests/test_oracle.py).
* tensor-core path == exact FP32 engine of the product on every block of C2 and 128 blocks of C3 -- two independent
  device implementations; plus the size-independent properties of a ComputeMatches list on every block.
* config 5: the run.sh sequence (scripts/run_pipeline.sh) around bin/match and around the reference binary (or its
  recorded file), `cmp`.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from frog_b200 import build, capi, pairsbin, synth
from oracle import oracle as O

sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_ref_golden as rg  # noqa: E402

pytestmark = pytest.mark.gpu


def spread_pairs(n_images, k, seed):
    """k distinct image pairs (i < j) spread over the group: the corners plus a seeded sample of all pairs."""
    allp = [(i, j) for i in range(n_images) for j in range(i + 1, n_images)]
    rng = np.random.default_rng(seed)
    pick = {0, len(allp) - 1, n_images - 2}
    while len(pick) < min(k, len(allp)):
        pick.add(int(rng.integers(len(allp))))
    return [allp[p] for p in sorted(pick)]


def check_list_properties(lists, n_first, n_second):
    """What every ComputeMatches list satisfies whatever the data: sorted by `second`, each row at most once
    (match.cpp:262, :323-327), indices in range."""
    for m, nf, ns in zip(lists, n_first, n_second):
        if m.shape[0] == 0:
            continue
        assert np.all(np.diff(m[:, 1].astype(np.int64)) > 0)
        assert m[:, 0].max() < nf and m[:, 1].max() < ns


@pytest.mark.parametrize("kind", ["iid", "bank"])
def test_c2_whole_group_bytes_vs_reference_binary(built, tmp_path, kind):
    lst = synth.write_group(str(tmp_path / "g"), kind, 10, 20000, fmt="bin")
    ref_out, out = str(tmp_path / "ref.bin"), str(tmp_path / "new.bin")
    r = subprocess.run([build.BIN, lst, "-o", out, "-d", "1"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    if os.path.exists(O.REF_BIN):
        O.run_ref_binary([lst, "-o", ref_out, "-d", "1"], threads=os.cpu_count())
        mine, ref = open(out, "rb").read(), open(ref_out, "rb").read()
        if mine != ref:
            pytest.fail(str(pairsbin.diff(pairsbin.parse(ref), pairsbin.parse(mine))))
    else:  # the reference binary's file for this group, as recorded
        assert rg.pairs_digest(out) == rg.load("c2_" + kind)[0]["pairs"], "pairs.bin differs from the reference's"
    assert pairsbin.parse(out).n_matches() > 100000


@pytest.mark.parametrize("name,n_img,n_pts,thr,rat", [("c3", 50, 50000, 1.0, 1.0), ("c4", 200, 20000, 1.0, 0.8)])
def test_big_groups_spread_blocks_vs_fast_oracle(built, name, n_img, n_pts, thr, rat):
    fast = O.FastLib()
    kps = [synth.make("iid", n_pts, i) for i in range(n_img)]
    pairs = spread_pairs(n_img, 64, seed=n_img)
    m = capi.Matcher(0)
    try:
        for i, k in enumerate(kps):
            m.upload(i, k.desc, k.scale, k.lap)
        pf, ps = [p[0] for p in pairs], [p[1] for p in pairs]
        res = m.match(pf, ps, thr, rat)
        got = res.all_pairs()
        st = m.stats()
        res.free()
    finally:
        m.close()
    assert st["score_launches"] >= 1 and st["rows_exact"] < 1e-3 * st["rows"]  # the tensor-core path did the work
    check_list_properties(got, [kps[i].n for i in pf], [kps[j].n for j in ps])
    n_matches = 0
    for (i, j), g in zip(pairs, got):
        a, b = kps[i], kps[j]
        want = fast.compute_matches((a.desc, a.scale, a.lap), (b.desc, b.scale, b.lap), thr, rat)
        assert np.array_equal(g, want), f"{name} block ({i},{j}): {g.shape[0]} vs {want.shape[0]} pairs"
        n_matches += g.shape[0]
    assert n_matches > 0


@pytest.mark.parametrize("name,n_img,n_pts,n_blocks", [("c2", 10, 20000, 45), ("c3", 50, 50000, 128)])
def test_tensor_path_equals_exact_engine_at_scale(built, name, n_img, n_pts, n_blocks):
    kps = [synth.make("iid", n_pts, i) for i in range(n_img)]
    pairs = spread_pairs(n_img, n_blocks, seed=7)
    m = capi.Matcher(0)
    try:
        for i, k in enumerate(kps):
            m.upload(i, k.desc, k.scale, k.lap)
        pf, ps = [p[0] for p in pairs], [p[1] for p in pairs]
        out = []
        for force_exact in (False, True):
            res = m.match(pf, ps, 1.0, 1.0, force_exact=force_exact)
            out.append(res.all_pairs())
            res.free()
    finally:
        m.close()
    check_list_properties(out[0], [kps[i].n for i in pf], [kps[j].n for j in ps])
    for p, (a, b) in enumerate(zip(*out)):
        assert np.array_equal(a, b), f"{name} block {pairs[p]}: tensor path {a.shape[0]} vs exact engine {b.shape[0]} pairs"


def test_config5_pipeline_cmp(built, tmp_path):
    """BASELINE.json config 5, as far as this image allows (no VTK: surf3d / frog are stand-ins, SURVEY.md 8c): the
    run.sh sequence with NPOINTS = 20000 keypoint files written in surf3d's .csv.gz format, once around bin/match
    and once around the reference binary; pairs.bin `cmp`'d (identical pairs.bin => identical frog input)."""
    n_img = 8
    kp_dir = tmp_path / "keypoints"
    synth.write_group(str(kp_dir), "bank", n_img, 20000, fmt="csv.gz", threads=8)
    outs = {}
    for tag, exe in (("new", build.BIN), ("ref", O.REF_BIN)):
        if tag == "ref" and not os.path.exists(exe):
            continue  # compared with the reference's file as recorded, below
        r, pairs = rg.run_pipeline(str(tmp_path), str(kp_dir), exe, n_img, tag)
        assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
        assert "Nb Match : " in r.stdout and f"read {n_img} images" in r.stdout and "Match time" in r.stdout
        outs[tag] = open(pairs, "rb").read()
    if "ref" in outs:
        assert outs["new"] == outs["ref"], "pairs.bin differs from the reference's"
    else:
        assert rg.pairs_digest(outs["new"]) == rg.load("config5")[0]["pairs"], "pairs.bin differs from the reference's"
    assert pairsbin.parse(outs["new"]).n_matches() > 10000
