"""GPU: the SURF3D producer (libfrogsurf.so through its C ABI, bin/surf3d) against the reference -- golden vectors
written by the verbatim reference build, the verbatim build itself where its .so travelled, and the numpy
restatement.  Integer work (cast, integral volume, flags, keypoint order) and FP32 / FP64 arithmetic replayed op for
op (responses, descriptors) are compared BIT FOR BIT; the sub-voxel interpolation (OpenCV SVD in the reference, absent
here) within 1 float ulp with the number of differing values reported (0 on every case so far).  The volumes no
fixture holds are compared with the verbatim build where oracle/_ref is built, else with its outputs as recorded in
tests/golden/ref."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from frog_b200 import build, surf

sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_ref_golden as rg  # noqa: E402
import make_surf_golden as mg  # noqa: E402
from oracle import surf_numpy as sn, surf_oracle as so  # noqa: E402

pytestmark = pytest.mark.gpu

GOLD = os.path.join(ROOT, "tests", "golden", "surf")
MANIFEST = json.load(open(os.path.join(GOLD, "manifest.json")))


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def pts_matrix(pts):
    return np.stack([pts["x"], pts["y"], pts["z"], pts["scale"], pts["response"]], 1)


def assert_points_close(got, want):
    """coordinates / scale within 1 ulp (interpolation solve), response identical"""
    assert got.shape == want.shape
    assert np.array_equal(bits(got[:, 4]), bits(want[:, 4]))
    ulp = np.abs(bits(got[:, :4]).astype(np.int64) - bits(want[:, :4]).astype(np.int64))
    assert ulp.max(initial=0) <= 1, f"{np.count_nonzero(ulp)} coordinate values differ, worst {ulp.max()} ulp"
    return int(np.count_nonzero(ulp))


@pytest.fixture(scope="module")
def producer(built):
    p = surf.Producer(0)
    p.keep_cast_volume(True)
    yield p
    p.close()


@pytest.mark.parametrize("name", ["small", "mid", "f32"])
def test_stages_match_golden(producer, name):
    m, g = MANIFEST[name], np.load(os.path.join(GOLD, name + ".npz"))
    vol = mg.case_volume(name)
    assert mg.sha(vol) == m["volume"]
    p = producer
    p.set_volume(vol)
    assert mg.sha(p.cast_volume()) == m["cast"]
    assert mg.sha(p.integral()) == m["integral"]
    n = p.detect(0.0)
    assert mg.layer_hashes(p.layers()) == m["layers"]  # responses, laplacian, isblob of every layer's interior
    for l in p.layers():                                 # and nothing written outside it
        lim = so.layer_limit(l["filter"], l["step"])
        inner = l["responses"][lim:l["depth"] - lim, lim:l["height"] - lim, lim:l["width"] - lim]
        assert np.count_nonzero(l["responses"]) == np.count_nonzero(inner)
    assert n == m["n_detected"]
    pts, _ = p.points(with_descriptors=False)
    differing = assert_points_close(pts_matrix(pts), g["det_xyzsr"])  # the reference's push_back order
    assert np.array_equal(pts["laplacian"], g["det_lap"])
    p.select(20000)
    p.describe(0, 5, True)
    pts, desc = p.points()
    differing += assert_points_close(pts_matrix(pts), g["xyzsr"])
    assert np.array_equal(pts["laplacian"], g["lap"])
    if differing == 0:
        assert np.array_equal(bits(desc), bits(g["desc"]))
    st = p.stats()
    assert st["n_clamped"] == 0 and st["n_points"] == m["n_points"] and st["ms_response_map"] > 0


def test_descriptors_on_reference_points_bit_exact(producer):
    """Given the reference's own keypoints, descriptors are identical to the last bit: SURF3D (radius 5, normalised;
    radius 4, raw sums) and the raw Haar type (24 r^3 values)."""
    g = np.load(os.path.join(GOLD, "small.npz"))
    p = producer
    p.set_volume(mg.case_volume("small"))
    p.set_points(g["xyzsr"][:, :4])
    p.describe(0, 5, True)
    assert np.array_equal(bits(p.points()[1]), bits(g["desc"]))
    p.set_points(g["r4_xyzsr"][:, :4])
    p.describe(0, 4, False)
    assert np.array_equal(bits(p.points()[1]), bits(g["r4_desc"]))
    p.set_points(g["raw_xyzsr"][:, :4])
    p.describe(1, 3, True)
    d = p.points()[1]
    assert d.shape == (len(g["raw_xyzsr"]), 24 * 27) and np.array_equal(bits(d), bits(g["raw_desc"]))
    with pytest.raises(surf.FrogSurfError):
        p.describe(2, 5, True)  # vtkImageResize sub-volumes: rejected, not approximated


def test_voxel_types_and_device_pointer(producer):
    """Every accepted voxel type, host and device pointers: cast + integral equal the numpy restatement."""
    import torch
    rng = np.random.default_rng(9)
    base = rng.integers(0, 200, (37, 45, 61))
    for dt, off in ((np.uint8, 0), (np.int16, -90), (np.uint16, 40000), (np.int32, -70000), (np.float32, -3.3)):
        vol = (base + off).astype(dt)
        producer.set_volume(vol)
        cast = sn.cast_shift(vol)
        assert np.array_equal(producer.cast_volume(), cast) and np.array_equal(producer.integral(), sn.integral(cast))
    dev = torch.from_numpy(vol).cuda()
    producer.set_volume_device(dev.data_ptr(), np.float32, vol.shape)
    assert np.array_equal(producer.integral(), sn.integral(cast))
    wide = rng.integers(-5, 2000, (3, 5, 1300)).astype(np.int16)  # rows longer than one scan block
    producer.set_volume(wide)
    assert np.array_equal(producer.integral(), sn.integral(sn.cast_shift(wide)))


def reference_surf(name, vol, n_points):
    """(hashes, keypoint arrays) of the verbatim build on `vol`: computed where oracle/_ref is built, else as recorded
    from it (tests/golden/ref, make_ref_golden.py)."""
    return rg.surf_outputs(True, vol, n_points) if so.available() else rg.load(name)


def test_fresh_volume_against_the_reference_build(producer):
    """A volume no fixture holds (four octaves: 400 voxels wide) against the reference's compiled code."""
    vol = rg.fresh_volume()
    want, ref = reference_surf("surf_fresh", vol, 3000)
    p = producer
    p.set_volume(vol)
    assert mg.sha(p.integral()) == want["integral"]
    n = p.detect(0.0)
    assert p.stats()["n_layers"] == 10
    assert mg.layer_hashes(p.layers()) == want["layers"]
    assert n == want["n_detected"]
    pts, _ = p.points(with_descriptors=False)
    differing = assert_points_close(pts_matrix(pts), ref["det_xyzsr"])
    p.select(3000)
    p.describe(0, 5, True)
    pts, desc = p.points()
    differing += assert_points_close(pts_matrix(pts), ref["xyzsr"])
    assert len(pts) == 3000 and np.array_equal(pts["laplacian"], ref["lap"])
    if differing == 0:
        assert mg.sha(desc) == want["desc"]
    p.set_points(ref["xyzsr"][:, :4])
    p.describe(0, 5, True)
    assert mg.sha(p.points()[1]) == want["desc"]


def test_cli_writes_the_reference_files(built, tmp_path):
    """bin/surf3d on a MetaImage volume: csv / csv.gz / bin byte-identical to the files the reference's writers
    produced for the same volume (spacing and origin applied), bounds json as surf3d.cxx:269-285 writes it."""
    c = mg.CASES["small"]
    mha = str(tmp_path / "small.mha")
    surf.write_metaimage(mha, mg.case_volume("small"), c["spacing"], c["origin"])
    base = str(tmp_path / "points")
    r = subprocess.run([build.SURF_BIN, mha, "-o", base, "-t", "0", "-n", "20000", "-bin", "1", "-csv", "1"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "Number of keypoints : 65" in r.stdout
    for fmt in ("csv", "csv.gz", "bin"):
        assert open(base + "." + fmt, "rb").read() == open(os.path.join(GOLD, "small_points." + fmt), "rb").read(), fmt
    b = json.load(open(base + ".json"))["bounds"]
    assert b["xmin"] == c["origin"][0] and abs(b["zmax"] - (c["origin"][2] + 119 * c["spacing"][2])) < 1e-9
    r = subprocess.run([build.SURF_BIN, mha, "-o", base + "9", "-n", "20000", "-gz", "9", "-precision", "4"],
                       capture_output=True, text=True)
    assert r.returncode == 0
    assert open(base + "9.csv.gz", "rb").read() == open(os.path.join(GOLD, "small_points_l9p4.csv.gz"), "rb").read()


def test_producer_feeds_matcher_like_run_sh(built, tmp_path):
    """run.sh:80-93 with both stages on the GPU: surf3d per volume -> list file -> match, against the same chain run
    by the reference's compiled code (its producer writes the .csv.gz files, its matcher pairs them): pairs.bin cmp.
    Where oracle/_ref is not built, against that chain's files as recorded (tests/golden/ref)."""
    import hashlib
    live = so.available() and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "match_ref"))
    want = rg.load("surf_run_sh")[0]
    vols = rg.run_sh_volumes()
    gdir, rdir = tmp_path / "gpu", tmp_path / "ref"
    gdir.mkdir()
    rdir.mkdir()
    for i, v in enumerate(vols):
        mha = str(tmp_path / f"v{i}.mha")
        surf.write_metaimage(mha, v, rg.RUN_SH_SPACING, rg.RUN_SH_ORIGIN(i))
        r = subprocess.run([build.SURF_BIN, mha, "-o", str(gdir / f"points{i}"), "-t", "0", "-n", "20000"], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        got = open(gdir / f"points{i}.csv.gz", "rb").read()
        if live:
            ref = so.RefSurf(v, rg.RUN_SH_SPACING, rg.RUN_SH_ORIGIN(i))
            ref.update(threshold=0.0, number_of_points=20000)
            ref.write(str(rdir / f"points{i}.csv.gz"), "csv.gz")
            assert got == open(rdir / f"points{i}.csv.gz", "rb").read()
        else:
            assert hashlib.sha256(got).hexdigest() == want["files"][i]
    for d in (gdir, rdir):
        open(d / "points.txt", "w").write("".join(f"{d}/points{i}.csv.gz\n" for i in range(len(vols))))
    r = subprocess.run([build.BIN, str(gdir / "points.txt"), "-o", str(gdir / "pairs.bin"), "-d", "1"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = open(gdir / "pairs.bin", "rb").read()
    if live:
        from oracle import oracle
        rr = oracle.run_ref_binary([str(rdir / "points.txt"), "-o", str(rdir / "pairs.bin"), "-d", "1"])
        assert rr.returncode == 0
        assert got == open(rdir / "pairs.bin", "rb").read()
    else:
        assert rg.pairs_digest(got) == want["pairs"]
    assert len(got) > 1000


def test_cli_point_file(built, tmp_path):
    """surf3d -p points.csv: descriptors at given points instead of detection (vtk3DSURF::ReadIPoints); with -n 30 the
    reference's partial_sort runs over 50 equal (zero) responses and decides which 30 survive and in what order."""
    c = mg.CASES["small"]
    g = np.load(os.path.join(GOLD, "pfile.npz"))
    mha = str(tmp_path / "small.mha")
    surf.write_metaimage(mha, mg.case_volume("small"), c["spacing"], c["origin"])
    pfile = os.path.join(GOLD, "pfile_points.csv")
    base = str(tmp_path / "p")
    r = subprocess.run([build.SURF_BIN, mha, "-o", base, "-p", pfile, "-bin", "1", "-csvgz", "0"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    rec = np.fromfile(base + ".bin", np.float32).reshape(-1, 54)
    assert rec.shape[0] == 50 and np.array_equal(bits(rec[:, 6:]), bits(g["desc"]))
    assert not rec[:, 4:6].any()  # laplacian and response stay 0 (Ipoint(), ipoint.h:33)
    r = subprocess.run([build.SURF_BIN, mha, "-o", base + "30", "-p", pfile, "-n", "30"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(base + "30.csv.gz", "rb").read() == open(os.path.join(GOLD, "pfile_points_n30.csv.gz"), "rb").read()


def test_odd_dimensions_against_the_reference_build(producer):
    """Odd sizes on every axis (131 x 103 x 117 voxels, z y x): the parity-split layout's half rows differ in length,
    the layers drop the last voxel of each axis."""
    vol = rg.odd_volume()
    want, ref = reference_surf("surf_odd", vol, 20000)
    p = producer
    p.set_volume(vol)
    assert mg.sha(p.integral()) == want["integral"]
    n = p.detect(0.0)
    assert mg.layer_hashes(p.layers()) == want["layers"]
    assert n == want["n_detected"] and n > 20
    pts, _ = p.points(with_descriptors=False)
    differing = assert_points_close(pts_matrix(pts), ref["det_xyzsr"])
    p.select(20000)
    p.describe(0, 5, True)
    pts, desc = p.points()
    differing += assert_points_close(pts_matrix(pts), ref["xyzsr"])
    assert np.array_equal(pts["laplacian"], ref["lap"])
    if differing == 0:
        assert mg.sha(desc) == want["desc"]
