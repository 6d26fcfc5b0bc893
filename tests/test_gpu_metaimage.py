"""GPU: volumes in every MetaImage encoding the reader accepts and in the element types int8 / uint32 / float64.  The
new types go through the producer's cast and integral exactly as the numpy restatement does; the encodings are
lossless, so bin/surf3d's files and bin/match's pairs.bin must be byte-identical to those of the plain .mha, whose
outputs are pinned to the reference by test_gpu_surf.py and test_gpu_volumes.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from frog_b200 import build, pairsbin, surf

sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_ref_golden as rg  # noqa: E402
import make_surf_golden as mg  # noqa: E402
from oracle import surf_numpy as sn  # noqa: E402

pytestmark = pytest.mark.gpu

OUTPUTS = (".csv.gz", ".csv", ".bin", ".json")


@pytest.fixture(scope="module")
def producer(built):
    p = surf.Producer(0)
    p.keep_cast_volume(True)
    yield p
    p.close()


def test_new_voxel_types_host_and_device(producer):
    """int8 / uint32 / float64 from host and device pointers: cast + integral equal the numpy restatement."""
    import torch
    rng = np.random.default_rng(11)
    base = rng.integers(0, 200, (37, 45, 61))
    frac = rng.random((37, 45, 61))
    cases = [
        (base - 120).astype(np.int8),                                        # negative int8
        (base.astype(np.uint64) * 10_000_000 + 2_100_000_000).astype(np.uint32),  # most values above INT_MAX
        (base.astype(np.uint64) * 1000).astype(np.uint32),
        base * 0.731 - 55.0 + frac * 1e-9,                                   # doubles that are not floats
        base + 1e301,                                                         # every value above 1e300
    ]
    assert (cases[1] > 2**31 - 1).mean() > 0.5 and not np.array_equal(cases[3], cases[3].astype(np.float32))
    for vol in cases:
        cast = sn.cast_shift(vol)
        producer.set_volume(vol)
        assert np.array_equal(producer.cast_volume(), cast) and np.array_equal(producer.integral(), sn.integral(cast))
        dev = torch.from_numpy(np.ascontiguousarray(vol).view(np.uint8)).cuda()
        torch.cuda.synchronize()
        producer.set_volume_device(dev.data_ptr(), vol.dtype, vol.shape)
        assert np.array_equal(producer.cast_volume(), cast) and np.array_equal(producer.integral(), sn.integral(cast))
    for dt, lo, hi in ((np.int8, -128, 128), (np.uint32, 0, 2**32), (np.float64, -3e9, 3e9)):
        wide = (rng.random((3, 5, 1300)) * (hi - lo) + lo) if dt == np.float64 else rng.integers(lo, hi, (3, 5, 1300))
        wide = wide.astype(dt)  # rows longer than one scan block
        producer.set_volume(wide)
        cast = sn.cast_shift(wide)
        assert np.array_equal(producer.cast_volume(), cast) and np.array_equal(producer.integral(), sn.integral(cast))


def surf3d(vol_path, base, extra=()):
    r = subprocess.run([build.SURF_BIN, vol_path, "-o", base, "-t", "0", "-n", "20000", "-bin", "1", "-csv", "1"] + list(extra),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    return {ext: open(base + ext, "rb").read() for ext in OUTPUTS}


ENCODINGS = {
    "zlib1": dict(compress=1), "zlib6": dict(compress=6), "zlib9": dict(compress=9),
    "gzip": dict(compress=6, gzip=True), "zlib_nosize": dict(compress=6, compressed_size=False),
    "raw_header0": dict(data_file="d.raw", header_size=0), "raw_header37": dict(data_file="d.raw", header_size=37),
    "raw_header_auto": dict(data_file="d.raw", header_size=-1), "zraw": dict(data_file="d.zraw", compress=6),
    "zraw_gzip_nosize": dict(data_file="d.zraw", compress=1, gzip=True, compressed_size=False),
    "big_endian": dict(byte_order=">"), "big_endian_zraw": dict(byte_order=">", data_file="d.zraw", compress=6),
    "element_msb": dict(byte_order=">", compress=9),
}


@pytest.mark.parametrize("name", ["small", "mid"])
def test_encodings_give_identical_files(built, tmp_path, name):
    c = mg.CASES[name]
    vol = mg.case_volume(name)
    plain = str(tmp_path / "plain.mha")
    surf.write_metaimage(plain, vol, c["spacing"], c["origin"])
    want = surf3d(plain, str(tmp_path / "plain"))
    assert len(want[".bin"]) > 0
    for enc, kw in ENCODINGS.items():
        p = tmp_path / (enc + (".mhd" if "data_file" in kw else ".mha"))
        surf.write_metaimage(str(p), vol, c["spacing"], c["origin"], **kw)
        if enc == "element_msb":
            p.write_bytes(p.read_bytes().replace(b"BinaryDataByteOrderMSB = True", b"ElementByteOrderMSB = True"))
        got = surf3d(str(p), str(tmp_path / enc))
        for ext in OUTPUTS:
            assert got[ext] == want[ext], (enc, ext)


def test_element_types_give_identical_files(built, tmp_path):
    """The f32 golden volume as MET_DOUBLE; a volume whose values fit int8 (and are non-negative) as MET_CHAR,
    MET_SHORT, MET_INT and MET_UINT."""
    f32 = mg.case_volume("f32")
    files = {}
    for dt in (np.float32, np.float64):
        p = str(tmp_path / f"f_{np.dtype(dt).name}.mha")
        surf.write_metaimage(p, f32.astype(dt))
        files[dt] = surf3d(p, str(tmp_path / f"f_{np.dtype(dt).name}"))
    assert files[np.float32] == files[np.float64] and len(files[np.float32][".bin"]) > 0
    small = mg.case_volume("small").astype(np.int64)
    small = (small - small.min()) * 127 // (small.max() - small.min())
    files = []
    for dt in (np.int8, np.int16, np.int32, np.uint32):
        p = str(tmp_path / f"s_{np.dtype(dt).name}.mha")
        surf.write_metaimage(p, small.astype(dt), compress=6)
        files.append(surf3d(p, str(tmp_path / f"s_{np.dtype(dt).name}")))
    assert all(f == files[0] for f in files) and len(files[0][".bin"]) > 0


def test_double_points_and_raw_descriptors(built, tmp_path):
    """-p points and -type 1 descriptors on a MET_DOUBLE volume equal those on the same values as MET_FLOAT."""
    f32 = mg.case_volume("f32")
    rng = np.random.default_rng(5)
    pts = np.stack([rng.uniform(8, 95, 40), rng.uniform(8, 100, 40), rng.uniform(8, 87, 40), rng.uniform(1.5, 4, 40)], 1)
    pfile = tmp_path / "pts.csv"
    pfile.write_text("".join("%.4f,%.4f,%.4f,%.4f\n" % tuple(p) for p in pts))
    out = {}
    for dt in (np.float32, np.float64):
        p = str(tmp_path / f"v_{np.dtype(dt).name}.mha")
        surf.write_metaimage(p, f32.astype(dt), compress=1)
        out[dt] = (surf3d(p, str(tmp_path / f"p_{np.dtype(dt).name}"), ["-p", str(pfile)]),
                   surf3d(p, str(tmp_path / f"r_{np.dtype(dt).name}"), ["-type", "1", "-r", "2", "-n", "300"]))
    assert out[np.float32] == out[np.float64]
    assert len(out[np.float32][0][".bin"]) == 40 * 54 * 4 and len(out[np.float32][1][".bin"]) > 0


def clamp_values(vol, lo, hi):
    """surf_io.cpp clamp_values<T>: through double against the float option values, replaced by (T)value."""
    v = vol.copy()
    lo32, hi32 = np.float32(lo), np.float32(hi)
    v[v.astype(np.float64) < np.float64(lo32)] = np.array(lo32).astype(v.dtype)
    v[v.astype(np.float64) > np.float64(hi32)] = np.array(hi32).astype(v.dtype)
    return v


@pytest.mark.parametrize("dtype", [np.int8, np.uint32, np.float64], ids=lambda d: np.dtype(d).name)
def test_clamp_on_new_types(built, tmp_path, dtype):
    small = mg.case_volume("small").astype(np.float64)
    unit = (small - small.min()) / (small.max() - small.min())
    vol, lo, hi = {
        np.int8: (np.round(unit * 250 - 125), -60, 70.0),
        np.uint32: (np.round(unit * 3.5e9), 1e8, 3e9),
        np.float64: (unit * 1234.5678 - 300.123456789, -0.25, 500.5),
    }[dtype]
    vol = vol.astype(dtype)
    p = str(tmp_path / "v.mha")
    surf.write_metaimage(p, vol, compress=6, byte_order=">")
    got = surf3d(p, str(tmp_path / "opt"), ["-cmin", repr(float(lo)), "-cmax", repr(float(hi))])
    q = str(tmp_path / "clamped.mha")
    clamped = clamp_values(vol, lo, hi)
    assert (clamped != vol).any()
    surf.write_metaimage(q, clamped)
    assert got == surf3d(q, str(tmp_path / "pre")) and len(got[".bin"]) > 0


# ---- bin/match over mixed encodings ------------------------------------------------------------------------------

def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def same_pairs(a, b):
    """Equal image by image, block by block; the names differ with the entries."""
    assert len(a.points) == len(b.points)
    for x, y in zip(a.points, b.points):
        assert np.array_equal(bits(x), bits(y))
    assert np.array_equal(np.asarray(a.rigids), np.asarray(b.rigids))
    assert [(i, j) for i, j, _ in a.blocks] == [(i, j) for i, j, _ in b.blocks]
    for (_, _, x), (_, _, y) in zip(a.blocks, b.blocks):
        assert np.array_equal(x, y)
    assert a.n_matches() > 0


@pytest.mark.parametrize("mode", ["one_shot", "gpus2", "serve"])
def test_match_mixed_encodings(built, tmp_path, mode):
    vols = rg.run_sh_volumes()
    plain, mixed = [], []
    for i, v in enumerate(vols):
        sp, org = rg.RUN_SH_SPACING, rg.RUN_SH_ORIGIN(i)
        p = str(tmp_path / f"plain{i}.mha")
        surf.write_metaimage(p, v, sp, org)
        plain.append(p)
        kw = [dict(data_file=f"m{i}.zraw", compress=6), dict(compress=1), dict(byte_order=">")][i % 3]
        m = str(tmp_path / (f"m{i}.mhd" if "data_file" in kw else f"m{i}.mha"))
        surf.write_metaimage(m, v, sp, org, **kw)
        mixed.append(m)
    kp = str(tmp_path / "kp0")
    surf3d(plain[0], kp)  # a keypoint file in both lists
    plain.append(kp + ".csv.gz")
    mixed.append(kp + ".csv.gz")
    (tmp_path / "plain.txt").write_text("".join(f + "\n" for f in plain))
    (tmp_path / "mixed.txt").write_text("".join(f + "\n" for f in mixed))
    env = dict(os.environ)
    extra = []
    if mode == "gpus2":
        extra = ["-gpus", "2"]
    elif mode == "serve":
        env.update(FROGMATCH_SOCKET=str(tmp_path / "fm.sock"), FROGMATCH_SERVE_IDLE="60")
        extra = ["-serve", "1"]
    args = ["-d", "1", "-surf3d", "-t 0 -n 20000"]
    try:
        for lst in ("plain", "mixed"):
            r = subprocess.run([build.BIN, str(tmp_path / f"{lst}.txt"), "-o", str(tmp_path / f"{lst}.bin")] + args + extra,
                               capture_output=True, text=True, timeout=600, env=env)
            assert r.returncode == 0, r.stderr
    finally:
        if mode == "serve":
            subprocess.run([build.BIN, "-serve-stop"], env=env, timeout=60)
    a, b = pairsbin.parse(str(tmp_path / "plain.bin")), pairsbin.parse(str(tmp_path / "mixed.bin"))
    assert [os.path.basename(n) for n in b.names] == [os.path.basename(n) for n in mixed]
    same_pairs(a, b)
