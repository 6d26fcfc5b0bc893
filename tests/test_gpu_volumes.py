"""Volume entries in bin/match's list (`-surf3d "<options>"`): the SURF3D producer runs in-process and its keypoints
are what `bin/surf3d <volume> <options>` -> .csv.gz -> the reader would give, bit for bit.  Checked at three levels:
the device conversion (fs_get_points_as_read, fs_debug_as_read) against the host writer + strtof, whole pairs.bin
files against the file chain, and the chain's digest recorded from the reference build.  The option refusals and the
load-time independence from libfrogsurf.so run without a GPU."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from frog_b200 import build, hostio, pairsbin, surf

sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_ref_golden as rg  # noqa: E402
import make_surf_golden as mg  # noqa: E402

gpu = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def run_sh_mha(tmp_path_factory):
    """The run.sh volumes as .mha files (spacing 0.75, origins as the recorded chain used)."""
    d = tmp_path_factory.mktemp("vols")
    paths = []
    for i, v in enumerate(rg.run_sh_volumes()):
        p = str(d / f"v{i}.mha")
        surf.write_metaimage(p, v, rg.RUN_SH_SPACING, rg.RUN_SH_ORIGIN(i))
        paths.append(p)
    return paths


def surf3d_csvgz(mha, out_base, opts):
    r = subprocess.run([build.SURF_BIN, mha, "-o", out_base] + opts, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return out_base + ".csv.gz"


def run_match(args, **kw):
    r = subprocess.run([build.BIN] + args, capture_output=True, text=True, timeout=600, **kw)
    assert r.returncode == 0, r.stderr
    return r


def chain_and_volumes(tmp, mhas, surf_opts, match_opts, entries=None):
    """pairs.bin of the file chain (surf3d per volume, then match over the .csv.gz list) and of match over the volume
    list; `entries` picks per image "mha" or "gz" for the second run (default: all volumes)."""
    files = [surf3d_csvgz(m, str(tmp / f"points{i}"), surf_opts) for i, m in enumerate(mhas)]
    (tmp / "files.txt").write_text("".join(f + "\n" for f in files))
    run_match([str(tmp / "files.txt"), "-o", str(tmp / "chain.bin")] + match_opts)
    entries = entries or ["mha"] * len(mhas)
    listed = [m if e == "mha" else f for m, f, e in zip(mhas, files, entries)]
    (tmp / "vols.txt").write_text("".join(f + "\n" for f in listed))
    r = run_match([str(tmp / "vols.txt"), "-o", str(tmp / "vols.bin"), "-surf3d", " ".join(surf_opts)] + match_opts)
    return pairsbin.parse(str(tmp / "chain.bin")), pairsbin.parse(str(tmp / "vols.bin")), listed, r


def assert_same_pairs(chain, vols, listed):
    """Equal after mapping names: the volume run names an image by its entry's base name."""
    assert [os.path.basename(n) for n in vols.names] == [os.path.basename(n) for n in listed]
    assert len(chain.points) == len(vols.points)
    for a, b in zip(chain.points, vols.points):
        assert np.array_equal(bits(a), bits(b))
    assert np.array_equal(np.asarray(chain.rigids), np.asarray(vols.rigids))
    assert [(i, j) for i, j, _ in chain.blocks] == [(i, j) for i, j, _ in vols.blocks]
    for (_, _, a), (_, _, b) in zip(chain.blocks, vols.blocks):
        assert np.array_equal(a, b)
    assert chain.n_matches() > 0


# ---- the device conversion --------------------------------------------------------------------------------------

CONVERSION_CASES = [
    ("run_sh0", -1, None), ("run_sh1", 0, None), ("run_sh2", 3, None), ("small", 4, None), ("small", 9, None),
    ("small", -1, None), ("run_sh0", 9, "aniso"), ("small", 6, "raw"), ("small", 9, "raw"), ("small", 12, "raw"),
]


@gpu
@pytest.mark.parametrize("case,precision,variant", CONVERSION_CASES)
def test_points_as_read_equals_written_file(built, tmp_path, case, precision, variant):
    """Producer.points_as_read == fsio_write_points(csv.gz) then hostio.read_keypoints, every float bit.  `aniso`:
    anisotropic spacing and a negative origin; `raw`: -type 1 -r 2 raw Haar descriptors, not normalised (large values;
    beyond 9 decimals every descriptor takes the host's snprintf path)."""
    if case == "small":
        c = mg.CASES["small"]
        vol, spacing, origin = mg.case_volume("small"), c["spacing"], c["origin"]
    else:
        i = int(case[-1])
        vol, spacing, origin = rg.run_sh_volumes()[i], rg.RUN_SH_SPACING, rg.RUN_SH_ORIGIN(i)
    if variant == "aniso":
        spacing, origin = (0.6, 1.1, 2.3), (-301.7, -0.123, -77.5)
    dtype, radius = (1, 2) if variant == "raw" else (0, 5)
    p = surf.Producer(0)
    try:
        p.set_volume(vol)
        p.detect(0.0)
        p.select(20000)
        p.describe(dtype, radius, variant != "raw")
        pts, desc = p.points()
        head, got = p.points_as_read(precision, spacing, origin)
    finally:
        p.close()
    assert len(pts) >= 50  # the small golden volume has 65 keypoints
    f = str(tmp_path / "points.csv.gz")
    surf.write_points(f, "csv.gz", pts, desc, spacing, origin, precision=precision)
    want_head, want_desc = hostio.read_keypoints(f, d_cap=desc.shape[1])
    assert np.array_equal(bits(head), bits(want_head))
    assert np.array_equal(bits(got), bits(want_desc))


@gpu
def test_debug_as_read_exhaustive(built):
    """fs_debug_as_read == the host formatter + strtof on every float in [-16, 16] and on 10^7 random float bit
    patterns (every exponent: zeros, subnormals, huge values, inf, nan), at precisions 0, 6 and 9."""
    top = int(np.float32(16.0).view(np.uint32))
    chunk = 1 << 25
    rng = np.random.default_rng(7)
    patterns = rng.integers(0, 1 << 32, 10 ** 7, dtype=np.uint64).astype(np.uint32).view(np.float32).astype(np.float64)
    for precision in (0, 6, 9):
        for sign in (0, 1 << 31):
            for a in range(0, top + 1, chunk):
                b = np.arange(a, min(a + chunk, top + 1), dtype=np.uint32) | np.uint32(sign)
                v = b.view(np.float32).astype(np.float64)
                got, want = surf.debug_as_read(v, precision), surf.as_read_host(v, precision)
                bad = np.flatnonzero(bits(got) != bits(want))
                assert bad.size == 0, (precision, v[bad[:5]], got[bad[:5]], want[bad[:5]])
        got, want = surf.debug_as_read(patterns, precision), surf.as_read_host(patterns, precision)
        same = (bits(got) == bits(want)) | (np.isnan(got) & np.isnan(want))
        assert same.all(), (precision, patterns[~same][:5])


# ---- whole runs against the file chain --------------------------------------------------------------------------

CHAIN_CASES = {
    "run_sh": (["-t", "0", "-n", "20000"], ["-d", "1"]),
    "precision4": (["-t", "0", "-n", "20000", "-precision", "4"], ["-d", "1"]),
    "clamp": (["-t", "0", "-n", "20000", "-cmin", "400", "-cmax", "1500"], ["-d", "1"]),
    "raw_haar": (["-t", "0", "-n", "3000", "-type", "1", "-r", "2"], ["-d", "1e9", "-d2", "0.9"]),
    "np_below_n": (["-t", "0", "-n", "20000"], ["-d", "1", "-np", "5000"]),
    "sym": (["-t", "0", "-n", "20000"], ["-d", "1", "-sym"]),
    "targ": (["-t", "0", "-n", "20000"], ["-d", "1", "-targ", "1"]),
}


@gpu
@pytest.mark.parametrize("name", sorted(CHAIN_CASES))
def test_volumes_match_file_chain(built, run_sh_mha, tmp_path, name):
    surf_opts, match_opts = CHAIN_CASES[name]
    chain, vols, listed, r = chain_and_volumes(tmp_path, run_sh_mha, surf_opts, match_opts)
    assert_same_pairs(chain, vols, listed)
    assert "Nb Match : " in r.stdout and "Output file : " in r.stdout


@gpu
def test_volumes_zwindow_rigid(built, run_sh_mha, tmp_path):
    """-zmin / -zmax applied after a rigid column of the list (z + zT), with -sp: the volume list carries the same
    rigid columns as the file list."""
    files = [surf3d_csvgz(m, str(tmp_path / f"points{i}"), ["-t", "0", "-n", "20000"]) for i, m in enumerate(run_sh_mha)]
    rig = [(0.0, 0.0, 0.0), (1.5, -2.0, 12.25), (0.0, 3.0, -20.0)]
    opts = ["-d", "1", "-zmin", "20", "-zmax", "90", "-sp", "0.5"]
    (tmp_path / "files.txt").write_text("".join(f"{f},{a},{b},{c}\n" for f, (a, b, c) in zip(files, rig)))
    (tmp_path / "vols.txt").write_text("".join(f"{m},{a},{b},{c}\n" for m, (a, b, c) in zip(run_sh_mha, rig)))
    run_match([str(tmp_path / "files.txt"), "-o", str(tmp_path / "chain.bin")] + opts)
    run_match([str(tmp_path / "vols.txt"), "-o", str(tmp_path / "vols.bin"), "-surf3d", "-t 0 -n 20000"] + opts)
    chain, vols = pairsbin.parse(str(tmp_path / "chain.bin")), pairsbin.parse(str(tmp_path / "vols.bin"))
    assert_same_pairs(chain, vols, run_sh_mha)
    assert 0 < len(vols.points[1]) < 20000


@gpu
def test_mixed_list(built, run_sh_mha, tmp_path):
    chain, vols, listed, _ = chain_and_volumes(tmp_path, run_sh_mha, ["-t", "0", "-n", "20000"], ["-d", "1"],
                                               entries=["mha", "gz", "mha"])
    assert_same_pairs(chain, vols, listed)


@gpu
def test_run_sh_reference_digest(built, run_sh_mha, tmp_path):
    """The volume run, re-emitted under the chain's names, has the digest recorded from the reference's own
    surf3d -> match chain."""
    (tmp_path / "vols.txt").write_text("".join(m + "\n" for m in run_sh_mha))
    r = run_match([str(tmp_path / "vols.txt"), "-o", str(tmp_path / "vols.bin"), "-d", "1", "-surf3d", "-t 0 -n 20000",
                   "-stats", str(tmp_path / "stats.json")])
    pf = pairsbin.parse(str(tmp_path / "vols.bin"))
    names = [f"points{i}.csv.gz" for i in range(len(run_sh_mha))]
    hostio.write_pairs_bin(str(tmp_path / "renamed.bin"), names, np.asarray(pf.rigids), pf.points, pf.blocks)
    assert rg.pairs_digest(str(tmp_path / "renamed.bin")) == rg.load("surf_run_sh")[0]["pairs"]
    import json
    st = json.load(open(tmp_path / "stats.json"))
    assert st["volumes"] == 3 and st["produce_s"] > 0 and st["produce_gpu_ms"] > 0
    assert "volume" not in r.stdout.lower()  # the reference's stdout lines only


@gpu
@pytest.mark.parametrize("mp", ["0", "1"])
def test_volumes_two_gpus(built, run_sh_mha, tmp_path, mp):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    chain, vols, listed, _ = chain_and_volumes(tmp_path, run_sh_mha, ["-t", "0", "-n", "20000"],
                                               ["-d", "1", "-gpus", "2", "-mp", mp])
    assert_same_pairs(chain, vols, listed)


@gpu
def test_volumes_resident_server(built, run_sh_mha, tmp_path):
    """-serve 1: the server keeps one producer context from job to job."""
    env = dict(os.environ, FROGMATCH_SOCKET=str(tmp_path / "fm.sock"), FROGMATCH_SERVE_IDLE="60")
    files = [surf3d_csvgz(m, str(tmp_path / f"points{i}"), ["-t", "0", "-n", "20000"]) for i, m in enumerate(run_sh_mha)]
    (tmp_path / "files.txt").write_text("".join(f + "\n" for f in files))
    (tmp_path / "vols.txt").write_text("".join(m + "\n" for m in run_sh_mha))
    run_match([str(tmp_path / "files.txt"), "-o", str(tmp_path / "chain.bin"), "-d", "1"])
    chain = pairsbin.parse(str(tmp_path / "chain.bin"))
    try:
        for k in range(2):
            run_match([str(tmp_path / "vols.txt"), "-o", str(tmp_path / f"served{k}.bin"), "-d", "1", "-surf3d", "-t 0 -n 20000",
                       "-serve", "1"], env=env)
            assert_same_pairs(chain, pairsbin.parse(str(tmp_path / f"served{k}.bin")), run_sh_mha)
    finally:
        subprocess.run([build.BIN, "-serve-stop"], env=env, timeout=60)
    assert not os.path.exists(tmp_path / "fm.sock")


@gpu
def test_bad_volume_named(built, run_sh_mha, tmp_path):
    """A compressed or unreadable .mha: exit 1, the file named."""
    comp = tmp_path / "comp.mha"
    comp.write_bytes(open(run_sh_mha[0], "rb").read().replace(b"CompressedData = False", b"CompressedData = True"))
    for bad in (str(comp), str(tmp_path / "missing.mha")):
        (tmp_path / "l.txt").write_text(f"{run_sh_mha[1]}\n{bad}\n")
        r = subprocess.run([build.BIN, str(tmp_path / "l.txt"), "-o", str(tmp_path / "o.bin")], capture_output=True, text=True,
                           timeout=300)
        assert r.returncode == 1 and bad in r.stderr, r.stderr


@gpu
def test_keypoint_list_without_libfrogsurf(built, golden_dir, tmp_path):
    """bin/match over keypoint files runs from a tree holding only bin/match and libfrogmatch.so."""
    (tmp_path / "bin").mkdir()
    (tmp_path / "frog_b200").mkdir()
    shutil.copy(build.BIN, tmp_path / "bin" / "match")
    shutil.copy(build.LIB, tmp_path / "frog_b200" / "libfrogmatch.so")
    r = subprocess.run([str(tmp_path / "bin" / "match"), os.path.join(golden_dir, "list_bin.txt"), "-o", str(tmp_path / "o.bin"),
                        "-d", "1"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert open(tmp_path / "o.bin", "rb").read() == open(os.path.join(golden_dir, "bin_runsh.pairs.bin"), "rb").read()


# ---- without a GPU --------------------------------------------------------------------------------------------

REFUSED = [["-s", "2"], ["-d", "100"], ["-m", "mask.mha"], ["-pad", "1"], ["-type", "2"], ["-json", "1"]]


@pytest.mark.parametrize("opt", REFUSED, ids=lambda o: o[0])
def test_surf3d_refusals_shared(built, tmp_path, opt):
    """An option bin/surf3d refuses is refused by -surf3d the same way (exit 7, same message), before any CUDA call."""
    (tmp_path / "l.txt").write_text(str(tmp_path / "v.mha") + "\n")
    a = subprocess.run([build.SURF_BIN, str(tmp_path / "v.mha")] + opt, capture_output=True, text=True)
    b = subprocess.run([build.BIN, str(tmp_path / "l.txt"), "-surf3d", " ".join(opt + ["-t", "0"])], capture_output=True, text=True)
    assert a.returncode == 7 and b.returncode == 7
    assert a.stderr == b.stderr and "needs a VTK image filter" in b.stderr
    assert b.stdout == ""


def test_surf3d_points_file_refused(built, tmp_path):
    (tmp_path / "l.txt").write_text(str(tmp_path / "v.mha") + "\n")
    r = subprocess.run([build.BIN, str(tmp_path / "l.txt"), "-surf3d", "-p pts.csv"], capture_output=True, text=True)
    assert r.returncode == 7 and "-p" in r.stderr


def test_match_does_not_link_libfrogsurf(built, tmp_path):
    """libfrogsurf.so is loaded at run time, only for lists that hold volumes; without it such a list fails clearly
    (before any CUDA call)."""
    r = subprocess.run(["readelf", "-d", build.BIN], capture_output=True, text=True)
    assert r.returncode == 0 and "libfrogmatch.so" in r.stdout and "libfrogsurf" not in r.stdout
    (tmp_path / "bin").mkdir()
    (tmp_path / "frog_b200").mkdir()
    shutil.copy(build.BIN, tmp_path / "bin" / "match")
    shutil.copy(build.LIB, tmp_path / "frog_b200" / "libfrogmatch.so")
    (tmp_path / "l.txt").write_text(str(tmp_path / "v.mha") + "\n")
    env = {k: v for k, v in os.environ.items() if k != "LD_LIBRARY_PATH"}
    r = subprocess.run([str(tmp_path / "bin" / "match"), str(tmp_path / "l.txt")], capture_output=True, text=True, env=env)
    assert r.returncode == 1 and "libfrogsurf.so" in r.stderr


def test_volume_plan(built, tmp_path):
    """The GPU plan counts a volume as -n keypoints (no CUDA call with -plan 1)."""
    v = tmp_path / "v.mha"
    surf.write_metaimage(str(v), np.zeros((8, 8, 8), np.int16))
    (tmp_path / "l.txt").write_text("".join(f"{v}\n" for _ in range(4)))
    r = subprocess.run([build.BIN, str(tmp_path / "l.txt"), "-plan", "1", "-surf3d", "-n 20000"], capture_output=True, text=True)
    assert r.returncode == 0 and "Planned GPUs : 1 (6 image pairs)" in r.stdout
