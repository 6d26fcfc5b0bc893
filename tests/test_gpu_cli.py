"""GPU: the drop-in executable.  bin/match must write byte-identical pairs.bin files to the
reference binary on every golden case and on a fresh group matched by the reference here."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT
from frog_b200 import build, pairsbin, synth
from oracle import oracle as O

sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_ref_golden as rg  # noqa: E402

pytestmark = pytest.mark.gpu
CASES = sorted(json.load(open(os.path.join(ROOT, "tests", "golden", "manifest.json"))).items())


@pytest.mark.parametrize("name,case", CASES)
def test_cli_golden_bytes(built, golden_dir, tmp_path, name, case):
    out = str(tmp_path / "pairs.bin")
    r = subprocess.run([build.BIN, os.path.join(golden_dir, case["list"]), "-o", out] + case["args"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert f"Nb Match : {case['nb_match']}" in r.stdout and "Pairing... " in r.stdout
    golden = open(os.path.join(golden_dir, name + ".pairs.bin"), "rb").read()
    mine = open(out, "rb").read()
    if mine != golden:
        pytest.fail(str(pairsbin.diff(pairsbin.parse(golden), pairsbin.parse(mine))))


def test_cli_exact_engine_and_stats(built, golden_dir, tmp_path):
    out, stats = str(tmp_path / "p.bin"), str(tmp_path / "s.json")
    r = subprocess.run([build.BIN, os.path.join(golden_dir, "list_bin.txt"), "-o", out, "-d", "1", "-exact", "1",
                        "-stats", stats, "-gpus", "1"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(out, "rb").read() == open(os.path.join(golden_dir, "bin_runsh.pairs.bin"), "rb").read()
    s = json.load(open(stats))
    assert s["image_pairs"] == 6 and s["rows_exact"] == s["rows"]


def test_cli_default_output_name(built, golden_dir, tmp_path):
    r = subprocess.run([build.BIN, os.path.join(golden_dir, "list_bin.txt")], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0, r.stderr
    assert os.path.exists(tmp_path / "out_list_bin_4.bin")  # match.cpp:671


def test_cli_vs_reference_binary_fresh_group(built, tmp_path):
    """Config 1 of BASELINE.json: 2 keypoint files (~5k points, csv.gz), defaults -d 0.22 -d2 1.  Against the reference
    binary where oracle/_ref is built, else against its file and match count as recorded in tests/golden/ref."""
    lst = synth.write_group(str(tmp_path / "g"), "bank", 2, 5000, fmt="csv.gz")
    ref_out, out = str(tmp_path / "ref.bin"), str(tmp_path / "new.bin")
    new = subprocess.run([build.BIN, lst, "-o", out], capture_output=True, text=True)
    assert new.returncode == 0, new.stderr
    if os.path.exists(O.REF_BIN):
        ref = O.run_ref_binary([lst, "-o", ref_out])
        assert open(out, "rb").read() == open(ref_out, "rb").read()
        nb = [l for l in ref.stdout.splitlines() if l.startswith("Nb Match")][0]
    else:
        want = rg.load("fresh_group")[0]
        assert rg.pairs_digest(out) == want["pairs"]
        nb = want["nb_match_line"]
    assert nb in new.stdout


@pytest.mark.parametrize("gather", ["host", "nccl"])
def test_cli_two_gpus_gather(built, golden_dir, tmp_path, gather):
    """-gpus 2: image pairs sharded over two GPUs, lists merged on the host or gathered to GPU 0 over NCCL;
    either way the file is the reference's, byte for byte."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    out, stats = str(tmp_path / "p.bin"), str(tmp_path / "s.json")
    r = subprocess.run([build.BIN, os.path.join(golden_dir, "list_bin.txt"), "-o", out, "-d", "1", "-gpus", "2",
                        "-gather", gather, "-stats", stats], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(out, "rb").read() == open(os.path.join(golden_dir, "bin_runsh.pairs.bin"), "rb").read()
    s = json.load(open(stats))
    assert s["gpus"] == 2 and s["gather"] == gather


def test_cli_two_gpus_worker_processes(built, golden_dir, tmp_path):
    """-mp 1: one forked worker process per GPU over the shared arena; same bytes."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    out, stats = str(tmp_path / "p.bin"), str(tmp_path / "s.json")
    r = subprocess.run([build.BIN, os.path.join(golden_dir, "list_bin.txt"), "-o", out, "-d", "1", "-gpus", "2", "-mp", "1",
                        "-stats", stats], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(out, "rb").read() == open(os.path.join(golden_dir, "bin_runsh.pairs.bin"), "rb").read()
    s = json.load(open(stats))
    assert s["gpus"] == 2 and s["processes"] == 2


def test_cli_resident_server(built, golden_dir, tmp_path):
    """-serve 1: the command line runs inside a resident server that keeps the CUDA contexts warm; stdout, exit code
    and pairs.bin are those of a one-shot run (relative paths resolve against the CLIENT's directory)."""
    env = dict(os.environ, FROGMATCH_SOCKET=str(tmp_path / "fm.sock"), FROGMATCH_SERVE_IDLE="60")
    golden = open(os.path.join(golden_dir, "bin_runsh.pairs.bin"), "rb").read()
    try:
        for k in range(3):
            r = subprocess.run([build.BIN, os.path.join(golden_dir, "list_bin.txt"), "-o", f"served{k}.bin", "-d", "1", "-serve", "1"],
                               capture_output=True, text=True, env=env, cwd=tmp_path, timeout=180)
            assert r.returncode == 0, r.stderr
            assert "Pairing... " in r.stdout and "Nb Match : " in r.stdout and f"Output file : served{k}.bin" in r.stdout
            assert open(tmp_path / f"served{k}.bin", "rb").read() == golden
        r = subprocess.run([build.BIN, "/nonexistent/list.txt", "-serve", "1"], capture_output=True, text=True, env=env, timeout=60)
        assert r.returncode == 1 and "Bad argument" in r.stderr  # errors and exit codes travel back too
        # a different flag set through the same server
        r = subprocess.run([build.BIN, os.path.join(golden_dir, "list_bin.txt"), "-o", str(tmp_path / "sym.bin"), "-d", "1", "-sym",
                            "-serve", "1"], capture_output=True, text=True, env=env, timeout=60)
        assert r.returncode == 0, r.stderr
        assert open(tmp_path / "sym.bin", "rb").read() == open(os.path.join(golden_dir, "bin_sym.pairs.bin"), "rb").read()
    finally:
        subprocess.run([build.BIN, "-serve-stop"], env=env, timeout=60)
    assert not os.path.exists(tmp_path / "fm.sock")


def test_cli_distance_side_output(built, golden_dir, tmp_path):
    """-dists f: one float32 squared distance per emitted match, in pairs.bin block order, equal (0 ulp; the north star
    allows 2) to what the reference's own norm() returns for that pair (oracle/_ref/libmatch_ref.so)."""
    import numpy as np
    from frog_b200 import hostio
    out, dists = str(tmp_path / "p.bin"), str(tmp_path / "d.f32")
    lst = os.path.join(golden_dir, "list_bin.txt")
    r = subprocess.run([build.BIN, lst, "-o", out, "-d", "1", "-dists", dists], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(out, "rb").read() == open(os.path.join(golden_dir, "bin_runsh.pairs.bin"), "rb").read()
    pf = pairsbin.parse(out)
    d = np.fromfile(dists, np.float32)
    assert d.shape[0] == pf.n_matches() > 0
    files = [l.strip() for l in open(lst) if l.strip()]
    descs = [hostio.read_keypoints(f)[1] for f in files]
    ref = O.RefLib() if os.path.exists(O.REF_LIB) else None
    off = 0
    for i, j, m in pf.blocks:
        n = m.shape[0]
        want = (ref.distances(descs[i], descs[j], m[:, 0], m[:, 1]) if ref is not None
                else O.norm_matrix_numpy(descs[j][m[:, 1]], descs[i])[np.arange(n), m[:, 0]])
        assert np.array_equal(d[off:off + n].view(np.uint32), want.view(np.uint32))
        off += n
