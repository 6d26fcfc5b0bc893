"""GPU: what the MetaImage encodings cost on the way from volumes to pairs.bin, on one B200.

    python scripts/gpu_metaimage_wall.py [--groups 32x256,8x400] [--out FILE]

The groups are gpu_volumes_wall.py's (V synthetic int16 volumes of size^3), each written in six encodings: raw .mha,
zlib level 1 and 6 as .mha and as .mhd + .zraw, and big-endian raw .mha.  Every file is read once before the timed
runs (page cache).  Per encoding:
  * the reader's time per volume through surf.read_metaimage, split into header, read, inflate and swap;
  * `bin/match vols.txt -surf3d "-t 0 -n 20000" -d 1` one-shot, and through a resident server (`-serve 1`) that one
    untimed call on the raw group started;
  * whether each pairs.bin equals the raw group's one-shot pairs.bin (names aside).
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from frog_b200 import build, surf  # noqa: E402
from gpu_surf_bench import bench_volume  # noqa: E402
from gpu_volumes_wall import run, same_pairs  # noqa: E402

SURF_OPTS = "-t 0 -n 20000"
ENCODINGS = {
    "raw_mha": dict(),
    "zlib1_mha": dict(compress=1),
    "zlib6_mha": dict(compress=6),
    "zlib1_mhd_zraw": dict(compress=1, data_file=True),
    "zlib6_mhd_zraw": dict(compress=6, data_file=True),
    "big_endian_mha": dict(byte_order=">"),
}


def volumes(n_vol, size):
    bases = [bench_volume(size, seed=100 + 8 * b) for b in range(4)]
    out = []
    for k in range(n_vol):
        rng = np.random.default_rng(1000 + k)
        v = np.roll(bases[k % 4], tuple(int(s) for s in rng.integers(-12, 13, 3)), (0, 1, 2))
        out.append(v + rng.integers(-4, 5, v.shape).astype(np.int16))
    return out


def write_encoding(d, vols, kw):
    os.makedirs(d)

    def one(k):
        ext = ".mhd" if kw.get("data_file") else ".mha"
        p = os.path.join(d, f"v{k}{ext}")
        args = dict(kw, data_file=f"v{k}.zraw") if kw.get("data_file") else kw
        surf.write_metaimage(p, vols[k], (0.75, 0.75, 0.75), (-100.0, -100.0, 5.0 * k), **args)
        return p

    with ThreadPoolExecutor(os.cpu_count()) as ex:  # zlib releases the GIL
        paths = list(ex.map(one, range(len(vols))))
    nbytes = 0
    for f in os.listdir(d):  # into the page cache
        nbytes += len(open(os.path.join(d, f), "rb").read())
    open(os.path.join(d, "vols.txt"), "w").write("".join(p + "\n" for p in paths))
    return paths, nbytes


def group(tmp, n_vol, size):
    vols = volumes(n_vol, size)
    res = dict(volumes=n_vol, size=size, encodings={})
    env = dict(os.environ, FROGMATCH_SOCKET=os.path.join(tmp, f"fm{n_vol}x{size}.sock"), FROGMATCH_SERVE_IDLE="300")
    gdir = os.path.join(tmp, f"g{n_vol}x{size}")
    ref = None
    try:
        for name, kw in ENCODINGS.items():
            d = os.path.join(gdir, name)
            paths, nbytes = write_encoding(d, vols, kw)
            phases = []
            for p in paths:
                ph = {}
                t = time.perf_counter()
                surf.read_metaimage(p, ph)
                ph["total_s"] = time.perf_counter() - t
                phases.append(ph)
            lst = os.path.join(d, "vols.txt")
            common = [build.BIN, lst, "-surf3d", SURF_OPTS, "-d", "1"]
            if ref is None:  # the raw group: starts the server, untimed
                run(common + ["-o", os.path.join(d, "warmup.bin"), "-serve", "1"], cwd=d, env=env)
            t_b = run(common + ["-o", os.path.join(d, "oneshot.bin")], cwd=d)
            t_c = run(common + ["-o", os.path.join(d, "served.bin"), "-serve", "1"], cwd=d, env=env)
            if ref is None:
                ref = os.path.join(d, "oneshot.bin")
            eq_b, n_match = same_pairs(ref, os.path.join(d, "oneshot.bin"))
            eq_c, _ = same_pairs(ref, os.path.join(d, "served.bin"))
            mean = {k: float(np.mean([ph[k] for ph in phases])) for k in phases[0]}
            res["encodings"][name] = dict(
                file_bytes=nbytes, read_per_volume_s=mean, read_max_s=float(max(ph["total_s"] for ph in phases)),
                oneshot_s=t_b, served_s=t_c, matches=n_match, oneshot_equals_raw=bool(eq_b), served_equals_raw=bool(eq_c))
            print(name, json.dumps(res["encodings"][name]), flush=True)
            for f in os.listdir(d):
                if not f.endswith(".bin"):
                    os.remove(os.path.join(d, f))
    finally:
        subprocess.run([build.BIN, "-serve-stop"], env=env, timeout=120)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--groups", default="32x256,8x400")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    out = dict(gpu=smi, host_cores=os.cpu_count(), page_cache="every file was read once before the timed runs",
               surf3d_options=SURF_OPTS, match_options="-d 1", groups=[])
    with tempfile.TemporaryDirectory() as tmp:
        for g in a.groups.split(","):
            n, s = (int(x) for x in g.split("x"))
            out["groups"].append(group(tmp, n, s))
    print(json.dumps(out))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(out, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
