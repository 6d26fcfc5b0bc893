"""GPU: wall time from MetaImage volumes to pairs.bin on one B200, three ways.

    python scripts/gpu_volumes_wall.py [--groups 32x256,8x400] [--out FILE]

  (a) run.sh's chain: one `bin/surf3d <vol> -t 0 -n 20000` process per volume, one after the other, then
      `bin/match list -d 1` over the .csv.gz files;
  (b) `bin/match vols.txt -surf3d "-t 0 -n 20000" -d 1`, one-shot;
  (c) the same command with `-serve 1`, timed after one warm-up call that starts the resident server.

Volumes: per group, V synthetic int16 volumes of size^3 (octant-seeded CT-like volumes as in gpu_surf_bench.py; four
bases per group, each volume a base shifted by its own offset plus its own noise, so no two volumes are alike), written
as .mha to a temporary directory and read once before timing: the three runs find them in the page cache.  The three
pairs.bin files must agree (names aside).  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from frog_b200 import build, pairsbin, surf  # noqa: E402
from gpu_surf_bench import bench_volume  # noqa: E402

SURF_OPTS = ["-t", "0", "-n", "20000"]


def run(cmd, **kw):
    t = time.perf_counter()
    r = subprocess.run(cmd, capture_output=True, text=True, **kw)
    if r.returncode != 0:
        raise RuntimeError(f"{cmd[:2]} failed: {r.stderr[-2000:]}")
    return time.perf_counter() - t


def same_pairs(a, b):
    pa, pb = pairsbin.parse(a), pairsbin.parse(b)
    return (len(pa.points) == len(pb.points)
            and all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(pa.points, pb.points))
            and [(i, j) for i, j, _ in pa.blocks] == [(i, j) for i, j, _ in pb.blocks]
            and all(np.array_equal(x, y) for (_, _, x), (_, _, y) in zip(pa.blocks, pb.blocks))), pa.n_matches()


def group(tmp, n_vol, size):
    d = os.path.join(tmp, f"g{n_vol}x{size}")
    os.makedirs(d)
    bases = [bench_volume(size, seed=100 + 8 * b) for b in range(4)]
    mhas = []
    for k in range(n_vol):
        rng = np.random.default_rng(1000 + k)
        v = np.roll(bases[k % 4], tuple(int(s) for s in rng.integers(-12, 13, 3)), (0, 1, 2))
        v = v + rng.integers(-4, 5, v.shape).astype(np.int16)
        p = os.path.join(d, f"v{k}.mha")
        surf.write_metaimage(p, v, (0.75, 0.75, 0.75), (-100.0, -100.0, 5.0 * k))
        mhas.append(p)
    del bases
    nbytes = sum(len(open(p, "rb").read()) for p in mhas)  # into the page cache
    vols = os.path.join(d, "vols.txt")
    open(vols, "w").write("".join(p + "\n" for p in mhas))

    # (a) the chain
    t_surf = 0.0
    files = []
    for k, p in enumerate(mhas):
        base = os.path.join(d, f"points{k}")
        t_surf += run([build.SURF_BIN, p, "-o", base] + SURF_OPTS, cwd=d)
        files.append(base + ".csv.gz")
    lst = os.path.join(d, "files.txt")
    open(lst, "w").write("".join(f + "\n" for f in files))
    t_match = run([build.BIN, lst, "-d", "1", "-o", os.path.join(d, "chain.bin")], cwd=d)
    # (b) one-shot
    stats = os.path.join(d, "stats.json")
    t_b = run([build.BIN, vols, "-surf3d", " ".join(SURF_OPTS), "-d", "1", "-o", os.path.join(d, "oneshot.bin"), "-stats", stats], cwd=d)
    st = json.load(open(stats))
    # (c) resident server
    env = dict(os.environ, FROGMATCH_SOCKET=os.path.join(d, "fm.sock"), FROGMATCH_SERVE_IDLE="120")
    try:
        t_warm = run([build.BIN, vols, "-surf3d", " ".join(SURF_OPTS), "-d", "1", "-o", os.path.join(d, "warmup.bin"), "-serve", "1"],
                     cwd=d, env=env)
        t_c = run([build.BIN, vols, "-surf3d", " ".join(SURF_OPTS), "-d", "1", "-o", os.path.join(d, "served.bin"), "-serve", "1"],
                  cwd=d, env=env)
    finally:
        subprocess.run([build.BIN, "-serve-stop"], env=env, timeout=120)
    eq_b, n_match = same_pairs(os.path.join(d, "chain.bin"), os.path.join(d, "oneshot.bin"))
    eq_c, _ = same_pairs(os.path.join(d, "chain.bin"), os.path.join(d, "served.bin"))
    for f in files + mhas:
        os.remove(f)
    return dict(volumes=n_vol, size=size, mha_bytes=nbytes, matches=n_match,
                a_chain_s=t_surf + t_match, a_surf3d_processes_s=t_surf, a_match_s=t_match,
                b_oneshot_s=t_b, c_served_s=t_c, c_warmup_call_s=t_warm,
                b_produce_s=st["produce_s"], b_produce_gpu_ms=st["produce_gpu_ms"], b_pairing_s=st["pairing_s"],
                oneshot_equals_chain=bool(eq_b), served_equals_chain=bool(eq_c))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--groups", default="32x256,8x400")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    out = dict(gpu=smi, page_cache="every .mha was read once before the timed runs", surf3d_options=" ".join(SURF_OPTS),
               match_options="-d 1", groups=[])
    with tempfile.TemporaryDirectory() as tmp:
        for g in a.groups.split(","):
            n, s = (int(x) for x in g.split("x"))
            out["groups"].append(group(tmp, n, s))
            print(json.dumps(out["groups"][-1]), flush=True)
    print(json.dumps(out))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(out, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
