"""Row tables (FM_FLAG_ROW_TABLE) and fm_result_select on one GPU: what a table-mode call costs over a plain fm_match,
and what re-deciding it at another setting costs against scoring again.

Workloads:
  c4        bench.py's C4 group (200 x 20 000 iid keypoints, D = 48, all 19 900 pairs row-major) on the tensor cores
  raw_haar  surf3d -type 1 raw Haar descriptors as the producer writes them (|desc|^2 far above 16: the exact FP32
            engine), --haar-volumes textured volumes of --haar-size^3 voxels, at most --haar-points keypoints each,
            radius 3 (d = 648), all pairs row-major

For each workload and each call flag set -- bench.py's (-d 1 -d2 0.8) and FROG.py's (-d 1e10 -d2 1) -- in one process:
  plain_ms   host clock around a synchronous fm_match with FM_FLAG_DEVICE_ONLY (lists resident), after warm-up
  table_ms   the same call with FM_FLAG_ROW_TABLE (includes allocating and freeing the table: each call owns its table)
  select_ms  host clock around a synchronous device-only fm_result_select of that table at each driver setting
             (reference default 0.22/1, run.sh 1/1, FROG.py 1e10/1, desk UI 0.5/0.998, bench 1/0.8), and its
             CUDA-event time (fm_result_stats ms_total)
  fresh_ms   the plain fm_match at that setting, which select replaces
and checks that every selected result's counts and lists (device views) and distances are byte-identical to the fresh
call's.  Medians over --reps calls.  Records the card name and power limit, read in the same process.

    python scripts/gpu_select_bench.py --out DIR [--reps 5] [--workloads c4,raw_haar]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from frog_b200 import capi, surf, synth  # noqa: E402
from frog_b200 import dist as fdist  # noqa: E402

FLAG_SETS = {"bench_d1_d2_0.8": (1.0, 0.8), "frog_d1e10_d2_1": (1e10, 1.0)}
SETTINGS = {"reference_0.22_1": (0.22, 1.0), "run_sh_1_1": (1.0, 1.0), "frog_py_1e10_1": (1e10, 1.0),
            "desk_0.5_0.998": (0.5, 0.998), "bench_1_0.8": (1.0, 0.8)}
# raw Haar distances are sums of squared raw Haar responses, far above 1: these settings also accept some of its rows
HAAR_SETTINGS = {"d_1e4_ratio_0.9": (1e4, 0.9), "d_1e5_ratio_1": (1e5, 1.0)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return [l.strip() for l in q.stdout.splitlines() if l.strip()]


def c4_images(n_images, n_points):
    return [(k.desc, k.scale, k.lap) for k in (synth.make("iid", n_points, i) for i in range(n_images))]


def haar_images(n_volumes, size, blobs, n_points):
    out = []
    for k in range(n_volumes):
        v = synth.make_volume((size, size, size), 60 + 10 * k, blobs_per_mvox=blobs, texture=250.0)
        pts, desc, _ = surf.run(v, descriptor_type=1, radius=3, number_of_points=n_points)
        out.append((np.ascontiguousarray(desc.reshape(len(pts), -1), np.float32), pts["scale"].astype(np.float32),
                    pts["laplacian"].astype(np.float32)))
    return out


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    times, out = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        times.append((time.perf_counter() - t0) * 1e3)
    return times, out


def device_snapshot(res, n_pairs, dev):
    """Counts, lists and distances of a device-only result, as device tensors (fetched distances: host bytes)."""
    res.wait()
    cptr, pptr = res.device_pointers()
    counts = fdist.as_torch_u32(cptr, n_pairs, dev).clone()
    lists = fdist.as_torch_u32(pptr, 2 * int(res.total), dev).clone()
    res.fetch()
    dist = b"".join(res.distances(p).tobytes() for p in range(n_pairs))
    return counts, lists, dist


def run_workload(m, name, images, reps, warmup, settings):
    n = len(images)
    pf = np.array([i for i in range(n) for j in range(i + 1, n)], np.uint32)
    ps = np.array([j for i in range(n) for j in range(i + 1, n)], np.uint32)
    dev = torch.device("cuda", 0)
    m.clear()
    for i, (d, s, l) in enumerate(images):
        m.upload(i, d, s, l)
    out = {"images": n, "points": [int(len(im[1])) for im in images], "d": int(images[0][0].shape[1]), "pairs": len(pf),
           "runs": {}}
    for fname, (dist, ratio) in FLAG_SETS.items():
        def plain():
            r = m.match(pf, ps, dist, ratio, device_only=True)
            st = r.stats()
            r.free()
            return st

        def table():
            r = m.match(pf, ps, dist, ratio, device_only=True, row_table=True)
            st = r.stats()
            r.free()
            return st

        plain_t, plain_st = timed(plain, reps, warmup)
        table_t, table_st = timed(table, reps, warmup)
        tab = m.match(pf, ps, dist, ratio, device_only=True, row_table=True)
        rows = tab.row_offset(len(pf))
        row = {"plain_ms_median": statistics.median(plain_t), "plain_ms": plain_t, "plain_event_ms": plain_st["ms_total"],
               "plain_two_phase_batches": plain_st["two_phase_batches"], "plain_rows_rejected_early": plain_st["rows_rejected_early"],
               "table_ms_median": statistics.median(table_t), "table_ms": table_t, "table_event_ms": table_st["ms_total"],
               "table_over_plain": statistics.median(table_t) / statistics.median(plain_t),
               "rows": rows, "table_bytes": 12 * rows, "select": {}}
        for sname, (sd, sr) in settings.items():
            def select():
                r = tab.select(sd, sr, device_only=True)
                st = r.stats()
                r.free()
                return st

            sel_t, sel_st = timed(select, reps, warmup)
            fresh_t, _ = timed(lambda: plain_at(m, pf, ps, sd, sr), reps, warmup)
            fresh = m.match(pf, ps, sd, sr, device_only=True, distances=True)
            want = device_snapshot(fresh, len(pf), dev)
            total = int(fresh.total)
            fresh.free()
            sel = tab.select(sd, sr, device_only=True, distances=True)
            got = device_snapshot(sel, len(pf), dev)
            sel.free()
            same = {"counts": bool(torch.equal(got[0], want[0])), "lists": bool(torch.equal(got[1], want[1])),
                    "distances": got[2] == want[2]}
            del got, want
            row["select"][sname] = {"setting": [sd, sr], "matches": total, "select_ms_median": statistics.median(sel_t),
                                    "select_ms": sel_t, "select_event_ms": sel_st["ms_total"],
                                    "fresh_ms_median": statistics.median(fresh_t), "fresh_ms": fresh_t,
                                    "fresh_over_select": statistics.median(fresh_t) / statistics.median(sel_t),
                                    "identical_to_fresh": same}
            print(json.dumps({name: {fname: {sname: {k: v for k, v in row["select"][sname].items()
                                                      if k not in ("select_ms", "fresh_ms")}}}}), flush=True)
        tab.free()
        torch.cuda.empty_cache()
        out["runs"][fname] = row
        print(json.dumps({name: {fname: {k: v for k, v in row.items() if k not in ("plain_ms", "table_ms", "select")}}}),
              flush=True)
    return out


def plain_at(m, pf, ps, dist, ratio):
    r = m.match(pf, ps, dist, ratio, device_only=True)
    r.free()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--workloads", default="c4,raw_haar")
    ap.add_argument("--images", type=int, default=200)
    ap.add_argument("--points", type=int, default=20000)
    ap.add_argument("--haar-volumes", type=int, default=8)
    ap.add_argument("--haar-size", type=int, default=192)
    ap.add_argument("--haar-blobs", type=float, default=4000.0, help="blobs per million voxels of the volumes")
    ap.add_argument("--haar-points", type=int, default=4000)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    out = {"cards": card(), "reps": a.reps, "warmup": a.warmup, "workloads": {}}
    print(json.dumps(out["cards"]), flush=True)
    m = capi.Matcher(0)
    try:
        for w in a.workloads.split(","):
            if w == "c4":
                images = c4_images(a.images, a.points)
                desc = f"c4: {a.images} images x {a.points} iid keypoints (D=48), all pairs row-major"
            elif w == "raw_haar":
                images = haar_images(a.haar_volumes, a.haar_size, a.haar_blobs, a.haar_points)
                desc = (f"raw_haar: surf3d -type 1 -r 3 raw Haar descriptors (as written) of {a.haar_volumes} textured "
                        f"{a.haar_size}^3 volumes ({a.haar_blobs:g} blobs per Mvoxel), at most {a.haar_points} keypoints "
                        f"each, all pairs row-major: exact FP32 engine")
            else:
                raise SystemExit(f"unknown workload {w!r}")
            settings = dict(SETTINGS, **HAAR_SETTINGS) if w == "raw_haar" else SETTINGS
            out["workloads"][w] = run_workload(m, w, images, a.reps, a.warmup, settings)
            out["workloads"][w]["workload"] = desc
    finally:
        m.close()
    out["cards_after"] = card()
    with open(os.path.join(a.out, "select_bench.json"), "w") as f:
        json.dump(out, f, indent=1)
    bad = [(w, f, s) for w, wr in out["workloads"].items() for f, fr in wr["runs"].items()
           for s, sr in fr["select"].items() if not all(sr["identical_to_fresh"].values())]
    if bad:
        raise SystemExit(f"selected lists differ from fresh calls: {bad}")


if __name__ == "__main__":
    main()
