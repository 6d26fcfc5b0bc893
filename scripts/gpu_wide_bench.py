"""Wide tensor-core path (descriptor lengths d != 48) against the exact engine on one GPU.

Workload per descriptor length d: 10 images x 20 000 keypoints with SURF3D scale and laplacian distributions
(frog_b200.synth), L2-normalised descriptors of length d drawn `bank`-style (shared prototypes + noise, so true matches
exist), all 45 image pairs, at -d 1 -d2 0.8 and -d 1 -d2 1.  Per run: descriptor pairs/s of both engines (the wide path
and FM_FLAG_FORCE_EXACT, CUDA-event time of the whole call), the kernel phase times, the executed tensor-core rate
(2 K_pad x scored_pairs over the wide scoring kernel's time), and whether both engines' match lists are identical.

    python scripts/gpu_wide_bench.py --out profiles/r7_wide_bench.json [--lengths 24,192,648,1000,3000]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from frog_b200 import capi, synth  # noqa: E402


def group(d: int, n_images: int, n: int, seed: int, noise: float = 0.1, outliers: float = 0.1):
    rng = np.random.default_rng(seed)

    def unit(x):
        x /= np.maximum(np.linalg.norm(x, axis=1, keepdims=True), 1e-30)
        return x

    proto = unit(rng.standard_normal((2 * n, d), dtype=np.float32))
    pscale = synth._scales(rng, 2 * n)
    plap = rng.integers(0, 2, 2 * n).astype(np.float32)
    out = []
    for _ in range(n_images):
        pick = rng.permutation(2 * n)[:n]
        desc = unit(proto[pick] + np.float32(noise / np.sqrt(d)) * rng.standard_normal((n, d), dtype=np.float32))
        o = rng.uniform(size=n) < outliers
        desc[o] = unit(rng.standard_normal((int(o.sum()), d), dtype=np.float32))
        scale = (pscale[pick] * (1.0 + rng.uniform(-0.03, 0.03, n))).astype(np.float32)
        out.append((np.ascontiguousarray(desc, np.float32), scale, plap[pick].copy()))
    return out


def gpu_info() -> dict:
    info = {}
    try:
        import torch
        info["card"] = torch.cuda.get_device_name(0)
    except Exception as e:  # torch is only used for the name
        info["card"] = f"unknown ({e})"
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, plim, sm, smax = [x.strip() for x in q.split(",")]
        info.update(smi_name=name, power_limit=plim, sm_clock=sm, sm_clock_max=smax)
    except Exception as e:
        info["nvidia_smi"] = f"unavailable ({e})"
    return info


def run(m, pf, ps, thr, rat, force_exact):
    res = m.match(pf, ps, thr, rat, force_exact=force_exact)
    lists = res.all_pairs()
    st = res.stats()
    res.free()
    return lists, st


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--lengths", default="24,192,648,1000,3000")
    ap.add_argument("--images", type=int, default=10)
    ap.add_argument("--points", type=int, default=20000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    pairs = [(i, j) for i in range(a.images) for j in range(i + 1, a.images)]
    pf, ps = [p[0] for p in pairs], [p[1] for p in pairs]
    m = capi.Matcher(0)
    result = dict(workload=f"{a.images} images x {a.points} keypoints, {len(pairs)} pairs, bank-style unit descriptors",
                  gpu=gpu_info(), version=capi.version(), runs=[])
    for d in [int(x) for x in a.lengths.split(",")]:
        t0 = time.time()
        images = group(d, a.images, a.points, seed=d)
        m.clear()
        for i, (x, s, l) in enumerate(images):
            m.upload(i, x, s, l)
        del images
        kpad = (d + 63) // 64 * 64
        for thr, rat in [(1.0, 0.8), (1.0, 1.0)]:
            run(m, pf, ps, thr, rat, False)  # warm-up
            wide = []
            for _ in range(a.reps):
                lists_w, st = run(m, pf, ps, thr, rat, False)
                wide.append(st)
            lists_x, stx = run(m, pf, ps, thr, rat, True)
            same = len(lists_w) == len(lists_x) and all(np.array_equal(g, w) for g, w in zip(lists_w, lists_x))
            best = min(wide, key=lambda s: s["ms_total"])
            rec = dict(
                d=d, k_pad=kpad, dist=thr, ratio=rat, identical=bool(same), matches=int(sum(len(x) for x in lists_w)),
                descriptor_pairs=best["descriptor_pairs"], scored_pairs=best["scored_pairs"],
                rows=best["rows"], rows_exact=best["rows_exact"], candidates=best["candidates"],
                rows_rejected_early=best["rows_rejected_early"],
                wide_ms_total=best["ms_total"], wide_ms_score=best["ms_score"], wide_ms_rescore=best["ms_rescore"],
                wide_ms_exact=best["ms_exact"], wide_ms_compact=best["ms_compact"],
                wide_ms_total_all=[s["ms_total"] for s in wide],
                exact_ms_total=stx["ms_total"], exact_ms_exact=stx["ms_exact"],
                wide_pairs_per_s=best["descriptor_pairs"] / (best["ms_total"] * 1e-3),
                exact_pairs_per_s=stx["descriptor_pairs"] / (stx["ms_total"] * 1e-3),
                speedup=stx["ms_total"] / best["ms_total"],
                executed_tflops=2.0 * kpad * best["scored_pairs"] / (best["ms_score"] * 1e-3) / 1e12,
            )
            result["runs"].append(rec)
            print(json.dumps(rec), flush=True)
        print(f"d={d}: {time.time() - t0:.1f} s", file=sys.stderr, flush=True)
    m.close()
    result["all_identical"] = all(r["identical"] for r in result["runs"])
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps(dict(all_identical=result["all_identical"],
                          speedups={f'{r["d"]}/{r["ratio"]}': round(r["speedup"], 1) for r in result["runs"]})))


if __name__ == "__main__":
    main()
