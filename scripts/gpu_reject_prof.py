"""Per-launch kernel times of two-phase scoring on 5.52 M rows, and the reject pass's work counted from the bands.

    python scripts/gpu_reject_prof.py [--lib PATH] [--label NAME] [--out FILE.json] [--counts-only]

24 iid images of 20 000 keypoints, all 276 pairs in one call, two-phase scoring forced (-d 1 -d2 0.8, the C4 gates):
2 warm-up calls, then 5 calls under torch.profiler with CUDA activities.  Prints and writes one JSON object: µs per
launch of every kernel, the card, its power limit and SM clocks (nvidia-smi, read right after the profiled calls), and
from a numpy replay of the reference's gates over the same images:
  * TMA operand bytes per launch: per 512-row unit with a step, its 16 KB row-operand tiles (one per 128-row quarter
    with rows: 1 to 4), plus 32 KB per 256-column step;
  * the number of units and steps, and per epilogue warp and step its four 128-column rounds (one per quarter's fill)
    split into skipped (no row of the warp has a column there), interior (every row of the warp accepts all 128
    columns) and edge (masked per score).
--lib points at another build of libfrogmatch.so, so that two builds can be alternated in one session.
--counts-only skips the GPU and prints the replay alone.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from frog_b200 import capi, synth  # noqa: E402

N_IMAGES, N_POINTS, THR, RATIO = 24, 20000, 1.0, 0.8
UNIT, TILE_ROWS, WARP_ROWS, STEP, ROUND = 512, 128, 32, 256, 128  # reject-pass unit = four 128-row quarters
OP_TILE_BYTES, STEP_BYTES = 16384, 32768


def _sorted_view(kp):
    """(scale, laplacian) in the library's sorted order: by the laplacian's top 16 pattern bits, then by scale."""
    s, lap = kp.scale, np.where(kp.lap == 0, np.float32(0), kp.lap).astype(np.float32)
    order = np.lexsort((s.view(np.uint32), lap.view(np.uint32) >> 16))
    return s[order], lap[order]


def _first_true(pred, lo, hi):
    lo, hi = lo.copy(), hi.copy()
    while np.any(lo < hi):
        act = lo < hi
        m = (lo + hi) >> 1
        p = pred(np.where(act, m, 0)) & act
        lo = np.where(act & ~p, m + 1, lo)
        hi = np.where(p, m, hi)
    return lo


def bands(col, row):
    """The reference's scale and laplacian gates as sorted column intervals [lo, hi) per sorted row."""
    sc, lc = _sorted_view(col)
    sr, lr = _sorted_view(row)
    lo = np.zeros(sr.shape[0], np.int64)
    hi = np.zeros(sr.shape[0], np.int64)
    for lap in np.unique(lr):
        rows = np.nonzero(lr == lap)[0]
        cls = np.nonzero(lc == lap)[0]
        if cls.size == 0:
            continue
        beg, end = int(cls[0]), int(cls[-1]) + 1
        x = sr[rows]
        b = np.full(rows.size, beg, np.int64)
        e = np.full(rows.size, end, np.int64)
        l0 = _first_true(lambda m: ~((x / sc[m]).astype(np.float64) > 1.3), b, e)
        h0 = _first_true(lambda m: (sc[m] / x).astype(np.float64) > 1.3, l0, e)
        lo[rows], hi[rows] = l0, np.maximum(h0, l0)
    return lo, hi


def replay(kps, pf, ps):
    """TMA bytes, steps and the epilogue's round kinds of one reject-pass launch over the pairs (pf: columns)."""
    tot = {"tma_operand_bytes_per_launch": 0, "units": 0, "steps": 0, "rounds_skipped": 0, "rounds_interior": 0,
           "rounds_edge": 0}
    for i, j in zip(pf, ps):
        lo, hi = bands(kps[i], kps[j])
        n = lo.shape[0]
        units = (n + UNIT - 1) // UNIT
        pad = units * UNIT - n
        lo = np.concatenate([lo, np.zeros(pad, np.int64)]).reshape(units, UNIT // WARP_ROWS, WARP_ROWS)
        hi = np.concatenate([hi, np.zeros(pad, np.int64)]).reshape(units, UNIT // WARP_ROWS, WARP_ROWS)
        ok = hi > lo
        big = np.int64(1) << 40
        cmin = np.where(ok, lo, big).min(2)    # [unit, 32-row group]
        cmax = np.where(ok, hi, 0).max(2)
        imin = np.where(ok, lo, 0).max(2)
        imax = np.where(ok, hi, big).min(2)
        umin, umax = cmin.min(1), cmax.max(1)
        has = umax > umin
        step0 = np.where(has, umin // STEP, 0)
        nst = np.where(has, (umax + STEP - 1) // STEP - step0, 0)
        tot["units"] += int(has.sum())
        tot["steps"] += int(nst.sum())
        tiles = np.minimum(UNIT // TILE_ROWS, (n - np.arange(units) * UNIT + TILE_ROWS - 1) // TILE_ROWS)  # quarters with rows
        tot["tma_operand_bytes_per_launch"] += int((tiles * has).sum()) * OP_TILE_BYTES + int(nst.sum()) * STEP_BYTES
        k = np.arange(int(nst.max()) if nst.size else 0)
        live = k[None, :] < nst[:, None]                       # [unit, step]
        for c in range(STEP // ROUND):  # the 32-row groups are the (quarter, lane quadrant) pairs: one fill each
            c0 = ((step0[:, None] + k[None, :]) * STEP + c * ROUND)[:, :, None]  # [unit, step, 1]
            need = (c0 < cmax[:, None, :]) & (c0 + ROUND > cmin[:, None, :])    # [unit, step, group]
            inter = (c0 >= imin[:, None, :]) & (c0 + ROUND <= imax[:, None, :])
            lv = np.broadcast_to(live[:, :, None], need.shape)
            tot["rounds_skipped"] += int((lv & ~need).sum())
            tot["rounds_interior"] += int((lv & need & inter).sum())
            tot["rounds_edge"] += int((lv & need & ~inter).sum())
    r = tot["rounds_skipped"] + tot["rounds_interior"] + tot["rounds_edge"]
    for key in ("skipped", "interior", "edge"):
        tot[f"frac_{key}"] = tot[f"rounds_{key}"] / max(r, 1)
    return tot


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks_event_reasons.sw_power_cap"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        return dict(zip(q.split(","), (x.strip() for x in out[0].split(",")))) if out else {}
    except (OSError, subprocess.SubprocessError):
        return {}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=capi.LIB_PATH)
    ap.add_argument("--label", default="")
    ap.add_argument("--out")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--counts-only", action="store_true")
    args = ap.parse_args()

    kps = [synth.make("iid", N_POINTS, i) for i in range(N_IMAGES)]
    pf = [i for i in range(N_IMAGES) for j in range(i + 1, N_IMAGES)]
    ps = [j for i in range(N_IMAGES) for j in range(i + 1, N_IMAGES)]
    out = {"label": args.label, "lib": os.path.basename(args.lib), "rows_per_launch": N_POINTS * len(pf)}
    out.update(replay(kps, pf, ps))
    if not args.counts_only:
        import torch
        from torch.profiler import ProfilerActivity, profile

        capi.LIB_PATH = os.path.abspath(args.lib)
        m = capi.Matcher(0)
        for i, k in enumerate(kps):
            m.upload(i, k.desc, k.scale, k.lap)
        capi.debug_set_option("two_phase", 1)
        try:
            for _ in range(args.warmup):
                m.match(pf, ps, THR, RATIO).free()
            m.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.calls):
                    m.match(pf, ps, THR, RATIO).free()
                m.synchronize()
            st = m.stats()
        finally:
            capi.debug_set_option("two_phase", -1)
            m.close()
        assert st["two_phase_batches"] >= 1, "two-phase scoring did not run"
        out["card"] = card()
        out["torch_device"] = torch.cuda.get_device_name(0)
        kern = {}
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            if t > 0:
                kern[e.key[:100]] = {"count": e.count, "us_per_launch": round(t / args.calls, 1)}
        out["kernels"] = kern
        rj = [v for k, v in kern.items() if "reject_kernel" in k]
        if rj:
            us = rj[0]["us_per_launch"]
            out["reject_us_per_launch"] = us
            out["tma_gb_per_s"] = out["tma_operand_bytes_per_launch"] / (us * 1e-6) / 1e9
            out["sm_cycles_per_step"] = us * 1e-6 * float(out["card"].get("clocks.max.sm", "0 MHz").split()[0]) * 1e6 \
                * min(148, out["units"]) / max(out["steps"], 1)
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
