"""Device groups (fm_group_*) at G = 1, 2, 4, 8 on the C4 group (bench.py's 200 x 20 000 iid images, all 19 900
pairs), at bench.py's flags (-d 1 -d2 0.8) and at FROG.py's (-d 1e10 -d2 1).

Per G and flag set, in one process:
  call_ms    host clock around a synchronous fm_group_match with FM_FLAG_DEVICE_ONLY (lists resident on the lead),
             after warm-up; median and min over --reps calls
  member_ms  the longest member's CUDA-event match time (fm_result_stats ms_total of the group result), so
             call_ms - member_ms is what the gather (and the host) add
  fetch_ms   fm_result_fetch of the lists to pinned host memory
  links_ms   fm_links_build on the lead (its CUDA-event time, and the host clock around the call)
and checks that the counts, the lists on the lead and the links are byte-identical to G = 1 (compared on the lead).
Records the card name and power limit.

    python scripts/gpu_group_scale.py --out DIR [--gpus 1,2,4,8] [--reps 5] [--same-device]

--same-device puts every member on GPU 0 (debug option "group_repeat"): no scaling, but the sharding and the gather
(as device-local stores) run on a box with one GPU, and the byte-identity checks hold at full size.
"""
from __future__ import annotations

import argparse
import ctypes as C
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

from frog_b200 import capi, synth  # noqa: E402
from frog_b200 import dist as fdist  # noqa: E402

FLAG_SETS = {"bench_d1_d2_0.8": (1.0, 0.8), "frog_d1e10_d2_1": (1e10, 1.0)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return [l.strip() for l in q.stdout.splitlines() if l.strip()]


def device_links(res, pf, ps, dev, n_points):
    """fm_links_build on the result; returns (offsets, links) as device tensors on the lead, build ms, host ms."""
    L = res._m._L
    h = C.c_void_p()
    t0 = time.perf_counter()
    res._m._check(L.fm_links_build(res._h, capi._ptr(pf), capi._ptr(ps), None, C.byref(h)))
    host_ms = (time.perf_counter() - t0) * 1e3
    try:
        L.fm_links_device_offsets.restype = C.c_void_p
        L.fm_links_device_data.restype = C.c_void_p
        total = int(L.fm_links_total(h))
        off_ptr, data_ptr = L.fm_links_device_offsets(h), L.fm_links_device_data(h)
        off = fdist.as_torch_u32(off_ptr, 2 * (n_points + 1), dev).clone()
        data = fdist.as_torch_u32(data_ptr, 2 * total, dev).clone()
        return off, data, float(L.fm_links_build_ms(h)), host_ms
    finally:
        L.fm_links_free(h)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--images", type=int, default=200)
    ap.add_argument("--points", type=int, default=20000)
    ap.add_argument("--same-device", action="store_true")
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    n_dev = torch.cuda.device_count()
    gs = [g for g in (int(x) for x in a.gpus.split(",")) if g <= n_dev or (a.same_device and n_dev)]
    if a.same_device:
        capi.debug_set_option("group_repeat", 1)
    if not gs or gs[0] != 1:
        raise SystemExit("needs G = 1 first (the reference of the byte-identity checks) and a CUDA device")
    images = [synth.make("iid", a.points, i) for i in range(a.images)]
    pf = np.array([i for i in range(a.images) for j in range(i + 1, a.images)], np.uint32)
    ps = np.array([j for i in range(a.images) for j in range(i + 1, a.images)], np.uint32)
    dev = torch.device("cuda", 0)
    out = {"cards": card(), "visible_gpus": n_dev, "workload": f"c4: {a.images} images x {a.points} iid keypoints (D=48), "
           f"all {len(pf)} pairs row-major", "same_device": a.same_device, "reps": a.reps, "warmup": a.warmup, "runs": {}}
    print(json.dumps(out["cards"]), flush=True)
    ref = {}
    for name, (dist, ratio) in FLAG_SETS.items():
        out["runs"][name] = {}
        for G in gs:
            g = capi.Group([0] * G if a.same_device else list(range(G)))
            t0 = time.perf_counter()
            for i, k in enumerate(images):
                g.upload_raw(i, k.desc.ctypes.data, k.scale.ctypes.data, k.lap.ctypes.data, k.n, k.desc.shape[1])
            g.synchronize()
            upload_s = time.perf_counter() - t0
            for _ in range(a.warmup):
                g.match(pf, ps, dist, ratio, device_only=True).free()
            times, member = [], []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                res = g.match(pf, ps, dist, ratio, device_only=True)
                times.append((time.perf_counter() - t0) * 1e3)
                member.append(res.stats()["ms_total"])
                res.free()
            res = g.match(pf, ps, dist, ratio, device_only=True)
            total = int(res.total)
            cptr, pptr = res.device_pointers()
            counts = fdist.as_torch_u32(cptr, len(pf), dev).clone()
            lists = fdist.as_torch_u32(pptr, 2 * total, dev).clone()
            off, links, links_ms, links_host_ms = device_links(res, pf, ps, dev, a.images * a.points)
            t0 = time.perf_counter()
            res.fetch()
            fetch_ms = (time.perf_counter() - t0) * 1e3
            st = res.stats()
            res.free()
            g.close()
            row = {"G": G, "matches": total, "list_bytes": 8 * total, "upload_s": upload_s,
                   "call_ms_median": statistics.median(times), "call_ms_min": min(times), "call_ms": times,
                   "member_ms_median": statistics.median(member), "member_ms": member,
                   "gather_and_host_ms_median": statistics.median([t - m for t, m in zip(times, member)]),
                   "fetch_ms": fetch_ms, "links_build_ms": links_ms, "links_host_ms": links_host_ms,
                   "kernel_launches": st["kernel_launches"], "descriptor_pairs": st["descriptor_pairs"]}
            if G == 1:
                ref[name] = (counts, lists, off, links)
                row["identical_to_G1"] = None
            else:
                rc, rl, ro, rk = ref[name]
                row["identical_to_G1"] = {"counts": bool(torch.equal(counts, rc)), "lists": bool(torch.equal(lists, rl)),
                                          "link_offsets": bool(torch.equal(off, ro)), "links": bool(torch.equal(links, rk))}
            row["speedup_vs_G1"] = out["runs"][name]["1"]["call_ms_median"] / row["call_ms_median"] if G > 1 else 1.0
            out["runs"][name][str(G)] = row
            print(json.dumps({name: {k: v for k, v in row.items() if k not in ("call_ms", "member_ms")}}), flush=True)
            del counts, lists, off, links
        ref.pop(name, None)
        torch.cuda.empty_cache()
    with open(os.path.join(a.out, "group_scale_same_device.json" if a.same_device else "group_scale.json"), "w") as f:
        json.dump(out, f, indent=1)
    bad = [(n, G) for n, runs in out["runs"].items() for G, r in runs.items()
           if r["identical_to_G1"] is not None and not all(r["identical_to_G1"].values())]
    if bad:
        raise SystemExit(f"lists or links differ from G = 1: {bad}")


if __name__ == "__main__":
    main()
