#!/usr/bin/env python
"""bench.py -- descriptor pairs/sec and match wall-time of the keypoint-matching hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c4|c3|c2|c1|dense]
                    [--dump-outputs DIR]

A step = one pass of the hot path (match.cpp:638-652: every image pair of a group through ComputeMatches)
over ONE synthetic keypoint group.  Default workload: BASELINE.json configs[3], the configuration the
north star is quoted on -- 200 images x 20 000 keypoints, random SURF3D-format descriptors (`iid` set,
SURVEY.md 8d), -d 1 -d2 0.8, all 19 900 image pairs = 7.96e12 descriptor pairs per step.

N > 1 is STRONG scaling of that one group: every rank holds all images (replicated, uploaded over its own
PCIe link), the image pairs are sharded over the ranks longest-processing-time-first (frog_b200.dist.shard_pairs,
the loop match.cpp:638-652 runs under OpenMP), no data-path collective; only the compacted match lists travel,
exact-size, to rank 0 over NCCL (NVLink).

One JSON line on rank 0:
  value     descriptor pairs/s, keypoints resident in HBM when the timed region starts (lists end on rank 0's GPU)
  e2e       the same through the C ABI from pinned HOST buffers: per step every image crosses PCIe once (rank r uploads
            images r, r+N, ...) and reaches the other GPUs by an NCCL all-gather over NVLink, then preparation + matching +
            list gather + D2H of all lists to rank 0's host memory
  roofline  tensor-core FLOP rate of the scoring kernel (96 FLOP per descriptor pair, DESIGN.md 4)
  wall      `bin/match` (the drop-in executable) process start -> exit on the same group at N GPUs, .bin and .csv.gz
  cpu_baseline  the verbatim reference match.cpp (oracle/_ref/match_ref) on this box's cores (N = 1 only)
`--impl reference` times that reference binary alone (rank 0), on images of the workload's real size.
"""
from __future__ import annotations

import argparse
import collections
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (images per group, keypoints per image, set, dist, ratio)
    "c1": (2, 5000, "bank", 0.22, 1.0),
    "c2": (10, 20000, "iid", 1.0, 1.0),
    "c3": (50, 50000, "iid", 1.0, 1.0),
    "c4": (200, 20000, "iid", 1.0, 0.8),
    # every keypoint in one laplacian class and at one scale: no column is gated out, the scoring kernel
    # executes every algorithmic pair (scored_fraction 1.0)
    "dense": (10, 20000, "dense", 1.0, 1.0),
}
FLOP_PER_PAIR = 96.0  # 2 * D, D = 48 (SURVEY.md 8d)
METRIC = "descriptor pairs/sec (keypoint matching, match.cpp ComputeMatches)"


def measured_traffic(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum of one scoring-kernel launch, from the committed ncu capture
    of this workload (profiles/); None for workloads that were not captured."""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            j = json.load(open(p))
            if j.get("workload") == workload:
                return float(j["dram_bytes_read"] + j["dram_bytes_write"])
    return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["bf16_tflops"]), float(j["hbm_gbs"]), "measured"
    return 1590.0, 6650.0, "fallback"


def workload_name(w, gpus):
    n_img, n_pts, kind, dist, ratio = WORKLOADS[w]
    s = (f"{w}: {n_img} images x {n_pts} keypoints, {kind} SURF3D descriptors (D=48), -d {dist:g} -d2 {ratio:g}, "
         f"all {n_img * (n_img - 1) // 2} image pairs of ONE group")
    if gpus > 1:
        s += f", sharded over {gpus} GPUs (images replicated, match lists gathered to rank 0 over NCCL)"
    return s


# --------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the unmodified reference binary on a bounded sample of the workload


def run_reference(list_path, dist, ratio, threads):
    from frog_b200 import pairsbin
    from oracle import oracle
    out = os.path.join(os.path.dirname(list_path), "ref_pairs.bin")
    t0 = time.perf_counter()
    res = oracle.run_ref_binary([list_path, "-o", out, "-d", dist, "-d2", ratio], threads=threads)
    wall = time.perf_counter() - t0
    # the reference prints " : <seconds>s" after each phase; the third one is "Pairing" (match.cpp:655)
    secs = [float(x) for x in re.findall(r" : ([0-9.eE+-]+)s$", res.stdout, flags=re.M)]
    pairing = secs[2] if len(secs) >= 3 else wall
    # Loaded (phantom-inclusive, match.cpp:179-208) keypoint counts come from the pairs.bin the reference
    # wrote: its per-image stdout lines are printed from OpenMP threads without a lock and interleave.
    n = np.array([p.shape[0] for p in pairsbin.parse(out).points], np.float64)
    pairs = (n.sum() ** 2 - (n ** 2).sum()) / 2.0  # sum_{i<j} N_i N_j
    return pairs, pairing, wall


def sample_images(cores, n_points, budget_s=14.0):
    """How many REAL-SIZE images of the workload the CPU sample holds.  The reference parallelises over image pairs
    only (match.cpp:638), one image pair of 20k x 20k keypoints is ~4-6 s on a core, so the sample is the image
    count whose n(n-1)/2 image pairs keep the cores busiest (fewest idle cores in the last OpenMP wave) within about
    `budget_s` seconds per run."""
    per_pair_s = float(n_points) ** 2 / 9.0e7
    best, best_eff = 3, -1.0
    for n in range(3, 65):
        p = n * (n - 1) // 2
        waves = -(-p // cores)
        if n > 3 and waves * per_pair_s > budget_s:
            break
        eff = p / float(waves * cores)
        if eff > best_eff + 1e-9:
            best, best_eff = n, eff
    return best


def reference_sample(workload, tmp):
    from frog_b200 import synth
    n_img, n_pts, kind, dist, ratio = WORKLOADS[workload]
    cores = os.cpu_count() or 1
    s_img = min(n_img, sample_images(cores, n_pts))
    lst = synth.write_group(tmp, kind, s_img, n_pts, fmt="bin")
    text = (f"{s_img} of the workload's {n_img} images, {n_pts} keypoints each ({kind}), "
            f"{s_img * (s_img - 1) // 2} image pairs, -d {dist:g} -d2 {ratio:g}, -nt {cores}")
    return lst, dist, ratio, cores, text


def parity_on_sample(list_path, ref_pairs_path, dist, ratio, device):
    """Checker leg: the product (C ABI, cuda:`device`) on the very keypoint files the reference binary just matched,
    lists compared block by block with the reference's pairs.bin (oracle/compare.py classifies differences)."""
    from frog_b200 import capi, hostio, pairsbin
    from oracle import compare
    files = [l.split(",")[0] for l in open(list_path).read().split("\n") if l.strip()]
    images = []
    for f in files:
        head, desc = hostio.read_keypoints(f)  # phantom record of .bin files included, as the reference loads them
        images.append((desc, np.ascontiguousarray(head[:, 3]), np.ascontiguousarray(head[:, 4])))
    ref = pairsbin.parse(ref_pairs_path).block_map()
    keys = sorted(ref)
    m = capi.Matcher(device)
    try:
        for i, (d, sc, lp) in enumerate(images):
            m.upload(i, d, sc, lp)
        res = m.match([k[0] for k in keys], [k[1] for k in keys], dist, ratio)
        ours = dict(zip(keys, res.all_pairs()))
        res.free()
    finally:
        m.close()
    rep = compare.compare_blocks(ours, ref, images, dist, ratio)
    rep["what"] = "product vs reference pairs.bin on the cpu_baseline sample, every image pair"
    return rep


def cpu_baseline(workload, parity_device=None):
    tmp = tempfile.mkdtemp(prefix="fm_cpu_")
    parity = None
    try:
        lst, dist, ratio, cores, text = reference_sample(workload, tmp)
        pairs, pairing, wall = run_reference(lst, dist, ratio, cores)
        if parity_device is not None:
            try:
                parity = parity_on_sample(lst, os.path.join(tmp, "ref_pairs.bin"), dist, ratio, parity_device)
            except Exception as e:
                parity = {"error": str(e)[:300]}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    out = {"value": pairs / pairing, "unit": "descriptor pairs/s", "cores": cores, "kind": "reference",
           "sample": text + "; reference's own Pairing timer (match.cpp:655)", "seconds": pairing, "wall_s": wall}
    if parity is not None:
        out["parity"] = parity
    return out


def bench_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    tmp = tempfile.mkdtemp(prefix="fm_ref_")
    try:
        lst, dist, ratio, cores, text = reference_sample(args.workload, tmp)
        times, walls, pairs = [], [], 0.0
        for it in range(args.warmup + args.steps):
            pairs, pairing, wall = run_reference(lst, dist, ratio, cores)
            if it >= args.warmup:
                times.append(pairing)
                walls.append(wall)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    t = float(np.mean(times))
    val = pairs / t
    sample = f"{text} per step = {pairs:.3g} descriptor pairs"
    line = {
        "impl": "reference", "metric": METRIC,
        "value": val, "unit": "descriptor pairs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_name(args.workload, args.gpus), "reference_sample": sample},
        "cpu_baseline": {"value": val, "unit": "descriptor pairs/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": val, "unit": "descriptor pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall": {"unit": "s", "what": "match_ref process start -> exit on the sample (.bin inputs)", "seconds": float(np.mean(walls))},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for l in self.proc.stdout:
            self.lines.append((time.time(), l.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                mx = float(f[1])
                if t0 <= ts <= t1 + 0.1:
                    sm.append(float(f[0]))
                    for nm, v in zip(names, f[3:7]):
                        if v.lower().startswith("active"):
                            reasons.add(nm)
            except ValueError:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def bin_match_wall(kps, kind, thr, ratio, gpus, formats):
    """Wall time of the drop-in executable on the same group: `bin/match list -o pairs.bin -d .. -d2 .. -gpus N`,
    process start to exit (the reference prints the same three phase timers, match.cpp:572-573, 611-612, 654-655).
    Two ways: one-shot (every call pays CUDA's start-up: ~0.55 s + ~0.65 s per further GPU on these boxes) and through
    the resident server (`-serve 1`, contexts warm; the call that starts the server is not the one timed)."""
    from frog_b200 import build, synth
    out = {"unit": "s", "what": "bin/match process start -> exit on the workload's group (files in the page cache); "
                                "*_served: the same command line with -serve 1 against a warm resident server", "gpus": gpus}
    cores = os.cpu_count() or 1
    ids = [x for x in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if x] or [str(g) for g in range(gpus)]
    for fmt in formats:
        tmp = tempfile.mkdtemp(prefix="fm_wall_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        env = dict(os.environ, FROGMATCH_SOCKET=os.path.join(tmp, "fm.sock"), FROGMATCH_SERVE_IDLE="120",
                   CUDA_VISIBLE_DEVICES=",".join(ids[:gpus]))
        try:
            lst = synth.write_group(tmp, kind, len(kps), kps[0].n, fmt=fmt, threads=min(cores, 32), keypoints=kps)
            stats = os.path.join(tmp, "stats.json")
            cmd = [build.BIN, lst, "-o", os.path.join(tmp, "pairs.bin"), "-d", repr(thr), "-d2", repr(ratio), "-gpus", str(gpus),
                   "-stats", stats]

            def one(extra):
                t0 = time.perf_counter()
                r = subprocess.run(cmd + extra, capture_output=True, text=True, env=env)
                wall = time.perf_counter() - t0
                if r.returncode != 0:
                    raise RuntimeError(f"bin/match failed ({r.returncode}): {r.stderr[-300:]}")
                secs = [float(x) for x in re.findall(r" : ([0-9.eE+-]+)s$", r.stdout, flags=re.M)]
                st = json.load(open(stats))
                return {"seconds": wall, "load_s": secs[0] if secs else None, "pairing_s": secs[2] if len(secs) > 2 else None,
                        "gpu_ms_max": st.get("gpu_ms_max"), "ctx_create_s": st.get("ctx_create_s"), "matches": st.get("matches"),
                        "gpus_used": st.get("gpus")}

            runs = [one([]) for _ in range(2)]
            best = min(runs, key=lambda x: x["seconds"])
            best["first_run_seconds"] = runs[0]["seconds"]
            out[fmt.replace(".", "_")] = best
            try:
                start = one(["-serve", "1"])  # starts the server: CUDA comes up for every visible GPU, once
                served = [one(["-serve", "1"]) for _ in range(2)]
                best = min(served, key=lambda x: x["seconds"])
                best["server_start_call_seconds"] = start["seconds"]
                out[fmt.replace(".", "_") + "_served"] = best
            finally:
                subprocess.run([build.BIN, "-serve-stop"], env=env, capture_output=True, timeout=120)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    return out


def producer_line(device, size=256, steps=5, warmup=3, points=20000):
    """The step before the path (SURVEY 8f-4): one size^3 volume through libfrogsurf.so (frog_b200.surf) -- host buffer
    in, keypoints + descriptors out -- with the reference's own producer code (oracle/_ref/libsurf_ref.so, all cores)
    timed on the same volume and the two outputs compared.  scripts/gpu_surf_bench.py is the full-size measurement."""
    import time
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import gpu_surf_bench as gsb
    from frog_b200 import surf
    from oracle import surf_oracle
    vol = gsb.bench_volume(size)
    p = surf.Producer(device)
    walls = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        p.set_volume(vol)
        n_det = p.detect(0.0)
        p.select(points)
        p.describe(0, 5, True)
        pts, desc = p.points()
        if it >= warmup:
            walls.append(time.perf_counter() - t0)
    st = p.stats()
    p.close()
    wall = float(np.median(walls))
    out = {"metric": "voxels/s through the SURF3D producer (surf3d -t 0 -n 20000, type 0)", "workload": f"{size}^3 int16 volume",
           "value": vol.size / wall, "unit": "voxels/s", "ms_per_volume": wall * 1e3,
           "gpu_ms": {k: st[k] for k in ("ms_integral", "ms_response_map", "ms_extrema", "ms_describe")},
           "n_detected": int(n_det), "n_points": int(len(pts)), "h2d_bytes": int(vol.nbytes), "d2h_bytes": int(pts.nbytes + desc.nbytes)}
    if surf_oracle.available():
        t0 = time.perf_counter()
        ref = surf_oracle.RefSurf(vol)
        rx, rlap, rdesc = ref.update(threshold=0.0, number_of_points=points)
        ref_s = time.perf_counter() - t0
        same = len(rx) == len(pts)
        g = np.stack([pts["x"], pts["y"], pts["z"], pts["scale"], pts["response"]], 1)
        out["cpu_baseline"] = {"kind": "reference", "seconds": ref_s, "value": vol.size / ref_s, "unit": "voxels/s", "cores": os.cpu_count()}
        out["parity"] = {"n_points": [int(len(pts)), int(len(rx))],
                         "point_values_differ": int(np.count_nonzero(g.view(np.uint32) != rx.view(np.uint32))) if same else None,
                         "descriptor_values_differ": int(np.count_nonzero(desc.view(np.uint32) != rdesc.view(np.uint32))) if same else None}
    return out


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, lists):
    """The match lists of the last timed step, as fm_match returns them: counts.npy [image pairs] and pairs.npy
    [matches, 2] ((first, second) keypoint indices, image pairs in (i, j) order, i < j), float64.  Above DUMP_BYTES
    pairs.npy holds a fixed seeded sample of the rows, whose indices are in pairs_rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    counts = np.array([m.shape[0] for m in lists], np.float64)
    pairs = np.concatenate([np.zeros((0, 2), np.uint32)] + list(lists)).astype(np.float64)
    np.save(os.path.join(out_dir, "counts.npy"), counts)
    cap = (DUMP_BYTES - counts.nbytes) // 24  # 16 bytes per sampled row + 8 for its index
    if pairs.shape[0] > cap:
        rows = np.sort(np.random.default_rng(0).choice(pairs.shape[0], cap, replace=False))
        np.save(os.path.join(out_dir, "pairs_rows.npy"), rows.astype(np.float64))
        pairs = pairs[rows]
    np.save(os.path.join(out_dir, "pairs.npy"), pairs)


def bench_ours(args):
    import torch
    import torch.distributed as dist

    from frog_b200 import capi, synth
    from frog_b200 import dist as fdist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the matcher has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # stdout carries exactly ONE JSON line: native libraries that write to fd 1 (NCCL prints its version banner
    # there) are pointed at stderr, the line itself goes to a private duplicate of the original stdout
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if world > 1:
        # NCCL on a high-priority stream: the list transfer of one step runs while the next step's scoring kernel
        # still has thread blocks waiting to be dispatched, and must not queue behind them
        opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        dist.init_process_group("nccl", device_id=dev, pg_options=opts)
        host_group = dist.new_group(backend="gloo")  # CPU-side barrier: idle ranks must not spin a kernel on their GPU
    n_img, n_pts, kind, thr, ratio = WORKLOADS[args.workload]
    for kv in args.debug_opt:
        k, v = kv.split("=")
        capi.debug_set_option(k, int(v))

    # ---- the synthetic group (the same on every rank), in pinned host memory -----------------------
    kps = [synth.make(kind, n_pts, i) for i in range(n_img)]
    host = []
    for k in kps:
        host.append((torch.from_numpy(k.desc).pin_memory(), torch.from_numpy(k.scale).pin_memory(),
                     torch.from_numpy(k.lap).pin_memory()))
    pf_all = [i for i in range(n_img) for j in range(i + 1, n_img)]
    ps_all = [j for i in range(n_img) for j in range(i + 1, n_img)]
    weights = [float(kps[i].n) * float(kps[j].n) for i, j in zip(pf_all, ps_all)]
    total_pairs = float(sum(weights))
    # ---- this rank's share of the image pairs (match.cpp:638-652 is the loop being sharded) ---------
    shards = fdist.shard_pairs(weights, world)
    mine = shards[rank]
    pf = [pf_all[p] for p in mine]
    ps = [ps_all[p] for p in mine]
    needed = sorted(set(pf) | set(ps))
    h2d_bytes = sum(host[i][0].numel() * 4 + host[i][1].numel() * 4 + host[i][2].numel() * 4 for i in needed)
    rows_rank = sum(kps[j].n for j in ps)  # one outer-loop row per keypoint of image `second`, per image pair

    # real (non-default) streams: handle 0 would mean "the context's own stream" to fm_set_stream
    stream = torch.cuda.Stream(device=dev)
    comm = torch.cuda.Stream(device=dev, priority=-1)  # list hand-off: NCCL transfers and D2H copies
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def upload_all(mm):
        for i in needed:
            d, s, l = host[i]
            mm.upload_raw(i, d.data_ptr(), s.data_ptr(), l.data_ptr(), d.shape[0], d.shape[1])

    # N > 1, end to end: every byte of the group crosses PCIe ONCE -- rank r copies images r, r + N, ... from its pinned
    # host memory to its GPU -- and reaches the other GPUs over NVLink (NCCL all-gather), instead of every rank pulling
    # the whole group over its own PCIe link.  fm_upload_image takes the gathered device pointers as they are.
    uniform = len({k.n for k in kps}) == 1 and world > 1 and n_img % world == 0
    mine_imgs = list(range(rank, n_img, world))
    if uniform:
        h_desc = torch.stack([host[i][0] for i in mine_imgs]).pin_memory()   # [n_local, n_pts, 48]
        h_scale = torch.stack([host[i][1] for i in mine_imgs]).pin_memory()
        h_lap = torch.stack([host[i][2] for i in mine_imgs]).pin_memory()
        g_bufs = [None, None]  # per e2e context: the gathered group, alive until that context's next upload

    def upload_sharded(mm, slot):
        """H2D of this rank's images + all-gather over NVLink, on the current stream; returns this rank's H2D bytes."""
        if not uniform:
            upload_all(mm)
            return h2d_bytes
        n_local = len(mine_imgs)
        loc = [h_desc.to(dev, non_blocking=True), h_scale.to(dev, non_blocking=True), h_lap.to(dev, non_blocking=True)]
        full = [torch.empty((world * n_local,) + t.shape[1:], dtype=t.dtype, device=dev) for t in loc]
        for f, t in zip(full, loc):
            dist.all_gather_into_tensor(f, t)  # rank-major: row r * n_local + k = image k * world + r
        g_bufs[slot] = (full, loc)
        d_all, s_all, l_all = full
        for i in needed:
            row = (i % world) * n_local + i // world
            mm.upload_raw(i, d_all[row].data_ptr(), s_all[row].data_ptr(), l_all[row].data_ptr(), d_all.shape[1], d_all.shape[2])
        return sum(t.numel() * 4 for t in (h_desc, h_scale, h_lap))

    class PinnedLists:
        """Rank 0's host-side landing area for the match lists; grows on demand."""

        def __init__(self):
            self.buf = torch.empty(1 << 20, dtype=torch.int32).pin_memory()

        def view(self, off, n):
            if off + n > self.buf.numel():
                nb = torch.empty(max(off + n, 2 * self.buf.numel()), dtype=torch.int32).pin_memory()
                nb[:off].copy_(self.buf[:off])
                self.buf = nb
            return self.buf[off:off + n]

    landing = PinnedLists()

    def hand_off(res, to_host):
        """Lists of a finished step to rank 0 (device; and on to pinned host memory with to_host).  The step's kernels
        are done (res.wait() returned), so nothing here waits for the compute stream: transfers run on `comm` beside
        the next step's kernels.  Returns the D2H bytes this rank copied."""
        d2h = 0
        cptr, pptr = res.device_pointers()
        counts = fdist.as_torch_u32(cptr, res.n_pairs, dev)
        pairs = fdist.as_torch_u32(pptr, 2 * int(res.total), dev)
        with torch.cuda.stream(comm):
            got = fdist.gather_match_lists(counts, pairs, 0) if world > 1 else ([counts], [pairs])
            if to_host and rank == 0:
                off = 0
                for c, p in zip(*got):
                    for t in (c, p):
                        if t.numel():
                            landing.view(off, t.numel()).copy_(t, non_blocking=True)
                            off += t.numel()
                d2h = off * 4
        comm.synchronize()  # lists have left this GPU / reached rank 0: the result's buffers may be reused
        return d2h

    # ---- resident: keypoints stay in HBM, K asynchronous fm_match calls back to back ---------------
    m = capi.Matcher(local)
    m.set_stream(stream.cuda_stream)
    upload_all(m)
    m.synchronize()
    retired = []
    host_ms = collections.defaultdict(float)

    class phase:
        def __init__(self, name):
            self.name = name

        def __enter__(self):
            self.t = time.perf_counter()

        def __exit__(self, *a):
            host_ms[self.name] += (time.perf_counter() - self.t) * 1e3

    def finish_resident(res, keep=False):
        with phase("wait_kernels"):
            res.wait()  # this step's kernels are done; the next step's are already queued behind them
        if world > 1:
            with phase("gather"):
                hand_off(res, to_host=False)
        retired.append((res.stats(), int(res.total)))
        if keep:
            return res
        res.free()

    def timed_resident(steps, warmup):
        prev = None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = 0.0
        for k in range(warmup + steps):
            if k == warmup:
                if prev is not None:
                    finish_resident(prev)
                    prev = None
                retired.clear()
                host_ms.clear()
                barrier()
                t0 = time.time()
                e0.record(stream)
            with torch.cuda.stream(stream):
                flush.zero_()  # evict the group from the 126 MB L2 between steps
                res = m.match(pf, ps, thr, ratio, device_only=True, asynchronous=True)
            if prev is not None:
                finish_resident(prev)
            prev = res
        last = finish_resident(prev, keep=bool(args.dump_outputs))  # with --dump-outputs: freed once it is written
        stream.wait_stream(comm)
        e1.record(stream)
        barrier()
        t1 = time.time()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), t0, t1, last

    sampler = ClockSampler(local) if rank == 0 else None
    ms_res, t0, t1, last = timed_resident(args.steps, args.warmup)
    clocks = sampler.stop(t0, t1) if sampler else None
    if args.dump_outputs:
        cptr, pptr = last.device_pointers()
        counts = fdist.as_torch_u32(cptr, last.n_pairs, dev)
        pairs = fdist.as_torch_u32(pptr, 2 * int(last.total), dev)
        got = fdist.gather_match_lists(counts, pairs, 0) if world > 1 else ([counts], [pairs])
        torch.cuda.synchronize()
        if rank == 0:
            dump_outputs(args.dump_outputs, fdist.assemble(shards, *got, len(pf_all)))
        last.free()
    stats = [o[0] for o in retired]
    matches_rank = retired[-1][1]
    res_host_ms = {k: round(v / args.steps, 4) for k, v in host_ms.items()}
    m.close()

    # ---- end to end: host buffers in, host lists out, through the C ABI ---------------------------
    # Two contexts on two streams, used alternately as a three-stage pipeline: while one runs step k's prep +
    # kernels, the other first hands step k-1's lists to rank 0's pinned host memory (NCCL gather for N > 1, then D2H)
    # and then uploads step k+1's images (H2D).  Every step's H2D and D2H is inside the timed region, which is
    # ONE CUDA-event bracket around all K steps (L2 flush writes included).
    streams = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
    ctxs = [capi.Matcher(local), capi.Matcher(local)]
    for mm, st in zip(ctxs, streams):
        mm.set_stream(st.cuda_stream)

    def e2e_start(mm, st):
        with torch.cuda.stream(st):
            flush.zero_()
            # prep + kernels queued, call returns; the lists reach the host in e2e_finish
            return mm.match(pf, ps, thr, ratio, device_only=True, asynchronous=True)

    def e2e_finish(res):
        with phase("wait_kernels"):
            res.wait()
        with phase("gather_d2h"):
            d2h = hand_off(res, to_host=True)
        res.free()
        return d2h

    h2d_step = [h2d_bytes]

    def timed_e2e(steps, warmup):
        d2h, total, prev = [], warmup + steps, None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctxs[0].clear()
        with torch.cuda.stream(streams[0]):
            upload_sharded(ctxs[0], 0)
        for k in range(total):
            cur, st = ctxs[k % 2], streams[k % 2]
            if k == warmup:
                if prev is not None:
                    d2h.append(e2e_finish(prev))
                    prev = None
                barrier()  # every stream of every rank is idle: start the clock
                host_ms.clear()
                e0.record(st)
                cur.clear()
                with torch.cuda.stream(st):
                    upload_sharded(cur, k % 2)  # pipeline fill: the first timed step's own upload is inside the region
            with phase("start_prep"):
                res = e2e_start(cur, st)  # step k: prep + kernels queued
            if k + 1 < total and k + 1 != warmup:
                # step k+1: H2D from pinned host memory, under step k's kernels.  Its context is the one that ran
                # step k-1; that step's lists live in the result's own buffers, not in the image arena.
                nxt = ctxs[(k + 1) % 2]
                with phase("clear"):
                    nxt.clear()
                with phase("upload_enqueue"), torch.cuda.stream(streams[(k + 1) % 2]):
                    h2d_step[0] = upload_sharded(nxt, (k + 1) % 2)
            if prev is not None:
                d2h.append(e2e_finish(prev))  # step k-1: lists to rank 0's pinned host memory, under step k's kernels
            prev = res
        d2h.append(e2e_finish(prev))
        last = streams[(total - 1) % 2]
        last.wait_stream(comm)
        e1.record(last)
        barrier()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), d2h[warmup:]

    ms_e2e, d2h_list = timed_e2e(args.steps, max(1, args.warmup))
    d2h_bytes = float(np.mean(d2h_list))
    e2e_host_ms = {k: round(v / args.steps, 4) for k, v in host_ms.items()}
    for mm in ctxs:
        mm.close()

    # whole-job aggregates
    agg = torch.tensor([float(h2d_step[0]), d2h_bytes, float(sum(s["kernel_launches"] for s in stats)), float(matches_rank)],
                       dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(agg, op=dist.ReduceOp.SUM)
    h2d_all, d2h_all, launches, matches_all = agg.tolist()

    torch.cuda.synchronize()
    if rank == 0:
        peak_tf, peak_gbs, which = peaks()
        n_launch = float(np.mean([s["score_launches"] for s in stats]))
        sc_ms = float(np.mean([s["ms_score"] / max(1, s["score_launches"]) for s in stats]))
        pairs_per_launch = float(np.mean([s["descriptor_pairs"] / max(1, s["score_launches"]) for s in stats]))
        scored_per_launch = float(np.mean([s["scored_pairs"] / max(1, s["score_launches"]) for s in stats]))
        achieved = FLOP_PER_PAIR * pairs_per_launch / (sc_ms * 1e-3) / 1e12 if sc_ms > 0 else 0.0
        executed = 2.0 * 64.0 * scored_per_launch / (sc_ms * 1e-3) / 1e12 if sc_ms > 0 else 0.0
        s0 = stats[-1]
        comp_bytes = 4.0 * s0["rows"] + 8.0 * matches_rank  # one 4-byte read per outer-loop row, one 8-byte write per match
        line = {
            "metric": METRIC,
            "value": total_pairs * args.steps / (ms_res * 1e-3), "unit": "descriptor pairs/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_res / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f16 operands / f32 accumulate + exact f32 rescoring",
            "data": "synthetic",
            "config": {"workload": workload_name(args.workload, world), "l2": "256 MiB flush buffer written between timed steps",
                       "timing": "value and e2e: one CUDA-event bracket around all steps (asynchronous fm_match calls, a step's "
                                 "list hand-off overlaps the next step's kernels), max over ranks; e2e alternates two contexts so "
                                 "a step's H2D upload overlaps the previous step's kernels",
                       "image_pairs_per_rank": [len(s) for s in shards], "matches_per_step": matches_all},
            "e2e": {"value": total_pairs * args.steps / (ms_e2e * 1e-3), "unit": "descriptor pairs/s",
                    "h2d_bytes_per_step": h2d_all, "d2h_bytes_per_step": d2h_all, "ms_per_step": ms_e2e / args.steps,
                    "nvlink_allgather_bytes_per_step": (float(h2d_all) * (world - 1) if (world > 1 and uniform) else 0.0),
                    "rank0_host_ms_per_step": e2e_host_ms},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": achieved / peak_tf, "traffic": measured_traffic(args.workload), "peak_source": which + " (cuBLAS bf16 burst)",
                         "kernel": "fm::score_kernel<false>" + (" (reject pass + capture pass)" if s0.get("two_phase_batches") else ""),
                         "kernel_ms": sc_ms, "launches_per_step": n_launch, "two_phase_batches_per_step": s0.get("two_phase_batches", 0),
                         "algorithmic_flop_per_launch": FLOP_PER_PAIR * pairs_per_launch,
                         "executed_tflops": executed, "executed_frac": executed / peak_tf,
                         "scored_fraction": scored_per_launch / max(1.0, pairs_per_launch), "rank": 0},
            # stream compaction (HBM-bound, DESIGN.md 4), rank 0's share, over the CUDA-event time of its kernel(s)
            "compaction": {"bound": "hbm", "unit": "GB/s", "peak": peak_gbs, "peak_source": which,
                           "achieved": comp_bytes / max(s0["ms_compact"] * 1e-3, 1e-12) / 1e9,
                           "frac": comp_bytes / max(s0["ms_compact"] * 1e-3, 1e-12) / 1e9 / peak_gbs,
                           "kernel_ms": s0["ms_compact"], "bytes": comp_bytes},
            "phases_ms": {k: s0[k] for k in ("ms_total", "ms_score", "ms_rescore", "ms_exact", "ms_compact", "ms_prep")},
            "rank0_host_ms_per_step": res_host_ms,
            "rows_exact_frac": s0["rows_exact"] / max(1, s0["rows"]), "candidates_per_row": s0["candidates"] / max(1, s0["rows"]),
            "rows_rejected_early_frac": s0["rows_rejected_early"] / max(1, s0["rows"]),
            # differences from the reference whose distance / ratio sits within 4 ulp of -d / -d2, counted on the
            # cpu_baseline sample (N = 1 runs; null when that leg did not run)
            "threshold_eps_count": None,
            "clocks": clocks,
        }
        if args.debug_opt:
            line["config"]["debug_opt"] = args.debug_opt
        if not args.no_wall:
            try:
                line["wall"] = bin_match_wall(kps, kind, thr, ratio, world, ["bin"] + ([] if args.no_wall_gz else ["csv.gz"]))
            except Exception as e:
                line["wall"] = {"unit": "s", "error": str(e)[:300]}
        if not args.no_cpu_baseline and world == 1:
            try:
                line["cpu_baseline"] = cpu_baseline(args.workload, parity_device=local)
                par = line["cpu_baseline"].get("parity") or {}
                if "threshold_eps_count" in par:
                    line["threshold_eps_count"] = par["threshold_eps_count"]
            except Exception as e:  # the baseline must never take the GPU numbers down with it
                line["cpu_baseline"] = {"value": None, "unit": "descriptor pairs/s", "cores": os.cpu_count(), "kind": "reference",
                                        "sample": f"failed: {e}"}
        if not args.no_producer and world == 1:
            try:
                line["producer"] = producer_line(local)  # (the reference producer's progress lines go to fd 1 = stderr here)
            except Exception as e:
                line["producer"] = {"error": str(e)[:300]}
        print(json.dumps(line), file=json_out, flush=True)
    if world > 1:
        dist.barrier(group=host_group)  # ranks > 0 wait here (on the CPU) while rank 0 times bin/match and the CPU baseline
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-wall", action="store_true")
    ap.add_argument("--no-producer", action="store_true", help="skip the SURF3D producer sub-measurement (N = 1 only)")
    ap.add_argument("--no-wall-gz", action="store_true")
    ap.add_argument("--debug-opt", action="append", default=[], metavar="NAME=VALUE",
                    help="kernel-study switch (include/frogmatch_debug.h), e.g. variant=1; not for reported numbers")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the match lists of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        bench_reference(args)
    else:
        bench_ours(args)


if __name__ == "__main__":
    main()
