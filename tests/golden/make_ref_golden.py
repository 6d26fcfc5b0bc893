"""Recorded reference outputs (tests/golden/ref) for the tests that compare the product with the verbatim reference
build on inputs no other fixture holds.  With them those tests run where the reference's sources are absent; where
oracle/_ref is built they compare with it live as well.

    python tests/golden/make_ref_golden.py [--reference] [--cpu-only] [--out DIR]

The committed values were written by this project (bin/match, bin/surf3d, libfrogsurf.so on a B200; the oracle's C
port for the CPU cases) at a commit where every one of these tests had passed against the verbatim reference build on
the same inputs: pairs.bin and keypoint files byte for byte, descriptors bit for bit, keypoint coordinates within the
1 ulp the tests allow.  --reference recomputes them from oracle/_ref instead (needs the reference sources, see
oracle/Makefile).  pairs.bin files are recorded as helpers.pairs_digest (image names cut to their base names, since
the files name the directory they were written in).

Cases (every input regenerated from a seed):
  c2_iid, c2_bank   10 x 20 000 keypoints (.bin), -d 1: pairs.bin                     tests/test_gpu_scale.py
  config5           run.sh around the matcher, 8 x 20 000 bank keypoints (.csv.gz)    tests/test_gpu_scale.py
  fresh_group       2 x 5 000 bank keypoints (.csv.gz), default flags: pairs.bin      tests/test_gpu_cli.py
  surf_fresh        400^3 volume (four octaves), 3000 keypoints                       tests/test_gpu_surf.py
  surf_odd          131 x 103 x 117 volume, every keypoint                            tests/test_gpu_surf.py
  surf_run_sh       three volumes through surf3d, then the matcher: files and pairs   tests/test_gpu_surf.py
  multi_member      keypoints loaded from a two-member .csv.gz                        tests/test_hostio.py
  match_all         -all lists of the port on three seeded image pairs                tests/test_oracle.py
"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
from frog_b200 import build, pairsbin, synth  # noqa: E402
from oracle import oracle as O, surf_oracle as so  # noqa: E402
import make_surf_golden as mg  # noqa: E402

OUT = os.path.join(HERE, "ref")
GPU_CASES = ("c2_iid", "c2_bank", "config5", "fresh_group", "surf_fresh", "surf_odd", "surf_run_sh")
CPU_CASES = ("multi_member", "match_all")
MATCH_ALL_THRESHOLDS = (0.22, 0.6, 5.0)


def pairs_digest(path_or_bytes) -> str:
    """SHA-256 of a pairs.bin's content with every image name cut to its base name."""
    pf = pairsbin.parse(path_or_bytes)
    h = hashlib.sha256()
    for name, rigid, pts in zip(pf.names, pf.rigids, pf.points):
        h.update(os.path.basename(name).encode("latin-1") + b"\0")
        h.update(np.asarray(rigid, "<f8").tobytes() + np.ascontiguousarray(pts, "<f4").tobytes())
    for i, j, m in pf.blocks:
        h.update(np.array([i, j, m.shape[0]], "<u4").tobytes() + np.ascontiguousarray(m, "<u4").tobytes())
    return h.hexdigest()


def load(name):
    """(manifest entry, arrays or None) of a recorded case."""
    entry = json.load(open(os.path.join(OUT, "manifest.json")))[name]
    npz = os.path.join(OUT, name + ".npz")
    return entry, (np.load(npz) if os.path.exists(npz) else None)


# ---- inputs -------------------------------------------------------------------------------------------------------

def fresh_volume():
    vol = synth.make_volume((100, 120, 400), 17, blobs_per_mvox=2500.0)
    return np.pad(vol, ((150, 150), (140, 140), (0, 0)), mode="reflect")  # 400 x 400 x 400


def odd_volume():
    return synth.make_volume((131, 103, 117), 5)


def run_sh_volumes():
    vols = [synth.make_volume((136, 128, 144), 30, blobs_per_mvox=3000.0)]
    vols.append(np.roll(vols[0], (3, -2, 4), (0, 1, 2)) + np.random.default_rng(1).integers(-6, 7, vols[0].shape).astype(np.int16))
    vols.append(synth.make_volume((136, 128, 144), 31, blobs_per_mvox=3000.0))
    return vols


RUN_SH_SPACING, RUN_SH_ORIGIN = (0.75, 0.75, 0.75), lambda i: (-50.0, -40.0, 10.0 * i)


def multi_member_files(d):
    """A .csv.gz of two gzip members (40 + 25 keypoints), a plain one, and their list file."""
    import gzip
    a, b = synth.make("bank", 40, 0), synth.make("bank", 25, 1)
    two = os.path.join(d, "two.csv.gz")
    open(two, "wb").write(gzip.compress(synth._text_lines(a), 6) + gzip.compress(synth._text_lines(b), 1))
    other = os.path.join(d, "other.csv.gz")
    synth.write_csv_gz(synth.make("bank", 50, 2), other)
    lst = os.path.join(d, "list.txt")
    open(lst, "w").write(f"{two}\n{other}\n")
    return two, lst, b


def match_all_cases():
    for seed in range(3):
        a, b = synth.make("bank", 300, seed), synth.make("bank", 260, seed + 5)
        for thr in MATCH_ALL_THRESHOLDS:
            for sym in (False, True):
                yield f"s{seed}_t{thr:g}_{'sym' if sym else 'plain'}", (a.desc, a.scale, a.lap), (b.desc, b.scale, b.lap), thr, sym


def run_pipeline(tmp, kp_dir, exe, n_img, tag):
    """run.sh (scripts/run_pipeline.sh) around one matcher executable with NPOINTS = 20000; returns the process."""
    res = os.path.join(tmp, f"res_{tag}")
    params = os.path.join(tmp, f"params_{tag}.sh")
    open(params, "w").write("\n".join([
        "export IMG_INPUT=(" + " ".join(f"image{k}.nii.gz" for k in range(n_img)) + ")",
        f"export RES_FOLDER={res}", "export SPACING=0.75", "export THRESHOLD=0", "export NPOINTS=20000",
        'export SURF_OTHER_PARAMS=""', "export MAX_DISTANCE=1", 'export MATCH_OTHER_PARAMS=""',
        'export REGISTRATION_OTHER_PARAMS=""']) + "\n")
    return subprocess.run(["bash", os.path.join(ROOT, "scripts", "run_pipeline.sh"), params, kp_dir, exe,
                           f"{sys.executable} {os.path.join(ROOT, 'scripts', 'read_pairs.py')}"],
                          capture_output=True, text=True, timeout=900), os.path.join(res, "pairs.bin")


# ---- one source of outputs: the product, or the verbatim reference build ------------------------------------------

def match_exe(reference):
    return O.REF_BIN if reference else build.BIN


def run_match(reference, args):
    if reference:
        return O.run_ref_binary(args, threads=os.cpu_count())
    r = subprocess.run([build.BIN] + args, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return r


def surf_outputs(reference, vol, n_points):
    """integral / layer hashes, the detector's keypoints in push_back order, the selected keypoints and the SHA-256 of
    their SURF3D descriptors (radius 5, normalised)."""
    if reference:
        ref = so.RefSurf(vol)
        rx, rlap, rdesc = ref.update(threshold=0.0, number_of_points=n_points)
        det, det_lap = ref.detect(0.0)
        integral, layers = ref.integral_volume(), ref.response_layers(0.0)
    else:
        from frog_b200 import surf
        p = surf.Producer(0)
        p.set_volume(vol)
        integral = p.integral()
        p.detect(0.0)
        layers = p.layers()
        pts, _ = p.points(with_descriptors=False)
        det, det_lap = xyzsr(pts), pts["laplacian"]
        p.select(n_points)
        p.describe(0, 5, True)
        pts, rdesc = p.points()
        rx, rlap = xyzsr(pts), pts["laplacian"]
        p.close()
    entry = dict(integral=mg.sha(integral), layers=mg.layer_hashes(layers), n_detected=int(len(det)), n_points=int(len(rx)),
                 desc=mg.sha(np.ascontiguousarray(rdesc, np.float32)))
    return entry, dict(det_xyzsr=np.ascontiguousarray(det, np.float32), det_lap=np.asarray(det_lap),
                       xyzsr=np.ascontiguousarray(rx, np.float32), lap=np.asarray(rlap))


def xyzsr(pts):
    return np.stack([pts["x"], pts["y"], pts["z"], pts["scale"], pts["response"]], 1)


def make_case(name, reference, tmp):
    if name in ("c2_iid", "c2_bank"):
        lst = synth.write_group(os.path.join(tmp, "g"), name[3:], 10, 20000, fmt="bin")
        run_match(reference, [lst, "-o", os.path.join(tmp, "pairs.bin"), "-d", "1"])
        out = os.path.join(tmp, "pairs.bin")
        return dict(pairs=pairs_digest(out), n_matches=pairsbin.parse(out).n_matches()), None
    if name == "fresh_group":
        lst = synth.write_group(os.path.join(tmp, "g"), "bank", 2, 5000, fmt="csv.gz")
        r = run_match(reference, [lst, "-o", os.path.join(tmp, "pairs.bin")])
        nb = [l for l in r.stdout.splitlines() if l.startswith("Nb Match")][0]
        return dict(pairs=pairs_digest(os.path.join(tmp, "pairs.bin")), nb_match_line=nb), None
    if name == "config5":
        kp_dir = os.path.join(tmp, "keypoints")
        synth.write_group(kp_dir, "bank", 8, 20000, fmt="csv.gz", threads=8)
        r, out = run_pipeline(tmp, kp_dir, match_exe(reference), 8, "gen")
        assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
        return dict(pairs=pairs_digest(out)), None
    if name == "surf_fresh":
        return surf_outputs(reference, fresh_volume(), 3000)
    if name == "surf_odd":
        return surf_outputs(reference, odd_volume(), 20000)
    if name == "surf_run_sh":
        files = []
        for i, v in enumerate(run_sh_volumes()):
            base = os.path.join(tmp, f"points{i}")
            if reference:
                ref = so.RefSurf(v, RUN_SH_SPACING, RUN_SH_ORIGIN(i))
                ref.update(threshold=0.0, number_of_points=20000)
                ref.write(base + ".csv.gz", "csv.gz")
            else:
                from frog_b200 import surf
                mha = os.path.join(tmp, f"v{i}.mha")
                surf.write_metaimage(mha, v, RUN_SH_SPACING, RUN_SH_ORIGIN(i))
                r = subprocess.run([build.SURF_BIN, mha, "-o", base, "-t", "0", "-n", "20000"], capture_output=True, text=True)
                assert r.returncode == 0, r.stderr
            files.append(base + ".csv.gz")
        lst = os.path.join(tmp, "points.txt")
        open(lst, "w").write("".join(f + "\n" for f in files))
        run_match(reference, [lst, "-o", os.path.join(tmp, "pairs.bin"), "-d", "1"])
        return dict(files=[hashlib.sha256(open(f, "rb").read()).hexdigest() for f in files],
                    pairs=pairs_digest(os.path.join(tmp, "pairs.bin"))), None
    if name == "multi_member":
        from frog_b200 import hostio
        two, lst, _ = multi_member_files(tmp)
        if reference:
            O.run_ref_binary([lst, "-o", os.path.join(tmp, "ref.bin"), "-d", "1"])
            head = pairsbin.parse(os.path.join(tmp, "ref.bin")).points[0]
        else:
            head = hostio.read_keypoints(two)[0]
        return dict(n_points=int(head.shape[0])), dict(points0=np.ascontiguousarray(head, np.float32))
    if name == "match_all":
        lib = O.RefLib() if reference else O.PortLib()
        return {}, {k: lib.compute_matches_all(a, b, thr, sym) for k, a, b, thr, sym in match_all_cases()}
    raise KeyError(name)


def main():
    reference = "--reference" in sys.argv
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else OUT
    names = CPU_CASES if "--cpu-only" in sys.argv else GPU_CASES + CPU_CASES
    os.makedirs(out, exist_ok=True)
    O.build(ref=reference)
    mpath = os.path.join(out, "manifest.json")
    manifest = json.load(open(mpath)) if os.path.exists(mpath) else {}
    for name in names:
        with tempfile.TemporaryDirectory(prefix="fm_gold_") as tmp:
            entry, arrays = make_case(name, reference, tmp)
        manifest[name] = entry
        if arrays is not None:
            np.savez_compressed(os.path.join(out, name + ".npz"), **arrays)
        print(name, {k: v for k, v in entry.items() if k != "layers"}, flush=True)
    json.dump(manifest, open(mpath, "w"), indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
