"""Reject-pass outputs of one library build, and a bitwise comparison of two builds' outputs.

    python scripts/gpu_reject_dump_cmp.py run LIB OUT.npz     # one build (LIB: a libfrogmatch.so)
    python scripts/gpu_reject_dump_cmp.py cmp A.npz B.npz     # exit 1 if any array differs

Two calls with two-phase scoring forced and the reject dump on (fm_debug_reject_rows): 24 iid images of 20 000
keypoints, all 276 pairs at -d 1 -d2 0.8 (the C4 gates), and 10 bank images of 16 000 keypoints, all pairs, -sym at
-d 1 -d2 0.9.  Saved per task: each row's certified_reject arguments (a1, a2, |a|^2, eps), rowstat, bands and the
sorted survivor list; per call the match lists and the scored_pairs counter.  scored_pairs includes the capture pass,
whose survivor units follow the order in which the reject pass appended survivors (atomics), so it varies from run to
run of one build; every other array must be bit-identical.
Run each build in its own process (the library path is fixed at load)."""
import os
import sys

import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from frog_b200 import capi, synth

def run(lib, out):
    capi.LIB_PATH = os.path.abspath(lib)
    res = {}
    for name, kind, n_img, npts, thr, rat, sym in (("iid276", "iid", 24, 20000, 1.0, 0.8, False),
                                                    ("banksym", "bank", 10, 16000, 1.0, 0.9, True)):
        kps = [synth.make(kind, npts, i) for i in range(n_img)]
        pf = [i for i in range(n_img) for j in range(i + 1, n_img)]
        ps = [j for i in range(n_img) for j in range(i + 1, n_img)]
        m = capi.Matcher(0)
        capi.debug_set_option("two_phase", 1)
        capi.debug_set_option("reject_dump", 1)
        for i, k in enumerate(kps):
            m.upload(i, k.desc, k.scale, k.lap)
        r = m.match(pf, ps, thr, rat, sym=sym)
        lists = r.all_pairs(); r.free()
        st = m.stats()
        assert st["two_phase_batches"] >= 1
        tasks = [(a, b) for a, b in zip(pf, ps)]
        if sym:
            tasks = [t for a, b in zip(pf, ps) for t in ((a, b), (b, a))]
        for t, (c, rw) in enumerate(tasks):
            d = m.debug_reject_rows(t, npts)
            assert d is not None
            for key in ("args", "rowstat", "bands", "survivors"):
                res[f"{name}/{t}/{key}"] = d[key]
        for p, l in enumerate(lists):
            res[f"{name}/list/{p}"] = np.asarray(l)
        res[f"{name}/scored_pairs"] = np.array([st.get("scored_pairs", 0)])
        capi.debug_set_option("reject_dump", 0)
        capi.debug_set_option("two_phase", -1)
        m.close()
    np.savez(out, **res)

def cmp(a, b):
    A, B = np.load(a), np.load(b)
    assert sorted(A.files) == sorted(B.files), "key sets differ"
    bad = [k for k in A.files if not k.endswith("/scored_pairs") and not (A[k].dtype == B[k].dtype and A[k].shape == B[k].shape and A[k].tobytes() == B[k].tobytes())]
    rows = sum(A[k].shape[0] for k in A.files if k.endswith("/args"))
    for k in (k for k in A.files if k.endswith("/scored_pairs")):
        print(f"{k} (not compared, varies run to run): {int(A[k][0])} vs {int(B[k][0])}")
    print(f"compared {len(A.files)} arrays, {rows} dumped rows; differing: {len(bad)} {bad[:10]}")
    for k in bad[:3]:
        print(k, A[k][:4], B[k][:4])
    return not bad

if __name__ == "__main__":
    if sys.argv[1] == "run":
        run(sys.argv[2], sys.argv[3])
    else:
        sys.exit(0 if cmp(sys.argv[2], sys.argv[3]) else 1)
