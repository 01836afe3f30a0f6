#!/usr/bin/env python
"""spn_match_pairs (include/spn_match.h): time per call over exhaustive pair lists, against the grouped gather +
spn_mutual_nn_match route of evaluations/posed_evaluation.py and against cv2.BFMatcher.knnMatch(k=2) + ratio test on a
host thread pool.

Workload: a pool of N = 32, 64 and 128 descriptor sets (every pair a < b: 496, 2 016 and 8 128 pairs), cap = 1000 rows
of C = 256, every set full (the matcher's work depends on the counts, not on the values).  Each set is 700 noisy views
(noise 0.3 per component) of rows of one seeded random base set in a random order plus 300 unrelated rows, all
L2-normalised, so that every filter keeps matches.
The pool is 33, 66 and 131 MB: the first two fit the 126 MB L2 after the first pass, the last does not.  Modes: mutual,
mutual + ratio 0.8, ratio 0.8 alone.  Reports, with the GPU's name, power limit and clocks read in the same run:
  * ms per spn_match_pairs call, CUDA events over --reps calls after warm-up (the pair-list upload included);
  * useful FLOP/s (2 n_a n_b C per direction, two directions with the mutual check) and executed FLOP/s (x3: the
    hi.hi + hi.lo + lo.hi tensor-core products);
  * mutual mode: ms of the grouped route (descriptors gathered 64 pairs at a time with index_select, then
    spn_mutual_nn_match), the same CUDA-event window, outputs asserted equal;
  * ms per pair of cv2 knnMatch(k=2) + ratio 0.8 on --cv2-pairs pairs (a SAMPLE, not the whole list) on a thread pool.

    python tools/bench_match.py [--reps 20] [--out profiles/r6_match.json]
"""
import argparse
import concurrent.futures as cf
import ctypes as C
import json
import math
import os
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from bench_nerf_export import gpu_info  # noqa: E402

CAP, DIM, GROUP = 1000, 256, 64
MODES = {"mutual": (True, 0.0), "mutual+ratio0.8": (True, 0.8), "ratio0.8": (False, 0.8)}


def event_ms(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def cv2_sample(desc, pairs, ratio, workers):
    import cv2

    def job(p):
        bf = cv2.BFMatcher(cv2.NORM_L2)
        knn = bf.knnMatch(desc[p[0]], desc[p[1]], k=2)
        return sum(1 for m in knn if len(m) == 2 and m[0].distance < ratio * m[1].distance)

    with cf.ThreadPoolExecutor(max_workers=workers) as pool:
        list(pool.map(job, pairs[:workers]))                 # warm-up
        t0 = time.perf_counter()
        kept = list(pool.map(job, pairs))
        dt = time.perf_counter() - t0
    return dt * 1e3 / len(pairs), int(sum(kept))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--sizes", default="32,64,128")
    ap.add_argument("--cv2-pairs", type=int, default=128)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_match needs a GPU")
    from superpoint_nerf_pytorch_b200 import _native
    ctx = _native.get_context(0)
    workers = max(1, min(32, (os.cpu_count() or 2) - 1))
    rec = {"gpu": gpu_info(), "cap": CAP, "C": DIM, "reps": args.reps, "cpu_workers": workers, "runs": []}
    for N in (int(s) for s in args.sizes.split(",")):
        rng = np.random.RandomState(N)
        base = rng.randn(CAP, DIM).astype(np.float32)
        host = rng.randn(N, CAP, DIM).astype(np.float32)
        for n in range(N):
            host[n, :700] = base[rng.permutation(CAP)[:700]] + 0.3 * host[n, :700]
        host /= np.linalg.norm(host, axis=-1, keepdims=True)
        desc = torch.from_numpy(host).cuda()
        counts = torch.full((N,), CAP, dtype=torch.int32, device="cuda")
        pairs = np.array([(a, b) for a in range(N) for b in range(a + 1, N)], np.int32)
        P = len(pairs)
        match = torch.empty((P, CAP), dtype=torch.int32, device="cuda")
        dist = torch.empty((P, CAP), dtype=torch.float32, device="cuda")
        ptr = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
        for mode, (mutual, ratio) in MODES.items():
            def call():
                ctx._call("spn_match_pairs", ctx.handle, ptr(desc), ptr(counts), N, CAP, DIM, C.c_void_p(pairs.ctypes.data), P,
                          int(mutual), C.c_float(ratio), C.c_float(math.inf), ptr(match), ptr(dist), ctx._s())
            ms = event_ms(call, args.reps)
            useful = 2.0 * CAP * CAP * DIM * P * (2 if mutual else 1)
            run = {"N": N, "pairs": P, "mode": mode, "ms_per_call": ms, "us_per_pair": ms * 1e3 / P,
                   "useful_tflops": useful / ms / 1e9, "executed_tflops": 3 * useful / ms / 1e9,
                   "matches": int((match >= 0).sum())}
            if mode == "mutual":
                ia = torch.from_numpy(pairs[:, 0].astype(np.int64)).cuda()
                ib = torch.from_numpy(pairs[:, 1].astype(np.int64)).cuda()
                ref = torch.empty_like(match)
                ref_d = torch.empty_like(dist)

                def grouped():
                    for g in range(0, P, GROUP):
                        sa, sb = ia[g:g + GROUP], ib[g:g + GROUP]
                        m, d = ctx.mutual_nn_match(desc.index_select(0, sa), counts.index_select(0, sa),
                                                   desc.index_select(0, sb), counts.index_select(0, sb))
                        ref[g:g + GROUP], ref_d[g:g + GROUP] = m, d
                gms = event_ms(grouped, args.reps)
                assert torch.equal(ref, match) and torch.equal(ref_d, dist), "pooled and grouped outputs differ"
                run.update(grouped_ms_per_call=gms, speedup_vs_grouped=gms / ms, outputs_equal=True)
            if not mutual:
                sample = [tuple(p) for p in pairs[np.random.RandomState(0).permutation(P)[:args.cv2_pairs]]]
                ms_pair, kept = cv2_sample(host, sample, ratio, workers)
                rows = np.array([q for q, p in enumerate(map(tuple, pairs)) if p in set(sample)])
                run.update(cv2_sample_pairs=len(sample), cv2_ms_per_pair=ms_pair, cv2_ms_extrapolated=ms_pair * P,
                           cv2_sample_matches=kept, gpu_sample_matches=int((match[torch.from_numpy(rows).cuda()] >= 0).sum()), note_cv2="cv2 timed on a sample of pairs; the extrapolation is per-pair time x P")
            rec["runs"].append(run)
            print(json.dumps(run), flush=True)
    rec["gpu_after"] = gpu_info()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(rec, indent=2) + "\n")
    print(json.dumps({"gpu": rec["gpu"]}))


if __name__ == "__main__":
    main()
