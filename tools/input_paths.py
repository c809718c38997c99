#!/usr/bin/env python3
"""Time per timepoint of HDDStream.online_microcluster_maintenance for every kind of input it takes without a host-side
float64 pass: float64 / float32 numpy rows (ordinary pageable memory, as a file reader hands them out) and float64 /
float32 CUDA tensors, each without and with the device min-max scaler.  numpy float64 without a scaler is the baseline
(bench.py's e2e_pageable path).  Workload: config C2 (synth.gen, 1e6 cells x 12 markers x 5 timepoints, seed 1234).

Every variant is first checked against the float64 path on the same rows widened to float64 -- assignments, stages,
both lists, counters and final clusters at every timepoint, bit for bit -- and then timed: a host clock around each call
(the call returns after its results are on the host, behind a stream synchronisation; the offline phase is included),
after one warm-up pass per variant, `--reps` passes taken in turn across the variants.

    python tools/input_paths.py --out DIR [--reps 5] [--scale 1.0]      # writes DIR/input_paths.json (one JSON line)
"""
import argparse
import json
import logging
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from chronoclust_b200.hddstream import HDDStream  # noqa: E402
from chronoclust_b200.synth import CONFIGS, config_params, gen  # noqa: E402

LOG = logging.getLogger("input_paths")


def snapshot(h):
    lists = [h.export_arrays(w) for w in (0, 1)]
    cl = [(c.members_in_claim_order, c.cumulative_weight, c.CF1, c.CF2, c.cluster_centroids,
           c.preferred_dimension_vector) for c in h.final_clusters]
    return h.last_assignment.copy(), h.last_stage.copy(), lists, h.counts(), cl


def same_bits(a, b):
    a, b = np.ascontiguousarray(a, np.float64), np.ascontiguousarray(b, np.float64)
    return a.shape == b.shape and (a.view(np.uint64) == b.view(np.uint64)).all()


def snapshots_equal(s, r):
    (a1, s1, l1, c1, k1), (a2, s2, l2, c2, k2) = s, r
    if not ((a1 == a2).all() and (s1 == s2).all() and c1 == c2 and len(k1) == len(k2)):
        return False
    for x, y in zip(l1, l2):
        if len(x[0]) != len(y[0]) or not ((x[0] == y[0]).all() and (x[1] == y[1]).all()):
            return False
        if not all(same_bits(p, q) for p, q in zip(x[2:], y[2:])):
            return False
    return all(list(m1) == list(m2) and same_bits(w1, w2) and all(same_bits(p, q) for p, q in zip(r1, r2))
               for (m1, w1, *r1), (m2, w2, *r2) in zip(k1, k2))


def run(h, Xs, scaler, times=None):
    h.reset()
    snaps = []
    for t, X in enumerate(Xs):
        t0 = time.perf_counter()
        h.online_microcluster_maintenance(X, t, scaler=scaler)
        if times is not None:
            times[t].append(time.perf_counter() - t0)
        else:
            snaps.append(snapshot(h))
    return snaps


def card(dev):
    import torch

    name = torch.cuda.get_device_name(dev)
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return {"gpu": name, "power_limit_and_max_sm_clock": q}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True, help="directory for input_paths.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of C2's cells per timepoint")
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args()
    import torch
    from sklearn.preprocessing import MinMaxScaler

    if not torch.cuda.is_available():
        sys.exit("input_paths.py measures on a CUDA device; none is visible")
    dev = args.device
    torch.cuda.set_device(dev)
    N, D, T, Cn, seed, _eps, _pi = CONFIGS["C2"]
    N = int(N * args.scale)
    cfg = config_params("C2")
    X64 = gen(N, D, T, Cn, seed)
    # raw rows for the scaled variants: markers on scales from 0.01 to 1e4, as a cytometer exports them
    sc = np.array([3.0, 250.0, 0.01, 17.0, 1e4, 2.0, 41.0, 0.5, 7.0, 900.0, 1.5, 60.0])[:D]
    sh = np.array([1.0, 100.0, 0.0, -4.0, 5e3, 0.5, -20.0, 0.25, 3.0, -450.0, 0.0, 30.0])[:D]
    R64 = [x * sc - sh for x in X64]
    sk = MinMaxScaler().fit(np.concatenate(R64, axis=0))
    X32 = [x.astype(np.float32) for x in X64]
    R32 = [x.astype(np.float32) for x in R64]
    cuda = lambda xs: [torch.from_numpy(x).cuda(dev) for x in xs]
    # name: (inputs, scaler, authority = the float64 numpy rows whose results the variant must reproduce)
    variants = {
        "numpy_f64": (X64, None, X64),
        "numpy_f64_scaled": (R64, sk, R64),
        "numpy_f32": (X32, None, [x.astype(np.float64) for x in X32]),
        "numpy_f32_scaled": (R32, sk, [x.astype(np.float64) for x in R32]),
        "cuda_f64": (cuda(X64), None, X64),
        "cuda_f64_scaled": (cuda(R64), sk, R64),
        "cuda_f32": (cuda(X32), None, [x.astype(np.float64) for x in X32]),
        "cuda_f32_scaled": (cuda(R32), sk, [x.astype(np.float64) for x in R32]),
    }
    handles = {k: HDDStream(cfg, LOG, device=dev) for k in variants}
    ref = HDDStream(cfg, LOG, device=dev)
    parity = {}
    for name, (xs, scaler, auth) in variants.items():  # (also the warm-up pass of every variant)
        parity[name] = all(snapshots_equal(s, r) for s, r in zip(run(handles[name], xs, scaler),
                                                                   run(ref, auth, scaler)))
    times = {k: [[] for _ in range(T)] for k in variants}
    for _ in range(args.reps):
        for name, (xs, scaler, _auth) in variants.items():
            run(handles[name], xs, scaler, times[name])
    res = {}
    for name, per_t in times.items():
        ms = np.array(per_t) * 1e3  # [T][reps]
        med = np.median(ms, axis=1)
        res[name] = {"ms_per_timepoint_median": [round(float(v), 3) for v in med],
                     "ms_per_timepoint_min": [round(float(v), 3) for v in ms.min(axis=1)],
                     "ms_per_timepoint_max": [round(float(v), 3) for v in ms.max(axis=1)],
                     "cells_per_s_median": float(N * T / (med.sum() * 1e-3)),
                     "bit_identical_to_float64_path": bool(parity[name])}
    base = res["numpy_f64"]["cells_per_s_median"]
    for r in res.values():
        r["vs_numpy_f64"] = round(r["cells_per_s_median"] / base, 3)
    out = {"metric": "online_microcluster_maintenance wall time per timepoint by input kind (offline phase included)",
           "workload": f"C2: {N} cells x {D} markers x {T} timepoints, synth.gen seed {seed}",
           "timing": f"host clock per call, 1 warm-up pass then {args.reps} passes alternating the variants",
           "card": card(dev), "variants": res}
    os.makedirs(args.out, exist_ok=True)
    line = json.dumps(out)
    with open(os.path.join(args.out, "input_paths.json"), "w") as f:
        f.write(line + "\n")
    print(line)
    if not all(parity.values()):
        sys.exit("a variant differs from the float64 path: " + ", ".join(k for k, v in parity.items() if not v))


if __name__ == "__main__":
    main()
