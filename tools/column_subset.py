#!/usr/bin/env python3
"""Clustering on a subset of the columns of wider rows: HDDStream.online_microcluster_maintenance(columns=) -- the gather
on the device -- against a gather by the caller (numpy fancy indexing / torch index_select) followed by a plain ingest.
Workload: config C3's cells (synth.gen, 2e6 cells x 40 markers x 5 timepoints, seed 1234) placed in rows 56 wide, the
40 markers at the non-contiguous columns {j < 56 : j % 7 not in (2, 5)} and uniform noise in the other 16.  Every input
kind (numpy float64 / float32, CUDA float64 / float32), without and with the device min-max scaler.

Every variant is first checked against the float64 path on the gathered rows -- assignments, stages, both lists,
counters and final clusters at every timepoint, bit for bit -- and then timed: a host clock around each call including
the caller's gather (the call returns after its results are on the host; the offline phase is included), after that
checking pass, `--reps` passes alternating the two forms.  cluster_statistics over all 56 columns is timed after the
last timepoint of each `columns=` variant, and its clustering columns are checked bit for bit against the statistics of
the gathered ingest.  One input kind's rows are held at a time.

    python tools/column_subset.py --out DIR [--reps 3] [--scale 1.0]      # writes DIR/column_subset.json (one JSON line)
"""
import argparse
import json
import logging
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from chronoclust_b200.hddstream import HDDStream  # noqa: E402
from chronoclust_b200.synth import CONFIGS, config_params, gen  # noqa: E402
from input_paths import card, snapshot, snapshots_equal  # noqa: E402

LOG = logging.getLogger("column_subset")
W = 56
COLS = [j for j in range(W) if j % 7 not in (2, 5)]  # 40 columns


def run(h, Xs, scaler, cols, gather, times=None):
    """one pass over the timepoints; gather: the caller-side gather applied before a plain ingest (cols then unused)"""
    h.reset()
    snaps = []
    for t, X in enumerate(Xs):
        t0 = time.perf_counter()
        if gather is not None:
            h.online_microcluster_maintenance(gather(X), t, scaler=scaler)
        else:
            h.online_microcluster_maintenance(X, t, scaler=scaler, columns=cols)
        if times is not None:
            times[t].append(time.perf_counter() - t0)
        else:
            snaps.append(snapshot(h))
    return snaps


def stats_bits(st, cols=None):
    arrs = (st.count, st.mean, st.median) if cols is None else (st.count, st.mean[:, cols], st.median[:, cols])
    return [np.ascontiguousarray(a).tobytes() for a in arrs]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True, help="directory for column_subset.json")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of C3's cells per timepoint")
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args()
    import torch
    from sklearn.preprocessing import MinMaxScaler

    if not torch.cuda.is_available():
        sys.exit("column_subset.py measures on a CUDA device; none is visible")
    dev = args.device
    torch.cuda.set_device(dev)
    N, D, T, Cn, seed, _eps, _pi = CONFIGS["C3"]
    N = int(N * args.scale)
    cfg = config_params("C3")
    rng = np.random.default_rng(seed)
    X = gen(N, D, T, Cn, seed)
    scale = np.linspace(0.01, 1e4, D)  # raw rows of the scaled variants: markers on scales from 0.01 to 1e4
    R = [x * scale - 3.0 for x in X]
    del X
    sk = MinMaxScaler().fit(np.concatenate(R, axis=0))

    def wide(xs, transform=None):
        out = []
        for x in xs:
            w = rng.uniform(-50.0, 50.0, size=(N, W))
            w[:, COLS] = x if transform is None else transform(x)
            out.append(w)
        return out

    # the rows the engine clusters: C3's cells (unscaled) or their raw counterparts (scaled), 56 wide
    base = {"unscaled": wide(R, sk.transform), "scaled": wide(R)}
    del R
    scalers = {"unscaled": None, "scaled": sk}
    ref = HDDStream(cfg, LOG, device=dev)
    authority = {}
    for s, xs in base.items():
        authority[s] = run(ref, [np.ascontiguousarray(x[:, COLS]) for x in xs], scalers[s], None, None)
        authority[s + "_stats"] = stats_bits(ref.cluster_statistics())
    idx = torch.tensor(COLS, device=f"cuda:{dev}")
    gathers = {"numpy": lambda x: np.ascontiguousarray(x[:, COLS]), "cuda": lambda x: x.index_select(1, idx)}
    res, parity = {}, {}
    for kind, dtype in (("numpy", np.float64), ("numpy", np.float32), ("cuda", np.float64), ("cuda", np.float32)):
        for s, xs in base.items():
            rows = [x.astype(dtype) for x in xs]
            if kind == "cuda":
                rows = [torch.from_numpy(x).cuda(dev) for x in rows]
            names = {f"{kind}_{np.dtype(dtype).name}_{s}_{form}": form for form in ("columns", "gather")}
            handles = {n: HDDStream(cfg, LOG, device=dev) for n in names}
            if dtype == np.float32:  # the authority of float32 rows: the float64 path on the widened float32 rows
                auth = run(ref, [np.ascontiguousarray(x[:, COLS].astype(np.float32), np.float64) for x in xs],
                           scalers[s], None, None)
                auth_stats = stats_bits(ref.cluster_statistics())
            else:
                auth, auth_stats = authority[s], authority[s + "_stats"]
            times = {n: [[] for _ in range(T)] for n in names}
            for n, form in names.items():
                g = gathers[kind] if form == "gather" else None
                parity[n] = all(snapshots_equal(a, b) for a, b in zip(run(handles[n], rows, scalers[s], COLS, g), auth))
            for _ in range(args.reps):
                for n, form in names.items():
                    run(handles[n], rows, scalers[s], COLS, gathers[kind] if form == "gather" else None, times[n])
            for n, per_t in times.items():
                ms = np.array(per_t) * 1e3  # [T][reps]
                med = np.median(ms, axis=1)
                res[n] = {"ms_per_timepoint_median": [round(float(v), 3) for v in med],
                          "ms_per_timepoint_min": [round(float(v), 3) for v in ms.min(axis=1)],
                          "ms_per_timepoint_max": [round(float(v), 3) for v in ms.max(axis=1)],
                          "cells_per_s_median": float(N * T / (med.sum() * 1e-3)),
                          "bit_identical_to_gathered_float64_path": bool(parity[n])}
            n = f"{kind}_{np.dtype(dtype).name}_{s}_columns"
            h = handles[n]  # its last pass ended on the last timepoint
            st = h.cluster_statistics()
            ok = st.mean.shape[1] == W and stats_bits(st, COLS) == auth_stats
            parity[n + "_statistics"] = ok
            sms = []
            for _ in range(3):
                t0 = time.perf_counter()
                h.cluster_statistics()
                sms.append((time.perf_counter() - t0) * 1e3)
            res[n]["cluster_statistics_56_columns_ms"] = [round(v, 3) for v in sms]
            res[n]["cluster_statistics_clustering_columns_bit_identical"] = bool(ok)
            del rows, handles
            torch.cuda.empty_cache()
    out = {"metric": "online_microcluster_maintenance wall time per timepoint, columns= vs a caller-side gather "
                     "(offline phase included)",
           "workload": f"C3 cells: {N} x {D} markers x {T} timepoints (synth.gen seed {seed}) in rows {W} wide, "
                       f"clustering columns {COLS}",
           "timing": f"host clock per call, gather included; 1 checking pass then {args.reps} passes alternating the forms",
           "card": card(dev), "variants": res}
    os.makedirs(args.out, exist_ok=True)
    line = json.dumps(out)
    with open(os.path.join(args.out, "column_subset.json"), "w") as f:
        f.write(line + "\n")
    print(line)
    if not all(parity.values()):
        sys.exit("a variant differs from the gathered float64 path: " + ", ".join(k for k, v in parity.items() if not v))


if __name__ == "__main__":
    main()
