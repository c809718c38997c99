#!/usr/bin/env python3
"""Time of HDDStream.cluster_statistics() per timepoint on configs C2 and C3 (synth.gen), and of the stateless
group_statistics on two shapes of grouping: one group holding 99 % of 1e6 cells, and G = 10 000 groups.

Every case is first compared with a host numpy group-by of the same values (np.median / np.mean per group, counts and
medians exactly, means to 1e-12 mean(|x|)); that group-by is also timed, for context.  Timing: a host clock around a call
that ends in a stream synchronisation (the outputs are on the host), after 3 warm-up calls, median of `--reps` calls.
Bytes: what the pipeline moves at least -- the rows read once, the column-major keys written once and read by the
median sort / radix passes -- over the HBM peak of 7.7 TB/s.  The card's name and power limit are recorded beside.

    python tools/cluster_stats.py --out DIR [--reps 20]      # writes DIR/cluster_stats.json
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
from chronoclust_b200.cellstats import group_statistics  # noqa: E402
from chronoclust_b200.hddstream import HDDStream  # noqa: E402
from chronoclust_b200.synth import CONFIGS, config_params, gen  # noqa: E402

HBM_PEAK = 7.7e12
LOG = logging.getLogger("cluster_stats")


def timed(fn, reps):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)) * 1e3, float(min(ts)) * 1e3


def host_groupby(V, groups, G):
    order = np.argsort(groups, kind="stable")
    sg = groups[order]
    cnt = np.zeros(G, np.int64)
    med, mean, scale = (np.full((G, V.shape[1]), np.nan) for _ in range(3))
    for g in range(G):
        x = V[order[np.searchsorted(sg, g):np.searchsorted(sg, g, "right")]]
        cnt[g] = len(x)
        if len(x):
            med[g], mean[g], scale[g] = np.median(x, axis=0), x.mean(axis=0), np.abs(x).mean(axis=0)
    return cnt, med, mean, scale


def equal(st, ref):
    cnt, med, mean, scale = ref
    okm = (st.median == med) | (np.isnan(st.median) & np.isnan(med))
    okn = (st.mean == mean) | (np.abs(st.mean - mean) <= 1e-12 * scale) | (np.isnan(st.mean) & np.isnan(mean))
    return bool((st.count == cnt).all() and okm.all() and okn.all())


def traffic(N, D, large_fraction, itemsize=8):
    """rows read + keys written + keys read by the sort (small groups) or by the 8 radix passes (large groups)"""
    keys = N * D * 8
    return N * D * itemsize + keys + keys * (1 + 7 * large_fraction)


def case(name, V, groups, G, reps, large_fraction):
    import torch

    Xd = torch.from_numpy(V).cuda()
    gd = torch.from_numpy(groups.astype(np.int32)).cuda()
    st = group_statistics(Xd, gd, G)
    t0 = time.perf_counter()
    ref = host_groupby(V, groups, G)
    host_ms = (time.perf_counter() - t0) * 1e3
    ms, best = timed(lambda: group_statistics(Xd, gd, G), reps)
    b = traffic(*V.shape, large_fraction)
    return {"case": name, "N": V.shape[0], "D": V.shape[1], "G": G, "equal_to_numpy": equal(st, ref), "ms_median": ms,
            "ms_min": best, "bytes": b, "bytes_over_hbm_peak_ms": b / HBM_PEAK * 1e3, "host_numpy_groupby_ms": host_ms}


def config_case(cname, reps):
    N, D, T, C, seed, *_ = CONFIGS[cname]
    h = HDDStream(config_params(cname), LOG)
    out = []
    for t, X in enumerate(gen(N, D, T, C, seed)):
        h.online_microcluster_maintenance(X, t)
        st = h.cluster_statistics()
        G = len(h.final_clusters)
        lab = h.cluster_labels_for_points()
        groups = np.where(lab < 0, G, lab)
        t0 = time.perf_counter()
        ref = host_groupby(X, groups, G + 1)
        host_ms = (time.perf_counter() - t0) * 1e3
        ms, best = timed(h.cluster_statistics, reps)
        large = float((np.bincount(groups, minlength=G + 1)[np.bincount(groups, minlength=G + 1) > 4096]).sum()) / N
        b = traffic(N, D, large)
        out.append({"case": f"{cname} t{t}", "N": N, "D": D, "G": G + 1, "equal_to_numpy": equal(st, ref), "ms_median": ms,
                    "ms_min": best, "bytes": b, "bytes_over_hbm_peak_ms": b / HBM_PEAK * 1e3, "host_numpy_groupby_ms": host_ms})
        print(json.dumps(out[-1]), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    if a.reps < 20:
        ap.error("--reps must be >= 20")
    import torch

    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this tool measures the GPU and has no CPU path")
    os.makedirs(a.out, exist_ok=True)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    rows = config_case("C2", a.reps) + config_case("C3", a.reps)
    rng = np.random.default_rng(7)
    N, D = 1_000_000, 12
    V = gen(N, D, 1, 20, 1234)[0]
    skew = np.where(rng.random(N) < 0.99, 0, rng.integers(1, 20, N))
    rows.append(case("skew: one group of 99 % of 1e6 cells", V, skew, 20, a.reps, 0.99))
    rows.append(case("balanced: 20 groups of 1e6 cells", V, rng.integers(0, 20, N), 20, a.reps, 1.0))
    rows.append(case("many groups: G = 10000", V, rng.integers(0, 10000, N), 10000, a.reps, 0.0))
    for r in rows[-3:]:
        print(json.dumps(r), flush=True)
    res = {"card": card[0] if card else "unknown", "hbm_peak_bytes_per_s": HBM_PEAK, "reps": a.reps, "cases": rows}
    with open(os.path.join(a.out, "cluster_stats.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
