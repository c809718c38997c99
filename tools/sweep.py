#!/usr/bin/env python3
"""Config C5 (BASELINE.json configs[4]): epsilon x upsilon x beta parameter sweep, 64 independent runs of the C2
workload, partitioned over the ranks (no data-path collective -- every run is its own ordered stream).  The runs differ
60x in cost (eps = 0.04 saturates the microclusters), so they are handed out dynamically: costliest first (smallest eps,
largest beta), every rank takes the next one from a shared counter (a TCPStore key -- control plane only).  The dataset is replicated on every device once; each run is a fresh handle fed device-resident
timepoints through ccb_ingest_device.  Prints one JSON line on rank 0.

    python tools/sweep.py [--scale 1.0]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 tools/sweep.py
"""
import argparse
import itertools
import json
import logging
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from chronoclust_b200.hddstream import HDDStream  # noqa: E402
from chronoclust_b200.synth import CONFIGS, config_params, gen  # noqa: E402

GRID = list(itertools.product((0.04, 0.045, 0.05, 0.055), (4.0, 5.5, 6.5, 8.0), (0.1, 0.2, 0.4, 0.8)))  # SURVEY 8d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--configs", type=int, default=len(GRID))
    a = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    N, D, T, Cn, seed, _, _ = CONFIGS["C2"]
    N = max(1000, int(N * a.scale))
    Xd = [torch.from_numpy(x).cuda(local) for x in gen(N, D, T, Cn, seed)]
    assign = torch.empty(N, dtype=torch.int32, device=f"cuda:{local}")
    stage = torch.empty(N, dtype=torch.uint8, device=f"cuda:{local}")
    grid = GRID[::max(1, len(GRID) // a.configs)][:a.configs] if a.configs < len(GRID) else GRID
    order = sorted(range(len(grid)), key=lambda i: (grid[i][0], -grid[i][2], grid[i][1]))  # costliest first
    store = None
    if world > 1:
        port = int(os.environ.get("MASTER_PORT", "29500")) + 17
        store = dist.TCPStore(os.environ.get("MASTER_ADDR", "127.0.0.1"), port, world, is_master=(rank == 0))

    def next_job():
        """Index into `order` of the next run nobody has taken yet (shared counter; single rank: a local one)."""
        if store is None:
            next_job.n += 1
            return next_job.n - 1
        return store.add("next_run", 1) - 1

    next_job.n = 0

    def run(i):
        eps, ups, beta = grid[i]
        cfg = dict(config_params("C2"), epsilon=eps, upsilon=ups, beta=beta)
        t0 = time.perf_counter()
        h = HDDStream(cfg, logging.getLogger("sweep"), device=local)
        h.dataset_dimensionality = D
        h._ensure_handle(D)
        for t in range(T):
            h.ingest_device(Xd[t].data_ptr(), N, D, t, assign.data_ptr(), stage.data_ptr())
        c = h.counts()
        torch.cuda.synchronize()
        st = h.stats()
        return {"epsilon": eps, "upsilon": ups, "beta": beta, "pcore": int(c[0]), "outlier": int(c[1]),
                "clusters": len(h.final_clusters), "seconds": round(time.perf_counter() - t0, 3),
                "blocks": st["bsv_blocks"], "rounds": st["bsv_rounds"], "outlier_stage_cells": st["bsv_outlier_stage_cells"],
                "cuts": [st["bsv_cuts_unknown"], st["bsv_cuts_rounds"], st["bsv_cuts_capacity"]]}

    run(order[-1])  # warm-up (module load, workspace growth) on the cheapest configuration
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    e0.record()
    res = []
    while True:
        j = next_job()
        if j >= len(order):
            break
        r = run(order[j])
        r["rank"] = rank
        res.append(r)
    e1.record()
    torch.cuda.synchronize()
    sec = e0.elapsed_time(e1) * 1e-3
    wall = time.perf_counter() - w0
    if dist is not None:
        tt = torch.tensor([sec, wall], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        sec, wall = float(tt[0]), float(tt[1])
        allres = [None] * world
        dist.all_gather_object(allres, res)
        res = [r for rr in allres for r in rr]
    if rank == 0:
        cells = len(grid) * N * T
        print(json.dumps({"metric": "cells/sec over the whole parameter sweep", "value": cells / sec, "unit": "cells/s",
                          "n_gpus": world, "configs": len(grid), "cells_per_config": N * T, "seconds": sec,
                          "wall_s": wall, "scaling": "strong",
                          "partition": "dynamic: costliest configuration first, shared counter, no data-path collective",
                          "runs_per_rank": [sum(1 for r in res if r.get("rank") == g) for g in range(world)],
                          "clusters_min_max": [min(r["clusters"] for r in res), max(r["clusters"] for r in res)],
                          "seconds_per_run_min_median_max": [min(r["seconds"] for r in res),
                                                             sorted(r["seconds"] for r in res)[len(res) // 2],
                                                             max(r["seconds"] for r in res)],
                          "slowest_over_fastest": max(r["seconds"] for r in res) / max(min(r["seconds"] for r in res), 1e-9),
                          "runs": res}))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
