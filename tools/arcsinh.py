#!/usr/bin/env python3
"""The arcsinh transform of cytometry intensities: HDDStream.online_microcluster_maintenance(cofactors=) -- asinh(x / c)
fused into the staging launch -- against a transform by the caller followed by a plain ingest (scaling.arcsinh on the
host -- ccbio_arcsinh_host, multithreaded -- or np.arcsinh for numpy rows; ccb_arcsinh for CUDA tensors).
Workload: config C3's cells (synth.gen, 2e6 cells x 40 markers x 5 timepoints, seed 1234) as raw intensities
raw = 5 sinh(6 x - 0.5), cofactor 5 on every marker, the engine's min-max scaler fitted on the transformed values.

Every form is first checked against the float64 path on host-transformed rows -- assignments, stages, both lists,
counters and final clusters at every timepoint, bit for bit (np.arcsinh is not the engine's definition: its check is
reported, not required) -- and then timed: a host clock around each call including the caller's transform, `--reps`
passes alternating the forms.  Then the staging launch alone (ccb_arcsinh: k_stage_rows_tx, no map, no scaler) with
CUDA events on 2e6 x 40 rows (640 MB of float64 in, larger than L2), with cofactor 5 and with cofactor 0 (the same
launch, the transform skipped), as time and bytes moved per second.

    python tools/arcsinh.py --out DIR [--reps 3] [--scale 1.0]      # writes DIR/arcsinh.json (one JSON line)
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
from chronoclust_b200 import _hostio, _lib  # noqa: E402
from chronoclust_b200.hddstream import HDDStream  # noqa: E402
from chronoclust_b200.scaling import arcsinh  # noqa: E402
from chronoclust_b200.synth import CONFIGS, config_params, gen  # noqa: E402
from input_paths import card, snapshot, snapshots_equal  # noqa: E402

LOG = logging.getLogger("arcsinh")
COF = 5.0


def run(h, Xs, scaler, form, times=None):
    """one pass over the timepoints; form: "cofactors" or a caller-side transform applied before a plain ingest"""
    h.reset()
    snaps = []
    for t, X in enumerate(Xs):
        t0 = time.perf_counter()
        if form == "cofactors":
            h.online_microcluster_maintenance(X, t, scaler=scaler, cofactors=COF)
        else:
            h.online_microcluster_maintenance(form(X), t, scaler=scaler)
        if times is not None:
            times[t].append(time.perf_counter() - t0)
        else:
            snaps.append(snapshot(h))
    return snaps


def staging_launch(dev, N, D, reps=20):
    """ms per ccb_arcsinh launch on float32 / float64 rows [N][D], cofactor 5 and 0, with CUDA events"""
    import torch

    out = {}
    y = torch.empty((N, D), dtype=torch.float64, device=f"cuda:{dev}")
    for dt in (torch.float64, torch.float32):
        x = (torch.rand((N, D), dtype=torch.float64, device=f"cuda:{dev}") * 6.0 - 0.5).sinh_().mul_(5.0).to(dt)
        code = _lib.DTYPE_F64 if dt == torch.float64 else _lib.DTYPE_F32
        for c in (COF, 0.0):
            cof = np.full(D, c)
            s = torch.cuda.current_stream(dev)
            call = lambda: _lib.check(_lib.lib().ccb_arcsinh(dev, s.cuda_stream, x.data_ptr(), code, N, D, D,
                                                             cof.ctypes.data, y.data_ptr()))
            for _ in range(3):
                call()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(s)
            for _ in range(reps):
                call()
            e1.record(s)
            e1.synchronize()
            ms = e0.elapsed_time(e1) / reps
            nbytes = N * D * (x.element_size() + 8)
            out[f"{str(dt).split('.')[-1]}_cofactor_{c:g}"] = {"ms": round(ms, 4), "GB_per_s": round(nbytes / ms / 1e6, 1)}
        del x
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", required=True, help="directory for arcsinh.json")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of C3's cells per timepoint")
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args()
    import torch
    from sklearn.preprocessing import MinMaxScaler

    if not torch.cuda.is_available():
        sys.exit("arcsinh.py measures on a CUDA device; none is visible")
    dev = args.device
    torch.cuda.set_device(dev)
    N, D, T, Cn, seed, _eps, _pi = CONFIGS["C3"]
    N = int(N * args.scale)
    cfg = config_params("C3")
    raw = [5.0 * np.sinh(6.0 * x - 0.5) for x in gen(N, D, T, Cn, seed)]
    cof = np.full(D, COF)
    sk = MinMaxScaler().fit(np.concatenate([_hostio.arcsinh_host(x, cof) for x in raw], axis=0))
    ref = HDDStream(cfg, LOG, device=dev)
    res, parity = {}, {}
    for kind, dtype in (("numpy", np.float64), ("numpy", np.float32), ("cuda", np.float64), ("cuda", np.float32)):
        rows = [x.astype(dtype) for x in raw]
        auth = run(ref, [_hostio.arcsinh_host(x, cof) for x in rows], sk, lambda x: x)
        if kind == "cuda":
            rows = [torch.from_numpy(x).cuda(dev) for x in rows]
            forms = {"cofactors": "cofactors", "ccb_arcsinh": lambda x: arcsinh(x, COF)}
        else:
            forms = {"cofactors": "cofactors", "arcsinh_host": lambda x: arcsinh(x, COF),
                     "np_arcsinh": lambda x: np.arcsinh(x / np.asarray(COF, x.dtype))}
        names = {f"{kind}_{np.dtype(dtype).name}_{f}": form for f, form in forms.items()}
        handles = {n: HDDStream(cfg, LOG, device=dev) for n in names}
        for n, form in names.items():
            parity[n] = all(snapshots_equal(a, b) for a, b in zip(run(handles[n], rows, sk, form), auth))
        times = {n: [[] for _ in range(T)] for n in names}
        for _ in range(args.reps):
            for n, form in names.items():
                run(handles[n], rows, sk, form, times[n])
        for n, per_t in times.items():
            ms = np.array(per_t) * 1e3  # [T][reps]
            med = np.median(ms, axis=1)
            res[n] = {"ms_per_timepoint_median": [round(float(v), 3) for v in med],
                      "cells_per_s_median": float(N * T / (med.sum() * 1e-3)),
                      "bit_identical_to_host_transformed_float64_path": bool(parity[n])}
        del rows, handles
        torch.cuda.empty_cache()
    out = {"metric": "online_microcluster_maintenance wall time per timepoint, cofactors= vs a caller-side transform "
                     "(offline phase included), and the staging launch alone",
           "workload": f"C3 cells: {N} x {D} markers x {T} timepoints (synth.gen seed {seed}) as 5 sinh(6 x - 0.5), "
                       f"cofactor {COF}, scaler on the transformed values",
           "timing": f"host clock per call, transform included; 1 checking pass then {args.reps} passes alternating the "
                     "forms; staging launch: CUDA events over 20 launches after 3 warm-up launches",
           "card": card(dev), "variants": res, "staging_launch_2e6x40": staging_launch(dev, 2_000_000, D)}
    os.makedirs(args.out, exist_ok=True)
    line = json.dumps(out)
    with open(os.path.join(args.out, "arcsinh.json"), "w") as f:
        f.write(line + "\n")
    print(line)
    bad = [k for k, v in parity.items() if not v and not k.endswith("np_arcsinh")]
    if bad:
        sys.exit("a variant differs from the host-transformed float64 path: " + ", ".join(bad))


if __name__ == "__main__":
    main()
