"""Per-timepoint wall time of the device-resident path without event timing (what bench.py's `value` sees).

    python tools/tp_wall.py C2 1.0 [chunk] [--eps 0.04] [--iters 12] [--bmin 2048]
                                  [--reps 3] [--tps 5] [--sweep "chunk=24576;iters=12"]
"""
import logging
import sys
import time

import torch

sys.path.insert(0, ".")
from chronoclust_b200.hddstream import HDDStream
from chronoclust_b200.synth import CONFIGS, config_params, gen


def opt(name, default, cast=float):
    if name in sys.argv:
        i = sys.argv.index(name)
        v = cast(sys.argv[i + 1])
        del sys.argv[i:i + 2]
        return v
    return default


eps_over = opt("--eps", None)
reps = opt("--reps", 3, int)
tps = opt("--tps", 0, int)
# several engine settings on the same data in one process: --sweep "chunk=24576;iters=12;bmin=4096,iters=16" ("" = defaults)
sweep = opt("--sweep", None, str)
settings = [dict(chunk=int(sys.argv[3]) if len(sys.argv) > 3 else 0, iters=opt("--iters", 0, int), bmin=opt("--bmin", 0, int))]
if sweep is not None:
    settings = []
    for item in sweep.split(";"):
        d = dict(chunk=0, iters=0, bmin=0)
        for kv in filter(None, item.split(",")):
            k, v = kv.split("=")
            d[k.strip()] = int(v)
        settings.append(d)
name = sys.argv[1] if len(sys.argv) > 1 else "C2"
scale = float(sys.argv[2]) if len(sys.argv) > 2 else 1.0
N, D, T, Cn, seed, eps, pi = CONFIGS[name]
N = int(N * scale)
T = tps or T
Xs = gen(N, D, T, Cn, seed)
prm = config_params(name)
if eps_over is not None:
    prm["epsilon"] = eps_over
Xd = [torch.from_numpy(x).cuda() for x in Xs]
a = torch.empty(N, dtype=torch.int32, device="cuda")
s = torch.empty(N, dtype=torch.uint8, device="cuda")
for cfg in settings:
    h = HDDStream(prm, logging.getLogger("q"), chunk=cfg["chunk"], bsv_iters=cfg["iters"], bsv_bmin=cfg["bmin"])
    h.dataset_dimensionality = D
    h._ensure_handle(D)
    print(f"# {name} x{scale} eps={eps_over} {cfg}")
    for rep in range(reps):
        h.reset()
        prev = h.stats()
        line = []
        tot = 0.0
        for t in range(T):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            h.ingest_device(Xd[t].data_ptr(), N, D, t, a.data_ptr(), s.data_ptr())
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            tot += dt
            st = h.stats()
            line.append(f"t{t} {dt*1e3:.1f}ms blocks={st['bsv_blocks']-prev['bsv_blocks']} rounds={st['bsv_rounds']-prev['bsv_rounds']} "
                        f"light={st['bsv_light_rounds']-prev['bsv_light_rounds']} "
                        f"cuts={st['bsv_cuts_unknown']-prev['bsv_cuts_unknown']}/{st['bsv_cuts_rounds']-prev['bsv_cuts_rounds']}/"
                        f"{st['bsv_cuts_capacity']-prev['bsv_cuts_capacity']} launches={st['kernel_launches']-prev['kernel_launches']}")
            prev = st
        print(f"rep {rep}: total {tot*1e3:.1f}ms | " + " | ".join(line))
    del h
