"""Exploratory timing of the CUDA path (not the bench contract): per-timepoint wall time and counters."""
import logging
import sys
import time

import numpy as np

sys.path.insert(0, ".")
from chronoclust_b200.hddstream import HDDStream
from chronoclust_b200.synth import CONFIGS, config_params, gen

name = sys.argv[1] if len(sys.argv) > 1 else "C2"
scale = float(sys.argv[2]) if len(sys.argv) > 2 else 1.0
N, D, T, Cn, seed, eps, pi = CONFIGS[name]
N = int(N * scale)
t0 = time.time()
Xs = gen(N, D, T, Cn, seed)
print(f"gen {time.time()-t0:.1f}s  N={N} D={D} T={T}")
chunk = int(sys.argv[4]) if len(sys.argv) > 4 else 0
iters = int(sys.argv[5]) if len(sys.argv) > 5 else 0
if "--chain" in sys.argv:  # per-key cycle counters of the replay kernel: only the debug build has them (build.py --debug)
    from chronoclust_b200 import _lib as _l0, build as _b0
    _l0.SO_PATH = _b0.build(debug=True)
h = HDDStream(config_params(name), logging.getLogger("q"), chunk=chunk, bsv_iters=iters)
prev = None
h._ensure_handle(D)
h.enable_timing()
for t, X in enumerate(Xs):
    t0 = time.time()
    h.online_microcluster_maintenance(X, t, run_offline=False)
    t1 = time.time()
    h.offline_clustering(t)
    t2 = time.time()
    st = h.stats()
    d = {k: st[k] - (prev[k] if prev else 0) for k in st}
    prev = st
    c = h.counts()
    print(f"t={t} online {t1-t0:.3f}s offline {t2-t1:.3f}s  {N/(t2-t0):.0f} cells/s  pcore={c[0]} outlier={c[1]} "
          f"clusters={len(h.final_clusters)}")
    print("   ", {k: v for k, v in d.items() if v})
    print("    gpu ms:", {k: (round(v[0], 2), v[1]) for k, v in h.timing(reset=True).items() if v[1]})
    if "--chain" in sys.argv:
        import ctypes as C
        from chronoclust_b200 import _lib
        buf = np.zeros((64, 8), dtype=np.int64)
        fn = _lib.lib().ccb_debug_chain
        fn.restype, fn.argtypes = C.c_int, [C.c_void_p, C.c_void_p, C.c_int32]
        _lib.check(fn(h._h, buf.ctypes.data_as(C.c_void_p), 64), h._h)
        print("    chain_p last launch [members, replay cyc, wait, mixed-stage cyc, contested, head cyc, tail cyc, clean stages]:")
        for j in np.argsort(-buf[:, 0])[:6]:
            print("      key", j, buf[j].tolist())
