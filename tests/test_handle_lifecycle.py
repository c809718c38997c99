"""Life cycle of a handle (-m gpu): reset and rerun, per-category timing switched on and off, recovery from a refused
allocation, and many handles created and destroyed.  Every run is compared with a stress golden bit for bit."""
import numpy as np
import pytest

from helpers import assert_clusters_equal, assert_list_equal, config_of, load, stress_inputs
from test_gpu_parity import clusters_of, make

pytestmark = pytest.mark.gpu

ENGINE_CATEGORIES = ("chain_p", "nearest", "verify", "speculate", "lists", "chain_o", "olist", "derive", "decide", "commit")


def golden():
    z = load("stress_downgrade.npz")  # 4 timepoints of 2 500 cells, decay and outlier deletions from the second one on
    return z, stress_inputs(z)


def run_series(h, z, Xs, what, steps=None):
    """Feeds timepoints `steps` (default: all) to h and compares h with the golden after each one."""
    ts = z["timestamps"].tolist()
    for i in range(len(ts)) if steps is None else steps:
        h.online_microcluster_maintenance(Xs[i], int(ts[i]))
        P = f"t{i}_"
        assert (h.last_assignment == z[P + "assign"]).all(), f"{what} t{i}: assignments differ"
        for which, name in ((0, "p_"), (1, "o_")):
            assert_list_equal(h.export_arrays(which), z, P + name, f"{what} t{i} list{which}")
        assert h.counts()[2:] == z[P + "counters"].tolist()
        assert_clusters_equal(clusters_of(h), z, P, f"{what} t{i}")


def test_reset_and_rerun_on_one_handle():
    z, Xs = golden()
    h = make(config_of(z))
    run_series(h, z, Xs, "first pass")
    h.reset()
    run_series(h, z, Xs, "after reset")
    assert h.stats()["points"] == 2 * sum(len(X) for X in Xs)


def test_timing_on_then_off_keeps_results():
    z, Xs = golden()
    h = make(config_of(z))
    h._ensure_handle(Xs[0].shape[1])
    h.enable_timing(True)
    run_series(h, z, Xs, "timing on", steps=[0, 1])
    t = h.timing(reset=True)
    for cat in ENGINE_CATEGORIES + ("maintenance", "offline", "copy"):
        assert t[cat][1] > 0, f"no timed launches in category {cat}: {t}"
    assert sum(ms for ms, _ in t.values()) > 0.0
    h.enable_timing(False)
    run_series(h, z, Xs, "timing off", steps=range(2, len(Xs)))
    assert all(n == 0 for _, n in h.timing().values())


def test_refused_allocation_leaves_handle_usable():
    from chronoclust_b200 import _lib

    z, Xs = golden()
    h = make(config_of(z))
    D = Xs[0].shape[1]
    h._ensure_handle(D)
    L = _lib.lib()
    _lib.check(L.ccb_begin_timepoint(h._h, 1.0, 0.0, D, 0, 1.0), h._h)
    # one row at a stride of 2^42 doubles: a 32 TiB staging buffer, refused before anything is copied
    x, assign, stage = np.zeros(D), np.zeros(1, np.int32), np.zeros(1, np.uint8)
    with pytest.raises(_lib.CCBError, match=r"error -3:"):
        _lib.check(L.ccb_ingest(h._h, _lib.ptr(x), 1, 1 << 42, _lib.ptr(assign), _lib.ptr(stage)), h._h)
    run_series(h, z, Xs, "after a refused allocation")


def test_handle_churn():
    z, Xs = golden()
    D = Xs[0].shape[1]
    for k in range(16):
        h = make(config_of(z))
        if k % 3 == 0:
            h._ensure_handle(D)  # created, never used
        elif k % 3 == 1:
            run_series(h, z, Xs, f"churn {k}", steps=[0])
        else:
            run_series(h, z, Xs, f"churn {k}", steps=[0, 1, 2])  # two decays: both graph slots were built
            assert h.stats()["bsv_blocks"] > 0
        del h
    run_series(make(config_of(z)), z, Xs, "after churn")
