"""Per-group cell statistics on the device (ccb_group_stats / ccb_cluster_stats, chronoclust_b200.cellstats,
HDDStream.cluster_statistics, app.run(cluster_statistics=True)) against numpy: counts, medians and linear quantiles bit for
bit, means to rounding and identical from call to call; the handle that computes them is unchanged by it."""
import csv
import logging
import os
import pickle

import numpy as np
import pytest

from helpers import STRESS_NAMES, config_of, load, stress_inputs
from test_input_paths import assert_same

LOG = logging.getLogger("test")
gpu = pytest.mark.gpu
QS = [0.0, 0.1, 0.25, 0.5, 0.75, 1.0]


# ---- numpy reference ---------------------------------------------------------------------------------------------------
def reference(V, groups, G, q=()):
    """count / mean / median / quantiles of every group of the rows V [N][D] (float64), and mean(|x|) for the tolerance"""
    D = V.shape[1]
    cnt = np.zeros(G, np.int64)
    mean, med, scale = (np.full((G, D), np.nan) for _ in range(3))
    qu = np.full((len(q), G, D), np.nan)
    order = np.argsort(groups, kind="stable")
    sg = groups[order]
    for g in range(G):
        x = V[order[np.searchsorted(sg, g, "left"):np.searchsorted(sg, g, "right")]]
        cnt[g] = len(x)
        if len(x) == 0:
            continue
        with np.errstate(all="ignore"):
            mean[g] = x.mean(axis=0)
            scale[g] = np.abs(x).mean(axis=0)
            med[g] = np.median(x, axis=0)
            if len(q):
                qu[:, g] = np.quantile(x, q, axis=0, method="linear")
    return cnt, mean, med, qu, scale


def same(a, b):
    """equal values (the sign of a zero free), NaN equal to NaN"""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and bool(((a == b) | (np.isnan(a) & np.isnan(b))).all())


def check(got, V, groups, G, q, what):
    cnt, mean, med, qu, scale = reference(V, groups, G, q)
    assert (got.count == cnt).all(), f"{what}: counts"
    assert same(got.median, med), f"{what}: medians differ at {np.argwhere(~((got.median == med) | np.isnan(med)))[:5]}"
    assert same(got.quantiles, qu), f"{what}: quantiles differ"
    exact = (got.mean == mean) | (np.isnan(got.mean) & np.isnan(mean))
    with np.errstate(invalid="ignore"):
        close = np.abs(got.mean - mean) <= 1e-12 * scale
    assert (exact | close).all(), f"{what}: means differ beyond 1e-12 mean(|x|)"


def bits(st):
    return [np.ascontiguousarray(a).view(np.uint8).tobytes() for a in st]


# ---- stateless kernel ----------------------------------------------------------------------------------------------------
def _run(X, groups, G, q, what, rows=None):
    from chronoclust_b200.cellstats import group_statistics

    got = group_statistics(X, groups, G, q)
    g = groups.cpu().numpy() if hasattr(groups, "cpu") else np.asarray(groups)
    check(got, np.asarray(rows if rows is not None else X, np.float64), g, G, q, what)
    assert bits(got) == bits(group_statistics(X, groups, G, q)), f"{what}: two calls differ"
    return got


@gpu
@pytest.mark.parametrize("D", [1, 3, 12, 40, 64])
def test_group_stats_balanced_groups_with_skipped_rows(D):
    """seven groups of ~2500 cells (one slice each) plus one of ~10000 (radix select), -1 rows left out"""
    rng = np.random.default_rng(D)
    N = 30000
    X = rng.normal(size=(N, D)) * rng.uniform(0.01, 100, D)
    g = rng.integers(-1, 8, N)
    g[rng.random(N) < 0.3] = 7
    _run(X, g, 8, QS, f"D={D}")


@gpu
@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_group_stats_row_strided_cuda_views(dtype):
    import torch

    rng = np.random.default_rng(3)
    N, D = 20000, 12
    big = torch.from_numpy(rng.normal(size=(N, D + 5))).to("cuda", getattr(torch, dtype))
    view = big[:, 2:2 + D]
    g = rng.integers(-1, 3, N)
    _run(view, torch.from_numpy(g).cuda(), 3, QS, f"cuda {dtype} view", rows=view.double().cpu().numpy())
    _run(view.cpu().numpy(), g, 3, QS, f"numpy {dtype} view")


@gpu
def test_group_stats_one_group_holds_99_percent():
    rng = np.random.default_rng(5)
    N, D = 400000, 3
    X = rng.normal(size=(N, D))
    g = np.where(rng.random(N) < 0.99, 0, rng.integers(1, 6, N))
    _run(X, g, 6, QS, "skew")


@gpu
def test_group_stats_thousands_of_tiny_groups():
    """G = 5000: groups of size 0, 1, 2 and some of a few hundred cells"""
    rng = np.random.default_rng(9)
    sizes = np.concatenate([np.zeros(1000, int), np.ones(1500, int), np.full(1500, 2), rng.integers(3, 400, 1000)])
    rng.shuffle(sizes)
    g = np.repeat(np.arange(5000), sizes)
    rng.shuffle(g)
    X = rng.normal(size=(len(g), 4))
    got = _run(X, g, 5000, QS, "G=5000")
    assert (got.count == sizes).all() and np.isnan(got.median[sizes == 0]).all()


@gpu
@pytest.mark.parametrize("big", [False, True], ids=["sorted-in-shared-memory", "radix-select"])
def test_group_stats_duplicates_zeros_infinities_nans(big):
    rng = np.random.default_rng(11)
    N, D, G = (60000 if big else 6000), 6, 4
    X = rng.integers(-3, 4, size=(N, D)).astype(np.float64)  # heavy duplicates
    X[:, 1] = np.where(rng.random(N) < 0.5, 0.0, -0.0)
    X[rng.random(N) < 0.01, 2] = np.inf
    X[rng.random(N) < 0.01, 3] = -np.inf
    g = rng.integers(-1, G, N)
    X[np.flatnonzero(g == 2)[:1], 4] = np.nan  # one NaN in group 2, marker 4
    X[:, 5] = np.where(rng.random(N) < 0.5, np.inf, -np.inf)
    got = _run(X, g, G, QS, "special values")
    assert np.isnan(got.median[2, 4]) and not np.isnan(got.median[1, 4])


@gpu
def test_group_stats_argument_errors():
    import torch

    from chronoclust_b200 import _lib

    X = torch.zeros((10, 3), dtype=torch.float64, device="cuda")
    g = torch.zeros(10, dtype=torch.int32, device="cuda")
    out = [np.zeros(4, np.int64), np.zeros(12), np.zeros(12), np.zeros(12)]
    L = _lib.lib()

    def call(G=1, nq=0, q=None, ld=3):
        qa = None if q is None else np.ascontiguousarray(q, np.float64)
        return L.ccb_group_stats(0, None, X.data_ptr(), _lib.DTYPE_F64, 10, ld, 3, g.data_ptr(), G, nq, _lib.ptr(qa),
                                 *[_lib.ptr(a) for a in out])

    assert call() == 0 and out[0][0] == 10
    assert call(G=0) == -1
    assert call(nq=1, q=[1.5]) == -1
    assert call(nq=1, q=[np.nan]) == -1
    assert call(ld=2) == -1


# ---- handle ----------------------------------------------------------------------------------------------------------------
def fixtures():
    out = []
    for name in STRESS_NAMES + ["c1"]:
        if name == "c1":
            z = load("c1.npz")
            Xs = [z[f"scaled{t}"] for t in range(5)]
            ts = list(range(5))
        else:
            z = load(f"stress_{name}.npz")
            Xs = stress_inputs(z)
            ts = [int(t) for t in z["timestamps"]]
        out.append((name, config_of(z), Xs, ts))
    return out


KINDS = ["numpy-f64", "numpy-f32", "cuda-f64", "cuda-f32"]


@gpu
@pytest.mark.parametrize("scaled", [False, True], ids=["unscaled", "scaled"])
@pytest.mark.parametrize("kind", KINDS)
def test_cluster_statistics_equal_numpy_grouped_by_cluster_labels(kind, scaled):
    """Every stress fixture and C1, every timepoint: HDDStream.cluster_statistics equals numpy over the cells grouped by
    cluster_labels_for_points() (the unclustered ones last); a handle that never asks stays bit-identical."""
    import torch
    from sklearn.preprocessing import MinMaxScaler

    from chronoclust_b200.hddstream import HDDStream

    for name, cfg, Xs, ts in fixtures():
        D = Xs[0].shape[1]
        sk = None
        if scaled:  # raw rows far from [0, 1]; the engine scales them on the device
            Xs = [x * np.linspace(0.5, 400.0, D) - np.linspace(-3.0, 50.0, D) for x in Xs]
            sk = MinMaxScaler().fit(np.concatenate(Xs, axis=0))
        dt = np.float32 if kind.endswith("f32") else np.float64
        a, b = HDDStream(dict(cfg), LOG), HDDStream(dict(cfg), LOG)
        for t, X in zip(ts, Xs):
            X = X.astype(dt)
            feed = torch.from_numpy(X).cuda() if kind.startswith("cuda") else X
            a.online_microcluster_maintenance(feed, t, scaler=sk)
            b.online_microcluster_maintenance(X, t, scaler=sk)
            V = X.astype(np.float64)
            if sk is not None:  # what the engine read, brought back: (x * scale_ + min_ - min_) / scale_
                V = (V * sk.scale_ + sk.min_ - sk.min_) / sk.scale_
            lab = a.cluster_labels_for_points()
            G = len(a.final_clusters)
            got = a.cluster_statistics(quantiles=QS)
            check(got, V, np.where(lab < 0, G, lab), G + 1, QS, f"{name} {kind} scaled={scaled} t{t}")
            assert bits(got) == bits(a.cluster_statistics(quantiles=QS))
            assert_same(a, b, f"{name} {kind} t{t}")


@gpu
def test_cluster_statistics_with_given_groups():
    from chronoclust_b200.hddstream import HDDStream

    z = load("c1.npz")
    h = HDDStream(dict(config_of(z)), LOG)
    h.online_microcluster_maintenance(z["scaled0"], 0, run_offline=False)
    with pytest.raises(ValueError):
        h.cluster_statistics()
    uids = h.export_arrays(0)[1]
    groups = np.arange(len(uids)) % 2  # every pcore MC a group of its own parity
    got = h.cluster_statistics(groups=groups)
    lut = {int(u): int(c) for u, c in zip(uids, groups)}
    cell = np.array([lut.get(int(u), 2) for u in h.last_assignment])
    check(got, z["scaled0"], cell, 3, (), "given groups")


@gpu
def test_cluster_statistics_state_errors(tmp_path):
    from chronoclust_b200 import _lib
    from chronoclust_b200.hddstream import HDDStream

    z = load("c1.npz")
    cfg = config_of(z)
    h = HDDStream(dict(cfg), LOG)
    with pytest.raises(_lib.CCBError):  # before any ingest
        h.cluster_statistics(groups=np.zeros(0, np.int32))
    h.online_microcluster_maintenance(z["scaled0"], 0)
    n = len(h.last_cluster_label)
    h.cluster_statistics()
    L = _lib.lib()
    big = [np.zeros(64 * 64) for _ in range(3)]

    def call(gop, G, q=()):
        qa = np.ascontiguousarray(q, np.float64)
        return L.ccb_cluster_stats(h._h, _lib.ptr(np.ascontiguousarray(gop, np.int32)), len(gop), G, len(qa),
                                   _lib.ptr(qa) if len(qa) else None, _lib.ptr(np.zeros(64, np.int64)),
                                   *[_lib.ptr(a) for a in big])

    assert call(np.full(n, -1), 1) == 0
    assert call(np.full(n + 1, -1), 1) == -1  # wrong n_pcore
    assert call(np.full(n, -1), -1) == -1     # G < 0
    assert call(np.full(n, 0), 0) == -1       # a group >= G
    assert call(np.full(n, -1), 1, [1.5]) == -1
    assert call(np.full(n, -1), 1, [-0.1]) == -1
    # after a timepoint start, a reset, an unpickling: no ingest to summarise
    L.ccb_begin_timepoint(h._h, float(h.mu), float(h.omicron), int(h.pi), 0, 1.0)
    assert call(np.full(n, -1), 1) == -4
    with pytest.raises(_lib.CCBError):
        h.cluster_statistics()
    h.online_microcluster_maintenance(z["scaled1"], 1)
    h.cluster_statistics()
    r = pickle.loads(pickle.dumps(h))
    with pytest.raises(_lib.CCBError):
        r.cluster_statistics(groups=np.full(len(r.export_arrays(0)[0]), -1))
    h.reset()
    with pytest.raises(_lib.CCBError):
        h.cluster_statistics(groups=np.full(len(h.export_arrays(0)[0]), -1))


# ---- app.run ----------------------------------------------------------------------------------------------------------------
def _c1_files(tmp_path, rows=None):
    import pandas as pd

    z = load("c1.npz")
    files = []
    for t in range(5):
        f = tmp_path / f"d{t}.csv"
        pd.DataFrame(z[f"raw{t}"][:rows], columns=["x", "y", "z"]).to_csv(f, index=False)
        files.append(str(f))
    return z, files


def _run_app(files, out, cfg, stats):
    from chronoclust_b200 import app

    out.mkdir()
    app.run(data=files, output_directory=str(out), param_beta=cfg["beta"], param_delta=cfg["delta"],
            param_epsilon=cfg["epsilon"], param_lambda=cfg["lambda"], param_k=cfg["k"], param_mu=cfg["mu"],
            param_pi=cfg["pi"], param_omicron=cfg["omicron"], param_upsilon=cfg["upsilon"], cluster_statistics=stats)


@gpu
def test_app_run_writes_cluster_statistics(tmp_path):
    import pandas as pd

    z, files = _c1_files(tmp_path)
    cfg = config_of(z)
    _run_app(files, tmp_path / "plain", cfg, False)
    _run_app(files, tmp_path / "stats", cfg, True)
    assert not os.path.exists(tmp_path / "plain" / "cluster_statistics.csv")
    for f in ["result.csv"] + [f"cluster_points_D{t}.csv" for t in range(5)]:
        assert open(tmp_path / "plain" / f, "rb").read() == open(tmp_path / "stats" / f, "rb").read(), f
    with open(tmp_path / "stats" / "result.csv") as f:
        result = list(csv.reader(f))
    col = result[0].index("tracking_by_lineage")
    with open(tmp_path / "stats" / "cluster_statistics.csv") as f:
        rows = list(csv.reader(f))
    assert rows[0] == ["timepoint", "tracking_by_lineage", "cell_count", "median_x", "median_y", "median_z", "mean_x",
                       "mean_y", "mean_z"]
    rows = rows[1:]
    for t in range(5):
        pts = pd.read_csv(tmp_path / "stats" / f"cluster_points_D{t}.csv", keep_default_na=False,
                          float_precision="round_trip")
        labels = list(dict.fromkeys(r[col] for r in result[1:] if r[0] == str(t))) + ["None"]
        mine = [r for r in rows if r[0] == str(t)]
        assert [r[1] for r in mine] == labels, f"t{t}: label rows"
        for r in mine:
            x = pts.loc[pts["cluster_id"].astype(str) == r[1], ["x", "y", "z"]].to_numpy(np.float64)
            assert int(r[2]) == len(x)
            got = np.array([float(v) for v in r[3:]])
            if len(x) == 0:
                assert np.isnan(got).all()
                continue
            assert same(got[:3], np.median(x, axis=0)), f"t{t} {r[1]}: medians"
            assert (np.abs(got[3:] - x.mean(axis=0)) <= 1e-12 * np.abs(x).mean(axis=0)).all(), f"t{t} {r[1]}: means"
            assert all(repr(float(v)) == v for v in r[3:])  # Python float repr: round-trips


@gpu
def test_app_run_cluster_statistics_without_clusters(tmp_path):
    z, files = _c1_files(tmp_path, rows=10)
    cfg = dict(beta=1, delta=0.05, epsilon=0.03, **{"lambda": 2}, k=4, mu=1, pi=3, omicron=0.000000435, upsilon=6.5)
    _run_app(files, tmp_path / "out", cfg, True)
    with open(tmp_path / "out" / "cluster_statistics.csv") as f:
        rows = list(csv.reader(f))[1:]
    assert [(r[0], r[1], r[2]) for r in rows] == [(str(t), "None", "10") for t in range(5)]


# ---- CPU: argument checks and row assembly -----------------------------------------------------------------------------------
def test_quantile_validation():
    from chronoclust_b200.cellstats import quantile_array

    assert quantile_array([0, 0.5, 1]).tolist() == [0.0, 0.5, 1.0]
    assert quantile_array(()).shape == (0,)
    for bad in ([1.5], [-0.1], [np.nan], [0.5, np.inf]):
        with pytest.raises(ValueError):
            quantile_array(bad)


def test_group_statistics_validates_before_any_device_call():
    pytest.importorskip("torch")
    from chronoclust_b200.cellstats import group_statistics

    X = np.zeros((5, 3))
    for args in [(X, np.zeros(4, int), 1), (X, np.zeros(5, int), 0), (X, np.full(5, 2), 2), (X, np.full(5, -2), 2),
                 (X, np.zeros(5), 1), (np.zeros(5), np.zeros(5, int), 1), (np.zeros((5, 65)), np.zeros(5, int), 1)]:
        with pytest.raises(ValueError):
            group_statistics(*args)
    with pytest.raises(ValueError):
        group_statistics(X, np.zeros(5, int), 1, quantiles=[np.nan])


def test_statistics_rows_order_merge_none_and_float_format():
    from chronoclust_b200 import app
    from chronoclust_b200.cellstats import GroupStats, statistics_rows

    class Cl(object):
        def __init__(self, cid, pcores):
            self.id, self.pcore_ids = cid, pcores

    class Fake(object):
        def export_arrays(self, which):
            return np.array([10, 11, 12, 13, 14]), np.array([4, 0, 3, 1, 2])

    # clusters in result.csv order; "B" twice (a label shared by two clusters merges), pcore 14 in none
    idx, uids, labels = app._pcore_labels(Fake(), [Cl("B", [11]), Cl("A", [10, 13]), Cl("B", [12])])
    assert labels == ["None", "B", "A"] and idx.tolist() == [2, 1, 1, 2, 0]
    st = GroupStats(np.array([3, 0, 7]), np.array([[0.1], [np.nan], [1 / 3]]), np.array([[2.5], [np.nan], [-0.0]]),
                    np.zeros((0, 3, 1)))
    rows = statistics_rows(4, labels + ["C"], st)
    assert [r[:3] for r in rows] == [[4, "B", 3], [4, "A", 0], [4, "C", 0], [4, "None", 7]]
    assert rows[0][3:] == [2.5, 0.1] and np.isnan(rows[1][3:]).all() and np.isnan(rows[2][3:]).all()
    import io

    buf = io.StringIO()
    csv.writer(buf).writerows(rows)
    line = buf.getvalue().splitlines()[-1].split(",")
    assert line == ["4", "None", "7", "-0.0", repr(1 / 3)] and float(line[4]) == 1 / 3
