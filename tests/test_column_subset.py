"""Clustering on a subset of the columns of wider rows -- HDDStream.online_microcluster_maintenance(columns=),
ccb_ingest_cols, app.run(clustering_markers=) -- gives bit for bit what the float64 path gives on the gathered rows
X[:, cols]: assignments, stages, both lists, counters, final clusters and `points`, for every input kind, with and without
the scaler.  cluster_statistics then covers every column of the rows.  The wide rows interleave columns of NaN and of
large values with the real ones, so that a gather reading a wrong column cannot pass."""
import csv
import os

import numpy as np
import pytest

from helpers import GOLDEN, STRESS_NAMES, config_of, load, stress_inputs
from test_cluster_stats import QS, bits, check
from test_input_paths import assert_same, make

gpu = pytest.mark.gpu
KINDS = ["numpy-f64", "numpy-f32", "cuda-f64", "cuda-f32"]
FILLERS = (np.nan, 3.0e30, -7.0e29)  # (representable in float32)


def widen(X, W, cols, dtype=np.float64):
    """rows W wide holding X's column d at column cols[d], filler columns elsewhere"""
    big = np.empty((len(X), W), np.float64)
    for j in range(W):
        big[:, j] = FILLERS[j % len(FILLERS)]
    big[:, cols] = X
    return big.astype(dtype)


def pattern(D, which, rng):
    """(W, cols) for D clustering columns"""
    if which == "permuted":  # a permuted subset of slightly wider rows
        W = min(64, D + 3)
        return W, rng.permutation(W)[:D].tolist()
    if which == "noncontiguous":  # every other column, in order
        W = min(64, 2 * D + 1)
        return W, (list(range(1, 2 * D, 2)) if 2 * D <= W else sorted(rng.permutation(W)[:D].tolist()))
    return D, rng.permutation(D).tolist()  # "all": every column, shuffled


def feed(big, kind, torch=None):
    if kind.startswith("cuda"):
        return torch.from_numpy(big).cuda()
    return big


def fixtures():
    out = []
    for name in STRESS_NAMES + ["c1"]:
        if name == "c1":
            z = load("c1.npz")
            out.append((name, config_of(z), [z[f"scaled{t}"] for t in range(5)], list(range(5))))
        else:
            z = load(f"stress_{name}.npz")
            out.append((name, config_of(z), stress_inputs(z), [int(t) for t in z["timestamps"]]))
    return out


def scaled_series(Xs):
    """raw rows far from [0, 1] and a MinMaxScaler fitted on them"""
    from sklearn.preprocessing import MinMaxScaler

    D = Xs[0].shape[1]
    Xs = [x * np.linspace(0.5, 400.0, D) - np.linspace(-3.0, 50.0, D) for x in Xs]
    return Xs, MinMaxScaler().fit(np.concatenate(Xs, axis=0))


def run_cols(cfg, Xs, ts, W, cols, kind, sk, what, **kw):
    """authority: the float64 host path on the gathered rows; other: columns= on the wide rows of `kind`"""
    import torch

    dt = np.float32 if kind.endswith("f32") else np.float64
    a, b = make(cfg, **kw), make(cfg, **kw)
    for t, X in zip(ts, Xs):
        big = widen(X, W, cols, dt)
        x = feed(big, kind, torch)
        before = big.copy() if isinstance(x, np.ndarray) else x.clone()
        a.online_microcluster_maintenance(np.ascontiguousarray(big[:, cols], np.float64), t, scaler=sk)
        b.online_microcluster_maintenance(x, t, scaler=sk, columns=cols)
        if isinstance(x, np.ndarray):
            assert before.tobytes() == x.tobytes(), f"{what}: the caller's rows were written"
        else:
            assert torch.equal(before.view(torch.uint8), x.view(torch.uint8)), f"{what}: the caller's tensor was written"
        assert b.dataset_dimensionality == len(cols)
        assert_same(a, b, f"{what} t{t}", points=True)
    return a, b


# ---- bit-exact against the gathered float64 path ---------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("scaled", [False, True], ids=["unscaled", "scaled"])
@pytest.mark.parametrize("kind", KINDS)
def test_columns_equal_the_gathered_float64_path(kind, scaled):
    """Every stress fixture and C1, each with a permuted, a non-contiguous and an all-columns-shuffled pattern"""
    rng = np.random.default_rng(2 * KINDS.index(kind) + scaled)
    for name, cfg, Xs, ts in fixtures():
        sk = None
        if scaled:
            Xs, sk = scaled_series(Xs)
        for which in ("permuted", "noncontiguous", "all"):
            W, cols = pattern(Xs[0].shape[1], which, rng)
            run_cols(cfg, Xs, ts, W, cols, kind, sk, f"{name} {kind} scaled={scaled} {which} W={W} cols={cols}")


@gpu
@pytest.mark.parametrize("D,W", [(1, 5), (13, 29), (24, 50), (40, 56), (64, 64)])
@pytest.mark.parametrize("kind", KINDS)
def test_columns_width_classes(kind, D, W):
    """a single column, D = 13 / 24 / 40 out of wider rows (several padded width classes of the engine), and D = 64 of
    W = 64 in a shuffled order; the scaler on every other kind"""
    from sklearn.preprocessing import MinMaxScaler

    from chronoclust_b200.synth import config_params, gen

    rng = np.random.default_rng(D * 100 + W)
    cols = rng.permutation(W)[:D].tolist()
    Xs = gen(6000, D, 2, 8, D + W)
    sk = None
    if kind in ("numpy-f32", "cuda-f64"):
        Xs = [x * 37.0 - 5.0 for x in Xs]
        sk = MinMaxScaler().fit(np.concatenate(Xs, axis=0))
    cfg = dict(config_params("C2"))
    run_cols(cfg, Xs, [0, 1], W, cols, kind, sk, f"{kind} D={D} W={W}")


@gpu
@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_columns_cuda_views_written_on_a_side_stream(dtype):
    """A row-strided view big[:, :W] (ld > W, NaN padding) of a CUDA tensor written on a side stream current at the time
    of the call: the handle waits for it, and the caller's tensor is bitwise unchanged."""
    import torch

    from chronoclust_b200.synth import config_params, gen

    cfg = config_params("C2")
    D, W = 12, 20
    rng = np.random.default_rng(4)
    cols = rng.permutation(W)[:D].tolist()
    a, b = make(cfg), make(cfg)
    side = torch.cuda.Stream()
    for t, X in enumerate(gen(30000, D, 2, 20, 21)):
        wide = widen(X, W, cols, getattr(np, dtype))
        src = torch.from_numpy(wide).cuda()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            big = torch.full((len(X), W + 5), float("nan"), dtype=getattr(torch, dtype), device="cuda")
            torch.cuda._sleep(50_000_000)
            big[:, :W].copy_(src)
            before = big.clone()
            b.online_microcluster_maintenance(big[:, :W], t, columns=cols)
            after = big.clone()
        torch.cuda.synchronize()
        a.online_microcluster_maintenance(np.ascontiguousarray(wide[:, cols], np.float64), t)
        assert torch.equal(before.view(torch.uint8), after.view(torch.uint8)), "the caller's tensor was written"
        assert_same(a, b, f"cuda {dtype} view t{t}", points=True)


@gpu
@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_columns_segmented_copy_pipeline(dtype):
    """N >= 262144: the W-wide host rows travel segment by segment into the staging buffer and are gathered behind each
    segment's copy; with timing on, the same rows take the single-segment branch.  A row-strided view (ld > W) too."""
    from chronoclust_b200.synth import config_params, gen

    cfg = config_params("C2")
    D, W = 12, 19
    cols = [17, 2, 5, 11, 0, 8, 14, 3, 9, 16, 6, 12]
    a, b, c, d = (make(cfg) for _ in range(4))
    c._ensure_handle(D)
    c.enable_timing(True)
    for t, X in enumerate(gen(300001, D, 2, 20, 7)):
        wide = widen(X, W, cols, getattr(np, dtype))
        padded = np.full((len(X), W + 3), np.nan, wide.dtype)
        padded[:, :W] = wide
        a.online_microcluster_maintenance(np.ascontiguousarray(wide[:, cols], np.float64), t)
        b.online_microcluster_maintenance(wide, t, columns=cols)
        c.online_microcluster_maintenance(wide, t, columns=cols)
        d.online_microcluster_maintenance(padded[:, :W], t, columns=cols)
        for h, what in ((b, "segmented"), (c, "single segment (timing)"), (d, "segmented, ld = W + 3")):
            assert_same(a, h, f"{dtype} {what} t{t}", points=(t == 1))
    assert c.timing()["copy"][1] > 0


# ---- statistics over the whole row -----------------------------------------------------------------------------------------
def whole_row_values(big, cols, sk):
    """what cluster_statistics reports after a column ingest: the raw rows widened, the clustering columns under a scaler
    transformed forth and back (two roundings each way)"""
    V = big.astype(np.float64)
    if sk is not None:
        x = V[:, cols]
        V[:, cols] = (x * sk.scale_ + sk.min_ - sk.min_) / sk.scale_
    return V


@gpu
@pytest.mark.parametrize("scaled", [False, True], ids=["unscaled", "scaled"])
@pytest.mark.parametrize("kind", KINDS)
def test_cluster_statistics_cover_every_column(kind, scaled):
    """cluster_statistics after a column ingest, on a stress fixture and C1: W columns, against a numpy group-by of the
    values above by cluster_labels_for_points()"""
    import torch

    rng = np.random.default_rng(17)
    for name, cfg, Xs, ts in [f for f in fixtures() if f[0] in ("c2like", "c1")]:
        sk = None
        if scaled:
            Xs, sk = scaled_series(Xs)
        W, cols = pattern(Xs[0].shape[1], "permuted", rng)
        dt = np.float32 if kind.endswith("f32") else np.float64
        h = make(cfg)
        for t, X in zip(ts, Xs):
            big = widen(X, W, cols, dt)
            h.online_microcluster_maintenance(feed(big, kind, torch), t, scaler=sk, columns=cols)
            lab = h.cluster_labels_for_points()
            G = len(h.final_clusters)
            got = h.cluster_statistics(quantiles=QS)
            assert got.mean.shape == (G + 1, W) and got.quantiles.shape == (len(QS), G + 1, W)
            check(got, whole_row_values(big, cols, sk), np.where(lab < 0, G, lab), G + 1, QS,
                  f"{name} {kind} scaled={scaled} t{t}")
            assert bits(got) == bits(h.cluster_statistics(quantiles=QS))
        h.online_microcluster_maintenance(np.ascontiguousarray(big[:, cols], np.float64), ts[-1] + 1, scaler=sk)
        assert h.cluster_statistics().mean.shape[1] == len(cols)  # a plain ingest: D columns again


# ---- app.run ----------------------------------------------------------------------------------------------------------------
def _files(tmp_path, tag, columns, extra):
    """C1's raw cells as CSV files with the columns `columns` (names among x, y, z and the keys of `extra`)"""
    import pandas as pd

    z = load("c1.npz")
    files = []
    for t in range(5):
        xyz = dict(zip("xyz", z[f"raw{t}"].T))
        n = len(z[f"raw{t}"])
        data = {c: (xyz[c] if c in xyz else extra[c](t, n)) for c in columns}
        f = tmp_path / f"{tag}_d{t}.csv"
        pd.DataFrame(data, columns=columns).to_csv(f, index=False)
        files.append(str(f))
    return z, files


EXTRA = {"cd3": lambda t, n: np.random.default_rng(t).normal(5e3, 900.0, n),
         "fsc": lambda t, n: np.random.default_rng(10 + t).integers(0, 260000, n).astype(np.float64),
         "nanny": lambda t, n: np.where(np.arange(n) % 7 == 0, np.nan, np.arange(n) * 0.25)}
WIDE = ["cd3", "x", "fsc", "y", "nanny", "z"]


def _run(files, out, stats=False, markers=None):
    from chronoclust_b200 import app

    z = load("c1.npz")
    cfg = config_of(z)
    out.mkdir()
    app.run(data=files, output_directory=str(out), gating_centroid_file=os.path.join(GOLDEN, "c1_gating_centroids.csv"),
            param_beta=cfg["beta"], param_delta=cfg["delta"], param_epsilon=cfg["epsilon"], param_lambda=cfg["lambda"],
            param_k=cfg["k"], param_mu=cfg["mu"], param_pi=cfg["pi"], param_omicron=cfg["omicron"],
            param_upsilon=cfg["upsilon"], cluster_statistics=stats, clustering_markers=markers)


@gpu
def test_app_run_clustering_markers(tmp_path):
    import pandas as pd

    _, narrow = _files(tmp_path, "narrow", ["x", "y", "z"], EXTRA)
    _, wide = _files(tmp_path, "wide", WIDE, EXTRA)
    _run(narrow, tmp_path / "narrow")
    _run(wide, tmp_path / "wide", stats=True, markers=["x", "y", "z"])
    got = open(tmp_path / "wide" / "result.csv", "rb").read()
    assert got == open(os.path.join(GOLDEN, "c1_result.csv"), "rb").read()
    assert got == open(tmp_path / "narrow" / "result.csv", "rb").read()
    lab = load("c1_labels.npz")
    with open(tmp_path / "wide" / "cluster_statistics.csv") as f:
        stats = list(csv.reader(f))
    assert stats[0][3:] == [f"median_{c}" for c in WIDE] + [f"mean_{c}" for c in WIDE]
    for t in range(5):
        w = pd.read_csv(tmp_path / "wide" / f"cluster_points_D{t}.csv", keep_default_na=False, float_precision="round_trip",
                        na_values=[""])
        n = pd.read_csv(tmp_path / "narrow" / f"cluster_points_D{t}.csv", keep_default_na=False,
                        float_precision="round_trip")
        parsed = pd.read_csv(wide[t])
        assert list(w.columns) == ["id", "cluster_id"] + WIDE
        assert (w["id"].to_numpy() == lab[f"ids{t}"]).all()
        assert (w["cluster_id"].astype(str).to_numpy() == lab[f"labels{t}"]).all()
        assert (w[["x", "y", "z"]].to_numpy() == n[["x", "y", "z"]].to_numpy()).all()
        for c in ("cd3", "fsc", "nanny"):
            a, b = w[c].to_numpy(np.float64), parsed[c].to_numpy(np.float64)
            assert ((a == b) | (np.isnan(a) & np.isnan(b))).all(), f"t{t} {c}"
        for r in (r for r in stats[1:] if r[0] == str(t)):
            x = w.loc[w["cluster_id"].astype(str) == r[1], WIDE].to_numpy(np.float64)
            assert int(r[2]) == len(x)
            got = np.array([float(v) for v in r[3:]])
            if len(x) == 0:
                continue
            with np.errstate(invalid="ignore"):
                med, mean, scale = np.median(x, axis=0), x.mean(axis=0), np.abs(x).mean(axis=0)
                assert ((got[:6] == med) | (np.isnan(got[:6]) & np.isnan(med))).all(), f"t{t} {r[1]}: medians"
                close = (np.abs(got[6:] - mean) <= 1e-12 * scale) | (np.isnan(got[6:]) & np.isnan(mean))
            assert close.all(), f"t{t} {r[1]}: means"


@gpu
def test_app_run_shuffled_clustering_markers(tmp_path):
    """clustering_markers in another order equals files whose columns are in that order"""
    import pandas as pd

    order = ["z", "x", "y"]
    _, narrow = _files(tmp_path, "narrow", order, EXTRA)
    _, wide = _files(tmp_path, "wide", WIDE, EXTRA)
    _run(narrow, tmp_path / "narrow")
    _run(wide, tmp_path / "wide", markers=order)
    assert open(tmp_path / "wide" / "result.csv", "rb").read() == open(tmp_path / "narrow" / "result.csv", "rb").read()
    for t in range(5):
        w = pd.read_csv(tmp_path / "wide" / f"cluster_points_D{t}.csv", keep_default_na=False, na_values=[""],
                        float_precision="round_trip")
        n = pd.read_csv(tmp_path / "narrow" / f"cluster_points_D{t}.csv", keep_default_na=False,
                        float_precision="round_trip")
        assert (w["cluster_id"].astype(str) == n["cluster_id"].astype(str)).all()
        assert (w[order].to_numpy() == n[order].to_numpy()).all()


# ---- errors -------------------------------------------------------------------------------------------------------------------
@gpu
def test_ingest_cols_rejects_bad_arguments():
    from chronoclust_b200 import _lib

    h = make(config_of(load("c1.npz")))
    h._ensure_handle(3)
    L = _lib.lib()
    X = np.zeros((10, 8), np.float64)
    assign, stage = np.zeros(10, np.int32), np.zeros(10, np.uint8)

    def call(cols, W=8, ld=8, dtype=_lib.DTYPE_F64, scale=None, min_=None):
        c = None if cols is None else _lib.ptr(np.ascontiguousarray(cols, np.int32))
        return L.ccb_ingest_cols(h._h, _lib.ptr(X), dtype, 0, 10, ld, W, c, scale, min_, _lib.ptr(assign), _lib.ptr(stage))

    ok = [5, 0, 2]
    L.ccb_begin_timepoint(h._h, 1.0, 0.0, 3, 0, 1.0)
    assert call(ok) == 0
    assert call(ok, W=2) == -1      # W < D
    assert call(ok, W=65, ld=65) == -1
    assert call(ok, ld=7) == -1     # ld < W
    assert call(None) == -1
    assert call([5, 0, 8]) == -1    # outside [0, W)
    assert call([5, -1, 2]) == -1
    assert call([5, 0, 5]) == -1    # repeated
    assert call(ok, dtype=7) == -1  # what ccb_ingest_ex rejects
    assert call(ok, scale=_lib.ptr(np.ones(3))) == -1
    assert (X == 0).all()


@gpu
def test_cluster_stats_state_after_a_column_ingest():
    from chronoclust_b200 import _lib

    z = load("c1.npz")
    h = make(config_of(z))
    big = widen(z["scaled0"], 7, [4, 1, 6])
    h.online_microcluster_maintenance(big, 0, columns=[4, 1, 6])
    assert h.cluster_statistics().mean.shape[1] == 7
    L = _lib.lib()
    L.ccb_begin_timepoint(h._h, float(h.mu), float(h.omicron), int(h.pi), 0, 1.0)
    n = len(h.export_arrays(0)[0])
    out = [np.zeros(64 * 8) for _ in range(3)]
    assert L.ccb_cluster_stats(h._h, _lib.ptr(np.full(n, -1, np.int32)), n, 1, 0, None, _lib.ptr(np.zeros(8, np.int64)),
                               *[_lib.ptr(a) for a in out]) == -4  # CCB_ESTATE
    with pytest.raises(_lib.CCBError):
        h.cluster_statistics()


@gpu
def test_columns_length_must_match_the_handle():
    z = load("c1.npz")
    h = make(config_of(z))
    big = widen(z["scaled0"], 7, [4, 1, 6])
    h.online_microcluster_maintenance(big, 0, columns=[4, 1, 6])
    with pytest.raises(ValueError):
        h.online_microcluster_maintenance(big, 1, columns=[4, 1])
    with pytest.raises(ValueError):
        h.online_microcluster_maintenance(big, 1, columns=[4, 1, 6], scaler=(np.ones(7), np.zeros(7)))


# ---- CPU: validation, headers, the per-column value rule ------------------------------------------------------------------------
@pytest.mark.parametrize("bad", [[], [0, 0], [7], [-1], [1.0], ["a"], [True], list(range(65)), 3])
def test_columns_validation(bad):
    from chronoclust_b200.hddstream import HDDStream, column_map

    with pytest.raises(ValueError):
        column_map(bad, 7)
    h = HDDStream(dict(config_of(load("c1.npz"))), None)
    with pytest.raises(ValueError):  # before any device work: no handle is created
        h.online_microcluster_maintenance(np.zeros((4, 7)), 0, columns=bad)
    assert h._h is None


def test_columns_validation_accepts_integer_sequences():
    from chronoclust_b200.hddstream import column_map

    assert column_map([3, 0, 5], 6).tolist() == [3, 0, 5]
    assert column_map(np.array([2, 1], np.int64), 3).dtype == np.int32
    assert column_map(range(64), 64).tolist() == list(range(64))
    with pytest.raises(ValueError):
        column_map([0], 65)  # rows wider than 64 columns


def test_clustering_markers_validation():
    from chronoclust_b200.app import clustering_columns

    attrs = ["cd3", "x", "fsc", "y", "z"]
    assert clustering_columns(attrs, None) is None
    assert clustering_columns(attrs, ["z", "x", "y"]) == [4, 1, 3]
    for bad in (["x", "w"], ["x", "x"], []):
        with pytest.raises(ValueError):
            clustering_columns(attrs, bad)


def test_app_run_rejects_bad_clustering_markers(tmp_path):
    import pandas as pd

    from chronoclust_b200 import app

    f = tmp_path / "d0.csv"
    pd.DataFrame(np.zeros((3, 3)), columns=["x", "y", "z"]).to_csv(f, index=False)
    for bad in (["x", "q"], ["y", "y"]):
        out = tmp_path / f"out_{bad[1]}"
        with pytest.raises(ValueError):
            app.run(data=[str(f)], output_directory=str(out), clustering_markers=bad)
        assert not os.path.exists(out / "result.csv")


def test_points_values_per_column_rule():
    from sklearn.preprocessing import MinMaxScaler

    from chronoclust_b200.app import points_values
    from chronoclust_b200.scaling import Scaler

    rng = np.random.default_rng(2)
    raw = rng.normal(100.0, 40.0, size=(50, 5))
    cols = [3, 0]
    sc = Scaler()
    sc.scaler = MinMaxScaler().fit(raw[:, cols])
    got = points_values(raw, sc, cols)
    exp = raw.copy()
    exp[:, cols] = sc.scaler.inverse_transform(sc.scaler.transform(raw[:, cols]))
    assert got.tobytes() == exp.tobytes()
    assert got[:, [1, 2, 4]].tobytes() == raw[:, [1, 2, 4]].tobytes()
    assert points_values(raw, None, cols) is raw
    full = Scaler()
    full.scaler = MinMaxScaler().fit(raw)
    assert points_values(raw, full, None).tobytes() == full.reverse_scaling(full.scale_data(raw)).tobytes()


def test_points_view_applies_the_column_map():
    from sklearn.preprocessing import MinMaxScaler

    from chronoclust_b200.hddstream import _PointsView

    rng = np.random.default_rng(1)
    cols = np.array([4, 0, 2], np.int32)
    wide = rng.normal(0.0, 30.0, size=(40, 6)).astype(np.float32)
    gathered = np.ascontiguousarray(wide[:, cols], np.float64)
    assign = rng.integers(0, 3, size=40).astype(np.int32)
    sk = MinMaxScaler().fit(gathered)
    for scaler in (None, (sk.scale_, sk.min_)):
        v, ref = _PointsView(), _PointsView()
        v.add(wide, assign, scaler, cols)
        ref.add(gathered, assign, scaler)
        for uid in range(3):
            a, b = v.points_of(uid), ref.points_of(uid)
            assert list(a.keys()) == list(b.keys()) and a == b


def test_result_and_points_headers():
    """result.csv's centroid columns are the clustering markers in the given order; the per-cell table and the statistics
    keep every column of the files in file order; without clustering_markers the headers are today's"""
    from chronoclust_b200 import app

    attrs = ["cd3", "x", "fsc", "y", "z"]
    cols = app.clustering_columns(attrs, ["y", "x"])
    result, points, stats = app.output_headers(attrs, [attrs[c] for c in cols], "gates.csv")
    assert result == ["timepoint", "cumulative_size", "pcore_ids", "pref_dimensions", "y", "x", "tracking_by_lineage",
                      "tracking_by_association", "predicted_label"]
    assert points == ["id", "cluster_id"] + attrs
    assert stats == ["timepoint", "tracking_by_lineage", "cell_count"] + [f"median_{a}" for a in attrs] + \
        [f"mean_{a}" for a in attrs]
    result, points, _ = app.output_headers(["x", "y", "z"], ["x", "y", "z"], None)
    assert result == ["timepoint", "cumulative_size", "pcore_ids", "pref_dimensions", "x", "y", "z",
                      "tracking_by_lineage", "tracking_by_association"]
    assert points == ["id", "cluster_id", "x", "y", "z"]
