"""The arcsinh transform of cytometry intensities: ccb_asinh (csrc/asinh.h) within 1 ulp of the correctly rounded asinh
and odd bit for bit; the host library (ccbio_arcsinh_host) and the device (ccb_arcsinh, the staging kernels) give the
same bits; and HDDStream.online_microcluster_maintenance(cofactors=), cluster_statistics and app.run(arcsinh_cofactors=)
give bit for bit what the float64 path gives on the host-transformed rows."""
import csv
import logging
import os
import shutil
import subprocess

import numpy as np
import pytest

from helpers import STRESS_NAMES, bits_equal, config_of, load, stress_inputs
from test_cluster_stats import QS, bits, check
from test_column_subset import whole_row_values, widen
from test_input_paths import assert_same, make

gpu = pytest.mark.gpu
KINDS = ["numpy-f64", "numpy-f32", "cuda-f64", "cuda-f32"]
CYCLE = (5.0, 150.0, 0.0, 2.5)  # cofactors by column: mass, flow, linear, another


def host(x, cof, threads=0):
    from chronoclust_b200 import _hostio

    return _hostio.arcsinh_host(x, np.asarray(cof, np.float64), threads)


def asinh1(v):
    """ccb_asinh of a float64 vector (cofactor 1: x / 1 is exact)"""
    return host(np.ascontiguousarray(v, np.float64).reshape(-1, 1), [1.0])[:, 0]


def value_set(n=1_000_000, seed=0):
    """log-uniform magnitudes over the whole double range, both signs, subnormals, the neighbourhoods of 2^-28, 2 and 2^28,
    +-0, +-inf and NaN"""
    rng = np.random.default_rng(seed)
    mag = np.ldexp(rng.uniform(1.0, 2.0, n), rng.integers(-1074, 1024, n))
    parts = [mag * rng.choice([-1.0, 1.0], n), np.ldexp(rng.uniform(0.0, 1.0, 2000), -1022)]
    for edge in (2.0 ** -28, 2.0, 2.0 ** 28):
        b = np.float64(edge).view(np.int64)
        near = (b + np.arange(-3000, 3001)).view(np.float64)
        parts += [near, -near, edge * rng.uniform(0.5, 2.0, 3000)]
    parts.append(np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1.0, -1.0, 0.5, 0.51877144]))
    v = np.concatenate(parts)
    return v[np.isfinite(v) | np.isnan(v) | np.isinf(v)]


def ulp_distance(a, b):
    """|a - b| in units in the last place, through the order-preserving integer map"""
    def key(x):
        i = x.view(np.int64)
        return np.where(i < 0, np.int64(-(2 ** 63)) - i, i)
    return np.abs(key(a) - key(b))


# ---- the definition (CPU) -----------------------------------------------------------------------------------------------
def test_ccb_asinh_within_one_ulp_of_mpmath():
    import mpmath

    v = value_set()
    got = asinh1(v)
    fin = np.isfinite(v)
    assert np.isnan(got[np.isnan(v)]).all()
    assert (got[np.isinf(v)] == v[np.isinf(v)]).all()
    z = v == 0
    assert (got[z].view(np.int64) == v[z].view(np.int64)).all(), "+-0 keep their sign"
    with mpmath.workprec(200):
        ref = np.array([float(mpmath.asinh(mpmath.mpf(float(x)))) for x in v[fin]])  # float(): correctly rounded
    d = ulp_distance(got[fin], ref)
    exact = float((d == 0).mean())
    print(f"ccb_asinh: {fin.sum()} finite values, {100 * exact:.2f} % correctly rounded, max {d.max()} ulp")
    assert d.max() <= 1, f"{(d > 1).sum()} values further than 1 ulp, e.g. {v[fin][d > 1][:5]}"
    assert exact > 0.7


def test_ccb_asinh_is_odd_bit_for_bit():
    v = value_set(200_000, seed=1)
    v = v[~np.isnan(v)]
    assert (asinh1(-v).view(np.int64) == (-asinh1(v)).view(np.int64)).all()


@pytest.mark.parametrize("layout", ["float64", "float32", "strided64", "strided32"])
def test_arcsinh_host_threads_give_identical_output(layout):
    rng = np.random.default_rng(3)
    X = rng.exponential(400.0, (50_000, 13)) * rng.choice([-1.0, 1.0], (50_000, 13))
    X[::97, 4] = np.nan
    if layout.startswith("strided"):
        X = np.concatenate([X, np.full((len(X), 5), np.nan)], axis=1)[:, :13]
    X = X.astype(np.float32 if layout.endswith("32") else np.float64)
    cof = [CYCLE[j % 4] for j in range(13)]
    one, many = host(X, cof, 1), host(X, cof, 16)
    assert one.tobytes() == many.tobytes()
    ref = np.array([[v if c == 0 else asinh1(np.array([np.float64(v) / c]))[0] for v, c in zip(row, cof)]
                    for row in X[:200].astype(np.float64)])
    assert bits_equal(np.nan_to_num(one[:200], nan=7.0), np.nan_to_num(ref, nan=7.0))


def test_cofactor_vector_validation():
    from chronoclust_b200.scaling import arcsinh, cofactor_vector

    assert cofactor_vector(5, 3).tolist() == [5.0, 5.0, 5.0]
    assert cofactor_vector(np.float32(150), 2).tolist() == [150.0, 150.0]
    assert cofactor_vector([5, 0, 2.5], 3).tolist() == [5.0, 0.0, 2.5]
    for bad in (-1.0, np.nan, np.inf, -np.inf, [5, 5], [5, -0.5, 1], [5, "a", 1], True, [1, None, 2], "5", None):
        with pytest.raises(ValueError):
            cofactor_vector(bad, 3)
    x32 = np.random.default_rng(0).exponential(100.0, (64, 3)).astype(np.float32)
    got = arcsinh(x32, [5, 0, 150])
    assert got.dtype == np.float64 and bits_equal(got[:, 1], x32[:, 1].astype(np.float64))
    assert bits_equal(got, host(x32, [5, 0, 150]))


def test_app_cofactor_options():
    from chronoclust_b200.app import arcsinh_cofactors_by_column, transform_gates

    attrs = ["cd3", "x", "fsc", "y"]
    assert arcsinh_cofactors_by_column(attrs, None, None) is None
    assert arcsinh_cofactors_by_column(attrs, None, 5).tolist() == [5.0] * 4
    assert arcsinh_cofactors_by_column(attrs, [1, 3], 5).tolist() == [0.0, 5.0, 0.0, 5.0]
    assert arcsinh_cofactors_by_column(attrs, [1, 3], {"cd3": 150, "x": 5}).tolist() == [150.0, 5.0, 0.0, 0.0]
    for bad in ({"cd4": 5}, {"x": -5}, {"x": np.nan}, -1, np.inf, [5, 5, 5, 5], "5"):
        with pytest.raises(ValueError):
            arcsinh_cofactors_by_column(attrs, [1, 3], bad)
    gates = {0: {(10.0, 20.0): "A", (-3.0, 0.5): "B"}, 2: {(1e4, 7.0): "C"}}
    got = transform_gates(gates, np.array([5.0, 0.0]))
    assert list(got) == [0, 2] and list(got[0].values()) == ["A", "B"]
    for day in gates:
        for (raw, name), (tx, name2) in zip(gates[day].items(), got[day].items()):
            assert name == name2 and tx[1] == raw[1] and tx[0] == asinh1(np.array([raw[0] / 5.0]))[0]


def test_points_values_per_column_rule():
    from sklearn.preprocessing import MinMaxScaler

    from chronoclust_b200.app import points_values
    from chronoclust_b200.scaling import Scaler

    rng = np.random.default_rng(5)
    raw = rng.normal(200.0, 150.0, (500, 4))
    cof = np.array([5.0, 0.0, 150.0, 0.0])  # columns 0, 2 transformed; 0, 1 clustering
    cols = [0, 1]
    tx = host(raw, cof)
    sc = Scaler()
    sc.scaler = MinMaxScaler().fit(tx[:, cols])
    got = points_values(raw, sc, cols, cof)
    assert bits_equal(got[:, cols], sc.reverse_scaling(sc.scale_data(tx[:, cols])))  # transformed + scaled, scaled
    assert bits_equal(got[:, 2], tx[:, 2]) and bits_equal(got[:, 3], raw[:, 3])    # transformed, raw
    assert bits_equal(points_values(raw, None, cols, cof), tx)
    assert points_values(raw, None, cols) is raw  # without the option: the parsed values, as before


def test_host_library_has_no_fma():
    from chronoclust_b200 import _hostio

    if shutil.which("objdump") is None:
        pytest.skip("objdump is not installed")
    _hostio.lib()
    dis = subprocess.run(["objdump", "-d", _hostio.SO_PATH], capture_output=True, text=True, check=True).stdout
    assert "ccbio_arcsinh_host" in dis and "vfmadd" not in dis and "vfnmadd" not in dis and "vfmsub" not in dis


# ---- host == device, pointwise (GPU) -------------------------------------------------------------------------------------
def device_arcsinh(x, cof):
    from chronoclust_b200.scaling import arcsinh

    return arcsinh(x, cof).cpu().numpy()


def same_bits_or_both_nan(a, b):
    return a.shape == b.shape and ((a.view(np.int64) == b.view(np.int64)) | (np.isnan(a) & np.isnan(b))).all()


@gpu
@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_device_equals_host_pointwise(dtype):
    import torch

    v = value_set()
    rng = np.random.default_rng(7)
    intens = np.concatenate([rng.exponential(300.0, 5_000_000), rng.normal(0.0, 80.0, 5_000_000)])
    for what, flat in (("value set", v), ("intensities", intens)):
        flat = flat.astype(getattr(np, dtype))
        D = 8
        n = len(flat) // D
        X = flat[:n * D].reshape(n, D)
        cof = [CYCLE[j % 4] if what == "intensities" else (1.0, 5.0, 0.0, 3e-300, 1e300, 150.0, 0.5, 7.0)[j]
               for j in range(D)]
        ref = host(X, cof)
        assert same_bits_or_both_nan(device_arcsinh(torch.from_numpy(X).cuda(), cof), ref), f"{what} {dtype}"
        pad = torch.full((n, D + 3), float("nan"), dtype=getattr(torch, dtype), device="cuda")
        pad[:, :D] = torch.from_numpy(X).cuda()
        assert same_bits_or_both_nan(device_arcsinh(pad[:, :D], cof), ref), f"{what} {dtype} strided"
        assert same_bits_or_both_nan(host(pad[:, :D].cpu().numpy(), cof), ref), f"{what} {dtype} host strided"


@gpu
def test_ccb_arcsinh_rejects_bad_arguments():
    import torch

    from chronoclust_b200 import _lib

    X = torch.zeros((4, 3), dtype=torch.float64, device="cuda")
    out = torch.empty((4, 3), dtype=torch.float64, device="cuda")
    L = _lib.lib()

    def call(cof, dtype=_lib.DTYPE_F64, ld=3, D=3):
        return L.ccb_arcsinh(0, None, X.data_ptr(), dtype, 4, ld, D, _lib.ptr(np.asarray(cof, np.float64)), out.data_ptr())

    assert call([5, 0, 1]) == 0
    for bad in ([5, -1, 1], [5, np.nan, 1], [np.inf, 0, 1]):
        assert call(bad) == -1
    assert call([5, 0, 1], dtype=3) == -1 and call([5, 0, 1], ld=2) == -1 and call([5] * 65, D=65, ld=65) == -1
    assert L.ccb_arcsinh(0, None, X.data_ptr(), 0, 4, 3, 3, None, out.data_ptr()) == -1
    torch.cuda.synchronize()


# ---- clustering (GPU) ---------------------------------------------------------------------------------------------------------
def intensities(Xs):
    """raw intensities raw = 5 sinh(6 x - 0.5) of generator rows x: cytometry-like, negative values included"""
    return [5.0 * np.sinh(6.0 * x - 0.5) for x in Xs]


def fixtures():
    from chronoclust_b200.synth import config_params, gen

    out = []
    for name in STRESS_NAMES + ["c1"]:
        if name == "c1":
            z = load("c1.npz")
            out.append((name, config_of(z), [z[f"scaled{t}"] for t in range(5)], list(range(5))))
        else:
            z = load(f"stress_{name}.npz")
            out.append((name, config_of(z), stress_inputs(z), [int(t) for t in z["timestamps"]]))
    cfg = dict(config_params("C2"))
    cfg["epsilon"] = 0.4  # (the transformed rows span about [-0.5, 5.5])
    out.append(("intensities", cfg, intensities(gen(20000, 10, 3, 12, 31)), [0, 1, 2]))
    return out


def run_tx(cfg, Xs, ts, W, cols, kind, scaled, what, **kw):
    """authority: the float64 host path on arcsinh_host(rows) (then gathered); other: cofactors= on the rows of `kind`"""
    import torch
    from sklearn.preprocessing import MinMaxScaler

    dt = np.float32 if kind.endswith("f32") else np.float64
    idx = list(range(W)) if cols is None else cols
    cof = np.array([CYCLE[j % 4] for j in range(W)])
    bigs = [(X.astype(dt) if cols is None else widen(X, W, cols, dt)) for X in Xs]
    txs = [host(b, cof) for b in bigs]
    sk = MinMaxScaler().fit(np.concatenate([t[:, idx] for t in txs], axis=0)) if scaled else None
    a, b = make(cfg, **kw), make(cfg, **kw)
    for t, big, tx in zip(ts, bigs, txs):
        x = torch.from_numpy(big).cuda() if kind.startswith("cuda") else big
        before = big.copy()
        a.online_microcluster_maintenance(np.ascontiguousarray(tx[:, idx]), t, scaler=sk)
        b.online_microcluster_maintenance(x, t, scaler=sk, columns=cols, cofactors=cof)
        after = x if isinstance(x, np.ndarray) else x.cpu().numpy()
        assert before.tobytes() == after.tobytes(), f"{what}: the caller's rows were written"
        assert_same(a, b, f"{what} t{t}", points=True)
    return a, b


@gpu
@pytest.mark.parametrize("scaled", [False, True], ids=["unscaled", "scaled"])
@pytest.mark.parametrize("kind", KINDS)
def test_cofactors_equal_the_host_transformed_float64_path(kind, scaled):
    rng = np.random.default_rng(11 + 2 * KINDS.index(kind) + scaled)
    for name, cfg, Xs, ts in fixtures():
        D = Xs[0].shape[1]
        run_tx(cfg, Xs, ts, D, None, kind, scaled, f"{name} {kind} scaled={scaled}")
        W = min(64, D + 3)
        cols = rng.permutation(W)[:D].tolist()
        run_tx(cfg, Xs, ts, W, cols, kind, scaled, f"{name} {kind} scaled={scaled} W={W} cols={cols}")


@gpu
@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_cofactors_segmented_and_single_segment_copy(dtype):
    """N >= 262144: host rows are transformed segment by segment behind the copies (float64 in place in the engine's
    buffer); with timing on, the single-segment branch; a row-strided view too"""
    from chronoclust_b200.synth import config_params, gen

    cfg = dict(config_params("C2"))
    cfg["epsilon"] = 0.4
    D = 12
    cof = np.array([CYCLE[j % 4] for j in range(D)])
    a, b, c, d = (make(cfg) for _ in range(4))
    c._ensure_handle(D)
    c.enable_timing(True)
    for t, X in enumerate(intensities(gen(300001, D, 2, 20, 7))):
        X = X.astype(getattr(np, dtype))
        padded = np.full((len(X), D + 3), np.nan, X.dtype)
        padded[:, :D] = X
        a.online_microcluster_maintenance(host(X, cof), t)
        b.online_microcluster_maintenance(X, t, cofactors=cof)
        c.online_microcluster_maintenance(X, t, cofactors=cof)
        d.online_microcluster_maintenance(padded[:, :D], t, cofactors=cof)
        for h, what in ((b, "segmented"), (c, "single segment (timing)"), (d, "segmented, ld = D + 3")):
            assert_same(a, h, f"{dtype} {what} t{t}", points=(t == 1))
    assert c.timing()["copy"][1] > 0


@gpu
@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_cofactors_cuda_view_written_on_a_side_stream(dtype):
    import torch

    from chronoclust_b200.synth import config_params, gen

    cfg = dict(config_params("C2"))
    cfg["epsilon"] = 0.4
    D = 12
    cof = np.array([CYCLE[j % 4] for j in range(D)])
    a, b = make(cfg), make(cfg)
    side = torch.cuda.Stream()
    for t, X in enumerate(intensities(gen(30000, D, 2, 20, 21))):
        X = X.astype(getattr(np, dtype))
        src = torch.from_numpy(X).cuda()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            big = torch.full((len(X), D + 5), float("nan"), dtype=getattr(torch, dtype), device="cuda")
            torch.cuda._sleep(50_000_000)
            big[:, :D].copy_(src)
            b.online_microcluster_maintenance(big[:, :D], t, cofactors=cof)
        torch.cuda.synchronize()
        a.online_microcluster_maintenance(host(X, cof), t)
        assert_same(a, b, f"cuda {dtype} view t{t}", points=True)


# ---- statistics (GPU) -----------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("with_cols", [False, True], ids=["all-columns", "columns"])
@pytest.mark.parametrize("scaled", [False, True], ids=["unscaled", "scaled"])
@pytest.mark.parametrize("kind", KINDS)
def test_cluster_statistics_in_transformed_space(kind, scaled, with_cols):
    import torch
    from sklearn.preprocessing import MinMaxScaler

    rng = np.random.default_rng(23)
    for name, cfg, Xs, ts in [f for f in fixtures() if f[0] in ("c2like", "intensities")]:
        D = Xs[0].shape[1]
        W = D + 3 if with_cols else D
        cols = rng.permutation(W)[:D].tolist() if with_cols else None
        idx = cols if with_cols else list(range(D))
        dt = np.float32 if kind.endswith("f32") else np.float64
        cof = np.array([CYCLE[j % 4] for j in range(W)])
        bigs = [(widen(X, W, cols, dt) if with_cols else X.astype(dt)) for X in Xs]
        sk = MinMaxScaler().fit(np.concatenate([host(b, cof)[:, idx] for b in bigs])) if scaled else None
        h = make(cfg)
        for t, big in zip(ts, bigs):
            x = torch.from_numpy(big).cuda() if kind.startswith("cuda") else big
            h.online_microcluster_maintenance(x, t, scaler=sk, columns=cols, cofactors=cof)
            lab = h.cluster_labels_for_points()
            G = len(h.final_clusters)
            got = h.cluster_statistics(quantiles=QS)
            assert got.mean.shape == (G + 1, W)
            check(got, whole_row_values(host(big, cof), idx, sk), np.where(lab < 0, G, lab), G + 1, QS,
                  f"{name} {kind} scaled={scaled} cols={cols} t{t}")
            assert bits(got) == bits(h.cluster_statistics(quantiles=QS))


# ---- app.run (GPU) ----------------------------------------------------------------------------------------------------------------
def _reread(values, columns, path):
    """values written as app.run's inputs are (DataFrame.to_csv) and parsed back as app.run parses them"""
    import pandas as pd

    pd.DataFrame(values, columns=columns).to_csv(path, index=False)
    return pd.read_csv(path).to_numpy(np.float64)


def _same_rows(a, b):
    return ((a.view(np.int64) == b.view(np.int64)) | (np.isnan(a) & np.isnan(b))).all(axis=1)


def _series(tmp_path, columns, cof):
    """C1's cells as raw intensities (columns x, y, z: 5 sinh(6 x - 0.5); cd3 / fsc: extra markers) and the same cells
    holding their arcsinh_host values under `cof` (by column), plus gating files in either unit.  pandas' CSV parser does
    not always give back the double that was written, so only the cells (and gates) whose transformed values read back
    exactly are kept: both runs then start from the same doubles."""
    z = load("c1.npz")
    raw_files, tx_files, g_raw, g_tx = [], [], [], []
    xyz = [columns.index(c) for c in "xyz"]
    for t in range(5):
        s = z[f"scaled{t}"]
        rng = np.random.default_rng(t)
        cells = {"x": 5.0 * np.sinh(6.0 * s[:, 0] - 0.5), "y": 5.0 * np.sinh(6.0 * s[:, 1] - 0.5),
                 "z": 5.0 * np.sinh(6.0 * s[:, 2] - 0.5), "cd3": rng.exponential(900.0, len(s)) - 100.0,
                 "fsc": rng.integers(0, 260000, len(s)).astype(np.float64)}
        rf, tf = tmp_path / f"raw_d{t}.csv", tmp_path / f"tx_d{t}.csv"
        parsed = _reread(np.stack([cells[c] for c in columns], axis=1), columns, rf)
        tx = host(parsed, cof)
        keep = _same_rows(_reread(parsed, columns, rf), parsed) & _same_rows(_reread(tx, columns, tf), tx)
        assert keep.mean() > 0.2
        parsed, tx = parsed[keep], tx[keep]
        assert _same_rows(_reread(parsed, columns, rf), parsed).all() and _same_rows(_reread(tx, columns, tf), tx).all()
        raw_files.append(str(rf))
        tx_files.append(str(tf))
        for k in range(0, len(parsed), len(parsed) // 3):
            g = parsed[k:k + 1, xyz]  # (read back exactly, as every kept cell)
            gt = tx[k:k + 1, xyz]
            g_raw.append((t, f"P{len(g_raw) % 5}", *g[0]))
            g_tx.append((t, g_raw[-1][1], *gt[0]))
    gates = []
    for name, rows in (("gates_raw.csv", g_raw), ("gates_tx.csv", g_tx)):
        import pandas as pd

        frame = pd.DataFrame(rows, columns=["Day", "PopName", "x", "y", "z"])
        frame.to_csv(tmp_path / name, index=False)
        back = pd.read_csv(tmp_path / name)[["x", "y", "z"]].to_numpy(np.float64)
        assert _same_rows(back, frame[["x", "y", "z"]].to_numpy(np.float64)).all()
        gates.append(str(tmp_path / name))
    return raw_files, tx_files, gates[0], gates[1]


def _app(files, out, gates, **kw):
    from chronoclust_b200 import app

    cfg = config_of(load("c1.npz"))
    app.run(data=files, output_directory=str(out), gating_centroid_file=gates, param_beta=cfg["beta"],
            param_delta=cfg["delta"], param_epsilon=cfg["epsilon"] * 6.0, param_lambda=cfg["lambda"], param_k=cfg["k"],
            param_mu=cfg["mu"], param_pi=cfg["pi"], param_omicron=cfg["omicron"], param_upsilon=cfg["upsilon"],
            cluster_statistics=True, **kw)


@gpu
@pytest.mark.parametrize("option", ["scalar", "dict"])
def test_app_run_arcsinh_cofactors(tmp_path, caplog, option):
    caplog.set_level(logging.INFO)
    if option == "scalar":
        columns, cof, kw = ["x", "y", "z"], np.array([5.0, 5.0, 5.0]), dict(arcsinh_cofactors=5)
        kw_tx = {}
    else:  # a transformed non-clustering marker (cd3) and a linear one (fsc)
        columns, cof = ["cd3", "x", "fsc", "y", "z"], np.array([150.0, 5.0, 0.0, 5.0, 5.0])
        kw = dict(arcsinh_cofactors={"x": 5, "y": 5, "z": 5, "cd3": 150}, clustering_markers=["x", "y", "z"])
        kw_tx = dict(clustering_markers=["x", "y", "z"])
    raw, tx, g_raw, g_tx = _series(tmp_path, columns, cof)
    _app(raw, tmp_path / "raw", g_raw, **kw)
    _app(tx, tmp_path / "tx", g_tx, **kw_tx)
    names = ["result.csv", "cluster_statistics.csv"] + [f"cluster_points_D{t}.csv" for t in range(5)]
    for f in names:
        a, b = open(tmp_path / "raw" / f, "rb").read(), open(tmp_path / "tx" / f, "rb").read()
        assert a == b, f"{option}: {f} differs"
    with open(tmp_path / "raw" / "result.csv") as f:
        rows = list(csv.reader(f))
    assert len(rows) > 5 and all(r[-1] for r in rows[1:]), "every cluster has a gating label"
    logged = [r.getMessage() for r in caplog.records if "arcsinh cofactors" in r.getMessage()]
    assert len(logged) == 1 and "x=5.0" in logged[0]


@gpu
def test_app_run_rejects_bad_cofactors_before_clustering(tmp_path):
    raw, _, g_raw, _ = _series(tmp_path, ["x", "y", "z"], np.array([5.0, 5.0, 5.0]))
    for bad in ({"q": 5}, -5, {"x": np.nan}):
        out = tmp_path / f"bad{len(os.listdir(tmp_path))}"
        with pytest.raises(ValueError):
            _app(raw, out, g_raw, arcsinh_cofactors=bad)
        assert not (out / "cluster_points_D0.csv").exists()


# ---- ABI (GPU) ------------------------------------------------------------------------------------------------------------------
@gpu
def test_ingest_tx_rejections_and_unchanged_ingest_ex_cols():
    from chronoclust_b200 import _lib

    h = make(config_of(load("c1.npz")))
    h._ensure_handle(3)
    L = _lib.lib()
    X = np.random.default_rng(0).normal(0.0, 1.0, (10, 8))
    X0 = X.copy()
    assign, stage = np.zeros(10, np.int32), np.zeros(10, np.uint8)
    P = lambda a: None if a is None else _lib.ptr(np.ascontiguousarray(a, np.int32 if np.asarray(a).dtype.kind == "i"
                                                                        else np.float64))

    def tx(cols, cof, W=8, ld=8, dtype=_lib.DTYPE_F64, scale=None, min_=None):
        return L.ccb_ingest_tx(h._h, _lib.ptr(X), dtype, 0, 10, ld, W, P(cols), P(cof), scale, min_, _lib.ptr(assign),
                               _lib.ptr(stage))

    def cols_(cols, W=8, ld=8, dtype=_lib.DTYPE_F64, scale=None, min_=None):
        return L.ccb_ingest_cols(h._h, _lib.ptr(X), dtype, 0, 10, ld, W, P(cols), scale, min_, _lib.ptr(assign),
                                 _lib.ptr(stage))

    ok, cof = [5, 0, 2], np.array([5.0, 0, 1, 2, 150, 0, 3, 4])
    L.ccb_begin_timepoint(h._h, 1.0, 0.0, 3, 0, 1.0)
    assert tx(ok, cof) == 0 and tx(ok, None) == 0 and tx(None, cof[:3], W=3) == 0 and tx(None, None, W=3) == 0
    for bad in (-1.0, np.nan, np.inf, -np.inf):
        c = cof.copy()
        c[6] = bad
        assert tx(ok, c) == -1, bad
    assert tx(None, cof, W=8) == -1  # W != D without a column map
    one = np.ones(3)
    for args in (dict(W=2), dict(W=65, ld=65), dict(ld=7), dict(dtype=7), dict(scale=_lib.ptr(one))):
        assert tx(ok, cof, **args) == -1 and cols_(ok, **args) == -1, args
    for c in ([5, 0, 8], [5, -1, 2], [5, 0, 5]):
        assert tx(c, cof) == -1 and cols_(c) == -1, c
    assert cols_(None) == -1
    assert L.ccb_ingest_ex(h._h, _lib.ptr(X), _lib.DTYPE_F64, 0, 10, 2, None, None, _lib.ptr(assign), _lib.ptr(stage)) == -1
    assert (X == X0).all()
    # ccb_ingest_ex / ccb_ingest_cols give what ccb_ingest_tx gives without cofactors
    from chronoclust_b200.synth import config_params, gen

    cfg = config_params("C2")
    Xs = gen(20000, 6, 2, 8, 3)
    W, cmap = 9, np.array([7, 1, 4, 0, 8, 2], np.int32)
    for variant in ("ex", "cols"):
        a, b = make(cfg), make(cfg)
        for t, x in enumerate(Xs):
            big = widen(x, W, cmap.tolist()) if variant == "cols" else x
            for hh in (a, b):
                hh._set_dataset_dependent_parameters(big, 6)
                hh._ensure_handle(6)
                _lib.check(L.ccb_begin_timepoint(hh._h, float(hh.mu), float(hh.omicron), int(hh.pi), int(t > 0),
                                                 1.0), hh._h)
            ua, sa, ub, sb = (np.empty(len(x), np.int32), np.empty(len(x), np.uint8),
                              np.empty(len(x), np.int32), np.empty(len(x), np.uint8))
            ld = big.shape[1]
            if variant == "ex":
                rc = L.ccb_ingest_ex(a._h, _lib.ptr(big), 0, 0, len(x), ld, None, None, _lib.ptr(ua), _lib.ptr(sa))
            else:
                rc = L.ccb_ingest_cols(a._h, _lib.ptr(big), 0, 0, len(x), ld, W, _lib.ptr(cmap), None, None, _lib.ptr(ua),
                                       _lib.ptr(sa))
            assert rc == 0
            assert L.ccb_ingest_tx(b._h, _lib.ptr(big), 0, 0, len(x), ld, ld, None if variant == "ex" else _lib.ptr(cmap),
                                   None, None, None, _lib.ptr(ub), _lib.ptr(sb)) == 0
            assert (ua == ub).all() and (sa == sb).all(), f"{variant} t{t}"
            for which in (0, 1):
                ga, gb = a.export_arrays(which), b.export_arrays(which)
                assert all(bits_equal(p, q) for p, q in zip(ga[2:], gb[2:]))
