"""Every way in to HDDStream.online_microcluster_maintenance -- float32 numpy rows, row-strided views, CPU tensors, CUDA
tensors, with and without the device scaler -- gives bit for bit what the float64 path gives on the same rows widened to
float64 (which the rest of the suite pins to the goldens and the oracle): assignments, stages, both lists, counters,
final clusters and the `points` of the microclusters, at every timepoint."""
import logging

import numpy as np
import pytest

from helpers import STRESS_NAMES, bits_equal, config_of, load, stress_inputs

LOG = logging.getLogger("test")
gpu = pytest.mark.gpu


def make(cfg, **kw):
    from chronoclust_b200.hddstream import HDDStream

    return HDDStream(dict(cfg), LOG, **kw)


def clusters_of(h):
    return [(c.members_in_claim_order, c.cumulative_weight, c.CF1, c.CF2, c.cluster_centroids,
             c.preferred_dimension_vector) for c in h.final_clusters]


def points_sample(h, n=3):
    """points dicts of the first n pcore and the first n outlier microclusters"""
    return [mc.points for mc in h.pcore_MC[:n] + h.outlier_MC[:n]]


def assert_same(a, b, what, points=False):
    assert (a.last_assignment == b.last_assignment).all(), \
        f"{what}: {(a.last_assignment != b.last_assignment).sum()} assignments differ"
    assert (a.last_stage == b.last_stage).all(), f"{what}: stages differ"
    for which in (0, 1):
        ga, gb = a.export_arrays(which), b.export_arrays(which)
        assert len(ga[0]) == len(gb[0]), f"{what}: list {which} length {len(ga[0])} != {len(gb[0])}"
        assert (ga[0] == gb[0]).all() and (ga[1] == gb[1]).all(), f"{what}: list {which} ids / uids differ"
        for n, x, y in zip(("w", "cf1", "cf2", "cen", "pref"), ga[2:], gb[2:]):
            assert bits_equal(x, y), f"{what}: list {which} {n} not bit-identical"
    assert a.counts() == b.counts(), f"{what}: counters"
    ca, cb = clusters_of(a), clusters_of(b)
    assert len(ca) == len(cb), f"{what}: {len(ca)} clusters != {len(cb)}"
    for c, ((m1, w1, *r1), (m2, w2, *r2)) in enumerate(zip(ca, cb)):
        assert list(m1) == list(m2) and bits_equal(w1, w2), f"{what}: cluster {c} claim order / weight"
        assert all(bits_equal(p, q) for p, q in zip(r1, r2)), f"{what}: cluster {c} sums"
    if points:
        pa, pb = points_sample(a), points_sample(b)
        assert len(pa) == len(pb)
        for x, y in zip(pa, pb):
            assert list(x.keys()) == list(y.keys()) and x == y, f"{what}: points differ"


def run_pair(cfg, Xs, feed, what, scaler=None, timestamps=None, **kw):
    """authority: the float64 host path on X.astype(float64); other: feed(X) for every timepoint X (float32 or float64)"""
    a, b = make(cfg, **kw), make(cfg, **kw)
    for i, X in enumerate(Xs):
        t = i if timestamps is None else int(timestamps[i])
        a.online_microcluster_maintenance(X.astype(np.float64), t, scaler=scaler)
        b.online_microcluster_maintenance(feed(X), t, scaler=scaler)
        assert_same(a, b, f"{what} t{i}", points=True)
    return a, b


def raw_series(N, D, T, C, seed, cast=np.float32):
    """gen() rows moved far from [0, 1] (per-marker scales from 0.01 to 1e4), in `cast`"""
    from chronoclust_b200.synth import gen

    sc = np.array([3.0, 250.0, 0.01, 17.0, 1e4, 2.0, 41.0, 0.5, 7.0, 900.0, 1.5, 60.0])[:D]
    sh = np.array([1.0, 100.0, 0.0, -4.0, 5e3, 0.5, -20.0, 0.25, 3.0, -450.0, 0.0, 30.0])[:D]
    return [(x * sc - sh).astype(cast) for x in gen(N, D, T, C, seed)]


def cuda_rows(x, dtype, side, extra=3):
    """x as the row-strided view big[:, :D] of a CUDA tensor of `dtype` whose padding columns hold NaN, written on the
    stream `side` only after a delay: a reader that does not wait for `side` sees NaN rows"""
    import torch

    src = torch.from_numpy(np.ascontiguousarray(x)).to("cuda", dtype)
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        big = torch.full((x.shape[0], x.shape[1] + extra), float("nan"), dtype=dtype, device="cuda")
        torch.cuda._sleep(50_000_000)
        big[:, :x.shape[1]].copy_(src)
    return big, big[:, :x.shape[1]]


# ---- host rows -------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", STRESS_NAMES + ["c1"])
def test_float32_host_rows_equal_the_widened_float64_path(name):
    if name == "c1":
        z = load("c1.npz")
        Xs = [z[f"scaled{t}"] for t in range(5)]
    else:
        z = load(f"stress_{name}.npz")
        Xs = stress_inputs(z)
    run_pair(config_of(z), [x.astype(np.float32) for x in Xs], lambda x: x, f"{name}/f32", timestamps=z["timestamps"])


@gpu
def test_float32_segmented_copy_pipeline():
    """N >= 262144 per timepoint: the float32 rows travel segment by segment into the float32 staging buffer and are
    widened behind each segment's copy; with timing on the same rows take the single-segment branch.  A row-strided
    float32 view (ld > D) goes through the same segments."""
    from chronoclust_b200.synth import config_params, gen

    cfg = config_params("C2")
    Xs = [x.astype(np.float32) for x in gen(300001, 12, 3, 20, 7)]
    a, b, c, d = (make(cfg) for _ in range(4))
    c._ensure_handle(12)
    c.enable_timing(True)
    for t, X in enumerate(Xs):
        big = np.full((X.shape[0], 17), np.nan, np.float32)
        big[:, :12] = X
        a.online_microcluster_maintenance(X.astype(np.float64), t)
        b.online_microcluster_maintenance(X, t)
        c.online_microcluster_maintenance(X, t)
        d.online_microcluster_maintenance(big[:, :12], t)
        for h, what in ((b, "segmented"), (c, "single segment (timing)"), (d, "segmented, ld = 17")):
            assert_same(a, h, f"{what} t{t}", points=(t == len(Xs) - 1))
    assert c.timing()["copy"][1] > 0


@gpu
def test_scaled_float32_raw_rows_host_and_device():
    """Raw float32 rows with a fitted MinMaxScaler, host and CUDA, equal the float64 scaled path on the widened raw rows
    (which test_device_scaler_matches_sklearn pins to scaling on the host first); 300001 rows take the segmented copy."""
    import torch
    from sklearn.preprocessing import MinMaxScaler

    cfg = {"beta": 0.2, "delta": 0.05, "epsilon": 0.05, "lambda": 2, "k": 4, "mu": 0.01, "pi": 0, "omicron": 0.00000435,
           "upsilon": 6.5}
    raw = raw_series(300001, 6, 2, 6, 5)
    sk = MinMaxScaler().fit(np.concatenate(raw, axis=0).astype(np.float64))
    run_pair(cfg, raw, lambda x: x, "host f32 scaled", scaler=sk)
    run_pair(cfg, raw, lambda x: torch.from_numpy(x).cuda(), "cuda f32 scaled", scaler=sk)


# ---- CUDA tensors ----------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("scaled", [False, True], ids=["unscaled", "scaled"])
@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_cuda_tensor_rows_equal_the_host_float64_path(dtype, scaled):
    """A row-strided view of a CUDA tensor, written on a side stream that is current at the time of the call: the handle
    waits for that stream, the results equal the host float64 path on the same (widened) rows, and the caller's tensor
    is bitwise unchanged."""
    import torch
    from sklearn.preprocessing import MinMaxScaler

    from chronoclust_b200.synth import config_params

    cfg = config_params("C2")
    raw = raw_series(40000, 12, 3, 20, 11, cast=np.float64)
    sk = MinMaxScaler().fit(np.concatenate(raw, axis=0))
    Xs = [(x if scaled else sk.transform(x)).astype(dtype) for x in raw]
    sk = sk if scaled else None
    a, b = make(cfg), make(cfg)
    side = torch.cuda.Stream()
    for t, X in enumerate(Xs):
        a.online_microcluster_maintenance(X.astype(np.float64), t, scaler=sk)
        big, view = cuda_rows(X, getattr(torch, dtype), side)
        with torch.cuda.stream(side):
            before = big.clone()
            b.online_microcluster_maintenance(view, t, scaler=sk)
            after = big.clone()
        torch.cuda.synchronize()
        assert torch.equal(before.view(torch.uint8), after.view(torch.uint8)), "the caller's tensor was written"
        assert isinstance(b.last_assignment, np.ndarray) and isinstance(b.last_stage, np.ndarray)
        assert_same(a, b, f"cuda {dtype} scaled={scaled} t{t}", points=True)
        # downstream of the per-cell results: unchanged
        assert (a.cluster_labels_for_points() == b.cluster_labels_for_points()).all()


@gpu
def test_points_identical_across_input_paths():
    """The points dicts of pcore and outlier microclusters (keys and coordinates) do not depend on how the rows came in."""
    import torch

    z = load("c1.npz")
    X32 = z["scaled0"].astype(np.float32)
    big = np.zeros((X32.shape[0], X32.shape[1] + 4), np.float32)
    big[:, :X32.shape[1]] = X32
    feeds = {
        "numpy f32": X32, "numpy f32 view": big[:, :X32.shape[1]], "numpy f32 fortran": np.asfortranarray(X32),
        "cpu tensor f32": torch.from_numpy(X32), "cuda f32": torch.from_numpy(X32).cuda(),
        "cuda f64": torch.from_numpy(X32.astype(np.float64)).cuda(),
        "cuda f32 view": torch.from_numpy(big).cuda()[:, :X32.shape[1]],
    }
    a = make(config_of(z))
    a.online_microcluster_maintenance(X32.astype(np.float64), 0)
    ref = points_sample(a, 4)
    assert sum(len(p) for p in ref) > 0
    for what, X in feeds.items():
        h = make(config_of(z))
        h.online_microcluster_maintenance(X, 0)
        got = points_sample(h, 4)
        assert len(got) == len(ref), what
        for p, q in zip(ref, got):
            assert list(p.keys()) == list(q.keys()) and p == q, what
            assert all(type(v) is float for row in q.values() for v in row), what


# ---- device scaler fit -----------------------------------------------------------------------------------------------
@gpu
def test_colminmax_ex_on_float32_rows():
    import torch

    from chronoclust_b200 import _lib
    from chronoclust_b200.scaling import Scaler

    rng = np.random.default_rng(8)
    N, D, ld = 70001, 7, 9
    buf = rng.normal(-20.0, 50.0, size=(N, ld)).astype(np.float32)
    buf[rng.random((N, ld)) < 0.001] = np.nan
    buf[:, 3] = -12.5  # constant column
    buf[:, 5] = np.nan
    buf[17, 5] = -0.0  # a column with one value
    wide = buf.astype(np.float64)
    t = torch.from_numpy(buf).cuda()
    mn = torch.empty(D, dtype=torch.float64, device="cuda")
    mx = torch.empty(D, dtype=torch.float64, device="cuda")
    _lib.check(_lib.lib().ccb_colminmax_ex(0, None, t.data_ptr(), _lib.DTYPE_F32, N, ld, D, mn.data_ptr(), mx.data_ptr()))
    torch.cuda.synchronize()
    assert bits_equal(mn.cpu().numpy(), np.nanmin(wide[:, :D], axis=0))
    assert bits_equal(mx.cpu().numpy(), np.nanmax(wide[:, :D], axis=0))
    fmn, fmx = Scaler.fit_columns_on_device(t[:, :D])
    assert bits_equal(fmn, np.nanmin(wide[:, :D], axis=0)) and bits_equal(fmx, np.nanmax(wide[:, :D], axis=0))
    fmn, fmx = Scaler.fit_columns_on_device(t.double()[:, :D])
    assert bits_equal(fmn, np.nanmin(wide[:, :D], axis=0)) and bits_equal(fmx, np.nanmax(wide[:, :D], axis=0))


# ---- rejections ------------------------------------------------------------------------------------------------------
@gpu
def test_ingest_ex_rejects_bad_arguments():
    import torch

    from chronoclust_b200 import _lib

    h = make(config_of(load("c1.npz")))
    h._ensure_handle(4)
    L = _lib.lib()
    X = np.zeros((10, 4), np.float64)
    assign, stage = np.zeros(10, np.int32), np.zeros(10, np.uint8)
    sc = np.ones(4)
    args = lambda dtype, ld, scale, min_: (h._h, _lib.ptr(X), dtype, 0, 10, ld, scale, min_, _lib.ptr(assign),
                                           _lib.ptr(stage))
    assert L.ccb_ingest_ex(*args(7, 4, None, None)) == -1  # CCB_EINVAL
    assert b"dtype" in L.ccb_last_error(h._h)
    assert L.ccb_ingest_ex(*args(_lib.DTYPE_F64, 4, _lib.ptr(sc), None)) == -1
    assert L.ccb_ingest_ex(*args(_lib.DTYPE_F64, 4, None, _lib.ptr(sc))) == -1
    assert L.ccb_ingest_ex(*args(_lib.DTYPE_F32, 3, None, None)) == -1
    t = torch.zeros((10, 4), dtype=torch.float64, device="cuda")
    out = torch.empty(2, 4, dtype=torch.float64, device="cuda")
    assert L.ccb_colminmax_ex(0, None, t.data_ptr(), 7, 10, 4, 4, out[0].data_ptr(), out[1].data_ptr()) == -1


@gpu
def test_cuda_tensor_on_another_device_is_rejected():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    z = load("c1.npz")
    h = make(config_of(z), device=0)
    with pytest.raises(ValueError):
        h.online_microcluster_maintenance(torch.from_numpy(z["scaled0"]).to("cuda:1"), 0)
    assert h._h is None  # rejected before the handle (or anything on the device) was touched


# ---- the dispatch helper (CPU) ---------------------------------------------------------------------------------------
def test_dispatch_passes_float_rows_without_a_copy():
    import torch

    from chronoclust_b200 import _lib
    from chronoclust_b200.hddstream import _input_rows

    x32 = np.arange(60, dtype=np.float32).reshape(10, 6)
    p, code, dev, ld, keep = _input_rows(x32, 0)
    assert (p, code, dev, ld) == (x32.ctypes.data, _lib.DTYPE_F32, False, 6) and keep is x32
    big = np.arange(90, dtype=np.float64).reshape(10, 9)
    view = big[:, :6]
    p, code, dev, ld, keep = _input_rows(view, 0)
    assert (p, code, dev, ld) == (big.ctypes.data, _lib.DTYPE_F64, False, 9) and keep is view
    big32 = big.astype(np.float32)
    p, code, dev, ld, _ = _input_rows(big32[2:, :4], 0)
    assert (p, code, dev, ld) == (big32.ctypes.data + 2 * 9 * 4, _lib.DTYPE_F32, False, 9)
    for t, c in ((torch.from_numpy(x32), _lib.DTYPE_F32), (torch.from_numpy(big)[:, :6], _lib.DTYPE_F64)):
        p, code, dev, ld, keep = _input_rows(t, 0)
        assert (p, code, dev, ld) == (t.data_ptr(), c, False, t.stride(0))
        assert keep.shape == tuple(t.shape) and (keep == t.numpy()).all()


@pytest.mark.parametrize("kind", ["fortran", "int", "column_strided", "list", "float16", "byteswapped"])
def test_dispatch_converts_other_inputs_to_float64_rows(kind):
    import torch

    from chronoclust_b200 import _lib
    from chronoclust_b200.hddstream import _input_rows

    base = np.arange(70, dtype=np.float64).reshape(10, 7) / 8.0
    x = {"fortran": np.asfortranarray(base), "int": (base * 8).astype(np.int64),
         "column_strided": np.repeat(base, 2, axis=1)[:, ::2], "list": base.tolist(),
         "float16": torch.from_numpy(base.astype(np.float16)), "byteswapped": base.astype(">f8")}[kind]
    p, code, dev, ld, keep = _input_rows(x, 0)
    assert code == _lib.DTYPE_F64 and not dev and ld == 7
    assert keep.dtype == np.float64 and keep.flags.c_contiguous and p == keep.ctypes.data
    assert bits_equal(keep, base * (8 if kind == "int" else 1))


def test_points_view_widens_float32_rows_before_the_scaler():
    """float32 rows hand out the coordinates the float64 path hands out for the widened rows, scaled or not."""
    from sklearn.preprocessing import MinMaxScaler

    from chronoclust_b200.hddstream import _PointsView

    rng = np.random.default_rng(1)
    X32 = rng.normal(0.0, 30.0, size=(50, 4)).astype(np.float32)
    X64 = X32.astype(np.float64)
    sk = MinMaxScaler().fit(X64)
    assign = rng.integers(0, 3, size=50).astype(np.int32)
    for scaler in (None, (sk.scale_, sk.min_)):
        v32, v64 = _PointsView(), _PointsView()
        v32.add(X32, assign, scaler)
        v64.add(X64, assign, scaler)
        for uid in range(3):
            a, b = v32.points_of(uid), v64.points_of(uid)
            assert list(a.keys()) == list(b.keys()) and a == b
            assert all(type(v) is float for row in a.values() for v in row)
