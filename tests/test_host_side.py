"""CPU suite for the host side: the C-ABI library loads and exports every declared symbol, the
lineage / association trackers behave like the reference's (scenarios of tests/tracking_test/*), the
parameter derivation matches hddstream.py:89-128 (unittest_hddstream.py:10-41)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from chronoclust_b200 import _lib, build

    build.build()
    L = C.CDLL(_lib.SO_PATH)
    header = open(os.path.join(ROOT, "include", "chronoclust_b200.h")).read()
    declared = set(re.findall(r"\b(ccb_[a-z0-9_]+)\s*\(", header))
    declared -= {"ccb_handle"}
    assert declared, "no declarations parsed"
    for name in sorted(declared):
        assert hasattr(L, name), f"{name} declared in the header but not exported"
    assert declared == set(_lib.SYMBOLS), (declared ^ set(_lib.SYMBOLS))


def test_no_cpu_fallback_without_device():
    """Without a CUDA device handle creation must fail loudly (this container has no GPU)."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import logging

    from chronoclust_b200 import _lib
    from chronoclust_b200.hddstream import HDDStream

    h = HDDStream({"beta": 0.2, "delta": 0.05, "epsilon": 0.03, "lambda": 2, "k": 4, "mu": 0.01, "pi": 3,
                   "omicron": 0.0, "upsilon": 6.5}, logging.getLogger("t"))
    with pytest.raises(_lib.CCBError):
        h.online_microcluster_maintenance(np.random.rand(10, 3), 0)


def test_product_does_not_import_oracle():
    import subprocess
    import sys

    code = ("import sys; sys.path.insert(0, %r); import chronoclust_b200.app, chronoclust_b200.hddstream; "
            "assert not any(m == 'oracle' or m.startswith('oracle.') for m in sys.modules), 'oracle imported'") % ROOT
    subprocess.check_call([sys.executable, "-c", code])
    for dirpath, _, files in os.walk(os.path.join(ROOT, "chronoclust_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src and "libcco" not in src


def test_dataset_dependent_parameters():
    """unittest_hddstream.py:10-41: pi = D when 0, mu = mu*N, omicron from the PREVIOUS N, upsilon = v*eps."""
    import logging

    from chronoclust_b200.hddstream import HDDStream

    cfg = {"beta": 0.5, "delta": 0.1, "epsilon": 0.2, "lambda": 1, "k": 3, "mu": 0.05, "pi": 0, "omicron": 0.01,
           "upsilon": 2}
    h = HDDStream(cfg, logging.getLogger("t"))
    assert h.upsilon == 2.0 * 0.2 and h.epsilon_squared == 0.2 ** 2 and h.delta_squared == 0.1 ** 2
    X = np.zeros((200, 7))
    h._set_dataset_dependent_parameters(X)
    assert h.pi == 7 and h.mu == 0.05 * 200 and h.omicron == 0.0
    h._set_dataset_dependent_parameters(np.zeros((50, 7)))
    assert h.omicron == 0.01 * 200 and h.mu == 0.05 * 50
    cfg["pi"] = 2.5
    h2 = HDDStream(cfg, logging.getLogger("t"))
    h2._set_dataset_dependent_parameters(X)
    assert h2.pi == round(2.5)
    with pytest.raises(SystemExit):
        HDDStream(dict(cfg, delta=1.5), logging.getLogger("t"))


def _cl(pcores, w=1.0):
    from chronoclust_b200.objects import Cluster

    return Cluster(list(pcores), [0.0], w, [1.0])


def test_lineage_new_split_merge():
    from chronoclust_b200.tracking import TrackByLineage

    t = TrackByLineage()
    a, b = _cl([0, 1], 5), _cl([2], 9)
    t.add_new_child_cluster(b)
    t.add_new_child_cluster(a)
    t.calculate_ids()
    assert [c.id for c in t.child_clusters] == ["A", "B"]  # sorted by weight, letters in that order
    t.transfer_child_to_parent()
    # split: pcores 0 and 1 part ways; the child with more parent pcores keeps the label
    c1, c2, c3 = _cl([0, 5], 3), _cl([1], 2), _cl([2], 9)
    for c in (c1, c2, c3):
        t.add_new_child_cluster(c)
    t.calculate_ids()
    ids = {tuple(c.pcore_ids): c.id for c in t.child_clusters}
    assert ids[(0, 5)] == "A" and ids[(1,)] == "A|1" and ids[(2,)] == "B"
    t.transfer_child_to_parent()
    # merge of A|1 and B, and A splits again -> A|2 (split counter remembered)
    m, s1, s2 = _cl([1, 2], 8), _cl([0], 1), _cl([5], 2)
    for c in (m, s1, s2):
        t.add_new_child_cluster(c)
    t.calculate_ids()
    ids = {tuple(c.pcore_ids): c.id for c in t.child_clusters}
    assert ids[(1, 2)] == "(A|1,B)"
    assert sorted([ids[(0,)], ids[(5,)]]) == ["A", "A|2"]


def test_lineage_more_than_26_clusters():
    from chronoclust_b200.tracking import TrackByLineage

    t = TrackByLineage()
    for i in range(28):
        t.add_new_child_cluster(_cl([i], i))
    t.calculate_ids()
    ids = [c.id for c in t.child_clusters]
    assert ids[:26] == list("ABCDEFGHIJKLMNOPQRSTUVWXYZ") and ids[26:] == ["AA", "BB"]


def test_historical_association():
    from chronoclust_b200.objects import Microcluster
    from chronoclust_b200.tracking import TrackByHistoricalAssociation

    def mc(pid, cen):
        return Microcluster(cf1=np.zeros(2), cf2=np.zeros(2), id=[pid], cumulative_weight=1,
                            preferred_dimension_vector=np.ones(2), cluster_centroids=np.array(cen, float))

    t = TrackByHistoricalAssociation()
    p1, p2 = _cl([0]), _cl([1])
    p1.id, p2.id = "A", "B"
    p1.pcore_objects, p2.pcore_objects = [mc(0, [0, 0])], [mc(1, [10, 10])]
    t.set_current_clusters([p1, p2])
    t.track_cluster_history()
    assert p1.get_historical_associates_as_str() == "None"
    t.transfer_current_to_previous()
    c = _cl([2, 3])
    c.id = "C"
    c.pcore_objects = [mc(2, [1, 1]), mc(3, [9, 9])]
    t.set_current_clusters([c])
    t.track_cluster_history()
    assert c.get_historical_associates_as_str() == "A&B"


def test_points_view_applies_the_device_scaler_on_the_host_side():
    """When raw rows were scaled on the device (ccb_ingest_scaled), Microcluster.points hands out x * scale_ + min_ of the
    requested rows -- the same two roundings (scaling/scaler.py:43-47 -> MinMaxScaler.transform)."""
    from sklearn.preprocessing import MinMaxScaler

    from chronoclust_b200.hddstream import _PointsView

    rng = np.random.default_rng(0)
    X = rng.normal(0.0, 30.0, size=(50, 4))
    sk = MinMaxScaler().fit(X)
    assign = rng.integers(0, 3, size=50).astype(np.int32)
    raw_view, scaled_view = _PointsView(), _PointsView()
    raw_view.add(X, assign, (sk.scale_, sk.min_))
    scaled_view.add(sk.transform(X), assign)
    for uid in range(3):
        a, b = raw_view.points_of(uid), scaled_view.points_of(uid)
        assert list(a.keys()) == list(b.keys()) == sorted(a.keys())
        assert a == b


def test_streamed_scaler_fit_equals_one_fit_over_all_timepoints(tmp_path):
    """Scaler fits file by file (partial_fit); the fitted vectors and the transform equal those of the reference's single
    fit over the concatenation of all timepoints (scaling/scaler.py:27-36), bit for bit."""
    from sklearn.preprocessing import MinMaxScaler

    from chronoclust_b200.scaling import Scaler

    rng = np.random.default_rng(4)
    parts, files = [], []
    for t in range(4):
        X = rng.normal(10.0 * t, 40.0, size=(300 + 17 * t, 5))
        X[:, 2] = 3.25  # a constant marker
        parts.append(X)
        f = tmp_path / f"d{t}.csv"
        np.savetxt(f, X, delimiter=",", header="a,b,c,d,e", comments="", fmt="%.17g")
        files.append(str(f))
    s = Scaler(files)
    import pandas as pd
    parts = [pd.read_csv(f, header=0, sep=',').to_numpy() for f in files]  # what both implementations see
    allc = np.concatenate(parts, axis=0)
    ref = MinMaxScaler().fit(allc)
    same = lambda a, b: (np.ascontiguousarray(a).view(np.uint64) == np.ascontiguousarray(b).view(np.uint64)).all()
    assert same(s.scaler.scale_, ref.scale_) and same(s.scaler.min_, ref.min_)
    assert same(s.scale_data(parts[1]), ref.transform(parts[1]))
    assert same(s.reverse_scaling(ref.transform(parts[2])), ref.inverse_transform(ref.transform(parts[2])))
    sc, mn = s.device_vectors()
    assert same(parts[3] * sc + mn, ref.transform(parts[3]))
    assert len(s.get_input_data()) == len(allc)


def test_hostio_repr_is_python_repr():
    """csrc/hostio.c formats float64 exactly like repr(float) (= what pandas' to_csv writes): shortest round-trip digits,
    positional / exponent notation switch at 1e-4 and 1e16, '.0' on integers, subnormals, signed zero, infinities."""
    import ctypes as C

    from chronoclust_b200 import _hostio

    L = _hostio.lib()
    buf = C.create_string_buffer(64)
    rng = np.random.default_rng(4)
    vals = [0.1, 5.0, 1e-5, 0.0001, 1e15, 1e16, 1e17, 1.5e-7, 123456789.0, 1e22, -0.0, 0.0, 1 / 3, 2 / 3, 1e-310, 5e-324,
            1.7976931348623157e308, float("inf"), -float("inf"), 9.999999999999999e15, 0.00011, 9.5e-5, 2.5e-4,
            1234567890123456.0, 12345678901234567.0, 2.2250738585072014e-308, 2.225073858507201e-308, 1e100, -1e-100]
    vals += rng.random(3000).tolist() + (rng.random(3000) * 1e6).tolist() + (rng.standard_normal(3000) * 1e-6).tolist()
    vals += np.exp(rng.uniform(-740, 709, 3000)).tolist() + np.round(rng.random(1000), 3).tolist()
    vals += rng.integers(-1000, 1000, 500).astype(float).tolist()
    for v in vals:
        n = L.ccbio_repr(v, buf)
        assert buf.raw[:n].decode() == repr(v), (repr(v), buf.raw[:n])
    assert L.ccbio_repr(float("nan"), buf) == 0  # an empty field, pandas' na_rep


def test_hostio_table_is_byte_identical_to_pandas(tmp_path):
    """The native multi-threaded writer of cluster_points_D{t}.csv against DataFrame.to_csv(index=False): same bytes,
    including quoted labels (merged lineage ids contain commas), quoted column names, NaN cells and a strided input."""
    import pandas as pd

    from chronoclust_b200 import _hostio

    rng = np.random.default_rng(9)
    N, D = 50_003, 7
    wide = rng.random((N, D + 2)) * np.array([1e-6, 1e-3, 1.0, 10.0, 1e3, 1e7, 1e17, 1.0, 1.0])
    X = wide[:, :D]  # row stride != D
    X[5, 3] = np.nan
    X[7, 0] = 1e-310
    X[9, 2] = -0.0
    labels = ["None", "A", "B|1", "(A,B)", 'q"x', "((A,B),C)|2"]
    li = rng.integers(0, len(labels), N).astype(np.int32)
    names = ["FSC-A", "x,y"] + [f"m{j}" for j in range(2, D)]
    cols = {"id": np.arange(N), "cluster_id": np.array(labels, dtype=object)[li]}
    for j in range(D):
        cols[names[j]] = X[:, j]
    pd.DataFrame(cols).to_csv(tmp_path / "pandas.csv", index=False)
    for threads in (0, 1, 3):
        _hostio.write_points_csv(tmp_path / "native.csv", ["id", "cluster_id"] + names, X, li, labels, threads=threads)
        assert open(tmp_path / "native.csv", "rb").read() == open(tmp_path / "pandas.csv", "rb").read()
    _hostio.write_points_csv(tmp_path / "empty.csv", ["id", "cluster_id"] + names, np.zeros((0, D)), np.zeros(0, np.int32), labels)
    assert open(tmp_path / "empty.csv").read() == ",".join(["id", "cluster_id", "FSC-A", '"x,y"'] + names[2:]) + "\n"


def _gating_case(seed=3, Q=37, P=11, D=6, k=4.0):
    from chronoclust_b200.objects import Cluster

    rng = np.random.default_rng(seed)
    gates = {tuple(rng.random(D).tolist()): f"pop{j}" for j in range(P)}
    clusters = []
    for q in range(Q):
        pref = np.where(rng.random(D) < 0.5, k, 1.0)
        clusters.append(Cluster([q], rng.random(D), 1.0, pref))
    first = next(iter(gates))
    clusters[0].centroid = np.array(first) + 1e-3   # a clear winner
    twin = tuple((np.array(first) + 2e-3).tolist())  # ... and an exact tie between two gates for cluster 1
    gates[twin] = "twin"
    clusters[1].centroid = np.array(first) + 1e-3
    clusters[1].preferred_dimensions = np.ones(D)
    return gates, clusters


def test_closest_gates_without_cuda_uses_the_reference_expression():
    """SURVEY 8f-4 host side: with no CUDA device the gating labels come from the reference's own scan
    (find_closest_gating, app.py:497-512): first strictly smaller distance wins, dict order."""
    from chronoclust_b200 import app

    gates, clusters = _gating_case()
    got = app.closest_gates(gates, clusters, None, 4.0)
    exp = []
    for c in clusters:
        best, lab = None, None
        for cen, name in gates.items():
            d = 0.0
            for ci, pi_, di in zip(c.centroid, cen, c.preferred_dimensions):
                d += ((float(pi_) - float(ci)) ** 2) / float(di)
            if best is None or d < best:
                best, lab = d, name
        exp.append(lab)
    assert got == exp and got[0] == "pop0"
    assert app.closest_gates(gates, [], None, 4.0) == []


def test_bench_dump_outputs_keeps_a_fixed_sample_under_the_budget(tmp_path):
    """bench.py --dump-outputs: below the budget every array is written whole; above it, every array of more than one row
    keeps the same seeded sample of its rows (row numbers written beside it), the same in every run."""
    import bench

    rng = np.random.default_rng(1)
    arrays = {"assign": rng.integers(0, 1000, 200_000).astype(np.float64), "cen": rng.random((5000, 12)), "w": np.ones(1)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, budget=1_000_000)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(os.listdir(tmp_path / "b")) == ["assign.npy", "assign_rows.npy", "cen.npy", "cen_rows.npy", "w.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 1_000_000 + 128 * len(files)  # (+ .npy headers)
    for name in ("assign", "cen"):
        rows = np.load(tmp_path / "a" / f"{name}_rows.npy").astype(np.int64)
        got = np.load(tmp_path / "a" / f"{name}.npy")
        assert len(rows) > 0 and (got == arrays[name][rows]).all() and (got == np.load(tmp_path / "b" / f"{name}.npy")).all()
    bench.dump_outputs(str(tmp_path / "whole"), arrays)
    assert sorted(os.listdir(tmp_path / "whole")) == ["assign.npy", "cen.npy", "w.npy"]
    assert (np.load(tmp_path / "whole" / "assign.npy") == arrays["assign"]).all()


def test_generated_documents_carry_no_unfilled_field():
    """DESIGN.md / README.md are generated from tools/templates/*.in by tools/fill_docs.py: no @FIELD@ may survive, and
    the text around the numbers must be the template's."""
    import re

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for name in ("DESIGN.md", "README.md"):
        doc = open(os.path.join(root, name), encoding="utf-8").read()
        tpl = open(os.path.join(root, "tools", "templates", name + ".in"), encoding="utf-8").read()
        assert not re.findall(r"@[A-Z0-9_]+@", doc), name
        # every literal stretch of the template (between two fields) occurs in the generated document
        for piece in re.split(r"@[A-Z0-9_]+@", tpl):
            assert piece in doc, f"{name} is out of date with its template near: {piece[:80]!r}"
