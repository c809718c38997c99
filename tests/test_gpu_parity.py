"""GPU suite (-m gpu): the CUDA path behind the C ABI against the golden vectors of the live reference
and against the CPU oracle on the same seeded inputs.  Bit-exact everywhere: assignments, list order,
ids, weights, CF1/CF2, centroids, preference vectors, cluster membership / set order / sums."""
import ctypes as C
import json
import logging
import os

import numpy as np
import pytest

from helpers import (GOLDEN, STRESS_NAMES, assert_clusters_equal, assert_list_equal, bits_equal, config_of, load,
                     stress_inputs)

pytestmark = pytest.mark.gpu

LOG = logging.getLogger("test")


def make(cfg, **kw):
    from chronoclust_b200.hddstream import HDDStream

    return HDDStream(dict(cfg), LOG, **kw)


def clusters_of(h):
    return [(c.members_in_claim_order, c.cumulative_weight, c.CF1, c.CF2, c.cluster_centroids,
             c.preferred_dimension_vector) for c in h.final_clusters]


def run_against_golden(z, Xs, what, **kw):
    h = make(config_of(z), **kw)
    for i, (t, X) in enumerate(zip(z["timestamps"].tolist(), Xs)):
        h.online_microcluster_maintenance(X, int(t))
        P = f"t{i}_"
        assert (h.last_assignment == z[P + "assign"]).all(), \
            f"{what} t{i}: {(h.last_assignment != z[P + 'assign']).sum()} assignments differ, first at " \
            f"{np.flatnonzero(h.last_assignment != z[P + 'assign'])[:5]}"
        for which, name in ((0, "p_"), (1, "o_")):
            assert_list_equal(h.export_arrays(which), z, P + name, f"{what} t{i} list{which}")
        assert h.counts()[2:] == z[P + "counters"].tolist()
        assert_clusters_equal(clusters_of(h), z, P, f"{what} t{i}")
    return h


# the ordered engine's knobs -- block length cap / smallest block / refinement rounds / graph vs stream launches -- never
# change results
BSV_KNOBS = [dict(), dict(chunk=96, bsv_bmin=32, bsv_iters=1), dict(chunk=2048, bsv_bmin=64, bsv_iters=2),
             dict(chunk=512, bsv_bmin=512, bsv_iters=6), dict(bsv_stream=1), dict(chunk=300, bsv_bmin=16, bsv_stream=1)]


@pytest.mark.parametrize("knobs", BSV_KNOBS, ids=lambda k: "-".join(f"{a}{b}" for a, b in k.items()) or "default")
@pytest.mark.parametrize("name", STRESS_NAMES)
def test_stress_matches_reference_bsv(name, knobs):
    z = load(f"stress_{name}.npz")
    h = run_against_golden(z, stress_inputs(z), f"{name}/bsv{knobs}", **knobs)
    st = h.stats()
    assert st["bsv_blocks"] > 0 and st["kernel_launches"] > 0


@pytest.mark.parametrize("chunk", [0, 97])
def test_c1_matches_reference(chunk):
    z = load("c1.npz")
    h = run_against_golden(z, [z[f"scaled{t}"] for t in range(5)], "c1", chunk=chunk)
    st = h.stats()
    assert st["kernel_launches"] > 0 and st["points"] == sum(z[f"scaled{t}"].shape[0] for t in range(5))


def test_points_view_matches_assignment():
    z = load("c1.npz")
    h = make(config_of(z))
    X = z["scaled0"]
    h.online_microcluster_maintenance(X, 0)
    seen = 0
    for mc in h.pcore_MC + h.outlier_MC:
        keys = list(mc.points.keys())
        assert keys == sorted(keys)
        assert (h.last_assignment[keys] == mc.prev_outlier_id).all()
        assert mc.points[keys[0]] == X[keys[0]].tolist()
        seen += len(keys)
    assert seen == X.shape[0]


@pytest.mark.parametrize("csr_min_m", [2048, 0], ids=["bitrows", "csr"])
def test_offline_sets_match_predecon(csr_min_m):
    """24 randomised pcore sets pushed through the reference's PreDeCon.run (predecon.py:49-120): neighbourhoods,
    subspace vectors, weighted neighbourhoods and the ordered cluster growth -- the latter through both of its
    device formulations (bit-row scan for small M, isolated-MC pre-pass + CSR lists for large M)."""
    _run_offline_sets(load("offline_sets.npz"), csr_min_m)


def _run_offline_sets(z, csr_min_m):
    for s in range(int(z["nset"])):
        P = f"s{s}_"
        D, M, k, pi, delta, E = z[P + "params"]
        D, M, pi = int(D), int(M), int(pi)
        cen, w, cf1, cf2, ids, core = (z[P + n] for n in ("cen", "w", "cf1", "cf2", "ids", "core"))
        wc, wn_ = w[core], w[~core]
        separable = not (len(wc) and len(wn_) and wc.min() <= wn_.max())
        mu = 0.0
        if separable:
            mu = float((wc.min() + wn_.max()) / 2) if len(wc) and len(wn_) else (0.0 if len(wc) else 1e300)
        cfg = {"beta": 0.0, "delta": float(delta), "epsilon": 1e150, "lambda": 0, "k": float(k), "mu": 0.0, "pi": pi,
               "omicron": 0.0, "upsilon": float(E) / 1e150}
        h = make(cfg, off_csr_min_m=csr_min_m if csr_min_m else 1)
        assert h.upsilon == float(E), "test construction: upsilon*epsilon must reproduce E exactly"
        h.dataset_dimensionality = D
        h._ensure_handle(D)
        h.pi, h.mu, h.omicron = pi, mu, 0.0
        from chronoclust_b200 import _lib
        _lib.check(_lib.lib().ccb_begin_timepoint(h._h, mu, 0.0, pi, 0, 1.0), h._h)
        h.import_arrays(0, ids, ids, w, cf1, cf2, cen, np.ones((M, D)))
        h.offline_clustering(0)
        got_core, nbr, wn, subw = h.offline_intermediates()
        exp_nbr = np.unpackbits(z[P + "nbr"])[:M * M].reshape(M, M)
        exp_wn = np.unpackbits(z[P + "wnbr"])[:M * M].reshape(M, M)
        assert (nbr == exp_nbr).all(), f"set {s}: neighbourhoods differ"
        assert bits_equal(subw, z[P + "subw"]), f"set {s}: subspace preference vectors differ"
        assert (wn == exp_wn).all(), f"set {s}: weighted neighbourhoods differ"
        if separable:
            assert (got_core.astype(bool) == core).all()
            assert_clusters_equal(clusters_of(h), z, P, f"offline set {s}")


def test_kats_on_device():
    """The reference's unit-test known answers through the CUDA path."""
    import torch
    from chronoclust_b200 import _lib

    kat = json.load(open(os.path.join(GOLDEN, "kat.json")))
    L = _lib.lib()
    # projected distance (unittest_microcluster.py:10-32) through kernel 1
    for case in kat["projdist"]:
        x = torch.tensor([case["pt"]], dtype=torch.float64, device="cuda")
        cen = torch.tensor([case["cen"]], dtype=torch.float64, device="cuda")
        mask = sum(1 << d for d, v in enumerate(case["pref"]) if v == 15.0)
        m = torch.tensor([mask], dtype=torch.int64, device="cuda")
        slot = torch.full((1,), -5, dtype=torch.int32, device="cuda")
        dist = torch.zeros(1, dtype=torch.float64, device="cuda")
        _lib.check(L.ccb_nearest(0, None, x.data_ptr(), 1, 3, 3, cen.data_ptr(), m.data_ptr(), 1, 15.0, slot.data_ptr(),
                                 dist.data_ptr()))
        torch.cuda.synchronize()
        assert slot.item() == 0 and dist.item() == case["dist"] and round(dist.item(), 2) == case["rounded"]
    # preference vector / CF / centroid after 10 ordered absorbs (unittest_microcluster.py:34-80)
    pts = np.ascontiguousarray(kat["prefvec"]["pts"], np.float64)
    for case in kat["prefvec"]["cases"]:
        cfg = {"beta": 1.0, "delta": case["delta2"] ** 0.5, "epsilon": 1e6, "lambda": 0, "k": case["k"], "mu": 1e9,
               "pi": 0, "omicron": 0.0, "upsilon": 1.0}
        h = make(cfg)
        h.delta_squared = case["delta2"]
        h.online_microcluster_maintenance(pts, 0, run_offline=False)
        ids, uids, w, cf1, cf2, cen, pref = h.export_arrays(1)
        assert len(ids) == 1 and w[0] == case["w"]
        assert bits_equal(cf1[0], case["cf1"]) and bits_equal(cf2[0], case["cf2"]) and bits_equal(cen[0], case["cen"])
        assert pref[0].tolist() == case["pref"]
    # radius^2 (unittest_microcluster.py:82-104) through the core flag: eps^2 just above / below the answer
    r = kat["radius2"]
    for eps2, expect in ((np.nextafter(r["r2"], 1.0), 1), (r["r2"], 1), (np.nextafter(r["r2"], 0.0), 0)):
        cfg = {"beta": 0.0, "delta": 0.5, "epsilon": float(eps2) ** 0.5, "lambda": 0, "k": 16.0, "mu": 0.0, "pi": 0,
               "omicron": 0.0, "upsilon": 1.0}
        h = make(cfg)
        h.epsilon_squared = float(eps2)
        h.dataset_dimensionality = 20
        h._ensure_handle(20)
        _lib.check(L.ccb_begin_timepoint(h._h, 0.0, 0.0, 20, 0, 1.0), h._h)
        one = lambda v: np.ascontiguousarray([v], np.float64)
        h.import_arrays(0, [0], [0], [r["w"]], one(r["cf1"]), one(r["cf2"]), one(r["cf1"]) / r["w"], one(r["pref"]))
        h.offline_clustering(0)
        assert h.offline_intermediates()[0][0] == expect


@pytest.mark.parametrize("D,M,k", [(3, 5, 4.0), (12, 300, 4.0), (40, 1000, 4.0), (12, 77, 3.0), (7, 4100, 1.0),
                                   (64, 33, 2.0)])
def test_kernel1_nearest_bit_exact(D, M, k):
    """Kernel 1 against a scalar restatement (sequential sum over d, true division, strict-< first wins)."""
    import torch
    from chronoclust_b200 import _lib
    from oracle.oracle import lib as olib, _p

    rng = np.random.default_rng(D * 1000 + M)
    N = 3000
    X = rng.random((N, D))
    cen = rng.random((M, D))
    cen[M // 2] = cen[0]  # exact tie between two microclusters: the earlier one must win
    maskbits = rng.random((M, D)) < 0.5
    maskbits[M // 2] = maskbits[0]
    pref = np.where(maskbits, k, 1.0)
    masks = np.array([sum(1 << d for d in range(D) if maskbits[j, d]) for j in range(M)], np.uint64).astype(np.int64)
    tX, tc = torch.from_numpy(X).cuda(), torch.from_numpy(cen).cuda()
    tm = torch.from_numpy(masks).cuda()
    slot = torch.empty(N, dtype=torch.int32, device="cuda")
    dist = torch.empty(N, dtype=torch.float64, device="cuda")
    _lib.check(_lib.lib().ccb_nearest(0, None, tX.data_ptr(), N, D, D, tc.data_ptr(), tm.data_ptr(), M, k,
                                      slot.data_ptr(), dist.data_ptr()))
    torch.cuda.synchronize()
    L = olib()
    exp_slot, exp_dist = np.zeros(N, np.int32), np.zeros(N)
    for i in range(0, N, 7):  # a sample of rows through the oracle's scalar kernel
        best, bd = -1, 0.0
        for j in range(M):
            d = L.cco_kat_projected_distance(_p(np.ascontiguousarray(cen[j])), _p(np.ascontiguousarray(pref[j])),
                                             _p(np.ascontiguousarray(X[i])), D)
            if best < 0 or d < bd:
                best, bd = j, d
        assert slot[i].item() == best and dist[i].item() == bd, (i, slot[i].item(), best, dist[i].item(), bd)


@pytest.mark.parametrize("D,M,k,tiny", [(12, 500, 4.0, 0.0), (12, 500, 4.0, 1e-160), (40, 200, 16.0, 1e-158),
                                        (12, 260, 4.0, 1e-200), (5, 90, 2.0, 3e-162)])
def test_kernel1_fused_weight_step_bit_exact(D, M, k, tiny):
    """Kernel 1 folds the power-of-two preference weight into the accumulate (fma(t*t, 1/k, acc)); that is the
    reference's acc + (t*t)/k (mc_functions.py:35-43) only while (t*t)/k stays normal.  Inputs whose squared
    differences fall into the subnormal range must take the unfused sequence: every row is compared with numpy's
    elementwise IEEE arithmetic (no contraction), summed over d in index order, first minimum wins."""
    import torch
    from chronoclust_b200 import _lib

    rng = np.random.default_rng(D * 77 + M)
    N = 2048
    X = rng.random((N, D))
    cen = rng.random((M, D))
    if tiny:
        # a band of cells and microclusters living at magnitude `tiny`: (x - c)^2 ~ 1e-320 (subnormal), / k loses bits
        X[::3] *= tiny
        cen[::2] *= tiny
        X[5::7, ::2] = 0.0
    maskbits = rng.random((M, D)) < 0.6
    pref = np.where(maskbits, k, 1.0)
    masks = np.array([sum(1 << d for d in range(D) if maskbits[j, d]) for j in range(M)], np.uint64).astype(np.int64)
    tX, tc, tm = torch.from_numpy(X).cuda(), torch.from_numpy(cen).cuda(), torch.from_numpy(masks).cuda()
    slot = torch.empty(N, dtype=torch.int32, device="cuda")
    dist = torch.empty(N, dtype=torch.float64, device="cuda")
    _lib.check(_lib.lib().ccb_nearest(0, None, tX.data_ptr(), N, D, D, tc.data_ptr(), tm.data_ptr(), M, k,
                                      slot.data_ptr(), dist.data_ptr()))
    torch.cuda.synchronize()
    acc = np.zeros((N, M))
    for d in range(D):
        t = X[:, d, None] - cen[None, :, d]
        t = t * t
        t = t / pref[None, :, d]
        acc = acc + t
    exp_slot = acc.argmin(axis=1)
    exp_dist = acc[np.arange(N), exp_slot]
    assert (slot.cpu().numpy() == exp_slot).all()
    assert bits_equal(dist.cpu().numpy(), exp_dist)
    if tiny > 1e-165:  # (1e-200 squares underflow to exact zeros: a tie-break case, first minimum wins)
        assert ((acc > 0) & (acc < 2.3e-308)).any(), "the fixture must reach the subnormal range"


@pytest.mark.parametrize("cfgname,N,T", [("C2", 60000, 3), ("C3", 20000, 2)])
def test_online_offline_vs_oracle_mid_size(cfgname, N, T):
    """CUDA vs the (reference-pinned) oracle at sizes the reference itself cannot reach in test time."""
    from chronoclust_b200.synth import CONFIGS, config_params, gen
    from oracle.oracle import OracleHDDStream

    _, D, _, Cn, seed, _, _ = CONFIGS[cfgname]
    cfg = config_params(cfgname)
    Xs = gen(N, D, T, Cn, seed)
    h, o = make(cfg), OracleHDDStream(cfg)
    for t, X in enumerate(Xs):
        h.online_microcluster_maintenance(X, t)
        o.online_microcluster_maintenance(X, t)
        assert (h.last_assignment == o.assign_uid).all(), f"t{t}: first diff at {np.flatnonzero(h.last_assignment != o.assign_uid)[:5]}"
        assert (h.last_stage == o.stage).all()
        for which in (0, 1):
            e = o.export(which)
            got = h.export_arrays(which)
            assert len(got[0]) == len(e)
            assert (got[0] == e.ids).all() and (got[1] == e.uids).all()
            for g, x in zip(got[2:], (e.w, e.cf1, e.cf2, e.cen, e.pref)):
                assert bits_equal(g, x)
        oc = o.clusters()
        hc = clusters_of(h)
        assert len(oc) == len(hc)
        for (m1, w1, a1, b1, c1, p1), (m2, w2, a2, b2, c2, p2) in zip(hc, oc):
            assert list(m1) == list(m2) and w1 == w2
            assert bits_equal(a1, a2) and bits_equal(b1, b2) and bits_equal(c1, c2) and bits_equal(p1, p2)
    st = h.stats()
    print(cfgname, st)


def test_app_run_matches_reference_files(tmp_path):
    """chronoclust_b200.app.run on the reference's synthetic d0-d4 with the integration test's parameters
    and gating file: result.csv byte-identical to the reference's golden file, cluster_points labels
    identical on every row (normal_test.py:78-157)."""
    import pandas as pd

    from chronoclust_b200 import app

    z = load("c1.npz")
    files = []
    for t in range(5):
        f = tmp_path / f"synthetic_d{t}.csv"
        pd.DataFrame(z[f"raw{t}"], columns=["x", "y", "z"]).to_csv(f, index=False)
        files.append(str(f))
    cfg = config_of(z)
    out = tmp_path / "out"
    out.mkdir()
    app.run(data=files, output_directory=str(out), gating_centroid_file=os.path.join(GOLDEN, "c1_gating_centroids.csv"),
            param_beta=cfg["beta"], param_delta=cfg["delta"], param_epsilon=cfg["epsilon"], param_lambda=cfg["lambda"],
            param_k=cfg["k"], param_mu=cfg["mu"], param_pi=cfg["pi"], param_omicron=cfg["omicron"],
            param_upsilon=cfg["upsilon"])
    got = open(out / "result.csv", "rb").read()
    exp = open(os.path.join(GOLDEN, "c1_result.csv"), "rb").read()
    assert got == exp, "result.csv differs from the reference's golden file"
    lab = load("c1_labels.npz")
    for t in range(5):
        df = pd.read_csv(out / f"cluster_points_D{t}.csv", keep_default_na=False)
        assert (df["id"].to_numpy() == lab[f"ids{t}"]).all()
        assert (df["cluster_id"].astype(str).to_numpy() == lab[f"labels{t}"]).all()
        assert np.abs(df[["x", "y", "z"]].to_numpy() - lab[f"xyz{t}"]).max() < 1e-12
    assert os.path.exists(out / "parameters.csv") and os.path.exists(out / "program_images" / "hddstream")
    # degenerate run (no_cluster_test.py:29-43, 70-85): beta = mu = 1 -> no cluster, every cell labelled None
    out2 = tmp_path / "out2"
    out2.mkdir()
    small = []
    for t in range(5):
        f = tmp_path / f"small_d{t}.csv"
        pd.DataFrame(z[f"raw{t}"][:10], columns=["x", "y", "z"]).to_csv(f, index=False)
        small.append(str(f))
    app.run(data=small, output_directory=str(out2), param_beta=1, param_delta=0.05, param_epsilon=0.03, param_lambda=2,
            param_k=4, param_mu=1, param_pi=3, param_omicron=0.000000435, param_upsilon=6.5)
    assert len(open(out2 / "result.csv").read().splitlines()) == 1
    for t in range(5):
        df = pd.read_csv(out2 / f"cluster_points_D{t}.csv", keep_default_na=False)
        assert len(df) == 10 and (df["cluster_id"] == "None").all()


def test_pickle_roundtrip_continues_identically():
    import pickle

    z = load("stress_churn.npz")
    Xs = stress_inputs(z)
    h = make(config_of(z))
    for t in range(2):
        h.online_microcluster_maintenance(Xs[t], t)
    h2 = pickle.loads(pickle.dumps(h))
    for t in range(2, len(Xs)):
        h2.online_microcluster_maintenance(Xs[t], t)
        P = f"t{t}_"
        assert (h2.last_assignment == z[P + "assign"]).all()
        for which, name in ((0, "p_"), (1, "o_")):
            assert_list_equal(h2.export_arrays(which), z, P + name, f"restored t{t} list{which}")
        assert_clusters_equal(clusters_of(h2), z, P, f"restored t{t}")


def test_stateless_offline_stages_match_handle_path():
    """The row-sharded stage functions (world = 1) against the handle-level offline phase and the golden
    PreDeCon results: neighbour / weighted-neighbour rows, masks, labels, claim order."""
    import torch

    from chronoclust_b200.offline_sharded import CudaStages, sharded_offline

    z = load("offline_sets.npz")
    st = CudaStages(0, dnrm2_ptr=None)
    for s in range(int(z["nset"])):
        P = f"s{s}_"
        D, M, k, pi, delta, E = z[P + "params"]
        D, M, pi = int(D), int(M), int(pi)
        cen, core = z[P + "cen"], z[P + "core"]
        tc = torch.from_numpy(np.ascontiguousarray(cen)).cuda()
        tcore = torch.from_numpy(core.astype(np.uint8)).cuda()
        lab, order, cl_off, ncl, info = sharded_offline(st, tc, tcore, M, D, float(k), pi, float(delta), float(E),
                                                        float(E) ** 2)
        # membership per emitted cluster equals the reference's id sets (clusters with members only)
        ids = z[P + "ids"]
        got = [sorted(int(ids[x]) for x in order[cl_off[c]:cl_off[c + 1]]) for c in range(ncl)
               if cl_off[c + 1] > cl_off[c]]
        off = z[P + "cl_off"]
        exp = [sorted(z[P + "cl_idlist"][off[c]:off[c + 1]].tolist()) for c in range(len(off) - 1)]
        assert got == exp, f"set {s}"
        assert info["neighbour_count"] == int(np.unpackbits(z[P + "nbr"])[:M * M].sum())


def test_offline_borderline_pairs_resolved_by_dnrm2():
    """Centroids placed exactly on the eps-boundary (3-4-5 triangles): the device must flag them and the
    host must settle them with dnrm2 (<= E is inclusive) -- in the handle's offline phase and in the stateless
    row-sharded stage, with the scipy dnrm2 and with the built-in one, over all rows and over two row halves."""
    import torch

    from chronoclust_b200.offline_sharded import CudaStages
    cfg = {"beta": 0.0, "delta": 0.5, "epsilon": 1.0, "lambda": 0, "k": 4.0, "mu": 0.0, "pi": 0, "omicron": 0.0,
           "upsilon": 5.0}
    h = make(cfg)
    D = 2
    h.dataset_dimensionality = D
    h._ensure_handle(D)
    from chronoclust_b200 import _lib
    _lib.check(_lib.lib().ccb_begin_timepoint(h._h, 0.0, 0.0, D, 0, 1.0), h._h)
    cen = np.array([[0.0, 0.0], [3.0, 4.0], [6.0, 8.0], [3.0, 4.0000000000000036]])  # |c0-c1| = 5 = E exactly
    M = len(cen)
    w = np.full(M, 10.0)
    h.import_arrays(0, np.arange(M), np.arange(M), w, cen * 10, (cen ** 2 + 0.01) * 10, cen, np.ones((M, D)))
    h.offline_clustering(0)
    core, nbr, wn, subw = h.offline_intermediates()
    assert h.stats()["borderline_pairs"] >= 2
    assert nbr[0, 1] == 1 and nbr[1, 0] == 1 and nbr[1, 2] == 1  # distance exactly E is a neighbour
    assert nbr[0, 2] == 0 and nbr[0, 3] == 0  # 10 > 5; 5.000000000000003 > 5
    tc = torch.from_numpy(cen).cuda()
    E = h.upsilon
    for st in (CudaStages(0, dnrm2_ptr=None), CudaStages(0, dnrm2_ptr=_lib.scipy_dnrm2_pointer())):
        for r0, r1 in ((0, M), (0, 2), (2, M)):
            rows = st.empty((r1 - r0, 1), torch.int32)
            cnt = st.empty((r1 - r0,), torch.int32)
            n = st.neighbours(tc, M, D, r0, r1, E, E ** 2, rows, cnt)
            got = np.unpackbits(rows.cpu().numpy().view(np.uint8), axis=1, bitorder="little")[:, :M]
            assert n >= 1, (st.dnrm2_ptr, r0, r1)
            assert (got == nbr[r0:r1]).all(), (st.dnrm2_ptr, r0, r1, got)
            assert (cnt.cpu().numpy() == nbr[r0:r1].sum(axis=1)).all(), (st.dnrm2_ptr, r0, r1)


def _growth_graph(rng, M, D, ngroups, p_edge, p_iso):
    """A random symmetric weighted-neighbourhood graph with isolated MCs, noise, border MCs shared between clusters and
    core MCs whose pdim exceeds pi: (bit rows, core flags, subspace masks, CSR entries of the non-isolated rows)."""
    words = (M + 31) // 32
    grp = rng.integers(0, ngroups, size=M)
    grp[rng.random(M) < p_iso] = -1  # isolated
    A = np.zeros((M, M), bool)
    for g in range(ngroups):
        idx = np.flatnonzero(grp == g)
        sub = rng.random((len(idx), len(idx))) < p_edge
        A[np.ix_(idx, idx)] = sub | sub.T
    bridges = rng.integers(0, M, size=(40, 2))  # a few edges between groups (border MCs reachable from two clusters)
    bridges = bridges[(grp[bridges[:, 0]] >= 0) & (grp[bridges[:, 1]] >= 0)]
    A[bridges[:, 0], bridges[:, 1]] = A[bridges[:, 1], bridges[:, 0]] = True
    np.fill_diagonal(A, True)
    bits = np.zeros((M, words * 32), np.uint8)
    bits[:, :M] = A
    wn = np.packbits(bits.reshape(M, words, 32), axis=2, bitorder="little").view(np.uint32).reshape(M, words)
    core = (rng.random(M) < 0.6).astype(np.uint8)
    pd = rng.integers(0, D + 1, size=M)
    sub = np.array([sum(1 << int(d) for d in rng.choice(D, size=int(k), replace=False)) for k in pd], np.int64)
    deg = A.sum(axis=1)
    nnz = int(deg[deg > 1].sum())  # an isolated row (WN(p) = {p}) owns no CSR entry
    return wn, core, sub, nnz


def test_cluster_growth_formulations_agree():
    """Kernel 4e has two formulations (bit-row scan; isolated pre-pass + CSR + merge by seed rank), and the CSR one walks
    the graph in one of three ways by its size: one warp over a shared-memory copy (22 bytes per entry fit 200 KB), one
    warp over global memory (mean list length <= 16), the 1024-thread walk (longer lists).  On a random graph for each
    walk, the CSR formulation must give the bit-row scan's labels, claim order and offsets."""
    import torch
    from chronoclust_b200.offline_sharded import CudaStages

    rng = np.random.default_rng(11)
    D, pi = 12, 8
    st = CudaStages(0)
    for walk, M, ngroups, p_edge, p_iso in (("warp", 3000, 60, 0.08, 0.3), ("smem", 1500, 60, 0.08, 0.3),
                                            ("block", 2000, 20, 0.3, 0.1)):
        wn, core, sub, nnz = _growth_graph(rng, M, D, ngroups, p_edge, p_iso)
        regime = "block" if nnz > 16 * M else "smem" if nnz * 22 + 64 <= 200 * 1024 else "warp"
        assert regime == walk, f"test construction: {nnz} CSR entries over {M} rows reach the {regime} walk"
        twn = torch.from_numpy(wn.view(np.int32)).cuda()
        tcore, tsub = torch.from_numpy(core).cuda(), torch.from_numpy(sub).cuda()
        res = []
        for min_m in (10 ** 8, 1):
            lab, order, cl_off, ncl = st.clusters(M, twn, tcore, tsub, 4.0, pi, csr_min_m=min_m)
            res.append((lab.copy(), order[:cl_off[-1]].copy(), cl_off.copy(), ncl))
        (l0, o0, c0, n0), (l1, o1, c1, n1) = res
        assert n0 == n1, walk
        assert (c0 == c1).all() and (o0 == o1).all() and (l0 == l1).all(), walk
        sizes = np.diff(c0)
        if walk == "warp":
            assert n0 > 100
            assert (sizes > 1).sum() > 20 and (sizes == 0).sum() > 0 and (l0 < 0).sum() > 0  # the fixture exercises every case
        else:
            assert (sizes > 1).sum() > 0 and (l0 < 0).sum() > 0, walk


@pytest.mark.parametrize("D,Q,P,k", [(3, 7, 5, 4.0), (12, 300, 257, 4.0), (40, 130, 999, 16.0), (12, 64, 100, 3.0),
                                     (5, 33, 1, 1.0)])
def test_assoc_scan_bit_exact(D, Q, P, k):
    """SURVEY 8f-1: ccb_assoc_nearest against numpy's elementwise IEEE arithmetic (microcluster.py:167-181 ->
    mc_functions.py:35-43 with the QUERY's centroid / preference vector), summed over d in index order, first wins."""
    import torch
    from chronoclust_b200 import _lib

    rng = np.random.default_rng(D * 31 + Q + P)
    cur, prev = rng.random((Q, D)), rng.random((P, D))
    if P > 3:
        prev[P // 2] = prev[1]  # exact tie: the earlier previous MC must win
    prefbits = rng.random((Q, D)) < 0.5
    pref = np.where(prefbits, k, 1.0)
    masks = np.array([sum(1 << d for d in range(D) if prefbits[q, d] and k != 1.0) for q in range(Q)], np.uint64).view(np.int64)
    tc, tp, tm = torch.from_numpy(cur).cuda(), torch.from_numpy(prev).cuda(), torch.from_numpy(masks).cuda()
    best = torch.empty(Q, dtype=torch.int32, device="cuda")
    dist = torch.empty(Q, dtype=torch.float64, device="cuda")
    _lib.check(_lib.lib().ccb_assoc_nearest(0, None, tc.data_ptr(), tm.data_ptr(), Q, tp.data_ptr(), P, D, k,
                                            best.data_ptr(), dist.data_ptr()))
    torch.cuda.synchronize()
    acc = np.zeros((Q, P))
    for d in range(D):
        t = prev[None, :, d] - cur[:, d, None]
        acc = acc + (t * t) / pref[:, d, None]
    exp = acc.argmin(axis=1)
    assert (best.cpu().numpy() == exp).all()
    assert bits_equal(dist.cpu().numpy(), acc[np.arange(Q), exp])


def test_historical_association_device_scan_matches_host_loop():
    """The tracker (tracking/cluster_tracker.py:127-144) with the scan on the device gives the associations of the
    host loop, on clusters built from the C1 golden microclusters of two consecutive timepoints."""
    from chronoclust_b200.objects import Cluster, Microcluster
    from chronoclust_b200.tracking import TrackByHistoricalAssociation

    z = load("c1.npz")

    def clusters_at(t):
        P = f"t{t}_p_"
        mcs = {int(i): Microcluster(z[P + "cf1"][j], z[P + "cf2"][j], id=[int(i)], cumulative_weight=float(z[P + "w"][j]),
                                    preferred_dimension_vector=z[P + "pref"][j], cluster_centroids=z[P + "cen"][j])
               for j, i in enumerate(z[P + "ids"].tolist())}
        off, idl = z[f"t{t}_cl_off"], z[f"t{t}_cl_idlist"]
        out = []
        for c in range(len(off) - 1):
            cl = Cluster([int(i) for i in idl[off[c]:off[c + 1]]])
            cl.id = f"K{t}_{c}"
            cl.add_pcore_objects(mcs)
            out.append(cl)
        return out

    res = []
    for min_pairs in (None, 0):
        tr = TrackByHistoricalAssociation()
        tr.device_scan_min_pairs = min_pairs
        tr.previous_timepoint_clusters = clusters_at(1)
        cur = clusters_at(2)
        tr.set_current_clusters(cur)
        tr.track_cluster_history()
        res.append([(sorted(c.historical_associates), sorted(c.historical_associates_pcores)) for c in cur])
    assert res[0] == res[1] and any(a for a, _ in res[0])


def test_full_size_c2_invariants():
    """BASELINE config C2 at FULL size (1e6 cells x 12 markers, 2 timepoints) -- too big for the oracle in test time, so
    the check is through properties that do not depend on the size:
      * the engine's knobs never change results: the default run (32 768-cell blocks, CUDA graph) and a run with 6 000-cell
        blocks on plain stream launches give bit-identical assignments, lists, statistics and clusters;
      * conservation at t0 (nothing decays yet): every cell is absorbed exactly once, so the weights are integers that
        sum to N, each MC's weight is the number of cells assigned to it, and sum(CF1) over all MCs equals the column
        sums of X to 1e-9 relative (the summation ORDER differs, the set of addends does not);
      * every per-cell uid names a live microcluster; created + upgraded counters agree with the list lengths."""
    from chronoclust_b200.synth import CONFIGS, config_params, gen

    N, D, _, Cn, seed, _, _ = CONFIGS["C2"]
    cfg = config_params("C2")
    Xs = gen(N, D, 2, Cn, seed)
    a, b = make(cfg), make(cfg, chunk=6000, bsv_bmin=256, bsv_stream=1)
    for t, X in enumerate(Xs):
        a.online_microcluster_maintenance(X, t)
        b.online_microcluster_maintenance(X, t)
        assert (a.last_assignment == b.last_assignment).all() and (a.last_stage == b.last_stage).all()
        for which in (0, 1):
            ga, gb = a.export_arrays(which), b.export_arrays(which)
            assert (ga[0] == gb[0]).all() and (ga[1] == gb[1]).all()
            for x, y in zip(ga[2:], gb[2:]):
                assert bits_equal(x, y)
        ca, cb = clusters_of(a), clusters_of(b)
        assert len(ca) == len(cb)
        for (m1, w1, *r1), (m2, w2, *r2) in zip(ca, cb):
            assert list(m1) == list(m2) and w1 == w2 and all(bits_equal(p, q) for p, q in zip(r1, r2))
        if t == 0:
            ids_p, uid_p, w_p, cf1_p = a.export_arrays(0)[:4]
            ids_o, uid_o, w_o, cf1_o = a.export_arrays(1)[:4]
            w, uid = np.concatenate([w_p, w_o]), np.concatenate([uid_p, uid_o])
            assert (w == np.round(w)).all() and w.sum() == N
            counts = np.bincount(a.last_assignment, minlength=int(uid.max()) + 1)
            assert (counts[uid] == w).all() and counts.sum() == N
            col = np.concatenate([cf1_p, cf1_o]).sum(axis=0)
            assert np.allclose(col, X.sum(axis=0), rtol=1e-9, atol=0.0)
        live = np.zeros(int(max(a.last_assignment.max(), 0)) + 2, bool)
        live[np.concatenate([a.export_arrays(0)[1], a.export_arrays(1)[1]])] = True
        assert live[a.last_assignment].all()
    st = a.stats()
    assert st["points"] == 2 * N and st["bsv_blocks"] > 0


EDGE_CFG = {"beta": 0.2, "delta": 0.05, "epsilon": 0.05, "lambda": 2, "k": 4, "mu": 0.01, "pi": 0, "omicron": 0.00000435,
            "upsilon": 6.5}


def _edge_series(kind):
    rng = np.random.default_rng(7)
    blob = lambda n, d: np.clip(0.5 + 0.02 * rng.standard_normal((n, d)), 0.0, 1.0)
    if kind == "d1":
        return EDGE_CFG, [blob(500, 1) for _ in range(3)]
    if kind == "d64":  # the widest preference mask (64 bits)
        return dict(EDGE_CFG, epsilon=0.2), [blob(300, 64) for _ in range(3)]
    if kind == "single_cell":
        return EDGE_CFG, [blob(1, 3) for _ in range(3)]
    if kind == "empty_timepoint":
        return EDGE_CFG, [blob(400, 3), np.zeros((0, 3)), blob(400, 3)]
    if kind == "identical_cells":  # zero variance, every distance an exact tie
        return EDGE_CFG, [np.full((257, 5), 0.25), np.full((64, 5), 0.25), np.full((300, 5), 0.75)]
    if kind == "k1_default":  # reference default k = 1: every preference weight is 1, pdim is always 0
        return dict(EDGE_CFG, k=1, pi=2), [blob(600, 4) for _ in range(3)]
    if kind == "no_cluster":  # nothing ever reaches the pcore threshold (no_cluster_test.py of the reference)
        return dict(EDGE_CFG, beta=1.0, mu=0.9), [rng.random((500, 3)) for _ in range(3)]
    if kind == "two_far_blobs_gap":  # timestamps with a gap: decay by 2^(-lambda * 3)
        return EDGE_CFG, [np.vstack([blob(300, 2), blob(300, 2) * 0.2]) for _ in range(3)]
    raise KeyError(kind)


@pytest.mark.parametrize("kind", ["d1", "d64", "single_cell", "empty_timepoint", "identical_cells", "k1_default",
                                  "no_cluster", "two_far_blobs_gap"])
def test_edge_shapes_vs_oracle(kind):
    """Edge cases of the hot path against the (reference-pinned) oracle, bit for bit: one marker, 64 markers, a single
    cell, an empty timepoint, identical cells (exact ties), the default k = 1, a run in which no cluster ever forms,
    and non-consecutive timestamps."""
    from oracle.oracle import OracleHDDStream

    cfg, Xs = _edge_series(kind)
    stamps = [0, 3, 4] if kind == "two_far_blobs_gap" else list(range(len(Xs)))
    h, o = make(cfg), OracleHDDStream(cfg)
    for t, X in zip(stamps, Xs):
        X = np.ascontiguousarray(X, np.float64)
        h.online_microcluster_maintenance(X, t)
        o.online_microcluster_maintenance(X, t)
        if len(X):
            assert (h.last_assignment == o.assign_uid).all() and (h.last_stage == o.stage).all()
        for which in (0, 1):
            e, got = o.export(which), h.export_arrays(which)
            assert len(got[0]) == len(e.ids) and (got[0] == e.ids).all() and (got[1] == e.uids).all()
            for g, x in zip(got[2:], (e.w, e.cf1, e.cf2, e.cen, e.pref)):
                assert bits_equal(g, x)
        oc, hc = o.clusters(), clusters_of(h)
        assert len(oc) == len(hc)
        for (m1, w1, *r1), (m2, w2, *r2) in zip(hc, oc):
            assert list(m1) == list(m2) and w1 == w2 and all(bits_equal(p, q) for p, q in zip(r1, r2))
    if kind == "no_cluster":
        assert len(h.final_clusters) == 0


def test_device_scaler_matches_sklearn():
    """SURVEY 8f-3.  (1) ccb_colminmax = np.nanmin / np.nanmax per column (what MinMaxScaler.partial_fit computes),
    negative values, NaNs and a strided layout included.  (2) Feeding RAW rows with a fitted sklearn MinMaxScaler
    (ccb_ingest_scaled: x * scale_ + min_ on the device, two roundings) gives bit for bit what scaling on the host first
    gives -- assignments, both lists, clusters, and the per-MC `points` coordinates."""
    import torch
    from sklearn.preprocessing import MinMaxScaler
    from chronoclust_b200 import _lib
    from chronoclust_b200.synth import gen

    rng = np.random.default_rng(3)
    N, D, ld = 70001, 7, 9
    buf = rng.normal(0.0, 50.0, size=(N, ld))
    buf[rng.random((N, ld)) < 0.001] = np.nan
    buf[:, 3] = 12.5  # constant column
    t = torch.from_numpy(buf).cuda()
    mn = torch.empty(D, dtype=torch.float64, device="cuda")
    mx = torch.empty(D, dtype=torch.float64, device="cuda")
    _lib.check(_lib.lib().ccb_colminmax(0, None, t.data_ptr(), N, ld, D, mn.data_ptr(), mx.data_ptr()))
    torch.cuda.synchronize()
    assert bits_equal(mn.cpu().numpy(), np.nanmin(buf[:, :D], axis=0))
    assert bits_equal(mx.cpu().numpy(), np.nanmax(buf[:, :D], axis=0))

    cfg = {"beta": 0.2, "delta": 0.05, "epsilon": 0.05, "lambda": 2, "k": 4, "mu": 0.01, "pi": 0, "omicron": 0.00000435,
           "upsilon": 6.5}
    raw = [x * np.array([3.0, 250.0, 0.01, 17.0, 1e4, 2.0]) - np.array([1.0, 100.0, 0.0, -4.0, 5e3, 0.5])
           for x in gen(300001, 6, 2, 6, 5)]  # >= 2 x 131 072 rows: the segmented copy path scales segment by segment
    sk = MinMaxScaler().fit(np.concatenate(raw, axis=0))
    a, b = make(cfg), make(cfg)
    for ts, X in enumerate(raw):
        a.online_microcluster_maintenance(sk.transform(X), ts)
        b.online_microcluster_maintenance(X, ts, scaler=sk)
        assert (a.last_assignment == b.last_assignment).all() and (a.last_stage == b.last_stage).all()
        for which in (0, 1):
            ga, gb = a.export_arrays(which), b.export_arrays(which)
            assert (ga[0] == gb[0]).all() and all(bits_equal(x, y) for x, y in zip(ga[2:], gb[2:]))
        ca, cb = clusters_of(a), clusters_of(b)
        assert len(ca) == len(cb) and all(list(m1) == list(m2) and w1 == w2 for (m1, w1, *_), (m2, w2, *_) in zip(ca, cb))
        pa, pb = a.pcore_MC[0].points, b.pcore_MC[0].points
        assert list(pa.keys()) == list(pb.keys()) and pa[next(iter(pa))] == pb[next(iter(pb))]


# ---- BASELINE sizes against the oracle (VERDICT r1: the benched configuration itself must be compared) -------------
def _assert_same_as_oracle(h, o, what):
    assert (h.last_assignment == o.assign_uid).all(), \
        f"{what}: {(h.last_assignment != o.assign_uid).sum()} assignments differ, first at " \
        f"{np.flatnonzero(h.last_assignment != o.assign_uid)[:5]}"
    assert (h.last_stage == o.stage).all(), f"{what}: per-cell stage differs"
    for which in (0, 1):
        e, got = o.export(which), h.export_arrays(which)
        assert len(got[0]) == len(e), f"{what}: list {which} has {len(got[0])} MCs, oracle {len(e)}"
        assert (got[0] == e.ids).all() and (got[1] == e.uids).all(), f"{what}: list {which} ids / order differ"
        for n, g, x in zip(("w", "cf1", "cf2", "cen", "pref"), got[2:], (e.w, e.cf1, e.cf2, e.cen, e.pref)):
            assert bits_equal(g, x), f"{what}: list {which} {n} not bit-identical"
    assert tuple(h.counts()[2:]) == tuple(o.counters), f"{what}: id counters differ"
    oc, hc = o.clusters(), clusters_of(h)
    assert len(oc) == len(hc), f"{what}: {len(hc)} clusters, oracle {len(oc)}"
    for c, ((m1, w1, *r1), (m2, w2, *r2)) in enumerate(zip(hc, oc)):
        assert list(m1) == list(m2) and w1 == w2, f"{what}: cluster {c} members / weight differ"
        assert all(bits_equal(p, q) for p, q in zip(r1, r2)), f"{what}: cluster {c} statistics not bit-identical"


@pytest.mark.parametrize("cfgname,T,scale,over", [
    ("C2", 5, 1.0, {}),                 # BASELINE configs[1] at full size: 1e6 cells x 12 markers x 5 timepoints
    ("C3", 2, 1.0, {}),                 # BASELINE configs[2] at full N: 2e6 cells x 40 markers (2 timepoints: oracle ~30 s)
    ("C2", 2, 0.5, {"epsilon": 0.04}),  # BASELINE configs[4] corner: the saturated regime (round / capacity cuts); the
                                        # oracle needs 45 s for ONE full timepoint there, hence 5e5 cells x 2
    ("C2", 2, 1.0, {"epsilon": 0.045, "upsilon": 4, "beta": 0.8}),  # another grid corner: late upgrades, long cold start
], ids=["C2-full", "C3-fullN-2tp", "C5-eps0.04", "C5-beta0.8"])
def test_baseline_sizes_vs_oracle(cfgname, T, scale, over):
    """The CUDA path against the (reference-pinned) oracle at BASELINE.json's own sizes, bit for bit after every
    timepoint: per-cell assignment and stage, both lists (order, ids, W / CF1 / CF2 / centroid / preference vector), id
    counters, every cluster (claim order, sums).  These sizes reach what the fixtures cannot: 20-35 k outlier MCs,
    kernel 1 over > 32 slabs, store growth inside the graph loop, need-list growth relaunches, capacity / round cuts."""
    from chronoclust_b200.synth import CONFIGS, config_params, gen
    from oracle.oracle import OracleHDDStream

    N, D, _, Cn, seed, _, _ = CONFIGS[cfgname]
    N = int(N * scale)
    cfg = dict(config_params(cfgname), **over)
    Xs = gen(N, D, T, Cn, seed)
    h, o = make(cfg), OracleHDDStream(cfg)
    for t, X in enumerate(Xs):
        h.online_microcluster_maintenance(X, t)
        o.online_microcluster_maintenance(X, t)
        _assert_same_as_oracle(h, o, f"{cfgname}{over} t{t}")
    st = h.stats()
    print(cfgname, over, {k: v for k, v in st.items() if v})
    assert st["points"] == N * T


def test_offline_c4_shape_vs_oracle():
    """The offline phase at M = 8192 potential microclusters x 40 markers from the C4 generator (SURVEY 8d) against the
    oracle's PreDeCon restatement: column slabs of kernel 4b, the guard band on real data, CSR growth with thousands of
    clusters, claim order and merged sums -- through ccb_offline, i.e. what HDDStream.offline_clustering calls."""
    from chronoclust_b200 import _lib
    from chronoclust_b200.synth import gen_offline_stress
    from oracle.oracle import OracleHDDStream, _p
    from oracle.oracle import lib as olib

    M, D = 8192, 40
    cen, w, _core = gen_offline_stress(M, D)
    rng = np.random.default_rng(11)
    cf1 = cen * w[:, None]
    cf2 = (cen * cen + rng.uniform(1e-5, 4e-3, size=(M, D))) * w[:, None]  # variances on both sides of delta^2
    ids = np.arange(M, dtype=np.int64)
    cfg = {"beta": 0.0, "delta": 0.05, "epsilon": 1e150, "lambda": 0, "k": 4.0, "mu": 0.0, "pi": D, "omicron": 0.0,
           "upsilon": 0.3 / 1e150}
    mu = 20.0
    o = OracleHDDStream(cfg)
    o._ensure(D)
    L = olib()
    for i in range(M):
        L.cco_import_mc(o._h, 0, int(ids[i]), int(ids[i]), float(w[i]), _p(np.ascontiguousarray(cf1[i])),
                        _p(np.ascontiguousarray(cf2[i])), _p(np.ascontiguousarray(cen[i])), _p(np.ones(D)))
    L.cco_set_thresholds(o._h, mu, 0.0, D)
    o.offline_clustering()
    oc = o.clusters()
    for csr in (0, 10 ** 8):  # CSR formulation (default at this M) and the bit-row scan
        h = make(cfg, off_csr_min_m=csr)
        assert h.upsilon == 0.3
        h.dataset_dimensionality = D
        h._ensure_handle(D)
        h.pi, h.mu, h.omicron = D, mu, 0.0
        _lib.check(_lib.lib().ccb_begin_timepoint(h._h, mu, 0.0, D, 0, 1.0), h._h)
        h.import_arrays(0, ids, ids, w, cf1, cf2, cen, np.ones((M, D)))
        h.offline_clustering(0)
        hc = clusters_of(h)
        assert len(hc) == len(oc) and len(hc) > 1000
        for c, ((m1, w1, *r1), (m2, w2, *r2)) in enumerate(zip(hc, oc)):
            assert list(m1) == list(m2) and w1 == w2, f"cluster {c} (csr_min_m={csr})"
            assert all(bits_equal(p, q) for p, q in zip(r1, r2)), f"cluster {c} statistics (csr_min_m={csr})"
    assert max(len(m) for m, *_ in oc) > 1


def test_colminmax_covers_every_element():
    """ADVICE r1: with D = 12 / D = 40 and N * D far above the grid size, every flat index must be visited -- the extreme
    values are planted exactly where a stride rounded UP to a multiple of D would skip (indices [threads, stride))."""
    import torch
    from chronoclust_b200 import _lib

    threads = 148 * 8 * 256
    for D, N in ((12, 200_003), (40, 100_001), (7, 70_001)):
        X = np.random.default_rng(D).uniform(-1.0, 1.0, size=(N, D))
        up = (threads + D - 1) // D * D
        for w in range(3):  # a few stride windows
            for e in range(threads + w * up, min(up + w * up, N * D)):
                X[e // D, e % D] = 5.0 + e if (e % 2) else -5.0 - e
        t = torch.from_numpy(X).cuda()
        mn = torch.empty(D, dtype=torch.float64, device="cuda")
        mx = torch.empty(D, dtype=torch.float64, device="cuda")
        _lib.check(_lib.lib().ccb_colminmax(0, None, t.data_ptr(), N, D, D, mn.data_ptr(), mx.data_ptr()))
        torch.cuda.synchronize()
        assert bits_equal(mn.cpu().numpy(), X.min(axis=0)) and bits_equal(mx.cpu().numpy(), X.max(axis=0)), f"D={D}"


def _nccl_offline_worker(rank, world, port, M, ret):
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(f"cuda:{rank}"))
    try:
        from chronoclust_b200 import _lib
        from chronoclust_b200.offline_sharded import CudaStages, sharded_offline
        from chronoclust_b200.synth import gen_offline_stress

        D, E = 40, 0.3
        cen, w, core = gen_offline_stress(M, D)
        tc = torch.from_numpy(cen).cuda(rank)
        tcore = torch.from_numpy(core.astype(np.uint8)).cuda(rank)
        st = CudaStages(rank, dnrm2_ptr=_lib.scipy_dnrm2_pointer())
        out = {}
        for name, stages in (("csr", st), ("bitrows", _WithoutCsr(st))):
            lab, order, cl_off, ncl, info = sharded_offline(stages, tc, tcore, M, D, 4.0, D, 0.05, E, E ** 2, dist=dist)
            out[name] = (lab.copy(), order[:cl_off[-1]].copy(), cl_off.copy(), int(ncl), info["exchange"], info["gather_bytes"])
        l1, o1, c1, n1, _ = sharded_offline(st, tc, tcore, M, D, 4.0, D, 0.05, E, E ** 2, dist=None)  # this rank alone
        ok = True
        for name, (lab, order, cl_off, ncl, exch, nbytes) in out.items():
            ok = ok and exch == name and ncl == n1 and (lab == l1).all() and (cl_off == c1).all() and (order == o1[:c1[-1]]).all()
        ret[rank] = (bool(ok), int(n1), out["csr"][5], out["bitrows"][5], l1.tolist() if rank == 0 else None,
                     o1[:c1[-1]].tolist() if rank == 0 else None, c1.tolist() if rank == 0 else None)
    finally:
        dist.destroy_process_group()


class _WithoutCsr:
    """A stage object without the CSR methods: sharded_offline then all-gathers the bit rows."""

    def __init__(self, st):
        self._st, self.torch = st, st.torch

    def __getattr__(self, name):
        if name in ("rowinfo", "fill", "clusters_csr"):
            raise AttributeError(name)
        return getattr(self._st, name)


def test_sharded_offline_nccl_matches_single_rank_and_oracle():
    """The row-sharded offline phase on 2 GPUs over NCCL -- both exchanges: per-rank CSR lists merged by an all-reduce, and
    the all-gather of the bit rows -- against (i) the same phase on one rank and (ii) the oracle's PreDeCon restatement:
    labels, claim order and cluster offsets identical.  Skipped on a box with fewer than 2 GPUs (run it with
    `gpurun --gpus 2`; the log of that run is committed under profiles/)."""
    import torch
    import torch.multiprocessing as mp

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from chronoclust_b200.synth import gen_offline_stress
    from oracle.oracle import OracleHDDStream, _p
    from oracle.oracle import lib as olib

    M, D = 6000, 40
    world = 2
    mgr = mp.get_context("spawn").Manager()
    ret = mgr.dict()
    mp.spawn(_nccl_offline_worker, args=(world, 29700 + os.getpid() % 200, M, ret), nprocs=world, join=True)
    assert all(ret[r][0] for r in range(world)), {r: ret[r][:4] for r in range(world)}
    assert ret[0][2] < ret[0][3], "the CSR exchange must move fewer bytes than the bit rows"
    # oracle: same microclusters (any CF consistent with the centroids; only centroids / weights / core flags matter here)
    cen, w, core = gen_offline_stress(M, D)
    cfg = {"beta": 0.0, "delta": 0.05, "epsilon": 1e150, "lambda": 0, "k": 4.0, "mu": 0.0, "pi": D, "omicron": 0.0,
           "upsilon": 0.3 / 1e150}
    o = OracleHDDStream(cfg)
    o._ensure(D)
    L = olib()
    cf1, cf2 = cen * w[:, None], (cen * cen) * w[:, None]  # zero variance: every MC passes the radius test of the core flag
    for i in range(M):
        L.cco_import_mc(o._h, 0, i, i, float(w[i]), _p(np.ascontiguousarray(cf1[i])), _p(np.ascontiguousarray(cf2[i])),
                        _p(np.ascontiguousarray(cen[i])), _p(np.ones(D)))
    L.cco_set_thresholds(o._h, 20.0, 0.0, D)  # core <=> W >= 20, the generator's flag
    o.offline_clustering()
    lab, order, cl_off = np.array(ret[0][4]), np.array(ret[0][5]), np.array(ret[0][6])
    members = [order[cl_off[c]:cl_off[c + 1]].tolist() for c in range(len(cl_off) - 1)]
    members = [m for m in members if m]  # (clusters without members have weight 0 and are dropped, predecon.py:83)
    oc = [list(m) for m, *_ in o.clusters()]
    assert members == oc, "2-GPU clusters differ from the oracle's"


def test_gating_scan_on_device_matches_reference_expression():
    """SURVEY 8f-4: the (clusters x gates) scan of app.closest_gates on the device (ccb_assoc_nearest2) gives the labels of
    the reference's own loop (find_closest_gating, app.py:497-512), with and without a scaler, including an exact tie
    between two gates (settled by the guard band + the reference expression: the first gate in dict order wins)."""
    from sklearn.preprocessing import MinMaxScaler

    from chronoclust_b200 import app
    from chronoclust_b200.scaling import Scaler
    from test_host_side import _gating_case

    for k in (4.0, 3.0, 1.0):
        gates, clusters = _gating_case(seed=int(k), Q=300, P=40, D=12, k=k)
        scan = app._device_gate_scan(np.array([c.centroid for c in clusters]),
                                     np.array([c.preferred_dimensions for c in clusters]),
                                     np.array([list(g) for g in gates]), k, 0)
        assert scan is not None and (scan[1] <= scan[2]).all()
        assert app.closest_gates(gates, clusters, None, k) == [app.find_closest_gating(gates, c, None) for c in clusters]
        sc = Scaler()
        sc.scaler = MinMaxScaler().fit(np.random.default_rng(1).random((50, 12)) * 7.0 - 2.0)
        assert app.closest_gates(gates, clusters, sc, k) == [app.find_closest_gating(gates, c, sc) for c in clusters]
