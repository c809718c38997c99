"""Every padded width the kernels are compiled for, against plain references.

Each hot-path kernel is instantiated once per padded width DP (csrc/api.cu: kDPs, round_dp), and much of its code depends
on DP at compile time: registers per lane of the replay record, the unsplit or split fast radius test, terms per lane,
which CONTESTED-group schedules exist, batch sizes, launch bounds, cells per thread and tile sizes of kernels 1 and 4b,
the straight-line or rolled sum of the exact radius test.  The rest of the GPU suite runs D = 1-7, 12, 40 and 64 only, so
here every class runs, at a width that fills it (D == DP) and at one that pads it (D < DP):

* the whole path (online + offline) against the oracle, bit for bit after every timepoint, in the regime where the
  ordered engine speculates, mismatches and replays;
* kernel 1, the association scans and the offline phase against numpy / the oracle, kernel by kernel;
* a strided device-resident ingest against a contiguous one;
* data far from the origin, where the fast radius test leaves the decision to the exact one.
"""
import ctypes as C
import logging
import os
import re

import numpy as np
import pytest

from helpers import bits_equal

LOG = logging.getLogger("test")
HERE = os.path.dirname(os.path.abspath(__file__))

# the whole path: every class above 12, filled and padded, and both sides of the NT = 2 boundary (DP 32 / 40)
WIDTHS = [13, 16, 17, 24, 29, 32, 33, 41, 48, 63]
# the kernel-level tests: every class, filled and padded
KERNEL_WIDTHS = [1, 3, 4, 7, 8, 11, 12] + WIDTHS + [40, 64]


def _kdps():
    src = open(os.path.join(HERE, "..", "chronoclust_b200", "csrc", "api.cu")).read()
    m = re.search(r"const int kDPs\[\] = \{([^}]*)\};", src)
    assert m, "kDPs not found in csrc/api.cu"
    return [int(v) for v in m.group(1).split(",")]


def _round_dp(D):
    return next(v for v in _kdps() if D <= v)


def test_width_lists_cover_every_class():
    """CPU guard: the width lists of this file keep up with the instantiations of csrc/api.cu."""
    dps = _kdps()
    assert max(KERNEL_WIDTHS) <= max(dps)
    for dp in dps:
        ds = [D for D in KERNEL_WIDTHS if _round_dp(D) == dp]
        assert dp in ds, f"no kernel test fills DP = {dp}"
        assert any(D < dp for D in ds), f"no kernel test pads DP = {dp}"
        if dp > 12:  # (the rest of the GPU suite runs the whole path at D <= 12 only)
            ws = [D for D in WIDTHS if _round_dp(D) == dp]
            assert any(D < dp for D in ws), f"no whole-path test pads DP = {dp}"
            assert dp in ws or dp in (40, 64), f"no whole-path test fills DP = {dp}"


def make(cfg, **kw):
    from chronoclust_b200.hddstream import HDDStream

    return HDDStream(dict(cfg), LOG, **kw)


def _cfg(D, c):
    """epsilon at c times the radius of a population of the generator (sigma = 0.025 per marker, r^2 ~ D sigma^2 / k)"""
    return {"beta": 0.2, "delta": 0.05, "epsilon": c * 0.025 * (D / 4) ** 0.5, "lambda": 2, "k": 4, "mu": 0.01, "pi": D,
            "omicron": 0.00000435, "upsilon": 6.5}


def _series(D, N=24000, T=3, shift=0.0):
    from chronoclust_b200.synth import gen

    return [np.ascontiguousarray(X + shift) for X in gen(N, D, T, 8, 4000 + D)]


def _same_state(a, b, what):
    """two handles: per-cell results, lists, counters and clusters bit-identical"""
    from test_gpu_parity import clusters_of

    assert (a.last_assignment == b.last_assignment).all() and (a.last_stage == b.last_stage).all(), what
    for which in (0, 1):
        ga, gb = a.export_arrays(which), b.export_arrays(which)
        assert len(ga[0]) == len(gb[0]) and (ga[0] == gb[0]).all() and (ga[1] == gb[1]).all(), what
        assert all(bits_equal(x, y) for x, y in zip(ga[2:], gb[2:])), what
    assert a.counts() == b.counts(), what
    ca, cb = clusters_of(a), clusters_of(b)
    assert len(ca) == len(cb), what
    for (m1, w1, *r1), (m2, w2, *r2) in zip(ca, cb):
        assert list(m1) == list(m2) and w1 == w2 and all(bits_equal(p, q) for p, q in zip(r1, r2)), what


def _run_vs_oracle(D, cfg, Xs, knobs=(dict(),)):
    from oracle.oracle import OracleHDDStream
    from test_gpu_parity import _assert_same_as_oracle

    hs, o = [make(cfg, **k) for k in knobs], OracleHDDStream(cfg)
    for t, X in enumerate(Xs):
        o.online_microcluster_maintenance(X, t)
        for h, k in zip(hs, knobs):
            h.online_microcluster_maintenance(X, t)
            _assert_same_as_oracle(h, o, f"D={D} {k} t{t}")
    return hs


# two settings of the engine's knobs (block length cap / smallest block / refinement rounds / stream launches) that must
# not change results
KNOBS = (dict(), dict(chunk=300, bsv_bmin=16, bsv_stream=1), dict(chunk=96, bsv_bmin=32, bsv_iters=1))


@pytest.mark.gpu
@pytest.mark.parametrize("c", [1.0, 1.3], ids=["saturated", "ordinary"])
@pytest.mark.parametrize("D", WIDTHS)
def test_whole_path_vs_oracle(D, c):
    """Online + offline phase against the oracle after every timepoint: per-cell assignment and stage, both lists in order
    with ids, W / CF1 / CF2 / centroid / preference bits, id counters, every cluster.  At DP 24 and 48 (saturated) the
    engine also runs with two other knob settings."""
    knobs = KNOBS if (D in (24, 48) and c == 1.0) else KNOBS[:1]
    hs = _run_vs_oracle(D, _cfg(D, c), _series(D), knobs)
    st = hs[0].stats()
    print(f"D={D} DP={_round_dp(D)} c={c}", {k: v for k, v in st.items() if v}, "clusters", len(hs[0].final_clusters))
    # the regime this width is here for: speculation that mismatched, cells decided by the outlier stage, upgrades,
    # kernel 1 at work, more than one cluster
    assert st["bsv_mismatches"] > 0 and st["bsv_outlier_stage_cells"] > 0, st
    assert st["upgrades"] > 0 and st["nearest_pairs"] > 0, st
    assert len(hs[0].final_clusters) >= 2


@pytest.mark.gpu
@pytest.mark.parametrize("D", [24, 40])
def test_far_from_origin_vs_oracle(D):
    """The same data shifted by 3 000 eps: the shape at the radius limit is unchanged, only the rounding of CF2 W - CF1^2
    grows.  The fast radius test of the pcore replay must then leave the close calls to the exact test (and
    k_bs_verify_p would catch a wrong one); either way the result is the oracle's, bit for bit."""
    cfg = _cfg(D, 1.0)
    hs = _run_vs_oracle(D, cfg, _series(D, shift=3000 * cfg["epsilon"]))
    st = hs[0].stats()
    print(f"D={D} shifted by 3000 eps:", {k: st[k] for k in ("bsv_rounds", "bsv_mismatches", "bsv_cuts_rounds")})


@pytest.mark.gpu
@pytest.mark.parametrize("D", [13, 24])
def test_strided_device_ingest(D):
    """HDDStream.ingest_device with X as a column slice of a wider device tensor (ld = D + 3) gives bit for bit what a
    contiguous copy gives.  An odd and an even width: the vectorised addend copy of k_bs_chain_o depends on the parity of
    D and ld."""
    import torch

    cfg = _cfg(D, 1.0)
    Xs = _series(D)
    N = Xs[0].shape[0]
    lds = (D, D + 3)
    hs = [make(cfg) for _ in lds]
    for h in hs:
        h.dataset_dimensionality = D
        h._ensure_handle(D)
    for t, X in enumerate(Xs):
        for h, ld in zip(hs, lds):
            buf = np.full((N, ld), np.nan)  # (the columns past D must never be read)
            buf[:, :D] = X
            tb = torch.from_numpy(buf).cuda()
            a = torch.empty(N, dtype=torch.int32, device="cuda")
            s = torch.empty(N, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            h.ingest_device(tb.data_ptr(), N, ld, t, a.data_ptr(), s.data_ptr())
            torch.cuda.synchronize()
            h.last_assignment, h.last_stage = a.cpu().numpy(), s.cpu().numpy()
        _same_state(hs[0], hs[1], f"D={D} ld={lds[1]} t{t}")
    st = hs[1].stats()
    print(f"D={D}", {k: v for k, v in st.items() if v})
    assert st["points"] == len(Xs) * N and st["bsv_outlier_stage_cells"] > 0 and len(hs[1].final_clusters) >= 2


def _masks(bits):
    return np.array([sum(1 << d for d in range(bits.shape[1]) if bits[j, d]) for j in range(bits.shape[0])],
                    np.uint64).view(np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("D", KERNEL_WIDTHS)
def test_kernel1_every_width(D):
    """Kernel 1 (ccb_nearest) against numpy's elementwise IEEE arithmetic, summed over d in index order, first minimum
    wins: k = 4 (the fused power-of-two weight step) with and without a band of subnormal squares (the unfused fallback),
    k = 3 (true division), exact ties between microclusters, M over several slabs and not a multiple of the tile, and X
    as a column slice of a wider device tensor (ld = D, D + 1, D + 3)."""
    import torch
    from chronoclust_b200 import _lib

    rng = np.random.default_rng(D * 101)
    N, M = 1500, 1337
    for k, tiny in ((4.0, 0.0), (4.0, 1e-160), (3.0, 0.0)):
        buf = rng.random((N, D + 3))
        cen = rng.random((M, D))
        if tiny:
            buf[::3] *= tiny
            cen[::2] *= tiny
            buf[5::7, :D:2] = 0.0
        cen[M // 2] = cen[0]  # exact ties between two microclusters: the earlier one must win
        cen[M - 1] = cen[7]
        buf[11, :D], buf[12, :D] = cen[0], cen[7]  # (cells at distance 0 from both of a pair)
        X = buf[:, :D]
        maskbits = rng.random((M, D)) < 0.6
        maskbits[M // 2] = maskbits[0]
        maskbits[M - 1] = maskbits[7]
        pref = np.where(maskbits, k, 1.0)
        acc = np.zeros((N, M))
        for d in range(D):
            t = X[:, d, None] - cen[None, :, d]
            acc = acc + (t * t) / pref[None, :, d]
        exp_slot = acc.argmin(axis=1)
        exp_dist = acc[np.arange(N), exp_slot]
        if tiny:
            assert ((acc > 0) & (acc < 2.3e-308)).any(), "the fixture must reach the subnormal range"
        assert exp_slot[11] == 0 and exp_slot[12] == 7, "the fixture must reach the ties"
        tc, tm = torch.from_numpy(cen).cuda(), torch.from_numpy(_masks(maskbits)).cuda()
        for ld in (D, D + 1, D + 3):
            tX = torch.from_numpy(np.ascontiguousarray(buf[:, :ld])).cuda()
            slot = torch.empty(N, dtype=torch.int32, device="cuda")
            dist = torch.empty(N, dtype=torch.float64, device="cuda")
            _lib.check(_lib.lib().ccb_nearest(0, None, tX.data_ptr(), N, ld, D, tc.data_ptr(), tm.data_ptr(), M, k,
                                              slot.data_ptr(), dist.data_ptr()))
            torch.cuda.synchronize()
            got = slot.cpu().numpy()
            assert (got == exp_slot).all(), f"k={k} tiny={tiny} ld={ld}: first differing cell {np.flatnonzero(got != exp_slot)[:5]}"
            assert bits_equal(dist.cpu().numpy(), exp_dist), f"k={k} tiny={tiny} ld={ld}: distances differ"


@pytest.mark.gpu
@pytest.mark.parametrize("D", KERNEL_WIDTHS)
def test_assoc_scans_every_width(D):
    """ccb_assoc_nearest and ccb_assoc_nearest2 against numpy (the QUERY's centroid and preference vector, summed over d in
    index order, first minimum wins), with exact ties, for k = 4 and k = 3 -- and the runner-up distance dist2 of
    ccb_assoc_nearest2: the smallest distance over every other previous microcluster."""
    import torch
    from chronoclust_b200 import _lib

    L = _lib.lib()
    rng = np.random.default_rng(D * 7 + 1)
    Q, P = 301, 517
    for k in (4.0, 3.0):
        cur, prev = rng.random((Q, D)), rng.random((P, D))
        prev[P // 2] = prev[1]  # exact tie: the earlier previous MC wins, and the runner-up equals the best
        cur[5] = prev[1]
        prefbits = rng.random((Q, D)) < 0.5
        pref = np.where(prefbits, k, 1.0)
        acc = np.zeros((Q, P))
        for d in range(D):
            t = prev[None, :, d] - cur[:, d, None]
            acc = acc + (t * t) / pref[:, d, None]
        exp = acc.argmin(axis=1)
        exp_d, exp_d2 = acc[np.arange(Q), exp], np.partition(acc, 1, axis=1)[:, 1]
        assert exp[5] == 1 and exp_d2[5] == exp_d[5] == 0.0
        tc, tp, tm = (torch.from_numpy(a).cuda() for a in (cur, prev, _masks(prefbits)))
        best = torch.empty(Q, dtype=torch.int32, device="cuda")
        dist = torch.empty(Q, dtype=torch.float64, device="cuda")
        dist2 = torch.empty(Q, dtype=torch.float64, device="cuda")
        _lib.check(L.ccb_assoc_nearest(0, None, tc.data_ptr(), tm.data_ptr(), Q, tp.data_ptr(), P, D, k, best.data_ptr(),
                                       dist.data_ptr()))
        torch.cuda.synchronize()
        assert (best.cpu().numpy() == exp).all() and bits_equal(dist.cpu().numpy(), exp_d), f"assoc k={k}"
        best.fill_(-7)
        dist.zero_()
        _lib.check(L.ccb_assoc_nearest2(0, None, tc.data_ptr(), tm.data_ptr(), Q, tp.data_ptr(), P, D, k, best.data_ptr(),
                                        dist.data_ptr(), dist2.data_ptr()))
        torch.cuda.synchronize()
        assert (best.cpu().numpy() == exp).all() and bits_equal(dist.cpu().numpy(), exp_d), f"assoc2 k={k}"
        assert bits_equal(dist2.cpu().numpy(), exp_d2), f"assoc2 k={k}: runner-up distances differ"


@pytest.mark.gpu
@pytest.mark.parametrize("D", KERNEL_WIDTHS)
def test_offline_every_width_vs_oracle(D):
    """The offline phase against the oracle's PreDeCon restatement: core flags, neighbour and weighted-neighbour matrices,
    subspace preference vectors and the clusters, bit for bit, with pairs planted exactly at distance E (a 3-4-5 triangle
    in two coordinates, every other coordinate equal) that the host settles with dnrm2.  Then the stateless stages
    (CudaStages.neighbours / subspace / weighted) over uneven row splits give the handle's rows."""
    import torch
    from chronoclust_b200 import _lib
    from chronoclust_b200.offline_sharded import CudaStages
    from chronoclust_b200.synth import gen_offline_stress
    from oracle.oracle import OracleHDDStream, _p
    from oracle.oracle import lib as olib
    from test_gpu_parity import clusters_of

    M = 1501
    s = max(1, round(0.3 * (D / 40) ** 0.5 * 64 / 5)) / 64  # E = 5 s: a neighbourhood radius of the generator's scale
    E = 5 * s
    cen, w, _core = gen_offline_stress(M, D, seed=D)
    cen = np.round(cen * 2.0 ** 30) / 2.0 ** 30  # (on a grid: c + 3 s and c + 4 s are exact, and so are the differences)
    if D >= 2:
        for a in range(0, 60, 6):  # planted pairs at distance exactly E
            b = a + 3 + 97 * a % (M - 70)
            cen[b] = cen[a]
            cen[b, 0] += 3 * s
            cen[b, 1] += 4 * s
    rng = np.random.default_rng(D)
    cf1 = cen * w[:, None]
    cf2 = (cen * cen + rng.uniform(1e-5, 4e-3, size=(M, D))) * w[:, None]  # variances on both sides of delta^2
    ids = np.arange(M, dtype=np.int64)
    cfg = {"beta": 0.0, "delta": 0.05, "epsilon": 2.0 ** 500, "lambda": 0, "k": 4.0, "mu": 0.0, "pi": D, "omicron": 0.0,
           "upsilon": E / 2.0 ** 500}  # (every MC passes the radius test of the core flag; upsilon * epsilon == E exactly)
    mu = 20.0
    o = OracleHDDStream(cfg)
    o._ensure(D)
    Lo = olib()
    for i in range(M):
        Lo.cco_import_mc(o._h, 0, int(ids[i]), int(ids[i]), float(w[i]), _p(np.ascontiguousarray(cf1[i])),
                         _p(np.ascontiguousarray(cf2[i])), _p(np.ascontiguousarray(cen[i])), _p(np.ones(D)))
    Lo.cco_set_thresholds(o._h, mu, 0.0, D)
    o.offline_clustering()
    h = make(cfg)
    assert h.upsilon == E, "test construction: upsilon * epsilon must reproduce E exactly"
    h.dataset_dimensionality = D
    h._ensure_handle(D)
    h.pi, h.mu, h.omicron = D, mu, 0.0
    _lib.check(_lib.lib().ccb_begin_timepoint(h._h, mu, 0.0, D, 0, 1.0), h._h)
    h.import_arrays(0, ids, ids, w, cf1, cf2, cen, np.ones((M, D)))
    h.offline_clustering(0)
    core, nbr, wn, subw = h.offline_intermediates()
    ocore, onbr, own, osubw = o.offline_intermediates()
    assert (core == ocore).all(), "core flags differ"
    assert (nbr == onbr).all(), f"neighbourhoods differ, first row {np.flatnonzero((nbr != onbr).any(axis=1))[:5]}"
    assert bits_equal(subw, osubw), "subspace preference vectors differ"
    assert (wn == own).all(), f"weighted neighbourhoods differ, first row {np.flatnonzero((wn != own).any(axis=1))[:5]}"
    hc, oc = clusters_of(h), o.clusters()
    assert len(hc) == len(oc)
    for c, ((m1, w1, *r1), (m2, w2, *r2)) in enumerate(zip(hc, oc)):
        assert list(m1) == list(m2) and w1 == w2 and all(bits_equal(p, q) for p, q in zip(r1, r2)), f"cluster {c}"
    st = h.stats()
    nb = int(nbr.sum()) - M
    print(f"D={D}: {nb} neighbour pairs, {st['borderline_pairs']} borderline, {int(core.sum())} core, {len(hc)} clusters")
    if D >= 2:
        assert st["borderline_pairs"] > 0
    assert 0 < nb < M * (M - 1) and len(hc) >= 2 and 0 < core.sum() < M

    # the stateless stages over uneven row splits (r0 odd) give the handle's rows
    stg = CudaStages(0, dnrm2_ptr=_lib.scipy_dnrm2_pointer())
    tc = torch.from_numpy(cen).cuda()
    words = (M + 31) // 32
    unpack = lambda r: np.unpackbits(r.cpu().numpy().view(np.uint8), axis=1, bitorder="little")[:, :M]
    splits = ((0, 37), (37, M))
    parts = []
    for r0, r1 in splits:
        rows = stg.empty((r1 - r0, words), torch.int32)
        cnt = stg.empty((r1 - r0,), torch.int32)
        sub = stg.empty((r1 - r0,), torch.int64)
        stg.neighbours(tc, M, D, r0, r1, E, E * E, rows, cnt)
        assert (unpack(rows) == nbr[r0:r1]).all(), f"rows [{r0}, {r1}): neighbour rows differ"
        assert (cnt.cpu().numpy() == nbr[r0:r1].sum(axis=1)).all()
        stg.subspace(tc, M, D, r0, r1, rows, cnt, h.delta, sub)
        parts.append((rows, sub))
    sub_all = torch.cat([p[1] for p in parts])
    exp_mask = _masks(subw == 4.0)
    assert (sub_all.cpu().numpy() == exp_mask).all(), "subspace masks differ"
    for (r0, r1), (rows, _) in zip(splits, parts):
        wrows = stg.empty((r1 - r0, words), torch.int32)
        stg.weighted(tc, M, D, r0, r1, rows, sub_all, 4.0, E * E, wrows)
        assert (unpack(wrows) == wn[r0:r1]).all(), f"rows [{r0}, {r1}): weighted neighbour rows differ"
