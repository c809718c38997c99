"""Timepoint-start maintenance -- kernel 3, k_maint_plan + k_maint_gather (csrc/online.cuh) -- against a plain model of the
reference's list loops and against the oracle.

Every timepoint after the first starts by decaying CF1, CF2 and W by f = 2^(-lambda dt), downgrading the pcore MCs with
W < beta*mu or pdim > pi (id <- prev_outlier_id, appended to the outlier list), deleting the outlier MCs with W <= omicron
and compacting both lists in order (hddstream.py:247-286, 516-549).  The reference removes inside `for mc in list` over the
list it mutates, so the element that follows a removed one is never examined.  Kernel 3 restates that sequential rule in
parallel: a thread-0 walk of the pcore list, and a two-state machine per chunk of ceil(total / 1024) outliers, chained
across the 1024 threads, with tombstones (W = -1) skipped.  Such code works on small lists and breaks at a chunk boundary
or a threshold tie, so the case grid places runs of removals on every chunk boundary and weights on both sides of both
thresholds, and covers underflowing factors and the growth of the outlier store inside ccb_begin_timepoint.

- CPU: reference_maintenance (the model) against the oracle's cco_begin_timepoint on the whole case grid, and the
  coverage of the long streams' construction.
- GPU: kernel 3 on the same lists against both, a follow-up ingest that reads the packed (centroid, weight) rows kernel 3
  rebuilt, and long irregular streams against the oracle after every timepoint, on both launch paths of the engine."""
import numpy as np
import pytest

from helpers import bits_equal

MAINT_THREADS = 1024  # threads of k_maint_plan: the outlier sequence is cut into chunks of ceil(total / 1024)
OUT_STORE0 = 8192  # entries of a new handle's outlier store


# ---- the model ----------------------------------------------------------------------------------------------------
class MC:
    __slots__ = ("id", "uid", "w", "cf1", "cf2", "cen", "pref")

    def __init__(self, id, uid, w, cf1, cf2, cen, pref):
        self.id, self.uid, self.w, self.cf1, self.cf2, self.cen, self.pref = id, uid, w, cf1, cf2, cen, pref


def reference_maintenance(pcore, outlier, f, beta_mu, omicron, pi):
    """hddstream.py:247-286 and 516-549 over Python lists of MC, in the reference's loop shape.  Mutates both lists and
    returns what it did: downgraded / deleted MCs, downgrades by weight only / pdim only / both, and the examined MCs that
    sit exactly on a threshold (W * f == beta*mu, W * f == omicron)."""
    for mc in pcore + outlier:  # one IEEE multiply each; centroid and preference vector untouched
        mc.w = mc.w * f
        mc.cf1 = mc.cf1 * f
        mc.cf2 = mc.cf2 * f
    n = dict(downgraded=0, deleted=0, weight=0, pdim=0, both=0, tie_beta_mu=0, tie_omicron=0)
    for mc in pcore:
        by_w = mc.w < beta_mu
        by_p = int((mc.pref > 1).sum()) > pi
        n["tie_beta_mu"] += mc.w == beta_mu
        if by_w or by_p:
            mc.id = mc.uid
            pcore.remove(mc)
            outlier.append(mc)
            n["downgraded"] += 1
            n["both" if by_w and by_p else "weight" if by_w else "pdim"] += 1
    # `del outlier[i]` is outlier.remove(mc) without its linear search: enumerate's count and the list iterator's index
    # advance together, so i is the position of mc in the list as it is now
    for i, mc in enumerate(outlier):
        n["tie_omicron"] += mc.w == omicron
        if mc.w <= omicron:
            del outlier[i]
            n["deleted"] += 1
    return n


def to_mcs(arrs):
    ids, uids, w, cf1, cf2, cen, pref = arrs
    return [MC(int(ids[j]), int(uids[j]), float(w[j]), cf1[j].copy(), cf2[j].copy(), cen[j].copy(), pref[j].copy())
            for j in range(len(ids))]


def from_mcs(mcs, D):
    if not mcs:
        return (np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0)) + tuple(np.zeros((0, D)) for _ in range(4))
    return (np.array([m.id for m in mcs], np.int64), np.array([m.uid for m in mcs], np.int64),
            np.array([m.w for m in mcs], np.float64)) + tuple(np.array([getattr(m, a) for m in mcs], np.float64)
                                                              for a in ("cf1", "cf2", "cen", "pref"))


def assert_lists_equal(got, exp, what):
    """(ids, uids, w, cf1, cf2, cen, pref) in list order, bit for bit."""
    assert len(got[0]) == len(exp[0]), f"{what}: {len(got[0])} MCs, expected {len(exp[0])}"
    assert (np.asarray(got[0]) == exp[0]).all(), f"{what}: ids / order differ, first at " \
        f"{np.flatnonzero(np.asarray(got[0]) != exp[0])[:5]}"
    assert (np.asarray(got[1]) == exp[1]).all(), f"{what}: uids differ"
    for name, g, e in zip(("w", "cf1", "cf2", "cen", "pref"), got[2:], exp[2:]):
        assert bits_equal(g, e), f"{what}: {name} not bit-identical"


# ---- the case grid ------------------------------------------------------------------------------------------------
LENGTHS = [0, 1, 2, 1023, 1024, 1025, 2047, 2048, 2049, 5000, 40000]
PATTERNS = ["none", "all", "alternating", "runs", "p0.1", "p0.5", "p0.9", "straddle"]
PCORES = ["empty", "single_kept", "single_down", "runs_weight", "pdim_only", "weight_pdim_both", "many",
          "down_and_deleted"]
SHAPES = [(D, k) for D in (1, 12, 33, 64) for k in (4.0, 3.0, 1.0)]
W_BM, W_OM = 40.0, 10.0  # weights that land exactly on beta*mu / omicron after the decay
BETA = 0.5


def _step(f, thr, up):
    """A weight whose product with f (> 0) is the double next to thr, above it (up) or below it."""
    t = np.nextafter(np.float64(thr), np.inf if up else -np.inf)
    w = t / np.float64(f)
    while not ((w * f > thr) if up else (w * f < thr)):
        w = np.nextafter(w, np.inf if up else 0.0)
    return float(w)


def _pattern(name, n, rng, total):
    """Which of n outliers are meant to be deletable (W * f <= omicron); total: length of the sequence kernel 3 cuts into
    chunks (the outliers and the downgraded pcore MCs behind them)."""
    if name == "none":
        return np.zeros(n, bool)
    if name == "all":
        return np.ones(n, bool)
    if name == "alternating":
        return np.arange(n) % 2 == 0
    if name == "runs":  # runs of 2..7 deletable MCs, 1..3 apart
        c, j = np.zeros(n, bool), 0
        while j < n:
            r = 2 + (j * 7 + 3) % 6
            c[j:j + r] = True
            j += r + 1 + j % 3
        return c
    if name.startswith("p"):
        return rng.random(n) < float(name[1:])
    if name == "straddle":  # runs starting at c*per - 1, c*per and c*per + 1 of every chunk boundary (2..4 long)
        c = np.zeros(n, bool)
        per = max(1, -(-total // MAINT_THREADS))
        for b in range(per, n, per):
            s = b + (b // per) % 3 - 1
            c[s:s + 2 + (b // per) % 3] = True
        return c
    raise KeyError(name)


class Case:
    """Two lists to be maintained, with the arguments of ccb_begin_timepoint / cco_begin_timepoint."""

    def __init__(self, D, k, f, P, O, beta_mu, omicron, pi):
        self.D, self.k, self.f, self.P, self.O, self.pi = D, k, f, P, O, pi
        self.beta_mu, self.omicron = beta_mu, omicron
        self.mu = beta_mu / BETA  # exact: BETA is a power of two, so BETA * mu == beta_mu
        assert BETA * self.mu == beta_mu
        self.counters = (int(P[0].max()) + 1 if len(P[0]) else 500000,
                         int(max([-1] + [int(a[1].max()) for a in (P, O) if len(a[1])])) + 1)

    def cfg(self):
        return {"beta": BETA, "delta": 0.05, "epsilon": 0.25, "lambda": 1, "k": self.k, "mu": 0.0, "pi": self.pi,
                "omicron": 0.0, "upsilon": 2.0}

    def model(self):
        P, O = to_mcs(self.P), to_mcs(self.O)
        n = reference_maintenance(P, O, self.f, self.beta_mu, self.omicron, self.pi)
        return from_mcs(P, self.D), from_mcs(O, self.D), n


def _rows(rng, D, k, w, pdim, uid0, ids=None, at=0.0):
    """MC rows in [at, at + 1]^D with sums that fit their centroid: CF1 = cen * W, CF2 = (cen^2 + 0.01 / D) * W."""
    n = len(w)
    w = np.asarray(w, np.float64)
    cen = at + rng.random((n, D))
    bits = np.zeros((n, D), bool)
    if k > 1.0:
        for j in range(n):
            bits[j, rng.permutation(D)[:pdim[j]]] = True
    uids = np.arange(uid0, uid0 + n, dtype=np.int64)
    return (uids if ids is None else ids, uids, w, cen * w[:, None], (cen * cen + 0.01 / D) * w[:, None], cen,
            np.where(bits, k, 1.0))


def _outlier_weights(cond, f, om, rng):
    """Deletable: 0 (live, not a tombstone), exactly on omicron, the next weight below it, or anything under it; kept: the
    next weight above omicron, or anything above it.  With f = 0 (omicron = 0) everything is deletable."""
    n = len(cond)
    w = np.empty(n)
    r = rng.integers(0, 4, n)
    top = W_OM if f > 0 else 50.0
    low = [0.0, top, _step(f, om, False) if f > 0 else 1.0]
    high = _step(f, om, True) if f > 0 else 0.0
    for j in range(n):
        if cond[j] or f == 0:
            w[j] = low[r[j]] if r[j] < 3 else rng.uniform(0.0, top)
        else:
            w[j] = high if r[j] < 2 else rng.uniform(W_OM, 3 * W_OM) + 1.0
    return w


def _pcore_spec(name, rng, D, k, pi, f, bm):
    """(weights, pdims) of a pcore list.  Kinds: K kept (exactly on beta*mu, or above), W downgraded by weight (the next
    weight below beta*mu, or anything between omicron and beta*mu), P downgraded by pdim only, B both, X downgraded by
    weight and deletable."""
    can_p = k > 1.0 and pi < D
    below = _step(f, bm, False) if f > 0 else 1.0
    kinds = {"empty": "", "single_kept": "K", "single_down": "W", "runs_weight": "KWWWWWKWWKWWWWWWWK",
             "pdim_only": "KPPKPKPPPK" if can_p else "KWWKWKWWWK", "weight_pdim_both": "KWPBBKPWWBK" if can_p else "KWWK",
             "down_and_deleted": "KXXXWXKXXWK",
             "many": "".join(rng.choice(list("KKKKWPBX" if can_p else "KKKKWWWX"), 3400))}[name]
    w, pd = [], []
    for c in kinds:
        if c == "K":
            w.append(W_BM if rng.random() < 0.5 else rng.uniform(W_BM, 4 * W_BM) + 1.0)
        elif c == "W":
            w.append(below if rng.random() < 0.5 else rng.uniform(W_OM + 1.0, W_BM - 1.0))
        elif c == "X":
            w.append(W_OM if rng.random() < 0.5 else rng.uniform(0.0, W_OM))
        else:  # P, B
            w.append(W_BM if c == "P" else rng.uniform(W_OM + 1.0, W_BM - 1.0))
        low_pd = c in "KWX"
        pd.append(int(rng.integers(0, pi + 1)) if low_pd or not can_p else int(rng.integers(pi + 1, D + 1)))
    if k == 1.0:
        pd = [0] * len(pd)
    return w, [min(p, D) for p in pd]


def make_case(n_out, pattern, pcores, D=12, k=4.0, f=0.5, seed=0, pi=None, om_tail=0):
    """f > 0: beta*mu = fl(W_BM * f) and omicron = fl(W_OM * f), so that the weights W_BM and W_OM land on them exactly;
    f == 0: beta*mu = 1 and omicron = 0, every decayed weight is 0.  om_tail: the last om_tail old outliers are
    deletable whatever the pattern (a run of deletions that goes on into the downgraded pcores)."""
    rng = np.random.default_rng([n_out, seed, D, int(k * 8)])
    pi = (D // 2) if pi is None else pi
    bm, om = (float(np.float64(W_BM) * f), float(np.float64(W_OM) * f)) if f > 0 else (1.0, 0.0)
    pw, pd = _pcore_spec(pcores, rng, D, k, pi, f, bm)
    moved, prev = 0, False  # the pcore pass, for the length of the outlier sequence
    for w, p in zip(pw, pd):
        prev = not prev and (w * f < bm or (k > 1.0 and p > pi))
        moved += prev
    cond = _pattern(pattern, n_out, rng, n_out + moved)
    if om_tail:
        cond[-om_tail:] = True
    ow = _outlier_weights(cond, f, om, rng)
    O = _rows(rng, D, k, ow, rng.integers(0, D + 1, n_out), 0)
    # pcore MCs far from every outlier (and from the cells of the follow-up ingests): those cells take the outlier stage
    P = _rows(rng, D, k, pw, pd, n_out + 7, ids=np.arange(900000, 900000 + len(pw), dtype=np.int64), at=10.0)
    return Case(D, k, f, P, O, bm, om, pi)


F_POW2, F_ODD = 0.5, 0.7071067811865476  # 2^-1 and 2^-0.5
GRID = ([("len", n, p, "runs_weight", 12, 4.0, F_POW2) for n in LENGTHS for p in PATTERNS]
        + [("pcore", n, "p0.5", pc, 12, 4.0, F_POW2) for n in (0, 1, 1025, 2049, 5000) for pc in PCORES]
        + [("tie", n, p, "weight_pdim_both", 12, 4.0, f) for n in (2, 1025, 5000) for p in ("p0.5", "straddle")
           for f in (F_POW2, F_ODD)]
        + [("underflow", n, "p0.5", pc, 12, 4.0, f) for n in (1, 2049) for pc in ("runs_weight", "many")
           for f in (0.0, 2.0 ** -1060, 7 * 5e-324)]
        + [("shape", 2049, "p0.5", "weight_pdim_both", D, k, F_POW2) for D, k in SHAPES])


def _cid(c):
    kind, n, p, pc, D, k, f = c
    return f"{kind}-n{n}-{p}-{pc}-D{D}-k{k:g}-f{f:.3g}"


def _case(c):
    kind, n, p, pc, D, k, f = c
    return make_case(n, p, pc, D=D, k=k, f=f, om_tail=5 if pc == "down_and_deleted" else 0)


# ---- the oracle ---------------------------------------------------------------------------------------------------
def oracle_of(case):
    from oracle.oracle import MCList, OracleHDDStream, lib

    o = OracleHDDStream(case.cfg())
    o._ensure(case.D)
    for which, arrs in ((0, case.P), (1, case.O)):
        o.import_list(which, MCList(*arrs))
    lib().cco_set_counters(o._h, *case.counters)
    return o


def oracle_maintain(case):
    from oracle.oracle import lib

    o = oracle_of(case)
    lib().cco_begin_timepoint(o._h, case.mu, case.omicron, case.pi, 1, case.f)
    return o, oracle_lists(o)


def oracle_lists(o):
    """Both lists of an OracleHDDStream as (ids, uids, w, cf1, cf2, cen, pref)."""
    return [(x.ids, x.uids, x.w, x.cf1, x.cf2, x.cen, x.pref) for x in (o.export(0), o.export(1))]


def _coverage_of_case(case, n):
    """What a case promises to reach, checked against the model's own counts."""
    nO, nP = len(case.O[0]), len(case.P[0])
    if nO + nP and case.f == 0.0:
        assert n["deleted"] > 0
    if nP > 2:
        assert n["downgraded"] > 0


@pytest.mark.parametrize("c", GRID, ids=_cid)
def test_model_matches_oracle(c):
    """The model against the oracle's cco_begin_timepoint: order, ids, uids and the bits of every field of both lists,
    and the numbers of downgraded and deleted MCs."""
    case = _case(c)
    P, O, n = case.model()
    _coverage_of_case(case, n)
    o, (oP, oO) = oracle_maintain(case)
    assert_lists_equal(oP, P, "pcore list")
    assert_lists_equal(oO, O, "outlier list")
    assert len(case.P[0]) - len(oP[0]) == n["downgraded"]
    assert len(case.O[0]) + n["downgraded"] - len(oO[0]) == n["deleted"]


def test_model_skip_next_and_ties():
    """Hand-worked lists: a removed MC hides its successor from the test, also across the two passes, and the thresholds
    are strict (< beta*mu) and inclusive (<= omicron)."""
    D, one = 2, np.ones(2)

    def mc(i, w, pdim=0):
        return MC(i, 100 + i, w, one * w, one * w, one, np.array([4.0] * pdim + [1.0] * (2 - pdim)))

    # pcore: 0 kept (tie), 1 down by weight, 2 skipped (down-worthy), 3 down by weight and pdim, 4 skipped, 5 kept
    P = [mc(0, 4.0), mc(1, 3.0), mc(2, 1.0), mc(3, 1.0, 2), mc(4, 1.0), mc(5, 9.0)]
    # outliers: 10 deleted (tie), 11 skipped (deletable), 12 kept, 13 deleted (W = 0); appended: 1 skipped, 3 deleted (tie)
    O = [mc(10, 1.0), mc(11, 0.5), mc(12, 3.0), mc(13, 0.0)]
    n = reference_maintenance(P, O, 0.5, 2.0, 0.5, 1)
    assert [m.id for m in P] == [0, 2, 4, 5]
    assert [(m.id, m.uid) for m in O] == [(11, 111), (12, 112), (101, 101)]
    assert n == dict(downgraded=2, deleted=3, weight=1, pdim=0, both=1, tie_beta_mu=1, tie_omicron=2)
    assert P[0].w == 2.0 and O[2].cf1.tolist() == [1.5, 1.5] and O[2].cen.tolist() == [1.0, 1.0]


# ---- kernel 3 on the device ---------------------------------------------------------------------------------------
def handle_of(case):
    from test_gpu_parity import make
    from chronoclust_b200 import _lib

    h = make(case.cfg())
    h.dataset_dimensionality = case.D
    h._ensure_handle(case.D)
    for which, arrs in ((0, case.P), (1, case.O)):
        h.import_arrays(which, *arrs)
    _lib.check(_lib.lib().ccb_set_counters(h._h, *case.counters), h._h)
    return h


def device_maintain(case):
    from chronoclust_b200 import _lib

    h = handle_of(case)
    st0 = h.stats()
    _lib.check(_lib.lib().ccb_begin_timepoint(h._h, case.mu, case.omicron, case.pi, 1, case.f), h._h)
    st1 = h.stats()
    return h, {k: st1[k] - st0[k] for k in ("downgraded", "deleted")}


def _follow_up(h, o, case, O_after, seed):
    """An ingest behind the maintenance, at the same stamp (no second maintenance): cells on and on both sides of the
    centroids of the outlier list (surviving and downgraded MCs), and cells in between.  The pcore MCs lie far away, so
    every cell goes through kernel 1 over the packed (centroid, weight) rows kernel 3 rebuilt, which no export shows."""
    from test_gpu_parity import _assert_same_as_oracle

    rng = np.random.default_rng(seed)
    cen = O_after[5] if len(O_after[5]) else rng.random((4, case.D))
    sel = cen[rng.integers(0, len(cen), 600)]
    off = 0.02 * rng.standard_normal(sel.shape)
    X = np.ascontiguousarray(np.vstack([sel[:100], sel[100:350] + off[100:350], sel[350:] - off[350:],
                                        rng.random((200, case.D))]), np.float64)
    for s in (h, o):
        s.dataset_size, s.last_data_timestamp = 4096, 9
        s.config = dict(s.config, mu=1.0, omicron=2.0 ** -12)  # beta*mu = 400: no upgrade moves an outlier MC
        s.online_microcluster_maintenance(X, 9)
    _assert_same_as_oracle(h, o, "ingest behind the maintenance")
    assert (o.stage == 1).sum() > 100, "the cells must be absorbed by outlier MCs"


@pytest.mark.gpu
@pytest.mark.parametrize("c", GRID, ids=_cid)
def test_kernel3_matches_model_and_oracle(c):
    """ccb_begin_timepoint on imported lists against the model and the oracle, bit for bit, with the downgrade and
    deletion counters; for the shape cases, an ingest behind it against the oracle."""
    case = _case(c)
    P, O, n = case.model()
    h, cnt = device_maintain(case)
    o, (oP, oO) = oracle_maintain(case)
    for which, exp, oexp, name in ((0, P, oP, "pcore list"), (1, O, oO, "outlier list")):
        got = h.export_arrays(which)
        assert_lists_equal(got, oexp, f"{name} vs the oracle")
        assert_lists_equal(got, exp, f"{name} vs the model")
    assert cnt == {"downgraded": n["downgraded"], "deleted": n["deleted"]}
    assert h.counts()[2:] == list(case.counters)
    if c[0] == "pcore" and c[3] == "many" and c[1] == 5000:
        assert len(case.O[0]) + len(case.P[0]) > OUT_STORE0, "the outlier store must grow inside ccb_begin_timepoint"
    if c[0] == "shape":
        _follow_up(h, o, case, O, seed=c[4] * 10 + int(c[5]))


@pytest.mark.gpu
def test_kernel3_tombstones_and_repeated_maintenance():
    """Three maintenances in a row on one handle, each behind two ingests at one stamp: the upgrades of the first ingest
    leave tombstones (W = -1) that the second one and kernel 3 run over (the state machine skips them without resetting),
    and the ping-pong stores flip every time."""
    from oracle.oracle import lib as olib
    from chronoclust_b200 import _lib
    from test_gpu_parity import _assert_same_as_oracle

    case = make_case(2049, "p0.5", "runs_weight", seed=3, pi=12)  # pi = D: absorbing MCs can be upgraded
    h, o = handle_of(case), oracle_of(case)
    rng = np.random.default_rng(5)
    X = np.ascontiguousarray(case.O[5][rng.integers(0, 2049, 3000)] + 0.01 * rng.standard_normal((3000, case.D)))
    mu, om = 2.0 ** -9 * 1500, 2.0 ** -12 * 1500
    deleted = 0
    for t, f in ((1, 0.5), (2, F_ODD), (3, 0.5)):
        for part in (X[:1500], X[1500:]):
            for s in (h, o):
                s.config = dict(s.config, mu=2.0 ** -9, omicron=2.0 ** -12)
                s.dataset_size, s.last_data_timestamp = 1500, t
                s.online_microcluster_maintenance(part, t)
            _assert_same_as_oracle(h, o, f"t{t}")
        pre = [to_mcs(x) for x in oracle_lists(o)]
        n = reference_maintenance(*pre, f, BETA * mu, om, case.pi)
        st0 = h.stats()
        _lib.check(_lib.lib().ccb_begin_timepoint(h._h, mu, om, case.pi, 1, f), h._h)
        olib().cco_begin_timepoint(o._h, mu, om, case.pi, 1, f)
        st1 = h.stats()
        assert (st1["downgraded"] - st0["downgraded"], st1["deleted"] - st0["deleted"]) == (n["downgraded"], n["deleted"])
        deleted += n["deleted"]
        for which, (oe, me) in enumerate(zip(oracle_lists(o), pre)):
            assert_lists_equal(h.export_arrays(which), oe, f"t{t} list {which} vs the oracle")
            assert_lists_equal(h.export_arrays(which), from_mcs(me, case.D), f"t{t} list {which} vs the model")
    assert h.stats()["upgrades"] > 0 and deleted > 0


# ---- long irregular streams ---------------------------------------------------------------------------------------
STREAM_D, STREAM_PI = 6, 3


def stream_series(lam, k, seed=11):
    """An irregular stream of 24 timepoints: (stamps, rows, config pi per timepoint).  Populations appear, drift and
    vanish; noise cells make outliers that are deleted; two stamps repeat (no maintenance, tombstones carried into the
    next ingest); pi drops to 1 at two timepoints, which downgrades the pcore MCs with 2-3 preferred dimensions (with a
    constant pi no pcore MC ever holds more than pi); one long gap (f = 0 for lambda > 0) is followed by a run of
    single-cell timepoints a long interval apart -- every maintenance keeps the MC after a removed one, so a list of n
    needs about log2(n) of them to run empty -- and then the stream is seeded again.  Outside that run N is a multiple of
    1024, so that mu = N / 256 and omicron = N_prev / 2048 are whole or half numbers: with lambda = 0 the weights are
    integers and tie with beta*mu and omicron."""
    rng = np.random.default_rng([seed, int(lam * 10), int(k)])
    D = STREAM_D
    tight = [rng.permutation(D)[:t] for t in (2, 3, 2, 1, 3, 2)]
    centre = rng.uniform(0.25, 0.75, (6, D))
    drift = rng.normal(0.0, 0.02, (6, D))
    alive = [range(0, 7), [*range(2, 10), 21, 22, 23], range(4, 10), range(0, 3), range(21, 24), range(6, 10)]

    def cells(t, n):
        parts = [rng.random((n // 3, D))]  # noise
        live = [p for p in range(6) if t in alive[p]]
        for p in live:
            sd = np.full(D, 0.06)
            sd[tight[p]] = 0.004
            m = (n - n // 3) // len(live) if live else 0
            parts.append(np.clip(centre[p] + drift[p] * t + sd * rng.standard_normal((m, D)), 0.0, 1.0))
        X = np.vstack(parts)
        return X[rng.permutation(len(X))][:n] if len(X) >= n else np.vstack([X, rng.random((n - len(X), D))])

    stamps = [0, 1, 2, 2, 3, 5, 6, 6, 8, 9] + [9 + 2400 * i for i in range(1, 12)] + [9 + 2400 * 11 + d for d in (1, 2, 3)]
    sizes = [2048, 3072, 2048, 1024, 4096, 3072, 2048, 1024, 3072, 2048] + [1] * 11 + [2048, 3072, 2048]
    pis = [STREAM_PI] * len(stamps)
    pis[5] = pis[9] = 1
    Xs = [np.ascontiguousarray(cells(i, n)) for i, n in enumerate(sizes)]
    return stamps, Xs, pis


def stream_cfg(lam, k):
    return {"beta": 0.5, "delta": 0.05, "epsilon": 0.15, "lambda": lam, "k": k, "mu": 2.0 ** -8, "pi": STREAM_PI,
            "omicron": 2.0 ** -11, "upsilon": 2.0}


STREAMS = [(lam, k) for lam in (0.0, 0.5, 2.0) for k in (4.0, 3.0)]


def run_stream(lam, k, handles=()):
    """Feeds the stream to the oracle (and to `handles`), runs the model on every maintenance over the oracle's lists
    before it, and compares each handle with the oracle after every timepoint and its counters with the model's.
    Returns the coverage the stream reached."""
    from oracle.oracle import OracleHDDStream
    from test_gpu_parity import _assert_same_as_oracle

    stamps, Xs, pis = stream_series(lam, k)
    cfg = stream_cfg(lam, k)
    o = OracleHDDStream(cfg)
    cov = dict(downgraded=0, deleted=0, weight=0, pdim=0, both=0, tie_beta_mu=0, tie_omicron=0, emptied=0, repeated=0,
               chunked=0)
    for i, (t, X, pi) in enumerate(zip(stamps, Xs, pis)):
        for s in (o,) + tuple(handles):
            s.config = dict(cfg, pi=pi)
        decay = t != o.last_data_timestamp
        f = 2 ** (-o.lambbda * (t - o.last_data_timestamp)) if decay else 1.0
        pre = [to_mcs(x) for x in oracle_lists(o)] if decay else None
        st0 = [hh.stats() if decay else None for hh in handles]
        o.online_microcluster_maintenance(X, t)
        if i > 0 and not decay:
            cov["repeated"] += 1
        if decay:
            cov["chunked"] += len(pre[1]) + len(pre[0]) > MAINT_THREADS
            n = reference_maintenance(pre[0], pre[1], f, o.beta * o.mu, o.omicron, o.pi)
            for key in n:
                cov[key] += n[key]
            cov["emptied"] += not pre[0] and not pre[1]
        for hh, s0 in zip(handles, st0):
            hh.online_microcluster_maintenance(X, t)
            _assert_same_as_oracle(hh, o, f"lambda {lam} k {k} t{i} (stamp {t})")
            if decay:
                s1 = hh.stats()
                assert (s1["downgraded"] - s0["downgraded"], s1["deleted"] - s0["deleted"]) == \
                    (n["downgraded"], n["deleted"]), f"t{i}: kernel 3's counters differ from the model's"
    return cov


def _assert_stream_coverage(cov, lam):
    assert cov["deleted"] >= 1000 and cov["weight"] >= 50 and cov["pdim"] >= 3 and cov["both"] >= 10, cov
    assert cov["repeated"] == 2, cov
    if lam < 1:  # (lambda = 2 decays the lists below two entries per thread)
        assert cov["chunked"] >= 1, cov
    if lam > 0:
        assert cov["emptied"] >= 1, cov
    else:
        assert cov["tie_beta_mu"] >= 10 and cov["tie_omicron"] >= 10, cov


@pytest.mark.parametrize("lam,k", STREAMS)
def test_stream_construction_coverage(lam, k):
    """The streams reach what they are for -- deletions, downgrades by weight and by pdim, repeated stamps, lists run
    empty (lambda > 0), exact ties (lambda = 0) -- counted by the model over the oracle's lists."""
    _assert_stream_coverage(run_stream(lam, k), lam)


@pytest.mark.gpu
@pytest.mark.parametrize("lam,k", STREAMS)
def test_long_irregular_stream_vs_oracle(lam, k):
    """The streams on the default graph engine and on stream launches with short blocks, against the oracle after every
    timepoint (every maintenance flips the ping-pong stores the cached graphs bake in), and kernel 3's counters against
    the model at every maintenance."""
    from test_gpu_parity import make

    cfg = stream_cfg(lam, k)
    hs = (make(cfg), make(cfg, bsv_stream=1, chunk=300))
    _assert_stream_coverage(run_stream(lam, k, hs), lam)
