"""CPU suite: the CONTESTED-group logic of the pcore replay (csrc/engine.cuh: fast / exact radius test, two cells per step,
eight cells per pass along predicted verdicts), modelled operation by operation in tests/proto/chain_group_model.c, on
microclusters grown to their radius limit (the regime where these paths run):

* the division-free fast test never contradicts the reference's radius test (utilities/mc_functions.py:45-56) when it
  decides -- and it does decide nearly always, otherwise it would be no shortcut.  Both of its forms are modelled: one
  integer per term (padded width DP <= 16) and the split high / low integers (DP > 16);
* both group schedules (DP <= 12, one register per lane) leave the verdicts and the state of the one-by-one replay, bit for
  bit, whatever the predictions are (right, wrong, random): predictions steer the work, never the result.  At DP >= 16 the
  device takes the cells one by one, and so does the model.
"""
import ctypes as C
import os
import subprocess

import pytest

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "proto")
SRC, SO = os.path.join(HERE, "chain_group_model.c"), os.path.join(HERE, "libchaingroup.so")


def lib():
    if not os.path.exists(SO) or os.path.getmtime(SO) < os.path.getmtime(SRC):
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-o", SO, SRC, "-lm"])
    L = C.CDLL(SO)
    L.cgm_run.restype = C.c_longlong
    L.cgm_run.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                          C.c_double, C.c_int, C.c_int, C.c_double, C.POINTER(C.c_longlong)]
    L.cgm_boundary.restype = None
    L.cgm_boundary.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int,
                               C.POINTER(C.c_longlong)]
    return L


def run(seed, D=12, div_mode=0, k=4.0, eps=0.05, delta=0.05, W0=2000.0, centre=1.0, sigma=0.03, far=0.3, groups=400, pred=2,
        contested=0.9):
    out = (C.c_longlong * 8)()
    bad = lib().cgm_run(seed, D, div_mode, k, eps, delta, W0, centre, sigma, far, groups, pred, contested, out)
    keys = ("fast_decided", "fast_undecided", "fast_wrong", "passes", "groups", "contested", "rejected")
    return bad, dict(zip(keys, list(out)))


# (the spread sigma puts the MC at its radius limit: with every dimension preferred r^2 ~ D sigma^2 / k against eps^2)
CASES = [
    dict(sigma=0.0305, far=0.3),                                     # C2-like: D = 12, k = 4 (a power of two: multiply by 1/k)
    dict(div_mode=1, k=3.0, sigma=0.0262, far=0.3),                  # k not a power of two: the reference's division
    dict(D=4, sigma=0.052, W0=300.0, far=0.3),                       # few markers, a light MC (coarse integer units)
    dict(D=15, sigma=0.0268, W0=50000.0, groups=200, far=0.3),       # padded DP = 16 record (two registers a lane), a heavy MC
    dict(delta=0.018, sigma=0.0185, far=0.3),                        # variances straddle delta^2: mixed preference masks
    dict(centre=40.0, eps=0.5, delta=0.5, sigma=0.3, far=0.3),       # far from the origin (cancellation in CF2 W - CF1^2)
    dict(far=0.0, contested=1.0, sigma=0.03), dict(far=1.0, contested=1.0, sigma=0.02), dict(contested=0.5, far=0.6),
]


@pytest.mark.parametrize("pred", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("case", range(len(CASES)))
def test_group_schedules_reproduce_the_one_by_one_replay(case, pred):
    tot = {"fast_decided": 0, "fast_undecided": 0, "rejected": 0, "contested": 0, "passes": 0, "groups": 0}
    for seed in range(1, 7):
        bad, st = run(seed, pred=pred, **CASES[case])
        assert bad == 0, f"case {case} pred {pred} seed {seed}: {bad} groups differ from the one-by-one replay ({st})"
        assert st["fast_wrong"] == 0, f"case {case} seed {seed}: the fast test contradicted the exact test ({st})"
        for k in tot:
            tot[k] += st[k]
    # the regime is the intended one: both verdicts occur, and the fast test is a shortcut (it decides > 95 %)
    assert 0.03 * tot["contested"] < tot["rejected"] < 0.97 * tot["contested"]
    assert tot["fast_decided"] > 20 * max(tot["fast_undecided"], 1) or tot["fast_undecided"] == 0
    if pred == 3:  # right predictions: one pass per group (+ the exact first member, undecided cells)
        assert tot["passes"] <= 1.15 * tot["groups"] + 6


def _sigma(D, k=4.0, f=1.05):
    """the per-dimension spread that puts an MC with every dimension preferred at its radius limit (eps = 0.05)"""
    return round(0.05 * (k / D) ** 0.5 * f, 4)


# wider records: the unsplit test at the padded DP = 16, the split test at DP = 24 / 40 / 64 (NT = 1 and NT = 2 terms a lane)
WIDE_CASES = [dict(D=16, sigma=_sigma(16))]
for _D in (24, 40, 64):
    WIDE_CASES += [
        dict(D=_D, sigma=_sigma(_D)),                                              # k = 4
        dict(D=_D, div_mode=1, k=3.0, sigma=_sigma(_D, 3.0)),                      # k = 3: the reference's division
        dict(D=_D, W0=50000.0, groups=200, sigma=_sigma(_D, f=1.03)),              # a heavy MC
        dict(D=_D, delta=0.018, sigma=0.0185, eps=round(0.05 * (_D / 12) ** 0.5, 4)),  # variances straddle delta^2
    ]
for _D in (16, 24, 40, 64):  # far from the origin: cancellation in CF2 W - CF1^2 (centre = 1 000 eps and 3 000 eps)
    WIDE_CASES += [dict(D=_D, centre=1000 * 0.05, sigma=_sigma(_D)), dict(D=_D, centre=3000 * 0.05, sigma=_sigma(_D))]


@pytest.mark.parametrize("case", WIDE_CASES, ids=lambda c: "-".join(f"{a}{b}" for a, b in c.items()))
def test_wide_records_fast_test_is_decision_exact(case):
    tot = {"fast_decided": 0, "fast_undecided": 0, "rejected": 0, "contested": 0}
    for seed in range(1, 7):
        bad, st = run(seed, pred=3, **case)
        assert bad == 0, f"seed {seed}: {bad} groups differ from the one-by-one replay with the exact test ({st})"
        assert st["fast_wrong"] == 0, f"seed {seed}: the fast test contradicted the exact test ({st})"
        for k in tot:
            tot[k] += st[k]
    assert 0.03 * tot["contested"] < tot["rejected"] < 0.97 * tot["contested"]
    assert tot["fast_decided"] > 20 * max(tot["fast_undecided"], 1) or tot["fast_undecided"] == 0, tot


@pytest.mark.parametrize("centre_eps", [1, 1000, 3000, 10000])
@pytest.mark.parametrize("D", [12, 16, 24, 40, 64])
def test_fast_test_at_the_boundary(D, centre_eps):
    """The fast test where only the fp64 error of its terms decides: eps^2 within 1e-11 .. 1e-5 (relative) of the r^2 the
    reference computes for the record.  Far from the origin that error grows like 2^-52 CF2 W' per term; the clearance
    of a decision follows that bound (ChainFast.mg), so no distance from the origin makes the fast test contradict the
    exact one -- it only leaves more records undecided."""
    out = (C.c_longlong * 3)()
    dec = und = 0
    for seed in range(1, 4):
        lib().cgm_boundary(seed, D, 0, 4.0, 0.05, 200.0, centre_eps * 0.05, _sigma(D, f=1.0), 100, out)
        assert out[2] == 0, f"seed {seed}: the fast test contradicted the exact test on {out[2]} of {out[0]} decided records"
        dec, und = dec + out[0], und + out[1]
    assert dec > 0 and und > 0, (dec, und)  # both sides of the clearance are reached
