/* CPU model of the CONTESTED-group logic of the pcore replay (chronoclust_b200/csrc/engine.cuh: bs_radius_test,
 * bs_radius_fast, bs_chain_slow_group, bs_chain_slow_group_pairs, bs_chain_slow_group_batch, the ChainFast setup of
 * k_bs_chain_p) -- TEST INFRASTRUCTURE, plain loops, one "lane" per
 * record element.  It answers two questions no GPU is needed for:
 *   (1) is the division-free FAST radius test decision-exact, i.e. does it agree with the exact test of
 *       utilities/mc_functions.py:45-56 (objects/microcluster.py:213-233) whenever it takes a decision -- unsplit (padded
 *       width DP <= 16) and split (DP > 16), at any distance from the origin?
 *   (2) does the EIGHT-CELLS-PER-PASS schedule (tentative records laid along predicted verdicts, -0.0 as the addend of a
 *       cell that does not join, restart behind the first deviation) leave bit for bit the state and the verdicts of the
 *       one-by-one replay, whatever the predictions are?
 * The arithmetic follows the device code operation by operation (no contraction except the one explicit fma).
 * Build: gcc -O2 -ffp-contract=off -shared -fPIC -o libchaingroup.so chain_group_model.c -lm */
#include <math.h>
#include <stdint.h>
#include <string.h>

#define MAXD 64
#define GS 8

typedef struct {
    double cf1[MAXD], cf2[MAXD], w;
} Rec;

typedef struct {
    int D, DP, div_mode;
    double delta2, eps2, k, wsel;
    /* ChainFast */
    double F, fs, invk, mg;
} Prm;

static int round_dp(int D) { /* csrc/api.cu: the padded width the kernels are instantiated for */
    static const int dps[] = {4, 8, 12, 16, 24, 32, 40, 48, 64};
    for (int i = 0; i < 9; ++i)
        if (D <= dps[i]) return dps[i];
    return -1;
}

static uint64_t rng_s;
static double urand(void) { /* xorshift64* -> (0, 1) */
    rng_s ^= rng_s >> 12;
    rng_s ^= rng_s << 25;
    rng_s ^= rng_s >> 27;
    return ((rng_s * 0x2545F4914F6CDD1DULL) >> 11) * (1.0 / 9007199254740992.0) + 1e-300;
}
static double nrand(void) { return sqrt(-2.0 * log(urand())) * cos(6.283185307179586 * urand()); }

static Rec rec_add(const Rec *v, const double *x, int D) { /* v + ADDEND(x) = (x, x*x, 1.0), element by element */
    Rec r = *v;
    for (int d = 0; d < D; ++d) {
        r.cf1[d] = v->cf1[d] + x[d];
        r.cf2[d] = v->cf2[d] + x[d] * x[d];
    }
    r.w = v->w + 1.0;
    return r;
}
static Rec rec_add_negzero(const Rec *v, int D) { /* the addend of a cell that does not join: -0.0 in every element */
    Rec r = *v;
    for (int d = 0; d < D; ++d) {
        r.cf1[d] = v->cf1[d] + -0.0;
        r.cf2[d] = v->cf2[d] + -0.0;
    }
    r.w = v->w + -0.0;
    return r;
}

/* bs_radius_test: the reference's radius test on the tentative record, terms summed in index order */
static double exact_r2(const Rec *nv, const Prm *p) {
    double r2 = 0.0;
    for (int d = 0; d < p->D; ++d) {
        const double q2 = nv->cf2[d] / nv->w;
        const double c = nv->cf1[d] / nv->w;
        const double var = q2 - c * c;
        const int bit = var <= p->delta2;
        const double t = bit ? (p->div_mode ? var / p->k : var * p->wsel) : var;
        r2 = r2 + t;
    }
    return r2;
}
static int exact_test(const Rec *nv, const Prm *p) { return exact_r2(nv, p) <= p->eps2; }

static int d2i_rn_sat(double v) { /* cvt.rni.s32.f64: saturating, NaN -> 0 */
    if (v != v) return 0;
    const double r = nearbyint(v);
    if (r >= 2147483647.0) return 2147483647;
    if (r <= -2147483648.0) return (-2147483647 - 1);
    return (int)r;
}
static int d2i_rd_sat(double v) { return d2i_rn_sat(floor(v)); }
static int d2i_ru_sat(double v) { return d2i_rn_sat(ceil(v)); }

/* bs_radius_fast: 1 absorbed, 0 rejected, 2 too close to call.  DP <= 16: one integer per term, TH = 2^25; DP > 16: the
 * term is split into a high integer and a low part in 2^-20 units (two redux.sync), TH = 2^23.  NT == 2 (DP > 32) only
 * changes which lane holds a term; the integer sums do not depend on it. */
static int fast_test(const Rec *nv, const Prm *p) {
    const int split = p->DP > 16;
    const int CL = split ? (1 << 24) : (1 << 26);
    const double wn = nv->w;
    const double wn2 = wn * wn;
    const double thr = wn2 * p->F;
    const double d2w = p->delta2 * wn2;
    const double tol = d2w * 0x1p-24;
    const int t_lo = d2i_rd_sat(thr - p->mg), t_hi = d2i_ru_sat(thr + p->mg);
    long long S = 0, L = 0; /* redux.sync.add.s32 of at most 64 terms of magnitude <= 2^24 (2^26 unsplit, <= 16 terms) */
    int amb = 0;
    for (int d = 0; d < p->D; ++d) {
        const double c1 = nv->cf1[d], c2 = nv->cf2[d];
        const double t = fma(-c1, c1, c2 * wn);
        const double diff = t - d2w;
        amb |= !(fabs(diff) > tol);
        const double tk = t * p->invk;
        const double v = (diff <= 0.0 ? tk : t) * p->fs;
        int hi = d2i_rn_sat(v);
        hi = hi > CL ? CL : hi;
        hi = hi < -(1 << 20) ? -(1 << 20) : hi;
        S += hi;
        if (split) {
            int lo = d2i_rn_sat((v - (double)hi) * 0x1p20);
            lo = lo > (1 << 20) ? (1 << 20) : lo;
            lo = lo < -(1 << 20) ? -(1 << 20) : lo;
            L += lo;
        }
    }
    if (amb) return 2;
    if (split) {
        const double tot = (double)(int)S + (double)(int)L * 0x1p-20;
        if (tot < thr - p->mg) return 1;
        if (tot > thr + p->mg) return 0;
        return 2;
    }
    return S < t_lo ? 1 : (S > t_hi ? 0 : 2);
}

/* ChainFast of a chain of n cells that starts at state v (engine.cuh, chain setup of k_bs_chain_p) */
static void chain_fast(Prm *p, const Rec *v, int n) {
    const double TH = p->DP > 16 ? 0x1p23 : 0x1p25;
    const double wmax = v->w + (double)(n + 1);
    p->F = TH / (wmax * wmax);
    p->fs = p->F / p->eps2;
    p->invk = p->div_mode ? 1.0 / p->k : p->wsel;
    /* clearance: rounding of the integer terms (unsplit) or of the low parts (split), plus the bound on the fp64 error of
     * the terms from the chain's start state, sum_d CF2_d / W (summed here in another order than the warp's: a bound) */
    double q2 = 0.0;
    for (int d = 0; d < p->D; ++d) q2 += v->cf2[d];
    p->mg = (p->DP > 16 ? 0.01 : (double)(p->D + 8)) + 0x1p-48 * TH * (q2 / v->w) / p->eps2;
}

/* one by one with the EXACT test: the semantics everything else has to reproduce */
static void group_reference(Rec *v, const double x[GS][MAXD], unsigned cg, int ncell, const Prm *p, unsigned *rej) {
    *rej = 0u;
    for (int q = 0; q < ncell; ++q) {
        const Rec nv = rec_add(v, x[q], p->D);
        int keep = 1;
        if ((cg >> q) & 1u) keep = exact_test(&nv, p);
        if (keep) *v = nv;
        else *rej |= 1u << q;
    }
}

typedef struct {
    long long fast_decided, fast_undecided, fast_wrong, passes, groups, contested, rejected;
} Stats;

/* bs_chain_slow_group: cell by cell, the fast test first, the exact test where it cannot call (and for the first member of
 * the chain).  The only schedule at DP >= 16, where the record takes more than one register per lane. */
static void group_onebyone(Rec *vio, const double x[GS][MAXD], unsigned cg, int ncell, const Prm *p, int exact_first,
                           unsigned *rej_out, Stats *st) {
    Rec v = *vio;
    unsigned rej = 0u;
    for (int q = 0; q < ncell; ++q) {
        const Rec nv = rec_add(&v, x[q], p->D);
        int keep = 1;
        if ((cg >> q) & 1u) {
            int r = (q == 0 && exact_first) ? 2 : fast_test(&nv, p);
            if (r == 2) {
                if (!(q == 0 && exact_first)) ++st->fast_undecided;
                r = exact_test(&nv, p);
            } else {
                ++st->fast_decided;
                if (exact_test(&nv, p) != r) ++st->fast_wrong;
            }
            keep = r != 0;
        }
        if (keep) v = nv;
        else rej |= 1u << q;
    }
    *vio = v;
    *rej_out = rej;
}

/* bs_chain_slow_group_batch */
static void group_batch(Rec *vio, const double x[GS][MAXD], unsigned cg, unsigned pg, int ncell, const Prm *p, int exact_first,
                        unsigned *rej_out, Stats *st) {
    Rec v = *vio;
    const unsigned live = (1u << ncell) - 1u;
    cg &= live;
    const unsigned pred = pg & cg;
    unsigned rej = 0u;
    int q0 = 0;
    if (exact_first && (cg & 1u)) {
        const Rec nv = rec_add(&v, x[0], p->D);
        if (exact_test(&nv, p)) v = nv;
        else rej |= 1u;
        q0 = 1;
    }
    while (q0 < ncell) {
        ++st->passes;
        const unsigned todo = live & ~((1u << q0) - 1u);
        const unsigned adv = todo & ~pred;
        Rec nv[GS], sb[GS], state = v;
        for (int q = 0; q < GS; ++q) {
            sb[q] = state;
            nv[q] = rec_add(&state, x[q], p->D);
            state = ((adv >> q) & 1u) ? rec_add(&state, x[q], p->D) : rec_add_negzero(&state, p->D);
        }
        unsigned accm = 0u, rejm = 0u;
        for (int q = 0; q < GS; ++q) {
            const int r = fast_test(&nv[q], p);
            accm |= (r == 1 ? 1u : 0u) << q;
            rejm |= (r == 0 ? 1u : 0u) << q;
        }
        const unsigned und = ~(accm | rejm);
        const unsigned dev = ((rejm & ~pred) | (accm & pred) | und) & cg & todo;
        int qs = ncell;
        if (dev) {
            qs = 0;
            while (!((dev >> qs) & 1u)) ++qs;
        }
        const int qe = qs < ncell - 1 ? qs : ncell - 1;
        /* every fast verdict this pass relies on (cells q0 .. qe that are CONTESTED and decided) against the exact test */
        for (int q = q0; q <= qe; ++q) {
            if (!((cg >> q) & 1u)) continue;
            if ((und >> q) & 1u) {
                ++st->fast_undecided;
                continue;
            }
            ++st->fast_decided;
            if (exact_test(&nv[q], p) != (int)((accm >> q) & 1u)) ++st->fast_wrong;
        }
        rej |= pred & todo & ((1u << qs) - 1u);
        int keep;
        if (dev) {
            if ((und >> qs) & 1u) keep = exact_test(&nv[qs], p);
            else keep = (accm >> qs) & 1u;
            rej |= (keep ? 0u : 1u) << qs;
        } else {
            keep = !((pred >> qe) & 1u);
        }
        v = keep ? nv[qe] : sb[qe];
        q0 = qs + 1;
    }
    *vio = v;
    *rej_out = rej;
}

/* bs_chain_slow_group_pairs (verdicts only; the state follows from them) */
static void group_pairs(Rec *vio, const double x[GS][MAXD], unsigned cg, int ncell, const Prm *p, int exact_first,
                        unsigned *rej_out, Stats *st) {
    Rec v = *vio;
    unsigned rej = 0u;
    for (int q = 0; q < ncell; q += 2) {
        const int hasB = q + 1 < ncell;
        const int cA = (cg >> q) & 1u, cB = hasB && ((cg >> (q + 1)) & 1u);
        const Rec nvA = rec_add(&v, x[q], p->D);
        int rA = 1, rB = 1, done = 0;
        Rec nvB = nvA;
        if (cA && cB && !(q == 0 && exact_first)) {
            const Rec nvB1 = rec_add(&nvA, x[q + 1], p->D), nvB0 = rec_add(&v, x[q + 1], p->D);
            rA = fast_test(&nvA, p);
            const int rB1 = fast_test(&nvB1, p), rB0 = fast_test(&nvB0, p);
            rB = rA ? rB1 : rB0;
            nvB = rA ? nvB1 : nvB0;
            done = rA != 2 && rB != 2;
            if (done) {
                st->fast_decided += 2;
                if (exact_test(&nvA, p) != rA) ++st->fast_wrong;
                if (exact_test(&nvB, p) != rB) ++st->fast_wrong;
            }
        }
        if (!done) {
            if (cA) {
                rA = (q == 0 && exact_first) ? 2 : fast_test(&nvA, p);
                if (rA == 2) rA = exact_test(&nvA, p);
            }
            if (hasB) {
                nvB = rec_add(rA ? &nvA : &v, x[q + 1], p->D);
                if (cB) {
                    rB = fast_test(&nvB, p);
                    if (rB == 2) rB = exact_test(&nvB, p);
                }
            }
        }
        if (hasB) {
            if (rB) v = nvB;
            else if (rA) v = nvA;
            rej |= ((cA && !rA) ? 1u : 0u) << q | ((cB && !rB) ? 1u : 0u) << (q + 1);
        } else {
            if (rA) v = nvA;
            rej |= ((cA && !rA) ? 1u : 0u) << q;
        }
    }
    *vio = v;
    *rej_out = rej;
}

/* One chain: an MC grown to weight ~W0 at its radius limit (cells drawn around a centre with per-dimension spread sigma,
 * absorbed under the exact test), then `ngroups` groups of eight cells replayed three ways.  pred_mode: 0 all "absorbed",
 * 1 all "rejected", 2 random, 3 the true verdicts, 4 the true verdicts with every fourth one flipped.
 * Returns the number of groups whose verdicts or final state (bit patterns) differ from the one-by-one replay; out[0..6] =
 * fast decided / undecided / wrong, passes, groups, CONTESTED cells, rejected cells. */
long long cgm_run(uint64_t seed, int D, int div_mode, double kk, double eps, double delta, double W0, double centre_scale,
                  double sigma, double far_frac, int ngroups, int pred_mode, double contested_frac, long long *out) {
    rng_s = seed * 0x9E3779B97F4A7C15ULL + 0x1234567ULL;
    Prm p;
    memset(&p, 0, sizeof p);
    p.D = D;
    p.DP = round_dp(D);
    p.div_mode = div_mode;
    p.k = kk;
    p.wsel = 1.0 / kk;
    p.eps2 = eps * eps;
    p.delta2 = delta * delta;
    double centre[MAXD];
    for (int d = 0; d < D; ++d) centre[d] = centre_scale * urand();
    Rec v;
    memset(&v, 0, sizeof v);
    /* seed the MC with one cell at the centre, then grow it under the exact test */
    v = rec_add(&v, centre, D);
    long long guard = 0;
    while (v.w < W0 && guard++ < 50 * (long long)W0 + 1000) {
        double x[MAXD];
        for (int d = 0; d < D; ++d) x[d] = centre[d] + sigma * nrand();
        const Rec nv = rec_add(&v, x, D);
        if (exact_test(&nv, &p)) v = nv;
    }
    chain_fast(&p, &v, ngroups * GS);
    Stats st;
    memset(&st, 0, sizeof st);
    long long bad = 0;
    Rec vb = v, vp = v;
    for (int g = 0; g < ngroups; ++g) {
        double x[GS][MAXD];
        unsigned cg = 0u;
        for (int q = 0; q < GS; ++q) {
            const int cont = urand() < contested_frac; /* a cell that is not CONTESTED is SAFE: close to the centre */
            const double s = cont ? (urand() < far_frac ? 3.0 * sigma : sigma) : 0.5 * sigma;
            for (int d = 0; d < D; ++d) x[q][d] = centre[d] + s * nrand();
            if (cont) cg |= 1u << q;
        }
        const int ncell = (g == ngroups - 1) ? 1 + (int)(urand() * 7.999) : GS; /* ragged tail */
        cg &= (1u << ncell) - 1u;
        Rec vr = v;
        unsigned rej_ref, rej_b, rej_p;
        group_reference(&vr, x, cg, ncell, &p, &rej_ref);
        unsigned pg;
        switch (pred_mode) {
        case 0: pg = 0u; break;
        case 1: pg = 0xffu; break;
        case 2: pg = (unsigned)(urand() * 256.0) & 0xffu; break;
        case 3: pg = rej_ref; break;
        default: pg = rej_ref ^ 0x88u; break;
        }
        if (p.DP <= 12) { /* the record is one register per lane (NH == 1): the two group schedules */
            group_batch(&vb, x, cg, pg, ncell, &p, g == 0, &rej_b, &st);
            group_pairs(&vp, x, cg, ncell, &p, g == 0, &rej_p, &st);
        } else {
            group_onebyone(&vb, x, cg, ncell, &p, g == 0, &rej_b, &st);
            vp = vb;
            rej_p = rej_b;
        }
        ++st.groups;
        st.contested += __builtin_popcount(cg);
        st.rejected += __builtin_popcount(rej_ref);
        if (rej_b != rej_ref || rej_p != rej_ref || memcmp(&vb, &vr, sizeof(Rec)) != 0 || memcmp(&vp, &vr, sizeof(Rec)) != 0) ++bad;
        v = vr;
        vb = vr; /* (keep the three replays on the reference state so that one divergence is counted once) */
        vp = vr;
    }
    out[0] = st.fast_decided;
    out[1] = st.fast_undecided;
    out[2] = st.fast_wrong;
    out[3] = st.passes;
    out[4] = st.groups;
    out[5] = st.contested;
    out[6] = st.rejected;
    return bad;
}

/* The fast test AT the decision boundary: a record of W cells drawn around a centre (coordinates centre_scale * U(0, 1)) with
 * spread sigma, and eps^2 placed at the reference's own r^2 of that record times 1 +- rho, rho log-uniform in
 * [1e-11, 1e-5] -- where the fp64 error of the fast test's terms decides.  ntrials records; out[0..2] = fast decided /
 * undecided / wrong. */
void cgm_boundary(uint64_t seed, int D, int div_mode, double kk, double delta, double W, double centre_scale, double sigma,
                  int ntrials, long long *out) {
    rng_s = seed * 0x9E3779B97F4A7C15ULL + 0x7654321ULL;
    Prm p;
    memset(&p, 0, sizeof p);
    p.D = D;
    p.DP = round_dp(D);
    p.div_mode = div_mode;
    p.k = kk;
    p.wsel = 1.0 / kk;
    p.delta2 = delta * delta;
    Stats st;
    memset(&st, 0, sizeof st);
    for (int it = 0; it < ntrials; ++it) {
        double centre[MAXD];
        for (int d = 0; d < D; ++d) centre[d] = centre_scale * urand();
        Rec v;
        memset(&v, 0, sizeof v);
        for (int i = 0; i < (int)W; ++i) {
            double x[MAXD];
            for (int d = 0; d < D; ++d) x[d] = centre[d] + sigma * nrand();
            v = rec_add(&v, x, D);
        }
        p.eps2 = 1.0; /* (exact_r2 does not read eps^2) */
        const double r2 = exact_r2(&v, &p);
        const double rho = exp(log(1e-11) + urand() * (log(1e-5) - log(1e-11)));
        p.eps2 = r2 * (urand() < 0.5 ? 1.0 - rho : 1.0 + rho);
        chain_fast(&p, &v, 0); /* (Wmax = W + 1, as for a chain whose last member brings W' to W) */
        const int r = fast_test(&v, &p);
        if (r == 2) {
            ++st.fast_undecided;
            continue;
        }
        ++st.fast_decided;
        if (r != exact_test(&v, &p)) ++st.fast_wrong;
    }
    out[0] = st.fast_decided;
    out[1] = st.fast_undecided;
    out[2] = st.fast_wrong;
}
