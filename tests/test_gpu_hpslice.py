"""GPU: slice sampling of continuous hypers on the device (msb_state_slice_hp / state.slice_hp).

Every update is replayed in fp64 from the restated Philox stream against the CPU checker's score_data summed over the
groups plus the numpy prior (niw: the rank-one form, itself held to the checker's closed form); chained updates of many
identical features follow the exact conditional, integrated numerically on the host, by KS.  The state a call leaves
scores like the same hypers set by hand, and the four-entity Gibbs chain with slice_hp after each sweep visits the
partitions and hyper means of the exact posterior.
"""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
from scipy import special, stats

import common_b200 as cb
import oracle_lib as ol
from common_b200 import hyperprior as hpr
from test_gpu_parity import _four_entities, make_state
from test_gpu_theta import Stream

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HPSL_TAG = 0x4850534c00000000
M, SHRINK_CAP = 128, 200
NEAR = 1e-12    # a decision within NEAR * sum_c |cell_c| of its boundary may go either way under a last-ulp difference


def hp_offset(desc, key):
    d = desc()
    name, p = d.name(), d._param()
    if name == "niw":
        return {"kappa": p, "nu": p + 1 + p * p}[key]
    return list(d.default_hyperparams()).index(key)


def support_lo(desc, key):
    d = desc()
    if d.name() == "nich" and key == "mu":
        return -math.inf
    if d.name() == "niw" and key == "nu":
        return d._param() - 1.0
    return 0.0


def niw_prep(st, d, gids, dim, h):
    """(log |psi|, [(n, log |B|, q) per group]) from the state's suffstats"""
    mu0, psi = h[:dim], h[dim + 1:dim + 1 + dim * dim].reshape(dim, dim)
    rows = []
    for g in gids:
        n = st.get_suffstats(d, g, "count")[0]
        if n == 0:
            rows.append((0.0, 0.0, 0.0))
            continue
        sx = st.get_suffstats(d, g, "sum_x", dim)
        B = psi + st.get_suffstats(d, g, "sum_xxT", dim * dim).reshape(dim, dim) - np.outer(sx, sx) / n
        v = sx / n - mu0
        rows.append((n, np.linalg.slogdet(B)[1], float(v @ np.linalg.solve(B, v))))
    return np.linalg.slogdet(psi)[1], np.array(rows)


def niw_cells(dim, kappa, nu, ld0, rows):
    n, ldB, q = rows[:, 0], rows[:, 1], rows[:, 2]
    j = np.arange(dim)[None, :]
    lg = np.sum(special.gammaln(0.5 * (nu + n[:, None] - j)) - special.gammaln(0.5 * (nu - j)), axis=1)
    kn = kappa + n
    ldn = ldB + np.log1p(kappa * n * q / kn)
    cells = -0.5 * n * dim * math.log(math.pi) + lg + 0.5 * nu * ld0 - 0.5 * (nu + n) * ldn + 0.5 * dim * np.log(kappa / kn)
    return np.where(n == 0, 0.0, cells)


def log_prior(prior, x, partner):
    if prior.kind == hpr.NONINFORMATIVE_BETA:
        return float(prior(x, partner))
    return float(prior(x))


def feature_target(oracle, desc, key, prior, h, ss_rows=None, niw=None):
    """f(x) -> (value, sum |cell|) for coordinate key of a feature with hp vector h (other coordinates as in h)"""
    m, off, lo = oracle.model(desc), hp_offset(desc, key), support_lo(desc, key)
    partner = h[1 - off] if prior.kind == hpr.NONINFORMATIVE_BETA else None

    def f(x):
        if not x > lo:
            return -math.inf, 0.0
        lp = log_prior(prior, x, partner)
        if lp == -math.inf:
            return lp, 0.0
        hx = h.copy()
        hx[off] = x
        if niw is not None:
            dim = desc()._param()
            cells = niw_cells(dim, hx[dim], hx[dim + 1 + dim * dim], *niw)
        else:
            cells = np.array([oracle.score_data(m, hx, r) for r in ss_rows])
        return lp + float(np.sum(cells)), float(np.sum(np.abs(cells)))
    return f


def alpha_target(prior, counts):
    ne, n = float(np.sum(counts > 0)), float(np.sum(counts))

    def f(x):
        if not x > 0.0:
            return -math.inf, 0.0
        lp = log_prior(prior, x, None)
        if lp == -math.inf:
            return lp, 0.0
        v = (ne - 1.0) * math.log(x) + math.lgamma(1.0 + x) - math.lgamma(n + x)
        return lp + v, abs(v)
    return f


def slice_replay(oracle, seed, counter, d, j, f, x0, w):
    """(new value, number of decisions within NEAR of their boundary, evaluations, capped)"""
    rs = Stream(oracle, seed, d, j, counter, HPSL_TAG)
    f0, _ = f(x0)
    assert math.isfinite(f0)
    y = f0 + math.log(rs.u_open())
    near, evals = 0, 1

    def above(x):
        nonlocal near, evals
        v, scale = f(x)
        evals += 1
        if math.isfinite(v) and abs(v - y) <= NEAR * max(scale, 1.0):
            near += 1
        return v > y

    L = x0 - w * rs.u53()
    R = L + w
    jl = int(M * rs.u53())
    jr = M - 1 - jl
    while jl > 0 and above(L):
        L -= w
        jl -= 1
    while jr > 0 and above(R):
        R += w
        jr -= 1
    for _ in range(SHRINK_CAP):
        x = L + rs.u53() * (R - L)
        if above(x):
            return x, near, evals, False
        if x < x0:
            L = x
        else:
            R = x
    return x0, near, evals, True


E1 = hpr.log_exponential(1.0)
# family -> {key: (prior, width)}: every prior kind, widths 0.01 .. 5
SPECS = {
    "bb": {("alpha", "beta"): (hpr.log_noninformative_beta_prior, 1.0)},
    "bnb": {"alpha": (hpr.log_exponential(0.5), 0.5), "beta": (hpr.log_normal(1.0, 4.0), 2.0)},
    "gp": {"alpha": (hpr.log_flat(0.01, 50.0), 5.0), "inv_beta": (E1, 0.01)},
    "nich": {"mu": (hpr.log_normal(0.0, 10.0), 0.3), "kappa": (E1, 1.0), "sigmasq": (hpr.log_flat(1e-3, 100.0), 2.0),
             "nu": (hpr.log_exponential(0.2), 5.0)},
    "bbnc": {"alpha": (E1, 0.05), "beta": (hpr.log_noninformative_beta_prior, 0.2)},
    "niw3": {"nu": (hpr.log_flat(2.0, 50.0), 3.0), "kappa": (E1, 1.0)},
    "niw64": {"kappa": (hpr.log_normal(1.0, 4.0), 0.7), "nu": (hpr.log_exponential(0.05), 5.0)},
}
CASES = {"every": [cb.bb, cb.bnb, cb.gp, cb.nich, cb.bbnc, cb.niw(3)], "niw64": [cb.niw(64), cb.bb]}
START = {"bnb": {"alpha": 2.5, "beta": 1.5, "r": 1.0}, "gp": {"alpha": 2.0, "inv_beta": 0.7},
         "niw64": {"nu": 70.0, "psi": np.eye(64) * 2.0}}


def spec_key(desc):
    d = desc()
    return "niw%d" % d._param() if d.name() == "niw" else d.name()


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("k", [3, 200, 700])
def test_updates_replay_in_fp64(ctx, oracle, case, k):
    descs = CASES[case]
    hp = {d: START[spec_key(desc)] for d, desc in enumerate(descs) if spec_key(desc) in START}
    st, view, z, gids, hp_flat, ss, counts = make_state(ctx, oracle, descs, max(1500, 6 * k), k, seed=k + len(descs),
                                                        mask_frac=0.05, extra_empty=2, hp=hp)
    hparams = {d: SPECS[spec_key(desc)] for d, desc in enumerate(descs)}
    if case == "niw64":
        hparams[1] = {"alpha": (hpr.log_flat(0.01, 10.0), 0.01)}
    cparam = {"alpha": (hpr.log_normal(1.0, 1.0), 0.5) if case == "niw64" else (E1, 1.0)}
    before = [np.concatenate([np.ravel(v) for v in st.get_component_hp(d).values()]) for d in range(len(descs))]
    alpha0 = st.get_cluster_hp()["alpha"]
    seed, counter = 100 + k, 7
    r = st.slice_hp(hparams, cparam, seed=seed, counter=counter)
    assert r["capped"] == 0
    got = r["values"]
    off = np.cumsum([0] + [oracle.ss_size(oracle.model(desc)) for desc in descs])
    near = total = 0
    for d, desc in enumerate(descs):
        h = before[d].copy()                                                   # the flat hp vector before the call
        niw = niw_prep(st, d, gids, desc()._param(), h) if desc().name() == "niw" else None
        j = 0
        for key, (prior, w) in hparams[d].items():
            for kk in (key if isinstance(key, tuple) else (key,)):
                f = feature_target(oracle, desc, kk, prior, h, ss[:, off[d]:off[d + 1]], niw)
                x0 = h[hp_offset(desc, kk)]
                want, n_near, _, cap = slice_replay(oracle, seed, counter, d, j, f, x0, w)
                assert not cap
                total += 1
                if n_near:
                    near += 1
                else:
                    assert abs(got[d][kk] - want) <= 1e-12 * abs(want), (d, kk, got[d][kk], want)
                h[hp_offset(desc, kk)] = got[d][kk]                            # the next spec conditions on the draw
                j += 1
    want, n_near, _, cap = slice_replay(oracle, seed, counter, len(descs), 0, alpha_target(cparam["alpha"][0], counts),
                                        alpha0, cparam["alpha"][1])
    total += 1
    if n_near:
        near += 1
    else:
        assert abs(got["alpha"] - want) <= 1e-12 * want
    print("slice_hp replay %s k=%d: %d of %d updates had a decision within %g of its boundary" % (case, k, near, total, NEAR))
    assert near <= 2
    st.close()


@pytest.mark.parametrize("dim", [3, 64])
def test_rank_one_niw_target_is_the_closed_form(ctx, oracle, dim):
    desc = cb.niw(dim)
    st, view, z, gids, hp_flat, ss, counts = make_state(ctx, oracle, [desc], 3000, 40, seed=dim, mask_frac=0.05, extra_empty=2,
                                                        hp={0: {"nu": dim + 3.0, "psi": np.eye(dim) * 1.5}})
    m = oracle.model(desc)
    for kappa, nu in [(1.0, dim + 3.0), (0.05, dim - 0.5), (40.0, 5.0 * dim)]:
        h = oracle.flat_hp(desc, {"kappa": kappa, "nu": nu, "psi": np.eye(dim) * 1.5})
        direct = np.array([oracle.score_data(m, h, ss[c]) for c in range(ss.shape[0])])
        rank1 = niw_cells(dim, kappa, nu, *niw_prep(st, 0, gids, dim, h))
        assert abs(rank1.sum() - direct.sum()) <= 1e-10 * np.abs(direct).sum(), (kappa, nu, rank1.sum(), direct.sum())
    st.close()


def _identical_features(ctx, oracle, desc, F, n, K, seed):
    """a state of F features that all hold the same column; (state, the one-feature suffstats rows, counts)"""
    arr1, z = cb.synth.make_dataset([desc], n, K, seed=seed)
    col = arr1[arr1.dtype.names[0]]
    arr = np.zeros(n, dtype=[("f%d" % d, arr1.dtype[0]) for d in range(F)])
    for d in range(F):
        arr["f%d" % d] = col
    st = cb.state(ctx, [desc] * F, max_groups=K + 2, cluster_hp={"alpha": 1.0})
    h = oracle.flat_hp(desc)
    st.bind(cb.numpy_dataview(arr))
    gids = [st.create_group() for _ in range(K)]
    st.add_values(np.asarray(gids)[z])
    ss, counts = ol.build_suffstats(oracle, [desc], h, cb.numpy_dataview(arr1), z, K)
    return st, ss, counts


def _cdf(f, lo, hi, npts=20000):
    """the normalised CDF of exp(f) on (lo, hi), integrated on a grid uniform in log(x - lo)"""
    u = np.linspace(math.log(hi - lo) - 26.0, math.log(hi - lo), npts)
    x = lo + np.exp(u)
    lf = np.array([f(v)[0] for v in x]) + u                                   # dx = (x - lo) du
    p = np.exp(lf - np.max(lf))
    c = np.concatenate([[0.0], np.cumsum(0.5 * (p[1:] + p[:-1]) * np.diff(u))])
    assert p[0] < 1e-9 * p.max() and p[-1] < 1e-9 * p.max(), "the grid does not hold the mass"
    return lambda v: np.interp(v, x, c / c[-1])


LAW = [("bb-alpha", cb.bb, "alpha", E1, 1.0, 0.0, 60.0),
       ("nich-kappa", cb.nich, "kappa", hpr.log_flat(0.05, 20.0), 2.0, 0.0, 20.0),
       ("gp-inv_beta", cb.gp, "inv_beta", hpr.log_exponential(0.5), 0.5, 0.0, 200.0),
       ("niw-nu", cb.niw(3), "nu", hpr.log_exponential(0.1), 3.0, 2.0, 600.0)]


@pytest.mark.parametrize("name,desc,key,prior,w,lo,hi", LAW, ids=[c[0] for c in LAW])
def test_chained_updates_follow_the_exact_conditional(ctx, oracle, name, desc, key, prior, w, lo, hi):
    F, K = 300, 6
    st, ss, counts = _identical_features(ctx, oracle, desc, F, 120, K, seed=len(name))
    h = oracle.flat_hp(desc)
    for it in range(30):
        assert st.slice_hp({d: {key: (prior, w)} for d in range(F)}, seed=41, counter=it)["capped"] == 0
    x = np.array([st.get_component_hp(d)[key] for d in range(F)])
    cdf = _cdf(feature_target(oracle, desc, key, prior, h, ss), lo, hi)
    r = stats.kstest(x, cdf)
    print("slice_hp law %s: KS p-value %.3g (mean %.4g)" % (name, r.pvalue, x.mean()))
    assert r.pvalue > 1e-3
    st.close()


def test_alpha_chain_follows_the_exact_conditional(ctx, oracle):
    st, view, z, gids, hp_flat, ss, counts = make_state(ctx, oracle, [cb.bb], 40, 5, seed=3, extra_empty=1)
    prior = hpr.log_exponential(1.0)
    xs = []
    for it in range(3100):
        v = st.slice_hp(cparam={"alpha": (prior, 1.0)}, seed=5, counter=it)["values"]["alpha"]
        if it >= 100 and it % 10 == 0:
            xs.append(v)
    r = stats.kstest(xs, _cdf(alpha_target(prior, counts), 0.0, 80.0))
    print("slice_hp law alpha: KS p-value %.3g over %d thinned draws" % (r.pvalue, len(xs)))
    assert r.pvalue > 1e-3
    st.close()


def _snapshot(st, gids, ncomp):
    ss = [st.get_suffstats(d, g, key, st._ss_counts(st._models[d], key)).tobytes()
          for d in range(ncomp) for g in gids for key in st._SS_KEYS[st._models[d].name()]]
    hps = [{k: np.asarray(v).tobytes() for k, v in st.get_component_hp(d).items()} for d in range(ncomp)]
    return st.assignments().tobytes(), ss, [st.groupsize(g) for g in gids], hps, st.get_cluster_hp()


def test_the_applied_state_scores_like_hypers_set_by_hand(ctx, oracle):
    descs = [cb.bb, cb.nich, cb.dd(16), cb.gp, cb.niw(3), cb.bbnc, cb.bnb]
    a, _, _, gids, _, _, _ = make_state(ctx, oracle, descs, 2000, 7, seed=4, mask_frac=0.05, extra_empty=1, hp={6: START["bnb"]})
    b, _, _, _, _, _, _ = make_state(ctx, oracle, descs, 2000, 7, seed=4, mask_frac=0.05, extra_empty=1, hp={6: START["bnb"]})
    before = _snapshot(a, gids, len(descs))
    hparams = {0: SPECS["bb"], 1: SPECS["nich"], 3: SPECS["gp"], 4: SPECS["niw3"], 6: SPECS["bnb"]}
    r = a.slice_hp(hparams, {"alpha": (E1, 1.0)}, seed=3, counter=1)
    after = _snapshot(a, gids, len(descs))
    assert after[:3] == before[:3]                                   # assignments, suffstats, group sizes
    for d in (2, 5):                                                 # features without a spec keep their hypers
        assert after[3][d] == before[3][d]
    for d, vals in r["values"].items():
        if d == "alpha":
            assert a.get_cluster_hp()["alpha"] == vals
            continue
        got = a.get_component_hp(d)
        for key, v in vals.items():
            assert got[key] == v, (d, key)
        b.set_component_hp(d, vals)
    b.set_cluster_hp({"alpha": r["values"]["alpha"]})
    _, sa = a.score_rows()
    _, sb = b.score_rows()
    assert np.array_equal(sa.view(np.uint32), sb.view(np.uint32))
    for d in range(len(descs)):
        for g in gids:
            assert a.score_likelihood(d, g) == b.score_likelihood(d, g)
    a.close(); b.close()


def test_gibbs_chain_with_slice_hp_visits_the_exact_posterior(ctx):
    """partitions x (alpha_d, beta_d) per feature x CRP alpha, every hyper under Exponential(1): the partition marginal
    and each hyper's posterior mean, integrated on a log grid on the host"""
    from math import lgamma
    arr, n, D, _, _, canon = _four_entities()
    data = np.stack([arr["f%d" % d] for d in range(D)], axis=1).astype(int)
    u = np.linspace(-12.0, 6.0, 500)
    x = np.exp(u)
    wx = np.exp(-x) * x * (u[1] - u[0])                               # Exponential(1) density times dx on the log grid
    A, B = x[:, None], x[None, :]
    lbab = special.betaln(A, B)

    def partitions(items):
        if not items:
            yield []
            return
        first, rest = items[0], items[1:]
        for p in partitions(rest):
            for i in range(len(p)):
                yield p[:i] + [[first] + p[i]] + p[i + 1:]
            yield [[first]] + p

    parts, logz, mean_a, mean_b, mean_al = [], [], [], [], []
    for p in partitions(list(range(n))):
        a = [0] * n
        for gi, g in enumerate(p):
            for e in g:
                a[e] = gi
        crp = len(p) * np.log(x) + special.gammaln(x) - special.gammaln(n + x) + sum(lgamma(len(g)) for g in p)
        wc = np.exp(crp) * wx
        lz, ma, mb = math.log(wc.sum()), [], []
        for d in range(D):
            s = np.zeros_like(lbab)
            for g in p:
                h = int(data[g, d].sum())
                s += special.betaln(A + h, B + len(g) - h) - lbab
            w2 = np.exp(s) * wx[:, None] * wx[None, :]
            lz += math.log(w2.sum())
            ma.append((w2 * A).sum() / w2.sum())
            mb.append((w2 * B).sum() / w2.sum())
        parts.append(canon(a)); logz.append(lz); mean_a.append(ma); mean_b.append(mb)
        mean_al.append((wc * x).sum() / wc.sum())
    pw = np.exp(np.array(logz) - max(logz))
    pw /= pw.sum()
    exact_part = dict(zip(parts, pw))
    exact = np.concatenate([pw @ np.array(mean_a), pw @ np.array(mean_b), [pw @ np.array(mean_al)]])

    st = cb.state(ctx, [cb.bb] * D, max_groups=8, cluster_hp={"alpha": 1.0})
    st.bind(cb.numpy_dataview(arr))
    g0 = st.create_group()
    st.add_values(np.full(n, g0))
    hparams = {d: {("alpha", "beta"): (E1, 1.0)} for d in range(D)}
    rng = np.random.default_rng(0)
    visits, trace = {}, []
    sweeps, burn = 4100, 100
    for it in range(sweeps):
        for eid in range(n):
            st.remove_value(eid)
            empties = st.empty_groups()
            if not empties:
                st.create_group()
            elif len(empties) > 1:
                for g in empties[1:]:
                    st.delete_group(g)
            gids, s = st.score_value(eid)
            p = np.exp(np.asarray(s, np.float64) - np.max(s))
            st.add_value(gids[int(rng.choice(len(gids), p=p / p.sum()))], eid)
        v = st.slice_hp(hparams, {"alpha": (E1, 1.0)}, seed=17, counter=it)["values"]
        if it >= burn:
            key = canon(st.assignments().tolist())
            visits[key] = visits.get(key, 0) + 1
            trace.append([v[d]["alpha"] for d in range(D)] + [v[d]["beta"] for d in range(D)] + [v["alpha"]])
    st.close()
    total = sweeps - burn
    worst = max(abs(visits.get(k, 0) / total - pk) for k, pk in exact_part.items())
    print("slice_hp chain: largest partition deviation %.4f" % worst)
    assert worst < 0.04, worst
    trace = np.array(trace)
    batches = trace.reshape(40, -1, trace.shape[1]).mean(axis=1)
    se = batches.std(axis=0, ddof=1) / math.sqrt(40)
    z_scores = (trace.mean(axis=0) - exact) / se
    print("slice_hp chain: hyper means %s, exact %s, z %s" % (trace.mean(axis=0), exact, z_scores))
    assert np.all(np.abs(z_scores) < 4.0), z_scores


def test_same_seed_and_counter_give_the_same_bits(ctx, oracle):
    descs = [cb.nich, cb.gp, cb.niw(4), cb.bb]
    a = make_state(ctx, oracle, descs, 3000, 50, seed=6, extra_empty=3)
    b = make_state(ctx, oracle, descs, 3000, 50, seed=6, extra_empty=3)
    hparams = {0: SPECS["nich"], 1: {"inv_beta": (E1, 0.5)}, 2: {"kappa": (E1, 1.0)}, 3: SPECS["bb"]}
    cp = {"alpha": (E1, 1.0)}
    ra = a[0].slice_hp(hparams, cp, seed=9, counter=4)
    rb = b[0].slice_hp(hparams, cp, seed=9, counter=4)
    assert ra == rb
    ra2 = a[0].slice_hp(hparams, cp, seed=9, counter=5)
    flat = lambda r: [v for d in sorted(r["values"], key=str) for v in (r["values"][d].values() if isinstance(r["values"][d], dict) else [r["values"][d]])]  # noqa: E731
    assert all(x != y for x, y in zip(flat(ra), flat(ra2)))
    a[0].close(); b[0].close()


def test_refusals_leave_the_state_untouched(ctx, oracle):
    descs = [cb.bb, cb.bnb, cb.niw(3), cb.nich, cb.gp, cb.dd(4), cb.bbnc]
    st, view, z, gids, hp, ss, counts = make_state(ctx, oracle, descs, 600, 4, seed=5, extra_empty=1, hp={1: START["bnb"]})
    before = _snapshot(st, gids, len(descs))
    lib = cb._lib

    def refused(hparams, cparam, match, status=lib.MSB_ERR_INVALID, counter=0):
        with pytest.raises(cb.MsbError, match=match) as e:
            st.slice_hp(hparams, cparam, counter=counter)
        assert e.value.status == status
        assert _snapshot(st, gids, len(descs)) == before

    ok = {0: {"alpha": (E1, 1.0)}, 3: {"mu": (E1, 1.0)}}
    nib = hpr.log_noninformative_beta_prior
    refused({**ok, 4: {"alpha": (E1, 0.0)}}, None, "feature 4: key 'alpha': the slice width must be finite and positive")
    refused({**ok, 4: {"alpha": (E1, -1.0)}}, None, "feature 4: key 'alpha': the slice width")
    refused({**ok, 4: {"alpha": (E1, np.nan)}}, None, "feature 4: key 'alpha': the slice width")
    refused({**ok, 4: {"alpha": (E1, np.inf)}}, None, "feature 4: key 'alpha': the slice width")
    refused({3: {"kappa": (hpr.log_flat(2.0, 2.0), 1.0)}}, None, "feature 3: key 'kappa': the flat prior needs finite lo < hi")
    refused({3: {"kappa": (hpr.log_flat(0.0, np.inf), 1.0)}}, None, "the flat prior")
    refused({3: {"kappa": (hpr.log_exponential(0.0), 1.0)}}, None, "feature 3: key 'kappa': the exponential prior")
    refused({3: {"kappa": (hpr.log_normal(0.0, -1.0), 1.0)}}, None, "feature 3: key 'kappa': the normal prior")
    refused({4: {"alpha": (nib, 1.0)}}, None, "feature 4: key 'alpha': the non-informative beta prior applies")
    refused(None, {"alpha": (nib, 1.0)}, "alpha: the non-informative beta prior applies")
    refused({0: {"alpha": (E1, 1.0), ("beta", "alpha"): (E1, 1.0)}}, None, "feature 0: key 'alpha': the key appears twice")
    refused({len(descs) + 1: {"alpha": (E1, 1.0)}}, None, "out of range")
    refused(ok, None, "below 2", counter=1 << 32)
    refused({1: {"r": (E1, 1.0)}}, None, "feature 1: key 'r': bnb's score_data drops")
    refused({5: {"alphas": (E1, 1.0)}}, None, "feature 5: key 'alphas': a vector hyper", lib.MSB_ERR_UNSUPPORTED)
    refused({2: {"mu": (E1, 1.0)}}, None, "msb_state_set_hp_grid", lib.MSB_ERR_UNSUPPORTED)
    refused({2: {"psi": (E1, 1.0)}}, None, "a vector hyper", lib.MSB_ERR_UNSUPPORTED)
    refused({0: {"gamma": (E1, 1.0)}}, None, "feature 0", lib.MSB_ERR_KEY)
    refused(None, {"beta": (E1, 1.0)}, "alpha", lib.MSB_ERR_KEY)
    # a current value where the target is not finite
    refused({3: {"kappa": (hpr.log_flat(2.0, 5.0), 1.0)}}, None, "feature 3: key 'kappa': the target .* is not finite at the current value")
    st.set_component_hp(2, {"nu": 2.0})                                   # niw(3): nu <= d - 1
    before = _snapshot(st, gids, len(descs))
    refused({2: {"kappa": (E1, 1.0)}}, None, "feature 2: key 'kappa': the target")
    st.set_component_hp(2, {"nu": 5.0})
    st.set_suffstats(6, gids[0], "heads", 5.0)
    st.set_suffstats(6, gids[0], "p", 0.0)                                # bbnc: p = 0 with heads
    before = _snapshot(st, gids, len(descs))
    refused({0: {"alpha": (E1, 1.0)}, 6: {"beta": (E1, 1.0)}}, None, "feature 6: key 'beta': the target")
    st.set_suffstats(6, gids[0], "p", 0.5)
    r = st.slice_hp({0: {"alpha": (E1, 1.0)}, 2: {"kappa": (E1, 1.0)}, 6: {"beta": (E1, 1.0)}}, {"alpha": (E1, 1.0)})
    assert r["capped"] == 0 and set(r["values"]) == {0, 2, 6, "alpha"}
    assert st.slice_hp() == {"capped": 0, "values": {}}
    st.close()


def test_two_ranks_draw_identical_hypers():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    port = 29900 + os.getpid() % 90
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "scripts", "check_slice_hp_replicas.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=850)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "all ok" in out.stdout


def test_cxx_batch_scorer_draws_what_python_draws(ctx, tmp_path):
    exe = str(tmp_path / "slice_hp")
    libdir = os.path.join(ROOT, "common_b200", "csrc")
    subprocess.check_call(["g++", "-std=c++14", "-O1", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cxx", "slice_hp.cpp"),
                           "-L" + libdir, "-lmscope_b200", "-Wl,-rpath," + libdir, "-o", exe])
    N, K = 90, 3
    i = np.arange(N)
    arr = np.zeros(N, dtype=[("f0", np.bool_), ("f1", np.uint32), ("f2", np.float32)])
    arr["f0"] = (i * 7) % 10 < 3 + 2 * (i % K)
    arr["f1"] = (i * 13) % 9 + 3 * (i % K)
    arr["f2"] = ((i % K) + 0.125 * (i % 7)).astype(np.float32)
    hparams = {0: {("alpha", "beta"): (hpr.log_noninformative_beta_prior, 1.0)}, 1: {"inv_beta": (hpr.log_exponential(2.0), 0.5)},
               2: {"mu": (hpr.log_normal(0.5, 2.0), 0.25), "nu": (hpr.log_flat(0.5, 30.0), 2.0)}}
    for seed, counter in [(1, 0), (5, 3), (77, 12345)]:
        st = cb.state(ctx, [cb.bb, cb.gp, cb.nich], max_groups=K + 1, cluster_hp={"alpha": 1.0})
        st.bind(cb.numpy_dataview(arr))
        gids = [st.create_group() for _ in range(K + 1)]                    # the last one stays empty
        st.add_values(np.asarray(gids)[i % K])
        v = st.slice_hp(hparams, {"alpha": (hpr.log_exponential(1.0), 1.0)}, seed=seed, counter=counter)["values"]
        st.close()
        want = [v[0]["alpha"], v[0]["beta"], v[1]["inv_beta"], v[2]["mu"], v[2]["nu"], v["alpha"]]
        out = subprocess.run([exe, str(seed), str(counter)], capture_output=True, text=True, timeout=120)
        assert out.returncode == 0, out.stdout + out.stderr
        assert out.stdout.split() == [str(int(np.float64(x).view(np.uint64))) for x in want]
