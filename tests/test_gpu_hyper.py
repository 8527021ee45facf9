"""GPU: hyperparameter inference on a grid (msb_state_hp_gibbs / state.hp_gibbs).

The weights of every family are held to the fp64 closed forms of the CPU checker summed over the groups, alpha's to the
closed form in numpy; every draw is replayed from the returned weights and the restated Philox uniform, and the draws
follow softmax(logw) in law.  A chain of the exact per-entity Gibbs step followed by hp_gibbs visits partitions, feature
hypers and alpha with the marginals of the enumerated joint posterior.
"""
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import common_b200 as cb
from common_b200.state import flat_hp
from test_gpu_parity import _four_entities, make_state

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HP_TAG = 0x4859505200000000
EVERY = [cb.bb, cb.bnb, cb.gp, cb.nich, cb.dd(9), cb.bbnc, cb.niw(3), cb.dm(12)]
CASES = {"every": EVERY, "niw64": [cb.niw(64), cb.bb]}


def random_point(desc, rng):
    """one hp dict of the family with every value moved away from the default (bnb keeps its r)"""
    d = desc()
    name, p = d.name(), d._param()
    if name in ("bb", "bbnc"):
        return {"alpha": rng.uniform(0.3, 4.0), "beta": rng.uniform(0.3, 4.0)}
    if name == "bnb":
        return {"alpha": rng.uniform(1.5, 5.0), "beta": rng.uniform(0.3, 4.0), "r": 1.0}
    if name == "gp":
        return {"alpha": rng.uniform(0.3, 4.0), "inv_beta": rng.uniform(0.2, 3.0)}
    if name == "nich":
        return {"mu": rng.normal(), "kappa": rng.uniform(0.2, 3.0), "sigmasq": rng.uniform(0.2, 3.0), "nu": rng.uniform(0.5, 5.0)}
    if name in ("dd", "dm"):
        return {"alphas": rng.uniform(0.2, 3.0, p)}
    a = rng.normal(size=(p, p))
    return {"mu": rng.normal(size=p) * 0.3, "kappa": rng.uniform(0.2, 3.0), "psi": a @ a.T / p + np.eye(p) * rng.uniform(0.5, 2.0),
            "nu": p + rng.uniform(0.5, 4.0)}


def philox_u53(oracle, seed, row, counter):
    r = oracle.philox_raw(seed, row, HP_TAG | counter)
    return ((r[0] >> 5) * 67108864.0 + (r[1] >> 6)) / 9007199254740992.0


def replay(w, u):
    """(choice, distance of u from the nearest cumulative boundary) from the weights"""
    w = np.asarray(w, np.float64)
    p = np.exp(w - w.max())
    c = np.cumsum(p)
    return int(np.argmax(c > u * c[-1])), float(np.min(np.abs(c / c[-1] - u)))


def alpha_closed_form(counts, alphas):
    ne, n = int(np.sum(counts > 0)), float(np.sum(counts))
    return np.array([(ne - 1) * math.log(a) + math.lgamma(1 + a) - math.lgamma(n + a) for a in alphas])


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("k", [3, 200, 700])
@pytest.mark.parametrize("G", [1, 7, 33])
def test_weights_agree_with_fp64_and_draws_replay(ctx, oracle, case, k, G):
    descs = CASES[case]
    n = max(1500, 6 * k)
    st, view, z, gids, hp, ss, counts = make_state(ctx, oracle, descs, n, k, seed=k + G, mask_frac=0.05, extra_empty=2)
    rng = np.random.default_rng(G * 1000 + k)
    grids, priors = [], []
    for d, desc in enumerate(descs):
        grids.append([random_point(desc, rng) for _ in range(G)])
        priors.append(rng.normal(size=G))
        st.set_hp_grid(d, grids[d], priors[d])
    alphas, alp = rng.uniform(0.1, 20.0, G), rng.normal(size=G)
    st.set_cluster_hp_grid(alphas, alp)
    seed, counter = 7 + G, 11 + k
    r = st.hp_gibbs(seed=seed, counter=counter, weights=True)
    off = 0
    for d, desc in enumerate(descs):
        m = oracle.model(desc)
        w = oracle.ss_size(m)
        cells = np.array([[oracle.score_data(m, flat_hp(desc(), pt), ss[c, off:off + w]) for c in range(ss.shape[0])]
                          for pt in grids[d]])
        want, scale = cells.sum(axis=1), np.abs(cells).sum(axis=1)
        got = r["logw"][d] - priors[d]
        assert np.all(np.abs(got - want) <= 1e-11 * scale), (desc().name(), np.max(np.abs(got - want) / scale))
        off += w
    assert np.all(np.abs(r["logw"]["alpha"] - alp - alpha_closed_form(counts, alphas)) <=
                  1e-13 * np.maximum(1.0, np.abs(alpha_closed_form(counts, alphas))))
    for key, row in [(d, d) for d in range(len(descs))] + [("alpha", len(descs))]:
        want, dist = replay(r["logw"][key], philox_u53(oracle, seed, row, counter))
        assert dist > 1e-12
        assert r["choice"][key] == want, key
    st.close()


def test_draws_follow_softmax_of_the_weights(ctx, oracle):
    from scipy import stats
    descs = [cb.bb, cb.dd(5), cb.nich, cb.gp]
    st, view, z, gids, hp, ss, counts = make_state(ctx, oracle, descs, 60, 3, seed=3, extra_empty=1)
    rng = np.random.default_rng(1)
    grids = [[random_point(desc, rng) for _ in range(4 + d)] for d, desc in enumerate(descs)]
    alphas = [0.3, 1.0, 3.0, 9.0, 27.0]
    for d in range(len(descs)):
        st.set_hp_grid(d, grids[d])
    st.set_cluster_hp_grid(alphas)
    first = st.hp_gibbs(weights=True)["logw"]
    # priors that flatten the posterior over each grid, up to a random tilt: every point gets a sizeable probability
    for d in range(len(descs)):
        st.set_hp_grid(d, grids[d], -first[d] + rng.uniform(-1, 1, len(grids[d])))
    st.set_cluster_hp_grid(alphas, -first["alpha"] + rng.uniform(-1, 1, len(alphas)))
    logw = st.hp_gibbs(weights=True)["logw"]
    hist = {key: np.zeros(len(w)) for key, w in logw.items()}
    N = 20000
    for counter in range(N):
        for key, c in st.hp_gibbs(seed=5, counter=counter)["choice"].items():
            hist[key][c] += 1
    for key, w in logw.items():
        p = np.exp(w - w.max())
        p /= p.sum()
        assert stats.chisquare(hist[key], p * N).pvalue > 1e-4, (key, hist[key], p * N)
    st.close()


def test_one_point_grids_set_every_family_exactly(ctx, oracle):
    descs = EVERY + [cb.dd(256)]
    st, view, z, gids, hp, ss, counts = make_state(ctx, oracle, descs, 800, 5, seed=2, extra_empty=1)
    rng = np.random.default_rng(3)
    pts = [random_point(desc, rng) for desc in descs]
    for d in range(len(descs)):
        st.set_hp_grid(d, [pts[d]])
    st.set_cluster_hp_grid([2.75])
    r = st.hp_gibbs()
    assert r["choice"] == dict({d: 0 for d in range(len(descs))}, alpha=0)
    for d, desc in enumerate(descs):
        got = st.get_component_hp(d)
        for key in desc().default_hyperparams():
            assert np.array_equal(np.asarray(got[key], np.float64).ravel(), np.asarray(pts[d][key], np.float64).ravel()), (d, key)
    assert st.get_cluster_hp()["alpha"] == 2.75
    st.close()


def _snapshot(st, gids, ncomp):
    ss = [st.get_suffstats(d, g, key, st._ss_counts(st._models[d], key)).tobytes()
          for d in range(ncomp) for g in gids for key in st._SS_KEYS[st._models[d].name()]]
    hps = [{k: np.asarray(v).tobytes() for k, v in st.get_component_hp(d).items()} for d in range(ncomp)]
    return st.assignments().tobytes(), ss, [st.groupsize(g) for g in gids], hps, st.get_cluster_hp()


def test_drawn_hypers_score_like_hypers_set_by_hand(ctx, oracle):
    descs = [cb.dd(256), cb.bb, cb.nich, cb.dd(16), cb.gp, cb.niw(3), cb.bbnc, cb.dm(6)]
    n, k = 2000, 7
    a, _, _, gids, _, _, _ = make_state(ctx, oracle, descs, n, k, seed=4, mask_frac=0.05, extra_empty=1)
    b, _, _, _, _, _, _ = make_state(ctx, oracle, descs, n, k, seed=4, mask_frac=0.05, extra_empty=1)
    a.sweep(seed=1, sweep=0); b.sweep(seed=1, sweep=0)
    rng = np.random.default_rng(8)
    with_grid = [0, 2, 3, 5, 7]
    grids = {d: [random_point(descs[d], rng) for _ in range(9)] for d in with_grid}
    before = _snapshot(a, gids, len(descs))
    for d in with_grid:
        a.set_hp_grid(d, grids[d])
    a.set_cluster_hp_grid([0.5, 2.0, 8.0])
    r = a.hp_gibbs(seed=3, counter=1)
    after = _snapshot(a, gids, len(descs))
    assert after[:3] == before[:3]                           # assignments, suffstats, group sizes
    for d in range(len(descs)):                              # features without a grid keep their hypers
        if d not in with_grid:
            assert after[3][d] == before[3][d]
    for d in with_grid:
        b.set_component_hp(d, grids[d][r["choice"][d]])
    b.set_cluster_hp({"alpha": [0.5, 2.0, 8.0][r["choice"]["alpha"]]})
    _, sa = a.score_rows()
    _, sb = b.score_rows()
    assert np.array_equal(sa.view(np.uint32), sb.view(np.uint32))
    a.sweep(seed=1, sweep=1); b.sweep(seed=1, sweep=1)
    assert np.array_equal(a.assignments(), b.assignments())
    a.close(); b.close()


@pytest.mark.parametrize("niw_points,other_points,k", [(2, 500, 10), (1, 200, 1), (3, 4000, 2)])
def test_small_niw_grid_beside_a_larger_grid(ctx, oracle, niw_points, other_points, k):
    """the niw scratch is sized by the niw grid, not by the largest grid of the state: a few niw points next to a much
    larger alpha or feature grid, few groups"""
    descs = [cb.niw(3), cb.bb]
    st, view, z, gids, hp, ss, counts = make_state(ctx, oracle, descs, 40 * k, k, seed=niw_points + k)
    rng = np.random.default_rng(k)
    niw = [random_point(cb.niw(3), rng) for _ in range(niw_points)]
    st.set_hp_grid(0, niw)
    st.set_hp_grid(1, [random_point(cb.bb, rng) for _ in range(other_points)])
    st.set_cluster_hp_grid(rng.uniform(0.1, 20.0, other_points))
    for counter in range(3):
        r = st.hp_gibbs(seed=2, counter=counter, weights=True)
        m, w = oracle.model(cb.niw(3)), oracle.ss_size(oracle.model(cb.niw(3)))
        cells = np.array([[oracle.score_data(m, flat_hp(cb.niw(3)(), pt), ss[c, :w]) for c in range(ss.shape[0])] for pt in niw])
        assert np.all(np.abs(r["logw"][0] - cells.sum(axis=1)) <= 1e-11 * np.abs(cells).sum(axis=1))
        assert len(r["logw"][1]) == other_points and np.all(np.isfinite(r["logw"][1]))
    st.close()


def test_same_seed_and_counter_give_the_same_bits(ctx, oracle):
    descs = [cb.dd(64), cb.nich, cb.niw(4), cb.bnb]
    st, view, z, gids, hp, ss, counts = make_state(ctx, oracle, descs, 3000, 150, seed=6, extra_empty=3)
    rng = np.random.default_rng(2)
    for d, desc in enumerate(descs):
        st.set_hp_grid(d, [random_point(desc, rng) for _ in range(17)], rng.normal(size=17))
    st.set_cluster_hp_grid(rng.uniform(0.1, 10, 17))
    r1 = st.hp_gibbs(seed=9, counter=4, weights=True)
    r2 = st.hp_gibbs(seed=9, counter=4, weights=True)
    assert r1["choice"] == r2["choice"]
    for key in r1["logw"]:
        assert np.array_equal(r1["logw"][key].view(np.uint64), r2["logw"][key].view(np.uint64)), key
    assert st.hp_gibbs(seed=9, counter=5)["choice"] != r1["choice"] or st.hp_gibbs(seed=10, counter=4)["choice"] != r1["choice"]
    st.close()


def test_gibbs_chain_with_hyper_steps_visits_the_exact_joint_posterior(ctx):
    from math import lgamma
    arr, n, D, _, _, canon = _four_entities()
    data = np.stack([arr["f%d" % d] for d in range(D)], axis=1).astype(int)
    ab = [0.5, 1.0, 2.0]
    ab_prior = np.log([0.2, 0.5, 0.3])
    alphas = [0.5, 1.5, 4.0]
    alpha_prior = np.log([0.3, 0.3, 0.4])

    def lbeta(a, b):
        return lgamma(a) + lgamma(b) - lgamma(a + b)

    def partitions(items):
        if not items:
            yield []
            return
        first, rest = items[0], items[1:]
        for p in partitions(rest):
            for i in range(len(p)):
                yield p[:i] + [[first] + p[i]] + p[i + 1:]
            yield [[first]] + p

    # the joint of (partition, theta_0, theta_1, theta_2, alpha): 15 x 3^3 x 3 states
    joint = {}
    for p in partitions(list(range(n))):
        a = [0] * n
        for gi, g in enumerate(p):
            for e in g:
                a[e] = gi
        key = canon(a)
        for ia, al in enumerate(alphas):
            crp = len(p) * math.log(al) + lgamma(al) - lgamma(n + al) + sum(lgamma(len(g)) for g in p) + alpha_prior[ia]
            for t in np.ndindex(3, 3, 3):
                s = crp
                for d in range(D):
                    c = ab[t[d]]
                    s += ab_prior[t[d]]
                    for g in p:
                        h = int(data[g, d].sum())
                        s += lbeta(c + h, c + len(g) - h) - lbeta(c, c)
                joint[(key, t, ia)] = s
    m = max(joint.values())
    z = sum(math.exp(v - m) for v in joint.values())
    marg_part, marg_feat, marg_alpha = {}, np.zeros((D, 3)), np.zeros(3)
    for (key, t, ia), v in joint.items():
        pr = math.exp(v - m) / z
        marg_part[key] = marg_part.get(key, 0.0) + pr
        for d in range(D):
            marg_feat[d, t[d]] += pr
        marg_alpha[ia] += pr

    st = cb.state(ctx, [cb.bb] * D, max_groups=8, cluster_hp={"alpha": 1.5})
    st.bind(cb.numpy_dataview(arr))
    g0 = st.create_group()
    st.add_values(np.full(n, g0))
    for d in range(D):
        st.set_hp_grid(d, [{"alpha": c, "beta": c} for c in ab], ab_prior)
    st.set_cluster_hp_grid(alphas, alpha_prior)
    rng = np.random.default_rng(0)
    visits, feat, alph = {}, np.zeros((D, 3)), np.zeros(3)
    sweeps, burn = 4000, 100
    for it in range(sweeps):
        for eid in range(n):
            st.remove_value(eid)
            empties = st.empty_groups()
            if not empties:
                st.create_group()
            elif len(empties) > 1:          # keep exactly one empty group, as the reference's assign kernel does
                for g in empties[1:]:
                    st.delete_group(g)
            gids, s = st.score_value(eid)
            p = np.exp(np.asarray(s, np.float64) - np.max(s))
            st.add_value(gids[int(rng.choice(len(gids), p=p / p.sum()))], eid)
        ch = st.hp_gibbs(seed=17, counter=it)["choice"]
        if it >= burn:
            key = canon(st.assignments().tolist())
            visits[key] = visits.get(key, 0) + 1
            for d in range(D):
                feat[d, ch[d]] += 1
            alph[ch["alpha"]] += 1
    st.close()
    total = sweeps - burn
    worst = max(abs(visits.get(k, 0) / total - pk) for k, pk in marg_part.items())
    assert worst < 0.04, ("partition", worst)
    assert np.max(np.abs(feat / total - marg_feat)) < 0.04, (feat / total, marg_feat)
    assert np.max(np.abs(alph / total - marg_alpha)) < 0.04, (alph / total, marg_alpha)


def test_refusals_leave_the_state_untouched(ctx, oracle):
    descs = [cb.bb, cb.bnb, cb.niw(3), cb.nich, cb.gp, cb.dd(4)]
    st, view, z, gids, hp, ss, counts = make_state(ctx, oracle, descs, 600, 4, seed=5)
    rng = np.random.default_rng(4)
    good = [[random_point(desc, rng) for _ in range(3)] for desc in descs]
    for d in range(len(descs)):
        st.set_hp_grid(d, good[d])
    st.set_cluster_hp_grid([0.5, 1.0])
    ref = st.hp_gibbs(seed=1, counter=0, weights=True)
    before = _snapshot(st, gids, len(descs))

    def refused(fn, match):
        with pytest.raises(cb.MsbError, match=match) as e:
            fn()
        assert e.value.status == cb._lib.MSB_ERR_INVALID
        assert _snapshot(st, gids, len(descs)) == before

    lib = cb._lib.load()
    pts = np.ones(3 * 4)
    lp = np.zeros(4)
    P = cb._lib.C.POINTER(cb._lib.C.c_double)
    refused(lambda: cb._lib.check(lib.msb_state_set_hp_grid(st.handle, 0, pts.ctypes.data_as(P), 4, 3, lp.ctypes.data_as(P))),
            "takes 2")                                                               # nhp not the family's
    refused(lambda: st.set_hp_grid(5, [{"alphas": [1.0, 2.0, 3.0]}]), "takes 4")
    refused(lambda: st.set_hp_grid(0, [{"alpha": np.nan, "beta": 1.0}]), "non-finite")
    refused(lambda: st.set_hp_grid(0, [{"alpha": 1.0, "beta": 1.0}], [np.inf]), "non-finite")
    refused(lambda: st.set_cluster_hp_grid([1.0, 0.0]), "positive")
    refused(lambda: st.set_cluster_hp_grid([1.0, -2.0]), "positive")
    refused(lambda: st.set_hp_grid(1, [{"alpha": 2.0, "beta": 1.0, "r": 1.0}, {"alpha": 2.0, "beta": 1.0, "r": 3.0}]),
            "bnb grid point 1 changes r")
    refused(lambda: st.hp_gibbs(counter=1 << 32), "below 2")
    refused(lambda: st.set_hp_grid(0, [{"alpha": 1.0, "beta": 1.0}] * 65536), "at most 65535")
    refused(lambda: st.set_cluster_hp_grid(np.ones(65536)), "at most 65535")
    with pytest.raises(ValueError, match="one log prior per grid point"):
        st.set_hp_grid(0, good[0], [0.0])
    assert _snapshot(st, gids, len(descs)) == before
    # the grids registered before the refusals are still the ones used
    again = st.hp_gibbs(seed=1, counter=0, weights=True)
    assert all(np.array_equal(again["logw"][key], ref["logw"][key]) for key in ref["logw"])
    st.set_hp_grid(0, good[0])
    st.set_hp_grid(1, good[1])
    st.set_cluster_hp_grid([0.5, 1.0])
    bad_psi = dict(good[2][1], psi=np.diag([1.0, -1.0, 1.0]))
    st.set_hp_grid(2, [good[2][0], bad_psi])
    refused(lambda: st.hp_gibbs(), "feature 2: grid point 1 has a NaN weight")
    st.set_hp_grid(2, good[2])
    st.set_hp_grid(3, [good[3][0], dict(good[3][0], kappa=-1.0)])
    refused(lambda: st.hp_gibbs(), "feature 3: grid point 1 has a NaN weight")
    st.set_hp_grid(3, good[3])
    st.set_hp_grid(4, [{"alpha": 1.0, "inv_beta": 0.0}, {"alpha": 2.0, "inv_beta": 0.0}])   # every group holds rows
    refused(lambda: st.hp_gibbs(), "feature 4: every grid point has weight -inf")
    st.set_hp_grid(4, None)
    st.set_component_hp(1, dict(good[1][0], r=2.0))                                  # r moved after the grid was set
    before = _snapshot(st, gids, len(descs))
    refused(lambda: st.hp_gibbs(), "changes r")
    st.close()


def test_two_ranks_draw_identical_hypers():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    port = 29500 + os.getpid() % 200
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "scripts", "check_hp_replicas.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=850)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "all ok" in out.stdout


def test_cxx_batch_scorer_draws_what_python_draws(ctx, tmp_path):
    exe = str(tmp_path / "hp_gibbs")
    libdir = os.path.join(ROOT, "common_b200", "csrc")
    subprocess.check_call(["g++", "-std=c++14", "-O1", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cxx", "hp_gibbs.cpp"),
                           "-L" + libdir, "-lmscope_b200", "-Wl,-rpath," + libdir, "-o", exe])
    N, K = 90, 3
    i = np.arange(N)
    arr = np.zeros(N, dtype=[("f0", np.bool_), ("f1", np.uint32), ("f2", np.float32)])
    arr["f0"] = (i * 7) % 10 < 3 + 2 * (i % K)
    arr["f1"] = (i * 13) % 9 + 3 * (i % K)
    arr["f2"] = ((i % K) + 0.125 * (i % 7)).astype(np.float32)
    st = cb.state(ctx, [cb.bb, cb.gp, cb.nich], max_groups=K + 1, cluster_hp={"alpha": 1.0})
    st.bind(cb.numpy_dataview(arr))
    gids = [st.create_group() for _ in range(K)]
    st.add_values(np.asarray(gids)[i % K])
    st.set_hp_grid(0, [{"alpha": 0.5, "beta": 0.5}, {"alpha": 1.0, "beta": 1.0}, {"alpha": 2.0, "beta": 3.0}], [0.0, -0.5, -1.0])
    st.set_hp_grid(1, [{"alpha": 1.0, "inv_beta": 1.0}, {"alpha": 2.0, "inv_beta": 0.5}, {"alpha": 4.0, "inv_beta": 1.0},
                       {"alpha": 0.5, "inv_beta": 2.0}], [0.0, 0.0, -0.25, 0.1])
    st.set_hp_grid(2, [{"mu": 0.0, "kappa": 1.0, "sigmasq": 1.0, "nu": 1.0}, {"mu": 1.0, "kappa": 0.5, "sigmasq": 2.0, "nu": 3.0}],
                   [0.0, 0.0])
    st.set_cluster_hp_grid([0.25, 1.0, 4.0, 16.0], [0.0, 0.0, 0.0, -2.0])
    for seed, counter in [(1, 0), (5, 3), (77, 12345)]:
        out = subprocess.run([exe, str(seed), str(counter)], capture_output=True, text=True, timeout=120)
        assert out.returncode == 0, out.stdout + out.stderr
        c = st.hp_gibbs(seed=seed, counter=counter)["choice"]
        assert [int(x) for x in out.stdout.split()] == [c[0], c[1], c[2], c["alpha"]]
    st.close()
