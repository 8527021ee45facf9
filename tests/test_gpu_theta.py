"""GPU: non-conjugate parameters on the device (msb_state_theta / state.theta, msb_state_redraw_empty / state.redraw_empty).

Every slice update and every Beta draw is replayed in fp64 from the restated Philox stream; the chained updates follow
the conjugate posterior Beta(alpha + heads, beta + tails) and the fresh draws the prior, by KS.  The state a call leaves
scores like the same p set by hand, and the sequential chain with redraw_empty and theta (Neal's algorithm 8, m = 1)
visits the partitions of four entities with bb's exact posterior.
"""
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import common_b200 as cb
import oracle_lib as ol
from test_gpu_parity import _four_entities, check, make_state

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THETA_TAG = 0x534c494300000000
AUX_TAG = 0x4155585000000000
SHRINK_CAP, STEP_CAP = 200, 1 << 20
NEAR = 1e-9     # a decision this close to its boundary may go either way under a last-ulp difference of log / lgamma


class Stream(object):
    """DrawStream of msb_draw.cuh: block b = philox4x32_10(seed, counter << 32 | gid, tag | feature << 16 | b)"""

    def __init__(self, oracle, seed, gid, feature, counter, tag):
        self.o, self.seed, self.idx, self.tag = oracle, seed, (counter << 32) | gid, tag | (feature << 16)
        self.blk, self.buf = 0, []

    def next(self):
        if not self.buf:
            self.buf = self.o.philox_raw(self.seed, self.idx, self.tag | self.blk)
            self.blk += 1
        return self.buf.pop(0)

    def u53(self):
        a = self.next() >> 5
        b = self.next() >> 6
        return (a * 67108864.0 + b) * (1.0 / 9007199254740992.0)

    def u_open(self):
        a = self.next() >> 6
        b = self.next() >> 6
        return (a * 67108864.0 + b + 0.5) * (1.0 / 4503599627370496.0)

    def normal(self):
        u1 = self.u53()
        u2 = self.u53()
        return math.sqrt(-2.0 * math.log1p(-u1)) * math.cos(6.283185307179586 * u2)

    def gamma(self, k):
        """(draw, smallest distance of an accept test from its boundary)"""
        boost, near = 1.0, math.inf
        if k < 1.0:
            boost = math.pow(1.0 - self.u53(), 1.0 / k)
            k += 1.0
        d = k - 1.0 / 3.0
        c = 1.0 / math.sqrt(9.0 * d)
        for _ in range(1000):
            z = self.normal()
            v = 1.0 + c * z
            if v <= 0.0:
                continue
            v = v * v * v
            u = 1.0 - self.u53()
            lhs, rhs = math.log(u), 0.5 * z * z + d - d * v + d * math.log(v)
            near = min(near, abs(lhs - rhs))
            if lhs < rhs:
                return boost * d * v, near
        return boost * d, near


def target(a, b, p, heads, tails):
    """bbnc's score_data (bbnc.cpp:61-73) at p, as score_data_cell evaluates it"""
    if p < 0.0 or p > 1.0:
        return -math.inf
    with np.errstate(all="ignore"):
        lp, l1p = np.log(np.float64(p)), np.log1p(-np.float64(p))
        lb = math.lgamma(a) + math.lgamma(b) - math.lgamma(a + b)
        return float((a - 1.0) * lp + (b - 1.0) * l1p - lb + heads * lp + tails * l1p)


def slice_replay(oracle, seed, counter, feature, gid, a, b, w, p0, heads, tails):
    """(new p, smallest |f - y| over the decisions taken, capped)"""
    f = lambda p: target(a, b, p, heads, tails)                                   # noqa: E731
    rs = Stream(oracle, seed, gid, feature, counter, THETA_TAG)
    y = f(p0) + math.log(rs.u_open())
    near = math.inf

    def above(x):
        nonlocal near
        v = f(x)
        if math.isfinite(v):
            near = min(near, abs(v - y))
        return v > y

    L = p0 - w * rs.u53()
    R = L + w
    n = 0
    while n <= STEP_CAP and above(L):
        L -= w
        n += 1
    m = 0
    while m <= STEP_CAP and above(R):
        R += w
        m += 1
    if n > STEP_CAP or m > STEP_CAP:
        return p0, near, True
    for _ in range(SHRINK_CAP):
        x = L + rs.u53() * (R - L)
        if above(x):
            return x, near, False
        if x < p0:
            L = x
        else:
            R = x
    return p0, near, True


def beta_replay(oracle, seed, counter, feature, gid, a, b):
    rs = Stream(oracle, seed, gid, feature, counter, AUX_TAG)
    x, n1 = rs.gamma(a)
    y, n2 = rs.gamma(b)
    return x / (x + y), min(n1, n2)


def get_p(st, d, gids):
    return np.array([st.get_suffstats(d, g, "p")[0] for g in gids])


def snapshot(st, gids, ncomp):
    """({(feature, gid, key): suffstat bits}, assignment bits)"""
    ss = {(d, g, key): st.get_suffstats(d, g, key, st._ss_counts(st._models[d], key)).tobytes()
          for d in range(ncomp) for g in gids for key in st._SS_KEYS[st._models[d].name()]}
    return ss, st.assignments().tobytes()


# (alpha, beta, width) per feature: widths from 0.01 to 5
REPLAY = [(1.0, 1.0, 0.01), (0.5, 2.0, 0.1), (3.0, 0.7, 0.5), (2.0, 5.0, 1.0), (1.5, 1.5, 5.0), (0.8, 0.8, 2.0), (4.0, 4.0, 0.05)]


def test_slice_updates_and_beta_draws_replay(ctx, oracle):
    K, D = 200, len(REPLAY)
    st = cb.state(ctx, [cb.bbnc] * D, max_groups=K + 4, cluster_hp={"alpha": 1.0})
    for d, (a, b, _) in enumerate(REPLAY):
        st.set_component_hp(d, {"alpha": a, "beta": b})
    gids = [st.create_group() for _ in range(K)]
    rng = np.random.default_rng(11)
    ht = {}
    for d in range(D):
        for c, g in enumerate(gids):
            heads, tails = (1e6, 3.0) if c == 0 else tuple(float(rng.integers(0, 10 ** rng.integers(0, 5))) for _ in range(2))
            ht[d, c] = heads, tails
            st.set_suffstats(d, g, "heads", heads)
            st.set_suffstats(d, g, "tails", tails)
            if c % 3 == 1:
                st.set_suffstats(d, g, "p", rng.uniform(0.02, 0.98))
    seed, counter = 1234, 5
    p0 = np.stack([get_p(st, d, gids) for d in range(D)])
    capped = st.theta({d: {"p": w} for d, (_, _, w) in enumerate(REPLAY)}, seed=seed, counter=counter)
    assert capped == 0
    p1 = np.stack([get_p(st, d, gids) for d in range(D)])
    near = 0
    for d, (a, b, w) in enumerate(REPLAY):
        for c, g in enumerate(gids):
            want, dist, cap = slice_replay(oracle, seed, counter, d, g, a, b, w, p0[d, c], *ht[d, c])
            assert not cap
            if dist < NEAR:
                near += 1
                continue
            assert abs(p1[d, c] - want) <= 1e-12 * abs(want), (d, c, p1[d, c], want)
    print("slice replay: %d of %d updates had a decision within %g of its boundary" % (near, K * D, NEAR))
    assert near <= 3
    assert np.all(p1 != p0)                          # every update moved (a shrink step lands on p0 with probability 0)
    assert np.all((p1 > 0) & (p1 < 1))
    # every group is empty: redraw_empty draws all of them
    st.redraw_empty(seed=seed, counter=counter + 1)
    p2 = np.stack([get_p(st, d, gids) for d in range(D)])
    near = 0
    for d, (a, b, _) in enumerate(REPLAY):
        for c, g in enumerate(gids):
            want, dist = beta_replay(oracle, seed, counter + 1, d, g, a, b)
            if dist < NEAR:
                near += 1
                continue
            assert abs(p2[d, c] - want) <= 1e-12 * max(abs(want), 1e-300), (d, c, p2[d, c], want)
    print("beta replay: %d of %d draws had an accept test within %g of its boundary" % (near, K * D, NEAR))
    assert near <= 3
    st.close()


@pytest.mark.parametrize("a,b,heads,tails,w", [(1.0, 1.0, 3, 7, 0.5),          # moderate
                                               (2.0, 2.0, 5000, 3000, 5.0),    # narrow posterior, wide width
                                               (0.7, 0.9, 0, 1, 0.01),         # wide posterior, tiny width
                                               (0.5, 3.0, 40, 0, 1.0)])        # mass at the edge p -> 1
def test_chained_updates_follow_the_conjugate_posterior(ctx, a, b, heads, tails, w):
    from scipy import stats
    K = 512
    st = cb.state(ctx, [cb.bbnc, cb.bb], max_groups=K, cluster_hp={"alpha": 1.0})
    st.set_component_hp(0, {"alpha": a, "beta": b})
    gids = [st.create_group() for _ in range(K)]
    for g in gids:
        st.set_suffstats(0, g, "heads", heads)
        st.set_suffstats(0, g, "tails", tails)
    for i in range(30):
        assert st.theta({0: {"p": w}}, seed=77, counter=i) == 0
    p = get_p(st, 0, gids)
    r = stats.kstest(p, stats.beta(a + heads, b + tails).cdf)
    print("theta law a=%g b=%g heads=%d tails=%d w=%g: KS p-value %.3g" % (a, b, heads, tails, w, r.pvalue))
    assert r.pvalue > 1e-3
    st.close()


@pytest.mark.parametrize("a,b", [(1.0, 1.0), (0.4, 2.5), (6.0, 0.8)])
def test_fresh_draws_follow_the_prior(ctx, a, b):
    from scipy import stats
    K = 600
    st = cb.state(ctx, [cb.bb, cb.bbnc], max_groups=K, cluster_hp={"alpha": 1.0})
    st.set_component_hp(1, {"alpha": a, "beta": b})
    gids = [st.create_group() for _ in range(K)]
    st.redraw_empty(seed=3, counter=9)
    p = get_p(st, 1, gids)
    r = stats.kstest(p, stats.beta(a, b).cdf)
    print("redraw_empty law a=%g b=%g: KS p-value %.3g" % (a, b, r.pvalue))
    assert r.pvalue > 1e-3
    st.close()


def test_the_state_after_theta_and_redraw_scores_like_p_set_by_hand(ctx, oracle):
    descs = [cb.bbnc, cb.bb, cb.bbnc, cb.nich, cb.bbnc]
    n, k = 2000, 9
    st, view, z, gids, hp, ss, counts = make_state(ctx, oracle, descs, n, k, seed=8, mask_frac=0.05, extra_empty=2,
                                                   hp={0: {"alpha": 2.0, "beta": 3.0}, 2: {"alpha": 0.6, "beta": 0.6}})
    ncomp = len(descs)
    offs = np.cumsum([0] + [oracle.ss_size(oracle.model(d)) for d in descs])
    hoffs = np.cumsum([0] + [oracle.hp_size(oracle.model(d)) for d in descs])
    before, assign = snapshot(st, gids, ncomp)
    assert st.theta({0: {"p": 0.3}, 2: {"p": 1.0}, 4: {"p": 0.0}}, seed=5, counter=1) == 0
    after, assign2 = snapshot(st, gids, ncomp)
    assert assign2 == assign
    # only p of the features with a width moved; heads / tails, width-0 and other features keep their bits
    assert {key for key in before if before[key] != after[key]} == {(d, g, "p") for d in (0, 2) for g in gids}
    for d in (0, 2):
        p = get_p(st, d, gids)
        ss[:, offs[d]] = p
        m = oracle.model(descs[d])
        for c, g in enumerate(gids):
            want = oracle.score_data(m, hp[hoffs[d]:hoffs[d + 1]], ss[c, offs[d]:offs[d + 1]])
            assert abs(st.score_likelihood(d, g) - want) <= 2e-6 * max(1.0, abs(want)), (d, c)
    _, S = st.score_rows()
    check(S, oracle.score_rows(descs, hp, ss, ol.logprior(counts, 1.0), view))
    # redraw_empty: only the empty groups' p change
    empty = set(st.empty_groups())
    assert len(empty) == 2
    mid, _ = snapshot(st, gids, ncomp)
    st.redraw_empty(seed=5, counter=2)
    end, _ = snapshot(st, gids, ncomp)
    assert {key for key in mid if mid[key] != end[key]} == {(d, g, "p") for d in (0, 2, 4) for g in empty}
    st.close()


def _bbnc_chain(ctx, sweeps, with_theta, seed=0):
    arr, n, D, alpha, exact, canon = _four_entities()
    st = cb.state(ctx, [cb.bbnc] * D, max_groups=8, cluster_hp={"alpha": alpha})
    for d in range(D):
        st.set_component_hp(d, {"alpha": 1.0, "beta": 1.0})
    st.bind(cb.numpy_dataview(arr))
    g0 = st.create_group()
    st.add_values(np.full(n, g0))
    rng = np.random.default_rng(seed)
    visits, burn, step = {}, 100, 0
    for it in range(sweeps):
        for eid in range(n):
            old = st.remove_value(eid)
            empties = st.empty_groups()
            if st.groupsize(old) == 0:          # a singleton: its group, with its p, is the auxiliary component
                for g in empties:
                    if g != old:
                        st.delete_group(g)
            else:                               # one auxiliary component with p fresh from the prior
                if not empties:
                    st.create_group()
                for g in empties[1:]:
                    st.delete_group(g)
                st.redraw_empty(seed=seed + 1, counter=step)
            step += 1
            gids, s = st.score_value(eid)       # log alpha + log p / log(1 - p) for the auxiliary group (m = 1)
            p = np.exp(np.asarray(s, np.float64) - np.max(s))
            st.add_value(gids[int(rng.choice(len(gids), p=p / p.sum()))], eid)
        if with_theta:
            assert st.theta({d: {"p": 0.5} for d in range(D)}, seed=seed + 2, counter=it) == 0
        if it >= burn:
            key = canon(st.assignments().tolist())
            visits[key] = visits.get(key, 0) + 1
    st.close()
    total = sum(visits.values())
    return max(abs(visits.get(k, 0) / total - pk) for k, pk in exact.items())


def test_algorithm8_chain_with_theta_visits_the_exact_posterior(ctx):
    """integrating p out of bbnc at alpha = beta = 1 gives bb's partition posterior: the chain of remove_value,
    redraw_empty (Neal's algorithm 8 with m = 1), score_value, draw, add_value, and theta after each sweep must visit it"""
    worst = _bbnc_chain(ctx, 3000, True)
    frozen = _bbnc_chain(ctx, 1500, False)
    print("algorithm 8 + theta: largest deviation from the exact posterior %.4f; without theta (p frozen at its draw): %.4f"
          % (worst, frozen))
    assert worst < 0.04, worst


def test_same_seed_and_counter_give_the_same_bits(ctx, oracle):
    descs = [cb.bbnc, cb.bbnc, cb.bb]
    a = make_state(ctx, oracle, descs, 3000, 40, seed=6, extra_empty=3)
    b = make_state(ctx, oracle, descs, 3000, 40, seed=6, extra_empty=3)
    gids = a[3]
    for st in (a[0], b[0]):
        st.redraw_empty(seed=9, counter=4)
        st.theta({0: {"p": 0.2}, 1: {"p": 2.0}}, seed=9, counter=4)
    pa = [get_p(a[0], d, gids) for d in (0, 1)]
    pb = [get_p(b[0], d, gids) for d in (0, 1)]
    assert all(np.array_equal(x.view(np.uint64), y.view(np.uint64)) for x, y in zip(pa, pb))
    a[0].theta({0: {"p": 0.2}, 1: {"p": 2.0}}, seed=9, counter=5)
    b[0].theta({0: {"p": 0.2}, 1: {"p": 2.0}}, seed=10, counter=4)
    qa = [get_p(a[0], d, gids) for d in (0, 1)]
    qb = [get_p(b[0], d, gids) for d in (0, 1)]
    for d in range(2):
        assert np.all(qa[d] != qb[d])
    a[0].close(); b[0].close()


def test_refusals_leave_the_state_untouched(ctx, oracle):
    descs = [cb.bbnc, cb.bb, cb.bbnc]
    st, view, z, gids, hp, ss, counts = make_state(ctx, oracle, descs, 600, 4, seed=5, extra_empty=1)

    def state_bits():
        _, S = st.score_rows(0, 1)
        return snapshot(st, gids, len(descs)), S.tobytes()

    before = state_bits()

    def refused(fn, match):
        with pytest.raises(cb.MsbError, match=match) as e:
            fn()
        assert e.value.status == cb._lib.MSB_ERR_INVALID
        assert state_bits() == before

    lib = cb._lib.load()
    refused(lambda: st.theta({0: {"p": -0.5}}), "feature 0: the slice width must be finite and non-negative")
    refused(lambda: st.theta({2: {"p": np.nan}}), "feature 2: the slice width must be finite")
    refused(lambda: st.theta({2: {"p": np.inf}}), "feature 2: the slice width must be finite")
    refused(lambda: st.theta({0: {"p": 0.5}, 1: {"p": 0.5}}), "feature 1: bb has no non-conjugate parameter")
    refused(lambda: st.theta({0: {"p": 0.5}}, counter=1 << 32), "below 2")
    refused(lambda: st.redraw_empty(counter=1 << 32), "below 2")
    w = np.full(2, 0.5)
    opts = cb._lib.ThetaOpts(0, 0, w.ctypes.data, 2)
    refused(lambda: cb._lib.check(lib.msb_state_theta(st.handle, cb._lib.C.byref(opts), None)), "2 widths for a state of 3 features")
    with pytest.raises(ValueError, match="no non-conjugate parameter 'q'"):
        st.theta({0: {"q": 0.5}})
    st.set_suffstats(0, gids[0], "heads", 5.0)
    st.set_suffstats(0, gids[0], "p", 0.0)                 # heads > 0: score_data is -inf at p = 0
    before = state_bits()
    refused(lambda: st.theta({0: {"p": 0.5}}), "feature 0: gid %d: the current p has a non-finite score_data" % gids[0])
    st.set_suffstats(0, gids[0], "p", 0.5)
    st.set_suffstats(2, gids[1], "p", 1.0)
    st.set_suffstats(2, gids[1], "tails", 3.0)
    before = state_bits()
    refused(lambda: st.theta({0: {"p": 0.5}, 2: {"p": 0.5}}), "feature 2: gid %d: the current p" % gids[1])
    st.set_suffstats(2, gids[1], "p", 0.5)
    assert cb._lib.load().msb_state_restore_group(st.handle, 1 << 32) == 0
    before = state_bits()
    refused(lambda: st.theta({0: {"p": 0.5}}), "gid 4294967296 does not fit the stream packing")
    refused(lambda: st.redraw_empty(), "gid 4294967296 does not fit the stream packing")
    st.delete_group(1 << 32)
    assert st.theta({0: {"p": 0.5}, 2: {"p": 0.5}}) == 0
    st.close()
    plain = cb.state(ctx, [cb.bb, cb.nich], max_groups=4, cluster_hp={"alpha": 1.0})
    plain.create_group()
    plain.redraw_empty(seed=1, counter=2)                  # no bbnc feature: nothing to do
    assert plain.theta({}) == 0
    plain.close()


def test_two_ranks_draw_identical_p():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    port = 29700 + os.getpid() % 200
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "scripts", "check_theta_replicas.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=850)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "all ok" in out.stdout


def test_cxx_batch_scorer_draws_what_python_draws(ctx, tmp_path):
    exe = str(tmp_path / "theta")
    libdir = os.path.join(ROOT, "common_b200", "csrc")
    subprocess.check_call(["g++", "-std=c++14", "-O1", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cxx", "theta.cpp"),
                           "-L" + libdir, "-lmscope_b200", "-Wl,-rpath," + libdir, "-o", exe])
    N, K = 90, 3
    i = np.arange(N)
    arr = np.zeros(N, dtype=[("f0", np.bool_), ("f1", np.bool_), ("f2", np.bool_)])
    arr["f0"] = (i * 7) % 10 < 3 + 2 * (i % K)
    arr["f1"] = (i * 13) % 9 < 2 + 3 * (i % K)
    arr["f2"] = (i * 5) % 11 < 4
    for seed, counter in [(1, 0), (5, 3), (77, 12345)]:
        st = cb.state(ctx, [cb.bbnc, cb.bb, cb.bbnc], max_groups=K + 2, cluster_hp={"alpha": 1.0})
        st.set_component_hp(0, {"alpha": 2.0, "beta": 0.5})
        st.bind(cb.numpy_dataview(arr))
        gids = [st.create_group() for _ in range(K + 1)]       # the last one stays empty
        st.add_values(np.asarray(gids)[i % K])
        st.redraw_empty(seed=seed, counter=counter)
        st.theta({0: {"p": 0.25}, 2: {"p": 1.5}}, seed=seed, counter=counter + 1)
        want = [str(int(st.get_suffstats(d, g, "p").view(np.uint64)[0])) for d in (0, 2) for g in gids]
        st.close()
        out = subprocess.run([exe, str(seed), str(counter)], capture_output=True, text=True, timeout=120)
        assert out.returncode == 0, out.stdout + out.stderr
        assert out.stdout.split() == want
