"""GPU: the posterior predictive of rows (msb_state_predict / state.predict).

The log predictive density, the responsibilities and the MAP group are restated in numpy from the GPU's own score bits
(the sampler's exp, a sequential fp64 sum, a float32 division) and must agree bit for bit (logp to 1e-14); logp is also
held to the fp64 closed forms.  The group draw is the sweep's, and every imputed cell is the draw the single-group call
makes for the same counter.
"""
import numpy as np
import numpy.ma as ma
import pytest

import common_b200 as cb
import oracle_lib as ol
from test_gpu_parity import make_state

pytestmark = pytest.mark.gpu

EVERY = [cb.bb, cb.bnb, cb.gp, cb.nich, cb.dd(9), cb.bbnc, cb.niw(3), cb.dm(4)]
CASES = {
    "every": (EVERY, 0.0),
    "mixed-masked": ([cb.bb, cb.gp, cb.nich, cb.dd(16), cb.bb, cb.nich, cb.bnb, cb.bbnc], 0.05),
    "niw64+scalars": ([cb.niw(64), cb.bb, cb.nich, cb.dd(16)], 0.0),
    "dm+scalars": ([cb.dm(12), cb.bb, cb.nich, cb.dd(16), cb.gp], 0.0),
}


def pseudocounts(counts, alpha=1.0):
    counts = np.asarray(counts, np.float64)
    nempty = int((counts == 0).sum())
    return np.where(counts != 0, counts.astype(np.float32), np.float32(alpha) / np.float32(max(nempty, 1))).astype(np.float32)


def restate(orc, S, counts):
    """numpy restatement of msb_state_predict from fp32 scores S[n, K]: (logp, resp, map column)"""
    m = S.max(axis=1)
    x = (S - m[:, None]).astype(np.float32)
    p = np.zeros_like(x)
    live = ~(x < -104.0)
    p[live] = np.frompyfunc(orc.expf, 1, 1)(x[live]).astype(np.float32)
    acc = np.cumsum(p.astype(np.float64), axis=1)[:, -1]          # sequential, column order
    resp = p / acc.astype(np.float32)[:, None]                      # float32 division
    logz = np.log(pseudocounts(counts).astype(np.float64).sum())
    logp = m.astype(np.float64) + np.log(acc) - logz
    return logp, resp.astype(np.float32), np.argmax(S == m[:, None], axis=1)


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("k", [3, 200, 390, 700])
def test_exact_given_the_gpus_score_bits_and_accurate_against_fp64(ctx, oracle, case, k):
    descs, mask_frac = CASES[case]
    n, lo = 1500, 37
    st, view, z, gids, hp, ss, counts = make_state(ctx, oracle, descs, n, k, seed=11, mask_frac=mask_frac, extra_empty=1)
    seed, counter = 91, 4
    r = st.predict(lo, n, responsibilities=True, map=True, draw=True, seed=seed, counter=counter)
    assert r["gids"] == gids
    S = st.read_last_scores()
    assert S.shape == (n - lo, k + 1)
    logp, resp, mcol = restate(oracle, S, counts)
    assert np.array_equal(r["resp"].view(np.uint32), resp.view(np.uint32))
    assert np.array_equal(r["map_gid"], np.asarray(gids)[mcol])
    assert np.max(np.abs(r["logp"] - logp) / np.maximum(1.0, np.abs(logp))) < 1e-14
    u = oracle.philox_u01_rows(seed, lo, n - lo, counter)
    assert np.array_equal(r["draw_gid"], np.asarray(gids)[oracle.sample_rows(S, u)])
    # against the fp64 closed forms: the logsumexp's error is bounded by the largest score error
    S64 = oracle.score_rows(descs, hp, ss, ol.logprior(counts, 1.0), view, lo, n)
    mx = S64.max(axis=1)
    want = mx + np.log(np.exp(S64 - mx[:, None]).sum(axis=1)) - np.log(pseudocounts(counts).astype(np.float64).sum())
    assert np.all(np.abs(r["logp"] - want) <= 1e-5 * np.maximum(1.0, np.abs(S64).max(axis=1)))
    st.close()


def _dd_bb_state(ctx, n_empty, with_masked_row=False):
    """dd(5) x bb: 300 training rows in 3 groups, then every one of the 10 value combinations bound unassigned"""
    rng = np.random.default_rng(5)
    ntr = 300
    z = np.arange(ntr) % 3
    theta = np.array([[.6, .2, .1, .05, .05], [.05, .05, .1, .2, .6], [.2, .2, .2, .2, .2]])
    dd = np.array([rng.choice(5, p=theta[g]) for g in z])
    bb = rng.random(ntr) < np.array([.9, .2, .5])[z]
    combos = [(c, b) for c in range(5) for b in (False, True)]
    rows = list(zip(dd, bb)) + combos + ([(0, False)] if with_masked_row else [])
    arr = np.zeros(len(rows), dtype=[("f0", np.int32), ("f1", np.bool_)])
    arr["f0"] = [r[0] for r in rows]
    arr["f1"] = [r[1] for r in rows]
    if with_masked_row:
        mask = np.zeros(len(rows), dtype=[("f0", np.bool_), ("f1", np.bool_)])
        mask[-1] = (True, True)
        arr = ma.array(arr, mask=mask)
    st = cb.state(ctx, [cb.dd(5), cb.bb], max_groups=8, cluster_hp={"alpha": 1.5})
    st.bind(cb.numpy_dataview(arr))
    gids = [st.create_group() for _ in range(3 + n_empty)]
    st.add_values(np.concatenate([np.asarray(gids)[z], -np.ones(len(rows) - ntr, np.int64)]))
    return st, ntr


@pytest.mark.parametrize("n_empty", [0, 1, 3])
def test_predictive_densities_of_every_value_sum_to_one(ctx, n_empty):
    st, ntr = _dd_bb_state(ctx, n_empty, with_masked_row=True)
    r = st.predict(ntr, ntr + 10, responsibilities=True)
    assert abs(np.exp(r["logp"]).sum() - 1.0) < 1e-5
    # a fully masked row: p(nothing observed) = 1, and the responsibilities are the CRP weights pc / Z
    m = st.predict(ntr + 10, ntr + 11, responsibilities=True)
    assert abs(m["logp"][0]) < 1e-6
    pc = pseudocounts([st.groupsize(g) for g in m["gids"]], 1.5).astype(np.float64)
    assert np.max(np.abs(m["resp"][0] - pc / pc.sum())) < 1e-6
    st.close()


def test_chunks_and_sub_ranges_do_not_change_the_results(ctx, oracle, monkeypatch):
    descs = [cb.bb, cb.gp, cb.nich, cb.dd(16), cb.niw(3), cb.bbnc]
    n, k = 3500, 200
    st, view, z, gids, hp, ss, counts = make_state(ctx, oracle, descs, n, k, seed=4, mask_frac=0.1, extra_empty=2)
    kw = dict(responsibilities=True, map=True, draw=True, impute=True, seed=3, counter=2)
    full = st.predict(**kw)
    monkeypatch.setenv("MSB_SCORES_MB", "1")         # 1 MB of scores: 1024-row chunks
    chunked = st.predict(**kw)
    monkeypatch.delenv("MSB_SCORES_MB")
    sub = st.predict(1000, 2500, **kw)
    for key in ("logp", "resp", "map_gid", "draw_gid"):
        assert np.array_equal(full[key], chunked[key]), key
        assert np.array_equal(full[key][1000:2500], sub[key]), key
    for d in range(len(descs)):
        assert np.array_equal(full["values"][d], chunked["values"][d], equal_nan=True)
        assert np.array_equal(full["values"][d][1000:2500], sub["values"][d], equal_nan=True)
    st.close()


def test_imputation_draws_what_the_single_group_calls_draw(ctx, oracle):
    descs = [cb.bb, cb.bnb, cb.gp, cb.nich, cb.dd(9), cb.bbnc, cb.niw(3)]
    n, k, D = 400, 4, 7
    st, view, z, gids, hp, ss, counts = make_state(ctx, oracle, descs, n, k, seed=8, mask_frac=0.1, extra_empty=2)
    seed, counter = 17, 3
    r = st.predict(draw=True, impute=True, seed=seed, counter=counter)
    arr = view._data
    mask = view._mask
    col = np.searchsorted(gids, r["draw_gid"])
    off = hoff = 0
    nmasked = 0
    for d, desc in enumerate(descs):
        m = oracle.model(desc)
        w, hw = oracle.ss_size(m), oracle.hp_size(m)
        name = desc().name()
        exact = name in ("bb", "bbnc", "dd", "gp", "bnb")
        got = r["values"][d]
        for row in range(n):
            cell_masked = bool(np.any(mask["f%d" % d][row]))
            if not cell_masked:
                want = np.asarray(arr["f%d" % d][row], np.float32 if name in ("nich", "niw") else np.float64)
                assert np.array_equal(np.asarray(got[row], np.float64), want.astype(np.float64)), (name, row)
                continue
            nmasked += 1
            c = int(col[row])
            ctr = (counter << 40) + row * D + d
            want = oracle.sample_value(m, hp[hoff:hoff + hw], ss[c, off:off + w], seed, ctr, 1)[0]
            dev = st.sample_value(d, gids[c], seed=seed, counter=ctr, n=1)[0]
            g = np.asarray(got[row], np.float64)
            if exact:
                assert g == want and g == dev, (name, row)
            else:
                assert np.max(np.abs(g - want) / np.maximum(1.0, np.abs(want))) < 1e-9, (name, row)
                assert np.max(np.abs(g - dev) / np.maximum(1.0, np.abs(dev))) < 1e-12, (name, row)
        off += w; hoff += hw
    assert nmasked > 150
    assert set(np.unique(r["draw_gid"])) > set(gids[:1])      # rows are drawn into several groups
    st.close()


def test_dm_imputation_is_unsupported_as_upstream(ctx, oracle):
    descs = [cb.dm(6), cb.bb, cb.nich]
    st, view, z, gids, hp, ss, counts = make_state(ctx, oracle, descs, 300, 3, seed=2, mask_frac=0.1)
    with pytest.raises(cb.MsbError, match="multinomial sampling unimplemented"):
        st.predict(impute=True)
    st.close()
    st, view, z, gids, hp, ss, counts = make_state(ctx, oracle, descs, 300, 3, seed=2)
    r = st.predict(impute=True)
    assert np.array_equal(r["values"][0], view._data["f0"].astype(np.float64))
    st.close()


def test_imputed_values_follow_the_posterior_predictive_law(ctx):
    from scipy import stats
    ntr = 300
    # the training rows of _dd_bb_state, then 2000 copies of one held-out row with dd(5) masked and bb = 1 observed: every copy is an
    # independent draw (its own row id), 10 counters give 20 000 draws
    rng = np.random.default_rng(5)
    z = np.arange(ntr) % 3
    theta = np.array([[.6, .2, .1, .05, .05], [.05, .05, .1, .2, .6], [.2, .2, .2, .2, .2]])
    dd = np.array([rng.choice(5, p=theta[g]) for g in z])
    bb = rng.random(ntr) < np.array([.9, .2, .5])[z]
    nh = 2000
    arr = np.zeros(ntr + nh, dtype=[("f0", np.int32), ("f1", np.bool_)])
    arr["f0"][:ntr] = dd
    arr["f1"][:ntr] = bb
    arr["f1"][ntr:] = True
    mask = np.zeros(ntr + nh, dtype=[("f0", np.bool_), ("f1", np.bool_)])
    mask["f0"][ntr:] = True
    st = cb.state(ctx, [cb.dd(5), cb.bb], max_groups=8, cluster_hp={"alpha": 1.5})
    st.bind(cb.numpy_dataview(ma.array(arr, mask=mask)))
    gids = [st.create_group() for _ in range(4)]
    st.add_values(np.concatenate([np.asarray(gids)[z], -np.ones(nh, np.int64)]))
    hist = np.zeros(5)
    for counter in range(10):
        r = st.predict(ntr, ntr + nh, responsibilities=True, impute=True, seed=29, counter=counter)
        hist += np.bincount(r["values"][0].astype(np.int64), minlength=5)
        assert np.all(r["values"][1] == 1.0)
    resp = r["resp"][0].astype(np.float64)
    law = np.zeros(5)
    for c, g in enumerate(r["gids"]):
        cnt = np.array([np.sum((z == c) & (dd == v)) for v in range(5)], np.float64) if c < 3 else np.zeros(5)
        law += resp[c] * (1.0 + cnt) / (5.0 + cnt.sum())      # dd(5) with alphas 1: (alpha_x + n_kx) / (sum alpha + n_k)
    law /= law.sum()
    assert stats.chisquare(hist, law * hist.sum()).pvalue > 1e-3
    st.close()


def test_predict_changes_nothing_of_the_state(ctx, oracle):
    descs = [cb.bb, cb.gp, cb.nich, cb.dd(16), cb.niw(3)]
    n, k = 1200, 6

    def snapshot(st, gids):
        ss = [st.get_suffstats(d, g, key, st._ss_counts(st._models[d], key)).tobytes()
              for d in range(len(descs)) for g in gids for key in st._SS_KEYS[st._models[d].name()]]
        return st.assignments().tobytes(), ss, [st.groupsize(g) for g in gids], st.score_likelihood(), st.last_timings()

    a, _, _, gids, _, _, _ = make_state(ctx, oracle, descs, n, k, seed=9, mask_frac=0.05, extra_empty=1)
    b, _, _, _, _, _, _ = make_state(ctx, oracle, descs, n, k, seed=9, mask_frac=0.05, extra_empty=1)
    a.sweep(seed=5, sweep=0); b.sweep(seed=5, sweep=0)
    before = snapshot(a, gids)
    a.predict(responsibilities=True, map=True, draw=True, impute=True, seed=5, counter=1)
    assert snapshot(a, gids) == before
    a.sweep(seed=5, sweep=1); b.sweep(seed=5, sweep=1)
    assert np.array_equal(a.assignments(), b.assignments())
    a.close(); b.close()
