"""The tile sampler's fast paths (common_b200/csrc/msb_score.cuh, sample_tile_kernel): the packed exp of a batch whose
x = s - max all lie in [-86, 0], and the walk's skip of a batch whose quotients provably leave every dart unchanged.
Both must keep the draws of util.hpp:125-156 bit for bit."""
import ctypes as C
import struct
from fractions import Fraction

import numpy as np
import pytest

import common_b200 as cb
from test_division_sequence import rn32, F


def f32(bits):
    return np.frombuffer(struct.pack("<I", bits), np.float32)[0]


def bexp(x):
    """biased exponent field of a binary32"""
    return (struct.unpack("<I", struct.pack("<f", float(x)))[0] >> 23) & 0xFF


def skip_rule(pmax, acc, d):
    """the walk's test: may a lane at dart d skip a batch whose largest p is pmax (acc in [1, 2^24], d >= 2^-60)?"""
    return bexp(pmax) <= bexp(acc) - 154 + bexp(d)


def step(d, p, acc):
    """one step of the walk in exact rational arithmetic: RN(d - RN(p / acc))"""
    q = rn32(F(p) / F(acc))
    return rn32(F(d) - F(q))


def test_skip_rule_leaves_the_dart_unchanged():
    rng = np.random.default_rng(3)
    darts = [np.float32(2.0 ** e) for e in range(-60, 1)]                                 # exact powers of two
    darts += [np.float32(np.nextafter(np.float32(2.0 ** e), np.float32(1))) for e in range(-60, 0)]
    darts += [np.float32(np.nextafter(np.float32(2.0 ** e), np.float32(0))) for e in range(-59, 1)]
    darts += [np.float32(1.0 - 2.0 ** -24), np.float32(0.25), np.float32(0.75)]
    darts += list(rng.uniform(0, 1, 40).astype(np.float32))
    accs = [np.float32(1.0), np.float32(np.nextafter(np.float32(1), np.float32(2))), np.float32(2.0 ** 24),
            np.float32(3.0), np.float32(200.0), np.float32(np.nextafter(np.float32(2.0), np.float32(0)))]
    skipped = changed = 0
    for d in darts:
        for acc in accs:
            h = Fraction(2) ** (bexp(d) - 127 - 25)
            edge = F(acc) * h                                    # acc * h: the boundary the rule stays below
            cands = set()
            for c in (edge, edge / 2, edge / 4, edge * 2):
                p = rn32(c)
                b = struct.unpack("<I", struct.pack("<f", float(p)))[0]
                for off in range(-3, 4):
                    if 0 < b + off < 0x7F800000:
                        cands.add(int(b + off))
            e_max = bexp(acc) - 154 + bexp(d)                    # the largest p the rule accepts: exponent e_max, all ones
            if 0 <= e_max < 255:
                cands.add((e_max << 23) | 0x7FFFFF)
            for b in cands:
                p = f32(b)
                if skip_rule(p, acc, d):
                    skipped += 1
                    assert step(d, p, acc) == d, (d, acc, p)       # the dart stays bit for bit, so no pick either
                elif step(d, p, acc) != d:
                    changed += 1
    assert skipped > 1000 and changed > 1000


def test_skip_rule_stays_within_a_factor_of_four_of_the_exact_bound():
    # p just below 2^(e_max - 126) is accepted, the next exponent is not: the rule gives up a factor of two at most for
    # rounding p up to a power of two and two for rounding acc down to one (here acc = 1, so only the first)
    d, acc = np.float32(0.5), np.float32(1.0)
    e_max = bexp(acc) - 154 + bexp(d)
    assert skip_rule(f32((e_max << 23) | 0x7FFFFF), acc, d)
    assert not skip_rule(f32((e_max + 1) << 23), acc, d)
    assert F(f32((e_max + 1) << 23)) * 2 == F(acc) * Fraction(2) ** (bexp(d) - 127 - 25)


@pytest.mark.gpu
def test_kernels_skip_rule_is_the_checked_one_and_exact(ctx):
    # the walk's own predicate (dart_keeps, msb_kernels.cuh) evaluated on the device over darts at and around powers of
    # two, sums at and around the ends of [1, 2^24], and exponents around the bound; every accepted case must leave the
    # dart unchanged for the largest p of that exponent, and the device must agree with skip_rule above
    from common_b200 import _lib
    darts = [np.float32(2.0 ** e) for e in range(-61, 2)] + [np.float32(np.nextafter(np.float32(2.0 ** e), np.float32(0)))
                                                              for e in range(-60, 1)]
    darts += [np.float32(0.75), np.float32(1.0 - 2.0 ** -24), np.float32(0.0), np.float32(np.nan), np.float32(-0.5)]
    accs = [np.float32(1.0), np.float32(np.nextafter(np.float32(1), np.float32(0))), np.float32(3.0),
            np.float32(2.0 ** 24), np.float32(np.nextafter(np.float32(2.0 ** 24), np.float32(2.0 ** 25))), np.float32(np.nan)]
    E, A, D = [], [], []
    for d in darts:
        for acc in accs:
            base = (bexp(acc) - 154 + bexp(d)) if np.isfinite(d) and np.isfinite(acc) else 100
            for e in sorted({0, 1, 254, 255} | {x for x in range(base - 3, base + 4) if 0 <= x <= 255}):
                E.append(e); A.append(acc); D.append(d)
    e = np.array(E, np.uint8); a = np.array(A, np.float32); d = np.array(D, np.float32)
    out = np.zeros(len(e), np.uint8)
    _lib.check(_lib.load().msb_selftest_skip_rule(ctx.handle, e.ctypes.data, a.ctypes.data, d.ctypes.data, len(e),
                                                 out.ctypes.data))
    accepted = 0
    for ei, ai, di, oi in zip(e, a, d, out):
        want = bool(1 <= ai <= 2.0 ** 24 and di >= 2.0 ** -60 and skip_rule(f32(int(ei) << 23), ai, di))
        assert bool(oi) == want, (int(ei), ai, di)
        if oi:
            accepted += 1
            p = f32((int(ei) << 23) | 0x7FFFFF)          # the largest p with that exponent
            assert step(di, p, ai) == di, (int(ei), ai, di)
    assert accepted > 500
    # at d = 1/2, acc = 1 the bound sits at exponent 99 (p < 2^-27): 99 passes, 100 does not
    out1 = np.zeros(2, np.uint8)
    e1 = np.array([99, 100], np.uint8); a1 = np.ones(2, np.float32); d1 = np.full(2, 0.5, np.float32)
    _lib.check(_lib.load().msb_selftest_skip_rule(ctx.handle, e1.ctypes.data, a1.ctypes.data, d1.ctypes.data, 2,
                                                 out1.ctypes.data))
    assert list(out1) == [1, 0]


@pytest.mark.gpu
def test_packed_exp_equals_scalar_exp_on_every_float_in_range(ctx):
    from common_b200 import _lib
    bad = C.c_uint64(1)
    _lib.check(_lib.load().msb_selftest_expf2(ctx.handle, C.byref(bad)))
    assert bad.value == 0


def crafted(k, n, seed):
    rng = np.random.default_rng(seed)
    h = n // 2
    s = rng.normal(0.0, 30.0, (n, k)).astype(np.float32)
    s[:h] = rng.uniform(-80, 0, (h, k))            # whole 32-row warps within exp's normal range: the packed path
    s[:h:37] = 0.0
    u = rng.uniform(0, 1, n).astype(np.float32)
    u[2::13] = 0.0
    u[3::13] = np.float32(1.0 - 2.0 ** -24)
    u[4::13] = np.float32(2.0 ** -rng.integers(1, 24, len(u[4::13])))           # darts at exact powers of two
    s[h + 1::9, 0] += 200.0                                                     # dead batches next to a dominant group
    # darts below 2^-60 meeting a p below 2^-100 before the dominant group: the division is redone with the IEEE operator
    tiny = slice(h + 5, n, 17)
    s[tiny, :] = -300.0
    s[tiny, 0] = -70.0                                                           # p ~ 2^-101
    s[tiny, k - 1] = 0.0
    u[tiny] = np.float32(2.0 ** -70)
    s[h + 6::19, rng.integers(0, k)] = np.nan
    s[h + 7::23, :] = -np.inf
    s[h + 8::29, rng.integers(0, k)] = -np.inf
    s[h + 9::31, :] = np.nan
    return s, u


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 7, 8, 9, 200, 372, 384])
def test_crafted_matrices_draw_like_the_checker(ctx, oracle, k, monkeypatch):
    # the discrete-log sampler takes the tile sampler when the tile fits (K <= 372: K * 33 floats within 48 KB), the
    # one-row-per-thread walk otherwise (384).  The first half of the rows lies in [-80, 0], so from K = 8 on whole warps
    # take the packed exp; K = 1 and 7 are a single padded batch (the scalar exp), K = 9 one packed batch and one padded.
    n = 2000
    s, u = crafted(k, n, seed=k)
    want = oracle.sample_rows(s, u)
    got = cb.sample_discrete_log(ctx, s, u)
    assert np.array_equal(got, want)
    monkeypatch.setenv("MSB_NO_TILE_SAMPLER", "1")
    assert np.array_equal(cb.sample_discrete_log(ctx, s, u), want)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [8, 200, 208, 216, 384])
def test_tables_only_row_maxima_give_the_same_scores_and_draws(ctx, oracle, k, monkeypatch):
    # dd(256) x 4 is the tables-only path: score_kernel's blocked epilogues leave the row maxima (K = 8 and 200: ragged
    # last k-tile of 8 groups, 208: of 16, 216: no ragged tile, 384: full k-tiles and the global-memory sampler).
    # Without them (MSB_NO_ROWMAX) and with the persistent kernel, which does not emit them, the samplers scan; the
    # scores and the draws must be the same bits in all three, and the draws the checker's.
    from test_gpu_parity import make_state
    descs = [cb.dd(256)] * 4
    n = 5000
    u = np.array([oracle.philox_u01(6, i, 0) for i in range(n)], np.float32)
    runs = []
    for env in (None, "MSB_NO_ROWMAX", "MSB_PERSISTENT"):
        if env:
            monkeypatch.setenv(env, "1")
        st, view, z, gids, hp, ss, counts = make_state(ctx, oracle, descs, n, k, seed=23, extra_empty=1)
        st.sweep(seed=6, sweep=0)
        S = st.read_last_scores().copy()
        a = np.searchsorted(gids, st.assignments()).astype(np.int32)
        assert np.array_equal(a, oracle.sample_rows(S, u))
        runs.append((S, a))
        st.close()
        if env:
            monkeypatch.delenv(env)
    for S, a in runs[1:]:
        assert np.array_equal(S.view(np.uint32), runs[0][0].view(np.uint32))
        assert np.array_equal(a, runs[0][1])


@pytest.mark.gpu
@pytest.mark.parametrize("k", [8, 200])
def test_sweep_with_bundled_row_maxima_draws_like_the_checker(ctx, oracle, k, monkeypatch):
    # the general score kernel leaves the row maxima and the tile sampler skips its first pass; without them it scans
    from test_gpu_parity import make_state
    descs = [cb.nich, cb.dd(16), cb.bb] * 2
    n = 4099
    got = {}
    for env in (None, "1"):
        if env:
            monkeypatch.setenv("MSB_NO_ROWMAX", env)
        st, view, z, gids, hp, ss, counts = make_state(ctx, oracle, descs, n, k, seed=17, extra_empty=1)
        st.sweep(seed=4, sweep=0)
        S = st.read_last_scores()
        got[env] = np.searchsorted(gids, st.assignments()).astype(np.int32)
        u = np.array([oracle.philox_u01(4, i, 0) for i in range(n)], np.float32)
        assert np.array_equal(got[env], oracle.sample_rows(S, u))
        st.close()
    assert np.array_equal(got[None], got["1"])
