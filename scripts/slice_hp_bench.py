#!/usr/bin/env python
"""Time of one slice-sampling update of continuous hypers (msb_state_slice_hp, DESIGN.md section 4.12) at the full
synth.config shapes:
  C3  every nich key (mu, kappa, sigmasq, nu) of all 128 features
  C4  niw(64) kappa and nu
  C5  the scalar keys of its bb, gp and nich features (dd has only its vector alphas: left out)
and alpha in each.  Priors: Normal(0, 100) on nich mu, Exponential(1) on the rest (Exponential(0.01) on niw nu); width 1.

For each shape it reports
  slice_hp       per call: the device time of its kernels (msb_ctx_profile event pairs, 5 calls after a warm-up) and
                 the host time of the whole call (it ends with a synchronise);
  evaluations    the mean number of target evaluations per spec, counted by the fp64 replay of tests/test_gpu_hpslice.py
                 on a sample of the call's specs (one feature per family, and alpha);
  sweep          the device-resident sweep of the same state (sum of its phase events);
  host_loop      the caller's loop without the call: per evaluation one set_component_hp and one
                 score_likelihood(component).  A stated number of pairs is timed on one feature per family and scaled by
                 the mean evaluations per spec times the number of feature specs.
The cost depends on K x D (and niw's d), not on N.  The card's name, power limit and maximum SM clock are read in the
same run.

    python scripts/slice_hp_bench.py [--configs C3 C4 C5] [--reps 5] [--host-pairs 20] [--out DIR]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import common_b200 as cb  # noqa: E402
from common_b200 import hyperprior as hpr  # noqa: E402
from hp_bench import sweep_ms  # noqa: E402
from predict_bench import card, kernel_ms  # noqa: E402

E1 = hpr.log_exponential(1.0)
KEYS = {"bb": {"alpha": E1, "beta": E1}, "gp": {"alpha": E1, "inv_beta": E1},
        "nich": {"mu": hpr.log_normal(0.0, 100.0), "kappa": E1, "sigmasq": E1, "nu": E1},
        "niw": {"kappa": E1, "nu": hpr.log_exponential(0.01)}}
WIDTH = 1.0


def specs_of(models):
    return {d: {k: (p, WIDTH) for k, p in KEYS[m().name()].items()} for d, m in enumerate(models) if m().name() in KEYS}


def count_evaluations(st, cfg, arr, hparams, before, alpha0, seed, counter, values):
    """evaluations per spec of one feature per family and of alpha, from the fp64 replay of the call just made"""
    import oracle_lib as ol
    from test_gpu_hpslice import alpha_target, feature_target, hp_offset, niw_prep, slice_replay
    oracle = ol.load()
    models = cfg["models"]
    gids = sorted(st.groups())                                  # the partition the sweeps left, empty groups included
    K = len(gids)
    z = np.searchsorted(gids, st.assignments())
    counts = np.bincount(z, minlength=K).astype(np.float64)
    evals, seen = [], set()
    for d, params in hparams.items():
        desc = models[d]
        if desc().name() in seen:
            continue
        seen.add(desc().name())
        h = before[d].copy()
        niw = niw_prep(st, d, gids, desc()._param(), h) if desc().name() == "niw" else None
        ss = None
        if niw is None:
            name = arr.dtype.names[d]
            one = np.zeros(len(arr), dtype=[(name, arr.dtype[name])])       # a packed one-field record
            one[name] = arr[name]
            ss, _ = ol.build_suffstats(oracle, [desc], h, cb.numpy_dataview(one), z, K)
        for j, (key, (prior, w)) in enumerate(params.items()):
            f = feature_target(oracle, desc, key, prior, h, ss, niw)
            _, _, n, _ = slice_replay(oracle, seed, counter, d, j, f, h[hp_offset(desc, key)], w)
            evals.append(n)
            h[hp_offset(desc, key)] = values[d][key]
    _, _, n, _ = slice_replay(oracle, seed, counter, len(models), 0, alpha_target(E1, counts), alpha0, WIDTH)
    return float(np.mean(evals)), float(n)


def make_state(ctx, cfg):
    """predict_bench's state (K groups in creation order), and its data for the replay's suffstats"""
    arr, z = cb.synth.make_dataset(cfg["models"], cfg["n"], cfg["k"], seed=73, storage=cfg.get("storage"))
    st = cb.state(ctx, cfg["models"], max_groups=cfg["k"] + 8, cluster_hp={"alpha": 1.0})
    st.bind(cb.numpy_dataview(arr))
    gids = np.asarray([st.create_group() for _ in range(cfg["k"])])
    st.add_values(gids[z])
    return st, arr, z


def host_loop(st, hparams, models, pairs):
    """seconds per (set_component_hp, score_likelihood(component)) pair, on one feature per family"""
    feats, seen = [], set()
    for d in hparams:
        if models[d]().name() not in seen:
            seen.add(models[d]().name())
            feats.append(d)
    per = []
    for d in feats:
        key = next(iter(hparams[d]))
        v = st.get_component_hp(d)[key]
        st.set_component_hp(d, {key: v})
        st.score_likelihood(d)                                                   # warm-up
        t0 = time.perf_counter()
        for _ in range(pairs):
            st.set_component_hp(d, {key: v})
            st.score_likelihood(d)
        per.append((time.perf_counter() - t0) / pairs)
    return float(np.mean(per)), feats


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=["C3", "C4", "C5"])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--host-pairs", type=int, default=20, help="(set_component_hp, score_likelihood) pairs timed per feature")
    ap.add_argument("--rows", type=int, default=None, help="override the config's N (the cost does not depend on it)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ctx = cb.Context(0)
    rec = {"card": card(), "configs": {}}
    for name in args.configs:
        cfg = cb.synth.config(name)
        if args.rows:
            cfg["n"] = args.rows
        st, arr, z = make_state(ctx, cfg)
        models = cfg["models"]
        hparams = specs_of(models)
        cparam = {"alpha": (E1, WIDTH)}
        nspecs = sum(len(v) for v in hparams.values())
        res = {"n": cfg["n"], "k": cfg["k"], "d": len(models), "feature_specs": nspecs, "width": WIDTH}
        counter = [0]

        def call():
            counter[0] += 1
            assert st.slice_hp(hparams, cparam, seed=3, counter=counter[0])["capped"] == 0
        prof = kernel_ms(ctx, call, args.reps)
        res["kernels_ms"] = {k: v for k, v in prof.items() if "slice" in k}
        res["device_ms"] = sum(res["kernels_ms"].values())
        t0 = time.perf_counter()
        for _ in range(args.reps):
            call()
        res["call_ms"] = (time.perf_counter() - t0) * 1e3 / args.reps
        res["sweep_ms"] = sweep_ms(st, args.reps)
        before = [np.concatenate([np.ravel(v) for v in st.get_component_hp(d).values()]) for d in range(len(models))]
        alpha0 = st.get_cluster_hp()["alpha"]
        values = st.slice_hp(hparams, cparam, seed=3, counter=10 ** 6)["values"]
        ev, ev_alpha = count_evaluations(st, cfg, arr, hparams, before, alpha0, 3, 10 ** 6, values)
        res["evaluations_per_spec"] = ev
        res["evaluations_alpha"] = ev_alpha
        per_pair, feats = host_loop(st, hparams, models, args.host_pairs)
        res["host_loop"] = {"features_timed": feats, "pairs_per_feature": args.host_pairs, "seconds_per_pair": per_pair,
                            "seconds_all_specs": per_pair * ev * nspecs}
        res["speedup_vs_host_loop"] = res["host_loop"]["seconds_all_specs"] * 1e3 / res["call_ms"]
        res["call_over_sweep"] = res["call_ms"] / res["sweep_ms"]
        st.close()
        del arr, z
        rec["configs"][name] = res
        print(json.dumps({name: res}), flush=True)
    rec["card_after"] = card()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "slice_hp_bench.json"), "w") as f:
            json.dump(rec, f, indent=1)
    print(json.dumps(rec))
    ctx.close()


if __name__ == "__main__":
    main()
