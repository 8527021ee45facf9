#!/usr/bin/env python
"""Time of the non-conjugate parameter steps (msb_state_theta and msb_state_redraw_empty, DESIGN.md section 4.11) on a
1M-row state of bbnc features only, at K = 200 x D = 32 and K = 1000 x D = 256 (data from synth.make_dataset, 8 more
groups left empty so that redraw_empty has work).

For each shape it reports
  theta, redraw_empty  per call: the device time of their kernels (msb_ctx_profile event pairs, 5 calls after a
                       warm-up) and the host time of the whole call (it ends with a synchronise);
  sweep                the device-resident sweep of the same state (sum of its phase events);
  host_loop            the runner's loop without these calls: per group and per density evaluation one set_suffstats of
                       p and one score_likelihood.  A stated number of (set_suffstats, score_likelihood) pairs is timed,
                       and scaled by the mean number of density evaluations of one slice update -- counted by a
                       restatement of the update in numpy on a sample of the state's groups -- times K x D.
The card's name, power limit and maximum SM clock are read in the same run.

    python scripts/theta_bench.py [--shapes 200x32 1000x256] [--rows 1000000] [--reps 5] [--host-evals 200] [--out DIR]
"""
import argparse
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import common_b200 as cb  # noqa: E402
from hp_bench import sweep_ms  # noqa: E402
from predict_bench import card, kernel_ms  # noqa: E402

WIDTH = 0.1


def slice_evals(a, b, p0, heads, tails, w, rng):
    """density evaluations of one slice update (stepping out, then shrinkage) at these values"""
    def f(p):
        if p <= 0.0 or p >= 1.0:
            return -math.inf
        return (a - 1.0 + heads) * math.log(p) + (b - 1.0 + tails) * math.log1p(-p)
    n = 1
    y = f(p0) + math.log(rng.random() or 0.5)
    L = p0 - w * rng.random()
    R = L + w
    while True:
        n += 1
        if not f(L) > y:
            break
        L -= w
    while True:
        n += 1
        if not f(R) > y:
            break
        R += w
    while True:
        x = L + rng.random() * (R - L)
        n += 1
        if f(x) > y:
            return n
        if x < p0:
            L = x
        else:
            R = x


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", nargs="+", default=["200x32", "1000x256"])
    ap.add_argument("--rows", type=int, default=1000000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--host-evals", type=int, default=200, help="(set_suffstats, score_likelihood) pairs timed")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ctx = cb.Context(0)
    rec = {"card": card(), "shapes": {}}
    for shape in args.shapes:
        K, D = (int(x) for x in shape.split("x"))
        models = [cb.bbnc] * D
        arr, z = cb.synth.make_dataset(models, args.rows, K, seed=73)
        st = cb.state(ctx, models, max_groups=K + 8, cluster_hp={"alpha": 1.0})
        st.bind(cb.numpy_dataview(arr))
        gids = np.asarray([st.create_group() for _ in range(K + 8)])
        st.add_values(gids[z])
        res = {"n": args.rows, "k": K + 8, "d": D, "width": WIDTH}
        tp = {d: {"p": WIDTH} for d in range(D)}
        counter = [0]

        def theta():
            counter[0] += 1
            assert st.theta(tp, seed=3, counter=counter[0]) == 0

        def redraw():
            counter[0] += 1
            st.redraw_empty(seed=3, counter=counter[0])

        for name, fn, prefix in (("theta", theta, "theta_"), ("redraw_empty", redraw, ("redraw_", "theta_commit"))):
            prof = kernel_ms(ctx, fn, args.reps)
            res[name + "_kernels_ms"] = {k: v for k, v in prof.items() if k.startswith(prefix)}
            res[name + "_device_ms"] = sum(res[name + "_kernels_ms"].values())
            t0 = time.perf_counter()
            for _ in range(args.reps):
                fn()
            res[name + "_call_ms"] = (time.perf_counter() - t0) * 1e3 / args.reps
        res["sweep_ms"] = sweep_ms(st, args.reps)
        # the host loop: a sample of the state's columns gives the mean number of evaluations of one update
        rng = np.random.default_rng(0)
        evals = []
        for _ in range(64):
            d, g = int(rng.integers(D)), int(gids[rng.integers(K)])
            p0, heads, tails = (float(st.get_suffstats(d, g, key)[0]) for key in ("p", "heads", "tails"))
            evals.append(slice_evals(1.0, 1.0, p0, heads, tails, WIDTH, rng))
        g0 = int(gids[0])
        p_keep = st.get_suffstats(0, g0, "p")
        st.set_suffstats(0, g0, "p", p_keep)
        st.score_likelihood(0, g0)                                                   # warm-up
        t0 = time.perf_counter()
        for i in range(args.host_evals):
            st.set_suffstats(0, g0, "p", p_keep)
            st.score_likelihood(0, g0)
        per_eval = (time.perf_counter() - t0) / args.host_evals
        res["host_loop"] = {"pairs_timed": args.host_evals, "seconds_per_pair": per_eval,
                            "evaluations_per_update": float(np.mean(evals)),
                            "seconds_all_groups": per_eval * float(np.mean(evals)) * (K + 8) * D}
        res["speedup_vs_host_loop"] = res["host_loop"]["seconds_all_groups"] * 1e3 / res["theta_call_ms"]
        res["theta_over_sweep"] = res["theta_call_ms"] / res["sweep_ms"]
        st.close()
        rec["shapes"][shape] = res
        print(json.dumps({shape: res}), flush=True)
    rec["card_after"] = card()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "theta_bench.json"), "w") as f:
            json.dump(rec, f, indent=1)
    print(json.dumps(rec))
    ctx.close()


if __name__ == "__main__":
    main()
