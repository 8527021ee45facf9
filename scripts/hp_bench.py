#!/usr/bin/env python
"""Time of one grid Gibbs step over the hypers (msb_state_hp_gibbs, DESIGN.md section 4.10) at the C2, C4 and C5 shapes.

Grids: C2 and C5 a 32-point grid on every feature, C4 (niw(64)) a 16-point (kappa, nu) grid, 32 points for alpha.
For each configuration it reports
  hp_gibbs   per call: the device time of its kernels (msb_ctx_profile event pairs) and the host time of the whole call
             (it ends with a synchronise), after one warm-up call;
  host_loop  the loop hp_gibbs replaces -- set_component_hp + score_likelihood per (feature, point), exp in numpy, the
             winner set -- in full at C2 and C4, on a stated subset of the features at C5 (scaled to all of them);
  sweep      the device-resident sweep of the same state (sum of its phase events).
The card's name, power limit and maximum SM clock are read in the same run.

    python scripts/hp_bench.py [--configs C2 C4 C5] [--reps 10] [--c5-features 8] [--out DIR]
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
import common_b200 as cb  # noqa: E402
from predict_bench import card, kernel_ms, make_state  # noqa: E402

HP_KERNELS = ("hp_", "niw_hp_")


def grid(desc, G):
    """G hp dicts around the defaults: one concentration / scale factor per point"""
    d = desc()
    name, c = d.name(), np.exp(np.linspace(-2.0, 2.0, G))
    if name == "niw":
        p = d._param()
        return [{"mu": np.zeros(p), "kappa": k, "psi": np.eye(p), "nu": p + v}
                for k in (0.1, 1.0, 10.0, 100.0) for v in (1.0, 8.0, 64.0, 256.0)][:G]
    if name == "dd":
        return [{"alphas": np.full(d._param(), x)} for x in c]
    if name == "bb":
        return [{"alpha": x, "beta": 1.0 / x} for x in c]
    if name == "gp":
        return [{"alpha": x, "inv_beta": 1.0} for x in c]
    return [{"mu": 0.0, "kappa": x, "sigmasq": 1.0, "nu": 1.0 + x} for x in c]   # nich


def host_loop(st, features, grids):
    """the caller's loop without the library's hp step: seconds for `features`"""
    t0 = time.perf_counter()
    for d in features:
        w = np.zeros(len(grids[d]))
        for g, pt in enumerate(grids[d]):
            st.set_component_hp(d, pt)
            w[g] = st.score_likelihood(d)
        p = np.exp(w - w.max())
        st.set_component_hp(d, grids[d][int(np.searchsorted(np.cumsum(p), np.random.rand() * p.sum(), side="right"))])
    return time.perf_counter() - t0


def sweep_ms(st, reps):
    for i in range(2):
        st.sweep(seed=1, sweep=i)
    tot = 0.0
    for i in range(reps):
        st.sweep(seed=1, sweep=100 + i)
        tot += sum(st.last_timings().values())
    return tot / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=["C2", "C4", "C5"])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--c5-features", type=int, default=8, help="features timed in the C5 host loop (spread over the families)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ctx = cb.Context(0)
    rec = {"card": card(), "configs": {}}
    for name in args.configs:
        cfg = cb.synth.config(name)
        st = make_state(ctx, cfg, 0.0)
        D = len(cfg["models"])
        G = 16 if name == "C4" else 32
        grids = [grid(m, G) for m in cfg["models"]]
        for d in range(D):
            st.set_hp_grid(d, grids[d])
        st.set_cluster_hp_grid(np.exp(np.linspace(-3.0, 3.0, 32)))
        res = {"n": cfg["n"], "k": cfg["k"], "d": D, "grid_points": G}
        counter = [0]

        def step():
            counter[0] += 1
            st.hp_gibbs(seed=3, counter=counter[0])
        prof = kernel_ms(ctx, step, args.reps)
        res["hp_gibbs_kernels_ms"] = {k: v for k, v in prof.items() if k.startswith(HP_KERNELS)}
        res["hp_gibbs_device_ms"] = sum(res["hp_gibbs_kernels_ms"].values())
        t0 = time.perf_counter()
        for _ in range(args.reps):
            step()
        res["hp_gibbs_call_ms"] = (time.perf_counter() - t0) * 1e3 / args.reps
        res["sweep_ms"] = sweep_ms(st, args.reps)
        if name == "C5":
            per = D // 4
            feats = [f * per + i for f in range(4) for i in range(max(1, args.c5_features // 4))]
        else:
            feats = list(range(D))
        host_loop(st, feats[:1], grids)                                   # warm-up
        s = host_loop(st, feats, grids)
        res["host_loop"] = {"features_timed": len(feats), "seconds": s, "seconds_all_features": s * D / len(feats)}
        res["speedup_vs_host_loop"] = res["host_loop"]["seconds_all_features"] * 1e3 / res["hp_gibbs_call_ms"]
        res["hp_gibbs_over_sweep"] = res["hp_gibbs_call_ms"] / res["sweep_ms"]
        st.close()
        rec["configs"][name] = res
        print(json.dumps({name: res}), flush=True)
    rec["card_after"] = card()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "hp_bench.json"), "w") as f:
            json.dump(rec, f, indent=1)
    print(json.dumps(rec))
    ctx.close()


if __name__ == "__main__":
    main()
