"""Kernel time of msb_state_predict at the C2 and C5 shapes (DESIGN.md section 4.9).

For each configuration, after warm-up, the per-call time of the predictive reduction kernel (predict_tile_kernel or
predict_rows_kernel, from msb_ctx_profile's CUDA event pairs) for
  logp        logp only,
  logp+resp   logp and the responsibilities,
  impute      logp, the group draw and the imputation of a dataset with 5 % of its cells masked
(the latter also reports the sampler's and impute_kernel's time), beside the sweep's sample phase on the same state.
The reduction's bytes are 4 N K read + 8 N written (+ 4 N K written with resp), reported over the measured HBM peak the
project uses (6539 GB/s).  The card's name, power limit and maximum SM clock are read in the same run.

    python scripts/predict_bench.py [--configs C2 C5] [--reps 10] [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import common_b200 as cb  # noqa: E402

HBM_GBPS = 6539.0   # measured HBM peak of a B200 (the figure the project's roofline uses)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, mhz = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": mhz}
    except Exception as e:  # the numbers are still measured; the record says the card could not be read
        return {"error": str(e)}


def make_state(ctx, cfg, mask_frac):
    arr, z = cb.synth.make_dataset(cfg["models"], cfg["n"], cfg["k"], seed=73, mask_frac=mask_frac, storage=cfg.get("storage"))
    st = cb.state(ctx, cfg["models"], max_groups=cfg["k"] + 8, cluster_hp={"alpha": 1.0})
    if cfg.get("hp"):
        for d in range(len(cfg["models"])):
            st.set_component_hp(d, cfg["hp"])
    st.bind(cb.numpy_dataview(arr))
    gids = np.asarray([st.create_group() for _ in range(cfg["k"])])
    st.add_values(gids[z])
    return st


def kernel_ms(ctx, fn, reps):
    """per-call ms of every kernel fn launches, over reps calls after one warm-up call"""
    fn()
    ctx.synchronize()
    ctx.profile(True)
    for _ in range(reps):
        fn()
    ctx.synchronize()
    prof = ctx.profile_read()
    ctx.profile(False)
    return {name: ms / reps for name, (cnt, ms) in prof.items()}


def pick(prof, prefix):
    return sum(v for name, v in prof.items() if name.startswith(prefix))


def sample_phase_ms(st, reps):
    for i in range(3):
        st.sweep(seed=73, sweep=1000 + i)
    ms = []
    for i in range(reps):
        st.sweep(seed=73, sweep=2000 + i)
        ms.append(st.last_timings()["sample"])
    return float(np.median(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=["C2", "C5"])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None, help="directory for predict_bench.json")
    args = ap.parse_args()
    ctx = cb.Context(0)
    rec = {"card": card(), "hbm_gbps": HBM_GBPS, "configs": {}}
    for name in args.configs:
        cfg = cb.synth.config(name)
        n, k = cfg["n"], cfg["k"]
        res = {"n": n, "k": k, "d": len(cfg["models"])}
        t0 = time.perf_counter()
        st = make_state(ctx, cfg, 0.0)
        K = st.ngroups()
        modes = {
            "logp": (lambda: st.predict(), 4.0 * n * K + 8.0 * n),
            "logp+resp": (lambda: st.predict(responsibilities=True), 8.0 * n * K + 8.0 * n),
        }
        for mode, (fn, nbytes) in modes.items():
            prof = kernel_ms(ctx, fn, args.reps if mode == "logp" else max(2, args.reps // 4))
            ms = pick(prof, "predict_")
            res[mode] = {"predict_ms": ms, "score_ms": pick(prof, "score_"), "bytes": nbytes,
                         "hbm_fraction": nbytes / (ms * 1e-3) / (HBM_GBPS * 1e9) if ms > 0 else None}
        res["sweep_sample_ms"] = sample_phase_ms(st, args.reps)
        st.close()
        st = make_state(ctx, cfg, 0.05)
        prof = kernel_ms(ctx, lambda: st.predict(impute=True, seed=5, counter=1), max(2, args.reps // 4))
        ms = pick(prof, "predict_")
        nbytes = 4.0 * n * K + 8.0 * n
        res["impute"] = {"predict_ms": ms, "sampler_ms": pick(prof, "sample_"), "impute_ms": pick(prof, "impute_kernel"),
                         "niw_factor_ms": pick(prof, "niw_predictive_factor_kernel"), "score_ms": pick(prof, "score_"),
                         "bytes": nbytes, "hbm_fraction": nbytes / (ms * 1e-3) / (HBM_GBPS * 1e9) if ms > 0 else None}
        res["impute_state_sweep_sample_ms"] = sample_phase_ms(st, args.reps)
        st.close()
        res["wall_s"] = time.perf_counter() - t0
        rec["configs"][name] = res
        print(json.dumps({name: res}), flush=True)
    rec["card_after"] = card()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "predict_bench.json"), "w") as f:
            json.dump(rec, f, indent=1)
    print(json.dumps(rec))
    ctx.close()


if __name__ == "__main__":
    main()
