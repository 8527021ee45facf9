#!/usr/bin/env python
"""bench.py -- row x group x feature scores/sec of the hot path on N B200s of one node.

A "step" is one full pass of the hot path over one batch of synthetic rows:
parameter build -> score (N x K matrix materialised) -> categorical draw ->
suffstat update (-> one all-reduce of the suffstat deltas when N > 1).

  python bench.py --gpus 1 --steps 5 --warmup 3
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...      # the CPU path, all host threads
  python bench.py ... --dump-outputs DIR    # + what the last timed step computed, as DIR/<config>_<name>.npy

Prints ONE JSON line (rank 0).  The headline keys (value, ms_per_step, roofline, e2e, cpu_baseline) are those of
--workload (default C2, BASELINE.json configs[1], at every N so that the per-N values are comparable).  The same
line carries, under "configs", one full record per BASELINE.json GPU configuration measured in the same run:

  N = 1 : C2, C3, C4, C5 at full size, each with phase times, roofline, an in-run parity spot check against the
          CPU oracle (scores of a row sample, the draw replayed from the GPU's own score bits, group counts rebuilt
          from the assignments) and the bandwidth-bound kernels against the HBM roof;
  N > 1 : C2 weak, C5 weak (1M rows per GPU) and C3 strong (4M rows / N per GPU), each with a cross-rank replica
          check (64-bit hash of the suffstat buffer, group sizes summing to the global row count).

Compact copies of the per-config figures are repeated as flat keys under "config" and in the closing "summary".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the tree it runs from as it found it (it may be read-only)

METRIC = "row_x_group_x_feature_scores_per_sec"
UNIT = "scores/s"

# per-unit byte sizes of SURVEY.md section 8(d) / BASELINE.md section 5
B_X = {"bb": 1, "dd": 1, "gp": 4, "nich": 4}
B_SS = {"bb": 8, "gp": 12, "nich": 12}
B_HP = {"bb": 8, "gp": 8, "nich": 16}


def algorithmic_bytes_score(descs, storage, n, k):
    """B = N sum b_x + K sum b_ss + sum b_hp + 4 N K   (score mode)"""
    bx = bss = bhp = 0
    for d, desc in enumerate(descs):
        m = desc()
        nm = m.name()
        if nm == "dd":
            C = m._param()
            bx += np.dtype(storage[d]).itemsize if storage and storage[d] is not None else 4
            bss += 4 * (C + 1); bhp += 4 * C
        elif nm == "niw":
            dim = m._param()
            bx += 4 * dim; bss += 4 * (1 + dim + dim * dim); bhp += 4 * (2 + dim + dim * dim)
        else:
            bx += B_X[nm]; bss += B_SS[nm]; bhp += B_HP[nm]
    return n * bx + k * bss + bhp + 4 * n * k


def column_bytes(descs):
    """bytes per row of the device columns the ingest kernel writes: Value-typed column + u32 score column + slow bit"""
    tot = 0
    for desc in descs:
        m = desc()
        nm = m.name()
        if nm == "niw":
            tot += 2 * 4 * m._param()           # raw + centred rows
        elif nm == "dm":
            tot += 4 * m._param()
        else:
            col = 4 if nm in ("gp", "bnb", "nich") else (1 if (nm != "dd" or m._param() + 1 <= 256) else 2)
            tot += col + 4 + 1.0 / 8
    return tot


class ClockSampler(object):
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md)"""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        """starts sampling, or resumes it after pause(): the rows of every sampling stretch are summarised together"""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, args=(self.proc,), daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self, proc):
        for line in proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def pause(self):
        """ends the running sampler; its rows are kept"""
        if not self.proc:
            return
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        self.thread.join(timeout=2)

    def stop(self):
        if not self.proc and not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.pause()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except ValueError:
                continue
            for nm, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def usable_cores():
    """host threads this process may really use: the affinity mask, capped by the cgroup CPU quota
    (os.cpu_count() reports the machine, not the container)"""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


def pin_rank_to_cores(local_rank, world):
    """each rank gets its own slice of the host cores (SCALE_r01: eight ranks shared one affinity mask, and the
    end-to-end pass -- host-side ctypes calls + pinned H2D copies -- lost 27 % at 8 GPUs)"""
    if world <= 1:
        return None
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = max(1, len(cores) // world)
        mine = cores[local_rank * per:(local_rank + 1) * per] or cores
        os.sched_setaffinity(0, mine)
        return len(mine)
    except Exception:
        return None


def build_workload(workload, rows, groups, rank, world, scaling):
    import common_b200 as cb
    cfg = cb.synth.config(workload)
    n_cfg = rows or cfg["n"]
    k = groups or cfg["k"]
    descs = cfg["models"]
    storage = cfg.get("storage")
    if scaling == "strong" and world > 1:
        # total work fixed: rank r holds rows [lo, hi) of the N-row workload (a multiple of K, so that the planted
        # assignment row mod K continues across shards)
        per = (n_cfg // world) // k * k
        lo = rank * per
        n = per if rank < world - 1 else n_cfg - lo
        n_total = n_cfg
    else:
        # weak scaling: every rank holds its own n rows of the same planted mixture (stream id = rank)
        n, lo, n_total = n_cfg, rank * n_cfg, n_cfg * world
    arr, z = cb.synth.make_dataset(descs, n, k, seed=73, stream=rank, storage=storage)
    return cfg, descs, storage, n, k, arr, z, lo, n_total


def cpu_reference_rate(descs, hp_by_feature, arr, z, k, budget_s, nthreads, f32=True):
    """times the CPU path (the reference's per-(row, group, feature) loop) on a bounded row sample.
    Uses oracle/_ref (the reference's own headers) when it was built, else the C port."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import common_b200 as cb
    import oracle_lib as ol
    import ref_lib
    orc = ol.load()
    hp = np.concatenate([orc.flat_hp(d, hp_by_feature) for d in descs])
    n_build = min(arr.shape[0], 200_000)
    view_all = cb.numpy_dataview(arr[:n_build])
    ss, counts = ol.build_suffstats(orc, descs, hp, view_all, z[:n_build], k)
    lp = ol.logprior(counts, 1.0)
    ref = ref_lib.load()
    kind = "reference-api" if ref is not None else "port"
    D = len(descs)

    def run(rows):
        view = cb.numpy_dataview(arr[:rows])
        t0 = time.perf_counter()
        if ref is not None:
            ref.score_rows(descs, hp, ss, lp, view, nthreads)
        else:
            orc.score_rows(descs, hp, ss, lp, view, nthreads=nthreads, f32=f32)
        return time.perf_counter() - t0

    rows = max(8, min(256, arr.shape[0]))
    t = run(rows)
    # grow the sample until it fills the budget (bounded by the data we have)
    while t < budget_s / 4 and rows < arr.shape[0]:
        rows = int(min(arr.shape[0], max(rows * 2, rows * (budget_s / 2) / max(t, 1e-6))))
        t = run(rows)
    noop_ns = None
    if ref is not None and hasattr(ref.lib, "ref_noop_overhead_ns"):
        noop_ns = ref.noop_overhead_ns()     # the reference's own noop model: what the plugin API costs per call
    return {"value": rows * k * D / t, "seconds": t, "rows": rows, "kind": kind, "cores": nthreads, "noop_ns": noop_ns,
            "sample": "%d of the workload's rows x K=%d groups x D=%d features, %s" % (
                rows, k, D, "reference headers (models/base.hpp, recarray/dataview.hpp) + restated family maths, libm logf/lgammaf"
                if ref is not None else "C port of the reference loop, libm logf/lgammaf")}


def workload_name(workload, descs, n, k):
    names = {}
    for d in descs:
        m = d()
        key = m.name() + ("(%d)" % m._param() if m._param() else "")
        names[key] = names.get(key, 0) + 1
    return "%s: %s, N=%d rows x K=%d groups x D=%d features" % (
        workload.upper(), " + ".join("%d x %s" % (c, nm) for nm, c in names.items()), n, k, len(descs))


def parity_check(st, descs, hp_by_feature, view, gids, k, alpha, seed, sweep_idx, rows, ncores):
    """In-run spot check of the state the timed steps left behind (untimed): the CPU oracle rebuilds the suffstats
    from the GPU's own assignments (add_value of every row), scores a sample of rows against them, and replays the
    draw from the GPU's own score bits and the same Philox uniforms."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ol
    orc = ol.load()
    t0 = time.perf_counter()
    hp = np.concatenate([orc.flat_hp(d, hp_by_feature) for d in descs])
    gids = np.asarray(gids)
    cols = np.searchsorted(gids, st.assignments()).astype(np.int32)
    n = cols.shape[0]
    ss, counts = ol.build_suffstats(orc, descs, hp, view, cols, k)
    counts_exact = bool(all(st.groupsize(int(g)) == int(counts[c]) for c, g in enumerate(gids)))
    rows = min(rows, n)
    lo = (n // 2) // 1024 * 1024
    if lo + rows > n:
        lo = 0
    hi = lo + rows
    res = st.sweep(lo, hi, seed=seed, sweep=sweep_idx)        # the production sweep on the sample: same kernels, same K and D
    S = st.read_last_scores()
    want = orc.score_rows(descs, hp, ss, ol.logprior(counts, alpha), view, lo, hi, nthreads=ncores)
    den = np.maximum(1.0, np.abs(want))
    err = float(np.max(np.abs(S - want) / den))
    abs_err = float(np.max(np.abs(S - want)))
    u = orc.philox_u01_rows(seed, lo, rows, sweep_idx)
    new_cols = np.searchsorted(gids, st.assignments()[lo:hi]).astype(np.int32)
    draws = orc.sample_rows(S, u)
    libm = orc.sample_rows_libm(S, u)
    return {"rows": int(rows), "row_lo": int(lo), "groups": int(k), "features": len(descs),
            "max_rel_err": err, "max_abs_err": abs_err, "rel_err_is": "|gpu - oracle| / max(1, |oracle|) per (row, group) score, oracle = fp64 closed forms",
            "tolerance": 1e-5, "draws_bit_exact": bool(np.array_equal(new_cols, draws)),
            "draws_differing_under_glibc_expf": int((libm != new_cols).sum()),
            "group_counts_exact": counts_exact, "moved_in_sample": int(res["moved"]),
            "ok": bool(err < 1e-5 and np.array_equal(new_cols, draws) and counts_exact),
            "seconds": time.perf_counter() - t0}


def replica_check(st, device, n_total, world):
    """every rank must hold bit-identical suffstats after the timed steps: all-gather of a position-weighted 64-bit
    checksum of the resident suffstat buffer; the group sizes must add up to the global row count"""
    import torch
    import torch.distributed as dist
    from common_b200 import dist as cbd
    ptr, cnt = st.suffstat_buffer()
    t = cbd.as_tensor(ptr, cnt, device)
    bits = t.view(torch.int64)
    w = (torch.arange(cnt, device=device, dtype=torch.int64) * 0x9E3779B1 + 1) | 1
    h = (bits * w).sum().reshape(1)                     # wraps modulo 2^64
    hs = [torch.zeros_like(h) for _ in range(world)]
    if world > 1:
        dist.all_gather(hs, h)
    else:
        hs = [h]
    vals = [int(x.item()) for x in hs]
    kmax = st.max_groups
    return {"identical": bool(len(set(vals)) == 1), "hash": "%016x" % (vals[0] & 0xFFFFFFFFFFFFFFFF), "ranks": world,
            "group_sizes_sum": int(round(float(t[:kmax].sum().item()))), "rows_total": int(n_total)}


DUMP_BYTES = 60 << 20   # --dump-outputs writes at most this much in all (64 MB less room for the .npy headers)


def dump_outputs(out_dir, tag, st, device, budget):
    """Writes what the last timed step left for a caller of the sweep as out_dir/<tag>_<name>.npy, in at most `budget`
    bytes: the group ids and sizes, every row's group id, a sample of the rows of the score matrix (of its last chunk of
    rows where the step scored in chunks) and the resident suffstats.  Where an array does not fit, a sample of it is
    written, drawn from a fixed seed: the same arguments give the same inputs and the same sample on every run, so two
    builds can be compared array for array.  The score matrix is read through the library's own reader, which knows
    the layout the step left it in; that is one host copy of the last chunk (a few GB at full size), untimed."""
    t0 = time.perf_counter()
    rng = np.random.default_rng(20_000)

    def sample(n, cap):
        return np.arange(n) if n <= cap else np.sort(rng.choice(n, max(1, int(cap)), replace=False))

    groups = np.asarray(st.groups(), np.int64)
    out = {"group_ids": groups.astype(np.float64),
           "group_sizes": np.asarray([st.groupsize(int(g)) for g in groups], np.float64)}
    left = budget - sum(a.nbytes for a in out.values())
    a = st.assignments()
    assert np.all(np.abs(a) < (1 << 24)), "group ids beyond the integers float32 holds exactly"
    out["assignments"] = a[sample(a.size, left // 2 // 4)].astype(np.float32)
    S = st.read_last_scores()
    out["scores"] = S[sample(S.shape[0], left // 4 // (4 * max(1, S.shape[1])))].astype(np.float32)
    del S
    ptr, cnt = st.suffstat_buffer()
    ss = np.empty(cnt, np.float64)
    if cnt:
        from common_b200 import dist as cbd
        ss = cbd.as_tensor(ptr, cnt, device).cpu().numpy()
    out["suffstats"] = ss[sample(cnt, left // 4 // 8)]
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in out.items():
        np.save(os.path.join(out_dir, "%s_%s.npy" % (tag, name)), arr)
    return {"shapes": {name: list(arr.shape) for name, arr in out.items()}, "seconds": time.perf_counter() - t0}


def run_config(ctx, device, stream, comm, workload, args, rank, local_rank, world, scaling, peaks, want_e2e, want_parity,
               want_kernels, want_cpu, dump_budget=0):
    """one BASELINE.json configuration: data, state, warm-up, timed steps, (e2e), (parity), (per-kernel HBM records)"""
    import torch
    import torch.distributed as dist
    import common_b200 as cb
    from common_b200 import dist as cbd

    t_cfg0 = time.perf_counter()
    rows_override = args.rows if workload.upper() == args.workload.upper() else 0
    groups_override = args.groups if workload.upper() == args.workload.upper() else 0
    cfg, descs, storage, n, k, arr, z, row_off, n_total = build_workload(workload, rows_override, groups_override, rank, world, scaling)
    D = len(descs)
    warmup = max(args.warmup, 3)
    steps = args.steps
    view = cb.numpy_dataview(arr)
    st = cb.state(ctx, descs, max_groups=k + 8, cluster_hp={"alpha": 1.0})
    st.max_groups = k + 8
    if cfg.get("hp"):
        for d in range(D):
            st.set_component_hp(d, cfg["hp"])
    st.bind(view)
    gids = np.asarray([st.create_group() for _ in range(k)])
    if world > 1:
        cbd.add_values_sharded(st, gids[z], device, comm, n_total)   # local rows -> delta buffer -> all-reduce -> every replica applies the sum
    else:
        st.add_values(gids[z])

    def step(i, s_=None):
        # everything is enqueued on the stream; nothing in a step waits for the device
        s_ = s_ or st
        if world > 1:
            r = s_.sweep(seed=73, sweep=i, row_id_offset=row_off, defer_apply=True, wait=False)
            s_.allreduce_deltas(comm, n_total)       # ncclAllReduce inside the library, on its stream, then apply
        else:
            r = s_.sweep(seed=73, sweep=i, wait=False)
        return r

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    for i in range(warmup):
        step(i)
    clocks = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        clocks.start()
    launches0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    phase = {"build": 0.0, "score": 0.0, "sample": 0.0, "update": 0.0, "apply": 0.0}
    units = 0
    e0.record(stream)
    for i in range(steps):
        r = step(warmup + i)
        units += r["units"]
    e1.record(stream)
    barrier()
    ms_total = e0.elapsed_time(e1)
    timed = min(steps, 64)   # the library keeps the phase events of the last 64 sweeps
    for back in range(timed):
        for kk, v in st.last_timings(back).items():
            phase[kk] += v * steps / timed
    launches = ctx.launch_count() - launches0
    dumped = None
    if dump_budget and rank == 0:   # before any further sweep changes the state the last timed step left
        clocks.pause()              # the sampler is to see the GPU under this load, not idle during the dump's copies
        dumped = dump_outputs(args.dump_outputs, workload.upper() + ("_strong" if scaling == "strong" else ""), st, device,
                              dump_budget)
    t = torch.tensor([ms_total], device=device, dtype=torch.float64)
    u = torch.tensor([float(units)], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(u, op=dist.ReduceOp.SUM)
    ms_total = float(t.item()); units_all = float(u.item())
    # nvidia-smi cannot sample faster than ~100 ms: when the timed region is shorter than ~1.5 s, every rank keeps the
    # same step running (untimed; the same count on every rank, derived from the agreed time, because a step holds a
    # collective when N > 1) until the sampler has seen the GPU under this load
    extra = 0
    if ms_total < 1500.0:
        extra = int(min(4000, max(1, np.ceil((1500.0 - ms_total) / max(ms_total / steps, 1e-3)))))
        if dumped is not None:
            clocks.start()
        for j in range(extra):
            step(warmup + steps + j)
        barrier()
    clk = None
    if rank == 0:
        clk = clocks.stop()
        clk["sampled_over"] = "timed region" if extra == 0 else "timed region + %d more untimed steps of the same workload" % extra
    value = units_all / (ms_total * 1e-3)
    ld_scores = st.last_scores()[1]

    rec = {"workload": workload_name(workload, descs, n_total if scaling == "strong" else n, k), "name": workload.upper(),
           "scaling": scaling, "n_gpus": world, "rows_per_gpu": n, "rows_total": n_total, "groups": k, "features": D,
           "steps": steps, "warmup": warmup, "ms_per_step": ms_total / steps, "value": value, "unit": UNIT,
           "phase_ms_per_step": {kk: v / steps for kk, v in phase.items()}, "gpu_launches": int(launches), "clocks": clk}
    if dumped:
        rec["dumped_outputs"] = dumped

    # ---- replicas (N > 1): bit-identical suffstats on every rank, group sizes add up --------------------------------
    if world > 1:
        rec["replica_check"] = replica_check(st, device, n_total, world)
        msg = st.last_allreduce_bytes()
        cnt = st.suffstat_buffer()[1]
        rec["nvlink_bytes_per_step"] = {"message_bytes": int(msg), "dtype": "int32" if msg == 4 * cnt else "float64",
                                        "per_rank_sent_ring": int(2 * (world - 1) * msg // world),
                                        "collective": "one all-reduce(sum) of the flat suffstat-delta buffer per step"}

    # ---- e2e: the same step through the public API from HOST buffers -------------------
    # The reference re-reads its borrowed host rows on every pass (recarray/dataview.hpp:194-217); here one
    # pass over host rows is: H2D of the records (pinned) -> AoS->SoA conversion -> sweep (score + draw +
    # suffstat update, + all-reduce) -> assignments back to pinned host memory.  Groups, hypers and
    # suffstats stay resident in HBM between passes, as they stay resident in the reference's state object.
    if want_e2e:
        raw, mraw = view.raw()
        pinned = torch.from_numpy(raw).pin_memory()
        out_host = [torch.empty(n, dtype=torch.int64).pin_memory() for _ in range(2)]
        out_np = [t_.numpy() for t_ in out_host]
        from common_b200.dataview import device_dataview
        dv2 = device_dataview(ctx, data=pinned.data_ptr(), n=n, types=view.types())
        s2 = cb.state(ctx, descs, max_groups=k + 8, cluster_hp={"alpha": 1.0})
        if cfg.get("hp"):
            for d in range(D):
                s2.set_component_hp(d, cfg["hp"])
        s2.bind(dv2)
        g2 = np.asarray([s2.create_group() for _ in range(k)])
        if world > 1:
            cbd.add_values_sharded(s2, g2[z], device, comm, n_total)
        else:
            s2.add_values(g2[z])

        dv2.upload(pinned.data_ptr())                # the first pass's records
        s2.prefetch()

        def e2e_step(i):
            # one ABI call per pass (msb_state_pass): refresh (this pass's columns, converted on the copy stream, become
            # current) -> H2D of the NEXT pass's records + their AoS -> SoA conversion into the second column buffer
            # (copy stream, under this pass's sweep) -> sweep (+ all-reduce) -> the previous pass's assignments have
            # landed in pinned memory -> D2H of this pass's assignments starts on the copy stream
            rr = s2.run_pass(seed=73, sweep=i, row_id_offset=row_off, next_data=pinned.data_ptr(), assign_out=out_np[i & 1],
                             comm=comm, global_rows=n_total)
            return rr["units"]

        for i in range(3):
            e2e_step(1000 + i)
        barrier()
        t0 = time.perf_counter()
        eu = 0
        # at least ~60 ms of passes: a handful of 2 ms passes timed by the host clock is mostly pipeline fill and jitter
        # (C2: 2.04 ms per pass over 20 passes, 2.18 over 5).  The count comes from the agreed step time: the same on every rank.
        esteps = max(3, steps, int(min(200, np.ceil(60.0 / max(ms_total / steps, 1e-3)))))
        for i in range(esteps):
            eu += e2e_step(2000 + i)
        s2.assignments_wait()                        # the last pass's result is on the host
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], device=device, dtype=torch.float64)
        uu = torch.tensor([float(eu)], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dist.all_reduce(uu, op=dist.ReduceOp.SUM)
        e2e_phase = {}
        for back in range(min(esteps, 16)):     # device phase times of the end-to-end passes themselves (the library's event ring)
            for kk, v in s2.last_timings(back).items():
                e2e_phase[kk] = e2e_phase.get(kk, 0.0) + v / min(esteps, 16)
        rec["e2e"] = {"value": float(uu.item()) / float(tt.item()), "unit": UNIT, "device_phase_ms_per_pass": e2e_phase,
                      "h2d_bytes_per_step": int(raw.nbytes), "d2h_bytes_per_step": int(n * 8),
                      "ms_per_step": float(tt.item()) * 1e3 / esteps, "steps": esteps,
                      "what": "per pass: one H2D of the host AoS records (pinned) + AoS->SoA conversion, both for the NEXT pass on a copy stream under this pass's sweep (double-buffered columns) -> sweep (score, draw, suffstat update"
                              + (", all-reduce" if world > 1 else "") + ") -> int64 assignments to pinned host memory (copied on the copy stream, waited for during the next pass; the last one inside the timed region); groups/hypers/suffstats resident in HBM"}
        s2.close(); dv2.close()
        del pinned, out_host

    if rank == 0:
        hbm = float(peaks.get("hbm_gbs", 6650.0))
        hbm_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        score_ms = phase["score"] / steps
        abytes = algorithmic_bytes_score(descs, storage, n, k)
        achieved = abytes / (score_ms * 1e-3) / 1e9 if score_ms > 0 else 0.0
        traffic, wf, tr = None, None, None
        sm_count = torch.cuda.get_device_properties(device).multi_processor_count
        try:  # DRAM bytes per launch of this kernel from the committed ncu capture (same workload, same size)
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(workload.upper())
            if tr and tr.get("rows") == n:
                traffic = tr.get("dram_bytes_per_launch")
                wf = tr.get("smem_wavefronts_per_launch")
        except Exception:
            pass
        has_niw = any(d().name() == "niw" for d in descs)
        roof = {"kernel": "score_kernel", "bound": "hbm", "achieved": achieved, "peak": hbm, "unit": "GB/s",
                "frac": achieved / hbm, "traffic": traffic, "algorithmic_bytes_per_launch": abytes,
                "launch_ms": score_ms, "peak_source": hbm_src,
                "traffic_source": (tr or {}).get("capture") if traffic else None,
                "note": "score kernels reuse every loaded value K times: the binding roof is shared-memory lookup / FP32 issue rate, see DESIGN.md"}
        if wf and score_ms > 0 and clk and clk.get("sm_mhz"):
            # the pipe that really binds this kernel: one 128-byte shared-memory wavefront per SM per clock
            roof["binding_resource"] = "shared-memory wavefronts (LSU data pipe, 1 per SM per clock)"
            roof["binding_wavefronts_per_launch"] = wf
            roof["binding_frac"] = wf / (score_ms * 1e-3 * clk["sm_mhz"] * 1e6 * sm_count)
        if has_niw:
            dims = [d()._param() for d in descs if d().name() == "niw"]
            flops = sum(2.0 * dd_ * dd_ * n * k for dd_ in dims)   # whitened-GEMM form, SURVEY.md section 8(d)
            ach = flops / (score_ms * 1e-3) / 1e12
            f16_peak = float(peaks.get("bf16_tflops", 0.0)) or 2250.0
            roof = {"kernel": "niw_tc16_kernel (+ operand conversion)", "bound": "tensor", "achieved": ach, "peak": f16_peak, "unit": "TFLOP/s",
                    "frac": ach / f16_peak, "traffic": traffic, "algorithmic_flops_per_launch": flops, "launch_ms": score_ms,
                    "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst; fp16 runs at the bf16 rate)" if peaks.get("bf16_tflops") else "nominal 2250 TFLOP/s",
                    "traffic_source": (tr or {}).get("capture") if traffic else None,
                    "note": "3 fp16 products per algorithmic product (hi*hi + hi*lo + lo*hi, scaled operands) for fp32-class accuracy, less the structurally zero triangle of W_k: tensor-pipe work = 1.875 x the algorithmic FLOPs"}
        if tr:   # the pipes ncu saw busy in the committed full-size capture of this kernel (profiles/traffic.json)
            for kk in ("fma_pipe_pct", "xu_pipe_pct", "lsu_pipe_pct", "tensor_pipe_pct", "issue_active_pct"):
                if kk in tr:
                    roof["ncu_" + kk] = tr[kk]
        rec["roofline"] = roof

        # ---- the bandwidth-bound kernels, each against the HBM roof (one extra untimed step with an event pair per launch)
        if want_kernels and world == 1:
            ctx.profile(True)
            st.refresh()                                  # AoS records -> columns (ingest_tile_kernel) on the compute stream
            rr = st.sweep(seed=73, sweep=10_000)
            prof = ctx.profile_read()
            ctx.profile(False)
            rowsize = int(view.raw()[0].nbytes // max(n, 1))
            moved = int(rr["moved"])
            bx = sum((4 * d()._param() if d().name() in ("niw", "dm") else B_X.get(d().name(), 4)) for d in descs)
            ss_doubles = st.suffstat_buffer()[1]
            byts = {
                "ingest_tile_kernel": n * (rowsize + column_bytes(descs)),
                "sample_tile_kernel": n * (4.0 * ld_scores + 8),
                "sample_blocked_kernel": n * (4.0 * ld_scores + 8),
                "update_kernel": n * 8.0 + moved * bx,
                "commit_assign_kernel": n * 12.0,
                "apply_delta_kernel": ss_doubles * 8.0 * 4,
                "niw_colmax_kernel": n * 1.0 * bx if has_niw else 0,
                "niw_convert_a16_kernel": n * 2.0 * bx if has_niw else 0,
                "update_niw_kernel": n * 8.0 + moved * bx,
            }
            lst = []
            for name, (cnt, ms) in prof.items():
                e = {"kernel": name, "launches": cnt, "ms": ms}
                b = byts.get(name.split("<")[0])
                if b:
                    e["bytes"] = int(b)
                    e["gbs"] = b / (ms * 1e-3) / 1e9 if ms > 0 else None
                    e["frac"] = e["gbs"] / hbm if ms > 0 else None
                lst.append(e)
            rec["kernels_one_step"] = lst
            rec["roofline_hbm_bound"] = [e for e in lst if "bytes" in e]

        if want_parity and world == 1:
            try:
                rec["parity"] = parity_check(st, descs, cfg.get("hp"), view, gids, k, 1.0, 73, 20_000, args.parity_rows, usable_cores())
            except Exception as ex:  # a failed checker must not hide the measurement
                rec["parity"] = {"ok": False, "error": repr(ex)[:300]}

        if want_cpu and world == 1:
            c = cpu_reference_rate(descs, cfg.get("hp"), arr, z, k, args.cpu_seconds, 1)
            rec["cpu_baseline"] = {"value": c["value"], "unit": UNIT, "cores": c["cores"],
                                   "kind": "port", "api": c["kind"], "sample": c["sample"],
                                   "api_overhead_ns_per_call": c["noop_ns"],
                                   "api_overhead_note": "the reference's own noop model (models/noop.hpp) in the perf_group.cpp loop: "
                                                        "the floor the plugin API itself puts under any per-value implementation"}
    rec["l2"] = "no explicit flush: each step streams the %.0f MB score matrix (> 126 MB L2)" % (4.0 * n * ld_scores / 1e6)
    rec["wall_s"] = time.perf_counter() - t_cfg0
    st.close()
    del arr, view
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C2")
    ap.add_argument("--configs", default=None,
                    help="comma list of the configurations measured next to the headline (default: C2,C3,C4,C5 at N=1; "
                         "C2,C5 weak + C3 strong at N>1; 'none' = headline only)")
    ap.add_argument("--rows", type=int, default=0)
    ap.add_argument("--groups", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--parity-rows", type=int, default=2048)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps of every configuration, write what its last timed step computed as "
                         "DIR/<config>_<name>.npy (float32 / float64, %d MiB at most in all; rank 0)" % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the GPU path computed: --impl b200 only")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    import common_b200 as cb

    if args.impl == "reference":
        if rank != 0:
            return 0
        cfg, descs, storage, n, k, arr, z, _, _ = build_workload(args.workload, args.rows, args.groups, 0, 1, "weak")
        name = workload_name(args.workload, descs, n, k)   # the same workload as the b200 arm; each step times a bounded sample of its rows
        n = min(n, 200_000)
        arr, z = arr[:n], z[:n]
        ncores = usable_cores()
        hpx = cfg.get("hp")
        rates = []
        for i in range(args.warmup + args.steps):
            r = cpu_reference_rate(descs, hpx, arr, z, k, max(2.0, args.cpu_seconds / max(1, args.steps)), ncores)
            if i >= args.warmup:
                rates.append(r)
        val = float(np.mean([r["value"] for r in rates]))
        ms = float(np.mean([r["seconds"] for r in rates]) * 1e3)
        line = {"metric": METRIC, "value": val, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": name, "rows_per_step": rates[-1]["rows"], "groups": k, "features": len(descs),
                           "sample": "each step scores rows_per_step of the workload's rows against all K groups x D features"},
                "cpu_baseline": {"value": val, "unit": UNIT, "cores": rates[-1]["cores"], "kind": "port", "api": rates[-1]["kind"], "sample": rates[-1]["sample"]},
                "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist

    cores_mine = pin_rank_to_cores(local_rank, world)
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    # the library's own (non-blocking) stream becomes torch's current stream: the timing events, the NCCL
    # collectives and the library's kernels are all ordered on it
    ctx = cb.Context(local_rank)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=device)
    torch.cuda.set_stream(stream)
    comm = None
    if world > 1:
        from common_b200 import dist as cbd
        comm = cbd.NcclComm(ctx, rank, world)    # the library's own ncclComm_t: the delta all-reduce runs inside the C ABI
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass

    head = args.workload.upper()
    if args.configs is None:
        plan = [("C2", "weak"), ("C3", "weak"), ("C4", "weak"), ("C5", "weak")] if world == 1 else \
               [("C2", "weak"), ("C5", "weak"), ("C3", "strong")]
        if args.rows or args.groups:
            plan = []
    elif args.configs.lower() in ("none", ""):
        plan = []
    else:
        plan = []
        for c in args.configs.split(","):
            c = c.strip()
            if ":" in c:
                plan.append((c.split(":")[0].upper(), c.split(":")[1]))
            else:
                plan.append((c.upper(), "weak"))
    if not any(w == head and s == "weak" for w, s in plan):
        plan.insert(0, (head, "weak"))
    plan.sort(key=lambda p: 0 if (p[0] == head and p[1] == "weak") else 1)   # headline first

    records = []
    for w, scal in plan:
        is_head = (w == head and scal == "weak")
        rec = run_config(ctx, device, stream, comm, w, args, rank, local_rank, world, scal, peaks,
                         want_e2e=not args.no_e2e, want_parity=not args.no_parity, want_kernels=True,
                         want_cpu=is_head and not args.no_cpu,
                         dump_budget=DUMP_BYTES // len(plan) if args.dump_outputs else 0)
        records.append(rec)
        import gc
        gc.collect()
        torch.cuda.empty_cache()

    if rank == 0:
        h = records[0]
        flat = {}
        for r in records:
            tag = r["name"] + ("_strong" if r["scaling"] == "strong" else "")
            flat[tag + "_ms_per_step"] = round(r["ms_per_step"], 4)
            flat[tag + "_value"] = r["value"]
            if "roofline" in r:
                flat[tag + "_roofline_frac"] = round(r["roofline"]["frac"], 4)
                flat[tag + "_roofline_bound"] = r["roofline"]["bound"]
                flat[tag + "_score_ms"] = round(r["roofline"]["launch_ms"], 4)
            if "e2e" in r:
                flat[tag + "_e2e_value"] = r["e2e"]["value"]
                flat[tag + "_e2e_ms_per_step"] = round(r["e2e"]["ms_per_step"], 4)
            if "parity" in r:
                flat[tag + "_parity_max_rel_err"] = r["parity"].get("max_rel_err")
                flat[tag + "_parity_draws_bit_exact"] = r["parity"].get("draws_bit_exact")
                flat[tag + "_parity_ok"] = r["parity"].get("ok")
            if "replica_check" in r:
                flat[tag + "_replicas_identical"] = r["replica_check"]["identical"]
                flat[tag + "_group_sizes_sum_ok"] = r["replica_check"]["group_sizes_sum"] == r["replica_check"]["rows_total"]
        line = {"metric": METRIC, "value": h["value"], "unit": UNIT, "n_gpus": world, "steps": h["steps"], "warmup": h["warmup"],
                "ms_per_step": h["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": dict({"workload": h["workload"], "rows_per_gpu": h["rows_per_gpu"], "groups": h["groups"], "features": h["features"],
                                "step": "param build + score (N x K fp32 materialised) + sample + suffstat update" + (" + all-reduce" if world > 1 else ""),
                                "l2": h["l2"], "host_cores_per_rank": cores_mine}, **flat),
                "phase_ms_per_step": h["phase_ms_per_step"],
                "roofline": h.get("roofline"),
                "gpu_launches": h["gpu_launches"], "clocks": h["clocks"]}
        if "e2e" in h:
            line["e2e"] = h["e2e"]
        if "cpu_baseline" in h:
            line["cpu_baseline"] = h["cpu_baseline"]
        if "parity" in h:
            line["parity"] = h["parity"]
        if "replica_check" in h:
            line["replica_check"] = h["replica_check"]
            line["nvlink_bytes_per_step"] = h["nvlink_bytes_per_step"]
        if "roofline_hbm_bound" in h:
            line["roofline_hbm_bound"] = h["roofline_hbm_bound"]
        line["configs"] = records
        # the closing key: what a reader of the last ~1.5 KB of the line still sees
        parts = []
        for r in records:
            tag = r["name"] + ("/strong" if r["scaling"] == "strong" else "")
            s = "%s %.3fms %.3gu/s" % (tag, r["ms_per_step"], r["value"])
            if "roofline" in r:
                s += " roof(%s)=%.3f" % (r["roofline"]["bound"], r["roofline"]["frac"])
            if "e2e" in r:
                s += " e2e=%.3fms" % r["e2e"]["ms_per_step"]
            if "parity" in r and "max_rel_err" in r["parity"]:
                s += " err=%.1e draws=%s counts=%s" % (r["parity"]["max_rel_err"], "exact" if r["parity"]["draws_bit_exact"] else "DIFFER",
                                                       "exact" if r["parity"]["group_counts_exact"] else "DIFFER")
            if "replica_check" in r:
                s += " replicas=%s sizes=%d/%d" % ("identical" if r["replica_check"]["identical"] else "DIFFER",
                                                  r["replica_check"]["group_sizes_sum"], r["replica_check"]["rows_total"])
            parts.append(s)
        line["summary"] = "; ".join(parts)
        print(json.dumps(line))
    if comm is not None:
        comm.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
