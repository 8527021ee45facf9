"""Mixture-model state on the device -- the caller side of the hot path.

Method names and meaning follow the reference's entity_based_state_object
(include/microscopes/common/entity_state.hpp:25-90) and group_manager
(include/microscopes/common/group_manager.hpp:48-306); the batched calls
(score_rows, sweep) are the data-parallel form of the same loop.
"""
import ctypes as C

import numpy as np

from . import _lib


def _dbl(values):
    a = np.ascontiguousarray(np.asarray(values, dtype=np.float64).ravel())
    return a, a.ctypes.data_as(C.POINTER(C.c_double))


def flat_hp(model, hp):
    """one hp dict with the keys of model.default_hyperparams() as the flat vector of the C ABI (include/mscope_b200.h,
    enum msb_family): the values in that key order"""
    return np.concatenate([np.asarray(hp[k], np.float64).ravel() for k in model.default_hyperparams()])


def slice_hp_specs(hparams, cparam, nfeatures):
    """the msb_slice_hp_spec list of state.slice_hp: (feature, key, width, prior kind, a, b) per update, the features in
    the order given, each feature's keys in its dict's order with a tuple key expanded in place, then alpha as feature
    ``nfeatures``"""
    specs = []
    items = list((hparams or {}).items()) + [(nfeatures, {k: v}) for k, v in (cparam or {}).items()]
    for d, params in items:
        for key, (prior, width) in params.items():
            if not hasattr(prior, "kind"):
                raise TypeError("component %r, key %r: the prior must be one of common_b200.hyperprior's" % (d, key))
            for k in (key if isinstance(key, tuple) else (key,)):
                specs.append((int(d), k, float(width), int(prior.kind), prior.a, prior.b))
    return specs


class state(object):
    def __init__(self, ctx, models, max_groups=64, cluster_hp=None):
        self._ctx = ctx
        self._models = [m() for m in models]
        descs = (_lib.ModelDesc * len(self._models))(*[m.c_desc() for m in self._models])
        h = C.c_void_p()
        _lib.check(_lib.load().msb_state_create(ctx.handle, descs, len(self._models), int(max_groups), C.byref(h)))
        self._h = h
        self._view = None
        self._grid_sizes = {}     # component (or "alpha") -> number of grid points registered
        ctx._adopt(self)
        if cluster_hp is not None:
            self.set_cluster_hp(cluster_hp)

    @property
    def handle(self):
        return self._h

    def models(self):
        return list(self._models)

    # ---- data ---------------------------------------------------------------
    def bind(self, view):
        dev = view.to_device(self._ctx) if hasattr(view, "to_device") else view
        _lib.check(_lib.load().msb_state_bind(self._h, dev.handle))
        self._view = dev

    def refresh(self):
        """the bound device dataview was re-uploaded in place: convert its records again
        (assignments and suffstats are kept)"""
        _lib.check(_lib.load().msb_state_refresh(self._h))

    def prefetch(self):
        """after an upload: convert the new records on the copy stream into the second column buffer;
        the next refresh() only swaps buffers"""
        _lib.check(_lib.load().msb_state_prefetch(self._h))

    # ---- hyperparameters (entity_state.hpp:41-49) -----------------------------
    def set_cluster_hp(self, hp):
        _lib.check(_lib.load().msb_state_set_cluster_hp(self._h, b"alpha", float(hp["alpha"])))

    def get_cluster_hp(self):
        v = C.c_double()
        _lib.check(_lib.load().msb_state_get_cluster_hp(self._h, b"alpha", C.byref(v)))
        return {"alpha": v.value}

    def set_component_hp(self, component, hp):
        for key, val in hp.items():
            a, p = _dbl(val)
            _lib.check(_lib.load().msb_state_set_hp(self._h, component, key.encode(), p, a.size))

    def get_component_hp(self, component):
        out = {}
        for key, default in self._models[component].default_hyperparams().items():
            shape = np.shape(default)
            a = np.zeros(int(np.prod(shape)) if shape else 1, np.float64)
            _lib.check(_lib.load().msb_state_get_hp(self._h, component, key.encode(),
                                                    a.ctypes.data_as(C.POINTER(C.c_double)), a.size))
            out[key] = a.reshape(shape) if shape else float(a[0])
        return out

    def set_hp_raw(self, component, key, values):
        a, p = _dbl(values)
        _lib.check(_lib.load().msb_state_set_hp(self._h, component, key.encode(), p, a.size))

    # ---- hyperparameter inference on a grid (msb_state_hp_gibbs) ------------------------------------------------
    def set_hp_grid(self, component, points, log_prior=None):
        """register a grid for the component's hypers: ``points`` a list of hp dicts, ``log_prior`` the caller's log
        hyperprior at each point (default: uniform).  points=None removes the grid"""
        lib = _lib.load()
        if points is None or len(points) == 0:
            _lib.check(lib.msb_state_set_hp_grid(self._h, component, None, 0, 0, None))
            self._grid_sizes.pop(component, None)
            return
        flat = np.stack([flat_hp(self._models[component], p) for p in points])
        a, pa = _dbl(flat)
        lp, plp = _dbl(np.zeros(len(points)) if log_prior is None else log_prior)
        if lp.size != len(points):
            raise ValueError("one log prior per grid point: %d points, %d log priors" % (len(points), lp.size))
        _lib.check(lib.msb_state_set_hp_grid(self._h, component, pa, flat.shape[0], flat.shape[1], plp))
        self._grid_sizes[component] = flat.shape[0]

    def set_cluster_hp_grid(self, alphas, log_prior=None):
        """register a grid for the CRP concentration; alphas=None removes it"""
        lib = _lib.load()
        if alphas is None or len(alphas) == 0:
            _lib.check(lib.msb_state_set_cluster_hp_grid(self._h, None, 0, None))
            self._grid_sizes.pop("alpha", None)
            return
        a, pa = _dbl(alphas)
        lp, plp = _dbl(np.zeros(a.size) if log_prior is None else log_prior)
        if lp.size != a.size:
            raise ValueError("one log prior per grid point: %d points, %d log priors" % (a.size, lp.size))
        _lib.check(lib.msb_state_set_cluster_hp_grid(self._h, pa, a.size, plp))
        self._grid_sizes["alpha"] = a.size

    def hp_gibbs(self, seed=0, counter=0, weights=False):
        """one Gibbs step over every registered grid (features and alpha), drawn on the device and applied to the state.
        Returns {"choice": {component: index, ..., "alpha": index}} for the grids that exist, and with weights=True
        also "logw": {same keys: float64 array of log_prior + log marginal per point}"""
        D = len(self._models)
        choice = np.full(D + 1, -1, np.int64)
        out = _lib.HpGibbsOut(choice.ctypes.data, None, 0)
        logw = None
        if weights:
            logw = np.zeros((D + 1, max(self._grid_sizes.values(), default=1)))
            out.logw, out.logw_ld = logw.ctypes.data, logw.shape[1]
        opts = _lib.HpGibbsOpts(int(seed), int(counter))
        _lib.check(_lib.load().msb_state_hp_gibbs(self._h, C.byref(opts), C.byref(out)))
        keys = list(range(D)) + ["alpha"]
        res = {"choice": {keys[d]: int(choice[d]) for d in range(D + 1) if choice[d] >= 0}}
        if weights:
            res["logw"] = {k: logw[d][:self._grid_sizes[k]].copy() for d, k in enumerate(keys) if choice[d] >= 0}
        return res

    # ---- non-conjugate parameters (msb_state_theta / msb_state_redraw_empty) --------------------------------------
    def theta(self, tparams, seed=0, counter=0):
        """one slice-sampling update of every group's non-conjugate parameter, for the features in ``tparams``, the
        runner's {component: {"p": width}} (bbnc is the one family with such a parameter).  Returns the number of
        updates that reached the shrink cap and kept their value"""
        widths = np.zeros(len(self._models))
        for d, params in tparams.items():
            for key, w in params.items():
                if key != "p":
                    raise ValueError("component %d: no non-conjugate parameter %r (bbnc's is 'p')" % (d, key))
                widths[d] = w
        out = _lib.ThetaOut()
        opts = _lib.ThetaOpts(int(seed), int(counter), widths.ctypes.data, widths.size)
        _lib.check(_lib.load().msb_state_theta(self._h, C.byref(opts), C.byref(out)))
        return out.capped

    def redraw_empty(self, seed=0, counter=0):
        """every empty group's bbnc p drawn afresh from Beta(alpha, beta): the auxiliary groups of Neal's algorithm 8"""
        _lib.check(_lib.load().msb_state_redraw_empty(self._h, int(seed), int(counter)))

    # ---- slice sampling of continuous hypers (msb_state_slice_hp) ------------------------------------------------
    def slice_hp(self, hparams=None, cparam=None, seed=0, counter=0):
        """one slice-sampling update of every listed scalar hyper, on the device and applied to the state.
        ``hparams`` is the runner's {component: {key: (prior, width)}}, ``cparam`` {"alpha": (prior, width)}, with the
        priors of common_b200.hyperprior; a tuple key such as ("alpha", "beta") gives one update per key, in that order.
        Returns {"capped": updates that reached the shrink cap, "values": {component: {key: value}, "alpha": value}}"""
        specs = slice_hp_specs(hparams, cparam, len(self._models))
        arr = (_lib.SliceHpSpec * max(len(specs), 1))()
        keys = [key.encode() for _, key, _, _, _, _ in specs]       # kept alive for the call
        for i, (d, _, w, kind, a, b) in enumerate(specs):
            arr[i] = _lib.SliceHpSpec(d, keys[i], w, kind, a, b)
        values = np.zeros(max(len(specs), 1))
        out = _lib.SliceHpOut(0, values.ctypes.data)
        opts = _lib.SliceHpOpts(int(seed), int(counter), arr, len(specs))
        _lib.check(_lib.load().msb_state_slice_hp(self._h, C.byref(opts), C.byref(out)))
        res = {}
        for i, (d, key, _, _, _, _) in enumerate(specs):
            if d == len(self._models):
                res["alpha"] = float(values[i])
            else:
                res.setdefault(d, {})[key] = float(values[i])
        return {"capped": out.capped, "values": res}

    # ---- suffstats (entity_state.hpp:51-54) --------------------------------------
    def get_suffstats(self, component, gid, key, count=1):
        a = np.zeros(count, np.float64)
        _lib.check(_lib.load().msb_state_get_ss(self._h, component, gid, key.encode(),
                                                a.ctypes.data_as(C.POINTER(C.c_double)), count))
        return a

    def set_suffstats(self, component, gid, key, values):
        a, p = _dbl(values)
        _lib.check(_lib.load().msb_state_set_ss(self._h, component, gid, key.encode(), p, a.size))

    # ---- groups (entity_state.hpp:30-38,87-89) -------------------------------------
    def nentities(self):
        v = C.c_size_t()
        _lib.check(_lib.load().msb_state_nentities(self._h, C.byref(v)))
        return v.value

    def ngroups(self):
        v = C.c_size_t()
        _lib.check(_lib.load().msb_state_ngroups(self._h, C.byref(v)))
        return v.value

    def ncomponents(self):
        return len(self._models)

    def groups(self):
        n = self.ngroups()
        buf = (C.c_size_t * max(n, 1))()
        out = C.c_size_t()
        _lib.check(_lib.load().msb_state_groups(self._h, buf, n, C.byref(out)))
        return [int(buf[i]) for i in range(out.value)]

    def empty_groups(self):
        n = self.ngroups()
        buf = (C.c_size_t * max(n, 1))()
        out = C.c_size_t()
        _lib.check(_lib.load().msb_state_empty_groups(self._h, buf, n, C.byref(out)))
        return [int(buf[i]) for i in range(out.value)]

    def groupsize(self, gid):
        v = C.c_size_t()
        _lib.check(_lib.load().msb_state_groupsize(self._h, gid, C.byref(v)))
        return v.value

    def create_group(self, rng=None):
        v = C.c_size_t()
        _lib.check(_lib.load().msb_state_create_group(self._h, C.byref(v)))
        return v.value

    def delete_group(self, gid):
        _lib.check(_lib.load().msb_state_delete_group(self._h, gid))

    def assignments(self, out=None):
        """gid per entity (-1 = unassigned); ``out``: optional int64 array (e.g. over pinned memory)"""
        n = self.nentities()
        a = np.empty(n, np.int64) if out is None else out
        assert a.dtype == np.int64 and a.size == n and a.flags.c_contiguous
        _lib.check(_lib.load().msb_state_assignments(self._h, a.ctypes.data, n))
        return a

    def assignments_async(self, out):
        """enqueue the copy of the assignments into ``out`` (int64, pinned); valid after assignments_wait()"""
        assert out.dtype == np.int64 and out.size == self.nentities() and out.flags.c_contiguous
        _lib.check(_lib.load().msb_state_assignments_async(self._h, out.ctypes.data, out.size))

    def assignments_wait(self):
        _lib.check(_lib.load().msb_state_assignments_wait(self._h))

    # ---- membership (entity_state.hpp:57-72) ------------------------------------------
    def add_value(self, gid, eid, rng=None):
        _lib.check(_lib.load().msb_state_add_value(self._h, gid, eid))

    def remove_value(self, eid, rng=None):
        v = C.c_size_t()
        _lib.check(_lib.load().msb_state_remove_value(self._h, eid, C.byref(v)))
        return v.value

    def add_values(self, gids, defer_apply=False):
        """bulk add_value; defer_apply leaves the suffstat changes in the delta buffer (all-reduce, then apply_deltas)"""
        a = np.ascontiguousarray(gids, dtype=np.int64)
        fn = _lib.load().msb_state_add_values_deferred if defer_apply else _lib.load().msb_state_add_values
        _lib.check(fn(self._h, a.ctypes.data, a.size))

    def score_value(self, eid, rng=None):
        k = self.ngroups()
        gids = (C.c_size_t * max(k, 1))()
        scores = np.zeros(max(k, 1), np.float32)
        n = C.c_size_t()
        _lib.check(_lib.load().msb_state_score_value(self._h, eid, gids, scores.ctypes.data_as(C.POINTER(C.c_float)),
                                                     k, C.byref(n)))
        return [int(gids[i]) for i in range(n.value)], scores[:n.value]

    # ---- marginal likelihoods (entity_state.hpp:74-86) ------------------------------------
    def score_assignment(self):
        v = C.c_float()
        _lib.check(_lib.load().msb_state_score_assignment(self._h, C.byref(v)))
        return v.value

    def score_likelihood(self, component=None, gid=None, rng=None):
        """score_likelihood(component, gid): one group's score_data; score_likelihood(component): summed over
        the groups; score_likelihood(): summed over components too"""
        if component is not None and gid is not None:
            v = C.c_float()
            _lib.check(_lib.load().msb_state_score_likelihood(self._h, component, gid, C.byref(v)))
            return v.value
        per = (C.c_float * len(self._models))()
        tot = C.c_float()
        _lib.check(_lib.load().msb_state_score_likelihood_all(self._h, per, len(self._models), C.byref(tot)))
        return tot.value if component is None else float(per[component])

    def score_joint(self):
        """score_assignment() + score_likelihood() (the quantity the reference's testutil compares)"""
        return self.score_assignment() + self.score_likelihood()

    # ---- batched ---------------------------------------------------------------------
    def score_rows(self, row_lo=0, row_hi=None, out=None):
        """(gids, scores[nrows, K]): log(pseudocount) + sum_d score_value for every row"""
        row_hi = self.nentities() if row_hi is None else row_hi
        k = self.ngroups()
        gids = (C.c_size_t * max(k, 1))()
        n = C.c_size_t()
        if out is None:
            out = np.empty((row_hi - row_lo, k), np.float32)
        _lib.check(_lib.load().msb_state_score_rows(self._h, row_lo, row_hi, out.ctypes.data, out.strides[0] // 4 if out.size else k,
                                                    0, gids, k, C.byref(n)))
        return [int(gids[i]) for i in range(n.value)], out

    def score_rows_f64(self, row_lo=0, row_hi=None):
        """(gids, float64 scores[nrows, K]) from the fp64 closed-form path"""
        row_hi = self.nentities() if row_hi is None else row_hi
        k = self.ngroups()
        gids = (C.c_size_t * max(k, 1))()
        n = C.c_size_t()
        out = np.zeros((row_hi - row_lo, k), np.float64)
        _lib.check(_lib.load().msb_state_score_rows_f64(self._h, row_lo, row_hi, out.ctypes.data, k, gids, k, C.byref(n)))
        return [int(gids[i]) for i in range(n.value)], out

    def score_rows_device(self, row_lo=0, row_hi=None):
        """scores stay on the device; returns (gids, device pointer, ld)"""
        row_hi = self.nentities() if row_hi is None else row_hi
        k = self.ngroups()
        gids = (C.c_size_t * max(k, 1))()
        n = C.c_size_t()
        _lib.check(_lib.load().msb_state_score_rows(self._h, row_lo, row_hi, None, 0, 1, gids, k, C.byref(n)))
        ptr, ld = C.c_void_p(), C.c_size_t()
        _lib.check(_lib.load().msb_state_last_scores(self._h, C.byref(ptr), C.byref(ld), None, None))
        return [int(gids[i]) for i in range(n.value)], ptr.value, ld.value

    def sweep(self, row_lo=0, row_hi=None, seed=0, sweep=0, uniforms=None, row_id_offset=0, defer_apply=False,
              wait=True):
        """one batched (synchronous) reassignment pass: every row is scored against the same frozen suffstats -- its own
        contribution included -- and all rows move at once.  Approximate by construction (see msb_state_sweep in
        include/mscope_b200.h); the exact chain is remove_value / score_value / add_value per entity.
        wait=False only enqueues it (sweep_wait() collects ``moved``)"""
        row_hi = self.nentities() if row_hi is None else row_hi
        opts = _lib.SweepOpts(int(seed), int(sweep), int(row_id_offset), None, 1 if defer_apply else 0,
                              0 if wait else _lib.SWEEP_ASYNC)
        keep = None
        if uniforms is not None:
            keep = np.ascontiguousarray(uniforms, dtype=np.float32)
            assert keep.size == row_hi - row_lo
            opts.uniforms = keep.ctypes.data
        res = _lib.SweepResult()
        _lib.check(_lib.load().msb_state_sweep(self._h, row_lo, row_hi, C.byref(opts), C.byref(res)))
        return {"rows": res.rows, "moved": res.moved, "units": res.units}

    def sweep_wait(self):
        res = _lib.SweepResult()
        _lib.check(_lib.load().msb_state_sweep_wait(self._h, C.byref(res)))
        return {"rows": res.rows, "moved": res.moved, "units": res.units}

    def predict(self, row_lo=0, row_hi=None, *, responsibilities=False, map=False, draw=False, impute=False, seed=0,
                counter=0, row_id_offset=0, uniforms=None):
        """posterior predictive of rows [row_lo, row_hi) of the bound dataview against the current suffstats (an assigned
        row's own contribution included: not leave-one-out).  Returns a dict with ``gids`` (the columns), ``logp``
        (log p(x_observed | state), float64), and where asked ``resp`` (float32 [nrows, K], the sampler's own
        probabilities), ``map_gid``, ``draw_gid`` (the sweep's draw with sweep word ``counter``) and ``values`` (one array
        per feature, [nrows] or [nrows, dim]: observed cells as stored, masked cells drawn from the drawn group's
        posterior predictive).  Nothing of the state changes."""
        row_hi = self.nentities() if row_hi is None else row_hi
        n = row_hi - row_lo
        k = self.ngroups()
        widths = [m._param() if m.name() in ("niw", "dm") else 1 for m in self._models]
        res = {"logp": np.zeros(n, np.float64)}
        out = _lib.PredictOut()
        out.logp = res["logp"].ctypes.data
        if responsibilities:
            res["resp"] = np.zeros((n, k), np.float32)
            out.resp, out.resp_ld = res["resp"].ctypes.data, k
        if map:
            res["map_gid"] = np.zeros(n, np.int64)
            out.map_gid = res["map_gid"].ctypes.data
        if draw or impute:
            res["draw_gid"] = np.zeros(n, np.int64)
            out.draw_gid = res["draw_gid"].ctypes.data
        if impute:
            vals = np.zeros((n, sum(widths)), np.float64)
            out.values, out.values_ld = vals.ctypes.data, vals.shape[1]
        opts = _lib.PredictOpts(int(seed), int(counter), int(row_id_offset), None)
        keep = None
        if uniforms is not None:
            keep = np.ascontiguousarray(uniforms, dtype=np.float32)
            assert keep.size == n
            opts.uniforms = keep.ctypes.data
        gids = (C.c_size_t * max(k, 1))()
        nc = C.c_size_t()
        _lib.check(_lib.load().msb_state_predict(self._h, row_lo, row_hi, C.byref(opts), C.byref(out), gids, k, C.byref(nc)))
        res["gids"] = [int(gids[i]) for i in range(nc.value)]
        if impute:
            res["values"], off = [], 0
            for m, w in zip(self._models, widths):
                res["values"].append(vals[:, off:off + w] if m.name() in ("niw", "dm") else vals[:, off])
                off += w
        return res

    def last_scores(self):
        """(device pointer, ld, nrows, ncols) of the score matrix the last score/sweep call wrote"""
        ptr, ld, nr, nc = C.c_void_p(), C.c_size_t(), C.c_size_t(), C.c_size_t()
        _lib.check(_lib.load().msb_state_last_scores(self._h, C.byref(ptr), C.byref(ld), C.byref(nr), C.byref(nc)))
        return ptr.value, ld.value, nr.value, nc.value

    def read_last_scores(self):
        """host copy of the score matrix the last score/sweep call left on the device"""
        _, _, nr, nc = self.last_scores()
        out = np.empty((nr, nc), np.float32)
        if out.size:
            _lib.check(_lib.load().msb_state_read_last_scores(self._h, out.ctypes.data, nc))
        return out

    def last_timings(self, back=0):
        """ms per phase of the last sweep (back=0) or of an earlier one (ring of 64 sweeps)"""
        a = (C.c_float * 5)()
        _lib.check(_lib.load().msb_state_timings(self._h, int(back), a, 5))
        return dict(zip(("build", "score", "sample", "update", "apply"), [float(x) for x in a]))

    def delta_buffer(self):
        ptr, n = C.c_void_p(), C.c_size_t()
        _lib.check(_lib.load().msb_state_delta_buffer(self._h, C.byref(ptr), C.byref(n)))
        return ptr.value, n.value

    def delta_buffer_i32(self):
        """(device pointer or None, count): the pending deltas as exact int32 (integer-valued states only)"""
        ptr, n = C.c_void_p(), C.c_size_t()
        _lib.check(_lib.load().msb_state_delta_buffer_i32(self._h, C.byref(ptr), C.byref(n)))
        return ptr.value, n.value

    def delta_from_i32(self):
        _lib.check(_lib.load().msb_state_delta_from_i32(self._h))

    def suffstat_buffer(self):
        ptr, n = C.c_void_p(), C.c_size_t()
        _lib.check(_lib.load().msb_state_suffstat_buffer(self._h, C.byref(ptr), C.byref(n)))
        return ptr.value, n.value

    def apply_deltas(self):
        _lib.check(_lib.load().msb_state_apply_deltas(self._h))

    def allreduce_deltas(self, comm, global_rows=0):
        """ncclAllReduce(sum) of the pending deltas inside the library (comm: dist.NcclComm or a raw ncclComm_t),
        then apply: every replica ends with the same suffstats"""
        h = comm.handle if hasattr(comm, "handle") else comm
        _lib.check(_lib.load().msb_state_allreduce_deltas(self._h, h, int(global_rows)))

    def last_allreduce_bytes(self):
        v = C.c_size_t()
        _lib.check(_lib.load().msb_state_last_allreduce_bytes(self._h, C.byref(v)))
        return v.value

    def run_pass(self, seed=0, sweep=0, row_id_offset=0, next_data=None, next_mask=None, assign_out=None, comm=None,
                 global_rows=0):
        """one pass over host rows in one ABI call (msb_state_pass): refresh -> upload + prefetch of the next pass's
        records -> asynchronous sweep (-> delta all-reduce) -> assignments of this pass on their way to ``assign_out``
        (a pinned int64 array); next_data / next_mask are host addresses (pinned)"""
        po = _lib.PassOpts()
        po.sweep = _lib.SweepOpts(int(seed), int(sweep), int(row_id_offset), None, 0, 0)
        po.next_data = next_data
        po.next_mask = next_mask
        po.assign_out = assign_out.ctypes.data if assign_out is not None else None
        po.nccl_comm = (comm.handle if hasattr(comm, "handle") else comm) if comm is not None else None
        po.global_rows = int(global_rows)
        res = _lib.SweepResult()
        _lib.check(_lib.load().msb_state_pass(self._h, C.byref(po), C.byref(res)))
        return {"rows": res.rows, "moved": res.moved, "units": res.units}

    def sample_value(self, component, gid, seed, counter=0, n=1):
        """group::sample_value (models/base.hpp:29) for one (feature, group): ``n`` draws from the posterior predictive,
        draw i from the Philox stream (seed, counter + i).  Returns an array of n values (n x dim for niw)."""
        m = self._models[component]
        width = m._param() if m.name() == "niw" else 1
        out = np.zeros((n, width), np.float64)
        _lib.check(_lib.load().msb_state_sample_value(self._h, component, gid, seed, counter, n,
                                                      out.ctypes.data_as(C.POINTER(C.c_double))))
        return out if width > 1 else out[:, 0]

    # ---- checkpoint / resume: the reference's wire format (microscopes/io/schema.proto) -----------------
    _SS_KEYS = {"dm": ("counts", "ratio"), "bbnc": ("p", "heads", "tails"), "bb": ("heads", "tails"), "bnb": ("count", "sum"), "gp": ("count", "sum", "log_prod"),
                "nich": ("count", "mean", "count_times_variance"), "dd": ("counts",), "niw": ("count", "sum_x", "sum_xxT")}

    _WIRE_FLOAT_KEYS = ("p", "ratio", "log_prod", "mean", "count_times_variance", "sum_x", "sum_xxT")   # float32 on the wire

    def _ss_counts(self, m, key):
        p = m._param() or 0
        return {"counts": p, "sum_x": p, "sum_xxT": p * p}.get(key, 1)

    def get_component_hp_bag(self, component):
        """hypers::get_hp (distributions.hpp:355-361): the component's Shared message"""
        from . import wire
        m = self._models[component]
        hp = self.get_component_hp(component)
        vals = {k: (np.asarray(v).ravel().tolist() if np.ndim(v) else v) for k, v in hp.items()}
        return wire.encode(m.name() + ".Shared", vals)

    def get_suffstats_bag(self, component, gid):
        """group::get_ss (distributions.hpp:300-306): one group's Group message"""
        from . import wire
        m = self._models[component]
        vals = {}
        for key in self._SS_KEYS[m.name()]:
            n = self._ss_counts(m, key)
            v = self.get_suffstats(component, gid, key, n)
            vals[key] = v.tolist() if n > 1 or key in ("counts", "sum_x", "sum_xxT") else float(v[0])
        return wire.encode(m.name() + ".Group", vals)

    def suffstats_identifiers(self, component):
        """entity_state.hpp:52: the identifiers under which the component's suffstats are kept -- the group ids"""
        if not 0 <= component < len(self._models):
            raise IndexError("bad component index")
        return self.groups()

    def set_component_hp_bag(self, component, bag):
        """entity_state.hpp:47 / hypers::set_hp (distributions.hpp:363-369): from the component's Shared message"""
        from . import wire
        m = self._models[component]
        hp = wire.decode(m.name() + ".Shared", bag)
        self.set_component_hp(component, {k: hp[k] for k in m.default_hyperparams()})

    def set_suffstats_bag(self, component, gid, bag):
        """entity_state.hpp:54 / group::set_ss (distributions.hpp:308-314): from one group's Group message"""
        from . import wire
        m = self._models[component]
        ss = wire.decode(m.name() + ".Group", bag)
        for key in self._SS_KEYS[m.name()]:
            self.set_suffstats(component, gid, key, ss[key])

    def serialize(self):
        """MixtureModelState{hypers[], groups = GroupManager{alpha, assignments[], groups[GroupData{id, data =
        MixtureModelGroup{suffstats[]}}]}} -- group_manager.hpp:285-298 with the mixture model's group payload"""
        from . import wire
        D = len(self._models)
        groups = [{"id": g, "data": wire.encode("MixtureModelGroup", {"suffstats": [self.get_suffstats_bag(d, g) for d in range(D)]})}
                  for g in self.groups()]
        gm = wire.encode("GroupManager", {"alpha": self.get_cluster_hp()["alpha"], "assignments": self.assignments().tolist(),
                                          "groups": groups})
        return wire.encode("MixtureModelState", {"hypers": [self.get_component_hp_bag(d) for d in range(D)], "groups": gm})

    @classmethod
    def deserialize(cls, ctx, models, view, blob, max_groups=None):
        """the inverse: group identifiers, assignments, hypers and suffstats as saved (group_manager.hpp:71-105)"""
        from . import wire
        top = wire.decode("MixtureModelState", blob)
        gm = wire.decode("GroupManager", top["groups"])
        ngroups = len(gm["groups"])
        st = cls(ctx, models, max_groups=max_groups or (ngroups + 8), cluster_hp={"alpha": gm["alpha"]})
        for d, bag in enumerate(top["hypers"]):
            st.set_component_hp_bag(d, bag)
        st.bind(view)
        for g in gm["groups"]:
            _lib.check(_lib.load().msb_state_restore_group(st._h, int(g["id"])))
        a = np.asarray(gm["assignments"], np.int64)
        assert a.size == st.nentities(), "the checkpoint holds another number of entities"
        st.add_values(a)        # membership, and the suffstats the data implies in full fp64 ...
        # ... then the saved ones -- but only where they say something else.  The wire carries its real-valued fields as
        # float32 (nich mean / count_times_variance, niw sum_x / sum_xxT, gp log_prod, dm ratio, bbnc p): overwriting an
        # fp64 statistic with its own float32 rounding would leave every later remove_value subtracting exact row values
        # from rounded sums (residuals in emptied groups, a resumed chain 1e-7 away from the uninterrupted one).  A field
        # whose data-implied value rounds to what was saved is therefore kept as rebuilt; a real difference (the caller
        # saved something the data does not imply) is restored as saved.
        for g in gm["groups"]:
            gid = int(g["id"])
            bags = wire.decode("MixtureModelGroup", g["data"])["suffstats"]
            for d, bag in enumerate(bags):
                m = st._models[d]
                name = m.name()
                saved = wire.decode(name + ".Group", bag)
                for key in cls._SS_KEYS[name]:
                    cnt = st._ss_counts(m, key)
                    cur = np.asarray(st.get_suffstats(d, gid, key, cnt), np.float64).ravel()
                    want = np.atleast_1d(np.asarray(saved[key], np.float64)).ravel()
                    if key in cls._WIRE_FLOAT_KEYS:
                        same = cur.size == want.size and np.array_equal(cur.astype(np.float32), want.astype(np.float32))
                    else:
                        same = cur.size == want.size and np.array_equal(cur, want)
                    if not same:
                        st.set_suffstats(d, gid, key, saved[key])
        return st

    def close(self):
        if self._h:
            _lib.load().msb_state_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def sample_discrete_log(ctx, scores, uniforms):
    """util.hpp:138-143 for every row of ``scores`` with one uniform each, on the device"""
    s = np.ascontiguousarray(scores, dtype=np.float32)
    u = np.ascontiguousarray(uniforms, dtype=np.float32)
    out = np.zeros(s.shape[0], np.int32)
    _lib.check(_lib.load().msb_sample_discrete_log(ctx.handle, s.ctypes.data, s.shape[0], s.shape[1], s.shape[1],
                                                   u.ctypes.data, out.ctypes.data))
    return out


def philox_uniforms(ctx, seed, sweep, row_lo, n):
    out = np.zeros(n, np.float32)
    _lib.check(_lib.load().msb_philox_uniforms(ctx.handle, seed, sweep, row_lo, n, out.ctypes.data))
    return out
