"""ctypes binding of libmscope_b200.so (the C ABI of include/mscope_b200.h).

This is the Python-side counterpart of the reference's Cython declarations
(microscopes/_models_h.pxd, microscopes/common/recarray/_dataview_h.pxd): it
only declares prototypes and turns status codes into exceptions, the way the
reference maps C++ exceptions with ``except +`` (_models_h.pxd:10-19).

There is no fallback: if the CUDA library is missing this module raises.
"""
import ctypes as C
import os
import weakref

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libmscope_b200.so")

MSB_OK, MSB_ERR_INVALID, MSB_ERR_CUDA, MSB_ERR_NOMEM, MSB_ERR_UNSUPPORTED, MSB_ERR_KEY, MSB_ERR_STATE = range(7)

# type_info.h:10-34
TYPE_B, TYPE_I8, TYPE_U8, TYPE_I16, TYPE_U16, TYPE_I32, TYPE_U32, TYPE_I64, TYPE_U64, TYPE_F32, TYPE_F64 = range(11)
# distributions.hpp:58-64
FAMILY_BB, FAMILY_BNB, FAMILY_GP, FAMILY_NICH, FAMILY_DD, FAMILY_NIW, FAMILY_BBNC, FAMILY_DM = range(8)


class MsbError(RuntimeError):
    """The reference throws std::runtime_error; the ABI returns a status + message."""

    def __init__(self, status, message):
        super().__init__(message)
        self.status = status


class RuntimeType(C.Structure):
    _fields_ = [("prim", C.c_int32), ("n", C.c_uint32), ("vec", C.c_int32)]


class ModelDesc(C.Structure):
    _fields_ = [("family", C.c_int32), ("dim", C.c_uint32)]


class SweepOpts(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("sweep", C.c_uint64), ("row_id_offset", C.c_uint64),
                ("uniforms", C.c_void_p), ("defer_apply", C.c_int32), ("flags", C.c_int32)]


SWEEP_ASYNC = 1
NCCL_UNIQUE_ID_BYTES = 128


class PassOpts(C.Structure):
    _fields_ = [("sweep", SweepOpts), ("next_data", C.c_void_p), ("next_mask", C.c_void_p), ("assign_out", C.c_void_p),
                ("nccl_comm", C.c_void_p), ("global_rows", C.c_uint64)]


class SweepResult(C.Structure):
    _fields_ = [("rows", C.c_uint64), ("moved", C.c_uint64), ("units", C.c_uint64)]


class PredictOpts(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("counter", C.c_uint64), ("row_id_offset", C.c_uint64), ("uniforms", C.c_void_p)]


class PredictOut(C.Structure):
    _fields_ = [("logp", C.c_void_p), ("resp", C.c_void_p), ("resp_ld", C.c_size_t), ("map_gid", C.c_void_p),
                ("draw_gid", C.c_void_p), ("values", C.c_void_p), ("values_ld", C.c_size_t)]


_P = C.c_void_p
_SZ = C.c_size_t
_PROTOS = {
    # name: (restype, argtypes)
    "msb_last_error": (C.c_char_p, []),
    "msb_abi_version": (C.c_int, []),
    "msb_ctx_create": (C.c_int, [C.c_int, _P, C.POINTER(_P)]),
    "msb_ctx_destroy": (C.c_int, [_P]),
    "msb_ctx_synchronize": (C.c_int, [_P]),
    "msb_ctx_stream": (_P, [_P]),
    "msb_ctx_launch_count": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "msb_ctx_profile": (C.c_int, [_P, C.c_int]),
    "msb_ctx_profile_read": (C.c_int, [_P, C.c_char_p, _SZ, C.POINTER(_SZ)]),
    "msb_dataview_create": (C.c_int, [_P, _P, _P, _SZ, C.POINTER(RuntimeType), _SZ, C.c_int, C.POINTER(_P)]),
    "msb_dataview_upload": (C.c_int, [_P, _P, _P]),
    "msb_dataview_destroy": (C.c_int, [_P]),
    "msb_dataview_size": (C.c_int, [_P, C.POINTER(_SZ)]),
    "msb_dataview_nfeatures": (C.c_int, [_P, C.POINTER(_SZ)]),
    "msb_dataview_rowsize": (C.c_int, [_P, C.POINTER(_SZ), C.POINTER(_SZ)]),
    "msb_dataview_get_row": (C.c_int, [_P, _SZ, _P, _P]),
    "msb_dataview_permute": (C.c_int, [_P, C.c_uint64]),
    "msb_dataview_reset_permutation": (C.c_int, [_P]),
    "msb_dataview_permutation": (C.c_int, [_P, C.POINTER(C.c_uint64), _SZ]),
    "msb_state_create": (C.c_int, [_P, C.POINTER(ModelDesc), _SZ, _SZ, C.POINTER(_P)]),
    "msb_state_destroy": (C.c_int, [_P]),
    "msb_state_bind": (C.c_int, [_P, _P]),
    "msb_state_refresh": (C.c_int, [_P]),
    "msb_state_prefetch": (C.c_int, [_P]),
    "msb_state_set_hp": (C.c_int, [_P, _SZ, C.c_char_p, C.POINTER(C.c_double), _SZ]),
    "msb_state_get_hp": (C.c_int, [_P, _SZ, C.c_char_p, C.POINTER(C.c_double), _SZ]),
    "msb_state_set_ss": (C.c_int, [_P, _SZ, _SZ, C.c_char_p, C.POINTER(C.c_double), _SZ]),
    "msb_state_get_ss": (C.c_int, [_P, _SZ, _SZ, C.c_char_p, C.POINTER(C.c_double), _SZ]),
    "msb_state_set_cluster_hp": (C.c_int, [_P, C.c_char_p, C.c_double]),
    "msb_state_get_cluster_hp": (C.c_int, [_P, C.c_char_p, C.POINTER(C.c_double)]),
    "msb_state_nentities": (C.c_int, [_P, C.POINTER(_SZ)]),
    "msb_state_ngroups": (C.c_int, [_P, C.POINTER(_SZ)]),
    "msb_state_groups": (C.c_int, [_P, C.POINTER(_SZ), _SZ, C.POINTER(_SZ)]),
    "msb_state_empty_groups": (C.c_int, [_P, C.POINTER(_SZ), _SZ, C.POINTER(_SZ)]),
    "msb_state_groupsize": (C.c_int, [_P, _SZ, C.POINTER(_SZ)]),
    "msb_state_create_group": (C.c_int, [_P, C.POINTER(_SZ)]),
    "msb_state_delete_group": (C.c_int, [_P, _SZ]),
    "msb_state_restore_group": (C.c_int, [_P, _SZ]),
    "msb_state_assignments": (C.c_int, [_P, _P, _SZ]),
    "msb_state_assignments_async": (C.c_int, [_P, _P, _SZ]),
    "msb_state_assignments_wait": (C.c_int, [_P]),
    "msb_state_add_values": (C.c_int, [_P, _P, _SZ]),
    "msb_state_add_values_deferred": (C.c_int, [_P, _P, _SZ]),
    "msb_state_add_value": (C.c_int, [_P, _SZ, _SZ]),
    "msb_state_remove_value": (C.c_int, [_P, _SZ, C.POINTER(_SZ)]),
    "msb_state_score_value": (C.c_int, [_P, _SZ, C.POINTER(_SZ), C.POINTER(C.c_float), _SZ, C.POINTER(_SZ)]),
    "msb_state_score_rows": (C.c_int, [_P, _SZ, _SZ, _P, _SZ, C.c_int, C.POINTER(_SZ), _SZ, C.POINTER(_SZ)]),
    "msb_state_score_rows_f64": (C.c_int, [_P, _SZ, _SZ, _P, _SZ, C.POINTER(_SZ), _SZ, C.POINTER(_SZ)]),
    "msb_state_score_likelihood": (C.c_int, [_P, _SZ, _SZ, C.POINTER(C.c_float)]),
    "msb_state_score_likelihood_all": (C.c_int, [_P, C.POINTER(C.c_float), _SZ, C.POINTER(C.c_float)]),
    "msb_state_score_assignment": (C.c_int, [_P, C.POINTER(C.c_float)]),
    "msb_sample_discrete_log": (C.c_int, [_P, _P, _SZ, _SZ, _SZ, _P, _P]),
    "msb_philox_uniforms": (C.c_int, [_P, C.c_uint64, C.c_uint64, C.c_uint64, _SZ, _P]),
    "msb_selftest_expf": (C.c_int, [_P, _P, _SZ, _P]),
    "msb_selftest_expf2": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "msb_selftest_division": (C.c_int, [_P, C.c_uint64, _SZ, C.POINTER(C.c_uint64)]),
    "msb_selftest_skip_rule": (C.c_int, [_P, _P, _P, _P, _SZ, _P]),
    "msb_state_sweep": (C.c_int, [_P, _SZ, _SZ, C.POINTER(SweepOpts), C.POINTER(SweepResult)]),
    "msb_state_sweep_wait": (C.c_int, [_P, C.POINTER(SweepResult)]),
    "msb_state_predict": (C.c_int, [_P, _SZ, _SZ, C.POINTER(PredictOpts), C.POINTER(PredictOut), C.POINTER(_SZ), _SZ,
                                    C.POINTER(_SZ)]),
    "msb_state_delta_buffer": (C.c_int, [_P, C.POINTER(_P), C.POINTER(_SZ)]),
    "msb_state_apply_deltas": (C.c_int, [_P]),
    "msb_state_delta_buffer_i32": (C.c_int, [_P, C.POINTER(_P), C.POINTER(_SZ)]),
    "msb_state_delta_from_i32": (C.c_int, [_P]),
    "msb_state_suffstat_buffer": (C.c_int, [_P, C.POINTER(_P), C.POINTER(_SZ)]),
    "msb_nccl_version": (C.c_int, [C.POINTER(C.c_int)]),
    "msb_nccl_unique_id": (C.c_int, [_P]),
    "msb_nccl_comm_create": (C.c_int, [_P, C.c_int, C.c_int, _P, C.POINTER(_P)]),
    "msb_nccl_comm_destroy": (C.c_int, [_P]),
    "msb_state_allreduce_deltas": (C.c_int, [_P, _P, C.c_uint64]),
    "msb_state_last_allreduce_bytes": (C.c_int, [_P, C.POINTER(_SZ)]),
    "msb_state_pass": (C.c_int, [_P, C.POINTER(PassOpts), C.POINTER(SweepResult)]),
    "msb_state_last_scores": (C.c_int, [_P, C.POINTER(_P), C.POINTER(_SZ), C.POINTER(_SZ), C.POINTER(_SZ)]),
    "msb_state_read_last_scores": (C.c_int, [_P, _P, _SZ]),
    "msb_state_last_timings": (C.c_int, [_P, C.POINTER(C.c_float), _SZ]),
    "msb_state_timings": (C.c_int, [_P, _SZ, C.POINTER(C.c_float), _SZ]),
    "msb_value_score": (C.c_int, [_P, C.POINTER(ModelDesc), C.POINTER(C.c_double), _SZ, C.POINTER(C.c_double), _SZ,
                                  _P, C.POINTER(RuntimeType), C.POINTER(C.c_float)]),
    "msb_value_add": (C.c_int, [_P, C.POINTER(ModelDesc), C.POINTER(C.c_double), _SZ, C.POINTER(C.c_double), _SZ,
                                _P, C.POINTER(RuntimeType)]),
    "msb_value_remove": (C.c_int, [_P, C.POINTER(ModelDesc), C.POINTER(C.c_double), _SZ, C.POINTER(C.c_double), _SZ,
                                   _P, C.POINTER(RuntimeType)]),
    "msb_value_score_data": (C.c_int, [_P, C.POINTER(ModelDesc), C.POINTER(C.c_double), _SZ, C.POINTER(C.c_double), _SZ,
                                       C.POINTER(C.c_float)]),
    "msb_value_sample": (C.c_int, [_P, C.POINTER(ModelDesc), C.POINTER(C.c_double), _SZ, C.POINTER(C.c_double), _SZ,
                                   C.c_uint64, C.c_uint64, _SZ, C.POINTER(C.c_double)]),
    "msb_state_sample_value": (C.c_int, [_P, _SZ, _SZ, C.c_uint64, C.c_uint64, _SZ, C.POINTER(C.c_double)]),
    "msb_model_hp_size": (_SZ, [C.POINTER(ModelDesc)]),
    "msb_model_ss_size": (_SZ, [C.POINTER(ModelDesc)]),
}

EXPORTED_SYMBOLS = tuple(sorted(_PROTOS))

_lib = None


def load():
    """dlopen the in-tree CUDA library; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "%s is missing: build it with common_b200/csrc/build.sh (nvcc, sm_100a). "
            "There is no CPU fallback for this path." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status):
    if status != MSB_OK:
        msg = load().msb_last_error().decode("utf-8", "replace")
        raise MsbError(status, msg)


class Context:
    """Device + stream.  One per process per GPU."""

    def __init__(self, device=0, stream=None):
        lib = load()
        h = _P()
        check(lib.msb_ctx_create(int(device), _P(stream) if stream else None, C.byref(h)))
        self._h = h
        self.device = int(device)
        self._children = weakref.WeakSet()  # states / dataviews that must be released before the context

    @property
    def handle(self):
        if not self._h:
            raise MsbError(MSB_ERR_STATE, "context is closed")
        return self._h

    def _adopt(self, child):
        self._children.add(child)

    def synchronize(self):
        check(load().msb_ctx_synchronize(self._h))

    def stream(self):
        return load().msb_ctx_stream(self._h)

    def launch_count(self):
        v = C.c_uint64()
        check(load().msb_ctx_launch_count(self._h, C.byref(v)))
        return v.value

    def profile(self, enable=True):
        """per-kernel CUDA event pairs around every launch from now on (diagnostics; off by default)"""
        check(load().msb_ctx_profile(self._h, 1 if enable else 0))

    def profile_read(self):
        """{kernel name: (launches, total ms)} of the launches recorded since profile(True)"""
        need = _SZ()
        check(load().msb_ctx_profile_read(self._h, None, 0, C.byref(need)))
        buf = C.create_string_buffer(need.value + 16)
        check(load().msb_ctx_profile_read(self._h, buf, len(buf), C.byref(need)))
        out = {}
        for line in buf.value.decode().splitlines():
            name, cnt, ms = line.rsplit("\t", 2)
            out[name.strip("()")] = (int(cnt), float(ms))
        return out

    def close(self):
        if self._h:
            for child in list(self._children):
                child.close()
            load().msb_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
