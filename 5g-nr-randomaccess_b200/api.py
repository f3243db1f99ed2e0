"""ctypes binding of librach_gpu (include/rach_gpu.h) -- the Python-side mirror of the C ABI.

The product path: RachSim -> ra_sim_create / ra_sim_run / ra_sim_stats in librach_gpu.so
(CUDA, sm_100a).  No CPU fallback: constructing a RachSim without a CUDA device raises.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RACH_GPU_LIB") or os.path.join(HERE, "librach_gpu.so")   # override: tuning builds only

RA_VARIANT_W, RA_VARIANT_U0, RA_VARIANT_N = 0, 1, 2
RA_DUMP_FIELDS = 16
HIST_DELAY, HIST_TX, HIST_FAIL = 0, 1, 2     # RA_HIST_*: timer, preambleTxCounter, failCount of the successful UEs
DUMP_NAMES = ["timer", "active", "txTime", "firstTxTime", "secondTxTime", "nowBackoff", "preamble",
              "preambleChange", "rarWindow", "maxRarCounter", "preambleTxCounter", "msg2Flag",
              "connectionRequest", "msg4Flag", "failCount", "sector"]


class RaParams(C.Structure):
    _fields_ = [("variant", C.c_int), ("nUE", C.c_int), ("distribution", C.c_int),
                ("nPreamble", C.c_int), ("backoffIndicator", C.c_int), ("nGrantUL", C.c_int),
                ("maxRarWindow", C.c_int), ("maxMsg2TxCount", C.c_int), ("accessTime", C.c_int),
                ("maxTimeMs", C.c_int), ("cellRadius", C.c_float), ("hBS", C.c_float),
                ("hUT", C.c_float), ("geometry", C.c_int), ("seed", C.c_ulonglong)]


class RaStats(C.Structure):
    _fields_ = [("simTimeMs", C.c_int), ("nSuccess", C.c_int), ("preambleTxSum", C.c_longlong),
                ("delaySum", C.c_longlong), ("failCountSum", C.c_longlong),
                ("continueFailed", C.c_longlong), ("finalSuccess", C.c_longlong),
                ("collisionPreambles", C.c_longlong), ("totalPreambleTxop", C.c_longlong),
                ("collisionScans", C.c_longlong), ("totalScans", C.c_longlong),
                ("updates", C.c_longlong), ("recordMoves", C.c_longlong)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


STATS_DTYPE = np.dtype([("simTimeMs", "<i4"), ("nSuccess", "<i4"), ("preambleTxSum", "<i8"),
                        ("delaySum", "<i8"), ("failCountSum", "<i8"), ("continueFailed", "<i8"),
                        ("finalSuccess", "<i8"), ("collisionPreambles", "<i8"),
                        ("totalPreambleTxop", "<i8"), ("collisionScans", "<i8"),
                        ("totalScans", "<i8"), ("updates", "<i8"), ("recordMoves", "<i8")])
assert STATS_DTYPE.itemsize == C.sizeof(RaStats)


class RaOptions(C.Structure):
    _fields_ = [("repOffset", C.c_int), ("dumpUEs", C.c_int), ("ctasPerSM", C.c_int),
                ("phaseTimers", C.c_int), ("histograms", C.c_int), ("reserved", C.c_int * 3)]


DUMP_CB = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_int, C.POINTER(RaStats), C.POINTER(C.c_int))

SYMBOLS = ["ra_sim_create", "ra_sim_create_ex", "ra_last_create_error", "ra_last_create_code", "ra_sim_run", "ra_sim_run_stream", "ra_sim_stats",
           "ra_sim_stats_all", "ra_sim_dump_ues", "ra_sim_geometry", "ra_sim_gains", "ra_sim_kernel_ms",
           "ra_sim_gpu_launches", "ra_sim_phase_cycles", "ra_sim_destroy", "ra_sim_last_error", "ra_params_default",
           "ra_horizon_ms", "ra_arrival_schedule", "ra_params_validate", "ra_version", "ra_hist_bins", "ra_sim_histogram"]

_lib = None


class RachError(RuntimeError):
    pass


def load_lib():
    """Load librach_gpu.so; raises loudly if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RachError("%s is missing: run `python __graft_entry__.py` (build()) first; "
                        "there is no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    lib.ra_sim_create.restype = vp
    lib.ra_sim_create.argtypes = [C.POINTER(RaParams), C.c_int, C.c_int, C.POINTER(C.c_int), C.c_int]
    lib.ra_sim_create_ex.restype = vp
    lib.ra_sim_create_ex.argtypes = [C.POINTER(RaParams), C.c_int, C.c_int, C.POINTER(C.c_int), C.c_int,
                                     C.POINTER(RaOptions)]
    lib.ra_last_create_error.restype = C.c_char_p
    lib.ra_sim_run.argtypes = [vp]
    lib.ra_sim_run_stream.argtypes = [vp, DUMP_CB, vp]
    lib.ra_sim_stats.argtypes = [vp, C.c_int, C.c_int, C.POINTER(RaStats)]
    lib.ra_sim_stats_all.argtypes = [vp, vp]
    lib.ra_sim_dump_ues.argtypes = [vp, C.c_int, C.c_int, vp]
    lib.ra_sim_geometry.argtypes = [vp, C.c_int, C.c_int, vp]
    lib.ra_sim_gains.argtypes = [vp, C.c_int, C.c_int, vp]
    lib.ra_sim_histogram.argtypes = [vp, C.c_int, C.c_int, vp]
    lib.ra_hist_bins.argtypes = [C.POINTER(RaParams), C.c_int]
    lib.ra_sim_kernel_ms.restype = C.c_double
    lib.ra_sim_kernel_ms.argtypes = [vp]
    lib.ra_sim_gpu_launches.restype = C.c_longlong
    lib.ra_sim_gpu_launches.argtypes = [vp]
    lib.ra_sim_phase_cycles.argtypes = [vp, vp]
    lib.ra_sim_destroy.argtypes = [vp]
    lib.ra_sim_destroy.restype = None
    lib.ra_sim_last_error.restype = C.c_char_p
    lib.ra_sim_last_error.argtypes = [vp]
    lib.ra_params_default.argtypes = [C.POINTER(RaParams), C.c_int]
    lib.ra_horizon_ms.argtypes = [C.POINTER(RaParams)]
    lib.ra_arrival_schedule.argtypes = [C.POINTER(RaParams), vp, C.c_int]
    lib.ra_params_validate.argtypes = [C.POINTER(RaParams), C.c_char_p, C.c_int]
    lib.ra_version.restype = C.c_char_p
    _lib = lib
    return lib


def default_params(**kw):
    """W defaults (RandomAccessWithNOMA.c:69-88) with overrides; variant=RA_VARIANT_N gives NOMA.c:41-57."""
    p = RaParams()
    load_lib().ra_params_default(C.byref(p), kw.get("variant", RA_VARIANT_W))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise AttributeError(k)
        setattr(p, k, v)
    return p


def validate_params(params):
    """(RA_OK, "") or (RA_E_INVAL, reason): the checks ra_sim_create applies, without a device."""
    buf = C.create_string_buffer(256)
    rc = load_lib().ra_params_validate(C.byref(params), buf, 256)
    return rc, buf.value.decode()


def hist_bins(params, kind):
    """Bins of histogram `kind` (HIST_*) for a point: horizon + 7 for HIST_DELAY, 256 otherwise; RA_E_INVAL (-1) for
    an unknown kind or HIST_FAIL on variant N / U0.  Needs no device."""
    return load_lib().ra_hist_bins(C.byref(params), kind)


def arrival_schedule(params):
    lib = load_lib()
    h = lib.ra_horizon_ms(C.byref(params))
    arr = np.zeros(h, dtype=np.int32)
    all_at = lib.ra_arrival_schedule(C.byref(params), arr.ctypes.data_as(C.c_void_p), h)
    return arr, all_at


class RachSim:
    """points x reps replications of the RACH state machine on the GPU(s)."""

    def __init__(self, points, reps=1, devices=None, rep_offset=0, dump_ues=False, ctas_per_sm=0, phase_timers=False,
                 histograms=False):
        lib = load_lib()
        self._lib = lib
        self.points = list(points)
        self.reps = int(reps)
        arr = (RaParams * len(self.points))(*self.points)
        opt = RaOptions(repOffset=rep_offset, dumpUEs=1 if dump_ues else 0, ctasPerSM=ctas_per_sm,
                        phaseTimers=1 if phase_timers else 0, histograms=1 if histograms else 0)
        if devices is None:
            dev, nd = None, 0
        else:
            dev, nd = (C.c_int * len(devices))(*devices), len(devices)
        self._h = lib.ra_sim_create_ex(arr, len(self.points), self.reps, dev, nd, C.byref(opt))
        if not self._h:
            raise RachError("ra_sim_create failed (%d): %s" % (lib.ra_last_create_code(), lib.ra_last_create_error().decode()))

    def _check(self, rc):
        if rc != 0:
            raise RachError("librach_gpu error %d: %s" % (rc, self._lib.ra_sim_last_error(self._h).decode()))

    def run(self):
        self._check(self._lib.ra_sim_run(self._h))
        return self

    def run_stream(self, on_replication):
        """ra_sim_run_stream: on_replication(point, rep, stats_dict, rows[nUE, 16]) is called for every replication as
        soon as it has finished on the GPU (completion order), while the kernel keeps running.  Needs dump_ues=True."""
        err = []

        def _cb(_user, point, rep, st, rows):
            try:
                n = self.points[point].nUE
                arr = np.ctypeslib.as_array(rows, shape=(n * RA_DUMP_FIELDS,)).reshape(n, RA_DUMP_FIELDS).copy()
                on_replication(point, rep, st.contents.as_dict(), arr)
            except Exception as e:      # never unwind through the C frames
                err.append(e)
        cb = DUMP_CB(_cb)
        self._check(self._lib.ra_sim_run_stream(self._h, cb, None))
        if err:
            raise err[0]
        return self

    def stats(self, point=0, rep=0):
        st = RaStats()
        self._check(self._lib.ra_sim_stats(self._h, point, rep, C.byref(st)))
        return st

    def stats_all(self):
        out = np.zeros(len(self.points) * self.reps, dtype=STATS_DTYPE)
        self._check(self._lib.ra_sim_stats_all(self._h, out.ctypes.data_as(C.c_void_p)))
        return out.reshape(len(self.points), self.reps)

    def dump_ues(self, point=0, rep=0):
        n = self.points[point].nUE
        out = np.zeros((n, RA_DUMP_FIELDS), dtype=np.int32)
        self._check(self._lib.ra_sim_dump_ues(self._h, point, rep, out.ctypes.data_as(C.c_void_p)))
        return out

    def geometry(self, point=0, rep=0):
        n = self.points[point].nUE
        out = np.zeros((n, 6), dtype=np.float32)
        self._check(self._lib.ra_sim_geometry(self._h, point, rep, out.ctypes.data_as(C.c_void_p)))
        return out

    def gains(self, point=0, rep=0):
        n = self.points[point].nUE
        out = np.zeros(n, dtype=np.float64)
        self._check(self._lib.ra_sim_gains(self._h, point, rep, out.ctypes.data_as(C.c_void_p)))
        return out

    def histogram(self, point, kind):
        """ra_sim_histogram: counts per value of `kind` (HIST_DELAY / HIST_TX / HIST_FAIL) over the UEs of `point` that
        finished, summed over its replications and devices.  Needs histograms=True and a run."""
        n = hist_bins(self.points[point], kind) if 0 <= point < len(self.points) else 1
        out = np.zeros(max(n, 1), dtype=np.uint64)
        self._check(self._lib.ra_sim_histogram(self._h, point, kind, out.ctypes.data_as(C.c_void_p)))
        return out

    def phase_cycles(self):
        out = np.zeros(10, dtype=np.uint64)
        self._check(self._lib.ra_sim_phase_cycles(self._h, out.ctypes.data_as(C.c_void_p)))
        return out

    @property
    def kernel_ms(self):
        return self._lib.ra_sim_kernel_ms(self._h)

    @property
    def gpu_launches(self):
        return self._lib.ra_sim_gpu_launches(self._h)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ra_sim_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
