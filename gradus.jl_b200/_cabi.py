"""ctypes mirror of include/gradus_b200.h and loader for libgradus_b200.so.

This is the same binding surface a Julia maintainer reaches with ``ccall`` (see
INTEGRATION.md).  There is no CPU fallback: if the CUDA library is missing or no
device is usable, every compute call raises."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libgradus_b200.so")

# ---- constants (include/gradus_b200.h) -------------------------------------
OK = 0
ERR_INVALID_ARGUMENT, ERR_NO_DEVICE, ERR_CUDA, ERR_UNSUPPORTED, ERR_NOMEM = -1, -2, -3, -4, -5
STATUS_OUT_OF_DOMAIN, STATUS_WITHIN_INNER_BOUNDARY, STATUS_INTERSECTED, STATUS_NO_STATUS = 0, 1, 2, 3
METRIC_KERR, METRIC_JP, METRIC_JOHANNSEN, METRIC_BUMBLEBEE, METRIC_KERR_NEWMAN, METRIC_MORRIS_THORNE, METRIC_DILATON_AXION = 0, 1, 2, 3, 4, 5, 6
GEOMETRY_NONE, GEOMETRY_THIN_DISC, GEOMETRY_SHAKURA_SUNYAEV, GEOMETRY_DATUM_PLANE, GEOMETRY_THICK_TABLE = 0, 1, 2, 3, 4
GEOMETRY_TARGET_POINT = 5  # gb200_trace_target only
GEOMETRY_THIN_DISC_ORDER = 6  # ImageOrder(ThinDisc, n): params inner_radius, outer_radius, n
CALLBACK_NONE, CALLBACK_UPPER_HEMISPHERE = 0, 1
POW_EXACT, POW_FAST32 = 0, 1
IC_RENDER_GRID, IC_POLAR_PLANE, IC_EXPLICIT, IC_CARTESIAN_PLANE, IC_IMPACT_PARAMETERS = 0, 1, 2, 3, 4
GRID_LINEAR, GRID_GEOMETRIC, GRID_INVERSE = 0, 1, 2
PF_SHADOW, PF_REDSHIFT, PF_DISC_RADIUS, PF_COORDINATE_TIME, PF_STATUS, PF_AFFINE_TIME, PF_RADIUS = 0, 1, 2, 3, 4, 5, 6
PF_EQUATORIAL_CROSSINGS = 7
EMISSIVITY_POWERLAW, EMISSIVITY_TABLE = 0, 1
PROFILE_TIME_NAN_LINEAR, PROFILE_TIME_LINEAR = 0, 1
FLAG_MAXITERS, FLAG_DT_MIN, FLAG_UNSTABLE = 1, 2, 4

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)


class Problem(C.Structure):
    _fields_ = [
        ("metric_kind", C.c_int32), ("geometry_kind", C.c_int32), ("callback_kind", C.c_int32), ("pow_mode", C.c_int32),
        ("metric_params", C.c_double * 8), ("observer", C.c_double * 4), ("geometry_params", C.c_double * 4),
        ("gtol", C.c_double), ("chart_inner", C.c_double), ("chart_outer", C.c_double), ("callback_delta", C.c_double),
        ("lambda_min", C.c_double), ("lambda_max", C.c_double), ("abstol", C.c_double), ("reltol", C.c_double),
        ("dtmax", C.c_double), ("mu", C.c_double), ("maxiters", C.c_int64),
    ]


class IC(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("grid_kind", C.c_int32), ("width", C.c_int64), ("height", C.c_int64),
        ("lo0", C.c_double), ("hi0", C.c_double), ("lo1", C.c_double), ("hi1", C.c_double),
        ("x", _dp * 4), ("v", _dp * 4), ("n", C.c_int64),
    ]


class Range(C.Structure):
    """Slot n holds ray first + (n // block) * stride * block + n % block (include/gradus_b200.h)."""

    _fields_ = [("first", C.c_int64), ("count", C.c_int64), ("stride", C.c_int64), ("block", C.c_int64)]

    def __init__(self, first=0, count=0, stride=1, block=1):
        super().__init__(first, count, stride, block)

    def indices(self):
        n = np.arange(self.count, dtype=np.int64)
        b = max(self.block, 1)
        return self.first + (n // b) * (self.stride * b) + n % b


class Endpoints(C.Structure):
    _fields_ = [
        ("status", _ip), ("lambda_max", _dp), ("x", _dp * 4), ("v", _dp * 4), ("x_init", _dp * 4), ("v_init", _dp * 4),
        ("naccept", _ip), ("nreject", _ip), ("flags", _ip),
    ]


class Emissivity(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n", C.c_int32), ("index", C.c_double), ("r", _dp), ("eps", _dp)]


class PlungingTable(C.Structure):
    _fields_ = [("n", C.c_int32), ("r", _dp), ("ut", _dp), ("ur", _dp), ("uphi", _dp)]


class LineProfileOpts(C.Structure):
    _fields_ = [("min_re", C.c_double), ("max_re", C.c_double), ("normalise", C.c_int32), ("bin_right_closed", C.c_int32)]


class DiscProfile(C.Structure):
    """gb200_disc_profile: ε(ρ) and the source-to-disc arrival time t(ρ) of the binned lag transfer function."""

    _fields_ = [("emissivity", Emissivity), ("time_kind", C.c_int32), ("n", C.c_int32), ("r", _dp), ("t", _dp)]


class LagTransferOpts(C.Structure):
    _fields_ = [("E0", C.c_double), ("t0", C.c_double), ("energy_lims", C.c_double * 2), ("time_lims", C.c_double * 2),
                ("N_E", C.c_int32), ("N_t", C.c_int32)]


class TfBranches(C.Structure):
    """gb200_tf_branches: one InterpolatingTransferBranches, flattened (branch 2k lower, 2k+1 upper of radius k)."""

    _fields_ = [("n_radii", C.c_int32), ("reserved", C.c_int32), ("r_e", _dp), ("gmin", _dp), ("gmax", _dp),
                ("off", C.POINTER(C.c_int64)), ("gs", _dp), ("f", _dp), ("t", _dp)]


class TfModel(C.Structure):
    _fields_ = [("table", C.c_int32), ("n_radii", C.c_int32), ("radii", _dp), ("rmin", C.c_double), ("g_scale", C.c_double),
                ("profile", DiscProfile)]


class TfQuadOpts(C.Structure):
    _fields_ = [("h", C.c_double), ("t0", C.c_double), ("upscale", C.c_int32), ("npoints", C.c_int32), ("nodes", _dp),
                ("weights", _dp), ("normalise", C.c_int32), ("reserved", C.c_int32)]


class DualIC(C.Structure):
    """gb200_dual_ic: impact parameters with seeded partials (forward-mode traces)."""

    _fields_ = [("n", C.c_int64), ("npartials", C.c_int32), ("reserved", C.c_int32), ("alpha", _dp), ("beta", _dp),
                ("dalpha", _dp), ("dbeta", _dp), ("height", _dp)]


class DualOut(C.Structure):
    _fields_ = [("status", _ip), ("lambda_max", _dp), ("x", _dp * 4), ("v", _dp * 4), ("g", _dp), ("dg", _dp),
                ("rho", _dp), ("drho", _dp), ("naccept", _ip), ("nreject", _ip), ("flags", _ip)]


DUAL_NORM_WITH_PARTIALS, DUAL_NORM_VALUES_ONLY = 0, 1


class Stats(C.Structure):
    _fields_ = [
        ("kernel_ms", C.c_double), ("total_ms", C.c_double), ("rays", C.c_int64), ("steps_accepted", C.c_int64),
        ("steps_rejected", C.c_int64), ("launches", C.c_int64), ("flagged", C.c_int64),
    ]


#: every symbol include/gradus_b200.h declares
EXPORTED_SYMBOLS = (
    "gb200_version", "gb200_init", "gb200_destroy", "gb200_last_error", "gb200_get_stats", "gb200_validate",
    "gb200_isco", "gb200_radiative_efficiency", "gb200_trace", "gb200_trace_batch", "gb200_trace_path", "gb200_build_plunging_table", "gb200_render", "gb200_lineprofile",
    "gb200_render_batch", "gb200_render_device", "gb200_lineprofile_device", "gb200_fp64_peak", "gb200_fp64_issue_probe", "gb200_debug_rhs", "gb200_debug_math", "gb200_debug_math_lo",
    "gb200_trace_dual", "gb200_trace_dual_batch", "gb200_trace_target",
    "gb200_set_cross_section", "gb200_bucket2d", "gb200_comm_init", "gb200_comm_destroy", "gb200_comm_size", "gb200_comm_context", "gb200_comm_lineprofile", "gb200_comm_render",
    "gb200_lagtransfer", "gb200_comm_lagtransfer", "gb200_tf_lineprofile", "gb200_tf_lagtransfer",
)


def dptr(a):
    """double* of a C-contiguous float64 numpy array (None -> NULL)."""
    if a is None:
        return C.cast(None, _dp)
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_dp)


def iptr(a):
    if a is None:
        return C.cast(None, _ip)
    assert a.dtype == np.int32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_ip)


class DualArrays:
    """Caller-owned inputs and outputs of one forward-mode trace call plus the ctypes views handed to the library."""

    def __init__(self, alpha, beta, dalpha, dbeta, height=None):
        self.alpha = np.ascontiguousarray(alpha, np.float64)
        self.beta = np.ascontiguousarray(beta, np.float64)
        n = self.alpha.size
        self.dalpha = np.ascontiguousarray(np.atleast_2d(np.asarray(dalpha, np.float64)))
        self.dbeta = np.ascontiguousarray(np.atleast_2d(np.asarray(dbeta, np.float64)))
        nd = self.dalpha.shape[0]
        if self.beta.shape != (n,) or self.dalpha.shape != (nd, n) or self.dbeta.shape != (nd, n) or nd not in (1, 2):
            raise ValueError("alpha, beta: (n,); dalpha, dbeta: (npartials, n) with npartials 1 or 2")
        self.height = None if height is None else np.ascontiguousarray(np.broadcast_to(np.asarray(height, np.float64), (n,)))
        self.n, self.npartials = n, nd
        self.ic = DualIC(n, nd, 0, dptr(self.alpha), dptr(self.beta), dptr(self.dalpha), dptr(self.dbeta), dptr(self.height))
        # one block for the outputs, pointers by address arithmetic (a numpy `.ctypes` view per array costs more than the rest)
        rows = 11 + 2 * nd  # lambda, x[4], v[4], g, rho, dg[nd], drho[nd]
        dbl, ints = np.zeros((rows, n)), np.zeros((4, n), np.int32)
        ints[0] = -1
        self._blocks = (dbl, ints)
        self.lambda_max, self.x, self.v, self.g, self.rho = dbl[0], dbl[1:5], dbl[5:9], dbl[9], dbl[10]
        self.dg, self.drho = dbl[11:11 + nd], dbl[11 + nd:11 + 2 * nd]
        self.status, self.naccept, self.nreject, self.flags = ints[0], ints[1], ints[2], ints[3]
        db, ib, dstep, istep = dbl.ctypes.data, ints.ctypes.data, 8 * n, 4 * n
        dp = lambda row: C.cast(db + row * dstep, _dp)  # noqa: E731
        ip = lambda row: C.cast(ib + row * istep, _ip)  # noqa: E731
        o = DualOut()
        o.status, o.lambda_max = ip(0), dp(0)
        for k in range(4):
            o.x[k], o.v[k] = dp(1 + k), dp(5 + k)
        o.g, o.rho, o.dg, o.drho = dp(9), dp(10), dp(11), dp(11 + nd)
        o.naccept, o.nreject, o.flags = ip(1), ip(2), ip(3)
        self.out = o


class EndpointArrays:
    """Caller-owned host SoA for `count` rays plus the ctypes view handed to the library."""

    def __init__(self, count, init=True, stats=True):
        n = int(count)
        # one block per element type, pointers by address arithmetic: building ~20 numpy `.ctypes` views per ensemble
        # cost more than tracing a thousand rays
        dbl = np.zeros((17 if init else 9, n))
        ints = np.zeros((4 if stats else 1, n), np.int32)
        ints[0] = -1
        self._blocks = (dbl, ints)
        self.lambda_max, self.x, self.v = dbl[0], dbl[1:5], dbl[5:9]
        self.x_init = dbl[9:13] if init else None
        self.v_init = dbl[13:17] if init else None
        self.status = ints[0]
        self.naccept, self.nreject, self.flags = (ints[1], ints[2], ints[3]) if stats else (None, None, None)
        db, ib, dstep, istep = dbl.ctypes.data, ints.ctypes.data, 8 * n, 4 * n
        null_d, null_i = C.cast(None, _dp), C.cast(None, _ip)
        e = Endpoints()
        e.status = C.cast(ib, _ip)
        e.lambda_max = C.cast(db, _dp)
        for k in range(4):
            e.x[k] = C.cast(db + (1 + k) * dstep, _dp)
            e.v[k] = C.cast(db + (5 + k) * dstep, _dp)
            e.x_init[k] = C.cast(db + (9 + k) * dstep, _dp) if init else null_d
            e.v_init[k] = C.cast(db + (13 + k) * dstep, _dp) if init else null_d
        e.naccept = C.cast(ib + istep, _ip) if stats else null_i
        e.nreject = C.cast(ib + 2 * istep, _ip) if stats else null_i
        e.flags = C.cast(ib + 3 * istep, _ip) if stats else null_i
        self.c = e


_lib = None


class GradusB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libgradus_b200 error {code}: {msg}")
        self.code = code


def load():
    """dlopen libgradus_b200.so and set prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GradusB200Error(ERR_NO_DEVICE, f"{LIB_PATH} not built; run __graft_entry__.build() (no CPU fallback exists)")
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    lib.gb200_version.restype = C.c_int
    lib.gb200_init.argtypes = [C.c_int, C.POINTER(vp)]
    lib.gb200_destroy.argtypes = [vp]
    lib.gb200_destroy.restype = None
    lib.gb200_last_error.argtypes = [vp]
    lib.gb200_last_error.restype = C.c_char_p
    lib.gb200_get_stats.argtypes = [vp, C.POINTER(Stats)]
    lib.gb200_validate.argtypes = [C.POINTER(Problem), C.POINTER(IC)]
    lib.gb200_isco.argtypes = [C.c_int32, _dp, _dp]
    lib.gb200_radiative_efficiency.argtypes = [C.c_int32, _dp, _dp]
    lib.gb200_trace.argtypes = [vp, C.POINTER(Problem), C.POINTER(IC), C.POINTER(Range), C.POINTER(Endpoints)]
    lib.gb200_trace_batch.argtypes = [vp, C.c_int32, C.POINTER(Problem), C.POINTER(IC), C.POINTER(Range), C.POINTER(Endpoints)]
    lib.gb200_trace_path.argtypes = [vp, C.POINTER(Problem), _dp, C.c_int32, _dp, _dp, _ip, _ip]
    lib.gb200_trace_target.argtypes = [vp, C.POINTER(Problem), C.POINTER(IC), C.POINTER(Range), _dp, C.c_double, C.POINTER(Endpoints), _dp]
    lib.gb200_build_plunging_table.argtypes = [vp, C.c_int32, _dp, C.c_int32, _dp, _dp, _dp, _dp, _ip]
    lib.gb200_render.argtypes = [vp, C.POINTER(Problem), C.POINTER(IC), C.POINTER(Range), _ip, C.c_int32,
                                 C.POINTER(PlungingTable), C.POINTER(_dp)]
    lib.gb200_lineprofile.argtypes = [vp, C.POINTER(Problem), C.POINTER(IC), C.POINTER(Range), C.POINTER(Emissivity),
                                      C.POINTER(PlungingTable), _dp, C.c_int32, C.POINTER(LineProfileOpts), _dp]
    lib.gb200_render_batch.argtypes = [vp, C.c_int32, C.POINTER(Problem), C.POINTER(IC), C.POINTER(Range), _ip, C.c_int32,
                                       C.POINTER(C.POINTER(PlungingTable)), C.POINTER(_dp)]
    lib.gb200_render_device.argtypes = [vp, C.POINTER(Problem), C.POINTER(IC), C.POINTER(Range), _ip, C.c_int32,
                                        C.POINTER(PlungingTable), C.POINTER(vp), vp, C.c_int]
    lib.gb200_lineprofile_device.argtypes = [vp, C.POINTER(Problem), C.POINTER(IC), C.POINTER(Range),
                                             C.POINTER(Emissivity), C.POINTER(PlungingTable), _dp, C.c_int32,
                                             C.POINTER(LineProfileOpts), vp, vp, C.c_int]
    lib.gb200_fp64_peak.argtypes = [vp, _dp]
    lib.gb200_fp64_issue_probe.argtypes = [vp, C.c_int32, _dp]
    lib.gb200_debug_rhs.argtypes = [vp, C.c_int32, _dp, C.c_int64, _dp, _dp]
    lib.gb200_debug_math.argtypes = [vp, C.c_int64, _dp, _dp]
    lib.gb200_debug_math_lo.argtypes = [vp, C.c_int64, _dp, _dp]
    lib.gb200_trace_dual.argtypes = [vp, C.POINTER(Problem), C.POINTER(DualIC), C.c_int32, C.POINTER(PlungingTable), C.POINTER(DualOut)]
    lib.gb200_trace_dual_batch.argtypes = [vp, C.c_int32, C.POINTER(Problem), C.POINTER(DualIC), C.c_int32,
                                           C.POINTER(C.POINTER(PlungingTable)), C.POINTER(DualOut)]
    lib.gb200_set_cross_section.argtypes = [vp, _dp, _dp, C.c_int32]
    lib.gb200_bucket2d.argtypes = [vp, C.c_int64, _dp, _dp, _dp, _dp, C.c_int32, _dp, C.c_int32, _dp]
    lib.gb200_comm_init.argtypes = [_ip, C.c_int32, C.POINTER(vp)]
    lib.gb200_comm_destroy.argtypes = [vp]
    lib.gb200_comm_destroy.restype = None
    lib.gb200_comm_size.argtypes = [vp]
    lib.gb200_comm_context.argtypes = [vp, C.c_int32]
    lib.gb200_comm_context.restype = vp
    lib.gb200_comm_lineprofile.argtypes = [vp, C.POINTER(Problem), C.POINTER(IC), C.POINTER(Emissivity), C.POINTER(PlungingTable), _dp, C.c_int32,
                                           C.POINTER(LineProfileOpts), _dp]
    lib.gb200_comm_render.argtypes = [vp, C.POINTER(Problem), C.POINTER(IC), _ip, C.c_int32, C.POINTER(PlungingTable), C.POINTER(_dp)]
    lag = [C.POINTER(Problem), C.POINTER(IC), C.POINTER(DiscProfile), C.POINTER(PlungingTable), C.POINTER(LagTransferOpts), _dp, _dp, _dp,
           C.POINTER(C.c_int64)]
    lib.gb200_lagtransfer.argtypes = [vp] + lag
    lib.gb200_comm_lagtransfer.argtypes = [vp] + lag
    tfq = [vp, C.c_int32, C.POINTER(TfBranches), C.c_int32, C.POINTER(TfModel), _dp, C.c_int32]
    lib.gb200_tf_lineprofile.argtypes = tfq + [C.POINTER(TfQuadOpts), _dp]
    lib.gb200_tf_lagtransfer.argtypes = tfq + [_dp, C.c_int32, C.POINTER(TfQuadOpts), _dp]
    for name in EXPORTED_SYMBOLS:
        fn = getattr(lib, name)
        if name not in ("gb200_destroy", "gb200_last_error", "gb200_version", "gb200_comm_destroy", "gb200_comm_context"):
            fn.restype = C.c_int
    _lib = lib
    return lib


def check(code, ctx=None):
    if code != OK:
        msg = load().gb200_last_error(ctx)
        raise GradusB200Error(code, msg.decode() if msg else "?")
