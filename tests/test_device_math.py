"""Device math and scalar helpers point by point.

The step-level parity tests see the helpers of kid_b200/csrc only through whole steps (1e-5 per cell, a few outliers
allowed), where an f64 power off by hundreds of ulps or a decade index one bin off next to 10**n moves only a handful of
cells.  Here each helper is evaluated on the device, as compiled for the step, and held to a contract of its own:

* tests/device_probe.cu includes the product headers unchanged and is compiled with the library's flags
  (kid_b200.build.BASE_FLAGS); one elementwise kernel evaluates a helper by id, with the KConst of a handle
  (hostinit::compute) as a __grid_constant__ launch parameter and the node tables uploaded as kidmp_init does.
* The host twin is kidmp_fastmath.h compiled by g++ -O2 -ffp-contract=off (the algorithm the device copy in
  kidmp_math.cuh restates with its own coefficients), plus glibc's powf / expf / logf / log10f, which the oracle calls.

The contract of the f64 routines (asserted below, stated in DESIGN.md section 4 and kidmp_fastmath.h):
  dexp  < 1 ulp for |x| < 704 (table path); <= 1 ulp + the subnormal ulp outside it (library exp)
  dlog  < 1.5 ulp where |log x| > 0.1; absolute < 1.5e-17 where |log x| <= 0.1 (near 1 the error is absolute)
  dpow  < 3 * (1 + |y log x|) ulp, plus |y| * 1.5e-17 relative where |log x| <= 0.1
and the f32 wrappers (pow_f, exp_f, log10_f, pow10_f, log_f) are within one ulp of the correctly rounded result,
and equal to it except for a few double-rounding misses per million.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "kid_b200", "csrc")
HERE = os.path.dirname(os.path.abspath(__file__))
LD = np.longdouble
_dp = C.POINTER(C.c_double)
_fp = C.POINTER(C.c_float)

DBL_MIN = np.finfo(np.float64).tiny
DBL_MAX = np.finfo(np.float64).max

# ---------------------------------------------------------------------------------------------------------------------
# host twin: kidmp_fastmath.h and glibc's f32 functions as vector functions

TWIN_SRC = r'''
#include "kidmp_fastmath.h"
#include <math.h>
using namespace kidmp;
static double et[KFM_N];
static LogNode lt[KFM_N];
static int ready = 0;
static void init() { if (!ready) { kfm_build_tables(et, lt); ready = 1; } }
extern "C" {
void twin_exp(const double* x, double* r, long n) { init(); for (long i = 0; i < n; ++i) r[i] = kfm_exp(x[i], et); }
void twin_log(const double* x, double* r, long n) { init(); for (long i = 0; i < n; ++i) r[i] = kfm_log(x[i], lt); }
void twin_pow(const double* x, const double* y, double* r, long n) {
  init(); for (long i = 0; i < n; ++i) r[i] = kfm_exp(y[i] * kfm_log(x[i], lt), et);
}
void libm_powf(const float* x, const float* y, float* r, long n) { for (long i = 0; i < n; ++i) r[i] = powf(x[i], y[i]); }
void libm_expf(const float* x, float* r, long n) { for (long i = 0; i < n; ++i) r[i] = expf(x[i]); }
void libm_logf(const float* x, float* r, long n) { for (long i = 0; i < n; ++i) r[i] = logf(x[i]); }
void libm_log10f(const float* x, float* r, long n) { for (long i = 0; i < n; ++i) r[i] = log10f(x[i]); }
}
'''


class Twin:
    def __init__(self, path):
        self.L = C.CDLL(path)
        for n in ("twin_exp", "twin_log"):
            getattr(self.L, n).argtypes = [_dp, _dp, C.c_long]
        self.L.twin_pow.argtypes = [_dp, _dp, _dp, C.c_long]
        self.L.libm_powf.argtypes = [_fp, _fp, _fp, C.c_long]
        for n in ("libm_expf", "libm_logf", "libm_log10f"):
            getattr(self.L, n).argtypes = [_fp, _fp, C.c_long]

    def _call(self, fn, dtype, *args):
        a = [np.ascontiguousarray(v, dtype) for v in np.broadcast_arrays(*args)]
        out = np.empty(a[0].shape, dtype)
        ptr = _dp if dtype == np.float64 else _fp
        fn(*[v.ctypes.data_as(ptr) for v in a], out.ctypes.data_as(ptr), out.size)
        return out

    def exp(self, x): return self._call(self.L.twin_exp, np.float64, x)
    def log(self, x): return self._call(self.L.twin_log, np.float64, x)
    def pow(self, x, y): return self._call(self.L.twin_pow, np.float64, x, y)
    def powf(self, x, y): return self._call(self.L.libm_powf, np.float32, x, y)
    def expf(self, x): return self._call(self.L.libm_expf, np.float32, x)
    def logf(self, x): return self._call(self.L.libm_logf, np.float32, x)
    def log10f(self, x): return self._call(self.L.libm_log10f, np.float32, x)


def _build_twin(d):
    os.makedirs(d, exist_ok=True)
    src = os.path.join(d, "twin.cpp")
    with open(src, "w") as f:
        f.write(TWIN_SRC)
    so = os.path.join(d, "libtwin.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-I", CSRC, src,
                           "-o", so])
    return Twin(so)


@pytest.fixture(scope="session")
def twin(tmp_path_factory):
    return _build_twin(str(tmp_path_factory.mktemp("twin")))


# ---------------------------------------------------------------------------------------------------------------------
# error measures

def ulp_err64(got, ref):
    """|got - ref| in ulps of f64 at ref (ref in long double; below DBL_MIN the ulp is the subnormal one, 2**-1074)."""
    ref = np.asarray(ref, LD)
    _, e = np.frexp(np.abs(ref))
    ulp = np.ldexp(LD(1), np.maximum(e.astype(np.int64) - 53, -1074))
    return np.abs(np.asarray(got, np.float64).astype(LD) - ref) / ulp


def f32_ord(x):
    """f32 values as integers in ulp order (adjacent floats differ by 1, +-inf one past +-FLT_MAX)."""
    b = np.ascontiguousarray(x, np.float32).view(np.int32).astype(np.int64)
    return np.where(b < 0, -(b & 0x7fffffff), b)


def ulp_dist32(a, b):
    return np.abs(f32_ord(a) - f32_ord(b))


def f64_bits(x):
    return np.ascontiguousarray(x, np.float64).view(np.int64)


# ---------------------------------------------------------------------------------------------------------------------
# correctly rounded f32 references: long double, and mpmath where long double cannot decide (near an f32 midpoint)

def _ld_ref(kind, x, y):
    x = np.asarray(x, np.float32).astype(LD)
    if kind == "exp":
        return np.exp(x)
    if kind == "log":
        return np.log(x)
    if kind == "log10":
        return np.log10(x)
    if kind == "pow10":
        return np.power(LD(10), x)
    return np.exp(np.asarray(y, np.float32).astype(LD) * np.log(x))      # pow, x > 0


def _mp_ref(kind, x, y):
    import mpmath
    with mpmath.workprec(200):
        X = mpmath.mpf(float(x))
        if kind == "exp":
            return mpmath.exp(X)
        if kind == "log":
            return mpmath.log(X)
        if kind == "log10":
            return mpmath.log10(X)
        if kind == "pow10":
            return mpmath.power(10, X)
        return mpmath.power(X, mpmath.mpf(float(y)))


def _mp_round_f32(v):
    import mpmath
    if mpmath.isinf(v) or abs(v) >= mpmath.mpf(2) ** 128:
        return np.float32(np.inf if v > 0 else -np.inf)
    if abs(v) < mpmath.mpf(2) ** -126:                                  # f32 subnormal: a multiple of 2**-149
        with mpmath.workprec(300):
            q = mpmath.nint(v * mpmath.mpf(2) ** 149)
        return np.float32(float(q) * 2.0 ** -149)
    with mpmath.workprec(24):
        return np.float32(float(+v))


def cr_f32(kind, x, y=None):
    """The correctly rounded f32 value of exp / log / log10 / 10** / pow at f32 arguments."""
    r = _ld_ref(kind, x, y)
    f = r.astype(np.float32)
    lo = np.nextafter(f, np.float32(-np.inf)).astype(LD)
    hi = np.nextafter(f, np.float32(np.inf)).astype(LD)
    fl = f.astype(LD)
    with np.errstate(invalid="ignore", over="ignore"):
        dist = np.minimum(np.abs(r - (fl + lo) / 2), np.abs(r - (fl + hi) / 2)) / np.abs(r)
    amb = np.nonzero(np.isfinite(f) & (dist < 2.0 ** -40))[0]
    xs = np.broadcast_to(np.asarray(x, np.float32), r.shape)
    ys = np.broadcast_to(np.asarray(y if y is not None else 0, np.float32), r.shape)
    for i in amb:
        f[i] = _mp_round_f32(_mp_ref(kind, xs[i], ys[i]))
    return f


# ---------------------------------------------------------------------------------------------------------------------
# point sets

def _around(v, k):
    """Every f64 within k ulps of each value of v."""
    b = f64_bits(np.asarray(v, np.float64))
    return (b[:, None] + np.arange(-k, k + 1)[None, :]).ravel().view(np.float64)


def _exp_node_boundaries():
    """+-3 ulps around every x where the table index k = round(x * 128 / ln 2) of the exp reduction changes, |x| < 704."""
    c0 = 184.6649652337873
    j = np.arange(-130000, 130000)
    x = _around((j + 0.5) / c0, 3)
    return x[np.abs(x) < 704]


def _log_node_boundaries():
    """+-2 ulps around every x where the log node index (hi word - 0x3fe60000) >> 13 changes, over all normal binades."""
    m = np.arange(-(0x3fe60000 - 0x00100000) // 0x2000, (0x7fe00000 - 0x3fe60000) // 0x2000 + 1)
    hi = 0x3fe60000 + m * 0x2000
    hi = hi[(hi >= 0x00100000) & (hi < 0x7ff00000)]
    x = _around((hi.astype(np.int64) << 32).view(np.float64), 2)
    return x[(x >= DBL_MIN) & (x <= DBL_MAX)]


def _log_points(rng):
    """Every binade from DBL_MIN to DBL_MAX (256 random mantissas each), and x = 1 +- k ulp."""
    e = np.repeat(np.arange(-1022, 1024), 256)
    x = np.ldexp(rng.uniform(1.0, 2.0, e.size), e)
    one = np.concatenate([_around([1.0], 2000), 1.0 + rng.uniform(-0.1, 0.1, 200_000)])
    return np.concatenate([x, one[one > 0]])


def _pow_points(rng, n):
    """x over the whole positive normal range, y such that |y log x| < 704."""
    lx = rng.uniform(-700, 700, n)
    x = np.exp(lx)
    x[: n // 4] = np.exp(rng.uniform(-40, 40, n // 4))
    lx = np.log(x)
    e = rng.uniform(-703.5, 703.5, n) * rng.choice([1.0, 0.1, 0.01], n)
    y = e / np.where(np.abs(lx) < 1e-300, 1.0, lx)
    keep = (np.abs(y * lx) < 703.9) & (x > DBL_MIN) & np.isfinite(y)
    return x[keep], y[keep]


# contract of the f64 routines (DESIGN.md section 4): measured maxima on the host twin over the point sets below, with a
# small margin - exp 0.998 ulp, log 1.42 ulp (|log x| > 0.1; 1.10 below |log x| = 700) / 1.35e-17 absolute (|log x| <= 0.1), pow 2.57
EXP_ULP = 1.0
LOG_ULP = 1.5
LOG_ABS = 1.5e-17
POW_C = 3.0


def pow_bound_ulp(x, y):
    """dpow's bound in ulps: POW_C * (1 + |y ln x|), plus |y| * LOG_ABS relative where |ln x| <= 0.1 (the absolute error
    of log near 1 is multiplied by y)."""
    lx = np.log(np.asarray(x, np.float64).astype(LD))
    yl = np.asarray(y, np.float64).astype(LD)
    near1 = np.abs(lx) <= 0.1
    return POW_C * (1 + np.abs(yl * lx)) + np.where(near1, np.abs(yl) * LOG_ABS / 2.0 ** -53, 0)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the host twin against long double / mpmath

def test_twin_exp_accuracy(twin):
    rng = np.random.default_rng(1)
    x = np.concatenate([rng.uniform(-703.999, 703.999, 1_000_000), rng.uniform(-1, 1, 200_000), _exp_node_boundaries(),
                        _around([704.0, -704.0], 1000)])
    fast = np.abs(x) < 704
    err = ulp_err64(twin.exp(x), np.exp(x.astype(LD)))
    assert err[fast].max() < EXP_ULP, err[fast].max()
    # |x| >= 704 takes the library exp: within one ulp, results subnormal below -708.4 (the subnormal ulp is absolute)
    xs = np.concatenate([x[~fast], rng.uniform(-745.1, -704, 100_000), rng.uniform(704, 709.78, 100_000)])
    assert ulp_err64(twin.exp(xs), np.exp(xs.astype(LD))).max() <= 1.0


def test_twin_log_accuracy(twin):
    rng = np.random.default_rng(2)
    x = np.concatenate([_log_points(rng), _log_node_boundaries()[::4], _around([DBL_MIN, DBL_MAX], 100)])
    x = x[(x >= DBL_MIN) & (x <= DBL_MAX)]
    ref = np.log(x.astype(LD))
    got = twin.log(x)
    big = np.abs(ref) > 0.1
    assert ulp_err64(got[big], ref[big]).max() < LOG_ULP
    assert np.abs(got[~big].astype(LD) - ref[~big]).max() < LOG_ABS
    # 1 +- k ulp: the error is absolute (log x ~ k * 2**-53), up to ~1e4 ulps of the result
    one = _around([1.0], 2000)
    assert np.abs(twin.log(one).astype(LD) - np.log(one.astype(LD))).max() < LOG_ABS


def test_twin_pow_accuracy(twin):
    rng = np.random.default_rng(3)
    x, y = _pow_points(rng, 1_000_000)
    ref = np.exp(y.astype(LD) * np.log(x.astype(LD)))
    err = ulp_err64(twin.pow(x, y), ref)
    assert (err <= pow_bound_ulp(x, y)).all(), (err / pow_bound_ulp(x, y)).max()


def test_twin_pow_f32_correctly_rounded_near_midpoints(twin):
    """The f32 rounding of the twin's x**y (= pow_f) against the correctly rounded value, with mpmath deciding the points
    long double cannot; x in e**+-40, y in +-2."""
    rng = np.random.default_rng(4)
    x = np.exp(rng.uniform(-40, 40, 300_000)).astype(np.float32)
    y = rng.uniform(-2, 2, 300_000).astype(np.float32)
    got = twin.pow(x.astype(np.float64), y.astype(np.float64)).astype(np.float32)
    cr = cr_f32("pow", x, y)
    assert ulp_dist32(got, cr).max() <= 1
    assert np.count_nonzero(got != cr) <= 3


def test_oracle_decade_index_d_around_every_decade():
    """kor_decade_index_d (M:1824-1833) on the f64 ulps around 10**n, the libgcc powi 10.**n and m * 10**n: the index is
    the decade's mantissa bin, and the array form equals the scalar calls."""
    from oracle import oracle
    x = _decade_points_d(8)
    n2, ntb = 4, 28
    got = oracle.decade_index_d_array(x, n2, ntb)
    assert np.array_equal(got, [oracle.decade_index_d(float(v), n2, ntb) for v in x])
    # an exact restatement where the bin is not on an edge: floor(x / 10**n) + 9 (n - n2), clamped
    xl = x.astype(LD)
    n = np.floor(np.log10(xl)).astype(np.int64)
    q = xl / np.power(LD(10), n)
    clear = (np.abs(q - np.round(q)) > 1e-12) & (q > 1 + 1e-12)
    want = np.clip(np.floor(q).astype(np.int64) + 9 * (n - n2), 1, ntb)
    assert np.array_equal(got[clear], want[clear])


def test_oracle_array_forms_equal_scalar_calls():
    from oracle import oracle
    rng = np.random.default_rng(5)
    n = 2000
    p = rng.uniform(3e4, 1.05e5, n).astype(np.float32)
    t = rng.uniform(170, 330, n).astype(np.float32)
    assert np.array_equal(oracle.rslf_array(p, t), np.float32([oracle.rslf(a, b) for a, b in zip(p, t)]))
    assert np.array_equal(oracle.rsif_array(p, t), np.float32([oracle.rsif(a, b) for a, b in zip(p, t)]))
    x = np.exp(rng.uniform(-30, 20, n)).astype(np.float32)
    assert np.array_equal(oracle.decade_index_array(x, -6, 37), [oracle.decade_index(v, -6, 37) for v in x])
    args = _aero_inputs(rng, n)
    for sp in "rsg":
        got = oracle.eff_aero_array(*args["eff_" + sp], sp)
        assert np.array_equal(got, np.float32([oracle.eff_aero(*a, sp) for a in zip(*args["eff_" + sp])]), sp)
    for name, fn, fa in (("demott", oracle.ice_demott, oracle.ice_demott_array), ("koop", oracle.ice_koop, oracle.ice_koop_array),
                         ("activ", oracle.activ_ncloud, oracle.activ_ncloud_array)):
        got = fa(*args[name])
        assert np.array_equal(got, np.float32([fn(*a) for a in zip(*args[name])]), name)


def test_probe_compiles_for_sm100a(probe_lib):
    """The probe (tests/device_probe.cu) compiles with the library's flags and includes the product headers unchanged."""
    out = subprocess.run(["/usr/local/cuda/bin/cuobjdump", "-lelf", probe_lib], capture_output=True, text=True)
    if out.returncode == 0:
        assert "sm_100a" in out.stdout
    assert os.path.getsize(probe_lib) > 0


# ---------------------------------------------------------------------------------------------------------------------
# point sets of the scalar helpers

def _powi10(n):
    """10.**n as libgcc __powisf2 builds it (kidmp_hostinit.h powi10), in f32."""
    m = abs(n)
    x = np.float32(10.0)
    y = x if m % 2 else np.float32(1.0)
    m >>= 1
    while m:
        x = np.float32(x * x)
        if m % 2:
            y = np.float32(y * x)
        m >>= 1
    return np.float32(np.float32(1.0) / y) if n < 0 else y


DECADES = range(-30, 31)


def _decade_points_f(k, rng=None):
    """f32 values within k ulps of 10**n, of the powi 10.**n and of m * 10**n (m = 2..9), n = -30..30; plus random."""
    c = []
    for n in DECADES:
        c += [np.float32(10.0 ** n), _powi10(n)] + [np.float32(m * 10.0 ** n) for m in range(2, 10)]
    b = np.float32(c).view(np.int32).astype(np.int64)
    x = (b[:, None] + np.arange(-k, k + 1)[None, :]).ravel().astype(np.int32).view(np.float32)
    if rng is not None:
        x = np.concatenate([x, np.float32(10.0) ** rng.uniform(-30, 30.9, 1_000_000).astype(np.float32)])
    return x[np.isfinite(x) & (x > 0)]


def _decade_points_d(k, rng=None):
    c = []
    for n in DECADES:
        c += [10.0 ** n, float(_powi10(n))] + [m * 10.0 ** n for m in range(2, 10)]
    x = _around(c, k)
    if rng is not None:
        x = np.concatenate([x, 10.0 ** rng.uniform(-30, 30.9, 1_000_000)])
    return x[x > 0]


def _aero_inputs(rng, n):
    f = lambda lo, hi: rng.uniform(lo, hi, n).astype(np.float32)
    lg = lambda lo, hi: np.exp(rng.uniform(np.log(lo), np.log(hi), n)).astype(np.float32)
    # the two aerosol diameters of the scheme, and larger ones: only those reach St > St2 and the 1.0 clamp of Eff
    Da = np.where(rng.random(n) < 0.5, np.where(rng.random(n) < 0.5, np.float32(0.04e-6), np.float32(0.8e-6)),
                  lg(1e-6, 2e-5)).astype(np.float32)
    eff = lambda: (lg(50e-6, 5e-3), Da, f(1.2e-5, 1.9e-5), f(0.3, 1.4), f(200, 310))
    return {"eff_r": eff(), "eff_s": eff(), "eff_g": eff(),
            "demott": (f(-60, -0.5), f(0.3, 1.4), lg(1e2, 1e8)),
            "koop": (f(180, 238), lg(1e-7, 1e-3), lg(1e-7, 1e-3), lg(1e6, 1e11), f(1, 120)),
            "activ": (f(230, 310), np.concatenate([lg(1e-3, 200, )[: n // 2], f(-5, 5)[: n - n // 2]]), lg(1e5, 2e10))}


# ---------------------------------------------------------------------------------------------------------------------
# the device probe

PROBE_FN = {n: i for i, n in enumerate((
    "dexp", "dlog", "dpow", "pow_f", "exp_f", "log10_f", "pow10_f", "log_f", "rslf", "rsif",
    "decade_idx_f", "decade_idx_d", "field_moment", "field_loga", "field_b", "graupel_n0_exp", "rain_lam", "ice_lam",
    "eff_aero_r", "eff_aero_s", "eff_aero_g", "ice_demott", "ice_koop", "activ_ncloud"))}

# the (n2, ntb) pairs of the decade indices the cell kernels take (kidmp_cells.cuh, S6: idx_c idx_i idx_i1 idx_r idx_s
# idx_g, then idx_r1 and idx_g1 of the f64 intercepts)
DECADE_F_PAIRS = (("nic2", 37), ("nii2", 64), ("nii3", 55), ("nir2", 37), ("nis2", 28), ("nig2", 28))
DECADE_D_PAIRS = (("nir3", 37), ("nig3", 28))


def probe_flags():
    """The flags libkidmp.so is built with (kid_b200.build.BASE_FLAGS, without the build-id define)."""
    from kid_b200 import build as kb
    return [*kb.BASE_FLAGS, "-I", CSRC]


@pytest.fixture(scope="session")
def probe_lib(tmp_path_factory):
    from kid_b200 import build as kb
    out = str(tmp_path_factory.mktemp("probe") / "libdevice_probe.so")
    subprocess.check_call([kb.nvcc_path(), *probe_flags(), "-o", out, os.path.join(HERE, "device_probe.cu")])
    return out


class Probe:
    """ctypes front of tests/device_probe.cu: run(name, *arrays) evaluates a helper on the device, on torch's current
    stream, with the KConst of a handle of (set_Nc, iiwarm)."""

    def __init__(self, path, set_Nc=100.0, iiwarm=0):
        L = C.CDLL(path)
        L.probe_kconst_size.restype = C.c_long
        L.probe_init.restype = C.c_int
        L.probe_init.argtypes = [C.c_float, C.c_int, C.c_void_p]
        L.probe_kconst.restype = C.c_double
        L.probe_kconst.argtypes = [C.c_void_p, C.c_char_p]
        L.probe_run.restype = C.c_int
        L.probe_run.argtypes = [C.c_int, C.c_long] + [C.c_void_p] * 5 + [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        self.L = L
        self.kc = C.create_string_buffer(L.probe_kconst_size())
        rc = L.probe_init(set_Nc, iiwarm, self.kc)
        assert rc == 0, "probe_init: cudaError %d" % rc

    def const(self, name):
        v = self.L.probe_kconst(self.kc, name.encode())
        assert np.isfinite(v), name
        return v

    def run(self, name, *args, i0=0, i1=0):
        import torch
        arrs = np.broadcast_arrays(*[np.asarray(a, np.float64) for a in args])
        ts = [torch.from_numpy(np.ascontiguousarray(a, np.float64).ravel()).cuda() for a in arrs]
        n = ts[0].numel()
        out = torch.empty(n, dtype=torch.float64, device="cuda")
        ptrs = [t.data_ptr() for t in ts] + [None] * (5 - len(ts))
        rc = self.L.probe_run(PROBE_FN[name], n, *ptrs, i0, i1, self.kc, out.data_ptr(),
                              torch.cuda.current_stream().cuda_stream)
        assert rc == 0, "probe_run(%s): cudaError %d" % (name, rc)
        return out.cpu().numpy().reshape(arrs[0].shape)

    def run32(self, name, *args, **kw):
        r = self.run(name, *args, **kw)
        assert np.array_equal(r.astype(np.float32).astype(np.float64), r, equal_nan=True), name
        return r.astype(np.float32)


@pytest.fixture(scope="session")
def probe(probe_lib):
    return Probe(probe_lib)


# ---------------------------------------------------------------------------------------------------------------------
# A. the device copy is the tested algorithm

@pytest.mark.gpu
def test_device_exp_log_pow_bit_identical_to_twin(probe, twin):
    """dexp / dlog / dpow (kidmp_math.cuh: own c_fm coefficients, own fm_*_core) against the host twin of
    kidmp_fastmath.h, bit for bit wherever both take the table path: >= 1e6 points each, every exp node boundary
    (|x| < 704), every log node boundary of every binade, both sides of the fm_exp_fast / fm_log_fast switches."""
    rng = np.random.default_rng(11)
    x = np.concatenate([rng.uniform(-704, 704, 1_000_000), rng.uniform(-1e-3, 1e-3, 10_000), _exp_node_boundaries(),
                        _around([704.0, -704.0], 200)])
    fast = np.abs(x) < 704
    d = probe.run("dexp", x)
    assert np.array_equal(f64_bits(d[fast]), f64_bits(twin.exp(x[fast]))), np.count_nonzero(
        f64_bits(d[fast]) != f64_bits(twin.exp(x[fast])))
    assert fast.sum() >= 1_000_000

    x = np.concatenate([np.ldexp(rng.uniform(1, 2, 1_000_000), rng.integers(-1022, 1024, 1_000_000)),
                        _log_node_boundaries(), _around([DBL_MIN, DBL_MAX], 200), _around([1.0], 500)])
    fast = (x >= DBL_MIN) & (x <= DBL_MAX)
    d = probe.run("dlog", x)
    bad = np.count_nonzero(f64_bits(d[fast]) != f64_bits(twin.log(x[fast])))
    assert bad == 0, bad
    assert fast.sum() >= 1_000_000

    xp, yp = _pow_points(rng, 1_200_000)
    xs = np.exp(rng.uniform(-700, 700, 20_000))                      # both sides of |y log x| = 704
    ys = np.concatenate([_around(704.0 / np.log(xs[:10_000]), 3), _around(-704.0 / np.log(xs[10_000:]), 3)])
    xp = np.concatenate([xp, np.repeat(xs, 7)])
    yp = np.concatenate([yp, ys])
    with np.errstate(over="ignore", invalid="ignore"):
        fast = (xp >= DBL_MIN) & (xp <= DBL_MAX) & (np.abs(yp * twin.log(xp)) < 704)
    d = probe.run("dpow", xp, yp)
    bad = np.count_nonzero(f64_bits(d[fast]) != f64_bits(twin.pow(xp[fast], yp[fast])))
    assert bad == 0, bad
    assert fast.sum() >= 1_000_000 and (~fast).sum() > 1000


# ---------------------------------------------------------------------------------------------------------------------
# B. accuracy outside the table path (long double references: 64-bit significand, 11 bits beyond f64)

@pytest.mark.gpu
def test_device_math_outside_fast_path(probe):
    rng = np.random.default_rng(12)
    # log of subnormal and DBL_MIN-adjacent x: the library log, within one ulp
    sub = rng.integers(1, 1 << 52, 100_000).view(np.float64)
    x = np.concatenate([sub, np.arange(1, 1001).view(np.float64), _around([DBL_MIN], 1000)])
    err = ulp_err64(probe.run("dlog", x), np.log(x.astype(LD)))
    assert err.max() <= 1.0, err.max()
    # exp beyond |x| = 704: normal results, overflow, subnormal results (x in [-745, -708]) and underflow to zero
    x = np.concatenate([rng.uniform(704, 709.78, 50_000), rng.uniform(-708.4, -704, 50_000),
                        rng.uniform(-745.13, -708.4, 100_000), _around([704.0, -704.0, -708.3964185322641], 100)])
    x = x[np.abs(x) >= 704]
    ref = np.exp(x.astype(LD))
    err = ulp_err64(probe.run("dexp", x), ref)
    sub = ref < LD(DBL_MIN)
    assert err[~sub].max() <= 1.0, err[~sub].max()
    assert err[sub].max() <= 2.0, err[sub].max()                     # one ulp + the absolute subnormal ulp
    assert np.all(probe.run("dexp", [709.79, 710.0, 800.0, 1e300]) == np.inf)
    assert np.all(probe.run("dexp", [-745.2, -746.0, -800.0, -1e300]) == 0.0)
    # x**y with |y log x| >= 704: results that overflow, underflow or are subnormal
    xb = np.exp(rng.uniform(-700, 700, 100_000))
    xb = xb[np.abs(np.log(xb)) > 1e-3]
    yb = rng.uniform(704, 760, xb.size) * rng.choice([-1.0, 1.0], xb.size) / np.log(xb)
    ref = np.exp(yb.astype(LD) * np.log(xb.astype(LD)))
    d = probe.run("dpow", xb, yb)
    over = ref > LD(DBL_MAX) * (1 + LD(1e-9))
    fin = ref < LD(DBL_MAX) * (1 - LD(1e-9))
    assert np.all(d[over] == np.inf)
    err = ulp_err64(d[fin], ref[fin])
    assert np.all(err <= pow_bound_ulp(xb[fin], yb[fin]) + 1)
    assert over.sum() > 1000 and (fin & (ref < LD(DBL_MIN))).sum() > 1000


# ---------------------------------------------------------------------------------------------------------------------
# C. special values, pinned

NAN = float("nan")
INF = float("inf")
SUB = 5e-324


@pytest.mark.gpu
def test_device_special_values_pinned(probe):
    """What dexp / dlog / dpow do at +-0, x < 0, +-inf, NaN and subnormals.

    dpow departs from C pow / glibc powf (which the reference's REAL ** REAL is under gfortran) in four cases: 0**0,
    1**+-inf, inf**0 and NaN**0 give NaN instead of 1, and a negative base gives NaN even for an integral exponent.
    None of them can be reached from the step; the call sites of pow_f / pow_d (= dpow):
      kidmp_cells.cuh   lc / lamc ...**obmr (347, 455, 932), xDc (454): base a ratio of nc, rc > R1 - positive;
                        exponent obmr = 1/3.  Dc_b (460) ...**(1/6): a negative or zero base is NaN / 0 in C too
                        (non-integral exponent).  diffu (408, 1102, 1150): (temp/273.15)**1.94, temp > 0.
                        smo1 / smo0 (431, 694, 807): smo2 / smob = rs*oams with rs > R1 - positive; the Field exponent
                        b_ is finite, and zero only with a positive base.  vtg, il9, il10, il11 (567, 574, 596, 749,
                        819, 1385): ilamg**bv_g / cge(9) / cge(11), ilamg = 1/lamg > 0, PARAMETER exponents 0.89,
                        3.89, 2.945.  mm, t1..t4_vts (1227-1233): Mrat, ils1, ils2 > 0 (snow moments of rs > R1),
                        exponents mu_s, cse(4), cse(10), cse(1), cse(7) - nonzero PARAMETERs (cse(1) = 3 is integral,
                        but the base is positive).
      kidmp_column.cuh  field_moment (56): smo2 > 0, as above.  rain_lam / ice_lam (112, 115): nr / rr, ni / ri of a
                        present species - positive; exponents obmr = obmi = 1/3.  lc (409) as at cells 347.
      kidmp_aero.cuh    eff_aero (19, 20, 28, 30): D**0.55 / D**0.89 with a mean diameter > 0, Sc**0.3333 with Sc > 0,
                        ((St - St2) / (St - St2 + 0.666667))**1.5 only where St > St2.  ice_demott (38):
                        (-tempc)**3.33 and nifa_cc**(0.0033 - 0.0264 tempc) are called below T_0 only (the Cooper /
                        DeMott block of S6 runs for cold cells): -tempc > 0 and the exponent > 0.0033, so 0**0 cannot
                        occur and 0**y (nifa = 0) is 0 as in C.
      (kidmp_kid.cuh:46 exner**(1/kappa) and kidmp_wrf.cuh:95, 99 are of the same kinds: positive bases, nonzero
      PARAMETER exponents.)
    No exponent is infinite or NaN for finite inputs, so 1**+-inf, inf**0 and NaN**0 need a state that is already
    infinite or NaN."""
    cases = [
        ("dexp", (0.0,), 1.0), ("dexp", (-0.0,), 1.0), ("dexp", (INF,), INF), ("dexp", (-INF,), 0.0),
        ("dexp", (NAN,), NAN), ("dexp", (SUB,), 1.0), ("dexp", (-SUB,), 1.0),
        ("dlog", (0.0,), -INF), ("dlog", (-0.0,), -INF), ("dlog", (-1.0,), NAN), ("dlog", (-SUB,), NAN),
        ("dlog", (INF,), INF), ("dlog", (-INF,), NAN), ("dlog", (NAN,), NAN), ("dlog", (1.0,), 0.0),
        ("dlog", (SUB,), float(np.log(LD(SUB)))),
        ("dpow", (0.0, 2.0), 0.0), ("dpow", (0.0, -2.0), INF), ("dpow", (-0.0, 3.0), 0.0), ("dpow", (-0.0, -3.0), INF),
        ("dpow", (2.0, 0.0), 1.0), ("dpow", (1.0, 5.0), 1.0), ("dpow", (INF, 2.0), INF), ("dpow", (INF, -2.0), 0.0),
        ("dpow", (NAN, 2.0), NAN), ("dpow", (2.0, NAN), NAN),
        ("dpow", (-2.0, 0.5), NAN),
        # the four departures from C pow (which gives 1, 1, 1, 1 and 4): pinned as NaN
        ("dpow", (0.0, 0.0), NAN), ("dpow", (1.0, INF), NAN), ("dpow", (1.0, -INF), NAN), ("dpow", (INF, 0.0), NAN),
        ("dpow", (NAN, 0.0), NAN), ("dpow", (-2.0, 2.0), NAN),
        ("pow_f", (0.0, 0.0), NAN), ("pow_f", (0.0, 1.5), 0.0), ("pow_f", (-2.0, 2.0), NAN), ("pow_f", (4.0, 0.5), 2.0),
        ("exp_f", (-INF,), 0.0), ("exp_f", (INF,), INF), ("exp_f", (100.0,), INF), ("exp_f", (-110.0,), 0.0),
        ("log10_f", (0.0,), -INF), ("log10_f", (-1.0,), NAN), ("log_f", (INF,), INF), ("pow10_f", (39.0,), INF),
    ]
    for name, args, want in cases:
        got = float(probe.run(name, *[np.array([a]) for a in args])[0])
        if np.isnan(want):
            assert np.isnan(got), (name, args, got)
        else:
            assert got == want and np.signbit(got) == np.signbit(want), (name, args, got, want)


# ---------------------------------------------------------------------------------------------------------------------
# D. the f32 wrappers are correctly rounded

def _f32(a):
    return np.asarray(a, np.float32)


def _check_cr(got, cr, what, per_million=5):
    d = ulp_dist32(got, cr)
    miss = int(np.count_nonzero(d))
    assert d.max() <= 1, (what, int(d.max()))
    assert miss <= 2 + per_million * got.size / 1e6, (what, miss, got.size)
    return miss


@pytest.fixture(scope="session")
def f32_points(probe):
    """Inputs of the f32 wrappers and their correctly rounded results (computed once per session)."""
    rng = np.random.default_rng(13)
    n = 1_000_000
    pts = {}
    # x**y: x in e**+-40, y in +-2, every run-time exponent of the kernels, results at the overflow edge and subnormal
    exps = [probe.const("obmr"), probe.const("obmi"), 0.55, 0.89, probe.const("Sc3"), 0.3333, 1.5, 3.33, 1.94, 1 / 6]
    tc0 = _f32(rng.uniform(-60, -0.1, 30_000))
    bfield = probe.run32("field_b", tc0, _f32(rng.choice([probe.const("cse0"), probe.const("cse12"), probe.const("cse15")],
                                                         30_000)))
    x = [np.exp(rng.uniform(-40, 40, n))]
    y = [rng.uniform(-2, 2, n)]
    for e in exps:
        x.append(np.exp(rng.uniform(-40, 40, 100_000)))
        y.append(np.full(100_000, e))
    x.append(np.exp(rng.uniform(-20, 3, bfield.size)))
    y.append(bfield)
    ye = rng.uniform(0.3, 3, 200_000) * rng.choice([-1, 1], 200_000)
    x.append(np.exp((88.72 + rng.uniform(-0.05, 0.05, 100_000)) / ye[:100_000]))         # overflow edge
    x.append(np.exp(rng.uniform(-104, -87.3, 100_000) / ye[100_000:]))                  # subnormal results
    y.append(ye)
    px, py = _f32(np.concatenate(x)), _f32(np.concatenate(y))
    ok = (px > 0) & np.isfinite(px)
    pts["pow_f"] = (px[ok], py[ok])
    edges = np.tile([88.7228391, -87.3365448, -103.972], 1000) + rng.uniform(-1e-4, 1e-4, 3000)
    pts["exp_f"] = (_f32(np.concatenate([rng.uniform(-104, 88.8, n), edges])),)
    allf = rng.integers(1, 0x7f800000, n).astype(np.int32).view(np.float32)              # every positive f32 binade
    pts["log10_f"] = (allf,)
    pts["log_f"] = (allf,)
    pts["pow10_f"] = (_f32(np.concatenate([rng.uniform(-45.2, 38.6, n), rng.uniform(-0.5, 0.5, 100_000)])),)
    kinds = {"pow_f": "pow", "exp_f": "exp", "log10_f": "log10", "log_f": "log", "pow10_f": "pow10"}
    return {k: (v, cr_f32(kinds[k], *v)) for k, v in pts.items()}


@pytest.mark.gpu
def test_f32_wrappers_correctly_rounded(probe, twin, f32_points):
    """pow_f, exp_f, log10_f, pow10_f, log_f (f64 evaluation rounded once, DESIGN.md section 4 rule 2): never more than
    one ulp from the correctly rounded value and equal to it but for a few double-rounding misses per million, in the
    normal range, at the f32 overflow edge and for subnormal results (the build keeps -ftz=false).  The differences from
    glibc (what the oracle calls) are printed: within one ulp for powf / expf / logf, two for log10f, which glibc does
    not round correctly (measured on a B200 build: 1.4 % of a million log10f results, all of them where glibc misses)."""
    libm = {"pow_f": twin.powf, "exp_f": twin.expf, "log10_f": twin.log10f, "log_f": twin.logf,
            "pow10_f": lambda y: twin.powf(np.float32(10), y)}
    for name, (args, cr) in f32_points.items():
        got = probe.run32(name, *args)
        miss = _check_cr(got, cr, name)
        lm = libm[name](*args)
        dl = ulp_dist32(got, lm)
        print("%-8s %8d points: %d not correctly rounded, %d differ from glibc (max %d ulp); glibc not correctly rounded: %d"
              % (name, got.size, miss, np.count_nonzero(dl), dl.max(), np.count_nonzero(lm != cr)))
        assert dl.max() <= 2, name                                  # glibc's log10f is up to 2 ulps off (the others 1)
        if name == "pow_f":
            res = cr[np.isfinite(cr)]
            assert np.count_nonzero(np.isinf(cr)) > 1000 and np.count_nonzero(res < np.finfo(np.float32).tiny) > 1000
    n = np.arange(0, 11)
    assert np.array_equal(probe.run32("pow10_f", n), _f32(10.0 ** n))    # 10**n exact in f32 for n <= 10
    assert probe.run32("pow_f", [4.0], [0.5])[0] == 2.0


# ---------------------------------------------------------------------------------------------------------------------
# E. bit-identical to the oracle where no transcendental is involved

@pytest.mark.gpu
def test_saturation_bit_identical_to_oracle(probe):
    """rslf / rsif (Horner polynomials in f32, no FMA) at every f32 temperature of [173.15, 333.15] K and four pressures,
    and at random (P, T) that reach both clamps (T - 273.16 < -80 and ESL > 0.15 P)."""
    from oracle import oracle
    t = np.arange(_f32(173.15).view(np.int32), _f32(333.15).view(np.int32) + 1, dtype=np.int32).view(np.float32)
    for P in (50000.0, 70000.0, 85000.0, 105000.0):
        p = np.full(t.size, P, np.float32)
        for fn, ofn in (("rslf", oracle.rslf_array), ("rsif", oracle.rsif_array)):
            got = probe.run32(fn, p, t)
            want = ofn(p, t)
            assert np.array_equal(got.view(np.int32), want.view(np.int32)), (fn, P, np.count_nonzero(got != want))
    rng = np.random.default_rng(14)
    p = _f32(np.exp(rng.uniform(np.log(100), np.log(1.1e5), 2_000_000)))
    tt = _f32(rng.uniform(150, 350, 2_000_000))
    for fn, ofn in (("rslf", oracle.rslf_array), ("rsif", oracle.rsif_array)):
        got = probe.run32(fn, p, tt)
        want = ofn(p, tt)
        assert np.array_equal(got.view(np.int32), want.view(np.int32)), fn
        clamped = np.isclose(want.astype(np.float64), 0.622 * 0.15 / 0.85, rtol=1e-5)
        assert clamped.sum() > 1000 and (tt < 193.16).sum() > 1000


@pytest.mark.gpu
def test_decade_index_bit_identical_to_oracle(probe):
    """decade_idx_f / decade_idx_d (kidmp_column.cuh) against the oracle's search (M:1762-1774, M:1824-1833) for every
    (n2, ntb) pair the cell kernels pass: every ulp within 40 of 10**n, of the powi 10.**n and of m * 10**n, n = -30..30,
    plus a million log-uniform values."""
    from oracle import oracle
    rng = np.random.default_rng(15)
    xf = _decade_points_f(40, rng)
    for name, ntb in DECADE_F_PAIRS:
        n2 = int(probe.const(name))
        got = probe.run("decade_idx_f", xf, i0=n2, i1=ntb).astype(np.int32)
        want = oracle.decade_index_array(xf, n2, ntb)
        assert np.array_equal(got, want), (name, xf[got != want][:5], got[got != want][:5], want[got != want][:5])
    xd = _decade_points_d(40, rng)
    for name, ntb in DECADE_D_PAIRS:
        n2 = int(probe.const(name))
        got = probe.run("decade_idx_d", xd, i0=n2, i1=ntb).astype(np.int32)
        want = oracle.decade_index_d_array(xd, n2, ntb)
        assert np.array_equal(got, want), (name, xd[got != want][:5], got[got != want][:5], want[got != want][:5])


# ---------------------------------------------------------------------------------------------------------------------
# F. helpers that mix f32 arithmetic with transcendentals

C_SA = _f32([0, 5.065339, -0.062659, -3.032362, 0.029469, -0.000285, 0.31255, 0.000204, 0.003199, 0.0, -0.015952])
C_SB = _f32([0, 0.476221, -0.015896, 0.165977, 0.007468, -0.000141, 0.060366, 0.000079, 0.000594, 0.0, -0.003577])


def _field_ab_f32(tc0, c):
    """loga_ / b_ of field_ab (M:1590-1599), operation by operation in f32 (products left to right, no FMA)."""
    def poly(s):
        return (s[1] + s[2] * tc0 + s[3] * c + s[4] * tc0 * c + s[5] * tc0 * tc0 + s[6] * c * c + s[7] * tc0 * tc0 * c
                + s[8] * tc0 * c * c + s[9] * tc0 * tc0 * tc0 + s[10] * c * c * c)
    return poly(C_SA), poly(C_SB)


@pytest.mark.gpu
def test_field_moment_and_graupel_intercept_against_f32_restatement(probe):
    """field_moment and graupel_n0_exp against a numpy f32 restatement whose transcendentals are correctly rounded
    (long double, mpmath at f32 midpoints): bit-identical but for counted double-rounding misses of pow_f / pow10_f /
    log10_f; field_ab's two polynomials bit for bit."""
    rng = np.random.default_rng(16)
    n = 300_000
    tc0 = _f32(rng.uniform(-60, -0.1, n))
    c = _f32(rng.choice([probe.const("cse0"), probe.const("cse12"), probe.const("cse15")], n))
    smo2 = _f32(np.exp(rng.uniform(np.log(1e-9), np.log(0.2), n)))
    la, b = _field_ab_f32(tc0, c)
    assert np.array_equal(probe.run32("field_loga", tc0, c).view(np.int32), la.view(np.int32))
    assert np.array_equal(probe.run32("field_b", tc0, c).view(np.int32), b.view(np.int32))
    want = cr_f32("pow10", la) * cr_f32("pow", smo2, b)
    got = probe.run32("field_moment", tc0, c, smo2)
    miss = np.count_nonzero(got != want)
    assert ulp_dist32(got, want).max() <= 2 and miss <= 2 + 10 * n / 1e6, miss

    # graupel intercept: xslw1 = 0.01 or 4.01 + log10(mvd_r), rg across 5e-5 (the MAX of M:1641) and both gonv clamps
    xslw1 = np.where(rng.random(n) < 0.3, np.float32(0.01),
                     np.float32(4.01) + cr_f32("log10", _f32(np.exp(rng.uniform(np.log(100e-6), np.log(5e-3), n)))))
    near = (np.float32(5e-5).view(np.int32) + rng.integers(-10_000, 10_001, 20_000)).astype(np.int32).view(np.float32)
    rg = _f32(np.concatenate([np.exp(rng.uniform(np.log(1e-8), np.log(2e-2), n - 20_000)), near]))
    ygra1 = np.float32(4.31) + cr_f32("log10", np.maximum(np.float32(5e-5), rg))
    zans1 = np.float32(3.1) + (np.float32(100) / (np.float32(300) * xslw1 * ygra1 / (np.float32(10) / xslw1 + np.float32(1)
                                                                                      + np.float32(0.25) * ygra1)
                                                  + np.float32(30) + np.float32(10) * ygra1))
    n0 = cr_f32("pow10", zans1).astype(np.float64)
    want = np.maximum(1e4, np.minimum(n0, 3e6))
    got = probe.run("graupel_n0_exp", xslw1, rg)
    miss = np.count_nonzero(got != want)
    assert ulp_dist32(got, want).max() <= 2 and miss <= 2 + 20 * n / 1e6, miss
    # the gonv_min clamp is met; gonv_max cannot be: for xslw1 >= 0.01 the denominator is > 30, so zans1 < 6.44 and
    # N0 < 2.8e6 whatever rg
    assert (n0 < 1e4).sum() > 100 and ((n0 > 1e4) & (n0 < 3e6)).sum() > 100 and n0.max() < 2.8e6


@pytest.mark.gpu
def test_rain_and_ice_slope_within_pow_f_contract(probe):
    """rain_lam / ice_lam: (am*c*o*n/q)**(1/3) with the f32 base restated operation by operation, against the correctly
    rounded power: within one ulp, equal but for a few misses per million."""
    rng = np.random.default_rng(17)
    n = 500_000
    num = _f32(np.exp(rng.uniform(np.log(1e-2), np.log(1e9), n)))
    q = _f32(np.exp(rng.uniform(np.log(1e-12), np.log(2e-2), n)))
    for fn, k in (("rain_lam", ("am_r", "crg2", "org2", "obmr")), ("ice_lam", ("am_i", "cig1", "oig1", "obmi"))):
        a, b, o, e = (_f32(probe.const(v)) for v in k)
        base = a * b * o * num / q
        ok = np.isfinite(base) & (base > 0)
        got = probe.run(fn, num[ok], q[ok]).astype(np.float32)
        _check_cr(got, cr_f32("pow", base[ok], np.full(ok.sum(), e, np.float32)), fn)


def _eff_aero_f64(D, Da, visc, rhoa, T, sp):
    """St, St2 and the unclamped Eff of eff_aero in f64 (to place each point relative to the branch conditions)."""
    D, Da, visc, rhoa, T = (np.asarray(v, np.float64) for v in (D, Da, visc, rhoa, T))
    if sp == "r":
        vt = -0.1021 + 4.932e3 * D - 0.9551e6 * D ** 2 + 0.07934e9 * D ** 3 - 0.002362e12 * D ** 4
    else:
        vt = (40.0 * D ** 0.55) if sp == "s" else (442.0 * D ** 0.89)
    mp = 0.0256e-6
    Cc = 1 + 2 * mp / Da * (1.257 + 0.4 * np.exp(-0.55 * Da / mp))
    diff = 1.3806503e-23 * T * Cc / (3 * np.pi * visc * Da)
    Re = 0.5 * rhoa * D * vt / visc
    Sc = visc / (rhoa * diff)
    St = Da * Da * vt * 1000 / (9 * visc * D)
    aval = 1 + np.log(1 + Re)
    St2 = (1.2 + aval / 12) / (1 + aval)
    Eff = 4 / (Re * Sc) * (1 + 0.4 * np.sqrt(Re) * Sc ** 0.3333 + 0.16 * np.sqrt(Re) * np.sqrt(Sc)) \
        + 4 * Da / D * (0.02 + Da / D * (1 + 2 * np.sqrt(Re)))
    Eff = Eff + np.where(St > St2, np.abs((St - St2) / (St - St2 + 0.666667)) ** 1.5, 0.0)
    return St, St2, Eff


@pytest.mark.gpu
def test_aerosol_functions_against_oracle(probe):
    """eff_aero ('r', 's', 'g'), ice_demott, ice_koop and activ_ncloud against the oracle (glibc's f32 functions).
    Outside a 1e-5 relative band around each branch condition (St > St2, the 1e-5 / 1.0 clamps of Eff, the log_J_rate
    cap at 20, prob_h > 0, the ta_Na / ta_Ww brackets and end clamps) the results agree to a few f32 ulps; the points
    that do not are printed and may only be the rare ones where one f32 ulp of an exp / log feeds a cancellation (the
    chemical-potential sum and 1 - exp(-J V dt) of ice_koop).  Inside a band the device value is the oracle's or the
    other branch's, which differ by at most the band."""
    from oracle import oracle
    rng = np.random.default_rng(18)
    n = 400_000
    args = _aero_inputs(rng, n)
    ULP = 4
    for sp in "rsg":
        a = args["eff_" + sp]
        got = probe.run32("eff_aero_" + sp, *a)
        want = oracle.eff_aero_array(*a, sp)
        St, St2, Eff = _eff_aero_f64(*a, sp)
        band = (np.abs(St - St2) <= 1e-5 * np.abs(St2)) | (np.abs(Eff - 1e-5) <= 1e-10) | (np.abs(Eff - 1) <= 1e-5)
        d = ulp_dist32(got, want)
        out = d[~band] > ULP
        print("eff_aero %s: %d points, %d in a band, %d bit-identical, %d outside the band beyond %d ulps"
              % (sp, n, band.sum(), np.count_nonzero(d == 0), out.sum(), ULP))
        assert out.sum() <= 1e-4 * n, sp
        assert np.all(np.abs(got[band].astype(np.float64) - want[band]) <= 2e-5 * np.abs(want[band]) + 1e-10), sp
        assert (St > St2).sum() > 1000 and (St < St2).sum() > 1000, sp

    got = probe.run32("ice_demott", *args["demott"])
    want = oracle.ice_demott_array(*args["demott"])
    d = ulp_dist32(got, want)
    print("ice_demott: %d bit-identical of %d, max %d ulps" % (np.count_nonzero(d == 0), n, d.max()))
    assert d.max() <= ULP

    temp, qv, qvs, naero, dt = args["koop"]
    got = probe.run32("ice_koop", *args["koop"])
    want = oracle.ice_koop_array(*args["koop"])
    t = temp.astype(np.float64)
    mu = 210368.0 + 131.438 * t - 3.32373e6 / t - 41729.1 * np.log(t)
    daw = qv.astype(np.float64) / qvs - np.exp(mu / (8.314 * t))
    logJ = -906.7 + 8502.0 * daw - 26924.0 * daw ** 2 + 29180.0 * daw ** 3
    band = np.abs(logJ - 20) <= 2e-4
    d = ulp_dist32(got, want)
    out = (d > ULP) & ~band
    print("ice_koop: %d points, %d bit-identical, %d nonzero, %d beyond %d ulps" % (
        n, np.count_nonzero(d == 0), np.count_nonzero(want), out.sum(), ULP))
    assert out.sum() <= 1e-3 * n
    assert np.count_nonzero(want > 0) > 1000 and np.count_nonzero(want == 0) > 1000 and (logJ > 20).sum() > 1000

    got = probe.run32("activ_ncloud", *args["activ"])
    want = oracle.activ_ncloud_array(*args["activ"])
    d = ulp_dist32(got, want)
    print("activ_ncloud: %d bit-identical of %d, max %d ulps" % (np.count_nonzero(d == 0), n, d.max()))
    assert d.max() <= ULP
