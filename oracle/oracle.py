"""ORACLE — TEST INFRASTRUCTURE ONLY.

ctypes wrapper over oracle/libthompson_oracle.so, the CPU restatement of the reference scheme
(/root/reference/module_mp_thompson09n.f90 = "M:", mphys_thompson09n.f90 = "I:").
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  PARITY UNPINNED by the reference (it ships no tests or vectors).
"""
import ctypes as C
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libthompson_oracle.so")
_fp = C.POINTER(C.c_float)
_dp = C.POINTER(C.c_double)


def build(force=False):
    srcs = [os.path.join(_HERE, f) for f in ("thompson_oracle.cpp", "thompson_oracle_step.inc", "thompson_oracle.h")]
    if force or not os.path.exists(_LIB) or any(
            os.path.exists(s) and os.path.getmtime(s) > os.path.getmtime(_LIB) for s in srcs):
        env = dict(os.environ)
        env.pop("CXX", None)
        subprocess.check_call(["make", "-C", _HERE, "-s"], env=env)
    return _LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB)
        L.kor_create.restype = C.c_void_p
        L.kor_create.argtypes = [C.c_float, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_int]
        L.kor_destroy.argtypes = [C.c_void_p]
        L.kor_init_seconds.restype = C.c_double
        L.kor_init_seconds.argtypes = [C.c_void_p]
        L.kor_table_size.restype = C.c_long
        L.kor_table_size.argtypes = [C.c_void_p, C.c_char_p]
        L.kor_get_table.restype = C.c_long
        L.kor_get_table.argtypes = [C.c_void_p, C.c_char_p, _dp, C.c_long]
        L.kor_mp_thompson.restype = C.c_int
        L.kor_mp_thompson.argtypes = [C.c_void_p, C.c_int, C.c_float] + [_fp] * 10 + [_fp, _fp, _fp, _dp]
        L.kor_step_aero.restype = C.c_int
        L.kor_step_aero.argtypes = [C.c_void_p, C.c_long, C.c_int, C.c_float] + [_fp] * 17 + [C.c_int]
        for name, args in (("kor_eff_aero", [C.c_float] * 5 + [C.c_char]), ("kor_ice_demott", [C.c_float] * 3),
                           ("kor_ice_koop", [C.c_float] * 5), ("kor_activ_ncloud", [C.c_float] * 3)):
            getattr(L, name).restype = C.c_float
            getattr(L, name).argtypes = args
        L.kor_step.restype = C.c_int
        L.kor_step.argtypes = [C.c_void_p, C.c_long, C.c_int, C.c_float, C.c_int] + [_fp] * 9 + [_fp, _fp, _fp, C.c_int]
        L.kor_kid_interface.restype = C.c_int
        L.kor_kid_interface.argtypes = ([C.c_void_p, C.c_long, C.c_int, C.c_float, C.c_float, C.c_float] + [_fp] * 8
                                        + [C.POINTER(_fp)] * 3 + [_fp, _fp, C.POINTER(_fp), _fp])
        L.kor_rate_names.restype = C.c_char_p
        for n in ("kor_rslf", "kor_rsif"):
            getattr(L, n).restype = C.c_float
            getattr(L, n).argtypes = [C.c_float, C.c_float]
        for n in ("kor_gammln", "kor_wgamma"):
            getattr(L, n).restype = C.c_float
            getattr(L, n).argtypes = [C.c_float]
        L.kor_gammp.restype = C.c_float
        L.kor_gammp.argtypes = [C.c_float, C.c_float]
        L.kor_calc_effect_rad.restype = C.c_int
        L.kor_calc_effect_rad.argtypes = [C.c_void_p, C.c_int] + [_fp] * 11
        L.kor_calc_effect_rad_aero.restype = C.c_int
        L.kor_calc_effect_rad_aero.argtypes = [C.c_void_p, C.c_int] + [_fp] * 11
        L.kor_mp_gt_driver.restype = C.c_int
        L.kor_mp_gt_driver.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float] + [_fp] * 22
        L.kor_decade_index.restype = C.c_int
        L.kor_decade_index.argtypes = [C.c_float, C.c_int, C.c_int]
        L.kor_decade_index_d.restype = C.c_int
        L.kor_decade_index_d.argtypes = [C.c_double, C.c_int, C.c_int]
        _ip = C.POINTER(C.c_int)
        for name, args in (("kor_rslf_array", [_fp] * 3), ("kor_rsif_array", [_fp] * 3),
                           ("kor_decade_index_array", [_fp, C.c_int, C.c_int, _ip]),
                           ("kor_decade_index_d_array", [_dp, C.c_int, C.c_int, _ip]),
                           ("kor_eff_aero_array", [_fp] * 5 + [C.c_char, _fp]), ("kor_ice_demott_array", [_fp] * 4),
                           ("kor_ice_koop_array", [_fp] * 6), ("kor_activ_ncloud_array", [_fp] * 4)):
            getattr(L, name).restype = None
            getattr(L, name).argtypes = args + [C.c_long]
        _lib = L
    return _lib


def default_cache_path():
    d = os.environ.get("KOR_CACHE_DIR", os.path.join(_HERE, "_cache"))
    os.makedirs(d, exist_ok=True)
    return os.path.join(d, "collection_tables.bin")


FIELDS = ("qv", "qc", "qi", "qr", "qs", "qg", "ni", "nr", "t")
TABLES_4D_G = ("tcg_racg", "tmr_racg", "tcr_gacr", "tmg_gacr", "tnr_racg", "tnr_gacr")
TABLES_4D_S = ("tcs_racs1", "tmr_racs1", "tcs_racs2", "tmr_racs2", "tcr_sacr1", "tms_sacr1",
               "tcr_sacr2", "tms_sacr2", "tnr_racs1", "tnr_racs2", "tnr_sacr1", "tnr_sacr2")
TABLES_SMALL = ("tpi_qcfz", "tni_qcfz", "tpi_qrfz", "tpg_qrfz", "tni_qrfz", "tnr_qrfz",
                "tps_iaus", "tni_iaus", "tpi_ide", "t_Efrw", "t_Efsw")
TABLE_SHAPES = {  # Fortran (column-major) shapes, M:386-423
    **{n: (28, 28, 37, 37) for n in TABLES_4D_G},
    **{n: (28, 9, 37, 37) for n in TABLES_4D_S},
    "tpi_qcfz": (37, 45), "tni_qcfz": (37, 45),
    "tpi_qrfz": (37, 37, 45), "tpg_qrfz": (37, 37, 45), "tni_qrfz": (37, 37, 45), "tnr_qrfz": (37, 37, 45),
    "tps_iaus": (64, 55), "tni_iaus": (64, 55), "tpi_ide": (64, 55),
    "t_Efrw": (100, 100), "t_Efsw": (100, 100),
}


class Oracle:
    """thompson_init (M:374-797) + mp_thompson (M:1156-3688) on the CPU."""

    def __init__(self, set_Nc=100.0, iiwarm=False, l_sediment=True, wp_double=False, cache=True, nthreads=None):
        L = lib()
        self.nthreads = nthreads or os.cpu_count() or 1
        cp = default_cache_path().encode() if cache else None
        self.h = L.kor_create(float(set_Nc), int(iiwarm), int(l_sediment), int(wp_double), cp, self.nthreads)
        self.iiwarm = bool(iiwarm)
        self.rate_names = L.kor_rate_names().decode().split(",")

    def close(self):
        if self.h:
            lib().kor_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def init_seconds(self):
        return lib().kor_init_seconds(self.h)

    def get(self, name):
        L = lib()
        n = L.kor_table_size(self.h, name.encode())
        if n < 0:
            raise KeyError(name)
        out = np.empty(n, dtype=np.float64)
        L.kor_get_table(self.h, name.encode(), out.ctypes.data_as(_dp), n)
        if name in TABLE_SHAPES:
            out = out.reshape(TABLE_SHAPES[name], order="F")
        return out

    def effect_rad(self, t, p, qv, qc, qi, ni, qs, nc=None):
        """calc_effectRad (M:4834-4935) for one column preset as at M:1112-1114; returns (re_qc, re_qi, re_qs).
        nc given: is_aerosol_aware = .true., the droplet number is read (M:4874)."""
        nz = len(t)
        arrs = [np.ascontiguousarray(v, dtype=np.float32) for v in (t, p, qv, qc, qi, ni, qs)]
        t, p, qv, qc, qi, ni, qs = arrs
        rc, ri, rs = (np.full(nz, v, np.float32) for v in (2.49e-6, 4.99e-6, 9.99e-6))
        P = lambda a: a.ctypes.data_as(_fp)
        if nc is not None:
            ncc = np.ascontiguousarray(nc, dtype=np.float32)
            r = lib().kor_calc_effect_rad_aero(self.h, nz, P(t), P(p), P(qv), P(qc), P(ncc), P(qi), P(ni), P(qs), P(rc), P(ri), P(rs))
            if r:
                raise RuntimeError("kor_calc_effect_rad_aero failed")
            return rc, ri, rs
        r = lib().kor_calc_effect_rad(self.h, nz, P(t), P(p), P(qv), P(qc), None, P(qi), P(ni), P(qs), P(rc), P(ri), P(rs))
        if r:
            raise RuntimeError("kor_calc_effect_rad failed")
        return rc, ri, rs

    def mp_gt_driver(self, dt, f3, pii, p, dz, acc, radii=True):
        """mp_gt_driver (M:806-1143).  f3: dict qv qc qr qi qs qg ni nr th of (nj, nk, ni) float32 arrays (C order =
        WRF's (i,k,j) Fortran order), updated in place; acc: dict rainnc rainncv sr [snownc snowncv graupelnc
        graupelncv] of (nj, ni) arrays, updated in place.  Returns dict re_cloud re_ice re_snow (or {})."""
        nj, nk, ni = f3["qv"].shape
        P = lambda a: a.ctypes.data_as(_fp) if a is not None else None
        for k in ("qv", "qc", "qr", "qi", "qs", "qg", "ni", "nr", "th"):
            assert f3[k].dtype == np.float32 and f3[k].flags.c_contiguous and f3[k].shape == (nj, nk, ni)
        re = {k: np.zeros((nj, nk, ni), np.float32) for k in ("re_cloud", "re_ice", "re_snow")} if radii else {}
        r = lib().kor_mp_gt_driver(
            self.h, ni, nk, nj, float(dt), *[P(f3[k]) for k in ("qv", "qc", "qr", "qi", "qs", "qg", "ni", "nr", "th")],
            P(np.ascontiguousarray(pii, np.float32)), P(np.ascontiguousarray(p, np.float32)),
            P(np.ascontiguousarray(dz, np.float32)), P(acc["rainnc"]), P(acc["rainncv"]), P(acc.get("snownc")),
            P(acc.get("snowncv")), P(acc.get("graupelnc")), P(acc.get("graupelncv")), P(acc["sr"]),
            P(re.get("re_cloud")), P(re.get("re_ice")), P(re.get("re_snow")))
        if r:
            raise RuntimeError("kor_mp_gt_driver failed")
        return re

    def column(self, dt, qv, qc, qi, qr, qs, qg, ni, nr, t, p, dz, nc=None, ppt=None, want_rates=False):
        """One mp_thompson call.  Arrays of nz (index 0 = lowest level); returns dict of new arrays."""
        nz = len(t)
        a = {k: np.ascontiguousarray(v, dtype=np.float32).copy()
             for k, v in zip(FIELDS, (qv, qc, qi, qr, qs, qg, ni, nr, t))}
        p = np.ascontiguousarray(p, dtype=np.float32)
        dz = np.ascontiguousarray(dz, dtype=np.float32)
        ppt4 = np.zeros(4, np.float32) if ppt is None else np.asarray(ppt, np.float32).copy()
        ncp = None
        if nc is not None:
            a["nc"] = np.ascontiguousarray(nc, dtype=np.float32).copy()
            ncp = a["nc"].ctypes.data_as(_fp)
        rates = np.zeros((36, nz), np.float64) if want_rates else None
        rc = lib().kor_mp_thompson(
            self.h, nz, float(dt), *[a[k].ctypes.data_as(_fp) for k in ("qv", "qc", "qi", "qr", "qs", "qg", "ni", "nr")],
            ncp, a["t"].ctypes.data_as(_fp), p.ctypes.data_as(_fp), dz.ctypes.data_as(_fp),
            ppt4.ctypes.data_as(_fp), rates.ctypes.data_as(_dp) if want_rates else None)
        if rc:
            raise RuntimeError("kor_mp_thompson rc=%d" % rc)
        a["ppt"] = ppt4
        if want_rates:
            a["rates"] = rates
        return a

    def step(self, dt, state, p, dz, layout="col_fastest", nthreads=None):
        """I:54-246 over many columns, in place on the float32 arrays in `state` (dict by FIELDS).
        layout 'k_fastest': arrays (ncol, nz); 'col_fastest': arrays (nz, ncol).  Returns ppt[4, ncol]."""
        lay = 0 if layout == "k_fastest" else 1
        t = state["t"]
        ncol, nz = (t.shape if lay == 0 else t.shape[::-1])
        for k in FIELDS:
            assert state[k].dtype == np.float32 and state[k].flags.c_contiguous and state[k].shape == t.shape
        assert p.dtype == np.float32 and p.flags.c_contiguous and p.shape == t.shape
        dz = np.ascontiguousarray(dz, np.float32)
        ppt = np.zeros((4, ncol), np.float32)
        rc = lib().kor_step(self.h, ncol, nz, float(dt), lay, *[state[k].ctypes.data_as(_fp) for k in FIELDS],
                            p.ctypes.data_as(_fp), dz.ctypes.data_as(_fp), ppt.ctypes.data_as(_fp),
                            int(nthreads or self.nthreads))
        if rc:
            raise RuntimeError("kor_step rc=%d" % rc)
        return ppt


    def step_aero(self, dt, state, nc, nwfa, nifa, p, w, dz, nwfa2d=None, nthreads=None):
        """mp_thompson with is_aerosol_aware = .true. (M:28) over the columns of (nz, ncol) float32 arrays, in place on
        `state` (dict by FIELDS), nc, nwfa, nifa; w: vertical velocity; nwfa2d (ncol) or None: the surface emission that
        mp_gt_driver adds to the lowest level after the step (M:1001).  Returns ppt[4, ncol]."""
        t = state["t"]
        nz, ncol = t.shape
        for a in list(state.values()) + [nc, nwfa, nifa, p, w]:
            assert a.dtype == np.float32 and a.flags.c_contiguous and a.shape == t.shape
        dz = np.ascontiguousarray(dz, np.float32)
        ppt = np.zeros((4, ncol), np.float32)
        n2 = np.ascontiguousarray(nwfa2d, np.float32) if nwfa2d is not None else None
        rc = lib().kor_step_aero(self.h, ncol, nz, float(dt), *[state[k].ctypes.data_as(_fp) for k in FIELDS],
                                 nc.ctypes.data_as(_fp), nwfa.ctypes.data_as(_fp), nifa.ctypes.data_as(_fp), p.ctypes.data_as(_fp),
                                 w.ctypes.data_as(_fp), dz.ctypes.data_as(_fp), n2.ctypes.data_as(_fp) if n2 is not None else None,
                                 ppt.ctypes.data_as(_fp), int(nthreads or self.nthreads))
        if rc:
            raise RuntimeError("kor_step_aero rc=%d" % rc)
        return ppt


def eff_aero(D, Da, visc, rhoa, temp, species):
    return float(lib().kor_eff_aero(D, Da, visc, rhoa, temp, species.encode()))


def ice_demott(tempc, rho, nifa):
    return float(lib().kor_ice_demott(tempc, rho, nifa))


def ice_koop(temp, qv, qvs, naero, dt):
    return float(lib().kor_ice_koop(temp, qv, qvs, naero, dt))


def activ_ncloud(Tt, Ww, NCCN):
    return float(lib().kor_activ_ncloud(Tt, Ww, NCCN))


HYD_PLANES = ("qc", "qr", "nr", "qi", "ni", "qs", "qg")


def kid_interface(o, kid, dt, p0=1.0e5, r_on_cp=287.05 / 1005.0):
    """I:28-246 on the oracle.  kid: dict of float32 (nx, nz) arrays 'theta', 'dtheta_adv', 'dtheta_div', 'exner',
    'qv', 'dqv_adv', 'dqv_div', plus '<m>', 'd<m>_adv', 'd<m>_div' for m in HYD_PLANES, and 'dz' (nz).
    Returns dict: 'dtheta_mphys', 'dqv_mphys', 'd<m>_mphys', 'ppt' [4, nx]."""
    nx, nz = kid["theta"].shape
    f = lambda a: np.ascontiguousarray(a, np.float32)
    a = {k: f(v) for k, v in kid.items()}
    out = {"dtheta_mphys": np.zeros((nx, nz), np.float32), "dqv_mphys": np.zeros((nx, nz), np.float32),
           "ppt": np.zeros((4, nx), np.float32)}
    for m in HYD_PLANES:
        out["d%s_mphys" % m] = np.zeros((nx, nz), np.float32)
    P = lambda x: x.ctypes.data_as(_fp)
    arr = lambda names: (_fp * 7)(*[P(a[n]) for n in names])
    hyd_out = (_fp * 7)(*[P(out["d%s_mphys" % m]) for m in HYD_PLANES])
    rc = lib().kor_kid_interface(o.h, nx, nz, float(dt), float(p0), float(r_on_cp), P(a["theta"]), P(a["dtheta_adv"]),
                                 P(a["dtheta_div"]), P(a["exner"]), P(a["qv"]), P(a["dqv_adv"]), P(a["dqv_div"]),
                                 P(a["dz"]), arr(HYD_PLANES), arr(["d%s_adv" % m for m in HYD_PLANES]),
                                 arr(["d%s_div" % m for m in HYD_PLANES]), P(out["dtheta_mphys"]), P(out["dqv_mphys"]),
                                 hyd_out, P(out["ppt"]))
    if rc:
        raise RuntimeError("kor_kid_interface rc=%d" % rc)
    return out


def rslf(p, t):
    return float(lib().kor_rslf(p, t))


def rsif(p, t):
    return float(lib().kor_rsif(p, t))


def decade_index(x, n2, ntb):
    """M:1762-1774: the table index of an f32 value (decade offset n2, ntb nodes)."""
    return int(lib().kor_decade_index(x, n2, ntb))


def decade_index_d(x, n2, ntb):
    """M:1824-1833: the same for an f64 value (the rain and graupel intercepts)."""
    return int(lib().kor_decade_index_d(x, n2, ntb))


def _array_call(fn, inputs, dtype, out_dtype, *scalars):
    """fn(in_0, ..., *scalars, out, n) over 1-D arrays broadcast to one length; returns out."""
    arrs = [np.ascontiguousarray(a, dtype) for a in np.broadcast_arrays(*[np.asarray(a) for a in inputs])]
    n = arrs[0].size
    out = np.empty(n, out_dtype)
    ptr = _dp if dtype == np.float64 else _fp
    optr = C.POINTER(C.c_int) if out_dtype == np.int32 else _fp
    fn(*[a.ravel().ctypes.data_as(ptr) for a in arrs], *scalars, out.ctypes.data_as(optr), n)
    return out


def rslf_array(p, t):
    return _array_call(lib().kor_rslf_array, (p, t), np.float32, np.float32)


def rsif_array(p, t):
    return _array_call(lib().kor_rsif_array, (p, t), np.float32, np.float32)


def decade_index_array(x, n2, ntb):
    return _array_call(lib().kor_decade_index_array, (x,), np.float32, np.int32, int(n2), int(ntb))


def decade_index_d_array(x, n2, ntb):
    return _array_call(lib().kor_decade_index_d_array, (x,), np.float64, np.int32, int(n2), int(ntb))


def eff_aero_array(D, Da, visc, rhoa, temp, species):
    return _array_call(lib().kor_eff_aero_array, (D, Da, visc, rhoa, temp), np.float32, np.float32, species.encode())


def ice_demott_array(tempc, rho, nifa):
    return _array_call(lib().kor_ice_demott_array, (tempc, rho, nifa), np.float32, np.float32)


def ice_koop_array(temp, qv, qvs, naero, dt):
    return _array_call(lib().kor_ice_koop_array, (temp, qv, qvs, naero, dt), np.float32, np.float32)


def activ_ncloud_array(Tt, Ww, NCCN):
    return _array_call(lib().kor_activ_ncloud_array, (Tt, Ww, NCCN), np.float32, np.float32)
