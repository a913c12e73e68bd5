"""ctypes binding of kid_b200/libkidmp.so (include/kidmp.h), used by the tests and bench.py.

This is plumbing only: every compute call goes through the C ABI into the CUDA kernels.  There is
no CPU path - on a machine without a CUDA device `Thompson(...)` raises `KidmpError`.
"""
import ctypes as C
import os
import numpy as np

from . import build as _build

NFIELDS = 9
FIELDS = ("qv", "qc", "qi", "qr", "qs", "qg", "ni", "nr", "t")
K_FASTEST, COL_FASTEST = 0, 1
NDIAG = 8
DIAG_NAMES = ("ppt_rain", "ppt_ice", "ppt_snow", "ppt_graupel", "lwp", "iwp", "active_columns", "columns")

_fp = C.POINTER(C.c_float)
_dp = C.POINTER(C.c_double)
_fpp = C.POINTER(_fp)


class KidmpError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [("set_Nc", C.c_float), ("iiwarm", C.c_int), ("l_sediment", C.c_int), ("wp_double", C.c_int),
                ("device", C.c_int), ("reuse_tables", C.c_int), ("table_cache_path", C.c_char_p),
                ("ndev", C.c_int), ("device_ids", C.POINTER(C.c_int))]


# every symbol include/kidmp.h declares: (restype, argtypes)
SYMBOLS = {
    "kidmp_init": (C.c_int, [C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "kidmp_finalize": (C.c_int, [C.c_void_p]),
    "kidmp_last_error": (C.c_char_p, [C.c_void_p]),
    "kidmp_build_id": (C.c_char_p, []),
    "kidmp_table_build_ms": (C.c_double, [C.c_void_p]),
    "kidmp_table_size": (C.c_long, [C.c_void_p, C.c_char_p]),
    "kidmp_get_table": (C.c_int, [C.c_void_p, C.c_char_p, _dp, C.c_long]),
    "kidmp_save_tables": (C.c_int, [C.c_void_p, C.c_char_p]),
    "kidmp_write_kid_cache": (C.c_int, [C.c_void_p, C.c_char_p, C.c_char_p]),
    "kidmp_read_kid_cache": (C.c_int, [C.c_void_p, C.c_char_p, C.c_char_p]),
    "kidmp_column": (C.c_int, [C.c_void_p, C.c_int, C.c_float] + [_fp] * 9 + [_fp, _fp, _fp]),
    "kidmp_step": (C.c_int, [C.c_void_p, C.c_long, C.c_int, C.c_float, C.c_int, _fpp, _fp, _fp, _fp]),
    "kidmp_state_alloc": (C.c_int, [C.c_void_p, C.c_long, C.c_int]),
    "kidmp_upload": (C.c_int, [C.c_void_p, C.c_int, _fpp, _fp, _fp]),
    "kidmp_step_resident": (C.c_int, [C.c_void_p, C.c_float]),
    "kidmp_download": (C.c_int, [C.c_void_p, C.c_int, _fpp, _fp]),
    "kidmp_step_device": (C.c_int, [C.c_void_p, C.c_long, C.c_int, C.c_float, C.POINTER(C.c_void_p), C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p]),
    "kidmp_step_device_aero": (C.c_int, [C.c_void_p, C.c_long, C.c_int, C.c_float, C.POINTER(C.c_void_p)] + [C.c_void_p] * 9),
    "kidmp_step_aero": (C.c_int, [C.c_void_p, C.c_long, C.c_int, C.c_float, C.c_int, _fpp] + [_fp] * 8),
    "kidmp_step_nc": (C.c_int, [C.c_void_p, C.c_long, C.c_int, C.c_float, C.c_int, _fpp, _fp, _fp, _fp, _fp]),
    "kidmp_step_device_nc": (C.c_int, [C.c_void_p, C.c_long, C.c_int, C.c_float, C.POINTER(C.c_void_p)] + [C.c_void_p] * 5),
    "kidmp_set_rates_buffer": (C.c_int, [C.c_void_p, C.c_void_p]),
    "kidmp_rate_names": (C.c_char_p, []),
    "kidmp_enable_rates": (C.c_int, [C.c_void_p, C.c_int]),
    "kidmp_get_rates": (C.c_int, [C.c_void_p, C.c_int, _fp]),
    "kidmp_diag": (C.c_int, [C.c_void_p, _dp]),
    "kidmp_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "kidmp_gpu_launches": (C.c_long, [C.c_void_p]),
    "kidmp_num_devices": (C.c_int, [C.c_void_p]),
    "kidmp_step_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_long)]),
    "kidmp_kernel_names": (C.c_char_p, []),
    "kidmp_last_kernel_ms": (C.c_int, [C.c_void_p, _fp, C.c_int]),
    "kidmp_sync": (C.c_int, [C.c_void_p]),
    "kidmp_last_step_ms": (C.c_int, [C.c_void_p, _fp]),
    "kidmp_tables_from_cache": (C.c_int, [C.c_void_p]),
    "kidmp_stream": (C.c_void_p, [C.c_void_p]),
    "kidmp_device_state": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                     C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
}



class KidColumns(C.Structure):
    """kidmp_kid_columns of include/kidmp.h."""
    _fields_ = [("nx", C.c_long), ("nz", C.c_int)] + [(n, _fp) for n in (
        "theta", "dtheta_adv", "dtheta_div", "exner", "qv", "dqv_adv", "dqv_div", "dz")] + [
        ("hyd", _fp * 7), ("dhyd_adv", _fp * 7), ("dhyd_div", _fp * 7),
        ("dtheta_mphys", _fp), ("dqv_mphys", _fp), ("dhyd_mphys", _fp * 7), ("ppt", _fp)]


class WrfFields(C.Structure):
    """kidmp_wrf_fields of include/kidmp.h."""
    _fields_ = [("ni", C.c_int), ("nk", C.c_int), ("nj", C.c_int)] + [(n, _fp) for n in (
        "qv", "qc", "qr", "qi", "qs", "qg", "ni_", "nr", "th", "pii", "p", "dz", "rainnc", "rainncv", "sr",
        "snownc", "snowncv", "graupelnc", "graupelncv", "re_cloud", "re_ice", "re_snow")]


class WrfAerosols(C.Structure):
    """kidmp_wrf_aerosols of include/kidmp.h."""
    _fields_ = [(n, _fp) for n in ("nc", "nwfa", "nifa", "w", "nwfa2d")]


SYMBOLS["kidmp_mp_gt_driver"] = (C.c_int, [C.c_void_p, C.POINTER(WrfFields), C.c_float])
SYMBOLS["kidmp_mp_gt_driver_aero"] = (C.c_int, [C.c_void_p, C.POINTER(WrfFields), C.POINTER(WrfAerosols), C.c_float])


class WrfTile(C.Structure):
    """kidmp_wrf_tile of include/kidmp.h: 0-based offsets and extents of the tile inside the memory box."""
    _fields_ = [(n, C.c_int) for n in ("i0", "ni", "k0", "nk", "j0", "nj")]


SYMBOLS["kidmp_mp_gt_driver_tile"] = (C.c_int, [C.c_void_p, C.POINTER(WrfFields), C.POINTER(WrfTile), C.POINTER(WrfAerosols),
                                                C.c_float])
SYMBOLS["kidmp_mp_gt_driver_tile_device"] = (C.c_int, [C.c_void_p, C.POINTER(WrfFields), C.POINTER(WrfTile),
                                                       C.POINTER(WrfAerosols), C.c_float, C.c_void_p])
SYMBOLS["kidmp_mp_gt_driver_tile_nc"] = (C.c_int, [C.c_void_p, C.POINTER(WrfFields), C.POINTER(WrfTile), _fp, C.c_float])
SYMBOLS["kidmp_mp_gt_driver_tile_device_nc"] = (C.c_int, [C.c_void_p, C.POINTER(WrfFields), C.POINTER(WrfTile), C.c_void_p,
                                                          C.c_float, C.c_void_p])
SYMBOLS["kidmp_kid_interface"] = (C.c_int, [C.c_void_p, C.POINTER(KidColumns), C.c_float, C.c_float, C.c_float])
HYD_PLANES = ("qc", "qr", "nr", "qi", "ni", "qs", "qg")

_lib = None


def lib_path():
    return _build.LIB


def load(build_if_missing=True):
    """dlopen the library (building it first when a source is newer and nvcc is available)."""
    global _lib
    if _lib is None:
        path = os.environ.get("KIDMP_LIB")          # tools/state_hash.py: compare two builds of the library bit for bit
        if not path:
            path = _build.LIB
            # under torchrun only local rank 0 rebuilds a stale library; the other ranks take the file that is there
            # (one build instead of eight, and nobody dlopens a file that is being replaced)
            if os.path.exists(path) and int(os.environ.get("LOCAL_RANK", "0")) != 0:
                build_if_missing = False
            if build_if_missing and _build.needs_build():
                _build.build(force=True)            # a compile error is an error: never fall back to a stale binary
        L = C.CDLL(path)
        for name, (res, args) in SYMBOLS.items():
            try:
                fn = getattr(L, name)
            except AttributeError:
                if os.environ.get("KIDMP_LIB"):         # an earlier build in an A/B run: it simply lacks the newer entry points
                    continue
                raise
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _ptrs(arrs):
    return (_fp * len(arrs))(*[a.ctypes.data_as(_fp) for a in arrs])


def _f32c(a):
    a = np.asarray(a)
    if a.dtype != np.float32 or not a.flags.c_contiguous:
        raise ValueError("float32 C-contiguous array required")
    return a


class Thompson:
    """One handle = thompson_init (M:374-797) done on one GPU, plus the column step entry points."""

    def __init__(self, set_Nc=100.0, iiwarm=False, l_sediment=True, wp_double=False, device=0,
                 table_cache=None, reuse_tables=False, devices=None):
        """devices: list of CUDA ordinals for ONE handle over several GPUs (kidmp_config::ndev), else `device`."""
        L = load()
        self._L = L
        ids = (C.c_int * len(devices))(*devices) if devices else None
        if devices and len(devices) > 1 and "KIDMP_NCCL_LIB" not in os.environ:
            try:                                      # the NCCL that torch ships, when there is no system libnccl.so.2
                import nvidia.nccl
                cand = os.path.join(os.path.dirname(nvidia.nccl.__file__), "lib", "libnccl.so.2")
                if os.path.exists(cand):
                    os.environ["KIDMP_NCCL_LIB"] = cand
            except Exception:
                pass
        cfg = Config(float(set_Nc), int(iiwarm), int(l_sediment), int(wp_double), int(device),
                     int(bool(reuse_tables and table_cache)), table_cache.encode() if table_cache else None,
                     len(devices) if devices else 0, ids)
        h = C.c_void_p()
        rc = L.kidmp_init(C.byref(cfg), C.byref(h))
        if rc:
            raise KidmpError(L.kidmp_last_error(None).decode())
        self.h = h
        self.iiwarm = bool(iiwarm)

    # -- lifecycle ------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "h", None):
            self._L.kidmp_finalize(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc:
            raise KidmpError(self._L.kidmp_last_error(self.h).decode())

    # -- tables -----------------------------------------------------------------------------------
    @property
    def table_build_ms(self):
        return self._L.kidmp_table_build_ms(self.h)

    @property
    def tables_from_cache(self):
        return bool(self._L.kidmp_tables_from_cache(self.h))

    def get(self, name):
        n = self._L.kidmp_table_size(self.h, name.encode())
        if n < 0:
            raise KeyError(name)
        out = np.empty(n, np.float64)
        self._ck(self._L.kidmp_get_table(self.h, name.encode(), out.ctypes.data_as(_dp), n))
        return out

    def save_tables(self, path):
        self._ck(self._L.kidmp_save_tables(self.h, path.encode()))

    def write_kid_cache(self, racg_path, racs_path):
        """KiD's list-directed text cache files run_data/racg_thompson09.data / racs_thompson09.data (M:3710-3728 ...)."""
        self._ck(self._L.kidmp_write_kid_cache(self.h, racg_path.encode(), racs_path.encode()))

    def read_kid_cache(self, racg_path, racs_path):
        self._ck(self._L.kidmp_read_kid_cache(self.h, racg_path.encode(), racs_path.encode()))

    # -- steps --------------------------------------------------------------------------------------
    def column(self, dt, qv, qc, qi, qr, qs, qg, ni, nr, t, p, dz, ppt=None):
        """Twin of `call mp_thompson(...)` for one column (M:1156-1162); returns dict of new arrays."""
        a = {k: np.ascontiguousarray(v, np.float32).copy() for k, v in zip(FIELDS, (qv, qc, qi, qr, qs, qg, ni, nr, t))}
        p = np.ascontiguousarray(p, np.float32)
        dz = np.ascontiguousarray(dz, np.float32)
        ppt4 = np.zeros(4, np.float32) if ppt is None else np.asarray(ppt, np.float32).copy()
        self._ck(self._L.kidmp_column(self.h, len(p), float(dt), *[a[k].ctypes.data_as(_fp) for k in FIELDS],
                                      p.ctypes.data_as(_fp), dz.ctypes.data_as(_fp), ppt4.ctypes.data_as(_fp)))
        a["ppt"] = ppt4
        return a

    def step(self, dt, state, p, dz, layout="col_fastest", set_nc=None):
        """Host arrays in, host arrays out (in place).  state: dict by FIELDS of float32 arrays,
        (nz, ncol) for 'col_fastest' or (ncol, nz) for 'k_fastest'.  Returns ppt[4, ncol].
        set_nc: float32 (ncol,) set_Nc [cm^-3] of every column (plain scheme, kidmp_step_nc); None = the handle's set_Nc."""
        lay = K_FASTEST if layout == "k_fastest" else COL_FASTEST
        t = _f32c(state["t"])
        ncol, nz = (t.shape if lay == K_FASTEST else t.shape[::-1])
        arrs = [_f32c(state[k]) for k in FIELDS]
        ppt = np.zeros((4, ncol), np.float32)
        args = (self.h, ncol, nz, float(dt), lay, _ptrs(arrs), _f32c(p).ctypes.data_as(_fp),
                np.ascontiguousarray(dz, np.float32).ctypes.data_as(_fp))
        if set_nc is None:
            self._ck(self._L.kidmp_step(*args, ppt.ctypes.data_as(_fp)))
        else:
            if np.shape(set_nc) != (ncol,):
                raise ValueError("set_nc shape %r, expected (%d,)" % (np.shape(set_nc), ncol))
            self._ck(self._L.kidmp_step_nc(*args, _f32c(set_nc).ctypes.data_as(_fp), ppt.ctypes.data_as(_fp)))
        return ppt

    def step_aero(self, dt, state, aero, p, w, dz, layout="col_fastest", nwfa2d=None):
        """kidmp_step_aero: the aerosol-aware step (is_aerosol_aware = .true.) on host arrays, in place.  state as in step;
        aero: dict nc nwfa nifa of float32 arrays shaped like the fields, updated in place; w the same shape; nwfa2d: float32
        (ncol,) surface emission or None.  Returns ppt[4, ncol]."""
        lay = K_FASTEST if layout == "k_fastest" else COL_FASTEST
        t = _f32c(state["t"])
        ncol, nz = (t.shape if lay == K_FASTEST else t.shape[::-1])
        for name, a in (("nc", aero["nc"]), ("nwfa", aero["nwfa"]), ("nifa", aero["nifa"]), ("w", w)):
            if np.shape(a) != t.shape:
                raise ValueError("%s shape %r, expected %r" % (name, np.shape(a), t.shape))
        if nwfa2d is not None and np.shape(nwfa2d) != (ncol,):
            raise ValueError("nwfa2d shape %r, expected (%d,)" % (np.shape(nwfa2d), ncol))
        arrs = [_f32c(state[k]) for k in FIELDS]
        ae = [_f32c(aero[k]) for k in ("nc", "nwfa", "nifa")]
        P = lambda a: a.ctypes.data_as(_fp)
        ppt = np.zeros((4, ncol), np.float32)
        self._ck(self._L.kidmp_step_aero(self.h, ncol, nz, float(dt), lay, _ptrs(arrs), *[P(a) for a in ae], P(_f32c(p)), P(_f32c(w)),
                                         P(np.ascontiguousarray(dz, np.float32)), P(_f32c(nwfa2d)) if nwfa2d is not None else None,
                                         P(ppt)))
        return ppt

    def state_alloc(self, ncol, nz):
        self._ck(self._L.kidmp_state_alloc(self.h, int(ncol), int(nz)))
        self.ncol, self.nz = int(ncol), int(nz)

    def upload(self, state, p, dz, layout="col_fastest"):
        lay = K_FASTEST if layout == "k_fastest" else COL_FASTEST
        arrs = [_f32c(state[k]) for k in FIELDS]
        self._ck(self._L.kidmp_upload(self.h, lay, _ptrs(arrs), _f32c(p).ctypes.data_as(_fp),
                                      np.ascontiguousarray(dz, np.float32).ctypes.data_as(_fp)))

    def step_resident(self, dt):
        self._ck(self._L.kidmp_step_resident(self.h, float(dt)))

    def download(self, state=None, layout="col_fastest", want_ppt=True):
        lay = K_FASTEST if layout == "k_fastest" else COL_FASTEST
        ppt = np.zeros((4, self.ncol), np.float32) if want_ppt else None
        fp = _ptrs([_f32c(state[k]) for k in FIELDS]) if state is not None else None
        self._ck(self._L.kidmp_download(self.h, lay, fp, ppt.ctypes.data_as(_fp) if want_ppt else None))
        return ppt

    def step_device(self, ncol, nz, dt, field_ptrs, p_ptr, dz_ptr, ppt_ptr, stream=None, set_nc_ptr=None):
        """Device pointers (ints, e.g. torch.Tensor.data_ptr()), COL_FASTEST layout; asynchronous.
        set_nc_ptr: device float32 [ncol] set_Nc of every column (kidmp_step_device_nc), None = the handle's set_Nc."""
        fp = (C.c_void_p * NFIELDS)(*[C.c_void_p(int(x)) for x in field_ptrs])
        s = C.c_void_p(int(stream)) if stream else None
        if set_nc_ptr is None:
            self._ck(self._L.kidmp_step_device(self.h, int(ncol), int(nz), float(dt), fp, C.c_void_p(int(p_ptr)),
                                               C.c_void_p(int(dz_ptr)), C.c_void_p(int(ppt_ptr)), s))
        else:
            self._ck(self._L.kidmp_step_device_nc(self.h, int(ncol), int(nz), float(dt), fp, C.c_void_p(int(p_ptr)),
                                                  C.c_void_p(int(dz_ptr)), C.c_void_p(int(set_nc_ptr)), C.c_void_p(int(ppt_ptr)), s))

    def step_device_aero(self, ncol, nz, dt, field_ptrs, nc_ptr, nwfa_ptr, nifa_ptr, p_ptr, w_ptr, dz_ptr, ppt_ptr, nwfa2d_ptr=None,
                         stream=None):
        """kidmp_step_device_aero: the aerosol-aware step (is_aerosol_aware = .true.); device pointers, COL_FASTEST."""
        fp = (C.c_void_p * NFIELDS)(*[C.c_void_p(int(x)) for x in field_ptrs])
        v = lambda x: C.c_void_p(int(x)) if x else None
        self._ck(self._L.kidmp_step_device_aero(self.h, int(ncol), int(nz), float(dt), fp, v(nc_ptr), v(nwfa_ptr), v(nifa_ptr),
                                                v(p_ptr), v(w_ptr), v(dz_ptr), v(nwfa2d_ptr), v(ppt_ptr), v(stream)))

    def device_state(self):
        f = (C.c_void_p * NFIELDS)()
        p, dz, ppt = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._ck(self._L.kidmp_device_state(self.h, f, C.byref(p), C.byref(dz), C.byref(ppt)))
        return [int(x) for x in f], int(p.value), int(dz.value), int(ppt.value)

    def set_option(self, name, value):
        """kidmp_set_option: tuning knobs that do not change results ("chunk": columns per launch, "timing": 0 / 1)."""
        self._ck(self._L.kidmp_set_option(self.h, name.encode(), int(value)))

    def mp_gt_driver(self, dt, f3, pii, p, dz, acc, radii=True, aerosols=None, tile=None, set_nc=None):
        """mp_gt_driver (M:806-1143) through kidmp_mp_gt_driver.  f3: dict qv qc qr qi qs qg ni nr th of (nj, nk, ni)
        float32 arrays (C order = WRF's (i,k,j) Fortran order), updated in place; pii, p, dz the same shape; acc: dict
        rainnc rainncv sr [snownc snowncv graupelnc graupelncv] of (nj, ni) arrays, updated in place.
        aerosols: dict nc nwfa nifa w of (nj, nk, ni) arrays [+ nwfa2d (nj, ni)]: is_aerosol_aware = .true. through
        kidmp_mp_gt_driver_aero (nc, nwfa, nifa updated in place).
        tile: (i0, ni, k0, nk, j0, nj) steps only that tile of the arrays, which are then the memory box (halo points and
        spare levels included), through kidmp_mp_gt_driver_tile; nothing outside the tile is read or written.
        radii: True = new zero arrays of the memory box's shape, returned (outside a tile they stay zero); a dict of
        re_cloud re_ice re_snow arrays = those, filled in place; False = no radii.
        set_nc: (nj, ni) float32 set_Nc [cm^-3] of every column of the memory box (plain scheme, kidmp_mp_gt_driver_tile_nc;
        read at the tile's cells only); None = the handle's set_Nc.
        Returns dict re_cloud re_ice re_snow (empty when radii is False)."""
        nj, nk, ni = f3["qv"].shape
        w, ae, re, keep = self._wrf_structs(f3, pii, p, dz, acc, radii, aerosols, (nj, nk, ni), lambda a: _f32c(a).ctypes.data_as(_fp))
        if set_nc is not None:
            if ae is not None:
                raise ValueError("set_nc is for the plain scheme: not with aerosols")
            if np.shape(set_nc) != (nj, ni):
                raise ValueError("set_nc shape %r, expected %r" % (np.shape(set_nc), (nj, ni)))
            t = WrfTile(*[int(x) for x in (tile if tile is not None else (0, ni, 0, nk, 0, nj))])
            self._ck(self._L.kidmp_mp_gt_driver_tile_nc(self.h, C.byref(w), C.byref(t), _f32c(set_nc).ctypes.data_as(_fp),
                                                        float(dt)))
        elif tile is not None:
            t = WrfTile(*[int(x) for x in tile])
            self._ck(self._L.kidmp_mp_gt_driver_tile(self.h, C.byref(w), C.byref(t), C.byref(ae) if ae is not None else None,
                                                     float(dt)))
        elif ae is not None:
            self._ck(self._L.kidmp_mp_gt_driver_aero(self.h, C.byref(w), C.byref(ae), float(dt)))
        else:
            self._ck(self._L.kidmp_mp_gt_driver(self.h, C.byref(w), float(dt)))
        return re

    def mp_gt_driver_device(self, dt, f3, pii, p, dz, acc, tile=None, radii=None, aerosols=None, stream=None, set_nc=None):
        """kidmp_mp_gt_driver_tile_device: the same step on device arrays (anything with data_ptr(), e.g. contiguous float32
        CUDA tensors of the shapes of mp_gt_driver), enqueued on `stream` (a torch.cuda.Stream, a cudaStream_t as int, or
        None = the handle's stream) without synchronising.  tile None = the whole memory box.  radii: dict re_cloud re_ice
        re_snow of device arrays (filled inside the tile) or None.  set_nc: (nj, ni) device array of set_Nc per column
        (plain scheme, kidmp_mp_gt_driver_tile_device_nc), None = the handle's set_Nc."""
        nj, nk, ni = f3["qv"].shape
        w, ae, _, keep = self._wrf_structs(f3, pii, p, dz, acc, radii or False, aerosols, (nj, nk, ni),
                                           lambda a: C.cast(C.c_void_p(int(a.data_ptr())), _fp))
        t = WrfTile(*[int(x) for x in (tile if tile is not None else (0, ni, 0, nk, 0, nj))])
        s = getattr(stream, "cuda_stream", stream)
        s = C.c_void_p(int(s)) if s else None
        if set_nc is not None:
            if ae is not None:
                raise ValueError("set_nc is for the plain scheme: not with aerosols")
            if tuple(set_nc.shape) != (nj, ni) or not set_nc.is_contiguous() or str(set_nc.dtype) != "torch.float32":
                raise ValueError("set_nc: float32 contiguous tensor of shape %r required" % ((nj, ni),))
            self._ck(self._L.kidmp_mp_gt_driver_tile_device_nc(self.h, C.byref(w), C.byref(t), C.c_void_p(int(set_nc.data_ptr())),
                                                               float(dt), s))
        else:
            self._ck(self._L.kidmp_mp_gt_driver_tile_device(self.h, C.byref(w), C.byref(t), C.byref(ae) if ae is not None else None,
                                                            float(dt), s))

    @staticmethod
    def _wrf_structs(f3, pii, p, dz, acc, radii, aerosols, shape3, addr):
        """kidmp_wrf_fields / kidmp_wrf_aerosols over the arrays; addr(a) gives an array's address."""
        nj, nk, ni = shape3
        w = WrfFields()
        w.ni, w.nk, w.nj = ni, nk, nj
        keep = []

        def ptr(a, shape):
            if tuple(a.shape) != shape:
                raise ValueError("array shape %r, expected %r" % (tuple(a.shape), shape))
            if hasattr(a, "is_contiguous") and (not a.is_contiguous() or str(a.dtype) != "torch.float32"):
                raise ValueError("float32 contiguous tensor required")
            keep.append(a)
            return addr(a)
        for name, key in (("qv", "qv"), ("qc", "qc"), ("qr", "qr"), ("qi", "qi"), ("qs", "qs"), ("qg", "qg"),
                          ("ni_", "ni"), ("nr", "nr"), ("th", "th")):
            setattr(w, name, ptr(f3[key], (nj, nk, ni)))
        w.pii, w.p, w.dz = ptr(pii, (nj, nk, ni)), ptr(p, (nj, nk, ni)), ptr(dz, (nj, nk, ni))
        for name in ("rainnc", "rainncv", "sr"):
            setattr(w, name, ptr(acc[name], (nj, ni)))
        for name in ("snownc", "snowncv", "graupelnc", "graupelncv"):
            if acc.get(name) is not None:
                setattr(w, name, ptr(acc[name], (nj, ni)))
        if radii is True:
            re = {k: np.zeros((nj, nk, ni), np.float32) for k in ("re_cloud", "re_ice", "re_snow")}
        else:
            re = dict(radii) if radii else {}
        for name, a in re.items():
            setattr(w, name, ptr(a, (nj, nk, ni)))
        ae = None
        if aerosols is not None:
            ae = WrfAerosols()
            for name in ("nc", "nwfa", "nifa", "w"):
                setattr(ae, name, ptr(aerosols[name], (nj, nk, ni)))
            if aerosols.get("nwfa2d") is not None:
                ae.nwfa2d = ptr(aerosols["nwfa2d"], (nj, ni))
        return w, ae, re, keep

    def kid_interface(self, kid, dt, p0=1.0e5, r_on_cp=287.05 / 1005.0):
        """mphys_thompson09_interfacen (I:28-246) without save_dg.  kid: dict of float32 (nx, nz) arrays 'theta',
        'dtheta_adv', 'dtheta_div', 'exner', 'qv', 'dqv_adv', 'dqv_div', '<m>', 'd<m>_adv', 'd<m>_div' for m in
        HYD_PLANES, and 'dz' (nz).  Returns 'dtheta_mphys', 'dqv_mphys', 'd<m>_mphys', 'ppt' [4, nx]."""
        nx, nz = kid["theta"].shape
        a = {k: np.ascontiguousarray(v, np.float32) for k, v in kid.items()}
        out = {"dtheta_mphys": np.zeros((nx, nz), np.float32), "dqv_mphys": np.zeros((nx, nz), np.float32),
               "ppt": np.zeros((4, nx), np.float32)}
        for m in HYD_PLANES:
            out["d%s_mphys" % m] = np.zeros((nx, nz), np.float32)
        P = lambda x: x.ctypes.data_as(_fp)
        c = KidColumns()
        c.nx, c.nz = nx, nz
        for n in ("theta", "dtheta_adv", "dtheta_div", "exner", "qv", "dqv_adv", "dqv_div", "dz"):
            setattr(c, n, P(a[n]))
        for j, m in enumerate(HYD_PLANES):
            c.hyd[j], c.dhyd_adv[j], c.dhyd_div[j] = P(a[m]), P(a["d%s_adv" % m]), P(a["d%s_div" % m])
            c.dhyd_mphys[j] = P(out["d%s_mphys" % m])
        c.dtheta_mphys, c.dqv_mphys, c.ppt = P(out["dtheta_mphys"]), P(out["dqv_mphys"]), P(out["ppt"])
        self._ck(self._L.kidmp_kid_interface(self.h, C.byref(c), float(dt), float(p0), float(r_on_cp)))
        return out

    def set_rates_buffer(self, ptr):
        self._ck(self._L.kidmp_set_rates_buffer(self.h, C.c_void_p(int(ptr)) if ptr else None))

    def enable_rates(self, on=True):
        self._ck(self._L.kidmp_enable_rates(self.h, int(bool(on))))

    def get_rates(self, ncol, nz, layout="k_fastest"):
        """The 36 save_dg rates of the last step of the resident state: (36, ncol, nz) for 'k_fastest', (36, nz, ncol) else."""
        lay = K_FASTEST if layout == "k_fastest" else COL_FASTEST
        out = np.zeros((36, ncol, nz) if lay == K_FASTEST else (36, nz, ncol), np.float32)
        self._ck(self._L.kidmp_get_rates(self.h, lay, out.ctypes.data_as(_fp)))
        return out

    @property
    def rate_names(self):
        return self._L.kidmp_rate_names().decode().split(",")

    def diag(self):
        out = np.zeros(NDIAG, np.float64)
        self._ck(self._L.kidmp_diag(self.h, out.ctypes.data_as(_dp)))
        return out

    def step_stats(self):
        """Counts of the last launch of the step kernels: cloudy columns, busy cells (total and per cell kernel), columns
        with sedimentation sub-steps."""
        out = (C.c_long * 8)()
        self._ck(self._L.kidmp_step_stats(self.h, out))
        names = ("cloudy_columns", "busy_cells", "cells_warm", "cells_ice", "cells_mixed_no_rain", "cells_full", "substep_columns",
                 "zero_copy_return")
        return {n: int(out[i]) for i, n in enumerate(names)}

    def last_kernel_ms(self):
        """{kernel group: ms} of the last launch, after set_option("timing", 1)."""
        names = self._L.kidmp_kernel_names().decode().split(",")
        out = (C.c_float * len(names))()
        self._ck(self._L.kidmp_last_kernel_ms(self.h, out, len(names)))
        return {n: float(out[i]) for i, n in enumerate(names)}

    def sync(self):
        self._ck(self._L.kidmp_sync(self.h))

    @property
    def gpu_launches(self):
        return int(self._L.kidmp_gpu_launches(self.h))

    @property
    def stream(self):
        return int(self._L.kidmp_stream(self.h) or 0)

    def last_step_ms(self):
        ms = C.c_float()
        self._ck(self._L.kidmp_last_step_ms(self.h, C.byref(ms)))
        return float(ms.value)
