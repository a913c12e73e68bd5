"""mp_gt_driver over memory and tile dimensions: kidmp_mp_gt_driver_tile (host arrays) and kidmp_mp_gt_driver_tile_device
(device arrays).  WRF and MPAS arrays are (ims:ime, kms:kme, jms:jme) with halo points around the tile and one spare level on
top (kme = kte + 1); a call steps one tile of them and must read and write nothing else: the OpenMP tiles of one patch run at
the same time on one shared array.  Inside the tile the result is the packed entry's on the same tile, bit for bit."""
import ctypes as C
import os
import re
import threading

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F3 = ("qv", "qc", "qr", "qi", "qs", "qg", "ni", "nr", "th")
IN3 = ("pii", "p", "dz")
RE3 = ("re_cloud", "re_ice", "re_snow")
ACC = ("rainnc", "rainncv", "sr", "snownc", "snowncv", "graupelnc", "graupelncv")
AE3 = ("nc", "nwfa", "nifa", "w")


# ---- CPU: the Fortran shim binds the new type and functions as the header declares them -----------------------------------
def _read(*parts):
    return open(os.path.join(ROOT, *parts)).read()


def test_shim_tile_type_lists_the_c_members_in_order():
    hdr, f90 = _read("include", "kidmp.h"), _read("kid_b200", "fortran", "mphys_thompson09n.f90")
    c_body = re.search(r"typedef struct kidmp_wrf_tile\s*\{(.*?)\}\s*kidmp_wrf_tile;", hdr, re.S).group(1)
    c_members = [n.strip() for decl in c_body.split(";") if decl.strip()
                 for n in re.sub(r"^\s*int\s+", "", decl).split(",")]
    f_body = re.search(r"type, bind\(C\) :: kidmp_wrf_tile(.*?)end type kidmp_wrf_tile", f90, re.S).group(1)
    f_members = [n.strip() for line in f_body.split("\n") if "::" in line.split("!")[0]
                 for n in line.split("!")[0].split("::")[1].split(",")]
    assert c_members == ["i0", "ni", "k0", "nk", "j0", "nj"]
    assert [m.lower() for m in f_members] == c_members
    assert re.search(r"integer\(c_int\)\s*::\s*i0", f_body)


def test_shim_tile_functions_are_declared_in_the_header():
    hdr = re.sub(r"/\*.*?\*/", "", _read("include", "kidmp.h"), flags=re.S)
    f90 = _read("kid_b200", "fortran", "mphys_thompson09n.f90")
    declared = set(re.findall(r"\b(kidmp_[a-z0-9_]+)\s*\(", hdr))
    bound = set(re.findall(r"bind\(C,\s*name='(kidmp_[a-z0-9_]+)'\)", f90))
    assert {"kidmp_mp_gt_driver_tile", "kidmp_mp_gt_driver_tile_device"} <= bound
    assert bound <= declared
    # ae by value, so that c_null_ptr selects the plain scheme
    for name in ("kidmp_mp_gt_driver_tile", "kidmp_mp_gt_driver_tile_device"):
        body = re.search(r"function %s\(.*?end function %s" % (name, name), f90, re.S).group(0)
        assert re.search(r"type\(c_ptr\), value :: ae\b", body), name
        assert re.search(r"type\(kidmp_wrf_tile\), intent\(in\) :: t\b", body), name


def test_binding_tile_struct_matches_the_header():
    from kid_b200 import kidmp
    assert [n for n, _ in kidmp.WrfTile._fields_] == ["i0", "ni", "k0", "nk", "j0", "nj"]
    assert C.sizeof(kidmp.WrfTile) == 6 * 4


# ---- GPU ------------------------------------------------------------------------------------------------------------------
def _wrf_case(ni, nk, nj, seed=3, warm=False):
    """(i,k,j) arrays of one tile from the synthetic cloudy domain: theta and Exner function instead of T, layer depths that
    differ from column to column, accumulators with a history (as tests/test_gpu_parity.py::_wrf_case)."""
    from kid_b200 import synth
    rng = np.random.default_rng(seed)
    st, p, dz = synth.make_domain(ni * nj, nz=nk, coherent=False, cloudy_fraction=0.6)
    st = {k: v.numpy().copy() for k, v in st.items()}
    p, dz = p.numpy().copy(), dz.numpy().copy()
    if warm:
        for k in ("qi", "qs", "qg", "ni"):
            st[k][:] = 0.0
    to3 = lambda a: np.ascontiguousarray(a.reshape(nk, nj, ni).transpose(1, 0, 2))     # [k][col] -> (nj, nk, ni)
    f3 = {k: to3(st[k]) for k in ("qv", "qc", "qr", "qi", "qs", "qg", "ni", "nr")}
    p3 = to3(p)
    pii = ((p3 / 1.0e5) ** (287.04 / 1004.0)).astype(np.float32)
    f3["th"] = (to3(st["t"]) / pii).astype(np.float32)
    stretch = (0.8 + 0.4 * rng.random((nj, 1, ni))).astype(np.float32)
    dz3 = np.ascontiguousarray(np.broadcast_to(dz.reshape(1, nk, 1), (nj, nk, ni)) * stretch).astype(np.float32)
    acc = {k: (rng.random((nj, ni)) * 3.0).astype(np.float32) for k in ACC}
    planes = lambda a: np.ascontiguousarray(a.transpose(1, 0, 2).reshape(nk, nj * ni))
    cube = lambda a: np.ascontiguousarray(a.reshape(nk, nj, ni).transpose(1, 0, 2))
    nc, nwfa, nifa, w = synth.make_aerosols(dict(st, t=planes(f3["th"] * pii)), planes(p3), seed=seed + 90)
    ae = {"nc": cube(nc), "nwfa": cube(nwfa), "nifa": cube(nifa), "w": cube(w),
          "nwfa2d": rng.uniform(0.0, 2.0e5, (nj, ni)).astype(np.float32)}
    vals = dict(f3, pii=pii, p=p3, dz=dz3, **acc)
    return vals, ae


def _nans(shape, tag):
    """Quiet NaNs whose payload names the array (tag) and the cell: any read-modify-write shows."""
    n = int(np.prod(shape))
    bits = np.uint32(0x7FC00000) | np.uint32(tag << 16) | (np.arange(n, dtype=np.uint32) & np.uint32(0xFFFF))
    return bits.view(np.float32).reshape(shape)


class Patch:
    """Memory-box arrays (NaN outside the tile) with one tile's case in them, and the same case packed on its own."""

    def __init__(self, ni, nk, nj, hi=(2, 3), hj=(1, 2), k0=0, spare=1, seed=3, warm=False, full=True, aero=False):
        vals, ae = _wrf_case(ni, nk, nj, seed, warm)
        self.mem_shape = (nj + hj[0] + hj[1], k0 + nk + spare, ni + hi[0] + hi[1])
        self.tile = (hi[0], ni, k0, nk, hj[0], nj)
        self.s3 = (slice(hj[0], hj[0] + nj), slice(k0, k0 + nk), slice(hi[0], hi[0] + ni))
        self.s2 = (self.s3[0], self.s3[2])
        names3 = F3 + IN3 + (RE3 if full else RE3[:2]) + (AE3 if aero else ())
        names2 = (ACC if full else ACC[:3]) + (("nwfa2d",) if aero else ())
        self.mem, self.packed = {}, {}
        for tag, name in enumerate(names3 + names2):
            three = name in names3
            shape = self.mem_shape if three else (self.mem_shape[0], self.mem_shape[2])
            a = _nans(shape, tag + 1)
            src = ae.get(name, vals.get(name))
            if src is not None:
                a[self.s3 if three else self.s2] = src
                self.packed[name] = src.copy()
            self.mem[name] = a
        self.before = {k: v.copy() for k, v in self.mem.items()}
        self.full, self.aero = full, aero

    def args(self, arrs=None):
        """mp_gt_driver's arguments over `arrs` (default: the memory box)."""
        a = self.mem if arrs is None else arrs
        f3 = {k: a[k] for k in F3}
        acc = {k: a[k] for k in ACC if k in a}
        radii = {k: a[k] for k in RE3 if k in a}
        ae = {k: a[k] for k in AE3 + ("nwfa2d",) if k in a} if self.aero else None
        return f3, a["pii"], a["p"], a["dz"], acc, radii, ae

    def run_packed(self, gpu, dt=20.0):
        """The packed entry (kidmp_mp_gt_driver[_aero]) on the tile alone: the reference bits."""
        f3, pii, p, dz, acc, _, ae = self.args(self.packed)
        re = gpu.mp_gt_driver(dt, f3, pii, p, dz, acc, radii=self.full, aerosols=ae)
        out = {k: v.copy() for k, v in self.packed.items()}
        out.update(re)
        return out

    def run_tile(self, gpu, dt=20.0):
        f3, pii, p, dz, acc, radii, ae = self.args()
        gpu.mp_gt_driver(dt, f3, pii, p, dz, acc, radii=radii, aerosols=ae, tile=self.tile)

    def check(self, got, want):
        """Outside the tile every cell of every array is bit-identical to before; inside it the bits are `want`'s."""
        for k, a in got.items():
            s = self.s3 if a.ndim == 3 else self.s2
            out_now, out_was = a.view(np.uint32).copy(), self.before[k].view(np.uint32).copy()
            out_now[s] = 0
            out_was[s] = 0
            assert np.array_equal(out_now, out_was), "%s: a cell outside the tile changed" % k
            if k in want:
                assert np.array_equal(a[s].view(np.uint32), want[k].view(np.uint32)), "%s: tile differs from the packed entry" % k
            else:                                                       # (radii not requested: not touched at all)
                assert np.array_equal(a.view(np.uint32), self.before[k].view(np.uint32)), k
        for k in F3 + ("rainnc",):
            assert np.isfinite(got[k][self.s3 if got[k].ndim == 3 else self.s2]).all(), k


# odd memory widths, ni = 1, nj = 1 (MPAS: one row of cells), ni not a multiple of 32 or 128, k0 = 1; halos on all four sides
# (except in j for the MPAS shape) and kme = kte + 1
CASES = {
    "odd": dict(ni=37, nk=30, nj=5, hi=(3, 3), hj=(2, 2)),
    "ni1": dict(ni=1, nk=25, nj=7, hi=(2, 2), hj=(1, 2)),
    "mpas": dict(ni=301, nk=20, nj=1, hi=(0, 6), hj=(0, 0)),
    "ni133": dict(ni=133, nk=24, nj=3, hi=(5, 5), hj=(5, 5)),
    "k0": dict(ni=40, nk=20, nj=4, hi=(2, 3), hj=(1, 2), k0=1, spare=2),
    "no_options": dict(ni=45, nk=22, nj=3, hi=(1, 1), hj=(1, 1), full=False),
}


@pytest.mark.gpu
@pytest.mark.parametrize("handle", ["gpu_mixed", "gpu_warm"])
@pytest.mark.parametrize("case", list(CASES))
def test_halo_and_spare_levels_are_never_touched(case, handle, request):
    gpu = request.getfixturevalue(handle)
    pt = Patch(warm=handle == "gpu_warm", **CASES[case])
    want = pt.run_packed(gpu)
    pt.run_tile(gpu)
    pt.check(pt.mem, want)


@pytest.mark.gpu
@pytest.mark.parametrize("with_nwfa2d", [True, False])
@pytest.mark.parametrize("case", ["odd", "ni1", "mpas", "k0"])
def test_aerosol_aware_tile(case, with_nwfa2d, gpu_mixed):
    pt = Patch(aero=True, seed=11, **CASES[case])
    if not with_nwfa2d:
        del pt.mem["nwfa2d"], pt.packed["nwfa2d"], pt.before["nwfa2d"]
    want = pt.run_packed(gpu_mixed)
    pt.run_tile(gpu_mixed)
    pt.check(pt.mem, want)


@pytest.mark.gpu
@pytest.mark.parametrize("aero", [False, True])
def test_whole_box_as_tile_equals_the_packed_entry(aero, gpu_mixed):
    pt = Patch(ni=50, nk=30, nj=6, hi=(0, 0), hj=(0, 0), spare=0, aero=aero)
    assert pt.mem_shape == (6, 30, 50) and pt.tile == (0, 50, 0, 30, 0, 6)
    want = pt.run_packed(gpu_mixed)
    pt.run_tile(gpu_mixed)
    pt.check(pt.mem, want)


@pytest.mark.gpu
def test_tile_against_the_oracle(gpu_mixed, oracle_mixed):
    """One tile against oracle_mixed.mp_gt_driver on the packed tile, with the tolerances of test_wrf_driver_entry."""
    from parity_util import assert_parity
    pt = Patch(ni=50, nk=60, nj=9, hi=(3, 4), hj=(2, 3))
    pt.run_tile(gpu_mixed)
    f3, pii, p, dz, acc, _, _ = pt.args({k: v.copy() for k, v in pt.packed.items()})
    rb = oracle_mixed.mp_gt_driver(20.0, f3, pii, p, dz, acc)
    got = {k: pt.mem[k][pt.s3].reshape(-1) for k in F3}
    assert_parity(got, {k: v.reshape(-1) for k, v in f3.items()}, fields=F3, what="tile mp_gt_driver state")
    for k in ACC:
        np.testing.assert_allclose(pt.mem[k][pt.s2], acc[k], rtol=1e-5, atol=1e-9, err_msg=k)
    assert (pt.mem["rainncv"][pt.s2] > 0).any()
    for k in RE3:
        np.testing.assert_allclose(pt.mem[k][pt.s3], rb[k], rtol=2e-5, err_msg=k)


def _to_dev(arrs):
    import torch
    return {k: torch.from_numpy(v.copy()).cuda() for k, v in arrs.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("aero", [False, True])
@pytest.mark.parametrize("case", ["odd", "ni1", "mpas", "k0", "no_options"])
def test_device_entry_on_a_torch_stream(case, aero, gpu_mixed):
    """The device entry on CUDA tensors, enqueued on a non-default stream: the bits of the host tile entry, the halo untouched,
    and kidmp_diag afterwards sees the step."""
    import torch
    if aero and not CASES[case].get("full", True):
        pytest.skip("covered without aerosols")
    pt = Patch(aero=aero, seed=5, **CASES[case])
    dev = _to_dev(pt.mem)
    gpu_mixed.diag()
    pt.run_tile(gpu_mixed)
    d_host = gpu_mixed.diag()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    f3, pii, p, dz, acc, radii, ae = pt.args(dev)
    with torch.cuda.stream(s):
        gpu_mixed.mp_gt_driver_device(20.0, f3, pii, p, dz, acc, tile=pt.tile, radii=radii, aerosols=ae, stream=s)
    d_dev = gpu_mixed.diag()                      # ordered after the step on `s` by the handle's event
    s.synchronize()
    got = {k: v.cpu().numpy() for k, v in dev.items()}
    want = {k: pt.mem[k][pt.s3 if pt.mem[k].ndim == 3 else pt.s2] for k in pt.mem if k in pt.packed or k in RE3 and pt.full}
    pt.check(got, want)
    assert d_dev[7] == d_host[7] == pt.tile[1] * pt.tile[5] and d_dev[6] == d_host[6] > 0
    np.testing.assert_allclose(d_dev, d_host, rtol=1e-12, atol=0)


@pytest.mark.gpu
def test_device_entry_twice_on_two_streams_and_the_whole_box(gpu_mixed):
    """Two device calls on two streams reuse the handle's planes in order; a whole-box device call equals the packed entry."""
    import torch
    pt = Patch(ni=64, nk=30, nj=4, hi=(0, 0), hj=(0, 0), spare=0)
    want = pt.run_packed(gpu_mixed)
    dev = _to_dev(pt.mem)
    f3, pii, p, dz, acc, radii, _ = pt.args(dev)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    gpu_mixed.mp_gt_driver_device(20.0, f3, pii, p, dz, acc, radii=radii, stream=s1)
    s1.synchronize()
    got = {k: v.cpu().numpy() for k, v in dev.items()}
    pt.check(got, want)
    # a second step of the same arrays on another stream, against the packed entry's second step
    gpu_mixed.mp_gt_driver_device(20.0, f3, pii, p, dz, acc, radii=radii, stream=s2)
    f3p, piip, pp, dzp, accp, _, _ = pt.args(pt.packed)
    re2 = gpu_mixed.mp_gt_driver(20.0, f3p, piip, pp, dzp, accp)
    s2.synchronize()
    for k in F3 + ACC:
        assert np.array_equal(dev[k].cpu().numpy().view(np.uint32), pt.packed[k].view(np.uint32)), k
    for k in RE3:
        assert np.array_equal(dev[k].cpu().numpy().view(np.uint32), re2[k].view(np.uint32)), k


@pytest.mark.gpu
def test_openmp_style_tiles_on_two_handles_at_once(gpu_mixed):
    """Two handles in two threads step two adjacent tiles of one shared patch at the same time: the union is one call over the
    combined tile, and nothing outside both tiles changes."""
    from kid_b200.kidmp import Thompson
    pt = Patch(ni=96, nk=40, nj=8, hi=(4, 4), hj=(3, 3), seed=21)
    whole = {k: v.copy() for k, v in pt.mem.items()}
    f3, pii, p, dz, acc, radii, _ = pt.args(whole)
    gpu_mixed.mp_gt_driver(20.0, f3, pii, p, dz, acc, radii=radii, tile=pt.tile)
    i0, ni, k0, nk, j0, nj = pt.tile
    tiles = [(i0, 40, k0, nk, j0, nj), (i0 + 40, ni - 40, k0, nk, j0, nj)]
    handles = [Thompson(set_Nc=100.0, iiwarm=False, l_sediment=True) for _ in tiles]
    errors = []
    barrier = threading.Barrier(len(tiles))

    def run(h, t):
        try:
            f3, pii, p, dz, acc, radii, _ = pt.args()
            barrier.wait()
            h.mp_gt_driver(20.0, f3, pii, p, dz, acc, radii=radii, tile=t)
        except Exception as e:                   # (reported below: an assertion in a thread would be lost)
            errors.append(e)
    threads = [threading.Thread(target=run, args=(h, t)) for h, t in zip(handles, tiles)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    for h in handles:
        h.close()
    assert not errors, errors
    for k in pt.mem:
        assert np.array_equal(pt.mem[k].view(np.uint32), whole[k].view(np.uint32)), k
    pt.check(pt.mem, {k: (whole[k][pt.s3] if whole[k].ndim == 3 else whole[k][pt.s2]) for k in whole})


def _raw_call(gpu, pt, tile, arrs=None, device=False, drop=None, ae=False):
    """The C entry called directly (rc, message), so that a field can be NULL."""
    f3, pii, p, dz, acc, radii, aed = pt.args(arrs)
    if device:
        addr = lambda a: C.cast(C.c_void_p(int(a.data_ptr())), C.POINTER(C.c_float))
    else:
        addr = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
    w, aes, _, keep = gpu._wrf_structs(f3, pii, p, dz, acc, radii, aed if ae else None, pt.mem_shape, addr)
    if drop:
        setattr(w, drop, None)
    from kid_b200.kidmp import WrfTile
    t = WrfTile(*tile)
    L = gpu._L
    if device:
        rc = L.kidmp_mp_gt_driver_tile_device(gpu.h, C.byref(w), C.byref(t), C.byref(aes) if aes is not None else None,
                                              20.0, None)
    else:
        rc = L.kidmp_mp_gt_driver_tile(gpu.h, C.byref(w), C.byref(t), C.byref(aes) if aes is not None else None, 20.0)
    return rc, L.kidmp_last_error(gpu.h).decode()


BAD_TILES = {
    "i_below": ((-1, 10, 0, 20, 0, 3), "inside the memory box"),
    "i_beyond": ((5, 20, 0, 20, 0, 3), "inside the memory box"),
    "k_beyond": ((0, 10, 1, 21, 0, 3), "inside the memory box"),
    "j_below": ((0, 10, 0, 20, -1, 3), "inside the memory box"),
    "j_beyond": ((0, 10, 0, 20, 2, 4), "inside the memory box"),
    "nk1": ((0, 10, 0, 1, 0, 3), "tile extents"),
    "ni0": ((0, 0, 0, 20, 0, 3), "tile extents"),
    "nj0": ((0, 10, 0, 20, 0, 0), "tile extents"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("device", [False, True])
def test_rejections_leave_every_array_as_it_was(device, gpu_mixed):
    """A tile outside the memory box on each axis, nk < 2, an empty extent, a null field: an error with a message, and every
    array bit-identical to before (the check comes before any copy or launch)."""
    import torch
    pt = Patch(ni=18, nk=20, nj=3, hi=(2, 4), hj=(1, 1), spare=1, aero=True)   # memory 24 x 21 x 5
    assert pt.mem_shape == (5, 21, 24)
    arrs = _to_dev(pt.mem) if device else pt.mem
    cases = [(t, msg, None) for t, msg in BAD_TILES.values()] + [(pt.tile, "null field 1", "qc"), (pt.tile, "null array", "pii")]
    for ae in (False, True):
        for tile, msg, drop in cases:
            rc, err = _raw_call(gpu_mixed, pt, tile, arrs, device=device, drop=drop, ae=ae)
            assert rc != 0 and msg in err, (tile, drop, ae, err)
    if device:
        torch.cuda.synchronize()
        arrs = {k: v.cpu().numpy() for k, v in arrs.items()}
    for k, a in arrs.items():
        assert np.array_equal(a.view(np.uint32), pt.before[k].view(np.uint32)), k
    # and the handle still works: the valid tile steps
    rc, err = _raw_call(gpu_mixed, pt, pt.tile)
    assert rc == 0, err


@pytest.mark.gpu
def test_multi_device_handle(gpu_mixed):
    """A handle over two GPUs steps a host tile on its first device (the same bits); its device entry is an error that touches
    nothing."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from kid_b200.kidmp import Thompson, KidmpError
    m = Thompson(set_Nc=100.0, iiwarm=False, l_sediment=True, devices=[0, 1])
    try:
        pt = Patch(**CASES["odd"])
        ref = Patch(**CASES["odd"])
        ref.run_tile(gpu_mixed)
        pt.run_tile(m)
        for k in pt.mem:
            assert np.array_equal(pt.mem[k].view(np.uint32), ref.mem[k].view(np.uint32)), k
        pd = Patch(**CASES["odd"])
        dev = _to_dev(pd.mem)
        f3, pii, p, dz, acc, radii, _ = pd.args(dev)
        with pytest.raises(KidmpError, match="single-device"):
            m.mp_gt_driver_device(20.0, f3, pii, p, dz, acc, tile=pd.tile, radii=radii)
        torch.cuda.synchronize()
        for k, v in dev.items():
            assert np.array_equal(v.cpu().numpy().view(np.uint32), pd.before[k].view(np.uint32)), k
    finally:
        m.close()
