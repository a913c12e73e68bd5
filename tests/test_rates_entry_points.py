"""The 36 save_dg process rates (M:2963-3120) through every entry point that steps, bit for bit against the device path.

KiD keeps these rates every time step: the Fortran shim and the C++ host twin turn them on with kidmp_enable_rates and read
them with kidmp_get_rates after kidmp_kid_interface.  The reference here is kidmp_step_device with a caller buffer filled with
NaN (regimes.Device), which tests/test_regimes.py pins to the oracle cell by cell; each domain is re-checked against the oracle
once below, so this file stands on its own.  Every other path must give the reference's bits after mapping the layout:
columns a step does not touch stay NaN in a caller buffer and are exactly 0 in the handle's own buffer (cleared every step).

Domains: D1 the regime domain (806 columns, 32 levels, dt = 20 s; every cell-kernel class), D2 the sediment case (24 columns,
dt = 120 s, hundreds of sub-steps), D3 3000 bench-like columns at dt = 60 s (k_substeps runs), D4 the columns of D1 repeated
to 3*1024 + 77 (two chunks or more of a host pipeline of 1024 columns).

Stale rates: kidmp_get_rates returns the rates of the handle's last step or fails; it never returns those of an earlier step,
of another domain, or memory no step wrote.  Every rate read here goes into a buffer with a NaN guard region after it, so a
copy of the wrong size shows as a failure, not as a write past the caller's array."""
import ctypes as C

import numpy as np
import pytest

import regimes as R

FIELDS = R.FIELDS
NR = 36
GUARD = NR * 7001 * 60               # floats after every rate buffer: the largest state any test here leaves on a handle
NAN_BITS = np.uint32(0x7FC00000)


# ---- helpers ------------------------------------------------------------------------------------------------------------
def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_bits(got, want, what):
    g, w = bits(got), bits(want)
    assert g.shape == w.shape, (what, g.shape, w.shape)
    if not np.array_equal(g, w):
        bad = np.argwhere(g != w)
        raise AssertionError("%s: %d of %d rates differ, first at %s: got %r want %r" % (
            what, len(bad), g.size, tuple(bad[0]), got[tuple(bad[0])], want[tuple(bad[0])]))


def active_columns(rates):
    """Columns of a NaN-filled caller buffer that the step wrote: every level of every rate, or none."""
    act = np.isfinite(rates).all(axis=(0, 1))
    assert np.isnan(rates[:, :, ~act]).all(), "a column partly written"
    return act


def own(rates):
    """The handle's own buffer for the step a caller buffer saw: 0 where the step wrote nothing."""
    out = rates.copy()
    out[:, :, ~active_columns(rates)] = 0.0
    return out


def read_rates(th, ncol, nz, layout="k_fastest"):
    """kidmp_get_rates into a buffer of (36, ncol, nz) ('k_fastest') or (36, nz, ncol) with GUARD NaN floats after it.
    Raises KidmpError when the call fails; fails the test when it wrote into the guard."""
    from kid_b200 import kidmp
    lay = kidmp.K_FASTEST if layout == "k_fastest" else kidmp.COL_FASTEST
    n = NR * ncol * nz
    buf = np.full(n + GUARD, np.nan, np.float32)
    rc = th._L.kidmp_get_rates(th.h, lay, buf.ctypes.data_as(kidmp._fp))
    spill = int((buf[n:].view(np.uint32) != NAN_BITS).sum())
    assert spill == 0, "kidmp_get_rates wrote %d floats past the %d of a (%d, %d) domain" % (spill, n, ncol, nz)
    if rc:
        raise kidmp.KidmpError(th._L.kidmp_last_error(th.h).decode())
    return buf[:n].reshape((NR, ncol, nz) if lay == kidmp.K_FASTEST else (NR, nz, ncol)).copy()


def check_own(th, want, what):
    """Both layouts of the handle's own buffer against a reference caller buffer want (36, nz, ncol)."""
    _, nz, ncol = want.shape
    w = own(want)
    assert_bits(read_rates(th, ncol, nz, "col_fastest"), w, what + " col_fastest")
    assert_bits(read_rates(th, ncol, nz, "k_fastest"), np.ascontiguousarray(w.transpose(0, 2, 1)), what + " k_fastest")


def ref_run(th, st, p, dz, dt):
    """The reference: kidmp_step_device with a NaN-filled caller buffer.  (state, ppt, rates (36, nz, ncol), step_stats)."""
    state, ppt, rates, _, stats = R.Device(st, p, dz, dt).run(th)
    return state, ppt, rates, stats


def host_arrays(st, layout, pinned=False):
    """Copies of the (nz, ncol) arrays in `layout`, pinned (page-locked through torch) or pageable; '_keep' holds the tensors."""
    import torch
    out, keep = {}, []
    for k, v in st.items():
        a = np.ascontiguousarray(v if layout == "col_fastest" else v.T)
        if pinned:
            t = torch.from_numpy(a.copy()).pin_memory()
            keep.append(t)
            out[k] = t.numpy()
        else:
            out[k] = a.copy()
    out["_keep"] = keep
    return out


def assert_state(arrs, want, layout, what):
    for k in FIELDS:
        a = arrs[k] if layout == "col_fastest" else arrs[k].T
        assert np.array_equal(bits(a), bits(want[k])), (what, k)


def columns(st, idx):
    return {k: np.ascontiguousarray(v[:, idx]) for k, v in st.items()}


class _DevArray:
    """A float32 device array at a raw address, for torch.as_tensor (the CUDA array interface)."""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"data": (int(ptr), False), "shape": tuple(shape), "typestr": "<f4", "version": 2,
                                         "strides": None}


def resident_p(th, nz, ncol):
    """The resident pressure plane [nz][ncol] of a single-device handle (kidmp_device_state)."""
    import torch
    th.sync()
    _, p_ptr, _, _ = th.device_state()
    return torch.as_tensor(_DevArray(p_ptr, (nz, ncol)), device="cuda").cpu().numpy().copy()


# ---- fixtures -----------------------------------------------------------------------------------------------------------
def _new(**kw):
    from kid_b200.kidmp import Thompson
    cfg = dict(set_Nc=100.0, iiwarm=False, l_sediment=True)
    cfg.update(kw)
    return Thompson(**cfg)


@pytest.fixture(scope="module")
def refh():
    """Reference handles: mixed phase (set_Nc 100) and warm rain (set_Nc 50), with sedimentation."""
    hs = {"mixed": _new(), "warm": _new(set_Nc=50.0, iiwarm=True)}
    yield hs
    for h in hs.values():
        h.close()


def _d4():
    st, p, dz, dt = R.regime_domain()
    idx = np.arange(3 * 1024 + 77) % st["t"].shape[1]
    return columns(st, idx), np.ascontiguousarray(p[:, idx]), dz, dt


def _build(name):
    if name == "D1":
        return R.regime_domain()
    if name == "D2":
        return R.build("sediment")
    if name == "D3":
        st, p, dz = R.bench_like(3000, 100.0)
        return st, p, dz, 60.0
    return _d4()


@pytest.fixture(scope="module")
def dom(refh):
    """Domain name -> dict st p dz dt, and the mixed handle's reference state, ppt, rates and step_stats."""
    cache = {}

    def get(name):
        if name not in cache:
            st, p, dz, dt = _build(name)
            state, ppt, rates, stats = ref_run(refh["mixed"], st, p, dz, dt)
            cache[name] = dict(st=st, p=p, dz=dz, dt=dt, state=state, ppt=ppt, rates=rates, stats=stats,
                               nz=st["t"].shape[0], ncol=st["t"].shape[1])
        return cache[name]
    return get


def oracle_rates(o, st, p, dz, dt, cols):
    """The oracle's rates (36, nz, len(cols)) of the given columns, f64."""
    nz = st["t"].shape[0]
    out = np.zeros((NR, nz, len(cols)), np.float64)
    for n, j in enumerate(cols):
        out[:, :, n] = o.column(dt, *[st[k][:, j] for k in FIELDS], p[:, j], dz, want_rates=True)["rates"]
    return out


def assert_oracle(o, st, p, dz, dt, got, what):
    """Device rates got (36, nz, ncol; NaN or 0 in untouched columns) against the oracle at RATE_TOL, no outlier; the oracle
    has no process in the columns the device left untouched."""
    ncol = st["t"].shape[1]
    ref = oracle_rates(o, st, p, dz, dt, range(ncol))
    act = np.isfinite(got).all(axis=(0, 1)) & (got != 0).any(axis=(0, 1))
    assert act.any(), what
    assert not ref[:, :, ~act].any(), "%s: the oracle has processes in %d columns the device left untouched" % (
        what, int(ref[:, :, ~act].any(axis=(0, 1)).sum()))
    cls = np.full(st["t"].shape, "", dtype=object)
    bad = R.rate_outliers(got[:, :, act], ref[:, :, act], o.rate_names, cls[:, act])
    assert not bad, "%s: %d rate outliers against the oracle:\n  %s" % (what, len(bad), "\n  ".join(bad[:20]))


# ---- the reference, anchored -------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["D1", "D2"])
def test_reference_matches_the_oracle(name, dom, oracle_mixed):
    d = dom(name)
    assert_oracle(oracle_mixed, d["st"], d["p"], d["dz"], d["dt"], d["rates"], name)


@pytest.mark.gpu
def test_domains_reach_every_kernel_that_writes_rates(dom):
    s1, s2, s3 = dom("D1")["stats"], dom("D2")["stats"], dom("D3")["stats"]
    assert min(s1["cells_warm"], s1["cells_ice"], s1["cells_mixed_no_rain"], s1["cells_full"]) > 0, s1
    assert s2["substep_columns"] > 0 and s3["substep_columns"] > 0, (s2, s3)
    r3 = dom("D3")["rates"]
    assert (~active_columns(r3)).any() and active_columns(r3).any()        # clear-sky and cloudy columns


# ---- kidmp_step ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [False, True], ids=["pageable", "pinned"])
@pytest.mark.parametrize("layout", ["col_fastest", "k_fastest"])
@pytest.mark.parametrize("name", ["D1", "D3"])
def test_host_step(name, layout, pinned, dom):
    d = dom(name)
    th = _new()
    try:
        th.enable_rates(True)
        arrs = host_arrays(d["st"], layout, pinned)
        pl = np.ascontiguousarray(d["p"] if layout == "col_fastest" else d["p"].T)
        th.step(d["dt"], arrs, pl, d["dz"], layout=layout)
        assert_state(arrs, d["state"], layout, name)
        check_own(th, d["rates"], "%s %s" % (name, layout))
    finally:
        th.close()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["pageable", "pinned", "chunk512"])
def test_host_step_of_pipeline_size(variant, dom, monkeypatch):
    """A column-fastest domain of at least two host-pipeline chunks: with rates kept it goes through the resident state."""
    d = dom("D4")
    monkeypatch.setenv("KIDMP_PIPE_CHUNK", "1024")
    th = _new()
    try:
        if variant == "chunk512":
            th.set_option("chunk", 512)
        th.enable_rates(True)
        for rep in range(2):
            arrs = host_arrays(d["st"], "col_fastest", variant == "pinned")
            th.step(d["dt"], arrs, d["p"], d["dz"])
            assert_state(arrs, d["state"], "col_fastest", "D4 %s" % variant)
            check_own(th, d["rates"], "D4 %s run %d" % (variant, rep))
    finally:
        th.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["D1", "D4"], ids=["resident", "pipeline"])
def test_step_nc_with_the_handles_own_value(name, dom, monkeypatch):
    d = dom(name)
    monkeypatch.setenv("KIDMP_PIPE_CHUNK", "1024")
    th = _new()
    try:
        th.enable_rates(True)
        arrs = host_arrays(d["st"], "col_fastest")
        th.step(d["dt"], arrs, d["p"], d["dz"], set_nc=np.full(d["ncol"], 100.0, np.float32))
        assert_state(arrs, d["state"], "col_fastest", name)
        check_own(th, d["rates"], "step_nc " + name)
    finally:
        th.close()


# ---- the resident state -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_three_resident_steps(dom, refh):
    """state_alloc / upload / step_resident x 3 on D3: after each step that step's rates (the reference steps the state
    downloaded before it)."""
    d = dom("D3")
    th = _new()
    try:
        th.enable_rates(True)
        th.state_alloc(d["ncol"], d["nz"])
        th.upload(d["st"], d["p"], d["dz"])
        for i in range(3):
            cur = {k: np.zeros((d["nz"], d["ncol"]), np.float32) for k in FIELDS}
            th.download(cur, want_ppt=False)
            th.step_resident(d["dt"])
            _, _, want, _ = ref_run(refh["mixed"], cur, d["p"], d["dz"], d["dt"])
            check_own(th, want, "resident step %d" % i)
    finally:
        th.close()


@pytest.mark.gpu
def test_column(dom):
    """kidmp_column: a cloudy column of D1 gives its rates in D1's reference; a clear-sky column of D3 gives all zeros."""
    d1, d3 = dom("D1"), dom("D3")
    j1 = int(np.flatnonzero(active_columns(d1["rates"]))[0])
    j3 = int(np.flatnonzero(~active_columns(d3["rates"]))[0])
    th = _new()
    try:
        th.enable_rates(True)
        for d, j, what in ((d1, j1, "cloudy"), (d3, j3, "clear")):
            out = th.column(d["dt"], *[d["st"][k][:, j] for k in FIELDS], d["p"][:, j], d["dz"])
            for k in FIELDS:
                assert np.array_equal(bits(out[k]), bits(d["state"][k][:, j])), (what, k)
            got = read_rates(th, 1, d["nz"], "k_fastest")[:, 0, :]
            assert_bits(got, own(d["rates"])[:, :, j], "column " + what)
            if what == "clear":
                assert not got.any()
    finally:
        th.close()


# ---- kidmp_kid_interface ------------------------------------------------------------------------------------------------
KID_CASES = [("mixed", 1, 60), ("mixed", 77, 60), ("mixed", 120, 120), ("warm", 1, 60), ("warm", 77, 60), ("warm", 120, 120)]
DT_KID = 5.0


def kid_inputs(nx, nz):
    from test_gpu_parity import _kid_case
    return _kid_case(nx, nz)


def kid_state(kid, dt, warm):
    """The state kidmp_kid_interface steps (kidmp_kid.cuh, I:60-95) in f32, as (nz, nx) arrays: state + (advective +
    divergence tendency) * dt, T = theta * exner.  Ice moments are zero on a warm handle."""
    dt = np.float32(dt)
    new = lambda x, a, b: (x + (a + b) * dt).astype(np.float32)
    st = {"t": (new(kid["theta"], kid["dtheta_adv"], kid["dtheta_div"]) * kid["exner"]).astype(np.float32),
          "qv": new(kid["qv"], kid["dqv_adv"], kid["dqv_div"])}
    for m in ("qc", "qr", "nr", "qi", "ni", "qs", "qg"):
        ice = m in ("qi", "ni", "qs", "qg")
        st[m] = np.zeros_like(kid["qv"]) if ice and warm else new(kid[m], kid["d%s_adv" % m], kid["d%s_div" % m])
    return {k: np.ascontiguousarray(v.T) for k, v in st.items()}


def kid_reference(th, refh, kid, handle, p0, roc):
    """Step kid on th (enable_rates already set as the test wants) and return (output, the reference (state in, p, rates))."""
    nx, nz = kid["theta"].shape
    out = th.kid_interface(kid, DT_KID, p0, roc)
    st = kid_state(kid, DT_KID, handle == "warm")
    p = resident_p(th, nz, nx)
    _, _, rates, _ = ref_run(refh[handle], st, p, kid["dz"], DT_KID)
    return out, st, p, rates


@pytest.mark.gpu
@pytest.mark.parametrize("handle,nx,nz", KID_CASES)
def test_kid_interface(handle, nx, nz, refh, oracle_mixed, oracle_warm):
    """The path KiD's shim and the C++ twin use: get_rates(k_fastest) after kidmp_kid_interface, and a caller buffer."""
    import torch
    kid, p0, roc = kid_inputs(nx, nz)
    warm = handle == "warm"
    th = _new(set_Nc=50.0, iiwarm=True) if warm else _new()
    try:
        th.enable_rates(True)
        _, st, p, want = kid_reference(th, refh, kid, handle, p0, roc)
        assert_bits(read_rates(th, nx, nz, "k_fastest"), np.ascontiguousarray(own(want).transpose(0, 2, 1)), "kid k_fastest")
        o = oracle_warm if warm else oracle_mixed
        assert_oracle(o, st, p, kid["dz"], DT_KID, want, "kid %s %dx%d" % (handle, nx, nz))
        th.enable_rates(False)
        buf = torch.full((NR, nz, nx), float("nan"), dtype=torch.float32, device="cuda")
        th.set_rates_buffer(buf.data_ptr())
        try:
            th.kid_interface(kid, DT_KID, p0, roc)
            th.sync()
        finally:
            th.set_rates_buffer(0)
        assert_bits(buf.cpu().numpy(), want, "kid caller buffer")
    finally:
        th.close()


# ---- the WRF tile entries -----------------------------------------------------------------------------------------------
WRF_CASES = ["odd", "ni1", "mpas", "k0"]


def wrf_patch(case):
    """A Patch of tests/test_wrf_tiles.py with one dz profile in every column (the reference step takes dz per level), and the
    state the tile steps as (nk, ni*nj) planes: T = th * pii in f32 (kidmp_wrf.cuh)."""
    from test_wrf_tiles import CASES, Patch
    pt = Patch(**CASES[case])
    prof = pt.packed["dz"][0, :, 0].copy()
    pt.packed["dz"][:] = prof[None, :, None]
    pt.mem["dz"][pt.s3] = pt.packed["dz"]
    pt.before["dz"] = pt.mem["dz"].copy()
    nj, nk, ni = pt.packed["qv"].shape
    planes = lambda a: np.ascontiguousarray(a.transpose(1, 0, 2).reshape(nk, nj * ni))
    st = {k: planes(pt.packed[w]) for k, w in zip(FIELDS[:8], ("qv", "qc", "qi", "qr", "qs", "qg", "ni", "nr"))}
    st["t"] = planes((pt.packed["th"] * pt.packed["pii"]).astype(np.float32))
    return pt, st, planes(pt.packed["p"]), prof


@pytest.mark.gpu
@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("case", WRF_CASES)
def test_wrf_tile(case, device, refh):
    """kidmp_mp_gt_driver_tile (own buffer) and kidmp_mp_gt_driver_tile_device (caller buffer [36][nk][ni*nj], column i + ni*j)."""
    import torch
    pt, st, p, dz = wrf_patch(case)
    nk, ncol = st["t"].shape
    _, _, want, _ = ref_run(refh["mixed"], st, p, dz, 20.0)
    assert active_columns(want).any()
    th = _new()
    try:
        if not device:
            th.enable_rates(True)
            f3, pii, pp, dzz, acc, radii, _ = pt.args()
            th.mp_gt_driver(20.0, f3, pii, pp, dzz, acc, radii=radii, tile=pt.tile)
            check_own(th, want, "wrf host " + case)
        else:
            dev = {k: torch.from_numpy(v.copy()).cuda() for k, v in pt.mem.items()}
            buf = torch.full((NR, nk, ncol), float("nan"), dtype=torch.float32, device="cuda")
            f3, pii, pp, dzz, acc, radii, _ = pt.args(dev)
            th.set_rates_buffer(buf.data_ptr())
            try:
                th.mp_gt_driver_device(20.0, f3, pii, pp, dzz, acc, tile=pt.tile, radii=radii)
                th.sync()
            finally:
                th.set_rates_buffer(0)
            assert_bits(buf.cpu().numpy(), want, "wrf device " + case)
    finally:
        th.close()


# ---- captured graphs ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("graphs", [1, 0])
def test_graph_replays_with_changed_buffers(graphs, dom, refh):
    """A slice of D1 stepped on the same device arrays: caller buffer X, then Y, then X again (the third step leaves Y as the
    second left it); then resident steps with the own buffer on, off and on again.  Every result has the reference's bits."""
    import torch
    d = dom("D1")
    idx = np.arange(0, d["ncol"], 7)
    st, p = columns(d["st"], idx), np.ascontiguousarray(d["p"][:, idx])
    _, _, want, _ = ref_run(refh["mixed"], st, p, d["dz"], d["dt"])
    assert active_columns(want).any()
    nz, ncol = st["t"].shape
    th = _new()
    try:
        th.set_option("graphs", graphs)
        dv = R.Device(st, p, d["dz"], d["dt"], rates=False)
        bx, by = (torch.empty((NR, nz, ncol), dtype=torch.float32, device="cuda") for _ in range(2))

        def step_into(buf):
            for k in FIELDS:
                dv.dev[k].copy_(dv.src[k])
            buf.fill_(float("nan"))
            torch.cuda.synchronize()
            th.set_rates_buffer(buf.data_ptr())
            try:
                th.step_device(ncol, nz, d["dt"], [dv.dev[k].data_ptr() for k in FIELDS], dv.p.data_ptr(), dv.dz.data_ptr(),
                               dv.ppt.data_ptr())
                th.sync()
            finally:
                th.set_rates_buffer(0)
            return buf.cpu().numpy()
        for n in range(2):
            assert_bits(step_into(bx), want, "X %d" % n)
            y = step_into(by)
            assert_bits(y, want, "Y %d" % n)
            assert_bits(step_into(bx), want, "X again %d" % n)
            assert_bits(by.cpu().numpy(), y, "Y after the step into X %d" % n)
        th.state_alloc(ncol, nz)
        for n, on in enumerate((True, False, True, True)):
            th.enable_rates(on)
            th.upload(st, p, d["dz"])
            th.step_resident(d["dt"])
            if on:
                check_own(th, want, "resident %d" % n)
            else:
                with pytest.raises(Exception):
                    read_rates(th, ncol, nz)
    finally:
        th.close()


# ---- stale rates and refusals -------------------------------------------------------------------------------------------
STALE_ENTRIES = ["step", "step_k_fastest", "step_pipeline", "step_nc", "resident", "column", "kid_interface", "wrf_host",
                 "wrf_device", "step_device"]


@pytest.mark.gpu
@pytest.mark.parametrize("entry", STALE_ENTRIES)
def test_no_stale_rates_after_another_domain(entry, dom, refh, monkeypatch):
    """enable_rates, a resident step of D1, then another domain through `entry`: get_rates returns that domain's rates or
    fails, never D1's (nor anything of D1's size)."""
    import torch
    from kid_b200.kidmp import KidmpError
    monkeypatch.setenv("KIDMP_PIPE_CHUNK", "1024")
    a = dom("D1")
    th = _new()
    try:
        th.enable_rates(True)
        th.step(a["dt"], host_arrays(a["st"], "col_fastest"), a["p"], a["dz"])
        check_own(th, a["rates"], "domain A")
        want = None                                       # (36, nz, ncol) of B, None: B writes no rates
        if entry in ("step", "step_k_fastest", "step_nc", "resident", "step_device"):
            b = dom("D3")
            want, nz, ncol = b["rates"], b["nz"], b["ncol"]
            if entry == "step":
                th.step(b["dt"], host_arrays(b["st"], "col_fastest"), b["p"], b["dz"])
            elif entry == "step_k_fastest":
                th.step(b["dt"], host_arrays(b["st"], "k_fastest"), np.ascontiguousarray(b["p"].T), b["dz"], layout="k_fastest")
            elif entry == "step_nc":
                th.step(b["dt"], host_arrays(b["st"], "col_fastest"), b["p"], b["dz"], set_nc=np.full(ncol, 100.0, np.float32))
            elif entry == "resident":
                th.state_alloc(ncol, nz)
                th.upload(b["st"], b["p"], b["dz"])
                th.step_resident(b["dt"])
            else:
                dv = R.Device(b["st"], b["p"], b["dz"], b["dt"], rates=False)
                th.step_device(ncol, nz, b["dt"], [dv.dev[k].data_ptr() for k in FIELDS], dv.p.data_ptr(), dv.dz.data_ptr(),
                               dv.ppt.data_ptr())
                th.sync()
                want = None
        elif entry == "step_pipeline":
            b = dom("D4")
            want, nz, ncol = b["rates"], b["nz"], b["ncol"]
            th.step(b["dt"], host_arrays(b["st"], "col_fastest"), b["p"], b["dz"])
        elif entry == "column":
            b = dom("D3")
            j = int(np.flatnonzero(active_columns(b["rates"]))[0])
            want, nz, ncol = b["rates"][:, :, j:j + 1], b["nz"], 1
            th.column(b["dt"], *[b["st"][k][:, j] for k in FIELDS], b["p"][:, j], b["dz"])
        elif entry == "kid_interface":
            kid, p0, roc = kid_inputs(77, 60)
            _, _, _, want = kid_reference(th, refh, kid, "mixed", p0, roc)
            nz, ncol = 60, 77
        else:
            pt, st, p, dz = wrf_patch("odd")
            nz, ncol = st["t"].shape
            _, _, want, _ = ref_run(refh["mixed"], st, p, dz, 20.0)
            if entry == "wrf_host":
                f3, pii, pp, dzz, acc, radii, _ = pt.args()
                th.mp_gt_driver(20.0, f3, pii, pp, dzz, acc, radii=radii, tile=pt.tile)
            else:
                dev = {k: torch.from_numpy(v.copy()).cuda() for k, v in pt.mem.items()}
                f3, pii, pp, dzz, acc, radii, _ = pt.args(dev)
                th.mp_gt_driver_device(20.0, f3, pii, pp, dzz, acc, tile=pt.tile, radii=radii)
                th.sync()
        if want is None:
            for shape in ((ncol, nz), (a["ncol"], a["nz"])):
                with pytest.raises(KidmpError):
                    read_rates(th, *shape)
        else:
            check_own(th, want, entry)
    finally:
        th.close()


@pytest.mark.gpu
def test_rates_before_the_first_step_are_refused(dom):
    """enable_rates on a handle that already holds a resident state: nothing has written the new buffer yet."""
    from kid_b200.kidmp import KidmpError
    d = dom("D1")
    th = _new()
    try:
        th.state_alloc(d["ncol"], d["nz"])
        th.upload(d["st"], d["p"], d["dz"])
        th.enable_rates(True)
        with pytest.raises(KidmpError):
            read_rates(th, d["ncol"], d["nz"])
        th.step_resident(d["dt"])
        check_own(th, d["rates"], "after the step")
        th.enable_rates(True)                               # (again: the buffer stays, its rates are not this call's)
        with pytest.raises(KidmpError):
            read_rates(th, d["ncol"], d["nz"])
        th.state_alloc(d["ncol"] - 1, d["nz"])
        with pytest.raises(KidmpError):
            read_rates(th, d["ncol"] - 1, d["nz"])
    finally:
        th.close()


AERO_ENTRIES = ["step_device_aero", "mp_gt_driver_aero", "tile_host_aero", "tile_device_aero"]


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["caller_buffer", "enable_rates"])
@pytest.mark.parametrize("entry", AERO_ENTRIES)
def test_aerosol_aware_steps_refuse_rates(entry, how, dom):
    """The aerosol-aware step has no process rates: with a caller buffer set or the own buffer on, every aerosol-aware entry
    fails before it copies or launches anything.  Inputs and the rates buffer keep their bits; the handle then steps as before."""
    import torch
    from kid_b200.kidmp import KidmpError
    from test_wrf_tiles import CASES, Patch
    d = dom("D1")
    th = _new()
    try:
        buf = None
        if how == "caller_buffer":
            buf = torch.full((NR, d["nz"], d["ncol"]), float("nan"), dtype=torch.float32, device="cuda")
            th.set_rates_buffer(buf.data_ptr())
        else:
            th.enable_rates(True)
            th.step(d["dt"], host_arrays(d["st"], "col_fastest"), d["p"], d["dz"])
            check_own(th, d["rates"], "before")
        if entry == "step_device_aero":
            nc, nwfa, nifa, w = R.aero_inputs(d["st"], d["p"])
            host = dict({k: d["st"][k] for k in FIELDS}, nc=nc, nwfa=nwfa, nifa=nifa, w=w, p=d["p"])
            dev = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in host.items()}
            ddz = torch.from_numpy(d["dz"]).cuda()
            ppt = torch.full((4, d["ncol"]), 7.0, dtype=torch.float32, device="cuda")
            torch.cuda.synchronize()
            with pytest.raises(KidmpError, match="process-rate"):
                th.step_device_aero(d["ncol"], d["nz"], d["dt"], [dev[k].data_ptr() for k in FIELDS], dev["nc"].data_ptr(),
                                    dev["nwfa"].data_ptr(), dev["nifa"].data_ptr(), dev["p"].data_ptr(), dev["w"].data_ptr(),
                                    ddz.data_ptr(), ppt.data_ptr())
            torch.cuda.synchronize()
            for k, v in host.items():
                assert np.array_equal(bits(dev[k].cpu().numpy()), bits(v)), k
            assert (ppt == 7.0).all()
        else:
            pt = Patch(aero=True, seed=11, **CASES["odd"])
            if entry == "mp_gt_driver_aero":
                pt = Patch(ni=50, nk=30, nj=6, hi=(0, 0), hj=(0, 0), spare=0, aero=True)
            f3, pii, p, dz, acc, radii, ae = pt.args()
            if entry == "tile_device_aero":
                dev = {k: torch.from_numpy(v.copy()).cuda() for k, v in pt.mem.items()}
                f3, pii, p, dz, acc, radii, ae = pt.args(dev)
                with pytest.raises(KidmpError, match="process-rate"):
                    th.mp_gt_driver_device(20.0, f3, pii, p, dz, acc, tile=pt.tile, radii=radii, aerosols=ae)
                torch.cuda.synchronize()
                got = {k: v.cpu().numpy() for k, v in dev.items()}
            else:
                with pytest.raises(KidmpError, match="process-rate"):
                    th.mp_gt_driver(20.0, f3, pii, p, dz, acc, radii=radii, aerosols=ae,
                                    tile=pt.tile if entry == "tile_host_aero" else None)
                got = pt.mem
            for k, v in got.items():
                assert np.array_equal(bits(v), bits(pt.before[k])), k
        if buf is not None:
            assert (bits(buf.cpu().numpy()) == NAN_BITS).all()
            th.set_rates_buffer(0)
        else:
            check_own(th, d["rates"], "after the refused call")
        arrs = host_arrays(d["st"], "col_fastest")
        th.step(d["dt"], arrs, d["p"], d["dz"])
        assert_state(arrs, d["state"], "col_fastest", "plain step after the refusal")
        if buf is None:
            check_own(th, d["rates"], "plain step after the refusal")
    finally:
        th.close()


# ---- multi-device handles -----------------------------------------------------------------------------------------------
def _device_sets():
    try:
        import torch
        n = torch.cuda.device_count()
    except Exception:
        n = 0
    return [[0, 1]] + ([[0, 1, 2]] if n >= 3 else [])


@pytest.fixture(params=_device_sets(), ids=lambda s: "devices%d" % len(s))
def multi(request):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    m = _new(devices=request.param)
    yield m
    m.close()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["col_fastest", "k_fastest"])
def test_multi_device_step(layout, multi, refh):
    st, p, dz = R.bench_like(7001, 100.0)
    _, _, want, _ = ref_run(refh["mixed"], st, p, dz, 60.0)
    multi.enable_rates(True)
    pl = np.ascontiguousarray(p if layout == "col_fastest" else p.T)
    multi.step(60.0, host_arrays(st, layout), pl, dz, layout=layout)
    assert_bits(read_rates(multi, 7001, 60), np.ascontiguousarray(own(want).transpose(0, 2, 1)), "multi step " + layout)


@pytest.mark.gpu
@pytest.mark.parametrize("nx", [77, 1])
def test_multi_device_kid_interface(nx, multi, refh):
    kid, p0, roc = kid_inputs(nx, 60)
    single = _new()
    try:
        single.enable_rates(True)
        single.kid_interface(kid, DT_KID, p0, roc)
        want = read_rates(single, nx, 60)
    finally:
        single.close()
    multi.enable_rates(True)
    multi.kid_interface(kid, DT_KID, p0, roc)
    assert_bits(read_rates(multi, nx, 60), want, "multi kid nx=%d" % nx)


@pytest.mark.gpu
def test_multi_device_column_and_wrf_tile(multi, dom, refh):
    d = dom("D1")
    j = int(np.flatnonzero(active_columns(d["rates"]))[0])
    multi.enable_rates(True)
    multi.step(d["dt"], host_arrays(d["st"], "k_fastest"), np.ascontiguousarray(d["p"].T), d["dz"], layout="k_fastest")
    multi.column(d["dt"], *[d["st"][k][:, j] for k in FIELDS], d["p"][:, j], d["dz"])
    assert_bits(read_rates(multi, 1, d["nz"])[:, 0, :], own(d["rates"])[:, :, j], "multi column")
    pt, st, p, dz = wrf_patch("odd")
    nk, ncol = st["t"].shape
    _, _, want, _ = ref_run(refh["mixed"], st, p, dz, 20.0)
    f3, pii, pp, dzz, acc, radii, _ = pt.args()
    multi.mp_gt_driver(20.0, f3, pii, pp, dzz, acc, radii=radii, tile=pt.tile)
    assert_bits(read_rates(multi, ncol, nk), np.ascontiguousarray(own(want).transpose(0, 2, 1)), "multi wrf tile")


@pytest.mark.gpu
def test_multi_device_smaller_step_after_a_larger_state(multi, refh):
    """state_alloc of 7001 columns, then a kidmp_step of 2001: get_rates writes the 2001 columns' rates and nothing after them."""
    st, p, dz = R.bench_like(2001, 100.0)
    _, _, want, _ = ref_run(refh["mixed"], st, p, dz, 60.0)
    multi.enable_rates(True)
    multi.state_alloc(7001, 60)
    multi.step(60.0, host_arrays(st, "k_fastest"), np.ascontiguousarray(p.T), dz, layout="k_fastest")
    assert_bits(read_rates(multi, 2001, 60), np.ascontiguousarray(own(want).transpose(0, 2, 1)), "multi after state_alloc")
