"""kidmp_step_aero: the aerosol-aware step (is_aerosol_aware = .true., M:28) on host arrays, in both layouts, through the chunk
pipeline (pageable and pinned arrays) and over several GPUs.

The reference of every check is kidmp_step_device_aero on device copies of the same inputs, whose parity with the oracle
test_gpu_parity.py::test_aerosol_aware_step establishes; the host entry must give the same bits: the nine fields, nc, nwfa, nifa
and ppt.  kidmp_diag's counts agree exactly; its f64 sums are bit-identical where the host entry steps the columns in the same
launches as the reference (the resident path), and agree to rounding where the pipeline or a second device adds the sums of its
chunks one after the other.  One comparison with the oracle ties the entry to the reference restatement as well."""
import contextlib
import os

import numpy as np
import pytest

import regimes
from parity_util import assert_parity, FIELDS

pytestmark = pytest.mark.gpu

AERO = ("nc", "nwfa", "nifa")
PIPE_CHUNK = 1024                                        # the smallest pipeline chunk kidmp_init takes


@contextlib.contextmanager
def _env(**kw):
    old = {k: os.environ.get(k) for k in kw}
    os.environ.update({k: str(v) for k, v in kw.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.fixture(scope="module")
def th():
    """A handle with the default pipeline chunk: the domains of these tests take the resident path (and are its reference)."""
    from kid_b200.kidmp import Thompson
    t = Thompson(set_Nc=100.0, iiwarm=False, l_sediment=True)
    yield t
    t.close()


@pytest.fixture(scope="module")
def piped():
    """A handle whose host pipeline cuts a column-fastest domain of 2048 columns or more into chunks of 1024."""
    from kid_b200.kidmp import Thompson
    with _env(KIDMP_PIPE_CHUNK=PIPE_CHUNK):
        t = Thompson(set_Nc=100.0, iiwarm=False, l_sediment=True)
    yield t
    t.close()


def _case(ncol, dt=10.0, dz=250.0, col0=123456, seed=20261018):
    """Mixed-phase columns (seven in ten cloudy, the rest clear sky) with aerosol inputs and a surface emission."""
    from kid_b200 import synth
    st, p, dzv = synth.make_domain(ncol, nz=60, nx=1024, dz=dz, col0=col0, cloudy_fraction=0.7, coherent=False)
    st = {k: v.numpy().copy() for k, v in st.items()}
    p = p.numpy().copy()
    nc, nwfa, nifa, w = synth.make_aerosols(st, p, seed=seed)
    nwfa2d = np.random.default_rng(seed).uniform(0.0, 1.0e5, ncol).astype(np.float32)
    return dict(st=st, ae=dict(nc=nc, nwfa=nwfa, nifa=nifa), p=p, w=w, dz=dzv.numpy().copy(), dt=dt, nwfa2d=nwfa2d)


def _regime_case():
    names = [c.name for c in regimes.CASES if c.aero]
    st, p, dz, dt = regimes.regime_domain(names)
    nc, nwfa, nifa, w = regimes.aero_inputs(st, p)
    nwfa2d = np.random.default_rng(3).uniform(0.0, 1.0e5, st["t"].shape[1]).astype(np.float32)
    return dict(st=st, ae=dict(nc=nc, nwfa=nwfa, nifa=nifa), p=p, w=w, dz=dz, dt=dt, nwfa2d=nwfa2d)


def device_ref(t, c, emit=True):
    """kidmp_step_device_aero on device copies of the inputs: (fields + nc nwfa nifa, ppt, diag, step_stats)."""
    import torch
    nz, ncol = c["st"]["t"].shape
    dev = {k: torch.from_numpy(c["st"][k].copy()).cuda() for k in FIELDS}
    dev.update({k: torch.from_numpy(c["ae"][k].copy()).cuda() for k in AERO})
    dp, dw, ddz = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (c["p"], c["w"], c["dz"]))
    dn2 = torch.from_numpy(c["nwfa2d"]).cuda() if emit else None
    ppt = torch.full((4, ncol), float("nan"), dtype=torch.float32, device="cuda")
    t.diag()
    torch.cuda.synchronize()
    t.step_device_aero(ncol, nz, c["dt"], [dev[k].data_ptr() for k in FIELDS], dev["nc"].data_ptr(), dev["nwfa"].data_ptr(),
                       dev["nifa"].data_ptr(), dp.data_ptr(), dw.data_ptr(), ddz.data_ptr(), ppt.data_ptr(),
                       nwfa2d_ptr=dn2.data_ptr() if emit else None)
    t.sync()
    return {k: v.cpu().numpy() for k, v in dev.items()}, ppt.cpu().numpy(), t.diag(), t.step_stats()


def _to(layout, a):
    return a.copy() if layout == "col_fastest" else np.ascontiguousarray(a.T)


def _from(layout, a):
    return a if layout == "col_fastest" else np.ascontiguousarray(a.T)


def host_step(t, c, layout="col_fastest", emit=True, pinned=(), diag=True):
    """kidmp_step_aero on host copies of the inputs in `layout`; the arrays named in `pinned` (FIELDS and AERO names, or "all")
    are page-locked.  Returns (fields + nc nwfa nifa as [nz][ncol], ppt, diag, step_stats)."""
    import torch
    names = FIELDS + AERO
    pin = set(names) if pinned == "all" else set(pinned)
    src = dict(c["st"], **c["ae"])
    arrs, keep = {}, []
    for k in names:
        a = _to(layout, src[k])
        if k in pin:
            tt = torch.from_numpy(a).pin_memory()
            keep.append(tt)
            a = tt.numpy()
        arrs[k] = a
    if diag:
        t.diag()
    ppt = t.step_aero(c["dt"], {k: arrs[k] for k in FIELDS}, {k: arrs[k] for k in AERO}, _to(layout, c["p"]), _to(layout, c["w"]),
                      c["dz"], layout=layout, nwfa2d=c["nwfa2d"] if emit else None)
    out = {k: _from(layout, arrs[k]).copy() for k in names}
    return out, ppt, t.diag() if diag else None, t.step_stats()


def assert_same(got, want, what, exact_diag=True):
    for k in FIELDS + AERO:
        assert np.array_equal(got[0][k], want[0][k]), "%s: %s differs in %d cells" % (what, k, int((got[0][k] != want[0][k]).sum()))
    assert np.array_equal(got[1], want[1]), "%s: ppt" % what
    if got[2] is not None and want[2] is not None:
        if exact_diag:
            assert np.array_equal(got[2], want[2]), "%s: diag %r != %r" % (what, got[2], want[2])
        else:
            assert np.array_equal(got[2][6:], want[2][6:]), what
            np.testing.assert_allclose(got[2][:6], want[2][:6], rtol=1e-12, atol=0, err_msg=what)


def _skipped(c, ref):
    """Columns that the step leaves as they were in all twelve planes, but for the lowest nwfa level (the emission)."""
    src = dict(c["st"], **c["ae"])
    same = np.ones(c["st"]["t"].shape[1], bool)
    for k in FIELDS + AERO:
        a, b = ref[0][k], src[k]
        same &= (a[1:] == b[1:]).all(0) if k == "nwfa" else (a == b).all(0)
    return same


# ---- the resident path: small domains and every KIDMP_K_FASTEST call -------------------------------------------------------
@pytest.mark.parametrize("emit", [True, False], ids=["nwfa2d", "no_nwfa2d"])
@pytest.mark.parametrize("layout", ["col_fastest", "k_fastest"])
@pytest.mark.parametrize("dt,dz", [(10.0, 250.0), (60.0, 100.0)], ids=["mixed", "substeps"])
def test_resident_path_is_the_device_step(th, layout, emit, dt, dz):
    c = _case(3000, dt=dt, dz=dz)
    ref = device_ref(th, c, emit)
    if dt > 30.0:
        assert ref[3]["substep_columns"] > 0                                # the sub-stepped columns ran
    got = host_step(th, c, layout, emit)
    assert_same(got, ref, "%s dt=%g %s" % (layout, dt, emit))
    assert got[3]["zero_copy_return"] == 0
    # the step did work: the droplet number moved, the emission reached the lowest level
    assert not np.array_equal(got[0]["nc"], c["ae"]["nc"])
    if emit:
        assert (got[0]["nwfa"][0] != c["ae"]["nwfa"][0]).mean() > 0.9


@pytest.mark.parametrize("emit", [True, False], ids=["nwfa2d", "no_nwfa2d"])
@pytest.mark.parametrize("layout", ["col_fastest", "k_fastest"])
def test_regime_cases(th, layout, emit):
    """The aerosol-aware cases of tests/regimes.py side by side, with aerosol inputs at the clamps of M:1392-1410."""
    c = _regime_case()
    assert_same(host_step(th, c, layout, emit), device_ref(th, c, emit), "regimes %s %s" % (layout, emit))


def test_against_the_oracle(th, oracle_mixed):
    """One step against the oracle's restatement, at the tolerance of test_aerosol_aware_step."""
    c = _case(2000, dt=10.0, col0=77777)
    got = host_step(th, c, "k_fastest")
    ref = {k: v.copy() for k, v in c["st"].items()}
    rae = {k: v.copy() for k, v in c["ae"].items()}
    ppt = oracle_mixed.step_aero(c["dt"], ref, rae["nc"], rae["nwfa"], rae["nifa"], c["p"], c["w"], c["dz"], nwfa2d=c["nwfa2d"])
    assert_parity(got[0], dict(ref, **rae), fields=FIELDS + AERO, what="kidmp_step_aero vs oracle", flip_fraction=1e-3)
    np.testing.assert_allclose(got[1], ppt, rtol=1e-4, atol=1e-9)


# ---- the chunk pipeline -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("emit", [True, False], ids=["nwfa2d", "no_nwfa2d"])
def test_pipeline(th, piped, emit):
    """5000 columns in five chunks of 1024: the copy path (pageable arrays, KIDMP_ZEROCOPY=0, one pageable aerosol array) and the
    zero-copy path (all twelve INOUT arrays pinned), which writes only the changed columns back - and, with nwfa2d, the lowest
    nwfa level of every column."""
    c = _case(5000, col0=300000)
    ref = device_ref(th, c, emit)
    skipped = _skipped(c, ref)
    assert skipped.sum() > 100                                          # clear-sky columns the zero-copy path leaves alone
    if emit:                                                            # (an emission below half an ulp of nwfa changes nothing)
        assert (ref[0]["nwfa"][0, skipped] != c["ae"]["nwfa"][0, skipped]).mean() > 0.99
    runs = [("pageable", (), {}, 0), ("pinned", "all", {}, 1), ("zerocopy off", "all", {"KIDMP_ZEROCOPY": 0}, 0),
            ("pageable nc", FIELDS + ("nwfa", "nifa"), {}, 0)]
    for what, pinned, env, zc in runs:
        with _env(**env):
            got = host_step(piped, c, emit=emit, pinned=pinned)
        assert_same(got, ref, "pipeline, %s" % what, exact_diag=False)
        assert got[3]["zero_copy_return"] == zc, what


def test_repeated_calls_on_one_handle(th, piped):
    """Plain and aerosol-aware steps of different sizes and layouts alternate on one handle: the pipeline buffer grows for the
    aerosol-aware layout and serves the plain one after it, the resident state and the aerosol planes are re-used, and the
    captured graphs of a size are replayed with new array contents."""
    from kid_b200 import synth

    def plain(t, ncol, layout, col0):
        st, p, dz = synth.make_domain(ncol, nz=60, nx=1024, col0=col0, cloudy_fraction=0.7, coherent=False)
        st = {k: _to(layout, v.numpy()) for k, v in st.items()}
        ppt = t.step(10.0, st, _to(layout, p.numpy()), dz.numpy(), layout=layout)
        return {k: _from(layout, v) for k, v in st.items()}, ppt

    # (the two calls of 700 step the same resident planes, the two of 4100 the same pipeline chunks: graph replays)
    seq = [("plain", 5000, "col_fastest"), ("aero", 5000, "col_fastest"), ("plain", 3000, "col_fastest"), ("aero", 700, "k_fastest"),
           ("aero", 700, "col_fastest"), ("aero", 6100, "col_fastest"), ("plain", 500, "k_fastest"), ("aero", 4100, "col_fastest"),
           ("aero", 4100, "col_fastest"), ("aero", 900, "k_fastest")]
    for i, (kind, ncol, layout) in enumerate(seq):
        col0 = 1000 * i + 400000                                       # new contents at every call
        what = "call %d: %s %d %s" % (i, kind, ncol, layout)
        if kind == "plain":
            got, want = plain(piped, ncol, layout, col0), plain(th, ncol, layout, col0)
            for k in FIELDS:
                assert np.array_equal(got[0][k], want[0][k]), (what, k)
            assert np.array_equal(got[1], want[1]), what
        else:
            c = _case(ncol, col0=col0, seed=i)
            got = host_step(piped, c, layout, pinned="all" if i % 2 else ())
            assert_same(got, device_ref(th, c), what, exact_diag=ncol < 2 * PIPE_CHUNK or layout == "k_fastest")


# ---- several GPUs -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["col_fastest", "k_fastest"])
def test_two_gpus_equal_one(th, layout):
    """kidmp_config::ndev = 2: each device its column range (pitched copies through each device's pipeline, or a contiguous (k,i)
    range), every device with its own drop-evaporation table; the same bits as the single-device handle, and the NCCL
    all-reduced diag.  The rates refusal covers every device of the handle."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs in this process")
    from kid_b200.kidmp import Thompson, KidmpError
    with _env(KIDMP_PIPE_CHUNK=PIPE_CHUNK):
        two = Thompson(devices=[0, 1])
    try:
        c = _case(5003, col0=250000)
        for emit in (True, False):
            ref = host_step(th, c, layout, emit)
            assert_same(host_step(two, c, layout, emit), ref, "two GPUs %s %s" % (layout, emit), exact_diag=False)
            assert_same(ref, device_ref(th, c, emit), "one GPU %s %s" % (layout, emit))
        assert two._L.kidmp_num_devices(two.h) == 2
        two.enable_rates(True)
        with pytest.raises(KidmpError, match="process-rate"):
            host_step(two, c, layout)
        two.enable_rates(False)
    finally:
        two.close()


# ---- refusals ---------------------------------------------------------------------------------------------------------------
def test_refusals_touch_nothing(th):
    """A refused call copies and launches nothing and leaves every array - and a NaN-filled rate buffer - bit for bit as it was;
    ncol = 0 succeeds and touches nothing."""
    import torch
    from kid_b200.kidmp import KidmpError, _fp, _ptrs
    c = _case(600)
    arrs = {k: v.copy() for k, v in dict(c["st"], **c["ae"]).items()}
    ppt = np.full((4, 600), 7.0, np.float32)
    before = {k: v.copy() for k, v in arrs.items()}
    L = th._L
    P = lambda a: a.ctypes.data_as(_fp)

    def call(ncol=600, nz=60, dt=10.0, drop=None):
        ptr = {k: P(arrs[k]) for k in AERO}
        ptr.update(p=P(c["p"]), w=P(c["w"]), dz=P(c["dz"]))
        if drop:
            ptr[drop] = None
        return L.kidmp_step_aero(th.h, ncol, nz, dt, 1, _ptrs([arrs[k] for k in FIELDS]), ptr["nc"], ptr["nwfa"], ptr["nifa"],
                                 ptr["p"], ptr["w"], ptr["dz"], P(c["nwfa2d"]), P(ppt))

    def untouched(what):
        for k, v in before.items():
            assert np.array_equal(arrs[k], v), (what, k)
        assert (ppt == 7.0).all(), what

    launches = th.gpu_launches
    for drop in ("nc", "nwfa", "nifa", "w", "p", "dz"):
        assert call(drop=drop) != 0 and b"null" in L.kidmp_last_error(th.h), drop
        untouched(drop)
    for nz in (1, 257):
        assert call(nz=nz) != 0 and b"nz" in L.kidmp_last_error(th.h)
        untouched("nz=%d" % nz)
    for dt in (0.0, -10.0, float("nan")):
        assert call(dt=dt) != 0 and b"dt" in L.kidmp_last_error(th.h)
        untouched("dt=%g" % dt)
    assert call(ncol=0) == 0
    assert L.kidmp_step_aero(th.h, 0, 60, 10.0, 1, None, None, None, None, None, None, None, None, None) == 0
    untouched("ncol=0")
    assert th.gpu_launches == launches
    # rates kept, or a caller's rate buffer: refused, the buffer not written
    rates = torch.full((36, 60, 600), float("nan"), dtype=torch.float32, device="cuda")
    bits = rates.view(torch.int32).clone()
    th.set_rates_buffer(rates.data_ptr())
    try:
        assert call() != 0 and b"process-rate" in L.kidmp_last_error(th.h)
        with pytest.raises(KidmpError, match="process-rate"):
            host_step(th, c, diag=False)
    finally:
        th.set_rates_buffer(0)
    torch.cuda.synchronize()
    assert torch.equal(rates.view(torch.int32), bits)
    untouched("rate buffer")
    th.enable_rates(True)
    try:
        assert call() != 0 and b"process-rate" in L.kidmp_last_error(th.h)
    finally:
        th.enable_rates(False)
    untouched("rates kept")
    assert th.gpu_launches == launches
    # the binding checks shapes the way step checks set_nc
    with pytest.raises(ValueError, match="nwfa2d"):
        th.step_aero(10.0, arrs, arrs, c["p"], c["w"], c["dz"], nwfa2d=np.zeros(599, np.float32))
    with pytest.raises(ValueError, match="w shape"):
        th.step_aero(10.0, arrs, arrs, c["p"], c["w"][:, :10], c["dz"])
    untouched("shape checks")
