"""Per-column cloud droplet number (kidmp_step_nc, kidmp_step_device_nc, kidmp_mp_gt_driver_tile_nc / _device_nc).

In the plain scheme set_Nc feeds nothing but Nt_c = set_Nc * 1e6 (M:381), and no lookup table depends on it.  So a column
stepped with per-column value v must come out, bit for bit, as the same column stepped by a handle made with set_Nc = v.  Every
GPU test here steps one handle with values drawn from VALUES in a seeded shuffle (the lanes of one warp differ) and compares each
column with the handle of its value: the nine fields, ppt, the 36 rates (device rates buffer) and, on the WRF entries, the radii
and accumulators.  VALUES holds the exact NINT ties of nu_c = MIN(15, NINT(1000e6 / Nt_c) + 2) (400, 2000) and both of its ends
(10 -> 15, 3000 -> 2)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import regimes as R
from parity_util import FIELDS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VALUES = np.array([10.0, 50.0, 100.0, 300.0, 400.0, 1000.0, 2000.0, 3000.0], np.float32)
ENTRIES = ("kidmp_step_nc", "kidmp_step_device_nc", "kidmp_mp_gt_driver_tile_nc", "kidmp_mp_gt_driver_tile_device_nc")
OWN = 100.0                                   # set_Nc of the handles that take per-column values


def shuffled(n, seed):
    """n values of VALUES, each about n/8 times, in a seeded random order."""
    return VALUES[np.random.default_rng(seed).permutation(np.arange(n) % len(VALUES))]


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_values_reach_the_ties_and_both_ends_of_nu_c():
    F = np.float32

    def nu_c(v):                              # M:1705 in f32; NINT rounds half away from zero
        return min(15, int(np.floor(np.float64(F(F(1000.0e6) / F(F(v) * F(1.0e6)))) + 0.5)) + 2)
    got = {float(v): nu_c(v) for v in VALUES}
    assert got[10.0] == 15 and got[3000.0] == 2
    for v, x in ((400.0, 2.5), (2000.0, 0.5)):
        assert F(F(1000.0e6) / F(F(v) * F(1.0e6))) == F(x)        # an exact tie in f32
    assert sorted(set(got.values())) == [2, 3, 5, 12, 15]
    v = shuffled(64, 1)
    assert len(set(v[:32])) > 1 and len(set(v[32:])) > 1


def test_entries_are_declared_bound_and_exported():
    from kid_b200 import kidmp
    hdr = open(os.path.join(ROOT, "include", "kidmp.h")).read()
    f90 = open(os.path.join(ROOT, "kid_b200", "fortran", "mphys_thompson09n.f90")).read()
    L = kidmp.load()
    for name in ENTRIES:
        assert re.search(r"\bint %s\(" % name, hdr), name
        assert name in kidmp.SYMBOLS and hasattr(L, name), name
    for name in ENTRIES[2:]:
        assert "bind(C, name='%s')" % name in f90, name


# ---- GPU: helpers ------------------------------------------------------------------------------------------------------
class Handles:
    """One handle per (set_Nc, iiwarm), made on first use and kept for the module: the per-value references and the handles
    that take per-column values (OWN)."""

    def __init__(self):
        self.h = {}

    def __call__(self, set_Nc, iiwarm=False):
        from kid_b200.kidmp import Thompson
        key = (float(set_Nc), bool(iiwarm))
        if key not in self.h:
            self.h[key] = Thompson(set_Nc=float(set_Nc), iiwarm=bool(iiwarm), l_sediment=True)
        return self.h[key]

    def close(self):
        for th in self.h.values():
            th.close()


@pytest.fixture(scope="module")
def handles():
    hs = Handles()
    yield hs
    hs.close()


@pytest.fixture(scope="module")
def oracles():
    """The oracle of each value (mixed phase, sedimentation), made on first use."""
    from oracle.oracle import Oracle
    made = {}

    def get(v):
        if float(v) not in made:
            made[float(v)] = Oracle(set_Nc=float(v), iiwarm=False, l_sediment=True)
        return made[float(v)]
    yield get
    for o in made.values():
        o.close()


class Dev:
    """Device copies of one input at fixed addresses (a handle with CUDA graphs on replays its capture while they stay)."""

    def __init__(self, st, p, dz, dt, rates=True):
        import torch
        self.nz, self.ncol = st["t"].shape
        self.dt = dt
        self.src = {k: torch.from_numpy(np.ascontiguousarray(st[k])).cuda() for k in FIELDS}
        self.dev = {k: v.clone() for k, v in self.src.items()}
        self.p, self.dz = torch.from_numpy(np.ascontiguousarray(p)).cuda(), torch.from_numpy(np.ascontiguousarray(dz)).cuda()
        self.ppt = torch.zeros((4, self.ncol), dtype=torch.float32, device="cuda")
        self.rates = torch.empty((36, self.nz, self.ncol), dtype=torch.float32, device="cuda") if rates else None

    def run(self, th, set_nc=None):
        """One kidmp_step_device[_nc] from the inputs (set_nc: a CUDA tensor [ncol] or None).  Returns a dict of device
        tensors: the fields, ppt, rates (NaN where the step wrote nothing), and diag / stats."""
        import torch
        for k in FIELDS:
            self.dev[k].copy_(self.src[k])
        if self.rates is not None:
            self.rates.fill_(float("nan"))
        th.set_rates_buffer(self.rates.data_ptr() if self.rates is not None else 0)
        th.diag()
        torch.cuda.synchronize()
        try:
            th.step_device(self.ncol, self.nz, self.dt, [self.dev[k].data_ptr() for k in FIELDS], self.p.data_ptr(),
                           self.dz.data_ptr(), self.ppt.data_ptr(), set_nc_ptr=set_nc.data_ptr() if set_nc is not None else None)
            th.sync()
        finally:
            th.set_rates_buffer(0)
        out = {k: self.dev[k].clone() for k in FIELDS}
        out["ppt"] = self.ppt.clone()
        if self.rates is not None:
            out["rates"] = self.rates.clone()
        out["diag"], out["stats"] = th.diag(), th.step_stats()
        return out


def _bits(t):
    import torch
    return t.view(torch.int32)


def assert_columns(got, want, cols, what):
    """got and want (dicts of device tensors, columns last) hold the same bits in columns `cols` (an index tensor)."""
    import torch
    for k in FIELDS + ("ppt", "rates"):
        if k in got and k in want:
            a, b = _bits(got[k]).index_select(-1, cols), _bits(want[k]).index_select(-1, cols)
            if not torch.equal(a, b):
                n = int((a != b).sum())
                raise AssertionError("%s: %s differs in %d cells" % (what, k, n))


def assert_per_value(handles, d, vals, got, iiwarm=False, what=""):
    """Every column of `got` (a per-column run of Dev d with values vals) against the handle of its value."""
    import torch
    refs = []
    for v in VALUES:
        cols = torch.from_numpy(np.flatnonzero(vals == v)).cuda()
        if cols.numel() == 0:
            continue
        ref = d.run(handles(v, iiwarm))
        assert_columns(got, ref, cols, "%s set_Nc %g" % (what, v))
        assert got["diag"][6] == ref["diag"][6] and got["diag"][7] == ref["diag"][7] == d.ncol, (what, v)
        refs.append(ref)
    return refs


def differs(a, b, k):
    import torch
    return not torch.equal(_bits(a[k]), _bits(b[k]))


# ---- GPU: the step against one handle per value ------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dt,iiwarm", [(10.0, False), (60.0, False), (60.0, True)], ids=["dt10", "dt60", "warm_dt60"])
def test_bench_domain_matches_one_handle_per_value(handles, dt, iiwarm):
    """65 536 bench-like columns of 60 levels; at dt = 60 s columns take sedimentation sub-steps (k_substeps)."""
    import torch
    st, p, dz = R.bench_like(65536, 100.0)
    d = Dev(st, p, dz, dt)
    vals = shuffled(d.ncol, 11)
    got = d.run(handles(OWN if not iiwarm else 50.0, iiwarm), torch.from_numpy(vals).cuda())
    if dt == 60.0:
        assert got["stats"]["substep_columns"] > 0, got["stats"]
    refs = assert_per_value(handles, d, vals, got, iiwarm, "bench dt=%g" % dt)
    assert differs(refs[0], refs[-1], "qc") and differs(refs[0], refs[-1], "rates")     # set_Nc matters on this domain
    # the domain sums of the per-column run: its own precipitation and water paths
    ppt = got["ppt"].double().sum(dim=1).cpu().numpy()
    np.testing.assert_allclose(got["diag"][:4], ppt, rtol=1e-9, atol=0)


@pytest.mark.gpu
def test_regime_cases_with_every_value_in_every_column(handles):
    """The 18 regime cases (tests/regimes.py): the regime domain eight times side by side, copy r with the shuffled values
    rotated by r, so every column of every case runs with every value; the sediment case, which has its own layers, alone."""
    import torch
    st, p, dz, dt = R.regime_domain()
    n = st["t"].shape[1]
    base = np.random.default_rng(5).permutation(np.arange(n) % len(VALUES))
    idx = np.concatenate([(base + r) % len(VALUES) for r in range(len(VALUES))])
    tile = lambda a: np.ascontiguousarray(np.tile(a, (1, len(VALUES))))
    d = Dev({k: tile(v) for k, v in st.items()}, tile(p), dz, dt)
    vals = VALUES[idx]
    got = d.run(handles(OWN), torch.from_numpy(vals).cuda())
    assert_per_value(handles, d, vals, got, what="regimes")
    sst, sp, sdz, sdt = R.build("sediment")
    d = Dev(sst, sp, sdz, sdt)
    vals = shuffled(d.ncol, 6)
    got = d.run(handles(OWN), torch.from_numpy(vals).cuda())
    assert_per_value(handles, d, vals, got, what="sediment")


@pytest.mark.gpu
@pytest.mark.parametrize("case", R.CASES, ids=str)
def test_regime_case_against_oracles_of_the_same_values(case, handles, oracles):
    """Each regime case with shuffled per-column values against the oracle of each column's value, with the allowances of
    tests/test_configurations.py (state at REL_TOL, rates at 1e-5, precipitation)."""
    import torch
    from test_configurations import STATE_ALLOW
    st, p, dz, dt = R.build(case)
    d = Dev(st, p, dz, dt)
    vals = shuffled(d.ncol, len(case.name))
    got = d.run(handles(OWN), torch.from_numpy(vals).cuda())
    state = {k: got[k].cpu().numpy() for k in FIELDS}
    ppt, rates = got["ppt"].cpu().numpy(), got["rates"].cpu().numpy()
    cls, _ = R.cell_classes(st, p)
    bad, rbad = [], []
    for v in VALUES:
        m = vals == v
        if not m.any():
            continue
        _, _, _, _, ref, ppt_ref, rates_ref = R.oracle_run(oracles(v), case)
        names = oracles(v).rate_names
        bad += R.cell_outliers({k: state[k][:, m] for k in FIELDS}, {k: ref[k][:, m] for k in FIELDS}, FIELDS, cls[:, m])
        active = m & np.isfinite(rates).all(axis=(0, 1))
        assert not rates_ref[:, :, m & ~active].any(), v
        rbad += R.rate_outliers(rates[:, :, active], rates_ref[:, :, active], names, cls[:, active])
        np.testing.assert_allclose(ppt[:, m], ppt_ref[:, m], rtol=1e-5, atol=1e-10, err_msg="%s set_Nc %g ppt" % (case.name, v))
    allow = max([n for (c, cfg), n in STATE_ALLOW.items() if c == case.name and not cfg.startswith("warm")] or [0])
    assert len(bad) <= allow, "%s state:\n  %s" % (case.name, "\n  ".join(bad[:20]))
    assert not rbad, "%s rates:\n  %s" % (case.name, "\n  ".join(rbad[:20]))


@pytest.mark.gpu
def test_uniform_values_of_the_handles_own_set_nc_equal_the_plain_step(handles):
    import torch
    st, p, dz = R.bench_like(20000, 100.0)
    d = Dev(st, p, dz, 60.0)
    th = handles(OWN)
    plain = d.run(th)
    got = d.run(th, torch.full((d.ncol,), OWN, dtype=torch.float32, device="cuda"))
    assert_columns(got, plain, torch.arange(d.ncol, device="cuda"), "uniform")
    np.testing.assert_array_equal(got["diag"], plain["diag"])


@pytest.mark.gpu
def test_every_schedule_gives_the_same_bits(handles):
    """Graphs, the simple-column path, the class kernels, the serial timing schedule and launch chunks below the domain (three
    chunks and a remainder: each chunk reads its own slice of set_nc) all give the per-value bits.  With graphs on, new values
    written into the same array between two replays are read by the replay."""
    import torch
    from kid_b200.kidmp import Thompson
    st, p, dz = R.bench_like(5000, 100.0)
    d = Dev(st, p, dz, 60.0)
    vals = shuffled(d.ncol, 21)
    nc = torch.from_numpy(vals).cuda()
    want = d.run(handles(OWN), nc)
    assert_per_value(handles, d, vals, want, what="schedules")
    allc = torch.arange(d.ncol, device="cuda")
    th = Thompson(set_Nc=OWN, iiwarm=False, l_sediment=True)
    try:
        for name, value in (("graphs", 0), ("graphs", 1), ("simple", 0), ("simple", 1), ("classes", 0), ("classes", 1),
                            ("timing", 1), ("timing", 0), ("chunk", 1536), ("chunk", 1 << 20)):
            th.set_option(name, value)
            for rep in range(2):
                got = d.run(th, nc)
                assert_columns(got, want, allc, "%s=%d run %d" % (name, value, rep))
                np.testing.assert_array_equal(got["diag"][6:], want["diag"][6:])
        # the same pointer, new contents: the replay of the captured step reads them
        got = d.run(th, nc)
        vals2 = shuffled(d.ncol, 22)
        nc.copy_(torch.from_numpy(vals2).cuda())
        got2 = d.run(th, nc)
        assert differs(got, got2, "qc")
        assert_per_value(handles, d, vals2, got2, what="new contents")
    finally:
        th.close()


@pytest.mark.gpu
def test_per_column_and_plain_runs_interleaved_on_one_handle(handles):
    """Plain and per-column steps alternate on one handle with graphs on, on the same arrays: each keeps its own bits (a graph
    captured for one is never replayed for the other)."""
    import torch
    from kid_b200.kidmp import Thompson
    st, p, dz = R.bench_like(8000, 100.0)
    d = Dev(st, p, dz, 60.0)
    vals = shuffled(d.ncol, 31)
    nc = torch.from_numpy(vals).cuda()
    allc = torch.arange(d.ncol, device="cuda")
    th = Thompson(set_Nc=OWN, iiwarm=False, l_sediment=True)
    try:
        plain, mixed = d.run(th), d.run(th, nc)
        assert differs(plain, mixed, "qc")
        assert_per_value(handles, d, vals, mixed, what="interleaved")
        for rep in range(3):
            assert_columns(d.run(th), plain, allc, "plain %d" % rep)
            assert_columns(d.run(th, nc), mixed, allc, "per-column %d" % rep)
        # the host entry on the resident state: the same, with the handle's own staging of the values
        host = {k: np.ascontiguousarray(v) for k, v in st.items()}
        ppt0 = th.step(60.0, {k: v.copy() for k, v in host.items()}, p, dz)
        for rep in range(2):
            a = {k: v.copy() for k, v in host.items()}
            ppt = th.step(60.0, a, p, dz, set_nc=vals)
            for k in FIELDS:
                assert np.array_equal(a[k].view(np.uint32), mixed[k].cpu().numpy().view(np.uint32)), (rep, k)
            assert np.array_equal(ppt.view(np.uint32), mixed["ppt"].cpu().numpy().view(np.uint32)), rep
            b = {k: v.copy() for k, v in host.items()}
            assert np.array_equal(th.step(60.0, b, p, dz).view(np.uint32), ppt0.view(np.uint32)), rep
            for k in FIELDS:
                assert np.array_equal(b[k].view(np.uint32), plain[k].cpu().numpy().view(np.uint32)), (rep, k)
    finally:
        th.close()


# ---- GPU: the host entry -----------------------------------------------------------------------------------------------
def _host_want(d, got_dev):
    return {k: got_dev[k].cpu().numpy() for k in FIELDS}, got_dev["ppt"].cpu().numpy()


def _assert_host(state, ppt, want, want_ppt, layout, what):
    for k in FIELDS:
        a = state[k] if layout == "col_fastest" else state[k].T
        assert np.array_equal(np.ascontiguousarray(a).view(np.uint32), want[k].view(np.uint32)), (what, k)
    assert np.array_equal(ppt.view(np.uint32), want_ppt.view(np.uint32)), what


def _host_arrays(st, layout, pinned):
    import torch
    out = {}
    for k, v in st.items():
        a = np.ascontiguousarray(v if layout == "col_fastest" else v.T)
        if pinned:
            t = torch.from_numpy(a.copy()).pin_memory()
            out[k] = t.numpy()
            out.setdefault("_keep", []).append(t)
        else:
            out[k] = a.copy()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [False, True], ids=["pageable", "pinned"])
@pytest.mark.parametrize("layout", ["col_fastest", "k_fastest"])
def test_host_entry(handles, layout, pinned):
    """kidmp_step_nc on the resident path, both layouts, pageable and pinned arrays; with the handle's own rates kept
    (kidmp_enable_rates), the rates of every column are those of its value's handle."""
    import torch
    from kid_b200.kidmp import Thompson
    st, p, dz = R.bench_like(6000, 100.0)
    d = Dev(st, p, dz, 60.0)
    vals = shuffled(d.ncol, 41)
    want = d.run(handles(OWN), torch.from_numpy(vals).cuda())
    assert_per_value(handles, d, vals, want, what="host reference")
    ws, wp = _host_want(d, want)
    th = Thompson(set_Nc=OWN, iiwarm=False, l_sediment=True)
    try:
        th.enable_rates(True)
        arrs = _host_arrays(st, layout, pinned)
        pp = np.ascontiguousarray(p if layout == "col_fastest" else p.T)
        ppt = th.step(60.0, arrs, pp, dz, layout=layout, set_nc=vals)
        _assert_host(arrs, ppt, ws, wp, layout, "host %s" % layout)
        rates = th.get_rates(d.ncol, d.nz, layout="col_fastest" if layout == "col_fastest" else "k_fastest")
        r = want["rates"].cpu().numpy()
        active = np.isfinite(r).all(axis=(0, 1))
        r = np.where(np.isnan(r), 0.0, r).astype(np.float32)            # (the handle's own buffer starts every step at zero)
        if layout == "k_fastest":
            rates = np.ascontiguousarray(rates.transpose(0, 2, 1))
        assert np.array_equal(rates.view(np.uint32), r.view(np.uint32)), layout
        assert active.any()
    finally:
        th.close()


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [False, True], ids=["pageable", "pinned"])
def test_host_entry_through_the_chunk_pipeline(handles, monkeypatch, pinned):
    """A column-fastest domain of at least two pipeline chunks goes through the host pipeline (KIDMP_PIPE_CHUNK = 1024 set
    before the handle is made): three chunks and a remainder, each with its slice of set_nc."""
    import torch
    from kid_b200.kidmp import Thompson
    st, p, dz = R.bench_like(3 * 1024 + 77, 100.0)
    d = Dev(st, p, dz, 60.0, rates=False)
    vals = shuffled(d.ncol, 51)
    want = d.run(handles(OWN), torch.from_numpy(vals).cuda())
    assert_per_value(handles, d, vals, want, what="pipeline reference")
    ws, wp = _host_want(d, want)
    monkeypatch.setenv("KIDMP_PIPE_CHUNK", "1024")
    th = Thompson(set_Nc=OWN, iiwarm=False, l_sediment=True)
    try:
        for rep in range(2):
            arrs = _host_arrays(st, "col_fastest", pinned)
            ppt = th.step(60.0, arrs, p, dz, set_nc=vals)
            _assert_host(arrs, ppt, ws, wp, "col_fastest", "pipeline %d" % rep)
            if pinned:
                assert th.step_stats()["zero_copy_return"] == 1          # (only the pipeline returns columns this way)
    finally:
        th.close()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["col_fastest", "k_fastest"])
def test_host_entry_on_two_gpus(handles, layout):
    import torch
    from kid_b200.kidmp import Thompson
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    st, p, dz = R.bench_like(7001, 100.0)
    d = Dev(st, p, dz, 60.0, rates=False)
    vals = shuffled(d.ncol, 61)
    want = d.run(handles(OWN), torch.from_numpy(vals).cuda())
    assert_per_value(handles, d, vals, want, what="two-GPU reference")
    ws, wp = _host_want(d, want)
    m = Thompson(set_Nc=OWN, iiwarm=False, l_sediment=True, devices=[0, 1])
    try:
        arrs = _host_arrays(st, layout, False)
        pp = np.ascontiguousarray(p if layout == "col_fastest" else p.T)
        ppt = m.step(60.0, arrs, pp, dz, layout=layout, set_nc=vals)
        _assert_host(arrs, ppt, ws, wp, layout, "two GPUs %s" % layout)
        assert m.diag()[7] == d.ncol
    finally:
        m.close()


@pytest.mark.gpu
@pytest.mark.parametrize("bad", [float("nan"), 0.0, -100.0], ids=["nan", "zero", "negative"])
def test_host_entry_rejects_a_bad_value_and_touches_nothing(handles, bad):
    from kid_b200 import kidmp
    st, p, dz = R.bench_like(3000, 100.0)
    th = handles(OWN)
    L = th._L
    vals = shuffled(3000, 71)
    vals[-1] = bad                                        # (the last value read)
    for layout in (kidmp.COL_FASTEST, kidmp.K_FASTEST):
        arrs = [np.ascontiguousarray(st[k] if layout == kidmp.COL_FASTEST else st[k].T) for k in FIELDS]
        before = [a.copy() for a in arrs] + [p.copy(), dz.copy(), vals.copy()]
        ppt = np.full((4, 3000), 7.0, np.float32)
        fp = C.cast(kidmp._ptrs(arrs), kidmp._fpp)
        P = lambda a: a.ctypes.data_as(kidmp._fp)
        rc = L.kidmp_step_nc(th.h, 3000, 60, 60.0, layout, fp, P(p), P(dz), P(vals), P(ppt))
        assert rc != 0 and b"set_nc[2999]" in L.kidmp_last_error(th.h)
        for a, b in zip(arrs + [p, dz, vals], before):
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
        assert (ppt == 7.0).all()
    with pytest.raises(kidmp.KidmpError, match="finite and positive"):
        th.step(60.0, {k: v.copy() for k, v in st.items()}, p, dz, set_nc=vals)


# ---- GPU: the WRF tile entries -----------------------------------------------------------------------------------------
NC_TAG = 0x3F                                     # NaN payload of set_nc2d outside the tile


def _wrf_patch(seed, **case):
    from test_wrf_tiles import Patch, _nans
    pt = Patch(seed=seed, **case)
    nj, ni = pt.mem_shape[0], pt.mem_shape[2]
    nc2d = _nans((nj, ni), NC_TAG)
    vals2 = shuffled(pt.tile[1] * pt.tile[5], seed).reshape(pt.tile[5], pt.tile[1])
    nc2d[pt.s2] = vals2
    return pt, nc2d, vals2


def _wrf_want(pt, handles, vals2, dt):
    """The tile's cells as the packed entry of each column's value's handle computes them."""
    orig = {k: v.copy() for k, v in pt.packed.items()}
    want = None
    for v in VALUES:
        pt.packed = {k: a.copy() for k, a in orig.items()}
        out = pt.run_packed(handles(v), dt)
        if want is None:
            want = {k: a.copy() for k, a in out.items()}
        m = vals2 == v
        for k, a in out.items():
            sel = np.broadcast_to(m[:, None, :], a.shape) if a.ndim == 3 else m
            want[k][sel] = a[sel]
    pt.packed = orig
    assert not np.array_equal(want["re_cloud"], out["re_cloud"])           # the radii follow the column's value
    return want


WRF_CASES = {"odd": dict(ni=37, nk=30, nj=5, hi=(3, 3), hj=(2, 2)),
             "k0": dict(ni=40, nk=20, nj=4, hi=(2, 3), hj=(1, 2), k0=1, spare=2),
             "mpas": dict(ni=301, nk=20, nj=1, hi=(0, 6), hj=(0, 0))}


@pytest.mark.gpu
@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("case", list(WRF_CASES))
def test_wrf_tile(handles, case, device):
    """kidmp_mp_gt_driver_tile_nc (host arrays) and kidmp_mp_gt_driver_tile_device_nc (CUDA tensors, on a non-default torch
    stream): inside the tile every array holds the bits of its column's value's handle (fields, accumulators, radii); every cell
    outside it, set_nc2d included, keeps its NaN with its own payload."""
    import torch
    pt, nc2d, vals2 = _wrf_patch(7 + len(case), **WRF_CASES[case])
    want = _wrf_want(pt, handles, vals2, 20.0)
    nc_before = nc2d.copy()
    th = handles(OWN)
    if not device:
        f3, pii, p, dz, acc, radii, _ = pt.args()
        th.mp_gt_driver(20.0, f3, pii, p, dz, acc, radii=radii, tile=pt.tile, set_nc=nc2d)
        got = pt.mem
    else:
        dev = {k: torch.from_numpy(v.copy()).cuda() for k, v in pt.mem.items()}
        dnc = torch.from_numpy(nc2d.copy()).cuda()
        torch.cuda.synchronize()
        s = torch.cuda.Stream()
        f3, pii, p, dz, acc, radii, _ = pt.args(dev)
        with torch.cuda.stream(s):
            th.mp_gt_driver_device(20.0, f3, pii, p, dz, acc, tile=pt.tile, radii=radii, stream=s, set_nc=dnc)
        s.synchronize()
        got = {k: v.cpu().numpy() for k, v in dev.items()}
        nc2d = dnc.cpu().numpy()
    pt.check(got, want)
    assert np.array_equal(nc2d.view(np.uint32), nc_before.view(np.uint32))


@pytest.mark.gpu
def test_wrf_host_tile_rejects_a_bad_value_inside_the_tile(handles):
    from kid_b200.kidmp import KidmpError
    pt, nc2d, _ = _wrf_patch(9, **WRF_CASES["odd"])
    i0, _, _, _, j0, _ = pt.tile
    nc2d[j0 + 1, i0 + 2] = -1.0
    f3, pii, p, dz, acc, radii, _ = pt.args()
    with pytest.raises(KidmpError, match=r"set_nc2d\(%d,%d\)" % (i0 + 2, j0 + 1)):
        handles(OWN).mp_gt_driver(20.0, f3, pii, p, dz, acc, radii=radii, tile=pt.tile, set_nc=nc2d)
    for k, a in pt.mem.items():
        assert np.array_equal(a.view(np.uint32), pt.before[k].view(np.uint32)), k
