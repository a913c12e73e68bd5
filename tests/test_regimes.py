"""Parity at the edges of the scheme: the directed cases of tests/regimes.py.

CPU tests (no GPU): every case still reaches the branch it was made for (its target fires in the oracle), its busy cells
fall in the kernel classes it claims, and the cases together hold every sort key of the cell list.
GPU tests: the CUDA step against the oracle case by case, cell by cell, rates included, with no outlier allowed unless a
count below names its cause; the class-specialised cell kernels against the general one (the "classes" option) bit for
bit; the schedule options on the regime domain; the aerosol-aware step on the cases that the aerosol switch changes.
"""
import numpy as np
import pytest

import regimes as R

FIELDS = R.FIELDS
AERO_FIELDS = FIELDS + ("nc", "nwfa", "nifa")

# Outliers allowed per (case, handle); every other case allows none.  Keep each a fixed count with its cause.
# sediment: dt = 120 s with hundreds of sedimentation sub-steps takes nearly all the graupel (rain: its number) out of the lowest
# levels; what is left there is a residual of 1e-5 to 1e-4 of the input, and a one-ulp difference of a fall speed between the
# device and the host evaluation of its power law (M:3318-3333), accumulated over the sub-steps, is a percent of that
# residual (the presumed cause: the outliers sit only there).  Observed on a B200: 4 cells (qg at the four lowest levels of one column) on the mixed handle, 2 (nr) on the warm one.
STATE_ALLOW = {("sediment", "mixed"): 4, ("sediment", "warm"): 2}
RATE_ALLOW = {}
AERO_ALLOW = {}

_oracle_cache = {}


def _oracle(o, case, handle):
    key = (case.name, handle)
    if key not in _oracle_cache:
        _oracle_cache[key] = R.oracle_run(o, case)
    return _oracle_cache[key]


# ---- CPU: the claims of the case table ---------------------------------------------------------------------------------
@pytest.mark.parametrize("case", R.CASES, ids=str)
def test_case_fires_its_target_in_the_oracle(case, oracle_mixed):
    st, p, dz, dt, out, ppt, rates = _oracle(oracle_mixed, case, "mixed")
    _, _, busy = R.classify(st, p)
    msgs = [t.check(st, p, out, rates, oracle_mixed.rate_names, busy) for t in case.targets]
    assert not any(msgs), (case.name, [m for m in msgs if m])


@pytest.mark.parametrize("case", R.CASES, ids=str)
def test_case_cells_fall_in_its_classes(case):
    st, p, dz, dt = R.build(case)
    cls, _ = R.cell_classes(st, p)
    got = set(cls[cls != ""])
    assert got == case.classes, (case.name, sorted(got), sorted(case.classes))
    assert (cls[:, 0::2] == "").any(), case.name                    # probe columns: idle levels around the busy ones


def test_cases_cover_every_sort_key():
    keys, warm_classes = set(), set()
    for case in R.CASES:
        st, p, dz, dt = R.build(case)
        keys |= R.cell_classes(st, p)[1]
        cls_w, _ = R.cell_classes(st, p, iiwarm=True)
        warm_classes |= set(cls_w[cls_w != ""])
    assert keys == set(range(64)), sorted(set(range(64)) - keys)
    assert warm_classes == {"WARM", "FULL"}                     # the two classes of an iiwarm handle


def test_thresholds_sit_on_both_sides_of_their_f32_values():
    """The spread of the cases holds each compared threshold exactly and one f32 step on either side of it."""
    t = np.concatenate([R.build(c)[0]["t"].ravel() for c in R.CASES])
    for thr in (R.HGFR, R.T_0, R.F(R.T_0 + R.F(0.1)), R.F(253.15)):
        assert {R.down(thr), thr, R.up(thr)} <= set(t.tolist()), thr
    st, p, dz, dt = R.build("cooper_ssati")
    s = R._ssati(st, p)
    # (qv / qvsi lies in [1, 2), where f32 values are 2**-23 apart: 0.25 - 2**-23 is the largest ssati below 0.25)
    assert (s == R.F(0.25)).any() and (s == R.F(0.25 - 2.0 ** -23)).any()
    st, p, dz, dt = R.build("vapour_warm")
    w = R._ssatw(st, p)
    assert (w == 0).any() and (w == R.F(2.0 ** -23)).any()             # saturated, and one f32 step above it


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _device_step(th, st, p, dz, dt, rates=True):
    return R.Device(st, p, dz, dt, rates).run(th)


@pytest.mark.gpu
@pytest.mark.parametrize("handle", ["mixed", "warm"])
@pytest.mark.parametrize("case", R.CASES, ids=str)
def test_case_parity_with_the_oracle(case, handle, gpu_mixed, gpu_warm, oracle_mixed, oracle_warm):
    """State cell by cell at REL_TOL, the 36 rates at 1e-5 relative, surface precipitation: the CUDA step against the oracle."""
    th, o = (gpu_mixed, oracle_mixed) if handle == "mixed" else (gpu_warm, oracle_warm)
    st, p, dz, dt, ref, ppt_ref, rates_ref = _oracle(o, case, handle)
    got, ppt, rates, _, _ = _device_step(th, st, p, dz, dt)
    cls, _ = R.cell_classes(st, p, iiwarm=handle == "warm")
    bad = R.cell_outliers(got, ref, FIELDS, cls)
    # clear-sky columns: the kernel leaves the buffer alone; every other column gets all of its levels
    active = np.isfinite(rates).all(axis=(0, 1))
    assert not rates_ref[:, :, ~active].any()
    rbad = R.rate_outliers(rates[:, :, active], rates_ref[:, :, active], o.rate_names, cls[:, active])
    print("REGIME %s/%s: %d state outliers, %d rate outliers" % (case.name, handle, len(bad), len(rbad)))
    assert len(bad) <= STATE_ALLOW.get((case.name, handle), 0), "%s/%s state:\n  %s" % (case.name, handle, "\n  ".join(bad[:20]))
    assert len(rbad) <= RATE_ALLOW.get((case.name, handle), 0), "%s/%s rates:\n  %s" % (case.name, handle, "\n  ".join(rbad[:20]))
    np.testing.assert_allclose(ppt, ppt_ref, rtol=1e-5, atol=1e-10, err_msg="%s/%s ppt" % (case.name, handle))


def _same(a, b, what):
    sa, pa, ra, da, _ = a
    sb, pb, rb, db, _ = b
    for k in FIELDS:
        assert np.array_equal(sa[k], sb[k]), (what, k, np.argwhere(sa[k] != sb[k])[:5])
    assert np.array_equal(pa, pb), what
    if ra is not None:
        assert np.array_equal(ra, rb, equal_nan=True), (what, "rates")
    assert da[6] == db[6] and da[7] == db[7], what
    assert np.allclose(da[:6], db[:6], rtol=1e-12, atol=0), what


@pytest.mark.gpu
def test_class_kernels_compute_what_the_general_kernel_computes():
    """Every class kernel computes bit for bit what k_cells<KC_FULL> computes for the same cell (kidmp_cells.cuh): the
    "classes" option 0 sends every busy cell to the general kernel.  One handle, CUDA graphs on, the option toggled between
    replays of the same arguments: the option is part of the graph key, or the second run would replay the first routing."""
    from kid_b200.kidmp import Thompson
    th = Thompson(set_Nc=100.0, iiwarm=False, l_sediment=True)
    try:
        inputs = [("regimes",) + R.regime_domain(), ("sediment",) + R.build("sediment")]
        for dt in (10.0, 60.0):
            inputs.append(("bench-like dt=%g" % dt,) + R.bench_like(40000, 100.0) + (dt,))
        for name, st, p, dz, dt in inputs:
            d = R.Device(st, p, dz, dt)
            runs = {}
            for classes in (1, 0, 1):
                th.set_option("classes", classes)
                r = d.run(th)
                runs.setdefault(classes, []).append(r)
                s = r[4]
                if classes == 0:
                    assert s["cells_full"] == s["busy_cells"] > 0, (name, s)
                    assert s["cells_warm"] == s["cells_ice"] == s["cells_mixed_no_rain"] == 0, (name, s)
            _same(runs[1][0], runs[0][0], name)
            _same(runs[1][0], runs[1][1], name + " (again)")
            if name == "regimes":
                s = runs[1][0][4]
                assert min(s["cells_warm"], s["cells_ice"], s["cells_mixed_no_rain"], s["cells_full"]) > 0, s
    finally:
        th.close()


@pytest.mark.gpu
def test_class_kernels_of_the_warm_handle():
    from kid_b200.kidmp import Thompson
    th = Thompson(set_Nc=50.0, iiwarm=True, l_sediment=True)
    try:
        d = R.Device(*R.regime_domain())
        runs = {}
        for classes in (1, 0):
            th.set_option("classes", classes)
            runs[classes] = d.run(th)
        _same(runs[1], runs[0], "iiwarm")
        s1, s0 = runs[1][4], runs[0][4]
        assert s1["cells_warm"] > 0 and s1["cells_full"] > 0 and s1["cells_ice"] == s1["cells_mixed_no_rain"] == 0, s1
        assert s0["cells_full"] == s0["busy_cells"] == s1["busy_cells"], s0
    finally:
        th.close()


AERO_CASES = [c for c in R.CASES if c.aero]


@pytest.mark.gpu
def test_aerosol_aware_class_kernels_compute_what_the_general_kernel_computes():
    from kid_b200.kidmp import Thompson
    th = Thompson(set_Nc=100.0, iiwarm=False, l_sediment=True)
    try:
        st, p, dz, dt = R.regime_domain({c.name for c in AERO_CASES})
        ae = R.aero_inputs(st, p, seed=1)
        runs = {}
        for classes in (1, 0):
            th.set_option("classes", classes)
            runs[classes] = R.aero_step(th, st, p, dz, dt, *ae)
        for k in AERO_FIELDS:
            assert np.array_equal(runs[1][0][k], runs[0][0][k]), k
        assert np.array_equal(runs[1][1], runs[0][1])
    finally:
        th.close()


@pytest.mark.gpu
def test_schedule_options_on_the_regime_domain():
    """"simple" 0 (every column through k_carries) and "graphs" 0 give the bits of the default schedule on the regime domain,
    whose T_0 + 0.1 cells sit exactly on the bound of a simple column."""
    from kid_b200.kidmp import Thompson
    st, p, dz, dt = R.regime_domain()
    res = {}
    for name, opts in (("default", {}), ("no_simple", {"simple": 0}), ("no_graph", {"graphs": 0})):
        th = Thompson(set_Nc=100.0, iiwarm=False, l_sediment=True)
        try:
            for k, v in opts.items():
                th.set_option(k, v)
            res[name] = [_device_step(th, st, p, dz, dt), _device_step(th, *R.build("sediment"))]
        finally:
            th.close()
    for name, r in res.items():
        for a, b in zip(r, res["default"]):
            _same(a, b, name)


@pytest.mark.gpu
@pytest.mark.parametrize("case", AERO_CASES, ids=str)
def test_aerosol_aware_case_parity_with_the_oracle(case, gpu_mixed, oracle_mixed):
    """kidmp_step_device_aero against oracle.step_aero on the freezing, T_0, nucleation and clamp cases, with the aerosol numbers
    at and beyond their clamps, droplet numbers over the whole nu_c range and updrafts < 0, = 0 and large."""
    st, p, dz, dt = R.build(case)
    nc, nwfa, nifa, w = R.aero_inputs(st, p, seed=len(case.name))
    ref = {k: v.copy() for k, v in st.items()}
    rnc, rnwfa, rnifa = nc.copy(), nwfa.copy(), nifa.copy()
    ppt_ref = oracle_mixed.step_aero(dt, ref, rnc, rnwfa, rnifa, p, w, dz)
    got, ppt = R.aero_step(gpu_mixed, st, p, dz, dt, nc, nwfa, nifa, w)
    ref.update(nc=rnc, nwfa=rnwfa, nifa=rnifa)
    cls, _ = R.cell_classes(st, p)
    bad = R.cell_outliers(got, ref, AERO_FIELDS, cls)
    print("REGIME aero %s: %d state outliers" % (case.name, len(bad)))
    assert len(bad) <= AERO_ALLOW.get(case.name, 0), "aero %s:\n  %s" % (case.name, "\n  ".join(bad[:20]))
    np.testing.assert_allclose(ppt, ppt_ref, rtol=1e-5, atol=1e-10, err_msg="aero %s ppt" % case.name)
