"""CPU tests of the oracle: known-answer values derived from the reference source text (SURVEY.md
section 4), properties the reference guarantees, and the committed golden fixtures.

M: = /root/reference/module_mp_thompson09n.f90.  The reference has no tests of its own
(PARITY UNPINNED): these pins are what the oracle is anchored to.
"""
import os

import numpy as np
import pytest

from oracle import oracle as orc
from oracle.oracle import FIELDS
from kid_b200 import synth

GOLD = os.path.join(os.path.dirname(__file__), "golden", "columns.npz")


def test_gamma_exponents_and_values(oracle_mixed):
    o = oracle_mixed
    # exponents, M:485-497, M:532-543, M:467-473, M:507-524
    np.testing.assert_allclose(o.get("cre"), [4, 1, 4, 7, 2, 5, 3.5, 7, 4, 2, 3, 2.5, 8], rtol=0, atol=1e-6)
    np.testing.assert_allclose(o.get("cge"), [4, 1, 4, 7, 7.89, 4.89, 5.89, 6.89, 3.89, 2, 2.945, 2.945], rtol=0, atol=1e-6)
    np.testing.assert_allclose(o.get("cie"), [1, 4, 5, 2, 2, 3.5, 2.5], rtol=0, atol=1e-6)
    np.testing.assert_allclose(o.get("cse"), [3, 4, 4, 3.55, 5.55, 5, 3.6357, 4.6357, 5.6357, 4.1857, 6.1857, 5.6357,
                                              2.55, 2.55, 1.6357, 1.775, 3.4107, 4.1857], rtol=0, atol=2e-6)
    crg, cgg, csg = o.get("crg"), o.get("cgg"), o.get("csg")
    # gamma(n) = (n-1)! through the NR Lanczos GAMMLN (M:4598-4620) in f32
    np.testing.assert_allclose(crg[[0, 3, 12]], [6.0, 720.0, 5040.0], rtol=2e-6)
    np.testing.assert_allclose(crg[[6, 11]], [3.3233511, 1.3293403], rtol=2e-6)
    np.testing.assert_allclose(cgg[[4, 5, 8, 10]], [4041.009, 20.363228, 5.2347646, 1.9021707], rtol=3e-6)
    np.testing.assert_allclose(csg[[3, 9, 12, 15]], [3.5132518, 7.612799, 1.377746, 0.9249857], rtol=3e-6)


def test_scalar_constants(oracle_mixed):
    s = oracle_mixed.get("scalars")
    Nt_c, Sc3, D0i, xm0s, xm0g, rho_not, t1_qr_qc, t1_qr_qi, t2_qr_qi, t1_qg_qc = s[:10]
    assert Nt_c == 100.0e6                                             # M:381
    np.testing.assert_allclose(Sc3, 0.85816807, rtol=1e-6)             # M:442
    np.testing.assert_allclose(D0i, 1.28984e-5, rtol=1e-5)             # M:445
    np.testing.assert_allclose(xm0s, 2.76e-9, rtol=1e-6)
    np.testing.assert_allclose(xm0g, 4.09062e-9, rtol=1e-5)
    np.testing.assert_allclose(rho_not, 1.1845211, rtol=1e-6)          # M:141
    np.testing.assert_allclose(t1_qr_qc, 22873.94, rtol=1e-6)          # M:560
    np.testing.assert_allclose(t2_qr_qi, 1.437212e9, rtol=1e-5)        # M:562
    np.testing.assert_allclose(t1_qg_qc, 1817.2275, rtol=2e-6)         # M:565
    np.testing.assert_allclose(s[13], 36.830105, rtol=2e-6)            # t2_qr_ev, M:575
    off = oracle_mixed.get("offsets")
    assert list(off.astype(int)) == [7, -6, -10, 0, -6, 6, -5, -5, 4, 0]   # nic1, nic2 ... niIN2, M:594-602, M:670


def test_bins(oracle_mixed):
    Dr, tN = oracle_mixed.get("Dr"), oracle_mixed.get("t_Nc")
    np.testing.assert_allclose(Dr[0], 5.1165e-5, rtol=1e-4)            # M:625-634
    np.testing.assert_allclose(Dr[99], 4.8862e-3, rtol=1e-4)
    np.testing.assert_allclose(tN[0], 1.0408e6, rtol=1e-4)
    assert np.all(np.diff(Dr) > 0)
    # geometric grid: constant ratio
    np.testing.assert_allclose(Dr[1:] / Dr[:-1], (0.005 / 50e-6) ** 0.01, rtol=1e-6)


def test_saturation(oracle_mixed):
    np.testing.assert_allclose(orc.rslf(1e5, 293.15), 0.0148923, rtol=1e-5)      # M:4656-4686
    np.testing.assert_allclose(orc.rslf(8e4, 273.15), 0.00478818, rtol=1e-5)
    np.testing.assert_allclose(orc.rsif(5e4, 253.15), 0.00128693, rtol=1e-5)     # M:4688-4717
    np.testing.assert_allclose(orc.rsif(3e4, 233.15), 0.000266049, rtol=1e-5)
    # ice saturation below water saturation under 0 C
    assert orc.rsif(6e4, 263.15) < orc.rslf(6e4, 263.15)


def test_decade_index():
    L = orc.lib()
    # r_r axis: 1e-6..1e-2, 37 nodes, nir2 = -6 (M:235-240, M:1840-1852)
    assert L.kor_decade_index(1.5e-6, -6, 37) == 1
    assert L.kor_decade_index(9.99e-6, -6, 37) == 9
    assert L.kor_decade_index(1.0e-5, -6, 37) in (9, 10)      # exactly on a decade: f32 rounding decides
    assert L.kor_decade_index(3.3e-4, -6, 37) == 9 * 2 + 3
    assert L.kor_decade_index(0.5, -6, 37) == 37              # clamped
    # monotone non-decreasing over the axis
    xs = np.exp(np.linspace(np.log(1.1e-6), np.log(9e-3), 4000)).astype(np.float32)
    idx = np.array([L.kor_decade_index(float(x), -6, 37) for x in xs])
    assert np.all(np.diff(idx) >= 0) and idx.min() == 1 and idx.max() <= 37


def test_tables_properties(oracle_mixed):
    o = oracle_mixed
    ef = o.get("t_Efrw")
    Dr, Dc = o.get("Dr"), o.get("Dc")
    assert ef.min() >= 0.0 and ef.max() <= 0.95 + 1e-7                               # M:4294
    assert np.all(ef[:, Dc < 3e-6] == 0.0) and np.all(ef[Dr < 50e-6, :] == 0.0)     # M:4256-4257
    ide = o.get("tpi_ide")
    assert ide.min() >= 0.0 and ide.max() <= 1.0                                     # M:4209-4219
    r_r = np.array([m * 10.0 ** d for d in range(-6, -2) for m in range(1, 10)] + [1e-2], np.float32)
    tmr = o.get("tmr_racg")                                                          # (g1, g, r1, r)
    assert np.all(tmr <= r_r[None, None, None, :].astype(np.float64) * (1 + 1e-12))  # M:3802
    # freezing probability grows as it gets colder (third axis = -T), M:4118-4150
    tpg = o.get("tpg_qrfz")
    assert np.all(np.diff(tpg, axis=2) >= -1e-30)
    # the sacr1 family is identically zero: a snowflake heavier than 2/3 of the drop never falls slower (M:3998-4028)
    assert not o.get("tcr_sacr1").any()


def _col(st, p, j):
    return [st[k][:, j].copy() for k in FIELDS], p[:, j].copy()


def test_no_micro_columns_unchanged(oracle_mixed):
    st, p, dz = synth.make_domain(512, nz=60, cloudy_fraction=0.0, coherent=False)
    ref = {k: v.numpy().copy() for k, v in st.items()}
    new = {k: v.copy() for k, v in ref.items()}
    ppt = oracle_mixed.step(10.0, new, p.numpy(), dz.numpy())
    for k in FIELDS:
        assert np.array_equal(new[k], ref[k]), k                        # early RETURN at M:1540 (U9)
    assert not ppt.any()


def test_warm_leaves_ice_untouched(oracle_warm):
    st, p, dz = synth.make_domain(256, nz=60, cloudy_fraction=1.0, coherent=False)
    ref = {k: v.numpy().copy() for k, v in st.items()}
    new = {k: v.copy() for k, v in ref.items()}
    oracle_warm.step(10.0, new, p.numpy(), dz.numpy())
    for k in ("qs", "qg"):
        assert np.array_equal(new[k], ref[k]), k                        # iiwarm gates S3/S4/S6/S10/S15
    assert not np.array_equal(new["qr"], ref["qr"])


def test_output_clamps(oracle_mixed):
    st, p, dz = synth.make_domain(512, nz=60, cloudy_fraction=1.0, coherent=False)
    new = {k: v.numpy().copy() for k, v in st.items()}
    oracle_mixed.step(10.0, new, p.numpy(), dz.numpy())
    assert new["qv"].min() >= 1e-10                                      # M:3624
    for k in ("qc", "qi", "qr", "qs", "qg"):
        q = new[k]
        assert np.all((q == 0) | (q > 1e-12)), k                         # M:3628-3685
    assert np.all(new["ni"][new["qi"] == 0] == 0) and np.all(new["nr"][new["qr"] == 0] == 0)
    rho = 0.622 * p.numpy() / (287.04 * new["t"] * (new["qv"] + 0.622))
    assert np.all(new["ni"] * rho <= 499e3 * 1.001)                      # M:3650
    assert np.isfinite(np.stack([new[k] for k in FIELDS])).all()


def test_water_budget(oracle_mixed):
    # total water (vapour + condensate) + surface precipitation is conserved up to the clamp leaks
    st, p, dz = synth.make_domain(256, nz=60, cloudy_fraction=1.0, coherent=False)
    old = {k: v.numpy().astype(np.float64) for k, v in st.items()}
    new32 = {k: v.numpy().copy() for k, v in st.items()}
    ppt = oracle_mixed.step(10.0, new32, p.numpy(), dz.numpy()).astype(np.float64)
    new = {k: v.astype(np.float64) for k, v in new32.items()}
    pn, dzn = p.numpy().astype(np.float64), dz.numpy().astype(np.float64)[:, None]

    def column_water(s):
        rho = 0.622 * pn / (287.04 * s["t"] * (s["qv"] + 0.622))
        return ((s["qv"] + s["qc"] + s["qr"] + s["qi"] + s["qs"] + s["qg"]) * rho * dzn).sum(0)
    before, after = column_water(old), column_water(new) + ppt.sum(0)
    # air density changes with the latent heating at fixed pressure, so the budget closes to ~1e-3
    np.testing.assert_allclose(after, before, rtol=5e-3)


def test_golden_fixtures_reproduced():
    g = np.load(GOLD)
    p, dz = g["in/p"], g["in/dz"]
    for tag, kw, dt in (("mixed_dt10", dict(set_Nc=100.0, iiwarm=False), 10.0),
                        ("warm_dt10", dict(set_Nc=50.0, iiwarm=True), 10.0),
                        ("nosed_dt10", dict(set_Nc=300.0, iiwarm=False, l_sediment=False), 10.0)):
        o = orc.Oracle(**kw)
        s = {k: g["in/" + k].copy() for k in FIELDS}
        ppt = o.step(dt, s, p.copy(), dz)
        for k in FIELDS:
            assert np.array_equal(s[k], g["%s/%s" % (tag, k)]), (tag, k)
        assert np.array_equal(ppt, g[tag + "/ppt"])
        o.close()


def test_single_column_equals_batched(oracle_mixed):
    g = np.load(GOLD)
    j = 3
    out = oracle_mixed.column(10.0, *[g["in/" + k][:, j] for k in FIELDS], g["in/p"][:, j], g["in/dz"])
    for k in FIELDS:
        assert np.array_equal(out[k], g["mixed_dt10/" + k][:, j]), k
    # layouts: K_FASTEST (KiD (k,i)) and COL_FASTEST give the same numbers
    s = {k: np.ascontiguousarray(g["in/" + k].T) for k in FIELDS}
    oracle_mixed.step(10.0, s, np.ascontiguousarray(g["in/p"].T), g["in/dz"], layout="k_fastest")
    for k in FIELDS:
        assert np.array_equal(s[k].T, g["mixed_dt10/" + k]), k


def test_rates_buffer(oracle_mixed):
    g = np.load(GOLD)
    j = 0
    out = oracle_mixed.column(10.0, *[g["in/" + k][:, j] for k in FIELDS], g["in/p"][:, j], g["in/dz"], want_rates=True)
    assert out["rates"].shape == (36, 60) and len(oracle_mixed.rate_names) == 36
    assert np.isfinite(out["rates"]).all() and np.abs(out["rates"]).max() > 0


# ---- calc_effectRad (M:4834-4935) and the mp_gt_driver algebra (M:986-1003, M:1110-1123) -------------------------
def test_effective_radii_known_answers(oracle_mixed):
    """Source-derived values: with is_aerosol_aware = .false. the droplet number is Nt_c (M:4875); for Nt_c = 100 cm^-3
    inu_c = MIN(15, NINT(1000.E6/Nt_c) + 2) = 12 and lamc = (Nt_c*am_r*g_ratio(12)/rc)**obmr (M:4892-4897), so the
    cloud radius is 0.5*(3+12)/lamc; the ice radius is 0.5*(3+mu_i)/lami with lami of M:4902; cells without the
    species keep the presets of M:1112-1114."""
    o = oracle_mixed
    nz = 6
    t = np.array([290., 285., 270., 255., 240., 225.], np.float32)
    p = np.array([9.5e4, 9.0e4, 7.0e4, 5.5e4, 4.0e4, 3.0e4], np.float32)
    qv = np.full(nz, 5e-3, np.float32)
    qc = np.array([0., 1e-3, 2e-4, 0., 0., 0.], np.float32)
    qi = np.array([0., 0., 0., 1e-5, 5e-5, 1e-6], np.float32)
    ni = np.array([0., 0., 0., 5e3, 2e4, 1e3], np.float32)
    qs = np.array([0., 0., 1e-4, 5e-4, 1e-3, 0.], np.float32)
    rc, ri, rs = o.effect_rad(t, p, qv, qc, qi, ni, qs)
    rho = 0.622 * p.astype(np.float64) / (287.04 * t * (qv + 0.622))
    am_r, am_i = np.pi * 1000.0 / 6.0, np.pi * 890.0 / 6.0
    g12 = 2730.0                                             # g_ratio(12), M:4857 (= (nu+3)(nu+2)(nu+1)... for nu = 12)
    for k in range(nz):
        if qc[k] > 0:
            lamc = (100.0e6 * am_r * g12 / (qc[k] * rho[k])) ** (1.0 / 3.0)
            want = min(max(0.5 * 15.0 / lamc, 2.51e-6), 50e-6)
            assert abs(rc[k] - want) / want < 1e-5
        else:
            assert rc[k] == np.float32(2.49e-6)
        if qi[k] > 0:
            lami = (am_i * 6.0 * ni[k] / qi[k]) ** (1.0 / 3.0)   # cig(2)*oig1 = Gamma(4)/Gamma(1) = 6 (mu_i = 0, bm_i = 3)
            want = min(max(0.5 * 3.0 / lami, 5.01e-6), 125e-6)
            assert abs(ri[k] - want) / want < 1e-5
        else:
            assert ri[k] == np.float32(4.99e-6)
        if qs[k] > 0:
            # M:4911-4946: 0.5 * M3/M2 with the Field et al. (2005) moment relation for order cse(1) = bm_s + 1 = 3
            sa = [5.065339, -0.062659, -3.032362, 0.029469, -0.000285, 0.31255, 0.000204, 0.003199, 0.0, -0.015952]
            sb = [0.476221, -0.015896, 0.165977, 0.007468, -0.000141, 0.060366, 0.000079, 0.000594, 0.0, -0.003577]
            tc0, c = min(-0.1, float(t[k]) - 273.15), 3.0
            poly = lambda s: (s[0] + s[1] * tc0 + s[2] * c + s[3] * tc0 * c + s[4] * tc0 * tc0 + s[5] * c * c
                              + s[6] * tc0 * tc0 * c + s[7] * tc0 * c * c + s[8] * tc0 ** 3 + s[9] * c ** 3)
            smob = qs[k] * rho[k] / 0.069
            want = min(max(0.5 * 10.0 ** poly(sa) * smob ** poly(sb) / smob, 10e-6), 999e-6)
            assert abs(rs[k] - want) / want < 2e-4, (k, rs[k], want)
        else:
            assert rs[k] == np.float32(9.99e-6)


def test_wrf_driver_algebra_on_the_oracle(oracle_mixed):
    """mp_gt_driver around one column equals mp_thompson on T = th*pii with that column's dz, th = T/pii back,
    and the accumulator formulas of M:990-1003."""
    from kid_b200 import synth
    o = oracle_mixed
    st, p, dz = synth.deep_column(nz=40)
    nk = 40
    pii = ((p / 1.0e5) ** (287.04 / 1004.0)).astype(np.float32)
    f3 = {k: st[k].reshape(1, nk, 1).copy() for k in ("qv", "qc", "qr", "qi", "qs", "qg", "ni", "nr")}
    f3["th"] = (st["t"] / pii).astype(np.float32).reshape(1, nk, 1)
    t_in = (f3["th"].reshape(nk) * pii).astype(np.float32)
    dz3 = (dz * np.float32(1.1)).astype(np.float32).reshape(1, nk, 1)
    acc = {k: np.full((1, 1), v, np.float32) for k, v in
           (("rainnc", 2.0), ("rainncv", 9.0), ("sr", 9.0), ("snownc", 1.0), ("snowncv", 9.0), ("graupelnc", 0.5), ("graupelncv", 9.0))}
    re = o.mp_gt_driver(15.0, f3, pii.reshape(1, nk, 1), p.reshape(1, nk, 1), dz3, acc)
    ref = o.column(15.0, st["qv"], st["qc"], st["qi"], st["qr"], st["qs"], st["qg"], st["ni"], st["nr"], t_in, p, dz3.reshape(nk))
    for k in ("qv", "qc", "qr", "qi", "qs", "qg", "ni", "nr"):
        assert np.array_equal(f3[k].reshape(nk), ref[k]), k
    assert np.array_equal(f3["th"].reshape(nk), (ref["t"] / pii).astype(np.float32))
    rain, ice, snow, grau = [np.float32(x) for x in ref["ppt"]]
    ncv = np.float32(np.float32(np.float32(rain + snow) + grau) + ice)
    assert acc["rainncv"][0, 0] == ncv
    assert acc["rainnc"][0, 0] == np.float32(np.float32(np.float32(np.float32(np.float32(2.0) + rain) + snow) + grau) + ice)
    assert acc["snowncv"][0, 0] == np.float32(snow + ice) and acc["graupelncv"][0, 0] == grau
    assert acc["sr"][0, 0] == np.float32(np.float32(np.float32(snow + grau) + ice) / np.float32(ncv + np.float32(1e-12)))
    rc, ri, rs = o.effect_rad(ref["t"], p, ref["qv"], ref["qc"], ref["qi"], ref["ni"], ref["qs"])
    assert np.array_equal(re["re_cloud"].reshape(nk), np.clip(rc, np.float32(2.49e-6), np.float32(50e-6)))
    assert np.array_equal(re["re_ice"].reshape(nk), np.clip(ri, np.float32(4.99e-6), np.float32(125e-6)))
    assert np.array_equal(re["re_snow"].reshape(nk), np.clip(rs, np.float32(9.99e-6), np.float32(999e-6)))


def test_decade_index_shortcut_of_the_kernels_equals_the_reference_search():
    """The kernels' decade-mantissa index (kidmp_column.cuh decade_idx_f: a bit-level guess of the decade, ONE division when
    the quotient is well inside [1, 10), the reference's three-candidate search otherwise) restated in float32 numpy,
    against the oracle's restatement of M:1762-1774 - on random values and on the ulps around every decade boundary."""
    from oracle.oracle import lib
    L = lib()

    def powi10(m):                                   # libgcc __powisf2, as kidmp_hostinit.h
        n = abs(m)
        x = np.float32(10.0)
        y = x if n % 2 else np.float32(1.0)
        n >>= 1
        while n:
            x = np.float32(x * x)
            if n % 2:
                y = np.float32(y * x)
            n >>= 1
        return np.float32(1.0) / y if m < 0 else y
    p10 = np.array([powi10(n) for n in range(-32, 32)], np.float32)

    def kernel_index(x, n2, ntb):
        x = np.float32(x)
        b = int(x.view(np.int32))
        l2 = np.float32(np.float32((b >> 23) - 127) + np.int32((b & 0x007fffff) | 0x3f800000).view(np.float32) - np.float32(1.0))
        n0 = int(np.rint(np.float32(l2 * np.float32(0.30103))))
        q0 = np.float32(x / p10[n0 + 32])
        n, qn = n0, q0
        if not (q0 > np.float32(1.00001) and q0 < np.float32(9.9999)):
            n = n0 + 1
            for nn in (-1, 0, 1):
                q = np.float32(x / p10[n0 + nn + 32])
                if q >= 1.0 and q < 10.0:
                    n = n0 + nn
                    break
            qn = np.float32(x / p10[n + 32])
        return max(1, min(int(qn) + 9 * (n - n2), ntb))

    rng = np.random.default_rng(5)
    vals = list(np.exp(rng.uniform(np.log(1e-9), np.log(1e7), 40000)).astype(np.float32))
    for d in range(-9, 8):                           # every float within 40 ulps of 10**d, and of 10**d as powi builds it
        for c in (np.float32(10.0) ** d, powi10(d)):
            base = int(np.float32(c).view(np.int32))
            vals += [np.int32(base + k).view(np.float32) for k in range(-40, 41)]
    bad = 0
    for x in vals:
        for n2, ntb in ((-6, 37), (-10, 64), (-2, 55)):
            if kernel_index(x, n2, ntb) != L.kor_decade_index(float(x), n2, ntb):
                bad += 1
    assert bad == 0, bad


def _horner_f32(c, x):
    """The Horner form of RSLF / RSIF (M:4656-4717) in f32, operation by operation like the kernels (no FMA)."""
    acc = np.full_like(x, np.float32(c[8]))
    for q in range(7, -1, -1):
        acc = (np.float32(c[q]) + x * acc).astype(np.float32)
    return acc


def test_saturation_over_ice_not_above_liquid():
    """k_classify marks a cell busy when it holds a hydrometeor or ssati > 0; the cell code would also run rates for
    ssatw > eps (M:2780).  At or below 0 C that adds nothing because e_s(ice) <= e_s(liquid) for the two polynomials over
    their whole argument range [-80, -0.01] C - checked here for EVERY f32 temperature in that range - and
    0.622 e / (p - e) and q / qvs - 1 are monotone in round-to-nearest arithmetic."""
    CL = [.611583699E03, .444606896E02, .143177157E01, .264224321E-1, .299291081E-3, .203154182E-5, .702620698E-8,
          .379534310E-11, -.321582393E-13]
    CI = [.609868993E03, .499320233E02, .184672631E01, .402737184E-1, .565392987E-3, .521693933E-5, .307839583E-7,
          .105785160E-9, .161444444E-12]
    lo, hi = np.float32(193.0).view(np.uint32), np.float32(273.15).view(np.uint32)
    worst = np.inf
    for b0 in range(int(lo), int(hi) + 1, 1 << 20):
        t = np.arange(b0, min(b0 + (1 << 20), int(hi) + 1), dtype=np.uint32).view(np.float32)
        x = np.maximum(np.float32(-80.0), (t - np.float32(273.16)).astype(np.float32))
        esl, esi = _horner_f32(CL, x), _horner_f32(CI, x)
        worst = min(worst, float((esl - esi).min()))
        assert (esi <= esl).all()
    assert worst >= 0.0
    # spot check of the helpers against the oracle's RSLF / RSIF
    for tt in (200.0, 233.15, 260.0, 273.15):
        x = np.maximum(np.float32(-80.0), np.float32(tt) - np.float32(273.16))
        e = float(_horner_f32(CL, np.array([x], np.float32))[0])
        pp = np.float32(50000.0)
        e = min(np.float32(e), pp * np.float32(0.15))
        assert np.float32(np.float32(0.622) * e / (pp - e)) == np.float32(orc.rslf(50000.0, tt))


def test_cell_class_rule_covers_every_species_set():
    """The rule of cell_kernel_class (kid_b200/csrc/kidmp_column.cuh): every (species set, cold, iiwarm) combination goes to a
    class whose kernel may hold those species (CellTraits of kidmp_cells.cuh)."""
    from regimes import QC, QI, QR, QS, QG, kernel_class as rule
    allowed = {"WARM": QC | QR, "ICE": QI | QS, "MIXNR": QC | QI | QS | QG, "FULL": 31}
    for sp in range(32):
        for cold in (False, True):
            for iiwarm in (False, True):
                kc = rule(sp, cold, iiwarm)
                assert sp & ~allowed[kc] == 0, (sp, cold, iiwarm, kc)
                if kc == "WARM" and not iiwarm:
                    assert not cold          # no freezing or nucleation can start in a cell of this class (M:2025)
                if kc == "ICE":
                    assert cold and not iiwarm


# ---- the aerosol-aware half (is_aerosol_aware = .true., M:28): functions and table, from the source text --------------------
def test_aerosol_functions_known_answers():
    """Eff_aero M:4354-4390, iceDeMott M:4720-4756, iceKoop M:4764-4789, activ_ncloud M:4451-4526 against the same formulas
    written out in float64 numpy (independent arithmetic: agreement to f32 rounding, 1e-5)."""
    PI, meanPath, boltz = 3.1415926536, 0.0256e-6, 1.3806503e-23

    def eff(D, Da, visc, rhoa, T, sp):
        vt = {"r": -0.1021 + 4.932e3 * D - 0.9551e6 * D**2 + 0.07934e9 * D**3 - 0.002362e12 * D**4,
              "s": 40.0 * D**0.55, "g": 442.0 * D**0.89}[sp]
        Cc = 1.0 + 2.0 * meanPath / Da * (1.257 + 0.4 * np.exp(-0.55 * Da / meanPath))
        diff = boltz * T * Cc / (3.0 * PI * visc * Da)
        Re, Sc = 0.5 * rhoa * D * vt / visc, visc / (rhoa * diff)
        St = Da * Da * vt * 1000.0 / (9.0 * visc * D)
        aval = 1.0 + np.log(1.0 + Re)
        St2 = (1.2 + 1.0 / 12.0 * aval) / (1.0 + aval)
        E = 4.0 / (Re * Sc) * (1.0 + 0.4 * np.sqrt(Re) * Sc**0.3333 + 0.16 * np.sqrt(Re) * np.sqrt(Sc)) \
            + 4.0 * Da / D * (0.02 + Da / D * (1.0 + 2.0 * np.sqrt(Re)))
        if St > St2:
            E += ((St - St2) / (St - St2 + 0.666667))**1.5
        return max(1e-5, min(E, 1.0))

    for D, Da, visc, rhoa, T, sp in ((1.0e-3, 0.04e-6, 1.7e-5, 1.0, 280.0, "r"), (3.0e-3, 0.8e-6, 1.8e-5, 1.1, 290.0, "r"),
                                     (5.0e-4, 0.04e-6, 1.6e-5, 0.8, 260.0, "s"), (2.0e-3, 0.8e-6, 1.6e-5, 0.7, 255.0, "s"),
                                     (2.0e-3, 0.04e-6, 1.6e-5, 0.8, 260.0, "g"), (6.0e-3, 0.8e-6, 1.5e-5, 0.6, 250.0, "g")):
        got = orc.eff_aero(D, Da, visc, rhoa, T, sp)
        assert 1e-5 <= got <= 1.0
        np.testing.assert_allclose(got, eff(D, Da, visc, rhoa, T, sp), rtol=2e-5, err_msg=str((D, Da, sp)))
    # the big, slow-diffusing aerosol is collected more efficiently by large drops than the small one is by Brownian motion here
    assert orc.eff_aero(3.0e-3, 0.8e-6, 1.8e-5, 1.1, 290.0, "r") > orc.eff_aero(3.0e-3, 0.04e-6, 1.8e-5, 1.1, 290.0, "r") * 0.1

    rho_not0 = 101325.0 / (287.05 * 273.15)
    for tempc, rho, nifa in ((-20.0, 0.8, 1.0e6), (-35.0, 0.5, 5.0e4), (-10.0, 1.0, 2.0e6)):
        cc = nifa * rho_not0 * 1e-6 / rho
        want = 5.94e-5 * (-tempc)**3.33 * cc**(-0.0264 * tempc + 0.0033) * rho / rho_not0 * 1000.0
        np.testing.assert_allclose(orc.ice_demott(tempc, rho, nifa), want, rtol=2e-5)
    assert orc.ice_demott(-20.0, 0.8, 1.0e6) > orc.ice_demott(-10.0, 0.8, 1.0e6) > 0.0          # colder: more nuclei

    def koop(temp, qv, qvs, naero, dt):
        satw = qv / qvs
        mu = 210368.0 + 131.438 * temp - 3.32373e6 / temp - 41729.1 * np.log(temp)
        a_w_i = np.exp(mu / (8.314 * temp))
        d = satw - a_w_i
        logJ = min(20.0, -906.7 + 8502.0 * d - 26924.0 * d * d + 29180.0 * d**3)
        prob = min(1.0 - np.exp(-(10.0**logJ) * (4.0 / 3.0 * PI * 2.5e-6**3) * dt), 1.0)
        return max(0.0, min(prob * naero, 1000.0e3)) if prob > 0 else 0.0

    # (the rate goes from 0 to the cap over a few hundredths of saturation ratio: cases on the ramp, below and above it)
    a_w_i_230 = float(np.exp((210368.0 + 131.438 * 230.0 - 3.32373e6 / 230.0 - 41729.1 * np.log(230.0)) / (8.314 * 230.0)))
    for temp, satw, naero, dt in ((230.0, a_w_i_230 + 0.30, 3.0e8, 10.0), (230.0, a_w_i_230 + 0.305, 3.0e8, 10.0),
                                  (230.0, a_w_i_230 + 0.20, 3.0e8, 10.0), (225.0, 1.05, 1.0e8, 60.0)):
        want = koop(temp, satw * 1.0e-4, 1.0e-4, naero, dt)
        got = orc.ice_koop(temp, np.float32(satw * 1.0e-4), 1.0e-4, naero, dt)
        if 0.0 < want < 1000.0e3:
            # log_J_rate is a difference of f32 terms of size 900 (rounding 6e-5 each) and satw an f32 quotient: 10**x turns a few
            # hundredths of log_J_rate into tens of per cent, on a ramp that spans thirty decades
            np.testing.assert_allclose(got, want, rtol=0.3)
        else:
            assert got == want
    assert orc.ice_koop(230.0, 0.5e-4, 1.0e-4, 3.0e8, 10.0) == 0.0                                # far below the activity threshold

    # tnccn_act is all ones in this reference (M:752-762): the activated number is the CCN number up to the rounding of the
    # bilinear weights
    for T, W, N in ((280.0, 0.5, 3.0e8), (250.0, 0.001, 5.0e6), (300.0, 50.0, 2.0e10), (270.0, -1.0, 1.0e8)):
        np.testing.assert_allclose(orc.activ_ncloud(T, W, N), N, rtol=3e-6)


def test_drop_evaporation_table(oracle_mixed):
    """table_dropEvap M:4400-4439: tnc_wev(i,j,k) is the running sum over the first i diameter bins of the droplet spectrum with
    number t_Nc(k) and content r_c(j): non-decreasing in i, and its last entry is (nearly) the whole number."""
    o = oracle_mixed
    tnc = o.get("tnc_wev").reshape(100, 37, 100, order="F")
    tpc = o.get("tpc_wev").reshape(100, 37, 100, order="F")
    assert np.isfinite(tnc).all() and (tnc >= 0).all() and (np.diff(tnc, axis=0) >= 0).all()
    assert (np.diff(tpc, axis=0) >= 0).all()
    t_Nc = o.get("t_Nc")
    # droplet spectra that lie inside the bin range integrate to their number and to their mass
    j, k = 20, 50
    np.testing.assert_allclose(tnc[-1, j, k], t_Nc[k], rtol=2e-2)
    r_c = 10.0 ** np.floor(np.arange(37) / 9.0 - 6.0) * (np.arange(37) % 9 + 1)                      # M:215-221 (1e-6 .. 1e-2)
    np.testing.assert_allclose(tpc[-1, j, k], r_c[j], rtol=3e-2)


def test_aerosol_aware_oracle_properties(oracle_mixed):
    """mp_thompson with is_aerosol_aware = .true. on the oracle: clear-sky columns stay bit for bit as they were (M:1540, the
    aerosol arrays too), the aerosol numbers stay inside their clamps (M:3628-3631), nc is zero exactly where there is no cloud
    water (M:3633-3635) and below Nt_c_max / rho elsewhere (M:3646), and without any aerosol-specific process active (no cloud,
    rain, snow, graupel; warm) the other fields are those of the default scheme."""
    st, p, dz = synth.make_domain(1500, nz=60, nx=1024, col0=123456, cloudy_fraction=0.5, coherent=False)
    nc, nwfa, nifa, w = synth.make_aerosols(st, p)
    ref = {k: v.numpy().copy() for k, v in st.items()}
    before = {k: v.copy() for k, v in ref.items()}
    a0 = (nc.copy(), nwfa.copy(), nifa.copy())
    pn = p.numpy().copy()
    oracle_mixed.step_aero(10.0, ref, nc, nwfa, nifa, pn, w, dz.numpy().copy())
    base = {k: v.copy() for k, v in before.items()}
    oracle_mixed.step(10.0, base, pn, dz.numpy().copy())
    clear = np.ones(1500, bool)
    for k in FIELDS:
        clear &= (base[k] == before[k]).all(0)
    assert clear.sum() > 100
    for k in FIELDS:
        assert np.array_equal(ref[k][:, clear], before[k][:, clear]), k
    for got, was in zip((nc, nwfa, nifa), a0):
        assert np.array_equal(got[:, clear], was[:, clear])
    rho = (np.float32(0.622) * pn / (np.float32(287.04) * ref["t"] * (ref["qv"] + np.float32(0.622))))
    cloudy = ~clear
    assert (nwfa[:, cloudy] * rho[:, cloudy] >= 11.1e6 * 0.999).all() and (nwfa[:, cloudy] * rho[:, cloudy] <= 9999.0e6 * 1.001).all()
    assert (nifa[:, cloudy] >= 0.5e6 * 0.01 * 0.999).all() and (nifa[:, cloudy] * rho[:, cloudy] <= 9999.0e6 * 1.001).all()
    assert ((nc == 0) == (ref["qc"] == 0))[:, cloudy].all()
    assert (nc[:, cloudy] * rho[:, cloudy] <= 1999.0e6 * 1.001).all()
    assert not any(np.isnan(ref[k]).any() for k in FIELDS)
