"""Effective radii of cloud water, cloud ice and snow (calc_effectRad, M:4834-4935, clamps M:1118-1122), cell by cell.

k_wrf_scatter (kid_b200/csrc/kidmp_wrf.cuh) computes the radii from the state the step leaves behind.  So the reference here is
the oracle's calc_effectRad fed with the GPU's own output state, not the oracle's step: a flipped cell of the step cannot hide
a radius error, and the radii must agree bit for bit.  pii = 1 everywhere (p still varies; the driver never ties pii to p), so
the th that comes back is, bit for bit, the t1d the radii were computed from; in the aerosol-aware call the returned nc is the
droplet number the cloud radius read.

The domain puts dense spreads across every edge of the radii, and the tests check afterwards, on the returned state, that both
sides of each edge are populated:
  * qc * rho across R1 and qi * rho across R1 (the preset radius below);
  * snow from 272.9 to 273.4 K: tc0 = min(-0.1, T - 273.15) is clamped in some cells and not in others;
  * contents and numbers whose radius falls below and above each clamp (2.51 / 50 um, 5.01 / 125 um, 10 / 999 um);
  * aerosol-aware: nc * rho below and above 100 m^-3 and on both sides of the NINT ties 1e9 / (k + 0.5), so inu_c = 3 .. 15.
After a step some edges cannot be reached, because the step clamps its own output (M:3623-3686): nc * rho <= Nt_c_max = 1999e6
(so inu_c = 2 and nc > 1e10 need a fixed Nt_c above 2e9, the set_Nc 3000 handle), ni * rho >= 8e8 * qi * rho > R2 wherever qi > R1
(the 300 um bound of the mean ice diameter); the 50 um bound of the cloud radius, which the clamp of M:1118 repeats, needs more
cloud water than one step leaves at Nt_c = 1e7 (autoconversion), or larger drops than the 100 um bound of the mean drop diameter
allows a prognostic nc (M:3636-3638: re_qc <= 47 um); the 125 um bound of the ice radius needs qi * rho > 6e-4 kg m^-3 at the
499e3 m^-3 cap of the ice number, and a mixed-phase step turns such ice into snow (qi <= 6e-4 after it, re_qi <= 112.5 um, the
300 um bound again), so only the iiwarm handle, whose step leaves the ice processes out, reaches it.
CPU test: the oracle's own step and calc_effectRad on this domain reach every branch.  GPU tests: the three driver entries
(kidmp_mp_gt_driver[_aero], kidmp_mp_gt_driver_tile with halo and k0 = 1, kidmp_mp_gt_driver_tile_device), plain and
aerosol-aware, on handles whose Nt_c gives inu_c = 12, 15, 5 (a NINT tie), 2 and 15 (through the min).
"""
import numpy as np
import pytest

import regimes as R

F = np.float32
NZ = 12
DT = 5.0
R1, R2 = F(1e-12), F(1e-6)
RE = ("re_cloud", "re_ice", "re_snow")
CLAMP = {"re_cloud": (F(2.51e-6), F(50e-6)), "re_ice": (F(5.01e-6), F(125e-6)), "re_snow": (F(10e-6), F(999e-6))}
OUTER = {"re_cloud": (F(2.49e-6), F(50e-6)), "re_ice": (F(4.99e-6), F(125e-6)), "re_snow": (F(9.99e-6), F(999e-6))}   # M:1118-1122
HANDLES = {"mixed": dict(set_Nc=100.0), "warm": dict(set_Nc=50.0, iiwarm=True),
           "nc400": dict(set_Nc=400.0), "nc3000": dict(set_Nc=3000.0), "nc10": dict(set_Nc=10.0)}
INU_C = {"mixed": 12, "warm": 15, "nc400": 5, "nc3000": 2, "nc10": 15}
# Radii allowed to differ from the oracle's by one ulp, per (handle, plain / aero, entry); the rest must be bit-identical.
# aero: one cloud radius (level 0 of column 6), where lamc = (nc * am_r * g_ratio / rc)**obmr has x = 6.613e18: glibc powf gives
# 1877008.625, the device's pow_f (f64 exp(y * log x), rounded once) 1877008.5.  It is the only cloud cell of the domain where the
# two differ (checked on the oracle's own step), and the only radius that differs on a B200, on every handle and entry.
ULP_ALLOW = {(h, "aero", e): 1 for h in HANDLES if h != "warm" for e in ("packed", "tile", "device")}


# ---- the domain ---------------------------------------------------------------------------------------------------------
def _groups():
    """(p_sfc, [cells]): each cell a dict t, qv, and any of qc qi ni qs (mixing ratios) and nc_rho (droplets per m^3)."""
    L = np.linspace
    G = np.geomspace
    out = []
    # cloud water content across R1 at rho ~ 0.45 (mixing ratios above R1 survive the input clamp, their density does not)
    out.append((4.2e4, [dict(t=F(283.0), rc=F(r), over="water") for r in L(0.55e-12, 1.6e-12, 48)]))
    # cloud water from below the lower radius clamp to the largest radii one step leaves
    out.append((9.0e4, [dict(t=F(t), qc=F(q), over="water") for t in (278.0, 288.0, 298.0) for q in G(1e-11, 1.5e-2, 36)]))
    # aerosol-aware droplet numbers: both sides of each NINT tie 1e9 / (k + 0.5) over a range of contents (the step moves nc * rho
    # by about 1e-6 relative)
    out.append((9.0e4, [dict(t=F(285.0), qc=F(q), nc_rho=1e9 / (k + 0.5) * (1.0 + j * 1e-6), over="water")
                        for k in range(1, 14) for j in (-4, -2, -1, 0, 1, 2, 4, 8) for q in (2e-5, 3e-4)]))
    # nc * rho across 100 m^-3: few large drops (the 100 um bound of the mean drop diameter sets nc from qc, M:3636-3638)
    out.append((9.0e4, [dict(t=F(285.0), rc=F(r), nc_rho=1.0, over="water") for r in G(1.5e-8, 8e-8, 36)]))
    # cloud ice: content across R1, and from the lower radius clamp (many small crystals) to the upper one (the 499e3 m^-3 cap);
    # input numbers across R2 (the step raises them to its 300 um bound)
    out.append((3.0e4, [dict(t=F(250.0), ri=F(r), ni_rho=F(1e5), over="ice") for r in L(0.55e-12, 1.6e-12, 24)]))
    out.append((5.0e4, [dict(t=F(t), qi=F(q), ni_rho=F(n), over="ice") for t in (245.0, 258.0) for q in G(1e-11, 5e-3, 24)
                        for n in (1e-7, 1.2e-6, 1e3, 4.9e5)]))
    # snow: T across 273.05 K (the tc0 clamp), and contents from the lower radius clamp to the upper one
    out.append((8.0e4, [dict(t=F(t), qs=F(q), over="water") for t in L(272.9, 273.4, 41) for q in (3e-5, 3e-4, 3e-3)]))
    out.append((6.0e4, [dict(t=F(t), qs=F(q), over="ice") for t in (250.0, 265.0) for q in G(1e-11, 3e-2, 30)]))
    return out


def radii_domain():
    """(state, p, dz, nc, nwfa, nifa, w): planes (nz, ncol) float32, the groups cut into columns of NZ cells."""
    cols = []
    dz = np.full(NZ, 200.0, np.float32)
    pz = R.pressure(dz, 1.0)
    for p_sfc, cells in _groups():
        for c0 in range(0, len(cells), NZ):
            chunk = cells[c0:c0 + NZ]
            chunk = chunk + [chunk[-1]] * (NZ - len(chunk))
            cols.append((p_sfc, chunk))
    ncol = len(cols)
    st = {k: np.zeros((NZ, ncol), np.float32) for k in R.FIELDS}
    p = np.zeros((NZ, ncol), np.float32)
    nc = np.zeros((NZ, ncol), np.float32)
    for j, (p_sfc, chunk) in enumerate(cols):
        for k, c in enumerate(chunk):
            pk = F(p_sfc * pz[k])
            t = c["t"]
            qv = R.qv_for(float(pk), t, 0.0, c["over"])
            rho = R.rho_of(pk, t, qv)
            st["t"][k, j], st["qv"][k, j], p[k, j] = t, qv, pk
            if "rc" in c:
                st["qc"][k, j] = R.q_for_r(c["rc"], float(pk), t, qv)
            if "ri" in c:
                st["qi"][k, j] = R.q_for_r(c["ri"], float(pk), t, qv)
            for f in ("qc", "qi", "qs"):
                if f in c:
                    st[f][k, j] = c[f]
            if "ni_rho" in c:
                st["ni"][k, j] = F(c["ni_rho"] / rho)
            if st["qc"][k, j] > 0:
                nc[k, j] = F(c.get("nc_rho", 1e8) / rho)
    rho = R.rho_arr(st, p)
    nwfa = np.broadcast_to(F(5e8) / rho, p.shape).astype(np.float32)
    nifa = np.broadcast_to(F(1e6) / rho, p.shape).astype(np.float32)
    w = np.zeros(p.shape, np.float32)
    return st, p, dz, nc, nwfa, nifa, w


def expected_radii(o, st, p, nc=None):
    """The oracle's calc_effectRad on a state (planes), with the clamps of M:1118-1122: dict of planes."""
    out = {k: np.zeros(st["t"].shape, np.float32) for k in RE}
    for j in range(st["t"].shape[1]):
        args = [st[k][:, j] for k in ("t",)] + [p[:, j]] + [st[k][:, j] for k in ("qv", "qc", "qi", "ni", "qs")]
        r = o.effect_rad(*args, nc=None if nc is None else nc[:, j])
        for name, v in zip(RE, r):
            lo, hi = OUTER[name]
            out[name][:, j] = np.maximum(lo, np.minimum(v, hi))
    return out


def branches(st, p, nc=None, Nt_c=None):
    """The branch of each cell in calc_effectRad, from a state in f32 as the kernel forms it: dict of boolean planes."""
    rho = R.rho_arr(st, p)
    rc, ri, rs = (np.maximum(R1, (st[f] * rho).astype(np.float32)) for f in ("qc", "qi", "qs"))
    ni = np.maximum(R2, (st["ni"] * rho).astype(np.float32))
    ncr = np.maximum(R2, (nc * rho).astype(np.float32)) if nc is not None else np.full(rho.shape, F(Nt_c))
    cloud = (rc > R1) & (ncr > R2)
    with np.errstate(divide="ignore"):
        x = (F(1000.0e6) / ncr).astype(np.float32)
    inu = np.where(ncr < F(100), 15, np.where(ncr > F(1e10), 2, np.minimum(15, np.floor(x.astype(np.float64) + 0.5) + 2)))
    tc = (st["t"] - F(273.15)).astype(np.float32)
    return {"cloud": cloud, "inu_c": np.where(cloud, inu, 0).astype(int), "nc": ncr,
            "rc_low": (st["qc"] > R1) & ~(rc > R1), "ri_low": (st["qi"] > R1) & ~(ri > R1),
            "ice": (ri > R1) & (ni > R2), "snow": rs > R1,
            "tc0_clamped": (rs > R1) & (tc > F(-0.1)), "tc0_free": (rs > R1) & ~(tc > F(-0.1))}


def _edges_reached(st, p, re, nc=None, Nt_c=None):
    """Which edges the cells of a stepped state sit on either side of: a dict name -> bool."""
    b = branches(st, p, nc, Nt_c)
    got = {"rc <= R1 < qc": b["rc_low"].any(), "rc > R1": b["cloud"].any(),
           "ri <= R1 < qi": b["ri_low"].any(), "ice": b["ice"].any(),
           "tc0 clamped": b["tc0_clamped"].any(), "tc0 free": b["tc0_free"].any()}
    for name in RE:
        lo, hi = CLAMP[name]
        sel = {"re_cloud": b["cloud"], "re_ice": b["ice"], "re_snow": b["snow"]}[name]
        v = re[name][sel]
        got[name + " at lower clamp"] = (v == lo).any()
        if name != "re_cloud":
            got[name + " at upper clamp"] = (v == hi).any()
        got[name + " inside"] = ((v > lo) & (v < hi)).any()
    return got, b


# ---- CPU: the domain reaches every branch in the oracle -------------------------------------------------------------------
@pytest.fixture(scope="module")
def oracles(oracle_mixed, oracle_warm):
    from oracle.oracle import Oracle
    out = {"mixed": oracle_mixed, "warm": oracle_warm}
    for name in ("nc400", "nc3000", "nc10"):
        out[name] = Oracle(**HANDLES[name])
    yield out
    for name in ("nc400", "nc3000", "nc10"):
        out[name].close()


def _oracle_step(o, st, p, dz, aero=None):
    s = {k: v.copy() for k, v in st.items()}
    if aero is None:
        o.step(DT, s, p, dz)
        return s, None
    nc, nwfa, nifa, w = (a.copy() for a in aero)
    o.step_aero(DT, s, nc, nwfa, nifa, p, w, dz)
    return s, nc


def test_domain_reaches_every_branch_in_the_oracle(oracles):
    st, p, dz, nc, nwfa, nifa, w = radii_domain()
    inu, seen = set(), {}
    runs = [(name, None) for name in HANDLES] + [("mixed", (nc, nwfa, nifa, w))]
    for name, aero in runs:
        o = oracles[name]
        s, ncs = _oracle_step(o, st, p, dz, aero)
        re = expected_radii(o, s, p, ncs)
        got, b = _edges_reached(s, p, re, ncs, np.float32(np.float32(HANDLES[name]["set_Nc"]) * np.float32(1e6)))
        for k, v in got.items():
            seen[k] = seen.get(k, False) or bool(v)
        inu |= set(np.unique(b["inu_c"][b["cloud"]]).tolist())
        if aero is None:
            assert set(np.unique(b["inu_c"][b["cloud"]]).tolist()) == {INU_C[name]}, name
        else:
            ncr = b["nc"][b["cloud"]]
            assert (ncr < 100).any() and (ncr > 100).any()
            # both sides of every tie k + 0.5, k = 1 .. 13
            x = (F(1000.0e6) / ncr).astype(np.float32)
            for k in range(1, 14):
                assert ((x < k + 0.5) & (x > k + 0.4)).any() and ((x > k + 0.5) & (x < k + 0.6)).any(), k
    assert inu == set(range(2, 16)), sorted(set(range(2, 16)) - inu)
    missing = [k for k, v in seen.items() if not v]
    assert not missing, missing


# ---- GPU --------------------------------------------------------------------------------------------------------------------
def _cube(a, ni, nj):
    nk = a.shape[0]
    return np.ascontiguousarray(a.reshape(nk, nj, ni).transpose(1, 0, 2))


def _planes(a):
    nj, nk, ni = a.shape
    return np.ascontiguousarray(a.transpose(1, 0, 2).reshape(nk, nj * ni))


F3 = ("qv", "qc", "qr", "qi", "qs", "qg", "ni", "nr", "th")


def _driver(th, entry, st, p, dz, aero=None):
    """One mp_gt_driver call through `entry` ('packed', 'tile': inside a memory box with a halo and k0 = 1, 'device') on the
    domain: pii = 1, so th = T.  Returns (state planes with 't' = the returned th, nc plane or None, radii planes)."""
    import torch
    nk, ncol = st["t"].shape
    ni, nj = ncol // 2, 2
    assert ni * nj == ncol
    f3 = {k: _cube(st[k], ni, nj) for k in F3 if k != "th"}
    f3["th"] = _cube(st["t"], ni, nj)
    ins = {"pii": np.ones_like(f3["th"]), "p": _cube(p, ni, nj),
           "dz": _cube(np.ascontiguousarray(np.broadcast_to(dz[:, None], (nk, ncol))), ni, nj)}
    acc = {k: np.zeros((nj, ni), np.float32) for k in ("rainnc", "rainncv", "sr", "snownc", "snowncv", "graupelnc", "graupelncv")}
    ae = None
    if aero is not None:
        ae = {k: _cube(a, ni, nj) for k, a in zip(("nc", "nwfa", "nifa", "w"), aero)}
    if entry == "tile":
        hi, hj, k0 = (2, 3), (1, 1), 1
        box = (nj + sum(hj), k0 + nk + 1, ni + sum(hi))
        s3 = (slice(hj[0], hj[0] + nj), slice(k0, k0 + nk), slice(hi[0], hi[0] + ni))
        s2 = (s3[0], s3[2])

        def embed(a):
            m = np.zeros(box if a.ndim == 3 else (box[0], box[2]), np.float32)
            m[s3 if a.ndim == 3 else s2] = a
            return m
        mf3, mins, macc = ({k: embed(v) for k, v in d.items()} for d in (f3, ins, acc))
        mae = {k: embed(v) for k, v in ae.items()} if ae is not None else None
        re = th.mp_gt_driver(DT, mf3, mins["pii"], mins["p"], mins["dz"], macc, aerosols=mae,
                             tile=(hi[0], ni, k0, nk, hj[0], nj))
        f3 = {k: v[s3] for k, v in mf3.items()}
        re = {k: v[s3] for k, v in re.items()}
        if ae is not None:
            ae = {k: v[s3] for k, v in mae.items()}
    elif entry == "packed":
        re = th.mp_gt_driver(DT, f3, ins["pii"], ins["p"], ins["dz"], acc, aerosols=ae)
    else:
        d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        df3, dins, dacc = ({k: d(v) for k, v in x.items()} for x in (f3, ins, acc))
        dae = {k: d(v) for k, v in ae.items()} if ae is not None else None
        dre = {k: torch.zeros_like(df3["th"]) for k in RE}
        torch.cuda.synchronize()
        th.mp_gt_driver_device(DT, df3, dins["pii"], dins["p"], dins["dz"], dacc, radii=dre, aerosols=dae)
        th.sync()
        f3 = {k: v.cpu().numpy() for k, v in df3.items()}
        re = {k: v.cpu().numpy() for k, v in dre.items()}
        if ae is not None:
            ae = {k: v.cpu().numpy() for k, v in dae.items()}
    out = {k: _planes(f3[k]) for k in F3 if k != "th"}
    out["t"] = _planes(f3["th"])
    return out, (_planes(ae["nc"]) if ae is not None else None), {k: _planes(v) for k, v in re.items()}


@pytest.fixture(scope="module")
def handles(gpu_mixed, gpu_warm, oracles):
    from kid_b200.kidmp import Thompson
    out = {"mixed": gpu_mixed, "warm": gpu_warm}
    for name in ("nc400", "nc3000", "nc10"):
        out[name] = Thompson(**HANDLES[name])
    yield out
    for name in ("nc400", "nc3000", "nc10"):
        out[name].close()


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["packed", "tile", "device"])
# (the aerosol-aware step is a mixed-phase scheme: not on the iiwarm handle)
@pytest.mark.parametrize("handle,aero", [(h, a) for h in HANDLES for a in (False, True) if not (a and h == "warm")],
                         ids=lambda v: {False: "plain", True: "aero"}.get(v, v) if isinstance(v, bool) else v)
def test_radii_equal_calc_effect_rad_of_the_returned_state(handle, aero, entry, handles, oracles):
    th, o = handles[handle], oracles[handle]
    st, p, dz, nc, nwfa, nifa, w = radii_domain()
    got, ncs, re = _driver(th, entry, st, p, dz, (nc, nwfa, nifa, w) if aero else None)
    want = expected_radii(o, got, p, ncs)
    Nt_c = np.float32(np.float32(HANDLES[handle]["set_Nc"]) * np.float32(1e6))
    reached, b = _edges_reached(got, p, want, ncs, Nt_c)
    if handle != "warm":
        reached.pop("re_ice at upper clamp")        # (only where the step leaves the ice alone, see the module docstring)
    missing = [k for k, v in reached.items() if not v]
    assert not missing, (handle, aero, entry, missing)
    if not aero:
        assert set(np.unique(b["inu_c"][b["cloud"]]).tolist()) == {INU_C[handle]}
    key = (handle, "aero" if aero else "plain", entry)
    nulp = 0
    for name in RE:
        a, e = re[name], want[name]
        diff = a.view(np.int32).astype(np.int64) - e.view(np.int32).astype(np.int64)
        bad = np.argwhere(diff != 0)
        print("RADII %s/%s/%s %s: %d cells differ, max %d ulp" % (key + (name, len(bad), np.abs(diff).max())))
        assert np.abs(diff).max() <= 1, "%s %s: %s" % (key, name, [(int(k), int(j), float(a[k, j]), float(e[k, j]))
                                                                    for k, j in bad[:10]])
        nulp += len(bad)
        assert (a >= OUTER[name][0]).all() and (a <= OUTER[name][1]).all()
    assert nulp <= ULP_ALLOW.get(key, 0), key
