"""Directed cases for the parity tests: columns placed on the thresholds, clamps and table edges of the step.

The synthetic domains of kid_b200/synth.py keep clear of the scheme's edges (no cloud water below 236 K, rain only in warm
air, moderate drop and crystal sizes, humidity near saturation), so some branches of the cell kernels never run in them, or
run in too few cells for a domain-wide outlier allowance to notice.  Every case here aims at one such regime.  A case is
  * a seeded, deterministic builder of (state, p, dz, dt), fields (nz, ncol) float32 in the device layout;
  * a target that the oracle must show on it: a process rate that is non-zero (or zero) in named cells, or a property of
    the state after the step;
  * the cell-kernel classes its busy cells fall in (cell_kernel_class of kid_b200/csrc/kidmp_column.cuh).
Each case has two kinds of column: PROBE columns (a few busy levels in an otherwise clear column: sedimentation carries the
result into idle cells below) and UNIFORM columns (every level in the regime).  The values spread over the columns include
the exact f32 threshold and np.nextafter on each side of it.  tests/test_regimes.py checks the claims on the CPU and
compares the CUDA step with the oracle case by case on the GPU; tests/test_configurations.py does the same under every handle
configuration.  The device-step helpers and the cell-by-cell outlier reports both use are at the end of this module.
M: = module_mp_thompson09n.f90.
"""
import numpy as np

from oracle import oracle as orc
from parity_util import FLOOR, REL_TOL

F = np.float32
FIELDS = ("qv", "qc", "qi", "qr", "qs", "qg", "ni", "nr", "t")
T_0, HGFR, R1, EPS = F(273.15), F(235.16), F(1e-12), F(1e-15)
R_C1 = R_R1 = F(1e-6)                     # first bins of r_c, r_r (kg m^-3), M:504-520
R_S1 = R_G1 = F(1e-5)                     # first bins of r_s, r_g
R_LAST = F(1e-2)                          # last bin of r_r, r_s, r_g
NZ = 32
PROBE = (NZ - 8, NZ - 7, NZ - 6)          # the busy levels of a probe column


def up(x):
    return np.nextafter(F(x), F(np.inf))


def down(x):
    return np.nextafter(F(x), F(-np.inf))


def rho_of(p, t, qv):
    """Air density exactly as the scheme forms it in f32 (M:1387)."""
    return F(F(F(0.622) * F(p)) / F(F(F(287.04) * F(t)) * F(F(qv) + F(0.622))))


# ---- the rule of cell_kernel_class (kid_b200/csrc/kidmp_column.cuh), shared with test_oracle_kat.py ------------------------
QC, QI, QR, QS, QG = 1, 2, 4, 8, 16
CLASSES = ("WARM", "ICE", "MIXNR", "FULL")


def kernel_class(sp, cold, iiwarm):
    ice = bool(sp & (QI | QS | QG))
    if iiwarm:
        return "FULL" if ice else "WARM"
    if not cold and not ice:
        return "WARM"
    if cold and not (sp & (QC | QR | QG)):
        return "ICE"
    return "FULL" if sp & QR else "MIXNR"


def classify(st, p):
    """The class byte of k_classify (kid_b200/csrc/kidmp_column.cuh) in numpy: (species bits, cold, busy) per cell.
    Saturation through the oracle's RSLF / RSIF, in f32 like the kernel."""
    sp = np.zeros(st["t"].shape, np.int64)
    for bit, k in ((QC, "qc"), (QI, "qi"), (QR, "qr"), (QS, "qs"), (QG, "qg")):
        sp |= np.where(st[k] > R1, bit, 0)
    t, qv = st["t"], np.maximum(F(1e-10), st["qv"])
    cold = t < T_0
    busy = sp != 0
    for k, j in zip(*np.nonzero(sp == 0)):
        tc = F(t[k, j] - F(273.15))
        qvsi = F(orc.rsif(float(p[k, j]), float(t[k, j]))) if tc <= 0 else F(orc.rslf(float(p[k, j]), float(t[k, j])))
        ssati = F(qv[k, j] / qvsi - F(1))
        if abs(ssati) < EPS:
            ssati = F(0)
        if not ssati > 0:
            continue
        ssatw = ssati
        if tc <= 0:
            ssatw = F(qv[k, j] / F(orc.rslf(float(p[k, j]), float(t[k, j]))) - F(1))
            if abs(ssatw) < EPS:
                ssatw = F(0)
        busy[k, j] = bool((t[k, j] < T_0 and ssati >= F(0.25)) or ssatw > EPS)
    return sp, cold, busy


def cell_classes(st, p, iiwarm=False):
    """Array of class names ('' for idle cells) and the set of sort keys (species bits | cold << 5) of the busy cells."""
    sp, cold, busy = classify(st, p)
    out = np.full(sp.shape, "", dtype=object)
    keys = set()
    for k, j in zip(*np.nonzero(busy)):
        out[k, j] = kernel_class(int(sp[k, j]), bool(cold[k, j]), iiwarm)
        keys.add(int(sp[k, j]) | int(cold[k, j]) << 5)
    return out, keys


# ---- humidity -----------------------------------------------------------------------------------------------------------
def qv_for(p, t, sat, over="water"):
    """The largest f32 qv with qv / qvs - 1 <= sat in f32 arithmetic (qvs over water or ice); sat == 0 gives qv == qvs."""
    qvs = F(orc.rslf(p, t)) if over == "water" or F(t - F(273.15)) > 0 else F(orc.rsif(p, t))
    q = F(qvs * (1.0 + float(sat)))
    s = lambda x: F(x / qvs - F(1))
    for _ in range(64):
        if s(q) > F(sat):
            q = down(q)
        elif s(up(q)) <= F(sat):
            q = up(q)
        else:
            break
    return q


def q_for_r(r, p, t, qv):
    """Mixing ratio whose f32 product with the cell's air density is the density r (kg m^-3), when one exists nearby."""
    rho = rho_of(p, t, qv)
    q = F(F(r) / rho)
    for _ in range(16):
        got = F(q * rho)
        if got == F(r):
            break
        q = up(q) if got < F(r) else down(q)
    return q


def n_for_mvd(q, rho, mvd, rho_w=1000.0, mu=0.0):
    """Number mixing ratio of a gamma(mu = 0) rain distribution of mass mixing ratio q and median volume diameter mvd."""
    lam = (3.672 + mu) / mvd
    return F(q * lam ** 3 / (np.pi * rho_w))


def ni_for_xdi(q, rho, xdi):
    """Number mixing ratio of cloud ice of mass mixing ratio q and mean diameter xDi = 4 / lam (M:1429-1431)."""
    lam = 4.0 / xdi
    return F(q * lam ** 3 / (np.pi * 890.0))


# ---- column assembly ----------------------------------------------------------------------------------------------------
def pressure(dz, p_sfc=9.0e4, scale=8000.0):
    """Level mid-point pressures of layers dz over a surface at p_sfc (an isothermal scale height)."""
    dz = np.asarray(dz, np.float64)
    z = np.cumsum(dz) - 0.5 * dz
    return (p_sfc * np.exp(-z / scale)).astype(np.float32)


def assemble(specs, nz=NZ, dz=250.0, dt=20.0, p_sfc=9.0e4, probe_levels=PROBE, seed=0):
    """specs: list of dicts, one per regime point: 't' (K) of the busy cells, 'cell' = f(p, t) -> dict of the fields of a busy
    cell (qv and any of qc qi qr qs qg ni nr), optional 't_below' (K) of the idle levels under the probe levels and 'under' =
    {'t', 'cell'}: two busy levels of another kind right under the probe levels of the probe column.  Every spec
    gives one PROBE and one UNIFORM column.  A seeded jitter of 1e-4 relative on the pressure tells the columns apart."""
    dzv = np.broadcast_to(np.asarray(dz, np.float32), (nz,)).astype(np.float32).copy()
    pz = pressure(dzv, p_sfc)
    rng = np.random.default_rng(seed)
    ncol = 2 * len(specs)
    st = {k: np.zeros((nz, ncol), np.float32) for k in FIELDS}
    p = np.zeros((nz, ncol), np.float32)
    for j in range(ncol):
        sp = specs[j // 2]
        uniform = j % 2 == 1
        p[:, j] = (pz * (1.0 + 1e-4 * (rng.random() - 0.5))).astype(np.float32)
        for k in range(nz):
            busy = uniform or k in probe_levels
            t = F(sp["t"]) if busy or k > max(probe_levels) else F(sp.get("t_below", sp["t"]))
            make = sp["cell"]
            if not uniform and "under" in sp and k in (min(probe_levels) - 2, min(probe_levels) - 1):
                busy, t, make = True, F(sp["under"]["t"]), sp["under"]["cell"]
            st["t"][k, j] = t
            if busy:
                for f, v in make(float(p[k, j]), t).items():
                    st[f][k, j] = v
            else:                                               # clear air, well below ice and water saturation: idle
                st["qv"][k, j] = qv_for(float(p[k, j]), t, -0.7, over="ice")
    return st, p, dzv, float(dt)


def cell(qv_sat=0.0, over="ice", **species):
    """A busy cell: humidity qv / qvs - 1 = qv_sat over ice (below 0 C) or water; species given as densities (kg m^-3) through
    'rc' 'ri' 'rr' 'rs' 'rg', or mixing ratios 'qc' ...; numbers as 'nr_mvd' (median volume diameter, m), 'nr' (kg^-1),
    'ni_xdi' (mean ice diameter, m), 'ni' (kg^-1)."""
    def make(p, t):
        qv = qv_for(p, t, qv_sat, over)
        out = {"qv": qv}
        for m in ("c", "i", "r", "s", "g"):
            if "r" + m in species:
                out["q" + m] = q_for_r(species["r" + m], p, t, qv)
            elif "q" + m in species:
                out["q" + m] = F(species["q" + m])
        rho = float(rho_of(p, t, qv))
        if "nr_mvd" in species:
            out["nr"] = n_for_mvd(float(out["qr"]), rho, species["nr_mvd"])
        elif "nr" in species:
            out["nr"] = F(species["nr"])
        if "ni_xdi" in species:
            out["ni"] = ni_for_xdi(float(out["qi"]), rho, species["ni_xdi"])
        elif "ni" in species:
            out["ni"] = F(species["ni"])
        return out
    return make


# ---- targets ------------------------------------------------------------------------------------------------------------
class Rate:
    """The oracle rate `name` (one of the 36 save_dg rates) is non-zero (nonzero=True) or exactly zero in the busy cells
    `where` selects: where(st_in, p) -> bool (nz, ncol)."""

    def __init__(self, name, where, nonzero=True):
        self.name, self.where, self.nonzero = name, where, nonzero

    def check(self, st_in, p, st_out, rates, names, busy):
        sel = self.where(st_in, p) & busy
        assert sel.any(), "rate target %s selects no busy cell" % self.name
        r = rates[names.index(self.name)]
        bad = sel & ((r == 0) if self.nonzero else (r != 0))
        return None if not bad.any() else "%s %s in %d of %d cells, first (k, col) %s" % (
            self.name, "zero" if self.nonzero else "non-zero", bad.sum(), sel.sum(), tuple(np.argwhere(bad)[0]))


class State:
    """A property of the state after the step: prop(st_in, p, st_out) -> bool (nz, ncol), required in every cell (busy or
    idle) that where(st_in, p) selects."""

    def __init__(self, what, where, prop):
        self.name, self.where, self.prop = what, where, prop

    def check(self, st_in, p, st_out, rates, names, busy):
        sel = self.where(st_in, p)
        assert sel.any(), "state target '%s' selects no cell" % self.name
        bad = sel & ~self.prop(st_in, p, st_out)
        return None if not bad.any() else "'%s' fails in %d of %d cells, first (k, col) %s" % (
            self.name, bad.sum(), sel.sum(), tuple(np.argwhere(bad)[0]))


def has(f, thr=R1):
    return lambda s, p: s[f] > thr


def t_in(lo=-np.inf, hi=np.inf, incl_hi=False):
    return lambda s, p: (s["t"] > lo) & ((s["t"] <= hi) if incl_hi else (s["t"] < hi))


def both(*fs):
    return lambda s, p: np.logical_and.reduce([f(s, p) for f in fs])


def rho_arr(s, p):
    return (F(0.622) * p / (F(287.04) * s["t"] * (np.maximum(F(1e-10), s["qv"]) + F(0.622)))).astype(np.float32)


class Case:
    def __init__(self, name, build, targets, classes, aero=False):
        self.name, self.build, self.targets, self.classes, self.aero = name, build, targets, set(classes), aero

    def __repr__(self):
        return self.name


# ---- the cases ----------------------------------------------------------------------------------------------------------
T_HGFR = (F(234.0), F(230.0), F(220.0), down(HGFR), HGFR, up(HGFR))


def _hgfr_cloud():
    specs = [{"t": t, "cell": cell(0.0, "ice", rc=r)} for t in T_HGFR
             for r in (F(3e-7), down(R_C1), R_C1, up(R_C1), F(3e-5), F(2e-4))]
    return assemble(specs, p_sfc=4.5e4, seed=1)


def _hgfr_rain():
    specs = [{"t": t, "cell": cell(0.0, "ice", rr=r, nr_mvd=5e-4)} for t in T_HGFR
             for r in (F(3e-7), down(R_R1), R_R1, up(R_R1), F(3e-5), F(2e-4))]
    return assemble(specs, p_sfc=4.5e4, seed=2)


def _hgfr_vapour():
    specs = [{"t": t, "cell": cell(s, "water")} for t in T_HGFR for s in (2e-3, 1e-2, 4e-2)]
    return assemble(specs, p_sfc=4.5e4, seed=3)


T_MELT = (down(T_0), T_0, up(T_0), F(T_0 + F(0.05)), down(T_0 + F(0.1)), F(T_0 + F(0.1)), up(T_0 + F(0.1)), F(T_0 + F(0.2)))


def _t0_melt():
    mixes = (dict(qs=F(3e-4)), dict(qs=F(1e-3), qg=F(5e-4)), dict(qi=F(2e-5), ni_xdi=80e-6, qs=F(2e-4)),
             dict(qi=F(5e-5), ni_xdi=150e-6), dict(qg=F(1e-3)))
    specs = [{"t": t, "t_below": F(276.0), "cell": cell(0.0, "water", **m)} for t in T_MELT for m in mixes]
    return assemble(specs, p_sfc=8.0e4, seed=4)


def _t0_rain():
    ts = (F(T_0 - F(0.2)), F(T_0 - F(0.05)), down(T_0), T_0, up(T_0))
    mixes = (dict(qr=F(1e-3), nr_mvd=1e-3, qs=F(1e-3)), dict(qr=F(5e-4), nr_mvd=6e-4, qg=F(1e-3)),
             dict(qr=F(2e-4), nr_mvd=4e-4, qs=F(3e-4), qg=F(3e-4), qi=F(1e-5), ni_xdi=60e-6))
    specs = [{"t": t, "t_below": F(276.0), "cell": cell(0.0, "water", **m)} for t in ts for m in mixes]
    return assemble(specs, p_sfc=8.0e4, seed=5)


def _cooper_cold():
    ts = (F(250.0), F(245.0), F(240.0), F(236.0), down(F(253.15)), F(253.15), up(F(253.15)))
    # ssatw one f32 step above zero (the smallest value above EPS that a division can give), and a little more
    specs = [{"t": t, "cell": cell(s, "water")} for t in ts for s in (1.2e-7, 1e-4, 1e-3)]
    return assemble(specs, p_sfc=5.0e4, seed=6)


SSATI_25 = (F(0.25), down(F(0.25)))          # (qv_for: the largest reachable ssati below 0.25 is 0.25 - 2**-23)


def _cooper_ssati():
    ts = (F(254.0), F(258.0), F(262.0), F(266.0), F(270.0), down(T_0))
    specs = [{"t": t, "cell": cell(s, "ice")} for t in ts for s in SSATI_25]
    return assemble(specs, p_sfc=6.0e4, seed=7)


def _cooper_cap():
    specs = [{"t": t, "cell": cell(s, "water")} for t in (F(200.0), F(205.0), F(210.0)) for s in (1.2e-7, 1e-3)]
    return assemble(specs, p_sfc=2.5e4, seed=8)


def _vapour_warm():
    specs = [{"t": t, "cell": cell(s, "water")} for t in (F(275.0), F(285.0), F(295.0)) for s in (0.0, 1.2e-7, 1e-3, 1e-2)]
    return assemble(specs, p_sfc=9.5e4, seed=9)


def _evap_dry():
    specs = [{"t": t, "cell": cell(rh - 1.0, "water", qc=F(q), qr=F(q), nr_mvd=2e-4)}
             for t in (F(280.0), F(290.0), F(300.0)) for rh in (0.2, 0.3, 0.4) for q in (1e-8, 1e-7, 1e-6)]
    return assemble(specs, p_sfc=9.5e4, seed=10)


def _rain_clamps():
    specs = []
    for t in (F(285.0), F(265.0)):
        for q in (1e-4, 2e-3):
            for n in (dict(nr_mvd=4e-3), dict(nr_mvd=6e-3), dict(nr_mvd=20e-6), dict(nr_mvd=30e-6), dict(nr=0.0)):
                specs.append({"t": t, "cell": cell(0.0, "water", qr=F(q), **n)})
    return assemble(specs, p_sfc=8.5e4, seed=11)


def _ice_clamps():
    specs = []
    for t in (F(250.0), F(228.0)):
        for q in (1e-6, 1e-4):
            for n in (dict(ni_xdi=2e-6), dict(ni_xdi=4e-6), dict(ni_xdi=400e-6), dict(ni_xdi=900e-6), dict(ni=0.0),
                      dict(ni=F(2.0e6)), dict(ni=F(6.0e6))):
                specs.append({"t": t, "cell": cell(0.05, "ice", qi=F(q), **n)})
    return assemble(specs, p_sfc=5.0e4, seed=12)


def _table_edges():
    specs = []
    for t in (F(265.0), F(277.0)):
        for rr, rs, rg in ((R_R1, R_S1, R_G1), (down(R_R1), down(R_S1), down(R_G1)), (up(R_R1), up(R_S1), up(R_G1)),
                           (R_LAST, R_LAST, R_LAST), (F(2e-2), F(3e-2), F(3e-2)), (F(1e-3), down(R_S1), F(3e-2)),
                           (F(3e-2), F(1e-3), down(R_G1))):
            specs.append({"t": t, "cell": cell(0.0, "water", rr=rr, nr_mvd=1e-3, rs=rs, rg=rg)})
    return assemble(specs, p_sfc=8.0e4, seed=13)


def _intercept_edges():
    specs = []
    for t in (F(268.0), F(255.0)):
        for q, mvd in ((1e-2, 2.4e-3), (2e-2, 2.5e-3), (1e-6, 40e-6), (3e-7, 38e-6), (5e-3, 2e-3), (1e-5, 60e-6)):
            for qg in (0.0, 3e-2, 2e-9):
                specs.append({"t": t, "cell": cell(0.0, "water", qr=F(q), nr_mvd=mvd, qg=F(qg))})
    return assemble(specs, p_sfc=7.0e4, seed=14)


T_TC = (F(T_0 - F(0.5)), F(T_0 - F(44.5)), F(T_0 - F(45.5)), F(T_0 - F(80.0)))


def _idx_tc():
    specs = [{"t": t, "cell": cell(0.0, "ice", qc=F(q), qr=F(q), nr_mvd=5e-4)} for t in T_TC for q in (2e-6, 1e-4, 1e-3)]
    return assemble(specs, p_sfc=4.0e4, seed=15)


def _sediment():
    # dt = 120 s over 20-50 m layers at 300-400 hPa (fall speeds grow with rho_not / rho): graupel, rain, snow and ice in
    # one column need tens to hundreds of sub-steps each (M:3242), far below the KP_NSTEP_MAX cap
    dz = np.linspace(20.0, 50.0, NZ).astype(np.float32)
    specs = [{"t": t, "t_below": F(275.0),
              "cell": cell(0.0, "water", qg=F(g), qr=F(r), nr_mvd=1.5e-3, qs=F(2e-3), qi=F(1e-4), ni_xdi=100e-6)}
             for t in (F(262.0), F(268.0), F(272.0)) for g in (5e-3, 1.5e-2) for r in (3e-3, 8e-3)]
    return assemble(specs, dz=dz, dt=120.0, p_sfc=3.5e4, seed=16)


def _inherited_speeds():
    # A level without a species takes the fall speed of the level above (M:3235), so a busy cell of the warm or the ice class
    # receives ice (or rain) falling from above with that speed.  The one-sector records of these classes supply the missing
    # ice (or rain) number as a constant (load_rec_a); it multiplies the inherited number speed in the flux leaving the cell.
    # Few, large crystals and drops keep the numbers small enough for the flux of that constant to show.  The warm cells sit at
    # exactly T_0 and water saturation, where nothing melts the arriving ice (S15 needs T > T_0, M:3584).
    specs = []
    for q in (2e-9, 1e-8, 5e-8):
        specs.append({"t": F(262.0), "cell": cell(0.0, "ice", qi=F(q), ni_xdi=250e-6),
                      "under": {"t": T_0, "cell": cell(0.0, "water", qc=F(1e-4))}})
    for q in (1e-6, 5e-6, 2e-5):
        specs.append({"t": F(276.0), "cell": cell(0.0, "water", qr=F(q), nr_mvd=2.2e-3),
                      "under": {"t": F(266.0), "cell": cell(0.0, "ice", qi=F(1e-5), ni_xdi=100e-6)}})
    return assemble(specs, p_sfc=7.0e4, seed=18)


def _species_sets():
    # every (species set, T < T_0) sort key of k_classify: 32 sets x cold / warm; a vapour-only cell is busy through
    # supersaturation over water
    specs = []
    for cold in (True, False):
        for sp in range(32):
            m = {}
            if sp & QC: m["qc"] = F(1e-4)
            if sp & QI: m.update(qi=F(1e-5), ni_xdi=60e-6)
            if sp & QR: m.update(qr=F(2e-4), nr_mvd=5e-4)
            if sp & QS: m["qs"] = F(2e-4)
            if sp & QG: m["qg"] = F(2e-4)
            specs.append({"t": F(266.0) if cold else F(279.0), "cell": cell(0.0 if sp else 2e-3, "water", **m)})
    return assemble(specs, p_sfc=7.5e4, seed=17)


def _cold(lo=-np.inf):
    return t_in(lo, T_0)


CASES = [
    Case("hgfr_cloud", _hgfr_cloud, [
        Rate("pri_wfz", both(has("qc"), t_in(hi=HGFR))),
        Rate("pri_wfz", both(has("qc"), t_in(lo=down(HGFR)), lambda s, p: s["qc"] * rho_arr(s, p) <= R_C1), nonzero=False),
        # (the limiter of S7 can leave a residual of a few 1e-11 kg/kg, M:2291-2387)
        State("no cloud water left below HGFR", both(has("qc"), t_in(hi=F(234.5))), lambda s, p, o: o["qc"] < F(1e-10))],
        {"MIXNR"}, aero=True),
    Case("hgfr_rain", _hgfr_rain, [
        Rate("pnr_rfz", both(has("qr"), t_in(hi=HGFR))),
        Rate("pnr_rfz", both(has("qr"), t_in(lo=down(HGFR)), lambda s, p: s["qr"] * rho_arr(s, p) <= R_R1), nonzero=False)],
        {"FULL"}, aero=True),
    Case("hgfr_vapour", _hgfr_vapour, [
        State("condensed and frozen below HGFR", both(lambda s, p: _ssatw(s, p) > 0, t_in(hi=F(234.5))),
              lambda s, p, o: (o["qc"] == 0) & (o["qi"] > 0))],
        {"ICE"}, aero=True),
    Case("t0_melt", _t0_melt, [
        Rate("prr_sml", both(has("qs"), t_in(lo=T_0))),
        Rate("prr_sml", both(has("qs"), t_in(hi=T_0, incl_hi=True)), nonzero=False),
        Rate("prr_gml", both(has("qg"), t_in(lo=T_0))),
        State("cloud ice melted at once above T_0 + 0.05", both(has("qi"), t_in(lo=F(T_0 + F(0.04)))),
              lambda s, p, o: o["qi"] < F(1e-10))],
        {"ICE", "MIXNR"}, aero=True),
    Case("t0_rain", _t0_rain, [
        Rate("pnr_rcs", both(has("qr"), has("qs"))),
        Rate("pnr_rcg", both(has("qr"), has("qg")))],
        {"FULL"}),
    Case("cooper_cold", _cooper_cold, [
        Rate("pni_inu", t_in(hi=F(253.15))),
        Rate("pni_inu", t_in(lo=down(F(253.15))), nonzero=False)],
        {"ICE"}, aero=True),
    Case("cooper_ssati", _cooper_ssati, [
        Rate("pni_inu", lambda s, p: _ssati(s, p) >= F(0.25)),
        Rate("pni_inu", lambda s, p: _ssati(s, p) < F(0.25), nonzero=False)],
        {"ICE"}, aero=True),
    Case("cooper_cap", _cooper_cap, [
        Rate("pni_inu", t_in(hi=F(211.0))),
        State("ice number at most the 250e3 m^-3 of Cooper's cap", t_in(hi=F(211.0)),
              lambda s, p, o: o["ni"] * rho_arr(o, p) <= F(250e3) * F(1.0001))],
        {"ICE"}, aero=True),
    Case("vapour_warm", _vapour_warm, [
        State("condensation from vapour alone", lambda s, p: _ssatw(s, p) > 0, lambda s, p, o: o["qc"] > 0),
        State("no condensation at saturation", lambda s, p: (_ssatw(s, p) == 0) & (s["t"] > T_0), lambda s, p, o: o["qc"] == 0)],
        {"WARM"}),
    Case("evap_dry", _evap_dry, [
        Rate("prv_rev", has("qr")),
        State("cloud water all evaporated", has("qc"), lambda s, p, o: o["qc"] == 0)],
        {"WARM"}),
    Case("rain_clamps", _rain_clamps, [
        State("rain mvd inside [0.75 D0r, 2.5 mm] after the step", lambda s, p: s["qr"] > 0,
              lambda s, p, o: _mvd_ok(o, p))],
        {"WARM", "FULL"}, aero=True),
    Case("ice_clamps", _ice_clamps, [
        State("ice number at most 499e3 m^-3 after the step", has("qi"),
              lambda s, p, o: o["ni"] * rho_arr(o, p) <= F(499e3) * F(1.0001)),
        Rate("pri_ide", has("qi"))],
        {"ICE"}, aero=True),
    Case("table_edges", _table_edges, [
        Rate("pnr_rcs", both(_cold(), lambda s, p: (s["qr"] * rho_arr(s, p) >= R_R1) & (s["qs"] * rho_arr(s, p) >= R_S1))),
        Rate("pnr_rcg", both(_cold(), lambda s, p: (s["qr"] * rho_arr(s, p) >= R_R1) & (s["qg"] * rho_arr(s, p) >= R_G1)))],
        {"FULL"}),
    Case("intercept_edges", _intercept_edges, [
        Rate("pnr_rfz", both(_cold(), lambda s, p: s["qr"] * rho_arr(s, p) > R_R1))],
        {"FULL"}),
    Case("idx_tc", _idx_tc, [
        Rate("pnr_rfz", lambda s, p: s["qr"] * rho_arr(s, p) > R_R1),
        Rate("pri_wfz", lambda s, p: s["qc"] * rho_arr(s, p) > R_C1)],
        {"FULL"}),
    Case("sediment", _sediment, [
        State("graupel reaches the ground in one step", lambda s, p: _probe_mask(s, level=0),
              lambda s, p, o: np.broadcast_to(o["ppt"][3] > 0, s["t"].shape))],
        {"FULL"}),
    Case("inherited_speeds", _inherited_speeds, [
        State("ice falls into the warm cells at T_0", lambda s, p: _probe_mask(s, PROBE[0] - 1) & (s["t"] == T_0),
              lambda s, p, o: o["qi"] > 0),
        State("rain falls into the ice cells", lambda s, p: _probe_mask(s, PROBE[0] - 1) & (s["qi"] > 0),
              lambda s, p, o: o["nr"] > 0)],
        {"WARM", "ICE"}),
    Case("species_sets", _species_sets, [
        State("every sort key present", lambda s, p: np.ones(s["t"].shape, bool), lambda s, p, o: np.ones(o["t"].shape, bool))],
        set(CLASSES)),
]
BY_NAME = {c.name: c for c in CASES}


def _ssati(s, p):
    out = np.full(s["t"].shape, -1.0, np.float32)
    for k, j in np.ndindex(*out.shape):
        qvsi = F(orc.rsif(float(p[k, j]), float(s["t"][k, j])))
        out[k, j] = F(s["qv"][k, j] / qvsi - F(1))
    return out


def _ssatw(s, p):
    out = np.full(s["t"].shape, -1.0, np.float32)
    for k, j in np.ndindex(*out.shape):
        out[k, j] = F(s["qv"][k, j] / F(orc.rslf(float(p[k, j]), float(s["t"][k, j]))) - F(1))
    return out


def _mvd_ok(o, p):
    rho = rho_arr(o, p).astype(np.float64)
    qr, nr = o["qr"].astype(np.float64), o["nr"].astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        lam = (np.pi * 1000.0 * nr / np.maximum(qr, 1e-30)) ** (1.0 / 3.0)
        mvd = 3.672 / lam
    return (qr == 0) | ((mvd >= 0.75 * 50e-6 * (1 - 1e-3)) & (mvd <= 2.5e-3 * (1 + 1e-3)))


def _probe_mask(s, level):
    m = np.zeros(s["t"].shape, bool)
    m[level, 0::2] = True
    return m


def build(case):
    return case.build() if isinstance(case, Case) else BY_NAME[case].build()


def regime_domain(names=None):
    """The columns of every case with the common layers and time step (all but 'sediment') side by side: (state, p, dz, dt)."""
    parts = [build(c) for c in CASES if (names is None or c.name in names) and c.name != "sediment"]
    dz, dt = parts[0][2], parts[0][3]
    assert all(np.array_equal(q[2], dz) and q[3] == dt for q in parts)
    st = {k: np.ascontiguousarray(np.concatenate([q[0][k] for q in parts], axis=1)) for k in FIELDS}
    return st, np.ascontiguousarray(np.concatenate([q[1] for q in parts], axis=1)), dz, dt


def oracle_run(o, case, with_rates=True):
    """The case through the oracle: (state in, p, dz, dt, state out (and its 'ppt'), ppt, rates (36, nz, ncol) or None)."""
    st, p, dz, dt = build(case)
    out = {k: v.copy() for k, v in st.items()}
    ppt = o.step(dt, out, p, dz)
    out["ppt"] = ppt
    rates = None
    if with_rates:
        nz, ncol = st["t"].shape
        rates = np.zeros((36, nz, ncol), np.float64)
        for j in range(ncol):
            r = o.column(dt, *[st[k][:, j] for k in FIELDS], p[:, j], dz, want_rates=True)
            rates[:, :, j] = r["rates"]
    return st, p, dz, dt, out, ppt, rates


def bench_like(ncol, dz):
    """Columns of the bench domain (kid_b200/synth.py, 60 levels of depth dz): (state, p, dz)."""
    from kid_b200 import synth
    st, p, dzv = synth.make_domain(ncol, nz=60, nx=1024, dz=dz, col0=300000)
    return {k: v.numpy().copy() for k, v in st.items()}, p.numpy().copy(), dzv.numpy().copy()


# ---- the CUDA step against the oracle, cell by cell (GPU tests) --------------------------------------------------------
RATE_TOL = 1e-5


def cell_outliers(got, ref, fields, cls):
    """One line per cell of `fields` where got and ref differ by more than REL_TOL (relative to max(|ref|, FLOOR))."""
    out = []
    for f in fields:
        a, b = got[f].astype(np.float64), ref[f].astype(np.float64)
        rel = np.abs(a - b) / np.maximum(np.abs(b), FLOOR.get(f, 1e-30))
        rel = np.where(a == b, 0.0, rel)
        for k, j in np.argwhere(~(rel <= REL_TOL)):
            out.append("col %d level %d %s: gpu %.9g oracle %.9g (rel %.2e, class %s)" % (j, k, f, a[k, j], b[k, j], rel[k, j],
                                                                                          cls[k, j] or "idle"))
    return out


def rate_outliers(got, ref, names, cls):
    """One line per (rate, cell) where the device rate differs from the oracle's (rounded to f32) by more than RATE_TOL."""
    out = []
    ref32 = ref.astype(np.float32).astype(np.float64)
    got = got.astype(np.float64)
    rel = np.abs(got - ref32) / np.maximum(np.abs(ref32), 1e-30)
    rel = np.where(got == ref32, 0.0, rel)
    for q, k, j in np.argwhere(~(rel <= RATE_TOL)):
        out.append("col %d level %d %s: gpu %.9g oracle %.9g (class %s)" % (j, k, names[q], got[q, k, j], ref32[q, k, j],
                                                                             cls[k, j] or "idle"))
    return out


class Device:
    """Device copies of one input, allocated once: every run() starts from the same inputs at the same addresses, so that a
    handle with CUDA graphs on replays its capture of the previous run unless a setting in the graph key changed."""

    def __init__(self, st, p, dz, dt, rates=True):
        import torch
        self.nz, self.ncol = st["t"].shape
        self.dt = dt
        self.src = {k: torch.from_numpy(st[k].copy()).cuda() for k in FIELDS}
        self.dev = {k: v.clone() for k, v in self.src.items()}
        self.p, self.dz = torch.from_numpy(p).cuda(), torch.from_numpy(dz).cuda()
        self.ppt = torch.zeros((4, self.ncol), dtype=torch.float32, device="cuda")
        self.rates = torch.empty((36, self.nz, self.ncol), dtype=torch.float32, device="cuda") if rates else None

    def run(self, th):
        """One step; returns (state, ppt, rates or None, diag, step_stats)."""
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
                           self.dz.data_ptr(), self.ppt.data_ptr())
            th.sync()
        finally:
            th.set_rates_buffer(0)
        return ({k: self.dev[k].cpu().numpy() for k in FIELDS}, self.ppt.cpu().numpy(),
                self.rates.cpu().numpy() if self.rates is not None else None, th.diag(), th.step_stats())


def aero_step(th, st, p, dz, dt, nc, nwfa, nifa, w):
    """kidmp_step_device_aero on device copies of the inputs: (state with nc nwfa nifa, ppt)."""
    import torch
    nz, ncol = st["t"].shape
    dev = {k: torch.from_numpy(st[k].copy()).cuda() for k in FIELDS}
    dnc, dnwfa, dnifa, dw = (torch.from_numpy(x.copy()).cuda() for x in (nc, nwfa, nifa, w))
    dp, ddz = torch.from_numpy(p).cuda(), torch.from_numpy(dz).cuda()
    ppt = torch.zeros((4, ncol), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    th.step_device_aero(ncol, nz, dt, [dev[k].data_ptr() for k in FIELDS], dnc.data_ptr(), dnwfa.data_ptr(), dnifa.data_ptr(),
                        dp.data_ptr(), dw.data_ptr(), ddz.data_ptr(), ppt.data_ptr())
    th.sync()
    out = {k: dev[k].cpu().numpy() for k in FIELDS}
    out.update(nc=dnc.cpu().numpy(), nwfa=dnwfa.cpu().numpy(), nifa=dnifa.cpu().numpy())
    return out, ppt.cpu().numpy()


def aero_inputs(st, p, seed=0):
    """Aerosol-aware inputs at the clamps of M:1392-1393 and M:1399-1410: water- and ice-friendly aerosol numbers below 11.1e6
    and above 9999e6 m^-3, droplet numbers that span nu_c = 2 .. 15, vertical velocity < 0, = 0 and large."""
    nz, ncol = st["t"].shape
    rng = np.random.default_rng(seed)
    rho = rho_arr(st, p)
    per_m3 = np.array([5e6, 11.1e6, 1e8, 1e9, 9999e6, 2e10], np.float32)
    nwfa = (per_m3[rng.integers(0, 6, (1, ncol))] / rho).astype(np.float32)
    nifa = (per_m3[rng.integers(0, 6, (1, ncol))] / rho).astype(np.float32)
    nc_m3 = np.array([5e9, 1e9, 5e8, 2e8, 1e8, 7.7e7, 7e7, 5e7], np.float32)      # nu_c = 2, 3, 4, 7, 12, 15, 16 -> 15, ...
    nc = np.where(st["qc"] > R1, nc_m3[rng.integers(0, len(nc_m3), (nz, ncol))] / rho, 0.0).astype(np.float32)
    w = np.array([-2.0, 0.0, 25.0], np.float32)[rng.integers(0, 3, (nz, ncol))].astype(np.float32)
    return nc, nwfa, nifa, w
