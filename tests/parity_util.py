"""Comparison helpers of the parity tests: CUDA path vs the CPU oracle on identical inputs.

Tolerance (BASELINE.json north_star): at most 1e-5 relative error per hydrometeor mass / number
after one step.  The scheme is full of discontinuous table indices and thresholds (SURVEY.md
section 7, hard part 1), so the report separates
  * bit-identical cells,
  * cells within REL_TOL (relative to max(|oracle|, floor of the field)),
  * outliers (index / threshold flips), which must stay below FLIP_FRACTION of the cells.
"""
import numpy as np

FIELDS = ("qv", "qc", "qi", "qr", "qs", "qg", "ni", "nr", "t")
REL_TOL = 1e-5
FLIP_FRACTION = 2e-4
# below these magnitudes a field value is physically nothing (the scheme's own R1 = 1e-12 kg/kg
# threshold for masses, and one particle per 1000 m^3 for numbers); differences there are
# compared absolutely
FLOOR = {"qv": 1e-10, "qc": 1e-12, "qi": 1e-12, "qr": 1e-12, "qs": 1e-12, "qg": 1e-12, "ni": 1e-3, "nr": 1e-3,
         "t": 1.0, "nc": 1e-3, "nwfa": 1e-3, "nifa": 1e-3}
# the constants of thompson_init (M:374-797) that the device keeps and the oracle exports: compared bit for bit
INIT_CONSTANTS = ("cre", "crg", "cse", "csg", "cge", "cgg", "cie", "cig", "cce1", "cce2", "cce3", "cce4", "cce5",
                  "ccg1", "ccg2", "ccg3", "ccg4", "ccg5", "ocg1", "ocg2", "scalars", "offsets",
                  "Dc", "Di", "Dr", "Ds", "Dg", "t_Nc", "dtc", "dti", "dtr", "dts", "dtg")


def compare_field(name, got, ref):
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    exact = (got == ref) | (np.isnan(got) & np.isnan(ref))
    denom = np.maximum(np.abs(ref), FLOOR[name] if name in FLOOR else 1e-30)
    rel = np.abs(got - ref) / denom
    rel = np.where(exact, 0.0, rel)
    rel = np.where(np.isfinite(rel), rel, np.inf)
    return {
        "n": int(ref.size),
        "exact": int(exact.sum()),
        "within": int((rel <= REL_TOL).sum()),
        "max_rel": float(rel.max()) if rel.size else 0.0,
        "p9999_rel": float(np.quantile(rel, 0.9999)) if rel.size else 0.0,
        "argmax": int(rel.argmax()) if rel.size else -1,
    }


def compare_states(got, ref, fields=FIELDS):
    """got/ref: dicts of arrays.  Returns {field: stats} plus '_all'."""
    out = {}
    n = ex = wi = 0
    for f in fields:
        s = compare_field(f, got[f], ref[f])
        out[f] = s
        n += s["n"]; ex += s["exact"]; wi += s["within"]
    out["_all"] = {"n": n, "exact": ex, "within": wi, "exact_frac": ex / max(n, 1), "within_frac": wi / max(n, 1),
                   "max_rel": max(out[f]["max_rel"] for f in fields)}
    return out


def assert_parity(got, ref, fields=FIELDS, flip_fraction=FLIP_FRACTION, what=""):
    st = compare_states(got, ref, fields)
    a = st["_all"]
    bad = a["n"] - a["within"]
    msg = "%s parity: %d/%d cells outside rel %.0e (allowed %.1e of cells); exact %.4f; per field %s" % (
        what, bad, a["n"], REL_TOL, flip_fraction, a["exact_frac"],
        {f: (st[f]["n"] - st[f]["within"], "%.2e" % st[f]["max_rel"]) for f in fields})
    assert bad <= max(0, int(flip_fraction * a["n"])), msg
    return st
