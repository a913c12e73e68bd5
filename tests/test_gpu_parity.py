"""GPU parity tests: the CUDA path through the C ABI vs the CPU oracle on identical seeded inputs.

Bar (BASELINE.json): <= 1e-5 relative per hydrometeor mass / number after one step, except for a
counted handful of index / threshold flip cells (parity_util.FLIP_FRACTION); lookup tables to
1e-12 relative; init constants bit-exact.  M:/I: cite the reference files.
"""
import os

import numpy as np
import pytest

from parity_util import assert_parity, compare_states, FIELDS, INIT_CONSTANTS

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden", "columns.npz")


def _domain(ncol, nz=60, **kw):
    from kid_b200 import synth
    st, p, dz = synth.make_domain(ncol, nz=nz, **kw)
    return {k: v.numpy().copy() for k, v in st.items()}, p.numpy().copy(), dz.numpy().copy()


def _both(g, o, dt, st, p, dz, layout="col_fastest"):
    a = {k: v.copy() for k, v in st.items()}
    b = {k: v.copy() for k, v in st.items()}
    pa = g.step(dt, a, p, dz, layout=layout)
    pb = o.step(dt, b, p, dz, layout=layout)
    return a, pa, b, pb


# ---- thompson_init: constants and lookup tables (M:374-797, M:3698-4343) ------------------------------
def test_init_constants_bit_exact(gpu_mixed, oracle_mixed):
    for name in INIT_CONSTANTS:
        assert np.array_equal(gpu_mixed.get(name), oracle_mixed.get(name).ravel()), name


def test_lookup_tables(gpu_mixed, oracle_mixed):
    from oracle.oracle import TABLE_SHAPES
    for name in TABLE_SHAPES:
        a = gpu_mixed.get(name)
        b = oracle_mixed.get(name).ravel(order="F")
        assert a.shape == b.shape, name
        rel = np.where(a == b, 0.0, np.abs(a - b) / np.maximum(np.abs(b), 1e-300))
        assert rel.max() < 1e-12, (name, rel.max())
    assert gpu_mixed.table_build_ms > 0


def test_tables_against_golden_samples(gpu_mixed):
    g = np.load(GOLD)
    for key in g.files:
        if key.startswith("table/") and key.endswith("/sample"):
            name = key.split("/")[1]
            t = gpu_mixed.get(name)
            s = t[:: max(1, t.size // 257)][:257]
            np.testing.assert_allclose(s, g[key], rtol=1e-12, atol=0, err_msg=name)
            tot = g["table/%s/sum" % name]
            np.testing.assert_allclose(t.sum(), tot[0], rtol=1e-11)
            assert float((t != 0).sum()) == tot[2]


def test_table_cache_roundtrip(gpu_mixed, tmp_path):
    from kid_b200.kidmp import Thompson
    path = str(tmp_path / "tables.bin")
    gpu_mixed.save_tables(path)
    t2 = Thompson(set_Nc=100.0, iiwarm=False, table_cache=path, reuse_tables=True)
    assert t2.tables_from_cache
    for name in ("tcg_racg", "tnr_sacr2", "tpg_qrfz", "tni_qcfz", "tpi_ide", "t_Efsw"):
        assert np.array_equal(t2.get(name), gpu_mixed.get(name)), name
    t2.close()
    # a cache written under other constants is refused and the tables are rebuilt (M:3874-3881 warns, we check)
    t3 = Thompson(set_Nc=100.0, iiwarm=False, wp_double=True, table_cache=path, reuse_tables=True)
    assert not t3.tables_from_cache
    t3.close()


# ---- mp_thompson (M:1156-3688) ---------------------------------------------------------------------------
def test_golden_columns(gpu_mixed, gpu_warm):
    g = np.load(GOLD)
    for th, tag, dt in ((gpu_mixed, "mixed_dt10", 10.0), (gpu_mixed, "mixed_dt60", 60.0), (gpu_warm, "warm_dt10", 10.0)):
        s = {k: g["in/" + k].copy() for k in FIELDS}
        ppt = th.step(dt, s, g["in/p"].copy(), g["in/dz"])
        ref = {k: g["%s/%s" % (tag, k)] for k in FIELDS}
        assert_parity(s, ref, what=tag, flip_fraction=1e-3)
        np.testing.assert_allclose(ppt, g[tag + "/ppt"], rtol=1e-5, atol=1e-12)


def test_no_sedimentation_switch(tmp_path):
    from kid_b200.kidmp import Thompson
    g = np.load(GOLD)
    th = Thompson(set_Nc=300.0, iiwarm=False, l_sediment=False)
    s = {k: g["in/" + k].copy() for k in FIELDS}
    ppt = th.step(10.0, s, g["in/p"].copy(), g["in/dz"])
    assert_parity(s, {k: g["nosed_dt10/" + k] for k in FIELDS}, what="l_sediment=F", flip_fraction=1e-3)
    assert not ppt[1:].any()                       # ice, snow, graupel do not fall (M:3449, M:3506, M:3555)
    assert ppt[0].any()                            # rain still does (U6)
    th.close()


def test_deep_mixed_phase_column(gpu_mixed, oracle_mixed):
    """BASELINE config 2: one deep column with every species present, through the mp_thompson twin."""
    from kid_b200 import synth
    st, p, dz = synth.deep_column()
    args = [st[k] for k in FIELDS]
    a = gpu_mixed.column(10.0, *args, p, dz, ppt=[1.0, 2.0, 3.0, 4.0])
    b = oracle_mixed.column(10.0, *args, p, dz, ppt=[1.0, 2.0, 3.0, 4.0])
    assert_parity(a, b, what="deep column", flip_fraction=0.0)
    np.testing.assert_allclose(a["ppt"], b["ppt"], rtol=1e-6)        # INOUT accumulators (M:1172)
    assert a["ppt"][0] > 1.0


def test_mixed_domain_one_step(gpu_mixed, oracle_mixed):
    st, p, dz = _domain(4096, cloudy_fraction=1.0, coherent=False)
    for dt in (10.0, 60.0):                        # dt = 60 s drives nstep > 1 in the sedimentation sub-stepping
        a, pa, b, pb = _both(gpu_mixed, oracle_mixed, dt, st, p, dz)
        stt = assert_parity(a, b, what="4096 mixed dt=%g" % dt)
        assert stt["_all"]["exact_frac"] > 0.995
        np.testing.assert_allclose(pa, pb, rtol=1e-5, atol=1e-10)


def test_cells_outside_tolerance_are_condensation_residuals(gpu_mixed, oracle_mixed):
    """Decision U13 (DESIGN.md section 4).  The handful of cells per million whose hydrometeor content differs from the oracle by
    more than 1e-5 are all of one kind: cloud water (once: rain) left over after condensation or evaporation took almost all of
    it.  The Newton iteration of S11 (M:2784-2789) works in f32 on numbers of the size of qv, so its result carries one ulp
    of qv (~5e-10 kg/kg) of rounding freedom (expf of the host's libm vs the f64-evaluated one here); a residual of 1e-5 ... 1e-7
    kg/kg inherits that absolute difference.  Checked: every such cell is qc or qr, its difference is below two ulp of qv,
    and temperature, vapour and total water of the cell agree to rounding."""
    seen = 0
    for kw, dt in ((dict(col0=7, cloudy_fraction=1.0, coherent=False), 1.0), (dict(col0=1000, cloudy_fraction=1.0, coherent=False), 20.0),
                   (dict(col0=0, cloudy_fraction=0.6, coherent=False), 60.0)):
        st, p, dz = _domain(4096, **kw)
        a, pa, b, pb = _both(gpu_mixed, oracle_mixed, dt, st, p, dz)
        for f in FIELDS:
            den = np.maximum(np.abs(b[f].astype(np.float64)), 1e-12 if f.startswith("q") else (1e-3 if f.startswith("n") else 1.0))
            rel = np.abs(a[f].astype(np.float64) - b[f]) / den
            bad = np.argwhere(rel > 1e-5)
            if len(bad) and f not in ("qc", "qr"):
                assert f in ("nr",) and len(bad) <= 2, (f, len(bad))         # the number that belongs to such a rain residual
                continue
            for k, j in bad:
                seen += 1
                qv = float(b["qv"][k, j])
                assert abs(float(a[f][k, j]) - float(b[f][k, j])) <= 2.5e-7 * qv + 1e-11, (f, k, j)
                assert abs(float(a["t"][k, j]) - float(b["t"][k, j])) <= 1e-4
                assert abs(float(a["qv"][k, j]) - float(b["qv"][k, j])) <= 2.5e-7 * qv
    assert seen <= 30


def test_conus_domain_one_step(gpu_mixed, oracle_mixed):
    st, p, dz = _domain(8192, col0=300000, nx=1024)            # the bench domain: ~30 % cloudy, coherent
    a, pa, b, pb = _both(gpu_mixed, oracle_mixed, 10.0, st, p, dz)
    assert_parity(a, b, what="bench domain")
    np.testing.assert_allclose(pa, pb, rtol=1e-5, atol=1e-10)


def test_warm_rain_domain(gpu_warm, oracle_warm):
    """BASELINE config 1 regime (iiwarm): S1,S2,S5,S7-S9,S11-S14,S16 only."""
    st, p, dz = _domain(2048, cloudy_fraction=1.0, coherent=False)
    a, pa, b, pb = _both(gpu_warm, oracle_warm, 1.0, st, p, dz)
    assert_parity(a, b, what="warm dt=1")
    for k in ("qs", "qg"):
        assert np.array_equal(a[k], st[k])         # ice species untouched when iiwarm
    np.testing.assert_allclose(pa, pb, rtol=1e-5, atol=1e-10)


def test_clear_sky_columns_bit_unchanged(gpu_mixed):
    st, p, dz = _domain(1000, cloudy_fraction=0.0, coherent=False)
    a = {k: v.copy() for k, v in st.items()}
    gpu_mixed.diag()                               # clear the accumulated domain sums
    ppt = gpu_mixed.step(10.0, a, p, dz)
    for k in FIELDS:
        assert np.array_equal(a[k], st[k]), k      # early RETURN at M:1540
    assert not ppt.any()
    d = gpu_mixed.diag()
    assert d[6] == 0 and d[7] == 1000


def test_tiny_species_are_zeroed_before_the_early_return(gpu_mixed, oracle_mixed):
    # U9: species <= R1 are zeroed in the caller's arrays even when the column takes the clear-sky exit
    st, p, dz = _domain(64, cloudy_fraction=0.0, coherent=False)
    st["qc"][5, :] = 5e-13; st["qi"][40, :] = 9e-13; st["ni"][40, :] = 10.0; st["nr"][3, :] = 2.0
    a, pa, b, pb = _both(gpu_mixed, oracle_mixed, 10.0, st, p, dz)
    for k in FIELDS:
        assert np.array_equal(a[k], b[k]), k
    assert not a["qc"].any() and not a["ni"].any() and not a["nr"].any()


def test_layouts_and_ragged_sizes(gpu_mixed, oracle_mixed):
    for ncol in (1, 31, 129, 1000):
        st, p, dz = _domain(ncol, cloudy_fraction=1.0, coherent=False)
        a, pa, b, pb = _both(gpu_mixed, oracle_mixed, 10.0, st, p, dz)
        assert_parity(a, b, what="ncol=%d" % ncol, flip_fraction=1e-3)
        # KiD (k,i) layout gives bitwise the same numbers as the device layout
        kt = {k: np.ascontiguousarray(v.T) for k, v in st.items()}
        pk = gpu_mixed.step(10.0, kt, np.ascontiguousarray(p.T), dz, layout="k_fastest")
        for k in FIELDS:
            assert np.array_equal(kt[k].T, a[k]), (ncol, k)
        assert np.array_equal(pk, pa)


def test_other_level_counts(gpu_mixed, oracle_mixed):
    """nz = 120 (BASELINE config 3, 2-D cumulus grid run as 120 independent columns) and odd sizes."""
    for nz, dzv in ((120, 125.0), (2, 400.0), (37, 400.0), (200, 75.0)):
        st, p, dz = _domain(120, nz=nz, dz=dzv, cloudy_fraction=1.0, coherent=False)
        a, pa, b, pb = _both(gpu_mixed, oracle_mixed, 5.0, st, p, dz)
        assert_parity(a, b, what="nz=%d" % nz, flip_fraction=1e-3)
        np.testing.assert_allclose(pa, pb, rtol=1e-5, atol=1e-10)


def test_errors_are_returned_not_raised_across_the_abi(gpu_mixed):
    from kid_b200.kidmp import KidmpError
    st, p, dz = _domain(4, nz=60)
    with pytest.raises(KidmpError):
        gpu_mixed.step(-1.0, st, p, dz)
    big = {k: np.zeros((300, 2), np.float32) for k in FIELDS}
    with pytest.raises(KidmpError) as e:
        gpu_mixed.step(1.0, big, np.ones((300, 2), np.float32), np.ones(300, np.float32))
    assert "nz" in str(e.value)
    with pytest.raises(KeyError):
        gpu_mixed.get("no_such_table")
    # an empty domain is the reference's `do i = 1, nx` with nx = 0 (I:54): a successful no-op, nothing is touched
    empty = {k: np.zeros((60, 0), np.float32) for k in FIELDS}
    ppt = gpu_mixed.step(10.0, empty, np.zeros((60, 0), np.float32), np.full(60, 250.0, np.float32))
    assert ppt.shape == (4, 0)
    with pytest.raises(KidmpError):
        gpu_mixed._ck(gpu_mixed._L.kidmp_step(gpu_mixed.h, -3, 60, 10.0, 1, None, None, None, None))


def test_resident_time_series(gpu_mixed, oracle_mixed):
    """Surface precipitation and LWP / IWP series over 60 steps of dt = 10 s stay within 0.1 % (north_star)."""
    from kid_b200.shard import diag_from_state
    st, p, dz = _domain(1024, col0=300000, nx=1024)
    ref = {k: v.copy() for k, v in st.items()}
    gpu_mixed.state_alloc(1024, 60)
    gpu_mixed.upload(st, p, dz)
    gpu_mixed.diag()
    series_g, series_o = [], []
    cur = {k: v.copy() for k, v in st.items()}
    for n in range(60):
        gpu_mixed.step_resident(10.0)
        series_g.append(gpu_mixed.diag())
        ppt = oracle_mixed.step(10.0, ref, p, dz)
        series_o.append(diag_from_state(ref, p, dz, ppt))
    sg, so = np.array(series_g), np.array(series_o)
    for j, name in ((0, "rain"), (2, "snow"), (3, "graupel"), (4, "lwp"), (5, "iwp")):
        scale = np.abs(so[:, j]).max()
        if scale > 0:
            assert np.abs(sg[:, j] - so[:, j]).max() <= 1e-3 * scale, name
    gpu_mixed.download(cur)
    assert_parity(cur, ref, what="state after 60 steps", flip_fraction=5e-3)


def test_process_rate_buffer(gpu_mixed, oracle_mixed):
    """The 36 save_dg rates of M:2963-3120 through the optional device buffer."""
    import torch
    g = np.load(GOLD)
    ncol, nz = g["in/p"].shape[1], 60
    rates = torch.full((36, nz, ncol), float("nan"), dtype=torch.float32, device="cuda")
    gpu_mixed.set_rates_buffer(rates.data_ptr())
    s = {k: g["in/" + k].copy() for k in FIELDS}
    gpu_mixed.step(10.0, s, g["in/p"].copy(), g["in/dz"])
    gpu_mixed.set_rates_buffer(0)
    got = rates.cpu().numpy()
    assert gpu_mixed.rate_names == oracle_mixed.rate_names
    nbad = 0
    for j in range(ncol):
        out = oracle_mixed.column(10.0, *[g["in/" + k][:, j] for k in FIELDS], g["in/p"][:, j], g["in/dz"], want_rates=True)
        ref = out["rates"].astype(np.float32)
        active = np.isfinite(got[:, :, j]).all()
        if not active:                             # clear-sky column: kernel left the buffer untouched
            assert not ref.any()
            continue
        rel = np.abs(got[:, :, j] - ref) / np.maximum(np.abs(ref), 1e-30)
        rel = np.where(got[:, :, j] == ref, 0.0, rel)
        nbad += int((rel > 1e-5).sum())
    assert nbad <= 5


def test_host_side_process_rates(gpu_mixed):
    """kidmp_enable_rates / kidmp_get_rates (what the Fortran shim's save_dg calls are fed from): the same numbers as the
    caller's device buffer, zero for clear-sky columns, in both layouts."""
    import torch
    g = np.load(GOLD)
    ncol, nz = g["in/p"].shape[1], 60
    dev = torch.full((36, nz, ncol), float("nan"), dtype=torch.float32, device="cuda")
    gpu_mixed.set_rates_buffer(dev.data_ptr())
    s = {k: g["in/" + k].copy() for k in FIELDS}
    gpu_mixed.step(10.0, s, g["in/p"].copy(), g["in/dz"])
    gpu_mixed.set_rates_buffer(0)
    want = np.nan_to_num(dev.cpu().numpy(), nan=0.0)          # untouched (clear-sky) columns: no process at all
    gpu_mixed.enable_rates(True)
    try:
        s2 = {k: g["in/" + k].copy() for k in FIELDS}
        gpu_mixed.step(10.0, s2, g["in/p"].copy(), g["in/dz"])
        got = gpu_mixed.get_rates(ncol, nz, layout="col_fastest")
        got_k = gpu_mixed.get_rates(ncol, nz, layout="k_fastest")
    finally:
        gpu_mixed.enable_rates(False)
    for k in FIELDS:
        assert np.array_equal(s[k], s2[k]), k
    assert np.array_equal(got, want)
    assert np.array_equal(got_k, want.transpose(0, 2, 1))
    assert np.abs(want).max() > 0


@pytest.mark.parametrize("layout", ["col_fastest", "k_fastest"])
def test_multi_device_handle_equals_single_device(layout):
    """kidmp_config::ndev = 2: one handle, the columns cut into two ranges, one per GPU, no exchange on the data path.  Column
    by column the same bits as a single-device handle; kidmp_diag returns the NCCL all-reduced sums of both devices."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs in this process")
    from kid_b200 import synth
    from kid_b200.kidmp import Thompson
    ncol, nz = (150001, 60) if layout == "col_fastest" else (5003, 60)
    st, p, dz = synth.make_domain(ncol, nz=nz, col0=250000, nx=1024)
    conv = (lambda a: a.numpy().copy()) if layout == "col_fastest" else (lambda a: np.ascontiguousarray(a.numpy().T))
    one, two = Thompson(device=0), Thompson(devices=[0, 1])
    try:
        a = {k: conv(v) for k, v in st.items()}
        b = {k: conv(v) for k, v in st.items()}
        pa, pb = conv(p), conv(p)
        for _ in range(2):
            ppt_a = one.step(10.0, a, pa, dz.numpy(), layout=layout)
            ppt_b = two.step(10.0, b, pb, dz.numpy(), layout=layout)
        for k in FIELDS:
            assert np.array_equal(a[k], b[k]), k
        assert np.array_equal(ppt_a, ppt_b)
        da, db = one.diag(), two.diag()
        assert da[6] == db[6] and da[7] == db[7] == 2 * ncol
        assert np.allclose(da[:6], db[:6], rtol=1e-12)
        assert two._L.kidmp_num_devices(two.h) == 2
    finally:
        one.close(); two.close()


def test_pinned_host_arrays_get_only_the_changed_columns_back(gpu_mixed):
    """kidmp_step with pinned host arrays: the chunk pipeline writes the changed columns straight into them (k_scatter_host)
    instead of copying every column back.  Same bits as with pageable arrays, clear-sky columns untouched, and a clear-sky
    column in which a species <= R1 is zeroed (M:1412-1489) does come back."""
    import torch
    from kid_b200 import synth
    ncol, nz = 140000, 60
    st, p, dz = synth.make_domain(ncol, nz=nz, col0=200000, nx=1024)
    clear = np.flatnonzero(~(sum(st[k] for k in ("qc", "qi", "qr", "qs", "qg")) > 0).any(0).numpy())
    st["qs"][7, int(clear[5])] = 5e-13                       # below R1 in a clear-sky column: must come back as 0
    a = {k: v.numpy().copy() for k, v in st.items()}
    b = {k: v.clone().pin_memory() for k, v in st.items()}
    bn = {k: v.numpy() for k, v in b.items()}
    ppt_a = gpu_mixed.step(10.0, a, p.numpy().copy(), dz.numpy())
    assert gpu_mixed.step_stats()["zero_copy_return"] == 0
    ppt_b = gpu_mixed.step(10.0, bn, p.numpy().copy(), dz.numpy())
    assert gpu_mixed.step_stats()["zero_copy_return"] == 1
    for k in FIELDS:
        assert np.array_equal(a[k], bn[k]), k
    assert np.array_equal(ppt_a, ppt_b)
    assert bn["qs"][7, int(clear[5])] == 0.0 and a["qs"][7, int(clear[5])] == 0.0
    j = int(clear[9])
    assert all(np.array_equal(bn[k][:, j], st[k][:, j].numpy()) for k in FIELDS)


def test_step_device_on_a_torch_stream(gpu_mixed, oracle_mixed):
    import torch
    from kid_b200 import synth
    st, p, dz = synth.make_domain(3000, nz=60, cloudy_fraction=1.0, coherent=False, device="cuda")
    ref = {k: v.cpu().numpy().copy() for k, v in st.items()}
    ppt = torch.zeros((4, 3000), dtype=torch.float32, device="cuda")
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        gpu_mixed.step_device(3000, 60, 10.0, [st[k].data_ptr() for k in FIELDS], p.data_ptr(), dz.data_ptr(),
                              ppt.data_ptr(), stream=s.cuda_stream)
    s.synchronize()
    pb = oracle_mixed.step(10.0, ref, p.cpu().numpy(), dz.cpu().numpy())
    assert_parity({k: st[k].cpu().numpy() for k in FIELDS}, ref, what="step_device")
    np.testing.assert_allclose(ppt.cpu().numpy(), pb, rtol=1e-5, atol=1e-10)


def test_shards_equal_whole_domain(gpu_mixed):
    """An N-way column split must reproduce the whole-domain run column for column, bitwise (SURVEY 8e)."""
    from kid_b200.shard import shard_range
    st, p, dz = _domain(5000, col0=300000, nx=1024)
    whole = {k: v.copy() for k, v in st.items()}
    gpu_mixed.diag()
    pw = gpu_mixed.step(10.0, whole, p, dz)
    dw = gpu_mixed.diag()
    dsum = np.zeros(8)
    for r in range(3):
        c0, c1 = shard_range(5000, r, 3)
        part = {k: np.ascontiguousarray(v[:, c0:c1]) for k, v in st.items()}
        pp = gpu_mixed.step(10.0, part, np.ascontiguousarray(p[:, c0:c1]), dz)
        for k in FIELDS:
            assert np.array_equal(part[k], whole[k][:, c0:c1]), (r, k)
        assert np.array_equal(pp, pw[:, c0:c1])
        dsum += gpu_mixed.diag()
    np.testing.assert_allclose(dsum, dw, rtol=1e-12)


# ---- mphys_thompson09_interfacen (I:28-246) -----------------------------------------------------------------
def _kid_case(nx, nz, seed=7):
    from kid_b200 import synth
    rng = np.random.default_rng(seed)
    st, p, dz = synth.make_domain(nx, nz=nz, cloudy_fraction=1.0, coherent=False)
    p0, r_on_cp = 1.0e5, 287.05 / 1005.0
    T = st["t"].numpy().T.copy(); pk = p.numpy().T.copy()
    exner = ((pk / p0) ** r_on_cp).astype(np.float32)
    kid = {"theta": (T / exner).astype(np.float32), "exner": exner, "qv": st["qv"].numpy().T.copy(), "dz": dz.numpy()}
    kid["dtheta_adv"] = (1e-3 * rng.standard_normal((nx, nz))).astype(np.float32)
    kid["dtheta_div"] = (1e-4 * rng.standard_normal((nx, nz))).astype(np.float32)
    kid["dqv_adv"] = (1e-7 * rng.standard_normal((nx, nz))).astype(np.float32)
    kid["dqv_div"] = (1e-8 * rng.standard_normal((nx, nz))).astype(np.float32)
    for m in ("qc", "qr", "nr", "qi", "ni", "qs", "qg"):
        x = st[m].numpy().T.copy()
        kid[m] = x
        kid["d%s_adv" % m] = (x * 1e-3 * rng.standard_normal((nx, nz))).astype(np.float32)
        kid["d%s_div" % m] = (x * 1e-4 * rng.standard_normal((nx, nz))).astype(np.float32)
    return kid, p0, r_on_cp


def test_kid_interface_tendencies(gpu_mixed, oracle_mixed, gpu_warm, oracle_warm):
    from oracle.oracle import kid_interface, HYD_PLANES
    for g, o, nx, nz in ((gpu_mixed, oracle_mixed, 120, 120), (gpu_warm, oracle_warm, 1, 60), (gpu_mixed, oracle_mixed, 77, 60)):
        kid, p0, roc = _kid_case(nx, nz)
        a = g.kid_interface(kid, 5.0, p0, roc)
        b = kid_interface(o, kid, 5.0, p0, roc)
        warm = g.iiwarm
        names = ["dtheta_mphys", "dqv_mphys"] + ["d%s_mphys" % m for m in (HYD_PLANES[:3] if warm else HYD_PLANES)]
        # tendencies are differences of nearly equal states: compare them on the scale of state/dt
        scale = {"dtheta_mphys": 300.0 / 5.0, "dqv_mphys": kid["qv"].max() / 5.0}
        for m in HYD_PLANES:
            scale["d%s_mphys" % m] = max(float(np.abs(kid[m]).max()), 1e-12) / 5.0
        for n in names:
            err = np.abs(a[n].astype(np.float64) - b[n]).max() / scale[n]
            assert err < 2e-6, (n, err)
            assert (a[n] == b[n]).mean() > 0.98, n
        np.testing.assert_allclose(a["ppt"], b["ppt"], rtol=1e-5, atol=1e-10)


def test_pipelined_host_step_equals_resident_step(gpu_mixed, monkeypatch):
    """kidmp_step cuts large column-fastest domains into chunks that overlap H2D, kernels and D2H;
    chunking must not change a single bit (columns are independent)."""
    from kid_b200.kidmp import Thompson
    st, p, dz = _domain(5000, col0=300000, nx=1024)
    whole = {k: v.copy() for k, v in st.items()}
    pw = gpu_mixed.step(10.0, whole, p, dz)                    # 5000 < 2 * 65536: plain path
    monkeypatch.setenv("KIDMP_PIPE_CHUNK", "1024")
    t2 = Thompson(set_Nc=100.0, iiwarm=False, l_sediment=True)
    piped = {k: v.copy() for k, v in st.items()}
    pp = t2.step(10.0, piped, p, dz)                           # 5 chunks through the three-stream pipeline
    for k in FIELDS:
        assert np.array_equal(piped[k], whole[k]), k
    assert np.array_equal(pp, pw)
    d = t2.diag()
    assert d[7] == 5000
    t2.close()


@pytest.mark.parametrize("name", ["warm1", "deep1", "cu2d"])
def test_kinematic_case_time_series(name):
    """BASELINE configs 1-3 through the KiD-facing entry (kidmp_kid_interface) under a minimal kinematic host:
    surface precipitation and LWP / IWP time series of the CUDA path stay within 0.1 % of the oracle's over the
    whole case (north_star acceptance criterion; the host is kid_b200/kinematic.py because KiD's is not in the reference)."""
    from kid_b200 import kinematic as km
    from kid_b200.kidmp import Thompson
    from oracle.oracle import Oracle, kid_interface
    c = km.CASES[name]()
    g = Thompson(set_Nc=c.set_Nc, iiwarm=c.iiwarm)
    o = Oracle(set_Nc=c.set_Nc, iiwarm=c.iiwarm)
    rg = km.run(c, g.kid_interface)
    ro = km.run(c, lambda kid, dt, p0, roc: kid_interface(o, kid, dt, p0, roc))
    for key in ("lwp", "iwp"):
        scale = np.abs(ro[key]).max()
        if scale > 0:
            assert np.abs(rg[key] - ro[key]).max() <= 1e-3 * scale, (name, key, np.abs(rg[key] - ro[key]).max() / scale)
    acc_g, acc_o = np.cumsum(rg["ppt"], axis=0), np.cumsum(ro["ppt"], axis=0)      # accumulated surface precipitation
    for j in range(4):
        scale = np.abs(acc_o[:, j]).max()
        if scale > 0:
            assert np.abs(acc_g[:, j] - acc_o[:, j]).max() <= 1e-3 * scale, (name, "ppt", j)
    assert ro["lwp"].max() > 0.1 and (c.iiwarm or ro["iwp"].max() > 0.01)          # the case actually rained / glaciated
    g.close(); o.close()


def test_cxx_host_twin(gpu_mixed, tmp_path):
    """The C++ twin of KiD's `module mphys_thompson09n` (kid_b200/host): a no-argument `mphys_thompson09_interfacen()` over
    module-style state gives exactly what the library returns for the same columns, and reports the same save_dg records."""
    import subprocess
    from kid_b200 import build
    from kid_b200.kidmp import HYD_PLANES
    exe = build.build_host()
    nx, nz, dt = 40, 60, 5.0
    kid, p0, roc = _kid_case(nx, nz, seed=11)
    order = ["theta", "dtheta_adv", "dtheta_div", "exner", "qv", "dqv_adv", "dqv_div", "dz"]
    for m in HYD_PLANES:
        order += [m, "d%s_adv" % m, "d%s_div" % m]
    with open(tmp_path / "in.bin", "wb") as f:
        for name in order:
            np.ascontiguousarray(kid[name], np.float32).tofile(f)
    r = subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin"), str(nx), str(nz), str(dt), "0"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    # nx > 1: 5 means + 5 per-column records + total_ppt_level (I:248-308), and the 36 process rates of every level of every
    # column that mp_thompson itself saves (M:3046-3120)
    assert "save_dg_calls=%d" % (11 + 36 * nx * nz) in r.stdout
    out = np.fromfile(tmp_path / "out.bin", np.float32)
    roc = float(np.float32(287.05) / np.float32(1005.0))             # the driver's physconst defaults, evaluated in f32
    ref = gpu_mixed.kid_interface(kid, dt, 1.0e5, roc)
    n = nx * nz
    names = ["dtheta_mphys", "dqv_mphys"] + ["d%s_mphys" % m for m in HYD_PLANES]
    for j, name in enumerate(names):
        assert np.array_equal(out[j * n:(j + 1) * n].reshape(nx, nz), ref[name]), name
    assert np.array_equal(out[9 * n:].reshape(4, nx), ref["ppt"])


def test_negative_and_tiny_inputs_follow_the_reference_clamps(gpu_mixed, oracle_mixed):
    """No error path exists in the reference: negative or tiny hydrometeor values are clamped / zeroed exactly like
    M:1387-1493 does (species <= R1 zeroed with their numbers, qv floored at 1e-10), never rejected."""
    st, p, dz = _domain(2048, cloudy_fraction=1.0, coherent=False)
    rng = np.random.default_rng(3)
    for k in ("qc", "qi", "qr", "qs", "qg", "ni", "nr"):
        m = rng.random(st[k].shape) < 0.05
        st[k][m] = -np.abs(st[k][m]) - np.float32(1e-9)
        m = rng.random(st[k].shape) < 0.05
        st[k][m] = np.float32(3e-13)
    m = rng.random(st["qv"].shape) < 0.01
    st["qv"][m] = np.float32(-1e-6)
    st["nr"][rng.random(st["nr"].shape) < 0.05] = 0.0            # rain mass without a number: M:1447-1451 rebuilds it
    st["ni"][rng.random(st["ni"].shape) < 0.05] = 0.0
    a, pa, b, pb = _both(gpu_mixed, oracle_mixed, 10.0, st, p, dz)
    assert_parity(a, b, what="clamped inputs")
    np.testing.assert_allclose(pa, pb, rtol=1e-5, atol=1e-10)
    for k in ("qc", "qi", "qr", "qs", "qg", "ni", "nr"):
        assert a[k].min() >= 0.0, k
    assert a["qv"].min() >= 1e-10


def test_full_size_domain_properties(gpu_mixed, oracle_mixed):
    """BASELINE config 4 at full size (1 048 576 columns x 60 levels, resident in HBM): size-independent properties of the
    scheme, shard independence, and a 4 096-column random sample against the oracle."""
    import torch
    from kid_b200 import synth
    ncol, nz, dt = 1024 * 1024, 60, 10.0
    st, p, dz = synth.make_domain(ncol, nz=nz, nx=1024, device="cuda")
    before = {k: v.clone() for k, v in st.items()}
    ppt = torch.zeros((4, ncol), dtype=torch.float32, device="cuda")
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    gpu_mixed.diag()
    with torch.cuda.stream(s):
        gpu_mixed.step_device(ncol, nz, dt, [st[k].data_ptr() for k in FIELDS], p.data_ptr(), dz.data_ptr(), ppt.data_ptr(),
                              stream=s.cuda_stream)
    s.synchronize()
    d = gpu_mixed.diag()
    assert d[7] == ncol and 0.2 * ncol < d[6] < 0.4 * ncol                         # ~30 % cloudy columns
    # (1) clear-sky columns come back bit-unchanged (early RETURN, M:1540); cloudy ones changed somewhere
    hyd = sum(before[k] for k in ("qc", "qi", "qr", "qs", "qg"))
    clear = (hyd.max(0).values == 0)
    changed = torch.zeros(ncol, dtype=torch.bool, device="cuda")
    for k in FIELDS:
        changed |= (st[k] != before[k]).any(0)
    untouched = ~changed
    assert int(untouched.sum()) >= int(0.6 * ncol)
    assert bool((untouched | ~clear).all()) or int((clear & changed).sum()) < 0.02 * ncol   # clear + supersaturated wrt ice may nucleate
    assert not bool(ppt[:, untouched].any())
    # (2) output clamps (M:3623-3686)
    assert float(st["qv"].min()) >= 1e-10
    for k in ("qc", "qi", "qr", "qs", "qg"):
        q = st[k]
        assert bool(((q == 0) | (q > 1e-12)).all()), k
    assert bool((st["ni"][st["qi"] == 0] == 0).all()) and bool((st["nr"][st["qr"] == 0] == 0).all())
    rho = 0.622 * p / (287.04 * st["t"] * (st["qv"] + 0.622))
    assert float((st["ni"] * rho).max()) <= 499e3 * 1.001
    assert bool(torch.isfinite(torch.stack([st[k] for k in FIELDS])).all())
    # (3) column water budget on the air mass of the input state: vapour + condensate + what reached the ground.
    # The scheme moves mass per volume between levels with each level's own, mid-step density (M:3378-3389), so the
    # budget in mixing-ratio terms closes to the relative density change of the step, not to round-off.
    r0 = 0.622 * p.double() / (287.04 * before["t"].double() * (before["qv"].double() + 0.622))
    def water(state):
        return ((state["qv"] + state["qc"] + state["qr"] + state["qi"] + state["qs"] + state["qg"]).double() * r0 * dz.double()[:, None]).sum(0)
    w0, w1 = water(before), water(st) + ppt.double().sum(0)
    rel = ((w1 - w0).abs() / w0)
    assert float(torch.quantile(rel[::16].float(), 0.99)) < 1e-3      # 99 % of the columns close to 0.1 %
    assert float(rel.max()) < 0.1                                      # the rest are the reference's own clamp leaks (M:2291-2387, U10)
    assert abs(float(w1.sum() - w0.sum())) / float(w0.sum()) < 1e-3
    # (4) domain sums of kidmp_diag equal the sums over the returned arrays
    np.testing.assert_allclose(d[:4], ppt.double().sum(1).cpu().numpy(), rtol=1e-9)
    # (5) the two halves of the domain give bitwise the same columns as the whole (SURVEY 8e)
    half = ncol // 2
    for h0 in (0, half):
        part = {k: before[k][:, h0:h0 + half].contiguous() for k in FIELDS}
        pp = torch.zeros((4, half), dtype=torch.float32, device="cuda")
        ph = p[:, h0:h0 + half].contiguous()
        torch.cuda.synchronize()                   # the slices were made on torch's default stream, the step runs on `s`
        with torch.cuda.stream(s):
            gpu_mixed.step_device(half, nz, dt, [part[k].data_ptr() for k in FIELDS], ph.data_ptr(), dz.data_ptr(), pp.data_ptr(),
                                  stream=s.cuda_stream)
        s.synchronize()
        for k in FIELDS:
            assert torch.equal(part[k], st[k][:, h0:h0 + half]), (h0, k)
        assert torch.equal(pp, ppt[:, h0:h0 + half])
    # (6) a random sample of cloudy columns against the oracle
    g = torch.Generator(device="cpu").manual_seed(5)
    cloudy_idx = torch.nonzero(changed).flatten().cpu()
    pick = cloudy_idx[torch.randperm(cloudy_idx.numel(), generator=g)[:4096]].sort().values
    sample_in = {k: before[k][:, pick.cuda()].cpu().numpy().copy() for k in FIELDS}
    sample_out = {k: st[k][:, pick.cuda()].cpu().numpy() for k in FIELDS}
    pb = oracle_mixed.step(dt, sample_in, p[:, pick.cuda()].cpu().numpy().copy(), dz.cpu().numpy())
    assert_parity(sample_out, sample_in, what="4096 cloudy columns of the 1M-column run")
    np.testing.assert_allclose(ppt[:, pick.cuda()].cpu().numpy(), pb, rtol=1e-5, atol=1e-10)


def test_kid_text_cache_roundtrip(gpu_mixed, tmp_path):
    """KiD's list-directed lookup-table files (run_data/racg_thompson09.data, racs_thompson09.data; M:3710-3728,
    M:3857-3894): written in the order and element order of the reference's write statements, and read back exactly."""
    import subprocess
    from kid_b200.kidmp import Thompson
    racg, racs = str(tmp_path / "racg_thompson09.data"), str(tmp_path / "racs_thompson09.data")
    gpu_mixed.write_kid_cache(racg, racs)
    n_racg, n_racs = 28 * 28 * 37 * 37, 28 * 9 * 37 * 37
    assert int(subprocess.run(["wc", "-w", racg], capture_output=True, text=True).stdout.split()[0]) == 6 * n_racg
    assert int(subprocess.run(["wc", "-w", racs], capture_output=True, text=True).stdout.split()[0]) == 12 * n_racs
    head = np.array(open(racg).readline().split(), np.float64)          # first record starts with tcg_racg(1,1,1,1), (2,1,1,1) ...
    assert np.array_equal(head, gpu_mixed.get("tcg_racg")[:3])
    with open(racs) as f:                                               # second table of the file starts after n_racs values
        vals = []
        for line in f:
            vals.extend(line.split())
            if len(vals) > n_racs + 3:
                break
    assert np.array_equal(np.array(vals[n_racs:n_racs + 3], np.float64), gpu_mixed.get("tmr_racs1")[:3])
    t2 = Thompson(set_Nc=100.0, iiwarm=False, wp_double=True)           # slightly different bins => different tables
    assert not np.array_equal(t2.get("tcr_gacr"), gpu_mixed.get("tcr_gacr"))
    t2.read_kid_cache(racg, racs)
    for name in ("tcg_racg", "tmr_racg", "tcr_gacr", "tmg_gacr", "tnr_racg", "tnr_gacr", "tcs_racs1", "tmr_racs2", "tms_sacr2",
                 "tnr_racs1", "tnr_sacr2"):
        assert np.array_equal(t2.get(name), gpu_mixed.get(name)), name
    t2.close()


# ---- the WRF / MPAS-shaped entry, mp_gt_driver (M:806-1143) + calc_effectRad (M:4834-4935) ----------------------
def _wrf_case(ni, nk, nj, seed=3):
    """(i,k,j) arrays from the synthetic cloudy domain: theta and Exner function instead of T, layer depths that
    differ from column to column (terrain-following levels), accumulators with a history."""
    rng = np.random.default_rng(seed)
    st, p, dz = _domain(ni * nj, nz=nk, coherent=False, cloudy_fraction=0.6)
    to3 = lambda a: np.ascontiguousarray(a.reshape(nk, nj, ni).transpose(1, 0, 2))     # [k][col] -> (nj, nk, ni)
    f3 = {k: to3(st[k]) for k in ("qv", "qc", "qr", "qi", "qs", "qg", "ni", "nr")}
    p3 = to3(p)
    pii = ((p3 / 1.0e5) ** (287.04 / 1004.0)).astype(np.float32)
    f3["th"] = (to3(st["t"]) / pii).astype(np.float32)
    stretch = (0.8 + 0.4 * rng.random((nj, 1, ni))).astype(np.float32)
    dz3 = np.ascontiguousarray(np.broadcast_to(dz.reshape(1, nk, 1), (nj, nk, ni)) * stretch).astype(np.float32)
    acc = {k: (rng.random((nj, ni)) * 3.0).astype(np.float32) for k in
           ("rainnc", "rainncv", "sr", "snownc", "snowncv", "graupelnc", "graupelncv")}
    return f3, pii, p3, dz3, acc


def test_wrf_driver_entry(gpu_mixed, oracle_mixed):
    ni, nk, nj = 50, 60, 9
    f3, pii, p3, dz3, acc = _wrf_case(ni, nk, nj)
    a3 = {k: v.copy() for k, v in f3.items()}
    b3 = {k: v.copy() for k, v in f3.items()}
    aa = {k: v.copy() for k, v in acc.items()}
    ab = {k: v.copy() for k, v in acc.items()}
    ra = gpu_mixed.mp_gt_driver(20.0, a3, pii, p3, dz3, aa)
    rb = oracle_mixed.mp_gt_driver(20.0, b3, pii, p3, dz3, ab)
    flat = lambda d: {k: v.reshape(-1) for k, v in d.items()}
    names = ("qv", "qc", "qi", "qr", "qs", "qg", "ni", "nr", "th")
    assert_parity(flat(a3), flat(b3), fields=names, what="mp_gt_driver state")
    for k in ("rainnc", "rainncv", "sr", "snownc", "snowncv", "graupelnc", "graupelncv"):
        np.testing.assert_allclose(aa[k], ab[k], rtol=1e-5, atol=1e-9, err_msg=k)
    assert (aa["rainncv"] > 0).any()                                      # (no frozen precipitation reaches this 303 K surface)
    assert (aa["rainnc"] >= acc["rainnc"]).all()                         # accumulated, not overwritten
    # radii: inside the clamps of M:1118-1122, equal to the oracle's, and not all at the presets
    lim = {"re_cloud": (2.49e-6, 50e-6), "re_ice": (4.99e-6, 125e-6), "re_snow": (9.99e-6, 999e-6)}
    for k, (lo, hi) in lim.items():
        assert ra[k].min() >= np.float32(lo) and ra[k].max() <= np.float32(hi), k
        assert (ra[k] > np.float32(lo) * 1.01).any(), k
        # where the state agrees to the bit the radius must too (up to the f32 rounding of one power); the bit-exact check of
        # the radii against calc_effectRad of the returned state is tests/test_effective_radii.py
        np.testing.assert_allclose(ra[k], rb[k], rtol=2e-5, err_msg=k)
    # optional arguments absent: snow / graupel accumulators and radii are simply not produced
    a4 = {k: v.copy() for k, v in f3.items()}
    a_min = {k: acc[k].copy() for k in ("rainnc", "rainncv", "sr")}
    r4 = gpu_mixed.mp_gt_driver(20.0, a4, pii, p3, dz3, a_min, radii=False)
    assert r4 == {}
    for k in names:
        assert np.array_equal(a4[k], a3[k]), k
    assert np.array_equal(a_min["rainnc"], aa["rainnc"])
    # a shared dz vector through kidmp_step gives the same columns as the same depths passed per column
    f5, _, _, _, acc5 = _wrf_case(ni, nk, nj)
    dz_same = np.ascontiguousarray(np.broadcast_to(dz3[0, :, 0].reshape(1, nk, 1), (nj, nk, ni))).astype(np.float32)
    a5 = {k: v.copy() for k, v in f5.items()}
    gpu_mixed.mp_gt_driver(20.0, a5, pii, p3, dz_same, acc5, radii=False)
    st = {k: np.ascontiguousarray(f5[k].transpose(1, 0, 2).reshape(nk, nj * ni)) for k in f5 if k != "th"}
    st["t"] = np.ascontiguousarray((f5["th"] * pii).transpose(1, 0, 2).reshape(nk, nj * ni))
    pcol = np.ascontiguousarray(p3.transpose(1, 0, 2).reshape(nk, nj * ni))
    gpu_mixed.step(20.0, st, pcol, np.ascontiguousarray(dz3[0, :, 0]))
    for k in ("qv", "qc", "qi", "qr", "qs", "qg", "ni", "nr"):
        assert np.array_equal(st[k], a5[k].transpose(1, 0, 2).reshape(nk, nj * ni)), k


# ---- the step is launched over chunks of columns: the chunking must not change a bit -------------------------------
@pytest.mark.parametrize("dt,dz,warm,ncol,nz", [(10.0, 250.0, False, 20000, 60), (60.0, 100.0, False, 20000, 60),
                                                (30.0, 120.0, False, 20000, 60), (20.0, 60.0, True, 20000, 60),
                                                (10.0, 125.0, False, 77, 120), (5.0, 250.0, False, 1, 60),
                                                (10.0, 250.0, False, 140001, 37)])
def test_chunked_steps_are_bit_identical(dt, dz, warm, ncol, nz):
    """kidmp_set_option("chunk"): columns per launch of the step kernels (the work buffers are sized for one chunk).
    Columns are independent, so the state after several steps is the same bit for bit for every chunk size; so are the
    per-column precipitation amounts.  dt=60/dz=100 puts most rain columns on the sub-stepped sedimentation path."""
    import torch
    from kid_b200 import synth
    from kid_b200.kidmp import Thompson
    res = {}
    for chunk in (1 << 20, 4096, 1000, 32):
        if chunk == 32 and ncol > 20000:
            continue
        th = Thompson(set_Nc=100.0, iiwarm=warm, l_sediment=True)
        th.set_option("chunk", chunk)
        kw = dict(col0=200000) if ncol >= 20000 else dict(coherent=False, cloudy_fraction=1.0 if ncol == 1 else 0.6)
        st, p, dzv = synth.make_domain(ncol, nz=nz, nx=1024, device="cuda", dz=dz, **kw)
        ppt = torch.zeros((4, ncol), dtype=torch.float32, device="cuda")
        acc = torch.zeros((4, ncol), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        for _ in range(3):
            th.step_device(ncol, nz, dt, [st[k].data_ptr() for k in FIELDS], p.data_ptr(), dzv.data_ptr(), ppt.data_ptr())
            th.sync()
            acc += ppt.double()
            torch.cuda.synchronize()
        res[chunk] = ({k: st[k].cpu().numpy() for k in FIELDS}, acc.cpu().numpy(), th.diag())
        th.close()
    ref = res[1 << 20]
    for chunk, r in res.items():
        for k in FIELDS:
            assert np.array_equal(r[0][k], ref[0][k]), (chunk, k)
        assert np.array_equal(r[1], ref[1]), chunk
        assert r[2][6] == ref[2][6] and r[2][7] == ref[2][7]               # active columns, columns
        assert np.allclose(r[2][:6], ref[2][:6], rtol=1e-12)               # f64 sums: the order of the partial sums changes
    assert ref[2][6] > 0                                                   # some columns were active


@pytest.mark.gpu
@pytest.mark.parametrize("dt,dz", [(10.0, 250.0), (60.0, 100.0), (30.0, 120.0), (20.0, 250.0)])
def test_schedule_options_are_bit_identical(dt, dz):
    """The knobs that only change how a step is scheduled leave every bit of the result alone: "graphs" 0 (plain launches
    instead of a replayed CUDA graph), "simple" (columns in which no fall speed can cross the thinnest layer in one
    step skip k_carries: k_finish settles the snow speed of M:3301 and the top sedimenting levels of M:3208 on its own sweep),
    "timing" 1 / 2 (kernels one after the other / the normal schedule with events).  dt=60/dz=100 makes most precipitating
    columns non-simple, dt=10/dz=250 nearly all of them simple, the two in between a mix: both paths meet the same numbers."""
    import torch
    from kid_b200 import synth
    from kid_b200.kidmp import Thompson
    ncol, nz = 40000, 60
    res = {}
    for name, opts in (("default", {}), ("no_graph", {"graphs": 0}), ("no_simple", {"simple": 0}),
                       ("timing1", {"timing": 1}), ("timing2", {"timing": 2})):
        th = Thompson(set_Nc=100.0, iiwarm=False, l_sediment=True)
        for k, v in opts.items():
            th.set_option(k, v)
        st, p, dzv = synth.make_domain(ncol, nz=nz, nx=1024, device="cuda", dz=dz, col0=300000)
        ppt = torch.zeros((4, ncol), dtype=torch.float32, device="cuda")
        acc = torch.zeros((4, ncol), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        for _ in range(3):
            th.step_device(ncol, nz, dt, [st[k].data_ptr() for k in FIELDS], p.data_ptr(), dzv.data_ptr(), ppt.data_ptr())
            th.sync()
            acc += ppt.double()
        if name.startswith("timing"):
            ms = th.last_kernel_ms()
            assert set(ms) >= {"classify", "cells_ice", "finish"} and all(v >= 0.0 for v in ms.values())
        res[name] = ({k: st[k].cpu().numpy() for k in FIELDS}, acc.cpu().numpy(), th.diag(), th.step_stats())
        th.close()
    ref = res["default"]
    assert ref[2][6] > 0 and ref[1][0].sum() > 0                              # active columns, rain at the surface
    for name, r in res.items():
        for k in FIELDS:
            assert np.array_equal(r[0][k], ref[0][k]), (name, k)
        assert np.array_equal(r[1], ref[1]), name
        assert r[2][6] == ref[2][6] and r[2][7] == ref[2][7], name
        assert np.allclose(r[2][:6], ref[2][:6], rtol=1e-12), name
        assert r[3]["busy_cells"] == ref[3]["busy_cells"] and r[3]["cloudy_columns"] == ref[3]["cloudy_columns"], name
    if dt > 30.0:
        assert ref[3]["substep_columns"] > 0                                    # the sub-stepped path ran


@pytest.mark.gpu
@pytest.mark.parametrize("dt,dz,ncol", [(10.0, 250.0, 6000), (60.0, 100.0, 3000), (1.0, 250.0, 2000)])
def test_aerosol_aware_step(dt, dz, ncol, gpu_mixed, oracle_mixed):
    """The second half of SURVEY section 8f-4: is_aerosol_aware = .true. (M:28).  kidmp_step_device_aero against the oracle's
    restatement of the same switch on the same columns: prognostic nc / nwfa / nifa, aerosol scavenging by rain, snow and graupel
    (Eff_aero), dust nucleation (iceDeMott), homogeneous freezing of aerosols (iceKoop), droplet activation (activ_ncloud) and the
    evaporation of the smallest droplets (table_dropEvap), the surface emission of mp_gt_driver (M:1001).  Three steps, so the
    prognostic numbers of one step feed the next.  Tolerance as everywhere: 1e-5 relative, a few flipped cells allowed."""
    import torch
    from kid_b200 import synth
    st, p, dzv = synth.make_domain(ncol, nz=60, nx=1024, dz=dz, col0=123456, cloudy_fraction=0.7, coherent=False)
    nc, nwfa, nifa, w = synth.make_aerosols(st, p)
    nwfa2d = (np.random.default_rng(5).uniform(0.0, 1.0e5, ncol)).astype(np.float32)
    ref = {k: v.numpy().copy() for k, v in st.items()}
    rnc, rnwfa, rnifa = nc.copy(), nwfa.copy(), nifa.copy()
    pn, dzn = p.numpy().copy(), dzv.numpy().copy()
    dev = {k: v.cuda() for k, v in st.items()}
    dnc, dnwfa, dnifa, dw = (torch.from_numpy(x).cuda() for x in (nc, nwfa, nifa, w))
    dp, ddz, dn2 = p.cuda(), dzv.cuda(), torch.from_numpy(nwfa2d).cuda()
    dppt = torch.zeros((4, ncol), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    for step in range(3):
        ppt_ref = oracle_mixed.step_aero(dt, ref, rnc, rnwfa, rnifa, pn, w, dzn, nwfa2d=nwfa2d)
        gpu_mixed.step_device_aero(ncol, 60, dt, [dev[k].data_ptr() for k in FIELDS], dnc.data_ptr(), dnwfa.data_ptr(), dnifa.data_ptr(),
                                   dp.data_ptr(), dw.data_ptr(), ddz.data_ptr(), dppt.data_ptr(), nwfa2d_ptr=dn2.data_ptr())
        gpu_mixed.sync()
        got = {k: dev[k].cpu().numpy() for k in FIELDS}
        got.update(nc=dnc.cpu().numpy(), nwfa=dnwfa.cpu().numpy(), nifa=dnifa.cpu().numpy())
        want = dict(ref, nc=rnc, nwfa=rnwfa, nifa=rnifa)
        assert_parity(got, want, fields=FIELDS + ("nc", "nwfa", "nifa"), what="aerosol-aware step %d dt=%g" % (step, dt), flip_fraction=1e-3)
        np.testing.assert_allclose(dppt.cpu().numpy(), ppt_ref, rtol=1e-4, atol=1e-9)
        # the next step starts from the oracle's state on both sides: flipped cells do not accumulate
        for k in FIELDS:
            dev[k].copy_(torch.from_numpy(ref[k]))
        dnc.copy_(torch.from_numpy(rnc)); dnwfa.copy_(torch.from_numpy(rnwfa)); dnifa.copy_(torch.from_numpy(rnifa))
    # the switch does something: the droplet number is no longer Nt_c / rho where there is cloud
    cloud = ref["qc"] > 1e-9
    rho = 0.622 * pn / (287.04 * ref["t"] * (ref["qv"] + 0.622))
    assert cloud.any() and np.abs(rnc[cloud] * rho[cloud] / 100.0e6 - 1.0).max() > 0.05
    # the drop-evaporation table of the first aerosol-aware step (k_table_wev) against the oracle's table_dropEvap, M:4400-4439
    np.testing.assert_allclose(gpu_mixed.get("tnc_wev"), oracle_mixed.get("tnc_wev").ravel(order="F"), rtol=1e-12, atol=1e-300)
    # and the default path of the same handle is untouched by it
    a, pa, b, pb = _both(gpu_mixed, oracle_mixed, 10.0, *_domain(512, cloudy_fraction=1.0, coherent=False))
    assert_parity(a, b, what="default step after aerosol-aware steps", flip_fraction=1e-3)


@pytest.mark.gpu
def test_wrf_driver_entry_aerosol_aware(gpu_mixed, oracle_mixed):
    """kidmp_mp_gt_driver_aero: mp_gt_driver with is_aerosol_aware = .true. (M:807-832, M:950-956, M:999-1007, M:4874).  The
    reference side is put together from the oracle's pieces exactly as mp_gt_driver does: t = th*pii, mp_thompson per column
    with the aerosol arrays, surface emission into the lowest level, th = t/pii, calc_effectRad with the prognostic nc."""
    ni, nk, nj = 40, 60, 6
    f3, pii, p3, dz3, acc = _wrf_case(ni, nk, nj)
    dz_same = np.ascontiguousarray(np.broadcast_to(dz3[0, :, 0].reshape(1, nk, 1), (nj, nk, ni))).astype(np.float32)
    planes = lambda a: np.ascontiguousarray(a.transpose(1, 0, 2).reshape(nk, nj * ni))
    cube = lambda a: np.ascontiguousarray(a.reshape(nk, nj, ni).transpose(1, 0, 2))
    st = {k: planes(f3[k]) for k in f3 if k != "th"}
    st["t"] = planes(f3["th"] * pii)
    pcol = planes(p3)
    from kid_b200 import synth
    nc, nwfa, nifa, w = synth.make_aerosols(st, pcol, seed=99)
    nwfa2d = np.random.default_rng(7).uniform(0.0, 2.0e5, (nj, ni)).astype(np.float32)
    ae = {"nc": cube(nc), "nwfa": cube(nwfa), "nifa": cube(nifa), "w": cube(w), "nwfa2d": nwfa2d.copy()}
    a3 = {k: v.copy() for k, v in f3.items()}
    aa = {k: v.copy() for k, v in acc.items()}
    ra = gpu_mixed.mp_gt_driver(20.0, a3, pii, p3, dz_same, aa, aerosols=ae)
    # the oracle, piece by piece
    ppt = oracle_mixed.step_aero(20.0, st, nc, nwfa, nifa, pcol, w, np.ascontiguousarray(dz3[0, :, 0]), nwfa2d=nwfa2d.reshape(-1))
    want = {k: st[k] for k in ("qv", "qc", "qi", "qr", "qs", "qg", "ni", "nr")}
    want["th"] = planes(cube(st["t"]) / pii)
    want.update(nc=nc, nwfa=nwfa, nifa=nifa)
    got = {k: planes(a3[k]) for k in a3}
    got.update(nc=planes(ae["nc"]), nwfa=planes(ae["nwfa"]), nifa=planes(ae["nifa"]))
    assert_parity(got, want, fields=("qv", "qc", "qi", "qr", "qs", "qg", "ni", "nr", "th", "nc", "nwfa", "nifa"),
                  what="mp_gt_driver_aero", flip_fraction=1e-3)
    tot = ppt.sum(0).reshape(nj, ni)
    np.testing.assert_allclose(aa["rainncv"], tot, rtol=1e-4, atol=1e-9)
    # the cloud radius follows the prognostic droplet number: equal to the oracle's calc_effectRad fed with nc, and
    # different from what the fixed Nt_c gives (bit for bit, on the state the step returns: tests/test_effective_radii.py)
    rc_want = np.zeros((nk, nj * ni), np.float32)
    rc_fixed = np.zeros((nk, nj * ni), np.float32)
    for c in range(0, nj * ni, 7):
        args = (st["t"][:, c], pcol[:, c], st["qv"][:, c], st["qc"][:, c], st["qi"][:, c], st["ni"][:, c], st["qs"][:, c])
        rc_want[:, c] = np.clip(oracle_mixed.effect_rad(*args, nc=nc[:, c])[0], np.float32(2.49e-6), np.float32(50e-6))
        rc_fixed[:, c] = np.clip(oracle_mixed.effect_rad(*args)[0], np.float32(2.49e-6), np.float32(50e-6))
    sel = slice(0, nj * ni, 7)
    same_state = (got["qc"][:, sel] == want["qc"][:, sel]) & (got["nc"][:, sel] == want["nc"][:, sel]) & (got["th"][:, sel] == want["th"][:, sel]) \
        & (got["qv"][:, sel] == want["qv"][:, sel])
    np.testing.assert_allclose(planes(ra["re_cloud"])[:, sel][same_state], rc_want[:, sel][same_state], rtol=2e-5)
    assert (np.abs(rc_want[:, sel] - rc_fixed[:, sel]) > 1e-7).any()


@pytest.mark.gpu
def test_graph_replay_of_small_domains_is_bit_identical():
    """The fifteen launches of a step that fits one chunk are captured once in a CUDA graph and replayed while the arguments stay
    the same ("graphs" option): small domains are launch-bound.  Same bits as plain launches, over several steps, also when the
    arguments change in between (another dt: a new capture) and when the handle's work buffers grow (a larger domain)."""
    import torch
    from kid_b200 import synth
    from kid_b200.kidmp import Thompson
    res = {}
    for graphs in (1, 0):
        th = Thompson(set_Nc=100.0, iiwarm=False, l_sediment=True)
        th.set_option("graphs", graphs)
        out = []
        for ncol, dts in ((700, (10.0, 10.0, 10.0, 30.0, 30.0, 10.0)), (3000, (20.0, 20.0)), (700, (10.0, 10.0))):
            st, p, dzv = synth.make_domain(ncol, nz=60, nx=1024, device="cuda", col0=4242, cloudy_fraction=0.8, coherent=False)
            ppt = torch.zeros((4, ncol), dtype=torch.float32, device="cuda")
            acc = torch.zeros((4, ncol), dtype=torch.float64, device="cuda")
            for dt in dts:
                th.step_device(ncol, 60, dt, [st[k].data_ptr() for k in FIELDS], p.data_ptr(), dzv.data_ptr(), ppt.data_ptr())
                th.sync()
                acc += ppt.double()
            out.append(({k: st[k].cpu().numpy() for k in FIELDS}, acc.cpu().numpy()))
        res[graphs] = (out, th.diag(), th.gpu_launches)
        th.close()
    for (sa, pa), (sb, pb) in zip(res[1][0], res[0][0]):
        for k in FIELDS:
            assert np.array_equal(sa[k], sb[k]), k
        assert np.array_equal(pa, pb) and pa.sum() > 0
    assert np.array_equal(res[1][1], res[0][1])                                 # the domain sums too
    assert res[1][2] == res[0][2]                                               # and the launch count is the kernels' either way
