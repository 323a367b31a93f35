"""CPU-only exercise of the HOST layer (units, thresholds, operators, frequencies, wrapping, options)
with the device functions replaced by oracle stand-ins (tests/fake_device.py).  Kernel parity is the job
of the -m gpu tests; this file pins the glue above the C ABI without a GPU."""
import inspect

import numpy as np
import pytest

import fake_device
from oracle import xclim_oracle as O
from xb_helpers import make_field

import test_gpu_batch as batch   # reuse the oracle compositions of the 50 indicators


@pytest.fixture
def host(monkeypatch):
    fake_device.install(monkeypatch)


def test_batch_of_50_host_glue(host):
    from xclim_b200 import calendar as xcal, indices
    data = batch._inputs()
    units = {"tas": "K", "tasmax": "K", "tasmin": "K", "pr": "mm/d"}
    fields = {k: make_field(v, "1981-01-01", calendar="noleap", units=units[k]) for k, v in data.items()}
    for name, var in indices.BATCH_INDICATORS:
        da, x = fields[var], data[var]
        fn = getattr(indices, name)
        freq = inspect.signature(fn).parameters["freq"].default
        poff = da.time.period_offsets(freq)
        if name in ("tx90p", "tx10p", "tn90p"):
            per = 10.0 if name == "tx10p" else 90.0
            pdoy = xcal.select_percentile(xcal.percentile_doy(da, window=5, per=per), per)
            got = fn(da, pdoy)
            tab = O.percentile_doy(x, da.time.year, da.time.doy, 5, per)[:, 0]
            exp = O.doy_threshold_count(x, tab, da.time.doy, poff, "<" if name == "tx10p" else ">")
        else:
            got = fn(da)
            exp = batch._oracle(name, x, poff, da.time, data)
        exp = np.asarray(exp)
        assert got.values.shape == exp.shape, name
        assert "units" in got.attrs, name
        np.testing.assert_allclose(got.values, exp, rtol=1e-5, atol=1e-6, equal_nan=True, err_msg=name)


def test_unit_strings_and_operator_validation(host):
    from xclim_b200 import generic, indices
    rng = np.random.default_rng(3)
    pr = rng.gamma(0.5, 4.0, (365, 2, 3)).astype(np.float32)
    da = make_field(pr, "2001-01-01", calendar="noleap", units="mm/d")
    a = indices.wetdays(da, thresh="1 mm/day")
    b = indices.wetdays(make_field(pr / 86400.0, "2001-01-01", calendar="noleap", units="kg m-2 s-1"), thresh="1 mm/day")
    assert a.attrs["units"] == "d" and a.values.dtype == np.int64
    # the same physical threshold expressed in the data's units counts (almost) the same days
    assert np.abs(a.values - b.values).max() <= 1
    with pytest.raises(ValueError, match="not recognized"):
        generic.threshold_count(da, "=>", 1.0, "YS")
    with pytest.raises(ValueError, match="not permitted"):
        generic.threshold_count(da, "==", 1.0, "YS", constrain=(">", ">="))
    with pytest.raises(NotImplementedError):
        generic.spell_length_statistics(da, 1.0, 3, "sum", "<", "max", "YS", min_gap=2, resample_before_rl=False)
    for wr, op_, thr_ in (("sum", "<", 1.0), ("min", ">=", 0.5), ("mean", ">", 2.0)):      # window > 1 with min_gap
        out = generic.spell_length_statistics(da, thr_, 3, wr, op_, ["max", "count"], "YS", min_gap=3)
        for o, red in zip(out, ("max", "count")):
            exp = O.spell_length_statistics(pr, thr_, 3, wr, op_, red, da.time.period_offsets("YS"), min_gap=3)
            np.testing.assert_array_equal(o.values, exp, err_msg=f"{wr} {op_} {red}")
    out = generic.spell_length_statistics(da, 1.0, 1, None, "<", "max", "MS", min_gap=2)
    exp = O.spell_length_statistics(pr, 1.0, 1, None, "<", "max", da.time.period_offsets("MS"), min_gap=2)
    np.testing.assert_array_equal(out.values, exp)
    assert len(out.coords["time"]) == 12


def test_bootstrap_unequal_blocks_host_loop(host):
    """The N(N-1) virtual-row loop of bootstrapping.py on a standard calendar: same numbers as the oracle's
    literal block replacement (365 <-> 366 conversion)."""
    from xclim_b200 import calendar as xcal, indices
    rng = np.random.default_rng(4)
    T = 366 + 365 * 3 + 366                      # 2000 .. 2004
    t = np.arange(T)
    x = (288 + 10 * np.sin(2 * np.pi * t / 365.25)[:, None] + 3 * rng.standard_normal((T, 3))).astype(np.float32)
    da = make_field(x, "2000-01-01", calendar="standard", units="K")
    base = da.isel_time(da.time.sel_years(2001, 2004))
    pdoy = xcal.select_percentile(xcal.percentile_doy(base, window=5, per=90.0), 90.0)
    got = indices.tx90p(da, pdoy, freq="YS", bootstrap=True)
    exp = O.bootstrap_doy_count(x, da.time.year, da.time.doy, da.time.period_offsets("YS"), (2001, 2004), window=5,
                                per=90.0, op=">", cal_max_doy=366)
    np.testing.assert_array_equal(got.values, exp)
    assert got.values.dtype == np.float64 and got.attrs["units"] == "d"


def test_more_index_entry_points(host):
    """Thin entry points added over the existing kernels: oracle compositions of the reference bodies."""
    from xclim_b200 import indices
    data = batch._inputs()
    K0 = 273.15
    mk = lambda k, u: make_field(data[k], "1981-01-01", calendar="noleap", units=u)  # noqa: E731
    pr, tx, tn = mk("pr", "mm/d"), mk("tasmax", "K"), mk("tasmin", "K")
    poff = pr.time.period_offsets("YS")
    # wet spells (indices/_threshold.py:3596-3733)
    np.testing.assert_array_equal(indices.wet_spell_total_length(pr).values,
                                  O.spell_length_statistics(data["pr"], 1.0, 3, "sum", ">=", "sum", poff))
    np.testing.assert_array_equal(indices.wet_spell_max_length(pr).values,
                                  O.spell_length_statistics(data["pr"], 1.0, 1, "sum", ">=", "max", poff))
    # warm days / nights (:2674-2745): thresholds in degC against data in K
    np.testing.assert_array_equal(indices.warm_day_frequency(tx).values,
                                  O.threshold_count(data["tasmax"], ">", 30 + K0, poff))
    np.testing.assert_array_equal(indices.warm_night_frequency(tn, thresh="5 degC").values,
                                  O.threshold_count(data["tasmin"], ">", 5 + K0, poff))
    # extreme temperature range (_multivariate.py:601-637)
    etr = indices.extreme_temperature_range(tn, tx, freq="MS")
    pm = pr.time.period_offsets("MS")
    exp = O.select_resample_op(data["tasmax"].astype(np.float64), "max", pm) - \
        O.select_resample_op(data["tasmin"].astype(np.float64), "min", pm)
    np.testing.assert_allclose(etr.values, exp, rtol=1e-6, equal_nan=True)
    assert etr.attrs["units"] == "K" and etr.attrs["units_metadata"] == "temperature: difference"
    # days with snow (_threshold.py:1817-1860): low < prsn <= high
    prsn = make_field((data["pr"] / 86400.0).astype(np.float32), "1981-01-01", calendar="noleap", units="kg m-2 s-1")
    got = indices.days_with_snow(prsn, low="1e-5 kg m-2 s-1", high="1e-4 kg m-2 s-1")
    x = prsn.values
    pj = prsn.time.period_offsets("YS-JUL")
    exp = np.stack([((x[s:e] > np.float32(1e-5)) & (x[s:e] <= np.float32(1e-4))).sum(0) for s, e in zip(pj[:-1], pj[1:])])
    np.testing.assert_array_equal(got.values, exp)
    assert got.attrs["units"] == "d"
    # wind maxima
    w = make_field(np.abs(data["tas"] - 270).astype(np.float32), "1981-01-01", calendar="noleap", units="m s-1")
    np.testing.assert_allclose(indices.sfcWindmax_max(w).values, O.select_resample_op(w.values.astype(np.float64), "max", poff))


def test_days_over_precip_thresh(host):
    """indices/_multivariate.py:1223-1233: the per-doy percentile clamped from below by the wet-day
    threshold, then the doy-threshold count."""
    from xclim_b200 import calendar as xcal, indices
    rng = np.random.default_rng(7)
    pr = rng.gamma(0.4, 6.0, size=(365 * 4, 2, 3)).astype(np.float32)
    pr[rng.random(pr.shape) < 0.5] = 0
    pr[rng.random(pr.shape) < 0.01] = np.nan
    da = make_field(pr, "1981-01-01", calendar="noleap", units="mm/d")
    per = xcal.select_percentile(xcal.percentile_doy(da, window=5, per=75.0), 75.0)
    tab = O.percentile_doy(pr, da.time.year, da.time.doy, 5, 75.0)[:, 0]
    for freq in ("YS", "MS"):
        poff = da.time.period_offsets(freq)
        got = indices.days_over_precip_thresh(da, per, thresh="1 mm/day", freq=freq)
        tp = np.where(tab > 1.0, tab, 1.0)
        exp = O.doy_threshold_count(pr, tp, da.time.doy, poff, ">")
        np.testing.assert_array_equal(got.values, exp)
        assert got.values.dtype == np.int64 and got.attrs["units"] == "d"
    # the clamp matters: many doy percentiles of this dry series are below 1 mm/d
    assert (tab < 1.0).any() and (tab > 1.0).any()


@pytest.mark.parametrize("freq", ["YS", "MS"])
def test_bootstrap_equal_blocks_host_logic(host, freq):
    """bootstrapping.py on a noleap calendar: base slice, step -> period map, merge of in-base (bootstrapped)
    and out-of-base (plain) periods, error behaviour -- against the oracle's literal bootstrap."""
    from xclim_b200 import calendar as xcal, indices
    rng = np.random.default_rng(8)
    T = 365 * 6
    t = np.arange(T)
    x = (288 + 10 * np.sin(2 * np.pi * t / 365)[:, None] + 3 * rng.standard_normal((T, 2))).astype(np.float32)
    da = make_field(x, "1981-01-01", calendar="noleap", units="K")
    base = da.isel_time(da.time.sel_years(1982, 1985))
    pdoy = xcal.select_percentile(xcal.percentile_doy(base, window=5, per=90.0), 90.0)
    got = indices.tx90p(da, pdoy, freq=freq, bootstrap=True)
    exp = O.bootstrap_doy_count(x, da.time.year, da.time.doy, da.time.period_offsets(freq), (1982, 1985), window=5,
                                per=90.0, op=">")
    np.testing.assert_array_equal(got.values, exp)
    plain = indices.tx90p(da, pdoy, freq=freq).values
    yrs = np.array([int(s[:4]) for s in da.time.period_labels(freq)])
    outside = (yrs < 1982) | (yrs > 1985)
    np.testing.assert_array_equal(got.values[outside], plain[outside])
    p_all = xcal.select_percentile(xcal.percentile_doy(da, per=90.0), 90.0)
    with pytest.raises(KeyError, match="all years are overlapping"):
        indices.tx90p(da, p_all, bootstrap=True)


def test_eqm_host_wrapper(host):
    """sdba.EmpiricalQuantileMapping: train / ds / adjust wrapping (dims, coords, dtype, errors)."""
    from xclim_b200 import sdba
    rng = np.random.default_rng(9)
    T, shape = 730, (2, 3)
    ref = (285 + 6 * rng.standard_normal((T,) + shape)).astype(np.float32)
    hist = (286.5 + 7 * rng.standard_normal((T,) + shape)).astype(np.float32)
    sim = (288.5 + 7 * rng.standard_normal((T,) + shape)).astype(np.float32)
    f = lambda a: make_field(a, "1981-01-01", calendar="noleap", units="K")  # noqa: E731
    qm = sdba.EmpiricalQuantileMapping.train(f(ref), f(hist), nquantiles=15, kind="+", group="time")
    ds = qm.ds
    assert ds["af"].values.shape == (15,) + shape and ds["hist_q"].dims[0] == "quantiles"
    np.testing.assert_allclose(ds["af"].coords["quantiles"], sdba.equally_spaced_nodes(15), rtol=1e-6)
    af, hq = O.eqm_train(ref, hist, 15, "+")
    np.testing.assert_allclose(ds["af"].values, af, rtol=1e-5, atol=1e-5)
    scen = qm.adjust(f(sim), interp="linear")
    np.testing.assert_allclose(scen.values, O.eqm_adjust(sim, af, hq, "+", "linear"), rtol=1e-5)
    assert scen.values.dtype == np.float32 and scen.values.shape == sim.shape and scen.attrs["units"] == "K"
    with pytest.raises(NotImplementedError):
        sdba.EmpiricalQuantileMapping.train(f(ref), f(hist), group="time.month")
    with pytest.raises(ValueError):
        sdba.EmpiricalQuantileMapping.train(f(ref), f(hist), kind="-")
    with pytest.raises(NotImplementedError):
        qm.adjust(f(sim), interp="cubic")


# ---- the bodies of the GPU parity tests, run on the CPU over the oracle-backed device functions -------------
# Every GPU test that talks to the package only through its public host API (no explicit .cuda() tensors,
# no error raised by the C library itself) is executed here as well: the comparison against the oracle is
# then trivial for the kernels, but every line of host code on the way (unit conversion, operator codes,
# period offsets, date ranges of the season functions, missing-value masks, bootstrap bookkeeping, wrapping)
# runs in the GPU-less suite too.
GPU_BODIES = {
    "test_gpu_missing": ["test_indicator_level_entry_points_apply_missing_any", "test_missing_masks"],
    "test_gpu_seasons": ["test_date_bounded_runs_parity", "test_growing_season_reference_known_answers",
                         "test_season_parity"],
    "test_gpu_boundary": ["test_first_last_run"],
    "test_gpu_period_stats": ["test_bivariate_heat_waves", "test_cdd_reference_known_answers",
                              "test_hot_spell_max_magnitude", "test_resample_reductions",
                              "test_run_length_module_masks", "test_run_length_quantile_reducers",
                              "test_run_length_reference_known_answers", "test_select_time_indexers_on_resample_ops",
                              "test_spell_length_statistics_window1", "test_threshold_count_all_ops"],
    "test_gpu_rolling_spells_eqm": ["test_dry_spell_reference_known_answers", "test_eqm_train_adjust",
                                    "test_rolling_reference_known_answers", "test_rolling_resample",
                                    "test_spell_length_statistics_min_gap", "test_spell_length_statistics_windows",
                                    "test_spell_mask_reference_truth_tables"],
    "test_gpu_bootstrap": ["test_bootstrap_error_behaviour", "test_bootstrap_matches_literal_restatement",
                           "test_bootstrap_standard_calendar_365_366_blocks"],
    "test_gpu_percentile": ["test_percentile_doy_mid_percentiles_selection_kernel",
                            "test_percentile_doy_reference_known_answers",
                            "test_percentile_doy_standard_calendar_and_366", "test_tx90p_counts",
                            "test_tx90p_reference_known_answer_leap_year"],
}
MAX_COMBOS = 4   # per test function: the oracle is slow, the host code paths repeat


def _gpu_body_cases():
    import importlib
    cases = []
    for mod, names in GPU_BODIES.items():
        m = importlib.import_module(mod)
        for name in names:
            fn = getattr(m, name)
            combos = [{}]
            for mk in [k for k in getattr(fn, "pytestmark", []) if k.name == "parametrize"]:
                keys = [n.strip() for n in mk.args[0].split(",")]
                grown = []
                for c in combos:
                    for val in mk.args[1]:
                        vals = tuple(val) if (isinstance(val, (tuple, list)) and len(keys) > 1) else (val,)
                        grown.append({**c, **dict(zip(keys, vals))})
                combos = grown
            step = max(1, len(combos) // MAX_COMBOS)
            for i, c in enumerate(combos[::step][:MAX_COMBOS]):
                cases.append(pytest.param(mod, name, c, id=f"{mod[9:]}.{name[5:]}-{i}"))
    return cases


@pytest.mark.parametrize("mod,name,kwargs", _gpu_body_cases())
def test_gpu_test_bodies_over_oracle_backed_device(host, mod, name, kwargs):
    import importlib
    getattr(importlib.import_module(mod), name)(None, **kwargs)


def test_atmos_generic_missing_any_wrapper(host):
    """atmos.<index> built by with_missing_any: the index value, NaN where the period has a missing step in
    ANY time-dependent input (core/indicator.py:1522-1549 + core/missing.py:310-322)."""
    from xclim_b200 import atmos, indices
    data = batch._inputs()                                     # 0.3 % NaN scattered in every variable
    units = {"tas": "K", "tasmax": "K", "tasmin": "K", "pr": "mm/d"}
    f = {k: make_field(v, "1981-01-01", calendar="noleap", units=units[k]) for k, v in data.items()}
    for name, var in [("frost_days", "tasmin"), ("dry_spell_frequency", "pr"), ("growing_degree_days", "tas"),
                      ("tx_max", "tasmax")]:
        freq = "MS"
        got = getattr(atmos, name)(f[var], freq=freq).values
        ref = getattr(indices, name)(f[var], freq=freq).values.astype(np.float64)
        miss = O.missing_any(data[var], f[var].time.period_offsets(freq))
        assert miss.any() and not miss.all()
        np.testing.assert_array_equal(np.isnan(got), miss | np.isnan(ref), err_msg=name)
        np.testing.assert_array_equal(got[~miss], ref[~miss], err_msg=name)
    # two time-dependent inputs: either one missing masks the period
    got = atmos.heat_wave_frequency(f["tasmin"], f["tasmax"], freq="MS") if hasattr(atmos, "heat_wave_frequency") else None
    hw = atmos.with_missing_any(indices.heat_wave_frequency)(f["tasmin"], f["tasmax"], freq="MS").values
    poff = f["tasmin"].time.period_offsets("MS")
    both = O.missing_any(data["tasmin"], poff) | O.missing_any(data["tasmax"], poff)
    np.testing.assert_array_equal(np.isnan(hw), both)
    assert got is None or np.array_equal(np.isnan(got.values), both)


def test_missing_masks_on_partly_covered_periods(host):
    """expected_count (core/missing.py:64-160): 400 days from 2000-01-01 -> 2001 holds 34 of 365 days."""
    from xclim_b200 import missing
    x = np.ones((400, 2), np.float32)
    x[10, 1] = np.nan
    da = make_field(x, "2000-01-01", units="K")
    np.testing.assert_array_equal(missing.missing_any(da, "YS").values, [[False, True], [True, True]])
    np.testing.assert_array_equal(missing.missing_pct(da, "YS", 0.5).values, [[False, False], [True, True]])
    np.testing.assert_array_equal(missing.missing_pct(da, "YS", 0.002).values, [[False, True], [True, True]])
    np.testing.assert_array_equal(missing.at_least_n_valid(da, "YS", 30).values, [[False, False], [False, False]])
    np.testing.assert_array_equal(missing.at_least_n_valid(da, "YS", 35).values, [[False, False], [True, True]])
    np.testing.assert_array_equal(missing.missing_wmo(da, "YS").values, [[False, False], [True, True]])
    # monthly: February 2001 holds 3 of its 28 days -> 25 missing days >= nm
    m = missing.missing_wmo(da, "MS").values
    assert not m[:13].any() and m[13].all()
    a = missing.missing_any(da, "MS").values
    assert a[0, 1] and not a[0, 0] and a[13].all() and not a[1:13].any()


def test_atmos_check_missing_options(host):
    """set_options(check_missing=..., missing_options=...) selects the criterion of atmos.* (core/options.py)."""
    import xclim_b200
    from xclim_b200 import atmos, indices
    a = np.arange(360.0)
    a[5:7] = np.nan           # 2 of 31 days missing in July
    a[40:45] = np.nan         # 5 consecutive days missing in August
    ts = make_field((a + 280).astype(np.float32), "2000-07-01", units="K")
    raw = indices.tg_max(ts, freq="MS").values
    assert np.isnan(atmos.tg_max(ts, freq="MS").values[:2]).all()                       # any
    with xclim_b200.set_options(check_missing="pct", missing_options={"tolerance": 0.1}):
        out = atmos.tg_max(ts, freq="MS").values
        assert out[0] == raw[0] and np.isnan(out[1])
    with xclim_b200.set_options(check_missing="wmo"):
        out = atmos.tg_max(ts, freq="MS").values
        assert out[0] == raw[0] and np.isnan(out[1])
    with xclim_b200.set_options(check_missing="at_least_n", missing_options={"n": 28}):
        out = atmos.tg_max(ts, freq="MS").values
        assert out[0] == raw[0] and np.isnan(out[1])
    with xclim_b200.set_options(check_missing="skip"):
        np.testing.assert_array_equal(atmos.tg_max(ts, freq="MS").values, raw)
    assert xclim_b200.options.OPTIONS["check_missing"] == "any"


def test_atmos_fused_entry_points_honour_check_missing(host):
    """The three hand-fused indicators (cdd, tg_mean, tx90p) follow set_options(check_missing=...) like the
    generic ``with_missing_any`` wrappers (ADVICE r1: they always applied MissingAny)."""
    import xclim_b200
    from xclim_b200 import atmos, calendar as xcal, indices
    rng = np.random.default_rng(21)
    T = 365 * 3
    x = (285 + 5 * rng.standard_normal((T, 2))).astype(np.float32)
    x[400:403, 0] = np.nan                      # 3 missing days in year 2 of cell 0
    tas = make_field(x, "2001-01-01", calendar="noleap", units="K")
    pr = make_field(np.abs(x - 285).astype(np.float32), "2001-01-01", calendar="noleap", units="mm/d")
    per = xcal.select_percentile(xcal.percentile_doy(tas, window=5, per=90.0), 90.0)
    cases = [(atmos.tg_mean, indices.tg_mean, (tas,), {}),
             (atmos.maximum_consecutive_dry_days, indices.maximum_consecutive_dry_days, (pr,), {}),
             (atmos.tx90p, indices.tx90p, (tas, per), {})]
    for ind, idx, args, kw in cases:
        raw = np.asarray(idx(*args, **kw).values, dtype=np.float64)
        assert np.isnan(ind(*args, **kw).values[1, 0])                                   # default: any
        with xclim_b200.set_options(check_missing="skip"):
            np.testing.assert_allclose(ind(*args, **kw).values, raw, rtol=1e-6)
        with xclim_b200.set_options(check_missing="pct", missing_options={"tolerance": 0.05}):
            out = ind(*args, **kw).values
            assert not np.isnan(out).any() and np.allclose(out, raw, rtol=1e-6)
        with xclim_b200.set_options(check_missing="at_least_n", missing_options={"n": 364}):
            assert np.isnan(ind(*args, **kw).values[1, 0])


def test_bootstrap_converts_table_units(host):
    """degC data against a K percentile table with bootstrap=True: the out-of-base periods are counted
    against the table converted to the data units (indices/_multivariate.py:1583; ADVICE r1)."""
    from xclim_b200 import calendar as xcal, indices
    rng = np.random.default_rng(22)
    T = 365 * 5
    t = np.arange(T)
    xk = (288 + 10 * np.sin(2 * np.pi * t / 365)[:, None] + 3 * rng.standard_normal((T, 3))).astype(np.float32)
    da_k = make_field(xk, "1981-01-01", calendar="noleap", units="K")
    # exactly representable shift so that both unit systems see the same ordering
    da_c = make_field((xk - np.float32(273.15)).astype(np.float32), "1981-01-01", calendar="noleap", units="degC")
    base_k = da_k.isel_time(da_k.time.sel_years(1982, 1984))
    per_k = xcal.select_percentile(xcal.percentile_doy(base_k, window=5, per=90.0), 90.0)
    got_c = indices.tx90p(da_c, per_k, freq="YS", bootstrap=True).values
    plain_c = indices.tx90p(da_c, per_k, freq="YS").values
    # out-of-base years (1981, 1985): bootstrap == plain count (tests/test_bootstrapping.py:69-71), and the
    # plain count itself is sane (about 10 % of days, not 0 or 365 as with an unconverted K table)
    np.testing.assert_array_equal(got_c[[0, 4]], plain_c[[0, 4]])
    assert (plain_c[[0, 4]] > 5).all() and (plain_c[[0, 4]] < 120).all()


def _check_run_batch_against_single_calls(exact=True, fields=None, names=None):
    """indices.run_batch (fused passes) == the one-call-per-indicator functions: values, dtypes, dims, attrs.
    (exact=False: the oracle stand-ins of the CPU suite sum in different precisions.)  ``fields`` default to the
    batch inputs on a 4 x 8 grid; ``names`` runs a subset of BATCH_INDICATORS."""
    from xclim_b200 import calendar as xcal, indices
    if fields is None:
        data = batch._inputs()
        units = {"tas": "K", "tasmax": "K", "tasmin": "K", "pr": "mm/d"}
        fields = {k: make_field(v, "1981-01-01", calendar="noleap", units=units[k]) for k, v in data.items()}
    per_of = {"tx90p": ("tasmax", 90.0), "tx10p": ("tasmax", 10.0), "tn90p": ("tasmin", 90.0)}
    want = [(n, v) for n, v in indices.BATCH_INDICATORS if names is None or n in names]
    pers = {(var, p_): xcal.select_percentile(xcal.percentile_doy(fields[var], window=5, per=p_), p_)
            for var, p_ in sorted({per_of[n] for n, _ in want if n in per_of})}
    fused = indices.run_batch(fields, pers, names=names)
    assert list(fused) == [n for n, _ in want]
    n_fused = 0
    for name, var in want:
        fn = getattr(indices, name)
        ref = fn(fields[var], pers[per_of[name]]) if name in per_of else fn(fields[var])
        got = fused[name]
        assert got.dims == ref.dims and got.values.dtype == ref.values.dtype, name
        if exact or np.issubdtype(ref.values.dtype, np.integer):
            np.testing.assert_array_equal(got.values, ref.values, err_msg=name)
        else:
            np.testing.assert_allclose(got.values, ref.values, rtol=2e-6, equal_nan=True, err_msg=name)
        assert got.attrs == ref.attrs, (name, got.attrs, ref.attrs)
        n_fused += indices.BATCH_FUSED[name] is not None
    if names is None:
        assert n_fused >= 42


def test_run_batch_fused_passes_host_logic(host):
    _check_run_batch_against_single_calls(exact=False)


def _check_reference_default_call_shapes():
    """Call shapes that used to raise (VERDICT r1): freq=None (the reference default of the run-length functions,
    indices/run_length.py:275-335), index="last" (run_length.py:223-272), array thresholds in threshold_count
    (indices/generic.py:329-335), tuple spell_reducer (generic.py:555-585)."""
    from xclim_b200 import Field, generic, run_length as rl
    rng = np.random.default_rng(33)
    T, shape = 365 * 2 + 30, (2, 3)
    x = rng.gamma(0.5, 4.0, (T,) + shape).astype(np.float32)
    x[rng.random(x.shape) < 0.01] = np.nan
    da = make_field(x, "2001-01-01", calendar="noleap", units="mm/d")
    mask = make_field((x > 1.0).astype(np.float32), "2001-01-01", calendar="noleap", units="")
    m = x > 1.0
    whole = np.array([0, T])
    # ---- freq=None: the statistic of the whole series, no time dimension
    for red, win in (("max", 1), ("sum", 3), ("count", 2), ("mean", 1), ("std", 1)):
        got = rl.rle_statistics(mask, red, win)            # freq=None is the default
        assert got.dims == da.dims[1:] and got.values.shape == shape
        exp = O.resample_and_rl(m, True, O.rle_statistics, poff=whole, reducer=red, window=win)[0]
        np.testing.assert_allclose(got.values, exp, rtol=1e-6)
    np.testing.assert_array_equal(rl.longest_run(mask).values,
                                  O.resample_and_rl(m, True, O.rle_statistics, poff=whole, reducer="max", window=1)[0])
    np.testing.assert_array_equal(rl.windowed_run_count(mask, 3).values,
                                  O.resample_and_rl(m, True, O.rle_statistics, poff=whole, reducer="sum", window=3)[0])
    fr = rl.first_run(mask, 3)
    np.testing.assert_array_equal(fr.values, O.first_run(m, 3, poff=whole)[0])
    assert fr.dims == da.dims[1:]
    cd = generic.cumulative_difference(da, 1.0, ">", freq=None)
    np.testing.assert_allclose(cd.values, O.cumulative_difference(x, 1.0, ">", whole)[0], rtol=1e-5)
    # ---- index="last": a run counts for the period of its last element
    poff = da.time.period_offsets("MS")
    got = rl.rle_statistics(mask, "max", 1, freq="MS", index="last").values
    exp = np.zeros((len(poff) - 1,) + shape, np.float32)
    for idx in np.ndindex(shape):
        col = m[(slice(None),) + idx]
        t = 0
        while t < T:
            if col[t]:
                e = t
                while e + 1 < T and col[e + 1]:
                    e += 1
                p = np.searchsorted(poff, e, side="right") - 1
                exp[(p,) + idx] = max(exp[(p,) + idx], e - t + 1)
                t = e + 1
            else:
                t += 1
    np.testing.assert_array_equal(got, exp)
    first = rl.rle_statistics(mask, "max", 1, freq="MS", index="first").values
    assert (first != got).any()
    with pytest.raises(ValueError):
        rl.rle_statistics(mask, "max", 1, freq="MS", index="middle")
    # ---- array thresholds: per cell and per time step, compared in float64
    thr_cell = (0.5 + rng.random(shape)).astype(np.float64)
    thr_full = (0.5 + rng.random((T,) + shape)).astype(np.float64)
    poff_y = da.time.period_offsets("YS")
    with np.errstate(invalid="ignore"):
        exp_cell = np.stack([(x[a:b].astype(np.float64) > thr_cell).sum(0) for a, b in O._groups(poff_y)])
        exp_full = np.stack([(x[a:b].astype(np.float64) >= thr_full[a:b]).sum(0) for a, b in O._groups(poff_y)])
    got = generic.threshold_count(da, ">", Field(thr_cell, da.dims[1:], None, {}, {}), "YS")
    np.testing.assert_array_equal(got.values, exp_cell)
    assert got.values.dtype == np.int64
    np.testing.assert_array_equal(generic.threshold_count(da, ">=", thr_full, "YS").values, exp_full)
    swapped = Field(np.moveaxis(thr_full, 0, -1).copy(), da.dims[1:] + ("time",), da.time, {}, {})
    np.testing.assert_array_equal(generic.threshold_count(da, ">=", swapped, "YS").values, exp_full)
    with pytest.raises(ValueError):
        generic.threshold_count(da, ">", np.zeros((3, 3)), "YS")
    # ---- tuple spell_reducer
    a, b = generic.spell_length_statistics(da, 1.0, 1, None, "<", ("max", "count"), "YS")
    np.testing.assert_array_equal(a.values, O.spell_length_statistics(x, 1.0, 1, None, "<", "max", poff_y))
    np.testing.assert_array_equal(b.values, O.spell_length_statistics(x, 1.0, 1, None, "<", "count", poff_y))


def test_reference_default_call_shapes(host):
    _check_reference_default_call_shapes()


def _check_spell_statistics_with_indexers():
    """select_time on the spell mask (indices/generic.py:557-558): the reference's known answer
    (tests/test_indices.py:4116-4126: 9), the whole-array `rle` variant, and a random case against the oracle."""
    import xclim_b200
    from xclim_b200 import generic, indices
    a = np.array([1] * 5 + [0] * 10 + [1] * 350, dtype=np.float32)
    pr = make_field(a, "1900-01-01", calendar="standard", units="mm/d")
    for fn in (indices.dry_spell_total_length, indices.dry_spell_max_length):
        out = fn(pr, window=7, op="sum", thresh="3.1 mm", freq="MS", date_bounds=("01-10", "12-31"))
        np.testing.assert_allclose(out.values, [9] + [0] * 11)
        assert out.values.dtype == np.float32 and out.attrs["units"] == "d"
        with xclim_b200.set_options(rle_nan_adjacent="drop"):       # the whole-array rle drops the run next to the NaN
            out = fn(pr, window=7, op="sum", thresh="3.1 mm", freq="MS", date_bounds=("01-10", "12-31"))
        np.testing.assert_allclose(out.values, [0] * 12)
    # without the indexer the spell is whole: 16 days (3 wet days fit in a 7-day window under 3.1 mm)
    np.testing.assert_allclose(indices.dry_spell_total_length(pr, window=7, op="sum", thresh="3.1 mm", freq="MS").values,
                               [16] + [0] * 11)
    # random: season JJA, window 3, both orders, against the oracle mask with NaN -> run break
    rng = np.random.default_rng(55)
    T, shape = 365 * 2, (2, 3)
    x = rng.gamma(0.4, 5.0, (T,) + shape).astype(np.float32)
    x[rng.random(x.shape) < 0.5] = 0
    da = make_field(x, "2001-01-01", calendar="noleap", units="mm/d")
    keep = da.time.select_mask(season="JJA")
    m = O.spell_mask(x, 3, "sum", "<", 1.0).astype(np.float32)
    m[~keep] = 0.0
    for freq in ("YS", "QS-DEC"):
        poff = da.time.period_offsets(freq)
        for red in ("max", "sum", "count"):
            for before in (True, False):
                got = generic.spell_length_statistics(da, 1.0, 3, "sum", "<", red, freq, resample_before_rl=before,
                                                      season="JJA")
                exp = O.resample_and_rl(m > 0, before, O.rle_statistics, poff=poff, reducer=red, window=1)
                np.testing.assert_array_equal(got.values, exp, err_msg=f"{freq} {red} {before}")
    # window == 1 with an indexer goes the same way
    got = generic.spell_length_statistics(da, 1.0, 1, None, "<", "max", "YS", month=[6, 7])
    k2 = da.time.select_mask(month=[6, 7])
    exp = O.resample_and_rl((x < 1.0) & k2[:, None, None], True, O.rle_statistics, poff=da.time.period_offsets("YS"),
                            reducer="max", window=1)
    np.testing.assert_array_equal(got.values, exp)


def test_spell_statistics_with_indexers(host):
    _check_spell_statistics_with_indexers()


def _check_rolling_with_indexers():
    """select_rolling_resample_op(**indexer): the selection applies to the ROLLED series (indices/generic.py:169-174)."""
    from xclim_b200 import generic
    rng = np.random.default_rng(66)
    T, shape = 365 * 2, (2, 4)
    x = rng.gamma(0.5, 4.0, (T,) + shape).astype(np.float32)
    x[rng.random(x.shape) < 0.01] = np.nan
    da = make_field(x, "2001-01-01", calendar="noleap", units="mm/d")
    for freq, idx in (("YS", {"season": "DJF"}), ("MS", {"month": [1, 7]}), ("YS", {"date_bounds": ("03-01", "06-15")})):
        keep = da.time.select_mask(**idx)
        poff = da.time.period_offsets(freq)
        for wop, op, center, w in (("sum", "max", False, 5), ("mean", "mean", True, 3), ("max", "min", False, 4)):
            got = generic.select_rolling_resample_op(da, op, w, window_center=center, window_op=wop, freq=freq, **idx)
            rolled = O.rolling(x.astype(np.float64), w, wop, center=center)
            rolled = np.where(keep[:, None, None], rolled, np.nan)
            exp = O.resample_reduce(rolled, poff, op)
            np.testing.assert_allclose(got.values, exp, rtol=1e-5, equal_nan=True, err_msg=f"{freq} {idx} {wop} {op}")


def test_rolling_with_indexers(host):
    _check_rolling_with_indexers()
