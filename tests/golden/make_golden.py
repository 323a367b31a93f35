"""Generate golden fixtures from the REFERENCE's own numpy/numba cores.  It needs an xclim source checkout
(the tests only read the committed .npz files):

    XCLIM_REFERENCE_ROOT=<xclim checkout> python tests/golden/make_golden.py

Outputs (committed):
  tests/golden/ref_run_length_1d.npz  -- statistics_run_1d / windowed_run_count_1d /
        windowed_run_events_1d / first_run_1d / _cumsum_reset_np on seeded boolean series
        (reference: indices/run_length.py:143-151, 1334-1477)
  tests/golden/ref_quantile.npz       -- calc_perc on seeded float32 samples with NaNs
        (reference: core/utils.py:279-557)
  tests/golden/ref_cffwis.npz         -- the fire-weather recurrences (_fire_weather_calc with its season,
        overwintering and dry-start modes) on seeded float32 weather series
        (reference: indices/fire/_cffwis.py:161-900)
  tests/golden/ref_cross_check.npz    -- statistics_run_1d and calc_perc on the inputs of
        cross_check_inputs()
  tests/golden/ref_cffwis_steps.npz   -- the three daily step functions of the fire-weather codes on a seeded
        sample of the inputs of cffwis_step_inputs()
  tests/golden/ref_cffwis_modes.npz   -- _fire_weather_calc on the cases of cffwis_mode_cases() and
        cffwis_branch_cases(): the seeded positions of sample_positions() of every float output, the whole season
        mask (bit-packed) and winter_pr
Nothing from the reference is copied into the repo: the functions are exec'ed where they lie
(tests/golden/_ref_extract.py) and only their numeric inputs/outputs are stored.
"""
from __future__ import annotations

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import _ref_extract as ref  # noqa: E402


def run_length_fixture(rng):
    rl = ref.load_run_length()
    n_series, T = 64, 120
    series = np.zeros((n_series, T), dtype=bool)
    for i in range(n_series):
        p = rng.uniform(0.05, 0.95)
        # persistent series: flip state with small probability so that long runs occur
        flips = rng.random(T) < rng.uniform(0.05, 0.5)
        state = rng.random() < p
        for t in range(T):
            if flips[t]:
                state = rng.random() < p
            series[i, t] = state
    series[0] = False
    series[1] = True
    series[2, :] = True
    series[2, 35] = False
    reducers = ["max", "min", "sum", "count", "mean", "std"]
    windows = [1, 2, 3, 5, 10]
    stats = np.zeros((len(reducers), len(windows), n_series), dtype=np.float64)
    wcount = np.zeros((len(windows), n_series), dtype=np.float64)
    wevents = np.zeros((len(windows), n_series), dtype=np.float64)
    first = np.zeros((len(windows), n_series), dtype=np.float64)
    for i in range(n_series):
        for wi, w in enumerate(windows):
            for ri, r in enumerate(reducers):
                stats[ri, wi, i] = rl["statistics_run_1d"](series[i], r, w)
            wcount[wi, i] = rl["windowed_run_count_1d"](series[i], w)
            wevents[wi, i] = rl["windowed_run_events_1d"](series[i], w)
            first[wi, i] = rl["first_run_1d"](series[i], w)
    cs_last = rl["_cumsum_reset_np"](series.astype(np.uint8).copy(), "last", np.uint8(1))
    cs_first = rl["_cumsum_reset_np"](series.astype(np.uint8).copy(), "first", np.uint8(1))
    np.savez_compressed(os.path.join(HERE, "ref_run_length_1d.npz"), series=series,
                        reducers=np.array(reducers), windows=np.array(windows), stats=stats,
                        wcount=wcount, wevents=wevents, first=first, cs_last=cs_last, cs_first=cs_first)


def quantile_fixture(rng):
    ut = ref.load_utils()
    cases = []
    for n in (1, 2, 3, 5, 7, 10, 30, 75, 148, 150):
        a = (280 + 10 * rng.standard_normal((40, n))).astype(np.float32)
        # NaNs: some rows partially, one row entirely
        for r in range(40):
            k = rng.integers(0, max(1, n // 3) + 1) if r % 3 == 0 else 0
            if k:
                a[r, rng.choice(n, size=k, replace=False)] = np.nan
        a[5, :] = np.nan
        # ties
        if n >= 5:
            a[7, : n // 2] = a[7, 0]
        cases.append(a)
    pers = np.array([10.0, 50.0, 90.0, 99.0, 0.0, 100.0])
    out = {}
    for i, a in enumerate(cases):
        out[f"x{i}"] = a
        for (al, be), tag in (((1 / 3, 1 / 3), "t8"), ((1.0, 1.0), "t7")):
            with np.errstate(all="ignore"):
                import warnings
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    q = ut["calc_perc"](a.copy(), list(pers), al, be)
            out[f"q{i}_{tag}"] = q
    out["percentiles"] = pers
    out["n_cases"] = np.array(len(cases))
    np.savez_compressed(os.path.join(HERE, "ref_quantile.npz"), **out)


def cffwis_inputs(seed=20260924, C=16, T=800):
    """Seeded float32 weather series (cells, T), time LAST as the reference's ufunc core takes them."""
    rng = np.random.default_rng(seed)
    lat = np.array([-60, -35, -29.9, -20, -15, -10, 0, 10, 14.9, 15, 25, 30, 40, 47.5, 60, 75], dtype=np.float64)[:C]
    t = np.arange(T)
    doy = t % 365
    mth = np.minimum(doy // 30.42, 11).astype(np.int64) + 1
    season = np.cos(2 * np.pi * (doy - 200) / 365)                      # northern summer
    amp = np.where(lat >= 0, 1.0, -1.0)[:, None] * (6 + 0.25 * np.abs(lat))[:, None]
    base = (22 - 0.35 * np.abs(lat))[:, None]
    tas = base + amp * season[None, :] + 3.0 * rng.standard_normal((C, T))
    wet = rng.random((C, T)) < 0.35
    pr = np.where(wet, rng.gamma(0.7, 5.0, size=(C, T)), 0.0)
    hurs = np.clip(55 + 20 * rng.standard_normal((C, T)) + 15 * wet, 5, 100)
    ws = np.abs(12 + 8 * rng.standard_normal((C, T)))
    snd = np.clip(0.25 * (-(tas - 1.0)) / 10 + 0.05 * rng.standard_normal((C, T)), 0, None) * (tas < 4)
    # a missing block and single missing values
    tas[3, 100:104] = np.nan
    pr[5, 300] = np.nan
    hurs[7, 50] = np.nan
    ws[9, 60] = np.nan
    f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)  # noqa: E731
    return dict(tas=f32(tas), pr=f32(pr), hurs=f32(hurs), ws=f32(ws), snd=f32(snd), mth=mth, lat=lat)


#: the modes of _fire_weather_calc the fixture covers (name -> keyword overrides)
CFFWIS_CASES = {
    "always_on": dict(season_method=None, outputs=["DC", "DMC", "FFMC", "ISI", "BUI", "FWI", "DSR"]),
    "wf93": dict(season_method="WF93", outputs=["DC", "DMC", "FFMC", "ISI", "BUI", "FWI", "season_mask"]),
    "wf93_end4": dict(season_method="WF93", temp_end_thresh=4.0, temp_condition_days=4, outputs=["DC", "season_mask"]),
    "la08_overwinter": dict(season_method="LA08", overwintering=True, outputs=["DC", "season_mask", "winter_pr"],
                            state="some"),
    "mask_cfs": dict(season_method="mask", dry_start="CFS", dmc_dry_factor=5, outputs=["DC", "DMC"], mask_from="wf93"),
    "gfwed_snow": dict(season_method="GFWED", dry_start="GFWED+SNOW", snow_cover_days=20, snow_min_mean_depth=0.05,
                       outputs=["DC", "DMC", "FFMC", "ISI", "BUI", "FWI", "season_mask"]),
    "gfwed_dry": dict(season_method="mask", dry_start="GFWED", outputs=["DC", "DMC", "FFMC"], mask_from="wf93"),
    "mask_ow_cfs_cont": dict(season_method="mask", overwintering=True, dry_start="CFS", initial_start_up=False,
                             outputs=["DC", "DMC", "FFMC", "winter_pr"], mask_from="la08_overwinter", state="all"),
    "dc_only_always_on": dict(season_method=None, outputs=["DC"], state="some"),
}


def cffwis_params(fw, **over):
    kw = {k: (v if not isinstance(v, tuple) else v[0]) for k, v in fw["default_params"].items()}
    kw.update(season_method=None, overwintering=False, dry_start=None, initial_start_up=True)
    kw.update({k: v for k, v in over.items() if k not in ("mask_from", "state")})
    return kw


def cffwis_state(inp, kind):
    C = inp["tas"].shape[0]
    rng = np.random.default_rng(77)
    nan = np.full(C, np.nan, np.float32)
    if kind is None:
        return nan.copy(), nan.copy(), nan.copy(), np.zeros(C, np.float32)
    dc0 = (50 + 300 * rng.random(C)).astype(np.float32)
    dmc0 = (5 + 40 * rng.random(C)).astype(np.float32)
    ffmc0 = (60 + 30 * rng.random(C)).astype(np.float32)
    wpr = (200 * rng.random(C)).astype(np.float32)
    if kind == "some":
        dc0[::3] = np.nan
        dmc0[1::3] = np.nan
        ffmc0[2::3] = np.nan
    return dc0, dmc0, ffmc0, wpr


def cffwis_fixture():
    fw = ref.load_cffwis()
    inp = cffwis_inputs()
    out = {k: v for k, v in inp.items()}
    masks = {}
    for name, over in CFFWIS_CASES.items():
        kw = cffwis_params(fw, **over)
        dc0, dmc0, ffmc0, wpr = cffwis_state(inp, over.get("state"))
        mask = masks[over["mask_from"]] if "mask_from" in over else None
        res = fw["_fire_weather_calc"](inp["tas"], inp["pr"], inp["hurs"], inp["ws"], inp["snd"], inp["mth"], inp["lat"],
                                       mask, dc0, dmc0, ffmc0, wpr, **kw)
        if len(kw["outputs"]) == 1:
            res = (res,)
        for oname, arr in zip(kw["outputs"], res):
            out[f"{name}__{oname}"] = np.asarray(arr)
            if oname == "season_mask":
                masks[name] = np.asarray(arr).astype(bool)
    np.savez_compressed(os.path.join(HERE, "ref_cffwis.npz"), **out)
    return out


def cross_check_inputs():
    """Seeded boolean series (time, series) for statistics_run_1d and float32 samples with NaNs (rows, samples)
    for calc_perc."""
    rng = np.random.default_rng(7)
    m = rng.random((200, 50)) < 0.6
    x = (rng.standard_normal((50, 150)) * 5 + 280).astype(np.float32)
    x[rng.random(x.shape) < 0.05] = np.nan
    return m, x


CROSS_CHECK_REDUCERS = ("max", "min", "sum", "count", "mean", "std")
CROSS_CHECK_WINDOWS = (1, 2, 4)
CROSS_CHECK_PERCENTILES = (10.0, 90.0)


def cross_check_fixture():
    import warnings
    rl, ut = ref.load_run_length(), ref.load_utils()
    m, x = cross_check_inputs()
    stats = np.array([[[rl["statistics_run_1d"](m[:, i], red, w) for i in range(m.shape[1])]
                       for w in CROSS_CHECK_WINDOWS] for red in CROSS_CHECK_REDUCERS], dtype=np.float64)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        perc = ut["calc_perc"](x.copy(), list(CROSS_CHECK_PERCENTILES), 1 / 3, 1 / 3)
    np.savez_compressed(os.path.join(HERE, "ref_cross_check.npz"), stats=stats, calc_perc=perc)


def cffwis_step_inputs(n=4000):
    """Seeded float32 arguments of the three daily step functions over their whole ranges, and the latitudes and
    months they are evaluated at."""
    rng = np.random.default_rng(3)
    t = (rng.uniform(-15, 38, n)).astype(np.float32)
    p = np.where(rng.random(n) < 0.5, 0, rng.gamma(0.8, 6, n)).astype(np.float32)
    w = rng.uniform(0, 50, n).astype(np.float32)
    h = rng.uniform(3, 100, n).astype(np.float32)
    f0 = rng.uniform(0, 101, n).astype(np.float32)
    d0 = rng.uniform(0, 200, n).astype(np.float32)
    c0 = rng.uniform(0, 900, n).astype(np.float32)
    return dict(t=t, p=p, w=w, h=h, f0=f0, d0=d0, c0=c0), (-50.0, -20.0, 0.0, 20.0, 50.0), (1, 4, 7, 10)


def cffwis_step_fixture(per_case=64):
    """DMC and DC of a seeded sample of `per_case` inputs at every (latitude, month), FFMC of 4 * `per_case`."""
    fw = ref.load_cffwis()
    a, lats, mths = cffwis_step_inputs()
    n = a["t"].size
    rng = np.random.default_rng(5)
    sel = np.array([[np.sort(rng.choice(n, per_case, replace=False)) for _ in mths] for _ in lats], dtype=np.int16)
    dmc = np.empty(sel.shape, np.float64)
    dc = np.empty(sel.shape, np.float64)
    for li, lat in enumerate(lats):
        for mi, mth in enumerate(mths):
            s = sel[li, mi]
            dmc[li, mi] = fw["_duff_moisture_code"](a["t"][s], a["p"][s], a["h"][s], mth, lat, a["d0"][s])
            dc[li, mi] = fw["_drought_code"](a["t"][s], a["p"][s], mth, lat, a["c0"][s])
    sel_f = np.sort(rng.choice(n, 4 * per_case, replace=False)).astype(np.int16)
    ffmc = fw["_fine_fuel_moisture_code"](a["t"][sel_f], a["p"][sel_f], a["w"][sel_f], a["h"][sel_f], a["f0"][sel_f])
    np.savez_compressed(os.path.join(HERE, "ref_cffwis_steps.npz"), sel=sel, dmc=dmc, dc=dc, sel_ffmc=sel_f,
                        ffmc=np.asarray(ffmc, np.float64))


def cffwis_mode_cases():
    """All combinations of season method x overwintering x dry start x initial_start_up (overwintering needs a
    season), each with random thresholds / window lengths / previous codes.  Yields (label, inputs (cells, T),
    (dc0, dmc0, ffmc0, winter_pr), season mask (cells, T) or None, outputs, keyword overrides)."""
    import itertools
    rng = np.random.default_rng(123)
    T = 320
    combos = itertools.product([None, "mask", "WF93", "LA08", "GFWED"], [False, True], [None, "CFS", "GFWED", "GFWED+SNOW"],
                               [True, False])
    for trial, (season, ow, dry, isu) in enumerate(combos):
        if ow and season is None:
            continue
        inp = cffwis_inputs(seed=1000 + trial, C=16, T=T)
        state = cffwis_state(inp, [None, "some", "all"][trial % 3])
        over = dict(season_method=season, overwintering=ow, dry_start=dry, initial_start_up=isu,
                    temp_condition_days=int(rng.integers(1, 6)), snow_condition_days=int(rng.integers(1, 6)),
                    snow_cover_days=int(rng.integers(5, 70)), temp_start_thresh=float(rng.uniform(8, 14)),
                    temp_end_thresh=float(rng.uniform(2, 7)), snow_thresh=float(rng.choice([0.01, 0.03])),
                    prec_thresh=float(rng.choice([1.0, 2.5])), dc_dry_factor=int(rng.integers(2, 7)),
                    dmc_dry_factor=int(rng.integers(1, 4)), snow_min_cover_frac=float(rng.uniform(0.3, 0.8)),
                    snow_min_mean_depth=float(rng.uniform(0.02, 0.1)), carry_over_fraction=float(rng.choice([0.5, 0.75, 1.0])),
                    wetting_efficiency_fraction=float(rng.choice([0.5, 0.75, 0.9])))
        outs = ["DC", "DMC", "FFMC", "ISI", "BUI", "FWI", "DSR"]
        mask = None
        if season == "mask":                      # a persistent random mask
            mask = np.zeros((16, T), bool)
            st = rng.random(16) < 0.5
            for t in range(T):
                st = np.where(rng.random(16) < 0.03, ~st, st)
                mask[:, t] = st
        elif season is not None:
            outs.append("season_mask")
        if ow:
            outs.append("winter_pr")
        yield f"{season},{ow},{dry},{isu}", inp, state, mask, outs, over


def cffwis_branch_cases():
    """Inputs drawn from the branch points of the equations (rain thresholds 0.5 / 1.5 / 2.8 mm and just above,
    humidity 0 and 100 %, calm and storm winds, temperatures at -2.8 / -1.1 / 21.1 degC, snow depth at its
    threshold, latitudes on the band edges, previous codes at 0 / 33 / 65 / 101), with and without missing values,
    under four modes.  Yields what cffwis_mode_cases() does."""
    rng = np.random.default_rng(7)
    C, T = 32, 240
    f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)   # noqa: E731
    for trial in range(6):
        tas = rng.choice([-45.0, -2.8, -1.1, 0.0, 21.1, 35.0, 50.0], size=(C, T)) + rng.normal(0, 0.5, (C, T))
        pr = rng.choice([0.0, 0.5, 0.50001, 1.5, 1.50001, 2.8, 2.80001, 50.0, 300.0], size=(C, T))
        hurs = rng.choice([0.0, 1e-3, 5.0, 50.0, 99.999, 100.0], size=(C, T))
        ws = rng.choice([0.0, 1e-3, 10.0, 100.0, 250.0], size=(C, T))
        snd = rng.choice([0.0, 0.01, 0.010001, 0.5], size=(C, T))
        if trial % 3 == 0:
            for a in (tas, pr, hurs, ws):
                a[rng.random((C, T)) < 0.002] = np.nan
        mth = rng.integers(1, 13, T).astype(np.int64)
        lat = rng.choice([-90, -30, -15, 15, 30, 90, -29.999, 14.999, 0], size=C).astype(np.float64)
        dc0, dmc0, ffmc0, wpr = cffwis_state({"tas": f32(tas)}, [None, "some", "all"][trial % 3])
        if trial % 3:
            dc0[:4], dmc0[:4], ffmc0[:4] = [0.0, 1e-3, 800.0, 2000.0], [0.0, 33.0, 65.0, 500.0], [0.0, 101.0, 50.0, 99.9]
        inp = dict(tas=f32(tas), pr=f32(pr), hurs=f32(hurs), ws=f32(ws), snd=f32(snd), mth=mth, lat=lat)
        for season, ow, dry in ((None, False, None), ("WF93", True, "CFS"), ("GFWED", False, "GFWED+SNOW"), ("LA08", True, None)):
            outs = ["DC", "DMC", "FFMC", "ISI", "BUI", "FWI", "DSR"] + (["season_mask"] if season else []) + \
                (["winter_pr"] if ow else [])
            over = dict(season_method=season, overwintering=ow, dry_start=dry, snow_cover_days=10)
            yield f"{trial} {season}", inp, (dc0, dmc0, ffmc0, wpr), None, outs, over


CFFWIS_CASE_GROUPS = {"modes": cffwis_mode_cases, "branch": cffwis_branch_cases}
CFFWIS_FLOAT_OUTPUTS = ("DC", "DMC", "FFMC", "ISI", "BUI", "FWI", "DSR")


def sample_positions(C, T, case, n_random=16):
    """(day, cell) positions stored of a (T, cells) output of case number `case`: the last day of every cell,
    which carries the whole recurrence, and `n_random` seeded positions."""
    rng = np.random.default_rng(case)
    t = np.concatenate([np.full(C, T - 1), rng.integers(0, T, n_random)])
    c = np.concatenate([np.arange(C), rng.integers(0, C, n_random)])
    return t, c


def cffwis_mode_fixture():
    """Per case group, one row per case: `<group>__<output>` the float outputs at sample_positions() (NaN rows
    where a case does not ask for the output), `<group>__season_mask` the whole (cells, T) mask bit-packed,
    `<group>__winter_pr` every cell."""
    import warnings
    fw = ref.load_cffwis()
    out = {}
    for group, make_cases in CFFWIS_CASE_GROUPS.items():
        cases = list(make_cases())
        C, T = cases[0][1]["tas"].shape
        n = len(cases)
        rows = {o: np.full((n, C + 16), np.nan, np.float32) for o in CFFWIS_FLOAT_OUTPUTS}
        rows["season_mask"] = np.zeros((n, C * T // 8), np.uint8)
        rows["winter_pr"] = np.full((n, C), np.nan, np.float32)
        for i, (_, inp, state, mask, outs, over) in enumerate(cases):
            kw = cffwis_params(fw, outputs=outs, **over)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                res = fw["_fire_weather_calc"](inp["tas"], inp["pr"], inp["hurs"], inp["ws"], inp["snd"], inp["mth"],
                                               inp["lat"], mask, *(s.copy() for s in state), **kw)
            t, c = sample_positions(C, T, i)
            for o, a in zip(outs, res):
                a = np.asarray(a)
                if o == "season_mask":
                    rows[o][i] = np.packbits(a.astype(bool))
                elif o == "winter_pr":
                    rows[o][i] = a
                else:
                    rows[o][i] = a[c, t]
        out.update({f"{group}__{o}": v for o, v in rows.items()})
    np.savez_compressed(os.path.join(HERE, "ref_cffwis_modes.npz"), **out)


def stored_cffwis_outputs(g, group, case, outs, C, T):
    """The reference's outputs of case number `case` of `group` in ref_cffwis_modes.npz: the float outputs at
    sample_positions(), the season mask (T, cells) and winter_pr whole."""
    exp = {}
    for o in outs:
        a = g[f"{group}__{o}"][case]
        exp[o] = np.unpackbits(a, count=C * T).astype(bool).reshape(C, T).T if o == "season_mask" else a
    return exp


if __name__ == "__main__":
    if not ref.available():
        raise SystemExit("reference sources not found: set XCLIM_REFERENCE_ROOT to an xclim source checkout")
    rng = np.random.default_rng(20260923)
    run_length_fixture(rng)
    quantile_fixture(rng)
    cffwis_fixture()
    cross_check_fixture()
    cffwis_step_fixture()
    cffwis_mode_fixture()
    print("golden fixtures written to", HERE)
