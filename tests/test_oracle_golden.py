"""Pin the CPU oracle: (1) against fixtures produced by the reference's own numpy/numba cores
(tests/golden/make_golden.py), (2) against the known-answer values held by the reference's tests,
(3) against outputs of the reference's own cores on seeded inputs (tests/golden/make_golden.py)."""
import os
import sys

import numpy as np
import pytest

from oracle import xclim_oracle as O

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import make_golden as mg  # noqa: E402


# ------------------------------------------------------------------ fixtures from the reference
def test_run_length_whole_array_path_matches_reference_1d(golden_dir):
    g = np.load(os.path.join(golden_dir, "ref_run_length_1d.npz"))
    series = g["series"].T  # (T, n_series): time on axis 0
    for ri, red in enumerate(g["reducers"]):
        for wi, w in enumerate(g["windows"]):
            got = O.rle_statistics(series, str(red), int(w))
            np.testing.assert_allclose(got, g["stats"][ri, wi], rtol=1e-12, err_msg=f"{red} w={w}")
    for wi, w in enumerate(g["windows"]):
        np.testing.assert_array_equal(O.windowed_run_count(series, int(w), poff=[0, series.shape[0]])[0], g["wcount"][wi])
        np.testing.assert_array_equal(O.windowed_run_events(series, int(w)), g["wevents"][wi])
        fr = O.first_run(series, int(w))
        exp = g["first"][wi]
        if int(w) == 1:
            # whole-array quirk (run_length.py:603-605): argmax == argmin also for ALL-True series
            alltrue = series.all(axis=0)
            np.testing.assert_array_equal(fr[~alltrue], exp[~alltrue])
            assert np.isnan(fr[alltrue]).all()
        else:
            np.testing.assert_array_equal(fr, exp)
    np.testing.assert_array_equal(O.cumsum_reset(series, "last").T, g["cs_last"])
    np.testing.assert_array_equal(O.cumsum_reset(series, "first").T, g["cs_first"])


def test_quantile_matches_reference_calc_perc(golden_dir):
    g = np.load(os.path.join(golden_dir, "ref_quantile.npz"))
    pers = g["percentiles"]
    for i in range(int(g["n_cases"])):
        x = g[f"x{i}"]
        for tag, (al, be) in {"t8": (1 / 3, 1 / 3), "t7": (1.0, 1.0)}.items():
            got = O.calc_perc(x, pers, al, be)
            exp = g[f"q{i}_{tag}"]
            assert got.dtype == exp.dtype and (x.shape[1] == 1 or got.dtype == np.float64)
            np.testing.assert_array_equal(got, exp, err_msg=f"case {i} {tag}")  # bit-exact


# ------------------------------------------------------------------ known answers of the reference tests
def test_known_answers_quantile():
    # tests/test_utils.py:27-75
    arr = np.asarray([15.0, 20.0, 35.0, 40.0, 50.0])
    assert O.nan_quantile(arr, [0.4], 1, 1)[0] == 29
    assert O.nan_quantile(arr, [0.4], 1 / 3, 1 / 3)[0] == 27
    assert O.nan_quantile(np.asarray([np.nan, 41.0, 41.0, 43.0, 43.0]), [0.5], 1 / 3, 1 / 3)[0] == 42.0
    assert np.isnan(O.nan_quantile(np.asarray([np.nan]), [0.5])[0])
    assert np.isnan(O.nan_quantile(np.asarray([]), [0.5])).all()


def test_known_answers_rle():
    # tests/test_run_length.py:100-130
    v = np.zeros(365)
    v[1:11] = 1
    out = O.rle(v != 0, index="first")
    exp = np.zeros(365); exp[1] = 10; exp[2:11] = np.nan
    np.testing.assert_array_equal(out, exp)
    out = O.rle(v != 0, index="last")
    exp = np.zeros(365); exp[1:10] = np.nan; exp[10] = 10
    np.testing.assert_array_equal(out, exp)


def _months(start_doy0=0, year_days=365, leap=False):
    dpm = [31, 29 if leap else 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31]
    return np.concatenate([[0], np.cumsum(dpm)])


def test_known_answers_rle_statistics():
    # tests/test_run_length.py:166-278 (year 2000 from July 1st = 365 days; monthly groups)
    from xclim_b200 import TimeAxis
    ta = TimeAxis.daily("2000-07-01", 365)
    poff = ta.period_offsets("ME")
    v = np.zeros(365); v[1:11] = 1
    lt = O.resample_and_rl(v != 0, True, O.rle_statistics, poff=poff, reducer="max", window=1)
    assert lt[0] == 10 and (lt[1:] == 0).all()
    lt = O.rle_statistics(v != 0, "max", 1, poff=poff)
    assert lt[0] == 10 and (lt[1:] == 0).all()
    # all true
    v = np.ones(365)
    lt = O.rle_statistics(v != 0, "max", 1, poff=poff)
    exp = np.zeros(12); exp[0] = 365
    np.testing.assert_array_equal(lt, exp)
    lt = O.resample_and_rl(v != 0, True, O.rle_statistics, poff=poff, reducer="max", window=1)
    np.testing.assert_array_equal(lt, np.diff(poff))
    # almost all true
    v = np.ones(365); v[35] = 0
    lt = O.resample_and_rl(v != 0, True, O.rle_statistics, poff=poff, reducer="max", window=1)
    assert lt[0] == 31 and lt[1] == 26
    lt = O.rle_statistics(v != 0, "max", 1, poff=poff)
    assert lt[0] == 35 and lt[1] == 365 - 35 - 1
    # other stats (:243-278), yearly group
    ta = TimeAxis.daily("2000-01-01", 365)
    py = ta.period_offsets("YS")
    m = v != 0
    assert O.resample_and_rl(m, True, O.rle_statistics, poff=py, reducer="min", window=1)[0] == 35
    assert O.resample_and_rl(m, True, O.rle_statistics, poff=py, reducer="mean", window=36)[0] == 329
    assert O.resample_and_rl(m, True, O.rle_statistics, poff=py, reducer="std", window=1)[0] == 147
    assert O.rle_statistics(m, "q90", 1, poff=py)[0] == pytest.approx(299.6)
    assert O.rle_statistics(m, "q10", 1, poff=py)[0] == pytest.approx(64.4)


def test_known_answers_windowed_runs():
    # tests/test_run_length.py:356-371
    a = np.zeros(50, bool)
    a[4:7] = True
    a[34:45] = True
    assert O.windowed_run_events(a, 3) == 2
    assert O.windowed_run_count(a, 3, poff=[0, 50])[0] == 14


def test_known_answers_cdd():
    # tests/test_indices.py:2354-2381 (pr_series: daily from 2000-01-01, kg m-2 s-1; thresh 1 mm/day)
    from xclim_b200 import TimeAxis
    ta = TimeAxis.daily("2000-01-01", 365)
    poff = ta.period_offsets("ME")
    thr = 1 / 86400
    a = (np.zeros(365) + 10).astype(np.float32); a[5:15] = 0
    assert O.maximum_consecutive_dry_days(a, thr, poff)[0] == 10
    a = (np.zeros(365) + 10).astype(np.float32); a[:10] = 0
    assert O.maximum_consecutive_dry_days(a, thr, poff)[0] == 10
    a = (np.zeros(365) + 10).astype(np.float32); a[5:35] = 0
    assert O.maximum_consecutive_dry_days(a, thr, poff, resample_before_rl=True)[0] == 26
    assert O.maximum_consecutive_dry_days(a, thr, poff, resample_before_rl=False)[0] == 30


def test_known_answers_percentile_doy():
    # tests/test_calendar.py:83-103
    yr = np.full(365, 2001); doy = np.arange(1, 366)
    x = np.arange(365, dtype=np.float64)
    assert O.percentile_doy(x, yr, doy, 5, 50)[2, 0] == 2
    x[1] = np.nan
    assert O.percentile_doy(x, yr, doy, 5, 50)[2, 0] == 2.5


def test_known_answers_tx90p_leap_year():
    # tests/test_indices.py:2594-2607: 366-day year 2000, per=10, monthly counts 30, 29, ..., 25 in June
    from xclim_b200 import TimeAxis
    ta = TimeAxis.daily("2000-01-01", 366)
    tas = np.arange(366, dtype=np.float64)
    t90 = O.percentile_doy(tas, ta.year, ta.doy, 5, 10.0)[:, 0]
    assert t90.shape == (366,)
    tas[175:180] = 1
    thresh = O.resample_doy(t90, ta.doy, cal_max_doy=366)
    out = O.threshold_count(tas, ">", thresh, ta.period_offsets("MS"), constrain=(">", ">="))
    assert out[0] == 30 and out[1] == 29 and out[5] == 25


def test_spell_mask_truth_tables():
    # tests/test_generic.py:702-751 (values transcribed)
    data = np.array([1, 2, 3, 2, 1, 2, 3, 2, 1], dtype=np.float32)
    cases = [
        (1, "min", ">=", 2, [False, True, True, True, False, True, True, True, False]),
        (3, "min", ">=", 2, [False, True, True, True, False, True, True, True, False]),
        (3, "max", ">=", 2, [True] * 9),
        (2, "mean", ">=", 2, [False, True, True, True, False, True, True, True, False]),  # see test below
    ]
    for win, red, op, thr, exp in cases[:3]:
        got = O.spell_mask(data, win, red, op, thr)
        np.testing.assert_array_equal(got, exp, err_msg=f"{win} {red} {op}")


# ------------------------------------------------------------------ stored outputs of the reference's cores
def test_against_stored_reference_outputs(golden_dir):
    g = np.load(os.path.join(golden_dir, "ref_cross_check.npz"))
    m, x = mg.cross_check_inputs()
    for ri, red in enumerate(mg.CROSS_CHECK_REDUCERS):
        for wi, w in enumerate(mg.CROSS_CHECK_WINDOWS):
            np.testing.assert_allclose(O.rle_statistics(m, red, w), g["stats"][ri, wi], rtol=1e-12, err_msg=f"{red} w={w}")
    np.testing.assert_array_equal(O.calc_perc(x, list(mg.CROSS_CHECK_PERCENTILES), 1 / 3, 1 / 3), g["calc_perc"])


def _warm(d1, d2, n=365, start="2000-01-01"):
    """tas = 0 K except 280 K between the two dates (tests/test_indices.py:1668-1672)."""
    import pandas as pd
    from xclim_b200 import TimeAxis
    idx = pd.date_range(start, periods=n, freq="D")
    tas = np.zeros(n, np.float32)
    tas[(idx >= d1) & (idx <= d2)] = 280
    return tas, TimeAxis.daily(start, n)


@pytest.mark.parametrize("d1,d2,mid_date,expected", [
    ("1950-01-01", "1951-01-01", "07-01", np.nan), ("2000-01-01", "2000-12-31", "07-01", 365),
    ("2000-07-10", "2001-01-01", "07-01", np.nan), ("2000-06-15", "2000-07-15", "07-01", 198),
    ("2000-06-15", "2000-07-25", "07-15", 208), ("2000-06-15", "2000-07-15", "10-01", 275),
    ("2000-06-15", "2000-07-15", "01-10", np.nan), ("2000-06-15", "2000-07-15", "06-15", np.nan)])
def test_known_answers_growing_season_end(d1, d2, mid_date, expected):
    # tests/test_indices.py:1654-1678
    tas, ta = _warm(d1, d2)
    mids = ta.date_index_in_periods("YS", mid_date)
    out = O.season(tas > np.float32(278.15), 5, [int(m) if m >= 0 else None for m in mids], ta.period_offsets("YS"), "end", ta.doy)
    np.testing.assert_array_equal(out[0], expected)


@pytest.mark.parametrize("d1,d2,expected", [("1950-01-01", "1951-01-01", 0), ("2000-01-01", "2000-12-31", 365),
                                            ("2000-07-10", "2001-01-01", 0), ("2000-06-15", "2001-01-01", 199),
                                            ("2000-06-15", "2000-07-15", 31)])
def test_known_answers_growing_season_length(d1, d2, expected):
    # tests/test_indices.py:1681-1700
    tas, ta = _warm(d1, d2)
    mids = ta.date_index_in_periods("YS", "07-01")
    out = O.season(tas >= np.float32(278.15), 6, [int(m) for m in mids], ta.period_offsets("YS"), "length", ta.doy)
    assert out[0] == expected


def test_known_answers_season_and_start():
    # tests/test_run_length.py:674-690 ; tests/test_indices.py:1625-1645
    t = np.zeros(360); t[140:150] = 1
    beg, end, length = O.season_group(t >= 1, 2, None, has_date=False)
    assert (beg, end, length) == (140, 150, 10)
    tg = np.zeros(365) - 1
    tg[10:14] += 6; tg[20:25] += 6; tg[30:36] += 6
    beg, _, _ = O.season_group(tg + 273.15 >= 278.15, 5, 182)
    assert beg == 20
    # south hemisphere (tests/test_indices.py:1702-1707): YS-JUL groups, mid_date 01-01
    from xclim_b200 import TimeAxis
    import pandas as pd
    idx = pd.date_range("2000-01-01", periods=730, freq="D")
    tas = np.zeros(730, np.float32); tas[(idx >= "2000-11-01") & (idx <= "2001-03-01")] = 280
    ta = TimeAxis.daily("2000-01-01", 730)
    mids = ta.date_index_in_periods("YS-JUL", "01-01")
    poff = ta.period_offsets("YS-JUL")
    rel = [int(m) - int(s) if m >= 0 else None for m, s in zip(mids, poff[:-1])]   # index inside each group
    out = O.season(tas >= np.float32(278.15), 6, rel, poff, "length", ta.doy)
    assert out[ta.period_labels("YS-JUL").index("2000-07-01")] == 121


def test_runs_with_holes_reference_known_answers():
    """tests/test_run_length.py:135-162 (values only): window_stop == 1 reproduces the input runs;
    stop runs of 3 bridge the one- and two-step gaps and keep the four-step gap."""
    from oracle import xclim_oracle as O
    values = np.zeros((365, 3))
    values[1:11] = 1
    np.testing.assert_array_equal(O.runs_with_holes(values != 0, 1, values == 0, 1), values)
    v = np.zeros(365)
    a = [0, 1, 0, 1, 1, 0, 0, 1, 1, 1, 1, 0, 0, 0, 0, 1, 1, 1, 1, 1, 0, 0, 0, 0]
    v[:len(a)] = a
    expected = v * 0
    expected[1:11] = 1
    expected[15:20] = 1
    np.testing.assert_array_equal(O.runs_with_holes(v == 1, 1, v == 0, 3), expected)
    # the same through spell_mask(min_gap=3) and the spell statistics (one period): runs of 10 and 5
    x = np.where(v == 1, 0.0, 5.0).astype(np.float32)[:, None]
    np.testing.assert_array_equal(O.spell_mask(x, 1, None, "<", 1.0, min_gap=3)[:, 0], expected.astype(bool))
    poff = np.array([0, 365], dtype=np.int32)
    assert O.spell_length_statistics(x, 1.0, 1, None, "<", "max", poff, min_gap=3)[0, 0] == 10
    assert O.spell_length_statistics(x, 1.0, 1, None, "<", "count", poff, min_gap=3)[0, 0] == 2


@pytest.mark.parametrize("op,expected", [(">", 6), (">=", 5), ("==", 5), ("!=", 1), ("lt", None), ("le", None)])
def test_known_answers_first_day_threshold_reached(op, expected):
    """tests/test_generic.py:343-383 (values): pr = 0, .001, ..., .007 then zeros; first day (doy) on
    which `pr op 0.004` holds after 01-01, window 1.  The '<' family uses the flipped vector (:361-383)."""
    a = np.zeros(365)
    a[:8] = np.arange(8) / 1000
    if expected is None:
        a[:8] = a[:8][::-1].copy()
        expected = {"lt": 5, "le": 4}[op]
    cond = O.compare(a[:, None], op, 0.004)
    idx = O.first_run_after_date(cond, 1, 0)[0]          # mid = index of 01-01 in the (single) group
    assert idx + 1 == expected                             # dayofyear of a series starting on 1 January


def test_known_answers_adjust_doy_calendar():
    """tests/test_calendar.py:142-200 (values): 360 -> 366, 366 -> 360, a 92-day window onto 93 days
    (all_leap JJA), and a leap DJF table onto a noleap axis keep their end points."""
    src = np.arange(360, dtype=np.float64)
    doy = np.concatenate([np.arange(1, 367), np.arange(1, 366)])          # 2000-01-01 .. 2001-12-31
    out = O.adjust_doy_calendar(src, doy, cal_max_doy=366)
    assert out.shape[0] == 366 and out[0] == src[0] and out[365] == src[359]
    src = np.arange(366, dtype=np.float64)
    out = O.adjust_doy_calendar(src, np.arange(1, 361), cal_max_doy=360)
    assert out.shape[0] == 360 and out[0] == src[0] and out[359] == src[365]
    src = np.arange(92, dtype=np.float64)                                  # doys 152..243 -> 153..244
    out = O.adjust_doy_calendar(src, np.arange(153, 245), cal_max_doy=366)
    assert out.shape[0] == 92 and out[0] == src[0] and out[-1] == src[-1]
    # the same table size as the calendar: returned untouched (:748-750)
    tab = np.arange(365, dtype=np.float64)
    assert O.adjust_doy_calendar(tab, np.arange(1, 366), cal_max_doy=365) is tab
    # resample_doy gathers by day of year
    np.testing.assert_array_equal(O.resample_doy(tab, np.array([1, 365, 2]), cal_max_doy=365), [0, 364, 1])


def _date_index(start, n, date):
    """Index of MM-DD in a standard-calendar daily series of n steps starting at `start` (None if absent)."""
    from xclim_b200 import TimeAxis
    ta = TimeAxis.daily(start, n)
    mm, dd = (int(v) for v in date.split("-"))
    hit = np.nonzero((ta.month == mm) & (ta.day == dd))[0]
    return (int(hit[0]) if hit.size else None), ta


@pytest.mark.parametrize("date,end,expected", [("07-01", 210, 70), ("07-01", 190, 50), ("04-01", 150, 0),
                                               ("11-01", 150, 165), (None, 150, 10)])
def test_known_answers_season_length_with_dates(date, end, expected):
    """tests/test_run_length.py:473-503."""
    t = np.zeros(360)
    t[140:end] = 1
    mid, _ = _date_index("2000-01-01", 360, date) if date else (None, None)
    _, _, length = O.season_group(t == 1, 1, mid, has_date=date is not None)
    assert length == expected


@pytest.mark.parametrize("coord,date,end,expected", [("dayofyear", "07-01", 210, 211), (False, "07-01", 190, 190),
                                                     ("dayofyear", "04-01", 150, np.nan),
                                                     ("dayofyear", "11-01", 150, 306)])
def test_known_answers_run_end_after_date(coord, date, end, expected):
    """tests/test_run_length.py:505-529."""
    t = np.zeros(360)
    t[140:end] = 1
    mid, ta = _date_index("2000-01-01", 360, date)
    v = O.run_end_after_date(t == 1, 1, mid)
    if coord and not np.isnan(v):
        v = ta.doy[int(v)]
    np.testing.assert_array_equal(v, expected)


@pytest.mark.parametrize("coord,date,beg,expected", [("dayofyear", "07-01", 210, 211), (False, "07-01", 190, 190),
                                                     ("dayofyear", "04-01", False, np.nan),
                                                     ("dayofyear", "11-01", 150, 306)])
def test_known_answers_first_run_after_date(coord, date, beg, expected):
    """tests/test_run_length.py:531-554."""
    t = np.zeros(365)
    if beg:
        t[beg:] = 1
    mid, ta = _date_index("2000-01-01", 365, date)
    v = O.first_run_after_date(t == 1, 1, mid)
    if coord and not np.isnan(v):
        v = ta.doy[int(v)]
    np.testing.assert_array_equal(v, expected)


@pytest.mark.parametrize("coord,date,end,expected", [("dayofyear", "07-01", 210, 183), (False, "07-01", 190, 182),
                                                     ("dayofyear", "04-01", 150, np.nan),
                                                     ("dayofyear", "11-01", 150, 150)])
def test_known_answers_last_run_before_date(coord, date, end, expected):
    """tests/test_run_length.py:556-579."""
    t = np.zeros(360)
    t[140:end] = 1
    mid, ta = _date_index("2000-01-01", 360, date)
    v = O.last_run_before_date(t == 1, 1, mid)
    if coord and not np.isnan(v):
        v = ta.doy[int(v)]
    np.testing.assert_array_equal(v, expected)
