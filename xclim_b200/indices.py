"""Index entry points (L3 of the reference) for the hot-path configurations.

Same names / arguments / units as ``xclim.indices`` so that they can be bound to the existing
``Indicator`` registry through ``compute=`` (core/indicator.py:471-518, 884-886).
"""
from __future__ import annotations

from . import generic
from .units import threshold_in_units_of


def maximum_consecutive_dry_days(pr, thresh="1 mm/day", op="<", freq="YS", resample_before_rl=True):
    """Longest spell with precipitation under a threshold -- indices/_threshold.py:2895-2937."""
    thr = threshold_in_units_of(thresh, pr)
    return generic.spell_length_statistics(pr, thr, 1, None, op, "max", freq, resample_before_rl=resample_before_rl)


def maximum_consecutive_wet_days(pr, thresh="1 mm/day", op=">=", freq="YS", resample_before_rl=True):
    """indices/_threshold.py:799-841 (``op`` in {">", ">="}, third positional argument like the reference)."""
    from . import _lib
    _lib.op_code(op, (">", ">="))
    thr = threshold_in_units_of(thresh, pr)
    return generic.spell_length_statistics(pr, thr, 1, None, op, "max", freq, resample_before_rl=resample_before_rl)


def tg_mean(tas, freq="YS"):
    """Mean of daily mean temperature -- indices/_simple.py:76-113."""
    return generic.select_resample_op(tas, op="mean", freq=freq)


def wetdays(pr, thresh="1.0 mm/day", freq="YS", op=">="):
    """indices/_threshold.py:2749-2789."""
    thr = threshold_in_units_of(thresh, pr)
    out = generic.threshold_count(pr, op, thr, freq, constrain=(">", ">="))
    return out.assign_attrs(units="d")


def dry_days(pr, thresh="0.2 mm/d", freq="YS", op="<"):
    """indices/_threshold.py:756-796."""
    thr = threshold_in_units_of(thresh, pr)
    out = generic.threshold_count(pr, op, thr, freq, constrain=("<", "<="))
    return out.assign_attrs(units="d")


# ------------------------------------------------------------------ percentile-threshold day counts
def _percentile_day_count(da, per, freq, bootstrap, op, constrain):
    """Shared body of tx90p & family -- indices/_multivariate.py:1583-1590:
    ``thresh = resample_doy(per, da); threshold_count(da, op, thresh, freq)``; the (lat, lon, time)
    float64 threshold array of the reference is never built: the kernel indexes the per-doy table."""
    import numpy as np

    from . import _lib, device
    from .calendar import adjust_table, table_on_device
    from .generic import _unwrap, _wrap_periods
    from .field import attrs_of

    code = _lib.op_code(op, constrain)
    if bootstrap:
        from .bootstrapping import bootstrap_doy_count
        return bootstrap_doy_count(da, per, freq, op, constrain)
    x2d, cell_shape, other, ta = _unwrap(da)
    table = _table_in_units_of(table_on_device(per, cell_shape, other, x2d.device), per, da)
    table, doy_idx = adjust_table(table, ta)
    out, _ = device.doy_threshold_count(x2d, ta.period_offsets(freq), doy_idx, table, code)
    attrs = attrs_of(da)
    attrs["units"] = "d"
    return _wrap_periods(da, out, cell_shape, other, ta, freq, attrs, dtype=np.int64)


def _table_in_units_of(table, per, da):
    """``convert_units_to(per, da)`` (indices/_multivariate.py:1583) on the device table: the conversions
    of the small unit table are affine, so two probe values give scale and offset."""
    from .field import attrs_of
    from .units import convert_units_to
    pu, du = attrs_of(per).get("units"), attrs_of(da).get("units")
    if pu is None or du is None or pu == du:
        return table
    f0, f1 = convert_units_to(f"0 {pu}", du), convert_units_to(f"1 {pu}", du)
    if f0 == 0.0 and f1 == 1.0:
        return table
    return table * (f1 - f0) + f0


def days_over_precip_thresh(pr, pr_per, thresh="1 mm/day", freq="YS", bootstrap=False, op=">"):
    """Days with precipitation over both a doy percentile and a wet-day threshold (ETCCDI R95p-days) --
    indices/_multivariate.py:1176-1233: ``tp = pr_per.where(pr_per > thresh, thresh)`` then the tx90p
    count; the clamp is applied to the per-doy table on the device."""
    import numpy as np
    import torch

    from . import _lib, device
    from .calendar import adjust_table, table_on_device
    from .field import attrs_of
    from .generic import _unwrap, _wrap_periods

    if bootstrap:
        raise NotImplementedError("days_over_precip_thresh(bootstrap=True) is not supported by the B200 hot path")
    code = _lib.op_code(op, (">", ">="))
    thr = threshold_in_units_of(thresh, pr) if isinstance(thresh, str) else float(thresh)
    x2d, cell_shape, other, ta = _unwrap(pr)
    table = _table_in_units_of(table_on_device(pr_per, cell_shape, other, x2d.device), pr_per, pr)
    table = torch.where(table > thr, table, torch.full_like(table, thr))     # NaN percentiles -> thresh
    table, doy_idx = adjust_table(table, ta)
    out, _ = device.doy_threshold_count(x2d, ta.period_offsets(freq), doy_idx, table, code)
    attrs = attrs_of(pr)
    attrs["units"] = "d"
    return _wrap_periods(pr, out, cell_shape, other, ta, freq, attrs, dtype=np.int64)


def tx90p(tasmax, tasmax_per, freq="YS", bootstrap=False, op=">"):
    """Days with daily maximum temperature over the 90th percentile -- indices/_multivariate.py:1534-1590."""
    return _percentile_day_count(tasmax, tasmax_per, freq, bootstrap, op, (">", ">="))


def tx10p(tasmax, tasmax_per, freq="YS", bootstrap=False, op="<"):
    """indices/_multivariate.py:1593-1650."""
    return _percentile_day_count(tasmax, tasmax_per, freq, bootstrap, op, ("<", "<="))


def tn90p(tasmin, tasmin_per, freq="YS", bootstrap=False, op=">"):
    """indices/_multivariate.py:1417-1473."""
    return _percentile_day_count(tasmin, tasmin_per, freq, bootstrap, op, (">", ">="))


def tn10p(tasmin, tasmin_per, freq="YS", bootstrap=False, op="<"):
    """indices/_multivariate.py:1476-1531."""
    return _percentile_day_count(tasmin, tasmin_per, freq, bootstrap, op, ("<", "<="))


def tg90p(tas, tas_per, freq="YS", bootstrap=False, op=">"):
    """indices/_multivariate.py:1300-1356."""
    return _percentile_day_count(tas, tas_per, freq, bootstrap, op, (">", ">="))


def tg10p(tas, tas_per, freq="YS", bootstrap=False, op="<"):
    """indices/_multivariate.py:1359-1414."""
    return _percentile_day_count(tas, tas_per, freq, bootstrap, op, ("<", "<="))


# ------------------------------------------------------------------ rolling / spell families
def max_n_day_precipitation_amount(pr, window=1, freq="YS"):
    """Highest precipitation amount cumulated over an n-day moving window -- indices/_simple.py:485-525:
    ``rate2amount(pr).rolling(time=window).sum(skipna=False).resample(time=freq).max()``.  The input
    is expected in mm/d (rate2amount is then the identity factor 1 d, core/units.py:853-937)."""
    from . import _lib, device
    from .field import attrs_of
    from .generic import _unwrap, _wrap_periods
    x2d, cell_shape, other, ta = _unwrap(pr)
    out = device.rolling_period_reduce(x2d, ta.period_offsets(freq), window, _lib.STATS["sum"], False,
                                       _lib.STATS["max"])
    attrs = attrs_of(pr)
    attrs["units"] = "mm"
    return _wrap_periods(pr, out, cell_shape, other, ta, freq, attrs)


def _dry_wet_spell(pr, thresh, window, op, win_reducer, spell_reducer, freq, resample_before_rl, **indexer):
    thr = threshold_in_units_of(thresh, pr)
    return generic.spell_length_statistics(pr, thr, window, win_reducer, op, spell_reducer, freq,
                                           resample_before_rl=resample_before_rl, **indexer)


def dry_spell_frequency(pr, thresh="1.0 mm", window=3, freq="YS", resample_before_rl=True, op="sum", **indexer):
    """indices/_threshold.py:3314-3382 (input in mm/d so that the daily amount equals the rate)."""
    return _dry_wet_spell(pr, thresh.replace(" mm", " mm/d") if isinstance(thresh, str) else thresh, window, "<", op,
                          "count", freq, resample_before_rl, **indexer)


def dry_spell_total_length(pr, thresh="1.0 mm", window=3, op="sum", freq="YS", resample_before_rl=True, **indexer):
    """indices/_threshold.py:3385-3454."""
    return _dry_wet_spell(pr, thresh.replace(" mm", " mm/d") if isinstance(thresh, str) else thresh, window, "<", op,
                          "sum", freq, resample_before_rl, **indexer)


def dry_spell_max_length(pr, thresh="1.0 mm", window=1, op="sum", freq="YS", resample_before_rl=True, **indexer):
    """indices/_threshold.py:3457-3522."""
    return _dry_wet_spell(pr, thresh.replace(" mm", " mm/d") if isinstance(thresh, str) else thresh, window, "<", op,
                          "max", freq, resample_before_rl, **indexer)


def wet_spell_frequency(pr, thresh="1.0 mm", window=3, freq="YS", resample_before_rl=True, op="sum", **indexer):
    """indices/_threshold.py:3525-3592."""
    return _dry_wet_spell(pr, thresh.replace(" mm", " mm/d") if isinstance(thresh, str) else thresh, window, ">=", op,
                          "count", freq, resample_before_rl, **indexer)


def wet_spell_total_length(pr, thresh="1.0 mm", window=3, op="sum", freq="YS", resample_before_rl=True, **indexer):
    """indices/_threshold.py:3596-3663."""
    return _dry_wet_spell(pr, thresh.replace(" mm", " mm/d") if isinstance(thresh, str) else thresh, window, ">=", op,
                          "sum", freq, resample_before_rl, **indexer)


def wet_spell_max_length(pr, thresh="1.0 mm", window=1, op="sum", freq="YS", resample_before_rl=True, **indexer):
    """indices/_threshold.py:3667-3733."""
    return _dry_wet_spell(pr, thresh.replace(" mm", " mm/d") if isinstance(thresh, str) else thresh, window, ">=", op,
                          "max", freq, resample_before_rl, **indexer)


def hot_spell_max_magnitude(tasmax, thresh="25.0 degC", window=3, freq="YS", resample_before_rl=True):
    """Largest cumulated exceedance of a hot spell -- indices/_threshold.py:2019-2073; the
    ``(tasmax - thresh).clip(0)`` array of the reference is never built."""
    from . import _lib, device
    from .field import attrs_of
    from .generic import _unwrap, _wrap_periods
    thr = threshold_in_units_of(thresh, tasmax)
    x2d, cell_shape, other, ta = _unwrap(tasmax)
    out = device.period_run_maxsum(x2d, ta.period_offsets(freq), _lib.OPS[">"], thr, window, resample_before_rl)
    attrs = attrs_of(tasmax)
    attrs["units"] = "K d"
    return _wrap_periods(tasmax, out, cell_shape, other, ta, freq, attrs)


# =====================================================================================================
# The index families of SURVEY.md section 2.2 (the "batch of 50 atmos indicators" configuration): thin
# entry points over the same few kernels.  Signatures/defaults follow xclim.indices; thresholds are
# converted on the host (a Python float reaches the kernel, compared in float32 like numpy >= 2).
# =====================================================================================================
def _resample(da, op, freq):
    return generic.select_resample_op(da, op=op, freq=freq)


def _count(da, thresh, op, freq, constrain):
    thr = threshold_in_units_of(thresh, da) if isinstance(thresh, str) else float(thresh)
    return generic.threshold_count(da, op, thr, freq, constrain=constrain).assign_attrs(units="d")


def _spell(da, thresh, op, constrain, reducer, window, freq, resample_before_rl, units="d", clip_below=None):
    """compare -> rl.resample_and_rl(<run statistic>, window) (e.g. indices/_threshold.py:204-214)."""
    import numpy as np

    from . import _lib, device
    from .field import attrs_of
    from .generic import _unwrap, _wrap_periods
    code = _lib.op_code(op, constrain)
    thr = threshold_in_units_of(thresh, da) if isinstance(thresh, str) else float(thresh)
    x2d, cell_shape, other, ta = _unwrap(da)
    out, _ = device.period_runstat(x2d, ta.period_offsets(freq), code, thr, _lib.RL_REDUCERS[reducer], window,
                                   resample_before_rl)
    if clip_below is not None:      # `max_l.where(max_l >= window, 0)` (indices/_threshold.py:311)
        out = out * (out >= clip_below)
    attrs = attrs_of(da)
    attrs["units"] = units
    return _wrap_periods(da, out, cell_shape, other, ta, freq, attrs, dtype=np.float32)


# ---- resample reductions (indices/_simple.py:46-303, 447-482; _multivariate.py:930-1056)
def tg_max(tas, freq="YS"):
    return _resample(tas, "max", freq)


def tg_min(tas, freq="YS"):
    return _resample(tas, "min", freq)


def tn_max(tasmin, freq="YS"):
    return _resample(tasmin, "max", freq)


def tn_mean(tasmin, freq="YS"):
    return _resample(tasmin, "mean", freq)


def tn_min(tasmin, freq="YS"):
    return _resample(tasmin, "min", freq)


def tx_max(tasmax, freq="YS"):
    return _resample(tasmax, "max", freq)


def tx_mean(tasmax, freq="YS"):
    return _resample(tasmax, "mean", freq)


def tx_min(tasmax, freq="YS"):
    return _resample(tasmax, "min", freq)


def max_1day_precipitation_amount(pr, freq="YS"):
    """indices/_simple.py:447-482 (input in mm/d: the daily amount in mm equals the rate)."""
    return _resample(pr, "max", freq).assign_attrs(units="mm")


def precip_accumulation(pr, freq="YS"):
    """indices/_multivariate.py:930-991 without phase separation (input in mm/d -> mm)."""
    return _resample(pr, "sum", freq).assign_attrs(units="mm")


def precip_average(pr, freq="YS"):
    """Mean daily precipitation amount -- indices/_multivariate.py:994-1054 without phase separation (input in
    mm/d -> mm)."""
    return _resample(pr, "mean", freq).assign_attrs(units="mm")


def sfcWind_max(sfcWind, freq="YS"):
    return _resample(sfcWind, "max", freq)


def sfcWind_mean(sfcWind, freq="YS"):
    return _resample(sfcWind, "mean", freq)


def sfcWind_min(sfcWind, freq="YS"):
    return _resample(sfcWind, "min", freq)


def sfcWindmax_max(sfcWindmax, freq="YS"):  # noqa: N802
    """indices/_simple.py:720-753."""
    return _resample(sfcWindmax, "max", freq)


def sfcWindmax_mean(sfcWindmax, freq="YS"):  # noqa: N802
    """indices/_simple.py:757-790."""
    return _resample(sfcWindmax, "mean", freq)


def sfcWindmax_min(sfcWindmax, freq="YS"):  # noqa: N802
    """indices/_simple.py:794-826."""
    return _resample(sfcWindmax, "min", freq)


def extreme_temperature_range(tasmin, tasmax, freq="YS"):
    """max(tasmax) - min(tasmin) per period -- indices/_multivariate.py:601-637 (both inputs in the same
    units; the result is a temperature difference)."""
    from .field import Field, attrs_of, is_xarray
    from .units import units_of
    if units_of(tasmax) != units_of(tasmin):
        raise NotImplementedError("extreme_temperature_range: give tasmax and tasmin in the same units")
    hi, lo = _resample(tasmax, "max", freq), _resample(tasmin, "min", freq)
    out = hi.values - lo.values            # numpy arrays or CUDA tensors
    u = attrs_of(tasmax).get("units", "")
    attrs = {**attrs_of(hi), "units": {"degC": "K", "°C": "K", "C": "K"}.get(u, u), "units_metadata": "temperature: difference"}
    if is_xarray(hi):
        return hi.copy(data=out).assign_attrs(**attrs)
    return Field(out, hi.dims, hi.time, dict(hi.coords), attrs, hi.name)


# ---- threshold counts (indices/_simple.py:334-444, _threshold.py:122-155, 2422-2632, 3135-3167)
def warm_day_frequency(tasmax, thresh="30 degC", freq="YS", op=">"):
    """indices/_threshold.py:2674-2712."""
    return _count(tasmax, thresh, op, freq, (">", ">="))


def warm_night_frequency(tasmin, thresh="22 degC", freq="YS", op=">"):
    """indices/_threshold.py:2716-2745."""
    return _count(tasmin, thresh, op, freq, (">", ">="))


def days_with_snow(prsn, low="0 kg m-2 s-1", high="1E6 kg m-2 s-1", freq="YS-JUL"):
    """Days with ``low < prsn <= high`` -- indices/_threshold.py:1817-1860 (``domain_count``)."""
    lo = threshold_in_units_of(low, prsn) if isinstance(low, str) else float(low)
    hi = threshold_in_units_of(high, prsn) if isinstance(high, str) else float(high)
    return generic.domain_count(prsn, lo, hi, freq).assign_attrs(units="d")


def frost_days(tasmin, thresh="0 degC", freq="YS"):
    return _count(tasmin, thresh, "<", freq, ("<", "<="))


def ice_days(tasmax, thresh="0 degC", freq="YS"):
    return _count(tasmax, thresh, "<", freq, ("<", "<="))


def hot_days(tasmax, thresh="25 degC", freq="YS"):
    return _count(tasmax, thresh, ">", freq, (">", ">="))


def tx_days_above(tasmax, thresh="25.0 degC", freq="YS", op=">"):
    return _count(tasmax, thresh, op, freq, (">", ">="))


def tx_days_below(tasmax, thresh="25.0 degC", freq="YS", op="<"):
    return _count(tasmax, thresh, op, freq, ("<", "<="))


def tn_days_above(tasmin, thresh="20.0 degC", freq="YS", op=">"):
    return _count(tasmin, thresh, op, freq, (">", ">="))


def tn_days_below(tasmin, thresh="-10.0 degC", freq="YS", op="<"):
    return _count(tasmin, thresh, op, freq, ("<", "<="))


def tg_days_above(tas, thresh="10.0 degC", freq="YS", op=">"):
    return _count(tas, thresh, op, freq, (">", ">="))


def tg_days_below(tas, thresh="10.0 degC", freq="YS", op="<"):
    return _count(tas, thresh, op, freq, ("<", "<="))


def calm_days(sfcWind, thresh="2 m s-1", freq="MS"):
    return _count(sfcWind, thresh, "<", freq, ("<", "<="))


def windy_days(sfcWind, thresh="10.8 m s-1", freq="MS"):
    return _count(sfcWind, thresh, ">=", freq, (">", ">="))


def _ratio(num, den):
    """``num / den`` in float64 for numpy arrays or CUDA tensors (set_options(device_outputs=True))."""
    import numpy as np
    if hasattr(num, "is_cuda"):
        import torch
        if not hasattr(den, "is_cuda"):
            den = torch.from_numpy(np.ascontiguousarray(den)).to(num.device)
        return num.to(torch.float64) / den.to(torch.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.asarray(num, dtype=np.float64) / den


def wetdays_prop(pr, thresh="1.0 mm/day", freq="YS", op=">="):
    """indices/_threshold.py:2792-2834: mean of the boolean wet-day mask per period."""
    import numpy as np
    from .field import time_axis_of as _ta
    cnt = _count(pr, thresh, op, freq, (">", ">="))
    n = np.diff(_ta(pr).period_offsets(freq)).reshape((-1,) + (1,) * (cnt.values.ndim - 1))
    out = _ratio(cnt.values, n)
    from .field import Field, is_xarray
    if is_xarray(cnt):
        return cnt.copy(data=out).assign_attrs(units="1")
    return Field(out, cnt.dims, cnt.time, dict(cnt.coords), {**cnt.attrs, "units": "1"}, cnt.name)


# ---- thresholded sums (indices/_threshold.py:680-753, 905-972, 2127-2166)
def growing_degree_days(tas, thresh="4.0 degC", freq="YS"):
    return generic.cumulative_difference(tas, threshold=thresh, op=">", freq=freq)


def cooling_degree_days(tas, thresh="18 degC", freq="YS"):
    return generic.cumulative_difference(tas, threshold=thresh, op=">", freq=freq)


def heating_degree_days(tas, thresh="17.0 degC", freq="YS"):
    return generic.cumulative_difference(tas, threshold=thresh, op="<", freq=freq)


def daily_pr_intensity(pr, thresh="1 mm/day", freq="YS", op=">="):
    """indices/_threshold.py:680-753: precipitation of wet days divided by the number of wet days."""
    import numpy as np
    thr = threshold_in_units_of(thresh, pr)
    s = generic.thresholded_statistics(pr, op, thr, "sum", freq, constrain=(">", ">="))
    wd = _count(pr, thr, op, freq, (">", ">="))
    out = _ratio(s.values, wd.values)
    from .field import Field, is_xarray
    if is_xarray(s):
        return s.copy(data=out).assign_attrs(units="mm d-1")
    return Field(out, s.dims, s.time, dict(s.coords), {**s.attrs, "units": "mm d-1"}, s.name)


# ---- spells on runs (indices/_threshold.py:158-313, 1476-1523, 1972-2016, 2169-2345, 2837-3000)
def cold_spell_days(tas, thresh="-10 degC", window=5, freq="YS-JUL", op="<", resample_before_rl=True):
    return _spell(tas, thresh, op, ("<", "<="), "sum", window, freq, resample_before_rl)


def cold_spell_frequency(tas, thresh="-10 degC", window=5, freq="YS-JUL", op="<", resample_before_rl=True):
    return _spell(tas, thresh, op, ("<", "<="), "count", window, freq, resample_before_rl, units="")


def cold_spell_max_length(tas, thresh="-10 degC", window=1, freq="YS-JUL", op="<", resample_before_rl=True):
    return _spell(tas, thresh, op, ("<", "<="), "max", 1, freq, resample_before_rl, clip_below=window)


def cold_spell_total_length(tas, thresh="-10 degC", window=3, freq="YS-JUL", op="<", resample_before_rl=True):
    return _spell(tas, thresh, op, ("<", "<="), "sum", window, freq, resample_before_rl)


def hot_spell_frequency(tasmax, thresh="30 degC", window=3, freq="YS", op=">", resample_before_rl=True):
    return _spell(tasmax, thresh, op, (">", ">="), "count", window, freq, resample_before_rl, units="")


def hot_spell_max_length(tasmax, thresh="30 degC", window=1, freq="YS", op=">", resample_before_rl=True):
    return _spell(tasmax, thresh, op, (">", ">="), "max", 1, freq, resample_before_rl, clip_below=window)


def hot_spell_total_length(tasmax, thresh="30 degC", window=3, freq="YS", op=">", resample_before_rl=True):
    return _spell(tasmax, thresh, op, (">", ">="), "sum", window, freq, resample_before_rl)


def heat_wave_index(tasmax, thresh="25.0 degC", window=5, freq="YS", op=">", resample_before_rl=True):
    return _spell(tasmax, thresh, op, (">", ">="), "sum", window, freq, resample_before_rl)


def frost_free_spell_max_length(tasmin, thresh="0.0 degC", window=1, freq="YS-JUL", op=">=", resample_before_rl=True):
    return _spell(tasmin, thresh, op, (">", ">="), "max", 1, freq, resample_before_rl, clip_below=window)


def maximum_consecutive_frost_days(tasmin, thresh="0.0 degC", freq="YS-JUL", resample_before_rl=True):
    return cold_spell_max_length(tasmin, thresh=thresh, window=1, freq=freq, op="<",
                                 resample_before_rl=resample_before_rl)


def maximum_consecutive_frost_free_days(tasmin, thresh="0 degC", freq="YS", resample_before_rl=True):
    return frost_free_spell_max_length(tasmin, thresh=thresh, window=1, freq=freq, op=">=",
                                       resample_before_rl=resample_before_rl)


def maximum_consecutive_tx_days(tasmax, thresh="25 degC", freq="YS", resample_before_rl=True):
    return hot_spell_max_length(tasmax, thresh=thresh, window=1, freq=freq, op=">",
                                resample_before_rl=resample_before_rl)


#: the (name, variable) list of the "batch of 50" configuration (BASELINE.json configs[4]); every entry is
#: parity-tested against the oracle in tests/test_gpu_batch.py
BATCH_INDICATORS = [
    ("tg_mean", "tas"), ("tg_max", "tas"), ("tg_min", "tas"), ("tn_mean", "tasmin"), ("tn_max", "tasmin"),
    ("tn_min", "tasmin"), ("tx_mean", "tasmax"), ("tx_max", "tasmax"), ("tx_min", "tasmax"),
    ("max_1day_precipitation_amount", "pr"), ("precip_accumulation", "pr"), ("max_n_day_precipitation_amount", "pr"),
    ("frost_days", "tasmin"), ("ice_days", "tasmax"), ("hot_days", "tasmax"), ("tx_days_above", "tasmax"),
    ("tx_days_below", "tasmax"), ("tn_days_above", "tasmin"), ("tn_days_below", "tasmin"), ("tg_days_above", "tas"),
    ("tg_days_below", "tas"), ("wetdays", "pr"), ("dry_days", "pr"), ("wetdays_prop", "pr"),
    ("growing_degree_days", "tas"), ("cooling_degree_days", "tas"), ("heating_degree_days", "tas"),
    ("daily_pr_intensity", "pr"),
    ("cold_spell_days", "tas"), ("cold_spell_frequency", "tas"), ("cold_spell_max_length", "tas"),
    ("cold_spell_total_length", "tas"), ("hot_spell_frequency", "tasmax"), ("hot_spell_max_length", "tasmax"),
    ("hot_spell_total_length", "tasmax"), ("hot_spell_max_magnitude", "tasmax"), ("heat_wave_index", "tasmax"),
    ("frost_free_spell_max_length", "tasmin"), ("maximum_consecutive_frost_days", "tasmin"),
    ("maximum_consecutive_frost_free_days", "tasmin"), ("maximum_consecutive_tx_days", "tasmax"),
    ("maximum_consecutive_dry_days", "pr"), ("maximum_consecutive_wet_days", "pr"),
    ("dry_spell_frequency", "pr"), ("dry_spell_total_length", "pr"), ("dry_spell_max_length", "pr"),
    ("wet_spell_frequency", "pr"), ("tx90p", "tasmax"), ("tx10p", "tasmax"), ("tn90p", "tasmin"),
]


# ---- seasons and dates (indices/_threshold.py:975-1395, 1526-1700)
def growing_season_start(tas, thresh="5.0 degC", mid_date="07-01", window=5, freq="YS", op=">="):
    return generic.season(tas, thresh, window, op, "start", freq, mid_date=mid_date, constrain=(">", ">="))


def growing_season_end(tas, thresh="5.0 degC", mid_date="07-01", window=5, freq="YS", op=">"):
    return generic.season(tas, thresh, window, op, "end", freq, mid_date=mid_date, constrain=(">", ">="))


def growing_season_length(tas, thresh="5.0 degC", window=6, mid_date="07-01", freq="YS", op=">="):
    return generic.season(tas, thresh, window, op, "length", freq, mid_date=mid_date, constrain=(">", ">="))


def frost_season_length(tasmin, window=5, mid_date="01-01", thresh="0.0 degC", freq="YS-JUL", op="<"):
    return generic.season(tasmin, thresh, window, op, "length", freq, mid_date=mid_date, constrain=("<", "<="))


def frost_free_season_start(tasmin, thresh="0.0 degC", window=5, mid_date="07-01", op=">=", freq="YS"):
    return generic.season(tasmin, thresh, window, op, "start", freq, mid_date=mid_date, constrain=(">", ">="))


def frost_free_season_end(tasmin, thresh="0.0 degC", window=5, mid_date="07-01", op=">=", freq="YS"):
    return generic.season(tasmin, thresh, window, op, "end", freq, mid_date=mid_date, constrain=(">", ">="))


def frost_free_season_length(tasmin, thresh="0.0 degC", window=5, mid_date="07-01", op=">=", freq="YS"):
    return generic.season(tasmin, thresh, window, op, "length", freq, mid_date=mid_date, constrain=(">", ">="))


def first_day_temperature_below(tas, thresh="0 degC", op="<", after_date="07-01", window=1, freq="YS"):
    return generic.first_day_threshold_reached(tas, threshold=thresh, op=op, after_date=after_date, window=window,
                                               freq=freq, constrain=("<", "<="))


def first_day_temperature_above(tas, thresh="0 degC", op=">", after_date="01-01", window=1, freq="YS"):
    return generic.first_day_threshold_reached(tas, threshold=thresh, op=op, after_date=after_date, window=window,
                                               freq=freq, constrain=(">", ">="))


def last_spring_frost(tasmin, thresh="0 degC", op="<", before_date="07-01", window=1, freq="YS"):
    """indices/_threshold.py:1526-1582: day of year of the last frost run before a date."""
    import numpy as np

    from . import _lib, seasons
    from .field import attrs_of
    from .generic import _unwrap, _wrap_periods
    code = _lib.op_code(op, ("<", "<="))
    thr = threshold_in_units_of(thresh, tasmin)
    x2d, cell_shape, other, ta = _unwrap(tasmin)
    out = seasons.last_run_before_date(x2d, ta, freq, code, thr, window, before_date)
    attrs = attrs_of(tasmin)
    attrs.update(units="", is_dayofyear=np.int32(1), calendar=ta.calendar)
    return _wrap_periods(tasmin, out, cell_shape, other, ta, freq, attrs, dtype=np.float64)


# ---- bivariate conditions (indices/_multivariate.py:646-880, 1653-1716; generic.py:1002-1073)
def _bivariate(v1, v2, th1, th2, op1, op2, reducer, window, freq, resample_before_rl, units, var_any=False,
               constrain=None, dtype=None):
    import numpy as np

    from . import _lib, device
    from .field import attrs_of
    from .generic import _unwrap, _wrap_periods
    c1, c2 = _lib.op_code(op1, constrain), _lib.op_code(op2, constrain)
    t1 = threshold_in_units_of(th1, v1) if isinstance(th1, str) else float(th1)
    t2 = threshold_in_units_of(th2, v2) if isinstance(th2, str) else float(th2)
    x1, cell_shape, other, ta = _unwrap(v1)
    x2, cs2, _, ta2 = _unwrap(v2)
    if cs2 != cell_shape or len(ta2) != len(ta):
        raise ValueError("the two variables must share the same grid and time axis")
    out = device.period_runstat2(x1, x2, ta.period_offsets(freq), c1, t1, c2, t2, _lib.RL_REDUCERS[reducer], window,
                                 resample_before_rl, var_any)
    attrs = attrs_of(v1)
    attrs["units"] = units
    return _wrap_periods(v1, out, cell_shape, other, ta, freq, attrs, dtype=dtype or np.float32)


def heat_wave_frequency(tasmin, tasmax, thresh_tasmin="22.0 degC", thresh_tasmax="30 degC", window=3, freq="YS", op=">",
                        resample_before_rl=True):
    return _bivariate(tasmin, tasmax, thresh_tasmin, thresh_tasmax, op, op, "count", window, freq, resample_before_rl,
                      "", constrain=(">", ">="))


def heat_wave_max_length(tasmin, tasmax, thresh_tasmin="22.0 degC", thresh_tasmax="30 degC", window=3, freq="YS", op=">",
                         resample_before_rl=True):
    return _bivariate(tasmin, tasmax, thresh_tasmin, thresh_tasmax, op, op, "max", window, freq, resample_before_rl,
                      "d", constrain=(">", ">="))


def heat_wave_total_length(tasmin, tasmax, thresh_tasmin="22.0 degC", thresh_tasmax="30 degC", window=3, freq="YS",
                           op=">", resample_before_rl=True):
    return _bivariate(tasmin, tasmax, thresh_tasmin, thresh_tasmax, op, op, "sum", window, freq, resample_before_rl,
                      "d", constrain=(">", ">="))


def tx_tn_days_above(tasmin, tasmax, thresh_tasmin="22 degC", thresh_tasmax="30 degC", freq="YS", op=">"):
    import numpy as np
    return _bivariate(tasmin, tasmax, thresh_tasmin, thresh_tasmax, op, op, "sum", 1, freq, True, "d",
                      constrain=(">", ">="), dtype=np.int64)


# ---- more thin entry points over the same kernels -----------------------------------------------------
def multiday_temperature_swing(tasmin, tasmax, thresh_tasmin="0 degC", thresh_tasmax="0 degC", window=1, op="mean",
                               op_tasmin="<=", op_tasmax=">", freq="YS", resample_before_rl=True):
    """Statistics of freeze-thaw spells (tasmin op_tasmin thresh AND tasmax op_tasmax thresh) --
    indices/_multivariate.py:426-510: ``op="count"`` is ``windowed_run_events``, the others
    ``rle_statistics(reducer=op)``, both through ``resample_and_rl``."""
    import numpy as np

    from . import _lib, device
    from .field import attrs_of
    from .generic import _unwrap, _wrap_periods
    if op not in _lib.RL_REDUCERS:
        raise NotImplementedError(f"op {op!r} is not supported by the B200 hot path")
    c1 = _lib.op_code(op_tasmin, ("<", "<="))
    c2 = _lib.op_code(op_tasmax, (">", ">="))
    t1 = threshold_in_units_of(thresh_tasmin, tasmin) if isinstance(thresh_tasmin, str) else float(thresh_tasmin)
    t2 = threshold_in_units_of(thresh_tasmax, tasmax) if isinstance(thresh_tasmax, str) else float(thresh_tasmax)
    x1, cell_shape, other, ta = _unwrap(tasmin)
    x2, cs2, _, ta2 = _unwrap(tasmax)
    if cs2 != cell_shape or len(ta2) != len(ta):
        raise ValueError("the two variables must share the same grid and time axis")
    out = device.period_runstat2(x1, x2, ta.period_offsets(freq), c1, t1, c2, t2, _lib.RL_REDUCERS[op], int(window),
                                 resample_before_rl, False)
    attrs = attrs_of(tasmin)
    attrs["units"] = "d"
    return _wrap_periods(tasmin, out, cell_shape, other, ta, freq, attrs, dtype=np.float32)


def daily_freezethaw_cycles(tasmin, tasmax, thresh_tasmin="0 degC", thresh_tasmax="0 degC", op_tasmin="<=",
                            op_tasmax=">", freq="YS"):
    """Days with tasmin <= 0 degC and tasmax > 0 degC -- indices/_multivariate.py:344-423
    (``multiday_temperature_swing(window=1, op="sum")``)."""
    return multiday_temperature_swing(tasmin, tasmax, thresh_tasmin, thresh_tasmax, 1, "sum", op_tasmin, op_tasmax,
                                      freq, True)


def high_precip_low_temp(pr, tas, pr_thresh="0.4 mm/d", tas_thresh="-0.2 degC", freq="YS"):
    """Days with precipitation at or above and temperature under a threshold --
    indices/_multivariate.py:1117-1171."""
    return generic.bivariate_count_occurrences(data_var1=pr, data_var2=tas, threshold_var1=pr_thresh,
                                               threshold_var2=tas_thresh, freq=freq, op_var1=">=", op_var2="<",
                                               var_reducer="all")


def first_snowfall(prsn, thresh="1 mm/day", freq="YS-JUL"):
    """Day of year of the first day with snowfall at or above a threshold -- indices/_threshold.py:1701-1753."""
    return generic.first_occurrence(prsn, thresh, freq, ">=")


def last_snowfall(prsn, thresh="1 mm/day", freq="YS-JUL"):
    """indices/_threshold.py:1757-1809."""
    return generic.last_occurrence(prsn, thresh, freq, ">=")


def snowfall_frequency(prsn, thresh="1 mm/day", freq="YS-JUL"):
    """Percentage of the (non-missing) days of each period with snowfall over a threshold --
    indices/_threshold.py:1863-1916: ``days_with_snow(low=thresh) / count * 100``."""
    import numpy as np

    from . import _lib, device
    from .field import attrs_of
    from .generic import _unwrap, _wrap_periods
    thr = threshold_in_units_of(thresh, prsn) if isinstance(thresh, str) else float(thresh)
    hi = threshold_in_units_of("1E6 kg m-2 s-1", prsn)
    x2d, cell_shape, other, ta = _unwrap(prsn)
    poff = ta.period_offsets(freq)
    above, valid = device.period_count(x2d, poff, _lib.OPS[">"], thr, want_valid=True)
    over, _ = device.period_count(x2d, poff, _lib.OPS[">"], hi)
    out = _ratio(above - over, valid) * 100.0
    attrs = attrs_of(prsn)
    attrs["units"] = "%"
    return _wrap_periods(prsn, out, cell_shape, other, ta, freq, attrs, dtype=np.float64)


def snowfall_intensity(prsn, thresh="1 mm/day", freq="YS-JUL"):
    """Mean snowfall rate (mm/day of liquid water) of the days at or above a threshold, 0 when there is
    none -- indices/_threshold.py:1919-1967.  The mean is taken in the data's units and scaled once."""
    import numpy as np

    from . import _lib, device
    from .field import attrs_of
    from .generic import _unwrap, _wrap_periods
    from .units import convert_units_to, units_of
    thr = threshold_in_units_of(thresh, prsn) if isinstance(thresh, str) else float(thresh)
    scale = convert_units_to(f"1 {units_of(prsn)}", "mm/d")      # data units -> mm/day
    x2d, cell_shape, other, ta = _unwrap(prsn)
    out, _ = device.period_reduce(x2d, ta.period_offsets(freq), _lib.STATS["mean"], _lib.TF_WHERE, _lib.OPS[">="], thr)
    out = out * float(scale)
    out = out.nan_to_num(nan=0.0) if hasattr(out, "nan_to_num") else np.nan_to_num(out, nan=0.0)
    attrs = attrs_of(prsn)
    attrs["units"] = "mm/day"
    return _wrap_periods(prsn, out, cell_shape, other, ta, freq, attrs)




# =====================================================================================================
# The batch as FUSED passes (SURVEY.md section 8d: "unique inputs once each"): every output that shares an
# input variable and a resampling frequency comes out of one streaming pass (``xc_period_multi_f32``).  The
# table below says, per indicator, which slot of which pass it is; thresholds, windows, operators and
# frequencies are read from the indicator functions' own defaults (so the two cannot drift apart), and
# tests/test_gpu_batch.py checks run_batch against the one-call-per-indicator results, values and attrs.
# Kinds: ("stat", name, units) | ("count", op_or_param) | ("prop",) | ("excess", op) | ("intensity",) |
#        ("spell", op, reducer) | ("maxlen", op) | ("maxsum",) | None = not fusable here (own kernel).
# =====================================================================================================
BATCH_FUSED = {
    "tg_mean": ("stat", "mean", None), "tg_max": ("stat", "max", None), "tg_min": ("stat", "min", None),
    "tn_mean": ("stat", "mean", None), "tn_max": ("stat", "max", None), "tn_min": ("stat", "min", None),
    "tx_mean": ("stat", "mean", None), "tx_max": ("stat", "max", None), "tx_min": ("stat", "min", None),
    "max_1day_precipitation_amount": ("stat", "max", "mm"), "precip_accumulation": ("stat", "sum", "mm"),
    "max_n_day_precipitation_amount": ("stat1", "max", "mm"),
    "frost_days": ("count", "<"), "ice_days": ("count", "<"), "hot_days": ("count", ">"),
    "tx_days_above": ("count", "op"), "tx_days_below": ("count", "op"), "tn_days_above": ("count", "op"),
    "tn_days_below": ("count", "op"), "tg_days_above": ("count", "op"), "tg_days_below": ("count", "op"),
    "wetdays": ("count", "op"), "dry_days": ("count", "op"), "wetdays_prop": ("prop",),
    "growing_degree_days": ("excess", ">"), "cooling_degree_days": ("excess", ">"),
    "heating_degree_days": ("excess", "<"), "daily_pr_intensity": ("intensity",),
    "cold_spell_days": ("spell", "sum"), "cold_spell_frequency": ("spell", "count"),
    "cold_spell_max_length": ("maxlen",), "cold_spell_total_length": ("spell", "sum"),
    "hot_spell_frequency": ("spell", "count"), "hot_spell_max_length": ("maxlen",),
    "hot_spell_total_length": ("spell", "sum"), "hot_spell_max_magnitude": ("maxsum",),
    "heat_wave_index": ("spell", "sum"), "frost_free_spell_max_length": ("maxlen",),
    "maximum_consecutive_frost_days": ("maxlen", "<"), "maximum_consecutive_frost_free_days": ("maxlen", ">="),
    "maximum_consecutive_tx_days": ("maxlen", ">"),
    "maximum_consecutive_dry_days": ("maxlen", "op"), "maximum_consecutive_wet_days": ("maxlen", "op"),
    "dry_spell_frequency": None, "dry_spell_total_length": None, "dry_spell_max_length": ("maxlen", "<"),
    "wet_spell_frequency": None, "tx90p": None, "tx10p": None, "tn90p": None,
}


class _PassBuilder:
    """Collects the outputs wanted from one (variable, freq) pass and packs them into ``_lib.MultiPlan``s
    (a pass that needs more conditions than one plan holds is split into several launches)."""

    def __init__(self):
        self.stats = {}          # name -> request key
        self.conds = {}          # (sgn, thr) -> {"n": bool, "max": wmax or None, "runs": {(kind, w)}, "ms": (w, sgn, thr0)}
        self.sums = {}           # (mode, sgn, thr, off_sgn, off) -> True

    def cond(self, op_code, thr):
        from . import device
        key = device.normalise_condition(op_code, thr)
        return self.conds.setdefault(key, {"n": False, "max": False, "runs": set(), "ms": None}), key

    def plans(self):
        """-> list of (plan, n_slots, {request key: (slot, is_int)}).  Layout of a plan (include/xclim_b200.h):
        the conditions that own run outputs come first, two output places each (a condition with more than two
        is listed again), the one with a largest-run-sum output is condition 0."""
        from . import _lib
        # units: one entry per condition place = (key, cond dict, [run outputs (<= 2)], wants n/max here?)
        places = []
        for key, c in sorted(self.conds.items(), key=lambda kv: (kv[1]["ms"] is None, -len(kv[1]["runs"]))):
            runs = sorted(c["runs"], key=lambda kw: (kw[1], kw[0]))
            chunks = [runs[i:i + 2] for i in range(0, len(runs), 2)] or [[]]
            for ci, ch in enumerate(chunks):
                places.append({"key": key, "c": c, "runs": ch, "first": ci == 0})
        sums = list(self.sums)
        out = []
        first = True
        while first or places or sums:
            plan = _lib.MultiPlan()
            plan.slot_sum = plan.slot_mean = plan.slot_min = plan.slot_max = -1
            where, n = {}, 0

            def slot(key, is_int=False):
                nonlocal n
                where[key] = (n, is_int)
                n += 1
                return n - 1
            if first:
                for st in self.stats:
                    setattr(plan, "slot_" + st, slot(("stat", st)))
            # pick the places of this launch: run-owning places first (at most MAX_RUNS / 2), a max-sum owner at 0
            take, rest = [], []
            n_run_places = 0     # a max-sum owner without runs of its own counts: it holds run place 0 (ncr += 1 below)
            have_ms = False
            for pl in places:
                owns_runs = bool(pl["runs"])
                owns_ms = pl["first"] and pl["c"]["ms"] is not None
                if len(take) >= _lib.MULTI_MAX_COND or (owns_runs and n_run_places >= _lib.MULTI_MAX_RUNS // 2) or \
                        (owns_ms and (have_ms or take)):
                    rest.append(pl)
                    continue
                if owns_ms and not owns_runs and n_run_places:      # must sit at 0: only as the first place
                    rest.append(pl)
                    continue
                take.append(pl)
                n_run_places += owns_runs or owns_ms
                have_ms = have_ms or owns_ms
            # order: max-sum owner, then run owners, then the plain ones
            take.sort(key=lambda pl: (not (pl["first"] and pl["c"]["ms"] is not None), not pl["runs"]))
            ncr = sum(1 for pl in take if pl["runs"])
            if take and take[0]["first"] and take[0]["c"]["ms"] is not None and not take[0]["runs"] and ncr:
                ncr += 1      # the max-sum owner occupies run place 0 without using it
            places = rest
            plan.n_cond = len(take)
            for j, pl in enumerate(take):
                sgn, thr = pl["key"]
                c = pl["c"]
                e = plan.cond[j]
                e.sgn, e.thr, e.wmax = sgn, thr, 1
                e.slot_n = slot(("n", sgn, thr), True) if (pl["first"] and c["n"]) else -1
                e.slot_max = slot(("max", sgn, thr)) if (pl["first"] and c["max"]) else -1
                for u in range(2):
                    if j < ncr:
                        r = plan.runs[2 * j + u]
                        r.cond, r.window, r.kind, r.slot = j, 1, 0, -1
                        if u < len(pl["runs"]):
                            kind, w = pl["runs"][u]
                            r.window, r.kind = int(w), 0 if kind == "sum" else 1
                            r.slot = slot((kind, sgn, thr, w))
                if j == 0 and pl["first"] and c["ms"] is not None:
                    w, ms_sgn, thr0 = c["ms"]
                    m = plan.msum[0]
                    m.cond, m.window, m.sgn, m.thr0 = 0, int(w), ms_sgn, thr0
                    m.slot = slot(("ms", sgn, thr, w))
                    plan.n_msum = 1
            plan.n_runs = 2 * ncr
            take_s, sums = sums[:_lib.MULTI_MAX_SUMS], sums[_lib.MULTI_MAX_SUMS:]
            plan.n_sums = len(take_s)
            for j, key in enumerate(take_s):
                mode, sgn, thr, off_sgn, off = key
                e = plan.sums[j]
                e.mode, e.sgn, e.thr, e.off_sgn, e.off = mode, sgn, thr, off_sgn, off
                e.slot = slot(("qsum",) + key)
            out.append((plan, n, where))
            first = False
        return out


def run_batch(fields, pers=None, names=None):
    """The indicators of ``BATCH_INDICATORS`` (or ``names``) over ``fields = {"tas": ..., "tasmax": ..., "tasmin":
    ..., "pr": ...}`` with one fused pass per (variable, frequency); ``pers[(variable, percentile)]`` are the
    ``percentile_doy`` tables of tx90p / tx10p / tn90p.  Returns ``{name: result}``: the same containers, dtypes,
    values and attrs as the one-call-per-indicator functions."""
    import inspect

    import numpy as np

    from . import _lib, device
    from .field import attrs_of, time_axis_of
    from .generic import _unwrap, _wrap_periods

    want = [(nm, var) for nm, var in BATCH_INDICATORS if names is None or nm in names]
    per_of = {"tx90p": ("tasmax", 90.0), "tx10p": ("tasmax", 10.0), "tn90p": ("tasmin", 90.0)}
    g = globals()
    unwrapped = {}
    passes = {}          # (var, freq) -> _PassBuilder
    todo = []            # (name, var, freq, spec, params, request keys)
    results = {}
    for nm, var in want:
        fn = g[nm]
        spec = BATCH_FUSED.get(nm)
        sig = inspect.signature(fn)
        par = {k: v.default for k, v in sig.parameters.items() if v.default is not inspect.Parameter.empty}
        if spec is None or par.get("resample_before_rl", True) is not True:
            results[nm] = fn(fields[var], pers[per_of[nm]]) if nm in per_of else fn(fields[var])
            continue
        da = fields[var]
        if var not in unwrapped:
            unwrapped[var] = _unwrap(da)
        freq = par["freq"]
        pb = passes.setdefault((var, freq), _PassBuilder())
        kind = spec[0]
        th = par.get("thresh")
        if isinstance(th, str) and th.endswith(" mm"):          # daily amounts on mm/d data (cf. dry_spell_max_length)
            th = th.replace(" mm", " mm/d")
        thr = threshold_in_units_of(th, da) if th is not None else None
        op = None
        if len(spec) > 1 and kind in ("count", "excess", "maxlen"):
            op = par["op"] if spec[1] == "op" else spec[1]
        elif "op" in par:
            op = par["op"]
        keys = None
        if kind == "stat1":       # rolling(window).sum() -> max: with the default window of 1 the rolled series IS the series
            if int(par.get("window", 1)) != 1:
                results[nm] = fn(fields[var])
                continue
            kind, spec = "stat", ("stat",) + tuple(spec[1:])
        if kind == "stat":
            pb.stats[spec[1]] = True
            keys = ("stat", spec[1])
        elif kind in ("count", "prop"):
            c, k = pb.cond(_lib.OPS[op], thr)
            c["n"] = True
            keys = ("n",) + k
        elif kind == "excess":
            sgn = 1.0 if op in (">", ">=") else -1.0
            key = (0, 0.0, 0.0, sgn, float(np.float32(thr)))
            pb.sums[key] = True
            keys = ("qsum",) + key
        elif kind == "intensity":
            c, k = pb.cond(_lib.OPS[op], thr)
            c["n"] = True
            key = (1, k[0], k[1], 0.0, 0.0)
            pb.sums[key] = True
            keys = (("qsum",) + key, ("n",) + k)
        elif kind == "spell":
            c, k = pb.cond(_lib.OPS[op], thr)
            c["runs"].add((spec[1], int(par["window"])))
            keys = (spec[1],) + k + (int(par["window"]),)
        elif kind == "maxlen":
            c, k = pb.cond(_lib.OPS[op], thr)
            c["max"] = True
            keys = ("max",) + k
        elif kind == "maxsum":
            c, k = pb.cond(_lib.OPS[">"], thr)
            c["ms"] = (int(par["window"]), 1.0, float(np.float32(thr)))
            keys = ("ms",) + k + (int(par["window"]),)
        todo.append((nm, var, freq, spec, par, keys))
    # ---- one launch (or a few) per (variable, frequency)
    slots = {}           # (var, freq, request key) -> device tensor (P, C)
    for (var, freq), pb in passes.items():
        x2d, cell_shape, other, ta = unwrapped[var]
        poff = ta.period_offsets(freq)
        for plan, n, where in pb.plans():
            buf = device.period_multi(x2d, poff, plan, n)
            for key, (sl, is_int) in where.items():
                slots[(var, freq, key)] = buf[sl].view(_torch_int32()) if is_int else buf[sl]
    # ---- wrap like the one-call-per-indicator functions
    for nm, var, freq, spec, par, keys in todo:
        da = fields[var]
        x2d, cell_shape, other, ta = unwrapped[var]
        attrs = attrs_of(da)
        kind = spec[0]
        get = lambda k: slots[(var, freq, k)]   # noqa: E731
        if kind == "stat" and BATCH_FUSED[nm][0] == "stat1":     # max_n_day_precipitation_amount: units only
            attrs["units"] = spec[2]
            results[nm] = _wrap_periods(da, get(keys), cell_shape, other, ta, freq, attrs)
        elif kind == "stat":
            from .units import to_agg_units_attrs
            attrs.update(to_agg_units_attrs(da, spec[1]))
            out = _wrap_periods(da, get(keys), cell_shape, other, ta, freq, attrs)
            results[nm] = out.assign_attrs(units=spec[2]) if spec[2] else out
        elif kind == "count":
            results[nm] = _wrap_periods(da, get(keys), cell_shape, other, ta, freq, attrs,
                                        dtype=np.int64).assign_attrs(units="d")
        elif kind == "prop":
            cnt = _wrap_periods(da, get(keys), cell_shape, other, ta, freq, attrs, dtype=np.int64).assign_attrs(units="d")
            n = np.diff(time_axis_of(da).period_offsets(freq)).reshape((-1,) + (1,) * (cnt.values.ndim - 1))
            results[nm] = _like(cnt, _ratio(cnt.values, n), units="1")
        elif kind == "excess":
            u = attrs.get("units", "")
            attrs["units"] = f"{u} d".strip()
            results[nm] = _wrap_periods(da, get(keys), cell_shape, other, ta, freq, attrs)
        elif kind == "intensity":
            s_ = _wrap_periods(da, get(keys[0]), cell_shape, other, ta, freq, attrs)
            wd = _wrap_periods(da, get(keys[1]), cell_shape, other, ta, freq, attrs, dtype=np.int64)
            results[nm] = _like(s_, _ratio(s_.values, wd.values), units="mm d-1")
        elif kind in ("spell", "maxlen"):
            attrs["units"] = "" if (kind == "spell" and spec[1] == "count") else "d"
            val = get(keys)
            if kind == "maxlen" and int(par.get("window", 1)) > 1:     # `max_l.where(max_l >= window, 0)`
                val = val * (val >= int(par["window"]))
            results[nm] = _wrap_periods(da, val, cell_shape, other, ta, freq, attrs, dtype=np.float32)
        elif kind == "maxsum":
            attrs["units"] = "K d"
            results[nm] = _wrap_periods(da, get(keys), cell_shape, other, ta, freq, attrs)
    return {nm: results[nm] for nm, _ in want}


def _torch_int32():
    import torch
    return torch.int32


def _like(template, values, units):
    from .field import Field, is_xarray
    if is_xarray(template):
        return template.copy(data=values).assign_attrs(units=units)
    return Field(values, template.dims, template.time, dict(template.coords), {**template.attrs, "units": units},
                 template.name)


# ---- end-to-end path: host-backed inputs stream through HBM in lat slabs (xclim_b200/streaming.py)
def _stream_entry_points():
    import inspect

    from .streaming import streamed
    g = globals()
    for nm, fn in list(g.items()):
        if nm.startswith("_") or not inspect.isfunction(fn) or fn.__module__ != __name__:
            continue
        g[nm] = streamed(fn)


_stream_entry_points()
