"""TEST INFRASTRUCTURE -- CPU restatement of the Canadian Forest Fire Weather Index System recurrences.

SURVEY.md section 8(f).4: "the FWI numba recurrences (fire/_cffwis.py:245-560) -- same per-cell streaming
shape, different math".  This module restates, in numpy on the repo's ``(time, cell)`` layout, what the
reference computes with numba ufuncs inside a Python loop over days (file:line relative to
``/root/reference/src/xclim/indices/fire/_cffwis.py``):

* the three moisture codes over one day: FFMC ``246-319``, DMC ``322-393``, DC ``396-446`` (Van Wagner 1987
  equations, cffdrs revisions), day-length tables ``196-242``;
* the derived indices ISI ``449-469``, BUI ``472-501``, FWI ``504-528``, DSR ``531-546``;
* the overwintered drought code ``549-583``;
* the fire-season masks ``590-677`` (WF93 / LA08 / GFWED);
* the day loop with its start-up / shut-down / overwintering / dry-start state machine ``680-873``.

Only ``tests/``, ``__graft_entry__.smoke()`` and the CPU legs of ``bench.py`` may import it.  It is pinned
against the reference's own functions executed where they lie (``tests/golden/ref_cffwis.npz``, made by
``tests/golden/make_golden.py``) in ``tests/test_fire_oracle.py``.

Arithmetic, as the reference does it for float32 inputs: the three codes are evaluated in float64 from the
float32 inputs and stored (and carried to the next day) as float32; ISI / BUI / FWI / DSR are float32 numpy
expressions of the stored codes.
"""
from __future__ import annotations

import numpy as np

# GFWED day-length tables (_cffwis.py:186-205): rows = latitude bands, columns = months
DAY_LENGTHS = np.array([
    [11.5, 10.5, 9.2, 7.9, 6.8, 6.2, 6.5, 7.4, 8.7, 10, 11.2, 11.8],
    [10.1, 9.6, 9.1, 8.5, 8.1, 7.8, 7.9, 8.3, 8.9, 9.4, 9.9, 10.2],
    12 * [9],
    [7.9, 8.4, 8.9, 9.5, 9.9, 10.2, 10.1, 9.7, 9.1, 8.6, 8.1, 7.8],
    [6.5, 7.5, 9, 12.8, 13.9, 13.9, 12.4, 10.9, 9.4, 8, 7, 6],
])
DAY_LENGTH_FACTORS = np.array([
    [6.4, 5.0, 2.4, 0.4, -1.6, -1.6, -1.6, -1.6, -1.6, 0.9, 3.8, 5.8],
    12 * [1.39],
    [-1.6, -1.6, -1.6, 0.9, 3.8, 5.8, 6.4, 5.0, 2.4, 0.4, -1.6, -1.6],
])

#: default_params of the reference (_cffwis.py:161-178), magnitudes only
DEFAULTS = dict(temp_start_thresh=12.0, temp_end_thresh=5.0, snow_thresh=0.01, temp_condition_days=3,
                snow_condition_days=3, carry_over_fraction=0.75, wetting_efficiency_fraction=0.75, dc_start=15,
                dmc_start=6, ffmc_start=85, prec_thresh=1.0, dc_dry_factor=5, dmc_dry_factor=2, snow_cover_days=60,
                snow_min_cover_frac=0.75, snow_min_mean_depth=0.1)


def day_length_band(lat):
    """Row of DAY_LENGTHS for each latitude (207-224)."""
    lat = np.asarray(lat, dtype=np.float64)
    if np.any((lat > 90) | (lat < -90)):
        raise ValueError("Invalid lat specified.")
    return np.select([lat < -30, lat < -15, lat < 15, lat < 30], [0, 1, 2, 3], 4)


def day_length_factor_band(lat):
    """Row of DAY_LENGTH_FACTORS for each latitude (227-242)."""
    lat = np.asarray(lat, dtype=np.float64)
    if np.any((lat > 90) | (lat < -90)):
        raise ValueError("Invalid lat specified.")
    return np.select([lat < -15, lat < 15], [0, 1], 2)


def _pmax(a, b):
    """Python / numba ``max(a, b)``: ``b`` only when ``b > a`` (a NaN ``a`` stays)."""
    return np.where(b > a, b, a)


def _pmin(a, b):
    return np.where(b < a, b, a)


def ffmc_step(t, p, w, h, f0):
    """Fine fuel moisture code after one day (246-319).  numba types ``np.sqrt(w)`` by its float32
    argument: the square root of the wind speed is a float32 operation, everything else float64."""
    root_w = np.sqrt(np.asarray(w, dtype=np.float32)).astype(np.float64)
    t, p, w, h, f0 = (np.asarray(v, dtype=np.float64) for v in (t, p, w, h, f0))
    with np.errstate(all="ignore"):
        mo = (147.2 * (101.0 - f0)) / (59.5 + f0)
        rf = p - 0.5
        gain = 42.5 * rf * np.exp(-100.0 / (251.0 - mo)) * (1.0 - np.exp(-6.93 / rf))
        wet_hi = (mo + gain) + (0.0015 * (mo - 150.0) ** 2) * np.sqrt(rf)
        wet = np.where(mo > 150.0, wet_hi, np.where(mo <= 150.0, mo + gain, mo))
        mo = np.where(p > 0.5, _pmin(wet, 250.0), mo)
        dry_term = 0.18 * (21.1 - t) * (1.0 - 1.0 / np.exp(0.115 * h))
        ed = 0.942 * h ** 0.679 + 11.0 * np.exp((h - 100.0) / 10.0) + dry_term
        ew = 0.618 * h ** 0.753 + 10.0 * np.exp((h - 100.0) / 10.0) + dry_term
        rate = 0.581 * np.exp(0.0365 * t)
        x = (100.0 - h) / 100.0
        kw_wet = (0.424 * (1.0 - x ** 1.7) + (0.0694 * root_w) * (1.0 - x ** 8)) * rate
        y = h / 100.0
        kw_dry = (0.424 * (1.0 - y ** 1.7) + (0.0694 * root_w) * (1.0 - y ** 8)) * rate
        m_below = np.where(mo < ew, ew - (ew - mo) / 10.0 ** kw_wet, mo)
        m_above = ed + (mo - ed) / 10.0 ** kw_dry
        m = np.where(mo < ed, m_below, np.where(mo == ed, mo, m_above))
        ffmc = (59.5 * (250.0 - m)) / (147.2 + m)
        ffmc = np.where(ffmc > 101.0, 101.0, np.where(ffmc <= 0.0, 0.0, ffmc))
    return ffmc


def dmc_step(t, p, h, mth, lat_band, d0):
    """Duff moisture code after one day (322-393).  ``lat_band`` = :func:`day_length_band` of the cells.
    ``np.log(dmc0)`` is a float32 operation under numba (float32 argument), everything else float64.  numba calls
    the C library's ``logf``, which rounds (all but) correctly.  numpy's own SIMD float32 log does not: on an
    AVX-512 host it is off by up to 3 ulp for about 4 % of arguments, and the rain branch (Eq. 15) amplifies that far
    beyond a float32 ulp of the code.  The float64 log rounded to float32 is the correctly rounded float32 log on
    every host."""
    with np.errstate(all="ignore"):
        log_d0 = np.log(np.asarray(d0, dtype=np.float32).astype(np.float64)).astype(np.float32).astype(np.float64)
    t, p, h, d0 = (np.asarray(v, dtype=np.float64) for v in (t, p, h, d0))
    dl = DAY_LENGTHS[lat_band, int(mth) - 1]
    with np.errstate(all="ignore"):
        rk = np.where(t < -1.1, 0.0, 1.894 * (t + 1.1) * (100.0 - h) * dl * 0.0001)
        rw = 0.92 * p - 1.27
        wmi = 20.0 + 280.0 / np.exp(0.023 * d0)
        b = np.where(d0 <= 33.0, 100.0 / (0.5 + 0.3 * d0),
                     np.where(d0 <= 65.0, 14.0 - 1.3 * log_d0, 6.2 * log_d0 - 17.2))
        wmr = wmi + (1000 * rw) / (48.77 + b * rw)
        after_rain = 43.43 * (5.6348 - np.log(wmr - 20.0))
        pr_ = np.where(p > 1.5, after_rain, d0)
        pr_ = _pmax(pr_, 0.0)
        dmc = _pmax(pr_ + rk, 0.0)
    return np.where(np.isnan(d0), np.nan, dmc)


def dc_step(t, p, mth, fac_band, c0):
    """Drought code after one day (396-446).  ``fac_band`` = :func:`day_length_factor_band` of the cells."""
    t, p, c0 = (np.asarray(v, dtype=np.float64) for v in (t, p, c0))
    fl = DAY_LENGTH_FACTORS[fac_band, int(mth) - 1]
    with np.errstate(all="ignore"):
        t = _pmax(t, -2.8)
        pe = _pmax((0.36 * (t + 2.8) + fl) / 2, 0.0)
        rw = 0.83 * p - 1.27
        smi = 800.0 * np.exp(-c0 / 400.0)
        dr = c0 - 400.0 * np.log(1.0 + ((3.937 * rw) / smi))
        rained = np.where(dr > 0.0, dr + pe, np.where(np.isnan(c0), np.nan, pe))
    return np.where(p > 2.8, rained, c0 + pe)


def initial_spread_index(ws, ffmc):
    """ISI (449-469) in the arithmetic of its float32 inputs."""
    with np.errstate(all="ignore"):
        mo = 147.2 * (101.0 - ffmc) / (59.5 + ffmc)
        ff = 19.1152 * np.exp(mo * -0.1386) * (1.0 + (mo ** 5.31) / 49300000.0)
        return ff * np.exp(0.05039 * ws)


def build_up_index(dmc, dc):
    """BUI (472-501)."""
    with np.errstate(all="ignore"):
        both0 = (dmc == 0) & (dc == 0)
        denom = np.where(both0, np.nan, dmc + 0.4 * dc)
        low = (0.8 * dc * dmc) / denom
        high = dmc - (1.0 - 0.8 * dc / denom) * (0.92 + (0.0114 * dmc) ** 1.7)
        bui = np.where(both0, 0, np.where(dmc <= 0.4 * dc, low, high))
        return np.clip(bui, 0, None)


def fire_weather_index(isi, bui):
    """FWI (504-528)."""
    with np.errstate(all="ignore"):
        fwi = np.where(bui <= 80.0, 0.1 * isi * (0.626 * bui ** 0.809 + 2.0),
                       0.1 * isi * (1000.0 / (25.0 + 108.64 / np.exp(0.023 * bui))))
        big = fwi > 1
        fwi = np.array(fwi)
        fwi[big] = np.exp(2.72 * (0.434 * np.log(fwi[big])) ** 0.647)
        return fwi


def daily_severity_rating(fwi):
    """DSR (531-546)."""
    with np.errstate(all="ignore"):
        return 0.0272 * fwi ** 1.77


def overwintering_drought_code(last_dc, winter_pr, carry_over_fraction=0.75, wetting_efficiency_fraction=0.75,
                               min_dc=15):
    """Season-starting drought code (549-583); NaN when an input is."""
    last_dc = np.asarray(last_dc, dtype=np.float64)
    winter_pr = np.asarray(winter_pr, dtype=np.float64)
    with np.errstate(all="ignore"):
        qf = 800 * np.exp(-last_dc / 400)
        qs = carry_over_fraction * qf + wetting_efficiency_fraction * (3.94 * winter_pr)
        dcs = _pmax(400 * np.log(800 / qs), float(min_dc))
    return np.where(np.isnan(last_dc) | np.isnan(winter_pr), np.nan, dcs)


def fire_season(tas, snd=None, method="WF93", temp_start_thresh=12.0, temp_end_thresh=5.0, temp_condition_days=3,
                snow_condition_days=3, snow_thresh=0.01):
    """Active-season mask ``(T, C)`` bool (590-677).  ``tas`` degC, ``snd`` m, both ``(T, C)``."""
    T = tas.shape[0]
    mask = np.zeros(tas.shape, dtype=bool)
    if method == "WF93":
        first = temp_condition_days + 1
    elif method in ("LA08", "GFWED"):
        first = max(temp_condition_days, snow_condition_days)
    else:
        raise ValueError("`method` must be one of 'WF93', 'LA08' or 'GFWED'.")
    nt, ns = temp_condition_days, snow_condition_days
    with np.errstate(all="ignore"):
        for it in range(first, T):
            if method == "WF93":                      # the nt days BEFORE today
                win = tas[it - nt:it]
                up = np.all(win > temp_start_thresh, axis=0)
                down = np.all(win < temp_end_thresh, axis=0)
            elif method == "LA08":                    # windows that END today
                up = np.all(snd[it - ns + 1:it + 1] <= snow_thresh, axis=0)
                down = (snd[it] > snow_thresh) | np.all(tas[it - nt + 1:it + 1] < temp_end_thresh, axis=0)
            else:                                     # GFWED: window means (float32 pairwise sums, as numpy)
                msnow = np.mean(np.ascontiguousarray(snd[it - ns + 1:it + 1].T), axis=-1)
                mtemp = np.mean(np.ascontiguousarray(tas[it - nt + 1:it + 1].T), axis=-1)
                up = (mtemp > temp_start_thresh) & (msnow < snow_thresh)
                down = (msnow >= snow_thresh) | (mtemp < temp_end_thresh)
            mask[it] = (mask[it - 1] | up) & ~down
    return mask


_ORDER = ["DC", "DMC", "FFMC", "ISI", "BUI", "FWI", "DSR"]


def complete_indexes(indexes=None):
    """The index list ``fire_weather_ufunc`` works with (:1046-1057): every index an asked one depends on is
    added, in the fixed order DC, DMC, FFMC, ISI, BUI, FWI, DSR."""
    want = set(indexes or _ORDER)
    for idx, needs in (("DSR", {"FWI"}), ("FWI", {"ISI", "BUI"}), ("BUI", {"DC", "DMC"}), ("ISI", {"FFMC"})):
        if idx in want:
            want |= needs
    return sorted(want, key=_ORDER.index)


def fire_weather_calc(tas, pr, hurs, ws, snd, mth, lat, season_mask, dc0, dmc0, ffmc0, winter_pr, *, outputs,
                      season_method=None, overwintering=False, dry_start=None, initial_start_up=True, **params):
    """The day loop (680-873) on ``(T, C)`` float32 series; per-cell ``lat`` and previous codes ``(C,)``.

    Returns a dict name -> array for every name in ``outputs`` (codes / indices ``(T, C)`` float32,
    ``season_mask`` ``(T, C)`` bool, ``winter_pr`` ``(C,)``).
    """
    P = dict(DEFAULTS)
    P.update(params)
    T, C = tas.shape
    f32 = np.float32
    codes = [k for k in ("DC", "DMC", "FFMC") if k in outputs]
    prev = {"DC": np.array(dc0, dtype=f32), "DMC": np.array(dmc0, dtype=f32), "FFMC": np.array(ffmc0, dtype=f32)}
    always_on = season_method is None
    if always_on:
        mask = np.ones((T, C), dtype=bool)
        for k, start in (("DC", "dc_start"), ("DMC", "dmc_start"), ("FFMC", "ffmc_start")):
            prev[k][np.isnan(prev[k])] = P[start]
    elif season_method == "mask":
        mask = np.asarray(season_mask, dtype=bool)
    else:
        mask = fire_season(tas, snd, season_method, P["temp_start_thresh"], P["temp_end_thresh"],
                           P["temp_condition_days"], P["snow_condition_days"], P["snow_thresh"])
    out = {}
    for name in outputs:
        if name == "winter_pr":
            out[name] = np.array(winter_pr, dtype=f32)
        elif name == "season_mask":
            out[name] = mask
        else:
            out[name] = np.full((T, C), np.nan, dtype=f32)
    band = day_length_band(lat)
    fband = day_length_factor_band(lat)
    saved_dc = np.array(dc0, dtype=f32)            # last season's DC / the dry-start accumulators
    saved_dmc = np.array(dmc0, dtype=f32)
    if overwintering and "DC" in codes:
        prev["DC"] = np.full(C, np.nan, dtype=f32)
    snow_mode = bool(dry_start) and "SNOW" in dry_start
    gfwed_mode = bool(dry_start) and "GFWED" in dry_start
    if dry_start:
        if not overwintering:
            saved_dc = np.where(np.isnan(saved_dc), f32(P["dc_start"]), saved_dc).astype(f32)
        saved_dmc = np.where(np.isnan(saved_dmc), f32(P["dmc_start"]), saved_dmc).astype(f32)
        wet_start = np.zeros(C, dtype=bool)
    m_int = mask.astype(np.int16)
    for it in range(T):
        if not always_on:
            if it == 0:
                delta = m_int[0] if initial_start_up else np.zeros(C, np.int16)
            else:
                delta = m_int[it] - m_int[it - 1]
            closing = delta == -1
            opening = delta == 1
            off = (delta == 0) & (m_int[it] == 0)
            if dry_start:
                with np.errstate(invalid="ignore"):
                    rainy = pr[it] > P["prec_thresh"]
                nsc = P["snow_cover_days"]
                if snow_mode and it >= nsc:
                    hist = np.ascontiguousarray(snd[it - nsc + 1:it + 1].T)          # (C, nsc)
                    with np.errstate(invalid="ignore"):
                        covered = np.count_nonzero(hist > P["snow_thresh"], axis=-1)
                        wet_start = opening & (covered / nsc >= P["snow_min_cover_frac"]) & \
                            (hist.mean(axis=-1) >= P["snow_min_mean_depth"])
            if "DC" in codes:
                if overwintering:
                    saved_dc[closing] = prev["DC"][closing]
                    wp = out["winter_pr"]
                    wp[closing] = pr[it][closing]
                    wp[off] = wp[off] + pr[it][off]
                    last = saved_dc[opening]
                    prev["DC"][opening] = np.where(
                        np.isnan(last), P["dc_start"],
                        overwintering_drought_code(last, wp[opening], P["carry_over_fraction"],
                                                   P["wetting_efficiency_fraction"], P["dc_start"]))
                    saved_dc[opening] = np.nan
                    wp[opening] = np.nan
                elif dry_start:
                    saved_dc[closing] = P["dc_start"]
                    if gfwed_mode:
                        idle = opening | off
                        saved_dc[idle & rainy] = 0
                        saved_dc[idle & ~rainy] = saved_dc[idle & ~rainy] + f32(P["dc_dry_factor"])
                    else:
                        saved_dc[off & rainy] = P["dc_start"]
                        saved_dc[off & ~rainy] = saved_dc[off & ~rainy] + f32(P["dc_dry_factor"])
                    if snow_mode:
                        saved_dc[wet_start] = P["dc_start"]
                    prev["DC"][opening] = saved_dc[opening]
                    saved_dc[opening] = np.nan
                else:
                    prev["DC"][opening] = P["dc_start"]
                prev["DC"][closing] = np.nan
            if "DMC" in codes:
                if dry_start:
                    saved_dmc[closing] = P["dmc_start"]
                    if gfwed_mode:
                        idle = opening | off
                        saved_dmc[idle & rainy] = 0
                        saved_dmc[idle & ~rainy] = saved_dmc[idle & ~rainy] + f32(P["dmc_dry_factor"])
                    else:
                        saved_dmc[off & rainy] = P["dmc_start"]
                        saved_dmc[off & ~rainy] = saved_dmc[off & ~rainy] + f32(P["dmc_dry_factor"])
                    if snow_mode:
                        saved_dmc[wet_start] = P["dmc_start"]
                    prev["DMC"][opening] = saved_dmc[opening]
                    saved_dmc[opening] = np.nan
                else:
                    prev["DMC"][opening] = P["dmc_start"]
                prev["DMC"][closing] = np.nan
            if "FFMC" in codes:
                prev["FFMC"][opening] = P["ffmc_start"]
                prev["FFMC"][closing] = np.nan
        if "DC" in outputs:
            out["DC"][it] = dc_step(tas[it], pr[it], mth[it], fband, prev["DC"])
        if "DMC" in outputs:
            out["DMC"][it] = dmc_step(tas[it], pr[it], hurs[it], mth[it], band, prev["DMC"])
        if "FFMC" in outputs:
            out["FFMC"][it] = ffmc_step(tas[it], pr[it], ws[it], hurs[it], prev["FFMC"])
        if "ISI" in outputs:
            out["ISI"][it] = initial_spread_index(ws[it], out["FFMC"][it])
        if "BUI" in outputs:
            out["BUI"][it] = build_up_index(out["DMC"][it], out["DC"][it])
        if "FWI" in outputs:
            out["FWI"][it] = fire_weather_index(out["ISI"][it], out["BUI"][it])
        if "DSR" in outputs:
            out["DSR"][it] = daily_severity_rating(out["FWI"][it])
        for k in codes:
            prev[k] = out[k][it].copy()
    return out
