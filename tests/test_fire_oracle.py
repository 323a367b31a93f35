"""The fire-weather oracle (oracle/fire_oracle.py) against the reference's own numba / numpy cores:
fixtures made by executing indices/fire/_cffwis.py where it lies (tests/golden/make_golden.py), the
reference tests' known answers (tests/test_cffwis.py:122-170), and the reference's step functions on a seeded
sample of their arguments (tests/golden/make_golden.py)."""
import os
import sys

import numpy as np
import pytest

from oracle import fire_oracle as FO

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import make_golden as mg  # noqa: E402


@pytest.fixture(scope="module")
def golden(golden_dir):
    return np.load(os.path.join(golden_dir, "ref_cffwis.npz"))


def case_inputs(g, name):
    """Inputs of case ``name`` of the fixture in the repo's (T, C) layout + the keyword arguments."""
    over = mg.CFFWIS_CASES[name]
    inp = {k: g[k] for k in ("tas", "pr", "hurs", "ws", "snd", "mth", "lat")}
    dc0, dmc0, ffmc0, wpr = mg.cffwis_state(inp, over.get("state"))
    mask = np.ascontiguousarray(g[over["mask_from"] + "__season_mask"].T) if "mask_from" in over else None
    kw = {k: v for k, v in over.items() if k not in ("mask_from", "state")}
    tc = lambda a: np.ascontiguousarray(a.T)   # noqa: E731  fixture arrays are (cells, time)
    args = (tc(inp["tas"]), tc(inp["pr"]), tc(inp["hurs"]), tc(inp["ws"]), tc(inp["snd"]), inp["mth"], inp["lat"], mask,
            dc0, dmc0, ffmc0, wpr)
    exp = {o: (g[f"{name}__{o}"].T if g[f"{name}__{o}"].ndim == 2 else g[f"{name}__{o}"]) for o in kw["outputs"]}
    return args, kw, exp


def eq30b_condition(fwi_out):
    """Condition number of Eq. 30b (_cffwis.py:527: fwi -> exp(2.72 (0.434 ln fwi)^0.647) for fwi > 1) at the
    OUTPUT value: d ln(out) / d ln(in) = 2.72 * 0.647 * 0.434^0.647 * (ln in)^-0.353 -- unbounded at in = 1, still 3
    at in = 1.05.  1 where the transform does not apply."""
    out = np.asarray(fwi_out, dtype=np.float64)
    with np.errstate(all="ignore"):
        ln_in = (np.log(out) / 2.72) ** (1.0 / 0.647) / 0.434
        k = 2.72 * 0.647 * 0.434 ** 0.647 * ln_in ** -0.353
    return np.where(out > 1.0, np.clip(np.nan_to_num(k, nan=1.0, posinf=200.0), 1.0, 200.0), 1.0)


def assert_index_close(got, exp, label, rtol=1e-5, atol=1e-6):
    """ISI / BUI / FWI / DSR within the 1e-5 of the north star, scaled by the condition number of the
    reference's own formula where that exceeds 1: Eq. 30b amplifies a relative difference of its float32 input
    (two correct float32 evaluations differ by an ulp or two: numpy's and glibc's already do) by up to 3 at
    FWI = 1.25 and without bound towards FWI = 1; DSR = 0.0272 FWI^1.77 multiplies it by another 1.77."""
    got, exp = np.asarray(got), np.asarray(exp)
    cond = np.ones(exp.shape)
    if label.endswith("FWI"):
        cond = np.maximum(eq30b_condition(exp), eq30b_condition(got))
    elif label.endswith("DSR"):
        with np.errstate(all="ignore"):
            cond = 1.77 * np.maximum(eq30b_condition((exp / 0.0272) ** (1 / 1.77)), eq30b_condition((got / 0.0272) ** (1 / 1.77)))
    assert np.array_equal(np.isnan(got), np.isnan(exp)), label
    with np.errstate(all="ignore"):
        err = np.abs(got.astype(np.float64) - exp.astype(np.float64))
        bound = atol + rtol * cond * np.abs(exp.astype(np.float64))
    bad = np.nan_to_num(err, nan=0.0) > np.nan_to_num(bound, nan=np.inf)
    assert not bad.any(), (f"{label}: {int(bad.sum())} values beyond tolerance, worst "
                           f"{float(np.nanmax(np.where(bad, err / np.maximum(np.abs(exp), 1e-30), 0))):.3g} relative")


def check_outputs(got, exp, name, exact_frac=0.995):
    for o, e in exp.items():
        if e.dtype == bool:
            np.testing.assert_array_equal(np.asarray(got[o]).astype(bool), e, err_msg=f"{name}:{o}")
        elif o in ("DC", "DMC", "FFMC", "winter_pr"):
            # float64 evaluation rounded to float32: identical but for the libm behind exp / log / pow
            np.testing.assert_allclose(got[o], e, rtol=2e-6, atol=0, equal_nan=True, err_msg=f"{name}:{o}")
            assert (got[o] == e).mean() + np.isnan(e).mean() > exact_frac, f"{name}:{o}"
        else:
            assert_index_close(got[o], e, f"{name}:{o}")


@pytest.mark.parametrize("name", list(mg.CFFWIS_CASES))
def test_oracle_matches_reference_fixture(golden, name):
    args, kw, exp = case_inputs(golden, name)
    check_outputs(FO.fire_weather_calc(*args, **kw), exp, name)


def test_reference_known_answers():
    """tests/test_cffwis.py:122-170."""
    for (dcf, wpr, a, b, mn), exp in (((300, 110, 0.75, 0.75, 15), 109.4657), ((300, 110, 1.0, 0.9, 15), 16.35315),
                                      ((100, 50, 0.75, 0.75, 15), 105.176), ((1, 550, 0.75, 0.75, 10), 10)):
        np.testing.assert_allclose(FO.overwintering_drought_code(dcf, wpr, a, b, mn), exp, rtol=1e-6)
    assert FO.build_up_index(np.float32(0), np.float32(0)) == 0
    assert FO.DAY_LENGTHS[FO.day_length_band(44), 0] == 6.5
    assert FO.DAY_LENGTH_FACTORS[FO.day_length_factor_band(44), 0] == -1.6
    with pytest.raises(ValueError):
        FO.day_length_band(91)


def test_step_functions_against_stored_reference_outputs(golden_dir):
    g = np.load(os.path.join(golden_dir, "ref_cffwis_steps.npz"))
    a, lats, mths = mg.cffwis_step_inputs()
    for li, lat in enumerate(lats):
        for mi, mth in enumerate(mths):
            s = g["sel"][li, mi]
            band = FO.day_length_band(np.full(s.size, lat))
            fb = FO.day_length_factor_band(np.full(s.size, lat))
            np.testing.assert_allclose(FO.dmc_step(a["t"][s], a["p"][s], a["h"][s], mth, band, a["d0"][s]), g["dmc"][li, mi],
                                       rtol=1e-6)     # the C library's float32 log is not correctly rounded everywhere
            np.testing.assert_allclose(FO.dc_step(a["t"][s], a["p"][s], mth, fb, a["c0"][s]), g["dc"][li, mi], rtol=1e-13)
    s = g["sel_ffmc"]
    np.testing.assert_allclose(FO.ffmc_step(a["t"][s], a["p"][s], a["w"][s], a["h"][s], a["f0"][s]), g["ffmc"], rtol=1e-12)
