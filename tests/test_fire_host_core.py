"""The DEVICE code of the fire-weather kernel (xclim_b200/csrc/fwi_core.cuh), compiled for the host, against
the reference fixtures and the oracle.  The CUDA kernel adds only the thread-to-cell mapping to this code
(xclim_b200/csrc/fwi.cu); its run on a GPU is tests/test_zzz_gpu_fire.py."""
import os

import numpy as np
import pytest

import fwi_host_build as hb
from oracle import fire_oracle as FO
from test_fire_oracle import case_inputs, check_outputs, golden, mg  # noqa: F401


@pytest.mark.parametrize("name", list(mg.CFFWIS_CASES))
def test_host_build_of_the_kernel_matches_reference_fixture(golden, name):  # noqa: F811
    args, kw, exp = case_inputs(golden, name)
    if kw.get("season_method") is None:
        args = args[:4] + (None,) + args[5:]      # snd is not needed: the library accepts NULL
    got = hb.run(*args, **kw)
    check_outputs(got, exp, name, exact_frac=0.99)


def test_host_build_matches_oracle_on_other_parameters():
    rng = np.random.default_rng(11)
    inp = mg.cffwis_inputs(seed=5, C=16, T=500)
    tc = lambda a: np.ascontiguousarray(a.T)   # noqa: E731
    dc0, dmc0, ffmc0, wpr = mg.cffwis_state(inp, "some")
    base = (tc(inp["tas"]), tc(inp["pr"]), tc(inp["hurs"]), tc(inp["ws"]), tc(inp["snd"]), inp["mth"], inp["lat"])
    cases = [
        dict(season_method="GFWED", temp_condition_days=9, snow_condition_days=12, outputs=["FFMC", "ISI", "season_mask"]),
        dict(season_method="LA08", snow_condition_days=5, temp_condition_days=2, dry_start="CFS", outputs=["DC", "DMC", "BUI", "season_mask"]),
        dict(season_method="GFWED", dry_start="GFWED+SNOW", snow_cover_days=61, snow_min_cover_frac=0.3,
             snow_min_mean_depth=0.02, outputs=["DC", "DMC", "season_mask"]),
        dict(season_method="WF93", overwintering=True, carry_over_fraction=1.0, wetting_efficiency_fraction=0.5,
             dc_start=20, outputs=["DC", "FWI", "DSR", "winter_pr", "season_mask"]),
        dict(season_method=None, ffmc_start=70, dmc_start=10, dc_start=200, outputs=["FWI"]),
    ]
    for kw in cases:
        asked = kw.pop("outputs")
        extra = [o for o in asked if o in ("season_mask", "winter_pr")]
        exp = FO.fire_weather_calc(*base, None, dc0, dmc0, ffmc0, wpr, outputs=FO.complete_indexes(
            [o for o in asked if o not in extra]) + extra, **kw)
        got = hb.run(*base, None, dc0, dmc0, ffmc0, wpr, outputs=asked, **kw)   # the library adds what it needs
        assert set(got) == set(asked)
        check_outputs(got, {k: np.asarray(exp[k]) for k in asked}, str(kw), exact_frac=0.99)
    assert rng is not None


def test_argument_checks_of_the_library():
    inp = {k: (v[:4, :400] if getattr(v, "ndim", 0) == 2 else v[:400] if k == "mth" else v[:4]) for k, v in mg.cffwis_inputs().items()}
    tc = lambda a: np.ascontiguousarray(a.T)   # noqa: E731
    a = (tc(inp["tas"]), tc(inp["pr"]), None, None, None, inp["mth"], inp["lat"], None, None, None, None, None)
    assert set(hb.run(*a, outputs=["DC"])) == {"DC"}
    with pytest.raises(ValueError, match="hurs"):
        hb.run(*a, outputs=["DMC"])
    with pytest.raises(ValueError, match="overwintering"):
        hb.run(*a, outputs=["DC"], overwintering=True)
    with pytest.raises(ValueError, match="snd"):
        hb.run(*a, outputs=["DC"], season_method="LA08")
    with pytest.raises(ValueError, match="1..32"):
        hb.run(*a, outputs=["DC"], season_method="WF93", temp_condition_days=40)


def test_parameter_struct_layouts_agree():
    """The product's ctypes struct (xclim_b200/_lib.py) and the one the host build was driven with lay
    XcFwiParams out identically (144 bytes; the doubles 8-aligned after 17 4-byte fields)."""
    import ctypes

    from xclim_b200 import _lib
    assert ctypes.sizeof(_lib.FwiParams) == ctypes.sizeof(hb.XcFwiParams) == 144
    for (n1, _), (n2, _) in zip(_lib.FwiParams._fields_, hb.XcFwiParams._fields_):
        assert n1 == n2 and getattr(_lib.FwiParams, n1).offset == getattr(hb.XcFwiParams, n2).offset
    assert _lib.FwiParams.snow_min_cover_frac.offset == 72 and _lib.FwiParams.in_scale.offset == 104


def test_elementwise_functions_of_the_host_build(golden):  # noqa: F811
    """ISI / BUI / FWI / DSR of the stored codes reproduce the reference's own arrays; the overwintered DC its
    tests' known answers (tests/test_cffwis.py:126-145)."""
    from test_fire_oracle import assert_index_close
    g = golden
    ws = g["ws"].T
    ffmc, dmc, dc = (g[f"always_on__{k}"].T for k in ("FFMC", "DMC", "DC"))
    assert_index_close(hb.elementwise("ISI", ws, ffmc), g["always_on__ISI"].T, "ISI")
    assert_index_close(hb.elementwise("BUI", dmc, dc), g["always_on__BUI"].T, "BUI")
    assert_index_close(hb.elementwise("FWI", g["always_on__ISI"].T, g["always_on__BUI"].T), g["always_on__FWI"].T, "FWI")
    assert_index_close(hb.elementwise("DSR", g["always_on__FWI"].T), g["always_on__DSR"].T, "DSR")
    for (dcf, wpr, a, b, mn), exp in (((300, 110, 0.75, 0.75, 15), 109.4657), ((300, 110, 1.0, 0.9, 15), 16.35315),
                                      ((100, 50, 0.75, 0.75, 15), 105.176), ((1, 550, 0.75, 0.75, 10), 10)):
        got = hb.elementwise("OWDC", np.array([dcf], np.float32), np.array([wpr], np.float32), (a, b, mn))
        np.testing.assert_allclose(got, exp, rtol=1e-6)
    assert np.isnan(hb.elementwise("OWDC", np.array([np.nan], np.float32), np.array([5.0], np.float32), (0.75, 0.75, 15)))[0]
    assert hb.elementwise("BUI", np.zeros(1, np.float32), np.zeros(1, np.float32))[0] == 0


def check_against_stored_reference(golden_dir, group, exact_frac):
    """The oracle and the host build of the device code on every case of `group` (tests/golden/make_golden.py)
    against the outputs of the reference's `_fire_weather_calc` stored for it: every stored value within the
    tolerances of check_outputs, and the bit-identical share of each code, over all cases, above `exact_frac`.
    Returns the number of cases."""
    g = np.load(os.path.join(golden_dir, "ref_cffwis_modes.npz"))
    tc = lambda a: np.ascontiguousarray(a.T)   # noqa: E731
    same = {}
    n = 0
    for i, (label, inp, state, mask, outs, over) in enumerate(mg.CFFWIS_CASE_GROUPS[group]()):
        C, T = inp["tas"].shape
        exp = mg.stored_cffwis_outputs(g, group, i, outs, C, T)
        t, c = mg.sample_positions(C, T, i)
        args = (tc(inp["tas"]), tc(inp["pr"]), tc(inp["hurs"]), tc(inp["ws"]), tc(inp["snd"]), inp["mth"], inp["lat"],
                None if mask is None else tc(mask), *state)
        for who, got in (("oracle", FO.fire_weather_calc(*args, outputs=outs, **over)),
                         ("host build", hb.run(*args, outputs=outs, **over))):
            got = {o: (np.asarray(v)[t, c] if o in mg.CFFWIS_FLOAT_OUTPUTS else np.asarray(v)) for o, v in got.items()}
            check_outputs(got, exp, f"{who}:{label}", exact_frac=0.0)
            for o in ("DC", "DMC", "FFMC", "winter_pr"):
                if o in exp:
                    k = same.setdefault((who, o), [0, 0])
                    k[0] += int(((got[o] == exp[o]) | np.isnan(exp[o])).sum())
                    k[1] += exp[o].size
        n += 1
    for (who, o), (k, m) in same.items():
        assert k / m > exact_frac, f"{who}:{o}: {k} of {m} values bit-identical"
    return n


def test_every_mode_combination_against_the_reference(golden_dir):
    """All combinations of season method x overwintering x dry start x initial_start_up, each with random
    thresholds / window lengths / previous codes: the oracle AND the host build of the device code against the
    reference's `_fire_weather_calc`."""
    assert check_against_stored_reference(golden_dir, "modes", exact_frac=0.98) == 72


def test_ring_mean_rounds_as_numpy_mean():
    """The GFWED season and the snow-aware dry start compare float32 window means with thresholds
    (_cffwis.py:661-668, 746-756): np_mean_f32 must round exactly as np.mean does (pairwise summation)."""
    import ctypes
    lib = hb.load()
    lib.fwi_host_np_mean.restype = ctypes.c_float
    rng = np.random.default_rng(4)
    for n in list(range(1, 41)) + [59, 60, 61, 64, 100, 127, 128]:
        for _ in range(6):
            vals = (rng.random(n) * rng.choice([1e-3, 1.0, 1e3], size=n)).astype(np.float32)
            head = int(rng.integers(0, n))
            ring = np.empty(n, np.float32)
            ring[(head + 1 + np.arange(n)) % n] = vals            # oldest value right after the head
            got = lib.fwi_host_np_mean(ring.ctypes.data_as(ctypes.c_void_p), ctypes.c_int32(n), ctypes.c_int32(head))
            assert np.float32(got) == np.mean(vals), (n, head)


def test_branch_point_inputs_against_the_reference(golden_dir):
    """Inputs drawn from the branch points of the equations (rain thresholds 0.5 / 1.5 / 2.8 mm and just above,
    humidity 0 and 100 %, calm and storm winds, temperatures at -2.8 / -1.1 / 21.1 degC, snow depth at its
    threshold, latitudes on the band edges, previous codes at 0 / 33 / 65 / 101), with and without missing
    values: oracle and host build of the device code against the reference's `_fire_weather_calc`."""
    assert check_against_stored_reference(golden_dir, "branch", exact_frac=0.97) == 24
