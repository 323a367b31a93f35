"""GPU: the fire-weather kernel (xc_fwi_f32) through the C ABI against the reference fixtures, the oracle and
through the host layer.  Written after the GPU budget of round 2 was spent: these have NOT run on hardware
yet (hence the file name that sorts last, and the looser share of bit-identical values asked for: CUDA's logf /
exp / pow differ from glibc's by an ulp now and then, which flips a float32 rounding that the recurrences then
carry for days; every value must still agree to 2e-6); the kernel's device code is verified on the CPU as a host build
(tests/test_fire_host_core.py)."""
import numpy as np
import pytest

from oracle import fire_oracle as FO
from test_fire_oracle import case_inputs, check_outputs, golden, mg  # noqa: F401

pytestmark = pytest.mark.gpu


def run_on_device(args, kw):
    import torch

    from xclim_b200 import device
    tas, pr, hurs, ws, snd, mth, lat, mask, dc0, dmc0, ffmc0, wpr = args
    outputs = kw["outputs"]
    over = {k: v for k, v in kw.items() if k != "outputs"}
    from xclim_b200.fire import default_params
    p = {k: (v if not isinstance(v, tuple) else v[0]) for k, v in default_params.items()}
    p.update({k: v for k, v in over.items() if k in p})
    dry = over.get("dry_start")
    P = device.fwi_params(over.get("season_method"), over.get("overwintering", False), dry,
                          over.get("initial_start_up", True), **p)
    d = lambda a, dt=torch.float32: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to("cuda", dt)  # noqa: E731
    res = device.fire_weather(d(tas), d(pr), d(hurs), d(ws), d(snd), mth, lat, d(mask, torch.uint8), d(dc0), d(dmc0),
                              d(ffmc0), d(wpr), outputs, P)
    torch.cuda.synchronize()
    return {k: (v.cpu().numpy().astype(bool) if k == "season_mask" else v.cpu().numpy()) for k, v in res.items()}


def test_elementwise_kernel_on_device(cuda, golden):  # noqa: F811
    import torch

    from test_fire_oracle import assert_index_close
    from xclim_b200 import device
    g = golden
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a.T)).cuda()   # noqa: E731
    ffmc, dmc, dc = (d(g[f"always_on__{k}"]) for k in ("FFMC", "DMC", "DC"))
    assert_index_close(device.fire_elementwise("ISI", d(g["ws"]), ffmc).cpu().numpy(), g["always_on__ISI"].T, "ISI")
    assert_index_close(device.fire_elementwise("BUI", dmc, dc).cpu().numpy(), g["always_on__BUI"].T, "BUI")
    assert_index_close(device.fire_elementwise("FWI", d(g["always_on__ISI"]), d(g["always_on__BUI"])).cpu().numpy(),
                       g["always_on__FWI"].T, "FWI")
    assert_index_close(device.fire_elementwise("DSR", d(g["always_on__FWI"])).cpu().numpy(), g["always_on__DSR"].T, "DSR")
    got = device.fire_elementwise("OWDC", torch.tensor([300.0, 100.0, 1.0], device="cuda"),
                                  torch.tensor([110.0, 50.0, 550.0], device="cuda"), (0.75, 0.75, 15))
    np.testing.assert_allclose(got.cpu().numpy(), [109.4657, 105.176, 15.0], rtol=1e-6)


@pytest.mark.parametrize("name", list(mg.CFFWIS_CASES))
def test_kernel_matches_reference_fixture(cuda, golden, name):  # noqa: F811
    args, kw, exp = case_inputs(golden, name)
    got = run_on_device(args, kw)
    check_outputs(got, exp, name, exact_frac=0.90)


def test_kernel_matches_oracle_on_a_wider_grid(cuda):
    """1500 cells (several CTAs, a ragged last one), 3 years, all latitude bands."""
    rng = np.random.default_rng(21)
    base = mg.cffwis_inputs(seed=31, C=16, T=1095)
    reps = 94
    C = 16 * reps - 4
    tile = lambda a: np.ascontiguousarray(np.tile(a, (reps, 1))[:C].T)   # noqa: E731  (T, C)
    tas, pr, hurs, ws, snd = (tile(base[k]) for k in ("tas", "pr", "hurs", "ws", "snd"))
    tas = (tas + rng.normal(0, 1.5, tas.shape)).astype(np.float32)
    pr = (pr * rng.uniform(0.5, 1.5, pr.shape)).astype(np.float32)
    lat = rng.uniform(-90, 90, C)
    dc0 = rng.uniform(20, 500, C).astype(np.float32)
    dc0[::7] = np.nan
    nanv = np.full(C, np.nan, np.float32)
    for kw in (dict(season_method=None, outputs=["DC", "DMC", "FFMC", "ISI", "BUI", "FWI", "DSR"]),
               dict(season_method="GFWED", dry_start="GFWED+SNOW", snow_cover_days=45, snow_min_mean_depth=0.03,
                    outputs=["DC", "DMC", "FFMC", "ISI", "BUI", "FWI", "season_mask"]),
               dict(season_method="LA08", overwintering=True, outputs=["DC", "season_mask", "winter_pr"])):
        args = (tas, pr, hurs, ws, snd, base["mth"], lat, None, dc0, nanv, nanv, np.zeros(C, np.float32))
        exp = FO.fire_weather_calc(*args, **kw)
        got = run_on_device(args, kw)
        check_outputs(got, {k: np.asarray(v) for k, v in exp.items()}, str(kw), exact_frac=0.90)


def test_host_layer_on_device(cuda):
    from test_fire_host_layer import check_bodies
    from xclim_b200 import Field, fire
    check_bodies(fire, Field)


def test_fire_weather_streams_from_files_on_device(cuda, tmp_path):
    from test_fire_host_layer import check_streaming
    check_streaming(tmp_path)



def test_kernel_every_mode_combination_against_the_oracle(cuda):
    """All season x overwintering x dry-start x initial_start_up combinations with random parameters: the kernel
    against the oracle, which tests/test_fire_host_core.py pins to the reference on the SAME combinations
    (there, with the host build of this kernel's device code)."""
    assert kernel_against_the_oracle(mg.cffwis_mode_cases()) == 72


def test_kernel_branch_point_inputs_against_the_oracle(cuda):
    """The branch-point inputs of tests/test_fire_host_core.py::test_branch_point_inputs_against_the_reference
    (there: oracle and host build against the reference), here the kernel against the oracle."""
    assert kernel_against_the_oracle(mg.cffwis_branch_cases()) == 24


def kernel_against_the_oracle(cases):
    tc = lambda a: np.ascontiguousarray(a.T)   # noqa: E731
    n = 0
    for label, inp, state, mask, outs, over in cases:
        args = (tc(inp["tas"]), tc(inp["pr"]), tc(inp["hurs"]), tc(inp["ws"]), tc(inp["snd"]), inp["mth"], inp["lat"],
                None if mask is None else tc(mask), *state)
        exp = FO.fire_weather_calc(*args, outputs=outs, **over)
        got = run_on_device(args, dict(outputs=outs, **over))
        check_outputs(got, {k: np.asarray(v) for k, v in exp.items()}, label, exact_frac=0.90)
        n += 1
    return n
