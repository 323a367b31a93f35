"""GPU parity for the 'batch of 50 atmos indicators' configuration (BASELINE.json configs[4]): every
index entry point of xclim_b200.indices.BATCH_INDICATORS against an oracle composition."""
import numpy as np
import pytest

from oracle import xclim_oracle as O
from xb_helpers import make_field

pytestmark = pytest.mark.gpu

def _inputs(shape=(4, 8)):
    rng = np.random.default_rng(61)
    T = 365 * 3
    t = np.arange(T)
    season = 14 * np.sin(2 * np.pi * (t % 365 - 110) / 365).reshape((T,) + (1,) * len(shape))
    tas = (278 + season + 4 * rng.standard_normal((T,) + shape)).astype(np.float32)
    spread = np.abs(4 + rng.standard_normal((T,) + shape)).astype(np.float32)
    tasmax = (tas + spread).astype(np.float32)
    tasmin = (tas - spread).astype(np.float32)
    pr = rng.gamma(0.4, 6.0, size=(T,) + shape).astype(np.float32)
    pr[rng.random(pr.shape) < 0.45] = 0
    for a in (tas, tasmax, tasmin, pr):
        a[rng.random(a.shape) < 0.003] = np.nan
    return {"tas": tas, "tasmax": tasmax, "tasmin": tasmin, "pr": pr}



from oracle.batch50 import oracle_indicator as _oracle  # noqa: E402


def test_batch_of_50_indicators(cuda):
    from xclim_b200 import indices
    data = _inputs()
    units = {"tas": "K", "tasmax": "K", "tasmin": "K", "pr": "mm/d"}
    fields = {k: make_field(v, "1981-01-01", calendar="noleap", units=units[k]) for k, v in data.items()}
    assert len(indices.BATCH_INDICATORS) == 50
    _check_indicators_against_oracle(data, fields)


def _check_indicators_against_oracle(data, fields):
    """Every indicator of BATCH_INDICATORS called on ``fields`` (built from the arrays ``data``) against the
    oracle compositions: integer-valued results exactly, float results to 1e-5."""
    from xclim_b200 import calendar as xcal, indices
    checked = 0
    for name, var in indices.BATCH_INDICATORS:
        da, x = fields[var], data[var]
        fn = getattr(indices, name)
        defaults = fn.__defaults__ or ()
        import inspect
        freq = inspect.signature(fn).parameters["freq"].default
        poff = da.time.period_offsets(freq)
        if name in ("tx90p", "tx10p", "tn90p"):
            per = 10.0 if name == "tx10p" else 90.0
            pdoy = xcal.select_percentile(xcal.percentile_doy(da, window=5, per=per), per)
            got = fn(da, pdoy).values
            tab = O.percentile_doy(x, da.time.year, da.time.doy, 5, per)[:, 0]
            exp = O.doy_threshold_count(x, tab, da.time.doy, poff, "<" if name == "tx10p" else ">")
        else:
            got = fn(da).values
            exp = _oracle(name, x, poff, da.time, data)
        exp = np.asarray(exp)
        assert got.shape == exp.shape, name
        if np.issubdtype(got.dtype, np.integer) or name.startswith(("cold_spell", "hot_spell_f", "hot_spell_m", "hot_spell_t",
                                                                   "heat_wave", "frost_free", "maximum_consecutive",
                                                                   "dry_spell", "wet_spell")) and name != "hot_spell_max_magnitude":
            np.testing.assert_array_equal(got, exp.astype(got.dtype), err_msg=name)       # integer-valued: exact
        else:
            np.testing.assert_allclose(got, exp, rtol=1e-5, atol=1e-6, equal_nan=True, err_msg=name)  # float: 1e-5
        checked += 1
    assert checked == 50


def test_device_outputs_option_matches_host_outputs(cuda):
    """set_options(device_outputs=True): device-resident Fields in, device-resident Fields out, the
    same values and dtypes as the host-materialised results."""
    import torch
    import xclim_b200
    from xclim_b200 import Field, indices, run_length
    data = _inputs()
    units = {"tas": "K", "tasmax": "K", "tasmin": "K", "pr": "mm/d"}
    host = {k: make_field(v, "1981-01-01", calendar="noleap", units=units[k]) for k, v in data.items()}
    dev = {k: Field(torch.from_numpy(v).cuda(), f.dims, f.time, dict(f.coords), dict(f.attrs)) for (k, v), f in
           zip(data.items(), host.values())}
    names = ["tg_mean", "wetdays", "maximum_consecutive_dry_days", "dry_spell_frequency", "growing_degree_days",
             "max_n_day_precipitation_amount", "hot_spell_max_magnitude", "cold_spell_days"]
    var_of = dict(indices.BATCH_INDICATORS)
    for name in names:
        fn = getattr(indices, name)
        ref = fn(host[var_of[name]])
        with xclim_b200.set_options(device_outputs=True):
            got = fn(dev[var_of[name]])
        assert isinstance(got, Field) and got.values.is_cuda, name
        assert got.numpy().dtype == ref.values.dtype, name
        np.testing.assert_array_equal(got.numpy(), ref.values, err_msg=name)
        assert got.attrs == ref.attrs
    # first_run with coord="dayofyear" does its index -> doy lookup on the device
    mask = host["pr"].assign_attrs()
    ref = run_length.first_run(Field((data["pr"] > 5).astype(np.float32), mask.dims, mask.time), 2, freq="YS",
                               coord="dayofyear")
    with xclim_b200.set_options(device_outputs=True):
        got = run_length.first_run(Field(torch.from_numpy((data["pr"] > 5).astype(np.float32)).cuda(), mask.dims,
                                         mask.time), 2, freq="YS", coord="dayofyear")
    np.testing.assert_array_equal(got.numpy(), ref.values)
    assert not xclim_b200.options.OPTIONS["device_outputs"]


def test_run_batch_fused_passes_match_single_calls(cuda):
    """The fused multi-output kernel behind indices.run_batch against the 50 single-output calls."""
    import test_host_layer_cpu as cpu_side
    cpu_side._check_run_batch_against_single_calls()


def test_run_batch_device_resident(cuda):
    import torch
    import xclim_b200
    from xclim_b200 import Field, calendar as xcal, indices
    data = _inputs()
    units = {"tas": "K", "tasmax": "K", "tasmin": "K", "pr": "mm/d"}
    host = {k: make_field(v, "1981-01-01", calendar="noleap", units=units[k]) for k, v in data.items()}
    dev = {k: Field(torch.from_numpy(v).cuda(), f.dims, f.time, dict(f.coords), dict(f.attrs)) for (k, v), f in
           zip(data.items(), host.values())}
    with xclim_b200.set_options(device_outputs=True):
        pers = {(var, p_): xcal.select_percentile(xcal.percentile_doy(dev[var], window=5, per=p_), p_)
                for var, p_ in (("tasmax", 90.0), ("tasmax", 10.0), ("tasmin", 90.0))}
        out = indices.run_batch(dev, pers)
    assert all(o.values.is_cuda for o in out.values())
    ref = indices.run_batch(host, {k: Field(v.numpy(), v.dims, v.time, dict(v.coords), dict(v.attrs)) for k, v in pers.items()})
    for name in out:
        np.testing.assert_array_equal(out[name].numpy(), ref[name].values, err_msg=name)
