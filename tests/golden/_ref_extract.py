"""Load the reference's pure numpy/numba cores WITHOUT copying them into this repo.

The reference package need not be importable (xarray, dask, pint ... may be absent), but its
numerical cores are plain numpy/numba functions.  This helper parses the reference source files
where they lie (``$XCLIM_REFERENCE_ROOT/src/xclim/...``), extracts the named top-level function
definitions with ``ast`` and ``exec``s them in a private namespace.  It is used ONLY by
``make_golden.py`` (fixture generation); the tests read the fixtures it wrote.
"""
from __future__ import annotations

import ast
import os
import warnings
from collections import namedtuple
from collections.abc import Sequence

import numpy as np

REF_ROOT = os.environ.get("XCLIM_REFERENCE_ROOT", "")

RUN_LENGTH_FUNCS = [
    "_cumsum_reset_np", "_rle_1d", "rle_1d", "first_run_1d", "statistics_run_1d",
    "windowed_run_count_1d", "windowed_run_events_1d",
]
UTILS_FUNCS = [
    "calc_perc", "nan_calc_percentiles", "_compute_virtual_index", "_get_gamma", "_get_indexes",
    "_linear_interpolation", "_nan_quantile",
]


def available() -> bool:
    return bool(REF_ROOT) and os.path.isfile(os.path.join(REF_ROOT, "src/xclim/indices/run_length.py"))


def _extract(relpath: str, names: list[str], extra_ns: dict) -> dict:
    path = os.path.join(REF_ROOT, relpath)
    with open(path) as f:
        src = f.read()
    tree = ast.parse(src)
    def _name(n):
        if isinstance(n, ast.FunctionDef):
            return n.name
        if isinstance(n, ast.Assign) and len(n.targets) == 1 and isinstance(n.targets[0], ast.Name):
            return n.targets[0].id          # module-level constant tables (e.g. DAY_LENGTHS)
        if isinstance(n, ast.AnnAssign) and isinstance(n.target, ast.Name):
            return n.target.id
        return None

    wanted = [n for n in tree.body if _name(n) in names]
    missing = set(names) - {_name(n) for n in wanted}
    if missing:
        raise RuntimeError(f"reference functions not found in {relpath}: {sorted(missing)}")
    mod = ast.Module(body=wanted, type_ignores=[])
    ns = dict(extra_ns)
    exec(compile(mod, path, "exec"), ns)  # noqa: S102 - executing the reference where it lies
    return {n: ns[n] for n in names}


def load_run_length() -> dict:
    try:
        from numba import njit
    except Exception:  # pragma: no cover
        def njit(f):
            return f

    class _XR:  # annotations only (from __future__ annotations is not in the extracted body)
        DataArray = object

    ns = {"np": np, "njit": njit, "namedtuple": namedtuple, "warn": warnings.warn,
          "Sequence": Sequence, "xr": _XR}
    return _extract("src/xclim/indices/run_length.py", RUN_LENGTH_FUNCS, ns)


def load_utils() -> dict:
    ns = {"np": np, "Sequence": Sequence}
    return _extract("src/xclim/core/utils.py", UTILS_FUNCS, ns)


CFFWIS_NAMES = [
    "default_params", "DAY_LENGTHS", "DAY_LENGTH_FACTORS", "_day_length", "_day_length_factor",
    "_fine_fuel_moisture_code", "_duff_moisture_code", "_drought_code", "initial_spread_index", "build_up_index",
    "fire_weather_index", "daily_severity_rating", "_overwintering_drought_code", "_fire_season",
    "_fire_weather_calc",
]


def load_cffwis() -> dict:
    """The numba / numpy cores of the Canadian Forest Fire Weather Index System
    (indices/fire/_cffwis.py:161-900), executed where they lie."""
    from collections import OrderedDict

    from numba import njit, vectorize

    class _XR:
        DataArray = object

    ns = {"np": np, "njit": njit, "vectorize": vectorize, "OrderedDict": OrderedDict, "xr": _XR,
          "Sequence": Sequence, "namedtuple": namedtuple}
    return _extract("src/xclim/indices/fire/_cffwis.py", CFFWIS_NAMES, ns)
