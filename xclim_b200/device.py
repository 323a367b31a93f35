"""Thin device layer: torch tensors for HBM buffers + ctypes calls into ``libxclim_b200.so``.

PyTorch is plumbing here (device memory, streams, pinned host staging); every computation is one
of the hand-written kernels behind the C ABI.  All functions take/return CUDA tensors laid out as
``(time, cell)`` float32 row-major -- the flattened view of the reference's ``(time, lat, lon)``.
"""
from __future__ import annotations

import warnings

import numpy as np
import torch

from . import _lib
from ._lib import check, load


def _require_cuda():
    if not torch.cuda.is_available():
        raise _lib.XclimB200Error("xclim_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")


def current_stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t) -> int | None:
    return None if t is None else t.data_ptr()


# ---------------------------------------------------------------------------------------- staging
def to_time_cell(values, time_axis: int, device=None):
    """Unwrap an array to a contiguous ``(T, C)`` float32 CUDA tensor.

    Returns ``(x2d, cell_shape)``.  numpy inputs are staged through pinned host memory; CUDA
    tensors already in ``(time, ...)`` float32 contiguous layout are used in place (zero copy).
    """
    _require_cuda()
    if isinstance(values, torch.Tensor):
        t = values
        if time_axis != 0:
            t = t.movedim(time_axis, 0)
        if t.dtype != torch.float32:
            t = t.to(torch.float32)
        if not t.is_cuda:
            t = t.contiguous().pin_memory().to(device or "cuda", non_blocking=True)
        t = t.contiguous()
    else:
        a = np.asarray(values)
        if time_axis != 0:
            a = np.moveaxis(a, time_axis, 0)
        if a.dtype != np.float32:
            if a.dtype.kind == "f":
                warnings.warn(f"xclim_b200 computes in float32: casting input from {a.dtype}", stacklevel=3)
            a = a.astype(np.float32)
        a = np.ascontiguousarray(a)
        h = torch.from_numpy(a)
        try:
            h = h.pin_memory()
        except RuntimeError:  # pragma: no cover - pinning can fail for huge buffers
            pass
        t = h.to(device or "cuda", non_blocking=True)
    cell_shape = tuple(t.shape[1:])
    return t.reshape(t.shape[0], -1), cell_shape


_small_cache: dict = {}


def dev_ints(arr, dtype, device) -> torch.Tensor:
    """Small integer index arrays (period offsets, doy index) cached per device."""
    a = np.ascontiguousarray(np.asarray(arr, dtype=dtype))
    key = (str(device), a.dtype.str, a.tobytes())
    t = _small_cache.get(key)
    if t is None:
        if len(_small_cache) > 256:
            _small_cache.clear()
        t = torch.from_numpy(a).to(device)
        _small_cache[key] = t
    return t


# ---------------------------------------------------------------------------------------- kernels
def period_count(x2d, poff, op_code, thr, cmp_f64=False, want_valid=False):
    T, C = x2d.shape
    P = len(poff) - 1
    poff_d = dev_ints(poff, np.int32, x2d.device)
    out = torch.empty((P, C), dtype=torch.int32, device=x2d.device)
    valid = torch.empty((P, C), dtype=torch.int32, device=x2d.device) if want_valid else None
    check(load().xc_period_count_f32(x2d.data_ptr(), T, C, x2d.stride(0), poff_d.data_ptr(), P, op_code,
                                     float(thr), int(bool(cmp_f64)), out.data_ptr(), _ptr(valid),
                                     current_stream_ptr()))
    return out, valid


def period_count_arr(x2d, poff, op_code, thr2d, per_time):
    """Counts against an array threshold: ``thr2d`` float64 ``(T, C)`` (per_time) or ``(1, C)`` (per cell)."""
    T, C = x2d.shape
    P = len(poff) - 1
    assert thr2d.dtype == torch.float64 and thr2d.is_contiguous() and thr2d.shape[-1] == C
    poff_d = dev_ints(poff, np.int32, x2d.device)
    out = torch.empty((P, C), dtype=torch.int32, device=x2d.device)
    check(load().xc_period_count_arr_f32(x2d.data_ptr(), T, C, x2d.stride(0), poff_d.data_ptr(), P, op_code,
                                         thr2d.data_ptr(), C if per_time else 0, out.data_ptr(), current_stream_ptr()))
    return out


def period_runstat(x2d, poff, op_code, thr, reducer_code, window, resample_before_rl=True, cmp_f64=False,
                   want_valid=False):
    T, C = x2d.shape
    P = len(poff) - 1
    poff_d = dev_ints(poff, np.int32, x2d.device)
    out = torch.empty((P, C), dtype=torch.float32, device=x2d.device)
    valid = torch.empty((P, C), dtype=torch.int32, device=x2d.device) if want_valid else None
    check(load().xc_period_runstat_f32(x2d.data_ptr(), T, C, x2d.stride(0), poff_d.data_ptr(), P, op_code,
                                       float(thr), int(bool(cmp_f64)), reducer_code, int(window),
                                       int(bool(resample_before_rl)), out.data_ptr(), _ptr(valid),
                                       current_stream_ptr()))
    return out, valid


def period_reduce(x2d, poff, stat_code, transform=0, op_code=0, thr=0.0, want_valid=False):
    T, C = x2d.shape
    P = len(poff) - 1
    poff_d = dev_ints(poff, np.int32, x2d.device)
    out = torch.empty((P, C), dtype=torch.float32, device=x2d.device)
    valid = torch.empty((P, C), dtype=torch.int32, device=x2d.device) if want_valid else None
    check(load().xc_period_reduce_f32(x2d.data_ptr(), T, C, x2d.stride(0), poff_d.data_ptr(), P, stat_code,
                                      transform, op_code, float(thr), out.data_ptr(), _ptr(valid),
                                      current_stream_ptr()))
    return out, valid


def synth(T, C, kind, seed, cell_offset=0, cells_per_lat=1440, n_lat_global=721, year_len=365, device="cuda"):
    """Synthetic (T, C) float32 input generated in HBM (kind 0 = pr mm/d, 1 = tasmax K)."""
    _require_cuda()
    out = torch.empty((T, C), dtype=torch.float32, device=device)
    check(load().xc_synth_f32(out.data_ptr(), T, C, C, cell_offset, cells_per_lat, n_lat_global, year_len,
                              kind, seed, current_stream_ptr()))
    return out


# ------------------------------------------------------------------------------------ percentiles
def percentile_doy(x2d, doy_index, year_index, n_doy, n_years, window, percentiles, alpha, beta,
                   force_generic=False, vrow=None):
    """(n_per, n_doy, C) float64 table of day-of-year percentiles (core/calendar.py:448-479).
    ``vrow`` (int32[T], -1 = missing): read the value of step t from row vrow[t] (bootstrap
    replacements on calendars with leap years)."""
    T, C = x2d.shape
    per = np.ascontiguousarray(np.atleast_1d(np.asarray(percentiles, dtype=np.float64)))
    doy = np.ascontiguousarray(np.asarray(doy_index, dtype=np.int16))
    yr = np.ascontiguousarray(np.asarray(year_index, dtype=np.int16))
    assert doy.size == T and yr.size == T
    lib = load()
    ws_bytes = int(lib.xc_percentile_doy_workspace_bytes(T, C, n_doy, n_years, window, per.size))
    ws = torch.empty(max(ws_bytes, 256), dtype=torch.uint8, device=x2d.device)
    out = torch.empty((per.size, n_doy, C), dtype=torch.float64, device=x2d.device)
    if force_generic:
        for i, p in enumerate(per):
            check(lib.xc_percentile_doy_generic_f32(x2d.data_ptr(), T, C, x2d.stride(0), doy.ctypes.data,
                                                    yr.ctypes.data, n_doy, n_years, int(window), float(p),
                                                    float(alpha), float(beta), out[i].data_ptr(), ws.data_ptr(),
                                                    ws.numel(), current_stream_ptr()))
    elif vrow is not None:
        vr = np.ascontiguousarray(np.asarray(vrow, dtype=np.int32))
        assert vr.size == T
        check(lib.xc_percentile_doy_vrow_f32(x2d.data_ptr(), T, C, x2d.stride(0), doy.ctypes.data, yr.ctypes.data,
                                             vr.ctypes.data, n_doy, n_years, int(window), per.ctypes.data, per.size,
                                             float(alpha), float(beta), out.data_ptr(), ws.data_ptr(), ws.numel(),
                                             current_stream_ptr()))
    else:
        check(lib.xc_percentile_doy_f32(x2d.data_ptr(), T, C, x2d.stride(0), doy.ctypes.data, yr.ctypes.data,
                                        n_doy, n_years, int(window), per.ctypes.data, per.size, float(alpha),
                                        float(beta), out.data_ptr(), ws.data_ptr(), ws.numel(),
                                        current_stream_ptr()))
    return out


def table_cell_major(table):
    """(n_per, n_doy, C) float64 doy-major table -> (C, n_doy, n_per), the reference's
    ``(*space, dayofyear, percentiles)`` order (core/calendar.py:479-483), transposed in HBM."""
    n_per, n_doy, C = table.shape
    assert table.dtype == torch.float64 and table.is_contiguous()
    out = torch.empty((C, n_doy, n_per), dtype=torch.float64, device=table.device)
    check(load().xc_table_cell_major_f64(table.data_ptr(), n_per, n_doy, C, out.data_ptr(), current_stream_ptr()))
    return out


def transpose_f64(m):
    """(A, B) float64 -> (B, A), tiled in shared memory (the layout kernel of table_cell_major with n_per = 1)."""
    A, B = m.shape
    assert m.dtype == torch.float64 and m.is_contiguous()
    out = torch.empty((B, A), dtype=torch.float64, device=m.device)
    check(load().xc_table_cell_major_f64(m.data_ptr(), 1, A, B, out.data_ptr(), current_stream_ptr()))
    return out


def doy_interp(table2d, doy_min, doy_max):
    """core/calendar.py:690-726 on a (n_src, C) float64 device table."""
    n_src, C = table2d.shape
    out = torch.empty((doy_max - doy_min + 1, C), dtype=torch.float64, device=table2d.device)
    check(load().xc_doy_interp_f64(table2d.data_ptr(), n_src, C, doy_min, doy_max, out.data_ptr(),
                                   current_stream_ptr()))
    return out


def doy_threshold_count(x2d, poff, doy_index, table2d, op_code, want_valid=False):
    """#{t in period : float64(x[t]) op table[doy[t]-1]} (indices/_multivariate.py:1583-1590)."""
    T, C = x2d.shape
    P = len(poff) - 1
    assert table2d.dtype == torch.float64 and table2d.is_contiguous() and table2d.shape[1] == C
    doy_index = np.asarray(doy_index)
    assert int(doy_index.max()) <= table2d.shape[0] and int(doy_index.min()) >= 1
    out = torch.empty((P, C), dtype=torch.int32, device=x2d.device)
    valid = torch.empty((P, C), dtype=torch.int32, device=x2d.device) if want_valid else None
    # whole years of equal length with doy == position in the year: the year-blocked kernel
    poff = np.asarray(poff)
    L = int(poff[1] - poff[0])
    if (op_code <= 3 and C % 4 == 0 and x2d.stride(0) % 4 == 0 and x2d.data_ptr() % 16 == 0
            and np.all(np.diff(poff) == L) and L == table2d.shape[0]
            and np.array_equal(doy_index[poff[0]:poff[-1]], np.tile(np.arange(1, L + 1), P))):
        check(load().xc_doy_threshold_count_years_f32(x2d.data_ptr(), T, C, x2d.stride(0), int(poff[0]), P, L,
                                                       table2d.data_ptr(), op_code, out.data_ptr(), _ptr(valid),
                                                       current_stream_ptr()))
        return out, valid
    poff_d = dev_ints(poff, np.int32, x2d.device)
    doy_d = dev_ints(doy_index, np.int16, x2d.device)
    check(load().xc_doy_threshold_count_f32(x2d.data_ptr(), T, C, x2d.stride(0), poff_d.data_ptr(), P,
                                            doy_d.data_ptr(), table2d.data_ptr(), table2d.shape[0], op_code,
                                            out.data_ptr(), _ptr(valid), current_stream_ptr()))
    return out, valid


# ------------------------------------------------------------------------------------ host-buffer path
def period_runstat_host(x_host, poff, op_code, thr, reducer_code, window, cmp_f64=False, want_valid=True,
                        workspace=None, out_host=None, valid_host=None):
    """End-to-end call with HOST buffers (the `_host` C-ABI entry point): ``x_host`` is a (T, C)
    float32 CPU tensor (ideally pinned); slabs are streamed H2D inside the call, results land in
    host memory.  Returns ``(out_host, valid_host, workspace)`` so that buffers can be reused."""
    _require_cuda()
    assert x_host.dtype == torch.float32 and x_host.is_contiguous() and not x_host.is_cuda
    T, C = x_host.shape
    P = len(poff) - 1
    poff_h = np.ascontiguousarray(np.asarray(poff, dtype=np.int32))
    lib = load()
    need = int(lib.xc_host_stream_workspace_bytes(T, C, poff_h.ctypes.data, P))
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device="cuda")
    if out_host is None:
        out_host = torch.empty((P, C), dtype=torch.float32).pin_memory()
    if want_valid and valid_host is None:
        valid_host = torch.empty((P, C), dtype=torch.int32).pin_memory()
    # the entry point works on its own non-blocking streams: nothing queued on torch's stream may still be
    # using a block the caching allocator has just recycled into `workspace`
    torch.cuda.current_stream().synchronize()
    check(lib.xc_period_runstat_f32_host(x_host.data_ptr(), T, C, poff_h.ctypes.data, P, op_code, float(thr),
                                         int(bool(cmp_f64)), reducer_code, int(window), out_host.data_ptr(),
                                         valid_host.data_ptr() if want_valid else None, workspace.data_ptr(),
                                         workspace.numel()))
    return out_host, (valid_host if want_valid else None), workspace


def bootstrap_doy_count(x2d, base_start, n_base_years, year_len, step_period, P, window, percentile, alpha, beta,
                        op_code):
    """(P, C) float64 bootstrapped exceedance counts for the in-base periods (0 elsewhere)."""
    T, C = x2d.shape
    sp = dev_ints(step_period, np.int32, x2d.device)
    assert sp.numel() == n_base_years * year_len
    scratch = torch.empty((P, C), dtype=torch.int32, device=x2d.device)
    out = torch.empty((P, C), dtype=torch.float64, device=x2d.device)
    check(load().xc_bootstrap_doy_count_f32(x2d.data_ptr(), T, C, x2d.stride(0), int(base_start), int(n_base_years),
                                            int(year_len), sp.data_ptr(), P, int(window), float(percentile),
                                            float(alpha), float(beta), op_code, scratch.data_ptr(), out.data_ptr(),
                                            current_stream_ptr()))
    return out


# ------------------------------------------------------------------------------------ rolling / spells
def rolling_period_reduce(x2d, poff, window, window_stat_code, center, stat_code):
    T, C = x2d.shape
    P = len(poff) - 1
    poff_d = dev_ints(poff, np.int32, x2d.device)
    out = torch.empty((P, C), dtype=torch.float32, device=x2d.device)
    check(load().xc_rolling_period_reduce_f32(x2d.data_ptr(), T, C, x2d.stride(0), poff_d.data_ptr(), P, int(window),
                                              window_stat_code, int(bool(center)), stat_code, out.data_ptr(),
                                              current_stream_ptr()))
    return out


def rolling_period_reduce_sel(x2d, poff, window, window_stat_code, center, stat_code, keep):
    """rolling_period_reduce with ``select_time`` on the rolled series (labels with keep[t] == 0 dropped)."""
    T, C = x2d.shape
    P = len(poff) - 1
    poff_d = dev_ints(poff, np.int32, x2d.device)
    k = dev_ints(np.asarray(keep, dtype=np.uint8), np.uint8, x2d.device)
    out = torch.empty((P, C), dtype=torch.float32, device=x2d.device)
    check(load().xc_rolling_period_reduce_sel_f32(x2d.data_ptr(), T, C, x2d.stride(0), poff_d.data_ptr(), P,
                                                  int(window), window_stat_code, int(bool(center)), stat_code,
                                                  k.data_ptr(), out.data_ptr(), current_stream_ptr()))
    return out


def spell_runstat(x2d, poff, window, window_stat_code, op_code, thr, reducer_code, resample_before_rl=True):
    T, C = x2d.shape
    P = len(poff) - 1
    poff_d = dev_ints(poff, np.int32, x2d.device)
    out = torch.empty((P, C), dtype=torch.float32, device=x2d.device)
    check(load().xc_spell_runstat_f32(x2d.data_ptr(), T, C, x2d.stride(0), poff_d.data_ptr(), P, int(window),
                                      window_stat_code, op_code, float(thr), reducer_code,
                                      int(bool(resample_before_rl)), out.data_ptr(), current_stream_ptr()))
    return out


def spell_mask(x2d, window, window_stat_code, op_code, thr, keep=None, drop_nan_adjacent=False):
    """(T, C) float32 spell mask with ``select_time`` applied (NaN out of season), see xc_spell_mask_f32."""
    T, C = x2d.shape
    k = None if keep is None else dev_ints(np.asarray(keep, dtype=np.uint8), np.uint8, x2d.device)
    out = torch.empty((T, C), dtype=torch.float32, device=x2d.device)
    check(load().xc_spell_mask_f32(x2d.data_ptr(), T, C, x2d.stride(0), int(window), window_stat_code, op_code,
                                   float(thr), _ptr(k), int(bool(drop_nan_adjacent)), out.data_ptr(),
                                   current_stream_ptr()))
    return out


# ------------------------------------------------------------------------------------ quantile mapping
def eqm_train(ref2d, hist2d, nq, kind_code):
    T, C = ref2d.shape
    assert hist2d.shape == ref2d.shape and ref2d.stride(0) == hist2d.stride(0)
    af = torch.empty((nq, C), dtype=torch.float32, device=ref2d.device)
    hq = torch.empty((nq, C), dtype=torch.float32, device=ref2d.device)
    lib = load()
    ws = torch.empty(int(lib.xc_eqm_train_workspace_bytes(T, C, int(nq))), dtype=torch.uint8, device=ref2d.device)
    check(lib.xc_eqm_train_f32(ref2d.data_ptr(), hist2d.data_ptr(), T, C, ref2d.stride(0), int(nq), kind_code,
                               af.data_ptr(), hq.data_ptr(), ws.data_ptr(), ws.numel(), current_stream_ptr()))
    return af, hq


def eqm_adjust(sim2d, af, hq, kind_code, interp_code):
    T, C = sim2d.shape
    scen = torch.empty((T, C), dtype=torch.float32, device=sim2d.device)
    check(load().xc_eqm_adjust_f32(sim2d.data_ptr(), T, C, sim2d.stride(0), af.data_ptr(), hq.data_ptr(),
                                   af.shape[0], kind_code, interp_code, scen.data_ptr(), current_stream_ptr()))
    return scen


def period_boundary_run(x2d, poff, op_code, thr, window, last=False, cmp_f64=False):
    """Index of the first (last) run of >= window steps per period, NaN if none (run_length.py:543-740)."""
    T, C = x2d.shape
    P = len(poff) - 1
    poff_d = dev_ints(poff, np.int32, x2d.device)
    out = torch.empty((P, C), dtype=torch.float32, device=x2d.device)
    check(load().xc_period_boundary_run_f32(x2d.data_ptr(), T, C, x2d.stride(0), poff_d.data_ptr(), P, op_code,
                                            float(thr), int(bool(cmp_f64)), int(window), int(bool(last)),
                                            out.data_ptr(), current_stream_ptr()))
    return out


def period_run_maxsum(x2d, poff, op_code, thr, window, resample_before_rl=True):
    """windowed_max_run_sum of the excess over ``thr`` per period (run_length.py:491-540)."""
    T, C = x2d.shape
    P = len(poff) - 1
    poff_d = dev_ints(poff, np.int32, x2d.device)
    out = torch.empty((P, C), dtype=torch.float32, device=x2d.device)
    check(load().xc_period_run_maxsum_f32(x2d.data_ptr(), T, C, x2d.stride(0), poff_d.data_ptr(), P, op_code,
                                          float(thr), int(window), int(bool(resample_before_rl)), out.data_ptr(),
                                          current_stream_ptr()))
    return out


def period_boundary_run_range(x2d, poff, range_lo, range_hi, op_code, thr, window, last=False, negate=False,
                              cell_lo=None, cmp_f64=False):
    """First/last run confined to [range_lo[p], range_hi[p]) of every period (run_length.py:1148-1331)."""
    T, C = x2d.shape
    P = len(poff) - 1
    poff_d = dev_ints(poff, np.int32, x2d.device)
    lo_d = dev_ints(range_lo, np.int32, x2d.device)
    hi_d = dev_ints(range_hi, np.int32, x2d.device)
    out = torch.empty((P, C), dtype=torch.float32, device=x2d.device)
    check(load().xc_period_boundary_run_range_f32(x2d.data_ptr(), T, C, x2d.stride(0), poff_d.data_ptr(),
                                                  lo_d.data_ptr(), hi_d.data_ptr(), P, op_code, float(thr),
                                                  int(bool(cmp_f64)), int(bool(negate)), int(window), int(bool(last)),
                                                  _ptr(cell_lo), out.data_ptr(), current_stream_ptr()))
    return out


def period_runstat2(x1, x2, poff, op1, thr1, op2, thr2, reducer_code, window, resample_before_rl=True, var_any=False):
    """Run statistics of (x1 op1 thr1) AND|OR (x2 op2 thr2) per period (heat_wave_* family)."""
    T, C = x1.shape
    assert x2.shape == x1.shape and x1.stride(0) == x2.stride(0)
    P = len(poff) - 1
    poff_d = dev_ints(poff, np.int32, x1.device)
    out = torch.empty((P, C), dtype=torch.float32, device=x1.device)
    check(load().xc_period_runstat2_f32(x1.data_ptr(), x2.data_ptr(), T, C, x1.stride(0), poff_d.data_ptr(), P, op1,
                                        float(thr1), op2, float(thr2), int(bool(var_any)), reducer_code, int(window),
                                        int(bool(resample_before_rl)), out.data_ptr(), current_stream_ptr()))
    return out


def mask_steps(x2d, keep):
    """``select_time`` with drop=False: NaN on the steps where ``keep`` is False (a new buffer)."""
    T, C = x2d.shape
    k = dev_ints(np.asarray(keep, dtype=np.uint8), np.uint8, x2d.device)
    out = torch.empty((T, C), dtype=torch.float32, device=x2d.device)
    check(load().xc_mask_steps_f32(x2d.data_ptr(), T, C, x2d.stride(0), k.data_ptr(), out.data_ptr(),
                                   current_stream_ptr()))
    return out


def period_runstat_gap(x2d, poff, op_code, thr, reducer_code, min_gap, window=1, cmp_f64=False):
    """Run statistics per period of the mask with holes < min_gap filled (generic.spell_mask(min_gap))."""
    T, C = x2d.shape
    P = len(poff) - 1
    poff_d = dev_ints(poff, np.int32, x2d.device)
    out = torch.empty((P, C), dtype=torch.float32, device=x2d.device)
    check(load().xc_period_runstat_gap_f32(x2d.data_ptr(), T, C, x2d.stride(0), poff_d.data_ptr(), P, op_code,
                                           float(thr), int(bool(cmp_f64)), reducer_code, int(window), int(min_gap),
                                           out.data_ptr(), current_stream_ptr()))
    return out


def period_run_quantile(x2d, poff, op_code, thr, q, window, resample_before_rl=True, cmp_f64=False):
    """Linear quantile ``q`` of the run lengths >= window per period (rle_statistics reducer "qNN")."""
    T, C = x2d.shape
    P = len(poff) - 1
    poff_h = np.ascontiguousarray(np.asarray(poff, dtype=np.int32))
    poff_d = dev_ints(poff_h, np.int32, x2d.device)
    out = torch.empty((P, C), dtype=torch.float32, device=x2d.device)
    check(load().xc_period_run_quantile_f32(x2d.data_ptr(), T, C, x2d.stride(0), poff_d.data_ptr(),
                                            poff_h.ctypes.data, P, op_code, float(thr), int(bool(cmp_f64)), float(q),
                                            int(window), int(bool(resample_before_rl)), out.data_ptr(),
                                            current_stream_ptr()))
    return out


# ------------------------------------------------------------------------------------ fused multi-output pass
def normalise_condition(op_code, thr):
    """(sgn, thr') with  x op thr  <=>  sgn * x > thr'  for every float32 x (NaN: False on both sides).
    ``thr`` is compared in float32 (numpy >= 2 weak-scalar rule, indices/generic.py:301-326).
    ``x >= -inf`` and ``x <= inf`` (true for every x but NaN) have no such form and are refused."""
    t = np.float32(thr)
    gt, lt, ge, le = _lib.OPS[">"], _lib.OPS["<"], _lib.OPS[">="], _lib.OPS["<="]
    if (op_code == ge and t == -np.inf) or (op_code == le and t == np.inf):
        raise NotImplementedError("the fused pass cannot express `x >= -inf` or `x <= inf`")
    if op_code == gt:
        return 1.0, float(t)
    if op_code == lt:
        return -1.0, float(-t)
    if op_code == ge:                      # x >= t  <=>  x > pred(t)
        return 1.0, float(np.nextafter(t, np.float32(-np.inf)))
    if op_code == le:                      # x <= t  <=>  -x >= -t  <=>  -x > pred(-t)
        return -1.0, float(np.nextafter(np.float32(-t), np.float32(-np.inf)))
    raise NotImplementedError("the fused pass takes the operators >, >=, <, <=")


def period_multi(x2d, poff, plan, n_slots):
    """One streaming pass producing every output of ``plan`` (a ``_lib.MultiPlan``); returns the
    ``(n_slots, P, C)`` float32 slot buffer (count slots hold int32 bits: view them with ``.view(torch.int32)``)."""
    import ctypes
    T, C = x2d.shape
    P = len(poff) - 1
    poff_d = dev_ints(poff, np.int32, x2d.device)
    out = torch.empty((max(1, n_slots), P, C), dtype=torch.float32, device=x2d.device)
    check(load().xc_period_multi_f32(x2d.data_ptr(), T, C, x2d.stride(0), poff_d.data_ptr(), P, ctypes.byref(plan),
                                     out.data_ptr(), int(n_slots), current_stream_ptr()))
    return out


# ------------------------------------------------------------------------------------ fire weather
FWI_OUTPUTS = ("DC", "DMC", "FFMC", "ISI", "BUI", "FWI", "DSR")


def fwi_params(season_method=None, overwintering=False, dry_start=None, initial_start_up=True, in_affine=None, **p):
    """``_lib.FwiParams`` from the keyword parameters of ``fire_weather_ufunc`` (indices/fire/_cffwis.py:161-178:
    thresholds compare in float32 with the float32 data, as numpy does for Python scalars)."""
    P = _lib.FwiParams()
    P.season_mode = _lib.FWI_SEASONS[season_method]
    P.dry_start = _lib.FWI_DRY_STARTS[dry_start]
    P.overwintering, P.initial_start_up = int(bool(overwintering)), int(bool(initial_start_up))
    for k in ("temp_condition_days", "snow_condition_days", "snow_cover_days"):
        setattr(P, k, int(p[k]))
    for k in ("temp_start_thresh", "temp_end_thresh", "snow_thresh", "prec_thresh", "snow_min_mean_depth", "dc_start",
              "dmc_start", "ffmc_start", "dc_dry_factor", "dmc_dry_factor", "snow_min_cover_frac", "carry_over_fraction",
              "wetting_efficiency_fraction"):
        setattr(P, k, float(p[k]))
    P.min_dc = float(p["dc_start"])
    for i, (scale, offset) in enumerate(in_affine or [(1.0, 0.0)] * 5):   # tas, pr, hurs, ws, snd
        P.in_scale[i], P.in_offset[i] = scale, offset
    return P


def fire_weather(tas, pr, hurs, ws, snd, month, lat, season_mask, dc0, dmc0, ffmc0, winter_pr, outputs, params):
    """The fire-weather day loop on ``(T, C)`` float32 device series (``xc_fwi_f32``).

    ``month`` int8[T] host array, ``lat`` float64[C] host array or device tensor; ``season_mask`` (T, C) uint8 / previous codes (C,)
    float32 device tensors or None.  ``outputs``: names among DC..DSR, "season_mask", "winter_pr".
    Returns a dict name -> device tensor.
    """
    import ctypes
    ref = tas if tas is not None else pr
    T, C = ref.shape
    dev = ref.device
    ld = ref.stride(0)
    for x in (tas, pr, hurs, ws, snd):
        if x is not None and (tuple(x.shape) != (T, C) or x.stride(0) != ld or x.dtype != torch.float32):
            raise ValueError("fire_weather: the inputs must share their (T, C) float32 layout")
    if season_mask is not None and (tuple(season_mask.shape) != (T, C) or season_mask.dtype != torch.uint8
                                    or season_mask.stride(0) != ld):
        raise ValueError("fire_weather: season_mask must be (T, C) uint8 with the layout of the inputs")
    month_d = dev_ints(np.asarray(month, dtype=np.int8), np.int8, dev)
    if lat is None or isinstance(lat, torch.Tensor):        # a float64 device tensor is used as it is
        lat_d = lat
    else:
        lat_d = torch.from_numpy(np.ascontiguousarray(lat, dtype=np.float64)).to(dev)
    if lat_d is not None and (lat_d.dtype != torch.float64 or lat_d.numel() != C):
        raise ValueError("fire_weather: lat must hold one float64 value per cell")
    out = {}
    for name in outputs:
        if name in FWI_OUTPUTS:      # outputs use the leading dimension of the inputs
            out[name] = torch.empty((T, ld), dtype=torch.float32, device=dev)[:, :C]
        elif name == "season_mask":
            out[name] = torch.empty((T, ld), dtype=torch.uint8, device=dev)[:, :C]
        elif name == "winter_pr":
            out[name] = torch.empty(C, dtype=torch.float32, device=dev)
        else:
            raise ValueError(f"unknown fire weather output {name!r}")
    optr = [_ptr(out.get(n)) for n in FWI_OUTPUTS]
    check(load().xc_fwi_f32(_ptr(tas), _ptr(pr), _ptr(hurs), _ptr(ws), _ptr(snd), _ptr(season_mask), month_d.data_ptr(),
                            _ptr(lat_d), _ptr(dc0), _ptr(dmc0), _ptr(ffmc0), _ptr(winter_pr), T, C, ld,
                            ctypes.byref(params), *optr, _ptr(out.get("season_mask")), _ptr(out.get("winter_pr")),
                            current_stream_ptr()))
    return out


def to_device_f32(values):
    """Any array (numpy, torch) as a float32 CUDA tensor of the same shape."""
    _require_cuda()
    if isinstance(values, torch.Tensor):
        return values.to(device="cuda", dtype=torch.float32)
    return torch.from_numpy(np.ascontiguousarray(np.asarray(values), dtype=np.float32)).to("cuda")


def fire_elementwise(kind, a, b=None, p=(0.0, 0.0, 0.0)):
    """One of the element-wise fire-weather functions on float32 device tensors (``xc_fwi_elementwise_f32``)."""
    if b is not None and tuple(b.shape) != tuple(a.shape):
        raise ValueError("fire_elementwise: the two inputs must share their shape")
    a = a.contiguous()
    b = None if b is None else b.contiguous()
    out = torch.empty_like(a)
    check(load().xc_fwi_elementwise_f32(_lib.FWI_ELEMENTWISE[kind], a.data_ptr(), _ptr(b), a.numel(), float(p[0]),
                                        float(p[1]), float(p[2]), out.data_ptr(), current_stream_ptr()))
    return out
