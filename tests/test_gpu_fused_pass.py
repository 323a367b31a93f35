"""The fused multi-output pass ``xc_period_multi_f32`` through its C ABI: a seeded random plan for each of the 38
instantiated plan shapes, on grids that take each cell width of the kernel (4 or 2 cells per thread on aligned grids
whose cell count and row stride are multiples of 4, 1 cell otherwise), against oracle compositions of the ORIGINAL
conditions ``x op thr`` -- not the ``sgn * x > thr'`` form the kernel evaluates.  Also: rejected plans, writes
outside the plan's slots, and ``indices.run_batch`` on grids of any width."""
import ctypes
import functools

import numpy as np
import pytest

from oracle import xclim_oracle as O
from xb_helpers import make_field

import test_gpu_batch as batch
import test_fused_plans_cpu as plans_cpu
import test_host_layer_cpu as host_side

pytestmark = pytest.mark.gpu

# (NC, NCR, NM, NS) of the instantiations in xc_period_multi_f32
SHAPES = [(0, 0, 0, 0), (0, 0, 0, 3)] + [(nc, ncr, nm, ns) for nc in (2, 4, 6) for ncr in (0, 1, 2) for nm in (0, 1)
                                         for ns in (0, 3)]
assert len(SHAPES) == 38
OPS = (">", "<", ">=", "<=")
EDGES = np.float32([0.0, -0.0, 1e-45, -1e-45, np.inf, -np.inf])
SENTINEL = np.int32(0x7FC0DEAD)      # a NaN payload the kernel never writes (its NaN is the canonical one)
GUARD = 64                           # floats after the last slot that must stay untouched
T = 1096
CMAX = 2052

# name: (cells, row padding, base offset in floats, cells per thread the dispatcher must pick: 4 (4 or 2) or 1)
LAYOUTS = {
    "C1": (1, 0, 0, 1),
    "C3": (3, 0, 0, 1),
    "C63": (63, 0, 0, 1),
    "C64": (64, 0, 0, 4),
    "C64_offset": (64, 0, 1, 1),
    "C64_ldx68": (64, 4, 0, 4),
    "C1031": (1031, 0, 0, 1),
    "C2052": (2052, 0, 0, 4),
}


def _vec_path(x_ptr, C, ldx, out_ptr):
    """Mirror of can_vec4 in csrc/period_stats.cu: 4 when the dispatcher takes the 4 / 2 cells per thread kernels."""
    return 4 if (C % 4 == 0 and ldx % 4 == 0 and x_ptr % 16 == 0 and out_ptr % 16 == 0) else 1


@functools.cache
def _data():
    """(T, CMAX) float32: values quantised to 0.5 (ties with the thresholds drawn from them), blocky columns whose runs
    cross period boundaries, sprinkled +-0, +-subnormal, NaN and (cells 0, 8, 16, ...) +-inf, and special cells: an
    all-NaN period (cell 1), all-NaN cells (2, 2050), cells where a condition holds every day (+-inf: 61, 62; +-100:
    63, 1030, 2051)."""
    rng = np.random.default_rng(7)
    x = (np.round(rng.standard_normal((T, CMAX)) * 6) / 2).astype(np.float32)
    starts = np.where(rng.random((T, CMAX)) < 1 / 20, np.arange(T)[:, None], 0)
    starts[0] = 0
    blocky = np.take_along_axis(x, np.maximum.accumulate(starts, axis=0), axis=0)
    cols = rng.random(CMAX) < 0.35
    cols[1] = cols[60] = True
    x[:, cols] = blocky[:, cols]
    edge = rng.random((T, CMAX)) < 0.02
    x[edge] = rng.choice(EDGES[:4], size=int(edge.sum()))
    edge[:, np.arange(CMAX) % 8 != 0] = False      # infinities in every 8th cell only
    x[edge] = rng.choice(EDGES, size=int(edge.sum()))
    x[rng.random((T, CMAX)) < 0.03] = np.nan
    x[:400, 1] = np.nan
    x[:, [2, 2050]] = np.nan
    x[:, 61], x[:, 62] = np.inf, -np.inf
    x[:, [63, 2051]], x[:, 1030] = 100.0, -100.0
    return x


@functools.cache
def _period_sets():
    """name -> period offsets (all within the T rows of _data)."""
    from xclim_b200 import TimeAxis
    out = {}
    for cal, start, n in (("noleap", "1981-01-01", 365 * 3), ("standard", "1999-01-01", 1096)):
        ta = TimeAxis.daily(start, n, cal)
        for freq in ("YS", "MS"):
            out[f"{freq}-{cal}"] = np.asarray(ta.period_offsets(freq), dtype=np.int32)
    lengths = [1, 2, 7, 8, 11, 12, 13, 366]
    out["lengths"] = np.cumsum([0] + lengths).astype(np.int32)
    out["from-37"] = (37 + np.cumsum([0] + lengths[::-1] + lengths)).astype(np.int32)
    assert all(p[-1] <= T for p in out.values()) and out["YS-standard"][-1] == 1096
    return out


def _threshold(rng, x, finite=False):
    u = rng.random()
    if u < 0.6 or finite and u >= 0.9:
        v = x[rng.integers(T), rng.integers(CMAX)]
        while not np.isfinite(v):
            v = x[rng.integers(T), rng.integers(CMAX)]
        return float(v)
    if u < 0.9:
        return float(rng.choice(np.float32([0.0, -0.0])))
    return float(rng.choice(EDGES[2:]))


def _condition(rng, x, ops=OPS, finite=False):
    while True:
        op, t = str(rng.choice(ops)), _threshold(rng, x, finite)
        if (op, t) not in ((">=", -np.inf), ("<=", np.inf)):      # no sgn * x > thr' form: refused
            return op, t


def _random_plan(i, shape):
    """A valid plan of shape ``shape`` and its description in original terms.  The declared counts round up on every
    other shape (n_cond 1 / 3 / 5, n_sums 1 / 2); entries beyond them hold live conditions aimed at a spare slot, which
    the dispatcher must neutralise."""
    from xclim_b200 import _lib, device
    nc, ncr, nm, ns = shape
    rng = np.random.default_rng(1000 + i)
    x = _data()
    n_cond = nc - 1 if (nc and i % 2 == 0 and nc - 1 >= max(ncr, 1)) else nc
    n_sums = 0 if ns == 0 else 1 + i % 3
    outs = []                   # (what, slot holder): slots are dealt below

    plan = _lib.MultiPlan()
    plan.n_cond, plan.n_runs, plan.n_msum, plan.n_sums = n_cond, 2 * ncr, nm, n_sums
    spec = {"conds": [], "runs": [], "msum": None, "sums": []}
    for st in ("sum", "mean", "min", "max"):
        outs.append((("stat", st), plan, "slot_" + st))
    for j in range(n_cond):
        if j == 0 and nm:       # the largest-run-sum runs on condition 0: x > t (excess x - t) or x < t (t - x)
            op, t = _condition(rng, x, (">", "<"), finite=True)
        else:
            op, t = _condition(rng, x)
        e = plan.cond[j]
        e.sgn, e.thr = device.normalise_condition(_lib.OPS[op], t)
        e.wmax = int(rng.integers(1, 5))
        spec["conds"].append((op, t, e.wmax))
        outs += [(("n", j), e, "slot_n"), (("max", j), e, "slot_max")]
    for k in range(2 * ncr):
        r = plan.runs[k]
        r.cond, r.window, r.kind = k // 2, int(rng.integers(1, 11)), int(rng.integers(0, 2))
        spec["runs"].append((k // 2, r.kind, r.window))
        outs.append((("run", k), r, "slot"))
    if nm:
        op, t, _ = spec["conds"][0]
        m = plan.msum[0]
        m.cond, m.window, m.sgn, m.thr0 = 0, int(rng.integers(1, 6)), 1.0 if op == ">" else -1.0, t
        spec["msum"] = (m.window, m.sgn, t)
        outs.append((("msum",), m, "slot"))
    for k in range(n_sums):
        s = plan.sums[k]
        op, t = _condition(rng, x)
        s.mode = k % 2 if i % 4 else 1 - k % 2
        if s.mode == 0:
            s.off_sgn, s.off = (1.0 if op in (">", ">=") else -1.0), t
        else:
            s.sgn, s.thr = device.normalise_condition(_lib.OPS[op], t)
        spec["sums"].append((s.mode, op, t))
        outs.append((("sum", k), s, "slot"))
    # about one output in five is not wanted (slot -1); the others take a random permutation of the slots, and two
    # spare slots at the end are named by nobody
    keep = [o for o in outs if rng.random() > 0.2] or outs[:1]
    order = rng.permutation(len(keep))
    named = {}
    for (what, holder, field), sl in zip(keep, order):
        setattr(holder, field, int(sl))
        named[int(sl)] = what
    for what, holder, field in outs:
        if what not in named.values():
            setattr(holder, field, -1)
    n_slots = len(keep) + 2
    spare = n_slots - 1
    for j in range(n_cond, _lib.MULTI_MAX_COND):
        e = plan.cond[j]
        e.sgn, e.thr, e.wmax, e.slot_n, e.slot_max = 1.0, -3.0e38, 1, spare, spare
    for k in range(2 * ncr, _lib.MULTI_MAX_RUNS):
        r = plan.runs[k]
        r.cond, r.window, r.kind, r.slot = 5, 1, 1, spare
    for k in range(nm, _lib.MULTI_MAX_MSUM):
        plan.msum[k].slot = spare
    for k in range(n_sums, _lib.MULTI_MAX_SUMS):
        s = plan.sums[k]
        s.mode, s.off_sgn, s.off, s.slot = 0, 1.0, -3.0e38, spare
    return plan, n_slots, named, spec


def _max_run_sum_steps(ex, window, poff):
    """O.windowed_max_run_sum per period, step by step in float64.  The oracle's cumulative-sum formulation subtracts
    running totals: it loses a run sum below 1e-16 of the period's running total (two subnormal excesses after a few
    ordinary ones come out as 0) and turns an infinite excess into inf - inf = NaN."""
    out = np.zeros((len(poff) - 1, ex.shape[1]))
    for p, (a, b) in enumerate(O._groups(poff)):
        L = np.zeros(ex.shape[1])
        rs = np.zeros(ex.shape[1])
        best = np.zeros(ex.shape[1])
        for t in range(a, b):
            on = ex[t] > 0
            best = np.where(~on & (L >= window), np.maximum(best, rs), best)
            L, rs = np.where(on, L + 1, 0), np.where(on, rs + ex[t], 0)
        out[p] = np.where(L >= window, np.maximum(best, rs), best)
    return out


def _expected(spec, what, x, poff):
    """-> (values (P, CMAX), 'int' | 'exact' | 'float') of one output, from the oracle on the original conditions."""
    x64 = x.astype(np.float64)
    kind = what[0]
    if kind == "stat":
        return O.resample_reduce(x64, poff, what[1]), ("float" if what[1] in ("sum", "mean") else "exact")
    if kind == "n":
        op, t, _ = spec["conds"][what[1]]
        return O.threshold_count(x, op, t, poff), "int"
    if kind == "max":
        op, t, wmax = spec["conds"][what[1]]
        return O.resample_and_rl(O.compare(x, op, t), True, O.rle_statistics, "max", wmax, poff=poff), "exact"
    if kind == "run":
        j, rkind, w = spec["runs"][what[1]]
        op, t, _ = spec["conds"][j]
        red = "sum" if rkind == 0 else "count"
        return O.resample_and_rl(O.compare(x, op, t), True, O.rle_statistics, red, w, poff=poff), "exact"
    if kind == "msum":
        w, sgn, t = spec["msum"]
        with np.errstate(invalid="ignore"):
            d = np.float32(sgn) * (x - np.float32(t))
        ex = np.where(np.isnan(x), 0, np.clip(d, 0, None)).astype(np.float64)
        return _max_run_sum_steps(ex, w, poff), "float"
    mode, op, t = spec["sums"][what[1]]
    if mode == 0:        # the float32 excess of cumulative_difference, summed exactly (multiples of 0.5)
        return O.cumulative_difference(x, t, op, poff), "float"
    return O.resample_reduce(np.where(O.compare(x, op, t), x64, 0.0), poff, "sum"), "float"


_expected_cache = {}


def _expected_all(i):
    """The plan of shape i and, per period set, every named slot's expected values (kept for the shape's layouts)."""
    if i not in _expected_cache:
        _expected_cache.clear()
        plan, n_slots, named, spec = _random_plan(i, SHAPES[i])
        x = _data()
        exp = {ps: {sl: _expected(spec, what, x, poff) for sl, what in named.items()}
               for ps, poff in _period_sets().items()}
        _expected_cache[i] = (plan, n_slots, named, exp)
    return _expected_cache[i]


def _launch(plan, n_slots, C, pad, off, poff, x=None):
    """Run the plan on the first C cells of ``x`` (default _data()) laid out with row stride C + pad, the input and
    the slot buffer both starting ``off`` floats into their allocations.  -> (status, vec path, slots (n_slots, P, C)
    as int32, the whole int32 output allocation)."""
    import torch
    from xclim_b200 import _lib, device
    x = _data() if x is None else x
    ldx = C + pad
    P = len(poff) - 1
    xs = torch.full((off + T * ldx,), 1.0e6, dtype=torch.float32)       # row padding: values no cell may read
    xs[off:].view(T, ldx)[:, :C] = torch.from_numpy(np.ascontiguousarray(x[:, :C]))
    xs = xs.cuda()
    out = torch.full((off + max(1, n_slots) * P * C + GUARD,), int(SENTINEL), dtype=torch.int32, device="cuda")
    poff_d = torch.from_numpy(np.ascontiguousarray(poff, dtype=np.int32)).cuda()
    x_ptr, out_ptr = xs.data_ptr() + 4 * off, out.data_ptr() + 4 * off
    st = _lib.load().xc_period_multi_f32(x_ptr, T, C, ldx, poff_d.data_ptr(), P, ctypes.byref(plan), out_ptr,
                                         n_slots, device.current_stream_ptr())
    torch.cuda.synchronize()
    whole = out.cpu().numpy()
    return st, _vec_path(x_ptr, C, ldx, out_ptr), whole[off:off + n_slots * P * C].reshape(n_slots, P, C), whole


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("i", range(len(SHAPES)), ids=["nc%d-ncr%d-nm%d-ns%d" % s for s in SHAPES])
def test_fused_pass_against_original_conditions(cuda, layout, i):
    C, pad, off, path = LAYOUTS[layout]
    plan, n_slots, named, exp = _expected_all(i)
    for ps, poff in _period_sets().items():
        st, vec, got, whole = _launch(plan, n_slots, C, pad, off, poff)
        assert st == 0, (ps, st)
        assert vec == path, "the layout does not take the path it is meant to"
        for sl in range(n_slots):
            msg = f"{layout} {ps} slot {sl} {named.get(sl)}"
            if sl not in named:       # unnamed and neutralised entries write nothing
                assert (got[sl] == SENTINEL).all(), msg
                continue
            e, how = exp[ps][sl]
            e = e[:, :C]
            if how == "int":
                np.testing.assert_array_equal(got[sl], e.astype(np.int32), err_msg=msg)
            elif how == "exact":
                np.testing.assert_array_equal(got[sl].view(np.float32), e, err_msg=msg)
            else:
                np.testing.assert_allclose(got[sl].view(np.float32), e.astype(np.float32), rtol=1e-6, atol=0,
                                           equal_nan=True, err_msg=msg)      # float64 accumulation, one rounding
        assert (whole[:off] == SENTINEL).all() and (whole[off + n_slots * got.shape[1] * C:] == SENTINEL).all(), \
            f"{layout} {ps}: write outside the slots"
        if layout == "C64_offset":    # 1 cell per thread == 4 / 2 cells per thread, bit for bit
            st4, vec4, got4, _ = _launch(plan, n_slots, C, 0, 0, poff)
            assert st4 == 0 and vec4 == 4
            np.testing.assert_array_equal(got, got4, err_msg=ps)


def _bad_plans():
    from xclim_b200 import _lib
    base, n_slots, _, _ = _random_plan(5, (4, 2, 1, 3))
    assert base.n_cond == 4 and base.n_runs == 4 and base.n_msum == 1

    def copy():
        p = _lib.MultiPlan()
        ctypes.memmove(ctypes.byref(p), ctypes.byref(base), ctypes.sizeof(p))
        return p
    out = {}
    p = copy()
    p.slot_sum = n_slots
    out["slot at n_slots"] = p
    p = copy()
    p.runs[1].slot = n_slots + 3
    out["run slot above n_slots"] = p
    p = copy()
    p.n_runs = 3
    out["odd n_runs"] = p
    p = copy()
    p.runs[2].cond = 0
    out["run output away from its condition"] = p
    p = copy()
    p.n_cond, p.n_runs = 0, 0
    out["max-sum without a condition"] = p
    return out, n_slots


@pytest.mark.parametrize("case", ["slot at n_slots", "run slot above n_slots", "odd n_runs",
                                  "run output away from its condition", "max-sum without a condition"])
def test_rejected_plans_launch_nothing(cuda, case):
    from xclim_b200 import _lib
    plans, n_slots = _bad_plans()
    poff = _period_sets()["YS-noleap"]
    for C, off in ((64, 0), (63, 0), (64, 1)):
        st, _, _, whole = _launch(plans[case], n_slots, C, 0, off, poff)
        assert st == _lib.XC_ERR_INVALID, (case, st)
        assert (whole == SENTINEL).all(), f"{case}: a kernel ran"


# ---------------------------------------------------------------------------------------- run_batch on any grid
def _awkward_fields(cells):
    """(host arrays, the Fields run_batch takes): the batch inputs on ``cells``, or ("unaligned", (4, 8)): device
    Fields on a contiguous tensor 4 bytes into its storage."""
    import torch
    from xclim_b200 import Field
    unaligned = cells[0] == "unaligned"
    shape = cells[1] if unaligned else cells
    data = batch._inputs(shape)
    units = {"tas": "K", "tasmax": "K", "tasmin": "K", "pr": "mm/d"}
    fields = {k: make_field(v, "1981-01-01", calendar="noleap", units=units[k]) for k, v in data.items()}
    if unaligned:
        dev = {}
        for k, v in data.items():
            flat = torch.empty(v.size + 1, dtype=torch.float32, device="cuda")
            t = flat[1:].view(v.shape)
            t.copy_(torch.from_numpy(v))
            assert t.is_contiguous() and t.data_ptr() % 16 != 0
            f = fields[k]
            dev[k] = Field(t, f.dims, f.time, dict(f.coords), dict(f.attrs))
        fields = dev
    return data, fields


@pytest.mark.parametrize("cells", [(1,), (3, 5), (7, 9), ("unaligned", (4, 8))], ids=["1", "3x5", "7x9", "4x8-unaligned"])
def test_run_batch_on_grids_of_any_width(cuda, cells):
    data, fields = _awkward_fields(cells)
    host_side._check_run_batch_against_single_calls(exact=True, fields=fields)
    batch._check_indicators_against_oracle(data, fields)


def test_plan_packing_under_random_subsets_on_the_kernel(cuda, monkeypatch):
    plans_cpu.check_random_subsets(monkeypatch, exact=True)


def test_plan_packing_of_random_passes_on_the_kernel(cuda):
    import torch
    from xclim_b200 import device
    plans_cpu.check_random_pass_builders(device.period_multi, lambda a: torch.from_numpy(a).cuda())
