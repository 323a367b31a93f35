"""Plan packing of the fused batch pass (indices._PassBuilder.plans) under random subsets of the batch: every plan
handed to ``xc_period_multi_f32`` keeps the ABI's invariants (include/xclim_b200.h: XcMultiPlan), and the subset's
fused results equal the one-call-per-indicator results.  The device layer is the oracle stand-in of
tests/fake_device.py; tests/test_gpu_fused_pass.py runs the same check on the kernel."""
import numpy as np
import pytest

import fake_device
from oracle import xclim_oracle as O
from xclim_b200 import _lib

import test_host_layer_cpu as host_side

N_SUBSETS = 30


@pytest.fixture
def host(monkeypatch):
    fake_device.install(monkeypatch)


def check_plan(plan, n_slots):
    """The checks of xc_period_multi_f32 on a plan (csrc/period_stats.cu), on the declared entries, plus: the named
    slots are unique and use every slot of the buffer."""
    assert 0 <= plan.n_cond <= _lib.MULTI_MAX_COND and 0 <= plan.n_msum <= _lib.MULTI_MAX_MSUM
    assert 0 <= plan.n_runs <= _lib.MULTI_MAX_RUNS and plan.n_runs % 2 == 0
    assert 0 <= plan.n_sums <= _lib.MULTI_MAX_SUMS
    assert plan.n_runs // 2 <= plan.n_cond, "run outputs need their condition"
    assert plan.n_msum == 0 or plan.n_cond > 0, "a largest-run-sum needs its condition"
    slots = [plan.slot_sum, plan.slot_mean, plan.slot_min, plan.slot_max]
    for j in range(plan.n_cond):
        c = plan.cond[j]
        assert c.sgn in (1.0, -1.0) and c.wmax >= 1
        slots += [c.slot_n, c.slot_max]
    for k in range(plan.n_runs):
        r = plan.runs[k]
        assert r.cond == k // 2 and r.window >= 1 and r.kind in (0, 1)
        slots.append(r.slot)
    for k in range(plan.n_msum):
        m = plan.msum[k]
        assert m.cond == 0 and m.window >= 1 and m.sgn in (1.0, -1.0)
        slots.append(m.slot)
    for k in range(plan.n_sums):
        assert plan.sums[k].mode in (0, 1)
        slots.append(plan.sums[k].slot)
    assert all(-1 <= s < n_slots for s in slots), slots
    named = [s for s in slots if s >= 0]
    assert sorted(named) == list(range(n_slots)), f"slots not unique or not all used: {named} of {n_slots}"


def check_random_subsets(monkeypatch, exact):
    """run_batch(names=subset) on N_SUBSETS seeded random subsets of BATCH_INDICATORS: every plan passes check_plan,
    the results equal the single calls, and the subsets reach every packing case of _PassBuilder.plans."""
    from xclim_b200 import device, indices
    seen = dict.fromkeys(("max-sum owner at place 0 with an unused run place", "condition listed again"), False)
    period_multi, plans = device.period_multi, indices._PassBuilder.plans

    def checked_period_multi(x2d, poff, plan, n_slots):
        check_plan(plan, n_slots)
        if plan.n_msum and plan.n_runs and plan.runs[0].slot < 0 and plan.runs[1].slot < 0:
            seen["max-sum owner at place 0 with an unused run place"] = True
        return period_multi(x2d, poff, plan, n_slots)

    def recorded_plans(self):
        out = plans(self)
        keys = [(p.cond[j].sgn, p.cond[j].thr) for p, _, _ in out for j in range(p.n_cond)]
        seen["condition listed again"] |= len(set(keys)) < len(keys)
        return out
    monkeypatch.setattr(device, "period_multi", checked_period_multi)
    monkeypatch.setattr(indices._PassBuilder, "plans", recorded_plans)
    names = [n for n, _ in indices.BATCH_INDICATORS]
    rng = np.random.default_rng(2024)
    for _ in range(N_SUBSETS):
        subset = set(rng.choice(names, size=int(rng.integers(1, len(names) + 1)), replace=False).tolist())
        host_side._check_run_batch_against_single_calls(exact=exact, names=subset)
    assert all(seen.values()), seen


def test_plan_packing_under_random_subsets(host, monkeypatch):
    check_random_subsets(monkeypatch, exact=False)


def _expected_request(key, req, x, poff):
    """The oracle value of one request of a _PassBuilder, from its original condition ``x op t``."""
    x64 = x.astype(np.float64)
    kind, op, t, w = req
    if kind == "stat":
        return O.resample_reduce(x64, poff, op)
    if kind == "n":
        return O.threshold_count(x, op, t, poff)
    if kind in ("max", "sum", "count"):
        return O.resample_and_rl(O.compare(x, op, t), True, O.rle_statistics, kind, w, poff=poff)
    if kind == "ms":
        d = np.float32(1 if op == ">" else -1) * (x - np.float32(t))
        ex = np.where(np.isnan(x), 0, np.clip(d, 0, None)).astype(np.float64)
        return O.resample_and_rl(ex, True, O.windowed_max_run_sum, w, poff=poff)
    if kind == "excess":
        return O.cumulative_difference(x, t, op, poff)
    return O.resample_reduce(np.where(O.compare(x, op, t), x64, 0.0), poff, "sum")


def check_random_pass_builders(period_multi, to_device):
    """_PassBuilder.plans on random requests beyond what the batch asks for -- up to 12 conditions, up to 3 run outputs
    per condition, two largest-run-sums, up to 5 conditional sums -- so that passes split into several launches.  Every
    plan passes check_plan, and every request's slot equals the oracle of its original condition."""
    from xclim_b200 import TimeAxis, device, indices
    rng = np.random.default_rng(77)
    T, C = 730, 16
    x = (np.round(rng.standard_normal((T, C)) * 6) / 2).astype(np.float32)
    x[rng.random(x.shape) < 0.03] = np.nan
    x2d = to_device(x)
    seen = dict.fromkeys(("pass split into several launches", "condition listed again",
                          "max-sum owner at place 0 with an unused run place"), False)
    for seed in range(20):
        rng = np.random.default_rng(seed)
        poff = TimeAxis.daily("1981-01-01", T, "noleap").period_offsets(("YS", "MS")[seed % 2])
        pb = indices._PassBuilder()
        req = {}
        for st in rng.permutation(["sum", "mean", "min", "max"])[:int(rng.integers(0, 5))]:
            pb.stats[str(st)] = True
            req[("stat", str(st))] = ("stat", str(st), None, None)
        n_ms = 0
        for _ in range(int(rng.integers(1, 13))):
            op, t = str(rng.choice([">", "<", ">=", "<="])), float(x[rng.integers(T), rng.integers(C)])
            if t != t:
                t = 0.0
            c, k = pb.cond(_lib.OPS[op], t)
            if rng.random() < 0.6:
                c["n"] = True
                req[("n",) + k] = ("n", op, t, None)
            if rng.random() < 0.4:
                c["max"] = True
                req[("max",) + k] = ("max", op, t, 1)
            for _ in range(int(rng.integers(0, 4))):
                kind, w = str(rng.choice(["sum", "count"])), int(rng.integers(1, 6))
                c["runs"].add((kind, w))
                req[(kind,) + k + (w,)] = (kind, op, t, w)
            if op in (">", "<") and c["ms"] is None and n_ms < 2 and rng.random() < 0.5:
                w = int(rng.integers(1, 5))
                c["ms"] = (w, 1.0 if op == ">" else -1.0, float(np.float32(t)))
                req[("ms",) + k + (w,)] = ("ms", op, t, w)
                n_ms += 1
        for _ in range(int(rng.integers(0, 6))):
            op, t = str(rng.choice([">", "<", ">=", "<="])), float(rng.integers(-8, 9)) / 2
            if rng.random() < 0.5:
                key = (0, 0.0, 0.0, 1.0 if op in (">", ">=") else -1.0, t)
                req[("qsum",) + key] = ("excess", op, t, None)
            else:
                key = (1,) + device.normalise_condition(_lib.OPS[op], t) + (0.0, 0.0)
                req[("qsum",) + key] = ("where", op, t, None)
            pb.sums[key] = True
        launches = pb.plans()
        seen["pass split into several launches"] |= len(launches) > 1
        keys = [(p.cond[j].sgn, p.cond[j].thr) for p, _, _ in launches for j in range(p.n_cond)]
        seen["condition listed again"] |= len(set(keys)) < len(keys)
        got = {}
        for plan, n, where in launches:
            check_plan(plan, n)
            if plan.n_msum and plan.n_runs and plan.runs[0].slot < 0 and plan.runs[1].slot < 0:
                seen["max-sum owner at place 0 with an unused run place"] = True
            buf = period_multi(x2d, poff, plan, n).cpu().numpy()
            for key, (sl, is_int) in where.items():
                got[key] = buf[sl].view(np.int32) if is_int else buf[sl]
        assert set(got) == set(req), seed
        for key, r in req.items():
            exp = _expected_request(key, r, x, poff)
            if r[0] in ("stat", "ms", "excess", "where") and r[1] not in ("min", "max"):
                np.testing.assert_allclose(got[key], exp.astype(np.float32), rtol=1e-6, atol=0, equal_nan=True,
                                           err_msg=f"{seed} {key}")
            else:
                np.testing.assert_array_equal(got[key], exp.astype(got[key].dtype), err_msg=f"{seed} {key}")
    assert all(seen.values()), seen


def test_plan_packing_of_random_passes(host):
    import torch
    check_random_pass_builders(fake_device.period_multi, torch.from_numpy)


@pytest.mark.parametrize("op,thr", [(">=", -np.inf), ("<=", np.inf)])
def test_conditions_without_a_fused_form_are_refused(op, thr):
    from xclim_b200 import device
    with pytest.raises(NotImplementedError):
        device.normalise_condition(_lib.OPS[op], thr)


@pytest.mark.parametrize("op", [">", "<", ">=", "<="])
def test_normalised_conditions_agree_with_the_operator(op):
    """sgn * x > thr' against x op thr in float32 over the edge values, thresholds at zero, subnormals, infinities
    and the neighbours of each threshold."""
    from oracle import xclim_oracle as O
    from xclim_b200 import device
    f32 = np.float32
    edges = f32([0.0, -0.0, 1e-45, -1e-45, 2e-45, np.inf, -np.inf, np.nan, 1.0, -1.0, 3.5, np.finfo(np.float32).max,
                 -np.finfo(np.float32).max, np.finfo(np.float32).tiny])
    x = np.concatenate([edges, np.nextafter(edges, f32(np.inf)), np.nextafter(edges, f32(-np.inf))])
    for t in edges[~np.isnan(edges)]:
        if (op, t) in ((">=", -np.inf), ("<=", np.inf)):
            continue
        sgn, thr = device.normalise_condition(_lib.OPS[op], float(t))
        with np.errstate(invalid="ignore"):
            got = f32(sgn) * x > f32(thr)
        np.testing.assert_array_equal(got, O.compare(x, op, float(t)), err_msg=f"{op} {t!r}")
