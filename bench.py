#!/usr/bin/env python
"""bench.py -- headline benchmark of the xclim_b200 hot path (contract: DESIGN.md section 6).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA kernels)
    python bench.py --impl reference --gpus N --steps K ...   # CPU arm: the oracle port on host cores
    python bench.py ... --dump-outputs DIR                    # + the last timed step's results as DIR/*.npy

Workload (BASELINE.json configs[1]): ``maximum_consecutive_dry_days`` (+ fused MissingAny valid
count) on ONE synthetic daily float32 ``pr`` grid of shape (10950, 721, 1440) in mm/d, yearly
periods.  One step = one pass of the hot path over the whole grid.  With N GPUs the grid is cut into
contiguous lat tiles (721 rows -> 91, 90, ..., 90 on 8 ranks; xclim_b200.multigpu.lat_tiles): every
rank owns one tile, there is no collective on the data path and ``value`` = 1,038,240 cells /
max-over-ranks time (STRONG scaling).  The optional NCCL gather of the (30, 721, 1440) result and
the replicated (weak) figure are reported as secondary keys.

Further sections of the same JSON line (BASELINE.json configs[2..4], each on this rank's lat tile):
``tx90p`` (percentile_doy + count, sub-case 3a), ``bootstrap`` (3b: 15-year base, bootstrap=True),
``eqm`` (EmpiricalQuantileMapping train + adjust), ``batch50`` (50 indicators), ``e2e`` (host
buffers through the Python index functions, H2D/D2H inside the timed region), ``cpu_baseline``.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

T_FULL, Y_FULL, X_FULL, YEAR = 10950, 721, 1440, 365
METRIC = "grid_cells_per_s:maximum_consecutive_dry_days(10950x721x1440,f32)"
UNIT = "grid-cells/s"
ALL_SECTIONS = ("parity", "weak", "gather", "tx90p", "bootstrap", "eqm", "batch50", "e2e", "fwi", "cpu")
DUMP_CELLS = 1 << 17   # --dump-outputs: 30 periods x 131,072 cells x 4 B x 2 arrays = 31 MB


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--lat", type=int, default=Y_FULL, help="lat rows of the GLOBAL grid (default: full 721)")
    ap.add_argument("--sections", default=",".join(ALL_SECTIONS),
                    help="comma list of secondary sections to run (default: all): " + ",".join(ALL_SECTIONS))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-tx90p", action="store_true")
    ap.add_argument("--cpu-lat", type=int, default=6, help="lat rows per worker of the bounded CPU sample")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step to DIR/<name>.npy (float32, (periods, cells), on a "
                         f"fixed seeded sample of at most {DUMP_CELLS} cells of the grid)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    sec = [s for s in a.sections.split(",") if s]
    if a.no_e2e and "e2e" in sec:
        sec.remove("e2e")
    if a.no_cpu and "cpu" in sec:
        sec.remove("cpu")
    if a.no_tx90p and "tx90p" in sec:
        sec.remove("tx90p")
    a.sections = sec
    return a


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock / throttle reasons with NVML during the timed region."""

    def __init__(self, index=0, period=0.002):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._th = None
        self.index, self.period = index, period
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        if self.nv is not None:
            try:   # the first NVML queries of a process take tens of ms: prime them outside the timed region
                self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)
                self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                pass
            self._th = threading.Thread(target=self._run, daemon=True)
            self._th.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._th:
            self._th.join(timeout=2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------ CPU arm
def _cpu_cdd_band(args):
    """One worker: `lat` rows of (10950, 1, 1440), processed row by row to bound memory.  The input
    distribution is the GPU arm's (10-day wet/dry regimes, exponential amounts), generated with numpy."""
    from oracle import xclim_oracle as O
    seed, lat, X = args
    rng = np.random.default_rng(seed)
    poff = np.arange(T_FULL // YEAR + 1) * YEAR
    busy = 0.0
    acc = 0.0
    for _ in range(lat):
        regime = np.repeat(rng.random((T_FULL // 10 + 1, 1, X)) < 0.5, 10, axis=0)[:T_FULL]
        dry = rng.random((T_FULL, 1, X), dtype=np.float32) < np.where(regime, np.float32(0.8), np.float32(0.3))
        x = rng.standard_exponential((T_FULL, 1, X), dtype=np.float32) * np.float32(6.0)
        x[dry] = 0.0
        t = time.perf_counter()
        out = O.maximum_consecutive_dry_days(x, 1.0, poff)
        miss = O.missing_any(x, poff)
        out = np.where(miss, np.nan, out)
        busy += time.perf_counter() - t
        acc += float(np.nansum(out))
    return busy, acc


def _cpu_procs():
    cores = os.cpu_count() or 1
    use = max(1, cores)          # every host core (bounded below by the memory check: ~3 GB per worker)
    try:
        import psutil
        use = max(1, min(use, int(psutil.virtual_memory().available // (3 << 30))))
    except Exception:
        pass
    return use


def cpu_arm(lat_rows: int, cores: int, steps: int = 1, warmup: int = 0):
    """Oracle port (numpy restatement of the reference's whole-array algorithm) on `cores`
    processes, each working on its own lat band of `lat_rows` rows.  Returns cells/s computed from
    the slowest worker's busy time (input generation excluded)."""
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    jobs = [(1000 + i, lat_rows, X_FULL) for i in range(cores)]
    times = []
    with ctx.Pool(cores) as pool:
        for it in range(warmup + steps):
            res = pool.map(_cpu_cdd_band, jobs)
            if it >= warmup:
                times.append(max(r[0] for r in res))
    cells = cores * lat_rows * X_FULL
    dt = float(np.mean(times))
    return cells / dt, dt, cells


def run_reference(args):
    """The reference arm: xclim itself is not importable offline (xarray / dask / pint / cftime are
    absent from the image and from /opt/wheelhouse), so the oracle port -- the numpy restatement of the
    reference's whole-array algorithm, pinned to the reference's own cores (tests/golden) -- is timed on
    every host core.  One step = ONE lat row per core (a bounded sample of the same workload, scaled by
    cells), so that --steps 20 --warmup 5 ends within a few minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    use = _cpu_procs()
    rows = 1
    value, dt, cells = cpu_arm(rows, use, steps=args.steps, warmup=min(args.warmup, 1))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "maximum_consecutive_dry_days (10950,721,1440) f32 pr mm/d, thresh 1 mm/day, op <, "
                               "freq=YS, fused MissingAny valid count",
                   "global_grid": [T_FULL, Y_FULL, X_FULL],
                   "note": "reference package not importable offline (xarray/dask/pint absent): the oracle port "
                           "(restatement, not reference) is timed on the host cores"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": use, "kind": "port",
                         "sample": f"{use} lat bands of (10950,{rows},1440) per step, one process per core, "
                                   f"{dt:.1f} s busy per step"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ our arm
def dump_outputs(path, out, valid, cell0, cells_total, rank, world):
    """Writes what one step returns, (out, valid) of the (periods, cells) tile starting at global cell `cell0`, on
    a sample of cells of the global grid that depends on nothing but its size: ``maximum_consecutive_dry_days.npy``
    and ``valid_days.npy`` (days with data per period; MissingAny masks the periods short of 365), float32, cells
    in global order."""
    import torch
    import torch.distributed as dist
    sel = np.sort(np.random.default_rng(0).choice(cells_total, min(DUMP_CELLS, cells_total), replace=False))
    mine = torch.from_numpy(sel[(sel >= cell0) & (sel < cell0 + out.shape[1])] - cell0).to(out.device)
    parts = [(out[:, mine].cpu().numpy(), valid[:, mine].cpu().numpy().astype(np.float32))]
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, parts[0])
        parts = gathered
    if rank == 0:
        os.makedirs(path, exist_ok=True)
        for i, name in enumerate(("maximum_consecutive_dry_days", "valid_days")):
            np.save(os.path.join(path, name + ".npy"), np.concatenate([p[i] for p in parts], axis=1))


def run_ours(args):
    import torch
    import torch.distributed as dist

    import bench_sections as S
    from xclim_b200 import _lib, device, multigpu

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(vals):
        tt = torch.tensor(list(vals), dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return [float(v) for v in tt.tolist()]

    ctx = S.Ctx(args=args, dev=dev, rank=rank, world=world, local=local, barrier=barrier,
                max_over_ranks=max_over_ranks, peak=S.measured_peak(ROOT), root=ROOT)
    T, Yg, X = T_FULL, args.lat, X_FULL
    tiles = multigpu.lat_tiles(Yg, world)
    r0, r1 = tiles[rank]
    ctx.rows, ctx.row0, ctx.n_lat_global = r1 - r0, r0, Yg
    C = ctx.rows * X
    P = T // YEAR
    poff = np.arange(P + 1, dtype=np.int32) * YEAR
    # ---- this rank's lat tile of the ONE global grid, generated in HBM by the stateless generator
    pr = device.synth(T, C, kind=0, seed=2, cell_offset=r0 * X, cells_per_lat=X, n_lat_global=Yg)
    op, red = _lib.OPS["<"], _lib.RL_REDUCERS["max"]
    launches = [0]

    def step():
        out, valid = device.period_runstat(pr, poff, op, 1.0, red, 1, resample_before_rl=True, want_valid=True)
        launches[0] += 1
        return out, valid

    warm = max(args.warmup, 3)
    for _ in range(warm):
        out, valid = step()
    barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    launches[0] = 0
    with ClockSampler(local) as clk:
        barrier()
        ev[0].record()
        for i in range(args.steps):
            out, valid = step()
            ev[i + 1].record()
        barrier()
    per_step = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    (total_ms,) = max_over_ranks([ev[0].elapsed_time(ev[args.steps])])
    ms_per_step = total_ms / args.steps
    cells_total = Yg * X
    value = cells_total / (ms_per_step * 1e-3)
    # ---- roofline of the dominant kernel (period_runstat_kernel) on THIS rank's tile
    alg_bytes = T * C * 4 + P * C * 4 + P * C * 4  # read x once; write out f32 + valid i32
    kern_ms = float(np.mean(per_step))
    achieved = alg_bytes / (kern_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": ctx.peak["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / ctx.peak["hbm_gbs"],
                "traffic": S.ncu_traffic(ROOT, "period_runstat_kernel", [T, ctx.rows, X]),
                "kernel": "period_runstat_kernel<LT,MAX,VEC4,VALID,FASTMAX>",
                "algorithmic_bytes": alg_bytes, "launch_ms": kern_ms, "tile": [T, ctx.rows, X],
                "peak_source": ctx.peak["source"]}
    out_max = float(out.max().item())
    n_missing = int((valid != YEAR).sum().item())
    assert 0 <= out_max <= YEAR
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, valid, r0 * X, Yg * X, rank, world)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": warm, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"maximum_consecutive_dry_days ({T},{Yg},{X}) f32 pr mm/d, thresh 1 mm/day, op <, "
                               f"freq=YS, fused MissingAny valid count",
                   "global_grid": [T, Yg, X],
                   "partition": f"one global grid, contiguous lat tiles over {world} rank(s): "
                                + ",".join(str(b - a) for a, b in tiles) + " rows; no collective on the data path",
                   "l2_policy": f"per-rank input {T * C * 4 / 1e9:.1f} GB >> 126 MB L2, read once per step "
                                "(no flush needed)"},
        "roofline": roofline, "gpu_launches": launches[0], "clocks": clk.summary(),
        "check": {"out_max_days": out_max, "periods_masked_missing": n_missing},
    }
    sec = args.sections

    def guarded(name, fn):
        """A secondary section must not cost the headline line: on ONE GPU its failure is recorded, not
        raised.  Under torchrun a rank that swallowed an error would leave the others waiting in the next
        barrier, so there the error propagates and torchrun ends the job."""
        if world > 1:
            return fn()
        try:
            return fn()
        except Exception as e:  # noqa: BLE001
            import traceback
            print(f"[bench] section {name} failed:\n{traceback.format_exc()}", file=sys.stderr, flush=True)
            try:
                torch.cuda.empty_cache()
            except Exception:  # noqa: BLE001  (a faulted context: nothing more to free)
                pass
            return {"error": f"{type(e).__name__}: {e}"[:400]}

    # ---- full-size parity: sampled cells of this tile (incl. the last CTA's) against the oracle
    if "parity" in sec:
        line["parity"] = S.parity_cdd(ctx, pr, poff, out, valid)
    if "gather" in sec and world > 1:
        line["gather"] = guarded("gather", lambda: S.gather_section(ctx, out, P))
    # ---- end to end through the Python index functions with host buffers
    if "e2e" in sec:
        affinity = os.sched_getaffinity(0)   # the e2e leg pins this process to the GPU's NUMA node
        try:
            line["e2e"] = guarded("e2e", lambda: S.e2e_section(ctx, pr, poff, out, valid))
        finally:
            os.sched_setaffinity(0, affinity)  # ... the CPU arm below must see every core again
    del pr, out, valid
    torch.cuda.empty_cache()
    if "weak" in sec and world > 1:
        line["weak_replicas"] = guarded("weak", lambda: S.weak_section(ctx))
    if "tx90p" in sec or "bootstrap" in sec:
        err = guarded("tx90p", lambda: S.tx90p_sections(ctx, line, want_3a="tx90p" in sec, want_3b="bootstrap" in sec))
        if isinstance(err, dict) and "error" in err:
            line.setdefault("tx90p", err)
    if "eqm" in sec:
        line["eqm"] = guarded("eqm", lambda: S.eqm_section(ctx))
    if "batch50" in sec:
        line["batch50"] = guarded("batch50", lambda: S.batch50_section(ctx))
    # ---- the fire-weather kernel: last GPU section, one GPU only, guarded (its first run on hardware)
    if "fwi" in sec and world == 1:
        line["fwi"] = guarded("fwi", lambda: S.fwi_section(ctx))
    # ---- CPU baseline (oracle port) on a bounded sample, rank 0, N == 1 only
    if rank == 0 and world == 1 and "cpu" in sec:
        use = _cpu_procs()
        v, dt, cells = cpu_arm(args.cpu_lat, use)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": use, "kind": "port",
                                "sample": f"{use} lat bands of (10950,{args.cpu_lat},1440), one process per core, "
                                          f"{dt:.1f} s (restatement, not reference: xclim is not importable here)"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    elif any(isinstance(v, dict) and "error" in v for v in line.values()):
        # a section failed (possibly with a faulted CUDA context): the line is out, skip the teardown
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    a = parse_args()
    # the contract is ONE JSON line on stdout: libraries that print to fd 1 (e.g. "NCCL version ...")
    # are sent to stderr, and only the final line goes to the real stdout
    sys.stdout.flush()
    _real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = _real_stdout
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
