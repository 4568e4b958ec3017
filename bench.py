#!/usr/bin/env python
"""bench.py — the hot path of BASELINE.json on B200: rows/s and fraction of HBM roofline, filter AND aggregate.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--rows R] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline workload (BASELINE.json configs[1], "C2"): SELECT a FROM t WHERE a > 0.5 over 1e8 synthetic Float64
rows per GPU — the fused predicate + order-preserving filter-gather kernel.  A "step" is one pass of that
operator over one 1e8-row batch.  Rows are partitioned by row range across ranks (no data-path collective for
filter/project), so scaling is weak: every rank filters its own 1e8-row batch and `value` is the total rows of
all ranks / max-over-ranks device time.  The aggregate half of the metric (configs[3], "C4": SELECT k, SUM(v),
COUNT(v) GROUP BY k over 1e8 rows / 1e5 Int64 keys) is measured with the same rules and reported at top level
next to it (`roofline_c4`, `e2e_c4`, `cpu_baseline_c4`); C3 and C5 are in `extra`.

  value         device-resident: the batch is already in HBM when the timed region starts
  e2e           through the C ABI with HOST buffers (dfgpu_filter_project_host): H2D of the batch from pinned
                memory, the kernel, and D2H of the compacted result into pinned memory, every step, pipelined
                by row-range chunk inside the library
  roofline      algorithmic bytes of the dominant kernel (8*N read + 8*N_sel written) / its average duration
                measured with CUDA events recorded around the launch on the launching stream
  sustained     with --sustained only: the same resident step repeated back to back for >= 0.5 s (the K timed
                steps of C2 last a few ms)
  roofline_c4   the same for k_hash_agg (16*N bytes read), e2e_c4 through dfgpu_aggregate_update_host
  extra         C3 (fused expr+filter) and C5 (1e6 keys, MIN/MAX/SUM, 1.25e8 rows per GPU = 1e9 rows on 8 GPUs;
                with N>1 C4 and C5 include the NCCL partial-aggregate merge), same timing rules
  checks        every aggregate result (also the merged multi-GPU one, on every rank) is compared with numpy /
                torch on the same rows: key set, COUNT, MIN, MAX bit-exact, SUM within 1e-9; a mismatch fails the run
  cpu_baseline  the CPU oracle (C++ restatement of the reference's single-threaded operators) on a bounded
                sample of the same workload, on this box's host cores (rank 0, N=1 only)

--impl reference times that CPU restatement alone (the reference is Rust; no toolchain here) on the SAME
config: one full 1e8-row C2 batch per step.

Every timed loop (value, e2e, C3, C4, e2e_c4, C5) runs exactly K = --steps steps after its warm-ups.

--dump-outputs DIR writes, on rank 0, what the last timed step returned to its caller, as DIR/<name>.npy:
  c2_a                        the C2 result column (Float64); above 4 Mi rows, the rows at 4 Mi positions drawn
                              once with numpy's default_rng(0) and kept in ascending order (32 MB)
  c4_key_hi, c4_key_lo        the C4 GROUP BY keys (Int64) as their signed high and unsigned low 32 bits, Float64
  c4_sum, c4_count            SUM(v) and COUNT(v) of C4 (Float64), all rows sorted by key (the engine's row order
                              is that of its hash table and may differ from run to run)
The inputs are seeded, so two runs with the same arguments see the same rows.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True  # a benchmark run leaves the source tree as it found it (no __pycache__)
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "rows/s filter+agg over 1e8-row Arrow batch (C2: SELECT a FROM t WHERE a>0.5, Float64)"
SUM_RTOL = 1e-9
DUMP_SAMPLE_ROWS = 1 << 22  # --dump-outputs: at most 4 Mi rows (32 MB of Float64) of the C2 result column
DUMP_MAX_BYTES = 64 << 20


def c2_config(n):
    """The `config` object of both arms (the reference arm must describe exactly what ours measures)."""
    return {"workload": "C2: SELECT a FROM t WHERE a > 0.5; a~U[0,1) Float64, %d rows per GPU, seed 42+rank" % n,
            "rows_per_gpu": n, "partitioning": "row-range, one batch per rank, no collective",
            "l2": "inputs (%.1f GB per step) larger than L2 (126 MB); no explicit flush" % (8.0 * n / 1e9)}


def ncu_traffic(key):
    """DRAM bytes per launch of the dominant kernel, from the committed ncu capture (profiles/)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(key)
    except Exception:
        return None


def scatter_ceiling(kernel_ms, n):
    """C4's second bound: the measured time of its bare scattered-access pattern (profiles/scatter_peak.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "scatter_peak.json")) as f:
            j = json.load(f)
        floor_ms = j["ldg_red_f64_red_u64_ms_per_1e8_rows"] * n / 1e8
        return {"bound": "lsu/l2-atomic", "floor_ms": floor_ms, "frac": floor_ms / kernel_ms, "source": j["source"]}
    except Exception:
        return None


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []
        self.nvml, self.samples, self.running = None, [], False

    def _nvml_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        ids = [x for x in vis.split(",") if x.strip().isdigit()]
        return int(ids[self.gpu]) if self.gpu < len(ids) else self.gpu

    def start(self):
        # NVML in a thread (one sample every ~2 ms: the timed region of the resident steps is only a few
        # ms long); nvidia-smi -lms 100 as the fallback
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._nvml_index())
            self.nvml = pynvml
            self.running = True
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        N = self.nvml
        while self.running:
            try:
                sm = N.nvmlDeviceGetClockInfo(self.h, N.NVML_CLOCK_SM)
                try:
                    rs = N.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = N.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                pw = N.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                self.samples.append((sm, rs, pw))
            except Exception:
                pass
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml:
            N = self.nvml
            self.running = False
            self.t.join(timeout=1)
            try:
                mx = float(N.nvmlDeviceGetMaxClockInfo(self.h, N.NVML_CLOCK_SM))
            except Exception:
                mx = None
            bits = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4}
            reasons = sorted({nm for _, rs, _ in self.samples for nm, b in bits.items() if rs & b})
            sm = [x[0] for x in self.samples]
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "power_w_max": max([x[2] for x in self.samples], default=None),
                    "samples": len(sm), "reasons": reasons, "source": "nvml, ~2 ms period, warm-up + timed steps (+ sustained loop)"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 100"}


def dist_setup(n_gpus):
    """Returns (rank, world, local_rank, torch or None)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world == 1:
        return 0, 1, 0, None
    # stdout carries exactly one JSON line: NCCL's version / debug banner (stdout by default) goes to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    import torch
    import torch.distributed as dist
    rank, local = int(os.environ["RANK"]), int(os.environ.get("LOCAL_RANK", os.environ["RANK"]))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local, torch


def barrier(torch):
    if torch is not None:
        import torch.distributed as dist
        dist.barrier()
        torch.cuda.synchronize()


def _reduce(torch, x, op):
    if torch is None:
        return x
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=getattr(dist.ReduceOp, op))
    return float(t.item())


def max_over_ranks(torch, x):
    return _reduce(torch, x, "MAX")


def sum_over_ranks(torch, x):
    return _reduce(torch, x, "SUM")


def allreduce_np(torch, arr, op):
    """Element-wise reduction of a numpy array over ranks (the CHECKER's path: torch.distributed, not the engine)."""
    if torch is None:
        return arr
    import torch.distributed as dist
    t = torch.from_numpy(np.ascontiguousarray(arr)).cuda()
    dist.all_reduce(t, op=getattr(dist.ReduceOp, op))
    return t.cpu().numpy()


def time_steps(ctx, torch, fn, steps, warmup, last=None):
    """W untimed warm-ups, then exactly K steps between barrier+sync, device events, max over ranks.
    `last`, if given, is the K-th step: the same work as `fn`, but it keeps its result for the caller."""
    for _ in range(warmup):
        fn()
    ctx.sync()
    barrier(torch)
    ctx.profile_enable(True)
    l0 = ctx.kernel_launches()
    ctx.timer_start()
    for i in range(steps):
        (last if last is not None and i == steps - 1 else fn)()
    ms = ctx.timer_stop()
    ctx.sync()
    barrier(torch)
    kms, kn = ctx.profile_get()
    ctx.profile_enable(False)
    return max_over_ranks(torch, ms), kms, kn, ctx.kernel_launches() - l0


def dump_sample(x):
    """`x` whole if it has at most DUMP_SAMPLE_ROWS rows, else its rows at DUMP_SAMPLE_ROWS positions drawn with
    default_rng(0), ascending: the same positions for the same length."""
    if len(x) <= DUMP_SAMPLE_ROWS:
        return x
    return x[np.sort(np.random.default_rng(0).choice(len(x), DUMP_SAMPLE_ROWS, replace=False))]


def write_outputs(d, arrays):
    """--dump-outputs: one DIR/<name>.npy per array, Float64 only, DUMP_MAX_BYTES in all."""
    assert all(a.dtype == np.float64 for a in arrays.values())
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, "outputs to dump: %d bytes" % total
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), np.ascontiguousarray(a))


def check_groupby(torch, got, k_raw, v, nkeys, want, what):
    """Compare a (possibly merged, global) GROUP BY result with numpy / pandas on the same rows.  `got`: result
    columns [key, aggregates...]; `want`: aggregate names in column order.  Dense per-key partials are computed
    from this rank's rows and combined over ranks with torch.distributed (independent of the engine's merge)."""
    from datafusion_archive_b200 import workloads
    cnt = allreduce_np(torch, np.bincount(k_raw, minlength=nkeys).astype(np.int64), "SUM")
    exp = {"count": cnt.astype(np.uint64)}
    if "sum" in want:
        exp["sum"] = allreduce_np(torch, np.bincount(k_raw, weights=v, minlength=nkeys), "SUM")
    if "min" in want or "max" in want:
        # torch scatter_reduce (amin / amax) on the GPU: an independent library implementation, and fast enough
        # for 1.25e8 rows per rank at N = 8 (numpy's minimum.at / a pandas groupby take minutes there)
        import torch as T
        kt, vt = T.from_numpy(np.ascontiguousarray(k_raw)).cuda(), T.from_numpy(np.ascontiguousarray(v)).cuda()
        mn = T.full((nkeys,), float("inf"), dtype=T.float64, device="cuda").scatter_reduce_(0, kt, vt, "amin").cpu().numpy()
        mx = T.full((nkeys,), float("-inf"), dtype=T.float64, device="cuda").scatter_reduce_(0, kt, vt, "amax").cpu().numpy()
        del kt, vt
        T.cuda.empty_cache()
        exp["min"] = allreduce_np(torch, mn, "MIN")
        exp["max"] = allreduce_np(torch, mx, "MAX")
    present = np.nonzero(cnt)[0]
    mixed = workloads.mix_keys(present.astype(np.int64))
    order = np.argsort(mixed)
    o = np.argsort(got[0])
    assert len(got[0]) == len(present), "%s: %d groups, expected %d" % (what, len(got[0]), len(present))
    assert np.array_equal(got[0][o], mixed[order]), what + ": key set differs"
    for j, name in enumerate(want):
        g, e = got[1 + j][o], exp[name][present][order]
        if name == "sum":
            np.testing.assert_allclose(g, e, rtol=SUM_RTOL, atol=0, err_msg=what + ": SUM")
        else:
            assert np.array_equal(g, e), "%s: %s differs" % (what, name.upper())
    return {"groups": int(len(present)), "checked": [w for w in want], "against": "numpy bincount (SUM, COUNT) / torch scatter_reduce (MIN, MAX) on the same rows"
            + ("; per-rank partials all-reduced with torch.distributed" if torch is not None else "")}


def run_ours(args):
    from datafusion_archive_b200 import engine, workloads
    rank, world, local, torch = dist_setup(args.gpus)
    if world != args.gpus:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d (launch with torch.distributed.run for N>1)" % (args.gpus, world))
    ctx = engine.GpuContext(local)
    peak, peak_src = hbm_peak()
    n = args.rows
    steps, warmup = args.steps, max(3, args.warmup)
    dumps = {}  # --dump-outputs: name -> array

    # ---- C2 (headline) -----------------------------------------------------------------------
    pin_in = engine.PinnedBuffer((n,), np.float64)
    arrays, pred, proj = workloads.c2(n, seed=42 + rank, out=pin_in.array)
    a = arrays[0]
    n_sel = int(np.count_nonzero(a > 0.5))
    batch = ctx.upload([a])
    state = {}

    def step_resident(keep=False):
        r = ctx.filter_project(batch, pred, proj)
        state["nrows"] = r.nrows
        if keep:
            state["r2"] = r
        else:
            r.free()

    def step_e2e():
        # the call a user of the engine makes for a host-resident batch: host buffers in, host buffers
        # out (pinned), H2D / kernel / D2H pipelined by row-range chunk inside the library
        r = ctx.filter_project_host([a], pred, proj)
        state["nrows"] = r.nrows
        state["e2e_out"] = r.host_view(0)[:1000].copy()
        r.free()

    sampler = ClockSampler(local)
    sampler.start()
    ms, kms, kn, launches = time_steps(ctx, torch, step_resident, steps, warmup, last=lambda: step_resident(keep=True))
    assert state["nrows"] == n_sel, "GPU row count %d != expected %d" % (state["nrows"], n_sel)
    r2 = state.pop("r2")
    if args.dump_outputs:
        dumps["c2_a"] = dump_sample(r2.columns()[0])
    r2.free()
    if args.sustained:
        # the same step back to back for >= 0.5 s (same kernel, clocks sampled throughout)
        sus_steps = max(steps, int(np.ceil(600.0 / max(ms / steps, 1e-3))))
        sms, skms, skn, _ = time_steps(ctx, torch, step_resident, sus_steps, 0)
    clocks = sampler.stop()
    total_rows = sum_over_ranks(torch, float(n))
    value = total_rows * steps / (ms / 1e3)
    kernel_ms = kms / steps  # device time of the dominant kernel per step (1 launch per step here)
    alg_bytes = 8.0 * n + 8.0 * n_sel
    achieved = alg_bytes / (kernel_ms / 1e3) / 1e9
    e2e_steps = steps
    ems, _, _, _ = time_steps(ctx, torch, step_e2e, e2e_steps, 3)
    assert state["nrows"] == n_sel and np.array_equal(state["e2e_out"], a[a > 0.5][:1000])
    e2e_value = total_rows * e2e_steps / (ems / 1e3)
    batch.free()

    cfg = c2_config(n)
    cfg["selectivity"] = n_sel / n
    out = {
        "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": cfg, "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "rows/s", "h2d_bytes_per_step": 8 * n, "d2h_bytes_per_step": 8 * n_sel + 32,
                "steps": e2e_steps, "ms_per_step": ems / e2e_steps,
                "path": "dfgpu_filter_project_host: pinned host batch -> chunked H2D | kernel | D2H pipeline -> pinned host result"},
        "gpu_launches": launches,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": ncu_traffic("k_filter_project:c2") if n == 100_000_000 else None, "kernel": "k_filter_project_tma", "kernel_ms": kernel_ms,
                     "algorithmic_bytes": alg_bytes, "peak_source": peak_src},
    }
    if args.sustained:
        out["sustained"] = {"steps": sus_steps, "seconds": sms / 1e3, "ms_per_step": sms / sus_steps, "kernel_ms": skms / sus_steps,
                            "value": total_rows * sus_steps / (sms / 1e3), "roofline_frac": alg_bytes / (skms / sus_steps / 1e3) / 1e9 / peak}

    # ---- C3 (extra) ---------------------------------------------------------------------------------
    extra = {}
    xs = steps
    try:
        arrays3, pred3, proj3 = workloads.c3(n, seed=142 + 10 * rank)
        b3 = ctx.upload(arrays3[:2])  # c, d are never referenced: not uploaded (the host layer prunes them the same way)
        sel3 = int(np.count_nonzero(arrays3[1] < arrays3[0]))

        def step3():
            r = ctx.filter_project(b3, pred3, proj3)
            state["n3"] = r.nrows
            r.free()
        ms3, kms3, kn3, _ = time_steps(ctx, torch, step3, xs, 3)
        assert state["n3"] == sel3
        k3 = kms3 / xs
        bytes3 = 16.0 * n + 16.0 * sel3
        extra["c3"] = {"workload": "C3: SELECT a+b, a*b FROM t WHERE b<a; 4 Float64 cols", "value": total_rows * xs / (ms3 / 1e3),
                       "unit": "rows/s", "ms_per_step": ms3 / xs, "kernel_ms": k3,
                       "roofline": {"bound": "hbm", "achieved": bytes3 / (k3 / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                                    "frac": bytes3 / (k3 / 1e3) / 1e9 / peak, "algorithmic_bytes": bytes3}}
        b3.free()
        del arrays3
    except Exception as e:  # pragma: no cover
        extra["c3"] = {"error": repr(e)}

    # ---- C4 (the aggregate half of the metric: top level) and C5 (extra); a failed check fails the run ----
    if world > 1:
        import torch.distributed as dist
        uid = [engine.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(rank, world, uid[0])
    merge = " + NCCL partial-aggregate merge (global result on every rank)" if world > 1 else ""

    pin_k, pin_v = engine.PinnedBuffer((n,), np.int64), engine.PinnedBuffer((n,), np.float64)
    arrays4, keys4, aggs4, kraw4 = workloads.c4(n, seed=46 + 10 * rank)
    pin_k.array[:] = arrays4[0]
    pin_v.array[:] = arrays4[1]
    arrays4 = [pin_k.array, pin_v.array]
    b4 = ctx.upload(arrays4)

    def step4(keep=False):
        r = ctx.aggregate(b4, keys4, aggs4)
        state["g4"] = r.nrows
        if keep:
            state["r4"] = r
        else:
            r.free()

    def step4_e2e():
        r = ctx.aggregate_host(arrays4, keys4, aggs4)
        state["g4e"] = r.nrows
        state["cols4e"] = r.columns()  # D2H of the (small) result is part of the step
        r.free()
    ms4, kms4, kn4, _ = time_steps(ctx, torch, step4, xs, 3, last=lambda: step4(keep=True))
    r4 = state.pop("r4")
    cols4 = r4.columns()
    r4.free()
    chk4 = check_groupby(torch, cols4, kraw4, arrays4[1], 100_000, ["sum", "count"], "C4")
    if args.dump_outputs:
        o = np.argsort(cols4[0], kind="stable")
        k = cols4[0][o]
        dumps["c4_key_hi"] = (k >> 32).astype(np.float64)
        dumps["c4_key_lo"] = (k & 0xFFFFFFFF).astype(np.float64)
        dumps["c4_sum"] = cols4[1][o].astype(np.float64)
        dumps["c4_count"] = cols4[2][o].astype(np.float64)
    k4 = kms4 / xs  # scan kernel time per step (a first batch runs two launches: 1 Mi-row sampled prefix + the rest)
    bytes4 = 16.0 * n
    out["roofline_c4"] = {"bound": "hbm", "achieved": bytes4 / (k4 / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                          "frac": bytes4 / (k4 / 1e3) / 1e9 / peak, "algorithmic_bytes": bytes4, "kernel": "k_hash_agg_lean", "kernel_ms": k4,
                          "traffic": ncu_traffic("k_hash_agg:c4") if n == 100_000_000 else None, "peak_source": peak_src,
                          "scatter_ceiling": scatter_ceiling(k4, n)}
    out["c4"] = {"workload": "C4: SELECT k, SUM(v), COUNT(v) FROM t GROUP BY k; 1e5 Int64 keys, %d rows per GPU%s" % (n, merge),
                 "value": total_rows * xs / (ms4 / 1e3), "unit": "rows/s", "ms_per_step": ms4 / xs, "steps": xs, "result_check": chk4}
    try:
        ems4, _, _, _ = time_steps(ctx, torch, step4_e2e, xs, 3)
        check_groupby(torch, state["cols4e"], kraw4, arrays4[1], 100_000, ["sum", "count"], "C4 e2e")
        out["e2e_c4"] = {"value": total_rows * xs / (ems4 / 1e3), "unit": "rows/s", "h2d_bytes_per_step": 16 * n,
                         "d2h_bytes_per_step": 24 * state["g4e"], "steps": xs, "ms_per_step": ems4 / xs,
                         "path": "dfgpu_aggregate_update_host: pinned host batch -> chunked H2D overlapped with the scan kernel -> result columns to host"}
    except AttributeError:
        out["e2e_c4"] = None
    b4.free()

    try:
        n5 = args.rows5 or (n * 5) // 4  # 1.25e8 rows per GPU: 8 GPUs = BASELINE's 1e9 rows
        arrays5, keys5, aggs5, kraw5 = workloads.c5(n5, seed=46 + 10 * rank)
        b5 = ctx.upload(arrays5)

        def step5(keep=False):
            r = ctx.aggregate(b5, keys5, aggs5)
            state["g5"] = r.nrows
            if keep:
                state["r5"] = r
            else:
                r.free()
        ms5, kms5, kn5, _ = time_steps(ctx, torch, step5, xs, 3, last=lambda: step5(keep=True))
        r5 = state.pop("r5")
        cols5 = r5.columns()
        r5.free()
        chk5 = check_groupby(torch, cols5, kraw5, arrays5[1], 1_000_000, ["min", "max", "sum"], "C5")
        k5 = kms5 / xs
        bytes5 = 16.0 * n5
        total5 = sum_over_ranks(torch, float(n5))
        extra["c5"] = {"workload": "C5: SELECT k, MIN(v), MAX(v), SUM(v) FROM t GROUP BY k; 1e6 Int64 keys, %d rows per GPU (%.3g rows in all)%s"
                                   % (n5, total5, merge),
                       "groups": state["g5"], "value": total5 * xs / (ms5 / 1e3), "unit": "rows/s", "ms_per_step": ms5 / xs, "kernel_ms": k5,
                       "roofline": {"bound": "hbm", "achieved": bytes5 / (k5 / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                                    "frac": bytes5 / (k5 / 1e3) / 1e9 / peak, "algorithmic_bytes": bytes5, "kernel": "k_hash_agg_lean"},
                       "result_check": chk5}
        b5.free()
        del arrays5
    except AssertionError:
        raise
    except Exception as e:  # pragma: no cover
        extra["c5"] = {"error": repr(e)}
    out["extra"] = extra

    # ---- CPU baselines (rank 0, N=1 only) -----------------------------------------------------------
    if world == 1 and not args.no_cpu:
        out["cpu_baseline"] = cpu_baseline(a, pred, proj, budget_s=12.0)
        out["cpu_baseline_c4"] = cpu_baseline_c4(arrays4, keys4, aggs4)
    ctx.close()
    if rank == 0:
        if args.dump_outputs:
            write_outputs(args.dump_outputs, dumps)
        print(json.dumps(out))
    if torch is not None:
        import torch.distributed as dist
        dist.destroy_process_group()


def cpu_baseline(a, pred, proj, budget_s):
    """The oracle (kind "port": the reference is Rust, not buildable here) on a bounded sample."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    cal = min(len(a), 4_000_000)
    t0 = time.perf_counter()
    O.filter_project([a[:cal]], pred, proj)
    rate = cal / (time.perf_counter() - t0)
    sample = int(min(len(a), max(cal, rate * budget_s / 3)))
    times = []
    for _ in range(3):
        t0 = time.perf_counter()
        O.filter_project([a[:sample]], pred, proj)
        times.append(time.perf_counter() - t0)
    return {"value": sample / float(np.median(times)), "unit": "rows/s", "cores": 1, "host_cores": os.cpu_count(), "kind": "port",
            "sample": "first %d rows of the C2 batch, one batch, median of 3 passes; single thread = the reference's execution model "
                      "(README.md:20; Rc/RefCell operators are !Send)" % sample}


def cpu_baseline_c4(arrays4, keys4, aggs4, sample=10_000_000):
    """C4 through the oracle's with_group_by restatement (per-row key vector -> FNV map -> boxed accumulators,
    aggregate.rs:787-952) on a stated prefix (BASELINE.md §2)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    sample = min(sample, len(arrays4[0]))
    sub = [x[:sample] for x in arrays4]
    t0 = time.perf_counter()
    O.aggregate(sub, keys4, aggs4)
    dt = time.perf_counter() - t0
    return {"value": sample / dt, "unit": "rows/s", "cores": 1, "host_cores": os.cpu_count(), "kind": "port",
            "sample": "first %d rows of the C4 batch, one batch, one pass (%.1f s); single thread" % (sample, dt)}


def run_reference(args):
    """Reference arm: the CPU restatement of the reference's operators on the host cores, same config as ours:
    one full C2 batch (rows_per_gpu rows) per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    from datafusion_archive_b200 import workloads
    n = args.rows
    arrays, pred, proj = workloads.c2(n, seed=42)
    steps, warmup = args.steps, max(3, args.warmup)
    state = {}
    for _ in range(warmup):
        state["out"] = O.filter_project(arrays, pred, proj)
    t0 = time.perf_counter()
    for _ in range(steps):
        state["out"] = O.filter_project(arrays, pred, proj)
    dt = time.perf_counter() - t0
    n_sel = len(state["out"][0])
    value = n * steps / dt
    cfg = c2_config(n)
    cfg["selectivity"] = n_sel / n
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": 1, "host_cores": os.cpu_count(), "kind": "port",
                         "sample": "each step = the whole %d-row C2 batch through oracle/df_oracle.cpp (C++ restatement; the reference is "
                                   "Rust and cannot be built in this image); 1 thread = the reference's execution model (README.md:20), "
                                   "rank 0 only" % n},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps of every timed loop (default: 20; reference arm: 5)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=100_000_000, help="rows per GPU")
    ap.add_argument("--rows5", type=int, default=0, help="rows per GPU of the C5 extra (default 1.25 x --rows)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--sustained", action="store_true", help="also repeat the C2 step back to back for >= 0.5 s (reported as `sustained`)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's C2 and C4 results to DIR/<name>.npy (Float64)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 5 if args.impl == "reference" else 20
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
