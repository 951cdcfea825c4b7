#!/usr/bin/env python
"""bench.py — BASELINE.json's metric: lin_reg-family rows/sec on B200 next to the reference's CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C1|C2|C3|C4|C5] [--impl ours|reference]

Default workload = BASELINE configs[1] (C2): pds.lin_reg on 1e8 rows x 32 f32 features, return_pred=True.
One "step" = one pass of the hot path over the resident synthetic frame.  ONE JSON line (rank 0):

  value         whole-job rows/s, inputs resident in HBM (CUDA events, max over ranks)
  e2e           the same metric through the reference-facing plugin symbol (`_polars_plugin_pl_*`) with PAGEABLE host
                Arrow buffers (what Polars hands a plugin): H2D of every input column and D2H of the result are inside
                the timed region; `pinned_value` repeats it with page-locked inputs
  roofline      the dominant kernel timed alone with CUDA events; algorithmic bytes per row as SURVEY.md §8d defines
                them, against the measured HBM peak (MEASURED_PEAKS.json)
  cpu_baseline  the reference's CPU path on this box's host cores (N = 1 only): C2/C5 = oracle/ref_port.c, the C/OpenMP
                restatement with the reference's per-phase thread structure (kind "port": the Rust crate cannot be
                built here, DESIGN.md §5); C1/C3/C4 = the numpy oracle on a stated slice
  parity        at-size check of THIS run's result against an independent path (f64 SIMT moments of the same frame /
                numpy f64 on a host slice / per-window and per-group definitions)

Other configs (BASELINE.json order): C1 lin_reg 100k x 4 f64 add_bias; C3 group_by 1e8 rows in ~1e4 groups x 8 f32;
C4 rolling_lin_reg window 1024 on 1e8 x 8 f32; C5 = one GPU's share (1.25e8 x 64 f32) of the 1e9 x 64 row-sharded fit.

N > 1 (torchrun, one process per GPU): every rank owns `rows` rows (weak scaling).  lin_reg (C2, C5): per step each
rank builds its partial moments, ONE all-reduce of the (p+2)^2 f64 moments over the library's own NCCL communicator
(pdsb_comm_init_rank / pdsb_dev_allreduce_f64) joins them, every rank solves redundantly and predicts its shard — in
the end-to-end leg too: each rank passes ITS host shard to the plugin symbol and the library fits ONE regression over
N x rows.  C3 / C4 shard without a collective (groups / rows with a read-only halo).
`--impl reference` times the CPU arm alone (rank 0 only), full-size steps.
`--dump-outputs DIR` writes what the last timed step returned (coefficients, status, per-row outputs) as DIR/<name>.npy,
at most 64 MB: per-row outputs longer than that keep a fixed seeded sample of rows.  Inputs are seeded, so two builds run
with the same arguments can be compared file for file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

CONFIGS = {
    # name: (rows per GPU, features, dtype, description)
    "C1": (100_000, 4, "f64", "pds.lin_reg 100k rows x 4 f64 features, add_bias=True (BASELINE configs[0])"),
    "C2": (100_000_000, 32, "f32", "pds.lin_reg 1e8 rows x 32 f32 features, add_bias=False, return_pred=True (BASELINE configs[1])"),
    "C3": (100_000_000, 8, "f32", "group_by(seg).agg(pds.lin_reg) ~1e4 groups x ~1e4 rows x 8 f32, add_bias=True (BASELINE configs[2])"),
    "C4": (100_000_000, 8, "f32", "pds.rolling_lin_reg window=1024 on 1e8 rows x 8 f32 (BASELINE configs[3])"),
    "C5": (125_000_000, 64, "f32", "pds.lin_reg 1e9 rows x 64 f32 row-sharded over 8 GPUs: one GPU's share = 1.25e8 rows "
                                   "(BASELINE configs[4]), return_pred=True"),
}
KW_LR = {"bias": False, "null_policy": "skip", "l1_reg": 0.0, "l2_reg": 0.0, "solver": "qr", "tol": 1e-5,
         "max_iter": 200, "weighted": False, "positive": False, "singular_x_tol": 1e-6}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--rows", type=int, default=None, help="rows per GPU (default: the config's)")
    ap.add_argument("--features", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-steps", type=int, default=3, help="passes of the CPU baseline inside the ours arm")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step computed as DIR/<name>.npy (rank 0)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    rows, feats, dtype, desc = CONFIGS[a.config]
    a.rows = a.rows or rows
    a.features = a.features or feats
    a.dtype = dtype
    a.desc = desc
    return a


class ClockSampler:
    """nvidia-smi sampler running during the timed region (B200_PROFILING.md clocks line)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int, uuid: str | None = None):
        self.index = index
        self.uuid = uuid          # "GPU-..." of the CUDA device in use: immune to CUDA_VISIBLE_DEVICES re-numbering
        self.samples = []
        self.proc = None
        self.nvml = []            # (sm_mhz, reason bitmask) every ~2 ms from NVML, when the library is loadable
        self.nvml_max = None
        self._run = False

    def _nvml_loop(self):
        # in-process NVML polling: nvidia-smi's own loop cannot go below ~100 ms, shorter than one default bench run
        try:
            import pynvml

            pynvml.nvmlInit()
            h = None
            if self.uuid:
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(self.uuid.encode() if isinstance(self.uuid, str) else self.uuid)
                except Exception:
                    h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.nvml_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            while self._run:
                mhz = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                try:
                    bits = int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                except Exception:
                    bits = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                self.nvml.append((mhz, bits))
                time.sleep(0.002)
        except Exception:
            pass

    def start(self):
        try:
            self._run = True
            self.nvml_thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.nvml_thread.start()
        except Exception:
            self._run = False
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        self._run = False
        try:
            out = self._stop_smi()
        except Exception as e:      # never let the sampler take the bench line down
            out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"sampler error: {e}"], "samples": 0}
        try:
            nv = list(self.nvml)
            smi_mhz = out.get("sm_mhz")
            nv_mhz = float(np.median([m for m, _ in nv])) if nv else None
            if len(nv) >= 3 and smi_mhz and abs(nv_mhz - smi_mhz) > 0.25 * smi_mhz:
                out["note"] = f"NVML samples ({nv_mhz:.0f} MHz) disagree with nvidia-smi; nvidia-smi reported"
            elif len(nv) >= 3:
                bits = 0
                for _, b in nv:
                    bits |= b
                names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
                reasons = set(out.get("reasons") or []) | {nm for m, nm in names.items() if bits & m}
                reasons.discard("nvidia-smi unavailable")
                out = {"sm_mhz": float(np.median([m for m, _ in nv])), "sm_max_mhz": self.nvml_max or out.get("sm_max_mhz"),
                       "reasons": sorted(reasons), "samples": len(nv), "source": "nvml (2 ms period) + nvidia-smi"}
        except Exception:
            pass
        return out

    def _stop_smi(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            parts = [x.strip() for x in s.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}




# ------------------------------------------------------------------------------------------------ helpers
def cpu_quota() -> float:
    """CPUs of the cgroup quota (cpu.max "quota period"), 0.0 when there is none."""
    try:
        a, b = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        return 0.0 if a == "max" else float(a) / float(b)
    except Exception:
        return 0.0


def host_threads() -> int:
    """Threads the CPU arm runs on: the cores this process may use — affinity mask, cut to the cgroup CPU quota when there
    is one (the B200 boxes report 128 cores under a 16-CPU quota; threads beyond the quota only get throttled).
    PDSB_BENCH_THREADS overrides."""
    if os.environ.get("PDSB_BENCH_THREADS"):
        return max(1, int(os.environ["PDSB_BENCH_THREADS"]))
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    q = cpu_quota()
    return max(1, min(n, int(q + 0.5))) if q >= 1.0 else n


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def committed_traffic(kernel: str, rows: int, p: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch from the committed `ncu --set full` capture of exactly
    this kernel and shape (profiles/traffic.json, written by profiles/ncu_traffic.py); None when no capture matches."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            for e in json.load(f):
                if e["kernel"] == kernel and e["rows"] == rows and e["features"] == p:
                    return e["dram_bytes"]
    except Exception:
        pass
    return None


def blas_threads(n):
    try:
        from threadpoolctl import threadpool_limits

        return threadpool_limits(limits=n)
    except Exception:
        import contextlib

        return contextlib.nullcontext()


def gen_host_lin_reg(rows, p, seed=208):
    """[y, x_0 .. x_{p-1}] float32 host columns, X ~ N(0,1), beta_j = ((j mod 7) - 3)/4, y = X beta + 0.1 N(0,1);
    columns are drawn by a thread pool (numpy releases the GIL) so 1e8 x 33 takes seconds, not a minute."""
    from concurrent.futures import ThreadPoolExecutor

    beta = ((np.arange(p) % 7) - 3.0) / 4.0
    cols = [np.empty(rows, dtype=np.float32) for _ in range(p + 1)]

    def fill(c):
        np.random.default_rng([seed, c]).standard_normal(rows, dtype=np.float32, out=cols[c])

    with ThreadPoolExecutor(max_workers=min(host_threads(), p + 1)) as ex:
        list(ex.map(fill, range(p + 1)))
    y = cols[0]
    y *= np.float32(0.1)
    blk = 1 << 22
    for s in range(0, rows, blk):
        e = min(rows, s + blk)
        acc = np.zeros(e - s, dtype=np.float32)
        for j in range(p):
            acc += np.float32(beta[j]) * cols[1 + j][s:e]
        y[s:e] += acc
    return cols


def cpu_lin_reg_port(cols, steps, warmup):
    """oracle/ref_port.c: the reference's pl_lr_pred_f32 data passes with its per-phase thread structure."""
    from oracle import ref_port

    ref_port.set_threads(host_threads())          # torchrun exports OMP_NUM_THREADS=1: ask for the cores explicitly
    for _ in range(max(0, warmup)):
        ref_port.lr_pred_f32(cols)
    tot, phases = 0.0, {}
    for _ in range(steps):
        c, pred, resid, t = ref_port.lr_pred_f32(cols)
        tot += t["total"]
        for k, v in t.items():
            phases[k] = phases.get(k, 0.0) + v / steps
    assert c is not None and len(pred) == len(cols[0])
    dt = tot / steps
    return len(cols[0]) / dt, dt, phases, ref_port.threads()


def lin_reg_workload(args):
    return (f"{args.desc}: {args.rows} rows x {args.features} {args.dtype} features per GPU; "
            f"step = moments + solve + predict/resid")


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args, rank):
    """The CPU arm alone, rank 0 only.  C2 / C5: ref_port.c at the config's full per-GPU size (same_config)."""
    if rank != 0:
        return
    cores = host_threads()
    if args.config in ("C2", "C5"):
        cols = gen_host_lin_reg(args.rows, args.features)
        v, dt, phases, thr = cpu_lin_reg_port(cols, args.steps, args.warmup)
        sample = (f"{args.steps} full-size steps of {args.rows} rows x {args.features} f32 through oracle/ref_port.c "
                  f"(C/OpenMP restatement of pl_lr_pred_f32; pack, resid and the output copies run on ONE thread as in the "
                  f"reference, Gram / X'y / predict on {thr} threads), {dt:.2f} s each; phases " +
                  ", ".join(f"{k} {s_:.2f}s" for k, s_ in phases.items() if k != "total"))
        cfg = {"workload": lin_reg_workload(args), "rows_per_gpu": args.rows, "features": args.features, "same_config": True}
        metric = "lin_reg rows/sec (f32, return_pred=True)"
    else:
        v, dt, sample, cores = cpu_other(args, args.steps, args.warmup)
        cfg = {"workload": f"{args.desc}", "rows_per_gpu": args.rows, "features": args.features}
        metric = METRICS[args.config]
    line = {"impl": "reference", "metric": metric, "value": v, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.dtype, "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": "rows/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


METRICS = {"C1": "lin_reg rows/sec (f64, add_bias, coefficients)", "C2": "lin_reg rows/sec (f32, return_pred=True)",
           "C3": "group_by lin_reg rows/sec (f32, ~1e4 groups)", "C4": "rolling_lin_reg rows/sec (f32, window 1024)",
           "C5": "lin_reg rows/sec (f32, return_pred=True)"}


def cpu_other(args, steps, warmup, host=None):
    """numpy-oracle CPU arm of C1 / C3 / C4 on a stated slice.  Returns (rows/s, s per step, sample text, cores)."""
    from oracle import lin_reg_oracle as orc

    p = args.features
    rng = np.random.default_rng(208)
    if args.config == "C1":
        n = args.rows
        X = rng.standard_normal((p, n))
        y = np.array([0.5, -0.25, 0.75, 0.1][:p] + [0.0] * max(0, p - 4)) @ X + 0.5 + 0.1 * rng.standard_normal(n)
        cols = [orc.Col("y", y)] + [orc.Col(f"x{i}", X[i]) for i in range(p)]
        kw = dict(KW_LR, bias=True, singular_x_tol=1e-12)
        with blas_threads(host_threads()):
            for _ in range(max(1, warmup)):
                orc.pl_lr(cols, kw, f32=False)
            t0 = time.perf_counter()
            for _ in range(steps):
                orc.pl_lr(cols, kw, f32=False)
            dt = (time.perf_counter() - t0) / steps
        return n / dt, dt, (f"{steps} full-size passes of oracle.pl_lr (numpy/OpenBLAS, up to {host_threads()} BLAS "
                            f"threads) on {n} x {p} f64 + bias, {dt * 1e3:.2f} ms each"), host_threads()
    if args.config == "C3":
        n_groups, gl = 200, 10_000
        kw = dict(KW_LR, bias=True)
        data = [(rng.standard_normal((p, gl), dtype=np.float32), rng.standard_normal(gl, dtype=np.float32)) for _ in range(n_groups)]
        with blas_threads(1):
            t0 = time.perf_counter()
            for _ in range(max(1, steps)):
                for X, y in data:
                    orc.pl_lr([orc.Col("y", y)] + [orc.Col(f"x{i}", X[i]) for i in range(p)], kw, f32=True)
            dt = (time.perf_counter() - t0) / max(1, steps)
        rows = n_groups * gl
        return rows / dt, dt, (f"oracle.pl_lr once per group (what Polars does with the plugin) on {n_groups} groups x {gl} rows "
                               f"x {p} f32, ONE thread, {dt:.2f} s per pass; the reference spreads groups over its rayon pool, "
                               f"so its ceiling is this times the core count"), 1
    # C4: the reference's rolling path is a sequential Woodbury walk on one thread (lr_online_solvers.rs:201-210)
    n = min(args.rows, 200_000)
    X = rng.standard_normal((p, n), dtype=np.float32)
    y = rng.standard_normal(n, dtype=np.float32)
    cols = [orc.Col("y", y)] + [orc.Col(f"x{i}", X[i]) for i in range(p)]
    kw = {"null_policy": "raise", "n": 1024, "bias": False, "lambda": 0.0, "min_size": min(p, 1024)}
    with blas_threads(1):
        t0 = time.perf_counter()
        for _ in range(steps):
            orc.pl_rolling_lr(cols, kw, f32=True)
        dt = (time.perf_counter() - t0) / steps
    return n / dt, dt, (f"oracle.pl_rolling_lr (sequential Woodbury walk like faer_rolling_lr, ONE thread as in the reference) on "
                        f"a {n}-row slice x {p} f32, window 1024, {dt:.2f} s per pass; the walk is O(n), so rows/s carries to 1e8"), 1


# ------------------------------------------------------------------------------------------------ ours arm
class Ctx:
    pass


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist

    from polars_ds_extension_b200 import parallel
    from polars_ds_extension_b200._lib import check, lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    check(lib().pdsb_set_device(local_rank))
    c = Ctx()
    c.torch, c.dist, c.args, c.rank, c.local_rank, c.world = torch, dist, args, rank, local_rank, world
    c.device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=c.device)
        parallel.init_world()           # the library's own NCCL communicator (include/pdsb.h, pdsb_comm_init_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_ok(flag):
        torch.cuda.synchronize()
        if world == 1:
            return bool(flag)
        t = torch.tensor([1.0 if flag else 0.0], dtype=torch.float64, device=c.device)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return float(t.item()) > 0.5

    def max_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], dtype=torch.float64, device=c.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    c.barrier, c.all_ok, c.max_over_ranks = barrier, all_ok, max_over_ranks
    w = {"C1": setup_c1, "C2": setup_lin_reg, "C5": setup_lin_reg, "C3": setup_grouped, "C4": setup_rolling}[args.config](c)

    from polars_ds_extension_b200 import device as dev

    warm = max(args.warmup, 3)
    for _ in range(warm):
        w["step"]()
    barrier()
    gpu_uuid = None
    try:
        u = str(torch.cuda.get_device_properties(c.device).uuid)
        gpu_uuid = u if u.startswith("GPU-") else "GPU-" + u
    except Exception:
        gpu_uuid = None
    sampler = ClockSampler(local_rank, gpu_uuid)
    if rank == 0:
        sampler.start()
    launches0 = dev.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        w["step"]()
    ev1.record()
    barrier()
    launches = dev.launch_count() - launches0
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, w["outputs"]())
    rows = args.rows
    value = rows * world * args.steps / (ms * 1e-3)

    # ---- roofline of the dominant kernel, timed alone on the launching stream ----
    for _ in range(3):
        w["kernel"]()
    torch.cuda.synchronize()
    reps = max(args.steps, 5)
    ev0.record()
    for _ in range(reps):
        w["kernel"]()
    ev1.record()
    torch.cuda.synchronize()
    k_ms = ev0.elapsed_time(ev1) / reps
    peak, peak_src = hbm_peak()
    achieved = w["alg_bytes"] / (k_ms * 1e-3) / 1e9
    parity = w["parity"]() if "parity" in w else None

    e2e = None
    if not args.no_e2e:
        e2e = w["e2e"]()
        if world > 1:                                   # unconditional on every rank (value None -> contributes 0)
            t_e = max_over_ranks(e2e["ms_per_step"] if e2e.get("value") else 0.0)
            if e2e.get("value"):
                e2e["ms_per_step"] = t_e
                e2e["value"] = rows * world / (t_e * 1e-3)
                e2e["h2d_bytes_per_step"] *= world
                e2e["d2h_bytes_per_step"] *= world
    cpu = None
    if rank == 0 and not args.no_cpu and world == 1:
        cpu = w["cpu"]()

    if rank == 0:
        cfg = dict(w["config"])
        cfg.update({"rows_per_gpu": rows, "features": args.features,
                    "parallelism": w.get("parallelism", "single GPU") if world > 1 else "single GPU",
                    "l2_policy": w.get("l2_policy", "inputs are larger than L2 (126 MB); no explicit flush")})
        line = {"metric": METRICS[args.config], "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps,
                "warmup": warm, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": args.dtype, "data": "synthetic", "config": cfg, "e2e": e2e,
                "gpu_launches": launches, "clocks": clocks,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": w.get("traffic"), "kernel": w["kernel_name"], "kernel_ms": k_ms,
                             "algorithmic_bytes": w["alg_bytes"], "peak_source": peak_src},
                "cpu_baseline": cpu, "parity": parity}
        print(json.dumps(line), flush=True)
    if world > 1:
        parallel.destroy_world()
        dist.destroy_process_group()


# ---------------------------------------------------------------- e2e through the plugin symbol (host buffers)
def plugin_e2e(c, symbol, make_inputs, names, kw, check_len, h2d_bytes, d2h_bytes, api):
    """Time `_polars_plugin_<symbol>` with host Arrow buffers: pageable first (the headline), then pinned.
    `all_ok` is a collective AND over the ranks; every rank calls it the same number of times whatever happens locally."""
    import pyarrow as pa

    from polars_ds_extension_b200 import _harness

    torch, args = c.torch, c.args
    out = {"value": None, "unit": "rows/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
           "api": api + " (Arrow C data, PAGEABLE host buffers)"}
    k = max(1, args.e2e_steps)
    for kind in ("pageable", "pinned"):
        err, inputs, dt = None, None, None
        try:
            inputs = [pa.array(a) for a in make_inputs(kind == "pinned")]      # zero-copy views of the host buffers
            for _ in range(2):                                              # warm-up (result pool, staging ring)
                res = _harness.call_plugin(symbol, inputs, names, kw)
                del res
        except Exception as e:  # noqa: BLE001
            err = f"{type(e).__name__}: {e}"
        if not c.all_ok(err is None):                                       # collective: also the start barrier
            out.setdefault("error", err or "the end-to-end leg failed on another rank")
            break
        try:
            t0 = time.perf_counter()
            for _ in range(k):
                res = _harness.call_plugin(symbol, inputs, names, kw)
                assert len(res) == check_len
                del res
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / k
        except Exception as e:  # noqa: BLE001
            err = f"{type(e).__name__}: {e}"
        if not c.all_ok(err is None):
            out.setdefault("error", err or "the end-to-end leg failed on another rank")
            break
        if kind == "pageable":
            out.update({"value": args.rows / dt, "ms_per_step": dt * 1e3, "steps": k,
                        "staged_bytes_per_step": int(lib_().pdsb_last_staged_bytes())})
        else:
            out["pinned_value"] = args.rows / c.max_over_ranks(dt) * c.world
            out["pinned_ms_per_step"] = dt * 1e3
        del inputs
    return out


def lib_():
    from polars_ds_extension_b200._lib import lib

    return lib()


def host_copy(torch, dev_rows, pinned):
    """Host copies of device rows (list of 1-D tensors), pageable or pinned, as numpy arrays."""
    out = []
    for r in dev_rows:
        h = torch.empty(r.shape, dtype=r.dtype, pin_memory=pinned)
        h.copy_(r)
        out.append(h.numpy())
    torch.cuda.synchronize()
    return out


DUMP_BYTES = 60 << 20       # --dump-outputs stays under 64 MB in all, .npy headers included


def dump_outputs(dirname, outputs, seed=208):
    """Write `outputs` (name -> device tensor, rows on the first axis) as DIR/<name>.npy: float64 tensors as float64,
    every other dtype as float32.  When the longest arrays do not fit DUMP_BYTES, all arrays of that length keep the same
    seeded sample of rows (sorted), so two runs with the same arguments write files that compare row for row."""
    import torch

    def size(v):
        return 8 if v.dtype == torch.float64 else 4

    os.makedirs(dirname, exist_ok=True)
    n = max(v.shape[0] for v in outputs.values())
    fixed = sum(v.numel() * size(v) for v in outputs.values() if v.shape[0] != n)
    per_row = sum(v[0].numel() * size(v) for v in outputs.values() if v.shape[0] == n)
    k = (DUMP_BYTES - fixed) // per_row
    sample = torch.from_numpy(np.unique(np.random.default_rng(seed).integers(0, n, k))) if n > k else None
    for name, v in outputs.items():
        if sample is not None and v.shape[0] == n:
            v = v.index_select(0, sample.to(v.device))
        np.save(os.path.join(dirname, f"{name}.npy"), v.cpu().numpy().astype(np.float64 if size(v) == 8 else np.float32))


# ---------------------------------------------------------------- C2 / C5: lin_reg, return_pred
def setup_lin_reg(c):
    from polars_ds_extension_b200 import device as dev
    from polars_ds_extension_b200._lib import METHOD_LSTSQ, check

    torch, args = c.torch, c.args
    rows, p, device = args.rows, args.features, c.device
    L = lib_()
    g = torch.Generator(device=device)
    g.manual_seed(208 + c.rank)
    ld = (rows + 31) // 32 * 32
    Z = torch.zeros((p + 1, ld), dtype=torch.float32, device=device)      # column-major [X | y]
    X, y = Z[:p], Z[p:]
    bt = ((torch.arange(p, device=device) % 7).float() - 3.0) / 4.0
    for j in range(p):
        X[j, :rows].normal_(generator=g)
    for s in range(0, rows, 1 << 24):
        e = min(rows, s + (1 << 24))
        y[0, s:e] = bt @ X[:, s:e]
    noise = torch.empty(rows, dtype=torch.float32, device=device).normal_(generator=g)
    y[0, :rows] += 0.1 * noise
    del noise
    host = {}
    if not c.args.no_e2e or not c.args.no_cpu:
        host["pageable"] = host_copy(torch, [y[0, :rows]] + [X[j, :rows] for j in range(p)], False)
    frame = dev.to_frame(Z, n=rows)                                      # the library's resident layout (include/pdsb.h)
    torch.cuda.synchronize()
    del X, y, Z
    torch.cuda.empty_cache()
    ncols, q1 = p + 1, p + 2
    M = torch.empty((q1, q1), dtype=torch.float64, device=device)
    beta = torch.empty((1, p), dtype=torch.float64, device=device)
    status = torch.zeros(4, dtype=torch.int32, device=device)
    pred = torch.empty((1, ld), dtype=torch.float32, device=device)
    resid = torch.empty((1, ld), dtype=torch.float32, device=device)
    tol = 1e-6  # default singular_x_tol of the f32 family (expr_linear.py:184-186)

    def step():
        dev.moments_frame(frame, rows, ncols, 0, p, p, 1, out=M)
        if c.world > 1:   # the only exchange of the row-sharded path: (p+2)^2 f64 partial moments over NCCL / NVLink
            check(L.pdsb_dev_allreduce_f64(M.data_ptr(), q1 * q1, torch.cuda.current_stream().cuda_stream))
        dev.solve(M, p, 1, add_bias=False, method=METHOD_LSTSQ, singular_x_tol=tol, beta=beta, status=status)
        dev.predict_frame(frame, rows, ncols, 0, p, p, 1, beta, status, False, pred, resid)

    def kernel():
        dev.moments_frame(frame, rows, ncols, 0, p, p, 1, out=M)

    def parity():
        """This run's coefficients / predictions against paths that share nothing with the tcgen05 kernel:
        (1) moments of the SAME resident frame by the SIMT kernel (exact f32 products, f64 accumulation) -> same solve;
        (2) numpy float64 predictions on a host slice; (3) the generating beta."""
        step()
        torch.cuda.synchronize()
        b_tc = beta.cpu().numpy()[0].copy()
        path = int(L.pdsb_last_moments_path())
        L.pdsb_set_moments_path(1)
        try:
            M2 = dev.moments_frame(frame, rows, ncols, 0, p, p, 1)
            if c.world > 1:
                check(L.pdsb_dev_allreduce_f64(M2.data_ptr(), q1 * q1, torch.cuda.current_stream().cuda_stream))
            b2, _ = dev.solve(M2, p, 1, add_bias=False, method=METHOD_LSTSQ, singular_x_tol=tol)
            b_simt = b2.cpu().numpy()[0]
        finally:
            L.pdsb_set_moments_path(0)
        out = {"moments_path": "tcgen05" if path == 1 else "simt",
               "coef_rel_err_vs_f64_accumulated_simt_moments": float(np.max(np.abs(b_tc - b_simt)) / np.max(np.abs(b_simt))),
               "coef_max_abs_err_vs_generating_beta": float(np.max(np.abs(b_tc - ((np.arange(p) % 7) - 3.0) / 4.0))),
               "tolerance": "1e-4 relative (north_star, f32)"}
        if "pageable" in host:
            m = min(rows, 1_000_000)
            hx = np.stack([a[:m] for a in host["pageable"][1:]]).astype(np.float64)
            ref = b_simt @ hx
            got = pred[0, :m].cpu().numpy().astype(np.float64)
            out["pred_rel_err_vs_numpy_f64_first_1e6_rows"] = float(np.max(np.abs(got - ref)) / np.max(np.abs(ref)))
        return out

    def e2e():
        def make(pinned):
            if pinned and "pinned" not in host:
                host["pinned"] = []
                for a in host["pageable"]:
                    t = torch.empty(a.shape, dtype=torch.float32, pin_memory=True)
                    t.numpy()[:] = a
                    host["pinned"].append(t.numpy())
            return host["pinned" if pinned else "pageable"]

        names = ["y"] + [f"x{i}" for i in range(p)]
        api = "_polars_plugin_pl_lr_pred_f32"
        if c.world > 1:
            api += f", collective over {c.world} ranks: ONE fit over {c.world} x {rows} rows, moments all-reduced inside the library"
        return plugin_e2e(c, "pl_lr_pred_f32", make, names, KW_LR, rows, (p + 1) * rows * 4, 2 * rows * 4, api)

    def cpu():
        v, dt, phases, thr = cpu_lin_reg_port(host["pageable"], max(1, args.cpu_steps), 1)
        return {"value": v, "unit": "rows/s", "cores": thr, "kind": "port",
                "sample": f"{max(1, args.cpu_steps)} full-size passes ({rows} rows x {p} f32) of oracle/ref_port.c, {dt:.2f} s each; "
                          "thread structure per phase as in the reference (pack / resid / output copies: 1 thread; Gram, X'y, "
                          f"predict: {thr} threads); phases " + ", ".join(f"{k} {s_:.2f}s" for k, s_ in phases.items() if k != "total")}

    def outputs():
        return {"coeffs": beta[0], "status": status[:1], "pred": pred[0, :rows], "resid": resid[0, :rows]}

    path_name = "tcgen05+TMA 3xTF32"
    return {"step": step, "kernel": kernel, "outputs": outputs, "alg_bytes": rows * (p + 1) * 4,
            "kernel_name": "moments (Gram X'X | X'y)",
            "traffic": committed_traffic("moments_frame", rows, p), "parity": parity, "e2e": e2e, "cpu": cpu,
            "parallelism": f"row-sharded x{c.world}, one f64 moments all-reduce per step (library NCCL communicator)",
            "config": {"workload": lin_reg_workload(args), "moments_kernel": path_name,
                       "resident_layout": "row-blocked frame [block][column][128] (library native, include/pdsb.h)"}}


# ---------------------------------------------------------------- C1: lin_reg 100k x 4 f64 + bias, coefficients only
def setup_c1(c):
    from polars_ds_extension_b200 import device as dev
    from polars_ds_extension_b200._lib import METHOD_LSTSQ

    torch, args = c.torch, c.args
    n, p, device = args.rows, args.features, c.device
    rng = np.random.default_rng(208)
    Xh = rng.standard_normal((p, n))
    bt = np.array(([0.5, -0.25, 0.75, 0.1] * ((p + 3) // 4))[:p])
    yh = bt @ Xh + 0.5 + 0.1 * rng.standard_normal(n)
    ld = (n + 31) // 32 * 32
    Z = torch.zeros((p + 1, ld), dtype=torch.float64, device=device)
    Z[:p, :n] = torch.from_numpy(Xh).to(device)
    Z[p, :n] = torch.from_numpy(yh).to(device)
    X, Y = Z[:p], Z[p:]
    q1 = p + 2
    M = torch.empty((q1, q1), dtype=torch.float64, device=device)
    beta = torch.empty((1, p + 1), dtype=torch.float64, device=device)
    status = torch.zeros(4, dtype=torch.int32, device=device)

    def step():
        dev.moments(X, Y, n=n, out=M)
        dev.solve(M, p, 1, add_bias=True, method=METHOD_LSTSQ, singular_x_tol=1e-12, beta=beta, status=status)

    def kernel():
        dev.moments(X, Y, n=n, out=M)

    def parity():
        step()
        ref, *_ = np.linalg.lstsq(np.column_stack([Xh.T, np.ones(n)]), yh, rcond=None)
        got = beta.cpu().numpy()[0]
        return {"coef_rel_err_vs_numpy_lstsq_f64": float(np.max(np.abs(got - ref)) / np.max(np.abs(ref))),
                "tolerance": "1e-6 relative (north_star, f64)"}

    def e2e():
        cols = [yh] + [np.ascontiguousarray(Xh[i]) for i in range(p)]
        kw = dict(KW_LR, bias=True, singular_x_tol=1e-12)
        c.args.e2e_steps = max(c.args.e2e_steps, 50)
        return plugin_e2e(c, "pl_lr", lambda pinned: cols, ["y"] + [f"x{i}" for i in range(p)], kw, 1,
                          (p + 1) * n * 8, (p + 1) * 8, "_polars_plugin_pl_lr (latency-bound: ~4 MB in, 40 B out)")

    def cpu():
        v, dt, sample, cores = cpu_other(args, 50, 3)
        return {"value": v, "unit": "rows/s", "cores": cores, "kind": "port", "sample": sample}

    return {"step": step, "kernel": kernel, "outputs": lambda: {"coeffs": beta[0], "status": status[:1]},
            "alg_bytes": n * (p + 1) * 8, "kernel_name": "moments f64 (K2a)", "parity": parity,
            "e2e": e2e, "cpu": cpu, "l2_policy": "4 MB of input: L2-resident after the first step, latency-bound by design",
            "config": {"workload": f"{args.desc}; step = moments + solve (coefficients)"}}


# ---------------------------------------------------------------- C3: group_by lin_reg (batched)
def setup_grouped(c):
    from polars_ds_extension_b200 import device as dev

    torch, args = c.torch, c.args
    n, p, device = args.rows, args.features, c.device
    g = torch.Generator(device=device)
    g.manual_seed(208 + c.rank)
    Z = torch.randn((p + 1, n), device=device, generator=g)
    Z[p] += (Z[:p] * 0.25).sum(0)
    sizes = torch.randint(8000, 12001, (int(n / 10000) + 2,), generator=torch.Generator().manual_seed(1 + c.rank))
    offs = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(sizes, 0)])
    offs = offs[offs < n]
    offs_h = torch.cat([offs, torch.tensor([n])])
    offs_d = offs_h.to(device)
    ng = offs_h.numel() - 1
    state = {}

    def step():
        state["out"] = dev.grouped_lin_reg(Z[:p], Z[p], offs_d, add_bias=True, singular_x_tol=1e-6)

    def parity():
        step()
        beta = state["out"][0].cpu().numpy()
        rng = np.random.default_rng(0)
        worst = 0.0
        for gi in rng.integers(0, ng, 50):
            a, b = int(offs_h[gi]), int(offs_h[gi + 1])
            Xg = np.column_stack([Z[:p, a:b].double().T.cpu().numpy(), np.ones(b - a)])
            ref, *_ = np.linalg.lstsq(Xg, Z[p, a:b].double().cpu().numpy(), rcond=None)
            worst = max(worst, float(np.max(np.abs(beta[gi] - ref)) / np.max(np.abs(ref))))
        return {"coef_rel_err_vs_numpy_lstsq_f64_50_random_groups": worst, "groups": ng, "tolerance": "1e-4 relative (f32)"}

    def e2e():
        host = {}

        def make(pinned):
            key = "pinned" if pinned else "pageable"
            if key not in host:
                host[key] = [offs_h.numpy()] + host_copy(torch, [Z[p]] + [Z[j] for j in range(p)], pinned)
            return host[key]

        kw = dict(KW_LR, bias=True)
        return plugin_e2e(c, "pl_lr_by_f32", make, ["offsets", "y"] + [f"x{i}" for i in range(p)], kw, ng,
                          (p + 1) * n * 4 + (ng + 1) * 8, ng * (p + 1) * 4,
                          "_polars_plugin_pl_lr_by_f32 (additive batched group_by entry, one launch sequence for all groups)")

    def cpu():
        v, dt, sample, cores = cpu_other(args, 1, 0)
        return {"value": v, "unit": "rows/s", "cores": cores, "kind": "port", "sample": sample}

    return {"step": step, "kernel": step, "outputs": lambda: dict(zip(("coeffs", "status"), state["out"])),
            "alg_bytes": n * (p + 1) * 4, "kernel_name": "grouped moments + batched solve (K5)",
            "parity": parity, "e2e": e2e, "cpu": cpu, "parallelism": f"groups partitioned over {c.world} ranks, no collective",
            "config": {"workload": f"{args.desc}; {ng} groups of 8000..12000 rows; step = per-group moments + batched solve"}}


# ---------------------------------------------------------------- C4: rolling_lin_reg window 1024
def setup_rolling(c):
    from polars_ds_extension_b200 import device as dev

    torch, args = c.torch, c.args
    n, p, device = args.rows, args.features, c.device
    W = 1024
    g = torch.Generator(device=device)
    g.manual_seed(208 + c.rank)
    Z = torch.randn((p + 1, n), device=device, generator=g)
    Z[p] += (Z[:p] * 0.25).sum(0)
    coeffs = torch.empty((n, p), dtype=torch.float32, device=device)
    pred = torch.empty(n, dtype=torch.float32, device=device)
    valid = torch.empty(n, dtype=torch.uint8, device=device)

    def step():
        dev.online_lin_reg(Z[:p], Z[p], W, p, coeffs=coeffs, pred=pred, valid=valid)

    def parity():
        step()
        rng = np.random.default_rng(0)
        worst = 0.0
        rows = rng.integers(W, n, 1000)
        for j in rows:
            j = int(j)
            Xw = Z[:p, j - W + 1:j + 1].double().T.cpu().numpy()
            yw = Z[p, j - W + 1:j + 1].double().cpu().numpy()
            ref = np.linalg.solve(Xw.T @ Xw, Xw.T @ yw)
            worst = max(worst, float(np.max(np.abs(coeffs[j].cpu().numpy() - ref)) / np.max(np.abs(ref))))
        return {"coef_rel_err_vs_per_window_ols_f64_1000_random_rows": worst, "tolerance": "1e-4 relative (f32)"}

    def e2e():
        host = {}

        def make(pinned):
            key = "pinned" if pinned else "pageable"
            if key not in host:
                host[key] = host_copy(torch, [Z[p]] + [Z[j] for j in range(p)], pinned)
            return host[key]

        kw = {"null_policy": "raise", "n": W, "bias": False, "lambda": 0.0, "min_size": min(p, W)}
        c.args.e2e_steps = min(c.args.e2e_steps, 2)
        return plugin_e2e(c, "pl_rolling_lr_f32", make, ["y"] + [f"x{i}" for i in range(p)], kw, n,
                          (p + 1) * n * 4, n * (p * 4 + 4 + 1), "_polars_plugin_pl_rolling_lr_f32")

    def cpu():
        v, dt, sample, cores = cpu_other(args, 1, 0)
        return {"value": v, "unit": "rows/s", "cores": cores, "kind": "port", "sample": sample}

    return {"step": step, "kernel": step, "outputs": lambda: {"coeffs": coeffs, "pred": pred, "valid": valid},
            "alg_bytes": n * ((p + 1) * 4 + p * 4 + 4 + 1),
            "kernel_name": "rolling window moments + per-row solve (K6, 3 launches)", "parity": parity, "e2e": e2e, "cpu": cpu,
            "parallelism": f"rows partitioned over {c.world} ranks (+ a read-only halo of window-1 rows), no collective",
            "config": {"workload": f"{args.desc}; step = chain sums + scan + per-row window solve, writes coeffs/pred/valid"}}


if __name__ == "__main__":
    main()
