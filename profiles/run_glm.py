"""GLM (IRLS) timing on a resident 1e8-row f64 problem: the whole `device.glm` fit, one fused IRLS iteration, and the
existing weighted moments kernel on the same X (the least any unfused iteration must read: X, z and w), for p = 8, 32, 64
and the Poisson and binomial families.

    python profiles/run_glm.py [rows] [out.txt]

Timing: CUDA events after warm-up.  One iteration = (fit with max_iter = 1 + K) - (fit with max_iter = 1), divided by K,
with tol = 0 so no fit stops early: the fused moments pass, the K3 solve and the per-iteration download + synchronise.
The fused iteration and the weighted moments alternate, REPS times each.  X (p x n) is larger than the 126 MB L2 at
every p.  A torch.profiler pass at the end gives the kernel-only times.  Bytes per row are what the algorithm must
read: fused (p + 1) * 8 (X, y), weighted moments (p + 2) * 8 (X, z, w); shares are of the 6570 GB/s HBM read rate
DESIGN.md uses as the peak.
"""
import subprocess
import sys

import torch

sys.path.insert(0, ".")
from polars_ds_extension_b200 import device as dev  # noqa: E402

HBM = 6570e9
rows = int(float(sys.argv[1])) if len(sys.argv) > 1 else 100_000_000
out_path = sys.argv[2] if len(sys.argv) > 2 else None
REPS, K = 5, 4
lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def timed(fn, reps=1):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps * 1e-3


say(f"device: {gpu_info()}")
say(f"rows = {rows:.0e}, f64, resident; repeats = {REPS}, iterations per differenced fit = {K}")
ld = (rows + 31) // 32 * 32
gen = torch.Generator(device="cuda").manual_seed(2026)
Xall = torch.randn((64, ld), dtype=torch.float64, device="cuda", generator=gen).mul_(0.125)   # var(eta) = p / 64
y = torch.empty(ld, dtype=torch.float64, device="cuda")
w = torch.rand((1, ld), dtype=torch.float64, device="cuda", generator=gen).add_(0.5)
z = torch.empty((1, ld), dtype=torch.float64, device="cuda")
say(f"{'family':9s} {'p':>3s} {'n_iter':>6s} {'fit ms':>9s} {'iter ms':>9s} {'wmom ms':>9s} {'iter/wmom':>9s} "
    f"{'B/row it':>8s} {'%HBM it':>7s} {'%HBM wm':>7s} {'host ms':>8s}")
for p in (8, 32, 64):
    X = Xall[:p]
    eta = torch.linspace(-1.0, 1.0, p, dtype=torch.float64, device="cuda") @ X + 0.2
    for family in ("poisson", "binomial"):
        y.copy_(torch.poisson(torch.exp(eta), generator=gen) if family == "poisson"
                else torch.bernoulli(torch.sigmoid(eta), generator=gen))
        z.copy_(y.view(1, -1))
        fit = lambda: dev.glm(X, y, family, add_bias=True, max_iter=100, tol=1e-8, n=rows)
        fit1 = lambda: dev.glm(X, y, family, add_bias=True, max_iter=1, tol=0.0, n=rows)
        fitk = lambda: dev.glm(X, y, family, add_bias=True, max_iter=1 + K, tol=0.0, n=rows)
        wmom = lambda: dev.moments(X, z, n=rows, w=w)
        _, n_iter = fit()                                   # warm-up of every shape the timed window uses
        fit1(); fitk(); wmom()
        torch.cuda.synchronize()
        t_fit = min(timed(fit) for _ in range(2))
        it_t, wm_t = [], []
        for _ in range(REPS):                               # alternate the two
            it_t.append((timed(fitk) - timed(fit1)) / K)
            wm_t.append(timed(wmom))
        t_it, t_wm = sorted(it_t)[REPS // 2], sorted(wm_t)[REPS // 2]
        b_it, b_wm = (p + 1) * 8, (p + 2) * 8
        say(f"{family:9s} {p:3d} {n_iter:6d} {t_fit * 1e3:9.2f} {t_it * 1e3:9.3f} {t_wm * 1e3:9.3f} {t_it / t_wm:9.2f} "
            f"{b_it:8d} {100 * b_it * rows / t_it / HBM:7.1f} {100 * b_wm * rows / t_wm / HBM:7.1f} "
            f"{(t_fit - n_iter * t_it) * 1e3:8.2f}")
        say(f"    spread: iteration {min(it_t) * 1e3:.3f}..{max(it_t) * 1e3:.3f} ms, "
            f"weighted moments {min(wm_t) * 1e3:.3f}..{max(wm_t) * 1e3:.3f} ms")
    del eta

# kernel-only times: one fit of K + 1 iterations and one weighted-moments call per p
say()
say("kernel times (torch.profiler, CUDA activity, mean per launch; binomial, the last y above):")
from torch.profiler import ProfilerActivity, profile  # noqa: E402

for p in (8, 32, 64):
    X = Xall[:p]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        dev.glm(X, y, "binomial", add_bias=True, max_iter=1 + K, tol=0.0, n=rows)
        dev.moments(X, z, n=rows, w=w)
        torch.cuda.synchronize()
    for ev in prof.key_averages():
        if "gram_dmma_side" in ev.key or "solve" in ev.key:
            name = "fused GLM side kernel" if "GlmRows" in ev.key else ("weighted side kernel" if "side" in ev.key else ev.key[:40])
            t = getattr(ev, "device_time", 0.0) or getattr(ev, "cuda_time", 0.0)
            if t:
                say(f"  p = {p:2d}  {name:28s} x{ev.count:2d}  {t / 1e3:8.3f} ms")

if out_path:
    with open(out_path, "w") as f:
        f.write("\n".join(lines) + "\n")
