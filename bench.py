#!/usr/bin/env python
"""bench.py -- Helmholtz source-solves/sec on the BASELINE.json headline configuration.

Workload (BASELINE.json configs[2], the one the metric is quoted on; fits one GPU):
  synthetic 512 x 512 grid, 256-element ring (256 one-hot sources, 193 receivers kept per source),
  16 frequencies linspace(300, 596) kHz, complex64.  One STEP = one evaluation of the joint
  (loss, grad) = per frequency: assemble + factorise + all-source forward sweeps + source estimate /
  residual / loss + all-source adjoint sweeps on the same factors + gradient; frequencies are sharded
  over the ranks and the packed (grad, loss) is all-reduced once.  Units per step = source-solves =
  nfreq x nsrc x 2 (forward + adjoint), factorisation amortised into them.  --gpus N shards the SAME 16-frequency sweep
  over N ranks (BASELINE configs[2] as stated: "strong" scaling, 16 / N frequencies per GPU); with N > 1 the line also
  carries `weak_scaling`: the rate with 16 frequencies kept on every GPU (a 16*N-frequency objective over the same band).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
  (N>1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

`value`  : device-resident inputs, CUDA events, max over ranks.
`e2e`    : same step through the C-ABI host entry ust_fwi_loss_grad_host (the call a reference maintainer binds):
           pinned HOST slowness + observed data copied host->device and (loss, grad) read back device->host inside
           the call (N > 1: ShardedFWI.loss_grad_host = the same copies through torch + the NCCL all-reduce).
`roofline`: the kernel class with the largest share of the step, per-launch CUDA-event timing from ust_profile on
           one extra step (run as a single launch chain so that per-launch times do not overlap);
           `step_roofline`: algorithmic flops of the whole step / ms_per_step against the same peak;
           `cpu_baseline`: the oracle's SciPy/SuperLU path on a bounded sample on the host cores.
`--impl reference`: the reference's CPU algorithm (oracle port; JAX is not installable here) on all host
           cores, one process per frequency, bounded sample per step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "helmholtz_source_solves_per_sec"
# dram__bytes_read.sum + dram__bytes_write.sum per launch at the default workload from `ncu --set full` captures:
#   sweep_gemm: profiles/ncu_tc2_sweep_r01.txt (a back-substitution launch, all 256 tiles live: 185.7 MB read + 20.0 MB
#               written; operand planes + C of such a launch are 218 MB, nothing is re-read from HBM)
#   gj_update : profiles/ncu_tc2_update_r01.txt (32 matrices updated in place: 64 MB of X read + written, planes emitted)
TRAFFIC = {"sweep_gemm": 205.7e6, "gj_update": None}
try:
    TRAFFIC.update(json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))))
except Exception:
    pass
UNIT = "source-solves/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--nsrc", type=int, default=256)
    ap.add_argument("--nfreq", type=int, default=16, help="frequencies in total (strong, default) / per GPU (weak)")
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"])
    ap.add_argument("--no-weak", action="store_true", help="N > 1: skip the extra weak-scaling measurement")
    ap.add_argument("--groups", type=int, default=0, help="launch chains (streams) per GPU; 0 = library default")
    ap.add_argument("--shard", default="freq", choices=["freq", "source"],
                    help="N > 1: shard the frequencies (configs[2]) or blocks of sources with the factorisation replicated (configs[3])")
    ap.add_argument("--config", default=None, choices=["cfg2", "cfg3", "cfg4", "cfg5"],
                    help="preset: cfg2 = 256^2 / 256 sources / 1 frequency; cfg3 = the default; cfg4 = 1024^2 / 1024 sources / 1 frequency, "
                         "source-block sharding; cfg5 = 2048^2 / 512 sources / one frequency per GPU (weak: 8 frequencies on 8 GPUs)")
    ap.add_argument("--dtype", default="c64", choices=["c64", "c128"])
    ap.add_argument("--engine", default="auto", choices=["auto", "simt", "tc2"])
    ap.add_argument("--cpu-cols", type=int, default=24, help="columns of the CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the (loss, grad) of the last timed step as DIR/loss.npy and DIR/grad.npy, for comparing two builds "
                         "output for output (the inputs are the same from run to run)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.config == "cfg2":
        a.n, a.nsrc, a.nfreq = 256, 256, 1
    elif a.config == "cfg4":
        a.n, a.nsrc, a.nfreq, a.shard = 1024, 1024, 1, "source"
    elif a.config == "cfg5":
        a.n, a.nsrc, a.nfreq, a.scaling = 2048, 512, 1, "weak"
    a.cfg_name = {"cfg2": "configs[1]", "cfg4": "configs[3]", "cfg5": "configs[4]"}.get(a.config, "configs[2]")
    return a


def workload(a):
    from waveforminversionust_b200 import geometry as G
    geom = G.ring_geometry(a.n, a.nsrc)
    f_hi = G.frequency_for_grid(a.n)  # 5.29 points per wavelength at the top frequency (596 kHz at 512)
    world = int(os.environ.get("WORLD_SIZE", "1")) if a.impl == "ours" else max(1, a.gpus)
    a.nfreq_total = a.nfreq * world if a.scaling == "weak" else a.nfreq
    freqs = np.linspace(f_hi * 300.0 / 596.0, f_hi, a.nfreq_total) if a.nfreq_total > 1 else np.array([f_hi])
    vel_true = G.blob_model(geom)
    vel0 = G.blob_model(geom, dc=15.0, seed=99)  # current estimate: heterogeneous, not the truth
    return geom, freqs, vel_true, vel0


def config_for(a, geom, freqs):
    """The workload description both arms print (identical dict for `ours` and `--impl reference`)."""
    return {"workload": f"{a.n}x{a.n} grid, {geom.tx_include.size}-element ring, {a.nfreq_total}-frequency sweep (BASELINE {a.cfg_name}); "
                        f"step = joint (loss, grad): factor + forward + adjoint + gradient per frequency",
            "grid": a.n, "sources": int(geom.tx_include.size), "receivers_per_source": int(geom.mask_indices.shape[1]),
            "frequencies": int(a.nfreq_total), "freq_khz": [round(float(f) / 1e3, 1) for f in (freqs[0], freqs[-1])]}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_sample(geom, freqs, vel0, ncols, dtype="c64"):
    """One frequency, `ncols` source columns, forward + adjoint through the oracle's spsolve path
    (re-factorising each call exactly as the reference does).  Returns seconds."""
    from oracle import helmholtz as oh
    f = float(freqs[-1])
    src = geom.dense_src()[:, :, :ncols]
    t0 = time.perf_counter()
    u = oh.solve_helmholtz(geom.xi, geom.yi, vel0, src, f, geom.a0, geom.L_PML, False, dtype=dtype)
    oh.solve_helmholtz(geom.xi, geom.yi, vel0, u, f, geom.a0, geom.L_PML, True, dtype=dtype)
    return time.perf_counter() - t0


def _ref_worker(args):
    n, nsrc, f, c1, c2, dtype = args
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    from waveforminversionust_b200 import geometry as G
    geom = G.ring_geometry(n, nsrc)
    vel0 = G.blob_model(geom, dc=15.0, seed=99)
    return cpu_sample(geom, [f], vel0, c1, dtype), cpu_sample(geom, [f], vel0, c2, dtype)


def run_reference(a):
    """Reference arm: the reference's own algorithm for this path on the host CPU.  JAX/jaxopt are not
    installable in this image, so this runs the oracle port (NumPy assembly + SciPy spsolve -> SuperLU,
    the same third-party arithmetic the reference calls, re-factorising on every call like the reference).
    SuperLU is single-threaded; frequencies are independent, so one process per frequency uses all host
    cores.  Each step is a bounded two-point sample (c1 and c2 of the nsrc source columns, forward +
    adjoint) from which the fixed (assembly + factorisation) and per-column costs of one solve call are
    separated; `value` is the rate those costs give for the FULL workload (all nsrc columns per call, so
    that the factorisation is amortised exactly as in the real run), which is the number the GPU arm's
    whole-job throughput should be compared with."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    geom, freqs, _, _ = workload(a)
    cores = os.cpu_count() or 1
    nproc = max(1, min(cores, a.nfreq))
    c2 = max(4, min(a.cpu_cols, 12))
    c1 = 2
    jobs = [(a.n, a.nsrc, float(freqs[-1 - (i % a.nfreq)]), c1, c2, a.dtype) for i in range(nproc)]
    ctx = mp.get_context("spawn")
    times, fits = [], []
    with ctx.Pool(nproc) as pool:
        for i in range(a.warmup + a.steps):
            if i < a.warmup and i > 0:
                continue  # one warm-up pass is enough to page SciPy in; keep the run within minutes
            t0 = time.perf_counter()
            res = pool.map(_ref_worker, jobs)
            if i >= a.warmup:
                times.append(time.perf_counter() - t0)
                t1 = float(np.mean([r[0] for r in res])); t2 = float(np.mean([r[1] for r in res]))
                per_col = max((t2 - t1) / (2 * (c2 - c1)), 1e-9)   # seconds per column per solve call
                fixed = max(t2 / 2 - per_col * c2, 0.0)            # assembly + factorisation per solve call
                fits.append((fixed, per_col))
    ms = 1e3 * float(np.mean(times))
    fixed = float(np.mean([f_[0] for f_ in fits])); per_col = float(np.mean([f_[1] for f_ in fits]))
    value = nproc * a.nsrc / (fixed + per_col * a.nsrc)  # nproc frequencies in flight, each nsrc columns per solve call
    sample = (f"{nproc} of {a.nfreq} frequencies in parallel (one process each, SuperLU is single-threaded), per step two "
              f"forward+adjoint spsolve samples with {c1} and {c2} of the {a.nsrc} source columns (re-factorising each call as the "
              f"reference does) -> {fixed:.2f} s fixed + {per_col * 1e3:.1f} ms/column per solve call; value = MODELLED rate for all "
              f"{a.nsrc} columns per call on {nproc} cores")
    emit({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
        "dtype": a.dtype, "data": "synthetic",
        "config": config_for(a, geom, freqs),
        "value_is": "modelled from a bounded two-point sample (fixed + per-column cost of one spsolve call), not a timed full solve",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": nproc, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


_REAL_STDOUT = None


def emit(obj):
    """The one JSON line of the contract, on the process's original stdout."""
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


class Harness:
    """One ShardedFWI engine + its synthetic observed data + the timing helpers, for one list of frequencies."""

    def __init__(self, a, torch, dist, geom, freqs, vel_true, vel0, rank, world, local):
        from waveforminversionust_b200 import geometry as G
        from waveforminversionust_b200.distributed import ShardedFWI
        self.a, self.torch, self.dist, self.geom, self.freqs = a, torch, dist, geom, freqs
        self.rank, self.world, self.local = rank, world, local
        self.dv = dv = torch.device(f"cuda:{local}")
        self.eng = eng = ShardedFWI(geom, freqs, dtype=a.dtype, device=local, rank=rank, world=world, engine=a.engine, shard=a.shard)
        if a.groups > 0:
            eng.plan.set_groups(a.groups)
        plan = eng.plan
        self.nl = nl = len(eng.local)
        self.nt_all = geom.tx_include.size
        self.nt = nt = len(eng.local_tx)  # this rank's transmitters (all of them unless --shard source)
        ne = geom.num_elements
        self.slow0 = torch.as_tensor((1.0 / vel0).astype(plan.real)).to(dv)
        # synthetic observed data from the true model with this solver: REC[f,t,e] = amp_t * u_t(element e)
        self.rec_local = rec_local = torch.zeros((max(nl, 1), max(nt, 1), ne), dtype=plan.tcplx, device=dv)
        if nl and nt:
            slow_true = torch.as_tensor((1.0 / vel_true).astype(plan.real)).to(dv)
            plan.fwi_loss_grad(slow_true, rec_local, eng.local_freqs)
            amp = torch.as_tensor(G.source_amplitudes(self.nt_all)[eng.local_tx]).to(dv, plan.tcplx)
            rx = torch.as_tensor((geom.y_idx * geom.Nx + geom.x_idx).astype(np.int64)).to(dv)
            for i in range(nl):
                U = plan.wavefield(i).reshape(geom.Ny * geom.Nx, nt)
                rec_local[i] = (U[rx, :].T * amp[:, None])
                del U
        torch.cuda.synchronize()
        self.units_per_step = len(freqs) * self.nt_all * 2

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps):
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(steps):
            out = fn()
        e1.record()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=self.dv)
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)
        return float(ms[0]), out

    def step_dev(self):
        return self.eng.loss_grad_device(self.slow0, self.rec_local)

    def close(self):
        self.eng.close()
        del self.rec_local, self.slow0
        self.torch.cuda.empty_cache()


def main():
    global _REAL_STDOUT
    a = parse()
    # stdout must carry exactly one JSON line: anything libraries print (NCCL's version banner, ...) is sent to stderr
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if a.impl == "reference":
        run_reference(a)
        return
    import torch
    import torch.distributed as dist
    from waveforminversionust_b200 import _lib

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus:
        if world == 1 and a.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    torch.cuda.set_device(local)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # stdout carries exactly one JSON line
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    L = _lib.lib()

    geom, freqs, vel_true, vel0 = workload(a)
    H = Harness(a, torch, dist, geom, freqs, vel_true, vel0, rank, world, local)
    eng, plan, nl, nt = H.eng, H.eng.plan, H.nl, H.nt
    eng_name = a.engine
    if a.dtype != "c64":
        eng_name = "simt"
    elif a.engine == "auto":
        eng_name = "tc2"
    KERNEL_LABEL = {
        ("tc2", "sweep_gemm"): "tc2_sweep_gemm_kernel (TMA-fed tcgen05 kind::f16 complex GEMM, K = n; FP32-accurate products from BF16x3 splits = "
                               "6 MMA passes, leading product drained to FP32 registers every 16 k)",
        ("tc2", "gj_update"): "tc2_gj_update_kernel (rank-64 update of the blocked Gauss-Jordan inversion: the same TMA-fed tcgen05 complex GEMM "
                              "with K = 64 on 128 x 64 tiles, two CTAs per SM, look-ahead pivot inversion riding on the launch)",
        ("simt", "sweep_gemm"): "sweep_gemm_kernel (complex GEMM on the CUDA cores: FP32 FMA, or for complex128 the FP64 tensor-core instruction mma.sync.m8n8k4.f64)",
        ("simt", "gj_update"): "gj_update_kernel (rank-64 update: FP32 FMA, or for complex128 FP64 mma.sync.m8n8k4)",
    }
    ENGINE_LABEL = {"tc2": "tcgen05-tma-bf16x3", "simt": "simt-fp32" if a.dtype == "c64" else "dmma-fp64"}
    units_per_step = H.units_per_step

    # ---- value: inputs resident in HBM ----
    for _ in range(a.warmup):
        H.step_dev()
    L.ust_launch_count_reset()
    clk = ClockSampler(local)
    if rank == 0:
        clk.start()
    ms_dev, (loss, grad) = H.timed(H.step_dev, a.steps)
    clocks = clk.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, loss, grad)
    launches = int(L.ust_launch_count())
    ms_step = ms_dev / a.steps
    value = units_per_step / (ms_step / 1e3)
    ok = bool(torch.isfinite(loss)) and bool(torch.isfinite(grad).all()) and plan.status() == 0
    if not ok:
        raise SystemExit("bench: non-finite result or singular block met")
    # size-independent correctness check of what was just timed: residual of forward columns of the first / last local frequency
    checks = None
    if nl and nt:
        res = [plan.residual_onehot(fi, ti) for fi in sorted({0, nl - 1}) for ti in sorted({0, nt // 2, nt - 1})]
        worst = max(r[0] / r[1] for r in res)
        checks = {"forward_residual_over_scale_max": worst, "what": "max over 6 (frequency, source) columns of ||H u - e_src|| / || |H||u| || "
                  "(complex64 rounding level ~1e-7, complex128 ~1e-16)", "status": plan.status()}
        if not worst < (1e-5 if a.dtype == "c64" else 1e-12):
            raise SystemExit(f"bench: forward residual check failed ({worst:.3e})")
    # host time to ENQUEUE one step (no synchronisation): how close the CPU launch rate is to the GPU's pace
    torch.cuda.synchronize()
    t_enq = time.perf_counter()
    H.step_dev()
    host_enqueue_ms = 1e3 * (time.perf_counter() - t_enq)
    torch.cuda.synchronize()

    # ---- e2e: HOST buffers through the reference-facing call ----
    slow_h = torch.empty(H.slow0.shape, dtype=H.slow0.dtype).pin_memory()
    slow_h.copy_(H.slow0.cpu())
    rec_h = torch.empty(H.rec_local[:max(nl, 1)].shape, dtype=H.rec_local.dtype).pin_memory()
    rec_h.copy_(H.rec_local.cpu())
    if world == 1:
        # the C-ABI host entry itself (ust_fwi_loss_grad_host): host pointers in, host results out, copies inside the call
        grad_h = torch.empty(H.slow0.shape, dtype=H.slow0.dtype).pin_memory()
        slow_np, rec_np, grad_np = slow_h.numpy(), rec_h.numpy(), grad_h.numpy()
        e2e_api = "ust_fwi_loss_grad_host (C ABI, pinned host buffers)"
        step_host = lambda: plan.fwi_loss_grad_host(slow_np, rec_np, eng.local_freqs, out_grad=grad_np)
    else:
        e2e_api = "ShardedFWI.loss_grad_host (pinned host buffers -> device, evaluation, NCCL all-reduce, device -> host)"
        step_host = lambda: eng.loss_grad_host(slow_h, rec_h[:nl] if nl else rec_h)
    step_host()
    ms_host, (loss_h, grad_h_out) = H.timed(step_host, a.steps)
    e2e_value = units_per_step / (ms_host / a.steps / 1e3)
    assert abs(float(loss_h) - float(loss)) <= 1e-6 * abs(float(loss))

    # ---- roofline: per-launch event timing on one extra step (single launch chain: no overlap between timed launches) ----
    roof, step_roof, kernels = None, None, {}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    tc_peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)))
    src = "measured (MEASURED_PEAKS.json, sustained bf16)" if peaks else "fallback (B200_PROFILING.md)"
    nI, M = geom.Nx - 2, geom.Ny - 2
    if nl and nt:
        plan.profile(True)
        H.step_dev()
        prof = plan.get_profile()
        plan.profile(False)
        csz = 8 if a.dtype == "c64" else 16
        # one-hot forward solves: column tiles that are still identically zero during elimination are skipped by the kernels
        # (sweep.cuh: sweep_tile_is_zero); count only the products that are executed
        tiles_n = -(-nt // 128)
        src_row = (geom.y_idx[geom.tx_include][eng.local_tx] - 1).astype(int)
        mid = M // 2
        skipped = 0
        if eng_name == "tc2" and tiles_n <= 8:
            for tn in range(tiles_n):
                rows = src_row[tn * 128:(tn + 1) * 128]
                skipped += int(np.sum(np.arange(0, mid) < rows.min())) + int(np.sum(np.arange(mid + 1, M) > rows.max()))
        gemm_units = 2 * (2 * M - 1) * tiles_n - skipped  # (block row, column tile) products per frequency: forward + adjoint solve
        nP = plan_np(geom)
        nblk = nP // 64
        inv_flops = nl * M * 8.0 * float(nI) ** 3  # Gauss-Jordan inverse = n^3 complex MACs per block row (SURVEY 8d)
        alg = {
            "sweep_gemm": ("tensor", nl * gemm_units * 8.0 * nI * nI * (nt / tiles_n)),
            "gj_update": ("tensor", inv_flops * (nblk - 1) / nblk),  # rank-64 updates of all block rows but the pivot row
            "gj_rowpanel": ("tensor", inv_flops / nblk),               # R = P * X_k,: (the 64 x 64 pivot inversions are the remaining O(n^2 * 64))
            "assemble": ("hbm", nl * geom.Nx * geom.Ny * (csz / 2 + 9 * csz)),
            "gradient": ("hbm", nl * geom.Nx * geom.Ny * nt * 2.0 * csz + geom.Nx * geom.Ny * csz),
        }
        for name, (bound, work) in alg.items():
            ms, cnt = prof[name]
            if cnt == 0 or ms <= 0:
                continue
            if bound == "tensor":
                ach, peak, unit = work / (ms * 1e-3) / 1e12, tc_peak, "TFLOP/s"
            else:
                ach, peak, unit = work / (ms * 1e-3) / 1e9, hbm_peak, "GB/s"
            kernels[name] = {"bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                             "launches": cnt, "ms_total": ms, "work_per_launch": work / cnt}
        for name in ("schur", "gj_panel", "tri_apply", "receiver", "t_split", "gj_pivot", "gj_k0"):
            ms, cnt = prof[name]
            kernels[name] = {"launches": cnt, "ms_total": ms}
        serial_ms = sum(v["ms_total"] for n_, v in kernels.items() if n_ != "gj_panel")  # gj_panel brackets gj_pivot + gj_rowpanel
        dom = max((n_ for n_ in kernels if "frac" in kernels[n_]), key=lambda n_: kernels[n_]["ms_total"])
        k = kernels[dom]
        roof = {"bound": k["bound"], "achieved": k["achieved"], "peak": k["peak"], "unit": k["unit"], "frac": k["frac"],
                "traffic": TRAFFIC.get(dom), "kernel_class": dom, "kernel": KERNEL_LABEL.get((eng_name, dom), dom), "peak_source": src,
                "algorithmic_work_per_launch": k["work_per_launch"], "avg_launch_ms": k["ms_total"] / k["launches"],
                "share_of_step": k["ms_total"] / serial_ms,
                "note": "per-launch times from a profiling step run as ONE launch chain (events around every launch); the timed steps overlap "
                        "the launch chains of the frequency groups, so ms_per_step is below the sum of the per-class totals"}
        fac_ms = sum(prof[c][0] for c in ("schur", "gj_k0", "gj_rowpanel", "gj_update", "gj_pivot"))
        kernels["factor_total"] = {"bound": "tensor", "ms_total": fac_ms, "achieved": inv_flops / (fac_ms * 1e-3) / 1e12, "peak": tc_peak,
                                   "unit": "TFLOP/s", "frac": inv_flops / (fac_ms * 1e-3) / 1e12 / tc_peak}
        step_flops = inv_flops + alg["sweep_gemm"][1]
        step_roof = {"bound": "tensor", "achieved": step_flops / (ms_step * 1e-3) / 1e12, "peak": tc_peak, "unit": "TFLOP/s",
                     "frac": step_flops / (ms_step * 1e-3) / 1e12 / tc_peak, "algorithmic_flops_per_step_this_rank": step_flops,
                     "what": "explicit-inverse factorisation 8 n^3 per block row + executed sweep products 8 n^2 per column and block row, "
                             "this rank's frequencies, over ms_per_step"}

    # ---- CPU baseline (rank 0, N=1 only): bounded sample of the same workload on the host cores ----
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        c1, c2 = max(2, a.cpu_cols // 6), a.cpu_cols
        t1 = cpu_sample(geom, freqs, vel0, c1, a.dtype)
        t2 = cpu_sample(geom, freqs, vel0, c2, a.dtype)
        per_col = max((t2 - t1) / (2 * (c2 - c1)), 1e-9)  # seconds per column per solve
        fixed = max(t2 / 2 - per_col * c2, 0.0)  # factorisation + assembly per solve call
        full = nt / (fixed + per_col * nt)
        cpu = {"value": 2 * c2 / t2, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": (f"oracle solve_helmholtz (SciPy spsolve -> SuperLU, single-threaded), {a.dtype}, {a.n}x{a.n} grid, 1 of "
                          f"{a.nfreq} frequencies (the highest), {c2} of {nt} source columns, forward + adjoint, {t2:.1f} s; with a "
                          f"{c1}-column run ({t1:.1f} s) this gives {fixed:.2f} s fixed + {per_col * 1e3:.1f} ms/column per solve call"),
               "modelled_full_columns": full, "host_cores_available": os.cpu_count()}

    device_bytes = plan.device_bytes
    h2d, d2h = eng.h2d_bytes, eng.d2h_bytes
    nfreq_local = nl

    # ---- N > 1: the weak-scaling rate beside the configured (strong) one ----
    weak = None
    if world > 1 and a.scaling == "strong" and a.shard == "freq" and not a.no_weak:
        H.close()
        import copy
        aw = copy.copy(a)
        aw.scaling = "weak"
        geom_w, freqs_w, vt_w, v0_w = workload(aw)
        HW = Harness(aw, torch, dist, geom_w, freqs_w, vt_w, v0_w, rank, world, local)
        for _ in range(a.warmup):
            HW.step_dev()
        ms_w, _ = HW.timed(HW.step_dev, a.steps)
        weak = {"value": HW.units_per_step / (ms_w / a.steps / 1e3), "unit": UNIT, "ms_per_step": ms_w / a.steps,
                "frequencies": len(freqs_w), "frequencies_per_gpu": HW.nl,
                "what": f"{a.nfreq} frequencies kept on every GPU: a {len(freqs_w)}-frequency objective over the same band"}
        H = HW

    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
            "dtype": a.dtype, "data": "synthetic",
            "config": config_for(a, geom, freqs),
            "impl_config": {"parallelism": f"{a.shard}-shard x{world}", "frequencies_per_gpu": nfreq_local, "sources_per_gpu": nt,
                            "l2": "working set per step (factors + wavefields, %.1f GB) >> 126 MB L2" % (device_bytes / 1e9),
                            "engine": ENGINE_LABEL[eng_name], "mma_passes_per_product": 6 if eng_name == "tc2" else None,
                            "launch_chains_per_gpu": a.groups if a.groups > 0 else "library default (2)"},
            "sec_per_fwi_iteration": ms_step / 1e3,
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_host / a.steps, "api": e2e_api,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, "host_enqueue_ms_per_step": host_enqueue_ms, "clocks": clocks, "roofline": roof,
            "step_roofline": step_roof, "kernels": kernels, "cpu_baseline": cpu, "weak_scaling": weak,
            "loss": float(loss), "device_bytes": device_bytes, "checks": checks,
        }
        emit(out)
    H.barrier()
    H.close()
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 64 << 20


def dump_outputs(d, loss, grad):
    """What the timed step hands its caller: the all-reduced loss (float64) and gradient (float32 for complex64, float64 for
    complex128).  A gradient larger than DUMP_BYTES is replaced by the entries at a fixed, seeded, sorted set of flat indices."""
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "loss.npy"), loss.detach().cpu().numpy().astype(np.float64))
    g = grad.detach().cpu().numpy().ravel()
    if g.nbytes > DUMP_BYTES - 4096:
        g = g[np.sort(np.random.default_rng(0).choice(g.size, (DUMP_BYTES - 4096) // g.itemsize, replace=False))]
    else:
        g = g.reshape(grad.shape)
    np.save(os.path.join(d, "grad.npy"), g)


def plan_np(geom):
    return ((geom.Nx - 2 + 63) // 64) * 64


if __name__ == "__main__":
    main()
