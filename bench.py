#!/usr/bin/env python
"""bench.py -- headline benchmark of the dense-GP hot path (BASELINE.json metric).

One "step" = one pass of the hot path over one batch of synthetic input (SURVEY.md 8d, config 2):
  assemble K (SE kernel, N=65536 1-D inputs, fp64) -> Cholesky(K + 0.1 I) -> logpdf(y)
  -> posterior mean & variance at N*=4096 test points.
`value`  = N / step time with inputs already resident in HBM (device pointers through the C ABI),
           timed with CUDA events on the library's own stream (max over ranks).
`e2e`    = the same through the public API with HOST numpy buffers (H2D/D2H inside the region).
`--impl reference` times the CPU restatement of the reference path (oracle fast path:
  NumPy + SciPy/OpenBLAS, all host threads) on a bounded sample and extrapolates with the
  N^3 / N^2 cost model (the reference is Julia; no julia binary in this image -- DESIGN.md).
`--dump-outputs DIR` writes what the last timed device step returned (logpdf, posterior mean and
  variance) as DIR/<name>.npy in float64, so two builds can be compared output for output on the
  same seeded inputs.
"""
from __future__ import annotations

import argparse
import gc
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

N_TRAIN = 65536
N_TEST = 4096
SIGMA2 = 0.1
DEFAULT_TRAILING = "ozaki"
DMMA_PEAK_TFLOPS = 37.1  # builder-measured, tools/mb_fp64_peak.cu on this pool's B200 (profiles/)


_OUT_FD = None  # set by main(): the process's ORIGINAL stdout; fd 1 itself is pointed at stderr


def emit(line: str):
    """Print the one JSON line.  Under main() everything else that writes to fd 1 (NCCL's version
    banner, torch warnings from C++) has been diverted to stderr, so stdout carries only this."""
    if _OUT_FD is None:
        print(line)
        sys.stdout.flush()
    else:
        os.write(_OUT_FD, (line + "\n").encode())


def make_inputs(n, ns):
    """SURVEY.md 8(d) config 2: x ~ U(0, n/32) (32 points per length-scale), y = sin(x)+0.3 eps."""
    rng = np.random.default_rng(123456)
    x = rng.uniform(0, n / 32, n)
    xs = rng.uniform(0, n / 32, ns)
    y = np.sin(x) + 0.3 * rng.standard_normal(n)
    return x, y, xs


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, **arrays):
    """Write each array as out_dir/<name>.npy (float64).  Outputs larger than DUMP_LIMIT_BYTES in all
    (only with a large --ns) are replaced by the same fixed, seeded sample of entries, whose indices
    are written too as sample_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        size = max(a.size for a in arrays.values())
        keep = size * DUMP_LIMIT_BYTES // (2 * total)  # half the budget: leaves room for the index
        idx = np.sort(np.random.default_rng(0).choice(size, keep, replace=False))
        arrays = {k: a[idx] if a.size == size else a for k, a in arrays.items()}
        arrays["sample_index"] = idx.astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline: oracle fast path (same LAPACK entry points as Julia+OpenBLAS)
# ------------------------------------------------------------------------------------------


def cpu_pipeline(x, y, xs, sigma2):
    """Fast-path restatement used for timing (BASELINE.md section 2); numerically identical to
    oracle/stheno_oracle.py's logpdf + posterior for a single SE process (checked in tests)."""
    import scipy.linalg as sla
    from oracle.stheno_oracle import pairwise_sqeuclidean
    t = {}
    t0 = time.perf_counter()
    K = pairwise_sqeuclidean(x.reshape(1, -1))
    np.multiply(K, -0.5, out=K)
    np.exp(K, out=K)
    K[np.diag_indices_from(K)] += sigma2
    K = np.asfortranarray(K)
    t["assemble"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    U = sla.cholesky(K, lower=False, overwrite_a=True, check_finite=False)
    t["chol"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    n = len(x)
    v = sla.solve_triangular(U, y, trans="T", lower=False, check_finite=False)
    lp = -(n * math.log(2 * math.pi) + 2 * np.sum(np.log(np.diag(U))) + v @ v) / 2
    alpha = sla.solve_triangular(U, v, lower=False, check_finite=False)
    t["solve"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    Kfs = np.exp(-0.5 * pairwise_sqeuclidean(x.reshape(1, -1), xs.reshape(1, -1)))
    mean = Kfs.T @ alpha
    V = sla.solve_triangular(U, np.asfortranarray(Kfs), trans="T", lower=False, overwrite_b=True,
                             check_finite=False)
    var = 1.0 - np.einsum("ij,ij->j", V, V)
    t["posterior"] = time.perf_counter() - t0
    return lp, mean, var, t


def cpu_extrapolate(t, n_s, ns_s, n, ns):
    """Scale measured phase times from the sample (n_s, ns_s) to (n, ns)."""
    r = n / n_s
    return (t["assemble"] * r * r + t["chol"] * r ** 3 + t["solve"] * r * r
            + t["posterior"] * r * r * (ns / ns_s))


def pin_cpu_threads():
    """Use every host core for the CPU arm, whatever the launcher exported: torchrun sets
    OMP_NUM_THREADS=1, which silently turned the round-1 reference arm into a 1-thread run."""
    want = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=want)
        got = max([p.get("num_threads", 1) for p in threadpool_info()] + [1])
        return got
    except Exception:
        return 1


def host_ram_gb():
    try:
        import psutil
        return psutil.virtual_memory().available / 1e9
    except Exception:
        return 0.0


def cpu_sample_size():
    """One fixed sample size per host class (NOT per thread count): N=32768 needs ~30 GB and ~1 min
    on a >= 32-core host; otherwise N=16384."""
    return 32768 if (host_ram_gb() >= 48 and (os.cpu_count() or 1) >= 32) else 16384


def run_cpu_sample(n_s=None, reps=1):
    """Time the oracle fast path at (n_s, n_s/16) `reps` times; per-phase minimum over the
    repetitions (the box is shared: minima are the reproducible statistic), plus the spread."""
    cores = pin_cpu_threads()
    if n_s is None:
        n_s = cpu_sample_size()
    ns_s = max(64, n_s // 16)
    x, y, xs = make_inputs(n_s, ns_s)
    runs = []
    for _ in range(reps):
        _, _, _, t = cpu_pipeline(x, y, xs, SIGMA2)
        runs.append(t)
    best = {k: min(r[k] for r in runs) for k in runs[0]}
    totals = [sum(r.values()) for r in runs]
    measured = sum(best.values())
    ext = cpu_extrapolate(best, n_s, ns_s, N_TRAIN, N_TEST)
    return dict(n_sample=n_s, ns_sample=ns_s, measured_s=measured, extrapolated_s=ext, phases=best,
                cores=cores, reps=reps, total_s_min=min(totals), total_s_max=max(totals),
                host_ram_gb=round(host_ram_gb(), 1))


# ------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
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
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
                for nm, val in zip(names, r[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        # "under load" = samples drawing more than half of the max observed power
        load = [s for s, p in zip(sm, pw) if pw and p >= 0.5 * max(pw)] or sm
        return {"sm_mhz": float(np.median(load)) if load else None,
                "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------


def gpu_main(args):
    import ctypes as C

    import torch
    import stheno_jl_b200 as sb
    from stheno_jl_b200 import lib as sblib
    from stheno_jl_b200.gp import Lowered, spec_dense, spec_diag, spec_symmetric

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group(backend="cpu:gloo,cuda:nccl", rank=rank, world_size=world)
        ids = [sblib.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        ctx = sblib.Context(local, rank, world, ids[0])
    else:
        ctx = sblib.Context(local)
    sblib.set_default_context(ctx)
    lib = sblib.load()
    ctx.set_option("trailing", 1 if args.trailing == "ozaki" else 0)

    n, ns = args.n, args.ns
    x, y, xs = make_inputs(n, ns)
    f = sb.gppp(lambda GP: dict(f=GP(sb.SEKernel())))

    # ---- device-resident arm: inputs live in HBM before the timed region -----------------------
    dev = torch.device("cuda", local)
    xd, yd, xsd = (torch.from_numpy(a).to(dev) for a in (x, y, xs))
    mean_d = torch.empty(ns, dtype=torch.float64, device=dev)
    var_d = torch.empty(ns, dtype=torch.float64, device=dev)
    lx = Lowered(f, sb.GPPPInput("f", xd))
    ls = Lowered(f, sb.GPPPInput("f", xsd))
    spec_k, spec_c, spec_d = spec_symmetric(lx), spec_dense(ls, lx), spec_diag(ls)
    noise = sblib.sb_noise()
    noise.sigma2, noise.diag, noise.dense = SIGMA2, None, None
    lp_out = (C.c_double * 1)()

    call_s = {"factor": 0.0, "logpdf": 0.0, "set_data": 0.0, "predict": 0.0, "destroy": 0.0}

    def device_step():
        h = C.c_void_p()
        info = C.c_int64(0)
        t0 = time.perf_counter()
        sblib.check(lib.sb_factor_create(ctx.h, C.byref(spec_k), C.byref(noise), C.byref(h), C.byref(info)), info)
        t1 = time.perf_counter()
        try:
            sblib.check(lib.sb_logpdf(ctx.h, h, yd.data_ptr(), 1, lp_out))           # zero-mean: delta = y
            t2 = time.perf_counter()
            sblib.check(lib.sb_factor_set_data(ctx.h, h, yd.data_ptr()))
            t3 = time.perf_counter()
            sblib.check(lib.sb_predict(ctx.h, h, C.byref(spec_c), C.byref(spec_d), mean_d.data_ptr(), var_d.data_ptr()))
            t4 = time.perf_counter()
        finally:
            lib.sb_factor_destroy(h)
        t5 = time.perf_counter()
        for k, v in zip(call_s, (t1 - t0, t2 - t1, t3 - t2, t4 - t3, t5 - t4)):
            call_s[k] += v
        return lp_out[0]

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        device_step()
    for k in call_s:
        call_s[k] = 0.0
    barrier()
    ctx.timings(reset=True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # The library runs on its own stream and every ABI call is synchronous; the device time of a
    # step is the sum of the CUDA-event phase timers the library records on that stream
    # (sb_timings.total_ms), cross-checked against the host wall clock around the same calls.
    t0 = time.perf_counter()
    ctx.mark(0)
    for _ in range(args.steps):
        lp = device_step()
    ctx.mark(1)
    dev_ms = ctx.elapsed_ms(0, 1)  # CUDA events on the launching (library) stream around K steps
    torch.cuda.synchronize()
    wall_dev = time.perf_counter() - t0
    tm = ctx.timings()
    clocks = sampler.stop() if rank == 0 else None
    step_ms = dev_ms / args.steps
    if dist is not None:
        tt = torch.tensor([step_ms, wall_dev * 1e3 / args.steps], dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        step_ms, wall_ms = tt.tolist()
    else:
        wall_ms = wall_dev * 1e3 / args.steps

    # ---- end-to-end arm: public API, host numpy buffers in, host numpy out ---------------------
    def e2e_step():
        fx = f(sb.GPPPInput("f", x), SIGMA2)
        lp = sb.logpdf(fx, y)
        post = sb.posterior(fx, y)
        m, v = sb.mean_and_var(post, sb.GPPPInput("f", xs))
        return lp, m, v

    e2e_step()
    e2e_s = 0.0
    for _ in range(args.steps):
        # A posterior and its factor refer to each other, so the previous step's device factor
        # (17 GB at N = 65536) is freed only by the cycle collector: free it before the next step.
        gc.collect()
        barrier()
        t0 = time.perf_counter()
        lp_e, m_e, v_e = e2e_step()
        torch.cuda.synchronize()
        e2e_s += time.perf_counter() - t0
    e2e_s /= args.steps
    if dist is not None:
        tt = torch.tensor([e2e_s], dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_s = tt.item()
    h2d = 8 * (n + n + n + ns + n)  # x (factor), delta (logpdf), delta (posterior), x*, x (cross spec)
    d2h = 8 * (2 * ns + 1)

    def shutdown():
        # collective, orderly teardown: NCCL communicator of the library first, then torch's
        if dist is not None:
            dist.barrier()
        sblib.set_default_context(None)
        ctx.close()
        if dist is not None:
            dist.destroy_process_group()

    if rank != 0:
        shutdown()
        return
    mean_h, var_h = mean_d.cpu().numpy(), var_d.cpu().numpy()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, logpdf=np.float64(lp), mean=mean_h, var=var_h)
    np.testing.assert_allclose(mean_h, m_e, rtol=1e-9, atol=1e-10)
    # ---- parity against the committed single-GPU result of the same seeded inputs -----------------
    # (tests/golden/config2_n1.json: written by a 1-GPU DMMA run, itself oracle-checked at N <= 32768
    #  and cross-checked against the tcgen05 path at full size in tests/test_gpu_parity.py)
    gold_path = os.path.join(ROOT, "tests", "golden", "config2_n1.json")
    parity = None
    if args.write_golden and args.gpus == 1 and (n, ns) == (N_TRAIN, N_TEST):
        idx = list(range(0, ns, 16))
        json.dump({"n": n, "ns": ns, "trailing": args.trailing, "logpdf": lp, "idx": idx,
                   "mean": [float(mean_h[i]) for i in idx], "var": [float(var_h[i]) for i in idx]},
                  open(gold_path, "w"))
    if os.path.exists(gold_path) and (n, ns) == (N_TRAIN, N_TEST):
        gd = json.load(open(gold_path))
        idx = np.array(gd["idx"])
        parity = {"logpdf_rel_err": abs(lp - gd["logpdf"]) / abs(gd["logpdf"]),
                  "mean_max_abs_err": float(np.max(np.abs(mean_h[idx] - np.array(gd["mean"])))),
                  "var_max_rel_err": float(np.max(np.abs(var_h[idx] - np.array(gd["var"])) / np.abs(np.array(gd["var"])))),
                  "reference": f"tests/golden/config2_n1.json (1 GPU, trailing={gd.get('trailing')})", "tolerance": 1e-10}
        parity["ok"] = bool(parity["logpdf_rel_err"] <= 1e-10 and parity["mean_max_abs_err"] <= 1e-9
                            and parity["var_max_rel_err"] <= 1e-8)

    # ---- roofline of the dominant kernel (the trailing update of the Cholesky) -----------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    traffic = None
    try:  # per-launch DRAM bytes of the shipped trailing kernel from a committed `ncu --set full` capture
        traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json"))).get(args.trailing)
    except Exception:
        pass
    t_ms = tm["trailing_kernel_ms"]
    fp64_tf = tm["trailing_flops"] / (t_ms * 1e-3) / 1e12 if t_ms else None
    if tm.get("trailing_int8_ops", 0) > 0:
        # tcgen05 kind::i8: 28 int8 MMAs per fp64 MMA.  Peak = 2 x the MEASURED dense bf16 tensor peak
        # (int8 runs at twice the bf16 rate on sm_100a); sustained figure: the kernel runs inside a long step.
        bf16 = peaks.get("bf16_tflops_sustained", 1400.0)
        peak = 2.0 * bf16
        ach = tm["trailing_int8_ops"] / (t_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": "ozaki_syrk_kernel (tcgen05.mma kind::i8 from TMEM, fp64 via 7 int8 digit planes)",
                "achieved": ach, "peak": peak, "unit": "TOP/s (int8)", "frac": ach / peak,
                "peak_source": ("2 x MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "2 x fallback 1400 TF (of fallback)"),
                "fp64_equivalent_tflops": fp64_tf, "vs_dmma_peak": fp64_tf / DMMA_PEAK_TFLOPS if fp64_tf else None,
                "launches": tm["trailing_launches"] // max(1, args.steps),
                "flops_per_step": tm["trailing_flops"] / args.steps,
                "int8_ops_per_step": tm["trailing_int8_ops"] / args.steps}
    else:
        roof = {"bound": "tensor", "kernel": "gemm_nt_kernel (fp64 DMMA SYRK trailing update)",
                "achieved": fp64_tf, "peak": DMMA_PEAK_TFLOPS, "unit": "TFLOP/s",
                "frac": (fp64_tf / DMMA_PEAK_TFLOPS) if fp64_tf else None,
                "peak_source": "builder-measured mma.sync m8n8k4 f64 microbenchmark (tools/mb_fp64_peak.cu, "
                               "profiles/mb_fp64_peak_r1.txt); MEASURED_PEAKS.json has no fp64 entry, "
                               "tcgen05 has no fp64 kind",
                "launches": tm["trailing_launches"] // max(1, args.steps),
                "flops_per_step": tm["trailing_flops"] / args.steps}
    roof["traffic"] = traffic["dram_bytes_per_launch"] if traffic else None
    if traffic:
        roof["traffic_algorithmic"] = traffic.get("algorithmic_bytes_per_launch")
        roof["traffic_source"] = traffic.get("source")
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    asm_bytes = (n * (n + 1) / 2 * 8 + n * 8)
    roof_asm = {"bound": "hbm", "kernel": "assemble_kernel<packed>", "achieved": asm_bytes / (tm["assemble_ms"] / args.steps * 1e-3) / 1e9,
                "peak": hbm_peak, "unit": "GB/s"}
    roof_asm["frac"] = roof_asm["achieved"] / hbm_peak
    phases = {k: tm[k] / args.steps for k in ("assemble_ms", "panel_ms", "trailing_ms", "comm_ms", "solve_ms", "predict_ms", "panel_chain_ms")}

    cb = None
    if args.gpus == 1 and not args.no_cpu:
        s = run_cpu_sample(16384, 1)
        cb = {"value": N_TRAIN / s["extrapolated_s"], "unit": "points/s", "cores": s["cores"], "kind": "port",
              "sample": f"oracle fast path (NumPy+SciPy/OpenBLAS, {s['cores']} threads) measured once at N={s['n_sample']}, "
                        f"N*={s['ns_sample']}: {s['measured_s']:.2f} s; value extrapolated to N={N_TRAIN}, N*={N_TEST} with the "
                        f"N^3 (chol) / N^2 (assemble, solves) / N^2 N* (posterior) model = {s['extrapolated_s']:.0f} s",
              "phases_s": s["phases"]}

    out = {
        "metric": "logpdf+posterior points/sec, N=65536 SE-GP fp64", "value": n / (step_ms * 1e-3),
        "unit": "points/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": step_ms, "wall_ms_per_step": wall_ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"config 2: SEKernel GP N={n} fp64, 1-D inputs U(0,N/32), sigma2=0.1: "
                               f"kernelmatrix + Cholesky logpdf + posterior mean/var at N*={ns}",
                   "n_train": n, "n_test": ns, "l2": "inputs >> L2 (17.2 GB factor; no flush needed)",
                   "trailing": args.trailing,
                   "parallelism": f"1-D block-cyclic columns x{args.gpus}, NCCL panel broadcast" if args.gpus > 1 else "single GPU"},
        "e2e": {"value": n / e2e_s, "unit": "points/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_s * 1e3},
        "gpu_launches": tm["kernel_launches"], "roofline": roof, "roofline_assemble": roof_asm,
        "phases_ms": phases, "host_call_ms": {k: v * 1e3 / args.steps for k, v in call_s.items()},
        "logpdf": lp, "parity_vs_n1": parity, "clocks": clocks,
    }
    if cb:
        out["cpu_baseline"] = cb
    emit(json.dumps(out))
    shutdown()


def reference_main(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    reps = max(1, min(args.steps, 3))
    if args.warmup > 0:
        run_cpu_sample(4096, 1)   # page in NumPy/SciPy/OpenBLAS, spin up the thread pool
    s = run_cpu_sample(reps=reps)
    ext = s["extrapolated_s"]
    val = N_TRAIN / ext
    out = {
        "impl": "reference", "metric": "logpdf+posterior points/sec, N=65536 SE-GP fp64", "value": val,
        "unit": "points/s", "n_gpus": args.gpus, "steps": reps, "steps_requested": args.steps, "warmup": args.warmup,
        "samples_run": reps, "ms_per_step": ext * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"config 2: SEKernel GP N={N_TRAIN} fp64: kernelmatrix + Cholesky logpdf + "
                               f"posterior mean/var at N*={N_TEST} (CPU restatement of the reference path; "
                               "Julia is not installed in this image)"},
        "cpu_baseline": {"value": val, "unit": "points/s", "cores": s["cores"], "kind": "port",
                         "sample": f"oracle fast path (NumPy + SciPy/OpenBLAS, {s['cores']} threads pinned with threadpoolctl) at "
                                   f"N={s['n_sample']}, N*={s['ns_sample']}: per-phase minimum over {reps} runs = {s['measured_s']:.2f} s "
                                   f"(whole-run min {s['total_s_min']:.2f} s, max {s['total_s_max']:.2f} s); extrapolated to "
                                   f"N={N_TRAIN}, N*={N_TEST} by the N^3 (chol) / N^2 (assemble, solves) / N^2 N* (posterior) model "
                                   f"= {ext:.0f} s.  A full N=65536 CPU step needs ~100 GB and ~10 min, so each step is this bounded sample.",
                         "phases_s": s["phases"], "host_ram_gb": s["host_ram_gb"]},
        "e2e": {"value": val, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=N_TRAIN)
    ap.add_argument("--ns", type=int, default=N_TEST)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--write-golden", action="store_true", help="(1 GPU) rewrite tests/golden/config2_n1.json")
    ap.add_argument("--trailing", default=os.environ.get("SB_BENCH_TRAILING", DEFAULT_TRAILING), choices=["dmma", "ozaki"],
                    help="Cholesky trailing update: fp64 DMMA (mma.sync) or tcgen05 int8 Ozaki slices")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="(b200) write the last timed step's logpdf, posterior mean and variance as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs records the device path: use it with --impl b200")
    global _OUT_FD
    sys.stdout.flush()
    _OUT_FD = os.dup(1)
    os.dup2(2, 1)  # from here on fd 1 == stderr for Python AND C libraries
    if args.impl == "reference":
        reference_main(args)
    else:
        gpu_main(args)


if __name__ == "__main__":
    main()
