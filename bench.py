#!/usr/bin/env python
"""bench.py — QR GFLOP/s (fp64) of qr! on the BASELINE workload, one JSON line on rank 0.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 3|2] [--m M --n N --nb NB]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[2], the one `metric` is quoted on): QR of a 32768 x 4096 fp64 matrix, A[i,j] ~ U[0,1) from
the counter-based generator (synthetic; mirrors rand at test/runtests.jl:45-46), DArray-style contiguous column blocks over
the N GPUs (strong scaling: total work fixed).  A "step" is one full factorisation qr!(A) of a fresh matrix.
  value : (2mn^2 - 2/3 n^3) / t, inputs resident in HBM, CUDA events, max over ranks.
  e2e   : the same through the host-buffer entry (pinned host A -> H2D -> factor -> D2H of A and alpha).
          Before every step the CPU rewrites the pinned buffer and then flushes its caches (1 GiB scratch write), both outside
          the timed region: the host-side analogue of the L2 flush, the input sits in DRAM.  Side figures: the same call with the
          buffer still dirty in the CPU caches (slower, noisy DMA) and with the buffer last written by a device-to-host copy.
  roofline : the dominant kernel class (a DMMA GEMM of the trailing update), algorithmic flops / CUDA-event time of that
             class, against a cuBLAS DGEMM burst measured in this run (MEASURED_PEAKS.json carries no fp64 entry).
  solve : warm H \\ b on the factorisation just computed (Q'b and back-substitution separately; test/runtests.jl:66).
  cpu_baseline : the oracle's C restatement of the reference algorithm on the host cores (bounded strided sample of the
             whole sweep) and LAPACK dgeqrf, the reference tests' own normaliser (test/runtests.jl:49,53-54).
--config 2 measures BASELINE configs[1] (8192 x 1024, nb = 1: the unblocked column loop) with an HBM roofline instead.
--impl reference times the CPU restatement alone (the reference is Julia; Julia is not installed) on the same config.
--dump-outputs DIR writes what the last timed qr! handed back, as float64 .npy files, so that two builds can be compared
output for output (the inputs depend on the arguments only): DIR/alpha.npy (n) and DIR/A.npy (m x k), the factored A at
the columns of `dump_columns` (all n when the factor fits in 48 MiB, else a fixed seeded sample of k columns).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "QR GFLOP/s (fp64)"
ORACLE_PIN = ("oracle = line-cited C restatement of the reference's recurrences; parity with the Julia binary itself is UNPINNED "
              "(no Julia in the image, no golden vectors upstream): pinned by LAPACK dgeqrf through the storage-format identity "
              "and by the reference's own test properties")


def qr_flops(m, n):
    return 2.0 * m * n * n - 2.0 / 3.0 * n ** 3


def make_config(m, n, world):
    """The same dictionary in both arms (`same_config`): it names the workload, not the implementation."""
    return {"workload": f"qr! of {m}x{n} fp64 (A ~ U[0,1) synthetic, column-major), DArray-style contiguous column blocks over {world} process(es)",
            "m": m, "n": n, "processes": world,
            "l2": "inputs (m*n*8 B per step) larger than L2; fresh matrix every step",
            "timing": "GPU arm: CUDA events around K back-to-back qr! calls, max over ranks; CPU arm: wall clock around a strided sample of the column sweep"}


# ---------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi during the timed region)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()                      # exact PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for k, nm in enumerate(names) if any(len(r) > 2 + k and r[2 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle's C restatement, bounded strided sample of the column sweep S:127-144
# ---------------------------------------------------------------------------------------------
def host_cores():
    """(physical cores, logical cpus) this process may run on.  torch.distributed.run exports OMP_NUM_THREADS=1: the CPU arm
    ignores it and sizes its OpenMP team from the affinity mask, one thread per physical core, the same on every box."""
    aff = os.sched_getaffinity(0)
    cores = set()
    try:
        cpu, phys = None, 0
        for line in open("/proc/cpuinfo"):
            k, _, v = line.partition(":")
            k, v = k.strip(), v.strip()
            if k == "processor":
                cpu, phys = int(v), 0
            elif k == "physical id":
                phys = int(v)
            elif k == "core id" and cpu in aff:
                cores.add((phys, int(v)))
    except Exception:
        pass
    return (len(cores) if cores else len(aff)), len(aff)


def cpu_stride(m, n):
    return 8 if qr_flops(m, n) > 2e11 else (2 if qr_flops(m, n) > 2e10 else 1)


def cpu_pass(co, A0shape, offset, stride, threads):
    m, n = A0shape
    A = co.fill_uniform(0, m, n)                    # untimed
    t = time.perf_counter()
    _, fl = co.qr_steps_strided(A, offset % stride, stride, threads)
    return fl, time.perf_counter() - t


def cpu_sample_desc(m, n, stride, threads, logical):
    return (f"every {stride}th column step (S:127-144: norm, alpha, scale, copy, trailing update of all columns to the right) of the "
            f"whole {m}x{n} sweep, offset rotating per pass; GFLOP/s = flops of the sampled steps / their wall time; "
            f"{threads} OpenMP threads = physical cores of the affinity mask ({logical} logical), threads over trailing-column "
            f"chunks as S:203-211")


def cpu_port_baseline(m, n, passes=2):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import dhqr_oracle as O
    co = O.COracle()
    threads, logical = host_cores()
    threads = int(os.environ.get("DHQR_CPU_THREADS", "0")) or threads
    stride = cpu_stride(m, n)
    cpu_pass(co, (min(m, 4096), min(n, 256)), 0, 1, threads)        # thread start-up, untimed
    fl = dt = 0.0
    for p in range(passes):
        f, d = cpu_pass(co, (m, n), p, stride, threads)
        fl, dt = fl + f, dt + d
    return {"value": fl / dt / 1e9, "unit": "GFLOP/s", "cores": threads, "kind": "port",
            "sample": cpu_sample_desc(m, n, stride, threads, logical) + f"; {passes} passes, {dt:.1f} s",
            "extrapolated_full_factorisation_s": qr_flops(m, n) / (fl / dt)}


def lapack_baseline(m, n, threads):
    """LAPACK dgeqrf, the 'stdlib' number the reference's own tests normalise to (test/runtests.jl:49, 53-54, 87-89)."""
    try:
        import numpy as np
        from scipy.linalg import lapack
        from threadpoolctl import threadpool_limits
        ns = min(n, 1024)
        a = np.asfortranarray(np.random.default_rng(0).random((m, ns)))
        with threadpool_limits(limits=threads):
            lapack.dgeqrf(np.asfortranarray(a[:2048, :128].copy()))
            t = time.perf_counter()
            lapack.dgeqrf(a, overwrite_a=1)
            dt = time.perf_counter() - t
        return {"value": qr_flops(m, ns) / dt / 1e9, "unit": "GFLOP/s", "threads": threads,
                "sample": f"scipy.linalg.lapack.dgeqrf (OpenBLAS) on the leading {m}x{ns} columns, {dt:.2f} s"}
    except Exception as e:
        return {"unavailable": f"{type(e).__name__}: {e}"}


def run_reference(args):
    """--impl reference: the reference's CPU path on the same config.  Julia is absent, so this is the oracle port (kind=port)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import dhqr_oracle as O
    co = O.COracle()
    m, n = args.m, args.n
    threads, logical = host_cores()
    threads = int(os.environ.get("DHQR_CPU_THREADS", "0")) or threads
    stride = cpu_stride(m, n)
    cpu_pass(co, (min(m, 4096), min(n, 256)), 0, 1, threads)
    fl = dt = 0.0
    for it in range(args.warmup + args.steps):
        f, d = cpu_pass(co, (m, n), it, stride, threads)
        if it >= args.warmup:
            fl, dt = fl + f, dt + d
    val = fl / dt / 1e9
    cb = {"value": val, "unit": "GFLOP/s", "cores": threads, "kind": "port",
          "sample": cpu_sample_desc(m, n, stride, threads, logical) + f"; {args.steps} timed passes, {dt:.1f} s"}
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": val, "unit": "GFLOP/s", "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(1, args.steps),
                      "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                      "config": make_config(m, n, args.gpus), "cpu_baseline": cb,
                      "e2e": {"value": val, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                      "gpu_launches": 0}))


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s of B200_PROFILING.md (of fallback: MEASURED_PEAKS.json absent on this box)"


def run_ours(args):
    import torch
    import torch.distributed as dist
    import dhqr_b200 as D

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        h = D.init_distributed(local)
    else:
        h = D.default_handle(local)

    m, n, nb = args.m, args.n, args.nb
    b = D.splits(world, n) if args.split == "even" else [128 * int(round(x / 128.0)) for x in D.balanced_splits(world, n, "trailing")]
    b[0], b[-1] = 0, n
    c0, nl = b[rank], b[rank + 1] - b[rank]
    flops = qr_flops(m, n)
    K, W = args.steps, args.warmup

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def red(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    def maxover(x):
        return red(x, dist.ReduceOp.MAX) if world > 1 else x

    def sumover(x):
        return red(x, dist.ReduceOp.SUM) if world > 1 else x

    # pool of fresh matrices so the timed region holds only qr! calls (inputs resident in HBM)
    pool_n = max(1, min(K, args.pool))
    pool = [D.colmajor_empty(m, nl, dev) for _ in range(pool_n)]
    alpha = torch.zeros(n, dtype=torch.float64, device=dev)

    def refill():
        for A in pool:
            D.fill_uniform_(A, 0, 0, c0, h)

    def step(A):
        D.householder_(D.ColumnBlockMatrix(A, n, c0, h) if world > 1 else A, alpha, nb, h)

    refill()
    for w in range(W):
        step(pool[w % pool_n])
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    total_ms, done = 0.0, 0
    launches = 0
    while done < K:
        g = min(pool_n, K - done)
        refill()
        barrier()
        la = h.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(g):
            step(pool[i])
        e1.record()
        barrier()
        total_ms += maxover(e0.elapsed_time(e1))
        launches += h.launch_count() - la
        done += g
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = total_ms / K
    value = flops / (ms_per_step * 1e-3) / 1e9
    launches_all = int(sumover(float(launches)))
    last = pool[(K - 1) % pool_n]                 # the last timed factorisation (alpha belongs to it)
    # taken before the legs below refactor pool[0] into the same alpha
    outputs = gather_outputs(torch, dist, last, alpha, m, n, c0, nl, world, dev) if args.dump_outputs else None

    # ---- parity of the last timed factorisation ------------------------------------------------------------------------
    parity = {"tolerance": 1e-13, "oracle_pin": ORACLE_PIN}
    if not args.no_check:
        try:
            parity["qr_residual_fro_rel"] = dist_residual(torch, dist, D, last, alpha, m, n, c0, nl, world, rank, dev, h, b)
        except Exception as e:
            sys.stderr.write(f"[bench] residual check failed on rank {rank}: {type(e).__name__}: {e}\n")
            parity["qr_residual_fro_rel"] = "check failed (see stderr)"
        if world > 1:
            # the same seed factored on ONE GPU (rank 0, private single-GPU handle): alpha must agree to rounding
            a1 = torch.zeros(n, dtype=torch.float64, device=dev)
            if rank == 0:
                h1 = D.Handle(local)
                A1 = D.colmajor_empty(m, n, dev)
                D.fill_uniform_(A1, 0, 0, 0, h1)
                D.householder_(A1, a1, nb, h1)
                torch.cuda.synchronize()
                del A1
                h1.close()
            dist.broadcast(a1, 0)
            parity["alpha_vs_single_gpu_inf_rel"] = maxover(float(((alpha - a1).abs().max() / a1.abs().max()).item()))
            parity["alpha_tolerance"] = 1e-12

    # ---- solve: warm H \ b on the last factorisation (S:317-321; the reference benchmarks qr!(A) \ b, T:66) ----------------
    solve = None
    if not args.no_solve:
        Hm = D.ColumnBlockMatrix(last, n, c0, h) if world > 1 else last
        bvec = torch.rand(m, dtype=torch.float64, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
        if world > 1:
            dist.broadcast(bvec, 0)
        work = bvec.clone()
        ks = 5
        tq = tb = 0.0
        for it in range(2 + ks):
            work.copy_(bvec)
            barrier()
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record()
            D.apply_qt_(work, Hm, h)
            e1.record()
            D.backsolve_(work, Hm, alpha, h)
            e2.record()
            barrier()
            if it >= 2:
                tq += maxover(e0.elapsed_time(e1))
                tb += maxover(e1.elapsed_time(e2))
        vbytes = 8.0 * (m * n - n * (n - 1) / 2.0)
        rbytes = 8.0 * n * (n - 1) / 2.0
        hp, hsrc = hbm_peak()
        solve = {"apply_qt_ms": tq / ks, "backsolve_ms": tb / ks, "ldiv_ms": (tq + tb) / ks,
                 "apply_qt_gbs": vbytes / (tq / ks * 1e-3) / 1e9, "apply_qt_frac_of_hbm": vbytes / (tq / ks * 1e-3) / 1e9 / hp,
                 "backsolve_gbs": rbytes / (tb / ks * 1e-3) / 1e9, "hbm_peak_gbs": hp, "hbm_peak_source": hsrc,
                 "algorithmic_bytes": {"apply_qt": vbytes, "backsolve": rbytes}, "nrhs": 1, "steps": ks,
                 "note": "warm, device-resident b; apply_qt reads every reflector once (S:232-242), back-substitution reads triu(R) (S:256-282)"}

    # ---- per-kernel-class profile (separate, untimed step) -> roofline of the dominant kernel ----
    h.set_option("profile", 1)
    refill()
    barrier()
    h.profile_reset()
    step(pool[0])
    torch.cuda.synchronize()
    prof = h.profile()
    h.set_option("profile", 0)
    roof = None
    if rank == 0:
        tot = sum(v["ms"] for v in prof.values())
        classes = {k: {"ms": round(v["ms"], 3), "count": v["count"],
                       "tflops": (v["work"] / (v["ms"] * 1e-3) / 1e12 if (k.startswith("k_gemm") or k in ("k_gram128", "k_vpk_rmul")) and v["ms"] > 0 else None)}
                   for k, v in prof.items()}
        if nb == 1:
            # unblocked column loop: one read + one write of the trailing matrix per reflector (S:198-213), HBM/L2 bound
            E = sum((m - j) * (n - j - 1) for j in range(n)) + sum(m - j for j in range(n))
            gbs = 16.0 * E / (ms_per_step * 1e-3) / 1e9
            hp, hsrc = hbm_peak()
            dom = "k_apply1_tma" if "k_apply1_tma" in prof else max(prof, key=lambda k: prof[k]["ms"])
            timed_kernel = ("k_unblocked_wave (the whole column loop as ONE persistent launch; `classes` below profiles the "
                            "one-launch-per-column path the profiler needs)") if m <= 8192 and world == 1 else dom
            roof = {"bound": "hbm", "kernel": timed_kernel, "achieved": gbs, "peak": hp, "unit": "GB/s", "frac": gbs / hp, "traffic": None,
                    "algorithmic_bytes_per_step": 16.0 * E, "peak_source": hsrc,
                    "note": "whole-factorisation algorithmic bytes / ms_per_step; the 64 MiB matrix is L2-resident (126 MB L2), so DRAM traffic is far below the algorithmic bytes and the fraction can exceed what HBM alone would allow",
                    "share_of_step": prof[dom]["ms"] / tot if tot else None, "classes": classes}
        else:
            peak = dgemm_peak(torch, dev)
            dom = max((k for k in prof if k.startswith("k_gemm")), key=lambda k: prof[k]["ms"], default=None)
            if dom:
                ach = prof[dom]["work"] / (prof[dom]["ms"] * 1e-3) / 1e12
                traffic, tnote = None, None
                try:
                    tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))[dom]
                    traffic, tnote = tj["dram_bytes_per_launch"], f"dram bytes of the largest launch ({tj['captured_launch']}), ncu --set full, {tj['source']}"
                except Exception:
                    pass
                roof = {"bound": "tensor", "kernel": dom, "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                        "traffic": traffic, "traffic_note": tnote,
                        "peak_source": "cuBLAS DGEMM 8192^3 burst measured in this run (MEASURED_PEAKS.json has no fp64 entry); tcgen05 has no f64 kind, the fp64 tensor pipe is DMMA",
                        "launches": prof[dom]["count"], "avg_launch_ms": prof[dom]["ms"] / max(1, prof[dom]["count"]),
                        "share_of_step": prof[dom]["ms"] / tot if tot else None,
                        "whole_qr_frac_of_peak": value / 1e3 / peak / world, "classes": classes}
                # what the library itself reaches at the two bulk shapes of step 0 (K = nb = 128 for C += V Y; a 128-row output for
                # W = V'C): a comparator for the shape, not a roofline denominator
                try:
                    roof["cublas_same_shape"] = cublas_bulk_shapes(torch, dev, m, max(nl - 3 * (nb or 128), 128), nb or 128)
                    roof["cublas_same_shape"]["note"] = ("cuBLAS DGEMM (torch fp64 addmm / mm) at the shapes of the step-0 bulk update; "
                                                         "k_gemm_cvy128 / k_gemm_vta128 averages above are over all 31 launches of the sweep")
                except Exception as ex:   # a comparator only: never fail the bench line on it
                    roof["cublas_same_shape"] = {"error": str(ex)[:200]}

    # ---- e2e: host buffers through the reference-facing entry ----
    e2e = None
    if not args.no_e2e:
        hostA = torch.empty((nl, m), dtype=torch.float64).pin_memory().t()      # column-major pinned (m, nl)
        src = D.colmajor_empty(m, nl, dev)
        D.fill_uniform_(src, 0, 0, c0, h)
        hostA.copy_(src)
        pristine = hostA.clone()
        host_alpha = torch.empty(n, dtype=torch.float64).pin_memory()
        Ke = max(1, args.e2e_steps)
        tot_s = 0.0
        # Host-side analogue of the L2 flush between device-timed iterations: after the CPU has rewritten the pinned buffer a good part of
        # it sits dirty in the CPU caches, and DMA reads of such lines are slower and noisy (3-8 ms per step, profiles/r02b_host_pipeline.txt).
        # Writing a scratch buffer larger than the last-level caches puts the input where a matrix that did not just come out of this
        # process's own memcpy would be: in DRAM.  Outside the timed region; the dirty-cache case is reported next to the headline.
        flush = torch.empty(1 << 27, dtype=torch.float64)
        for it in range(2 + Ke):
            hostA.copy_(pristine)
            flush.fill_(float(it))
            barrier()
            t0 = time.perf_counter()
            if world == 1:
                import ctypes as C
                D._lib.call("dhqr_qr_host_f64", h.raw, m, n, C.c_void_p(hostA.data_ptr()), m, C.c_void_p(host_alpha.data_ptr()), nb)
            else:
                dA = pool[0]
                dA.copy_(hostA, non_blocking=True)
                step(dA)
                hostA.copy_(dA, non_blocking=True)
                host_alpha.copy_(alpha, non_blocking=True)
                torch.cuda.synchronize()
            dt = maxover(time.perf_counter() - t0)
            if it >= 2:
                tot_s += dt
        e2e = {"value": flops / (tot_s / Ke) / 1e9, "unit": "GFLOP/s", "h2d_bytes_per_step": int(sumover(float(m * nl * 8))),
               "d2h_bytes_per_step": int(sumover(float(m * nl * 8))) + n * 8, "ms_per_step": 1e3 * tot_s / Ke, "steps": Ke, "warmup": 2,
               "path": "dhqr_qr_host_f64 (C-ABI, pinned host buffers)" if world == 1 else "pinned host block -> qr_ -> host (per rank)",
               "input": "pinned host buffer rewritten by the CPU (copy from a pageable tensor) before every step, then the CPU caches flushed by "
                        "writing a 1 GiB scratch buffer (the input sits in DRAM); both outside the timed region"}
        if world == 1:
            # the same call in the two other states of the pinned buffer: still dirty in the CPU caches (rewritten by the CPU, no flush),
            # and last written by a device-to-host copy (as if it had arrived by DMA from a NIC or a disk)
            def e2e_variant(refresh):
                import ctypes as C
                tot2, K2 = 0.0, 4
                for it in range(1 + K2):
                    refresh()
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    D._lib.call("dhqr_qr_host_f64", h.raw, m, n, C.c_void_p(hostA.data_ptr()), m, C.c_void_p(host_alpha.data_ptr()), nb)
                    if it >= 1:
                        tot2 += time.perf_counter() - t0
                return {"ms_per_step": 1e3 * tot2 / K2, "value": flops / (tot2 / K2) / 1e9, "steps": K2}
            for key, refresh in (("input_dirty_in_cpu_caches", lambda: hostA.copy_(pristine)), ("input_written_by_dma", lambda: hostA.copy_(src))):
                try:
                    e2e[key] = e2e_variant(refresh)
                except Exception as ex:       # side figures only: never fail the bench line on them
                    e2e[key] = {"error": str(ex)[:200]}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_port_baseline(m, n)
        cpu["lapack_dgeqrf"] = lapack_baseline(m, n, cpu["cores"])

    if rank == 0:
        cfg = make_config(m, n, world)
        out = {"metric": METRIC, "value": value, "unit": "GFLOP/s", "n_gpus": world, "steps": K, "warmup": W,
               "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
               "dtype": "f64", "data": "synthetic", "config": cfg,
               "impl_details": {"nb": nb or 128, "cols_per_gpu": nl, "column_boundaries": b, "split": args.split, "wide_panels": h.get_option("wide_panels"),
                                "wide_redone": h.get_option("wide_redone"), "baseline_config": args.config},
               "clocks": clocks, "gpu_launches": launches_all, "e2e": e2e, "roofline": roof, "cpu_baseline": cpu,
               "solve": solve, "parity": parity}
        if outputs is not None:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
        print(json.dumps(out))
    if world > 1:
        D.shutdown_distributed()
        dist.destroy_process_group()


def dist_residual(torch, dist, D, Hloc, alpha, m, n, c0, nl, world, rank, dev, h, bnd):
    """||QR - A0||_F / ||A0||_F.  Every rank rebuilds ITS columns of Q R from all the reflectors (gathered panel by panel from
    their owners) in torch fp64 on the GPU, compares with its regenerated columns of A0, and the squared norms are summed
    over ranks.  Size independent; a wrong or wrongly ordered V anywhere shows up here (unlike a column-norm check)."""
    R = torch.zeros(m, nl, dtype=torch.float64, device=dev)
    gl = torch.arange(c0, c0 + nl, device=dev)
    rows = torch.arange(n, device=dev)
    Rtop = torch.where(rows[:, None] < gl[None, :], Hloc[:n], torch.zeros((), dtype=torch.float64, device=dev))
    R[:n] = Rtop
    if nl:
        R[gl, torch.arange(nl, device=dev)] = alpha[c0:c0 + nl]
    panels = []
    for r in range(world):
        for o in range(bnd[r], bnd[r + 1], 128):
            panels.append((r, o, min(128, bnd[r + 1] - o)))
    for owner, k, kb in reversed(panels):                       # Q R = H_1 (H_2 (... H_n R))
        if world > 1:
            V = torch.empty(m - k, kb, dtype=torch.float64, device=dev)
            if owner == rank:
                V.copy_(Hloc[k:, k - c0:k - c0 + kb])
            dist.broadcast(V, owner)
        else:
            V = Hloc[k:, k:k + kb]
        V = torch.tril(V)
        Tinv = torch.eye(kb, dtype=torch.float64, device=dev) + torch.triu(V.T @ V, 1)      # T^{-1} = I + striu(V'V)
        if nl:
            R[k:] -= V @ torch.linalg.solve_triangular(Tinv, V.T @ R[k:], upper=True)
    A0 = D.colmajor_empty(m, nl, dev)
    D.fill_uniform_(A0, 0, 0, c0, h)
    num = float(((R - A0) ** 2).sum().item()) if nl else 0.0
    den = float((A0 ** 2).sum().item()) if nl else 0.0
    if world > 1:
        t = torch.tensor([num, den], dtype=torch.float64, device=dev)
        dist.all_reduce(t)
        num, den = float(t[0].item()), float(t[1].item())
    return (num / den) ** 0.5


DUMP_A_BYTES = 48 << 20          # keeps a dump under 64 MB with alpha (8n bytes) beside it


def dump_columns(m, n):
    """Global columns of the factored A that --dump-outputs writes: all of them when they fit in DUMP_A_BYTES, else a
    sorted sample drawn with a fixed seed, so that every run with the same m and n writes the same columns."""
    import numpy as np
    k = min(n, max(1, DUMP_A_BYTES // (8 * m)))
    if k == n:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))


def gather_outputs(torch, dist, Hloc, alpha, m, n, c0, nl, world, dev):
    """The arrays qr!(A) hands back, as host arrays: the factored A at the columns of dump_columns, and alpha (replicated
    on every rank).  Each rank fills the sampled columns it owns and a sum over ranks assembles them."""
    cols = dump_columns(m, n)
    S = torch.zeros(m, len(cols), dtype=torch.float64, device=dev)
    mine = [(s, int(j) - c0) for s, j in enumerate(cols) if c0 <= j < c0 + nl]
    if mine:
        dst, src = zip(*mine)
        S[:, list(dst)] = Hloc[:, list(src)]
    if world > 1:
        dist.all_reduce(S)
    return {"A": S.cpu().numpy(), "alpha": alpha.cpu().numpy()}


def dgemm_peak(torch, dev, nn=8192):
    a = torch.rand(nn, nn, dtype=torch.float64, device=dev)
    b = torch.rand(nn, nn, dtype=torch.float64, device=dev)
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return 2.0 * nn ** 3 / (best * 1e-3) / 1e12


def cublas_bulk_shapes(torch, dev, rows, ncols, nb):
    """TFLOP/s of cuBLAS DGEMM at the two bulk-update shapes: C(rows x ncols) += V(rows x nb) Y(nb x ncols) and W(nb x ncols) = V'C."""
    V = torch.rand(nb, rows, dtype=torch.float64, device=dev)       # = V' row-major, i.e. V column-major
    Y = torch.rand(ncols, nb, dtype=torch.float64, device=dev)      # = Y' row-major
    Ct = torch.rand(ncols, rows, dtype=torch.float64, device=dev)   # = C' row-major, i.e. C column-major

    def best_ms(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        best = 1e30
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return best
    fl = 2.0 * rows * ncols * nb
    t_cvy = best_ms(lambda: torch.addmm(Ct, Y, V, out=Ct))           # C' += Y'V'  (K = nb)
    t_vta = best_ms(lambda: torch.mm(V, Ct.t()))                      # W = V'C     (K = rows)
    return {"rows": rows, "ncols": ncols, "k": nb, "cvy_tflops": fl / (t_cvy * 1e-3) / 1e12, "vta_tflops": fl / (t_vta * 1e-3) / 1e12}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=[2, 3], help="BASELINE.json config (1-based): 3 = 32768x4096 blocked (default, the metric's config), 2 = 8192x1024 unblocked")
    ap.add_argument("--m", type=int, default=0)
    ap.add_argument("--n", type=int, default=0)
    ap.add_argument("--nb", type=int, default=-1)
    ap.add_argument("--pool", type=int, default=8)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--no-solve", action="store_true")
    ap.add_argument("--split", default="even", choices=["even", "balanced"],
                    help="column blocks: DArray default (even) or the reference's load-balanced contiguous split (T:35), rounded to panels")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the factored A (column sample) and alpha of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours: the reference arm times a strided sample of the column sweep, not a whole qr!")
    dm, dn, dnb = (8192, 1024, 1) if args.config == 2 else (32768, 4096, 0)
    args.m, args.n = args.m or dm, args.n or dn
    args.nb = dnb if args.nb < 0 else args.nb
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
