#!/usr/bin/env python3
"""bench.py — objective+gradient evaluations/sec of the traceobjgrad hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cnot2] [--batch B] [--impl reference] [--dump-outputs DIR]

One "step" = one batched obj+grad evaluation (`jq_traceobjgrad_batch`) of B synthetic pcof candidates per GPU on the
named BASELINE configuration (default: cnot2, "batched random pcof evaluations").  Ranks shard the candidates
(weak scaling, no data-path collective).  Prints ONE JSON line on rank 0.

  value     device-resident throughput: inputs already in HBM, CUDA events on the launching stream, max over ranks
  e2e       same metric through the host-pointer C-ABI call (pinned host buffers, H2D + D2H inside the timed region)
  roofline  algorithmic FP64 flops (SURVEY.md 8d formula) / kernel time, against the FP64 FMA peak measured in-run
  cpu_baseline   the CPU oracle (a port: the Julia reference cannot run in this image) on a bounded sample
  extra.per_config (N = 1)   every named BASELINE shape — rabi, cnot1, cnot2, cnot3, risk-neutral 9-node quadrature x B
            candidates, the 1001-point epsilon sweep — with evals/s, roofline fractions and ITS OWN bounded CPU baseline
  extra.single_eval_latency (N = 1)   one pcof per call, the reference's real call pattern (Ipopt callback)
  extra.risk_neutral_sample_sharded   noise samples sharded over the ranks + the path's one NCCL all-reduce per evaluation:
            weak (16384 samples per GPU) and strong (16384 samples in total; the 1001-point sweep) scaling, and a parity
            self-check of the sharded + all-reduced result against one rank evaluating every sample (<= 1e-12)
  --impl reference   the same oracle with every host thread, as the reference arm
  --dump-outputs DIR   after the timed steps, the arrays the last timed step returned (infid, leak, trace_infid, grad, and
            infidgrad / leakgrad when objFuncType != 1) as DIR/<name>.npy in float64, so that two builds can be compared output for
            output on the same seeded inputs; above DUMP_BYTES a fixed, seeded sample of the candidates is written
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

WORKLOADS = ["rabi", "cnot1", "cnot2", "cnot3", "risk_neutral"]
# candidates per GPU per step: multiples of the resident-CTA wave of the kernel that serves the shape
DEFAULT_BATCH = {"rabi": 262144, "cnot1": 37888, "cnot2": 16384, "cnot3": 2368, "risk_neutral": 3946}
KERNEL_NAMES = {1: "jq_generic_kernel", 2: "jq_traj_kernel<SlotLane>", 3: "jq_traj_kernel<FiberLane>", 4: "jq_traj_kernel<TileLane>", 5: "jq_traj_kernel<latency layout, pipelined roles>", 6: "jq_dense_kernel (FP64 MMA)",
                7: "time-parallel: jq_traj_kernel<segment sweeps> + jq_seg_chain joins"}
DUMP_BYTES = 64_000_000          # --dump-outputs: bytes written per run, .npy headers included


def dump_outputs(out, directory, suffix="", budget=DUMP_BYTES):
    """Write the CUDA tensors of one evaluate_device() result as <directory>/<name><suffix>.npy (float64).  When they exceed `budget`
    bytes, only a sample of the candidates (first axis) is written: the same rows, in ascending order, for every run with the same
    arguments.  Returns what was written, for the JSON line."""
    arrs = {k: v.cpu().numpy() for k, v in out.items()}
    nbatch = next(iter(arrs.values())).shape[0]
    total = sum(a.nbytes for a in arrs.values())
    room = budget - 256 * len(arrs)                    # an .npy header takes 128 bytes here; leave twice that
    rows = None
    if total > room:
        rows = np.sort(np.random.default_rng(0).choice(nbatch, nbatch * room // total, replace=False))
        arrs = {k: a[rows] for k, a in arrs.items()}
    os.makedirs(directory, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(directory, f"{k}{suffix}.npy"), a)
    return {"dir": directory, "arrays": {k + suffix: list(a.shape) for k, a in arrs.items()},
            "candidates_written": nbatch if rows is None else len(rows), "candidates": nbatch,
            "sample": None if rows is None else "rows np.sort(np.random.default_rng(0).choice(candidates, candidates_written, replace=False))"}


def alg_flops_per_eval(p, npar, dense=False):
    """SURVEY.md section 8(d): algorithmic flops of one obj+grad evaluation (structural nonzeros, FMA = 2).
    dense=True: the same scheme with every operator product counted as a full n x n contraction (what a
    tensor-core formulation would have to execute)."""
    n, m, J, Nc, Nf = p.Ntot, p.N, p.linear_solver.max_iter, p.Ncoupled, p.Nfreq
    h0 = np.asarray(p.Hconst)
    nnzK = n + int(np.count_nonzero(h0 - np.diag(np.diag(h0)))) + sum(int(np.count_nonzero(h)) for h in p.Hsym_ops)
    nnzS = sum(int(np.count_nonzero(h)) for h in p.Hanti_ops)
    nnzq = [int(np.count_nonzero(h)) for h in p.Hsym_ops]
    if dense:
        nnzK, nnzS, nnzq = n * n, n * n, [n * n] * Nc
    f_state = 2 * m * (4 * nnzK + (4 + 2 * J) * nnzS) + (9 + 4 * J) * n * m
    f_adj = 2 * m * (4 * nnzK + (4 + 2 * J) * nnzS) + (16 + 4 * J) * n * m
    f_pen = 6 * n * m
    f_grad = sum(12 * m * z for z in nnzq) + 16 * n * m + 96 * Nc * Nf
    f_ctrl = 160 * Nc * Nf + 8 * sum(nnzq)
    return p.nsteps * ((f_state + f_pen + f_ctrl) + (f_state + f_adj + f_grad + f_ctrl))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_baseline_run(cfg, pcof, shifts, nthreads, budget_s):
    """Time the oracle on a bounded sample of the same workload; returns (evals_per_sec, n_evals, seconds)."""
    from oracle import oracle_traceobjgrad
    nsamp = 1 if shifts is None else len(shifts)
    t0 = time.perf_counter()
    oracle_traceobjgrad(cfg.params, pcof[:1], None if shifts is None else shifts[:1], nthreads=1)
    t_one = time.perf_counter() - t0
    ncand = int(max(1, min(len(pcof), (budget_s / max(t_one, 1e-6)) * nthreads / nsamp)))
    ncand = max(ncand, min(len(pcof), -(-nthreads // nsamp)))      # at least one trajectory per thread
    t0 = time.perf_counter()
    oracle_traceobjgrad(cfg.params, pcof[:ncand], shifts, nthreads=nthreads)
    dt = time.perf_counter() - t0
    return ncand * nsamp / dt, ncand * nsamp, dt


def ncu_summary(workload):
    """Per-launch DRAM traffic and executed-FP64-flop fraction from the committed `ncu --set full` captures (profiles/)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_summary.json"))).get(workload)
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cnot2", choices=WORKLOADS)
    ap.add_argument("--batch", type=int, default=0, help="pcof candidates per GPU per step (0 = per-workload default)")
    ap.add_argument("--kernel", type=int, default=0, help="0 auto, 1 generic, 2 slot layout, 3 fibre layout, 4 tile layout")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU work for the cpu_baseline sample")
    ap.add_argument("--per-config-cpu-budget", type=float, default=2.5, help="seconds of CPU work per extra.per_config baseline")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the arrays the last timed step returned as DIR/<name>.npy (float64; a seeded sample of the candidates "
                         "above 64 MB); with several ranks each rank writes <name>_rank<r>.npy")
    args = ap.parse_args()
    if args.impl != "reference" and args.warmup < 3:
        args.warmup = 3          # timing rules: at least 3 warm-up steps; the JSON line reports the value actually used
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed; the reference arm has no timed GPU step")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    from juqbox_b200 import configs
    cfg = configs.example(args.workload)
    B = args.batch or DEFAULT_BATCH[args.workload]
    shifts_h = configs.noise_shift(cfg.params.Ntot, cfg.nodes) if args.workload == "risk_neutral" else None
    nsamp = 1 if shifts_h is None else len(shifts_h)
    npar = cfg.nCoeff
    workload = {"workload": f"{args.workload} (examples/{'Risk_Neutral/swap-02-risk-neutral' if args.workload == 'risk_neutral' else args.workload + '-setup'}.jl, Stormer-Verlet)",
                "n": cfg.params.Ntot, "m": cfg.params.N, "nsteps": cfg.params.nsteps, "neumann_terms": cfg.params.linear_solver.max_iter,
                "npar": npar, "candidates_per_gpu": B, "noise_samples": nsamp, "state_steps_per_eval": 3 * cfg.params.nsteps,
                "l2": "flushed (256 MiB write) between timed steps"}

    # ------------------------------------------------------------------ reference arm: CPU oracle, all host threads
    if args.impl == "reference":
        if rank != 0:
            return 0
        from oracle import max_threads
        nthr = max_threads()
        pc = configs.synthetic_pcof(cfg, B)
        vals, sample = [], None
        budget = max(2.0, min(30.0, 150.0 / max(1, args.steps + args.warmup)))
        for it in range(args.warmup + args.steps):
            v, ne, dt = cpu_baseline_run(cfg, pc, shifts_h, nthr, budget)
            sample = f"{ne} obj+grad evaluations of the {B}-candidate batch per step, {nthr} threads"
            if it >= args.warmup:
                vals.append((ne, dt))
        tot_e, tot_t = sum(v[0] for v in vals), sum(v[1] for v in vals)
        val = tot_e / tot_t
        print(json.dumps({"impl": "reference", "metric": "objective+gradient evals/sec (traceobjgrad)", "value": val, "unit": "evals/s",
                          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(1, args.steps),
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                          "config": workload,
                          "cpu_baseline": {"value": val, "unit": "evals/s", "cores": nthr, "kind": "port", "sample": sample},
                          "e2e": {"value": val, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0

    # ------------------------------------------------------------------ our arm
    import torch
    import torch.distributed as dist
    import juqbox_b200 as jq
    from juqbox_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    launches = 0                                         # kernels of this library launched inside timed regions
    wa = jq.Working_Arrays(cfg.params, npar, device=local_rank)
    wa.set_kernel(args.kernel)
    pc_h = configs.synthetic_pcof(cfg, B, seed_offset=rank)
    pc_d = torch.from_numpy(pc_h).to(dev)
    sh_d = torch.from_numpy(shifts_h).to(dev) if shifts_h is not None else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)
    out = None

    def step():
        nonlocal out
        out = wa.evaluate_device(pc_d, sh_d, None, True, out=out, stream=stream)

    for _ in range(args.warmup):
        flush.fill_(1)
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kernel_ms = []
    barrier()
    for e0, e1 in evs:
        flush.fill_(1)
        e0.record(stream)
        step()
        e1.record(stream)
        kernel_ms.append(wa.last_kernel_ms)      # library's own events around the trajectory kernel (synchronises)
    barrier()
    dumped = None
    if args.dump_outputs:
        dumped = dump_outputs(out, args.dump_outputs, f"_rank{rank}" if world > 1 else "", DUMP_BYTES // world)
    launches += 2 * args.steps
    total_ms = max_over_ranks(sum(e0.elapsed_time(e1) for e0, e1 in evs))
    evals_per_step = world * B * nsamp
    value = evals_per_step * args.steps / (total_ms * 1e-3)
    kern_ms = float(np.mean(kernel_ms))
    used_kernel = wa.last_kernel

    # ---- end to end through the host-pointer C ABI, pinned host buffers
    pin_in = torch.from_numpy(pc_h).pin_memory()
    pc_pin = pin_in.numpy()
    pins = {k: torch.zeros((B, nsamp) + ((npar,) if k == "grad" else ()), dtype=torch.float64).pin_memory()
            for k in ("infid", "leak", "trace_infid", "grad")}          # pinned result buffers, reused like Working_Arrays
    r = {k: v.numpy() for k, v in pins.items()}
    for _ in range(1):
        r = wa.evaluate(pc_pin, shifts_h, out=r)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r = wa.evaluate(pc_pin, shifts_h, out=r)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches += 2 * args.steps
    e2e_val = evals_per_step * args.steps / e2e_s
    h2d = pc_pin.nbytes + (shifts_h.nbytes if shifts_h is not None else 0)
    d2h = sum(r[k].nbytes for k in ("infid", "leak", "trace_infid", "grad"))       # objFuncType 1: infidgrad aliases grad

    # ---- roofline of the dominant (trajectory) kernel
    flops_eval = alg_flops_per_eval(cfg.params, npar)
    peak = _lib.fp64_peak_tflops(local_rank)
    peak3 = _lib.fp64_peak_tflops(local_rank, three_operand=True)
    achieved = flops_eval * B * nsamp / (kern_ms * 1e-3) / 1e12
    peak_dmma = _lib.fp64_peak_tflops(local_rank, tensor=True)
    dense_ratio = alg_flops_per_eval(cfg.params, npar, dense=True) / flops_eval
    ns = ncu_summary(args.workload)
    same_launch = bool(ns and ns.get("evals_per_launch") == B * nsamp and ns.get("kernel") == used_kernel)
    roofline = {"bound": "fp64_fma",
                "bound_note": "compute roofline in TFLOP/s (the contract's 'tensor' class), but on the FP64 FMA pipe: B200 has no faster "
                              "FP64 tensor path (tensor_pipe below), and HBM carries ~1 KB per 1.4e8-flop evaluation (traffic)",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
                "traffic": ns["dram_bytes_per_launch"] if same_launch else None,
                "peak_source": "jq_fp64_peak DFMA micro-benchmark measured in this run (MEASURED_PEAKS.json has no FP64 entry); "
                               "against ncu's dfma peak_sustained (64/clk/SM x 148 SMs x sm_mhz) the fraction is frac_vs_ncu_sustained_peak",
                "frac_vs_ncu_sustained_peak": (achieved / (2 * 64 * 148 * clocks["sm_mhz"] * 1e-6)) if clocks and clocks.get("sm_mhz") else None,
                "executed_fp64_frac_ncu": ns.get("executed_fp64_flop_frac") if ns else None,
                "peak_no_operand_reuse": peak3, "frac_of_peak_no_operand_reuse": achieved / peak3 if peak3 else None,
                "tensor_pipe": {"util": 0.0, "fp64_mma_peak": peak_dmma, "dense_to_nnz_flop_ratio": dense_ratio,
                                "nnz_equivalent_ceiling": peak_dmma / dense_ratio if dense_ratio else None,
                                "note": "FP64 MMA (mma.sync m16n8k16) peak measured in this run; a dense contraction executes "
                                        "dense_to_nnz_flop_ratio x the structural flops, so its ceiling in this line's units is "
                                        "nnz_equivalent_ceiling TFLOP/s; the path stays on the DFMA pipe when that is below `achieved`"},
                "alg_flops_per_eval": flops_eval, "kernel_ms": kern_ms, "kernel": KERNEL_NAMES[used_kernel],
                "hbm_alg_bytes_per_launch": 8 * (B * npar + nsamp * cfg.params.Ntot + B * nsamp * (4 + npar))}

    # ---- CPU baseline (rank 0, N = 1 only)
    cpu = None
    nthr = 1
    if rank == 0 and world == 1:
        from oracle import max_threads
        v1, ne1, dt1 = cpu_baseline_run(cfg, pc_h, shifts_h, 1, args.cpu_budget * 0.4)
        nthr = max_threads()
        vN, neN, dtN = cpu_baseline_run(cfg, pc_h, shifts_h, nthr, args.cpu_budget)
        cpu = {"value": vN, "unit": "evals/s", "cores": nthr, "kind": "port",
               "sample": f"{neN} obj+grad evaluations from the same batch in {dtN:.1f}s on {nthr} threads (pthread pool over trajectories)",
               "single_thread": {"value": v1, "cores": 1, "sample": f"{ne1} evaluations in {dt1:.1f}s"}}

    def time_launches(fn, reps):
        """CUDA-event time per call of `fn` on `stream`, max over ranks, after one warm-up call."""
        fn()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(reps):
            fn()
        b.record(stream)
        barrier()
        return max_over_ranks(a.elapsed_time(b)) / reps

    extra = {}
    # ---- extra.per_config: every named shape at 1 GPU with its own CPU baseline (north_star: "each named problem shape ...
    #      CPU path timed in the same run")
    if not args.no_extra and world == 1:
        per = {}
        legs = [(n, None) for n in WORKLOADS] + [("risk_neutral", "sweep1001")]
        for name, variant in legs:
            c = configs.example(name)
            Bc = DEFAULT_BATCH[name]
            sh = wts = None
            label = name
            if name == "risk_neutral" and variant is None:
                sh = configs.noise_shift(c.params.Ntot, c.nodes)             # 9 Gauss-Legendre nodes (swap-02-risk-neutral.jl:45-49)
                label = "risk_neutral_9node"
            elif variant == "sweep1001":
                eps = np.linspace(-2 * np.pi * 3e-2, 2 * np.pi * 3e-2, 1001)   # examples/Risk_Neutral/run_all.jl:70-72
                sh = configs.noise_shift(c.params.Ntot, eps)
                Bc, label = 1, "risk_neutral_sweep1001"
            ns_c = 1 if sh is None else len(sh)
            pch = configs.synthetic_pcof(c, Bc)
            w2 = jq.Working_Arrays(c.params, c.nCoeff, device=local_rank)
            pcd = torch.from_numpy(pch).to(dev)
            shd = torch.from_numpy(sh).to(dev) if sh is not None else None
            o2 = None

            def leg():
                nonlocal o2
                o2 = w2.evaluate_device(pcd, shd, None, True, out=o2, stream=stream)
            reps = 2 if name == "cnot3" else 3
            leg()
            kms = []
            for _ in range(reps):
                flush.fill_(1)
                leg()
                kms.append(w2.last_kernel_ms)
            launches += 2 * reps
            kms = float(np.mean(kms))
            fl = alg_flops_per_eval(c.params, c.nCoeff)
            ev = Bc * ns_c / (kms * 1e-3)
            vC, neC, dtC = cpu_baseline_run(c, pch, sh, nthr, args.per_config_cpu_budget)
            nsum = ncu_summary(label) or ncu_summary(name)
            per[label] = {"candidates": Bc, "noise_samples": ns_c, "n": c.params.Ntot, "m": c.params.N, "nsteps": c.params.nsteps,
                          "kernel": KERNEL_NAMES[w2.last_kernel], "kernel_ms": kms, "evals_per_sec": ev,
                          "state_steps_per_sec": ev * 3 * c.params.nsteps, "alg_tflops": ev * fl / 1e12,
                          "frac": ev * fl / 1e12 / peak, "executed_fp64_frac_ncu": nsum.get("executed_fp64_flop_frac") if nsum else None,
                          "cpu_baseline": {"value": vC, "unit": "evals/s", "cores": nthr, "kind": "port",
                                           "sample": f"{neC} evaluations in {dtC:.1f}s"},
                          "speedup_vs_cpu_all_threads": ev / vC}
            w2.close()
        extra["per_config"] = per

        # ---- one pcof per call: the reference's own call pattern (eval_f_g_grad! from an Ipopt callback).  Automatic mode takes the
        # time-parallel evaluation (kernel 7); the single-sweep latency kernel (5) is timed beside it and must agree to 1e-12
        lat = {}
        from oracle import oracle_traceobjgrad
        for name in ("cnot1", "cnot2", "cnot3", "risk_neutral"):
            c = configs.example(name)
            sh = configs.noise_shift(c.params.Ntot, c.nodes) if name == "risk_neutral" else None
            wts = c.weights if name == "risk_neutral" else None
            w2 = jq.Working_Arrays(c.params, c.nCoeff, device=local_rank)
            p1 = configs.synthetic_pcof(c, 1)
            row, results = {}, {}
            for kern in (0, 5):
                try:
                    w2.set_kernel(kern)
                except Exception:
                    continue
                results[kern] = w2.evaluate(p1, sh, wts)
                ts = []
                for _ in range(3):
                    t0 = time.perf_counter()
                    w2.evaluate(p1, sh, wts)
                    ts.append((time.perf_counter() - t0) * 1e3)
                launches += 4 * int(w2.query(2))
                key = "automatic" if kern == 0 else "single_sweep"
                row[key] = {"kernel": KERNEL_NAMES[w2.last_kernel], "kernel_ms": w2.last_kernel_ms, "host_call_ms": min(ts),
                            "launches": int(w2.query(2)), "time_segments": int(w2.query(7))}
            if 0 in results and 5 in results:
                g0, g5 = results[0]["grad"].ravel(), results[5]["grad"].ravel()
                row["rel_grad_diff"] = float(np.linalg.norm(g0 - g5) / np.linalg.norm(g5))
                row["abs_infid_diff"] = float(np.abs(results[0]["infid"] - results[5]["infid"]).max())
            t0 = time.perf_counter()
            oracle_traceobjgrad(c.params, p1, sh, nthreads=min(nthr, 1 if sh is None else len(sh)))
            row.update({"trajectories": 1 if sh is None else len(sh), "cpu_ms": (time.perf_counter() - t0) * 1e3,
                        "cpu_threads": min(nthr, 1 if sh is None else len(sh))})
            lat[name] = row
            w2.close()
        extra["single_eval_latency"] = lat

    # ---- extra: risk-neutral evaluation with the sample shard + NCCL all-reduce (the path's one exchange step)
    if not args.no_extra:
        rn = configs.example("risk_neutral")
        ep_max = 2 * np.pi * 2e-2
        wr = jq.Working_Arrays(rn.params, rn.nCoeff, device=local_rank)
        if world > 1:
            wr.comm_init(rank, world)                        # the library's own NCCL communicator (jq_comm_init)
        pcr_h = configs.synthetic_pcof(rn, 1)
        pcr = torch.from_numpy(pcr_h).to(dev)

        def sharded_leg(nodes, weights, reps):
            """Each rank evaluates its contiguous shard of (nodes, weights); the call ends with the library's one grouped
            ncclAllReduce(sum) of 3 + Npar doubles.  Returns (ms per risk-neutral evaluation, result dict of this rank)."""
            per_rank = -(-len(nodes) // world)
            sl = slice(rank * per_rank, min(len(nodes), (rank + 1) * per_rank))
            shr = torch.from_numpy(configs.noise_shift(rn.params.Ntot, nodes[sl])).to(dev)
            wtr = torch.from_numpy(np.ascontiguousarray(weights[sl])).to(dev)
            res = {}

            def f():
                res["o"] = wr.evaluate_device(pcr, shr, wtr, True, out=res.get("o"), stream=stream)
            ms = time_launches(f, reps)
            return ms, res["o"]

        def midpoint(S):
            # uniform additive noise on +-ep_max/2 (BASELINE config 5), midpoint rule: node k of S, weight 1/S
            return (np.arange(S) + 0.5) / S * ep_max - 0.5 * ep_max, np.full(S, 1.0 / S)

        S = 16384                                            # noise samples per GPU (weak scaling)
        nodes, weights = midpoint(S * world)
        ms, o = sharded_leg(nodes, weights, args.steps)
        launches += 2 * args.steps
        rnleg = {"samples_per_gpu": S, "evals_per_sec": world * S / (ms * 1e-3), "ms_per_risk_neutral_evaluation": ms,
                 "allreduce_doubles": 3 + rn.nCoeff,
                 "collective": "ncclAllReduce(sum, f64) inside jq_traceobjgrad_batch_device" if world > 1 else "none (1 GPU)",
                 "objective": float(o["infid"][0].item() + o["leak"][0].item())}
        if rank == 0 and world == 1:
            vC, neC, dtC = cpu_baseline_run(rn, pcr_h, configs.noise_shift(rn.params.Ntot, nodes[:1024]), nthr, args.per_config_cpu_budget)
            rnleg["cpu_baseline"] = {"value": vC, "unit": "evals/s", "cores": nthr, "kind": "port",
                                     "sample": f"{neC} sample evaluations (first 1024 nodes, one pcof) in {dtC:.1f}s"}
            rnleg["speedup_vs_cpu_all_threads"] = rnleg["evals_per_sec"] / vC
        # strong scaling: the same 16384 samples in total, and the reference's own 1001-point epsilon sweep
        nodes_s, weights_s = midpoint(S)
        ms_s, _ = sharded_leg(nodes_s, weights_s, args.steps)
        eps = np.linspace(-2 * np.pi * 3e-2, 2 * np.pi * 3e-2, 1001)
        ms_w, _ = sharded_leg(eps, np.full(1001, 1.0 / 1001), args.steps)
        launches += 4 * args.steps
        rnleg["strong_scaling"] = {"samples_total_16384": {"ms_per_evaluation": ms_s, "evals_per_sec": S / (ms_s * 1e-3)},
                                   "sweep_1001": {"ms_per_evaluation": ms_w, "evals_per_sec": 1001 / (ms_w * 1e-3)},
                                   "note": "total work fixed, samples split in contiguous shards over the ranks; one all-reduce per evaluation"}
        # parity self-check of the exchange step: sharded + all-reduced vs every sample on this rank alone (no communicator)
        if world > 1:
            Sp = 64 * world
            nodes_p, weights_p = midpoint(Sp)
            weights_p = weights_p * (1.0 + 0.25 * np.cos(np.arange(Sp)))          # non-uniform weights
            _, o_sh = sharded_leg(nodes_p, weights_p, 1)
            w1 = jq.Working_Arrays(rn.params, rn.nCoeff, device=local_rank)
            o_all = w1.evaluate_device(pcr, torch.from_numpy(configs.noise_shift(rn.params.Ntot, nodes_p)).to(dev),
                                       torch.from_numpy(weights_p).to(dev), True, stream=stream)
            torch.cuda.synchronize()
            g_sh, g_all = o_sh["grad"][0].cpu().numpy(), o_all["grad"][0].cpu().numpy()
            f_sh = float(o_sh["infid"][0].item() + o_sh["leak"][0].item())
            f_all = float(o_all["infid"][0].item() + o_all["leak"][0].item())
            err = max(abs(f_sh - f_all) / abs(f_all), float(np.linalg.norm(g_sh - g_all) / np.linalg.norm(g_all)))
            err = max_over_ranks(err)
            rnleg["nccl_parity"] = {"ok": bool(err <= 1e-12), "max_rel_err_over_ranks": err, "samples": Sp, "tolerance": 1e-12,
                                    "what": "objective and gradient: sample shards + ncclAllReduce vs one rank evaluating all samples"}
            w1.close()
        extra["risk_neutral_sample_sharded"] = rnleg
        wr.close()

    # ---- extra (N > 1): ONE cnot3 evaluation shared out over the GPUs (jq_comm_set_cooperative): the time segments of the time-parallel
    # path are split over the ranks, the propagators all-gathered, every rank returns the single-GPU bits
    if not args.no_extra and world > 1:
        c3 = configs.example("cnot3")
        w3 = jq.Working_Arrays(c3.params, c3.nCoeff, device=local_rank)
        w3.comm_init(rank, world)
        p3 = configs.synthetic_pcof(c3, 1)
        coop = {}
        res3 = {}
        for mode in ("replicated", "cooperative"):
            w3.comm_set_cooperative(mode == "cooperative")
            res3[mode] = w3.evaluate(p3)
            ts, ks = [], []
            for _ in range(3):
                dist.barrier()
                t0 = time.perf_counter()
                w3.evaluate(p3)
                ts.append((time.perf_counter() - t0) * 1e3)
                ks.append(w3.last_kernel_ms)
            launches += 4 * int(w3.query(2))
            coop[mode] = {"kernel": KERNEL_NAMES[w3.last_kernel], "time_segments": int(w3.query(7)), "kernels_ms": max_over_ranks(min(ks)),
                          "host_call_ms": max_over_ranks(min(ts))}
        g0, g1 = res3["replicated"]["grad"].ravel(), res3["cooperative"]["grad"].ravel()
        coop["rel_grad_diff"] = max_over_ranks(float(np.linalg.norm(g0 - g1) / np.linalg.norm(g0)))
        coop["note"] = "one pcof, every rank the same arguments; cooperative: segments of the propagator launch sharded, one in-place ncclAllGather per propagator array"
        extra["cooperative_single_eval_cnot3"] = coop
        w3.comm_destroy()
        w3.close()

    if rank == 0:
        line = {"metric": "objective+gradient evals/sec (traceobjgrad)", "value": value, "unit": "evals/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload,
                "state_steps_per_sec": value * 3 * cfg.params.nsteps,
                "e2e": {"value": e2e_val, "unit": "evals/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
                "gpu_launches": int(launches), "gpu_launches_note": "trajectory kernel + finalize/weighted-sum kernel per evaluation, all legs of this run",
                "roofline": roofline, "clocks": clocks, "extra": extra}
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if dumped is not None:
            line["dump_outputs"] = dumped
        print(json.dumps(line))
    wa.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
