#!/usr/bin/env python
"""bench.py -- particle-observation steps/s of the bootstrap particle filter (BASELINE.json metric), config C2:
SIR [100,1,0], theta=(0.003,0.1), 100 observations (tests/golden/sir_c2.csv), 2^20 particles, systematic resampling
after every observation, on N B200s of one node (N > 1: independent replicas, one per GPU -- a single filter does not
shard, SURVEY.md 8e; `scaling` = weak).

A "step" is one full particle-filter log-likelihood evaluation (estimate_likelihood) = 2^20 x 100 particle-observation
steps.  `value` is measured with theta and the result resident in HBM (dpomp_pf_loglik_device); `e2e` is the same metric
through the public API closure get_particle_filter_lpdf(model, y)(theta) with HOST buffers.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step of each C2 loop returned, as DIR/<name>.npy: `loglik` (device-resident
path) with `population` (the filter's particles after that call, n x C, exact in float32), `loglik_e2e` (public API
closure) and `loglik_f64_loop`.  Seeds, theta and data are fixed, so the same arguments give the same inputs on every run
and two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

N_PARTICLES = 1 << 20
WORKLOAD = "C2: SIR [100,1,0] theta=(0.003,0.1), T=100 obs (tests/golden/sir_c2.csv), 2^20 particles, systematic resampling every obs"
METRIC = "particle-obs steps/sec (bootstrap PF)"
UNIT = "particle-observation steps/s"


def load_c2():
    import dpomp_b200 as dp

    model = dp.generate_model("SIR", [100, 1, 0])
    y = dp.get_observations(os.path.join(ROOT, "tests", "golden", "sir_c2.csv"))
    return dp, model, y, np.array([0.003, 0.1])


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU with NVML while the timed region runs."""

    def __init__(self, index: int, period_s: float = 0.01):
        super().__init__(daemon=True)
        self.index, self.period, self.samples, self.reasons, self.max_mhz = index, period_s, [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as exc:  # pragma: no cover
            self.err = repr(exc)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def ncu_traffic():
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the two PF kernels from the committed
    `ncu --set full` capture of this command (profiles/r1_ncu_full_metrics.csv); None when the file is missing."""
    import csv

    import glob

    cands = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_full_metrics.csv")))
    path = cands[-1] if cands else os.path.join(ROOT, "profiles", "r1_ncu_full_metrics.csv")
    ncu_traffic.source = os.path.relpath(path, ROOT)
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    try:
        rows = {r[0]: r for r in csv.reader(open(path)) if r}
        names = rows["Kernel Name"][2:]
        out = {}
        for key in ("pf_sim_weight_kernel", "pf_resample_kernel"):
            cols = [i for i, n in enumerate(names) if key in n]
            tot = 0.0
            for metric in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                r = rows[metric]
                tot += sum(float(r[2 + i].replace(",", "")) for i in cols) / max(len(cols), 1) * scale.get(r[1], 1.0)
            out[key] = tot if cols else None
            r = rows.get("smsp__inst_executed.sum")
            if r and cols:  # executed warp instructions per launch, for the issue-rate view of the same kernels
                out[key + ":warp_inst"] = sum(float(r[2 + i].replace(",", "")) for i in cols) / len(cols)
        return out
    except Exception:
        return {}


def cpu_baseline(dp, model, y, theta, n_particles: int, threads: int):
    """The oracle port (kind 'port': Julia is not installed, the reference itself cannot run) on the host cores."""
    from oracle import oracle as orc

    cm = dp.compile_model(model, y)
    t0 = time.perf_counter()
    ll, ev = orc.pf_loglik(cm.desc, theta, n_particles, 1, key=12345, threads=threads)
    dt = time.perf_counter() - t0
    return n_particles * len(y) / dt, dt, ll, ev


SMC2_OUTER, SMC2_NPF = 8192, 4096


def run_smc2(dp, world, rank, barrier):
    """BASELINE config C4: LOTKA [70,70], SMC^2 with 8192 theta-particles x 4096 state particles, T = 30 observations
    (tests/golden/lotka_c4.csv), prior U(0,(1,0.01,1)), ess_rs_crit 0.3, independent proposals.  theta-particles are
    sharded over the ranks (NCCL all-gather of weights, all-to-all of migrating filters).  One full run_ibis_analysis."""
    import torch

    model = dp.generate_model("LOTKA", [70, 70])
    model.prior = dp.UniformProduct([0, 0, 0], [1.0, 0.01, 1.0])
    y = dp.get_observations(os.path.join(ROOT, "tests", "golden", "lotka_c4.csv"))
    comm = dp.Comm() if world > 1 else None
    # warm-up with the SAME collective shapes as the timed run (all 8192 theta-particles, fewer state particles, enough
    # observations to reach a resample-move step): NCCL connects lazily per algorithm / protocol / message size class, and a
    # smaller warm-up left 0.15 s of connection set-up inside the timed region at 8 ranks
    dp.run_ibis_analysis(model, y[:12], np=SMC2_OUTER, npf=256, seed=3, comm=comm, verbose=False)
    import gc

    gc.collect()  # release the warm-up handles now: cudaFree synchronises and must not land in the timed region
    # the two filter banks (resident + proposal) of this rank are allocated before the timed region and outlive it, like
    # the workspace of the PF metric: the timed region is the analysis on resident workspaces
    lo, hi = (comm.bounds(SMC2_OUTER) if comm is not None else (0, SMC2_OUTER))
    dm = dp.device_model(dp.get_private_model(model, y))
    banks = [dp.ParticleFilter(dm, SMC2_NPF, max(hi - lo, 1), 1, seed=1 + k) for k in range(2)]
    it = iter(banks)
    barrier()
    t0 = time.perf_counter()
    res = dp.run_ibis_analysis(model, y, np=SMC2_OUTER, npf=SMC2_NPF, seed=1, comm=comm, verbose=False,
                               pf_factory=lambda nb, sd: next(it))
    barrier()
    dt = time.perf_counter() - t0
    tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        import torch.distributed as dist

        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dt = float(tt.item())
    n_rs = int(res.k_log[0] // SMC2_OUTER)
    out = {"metric": "SMC^2 theta-particle-observation updates/s", "value": SMC2_OUTER * len(y) / dt, "unit": "theta-particle-obs/s",
           "wall_s": dt, "n_gpus": world, "scaling": "strong",
           "config": {"workload": f"C4: LOTKA [70,70], {SMC2_OUTER} theta x {SMC2_NPF} state particles, T={len(y)}, prior U(0,(1,0.01,1)), "
                                  "ess_rs_crit 0.3, ind_prop, n_props 1; filter banks allocated before the timed region", "resample_mutate_steps": n_rs},
           "minus_log_evidence": [float(v) for v in res.bme], "posterior_mean": [float(v) for v in res.mu],
           "acceptance_rate": float(res.k_log[1] / max(res.k_log[0], 1)),
           "rank0_phase_seconds": {k: round(float(v), 4) for k, v in sorted(getattr(res, "timers", {}).items())}}
    if world == 1 and rank == 0:
        from oracle import oracle as orc

        cm = dp.compile_model(model, y)
        n_o, n_p = 128, 512
        th0 = model.prior.rand(n_o, np.random.default_rng(5))
        t0 = time.perf_counter()
        o = orc.run_pibis(cm.desc, th0, model.prior.lower, model.prior.upper, npf=n_p, seed=7, threads=orc.max_threads())
        dtc = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": n_o * len(y) / dtc, "unit": "theta-particle-obs/s", "cores": orc.max_threads(), "kind": "port",
                               "sample": f"{n_o} theta x {n_p} state particles (1/64 of the theta-particles, 1/8 of the state particles), {dtc:.1f} s",
                               "inner_pf_steps_per_s": o["pf_steps"] / dtc}
    return out


def _max_over_ranks(dt, world):
    import torch

    tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        import torch.distributed as dist

        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    return float(tt.item())


def _sha16(*arrays):
    import hashlib

    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:16]


def _seir_c3(dp):
    model = dp.generate_model("SEIR", [100, 0, 1, 0])
    model.prior = dp.UniformProduct([0, 0, 0], [0.02, 1.0, 0.5])
    y = dp.get_observations(os.path.join(ROOT, "tests", "golden", "seir_c3.csv"))
    return model, y


PMCMC_CHAINS, PMCMC_NPF, PMCMC_STEPS = 64, 65536, 41


def run_pmcmc_c3(dp, world, rank, barrier):
    """BASELINE config C3: SEIR [100,0,1,0], pMCMC (src/hmm_mcmc.jl:349-365, 166-211) with 64 independent chains x 65536
    particles, T = 100 observations (tests/golden/seir_c3.csv), prior U(0,(0.02,1,0.5)).  Chains are sharded over the
    ranks (strong scaling: the total work is fixed); no communication until the final gather of the samples.  The timed
    region is PMCMC_STEPS - 1 Metropolis-Hastings steps of every chain (plus the initial evaluation) on a pre-allocated
    filter bank."""
    import gc

    model, y = _seir_c3(dp)
    hmm = dp.get_private_model(model, y)
    comm = dp.Comm() if world > 1 else None
    lo, hi = (comm.bounds(PMCMC_CHAINS) if comm is not None else (0, PMCMC_CHAINS))
    th0 = np.tile(np.array([[0.005], [0.2], [0.1]]), (1, PMCMC_CHAINS)) * np.random.default_rng(1).uniform(0.8, 1.25, (3, PMCMC_CHAINS))
    pf = dp.ParticleFilter(dp.device_model(hmm), PMCMC_NPF, max(hi - lo, 1), 1, seed=2)
    factory = lambda nb, sd: pf
    dp.run_pmcmc(hmm, th0, steps=4, adapt_period=2, p=PMCMC_NPF, seed=1, comm=comm, pf_factory=factory, verbose=False)
    gc.collect()
    barrier()
    t0 = time.perf_counter()
    res = dp.run_pmcmc(hmm, th0, steps=PMCMC_STEPS, adapt_period=PMCMC_STEPS // 2, p=PMCMC_NPF, seed=2, comm=comm,
                       pf_factory=factory, verbose=False)
    barrier()
    dt = _max_over_ranks(time.perf_counter() - t0, world)
    evals = PMCMC_CHAINS * PMCMC_STEPS  # one PF evaluation per chain and step (the first one is the initial point)
    return {"metric": "pMCMC chain-steps/s", "value": evals / dt, "unit": "PF evaluations (chain x MH step)/s", "wall_s": dt,
            "n_gpus": world, "scaling": "strong", "particle_obs_steps_per_s": evals * PMCMC_NPF * len(y) / dt,
            "config": {"workload": f"C3: SEIR [100,0,1,0], {PMCMC_CHAINS} chains x {PMCMC_NPF} particles, T={len(y)}, {PMCMC_STEPS} "
                                   "MH steps per chain, prior U(0,(0.02,1,0.5)); filter bank allocated before the timed region"},
            "ms_per_mh_step": 1e3 * dt / PMCMC_STEPS,
            "mean_acceptance": float(res.accepted.mean() / (PMCMC_STEPS - 1)),
            "samples_sha16": _sha16(res.samples.theta), "posterior_mean": [float(v) for v in res.samples.mu],
            "rank0_phase_seconds": {k: round(float(v) * (1e-3 if k.endswith("_ms") else 1.0), 4) for k, v in sorted(res.timers.items())}}


MBPI_OUTER = 16384


def run_mbp_ibis_c5(dp, world, rank, barrier):
    """BASELINE config C5: SEIR data of C3, MBP-IBIS (src/hmm_ibis.jl:140-244) with 16384 theta-particles, n_props 3,
    ess_rs_crit 0.5, ind_prop false, STRATIFIED outer resampling; theta-particles and their trajectories are sharded over
    the ranks, trajectories migrate after every outer resample (two-phase all-to-all-v over NCCL)."""
    import gc

    model, y = _seir_c3(dp)
    hmm = dp.get_private_model(model, y)
    comm = dp.Comm() if world > 1 else None
    lo, hi = (comm.bounds(MBPI_OUTER) if comm is not None else (0, MBPI_OUTER))
    th0 = model.prior.rand(MBPI_OUTER, np.random.default_rng(3))
    ptcls = dp.MbpParticles(dp.device_model(hmm), max(hi - lo, 1), seed=4)
    # warm-up = one full analysis on the same store (0.2 s): NCCL sets up its send / receive connections lazily at the first
    # migration (0.3 s at two ranks), and a shortened data set does not reach a resample-move step.  Same seed as the timed
    # run, so the growable trajectory store has reached the capacity this analysis needs (the store is reset, nothing else
    # is kept: the timed run simulates, proposes and migrates everything again)
    dp.run_mbp_ibis(hmm, th0, 0.5, 3, False, 1.002, seed=4, comm=comm, outer_rs=dp.rs_stratified, verbose=False,
                    particles_factory=lambda n, sd: ptcls)
    gc.collect()
    barrier()
    t0 = time.perf_counter()
    r = dp.run_mbp_ibis(hmm, th0, 0.5, 3, False, 1.002, seed=4, comm=comm, outer_rs=dp.rs_stratified, verbose=False,
                        particles_factory=lambda n, sd: ptcls)
    barrier()
    dt = _max_over_ranks(time.perf_counter() - t0, world)
    return {"metric": "MBP-IBIS theta-particle-observation updates/s", "value": MBPI_OUTER * len(y) / dt, "unit": "theta-particle-obs/s",
            "wall_s": dt, "n_gpus": world, "scaling": "strong",
            "config": {"workload": f"C5: SEIR [100,0,1,0], {MBPI_OUTER} theta-particles (one trajectory each), T={len(y)}, n_props 3, "
                                   "ess_rs_crit 0.5, ind_prop false, stratified outer resampling; trajectory store allocated before the timed region",
                       "resample_mutate_steps": int(r.k_log[0] // (3 * MBPI_OUTER))},
            "minus_log_evidence": [float(v) for v in r.bme], "posterior_mean": [float(v) for v in r.mu],
            "acceptance_rate": float(r.k_log[1] / max(r.k_log[0], 1)),
            "result_sha16": _sha16(r.theta, r.weight, r.bme),
            "rank0_phase_seconds": {k: round(float(v), 4) for k, v in sorted(getattr(r, "timers", {}).items())}}


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port, all host threads) on the same config and metric."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dp, model, y, theta = load_c2()
    from oracle import oracle as orc

    # torchrun exports OMP_NUM_THREADS=1: take the cores this process may run on and pass the count explicitly (the oracle's
    # num_threads clause overrides the environment), so the arm uses the same threads at every --gpus N
    threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    rate = 0.0
    for _ in range(max(1, min(args.warmup, 2))):
        rate = max(rate, cpu_baseline(dp, model, y, theta, 1 << 15, threads)[0])
    # one step = the full 2^20-particle workload when it fits the per-step budget, else a power-of-two sample of it
    budget_s = min(4.0, 150.0 / max(args.steps, 1))
    n_sample = N_PARTICLES
    while n_sample > (1 << 14) and n_sample * len(y) / rate > budget_s:
        n_sample >>= 1
    t_total, units = 0.0, 0
    for _ in range(args.steps):
        v, dt, _, _ = cpu_baseline(dp, model, y, theta, n_sample, threads)
        t_total += dt
        units += n_sample * len(y)
    value = units / t_total
    sample = (f"{n_sample} of {N_PARTICLES} particles x {len(y)} observations per step, OpenMP over particles on {threads} threads "
              f"(thread count passed explicitly: independent of OMP_NUM_THREADS / torchrun)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "note": "CPU restatement of the reference algorithm (oracle/dpomp_oracle.c); "
                   "the Julia reference cannot run here (no julia in the image)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print_json(line)


def _json_only_stdout():
    """Everything except the final JSON line goes to stderr (NCCL and the analysis drivers print to fd 1)."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, "w")


def main():
    global print_json
    out = _json_only_stdout()
    print_json = lambda obj: (out.write(json.dumps(obj) + "\n"), out.flush())
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-smc2", action="store_true", help="skip the SMC^2 (config C4) secondary measurement")
    ap.add_argument("--no-outer", action="store_true", help="skip the pMCMC (C3) and MBP-IBIS (C5) secondary measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step of each C2 loop to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the particle-filter path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    dp, model, y, theta = load_c2()
    hmm = dp.get_private_model(model, y)
    dm = dp.device_model(hmm)
    T = len(y)
    units_per_step = N_PARTICLES * T

    pf = dp.ParticleFilter(dm, N_PARTICLES, 1, 1, seed=1000 + rank, device=local_rank)
    theta_dev = torch.tensor(theta, dtype=torch.float64, device="cuda")
    out_dev = torch.zeros(1, dtype=torch.float64, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def device_step():
        pf.loglik_device(theta_dev.data_ptr(), 1, out_dev.data_ptr())

    for _ in range(args.warmup):
        device_step()
    sampler = ClockSampler(local_rank)
    sampler.start()

    # ---- timed region 1: device-resident (value) -------------------------------------------------------------
    barrier()
    wall = dev_ms = 0.0
    launches = events = 0
    for _ in range(args.steps):
        flush.zero_()  # L2 flush between timed iterations (excluded from the step time)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        device_step()  # synchronous on return
        wall += time.perf_counter() - t0
        ms, nl = pf.last_timing()
        dev_ms += ms
        launches += nl
        events += pf.last_event_count()
    barrier()
    ll_last = float(out_dev.item())
    dumps = {}
    if args.dump_outputs:
        dumps["loglik"] = np.array([ll_last])
        dumps["population"] = pf.get_pop(1).astype(np.float32)

    # ---- timed region 2: end to end through the public API closure, host theta -> host float -------------------
    f = dp.get_particle_filter_lpdf(model, y, np=N_PARTICLES, seed=2000 + rank, device=local_rank)
    theta_pinned = torch.tensor(theta, dtype=torch.float64).pin_memory().numpy()
    for _ in range(3):
        f(theta_pinned)
    barrier()
    wall_e2e = 0.0
    for _ in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ll_e2e = f(theta_pinned)
        wall_e2e += time.perf_counter() - t0
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs:
        dumps["loglik_e2e"] = np.array([ll_e2e])

    # ---- roofline pass: CUDA events around every kernel launch of the same step --------------------------------
    pf.set_kernel_timing(True)
    k_ms = np.zeros(2)
    k_n = np.zeros(2, dtype=np.int64)
    roof_steps = args.steps
    for _ in range(roof_steps):
        flush.zero_()
        torch.cuda.synchronize()
        device_step()
        (m0, m1), (n0, n1) = pf.last_kernel_timing()
        k_ms += (m0, m1)
        k_n += (n0, n1)
    pf.set_kernel_timing(False)

    # ---- secondary metric of BASELINE.json: SMC^2 theta-particles/s on config C4, sharded over the ranks ------------
    # ---- reference-precision throughput: the same C2 step with the f64 event loop (DPOMP_SIM_F64) ----------------------
    pf64 = dp.ParticleFilter(dm, N_PARTICLES, 1, 1, seed=3000 + rank, device=local_rank, sim_precision=dp._capi.SIM_F64)
    for _ in range(2):
        pf64.loglik_device(theta_dev.data_ptr(), 1, out_dev.data_ptr())
    f64_steps = args.steps
    barrier()
    wall_f64 = 0.0
    for _ in range(f64_steps):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pf64.loglik_device(theta_dev.data_ptr(), 1, out_dev.data_ptr())
        wall_f64 += time.perf_counter() - t0
    barrier()
    ll_f64 = float(out_dev.item())
    del pf64
    if args.dump_outputs:
        dumps["loglik_f64_loop"] = np.array([ll_f64])
        if rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in dumps.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)

    smc2 = pmcmc = mbpi = None
    if not args.no_smc2:
        smc2 = run_smc2(dp, world, rank, barrier)
    if not args.no_outer:
        pmcmc = run_pmcmc_c3(dp, world, rank, barrier)
        mbpi = run_mbp_ibis_c5(dp, world, rank, barrier)

    # max over ranks
    t = torch.tensor([wall, dev_ms, wall_e2e, wall_f64], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    wall, dev_ms, wall_e2e, wall_f64 = (float(v) for v in t.tolist())

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        C = 3
        # algorithmic bytes per particle per launch (SURVEY.md 8d): K1 sim+weight R 4C, W 4C+8; fused K2-K5 (scan R8 W8,
        # search R8 W4, gather R 4+4C W 4C)
        alg = {"pf_sim_weight_kernel": 8 * C + 8, "pf_resample_kernel": 8 * C + 40}
        names = ["pf_sim_weight_kernel", "pf_resample_kernel"]
        traffic = ncu_traffic()
        kernels = {}
        for i, nm in enumerate(names):
            if k_n[i]:
                avg_ms = k_ms[i] / k_n[i]
                ach = alg[nm] * N_PARTICLES / (avg_ms * 1e-3) / 1e9
                kernels[nm] = {"ncu_dram_bytes_per_launch": traffic.get(nm), "avg_launch_us": 1e3 * avg_ms, "launches_per_step": int(k_n[i] // roof_steps),
                               "share_of_kernel_time": float(k_ms[i] / k_ms.sum()), "alg_bytes_per_particle": alg[nm],
                               "achieved_gbs": ach, "frac_of_hbm_peak": ach / hbm_peak}
                wi = traffic.get(nm + ":warp_inst")
                if wi:  # issue-rate view: executed warp instructions (ncu) / measured launch time vs SMs x 4 schedulers x clock
                    sm_clock = float((clocks or {}).get("sm_max_mhz") or 1965.0) * 1e6
                    issue_peak = torch.cuda.get_device_properties(local_rank).multi_processor_count * 4 * sm_clock
                    kernels[nm].update({"ncu_warp_inst_per_launch": wi, "warp_inst_per_s": wi / (avg_ms * 1e-3),
                                        "frac_of_issue_peak": wi / (avg_ms * 1e-3) / issue_peak})
        dom = max(kernels, key=lambda k: kernels[k]["share_of_kernel_time"])
        value = world * units_per_step * args.steps / wall
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 event loop + f64 weights/scan (int32 state)", "data": "synthetic",
            "config": {"workload": WORKLOAD, "parallelism": f"replicas x{world} (one independent filter per GPU)",
                       "l2": "256 MiB flush buffer written between timed iterations; per-filter working set (33 MB) is L2 resident within a step by construction",
                       "timing": "per-step host bracket around the synchronous C-ABI call, max over ranks; device_ms_per_step = CUDA events on the handle's stream"},
            "device_ms_per_step": dev_ms / args.steps,
            "events_per_step": events / args.steps, "events_per_sec": world * events / wall,
            "loglik_last": ll_last,
            "e2e": {"value": world * units_per_step * args.steps / wall_e2e, "unit": UNIT, "h2d_bytes_per_step": int(theta.nbytes),
                    "d2h_bytes_per_step": 8, "ms_per_step": 1e3 * wall_e2e / args.steps, "loglik_last": ll_e2e,
                    "api": "get_particle_filter_lpdf(model, y; np=2^20)(theta)"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"kernel": dom, "bound": "hbm", "achieved": kernels[dom]["achieved_gbs"], "peak": hbm_peak, "unit": "GB/s",
                         "frac": kernels[dom]["frac_of_hbm_peak"], "traffic": traffic.get(dom), "peak_source": peak_src,
                         "traffic_source": f"{getattr(ncu_traffic, 'source', 'profiles/')} (ncu --set full of this command; bytes per launch; the 33 MB working set is L2 resident)",
                         "note": "the simulate kernel is instruction-issue / latency bound, not HBM bound (DESIGN.md 4.1); frac is its HBM-roofline fraction, roofline_kernels[*].frac_of_issue_peak the issue-rate view (ncu warp instructions / measured launch time)"},
            "roofline_kernels": kernels,
            "roofline_kernels_note": "avg_launch_us / share_of_kernel_time come from a separate pass with CUDA events around EVERY launch, "
                                     "which serialises the programmatic-dependent-launch chain: they are upper bounds (their sum exceeds ms_per_step); "
                                     "value / ms_per_step are measured without per-launch events",
            "value_f64_loop": {"value": world * units_per_step * f64_steps / wall_f64, "unit": UNIT, "ms_per_step": 1e3 * wall_f64 / f64_steps,
                               "steps": f64_steps, "loglik_last": ll_f64,
                               "note": "same C2 step with DPOMP_SIM_F64: rates, waiting times and event choice in f64 with the reference's "
                                       "expressions (the draw-for-draw parity loop)"},
            "roofline_pipeline": {"alg_bytes_per_step": 16 * C + 48, "achieved_gbs": (16 * C + 48) * value / world / 1e9,
                                  "frac_of_hbm_peak": (16 * C + 48) * value / world / 1e9 / hbm_peak},
        }
        if smc2 is not None:
            line["smc2"] = smc2
        if pmcmc is not None:
            line["pmcmc_c3"] = pmcmc
        if mbpi is not None:
            line["mbp_ibis_c5"] = mbpi
        if world == 1 and not args.no_cpu_baseline:
            from oracle import oracle as orc

            th = orc.max_threads()
            v_all, dt_all, ll_cpu, _ = cpu_baseline(dp, model, y, theta, N_PARTICLES, th)
            v_one, dt_one, _, _ = cpu_baseline(dp, model, y, theta, 1 << 16, 1)
            line["cpu_baseline"] = {"value": v_all, "unit": UNIT, "cores": th, "kind": "port",
                                    "sample": f"the full workload once (2^20 particles x {T} obs, {dt_all:.1f} s), OpenMP over particles",
                                    "single_thread_value": v_one, "single_thread_sample": f"2^16 particles x {T} obs ({dt_one:.1f} s)",
                                    "loglik": ll_cpu}
        print_json(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
