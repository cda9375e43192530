"""Data-augmented MCMC (run_std_mcmc) on SIS / pooley.csv: device time per dpomp_da_step launch and chain-steps/s at 16, 1024
and 16384 lock-step chains with traj_props 1 and 16, and the single-core rate of the oracle's proposals for comparison.
Writes nothing to the tree; prints one line per configuration (and the GPU's name and power limit)."""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

import dpomp_b200 as dp
from oracle import da_oracle as dao

try:
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip())
except OSError:
    pass
model = dp.generate_model("SIS", [100, 1])
model.prior = dp.UniformProduct([0, 0], [0.01, 0.5])
y = dp.get_observations(os.path.join(ROOT, "tests", "golden", "pooley.csv"))
hmm = dp.get_private_model(model, y)
theta = np.array([0.003, 0.1])
for n in (16, 1024, 16384):
    th = theta[:, None] * np.random.default_rng(1).uniform(0.9, 1.1, size=(2, n))
    r = dp.run_std_mcmc(hmm, th, 3, 2, seed=2, verbose=False)  # generate_x0 + a warm-up step
    pt = r.particles
    lens = pt.lengths(np.arange(1, n + 1))
    for tp in (1, 16):
        kind = np.ones(n, dtype=np.uint8)
        pt.da_step(th, th, kind, tp, 3)
        reps = 20 if n < 16384 else 8
        t = time.perf_counter()
        for _ in range(reps):
            pt.da_step(th, th, kind, tp, 3)  # synchronous: the call ends with a stream synchronise
        dt = (time.perf_counter() - t) / reps
        print(f"chains {n:6d} traj_props {tp:2d}: {1e3 * dt:8.2f} ms per step, {n / dt:.3e} chain-steps/s, "
              f"{n * (tp + 1) / dt:.3e} walks/s (mean {lens.mean():.0f} events per trajectory)")
    th2 = np.ascontiguousarray(th[:, 0])
cm = dp.compile_model(model, y)
fc, times, types, ll = pt.get_particle(1)
t = np.zeros(len(times) + 4096); ty = np.zeros(len(times) + 4096, dtype=np.int32)
t[: len(times)] = times; ty[: len(times)] = types
ln, reps = len(times), 200
start = time.perf_counter()
for k in range(reps):
    ln = dao.da_props(cm.desc, th2, t, ty, ln, 196000, 16, 3, 1000 + k, 0)[0]
dt = (time.perf_counter() - start) / reps
print(f"oracle, one core, traj_props 16: {1e3 * dt:.2f} ms per chain-step ({1 / dt:.3e} chain-steps/s, {len(times)} events)")
