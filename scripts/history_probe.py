"""Cost of the hidden-state history (dpomp_pf_set_history) on config C2 (SIR, 1 x 2^20 particles, T = 100) and on the C3
per-chain shape (SEIR, 64 x 65536 particles, T = 100), f32 event loop, systematic resampling:
  * device time per filter call with the history off, MOMENTS, and MOMENTS | PATHS, alternated in one process;
  * per-launch time of pf_history_kernel (torch.profiler, CUDA activity) against the bytes it moves;
  * time of get_filtered_moments and of sample_paths.
Prints the GPU's name and power limit, then one line per number.  Writes nothing to the tree."""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

import dpomp_b200 as dp

print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip())
REPS = int(os.environ.get("HISTORY_PROBE_REPS", "6"))
CASES = [("C2", "SIR", [100, 1, 0], "sir_c2.csv", [0.003, 0.1], 1 << 20, 1),
         ("C3 shape", "SEIR", [100, 0, 1, 0], "seir_c3.csv", [0.005, 0.2, 0.1], 65536, 64)]
for name, mname, ic, csv, theta, n, nb in CASES:
    model = dp.generate_model(mname, ic)
    y = dp.get_observations(os.path.join(ROOT, "tests", "golden", csv))
    dm = dp.device_model(dp.get_private_model(model, y))
    th = np.tile(np.asarray(theta)[:, None], (1, nb))
    pfs = {}
    for label, flags in (("off", None), ("MOMENTS", (True, False)), ("MOMENTS|PATHS", (True, True))):
        pf = dp.ParticleFilter(dm, n, nb, 1, seed=7)
        if flags:
            pf.set_history(*flags)
        pf.loglik(th)  # warm-up (module load, two-per-lane choice from the previous call)
        pf.loglik(th)
        pfs[label] = pf
    times = {k: [] for k in pfs}
    for _ in range(REPS):  # alternate the three handles
        for k, pf in pfs.items():
            pf.loglik(th)
            times[k].append(pf.last_timing()[0])
    tile, _ = pfs["off"].geometry()
    n_pad = -(-n // tile) * tile
    C, T = len(ic), len(y)
    base = np.median(times["off"])
    for k, v in times.items():
        print(f"{name}: history {k:14s} {np.median(v):8.3f} ms per call (min {np.min(v):.3f}, max {np.max(v):.3f}; "
              f"{100 * (np.median(v) / base - 1):+.1f} % vs off)")
    pf = pfs["MOMENTS|PATHS"]
    print(f"{name}: PATHS history memory {T * nb * n_pad * (4 * C + 4) / 1e9:.2f} GB")
    # per-launch time of the record kernel
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        pf.loglik(th)
    durs = [e.device_time for e in prof.events() if "pf_history_kernel" in e.name]
    rd, wr = nb * n_pad * (4 * C + 8), nb * n_pad * 4 * C
    if durs:
        us = float(np.median(durs))
        print(f"{name}: pf_history_kernel (MOMENTS|PATHS) {len(durs)} launches, median {us:.1f} us, reads {rd / 1e6:.1f} MB, "
              f"writes {wr / 1e6:.1f} MB -> {(rd + wr) / (us * 1e-6) / 1e12:.2f} TB/s")
    t0 = time.perf_counter()
    pf.filtered_moments()
    print(f"{name}: get_filtered_moments {1e3 * (time.perf_counter() - t0):.2f} ms (host wall, includes the copy)")
    for n_paths in (1, 1000):
        key = pf.next_stream_key()
        pf.loglik(th)
        t0 = time.perf_counter()
        pf.sample_paths(n_paths, key)
        print(f"{name}: sample_paths({n_paths}) {1e3 * (time.perf_counter() - t0):.2f} ms (host wall, includes the copy)")
    del pfs, pf
    torch.cuda.empty_cache()
