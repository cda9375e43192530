"""Cost of the count observation families on the C2 shape: SIR [100,1,0], theta = (0.003, 0.1), the 100 observations of
tests/golden/sir_c2.csv, 2^20 particles, systematic resampling, f32 event loop.  The same data are observed through the
Gaussian model of bench.py (sigma 2; the predefined SIR kernels) and through a Poisson (rho = 1), a binomial (p = 0.9) and a
negative binomial (rho = 1, k = 10) law of I, which run on the generic rate-table kernels.  The four models are timed in one
process, alternating call by call after a warm-up; each call is one full log-likelihood (100 observations), timed with the
CUDA events of the filter handle.  Prints the card name and power limit, then one line per model (median / min over calls).

    python scripts/count_obs_probe.py [--calls 20] [--warmup 3] [--particles 1048576] [--json OUT]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, check=True).stdout.strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError):
        return "unknown"


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--particles", type=int, default=1 << 20)
    ap.add_argument("--json", help="also write the results to this file")
    args = ap.parse_args()

    import dpomp_b200 as dp

    y = dp.get_observations(os.path.join(ROOT, "tests", "golden", "sir_c2.csv"))
    theta = np.array([0.003, 0.1])
    models = {
        "gaussian": dp.partial_gaussian_obs_model(2.0),
        "poisson": dp.partial_poisson_obs_model(1.0),
        "binomial": dp.partial_binomial_obs_model(0.9),
        "negbin": dp.partial_negbin_obs_model(1.0, 10.0),
    }
    filters = {}
    for name, om in models.items():
        model = dp.generate_custom_model("SIR", dp.generate_model("SIR", [100, 1, 0]).rate_function, [100, 1, 0],
                                         [[-1, 1, 0], [0, -1, 1]], obs_model=om)
        filters[name] = dp.ParticleFilter(dp.device_model(dp.get_private_model(model, y)), args.particles, 1, 1, seed=7)
    for _ in range(args.warmup):
        for pf in filters.values():
            pf.loglik(theta)
    ms = {name: [] for name in filters}
    ll = {name: [] for name in filters}
    for _ in range(args.calls):
        for name, pf in filters.items():
            ll[name].append(pf.loglik(theta)[0])
            ms[name].append(pf.last_timing()[0])
    gpu = card()
    print(f"card: {gpu}; C2 shape, {args.particles} particles x {len(y)} observations, f32 loop, {args.calls} alternating calls")
    base = float(np.median(ms["gaussian"]))
    out = dict(card=gpu, particles=args.particles, observations=len(y), calls=args.calls, models={})
    for name in filters:
        med, lo = float(np.median(ms[name])), float(np.min(ms[name]))
        out["models"][name] = dict(median_ms=med, min_ms=lo, ratio_to_gaussian=med / base, mean_loglik=float(np.mean(ll[name])))
        print(f"  {name:9s} median {med:8.3f} ms  min {lo:8.3f} ms  x{med / base:5.2f} of the Gaussian  mean log-lik {np.mean(ll[name]):.2f}")
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
