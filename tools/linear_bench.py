"""Cost of the linear terms (xfb_set_linear_terms): ms per RK4 step with the terms off and on, alternated on one handle
per grid, with the card's name and power limit.

    python tools/linear_bench.py [1024 4096 8192 16384] [--steps 20] [--rounds 3]

Prints one JSON line per grid.  The "on" runs set beta, drag and order-4 hyperviscosity together (the LIN instances of
K-COL); "off" switches them back to zero (the default instances)."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import fields  # noqa: E402
import xlab_fftbarotropic_b200 as xfb  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception:
        return "unknown"


def dt_for(n):
    return {1024: 4.0, 2048: 2.0, 4096: 1.0, 8192: 0.5, 16384: 0.25}.get(n, 1.0)


def timed(b, steps, dt):
    b.step(2, dt)                 # (re)captures the step graph outside the window
    b.sync()
    t0 = time.perf_counter()
    b.step(steps, dt)
    b.sync()
    return (time.perf_counter() - t0) * 1e3 / steps


def main():
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("grids", type=int, nargs="*", default=[1024, 4096, 8192, 16384])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    gpu = card()
    for n in a.grids:
        dt = dt_for(n)
        k0 = 2 * np.pi / 600000.0
        kd = 2 * np.ceil(n / 3.0) ** 2
        beta, mu, nu_h = 2.3e-11, 1e-6, 0.5 / (dt * (kd * k0 * k0) ** 4)
        b = xfb.Backend(n)
        b.set_vorticity(fields.elliptic(n))
        off, on = [], []
        for _ in range(a.rounds):
            b.set_linear_terms(0.0, 0.0, 0.0)
            off.append(timed(b, a.steps, dt))
            b.set_linear_terms(beta, mu, nu_h, 4)
            on.append(timed(b, a.steps, dt))
        b.close()
        print(json.dumps({"grid": n, "gpu": gpu, "steps": a.steps, "ms_per_step_off": [round(x, 4) for x in off],
                          "ms_per_step_on": [round(x, 4) for x in on],
                          "overhead_pct": round(100.0 * (min(on) / min(off) - 1.0), 2)}), flush=True)


if __name__ == "__main__":
    main()
