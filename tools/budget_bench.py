"""Time xfb_get_spectral_budget on the elliptic vortex after warm-up steps: per grid, milliseconds per call without and
with a source, each for totals only (nshells = 0) and for every shell, next to the milliseconds of one step of the
same handle (host clock around K calls, each of which ends in a stream synchronise), and the GPU name and power limit
read in the same run.

    python tools/budget_bench.py 1024 4096 8192 16384 [--calls 20]

Prints one JSON line per grid.  No torch import (a fresh box pays a minute for it)."""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import fields  # noqa: E402
import xlab_fftbarotropic_b200 as xfb  # noqa: E402
from spectrum_bench import gpu_info  # noqa: E402


def per_call_ms(fn, calls):
    for _ in range(3):
        fn()
    t0 = time.perf_counter()
    for _ in range(calls):
        fn()
    return round((time.perf_counter() - t0) * 1e3 / calls, 4)


def main():
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("grids", type=int, nargs="*", default=[1024, 4096, 8192, 16384])
    ap.add_argument("--calls", type=int, default=20)
    a = ap.parse_args()
    name, power = gpu_info()
    for n in a.grids:
        dt = {1024: 4.0, 4096: 1.0, 8192: 0.5, 16384: 0.25}.get(n, 1.0)
        b = xfb.Backend(n)
        b.set_vorticity(fields.elliptic(n))
        b.step(3, dt)
        b.sync()
        out = {"grid": n, "gpu": name, "power_limit": power, "shells": xfb.capi.shells_all(n, n, 600000.0)}

        def step():
            b.step(1, dt)
            b.sync()

        out["ms_step"] = per_call_ms(step, a.calls)
        for src_tag in ("no_source", "source"):
            if src_tag == "source":
                x = np.arange(n, dtype=np.float32) / n
                b.set_source((2e-9 * np.sin(2 * np.pi * (3 * x[:, None] + 2 * x[None, :]))).astype(np.float32))
                out["ms_step_source"] = per_call_ms(step, a.calls)
            for tag, nsh in (("totals", 0), ("all_shells", None)):
                out[f"ms_budget_{src_tag}_{tag}"] = per_call_ms(lambda: b.spectral_budget(nsh), a.calls)
        print(json.dumps(out), flush=True)
        b.close()


if __name__ == "__main__":
    main()
