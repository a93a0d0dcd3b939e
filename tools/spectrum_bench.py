"""Time xfb_get_energy_spectrum on the elliptic vortex after warm-up steps: per grid, milliseconds per call with
nshells = 0 (totals only) and with every shell (host clock around K calls, each of which ends in a stream synchronise),
the state bytes read (nx * pitch * 8) and the rate they imply, and the GPU name and power limit read in the same run.

    python tools/spectrum_bench.py 1024 4096 8192 16384 [--calls 50]

Prints one JSON line per grid.  No torch import (a fresh box pays a minute for it)."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import fields  # noqa: E402
import xlab_fftbarotropic_b200 as xfb  # noqa: E402


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        name, power = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return name, power
    except Exception as e:          # the numbers still stand; say that the device could not be named
        return f"unknown ({e})", "unknown"


def main():
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("grids", type=int, nargs="*", default=[1024, 4096, 8192, 16384])
    ap.add_argument("--calls", type=int, default=50)
    a = ap.parse_args()
    name, power = gpu_info()
    for n in a.grids:
        b = xfb.Backend(n)
        b.set_vorticity(fields.elliptic(n))
        b.step(3, {1024: 4.0, 4096: 1.0, 8192: 0.5, 16384: 0.25}.get(n, 1.0))
        b.sync()
        pitch = xfb.slab_partition(n, n, 1, 1, 0)["chunk_cols"] if xfb.capi.load().xfb_size_supported(n, n) == 1 else n // 2 + 1
        nbytes = n * pitch * 8
        out = {"grid": n, "gpu": name, "power_limit": power, "state_bytes": nbytes, "shells": xfb.capi.shells_all(n, n, 600000.0)}
        for tag, nsh in (("totals", 0), ("all_shells", None)):
            for _ in range(5):
                b.energy_spectrum(nsh)
            t0 = time.perf_counter()
            for _ in range(a.calls):
                b.energy_spectrum(nsh)
            ms = (time.perf_counter() - t0) * 1e3 / a.calls
            out[f"ms_{tag}"] = round(ms, 4)
            out[f"GBps_{tag}"] = round(nbytes / (ms * 1e-3) / 1e9, 1)
        print(json.dumps(out), flush=True)
        b.close()


if __name__ == "__main__":
    main()
