"""Golden record files for tests/test_host_programs.py: what the reference main.cpp writes for main.out's two
comparison runs, so that those tests need nothing outside the repository.

Run after `python __graft_entry__.py` (it needs oracle/_ref/liboracle.so and bin/makefield-elliptic-vortex.out):
    python tests/golden/make_golden_records.py

  ref_records.npz
    n256_*   elliptic vortex at 256^2 (ref_n256.npz `elliptic_init`), dt = 3 s, 5 steps recorded every 2: steps 0, 2, 4
    n768_*   the reference's default grid: makefield-elliptic-vortex.out's 768^2 field, dt = 3 s, 6 steps recorded every 3
    Each of vort / psi / u / v at each record step is stored like ref_kuo1024.npz (make_golden_headline.py):
      <kind>_<step>_sub  every 8th (256^2) or 24th (768^2) point in both directions, float32
      <kind>_<step>_blk  float64 sums and sums of squares over 16 x 16 blocks (the whole field enters through them)
    source   "reference" when the unmodified reference binary was run, "restatement" when oracle/barotropic_oracle.c was.
             The restatement writes the reference binary's record files bit for bit: tests/test_oracle.py checks that
             against ref_n64.npz and ref_n256.npz, which the reference binary wrote.
"""
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
from oracle import build_oracle, oracle as orc  # noqa: E402
from make_golden_headline import reduce_field  # noqa: E402

KINDS = (("vort", orc.VORT), ("psi", orc.PSI), ("u", orc.U), ("v", orc.V))


def records(v0, n, dt, steps, rec):
    """{(kind, step): field} of the reference main.cpp's record files for `steps` steps recorded every `rec`"""
    if build_oracle.build_reference(n, programs=("main",)):
        return orc.run_reference_main(v0, n, dt, steps, rec), "reference"
    o = orc.Oracle(n)
    o.set_vorticity(v0)
    out = {}
    for s in range(steps):
        if s % rec == 0:
            for kind, which in KINDS:
                out[(kind, s)] = o.get_field(which)
        o.step(1, dt)
    return out, "restatement"


def main():
    out = {}
    sources = set()
    v256 = np.load(os.path.join(HERE, "ref_n256.npz"))["elliptic_init"]
    with tempfile.TemporaryDirectory() as d:
        os.makedirs(os.path.join(d, "input"))
        subprocess.run([os.path.join(ROOT, "xlab_fftbarotropic_b200", "bin", "makefield-elliptic-vortex.out")], cwd=d,
                       check=True, stderr=subprocess.DEVNULL)
        v768 = np.fromfile(os.path.join(d, "input", "initial_vorticity.bin"), dtype="<f4").reshape(768, 768)
    for tag, v0, n, steps, rec, stride in (("n256", v256, 256, 5, 2, 8), ("n768", v768, 768, 6, 3, 24)):
        r, src = records(v0, n, 3.0, steps, rec)
        sources.add(src)
        for s in range(0, steps, rec):
            for kind, _ in KINDS:
                for key, val in reduce_field(r[(kind, s)], stride).items():
                    out[f"{tag}_{kind}_{s}_{key}"] = val
    out["source"] = np.array(",".join(sorted(sources)))
    np.savez_compressed(os.path.join(HERE, "ref_records.npz"), **out)
    print("record golden vectors written to", HERE, "from the", out["source"])


if __name__ == "__main__":
    main()
