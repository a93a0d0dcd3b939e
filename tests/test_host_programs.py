"""Host C++ programs: generators byte-identical to the reference (CPU), main.out / invert_pres.out against
the reference main.cpp's record files on the same input (GPU): stored in tests/golden/ref_records.npz
(tests/golden/make_golden_records.py), and every full field against the CPU restatement run live."""
import hashlib
import json
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import check_golden, rel_l2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "xlab_fftbarotropic_b200", "bin")
GOLD = os.path.join(ROOT, "tests", "golden")
KINDS = ("vort", "psi", "u", "v")


def _reference_records(v0, n, dt, steps, rec):
    """{(kind, step): field} of the reference main.cpp's record files, from the CPU restatement (which writes them bit
    for bit, tests/test_oracle.py)"""
    from oracle import oracle as orc
    o = orc.Oracle(n)
    o.set_vorticity(v0)
    out = {}
    for s in range(steps):
        if s % rec == 0:
            for kind in KINDS:
                out[(kind, s)] = o.get_field(getattr(orc, kind.upper()))
        o.step(1, dt)
    return out


def _check_records(d, tag, ref, stride, tol=1e-5):
    """main.out's record files in `d` against ref_records.npz[<tag>_<kind>_<step>] and the full restatement fields"""
    gold = np.load(os.path.join(GOLD, "ref_records.npz"))
    for (kind, s), exp in sorted(ref.items()):
        got = np.fromfile(os.path.join(d, f"output/{kind}_step_{s}.bin"), dtype="<f4").reshape(exp.shape)
        check_golden(got, gold, f"{tag}_{kind}_{s}", stride, tol)         # the reference binary's record file
        assert rel_l2(got, exp) < tol, (kind, s)                          # the restatement, full field


def test_generators_byte_identical_to_reference():
    md5 = json.load(open(os.path.join(GOLD, "generators.json")))
    with tempfile.TemporaryDirectory() as d:
        os.makedirs(os.path.join(d, "input"))
        for name, want in md5.items():
            subprocess.run([os.path.join(BIN, name + ".out")], cwd=d, check=True, stderr=subprocess.DEVNULL)
            got = hashlib.md5(open(os.path.join(d, "input", "initial_vorticity.bin"), "rb").read()).hexdigest()
            assert got == want, name


def _forcing_stream(src, steps, new_at, clear_at=None):
    """the byte stream of src/vort_src_input.cpp:43-61: one flag byte per step, a field after a flag of 1"""
    out = bytearray()
    for step in range(steps):
        if step == new_at:
            out += b"\x01" + src.tobytes()
        elif clear_at is not None and step == clear_at:
            out += b"\x01" + np.zeros_like(src).tobytes()
        else:
            out += b"\x00"
    return bytes(out)


@pytest.mark.gpu
def test_live_fifo_producer_against_the_reference_forcing_program():
    """test/02-test_invert_pressure/example.sh:9-13: `mkfifo fifo; vort_src_input.out > fifo & main.out -f fifo` -- a real
    named pipe fed by a concurrent producer, for our main.out AND for the unmodified reference program that reads the
    pipe (src/main-shallow-water.cpp, built at 256^2 in oracle/_ref); the record files must agree."""
    import threading
    import fields
    ref_exe = os.path.join(ROOT, "oracle", "_ref", "main-shallow-water_n256.out")
    if not os.path.exists(ref_exe):
        pytest.skip("oracle/_ref/main-shallow-water_n256.out is built where /root/reference exists")
    n, steps, rec = 256, 7, 3
    v0 = fields.gaussian(n)
    src = (fields.kuo2004(n) * np.float32(1e-4)).astype(np.float32)
    stream = _forcing_stream(src, steps, new_at=1, clear_at=4)
    results = {}
    for tag in ("xfb", "ref"):
        with tempfile.TemporaryDirectory() as d:
            os.makedirs(os.path.join(d, "input"))
            os.makedirs(os.path.join(d, "output"))
            v0.tofile(os.path.join(d, "input", "initial_vorticity.bin"))
            fifo = os.path.join(d, "vort_src_fifo")
            os.mkfifo(fifo)

            def produce():
                with open(fifo, "wb") as fh:          # blocks until the model opens the pipe for reading
                    for k in range(0, len(stream), 65536):
                        fh.write(stream[k:k + 65536])

            th = threading.Thread(target=produce, daemon=True)
            th.start()
            if tag == "xfb":
                cmd = [os.path.join(BIN, "main.out"), "-n", str(n), "-t", str(steps), "-r", str(rec), "-f", "vort_src_fifo"]
                env = os.environ
            else:
                cmd = [ref_exe, "-f", "vort_src_fifo"]
                env = dict(os.environ, XFB_DT="3.0", XFB_TOTAL_STEPS=str(steps), XFB_RECORD_STEP=str(rec))
            r = subprocess.run(cmd, cwd=d, capture_output=True, text=True, env=env, timeout=300)
            th.join(timeout=30)
            assert r.returncode == 0, r.stderr[-2000:]
            assert not th.is_alive()
            log = [ln.strip() for ln in open(os.path.join(d, "log")) if ln.strip()]
            results[tag] = (log, {p: np.fromfile(os.path.join(d, p), dtype="<f4").reshape(n, n) for p in log})
    assert results["xfb"][0] == results["ref"][0]
    for p in results["ref"][0]:
        a, b = results["xfb"][1][p], results["ref"][1][p]
        if "vort_src_input" in p:
            assert np.array_equal(a, b), p            # the forcing field itself: step 0 zeros, step 3 src, step 6 zeros
        else:
            assert rel_l2(a, b) < 1e-5, p


@pytest.mark.gpu
def test_script_recipe_forcing():
    """SCRIPT recipe (`[time] [binary filename]` lines, '#' comments: format at src/vorticity_source.cpp:13-19; the
    reference's readScript is an empty stub, :100-110): the field of the last line whose time <= t is active."""
    from oracle import oracle as orc
    import fields
    n, dt = 256, 3.0
    v0 = fields.gaussian(n)
    src_a = (fields.kuo2004(n) * np.float32(1e-4)).astype(np.float32)
    src_b = (fields.elliptic(n) * np.float32(-5e-5)).astype(np.float32)
    with tempfile.TemporaryDirectory() as d:
        os.makedirs(os.path.join(d, "input"))
        os.makedirs(os.path.join(d, "output"))
        v0.tofile(os.path.join(d, "input", "initial_vorticity.bin"))
        src_a.tofile(os.path.join(d, "src_a.bin"))
        src_b.tofile(os.path.join(d, "src_b.bin"))
        with open(os.path.join(d, "recipe.txt"), "w") as fh:
            fh.write("# time  file\n3.0 src_a.bin   # active from step 1 (t = 3 s)\n\n9.0 src_b.bin\n")
        r = subprocess.run([os.path.join(BIN, "main.out"), "-n", str(n), "-t", "6", "-r", "5", "-d", str(dt), "-s", "recipe.txt"],
                           cwd=d, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        o = orc.Oracle(n)
        o.set_vorticity(v0)
        o.step(1, dt)                 # step 0: t = 0, nothing active
        o.set_source(src_a)
        o.step(2, dt)                 # steps 1, 2: t = 3, 6
        o.set_source(src_b)
        o.step(2, dt)                 # steps 3, 4: t = 9, 12
        got = np.fromfile(os.path.join(d, "output/vort_step_5.bin"), dtype="<f4").reshape(n, n)
        assert rel_l2(got, o.get_field(orc.VORT)) < 1e-5
        assert np.array_equal(np.fromfile(os.path.join(d, "output/vort_src_input_step_5.bin"), dtype="<f4").reshape(n, n), src_b)
        # a recipe that names a missing file stops the run instead of integrating with a stale buffer
        with open(os.path.join(d, "bad.txt"), "w") as fh:
            fh.write("0.0 nowhere.bin\n")
        r2 = subprocess.run([os.path.join(BIN, "main.out"), "-n", str(n), "-t", "2", "-s", "bad.txt"], cwd=d, capture_output=True, text=True)
        assert r2.returncode != 0


@pytest.mark.gpu
def test_main_out_matches_reference_binary():
    n, steps, rec = 256, 5, 2
    g = np.load(os.path.join(GOLD, "ref_n256.npz"))
    v0 = g["elliptic_init"]
    ref = _reference_records(v0, n, 3.0, steps, rec)
    with tempfile.TemporaryDirectory() as d:
        os.makedirs(os.path.join(d, "input"))
        os.makedirs(os.path.join(d, "output"))
        v0.tofile(os.path.join(d, "input", "initial_vorticity.bin"))
        r = subprocess.run([os.path.join(BIN, "main.out"), "-n", str(n), "-t", str(steps), "-r", str(rec)], cwd=d,
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert "# Step 0, time = 0.00, record now!" in r.stdout and "Program ends. Congrats!" in r.stdout
        log = [ln.strip() for ln in open(os.path.join(d, "log"))]
        want = [f"output/{k}_step_{s}.bin" for s in (0, 2, 4) for k in ("vort_src_input", "vort", "psi", "u", "v")]
        assert log == want                                   # same files, same order as the reference's log
        _check_records(d, "n256", ref, 8)


@pytest.mark.gpu
def test_example_sh_default_grid_768():
    """test/01-runtest/example.sh with the reference's compile-time defaults: makefield-elliptic-vortex.out writes
    input/initial_vorticity.bin at NPTS = 768 (src/configuration.hpp:18), main.out runs it with no size flag;
    compared file by file with the reference's record files at 768 (shortened to 6 steps, record every 3)."""
    n, steps, rec = 768, 6, 3
    with tempfile.TemporaryDirectory() as d:
        os.makedirs(os.path.join(d, "input"))
        os.makedirs(os.path.join(d, "output"))
        subprocess.run([os.path.join(BIN, "makefield-elliptic-vortex.out")], cwd=d, check=True, stderr=subprocess.DEVNULL)
        v0 = np.fromfile(os.path.join(d, "input", "initial_vorticity.bin"), dtype="<f4")
        assert v0.size == n * n
        v0 = v0.reshape(n, n)
        ref = _reference_records(v0, n, 3.0, steps, rec)
        r = subprocess.run([os.path.join(BIN, "main.out"), "-t", str(steps), "-r", str(rec)], cwd=d, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        _check_records(d, "n768", ref, 24)


@pytest.mark.gpu
def test_main_out_fifo_forcing_and_invert_pres():
    from oracle import oracle as orc
    import fields
    n = 256
    v0 = fields.gaussian(n)
    src = (fields.kuo2004(n) * np.float32(1e-4)).astype(np.float32)
    with tempfile.TemporaryDirectory() as d:
        os.makedirs(os.path.join(d, "input"))
        os.makedirs(os.path.join(d, "output"))
        v0.tofile(os.path.join(d, "input", "initial_vorticity.bin"))
        # forcing stream: step 0 no change, step 1 new field, steps 2.. no change   (vort_src_input.cpp:43-61)
        with open(os.path.join(d, "forcing.bin"), "wb") as fh:
            fh.write(b"\x00")
            fh.write(b"\x01")
            fh.write(src.tobytes())
            fh.write(b"\x00" * 8)
        r = subprocess.run([os.path.join(BIN, "main.out"), "-n", str(n), "-t", "4", "-r", "3", "-f", "forcing.bin"],
                           cwd=d, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        o = orc.Oracle(n)
        o.set_vorticity(v0)
        o.step(1, 3.0)
        o.set_source(src)
        o.step(2, 3.0)
        got = np.fromfile(os.path.join(d, "output/vort_step_3.bin"), dtype="<f4").reshape(n, n)
        assert rel_l2(got, o.get_field(orc.VORT)) < 1e-5
        assert np.array_equal(np.fromfile(os.path.join(d, "output/vort_src_input_step_3.bin"), dtype="<f4").reshape(n, n), src)
        # pressure inversion pipeline of test/01-runtest/invert.sh: psi_step_N.bin => pres_step_N.bin
        r2 = subprocess.run([os.path.join(BIN, "invert_pres.out"), "-n", str(n), "-x", "3", "-y", "5"], cwd=d,
                            input="output/psi_step_3.bin=>output/pres_step_3.bin\nnot a pair\n", capture_output=True, text=True)
        assert r2.returncode == 0 and "Error reading input: not a pair" in r2.stdout
        psi = np.fromfile(os.path.join(d, "output/psi_step_3.bin"), dtype="<f4").reshape(n, n)
        pres = np.fromfile(os.path.join(d, "output/pres_step_3.bin"), dtype="<f4").reshape(n, n)
        assert rel_l2(pres, o.invert_pres(psi, 3, 5)) < 1e-5


@pytest.mark.gpu
def test_gpu_against_golden_reference_files():
    """the CUDA path against files written by the unmodified reference binary (committed fixtures)"""
    import xlab_fftbarotropic_b200 as xfb
    g = np.load(os.path.join(GOLD, "ref_n256.npz"))
    b = xfb.Backend(256)
    b.set_vorticity(g["elliptic_init"])
    b.step(1, 3.0)
    for kind, which in (("vort", xfb.capi.VORT), ("psi", xfb.capi.PSI), ("u", xfb.capi.U), ("v", xfb.capi.V)):
        assert rel_l2(b.get_field(which), g[f"elliptic_{kind}_1"]) < 1e-5, kind
    assert rel_l2(b.invert_pres(g["elliptic_psi_1"], 3, 5), g["elliptic_pres_1"]) < 1e-5
    b.set_vorticity(g["kuo_init"])
    b.step(10, 3.0)
    assert rel_l2(b.get_field(xfb.capi.VORT), g["kuo_vort_10"]) < 1e-5
    b.close()


@pytest.mark.gpu
def test_main_out_ensemble_members_flag():
    """main.out -b <members>: per-member initial files (`%d` in -i), reference file names for member 0 and `.m<k>` for
    the others; every member must equal its own single-member run bit for bit"""
    import fields
    n, steps, rec = 256, 4, 3
    inits = [fields.gaussian_member(n, m) for m in range(3)]
    with tempfile.TemporaryDirectory() as d:
        os.makedirs(os.path.join(d, "input"))
        os.makedirs(os.path.join(d, "output"))
        for m, v in enumerate(inits):
            v.tofile(os.path.join(d, "input", f"init_{m}.bin"))
        r = subprocess.run([os.path.join(BIN, "main.out"), "-n", str(n), "-t", str(steps), "-r", str(rec), "-b", "3", "-i", "init_%d.bin", "-q"],
                           cwd=d, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        ens = {}
        for m in range(3):
            suffix = "" if m == 0 else f".m{m}"
            ens[m] = np.fromfile(os.path.join(d, f"output/vort_step_3{suffix}.bin"), dtype="<f4")
        log = [ln.strip() for ln in open(os.path.join(d, "log")) if ln.strip()]
        assert log[:3] == ["output/vort_src_input_step_0.bin", "output/vort_src_input_step_0.m1.bin", "output/vort_src_input_step_0.m2.bin"]
        for m in range(3):
            with tempfile.TemporaryDirectory() as d1:
                os.makedirs(os.path.join(d1, "input"))
                os.makedirs(os.path.join(d1, "output"))
                inits[m].tofile(os.path.join(d1, "input", "initial_vorticity.bin"))
                r1 = subprocess.run([os.path.join(BIN, "main.out"), "-n", str(n), "-t", str(steps), "-r", str(rec), "-q"], cwd=d1,
                                    capture_output=True, text=True)
                assert r1.returncode == 0, r1.stderr
                one = np.fromfile(os.path.join(d1, "output/vort_step_3.bin"), dtype="<f4")
            assert np.array_equal(ens[m], one), m


def _gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.gpu
def test_main_out_multi_gpu_modes():
    """main.out -G 2 (ensemble members over two devices) and -S 2 (one grid slab-decomposed over two devices, one forked
    rank per GPU, every rank reading and writing its own rows of the same files) against the single-GPU run"""
    if _gpu_count() < 2:
        pytest.skip("needs two GPUs")
    import fields
    n, steps, rec = 512, 4, 3
    v0 = fields.kuo2004(n)
    outs = {}
    for tag, extra in (("one", []), ("slab", ["-S", "2"]), ("ens", ["-b", "2", "-G", "2"])):
        with tempfile.TemporaryDirectory() as d:
            os.makedirs(os.path.join(d, "input"))
            os.makedirs(os.path.join(d, "output"))
            v0.tofile(os.path.join(d, "input", "initial_vorticity.bin"))
            r = subprocess.run([os.path.join(BIN, "main.out"), "-n", str(n), "-t", str(steps), "-r", str(rec), *extra], cwd=d,
                               capture_output=True, text=True, timeout=600)
            assert r.returncode == 0, r.stderr[-2000:]
            assert "Program ends. Congrats!" in r.stdout
            names = ["vort_step_3.bin", "psi_step_3.bin", "u_step_0.bin"] + (["vort_step_3.m1.bin"] if tag == "ens" else [])
            outs[tag] = {k: np.fromfile(os.path.join(d, "output", k), dtype="<f4") for k in names}
            outs[tag]["log"] = [ln.strip() for ln in open(os.path.join(d, "log")) if ln.strip()]
    for k in ("vort_step_3.bin", "psi_step_3.bin", "u_step_0.bin"):
        assert rel_l2(outs["slab"][k], outs["one"][k]) < 2e-6, k
        assert np.array_equal(outs["ens"][k], outs["one"][k]), k
    assert np.array_equal(outs["ens"]["vort_step_3.m1.bin"], outs["one"]["vort_step_3.bin"])
    assert outs["slab"]["log"] == outs["one"]["log"]
