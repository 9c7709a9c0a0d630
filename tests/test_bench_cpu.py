"""bench.py --dump-outputs on the CPU reference arm (no GPU needed): the files hold what the last timed step returned,
in float64, identical from run to run and equal to the serial oracle stepping the same workload."""
import json
import os
import subprocess
import sys

import numpy as np

from common import base_kw, synth_psi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    env = dict(os.environ, OMP_NUM_THREADS="1")   # the OpenMP sweep repeats its bits with one thread only
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stdout + out.stderr
    return out


def test_dump_outputs_reference_arm(tmp_path):
    from oracle import oracle as O
    N, nl, steps, warmup = 64, 2, 3, 1
    for d in ("a", "b"):
        out = _bench("--impl", "reference", "--N", str(N), "--nl", str(nl), "--steps", str(steps), "--warmup", str(warmup),
                     "--dump-outputs", str(tmp_path / d))
        line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        assert line["config"]["timed_steps"] == steps
    got = {}
    for name in ("dt", "t", "psi", "q"):
        a, b = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert a.dtype == np.float64 and np.array_equal(a, b), name
        got[name] = a
    m = O.Model(O.make_params(**base_kw(N, nl)))
    m.set(O.PSI, synth_psi(N, nl))
    m.set_const()
    dts = [m.step() for _ in range(warmup + steps)]
    assert got["dt"].tolist() == [dts[-1]] and got["t"].tolist() == [m.t]
    assert np.array_equal(got["psi"], m.get(O.PSI).ravel()) and np.array_equal(got["q"], m.get(O.Q).ravel())
    m.close()


def test_dump_sample_is_fixed():
    """fields larger than DUMP_SAMPLE values are cut to the same sorted sample of distinct cells on every run"""
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import numpy as np, bench\n"
            "n = 4096 * 4096 * 4\n"
            "i, j = bench.dump_indices(n), bench.dump_indices(n)\n"
            "assert np.array_equal(i, j) and i.size == bench.DUMP_SAMPLE and (np.diff(i) > 0).all() and 0 <= i[0] and i[-1] < n\n"
            "assert np.array_equal(bench.dump_indices(1000), np.arange(1000))\n"
            "print('ok')\n") % ROOT
    out = subprocess.run([sys.executable, "-B", "-c", code], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 0 and "ok" in out.stdout, out.stdout + out.stderr


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr
