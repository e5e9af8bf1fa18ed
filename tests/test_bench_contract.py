"""Checks of bench.py's contract: the reference arm prints exactly one JSON line with the agreed keys, our arm refuses to
run without a CUDA device (the product has no CPU path), and --dump-outputs writes the timed proof's transcript."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "gkr_prover_gates_per_s" and d["unit"] == "gates/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_our_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "3"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode != 0
    assert "no CUDA device" in (r.stderr + r.stdout)
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]   # no number without a GPU


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode != 0 and "--steps must be at least 1" in r.stderr
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_dump_outputs_keeps_every_bit(tmp_path):
    """--dump-outputs stores field elements as float32 bytes: exact, and any changed element differs by >= 1 somewhere"""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    P = (1 << 61) - 1
    rng = np.random.default_rng(5)
    tr = np.zeros(1000, [("re", "<u8"), ("im", "<u8")])
    tr["re"] = rng.integers(0, P, len(tr), dtype=np.uint64)
    tr["im"] = rng.integers(0, P, len(tr), dtype=np.uint64)
    tr[0] = (P - 1, 0)
    bench.dump_outputs(str(tmp_path / "out"), tr)
    d = np.load(tmp_path / "out" / "transcript.npy")
    assert d.dtype == np.float32 and d.shape == (len(tr), 16)
    assert (d.astype(np.uint8).view(tr.dtype).ravel() == tr).all()


@pytest.mark.gpu
def test_dump_outputs_is_the_proof_of_the_timed_circuit(tmp_path, B, O, sha_circuit):
    """bench.py --dump-outputs on a small workload: one JSON line, and the dumped transcript is the oracle's proof of the same
    circuit (SHA256_64 x 2) with the same challenges"""
    import numpy as np
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--instances", "2",
                        "--no-extras", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    assert len([l for l in r.stdout.splitlines() if l.strip()]) == 1, r.stdout[-2000:]
    assert json.loads(r.stdout)["steps"] == 2
    got = np.load(tmp_path / "transcript.npy").astype(np.uint8).view(B.F_DTYPE).ravel()
    want, _, _ = O.OracleCircuit(sha_circuit.replicate(2).expand().flat()).prove()
    assert (got["re"] == want["re"]).all() and (got["im"] == want["im"]).all()


_GUARD_SCRIPT = r'''
import ctypes, os, sys
sys.argv = ["bench.py"]
sys.path.insert(0, %r)
import bench
line = {"metric": "m", "value": 1}
g = bench.LineGuard(line, armed=True, deadline_s=float(os.environ["DL"]))
g.leg("failing_leg", lambda: 1 / 0)
g.leg("fine_leg", lambda: {"x": 2})
sys.stderr.write("READY\n"); sys.stderr.flush()
if os.environ["MODE"] == "ok":
    g.finish(); g.finish()           # the line is printed once
else:
    libc = ctypes.CDLL(None)
    while True:                      # a main thread stuck inside a C call (a collective whose peer died)
        libc.sleep(30)
'''


def _run_guard(mode, deadline, send_term=False):
    import signal
    import time
    p = subprocess.Popen([sys.executable, "-c", _GUARD_SCRIPT % ROOT], env=dict(os.environ, MODE=mode, DL=str(deadline)),
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    if send_term:
        assert p.stderr.readline().strip() == "READY"   # the guard is installed
        time.sleep(1)                                    # main thread inside libc.sleep
        p.send_signal(signal.SIGTERM)
    out, err = p.communicate(timeout=120)
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1, (out, err[-2000:])
    return p.returncode, json.loads(lines[0])


def test_bench_line_survives_failing_hanging_and_terminated_legs():
    """bench.py's LineGuard: a side measurement that throws fills its own slot; a hang after the timed regions or a
    SIGTERM from the launcher still yields the ONE JSON line (with a note), printed exactly once."""
    rc, d = _run_guard("ok", 60)
    assert rc == 0 and d["value"] == 1 and "ZeroDivisionError" in d["failing_leg"]["error"] and d["fine_leg"] == {"x": 2}
    assert "extras_error" not in d
    rc, d = _run_guard("hang", 2)
    assert rc == 0 and d["value"] == 1 and "did not finish" in d["extras_error"]
    rc, d = _run_guard("hang", 120, send_term=True)
    assert rc != 0 and d["value"] == 1 and "signal" in d["extras_error"]
