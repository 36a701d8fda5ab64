"""CPU suite: the reference arm of bench.py (`--impl reference`) -- the one bench leg that needs no GPU.  It must print exactly
one JSON line with the contract's keys, time the unmodified reference's own modules when the tree (or its staged copy) is
importable, and fall back to the oracle port when it is not."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra):
    env = dict(os.environ)
    env.update(env_extra)
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "1"], cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-1500:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout[-1500:]
    return json.loads(lines[0])


@pytest.mark.parametrize("mode", ["default", "no_reference_tree"])
def test_reference_arm_prints_one_contract_line(mode):
    from oracle import ref_shim
    d = _run({} if mode == "default" else {"CFT_REFERENCE_ROOT": "/nonexistent"})
    assert d["impl"] == "reference" and d["unit"] == "pairs/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["metric"].startswith("RGB+IR pairs/sec") and d["gpu_launches"] == 0 and d["dtype"] == "f32"
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["value"] == d["value"] and cb["cores"] >= 1
    want = "reference" if (mode == "default" and ref_shim.available()) else "port"
    assert cb["kind"] == want, cb


def test_reference_arm_times_every_step_and_dumps_the_last_output(tmp_path, monkeypatch):
    """`--steps` is the number of timed forwards, and `--dump-outputs` writes what the last of them returned: the arm's
    forward is replaced by one that counts its calls and returns a distinct z each time."""
    import numpy as np
    import torch
    import bench
    calls = []

    def fwd():
        calls.append(None)
        return torch.full((1, 7, 8), float(len(calls))), None
    monkeypatch.setattr(bench, "cpu_forward", lambda batch: (fwd, "port", "counting stub"))
    monkeypatch.setattr(bench, "best_thread_count", lambda f: 1)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--steps", "11", "--warmup", "1",
                                      "--dump-outputs", str(tmp_path)])
    bench.main()
    assert len(calls) == 11                                        # warm-up 1 = the thread probe only (stubbed here)
    z = np.load(tmp_path / "z.npy")
    assert z.dtype == np.float32 and z.shape == (1, 7, 8) and (z == 11.0).all()
    for steps in ("0", "-3"):
        monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--steps", steps])
        with pytest.raises(SystemExit):
            bench.main()
