"""bench.py --impl reference on the CPU: exactly one JSON line on stdout with the keys of the measurement contract."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--n", "4096"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "schnorr_sig_verifies_per_sec" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_reference_arm_dumps_the_verdicts_of_its_last_step(tmp_path):
    import numpy as np
    from rusty_kaspa_b200 import workload as W
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--n", "4096",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    st = np.load(tmp_path / "status.npy")
    _, _, _, kind = W.schnorr_triples(4096, seed=0x6B61737061)
    assert st.dtype == np.float32 and st.shape == (4096,)
    assert ((st == 1) == (kind == 0)).all()


def test_dump_outputs_samples_large_outputs_the_same_way_every_time(tmp_path, monkeypatch):
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 4000)
    arrays = {"status": np.arange(8000, dtype=np.uint8), "bitmap": np.arange(1000, dtype=np.uint8)}
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    sizes = 0
    for name in arrays:
        a, b = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert a.dtype == np.float32 and (a == b).all() and 0 < len(a) < len(arrays[name])
        sizes += a.nbytes
    assert sizes <= 4000
    bench.dump_outputs(str(tmp_path / "c"), {"status": np.arange(10, dtype=np.uint8)})
    assert (np.load(tmp_path / "c" / "status.npy") == np.arange(10)).all()
