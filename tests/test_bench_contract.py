"""bench.py contract, CPU side: the reference arm (`--impl reference`: the CPU oracle on the host cores, no GPU involved) must
print exactly ONE JSON line on stdout carrying the keys the driver parses, with the same `config`, `metric` and `unit` the GPU
arm reports.  (The GPU arm itself is exercised on the GPU box: profiles/r02_bench_n1.json.)"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    sys.path.insert(0, ROOT)
    import bench
    assert d["impl"] == "reference" and d["metric"] == "r1cs_proofs_per_sec" and d["unit"] == "proofs/s"
    assert d["config"] == bench.config_dict() and "2^20" in d["config"]["workload"]
    assert d["steps"] == 1 and d["warmup"] == 0 and d["n_gpus"] == 1
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_dumps_last_step_outputs(tmp_path):
    """--dump-outputs writes the proof and commitments the timed steps computed, as float32 byte values that equal a fresh oracle
    proof of the same instance"""
    import numpy as np
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    sys.path.insert(0, ROOT)
    import bench
    import oracle_lib as ol
    from bulletproofs_gadgets_b200 import gadgets
    inst = gadgets.merkle_tree_instances(bench.REF_SAMPLE_LEAVES, [None], trace_on_device=False)[0]
    try:
        _, proof, V = bench.oracle_prove(inst, 1 << 16, bytes(32), os.cpu_count() or 1)
    finally:
        ol.lib().bpo_set_threads(1)
    for name, want in (("proofs", proof), ("commitments", V)):
        got = np.load(str(tmp_path / (name + ".npy")))
        assert got.dtype == np.float32 and got.shape == (1, len(want))
        assert bytes(got[0].astype(np.uint8)) == want


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""
