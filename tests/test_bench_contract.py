"""bench.py's CPU-only legs and the JSON contract of its line (the GPU arm is exercised on the box).  The reference arm
(`--impl reference`) must run without the engine, print ONE JSON line and carry the keys the driver compares across arms."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--n", "3000", "--ref-sample", "3000", "--keys", "64",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "Ed25519 verifies/s" and d["unit"] == "verifies/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["value"] > 1000 and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and abs(d["cpu_baseline"]["value"] - d["value"]) < 1e-6
    assert d["e2e"] == {"value": d["value"], "unit": "verifies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "config[1]" in d["config"]["workload"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"], capture_output=True,
                         text=True, cwd=ROOT, env=env, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_input_synthesis_with_the_oracle_signer_matches_openssl():
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import hashlib
    import bench
    from oracle_api import Oracle
    from cryptography.hazmat.primitives.asymmetric.ed25519 import Ed25519PublicKey
    o = Oracle()
    inp = bench.make_inputs(500, 16, 512, seed=9, corrupt_frac=0.02, oracle=o)
    assert inp["sig"].shape == (500, 64) and inp["msgs"].shape == (500, 512) and int(inp["corrupted"].sum()) == 10
    for i in range(0, 500, 37):
        if inp["corrupted"][i]:
            continue
        d = hashlib.sha512(inp["msgs"][i].tobytes()).digest()[:32]
        Ed25519PublicKey.from_public_bytes(inp["pk"][i].tobytes()).verify(inp["sig"][i].tobytes(), d)   # raises on a bad signature
    ok = o.verify_rec128(__import__("numpy").concatenate([inp["sig"], inp["pk"], o.digest32_batch(inp["msgs"].reshape(-1), __import__("numpy").arange(501, dtype="uint64") * 512)], axis=1))
    assert (ok == ~inp["corrupted"]).all()


def test_dumped_outputs_are_float32_and_large_ones_a_fixed_row_sample(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    monkeypatch.setattr(bench, "DUMP_MAX_ELEMS", 64)
    flags = np.arange(64) % 3 == 0
    big = np.arange(100 * 4, dtype=np.int32).reshape(100, 4)
    bench.write_outputs(str(tmp_path / "a"), small=flags, big=big)
    bench.write_outputs(str(tmp_path / "b"), big=big)
    small, got = np.load(tmp_path / "a" / "small.npy"), np.load(tmp_path / "a" / "big.npy")
    assert small.dtype == np.float32 and (small == flags).all()
    assert got.dtype == np.float32 and got.shape == (16, 4) and (np.load(tmp_path / "b" / "big.npy") == got).all()
    rows = got[:, 0].astype(int) // 4
    assert (np.diff(rows) > 0).all() and (got == big[rows]).all()


class _OracleSigner:
    """The engine's load-generation signer answered by the CPU oracle: RFC 8032 signing is deterministic, so bench.make_inputs
    produces the same records through it as through the engine."""

    def __init__(self, o):
        self.o = o

    def keygen_batch(self, seeds):
        return self.o.keygen_batch(seeds)

    def digest32_batch(self, data, off):
        return self.o.digest32_batch(data, off)

    def sign_digests(self, seeds, pks, digests, key_idx):
        import numpy as np
        return self.o.sign_batch(seeds, pks, key_idx, digests.reshape(-1), np.arange(len(key_idx) + 1, dtype=np.uint64) * 32)


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_steps_verdicts_and_digests(tmp_path):
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import bench
    from oracle_api import Oracle
    n = 3000
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--n", str(n), "--keys", "16", "--steps", "2", "--warmup", "1", "--no-strong",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 2
    o = Oracle()
    inp = bench.make_inputs(n, 16, 512, seed=1234, corrupt_frac=0.01, engine=_OracleSigner(o))
    accept, digest = np.load(tmp_path / "accept.npy"), np.load(tmp_path / "digest.npy")
    assert accept.dtype == np.float32 and digest.dtype == np.float32
    assert (accept == ~inp["corrupted"]).all()
    assert (digest == o.digest32_batch(inp["msgs"].reshape(-1), np.arange(n + 1, dtype=np.uint64) * 512)).all()
