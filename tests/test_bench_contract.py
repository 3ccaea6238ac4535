"""CPU: bench.py's reference arm prints one JSON line with the contract's keys (tiny sample), and the GPU arm's
helpers parse MEASURED_PEAKS / fall back as documented."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_contract_json():
    env = dict(os.environ, B200H_REF_SAMPLE="64")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, env=env, cwd=ROOT, timeout=300)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "GiB/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, env=env, cwd=ROOT, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_hbm_peak_source():
    sys.path.insert(0, ROOT)
    import bench

    peak, src = bench.hbm_peak_gbs()
    assert peak > 1000 and ("measured" in src or "fallback" in src)


def test_e2e_leg_of_the_gpu_arm_runs_on_the_host_layer(fake_backend, monkeypatch):
    """bench.py's headline e2e leg (run_map_pump + NullStub + _null_put) is ordinary host code around the hash call:
    with the oracle-backed stand-in for the context it must push every payload through the real
    InputPreprocessor / InputPumper, keep the per-window digest tables, and tell BlobCreate the digests hashlib gives."""
    import base64
    import hashlib

    import numpy as np

    sys.path.insert(0, ROOT)
    import bench
    from modal_client_b200 import blob_utils, parallel_map

    monkeypatch.setattr(blob_utils, "_upload_to_s3_url", bench._null_put)
    monkeypatch.setattr(parallel_map, "HASH_WINDOW_BYTES", 64 * 1024)
    payloads = [bytes([i % 251, (i * 7) % 256]) * (1000 + 13 * i) for i in range(150)]
    stub = bench.NullStub()
    dt, batches, tables = bench.run_map_pump(payloads, stub)
    assert dt > 0 and batches >= 4 and stub.inputs_put == len(payloads)
    sha = np.concatenate([t[0] for t in tables])
    md5 = np.concatenate([t[1] for t in tables])
    assert [r.content_length for r in stub.blob_requests] == [len(p) for p in payloads]
    for i, (r, p) in enumerate(zip(stub.blob_requests, payloads)):
        assert base64.b64decode(r.content_sha256_base64) == hashlib.sha256(p).digest() == sha[i].tobytes()
        assert base64.b64decode(r.content_md5) == hashlib.md5(p).digest() == md5[i].tobytes()
    assert set(bench.run_map_pump.last_stats) == {"collect_s", "wait_context_s", "hash_call_s", "wait_hash_s"}


def test_dump_outputs_writes_float32_tables_within_the_size_bound(tmp_path, monkeypatch):
    """--dump-outputs: every table as float32 <name>.npy; past the byte bound, the same seeded rows of each (twice the
    same), with their indices in rows.npy."""
    import numpy as np

    sys.path.insert(0, ROOT)
    import bench

    rng = np.random.default_rng(5)
    tables = {"sha256": rng.integers(0, 256, (1000, 32), dtype=np.uint8),
              "md5": rng.integers(0, 256, (1000, 16), dtype=np.uint8)}
    bench.dump_outputs(str(tmp_path / "full"), tables)
    for name, t in tables.items():
        got = np.load(tmp_path / "full" / f"{name}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, t)
    assert not (tmp_path / "full" / "rows.npy").exists()

    monkeypatch.setattr(bench, "OUTPUT_DUMP_BYTES", 100 * 48 * 4)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), tables)
    total = sum(f.stat().st_size for f in (tmp_path / "a").iterdir())
    assert total <= 100 * 48 * 4 + 3 * 128  # .npy headers
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert rows.dtype == np.float64 and np.array_equal(rows, np.load(tmp_path / "b" / "rows.npy"))
    for name, t in tables.items():
        got = np.load(tmp_path / "a" / f"{name}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, t[rows.astype(np.int64)])
        assert np.array_equal(got, np.load(tmp_path / "b" / f"{name}.npy"))
