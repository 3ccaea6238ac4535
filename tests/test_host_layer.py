"""Host layer (drop-in hash_utils / blob_utils / segment payload): every test runs twice -- on the
oracle-backed stand-in (CPU, host logic only) and on the real library (GPU marker)."""
import asyncio
import base64
import hashlib
import io
import os
import random
from pathlib import Path, PurePosixPath

import numpy as np
import pytest

from modal_client_b200 import blob_utils, hash_utils
from modal_client_b200.exception import ExecutionError
from modal_client_b200.synth import materialize, synth_bytes
from tests.blob_server import FakeBlobStub, running_blob_server


@pytest.fixture(params=["fake", pytest.param("gpu", marks=pytest.mark.gpu)])
def backend(request):
    return request.getfixturevalue("fake_backend" if request.param == "fake" else "gpu_backend")


# ----------------------------------------------------------------------------------------- hash_utils


def test_hash_utils_golden(backend, golden):
    doc = golden("hash_utils.json")
    for c in doc["bytes_cases"]:
        data = materialize(c["input"])
        if len(data) > 2_000_000 and backend.device < 0:
            continue  # keep the CPU suite quick
        up = hash_utils.get_upload_hashes(data)
        assert (up.md5_base64, up.sha256_base64) == (c["md5_base64"], c["sha256_base64"])
        assert (up.md5_hex(), up.sha256_hex()) == (c["md5_hex"], c["sha256_hex"])
        assert hash_utils.get_sha256_hex(data) == c["get_sha256_hex"]
        assert hash_utils.get_sha256_base64(io.BytesIO(data)) == c["get_sha256_base64"]
        assert hash_utils.get_md5_base64(data) == c["get_md5_base64"]
    for c in doc["stream_cases"]:
        fp = io.BytesIO(materialize(c["input"]))
        fp.seek(c["pos"])
        up = hash_utils.get_upload_hashes(fp)
        assert fp.tell() == c["pos_after"]
        assert (up.md5_base64, up.sha256_base64) == (c["md5_base64"], c["sha256_base64"])
    for c in doc["supplied_cases"]:
        up = hash_utils.get_upload_hashes(materialize(c["input"]), **c["kwargs"])
        assert (up.md5_base64, up.sha256_base64) == (c["md5_base64"], c["sha256_base64"])


def test_supplied_digests_skip_the_gpu(fake_backend):
    up = hash_utils.get_upload_hashes(b"x" * 100, sha256_hex="ab" * 32, md5_hex="cd" * 16)
    assert fake_backend.calls == []
    assert base64.b64decode(up.sha256_base64).hex() == "ab" * 32


def test_update_rejects_text_streams(backend):
    with pytest.raises(ValueError, match="Only accepts bytes"):
        hash_utils.get_sha256_hex(io.StringIO("not bytes"))


def test_stream_uses_patched_chunk_size(backend, monkeypatch):
    monkeypatch.setattr(hash_utils, "HASH_CHUNK_SIZE", 7)
    data = synth_bytes(5, 1000)
    assert hash_utils.get_sha256_hex(io.BytesIO(data)) == hashlib.sha256(data).hexdigest()


def test_many_equals_one_by_one(backend):
    payloads = [synth_bytes(40 + i, n) for i, n in enumerate([0, 1, 64, 4097, 262144, 70000])]
    many = hash_utils.get_upload_hashes_many(payloads)
    for p, h in zip(payloads, many):
        assert h.sha256_hex() == hashlib.sha256(p).hexdigest() and h.md5_hex() == hashlib.md5(p).hexdigest()
    assert hash_utils.get_upload_hashes_many([]) == []


# --------------------------------------------------------------------------------------- FileUploadSpec


def _patch(monkeypatch, patch):
    for k, v in patch.items():
        monkeypatch.setattr(blob_utils, k, v)


def test_file_specs_golden(backend, golden, monkeypatch, tmp_path):
    batch, expect = [], []
    for i, c in enumerate(golden("file_specs.json")["cases"]):
        with monkeypatch.context() as mp:
            _patch(mp, c["patch"])
            data = materialize(c["input"])
            spec = blob_utils.get_file_upload_spec_from_fileobj(io.BytesIO(data), PurePosixPath(c["mount_filename"]), 0o100644 if not c["patch"] else 0o755)
            got = (spec.use_blob, spec.sha256_hex, spec.md5_hex, spec.mode, spec.size, spec.mount_filename, spec.content is not None)
            want = (c["use_blob"], c["sha256_hex"], c["md5_hex"], c["mode"], c["size"], c["mount_filename"], c["has_content"])
            assert got == want
            assert spec.read_content() == data
            if spec.content is not None:
                assert spec.content == data
        if not c["patch"]:
            f = tmp_path / f"f{i}.bin"
            f.write_bytes(data)
            os.chmod(f, 0o644)
            batch.append((f, PurePosixPath(c["mount_filename"]), None))
            expect.append(c)
    # the batched builder returns the same fields (mode from stat)
    specs = blob_utils.get_file_upload_specs(batch)
    for (f, _, _), spec, c in zip(batch, specs, expect):
        assert (spec.use_blob, spec.sha256_hex, spec.md5_hex, spec.size, spec.content is not None) == (
            c["use_blob"], c["sha256_hex"], c["md5_hex"], c["size"], c["has_content"])
        assert spec.mode == 0o644 and spec.source_is_path and spec.read_content() == f.read_bytes()
        one = blob_utils.get_file_upload_spec_from_path(f, PurePosixPath(c["mount_filename"]))
        assert (one.sha256_hex, one.md5_hex, one.mode, one.use_blob) == (spec.sha256_hex, spec.md5_hex, spec.mode, spec.use_blob)


def test_batched_specs_placeholder_md5_class(backend, monkeypatch, tmp_path):
    monkeypatch.setattr(blob_utils, "LARGE_FILE_LIMIT", 4096)
    monkeypatch.setattr(blob_utils, "MULTIPART_UPLOAD_THRESHOLD", 10000)
    files = []
    for i, n in enumerate([100, 4096, 10000, 10001, 30000]):
        f = tmp_path / f"g{i}"
        f.write_bytes(synth_bytes(70 + i, n))
        files.append((f, PurePosixPath(f"/m/g{i}"), 0o600))
    specs = blob_utils.get_file_upload_specs(files)
    assert [s.use_blob for s in specs] == [False, True, True, True, True]
    assert [s.md5_hex == "baadbaad" * 4 for s in specs] == [False, False, False, True, True]
    for (f, _, _), s in zip(files, specs):
        assert s.sha256_hex == hashlib.sha256(f.read_bytes()).hexdigest() and s.mode == 0o600


# ------------------------------------------------------------------------------------- FileUploadSpec2


def test_blocks_golden(backend, golden, monkeypatch):
    doc = golden("blocks.json")
    for c in doc["find_end_of_block"]:
        data = materialize(c["input"])
        assert blob_utils._find_end_of_block(lambda d=data: io.BytesIO(d), c["start"], c["end"]) == c["result"]
    for c in doc["spec2"]:
        data = materialize(c["input"])
        if len(data) > 20_000_000 and backend.device < 0:
            continue
        with monkeypatch.context() as mp:
            _patch(mp, c["patch"])
            spec = asyncio.run(blob_utils.FileUploadSpec2.from_fileobj(io.BytesIO(data), PurePosixPath(c["path"]),
                                                                       asyncio.Semaphore(2), 0o644))
            assert [[b.start, b.end, b.contents_sha256.hex()] for b in spec.blocks] == c["blocks"]
            assert (spec.size, spec.mode, spec.path) == (c["size"], c["mode"], c["path"])
            if spec.blocks:
                src = lambda d=data: io.BytesIO(d)  # noqa: E731
                blk = blob_utils._gather_block(src, len(spec.blocks) - 1)
                assert [blk.start, blk.end, blk.contents_sha256.hex()] == c["blocks"][-1]
                assert blob_utils._hash_range_sha256(src, blk.start, blk.end) == blk.contents_sha256


def test_spec2_batched_tree(backend, monkeypatch, tmp_path):
    monkeypatch.setattr(blob_utils, "BLOCK_SIZE", 1000)
    files, contents = [], []
    rng = random.Random(3)
    for i, n in enumerate([0, 1, 999, 1000, 1001, 5500, 12345]):
        data = bytearray(synth_bytes(80 + i, n))
        for _ in range(3):
            if n > 10:
                a = rng.randrange(n)
                data[a : a + rng.randrange(1, 700)] = bytes(min(n, a + 700) - a)[: len(data[a : a + 700])]
        data = bytes(data[:n])
        f = tmp_path / f"t{i}"
        f.write_bytes(data)
        files.append((f, PurePosixPath(f"/v/t{i}"), 0o644))
        contents.append(data)
    specs = asyncio.run(blob_utils.file_upload_specs2(files))
    for data, spec in zip(contents, specs):
        assert spec.size == len(data) and len(spec.blocks) == -(-len(data) // 1000)
        for b in spec.blocks:
            block = data[b.start : b.start + 1000]
            assert b.end == b.start + len(block.rstrip(b"\0"))
            assert b.contents_sha256 == hashlib.sha256(data[b.start : b.end]).digest()
        one = asyncio.run(blob_utils.FileUploadSpec2.from_path(Path(spec.source_description), PurePosixPath(spec.path),
                                                               asyncio.Semaphore(1)))
        assert one.blocks == spec.blocks and one.mode == spec.mode


# ------------------------------------------------------------------------------------------- uploads


def test_multipart_digests_golden(backend, golden):
    for c in golden("multipart.json")["cases"]:
        parts, etag = blob_utils.multipart_part_digests(materialize(c["input"]), c["part_len"])
        assert [p.hex() for p in parts] == c["part_md5_hex"] and etag == c["etag"]


def test_blob_upload_single_and_multipart_round_trip(backend, monkeypatch):
    monkeypatch.setattr(blob_utils, "DEFAULT_SEGMENT_CHUNK_SIZE", 128)

    async def run():
        async with running_blob_server() as (host, store):
            stub = FakeBlobStub(host, multipart_threshold=1024)
            small = synth_bytes(90, 700)
            bid = await blob_utils.blob_upload(small, stub)
            assert store.blobs[bid] == small
            req = stub.requests[-1]
            assert req.content_length == 700
            assert req.content_md5 == base64.b64encode(hashlib.md5(small).digest()).decode()
            assert req.content_sha256_base64 == base64.b64encode(hashlib.sha256(small).digest()).decode()
            # 256 parts + a half part of random bytes, like py/test/blob_test.py:56-66
            big = synth_bytes(91, 256 * 1024 + 512)
            bid = await blob_utils.blob_upload(big, stub)
            assert store.blobs[bid] == big and len(store.parts[bid]) == 257
            # file object path (blob_upload_file) and str payload auto-encoding
            fp = io.BytesIO(big)
            bid = await blob_utils.blob_upload_file(fp, stub)
            assert store.blobs[bid] == big
            bid = await blob_utils.blob_upload("héllo", stub)
            assert store.blobs[bid] == "héllo".encode("utf8")
            # batched pump-style upload keeps order
            payloads = [synth_bytes(100 + i, n) for i, n in enumerate([10, 2000, 999, 5000])]
            out = await blob_utils.blob_upload_many(payloads, stub)
            assert [store.blobs[o[0]] for o in out] == payloads
            assert (await blob_utils.format_blob_data(b"tiny", stub)) == {"data": b"tiny"}
            await blob_utils.ClientSessionRegistry.close_session()

    asyncio.run(run())


def test_blob_download_round_trip_and_failure(backend, monkeypatch):
    """blob_download / blob_iter (py/test/blob_test.py:25-46: upload, download, compare; bl-failure -> error)."""
    monkeypatch.setenv("RETRY_N_ATTEMPTS_OVERRIDE", "2")

    async def run():
        async with running_blob_server() as (host, store):
            stub = FakeBlobStub(host, multipart_threshold=1024)
            for payload in (b"", synth_bytes(92, 700), synth_bytes(93, 5000)):
                bid = await blob_utils.blob_upload(payload, stub)
                assert await blob_utils.blob_download(bid, stub) == payload
                got = b"".join([c async for c in blob_utils.blob_iter(bid, stub)])
                assert got == payload
            with pytest.raises(ExecutionError, match="failed with status 500"):
                await blob_utils.blob_download("bl-failure", stub)
            with pytest.raises(ExecutionError, match="failed with status 500"):
                async for _ in blob_utils.blob_iter("bl-failure", stub):
                    pass
            await blob_utils.ClientSessionRegistry.close_session()

    asyncio.run(run())


def test_upload_integrity_failures(backend, monkeypatch):
    monkeypatch.setenv("RETRY_N_ATTEMPTS_OVERRIDE", "2")

    async def run():
        async with running_blob_server() as (host, store):
            stub = FakeBlobStub(host, multipart_threshold=1 << 20, providers=1)
            with pytest.raises(ExecutionError, match="failed with status 500"):
                await blob_utils.blob_upload(b"FAILURE", stub)
            assert store.puts == 2  # retried once
            store.corrupt_etag = True
            with pytest.raises(ExecutionError, match="checksum mismatch"):
                await blob_utils.blob_upload(b"some payload", stub)
            await blob_utils.ClientSessionRegistry.close_session()

    asyncio.run(run())


def test_segment_payload_md5_and_reset(backend):
    from modal_client_b200.bytes_io_segment_payload import BytesIOSegmentPayload

    class Sink:
        def __init__(self):
            self.data = b""

        async def write(self, chunk):
            self.data += bytes(chunk)

    async def run():
        data = synth_bytes(95, 5000)
        pl = BytesIOSegmentPayload(io.BytesIO(data), segment_start=1000, segment_length=3000, chunk_size=777)
        sink = Sink()
        await pl.write_with_length(sink, None)
        assert sink.data == data[1000:4000] and pl.remaining_bytes() == 0
        assert pl.md5_checksum().hexdigest() == hashlib.md5(data[1000:4000]).hexdigest()
        with pytest.raises(RuntimeError):
            with pl.reset_on_error():
                raise RuntimeError("boom")
        assert pl.num_bytes_read == 0
        sink2 = Sink()
        await pl.write(sink2)
        assert sink2.data == data[1000:4000]
        assert pl.md5_checksum().hexdigest() == hashlib.md5(data[1000:4000]).hexdigest()
        known = BytesIOSegmentPayload(io.BytesIO(data), 0, 5000, md5_digest=hashlib.md5(data).digest())
        assert known.md5_checksum().hexdigest() == hashlib.md5(data).hexdigest() and known.size == 5000

    asyncio.run(run())


def test_byte_budget_limits_inflight():
    async def run():
        budget = blob_utils._ByteBudget(100)
        live, peak = 0, 0

        async def job(n):
            nonlocal live, peak
            async with budget.acquire(n):
                live += n
                peak = max(peak, live)
                await asyncio.sleep(0.01)
                live -= n

        await asyncio.gather(*(job(40) for _ in range(6)), job(500))
        assert peak <= 500 and budget._available == 100

    asyncio.run(run())


def test_use_md5_hosts():
    assert blob_utils.use_md5("https://bucket.s3.amazonaws.com/x") and blob_utils.use_md5("https://a.r2.cloudflarestorage.com/y")
    assert not blob_utils.use_md5("http://localhost:9000/x") and not blob_utils.use_md5("http://127.0.0.1:1/x")
    with pytest.raises(Exception, match="Unknown S3 host"):
        blob_utils.use_md5("https://example.com/x")


def test_bounded_map_order_bound_and_failure():
    """async_utils.bounded_map: results in input order, never more than `concurrency` calls in flight, a fixed number
    of tasks whatever the input length, first failure cancels the rest."""
    from modal_client_b200.async_utils import bounded_map

    async def run():
        live, peak, started = 0, 0, []

        async def fn(x):
            nonlocal live, peak
            live += 1
            peak = max(peak, live)
            started.append(x)
            await asyncio.sleep(0.001 * (x % 3))
            live -= 1
            return x * x

        before = len(asyncio.all_tasks())
        out = await bounded_map(range(200), fn, concurrency=7)
        assert out == [x * x for x in range(200)] and peak == 7 and len(asyncio.all_tasks()) == before
        assert await bounded_map([], fn, concurrency=3) == []
        assert await bounded_map([5], fn, concurrency=100) == [25]

        async def boom(x):
            await asyncio.sleep(0.001)
            if x == 13:
                raise ValueError("thirteen")
            await asyncio.sleep(0.05)
            return x

        started.clear()
        with pytest.raises(ValueError, match="thirteen"):
            await bounded_map(range(1000), boom, concurrency=4)
        await asyncio.sleep(0.1)
        assert len(asyncio.all_tasks()) == before  # the workers were cancelled, nothing keeps running

    asyncio.run(run())


def test_patchable_constants_equal_the_references(golden):
    """Every module constant of the path that callers / tests patch has the reference's name and value
    (hash_utils.py:11, blob_utils.py:40-63, function_utils thresholds, parallel_map chunk sizes, mount / NFS / volume timeouts),
    as oracle/gen_golden.py read them from the reference into tests/golden/seam.json."""
    import importlib

    want = golden("seam.json")["constants"]
    assert set(want) == {"hash_utils", "blob_utils", "mount", "volume", "network_file_system", "parallel_map"}
    for module, constants in want.items():
        ours = importlib.import_module(f"modal_client_b200.{module}")
        for name, value in constants.items():
            assert getattr(ours, name) == value, f"{module}.{name}"


def test_batched_specs_hash_the_bytes_they_cache_and_redo_files_that_grew(fake_backend, tmp_path, monkeypatch):
    """ADVICE r1: (1) a cached-content file is read once and exactly those bytes are hashed; (2) a file that grew between
    the stat and the read is not silently reported with the digest of its old prefix."""
    import hashlib

    small = tmp_path / "small.bin"
    small.write_bytes(b"s" * 1000)
    grown = tmp_path / "grown.bin"
    grown.write_bytes(b"g" * 300_000)  # streamed class (>= 256 KiB)
    real_stat = fake_backend.stat_files
    calls = {"n": 0}

    def stale_first_stat(paths):
        sizes, modes = real_stat(paths)
        calls["n"] += 1
        if calls["n"] == 1:  # what a stat taken before the file was appended to would have said
            sizes = sizes.copy()
            sizes[[i for i, p in enumerate(paths) if p.endswith(b"grown.bin")]] = 299_000
        return sizes, modes

    monkeypatch.setattr(fake_backend, "stat_files", stale_first_stat)
    reads = []
    real_open = open

    def counting_open(path, *a, **k):
        reads.append(str(path))
        return real_open(path, *a, **k)

    monkeypatch.setattr("builtins.open", counting_open)
    specs = blob_utils.get_file_upload_specs([(small, "small.bin", None), (grown, "grown.bin", None)], cache_small_content=True)
    monkeypatch.undo()
    assert specs[0].content == b"s" * 1000 and specs[0].sha256_hex == hashlib.sha256(b"s" * 1000).hexdigest()
    assert sum(1 for r in reads if r.endswith("small.bin")) == 1, "the cached file must be read exactly once"
    assert specs[1].size == 300_000 and specs[1].sha256_hex == hashlib.sha256(b"g" * 300_000).hexdigest()
    assert specs[1].md5_hex == hashlib.md5(b"g" * 300_000).hexdigest()


# ------------------------------------------------------------------------- async helpers of the upload path


def test_retry_counts_attempts_like_the_reference(monkeypatch):
    """Cases of py/test/async_utils_test.py:75-121: default 3 attempts, n_attempts=5, the bare-decorator form, the
    delay sequence base * factor^k capped at max_delay, the per-attempt timeout, RETRY_N_ATTEMPTS_OVERRIDE."""
    import asyncio

    from modal_client_b200 import async_utils
    from modal_client_b200.async_utils import retry

    class Boom(Exception):
        pass

    def fail_n_times(n):
        calls = {"n": 0}

        async def fn(x):
            calls["n"] += 1
            if calls["n"] <= n:
                raise Boom(calls["n"])
            return x + 1

        return fn

    async def run():
        assert await retry(fail_n_times(2))(42) == 43  # bare form, 3 attempts
        with pytest.raises(Boom):
            await retry(fail_n_times(3))(42)
        assert await retry(n_attempts=5)(fail_n_times(4))(42) == 43
        with pytest.raises(Boom):
            await retry(n_attempts=5)(fail_n_times(5))(42)

        delays = []
        real_sleep = asyncio.sleep

        async def fake_sleep(d):
            delays.append(d)
            await real_sleep(0)

        monkeypatch.setattr(async_utils.asyncio, "sleep", fake_sleep)
        try:
            fn = retry(n_attempts=5, base_delay=1, delay_factor=2, max_delay=2, attempt_timeout=None)(fail_n_times(4))
            assert await fn(0) == 1 and delays == [1, 2, 2, 2]
        finally:
            monkeypatch.setattr(async_utils.asyncio, "sleep", real_sleep)

        @retry(n_attempts=2, attempt_timeout=0.01)
        async def hangs():
            await asyncio.sleep(1)

        with pytest.raises(asyncio.TimeoutError):
            await hangs()

        @retry(n_attempts=3)
        async def cancelled():
            raise asyncio.CancelledError()

        with pytest.raises(asyncio.CancelledError):
            await cancelled()

        monkeypatch.setenv("RETRY_N_ATTEMPTS_OVERRIDE", "1")
        with pytest.raises(Boom):
            await retry(n_attempts=5)(fail_n_times(1))(0)

    asyncio.run(run())
