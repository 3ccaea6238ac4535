"""The drop-in seam from the reference's side: what the reference's UNMODIFIED blob_utils.py (spec builder, volumefs2
block gatherer, multipart upload) asked of hash_utils / _hash_range_sha256 / BytesIOSegmentPayload, and what its own
hashlib-backed versions answered, was recorded by oracle/gen_golden.py (tests/golden/seam.json, file_specs.json,
blocks.json).  Each test replays those calls on modal_client_b200 and must get the reference's answers."""
import asyncio
import hashlib
import io
from contextlib import contextmanager

import aiohttp
import pytest

from modal_client_b200 import hash_utils as our_hash_utils
from modal_client_b200.synth import materialize


@pytest.fixture(params=["fake", pytest.param("gpu", marks=pytest.mark.gpu)])
def backend(request):
    return request.getfixturevalue("fake_backend" if request.param == "fake" else "gpu_backend")


@pytest.fixture
def seam(backend, golden):
    return golden("seam.json")


def test_reference_spec_builder_on_our_hashes_reproduces_its_golden(seam, golden):
    cases = golden("file_specs.json")["cases"]
    assert len(seam["spec_builder_calls"]) == len(cases)
    for c, calls in zip(cases, seam["spec_builder_calls"]):
        data = materialize(c["input"])
        assert len(calls) == 1
        for call in calls:
            if call["stream"]:
                arg = io.BytesIO(data)
                arg.seek(call["pos"])
            else:
                arg = data
            up = our_hash_utils.get_upload_hashes(arg, **call["kwargs"])
            assert (up.sha256_hex(), up.md5_hex()) == (call["sha256_hex"], call["md5_hex"])
            if call["stream"]:
                assert arg.tell() == call["pos_after"]
        # the spec the reference built carries the digests of its last call
        assert (calls[-1]["sha256_hex"], calls[-1]["md5_hex"]) == (c["sha256_hex"], c["md5_hex"])


def test_reference_block_gatherer_on_our_hashes_reproduces_its_golden(seam, monkeypatch, backend, golden):
    # _hash_range_sha256 uses hashlib directly in the reference (blob_utils.py:648): the seam for volumefs2 is that
    # function, called by the reference's _gather_block on every range its _find_end_of_block chose
    from modal_client_b200 import blob_utils as ours

    for c in golden("blocks.json")["spec2"]:
        data = materialize(c["input"])
        if len(data) > 20_000_000 and backend.device < 0:
            continue  # the oracle-backed stand-in is slow; the GPU variant runs every case

        @contextmanager
        def source(data=data):
            yield io.BytesIO(data)

        with monkeypatch.context() as mp:
            for name, value in c["patch"].items():
                mp.setattr(ours, name, value)
            block = ours.BLOCK_SIZE
            for i, (start, end, sha) in enumerate(c["blocks"]):
                assert start == i * block and start <= end <= min(start + block, len(data))
                assert ours._hash_range_sha256(source, start, end).hex() == sha


def test_reference_multipart_upload_on_our_segment_payload(seam):
    """Second seam: the segment payloads the reference's perform_multipart_upload (blob_utils.py:159-234) builds, as our
    BytesIOSegmentPayload (per-part MD5 from the hash path), PUT through aiohttp to the fake blob server.  Like the
    reference's _upload_to_s3_url, every part's ETag is checked against `payload.md5_checksum().hexdigest()`, the
    assembled md5-of-md5s ETag against the server's, and a corrupted ETag must not match."""
    from modal_client_b200 import bytes_io_segment_payload as our_payload
    from tests.blob_server import running_blob_server

    mp = seam["multipart"]
    data = materialize(mp["input"])
    parts = mp["payloads"]
    assert len(parts) == 11 and sum(p["segment_length"] for p in parts) == len(data)

    async def put(session, url, rec):
        reader = io.BytesIO(data)
        reader.seek(rec["initial_pos"])
        payload = our_payload.BytesIOSegmentPayload(reader, rec["segment_start"], rec["segment_length"], rec["chunk_size"])
        with payload.reset_on_error():
            async with session.put(url, data=payload, skip_auto_headers=["content-type"]) as resp:
                assert resp.status == 200
                return resp.headers["ETag"].strip('"'), payload.md5_checksum().hexdigest()

    async def run():
        async with running_blob_server() as (host, store), aiohttp.ClientSession() as session:
            for i, rec in enumerate(parts):
                etag, local = await put(session, f"{host}/upload?blob_id=bl-x&part_number={i + 1}", rec)
                assert etag == local == rec["md5_hex"]
                assert hashlib.sha256(store.parts["bl-x"][i + 1]).hexdigest() == rec["sent_sha256"]
            async with session.post(f"{host}/complete_multipart?blob_id=bl-x") as resp:
                body = await resp.text()
            joined = b"".join(bytes.fromhex(rec["md5_hex"]) for rec in parts)
            assert f"{hashlib.md5(joined).hexdigest()}-{len(parts)}" in body
            assert store.blobs["bl-x"] == data
            # a corrupted ETag from the server is what the reference's check against our MD5 catches
            store.corrupt_etag = True
            etag, local = await put(session, f"{host}/upload?blob_id=bl-y&part_number=1", parts[0])
            assert etag != local

    asyncio.run(run())
