"""put_tensor / b200h_hash_device_parts without a GPU: the ABI surface, argument validation, and the volumefs1 / v2
request flow of tensors on an oracle-backed stand-in (host-backed readers), compared with put_file(BytesIO(same bytes))."""
import asyncio
import ctypes
import io
import os
import types

import numpy as np
import pytest
import torch
from aiohttp import web

from modal_client_b200 import _backend, _lib, blob_utils, volume
from modal_client_b200.synth import synth_bytes
from oracle import c_oracle
from tests.blob_server import running_blob_server
from tests.fake_backend import FakeContext
from tests.test_volume_upload import FakeVolumeStub, _add_block_route

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def oracle_parts(buffers, part_len, flags):
    """What b200h_hash_device_parts returns for these buffers (bytes), restated on the C oracle:
    (sha[rows,32]|None, md5[rows,16]|None, trimmed[rows], etags[n,16]|None) as raw rows."""
    shas, md5s, ends, etags = [], [], [], []
    for data in buffers:
        a = np.frombuffer(data, np.uint8)
        if part_len == 0:
            starts, lens = np.zeros(1, np.uint64), np.array([a.size], np.uint64)
        else:
            starts = np.arange(0, a.size, part_len, dtype=np.uint64)
            lens = np.minimum(part_len, a.size - starts).astype(np.uint64)
        s, m, e = c_oracle.hash_batch(a if a.size else np.zeros(1, np.uint8), starts, lens, sha=True, md5=True,
                                      trim=bool(flags & _lib.TRIM_ZEROS))
        shas.append(s)
        md5s.append(m)
        ends.append(e)
        etags.append(np.frombuffer(c_oracle.md5(m.tobytes()), np.uint8))
    sha = np.concatenate(shas) if shas else np.zeros((0, 32), np.uint8)
    md5 = np.concatenate(md5s) if md5s else np.zeros((0, 16), np.uint8)
    trimmed = np.concatenate(ends) if ends else np.zeros(0, np.uint64)
    return (sha if flags & _lib.SHA256 else None, md5 if flags & _lib.MD5 else None, trimmed,
            np.stack(etags) if etags else np.zeros((0, 16), np.uint8))


class FakeDeviceContext(FakeContext):
    """The stand-in with ``hash_device_parts`` over host memory: the readers of these tests wrap CPU tensors, whose
    data_ptr() is a host address."""

    def hash_device_parts(self, ptrs, sizes, part_len, flags=_lib.SHA256 | _lib.MD5, want_etag=False):
        self.calls.append(("hash_device_parts", len(ptrs), part_len, flags))
        bufs = [bytes((ctypes.c_uint8 * int(n)).from_address(int(p))) if n else b"" for p, n in zip(ptrs, sizes)]
        s, m, t, e = oracle_parts(bufs, part_len, flags)
        return s, m, t, (e if want_etag else None)


def test_device_parts_symbols_exported_and_declared():
    header = open(os.path.join(ROOT, "include", "b200hash.h")).read()
    L = _lib.load_library()
    for sym in ("b200h_hash_device_parts", "b200h_group_hash_device_parts"):
        assert sym in _lib.ABI_SYMBOLS and f"int {sym}(" in header and hasattr(L, sym)


def test_device_parts_rejects_null_handles_without_a_gpu():
    L = _lib.load_library()
    sizes = (ctypes.c_uint64 * 1)(16)
    bufs = (ctypes.c_void_p * 1)(None)
    out = (ctypes.c_uint8 * 64)()
    assert L.b200h_hash_device_parts(None, bufs, sizes, 1, 0, _lib.SHA256, out, None, None, None) == -1
    assert L.b200h_group_hash_device_parts(None, bufs, sizes, 1, 0, _lib.SHA256, out, None, None, None) == -1


def test_put_tensor_validates_at_call_time(fake_backend):
    batch = volume._BatchBase("vo", client=None)
    with pytest.raises(ValueError, match="CUDA tensor"):
        batch.put_tensor(torch.zeros(4), "/w.bin")
    with pytest.raises(ValueError, match="CUDA tensor"):
        batch.put_tensor(b"not a tensor", "/w.bin")
    with pytest.raises(ValueError) as put_file_err:
        batch.put_file(io.BytesIO(b"x"), "/")
    with pytest.raises(ValueError) as put_tensor_err:
        batch.put_tensor(torch.zeros(4), "/")
    assert str(put_tensor_err.value) == str(put_file_err.value)
    with pytest.raises(ValueError, match="contiguous CUDA tensor"):
        from modal_client_b200.function_utils import DevicePayload

        batch.put_tensor(DevicePayload(torch.zeros(4)), "/w.bin")
    assert batch._tensors == []


def test_context_devices_covers_contexts_and_groups():
    assert volume._context_devices(types.SimpleNamespace(device=3)) == [3]
    assert volume._context_devices(types.SimpleNamespace(devices=[0, 0, 1], device=0)) == [0, 0, 1]
    assert volume._context_devices(FakeContext()) is None  # the stand-in: any device


def test_host_backed_reader_reads_seeks_and_counts():
    t = torch.arange(1000, dtype=torch.int32)
    raw = t.numpy().tobytes()
    r = blob_utils.DeviceBufferReader(t)
    assert r.nbytes == len(raw) and r.seek(0, os.SEEK_END) == len(raw) and r.seek(10) == 10
    assert r.read(7) == raw[10:17] and r.tell() == 17
    c = r.clone()
    assert c.tell() == 0 and c.read() == raw
    with r.clone() as c2:
        c2.seek(len(raw) - 3)
        assert c2.read(100) == raw[-3:] and c2.read(5) == b""
    assert r.bytes_to_host == 7 + len(raw) + 3


def _tensors_and_bytes():
    out = []
    for i, (dtype, n) in enumerate([(torch.float32, 5000), (torch.uint8, 0), (torch.int16, 6000), (torch.uint8, 70_001),
                                    (torch.float64, 3)]):
        raw = bytearray(synth_bytes(40 + i, n * torch.empty(0, dtype=dtype).element_size()))
        if len(raw) > 3000:
            raw[-900:] = bytes(900)  # trailing zero run: trimmed blocks
        t = torch.frombuffer(bytearray(raw), dtype=torch.uint8).view(dtype) if raw else torch.empty(0, dtype=dtype)
        out.append((t, bytes(raw), f"/t/w{i}.bin"))
    return out


def test_v1_tensor_rows_equal_put_file_rows(monkeypatch):
    ctx = FakeDeviceContext()
    monkeypatch.setattr(_backend, "_override", ctx)
    monkeypatch.setattr(blob_utils, "LARGE_FILE_LIMIT", 20_000)  # the 70 001-byte tensor becomes a blob
    items = _tensors_and_bytes()

    async def upload(use_tensors):
        async with running_blob_server() as (host, store):
            stub = FakeVolumeStub(host, store, 8 << 20)
            sent = []
            orig = stub.VolumePutFiles

            async def record(req):
                sent.append(req)
                return await orig(req)

            stub.VolumePutFiles = record
            async with volume.VolumeUploadContextManager("vo-1", types.SimpleNamespace(stub=stub)) as batch:
                for t, raw, path in items:
                    if use_tensors:
                        batch._tensors.append((blob_utils.DeviceBufferReader(t), path, 0o600))
                    else:
                        batch.put_file(io.BytesIO(raw), path, mode=0o600)
            await blob_utils.ClientSessionRegistry.close_session()
            return sent[0].files, {k: v[0] for k, v in stub.volume_files.items()}, sorted(store.blobs.values())

    got_rows, got_files, got_blobs = asyncio.run(upload(True))
    want_rows, want_files, want_blobs = asyncio.run(upload(False))
    assert got_rows == want_rows and got_files == want_files and got_blobs == want_blobs
    assert got_files == {path: raw for _, raw, path in items}
    assert any(c[0] == "hash_device_parts" and c[2] == 0 for c in ctx.calls)


def test_v2_tensor_request_equals_put_file_request(monkeypatch):
    BS = 4096
    monkeypatch.setattr(blob_utils, "BLOCK_SIZE", BS)
    ctx = FakeDeviceContext()
    monkeypatch.setattr(_backend, "_override", ctx)
    items = _tensors_and_bytes()

    async def upload(use_tensors):
        async with running_blob_server() as (host, store):
            holder = {}
            stub = FakeVolumeStub(host, store, BS)
            holder["stub"] = stub
            app = web.Application(client_max_size=1 << 26)
            app.add_routes([web.put("/block/{token}", _add_block_route(store, holder, BS))])
            runner = web.AppRunner(app)
            await runner.setup()
            site = web.TCPSite(runner, "127.0.0.1", 0)
            await site.start()
            stub.host = f"http://127.0.0.1:{site._server.sockets[0].getsockname()[1]}"
            sent = []
            orig = stub.VolumePutFiles2

            async def record(req):
                sent.append(req)
                return await orig(req)

            stub.VolumePutFiles2 = record
            readers = []
            try:
                async with volume.VolumeUploadContextManager2("vo-2", types.SimpleNamespace(stub=stub)) as batch:
                    for t, raw, path in items:
                        if use_tensors:
                            readers.append(blob_utils.DeviceBufferReader(t))
                            batch._tensors.append((readers[-1], path, 0o640))
                        else:
                            batch.put_file(io.BytesIO(raw), path, mode=0o640)
            finally:
                await runner.cleanup()
                await blob_utils.ClientSessionRegistry.close_session()
            return sent, {k: v[0] for k, v in stub.volume_files.items()}, stub.blocks, readers

    got_reqs, got_files, got_blocks, readers = asyncio.run(upload(True))
    want_reqs, want_files, _, _ = asyncio.run(upload(False))
    assert [r.files for r in got_reqs] == [r.files for r in want_reqs]
    assert got_files == want_files == {path: raw for _, raw, path in items}
    # only the trimmed bytes of the blocks PUT crossed to the host
    assert sum(r.bytes_to_host for r in readers) == sum(len(b) for b in got_blocks.values())
    assert ("hash_device_parts", len(items), BS, _lib.SHA256 | _lib.TRIM_ZEROS) in ctx.calls
