"""put_tensor and b200h_hash_device_parts on the GPU: device parts bit for bit against the C oracle, the volumefs1 / v2
requests of put_tensor against those of put_file(BytesIO(same bytes)), only missing bytes crossing to the host, stream
ordering, and device groups (residency-aware deal)."""
import asyncio
import io
import types

import numpy as np
import pytest

from modal_client_b200 import _backend, _lib, batch, blob_utils, volume
from tests.blob_server import running_blob_server
from tests.test_volume_tensor_cpu import oracle_parts
from tests.test_volume_upload import FakeVolumeStub, _add_block_route

pytestmark = pytest.mark.gpu

MiB = 1 << 20
BLK = 8 * MiB
SIZES = [0, 1, 63, 64, BLK - 1, BLK, BLK + 1, 3 * BLK + 5, 2 * BLK + 100]


def _torch():
    import torch

    return torch


def _host_hex(t):
    return np.frombuffer(t.tobytes().hex().encode("ascii"), np.uint8).reshape(t.shape[0], 2 * t.shape[1])


@pytest.fixture(scope="module")
def slab():
    """One uint8 tensor; the buffers are slices of it at odd byte offsets, with trailing zero runs and blank blocks."""
    torch = _torch()
    g = torch.Generator(device="cuda").manual_seed(7)
    total = sum(SIZES) + 64 * len(SIZES) + 1
    t = torch.randint(0, 256, (total,), dtype=torch.uint8, device="cuda", generator=g)
    views, at = [], 1
    for i, n in enumerate(SIZES):
        v = t[at : at + n]
        if n > 4096 and i % 2:
            v[n - 3000 :] = 0  # trailing zeros
        if n == 3 * BLK + 5:
            v[BLK : 2 * BLK] = 0  # a fully blank block
        views.append(v)
        at += n + 64 + (i % 2)  # alternate odd / even starts
    torch.cuda.synchronize()
    return views, [v.cpu().numpy().tobytes() for v in views]


def _check(got, want, flags, etag_wanted):
    s, m, t, e = got
    ws, wm, wt, we = want
    hexed = bool(flags & _lib.HEX_OUT)
    if flags & _lib.SHA256:
        assert np.array_equal(s, _host_hex(ws) if hexed else ws)
    if flags & _lib.MD5:
        assert np.array_equal(m, _host_hex(wm) if hexed else wm)
    assert np.array_equal(t, wt)
    if etag_wanted:
        assert np.array_equal(e, we)


FLAG_SETS = [_lib.SHA256, _lib.SHA256 | _lib.TRIM_ZEROS, _lib.MD5, _lib.SHA256 | _lib.MD5,
             _lib.SHA256 | _lib.MD5 | _lib.HEX_OUT]


@pytest.mark.parametrize("flags", FLAG_SETS)
@pytest.mark.parametrize("part_len", [BLK, 0, 4096 + 3])
@pytest.mark.parametrize("outputs", ["host", "device"])
def test_device_parts_match_oracle(gpu_backend, slab, flags, part_len, outputs):
    torch = _torch()
    views, raw = slab
    if part_len == 0 and flags not in (_lib.SHA256 | _lib.MD5, _lib.SHA256 | _lib.TRIM_ZEROS):
        views, raw = views[:6], raw[:6]  # whole-buffer digests are serial chains: the long ones once per kind
    want_etag = bool(flags & _lib.MD5)
    want = oracle_parts(raw, part_len, flags)
    ptrs, sizes = [v.data_ptr() for v in views], [v.numel() for v in views]
    if outputs == "host":
        got = gpu_backend.hash_device_parts(ptrs, sizes, part_len, flags, want_etag)
    else:
        rows, wide = want[2].size, 2 if flags & _lib.HEX_OUT else 1
        d = {k: torch.zeros(max(rows * w, 1), dtype=torch.uint8, device="cuda")
             for k, w in (("sha", 32 * wide), ("md5", 16 * wide), ("trim", 8))}
        d["etag"] = torch.zeros(max(len(views) * 16, 1), dtype=torch.uint8, device="cuda")
        gpu_backend.hash_device_parts(ptrs, sizes, part_len, flags, want_etag, out_sha=d["sha"].data_ptr(),
                                      out_md5=d["md5"].data_ptr(), out_trimmed=d["trim"].data_ptr(),
                                      out_etag=d["etag"].data_ptr() if want_etag else 0)
        h = {k: v.cpu().numpy() for k, v in d.items()}
        got = (h["sha"][: rows * 32 * wide].reshape(rows, 32 * wide), h["md5"][: rows * 16 * wide].reshape(rows, 16 * wide),
               h["trim"][: rows * 8].view(np.uint64), h["etag"][: len(views) * 16].reshape(len(views), 16))
    _check(got, want, flags, want_etag)


def test_one_gib_buffer_blocks_and_etag(gpu_backend):
    torch = _torch()
    g = torch.Generator(device="cuda").manual_seed(11)
    t = torch.randint(0, 256, ((1 << 30) + 1,), dtype=torch.uint8, device="cuda", generator=g)
    v = t[1:]
    v[5 * BLK : 7 * BLK] = 0
    v[-123_457:] = 0
    raw = v.cpu().numpy().tobytes()
    for flags in (_lib.SHA256 | _lib.TRIM_ZEROS, _lib.MD5):
        got = gpu_backend.hash_device_parts([v.data_ptr()], [v.numel()], BLK, flags, bool(flags & _lib.MD5))
        _check(got, oracle_parts([raw], BLK, flags), flags, bool(flags & _lib.MD5))


def test_rejects_buffers_not_on_the_context_device(gpu_backend):
    host = np.zeros(4096, np.uint8)
    with pytest.raises(_lib.B200HashError, match="buffer 1 is host memory"):
        gpu_backend.hash_device_parts([0, host.ctypes.data], [0, host.size], 0, _lib.SHA256)
    one = _torch().ones(10, dtype=_torch().uint8, device="cuda")
    sha, _, _, _ = gpu_backend.hash_device_parts([one.data_ptr()], [10], 0, _lib.SHA256)  # still usable
    assert np.array_equal(sha, oracle_parts([bytes([1] * 10)], 0, _lib.SHA256)[0])


def test_work_queued_on_the_current_stream_is_hashed(gpu_backend):
    torch = _torch()
    src = torch.randint(0, 256, (256 * MiB,), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    want = oracle_parts([src.cpu().numpy().tobytes()], BLK, _lib.SHA256)[0]
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        t = torch.zeros_like(src)
        for _ in range(8):  # keep the stream busy so the copy lands late
            t.add_(1)
        t.copy_(src)
        table = batch.hash_blocks_tensors([t], BLK, sha256=True, ctx=gpu_backend)  # no synchronisation before
    assert np.array_equal(table.sha256, want)


# ---------------------------------------------------------------------------------------------- put_tensor


def _random_tensors():
    torch = _torch()
    g = torch.Generator(device="cuda").manual_seed(5)
    base = torch.randint(0, 256, (3 * MiB + 7,), dtype=torch.uint8, device="cuda", generator=g)
    f32 = torch.randn(300_000, device="cuda", generator=g)
    f32[-20_000:] = 0  # trailing zeros
    bf16 = torch.randn(250_000, device="cuda", generator=g).to(torch.bfloat16)
    i64 = torch.randint(-(2**40), 2**40, (200_001,), device="cuda", generator=g)
    rep = torch.cat([base[:64 * 1024]] * 6)  # repeated blocks
    return {"/w/f32.bin": f32, "/w/bf16.bin": bf16, "/w/i64.bin": i64, "/w/odd.bin": base[1:],
            "/w/odd_copy.bin": base[1:].clone(), "/w/rep.bin": rep, "/w/empty.bin": base[:0],
            "/w/big.bin": torch.randint(0, 256, (12 * MiB,), dtype=torch.uint8, device="cuda", generator=g)}


def _raw(t):
    return t.reshape(-1).view(_torch().uint8).cpu().numpy().tobytes()


def test_put_tensor_v2_equals_put_file(gpu_backend, monkeypatch):
    BS = 64 * 1024
    monkeypatch.setattr(blob_utils, "BLOCK_SIZE", BS)
    tensors = _random_tensors()

    async def upload(use_tensors):
        async with running_blob_server() as (host, store):
            holder = {}
            stub = FakeVolumeStub(host, store, BS)
            holder["stub"] = stub
            from aiohttp import web

            app = web.Application(client_max_size=1 << 26)
            app.add_routes([web.put("/block/{token}", _add_block_route(store, holder, BS))])
            runner = web.AppRunner(app)
            await runner.setup()
            site = web.TCPSite(runner, "127.0.0.1", 0)
            await site.start()
            stub.host = f"http://127.0.0.1:{site._server.sockets[0].getsockname()[1]}"
            sent, orig = [], stub.VolumePutFiles2

            async def record(req):
                sent.append(req)
                return await orig(req)

            stub.VolumePutFiles2 = record
            try:
                async with volume.VolumeUploadContextManager2("vo-2", types.SimpleNamespace(stub=stub)) as b:
                    for path, t in tensors.items():
                        if use_tensors:
                            b.put_tensor(t, path)
                        else:
                            b.put_file(io.BytesIO(_raw(t)), path, mode=0o644)
                    readers = [r for r, _, _ in b._tensors]
            finally:
                await runner.cleanup()
                await blob_utils.ClientSessionRegistry.close_session()
            return sent, stub, readers

    got, stub, readers = asyncio.run(upload(True))
    want, _, _ = asyncio.run(upload(False))
    assert [r.files for r in got] == [r.files for r in want]
    assert {k: v[0] for k, v in stub.volume_files.items()} == {p: _raw(t) for p, t in tensors.items()}
    assert stub.block_puts == len(stub.blocks)  # equal tensors and repeated blocks were PUT once
    assert sum(r.bytes_to_host for r in readers) == sum(len(b) for b in stub.blocks.values())


def test_put_tensor_v1_equals_put_file(gpu_backend, monkeypatch):
    monkeypatch.setattr(blob_utils, "LARGE_FILE_LIMIT", 1 * MiB)  # most tensors become blobs; big.bin goes multipart
    tensors = _random_tensors()

    async def upload(use_tensors):
        async with running_blob_server() as (host, store):
            stub = FakeVolumeStub(host, store, 8 * MiB)
            sent, orig = [], stub.VolumePutFiles

            async def record(req):
                sent.append(req)
                return await orig(req)

            stub.VolumePutFiles = record
            async with volume.VolumeUploadContextManager("vo-1", types.SimpleNamespace(stub=stub)) as b:
                for path, t in tensors.items():
                    if use_tensors:
                        b.put_tensor(t, path, mode=0o600)
                    else:
                        b.put_file(io.BytesIO(_raw(t)), path, mode=0o600)
            await blob_utils.ClientSessionRegistry.close_session()
            creates = sorted((r.content_md5, r.content_sha256_base64, r.content_length) for r in stub.requests)
            return sent[0].files, {k: v[0] for k, v in stub.volume_files.items()}, creates, sorted(store.blobs.values())

    got = asyncio.run(upload(True))
    want = asyncio.run(upload(False))
    assert got == want  # MountFile rows, contents, BlobCreate digests, blob bytes (the multipart ETag is checked on completion)
    assert got[1] == {p: _raw(t) for p, t in tensors.items()}
    assert any(length > 8 * MiB for _, _, length in got[2])  # the multipart path ran


def test_put_tensor_rejects_cpu_and_uncovered_tensors(gpu_backend):
    torch = _torch()
    b = volume._BatchBase("vo", client=None)
    with pytest.raises(ValueError, match="CUDA tensor"):
        b.put_tensor(torch.zeros(3), "/x")
    with pytest.raises(ValueError, match="contiguous"):
        b.put_tensor(torch.zeros(4, 4, device="cuda").t(), "/x")
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError, match="cuda:1"):
            b.put_tensor(torch.zeros(3, device="cuda:1"), "/x")


# --------------------------------------------------------------------------------------------------- groups


@pytest.fixture(scope="module", params=["0,0", "every device"])
def group(request):
    torch = _torch()
    if request.param == "every device":
        if torch.cuda.device_count() < 2:
            pytest.skip(f"a group over distinct GPUs needs 2 or more; this box has {torch.cuda.device_count()}")
        devices = list(range(torch.cuda.device_count()))
    else:
        devices = [0, 0]
    g = _lib.DeviceGroup(devices, pinned_bytes=64 * MiB, device_bytes=512 * MiB, min_share_bytes=1)
    yield g
    g.close()


@pytest.mark.parametrize("flags", [_lib.SHA256 | _lib.TRIM_ZEROS, _lib.SHA256 | _lib.MD5,
                                   _lib.SHA256 | _lib.MD5 | _lib.HEX_OUT])
def test_group_device_parts_equal_rows(group, slab, flags):
    torch = _torch()
    views, raw = slab
    # every device of the group holds a copy of the slab's buffers
    bufs, data = [], []
    for d in sorted(set(group.devices)):
        bufs += [v.to(f"cuda:{d}") for v in views]
        data += raw
    torch.cuda.synchronize()
    want_etag = bool(flags & _lib.MD5)
    got = group.hash_device_parts([b.data_ptr() for b in bufs], [b.numel() for b in bufs], BLK, flags, want_etag)
    _check(got, oracle_parts(data, BLK, flags), flags, want_etag)
    split = group.last_split()
    assert sum(s["messages"] for s in split) == got[2].size
    assert sum(s["bytes"] for s in split) == sum(b.numel() for b in bufs)
    assert sum(1 for s in split if s["messages"]) >= 2
    for s in split:  # every member only hashed bytes on its own device
        if s["messages"]:
            assert s["bytes"] <= sum(b.numel() for b in bufs if b.device.index == s["device"])


def test_group_rejects_foreign_buffers_and_stays_usable(group):
    torch = _torch()
    host = np.ones(100, np.uint8)
    with pytest.raises(_lib.B200HashError, match="buffer 0 is host memory"):
        group.hash_device_parts([host.ctypes.data], [100], 0, _lib.SHA256)
    t = torch.ones(100, dtype=torch.uint8, device="cuda")
    sha, _, _, _ = group.hash_device_parts([t.data_ptr()], [100], 0, _lib.SHA256)
    assert np.array_equal(sha, oracle_parts([bytes([1] * 100)], 0, _lib.SHA256)[0])


def test_put_tensor_on_an_uncovered_device(monkeypatch):
    torch = _torch()
    if torch.cuda.device_count() < 2:
        pytest.skip("needs a second GPU outside the group")
    g = _lib.DeviceGroup([0, 0], pinned_bytes=64 * MiB, device_bytes=512 * MiB, min_share_bytes=1)
    try:
        monkeypatch.setattr(_backend, "_override", g)
        b = volume._BatchBase("vo", client=None)
        with pytest.raises(ValueError, match="cuda:1"):
            b.put_tensor(torch.zeros(8, device="cuda:1"), "/x")
        t1 = torch.ones(64, dtype=torch.uint8, device="cuda:1")
        with pytest.raises(_lib.B200HashError, match="buffer 0 is on cuda:1, which is not in the group"):
            g.hash_device_parts([t1.data_ptr()], [64], 0, _lib.SHA256)
        t0 = torch.ones(64, dtype=torch.uint8, device="cuda:0")
        sha, _, _, _ = g.hash_device_parts([t0.data_ptr()], [64], 0, _lib.SHA256)
        assert np.array_equal(sha, oracle_parts([bytes([1] * 64)], 0, _lib.SHA256)[0])
    finally:
        g.close()
