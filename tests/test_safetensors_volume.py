"""put_safetensors and b200h_hash_device_segments on the GPU: rows bit for bit against the C oracle over the
concatenated bytes and against hash_device_parts over a torch.cat of the segments, windows, the volumefs1 / v2
requests of put_safetensors against those of put_file(BytesIO(the same file bytes)), only changed blocks PUT on a
re-save, stream ordering, and device groups."""
import asyncio
import io
import types

import numpy as np
import pytest

from modal_client_b200 import _backend, _lib, batch, blob_utils, volume
from tests.blob_server import running_blob_server
from tests.test_volume_tensor import FLAG_SETS, _check, _host_hex  # noqa: F401  (shared helpers)
from tests.test_volume_tensor_cpu import oracle_parts
from tests.test_volume_upload import FakeVolumeStub, _add_block_route

pytestmark = pytest.mark.gpu

MiB = 1 << 20
BLK = 8 * MiB

# segment sizes of the files of one call (a file = its list); chosen to hit every row kind
LAYOUTS = {
    "safetensors_like": [[136, 20 * MiB + 3, 5, 0, 1, 9 * MiB] + [4] * 700 + [3 * MiB + 17], [0, 0], []],
    "thousands_in_one_part": [[4] * 3000 + [BLK], [BLK - 2, 1, 1, 2, BLK]],
    "on_part_boundaries": [[BLK, BLK, 0, BLK], [4099, 4099, 4099 * 3]],
    "trailing_zeros_across_segments": [[5 * MiB, 2 * MiB, 4 * MiB, 3], [1000, 3]],
}
ZERO_TAILS = {"trailing_zeros_across_segments"}  # every segment after the first of a file is all zeros


def _torch():
    import torch

    return torch


@pytest.fixture(scope="module")
def layouts():
    """name -> (files as lists of CUDA uint8 views at odd and even addresses, the concatenated bytes of each file)."""
    torch = _torch()
    g = torch.Generator(device="cuda").manual_seed(3)
    out = {}
    for name, files in LAYOUTS.items():
        total = sum(sum(f) + 17 * len(f) + 1 for f in files) + 1
        slab = torch.randint(0, 256, (total,), dtype=torch.uint8, device="cuda", generator=g)
        views, at = [], 1
        for f in files:
            vs = []
            for k, n in enumerate(f):
                v = slab[at : at + n]
                if name in ZERO_TAILS and k:
                    v.zero_()
                vs.append(v)
                at += n + 1 + (k % 16)  # every alignment of source against destination
            views.append(vs)
        torch.cuda.synchronize()
        out[name] = (views, [b"".join(v.cpu().numpy().tobytes() for v in vs) for vs in views])
    return out


def _segs(views):
    return [[(v.data_ptr(), v.numel()) for v in vs] for vs in views]


@pytest.mark.parametrize("name", list(LAYOUTS))
@pytest.mark.parametrize("flags", FLAG_SETS)
@pytest.mark.parametrize("part_len", [BLK, 0, 4096 + 3])
@pytest.mark.parametrize("outputs", ["host", "device"])
def test_device_segments_match_oracle(gpu_backend, layouts, name, flags, part_len, outputs):
    torch = _torch()
    if part_len == 0 and outputs == "device" and flags != FLAG_SETS[-1]:
        pytest.skip("whole-file digests are serial chains: device outputs once, with every column")
    views, raw = layouts[name]
    want_etag = bool(flags & _lib.MD5)
    want = oracle_parts(raw, part_len, flags)
    if outputs == "host":
        got = gpu_backend.hash_device_segments(_segs(views), part_len, flags, want_etag)
    else:
        rows, wide = want[2].size, 2 if flags & _lib.HEX_OUT else 1
        d = {k: torch.zeros(max(rows * w, 1), dtype=torch.uint8, device="cuda")
             for k, w in (("sha", 32 * wide), ("md5", 16 * wide), ("trim", 8))}
        d["etag"] = torch.zeros(max(len(views) * 16, 1), dtype=torch.uint8, device="cuda")
        gpu_backend.hash_device_segments(_segs(views), part_len, flags, want_etag, out_sha=d["sha"].data_ptr(),
                                         out_md5=d["md5"].data_ptr(), out_trimmed=d["trim"].data_ptr(),
                                         out_etag=d["etag"].data_ptr() if want_etag else 0)
        h = {k: v.cpu().numpy() for k, v in d.items()}
        got = (h["sha"][: rows * 32 * wide].reshape(rows, 32 * wide), h["md5"][: rows * 16 * wide].reshape(rows, 16 * wide),
               h["trim"][: rows * 8].view(np.uint64), h["etag"][: len(views) * 16].reshape(len(views), 16))
    _check(got, want, flags, want_etag)


def test_trailing_zeros_across_segments_are_trimmed_like_the_file(gpu_backend, layouts):
    views, raw = layouts["trailing_zeros_across_segments"]
    _, _, trimmed, _ = gpu_backend.hash_device_segments(_segs(views), BLK, _lib.SHA256 | _lib.TRIM_ZEROS)
    first = len(raw[0].rstrip(b"\0"))
    assert trimmed[0] == first and first < 5 * MiB + 1 and trimmed[1] == 0  # block 1 is blank: trimmed to nothing


@pytest.mark.parametrize("name", list(LAYOUTS))
def test_device_segments_equal_device_parts_of_the_concatenation(gpu_backend, layouts, name):
    torch = _torch()
    views, _ = layouts[name]
    cats = [torch.cat(vs) if vs else torch.empty(0, dtype=torch.uint8, device="cuda") for vs in views]
    flags = _lib.SHA256 | _lib.MD5 | _lib.TRIM_ZEROS
    a = gpu_backend.hash_device_segments(_segs(views), BLK, flags, True)
    b = gpu_backend.hash_device_parts([c.data_ptr() for c in cats], [c.numel() for c in cats], BLK, flags, True)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("cap", ["1", "65536", str(9 * MiB)])
def test_windows_give_the_same_rows(gpu_backend, layouts, monkeypatch, cap):
    views, raw = layouts["safetensors_like"]
    flags = _lib.SHA256 | _lib.MD5 | _lib.TRIM_ZEROS
    want = gpu_backend.hash_device_segments(_segs(views), BLK, flags, True)
    monkeypatch.setenv("B200H_GATHER_BYTES", cap)
    sizes = [[n for _, n in f] for f in _segs(views)]
    seg_of = np.cumsum([0] + [len(f) for f in sizes])
    assert _lib.segments_preview([n for f in sizes for n in f], seg_of, BLK)["window_bytes"].size >= (2 if cap != str(9 * MiB) else 1)
    got = gpu_backend.hash_device_segments(_segs(views), BLK, flags, True)
    for x, y in zip(got, want):
        assert np.array_equal(x, y)
    _check(got, oracle_parts(raw, BLK, flags), flags, True)


def test_rejects_segments_not_on_the_context_device(gpu_backend):
    torch = _torch()
    host = np.zeros(4096, np.uint8)
    t = torch.ones(100, dtype=torch.uint8, device="cuda")
    with pytest.raises(_lib.B200HashError, match="file 1 segment 2 is host memory"):
        gpu_backend.hash_device_segments([[(t.data_ptr(), 100)], [(t.data_ptr(), 100), (host.ctypes.data, host.size)]],
                                         0, _lib.SHA256)
    sha, _, _, _ = gpu_backend.hash_device_segments([[(t.data_ptr(), 50), (t.data_ptr() + 50, 50)]], 0, _lib.SHA256)
    assert np.array_equal(sha, oracle_parts([bytes([1] * 100)], 0, _lib.SHA256)[0])  # still usable


def test_work_queued_on_a_side_stream_is_hashed(gpu_backend):
    torch = _torch()
    src = torch.randint(0, 256, (96 * MiB,), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    want = oracle_parts([src.cpu().numpy().tobytes()], BLK, _lib.SHA256)[0]
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        t = torch.zeros_like(src)
        for _ in range(8):  # keep the stream busy so the copy lands late
            t.add_(1)
        t.copy_(src)
        parts = [t[: 3 * MiB + 1], t[3 * MiB + 1 : 50 * MiB], t[50 * MiB :]]
        table = batch.hash_blocks_segments([parts], BLK, sha256=True, ctx=gpu_backend)  # no synchronisation before
    assert np.array_equal(table.sha256, want)


# ------------------------------------------------------------------------------------------- put_safetensors


def _state_dict(seed=5):
    torch = _torch()
    g = torch.Generator(device="cuda").manual_seed(seed)
    sd = {}
    for i in range(6):
        sd[f"model.layers.{i}.mlp.weight"] = torch.randn(1024, 1536 + i, device="cuda", generator=g).to(torch.bfloat16)
        sd[f"model.layers.{i}.norm.weight"] = torch.randn(1024, device="cuda", generator=g)
        sd[f"model.layers.{i}.scale"] = torch.randn((), device="cuda", generator=g)
    sd["embed.weight"] = torch.randn(4000, 1000, device="cuda", generator=g)
    sd["embed.weight"][-500:] = 0  # a zero run that crosses into the next tensor's blocks
    sd["head.bias"] = torch.zeros(7, dtype=torch.float16, device="cuda")
    sd["mask"] = torch.ones(33, dtype=torch.bool, device="cuda")
    sd["empty"] = torch.empty(0, 4, device="cuda")
    torch.cuda.synchronize()
    return sd


def _file(sd, md=None):
    torch = _torch()
    header, ordered = blob_utils.safetensors_layout(sd, md)
    return header + b"".join(t.reshape(-1).view(torch.uint8).cpu().numpy().tobytes() for _, t in ordered)


async def _upload_v2(files, use_segments, BS):
    from aiohttp import web

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
        sent, orig = [], stub.VolumePutFiles2

        async def record(req):
            sent.append(req)
            return await orig(req)

        stub.VolumePutFiles2 = record
        try:
            async with volume.VolumeUploadContextManager2("vo-2", types.SimpleNamespace(stub=stub)) as b:
                for path, (sd, md) in files.items():
                    if use_segments:
                        b.put_safetensors(sd, path, metadata=md)
                    else:
                        b.put_file(io.BytesIO(_file(sd, md)), path, mode=0o644)
                readers = [r for r, _, _ in b._safetensors]
        finally:
            await runner.cleanup()
            await blob_utils.ClientSessionRegistry.close_session()
        return sent, stub, readers


def test_put_safetensors_v2_equals_put_file(gpu_backend, monkeypatch):
    BS = 1 * MiB
    monkeypatch.setattr(blob_utils, "BLOCK_SIZE", BS)
    files = {"/ckpt/a.safetensors": (_state_dict(5), {"format": "pt"}), "/ckpt/b.safetensors": (_state_dict(6), None)}
    got, stub, readers = asyncio.run(_upload_v2(files, True, BS))
    want, _, _ = asyncio.run(_upload_v2(files, False, BS))
    assert [r.files for r in got] == [r.files for r in want]
    contents = {k: v[0] for k, v in stub.volume_files.items()}
    assert contents == {p: _file(sd, md) for p, (sd, md) in files.items()}
    assert sum(r.bytes_to_host for r in readers) == sum(len(b) for b in stub.blocks.values())
    st = pytest.importorskip("safetensors.torch")
    back = st.load(contents["/ckpt/a.safetensors"])
    sd = files["/ckpt/a.safetensors"][0]
    assert set(back) == set(sd) and all(torch_equal(back[k], sd[k]) for k in sd)


def torch_equal(host, dev):
    return _torch().equal(host, dev.cpu())


def test_resave_with_one_tensor_changed_changes_only_its_blocks(gpu_backend, monkeypatch):
    # A volumefs2 server asks only for blocks whose SHA-256 it lacks: after a first save, a re-save sends exactly the
    # blocks whose digests changed, which must be the blocks that overlap the changed tensor.
    BS = 1 * MiB
    monkeypatch.setattr(blob_utils, "BLOCK_SIZE", BS)
    sd = _state_dict(7)
    first, _, _ = asyncio.run(_upload_v2({"/m.safetensors": (sd, None)}, True, BS))
    name = "model.layers.3.mlp.weight"
    sd[name][100:200] += 1
    header, ordered = blob_utils.safetensors_layout(sd)
    names = [n for n, _ in ordered]
    begin = len(header) + sum(t.numel() * t.element_size() for _, t in ordered[: names.index(name)])
    end = begin + sd[name].numel() * sd[name].element_size()
    second, stub, _ = asyncio.run(_upload_v2({"/m.safetensors": (sd, None)}, True, BS))
    a, b = first[0].files[0].blocks, second[0].files[0].blocks
    changed = {i for i, (x, y) in enumerate(zip(a, b)) if x.contents_sha256 != y.contents_sha256}
    overlapping = {i for i in range(len(b)) if i * BS < end and begin < (i + 1) * BS}
    assert len(a) == len(b) and changed and changed <= overlapping
    assert {k: v[0] for k, v in stub.volume_files.items()} == {"/m.safetensors": _file(sd)}


def test_put_safetensors_v1_equals_put_file(gpu_backend, monkeypatch):
    monkeypatch.setattr(blob_utils, "LARGE_FILE_LIMIT", 1 * MiB)  # blobs; the 40 MB file goes multipart
    small = {k: v for k, v in _state_dict(8).items() if "embed" not in k}
    files = {"/v1/a.safetensors": (_state_dict(5), {"format": "pt"}), "/v1/small.safetensors": (small, None)}

    async def upload(use_segments):
        async with running_blob_server() as (host, store):
            stub = FakeVolumeStub(host, store, 8 * MiB)
            sent, orig = [], stub.VolumePutFiles

            async def record(req):
                sent.append(req)
                return await orig(req)

            stub.VolumePutFiles = record
            async with volume.VolumeUploadContextManager("vo-1", types.SimpleNamespace(stub=stub)) as b:
                for path, (sd, md) in files.items():
                    if use_segments:
                        b.put_safetensors(sd, path, metadata=md, mode=0o600)
                    else:
                        b.put_file(io.BytesIO(_file(sd, md)), path, mode=0o600)
            await blob_utils.ClientSessionRegistry.close_session()
            creates = sorted((r.content_md5, r.content_sha256_base64, r.content_length) for r in stub.requests)
            return sent[0].files, {k: v[0] for k, v in stub.volume_files.items()}, creates, sorted(store.blobs.values())

    got = asyncio.run(upload(True))
    want = asyncio.run(upload(False))
    assert got == want
    assert got[1] == {p: _file(sd, md) for p, (sd, md) in files.items()}
    assert any(length > 8 * MiB for _, _, length in got[2])  # the multipart path ran


def test_put_safetensors_rejects_bad_tensors(gpu_backend):
    torch = _torch()
    b = volume._BatchBase("vo", client=None)
    with pytest.raises(ValueError, match="'w' is not contiguous"):
        b.put_safetensors({"w": torch.zeros(4, 4, device="cuda").t()}, "/x")
    base = torch.zeros(8, device="cuda")
    with pytest.raises(ValueError, match="share storage"):
        b.put_safetensors({"a": base[:4], "b": base[4:]}, "/x")
    with pytest.raises(ValueError, match="'c' has dtype torch.complex128"):
        b.put_safetensors({"c": torch.zeros(2, dtype=torch.complex128, device="cuda")}, "/x")
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError, match="one device"):
            b.put_safetensors({"a": torch.zeros(2, device="cuda:0"), "b": torch.zeros(2, device="cuda:1")}, "/x")
    assert b._safetensors == []


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
def test_group_device_segments_equal_rows(group, layouts, flags):
    torch = _torch()
    views, raw = layouts["safetensors_like"]
    files, data = [], []
    for d in sorted(set(group.devices)):  # every device of the group holds a copy of the files
        files += [[v.to(f"cuda:{d}") for v in vs] for vs in views]
        data += raw
    torch.cuda.synchronize()
    want_etag = bool(flags & _lib.MD5)
    got = group.hash_device_segments(_segs(files), BLK, flags, want_etag)
    _check(got, oracle_parts(data, BLK, flags), flags, want_etag)
    split = group.last_split()
    assert sum(s["messages"] for s in split) == got[2].size
    assert sum(s["bytes"] for s in split) == sum(len(r) for r in data)
    assert sum(1 for s in split if s["messages"]) >= 2


def test_group_rejects_a_file_on_two_devices_and_stays_usable(group):
    torch = _torch()
    host = np.ones(100, np.uint8)
    t = torch.ones(100, dtype=torch.uint8, device="cuda")
    with pytest.raises(_lib.B200HashError, match="file 0 segment 1 is host memory"):
        group.hash_device_segments([[(t.data_ptr(), 100), (host.ctypes.data, 100)]], 0, _lib.SHA256)
    if torch.cuda.device_count() > 1:
        t1 = torch.ones(100, dtype=torch.uint8, device="cuda:1")
        with pytest.raises(_lib.B200HashError, match="file 2 has segments on cuda:0 and cuda:1"):
            group.hash_device_segments([[], [], [(t.data_ptr(), 100), (t1.data_ptr(), 100)]], 0, _lib.SHA256)
    sha, _, _, _ = group.hash_device_segments([[(t.data_ptr(), 60), (t.data_ptr() + 60, 40)]], 0, _lib.SHA256)
    assert np.array_equal(sha, oracle_parts([bytes([1] * 100)], 0, _lib.SHA256)[0])
