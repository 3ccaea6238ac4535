"""put_safetensors / b200h_hash_device_segments without a GPU: the ABI surface, the row and piece table against a plain
Python restatement, the safetensors framing against the golden (and the installed package where there is one),
argument validation, the segments reader over CPU tensors, and the volumefs1 / v2 request flow on an oracle-backed
stand-in compared with put_file(BytesIO(the same file bytes))."""
import asyncio
import ctypes
import hashlib
import io
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch
from aiohttp import web

from modal_client_b200 import _backend, _lib, blob_utils, volume
from oracle.gen_safetensors_golden import state_dict_from_recipe
from tests.blob_server import running_blob_server
from tests.test_volume_tensor_cpu import FakeDeviceContext, oracle_parts
from tests.test_volume_upload import FakeVolumeStub, _add_block_route

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = json.load(open(os.path.join(ROOT, "tests", "golden", "safetensors.json")))
MiB = 1 << 20


def file_bytes(tensors, metadata=None) -> bytes:
    header, ordered = blob_utils.safetensors_layout(tensors, metadata)
    return header + b"".join(t.reshape(-1).view(torch.uint8).numpy().tobytes() for _, t in ordered)


class FakeSegmentsContext(FakeDeviceContext):
    """The stand-in with ``hash_device_segments`` over host memory: the files are concatenated and hashed by the C
    oracle, which is what the GPU rows must equal."""

    def hash_device_segments(self, files, part_len, flags=_lib.SHA256 | _lib.MD5, want_etag=False):
        self.calls.append(("hash_device_segments", len(files), part_len, flags))
        bufs = [b"".join(bytes((ctypes.c_uint8 * int(n)).from_address(int(p))) for p, n in f if n) for f in files]
        s, m, t, e = oracle_parts(bufs, part_len, flags)
        return s, m, t, (e if want_etag else None)


# ---- ABI -------------------------------------------------------------------------------------------------------


def test_segments_symbols_exported_and_declared():
    header = open(os.path.join(ROOT, "include", "b200hash.h")).read()
    L = _lib.load_library()
    for sym in ("b200h_hash_device_segments", "b200h_group_hash_device_segments", "b200h_segments_preview"):
        assert sym in _lib.ABI_SYMBOLS and f"int {sym}(" in header and hasattr(L, sym)


def test_segments_reject_null_handles_without_a_gpu():
    L = _lib.load_library()
    sizes = (ctypes.c_uint64 * 1)(16)
    seg_of = (ctypes.c_uint64 * 2)(0, 1)
    segs = (ctypes.c_void_p * 1)(None)
    out = (ctypes.c_uint8 * 64)()
    assert L.b200h_hash_device_segments(None, segs, sizes, seg_of, 1, 0, _lib.SHA256, out, None, None, None) == -1
    assert L.b200h_group_hash_device_segments(None, segs, sizes, seg_of, 1, 0, _lib.SHA256, out, None, None, None) == -1
    bad_of = (ctypes.c_uint64 * 2)(1, 0)  # decreasing
    n = ctypes.c_uint64()
    assert L.b200h_segments_preview(sizes, bad_of, 1, 0, 0, ctypes.byref(n), None, None, None, None, None) == -1


# ---- the row / piece table -----------------------------------------------------------------------------------


def restated_preview(seg_sizes, seg_of, part_len, window_bytes):
    """Plain-Python restatement of b200h_segments_preview (include/b200hash.h)."""
    rows = []  # (gathered, a, b, len)
    for i in range(len(seg_of) - 1):
        segs = list(range(seg_of[i], seg_of[i + 1]))
        starts, at = {}, 0
        for s in segs:
            starts[s] = at
            at += seg_sizes[s]
        size = at
        parts = [(0, size)] if part_len == 0 else [(o, min(part_len, size - o)) for o in range(0, size, part_len)]
        for off, ln in parts:
            if ln == 0:
                rows.append([False, seg_of[i], 0, 0])
                continue
            touched = [s for s in segs if seg_sizes[s] and starts[s] < off + ln and off < starts[s] + seg_sizes[s]]
            if len(touched) == 1:
                rows.append([False, touched[0], off - starts[touched[0]], ln])
            else:
                rows.append([True, None, len(touched), ln])
    windows, cur, any_ = [0], 0, False
    for r in rows:
        if not r[0]:
            continue
        p = (r[3] + 15) // 16 * 16
        if any_ and windows[-1] + p > window_bytes:
            windows.append(0)
        windows[-1] += p
        r[1] = len(windows) - 1
        any_ = True
    return rows, windows


def random_layouts(rng):
    yield [], [0]
    yield [0, 0], [0, 1, 2]
    yield [1, 0, 1, 1], [0, 4]
    yield [64, 64, 0, 64], [0, 2, 4]  # boundaries exactly on part boundaries
    yield [4] * 5000 + [3 * MiB], [0, 5001]  # thousands of segments inside one part
    yield [5 * MiB, 3 * MiB, 8 * MiB, 1], [0, 1, 2, 4]
    for _ in range(40):
        n_files = int(rng.integers(1, 5))
        counts = rng.integers(0, 12, n_files)
        sizes = []
        for _ in range(int(counts.sum())):
            kind = rng.integers(0, 5)
            sizes.append(int([0, 1, rng.integers(2, 200), rng.integers(200, 3 * MiB), 64 * rng.integers(1, 4)][kind]))
        yield sizes, [0] + np.cumsum(counts).tolist()


@pytest.mark.parametrize("part_len", [0, 64, 5 * MiB, 8 * MiB])
@pytest.mark.parametrize("window_bytes", [1, 4096, 3 * MiB, 4 << 30])
def test_segments_preview_matches_restatement(part_len, window_bytes):
    rng = np.random.default_rng(part_len + window_bytes)
    for sizes, seg_of in random_layouts(rng):
        if part_len == 64 and sum(sizes) > 1 * MiB:
            continue  # keeps the restatement fast; the large layouts run at the MiB part sizes
        got = _lib.segments_preview(sizes, seg_of, part_len, window_bytes)
        rows, windows = restated_preview(sizes, seg_of, part_len, window_bytes)
        assert got["gathered"].tolist() == [r[0] for r in rows], (sizes, seg_of)
        assert got["a"].tolist() == [r[1] for r in rows], (sizes, seg_of)
        assert got["b"].tolist() == [r[2] for r in rows], (sizes, seg_of)
        assert got["window_bytes"].tolist() == windows, (sizes, seg_of)


def test_segments_preview_of_a_safetensors_file_gathers_one_block_per_boundary():
    # header + two 20 MiB tensors: 8 MiB blocks, one straddles header|t0 (block 0), one t0|t1
    header = 8 + 120
    got = _lib.segments_preview([header, 20 * MiB, 20 * MiB], [0, 3], 8 * MiB)
    assert got["gathered"].tolist() == [True, False, True, False, False, False]
    assert got["b"][0] == 2 and got["b"][2] == 2 and got["window_bytes"].tolist() == [16 * MiB]


# ---- the safetensors framing -----------------------------------------------------------------------------------


@pytest.mark.parametrize("case", GOLDEN["cases"], ids=[c["name"] for c in GOLDEN["cases"]])
def test_safetensors_layout_equals_golden(case):
    tensors = state_dict_from_recipe(case["tensors"])
    header, ordered = blob_utils.safetensors_layout(tensors, case["metadata"])
    assert header.hex() == case["header_hex"]
    data = file_bytes(tensors, case["metadata"])
    assert len(data) == case["size"] and hashlib.sha256(data).hexdigest() == case["sha256"]
    assert sorted(n for n, _ in ordered) == sorted(tensors)


@pytest.mark.parametrize("case", GOLDEN["cases"], ids=[c["name"] for c in GOLDEN["cases"]])
def test_safetensors_layout_equals_installed_package(case):
    st = pytest.importorskip("safetensors.torch")
    tensors = state_dict_from_recipe(case["tensors"])
    data = file_bytes(tensors, case["metadata"])
    assert data == st.save(tensors, case["metadata"])
    back = st.load(data)
    assert set(back) == set(tensors) and all(torch.equal(back[k].reshape(-1).view(torch.uint8), tensors[k].reshape(-1).view(torch.uint8))
                                             for k in tensors if tensors[k].numel())


def test_safetensors_layout_rejects_other_dtypes_by_name():
    with pytest.raises(ValueError, match="'w.q'.*complex128"):
        blob_utils.safetensors_layout({"a": torch.zeros(1), "w.q": torch.zeros(2, dtype=torch.complex128)})


def test_product_never_imports_safetensors():
    code = ("import sys; import modal_client_b200, modal_client_b200.volume, modal_client_b200.blob_utils as b, torch;"
            "b.safetensors_layout({'a': torch.zeros(2)}, {'k': 'v'});"
            "assert not any(m == 'safetensors' or m.startswith('safetensors.') for m in sys.modules), 'imported'")
    subprocess.run([sys.executable, "-c", code], cwd=ROOT, check=True)


# ---- validation --------------------------------------------------------------------------------------------------


def test_put_safetensors_validates_at_call_time(fake_backend):
    batch = volume._BatchBase("vo", client=None)
    with pytest.raises(ValueError, match="str tensor names"):
        batch.put_safetensors({1: torch.zeros(1)}, "/m.safetensors")
    with pytest.raises(ValueError, match="__metadata__"):
        batch.put_safetensors({"__metadata__": torch.zeros(1)}, "/m.safetensors")
    with pytest.raises(ValueError, match="'w' is not a CUDA tensor"):
        batch.put_safetensors({"w": torch.zeros(4)}, "/m.safetensors")
    with pytest.raises(ValueError, match="metadata must map str to str"):
        batch.put_safetensors({"w": torch.zeros(4)}, "/m.safetensors", metadata={"step": 3})
    with pytest.raises(ValueError) as put_file_err:
        batch.put_file(io.BytesIO(b"x"), "/")
    with pytest.raises(ValueError) as put_st_err:
        batch.put_safetensors({"w": torch.zeros(4)}, "/")
    assert str(put_st_err.value) == str(put_file_err.value)
    assert batch._safetensors == []


# ---- the reader ---------------------------------------------------------------------------------------------------


def test_host_backed_segments_reader_reads_seeks_clones_and_counts():
    tensors = {"b": torch.arange(1000, dtype=torch.int32), "a": torch.ones(33, dtype=torch.bfloat16),
               "z": torch.zeros(0), "s": torch.tensor(2.5)}
    header, ordered = blob_utils.safetensors_layout(tensors)
    raw = file_bytes(tensors)
    r = blob_utils.DeviceSegmentsReader(header, [t for _, t in ordered])
    assert r.nbytes == len(raw) and r.seek(0, os.SEEK_END) == len(raw) and r.seek(len(header) - 5) == len(header) - 5
    assert r.read(50) == raw[len(header) - 5 : len(header) + 45] and r.tell() == len(header) + 45
    c = r.clone()
    assert c.tell() == 0 and c.read() == raw
    with r.clone() as c2:
        c2.seek(len(raw) - 3)
        assert c2.read(100) == raw[-3:] and c2.read(5) == b""
    assert r.bytes_to_host == 50 + len(raw) + 3
    segs = r.segments(3, len(header))  # part of the header and the first bytes of the first tensor
    assert [n for _, n in segs] == [len(header) - 3, 3]


# ---- request flow on the stand-in -------------------------------------------------------------------------------


def _state_dicts():
    out = []
    for i, n in enumerate([3, 1, 40]):
        g = torch.Generator().manual_seed(i)
        sd = {f"layer.{k}.w": torch.randn(int(torch.randint(0, 700, (1,), generator=g)), generator=g) for k in range(n)}
        sd[f"layer.{n}.mask"] = torch.zeros(3000, dtype=torch.uint8)  # trailing zeros: trimmed blocks
        sd["bias"] = torch.arange(17, dtype=torch.int64)
        out.append((sd, {"format": "pt"} if i else None, f"/ckpt/m{i}.safetensors"))
    return out


def _reader(sd, md):
    header, ordered = blob_utils.safetensors_layout(sd, md)
    return blob_utils.DeviceSegmentsReader(header, [t for _, t in ordered])


def test_v1_safetensors_rows_equal_put_file_rows(monkeypatch):
    ctx = FakeSegmentsContext()
    monkeypatch.setattr(_backend, "_override", ctx)
    monkeypatch.setattr(blob_utils, "LARGE_FILE_LIMIT", 20_000)  # the 40-tensor file becomes a blob
    items = _state_dicts()

    async def upload(use_segments):
        async with running_blob_server() as (host, store):
            stub = FakeVolumeStub(host, store, 8 << 20)
            sent = []
            orig = stub.VolumePutFiles

            async def record(req):
                sent.append(req)
                return await orig(req)

            stub.VolumePutFiles = record
            async with volume.VolumeUploadContextManager("vo-1", types.SimpleNamespace(stub=stub)) as batch:
                for sd, md, path in items:
                    if use_segments:
                        batch._safetensors.append((_reader(sd, md), path, 0o600))
                    else:
                        batch.put_file(io.BytesIO(file_bytes(sd, md)), path, mode=0o600)
            await blob_utils.ClientSessionRegistry.close_session()
            return sent[0].files, {k: v[0] for k, v in stub.volume_files.items()}, sorted(store.blobs.values())

    got_rows, got_files, got_blobs = asyncio.run(upload(True))
    want_rows, want_files, want_blobs = asyncio.run(upload(False))
    assert got_rows == want_rows and got_files == want_files and got_blobs == want_blobs
    assert got_files == {path: file_bytes(sd, md) for sd, md, path in items}
    assert any(c[0] == "hash_device_segments" and c[2] == 0 for c in ctx.calls)


def test_v2_safetensors_request_equals_put_file_request(monkeypatch):
    BS = 4096
    monkeypatch.setattr(blob_utils, "BLOCK_SIZE", BS)
    ctx = FakeSegmentsContext()
    monkeypatch.setattr(_backend, "_override", ctx)
    items = _state_dicts()

    async def upload(use_segments):
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
                    for sd, md, path in items:
                        if use_segments:
                            readers.append(_reader(sd, md))
                            batch._safetensors.append((readers[-1], path, 0o640))
                        else:
                            batch.put_file(io.BytesIO(file_bytes(sd, md)), path, mode=0o640)
            finally:
                await runner.cleanup()
                await blob_utils.ClientSessionRegistry.close_session()
            return sent, {k: v[0] for k, v in stub.volume_files.items()}, stub.blocks, readers

    got_reqs, got_files, got_blocks, readers = asyncio.run(upload(True))
    want_reqs, want_files, _, _ = asyncio.run(upload(False))
    assert [r.files for r in got_reqs] == [r.files for r in want_reqs]
    assert got_files == want_files == {path: file_bytes(sd, md) for sd, md, path in items}
    assert sum(r.bytes_to_host for r in readers) == sum(len(b) for b in got_blocks.values())
    assert ("hash_device_segments", len(items), BS, _lib.SHA256 | _lib.TRIM_ZEROS) in ctx.calls
    st = pytest.importorskip("safetensors.torch")
    for sd, md, path in items:
        back = st.load(got_files[path])
        assert set(back) == set(sd) and all(torch.equal(back[k], sd[k]) for k in sd)
