"""tools/tensor_volume_bench.py -- Volume.batch_upload (volumefs2) of a state-dict-like set of CUDA tensors: put_tensor
against the way without it (t.cpu() -> a file on tmpfs -> put_file), one JSON line per measurement.

The set: log-normal tensor sizes (sigma 1.5, >= 4 KiB) summing to --total-gib, random bytes made on the GPU.  The null
VolumePutFiles2 reports --missing percent of the blocks missing in its first answer (a fixed pseudo-random selection)
and none in the second; missing blocks are PUT to an in-process aiohttp server that reads and discards the body.  Per
run: wall time of the whole batch, bytes copied device -> host (DeviceBufferReader.bytes_to_host for put_tensor; the
.cpu() copies for the file way, whose PUTs then read the files again), and for put_tensor the hash on its own
(tensor_upload_specs2: wall time and lane_hash device time from CUDA events).  Every path is warmed up on a small set
first.  The card name and power limit are read with nvidia-smi (query only) in the same run.
usage: python tools/tensor_volume_bench.py [--out profiles/r4_tensor_volume_bench.jsonl] [--total-gib 16]
                                           [--missing 0,50,100] [--dir /dev/shm]"""
import argparse
import asyncio
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
import types

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

from modal_client_b200 import _backend, _lib, blob_utils, volume

MiB, GiB = 1 << 20, 1 << 30


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout
    return [line.strip() for line in out.strip().splitlines()]


def state_dict(total_bytes, seed=0):
    import torch

    rng = np.random.default_rng(seed)
    sizes = []
    while sum(sizes) < total_bytes:
        sizes.append(int(max(4096, rng.lognormal(np.log(16 * MiB), 1.5))))
    sizes[-1] -= sum(sizes) - total_bytes
    if sizes[-1] < 4096:
        sizes.pop()
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randint(0, 256, (n,), dtype=torch.uint8, device="cuda", generator=g) for n in sizes]


class NullStub:
    """VolumePutFiles2 that lacks `missing_pct` percent of the blocks the first time it sees a batch."""

    def __init__(self, url, missing_pct):
        self.url, self.pct, self.rounds = url, missing_pct, 0

    async def VolumePutFiles2(self, req):
        self.rounds += 1
        if self.rounds > 1:
            return types.SimpleNamespace(missing_blocks=[])
        return types.SimpleNamespace(missing_blocks=[
            types.SimpleNamespace(file_index=fi, block_index=bi, put_url=f"{self.url}/block")
            for fi, f in enumerate(req.files) for bi in range(len(f.blocks))
            if (fi * 1_000_003 + bi * 7919) % 100 < self.pct])


async def upload(tensors, url, pct, way, where):
    stub = NullStub(url, pct)
    client = types.SimpleNamespace(stub=stub)
    readers = []
    t0 = time.perf_counter()
    async with volume.VolumeUploadContextManager2("vo-bench", client) as b:
        for i, t in enumerate(tensors):
            if way == "put_tensor":
                b.put_tensor(t, f"/ckpt/t{i}.bin")
            else:
                path = os.path.join(where, f"t{i}.bin")
                t.cpu().numpy().tofile(path)
                b.put_file(path, f"/ckpt/t{i}.bin")
        readers = [r for r, _, _ in b._tensors]
    wall = time.perf_counter() - t0
    to_host = sum(r.bytes_to_host for r in readers) if way == "put_tensor" else sum(t.numel() for t in tensors)
    return wall, to_host


async def main_async(args):
    import torch
    from aiohttp import web

    put_bytes = [0]

    async def put_block(request):
        async for chunk in request.content.iter_any():
            put_bytes[0] += len(chunk)
        return web.Response(text="ok")

    app = web.Application(client_max_size=64 * MiB)
    app.add_routes([web.put("/block", put_block)])
    runner = web.AppRunner(app)
    await runner.setup()
    site = web.TCPSite(runner, "127.0.0.1", 0)
    await site.start()
    url = f"http://127.0.0.1:{site._server.sockets[0].getsockname()[1]}"
    ctx = _lib.Context(0)
    _backend.set_context(ctx)
    cards = card()
    total = int(args.total_gib * GiB)
    tensors = state_dict(total)
    torch.cuda.synchronize()
    out = open(args.out, "a") if args.out else None

    def emit(rec):
        rec.update(cards=cards, tensors=len(tensors), total_bytes=sum(t.numel() for t in tensors))
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    room = shutil.disk_usage(args.dir).free
    tmp = tempfile.mkdtemp(dir=args.dir)
    file_way = room > 1.2 * total
    try:
        for way in ("put_tensor",) + (("cpu_file_put_file",) if file_way else ()):  # warm-up of both paths
            await upload(tensors[:8], url, 100, way, tmp)
        # the hash alone: every block of every tensor in one device call
        items = [(blob_utils.DeviceBufferReader(t), f"/t{i}", 0o644) for i, t in enumerate(tensors)]
        ctx.profile_enable(True)
        ctx.profile_read()
        t0 = time.perf_counter()
        specs = blob_utils.tensor_upload_specs2(items)
        hash_wall = time.perf_counter() - t0
        lane_ms, launches = ctx.profile_read()
        ctx.profile_enable(False)
        emit({"leg": "hash", "blocks": sum(len(s.blocks) for s in specs), "wall_ms": hash_wall * 1e3,
              "lane_hash_device_ms": lane_ms, "lane_hash_launches": launches,
              "device_GBps": sum(t.numel() for t in tensors) / lane_ms / 1e6 if lane_ms else None})
        for pct in args.missing:
            for way in ("put_tensor", "cpu_file_put_file"):
                if way != "put_tensor" and not file_way:
                    emit({"leg": "upload", "way": way, "missing_pct": pct,
                          "result": f"not measured: {args.dir} has {room / GiB:.1f} GiB free"})
                    continue
                put_bytes[0] = 0
                wall, to_host = await upload(tensors, url, pct, way, tmp)
                emit({"leg": "upload", "way": way, "missing_pct": pct, "wall_s": wall, "bytes_to_host": to_host,
                      "bytes_put": put_bytes[0]})
                for f in os.listdir(tmp):
                    os.unlink(os.path.join(tmp, f))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
        await blob_utils.ClientSessionRegistry.close_session()
        await runner.cleanup()
        ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r4_tensor_volume_bench.jsonl")
    ap.add_argument("--total-gib", type=float, default=16)
    ap.add_argument("--missing", type=lambda s: [int(x) for x in s.split(",")], default=[0, 50, 100])
    ap.add_argument("--dir", default="/dev/shm")
    asyncio.run(main_async(ap.parse_args()))


if __name__ == "__main__":
    main()
