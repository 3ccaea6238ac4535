"""tools/safetensors_volume_bench.py -- Volume.batch_upload (volumefs2) of one state dict as a safetensors file: the
put_safetensors leg of tools/tensor_volume_bench.py, one JSON line per measurement.

Same state dict (log-normal uint8 tensors summing to --total-gib, random bytes made on the GPU), same null
VolumePutFiles2 and discarding block server, same --missing.  Three ways: put_safetensors; today's way without it
(safetensors.torch.save_file to --dir, then put_file; only where the safetensors package is installed); and
put_tensor per tensor, which uploads the same bytes without any framing (one file per tensor).  Per run: wall time,
bytes copied device -> host, bytes PUT.  Alone: the hash of put_safetensors (safetensors_upload_specs2: wall time,
lane_hash device time, gather_pieces_kernel device time from torch.profiler, scratch bytes from the row table) and the
same for put_tensor (tensor_upload_specs2).  Every path is warmed up on a small dict first; the card name and power
limit are read with nvidia-smi (query only) in the same run.
usage: python tools/safetensors_volume_bench.py [--out profiles/r5_safetensors_volume_bench.jsonl] [--total-gib 16]
                                                [--missing 0,50,100] [--dir /dev/shm]"""
import argparse
import asyncio
import json
import os
import shutil
import sys
import tempfile
import time
import types

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np

from modal_client_b200 import _backend, _lib, blob_utils, volume
from tensor_volume_bench import GiB, MiB, NullStub, card, state_dict


async def upload(sd, url, pct, way, where):
    stub = NullStub(url, pct)
    client = types.SimpleNamespace(stub=stub)
    t0 = time.perf_counter()
    async with volume.VolumeUploadContextManager2("vo-bench", client) as b:
        if way == "put_safetensors":
            b.put_safetensors(sd, "/ckpt/model.safetensors")
        elif way == "put_tensor":
            for name, t in sd.items():
                b.put_tensor(t, f"/ckpt/{name}.bin")
        else:
            import safetensors.torch as st

            path = os.path.join(where, "model.safetensors")
            st.save_file(sd, path)
            b.put_file(path, "/ckpt/model.safetensors")
        readers = [r for r, _, _ in b._safetensors] + [r for r, _, _ in b._tensors]
    wall = time.perf_counter() - t0
    to_host = sum(r.bytes_to_host for r in readers) if readers else sum(t.numel() for t in sd.values())
    return wall, to_host


def hash_alone(ctx, specs_fn, items):
    """(wall s, lane_hash device ms, gather_pieces_kernel device ms, blocks) of one spec call."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    ctx.profile_enable(True)
    ctx.profile_read()
    t0 = time.perf_counter()
    specs = specs_fn(items)
    wall = time.perf_counter() - t0
    lane_ms, _ = ctx.profile_read()
    ctx.profile_enable(False)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:  # a run of its own: tracing slows the host
        specs_fn(items)
        torch.cuda.synchronize()
    gather_us = sum(e.device_time_total for e in prof.key_averages() if "gather_pieces_kernel" in e.key)
    return wall, lane_ms, gather_us / 1e3, sum(len(s.blocks) for s in specs)


async def main_async(args):
    import torch
    from aiohttp import web

    try:
        import safetensors.torch  # noqa: F401

        have_st = True
    except ImportError:
        have_st = False
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
    sd = {f"t{i:05d}": t for i, t in enumerate(state_dict(total))}
    torch.cuda.synchronize()
    out = open(args.out, "a") if args.out else None

    def emit(rec):
        rec.update(cards=cards, tensors=len(sd), total_bytes=sum(t.numel() for t in sd.values()))
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    room = shutil.disk_usage(args.dir).free
    tmp = tempfile.mkdtemp(dir=args.dir)
    file_way = have_st and room > 1.2 * total
    ways = ("put_safetensors", "put_tensor") + (("save_file_put_file",) if file_way else ())
    try:
        small = dict(list(sd.items())[:8])
        for way in ways:
            await upload(small, url, 100, way, tmp)
        header, ordered = blob_utils.safetensors_layout(sd)
        reader = blob_utils.DeviceSegmentsReader(header, [t for _, t in ordered])
        sizes = [len(header)] + [t.numel() for _, t in ordered]
        scratch = int(_lib.segments_preview(sizes, [0, len(sizes)], blob_utils.BLOCK_SIZE)["window_bytes"].max())
        wall, lane_ms, gather_ms, blocks = hash_alone(ctx, blob_utils.safetensors_upload_specs2,
                                                      [(reader, "/m.safetensors", 0o644)])
        emit({"leg": "hash", "way": "put_safetensors", "blocks": blocks, "wall_ms": wall * 1e3,
              "lane_hash_device_ms": lane_ms, "gather_device_ms": gather_ms, "scratch_bytes": scratch})
        items = [(blob_utils.DeviceBufferReader(t), f"/{n}", 0o644) for n, t in sd.items()]
        wall, lane_ms, gather_ms, blocks = hash_alone(ctx, blob_utils.tensor_upload_specs2, items)
        emit({"leg": "hash", "way": "put_tensor", "blocks": blocks, "wall_ms": wall * 1e3,
              "lane_hash_device_ms": lane_ms, "gather_device_ms": gather_ms, "scratch_bytes": 0})
        for pct in args.missing:
            for way in ("put_safetensors", "put_tensor", "save_file_put_file"):
                if way not in ways:
                    why = "safetensors is not installed" if not have_st else f"{args.dir} has {room / GiB:.1f} GiB free"
                    emit({"leg": "upload", "way": way, "missing_pct": pct, "result": f"not measured: {why}"})
                    continue
                put_bytes[0] = 0
                wall, to_host = await upload(sd, url, pct, way, tmp)
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
    ap.add_argument("--out", default="profiles/r5_safetensors_volume_bench.jsonl")
    ap.add_argument("--total-gib", type=float, default=16)
    ap.add_argument("--missing", type=lambda s: [int(x) for x in s.split(",")], default=[0, 50, 100])
    ap.add_argument("--dir", default="/dev/shm")
    asyncio.run(main_async(ap.parse_args()))


if __name__ == "__main__":
    main()
