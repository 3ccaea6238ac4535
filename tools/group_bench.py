"""tools/group_bench.py -- device groups (one process, several GPUs) through the API, one JSON line per measurement.

  (a) batch.hash_table_host over 8 GiB of C5 messages (4 / 16 / 64 MiB), from pageable and from host_alloc memory;
  (b) blob_utils.file_upload_specs2 (C3-v2) and get_file_upload_specs (C3-v1) over a log-normal tree (files_bench.py's);
  (c) Volume.batch_upload (volumefs2) over that tree against null RPCs: config 3 through the API;
  (d) the min_share_bytes crossover: one member against a forced split over two, growing batches of 256 KiB messages
      (short enough that the batch, not one message's serial chain, sets the time).
Groups [0], [0,0], [0,1], [0..3], [0..7]; a group needing more GPUs than the box has is written as "not measured".
Every shape is warmed up first; times are the median of --steps host-clock runs around calls that return only once the
digests are in host memory.  The card name and power limit are read with nvidia-smi (query only) in the same run.
usage: python tools/group_bench.py [--out profiles/r3_group_bench.jsonl] [--tree-gib 16] [--tree-files 100000]
                                   [--steps 3] [--dir /dev/shm] [--legs c5,sweep,tree]"""
import argparse
import asyncio
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time
import types
from pathlib import Path, PurePosixPath

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

from modal_client_b200 import _backend, _lib, batch, blob_utils, volume
from modal_client_b200.synth import synth_array

MiB, GiB = 1 << 20, 1 << 30
GROUPS = {"[0]": [0], "[0,0]": [0, 0], "[0,1]": [0, 1], "[0..3]": [0, 1, 2, 3], "[0..7]": list(range(8))}


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout
    return [line.strip() for line in out.strip().splitlines()]


def timed(fn, steps):
    fn()  # warm-up of this exact shape
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts)


class NullVolumeStub:
    """VolumePutFiles2 that already holds every block: the upload costs the client its hashing and request building."""

    async def VolumePutFiles2(self, request):
        self.files = len(request.files)
        return types.SimpleNamespace(missing_blocks=[])


def build_tree(where, n, total_gib):
    root = Path(tempfile.mkdtemp(prefix="b200h_group_tree_", dir=where))
    rng = np.random.default_rng(0)
    sigma = 1.5
    sizes = np.clip(rng.lognormal(np.log(102400) - sigma**2 / 2, sigma, n), 1, 1 << 28)
    sizes = np.maximum(1, (sizes * (total_gib * GiB / sizes.sum())).astype(np.int64))
    blob = synth_array(9, int(sizes.max()) + MiB)
    files = []
    for i, s in enumerate(sizes):
        d = root / f"d{i % 64}"
        if i < 64:
            d.mkdir()
        p = d / f"f{i}.bin"
        with open(p, "wb") as f:
            f.write(blob[i % 4096 : i % 4096 + int(s)].tobytes())
        files.append((p, PurePosixPath(f"/vol/d{i % 64}/f{i}.bin"), None))
    return root, files, int(sizes.sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r3_group_bench.jsonl")
    ap.add_argument("--tree-gib", type=float, default=16.0)
    ap.add_argument("--tree-files", type=int, default=100_000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--dir", default="/dev/shm" if os.path.isdir("/dev/shm") else "/tmp")
    ap.add_argument("--legs", default="c5,sweep,tree")
    a = ap.parse_args()
    legs = set(a.legs.split(","))
    ndev = _lib.load_library().b200h_device_count()
    if ndev < 1:
        raise SystemExit("no CUDA device: this benchmark measures the GPU and has nothing to fall back to")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    out = open(a.out, "w")

    def emit(**row):
        line = json.dumps(row)
        print(line, flush=True)
        out.write(line + "\n")
        out.flush()

    emit(kind="host", cards=card(), device_count=ndev, cpus=os.cpu_count())
    runnable = {k: v for k, v in GROUPS.items() if max(v) < ndev}
    for k in GROUPS:
        if k not in runnable:
            emit(kind="group", group=k, result="not measured", why=f"needs {max(GROUPS[k]) + 1} GPUs, box has {ndev}")

    # (a) C5 over 8 GiB
    total = 8 * GiB
    pageable = synth_array(21, total)
    home = _lib.Context(0)
    pinned = home.host_alloc(total)
    pinned[:] = pageable
    for name, devs in runnable.items() if "c5" in legs else ():
        g = _lib.DeviceGroup(devs)
        for mib in (4, 16, 64):
            n = total // (mib * MiB)
            lens = np.full(n, mib * MiB, np.uint64)
            offs = np.arange(n, dtype=np.uint64) * np.uint64(mib * MiB)
            for src_name, src in (("pageable", pageable), ("host_alloc", pinned)):
                dt = timed(lambda: batch.hash_table_host(src, offs, lens, ctx=g), a.steps)
                emit(kind="c5", group=name, msg_mib=mib, source=src_name, gib=total / GiB, seconds=round(dt, 4),
                     gib_s=round(total / GiB / dt, 2), split=g.last_split())
        g.close()

    # (d) crossover: one member vs. a forced split over two
    pair = "[0,1]" if "[0,1]" in runnable else "[0,0]"
    one = _lib.DeviceGroup([0], min_share_bytes=1)
    two = _lib.DeviceGroup(GROUPS[pair], min_share_bytes=1)
    for mib_total in (16, 64, 256, 1024, 4096) if "sweep" in legs else ():
        n = mib_total * 4
        lens = np.full(n, 256 << 10, np.uint64)
        offs = np.arange(n, dtype=np.uint64) * np.uint64(256 << 10)
        for src_name, src in (("pageable", pageable), ("host_alloc", pinned)):
            t1 = timed(lambda: one.hash_batch_host(src, offs, lens, _lib.SHA256 | _lib.MD5), max(a.steps, 5))
            t2 = timed(lambda: two.hash_batch_host(src, offs, lens, _lib.SHA256 | _lib.MD5), max(a.steps, 5))
            emit(kind="min_share_sweep", pair=pair, msg_kib=256, batch_mib=mib_total, per_member_mib=mib_total / 2,
                 source=src_name, one_ms=round(t1 * 1e3, 3), split_ms=round(t2 * 1e3, 3), split_faster=t2 < t1)
    one.close()
    two.close()
    home.host_free(pinned)
    del pageable

    if "tree" not in legs:
        return
    # (b) + (c) over one tree
    free = shutil.disk_usage(a.dir).free
    tree_gib = min(a.tree_gib, 0.4 * free / GiB, 100.0)
    t0 = time.perf_counter()
    root, files, nbytes = build_tree(a.dir, min(a.tree_files, 1_000_000), tree_gib)
    emit(kind="tree", dir=a.dir, files=len(files), gib=round(nbytes / GiB, 2), written_s=round(time.perf_counter() - t0, 1),
         dir_free_gib=round(free / GiB, 1))
    try:
        for name, devs in runnable.items():
            g = _lib.DeviceGroup(devs)
            _backend.set_context(g)
            try:
                dt = timed(lambda: asyncio.run(blob_utils.file_upload_specs2(files)), a.steps)
                emit(kind="c3v2_specs", group=name, seconds=round(dt, 3), gib_s=round(nbytes / GiB / dt, 2),
                     split=g.last_split())
                dt = timed(lambda: blob_utils.get_file_upload_specs(files, cache_small_content=False), a.steps)
                emit(kind="c3v1_specs", group=name, seconds=round(dt, 3), gib_s=round(nbytes / GiB / dt, 2),
                     split=g.last_split())

                async def upload():
                    client = types.SimpleNamespace(stub=NullVolumeStub())
                    async with volume.VolumeUploadContextManager2("vo-null", client) as b:
                        b.put_directory(root, "/vol")

                dt = timed(lambda: asyncio.run(upload()), a.steps)
                emit(kind="c3_batch_upload_v2", group=name, seconds=round(dt, 3), gib_s=round(nbytes / GiB / dt, 2),
                     split=g.last_split())
            finally:
                _backend.set_context(None)
                g.close()
    finally:
        shutil.rmtree(root, ignore_errors=True)
    out.close()


if __name__ == "__main__":
    main()
