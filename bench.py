#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 blob-ingest / content-hash path.

Workload (BASELINE.json configs[1]): the Function.map input pump -- 100 000 pickled inputs of
256 KiB each (24.4 GiB), fused SHA-256 + MD5 per payload -- per GPU (weak scaling; payload sets are
independent, no data-path collective; the per-rank digest tables are all-gathered over NCCL).

  value     GiB/s with the payloads already resident in HBM (CUDA events, max over ranks)
  e2e       GiB/s through the plugin call itself: 100 000 pageable Python ``bytes`` -> parallel_map.InputPreprocessor
            (one GPU hash batch per byte-budgeted window, pack + H2D + kernels + D2H digests) -> BlobCreate / PUT per
            input -> parallel_map.InputPumper, against a null control plane / object store
  e2e_pinned  the same payloads through batch.hash_table_host on page-locked host memory (round 1's e2e figure)
  roofline  lane_hash_kernel: algorithmic bytes / measured kernel time vs the measured HBM copy peak
  cpu_baseline  the reference's own get_upload_hashes (unmodified hash_utils.py from the checkout named by
            B200H_REFERENCE_ROOT, through oracle/ref_shim.py; oracle/ref_port.py without one) on the host cores,
            bounded sample

`--steps` timed steps (after `--warmup` untimed ones) are run on every leg above but the CPU baseline.
`--impl reference` times that same reference implementation (hashlib underneath, all host threads) on the same
workload shape and prints the same JSON line.
`--dump-outputs DIR` writes, after the timed steps, the digest tables the last step of each GPU leg returned as
float32 DIR/<name>.npy (one row per message, one column per digest byte): sha256 / md5 (HBM-resident),
e2e_pinned_sha256 / e2e_pinned_md5, e2e_sha256 / e2e_md5 (as BlobCreate received them).  The payloads are
generated from a fixed seed, so two builds can be compared output for output.  Past OUTPUT_DUMP_BYTES in all, a
fixed, seeded sample of rows is written, with their indices in rows.npy.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GiB = float(1 << 30)
N_MSG = int(os.environ.get("B200H_BENCH_NMSG", 100_000))
MSG_BYTES = int(os.environ.get("B200H_BENCH_MSG_BYTES", 256 * 1024))
METRIC = "GiB/s hashed+chunked (SHA-256+MD5) on synthetic blobs"
WORKLOAD = f"Function.map input pump: {N_MSG} x {MSG_BYTES // 1024} KiB pickled inputs blobified, per GPU"


def hbm_peak_gbs() -> tuple[float, str]:
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows: list[list[str]] = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.idx)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def halt(self) -> list:
        """Stop sampling and return the raw rows (lets a caller merge several timed regions)."""
        if self.proc:
            time.sleep(0.25)
            self.proc.terminate()
        return self.rows

    @staticmethod
    def summarize(rows: list, available: bool = True) -> dict:
        if not available:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm, smax, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                smax.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}

    def stop(self) -> dict:
        rows = self.halt()
        return self.summarize(rows, self.proc is not None)


OUTPUT_DUMP_BYTES = 64 * 10**6


def dump_outputs(out_dir: str, tables: dict) -> None:
    """``tables``: name -> uint8[n, k] digest table (the same n for all).  Each is written as float32
    ``out_dir/<name>.npy``; if that would pass OUTPUT_DUMP_BYTES, the same fixed, seeded sample of rows of every
    table is written instead, and the sampled row indices as float64 ``rows.npy``."""
    import numpy as np

    n = len(next(iter(tables.values())))
    row_bytes = sum(4 * t.shape[1] for t in tables.values())
    budget = OUTPUT_DUMP_BYTES - 4096  # room for the .npy headers
    rows = None
    if n * row_bytes > budget:
        rows = np.sort(np.random.default_rng(0).choice(n, budget // (row_bytes + 8), replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in tables.items():
        assert len(t) == n, name
        np.save(os.path.join(out_dir, f"{name}.npy"), (t if rows is None else t[rows]).astype(np.float32))
    if rows is not None:
        np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))


def env_rank():
    return (int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0)))


# ----------------------------------------------------------------------------------- reference arm


def cpu_payloads(n: int, seed: int) -> list[bytes]:
    from modal_client_b200.synth import synth_bytes

    return [synth_bytes(seed, MSG_BYTES, start=i * MSG_BYTES) for i in range(n)]


_REF = None


def reference_hasher():
    """(callable, kind): the reference's OWN ``get_upload_hashes`` (unmodified hash_utils.py from the checkout named
    by B200H_REFERENCE_ROOT, loaded through oracle/ref_shim.py) -> kind "reference"; without one, the hashlib
    port in oracle/ref_port.py -> kind "port".  Both make exactly the same hashlib calls."""
    global _REF
    if _REF is None:
        from oracle import ref_port, ref_shim  # allowed here: CPU baseline / reference arm only

        try:
            h, _, _ = ref_shim.load()
            _REF = (h.get_upload_hashes, "reference")
        except Exception:
            _REF = (ref_port.upload_hashes, "port")
    return _REF


def host_description() -> dict:
    """What SURVEY 8(d) asks to be stated next to the CPU baseline: logical CPUs, CPU model, SHA extensions, OpenSSL."""
    import ssl

    model, sha_ni = "unknown", False
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name") and model == "unknown":
                    model = line.split(":", 1)[1].strip()
                elif line.startswith("flags"):
                    sha_ni = " sha_ni" in line
                    break
    except OSError:
        pass
    return {"logical_cpus": os.cpu_count() or 1, "cpu_model": model, "sha_ni": sha_ni, "openssl": ssl.OPENSSL_VERSION}


def run_cpu_pool(payloads: list[bytes], workers: int) -> float:
    from concurrent.futures import ThreadPoolExecutor

    fn, _ = reference_hasher()
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=workers) as ex:
        list(ex.map(fn, payloads))
    return time.perf_counter() - t0


def best_pool_workers(probe: list[bytes], repeats: int = 1) -> int:
    """"All the host threads it can use": try the reference's default pool size (min(32, ncpu+4)), half and
    all logical CPUs on a warm-up slice and keep the fastest (python thread pools do not scale to every core)."""
    ncpu = os.cpu_count() or 1
    workers, best = ncpu, None
    for w in sorted({min(32, ncpu + 4), max(1, ncpu // 2), ncpu}):
        for _ in range(repeats):
            t = run_cpu_pool(probe, w)
        if best is None or t < best:
            workers, best = w, t
    return workers


def run_reference(args) -> None:
    rank, world, _ = env_rank()
    if rank != 0:
        return
    sample_n = int(os.environ.get("B200H_REF_SAMPLE", 16384))  # 4 GiB of 256 KiB payloads per step
    payloads = cpu_payloads(sample_n, 0xB200)
    workers = best_pool_workers(payloads[: max(1024, sample_n // 4)], max(1, args.warmup))
    times = [run_cpu_pool(payloads, workers) for _ in range(args.steps)]
    total = sum(times)
    gibs = sample_n * MSG_BYTES * args.steps / GiB / total
    what = "the reference's own get_upload_hashes" if reference_hasher()[1] == "reference" else "get_upload_hashes port"
    sample = f"{sample_n} of {N_MSG} payloads x {MSG_BYTES // 1024} KiB per step, hashlib SHA-256+MD5 via {what}, ThreadPool({workers})"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(gibs, 3), "unit": "GiB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * total / args.steps, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": round(gibs, 3), "unit": "GiB/s", "cores": workers, "kind": reference_hasher()[1],
                         "sample": sample, "host": host_description()},
        "e2e": {"value": round(gibs, 3), "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ----------------------------------------------------------------------------------------- GPU arm


class _NullBlobResponse:
    """What BlobCreate answers for a single-part upload (modal_proto/api.proto BlobCreateResponse): one blob id and
    one pre-signed URL.  The null stub hands the same object back for every request."""

    blob_ids = ["bl-null"]

    class _Urls:
        items = ["null://put"]

    upload_urls = _Urls()

    def WhichOneof(self, _name):
        return "upload_urls"


class NullStub:
    """Control plane + object store that cost nothing: BlobCreate keeps the request (so the digests the pump
    computed can be checked afterwards), FunctionPutInputs counts items."""

    def __init__(self):
        self.blob_requests = []
        self.inputs_put = 0
        self._resp = _NullBlobResponse()

    async def BlobCreate(self, request):
        self.blob_requests.append(request)
        return self._resp

    async def FunctionPutInputs(self, request):
        self.inputs_put += len(request.inputs)


async def _null_put(upload_url, payload, content_md5_b64=None, content_type="application/octet-stream"):
    """Stand-in for blob_utils._upload_to_s3_url: the payload object is built and handed over, no byte leaves."""
    return payload.md5_checksum().hexdigest()


def run_map_pump(payloads, stub) -> float:
    """One pass of the REAL plugin path over pageable ``bytes``: parallel_map.InputPreprocessor (collect -> one GPU
    hash batch per window -> BlobCreate + PUT per input) feeding parallel_map.InputPumper, as Function.map drives
    them (py/modal/parallel_map.py:90-198, _utils/blob_utils.py:338-352).  The inputs are already in wire format
    (``serializer`` = identity: "pickled inputs"), every one above the blob threshold.  Returns seconds."""
    import asyncio
    import types

    from modal_client_b200 import parallel_map

    fn = types.SimpleNamespace(_use_method_name="", _max_object_size_bytes=1, _metadata=object(), object_id="fu-bench")
    client = types.SimpleNamespace(stub=stub)

    async def main():
        raw, done = asyncio.Queue(), asyncio.Queue()
        for p in payloads:
            raw.put_nowait(p)
        raw.put_nowait(None)
        pre = parallel_map.InputPreprocessor(client, raw_input_queue=raw, processed_input_queue=done, function=fn,
                                             serializer=lambda p: p)
        pre.keep_digest_tables = True  # the per-window (sha, md5) tables, for the multi-GPU all-gather
        pump = parallel_map.InputPumper(client, input_queue=done, function=fn, function_call_id="fc-bench")

        async def drive(gen):
            async for _ in gen:
                pass

        t0 = time.perf_counter()
        await asyncio.gather(drive(pre.drain_input_generator()), drive(pump.pump_inputs()))
        dt = time.perf_counter() - t0
        assert pump.inputs_sent == len(payloads)
        run_map_pump.last_stats = {k: round(v, 4) for k, v in pre.stats.items()}
        return dt, pre.hash_batches, pre.digest_tables

    return asyncio.run(main())


def run_gpu(args) -> None:
    import numpy as np
    import torch
    import torch.distributed as dist

    from modal_client_b200 import _backend, _lib, batch, blob_utils, parallel_map, sharding

    rank, world, local_rank = env_rank()
    # a run that is still going after 13 minutes is hung (a normal one takes about one): say where, and end it,
    # instead of holding the box until somebody else's limit kills it silently
    import faulthandler

    faulthandler.dump_traceback_later(int(os.environ.get("B200H_BENCH_WATCHDOG_S", 780)), exit=True)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    all_cpus = os.sched_getaffinity(0)
    numa_bound = sharding.bind_process_to_gpu_node(local_rank)  # one process per GPU: stay next to it
    if world > 1:
        opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)  # the gather slips in between hash kernels
        dist.init_process_group("nccl", device_id=dev, pg_options=opts)
    ctx = _lib.Context(local_rank, pinned_bytes=512 << 20, device_bytes=8 << 30)
    _backend.set_context(ctx)
    BOTH = _lib.SHA256 | _lib.MD5
    total_bytes = N_MSG * MSG_BYTES
    seed = 0xB200 + rank

    # ---- synthetic payload set, generated on the device (same stream as synth.py on the CPU)
    data = torch.empty(total_bytes, dtype=torch.uint8, device=dev)
    ctx.fill_synth_device(data.data_ptr(), total_bytes, seed)
    off = torch.arange(N_MSG, dtype=torch.int64, device=dev) * MSG_BYTES
    ln = torch.full((N_MSG,), MSG_BYTES, dtype=torch.int64, device=dev)
    len_h = np.full(N_MSG, MSG_BYTES, dtype=np.uint64)  # the lengths on the host: the hash call then only enqueues
    # ONE packed digest table per step: n x 32 SHA-256 rows followed by n x 16 MD5 rows (48 B per message), double
    # buffered so that the all-gather of step k (side stream) overlaps the hash kernel of step k+1.
    NBUF = 2
    tabs = [torch.empty(N_MSG * 48, dtype=torch.uint8, device=dev) for _ in range(NBUF)]
    gathered = [torch.empty(world * N_MSG * 48, dtype=torch.uint8, device=dev) for _ in range(NBUF)] if world > 1 else None
    stream = torch.cuda.Stream(device=dev)  # non-default stream: the library launches on this very handle
    side = torch.cuda.Stream(device=dev)
    hashed = [torch.cuda.Event() for _ in range(NBUF)]
    gathered_ev = [torch.cuda.Event() for _ in range(NBUF)]
    torch.cuda.set_stream(stream)
    torch.cuda.synchronize()
    step_no = [0]

    def step():
        b = step_no[0] % NBUF
        step_no[0] += 1
        tab = tabs[b]
        if world > 1 and step_no[0] > NBUF:
            stream.wait_event(gathered_ev[b])  # the gather that last read this buffer
        ctx.hash_batch_device(data.data_ptr(), off.data_ptr(), ln.data_ptr(), N_MSG, BOTH, tab.data_ptr(),
                              tab.data_ptr() + 32 * N_MSG, 0, stream.cuda_stream, h_lengths=len_h)
        if world > 1:  # the path's only exchange: all-gather of the fixed-width digest table, off the hash stream
            hashed[b].record(stream)
            with torch.cuda.stream(side):
                side.wait_event(hashed[b])
                dist.all_gather_into_tensor(gathered[b], tab)
                gathered_ev[b].record(side)

    def drain():
        if world > 1:
            stream.wait_stream(side)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    drain()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count
    syncs0 = ctx.plan_sync_count
    ctx.profile_enable(True)
    ctx.profile_read()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    drain()
    ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    kern_ms, kern_n = ctx.profile_read()
    ctx.profile_enable(False)
    launches = ctx.launch_count - launches0
    plan_syncs = ctx.plan_sync_count - syncs0
    clock_rows = sampler.halt() if rank == 0 else []
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * total_bytes * args.steps / GiB / (ms / 1e3)
    last = tabs[(step_no[0] - 1) % NBUF].cpu().numpy()
    sha_dev, md5_dev = last[: 32 * N_MSG].reshape(-1, 32), last[32 * N_MSG :].reshape(-1, 16)
    gather_ok = None
    if world > 1:  # every rank holds every rank's table: this rank's slice must be its own table
        g = gathered[(step_no[0] - 1) % NBUF]
        gather_ok = bool(torch.equal(g[rank * N_MSG * 48 : (rank + 1) * N_MSG * 48], tabs[(step_no[0] - 1) % NBUF]))

    # ---- (secondary) end to end on page-locked host buffers: hash_table_host, digests to host
    host = ctx.host_alloc(total_bytes)
    torch.from_numpy(host).copy_(data)  # host bytes == device bytes
    torch.cuda.synchronize()
    del data
    torch.cuda.empty_cache()
    off_h = (np.arange(N_MSG, dtype=np.uint64) * np.uint64(MSG_BYTES))
    e2e_steps = args.steps
    e2e_warm = args.warmup

    def all_gather_host_table(packed: np.ndarray):
        if world > 1:  # every rank ends the step holding the whole job's digest table
            sharding.all_gather_table(packed, [N_MSG] * world, device=dev)

    def pinned_step():
        tab = batch.hash_table_host(host, off_h, len_h, ctx=ctx)
        all_gather_host_table(tab.packed())
        return tab

    for _ in range(e2e_warm):  # warm-up (first call allocates the wave buffers)
        pinned_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        table = pinned_step()
    barrier()
    pinned_s = time.perf_counter() - t0
    same = bool(np.array_equal(table.sha256, sha_dev) and np.array_equal(table.md5, md5_dev))

    # ---- (headline) end to end through the plugin call: pageable bytes -> map input pump -> BlobCreate/PUT (null)
    payloads = [host[i * MSG_BYTES:(i + 1) * MSG_BYTES].tobytes() for i in range(N_MSG)]  # ordinary Python bytes
    ctx.host_free(host)
    blob_utils._upload_to_s3_url = _null_put
    launches_pump0 = ctx.launch_count

    def pump_step():
        stub = NullStub()
        dt, batches, tables = run_map_pump(payloads, stub)
        return stub, dt, batches, tables

    def pump_table(tables) -> np.ndarray:
        """uint8[n, 48] digest table of one pump pass, from the per-window tables the preprocessor kept."""
        sha = np.concatenate([t[0] for t in tables])
        md5 = np.concatenate([t[1] for t in tables])
        return np.concatenate([sha, md5], axis=1)

    def requests_table(stub) -> np.ndarray:
        """The same table as the control plane received it (base64 fields of the BlobCreate requests)."""
        import base64

        rows = [base64.b64decode(r.content_sha256_base64) + base64.b64decode(r.content_md5) for r in stub.blob_requests]
        return np.frombuffer(b"".join(rows), np.uint8).reshape(-1, 48)

    for _ in range(e2e_warm):
        pump_step()
    barrier()
    sampler2 = ClockSampler(local_rank)
    if rank == 0:
        sampler2.start()
    t0 = time.perf_counter()
    pump_batches = 0
    for _ in range(e2e_steps):
        stub, _dt, pump_batches, tables = pump_step()
        if world > 1:
            all_gather_host_table(pump_table(tables))
    barrier()
    pump_s = time.perf_counter() - t0
    pump_launches = (ctx.launch_count - launches_pump0)
    clocks = None
    if rank == 0:  # clocks sampled inside the timed regions (HBM-resident steps and the headline e2e steps)
        clocks = ClockSampler.summarize(clock_rows + sampler2.halt(), sampler.proc is not None)
    t = torch.tensor([pinned_s, pump_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    pinned_s, pump_s = float(t[0].item()), float(t[1].item())
    pinned_value = world * total_bytes * e2e_steps / GiB / pinned_s
    pump_value = world * total_bytes * e2e_steps / GiB / pump_s
    ptab = requests_table(stub)  # what BlobCreate was told, checked after the timed region
    pump_same = bool(len(ptab) == N_MSG and np.array_equal(ptab[:, :32], sha_dev) and np.array_equal(ptab[:, 32:], md5_dev))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"sha256": sha_dev, "md5": md5_dev, "e2e_pinned_sha256": table.sha256,
                                         "e2e_pinned_md5": table.md5, "e2e_sha256": ptab[:, :32], "e2e_md5": ptab[:, 32:]})

    # ---- CPU baseline (rank 0, N=1): the reference's hashlib path on a bounded sample of the same bytes
    cpu = None
    parity = "tables device==pinned-host: %s; device==map-pump: %s" % ("exact" if same else "MISMATCH",
                                                                        "exact" if pump_same else "MISMATCH")
    if gather_ok is not None:
        parity += "; all-gathered slice == own table: %s" % ("exact" if gather_ok else "MISMATCH")
    if rank == 0 and world == 1:
        os.sched_setaffinity(0, all_cpus)  # the reference's thread pool gets every host core again
        sample_n = min(int(os.environ.get("B200H_CPU_SAMPLE", 16384)), N_MSG)
        sample = payloads[:sample_n]
        from concurrent.futures import ThreadPoolExecutor

        ref_fn, ref_kind = reference_hasher()
        workers = best_pool_workers(sample[:4096])
        t0 = time.perf_counter()
        with ThreadPoolExecutor(max_workers=workers) as ex:
            hashes = list(ex.map(ref_fn, sample))
        pool_s = time.perf_counter() - t0
        serial_n = min(2048, sample_n)
        t0 = time.perf_counter()
        for p_ in sample[:serial_n]:
            ref_fn(p_)
        serial_s = time.perf_counter() - t0
        ok = all(h.sha256_hex() == table.sha256_hex(i) and h.md5_hex() == table.md5_hex(i)
                 for i, h in enumerate(hashes))
        parity += "; GPU vs hashlib on %d payloads: %s" % (sample_n, "exact" if ok else "MISMATCH")
        cpu = {"value": round(sample_n * MSG_BYTES / GiB / pool_s, 3), "unit": "GiB/s", "cores": workers, "kind": ref_kind,
               "sample": f"first {sample_n} of {N_MSG} payloads ({sample_n * MSG_BYTES / GiB:.1f} GiB), hashlib SHA-256+MD5 "
                         f"({'reference get_upload_hashes' if ref_kind == 'reference' else 'get_upload_hashes port'}), "
                         f"ThreadPool({workers})",
               "serial_value": round(serial_n * MSG_BYTES / GiB / serial_s, 3),
               "serial_note": "one thread, as the reference's map pump really runs it (blob_utils.py:345)",
               "host": host_description()}

    if rank == 0:
        peak, peak_src = hbm_peak_gbs()
        kern_avg_ms = kern_ms / max(kern_n, 1)
        achieved = total_bytes / 1e9 / (kern_avg_ms / 1e3) if kern_n else None
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                traffic = json.load(f).get("lane_hash_kernel_dram_bytes_per_launch")
        except Exception:
            pass
        out = {
            "metric": METRIC, "value": round(value, 3), "unit": "GiB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "bytes_per_gpu_per_step": total_bytes, "digests": "sha256+md5 fused",
                       "l2": "inputs (24.4 GiB/GPU) larger than L2, no flush needed", "parallelism": f"shard{world}",
                       "collective": ("nccl all_gather of ONE packed 48-B-row digest table per step on a side stream, "
                                      "double buffered (gather k overlaps hash k+1)") if world > 1 else "none",
                       "host_syncs_in_timed_region": int(plan_syncs), "process_bound_to_gpu_numa_node": bool(numa_bound)},
            "roofline": {"bound": "hbm", "achieved": round(achieved, 1) if achieved else None, "peak": peak, "unit": "GB/s",
                         "frac": round(achieved / peak, 4) if achieved else None, "traffic": traffic,
                         "peak_source": peak_src, "kernel": "lane_hash_kernel<sha256,md5>",
                         "kernel_avg_ms": round(kern_avg_ms, 4), "kernel_launches_timed": kern_n,
                         "int_alu_peak": 1018.0, "int_alu_frac": round(achieved / 1018.0, 4) if achieved else None,
                         "note": "hbm frac per the contract; the binding limit is INT32 issue: 1168 ALU-pipe instr per "
                                 "64 B block at 0.5 warp-instr/clk/SMSP x 592 SMSP x 1.965 GHz = 1018 GB/s (DESIGN.md 5.1)"},
            "cpu_baseline": cpu,
            "e2e": {"value": round(pump_value, 3), "unit": "GiB/s", "h2d_bytes_per_step": total_bytes + 16 * N_MSG,
                    "d2h_bytes_per_step": 56 * N_MSG, "steps": e2e_steps,
                    "api": "parallel_map.InputPreprocessor -> hash_utils.get_upload_hashes_many -> blob_utils._blob_upload_row "
                           "-> parallel_map.InputPumper over 100 000 pageable Python bytes (wire-format inputs, identity "
                           "serializer), null BlobCreate / PUT / FunctionPutInputs"
                           + (" + sharding.all_gather_table (NCCL)" if world > 1 else ""),
                    "hash_batches_per_step": pump_batches,
                    "window_bytes": parallel_map.HASH_WINDOW_BYTES, "windows_in_flight": parallel_map.HASH_WINDOWS_IN_FLIGHT,
                    "gpu_launches": int(pump_launches),
                    "stage_seconds_last_step": getattr(run_map_pump, "last_stats", None),
                    "seconds_last_step": round(_dt, 4)},
            "e2e_pinned": {"value": round(pinned_value, 3), "unit": "GiB/s", "steps": e2e_steps,
                           "api": "batch.hash_table_host on page-locked host memory (one call, 100 000 messages)"
                                  + (" + sharding.all_gather_table (NCCL)" if world > 1 else "")},
            "gpu_launches": int(launches), "clocks": clocks, "parity": parity,
        }
        print(json.dumps(out))
    _backend.set_context(None)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    faulthandler.cancel_dump_traceback_later()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's digest tables as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
