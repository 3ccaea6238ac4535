"""ctypes binding of libb200hash.so (C ABI: include/b200hash.h).

There is deliberately no CPU fallback in this package: if the shared library is missing, or no B200
is visible, every entry point raises ``B200HashError``.  ``build_library()`` (re)builds the .so in-tree
with nvcc for sm_100a (cross-compiles without a GPU).
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import threading
from typing import Sequence

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200H_LIB") or os.path.join(_PKG, "libb200hash.so")  # override: experiments only
CSRC = os.path.join(_PKG, "csrc")

SHA256 = 1
MD5 = 2
TRIM_ZEROS = 4
HEX_OUT = 32  # digest outputs as lowercase ASCII hex rows (64 / 32 chars), formatted on the device
NO_OUTLIERS = 16  # keep every message on the lane kernel: device batches then only enqueue (include/b200hash.h)

#: every symbol include/b200hash.h declares (tests check the .so exports all of them)
ABI_SYMBOLS = (
    "b200h_create", "b200h_destroy", "b200h_last_error", "b200h_version", "b200h_device_count",
    "b200h_host_alloc", "b200h_host_free", "b200h_hash_batch_host", "b200h_hash_batch_device",
    "b200h_hash_fixed_parts", "b200h_stat_files", "b200h_hash_files", "b200h_stream_new", "b200h_stream_update", "b200h_stream_digest",
    "b200h_stream_reset", "b200h_stream_free", "b200h_fill_synth_device", "b200h_launch_count",
    "b200h_profile_enable", "b200h_profile_read", "b200h_dedupe_host", "b200h_dedupe_device",
    "b200h_last_outlier_count", "b200h_hash_batch_device_hl", "b200h_combine_stats", "b200h_plan_sync_count",
    "b200h_stream_copy", "b200h_stream_copy_isa", "b200h_plan_preview", "b200h_pack_preview",
    "b200h_group_create", "b200h_group_destroy", "b200h_group_last_error", "b200h_group_size", "b200h_group_member",
    "b200h_group_hash_batch_host", "b200h_group_hash_files", "b200h_group_last_split", "b200h_group_split_preview",
    "b200h_hash_device_parts", "b200h_group_hash_device_parts",
    "b200h_hash_device_segments", "b200h_group_hash_device_segments", "b200h_segments_preview",
)


class B200HashError(RuntimeError):
    """The CUDA library is missing or a GPU call failed.  Never swallowed, never replaced by CPU work."""


def build_library(force: bool = False, verbose: bool = False) -> str:
    srcs = [os.path.join(CSRC, f) for f in ("b200hash_kernels.cu", "b200hash_dedupe.cu", "b200hash_api.cu",
                                            "b200hash_group.cu", "b200hash_device_parts.cu", "b200hash_device_segments.cu",
                                            "b200hash_internal.h", "b200blob_host.cpp",
                                            "b200pack_copy.cpp", "b200hash_kernels.cuh", "b200pack_team.h")]
    srcs += [os.path.join(os.path.dirname(_PKG), "include", h) for h in ("b200hash.h", "b200blob.h")]
    stale = not os.path.exists(LIB_PATH) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs)
    if force or stale:
        cmd = ["make", "-C", CSRC] + (["-B"] if force else [])
        out = subprocess.run(cmd, capture_output=True, text=True)
        if verbose or out.returncode:
            print(out.stdout, out.stderr)
        if out.returncode:
            raise B200HashError(f"building libb200hash.so failed:\n{out.stdout}\n{out.stderr}")
    return LIB_PATH


_lib = None
_lib_lock = threading.Lock()


def load_library() -> ctypes.CDLL:
    """dlopen libb200hash.so and declare prototypes.  Works without a GPU (symbols only)."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise B200HashError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  modal_client_b200 has no CPU fallback."
            )
        L = ctypes.CDLL(LIB_PATH)
        vp, u64, u32, i32, sz = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int, ctypes.c_size_t
        L.b200h_create.argtypes = [i32, sz, sz, ctypes.POINTER(vp)]
        L.b200h_create.restype = i32
        L.b200h_destroy.argtypes = [vp]
        L.b200h_destroy.restype = None
        L.b200h_last_error.argtypes = [vp]
        L.b200h_last_error.restype = ctypes.c_char_p
        L.b200h_version.argtypes = []
        L.b200h_version.restype = ctypes.c_char_p
        L.b200h_device_count.argtypes = []
        L.b200h_device_count.restype = i32
        L.b200h_host_alloc.argtypes = [vp, sz]
        L.b200h_host_alloc.restype = vp
        L.b200h_host_free.argtypes = [vp, vp]
        L.b200h_host_free.restype = None
        L.b200h_hash_batch_host.argtypes = [vp, vp, vp, vp, u64, u32, vp, vp, vp]
        L.b200h_hash_batch_host.restype = i32
        L.b200h_hash_batch_device.argtypes = [vp, vp, vp, vp, u64, u32, vp, vp, vp, vp]
        L.b200h_hash_batch_device.restype = i32
        L.b200h_hash_batch_device_hl.argtypes = [vp, vp, vp, vp, vp, u64, u32, vp, vp, vp, vp]
        L.b200h_hash_batch_device_hl.restype = i32
        L.b200h_combine_stats.argtypes = [vp, ctypes.POINTER(u64), ctypes.POINTER(u64)]
        L.b200h_combine_stats.restype = i32
        L.b200h_plan_sync_count.argtypes = [vp]
        L.b200h_plan_sync_count.restype = u64
        L.b200h_hash_fixed_parts.argtypes = [vp, vp, u64, u64, u32, vp, vp, vp, vp, ctypes.POINTER(u64)]
        L.b200h_hash_fixed_parts.restype = i32
        L.b200h_stat_files.argtypes = [vp, vp, u64, vp, vp]
        L.b200h_stat_files.restype = i32
        L.b200h_hash_files.argtypes = [vp, vp, u64, vp, u64, u32, vp, vp, vp]
        L.b200h_hash_files.restype = i32
        L.b200h_stream_new.argtypes = [vp, u32, ctypes.POINTER(vp)]
        L.b200h_stream_new.restype = i32
        L.b200h_stream_update.argtypes = [vp, vp, u64]
        L.b200h_stream_update.restype = i32
        L.b200h_stream_digest.argtypes = [vp, vp, vp]
        L.b200h_stream_digest.restype = i32
        L.b200h_stream_reset.argtypes = [vp]
        L.b200h_stream_reset.restype = i32
        L.b200h_stream_free.argtypes = [vp]
        L.b200h_stream_free.restype = None
        L.b200h_fill_synth_device.argtypes = [vp, vp, u64, u64, u64, vp]
        L.b200h_fill_synth_device.restype = i32
        L.b200h_launch_count.argtypes = [vp]
        L.b200h_launch_count.restype = u64
        L.b200h_profile_enable.argtypes = [vp, i32]
        L.b200h_profile_enable.restype = i32
        L.b200h_profile_read.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(u64)]
        L.b200h_profile_read.restype = i32
        L.b200h_last_outlier_count.argtypes = [vp, ctypes.POINTER(u32)]
        L.b200h_last_outlier_count.restype = i32
        L.b200h_dedupe_host.argtypes = [vp, vp, u64, u32, vp, ctypes.POINTER(u64)]
        L.b200h_dedupe_host.restype = i32
        L.b200h_dedupe_device.argtypes = [vp, vp, u64, u32, vp, vp, vp]
        L.b200h_dedupe_device.restype = i32
        L.b200h_stream_copy.argtypes = [vp, vp, sz]
        L.b200h_stream_copy.restype = None
        L.b200h_stream_copy_isa.argtypes = []
        L.b200h_stream_copy_isa.restype = ctypes.c_char_p
        L.b200h_plan_preview.argtypes = [vp, u64, u32, u32, ctypes.POINTER(u32), ctypes.POINTER(u32)]
        L.b200h_plan_preview.restype = i32
        L.b200h_pack_preview.argtypes = [vp, vp, vp, u64, vp, u64, u64, i32, vp]
        L.b200h_pack_preview.restype = i32
        L.b200h_group_create.argtypes = [vp, i32, sz, sz, u64, ctypes.POINTER(vp)]
        L.b200h_group_create.restype = i32
        L.b200h_group_destroy.argtypes = [vp]
        L.b200h_group_destroy.restype = None
        L.b200h_group_last_error.argtypes = [vp]
        L.b200h_group_last_error.restype = ctypes.c_char_p
        L.b200h_group_size.argtypes = [vp]
        L.b200h_group_size.restype = i32
        L.b200h_group_member.argtypes = [vp, i32]
        L.b200h_group_member.restype = vp
        L.b200h_group_hash_batch_host.argtypes = [vp, vp, vp, vp, u64, u32, vp, vp, vp]
        L.b200h_group_hash_batch_host.restype = i32
        L.b200h_group_hash_files.argtypes = [vp, vp, u64, vp, u64, u32, vp, vp, vp]
        L.b200h_group_hash_files.restype = i32
        L.b200h_group_last_split.argtypes = [vp, vp, vp, vp, vp]
        L.b200h_group_last_split.restype = i32
        L.b200h_group_split_preview.argtypes = [vp, u64, i32, u64, vp, ctypes.POINTER(i32)]
        L.b200h_group_split_preview.restype = i32
        L.b200h_hash_device_parts.argtypes = [vp, vp, vp, u64, u64, u32, vp, vp, vp, vp]
        L.b200h_hash_device_parts.restype = i32
        L.b200h_group_hash_device_parts.argtypes = [vp, vp, vp, u64, u64, u32, vp, vp, vp, vp]
        L.b200h_group_hash_device_parts.restype = i32
        L.b200h_hash_device_segments.argtypes = [vp, vp, vp, vp, u64, u64, u32, vp, vp, vp, vp]
        L.b200h_hash_device_segments.restype = i32
        L.b200h_group_hash_device_segments.argtypes = [vp, vp, vp, vp, u64, u64, u32, vp, vp, vp, vp]
        L.b200h_group_hash_device_segments.restype = i32
        L.b200h_segments_preview.argtypes = [vp, vp, u64, u64, u64, ctypes.POINTER(u64), ctypes.POINTER(u64), vp, vp, vp, vp]
        L.b200h_segments_preview.restype = i32
        _lib = L
        return L


# CPython keeps a bytes object's payload at a fixed offset behind its header; taking the address this way
# avoids building one numpy view per payload (3 us each) when a batch holds 10^5..10^6 small payloads.
_BYTES_HDR = bytes.__basicsize__ - 1
_probe = b"b200hash-address-probe"
_FAST_BYTES_ADDR = ctypes.string_at(id(_probe) + _BYTES_HDR, len(_probe)) == _probe


def _np_ptr(a: np.ndarray | None):
    return None if a is None else ctypes.c_void_p(a.ctypes.data)


def plan_preview(lengths, flags: int = SHA256 | MD5, sm_count: int = 148) -> tuple[int, int]:
    """(messages routed to the chain kernel, messages in the long lane queue) for a batch with these lengths on a
    device with ``sm_count`` SMs -- the library's host-side planner (no context, no GPU needed)."""
    L = load_library()
    ln = np.ascontiguousarray(lengths, dtype=np.uint64)
    c, l = ctypes.c_uint32(), ctypes.c_uint32()
    rc = L.b200h_plan_preview(_np_ptr(ln) if ln.size else None, ln.size, flags, sm_count, ctypes.byref(c), ctypes.byref(l))
    if rc != 0:
        raise B200HashError(f"b200h_plan_preview failed ({rc})")
    return c.value, l.value


def group_split_preview(lengths, nmembers: int, min_share_bytes: int = 0) -> tuple[np.ndarray, int]:
    """(owner uint32[n], members used k): how a device group of ``nmembers`` deals a batch with these lengths --
    the library's own split (no group, no GPU).  ``min_share_bytes`` 0 = the library default."""
    L = load_library()
    ln = np.ascontiguousarray(lengths, dtype=np.uint64)
    owner = np.empty(max(ln.size, 1), np.uint32)
    k = ctypes.c_int()
    rc = L.b200h_group_split_preview(_np_ptr(ln), ln.size, nmembers, min_share_bytes, _np_ptr(owner), ctypes.byref(k))
    if rc != 0:
        raise B200HashError(f"b200h_group_split_preview failed ({rc})")
    return owner[: ln.size], k.value


def _segment_table(files) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
    """files: per file a sequence of (address, nbytes) segments -> (addresses, sizes, seg_of[n_files + 1])."""
    counts = [len(f) for f in files]
    seg_of = np.zeros(len(files) + 1, np.uint64)
    np.cumsum(counts, out=seg_of[1:])
    segs = [s for f in files for s in f]
    addr = np.fromiter((int(a) for a, _ in segs), dtype=np.uint64, count=len(segs))
    size = np.fromiter((int(n) for _, n in segs), dtype=np.uint64, count=len(segs))
    return addr, size, seg_of


def _segment_rows(sizes: np.ndarray, seg_of: np.ndarray, part_len: int) -> int:
    csum = np.zeros(sizes.size + 1, np.uint64)
    np.cumsum(sizes, out=csum[1:])
    file_sizes = csum[seg_of[1:].astype(np.int64)] - csum[seg_of[:-1].astype(np.int64)]
    return int(file_sizes.size) if part_len == 0 else int(((file_sizes + np.uint64(part_len - 1)) // np.uint64(part_len)).sum())


def segments_preview(seg_sizes, seg_of, part_len: int, window_bytes: int = 0) -> dict:
    """The row table ``b200h_hash_device_segments`` builds for files made of segments of these sizes (file i = segments
    [seg_of[i], seg_of[i + 1])) -- the library's own code, no context, no GPU.  ``window_bytes`` 0 = the
    B200H_GATHER_BYTES cap.  -> {"gathered": bool[rows], "a": uint64[rows], "b": uint64[rows],
    "window_bytes": uint64[windows]}: an in-place row has a = segment, b = offset in it; a gathered row has a = window,
    b = pieces."""
    L = load_library()
    sz = np.ascontiguousarray(seg_sizes, dtype=np.uint64)
    so = np.ascontiguousarray(seg_of, dtype=np.uint64)
    nf = max(int(so.size) - 1, 0)
    rows, wins = ctypes.c_uint64(), ctypes.c_uint64()
    args = (_np_ptr(sz) if sz.size else None, _np_ptr(so) if so.size else None, nf, part_len, window_bytes)
    rc = L.b200h_segments_preview(*args, ctypes.byref(rows), ctypes.byref(wins), None, None, None, None)
    if rc != 0:
        raise B200HashError(f"b200h_segments_preview failed ({rc})")
    g = np.zeros(max(rows.value, 1), np.uint8)
    a, b = np.zeros(max(rows.value, 1), np.uint64), np.zeros(max(rows.value, 1), np.uint64)
    wb = np.zeros(max(wins.value, 1), np.uint64)
    rc = L.b200h_segments_preview(*args, ctypes.byref(rows), ctypes.byref(wins), _np_ptr(g), _np_ptr(a), _np_ptr(b),
                                  _np_ptr(wb))
    if rc != 0:
        raise B200HashError(f"b200h_segments_preview failed ({rc})")
    r, w = rows.value, wins.value
    return {"gathered": g[:r].astype(bool), "a": a[:r], "b": b[:r], "window_bytes": wb[:w]}


def pack_preview(base, offsets, lengths, threads: int = 16, slot_bytes: int = 256 << 20, dst: np.ndarray | None = None):
    """(packed uint8 buffer, packed offsets uint64[n]): the staging step of the *_host entry points on its own -- the
    messages gathered by the library's packer team into the layout a wave has in HBM.  ``base`` may be None with
    absolute addresses in ``offsets``.  No context, no GPU."""
    L = load_library()
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    ln = np.ascontiguousarray(lengths, dtype=np.uint64)
    need = int(((ln + np.uint64(15)) & ~np.uint64(15)).sum()) if ln.size else 0
    if dst is None:
        dst = np.empty(max(need, 1), np.uint8)
    out = np.empty(max(ln.size, 1), np.uint64)
    bp = None if base is None else ctypes.c_void_p(np.asarray(base).ctypes.data)
    rc = L.b200h_pack_preview(bp, _np_ptr(off), _np_ptr(ln), ln.size, _np_ptr(dst), dst.size, slot_bytes, threads, _np_ptr(out))
    if rc != 0:
        raise B200HashError(f"b200h_pack_preview failed ({rc})")
    return dst, out[: ln.size]


class Context:
    """One libb200hash context bound to one GPU.  Thread-safe (calls serialise inside the library)."""

    def __init__(self, device: int = 0, pinned_bytes: int = 0, device_bytes: int = 0):
        self._L = load_library()
        h = ctypes.c_void_p()
        rc = self._L.b200h_create(device, pinned_bytes, device_bytes, ctypes.byref(h))
        if rc != 0:
            msg = (self._L.b200h_last_error(None) or b"").decode()
            raise B200HashError(f"b200h_create(device={device}) failed ({rc}): {msg}")
        self._h = h
        self.device = device

    # -- plumbing
    def _check(self, rc: int, what: str):
        if rc != 0:
            msg = (self._L.b200h_last_error(self._h) or b"").decode()
            raise B200HashError(f"{what} failed ({rc}): {msg}")

    def close(self):
        if getattr(self, "_h", None):
            self._L.b200h_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launch_count(self) -> int:
        return int(self._L.b200h_launch_count(self._h))

    @property
    def last_outlier_count(self) -> int:
        """Messages of the most recent batch that went to the outlier (chain) kernel; synchronises."""
        c = ctypes.c_uint32()
        self._check(self._L.b200h_last_outlier_count(self._h, ctypes.byref(c)), "b200h_last_outlier_count")
        return int(c.value)

    @property
    def plan_sync_count(self) -> int:
        """Enqueues that had to synchronise their stream to read the planner's outlier count back."""
        return int(self._L.b200h_plan_sync_count(self._h))

    def combine_stats(self) -> tuple[int, int]:
        """(GPU batches issued, caller requests served) by the combining queue of small hash_batch_host calls."""
        g, r = ctypes.c_uint64(), ctypes.c_uint64()
        self._check(self._L.b200h_combine_stats(self._h, ctypes.byref(g), ctypes.byref(r)), "b200h_combine_stats")
        return int(g.value), int(r.value)

    def profile_enable(self, on: bool = True):
        self._check(self._L.b200h_profile_enable(self._h, int(on)), "b200h_profile_enable")

    def profile_read(self) -> tuple[float, int]:
        ms, n = ctypes.c_double(), ctypes.c_uint64()
        self._check(self._L.b200h_profile_read(self._h, ctypes.byref(ms), ctypes.byref(n)), "b200h_profile_read")
        return ms.value, n.value

    # -- pinned host memory
    def host_alloc(self, nbytes: int) -> np.ndarray:
        """uint8[nbytes] view of page-locked memory (freed with host_free)."""
        p = self._L.b200h_host_alloc(self._h, nbytes)
        if not p:
            self._check(-3, "b200h_host_alloc")
        buf = (ctypes.c_uint8 * max(nbytes, 1)).from_address(p)
        arr = np.frombuffer(buf, dtype=np.uint8, count=nbytes)
        arr.flags.writeable = True
        arr_base = arr  # keep ctypes buffer alive via arr.base
        self._pinned = getattr(self, "_pinned", {})
        self._pinned[arr_base.ctypes.data] = p
        return arr

    def host_free(self, arr: np.ndarray):
        p = getattr(self, "_pinned", {}).pop(arr.ctypes.data, None)
        if p:
            self._L.b200h_host_free(self._h, p)

    # -- batch over host memory
    def hash_batch_host(self, base, offsets, lengths, flags: int = SHA256 | MD5, *, out_sha: int = 0, out_md5: int = 0,
                        out_trimmed: int = 0):
        """base: uint8 ndarray / bytes-like / int address / None (absolute addresses in offsets).
        -> (sha[n,32] | None, md5[n,16] | None, trimmed[n])
        out_sha / out_md5 / out_trimmed: raw addresses (host or DEVICE memory, e.g. a CUDA tensor's data_ptr()) that
        receive the columns instead of fresh numpy arrays; the corresponding element of the result is then None."""
        off = np.ascontiguousarray(offsets, dtype=np.uint64)
        ln = np.ascontiguousarray(lengths, dtype=np.uint64)
        n = int(off.size)
        assert ln.size == n
        keep = None
        if base is None:
            bp = None
        elif isinstance(base, int):
            bp = ctypes.c_void_p(base)
        elif isinstance(base, np.ndarray):
            assert base.dtype == np.uint8 and base.flags.c_contiguous
            bp = ctypes.c_void_p(base.ctypes.data)
        else:
            keep = np.frombuffer(base, dtype=np.uint8)
            bp = ctypes.c_void_p(keep.ctypes.data) if keep.size else ctypes.c_void_p(off.ctypes.data)
        wide = 2 if flags & HEX_OUT else 1  # hex rows are twice as wide
        sha = np.empty((n, 32 * wide), np.uint8) if (flags & SHA256 and not out_sha) else None
        md5 = np.empty((n, 16 * wide), np.uint8) if (flags & MD5 and not out_md5) else None
        trimmed = None if out_trimmed else np.empty(n, np.uint64)
        self._batch_host(bp, _np_ptr(off), _np_ptr(ln), n, flags,
                         ctypes.c_void_p(out_sha) if out_sha else _np_ptr(sha),
                         ctypes.c_void_p(out_md5) if out_md5 else _np_ptr(md5),
                         ctypes.c_void_p(out_trimmed) if out_trimmed else _np_ptr(trimmed))
        del keep
        return sha, md5, trimmed

    def _batch_host(self, *args):
        self._check(self._L.b200h_hash_batch_host(self._h, *args), "b200h_hash_batch_host")

    def hash_buffers(self, bufs: Sequence, flags: int = SHA256 | MD5):
        """Hash many separate bytes-like objects without packing them in Python: their addresses go to
        the library as absolute offsets (base=NULL) and it gathers them into its pinned staging ring."""
        n = len(bufs)
        if _FAST_BYTES_ADDR and n and set(map(type, bufs)) == {bytes}:
            # C-level passes only (map + fromiter): this runs on a worker thread that holds the GIL meanwhile
            off = np.fromiter(map(id, bufs), dtype=np.uint64, count=n)
            off += np.uint64(_BYTES_HDR)
            ln = np.fromiter(map(len, bufs), dtype=np.uint64, count=n)
            return self.hash_batch_host(None, off, ln, flags)  # `bufs` keeps the objects alive for the call
        views = [np.frombuffer(b, dtype=np.uint8) for b in bufs]
        off = np.fromiter((v.ctypes.data if v.size else 0 for v in views), dtype=np.uint64, count=n)
        ln = np.fromiter((v.size for v in views), dtype=np.uint64, count=n)
        out = self.hash_batch_host(None, off, ln, flags)
        del views
        return out

    # -- batch over device memory (raw pointers: torch tensors' data_ptr())
    def hash_batch_device(self, d_base: int, d_offsets: int, d_lengths: int, n: int, flags: int, d_sha: int, d_md5: int,
                          d_trimmed: int = 0, stream: int = 0, h_lengths: np.ndarray | None = None):
        """h_lengths: the same lengths as a host uint64 array -- the library then routes outliers without reading
        anything back and the call only enqueues (b200h_hash_batch_device_hl); so does ``flags | NO_OUTLIERS``."""
        if h_lengths is not None:
            hl = np.ascontiguousarray(h_lengths, dtype=np.uint64)
            assert hl.size == n
            rc = self._L.b200h_hash_batch_device_hl(self._h, d_base or None, d_offsets, d_lengths, _np_ptr(hl), n, flags,
                                                    d_sha or None, d_md5 or None, d_trimmed or None, stream or None)
        else:
            rc = self._L.b200h_hash_batch_device(self._h, d_base or None, d_offsets, d_lengths, n, flags, d_sha or None,
                                                 d_md5 or None, d_trimmed or None, stream or None)
        self._check(rc, "b200h_hash_batch_device")

    def hash_fixed_parts(self, data, part_len: int, flags: int = SHA256 | MD5, want_etag: bool = False):
        """-> (sha[np,32]|None, md5[np,16]|None, trimmed[np], etag bytes|None)"""
        if isinstance(data, np.ndarray):
            a = data
        else:
            a = np.frombuffer(data, dtype=np.uint8)
        total = int(a.size)
        nparts = -(-total // part_len) if total else 0
        sha = np.empty((nparts, 32), np.uint8) if flags & SHA256 else None
        md5 = np.empty((nparts, 16), np.uint8) if flags & MD5 else None
        trimmed = np.empty(nparts, np.uint64)
        etag = np.empty(16, np.uint8) if want_etag else None
        got = ctypes.c_uint64()
        bp = ctypes.c_void_p(a.ctypes.data) if total else None
        rc = self._L.b200h_hash_fixed_parts(self._h, bp, total, part_len, flags, _np_ptr(sha), _np_ptr(md5),
                                            _np_ptr(trimmed), _np_ptr(etag), ctypes.byref(got))
        self._check(rc, "b200h_hash_fixed_parts")
        assert got.value == nparts
        return sha, md5, trimmed, (etag.tobytes() if want_etag else None)

    # -- buffers already in device memory, split into parts (b200h_hash_device_parts)
    def hash_device_parts(self, ptrs, sizes, part_len: int, flags: int = SHA256 | MD5, want_etag: bool = False, *,
                          out_sha: int = 0, out_md5: int = 0, out_trimmed: int = 0, out_etag: int = 0):
        """ptrs: device addresses (e.g. CUDA tensors' data_ptr()) of n buffers on this context's device, sizes their
        byte counts.  -> (sha[rows,32]|None, md5[rows,16]|None, trimmed[rows], etags[n,16]|None); rows = n (part_len 0)
        or the buffer-major list of ceil(size/part_len) parts.  out_*: raw addresses (host or device memory) that
        receive a column instead of a fresh numpy array; that element of the result is then None."""
        p = np.ascontiguousarray(ptrs, dtype=np.uint64)
        sz = np.ascontiguousarray(sizes, dtype=np.uint64)
        n = int(p.size)
        assert sz.size == n
        rows = n if part_len == 0 else int(((sz + np.uint64(part_len - 1)) // np.uint64(part_len)).sum())
        wide = 2 if flags & HEX_OUT else 1
        sha = np.empty((rows, 32 * wide), np.uint8) if (flags & SHA256 and not out_sha) else None
        md5 = np.empty((rows, 16 * wide), np.uint8) if (flags & MD5 and not out_md5) else None
        trimmed = None if out_trimmed else np.empty(rows, np.uint64)
        etag = np.empty((n, 16), np.uint8) if (want_etag and not out_etag) else None
        self._device_parts(_np_ptr(p) if n else None, _np_ptr(sz) if n else None, n, part_len, flags,
                           ctypes.c_void_p(out_sha) if out_sha else _np_ptr(sha),
                           ctypes.c_void_p(out_md5) if out_md5 else _np_ptr(md5),
                           ctypes.c_void_p(out_trimmed) if out_trimmed else _np_ptr(trimmed),
                           ctypes.c_void_p(out_etag) if out_etag else _np_ptr(etag))
        return sha, md5, trimmed, etag

    def _device_parts(self, *args):
        self._check(self._L.b200h_hash_device_parts(self._h, *args), "b200h_hash_device_parts")

    # -- files made of device segments, e.g. a safetensors header plus its tensors (b200h_hash_device_segments)
    def hash_device_segments(self, files, part_len: int, flags: int = SHA256 | MD5, want_etag: bool = False, *,
                             out_sha: int = 0, out_md5: int = 0, out_trimmed: int = 0, out_etag: int = 0):
        """files: per file, a sequence of ``(device address, nbytes)`` segments on this context's device; the file is
        their concatenation.  Rows and results exactly as ``hash_device_parts`` with one buffer per file holding those
        bytes: -> (sha[rows,32]|None, md5[rows,16]|None, trimmed[rows], etags[n,16]|None).  Parts that straddle
        segments are gathered into scratch on the device first (B200H_GATHER_BYTES caps it)."""
        addr, sz, seg_of = _segment_table(files)
        n = len(files)
        rows = _segment_rows(sz, seg_of, part_len)
        wide = 2 if flags & HEX_OUT else 1
        sha = np.empty((rows, 32 * wide), np.uint8) if (flags & SHA256 and not out_sha) else None
        md5 = np.empty((rows, 16 * wide), np.uint8) if (flags & MD5 and not out_md5) else None
        trimmed = None if out_trimmed else np.empty(rows, np.uint64)
        etag = np.empty((n, 16), np.uint8) if (want_etag and not out_etag) else None
        self._device_segments(_np_ptr(addr) if addr.size else None, _np_ptr(sz) if sz.size else None,
                              _np_ptr(seg_of), n, part_len, flags,
                              ctypes.c_void_p(out_sha) if out_sha else _np_ptr(sha),
                              ctypes.c_void_p(out_md5) if out_md5 else _np_ptr(md5),
                              ctypes.c_void_p(out_trimmed) if out_trimmed else _np_ptr(trimmed),
                              ctypes.c_void_p(out_etag) if out_etag else _np_ptr(etag))
        return sha, md5, trimmed, etag

    def _device_segments(self, *args):
        self._check(self._L.b200h_hash_device_segments(self._h, *args), "b200h_hash_device_segments")

    # -- files: stat + read + hash entirely inside the library (native reader threads, no mmap / Python I/O)
    @staticmethod
    def _c_paths(paths):
        # callers that make several calls over one tree pass the paths already encoded (bytes) to pay fsencode once
        enc = paths if (len(paths) and type(paths[0]) is bytes) else [os.fsencode(p) for p in paths]
        return enc, (ctypes.c_char_p * len(enc))(*enc)

    def stat_files(self, paths) -> tuple[np.ndarray, np.ndarray]:
        """-> (sizes uint64[n], permission bits uint32[n]); raises for missing / non-regular files."""
        keep, arr = self._c_paths(paths)
        n = len(keep)
        sizes, modes = np.zeros(n, np.uint64), np.zeros(n, np.uint32)
        self._check(self._L.b200h_stat_files(self._h, arr, n, _np_ptr(sizes), _np_ptr(modes)), "b200h_stat_files")
        return sizes, modes

    def hash_files(self, paths, sizes, part_len: int = 0, flags: int = SHA256 | MD5):
        """-> (sha[rows,32]|None, md5[rows,16]|None, trimmed[rows]); rows = n files (part_len 0) or the
        file-major list of ceil(size/part_len) parts."""
        keep, arr = self._c_paths(paths)
        sizes = np.ascontiguousarray(sizes, dtype=np.uint64)
        n = len(keep)
        rows = n if part_len == 0 else int(((sizes + np.uint64(part_len - 1)) // np.uint64(part_len)).sum())
        wide = 2 if flags & HEX_OUT else 1
        sha = np.empty((rows, 32 * wide), np.uint8) if flags & SHA256 else None
        md5 = np.empty((rows, 16 * wide), np.uint8) if flags & MD5 else None
        trimmed = np.empty(rows, np.uint64)
        self._files(arr, n, _np_ptr(sizes), part_len, flags, _np_ptr(sha), _np_ptr(md5), _np_ptr(trimmed))
        return sha, md5, trimmed

    def _files(self, *args):
        self._check(self._L.b200h_hash_files(self._h, *args), "b200h_hash_files")

    # -- dedupe of a digest table (first occurrence of every content)
    def dedupe(self, keys: np.ndarray) -> tuple[np.ndarray, int]:
        """keys: uint8[n, 32] (SHA-256 rows) or uint8[n, 16] (MD5 rows) on the host.
        -> (first uint32[n] with first[i] = smallest j such that keys[j] == keys[i], number of distinct rows)"""
        k = np.ascontiguousarray(keys, dtype=np.uint8)
        if k.ndim != 2 or k.shape[1] not in (16, 32):
            raise ValueError("keys must be uint8[n, 32] or uint8[n, 16]")
        n = int(k.shape[0])
        first = np.empty(n, np.uint32)
        nd = ctypes.c_uint64()
        rc = self._L.b200h_dedupe_host(self._h, _np_ptr(k) if n else None, n, k.shape[1], _np_ptr(first) if n else None,
                                       ctypes.byref(nd))
        self._check(rc, "b200h_dedupe_host")
        return first, int(nd.value)

    def dedupe_device(self, d_keys: int, n: int, key_bytes: int, d_first: int, d_ndistinct: int = 0, stream: int = 0):
        rc = self._L.b200h_dedupe_device(self._h, d_keys or None, n, key_bytes, d_first or None, d_ndistinct or None,
                                         stream or None)
        self._check(rc, "b200h_dedupe_device")

    def fill_synth_device(self, d_ptr: int, nbytes: int, seed: int, start: int = 0, stream: int = 0):
        self._check(self._L.b200h_fill_synth_device(self._h, d_ptr, nbytes, seed, start, stream or None),
                    "b200h_fill_synth_device")

    def stream(self, flags: int = SHA256 | MD5) -> "DigestStream":
        return DigestStream(self, flags)


class DeviceGroup(Context):
    """One context per listed device, driven as one (include/b200hash.h, device groups).  ``hash_batch_host`` (and so
    ``hash_buffers``) and ``hash_files`` deal each batch over the members by bytes and hash the shares at the same time;
    ``hash_device_parts`` / ``hash_device_segments`` deal the parts of device buffers (files) over the members on each
    buffer's (file's) device;
    every other method runs on the home member (``devices[0]``), whose handle this object carries as a Context.
    ``devices=None`` means every visible device; a device may repeat.  ``min_share_bytes`` 0 = the library default."""

    def __init__(self, devices: Sequence[int] | None = None, pinned_bytes: int = 0, device_bytes: int = 0,
                 min_share_bytes: int = 0):
        self._L = load_library()
        if devices is None:
            devices = list(range(self._L.b200h_device_count()))
        devs = (ctypes.c_int * max(len(devices), 1))(*devices)
        g = ctypes.c_void_p()
        rc = self._L.b200h_group_create(devs, len(devices), pinned_bytes, device_bytes, min_share_bytes, ctypes.byref(g))
        if rc != 0:
            msg = (self._L.b200h_group_last_error(None) or b"").decode()
            raise B200HashError(f"b200h_group_create(devices={list(devices)}) failed ({rc}): {msg}")
        self._g = g
        self.devices = [int(d) for d in devices]
        self._members = [ctypes.c_void_p(self._L.b200h_group_member(g, i)) for i in range(len(self.devices))]
        self._h = self._members[0]  # borrowed: the group owns it
        self.device = self.devices[0]

    def _gcheck(self, rc: int, what: str):
        if rc != 0:
            msg = (self._L.b200h_group_last_error(self._g) or b"").decode()
            raise B200HashError(f"{what} failed ({rc}): {msg}")

    def _batch_host(self, *args):
        self._gcheck(self._L.b200h_group_hash_batch_host(self._g, *args), "b200h_group_hash_batch_host")

    def _files(self, *args):
        self._gcheck(self._L.b200h_group_hash_files(self._g, *args), "b200h_group_hash_files")

    def _device_parts(self, *args):
        # every buffer is hashed by the members on the device that holds it
        self._gcheck(self._L.b200h_group_hash_device_parts(self._g, *args), "b200h_group_hash_device_parts")

    def _device_segments(self, *args):
        # every file is hashed by the members on the device that holds its segments
        self._gcheck(self._L.b200h_group_hash_device_segments(self._g, *args), "b200h_group_hash_device_segments")

    def close(self):
        if getattr(self, "_g", None):
            self._L.b200h_group_destroy(self._g)
        self._g = None
        self._h = None  # never destroyed on its own: it belonged to the group

    @property
    def launch_count(self) -> int:
        return sum(int(self._L.b200h_launch_count(h)) for h in self._members) if getattr(self, "_g", None) else 0

    def last_split(self) -> list[dict]:
        """Per member, what the last batch call did: device, messages, payload bytes, bytes that went through the
        member's pinned staging ring (0 = DMAed straight from page-locked memory), wall ms inside the member."""
        m = len(self.devices)
        msgs, nbytes, staged = np.zeros(m, np.uint64), np.zeros(m, np.uint64), np.zeros(m, np.uint64)
        ms = np.zeros(m, np.float64)
        self._gcheck(self._L.b200h_group_last_split(self._g, _np_ptr(msgs), _np_ptr(nbytes), _np_ptr(staged), _np_ptr(ms)),
                     "b200h_group_last_split")
        return [{"device": d, "messages": int(a), "bytes": int(b), "staged_bytes": int(s), "busy_ms": float(t)}
                for d, a, b, s, t in zip(self.devices, msgs, nbytes, staged, ms)]


class DigestStream:
    """hashlib-object shaped incremental digest (update / digest / reset); state lives on the GPU."""

    def __init__(self, ctx: Context, flags: int):
        self._ctx = ctx
        self._flags = flags
        h = ctypes.c_void_p()
        ctx._check(ctx._L.b200h_stream_new(ctx._h, flags, ctypes.byref(h)), "b200h_stream_new")
        self._h = h

    def update(self, data) -> None:
        v = np.frombuffer(data, dtype=np.uint8)
        if v.size:
            self._ctx._check(self._ctx._L.b200h_stream_update(self._h, ctypes.c_void_p(v.ctypes.data), v.size),
                             "b200h_stream_update")

    def digests(self) -> tuple[bytes | None, bytes | None]:
        sha = np.empty(32, np.uint8)
        md5 = np.empty(16, np.uint8)
        self._ctx._check(self._ctx._L.b200h_stream_digest(self._h, _np_ptr(sha), _np_ptr(md5)), "b200h_stream_digest")
        return (sha.tobytes() if self._flags & SHA256 else None, md5.tobytes() if self._flags & MD5 else None)

    def reset(self) -> None:
        self._ctx._check(self._ctx._L.b200h_stream_reset(self._h), "b200h_stream_reset")

    def close(self):
        if getattr(self, "_h", None) and getattr(self._ctx, "_h", None):
            self._ctx._L.b200h_stream_free(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default: dict[int, Context] = {}
_default_lock = threading.Lock()


def default_context(device: int | None = None) -> Context:
    """Process-wide context per device (LOCAL_RANK picks the device under torchrun)."""
    if device is None:
        device = int(os.environ.get("B200H_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    with _default_lock:
        ctx = _default.get(device)
        if ctx is None:
            ctx = _default[device] = Context(device)
        return ctx
