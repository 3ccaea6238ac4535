"""Batch front door of the B200 hash path: many independent messages in, one digest table out.

This is the call the accelerated callers make (map input pump, Volume.batch_upload v1/v2, multipart
parts): the reference hashes one payload / file / block at a time with hashlib
(py/modal/_utils/blob_utils.py:345,459-474,640-664); here the whole set goes to the GPU in one call.
"""
from __future__ import annotations

import base64
import dataclasses
from typing import Sequence

import numpy as np

from . import _lib
from ._backend import get_context
from ._lib import MD5, SHA256, TRIM_ZEROS, Context, default_context


@dataclasses.dataclass
class DigestTable:
    """Fixed-width digest table, row i = message i.  ``sha256``: uint8[n,32] or None; ``md5``:
    uint8[n,16] or None; ``hashed_len``: uint64[n] bytes actually hashed (differs from the input
    length only with zero trimming)."""

    sha256: np.ndarray | None
    md5: np.ndarray | None
    hashed_len: np.ndarray

    def __len__(self) -> int:
        return int(self.hashed_len.size)

    def sha256_hex(self, i: int) -> str:
        return self.sha256[i].tobytes().hex()

    def md5_hex(self, i: int) -> str:
        return self.md5[i].tobytes().hex()

    def sha256_base64(self, i: int) -> str:
        return base64.b64encode(self.sha256[i].tobytes()).decode("ascii")

    def md5_base64(self, i: int) -> str:
        return base64.b64encode(self.md5[i].tobytes()).decode("ascii")

    def first_occurrence(self, ctx: Context | None = None) -> tuple[np.ndarray, int]:
        """In-batch dedupe on the GPU: ``first[i]`` = smallest row index carrying the same SHA-256 (MD5 when the
        table has no SHA-256 column) as row i, and the number of distinct contents.  What ``_Mount._load_mount``
        does one file at a time with its ``accounted_hashes`` set (py/modal/mount.py:498,518-534)."""
        keys = self.sha256 if self.sha256 is not None else self.md5
        if keys is None:
            raise ValueError("the table holds no digests")
        return (ctx or get_context()).dedupe(keys)

    def packed(self) -> np.ndarray:
        """uint8[n,48]: sha256 || md5 per row -- the table the ranks all-gather."""
        n = len(self)
        out = np.zeros((n, 48), np.uint8)
        if self.sha256 is not None:
            out[:, :32] = self.sha256
        if self.md5 is not None:
            out[:, 32:] = self.md5
        return out


def hash_table_host(base, offsets, lengths, *, sha256: bool = True, md5: bool = True, trim_zeros: bool = False,
                    ctx: Context | None = None) -> DigestTable:
    """Hash messages ``base[offsets[i] : offsets[i]+lengths[i]]`` that live in host memory
    (page-locked memory from ``Context.host_alloc`` is DMA'd directly; anything else is staged)."""
    ctx = ctx or get_context()
    flags = (SHA256 if sha256 else 0) | (MD5 if md5 else 0) | (TRIM_ZEROS if trim_zeros else 0)
    s, m, t = ctx.hash_batch_host(base, offsets, lengths, flags)
    return DigestTable(s, m, t)


def hash_table_buffers(bufs: Sequence, *, sha256: bool = True, md5: bool = True, ctx: Context | None = None) -> DigestTable:
    """Hash many separate bytes-like objects (e.g. serialized map inputs) in one GPU batch."""
    ctx = ctx or get_context()
    flags = (SHA256 if sha256 else 0) | (MD5 if md5 else 0)
    s, m, t = ctx.hash_buffers(bufs, flags)
    return DigestTable(s, m, t)


def hash_table_tensors(tensors: Sequence, *, sha256: bool = True, md5: bool = True, ctx: Context | None = None):
    """Digest the raw bytes of CUDA tensors where they are (no host round trip): message i is the storage of
    contiguous tensor i.  Returns ``(sha uint8[n,32] | None, md5 uint8[n,16] | None)`` as CUDA tensors on the
    same device, ordered on the current torch stream.  This is the entry point for map inputs that are already
    tensors in HBM (SURVEY 8f-4): nothing is pickled or copied before hashing."""
    import torch

    ctx = ctx or get_context()
    n = len(tensors)
    dev = tensors[0].device if n else torch.device("cuda", ctx.device)
    for t in tensors:
        if not (t.is_cuda and t.is_contiguous() and t.device == dev):
            raise ValueError("hash_table_tensors needs contiguous CUDA tensors on one device")
    if n and dev.index is not None and getattr(ctx, "device", dev.index) not in (dev.index, -1):
        raise ValueError(f"tensors live on cuda:{dev.index} but the context is bound to cuda:{ctx.device}")
    addr = torch.tensor([t.data_ptr() for t in tensors], dtype=torch.int64)
    size = torch.tensor([t.numel() * t.element_size() for t in tensors], dtype=torch.int64)
    d_addr, d_size = addr.to(dev, non_blocking=False), size.to(dev, non_blocking=False)
    d_sha = torch.empty((n, 32), dtype=torch.uint8, device=dev) if sha256 else None
    d_md5 = torch.empty((n, 16), dtype=torch.uint8, device=dev) if md5 else None
    flags = (SHA256 if sha256 else 0) | (MD5 if md5 else 0)
    stream = torch.cuda.current_stream(dev)
    # absolute device addresses as offsets from a NULL base
    # the sizes are known here, so the library routes outliers on the host: the call only enqueues
    ctx.hash_batch_device(0, d_addr.data_ptr(), d_size.data_ptr(), n, flags, d_sha.data_ptr() if sha256 else 0,
                          d_md5.data_ptr() if md5 else 0, 0, stream.cuda_stream,
                          h_lengths=size.numpy().astype(np.uint64))
    # the library launched on this stream (or, for the legacy default stream, on its own): make the result
    # visible to the caller's stream before the offset tensors can be freed
    if stream.cuda_stream == 0:
        torch.cuda.synchronize(dev)
    else:
        d_addr.record_stream(stream)
        d_size.record_stream(stream)
    return d_sha, d_md5


def ready_event(tensor):
    """A CUDA event recorded on ``tensor``'s current torch stream: once it has completed, every write queued so far on
    that stream is visible to the library's own streams.  Record it when a tensor is queued, wait on it before
    hashing -- a wait on one event, not a device-wide synchronisation."""
    import torch

    ev = torch.cuda.Event()
    ev.record(torch.cuda.current_stream(tensor.device))
    return ev


def hash_blocks_tensors(tensors: Sequence, part_len: int, *, sha256: bool = True, md5: bool = False,
                        trim_zeros: bool = False, ctx: Context | None = None, ready: Sequence | None = None) -> DigestTable:
    """Digest the raw bytes (``numel * element_size`` from ``data_ptr()``) of contiguous CUDA tensors of any dtype where
    they are, split into ``part_len``-byte parts (``part_len`` 0: one row per tensor): ``b200h_hash_device_parts``.
    Rows are tensor-major, ceil(nbytes / part_len) per tensor; with ``trim_zeros`` these are the volumefs2 blocks of the
    tensor's bytes.  ``ready``: events from ``ready_event`` recorded when the tensors were queued (default: recorded
    now); the call waits on them, so work already queued on each tensor's stream is part of what is hashed.  A device
    group hashes every tensor on the members on its device."""
    ctx = ctx or get_context()
    for t in tensors:
        if not (getattr(t, "is_cuda", False) and t.is_contiguous()):
            raise ValueError("hash_blocks_tensors needs contiguous CUDA tensors")
    for ev in (ready if ready is not None else [ready_event(t) for t in tensors]):
        ev.synchronize()
    flags = (SHA256 if sha256 else 0) | (MD5 if md5 else 0) | (TRIM_ZEROS if trim_zeros else 0)
    s, m, t, _ = ctx.hash_device_parts([x.data_ptr() for x in tensors], [x.numel() * x.element_size() for x in tensors],
                                       part_len, flags)
    return DigestTable(s, m, t)


def hash_blocks_segments(files: Sequence[Sequence], part_len: int, *, sha256: bool = True, md5: bool = False,
                         trim_zeros: bool = False, ctx: Context | None = None, ready: Sequence | None = None) -> DigestTable:
    """``hash_blocks_tensors`` for files made of several tensors: file i is the raw bytes of the contiguous CUDA tensors
    ``files[i]`` back to back (a safetensors file is its header as a uint8 tensor, then its tensors).  The rows are
    exactly those of ``hash_blocks_tensors`` over one tensor per file holding the concatenated bytes, without building
    it: ``b200h_hash_device_segments`` gathers only the parts that straddle two tensors.  ``ready`` as for
    ``hash_blocks_tensors`` (default: one event per tensor, recorded now)."""
    ctx = ctx or get_context()
    for f in files:
        for t in f:
            if not (getattr(t, "is_cuda", False) and t.is_contiguous()):
                raise ValueError("hash_blocks_segments needs contiguous CUDA tensors")
    for ev in (ready if ready is not None else [ready_event(t) for f in files for t in f]):
        ev.synchronize()
    flags = (SHA256 if sha256 else 0) | (MD5 if md5 else 0) | (TRIM_ZEROS if trim_zeros else 0)
    s, m, t, _ = ctx.hash_device_segments([[(x.data_ptr(), x.numel() * x.element_size()) for x in f] for f in files],
                                          part_len, flags)
    return DigestTable(s, m, t)


__all__ = ["DigestTable", "hash_table_host", "hash_table_buffers", "hash_table_tensors", "hash_blocks_tensors",
           "hash_blocks_segments", "ready_event", "Context", "default_context", "_lib"]
