"""Drop-in for the hashing / chunking half of the reference's ``modal/_utils/blob_utils.py``.

Same public names, size classes, thresholds and integrity checks as the reference
(py/modal/_utils/blob_utils.py), with every digest produced by libb200hash on the B200:

=============================  ===========================================================================
reference (file:line)          here
=============================  ===========================================================================
``_get_file_upload_spec``      same semantics per file; ``get_file_upload_specs`` hashes a whole *list* of
  :446-487                     files in one GPU batch (what ``Volume.batch_upload`` v1 / ``Mount`` need)
``_gather_blocks`` … :622-705  one ``b200h_hash_fixed_parts(TRIM_ZEROS)`` call per file: the zero-trim scan and
                               the SHA-256 of every 8 MiB block run on the device, the file is read ONCE
``perform_multipart_upload``   all part MD5s + the md5-of-md5s ETag come from one GPU call before any byte is
  :159-234                     sent; the per-chunk CPU re-hash inside the payload disappears
``_blob_upload`` … :271-374    unchanged control flow (BlobCreate -> single PUT | multipart), GPU digests
=============================  ===========================================================================

Module constants stay patchable module globals read at call time, because the reference's tests patch
them by dotted name (py/test/blob_test.py:57, py/test/volume_test.py:489).
"""
from __future__ import annotations

import asyncio
import dataclasses
import functools
import gc
import io
import json
import mmap
import os
import platform
import threading
import time
from collections.abc import Callable, Sequence
from contextlib import AbstractContextManager, asynccontextmanager, contextmanager
from io import BytesIO, FileIO
from pathlib import Path, PurePosixPath
from typing import Any, BinaryIO, ContextManager
from urllib.parse import urlparse

import numpy as np

from . import _lib, _wire, hash_utils
from ._backend import get_context
from ._logging import logger
from ._wire import BlobCreateRequest
from .async_utils import asyncnullcontext, bounded_map, gather_cancel_on_error, retry
from .bytes_io_segment_payload import BytesIOSegmentPayload, KnownBytesBody
from .exception import ExecutionError
from .hash_utils import UploadHashes, get_upload_hashes
from .http_utils import ClientSessionRegistry

MAX_OBJECT_SIZE_BYTES = 2 * 1024 * 1024  # function inputs/outputs above this go to blob storage
MAX_ASYNC_OBJECT_SIZE_BYTES = 8 * 1024  # ... for async (spawn) calls
LARGE_FILE_LIMIT = 4 * 1024 * 1024  # files at least this big are uploaded as blobs
BLOB_MAX_PARALLELISM = 20
DEFAULT_SEGMENT_CHUNK_SIZE = 2**24
MULTIPART_UPLOAD_THRESHOLD = 1024**3  # above this no whole-file MD5 is computed (placeholder instead)
MULTIPART_INFLIGHT_BYTES_MAX = 2 * 1024**3
MULTIPART_INFLIGHT_BYTES_MIN = 256 * 1024 * 1024
MULTIPART_INFLIGHT_MEMORY_FRACTION = 0.5
BLOCK_SIZE: int = 8 * 1024 * 1024  # volumefs2 block
SMALL_FILE_INLINE_LIMIT = 256 * 1024  # below this the content is cached in the spec
_MD5_PLACEHOLDER = "baadbaad" * 4


# --------------------------------------------------------------------------------------- byte budget


class _ByteBudget:
    """Caps the bytes in flight across concurrent part uploads (reference :66-91)."""

    def __init__(self, total: int):
        self._total = total
        self._available = total
        self._cond = asyncio.Condition()

    @classmethod
    def from_system_memory(cls) -> "_ByteBudget":
        return cls(_get_multipart_inflight_budget())

    @asynccontextmanager
    async def acquire(self, n: int):
        async with self._cond:
            # a request larger than the whole budget is admitted once nothing else is in flight
            await self._cond.wait_for(lambda: self._available >= min(n, self._total))
            self._available -= n
        try:
            yield
        finally:
            async with self._cond:
                self._available += n
                self._cond.notify_all()


def _get_multipart_inflight_budget() -> int:
    try:
        import psutil

        available = psutil.virtual_memory().available
    except Exception:
        try:
            available = os.sysconf("SC_AVPHYS_PAGES") * os.sysconf("SC_PAGE_SIZE")
        except (AttributeError, ValueError, OSError):
            return MULTIPART_INFLIGHT_BYTES_MIN
    want = int(available * MULTIPART_INFLIGHT_MEMORY_FRACTION)
    return min(max(want, MULTIPART_INFLIGHT_BYTES_MIN), MULTIPART_INFLIGHT_BYTES_MAX)


# ------------------------------------------------------------------------------ views of file contents


@contextmanager
def _readonly_view(fp: BinaryIO):
    """uint8 ndarray over the whole content of ``fp`` without copying when possible:
    BytesIO -> its buffer; real file -> a private read-only mmap; anything else -> one read()."""
    if isinstance(fp, BytesIO):
        buf = fp.getbuffer()
        arr = np.frombuffer(buf, dtype=np.uint8)
        try:
            yield arr
        finally:
            del arr
            buf.release()  # callers drop their references first (see _with_view)
        return
    try:
        fd = fp.fileno()
        size = os.fstat(fd).st_size
    except (OSError, AttributeError, ValueError):
        fd, size = None, 0
    if fd is not None and size > 0:
        mm = mmap.mmap(fd, 0, access=mmap.ACCESS_READ)
        try:
            arr = np.frombuffer(mm, dtype=np.uint8)
            yield arr
            del arr
        finally:
            mm.close()
        return
    pos = fp.tell()
    fp.seek(0)
    data = fp.read()
    fp.seek(pos)
    yield np.frombuffer(data, dtype=np.uint8)


def _with_view(fp: BinaryIO, fn):
    """fn(view) over the content of ``fp``; the view is dropped before the underlying buffer is released,
    so BytesIO objects stay closable/resizable afterwards."""
    with _readonly_view(fp) as view:
        try:
            return fn(view)
        finally:
            del view


# ------------------------------------------------------------------------------------ single-part PUT


@retry(n_attempts=3, base_delay=0.3, attempt_timeout=None)
async def _upload_to_s3_url(
    upload_url,
    payload,
    content_md5_b64: str | None = None,
    content_type: str | None = "application/octet-stream",
) -> str:
    """PUT one payload; returns the object's ETag after checking it against the local MD5
    (reference :110-156: S3's single-part ETag is the quoted MD5 hex of the body)."""
    with payload.reset_on_error():
        body = payload.as_payload() if isinstance(payload, KnownBytesBody) else payload
        headers = {}
        if content_md5_b64 and use_md5(upload_url):
            headers["Content-MD5"] = content_md5_b64
        if content_type:
            headers["Content-Type"] = content_type
        async with ClientSessionRegistry.get_session().put(
            upload_url, data=body, headers=headers, skip_auto_headers=["content-type"] if content_type is None else []
        ) as resp:
            if resp.status == 503:  # S3 SlowDown
                logger.debug("Received SlowDown signal from S3, sleeping for 1 second before retrying.")
                await asyncio.sleep(1)
            if resp.status != 200:
                try:
                    text = await resp.text()
                except Exception:
                    text = "<no body>"
                raise ExecutionError(f"Put to url {upload_url} failed with status {resp.status}: {text}")
            etag = resp.headers["ETag"].strip()
            if etag[:2] in ("W/", "w/"):
                etag = etag[2:]
            if len(etag) >= 2 and etag[0] == '"' and etag[-1] == '"':
                etag = etag[1:-1]
            local_md5_hex = payload.md5_checksum().hexdigest()
            if local_md5_hex != etag:
                raise ExecutionError(f"Local data and remote data checksum mismatch ({local_md5_hex} vs {etag})")
            return etag


# ------------------------------------------------------------------------------------------ multipart


def multipart_part_digests(data, part_length: int) -> tuple[list[bytes], str]:
    """All part MD5s of ``data`` split every ``part_length`` bytes plus the expected combined ETag
    ``md5(md5_0 || md5_1 || ...).hex() + "-<n>"`` -- one GPU call (reference :194-219 does n hashlib passes
    on executor threads and one more on the loop thread)."""
    _, md5, _, etag = get_context().hash_fixed_parts(data, part_length, _lib.MD5, want_etag=True)
    parts = [md5[i].tobytes() for i in range(len(md5))]
    return parts, f"{etag.hex()}-{len(parts)}"


async def perform_multipart_upload(
    data_file: BinaryIO | BytesIO | FileIO,
    *,
    content_length: int,
    max_part_size: int,
    part_urls: list[str],
    completion_url: str,
    upload_chunk_size: int = DEFAULT_SEGMENT_CHUNK_SIZE,
    progress_report_cb: Callable | None = None,
    byte_budget: _ByteBudget | None = None,
) -> None:
    # 1. hash every part on the GPU before sending anything
    on_device = isinstance(data_file, (DeviceBufferReader, DeviceSegmentsReader))
    start_pos = data_file.tell() if isinstance(data_file, (BytesIO, DeviceBufferReader, DeviceSegmentsReader)) else 0
    if on_device:  # tensors' bytes: the parts are hashed where they are, nothing is copied to the host for it
        part_md5, expected_etag = await asyncio.to_thread(data_file.part_digests, start_pos, content_length, max_part_size)
    else:
        part_md5, expected_etag = await asyncio.to_thread(
            _with_view, data_file,
            lambda whole: multipart_part_digests(whole[start_pos : start_pos + content_length], max_part_size))
    if len(part_md5) > len(part_urls):
        raise ExecutionError(f"{len(part_md5)} parts but only {len(part_urls)} part URLs")

    # 2. one independent reader per part (no shared file position)
    if isinstance(data_file, BytesIO):
        view = data_file.getbuffer()
        readers: list[BinaryIO] = [BytesIO(view) for _ in part_urls]
        for rdr in readers:
            rdr.seek(start_pos)
    elif on_device:
        readers = [data_file.clone() for _ in part_urls]
        for rdr in readers:
            rdr.seek(start_pos)
    else:
        readers = [open(data_file.name, "rb") for _ in part_urls]

    async def send(url: str, payload) -> str:
        async with byte_budget.acquire(4 * payload.chunk_size) if byte_budget else asyncnullcontext():
            return await _upload_to_s3_url(url, payload=payload, content_type=None)

    jobs, offset, left = [], 0, content_length
    for i, (rdr, url) in enumerate(zip(readers, part_urls)):
        n = min(left, max_part_size)
        payload = BytesIOSegmentPayload(rdr, segment_start=offset, segment_length=n, chunk_size=upload_chunk_size,
                                        progress_report_cb=progress_report_cb,
                                        md5_digest=part_md5[i] if i < len(part_md5) else None)
        jobs.append(send(url, payload))
        offset += n
        left -= n
    try:
        part_etags = await gather_cancel_on_error(*jobs)
    finally:
        if not isinstance(data_file, BytesIO):
            for rdr in readers:
                rdr.close()

    xml = ["<CompleteMultipartUpload>"]
    for number, etag in enumerate(part_etags, 1):
        xml.append(f'<Part>\n<PartNumber>{number}</PartNumber>\n<ETag>"{etag}"</ETag>\n</Part>')
    xml.append("</CompleteMultipartUpload>")
    # each part's ETag was already checked against the GPU digest in _upload_to_s3_url, so the device-side
    # md5-of-md5s is exactly what the store must report for the assembled object
    if len(part_md5) != len(part_etags):
        expected_etag = _etag_from_part_hexes(part_etags)
    resp = await ClientSessionRegistry.get_session().post(
        completion_url, data="\n".join(xml).encode("ascii"), skip_auto_headers=["content-type"]
    )
    if resp.status != 200:
        try:
            msg = await resp.text()
        except Exception:
            msg = "<no body>"
        raise ExecutionError(f"Error when completing multipart upload: {resp.status}\n{msg}")
    body_text = await resp.text()
    if expected_etag not in body_text:
        raise ExecutionError(f"Hash mismatch on multipart upload assembly: {expected_etag} not in {body_text}")


def _etag_from_part_hexes(part_etags: Sequence[str]) -> str:
    raw = b"".join(bytes.fromhex(e) for e in part_etags)
    _, md5, _ = get_context().hash_buffers([raw], _lib.MD5)
    return f"{md5[0].tobytes().hex()}-{len(part_etags)}"


# ---------------------------------------------------------------------------------------- blob upload


def get_content_length(data: BinaryIO) -> int:
    """Bytes from the current position to the end of the stream."""
    here = data.tell()
    end = data.seek(0, os.SEEK_END)
    data.seek(here)
    return end - here


async def _blob_upload_with_fallback(items, blob_ids: list[str], callback, content_length: int) -> tuple[str, bool, int]:
    """Try each storage provider in order; report whether R2 failed and the R2 throughput (reference :246-268)."""
    r2_failed, r2_bps = False, 0
    for idx, (item, blob_id) in enumerate(zip(items, blob_ids)):
        is_r2 = blob_id.endswith(":r2")
        try:
            t0 = time.monotonic_ns()
            await callback(item)
            if is_r2:
                r2_bps = (content_length * 1_000_000_000) // max(time.monotonic_ns() - t0, 1)
            return blob_id, r2_failed, r2_bps
        except Exception:
            r2_failed = r2_failed or is_r2
            if idx == len(items) - 1:
                raise
    raise ExecutionError("Failed to upload blob")


async def _blob_upload(
    upload_hashes: UploadHashes,
    data: bytes | BinaryIO,
    stub,
    progress_report_cb: Callable | None = None,
    byte_budget: _ByteBudget | None = None,
    _blob_create_response=None,
) -> tuple[str, bool, int]:
    """BlobCreate with the precomputed digests, then a single PUT or a multipart upload (reference :271-335).
    The map pump calls this once per blobified input, 10^5 times per map: a ``bytes`` payload is not wrapped in a
    reader (nor is its aiohttp payload object built) before a PUT actually needs one."""
    if isinstance(data, bytes):
        reader, content_length = None, len(data)
    else:
        reader, content_length = data, get_content_length(data)
    resp = _blob_create_response  # set when _blob_upload_bytes already made the request
    if resp is None:
        resp = await stub.BlobCreate(
            BlobCreateRequest(
                content_md5=upload_hashes.md5_base64,
                content_sha256_base64=upload_hashes.sha256_base64,
                content_length=content_length,
            )
        )
    if resp.WhichOneof("upload_types_oneof") == "multiparts":
        if reader is None:
            reader = BytesIO(data)

        async def send_multipart(part):
            return await perform_multipart_upload(
                reader,
                content_length=content_length,
                max_part_size=part.part_length,
                part_urls=part.upload_urls,
                completion_url=part.completion_url,
                upload_chunk_size=DEFAULT_SEGMENT_CHUNK_SIZE,
                progress_report_cb=progress_report_cb,
                byte_budget=byte_budget,
            )

        result = await _blob_upload_with_fallback(resp.multiparts.items, resp.blob_ids, send_multipart, content_length)
    else:
        payload = None

        async def send_single(url):
            nonlocal payload
            if payload is None:
                # the whole-blob MD5 is already in upload_hashes: hand it to the payload instead of re-hashing
                raw = getattr(upload_hashes, "md5_raw", None)
                if raw is None and _is_real_md5(upload_hashes):
                    raw = bytes.fromhex(upload_hashes.md5_hex())
                if reader is None and raw is not None:
                    payload = KnownBytesBody(data, raw, progress_report_cb)  # in memory, digest known: no reader at all
                else:
                    payload = BytesIOSegmentPayload(
                        reader if reader is not None else BytesIO(data), segment_start=0, segment_length=content_length,
                        progress_report_cb=progress_report_cb, md5_digest=raw)
            return await _upload_to_s3_url(url, payload, content_md5_b64=upload_hashes.md5_base64)

        result = await _blob_upload_with_fallback(resp.upload_urls.items, resp.blob_ids, send_single, content_length)
    if progress_report_cb:
        progress_report_cb(complete=True)
    return result


async def _blob_upload_bytes(upload_hashes: UploadHashes, data: bytes, stub) -> tuple[str, bool, int]:
    """``_blob_upload`` for an in-memory payload whose digests came out of a GPU batch (see ``_blob_upload_row``)."""
    return await _blob_upload_row(upload_hashes.md5_base64, upload_hashes.sha256_base64,
                                  getattr(upload_hashes, "md5_raw", None), data, stub)


async def _blob_upload_row(md5_b64: str, sha256_b64: str, md5_raw: bytes | None, data: bytes, stub) -> tuple[str, bool, int]:
    """``_blob_upload`` for the map pump's case -- an in-memory payload and its row of a GPU digest table (base64
    columns + the raw MD5) -- with the single-PUT branch and the provider fallback written out flat (same BlobCreate
    request, same fallback order, same r2 bookkeeping as ``_blob_upload`` / ``_blob_upload_with_fallback``): 10^5 of
    these run per map on the event-loop thread, and every coroutine frame, closure and temporary object per input is
    paid there.  Anything else (multipart answer, digest unknown) goes through the general function."""
    resp = await stub.BlobCreate(BlobCreateRequest(content_md5=md5_b64, content_sha256_base64=sha256_b64,
                                                   content_length=len(data)))  # keywords: the real class is a protobuf
    if md5_raw is None or resp.WhichOneof("upload_types_oneof") != "upload_urls":
        return await _blob_upload(hash_utils._UploadHashesRaw(md5_b64, sha256_b64, md5_raw), data, stub,
                                  _blob_create_response=resp)
    body = KnownBytesBody(data, md5_raw)
    urls, blob_ids = resp.upload_urls.items, resp.blob_ids
    if len(urls) == 1 and not blob_ids[0].endswith(":r2"):  # the common answer: one provider, nothing to fall back to
        await _upload_to_s3_url(urls[0], body, content_md5_b64=md5_b64)
        return blob_ids[0], False, 0
    r2_failed, last = False, len(urls) - 1
    for idx, url in enumerate(urls):
        blob_id = blob_ids[idx]
        is_r2 = blob_id.endswith(":r2")
        try:
            if is_r2:
                t0 = time.monotonic_ns()
                await _upload_to_s3_url(url, body, content_md5_b64=md5_b64)
                return blob_id, r2_failed, (len(data) * 1_000_000_000) // max(time.monotonic_ns() - t0, 1)
            await _upload_to_s3_url(url, body, content_md5_b64=md5_b64)
            return blob_id, r2_failed, 0
        except Exception:
            r2_failed = r2_failed or is_r2
            if idx == last:
                raise
    raise ExecutionError("Failed to upload blob")


def _is_real_md5(h: UploadHashes) -> bool:
    return bool(h.md5_base64) and h.md5_hex() != _MD5_PLACEHOLDER


def _is_real_md5_hex(md5_hex: str | None) -> bool:
    return bool(md5_hex) and md5_hex != _MD5_PLACEHOLDER


async def blob_upload_with_r2_failure_info(payload: bytes, stub) -> tuple[str, bool, int]:
    if isinstance(payload, str):
        logger.debug("Blob uploading string, not bytes - auto-encoding as utf8")
        payload = payload.encode("utf8")
    t0 = time.time()
    hashes = get_upload_hashes(payload)
    out = await _blob_upload(hashes, payload, stub)
    mib = len(payload) / (1 << 20)
    dt = max(time.time() - t0, 0.001)
    logger.debug(f"Uploaded large blob of size {mib:.2f} MiB ({mib / dt:.2f} MiB/s, total {dt:.2f}s). {out[0]}")
    return out


async def blob_upload(payload: bytes, stub) -> str:
    blob_id, _, _ = await blob_upload_with_r2_failure_info(payload, stub)
    return blob_id


async def blob_upload_many(payloads: Sequence[bytes], stub, concurrency: int | None = None) -> list[tuple[str, bool, int]]:
    """The batched form the map pump uses: hash all payloads in ONE GPU batch, then run the uploads with
    the reference's concurrency (BLOB_MAX_PARALLELISM).  Order is preserved."""
    payloads = [p.encode("utf8") if isinstance(p, str) else p for p in payloads]
    hashes = await asyncio.to_thread(hash_utils.get_upload_hashes_many, payloads)
    jobs = list(zip(hashes, payloads))
    return await bounded_map(jobs, lambda hp: _blob_upload(hp[0], hp[1], stub), concurrency or BLOB_MAX_PARALLELISM)


async def format_blob_data(data: bytes, api_stub) -> dict[str, Any]:
    return {"data_blob_id": await blob_upload(data, api_stub)} if len(data) > MAX_OBJECT_SIZE_BYTES else {"data": data}


async def blob_upload_file(
    file_obj: BinaryIO,
    stub,
    progress_report_cb: Callable | None = None,
    sha256_hex: str | None = None,
    md5_hex: str | None = None,
    byte_budget: _ByteBudget | None = None,
) -> str:
    hashes = get_upload_hashes(file_obj, sha256_hex=sha256_hex, md5_hex=md5_hex)
    blob_id, _, _ = await _blob_upload(hashes, file_obj, stub, progress_report_cb, byte_budget=byte_budget)
    return blob_id


# ------------------------------------------------------------------------------------------- download


@retry(n_attempts=5, base_delay=0.1, attempt_timeout=None)
async def _download_from_url(download_url: str) -> bytes:
    """GET one blob (reference :377-388; no integrity check there either: blobs are addressed by id)."""
    async with ClientSessionRegistry.get_session().get(download_url) as s3_resp:
        if s3_resp.status == 503:  # S3 SlowDown
            logger.debug("Received SlowDown signal from S3, sleeping for 1 second before retrying.")
            await asyncio.sleep(1)
        if s3_resp.status != 200:
            text = await s3_resp.text()
            raise ExecutionError(f"Get from url failed with status {s3_resp.status}: {text}")
        return await s3_resp.read()


async def blob_download(blob_id: str, stub) -> bytes:
    """Read a whole blob into memory (reference :391-404)."""
    logger.debug(f"Downloading large blob {blob_id}")
    t0 = time.time()
    resp = await stub.BlobGet(_wire.BlobGetRequest(blob_id=blob_id))
    data = await _download_from_url(resp.download_url)
    size_mib = len(data) / 1024 / 1024
    dur_s = max(time.time() - t0, 0.001)
    logger.debug(f"Downloaded large blob {blob_id} of size {size_mib:.2f} MiB ({size_mib / dur_s:.2f} MiB/s, total {dur_s:.2f}s)")
    return data


async def blob_iter(blob_id: str, stub):
    """Stream a blob chunk by chunk (reference :407-422)."""
    resp = await stub.BlobGet(_wire.BlobGetRequest(blob_id=blob_id))
    async with ClientSessionRegistry.get_session().get(resp.download_url) as s3_resp:
        if s3_resp.status == 503:
            logger.debug("Received SlowDown signal from S3, sleeping for 1 second before retrying.")
            await asyncio.sleep(1)
        if s3_resp.status != 200:
            text = await s3_resp.text()
            raise ExecutionError(f"Get from url failed with status {s3_resp.status}: {text}")
        async for chunk in s3_resp.content.iter_any():
            yield chunk


# ------------------------------------------------------------------------------- FileUploadSpec (v1)


@dataclasses.dataclass(slots=True)
class FileUploadSpec:
    source: Callable[[], AbstractContextManager | BinaryIO]
    source_description: Any
    source_is_path: bool
    mount_filename: str

    use_blob: bool
    sha256_hex: str
    md5_hex: str
    mode: int  # permission bits (low 12 bits of st_mode)
    size: int
    content: bytes | None = None  # cached for very small files

    def read_content(self) -> bytes:
        with self.source() as fp:
            fp.seek(0)
            return fp.read()


def _size_class(size: int) -> tuple[bool, bool, bool]:
    """-> (use_blob, want_md5, cache_content) for a file of ``size`` bytes (reference :459-474)."""
    if size >= LARGE_FILE_LIMIT:
        return True, not (size > MULTIPART_UPLOAD_THRESHOLD), False
    return False, True, size < SMALL_FILE_INLINE_LIMIT


def _get_file_upload_spec(
    source: Callable[[], AbstractContextManager | BinaryIO],
    source_description: Any,
    mount_filename: PurePosixPath,
    mode: int,
) -> FileUploadSpec:
    content = None
    with source() as fp:
        size = fp.seek(0, os.SEEK_END)  # the current position is ignored: uploads start at 0
        fp.seek(0)
        use_blob, want_md5, cache = _size_class(size)
        if cache:
            content = fp.read()
            hashes = get_upload_hashes(content)
        else:
            hashes = get_upload_hashes(fp, md5_hex=None if want_md5 else _MD5_PLACEHOLDER)
    return FileUploadSpec(
        source=source,
        source_description=source_description,
        source_is_path=isinstance(source_description, Path),
        mount_filename=mount_filename.as_posix(),
        use_blob=use_blob,
        sha256_hex=hashes.sha256_hex(),
        md5_hex=hashes.md5_hex(),
        mode=mode & 0o7777,
        size=size,
        content=content,
    )


def _default_mode(filename: Path) -> int:
    return os.stat(filename).st_mode & (0o7777 if platform.system() != "Windows" else 0o7755)


def get_file_upload_spec_from_path(
    filename: Path, mount_filename: PurePosixPath, mode: int | None = None
) -> FileUploadSpec:
    return _get_file_upload_spec(lambda: open(filename, "rb"), filename, mount_filename, mode or _default_mode(filename))


def get_file_upload_spec_from_fileobj(fp: BinaryIO, mount_filename: PurePosixPath, mode: int) -> FileUploadSpec:
    @contextmanager
    def source():
        fp.seek(0)
        yield fp

    return _get_file_upload_spec(source, str(fp), mount_filename, mode)


def get_file_upload_specs(
    files: Sequence[tuple[Path | str, PurePosixPath | str, int | None]],
    cache_small_content: bool | None = None,
) -> list[FileUploadSpec]:
    """Batched ``get_file_upload_spec_from_path``: every file of a ``Volume.batch_upload`` / ``Mount`` goes
    to the GPU in one batch (the reference fans the per-file hashlib loops over a ThreadPoolExecutor,
    py/modal/volume.py:1209-1216, py/modal/mount.py:467-485).  Sizes/modes come from ``b200h_stat_files`` and
    the bytes are read by the library's native reader threads straight into its pinned staging ring
    (``b200h_hash_files``): no per-file Python I/O, no mmap.
    Same size classes / placeholder MD5 as ``_get_file_upload_spec``.  ``content`` (the reference's
    "avoid the double read" cache for files < 256 KiB) is filled when ``cache_small_content`` is true;
    the default (None) does so only for batches of <= 4096 files -- for a million-file tree the extra
    Python read per file would cost more than the hashing."""
    if not files:
        return []
    ctx = get_context()
    n = len(files)
    paths = [os.fsencode(f[0]) for f in files]  # encoded once for the stat and the hash calls
    sizes, modes = ctx.stat_files(paths)
    # size classes, vectorised (same comparisons as _size_class)
    use_blob = sizes >= LARGE_FILE_LIMIT
    want_md5 = ~(use_blob & (sizes > MULTIPART_UPLOAD_THRESHOLD))
    cacheable = ~use_blob & (sizes < SMALL_FILE_INLINE_LIMIT)
    if cache_small_content is None:
        cache_small_content = n <= 4096
    # Files whose content is cached in the spec (< 256 KiB, like the reference's "read once" class) are read ONCE, here,
    # and those very bytes are hashed -- the digest can never disagree with spec.content, whatever happens to the
    # file meanwhile.  Everything else is read by the library's native reader.
    contents: dict[int, bytes] = {}
    if cache_small_content:
        for i in np.flatnonzero(cacheable).tolist():
            with open(files[i][0], "rb") as f:
                contents[i] = f.read()
        if contents:
            idx = np.fromiter(contents.keys(), dtype=np.int64, count=len(contents))
            sizes[idx] = [len(c) for c in contents.values()]
    from_memory = np.zeros(n, bool)
    if contents:
        from_memory[list(contents.keys())] = True
    # one fused SHA-256+MD5 batch for the files that need both, a SHA-only batch for the > 1 GiB class.  The digest
    # columns come back as the hex text the wire rows carry (FileUploadSpec / MountFile.sha256_hex), formatted on the
    # device from the digest table (B200H_HEX_OUT) -- no per-row conversion on the host.
    HEX = _lib.HEX_OUT
    sha_all = np.empty((n, 64), np.uint8)
    md5_all = np.full((n, 32), ord("0"), np.uint8)
    if contents:
        idx = np.flatnonzero(from_memory)
        sha, md5, _ = ctx.hash_buffers([contents[i] for i in idx.tolist()], _lib.SHA256 | _lib.MD5 | HEX)
        sha_all[idx], md5_all[idx] = sha, md5
    both = np.flatnonzero(want_md5 & ~from_memory)
    sha_only = np.flatnonzero(~want_md5 & ~from_memory)
    if both.size:
        sha, md5, _ = ctx.hash_files([paths[i] for i in both] if both.size != n else paths, sizes[both], 0,
                                     _lib.SHA256 | _lib.MD5 | HEX)
        sha_all[both], md5_all[both] = sha, md5
    if sha_only.size:
        sha, _, _ = ctx.hash_files([paths[i] for i in sha_only], sizes[sha_only], 0, _lib.SHA256 | HEX)
        sha_all[sha_only] = sha
    # A file that GREW between the stat and the read was hashed as its old prefix (a file that shrank fails the read):
    # stat again and redo the few that changed one at a time, the reference's way (one open, size and bytes together).
    redo: dict[int, FileUploadSpec] = {}
    streamed = np.flatnonzero(~from_memory)
    if streamed.size:
        sizes_after, _ = ctx.stat_files([paths[i] for i in streamed] if streamed.size != n else paths)
        for i in streamed[sizes_after != sizes[streamed]].tolist():
            filename, mount_filename, mode = files[i]
            redo[i] = get_file_upload_spec_from_path(Path(filename), PurePosixPath(mount_filename), mode)
    sha_hex, md5_hex = sha_all.tobytes().decode("ascii"), md5_all.tobytes().decode("ascii")  # sliced per file below
    sizes_l, modes_l = sizes.tolist(), modes.tolist()
    use_blob_l, want_md5_l = use_blob.tolist(), want_md5.tolist()
    # The per-file Python work below is what is left of a million-file tree once hashing takes a fraction of a second,
    # so it is kept to positional construction and precomputed columns (~2.5 us per file).
    partial, spec_cls, placeholder = functools.partial, FileUploadSpec, _MD5_PLACEHOLDER
    specs = []
    append = specs.append
    # a million small objects allocated in one go: without this the cyclic GC rescans the growing list again and again
    gc_was_on = gc.isenabled()
    gc.disable()
    try:
        _build_specs(files, append, spec_cls, partial, placeholder, contents, use_blob_l, want_md5_l,
                     sha_hex, md5_hex, modes_l, sizes_l)
    finally:
        if gc_was_on:
            gc.enable()
    for i, spec in redo.items():
        specs[i] = spec
    return specs


def _build_specs(files, append, spec_cls, partial, placeholder, contents, use_blob_l, want_md5_l,
                 sha_hex, md5_hex, modes_l, sizes_l) -> None:
    get_content = contents.get
    for i, (filename, mount_filename, mode) in enumerate(files):
        content = get_content(i)  # the bytes that were hashed (cached class only)
        append(
            spec_cls(
                partial(open, filename, "rb"),                                        # source
                filename if isinstance(filename, Path) else Path(filename),           # source_description
                True,                                                                 # source_is_path
                mount_filename if type(mount_filename) is str                         # posix string from a trusted walk
                else str(mount_filename) if type(mount_filename) is PurePosixPath
                else PurePosixPath(mount_filename).as_posix(),
                use_blob_l[i],
                sha_hex[64 * i : 64 * i + 64],
                md5_hex[32 * i : 32 * i + 32] if want_md5_l[i] else placeholder,
                (mode if mode else modes_l[i]) & 0o7777,
                sizes_l[i],
                content,
            )
        )


def first_occurrence_of_specs(specs: Sequence[FileUploadSpec]) -> tuple[list[int], int]:
    """In-batch dedupe of a list of specs by content (SHA-256), computed on the GPU over the digest table:
    ``first[i]`` is the index of the first spec with the same content as spec i.  The reference's counterpart is
    the ``accounted_hashes`` set walked file by file in ``_Mount._load_mount`` (py/modal/mount.py:498,518-534)."""
    n = len(specs)
    if n == 0:
        return [], 0
    keys = np.frombuffer(bytes.fromhex("".join(s.sha256_hex for s in specs)), np.uint8).reshape(n, 32)
    first, ndistinct = get_context().dedupe(keys)
    return first.tolist(), ndistinct


# ---------------------------------------------------------------------------- FileUploadSpec2 (v2)

_FileUploadSource2 = Callable[[], ContextManager[BinaryIO]]


@dataclasses.dataclass
class FileUploadBlock:
    start: int  # inclusive byte offset of the block in the file
    end: int  # exclusive end after dropping the block's trailing zero bytes
    contents_sha256: bytes  # raw 32-byte SHA-256 of [start, end)


def _blocks_of(view: np.ndarray) -> list[FileUploadBlock]:
    """All ceil(size/BLOCK_SIZE) blocks of one file image: trim scan + SHA-256 per block on the device."""
    if view.size == 0:
        return []
    sha, _, trimmed, _ = get_context().hash_fixed_parts(view, BLOCK_SIZE, _lib.SHA256 | _lib.TRIM_ZEROS)
    return [
        FileUploadBlock(start=i * BLOCK_SIZE, end=i * BLOCK_SIZE + int(trimmed[i]), contents_sha256=sha[i].tobytes())
        for i in range(len(trimmed))
    ]


@dataclasses.dataclass
class FileUploadSpec2:
    source: _FileUploadSource2
    source_description: str | Path

    path: str
    blocks: list[FileUploadBlock]  # 8 MiB blocks
    mode: int
    size: int

    @staticmethod
    async def from_path(
        filename: Path, mount_filename: PurePosixPath, hash_semaphore: asyncio.Semaphore, mode: int | None = None
    ) -> "FileUploadSpec2":
        def source():
            return open(filename, "rb")

        return await FileUploadSpec2._create(source, filename, mount_filename, mode or _default_mode(filename),
                                             hash_semaphore)

    @staticmethod
    async def from_fileobj(
        source_fp: BinaryIO | BytesIO, mount_filename: PurePosixPath, hash_semaphore: asyncio.Semaphore, mode: int
    ) -> "FileUploadSpec2":
        try:
            fileno = source_fp.fileno()

            def source():
                fp = os.fdopen(os.dup(fileno), "rb")
                fp.seek(0)
                return fp

        except OSError:  # BytesIO-like: no descriptor
            buffer = source_fp.getbuffer()

            def source():
                return BytesIO(buffer)

        return await FileUploadSpec2._create(source, str(source), mount_filename, mode, hash_semaphore)

    @staticmethod
    async def _create(
        source: _FileUploadSource2,
        source_description: str | Path,
        mount_filename: PurePosixPath,
        mode: int,
        hash_semaphore: asyncio.Semaphore,
    ) -> "FileUploadSpec2":
        with source() as fp:
            size = fp.seek(0, os.SEEK_END)
        blocks = await _gather_blocks(source, size, hash_semaphore)
        return FileUploadSpec2(source=source, source_description=source_description, path=mount_filename.as_posix(),
                               blocks=blocks, mode=mode & 0o7777, size=size)


async def _gather_blocks(source: _FileUploadSource2, size: int, hash_semaphore: asyncio.Semaphore) -> list[FileUploadBlock]:
    """Block list of one file.  The reference launches one thread task per block, each reading its block
    twice (rstrip pass + SHA pass, :640-664); here the file image is handed to the GPU once and all its
    blocks are trimmed and hashed by one batch."""
    if size == 0:
        return []

    def run() -> list[FileUploadBlock]:
        with source() as fp:
            return _with_view(fp, lambda view: _blocks_of(view[:size]))

    async with hash_semaphore:
        return await asyncio.to_thread(run)


def _read_range(source: _FileUploadSource2, start: int, end: int) -> bytes:
    with source() as fp:
        fp.seek(start)
        out = bytearray()
        while len(out) < end - start:
            chunk = fp.read(end - start - len(out))
            if not chunk:
                break
            out += chunk
        return bytes(out)


def _gather_block(source: _FileUploadSource2, block_idx: int) -> FileUploadBlock:
    start = block_idx * BLOCK_SIZE
    data = _read_range(source, start, start + BLOCK_SIZE)
    sha, _, trimmed = get_context().hash_batch_host(np.frombuffer(data, dtype=np.uint8), [0], [len(data)],
                                                    _lib.SHA256 | _lib.TRIM_ZEROS)
    return FileUploadBlock(start=start, end=start + int(trimmed[0]), contents_sha256=sha[0].tobytes())


def _hash_range_sha256(source: _FileUploadSource2, start, end) -> bytes:
    data = _read_range(source, start, end)
    sha, _, _ = get_context().hash_buffers([data], _lib.SHA256)
    return sha[0].tobytes()


def _find_end_of_block(source: _FileUploadSource2, start: int, end: int) -> int | None:
    """Index just past the last non-zero byte of [start, end) -- ``start`` for an empty or all-zero range.
    (The reference docstring's ``(…, 0, 3) -> 4`` example is stale: its code, like this, returns 3.)"""
    data = _read_range(source, start, end)
    if not data:
        return start
    _, _, trimmed = get_context().hash_batch_host(np.frombuffer(data, dtype=np.uint8), [0], [len(data)],
                                                  _lib.SHA256 | _lib.TRIM_ZEROS)
    return start + int(trimmed[0])


async def file_upload_specs2(
    files: Sequence[tuple[Path, PurePosixPath, int | None]],
) -> list[FileUploadSpec2]:
    """Batched ``FileUploadSpec2.from_path`` for a whole ``batch_upload``: the blocks of ALL files form one
    GPU batch (so a tree of many small files is as efficient as one big file), read by the library's native
    reader threads (``b200h_hash_files`` with part_len = BLOCK_SIZE and zero trimming)."""
    if not files:
        return []

    def run() -> list[FileUploadSpec2]:
        ctx = get_context()
        paths = [os.fsencode(f[0]) for f in files]  # encoded once for the stat and the hash calls
        sizes, modes = ctx.stat_files(paths)
        sha, _, trimmed = ctx.hash_files(paths, sizes, BLOCK_SIZE, _lib.SHA256 | _lib.TRIM_ZEROS)
        out, row = [], 0
        sizes_l, modes_l, trimmed_l, sha_raw = sizes.tolist(), modes.tolist(), trimmed.tolist(), sha.tobytes()
        block_cls, spec_cls, partial, bs = FileUploadBlock, FileUploadSpec2, functools.partial, BLOCK_SIZE
        gc_was_on = gc.isenabled()
        gc.disable()  # bulk allocation of small objects: keep the cyclic GC from rescanning the growing lists
        try:
            for i, (filename, mount_filename, mode) in enumerate(files):
                size = sizes_l[i]
                blocks = []
                for start in range(0, size, bs):
                    blocks.append(block_cls(start, start + trimmed_l[row], sha_raw[32 * row : 32 * row + 32]))
                    row += 1
                out.append(
                    spec_cls(
                        source=partial(open, filename, "rb"),
                        source_description=filename if isinstance(filename, Path) else Path(filename),
                        path=mount_filename if type(mount_filename) is str
                        else str(mount_filename) if type(mount_filename) is PurePosixPath
                        else PurePosixPath(mount_filename).as_posix(),
                        blocks=blocks,
                        mode=(mode if mode else modes_l[i]) & 0o7777,
                        size=size,
                    )
                )
        finally:
            if gc_was_on:
                gc.enable()
        return out

    return await asyncio.to_thread(run)


# ------------------------------------------------------------------------- tensors already in HBM


class _ByteCounter:
    def __init__(self):
        self._lock = threading.Lock()
        self.total = 0

    def add(self, n: int) -> None:
        with self._lock:
            self.total += n


class DeviceBufferReader(io.RawIOBase):
    """Read-only, seekable binary file object over the raw bytes of a contiguous tensor (``numel * element_size`` from
    ``data_ptr()``).  ``read(n)`` copies only that range to the host, ``stage_bytes`` at a time through a small pinned
    buffer, so host memory is bounded by the reads in flight (the PUTs), never by the tensor size.  ``clone()`` gives
    an independent reader (own position and staging buffer) over the same bytes; every clone adds to the same
    ``bytes_to_host`` count, which is what crossed PCIe.  Used as a spec's ``source()``, it lets ``_put_missing_blocks``,
    ``BytesIOSegmentPayload`` and ``blob_upload_file`` run unchanged.

    The reader waits, before its first copy, on a CUDA event recorded on the tensor's current stream when the reader
    was made (``ready``): work queued before that is visible, later writes to the tensor are not allowed until the
    upload is done.  A CPU tensor is read with plain copies (host-backed reader, for host-side tests)."""

    def __init__(self, tensor, *, stage_bytes: int = 4 << 20, _root: "DeviceBufferReader | None" = None):
        super().__init__()
        if _root is None:
            if not tensor.is_contiguous():
                raise ValueError("DeviceBufferReader needs a contiguous tensor")
            self.tensor = tensor
            self.nbytes = tensor.numel() * tensor.element_size()
            self._flat = tensor.reshape(-1).view(_torch().uint8) if self.nbytes else None
            self._counter = _ByteCounter()
            self._ready = None
            if tensor.is_cuda:
                from .batch import ready_event

                self._ready = ready_event(tensor)
        else:
            self.tensor, self.nbytes, self._flat = _root.tensor, _root.nbytes, _root._flat
            self._counter, self._ready = _root._counter, _root._ready
        self._stage_bytes = stage_bytes
        self._pos = 0
        self._pin = self._pin_np = self._stream = None

    # ---- what the hash and upload layers ask -----------------------------------------------------------------
    @property
    def data_ptr(self) -> int:
        return self.tensor.data_ptr()

    @property
    def device(self):
        return self.tensor.device

    @property
    def bytes_to_host(self) -> int:
        """Bytes this reader and its clones have copied to the host so far."""
        return self._counter.total

    def wait_ready(self) -> None:
        """Block until the work queued on the tensor's stream before the reader was made has finished."""
        if self._ready is not None:
            self._ready.synchronize()

    def clone(self) -> "DeviceBufferReader":
        return DeviceBufferReader(None, stage_bytes=self._stage_bytes, _root=self)

    def part_digests(self, start: int, length: int, part_length: int) -> tuple[list[bytes], str]:
        """``multipart_part_digests`` of bytes [start, start + length), hashed on the device where they are: the part
        MD5s and the multipart ETag from one ``b200h_hash_device_parts(part_length, MD5)`` call."""
        self.wait_ready()
        _, md5, _, etag = get_context().hash_device_parts([self.data_ptr + start], [length], part_length, _lib.MD5,
                                                          want_etag=True)
        return [md5[i].tobytes() for i in range(len(md5))], f"{etag[0].tobytes().hex()}-{len(md5)}"

    # ---- io.RawIOBase ------------------------------------------------------------------------------------------
    def readable(self) -> bool:
        return True

    def seekable(self) -> bool:
        return True

    def tell(self) -> int:
        return self._pos

    def seek(self, offset: int, whence: int = os.SEEK_SET) -> int:
        base = {os.SEEK_SET: 0, os.SEEK_CUR: self._pos, os.SEEK_END: self.nbytes}[whence]
        if base + offset < 0:
            raise ValueError("negative seek position")
        self._pos = base + offset
        return self._pos

    def read(self, size: int = -1) -> bytes:
        n = max(0, self.nbytes - self._pos) if size is None or size < 0 else size
        buf = bytearray(min(n, max(0, self.nbytes - self._pos)))
        got = self.readinto(buf)
        return bytes(buf) if got == len(buf) else bytes(buf[:got])

    def readinto(self, b) -> int:
        dst = np.frombuffer(memoryview(b).cast("B"), np.uint8)
        n = max(0, min(dst.size, self.nbytes - self._pos))
        if n == 0:
            return 0
        self._copy(self._pos, dst[:n])
        self._pos += n
        self._counter.add(n)
        return n

    def close(self) -> None:
        self._pin = self._pin_np = self._stream = None
        super().close()

    def _copy(self, at: int, dst: np.ndarray) -> None:
        self._stage(self._flat[at : at + dst.size], dst)

    def _stage(self, src, dst: np.ndarray) -> None:
        """dst[:] = the uint8 tensor ``src``, through the pinned staging buffer when it is on the GPU."""
        if not src.is_cuda:
            dst[:] = src.numpy()
            return
        torch = _torch()
        self.wait_ready()
        if self._pin is None:
            self._pin = torch.empty(min(self._stage_bytes, self.nbytes), dtype=torch.uint8, pin_memory=True)
            self._pin_np = self._pin.numpy()
            self._stream = torch.cuda.Stream(device=src.device)
        step = self._pin.numel()
        with torch.cuda.stream(self._stream):
            for o in range(0, dst.size, step):
                k = min(step, dst.size - o)
                self._pin[:k].copy_(src[o : o + k], non_blocking=True)
                self._stream.synchronize()
                dst[o : o + k] = self._pin_np[:k]


class DeviceSegmentsReader(DeviceBufferReader):
    """Read-only, seekable binary file object over a file made of segments: ``header`` (host bytes) followed by the
    raw bytes of contiguous ``tensors``, back to back -- a safetensors file whose tensors stay in HBM.  Reads, clones,
    ``bytes_to_host`` and ``wait_ready`` behave as for ``DeviceBufferReader``; a read of the header range is served
    from the host bytes (and counted like any other byte read).  The header also lives in a small CUDA tensor on the
    tensors' device, so the hash calls see device segments only.  The ready event is recorded on the device's current
    stream when the reader is made.  With CPU tensors every read is a plain copy (host-backed reader, for host-side
    tests)."""

    def __init__(self, header: bytes, tensors: Sequence, *, stage_bytes: int = 4 << 20,
                 _root: "DeviceSegmentsReader | None" = None):
        io.RawIOBase.__init__(self)
        if _root is None:
            torch = _torch()
            self.header = bytes(header)
            self.tensors = list(tensors)
            self._flats = [t.reshape(-1).view(torch.uint8) for t in self.tensors]
            dev = self.tensors[0].device if self.tensors else torch.device("cpu")
            host_header = torch.frombuffer(bytearray(self.header), dtype=torch.uint8)
            self._header_t = host_header.to(dev) if dev.type == "cuda" else host_header
            sizes = [len(self.header)] + [int(f.numel()) for f in self._flats]
            self._starts = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
            self.nbytes = int(self._starts[-1])
            self._counter = _ByteCounter()
            self._ready = None
            if dev.type == "cuda":
                from .batch import ready_event

                self._ready = ready_event(self._header_t)
        else:
            self.header, self.tensors, self._flats, self._header_t = _root.header, _root.tensors, _root._flats, _root._header_t
            self._starts, self.nbytes, self._counter, self._ready = _root._starts, _root.nbytes, _root._counter, _root._ready
        self._stage_bytes = stage_bytes
        self._pos = 0
        self._pin = self._pin_np = self._stream = None

    @property
    def data_ptr(self) -> int:
        raise TypeError("a DeviceSegmentsReader has no single buffer: use segments()")

    @property
    def device(self):
        return self._header_t.device

    def segments(self, start: int = 0, length: int | None = None) -> list[tuple[int, int]]:
        """(device address, nbytes) of the pieces of the header tensor and the tensors that make up bytes
        [start, start + length) of the file: the segment list of ``hash_device_segments``."""
        end = self.nbytes if length is None else start + length
        out = []
        for i, t in enumerate([self._header_t] + self._flats):
            lo, hi = max(start, int(self._starts[i])), min(end, int(self._starts[i + 1]))
            if hi > lo:
                out.append((t.data_ptr() + lo - int(self._starts[i]), hi - lo))
        return out

    def clone(self) -> "DeviceSegmentsReader":
        return DeviceSegmentsReader(b"", (), stage_bytes=self._stage_bytes, _root=self)

    def part_digests(self, start: int, length: int, part_length: int) -> tuple[list[bytes], str]:
        """``multipart_part_digests`` of bytes [start, start + length), hashed on the device where they are: the part
        MD5s and the multipart ETag from one ``b200h_hash_device_segments(part_length, MD5)`` call."""
        self.wait_ready()
        _, md5, _, etag = get_context().hash_device_segments([self.segments(start, length)], part_length, _lib.MD5,
                                                             want_etag=True)
        return [md5[i].tobytes() for i in range(len(md5))], f"{etag[0].tobytes().hex()}-{len(md5)}"

    def _copy(self, at: int, dst: np.ndarray) -> None:
        end = at + dst.size
        hl = len(self.header)
        if at < hl:
            k = min(end, hl) - at
            dst[:k] = np.frombuffer(self.header, np.uint8, count=k, offset=at)
        for i, f in enumerate(self._flats):
            lo, hi = max(at, int(self._starts[i + 1])), min(end, int(self._starts[i + 2]))
            if hi > lo:
                base = int(self._starts[i + 1])
                self._stage(f[lo - base : hi - base], dst[lo - at : hi - at])


def _torch():
    import torch

    return torch


def _reader_digests(readers: Sequence[DeviceBufferReader], part_len: int, flags: int, want_etag: bool = False):
    """One ``hash_device_parts`` call over the bytes of every reader's tensor, once the work queued on each tensor's
    stream has finished."""
    for r in readers:
        r.wait_ready()
    return get_context().hash_device_parts([r.data_ptr for r in readers], [r.nbytes for r in readers], part_len, flags,
                                           want_etag)


def tensor_upload_specs(items: Sequence[tuple[DeviceBufferReader, PurePosixPath | str, int]]) -> list[FileUploadSpec]:
    """``FileUploadSpec`` (volumefs1) for tensors queued with ``put_tensor``: whole-buffer SHA-256 + MD5 of each tensor's
    bytes on the device (``hash_device_parts`` with part_len 0), the size classes of ``_size_class``.  Each digest of a
    whole buffer is ONE serial chain on the chain kernel, about 71 MB/s (DESIGN §5.4): roughly 15 s for 1 GiB.  The
    multipart part MD5s are computed later on the device as well (``perform_multipart_upload``)."""
    if not items:
        return []
    readers = [r for r, _, _ in items]
    sizes = [r.nbytes for r in readers]
    classes = [_size_class(s) for s in sizes]
    sha_hex, md5_hex = [""] * len(items), [_MD5_PLACEHOLDER] * len(items)
    for want_md5 in (True, False):
        idx = [i for i, c in enumerate(classes) if c[1] == want_md5]
        if not idx:
            continue
        sha, md5, _, _ = _reader_digests([readers[i] for i in idx], 0, _lib.SHA256 | (_lib.MD5 if want_md5 else 0))
        for row, i in enumerate(idx):
            sha_hex[i] = sha[row].tobytes().hex()
            if want_md5:
                md5_hex[i] = md5[row].tobytes().hex()
    return [
        FileUploadSpec(source=r.clone, source_description=f"<tensor {tuple(r.tensor.shape)} {r.tensor.dtype}>",
                       source_is_path=False, mount_filename=PurePosixPath(remote).as_posix(), use_blob=classes[i][0],
                       sha256_hex=sha_hex[i], md5_hex=md5_hex[i], mode=mode & 0o7777, size=sizes[i])
        for i, (r, remote, mode) in enumerate(items)
    ]


def tensor_upload_specs2(items: Sequence[tuple[DeviceBufferReader, PurePosixPath | str, int]]) -> list[FileUploadSpec2]:
    """``FileUploadSpec2`` (volumefs2) for tensors queued with ``put_tensor``: every 8 MiB block of every tensor in ONE
    ``hash_device_parts(BLOCK_SIZE, SHA256 | TRIM_ZEROS)`` call, the blocks exactly as ``file_upload_specs2`` builds
    them.  Only the trimmed bytes of the blocks the server reports missing are ever copied to the host."""
    if not items:
        return []
    readers = [r for r, _, _ in items]
    bs = BLOCK_SIZE
    sha, _, trimmed, _ = _reader_digests(readers, bs, _lib.SHA256 | _lib.TRIM_ZEROS)
    trimmed_l, sha_raw = trimmed.tolist(), sha.tobytes()
    out, row = [], 0
    for r, remote, mode in items:
        blocks = []
        for start in range(0, r.nbytes, bs):
            blocks.append(FileUploadBlock(start, start + trimmed_l[row], sha_raw[32 * row : 32 * row + 32]))
            row += 1
        out.append(FileUploadSpec2(source=r.clone, source_description=f"<tensor {tuple(r.tensor.shape)} {r.tensor.dtype}>",
                                   path=PurePosixPath(remote).as_posix(), blocks=blocks, mode=mode & 0o7777,
                                   size=r.nbytes))
    return out


# ------------------------------------------------------------------------- safetensors files straight from HBM

# safetensors dtype names in data order (the library sorts tensors by this rank, then by name), as torch dtype names
_SAFETENSORS_DTYPES = (
    ("U64", "uint64"), ("I64", "int64"), ("F64", "float64"), ("C64", "complex64"), ("F32", "float32"),
    ("U32", "uint32"), ("I32", "int32"), ("BF16", "bfloat16"), ("F16", "float16"), ("U16", "uint16"),
    ("I16", "int16"), ("F8_E4M3", "float8_e4m3fn"), ("F8_E5M2", "float8_e5m2"), ("I8", "int8"), ("U8", "uint8"),
    ("BOOL", "bool"),
)


def safetensors_layout(tensors, metadata: dict[str, str] | None = None) -> tuple[bytes, list[tuple[str, Any]]]:
    """The safetensors framing of a state dict without the safetensors package: ``(header, [(name, tensor), ...])``
    such that ``header`` followed by the raw bytes of the tensors in that order is byte for byte what
    ``safetensors.torch.save(tensors, metadata)`` returns.  The header is the 8-byte little-endian length of the JSON,
    then compact JSON (UTF-8, ``__metadata__`` first, then the tensors in data order: by dtype rank, then name), padded
    with spaces to a multiple of 8.  A dtype safetensors cannot store is a ``ValueError`` naming the tensor."""
    torch = _torch()
    rank = {getattr(torch, tn): (i, st) for i, (st, tn) in enumerate(_SAFETENSORS_DTYPES) if hasattr(torch, tn)}
    keyed = []
    for name, t in tensors.items():
        if t.dtype not in rank:
            raise ValueError(f"tensor {name!r} has dtype {t.dtype}, which safetensors cannot store")
        keyed.append((rank[t.dtype][0], name, t))
    keyed.sort(key=lambda x: (x[0], x[1]))
    head: dict[str, Any] = {}
    if metadata is not None:
        head["__metadata__"] = dict(metadata)
    at = 0
    for _, name, t in keyed:
        n = t.numel() * t.element_size()
        head[name] = {"dtype": rank[t.dtype][1], "shape": list(t.shape), "data_offsets": [at, at + n]}
        at += n
    js = json.dumps(head, ensure_ascii=False, separators=(",", ":")).encode("utf-8")
    js += b" " * (-len(js) % 8)
    return len(js).to_bytes(8, "little") + js, [(name, t) for _, name, t in keyed]


def _segments_digests(readers: Sequence[DeviceSegmentsReader], part_len: int, flags: int):
    """One ``hash_device_segments`` call over every reader's file, once the work queued before each was made is done."""
    for r in readers:
        r.wait_ready()
    return get_context().hash_device_segments([r.segments() for r in readers], part_len, flags)


def _safetensors_description(r: DeviceSegmentsReader) -> str:
    return f"<safetensors: {len(r.tensors)} tensors, {r.nbytes} bytes>"


def safetensors_upload_specs(items: Sequence[tuple[DeviceSegmentsReader, PurePosixPath | str, int]]) -> list[FileUploadSpec]:
    """``FileUploadSpec`` (volumefs1) for files queued with ``put_safetensors``: whole-file SHA-256 (+ MD5 by
    ``_size_class``) on the device.  A file of several segments is gathered whole into scratch first, then each digest
    is ONE serial chain, about 71 MB/s (DESIGN §5.4): roughly 15 s per GiB."""
    if not items:
        return []
    readers = [r for r, _, _ in items]
    classes = [_size_class(r.nbytes) for r in readers]
    sha_hex, md5_hex = [""] * len(items), [_MD5_PLACEHOLDER] * len(items)
    for want_md5 in (True, False):
        idx = [i for i, c in enumerate(classes) if c[1] == want_md5]
        if not idx:
            continue
        sha, md5, _, _ = _segments_digests([readers[i] for i in idx], 0, _lib.SHA256 | (_lib.MD5 if want_md5 else 0))
        for row, i in enumerate(idx):
            sha_hex[i] = sha[row].tobytes().hex()
            if want_md5:
                md5_hex[i] = md5[row].tobytes().hex()
    return [
        FileUploadSpec(source=r.clone, source_description=_safetensors_description(r), source_is_path=False,
                       mount_filename=PurePosixPath(remote).as_posix(), use_blob=classes[i][0], sha256_hex=sha_hex[i],
                       md5_hex=md5_hex[i], mode=mode & 0o7777, size=r.nbytes)
        for i, (r, remote, mode) in enumerate(items)
    ]


def safetensors_upload_specs2(items: Sequence[tuple[DeviceSegmentsReader, PurePosixPath | str, int]]) -> list[FileUploadSpec2]:
    """``FileUploadSpec2`` (volumefs2) for files queued with ``put_safetensors``: every 8 MiB block of every file in ONE
    ``hash_device_segments(BLOCK_SIZE, SHA256 | TRIM_ZEROS)`` call, the blocks exactly as ``file_upload_specs2`` builds
    them from the same bytes.  Only the trimmed bytes of the blocks the server reports missing are copied to the host."""
    if not items:
        return []
    readers = [r for r, _, _ in items]
    bs = BLOCK_SIZE
    sha, _, trimmed, _ = _segments_digests(readers, bs, _lib.SHA256 | _lib.TRIM_ZEROS)
    trimmed_l, sha_raw = trimmed.tolist(), sha.tobytes()
    out, row = [], 0
    for r, remote, mode in items:
        blocks = []
        for start in range(0, r.nbytes, bs):
            blocks.append(FileUploadBlock(start, start + trimmed_l[row], sha_raw[32 * row : 32 * row + 32]))
            row += 1
        out.append(FileUploadSpec2(source=r.clone, source_description=_safetensors_description(r),
                                   path=PurePosixPath(remote).as_posix(), blocks=blocks, mode=mode & 0o7777,
                                   size=r.nbytes))
    return out


def use_md5(url: str) -> bool:
    """Attach Content-MD5 only for real S3 / R2 hosts (moto and local fakes reject it; reference :708-727)."""
    host = urlparse(url).netloc.split(":")[0]
    if host.endswith((".amazonaws.com", ".r2.cloudflarestorage.com")):
        return True
    if host == "localhost":
        return False
    try:
        import ipaddress

        addr = ipaddress.ip_address(host)
        if addr.is_private or addr.is_loopback:
            return False
    except ValueError:
        pass
    raise Exception(f"Unknown S3 host: {host}")
