"""``Volume.batch_upload()`` on the B200 hash path.

Counterparts of ``_VolumeUploadContextManager`` (volumefs1: whole-file SHA-256 + MD5, dedupe through
``MountPutFile``, py/modal/volume.py:1181-1333) and ``_VolumeUploadContextManager2`` (volumefs2: SHA-256 of every
zero-trimmed 8 MiB block, ``VolumePutFiles2`` missing-block loop, :1345-1574).  Same ``put_file`` /
``put_directory`` surface and the same RPC / PUT sequence; what changes is *when hashing happens*: the reference
hashes file by file (ThreadPoolExecutor) or block by block (``to_thread`` under a semaphore); here every path
queued in the batch is handed to ``blob_utils.get_file_upload_specs`` / ``file_upload_specs2`` -- ONE GPU
batch for the whole tree -- before the first RPC goes out.  File objects (``BytesIO`` / open files) keep the
per-object spec builders.  CUDA tensors (``put_tensor``) are hashed in HBM by ``blob_utils.tensor_upload_specs`` /
``tensor_upload_specs2`` -- one device call per batch -- and read back only for the bytes that are sent; state dicts
(``put_safetensors``) likewise, framed as safetensors files, by ``safetensors_upload_specs`` / ``_specs2``.
"""
from __future__ import annotations

import asyncio
import functools
import os
import time
from collections.abc import Callable
from io import BytesIO
from pathlib import Path, PurePosixPath
from typing import Any, BinaryIO

import numpy as np

from . import _wire, blob_utils
from ._logging import logger
from .async_utils import bounded_map, retry
from .blob_utils import FileUploadSpec, FileUploadSpec2, _ByteBudget
from .exception import ExecutionError
from .http_utils import ClientSessionRegistry

VOLUME_PUT_FILE_CLIENT_TIMEOUT = 60 * 60  # seconds a single file may take to become visible (volume.py:79)


class VolumeUploadTimeoutError(TimeoutError):
    pass


class _BatchBase:
    def __init__(self, volume_id: str, client, progress_cb: Callable[..., Any] | None = None, force: bool = False):
        self._volume_id = volume_id
        self._client = client
        self._progress_cb = progress_cb or (lambda *_, **__: None)
        self._force = force
        self._paths: list[tuple[Path | str, str, int | None]] = []  # (local path, remote posix path, mode)
        self._fileobjs: list[tuple[BinaryIO, PurePosixPath, int]] = []
        self._tensors: list[tuple[blob_utils.DeviceBufferReader, str, int]] = []
        self._safetensors: list[tuple[blob_utils.DeviceSegmentsReader, str, int]] = []

    async def __aenter__(self):
        return self

    def put_file(self, local_file: Path | str | BinaryIO | BytesIO, remote_path: PurePosixPath | str, mode: int | None = None):
        """Queue one file (path or readable file object; objects must stay readable until the batch exits)."""
        remote = PurePosixPath(remote_path).as_posix()
        if remote.endswith("/"):
            raise ValueError(f"remote_path ({remote}) must refer to a file - cannot end with /")
        if isinstance(local_file, (str, Path)):
            self._paths.append((local_file, remote, mode))
        else:
            self._fileobjs.append((local_file, PurePosixPath(remote), mode or 0o644))

    def put_tensor(self, tensor, remote_path: PurePosixPath | str, mode: int | None = None):
        """Queue the raw bytes of a contiguous CUDA tensor (or a ``function_utils.DevicePayload``) as one file at
        ``remote_path`` (mode 0o644 unless given): ``numel * element_size`` bytes from ``data_ptr()``, any dtype, no
        header.  A state dict that should load back as a checkpoint goes through ``put_safetensors``, which frames it
        as a safetensors file with the tensors still in HBM.

        The bytes are hashed where they are, on the GPU that holds them (each GPU of a device group hashes its own
        tensors), in one call for all tensors of the batch; only bytes that must be sent are copied to the host, through
        a small pinned buffer.  volumefs2 sends the zero-trimmed 8 MiB blocks the server reports missing, so re-saving
        mostly unchanged weights moves little.  volumefs1 needs a whole-tensor SHA-256 (+ MD5 up to 1 GiB): each is one
        serial chain on the device, about 71 MB/s -- roughly 15 s per GiB -- and the whole content is uploaded when
        the server lacks it.

        Work already queued on the tensor's current stream is part of what is uploaded.  The tensor must not be modified
        (nor freed and reused) until the batch exits, like a queued file object.  Raises ``ValueError`` now for a
        non-CUDA or non-contiguous tensor, a tensor on a device the current context or device group does not cover, or
        a ``remote_path`` that ends in ``/``."""
        from .function_utils import DevicePayload

        remote = PurePosixPath(remote_path).as_posix()
        if remote.endswith("/"):
            raise ValueError(f"remote_path ({remote}) must refer to a file - cannot end with /")
        if isinstance(tensor, DevicePayload):
            tensor = tensor.tensor
        if not getattr(tensor, "is_cuda", False):
            raise ValueError(f"put_tensor needs a CUDA tensor, got {getattr(tensor, 'device', type(tensor).__name__)}; "
                             "queue host data with put_file")
        if not tensor.is_contiguous():
            raise ValueError("put_tensor needs a contiguous tensor: call .contiguous() first")
        covered = _context_devices(blob_utils.get_context())
        if covered is not None and tensor.device.index not in covered:
            raise ValueError(f"the tensor is on cuda:{tensor.device.index}, which the current context / device group "
                             f"does not cover (devices {sorted(set(covered))})")
        self._tensors.append((blob_utils.DeviceBufferReader(tensor), remote, mode or 0o644))

    def put_safetensors(self, tensors, remote_path: PurePosixPath | str, *, metadata: dict[str, str] | None = None,
                        mode: int | None = None):
        """Queue a state dict as one safetensors file at ``remote_path`` (mode 0o644 unless given): byte for byte what
        ``safetensors.torch.save(tensors, metadata)`` writes (``blob_utils.safetensors_layout``), without copying the
        tensors out of HBM to build it.  The file is the small header followed by the tensors' raw bytes; its blocks
        are hashed on the GPU that holds the tensors (parts that straddle two tensors are gathered there first), in one
        call for every file of the batch, and only the bytes that must be sent are copied to the host.  volumefs2
        sends the zero-trimmed 8 MiB blocks the server reports missing, so re-saving a fine-tune whose frozen layers
        did not change sends little more than the changed tensors' blocks.  volumefs1 needs a whole-file SHA-256
        (+ MD5 up to 1 GiB): the file is gathered whole into scratch on the device and each digest is one serial
        chain, about 71 MB/s -- roughly 15 s per GiB.

        Work already queued on the device's current stream is part of what is uploaded; the tensors must not be
        modified (nor freed and reused) until the batch exits.  Raises ``ValueError`` now, queueing nothing, for a
        non-str name or one equal to ``__metadata__``, a non-CUDA or non-contiguous tensor, tensors on more than one
        device or on a device the current context / device group does not cover, tensors that share storage, a dtype
        safetensors cannot store, non-str metadata, or a ``remote_path`` that ends in ``/``."""
        remote = PurePosixPath(remote_path).as_posix()
        if remote.endswith("/"):
            raise ValueError(f"remote_path ({remote}) must refer to a file - cannot end with /")
        if metadata is not None and not all(isinstance(k, str) and isinstance(v, str) for k, v in metadata.items()):
            raise ValueError("put_safetensors metadata must map str to str")
        devices, storages = set(), {}
        for name, t in tensors.items():
            if not isinstance(name, str):
                raise ValueError(f"put_safetensors needs str tensor names, got {name!r}")
            if name == "__metadata__":
                raise ValueError("'__metadata__' is reserved by the safetensors format and cannot name a tensor")
            if not getattr(t, "is_cuda", False):
                raise ValueError(f"tensor {name!r} is not a CUDA tensor "
                                 f"({getattr(t, 'device', type(t).__name__)}); put_safetensors uploads from HBM")
            if not t.is_contiguous():
                raise ValueError(f"tensor {name!r} is not contiguous: call .contiguous() first")
            devices.add(t.device.index)
            if t.numel() and t.untyped_storage().nbytes():
                other = storages.setdefault(t.untyped_storage().data_ptr(), name)
                if other != name:
                    raise ValueError(f"tensors {other!r} and {name!r} share storage, which safetensors refuses: "
                                     "save a .clone() of one of them")
        if len(devices) > 1:
            raise ValueError(f"put_safetensors needs every tensor on one device, got cuda:{sorted(devices)}")
        header, ordered = blob_utils.safetensors_layout(tensors, metadata)
        if devices:
            device = devices.pop()
            covered = _context_devices(blob_utils.get_context())
            if covered is not None and device not in covered:
                raise ValueError(f"the tensors are on cuda:{device}, which the current context / device group "
                                 f"does not cover (devices {sorted(set(covered))})")
        else:
            raise ValueError("put_safetensors needs at least one CUDA tensor (the file is built on its device)")
        reader = blob_utils.DeviceSegmentsReader(header, [t for _, t in ordered])
        self._safetensors.append((reader, remote, mode or 0o644))

    def put_directory(self, local_path: Path | str, remote_path: PurePosixPath | str, recursive: bool = True):
        """Queue every regular file below ``local_path`` (directories and special files are skipped).

        Same selection as the reference's ``rglob("*")`` + ``is_file()`` (py/modal/volume.py:1279-1284): symlinks to
        files count, symlinked directories are not descended into, fifos / devices are skipped.  The walk itself is
        ``os.scandir`` on plain strings: with hashing down to a fraction of a second, ``pathlib``'s ~15 us per file
        (glob + ``is_file`` + ``relative_to`` + ``/``) would be most of a million-file upload."""
        local_path = Path(local_path)
        assert local_path.is_dir()
        remote_root = PurePosixPath(remote_path).as_posix().rstrip("/")
        append = self._paths.append
        for abs_path, rel_posix in _walk_files(os.fspath(local_path), recursive):
            append((abs_path, f"{remote_root}/{rel_posix}", None))


def _context_devices(ctx) -> list[int] | None:
    """CUDA devices a context (one device) or a device group (its members' devices) hashes on; None when unknown."""
    devices = getattr(ctx, "devices", None)
    if devices is None:
        device = getattr(ctx, "device", None)
        devices = None if device is None or device < 0 else [device]
    return devices


def _walk_files(root: str, recursive: bool):
    """Yield (absolute path, path relative to ``root`` in posix form) of every regular file (or symlink to one)."""
    stack = [(root, "")]
    sep_is_posix = os.sep == "/"
    while stack:
        d, rel = stack.pop()
        try:
            it = os.scandir(d)
        except OSError:
            continue  # vanished or unreadable directory: pathlib's glob skips those too
        with it:
            for e in it:
                name = e.name
                try:
                    if e.is_dir(follow_symlinks=False):
                        if recursive:
                            stack.append((e.path, f"{rel}{name}/"))
                    elif e.is_file():  # follows symlinks, like Path.is_file()
                        yield e.path, (f"{rel}{name}" if sep_is_posix else f"{rel}{name}".replace(os.sep, "/"))
                except OSError:
                    continue


class VolumeUploadContextManager(_BatchBase):
    """volumefs1 batch upload: one fused SHA-256+MD5 GPU batch over all queued paths, then dedupe + upload."""

    def __init__(self, volume_id: str, client, progress_cb=None, force: bool = False):
        super().__init__(volume_id, client, progress_cb, force)
        self._byte_budget = _ByteBudget.from_system_memory()

    async def __aexit__(self, exc_type, exc_val, exc_tb):
        if exc_val:
            return
        specs: list[FileUploadSpec] = await asyncio.to_thread(blob_utils.get_file_upload_specs, self._paths)
        for fp, remote, mode in self._fileobjs:
            specs.append(await asyncio.to_thread(blob_utils.get_file_upload_spec_from_fileobj, fp, remote, mode))
        specs.extend(await asyncio.to_thread(blob_utils.tensor_upload_specs, self._tensors))
        specs.extend(await asyncio.to_thread(blob_utils.safetensors_upload_specs, self._safetensors))
        logger.debug(f"Computed checksums for {len(specs)} files on the GPU")
        # In-batch dedupe on the digest table, computed on the GPU (b200h_dedupe_host; what Mount does with a set,
        # py/modal/mount.py:498,518-534): each distinct content is checked / uploaded once, however many paths carry
        # it; the other paths only appear in the file index.  20 uploads in flight, like the reference (volume.py:1220).
        first, _ = await asyncio.to_thread(blob_utils.first_occurrence_of_specs, specs)
        owners = [i for i, f in enumerate(first) if f == i]
        await bounded_map(owners, lambda i: self._upload_file(specs[i]), concurrency=20)
        for i, spec in enumerate(specs):
            if first[i] != i:  # a copy of something already sent: account for it in the progress display
                self._progress_cb(task_id=self._progress_cb(name=spec.mount_filename, size=spec.size), complete=True)
        files = [_wire.MountFile(filename=s.mount_filename, sha256_hex=s.sha256_hex, mode=s.mode) for s in specs]
        self._progress_cb(complete=True)
        request = _wire.VolumePutFilesRequest(volume_id=self._volume_id, files=files,
                                              disallow_overwrite_existing_files=not self._force)
        try:
            await self._client.stub.VolumePutFiles(request)
        except Exception as exc:
            if type(exc).__name__ == "AlreadyExistsError":
                raise FileExistsError(str(exc))
            raise

    async def _upload_file(self, spec: FileUploadSpec):
        task_id = self._progress_cb(name=spec.mount_filename, size=spec.size)
        stub = self._client.stub
        response = await stub.MountPutFile(_wire.MountPutFileRequest(sha256_hex=spec.sha256_hex))
        if response.exists:  # content-addressed dedupe: nothing to send
            self._progress_cb(task_id=task_id, complete=True)
        else:
            started = time.monotonic()
            if spec.use_blob:
                with spec.source() as fp:
                    blob_id = await blob_utils.blob_upload_file(
                        fp, stub, functools.partial(self._progress_cb, task_id), sha256_hex=spec.sha256_hex,
                        md5_hex=spec.md5_hex, byte_budget=self._byte_budget)
                request2 = _wire.MountPutFileRequest(data_blob_id=blob_id, sha256_hex=spec.sha256_hex)
            else:
                content = spec.content if spec.content is not None else await asyncio.to_thread(spec.read_content)
                request2 = _wire.MountPutFileRequest(data=content, sha256_hex=spec.sha256_hex)
                self._progress_cb(task_id=task_id, complete=True)
            while True:
                response = await stub.MountPutFile(request2)
                if response.exists:
                    break
                if time.monotonic() - started >= VOLUME_PUT_FILE_CLIENT_TIMEOUT:
                    raise VolumeUploadTimeoutError(f"Uploading of {spec.source_description} timed out")
        return _wire.MountFile(filename=spec.mount_filename, sha256_hex=spec.sha256_hex, mode=spec.mode)


class VolumeUploadContextManager2(_BatchBase):
    """volumefs2 batch upload: all 8 MiB blocks of all queued files form one GPU batch (trim scan + SHA-256)."""

    def __init__(self, volume_id: str, client, progress_cb=None, force: bool = False,
                 hash_concurrency: int | None = None, put_concurrency: int = 128):
        super().__init__(volume_id, client, progress_cb, force)
        # the reference hashes blocks under a semaphore of ``hash_concurrency`` = cpu_count executor threads
        # (volume.py:1358,1383); here every block of every file is one GPU batch, so the knob is accepted and unused
        self._hash_concurrency = hash_concurrency
        self._put_concurrency = put_concurrency

    async def __aexit__(self, exc_type, exc_val, exc_tb):
        if exc_val:
            return
        specs: list[FileUploadSpec2] = await blob_utils.file_upload_specs2(self._paths)
        one_at_a_time = asyncio.Semaphore(1)
        for fp, remote, mode in self._fileobjs:
            specs.append(await FileUploadSpec2.from_fileobj(fp, remote, one_at_a_time, mode))
        specs.extend(await asyncio.to_thread(blob_utils.tensor_upload_specs2, self._tensors))
        specs.extend(await asyncio.to_thread(blob_utils.safetensors_upload_specs2, self._safetensors))
        await self._put_file_specs(specs)

    async def _put_file_specs(self, file_specs: list[FileUploadSpec2]):
        put_responses: dict[bytes, bytes] = {}
        B = _wire.VolumePutFiles2Request
        for _attempt in range(2):  # once to learn the missing blocks, once more with every put_response
            files = [
                B.File(path=s.path, mode=s.mode, size=s.size,
                       blocks=[B.Block(contents_sha256=b.contents_sha256, put_response=put_responses.get(b.contents_sha256))
                               for b in s.blocks])
                for s in file_specs
            ]
            request = B(volume_id=self._volume_id, files=files, disallow_overwrite_existing_files=not self._force)
            try:
                response = await self._client.stub.VolumePutFiles2(request)
            except Exception as exc:
                if type(exc).__name__ == "AlreadyExistsError":
                    raise FileExistsError(str(exc))
                raise
            if not response.missing_blocks:
                break
            await _put_missing_blocks(file_specs, response.missing_blocks, put_responses, self._put_concurrency,
                                      self._progress_cb)
        else:
            raise RuntimeError("Did not succeed at uploading all files despite supplying all missing blocks")
        self._progress_cb(complete=True)


async def _put_missing_blocks(file_specs, missing_blocks, put_responses: dict[bytes, bytes], put_concurrency: int,
                              progress_cb: Callable[..., Any]):
    """PUT each block the server reported missing (only the zero-trimmed bytes travel) and remember the
    server's put_response per block digest (py/modal/volume.py:1500-1574)."""
    from .bytes_io_segment_payload import BytesIOSegmentPayload

    pending: dict[str, tuple[Any, set[int]]] = {}

    async def put_one(mb) -> tuple[bytes, bytes]:
        spec = file_specs[mb.file_index]
        block = spec.blocks[mb.block_index]
        if spec.path not in pending:
            pending[spec.path] = (progress_cb(name=spec.path, size=spec.size), set())
        task_id, waiting = pending[spec.path]
        waiting.add(mb.block_index)
        report = functools.partial(progress_cb, task_id=task_id)

        @retry(n_attempts=11, base_delay=0.5, attempt_timeout=None)  # reference: volume.py:1542
        async def attempt(payload) -> bytes:
            with payload.reset_on_error(subtract_progress=True):
                async with ClientSessionRegistry.get_session().put(mb.put_url, data=payload) as resp:
                    if resp.status != 200:
                        raise ExecutionError(f"block PUT failed with status {resp.status}: {await resp.text()}")
                    return await resp.content.read()

        with spec.source() as fp:
            # the block digest is already known (GPU batch): no re-hash while sending
            payload = BytesIOSegmentPayload(fp, block.start, block.end - block.start, chunk_size=256 * 1024,
                                            progress_report_cb=report, md5_digest=b"\0" * 16)
            data = await attempt(payload)
        waiting.discard(mb.block_index)
        if not waiting:
            report(complete=True)
        return block.contents_sha256, data

    # Identical blocks (the same content in several files, repeated runs inside one file) are sent once per round: the
    # put_response is kept per digest anyway (py/modal/volume.py:1464,1569).  First occurrences come from the GPU
    # dedupe over the digests of the missing blocks; the reference uploads every listed block.
    missing = list(missing_blocks)
    if len(missing) > 1:
        keys = np.frombuffer(b"".join(file_specs[mb.file_index].blocks[mb.block_index].contents_sha256 for mb in missing),
                             np.uint8).reshape(len(missing), 32)
        first, _ = await asyncio.to_thread(blob_utils.get_context().dedupe, keys)
        missing = [mb for i, mb in enumerate(missing) if first[i] == i]
    for digest, resp in await bounded_map(missing, put_one, concurrency=put_concurrency):
        put_responses[digest] = resp


# ---------------------------------------------------------------------------------- the reference's names

# enum VolumeFsVersion, modal_proto/api.proto:312-316
VOLUME_FS_VERSION_UNSPECIFIED, VOLUME_FS_VERSION_V1, VOLUME_FS_VERSION_V2 = 0, 1, 2


class _AbstractVolumeUploadContextManager:
    """The interface ``Volume.batch_upload`` hands out, and the version switch behind it (py/modal/volume.py:1137-1173)."""

    async def __aenter__(self): ...

    async def __aexit__(self, exc_type, exc_val, exc_tb): ...

    def put_file(self, local_file, remote_path, mode=None): ...

    def put_directory(self, local_path, remote_path, recursive=True): ...

    def put_tensor(self, tensor, remote_path, mode=None): ...

    def put_safetensors(self, tensors, remote_path, *, metadata=None, mode=None): ...

    @staticmethod
    def resolve(version, object_id: str, client, progress_cb: Callable[..., Any] | None = None, force: bool = False):
        if version in (None, VOLUME_FS_VERSION_UNSPECIFIED, VOLUME_FS_VERSION_V1):
            return VolumeUploadContextManager(object_id, client, progress_cb=progress_cb, force=force)
        if version == VOLUME_FS_VERSION_V2:
            return VolumeUploadContextManager2(object_id, client, progress_cb=progress_cb, force=force)
        raise RuntimeError(f"unsupported volume version: {version}")


# The reference keeps the implementation under the underscore name and exports a synchronicity wrapper under the plain
# one; there is no wrapper layer here, so both names mean the class itself.
AbstractVolumeUploadContextManager = _AbstractVolumeUploadContextManager
_VolumeUploadContextManager = VolumeUploadContextManager
_VolumeUploadContextManager2 = VolumeUploadContextManager2

