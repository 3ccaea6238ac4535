"""oracle/ref_shim.py -- TEST INFRASTRUCTURE ONLY; needs a source checkout of the original modal client,
named by ``B200H_REFERENCE_ROOT``.

Loads the reference's UNMODIFIED hash_utils.py / blob_utils.py / bytes_io_segment_payload.py
straight from <checkout>/py/modal/_utils without grpclib / synchronicity / generated
protos, by pre-seeding sys.modules so that modal/__init__.py never executes (SURVEY.md
Appendix A).  Used by oracle/gen_golden.py to produce tests/golden/*.json, which is all the tests read.
"""
from __future__ import annotations

import asyncio
import contextlib
import importlib
import logging
import os
import sys
import types


def _candidates():
    """Where an unmodified copy of the reference's ``modal`` package may live: below ``B200H_REFERENCE_ROOT``
    (a source checkout, or a ``pip install --target`` of one)."""
    env = os.environ.get("B200H_REFERENCE_ROOT")
    if env:
        yield os.path.join(env, "py", "modal")
        yield os.path.join(env, "modal")


def package_dir() -> str | None:
    for c in _candidates():
        if os.path.isfile(os.path.join(c, "_utils", "hash_utils.py")):
            return c
    return None


def _stub(name: str, **attrs) -> types.ModuleType:
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


_loaded = None


def load():
    """-> (ref_hash_utils, ref_blob_utils, ref_segment_payload) modules of the reference."""
    global _loaded
    if _loaded is not None:
        return _loaded
    pkg = package_dir()
    if pkg is None:
        raise RuntimeError("no copy of the reference found (set B200H_REFERENCE_ROOT)")
    if "modal" in sys.modules and not getattr(sys.modules["modal"], "_b200h_shim", False):
        raise RuntimeError("a real `modal` package is already imported; shim needs a clean process")

    class ExecutionError(Exception):
        pass

    def retry(direct_fn=None, **_kw):
        passthrough = lambda fn: fn  # noqa: E731
        return passthrough(direct_fn) if direct_fn else passthrough

    @contextlib.asynccontextmanager
    async def asyncnullcontext(*_a, **_k):
        yield

    class TaskContext:
        @staticmethod
        async def gather(*coros):
            return await asyncio.gather(*coros)

    shell = _stub("modal", _b200h_shim=True)
    shell.__path__ = []
    _stub("modal.config", logger=logging.getLogger("modal-ref"), config={})
    _stub("modal.exception", ExecutionError=ExecutionError)
    utils = _stub("modal._utils")
    utils.__path__ = [os.path.join(pkg, "_utils")]
    _stub(
        "modal._utils.async_utils",
        retry=retry,
        asyncnullcontext=asyncnullcontext,
        TaskContext=TaskContext,
        on_shutdown=lambda coro: None,
    )
    _stub("modal_proto").__path__ = []
    _stub("modal_proto.api_pb2")
    _stub("modal_proto.modal_api_grpc", ModalClientModal=object)
    h = importlib.import_module("modal._utils.hash_utils")
    b = importlib.import_module("modal._utils.blob_utils")
    s = importlib.import_module("modal._utils.bytes_io_segment_payload")
    _loaded = (h, b, s)
    return _loaded


def load_blob_utils_on(hash_utils_module):
    """The reference's UNMODIFIED blob_utils.py executed with ``modal._utils.hash_utils`` replaced by
    ``hash_utils_module`` -- i.e. the drop-in seam exercised from the reference's side: its own spec builders,
    block gatherer and multipart code calling somebody else's ``get_upload_hashes``.  The substitution only
    lasts for the import; the module returned is private (not left in sys.modules)."""
    import importlib.util
    from unittest import mock

    load()  # stubs for modal.config / exception / async_utils / protobufs
    path = os.path.join(package_dir(), "_utils", "blob_utils.py")
    name = "modal._utils.blob_utils_dropin"
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    mod.__package__ = "modal._utils"
    with mock.patch.dict(sys.modules, {"modal._utils.hash_utils": hash_utils_module, name: mod}):
        spec.loader.exec_module(mod)
    return mod
