"""modal_client_b200 -- B200-native blob-ingest / content-hash path behind the Modal client's function surface.

Drop-in modules (same names as the reference's ``modal/_utils``): ``hash_utils``, ``blob_utils``,
``bytes_io_segment_payload``, ``function_utils``, ``parallel_map``.  B200 additions: ``batch`` (digest
tables), ``sharding`` (multi-GPU, one process per GPU), ``use_devices`` (one process, several GPUs), ``_lib``
(ctypes binding of libb200hash.so, C ABI in include/b200hash.h).
All arithmetic runs in hand-written sm_100a CUDA; there is no CPU fallback.
"""
__version__ = "0.1.0"

from . import _lib  # noqa: F401  (symbols only; touching the GPU happens on first use)
from ._backend import use_devices  # noqa: F401
from .batch import DigestTable, hash_table_buffers, hash_table_host  # noqa: F401
from .hash_utils import UploadHashes, get_upload_hashes, get_upload_hashes_many  # noqa: F401
