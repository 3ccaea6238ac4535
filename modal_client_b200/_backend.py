"""Where the host layer gets its GPU context from.

Everything above the C ABI (hash_utils, blob_utils, batch planners) calls ``get_context()``; by default
that is the process-wide ``_lib.default_context()`` (device = LOCAL_RANK).  ``set_context`` lets an
application pin a specific context.  ``use_devices`` (or ``B200H_DEVICES``) opts one process into a device
group: every batched call then deals its messages over several GPUs (``_lib.DeviceGroup``).  There is no CPU
implementation behind this seam: the unit tests substitute an oracle-backed stand-in here to exercise host logic
on machines without a GPU, which is test scaffolding, not a fallback -- production code never does that.
"""
from __future__ import annotations

import os
import threading

from . import _lib

_override = None
_devices = None  # None: one GPU (the default); "all" or a list of device ids: a device group
_devices_from_env = False  # B200H_DEVICES is read once, on the first get_context()
_group = None
_group_lock = threading.Lock()


def set_context(ctx) -> None:
    global _override
    _override = ctx


def _parse_devices(spec):
    if spec is None:
        return None
    if isinstance(spec, str) and spec.strip().lower() == "all":
        ids = "all"
    elif isinstance(spec, str):
        try:
            ids = [int(x) for x in spec.split(",")]
        except ValueError:
            raise ValueError(f"devices must be 'all' or a comma-separated list of device ids, got {spec!r}") from None
    else:
        ids = list(spec)
        if not all(isinstance(d, int) and not isinstance(d, bool) for d in ids):
            raise ValueError(f"devices must be 'all' or a list of device ids, got {spec!r}")
    if ids != "all" and (not ids or min(ids) < 0):
        raise ValueError(f"devices must name at least one device id >= 0, got {spec!r}")
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        raise ValueError("a device group cannot be used under torchrun (WORLD_SIZE > 1): every rank already owns one "
                         "GPU; shard across ranks with sharding.hash_table_sharded instead")
    return ids


def use_devices(devices) -> None:
    """Hash this process's batches on several GPUs: ``"all"``, a list of device ids (``[0, 1, 2, 3]``; a device may
    repeat) or a string like ``"0,1,2,3"``.  ``None`` restores the default of one GPU.  The environment variable
    ``B200H_DEVICES`` (``all`` / ``0,1,2,3``) does the same on the first ``get_context()``."""
    global _devices, _group, _devices_from_env
    parsed = _parse_devices(devices)
    with _group_lock:
        _devices, _group, _devices_from_env = parsed, None, True


def get_context():
    global _devices, _devices_from_env, _group
    if _override is not None:
        return _override
    if not _devices_from_env:
        with _group_lock:
            if not _devices_from_env:
                _devices = _parse_devices(os.environ.get("B200H_DEVICES") or None)
                _devices_from_env = True
    if _devices is None:
        return _lib.default_context()
    with _group_lock:
        if _group is None:
            _group = _lib.DeviceGroup(None if _devices == "all" else _devices)
        return _group


_pool: list = []


def context_pool(n: int) -> list:
    """``n`` contexts on this process's device for callers that keep several host batches in flight (the map pump
    hashes window k+1 while window k's tail is still on the GPU): the current context plus ``n-1`` more on the same
    device, created on first use.  A device group is returned ``n`` times: each window is already split over its
    members.  A stand-in installed by the tests is returned ``n`` times."""
    first = get_context()
    if isinstance(first, _lib.DeviceGroup) or not isinstance(first, _lib.Context):
        return [first] * n
    while len(_pool) < n - 1 or any(c.device != first.device or not getattr(c, "_h", None) for c in _pool):
        _pool[:] = [c for c in _pool if c.device == first.device and getattr(c, "_h", None)]
        if len(_pool) >= n - 1:
            break
        _pool.append(_lib.Context(first.device))
    return [first] + _pool[: n - 1]
