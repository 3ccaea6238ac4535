"""Device groups on the GPU: batches split over several contexts, checked bit for bit against the oracle.

Groups [0, 0] and [0, 0, 0, 0] put several members on one B200, which covers the whole split-and-scatter path on a
single-GPU box; the group over every visible device needs two or more.  min_share_bytes=1 makes small batches split."""
import os
import threading

import numpy as np
import pytest

from modal_client_b200 import _backend, _lib
from modal_client_b200.synth import synth_array
from oracle import c_oracle
from tests.test_host_layer import test_blocks_golden as blocks_golden
from tests.test_host_layer import test_file_specs_golden as file_specs_golden
from tests.test_mount_upload import test_load_mount_checksums_dedupes_and_uploads as load_mount_checksums
from tests.test_volume_upload import test_batch_upload_v2_missing_block_loop as batch_upload_v2_missing_block_loop

pytestmark = pytest.mark.gpu

MiB = 1 << 20
SM = _lib.SHA256 | _lib.MD5


def _device_count():
    import torch

    return torch.cuda.device_count()


@pytest.fixture(scope="module", params=["0,0", "0,0,0,0", "every device"])
def group(request):
    if request.param == "every device":
        n = _device_count()
        if n < 2:
            pytest.skip(f"a group over distinct GPUs needs 2 or more; this box has {n}")
        devices = list(range(n))
    else:
        devices = [int(d) for d in request.param.split(",")]
    g = _lib.DeviceGroup(devices, pinned_bytes=64 * MiB, device_bytes=512 * MiB, min_share_bytes=1)
    yield g
    g.close()


def _mixed_batch(seed=3):
    """Mixed lengths at unaligned offsets, with blank messages and trailing-zero runs for TRIM_ZEROS."""
    rng = np.random.default_rng(seed)
    lens = [0, 1, 55, 56, 64, 65, 4096, 256 * 1024, 8 * MiB, 64 * MiB]
    lens += rng.integers(0, 300_000, 60).tolist()
    lens = np.array(lens, np.uint64)
    rng.shuffle(lens)
    gaps = rng.integers(1, 40, lens.size).astype(np.uint64)
    offs = (np.concatenate([[0], np.cumsum(lens + gaps)])[:-1] + 3).astype(np.uint64)
    total = int(offs[-1] + lens[-1]) + 64
    buf = synth_array(seed, total).copy()
    for i in range(0, lens.size, 7):  # blank messages
        buf[int(offs[i]) : int(offs[i] + lens[i])] = 0
    for i in range(3, lens.size, 5):  # trailing zeros
        o, n = int(offs[i]), int(lens[i])
        buf[o + n // 2 : o + n] = 0
    return buf, offs, lens


def _hex(rows):
    return np.frombuffer(rows.tobytes().hex().encode(), np.uint8).reshape(rows.shape[0], 2 * rows.shape[1])


@pytest.fixture(scope="module")
def mixed():
    buf, offs, lens = _mixed_batch()
    plain = c_oracle.hash_batch(buf, offs, lens, trim=False)
    trimmed = c_oracle.hash_batch(buf, offs, lens, trim=True)
    return buf, offs, lens, plain, trimmed


FLAG_SETS = [SM, _lib.SHA256, _lib.MD5, SM | _lib.TRIM_ZEROS, SM | _lib.HEX_OUT]


def _check(flags, got, plain, trimmed):
    s, m, e = trimmed if flags & _lib.TRIM_ZEROS else plain
    if flags & _lib.HEX_OUT:
        s, m = _hex(s), _hex(m)
    sha, md5, ln = got
    assert (sha is None) == (not flags & _lib.SHA256) and (md5 is None) == (not flags & _lib.MD5)
    if sha is not None:
        assert np.array_equal(sha, s)
    if md5 is not None:
        assert np.array_equal(md5, m)
    assert np.array_equal(ln, e)


@pytest.mark.parametrize("flags", FLAG_SETS)
@pytest.mark.parametrize("source", ["pageable", "host_alloc"])
def test_hash_batch_host_matches_the_oracle(group, mixed, flags, source):
    buf, offs, lens, plain, trimmed = mixed
    if source == "host_alloc":
        base = group.host_alloc(buf.size)
        base[:] = buf
    else:
        base = buf
    try:
        _check(flags, group.hash_batch_host(base, offs, lens, flags), plain, trimmed)
        split = group.last_split()
        assert sum(1 for r in split if r["messages"]) == min(len(group.devices), lens.size)
        assert sum(r["messages"] for r in split) == lens.size and sum(r["bytes"] for r in split) == int(lens.sum())
    finally:
        if source == "host_alloc":
            group.host_free(base)


def _device_tables(group, flags, n, device):
    import torch

    wide = 2 if flags & _lib.HEX_OUT else 1
    dev = torch.device("cuda", device)
    sha = torch.full((n, 32 * wide), 7, dtype=torch.uint8, device=dev)
    md5 = torch.full((n, 16 * wide), 7, dtype=torch.uint8, device=dev)
    ln = torch.zeros(n, dtype=torch.int64, device=dev)
    return sha, md5, ln


@pytest.mark.parametrize("flags", [SM, SM | _lib.TRIM_ZEROS, SM | _lib.HEX_OUT])
@pytest.mark.parametrize("table", ["home", "other member"])
def test_device_outputs_land_in_one_table(group, mixed, flags, table):
    buf, offs, lens, plain, trimmed = mixed
    if table == "home":
        device = group.devices[0]
    else:
        others = [d for d in group.devices if d != group.devices[0]]
        if not others:
            pytest.skip("every member sits on the home device: no other device to hold the table")
        device = others[0]
    sha, md5, ln = _device_tables(group, flags, lens.size, device)
    got = group.hash_batch_host(buf, offs, lens, flags, out_sha=sha.data_ptr(), out_md5=md5.data_ptr(),
                                out_trimmed=ln.data_ptr())
    assert got == (None, None, None)
    import torch

    torch.cuda.synchronize(device)
    _check(flags, (sha.cpu().numpy(), md5.cpu().numpy(), ln.cpu().numpy().astype(np.uint64)), plain, trimmed)


def test_device_outputs_on_two_devices_are_refused(group, mixed):
    if len(set(group.devices)) < 2:
        pytest.skip("needs members on two distinct GPUs")
    buf, offs, lens, _, _ = mixed
    sha, _, _ = _device_tables(group, SM, lens.size, group.devices[0])
    _, md5, _ = _device_tables(group, SM, lens.size, group.devices[1])
    with pytest.raises(_lib.B200HashError, match="one device"):
        group.hash_batch_host(buf, offs, lens, SM, out_sha=sha.data_ptr(), out_md5=md5.data_ptr())


def test_pinned_source_is_dma_ed_by_every_member(group):
    """host_alloc memory is portable: every member DMAs its share straight from it, nothing is re-staged."""
    lens = np.full(32, 4 * MiB, np.uint64)
    offs = (np.arange(32, dtype=np.uint64) * np.uint64(4 * MiB + 16)).astype(np.uint64)
    data = synth_array(11, int(offs[-1] + lens[-1]))
    pinned = group.host_alloc(data.size)
    try:
        pinned[:] = data
        want = c_oracle.hash_batch(data, offs, lens)
        _check(SM, group.hash_batch_host(pinned, offs, lens, SM), want, want)
        used = [r for r in group.last_split() if r["messages"]]
        assert len(used) == min(len(group.devices), 32)
        assert all(r["staged_bytes"] == 0 for r in used), group.last_split()
    finally:
        group.host_free(pinned)
    _check(SM, group.hash_batch_host(data, offs, lens, SM), want, want)  # pageable: every byte goes through the ring
    assert all(r["staged_bytes"] == r["bytes"] for r in group.last_split())


def test_small_batch_stays_home_at_the_default_threshold(mixed):
    buf, offs, lens, plain, trimmed = mixed
    g = _lib.DeviceGroup([0, 0], pinned_bytes=64 * MiB, device_bytes=512 * MiB)
    try:
        small = lens < 300_000
        _check(SM, g.hash_batch_host(buf, offs[small], lens[small], SM),
               tuple(x[small] for x in plain), tuple(x[small] for x in trimmed))
        split = g.last_split()
        assert split[0]["messages"] == int(small.sum()) and split[1]["messages"] == 0
        # at the same threshold, 1 GiB of 8 MiB messages is dealt over both members
        lens8 = np.full(128, 8 * MiB, np.uint64)
        big = synth_array(5, int(lens8.sum()))
        offs8 = np.arange(128, dtype=np.uint64) * np.uint64(8 * MiB)
        want = c_oracle.hash_batch(big, offs8, lens8)
        _check(SM, g.hash_batch_host(big, offs8, lens8, SM), want, want)
        assert [r["messages"] for r in g.last_split()] == [64, 64]
    finally:
        g.close()


# ------------------------------------------------------------------------------------------------------ files


@pytest.fixture(scope="module")
def tree(tmp_path_factory):
    root = tmp_path_factory.mktemp("group_tree")
    rng = np.random.default_rng(9)
    sizes = [0, 0, 1, 8 * MiB, 8 * MiB + 1, 3 * 8 * MiB + 5, 16 * MiB, 12 * MiB] + rng.integers(0, 200_000, 80).tolist()
    paths, contents = [], []
    for i, n in enumerate(sizes):
        data = synth_array(100 + i, n).copy()
        if i == 6:
            data[:] = 0  # blank blocks
        if i == 7:
            data[5 * MiB :] = 0  # a block with trailing zeros, then a blank one
        p = root / f"f{i:03d}.bin"
        p.write_bytes(data.tobytes())
        paths.append(str(p))
        contents.append(data)
    return paths, contents


def _oracle_files(contents, part_len, trim):
    offs, lens, chunks, at = [], [], [], 0
    for c in contents:
        spans = [(0, c.size)] if part_len == 0 else [(o, min(part_len, c.size - o)) for o in range(0, c.size, part_len)]
        for o, n in spans:
            offs.append(at + o)
            lens.append(n)
        chunks.append(c)
        at += c.size
    buf = np.concatenate(chunks) if chunks else np.zeros(0, np.uint8)
    return c_oracle.hash_batch(buf, np.array(offs, np.uint64), np.array(lens, np.uint64), trim=trim)


@pytest.mark.parametrize("part_len, flags", [(0, SM), (8 * MiB, _lib.SHA256 | _lib.TRIM_ZEROS)])
def test_hash_files_matches_the_oracle_and_one_context(group, tree, part_len, flags):
    paths, contents = tree
    sizes, _ = group.stat_files(paths)
    got = group.hash_files(paths, sizes, part_len, flags)
    want = _oracle_files(contents, part_len, bool(flags & _lib.TRIM_ZEROS))
    _check(flags, got, want, want)
    assert sum(1 for r in group.last_split() if r["messages"]) > 1
    one = _lib.Context(0, pinned_bytes=64 * MiB, device_bytes=512 * MiB)
    try:
        ref = one.hash_files(paths, sizes, part_len, flags)
    finally:
        one.close()
    for a, b in zip(got, ref):
        assert (a is None and b is None) or np.array_equal(a, b)


def test_file_truncated_after_stat_names_the_path_and_the_group_recovers(group, tmp_path):
    paths = []
    for i in range(12):
        p = tmp_path / f"t{i}.bin"
        p.write_bytes(synth_array(300 + i, 3 * MiB + i).tobytes())
        paths.append(str(p))
    sizes, _ = group.stat_files(paths)
    victim = paths[5]
    os.truncate(victim, 1000)
    with pytest.raises(_lib.B200HashError, match=rf"member \d+ \(cuda:\d+\): .*{os.path.basename(victim)}"):
        group.hash_files(paths, sizes, 0, SM)
    sizes, _ = group.stat_files(paths)
    contents = [np.fromfile(p, np.uint8) for p in paths]
    want = _oracle_files(contents, 0, False)
    _check(SM, group.hash_files(paths, sizes, 0, SM), want, want)


def test_concurrent_callers_get_their_own_rows(group):
    results, errors = {}, []

    def worker(t):
        try:
            rng = np.random.default_rng(50 + t)
            lens = rng.integers(0, 2 * MiB, 40 + t).astype(np.uint64)
            offs = (np.concatenate([[0], np.cumsum(lens)])[:-1]).astype(np.uint64)
            buf = synth_array(60 + t, int(lens.sum()) + 1)
            for _ in range(3):
                got = group.hash_batch_host(buf, offs, lens, SM)
            results[t] = (got, c_oracle.hash_batch(buf, offs, lens))
        except Exception as e:  # surfaced below
            errors.append(e)

    threads = [threading.Thread(target=worker, args=(t,)) for t in range(4)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors
    for got, want in results.values():
        _check(SM, got, want, want)


def test_launch_count_sums_the_members(group, mixed):
    buf, offs, lens, _, _ = mixed
    before = group.launch_count
    group.hash_batch_host(buf, offs, lens, SM)
    assert group.launch_count >= before + min(len(group.devices), lens.size)


# ---------------------------------------------------------------------------- drop-in checks through a group


@pytest.fixture
def group_backend(group, monkeypatch):
    monkeypatch.setattr(_backend, "_override", group)
    return group


def test_file_specs_golden_through_a_group(group_backend, golden, monkeypatch, tmp_path):
    file_specs_golden(group_backend, golden, monkeypatch, tmp_path)


def test_blocks_golden_through_a_group(group_backend, golden, monkeypatch):
    blocks_golden(group_backend, golden, monkeypatch)


def test_batch_upload_v2_through_a_group(group_backend, monkeypatch, tmp_path):
    batch_upload_v2_missing_block_loop(group_backend, monkeypatch, tmp_path)


def test_mount_checksums_through_a_group(group_backend, monkeypatch, tmp_path):
    load_mount_checksums(group_backend, monkeypatch, tmp_path)
