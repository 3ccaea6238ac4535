"""Mount creation (select -> GPU checksums -> GPU dedupe -> MountPutFile / blob upload -> MountGetOrCreate) against an
in-process fake that follows the reference's test servicer (py/test/conftest.py:2224-2231 MountPutFile,
:2233-2263 MountGetOrCreate) and the expectations of py/test/mount_test.py (sha256_hex equals hashlib on the file
bytes; blob path above LARGE_FILE_LIMIT; ignored files are not uploaded)."""
import asyncio
import hashlib
import os
import time
import types
from pathlib import Path, PurePosixPath

import numpy as np
import pytest

from modal_client_b200 import _wire, blob_utils, mount
from modal_client_b200.exception import ExecutionError
from modal_client_b200.synth import synth_bytes
from oracle import ref_port
from tests.blob_server import FakeBlobStub, running_blob_server


@pytest.fixture(params=["fake", pytest.param("gpu", marks=pytest.mark.gpu)])
def backend(request):
    return request.getfixturevalue("fake_backend" if request.param == "fake" else "gpu_backend")


class FakeMountStub(FakeBlobStub):
    def __init__(self, host, store):
        super().__init__(host, multipart_threshold=10_000_000)
        self.store = store
        self.files_sha2data, self.mount_contents, self.deployed_mounts = {}, {}, {}
        self.n_mounts = 0
        self.exist_checks, self.data_puts = [], []
        self.last_request = None

    async def MountPutFile(self, req):
        if req.WhichOneof("data_oneof") is not None:
            self.data_puts.append(req.sha256_hex)
            self.files_sha2data[req.sha256_hex] = {"data": req.data, "data_blob_id": req.data_blob_id}
            return types.SimpleNamespace(exists=True)
        self.exist_checks.append(req.sha256_hex)
        return types.SimpleNamespace(exists=req.sha256_hex in self.files_sha2data)

    async def MountGetOrCreate(self, req):
        self.last_request = req
        k = (req.deployment_name, req.namespace)
        if req.object_creation_type == _wire.OBJECT_CREATION_TYPE_CREATE_FAIL_IF_EXISTS and k in self.deployed_mounts:
            raise RuntimeError("already exists")
        self.n_mounts += 1
        mount_id = f"mo-{self.n_mounts}"
        if req.deployment_name:
            self.deployed_mounts[k] = mount_id
        self.mount_contents[mount_id] = {f.filename: (f.sha256_hex, f.mode) for f in req.files}
        return types.SimpleNamespace(mount_id=mount_id, handle_metadata=types.SimpleNamespace(
            content_checksum_sha256_hex="deadbeef"))

    def content_of(self, sha):
        d = self.files_sha2data[sha]
        return d["data"] if d["data"] is not None else self.store.blobs[d["data_blob_id"]]


def _make_tree(tmp_path):
    root = tmp_path / "pkg"
    (root / "sub" / "__pycache__").mkdir(parents=True)
    (root / ".git").mkdir()
    files = {
        "a.py": synth_bytes(1, 15),
        "sub/b.py": synth_bytes(2, 4000),
        "sub/c.bin": synth_bytes(3, 70_000),       # above the (patched) blob limit
        "sub/copy_of_a.py": synth_bytes(1, 15),    # same content as a.py -> deduped on the GPU
        "sub/copy2_of_a.py": synth_bytes(1, 15),
        "empty": b"",
        "sub/__pycache__/b.pyc": b"ignored bytecode",
        ".git/config": b"ignored dot dir",
    }
    for rel, data in files.items():
        (root / rel).write_bytes(data)
    os.chmod(root / "a.py", 0o755)
    return root, files


class PruningIgnore:
    """Shaped like the reference's pattern matchers: callable on the relative path, can prune directories."""

    def __init__(self):
        self.asked = []

    def can_prune_directories(self):
        return True

    def __call__(self, rel: Path) -> bool:
        self.asked.append(rel.as_posix())
        return rel.parts[0] == ".git" or "__pycache__" in rel.parts or rel.suffix == ".pyc"


def test_select_files_entries(tmp_path):
    root, files = _make_tree(tmp_path)
    ign = PruningIgnore()
    d = mount._MountDir(root, PurePosixPath("/root/pkg"), ign, True)
    sel = dict((r.as_posix(), p) for p, r in mount._select_files([d]))
    assert sorted(sel) == sorted(f"/root/pkg/{k}" for k in files if ".git" not in k and "__pycache__" not in k)
    assert not any(a.startswith(".git/") or a.startswith("sub/__pycache__/") for a in ign.asked)  # pruned, never walked
    flat = mount._MountDir(root, PurePosixPath("/x"), recursive=False)
    assert sorted(r.as_posix() for _, r in mount._select_files([flat])) == ["/x/a.py", "/x/empty"]
    one = mount._MountFile(root / "a.py", PurePosixPath("/root/a.py"))
    # overlapping entries select a (local, remote) pair once; the same local file under two names twice
    both = mount._select_files([d, d, one])
    assert len(both) == len(sel) + 1
    with pytest.raises(FileNotFoundError):
        mount._select_files([mount._MountFile(root / "nope", PurePosixPath("/n"))])
    with pytest.raises(NotADirectoryError):
        mount._select_files([mount._MountDir(root / "a.py", PurePosixPath("/n"))])
    with pytest.raises(FileNotFoundError):
        mount._select_files([mount._MountDir(root / "nodir", PurePosixPath("/n"))])


def test_load_mount_checksums_dedupes_and_uploads(backend, monkeypatch, tmp_path):
    monkeypatch.setattr(blob_utils, "LARGE_FILE_LIMIT", 20_000)

    async def run():
        async with running_blob_server() as (host, store):
            stub = FakeMountStub(host, store)
            root, files = _make_tree(tmp_path)
            entries = [mount._MountDir(root, PurePosixPath("/root/pkg"), PruningIgnore(), True)]
            resp = await mount.load_mount(entries, stub, app_id="ap-1")
            assert resp.mount_id == "mo-1" and stub.last_request.app_id == "ap-1"
            assert stub.last_request.object_creation_type == _wire.OBJECT_CREATION_TYPE_ANONYMOUS_OWNED_BY_APP
            kept = {k: v for k, v in files.items() if ".git" not in k and "__pycache__" not in k}
            index = stub.mount_contents["mo-1"]
            assert sorted(index) == sorted(f"/root/pkg/{k}" for k in kept)
            for rel, data in kept.items():
                sha, mode = index[f"/root/pkg/{rel}"]
                assert sha == hashlib.sha256(data).hexdigest()  # what py/test/mount_test.py:41,45,172 pin
                assert stub.content_of(sha) == data
            assert index["/root/pkg/a.py"][1] == 0o755
            # three paths share one content: ONE existence check and ONE data put for it (mount.py:518-534)
            distinct = {hashlib.sha256(d).hexdigest() for d in kept.values()}
            assert sorted(stub.exist_checks) == sorted(distinct) and sorted(stub.data_puts) == sorted(distinct)
            assert len(store.blobs) == 1  # only sub/c.bin went through the blob path
            # a second mount of the same tree: everything exists, nothing is sent
            stub.exist_checks.clear(), stub.data_puts.clear()
            resp2 = await mount.load_mount(entries, stub, deployment_name="my-mount", environment_name="main")
            assert resp2.mount_id == "mo-2" and stub.data_puts == [] and sorted(stub.exist_checks) == sorted(distinct)
            assert stub.last_request.object_creation_type == _wire.OBJECT_CREATION_TYPE_CREATE_FAIL_IF_EXISTS
            await mount.load_mount(entries, stub, deployment_name="other", allow_overwrite=True)
            assert stub.last_request.object_creation_type == _wire.OBJECT_CREATION_TYPE_CREATE_IF_MISSING
            # empty mount: still registered (the reference logs a warning)
            (tmp_path / "nothing").mkdir()
            await mount.load_mount([mount._MountDir(tmp_path / "nothing", PurePosixPath("/e"))], stub)
            assert stub.last_request.files == [] and stub.last_request.object_creation_type == _wire.OBJECT_CREATION_TYPE_EPHEMERAL
            await blob_utils.ClientSessionRegistry.close_session()

    asyncio.run(run())


def test_load_mount_build_validation_and_timeout(backend, monkeypatch, tmp_path):
    async def run():
        async with running_blob_server() as (host, store):
            stub = FakeMountStub(host, store)
            f = tmp_path / "late.py"
            f.write_bytes(b"print('hi')")
            entries = [mount._MountFile(f, PurePosixPath("/root/late.py"))]
            past = time.time() - 3600
            os.utime(f, (past + 1800, past + 1800))  # modified after the build started
            with pytest.raises(ExecutionError, match="modified during build"):
                await mount.load_mount(entries, stub, build_start=past, build_validation="error")
            with pytest.warns(UserWarning, match="modified during build"):
                await mount.load_mount(entries, stub, build_start=past, build_validation="warn")
            await mount.load_mount(entries, stub, build_start=past, build_validation="ignore")
            # a server that never acknowledges the data times out with the reference's exception type
            monkeypatch.setattr(mount, "MOUNT_PUT_FILE_CLIENT_TIMEOUT", 0.05)

            async def never(req):
                await asyncio.sleep(0.01)
                return types.SimpleNamespace(exists=False)

            stub.MountPutFile = never
            with pytest.raises(mount.MountUploadTimeoutError):
                await mount.load_mount(entries, stub)

    asyncio.run(run())


def test_first_occurrence_of_specs_follows_the_set_walk(backend, tmp_path):
    root, files = _make_tree(tmp_path)
    specs = mount.get_file_specs([mount._MountDir(root, PurePosixPath("/m"))])
    first, nd = blob_utils.first_occurrence_of_specs(specs)
    want, want_nd = ref_port.first_occurrence([bytes.fromhex(s.sha256_hex) for s in specs])
    assert first == want and nd == want_nd == len({hashlib.sha256(d).digest() for d in files.values()})
    assert blob_utils.first_occurrence_of_specs([]) == ([], 0)


def test_mount_dir_symlinked_file_keeps_its_name(backend, tmp_path):
    """py/test/mount_test.py `test_mount_directory_with_symlinked_file`: a symlink inside the mounted directory is
    uploaded under the LINK's name with the TARGET's content (local paths are resolved per file, not for the directory)."""
    target_dir = tmp_path / "elsewhere"
    target_dir.mkdir()
    (target_dir / "real.txt").write_bytes(b"real content")
    root = tmp_path / "mounted"
    root.mkdir()
    os.symlink(target_dir / "real.txt", root / "alias.txt")
    sel = mount._select_files([mount._MountDir(root, PurePosixPath("/m"))])
    assert [(p, r.as_posix()) for p, r in sel] == [((target_dir / "real.txt").resolve(), "/m/alias.txt")]
    specs = mount.get_file_specs([mount._MountDir(root, PurePosixPath("/m"))])
    assert [(s.mount_filename, s.sha256_hex) for s in specs] == [("/m/alias.txt", hashlib.sha256(b"real content").hexdigest())]
    # a file that disappears after selection is skipped, not fatal
    ghost = root / "ghost.tmp"
    ghost.write_bytes(b"x")
    entries = [mount._MountDir(root, PurePosixPath("/m"))]
    real_select = mount._select_files

    def select_then_delete(e):
        out = real_select(e)
        ghost.unlink(missing_ok=True)
        return out

    import unittest.mock as um
    with um.patch.object(mount, "_select_files", select_then_delete):
        specs = mount.get_file_specs(entries)
    assert [s.mount_filename for s in specs] == ["/m/alias.txt"]


def _selection_cases(tmp_path):
    from oracle import gen_golden

    gen_golden.build_mount_tree(str(tmp_path))
    ours = {"_MountDir": mount._MountDir, "_MountFile": mount._MountFile}
    return gen_golden, {name: gen_golden.normalise_selection(mount._select_files(entries), str(tmp_path))
                        for name, entries in gen_golden.mount_cases(ours, str(tmp_path)).items()}


def test_mount_selection_matches_reference_golden(tmp_path):
    """_MountFile / _MountDir / _select_files select exactly what the reference's own classes select on the fixture
    tree of oracle/gen_golden.py (tests/golden/mount_select.json was produced by executing py/modal/mount.py:89-196
    unmodified): symlinked files under the link's name, symlinked directories not descended into, dangling links
    listed by the recursive walk but not by the flat one, ignore predicate applied to relative paths, overlaps merged."""
    import json

    golden = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "mount_select.json")))
    _, got = _selection_cases(tmp_path)
    assert got == golden["cases"]
    assert len(golden["cases"]["dir_recursive"]) == 10 and len(golden["cases"]["dir_flat"]) == 4


def test_mount_selection_matches_live_reference(tmp_path):
    """The reference's selection was recorded on this very fixture tree and for every case built here: the tree and
    the case names stored with tests/golden/mount_select.json are the ones oracle/gen_golden.py builds today."""
    import json

    golden = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "mount_select.json")))
    gen_golden, got = _selection_cases(tmp_path)
    assert golden["tree"] == {k: list(v) for k, v in gen_golden.MOUNT_TREE.items()}
    assert got == golden["cases"]
