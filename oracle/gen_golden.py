"""oracle/gen_golden.py -- regenerates tests/golden/*.json from the UNMODIFIED reference.

Needs a source checkout of the original modal client:  ``B200H_REFERENCE_ROOT=<checkout> python -m oracle.gen_golden``
Inputs are stored as small recipes (modal_client_b200.synth.materialize), outputs are whatever the
reference's own functions returned.  The tests only read the JSON, so they need no copy of the reference.
"""
from __future__ import annotations

import asyncio
import io
import json
import os
from pathlib import PurePosixPath

from modal_client_b200.synth import materialize
from oracle import ref_shim

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
MiB = 1 << 20


def synth(seed, size):
    return {"kind": "synth", "seed": seed, "size": size}


def rep(unit: bytes, count: int):
    return {"kind": "repeat", "unit": unit.hex(), "count": count}


def cat(*parts):
    return {"kind": "concat", "parts": list(parts)}


def lit(b: bytes):
    return {"kind": "literal", "hex": b.hex()}


def gen_hash_utils(h):
    cases = []
    sizes = [0, 1, 3, 55, 56, 57, 63, 64, 65, 119, 120, 121, 127, 128, 129, 1000, 4095, 4096, 65535, 65536,
             65537, 131072 + 5, 262144, MiB + 3]
    recipes = [synth(100 + i, n) for i, n in enumerate(sizes)]
    recipes += [
        lit(b"abc"),
        lit(b"hello world"),
        lit(b"this is a test"[:15]),
        rep(b"a", 4 * MiB + 1),  # py/test/mount_test.py:45
        rep(b"A", 1),  # py/test/mount_test.py:172
        rep(b"*", 10_000_000),  # py/test/blob_test.py:50
        rep(b"\0", 70000),
        cat(synth(7, 1000), {"kind": "zeros", "size": 5000}),
    ]
    for r in recipes:
        data = materialize(r)
        up = h.get_upload_hashes(data)
        up_stream = h.get_upload_hashes(io.BytesIO(data))
        assert up == up_stream
        cases.append(
            {
                "input": r,
                "md5_base64": up.md5_base64,
                "sha256_base64": up.sha256_base64,
                "md5_hex": up.md5_hex(),
                "sha256_hex": up.sha256_hex(),
                "get_sha256_hex": h.get_sha256_hex(data),
                "get_sha256_base64": h.get_sha256_base64(io.BytesIO(data)),
                "get_md5_base64": h.get_md5_base64(data),
            }
        )
    # stream semantics: hash from the current position, position restored (hash_utils.py:20,29)
    stream_cases = []
    for seed, size, pos in [(300, 200000, 0), (301, 200000, 77), (302, 65536 * 3, 65536), (303, 10, 10)]:
        r = synth(seed, size)
        fp = io.BytesIO(materialize(r))
        fp.seek(pos)
        up = h.get_upload_hashes(fp)
        stream_cases.append({"input": r, "pos": pos, "pos_after": fp.tell(), "md5_base64": up.md5_base64,
                             "sha256_base64": up.sha256_base64})
    # supplied digests are passed through and not recomputed (hash_utils.py:74-93)
    supplied = []
    r = synth(310, 5000)
    data = materialize(r)
    for kw in ({"sha256_hex": "11" * 32}, {"md5_hex": "22" * 16}, {"sha256_hex": "ab" * 32, "md5_hex": "cd" * 16}):
        up = h.get_upload_hashes(data, **kw)
        supplied.append({"input": r, "kwargs": kw, "md5_base64": up.md5_base64, "sha256_base64": up.sha256_base64})
    return {"source": "py/modal/_utils/hash_utils.py (unmodified, via oracle/ref_shim.py)", "bytes_cases": cases,
            "stream_cases": stream_cases, "supplied_cases": supplied}


def gen_file_specs(b):
    out = []
    sizes = [0, 11, 256 * 1024 - 1, 256 * 1024, 256 * 1024 + 1, 4 * MiB - 1, 4 * MiB, 4 * MiB + 1]
    for i, n in enumerate(sizes):
        r = synth(400 + i, n)
        spec = b.get_file_upload_spec_from_fileobj(io.BytesIO(materialize(r)), PurePosixPath("/d/f.bin"), 0o100644)
        out.append({"input": r, "patch": {}, "use_blob": spec.use_blob, "sha256_hex": spec.sha256_hex,
                    "md5_hex": spec.md5_hex, "mode": spec.mode, "size": spec.size,
                    "mount_filename": spec.mount_filename, "has_content": spec.content is not None})
    # "> 1 GiB" class (placeholder MD5, no MD5 computed) with the thresholds patched down, as the
    # reference's tests patch module globals (py/test/blob_test.py:57)
    patch = {"LARGE_FILE_LIMIT": 4096, "MULTIPART_UPLOAD_THRESHOLD": 10000}
    saved = {k: getattr(b, k) for k in patch}
    try:
        for k, v in patch.items():
            setattr(b, k, v)
        for i, n in enumerate([4095, 4096, 10000, 10001, 50000]):
            r = synth(420 + i, n)
            spec = b.get_file_upload_spec_from_fileobj(io.BytesIO(materialize(r)), PurePosixPath("x"), 0o755)
            out.append({"input": r, "patch": patch, "use_blob": spec.use_blob, "sha256_hex": spec.sha256_hex,
                        "md5_hex": spec.md5_hex, "mode": spec.mode, "size": spec.size,
                        "mount_filename": spec.mount_filename, "has_content": spec.content is not None})
    finally:
        for k, v in saved.items():
            setattr(b, k, v)
    return {"source": "py/modal/_utils/blob_utils.py:446-516 (unmodified)", "cases": out}


def gen_blocks(b):
    eob = []
    for data, start, end in [(b"abc123\0\0\0", 0, 1024), (b"abc123\0\0\0", 3, 1024), (b"abc123\0\0\0", 0, 3),
                             (b"abc123\0\0\0a", 0, 9), (b"\0\0\0", 0, 3), (b"\0\0\0\0\0\0", 3, 6), (b"", 0, 1024),
                             (b"\0\0x\0", 1, 4), (b"x", 0, 1)]:
        eob.append({"input": lit(data), "start": start, "end": end,
                    "result": b._find_end_of_block(lambda d=data: io.BytesIO(d), start, end)})

    async def spec2(data):
        sem = asyncio.Semaphore(4)
        return await b.FileUploadSpec2.from_fileobj(io.BytesIO(data), PurePosixPath("/v/file"), sem, 0o644)

    B = 8 * MiB
    recipes = [
        (cat(rep(b"a", 1), {"kind": "zeros", "size": B - 1}, rep(b"a", 1), {"kind": "zeros", "size": B - 1},
             lit(b"cdef")), {}),  # py/test/volume_test.py:537 blank-block file
        (cat(rep(b"A", 2 * B - 2), lit(b"B\0")), {}),  # py/test/volume_test.py:325-326 trailing zero regression
        (synth(500, 100), {}),
        (synth(501, B), {}),
        (synth(502, 2 * B), {}),
        (synth(503, 4 * B + 4711), {}),
        ({"kind": "zeros", "size": B + 17}, {}),
        (synth(504, 0), {}),
        (rep(b"hello world, this is a lot of text", 250_000), {}),  # py/test/volume_test.py:509
        # small block size (module global patched, read at call time: blob_utils.py:630,641)
        (cat(synth(510, 700), {"kind": "zeros", "size": 900}, synth(511, 300), {"kind": "zeros", "size": 2100},
             synth(512, 1)), {"BLOCK_SIZE": 1000}),
        (synth(513, 64 * 1000), {"BLOCK_SIZE": 1000}),
        (cat({"kind": "zeros", "size": 63}, lit(b"\x01"), {"kind": "zeros", "size": 64}), {"BLOCK_SIZE": 64}),
    ]
    specs = []
    for r, patch in recipes:
        saved = {k: getattr(b, k) for k in patch}
        try:
            for k, v in patch.items():
                setattr(b, k, v)
            s = asyncio.run(spec2(materialize(r)))
        finally:
            for k, v in saved.items():
                setattr(b, k, v)
        specs.append({"input": r, "patch": patch, "size": s.size, "mode": s.mode, "path": s.path,
                      "blocks": [[blk.start, blk.end, blk.contents_sha256.hex()] for blk in s.blocks]})
    return {"source": "py/modal/_utils/blob_utils.py:522-705 (unmodified)", "find_end_of_block": eob, "spec2": specs}


class _Sink:
    """Stand-in for aiohttp's stream writer: collects what the payload writes."""

    def __init__(self):
        self.chunks = []

    async def write(self, chunk):
        self.chunks.append(bytes(chunk))


def gen_multipart(b, seg):
    """Drives the reference's perform_multipart_upload / BytesIOSegmentPayload with a fake S3 that
    behaves like the reference's own test server (py/test/conftest.py:3364-3391): part ETag = md5 of
    the received body; completion body carries md5(concat(md5(part)))-N.  The reference *verifies*
    both (blob_utils.py:143-154,231-234); a recorded value is one the reference accepted."""
    import hashlib

    out = []

    async def run(data: bytes, part_len: int, chunk: int):
        received = {}

        async def fake_put(upload_url, payload, content_md5_b64=None, content_type=None):
            sink = _Sink()
            with payload.reset_on_error():
                await payload.write_with_length(sink, None)
                body = b"".join(sink.chunks)
                received[upload_url] = body
                etag = hashlib.md5(body).hexdigest()
                assert payload.md5_checksum().hexdigest() == etag  # the check at blob_utils.py:150-152
                return etag

        class Resp:
            status = 200

            def __init__(self, text):
                self._t = text

            async def text(self):
                return self._t

        class Session:
            async def post(self, url, data=None, skip_auto_headers=None):
                parts = [received[u] for u in urls]
                cat_md5 = hashlib.md5(b"".join(hashlib.md5(p).digest() for p in parts)).hexdigest()
                self.etag = f"{cat_md5}-{len(parts)}"
                return Resp(f'<etag>"{self.etag}"</etag>')

        nparts = -(-len(data) // part_len)
        urls = [f"part-{i}" for i in range(nparts)]
        session = Session()
        saved_put, saved_reg = b._upload_to_s3_url, b.ClientSessionRegistry

        class Reg:
            @staticmethod
            def get_session():
                return session

        b._upload_to_s3_url, b.ClientSessionRegistry = fake_put, Reg
        try:
            await b.perform_multipart_upload(io.BytesIO(data), content_length=len(data), max_part_size=part_len,
                                             part_urls=urls, completion_url="done", upload_chunk_size=chunk)
        finally:
            b._upload_to_s3_url, b.ClientSessionRegistry = saved_put, saved_reg
        assert b"".join(received[u] for u in urls) == data
        return [hashlib.md5(received[u]).hexdigest() for u in urls], session.etag

    for r, part_len, chunk in [
        (synth(600, 256 * 1024 + 512), 1024, 128),  # py/test/blob_test.py:56-66: 256 parts + a half part
        (synth(601, 5 * MiB + 123), MiB, 1 << 16),
        (synth(602, 3 * 4096), 4096, 4096),
        (synth(603, 100), 4096, 4096),
        (rep(b"\0", 300000), 65536, 1 << 16),
    ]:
        part_md5, etag = asyncio.run(run(materialize(r), part_len, chunk))
        out.append({"input": r, "part_len": part_len, "part_md5_hex": part_md5, "etag": etag})
    return {"source": "py/modal/_utils/blob_utils.py:159-234 + bytes_io_segment_payload.py (unmodified)", "cases": out}


# ---------------------------------------------------------------------------------- mount file selection

MOUNT_TREE = {  # relative path -> ("file", seed, size) | ("link", target relative to the tmp dir) ; dirs are implied
    "pkg/a.py": ("file", 1, 15),
    "pkg/sub/b.py": ("file", 2, 400),
    "pkg/sub/c.bin": ("file", 3, 70_000),
    "pkg/sub/__pycache__/b.pyc": ("file", 4, 30),
    "pkg/.git/config": ("file", 5, 20),
    "pkg/.hidden": ("file", 6, 5),
    "pkg/empty": ("file", 7, 0),
    "pkg/sp ace/x y.txt": ("file", 8, 9),
    "pkg/alias.txt": ("link", "outside/real.txt"),
    "pkg/linked_dir": ("link", "outside"),
    "pkg/dangling": ("link", "outside/nope"),
    "outside/real.txt": ("file", 9, 12),
}


def build_mount_tree(root):
    """Materialise MOUNT_TREE below ``root`` (used by this generator and by tests/test_mount_upload.py)."""
    from modal_client_b200.synth import synth_bytes

    for rel, spec in MOUNT_TREE.items():
        p = os.path.join(root, rel)
        os.makedirs(os.path.dirname(p), exist_ok=True)
        if spec[0] == "file":
            with open(p, "wb") as f:
                f.write(synth_bytes(spec[1], spec[2]))
    for rel, spec in MOUNT_TREE.items():
        if spec[0] == "link":
            os.symlink(os.path.join(root, spec[1]), os.path.join(root, rel))


def mount_ignore(rel) -> bool:
    """The ignore predicate of the golden cases (plain callable: no directory pruning in the reference)."""
    return rel.suffix == ".pyc" or any(part.startswith(".") for part in rel.parts)


def reference_mount_entries():
    """The reference's OWN ``_MountEntry`` / ``_MountFile`` / ``_MountDir`` / ``_select_files`` (py/modal/mount.py:89-196),
    compiled from the unmodified source file: only these four definitions are executed, in a namespace holding the
    standard-library names they use and a stand-in for ``modal.file_pattern_matcher._AbstractPatternMatcher``."""
    import abc
    import ast
    import dataclasses
    import types
    import typing
    from collections.abc import Callable, Generator
    from pathlib import Path

    path = os.path.join(os.path.dirname(ref_shim.package_dir()), "modal", "mount.py")
    tree = ast.parse(open(path).read())
    wanted = {"_MountEntry", "_select_files", "_MountFile", "_MountDir"}
    body = [n for n in tree.body if getattr(n, "name", None) in wanted]
    assert {n.name for n in body} == wanted

    class _AbstractPatternMatcher:  # nothing in the golden cases is one
        pass

    fake_modal = types.SimpleNamespace(file_pattern_matcher=types.SimpleNamespace(_AbstractPatternMatcher=_AbstractPatternMatcher))
    ns = {"abc": abc, "dataclasses": dataclasses, "os": os, "typing": typing, "Path": Path, "PurePosixPath": PurePosixPath,
          "Callable": Callable, "Generator": Generator, "modal": fake_modal}
    exec(compile(ast.Module(body=body, type_ignores=[]), path, "exec"), ns)
    return ns


def mount_cases(entries_ns, root):
    """name -> list of entries, built from the classes in ``entries_ns`` (the reference's or ours)."""
    from pathlib import Path

    D, F = entries_ns["_MountDir"], entries_ns["_MountFile"]
    pkg = Path(root) / "pkg"
    nothing = lambda _p: False  # noqa: E731
    return {
        "dir_recursive": [D(pkg, PurePosixPath("/root/pkg"), nothing, True)],
        "dir_recursive_ignore": [D(pkg, PurePosixPath("/root/pkg"), mount_ignore, True)],
        "dir_flat": [D(pkg, PurePosixPath("/x"), nothing, False)],
        "file_and_overlap": [F(pkg / "a.py", PurePosixPath("/root/a.py")), D(pkg / "sub", PurePosixPath("/s"), nothing, True),
                             D(pkg / "sub", PurePosixPath("/s"), nothing, True)],
        "file_via_symlink": [F(pkg / "alias.txt", PurePosixPath("/root/alias.txt"))],
    }


def normalise_selection(pairs, root):
    """[(local Path, remote PurePosixPath)] -> sorted [[local relative to the resolved root, remote posix]]."""
    from pathlib import Path

    base = Path(root).resolve()
    return sorted([os.path.relpath(str(p), str(base)), r.as_posix()] for p, r in pairs)


def gen_mount_select():
    import tempfile

    ns = reference_mount_entries()
    with tempfile.TemporaryDirectory() as tmp:
        build_mount_tree(tmp)
        cases = {name: normalise_selection(ns["_select_files"](entries), tmp) for name, entries in mount_cases(ns, tmp).items()}
    return {"source": "py/modal/mount.py:89-196 (_MountFile, _MountDir, _select_files; unmodified source, executed)",
            "tree": {k: list(v) for k, v in MOUNT_TREE.items()}, "cases": cases}


# ------------------------------------------------------------------ what the reference's callers see of the seam


def _reference_constant(rel, name):
    """A module constant of the reference read from its source text (modules that need the control plane to import)."""
    import re

    text = open(os.path.join(os.path.dirname(ref_shim.package_dir()), "modal", rel)).read()
    m = re.search(rf"^{name}\s*(?::[^=]+)?=\s*\(?\s*([^#\n]+)", text, flags=re.M)
    return eval(m.group(1).strip().rstrip(")"))  # noqa: S307 - arithmetic literals of the reference


def gen_seam(h, b, seg):
    """What crosses the drop-in seam when the reference's own callers run: the patchable module constants, the
    get_upload_hashes calls of its spec builder (argument kind, stream position, supplied digests, what came back),
    the BytesIOSegmentPayload objects its multipart upload builds (segment, chunk size, bytes sent, MD5 checked
    against the ETag), and its get_upload_hashes / _find_end_of_block on a few more inputs."""
    import hashlib

    constants = {"hash_utils": {"HASH_CHUNK_SIZE": h.HASH_CHUNK_SIZE},
                 "blob_utils": {k: getattr(b, k) for k in ["MAX_OBJECT_SIZE_BYTES", "MAX_ASYNC_OBJECT_SIZE_BYTES",
                                                           "LARGE_FILE_LIMIT", "BLOB_MAX_PARALLELISM",
                                                           "DEFAULT_SEGMENT_CHUNK_SIZE", "MULTIPART_UPLOAD_THRESHOLD",
                                                           "BLOCK_SIZE"]}}
    for rel, name in [("mount.py", "MOUNT_PUT_FILE_CLIENT_TIMEOUT"), ("volume.py", "VOLUME_PUT_FILE_CLIENT_TIMEOUT"),
                      ("network_file_system.py", "NETWORK_FILE_SYSTEM_PUT_FILE_CLIENT_TIMEOUT"),
                      ("parallel_map.py", "MAP_INVOCATION_CHUNK_SIZE"),
                      ("parallel_map.py", "SPAWN_MAP_INVOCATION_CHUNK_SIZE")]:
        constants.setdefault(rel[:-3], {})[name] = _reference_constant(rel, name)

    # the spec builder's calls into hash_utils, one list per tests/golden/file_specs.json case
    spec_calls = []
    real = b.get_upload_hashes

    def recording(data, **kw):
        is_stream = not isinstance(data, (bytes, bytearray, memoryview))
        call = {"stream": is_stream, "pos": data.tell() if is_stream else None, "kwargs": kw}
        up = real(data, **kw)
        call.update(pos_after=data.tell() if is_stream else None, sha256_hex=up.sha256_hex(), md5_hex=up.md5_hex())
        spec_calls[-1].append(call)
        return up

    b.get_upload_hashes = recording
    try:
        for c in json.load(open(os.path.join(OUT, "file_specs.json")))["cases"]:
            saved = {k: getattr(b, k) for k in c["patch"]}
            spec_calls.append([])
            try:
                for k, v in c["patch"].items():
                    setattr(b, k, v)
                b.get_file_upload_spec_from_fileobj(io.BytesIO(materialize(c["input"])), PurePosixPath(c["mount_filename"]),
                                                    0o100644 if not c["patch"] else 0o755)
            finally:
                for k, v in saved.items():
                    setattr(b, k, v)
    finally:
        b.get_upload_hashes = real

    # the multipart upload's segment payloads (the reference checks each one's MD5 against the part's ETag)
    payloads = []

    class RecordingPayload(seg.BytesIOSegmentPayload):
        def __init__(self, bytes_io, segment_start, segment_length, chunk_size, progress_report_cb=None):
            super().__init__(bytes_io, segment_start, segment_length, chunk_size, progress_report_cb)
            payloads.append({"initial_pos": self.initial_seek_pos, "segment_start": segment_start,
                             "segment_length": segment_length, "chunk_size": chunk_size})

    part_etags = {}

    async def put(upload_url, payload, content_md5_b64=None, content_type=None):
        sink = _Sink()
        with payload.reset_on_error():  # which resets the payload on the way out, as in blob_utils.py:118
            await payload.write(sink)
            body = b"".join(sink.chunks)
            part_etags[int(upload_url)] = hashlib.md5(body).digest()  # what S3 answers: the MD5 of the body it got
            local = payload.md5_checksum().hexdigest()
            assert local == part_etags[int(upload_url)].hex()  # the check at blob_utils.py:150-152
        payloads[int(upload_url)].update(sent_sha256=hashlib.sha256(body).hexdigest(), md5_hex=local)
        return local

    class Session:
        async def post(self, url, data=None, skip_auto_headers=None):
            joined = b"".join(part_etags[i] for i in sorted(part_etags))
            etag = f"{hashlib.md5(joined).hexdigest()}-{len(part_etags)}"

            class Resp:
                status = 200

                async def text(self):
                    return f'<ETag>"{etag}"</ETag>'
            return Resp()

    class Reg:
        get_session = staticmethod(Session)

    mp_input, part_len, chunk = synth(77, 10 * 1000 + 123), 1000, 256
    data = materialize(mp_input)
    saved = b._upload_to_s3_url, b.ClientSessionRegistry, seg.BytesIOSegmentPayload
    b._upload_to_s3_url, b.ClientSessionRegistry, seg.BytesIOSegmentPayload = put, Reg, RecordingPayload
    try:
        asyncio.run(b.perform_multipart_upload(io.BytesIO(data), content_length=len(data), max_part_size=part_len,
                                               part_urls=[str(i) for i in range(11)], completion_url="done",
                                               upload_chunk_size=chunk))
    finally:
        b._upload_to_s3_url, b.ClientSessionRegistry, seg.BytesIOSegmentPayload = saved

    upload_hashes = []
    for seed, n in [(900, 0), (901, 1), (902, 70001), (903, 300000)]:
        r = synth(seed, n)
        d = materialize(r)
        up = h.get_upload_hashes(io.BytesIO(d))
        upload_hashes.append({"input": r, "md5_base64": up.md5_base64, "sha256_base64": up.sha256_base64,
                              "end_of_block_with_9_zeros": b._find_end_of_block(lambda: io.BytesIO(d + bytes(9)), 0, n + 9)})
    return {"source": "py/modal/_utils/{hash_utils,blob_utils,bytes_io_segment_payload}.py and the constants of "
                      "mount.py / volume.py / network_file_system.py / parallel_map.py (unmodified, executed or read)",
            "constants": constants, "spec_builder_calls": spec_calls,
            "multipart": {"input": mp_input, "part_len": part_len, "chunk": chunk, "payloads": payloads},
            "upload_hashes": upload_hashes}


def main():
    h, b, seg = ref_shim.load()
    os.makedirs(OUT, exist_ok=True)
    for name, doc in [("hash_utils.json", gen_hash_utils(h)), ("file_specs.json", gen_file_specs(b)),
                      ("blocks.json", gen_blocks(b)), ("multipart.json", gen_multipart(b, seg)),
                      ("mount_select.json", gen_mount_select()), ("seam.json", gen_seam(h, b, seg))]:
        with open(os.path.join(OUT, name), "w") as f:
            json.dump(doc, f, indent=1, sort_keys=True)
            f.write("\n")
        print("wrote", name)


if __name__ == "__main__":
    main()
