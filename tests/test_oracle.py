"""CPU: pins the oracle (oracle/hash_oracle.c + oracle/ref_port.py) against
(1) published known-answer vectors (FIPS 180-4 / NIST CAVS examples, RFC 1321 A.5),
(2) hashlib on seeded inputs, (3) tests/golden/*.json written by the unmodified reference."""
import base64
import hashlib
import io

import numpy as np
import pytest

from modal_client_b200.synth import materialize, synth_bytes
from oracle import c_oracle, ref_port

SHA_KAT = [
    (b"", "e3b0c44298fc1c149afbf4c8996fb92427ae41e4649b934ca495991b7852b855"),
    (b"abc", "ba7816bf8f01cfea414140de5dae2223b00361a396177a9cb410ff61f20015ad"),
    (b"abcdbcdecdefdefgefghfghighijhijkijkljklmklmnlmnomnopnopq",
     "248d6a61d20638b8e5c026930c3e6039a33ce45964ff2167f6ecedd419db06c1"),
    (b"abcdefghbcdefghicdefghijdefghijkefghijklfghijklmghijklmnhijklmnoijklmnopjklmnopqklmnopqrlmnopqrsmnopqrstnopqrstu",
     "cf5b16a778af8380036ce59e7b0492370b249b11e8f07a51afac45037afee9d1"),
    (b"a" * 1_000_000, "cdc76e5c9914fb9281a1c7e284d73e67f1809a48a497200e046d39ccc7112cd0"),
]
MD5_KAT = [  # RFC 1321 appendix A.5
    (b"", "d41d8cd98f00b204e9800998ecf8427e"),
    (b"a", "0cc175b9c0f1b6a831c399e269772661"),
    (b"abc", "900150983cd24fb0d6963f7d28e17f72"),
    (b"message digest", "f96b697d7cb7938d525a2f31aaf161d0"),
    (b"abcdefghijklmnopqrstuvwxyz", "c3fcd3d76192e4007dfb496cca67e13b"),
    (b"ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789", "d174ab98d277d9f5a5611c2c9f419d9f"),
    (b"1234567890" * 8, "57edf4a22be3c955ac49da2e2107b67a"),
]


@pytest.mark.parametrize("msg,hexd", SHA_KAT)
def test_c_oracle_sha256_known_answers(msg, hexd):
    assert c_oracle.sha256(msg).hex() == hexd


@pytest.mark.parametrize("msg,hexd", MD5_KAT)
def test_c_oracle_md5_known_answers(msg, hexd):
    assert c_oracle.md5(msg).hex() == hexd


def test_c_oracle_vs_hashlib_every_length_to_300():
    stream = synth_bytes(1, 300)
    for n in range(301):
        m = stream[:n]
        assert c_oracle.sha256(m) == hashlib.sha256(m).digest(), n
        assert c_oracle.md5(m) == hashlib.md5(m).digest(), n


def test_c_oracle_batch_and_trim_vs_hashlib():
    rng = np.random.default_rng(0)
    lens = rng.integers(0, 5000, size=200)
    offs = np.concatenate([[0], np.cumsum(lens + rng.integers(0, 9, size=200))])[:-1]
    buf = bytearray(synth_bytes(2, int(offs[-1] + lens[-1]) + 16))
    for o, n in zip(offs[::3], lens[::3]):  # plant trailing zero runs
        z = min(int(n), int(rng.integers(0, 200)))
        buf[int(o + n - z) : int(o + n)] = bytes(z)
    buf = bytes(buf)
    s, m, e = c_oracle.hash_batch(buf, offs, lens, trim=True)
    for i, (o, n) in enumerate(zip(offs, lens)):
        msg = buf[int(o) : int(o + n)].rstrip(b"\0")
        assert e[i] == len(msg)
        assert s[i].tobytes() == hashlib.sha256(msg).digest()
        assert m[i].tobytes() == hashlib.md5(msg).digest()


def test_golden_hash_utils(golden):
    doc = golden("hash_utils.json")
    for c in doc["bytes_cases"]:
        data = materialize(c["input"])
        assert c_oracle.sha256(data).hex() == c["sha256_hex"]
        assert c_oracle.md5(data).hex() == c["md5_hex"]
        up = ref_port.upload_hashes(data)
        assert (up.md5_base64, up.sha256_base64) == (c["md5_base64"], c["sha256_base64"])
        assert ref_port.sha256_hex(io.BytesIO(data)) == c["get_sha256_hex"]
        assert ref_port.sha256_base64(data) == c["get_sha256_base64"]
        assert ref_port.md5_base64(io.BytesIO(data)) == c["get_md5_base64"]
    for c in doc["stream_cases"]:
        fp = io.BytesIO(materialize(c["input"]))
        fp.seek(c["pos"])
        up = ref_port.upload_hashes(fp)
        assert fp.tell() == c["pos_after"] == c["pos"]
        assert (up.md5_base64, up.sha256_base64) == (c["md5_base64"], c["sha256_base64"])
    for c in doc["supplied_cases"]:
        up = ref_port.upload_hashes(materialize(c["input"]), **c["kwargs"])
        assert (up.md5_base64, up.sha256_base64) == (c["md5_base64"], c["sha256_base64"])


def test_golden_file_specs(golden, monkeypatch):
    for c in golden("file_specs.json")["cases"]:
        p = c["patch"]
        monkeypatch.setattr(ref_port, "BIG_FILE", p.get("LARGE_FILE_LIMIT", 4 << 20))
        monkeypatch.setattr(ref_port, "NO_MD5_ABOVE", p.get("MULTIPART_UPLOAD_THRESHOLD", 1 << 30))
        f = ref_port.file_spec_fields(io.BytesIO(materialize(c["input"])))
        assert f["use_blob"] == c["use_blob"] and f["size"] == c["size"]
        assert f["sha256_hex"] == c["sha256_hex"] and f["md5_hex"] == c["md5_hex"]
        assert (f["content"] is not None) == c["has_content"]


def test_golden_blocks(golden):
    doc = golden("blocks.json")
    for c in doc["find_end_of_block"]:
        data = materialize(c["input"])
        assert ref_port.block_end(data, c["start"], c["end"]) == c["result"]
        assert c["start"] + c_oracle.trimmed_len(data[c["start"] : c["end"]]) == c["result"]
    for c in doc["spec2"]:
        data = materialize(c["input"])
        bs = c["patch"].get("BLOCK_SIZE", 8 << 20)
        got = ref_port.gather_blocks(data, bs)
        assert [[s, e, d.hex()] for s, e, d in got] == c["blocks"]
        starts = np.arange(0, len(data), bs, dtype=np.uint64)
        lens = np.minimum(bs, len(data) - starts).astype(np.uint64)
        s, _, e = c_oracle.hash_batch(data, starts, lens, md5=False, trim=True)
        assert [[int(a), int(a + b), h.tobytes().hex()] for a, b, h in zip(starts, e, s)] == c["blocks"]


def test_golden_multipart(golden):
    for c in golden("multipart.json")["cases"]:
        data = materialize(c["input"])
        parts, etag = ref_port.multipart_etag(data, c["part_len"])
        assert [p.hex() for p in parts] == c["part_md5_hex"] and etag == c["etag"]
        cparts, cetag = c_oracle.multipart_md5(data, c["part_len"])
        assert [p.tobytes().hex() for p in cparts] == c["part_md5_hex"]
        assert f"{cetag.hex()}-{len(cparts)}" == c["etag"]


def test_live_reference_agrees_with_port(golden):
    """The reference's get_upload_hashes / _find_end_of_block on seeded inputs, as recorded in tests/golden/seam.json."""
    cases = golden("seam.json")["upload_hashes"]
    assert [(c["input"]["seed"], c["input"]["size"]) for c in cases] == [(900, 0), (901, 1), (902, 70001), (903, 300000)]
    for c in cases:
        data = materialize(c["input"])
        assert data == synth_bytes(c["input"]["seed"], c["input"]["size"])
        p = ref_port.upload_hashes(io.BytesIO(data))
        assert (c["md5_base64"], c["sha256_base64"]) == (p.md5_base64, p.sha256_base64)
        assert base64.b64decode(c["sha256_base64"]) == c_oracle.sha256(data)
        n = len(data)
        assert c["end_of_block_with_9_zeros"] == ref_port.block_end(data + bytes(9), 0, n + 9)


def test_first_occurrence_is_the_set_walk_of_the_mount_uploader():
    """oracle.ref_port.first_occurrence restates mount.py:498,518-534: a digest already accounted for is skipped."""
    from oracle import ref_port

    keys = [b"a" * 32, b"b" * 32, b"a" * 32, b"c" * 32, b"b" * 32, b"a" * 32]
    assert ref_port.first_occurrence(keys) == ([0, 1, 0, 3, 1, 0], 3)
    assert ref_port.first_occurrence([]) == ([], 0)
    # against the literal reference behaviour: walk with a set, count what would be sent
    accounted, sent = set(), []
    for i, k in enumerate(keys):
        if k in accounted:
            continue
        accounted.add(k)
        sent.append(i)
    first, nd = ref_port.first_occurrence(keys)
    assert [i for i, f in enumerate(first) if f == i] == sent and nd == len(accounted)
