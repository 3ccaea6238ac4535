"""oracle/gen_safetensors_golden.py -- regenerates tests/golden/safetensors.json from the installed safetensors package.

``python -m oracle.gen_safetensors_golden``.  Every case is a small recipe -- tensor names, dtypes, shapes and a seed
per tensor (``state_dict_from_recipe``) -- plus what ``safetensors.torch.save`` returned for it: the header bytes and
the SHA-256 of the whole file.  Metadata has at most one key: safetensors writes a metadata map of several keys in
an order that changes from process to process (a Rust HashMap), so only a single key has one right answer.  The
tests rebuild the dicts from the recipes and compare
``blob_utils.safetensors_layout`` with the stored answers, so they need no safetensors package.
"""
from __future__ import annotations

import hashlib
import json
import os

import torch

from modal_client_b200.synth import synth_bytes

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "safetensors.json")

DTYPES = {"F64": "float64", "F32": "float32", "F16": "float16", "BF16": "bfloat16", "I64": "int64", "I32": "int32",
          "I16": "int16", "I8": "int8", "U8": "uint8", "BOOL": "bool", "F8_E4M3": "float8_e4m3fn",
          "F8_E5M2": "float8_e5m2", "C64": "complex64", "U64": "uint64", "U32": "uint32", "U16": "uint16"}


def state_dict_from_recipe(tensors: list[dict]) -> dict[str, torch.Tensor]:
    """{name: tensor} with bytes = synth_bytes(seed, nbytes) (BOOL: the low bit of each byte)."""
    out = {}
    for t in tensors:
        dtype = getattr(torch, DTYPES[t["dtype"]])
        n = 1
        for d in t["shape"]:
            n *= d
        raw = bytearray(synth_bytes(t["seed"], n * torch.empty(0, dtype=dtype).element_size()))
        if dtype == torch.bool:
            raw = bytearray(b & 1 for b in raw)
        flat = torch.frombuffer(raw, dtype=torch.uint8).view(dtype) if raw else torch.empty(0, dtype=dtype)
        out[t["name"]] = flat.reshape(t["shape"])
    return out


def _t(name, dtype, shape, seed):
    return {"name": name, "dtype": dtype, "shape": list(shape), "seed": seed}


def cases() -> list[dict]:
    every = [_t(f"t_{k.lower()}", k, (3, 5), 100 + i) for i, k in enumerate(DTYPES)]
    return [
        {"name": "empty", "metadata": None, "tensors": []},
        {"name": "empty_with_metadata", "metadata": {"format": "pt"}, "tensors": []},
        {"name": "every_dtype", "metadata": None, "tensors": every},
        {"name": "every_dtype_reversed_names", "metadata": {"z": "2"},
         "tensors": [dict(t, name=f"{99 - i:02d}_{t['name']}") for i, t in enumerate(every)]},
        {"name": "scalars_and_zero_size", "metadata": None,
         "tensors": [_t("s", "F32", (), 1), _t("z0", "F16", (0,), 2), _t("z1", "I64", (4, 0, 2), 3),
                     _t("b", "BOOL", (), 4), _t("x", "U8", (7,), 5)]},
        {"name": "names_sort_by_dtype_first", "metadata": None,
         "tensors": [_t("a", "U8", (5,), 6), _t("b", "F64", (2,), 7), _t("c", "BF16", (3,), 8), _t("d", "I64", (1,), 9),
                     _t("A", "U8", (2,), 10), _t("B", "F32", (1, 1), 11)]},
        {"name": "unusual_names", "metadata": {"note ü☃": "café \"quoted\" \\ back\u0001slash\n"},
         "tensors": [_t("café.weight", "F32", (2, 2), 12), _t("☃", "F32", (1,), 13),
                     _t("q\"uote", "F32", (1,), 14), _t("ctl\u0001\u001f\t\n", "F32", (1,), 15),
                     _t("back\\slash/", "F32", (1,), 16), _t("\U0001f600", "F32", (1,), 17), _t("Z", "F32", (1,), 18)]},
        {"name": "layer_stack", "metadata": {"format": "pt"},
         "tensors": [_t(f"model.layers.{i}.{p}", dt, shp, 200 + 10 * i + j) for i in range(3)
                     for j, (p, dt, shp) in enumerate([("mlp.weight", "BF16", (64, 96)), ("norm.weight", "F32", (64,)),
                                                       ("attn.scale", "F32", ()), ("mask", "BOOL", (9,)),
                                                       ("q.weight", "F8_E4M3", (33, 7))])]},
    ]


def main() -> None:
    import safetensors
    import safetensors.torch as st

    out = {"safetensors_version": safetensors.__version__, "cases": []}
    for case in cases():
        data = st.save(state_dict_from_recipe(case["tensors"]), case["metadata"])
        hlen = 8 + int.from_bytes(data[:8], "little")
        out["cases"].append(dict(case, header_hex=data[:hlen].hex(), size=len(data),
                                 sha256=hashlib.sha256(data).hexdigest()))
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1, ensure_ascii=True)
        f.write("\n")


if __name__ == "__main__":
    main()
