#!/usr/bin/env python
"""Compression ratio of the kernel's parse (its sequential CPU twin, tools/lz4_tile_model.c) on data kinds beyond the bench's
Silesia-like set, next to liblz4's: linked blocks (what the reference emits) and independent blocks (what any block-parallel
compressor is limited to).  Development tool: CPU only, reads files that happen to be installed in the build container.

--linked adds the linked-block twin (tile_model.frame_linked: block j sees the W raw bytes before it, the table seeded
with every (1 << s)-th window position) for W in LINKED_WINDOWS and s in LINKED_SEED_LOGS; its output is
profiles/linked_ratio_cpu_twin.jsonl."""
import glob
import json
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import oracle  # noqa: E402
import oracle.reflib as ref  # noqa: E402
from skyplane_b200 import synth  # noqa: E402
from tools import tile_model as tm  # noqa: E402


def cat(pattern, limit):
    out = bytearray()
    for f in sorted(glob.glob(pattern, recursive=True)):
        if os.path.isfile(f) and not os.path.islink(f):
            try:
                out += open(f, "rb").read()
            except OSError:
                pass
        if len(out) >= limit:
            break
    return bytes(out[:limit])


def kinds():
    r = np.random.default_rng(1)
    walk = np.cumsum(r.integers(-3, 4, size=1 << 19))
    py = cat("/usr/lib/python3*/**/*.py", 8 << 20)
    return {
        "silesia-like 4 x 4 MiB (bench set)": b"".join(synth.silesia_like_chunk(i, 4 << 20) for i in range(4)),
        "shared objects 8 MiB": cat("/usr/lib/x86_64-linux-gnu/*.so*", 8 << 20),
        "python sources 8 MiB": py,
        "c headers 8 MiB": cat("/usr/local/cuda/include/**/*.h", 8 << 20),
        "utf-16 text 4 MiB": py[: 2 << 20].decode("latin1").encode("utf-16-le"),
        "float64 walk 4 MiB": (walk * 0.25).astype("<f8").tobytes(),
        "int64 ids 4 MiB": (np.arange(1 << 19, dtype="<i8") * 7 + 1000).tobytes(),
        "int32 walk 4 MiB": synth._numeric(np.random.default_rng(7), 4 << 20),
        "rgb runs 3 MiB": np.repeat(r.integers(0, 255, size=(1 << 12, 3), dtype=np.uint8), 256, axis=0).tobytes(),
        "int16 audio-like 4 MiB": (np.sin(np.arange(1 << 21) / 50) * 3000 + r.integers(-2, 3, size=1 << 21)).astype("<i2").tobytes(),
    }


LINKED_WINDOWS = (4096, 8192, 16384, 32768, 65536)  # 4 KiB: what fits the kernel's shared memory next to a 4096-entry table
LINKED_SEED_LOGS = (0, 1, 2)


if __name__ == "__main__":
    linked = "--linked" in sys.argv
    for name, d in kinds().items():
        if not d:
            continue
        raw = len(d)
        ours = len(tm.frame(d))
        linked = len(ref.lz4f_compress(d))
        indep = len(oracle.lz4f_compress_indep(d)) if hasattr(oracle, "lz4f_compress_indep") else None
        row = {"data": name, "bytes": raw, "kernel_parse_ratio": round(raw / ours, 4), "liblz4_linked_ratio": round(raw / linked, 4),
               "vs_reference": round(linked / ours, 4)}
        if indep:
            row["liblz4_independent_blocks_ratio"] = round(raw / indep, 4)
            row["vs_liblz4_independent"] = round(indep / ours, 4)
        if linked:
            for w in LINKED_WINDOWS:
                for sl in LINKED_SEED_LOGS:
                    fr = tm.frame_linked(d, tm.kernel_opts(), w, sl)
                    assert ref.lz4f_decompress(fr, raw) == d
                    row[f"linked_w{w >> 10}k_seed{1 << sl}_ratio"] = round(raw / len(fr), 4)
        print(json.dumps(row), flush=True)
