"""Python face of tools/lz4_tile_model.c, the sequential CPU twin of the GPU block compressor (development / test tool,
not product code).  frame(data) assembles the LZ4 frame the GPU stage must emit byte for byte, frame_linked(data, ...) the
one it emits with SKY_F_LINKED."""
from __future__ import annotations

import ctypes
import subprocess
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
_SO = ROOT / "tools" / "bin" / "liblz4tile.so"
_SRC = ROOT / "tools" / "lz4_tile_model.c"
_lib = None


class Opts(ctypes.Structure):
    _fields_ = [("entries", ctypes.c_int), ("seg_slots", ctypes.c_int), ("max_step_log", ctypes.c_int), ("back_ext", ctypes.c_int),
                ("clip", ctypes.c_int), ("group_lag", ctypes.c_int), ("near_mask", ctypes.c_int)]


class Stats(ctypes.Structure):
    _fields_ = [(n, ctypes.c_uint64) for n in ("probes", "hits", "accepted", "segments")]


def kernel_opts(entries: int = 4096, seg_slots: int = 1024, max_step_log: int = 4) -> Opts:
    """The options the kernel in skyplane_b200/csrc/lz4.cuh implements."""
    return Opts(entries, seg_slots, max_step_log, 1, 1, 1, 0x8C)


def lib():
    global _lib
    if _lib is None:
        _SO.parent.mkdir(exist_ok=True)
        if not _SO.exists() or _SO.stat().st_mtime < _SRC.stat().st_mtime:
            subprocess.check_call(["gcc", "-O2", "-shared", "-fPIC", "-o", str(_SO), str(_SRC)])
        _lib = ctypes.CDLL(str(_SO))
        _lib.tile_compress_block.argtypes = [ctypes.c_char_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.POINTER(Opts)]
        _lib.tile_compress_block.restype = ctypes.c_uint32
        _lib.tile_compress_block_linked.argtypes = [ctypes.c_char_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_char_p,
                                                    ctypes.POINTER(Opts), ctypes.c_int]
        _lib.tile_compress_block_linked.restype = ctypes.c_uint32
    return _lib


def _xxh32_small(b: bytes) -> int:  # XXH32, seed 0, inputs < 16 bytes (the frame descriptor)
    P1, P2, P3, P4, P5, M = 2654435761, 2246822519, 3266489917, 668265263, 374761393, 0xFFFFFFFF
    rotl = lambda x, s: ((x << s) | (x >> (32 - s))) & M  # noqa: E731
    h = (P5 + len(b)) & M
    i = 0
    while i + 4 <= len(b):
        h = (rotl((h + int.from_bytes(b[i:i + 4], "little") * P3) & M, 17) * P4) & M
        i += 4
    while i < len(b):
        h = (rotl((h + b[i] * P5) & M, 11) * P1) & M
        i += 1
    h ^= h >> 15
    h = (h * P2) & M
    h ^= h >> 13
    h = (h * P3) & M
    return h ^ (h >> 16)


def blocks(data: bytes, o: Opts):
    """-> list of (compressed size or 0 when stored raw, block bytes as they appear in the frame)."""
    L = lib()
    buf = ctypes.create_string_buffer(65536 + 4096)
    out = []
    for pos in range(0, len(data), 65536):
        blk = data[pos:pos + 65536]
        c = L.tile_compress_block(blk, len(blk), buf, ctypes.byref(o))
        out.append((c, buf.raw[:c] if c else blk))
    return out


def blocks_linked(data: bytes, o: Opts, W: int, seed_step_log: int):
    """blocks() for a linked frame: block j >= 1 sees the W raw bytes before it as its window."""
    L = lib()
    buf = ctypes.create_string_buffer(65536 + 4096)
    out = []
    for pos in range(0, len(data), 65536):
        blk, win = data[pos:pos + 65536], data[max(0, pos - W):pos]
        c = L.tile_compress_block_linked(win, len(win), blk, len(blk), buf, ctypes.byref(o), seed_step_log)
        out.append((c, buf.raw[:c] if c else blk))
    return out


def _frame(data: bytes, flg: int, blks) -> bytes:
    if not data:
        d = bytes([0x60, 0x40])
        return bytes([0x04, 0x22, 0x4D, 0x18]) + d + bytes([(_xxh32_small(d) >> 8) & 0xFF]) + bytes(4)
    d = bytes([flg, 0x40]) + len(data).to_bytes(8, "little")
    fr = bytearray(bytes([0x04, 0x22, 0x4D, 0x18]) + d + bytes([(_xxh32_small(d) >> 8) & 0xFF]))
    for c, b in blks:
        fr += (c if c else (len(b) | 0x80000000)).to_bytes(4, "little") + b
    return bytes(fr + bytes(4))


def frame(data: bytes, o: Opts | None = None) -> bytes:
    o = o or kernel_opts()
    return _frame(data, 0x68, blocks(data, o))


def frame_linked(data: bytes, o: Opts | None = None, W: int = 4096, seed_step_log: int = 0) -> bytes:
    """The frame SKY_F_LINKED emits: FLG 0x48 (linked blocks, content size) when the chunk has more than one block; a chunk
    of one block gets FLG 0x68 as liblz4 gives it (a single block is independent either way)."""
    o = o or kernel_opts()
    return _frame(data, 0x48 if len(data) > 65536 else 0x68, blocks_linked(data, o, W, seed_step_log))
