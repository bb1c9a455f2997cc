"""CPU oracle for the chunk stage -- TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this package.  ``skyplane_b200`` never does.

``oracle.skyoracle.c`` is a plain-C restatement of the reference's per-chunk arithmetic
(``lz4.frame.compress`` at skyplane/gateway/operators/gateway_operator.py:359,
``lz4.frame.decompress`` at skyplane/gateway/operators/gateway_receiver.py:196 and
``hashlib.md5`` at skyplane/obj_store/s3_interface.py:181-192); this module is its ctypes face.
``oracle.reflib`` binds the system ``liblz4.so.1`` -- the library python-lz4 wraps -- and
``hashlib``; it is the reference engine the restatement is pinned against.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from pathlib import Path

_HERE = Path(__file__).resolve().parent
_LIB_PATH = _HERE / "libskyoracle.so"


def build(force: bool = False) -> Path:
    """Compile oracle/skyoracle.c with gcc (a few hundred ms)."""
    src = _HERE / "skyoracle.c"
    if force or not _LIB_PATH.exists() or _LIB_PATH.stat().st_mtime < src.stat().st_mtime:
        subprocess.check_call(["make", "-C", str(_HERE), "-B", "libskyoracle.so"], stdout=subprocess.DEVNULL)
    return _LIB_PATH


_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        build()
        L = ctypes.CDLL(str(_LIB_PATH))
        u8p, u64, u32 = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32
        L.sky_oracle_md5.argtypes = [u8p, u64, u8p]
        L.sky_oracle_md5.restype = None
        L.sky_oracle_xxh32.argtypes = [u8p, u64, u32]
        L.sky_oracle_xxh32.restype = u32
        L.sky_oracle_lz4f_bound.argtypes = [u64]
        L.sky_oracle_lz4f_bound.restype = u64
        L.sky_oracle_lz4f_decode.argtypes = [u8p, u64, u8p, u64, ctypes.POINTER(u64), ctypes.POINTER(u64), ctypes.POINTER(u32 * 4)]
        L.sky_oracle_lz4f_decode.restype = ctypes.c_int
        for name in ("sky_oracle_lz4f_compress", "sky_oracle_lz4f_compress_indep"):
            f = getattr(L, name)
            f.argtypes = [u8p, u64, u8p, u64]
            f.restype = ctypes.c_int64
        L.sky_oracle_chunk_stage.argtypes = [u8p, u64, u8p, u64, u8p]
        L.sky_oracle_chunk_stage.restype = ctypes.c_int64
        L.sky_oracle_secretbox_seal.argtypes = [u8p, u8p, u8p, u64, u8p]
        L.sky_oracle_secretbox_seal.restype = None
        L.sky_oracle_secretbox_open.argtypes = [u8p, u8p, u8p, u64, u8p]
        L.sky_oracle_secretbox_open.restype = ctypes.c_int
        L.sky_oracle_strerror.argtypes = [ctypes.c_int]
        L.sky_oracle_strerror.restype = ctypes.c_char_p
        _lib = L
    return _lib


class OracleError(ValueError):
    def __init__(self, code: int):
        self.code = code
        super().__init__(f"oracle error {code}: {lib().sky_oracle_strerror(code).decode()}")


def _ro(buf):
    """Read-only view -> (address, length, keepalive) without copying."""
    mv = memoryview(buf).cast("B")
    n = mv.nbytes
    if n == 0:
        return None, 0, mv
    if mv.readonly:
        arr = (ctypes.c_char * n).from_buffer_copy(mv) if not isinstance(buf, bytes) else None
        if arr is None:
            return ctypes.cast(ctypes.c_char_p(buf), ctypes.c_void_p), n, buf
        return ctypes.cast(arr, ctypes.c_void_p), n, arr
    arr = (ctypes.c_char * n).from_buffer(mv)
    return ctypes.cast(arr, ctypes.c_void_p), n, arr


def md5(data) -> bytes:
    p, n, _k = _ro(data)
    out = ctypes.create_string_buffer(16)
    lib().sky_oracle_md5(p, n, ctypes.cast(out, ctypes.c_void_p))
    return out.raw


def xxh32(data, seed: int = 0) -> int:
    p, n, _k = _ro(data)
    return lib().sky_oracle_xxh32(p, n, seed)


def lz4f_bound(n: int) -> int:
    return lib().sky_oracle_lz4f_bound(n)


def _compress(fn, data) -> bytes:
    p, n, _k = _ro(data)
    cap = lz4f_bound(n)
    out = ctypes.create_string_buffer(cap)
    r = fn(p, n, ctypes.cast(out, ctypes.c_void_p), cap)
    if r < 0:
        raise OracleError(int(r))
    return out.raw[:r]


def lz4f_compress(data) -> bytes:
    """Byte-for-byte what ``lz4.frame.compress(data)`` (python-lz4 defaults) returns."""
    return _compress(lib().sky_oracle_lz4f_compress, data)


def lz4f_compress_indep(data) -> bytes:
    """Same compressor, every 64 KiB block independent (FLG 0x68) -- the GPU stage's layout."""
    return _compress(lib().sky_oracle_lz4f_compress_indep, data)


def lz4f_decode(frame, max_out: int | None = None, with_info: bool = False):
    """Strict LZ4 frame decoder: rejects what ``lz4.frame.decompress`` rejects, and additionally enforces the block
    format's end-of-block rules (last match >= 12 bytes before the block end, last 5 bytes literals) and offset != 0,
    which liblz4 lets through in a few cases. Raises OracleError."""
    p, n, _k = _ro(frame)
    if max_out is None:
        mv = memoryview(frame).cast("B")
        max_out = int.from_bytes(bytes(mv[6:14]), "little") if n >= 14 and (mv[4] & 0x08) else max(64, n * 255)
    out = ctypes.create_string_buffer(max(1, max_out))
    olen, used = ctypes.c_uint64(0), ctypes.c_uint64(0)
    info = (ctypes.c_uint32 * 4)()
    rc = lib().sky_oracle_lz4f_decode(p, n, ctypes.cast(out, ctypes.c_void_p), max_out, ctypes.byref(olen), ctypes.byref(used), ctypes.byref(info))
    if rc != 0:
        raise OracleError(rc)
    data = out.raw[: olen.value]
    if with_info:
        return data, {"flg": info[0], "bd": info[1], "blocks": info[2], "raw_blocks": info[3], "consumed": used.value}
    return data


def chunk_stage(data):
    """The reference's serial pair for one chunk: (lz4 frame, md5 digest)."""
    p, n, _k = _ro(data)
    cap = lz4f_bound(n)
    out = ctypes.create_string_buffer(cap)
    dig = ctypes.create_string_buffer(16)
    r = lib().sky_oracle_chunk_stage(p, n, ctypes.cast(out, ctypes.c_void_p), cap, ctypes.cast(dig, ctypes.c_void_p))
    if r < 0:
        raise OracleError(int(r))
    return out.raw[:r], dig.raw


def secretbox_seal(key: bytes, nonce: bytes, msg) -> bytes:
    """tag(16) || ciphertext, i.e. nacl.bindings.crypto_secretbox(msg, nonce, key) (SecretBox.encrypt minus the nonce prefix)."""
    assert len(key) == 32 and len(nonce) == 24
    p, n, _k = _ro(msg)
    out = ctypes.create_string_buffer(16 + n)
    lib().sky_oracle_secretbox_seal(ctypes.cast(ctypes.c_char_p(key), ctypes.c_void_p), ctypes.cast(ctypes.c_char_p(nonce), ctypes.c_void_p),
                                    p, n, ctypes.cast(out, ctypes.c_void_p))
    return out.raw


def secretbox_open(key: bytes, nonce: bytes, boxed) -> bytes:
    assert len(key) == 32 and len(nonce) == 24
    p, n, _k = _ro(boxed)
    out = ctypes.create_string_buffer(max(1, n))
    rc = lib().sky_oracle_secretbox_open(ctypes.cast(ctypes.c_char_p(key), ctypes.c_void_p), ctypes.cast(ctypes.c_char_p(nonce), ctypes.c_void_p),
                                         p, n, ctypes.cast(out, ctypes.c_void_p))
    if rc != 0:
        raise ValueError("secretbox: authentication failed")
    return out.raw[: n - 16]
