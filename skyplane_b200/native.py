"""ctypes face of libskychunk.so (include/skychunk.h).  No torch, no numpy required.

The library is CUDA-only: if it is missing it is built with nvcc; if nvcc or a GPU is missing the
calls raise ``SkyChunkError`` -- there is deliberately no CPU fallback on the product path.
"""
from __future__ import annotations

import ctypes
from pathlib import Path
from typing import Optional, Sequence

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libskychunk.so"

SKY_OK = 0
SKY_E_INVALID, SKY_E_NOGPU, SKY_E_CUDA, SKY_E_CAPACITY, SKY_E_BUSY, SKY_E_TICKET, SKY_E_NOMEM, SKY_E_NOKEY = -1, -2, -3, -4, -5, -6, -7, -8
F_LZ4, F_MD5, F_MD5_EXCLUSIVE, F_NO_PACING, F_E2EE, F_LINKED = 1, 2, 4, 8, 16, 32
BOX_OVERHEAD = 40
# sky_decode status codes
D_OK, D_BAD_HEADER, D_CORRUPT, D_SIZE, D_UNSUPPORTED, D_LAYOUT, D_TRUNCATED, D_AUTH = 0, -1, -2, -3, -4, -5, -6, -7
D_NAMES = {0: "ok", -1: "bad frame header", -2: "corrupt block", -3: "size mismatch", -4: "unsupported frame feature",
           -5: "unexpected block layout", -6: "truncated frame", -7: "box authentication failed"}

_vp, _u64, _u32, _i32, _str = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int, ctypes.c_char_p
_p_vp, _p_u64, _p_i32, _p_f32 = (ctypes.POINTER(t) for t in (_vp, _u64, _i32, ctypes.c_float))
# every symbol include/skychunk.h declares, name: (restype, argtypes) (tests check the .so exports exactly these)
_ABI = {
    "sky_strerror": (_str, [_i32]),
    "sky_last_error": (_str, [_vp]),
    "sky_abi_version": (_i32, []),
    "sky_device_count": (_i32, [_p_i32]),
    "sky_device_pci_bus_id": (_i32, [_i32, _str, _i32]),
    "sky_kernel_config": (_u32, [_i32]),
    "sky_frame_bound": (_u64, [_u64]),
    "sky_ctx_create": (_i32, [_i32, _u64, _u32, _u32, _p_vp]),
    "sky_ctx_destroy": (_i32, [_vp]),
    "sky_pinned_alloc": (_vp, [_u64]),
    "sky_pinned_free": (_i32, [_vp]),
    "sky_submit": (_i32, [_vp, _u32, _p_vp, _p_u64, _p_vp, _p_u64, _p_u64]),
    "sky_wait": (_i32, [_vp, _u64, _p_u64, _vp, _p_f32]),
    "sky_submit_flags": (_i32, [_vp, _u32, _p_vp, _p_u64, _p_vp, _p_u64, _u32, _str, _p_u64]),
    "sky_set_e2ee_key": (_i32, [_vp, _str]),
    "sky_box_bound": (_u64, [_u64]),
    "sky_process_device": (_i32, [_vp, _u32, _vp, _p_u64, _p_u64, _vp, _p_u64, _p_u64, _u32, _vp, _p_u64, _vp, _p_f32]),
    "sky_decode_device": (_i32, [_vp, _u32, _vp, _p_u64, _p_u64, _vp, _p_u64, _p_u64, _vp, _p_i32, _vp, _p_f32]),
    "sky_decode": (_i32, [_vp, _u32, _p_vp, _p_u64, _p_vp, _p_u64, _p_i32, _vp, _p_f32]),
    "sky_decode_flags": (_i32, [_vp, _u32, _p_vp, _p_u64, _p_vp, _p_u64, _u32, _p_i32, _vp, _p_f32]),
    "sky_device_alloc": (_i32, [_vp, _u64, _p_vp]),
    "sky_device_free": (_i32, [_vp, _vp]),
    "sky_memcpy_h2d": (_i32, [_vp, _vp, _vp, _u64]),
    "sky_memcpy_d2h": (_i32, [_vp, _vp, _vp, _u64]),
    "sky_launch_count": (_u64, [_vp]),
}
ABI_SYMBOLS = tuple(_ABI)


class SkyChunkError(RuntimeError):
    def __init__(self, code: int, detail: str = ""):
        self.code = code
        msg = f"libskychunk error {code}: {_strerror(code)}"
        if detail:
            msg += f" [{detail}]"
        super().__init__(msg)


_lib: Optional[ctypes.CDLL] = None


def _strerror(code: int) -> str:
    try:
        return lib().sky_strerror(code).decode()
    except Exception:
        return "?"


def lib() -> ctypes.CDLL:
    """Load (building first if needed) libskychunk.so."""
    global _lib
    if _lib is not None:
        return _lib
    import os

    from skyplane_b200 import build as _build

    override = os.environ.get("SKYCHUNK_LIB")  # tuning builds (tools/): same ABI, different kernel constants
    if override:
        L = ctypes.CDLL(override)
    else:
        if _build.needs_build():
            _build.build()
        L = ctypes.CDLL(str(LIB_PATH))
    for name, (restype, argtypes) in _ABI.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = restype, argtypes
    _lib = L
    return L


def device_pci_bus_id(device: int) -> str:
    """PCI bus id of CUDA device `device` in CUDA's own device order (honours CUDA_VISIBLE_DEVICES)."""
    buf = ctypes.create_string_buffer(32)
    rc = lib().sky_device_pci_bus_id(device, buf, 32)
    if rc != SKY_OK:
        raise SkyChunkError(rc)
    return buf.value.decode().lower()


def kernel_config() -> dict:
    """Compile-time constants of the loaded build (sky_kernel_config).  linked_window = 0: no F_LINKED in this build."""
    L = lib()
    return {"lz4_entries": L.sky_kernel_config(0), "warps": L.sky_kernel_config(1), "seg_slots": L.sky_kernel_config(2),
            "max_step_log": L.sky_kernel_config(3), "linked_window": L.sky_kernel_config(4),
            "linked_seed_log": L.sky_kernel_config(5), "linked_entries": L.sky_kernel_config(6)}


def require_linked() -> None:
    """Raise unless the loaded build has F_LINKED (a build without it would send independent frames)."""
    if not kernel_config()["linked_window"]:
        raise SkyChunkError(SKY_E_INVALID, "this libskychunk build has no linked-block mode (sky_kernel_config(4) == 0)")


def frame_bound(n: int) -> int:
    return int(lib().sky_frame_bound(n))


def round16(x: int) -> int:
    return (x + 15) & ~15


def _split_digests(buf, n: int) -> list:
    """n 16-byte MD5 digests packed back to back in `buf` -> list of bytes."""
    raw = bytes(buf)
    return [raw[16 * i : 16 * i + 16] for i in range(n)]


def device_count() -> int:
    n = ctypes.c_int(0)
    rc = lib().sky_device_count(ctypes.byref(n))
    if rc != SKY_OK:
        return 0
    return n.value


class PinnedBuffer:
    """Page-locked host memory exposed as a writable memoryview (``.view``) and address (``.addr``)."""

    def __init__(self, nbytes: int):
        self.nbytes = int(nbytes)
        self.addr = lib().sky_pinned_alloc(self.nbytes)
        if not self.addr:
            raise SkyChunkError(SKY_E_NOMEM, "sky_pinned_alloc failed (no CUDA device?)")
        self._arr = (ctypes.c_ubyte * max(1, self.nbytes)).from_address(self.addr)
        self.view = memoryview(self._arr).cast("B")[: self.nbytes]

    def close(self):
        if self.addr:
            self.view.release()
            del self._arr
            lib().sky_pinned_free(self.addr)
            self.addr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Context:
    """One sky_ctx: a GPU, its streams, metadata arrays and (n_slots > 0) staging slabs."""

    def __init__(self, device: int = 0, max_batch_bytes: int = 1 << 30, max_chunks: int = 1024, n_slots: int = 2):
        self._h = ctypes.c_void_p()
        self.device = device
        self.max_chunks = max_chunks
        self.max_batch_bytes = max_batch_bytes
        rc = lib().sky_ctx_create(device, max_batch_bytes, max_chunks, n_slots, ctypes.byref(self._h))
        if rc != SKY_OK:
            detail = lib().sky_last_error(None).decode()
            self._h = ctypes.c_void_p()
            raise SkyChunkError(rc, detail)
        self._inflight = {}

    # ------------------------------------------------------------------ helpers
    def _check(self, rc: int):
        if rc != SKY_OK:
            raise SkyChunkError(rc, lib().sky_last_error(self._h).decode())

    def close(self):
        if self._h:
            lib().sky_ctx_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self) -> int:
        return int(lib().sky_launch_count(self._h))

    # ------------------------------------------------------------------ host-buffer path
    def set_e2ee_key(self, key: Optional[bytes]):
        """32-byte SecretBox key for F_E2EE batches (None switches it off)."""
        if key is not None and len(key) != 32:
            raise ValueError("SecretBox keys are 32 bytes")
        self._check(lib().sky_set_e2ee_key(self._h, key))

    def submit(self, src_addrs: Sequence[int], src_lens: Sequence[int], dst_addrs: Optional[Sequence[int]], dst_caps: Optional[Sequence[int]],
               flags: int = 0, nonces: Optional[bytes] = None) -> int:
        """flags = F_MD5: digests only (dst may be None). | F_E2EE: dst receives sealed boxes; nonces = 24 bytes per chunk."""
        n = len(src_addrs)
        A = ctypes.c_void_p * n
        U = ctypes.c_uint64 * n
        args = (A(*src_addrs), U(*src_lens), A(*dst_addrs) if dst_addrs is not None else None, U(*dst_caps) if dst_caps is not None else None, nonces)
        if nonces is not None and len(nonces) != 24 * n:
            raise ValueError("need 24 nonce bytes per chunk")
        t = ctypes.c_uint64(0)
        self._check(lib().sky_submit_flags(self._h, n, args[0], args[1], args[2], args[3], flags, nonces, ctypes.byref(t)))
        self._inflight[t.value] = (n, args)  # keep the pointer arrays alive until wait()
        return t.value

    def wait(self, ticket: int):
        """-> (out_lens: list[int], digests: list[bytes], kernel_ms: float)"""
        n, _keep = self._inflight.pop(ticket)
        out = (ctypes.c_uint64 * n)()
        md5 = (ctypes.c_ubyte * (16 * n))()
        ms = ctypes.c_float(0)
        self._check(lib().sky_wait(self._h, ticket, out, md5, ctypes.byref(ms)))
        return list(out), _split_digests(md5, n), ms.value

    # ------------------------------------------------------------------ device-resident path
    def process_device(self, d_src: int, src_off: Sequence[int], src_len: Sequence[int], d_dst: int, dst_off: Sequence[int],
                       dst_cap: Sequence[int], flags: int = 0, stream: int = 0):
        """-> (out_lens, digests, kernel_ms). Pointers are raw device addresses (e.g. tensor.data_ptr())."""
        n = len(src_len)
        U = ctypes.c_uint64 * n
        out = U()
        md5 = (ctypes.c_ubyte * (16 * n))()
        ms = ctypes.c_float(0)
        self._check(
            lib().sky_process_device(self._h, n, d_src, U(*src_off), U(*src_len), d_dst, U(*dst_off), U(*dst_cap), flags,
                                     stream or None, out, md5, ctypes.byref(ms))
        )
        return list(out), _split_digests(md5, n), ms.value

    # ------------------------------------------------------------------ receiver side
    def decode_device(self, d_frames: int, frame_off: Sequence[int], frame_len: Sequence[int], d_out: int, out_off: Sequence[int],
                      raw_len: Sequence[int], stream: int = 0):
        """-> (status: list[int], digests: list[bytes], kernel_ms)."""
        n = len(frame_len)
        U = ctypes.c_uint64 * n
        st = (ctypes.c_int32 * n)()
        md5 = (ctypes.c_ubyte * (16 * n))()
        ms = ctypes.c_float(0)
        self._check(lib().sky_decode_device(self._h, n, d_frames, U(*frame_off), U(*frame_len), d_out, U(*out_off), U(*raw_len),
                                            stream or None, st, md5, ctypes.byref(ms)))
        return list(st), _split_digests(md5, n), ms.value

    def decode(self, frame_addrs: Sequence[int], frame_lens: Sequence[int], dst_addrs: Sequence[int], raw_lens: Sequence[int], flags: int = 0):
        """Host buffers, synchronous. -> (status, digests, kernel_ms).  flags = F_E2EE: the payloads are sealed boxes."""
        n = len(frame_addrs)
        A = ctypes.c_void_p * n
        U = ctypes.c_uint64 * n
        st = (ctypes.c_int32 * n)()
        md5 = (ctypes.c_ubyte * (16 * n))()
        ms = ctypes.c_float(0)
        self._check(lib().sky_decode_flags(self._h, n, A(*frame_addrs), U(*frame_lens), A(*dst_addrs), U(*raw_lens), flags, st, md5, ctypes.byref(ms)))
        return list(st), _split_digests(md5, n), ms.value

    # ------------------------------------------------------------------ torch-free device memory
    def device_alloc(self, nbytes: int) -> int:
        p = ctypes.c_void_p()
        self._check(lib().sky_device_alloc(self._h, nbytes, ctypes.byref(p)))
        return p.value

    def device_free(self, dptr: int):
        self._check(lib().sky_device_free(self._h, dptr))

    def h2d(self, dptr: int, data) -> None:
        mv = memoryview(data).cast("B")
        if mv.nbytes == 0:
            return
        buf = (ctypes.c_ubyte * mv.nbytes).from_buffer_copy(mv) if mv.readonly else (ctypes.c_ubyte * mv.nbytes).from_buffer(mv)
        self._check(lib().sky_memcpy_h2d(self._h, dptr, ctypes.addressof(buf), mv.nbytes))

    def d2h(self, dptr: int, nbytes: int) -> bytes:
        if nbytes == 0:
            return b""
        buf = (ctypes.c_ubyte * nbytes)()
        self._check(lib().sky_memcpy_d2h(self._h, ctypes.addressof(buf), dptr, nbytes))
        return bytes(buf)
