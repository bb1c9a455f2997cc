"""ChunkStage: the host side of the B200 compress+hash stage (pinned staging + libskychunk).

This is what replaces, for a batch of chunks, the reference's two per-chunk CPU calls
(``lz4.frame.compress`` at skyplane/gateway/operators/gateway_operator.py:359 and the
``hashlib.md5`` loop at skyplane/obj_store/s3_interface.py:181-192).  Chunk bytes are read
straight into page-locked host memory, shipped to HBM, compressed + hashed by one fused kernel
launch, and the frames land in page-locked memory ready for ``sock.sendall``.

No CPU fallback: constructing a ChunkStage without a CUDA device raises SkyChunkError.
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from typing import List, Optional, Sequence, Union

from skyplane_b200 import native

BytesLike = Union[bytes, bytearray, memoryview]


@dataclass
class StageResult:
    """What the sender needs for one chunk (gateway_operator.py:367-372)."""

    frame: memoryview  # wire payload (view into the slot's pinned memory; valid until the slot is reused): the LZ4 frame,
    #                    or the chunk itself when compression is off, sealed in a SecretBox when E2EE is on
    md5: bytes  # 16 raw bytes == hashlib.md5(chunk).digest()
    raw_len: int  # WireProtocolHeader.raw_data_len
    comp_len: int  # WireProtocolHeader.data_len (length of `frame`)
    is_compressed: bool = True  # WireProtocolHeader.is_compressed
    is_encrypted: bool = False

    def frame_bytes(self) -> bytes:
        return bytes(self.frame)


class _Slot:
    def __init__(self, in_bytes: int, out_bytes: int):
        self.inp = native.PinnedBuffer(in_bytes)
        self.out = native.PinnedBuffer(out_bytes)
        self.reset()

    def reset(self):
        self.in_off: List[int] = []
        self.lens: List[int] = []
        self.out_off: List[int] = []
        self.in_used = 0
        self.out_used = 0
        self.ticket: Optional[int] = None
        self.flags = 0

    def reserve(self, n: int) -> memoryview:
        """Reserve room for an n-byte chunk; returns the writable pinned view to fill."""
        bound = native.frame_bound(n) + native.BOX_OVERHEAD  # (room for the SecretBox nonce + tag when E2EE is on)
        if self.in_used + native.round16(n) > self.inp.nbytes or self.out_used + native.round16(bound) > self.out.nbytes:
            raise native.SkyChunkError(native.SKY_E_CAPACITY, "batch exceeds the stage's staging buffers")
        off = self.in_used
        self.in_off.append(off)
        self.lens.append(n)
        self.out_off.append(self.out_used)
        self.in_used += native.round16(n)
        self.out_used += native.round16(bound)
        return self.inp.view[off : off + n]


class ChunkStage:
    def __init__(self, device: int = 0, max_batch_bytes: int = 256 << 20, max_chunks: int = 256, n_slots: int = 2):
        if n_slots < 1:
            raise ValueError("n_slots must be >= 1")
        self.ctx = native.Context(device, max_batch_bytes, max_chunks, n_slots)
        self.max_chunks = max_chunks
        self.max_batch_bytes = max_batch_bytes
        in_bytes = native.round16(max_batch_bytes) + 16 * max_chunks
        out_bytes = max_batch_bytes + 4 * (max_batch_bytes // 65536 + 1) + 128 * max_chunks
        self._slots = [_Slot(in_bytes, out_bytes) for _ in range(n_slots)]
        self._free = list(self._slots)

    # ------------------------------------------------------------------ async API
    def begin(self) -> _Slot:
        """Take a free staging slot (raises SKY_E_BUSY if every slot has an un-collected batch)."""
        if not self._free:
            raise native.SkyChunkError(native.SKY_E_BUSY, "collect() an earlier batch first")
        s = self._free.pop()
        s.reset()
        return s

    def release(self, slot: _Slot):
        """Give back a slot taken with begin() that was never launched."""
        slot.reset()
        self._free.append(slot)

    def fits(self, slot: _Slot, n: int) -> bool:
        return (
            len(slot.lens) < self.max_chunks
            and slot.in_used + native.round16(n) <= slot.inp.nbytes
            and slot.out_used + native.round16(native.frame_bound(n) + native.BOX_OVERHEAD) <= slot.out.nbytes
        )

    def add_bytes(self, slot: _Slot, data: BytesLike) -> int:
        mv = memoryview(data).cast("B")
        dst = slot.reserve(mv.nbytes)
        if mv.nbytes:
            dst[:] = mv
        return len(slot.lens) - 1

    def add_file(self, slot: _Slot, path: os.PathLike, length: int) -> int:
        """Read exactly `length` bytes of a chunk file into pinned memory (gateway_operator.py:350-352)."""
        dst = slot.reserve(length)
        got = 0
        with open(path, "rb", buffering=0) as f:
            while got < length:
                r = f.readinto(dst[got:])
                if not r:
                    break
                got += r
            extra = f.read(1) if got == length else b""
        if got != length or extra:
            slot.in_off.pop(); slot.lens.pop(); slot.out_off.pop()
            raise AssertionError(f"chunk file {path} has size != {length}")
        return len(slot.lens) - 1

    def add_stream(self, slot: _Slot, body, length: int) -> int:
        """Ingest without a chunk file (SURVEY.md section 8f row 3): fill the next staging range straight from a streaming
        body -- any object with ``readinto(buffer)`` (a file, a socket file, ``io.BufferedReader`` around an HTTP response,
        botocore's ``StreamingBody._raw_stream``) or ``read(n)`` -- the way ``download_object`` loops over 64 KiB pieces
        (skyplane/obj_store/s3_interface.py:183-191), minus the tmpfs file and minus the host-side MD5 (the GPU supplies it)."""
        dst = slot.reserve(length)
        got = 0
        readinto = getattr(body, "readinto", None)
        while got < length:
            if readinto is not None:
                r = readinto(dst[got:])
            else:
                piece = body.read(min(length - got, 1 << 20))
                r = len(piece)
                dst[got : got + r] = piece
            if not r:
                break
            got += r
        if got != length:
            slot.in_off.pop(); slot.lens.pop(); slot.out_off.pop()
            slot.in_used -= native.round16(length)
            slot.out_used -= native.round16(native.frame_bound(length) + native.BOX_OVERHEAD)
            raise EOFError(f"stream ended after {got} of {length} bytes")
        return len(slot.lens) - 1

    def set_e2ee_key(self, key: Optional[bytes]):
        """SecretBox key (32 bytes) for encrypt=True batches / decode(encrypted=True); None switches E2EE off."""
        self.ctx.set_e2ee_key(key)
        self._has_key = key is not None

    def launch(self, slot: _Slot, compress: bool = True, encrypt: bool = False, nonces: Optional[bytes] = None,
               linked: bool = False) -> _Slot:
        """compress=False is the reference's `compress: false` (digest only, the chunk passes through);
        encrypt=True seals every payload with the stage's key (nonces: 24 bytes per chunk, default os.urandom);
        linked=True emits linked-block frames (F_LINKED: better ratio on text; no effect without compression)."""
        if not slot.lens:
            raise ValueError("empty batch")
        if linked:
            native.require_linked()
        base_in, base_out = slot.inp.addr, slot.out.addr
        src = [base_in + o for o in slot.in_off]
        flags = native.F_MD5 | (native.F_LZ4 if compress else 0) | (native.F_E2EE if encrypt else 0) | (native.F_LINKED if linked else 0)
        if encrypt and nonces is None:
            nonces = os.urandom(24 * len(slot.lens))  # what nacl.utils.random(24) draws per message
        if compress or encrypt:
            dst = [base_out + o for o in slot.out_off]
            caps = [(native.frame_bound(n) if compress else n) + (native.BOX_OVERHEAD if encrypt else 0) for n in slot.lens]
        else:
            dst = caps = None
        slot.flags = flags
        slot.ticket = self.ctx.submit(src, slot.lens, dst, caps, flags, nonces)
        return slot

    def collect(self, slot: _Slot) -> List[StageResult]:
        out_lens, digests, self.last_kernel_ms = self.ctx.wait(slot.ticket)
        comp, enc = bool(slot.flags & native.F_LZ4), bool(slot.flags & native.F_E2EE)
        res = []
        for io, o, cl, dg, n in zip(slot.in_off, slot.out_off, out_lens, digests, slot.lens):
            payload = slot.out.view[o : o + cl] if (comp or enc) else slot.inp.view[io : io + n]
            res.append(StageResult(frame=payload, md5=dg, raw_len=n, comp_len=len(payload), is_compressed=comp, is_encrypted=enc))
        slot.ticket = None
        self._free.append(slot)
        return res

    # ------------------------------------------------------------------ sync convenience
    def process(self, chunks: Sequence[BytesLike], compress: bool = True, encrypt: bool = False, nonces: Optional[bytes] = None,
                linked: bool = False) -> List[StageResult]:
        """Compress + hash (+ seal) a list of in-memory chunks; payloads are returned as independent bytes."""
        out: List[StageResult] = []
        i = 0
        while i < len(chunks):
            slot = self.begin()
            j = i
            while j < len(chunks) and self.fits(slot, memoryview(chunks[j]).nbytes):
                self.add_bytes(slot, chunks[j])
                j += 1
            if j == i:
                self.release(slot)
                raise native.SkyChunkError(native.SKY_E_CAPACITY, f"chunk of {memoryview(chunks[i]).nbytes} bytes exceeds max_batch_bytes")
            self.launch(slot, compress, encrypt, nonces[24 * i : 24 * j] if nonces is not None else None, linked)
            for r in self.collect(slot):
                out.append(StageResult(frame=memoryview(bytes(r.frame)), md5=r.md5, raw_len=r.raw_len, comp_len=r.comp_len,
                                       is_compressed=r.is_compressed, is_encrypted=r.is_encrypted))
            i = j
        return out

    # ------------------------------------------------------------------ receiver side
    def decode(self, frames: Sequence[BytesLike], raw_lens: Sequence[int], encrypted: bool = False):
        """Decode LZ4 frames and digest the decoded bytes (gateway_receiver.py:195-201 + the missing hash check);
        encrypted=True: the payloads are SecretBox messages, opened on the device first (gateway_receiver.py:191-193).
        -> list of (data: bytes | None, md5: bytes, status: int); data is None when status != 0."""
        out = []
        i = 0
        if self._free is None or not self._free:
            raise native.SkyChunkError(native.SKY_E_BUSY, "collect() pending batches before decode()")
        slot = self._free[-1]  # its pinned buffers are idle: frames are staged in `out`, decoded bytes land in `inp`
        while i < len(frames):
            f_off, o_off, fp, op = [], [], 0, 0
            j = i
            while j < len(frames) and j - i < self.max_chunks:
                fl, rl = memoryview(frames[j]).nbytes, raw_lens[j]
                if fp + native.round16(fl) > slot.out.nbytes or op + native.round16(rl) > slot.inp.nbytes:
                    break
                slot.out.view[fp : fp + fl] = memoryview(frames[j]).cast("B")
                f_off.append(fp)
                o_off.append(op)
                fp += native.round16(fl)
                op += native.round16(rl)
                j += 1
            if j == i:
                raise native.SkyChunkError(native.SKY_E_CAPACITY, "frame exceeds the stage's staging buffers")
            lens = [memoryview(frames[k]).nbytes for k in range(i, j)]
            raws = list(raw_lens[i:j])
            st, dg, self.last_kernel_ms = self.ctx.decode([slot.out.addr + o for o in f_off], lens, [slot.inp.addr + o for o in o_off], raws,
                                                          native.F_E2EE if encrypted else 0)
            for k in range(j - i):
                data = bytes(slot.inp.view[o_off[k] : o_off[k] + raws[k]]) if st[k] == 0 else None
                out.append((data, dg[k], st[k]))
            i = j
        return out

    def close(self):
        self.ctx.close()
        for s in self._slots:
            s.inp.close()
            s.out.close()
        self._slots = []
        self._free = []
