"""Hand-built LZ4 frames for the decoder tests, and the plain sequential semantics they are checked against.

A block is written as a list of sequences ``(literals, offset, match_len)``; the last one has ``offset = match_len =
None`` (literals only).  ``decode_plain`` is the byte-at-a-time meaning of such a list, ``seq`` / ``frame`` are its
encoding.  The corpus builders at the bottom label every frame with what the strict oracle, liblz4 and the GPU decoder
must say about it, so the CPU tests (tests/test_decode_conformance.py) and the GPU tests
(tests/test_gpu_decode_edges.py) check the same frames against the same expectations.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np

import oracle

MAGIC = b"\x04\x22\x4d\x18"
BLOCK = 65536
MF_LIMIT = 12  # a match must start at least 12 bytes before the end of its block
LAST_LITERALS = 5  # the last 5 bytes of a block are literals

# GPU decoder statuses (skyplane_b200.native.D_*; repeated here so that the module imports without the library)
D_OK, D_BAD_HEADER, D_CORRUPT, D_SIZE, D_UNSUPPORTED, D_LAYOUT, D_TRUNCATED = 0, -1, -2, -3, -4, -5, -6
# oracle error codes (oracle/skyoracle.c)
E_TRUNCATED, E_MAGIC, E_HEADER, E_BLOCKSIZE, E_CORRUPT, E_SIZE, E_UNSUPPORTED = -1, -2, -3, -4, -5, -7, -8


# ------------------------------------------------------------------------------------------------ encoding
def _ext(n: int) -> bytes:
    """LZ4 length extension: 255-bytes while n >= 255, then the remainder."""
    return b"\xff" * (n // 255) + bytes([n % 255])


def seq(literals: bytes, offset: Optional[int] = None, match_len: Optional[int] = None) -> bytes:
    """One LZ4 sequence: token, literal-length extension, literals, then (unless literals-only) offset and match-length
    extension.  No validation: malformed sequences are built on purpose."""
    ll = len(literals)
    tok_m = 0 if match_len is None else min(match_len - 4, 15)
    out = bytes([(min(ll, 15) << 4) | tok_m])
    if ll >= 15:
        out += _ext(ll - 15)
    out += literals
    if match_len is not None:
        out += offset.to_bytes(2, "little")
        if match_len - 4 >= 15:
            out += _ext(match_len - 4 - 15)
    return out


def block(seqs: Sequence[tuple]) -> bytes:
    return b"".join(seq(*s) for s in seqs)


def header(independent: bool = True, content_size: Optional[int] = None, bd: int = 0x40, flg_extra: int = 0) -> bytes:
    flg = 0x40 | (0x20 if independent else 0) | (0x08 if content_size is not None else 0) | flg_extra
    d = bytes([flg, bd]) + (content_size.to_bytes(8, "little") if content_size is not None else b"")
    return MAGIC + d + bytes([(oracle.xxh32(d) >> 8) & 0xFF])


def frame(blocks: Sequence[Tuple[bool, bytes]], independent: bool = True, content_size: Optional[int] = None, bd: int = 0x40,
          flg_extra: int = 0, content: Optional[bytes] = None) -> bytes:
    """Frame from ``(stored, payload)`` blocks, EndMark appended.  ``flg_extra`` is OR-ed into FLG: with 0x10 (block
    checksum) every block is followed by its XXH32, with 0x04 (content checksum) the XXH32 of ``content`` follows the
    EndMark."""
    out = bytearray(header(independent, content_size, bd, flg_extra))
    for stored, payload in blocks:
        out += (len(payload) | (0x80000000 if stored else 0)).to_bytes(4, "little") + payload
        if flg_extra & 0x10:
            out += oracle.xxh32(payload).to_bytes(4, "little")
    out += bytes(4)
    if flg_extra & 0x04:
        out += oracle.xxh32(content or b"").to_bytes(4, "little")
    return bytes(out)


# ------------------------------------------------------------------------------------------------ plain semantics
def decode_plain(seqs: Sequence[tuple], prior: bytes = b"") -> bytes:
    """The output of one block's sequences, one byte at a time; matches may reach into ``prior`` (earlier blocks of a
    linked frame).  Returns only the block's own bytes."""
    out = bytearray(prior)
    for s in seqs:
        lit, off, ml = (tuple(s) + (None, None))[:3]
        out += lit
        if ml is not None:
            assert 0 < off <= len(out), "decode_plain: offset outside the output"
            for _ in range(ml):
                out.append(out[-off])
    return bytes(out[len(prior):])


def block_sequences(blk: bytes) -> List[Tuple[int, Optional[int], Optional[int]]]:
    """Walk a well-formed compressed block -> [(lit_len, match_start, match_len)], positions relative to the block's first
    output byte; the final sequence has match_start = match_len = None."""
    ip, op, out = 0, 0, []
    while True:
        t = blk[ip]
        ip += 1
        ll = t >> 4
        if ll == 15:
            while True:
                s = blk[ip]
                ip += 1
                ll += s
                if s != 255:
                    break
        ip += ll
        op += ll
        assert ip <= len(blk), "literals run past the block"
        if ip == len(blk):
            out.append((ll, None, None))
            return out
        ip += 2
        ml = t & 15
        if ml == 15:
            while True:
                s = blk[ip]
                ip += 1
                ml += s
                if s != 255:
                    break
        ml += 4
        out.append((ll, op, ml))
        op += ml


def check_block_end_rules(blk: bytes, decoded_len: int) -> None:
    """Assert the LZ4 block format's end-of-block rules: the last 5 bytes are literals and the last match starts at least
    12 bytes before the end of the block."""
    seqs = block_sequences(blk)
    total = sum(ll + (ml or 0) for ll, _, ml in seqs)
    assert total == decoded_len, f"block decodes to {total} bytes, expected {decoded_len}"
    for ll, start, ml in seqs:
        if ml is not None:
            assert start + MF_LIMIT <= decoded_len, f"match at {start} starts less than 12 bytes before the end ({decoded_len})"
            assert start + ml + LAST_LITERALS <= decoded_len, f"match [{start}, {start + ml}) ends inside the last 5 bytes ({decoded_len})"


def frame_blocks(fr: bytes):
    """-> (header length, [(offset of the block header, stored, payload)]) for a frame without block checksums."""
    flg = fr[4]
    ip = 4 + 2 + (8 if flg & 0x08 else 0) + 1
    hdr, out = ip, []
    while True:
        w = int.from_bytes(fr[ip:ip + 4], "little")
        if w == 0:
            return hdr, out
        sz = w & 0x7FFFFFFF
        out.append((ip, bool(w >> 31), fr[ip + 4:ip + 4 + sz]))
        ip += 4 + sz


# ------------------------------------------------------------------------------------------------ corpus
@dataclass
class Case:
    name: str
    frame: bytes
    raw_len: int  # what the receiver expects (WireProtocolHeader.raw_data_len)
    want: Optional[bytes] = None  # what the sequences mean (decoded bytes of a valid frame)
    gpu: int = D_OK  # status the GPU decoder must return
    oracle_err: Optional[int] = None  # error code the oracle raises (None: it decodes to `want`)
    liblz4_ok: bool = True


def _rng(seed):
    return np.random.default_rng(seed)


def _single(name, seqs, independent=True, sized=True, **kw):
    want = decode_plain(seqs)
    fr = frame([(False, block(seqs))], independent, len(want) if sized else None)
    return Case(name, fr, len(want), want, **kw)


MATCH_OFFSETS = list(range(1, 41)) + [63, 64, 65, 255, 256, 4095]
MATCH_LENS = [4, 5, 18, 19, 31, 32, 33, 63, 64, 65, 273, 274, 1000]
LITERAL_RUNS = [0, 1, 14, 15, 16, 63, 64, 65, 269, 270, 271, 4000]
TAIL = 12  # literals closing a block: with them even a final 4-byte match starts >= 12 bytes before the end


def valid_cases() -> List[Case]:
    """Frames every conforming decoder must accept, with the bytes they decode to."""
    r = _rng(2024)
    cases = []
    # every match length at every short offset (warp_match_copy's period path) and at a few long ones (32-byte rounds)
    for off in MATCH_OFFSETS:
        seqs = [(r.bytes(off), off, MATCH_LENS[0])]
        seqs += [(r.bytes(1 + i % 3), off, ml) for i, ml in enumerate(MATCH_LENS[1:])]
        seqs += [(r.bytes(TAIL),)]
        cases.append(_single(f"offset{off}", seqs))
    # literal runs at the token / extension boundaries, inside a block and as its last sequence
    seqs = [(r.bytes(20), 20, 8)] + [(r.bytes(n), 5, 4 + n % 11) for n in LITERAL_RUNS] + [(r.bytes(TAIL),)]
    cases.append(_single("literal_runs", seqs))
    for n in LITERAL_RUNS[1:]:
        if n >= LAST_LITERALS:
            cases.append(_single(f"final_literals{n}", [(r.bytes(30), 9, 40), (r.bytes(n),)]))
        cases.append(_single(f"literals_only{n}", [(r.bytes(n),)]))
    cases.append(phase_case(r))
    # matches reaching exactly the first byte of an independent block, in the first block and in a later one
    lead = r.bytes(BLOCK)
    seqs = [(r.bytes(40), 40, 300), (r.bytes(30),)]
    cases.append(_single("offset_to_first_block_start", seqs))
    body = decode_plain(seqs)
    cases.append(Case("offset_to_later_block_start", frame([(True, lead), (False, block(seqs))], True, BLOCK + len(body)), BLOCK + len(body),
                      lead + body))
    # linked frames: reach 65535 bytes back into the previous (stored) block; an overlapping period-3 match straddling
    # the boundary; a compressed block -> stored block -> compressed block chain
    s1 = [(b"Q", 65535, 1000), (r.bytes(20),)]
    b1 = decode_plain(s1, lead)
    cases.append(Case("linked_offset65535", frame([(True, lead), (False, block(s1))], False, BLOCK + len(b1)), BLOCK + len(b1), lead + b1))
    full0 = [(r.bytes(64), 64, BLOCK - 64 - 5), (r.bytes(5),)]
    o0 = decode_plain(full0)
    s1 = [(b"", 3, 100), (r.bytes(200), 40000, 3000), (r.bytes(9),)]
    o1 = decode_plain(s1, o0)
    fr = frame([(False, block(full0)), (False, block(s1))], False, BLOCK + len(o1))
    cases.append(Case("linked_period3_across_boundary", fr, BLOCK + len(o1), o0 + o1))
    mid = r.bytes(BLOCK)
    s2 = [(r.bytes(3), 65535 - 7, 500), (b"", 1, 64), (r.bytes(6),)]
    o2 = decode_plain(s2, o0 + mid)
    fr = frame([(False, block(full0)), (True, mid), (False, block(s2))], False, 2 * BLOCK + len(o2))
    cases.append(Case("linked_stored_then_compressed", fr, 2 * BLOCK + len(o2), o0 + mid + o2))
    # frames without a content size (independent and linked, one and several blocks)
    cases.append(_single("no_content_size", [(r.bytes(50), 17, 300), (r.bytes(13),)], sized=False))
    fr = frame([(False, block(full0)), (False, block(s1))], False, None)
    cases.append(Case("linked_no_content_size", fr, BLOCK + len(o1), o0 + o1))
    fr = frame([(True, lead), (False, block(seqs))], True, None)
    cases.append(Case("indep_no_content_size", fr, BLOCK + len(body), lead + body))
    # the empty frame with a content size of 0 (19 bytes) and without one (11 bytes, what the GPU sender emits)
    cases.append(Case("empty_sized", frame([], True, 0), 0, b""))
    cases.append(Case("empty", frame([], True, None), 0, b""))
    # blocks ending exactly at the limits: 5 final literals; the last match starting exactly 12 bytes before the end
    for size in (BLOCK, 1000):
        cases.append(_single(f"final5_{size}", [(r.bytes(64), 64, size - 64 - 5), (r.bytes(5),)]))
        cases.append(_single(f"mflimit_{size}", [(r.bytes(64), 64, size - 64 - 15), (r.bytes(3), 64, 7), (r.bytes(5),)]))
        cases.append(_single(f"mflimit_nolit_{size}", [(r.bytes(64), 64, size - 64 - 12), (b"", 64, 7), (r.bytes(5),)]))
    return cases


def phase_case(r) -> Case:
    """One block in which a literal run of >= 64 bytes starts at every (output position mod 16) x (frame position mod 4):
    warp_copy's funnel-shift path depends on both (the GPU places frames and outputs 16-byte aligned)."""
    seqs, ip, op = [], 15 + 4, 0  # ip: frame position (header with content size + block header), op: output position

    def push(s):
        nonlocal ip, op
        seqs.append(s)
        ip += len(seq(*s))
        op += len(s[0]) + s[2]

    push((r.bytes(32), 5, 4))
    for a in range(16):
        for b in range(4):
            # setter: k literals + a match of 19..34 bytes (4 + k encoded bytes) puts the next run at phase (a, b); the run
            # itself is a token and one extension byte, then its literals
            k = (b - ip - 6) % 4
            push((r.bytes(k), 7, 19 + (a - op - k - 19) % 16))
            assert (ip + 2) % 4 == b and op % 16 == a
            push((r.bytes(64 + (a * 4 + b) % 9), 3, 4))
    seqs.append((r.bytes(TAIL),))
    want = decode_plain(seqs)
    return Case("literal_phases", frame([(False, block(seqs))], True, len(want)), len(want), want)


def rejected_cases() -> List[Case]:
    """Malformed frames: the oracle's error code and the exact GPU status.  liblz4 rejects them too, except the few marked
    liblz4_ok (it is more lenient than the format there)."""
    r = _rng(7)
    lead = r.bytes(BLOCK)
    cases = []

    def single(name, blk, raw, gpu, err=E_CORRUPT, sized=True):
        cases.append(Case(name, frame([(False, blk)], True, raw if sized else None), raw, None, gpu, err, False))

    s = [(r.bytes(40), 41, 300), (r.bytes(30),)]
    single("offset_before_first_block", block(s), 40 + 300 + 30, D_CORRUPT)
    raw = BLOCK + 370
    cases.append(Case("offset_before_later_block", frame([(True, lead), (False, block(s))], True, raw), raw, None, D_CORRUPT, E_CORRUPT, False))
    # liblz4 1.9.4 accepts offset 0 (it copies whatever its output buffer holds); the format forbids it
    cases.append(Case("offset_zero", frame([(False, block([(r.bytes(40), 0, 300), (r.bytes(30),)]))], True, 370), 370, None, D_CORRUPT,
                      E_CORRUPT, True))
    single("ends_after_offset", block([(r.bytes(40), 8, 10)]), 50, D_CORRUPT)
    single("match_extension_missing", block([(r.bytes(40), 8, 500)])[:-2], 540, D_CORRUPT)
    single("literals_past_block", seq(r.bytes(10))[:-5], 10, D_CORRUPT)
    single("literal_extension_past_block", b"\xf0\xff\xff", 15 + 510, D_CORRUPT)
    single("literal_extension_missing", b"\xf0", 15, D_CORRUPT)
    single("match_extension_past_block", seq(r.bytes(20), 4, 200)[:-1], 220, D_CORRUPT)
    single("match_extension_255_past_block", seq(r.bytes(20), 4, 4 + 15 + 300)[:-1], 339, D_CORRUPT)
    # a block decoding to more than 64 KiB (followed by a second block so that the GPU's block table fits the frame)
    big = [(r.bytes(64), 64, BLOCK), (r.bytes(TAIL),)]
    raw = BLOCK + 100
    fr = frame([(False, block(big)), (True, r.bytes(100))], True, raw)
    cases.append(Case("block_over_64KiB", fr, raw, None, D_CORRUPT, E_CORRUPT, False))
    # a block size word above the 64 KiB maximum
    fr = frame([(True, r.bytes(BLOCK + 1))], True, BLOCK + 1)
    cases.append(Case("block_word_over_64KiB", fr, BLOCK + 1, None, D_CORRUPT, E_BLOCKSIZE, False))
    cases += end_rule_cases()
    # header / size classes
    good = frame([(False, block([(r.bytes(30), 9, 40), (r.bytes(7),)]))], True, 77)
    cases.append(Case("bad_magic", b"\x05" + good[1:], 77, None, D_BAD_HEADER, E_MAGIC, False))
    cases.append(Case("bad_header_checksum", good[:14] + bytes([good[14] ^ 1]) + good[15:], 77, None, D_BAD_HEADER, E_HEADER, False))
    cases.append(Case("bad_version", header(True, 77, flg_extra=0x80) + good[15:], 77, None, D_BAD_HEADER, E_HEADER, False))
    lying = frame([(False, block([(r.bytes(30), 9, 40), (r.bytes(7),)]))], True, 78)  # decodes to 77 bytes
    cases.append(Case("content_size_mismatch", lying, 77, None, D_SIZE, E_SIZE, False))
    return cases


def end_rule_cases() -> List[Case]:
    """Blocks breaking the end-of-block rules.  liblz4 rejects all but the last two; the oracle and the GPU decoder reject
    every one (the format's rules are slightly stricter than liblz4's check of them)."""
    r = _rng(11)
    out = []

    def add(name, seqs, liblz4_ok=False):
        want = decode_plain(seqs)
        out.append(Case(name, frame([(False, block(seqs))], True, len(want)), len(want), want, D_CORRUPT, E_CORRUPT, liblz4_ok))

    add("short_final4_noext", [(r.bytes(8), 8, 10), (r.bytes(4),)])
    add("short_final0", [(r.bytes(32), 8, 20), (b"",)])
    add("short_final0_two_matches", [(r.bytes(8), 8, 30), (r.bytes(2), 8, 30), (b"",)])
    add("full_final4", [(r.bytes(64), 64, BLOCK - 64 - 4), (r.bytes(4),)])
    add("full_match_starts_11_before_end", [(r.bytes(64), 64, BLOCK - 64 - 19), (r.bytes(8), 64, 4), (r.bytes(7),)])
    # liblz4 accepts these two: its decoder checks the output-side rules against the room left in its 64 KiB block buffer,
    # not against the block's real length.  Only a non-conformant encoder produces them; the oracle and the GPU refuse them.
    add("short_match_starts_11_before_end", [(r.bytes(64), 64, 1000 - 64 - 19), (r.bytes(8), 64, 4), (r.bytes(7),)], liblz4_ok=True)
    add("short_final4_after_extended_match", [(r.bytes(8), 8, 4 + 15 + 3), (r.bytes(4),)], liblz4_ok=True)
    return out


def layout_cases() -> List[Case]:
    """Valid LZ4 frames outside the layout the GPU decoder handles (64 KiB blocks, only the last one short, no checksums):
    liblz4 decodes them, the GPU decoder reports D_LAYOUT / D_UNSUPPORTED."""
    r = _rng(13)
    cases = []
    data = r.bytes(100)
    for bd in (0x50, 0x60, 0x70):
        cases.append(Case(f"bd{bd:#x}", frame([(True, data)], True, 100, bd=bd), 100, data, D_LAYOUT, None))
    seqs = [(r.bytes(64), 64, 100000), (r.bytes(TAIL),)]
    want = decode_plain(seqs)
    cases.append(Case("bd0x50_block_over_64KiB", frame([(False, block(seqs))], True, len(want), bd=0x50), len(want), want, D_LAYOUT, None))
    a, short, c = r.bytes(BLOCK), [(r.bytes(64), 64, 60000 - 64 - 7), (r.bytes(7),)], r.bytes(10000)
    want = a + decode_plain(short) + c
    fr = frame([(True, a), (False, block(short)), (True, c)], True, len(want))
    cases.append(Case("short_middle_block", fr, len(want), want, D_LAYOUT, None))
    a, b = r.bytes(1000), r.bytes(BLOCK)
    cases.append(Case("short_stored_first_block", frame([(True, a), (True, b)], True, len(a + b)), len(a + b), a + b, D_LAYOUT, None))
    seqs = [(r.bytes(30), 9, 400), (r.bytes(9),)]
    want = decode_plain(seqs)
    fr = frame([(False, block(seqs))], True, len(want), flg_extra=0x04, content=want)
    cases.append(Case("content_checksum", fr, len(want), want, D_UNSUPPORTED, E_UNSUPPORTED))
    fr = frame([(False, block(seqs))], True, len(want), flg_extra=0x10)
    cases.append(Case("block_checksum", fr, len(want), want, D_UNSUPPORTED, E_UNSUPPORTED))
    return cases


def boundary_cuts(fr: bytes, seeded: int, seed: int, margin: int = 24) -> List[int]:
    """Proper-prefix lengths of `fr`: every cut within `margin` bytes of a header / block boundary, plus `seeded` seeded
    cuts anywhere."""
    hdr, blocks = frame_blocks(fr)
    marks = [0, hdr] + [ip for ip, _, _ in blocks] + [ip + 4 for ip, _, _ in blocks] + [len(fr) - 4, len(fr)]
    cuts = {k for m in marks for k in range(m - margin, m + margin + 1) if 0 <= k < len(fr)}
    cuts |= {int(k) for k in _rng(seed).integers(0, len(fr), size=seeded)}
    return sorted(cuts)


def prefix_sets():
    """-> [(name, frame, raw_len, prefix lengths)]: proper prefixes that must all be reported as truncated."""
    from skyplane_b200 import synth
    import oracle.reflib as ref

    empty = frame([], True, None)
    text = (b"abcdefg" * (3 * BLOCK // 7 + 200))[:3 * BLOCK + 777]
    small = oracle.lz4f_compress_indep(text)
    assert len(small) < 1024
    sil = synth.silesia_like_chunk(5, 5 * BLOCK + 1234)
    indep = oracle.lz4f_compress_indep(sil)
    linked = ref.lz4f_compress(sil)
    return [("empty", empty, 0, list(range(len(empty)))),
            ("compressible", small, len(text), list(range(len(small)))),
            ("silesia_indep", indep, len(sil), boundary_cuts(indep, 256, 1)),
            ("silesia_linked", linked, len(sil), boundary_cuts(linked, 256, 2))]
