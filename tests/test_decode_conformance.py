"""Labels of the hand-built LZ4 frame corpus (tests/lz4_craft.py), settled on the CPU: what the strict oracle decoder,
liblz4 (LZ4F_decompress, what lz4.frame.decompress calls at gateway_receiver.py:196) and pyarrow say about each frame.
tests/test_gpu_decode_edges.py holds the GPU decoder to the same labels."""
import numpy as np
import pytest

import lz4_craft as craft
import oracle
import oracle.reflib as ref
from skyplane_b200 import synth

pytestmark = pytest.mark.skipif(not ref.available(), reason="liblz4.so.1 not present")


def _liblz4(c):
    return ref.lz4f_decompress(c.frame, max(c.raw_len, craft.BLOCK))


def test_valid_corpus_decodes_to_the_plain_bytes():
    try:
        import pyarrow as pa
    except ImportError:
        pa = None
    cases = craft.valid_cases()
    assert len({c.name for c in cases}) == len(cases)
    for c in cases:
        assert len(c.want) == c.raw_len, c.name
        assert oracle.lz4f_decode(c.frame, c.raw_len) == c.want, c.name
        assert _liblz4(c) == c.want, c.name
        if pa is not None and c.raw_len:
            assert pa.decompress(c.frame, decompressed_size=c.raw_len, codec="lz4").to_pybytes() == c.want, c.name
        # every valid case is also a conforming one: the end-of-block rules hold in each compressed block
        pos = 0
        for _, stored, payload in craft.frame_blocks(c.frame)[1]:
            n = min(craft.BLOCK, c.raw_len - pos)
            if not stored:
                craft.check_block_end_rules(payload, n)
            pos += n


def test_corpus_reaches_every_offset_length_and_literal_boundary():
    cases = {c.name: c for c in craft.valid_cases()}
    for off in craft.MATCH_OFFSETS:
        seqs = craft.block_sequences(craft.frame_blocks(cases[f"offset{off}"].frame)[1][0][2])
        assert [ml for _, _, ml in seqs[:-1]] == craft.MATCH_LENS
    seqs = craft.block_sequences(craft.frame_blocks(cases["literal_runs"].frame)[1][0][2])
    assert [ll for ll, _, _ in seqs[1:-1]] == craft.LITERAL_RUNS


def test_literal_runs_start_at_every_output_and_frame_phase():
    c = craft.phase_case(np.random.default_rng(0))
    hdr, blocks = craft.frame_blocks(c.frame)
    ip, _, blk = blocks[0]
    ip += 4  # first byte of the block's sequences
    seen, op, k = set(), 0, 0
    while k < len(blk):  # walk the encoding again, recording where every literal run of >= 64 bytes starts
        t = blk[k]
        k += 1
        ll = t >> 4
        if ll == 15:
            while True:
                s = blk[k]
                k += 1
                ll += s
                if s != 255:
                    break
        if ll >= 64:
            seen.add((op % 16, (ip + k) % 4))
        k += ll
        op += ll
        if k == len(blk):
            break
        ml = t & 15
        k += 2
        if ml == 15:
            while True:
                s = blk[k]
                k += 1
                ml += s
                if s != 255:
                    break
        op += ml + 4
    assert seen == {(a, b) for a in range(16) for b in range(4)}
    assert oracle.lz4f_decode(c.frame, c.raw_len) == c.want == _liblz4(c)


def test_rejected_by_the_oracle_and_liblz4():
    cases = craft.rejected_cases()
    assert len({c.name for c in cases}) == len(cases)
    # where liblz4 is more lenient than the format: offset 0, and two end-of-block violations in short blocks
    assert [c.name for c in cases if c.liblz4_ok] == ["offset_zero", "short_match_starts_11_before_end", "short_final4_after_extended_match"]
    for c in cases:
        with pytest.raises(oracle.OracleError) as e:
            oracle.lz4f_decode(c.frame, c.raw_len)
        assert e.value.code == c.oracle_err, c.name
        if c.liblz4_ok:
            assert len(_liblz4(c)) == c.raw_len, c.name
        else:
            with pytest.raises(ValueError):
                _liblz4(c)
                pytest.fail(f"liblz4 accepted {c.name}")


def test_end_of_block_rules_are_enforced():
    """The oracle rejects every block breaking the format's end-of-block rules (the last 5 bytes are literals, the last
    match starts at least 12 bytes before the end).  liblz4 rejects all but two kinds, both in short blocks: it checks the
    rules against the room left in its 64 KiB block buffer rather than the block's real end.  Only a non-conformant encoder
    emits such a block; the oracle and the GPU decoder refuse it on purpose."""
    cases = craft.end_rule_cases()
    assert [c.name for c in cases if c.liblz4_ok] == ["short_match_starts_11_before_end", "short_final4_after_extended_match"]
    for c in cases:
        with pytest.raises(oracle.OracleError) as e:
            oracle.lz4f_decode(c.frame, c.raw_len)
        assert e.value.code == craft.E_CORRUPT, c.name
        if c.liblz4_ok:
            assert _liblz4(c) == c.want, c.name
        else:
            with pytest.raises(ValueError):
                _liblz4(c)
                pytest.fail(f"liblz4 accepted {c.name}")


def test_gpu_layout_limits_are_valid_lz4():
    """Frames liblz4 decodes that lie outside the GPU decoder's layout (64 KiB blocks, only the last one short, no
    checksums).  liblz4's verdict is pinned so that the divergence is on record."""
    for c in craft.layout_cases():
        assert _liblz4(c) == c.want, c.name
        if c.oracle_err is None:
            assert oracle.lz4f_decode(c.frame, c.raw_len) == c.want, c.name
        else:
            with pytest.raises(oracle.OracleError) as e:
                oracle.lz4f_decode(c.frame, c.raw_len)
            assert e.value.code == c.oracle_err, c.name


def test_every_proper_prefix_is_truncated():
    """A receiver polls a payload that is still arriving: every proper prefix of a valid frame must read as truncated,
    never as corrupt (GatewayDecompressVerify re-queues only truncated frames)."""
    for name, fr, raw, cuts in craft.prefix_sets():
        assert oracle.lz4f_decode(fr, raw) is not None
        for k in cuts:
            with pytest.raises(oracle.OracleError) as e:
                oracle.lz4f_decode(fr[:k], raw)
            assert e.value.code == craft.E_TRUNCATED, (name, k)
        assert len(cuts) >= min(len(fr), 256), name


def _encoder_inputs():
    lens = list(range(13, 201)) + [1000, 4096, 65536, 65537, 65536 + 13, 65536 + 14, 70000, 131089]
    return [d for n in lens for d in (bytes(n), (b"abcdefg" * (n // 7 + 1))[:n], (b"it was the best of times " * (n // 25 + 1))[:n],
                                     synth.silesia_like_chunk(n, n))]


def test_our_encoders_obey_the_end_of_block_rules():
    """liblz4 checks the output-side rules against 64 KiB of room, not the block's real length, so it would not notice an
    encoder breaking them in a short last block; the GPU decoder and the oracle would refuse such a frame."""
    import sys
    from pathlib import Path

    sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
    from tools import tile_model

    datas = _encoder_inputs()
    checked = 0
    for enc in (tile_model.frame, oracle.lz4f_compress_indep, oracle.lz4f_compress):
        for d in datas:
            pos = 0
            for _, stored, payload in craft.frame_blocks(enc(d))[1]:
                n = min(craft.BLOCK, len(d) - pos)
                if not stored:
                    craft.check_block_end_rules(payload, n)
                    checked += 1
                pos += n
    assert checked > 2 * len(datas)
