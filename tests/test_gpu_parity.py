"""GPU parity tests: the fused CUDA stage, called through the C ABI, against the CPU oracle,
the reference's engines (liblz4 decoder / hashlib) and the committed golden vectors.

Bars: MD5 bit-exact; LZ4 frames decode bit-identically with three independent decoders (strict oracle
decoder, liblz4's LZ4F_decompress = what lz4.frame.decompress calls at gateway_receiver.py:196, pyarrow);
compression ratio >= 0.95 x the reference's on the compressible workload (16 x 16 MiB); frames byte-identical to the
sequential twin of the kernel's parse (tools/lz4_tile_model.c).
"""
import hashlib

import numpy as np
import pytest

import oracle
import oracle.reflib as ref
from gpu_util import run_device
from skyplane_b200 import native, synth
from skyplane_b200.stage import ChunkStage

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(300, method="thread")]

RNG = np.random.default_rng(77)
EDGE_LENS = [0, 1, 2, 11, 12, 13, 14, 15, 16, 17, 55, 56, 63, 64, 65, 119, 120, 128, 255, 4096, 65535, 65536, 65537,
             65536 + 12, 65536 + 13, 131072, 131073, 200000, (1 << 20) - 1, 1 << 20, (1 << 20) + 1]


@pytest.fixture(scope="module")
def ctx():
    c = native.Context(0, 1 << 30, 4096, 0)
    yield c
    c.close()


def kinds(n, rng=RNG):
    return {
        "random": rng.bytes(n),
        "zeros": bytes(n),
        "period7": (b"abcdefg" * (n // 7 + 1))[:n],
        "text": (b"it was the best of times, it was the worst of times; " * (n // 50 + 1))[:n],
        "half": (b"lorem ipsum dolor sit amet " * (n // 54 + 1))[: n // 2] + rng.bytes(n - n // 2),
    }


def check_frame(frame: bytes, data: bytes):
    n = len(data)
    assert len(frame) <= native.frame_bound(n)
    out, info = oracle.lz4f_decode(frame, n, with_info=True)
    assert out == data
    assert info["consumed"] == len(frame)
    assert info["bd"] == 0x40 and info["flg"] == (0x68 if n else 0x60)
    assert info["blocks"] == (n + 65535) // 65536
    assert ref.lz4f_decompress(frame, n) == data  # the reference's decoder
    return info


# ---------------------------------------------------------------- MD5
def test_md5_golden_vectors(ctx, golden):
    g = golden["md5_kat"]
    msgs = [bytes.fromhex(c["msg_hex"]) for c in g["rfc1321"]] + [bytes(c["len"]) for c in g["zeros"]]
    want = [c["md5"] for c in g["rfc1321"]] + [c["md5"] for c in g["zeros"]]
    _, digests, _, _ = run_device(ctx, msgs)
    assert [d.hex() for d in digests] == want
    _, digests, _, _ = run_device(ctx, msgs, flags=native.F_MD5)  # MD5-only launch
    assert [d.hex() for d in digests] == want


def test_md5_ragged_batch_matches_hashlib(ctx):
    msgs = [RNG.bytes(n) for n in EDGE_LENS] + [RNG.bytes(int(n)) for n in RNG.integers(0, 300000, size=70)]
    _, digests, _, _ = run_device(ctx, msgs)
    for m, d in zip(msgs, digests):
        assert d == hashlib.md5(m).digest() == oracle.md5(m), len(m)


# ---------------------------------------------------------------- LZ4 frames
def test_empty_chunk_frame_is_byte_identical_to_liblz4(ctx, golden):
    empty = [c for c in golden["lz4_frames"]["cases"] if c["name"] == "empty"][0]
    frames, digests, lens, _ = run_device(ctx, [b"", b"x", b""])
    assert frames[0].hex() == frames[2].hex() == empty["frame_hex"] and lens[0] == 11
    assert digests[0].hex() == empty["md5"]
    check_frame(frames[1], b"x")


def test_golden_inputs_roundtrip(ctx, golden):
    cases = golden["lz4_frames"]["cases"]
    datas = [bytes.fromhex(c["input_hex"]) for c in cases]
    frames, digests, _, _ = run_device(ctx, datas)
    for c, d, f, dg in zip(cases, datas, frames, digests):
        check_frame(f, d)
        assert dg.hex() == c["md5"], c["name"]
        # our frame must decode to what the reference's own frame decodes to
        assert oracle.lz4f_decode(bytes.fromhex(c["frame_hex"]), len(d)) == oracle.lz4f_decode(f, len(d))


@pytest.mark.parametrize("kind", ["random", "zeros", "period7", "text", "half"])
def test_edge_lengths_roundtrip(ctx, kind):
    datas = [kinds(n)[kind] for n in EDGE_LENS]
    frames, digests, lens, _ = run_device(ctx, datas)
    for d, f, dg, ln in zip(datas, frames, digests, lens):
        assert ln == len(f)
        info = check_frame(f, d)
        assert dg == hashlib.md5(d).digest()
        if kind == "random" and len(d) >= 64:
            assert info["raw_blocks"] == info["blocks"] and len(f) == native.frame_bound(len(d))
        if kind == "zeros" and len(d) >= 4096:
            tiny_tail = 1 if 0 < len(d) % 65536 < 13 else 0  # a sub-13-byte last block cannot shrink: stored raw, like liblz4
            assert info["raw_blocks"] == tiny_tail and len(f) < len(d) // 50


def test_incompressible_frame_equals_reference_payload(ctx):
    """For all-raw frames the bytes after the 15-byte header equal the reference's frame byte for byte
    (only FLG's B.Indep bit and the header checksum differ)."""
    d = synth.random_chunk(3, 8 << 20)
    (f,), (dg,), _, _ = run_device(ctx, [d])
    r = ref.lz4f_compress(d)
    assert len(f) == len(r) == 8389139
    assert f[15:] == r[15:] and f[:4] == r[:4] and f[5:14] == r[5:14]
    assert f[4] == 0x68 and r[4] == 0x48
    assert f == oracle.lz4f_compress_indep(d)
    assert dg == hashlib.md5(d).digest()


def test_mixed_compressibility_moves_blocks_correctly(ctx):
    """Compressed blocks followed by stored blocks (and vice versa) exercise the slide-left / chain logic."""
    z, r, t = bytes(65536), RNG.bytes(65536), (b"abcdefghij" * 6554)[:65536]
    layouts = [z + r + z + r + r + t + r[:100], r + r + z + z + t + r, t * 5 + r[:7], r[:65535] + z + r[:1], z * 3 + r * 3 + z[:5]]
    frames, digests, _, _ = run_device(ctx, layouts)
    for d, f, dg in zip(layouts, frames, digests):
        check_frame(f, d)
        assert dg == hashlib.md5(d).digest()


def test_long_matches_and_long_literal_runs(ctx):
    a = RNG.bytes(1000)
    datas = [a + bytes(60000) + a, RNG.bytes(300) + b"Q" * 65000, (RNG.bytes(70) * 1000)[:65536], RNG.bytes(20000) + bytes(45536)]
    frames, _, _, _ = run_device(ctx, datas)
    for d, f in zip(datas, frames):
        check_frame(f, d)


def _twin_opts():
    import sys
    from pathlib import Path

    sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
    from tools import tile_model

    k = native.kernel_config()
    return tile_model, tile_model.kernel_opts(k["lz4_entries"], k["seg_slots"], k["max_step_log"])


def test_frames_equal_sequential_twin(ctx):
    """The warp-parallel parse is specified by a sequential program (tools/lz4_tile_model.c): same table rule, same tile
    parse, same emission.  Frames must be byte-identical -- this pins every lane-level shortcut of the kernel (group-wise
    table lookups with atomic-max updates, in-group hash compares, fused forward/backward compare, per-segment parsers, carried literals, batched emission, stride doubling) to plain sequential semantics."""
    tm, o = _twin_opts()
    a = RNG.bytes(1000)
    datas = [kinds(n)[k] for n in (13, 300, 4096, 65536, 65537, 200000) for k in ("zeros", "period7", "text", "half", "random")]
    datas += [synth.silesia_like_chunk(40 + i, (1 << 20) + 777 * i) for i in range(6)]
    datas += [a + bytes(60000) + a, RNG.bytes(300) + b"Q" * 65000, (RNG.bytes(70) * 1000)[:65536], RNG.bytes(40000) + synth.silesia_like_chunk(3, 90000)]
    frames, _, _, _ = run_device(ctx, datas)
    for i, (d, f) in enumerate(zip(datas, frames)):
        want = tm.frame(d, o)
        assert f == want, f"chunk {i} (len {len(d)}): GPU frame {len(f)} B != twin {len(want)} B"


def test_ratio_parity_on_silesia_like(ctx):
    datas = [synth.silesia_like_chunk(i, 16 << 20) for i in range(16)]
    frames, digests, _, _ = run_device(ctx, datas)
    gpu = sum(map(len, frames))
    refsz = sum(len(ref.lz4f_compress(d)) for d in datas)
    indep = sum(len(oracle.lz4f_compress_indep(d)) for d in datas)
    total = sum(map(len, datas))
    print(f"ratio gpu {total / gpu:.3f} reference(linked) {total / refsz:.3f} oracle(indep) {total / indep:.3f}")
    for d, f, dg in zip(datas, frames, digests):
        check_frame(f, d)
        assert dg == hashlib.md5(d).digest()
    assert (total / gpu) >= 0.95 * (total / refsz)


def test_batch_of_8mib_chunks(ctx):
    """BASELINE config 2 shape (smaller batch): uniform random 8 MiB chunks, one launch."""
    n = 48
    datas = [synth.random_chunk(i, 8 << 20) for i in range(n)]
    frames, digests, lens, ms = run_device(ctx, datas)
    assert all(l == 8389139 for l in lens)
    for i in (0, 17, n - 1):
        check_frame(frames[i], datas[i])
    for d, dg in zip(datas, digests):
        assert dg == hashlib.md5(d).digest()
    # checksum-of-checksums: size independent summary equals the CPU side's
    assert hashlib.md5(b"".join(digests)).digest() == hashlib.md5(b"".join(hashlib.md5(d).digest() for d in datas)).digest()


def test_multipart_sized_chunks(ctx):
    """64 MiB is the reference's multipart part size (skyplane/api/config.py:115-118): 1024 block rows per chunk,
    frame offsets beyond 2^26, ragged companions in the same launch."""
    big = synth.silesia_like_chunk(80, 16 << 20) * 4  # 64 MiB, compressible
    odd = synth.random_chunk(81, (33 << 20) + 12345)  # 33 MiB + change, incompressible
    datas = [big, odd, b"tail" * 1000]
    frames, digests, lens, _ = run_device(ctx, datas)
    for d, f, dg in zip(datas, frames, digests):
        info = check_frame(f, d)
        assert dg == hashlib.md5(d).digest()
    assert len(frames[1]) == native.frame_bound(len(odd)) and len(frames[0]) < len(big) * 0.6


@pytest.mark.timeout(120, method="thread")
def test_compressor_slower_than_digest_with_many_rows(ctx):
    """Many compressible multi-row chunks: the MD5 lanes finish long before the LZ4 warps, so the tail rows are
    released against a 'digest finished' progress word (regression: that comparison once wrapped and hung)."""
    base = [synth.silesia_like_chunk(70 + i, 12 * 65536 + 4321 * i) for i in range(6)]
    datas = [base[i % 6] for i in range(420)]
    frames, digests, lens, _ = run_device(ctx, datas)
    want = [hashlib.md5(d).digest() for d in base]
    assert digests == [want[i % 6] for i in range(420)]
    for i in (0, 1, 2, 3, 4, 5, 417, 419):
        check_frame(frames[i], datas[i])
    assert all(frames[i] == frames[i % 6] for i in range(420))  # same input -> same frame, whatever warp did it


def test_run_to_run_determinism(ctx):
    datas = [synth.silesia_like_chunk(9, 3 << 20), kinds(200000)["half"]]
    a = run_device(ctx, datas)[0]
    b = run_device(ctx, datas)[0]
    assert a == b


def test_stage_flags(ctx):
    datas = [synth.silesia_like_chunk(2, 1 << 20), b"abc"]
    frames, digests, lens, _ = run_device(ctx, datas, flags=native.F_LZ4)
    for d, f in zip(datas, frames):
        check_frame(f, d)
    assert all(dg == bytes(16) for dg in digests)  # MD5 stage not run
    _, digests, lens, _ = run_device(ctx, datas, flags=native.F_MD5 | native.F_MD5_EXCLUSIVE)
    assert [dg for dg in digests] == [hashlib.md5(d).digest() for d in datas] and all(l == 0 for l in lens)
    frames, digests, _, _ = run_device(ctx, datas, flags=native.F_LZ4 | native.F_MD5 | native.F_NO_PACING)
    for d, f, dg in zip(datas, frames, digests):
        check_frame(f, d)
        assert dg == hashlib.md5(d).digest()
    frames, digests, _, _ = run_device(ctx, datas, flags=native.F_LZ4 | native.F_MD5 | native.F_MD5_EXCLUSIVE)
    for d, f, dg in zip(datas, frames, digests):
        check_frame(f, d)
        assert dg == hashlib.md5(d).digest()


# ---------------------------------------------------------------- ABI error behaviour
def test_abi_argument_errors(ctx):
    d = ctx.device_alloc(4096)
    misaligned = (([8], [10], [0], [64]), native.SKY_E_INVALID, "src_off[0] or dst_off[0] is not a multiple of 16")
    too_small = (([0], [100], [0], [100]), native.SKY_E_CAPACITY, "dst_cap[0] < sky_frame_bound(src_len[0])")
    try:
        # invalid, capacity, invalid again on one ctx: each error's detail names its own cause, never an earlier one's
        for (src_off, src_len, dst_off, dst_cap), code, cause in (misaligned, too_small, misaligned):
            with pytest.raises(native.SkyChunkError) as e:
                ctx.process_device(d, src_off, src_len, d + 1024, dst_off, dst_cap)
            assert e.value.code == code
            assert cause in str(e.value)
            assert all(other not in str(e.value) for _, _, other in (misaligned, too_small) if other != cause)
        small = native.Context(0, 1 << 20, 2, 0)
        with pytest.raises(native.SkyChunkError) as e:
            small.process_device(d, [0, 16, 32], [1, 1, 1], d + 1024, [0, 32, 64], [32, 32, 32])
        assert e.value.code == native.SKY_E_CAPACITY and "n = 3 > max_chunks = 2" in str(e.value)
        small.close()
        with pytest.raises(native.SkyChunkError) as e:  # no ctx to hold the detail: it is the calling thread's
            native.Context(0, 1 << 20, 0, 0)
        assert e.value.code == native.SKY_E_INVALID and "max_chunks == 0" in str(e.value)
    finally:
        ctx.device_free(d)


# ---------------------------------------------------------------- host-buffer path (sky_submit / sky_wait)
def test_host_path_pipelined_slots():
    stage = ChunkStage(0, max_batch_bytes=64 << 20, max_chunks=64, n_slots=2)
    try:
        batch_a = [synth.silesia_like_chunk(20 + i, 2 << 20) for i in range(6)] + [b"", b"tiny"]
        batch_b = [synth.random_chunk(30 + i, (1 << 20) + i) for i in range(5)]
        sa, sb = stage.begin(), stage.begin()
        for c in batch_a:
            stage.add_bytes(sa, c)
        for c in batch_b:
            stage.add_bytes(sb, c)
        stage.launch(sa)
        stage.launch(sb)
        with pytest.raises(native.SkyChunkError):
            stage.begin()  # both slots in flight
        rb = stage.collect(sb)  # out of order
        ra = stage.collect(sa)
        for data, res in ((batch_a, ra), (batch_b, rb)):
            for d, r in zip(data, res):
                check_frame(bytes(r.frame), d)
                assert r.md5 == hashlib.md5(d).digest() and r.raw_len == len(d) and r.comp_len == len(r.frame)
        out = stage.process([b"hello world" * 1000, synth.random_chunk(1, 100000)])
        assert [r.md5 for r in out] == [hashlib.md5(b"hello world" * 1000).digest(), hashlib.md5(synth.random_chunk(1, 100000)).digest()]
        assert stage.ctx.launches == 3
    finally:
        stage.close()
