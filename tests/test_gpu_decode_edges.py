"""The receiver-side GPU decoder (csrc/lz4dec.cuh through sky_decode_device / sky_decode_flags) on the hand-built corpus
of tests/lz4_craft.py, on every truncation a still-arriving payload can show, inside guard bands, and at chunk counts
past the point where the digest loops wrap.  Expected statuses and bytes come from the corpus labels that
tests/test_decode_conformance.py settles against the oracle and liblz4."""
import hashlib
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import lz4_craft as craft
import oracle
import oracle.reflib as ref
from gpu_util import run_device
from skyplane_b200 import native, synth
from skyplane_b200.stage import ChunkStage

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600, method="thread")]
ROOT = Path(__file__).resolve().parent.parent
GAP, SLACK = 4096, 65536  # untouched bytes between regions and after the last one
_PATTERN = ((np.arange(256) * 131 + 7) & 0xFF).astype(np.uint8)


@pytest.fixture(scope="module")
def ctx():
    c = native.Context(0, 1 << 30, 4096, 0)
    yield c
    c.close()


def pattern(n):
    """Position-dependent fill, (i * 131 + 7) & 0xFF (period 256)."""
    return np.tile(_PATTERN, n // 256 + 1)[:n].copy()


def layout(sizes, gap=GAP):
    """16-byte aligned offsets with `gap` pattern bytes after each region -> (offsets, slab size)."""
    offs, p = [], 0
    for s in sizes:
        offs.append(p)
        p += native.round16(s) + gap
    return offs, p + SLACK


def slab(blobs, offs, total):
    buf = pattern(total)
    for b, o in zip(blobs, offs):
        buf[o:o + len(b)] = np.frombuffer(b, np.uint8)
    return buf


def assert_outside_untouched(after, before, offs, sizes, what):
    mask = np.ones(len(after), bool)
    for o, s in zip(offs, sizes):
        mask[o:o + native.round16(s)] = False
    changed = np.flatnonzero((after != before) & mask)
    assert changed.size == 0, f"{what}: {changed.size} bytes changed outside the regions, first at {changed[0]}"


def decode_guarded(ctx, frames, raw_lens, gap=GAP):
    """sky_decode_device with every frame and output region surrounded by pattern bytes.  The frame slab must come back
    unchanged and nothing outside [out_off, out_off + round16(raw_len)) may change.  -> (outputs, digests, statuses)"""
    f_off, f_total = layout([len(f) for f in frames], gap)
    o_off, o_total = layout(raw_lens, gap)
    fs, os_ = slab(frames, f_off, f_total), pattern(o_total)
    d_f, d_o = ctx.device_alloc(f_total), ctx.device_alloc(o_total)
    try:
        ctx.h2d(d_f, fs)
        ctx.h2d(d_o, os_)
        st, dg, _ = ctx.decode_device(d_f, f_off, [len(f) for f in frames], d_o, o_off, list(raw_lens))
        f_after = np.frombuffer(ctx.d2h(d_f, f_total), np.uint8)
        o_after = np.frombuffer(ctx.d2h(d_o, o_total), np.uint8)
    finally:
        ctx.device_free(d_f)
        ctx.device_free(d_o)
    assert np.array_equal(f_after, fs), "the decoder wrote into the frame slab"
    assert_outside_untouched(o_after, os_, o_off, raw_lens, "decode")
    return [o_after[o:o + r].tobytes() for o, r in zip(o_off, raw_lens)], dg, st


def encode_guarded(ctx, datas, extra_cap=0, gap=GAP, flags=0):
    """sky_process_device with guard bands around every input and frame region; dst_cap = frame_bound + extra_cap.
    -> (frames, digests)"""
    lens = [len(d) for d in datas]
    caps = [native.frame_bound(n) + extra_cap for n in lens]
    s_off, s_total = layout(lens, gap)
    d_off, d_total = layout(caps, gap)
    ins, outs = slab(datas, s_off, s_total), pattern(d_total)
    d_in, d_out = ctx.device_alloc(s_total), ctx.device_alloc(d_total)
    try:
        ctx.h2d(d_in, ins)
        ctx.h2d(d_out, outs)
        out_lens, digests, _ = ctx.process_device(d_in, s_off, lens, d_out, d_off, caps, flags)
        i_after = np.frombuffer(ctx.d2h(d_in, s_total), np.uint8)
        o_after = np.frombuffer(ctx.d2h(d_out, d_total), np.uint8)
    finally:
        ctx.device_free(d_in)
        ctx.device_free(d_out)
    assert np.array_equal(i_after, ins), "the compressor wrote into the input slab"
    assert_outside_untouched(o_after, outs, d_off, caps, "encode")
    return [o_after[o:o + n].tobytes() for o, n in zip(d_off, out_lens)], digests


def _md5(b):
    return hashlib.md5(b).digest()


# ---------------------------------------------------------------- the corpus
def test_corpus_in_one_batch(ctx):
    """Valid frames placed between malformed ones: every status is the exact one for its class, the valid neighbours of
    failing frames decode intact (their MD5 lanes wait on the failed chunks' blocks), and the batch terminates."""
    valid = craft.valid_cases()
    bad = craft.rejected_cases() + craft.layout_cases()
    batch = []
    for i in range(max(len(valid), len(bad))):
        batch += [bad[i % len(bad)], valid[i % len(valid)]]
    outs, digests, status = decode_guarded(ctx, [c.frame for c in batch], [c.raw_len for c in batch])
    wrong = [(c.name, s, c.gpu) for c, s in zip(batch, status) if s != c.gpu]
    assert not wrong, f"(case, status, expected): {wrong}"
    for c, o, dg in zip(batch, outs, digests):
        if c.gpu == native.D_OK:
            assert o == c.want, c.name
            assert dg == _md5(c.want), c.name


def test_end_of_block_violations_are_corrupt(ctx):
    """The format's end-of-block rules, including the two short-block cases liblz4 lets through."""
    cases = craft.end_rule_cases()
    ok = [c for c in craft.valid_cases() if c.name.startswith(("final5_", "mflimit_"))]  # exactly at the limits
    _, _, status = decode_guarded(ctx, [c.frame for c in cases + ok], [c.raw_len for c in cases + ok])
    assert {c.name: s for c, s in zip(cases + ok, status)} == {c.name: c.gpu for c in cases + ok}
    assert all(c.gpu == native.D_CORRUPT for c in cases) and all(c.gpu == native.D_OK for c in ok)


def test_decode_writes_stay_inside_regions(ctx):
    """Real frames (ours, liblz4's linked ones) and damaged copies of them between guard bands."""
    rng = np.random.default_rng(21)
    datas = [synth.silesia_like_chunk(30 + i, (1 << 20) + 4099 * i) for i in range(3)] + [rng.bytes(70001), bytes(131075), b"x" * 13]
    frames = run_device(ctx, datas)[0] + [ref.lz4f_compress(d) for d in datas]
    raws = [len(d) for d in datas] * 2
    damaged = []
    for i, f in enumerate(frames):
        g = bytearray(f)
        for k in range(20 + i, len(g) - 8, 257 + 31 * i):
            g[k] ^= 0xA5
        damaged.append(bytes(g))
    outs, digests, status = decode_guarded(ctx, frames + damaged, raws + raws)
    for d, o, dg, st in zip(datas * 2, outs, digests, status):
        assert st == 0 and o == d and dg == _md5(d)
    for f, r, o, st in zip(damaged, raws, outs[len(frames):], status[len(frames):]):
        try:
            want = oracle.lz4f_decode(f, r)
        except oracle.OracleError:
            want = None
        assert st != 0 if want is None else (st != 0 or o == want)


# ---------------------------------------------------------------- truncation
def test_every_proper_prefix_is_truncated(ctx):
    """GatewayDecompressVerify re-queues a still-growing payload only while the status is D_TRUNCATED."""
    for name, fr, raw, cuts in craft.prefix_sets():
        _, _, status = decode_guarded(ctx, [fr[:k] for k in cuts] + [fr], [raw] * (len(cuts) + 1), gap=64)
        assert status[-1] == native.D_OK, name
        wrong = [(k, s) for k, s in zip(cuts, status) if s != native.D_TRUNCATED]
        assert not wrong, f"{name}: (prefix length, status) {wrong[:20]}"


def test_every_proper_prefix_of_a_box_fails_authentication():
    data = b"abcdefgh" * 40 + np.random.default_rng(4).bytes(60)
    stage = ChunkStage(0, max_batch_bytes=16 << 20, max_chunks=1024, n_slots=1)
    try:
        stage.set_e2ee_key(bytes(range(32)))
        (r,) = stage.process([data], encrypt=True)
        box = bytes(r.frame)
        assert len(box) < 1000
        boxes = [box] + [box[:k] for k in range(1, len(box))] + [box]
        res = stage.decode(boxes, [len(data)] * len(boxes), encrypted=True)
        for o, dg, st in (res[0], res[-1]):
            assert st == native.D_OK and o == data and dg == _md5(data)
        wrong = [(k, st) for k, (o, dg, st) in enumerate(res[1:-1], 1) if st != native.D_AUTH or o is not None]
        assert not wrong, f"(prefix length, status) {wrong[:20]}"
    finally:
        stage.close()


# ---------------------------------------------------------------- the sender's side of the same contracts
@pytest.mark.parametrize("extra_cap", [0, 4096 + 5])
def test_encode_writes_stay_inside_regions(ctx, extra_cap):
    from test_gpu_parity import _twin_opts, kinds

    tm, o = _twin_opts()
    rng = np.random.default_rng(31)
    datas = [kinds(n, rng)[k] for n in (0, 1, 13, 100, 4096, 65535, 65537, 200000) for k in ("random", "zeros", "text", "half")]
    datas += [synth.silesia_like_chunk(60 + i, (1 << 20) + 333 * i) for i in range(2)]
    frames, digests = encode_guarded(ctx, datas, extra_cap)
    for d, f, dg in zip(datas, frames, digests):
        assert f == tm.frame(d, o), len(d)
        assert dg == _md5(d)


def test_gpu_frames_obey_end_of_block_rules(ctx):
    """liblz4 would not notice a short last block breaking the rules (it checks them against 64 KiB of room)."""
    from test_gpu_parity import EDGE_LENS, kinds

    rng = np.random.default_rng(41)
    datas = [kinds(n, rng)[k] for k in ("random", "zeros", "period7", "text", "half") for n in EDGE_LENS]
    datas += [synth.silesia_like_chunk(40 + i, (1 << 20) + 777 * i) for i in range(6)]
    frames = run_device(ctx, datas)[0]
    checked = 0
    for d, f in zip(datas, frames):
        pos = 0
        for _, stored, payload in craft.frame_blocks(f)[1]:
            n = min(craft.BLOCK, len(d) - pos)
            if not stored:
                craft.check_block_end_rules(payload, n)
                checked += 1
            pos += n
    assert checked > 100


# ---------------------------------------------------------------- batch sizes
def test_large_chunk_counts():
    """More digest groups than 4 x grid (fused kernel: the digest CTAs stop growing) and 4 x sm_count (decode kernel:
    the MD5 group loop wraps)."""
    import torch

    sm = torch.cuda.get_device_properties(0).multi_processor_count
    n = 32 * (8 * sm + 2) + 7
    rng = np.random.default_rng(51)
    lens = [0 if rng.random() < 0.1 else int(rng.integers(1, 301)) for _ in range(n - 3)]
    lens[n // 3:n // 3] = [65535, 65537, 1 << 20]  # rows > 1
    pool = synth.silesia_like_chunk(52, sum(lens))
    starts = np.cumsum([0] + lens)
    datas = [pool[a:a + k] for a, k in zip(starts, lens)]
    c = native.Context(0, 1 << 28, n, 0)
    try:
        frames, digests = encode_guarded(c, datas, gap=64)
        assert [dg == _md5(d) for d, dg in zip(datas, digests)] == [True] * n
        assert all(oracle.lz4f_decode(f, len(d)) == d for d, f in zip(datas, frames))
        outs, dg2, status = decode_guarded(c, frames, lens, gap=64)
        assert status == [0] * n
        assert outs == datas and dg2 == digests
        frames, digests = encode_guarded(c, [b""] * 33)
        assert frames == [frames[0]] * 33 and len(frames[0]) == 11 and digests == [_md5(b"")] * 33
        outs, dg2, status = decode_guarded(c, frames, [0] * 33)
        assert status == [0] * 33 and dg2 == digests
    finally:
        c.close()


MD5_WARPS_CHILD = r"""
import hashlib, sys
import numpy as np
root = sys.argv[1]
sys.path[:0] = [root, root + "/tests"]
from gpu_util import run_device
from skyplane_b200 import native, synth
from tools import tile_model

rng = np.random.default_rng(int(sys.argv[2]))
ctx = native.Context(0, 1 << 30, 256, 0)
datas = [synth.silesia_like_chunk(int(s), int(n)) if s % 2 else rng.bytes(int(n))
         for s, n in zip(range(200), rng.integers(0, 300_000, size=200))]
_, digests, _, _ = run_device(ctx, datas, flags=native.F_MD5)
assert [d == hashlib.md5(x).digest() for x, d in zip(datas, digests)] == [True] * 200, "F_MD5 digests"
_, digests, _, _ = run_device(ctx, datas)
assert [d == hashlib.md5(x).digest() for x, d in zip(datas, digests)] == [True] * 200, "LZ4 + MD5 digests"
k = native.kernel_config()
o = tile_model.kernel_opts(k["lz4_entries"], k["seg_slots"], k["max_step_log"])
big = [synth.silesia_like_chunk(70 + i, 2 << 20) for i in range(8)]
frames, digests, _, _ = run_device(ctx, big)
assert [f == tile_model.frame(d, o) for d, f in zip(big, frames)] == [True] * 8, "frames differ from the twin"
assert [g == hashlib.md5(d).digest() for d, g in zip(big, digests)] == [True] * 8
ctx.close()
print("MD5_WARPS_OK")
"""


@pytest.mark.parametrize("warps", [1, 2, 4])
def test_md5_warps_per_digest_cta(warps):
    """SKYCHUNK_MD5_WARPS is read once per process, so each layout runs in a child process."""
    env = dict(os.environ, SKYCHUNK_MD5_WARPS=str(warps), PYTHONPATH=str(ROOT))
    r = subprocess.run([sys.executable, "-c", MD5_WARPS_CHILD, str(ROOT), str(warps)], env=env, capture_output=True, text=True, timeout=500)
    assert r.returncode == 0 and "MD5_WARPS_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
