"""SKY_F_LINKED on the GPU: linked-block frames byte-identical to the sequential twin (tools/tile_model.frame_linked with
the build's sky_kernel_config), decodable by liblz4, pyarrow, the oracle and sky_decode, with the default mode's digests."""
import hashlib
import os
import socket
import sys
import threading
from pathlib import Path

import numpy as np
import pytest

import oracle
import oracle.reflib as ref
from gpu_util import run_device
from skyplane_b200 import native, synth, wire
from skyplane_b200.chunk import Chunk
from skyplane_b200.stage import ChunkStage
from test_gpu_decode_edges import encode_guarded
from test_linked_model import decode_all, offsets_and_end_rules

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from tools import tile_model as tm  # noqa: E402

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600, method="thread")]
LZ4_LINKED = native.F_LZ4 | native.F_MD5 | native.F_LINKED


@pytest.fixture(scope="module")
def ctx():
    c = native.Context(0, 1 << 30, 4096, 1)
    yield c
    c.close()


def twin(d: bytes) -> bytes:
    k = native.kernel_config()
    return tm.frame_linked(d, tm.kernel_opts(k["linked_entries"], k["seg_slots"], k["max_step_log"]), k["linked_window"], k["linked_seed_log"])


def ragged(seed=0):
    rng = np.random.default_rng(seed)
    lens = [0, 1, 12, 13, 4096, 65535, 65536, 65537, 2 * 65536 - 1, 2 * 65536 + 1, (1 << 20) + 3, 3 << 20]
    lens += [int(n) for n in rng.integers(0, 600_000, size=20)]
    out = []
    for i, n in enumerate(lens):
        k = i % 5
        out.append([rng.bytes(n), bytes(n), (b"abcdefg" * (n // 7 + 1))[:n],
                    (b"it was the best of times, it was the worst of times; " * (n // 50 + 1))[:n], synth.silesia_like_chunk(i, n)][k])
    return out


def test_config_reports_linked_mode():
    k = native.kernel_config()
    assert k["linked_window"] > 0 and k["linked_window"] % 1024 == 0 and k["linked_entries"] >= 128


def test_frames_equal_twin_device_path(ctx):
    datas = ragged(1)
    frames, digests, _, _ = run_device(ctx, datas, flags=LZ4_LINKED)
    _, dflt_digests, _, _ = run_device(ctx, datas)
    for d, f, g, g0 in zip(datas, frames, digests, dflt_digests):
        assert g == g0 == hashlib.md5(d).digest()
        assert f == twin(d), len(d)
        decode_all(f, d)
        offsets_and_end_rules(f, d)
        assert f[4] == (0x60 if not d else 0x68 if len(d) <= 65536 else 0x48)


def test_frames_equal_twin_host_path_and_sky_decode(ctx):
    datas = ragged(2)
    bufs = [native.PinnedBuffer(max(1, len(d))) for d in datas]
    outs = [native.PinnedBuffer(native.frame_bound(len(d))) for d in datas]
    try:
        for b, d in zip(bufs, datas):
            b.view[:len(d)] = d
        t = ctx.submit([b.addr for b in bufs], [len(d) for d in datas], [o.addr for o in outs],
                       [native.frame_bound(len(d)) for d in datas], LZ4_LINKED)
        lens, digests, _ = ctx.wait(t)
        frames = [bytes(o.view[:n]) for o, n in zip(outs, lens)]
        assert [f == twin(d) for d, f in zip(datas, frames)] == [True] * len(datas)
        assert [g == hashlib.md5(d).digest() for d, g in zip(datas, digests)] == [True] * len(datas)
        dst = [native.PinnedBuffer(max(1, len(d))) for d in datas]
        src = [native.PinnedBuffer(max(1, len(f))) for f in frames]
        for s, f in zip(src, frames):
            s.view[:len(f)] = f
        st, dg, _ = ctx.decode([s.addr for s in src], [len(f) for f in frames], [b.addr for b in dst], [len(d) for d in datas])
        assert st == [0] * len(datas) and dg == digests
        assert [bytes(b.view[:len(d)]) == d for b, d in zip(dst, datas)] == [True] * len(datas)
    finally:
        for b in bufs + outs:
            b.close()


def test_incompressible_frames_equal_liblz4(ctx):
    rng = np.random.default_rng(3)
    datas = [rng.bytes(n) for n in (65537, 3 * 65536 + 5, 1 << 20)]
    frames = run_device(ctx, datas, flags=LZ4_LINKED)[0]
    assert frames == [ref.lz4f_compress(d) for d in datas]


def test_e2ee_box_holds_the_linked_frame():
    nacl = pytest.importorskip("nacl.secret")
    key = bytes(range(32))
    st = ChunkStage(0, max_batch_bytes=32 << 20, max_chunks=16, n_slots=1)
    try:
        st.set_e2ee_key(key)
        datas = [synth.silesia_like_chunk(5, 3 << 20), b"", b"q" * 13, synth.random_chunk(2, 200000)]
        nonces = os.urandom(24 * len(datas))
        res = st.process(datas, encrypt=True, nonces=nonces, linked=True)
        box = nacl.SecretBox(key)
        for i, (d, r) in enumerate(zip(datas, res)):
            fr = box.decrypt(bytes(r.frame))
            assert bytes(r.frame[:24]) == nonces[24 * i:24 * i + 24] and fr == twin(d)
        out = st.decode([bytes(r.frame) for r in res], [len(d) for d in datas], encrypted=True)
        assert [(data, s) for data, _, s in out] == [(d, 0) for d in datas]
    finally:
        st.close()


def test_guard_bands_and_determinism(ctx):
    datas = ragged(4)
    f1, g1 = encode_guarded(ctx, datas, flags=LZ4_LINKED)
    f2, g2 = encode_guarded(ctx, datas, flags=LZ4_LINKED)
    assert f1 == f2 and g1 == g2
    assert [f == twin(d) for d, f in zip(datas, f1)] == [True] * len(datas)


def test_large_chunk_count():
    import torch

    sm = torch.cuda.get_device_properties(0).multi_processor_count
    n = 32 * (8 * sm + 2) + 7
    rng = np.random.default_rng(61)
    lens = [0 if rng.random() < 0.1 else int(rng.integers(1, 301)) for _ in range(n - 3)]
    lens[n // 3:n // 3] = [65535, 65537, 1 << 20]
    pool = synth.silesia_like_chunk(62, sum(lens))
    starts = np.cumsum([0] + lens)
    datas = [pool[a:a + k] for a, k in zip(starts, lens)]
    c = native.Context(0, 1 << 28, n, 0)
    try:
        frames, digests = encode_guarded(c, datas, gap=64, flags=LZ4_LINKED)
        assert [g == hashlib.md5(d).digest() for d, g in zip(datas, digests)] == [True] * n
        assert [f == twin(d) for d, f in zip(datas, frames)] == [True] * n
    finally:
        c.close()


def test_ratio_not_below_default(ctx):
    datas = [synth.silesia_like_chunk(100 + i, 16 << 20) for i in range(16)]
    linked = run_device(ctx, datas, flags=LZ4_LINKED)[2]
    dflt = run_device(ctx, datas)[2]
    assert sum(linked) <= sum(dflt)


def test_sender_linked_to_receiver_stage_over_a_socket():
    """The receiver needs nothing new: linked payloads sent from the pinned slot decode on the receiver's stage."""
    datas = [synth.silesia_like_chunk(80 + i, (2 << 20) + 999 * i) for i in range(3)] + [synth.random_chunk(3, 1 << 20), b"", b"z" * 13]
    chunks = [Chunk("src", "dst", "%032x" % (0xBEE000 + i), len(d), partition_id="0") for i, d in enumerate(datas)]
    send_stage = ChunkStage(0, max_batch_bytes=32 << 20, max_chunks=16, n_slots=1)
    recv_stage = ChunkStage(0, max_batch_bytes=32 << 20, max_chunks=16, n_slots=1)
    a, b = socket.socketpair()
    got = []

    def receiver():
        slot = recv_stage._free[-1]
        off = 0
        for _ in chunks:
            h, n = wire.recv_chunk(b, slot.out.view[off:])
            got.append((h, off, n))
            off += native.round16(n)

    t = threading.Thread(target=receiver)
    t.start()
    try:
        slot = send_stage.begin()
        for d in datas:
            send_stage.add_bytes(slot, d)
        send_stage.launch(slot, linked=True)
        results = send_stage.collect(slot)
        wire.send_results(a, chunks, results)
        t.join(60)
        rslot = recv_stage._free[-1]
        frames = [bytes(rslot.out.view[off: off + n]) for _, off, n in got]
        assert [f == twin(d) for f, d in zip(frames, datas)] == [True] * len(datas)
        out = recv_stage.decode(frames, [h.raw_data_len for h, _, _ in got])
        assert [(data, dg, st) for data, dg, st in out] == [(d, hashlib.md5(d).digest(), 0) for d in datas]
    finally:
        a.close()
        b.close()
        send_stage.close()
        recv_stage.close()


DRIVER = r"""
import functools, json, sys
from pathlib import Path
from skyplane_b200.harness import run_stream
from skyplane_b200.operators import GatewayCompressHash
base = Path(sys.argv[1])
files = sorted((base / "pool").glob("*.bin"), key=lambda p: int(p.stem))
op = functools.partial(GatewayCompressHash, block_linked=True)
res = run_stream(base / "chunks", files, [p.stat().st_size for p in files], 12, n_workers=2, max_batch_chunks=4,
                 max_batch_bytes=32 << 20, keep_frames=True, operator_cls=op)
print("RESULT " + json.dumps(res))
"""


def test_operator_sends_linked_frames_to_the_receiver(tmp_path):
    """GatewayCompressHash(block_linked=True) in forked workers; the receiver's stage decodes what it wrote."""
    import json
    import subprocess

    (tmp_path / "pool").mkdir()
    pool = [synth.silesia_like_chunk(90, 3 << 20), synth.random_chunk(1, 1 << 20), b"", b"x" * 13, synth.silesia_like_chunk(91, 65536)]
    for k, d in enumerate(pool):
        (tmp_path / "pool" / f"{k}.bin").write_bytes(d)
    root = Path(__file__).resolve().parent.parent
    r = subprocess.run([sys.executable, "-c", DRIVER, str(tmp_path)], capture_output=True, text=True,
                       env=dict(os.environ, PYTHONPATH=str(root)), timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    res = json.loads([l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1][len("RESULT "):])
    assert len(res["records"]) == 12
    frames, datas = [], []
    for rec in res["records"]:
        d = pool[rec["pool_index"]]
        f = Path(rec["frame_path"]).read_bytes()
        assert rec["md5"] == hashlib.md5(d).hexdigest() and f == twin(d)
        frames.append(f)
        datas.append(d)
    st = ChunkStage(0, max_batch_bytes=64 << 20, max_chunks=16, n_slots=1)
    try:
        out = st.decode(frames, [len(d) for d in datas])
        assert [(x, s) for x, _, s in out] == [(d, 0) for d in datas]
    finally:
        st.close()


def test_operator_built_from_program_json(tmp_path):
    import multiprocessing as mp

    from skyplane_b200.chunk_store import ChunkStore
    from skyplane_b200.program import build_operator_graph

    program = [{"partitions": ["0"], "value": [{"op_type": "compress_hash", "handle": "a", "num_gpus": 1, "block_linked": True,
                                                "max_batch_chunks": 4, "max_batch_bytes": 16 << 20, "children": []}]}]
    g = build_operator_graph(program, ChunkStore(tmp_path), "test:r", mp.Event(), mp.Queue())
    op = g.operators["compress_hash_a"]
    assert op.block_linked
    stage = op._get_stage()
    try:
        datas = [synth.silesia_like_chunk(95, (1 << 20) + 7), b"", b"w" * 70000]
        res = stage.process(datas, linked=op.block_linked)
        assert [bytes(r.frame) for r in res] == [twin(d) for d in datas]
    finally:
        op.worker_exit(0)
