"""Gateway operator plugin surface + the B200 compress/hash operator.

``GatewayOperator`` keeps the reference's contract (skyplane/gateway/operators/gateway_operator.py:32-122):
same constructor arguments, ``start_workers`` forks ``n_processes`` workers running
``worker_loop(worker_id, *self.args)``, ``process(chunk_req, *args) -> bool`` where True forwards
the request to ``output_queue``, False re-queues it, and an exception stops the gateway through
``error_event`` / ``error_queue``.

``GatewayCompressHash`` is the new stage (integration choice (ii) of SURVEY.md section 8b: a new
op_type placed between ``read_object_store`` and ``send``).  Per chunk it
  * reads ``<chunk_dir>/<chunk_id>.chunk`` into pinned memory (gateway_operator.py:350-352),
  * runs the fused LZ4-frame + MD5 kernel on the worker's GPU (worker_id -> device),
  * writes the frame to ``<chunk_id>.chunk.lz4`` and sets ``chunk.md5_hash`` (chunk.py:21),
  * reports ``compressed_size_bytes`` / ``uncompressed_size_bytes`` in the ``complete`` status record so the
    daemon's ``/api/v1/profile/compression`` endpoint lights up (gateway_daemon_api.py:130-134).
Its ``worker_loop`` drains a *batch* of requests per launch (the reference's loop sleeps 0.1 s per chunk,
gateway_operator.py:102, which would cap a worker below 10 chunks/s) but keeps the same state logging
and error conventions.  CUDA is initialised lazily inside the worker process, never in ``__init__``
(workers are forked, gateway_operator.py:66-70).
"""
from __future__ import annotations

import os
import queue
import time
import traceback
from abc import ABC, abstractmethod
from multiprocessing import Event, Process, Queue
from typing import List, Optional

from skyplane_b200.chunk import ChunkRequest, ChunkState
from skyplane_b200.chunk_store import ChunkStore
from skyplane_b200.gateway_queue import GatewayQueue


class GatewayOperator(ABC):
    def __init__(
        self,
        handle: str,
        region: str,
        input_queue: GatewayQueue,
        output_queue: Optional[GatewayQueue],
        error_event,
        error_queue: Queue,
        chunk_store: ChunkStore,
        n_processes: Optional[int] = 1,
    ):
        self.handle = handle
        self.region = region
        self.input_queue = input_queue
        self.output_queue = output_queue
        self.chunk_store = chunk_store
        self.error_event = error_event
        self.error_queue = error_queue
        self.n_processes = n_processes
        self.args = ()  # extra positional args handed to worker_loop / process
        self.processes: List[Process] = []
        self.exit_flags = [Event() for _ in range(self.n_processes)]
        self.worker_id: Optional[int] = None  # process-local

    def start_workers(self):
        for i in range(self.n_processes):
            p = Process(target=self.worker_loop, args=(i,) + self.args)
            p.start()
            self.processes.append(p)

    def stop_workers(self):
        for flag in self.exit_flags:
            flag.set()
        for p in self.processes:
            p.join()
        self.processes = []

    def _running(self, worker_id: int) -> bool:
        return not self.exit_flags[worker_id].is_set() and not self.error_event.is_set()

    def _fail(self, worker_id: int, exc: BaseException):
        print(f"[{self.handle}:{worker_id}] Exception: {exc}")
        self.error_queue.put(traceback.format_exc())
        self.error_event.set()
        self.exit_flags[worker_id].set()

    def worker_loop(self, worker_id: int, *args):
        """One request at a time, as the reference does (gateway_operator.py:79-115)."""
        self.worker_id = worker_id
        while self._running(worker_id):
            try:
                try:
                    chunk_req = self.input_queue.get_nowait(self.handle)
                except queue.Empty:
                    time.sleep(0.001)
                    continue
                self.chunk_store.log_chunk_state(chunk_req, ChunkState.in_progress, operator_handle=self.handle, worker_id=worker_id)
                if self.process(chunk_req, *args):
                    self.chunk_store.log_chunk_state(chunk_req, ChunkState.complete, operator_handle=self.handle, worker_id=worker_id)
                    if self.output_queue is not None:
                        self.output_queue.put(chunk_req)
                else:
                    time.sleep(0.1)
                    self.input_queue.put(chunk_req)
            except Exception as e:
                self._fail(worker_id, e)
        self.worker_exit(worker_id)

    def worker_exit(self, worker_id: int):
        pass

    @abstractmethod
    def process(self, chunk_req: ChunkRequest, *args) -> bool:
        ...


class GatewayCompressHash(GatewayOperator):
    """B200 stage: LZ4 frame + MD5 per chunk, batched per kernel launch."""

    def __init__(
        self,
        handle: str,
        region: str,
        input_queue: GatewayQueue,
        output_queue: Optional[GatewayQueue],
        error_event,
        error_queue: Queue,
        chunk_store: ChunkStore,
        n_processes: Optional[int] = 1,
        use_compression: Optional[bool] = True,
        max_batch_chunks: int = 64,
        max_batch_bytes: int = 512 << 20,
        n_gpus: Optional[int] = None,
        keep_frames_on_disk: bool = True,
        read_threads: int = 12,
        ingest_read_local: bool = True,
        e2ee_key_bytes: Optional[bytes] = None,
        sink=None,
        n_slots: int = 4,
        block_linked: bool = False,
    ):
        """use_compression / e2ee_key_bytes: GatewaySender's arguments of the same name (gateway_operator.py:154-168):
        ``use_compression=False`` digests the chunk and lets it pass through uncompressed (``is_compressed=False``);
        ``e2ee_key_bytes`` seals every payload in a SecretBox on the GPU.
        sink: ``callable(worker_id) -> socket``, called once in each worker.  With a sink the worker sends every payload
        straight from the pinned staging slot (``wire.send_results``: WireProtocolHeader + payload, no intermediate bytes
        object, no frame file) -- the tail of ``GatewaySender.process`` (gateway_operator.py:367-402).
        block_linked: linked-block frames (``native.F_LINKED``), a few percent smaller on text; any LZ4 frame decoder, and
        so the receiver, reads them unchanged.  Raises when the worker creates its stage on a build without linked mode."""
        super().__init__(handle, region, input_queue, output_queue, error_event, error_queue, chunk_store, n_processes)
        self.use_compression = True if use_compression is None else bool(use_compression)
        self.block_linked = bool(block_linked)
        self.e2ee_key_bytes = e2ee_key_bytes
        self.sink = sink
        # batches in flight per worker: a batch of 8 MiB chunks spends >= 70 ms on the GPU whatever its size (one serial MD5
        # chain per chunk), so throughput = chunks in flight / 70 ms -- keep several batches going (one slot is being read
        # into, the others are on the GPU; measured 18.8 / 26.5 / 27.2 / 26.2 GB/s with 3 / 4 / 5 / 6 slots of 128 chunks)
        self.n_slots = max(2, n_slots)
        self._sock = None
        self.max_batch_chunks = max_batch_chunks
        self.max_batch_bytes = max_batch_bytes
        self.n_gpus = n_gpus
        self.keep_frames_on_disk = keep_frames_on_disk
        self.read_threads = read_threads
        self.ingest_read_local = ingest_read_local
        self._stage = None  # created lazily in the worker process (fork + CUDA)
        self._readers = None  # thread pool for chunk-file reads, also per process

    # -- per-process GPU state ---------------------------------------------------------------
    def _get_stage(self):
        if self._stage is None:
            from skyplane_b200 import native
            from skyplane_b200.stage import ChunkStage

            ngpu = self.n_gpus or native.device_count()
            if ngpu <= 0:
                raise native.SkyChunkError(native.SKY_E_NOGPU, "GatewayCompressHash needs a CUDA device; there is no CPU fallback")
            device = (self.worker_id or 0) % ngpu
            if ngpu > 1:
                from skyplane_b200.numa import bind_to_gpu

                bind_to_gpu(device)  # pinned staging buffers on the GPU's own socket
            if self.block_linked:
                native.require_linked()
            self._stage = ChunkStage(device, self.max_batch_bytes, self.max_batch_chunks, n_slots=self.n_slots)
            if self.e2ee_key_bytes is not None:
                self._stage.set_e2ee_key(self.e2ee_key_bytes)
        return self._stage

    def _grow_stage(self, n: int):
        """A chunk larger than the staging slots (e.g. a 64 MiB multipart part behind a small max_batch_bytes): rebuild the
        stage with room for it instead of stopping the gateway.  Only called while no batch is in flight."""
        if self._stage is not None:
            self._stage.close()
            self._stage = None
        self.max_batch_bytes = max(self.max_batch_bytes, (n + (1 << 20)) & ~((1 << 20) - 1))

    def worker_exit(self, worker_id: int):
        if self._sock is not None:
            try:
                self._sock.close()
            except OSError:
                pass
            self._sock = None
        if self._readers is not None:
            self._readers.shutdown(wait=True)
            self._readers = None
        if self._stage is not None:
            self._stage.close()
            self._stage = None

    # -- the plugin method ---------------------------------------------------------------------
    def process(self, chunk_req: ChunkRequest, *args) -> bool:
        return self.process_batch([chunk_req])[0]

    # -- batch plumbing -------------------------------------------------------------------------
    def _read_into(self, path, view, n: int, offset: Optional[int] = None) -> bool:
        """Read exactly n bytes into pinned memory.  offset None: `path` is a chunk file that must hold exactly n
        bytes (False if it is not complete yet); otherwise the byte range [offset, offset+n) of a source object."""
        try:
            with open(path, "rb", buffering=0) as f:
                if offset:
                    f.seek(offset)
                got = 0
                while got < n:
                    r = f.readinto(view[got:])
                    if not r:
                        return False
                    got += r
                return True if offset is not None else not f.read(1)
        except FileNotFoundError:
            return False

    def _source_of(self, chunk_req: ChunkRequest):
        """-> (path, offset or None, ready).  ``src_type == "read_local"`` (skyplane/chunk.py:54) ingests the byte range
        straight from the source file into the staging slot -- no tmpfs chunk file in between (SURVEY.md section 8f
        row 3 for the POSIX case); every other request reads ``<chunk_id>.chunk`` as GatewaySender does."""
        chunk = chunk_req.chunk
        n = chunk.chunk_length_bytes
        if self.ingest_read_local and chunk_req.src_type == "read_local":
            off = chunk.file_offset_bytes or 0
            try:
                return chunk.src_key, off, os.stat(chunk.src_key).st_size >= off + n
            except FileNotFoundError:
                return chunk.src_key, off, False
        path = self.chunk_store.get_chunk_file_path(chunk.chunk_id)
        try:
            return path, None, os.stat(path).st_size == n  # upstream writes the file before queueing (gateway_operator.py:567-570)
        except FileNotFoundError:
            return path, None, False

    def _stage_reads(self, reqs: List[ChunkRequest]):
        """Reserve room in a free staging slot for as many of `reqs` as fit and START reading them into pinned memory
        (thread pool; file -> pinned copies release the GIL).  Nothing here touches the GPU.
        -> (slot or None, jobs [(index, future)], not-ready indices, leftover indices)"""
        stage = self._get_stage()
        slot = stage.begin()
        not_ready, leftover, jobs = [], [], []
        for i, r in enumerate(reqs):
            chunk = r.chunk
            n = chunk.chunk_length_bytes
            if n > stage.max_batch_bytes:
                for _, fut in jobs:
                    fut.result()  # (reads into the slot we are about to give back must be over first)
                stage.release(slot)
                if len(stage._free) < len(stage._slots):  # batches in flight: come back when they have been collected
                    return None, [], [], list(range(len(reqs)))
                self._grow_stage(n)
                if n > self._get_stage().max_batch_bytes:
                    raise ValueError(f"chunk {chunk.chunk_id} ({n} B) exceeds what the stage can be grown to")
                return self._stage_reads(reqs)
            path, offset, ready = self._source_of(r)
            if not ready:
                not_ready.append(i)
            elif not stage.fits(slot, n):
                leftover.append(i)
            else:
                if self._readers is None:
                    from concurrent.futures import ThreadPoolExecutor

                    self._readers = ThreadPoolExecutor(max_workers=self.read_threads)
                jobs.append((i, self._readers.submit(self._read_into, path, slot.reserve(n), n, offset)))
        if jobs:
            return slot, jobs, not_ready, leftover
        stage.release(slot)
        if leftover:
            raise RuntimeError("staging slot cannot hold a single chunk")
        return None, [], not_ready, leftover

    def _launch_staged(self, slot, jobs) -> bool:
        """Wait for the reads of a staged batch and launch it.  False: a file changed under us -- the slot is given back and
        the whole batch must be retried later rather than hash partial data."""
        stage = self._get_stage()
        if not all([fut.result() for _, fut in jobs]):
            stage.release(slot)
            return False
        linked = {"linked": True} if self.block_linked else {}  # (only when asked for: stage look-alikes need not know it)
        stage.launch(slot, compress=self.use_compression, encrypt=self.e2ee_key_bytes is not None, **linked)
        return True

    def _launch(self, reqs: List[ChunkRequest]):
        """Stage as many of `reqs` as fit one slot, read them and launch them (synchronously).
        -> (slot or None, launched indices, not-ready indices, leftover indices)"""
        slot, jobs, not_ready, leftover = self._stage_reads(reqs)
        if slot is None:
            return None, [], not_ready, leftover
        idx = [i for i, _ in jobs]
        if not self._launch_staged(slot, jobs):
            return None, [], idx + not_ready, leftover
        return slot, idx, not_ready, leftover

    def _finish(self, slot, reqs: List[ChunkRequest]):
        """Collect a launched batch: sets md5_hash, hands the payloads on (socket sink, or payload files), attaches the
        size metadata.  The slot's pinned views stay valid until the slot is reused, i.e. until this returns."""
        results = self._get_stage().collect(slot)
        for r, res in zip(reqs, results):
            r.chunk.md5_hash = res.md5
            r._stage_meta = {"compressed_size_bytes": res.comp_len, "uncompressed_size_bytes": res.raw_len}
        if self.sink is not None:
            from skyplane_b200 import wire

            if self._sock is None:
                self._sock = self.sink(self.worker_id or 0)
            wire.send_results(self._sock, [r.chunk for r in reqs], results)
        elif self.keep_frames_on_disk:
            for r, res in zip(reqs, results):
                if res.is_compressed or res.is_encrypted:  # (a plain pass-through chunk is already on disk as <id>.chunk)
                    path = self.chunk_store.get_compressed_file_path(r.chunk.chunk_id)
                    tmp = path.with_name(path.name + ".part")
                    with open(tmp, "wb") as f:
                        f.write(res.frame)
                    os.replace(tmp, path)  # readers never see a half-written payload

    def process_batch(self, reqs: List[ChunkRequest]) -> List[bool]:
        """Compress + hash a batch synchronously. One bool per request (False = chunk file not ready yet, retry)."""
        ok = [True] * len(reqs)
        todo = list(range(len(reqs)))
        while todo:
            sub = [reqs[i] for i in todo]
            slot, launched, not_ready, leftover = self._launch(sub)
            for k in not_ready:
                ok[todo[k]] = False
            if slot is not None:
                self._finish(slot, [sub[k] for k in launched])
            todo = [todo[k] for k in leftover]
        return ok

    def _complete(self, worker_id: int, r: ChunkRequest):
        meta = r.__dict__.pop("_stage_meta", None)
        self.chunk_store.log_chunk_state(r, ChunkState.complete, operator_handle=self.handle, worker_id=worker_id, metadata=meta)
        if self.output_queue is not None:
            self.output_queue.put(r)

    def _complete_many(self, worker_id: int, reqs: List[ChunkRequest]):
        """`complete` records and the hand-over to the next operator for a whole batch: one queue element each."""
        metas = [r.__dict__.pop("_stage_meta", None) for r in reqs]
        self.chunk_store.log_chunk_states(reqs, ChunkState.complete, operator_handle=self.handle, worker_id=worker_id, metadata=metas)
        if self.output_queue is not None:
            self.output_queue.put_many(reqs)

    def worker_loop(self, worker_id: int, *args):
        """Batch-draining loop with the reference's logging / error conventions.  Three things overlap: the chunk files of
        batch k+1 are read into a free staging slot by the reader threads while batch k is on the GPU (several batches are)
        and while this thread waits for the oldest batch's payloads to come back (`_finish`)."""
        self.worker_id = worker_id
        inflight = []  # [(slot, reqs)] oldest first
        reading = None  # (slot, jobs, cand): a batch whose chunk files are being read into its slot
        backlog: List[ChunkRequest] = []  # dequeued but not yet staged (did not fit the slot)
        try:
            while self._running(worker_id):
                try:
                    progressed = False
                    if reading is not None and (not inflight or all(fut.done() for _, fut in reading[1])):
                        slot, jobs, cand = reading
                        reading = None
                        progressed = True
                        if self._launch_staged(slot, jobs):
                            inflight.append((slot, [cand[i] for i, _ in jobs]))
                        else:
                            for i, _ in jobs:
                                self.input_queue.put(cand[i])
                    if reading is None:
                        stage_free = self._stage is None or bool(self._stage._free)
                        if backlog and inflight and max(r.chunk.chunk_length_bytes for r in backlog) > self.max_batch_bytes:
                            stage_free = False  # an oversize chunk waits for the stage to drain, then the stage is rebuilt
                        if stage_free:
                            room = self.max_batch_chunks - len(backlog)
                            fresh = self.input_queue.get_batch_nowait(room, self.handle) if room > 0 else []
                            if fresh:
                                self.chunk_store.log_chunk_states(fresh, ChunkState.in_progress, operator_handle=self.handle, worker_id=worker_id)
                            cand = backlog + fresh
                            if cand:
                                slot, jobs, not_ready, leftover = self._stage_reads(cand)
                                if slot is not None:
                                    reading = (slot, jobs, cand)
                                    progressed = True
                                backlog = [cand[k] for k in leftover]
                                if not_ready:
                                    time.sleep(0.1 if slot is None and not inflight else 0)
                                    for k in not_ready:
                                        self.input_queue.put(cand[k])
                    if inflight and (reading is None or len(inflight) >= self.n_slots - 1):
                        slot, reqs = inflight.pop(0)  # (blocks until that batch's payloads are back; the readers keep going)
                        self._finish(slot, reqs)
                        self._complete_many(worker_id, reqs)
                    elif not progressed:
                        time.sleep(0.0002 if reading is not None else 0.0005)  # reads under way / nothing queued
                except Exception as e:
                    self._fail(worker_id, e)
            # drain what is already staged / on the GPU so no accepted chunk is lost on a clean stop
            if not self.error_event.is_set():
                if reading is not None:
                    slot, jobs, cand = reading
                    if self._launch_staged(slot, jobs):
                        inflight.append((slot, [cand[i] for i, _ in jobs]))
                for slot, reqs in inflight:
                    self._finish(slot, reqs)
                    self._complete_many(worker_id, reqs)
        finally:
            self.worker_exit(worker_id)


class ChecksumMismatchException(Exception):
    """Same name as skyplane/exceptions.py:44-48: the decoded chunk's MD5 differs from Chunk.md5_hash."""


class GatewayDecompressVerify(GatewayOperator):
    """Receiving side (SURVEY.md section 8f row 1): what gateway_receiver.py:191-233 does after the socket read.

    ``<chunk_id>.chunk.lz4`` (the wire payload) -> [SecretBox open on the GPU] -> LZ4 frame decode on the GPU ->
    ``<chunk_id>.chunk`` of exactly ``chunk_length_bytes`` bytes (the size check at gateway_receiver.py:213-218), and --
    closing the reference's "# todo check hash" (gateway_receiver.py:231) -- the digest of the decoded bytes is compared
    with ``chunk.md5_hash`` when the sender supplied one.  Requests are drained in batches (one decode launch per batch);
    a payload that is missing or still being written is re-queued like GatewayWaitReceiver does (gateway_operator.py:131-150);
    a complete but corrupt payload, a forged box or a digest mismatch raises, which stops the gateway through
    ``error_event`` like any other operator failure."""

    def __init__(self, *args, max_batch_chunks: int = 64, max_batch_bytes: int = 512 << 20, n_gpus: Optional[int] = None,
                 remove_frames: bool = True, e2ee_key_bytes: Optional[bytes] = None, stale_retries: int = 50, **kwargs):
        super().__init__(*args, **kwargs)
        self.max_batch_chunks = max_batch_chunks
        self.max_batch_bytes = max_batch_bytes
        self.n_gpus = n_gpus
        self.remove_frames = remove_frames
        self.e2ee_key_bytes = e2ee_key_bytes
        self.stale_retries = stale_retries  # re-queues of an unchanged, undecodable payload before it counts as corrupt
        self._stage = None
        self._seen = {}  # chunk_id -> (payload size at the last attempt, attempts at that size)

    def _get_stage(self):
        if self._stage is None:
            from skyplane_b200 import native
            from skyplane_b200.stage import ChunkStage

            ngpu = self.n_gpus or native.device_count()
            if ngpu <= 0:
                raise native.SkyChunkError(native.SKY_E_NOGPU, "GatewayDecompressVerify needs a CUDA device; there is no CPU fallback")
            self._stage = ChunkStage((self.worker_id or 0) % ngpu, self.max_batch_bytes, self.max_batch_chunks, n_slots=1)
            if self.e2ee_key_bytes is not None:
                self._stage.set_e2ee_key(self.e2ee_key_bytes)
        return self._stage

    def worker_exit(self, worker_id: int):
        if self._stage is not None:
            self._stage.close()
            self._stage = None

    def process(self, chunk_req: ChunkRequest, *args) -> bool:
        return self.process_batch([chunk_req])[0]

    def _still_arriving(self, chunk_id: str, size: int) -> bool:
        """True while an undecodable payload may simply be incomplete: its size changed since the last look, or it has not
        been looked at `stale_retries` times yet (each re-queue waits 0.1 s)."""
        last, tries = self._seen.get(chunk_id, (None, 0))
        tries = tries + 1 if last == size else 1
        self._seen[chunk_id] = (size, tries)
        return tries <= self.stale_retries

    def process_batch(self, reqs: List[ChunkRequest]) -> List[bool]:
        """One bool per request: False = payload not there / not complete yet (re-queue)."""
        from skyplane_b200 import native

        ok = [False] * len(reqs)
        ready, frames = [], []
        total = 0
        for i, r in enumerate(reqs):
            fpath = self.chunk_store.get_compressed_file_path(r.chunk.chunk_id)
            try:
                frame = fpath.read_bytes()
            except FileNotFoundError:
                continue  # payload not received yet: retry
            if total + len(frame) + r.chunk.chunk_length_bytes > self.max_batch_bytes and ready:
                continue  # next batch
            total += len(frame) + r.chunk.chunk_length_bytes
            ready.append(i)
            frames.append(frame)
        if not ready:
            return ok
        encrypted = self.e2ee_key_bytes is not None
        out = self._get_stage().decode(frames, [reqs[i].chunk.chunk_length_bytes for i in ready], encrypted=encrypted)
        for i, frame, (data, digest, status) in zip(ready, frames, out):
            chunk = reqs[i].chunk
            if status in (native.D_TRUNCATED, native.D_BAD_HEADER, native.D_AUTH) and self._still_arriving(chunk.chunk_id, len(frame)):
                continue  # a writer may still be appending (a short box fails authentication, a short frame is truncated)
            if status != 0:
                raise ValueError(f"chunk {chunk.chunk_id}: payload rejected ({native.D_NAMES.get(status, status)})")
            want = chunk.md5_hash
            if isinstance(want, str):  # a digest that crossed a JSON hop un-normalised
                want = bytes.fromhex(want)
            if want is not None and bytes(want) != digest:
                raise ChecksumMismatchException(f"chunk {chunk.chunk_id}: md5 {digest.hex()} != expected {bytes(want).hex()}")
            path = self.chunk_store.get_chunk_file_path(chunk.chunk_id)
            tmp = path.with_name(path.name + ".part")
            with open(tmp, "wb") as f:
                f.write(data)
            os.replace(tmp, path)
            chunk.md5_hash = digest  # lets the upload step send Content-MD5 (gateway_operator.py:640)
            self._seen.pop(chunk.chunk_id, None)
            if self.remove_frames:
                self.chunk_store.get_compressed_file_path(chunk.chunk_id).unlink(missing_ok=True)
            ok[i] = True
        return ok

    def worker_loop(self, worker_id: int, *args):
        """Batch-draining loop with the reference's logging / error conventions (gateway_operator.py:79-115)."""
        self.worker_id = worker_id
        try:
            while self._running(worker_id):
                try:
                    reqs = self.input_queue.get_batch_nowait(self.max_batch_chunks, self.handle)
                    if not reqs:
                        time.sleep(0.001)
                        continue
                    self.chunk_store.log_chunk_states(reqs, ChunkState.in_progress, operator_handle=self.handle, worker_id=worker_id)
                    done = self.process_batch(reqs)
                    good = [r for r, g in zip(reqs, done) if g]
                    if good:
                        self.chunk_store.log_chunk_states(good, ChunkState.complete, operator_handle=self.handle, worker_id=worker_id)
                        if self.output_queue is not None:
                            self.output_queue.put_many(good)
                    retry = [r for r, good in zip(reqs, done) if not good]
                    if retry:
                        if len(retry) == len(reqs):
                            time.sleep(0.1)  # nothing was ready: the reference's re-queue pause (gateway_operator.py:103-106)
                        for r in retry:
                            self.input_queue.put(r)
                except Exception as e:
                    self._fail(worker_id, e)
        finally:
            self.worker_exit(worker_id)
