#!/usr/bin/env python
"""bench.py -- chunk-pipeline GB/s (raw input) of the fused LZ4-frame + MD5 stage on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA stage
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path on the host cores

Workload = BASELINE.json configs[1]: 1024 x 8 MiB uniform-random chunks per GPU (chunk i =
numpy default_rng(1000+i) for host buffers; torch's CUDA generator for the device-resident set).
One "step" = one pass of the hot path over that batch.

  value     whole-job raw-input GB/s with the batch resident in HBM (device path, sky_process_device);
            timed with CUDA events on the launching stream, barrier + synchronize on both sides, MAX over ranks.
  e2e       the same metric through the host-buffer C ABI (sky_submit / sky_wait, what
            GatewayCompressHash.process uses): pinned host chunks -> H2D -> fused kernel -> D2H of the frames.
  roofline  dominant (only) kernel: algorithmic HBM bytes per launch (input read once + frame written once)
            / its CUDA-event duration, against MEASURED_PEAKS.json's hbm_gbs; plus the MD5 dependent-chain bound.
  cpu_baseline  lz4.frame.compress + hashlib.md5 per chunk on the host cores (liblz4.so.1 via ctypes with
            python-lz4's default preferences; oracle port if liblz4 is absent), bounded sample, median of 3 passes,
            with the host facts that decide it (cgroup cpu.max, cpuset, load average, single-core rate).
  config3   BASELINE.json configs[2] as a sub-record: 1024 x 16 MiB Silesia-like chunks per GPU, device-resident,
            GB/s + compression ratio against the reference's ratio on the same chunks + a decode round trip.
  queue_e2e the gateway plugin path (GatewayCompressHash workers behind a GatewayQueue, chunk files on tmpfs), a bounded
            stream, run as a subprocess after the timed regions (rank 0 only).
Only the cpu_baseline / --impl reference legs touch oracle/.

--dump-outputs DIR  writes what the last timed step of `value` (and of config3, prefixed config3_) handed back, as .npy
            (rank 0): frame_lens (float64, one per chunk), md5 (float32 bytes, chunks x 16) and frame_bytes_sample (float32,
            chunks x up to 4096 bytes of each frame at fixed, seeded relative positions).  Inputs are seeded, so two builds
            run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (it may be read-only); forked workers inherit this

METRIC = "chunk-pipeline GB/s (raw input)"
UNIT = "GB/s"
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
MD5_FLOOR_GBS_AT_1965 = 64 * 1.965e9 / (64 * 16.28) / 1e9  # 0.1207 GB/s per chain: 64 B per 64 steps x 16.28 cycles


# ============================================================================ CPU reference leg
_POOL = None
_COMP = None


def _cpu_init(pool_chunks, chunk_bytes, use_ref, workload="random"):
    """Runs in each worker process: build the chunk pool once (seeded -> identical in every worker)."""
    global _POOL, _COMP
    import numpy as np

    if workload == "random":
        _POOL = [np.random.default_rng(1000 + i).bytes(chunk_bytes) for i in range(pool_chunks)]
    else:
        from skyplane_b200 import synth

        _POOL = [synth.silesia_like_chunk(2000 + i, chunk_bytes) for i in range(pool_chunks)]
    if use_ref:
        import oracle.reflib as ref

        _COMP = ref.Compressor(chunk_bytes)
    else:
        import oracle

        oracle.lib()
        _COMP = None


def _cpu_task(i):
    """The reference's serial pair for one chunk: lz4.frame.compress(data) then hashlib.md5(data).digest()."""
    import ctypes
    import hashlib

    data = _POOL[i % len(_POOL)]
    if _COMP is not None:
        addr = ctypes.cast(ctypes.c_char_p(data), ctypes.c_void_p).value
        clen = _COMP.compress_into(addr, len(data))
        dg = hashlib.md5(data).digest()
    else:
        import oracle

        frame, dg = oracle.chunk_stage(data)
        clen = len(frame)
    return clen, dg[0]


def host_facts() -> dict:
    """What decides a CPU number on a shared box: the cores this process may use, the cgroup quota, the load."""
    def rd(path):
        try:
            return open(path).read().strip()
        except OSError:
            return None

    quota = rd("/sys/fs/cgroup/cpu.max")  # cgroup v2: "max 100000" or "<quota_us> <period_us>"
    if quota is None:  # cgroup v1
        q1, p1 = rd("/sys/fs/cgroup/cpu/cpu.cfs_quota_us"), rd("/sys/fs/cgroup/cpu/cpu.cfs_period_us")
        if q1 and p1:
            quota = "max " + p1 if q1.startswith("-") else f"{q1} {p1}"
    eff = None
    if quota and not quota.startswith("max"):
        try:
            q, per = quota.split()
            eff = float(q) / float(per)
        except ValueError:
            pass
    aff = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else None
    return {"cpu_model": cpu_model(), "os_cpu_count": os.cpu_count(), "sched_affinity": aff, "cgroup_cpu_max": quota,
            "cgroup_quota_cores": eff, "cpuset_effective": rd("/sys/fs/cgroup/cpuset.cpus.effective"),
            "loadavg": list(os.getloadavg()), "usable_cores": min(x for x in (aff, eff, os.cpu_count()) if x)}


class CpuReference:
    """All host cores, one chunk per task -- mirrors the reference's process-per-worker model
    (gateway_operator.py:66-70).  Must be constructed before CUDA is initialised (fork)."""

    def __init__(self, chunk_bytes: int, pool_chunks: int = 16, workload: str = "random"):
        import multiprocessing as mp

        import oracle.reflib as ref

        self.use_ref = ref.available()
        self.kind = "reference" if self.use_ref else "port"
        # one worker process per core this process may really use: the cgroup quota counts (a 1-GPU lease of this pool gets
        # 16 of the host's 128 cores; 128 workers on a 16-core quota only add throttling noise)
        self.cores = max(1, int(host_facts()["usable_cores"] + 0.5))
        self.chunk_bytes = chunk_bytes
        self.pool_chunks = pool_chunks
        self.engine = (f"liblz4 {ref.version()} LZ4F_compressFrame via ctypes (python-lz4 default prefs) + hashlib.md5"
                       if self.use_ref else "oracle/skyoracle.c port (liblz4.so.1 not found) incl. its MD5")
        self.pool = mp.get_context("fork").Pool(self.cores, initializer=_cpu_init, initargs=(pool_chunks, chunk_bytes, self.use_ref, workload))
        self.workload = workload
        self.pool.map(_cpu_task, range(self.cores * 2))  # touch every worker
        self.last_ratio = None

    def run(self, n_chunks: int) -> float:
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_task, range(n_chunks), chunksize=max(1, n_chunks // (self.cores * 8)))
        dt = time.perf_counter() - t0
        self.last_ratio = n_chunks * self.chunk_bytes / sum(r[0] for r in res)
        return dt

    def pool_ratio(self) -> float:
        """The reference's compression ratio over the distinct pool chunks (what config3's GPU ratio is compared with)."""
        res = self.pool.map(_cpu_task, range(self.pool_chunks))
        return self.pool_chunks * self.chunk_bytes / sum(r[0] for r in res)

    def single_core_gbs(self, n: int = 4) -> float:
        """One worker, n chunks back to back: the per-core rate the all-core number should be a multiple of."""
        t0 = time.perf_counter()
        self.pool.apply(_cpu_serial, (n,))
        return n * self.chunk_bytes / (time.perf_counter() - t0) / 1e9

    def measure(self, n_chunks: int, passes: int = 3) -> dict:
        gbs = sorted(n_chunks * self.chunk_bytes / self.run(n_chunks) / 1e9 for _ in range(passes))
        single = self.single_core_gbs()
        med = gbs[len(gbs) // 2]
        return {"value": med, "unit": UNIT, "cores": self.cores, "kind": self.kind, "passes_gbs": [round(g, 3) for g in gbs],
                "spread": (gbs[-1] - gbs[0]) / med if med else None, "single_core_gbs": single,
                "effective_parallelism": med / single if single else None, "per_core_gbs": med / self.cores, "ratio": self.last_ratio,
                "host": host_facts(),
                "sample": f"{n_chunks} x {self.chunk_bytes >> 20} MiB {self.workload} chunks per pass (pool of {self.pool_chunks} distinct, seeded), "
                          f"median of {passes} passes, {self.cores} worker processes, {self.engine}"}

    def close(self):
        self.pool.close()
        self.pool.join()


def _cpu_serial(n):
    for i in range(n):
        _cpu_task(i)
    return n


def cpu_model() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def workload_config(args, world: int) -> dict:
    """The same `config` for both arms: it names the workload, not the implementation."""
    return {"workload": f"{args.chunks} x {args.chunk_mib} MiB {args.workload} chunks per GPU, one pass of LZ4-frame + MD5 per step",
            "chunks_per_gpu": args.chunks, "chunk_bytes": args.chunk_mib << 20, "parallelism": f"chunk-sharded x{world}, no collective",
            "l2": "inputs (8 GiB/GPU) far exceed the 126 MB L2; no explicit flush"}


# ============================================================================ helpers
class ClockSampler:
    """nvidia-smi clock / throttle sampling during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self) -> dict:
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.p.terminate()
        try:
            self.p.wait(5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(names, r[5:9]):
                if v.strip().lower() == "active":
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (copy, read+write bytes)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback 6.65 TB/s (B200_PROFILING.md; MEASURED_PEAKS.json absent)"


# ============================================================================ reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return 0
    chunk_bytes = args.chunk_mib << 20
    ref = CpuReference(chunk_bytes, workload=args.workload)
    n = args.ref_chunks or args.chunks
    for _ in range(args.warmup):
        ref.run(max(ref.cores, n // 8))
    t = [ref.run(n) for _ in range(args.steps)]
    total = sum(t)
    value = n * chunk_bytes * args.steps / total / 1e9
    per_step = sorted(n * chunk_bytes / x / 1e9 for x in t)
    single = ref.single_core_gbs()
    cfg = workload_config(args, world)  # identical to the GPU arm's `config`: both arms name the workload, nothing else
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u32",
        "data": "synthetic", "config": cfg, "details": {"compression_ratio": ref.last_ratio},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": ref.cores, "kind": ref.kind, "single_core_gbs": single,
                         "effective_parallelism": value / single if single else None, "per_core_gbs": value / ref.cores,
                         "step_gbs_min_median_max": [per_step[0], per_step[len(per_step) // 2], per_step[-1]], "host": host_facts(),
                         "sample": f"{n} x {args.chunk_mib} MiB {args.workload} chunks per step on this ONE host whatever --gpus says (pool of 16 "
                                   f"distinct, seeded), {ref.cores} worker processes, {ref.engine}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    ref.close()
    print(json.dumps(line))
    return 0


# ============================================================================ GPU arm
def fill_device_input(torch, native, dev, workload, n_chunks, chunk_bytes, rank):
    """Synthetic batch resident in HBM (outside any timed region). -> (tensor, stride)"""
    stride_in = native.round16(chunk_bytes)
    d_in = torch.empty(n_chunks * stride_in + 64, dtype=torch.uint8, device=dev)
    if workload == "random":
        g = torch.Generator(device=dev)
        g.manual_seed(1000 + rank)
        step_e = 1 << 28
        for o in range(0, d_in.numel(), step_e):
            e = min(d_in.numel(), o + step_e)
            d_in[o:e] = torch.randint(0, 256, (e - o,), dtype=torch.uint8, device=dev, generator=g)
    else:
        from skyplane_b200 import synth

        pool = [torch.frombuffer(bytearray(synth.silesia_like_chunk(2000 + i, chunk_bytes)), dtype=torch.uint8).to(dev) for i in range(16)]
        for i in range(n_chunks):
            d_in[i * stride_in: i * stride_in + chunk_bytes] = pool[(i + rank) % 16]
    return d_in, stride_in


DUMP_SAMPLE_BYTES = 4 << 20  # frame bytes sampled per record: 16 MiB as float32, so value + config3 stay under 64 MB


def sample_outputs(torch, np, d_out, dst_off, out_lens, digests) -> dict:
    """What a caller of the device path holds after a step, as float arrays: every frame length and digest, and each frame's
    bytes at the same fixed, seeded relative positions."""
    n = len(out_lens)
    m = max(1, min(4096, DUMP_SAMPLE_BYTES // n))
    u = np.sort(np.random.default_rng(0).random(m))
    lens = np.asarray(out_lens, dtype=np.int64)
    pos = np.asarray(dst_off, dtype=np.int64)[:, None] + (u[None, :] * lens[:, None]).astype(np.int64)
    sample = d_out[torch.from_numpy(pos.ravel()).to(d_out.device)].float().cpu().numpy().reshape(n, m)
    md5 = np.frombuffer(b"".join(digests), dtype=np.uint8).reshape(n, 16).astype(np.float32)
    return {"frame_lens": lens.astype(np.float64), "md5": md5, "frame_bytes_sample": sample}


def device_resident_run(torch, native, dev, local, workload, n_chunks, chunk_bytes, rank, steps, warmup, sample_clocks=True, verify_decode=False,
                        dump=False):
    """K timed passes of the fused kernel over a batch resident in HBM, CUDA events on the launching stream."""
    import hashlib

    import numpy as np

    d_in, stride_in = fill_device_input(torch, native, dev, workload, n_chunks, chunk_bytes, rank)
    bound = native.frame_bound(chunk_bytes)
    stride_out = native.round16(bound)
    d_out = torch.empty(n_chunks * stride_out + 64, dtype=torch.uint8, device=dev)
    src_off = [i * stride_in for i in range(n_chunks)]
    dst_off = [i * stride_out for i in range(n_chunks)]
    lens, caps = [chunk_bytes] * n_chunks, [bound] * n_chunks
    ctx = native.Context(local, n_chunks * stride_in, n_chunks, 0)
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        return ctx.process_device(d_in.data_ptr(), src_off, lens, d_out.data_ptr(), dst_off, caps, 0, stream)

    for _ in range(warmup):
        step()
    sampler = ClockSampler(local) if sample_clocks else None
    torch.cuda.synchronize()
    if sampler:
        sampler.start()
    launches0 = ctx.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms = []
    ev0.record()
    for _ in range(steps):
        out_lens, digests, kms = step()
        kernel_ms.append(kms)
    ev1.record()
    torch.cuda.synchronize()
    elapsed = ev0.elapsed_time(ev1) / 1e3
    clocks = sampler.stop() if sampler else None
    launches = ctx.launches - launches0
    # parity spot check of the last timed step, outside the timed region (hashlib is stdlib, not the oracle)
    host0 = d_in[:chunk_bytes].cpu().numpy().tobytes()
    if digests[0] != hashlib.md5(host0).digest():
        raise SystemExit("MD5 mismatch against hashlib on chunk 0 -- refusing to report a number")
    roundtrip = None
    if verify_decode:
        # the frames just produced, decoded by the receiver-side kernels, must give the input back (+ the same digests)
        k = min(n_chunks, 64)
        d_back = torch.empty(k * stride_in + 64, dtype=torch.uint8, device=dev)
        st, dg2, _ = ctx.decode_device(d_out.data_ptr(), dst_off[:k], out_lens[:k], d_back.data_ptr(), src_off[:k], lens[:k], 0)
        roundtrip = all(x == 0 for x in st) and dg2 == digests[:k] and bool(torch.equal(d_back[: k * stride_in - (stride_in - chunk_bytes)], d_in[: k * stride_in - (stride_in - chunk_bytes)]))
        del d_back
        if not roundtrip:
            raise SystemExit("LZ4 frames do not decode back to the input -- refusing to report a number")
    res = {"elapsed": elapsed, "kernel_ms": statistics.mean(kernel_ms), "frame_bytes": sum(out_lens), "launches": launches,
           "clocks": clocks, "roundtrip": roundtrip, "total_in": n_chunks * chunk_bytes,
           "outputs": sample_outputs(torch, np, d_out, dst_off, out_lens, digests) if dump else None}
    ctx.close()
    del d_in, d_out
    torch.cuda.empty_cache()
    return res


def host_copy_ceiling(torch, dev, seconds: float = 1.0):
    """Pinned H2D and D2H running at the same time on this rank's GPU, no kernel: the ceiling of the e2e number.
    Under torchrun every rank runs it at the same moment, so shared host limits (DRAM, IIO) are in the figure."""
    n = 1 << 30
    h_in = torch.empty(n, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(n, dtype=torch.uint8).pin_memory()
    d_a = torch.empty(n, dtype=torch.uint8, device=dev)
    d_b = torch.empty(n, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

    def both():
        with torch.cuda.stream(s1):
            d_a.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_b, non_blocking=True)

    both()
    torch.cuda.synchronize()
    reps = 0
    t0 = time.perf_counter()
    while True:
        both()
        reps += 1
        torch.cuda.synchronize()
        if time.perf_counter() - t0 > seconds:
            break
    dt = time.perf_counter() - t0
    del h_in, h_out, d_a, d_b
    return n * reps / dt / 1e9  # GB/s per direction, both directions busy


def run_gpu(args):
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    chunk_bytes = args.chunk_mib << 20
    n_chunks = args.chunks
    do_c3 = not args.no_config3 and args.workload == "random"

    # ---- CPU legs first: they fork, so they must run before CUDA exists in this process (rank 0, N=1 only)
    cpu = None
    ref_ratio3 = None
    if world == 1 and not args.no_cpu_baseline:
        ref = CpuReference(chunk_bytes, workload=args.workload)
        cpu = ref.measure(args.cpu_chunks, passes=3)
        ref.close()
    if rank == 0 and do_c3:
        ref3 = CpuReference(16 << 20, pool_chunks=16, workload="silesia")  # the reference's ratio on config3's 16 distinct chunks
        ref_ratio3 = ref3.pool_ratio()
        ref3.close()

    import hashlib

    import numpy as np
    import torch

    from skyplane_b200 import native
    from skyplane_b200.sharding import max_over_ranks

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the stage has no CPU fallback (use --impl reference for the CPU arm)")
    from skyplane_b200.numa import bind_to_gpu

    numa_node = bind_to_gpu(local) if world > 1 else None  # pinned staging on the GPU's own socket
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    # ---- value: device-resident batch, CUDA events, MAX over ranks
    barrier()
    dump = bool(args.dump_outputs) and rank == 0
    r = device_resident_run(torch, native, dev, local, args.workload, n_chunks, chunk_bytes, rank, args.steps, args.warmup, dump=dump)
    barrier()
    elapsed = max_over_ranks(r["elapsed"], dev)
    clocks, gpu_launches = r["clocks"], r["launches"]
    total_in, frame_bytes, k_ms = r["total_in"], r["frame_bytes"], r["kernel_ms"]
    value = world * total_in * args.steps / elapsed / 1e9
    ratio = total_in / frame_bytes
    peak, peak_src = measured_peak()
    algo_bytes = total_in + frame_bytes + 16 * n_chunks  # input read once + frame written once + digests
    achieved = algo_bytes / (k_ms * 1e-3) / 1e9
    clk = ((clocks or {}).get("sm_mhz") or 1965.0) / 1965.0
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
        "peak_source": peak_src, "kernel": "sky_fused_kernel", "kernel_ms": k_ms,
        "algorithmic_bytes_per_launch": algo_bytes,
        "raw_input_gbs": total_in / (k_ms * 1e-3) / 1e9, "raw_input_frac_of_peak": total_in / (k_ms * 1e-3) / 1e9 / peak,
        # secondary bound (SURVEY.md section 8d): one MD5 chain per chunk; chain time = 64-byte blocks x cycles/block
        "md5_chain": {"streams": n_chunks, "bytes_per_stream": chunk_bytes,
                      "per_stream_gbs": chunk_bytes / (k_ms * 1e-3) / 1e9,
                      # floor measured by tools/md5_chain_bench.cu (profiles/r1_md5_chain_microbench.txt): 16.28 cycles per
                      # MD5 step x 64 steps per 64-byte block, scaled to the SM clock seen during this run
                      "per_stream_floor_gbs": MD5_FLOOR_GBS_AT_1965 * clk,
                      "bound_gbs": n_chunks * MD5_FLOOR_GBS_AT_1965 * clk,
                      "frac_of_bound": (total_in / (k_ms * 1e-3) / 1e9) / (n_chunks * MD5_FLOOR_GBS_AT_1965 * clk),
                      "note": "kernel time >= one chunk's serial MD5 chain; the batch cannot exceed streams x per_stream_floor_gbs"},
    }
    prof = ROOT / "profiles" / "traffic_latest.json"
    if prof.exists():
        try:
            roofline["traffic"] = json.loads(prof.read_text()).get("dram_bytes_per_launch")
        except Exception:
            pass

    # ---- e2e: host-buffer C ABI path, pinned host chunks, H2D + kernel + D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        stride_in = native.round16(chunk_bytes)
        bound = native.frame_bound(chunk_bytes)
        stride_out = native.round16(bound)
        sub = min(args.e2e_batch, n_chunks)
        n_sub = (n_chunks + sub - 1) // sub
        slots = args.e2e_slots
        ectx = native.Context(local, sub * stride_in, sub, slots)
        pool_n = min(64 if args.workload == "random" else 16, n_chunks)  # distinct host chunks, recycled
        pin_in = native.PinnedBuffer(pool_n * stride_in)
        if args.workload == "random":
            for i in range(pool_n):
                pin_in.view[i * stride_in: i * stride_in + chunk_bytes] = np.random.default_rng(1000 + i + 64 * rank).bytes(chunk_bytes)
        else:
            from skyplane_b200 import synth

            for i in range(pool_n):
                pin_in.view[i * stride_in: i * stride_in + chunk_bytes] = synth.silesia_like_chunk(2000 + i + 64 * rank, chunk_bytes)
        pin_out = [native.PinnedBuffer(sub * stride_out) for _ in range(slots)]

        class Pipe:
            """Continuous sky_submit / sky_wait pipeline: `slots` sub-batches in flight, across step boundaries."""

            def __init__(self):
                self.inflight = []
                self.h2d = self.d2h = self.done = 0
                self.last_dg = None
                self.b = 0

            def push_step(self):
                for b in range(n_sub):
                    lo, hi = b * sub, min(n_chunks, (b + 1) * sub)
                    if len(self.inflight) == slots:
                        self.pop()
                    ob = pin_out[self.b % slots]
                    self.b += 1
                    src = [pin_in.addr + ((i % pool_n) * stride_in) for i in range(lo, hi)]
                    dst = [ob.addr + (i - lo) * stride_out for i in range(lo, hi)]
                    t = ectx.submit(src, [chunk_bytes] * (hi - lo), dst, [bound] * (hi - lo))
                    self.h2d += (hi - lo) * chunk_bytes
                    self.inflight.append(t)

            def pop(self):
                ol, dg, _ = ectx.wait(self.inflight.pop(0))
                self.d2h += sum(ol) + 24 * len(ol)
                self.done += len(ol)
                self.last_dg = dg

            def drain(self):
                while self.inflight:
                    self.pop()

        pipe = Pipe()
        for _ in range(max(1, min(2, args.warmup))):
            pipe.push_step()
        pipe.drain()
        dg = pipe.last_dg
        lastc = ((n_chunks - 1) % pool_n) * stride_in
        if dg[-1] != hashlib.md5(bytes(pin_in.view[lastc: lastc + chunk_bytes])).digest():
            raise SystemExit("e2e MD5 mismatch against hashlib")
        barrier()
        el0 = ectx.launches
        pipe = Pipe()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pipe.push_step()
        pipe.drain()  # every frame of all K steps is back in host memory
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        assert pipe.done == n_chunks * args.steps
        h2d, d2h = pipe.h2d // args.steps, pipe.d2h // args.steps
        barrier()
        dt = max_over_ranks(dt, dev)
        e2e = {"value": world * total_in * args.steps / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "ms_per_step": dt / args.steps * 1e3, "sub_batches": n_sub, "slots_in_flight": slots, "gpu_launches": ectx.launches - el0,
               "api": "sky_submit/sky_wait (host-buffer C ABI used by GatewayCompressHash.process); wall clock incl. host sync"}
        ectx.close()
        del pin_in, pin_out
        # the ceiling this number lives under: concurrent pinned H2D + D2H on every rank's GPU at once, no kernel
        barrier()
        ceil_rank = host_copy_ceiling(torch, dev)
        barrier()
        ceil_all = world * (-max_over_ranks(-ceil_rank, dev))  # world x the slowest rank's rate
        e2e["host_ceiling_gbs"] = ceil_all
        e2e["frac_of_host_ceiling"] = e2e["value"] / ceil_all if ceil_all else None
        e2e["host_ceiling_note"] = "pinned H2D+D2H both busy on all ranks' GPUs at once (1 GiB copies, ~1 s): GB/s per direction, summed over ranks (slowest rank x world)"

    # ---- config3 (BASELINE.json configs[2]): 1024 x 16 MiB Silesia-like, device-resident, ratio parity + decode round trip
    config3 = None
    if do_c3:
        barrier()
        c3 = device_resident_run(torch, native, dev, local, "silesia", args.c3_chunks, 16 << 20, rank, max(2, args.steps // 2), 2,
                                 sample_clocks=False, verify_decode=True, dump=dump)
        barrier()
        el3 = max_over_ranks(c3["elapsed"], dev)
        steps3 = max(2, args.steps // 2)
        gpu_ratio = c3["total_in"] / c3["frame_bytes"]
        algo3 = c3["total_in"] + c3["frame_bytes"] + 16 * args.c3_chunks
        config3 = {"workload": f"{args.c3_chunks} x 16 MiB Silesia-like chunks per GPU (16 distinct, seeded), device-resident, fused LZ4-frame+MD5",
                   "value": world * c3["total_in"] * steps3 / el3 / 1e9, "unit": UNIT, "steps": steps3, "kernel_ms": c3["kernel_ms"],
                   "compression_ratio": gpu_ratio, "reference_ratio": ref_ratio3,
                   "ratio_vs_reference": (gpu_ratio / ref_ratio3) if ref_ratio3 else None,
                   "decode_roundtrip_64_chunks": c3["roundtrip"],
                   "roofline_achieved_gbs": algo3 / (c3["kernel_ms"] * 1e-3) / 1e9, "roofline_frac": algo3 / (c3["kernel_ms"] * 1e-3) / 1e9 / peak,
                   "md5_chain_bound_gbs": args.c3_chunks * MD5_FLOOR_GBS_AT_1965 * clk}

    # ---- queue_e2e: the plugin path (GatewayQueue -> forked GatewayCompressHash workers -> chunk files on tmpfs), bounded stream
    queue_e2e = None
    if not args.no_queue_e2e:
        barrier()
        if rank == 0:
            cmd = [sys.executable, "-m", "skyplane_b200.harness", "--gpus", str(world), "--chunks", str(args.queue_chunks * world), "--chunk-mib",
                   str(args.chunk_mib), "--workload", args.workload if args.workload == "random" else "silesia", "--pool", "32", "--batch", "128", "--slots", "4"]
            env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT")}
            env["PYTHONDONTWRITEBYTECODE"] = "1"
            try:
                out = subprocess.run(cmd, capture_output=True, text=True, timeout=240, cwd=str(ROOT), env=env)
                queue_e2e = json.loads(out.stdout.strip().splitlines()[-1]) if out.returncode == 0 else {"error": out.stderr[-400:]}
            except Exception as e:  # a broken harness must not take the bench line down with it
                queue_e2e = {"error": repr(e)}
        barrier()

    if dump:
        dump_dir = Path(args.dump_outputs)
        dump_dir.mkdir(parents=True, exist_ok=True)
        for prefix, rec in (("", r), ("config3_", c3 if do_c3 else None)):
            for name, arr in ((rec or {}).get("outputs") or {}).items():
                np.save(dump_dir / f"{prefix}{name}.npy", arr)

    if rank == 0:
        cfg = workload_config(args, world)
        details = {"compression_ratio": ratio, "numa_node_rank0": numa_node, "kernel_build": native.kernel_config()}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": elapsed / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/u32", "data": "synthetic", "config": cfg, "details": details,
            "e2e": e2e, "gpu_launches": gpu_launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "config3": config3, "queue_e2e": queue_e2e,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--chunks", type=int, default=1024, help="chunks per GPU per step")
    ap.add_argument("--chunk-mib", type=int, default=8)
    ap.add_argument("--workload", choices=["random", "silesia"], default="random")
    ap.add_argument("--e2e-batch", type=int, default=256, help="chunks per sky_submit call")
    ap.add_argument("--e2e-slots", type=int, default=4, help="sky_submit batches in flight")
    ap.add_argument("--ref-chunks", type=int, default=0, help="chunks per step of the reference arm (default: --chunks)")
    ap.add_argument("--cpu-chunks", type=int, default=1024, help="chunks in the cpu_baseline sample")
    ap.add_argument("--c3-chunks", type=int, default=1024, help="chunks per GPU of the config3 sub-record (16 MiB each)")
    ap.add_argument("--queue-chunks", type=int, default=1024, help="chunks per GPU streamed through the gateway-queue harness")
    ap.add_argument("--no-config3", action="store_true")
    ap.add_argument("--no-queue-e2e", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the last timed step's outputs as .npy files into DIR")
    args = ap.parse_args()
    if args.warmup < 3 and args.impl == "b200":
        print("note: timing rules ask for >= 3 warm-up steps", file=sys.stderr)
    sys.exit(run_reference(args) if args.impl == "reference" else run_gpu(args))


if __name__ == "__main__":
    main()
