#!/usr/bin/env python
"""Default vs linked-block (F_LINKED) frames on one GPU, device-resident: what the linked mode costs and gains.

  config3    1024 x 16 MiB Silesia-like chunks (bench.py's config3 data): fused LZ4+MD5 and LZ4-only kernel GB/s, ratio, and
             the reference's (liblz4, linked blocks) ratio on the same 16 distinct chunks
  text       ratio of both modes on the text kinds of tools/ratio_kinds.py (files installed on the machine that runs this)
  decode     sky_decode_device GB/s (decoded bytes / kernel time, MD5 of the output included) of the config3 frames of each mode;
             a linked frame's blocks decode one after another

Modes alternate step by step; kernel times are medians over --steps launches after --warmup.  The card's name, power limit and
SM clock are read in the same run and written next to the numbers.  Prints one JSON object (and writes it to --out)."""
import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def gpu_facts():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(zip(q.split(","), (x.strip() for x in r.stdout.strip().split(",")))) if r.returncode == 0 else {"error": r.stderr.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chunks", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    import oracle.reflib as ref
    from skyplane_b200 import native, synth
    from tools.ratio_kinds import kinds

    dev = torch.device("cuda:0")
    n, cb = args.chunks, 16 << 20
    pool_bytes = [synth.silesia_like_chunk(2000 + i, cb) for i in range(16)]
    stride_in, bound = native.round16(cb), native.frame_bound(cb)
    stride_out = native.round16(bound)
    d_in = torch.empty(n * stride_in + 64, dtype=torch.uint8, device=dev)
    pool = [torch.frombuffer(bytearray(b), dtype=torch.uint8).to(dev) for b in pool_bytes]
    for i in range(n):
        d_in[i * stride_in: i * stride_in + cb] = pool[i % 16]
    del pool
    outs = {m: torch.empty(n * stride_out + 64, dtype=torch.uint8, device=dev) for m in ("default", "linked")}
    src_off, dst_off = [i * stride_in for i in range(n)], [i * stride_out for i in range(n)]
    ctx = native.Context(0, n * stride_in, n, 0)
    stream = torch.cuda.current_stream().cuda_stream
    flags = {"default": 0, "linked": native.F_LINKED}
    before = gpu_facts()

    def step(mode, stages):
        return ctx.process_device(d_in.data_ptr(), src_off, [cb] * n, outs[mode].data_ptr(), dst_off, [bound] * n,
                                  stages | flags[mode], stream)

    res = {"gpu_before": before, "config3": {}, "text": {}, "decode": {}}
    frame_lens = {}
    for label, stages in (("fused", 0), ("lz4_only", native.F_LZ4)):
        ms = {"default": [], "linked": []}
        for k in range(args.warmup + args.steps):
            for mode in ("default", "linked") if k % 2 == 0 else ("linked", "default"):
                lens, _, kms = step(mode, stages)
                if k >= args.warmup:
                    ms[mode].append(kms)
                frame_lens[mode] = lens
        for mode in ms:
            med = statistics.median(ms[mode])
            res["config3"][f"{label}_{mode}"] = {"kernel_ms_median": round(med, 3), "kernel_ms_all": [round(x, 3) for x in ms[mode]],
                                                 "GBps": round(n * cb / med / 1e6, 2)}
    ref_ratio = sum(map(len, pool_bytes)) / sum(len(ref.lz4f_compress(b)) for b in pool_bytes)
    for mode in ("default", "linked"):
        ratio = n * cb / sum(frame_lens[mode])
        res["config3"][f"ratio_{mode}"] = round(ratio, 4)
        res["config3"][f"ratio_{mode}_vs_reference"] = round(ratio / ref_ratio, 4)
    res["config3"]["reference_ratio"] = round(ref_ratio, 4)

    # decode the frames of the last step of each mode (fused: frame_lens are the same as LZ4-only's)
    d_back = torch.empty(n * stride_in + 64, dtype=torch.uint8, device=dev)
    dms = {"default": [], "linked": []}
    for k in range(args.warmup + args.steps):
        for mode in ("default", "linked") if k % 2 == 0 else ("linked", "default"):
            st, _, kms = ctx.decode_device(outs[mode].data_ptr(), dst_off, frame_lens[mode], d_back.data_ptr(), src_off, [cb] * n, stream)
            if any(st):
                raise SystemExit(f"{mode} frames do not decode: {sorted(set(st))}")
            if k >= args.warmup:
                dms[mode].append(kms)
    if not torch.equal(d_back, d_in):
        raise SystemExit("decoded bytes differ from the input")
    for mode in dms:
        med = statistics.median(dms[mode])
        res["decode"][mode] = {"kernel_ms_median": round(med, 3), "kernel_ms_all": [round(x, 3) for x in dms[mode]],
                               "GBps": round(n * cb / med / 1e6, 2)}
    del d_back, d_in, outs
    torch.cuda.empty_cache()

    ks = kinds()
    for name in ("python sources 8 MiB", "c headers 8 MiB", "utf-16 text 4 MiB", "silesia-like 4 x 4 MiB (bench set)"):
        d = ks[name]
        if not d:
            continue
        chunks = [d[o:o + (1 << 20)] for o in range(0, len(d), 1 << 20)]  # 1 MiB chunks, like the study's frames but per chunk
        row = {"bytes": len(d), "liblz4_linked_ratio": round(len(d) / sum(len(ref.lz4f_compress(c)) for c in chunks), 4)}
        c2 = native.Context(0, len(d) + 16 * len(chunks) + 4096, len(chunks), 1)
        for mode in ("default", "linked"):
            bufs = [native.PinnedBuffer(len(c)) for c in chunks]
            obufs = [native.PinnedBuffer(native.frame_bound(len(c))) for c in chunks]
            for b, c in zip(bufs, chunks):
                b.view[:len(c)] = c
            t = c2.submit([b.addr for b in bufs], [len(c) for c in chunks], [o.addr for o in obufs],
                          [native.frame_bound(len(c)) for c in chunks], native.F_LZ4 | native.F_MD5 | flags[mode])
            lens, _, _ = c2.wait(t)
            row[f"{mode}_ratio"] = round(len(d) / sum(lens), 4)
            for b in bufs + obufs:
                b.close()
        c2.close()
        res["text"][name] = row
    ctx.close()
    res["gpu_after"] = gpu_facts()
    res["config"] = native.kernel_config()
    res["chunks"], res["chunk_bytes"], res["steps"], res["warmup"] = n, cb, args.steps, args.warmup
    out = json.dumps(res, indent=1)
    print(out)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(out + "\n")


if __name__ == "__main__":
    main()
