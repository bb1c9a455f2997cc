// skychunk.cu -- fused LZ4-frame + MD5 chunk stage for B200 (sm_100a) and its C ABI (include/skychunk.h).
//
// One persistent kernel per batch (sky_fused_kernel), two CTAs per SM, 14 warps per CTA, one role per CTA at a time:
//   * digest CTAs : the first few CTAs carry the MD5 groups -- 32 chunks per warp, lane = chunk (md5.cuh), one MD5 warp
//                   per CTA while the groups are few.  An MD5 chain is latency bound (3 dependent ALU ops per step, one
//                   64-byte block per 1042 cycles) and keeps its scheduler's issue port busy; when a CTA's groups are done
//                   it joins the compressors.
//   * compressor CTAs : one 64 KiB block at a time, claimed from a global atomic counter in row-major order (block row j of
//                   every chunk, then row j+1 ...): bulk-load the block into shared memory, warps 0-1 probe, warps 2-13
//                   parse segment by segment into an L2-resident scratch (lz4.cuh), warp 0 plans the block's layout.
// Output placement (single pass, no compaction kernel): a block's final place in the frame is only known when every block
// before it has been sized, so one per-chunk word orders the blocks:
//   OFF = (next block index << 40) | frame offset of that block: a prefix sum handed from block j-1 to block j as soon as
//         j-1 knows its compressed size -- before it has written a byte, so offsets race down the chain.
// Block j sizes itself from its segments' records, waits for OFF (its final position), publishes OFF for j+1 and then
// writes its bytes to the final place exactly once (stored blocks straight from the input).  The last block's CTA writes
// the EndMark and the frame length.
//
// HBM-read sharing: when MD5 is the slower stage, LZ4 work for block row j is released only when the MD5 lanes have entered
// that row (per-group progress word), so a row is pulled from HBM once and the lanes find it in L2.
//
// Host side: sky_ctx owns a stream, pinned + device metadata arrays, and (optionally) per-slot input /
// output slabs for the host-buffer path (H2D -> kernel -> D2H on one stream per slot).
// There is NO CPU fallback anywhere in this file: without a CUDA device every entry point fails.

#include <cuda_runtime.h>
#include <inttypes.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <numeric>
#include <string>
#include <vector>

#include "../../include/skychunk.h"
#include "lz4.cuh"
#include "lz4dec.cuh"
#include "md5.cuh"
#include "secretbox.cuh"

namespace sky {

#ifndef SKY_PARSERS
#define SKY_PARSERS 12
#endif
constexpr int kParsers = SKY_PARSERS;     // parser warps per CTA
constexpr int kProbers = 2;               // prober warps (0 and 1): they take alternate 256-slot batches
constexpr int kWarps = kProbers + kParsers;
constexpr int kThreads = kWarps * 32;
#ifndef SKY_RING_EXTRA
#define SKY_RING_EXTRA 2
#endif
constexpr int kMd5WarpsPerCta = 4;        // digest CTAs run 4 MD5 groups (one per SM sub-partition), see sky_fused_kernel
constexpr uint32_t kRingBytes = SKY_MD5_SLOTS * 2048;  // MD5 staging ring: slots x 64 B x 32 lanes
constexpr uint32_t kLoadPiece = 8192;     // bytes per bulk copy of the block load
constexpr int kCtasPerSm = 2;             // fused kernel: 2 x ~110 KiB of shared memory per SM
constexpr int kOffBits = 40;
constexpr uint64_t kOffMask = (1ull << kOffBits) - 1;

// Linked blocks (SKY_F_LINKED): block j >= 1 of a chunk is parsed with the kLinkedWindow raw bytes before it in shared
// memory ([window | block]), the table seeded with every (1 << kLinkedSeedLog)-th window position.  The window is what
// fits next to a 4096-entry table once the linked kernel gives up the ring's spare slots (DESIGN.md §4.2: a smaller
// table loses more ratio than a larger window gains).  A multiple of 1024, so that no probe group straddles the point
// where window coordinates wrap modulo 65536 (probe_batch).
#ifndef SKY_LINKED_WINDOW
#define SKY_LINKED_WINDOW 4096
#endif
#ifndef SKY_LINKED_SEED_LOG
#define SKY_LINKED_SEED_LOG 0
#endif
constexpr uint32_t kLinkedWindow = SKY_LINKED_WINDOW;
constexpr uint32_t kLinkedSeedLog = SKY_LINKED_SEED_LOG;
static_assert(kLinkedWindow % 1024 == 0 && kLinkedWindow <= kBlock, "SKY_LINKED_WINDOW must be a multiple of 1024, at most 64 KiB");

// ---- shared-memory layout of the fused kernel (dynamic, 128-byte aligned base) -------------------------
struct BlockDesc {            // written by the prober's lane 0, read by every warp after the block-start barrier
    const uint8_t *src;       // block start in the chunk (16-byte aligned)
    uint8_t *dst;             // chunk's frame region
    uint32_t c, j, L, last;   // chunk, block index, block length, 1 = last block of the chunk
    uint32_t valid, pad;
};
template <int kRing>
struct Ctl {
    uint64_t in_full;               // bulk copy of the block has landed
    uint64_t full[kRing], empty[kRing];
    BlockDesc desc[2];              // by block-iteration parity
    uint32_t claim;                 // next segment sequence number a parser may take (runs across blocks)
    volatile uint32_t block_end_seq;  // sequence number after the current block's last segment (0xffffffff while probing)
    volatile uint32_t nseg;
    volatile uint32_t seg_hit[4];     // per segment (mod 4): OR of its batches' hit masks (decides the stride two segments on)
    uint32_t csize, raw, last_lits, tail_off;   // plan results: compressed size, stored?, final literal run and where it goes
    uint32_t data_lo, data_hi;                  // frame offset of the block's first data byte
};
// kLinked: the block buffer has room for the window in front of the block, paid for by the ring's spare slots.
template <bool kLinked>
struct Smem {
    static constexpr int kRing = kParsers + (kLinked ? 0 : SKY_RING_EXTRA);  // segment slots between the prober and the parsers
    static constexpr uint32_t kWin = kLinked ? kLinkedWindow : 0;
    static constexpr uint32_t kInBytes = kWin + kBlock + 128;  // + slack: unaligned 4-byte reads may touch the word after the last byte
    static constexpr uint32_t kInOff = 0;
    static constexpr uint32_t kTabOff = kInOff + kInBytes;
    static constexpr uint32_t kRingOff = kTabOff + kTableBytes;
    static constexpr uint32_t kRecOff = kRingOff + kRing * (uint32_t)sizeof(SegSlot);
    static constexpr uint32_t kPlanOff = kRecOff + kMaxSegs * (uint32_t)sizeof(SegRec);
    static constexpr uint32_t kCtlOff = kPlanOff + kMaxSegs * (uint32_t)sizeof(SegPlan);
    static constexpr uint32_t kBytes = (kCtlOff + (uint32_t)sizeof(Ctl<kRing>) + 127u) & ~127u;
    static_assert(kBytes <= 232448 / 2 - 1024, "two CTAs per SM need <= 112.5 KiB each: lower SKY_PARSERS, SKY_LZ4_ENTRIES or SKY_LINKED_WINDOW");
    static_assert(kMd5WarpsPerCta * kRingBytes <= kInBytes, "the MD5 rings live in the block buffer of a digest CTA");
};
constexpr uint32_t kSmemBytes = Smem<false>::kBytes;
constexpr uint32_t kLinkedSmemBytes = Smem<true>::kBytes;
static_assert(kEntries % 128 == 0, "SKY_LZ4_ENTRIES must be a multiple of 128");
static_assert(sizeof(SegSlot) % 16 == 0 && sizeof(SegRec) == 16 && sizeof(SegPlan) == 16, "layout");

struct ChunkDesc {
    const uint8_t *src;  // 16-byte aligned
    uint8_t *dst;        // 16-byte aligned
    uint64_t len;
    uint32_t nblk;
    uint32_t group;  // MD5 group (warp) that digests this chunk
};

struct Params {
    const ChunkDesc *chunks;
    const uint32_t *md5_order;  // chunk indices, longest first, padded with 0xffffffff to 32*n_groups
    uint64_t *chain;            // per chunk OFF word: (next block index << 40) | frame offset of that block
    uint32_t *md5_progress;     // per MD5 group: 0 = not started, else 1 + 64 KiB rows consumed (0xffffffff = done)
    uint64_t *out_len;          // per chunk frame length
    uint8_t *md5_out;           // 16 bytes per chunk
    uint32_t *counters;         // [0] = LZ4 work counter
    uint8_t *scratch;           // kScratchBytes per CTA: where a block's segments are compressed before its frame offset is known
    uint32_t n_chunks;
    uint32_t n_groups;
    uint32_t n_md5_ctas;        // CTAs 0..n_md5_ctas-1 digest (4 groups each at a time) before they compress
    uint32_t rows;  // max(1, max nblk)
    uint32_t flags;
};

__device__ __forceinline__ uint64_t ld_acquire(const uint64_t *p) {
    uint64_t v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t ld_acquire32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(uint64_t *p, uint64_t v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_release32(uint32_t *p, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// named-barrier token between the two prober warps: the releaser arrives, the waiter syncs (ids 1 and 2, 64 threads)
template <int kId>
__device__ __forceinline__ void bar_arrive() { asm volatile("bar.arrive %0, 64;" ::"n"(kId) : "memory"); }
template <int kId>
__device__ __forceinline__ void bar_wait() { asm volatile("bar.sync %0, 64;" ::"n"(kId) : "memory"); }
__device__ __forceinline__ uint32_t ld_relaxed32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Prober lane 0: claim the next block that has LZ4 work (empty chunks are finished on the spot), wait until the chunk's
// MD5 lanes are close (so the block is read from HBM once), and describe it to the CTA.
template <bool kLinked>
__device__ __forceinline__ void claim_block(const Params &p, BlockDesc *d, bool pace) {
    const uint32_t total = p.rows * p.n_chunks;
    for (;;) {
        const uint32_t w = atomicAdd(p.counters, 1u);
        if (w >= total) {
            d->valid = 0;
            return;
        }
        const uint32_t c = w % p.n_chunks, j = w / p.n_chunks;  // row-major: block row j of every chunk, then row j+1
        const ChunkDesc cd = p.chunks[c];
        if (cd.nblk == 0) {
            if (j == 0) {  // empty chunk: 7-byte header + EndMark
                const uint32_t h = write_frame_header(cd.dst, 0);
                cd.dst[h] = cd.dst[h + 1] = cd.dst[h + 2] = cd.dst[h + 3] = 0;
                p.out_len[c] = h + 4;
            }
            continue;
        }
        if (j >= cd.nblk) continue;
        if (pace) {
            // stay at most one 64 KiB row ahead of the MD5 lanes of this chunk (only while they are running); the last
            // rows may run up to kTailLead rows ahead so the compressor's own latency for the final row overlaps the
            // digest's last rows instead of trailing them
            const uint32_t *pw = p.md5_progress + cd.group;
            constexpr uint32_t kTailLead = 8;
            const uint32_t lead = (cd.nblk - j <= kTailLead) ? kTailLead : 0;
            unsigned ns = 64;
            for (;;) {
                const uint32_t pr = ld_relaxed32(pw);
                // pr: 0 = digest not started, 0xffffffff = finished, else 1 + rows consumed (64-bit compare: no wrap)
                if (pr == 0 || (uint64_t)j + 1 <= (uint64_t)pr + lead) break;
                __nanosleep(ns);
                if (ns < 4096) ns <<= 1;
            }
        }
        const uint64_t boff = (uint64_t)j * kBlock;
        d->src = cd.src + boff;
        d->dst = cd.dst;
        d->c = c;
        d->j = j;
        d->L = (uint32_t)min((uint64_t)kBlock, cd.len - boff);
        d->last = (j + 1 == cd.nblk);
        d->valid = 1;
        if (j == 0) write_frame_header(cd.dst, cd.len, kLinked);
        return;
    }
}

// Fused LZ4-frame + MD5 kernel.  Grid = 2 CTAs per SM, kWarps warps each.
//   digest CTAs (blockIdx < n_md5_ctas): warps 0..3 each carry one MD5 group (32 chunks, lane = chunk, md5.cuh) at a time;
//       when the groups are done the CTA joins the compressors.
//   compressor CTAs: one 64 KiB block at a time -- bulk-load it into shared memory, warp 0 probes, warps 1.. parse
//       (lz4.cuh), warp 0 plans the block's layout and takes its frame offset from the OFF chain, all warps write it out.
// OFF chain (per chunk): (next block index << 40) | frame offset of that block -- a prefix sum handed from block j-1 to
// block j as soon as j-1 knows its compressed size.  Waiting is deadlock-free: a CTA only waits on lower-numbered work
// items, all of which were claimed earlier by running CTAs.
// kLinked (sky_fused_linked_kernel): block j >= 1 is parsed behind its window (lz4.cuh parse_segment), frames get FLG 0x48.
// Each block's window is raw input, already in HBM: no block waits on another block's compression.
template <bool kLinked>
__device__ __forceinline__ void fused_body(const Params &p) {
    using S = Smem<kLinked>;
    constexpr int kRing = S::kRing;
    constexpr uint32_t kInOff = S::kInOff, kTabOff = S::kTabOff, kRingOff = S::kRingOff;
    extern __shared__ __align__(128) uint8_t smem[];
    const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t *in = smem + kInOff;
    uint32_t *tab = reinterpret_cast<uint32_t *>(smem + kTabOff);
    SegSlot *ring = reinterpret_cast<SegSlot *>(smem + kRingOff);
    SegRec *recs = reinterpret_cast<SegRec *>(smem + S::kRecOff);
    SegPlan *plans = reinterpret_cast<SegPlan *>(smem + S::kPlanOff);
    Ctl<kRing> *ctl = reinterpret_cast<Ctl<kRing> *>(smem + S::kCtlOff);
    uint32_t smem_s = smem_u32(smem);  // shared-window address of the CTA's buffer, kept in a register: left to itself the
    asm volatile("" : "+r"(smem_s));   // compiler re-derives it (S2UR SR_CgaCtaId + ULEA) at the top of every prober batch

    const bool do_md5 = (p.flags & SKY_F_MD5) != 0, do_lz4 = (p.flags & SKY_F_LZ4) != 0;
    if (warp == 0 && lane == 0) {
        mbar_init(&ctl->in_full, 1);
        for (int i = 0; i < kRing; i++) {
            mbar_init(&ctl->full[i], 1);
            mbar_init(&ctl->empty[i], 1);
        }
        ctl->claim = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (do_md5 && blockIdx.x < p.n_md5_ctas) {
        if (warp < kMd5WarpsPerCta) {
            for (uint32_t g = warp * p.n_md5_ctas + blockIdx.x; g < p.n_groups; g += p.n_md5_ctas * kMd5WarpsPerCta) {
                const uint32_t c = p.md5_order[g * 32 + lane];
                const bool active = c != 0xffffffffu;
                const uint8_t *src = nullptr;
                uint64_t len = 0;
                if (active) {
                    src = p.chunks[c].src;
                    len = p.chunks[c].len;
                }
                volatile uint32_t *prog = p.md5_progress + g;
                if (lane == 0) *prog = 1u;  // started, 0 rows consumed
                md5_warp(reinterpret_cast<uint32_t *>(in + warp * kRingBytes), src, len, active, p.md5_out + (size_t)(active ? c : 0) * 16,
                         lane, prog);
                if (lane == 0) *prog = 0xffffffffu;
                __syncwarp();
            }
        }
        if (!do_lz4) return;
        __syncthreads();  // the rings overlapped the block buffer
    }
    if (!do_lz4) return;

    const bool pace = do_md5 && !(p.flags & SKY_F_NO_PACING);
    uint8_t *scratch = p.scratch + (size_t)blockIdx.x * kScratchBytes;
    uint32_t gseq = 0;        // probers: sequence number of the next segment they publish (runs across blocks)
    uint32_t batches_done = 0;  // prober 0: nothing to wait for before the kernel's very first batch
    uint32_t my_seq = 0;      // parser: the sequence number it holds a claim on
    bool have_claim = false;
    uint32_t in_phase = 0;
    for (uint32_t it = 0;; it++) {
        BlockDesc *dsc = &ctl->desc[it & 1];
        if (warp == 0 && lane == 0) {
            claim_block<kLinked>(p, dsc, pace);
            ctl->block_end_seq = 0xffffffffu;
            ctl->nseg = 0;
        }
        __syncthreads();  // (also: every warp is done with the previous block's buffer, records and plan)
        if (!dsc->valid) break;
        const uint8_t *src = dsc->src;
        const uint32_t L = dsc->L;
        const uint32_t base = kLinked && dsc->j > 0 ? S::kWin : 0u;  // window bytes in front of the block in shared memory

        if (warp < kProbers) {
            // ---------------------------------------------------------------- probers (warps 0 and 1, alternate batches of every segment)
            if (warp == 0) {
                if (lane == 0) {
                    const uint32_t bytes = (L + 15u) & ~15u;  // (the input slab is readable up to the next multiple of 16)
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic reads of the old block before the async write
                    mbar_arrive_expect_tx(&ctl->in_full, bytes + base);
                    if (kLinked && base) bulk_load(in, src - base, base, &ctl->in_full);  // the window: the raw bytes before the block
                    for (uint32_t o = 0; o < bytes; o += kLoadPiece)  // several copies in flight: the pieces stream in parallel
                        bulk_load(in + base + o, src + o, min(kLoadPiece, bytes - o), &ctl->in_full);
                }
                // clear the table meanwhile: entry 0 = (position 0, tag 0) doubles as "empty".  (Warp 1's first table access
                // follows warp 0's first table phase through the token, so it sees the cleared table.)
                uint4 *t4 = reinterpret_cast<uint4 *>(tab);
                const uint4 z = make_uint4(0, 0, 0, 0);
#pragma unroll 4
                for (uint32_t k = lane; k < kEntries / 4; k += 32) t4[k] = z;
                __syncwarp();
            }
            mbar_wait(&ctl->in_full, in_phase);
            in_phase ^= 1;
            if constexpr (kLinked) {
                if (warp == 0 && base && L >= kMfLimit + 1) {
                    // seed the table with the window: inserts only, no hits (positions < 65536 here: the max keeps the last)
                    for (uint32_t q = lane << kLinkedSeedLog; q < S::kWin; q += 32u << kLinkedSeedLog) {
                        const uint32_t hf = load32s(smem_s + kInOff, q) * 2654435761u + lds8(smem_s + kInOff + q + 4) * 0x85EBCA6Bu;
                        red_max_s(smem_s + kTabOff + __umulhi(hf, kEntries) * 4u, __byte_perm(q, hf, 0x1065));
                    }
                    __syncwarp();
                }
            }
            uint32_t nseg = 0;
            if (L >= kMfLimit + 1) {
                const uint32_t mflimit = base + L - kMfLimit;
                uint32_t seg_pos = base, slog = 0;
                while (seg_pos <= mflimit) {
                    if (nseg >= 2) {  // the verdict on segment nseg-2 decides this segment's stride
                        const bool h = ctl->seg_hit[(nseg - 2) & 3u] != 0u;
                        slog = h ? 0u : min(slog + 1u, kMaxStepLog);
                    }
                    const uint32_t si = gseq % kRing, ph = (gseq / kRing) & 1u;
                    SegSlot *slot = ring + si;
#pragma unroll 1
                    for (uint32_t b = warp; b < 4; b += kProbers) {
                        const uint32_t slot_s = smem_s + kRingOff + si * (uint32_t)sizeof(SegSlot);
                        const uint32_t hits = probe_batch<kLinked>(smem_s + kInOff, smem_s + kTabOff, slot_s + (uint32_t)offsetof(SegSlot, offs),
                                                          slot_s + (uint32_t)offsetof(SegSlot, masks), seg_pos, slog, b, mflimit, lane, [&]() {
                            // my turn at the table: the other prober has finished the previous batch
                            if (warp == 0) {
                                if (batches_done) bar_wait<2>();
                                if (b == 0) mbar_wait(&ctl->empty[si], ph ^ 1u);  // the ring slot is free again
                            } else {
                                bar_wait<1>();
                            }
                        });
                        batches_done = 1;
                        if (lane == 0) {
                            ctl->seg_hit[nseg & 3u] = (b == 0 ? 0u : ctl->seg_hit[nseg & 3u]) | hits;
                            if (b == 0) {
                                slot->seg_pos = seg_pos;
                                slot->slog = slog;
                                slot->sidx = nseg;
                            }
                        }
                        __syncwarp();
                        if (b == 3 && lane == 0) mbar_arrive(&ctl->full[si]);  // (release: both probers' slot writes are ordered before it)
                        __threadfence_block();
                        if (warp == 0) bar_arrive<1>(); else bar_arrive<2>();  // pass the token
                    }
                    seg_pos += kSegSlots << slog;
                    gseq++;
                    nseg++;
                }
            }
            if (warp == kProbers - 1 && lane == 0) {
                ctl->nseg = nseg;
                __threadfence_block();
                atomicExch(const_cast<uint32_t *>(&ctl->block_end_seq), gseq);  // (atomic: the parsers poll this word)
            }
        } else {
            // ---------------------------------------------------------------- parsers
            mbar_wait(&ctl->in_full, in_phase);  // the block is in shared memory (the prober may still be clearing the table)
            in_phase ^= 1;
            for (;;) {
                if (!have_claim) {
                    uint32_t t = 0;
                    if (lane == 0) t = atomicAdd(&ctl->claim, 1u);
                    my_seq = __shfl_sync(kFull, t, 0);
                    have_claim = true;
                }
                const uint32_t si = my_seq % kRing, ph = (my_seq / kRing) & 1u;
                bool got = true;
                // (mbarrier.try_wait's hardware suspend ends at every barrier event in the CTA, a few dozen ns apart here, so the
                // waiting loops are a quarter of the instructions issued -- but replacing them with timed sleeps gained
                // nothing (r2_29: 115.9 vs 116.3 GB/s): the issue slots they take are not the ones the parsers lack.)
                while (!mbar_try_wait_hint(&ctl->full[si], ph, 1000u)) {
                    if (atomicAdd(const_cast<uint32_t *>(&ctl->block_end_seq), 0u) <= my_seq) {  // no such segment in this block: keep the claim
                        got = mbar_try_wait(&ctl->full[si], ph);
                        break;
                    }
                }
                if (!got) break;
                const SegSlot *slot = ring + si;
                const uint32_t sidx = slot->sidx;
                uint8_t *scr = scratch + (slot->seg_pos - base) + sidx * kSegPad;
                const SegRec r = parse_segment<kLinked>(in, slot, scr, base + L, lane, base);
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(&ctl->empty[si]);
                    recs[sidx] = r;
                }
                have_claim = false;
            }
        }
        __syncthreads();

        // ---------------------------------------------------------------- plan (warp 0)
        const uint32_t nseg = ctl->nseg;
        if (warp == 0) {
            // String the segments together: the literals a segment leaves behind its last match (or a whole segment without
            // a match) are carried into the next first sequence.  carry_out(s) = has_match(s) ? t(s) : carry_in(s) + t(s) is
            // a scan of (reset, add) pairs: every lane folds its kPlanPerLane consecutive segments, the lanes are scanned with
            // shuffles, then every lane replays its segments with the true carry and sizes them; a second scan places them.
            constexpr uint32_t kPlanPerLane = (kMaxSegs + 31) / 32;
            uint32_t csize = 0;
            {
                const uint32_t s0 = lane * kPlanPerLane;
                uint32_t has = 0, val = 0;  // this lane's segments as one function of the incoming carry
                for (uint32_t k = 0; k < kPlanPerLane; k++) {
                    const uint32_t sg = s0 + k;
                    if (sg < nseg) {
                        const SegRec r = recs[sg];
                        const uint32_t t = r.off_t >> 16;
                        if (r.lead_ml >> 16) { has = 1; val = t; } else val += t;
                    }
                }
                uint32_t ihas = has, ival = val;  // inclusive scan of the composition (earlier lanes first)
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t ph_ = __shfl_up_sync(kFull, ihas, d), pv = __shfl_up_sync(kFull, ival, d);
                    if ((int)lane >= d && !ihas) { ihas = ph_; ival += pv; }
                }
                uint32_t carry = __shfl_up_sync(kFull, ival, 1);  // what reaches this lane's first segment
                if (lane == 0) carry = 0;
                const uint32_t carry_end = __shfl_sync(kFull, ival, 31);  // literals behind the block's last match
                uint32_t fll[kPlanPerLane], fsz[kPlanPerLane], msz[kPlanPerLane], mine_total = 0;
#pragma unroll
                for (uint32_t k = 0; k < kPlanPerLane; k++) {
                    const uint32_t sg = s0 + k;
                    fll[k] = fsz[k] = msz[k] = 0;
                    if (sg < nseg) {
                        const SegRec r = recs[sg];
                        const uint32_t ml = r.lead_ml >> 16, t = r.off_t >> 16;
                        msz[k] = r.mbytes;
                        if (ml) {
                            fll[k] = carry + (r.lead_ml & 0xffffu);
                            fsz[k] = seq_bytes_fast(fll[k], ml);
                            carry = t;
                        } else carry += t;
                        mine_total += fsz[k] + msz[k];
                    }
                }
                uint32_t incl = mine_total;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t t = __shfl_up_sync(kFull, incl, d);
                    if ((int)lane >= d) incl += t;
                }
                uint32_t o = incl - mine_total;
                const uint32_t total = __shfl_sync(kFull, incl, 31);
#pragma unroll
                for (uint32_t k = 0; k < kPlanPerLane; k++) {
                    const uint32_t sg = s0 + k;
                    if (sg < nseg) {
                        SegPlan pl;
                        pl.foff = o;
                        pl.moff = o + fsz[k];
                        pl.fll = fll[k];
                        pl.pad = 0;
                        plans[sg] = pl;
                        o += fsz[k] + msz[k];
                    }
                }
                const uint32_t last = nseg == 0 ? L : carry_end;
                if (lane == 0) {
                    ctl->last_lits = last;
                    ctl->tail_off = total;  // where the final literal run starts (relative to the block's first data byte)
                }
                csize = total + 1 + last + (last >= 15 ? (last - 15) / 255 + 1 : 0);
            }
            const bool raw = csize > L - 1;  // LZ4F_makeBlock: a block that does not shrink is stored
            // OFF chain: learn where this block starts, tell the successor at once
            uint64_t st = 0;
            if (lane == 0) {
                uint64_t *cw = p.chain + dsc->c;
                unsigned ns = 128;
                while (((st = ld_acquire(cw)) >> kOffBits) != dsc->j) {
                    __nanosleep(ns);
                    if (ns < 2048) ns <<= 1;
                }
                const uint64_t off = st & kOffMask;
                const uint32_t bsize = raw ? L : csize;
                const uint64_t end = off + 4 + bsize;
                if (!dsc->last) st_release(p.chain + dsc->c, ((uint64_t)(dsc->j + 1) << kOffBits) | end);
                uint8_t *hdr = dsc->dst + off;
                const uint32_t hword = raw ? (L | 0x80000000u) : csize;
                hdr[0] = (uint8_t)hword; hdr[1] = (uint8_t)(hword >> 8); hdr[2] = (uint8_t)(hword >> 16); hdr[3] = (uint8_t)(hword >> 24);
                if (dsc->last) {
                    uint8_t *e = dsc->dst + end;
                    e[0] = e[1] = e[2] = e[3] = 0;  // EndMark
                    p.out_len[dsc->c] = end + 4;
                }
                ctl->csize = csize;
                ctl->raw = raw;
                const uint64_t data = off + 4;
                ctl->data_hi = (uint32_t)(data >> 32);
                ctl->data_lo = (uint32_t)data;
            }
        }
        __syncthreads();

        // ---------------------------------------------------------------- write the block to its final place (all warps)
        {
            uint8_t *out = dsc->dst + (((uint64_t)ctl->data_hi << 32) | ctl->data_lo);
            if (ctl->raw) {
                // stored block: straight from the input (L2-hot: the bulk load just pulled it), 16-byte-aligned slices per warp
                const uint32_t per = (((L + kWarps - 1) / kWarps) + 15u) & ~15u;
                const uint32_t lo = warp * per;
                if (lo < L) warp_copy_stream<true>(out + lo, src + lo, min(per, L - lo), lane);
            } else {
                for (uint32_t s = warp; s < nseg; s += kWarps) {
                    const SegRec r = recs[s];
                    const SegPlan pl = plans[s];
                    const uint32_t ml = r.lead_ml >> 16;
                    if (ml) {
                        const uint32_t lit_start = r.seg_pos + (r.lead_ml & 0xffffu) - pl.fll;
                        emit_seq(out, pl.foff, src, lit_start, pl.fll, ml, r.off_t & 0xffffu, lane);
                    }
                    if (r.mbytes) warp_copy_stream<false>(out + pl.moff, scratch + r.seg_pos + s * kSegPad, r.mbytes, lane);
                }
                if (warp == kWarps - 1) {
                    const uint32_t ll = ctl->last_lits;
                    emit_seq(out, ctl->tail_off, src, L - ll, ll, 0, 0, lane);
                }
            }
        }
    }
}

__global__ void __launch_bounds__(kThreads, 2) sky_fused_kernel(const Params p) { fused_body<false>(p); }
__global__ void __launch_bounds__(kThreads, 2) sky_fused_linked_kernel(const Params p) { fused_body<true>(p); }


// ------------------------------------------------------------------------------------ receiver side
struct DecParams {
    DecChunk *chunks;
    DecBlock *blocks;
    int32_t *status;     // per chunk, 0 = ok (mapped host memory)
    uint32_t *done;      // per chunk: leading blocks fully decoded (linked frames wait on it)
    uint32_t *counter;   // work counter
    uint32_t *blk_done;  // per block: 1 once decoded (gates the MD5 lanes)
    const uint32_t *md5_order;
    uint8_t *md5_out;    // null = no digest
    uint32_t n_chunks;
    uint32_t n_groups;
    uint32_t rows;
};

__global__ void sky_frame_index_kernel(const DecParams p) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.n_chunks) return;
    DecChunk cd = p.chunks[c];
    int32_t st = kDecOk;
    frame_index(cd, p.blocks + cd.blk_base, &st);
    p.chunks[c].linked = cd.linked;
    p.status[c] = st;
}

// Gate for the MD5 lanes of the receiver: row `row` of a chunk may be hashed once its block has been decoded.
struct DecRowGate {
    const uint32_t *flags;  // this lane's chunk: one word per block, non-zero = decoded (or failed: hash garbage, status says so)
    __device__ __forceinline__ void operator()(uint64_t row, bool wants) const {
        unsigned ns = 128;
        for (;;) {
            const bool ready = !wants || ld_acquire32(flags + row) != 0;
            if (__all_sync(kFull, ready)) break;
            __nanosleep(ns);
            if (ns < 4096) ns <<= 1;
        }
    }
};

// Persistent: warps 0..3 of a CTA may host an MD5 group (digest of the decoded bytes, following the decode through
// per-block flags); every other warp (and MD5 warps once their groups are done) decodes blocks.
__global__ void __launch_bounds__(512, 1) sky_decode_kernel(const DecParams p) {
    extern __shared__ __align__(128) uint8_t smem[];
    const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (p.md5_out && warp < kMd5WarpsPerCta) {
        const uint32_t md5_slots = gridDim.x * kMd5WarpsPerCta;
        for (uint32_t g = warp * gridDim.x + blockIdx.x; g < p.n_groups; g += md5_slots) {
            const uint32_t c = p.md5_order[g * 32 + lane];
            const bool active = c != 0xffffffffu;
            const uint8_t *src = nullptr;
            uint64_t len = 0;
            DecRowGate gate{nullptr};
            if (active) {
                src = p.chunks[c].out;
                len = p.chunks[c].raw_len;
                gate.flags = p.blk_done + p.chunks[c].blk_base;
            }
            md5_warp(reinterpret_cast<uint32_t *>(smem + warp * kRingBytes), src, len, active, p.md5_out + (size_t)(active ? c : 0) * 16,
                     lane, nullptr, gate);
            __syncwarp();
        }
    }
    const uint32_t total = p.rows * p.n_chunks;
    for (;;) {
        uint32_t w = 0;
        if (lane == 0) w = atomicAdd(p.counter, 1u);
        w = __shfl_sync(kFull, w, 0);
        if (w >= total) break;
        const uint32_t c = w % p.n_chunks, j = w / p.n_chunks;
        const DecChunk cd = p.chunks[c];
        if (j >= cd.nblk) continue;
        int32_t st = *reinterpret_cast<volatile int32_t *>(p.status + c);
        const uint64_t pos = (uint64_t)j * kBlock;
        const uint32_t want = (uint32_t)min((uint64_t)kBlock, cd.raw_len - pos);
        if (cd.linked) {  // matches may reach into earlier blocks: decode in order within the chunk
            if (lane == 0) {
                unsigned ns = 64;
                while (ld_acquire32(p.done + c) < j) {
                    __nanosleep(ns);
                    if (ns < 2048) ns <<= 1;
                }
            }
            __syncwarp();
            st = *reinterpret_cast<volatile int32_t *>(p.status + c);
        }
        if (st == kDecOk) {
            const DecBlock b = p.blocks[cd.blk_base + j];
            const uint32_t sz = b.word & 0x7FFFFFFFu;
            if (b.word & 0x80000000u) {
                if (sz != want) st = kDecLayout;
                else warp_copy(cd.out + pos, cd.frame + b.off, sz, lane);
            } else {
                st = lz4_decode_block(cd.frame + b.off, sz, cd.out, pos, want, cd.linked ? 0 : pos, lane);
            }
            if (st != kDecOk && lane == 0) atomicMin(p.status + c, st);
        }
        __syncwarp();
        if (lane == 0) {
            __threadfence();
            if (cd.linked) st_release32(p.done + c, j + 1);
            st_release32(p.blk_done + cd.blk_base + j, 1u);  // lets the MD5 lane of this chunk enter the row
        }
    }
}

// ---- E2EE glue: describe one box per chunk once the frame lengths exist (they are only known on the device).
// Box i of a batch sits in the box slab at the offset of chunk i's frame in the frame slab + 64*i + 8: the box is 40 bytes
// longer than its payload, and box + 40 (the ciphertext) is 16-byte aligned like the payload.
__host__ __device__ inline uint64_t box_offset(uint64_t frame_off, uint32_t i) { return frame_off + 64ull * i + 8; }

// Both setup kernels end here: blk_base[i] = the 64-byte stream blocks of the boxes before box i (block 0's second half
// covers message bytes [0, 32), hence len + 32), blk_base[n] = their total; sky_box_xor_kernel splits its work by it.
__device__ void box_block_prefix(const BoxChunk *bc, uint64_t *blk_base, uint32_t n) {
    __syncthreads();
    if (threadIdx.x == 0) {
        uint64_t acc = 0;
        for (uint32_t i = 0; i < n; i++) {
            blk_base[i] = acc;
            acc += (bc[i].len + 32 + 63) / 64;
        }
        blk_base[n] = acc;
    }
}

// seal: msg = the chunk's frame (or, without LZ4, its raw bytes); the nonce is copied in, out_len becomes the box length.
__global__ void sky_box_setup_kernel(BoxChunk *bc, uint64_t *blk_base, const ChunkDesc *desc, uint32_t n, uint64_t *out_len,
                                     const uint8_t *frame_slab, uint8_t *box_slab, const uint8_t *nonces, int use_frames) {
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
        const ChunkDesc d = desc[i];
        BoxChunk b;
        b.box = box_slab + box_offset(d.dst - frame_slab, i);
        b.msg = use_frames ? d.dst : d.src;
        b.len = use_frames ? out_len[i] : d.len;
        for (int k = 0; k < 24; k++) b.box[k] = nonces[24ull * i + k];
        bc[i] = b;
        out_len[i] = b.len + kBoxOverhead;
    }
    box_block_prefix(bc, blk_base, n);
}
// open: the boxes were copied into box_slab; the plaintext frame goes to frame_slab + frame_off[i].
__global__ void sky_box_open_setup_kernel(BoxChunk *bc, uint64_t *blk_base, uint32_t n, const uint64_t *box_len,
                                          const uint64_t *frame_off, uint8_t *frame_slab, uint8_t *box_slab) {
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
        BoxChunk b;
        b.box = box_slab + box_offset(frame_off[i], i);
        b.msg = frame_slab + frame_off[i];
        b.len = box_len[i] >= (uint64_t)kBoxOverhead ? box_len[i] - kBoxOverhead : 0;
        bc[i] = b;
    }
    box_block_prefix(bc, blk_base, n);
}

}  // namespace sky

// ======================================================================================= host side
using namespace sky;

// One allocation that frees itself: device or pinned host memory, an event or a stream.  Every allocation a slot or the
// ctx makes is held by one of these members, so a half-built ctx is torn down by the same destructors as a finished one.
// put() frees what the handle held and gives the allocating call the pointer to fill.
template <class T, cudaError_t (*Free)(void *)>
struct Owned {
    T *p = nullptr;
    Owned() = default;
    Owned(Owned &&o) noexcept : p(o.p) { o.p = nullptr; }
    ~Owned() { reset(); }
    void reset() { if (p) Free(p); p = nullptr; }
    T **put() { reset(); return &p; }
    operator T *() const { return p; }
};
inline cudaError_t destroy_event(void *e) { return cudaEventDestroy(static_cast<cudaEvent_t>(e)); }
inline cudaError_t destroy_stream(void *s) { return cudaStreamDestroy(static_cast<cudaStream_t>(s)); }
template <class T> using Dev = Owned<T, cudaFree>;
template <class T> using Pinned = Owned<T, cudaFreeHost>;
using Event = Owned<CUevent_st, destroy_event>;
using Stream = Owned<CUstream_st, destroy_stream>;

struct Slot {
    Stream stream;
    Dev<uint8_t> d_in, d_out;  // host path (n_slots > 0): input slab, frame slab
    Event ev_k0, ev_k1;        // start / end of the slot's kernels (kernel_ms): the fused kernel, or frame index + decode
    Event ev_res;              // results (sizes + digests) are on the host
    Event ev_h2d, ev_d2h;      // input landed (on ctx->st_h2d) / frames landed (on ctx->st_d2h)
    Event ev_h0, ev_d0, ev_d1; // SKYCHUNK_TRACE only: H2D start, D2H start / end
    bool d2h_issued = false;
    // per-batch metadata (pinned host mirrors + device arrays)
    Pinned<ChunkDesc> h_desc; Dev<ChunkDesc> d_desc;
    Pinned<uint32_t> h_order; Dev<uint32_t> d_order;
    Pinned<uint64_t> h_chain; Dev<uint64_t> d_chain;
    Dev<uint32_t> d_progress;
    // results live in MAPPED pinned host memory: the kernel stores sizes / digests straight over PCIe, so no small
    // device->host copies sit in a copy-engine queue behind multi-GiB frame copies
    Pinned<uint64_t> h_outlen; uint64_t *d_outlen = nullptr;  // same allocation, host / device view
    Pinned<uint8_t> h_md5; uint8_t *d_md5 = nullptr;
    Dev<uint32_t> d_counters;
    Dev<uint8_t> d_scratch;  // compress scratch: kScratchBytes per CTA of the grid (kernels of different slots overlap)
    // receiver side
    Pinned<DecChunk> h_dchunks; Dev<DecChunk> d_dchunks;
    Dev<DecBlock> d_dblocks;      // block table, dblocks_cap entries
    Dev<uint32_t> d_block_flags;  // per block: 1 once decoded (gates the MD5 lanes), dblocks_cap entries
    uint64_t dblocks_cap = 0;
    Dev<uint32_t> d_blocks_done;  // per chunk: leading blocks decoded (linked frames decode in order)
    Pinned<int32_t> h_dstatus; Dev<int32_t> d_dstatus;
    // E2EE (allocated when a key is set): box slab, per-chunk box descriptors, stream-block prefix, subkeys, nonces
    Dev<uint8_t> d_box;
    Dev<BoxChunk> d_bchunks;
    Dev<uint64_t> d_blkbase;
    Dev<uint32_t> d_sub;
    Pinned<uint8_t> h_nonce; Dev<uint8_t> d_nonce;
    Pinned<uint64_t> h_boxmeta; Dev<uint64_t> d_boxmeta;  // open side: box_len | frame_off (2 x n)
    Pinned<int32_t> h_bstatus; Dev<int32_t> d_bstatus;
    uint32_t flags = 0;
    // in-flight ticket
    bool busy = false;
    uint64_t ticket = 0;
    uint32_t n = 0;
    std::vector<void *> dst;
    std::vector<uint64_t> out_off;
};

struct sky_ctx {
    int device = 0;
    int sm_count = 0;
    uint32_t max_chunks = 0;
    uint64_t in_cap = 0, out_cap = 0;
    std::vector<Slot> slots;  // slots[0] doubles as the metadata holder for sky_process_device
    uint64_t next_ticket = 1;
    uint64_t launches = 0;
    std::string err;  // sky_last_error
    // Host path: every slot's input copies go FIFO through one H2D stream and every frame copy through one D2H
    // stream, so the two directions use different copy engines and batch k's frames leave while batch k+1's
    // input arrives (per-slot streams put both directions of all slots into one in-order engine queue).
    Stream st_h2d, st_d2h;
    Dev<uint8_t> d_key;  // 32-byte SecretBox key (null: E2EE off)
    bool trace = false;  // SKYCHUNK_TRACE=1: print per-batch device timeline to stderr
    Event ev_base;
    // a copy on the shared streams may still read a slot's slabs: wait for all of them before the members free themselves
    ~sky_ctx() {
        cudaSetDevice(device);
        for (auto &s : slots)
            if (s.stream) cudaStreamSynchronize(s.stream);
        if (st_h2d) cudaStreamSynchronize(st_h2d);
        if (st_d2h) cudaStreamSynchronize(st_d2h);
    }
};

static thread_local std::string g_err;  // sky_last_error(NULL)

// Every failing return of an entry point goes through here: the detail goes to the ctx, or to the calling thread when
// there is none, so sky_last_error always describes the latest failure.
__attribute__((format(printf, 3, 4))) static int fail(sky_ctx *ctx, int rc, const char *fmt, ...) {
    char b[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(b, sizeof b, fmt, ap);
    va_end(ap);
    (ctx ? ctx->err : g_err) = b;
    return rc;
}

#define CK(ctx, call)                                                                                                   \
    do {                                                                                                                \
        const cudaError_t e_ = (call);                                                                                  \
        if (e_ != cudaSuccess) return fail(ctx, SKY_E_CUDA, "%s -> %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

static uint64_t round16(uint64_t x) { return (x + 15) & ~15ull; }

// Offsets of n regions of len(i) bytes packed back to back into a slab, each at a 16-byte aligned offset; end = bytes used.
template <class Len>
static std::vector<uint64_t> pack16(uint32_t n, Len len, uint64_t &end) {
    std::vector<uint64_t> off(n);
    end = 0;
    for (uint32_t i = 0; i < n; i++) {
        off[i] = end;
        end += round16(len(i));
    }
    return off;
}

// Stage flags 0 mean LZ4 + MD5.
static uint32_t with_default_stages(uint32_t flags) {
    return (flags & (SKY_F_LZ4 | SKY_F_MD5)) ? flags : flags | SKY_F_LZ4 | SKY_F_MD5;
}

static uint64_t nblocks(uint64_t len) { return (len + kBlock - 1) / kBlock; }
// 64 KiB block rows of a batch: max(1, blocks of its longest chunk).  The kernels hold a block index in 24 bits (the
// fused kernel's OFF word) and number their work items (rows x n) in 32.
static int block_rows(sky_ctx *ctx, uint32_t n, const uint64_t *len, uint32_t *rows) {
    uint64_t r = 1;
    for (uint32_t i = 0; i < n; i++) r = std::max(r, nblocks(len[i]));
    if (r >= (1ull << 24) || r * n >= 0xffffffffull)
        return fail(ctx, SKY_E_CAPACITY, "%" PRIu64 " block rows x %u chunks exceed the kernels' block and work counters", r, n);
    *rows = (uint32_t)r;
    return SKY_OK;
}

// MD5 lane assignment: chunk indices, longest chunk first so a warp's 32 lanes carry similar lengths, padded with
// 0xffffffff to whole groups of 32.  Returns the number of groups.
static uint32_t md5_lane_order(uint32_t *order, uint32_t n, const uint64_t *len) {
    const uint32_t ng = (n + 31) / 32;
    std::iota(order, order + n, 0u);
    std::stable_sort(order, order + n, [&](uint32_t a, uint32_t b) { return len[a] > len[b]; });
    std::fill(order + n, order + ng * 32, 0xffffffffu);
    return ng;
}

extern "C" {

const char *sky_strerror(int code) {
    switch (code) {
    case SKY_OK: return "ok";
    case SKY_E_INVALID: return "invalid argument";
    case SKY_E_NOGPU: return "no CUDA device available (this library has no CPU fallback)";
    case SKY_E_CUDA: return "CUDA error";
    case SKY_E_CAPACITY: return "capacity exceeded";
    case SKY_E_BUSY: return "all slots busy";
    case SKY_E_TICKET: return "unknown ticket";
    case SKY_E_NOMEM: return "out of memory";
    case SKY_E_NOKEY: return "SKY_F_E2EE without a key (sky_set_e2ee_key) or without nonces";
    default: return "unknown error";
    }
}

const char *sky_last_error(const sky_ctx *ctx) { return ctx ? ctx->err.c_str() : g_err.c_str(); }
int sky_abi_version(void) { return SKY_ABI_VERSION; }

int sky_device_count(int *count) {
    if (!count) return fail(nullptr, SKY_E_INVALID, "count is NULL");
    int n = 0;
    const cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        *count = 0;
        return fail(nullptr, SKY_E_NOGPU, "cudaGetDeviceCount -> %s", cudaGetErrorString(e));
    }
    *count = n;
    return SKY_OK;
}

int sky_device_pci_bus_id(int device, char *buf, int len) {
    if (!buf || len < 16) return fail(nullptr, SKY_E_INVALID, "buf is NULL or len < 16");
    const cudaError_t e = cudaDeviceGetPCIBusId(buf, len, device);
    if (e != cudaSuccess) return fail(nullptr, e == cudaErrorInvalidDevice ? SKY_E_INVALID : SKY_E_NOGPU, "%s", cudaGetErrorString(e));
    return SKY_OK;
}

uint32_t sky_kernel_config(int what) {
    switch (what) {
    case 0: return kEntries;
    case 1: return (uint32_t)kWarps;
    case 2: return kSegSlots;
    case 3: return kMaxStepLog;
    case 4: return kLinkedWindow;
    case 5: return kLinkedSeedLog;
    case 6: return kEntries;  // the linked kernel keeps the default table
    default: return 0;
    }
}

uint64_t sky_frame_bound(uint64_t n) {
    if (n == 0) return 11;
    return 15 + n + 4 * ((n + kBlock - 1) / kBlock) + 4;
}

// Everything a slot needs for any batch: metadata, results, decode arrays, stream and events (+ the slabs on the host path).
static int alloc_slot(sky_ctx *ctx, Slot &s, bool slabs) {
    const size_t nc = ctx->max_chunks, ng = (nc + 31) / 32 * 32;
    CK(ctx, cudaMallocHost(s.h_desc.put(), nc * sizeof(ChunkDesc)));
    CK(ctx, cudaMallocHost(s.h_order.put(), ng * sizeof(uint32_t)));
    CK(ctx, cudaMallocHost(s.h_chain.put(), nc * sizeof(uint64_t)));
    CK(ctx, cudaHostAlloc(s.h_outlen.put(), nc * sizeof(uint64_t), cudaHostAllocMapped | cudaHostAllocPortable));
    CK(ctx, cudaHostAlloc(s.h_md5.put(), nc * 16, cudaHostAllocMapped | cudaHostAllocPortable));
    CK(ctx, cudaHostGetDevicePointer(&s.d_outlen, s.h_outlen, 0));
    CK(ctx, cudaHostGetDevicePointer(&s.d_md5, s.h_md5, 0));
    CK(ctx, cudaEventCreateWithFlags(s.ev_h2d.put(), cudaEventDisableTiming));
    CK(ctx, cudaEventCreateWithFlags(s.ev_d2h.put(), cudaEventDisableTiming));
    CK(ctx, cudaMalloc(s.d_desc.put(), nc * sizeof(ChunkDesc)));
    CK(ctx, cudaMalloc(s.d_order.put(), ng * sizeof(uint32_t)));
    CK(ctx, cudaMalloc(s.d_chain.put(), nc * sizeof(uint64_t)));
    CK(ctx, cudaMalloc(s.d_counters.put(), 64));
    CK(ctx, cudaMalloc(s.d_scratch.put(), (size_t)ctx->sm_count * kCtasPerSm * kScratchBytes));
    CK(ctx, cudaMallocHost(s.h_dchunks.put(), nc * sizeof(DecChunk)));
    CK(ctx, cudaMalloc(s.d_dchunks.put(), nc * sizeof(DecChunk)));
    CK(ctx, cudaMallocHost(s.h_dstatus.put(), nc * sizeof(int32_t)));
    CK(ctx, cudaMalloc(s.d_dstatus.put(), nc * sizeof(int32_t)));
    CK(ctx, cudaMalloc(s.d_blocks_done.put(), nc * sizeof(uint32_t)));
    CK(ctx, cudaMalloc(s.d_progress.put(), (ng / 32 + 1) * sizeof(uint32_t)));
    CK(ctx, cudaStreamCreateWithFlags(s.stream.put(), cudaStreamNonBlocking));
    CK(ctx, cudaEventCreate(s.ev_k0.put()));
    CK(ctx, cudaEventCreate(s.ev_k1.put()));
    CK(ctx, cudaEventCreate(s.ev_res.put()));
    CK(ctx, cudaEventCreate(s.ev_h0.put()));
    CK(ctx, cudaEventCreate(s.ev_d0.put()));
    CK(ctx, cudaEventCreate(s.ev_d1.put()));
    if (slabs) {
        cudaError_t e = cudaMalloc(s.d_in.put(), ctx->in_cap);
        if (e == cudaSuccess) e = cudaMalloc(s.d_out.put(), ctx->out_cap);
        if (e != cudaSuccess) return fail(ctx, SKY_E_NOMEM, "cudaMalloc(slab) -> %s", cudaGetErrorString(e));
    }
    return SKY_OK;
}

static int init_ctx(sky_ctx *ctx, uint64_t max_batch_bytes, uint32_t n_slots) {
    CK(ctx, cudaSetDevice(ctx->device));
    cudaDeviceProp prop;
    CK(ctx, cudaGetDeviceProperties(&prop, ctx->device));
    ctx->sm_count = prop.multiProcessorCount;
    cudaError_t e = cudaFuncSetAttribute(sky_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(sky_fused_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(sky_fused_linked_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLinkedSmemBytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(sky_fused_linked_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (e != cudaSuccess) return fail(ctx, SKY_E_CUDA, "cudaFuncSetAttribute(smem) -> %s (built for sm_100a only)", cudaGetErrorString(e));
    // every chunk is placed at a 16-byte aligned offset; frames need bound(len) each
    const uint64_t max_chunks = ctx->max_chunks;
    ctx->in_cap = round16(max_batch_bytes) + 16 * max_chunks + 256;
    ctx->out_cap = max_batch_bytes + max_chunks * (64 + 4 * 2) + 4 * (max_batch_bytes / kBlock + 1) + 256;
    ctx->slots.resize(n_slots ? n_slots : 1);
    for (auto &s : ctx->slots)
        if (int rc = alloc_slot(ctx, s, n_slots != 0)) return rc;
    if (n_slots) {
        CK(ctx, cudaStreamCreateWithFlags(ctx->st_h2d.put(), cudaStreamNonBlocking));
        CK(ctx, cudaStreamCreateWithFlags(ctx->st_d2h.put(), cudaStreamNonBlocking));
    }
    ctx->trace = getenv("SKYCHUNK_TRACE") != nullptr;
    if (ctx->trace) {
        CK(ctx, cudaEventCreate(ctx->ev_base.put()));
        CK(ctx, cudaEventRecord(ctx->ev_base, ctx->slots[0].stream));
    }
    return SKY_OK;
}

int sky_ctx_create(int device, uint64_t max_batch_bytes, uint32_t max_chunks, uint32_t n_slots, sky_ctx **out) {
    if (!out || max_chunks == 0) return fail(nullptr, SKY_E_INVALID, "out is NULL or max_chunks == 0");
    *out = nullptr;
    int ndev = 0;
    if (int rc = sky_device_count(&ndev)) return rc;
    if (device < 0 || device >= ndev) return fail(nullptr, SKY_E_INVALID, "device %d of %d", device, ndev);
    sky_ctx *ctx = new (std::nothrow) sky_ctx();
    if (!ctx) return fail(nullptr, SKY_E_NOMEM, "new sky_ctx");
    ctx->device = device;
    ctx->max_chunks = max_chunks;
    if (int rc = init_ctx(ctx, max_batch_bytes, n_slots)) {
        g_err = ctx->err;  // this ctx is never handed out
        delete ctx;
        return rc;
    }
    *out = ctx;
    return SKY_OK;
}

int sky_ctx_destroy(sky_ctx *ctx) {
    if (!ctx) return fail(ctx, SKY_E_INVALID, "ctx is NULL");
    delete ctx;
    return SKY_OK;
}

void *sky_pinned_alloc(uint64_t bytes) {
    void *p = nullptr;
    const cudaError_t e = cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable);
    if (e == cudaSuccess) return p;
    fail(nullptr, SKY_E_NOMEM, "cudaHostAlloc(%" PRIu64 ") -> %s", bytes, cudaGetErrorString(e));
    return nullptr;
}
int sky_pinned_free(void *p) {
    if (p) CK(nullptr, cudaFreeHost(p));
    return SKY_OK;
}

uint64_t sky_box_bound(uint64_t n) { return sky_frame_bound(n) + kBoxOverhead; }

// E2EE arrays of a slot, made once (d_box last: a partly failed earlier attempt is made again).
static int alloc_box(sky_ctx *ctx, Slot &s) {
    if (s.d_box) return SKY_OK;
    const size_t nc = ctx->max_chunks;
    CK(ctx, cudaMalloc(s.d_bchunks.put(), nc * sizeof(BoxChunk)));
    CK(ctx, cudaMalloc(s.d_blkbase.put(), (nc + 1) * sizeof(uint64_t)));
    CK(ctx, cudaMalloc(s.d_sub.put(), nc * 16 * sizeof(uint32_t)));
    CK(ctx, cudaMalloc(s.d_nonce.put(), nc * 24));
    CK(ctx, cudaMallocHost(s.h_nonce.put(), nc * 24));
    CK(ctx, cudaMalloc(s.d_boxmeta.put(), 2 * nc * sizeof(uint64_t)));
    CK(ctx, cudaMallocHost(s.h_boxmeta.put(), 2 * nc * sizeof(uint64_t)));
    CK(ctx, cudaMalloc(s.d_bstatus.put(), nc * sizeof(int32_t)));
    CK(ctx, cudaMallocHost(s.h_bstatus.put(), nc * sizeof(int32_t)));
    CK(ctx, cudaMalloc(s.d_box.put(), ctx->out_cap + 64 * nc + 256));
    return SKY_OK;
}

int sky_set_e2ee_key(sky_ctx *ctx, const uint8_t *key32) {
    if (!ctx) return fail(ctx, SKY_E_INVALID, "ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    if (!key32) {
        ctx->d_key.reset();
        return SKY_OK;
    }
    if (!ctx->d_key) CK(ctx, cudaMalloc(ctx->d_key.put(), 32));
    CK(ctx, cudaMemcpy(ctx->d_key, key32, 32, cudaMemcpyHostToDevice));
    for (auto &s : ctx->slots)
        if (int rc = alloc_box(ctx, s)) return rc;
    return SKY_OK;
}

// Seal the batch's frames (or raw chunks) on `st` after the fused kernel: setup -> keys -> xor -> tag.
static int launch_seal(sky_ctx *ctx, Slot &s, cudaStream_t st, uint32_t n, uint8_t *d_dst, uint32_t flags) {
    const int use_frames = (flags & SKY_F_LZ4) ? 1 : 0;
    sky_box_setup_kernel<<<1, 256, 0, st>>>(s.d_bchunks, s.d_blkbase, s.d_desc, n, s.d_outlen, d_dst, s.d_box, s.d_nonce, use_frames);
    CK(ctx, cudaGetLastError());
    sky_box_keys_kernel<<<(n + 63) / 64, 64, 0, st>>>(s.d_bchunks, n, ctx->d_key, s.d_sub);
    CK(ctx, cudaGetLastError());
    sky_box_xor_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(s.d_bchunks, s.d_blkbase, n, s.d_sub, 0);
    CK(ctx, cudaGetLastError());
    sky_box_tag_kernel<<<n, kPolyThreads, 0, st>>>(s.d_bchunks, s.d_sub, 0, nullptr);
    CK(ctx, cudaGetLastError());
    ctx->launches += 4;
    return SKY_OK;
}

// Fills the slot's metadata for a batch and enqueues: meta H2D, counter reset, fused kernel, results D2H.
// `meta_st`: stream the three small metadata copies ride on (the H2D stream on the host path, so they are
// never queued behind another batch's frame copies); `st`: the stream the kernel runs on.
static int launch_batch(sky_ctx *ctx, Slot &s, cudaStream_t st, cudaStream_t meta_st, uint32_t n, const uint8_t *d_src,
                        const uint64_t *src_off, const uint64_t *src_len, uint8_t *d_dst, const uint64_t *dst_off, uint32_t flags) {
    uint32_t rows;
    if (int rc = block_rows(ctx, n, src_len, &rows)) return rc;
    for (uint32_t i = 0; i < n; i++) {
        ChunkDesc &d = s.h_desc[i];
        d.src = d_src + src_off[i];
        d.dst = d_dst + dst_off[i];
        d.len = src_len[i];
        d.nblk = (uint32_t)nblocks(src_len[i]);
        s.h_chain[i] = 15;  // block 0 starts right after the 15-byte frame header
    }
    const uint32_t ng = md5_lane_order(s.h_order, n, src_len);
    for (uint32_t i = 0; i < n; i++) s.h_desc[s.h_order[i]].group = i / 32;

    CK(ctx, cudaMemcpyAsync(s.d_desc, s.h_desc, n * sizeof(ChunkDesc), cudaMemcpyHostToDevice, meta_st));
    CK(ctx, cudaMemcpyAsync(s.d_order, s.h_order, ng * 32 * sizeof(uint32_t), cudaMemcpyHostToDevice, meta_st));
    CK(ctx, cudaMemcpyAsync(s.d_chain, s.h_chain, n * sizeof(uint64_t), cudaMemcpyHostToDevice, meta_st));
    if (meta_st != st) {
        CK(ctx, cudaEventRecord(s.ev_h2d, meta_st));  // input (enqueued earlier on meta_st) + metadata have landed
        CK(ctx, cudaStreamWaitEvent(st, s.ev_h2d, 0));
    }
    CK(ctx, cudaMemsetAsync(s.d_counters, 0, 64, st));
    CK(ctx, cudaMemsetAsync(s.d_progress, 0, (ng + 1) * sizeof(uint32_t), st));
    memset(s.h_outlen, 0, n * sizeof(uint64_t));  // host-side clear (mapped memory; the slot is idle here)
    memset(s.h_md5, 0, (size_t)n * 16);

    Params p;
    p.chunks = s.d_desc;
    p.md5_order = s.d_order;
    p.chain = s.d_chain;
    p.md5_progress = s.d_progress;
    p.out_len = s.d_outlen;
    p.md5_out = s.d_md5;
    p.counters = s.d_counters;
    p.scratch = s.d_scratch;
    p.n_chunks = n;
    p.n_groups = ng;
    const uint32_t grid = (uint32_t)ctx->sm_count * kCtasPerSm;
    // digest CTAs: 4 groups (one per SM sub-partition) each; with few groups spread them one per CTA first.  (Tried in
    // r2_30 / r2_31: whole digest SMs -- 4 or 8 MD5 warps on a few SMs, nothing else there -- so that fewer block buffers
    // sit idle.  With 8 or 16 MiB chunks the MD5 warps then ran at half their chain rate (0.061 GB/s per chunk; with 1 MiB
    // chunks at the full 0.118), so the spread-out arrangement stays.)
    {
        // MD5 warps per digest CTA while the groups are few: 1 = one warp in each of up to sm_count / 4 CTAs (default);
        // SKYCHUNK_MD5_WARPS=2 packs two per CTA so that half as many block buffers sit idle in the fused kernel (tuning knob)
        static const uint32_t md5_warps = [] {
            const char *e = getenv("SKYCHUNK_MD5_WARPS");
            const int v = e ? atoi(e) : 1;
            return (uint32_t)(v >= 1 && v <= kMd5WarpsPerCta ? v : 1);
        }();
        p.n_md5_ctas = (flags & SKY_F_MD5) ? std::min(grid, std::max((ng + kMd5WarpsPerCta - 1) / kMd5WarpsPerCta,
                                                                     std::min((ng + md5_warps - 1) / md5_warps, (uint32_t)ctx->sm_count / 4))) : 0;
    }
    p.rows = rows;
    p.flags = flags;
    CK(ctx, cudaEventRecord(s.ev_k0, st));
    if ((flags & SKY_F_LINKED) && (flags & SKY_F_LZ4)) sky_fused_linked_kernel<<<grid, kThreads, kLinkedSmemBytes, st>>>(p);
    else sky_fused_kernel<<<grid, kThreads, kSmemBytes, st>>>(p);
    CK(ctx, cudaGetLastError());
    CK(ctx, cudaEventRecord(s.ev_k1, st));
    ctx->launches++;
    if (flags & SKY_F_E2EE)
        if (int rc = launch_seal(ctx, s, st, n, d_dst, flags)) return rc;
    CK(ctx, cudaEventRecord(s.ev_res, st));  // kernel(s) done => sizes + digests are in host memory
    return SKY_OK;
}

// Frame copies need the compressed sizes, which only exist after the kernel.  Every host-path entry point
// calls this: for each in-flight slot whose sizes have reached the host (ev_res done) it enqueues the exact-length
// D2H copies on the ctx's D2H stream, so batch k's D2H overlaps batch k+1's H2D and kernel without a helper thread.
static int issue_d2h(sky_ctx *ctx, Slot &s) {
    CK(ctx, cudaStreamWaitEvent(ctx->st_d2h, s.ev_res, 0));
    if (ctx->trace) CK(ctx, cudaEventRecord(s.ev_d0, ctx->st_d2h));
    for (uint32_t i = 0; i < s.n; i++) {
        if (s.h_outlen[i] == 0) continue;  // MD5-only batch without E2EE: nothing comes back but the digests
        const uint8_t *from = (s.flags & SKY_F_E2EE) ? s.d_box + box_offset(s.out_off[i], i) : s.d_out + s.out_off[i];
        CK(ctx, cudaMemcpyAsync(s.dst[i], from, s.h_outlen[i], cudaMemcpyDeviceToHost, ctx->st_d2h));
    }
    if (ctx->trace) CK(ctx, cudaEventRecord(s.ev_d1, ctx->st_d2h));
    CK(ctx, cudaEventRecord(s.ev_d2h, ctx->st_d2h));
    s.d2h_issued = true;
    return SKY_OK;
}
static int progress(sky_ctx *ctx) {
    for (auto &s : ctx->slots) {
        if (!s.busy || s.d2h_issued) continue;
        cudaError_t q = cudaEventQuery(s.ev_res);
        if (q == cudaErrorNotReady) continue;
        CK(ctx, q);
        if (int rc = issue_d2h(ctx, s)) return rc;
    }
    return SKY_OK;
}

int sky_process_device(sky_ctx *ctx, uint32_t n, const void *d_src, const uint64_t *src_off, const uint64_t *src_len,
                       void *d_dst, const uint64_t *dst_off, const uint64_t *dst_cap, uint32_t flags, void *stream,
                       uint64_t *out_len, uint8_t *md5, float *kernel_ms) {
    if (!ctx || n == 0 || !src_off || !src_len || !dst_off || !dst_cap || !d_dst) return fail(ctx, SKY_E_INVALID, "NULL argument or n == 0");
    if (flags & SKY_F_E2EE) return fail(ctx, SKY_E_INVALID, "SKY_F_E2EE is a host-path feature (sky_submit_flags)");
    if (n > ctx->max_chunks) return fail(ctx, SKY_E_CAPACITY, "n = %u > max_chunks = %u", n, ctx->max_chunks);
    if ((reinterpret_cast<uintptr_t>(d_src) & 15) || (reinterpret_cast<uintptr_t>(d_dst) & 15))
        return fail(ctx, SKY_E_INVALID, "d_src or d_dst is not 16-byte aligned");
    for (uint32_t i = 0; i < n; i++) {
        if ((src_off[i] & 15) || (dst_off[i] & 15)) return fail(ctx, SKY_E_INVALID, "src_off[%u] or dst_off[%u] is not a multiple of 16", i, i);
        if (dst_cap[i] < sky_frame_bound(src_len[i])) return fail(ctx, SKY_E_CAPACITY, "dst_cap[%u] < sky_frame_bound(src_len[%u])", i, i);
        if (src_len[i] && !d_src) return fail(ctx, SKY_E_INVALID, "d_src is NULL");
    }
    CK(ctx, cudaSetDevice(ctx->device));
    Slot &s = ctx->slots[0];
    if (s.busy) return fail(ctx, SKY_E_BUSY, "slot 0 holds a batch that was not waited for");
    cudaStream_t st = stream ? (cudaStream_t)stream : s.stream;
    flags = with_default_stages(flags);
    if (int rc = launch_batch(ctx, s, st, st, n, (const uint8_t *)d_src, src_off, src_len, (uint8_t *)d_dst, dst_off, flags)) return rc;
    CK(ctx, cudaStreamSynchronize(st));
    if (out_len) memcpy(out_len, s.h_outlen, n * sizeof(uint64_t));
    if (md5) memcpy(md5, s.h_md5, (size_t)n * 16);
    if (kernel_ms) CK(ctx, cudaEventElapsedTime(kernel_ms, s.ev_k0, s.ev_k1));
    return SKY_OK;
}

int sky_submit(sky_ctx *ctx, uint32_t n, const void *const *src, const uint64_t *src_len, void *const *dst,
               const uint64_t *dst_cap, uint64_t *ticket) {
    return sky_submit_flags(ctx, n, src, src_len, dst, dst_cap, 0, nullptr, ticket);
}

int sky_submit_flags(sky_ctx *ctx, uint32_t n, const void *const *src, const uint64_t *src_len, void *const *dst,
                     const uint64_t *dst_cap, uint32_t flags, const uint8_t *nonces, uint64_t *ticket) {
    if (!ctx || n == 0 || !src || !src_len || !ticket) return fail(ctx, SKY_E_INVALID, "NULL argument or n == 0");
    flags = with_default_stages(flags);
    const bool e2ee = (flags & SKY_F_E2EE) != 0, frames = (flags & SKY_F_LZ4) != 0;
    const bool returns_data = frames || e2ee;  // MD5-only without E2EE: only digests come back
    if (returns_data && (!dst || !dst_cap)) return fail(ctx, SKY_E_INVALID, "dst or dst_cap is NULL");
    if (e2ee && (!ctx->d_key || !nonces)) return fail(ctx, SKY_E_NOKEY, ctx->d_key ? "nonces is NULL" : "no key (sky_set_e2ee_key)");
    if (n > ctx->max_chunks) return fail(ctx, SKY_E_CAPACITY, "n = %u > max_chunks = %u", n, ctx->max_chunks);
    Slot *sp = nullptr;
    for (auto &s : ctx->slots)
        if (!s.busy && s.d_in) { sp = &s; break; }
    if (!sp)
        return ctx->slots[0].d_in ? fail(ctx, SKY_E_BUSY, "all %zu slots hold batches that were not waited for", ctx->slots.size())
                                  : fail(ctx, SKY_E_INVALID, "the ctx was created without slots (n_slots = 0)");
    Slot &s = *sp;
    CK(ctx, cudaSetDevice(ctx->device));
    if (int rc = progress(ctx)) return rc;
    for (uint32_t i = 0; i < n; i++) {
        if (src_len[i] && !src[i]) return fail(ctx, SKY_E_INVALID, "src[%u] is NULL", i);
        const uint64_t need = (frames ? sky_frame_bound(src_len[i]) : src_len[i]) + (e2ee ? kBoxOverhead : 0);
        if (returns_data && (!dst[i] || dst_cap[i] < need)) return fail(ctx, SKY_E_CAPACITY, "dst[%u] is NULL or dst_cap[%u] < %" PRIu64, i, i, need);
    }
    uint64_t in_end, out_end;
    std::vector<uint64_t> in_off = pack16(n, [&](uint32_t i) { return src_len[i]; }, in_end);
    std::vector<uint64_t> out_off = pack16(n, [&](uint32_t i) { return sky_frame_bound(src_len[i]); }, out_end);
    if (in_end > ctx->in_cap || out_end > ctx->out_cap) return fail(ctx, SKY_E_CAPACITY, "the batch exceeds a slot's input or frame slab");
    if (ctx->trace) CK(ctx, cudaEventRecord(s.ev_h0, ctx->st_h2d));
    for (uint32_t i = 0; i < n; i++)
        if (src_len[i]) CK(ctx, cudaMemcpyAsync(s.d_in + in_off[i], src[i], src_len[i], cudaMemcpyHostToDevice, ctx->st_h2d));

    // No MD5 pacing on the host path: paced LZ4 warps keep every CTA resident for the whole MD5 chain (tens of
    // ms), which would serialise the kernels of different slots; unpaced, a batch's LZ4 CTAs retire in a few ms
    // and the next slot's kernel overlaps this one's MD5 tail.
    if (e2ee) {
        memcpy(s.h_nonce, nonces, 24ull * n);
        CK(ctx, cudaMemcpyAsync(s.d_nonce, s.h_nonce, 24ull * n, cudaMemcpyHostToDevice, ctx->st_h2d));
    }
    s.flags = flags;
    if (int rc = launch_batch(ctx, s, s.stream, ctx->st_h2d, n, s.d_in, in_off.data(), src_len, s.d_out, out_off.data(), flags | SKY_F_NO_PACING))
        return rc;
    s.busy = true;
    s.d2h_issued = false;
    s.ticket = ctx->next_ticket++;
    s.n = n;
    if (returns_data) s.dst.assign(dst, dst + n); else s.dst.assign(n, nullptr);
    s.out_off.swap(out_off);
    *ticket = s.ticket;
    return SKY_OK;
}

int sky_wait(sky_ctx *ctx, uint64_t ticket, uint64_t *out_len, uint8_t *md5, float *kernel_ms) {
    if (!ctx) return fail(ctx, SKY_E_INVALID, "ctx is NULL");
    Slot *sp = nullptr;
    for (auto &s : ctx->slots)
        if (s.busy && s.ticket == ticket) { sp = &s; break; }
    if (!sp) return fail(ctx, SKY_E_TICKET, "ticket %" PRIu64 " is not in flight", ticket);
    Slot &s = *sp;
    CK(ctx, cudaSetDevice(ctx->device));
    if (int rc = progress(ctx)) return rc;
    if (!s.d2h_issued) {
        CK(ctx, cudaEventSynchronize(s.ev_res));  // sizes + digests are on the host now
        if (int rc = issue_d2h(ctx, s)) return rc;
    }
    if (int rc = progress(ctx)) return rc;  // let later batches' copies queue up behind ours
    CK(ctx, cudaEventSynchronize(s.ev_d2h));
    if (out_len) memcpy(out_len, s.h_outlen, s.n * sizeof(uint64_t));
    if (md5) memcpy(md5, s.h_md5, (size_t)s.n * 16);
    if (kernel_ms) CK(ctx, cudaEventElapsedTime(kernel_ms, s.ev_k0, s.ev_k1));
    if (ctx->trace) {
        float h0 = 0, k0 = 0, k1 = 0, rs = 0, d0 = 0, d1 = 0;
        cudaEventElapsedTime(&h0, ctx->ev_base, s.ev_h0);
        cudaEventElapsedTime(&k0, ctx->ev_base, s.ev_k0);
        cudaEventElapsedTime(&k1, ctx->ev_base, s.ev_k1);
        cudaEventElapsedTime(&rs, ctx->ev_base, s.ev_res);
        cudaEventElapsedTime(&d0, ctx->ev_base, s.ev_d0);
        cudaEventElapsedTime(&d1, ctx->ev_base, s.ev_d1);
        fprintf(stderr, "[skychunk trace] ticket %llu: h2d %.1f..%.1f kernel %.1f..%.1f results %.1f d2h %.1f..%.1f ms\n",
                (unsigned long long)s.ticket, h0, k0, k0, k1, rs, d0, d1);
    }
    s.busy = false;
    return SKY_OK;
}

int sky_device_alloc(sky_ctx *ctx, uint64_t bytes, void **dptr) {
    if (!ctx || !dptr) return fail(ctx, SKY_E_INVALID, "ctx or dptr is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    const cudaError_t e = cudaMalloc(dptr, bytes ? bytes : 16);
    if (e != cudaSuccess) return fail(ctx, SKY_E_NOMEM, "cudaMalloc(%" PRIu64 ") -> %s", bytes, cudaGetErrorString(e));
    return SKY_OK;
}
int sky_device_free(sky_ctx *ctx, void *dptr) {
    if (!ctx) return fail(ctx, SKY_E_INVALID, "ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaFree(dptr));
    return SKY_OK;
}
int sky_memcpy_h2d(sky_ctx *ctx, void *dptr, const void *host, uint64_t bytes) {
    if (!ctx) return fail(ctx, SKY_E_INVALID, "ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpy(dptr, host, bytes, cudaMemcpyHostToDevice));
    return SKY_OK;
}
int sky_memcpy_d2h(sky_ctx *ctx, void *host, const void *dptr, uint64_t bytes) {
    if (!ctx) return fail(ctx, SKY_E_INVALID, "ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpy(host, dptr, bytes, cudaMemcpyDeviceToHost));
    return SKY_OK;
}

// ---------------------------------------------------------------------------------- receiver side
// Enqueues index + decode (+ MD5 of the decoded bytes through the fused kernel's MD5 role) on `st`.
static int launch_decode(sky_ctx *ctx, Slot &s, cudaStream_t st, uint32_t n, const uint8_t *d_frames, const uint64_t *frame_off,
                         const uint64_t *frame_len, uint8_t *d_out, const uint64_t *out_off, const uint64_t *raw_len) {
    uint32_t rows;
    if (int rc = block_rows(ctx, n, raw_len, &rows)) return rc;
    uint64_t nblk_total = 0;
    for (uint32_t i = 0; i < n; i++) {
        DecChunk &d = s.h_dchunks[i];
        d.frame = d_frames + frame_off[i];
        d.out = d_out + out_off[i];
        d.frame_len = frame_len[i];
        d.raw_len = raw_len[i];
        d.nblk = (uint32_t)nblocks(raw_len[i]);
        d.blk_base = nblk_total;
        d.linked = 0;
        nblk_total += d.nblk;
    }
    if (nblk_total + 1 > s.dblocks_cap) {  // grow the block arrays (the previous decode on `st` may still use them)
        CK(ctx, cudaStreamSynchronize(st));
        s.dblocks_cap = 0;
        CK(ctx, cudaMalloc(s.d_dblocks.put(), (nblk_total + 1) * sizeof(DecBlock)));
        CK(ctx, cudaMalloc(s.d_block_flags.put(), (nblk_total + 1) * sizeof(uint32_t)));
        s.dblocks_cap = nblk_total + 1;
    }
    CK(ctx, cudaMemcpyAsync(s.d_dchunks, s.h_dchunks, n * sizeof(DecChunk), cudaMemcpyHostToDevice, st));
    CK(ctx, cudaMemsetAsync(s.d_counters, 0, 64, st));
    CK(ctx, cudaMemsetAsync(s.d_blocks_done, 0, n * sizeof(uint32_t), st));
    CK(ctx, cudaMemsetAsync(s.d_dstatus, 0, n * sizeof(int32_t), st));
    CK(ctx, cudaMemsetAsync(s.d_block_flags, 0, (nblk_total + 1) * sizeof(uint32_t), st));
    const uint32_t ng = md5_lane_order(s.h_order, n, raw_len);
    CK(ctx, cudaMemcpyAsync(s.d_order, s.h_order, ng * 32 * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    memset(s.h_md5, 0, (size_t)n * 16);
    DecParams p;
    p.chunks = s.d_dchunks;
    p.blocks = s.d_dblocks;
    p.status = s.d_dstatus;
    p.done = s.d_blocks_done;
    p.counter = s.d_counters;
    p.blk_done = s.d_block_flags;
    p.md5_order = s.d_order;
    p.md5_out = s.d_md5;
    p.n_chunks = n;
    p.n_groups = ng;
    p.rows = rows;
    CK(ctx, cudaEventRecord(s.ev_k0, st));
    sky_frame_index_kernel<<<(n + 127) / 128, 128, 0, st>>>(p);
    CK(ctx, cudaGetLastError());
    sky_decode_kernel<<<ctx->sm_count, 512, kMd5WarpsPerCta * kRingBytes, st>>>(p);
    CK(ctx, cudaGetLastError());
    CK(ctx, cudaEventRecord(s.ev_k1, st));
    ctx->launches += 2;
    CK(ctx, cudaMemcpyAsync(s.h_dstatus, s.d_dstatus, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    return SKY_OK;
}

int sky_decode_device(sky_ctx *ctx, uint32_t n, const void *d_frames, const uint64_t *frame_off, const uint64_t *frame_len,
                      void *d_out, const uint64_t *out_off, const uint64_t *raw_len, void *stream, int32_t *status, uint8_t *md5,
                      float *kernel_ms) {
    if (!ctx || n == 0 || !d_frames || !frame_off || !frame_len || !out_off || !raw_len) return fail(ctx, SKY_E_INVALID, "NULL argument or n == 0");
    if (n > ctx->max_chunks) return fail(ctx, SKY_E_CAPACITY, "n = %u > max_chunks = %u", n, ctx->max_chunks);
    if (reinterpret_cast<uintptr_t>(d_out) & 15) return fail(ctx, SKY_E_INVALID, "d_out is not 16-byte aligned");
    for (uint32_t i = 0; i < n; i++) {
        if (out_off[i] & 15) return fail(ctx, SKY_E_INVALID, "out_off[%u] is not a multiple of 16", i);
        if (raw_len[i] && !d_out) return fail(ctx, SKY_E_INVALID, "d_out is NULL");
    }
    CK(ctx, cudaSetDevice(ctx->device));
    Slot &s = ctx->slots[0];
    if (s.busy) return fail(ctx, SKY_E_BUSY, "slot 0 holds a batch that was not waited for");
    cudaStream_t st = stream ? (cudaStream_t)stream : s.stream;
    if (int rc = launch_decode(ctx, s, st, n, (const uint8_t *)d_frames, frame_off, frame_len, (uint8_t *)d_out, out_off, raw_len)) return rc;
    CK(ctx, cudaStreamSynchronize(st));
    if (status) memcpy(status, s.h_dstatus, n * sizeof(int32_t));
    if (md5) memcpy(md5, s.h_md5, (size_t)n * 16);
    if (kernel_ms) CK(ctx, cudaEventElapsedTime(kernel_ms, s.ev_k0, s.ev_k1));  // index + decode + MD5
    return SKY_OK;
}

int sky_decode(sky_ctx *ctx, uint32_t n, const void *const *frames, const uint64_t *frame_len, void *const *dst,
               const uint64_t *raw_len, int32_t *status, uint8_t *md5, float *kernel_ms) {
    return sky_decode_flags(ctx, n, frames, frame_len, dst, raw_len, 0, status, md5, kernel_ms);
}

int sky_decode_flags(sky_ctx *ctx, uint32_t n, const void *const *frames, const uint64_t *frame_len, void *const *dst,
                     const uint64_t *raw_len, uint32_t flags, int32_t *status, uint8_t *md5, float *kernel_ms) {
    if (!ctx || n == 0 || !frames || !frame_len || !dst || !raw_len) return fail(ctx, SKY_E_INVALID, "NULL argument or n == 0");
    if (n > ctx->max_chunks) return fail(ctx, SKY_E_CAPACITY, "n = %u > max_chunks = %u", n, ctx->max_chunks);
    Slot &s = ctx->slots[0];
    if (s.busy) return fail(ctx, SKY_E_BUSY, "slot 0 holds a batch that was not waited for");
    if (!s.d_in) return fail(ctx, SKY_E_INVALID, "the ctx was created without slots (n_slots = 0)");
    const bool e2ee = (flags & SKY_F_E2EE) != 0;
    if (e2ee && !ctx->d_key) return fail(ctx, SKY_E_NOKEY, "no key (sky_set_e2ee_key)");
    CK(ctx, cudaSetDevice(ctx->device));
    for (uint32_t i = 0; i < n; i++)
        if (!frames[i] || (raw_len[i] && !dst[i])) return fail(ctx, SKY_E_INVALID, "frames[%u] or dst[%u] is NULL", i, i);
    // roles swap on the way back: frames (<= bound) go into the frame slab, decoded bytes into the input slab
    uint64_t f_end, o_end;
    const std::vector<uint64_t> f_off = pack16(n, [&](uint32_t i) { return frame_len[i]; }, f_end);
    const std::vector<uint64_t> o_off = pack16(n, [&](uint32_t i) { return raw_len[i]; }, o_end);
    if (f_end > ctx->out_cap || o_end > ctx->in_cap) return fail(ctx, SKY_E_CAPACITY, "the batch exceeds slot 0's frame or output slab");
    std::vector<uint64_t> f_len(frame_len, frame_len + n);
    if (e2ee) {
        // the payloads are boxes (nonce | tag | ciphertext): check the tags, decrypt into the frame slab, then decode as usual
        if (int rc = alloc_box(ctx, s)) return rc;
        for (uint32_t i = 0; i < n; i++) {
            s.h_boxmeta[i] = frame_len[i];
            s.h_boxmeta[n + i] = f_off[i];
            CK(ctx, cudaMemcpyAsync(s.d_box + box_offset(f_off[i], i), frames[i], frame_len[i], cudaMemcpyHostToDevice, s.stream));
            f_len[i] = frame_len[i] >= (uint64_t)kBoxOverhead ? frame_len[i] - kBoxOverhead : 0;
        }
        CK(ctx, cudaMemcpyAsync(s.d_boxmeta, s.h_boxmeta, 2ull * n * sizeof(uint64_t), cudaMemcpyHostToDevice, s.stream));
        sky_box_open_setup_kernel<<<1, 256, 0, s.stream>>>(s.d_bchunks, s.d_blkbase, n, s.d_boxmeta, s.d_boxmeta + n, s.d_out, s.d_box);
        CK(ctx, cudaGetLastError());
        sky_box_keys_kernel<<<(n + 63) / 64, 64, 0, s.stream>>>(s.d_bchunks, n, ctx->d_key, s.d_sub);
        CK(ctx, cudaGetLastError());
        sky_box_tag_kernel<<<n, kPolyThreads, 0, s.stream>>>(s.d_bchunks, s.d_sub, 1, s.d_bstatus);
        CK(ctx, cudaGetLastError());
        sky_box_xor_kernel<<<ctx->sm_count * 8, 256, 0, s.stream>>>(s.d_bchunks, s.d_blkbase, n, s.d_sub, 1);
        CK(ctx, cudaGetLastError());
        CK(ctx, cudaMemcpyAsync(s.h_bstatus, s.d_bstatus, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s.stream));
        ctx->launches += 4;
    } else {
        for (uint32_t i = 0; i < n; i++)
            CK(ctx, cudaMemcpyAsync(s.d_out + f_off[i], frames[i], frame_len[i], cudaMemcpyHostToDevice, s.stream));
    }
    if (int rc = sky_decode_device(ctx, n, s.d_out, f_off.data(), f_len.data(), s.d_in, o_off.data(), raw_len, s.stream, status, md5, kernel_ms))
        return rc;
    if (e2ee) {
        for (uint32_t i = 0; i < n; i++)
            if (s.h_bstatus[i] != 0 || frame_len[i] < (uint64_t)kBoxOverhead) {  // forged or truncated box: never hand its bytes out
                s.h_dstatus[i] = SKY_D_AUTH;
                if (status) status[i] = SKY_D_AUTH;
            }
    }
    for (uint32_t i = 0; i < n; i++)
        if (raw_len[i] && s.h_dstatus[i] == 0)
            CK(ctx, cudaMemcpyAsync(dst[i], s.d_in + o_off[i], raw_len[i], cudaMemcpyDeviceToHost, s.stream));
    CK(ctx, cudaStreamSynchronize(s.stream));
    return SKY_OK;
}

uint64_t sky_launch_count(const sky_ctx *ctx) { return ctx ? ctx->launches : 0; }

}  // extern "C"
