// lz4.cuh -- LZ4 block compressor for sm_100a: helpers shared by all formulations, and the CTA-per-block compressor
// (prober / parser warps over a shared-memory copy of the block) that sky_fused_kernel runs.
//
// Replaces, per 64 KiB block, what lz4.frame.compress(data) does inside
// skyplane/gateway/operators/gateway_operator.py:358-361 (liblz4's level-0 "fast" compressor:
// single-candidate hash table, greedy, skip acceleration).  The GPU formulation (details above each part below):
//   * one CTA owns one independent 64 KiB block at a time (frame flag B.Indep, so no cross-block state);
//   * the match table is 4096 x (pos16 << 16 | tag16) in shared memory; a probe never reads the candidate's bytes;
//   * 32 probe slots are one warp instruction; the stride between slots doubles over data without hits;
//   * parser warps verify and extend the hits of whole segments independently and emit standard LZ4 sequences;
//   * blocks that do not shrink are stored raw (bit 31 of the block header), like LZ4F_makeBlock;
//   * linked blocks (SKY_F_LINKED): the block is parsed behind a window of the input before it (parse_segment).
// Output is a standard LZ4 block: decodable by lz4.frame.decompress (gateway_receiver.py:196).
// tools/lz4_tile_model.c is the sequential twin of the parse; frames are byte-identical to it (tests).
#pragma once
#include <stdint.h>

namespace sky {

constexpr uint32_t kBlock = 65536;       // BD = 0x40
#ifndef SKY_LZ4_ENTRIES
#define SKY_LZ4_ENTRIES 4096
#endif
constexpr uint32_t kEntries = SKY_LZ4_ENTRIES;  // match-table entries per CTA (u32 each: pos16 << 16 | tag16); any multiple of 128
constexpr uint32_t kTableBytes = kEntries * 4;
constexpr uint32_t kMinMatch = 4;
constexpr uint32_t kMfLimit = 12;        // a match must start >= 12 bytes before the block end
constexpr uint32_t kLastLiterals = 5;    // the last 5 bytes are always literals
constexpr unsigned kFull = 0xffffffffu;

// ---- warp copy: dst and src arbitrarily aligned; regions disjoint, or dst < src (forward move) ----
// Over-reads at most 3 bytes past src+n (inside the same 4-byte word group); never over-writes.
__device__ __forceinline__ void warp_copy(uint8_t *dst, const uint8_t *src, uint32_t n, unsigned lane) {
    if (n < 64) {
        for (uint32_t base = 0; base < n; base += 32) {
            const uint32_t k = base + lane;
            uint8_t b = 0;
            if (k < n) b = src[k];
            __syncwarp();
            if (k < n) dst[k] = b;
        }
        return;
    }
    const uint32_t head = (16u - (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u;  // < 16 <= n
    uint8_t hb = 0;
    if (lane < head) hb = src[lane];
    __syncwarp();
    if (lane < head) dst[lane] = hb;
    dst += head;
    src += head;
    n -= head;
    const uint32_t nvec = n >> 4;
    const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(src) & 3u) * 8u;
    const uint32_t *sw = reinterpret_cast<const uint32_t *>(reinterpret_cast<uintptr_t>(src) & ~(uintptr_t)3);
    uint4 *dv = reinterpret_cast<uint4 *>(dst);
    for (uint32_t base = 0; base < nvec; base += 32) {
        const uint32_t k = base + lane;
        uint4 o = make_uint4(0, 0, 0, 0);
        if (k < nvec) {
            const uint32_t *q = sw + 4 * (size_t)k;
            const uint32_t w0 = q[0], w1 = q[1], w2 = q[2], w3 = q[3];
            const uint32_t w4 = sh ? q[4] : 0u;
            o.x = __funnelshift_r(w0, w1, sh);
            o.y = __funnelshift_r(w1, w2, sh);
            o.z = __funnelshift_r(w2, w3, sh);
            o.w = __funnelshift_r(w3, w4, sh);
        }
        __syncwarp();  // every lane has its source words before any lane overwrites (forward move)
        if (k < nvec) dv[k] = o;
    }
    const uint32_t done = nvec << 4, tail = n & 15u;
    uint8_t tb = 0;
    if (lane < tail) tb = src[done + lane];
    __syncwarp();
    if (lane < tail) dst[done + lane] = tb;
}

// ---- streaming warp copy for DISJOINT regions: 16-byte loads (4 in flight per lane), 16-byte streaming stores (the
// frame is never re-read here: keep L2 for the input rows and the scratch).  src 16-byte aligned; dst arbitrary.
// kReadOnly: the source is kernel-read-only input (ld.global.nc); otherwise it was written by this warp (ld.global.cg).
template <bool kReadOnly>
__device__ __forceinline__ uint32_t ld_stream32(const uint32_t *p) { return kReadOnly ? __ldg(p) : __ldcg(p); }
template <bool kReadOnly>
__device__ __forceinline__ uint4 ld_stream128(const uint4 *p) { return kReadOnly ? __ldg(p) : __ldcg(p); }

template <bool kReadOnly>
__device__ __forceinline__ void warp_copy_stream(uint8_t *dst, const uint8_t *__restrict__ src, uint32_t n, unsigned lane) {
    const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 15u);
    if (mis == 0) {
        const uint4 *sv = reinterpret_cast<const uint4 *>(src);
        uint4 *dv = reinterpret_cast<uint4 *>(dst);
        const uint32_t nvec = n >> 4;
        uint32_t k = lane;
        for (; k + 96 < nvec; k += 128) {
            const uint4 a = ld_stream128<kReadOnly>(sv + k), b = ld_stream128<kReadOnly>(sv + k + 32),
                        c = ld_stream128<kReadOnly>(sv + k + 64), d = ld_stream128<kReadOnly>(sv + k + 96);
            __stcs(dv + k, a); __stcs(dv + k + 32, b); __stcs(dv + k + 64, c); __stcs(dv + k + 96, d);
        }
        for (; k < nvec; k += 32) __stcs(dv + k, ld_stream128<kReadOnly>(sv + k));
        const uint32_t done = nvec << 4;
        if (lane < (n & 15u)) dst[done + lane] = src[done + lane];
        return;
    }
    // dst = 16-byte aligned base + mis: build each aligned 16-byte store from two consecutive source vectors
    const uint32_t head = 16u - mis;  // bytes until dst is aligned
    if (n <= head + 16) {
        for (uint32_t k = lane; k < n; k += 32) dst[k] = src[k];
        return;
    }
    if (lane < head) dst[lane] = src[lane];
    uint4 *dv = reinterpret_cast<uint4 *>(dst + head);
    const uint32_t rem = n - head, nvec = rem >> 4;
    const uint32_t *sw = reinterpret_cast<const uint32_t *>(src);  // src + head = word (head>>2), byte shift (head&3)
    const uint32_t wsh = head >> 2, bsh = (head & 3u) * 8u;
    for (uint32_t k = lane; k < nvec; k += 32) {
        const uint32_t *q = sw + wsh + 4 * (size_t)k;
        const uint32_t w0 = ld_stream32<kReadOnly>(q), w1 = ld_stream32<kReadOnly>(q + 1), w2 = ld_stream32<kReadOnly>(q + 2),
                       w3 = ld_stream32<kReadOnly>(q + 3);
        const uint32_t w4 = bsh ? ld_stream32<kReadOnly>(q + 4) : 0u;
        uint4 o;
        o.x = __funnelshift_r(w0, w1, bsh);
        o.y = __funnelshift_r(w1, w2, bsh);
        o.z = __funnelshift_r(w2, w3, bsh);
        o.w = __funnelshift_r(w3, w4, bsh);
        __stcs(dv + k, o);
    }
    const uint32_t done = head + (nvec << 4);
    if (lane < (rem & 15u)) dst[done + lane] = src[done + lane];
}

// ---- XXH32 of the frame descriptor (2 or 10 bytes), for the header checksum byte -----------------
__device__ __forceinline__ uint32_t rotl32(uint32_t x, int s) { return __funnelshift_l(x, x, s); }
__device__ __forceinline__ uint32_t xxh32_small(const uint8_t *p, uint32_t len) {  // len < 16, seed 0
    constexpr uint32_t P1 = 2654435761u, P2 = 2246822519u, P3 = 3266489917u, P4 = 668265263u, P5 = 374761393u;
    uint32_t h = P5 + len;
    uint32_t i = 0;
    for (; i + 4 <= len; i += 4) {
        const uint32_t v = p[i] | (p[i + 1] << 8) | (p[i + 2] << 16) | ((uint32_t)p[i + 3] << 24);
        h = rotl32(h + v * P3, 17) * P4;
    }
    for (; i < len; i++) h = rotl32(h + p[i] * P5, 11) * P1;
    h ^= h >> 15;
    h *= P2;
    h ^= h >> 13;
    h *= P3;
    h ^= h >> 16;
    return h;
}

// Writes the frame header for an n-byte chunk at dst; returns its size (15, or 7 when n == 0).  linked: FLG 0x48 (linked
// blocks) when the chunk has more than one block; one block keeps 0x68, as LZ4F_compressFrame switches a single-block
// input to independent blocks.  Single thread.
__device__ __forceinline__ uint32_t write_frame_header(uint8_t *dst, uint64_t n, bool linked = false) {
    uint8_t d[10];
    d[1] = 0x40;  // BD: 64 KiB blocks
    dst[0] = 0x04; dst[1] = 0x22; dst[2] = 0x4D; dst[3] = 0x18;
    if (n == 0) {
        d[0] = 0x60;  // v01 | B.Indep ; content size omitted (0 means "unknown" to LZ4F)
        dst[4] = d[0]; dst[5] = d[1];
        dst[6] = (uint8_t)(xxh32_small(d, 2) >> 8);
        return 7;
    }
    d[0] = linked && n > kBlock ? 0x48 : 0x68;  // v01 | C.Size (| B.Indep)
#pragma unroll
    for (int i = 0; i < 8; i++) d[2 + i] = (uint8_t)(n >> (8 * i));
#pragma unroll
    for (int i = 0; i < 10; i++) dst[4 + i] = d[i];
    dst[14] = (uint8_t)(xxh32_small(d, 10) >> 8);
    return 15;
}

// ---- sequence emission ----------------------------------------------------------------------------
// Emits token, literal-length bytes, literals, offset, match-length bytes.  All lanes call it with
// warp-uniform arguments; returns the new output cursor.
__device__ __forceinline__ uint32_t emit_seq(uint8_t *out, uint32_t op, const uint8_t *src, uint32_t anchor, uint32_t ll,
                                            uint32_t ml, uint32_t offset, unsigned lane) {
    const uint32_t mcode = ml ? ml - kMinMatch : 0;
    if (lane == 0) out[op] = (uint8_t)(((ll < 15 ? ll : 15) << 4) | (mcode < 15 ? mcode : 15));
    op += 1;
    if (ll >= 15) {
        const uint32_t r = ll - 15, n255 = r / 255;
        for (uint32_t k = lane; k < n255; k += 32) out[op + k] = 255;
        if (lane == 0) out[op + n255] = (uint8_t)(r - n255 * 255);
        op += n255 + 1;
    }
    warp_copy(out + op, src + anchor, ll, lane);
    op += ll;
    if (ml) {
        if (lane == 0) {
            out[op] = (uint8_t)offset;
            out[op + 1] = (uint8_t)(offset >> 8);
        }
        op += 2;
        if (mcode >= 15) {
            const uint32_t r = mcode - 15, n255 = r / 255;
            for (uint32_t k = lane; k < n255; k += 32) out[op + k] = 255;
            if (lane == 0) out[op + n255] = (uint8_t)(r - n255 * 255);
            op += n255 + 1;
        }
    }
    return op;
}

// =====================================================================================================
// CTA-per-block compressor.  One CTA owns one 64 KiB block at a time:
//   * the block is brought into shared memory with ONE bulk async copy (TMA 1-D, cp.async.bulk + mbarrier);
//   * warp 0 (the prober) walks the block segment by segment (kSegSlots probe slots each): hash 5 bytes, ONE
//     shared-memory lookup of (pos16 | tag16) per slot, no byte of the candidate is read; the 32 slots of a group look the
//     table up together and then replace their entries (atomic max: the last slot stays); short periods inside a group
//     are caught by comparing hashes 3, 4 and 8 lanes apart.  Per segment it publishes a
//     hit bit mask and the candidate offsets through a ring of shared-memory slots (mbarrier full / empty pairs);
//   * the parser warps each take whole segments from the ring and parse them INDEPENDENTLY (cursor and anchor start at the
//     segment start, matches are clipped to the segment end): per accepted match one warp-wide round compares 23 bytes
//     ahead and 8 bytes behind -- verification, forward and backward extension in one ballot, all from shared memory --
//     sequences are recorded one per lane and emitted 32 at a time into the segment's scratch area (L2-resident);
//   * after a CTA barrier warp 0 strings the segments together (literals a segment leaves behind are carried into the
//     next segment's first sequence), learns the block's frame offset from the OFF chain, and all warps write the block to
//     its final place exactly once.
// tools/lz4_tile_model.c is the sequential twin of exactly these rules (frames are byte-identical, tested).
#ifndef SKY_COOP_LIT
#define SKY_COOP_LIT 16
#endif
#ifndef SKY_MAX_STEP_LOG
#define SKY_MAX_STEP_LOG 4
#endif
#define SKY_SEG_GROUPS 32   // (fixed: 4 prober batches of 8 groups; a parser lane holds one group's hit mask)
constexpr uint32_t kCoopLit = SKY_COOP_LIT;          // literal runs at least this long are copied by the whole warp
constexpr uint32_t kMaxStepLog = SKY_MAX_STEP_LOG;   // probe stride doubles after a segment without a hit, up to 1 << this
constexpr int kSegGroups = SKY_SEG_GROUPS;           // a segment = this many warp-wide groups of probe slots (<= 32)
constexpr uint32_t kSegSlots = kSegGroups * 32;
constexpr uint32_t kMaxSegs = kBlock / kSegSlots;    // most segments a block can have (stride 1 throughout)
constexpr uint32_t kSegPad = 80;                     // scratch slack per segment: a segment's sequences can outgrow it by < 70 B
constexpr uint32_t kScratchBytes = kBlock + kMaxSegs * kSegPad + 1024;  // per-CTA compressed-segment scratch (global, L2)
static_assert(kSegGroups >= 1 && kSegGroups <= 32, "SKY_SEG_GROUPS must be 1..32");

// ring slot: what the prober hands a parser for one segment
struct SegSlot {
    uint16_t offs[kSegSlots];   // slot i: position - candidate position (valid where the hit bit is set)
    uint32_t masks[32];         // group g: hit bits of its 32 slots (groups >= kSegGroups: 0)
    uint32_t seg_pos, slog, sidx, pad;
};
// what a parser leaves behind for one segment
struct SegRec {
    uint32_t seg_pos;
    uint32_t lead_ml;   // first sequence: literals from the segment start | match length << 16 (0 = no match in the segment)
    uint32_t off_t;     // first sequence's offset | trailing literal bytes << 16
    uint32_t mbytes;    // bytes of the 2nd.. sequences in the segment's scratch area
};
struct SegPlan {
    uint32_t foff, moff;  // where the first sequence / the rest go, relative to the block's first data byte
    uint32_t fll, pad;    // first sequence's full literal length (carry + lead)
};

// ---- mbarrier / bulk-copy primitives (shared::cta) -----------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
// Explicit shared-state-space accessors on 32-bit shared addresses: the hot loops must compile to LDS / STS with 32-bit
// address arithmetic, whatever the compiler can or cannot infer about a pointer's address space.
__device__ __forceinline__ uint32_t lds32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds16(uint32_t a) {
    uint16_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds8(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts16(uint32_t a, uint32_t v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"((uint16_t)v) : "memory"); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// try_wait with a suspend-time hint (ns): the waiting warp is parked by the hardware instead of spinning through the
// scheduler -- a spinning parser would take issue slots from the prober it is waiting for
__device__ __forceinline__ bool mbar_try_wait_hint(uint64_t *bar, uint32_t parity, uint32_t ns) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(ns) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait_hint(bar, parity, 20000u)) {}
}
// global -> shared bulk async copy (TMA 1-D): bytes multiple of 16, both addresses 16-byte aligned; completes on `bar`
__device__ __forceinline__ void bulk_load(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ uint32_t div255(uint32_t x) { return (x * 0x8081u) >> 23; }  // exact for x < 65536
__device__ __forceinline__ uint32_t seq_bytes_fast(uint32_t ll, uint32_t ml) {           // ll, ml < 65536
    uint32_t s = 1 + ll + (ll >= 15 ? div255(ll - 15) + 1 : 0);
    if (ml) s += 2 + (ml >= 19 ? div255(ml - 19) + 1 : 0);
    return s;
}
// unaligned little-endian 32-bit read from the shared-memory copy of the block (in_s = its 32-bit shared address)
__device__ __forceinline__ uint32_t load32s(uint32_t in_s, uint32_t pos) {
    const uint32_t a = in_s + (pos & ~3u);
    return __funnelshift_r(lds32(a), lds32(a + 4), (pos & 3u) * 8u);
}

// ---- cooperative forward extension in shared memory: all lanes compare 4 bytes each per round
__device__ __forceinline__ uint32_t extend_coop_s(uint32_t in32, uint32_t mpos, uint32_t mcand, uint32_t mlen, uint32_t maxlen,
                                                  unsigned lane) {
    for (;;) {
        const uint32_t o = mlen + lane * 4;
        uint32_t cnt = 0;
        if (o < maxlen) {
            const uint32_t x = load32s(in32, mpos + o) ^ load32s(in32, mcand + o);
            cnt = x ? (uint32_t)(__ffs(x) - 1) >> 3 : 4u;
            cnt = min(cnt, maxlen - o);
        }
        const unsigned fullm = __ballot_sync(kFull, cnt == 4);
        if (fullm == kFull) {
            mlen += 128;
            continue;
        }
        const int f = __ffs(~fullm) - 1;
        return mlen + 4 * f + __shfl_sync(kFull, cnt, f);
    }
}

// ---- emission of up to 32 recorded sequences, one per lane ------------------------------------------
// q0 = literal length | match length << 16, q1 = literal start | offset << 16 (lane k = k-th sequence).  Literals come
// from the shared-memory copy of the block, output goes to the segment's scratch area.  Sizes go through a warp scan; every
// lane writes its own token, length bytes, literals (runs >= kCoopLit: one warp copy each), offset and match-length bytes.
// skip_first: lane 0 holds the segment's FIRST sequence, which is not emitted here (its literal run is completed with the
// literals carried over from earlier segments when the block is assembled).
// (One copy per kernel: kLinked only keeps the linked kernel's call from changing how the default kernel's is compiled.)
template <bool kLinked>
__device__ __noinline__ uint32_t flush_seqs(uint8_t *__restrict__ out, uint32_t op, const uint8_t *in, uint32_t q0, uint32_t q1,
                                            uint32_t nseq, bool skip_first, unsigned lane) {
    const uint32_t in32 = smem_u32(in);
    const bool act = lane < nseq && !(skip_first && lane == 0);
    const uint32_t ll = q0 & 0xffffu, ml = q0 >> 16, lit = q1 & 0xffffu, off = q1 >> 16;
    const uint32_t mcode = ml - kMinMatch;
    const uint32_t nl = ll >= 15 ? div255(ll - 15) + 1 : 0, nm = mcode >= 15 ? div255(mcode - 15) + 1 : 0;
    const uint32_t sz = act ? 3 + ll + nl + nm : 0;
    uint32_t incl = sz;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(kFull, incl, d);
        if ((int)lane >= d) incl += t;
    }
    const uint32_t total = __shfl_sync(kFull, incl, 31);
    uint32_t lit_o = 0;
    if (act) {
        uint32_t o = op + incl - sz;
        out[o++] = (uint8_t)(((ll < 15 ? ll : 15) << 4) | (mcode < 15 ? mcode : 15));
        if (nl) {
            for (uint32_t k = 0; k + 1 < nl; k++) out[o + k] = 255;
            out[o + nl - 1] = (uint8_t)(ll - 15 - (nl - 1) * 255);
            o += nl;
        }
        lit_o = o;
        if (ll < kCoopLit) {
            uint32_t k = 0;
            for (; k + 4 <= ll; k += 4) {  // 4 literal bytes per round: one unaligned read, four byte stores
                const uint32_t w = load32s(in32, lit + k);
                out[o + k] = (uint8_t)w;
                out[o + k + 1] = (uint8_t)(w >> 8);
                out[o + k + 2] = (uint8_t)(w >> 16);
                out[o + k + 3] = (uint8_t)(w >> 24);
            }
            const uint32_t rem = ll - k;
            if (rem) {
                const uint32_t w = load32s(in32, lit + k);
                out[o + k] = (uint8_t)w;
                if (rem > 1) out[o + k + 1] = (uint8_t)(w >> 8);
                if (rem > 2) out[o + k + 2] = (uint8_t)(w >> 16);
            }
        }
        o += ll;
        out[o] = (uint8_t)off;
        out[o + 1] = (uint8_t)(off >> 8);
        o += 2;
        if (nm) {
            for (uint32_t k = 0; k + 1 < nm; k++) out[o + k] = 255;
            out[o + nm - 1] = (uint8_t)(mcode - 15 - (nm - 1) * 255);
        }
    }
    __syncwarp();
    unsigned big = __ballot_sync(kFull, act && ll >= kCoopLit);
    while (big) {  // long literal runs: one warp-wide copy each (generic loads: the source is shared memory)
        const int l = __ffs(big) - 1;
        big &= big - 1;
        warp_copy(out + __shfl_sync(kFull, lit_o, l), in + __shfl_sync(kFull, lit, l), __shfl_sync(kFull, ll, l), lane);
    }
    return op + total;
}

// ---- prober: one batch of 8 groups (256 probe slots) of a segment.
// Phase A -- everything that does not depend on the table, for all 8 groups: input words, the 5-byte hash, the table index,
// the entry this slot will leave behind (pos16 << 16 | tag16), and the in-group candidates: a lane whose 32-bit hash equals
// that of the lane 3, 4 or 8 places below it takes that lane's slot as its candidate (three shuffles; periods 1, 2, 3, 4
// and 8 -- runs, UTF-16, pixels, words, doubles -- which the table cannot know yet because a group looks the table up before
// any of its slots is inserted).  Nothing here orders the lanes by hash: round 2's first formulation used match.any for
// that, and at 58 cycles of the SM's one ADU pipe per instruction it was what bounded the kernel (profiles/README.md).
// `turn()` is called between the phases: it returns when the other prober has finished the previous batch's table phase.
// Phase B -- the 8 table lookups and updates back to back: every lane reads its entry, then every lane max-es its own in
// (position in the high half: of the lanes that share an index the highest one stays, exactly what inserting the slots in
// order leaves behind).  The LSU keeps a warp's shared-memory accesses in order, so group k+1's lookup sees group k's
// update without waiting for group k's lookup to return.  Phase C -- consume the lookups: hit masks and candidate offsets
// into the segment's ring slot.  Returns the OR of the batch's hit masks.
// Slots past the last probe position (p > mflimit, only at the very end of a block, always the highest lanes) hash a
// clamped position: the entries they leave in the table no later lookup can observe, and the hits they report the parser
// masks out (parse_segment), so the prober spends nothing on them.
// kLinked (positions are window coordinates, up to window + 64 KiB, kept modulo 65536 in the entry): every lane first
// stores its entry, then max-es it in.  The store replaces whatever an earlier group left, which the max alone would keep
// once positions wrap; the max then picks the group's last slot.  A group never straddles the wrap (window coordinate
// 65536 = block position 65536 - W, a multiple of 1024 and so a group boundary), so the max sees no wrap inside a group.
// The offset (mine - e) >> 16 is then (position - entry) mod 65536: always 1..65535 for a hit.
__device__ __forceinline__ uint32_t bfind(uint32_t x) {  // index of the highest set bit (0xffffffff for 0): one FLO
    uint32_t r;
    asm("bfind.u32 %0, %1;" : "=r"(r) : "r"(x));
    return r;
}
// n = (the slot distance d << slog) << 16 if the lane d = 3, 4 or 8 places below has my hash (the nearest one), else unchanged
__device__ __forceinline__ void near_slot(uint32_t &n, uint32_t hf, uint32_t c3, uint32_t c4, uint32_t c8) {
    asm volatile(
        "{\n\t"
        ".reg .pred p, q;\n\t"
        ".reg .b32 t;\n\t"
        "shfl.sync.up.b32 t|p, %1, 8, 0, 0xffffffff;\n\t"
        "setp.eq.and.u32 q, t, %1, p;\n\t"
        "selp.u32 %0, %4, %0, q;\n\t"
        "shfl.sync.up.b32 t|p, %1, 4, 0, 0xffffffff;\n\t"
        "setp.eq.and.u32 q, t, %1, p;\n\t"
        "selp.u32 %0, %3, %0, q;\n\t"
        "shfl.sync.up.b32 t|p, %1, 3, 0, 0xffffffff;\n\t"
        "setp.eq.and.u32 q, t, %1, p;\n\t"
        "selp.u32 %0, %2, %0, q;\n\t"
        "}"
        : "+r"(n)
        : "r"(hf), "r"(c3), "r"(c4), "r"(c8));
}
__device__ __forceinline__ void red_max_s(uint32_t a, uint32_t v) {
    asm volatile("red.shared.max.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
template <bool kLinked = false, class Turn>
__device__ __forceinline__ uint32_t probe_batch(uint32_t in_s, uint32_t tab_s, uint32_t offs_s, uint32_t masks_s, uint32_t seg_pos,
                                                uint32_t slog, uint32_t batch, uint32_t mflimit, unsigned lane, Turn turn) {
    const uint32_t pstep = 32u << slog;
    uint32_t p = seg_pos + ((batch * 256u + lane) << slog);
    // p & 3 is the same for every group of the segment (p advances by a multiple of 32): byte selectors are loop-invariant
    const uint32_t selv = 0x3210u + 0x1111u * (p & 3u), selb = 0x4440u | (p & 3u);
    const uint32_t offs_l = offs_s + (batch * 256u + lane) * 2u;
    const uint32_t c3 = 0x30000u << slog, c4 = 0x40000u << slog, c8 = 0x80000u << slog;
    uint32_t idx[8], mine[8], e[8], near[8], anyhit = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const uint32_t pc = min(p, mflimit);
        const uint32_t a = in_s + (pc & ~3u);
        const uint32_t w0 = lds32(a), w1 = lds32(a + 4);
        uint32_t hf = __byte_perm(w0, w1, selv) * 2654435761u;
        hf = __byte_perm(w1, 0u, selb) * 0x85EBCA6Bu + hf;  // fifth byte
        idx[k] = __umulhi(hf, kEntries) * 4u;               // byte offset of the table entry
        mine[k] = __byte_perm(p, hf, 0x1065);               // pos16 << 16 | hash bytes 1-2 as the tag
        near[k] = 0u;
        near_slot(near[k], hf, c3, c4, c8);
        p += pstep;
    }
    turn();
#pragma unroll
    for (int k = 0; k < 8; k++) {
        e[k] = lds32(tab_s + idx[k]);
        __syncwarp();  // (orders the lanes' table reads of this group before its updates)
        if (kLinked) {
            sts32(tab_s + idx[k], mine[k]);
            __syncwarp();
        }
        red_max_s(tab_s + idx[k], mine[k]);
        __syncwarp();
    }
#pragma unroll
    for (int k = 0; k < 8; k++) {
        uint32_t d = mine[k] - e[k];  // tags equal <=> low half 0 (then no borrow: the high half is the distance, >= 1 for
        if (near[k]) d = near[k];     // a real entry, 0 only for slot 0 against the empty table)
        const uint32_t off = d >> 16;
        const unsigned hits = __ballot_sync(kFull, (d & 0xffffu) == 0u && off != 0u);
        anyhit |= hits;
        if (lane == 0) sts32(masks_s + (batch * 8u + (uint32_t)k) * 4u, hits);
        sts16(offs_l + (uint32_t)k * 64u, off);
    }
    return anyhit;
}

// ---- parser: one segment.  in = shared-memory copy of the block, scr = this segment's scratch area.
// (Hits only exist at positions <= L-12 inside the segment, so a hit position is always below the match limit.)
// Linked blocks: in = [window | block], base = the window's length, L = base + block length; positions are window
// coordinates, so candidates (and the backward extension's min(pos - anchor, cand, 8)) may reach into the window.  What
// the segment hands on (record, literal starts) is relative to the block.
template <bool kLinked = false>
__device__ __forceinline__ SegRec parse_segment(const uint8_t *in, const SegSlot *slot, uint8_t *__restrict__ scr, uint32_t L,
                                                unsigned lane, uint32_t base = 0) {
    const uint32_t in32 = smem_u32(in), offs_s = smem_u32(slot->offs);
    const uint32_t seg_pos = slot->seg_pos, slog = slot->slog;
    const uint32_t mflimit = L - kMfLimit, matchlimit = L - kLastLiterals;
    // group `lane` of the segment: only slots at positions <= mflimit were probed for real (the rest: block tail)
    const uint32_t n_real = ((mflimit - seg_pos) >> slog) + 1u;  // (seg_pos <= mflimit for every segment)
    const uint32_t mymask = slot->masks[lane] & ~__funnelshift_lc(0u, 0xffffffffu, min(max(n_real, lane * 32u) - lane * 32u, 32u));
    const uint32_t seg_lim = seg_pos + (kSegSlots << slog);
    const uint32_t mlim = min(matchlimit, seg_lim);                 // matches end at or before this
    const uint32_t seg_end = seg_lim > mflimit ? L : seg_lim;      // the last segment owns the block's tail
    const uint32_t round_up = (1u << slog) - 1u;
    const uint32_t dl = lane < 23 ? lane : lane - 32u;      // byte this lane compares: +0..+22 ahead, -1..-8 behind (lane 31 = -1)
    const uint32_t jrel = lane < 23 ? lane : 31u - lane;    // its distance from the match start
    const bool fwd_lane = lane < 23;
    uint32_t anchor = seg_pos, cur = seg_pos, nseq = 0, q0 = 0, q1 = 0, mbytes = 0;
    uint32_t first_q0 = 0, first_q1 = 0;
    bool first_pending = true;  // the segment's first sequence sits in lane 0 of the first batch
    unsigned nz = __ballot_sync(kFull, mymask != 0u);
    uint32_t m = 0, gbase = 0, sbase = 0;
    for (;;) {
        if (m == 0) {
            if (nz == 0) break;
            const int g = __ffs(nz) - 1;
            nz &= nz - 1;
            m = __shfl_sync(kFull, mymask, g);
            sbase = (uint32_t)g * 32u;
            gbase = seg_pos + (sbase << slog);
            m &= __funnelshift_lc(0u, 0xffffffffu, (max(cur, gbase) - gbase + round_up) >> slog);  // slots the cursor has passed
            if (m == 0) continue;
        }
        const uint32_t bit = bfind(m & (0u - m));  // lowest set bit: two ALU ops + one FLO (ffs is BREV + FLO, both on the XU pipe)
        uint32_t pos = gbase + (bit << slog);
        const uint32_t off = lds16(offs_s + (sbase + bit) * 2u);
        const uint32_t cand = pos - off;
        const uint32_t maxlen = mlim - pos;
        const uint32_t room = min(min(pos - anchor, cand), 8u);
        bool ok = false;
        if (jrel < (fwd_lane ? maxlen : room)) ok = lds8(in32 + pos + dl) == lds8(in32 + cand + dl);
        const unsigned z = ~__ballot_sync(kFull, ok) | 0x00800000u;  // bit 23 = stop bit of the forward scan
        uint32_t mlen = bfind(z & (0u - z));                       // 0..23
        if (mlen - kMinMatch >= 23u - kMinMatch) {  // rare: a tag collision (< 4), or the match runs past the 23 bytes compared
            if (mlen < kMinMatch) {
                m &= m - 1;
                continue;
            }
            if (maxlen > 23u) mlen = extend_coop_s(in32, pos, cand, 23u, maxlen, lane);
        }
        const uint32_t back = (uint32_t)__clz(z);  // 0..8 (lane 31 = byte -1)
        const uint32_t end = pos + mlen;
        pos -= back;
        mlen += back;
        const uint32_t r0 = (pos - anchor) | (mlen << 16), r1 = (anchor - base) | (off << 16);
        if (lane == nseq) {
            q0 = r0;
            q1 = r1;
        }
        anchor = cur = end;
        m &= __funnelshift_lc(0u, 0xffffffffu, (cur - gbase + round_up) >> slog);
        if (++nseq == 32) {
            if (first_pending) {
                first_q0 = __shfl_sync(kFull, q0, 0);
                first_q1 = __shfl_sync(kFull, q1, 0);
            }
            mbytes = flush_seqs<kLinked>(scr, mbytes, in + base, q0, q1, 32, first_pending, lane);
            first_pending = false;
            nseq = 0;
        }
    }
    if (nseq) {
        if (first_pending) {
            first_q0 = __shfl_sync(kFull, q0, 0);
            first_q1 = __shfl_sync(kFull, q1, 0);
        }
        mbytes = flush_seqs<kLinked>(scr, mbytes, in + base, q0, q1, nseq, first_pending, lane);
    }
    SegRec r;
    r.seg_pos = seg_pos - base;
    r.lead_ml = first_q0;                                            // lead literals | match length << 16 (0: no match)
    r.off_t = (first_q1 >> 16) | ((seg_end - anchor) << 16);        // offset | trailing literals << 16
    r.mbytes = mbytes;
    return r;
}

}  // namespace sky
