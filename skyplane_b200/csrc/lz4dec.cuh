// lz4dec.cuh -- LZ4 frame decoder for the receiving gateway (SURVEY.md section 8f row 1), sm_100a.
//
// Replaces lz4.frame.decompress(to_write) at skyplane/gateway/operators/gateway_receiver.py:195-201.
// Two device steps:
//   frame_index : one lane per chunk checks the frame header (magic, FLG, BD, content size, header checksum)
//                 and walks the block headers, producing a block table (offset, size word) per chunk;
//   block decode: one warp per 64 KiB block.  Frames whose blocks are independent (what the B200 sender
//                 emits) decode fully in parallel; linked-block frames (what the reference's CPU sender emits)
//                 decode block j after block j-1 of the same chunk (matches may reach into earlier output).
// Every read and write is bounds-checked: a malformed frame yields an error status, never an out-of-range access.
// It rejects what liblz4 rejects, and additionally enforces the block format's end-of-block rules (a match starts at
// least 12 bytes before the end of its block, the last 5 bytes are literals) and offset != 0: liblz4 checks the former
// against the room left in its 64 KiB block buffer rather than the block's real end, and lets offset 0 through.
// The decoded size of block j is taken to be min(64 KiB, raw_len - j*64 KiB) -- true for liblz4 and for our
// encoder (only the last block is short); anything else is reported as SKY_D_LAYOUT.
#pragma once
#include <stdint.h>

#include "lz4.cuh"

namespace sky {

constexpr int32_t kDecOk = 0;
constexpr int32_t kDecBadHeader = -1;   // magic / version / reserved bits / block size id / header checksum
constexpr int32_t kDecCorrupt = -2;     // malformed sequence, offset out of range, overrun
constexpr int32_t kDecSize = -3;        // content size or decoded size differs from the expected raw length
constexpr int32_t kDecUnsupported = -4; // dictID / checksummed frames (never produced on this path)
constexpr int32_t kDecLayout = -5;      // block structure does not match 64 KiB blocks with a short last one
constexpr int32_t kDecTruncated = -6;   // frame ends inside a header or block

struct DecChunk {
    const uint8_t *frame;  // frame bytes (any alignment)
    uint8_t *out;          // decoded bytes (16-byte aligned)
    uint64_t frame_len;
    uint64_t raw_len;      // expected decoded size (WireProtocolHeader.raw_data_len)
    uint64_t blk_base;     // index of this chunk's first entry in the block table
    uint32_t nblk;
    uint32_t linked;       // written by frame_index: 1 = blocks may reference earlier blocks
};

struct DecBlock {
    uint64_t off;    // offset of the block's data inside the frame
    uint32_t word;   // block header word (bit 31 = stored raw)
    uint32_t pad;
};

__device__ __forceinline__ uint32_t rd32(const uint8_t *p) {
    return p[0] | (p[1] << 8) | (p[2] << 16) | ((uint32_t)p[3] << 24);
}

// One thread per chunk.
__device__ __forceinline__ void frame_index(DecChunk &cd, DecBlock *tbl, int32_t *status) {
    const uint8_t *f = cd.frame;
    const uint64_t n = cd.frame_len;
    auto fail = [&](int32_t code) { *status = code; };
    if (n < 7 + 4) return fail(kDecTruncated);
    if (rd32(f) != 0x184D2204u) return fail(kDecBadHeader);
    const uint8_t flg = f[4], bd = f[5];
    if ((flg >> 6) != 1 || (flg & 0x02) || (bd & 0x8F)) return fail(kDecBadHeader);
    if (((bd >> 4) & 7) != 4) return fail(((bd >> 4) & 7) < 4 ? kDecBadHeader : kDecLayout);  // 64 KiB blocks only
    if (flg & 0x15) return fail(kDecUnsupported);  // block checksum / content checksum / dictID
    const bool has_size = flg & 0x08;
    const uint32_t hdr = 4 + 2 + (has_size ? 8 : 0) + 1;
    if (n < hdr + 4) return fail(kDecTruncated);
    uint8_t d[10];
    for (uint32_t i = 0; i < hdr - 5; i++) d[i] = f[4 + i];
    if ((uint8_t)(xxh32_small(d, hdr - 5) >> 8) != f[hdr - 1]) return fail(kDecBadHeader);
    if (has_size) {
        uint64_t cs = 0;
        for (int i = 0; i < 8; i++) cs |= (uint64_t)f[6 + i] << (8 * i);
        if (cs != cd.raw_len) return fail(kDecSize);
    }
    cd.linked = (flg & 0x20) ? 0u : 1u;
    uint64_t ip = hdr;
    for (uint32_t j = 0; j < cd.nblk; j++) {
        if (n - ip < 4) return fail(kDecTruncated);
        const uint32_t w = rd32(f + ip);
        ip += 4;
        const uint32_t sz = w & 0x7FFFFFFFu;
        if (w == 0) return fail(kDecSize);       // EndMark before all expected blocks
        if (sz > kBlock) return fail(kDecCorrupt);  // larger than the frame's block maximum
        if (n - ip < sz) return fail(kDecTruncated);
        tbl[j].off = ip;
        tbl[j].word = w;
        tbl[j].pad = 0;
        ip += sz;
    }
    if (n - ip < 4) return fail(kDecTruncated);
    if (rd32(f + ip) != 0) return fail(kDecSize);  // more blocks than the expected raw length allows
}

// Copy `n` bytes from `op - offset` to `op` (LZ4 match semantics: the source may overlap the destination).
__device__ __forceinline__ void warp_match_copy(uint8_t *op, uint32_t offset, uint32_t n, unsigned lane) {
    const uint8_t *s = op - offset;
    if (offset >= 32) {
        for (uint32_t base = 0; base < n; base += 32) {  // rounds of 32 bytes never read what the same round writes
            const uint32_t k = base + lane;
            uint8_t b = 0;
            if (k < n) b = s[k];
            __syncwarp();
            if (k < n) op[k] = b;
            __syncwarp();
        }
    } else {
        // period `offset` < 32: byte k of the match equals s[k mod offset], and those bytes are final already
        uint32_t ph = lane % offset;
        const uint32_t adv = 32u % offset;
        for (uint32_t k = lane; k < n; k += 32) {
            op[k] = s[ph];
            ph += adv;
            if (ph >= offset) ph -= offset;
        }
        __syncwarp();
    }
}

// One warp decodes one compressed block: src[0, slen) -> out[pos, pos + want); `low` = lowest output position a
// match may reference.  Returns kDecOk or an error; all lanes return the same value.
__device__ __forceinline__ int32_t lz4_decode_block(const uint8_t *src, uint32_t slen, uint8_t *out, uint64_t pos, uint32_t want,
                                                   uint64_t low, unsigned lane) {
    uint32_t ip = 0;
    uint64_t op = pos;
    const uint64_t oend = pos + want;
    if (slen == 0) return kDecCorrupt;
    for (;;) {
        if (ip >= slen) return kDecCorrupt;
        const uint32_t token = src[ip++];
        uint32_t ll = token >> 4;
        if (ll == 15) {
            uint32_t s;
            do {
                if (ip >= slen) return kDecCorrupt;
                s = src[ip++];
                ll += s;
            } while (s == 255 && ll < (1u << 24));
        }
        if (ll > slen - ip || op + ll > oend) return kDecCorrupt;
        warp_copy(out + op, src + ip, ll, lane);
        ip += ll;
        op += ll;
        if (ip == slen) break;  // last sequence: literals only
        if (slen - ip < 2) return kDecCorrupt;
        const uint32_t offset = src[ip] | (src[ip + 1] << 8);
        ip += 2;
        if (offset == 0 || offset > op - low) return kDecCorrupt;
        uint32_t ml = token & 15;
        if (ml == 15) {
            uint32_t s;
            do {
                if (ip >= slen) return kDecCorrupt;
                s = src[ip++];
                ml += s;
            } while (s == 255 && ml < (1u << 24));
        }
        ml += kMinMatch;
        if (op + kMfLimit > oend || op + ml + kLastLiterals > oend) return kDecCorrupt;  // end-of-block rules
        __syncwarp();  // the literals just written may be the match source
        warp_match_copy(out + op, offset, ml, lane);
        op += ml;
    }
    return op == oend ? kDecOk : kDecLayout;
}

}  // namespace sky
