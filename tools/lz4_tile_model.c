/*
 * lz4_tile_model.c -- sequential CPU twin of the round-2 GPU block compressor (skyplane_b200/csrc/lz4.cuh).
 *
 * NOT the reference's algorithm (that is oracle/skyoracle.c) and NOT product code: a development tool.  It replays the
 * kernel's parse on the host, byte for byte, so (a) design options can be compared for compression ratio without a GPU
 * (tools/tile_study.py) and (b) the GPU output can be diffed against a sequential implementation of the same rules
 * (tests/test_tools_model.py, tests/test_gpu_parity.py::test_frames_equal_sequential_twin).
 *
 * The parse, per 64 KiB block (the kernel runs it with one CTA per block: a prober warp and several parser warps):
 *   segment = seg_slots probe slots, slot i at position seg_pos + (i << slog); segments tile the block back to back.
 *             slog starts at 0 for the first two segments; segment s+2's slog is 0 if segment s had any hit, else segment
 *             s+1's slog plus one (up to max_step_log) -- one segment of delay, so the kernel's two prober warps never
 *             wait for each other's verdict.
 *   probe   = 32 slots (a group) at a time: hash 5 bytes, look the table entry (pos16 | tag16) up; hit = tag equal and
 *             entry older than the slot.  A slot whose full 32-bit hash equals that of the slot 3, 4 or 8 places before it
 *             in the same group takes that one as its candidate instead (short periods: pixels, words, doubles -- the
 *             table cannot know them yet).  Then the group's slots replace their table entries, the last one staying.
 *             No byte of the candidate is read here.
 *   parse   = per segment, independently of every other segment: cursor and anchor start at the segment start; walk the
 *             hits at or after the cursor; measure the real match length from byte 0 (this is also the verification),
 *             clipped to the segment end (and to the block's last-5-bytes rule); drop it if < 4; extend backwards by up
 *             to 8 bytes but not past the anchor; record the sequence; cursor = anchor = match end.
 *   emit    = the block's sequences are the segments' sequences in order; literals a segment leaves behind its last match
 *             (or a whole segment without a match) are carried into the next sequence.  Standard LZ4 block format.
 *             A block whose compressed size would exceed L-1 is stored raw (return 0), as LZ4F_makeBlock does.
 *
 * Linked blocks (tile_compress_block_linked): the block is parsed in a buffer [window | block] whose window is the W raw
 * bytes before the block.  All positions are window coordinates; the table holds them modulo 65536 (pos16), so an offset
 * is (position - entry) mod 65536, which keeps every offset in 1..65535.  Before the block's first segment the table is
 * seeded with the window positions 0, s, 2s, ... (s = 1 << seed_step_log), inserted in order without reporting hits.
 * After that the parse is the one above: candidates may lie in the window, a match that starts there may run on into the
 * block, backward extension stops at min(pos - anchor, cand, 8).  With W = 0 it is tile_compress_block exactly.
 *
 * Build: gcc -O2 -shared -fPIC -o tools/bin/liblz4tile.so tools/lz4_tile_model.c
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define MINMATCH 4
#define MFLIMIT 12
#define LASTLITERALS 5

typedef struct {
    int entries;       /* table entries (kernel: 4096; index = mulhi(hash, entries)) */
    int seg_slots;     /* probe slots per segment (kernel: 1024) */
    int max_step_log;  /* largest probe stride = 1 << this (kernel: 4) */
    int back_ext;      /* 1 = extend accepted matches backwards by up to 8 bytes (kernel: 1) */
    int clip;          /* 1 = matches end at the segment end (kernel: 1; 0 shows what the segment independence costs) */
    int group_lag;     /* 1 = the 32 slots of a group all look the table up before any of them is inserted (kernel: 1);
                          0 = every slot sees the slots before it (study variant: what a fully sequential probe would find) */
    int near_mask;     /* with group_lag: bit d-1 set = a slot also compares its 5-byte hash with the slot d places before it
                          in its group; the nearest equal one is its candidate, ahead of the table's (kernel: 0x8c = 3, 4, 8) */
} tile_opts;

static uint32_t rd32(const uint8_t *p) { uint32_t v; memcpy(&v, p, 4); return v; }

static uint32_t emit(uint8_t *out, uint32_t op, const uint8_t *src, uint32_t anchor, uint32_t ll, uint32_t ml, uint32_t off) {
    uint32_t mcode = ml ? ml - MINMATCH : 0;
    out[op++] = (uint8_t)(((ll < 15 ? ll : 15) << 4) | (mcode < 15 ? mcode : 15));
    if (ll >= 15) { uint32_t r = ll - 15; for (; r >= 255; r -= 255) out[op++] = 255; out[op++] = (uint8_t)r; }
    memcpy(out + op, src + anchor, ll); op += ll;
    if (ml) {
        out[op++] = (uint8_t)off; out[op++] = (uint8_t)(off >> 8);
        if (mcode >= 15) { uint32_t r = mcode - 15; for (; r >= 255; r -= 255) out[op++] = 255; out[op++] = (uint8_t)r; }
    }
    return op;
}

static uint32_t hash5(const uint8_t *p) { return rd32(p) * 2654435761u + p[4] * 0x85EBCA6Bu; }  /* 5 bytes, two 32-bit multiplies */
static uint32_t hidx(uint32_t hf, const tile_opts *o) { return (uint32_t)(((uint64_t)hf * (uint32_t)o->entries) >> 32); }
static uint32_t htag(uint32_t hf) { return (hf >> 8) & 0xffffu; }  /* hash bytes 1-2: one PRMT in the kernel */

typedef struct { uint64_t probes, hits, accepted, segments; } tile_stats;
static tile_stats g_stats;
void tile_model_stats(tile_stats *s, int reset) { *s = g_stats; if (reset) memset(&g_stats, 0, sizeof g_stats); }

/* The block is src[base .. base + BL); src[0 .. base) is its window.  Positions are window coordinates (base = 0: block
 * coordinates).  Returns compressed size, or 0 if the block does not shrink (store raw); out capacity >= BL + 2048. */
static uint32_t compress_block_at(const uint8_t *src, uint32_t base, uint32_t BL, uint8_t *out, const tile_opts *o, int seed_step_log) {
    const uint32_t S = (uint32_t)o->seg_slots, limit = BL - 1, L = base + BL;
    uint32_t *tab = calloc((size_t)o->entries, 4);  /* pos16 | tag << 16 ; 0 = (pos 0, tag 0) = "empty" */
    uint16_t *off = malloc(2 * S);
    uint8_t *hit = malloc(S);
    uint32_t anchor = base /* start of the literals not yet emitted */, op = 0, result = 0;
    uint32_t ghf[32];
    if (BL >= MFLIMIT + 1) {
        const uint32_t mflimit = L - MFLIMIT, matchlimit = L - LASTLITERALS;
        for (uint32_t q = 0; q < base; q += 1u << seed_step_log) {  /* window seeding: inserts only, the last one stays */
            const uint32_t hf = hash5(src + q);
            tab[hidx(hf, o)] = (q & 0xffffu) | (htag(hf) << 16);
        }
        uint32_t seg_pos = base, slog = 0, slog_next = 0;  /* slog of this segment / of the next one */
        while (seg_pos <= mflimit) {
            g_stats.segments++;
            /* ---- probe, one group of 32 slots at a time */
            int anyhit = 0;
            for (uint32_t g = 0; g < S; g += 32) {
                for (uint32_t i = g; i < g + 32; i++) {
                    const uint32_t p = seg_pos + (i << slog);
                    hit[i] = 0;
                    ghf[i - g] = 0;
                    if (p > mflimit) continue;
                    const uint32_t hf = hash5(src + p);
                    const uint32_t e = tab[hidx(hf, o)], eoff = (p - e) & 0xffffu;  /* (p - entry) mod 65536 */
                    ghf[i - g] = hf;
                    g_stats.probes++;
                    if ((e >> 16) == htag(hf) && eoff != 0) { hit[i] = 1; off[i] = (uint16_t)eoff; }
                    if (o->group_lag) {  /* an equal hash 3, 4 or 8 slots back in the group is the nearer candidate */
                        for (uint32_t d = 1; d <= i - g; d++)
                            if ((((uint32_t)o->near_mask >> (d - 1)) & 1u) && ghf[i - g - d] == hf) { hit[i] = 1; off[i] = (uint16_t)(d << slog); break; }
                    } else tab[hidx(hf, o)] = (p & 0xffffu) | (htag(hf) << 16);
                    if (hit[i]) { anyhit = 1; g_stats.hits++; }
                }
                if (o->group_lag)  /* the group's slots replace the table entries in slot order (the last one stays) */
                    for (uint32_t i = g; i < g + 32; i++) {
                        const uint32_t p = seg_pos + (i << slog);
                        if (p <= mflimit) tab[hidx(ghf[i - g], o)] = (p & 0xffffu) | (htag(ghf[i - g]) << 16);
                    }
            }
            /* ---- parse: depends on nothing outside this segment */
            const uint32_t seg_lim = seg_pos + (S << slog);  /* first byte of the next segment */
            const uint32_t mlim = (o->clip && seg_lim < matchlimit) ? seg_lim : matchlimit;
            uint32_t cur = seg_pos, lanchor = seg_pos;  /* local cursor / anchor */
            if (!o->clip && anchor > seg_pos) cur = lanchor = anchor;  /* (study variant: one parse across segments) */
            for (uint32_t i = 0; i < S; i++) {
                if (!hit[i]) continue;
                uint32_t pos = seg_pos + (i << slog);
                if (pos < cur || pos >= mlim) continue;
                uint32_t cand = pos - off[i];
                const uint32_t maxlen = mlim - pos;
                uint32_t mlen = 0;
                while (mlen < maxlen && src[pos + mlen] == src[cand + mlen]) mlen++;
                if (mlen < MINMATCH) continue;
                if (o->back_ext) {
                    uint32_t room = pos - lanchor;
                    if (cand < room) room = cand;
                    if (room > 8) room = 8;
                    uint32_t b = 0;
                    while (b < room && src[pos - 1 - b] == src[cand - 1 - b]) b++;
                    pos -= b; cand -= b; mlen += b;
                }
                op = emit(out, op, src, anchor, pos - anchor, mlen, pos - cand);
                anchor = cur = lanchor = pos + mlen;
                g_stats.accepted++;
                if (op > BL + 1024) goto done;  /* (model only) hopeless and about to overrun the caller's buffer */
            }
            seg_pos = seg_lim;
            {   /* this segment's verdict decides the stride two segments on */
                const uint32_t after = anyhit ? 0 : (slog_next < (uint32_t)o->max_step_log ? slog_next + 1 : slog_next);
                slog = slog_next;
                slog_next = after;
            }
        }
    }
    if (L - anchor + (L - anchor) / 255 + 2 + op <= BL + 2040) op = emit(out, op, src, anchor, L - anchor, 0, 0);
    else op = BL;  /* cannot fit anyway */
    if (op <= limit) result = op;
done:
    free(tab); free(off); free(hit);
    return result;
}

/* returns compressed size, or 0 if the block does not shrink (store raw); out capacity >= L + 2048 */
uint32_t tile_compress_block(const uint8_t *src, uint32_t L, uint8_t *out, const tile_opts *o) {
    return compress_block_at(src, 0, L, out, o, 0);
}

/* Linked block: win = the win_len raw bytes just before src (the previous block's tail; win_len 0 for a frame's first block).
 * Same return value and out capacity as tile_compress_block. */
uint32_t tile_compress_block_linked(const uint8_t *win, uint32_t win_len, const uint8_t *src, uint32_t L, uint8_t *out,
                                    const tile_opts *o, int seed_step_log) {
    uint8_t *buf = malloc((size_t)win_len + L + 1);
    memcpy(buf, win, win_len);
    memcpy(buf + win_len, src, L);
    const uint32_t r = compress_block_at(buf, win_len, L, out, o, seed_step_log);
    free(buf);
    return r;
}
