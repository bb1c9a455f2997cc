/*
 * skychunk.h -- C ABI of the B200 chunk-processing stage (libskychunk.so).
 *
 * Drop-in boundary for the per-chunk hot path of Skyplane's gateway.  The reference has no FFI
 * (it is pure Python); these entry points replace, for one batch of chunks, the two calls
 *     data = lz4.frame.compress(data)          skyplane/gateway/operators/gateway_operator.py:358-361
 *     m = hashlib.md5(); m.update(b); digest   skyplane/obj_store/s3_interface.py:181-192
 * and hand back exactly what the sender needs for its wire header (gateway_operator.py:367-372):
 * the frame bytes, their length, and the 16-byte digest for Chunk.md5_hash (skyplane/chunk.py:21).
 *
 * Conventions: plain pointers and sizes, no exceptions, 0 = success / negative = error code.
 * The caller owns every host buffer; the library owns device memory, streams and events.
 * One sky_ctx per process per GPU; calls on one ctx are not thread-safe (the reference runs one
 * process per worker, gateway_operator.py:66-70).  A ctx must be created in the process that uses
 * it (after fork), never inherited.
 *
 * Output format: one LZ4 frame per chunk that lz4.frame.decompress (gateway_receiver.py:196)
 * restores bit-exactly: magic, FLG=0x68 (v01, independent blocks, content size), BD=0x40 (64 KiB),
 * u64le content size, header checksum, blocks (bit 31 set = stored raw), EndMark.  A zero-length
 * chunk yields the 11-byte frame liblz4 itself emits (content size omitted).  SKY_F_LINKED: FLG=0x48 (linked blocks).
 */
#ifndef SKYCHUNK_H
#define SKYCHUNK_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SKY_API __attribute__((visibility("default")))
#else
#define SKY_API
#endif

#define SKY_ABI_VERSION 2

/* error codes */
#define SKY_OK 0
#define SKY_E_INVALID (-1)   /* bad argument (null pointer, misaligned device pointer, n == 0 ...) */
#define SKY_E_NOGPU (-2)     /* no CUDA device / driver: there is NO CPU fallback */
#define SKY_E_CUDA (-3)      /* a CUDA call failed; see sky_last_error() */
#define SKY_E_CAPACITY (-4)  /* batch exceeds what the ctx was created for, or dst_cap < sky_frame_bound() */
#define SKY_E_BUSY (-5)      /* all slots hold un-waited tickets */
#define SKY_E_TICKET (-6)    /* unknown / already consumed ticket */
#define SKY_E_NOMEM (-7)
#define SKY_E_NOKEY (-8)     /* SKY_F_E2EE without sky_set_e2ee_key() / without nonces */

/* stage selection (0 = LZ4 + MD5).  SKY_F_MD5 alone is the reference's `compress: false` (gateway_daemon.py:235,
 * gateway_operator.py:358): the chunk is digested and passes through uncompressed. */
#define SKY_F_LZ4 1u
#define SKY_F_MD5 2u
/* accepted and ignored since ABI 2 (round 1 kept an SM sub-partition free for each MD5 warp; digest groups now run in
 * CTAs of their own) */
#define SKY_F_MD5_EXCLUSIVE 4u
/* do not pace LZ4 work to the MD5 lanes' progress (pacing lets the lanes read the input from L2; sky_submit always
 * runs unpaced so that the kernels of different slots overlap) */
#define SKY_F_NO_PACING 8u
/* end-to-end encryption behind the frame (sky_submit_flags / sky_decode_flags): every payload becomes PyNaCl's
 * SecretBox.encrypt() message  nonce(24) | tag(16) | ciphertext  (XSalsa20-Poly1305), as GatewaySender does with
 * e2ee_key_bytes (gateway_operator.py:183-186, :362-364) and the receiver undoes (gateway_receiver.py:191-193). */
#define SKY_F_E2EE 16u
#define SKY_BOX_OVERHEAD 40u
/* linked blocks (sky_submit_flags / sky_process_device): a block's matches may also reach into the 4 KiB of input before
 * it (sky_kernel_config(4)), as the reference's frames do -- FLG 0x48 instead of 0x68 for chunks of more than one block,
 * a better ratio on text, and the receiver decodes the blocks of a chunk in order.  A chunk of at most 64 KiB gets the
 * same FLG as liblz4 gives it (0x68).  Composes with SKY_F_E2EE (the box holds the linked frame); no effect without
 * SKY_F_LZ4.  sky_frame_bound / sky_box_bound are unchanged. */
#define SKY_F_LINKED 32u

typedef struct sky_ctx sky_ctx;

SKY_API const char *sky_strerror(int code);
/* Detail of the latest failed call on this ctx.  ctx = NULL: of the latest failed call on this thread that had no ctx
 * (sky_ctx_create, the device queries, sky_pinned_alloc / sky_pinned_free, a NULL ctx argument). */
SKY_API const char *sky_last_error(const sky_ctx *ctx);
SKY_API int sky_abi_version(void);
SKY_API int sky_device_count(int *count);
/* PCI bus id ("0000:1b:00.0") of CUDA device `device` as the CUDA runtime orders devices (honours CUDA_VISIBLE_DEVICES,
 * unlike nvidia-smi -i); the host side maps it to the GPU's NUMA node before pinning staging memory. */
SKY_API int sky_device_pci_bus_id(int device, char *buf, int len);
/* Compile-time constants of the kernels in this build (tuning builds differ): what = 0 -> LZ4 match-table entries per
 * CTA, 1 -> warps per CTA of the fused kernel, 2 -> probe slots per segment, 3 -> log2 of the largest probe stride,
 * 4 -> SKY_F_LINKED window bytes (0 = no linked mode in this build), 5 -> log2 of the stride at which the window seeds
 * the match table, 6 -> match-table entries in linked mode.  Unknown `what` returns 0.  Parity tests feed these to the sequential twin of the compressor (tools/lz4_tile_model.c). */
SKY_API uint32_t sky_kernel_config(int what);

/* Worst-case frame bytes for an n-byte chunk: 15 + n + 4*ceil(n/65536) + 4 (11 when n == 0). */
SKY_API uint64_t sky_frame_bound(uint64_t n);

/* Create a context on `device` able to hold batches of up to max_chunks chunks totalling
 * max_batch_bytes input bytes.  n_slots >= 1 batches may be in flight through sky_submit at once
 * (each slot owns an input slab, an output slab and a stream); n_slots == 0 creates a ctx for
 * sky_process_device only (no slabs). */
SKY_API int sky_ctx_create(int device, uint64_t max_batch_bytes, uint32_t max_chunks, uint32_t n_slots, sky_ctx **out);
SKY_API int sky_ctx_destroy(sky_ctx *ctx);

/* Page-locked host memory for staging chunk bytes (cudaHostAlloc, portable). */
SKY_API void *sky_pinned_alloc(uint64_t bytes);
SKY_API int sky_pinned_free(void *p);

/* ---- host-buffer path (what GatewayOperator.process uses) -------------------------------------
 * sky_submit: asynchronously copies n chunks host->device, runs the fused kernel, and stages the
 *   per-chunk sizes and digests back.  src[i]/src_len[i] = chunk bytes; dst[i]/dst_cap[i] = where
 *   the frame goes (dst_cap[i] >= sky_frame_bound(src_len[i])).  All host buffers must stay valid
 *   until sky_wait returns.  Pinned buffers make the copies truly asynchronous.
 * sky_wait: blocks until the batch is done, copies each frame device->host (exact length), and
 *   fills out_len[n], md5[16*n].  kernel_ms (optional) = device time of the fused kernel. */
SKY_API int sky_submit(sky_ctx *ctx, uint32_t n, const void *const *src, const uint64_t *src_len, void *const *dst,
               const uint64_t *dst_cap, uint64_t *ticket);
SKY_API int sky_wait(sky_ctx *ctx, uint64_t ticket, uint64_t *out_len, uint8_t *md5, float *kernel_ms);
/* sky_submit with stage flags.  flags = SKY_F_MD5: digests only (dst / dst_cap may be NULL, out_len comes back 0: the
 *   caller forwards its own input bytes, is_compressed = False).  | SKY_F_E2EE: what comes back in dst[i] is the sealed
 *   box of the frame (or of the raw chunk when SKY_F_LZ4 is off), out_len[i] = its length = payload + SKY_BOX_OVERHEAD,
 *   dst_cap[i] >= sky_box_bound(src_len[i]); nonces = 24 bytes per chunk chosen by the caller (nacl.utils.random(24)).
 *   The key is the ctx's (sky_set_e2ee_key; key32 = NULL switches E2EE off). */
SKY_API int sky_submit_flags(sky_ctx *ctx, uint32_t n, const void *const *src, const uint64_t *src_len, void *const *dst,
                     const uint64_t *dst_cap, uint32_t flags, const uint8_t *nonces, uint64_t *ticket);
SKY_API int sky_set_e2ee_key(sky_ctx *ctx, const uint8_t *key32);
SKY_API uint64_t sky_box_bound(uint64_t n); /* sky_frame_bound(n) + SKY_BOX_OVERHEAD */

/* ---- device-resident path (kernel metric; inputs already in HBM) ------------------------------
 * Chunk i is d_src[src_off[i] .. +src_len[i]) ; its frame is written at d_dst + dst_off[i]
 * (capacity dst_cap[i] >= sky_frame_bound(src_len[i])).  src_off/dst_off must be multiples of 16
 * and both regions must be readable/writable up to the next multiple of 16.  `stream` is a
 * cudaStream_t (NULL = the ctx's own stream).  Synchronous: returns after the results are on the
 * host.  flags: SKY_F_* (0 = LZ4 + MD5). */
SKY_API int sky_process_device(sky_ctx *ctx, uint32_t n, const void *d_src, const uint64_t *src_off, const uint64_t *src_len,
                       void *d_dst, const uint64_t *dst_off, const uint64_t *dst_cap, uint32_t flags, void *stream,
                       uint64_t *out_len, uint8_t *md5, float *kernel_ms);

/* ---- receiver side: LZ4 frame decode + digest of the decoded bytes -----------------------------------
 * Replaces lz4.frame.decompress(to_write) (skyplane/gateway/operators/gateway_receiver.py:195-201) and supplies
 * the digest for the "# todo check hash" at gateway_receiver.py:231.  raw_len[i] is the expected decoded size
 * (WireProtocolHeader.raw_data_len, skyplane/chunk.py:100).  Accepts the frames this library emits (independent
 * 64 KiB blocks) and the reference sender's (linked blocks); status[i] = 0 or a SKY_D_* code (a bad frame is an
 * error status, never a crash); md5[16*i..] = MD5 of the decoded bytes.
 * sky_decode_device: frames and output already in HBM (out_off multiples of 16; each frame region must be readable
 * up to the next multiple of 4 bytes, each output region writable up to the next multiple of 16).  sky_decode: host
 * buffers, synchronous, through slot 0's slabs (needs n_slots >= 1). */
#define SKY_D_OK 0
#define SKY_D_BAD_HEADER (-1)
#define SKY_D_CORRUPT (-2)
#define SKY_D_SIZE (-3)
#define SKY_D_UNSUPPORTED (-4)
#define SKY_D_LAYOUT (-5)
#define SKY_D_TRUNCATED (-6)
#define SKY_D_AUTH (-7) /* SKY_F_E2EE: the box's Poly1305 tag does not verify (nacl.exceptions.CryptoError in the reference) */
SKY_API int sky_decode_device(sky_ctx *ctx, uint32_t n, const void *d_frames, const uint64_t *frame_off, const uint64_t *frame_len,
                      void *d_out, const uint64_t *out_off, const uint64_t *raw_len, void *stream, int32_t *status, uint8_t *md5,
                      float *kernel_ms);
SKY_API int sky_decode(sky_ctx *ctx, uint32_t n, const void *const *frames, const uint64_t *frame_len, void *const *dst,
               const uint64_t *raw_len, int32_t *status, uint8_t *md5, float *kernel_ms);
/* sky_decode with flags: SKY_F_E2EE = the payloads are sealed boxes; tags are checked and the boxes opened on the device
 * before the frames are decoded (status SKY_D_AUTH for a forged / truncated box, whose bytes are never returned). */
SKY_API int sky_decode_flags(sky_ctx *ctx, uint32_t n, const void *const *frames, const uint64_t *frame_len, void *const *dst,
                     const uint64_t *raw_len, uint32_t flags, int32_t *status, uint8_t *md5, float *kernel_ms);

/* Device-memory helpers so a host without torch can drive the device path. */
SKY_API int sky_device_alloc(sky_ctx *ctx, uint64_t bytes, void **dptr);
SKY_API int sky_device_free(sky_ctx *ctx, void *dptr);
SKY_API int sky_memcpy_h2d(sky_ctx *ctx, void *dptr, const void *host, uint64_t bytes);
SKY_API int sky_memcpy_d2h(sky_ctx *ctx, void *host, const void *dptr, uint64_t bytes);

/* Number of kernel launches issued through this ctx so far (bench.py's gpu_launches). */
SKY_API uint64_t sky_launch_count(const sky_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* SKYCHUNK_H */
