/*
 * lz4b200.h -- C ABI of liblz4b200.so: the B200 (sm_100a) LZ4 r93 block codec behind lz4net's service boundary.
 *
 * This is the drop-in boundary of the path (SURVEY.md 8b).  lz4net's native services (LZ4mm / LZ4cc) reach the
 * codec through exactly four C functions (src/LZ4cc/LZ4Codec.64.cpp:35,88,95,143 -> original/lz4.h:59-60,101,116,
 * original/lz4hc.h:57); a `CudaLZ4Service : ILZ4Service` (src/LZ4/ILZ4Service.cs:30-36) binds the entry points
 * below with [DllImport] exactly like CppMM64LZ4Service (src/LZ4/Services/CppMM64LZ4Service.cs:38-51) binds those.
 * INTEGRATION.md shows the managed stub.  Plain pointers and sizes only; no torch / CUDA types in any signature
 * (a `void* stream` is a cudaStream_t passed opaquely; NULL = the CUDA default stream, as everywhere in CUDA).
 *
 * Conventions shared with the reference:
 *   - encoders return bytes written, 0 = output too small / failed              (original/lz4.h:48-60)
 *   - known-size decode returns bytes READ from the source, < 0 = malformed     (original/lz4.h:96-101)
 *   - unknown-size decode returns bytes WRITTEN, < 0 = malformed                (original/lz4.h:104-116)
 *   - compressed bytes are identical to lz4net's LZ4Codec.Encode / EncodeHC on the same input
 * There is no CPU fallback: every entry point fails (LZ4B200_E_*) when no sm_100 device / kernel image is usable.
 */
#ifndef LZ4B200_H
#define LZ4B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LZ4B200_VERSION 100            /* 0.1.0 */

/* encoder selection (ILZ4Service.Encode vs EncodeHC, src/LZ4/ILZ4Service.cs:33-34) */
#define LZ4B200_MODE_FAST 0
#define LZ4B200_MODE_HC   1

/* where the buffers of a batch call live */
#define LZ4B200_MEM_HOST   0           /* src/dst/offset/length arrays are host memory; copies are inside the call */
#define LZ4B200_MEM_DEVICE 1           /* everything is device memory on the context's GPU; the call only enqueues */

/* status codes (batch / context calls).  Per-block results are reported in out_len[], never here. */
#define LZ4B200_OK            0
#define LZ4B200_E_ARG        -1
#define LZ4B200_E_NODEVICE   -2        /* no CUDA device, or not compute capability 10.x */
#define LZ4B200_E_CUDA       -3        /* a CUDA runtime call failed; see lz4b200_last_error() */
#define LZ4B200_E_NOMEM      -4
#define LZ4B200_E_FORMAT     -5        /* malformed LZ4Stream / Wrap framing, or a chunk that does not decode */

typedef struct lz4b200_ctx lz4b200_ctx;

int         lz4b200_version(void);
const char* lz4b200_last_error(void);                 /* thread-local, never NULL */
int         lz4b200_device_count(void);               /* usable (cc 10.x) devices; 0 if none */

/* A context owns one device's stream, scratch (HC chain tables, staging) and tuning knobs.  Unlike the reference
 * (stateless: tables are allocated per call, src/LZ4ps/LZ4Codec.Safe.cs:407) the GPU path has state.
 * Contexts are internally locked: one batch call at a time per context; use one context per caller thread/GPU. */
int  lz4b200_create(lz4b200_ctx** out, int device);
void lz4b200_destroy(lz4b200_ctx* ctx);
int  lz4b200_synchronize(lz4b200_ctx* ctx);           /* wait for everything enqueued through this context */

/* LZ4_compressBound (original/lz4.h:85) == LZ4Codec.MaximumOutputLength (src/LZ4/LZ4Codec.cs:313-316) */
int  lz4b200_compress_bound(int input_size);

/* ---- batched entry points: n_blocks independent blocks, one launch -------------------------------------------
 * Block i reads  src + src_off[i], src_len[i] bytes   and writes at  dst + dst_off[i], at most dst_cap[i] bytes.
 * out_len[i] receives the per-block return value of the corresponding single-block function below.
 *
 * encode:  LZ4_compress_limitedOutput / LZ4_compressHC_limitedOutput semantics per block (0 = did not fit).
 * decode:  known_len != 0 -> LZ4_uncompress (dst_cap[i] is the exact decoded size; out_len[i] = bytes read,
 *                            the caller compares it with src_len[i] like src/LZ4cc/LZ4Codec.64.cpp:88-93);
 *          known_len == 0 -> LZ4_uncompress_unknownOutputSize (dst_cap[i] = capacity; out_len[i] = bytes written).
 * MEM_DEVICE: asynchronous on `stream`; MEM_HOST: synchronous, chunked + overlapped copies inside the call.
 * Returns LZ4B200_OK or a negative status; malformed / too-small blocks are NOT a call failure. */
int lz4b200_encode_batch(lz4b200_ctx* ctx,
                         const void* src, const int64_t* src_off, const int32_t* src_len,
                         void* dst, const int64_t* dst_off, const int32_t* dst_cap,
                         int32_t* out_len, int32_t n_blocks, int mode, int mem, void* stream);

int lz4b200_decode_batch(lz4b200_ctx* ctx,
                         const void* src, const int64_t* src_off, const int32_t* src_len,
                         void* dst, const int64_t* dst_off, const int32_t* dst_cap,
                         int32_t* out_len, int32_t n_blocks, int known_len, int mem, void* stream);

/* Host-memory encode with PACKED output: block i's compressed bytes land at dst + out_off[i] (out_off has n_blocks+1
 * entries; out_off[n_blocks] = total bytes written <= dst_total_cap), back to back in block order -- the layout the
 * LZ4Stream chunk writer (src/LZ4/LZ4Stream.cs:262-266) and any transport want, and the one that moves only compLen
 * bytes per block back over PCIe.  dst_cap[i] is still the per-block limit of LZ4_compress_limitedOutput (a block that
 * does not fit reports out_len[i] = 0 and occupies no bytes). */
int lz4b200_encode_batch_packed(lz4b200_ctx* ctx,
                                const void* src, const int64_t* src_off, const int32_t* src_len, const int32_t* dst_cap,
                                void* dst, int64_t dst_total_cap, int64_t* out_off, int32_t* out_len,
                                int32_t n_blocks, int mode);

/* Compaction of fixed-stride encoder slots into one contiguous payload (device memory only): the batched form of
 * the Buffer.BlockCopy trim in LZ4Codec.Encode (src/LZ4/LZ4Codec.cs:357-364).  out_off[i] (int64, n_blocks+1
 * entries) = exclusive prefix sum of max(len[i],0); block i's bytes are copied to packed + out_off[i]. */
int lz4b200_compact(lz4b200_ctx* ctx, const void* slots, const int64_t* slot_off, const int32_t* len,
                    void* packed, int64_t* out_off, int32_t n_blocks, void* stream);

/* ---- single-block entry points (host pointers), 1:1 with the reference's native API -------------------------- */
/* original/lz4.h:59-60  LZ4_compress_limitedOutput */
int lz4b200_compress_limitedOutput(const char* source, char* dest, int isize, int maxOutputSize);
/* original/lz4hc.h:57   LZ4_compressHC_limitedOutput */
int lz4b200_compressHC_limitedOutput(const char* source, char* dest, int isize, int maxOutputSize);
/* original/lz4.h:101    LZ4_uncompress.  `isize` (the compressed length every managed caller holds,
 * src/LZ4pn/LZ4Codec.Unsafe.cs:366-371) is added because the bytes must be staged to the device; reads never pass it. */
int lz4b200_uncompress(const char* source, char* dest, int isize, int osize);
/* original/lz4.h:116    LZ4_uncompress_unknownOutputSize */
int lz4b200_uncompress_unknownOutputSize(const char* source, char* dest, int isize, int maxOutputSize);

/* ---- framing built on the batch calls ("next" rows of SURVEY.md 8f) ------------------------------------------
 * LZ4Stream chunk format (src/LZ4/LZ4Stream.cs:239-312): varint(flags) varint(rawLen) [varint(compLen)] payload.
 * stream_encode cuts `src` into block_size chunks, encodes all of them in one batch and writes the exact byte
 * stream an LZ4Stream(..., Compress, highCompression, block_size) would have produced for one Write + Close.
 * Returns bytes written, or a negative status (LZ4B200_E_ARG if dst_cap is too small / the stream is malformed). */
int64_t lz4b200_stream_bound(int64_t n, int32_t block_size);
int64_t lz4b200_stream_encode(lz4b200_ctx* ctx, const void* src, int64_t n, int32_t block_size, int high_compression,
                              void* dst, int64_t dst_cap);
int64_t lz4b200_stream_decoded_size(const void* src, int64_t n);     /* sum of rawLen over all chunks, <0 = malformed */
int64_t lz4b200_stream_decode(lz4b200_ctx* ctx, const void* src, int64_t n, void* dst, int64_t dst_cap);

/* LZ4Stream framing on device memory (src, dst on the context's GPU).  Ordered on `stream`: the call waits for
 * work already queued there, and returns once its result is known.
 * Each call returns exactly what its host twin above returns for the same bytes -- bytes written, the total raw size,
 * LZ4B200_E_ARG (dst_cap below lz4b200_stream_bound / below the total; no byte of dst is written then) or
 * LZ4B200_E_FORMAT -- and the encoder writes the same bytes.  src and dst may have any alignment; no byte outside
 * [src, src + n) is parsed.  The compressed bytes never cross PCIe: only the sizes come back to the host.
 * decoded_size walks the chunk headers on the device (one thread: each header's position depends on the one before);
 * decode walks them again, then copies the stored chunks and decodes all compressed ones in one batch. */
int64_t lz4b200_stream_encode_device(lz4b200_ctx* ctx, const void* src, int64_t n, int32_t block_size,
                                     int high_compression, void* dst, int64_t dst_cap, void* stream);
int64_t lz4b200_stream_decoded_size_device(lz4b200_ctx* ctx, const void* src, int64_t n, void* stream);
int64_t lz4b200_stream_decode_device(lz4b200_ctx* ctx, const void* src, int64_t n, void* dst, int64_t dst_cap, void* stream);

/* LZ4Codec.Wrap / Unwrap packet (src/LZ4/LZ4Codec.cs:510-543,574-599): u32le rawLen, u32le storedLen, payload. */
int lz4b200_wrap(lz4b200_ctx* ctx, const void* src, int32_t n, int high_compression, void* dst, int32_t dst_cap);
int lz4b200_unwrap_size(const void* src, int32_t n);
int lz4b200_unwrap(lz4b200_ctx* ctx, const void* src, int32_t n, void* dst, int32_t dst_cap);

/* The same for n packets at once: ONE encode / decode batch instead of one H2D + launch + D2H per packet.  Packet i is
 * byte for byte what lz4b200_wrap makes of input i.  wrap_batch: dst_cap[i] >= src_len[i] + 8; out_len[i] = packet size.
 * unwrap_batch: dst_cap[i] >= lz4b200_unwrap_size(packet i); out_len[i] = bytes restored or a negative status. */
int lz4b200_wrap_batch(lz4b200_ctx* ctx, const void* src, const int64_t* src_off, const int32_t* src_len, int high_compression,
                       void* dst, const int64_t* dst_off, const int32_t* dst_cap, int32_t* out_len, int32_t n);
int lz4b200_unwrap_batch(lz4b200_ctx* ctx, const void* src, const int64_t* src_off, const int32_t* src_len,
                         void* dst, const int64_t* dst_off, const int32_t* dst_cap, int32_t* out_len, int32_t n);

/* ---- host buffers the caller keeps for a while (a pinned byte[] behind a GCHandle, a native arena) --------------------
 * Host-memory batches copy straight from / to the caller's buffers.  From pageable memory the driver stages every copy
 * through its own pinned bounce buffers, synchronously; page-locking a long-lived buffer once (cudaHostRegister) lets the
 * same calls run at the full pipelined rate.  Optional: everything works without it. */
int lz4b200_host_register(void* ptr, int64_t bytes);
int lz4b200_host_unregister(void* ptr);

/* ---- one stream, several GPUs of one node (BASELINE configs[3]; lz4net_b200/shard.py StreamWindow) --------------------
 * Asynchronous copy between device buffers of two GPUs (either side may be memory another process exported with CUDA
 * IPC), ordered on `stream` of the CURRENT device, executed by the copy engines over NVLink -- it overlaps codec kernels,
 * which a send/recv kernel of a communication library does not.  Enables peer access on first use. */
int lz4b200_peer_copy(void* dst, const void* src, int64_t bytes, void* stream);

/* ---- synthetic workload generator (bench/test utility; device memory) ----------------------------------------
 * Fills n_blocks * block_size bytes at dst with entropy class cls (0 E0, 1 E50, 2 E100, 3 ETEXT), block index
 * first_block + i, exactly as lz4net_b200/synth.py defines them. */
int lz4b200_synth_fill(lz4b200_ctx* ctx, void* dst, int64_t n_blocks, int32_t block_size, int cls, uint64_t seed,
                       int64_t first_block, void* stream);

/* Tuning knobs (bench / profiling only).  key: "decode_lanes" (4|8|16|32 lanes per block, +100 = the output-staged
 * variant; 1 = the lane-per-block decoder), "decode_lanes_auto" (the decoder is
 * picked per batch from the compression ratio: the default), "encode_ctas_per_sm" (encoder warps = blocks in
 * flight per SM, 0 = as many as shared memory allows: 14), "encode_variant" (1 = always exact same-hash votes, 2 = resolved
 * through the table: default),
 * "encode_prefetch" (bytes of input kept prefetched ahead of the parse; 0 off, < 0 L2 only), "encode_lane_copy_max" /
 * "encode_probe_max" / "encode_wide_min" (path-selection heuristics of the fast encoder, lz4_encode.cuh EncTune: they
 * never change the emitted bytes), "hc_kernel" (which LZ4HC kernel encodes a batch: -1 = chosen per batch, the default -- at most
 * three blocks per SM: kernel 1, larger batches: kernel 2, batches made mostly of blocks above 64 KiB: kernel 0; 0 = one
 * thread per block, any block size; 1 / 2 = one warp per block on a static index of the block's hash buckets, blocks of at
 * most 64 KiB -- 1 stages the block in shared memory, 2 reads it through L1 -- larger blocks and the rare block whose chains
 * depend on the parse go to kernel 0 inside the same call), "hc_warps_per_sm" (kernels 1 / 2: blocks in flight per SM,
 * 0 = the default: 3 / 32),
 * "hc_concurrency" (kernel 0: blocks in flight), "host_chunk_mb" (bytes per pipeline stage of host-memory batches).
 * Returns LZ4B200_OK or LZ4B200_E_ARG. */
int lz4b200_set_option(lz4b200_ctx* ctx, const char* key, int64_t value);
/* The current value of an integer option ("hc_kernel", "hc_warps_per_sm", "hc_concurrency", "decode_lanes",
 * "encode_variant", "encode_ctas_per_sm").  Returns LZ4B200_OK or LZ4B200_E_ARG. */
int lz4b200_get_option(lz4b200_ctx* ctx, const char* key, int64_t* value);

/* Kernel launches issued through this context since creation (bench.py reports it as gpu_launches). */
int64_t lz4b200_launch_count(lz4b200_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* LZ4B200_H */
