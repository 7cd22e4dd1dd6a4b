/*
 * dlz4_b200.h -- C ABI of the B200-native LZ4 block codec (libdlz4_b200.so).
 *
 * Drop-in boundary for the raw block layer and the batched block path of divortio-lz4.
 * Every entry point names the reference interface it replaces (paths relative to the
 * reference repository).  Plain pointers and sizes only; no torch / CUDA types in signatures
 * (a CUDA stream is passed as an opaque void* holding a cudaStream_t; NULL = the context's own stream, so pass
 * cudaStreamLegacy (0x1) to mean the legacy default stream).
 *
 * There is no CPU fallback: every call runs CUDA kernels on the context's device and returns
 * DLZ4_E_CUDA (with dlz4_last_error() text) when the device or driver is not usable.
 *
 * Status codes: 0 = ok; 1..4 are decompressBlock's four errors, 5..7 decompressBuffer's three
 * (dlz4_strerror returns the reference's exact exception strings for them); >= 8 are additions.
 */
#ifndef DLZ4_B200_H
#define DLZ4_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DLZ4_OK                  0
#define DLZ4_E_OUTPUT_TOO_SMALL  1   /* "LZ4: Output Buffer Too Small"          src/block/blockDecompress.js:74  */
#define DLZ4_E_MALFORMED         2   /* "LZ4: Malformed Input"                  src/block/blockDecompress.js:75  */
#define DLZ4_E_OFFSET_ZERO       3   /* "LZ4: Invalid Offset 0"                 src/block/blockDecompress.js:128 */
#define DLZ4_E_DICT_OOB          4   /* "LZ4: Dictionary Offset Out of Bounds"  src/block/blockDecompress.js:151 */
#define DLZ4_E_BAD_MAGIC         5   /* "LZ4: Invalid Magic Number"             src/buffer/bufferDecompress.js:60  */
#define DLZ4_E_BAD_VERSION       6   /* "LZ4: Unsupported Version N"            src/buffer/bufferDecompress.js:67  */
#define DLZ4_E_CONTENT_CHECKSUM  7   /* "LZ4: Content Checksum Error"           src/buffer/bufferDecompress.js:216 */
#define DLZ4_E_BLOCK_CHECKSUM    8   /* extension: block checksum mismatch (only when verify_block_checksums) */
#define DLZ4_E_HEADER_CHECKSUM   9   /* extension: header checksum mismatch (only when strict)                */
#define DLZ4_E_INVALID_ARG      20
#define DLZ4_E_TOO_LARGE        21   /* input >= 2 GiB in one call: the reference takes len|0 (bufferCompress.js:127) */
#define DLZ4_E_CUDA             30   /* CUDA runtime/driver failure; see dlz4_last_error() */

#define DLZ4_HASH_ENTRIES    16384   /* Int32Array(16384): src/buffer/bufferCompress.js:21,55 */

/* Initial hash-table state for compress_blocks (SURVEY 8d config 4 "table modes"). */
#define DLZ4_WARM_NONE     0   /* fresh zero table per block (compressBuffer independent blocks, bufferCompress.js:234-236) */
#define DLZ4_WARM_JENKINS  1   /* table warmed from the prefix as compressBuffer does (bufferCompress.js:186-204) */
#define DLZ4_WARM_TABLE    2   /* caller-supplied int32[16384] copied per block (blockCompress.js:27 hashTable) */

/* History mode for decompress_blocks. */
#define DLZ4_HIST_RAW      0   /* every block has its own output base; history = dictionary only
                                  (decompressBlock(msg,0,len,out_i,0,dict), blockDecompress.js:142-147) */
#define DLZ4_HIST_FRAME    1   /* all blocks write one output buffer; block history = dictionary ++ dst[0..dst_off[i])
                                  (bufferDecompress.js:153), the caller's bytes of dst included: the host-pointer variant
                                  uploads all of dst in this mode */

typedef struct dlz4_ctx dlz4_ctx;

/* ---- lifecycle -------------------------------------------------------------------------- */
/* Creates a context bound to CUDA device `device` (one per process/GPU; one stream, reusable scratch). */
int dlz4_init(int device, dlz4_ctx **ctx);
void dlz4_shutdown(dlz4_ctx *ctx);
/* Reference exception text for a status code ("LZ4: Malformed Input", ...). */
const char *dlz4_strerror(int status);
/* Text of the last CUDA failure seen by this context ("" if none). */
const char *dlz4_last_error(const dlz4_ctx *ctx);
/* Number of kernels this context has launched so far (bench.py "gpu_launches"). */
uint64_t dlz4_launch_count(const dlz4_ctx *ctx);
/* Device time in ms of the most recent host-pointer call's kernel section (CUDA events). */
float dlz4_last_kernel_ms(const dlz4_ctx *ctx);
/* Measurement aid (bench.py "roofline"): with enable != 0 the next batches of fresh blocks <= 64 KiB record CUDA events
 * around the match finder (k_parse_pw) and the encoder (k_encode_blocks) on the stream they run on.  finder_ms /
 * encoder_ms (nullable) receive the durations of the most recent probed batch (the call waits for it). */
int dlz4_kernel_probe(dlz4_ctx *ctx, int enable, float *finder_ms, float *encoder_ms);
/* Segment-parallel compression (linked-block chains, bufferCompress.js:182,219,234, and independent blocks > 64 KiB): how
 * many segments the most recent frame call used, how many of them had to be re-run because the speculative start state
 * differed from the serial parse's, and in how many rounds.  The output bytes are those of the serial loop either way. */
void dlz4_segment_stats(const dlz4_ctx *ctx, uint32_t *segments, uint32_t *reruns, uint32_t *rounds);

/* Page-locked host memory, so host-pointer calls copy at the full PCIe rate (an N-API addon backs its external
 * ArrayBuffers with it).  Any host pointer is accepted everywhere; pageable ones are simply slower. */
void *dlz4_pinned_alloc(uint64_t bytes);
void dlz4_pinned_free(void *p);
/* Page-locks / releases memory the caller already owns (a Node Buffer's backing store, a mapping shared by the ranks of a
 * box): the way ordinary caller-owned Uint8Arrays (bufferCompress.js:100) reach the pinned PCIe rate without a bounce copy. */
int dlz4_host_register(void *p, uint64_t bytes);
int dlz4_host_unregister(void *p);

/* Worst-case compressed size of one n-byte block: n + n/255 + 16. */
uint64_t dlz4_compress_bound(uint64_t n);
/* Worst-case frame size for n input bytes. */
uint64_t dlz4_frame_bound(uint64_t n);
/* Contiguous block range [first, first+count) owned by `rank` of `world` (SURVEY 8e: block i -> GPU floor(i*G/n)). */
void dlz4_shard_range(uint64_t nblocks, uint32_t world, uint32_t rank, uint64_t *first, uint64_t *count);

/* ---- batched raw blocks: replaces the per-block calls compressBlock() / decompressBlock() ----
 * compressBlock(src, output, srcStart, srcLen, hashTable, outputOffset)   src/block/blockCompress.js:31
 *   block i = src[src_off[i] .. +src_len[i]); its output goes to dst[dst_off[i] ..) (give it
 *   dlz4_compress_bound(src_len[i]) bytes) and its length to comp_len[i].
 *   prefix/prefix_len: optional bytes that logically precede EVERY block (the caller-side
 *   "dict ++ msg" working buffer, srcStart = prefix_len); warm selects the initial table.
 *   Bytes are identical to the reference for the same (prefix, table, block).
 * Pointers of the _dev variants are device pointers (off/len arrays too).
 *   Host variant only: dst_off == NULL selects PACKED output -- block i is written directly behind block i-1 (its offset
 *   is the running sum of comp_len[]); blocks must then be ascending and disjoint in src, and the call runs as a chunked
 *   pipeline (H2D of chunk c+1, kernels of chunk c, D2H of chunk c-1 overlap), moving only real bytes over PCIe; prefix,
 *   warm and init_table apply as in the strided form (uploaded once, before the first chunk).
 *   dlz4_decompress_blocks accepts that layout with src_off == NULL.
 *   max_block_len: an upper bound of src_len[] known to the caller (0xFFFFFFFF if unknown); blocks of at most
 *   64 KiB with no prefix and DLZ4_WARM_NONE take the match finder + encoder pair (k_parse_pw, k_encode_blocks); batches of
 *   uniform blocks > 64 KiB are cut into segments (the call then reads the descriptors back and synchronises the stream).
 *   The match finder's record scratch is (max_block_len / 4 + 2) x 8 bytes per block, kept by the context and capped at
 *   2.25 GiB per launch: a larger batch (more than 16 384 blocks of 64 KiB, or many small blocks behind one 64 KiB block)
 *   runs as several launches on `stream`.  Growing the scratch synchronises the device.
 */
int dlz4_compress_blocks_dev(dlz4_ctx *ctx, const uint8_t *src, const uint64_t *src_off, const uint32_t *src_len,
                             uint32_t nblocks, uint32_t max_block_len, const uint8_t *prefix, uint32_t prefix_len, int warm,
                             const int32_t *init_table, uint8_t *dst, const uint64_t *dst_off,
                             uint32_t *comp_len, void *stream);
int dlz4_compress_blocks(dlz4_ctx *ctx, const uint8_t *src, uint64_t src_bytes, const uint64_t *src_off,
                         const uint32_t *src_len, uint32_t nblocks, const uint8_t *prefix, uint32_t prefix_len,
                         int warm, const int32_t *init_table, uint8_t *dst, uint64_t dst_bytes,
                         const uint64_t *dst_off, uint32_t *comp_len);

/* decompressBlock(input, inputOffset, inputSize, output, outputOffset, dictionary)   src/block/blockDecompress.js:30
 *   block i = src[src_off[i] .. +src_len[i]) decodes to dst[dst_off[i] ..) with capacity dst_cap[i];
 *   out_len[i] = bytes written, status[i] = 0 or DLZ4_E_* (1..4).  Returns the first non-zero status (host
 *   variant) or DLZ4_OK/CUDA error (_dev variant: read status[] yourself).
 *   Batches of fewer than 1024 blocks without dictionary are inspected (descriptors read back, the stream synchronised): uniform
 *   blocks > 64 KiB tiling one output range go to the jump decoder (parallel inside every block); everything else is one
 *   warp per block, asynchronous on `stream`.
 */
int dlz4_decompress_blocks_dev(dlz4_ctx *ctx, const uint8_t *src, const uint64_t *src_off, const uint32_t *src_len,
                               uint32_t nblocks, uint8_t *dst, const uint64_t *dst_off, const uint32_t *dst_cap,
                               const uint8_t *dict, uint32_t dict_len, int hist_mode,
                               uint32_t *out_len, uint8_t *status, void *stream);
int dlz4_decompress_blocks(dlz4_ctx *ctx, const uint8_t *src, uint64_t src_bytes, const uint64_t *src_off,
                           const uint32_t *src_len, uint32_t nblocks, uint8_t *dst, uint64_t dst_bytes,
                           const uint64_t *dst_off, const uint32_t *dst_cap, const uint8_t *dict, uint32_t dict_len,
                           int hist_mode, uint32_t *out_len, uint8_t *status);

/* ---- single raw block: LZ4.compressRaw / LZ4.decompressRaw (src/lz4.js:32-33) ----------------
 * Same argument meaning as the JS functions; `table` (int32[16384], value = position+1, <=0 empty)
 * is read and written back so linked use across calls behaves as in the reference.
 */
int dlz4_compress_block(dlz4_ctx *ctx, const uint8_t *src, uint64_t src_total, int32_t src_start, int32_t src_len,
                        int32_t *table, uint8_t *output, uint64_t output_total, int32_t output_offset,
                        int32_t *written);
int dlz4_decompress_block(dlz4_ctx *ctx, const uint8_t *input, uint64_t input_total, int64_t input_offset,
                          int64_t input_size, uint8_t *output, uint64_t output_total, int64_t output_offset,
                          const uint8_t *dictionary, uint64_t dict_len, int64_t *written);

/* ---- xxHash32: xxHash32(input, seed)   src/xxhash32/xxhash32.js:21 -----------------------------
 * batch: out[i] = xxh32(base[off[i] .. +len[i]), seed), one independent hash per item (per-block checksums).
 * stream: one hash over a whole buffer (contentChecksum; serial 4-lane chain, single warp).
 */
int dlz4_xxh32_batch_dev(dlz4_ctx *ctx, const uint8_t *base, const uint64_t *off, const uint32_t *len, uint32_t n,
                         uint32_t seed, uint32_t *out, void *stream);
int dlz4_xxh32_stream_dev(dlz4_ctx *ctx, const uint8_t *data, uint64_t len, uint32_t seed, uint32_t *out, void *stream);
int dlz4_xxh32(dlz4_ctx *ctx, const uint8_t *data, uint64_t len, uint32_t seed, uint32_t *out);
/* The same hash started asynchronously in one of 32 slots, each a serial chain on its own stream (xxhash32.js:34-57 is one
 * chain per stream; the content checksums of DIFFERENT frames, bufferCompress.js:248-252, are independent).  data: a device
 * pointer or PAGE-LOCKED host memory (dlz4_pinned_alloc / dlz4_host_register), which the kernel reads in place over PCIe;
 * pageable memory is refused with DLZ4_E_INVALID_ARG.  dlz4_xxh32_wait blocks until the slot's hash is there. */
int dlz4_xxh32_async(dlz4_ctx *ctx, int slot, const uint8_t *data, uint64_t len, uint32_t seed);
int dlz4_xxh32_wait(dlz4_ctx *ctx, int slot, uint32_t *out);
int dlz4_xxh32_batch(dlz4_ctx *ctx, const uint8_t *base, uint64_t base_bytes, const uint64_t *off,
                     const uint32_t *len, uint32_t n, uint32_t seed, uint32_t *out);

/* ---- frame API: the block loops of compressBuffer / decompressBuffer as one batched GPU pass ----
 * compressBuffer(input, dictionary, maxBlockSize, blockIndependence, contentChecksum, addContentSize, outputBuffer)
 *   src/buffer/bufferCompress.js:100 (block loop :209-239).  block_checksum is an addition (LZ4 frame spec;
 *   the reference writer has no such option): with 0 the frame is byte-identical to the reference's.
 */
typedef struct dlz4_frame_opts {
    uint32_t max_block_size;      /* quantised as getBlockId does: <=64K,<=256K,<=1M, else 4M (bufferCompress.js:77-82) */
    int32_t  block_independence;  /* default 0 in the reference (linked blocks = serial chain kernel) */
    int32_t  content_checksum;
    int32_t  add_content_size;    /* default 1 in the reference */
    int32_t  block_checksum;      /* addition */
} dlz4_frame_opts;

int dlz4_frame_compress(dlz4_ctx *ctx, const uint8_t *input, uint64_t input_len, const uint8_t *dictionary,
                        uint64_t dict_len, const dlz4_frame_opts *opts, uint8_t *output, uint64_t output_cap,
                        uint64_t *output_len);

/* decompressBuffer(input, dictionary, verifyChecksum)   src/buffer/bufferDecompress.js:51 (block loop :133-192).
 *   dlz4_frame_info parses the header and walks the block table on the host so the caller can size `output`
 *   (content size if present, else nblocks * blockMaxSize as an upper bound).
 *   flags: bit0 verify content checksum (the reference's verifyChecksum), bit1 verify block checksums (addition),
 *          bit2 verify header checksum (addition).
 */
typedef struct dlz4_frame_info_t {
    uint64_t content_size;        /* 0 when absent */
    uint64_t max_decoded;         /* upper bound for the decoded length */
    uint32_t nblocks;
    uint32_t block_max_size;
    uint8_t  flg, bd, has_content_size, has_content_checksum, has_block_checksum, has_dict_id, block_independence, pad;
    uint32_t dict_id;
    int32_t  version;
    uint64_t frame_bytes;         /* bytes of this frame: header .. EndMark [content checksum] */
} dlz4_frame_info_t;
int dlz4_frame_info(const uint8_t *frame, uint64_t frame_len, dlz4_frame_info_t *info);
int dlz4_frame_decompress(dlz4_ctx *ctx, const uint8_t *frame, uint64_t frame_len, const uint8_t *dictionary,
                          uint64_t dict_len, uint32_t flags, uint8_t *output, uint64_t output_cap,
                          uint64_t *output_len);

/* ---- single frames in device memory: dlz4_frame_compress / dlz4_frame_info / dlz4_frame_decompress on CUDA buffers ----
 * src, dictionary, frame and dst are device pointers of any alignment; every other pointer is host memory.  A call stages
 * what it reads in the context's scratch with one device-to-device copy, then runs the host call's code paths (the
 * segment-parallel compressor, the jump decoder, ...) and produces the same bytes and statuses.  Work is queued on `stream`
 * (NULL = the context's stream), and the call has synchronised `stream` when it returns, because its results are host values:
 *   compress:   twice -- once for the compressed body's length (it places the EndMark and sizes *frame_len), once at the end.
 *   info:       once -- for the header bytes and the block walk's count, bound and end.
 *   decompress: three times (twice for a frame without blocks, or on an error found before decoding) plus the decode
 *               route's own one or two -- for the header and the block count, for the block table
 *               (it sizes the jump decoder's scratch and selects the decode route), and for the final status.
 * Not covered: block ranges (use the host calls) and the stream classes.  Concatenated and skippable frames: the
 * dlz4_frames_*_dev calls below. */
/* dlz4_frame_compress on device memory.  dst_cap must be at least dlz4_frame_bound(src_len) (else DLZ4_E_OUTPUT_TOO_SMALL;
 * no silent truncation here).  *frame_len (host) = the frame's length.  The independent 64 KiB-block frames that the host call
 * sends through its chunked PCIe pipeline take the ordinary block compressor here; the bytes are the same. */
int dlz4_frame_compress_dev(dlz4_ctx *ctx, const uint8_t *src, uint64_t src_len, const uint8_t *dictionary, uint64_t dict_len,
                            const dlz4_frame_opts *opts /* host */, uint8_t *dst, uint64_t dst_cap, uint64_t *frame_len,
                            void *stream);
/* dlz4_frame_info on a frame in device memory: same fields, same status for every input. */
int dlz4_frame_info_dev(dlz4_ctx *ctx, const uint8_t *frame, uint64_t frame_len, dlz4_frame_info_t *info /* host */,
                        void *stream);
/* dlz4_frame_decompress on device memory: same flags.  Return value and *output_len (host) are what dlz4_frame_decompress
 * returns for the same bytes, dictionary, flags and output_cap.  dst bytes beyond *output_len, and all of dst on error, are
 * unspecified.  Checksums are computed and compared on the device. */
int dlz4_frame_decompress_dev(dlz4_ctx *ctx, const uint8_t *frame, uint64_t frame_len, const uint8_t *dictionary,
                              uint64_t dict_len, uint32_t flags, uint8_t *dst, uint64_t output_cap, uint64_t *output_len,
                              void *stream);

/* ---- batched frames: LZ4.compress / LZ4.decompress once per message, for many messages in one GPU pass ----
 * Every frame of a batch shares one option set (opts on compress, flags on decompress) and one optional dictionary; frame i
 * comes out exactly as the single-frame call makes it, byte for byte and status for status.  Per-frame work is one thread or
 * one warp per frame; inside a frame the block table stays a short serial loop.  This is the path for many small frames: one
 * warp per frame decodes a batch of a few large frames more slowly than dlz4_frame_decompress's jump decoder, and a linked
 * frame of several blocks compresses on one warp instead of the segment engine (the crossover is measured by
 * tools/frame_batch_bench.py and recorded in DESIGN.md).
 * _dev variants take device pointers, queue their work on `stream` and synchronise it once, to read the block count back.
 * Host variants stage through the context's scratch (pageable memory works) and return when the results are in place.
 * A frame of 0x7FFF0000 bytes or more makes the call return DLZ4_E_TOO_LARGE, as dlz4_frame_compress does.
 *
 * Compress: frame i = dlz4_frame_compress(src[src_off[i] .. +src_len[i]), dictionary, opts), frames packed back to back:
 *   frame i is dst[frame_off[i] .. frame_off[i+1]) (frame_off has nframes + 1 entries).  dst_cap must be at least the sum of
 *   dlz4_frame_bound(src_len[i]) (else DLZ4_E_OUTPUT_TOO_SMALL).  max_len: an upper bound of src_len[] (_dev only).
 *   Host variant: src holds src_bytes bytes, dst dst_cap bytes. */
int dlz4_frames_compress_batch_dev(dlz4_ctx *ctx, const uint8_t *src, const uint64_t *src_off, const uint32_t *src_len,
                                   uint32_t nframes, uint32_t max_len, const uint8_t *dictionary, uint32_t dict_len,
                                   const dlz4_frame_opts *opts /* host */, uint8_t *dst, uint64_t dst_cap, uint64_t *frame_off,
                                   void *stream);
int dlz4_frames_compress_batch(dlz4_ctx *ctx, const uint8_t *src, uint64_t src_bytes, const uint64_t *src_off,
                               const uint32_t *src_len, uint32_t nframes, const uint8_t *dictionary, uint32_t dict_len,
                               const dlz4_frame_opts *opts, uint8_t *dst, uint64_t dst_cap, uint64_t *frame_off);
/* Sizing pass: max_decoded[i] = dlz4_frame_info(frame i).max_decoded, status[i] = its status (0, 2, 5 or 6; max_decoded[i] = 0
 * on error).  Frame i is src[frame_off[i] .. +frame_len[i]). */
int dlz4_frames_batch_info_dev(dlz4_ctx *ctx, const uint8_t *src, const uint64_t *frame_off, const uint64_t *frame_len,
                               uint32_t nframes, uint64_t *max_decoded, uint8_t *status, void *stream);
int dlz4_frames_batch_info(dlz4_ctx *ctx, const uint8_t *src, uint64_t src_bytes, const uint64_t *frame_off,
                           const uint64_t *frame_len, uint32_t nframes, uint64_t *max_decoded, uint8_t *status);
/* Decompress: the first frame in src[frame_off[i] .. +frame_len[i]) (bytes after it are ignored, as in the single-frame call)
 *   decodes to dst[dst_off[i] .. +dst_cap[i]); status[i] / out_len[i] are what dlz4_frame_decompress(frame i, dictionary, flags,
 *   output_cap = dst_cap[i]) returns (out_len[i] = 0 on error).  Bytes of dst[dst_off[i] + out_len[i] .. +dst_cap[i]) are
 *   unspecified afterwards.  The host variant returns the first non-zero status, like dlz4_decompress_blocks. */
int dlz4_frames_decompress_batch_dev(dlz4_ctx *ctx, const uint8_t *src, const uint64_t *frame_off, const uint64_t *frame_len,
                                     uint32_t nframes, const uint8_t *dictionary, uint32_t dict_len, uint32_t flags,
                                     uint8_t *dst, const uint64_t *dst_off, const uint64_t *dst_cap, uint64_t *out_len,
                                     uint8_t *status, void *stream);
int dlz4_frames_decompress_batch(dlz4_ctx *ctx, const uint8_t *src, uint64_t src_bytes, const uint64_t *frame_off,
                                 const uint64_t *frame_len, uint32_t nframes, const uint8_t *dictionary, uint32_t dict_len,
                                 uint32_t flags, uint8_t *dst, uint64_t dst_bytes, const uint64_t *dst_off,
                                 const uint64_t *dst_cap, uint64_t *out_len, uint8_t *status);

/* SURVEY 8 f3: a buffer of several concatenated frames (what `cat a.lz4 b.lz4` or the lz4 CLI with several inputs produces) with
 * skippable frames (magic 0x184D2A50..5F, u32 size, payload) between them.  bufferDecompress.js:51-220 stops at the first
 * EndMark; the reference's stream decoder loops over frames (src/shared/lz4Decode.js:262-266).  Decodes every LZ4 frame in
 * order into `output` (same flags as dlz4_frame_decompress), skips skippable frames, and reports how many frames it decoded.
 * Trailing bytes that are not a frame are DLZ4_E_BAD_MAGIC.
 */
int dlz4_frames_decompress(dlz4_ctx *ctx, const uint8_t *data, uint64_t data_len, const uint8_t *dictionary, uint64_t dict_len,
                           uint32_t flags, uint8_t *output, uint64_t output_cap, uint64_t *output_len, uint32_t *frames);
/* Sum of the decoded-size bounds of all LZ4 frames in `data` (to size `output`), and their count. */
int dlz4_frames_info(const uint8_t *data, uint64_t data_len, uint64_t *max_decoded, uint32_t *frames);

/* ---- concatenated frames in device memory: inputs of any size, and the frame loop above, on CUDA buffers ----
 * Pointer conventions of dlz4_frame_*_dev: src, dictionary, data and dst are device pointers of any alignment and without
 * slack after their end; every other pointer is host memory; work is queued on `stream` (NULL = the context's stream).
 *
 * Compress: frame k = dlz4_frame_compress(src[k*frame_bytes .. min((k+1)*frame_bytes, src_len)), dictionary, opts), frames back
 *   to back in dst (src_len == 0 gives one empty frame).  1 <= frame_bytes < 0x7FFF0000 (else DLZ4_E_INVALID_ARG /
 *   DLZ4_E_TOO_LARGE).  dst_cap must be at least the sum of dlz4_frame_bound over the spans (else DLZ4_E_OUTPUT_TOO_SMALL, before
 *   any work).  frame_off (nullable) receives nframes + 1 entries: frame k is dst[frame_off[k] .. frame_off[k+1]).  The content
 *   checksums of all frames run side by side, one serial chain each, beside the block work.  `stream` is synchronised once per
 *   frame (its body length places the next frame) and once at the end.
 * Info: dlz4_frames_info on device memory -- the same *max_decoded, *frames and status for every input.  One synchronisation.
 * Decompress: dlz4_frames_decompress on device memory -- the same return value, *output_len and *frames as the host call for
 *   the same bytes, dictionary, flags and output_cap.  dst beyond *output_len, and all of dst on error, are unspecified.
 *   Frames whose max_decoded is below a size threshold decode in groups, one warp per frame; larger ones one at a time
 *   through dlz4_frame_decompress_dev's decoders.  `stream` is synchronised for the frame walk (twice when the sequence has
 *   more than 4096 frames), for the parse, once per group of small frames, for each large frame's block table and decode
 *   route, and once at the end for the statuses. */
int dlz4_frames_compress_dev(dlz4_ctx *ctx, const uint8_t *src, uint64_t src_len, uint64_t frame_bytes, const uint8_t *dictionary,
                             uint64_t dict_len, const dlz4_frame_opts *opts /* host */, uint8_t *dst, uint64_t dst_cap,
                             uint64_t *frame_off, uint64_t *out_len, uint32_t *nframes, void *stream);
int dlz4_frames_info_dev(dlz4_ctx *ctx, const uint8_t *data, uint64_t data_len, uint64_t *max_decoded, uint32_t *frames,
                         void *stream);
int dlz4_frames_decompress_dev(dlz4_ctx *ctx, const uint8_t *data, uint64_t data_len, const uint8_t *dictionary,
                               uint64_t dict_len, uint32_t flags, uint8_t *dst, uint64_t output_cap, uint64_t *output_len,
                               uint32_t *frames, void *stream);

/* SURVEY 8 f1 (streaming codec, src/shared/lz4Encode.js / lz4Decode.js) -- the two pieces the stream classes need below them.
 *
 * Stateful xxh32 (the reference's XXHash32 class, update()/digest()): the stripe loop runs on the GPU with the four
 * accumulators carried in `v`; the host keeps the < 16-byte tail and finishes the digest (merge + tail + avalanche).
 */
typedef struct dlz4_xxh32_state {
    uint32_t v[4];
    uint64_t total;
    uint8_t  mem[16];
    uint32_t memsize;
    uint32_t seed;
} dlz4_xxh32_state;
void dlz4_xxh32_reset(dlz4_xxh32_state *s, uint32_t seed);
int dlz4_xxh32_update(dlz4_ctx *ctx, dlz4_xxh32_state *s, const uint8_t *data, uint64_t len);
uint32_t dlz4_xxh32_digest(const dlz4_xxh32_state *s);
/* LZ4Encoder._flushBlock for every full block of an add() at once (lz4Encode.js:215-298, linked mode): blocks of
 * block_size tile work[start, start + total), history is work[0, start), `table` (int32[16384], position + 1 in `work`) is
 * the carried state, read and written.  Block k's bytes go to dst + k * dst_stride, its size to comp_len[k].  Long runs take
 * the segment-parallel engine; the table returned is the serial loop's. */
int dlz4_chain_compress(dlz4_ctx *ctx, const uint8_t *work, uint64_t work_len, int32_t start, int32_t total, int32_t block_size,
                        int32_t *table, uint8_t *dst, uint64_t dst_stride, uint32_t *comp_len);
/* The same flush with the output already in frame-body form and the working buffer given as TWO host pieces that are joined
 * on the device (head = 64 KiB window ++ pending bytes, tail = the caller's new chunk: no host-side concatenation).  Blocks of
 * block_size tile [start, start + total) of head ++ tail.  linked != 0: one chain carrying `table` (in/out); linked == 0: fresh
 * independent blocks (lz4Encode.js:240-242; table unused).  body <- [u32 size | stored bit][payload] per block with the
 * stored-block rule of lz4Encode.js:263-273; piece_len[k] = length of block k's piece (4 + payload). */
int dlz4_stream_blocks(dlz4_ctx *ctx, const uint8_t *head, uint64_t head_len, const uint8_t *tail, uint64_t tail_len, int32_t start,
                       int32_t total, int32_t block_size, int linked, int32_t *table, uint8_t *body, uint64_t body_cap,
                       uint64_t *body_len, uint32_t *piece_len);

/* dlz4_frame_decompress that also reports every block's decoded length (block_out_len[nblocks], nullable): the stream
 * decoder hands out one chunk per block like LZ4Decoder.update (lz4Decode.js:206-245). */
int dlz4_frame_decompress_ex(dlz4_ctx *ctx, const uint8_t *frame, uint64_t frame_len, const uint8_t *dictionary,
                             uint64_t dict_len, uint32_t flags, uint8_t *output, uint64_t output_cap, uint64_t *output_len,
                             uint32_t *block_out_len);

/* Device-resident frame assembly used by the sharded path (SURVEY 8e): given the per-block compressed
 * lengths and the worst-case-strided scratch produced by dlz4_compress_blocks_dev, writes
 * [u32 size|stored][data][u32 xxh32]* for blocks [0,nblocks) into d_segment and its length to *d_segment_len.
 */
int dlz4_frame_pack_dev(dlz4_ctx *ctx, const uint8_t *src, const uint64_t *src_off, const uint32_t *src_len,
                        const uint8_t *comp, const uint64_t *comp_off, const uint32_t *comp_len, uint32_t nblocks,
                        int block_checksum, uint8_t *segment, uint64_t *block_pos /* nblocks+1 */, void *stream);

/* ---- sharded frames (SURVEY 8e: block i -> GPU floor(i*G/n); one process and one context per GPU) ----------------------
 * The block loop of compressBuffer (bufferCompress.js:209-239) over one rank's contiguous range of INDEPENDENT blocks.
 * dlz4_frame_body_compress compresses `input` (the rank's slice, < 2 GiB, whole blocks except at the frame's end) and packs
 * [u32 size | stored bit][payload][u32 xxh32]* -- exactly the bytes dlz4_frame_compress writes for those blocks -- in
 * device memory; *body_len = its length.  The host then scans the ranks' lengths and every rank copies its body to its
 * place in the host frame with dlz4_frame_body_fetch (no collective touches the data).  Header and EndMark come from
 * dlz4_frame_header / four zero bytes.
 */
int dlz4_frame_body_compress(dlz4_ctx *ctx, const uint8_t *input, uint64_t input_len, uint32_t max_block_size,
                             int block_checksum, uint64_t *body_len);
int dlz4_frame_body_fetch(dlz4_ctx *ctx, uint8_t *dst, uint64_t dst_cap);
/* The frame header every path writes (bufferCompress.js:147-178): magic, FLG, BD, [content size u64], [dictID], HC.
 * Returns its length (7..19).  Host-only arithmetic (xxh32 of <= 14 bytes). */
size_t dlz4_frame_header(const dlz4_frame_opts *opts, uint64_t content_len, int have_dict, uint32_t dict_id, uint8_t out[19]);
/* The block loop of decompressBuffer (bufferDecompress.js:133-192) over blocks [first_block, first_block + block_count) of an
 * independent-block frame: decodes them into `output` (block first_block at output[0]); block_out_len (nullable) receives the
 * decoded length of each block of the range so that the caller can check that inner blocks are full before trusting the
 * i * blockMaxSize placement.  flags as dlz4_frame_decompress, except that the content checksum is never verified over a
 * part (use the relay below).  A linked-block frame is accepted only as a whole (first_block == 0, all blocks). */
int dlz4_frame_decompress_range(dlz4_ctx *ctx, const uint8_t *frame, uint64_t frame_len, uint32_t first_block,
                                uint32_t block_count, const uint8_t *dictionary, uint64_t dict_len, uint32_t flags,
                                uint8_t *output, uint64_t output_cap, uint64_t *output_len, uint32_t *block_out_len);
/* Whole-stream content checksum across ranks (xxhash32.js:34-57 is one serial chain: "replicas only", SURVEY 8e): a relay.
 * Rank r receives the 16-byte accumulator state from rank r-1, runs the stripe loop over the bytes its last
 * dlz4_frame_body_compress (which = DLZ4_RESIDENT_INPUT) or dlz4_frame_decompress[_range] (DLZ4_RESIDENT_OUTPUT) call left
 * on its GPU -- nothing is uploaded twice -- and passes the state on; the last rank calls dlz4_xxh32_digest.  Pieces before
 * the last must be multiples of 16 bytes (whole blocks are). */
#define DLZ4_RESIDENT_INPUT   0
#define DLZ4_RESIDENT_OUTPUT  1
int dlz4_xxh32_update_resident(dlz4_ctx *ctx, dlz4_xxh32_state *s, int which);

#ifdef __cplusplus
}
#endif
#endif /* DLZ4_B200_H */
