/*
 * include/b2c.h -- C ABI of libb200comp.so, the B200 (sm_100a) block-compression engine.
 *
 * This is the drop-in boundary for klauspost/compress's block codec hot path.  The reference
 * has no FFI of its own (pure Go + Go assembler, CGO_ENABLED=0); the entry points below are what a
 * cgo shim would bind in place of the per-block work of
 *     zstd.Encoder.EncodeAll / encodeAll        zstd/encoder.go:722,731   -> b2c_zstd_encode_*
 *     zstd.Decoder.DecodeAll / runDecoder       zstd/decoder.go:319, framedec.go:330 -> b2c_zstd_decode_*
 *     huff0.Compress4X / Compress1X             huff0/compress.go:27,14   -> b2c_huf_compress_device
 *     s2.Encode / s2.Writer custom encoder hook s2/encode.go:29, s2/writer.go:1052 -> b2c_s2_*
 * (see INTEGRATION.md for the cgo stubs).  Conventions follow the reference's Go<->asm seam
 * (zstd/seqdec_asm.go:17-78, s2/encodeblock_amd64.go:14-42): the caller owns all memory, nothing is
 * retained past return, sizes are plain integers, results are byte counts or negative error codes.
 *
 * Batched on purpose: one call = N independent chunks (a 64 KiB chunk per kernel launch would be
 * launch-bound); a chunk is what one EncodeAll call / one s2 block is in the reference.
 * No CPU fallback exists: every entry point fails with B2C_ERR_NO_DEVICE without a CUDA device.
 */
#ifndef B2C_H
#define B2C_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2C_API __attribute__((visibility("default")))

/* error codes (returned negative, also stored per chunk in sizes_out) */
enum {
    B2C_OK = 0,
    B2C_ERR_NO_DEVICE = -100,   /* no CUDA device / driver: the product never falls back to the CPU */
    B2C_ERR_CUDA = -101,        /* a CUDA runtime call failed (see b2c_last_cuda_error) */
    B2C_ERR_ARG = -102,
    B2C_ERR_TOO_BIG = -3,       /* chunk larger than the level's block size (zstd: 64 KiB at level 1) */
    B2C_ERR_DST_SMALL = -4,     /* destination slot smaller than the encoded chunk */
    B2C_ERR_CORRUPT = -5,       /* decoder: invalid stream (maps to the zstd package's decode errors) */
    B2C_ERR_MAGIC = -7,         /* zstd.ErrMagicMismatch */
    B2C_ERR_WINDOW = -8,        /* zstd.ErrWindowSizeExceeded / ErrWindowSizeTooSmall / ErrBlockTooBig-class */
    B2C_ERR_CRC = -9,           /* zstd.ErrCRCMismatch */
    B2C_ERR_SIZE = -10,         /* zstd.ErrFrameSizeExceeded / ErrFrameSizeMismatch / ErrDecoderSizeExceeded */
    B2C_ERR_UNSUPPORTED = -11
};

/* flags for the zstd encoder */
enum {
    B2C_ZSTD_CRC = 1,    /* append XXH64 content checksum (zstd.WithEncoderCRC, default true) */
    B2C_ZSTD_FRAME = 2   /* emit one complete frame per chunk (EncodeAll); otherwise bare blocks */
};

/* S2 block encoder: level and flags.  B2C_S2_FAST = s2.Encode's match finder class (s2/encode.go:29, encodeBlockGo),
 * B2C_S2_BETTER = s2.EncodeBetter's (s2/encode.go:117, encodeBlockBetterGo64K in s2/encode_better.go:485: long 7-byte +
 * short 4-byte table, long preferred, lazy step).  B2C_S2_SNAPPY selects Snappy-compatible output (s2.EncodeSnappy /
 * EncodeSnappyBetter, s2/encode.go:204,248: no repeat tags, copies <= 64). */
enum { B2C_S2_FAST = 1, B2C_S2_BETTER = 2 };
enum { B2C_S2_SNAPPY = 1 };

/* huff0: number of streams (huff0.Compress4X / Compress1X, huff0/compress.go:27,14) */
enum { B2C_HUF_1X = 0, B2C_HUF_4X = 1 };
/* huff0 results besides byte counts: the package's sentinel errors (huff0/huff0.go:30-42) */
enum { B2C_HUF_ERR_INCOMPRESSIBLE = -1, B2C_HUF_ERR_USE_RLE = -2 };   /* ErrTooBig = B2C_ERR_TOO_BIG */

/* zstd levels (zstd.EncoderLevel, zstd/encoder_options.go:163-190): SpeedFastest = 64 KiB blocks, one hash table
 * (zstd/enc_fast.go); SpeedDefault = 128 KiB blocks, long + short table with a lazy step (zstd/enc_dfast.go) */
enum { B2C_LEVEL_FASTEST = 1, B2C_LEVEL_DEFAULT = 2, B2C_LEVEL_BETTER = 3 };   /* 3: SpeedBetterCompression (zstd/enc_better.go), 128 KiB blocks */

typedef struct b2c_ctx b2c_ctx;

B2C_API int b2c_device_count(void);
/* One context per GPU per host thread.  max_chunks bounds the batch size of the host-buffer calls. */
B2C_API b2c_ctx *b2c_ctx_create(int device, size_t max_chunks);
B2C_API void b2c_ctx_destroy(b2c_ctx *ctx);
B2C_API const char *b2c_strerror(int code);
B2C_API const char *b2c_last_cuda_error(b2c_ctx *ctx);
B2C_API int b2c_sm_count(b2c_ctx *ctx);
/* number of kernel launches issued through this context so far (bench.py's gpu_launches) */
B2C_API uint64_t b2c_launch_count(b2c_ctx *ctx);

/* Per-kernel timing of the encode pipeline with CUDA events recorded on the launching stream (bench.py's
 * roofline).  b2c_profile_enable(ctx, 1) starts collecting; b2c_profile_read synchronises the device and returns in
 * ms[0..5] the summed durations of {xxh64, parse, histograms, tables, chains, pack} over the *ncalls encode launches
 * since (a device-resident call larger than the work pool is several launches).  The histograms are counted inside the
 * parse kernel, so ms[2] is an empty interval (about 0 ms), kept so that the slots keep their meaning. */
B2C_API int b2c_profile_enable(b2c_ctx *ctx, int on);
B2C_API int b2c_profile_read(b2c_ctx *ctx, double *ms, uint32_t *ncalls);
/* The same for zstd decode: ms[0..5] = {scan, literals, sequences, execute, xxh64, one-warp decoder} summed over the decode
 * launches since b2c_decode_profile_enable(ctx, 1); while enabled every decode launch synchronises its stream. */
B2C_API int b2c_decode_profile_enable(b2c_ctx *ctx, int on);
B2C_API int b2c_decode_profile_read(b2c_ctx *ctx, double *ms);
/* diagnostics: of the first nchunks inputs of the most recent decode launch, how many the staged kernels completed (the
 * rest were decoded by the one-warp decoder).  Synchronises the device. */
B2C_API int b2c_decode_staged_count(b2c_ctx *ctx, uint32_t nchunks, uint32_t *staged);
B2C_API int b2c_s2_decode_staged_count(b2c_ctx *ctx, uint32_t nchunks, uint32_t *staged);   /* the same for S2 block decode */

/* Encoder.MaxEncodedSize for one chunk of n bytes (zstd/encoder.go:843-873) */
B2C_API size_t b2c_zstd_bound(size_t n, int level);

/*
 * Device-resident batch (throughput path; bench `value`).  Chunk i is read from
 * d_src + i*src_stride (size d_sizes[i], or size_all when d_sizes == NULL) and written to
 * d_dst + i*dst_stride (capacity dst_stride); d_out_sizes[i] receives the encoded size or a
 * negative error.  All pointers are device pointers; `stream` is a cudaStream_t (NULL = default).
 * Asynchronous: returns after enqueueing.
 */
B2C_API int b2c_zstd_encode_device(b2c_ctx *ctx, int level, int flags, const void *d_src, size_t src_stride,
                                   const uint32_t *d_sizes, uint32_t size_all, void *d_dst, size_t dst_stride,
                                   int64_t *d_out_sizes, uint32_t nchunks, void *stream);

/*
 * Host-buffer batch (the call a cgo shim makes; bench `e2e`).  srcs[i]/dsts[i] are host pointers;
 * the library stages through pinned memory, copies H2D, encodes, packs and copies D2H.
 * sizes_out[i] = encoded bytes or negative error.  Synchronous.
 */
B2C_API int b2c_zstd_encode_chunks(b2c_ctx *ctx, int level, int flags, const void *const *srcs,
                                   const size_t *src_sizes, void *const *dsts, const size_t *dst_caps,
                                   int64_t *sizes_out, size_t n);

/*
 * Contiguous host input -> packed host output: src is cut into chunk_size pieces (<= 64 KiB at level 1), each
 * encoded as one frame, frames written back to back into h_dst (a valid zstd stream: concatenated frames,
 * zstd/encoder.go:719).  sizes_out[i] / offsets_out[i] describe frame i; *total_out is the stream length.
 * Double-buffered: H2D, kernels and D2H of consecutive batches overlap.  Synchronous.  h_src / h_dst may be pinned
 * (copied directly at PCIe rate) or ordinary pageable memory such as a Go slice (then the library stages them through
 * its own pinned buffers with several host threads; no cudaHostRegister by the caller is needed).
 */
B2C_API int b2c_zstd_encode_packed(b2c_ctx *ctx, int level, int flags, const void *h_src, size_t src_bytes,
                                   uint32_t chunk_size, void *h_dst, size_t dst_cap, int64_t *sizes_out,
                                   uint64_t *offsets_out, size_t *total_out);

/*
 * Frame mode: zstd.Encoder.EncodeAll for inputs of any size (zstd/encoder.go:722-840, the multi-block branch :796-830):
 * ONE frame per input -- frame header with the content size (frameHeader.appendTo, zstd/frameenc.go:25-92), the blocks,
 * the XXH64 of the whole content (B2C_ZSTD_CRC).  Blocks are 48 KiB at level 1 and 96 KiB at levels 2-3; the match
 * finder of every block also sees the 16 / 32 KiB before it (the reference's history, fastBase.addBlock,
 * zstd/enc_base.go:57-199), so match offsets reach back across blocks.  Blocks of a frame are encoded in parallel and
 * entropy-coded independently (no repeat-mode tables).
 * _device: frame f is h_src_sizes[f] bytes at d_src + h_src_offsets[f] (HOST arrays; 16-byte aligned offsets are
 * fastest); frames are written back to back into d_dst; d_dst_offsets[f] / d_out_sizes[f] (DEVICE arrays) receive
 * every frame's position and size (negative = error).  Asynchronous on `stream`.
 * b2c_zstd_encode_frames: host pointers in and out, one frame per (srcs[i], dsts[i]); synchronous.
 */
B2C_API size_t b2c_zstd_frame_bound(size_t n, int level);
B2C_API int b2c_zstd_encode_frames_device(b2c_ctx *ctx, int level, int flags, const void *d_src,
                                          const uint64_t *h_src_offsets, const uint64_t *h_src_sizes, uint32_t nframes,
                                          void *d_dst, uint64_t dst_cap, uint64_t *d_dst_offsets, int64_t *d_out_sizes,
                                          void *stream);
B2C_API int b2c_zstd_encode_frames(b2c_ctx *ctx, int level, int flags, const void *const *srcs, const size_t *src_sizes,
                                   void *const *dsts, const size_t *dst_caps, int64_t *sizes_out, size_t n);

/* Debug/parity hook used by tests: encode device-resident chunks and also dump, per chunk,
 * {nseq, nlit, kind, litMode}, the (litLen, matchLen-3, offset) triples and the literal bytes (rows of the level's
 * block size), so the entropy stage can be compared byte-for-byte with the oracle's blockEnc.encode. */
B2C_API int b2c_zstd_encode_device_debug(b2c_ctx *ctx, int level, int flags, const void *d_src, size_t src_stride,
                                         const uint32_t *d_sizes, uint32_t size_all, void *d_dst, size_t dst_stride,
                                         int64_t *d_out_sizes, uint32_t nchunks, uint32_t *d_dbg_hdr,
                                         uint32_t *d_dbg_seqs, uint8_t *d_dbg_lits, uint32_t dbg_seq_cap, void *stream);

/* Profiling hook: like b2c_zstd_encode_device (all chunks size_all bytes) but thread 0 of every CTA also
 * stores clock64() at 15 phase boundaries into d_cycles[chunk][16] (tools/phase_times.py). */
B2C_API int b2c_zstd_encode_device_timed(b2c_ctx *ctx, int flags, const void *d_src, size_t src_stride,
                                         uint32_t size_all, void *d_dst, size_t dst_stride, int64_t *d_out_sizes,
                                         uint32_t nchunks, unsigned long long *d_cycles, void *stream);

/*
 * zstd decode (zstd.Decoder.DecodeAll, zstd/decoder.go:319; per-block work of frameDec.runDecoder,
 * zstd/framedec.go:330).  Input i is a complete zstd stream (one or more frames, skippable frames allowed,
 * no dictionary) of d_src_sizes[i] bytes at d_src + (d_src_offsets ? d_src_offsets[i] : i*src_stride); its
 * content is written to d_dst + (d_dst_offsets ? d_dst_offsets[i] : i*dst_stride), at most dst_cap bytes.
 * d_out_sizes[i] = decoded bytes, or a negative error (B2C_ERR_CORRUPT, B2C_ERR_DST_SMALL, ...; checksum,
 * window and frame-size violations are reported as the reference reports them, see b2c_strerror).
 * One warp decodes one input: throughput comes from batching many inputs.  Asynchronous.
 */
B2C_API int b2c_zstd_decode_device(b2c_ctx *ctx, const void *d_src, size_t src_stride, const uint64_t *d_src_offsets,
                                   const uint32_t *d_src_sizes, void *d_dst, size_t dst_stride,
                                   const uint64_t *d_dst_offsets, uint32_t dst_cap, int64_t *d_out_sizes,
                                   uint32_t nchunks, void *stream);

/* Host-buffer batch decode (the call a cgo shim makes for a batch of DecodeAll calls).  Synchronous. */
B2C_API int b2c_zstd_decode_chunks(b2c_ctx *ctx, const void *const *srcs, const size_t *src_sizes, void *const *dsts,
                                   const size_t *dst_caps, int64_t *sizes_out, size_t n);

/*
 * S2 / Snappy blocks (s2.Encode / s2.EncodeSnappy / s2.Decode, s2/encode.go:29,204, s2/decode.go:58; per-block work
 * of s2.Writer with WriterBlockSize(64 KiB), the seam WriterCustomEncoder exposes, s2/writer.go:1052).
 * Block i (<= 64 KiB of input) becomes uvarint(len) + tag stream, or uvarint + one literal when it does not shrink.
 * Argument conventions are those of the zstd calls above.  Decode accepts any S2 or Snappy block whose decoded
 * length fits dst_cap (repeat tags, 4-byte offsets and long literals included); results are decoded bytes or
 * B2C_ERR_CORRUPT (s2.ErrCorrupt) / B2C_ERR_DST_SMALL.
 */
B2C_API size_t b2c_s2_bound(size_t n);   /* s2.MaxEncodedLen, s2/encode.go:389; 0 = too large */
B2C_API int b2c_s2_encode_device(b2c_ctx *ctx, int level, int flags, const void *d_src, size_t src_stride,
                                 const uint32_t *d_sizes, uint32_t size_all, void *d_dst, size_t dst_stride,
                                 int64_t *d_out_sizes, uint32_t nchunks, void *stream);
B2C_API int b2c_s2_decode_device(b2c_ctx *ctx, const void *d_src, size_t src_stride, const uint64_t *d_src_offsets,
                                 const uint32_t *d_src_sizes, void *d_dst, size_t dst_stride,
                                 const uint64_t *d_dst_offsets, uint32_t dst_cap, int64_t *d_out_sizes,
                                 uint32_t nchunks, void *stream);
B2C_API int b2c_s2_encode_chunks(b2c_ctx *ctx, int level, int flags, const void *const *srcs, const size_t *src_sizes,
                                 void *const *dsts, const size_t *dst_caps, int64_t *sizes_out, size_t n);
B2C_API int b2c_s2_decode_chunks(b2c_ctx *ctx, const void *const *srcs, const size_t *src_sizes, void *const *dsts,
                                 const size_t *dst_caps, int64_t *sizes_out, size_t n);

/*
 * S2 / Snappy STREAMS (the framing format: s2.Writer.EncodeBuffer, s2/writer.go:357-470, and s2.Reader over a buffer,
 * s2/reader.go:249-420; constants and the masked CRC32-C: s2/s2.go:75-126).  A stream = the identifier chunk, then per
 * block (<= 64 KiB here, WriterBlockSize) one chunk: type (0 compressed, 1 uncompressed), 24-bit length, checksum of the
 * uncompressed bytes, payload.  level / flags as for the block encoders (B2C_S2_SNAPPY writes a Snappy stream).
 * _encode_stream_device: device buffers, asynchronous; *d_total (device u64) = stream bytes, *d_err (device i32) = 0 or a
 * negative error.  _encode_stream / _decode_stream: host buffers, synchronous.  The reader accepts what s2.Reader accepts
 * (blocks up to 4 MiB, skippable and padding chunks, Snappy streams) and returns its errors: B2C_ERR_CORRUPT, B2C_ERR_CRC,
 * B2C_ERR_UNSUPPORTED (reserved unskippable chunk), B2C_ERR_DST_SMALL.
 */
B2C_API size_t b2c_s2_stream_bound(size_t n, size_t block);
B2C_API int b2c_s2_encode_stream_device(b2c_ctx *ctx, int level, int flags, const void *d_src, uint64_t n, uint32_t block,
                                        void *d_dst, uint64_t dst_cap, uint64_t *d_total, int32_t *d_err, void *stream);
B2C_API int b2c_s2_encode_stream(b2c_ctx *ctx, int level, int flags, const void *src, size_t n, uint32_t block, void *dst,
                                 size_t cap, size_t *out_len);
B2C_API int b2c_s2_decode_stream(b2c_ctx *ctx, const void *src, size_t n, void *dst, size_t cap, size_t *out_len);

/*
 * Standalone huff0 blocks (huff0.Compress4X / Compress1X with a fresh Scratch, huff0/compress.go:14-141;
 * huff0.ReadTable + Decoder.Decompress4X / Decompress1X, huff0/decompress.go:29,234,622).  Block i (<= 262143
 * bytes) -> table description + (jump table +) streams, byte-identical to the reference's output;
 * d_out_sizes[i] = bytes, or B2C_HUF_ERR_INCOMPRESSIBLE / B2C_HUF_ERR_USE_RLE / B2C_ERR_TOO_BIG /
 * B2C_ERR_DST_SMALL.  dst_stride (= slot capacity) and d_dst must be multiples of 4.
 * Decompress needs the exact decoded size of every block (the dstSize argument of Decompress4X).
 */
B2C_API int b2c_huf_compress_device(b2c_ctx *ctx, int flags, const void *d_src, size_t src_stride, const uint32_t *d_sizes,
                                    uint32_t size_all, void *d_dst, size_t dst_stride, int64_t *d_out_sizes,
                                    uint32_t nchunks, void *stream);
B2C_API int b2c_huf_decompress_device(b2c_ctx *ctx, int flags, const void *d_src, size_t src_stride,
                                      const uint32_t *d_src_sizes, void *d_dst, size_t dst_stride,
                                      const uint32_t *d_dst_sizes, int64_t *d_out_sizes, uint32_t nchunks, void *stream);

/* Host-buffer forms of the huff0 calls (the call a cgo shim makes): blocks[i] in ordinary host memory, results per
 * element as above.  b2c_huf_decompress_chunks takes the EXACT decoded size of every block in dst_sizes (the dstSize
 * argument of Decoder.Decompress4X, huff0/decompress_asm.go:27-31).  b2c_huf_read_table is huff0.ReadTable
 * (huff0/decompress.go:29-166): rows[i] receives 260 bytes -- [0] actualTableLog, [1] 0, [2..3] the size of the table
 * description in bytes (little endian; the streams start there), [4..259] the code length of every symbol (0 = absent) --
 * and sizes_out[i] the same size, or a negative error. */
B2C_API int b2c_huf_compress_chunks(b2c_ctx *ctx, int flags, const void *const *srcs, const size_t *src_sizes,
                                    void *const *dsts, const size_t *dst_caps, int64_t *sizes_out, size_t n);
B2C_API int b2c_huf_decompress_chunks(b2c_ctx *ctx, int flags, const void *const *srcs, const size_t *src_sizes,
                                      void *const *dsts, const size_t *dst_sizes, int64_t *sizes_out, size_t n);
B2C_API int b2c_huf_read_table(b2c_ctx *ctx, const void *const *srcs, const size_t *src_sizes, void *const *rows,
                               int64_t *sizes_out, size_t n);

/*
 * Coalescing queue: the shim's answer to the reference's one-block-per-call seams.  zstd.Encoder.EncodeAll may be
 * called concurrently (zstd/encoder.go:717-729), s2.WriterCustomEncoder's hook runs on one goroutine per block
 * (s2/writer.go:1052-1064, :455-461) and so do Decoder.DecodeAll / s2.Decode.  Every b2c_queue_* call blocks like the
 * function it replaces; a dispatcher thread owned by the queue gathers the calls that are pending (waiting up to
 * linger_us for more, at most max_batch per dispatch), issues one batched device call per kind of request and returns
 * each caller its byte count or negative error.  Thread-safe; src/dst are ordinary host memory, valid for the call.
 * b2c_queue_zstd_encode is EncodeAll for any input size: inputs of at most one block become single-block frames, larger
 * ones one multi-block frame each (frame mode); S2 blocks larger than 64 KiB are refused with B2C_ERR_TOO_BIG.
 */
typedef struct b2c_queue b2c_queue;
B2C_API b2c_queue *b2c_queue_create(int device, size_t max_batch, unsigned linger_us);
B2C_API void b2c_queue_destroy(b2c_queue *q);
B2C_API int64_t b2c_queue_zstd_encode(b2c_queue *q, int level, int flags, const void *src, size_t n, void *dst, size_t cap);
B2C_API int64_t b2c_queue_zstd_decode(b2c_queue *q, const void *src, size_t n, void *dst, size_t cap);
B2C_API int64_t b2c_queue_s2_encode(b2c_queue *q, int level, int flags, const void *src, size_t n, void *dst, size_t cap);
B2C_API int64_t b2c_queue_s2_decode(b2c_queue *q, const void *src, size_t n, void *dst, size_t cap);
B2C_API int b2c_queue_stats(b2c_queue *q, uint64_t *calls, uint64_t *batches);

#ifdef __cplusplus
}
#endif
#endif
