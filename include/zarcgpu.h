/* libzarcgpu — C ABI of the B200-native zarc content path.
 *
 * This is the drop-in boundary: every entry point replaces one call the reference (passcod/zarc,
 * Rust) makes into the `blake3` / `zstd-safe` crates on its content path, or batches many of them.
 * File:line citations are relative to the reference tree.  Plain pointers and sizes only; no
 * exceptions cross the boundary; the caller owns every buffer; contexts are opaque handles.
 *
 * Error convention = libzstd's (what crates/zarc/src/lib.rs:27-30 and decode/error.rs:35-38 map):
 * functions return size_t; values for which zg_is_error() is true are error codes; names via
 * zg_error_name().  Error numbers are libzstd 1.5.5's ZSTD_ErrorCode values.
 *
 * All content bytes are processed by hand-written sm_100a CUDA kernels; there is no CPU fallback.
 * Without a CUDA device every compute call returns ZG_error_no_device.
 */
#ifndef ZARCGPU_H
#define ZARCGPU_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZG_DIGEST_LEN 32 /* DigestType::digest_len(), crates/zarc/src/integrity.rs:98-104 */

typedef enum {
	ZG_error_no_error = 0,
	ZG_error_GENERIC = 1,
	ZG_error_prefix_unknown = 10,
	ZG_error_frameParameter_unsupported = 14,
	ZG_error_frameParameter_windowTooLarge = 16,
	ZG_error_corruption_detected = 20,
	ZG_error_checksum_wrong = 22,
	ZG_error_dictionary_wrong = 32,
	ZG_error_parameter_unsupported = 40,
	ZG_error_parameter_outOfBound = 42,
	ZG_error_memory_allocation = 64,
	ZG_error_dstSize_tooSmall = 70,
	ZG_error_srcSize_wrong = 72,
	ZG_error_dstBuffer_null = 74,
	ZG_error_device = 110,    /* a CUDA call failed (ours; below libzstd's maxCode 120) */
	ZG_error_no_device = 111, /* no CUDA device: the library never falls back to the CPU */
	ZG_error_maxCode = 120
} zg_error_code;

/* zstd_safe::get_error_name / ZSTD_isError (crates/zarc/src/lib.rs:28, decode/error.rs:36) */
int zg_is_error(size_t code);
const char* zg_error_name(size_t code);
zg_error_code zg_get_error_code(size_t code);

/* ---- device -------------------------------------------------------------------------------- */
int zg_device_count(void);
size_t zg_set_device(int device);
const char* zg_build_info(void); /* "sm_100a" for the product build */
/* page-locked host memory for callers that want full-rate host<->device copies (optional) */
void* zg_alloc_pinned(size_t bytes);
void zg_free_pinned(void* p);

/* ---- parameters (libzstd's ZSTD_cParameter numbers; crates/zarc/src/encode.rs:12,84-89;
 *      CLI mapping crates/zarc-cli/src/pack.rs:89-114,140-195,227-237) ---------------------- */
/* ZG_c_compressionLevel: -131072 .. 22 (0 = 3).  A negative level is libzstd's "fast" strategy with an acceleration
 * of -level: every literals section is Raw (no Huffman), and from -2 down the match finder probes pairs of positions
 * -level + 1 bytes apart (more after long stretches without a match).  The lower the level, the larger the frames.
 * Speed does not fall in step: measured on a B200, -1 packs faster than level 1 (no Huffman step), -2 to -4 are no
 * faster than -1 and can be slower than level 1 (the sampled parse advances less per step of the match finder), and
 * from about -5 down the sampling makes packing faster again (see profiles/fast_levels_1gpu.json).  An explicit
 * ZG_c_strategy >= 2 or ZG_c_searchLog overrides fast mode, as in libzstd: the level then acts as level 1.
 * ZG_c_hashLog, ZG_c_minMatch and ZG_c_windowLog keep their meaning at negative levels.  Setting a negative level
 * returns 0. */
typedef enum {
	ZG_c_compressionLevel = 100,
	ZG_c_windowLog = 101,
	ZG_c_hashLog = 102,
	ZG_c_chainLog = 103,
	ZG_c_searchLog = 104,
	ZG_c_minMatch = 105,
	ZG_c_targetLength = 106,
	ZG_c_strategy = 107,
	ZG_c_contentSizeFlag = 200,
	ZG_c_checksumFlag = 201,
	ZG_c_dictIDFlag = 202
} zg_cparameter;
typedef enum { ZG_reset_session_only = 1, ZG_reset_parameters = 2, ZG_reset_session_and_parameters = 3 } zg_reset_directive;

/* ---- BLAKE3 (replaces blake3::hash at encode/content_frame.rs:26, integrity.rs:110, and
 *      blake3::Hasher::{new,update,finalize} at decode/frame_iterator.rs:54,99,77) ------------ */
size_t zg_blake3(const void* data, size_t len, uint8_t out[ZG_DIGEST_LEN]);
typedef struct zg_hasher zg_hasher;
zg_hasher* zg_hasher_new(void);
size_t zg_hasher_update(zg_hasher*, const void* data, size_t len);
size_t zg_hasher_finalize(zg_hasher*, uint8_t out[ZG_DIGEST_LEN]); /* does not consume, like blake3 */
void zg_hasher_free(zg_hasher*);

/* ---- compression context (replaces zstd_safe::CCtx; encode.rs:61-62,84-89,
 *      encode/content_frame.rs:37-39, encode/lowlevel_frames.rs:30) --------------------------- */
typedef struct zg_cctx zg_cctx;
zg_cctx* zg_cctx_create(void);                                 /* CCtx::try_create, NULL on failure */
void zg_cctx_free(zg_cctx*);
size_t zg_cctx_init(zg_cctx*, int level);                       /* CCtx::init(level); 0 => default 3; < 0: fast, see above */
size_t zg_cctx_set_parameter(zg_cctx*, int param, int value);   /* returns the value set, like libzstd */
size_t zg_cctx_reset(zg_cctx*, int directive);                  /* CCtx::reset */
size_t zg_cctx_set_stream(zg_cctx*, void* cuda_stream);         /* run on a caller-owned cudaStream_t */
/* One complete Zstandard frame (header, blocks, XXH64 trailer when checksumFlag) into dst.
 * src/dst are HOST buffers.  Returns the frame length, or dstSize_tooSmall (never overruns). */
size_t zg_compress2(zg_cctx*, void* dst, size_t dst_capacity, const void* src, size_t src_size);
size_t zg_compress_bound(size_t src_size);

/* ---- decompression context (replaces zstd_safe::DCtx; decode/zstd_iterator.rs:29,88-153) ---- */
typedef struct zg_dctx zg_dctx;
typedef struct { void* dst; size_t size; size_t pos; } zg_out_buffer;      /* zstd_safe::OutBuffer */
typedef struct { const void* src; size_t size; size_t pos; } zg_in_buffer; /* zstd_safe::InBuffer */
zg_dctx* zg_dctx_create(void);
void zg_dctx_free(zg_dctx*);
size_t zg_dctx_set_stream(zg_dctx*, void* cuda_stream);
size_t zg_dctx_set_verify_checksum(zg_dctx*, int on); /* default 1, like libzstd */
/* Streaming decode with DCtx::decompress_stream's contract: consumes input, produces output,
 * returns 0 when the frame is complete and fully flushed, a non-zero hint otherwise. */
size_t zg_decompress_stream(zg_dctx*, zg_out_buffer* output, zg_in_buffer* input);
size_t zg_dstream_in_size(void);  /* DCtx::in_size()  = 131075 */
size_t zg_dstream_out_size(void); /* DCtx::out_size() = 131072 */
/* One-shot: decode exactly one frame at src (HOST buffers). Returns bytes written. */
size_t zg_decompress(zg_dctx*, void* dst, size_t dst_capacity, const void* src, size_t src_size);
size_t zg_find_frame_compressed_size(const void* src, size_t src_size);

/* ---- batched content path: the real hot path ------------------------------------------------
 * zg_pack_batch == for each file i in order: Encoder::add_data_frame(blob[off[i]..off[i]+len[i]])
 * (encode/content_frame.rs:20-60), with the Encoder's dedup map and running offset kept inside
 * the cctx across calls (cleared by zg_cctx_reset(ZG_reset_session_and_parameters) or
 * zg_cctx_reset_archive).
 *
 *   digests[i]      BLAKE3 of file i                                        (content_frame.rs:26)
 *   first[i]        1 if file i's content was not seen before (this call or earlier), else 0 (:30)
 *   frame_off[i]    archive offset of the frame holding file i's content    (Frame.offset, :22,:51)
 *   frame_len[i]    that frame's length incl. header and checksum           (Frame.length, :54)
 *   frames_out      the new frames, concatenated in insertion order; frames_out[0] sits at the
 *                   archive offset the cctx had on entry (zg_cctx_archive_offset)
 *   *frames_bytes   bytes appended to frames_out
 * Returns 0 or an error (dstSize_tooSmall if frames_cap is too small; nothing is overrun).
 * The `_dev` variant takes DEVICE pointers for every array and runs on the cctx stream.
 */
size_t zg_cctx_reset_archive(zg_cctx*, uint64_t first_frame_offset /* 12 after FILE_MAGIC, encode.rs:65 */);
uint64_t zg_cctx_archive_offset(const zg_cctx*);
size_t zg_pack_batch(zg_cctx*, const uint8_t* blob, const uint64_t* off, const uint64_t* len, uint64_t n_files,
                     uint8_t* digests, uint8_t* first, uint64_t* frame_off, uint64_t* frame_len,
                     uint8_t* frames_out, uint64_t frames_cap, uint64_t* frames_bytes);
size_t zg_pack_batch_dev(zg_cctx*, const uint8_t* blob, const uint64_t* off, const uint64_t* len, uint64_t n_files,
                         uint8_t* digests, uint8_t* first, uint64_t* frame_off, uint64_t* frame_len,
                         uint8_t* frames_out, uint64_t frames_cap, uint64_t* frames_bytes /* HOST */);

/* add_data_frame with its two decisions supplied by the caller, for archives packed by several GPUs (one rank per
 * GPU, files sharded; SURVEY.md 8e): `digests_in` (NULL: compute here) are the BLAKE3 digests of content_frame.rs:26,
 * which the ranks need BEFORE this call to take the first-occurrence decision of content_frame.rs:30 over the global
 * file order (zg_dedup_dev on the all-gathered digests); `select[i]` (NULL: all ones) is that decision.  A file with
 * select[i] == 0 gets no frame here: first[i] = 0, and frame_off[i] / frame_len[i] name the frame of an earlier identical
 * file of this context if there is one, else 0 / 0.  Device pointers. */
size_t zg_pack_batch_dev_ex(zg_cctx*, const uint8_t* blob, const uint64_t* off, const uint64_t* len, uint64_t n_files,
                            const uint8_t* digests_in, const uint8_t* select, uint8_t* digests, uint8_t* first,
                            uint64_t* frame_off, uint64_t* frame_len, uint8_t* frames_out, uint64_t frames_cap,
                            uint64_t* frames_bytes /* HOST */);

/* zg_unpack_batch == for each entry k: Decoder::read_content_frame -> FrameIterator drained
 * (decode/frame_iterator.rs:14-27,94-103) + verify() (:77,86-88).
 *   archive[off[k] .. off[k]+len[k])  one Zstandard frame (Frame.offset / Frame.length)
 *   ulen[k]                           Frame.uncompressed
 *   out[out_off[k] .. +ulen[k])       decoded bytes
 *   digests (may be NULL)             expected BLAKE3; ok[k] = 1 match, 0 mismatch (verify())
 *   status[k]                         0 or the zstd error code for frame k
 * Returns 0 if every frame decoded, else the error of the lowest failing k (others still decode).
 * A digest mismatch is NOT an error at this boundary (frame_iterator.rs:86-88, unpack.rs:118-120).
 * Host buffers (page-locked ones overlap the copies with the kernels): the batch goes through in slices, two of them
 * decoding at once -- the call runs one extra host thread while it lasts and the context keeps a helper context; results
 * do not depend on the slicing.  A context serves one call at a time (the reference owns one DCtx per frame iterator,
 * decode/zstd_iterator.rs:29; concurrent callers use one zg_dctx each).
 */
size_t zg_unpack_batch(zg_dctx*, const uint8_t* archive, uint64_t archive_len, uint64_t n_frames,
                       const uint64_t* off, const uint64_t* len, const uint64_t* ulen, const uint8_t* digests,
                       uint8_t* out, uint64_t out_cap, const uint64_t* out_off, uint8_t* ok, uint32_t* status);
size_t zg_unpack_batch_dev(zg_dctx*, const uint8_t* archive, uint64_t archive_len, uint64_t n_frames,
                           const uint64_t* off, const uint64_t* len, const uint64_t* ulen, const uint8_t* digests,
                           uint8_t* out, uint64_t out_cap, const uint64_t* out_off, uint8_t* ok, uint32_t* status);

/* Device-pointer entry points (`*_dev`): the kernels read their inputs as ALIGNED 4-byte words, so the word that holds
 * a buffer's last byte may be read whole -- up to 3 bytes past the end, inside the same aligned word, never written and
 * never used.  On a GPU such a word cannot leave the allocation; a byte-exact checker wants 4 bytes of slack after
 * `archive`, `blob` and `out`.  The host-buffer entry points stage through padded device buffers of their own. */

/* ---- building blocks exposed for tests / roofline measurement (device pointers) ------------- */
size_t zg_blake3_batch_dev(void* cuda_stream, const uint8_t* blob, const uint64_t* off, const uint64_t* len,
                           uint64_t n, uint8_t* digests);
size_t zg_blake3_batch(const uint8_t* blob, const uint64_t* off, const uint64_t* len, uint64_t n, uint8_t* digests);
size_t zg_xxh64_batch_dev(void* cuda_stream, const uint8_t* blob, const uint64_t* off, const uint64_t* len,
                          uint64_t n, uint64_t* hashes);
size_t zg_xxh64_batch(const uint8_t* blob, const uint64_t* off, const uint64_t* len, uint64_t n, uint64_t* hashes);
/* exclusive prefix sum of frame lengths -> archive offsets (content_frame.rs:22,45); `base` is
 * this rank's starting offset (after the cross-rank allgather of per-rank totals). */
size_t zg_assign_offsets_dev(void* cuda_stream, const uint64_t* frame_len, uint64_t n, uint64_t base, uint64_t* frame_off);

/* ---- synthetic corpora (SURVEY.md §8d): workload generation, not part of the content path --- */
size_t zg_corpus_generate_dev(void* cuda_stream, uint8_t* out, const uint64_t* seg_off, const uint32_t* seg_len,
                              const uint8_t* seg_kind, const uint64_t* seg_key, uint64_t n_segments);
size_t zg_corpus_generate_host(uint8_t* out, const uint64_t* seg_off, const uint32_t* seg_len,
                               const uint8_t* seg_kind, const uint64_t* seg_key, uint64_t n_segments);

/* first[i] = 1 iff digests[i] does not occur at a smaller index; rep[i] = that smallest index.
 * Device pointers.  (content_frame.rs:30 over an ordered digest list gathered from several GPUs.) */
size_t zg_dedup_dev(void* cuda_stream, const uint8_t* digests, uint64_t n, uint8_t* first, uint64_t* rep);

/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
uint64_t zg_kernel_launch_count(void);
/* optional per-kernel device timing (CUDA events on the launching stream) for roofline reports.
 * k: 0 BLAKE3, 1 Zstd encode, 2 Zstd decode, 3 frame assemble, 4 XXH64, 5 dedup,
 * 9 Huffman literals decoded ahead of the fused decoder (part of 2) */
void zg_profile_enable(int on);
size_t zg_profile_read(int k, double* total_ms, uint64_t* launches);

#ifdef __cplusplus
}
#endif
#endif
