/*
 * zeekstd_b200.h -- C ABI of the B200-native seekable-zstd codec.
 *
 * Drop-in boundary for the hot path of rorosen/zeekstd.  The reference crosses into native code
 * (libzstd via zstd-safe) at exactly these call sites, which this ABI replaces:
 *
 *   lib/src/encode.rs:341-345   cctx.compress_stream2(out, in, ZSTD_e_continue)   -> zk_compress_frames*
 *   lib/src/encode.rs:444-448   cctx.compress_stream2(out, empty, ZSTD_e_end)     -> zk_compress_frames*
 *   lib/src/encode.rs:281-284   cctx.set_parameter(CompressionLevel/ChecksumFlag)  -> level / checksum args
 *   lib/src/encode.rs:504-506   cctx.reset(SessionOnly)                            -> (frames are independent)
 *   lib/src/decode.rs:243-245   dctx.decompress_stream(out, in)                    -> zk_decompress_frames*
 *   lib/src/decode.rs:354-356   dctx.reset(SessionOnly)                            -> (stateless per call)
 *   lib/src/error.rs:68,125     zstd_safe::get_error_name                          -> zk_error_name
 *
 * The libzstd interface is a one-context, 128 KiB-at-a-time stream; it cannot express a batch.  Each
 * independent frame of the seekable format (seekable_format.md:23-29) is one unit of data parallelism,
 * so the batch entry points take whole frames.  On top of them the "mirror" layer (zk_raw_encoder_*,
 * zk_encoder_*, zk_decoder_*, zk_seek_table_*) re-exposes the reference's Rust API surface one C
 * function per method so that a Rust (or any FFI) wrapper is mechanical -- see INTEGRATION.md.
 *
 * Conventions
 *   - plain C, opaque handles, no exceptions cross the boundary, caller owns all byte buffers;
 *   - return value int32_t: 0 = ok, < 0 = error (ZK_ERR_* or -(libzstd ZSTD_ErrorCode), e.g. -20
 *     corruption_detected, -22 checksum_wrong, -70 dstSize_tooSmall) -- the numeric zstd codes are kept
 *     so that Error::is_zstd()/get_error_name() (error.rs:40-45,101-113) stay meaningful;
 *   - a zk_ctx is NOT thread-safe (one per host thread / GPU), like CCtx/DCtx; calls are synchronous;
 *   - there is NO CPU fallback: zk_ctx_create fails with ZK_ERR_NO_DEVICE when no CUDA device exists.
 */
#ifndef ZEEKSTD_B200_H
#define ZEEKSTD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ constants (lib/src/lib.rs:49-62) */
#define ZK_SEEKABLE_MAGIC_NUMBER 0x8F92EAB1u
#define ZK_SEEKABLE_MAX_FRAMES 0x08000000u
#define ZK_SEEK_TABLE_INTEGRITY_SIZE 9u
#define ZK_SEEKABLE_MAX_FRAME_SIZE 0x40000000u
#define ZK_SKIPPABLE_HEADER_SIZE 8u
#define ZK_DEFAULT_FRAME_SIZE 0x200000u /* FrameSizePolicy::default(), encode.rs:33-39 */

/* ------------------------------------------------------------------ errors (lib/src/error.rs:101-113) */
#define ZK_OK 0
#define ZK_ERR_NUMBER_CONVERSION (-1001) /* Kind::NumberConversionFailed */
#define ZK_ERR_OFFSET_OUT_OF_RANGE (-1002) /* Kind::OffsetOutOfRange       */
#define ZK_ERR_FRAME_INDEX_TOO_LARGE (-1003) /* Kind::FrameIndexTooLarge     */
#define ZK_ERR_IO (-1004) /* Kind::IO                     */
#define ZK_ERR_NO_DEVICE (-1005) /* no CUDA device / CUDA failure: the product never falls back to the CPU */
#define ZK_ERR_INVALID_ARG (-1006)
#define ZK_ERR_CUDA (-1007) /* a CUDA runtime call or a kernel failed after the context was created; zk_last_cuda_error() has the text */
/* Kind::Zstd(code): returned as -(ZSTD_ErrorCode), i.e. in [-120, -1] */
#define ZK_ERR_ZSTD(code) (-(int32_t)(code))
#define ZK_IS_ZSTD_ERR(rc) ((rc) < 0 && (rc) > -1000)

const char* zk_error_name(int32_t rc);
/* cudaGetErrorString of the most recent CUDA failure seen by this thread ("" if none) */
const char* zk_last_cuda_error(void);

/* ------------------------------------------------------------------ context (CCtx/DCtx, encode.rs:130, decode.rs:31) */
typedef struct zk_ctx zk_ctx;
int32_t zk_ctx_create(int32_t device_ordinal, uint32_t flags, zk_ctx** out);
void zk_ctx_destroy(zk_ctx* ctx);
/* number of CUDA kernels this context has launched so far (bench.py reports it as gpu_launches) */
uint64_t zk_ctx_kernel_launches(const zk_ctx* ctx);
/* kernel-only device time (ms, CUDA events on the context's stream) of the most recent batch call */
float zk_ctx_last_device_ms(const zk_ctx* ctx);
const char* zk_version(void);
/* per-kernel device time (CUDA events on the launching stream), accumulated while enabled.
 * slots: 0 scan, 1 seq, 2 huf, 3 exec, 4 xxh64, 5 match, 6 entropy-enc, 7 frame assembly; arrays of 8 */
void zk_ctx_profile(zk_ctx* ctx, int32_t enable);
void zk_ctx_profile_read(const zk_ctx* ctx, float* ms, uint32_t* launches);

/* ------------------------------------------------------------------ batch codec: the hot path */
/* Upper bound of the compressed size of n input bytes cut into frames of frame_size (excl. seek table). */
size_t zk_compress_bound(size_t n, uint32_t frame_size);

/*
 * Compress src[0..n) into ceil(n / frame_size) independent zstd frames written back to back into dst
 * (FrameSizePolicy::Uncompressed, encode.rs:528-544).  c_sizes / d_sizes (capacity frames_cap) receive
 * what RawEncoder would pass to SeekTable::log_frame (encode.rs:466).  n == 0 produces one empty frame,
 * like Encoder::finish() on an empty stream (encode.rs:755-756).  HOST pointers (pinned memory is faster).
 */
int32_t zk_compress_frames(zk_ctx* ctx, const uint8_t* src, size_t n, uint32_t frame_size, int32_t level,
                           int32_t checksum, uint8_t* dst, size_t dst_cap, uint32_t* c_sizes, uint32_t* d_sizes,
                           uint32_t frames_cap, uint32_t* n_frames, size_t* dst_len);

/*
 * Decompress n_frames seek-table entries.  Entry f occupies comp[c_off[f] .. c_off[f+1]) and decodes to
 * dst[d_off[f] .. d_off[f+1]) (the N+1 cumulative offsets of SeekTable, seek_table.rs:97-101, rebased by
 * the caller to the two pointers).  status[f] (optional) = 0 or -(zstd code).  With verify_checksum != 0
 * frames that carry a content checksum are verified (-22 on mismatch).  HOST pointers.
 * Returns 0 or the first failing frame's status.
 */
int32_t zk_decompress_frames(zk_ctx* ctx, const uint8_t* comp, const uint64_t* c_off, const uint64_t* d_off,
                             uint32_t n_frames, uint8_t* dst, int32_t verify_checksum, int32_t* status);

/* Range reads (SURVEY.md 8f.1; decode.rs:228-266 decodes a frame only as far as offset_limit): like
 * zk_decompress_frames, but entry i is only guaranteed to hold its first d_need[i] bytes afterwards (the decoder stops at
 * the first block boundary at or after that point; the rest of the entry's output range is unspecified).  A prefix is
 * not checksum-verified, as in the reference (decode.rs:425-427).  d_need == NULL or d_need[i] >= the entry's size: everything. */
int32_t zk_decompress_frames_upto(zk_ctx* ctx, const uint8_t* comp, const uint64_t* c_off, const uint64_t* d_off,
                                  uint32_t n_frames, uint8_t* dst, const uint32_t* d_need, int32_t verify_checksum, int32_t* status);

/*
 * Prefix / patch mode: the same calls with a raw-content prefix that precedes EVERY frame (the reference re-applies it per
 * frame: cctx.ref_prefix at each frame start, encode.rs:332-338; dctx.ref_prefix before the first frame and after every frame
 * end, decode.rs:211-214, 246-255).  Matches may reach back into the prefix; frames made this way only decode with the same
 * prefix (libzstd: ZSTD_CCtx_refPrefix / ZSTD_DCtx_refPrefix).  prefix == NULL or prefix_len == 0: the plain calls.  HOST pointers.
 */
int32_t zk_compress_frames_prefix(zk_ctx* ctx, const uint8_t* src, size_t n, uint32_t frame_size, int32_t level,
                                  int32_t checksum, const uint8_t* prefix, size_t prefix_len, uint8_t* dst, size_t dst_cap,
                                  uint32_t* c_sizes, uint32_t* d_sizes, uint32_t frames_cap, uint32_t* n_frames, size_t* dst_len);
int32_t zk_decompress_frames_prefix(zk_ctx* ctx, const uint8_t* comp, const uint64_t* c_off, const uint64_t* d_off,
                                    uint32_t n_frames, uint8_t* dst, const uint32_t* d_need, int32_t verify_checksum,
                                    int32_t* status, const uint8_t* prefix, size_t prefix_len);

/*
 * Context parameters (the ones the reference's CLI sets on its CCtx / DCtx for patch files, cli/src/compress.rs:31-37,
 * cli/src/decompress.rs:53-62).  A zk_ctx plays both roles, so both kinds live on it.  They are sticky, like libzstd's, and apply
 * to every batch and mirror call made on the context.  Value 0 restores the default.  Unknown parameter: ZK_ERR_ZSTD(40)
 * (parameter_unsupported); value out of range: ZK_ERR_ZSTD(42) (parameter_outOfBound).
 *
 *   ZK_C_WINDOW_LOG (0, 10..30)          the Window_Descriptor announces max(the level's own window, 2^value); no offset the
 *                                        encoder emits exceeds the announced window.  Values below a level's window change nothing.
 *   ZK_C_ENABLE_LONG_DISTANCE_MATCHING   0 / 1.  Takes effect in prefix calls only: the part of the prefix the window reaches is
 *   (0, 1)                               indexed on the device and every block of every frame searches it.  With window log 0 the
 *                                        window is 2^27, as in libzstd.  Without a prefix it is a no-op for now (no in-frame
 *                                        long-distance matching yet).
 *   ZK_D_WINDOW_LOG_MAX (0, 10..30)      frames announcing a window above 2^value are refused (ZK_ERR_ZSTD(16)); default (0):
 *                                        2^27 + 1, the limit of a default ZSTD_DCtx.
 *
 * Window logs stop at 30, one below libzstd's 64-bit maximum: the decoder keeps every concrete offset below 2^31.
 */
#define ZK_C_WINDOW_LOG 101                      /* = ZSTD_c_windowLog */
#define ZK_C_ENABLE_LONG_DISTANCE_MATCHING 160   /* = ZSTD_c_enableLongDistanceMatching */
#define ZK_D_WINDOW_LOG_MAX 100                  /* = ZSTD_d_windowLogMax */
#define ZK_WINDOWLOG_MIN 10
#define ZK_WINDOWLOG_MAX 30
int32_t zk_ctx_set_cparameter(zk_ctx* ctx, int32_t param, int32_t value);
int32_t zk_ctx_set_dparameter(zk_ctx* ctx, int32_t param, int32_t value);

/*
 * Device-resident variants (zero-copy; used for roofline measurements and multi-GPU pipelines).
 * d_* are CUDA device pointers, 16-byte aligned, with >= 16 readable bytes after the last byte;
 * offset / size arrays stay on the HOST.  cuda_stream is a cudaStream_t (NULL = the context's own
 * non-blocking stream; pass cudaStreamLegacy (0x1) to order the work on the legacy default stream, e.g.
 * after PyTorch ops).  The call returns after the work has completed on that stream.
 */
int32_t zk_compress_frames_dev(zk_ctx* ctx, const void* d_src, size_t n, uint32_t frame_size, int32_t level,
                               int32_t checksum, void* d_dst, size_t dst_cap, uint32_t* c_sizes, uint32_t* d_sizes,
                               uint32_t frames_cap, uint32_t* n_frames, size_t* dst_len, void* cuda_stream);
int32_t zk_decompress_frames_dev(zk_ctx* ctx, const void* d_comp, const uint64_t* c_off, const uint64_t* d_off,
                                 uint32_t n_frames, void* d_dst, int32_t verify_checksum, int32_t* status,
                                 void* cuda_stream);

/* ------------------------------------------------------------------ SeekTable (lib/src/seek_table.rs) */
typedef struct zk_seek_table zk_seek_table;
typedef enum { ZK_FORMAT_HEAD = 0, ZK_FORMAT_FOOT = 1 } zk_format; /* seek_table.rs:228-241 */

zk_seek_table* zk_seek_table_new(void);                                             /* SeekTable::new  :314 */
void zk_seek_table_free(zk_seek_table* st);
zk_seek_table* zk_seek_table_clone(const zk_seek_table* st);
/* SeekTable::from_seekable_format over a memory span (BytesWrapper), seek_table.rs:379-436 */
int32_t zk_seek_table_from_bytes(const uint8_t* buf, size_t len, zk_format format, zk_seek_table** out);
int32_t zk_seek_table_log_frame(zk_seek_table* st, uint32_t c_size, uint32_t d_size); /* :513-525 */
uint32_t zk_seek_table_num_frames(const zk_seek_table* st);                           /* :540 */
uint32_t zk_seek_table_frame_index_comp(const zk_seek_table* st, uint64_t offset);    /* :560 */
uint32_t zk_seek_table_frame_index_decomp(const zk_seek_table* st, uint64_t offset);  /* :580 */
int32_t zk_seek_table_frame_start_comp(const zk_seek_table* st, uint32_t index, uint64_t* out);
int32_t zk_seek_table_frame_start_decomp(const zk_seek_table* st, uint32_t index, uint64_t* out);
int32_t zk_seek_table_frame_end_comp(const zk_seek_table* st, uint32_t index, uint64_t* out);
int32_t zk_seek_table_frame_end_decomp(const zk_seek_table* st, uint32_t index, uint64_t* out);
int32_t zk_seek_table_frame_size_comp(const zk_seek_table* st, uint32_t index, uint64_t* out);
int32_t zk_seek_table_frame_size_decomp(const zk_seek_table* st, uint32_t index, uint64_t* out);
uint64_t zk_seek_table_max_frame_size_comp(const zk_seek_table* st);
uint64_t zk_seek_table_max_frame_size_decomp(const zk_seek_table* st);
uint64_t zk_seek_table_size_comp(const zk_seek_table* st);
uint64_t zk_seek_table_size_decomp(const zk_seek_table* st);
/* copies the N+1 cumulative offsets (c then d may be NULL); returns N+1 */
uint32_t zk_seek_table_offsets(const zk_seek_table* st, uint64_t* c_off, uint64_t* d_off, uint32_t cap);

/* Serializer (seek_table.rs:955-1051): resumable at byte granularity */
typedef struct zk_serializer zk_serializer;
zk_serializer* zk_seek_table_into_serializer(const zk_seek_table* st, zk_format format); /* :885-905 */
void zk_serializer_free(zk_serializer* s);
size_t zk_serializer_write_into(zk_serializer* s, uint8_t* buf, size_t len);          /* :967-1005 */
void zk_serializer_reset(zk_serializer* s);                                            /* :1021 */
size_t zk_serializer_encoded_len(const zk_serializer* s);                             /* :1038 */

/* ------------------------------------------------------------------ EncodeOptions / RawEncoder / Encoder (lib/src/encode.rs) */
typedef struct zk_encode_options zk_encode_options;
typedef struct zk_raw_encoder zk_raw_encoder;
typedef struct zk_encoder zk_encoder;
typedef enum { ZK_POLICY_COMPRESSED = 0, ZK_POLICY_UNCOMPRESSED = 1 } zk_frame_size_policy; /* encode.rs:21-31 */
typedef struct { size_t in_progress, out_progress; } zk_compression_progress;           /* encode.rs:43-65 */
typedef struct { size_t out_progress, data_left; } zk_epilogue_progress;                /* encode.rs:69-92 */
/* Write sink (W: std::io::Write, encode.rs:570): must consume all len bytes; return 0 on success */
typedef int32_t (*zk_write_fn)(void* user, const uint8_t* data, size_t len);
typedef int32_t (*zk_flush_fn)(void* user);

zk_encode_options* zk_encode_options_new(zk_ctx* ctx);                                  /* encode.rs:124 */
void zk_encode_options_free(zk_encode_options* o);
void zk_encode_options_frame_size_policy(zk_encode_options* o, zk_frame_size_policy kind, uint32_t size); /* :158 */
void zk_encode_options_checksum_flag(zk_encode_options* o, int32_t flag);               /* :166 */
void zk_encode_options_compression_level(zk_encode_options* o, int32_t level);          /* :176 */
/* consume the options (like `self`) */
int32_t zk_encode_options_into_raw_encoder(zk_encode_options* o, zk_raw_encoder** out); /* :188 */
int32_t zk_encode_options_into_encoder(zk_encode_options* o, zk_write_fn write, zk_flush_fn flush, void* user,
                                       zk_encoder** out);                               /* :204 */

void zk_raw_encoder_free(zk_raw_encoder* e);
int32_t zk_raw_encoder_compress(zk_raw_encoder* e, const uint8_t* input, size_t in_len, uint8_t* output,
                                size_t out_len, zk_compression_progress* progress);     /* :398 / 311-354 */
/* RawEncoder::compress_with_prefix: the prefix given at a frame's FIRST call is that frame's raw-content prefix (it must stay
 * valid until the frame is closed -- 'b: 'a in the reference); NULL = none */
int32_t zk_raw_encoder_compress_with_prefix(zk_raw_encoder* e, const uint8_t* input, size_t in_len, uint8_t* output,
                                            size_t out_len, const uint8_t* prefix, size_t prefix_len,
                                            zk_compression_progress* progress);            /* :311-354 */
int32_t zk_raw_encoder_end_frame(zk_raw_encoder* e, uint8_t* output, size_t out_len,
                                 zk_epilogue_progress* progress);                       /* :438-472 */
const zk_seek_table* zk_raw_encoder_seek_table(const zk_raw_encoder* e);               /* :479 */
zk_seek_table* zk_raw_encoder_into_seek_table(zk_raw_encoder* e);                      /* :492 (consumes e) */
void zk_raw_encoder_reset_frame(zk_raw_encoder* e);                                     /* :501-507 */
void zk_raw_encoder_reset_seek_table(zk_raw_encoder* e);                                /* :524 */

void zk_encoder_free(zk_encoder* e);
int32_t zk_encoder_compress(zk_encoder* e, const uint8_t* buf, size_t len, size_t* consumed); /* :692 / 641-665 */
int32_t zk_encoder_compress_with_prefix(zk_encoder* e, const uint8_t* buf, size_t len, const uint8_t* prefix,
                                        size_t prefix_len, size_t* consumed);               /* :641-665 */
int32_t zk_encoder_end_frame(zk_encoder* e, size_t* written);                          /* :704-717 */
int32_t zk_encoder_flush(zk_encoder* e);                                                /* impl Write::flush :796 */
/* finish()/finish_format() consume the encoder; *total = bytes written to the sink incl. seek table */
int32_t zk_encoder_finish(zk_encoder* e, uint64_t* total);                              /* :743 */
int32_t zk_encoder_finish_format(zk_encoder* e, zk_format format, uint64_t* total);     /* :755-775 */
uint64_t zk_encoder_written_compressed(const zk_encoder* e);                            /* :615 */
const zk_seek_table* zk_encoder_seek_table(const zk_encoder* e);                        /* :609 */

/* ------------------------------------------------------------------ Seekable source + Decoder (lib/src/seekable.rs, decode.rs) */
/* trait Seekable (seekable.rs:16-39) as callbacks.  whence: 0 = OffsetFrom::Start(u64), 1 = OffsetFrom::End(i64) */
typedef struct {
    void* user;
    int64_t (*set_offset)(void* user, int32_t whence, int64_t offset); /* -> new absolute position or < 0 */
    int64_t (*read)(void* user, uint8_t* buf, size_t len);             /* -> bytes read (0 = EOF) or < 0 */
} zk_seekable;

typedef struct zk_decode_options zk_decode_options;
typedef struct zk_decoder zk_decoder;

/* DecodeOptions::new(src) with src = BytesWrapper over memory (seekable.rs:43-97); bytes must outlive the decoder */
zk_decode_options* zk_decode_options_new_bytes(zk_ctx* ctx, const uint8_t* src, size_t len);
/* DecodeOptions::new(src) with a generic Seekable */
zk_decode_options* zk_decode_options_new_seekable(zk_ctx* ctx, zk_seekable src);
void zk_decode_options_free(zk_decode_options* o);
void zk_decode_options_seek_table(zk_decode_options* o, const zk_seek_table* st);     /* decode.rs:69 (copied) */
void zk_decode_options_lower_frame(zk_decode_options* o, uint32_t index);              /* :77 */
void zk_decode_options_upper_frame(zk_decode_options* o, uint32_t index);              /* :85 */
void zk_decode_options_offset(zk_decode_options* o, uint64_t offset);                  /* :95 */
void zk_decode_options_offset_limit(zk_decode_options* o, uint64_t limit);             /* :105 */
int32_t zk_decode_options_into_decoder(zk_decode_options* o, zk_decoder** out);        /* :111 / 152-187 (consumes o) */

void zk_decoder_free(zk_decoder* d);
int32_t zk_decoder_decompress(zk_decoder* d, uint8_t* buf, size_t len, size_t* produced); /* :314 / 201-270 */
/* Decoder::decompress_with_prefix: every frame is decoded against the raw-content prefix (decode.rs:211-214, 246-255) */
int32_t zk_decoder_decompress_with_prefix(zk_decoder* d, uint8_t* buf, size_t len, const uint8_t* prefix,
                                          size_t prefix_len, size_t* produced);            /* :201-270 */
void zk_decoder_reset(zk_decoder* d);                                                    /* :346-350 */
int32_t zk_decoder_set_lower_frame(zk_decoder* d, uint32_t index, uint64_t* offset);    /* :367 */
int32_t zk_decoder_set_upper_frame(zk_decoder* d, uint32_t index, uint64_t* offset);    /* :383 */
int32_t zk_decoder_set_offset(zk_decoder* d, uint64_t offset);                           /* :402-414 */
int32_t zk_decoder_set_offset_limit(zk_decoder* d, uint64_t limit);                      /* :432-437 */
uint64_t zk_decoder_read_compressed(const zk_decoder* d);                                /* :448 */
uint64_t zk_decoder_offset(const zk_decoder* d);                                         /* :458 */
uint64_t zk_decoder_offset_limit(const zk_decoder* d);                                   /* :463 */
const zk_seek_table* zk_decoder_seek_table(const zk_decoder* d);                        /* :453 */
/* impl Seek for Decoder (decode.rs:545-579): whence 0 = Start, 1 = End, 2 = Current */
int32_t zk_decoder_seek(zk_decoder* d, int32_t whence, int64_t offset, uint64_t* new_offset);

#ifdef __cplusplus
}
#endif
#endif /* ZEEKSTD_B200_H */
