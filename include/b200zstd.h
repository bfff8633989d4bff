/*
 * b200zstd.h -- C ABI of the B200-native zstd block decompressor (libb200zstd.so).
 *
 * Drop-in boundary for the decode hot path of ruzstd (KillingSpark/zstd-rs @ eb7e03cc, crate ruzstd 0.9.1).
 * Everything below replaces work that the reference does inside
 *     BlockDecoder::decompress_block            ruzstd/src/decoding/block_decoder.rs:97-197
 * called from the block loops of
 *     FrameDecoder::decode_blocks               ruzstd/src/decoding/frame_decoder.rs:309-377
 *     FrameDecoder::decode_from_to              ruzstd/src/decoding/frame_decoder.rs:439-529
 * i.e. decode_literals (literals_section_decoder.rs:12), decode_sequences (sequence_section_decoder.rs:14),
 * execute_sequences (sequence_execution.rs:5) and DecodeBuffer::{push,repeat} (decode_buffer.rs:74,79), with
 * HuffmanTable / FSETable (huff0_decoder.rs:57, fse_decoder.rs:59) built and kept on the GPU.
 *
 * Plain C: opaque handles, pointers and sizes only.  No torch / CUDA types in any signature (a stream is passed
 * as void*).  No process-global state; a handle may migrate between threads but is used by one at a time
 * (the reference's FrameDecoder is Send + Sync, tests/mod.rs:37-45).  Nothing here ever falls back to a CPU
 * decoder: if no CUDA device is usable, b200z_ctx_create fails with B200Z_ERR_NO_DEVICE and every other entry
 * point needs a ctx.
 *
 * Error convention: int return, 0 = ok, >0 = b200z_error (one code per leaf of the reference's nested error
 * enums, decoding/errors.rs; numbering shared with the test oracle).  b200z_*_last_stage tells which stage
 * raised it (the nesting path in the reference).
 */
#ifndef B200ZSTD_H
#define B200ZSTD_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200Z_ABI_VERSION 1

typedef enum b200z_error {

    B200Z_OK = 0,
    /* ReadFrameHeaderError (errors.rs:95-104) */
    B200Z_ERR_MAGIC_NUMBER_READ = 1,
    B200Z_ERR_BAD_MAGIC_NUMBER = 2,
    B200Z_ERR_FRAME_DESCRIPTOR_READ = 3,
    B200Z_ERR_INVALID_FRAME_DESCRIPTOR = 4,
    B200Z_ERR_WINDOW_DESCRIPTOR_READ = 5,
    B200Z_ERR_DICTIONARY_ID_READ = 6,
    B200Z_ERR_FRAME_CONTENT_SIZE_READ = 7,
    B200Z_ERR_SKIP_FRAME = 8,
    /* FrameHeaderError (errors.rs:34-42) / FrameDecoderError (errors.rs:472-486) */
    B200Z_ERR_WINDOW_TOO_BIG = 10,
    B200Z_ERR_WINDOW_TOO_SMALL = 11,
    B200Z_ERR_WINDOW_SIZE_TOO_BIG = 12,
    B200Z_ERR_DICT_NOT_PROVIDED = 13,
    B200Z_ERR_NOT_YET_INITIALIZED = 14,
    B200Z_ERR_FAILED_TO_READ_CHECKSUM = 15,
    B200Z_ERR_FAILED_TO_DRAIN_DECODEBUFFER = 16,
    B200Z_ERR_FAILED_TO_SKIP_FRAME = 17,
    B200Z_ERR_TARGET_TOO_SMALL = 18,
    /* BlockHeaderReadError (errors.rs:156-161) */
    B200Z_ERR_BLOCK_HEADER_READ = 20,
    B200Z_ERR_FOUND_RESERVED_BLOCK = 21,
    B200Z_ERR_BLOCK_SIZE_TOO_LARGE = 22,
    /* DecodeBlockContentError / DecompressBlockError (errors.rs:345-350, 256-267) */
    B200Z_ERR_DECODER_STATE_IS_FAILED = 30,
    B200Z_ERR_EXPECTED_HEADER_OF_PREVIOUS_BLOCK = 31,
    B200Z_ERR_BLOCK_BODY_READ = 32,
    B200Z_ERR_BLOCK_CONTENT_READ = 33,
    B200Z_ERR_MALFORMED_SECTION_HEADER = 34,
    /* LiteralsSectionParseError / SequencesHeaderParseError (errors.rs:816-820, 870-872) */
    B200Z_ERR_LITSEC_ILLEGAL_TYPE = 40,
    B200Z_ERR_LITSEC_GET_BITS = 41,
    B200Z_ERR_LITSEC_NOT_ENOUGH_BYTES = 42,
    B200Z_ERR_SEQHDR_NOT_ENOUGH_BYTES = 45,
    /* DecompressLiteralsError (errors.rs:586-598) */
    B200Z_ERR_LIT_MISSING_COMPRESSED_SIZE = 50,
    B200Z_ERR_LIT_MISSING_NUM_STREAMS = 51,
    B200Z_ERR_LIT_GET_BITS = 52,
    B200Z_ERR_LIT_UNINITIALIZED_HUFFMAN_TABLE = 55,
    B200Z_ERR_LIT_MISSING_BYTES_FOR_JUMP_HEADER = 56,
    B200Z_ERR_LIT_MISSING_BYTES_FOR_LITERALS = 57,
    B200Z_ERR_LIT_EXTRA_PADDING = 58,
    B200Z_ERR_LIT_BITSTREAM_READ_MISMATCH = 59,
    B200Z_ERR_LIT_DECODED_LITERAL_COUNT_MISMATCH = 60,
    /* HuffmanTableError (errors.rs:991-1028) */
    B200Z_ERR_HUF_GET_BITS = 70,
    B200Z_ERR_HUF_FSE_DECODER = 71,
    B200Z_ERR_HUF_SOURCE_IS_EMPTY = 72,
    B200Z_ERR_HUF_NOT_ENOUGH_BYTES_FOR_WEIGHTS = 73,
    B200Z_ERR_HUF_EXTRA_PADDING = 74,
    B200Z_ERR_HUF_TOO_MANY_WEIGHTS = 75,
    B200Z_ERR_HUF_MISSING_WEIGHTS = 76,
    B200Z_ERR_HUF_LEFTOVER_NOT_POWER_OF_2 = 77,
    B200Z_ERR_HUF_NOT_ENOUGH_BYTES_TO_DECOMPRESS_WEIGHTS = 78,
    B200Z_ERR_HUF_FSE_TABLE_USED_TOO_MANY_BYTES = 79,
    B200Z_ERR_HUF_NOT_ENOUGH_BYTES_IN_SOURCE = 80,
    B200Z_ERR_HUF_WEIGHT_BIGGER_THAN_MAX_NUM_BITS = 81,
    B200Z_ERR_HUF_MAX_BITS_TOO_HIGH = 82,
    /* FSETableError (errors.rs:892-908); the same leaf can surface under Huffman weights, sequence
     * tables or a dictionary -- the code is the leaf, zo_last_error_stage() tells where. */
    B200Z_ERR_FSE_ACC_LOG_IS_ZERO = 90,
    B200Z_ERR_FSE_ACC_LOG_TOO_BIG = 91,
    B200Z_ERR_FSE_GET_BITS = 92,
    B200Z_ERR_FSE_PROBABILITY_COUNTER_MISMATCH = 93,
    B200Z_ERR_FSE_TOO_MANY_SYMBOLS = 94,
    B200Z_ERR_FSE_TABLE_IS_UNINITIALIZED = 95, /* FSEDecoderError::TableIsUninitialized (errors.rs:957-960) */
    /* DecodeSequenceError (errors.rs:726-739) */
    B200Z_ERR_SEQ_EXTRA_PADDING = 100,
    B200Z_ERR_SEQ_UNSUPPORTED_OFFSET = 101,
    B200Z_ERR_SEQ_ZERO_OFFSET = 102,
    B200Z_ERR_SEQ_NOT_ENOUGH_BYTES_FOR_NUM_SEQUENCES = 103,
    B200Z_ERR_SEQ_EXTRA_BITS = 104,
    B200Z_ERR_SEQ_MISSING_COMPRESSION_MODE = 105,
    B200Z_ERR_SEQ_MISSING_BYTE_FOR_RLE_LL_TABLE = 106,
    B200Z_ERR_SEQ_MISSING_BYTE_FOR_RLE_OF_TABLE = 107,
    B200Z_ERR_SEQ_MISSING_BYTE_FOR_RLE_ML_TABLE = 108,
    /* ExecuteSequencesError / DecodeBufferError (errors.rs:683-687, 393-396) */
    B200Z_ERR_EXEC_NOT_ENOUGH_BYTES_FOR_SEQUENCE = 110,
    B200Z_ERR_EXEC_ZERO_OFFSET = 111,
    B200Z_ERR_EXEC_NOT_ENOUGH_BYTES_IN_DICTIONARY = 112,
    B200Z_ERR_EXEC_OFFSET_TOO_BIG = 113,
    /* DictionaryDecodeError (errors.rs:419-424) */
    B200Z_ERR_DICT_NOT_ENOUGH_BYTES = 120,
    B200Z_ERR_DICT_BAD_MAGIC_NUM = 121,
    /* Places where the reference would panic (assert!/unreachable!/index out of bounds) instead of
     * returning an error; SURVEY.md Appendix B.8.  Never produced by spec-valid input. */
    B200Z_ERR_REFERENCE_WOULD_PANIC = 200,
    /* Resource limits of this build (documented deviations, never hit by spec-valid input). */
    B200Z_ERR_BLOCK_OUTPUT_LIMIT = 210,
    B200Z_ERR_INVALID_ARGUMENT = 220,
    B200Z_ERR_OUT_OF_MEMORY = 221
    ,
    /* this build only */
    B200Z_ERR_NO_DEVICE = 230,
    B200Z_ERR_CUDA = 231
} b200z_error;

/* stage that raised the error == nesting path of the reference's FrameDecoderError (errors.rs:472-486) */
typedef enum b200z_stage {
    B200Z_STAGE_NONE = 0,
    B200Z_STAGE_FRAME_HEADER = 1, /* ReadFrameHeaderError / FrameHeaderError                          */
    B200Z_STAGE_BLOCK_HEADER = 2, /* FailedToReadBlockHeader(BlockHeaderReadError)                    */
    B200Z_STAGE_BLOCK_BODY = 3,   /* FailedToReadBlockBody(DecodeBlockContentError / section headers) */
    B200Z_STAGE_LITERALS = 4,     /* ... DecompressLiteralsError                                      */
    B200Z_STAGE_SEQUENCES = 5,    /* ... DecodeSequenceError                                          */
    B200Z_STAGE_EXECUTE = 6,      /* ... ExecuteSequencesError                                        */
    B200Z_STAGE_CHECKSUM = 7,     /* FailedToReadChecksum                                             */
    B200Z_STAGE_DICTIONARY = 8,   /* DictionaryDecodeError                                            */
    B200Z_STAGE_DRAIN = 9         /* FailedToDrainDecodebuffer                                        */
} b200z_stage;

const char *b200z_error_name(int code);
int b200z_abi_version(void);

/* ------------------------------------------------------------------------------------------------------------
 * Device context: pins one CUDA device, owns its stream(s) and scratch pools.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct b200z_ctx b200z_ctx;
int b200z_ctx_create(int device_ordinal, b200z_ctx **out);
void b200z_ctx_destroy(b200z_ctx *ctx);
const char *b200z_ctx_last_error_message(const b200z_ctx *ctx);
/* the CUDA stream (cudaStream_t as void*) all work of this ctx is enqueued on; for event timing by callers */
void *b200z_ctx_stream(const b200z_ctx *ctx);
/* Context flags.  B200Z_FLAG_CHECKSUM: the batch entry also computes every frame's content checksum on the GPU (XXH64 seed 0 over
 * the plaintext, the hash the reference feeds while draining, decode_buffer.rs:225-226,290,301) and returns it in
 * b200z_frame_result.calculated_checksum -- like the reference it is reported, never enforced (frame_decoder.rs:253-270).
 * Device output buffers must be readable 8 bytes past their end when this flag is set. */
#define B200Z_FLAG_CHECKSUM 1u
void b200z_ctx_set_flags(b200z_ctx *ctx, uint32_t flags);
uint32_t b200z_ctx_flags(const b200z_ctx *ctx);
/* number of this library's kernel launches since ctx creation (bench.py's gpu_launches) */
uint64_t b200z_ctx_kernel_launches(const b200z_ctx *ctx);

/* ------------------------------------------------------------------------------------------------------------
 * Dictionaries (device resident).  Replaces Dictionary::decode_dict (decoding/dictionary.rs:45-126) +
 * FrameDecoder::add_dict (frame_decoder.rs:224-227); tables are expanded on the GPU.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct b200z_dict b200z_dict;
int b200z_dict_create(b200z_ctx *ctx, const uint8_t *raw, size_t len, b200z_dict **out);
/* EXTENSION (not in the reference, SURVEY.md 8c gap): raw-content dictionary = content only, offset history
 * [1,4,8], no entropy tables.  Frames compressed against it carry no dict id; select it with force_dict /
 * the `forced_dict` argument. */
int b200z_dict_create_raw_content(b200z_ctx *ctx, uint32_t id, const uint8_t *content, size_t len, b200z_dict **out);
uint32_t b200z_dict_id(const b200z_dict *d);
int b200z_dict_offset_history(const b200z_dict *d, uint32_t out[3]);
size_t b200z_dict_content_size(const b200z_dict *d);
void b200z_dict_destroy(b200z_dict *d);

/* ------------------------------------------------------------------------------------------------------------
 * Tier 1 -- batch entry: many independent frames in one submission (the throughput path; frames shard
 * across GPUs by giving each rank's ctx its own sub-list).  For each frame this does what
 *   FrameDecoder::reset + [force_dict] + decode_blocks(BlockDecodingStrategy::All) + read
 * does in the reference (tests/decode_corpus.rs:76-100), for all frames at once.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct b200z_frame_io {
    uint64_t src_off;  /* byte offset of the frame (magic number first) inside `input`          */
    uint64_t src_size; /* bytes available for this frame (may exceed the frame; see bytes_read) */
    uint64_t out_off;  /* where this frame's plaintext goes inside `output`                     */
    uint64_t out_cap;  /* room reserved there; TargetTooSmall if the frame needs more           */
} b200z_frame_io;

typedef struct b200z_frame_result {
    uint64_t out_size;       /* plaintext bytes produced at out_off                                        */
    uint64_t bytes_read;     /* FrameDecoder::bytes_read_from_source (frame_decoder.rs:273)                */
    uint64_t content_size;   /* FrameDecoder::content_size (frame_decoder.rs:246)                          */
    uint64_t window_size;    /* FrameHeader::window_size (frame.rs:116)                                    */
    int32_t status;          /* 0 or b200z_error                                                           */
    int32_t stage;           /* b200z_stage of the error                                                   */
    uint32_t blocks_decoded; /* FrameDecoder::blocks_decoded (frame_decoder.rs:297)                        */
    uint32_t error_block;    /* index of the block that failed (when status != 0 in stages 2..6)           */
    uint32_t has_checksum;   /* frame carries a content checksum                                           */
    uint32_t checksum_from_data;  /* get_checksum_from_data (frame_decoder.rs:254)                         */
    uint32_t has_dict_id;
    uint32_t dict_id;        /* FrameHeader::dictionary_id (frame.rs:142)                                  */
    uint32_t has_calculated_checksum; /* 1 when the context ran the GPU checksum stage (B200Z_FLAG_CHECKSUM)   */
    uint32_t calculated_checksum;     /* get_calculated_checksum (frame_decoder.rs:262): XXH64(seed 0) low 32 bits */
} b200z_frame_result;

#define B200Z_MEM_HOST 0
#define B200Z_MEM_DEVICE 1

/* One-shot: plan on the host, copy in (if host memory), run the kernels, copy out (if host memory), fill
 * `results[nframes]`.  Returns 0 if the submission ran (per-frame outcome in results[i].status) or a
 * b200z_error for a submission-level failure.  `dicts`/`ndicts`: dictionaries selectable by frame dict id
 * (FrameDecoder::add_dict); `forced_dict`: applied to every frame after init (FrameDecoder::force_dict,
 * frame_decoder.rs:229) or NULL.  `max_window_size` 0 = the reference default 128 MiB (frame_decoder.rs:25). */
int b200z_decode_frames_batch(b200z_ctx *ctx, const uint8_t *input, size_t input_len, int input_mem,
                              const b200z_frame_io *frames, size_t nframes, const b200z_dict *const *dicts,
                              size_t ndicts, const b200z_dict *forced_dict, uint64_t max_window_size,
                              uint8_t *output, size_t output_cap, int output_mem, b200z_frame_result *results);

/* Split form of the same call, for device-resident pipelines and for timing the kernels alone:
 *   prepare: host plan (frame/block/section header walk) + upload of input and descriptors into HBM
 *   run:     ONLY kernel launches on the ctx stream (async), input/descriptors/tables/output all in HBM
 *   finish:  synchronise and fetch per-frame results */
typedef struct b200z_batch b200z_batch;
int b200z_batch_prepare(b200z_ctx *ctx, const uint8_t *input, size_t input_len, int input_mem,
                        const b200z_frame_io *frames, size_t nframes, const b200z_dict *const *dicts, size_t ndicts,
                        const b200z_dict *forced_dict, uint64_t max_window_size, b200z_batch **out);
int b200z_batch_run(b200z_batch *b, uint8_t *d_output, size_t output_cap);
int b200z_batch_finish(b200z_batch *b, b200z_frame_result *results);
/* b200z_batch_run with a CUDA event between kernels: synchronises and returns each kernel's device milliseconds
 * (stage_ms[i] for kernel b200z_stage_kernel_name(i), i < b200z_num_stages()).  Profiling aid for bench.py. */
int b200z_batch_run_profile(b200z_batch *b, uint8_t *d_output, size_t output_cap, float *stage_ms, size_t nstages);
/* one pass exactly as b200z_batch_run launches it, with events on the stream: out_ms[0..3] = completion time, relative to the
 * start of the pass, of k_setup, of k_huf, of the pair k_fse + k_exec (k_exec runs beside k_fse as its programmatic dependent)
 * and of k_exec_cta + the k_exec launch that takes what it handed back (n >= 4) */
int b200z_batch_run_timeline(b200z_batch *b, uint8_t *d_output, size_t output_cap, float *out_ms, size_t n);
int b200z_num_stages(void);
const char *b200z_stage_kernel_name(int stage);
/* facts about a prepared batch: [0] frames [1] blocks [2] compressed blocks [3] input bytes planned
 * [4] literal-scratch bytes [5] sequences [6] kernel launches per run */
int b200z_batch_info(const b200z_batch *b, uint64_t out[8]);
/* per-stage device pointers for kernel-level parity tests (tests/ only): literals scratch and sequence
 * scratch of the LAST run, laid out exactly as the oracle's trace (oracle/ruzstd_oracle.h zo_block_trace) */
int b200z_batch_debug_literals(b200z_batch *b, uint32_t block, uint8_t *host_out, size_t cap, size_t *len);
int b200z_batch_debug_sequences(b200z_batch *b, uint32_t block, uint32_t *host_out_ll_ml_of, size_t cap_seqs, size_t *nseq);
/* bit 0: the block's `of` column holds raw offset_values; otherwise offsets after do_offset_history
 * (sequence_execution.rs:59-118), symbolic where they depend on the repeat-offset history at the block's start:
 * tag << 30 | decrements, tag 1..3 = history slot + 1 */
int b200z_batch_debug_block_flags(b200z_batch *b, uint32_t block, uint32_t *flags);
/* execution scheduling counters of the last run (tests / profiling): [0] frames given to k_exec_cta (block assembled in
 * shared memory), [1] frames it handed back to k_exec (one warp per frame), [2] OR of the reasons, [3] blocks handed back */
int b200z_batch_debug_sched(b200z_batch *b, uint32_t out[4]);
/* Host-only views of a submission's scheduling decisions (no context, no device; for CPU tests of the host logic).
 * b200z_debug_route_frames: which frames k_exec_cta would take (largest first) given each frame's work (sequences + compressed
 * bytes / 16) and whether it is eligible (>= 2 blocks, >= 4096 compressed bytes, no dictionary); cta_frames has room for nframes.
 * b200z_debug_fse_order: the order in which k_fse takes the blocks (row by row across the warp kernel's frames, by decreasing
 * sequence count inside a row, k_exec_cta's frames last); *n_order = 0 means descriptor order; order has room for nblocks_total. */
int b200z_debug_route_frames(const uint64_t *work, const uint8_t *eligible, size_t nframes, uint32_t sms, uint32_t *cta_frames, size_t *n_cta);
int b200z_debug_fse_order(const uint32_t *first_block, const uint32_t *nblocks, const uint8_t *on_cta, size_t nframes, const uint32_t *nseq,
                          size_t nblocks_total, uint32_t *order, size_t *n_order);
void b200z_batch_destroy(b200z_batch *b);

/* ------------------------------------------------------------------------------------------------------------
 * Tier 1b -- block-level batch entry: the thin FFI for a host that keeps the reference's OWN frame / block /
 * section header parsing (frame.rs:6-85, block_decoder.rs:201-247, literals_section.rs:117-223,
 * sequence_section.rs:108-167) and ships compressed blocks.  It replaces the one call site of the hot path,
 * BlockDecoder::decompress_block (block_decoder.rs:97-197, called at :140-145 / :176-183), for many blocks of many
 * frames at once.  A descriptor carries what decompress_block has in hand when it calls decode_literals /
 * decode_sequences / execute_sequences.  The entropy tables are built on the GPU from the descriptions inside the
 * block content, so the "table pool" is implicit: Repeat / Treeless modes refer to the tables of the previous block
 * of the same frame (blocks of a frame are consecutive and in order), or to the frame's dictionary.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct b200z_block_desc {
    uint64_t src_off;             /* offset of the block CONTENT (after the 3-byte header) in `compressed`            */
    uint32_t content_size;        /* BlockHeader::content_size (block.rs:31-43)                                        */
    uint32_t block_type;          /* 0 Raw, 1 RLE, 2 Compressed                                                        */
    uint32_t decompressed_size;   /* BlockHeader::decompressed_size (Raw / RLE blocks)                                 */
    uint32_t last_block;
    /* what LiteralsSection::parse_from_header gave (literals_section.rs:9-28); checked against the content */
    uint32_t literals_type;       /* 0 Raw, 1 RLE, 2 Compressed, 3 Treeless                                            */
    uint32_t regenerated_size;
    uint32_t compressed_size;     /* 0 for Raw / RLE literals                                                          */
    uint32_t num_streams;         /* 1 or 4 (Compressed / Treeless), else 0                                            */
    /* what SequencesHeader::parse_from_header gave (sequence_section.rs:10-19) */
    uint32_t num_sequences;
    uint32_t modes;               /* the compression-modes byte (0 when num_sequences == 0)                            */
} b200z_block_desc;

typedef struct b200z_block_frame {
    uint64_t out_off;             /* where the frame's byte 0 goes inside `output`                                     */
    uint64_t out_cap;
    uint64_t window_size;         /* FrameHeader::window_size (frame.rs:116)                                           */
    const b200z_dict *dict;       /* dictionary in use (initial tables, offset history, content) or NULL               */
    uint32_t first_block;         /* index of the frame's first descriptor                                             */
    uint32_t num_blocks;
} b200z_block_frame;

typedef struct b200z_block_status {
    int32_t status;               /* 0, a b200z_error, or B200Z_BLOCK_NOT_REACHED (an earlier block of the frame failed) */
    int32_t stage;
    uint32_t out_size;            /* bytes this block added to the frame's output                                      */
    uint32_t reserved;
} b200z_block_status;
#define B200Z_BLOCK_NOT_REACHED (-1)

/* Decodes `nblocks` blocks of `nframes` frames.  `compressed` / `output` are host or device memory (B200Z_MEM_*).
 * Returns 0 when the submission ran; per-block outcomes in status[nblocks], per-frame totals in frame_out_size[nframes]
 * (either may be NULL).  B200Z_ERR_INVALID_ARGUMENT when a descriptor disagrees with the section headers found in the
 * block content. */
int b200z_decode_blocks_batch(b200z_ctx *ctx, const b200z_block_desc *blocks, size_t nblocks, const b200z_block_frame *frames,
                              size_t nframes, const uint8_t *compressed, size_t compressed_len, int compressed_mem, uint8_t *output,
                              size_t output_cap, int output_mem, b200z_block_status *status, uint64_t *frame_out_size);

/* ------------------------------------------------------------------------------------------------------------
 * Tier 2 -- mirror of ruzstd's FrameDecoder (decoding/frame_decoder.rs:154-627), GPU-backed.
 * Same names, argument meaning and error behaviour; `read_cb` has io::Read::read semantics.
 * ---------------------------------------------------------------------------------------------------------- */
typedef long (*b200z_read_fn)(void *user, uint8_t *buf, size_t len);        /* bytes read, 0 = EOF, <0 = error */
typedef long (*b200z_write_fn)(void *user, const uint8_t *buf, size_t len); /* bytes written, 0 = full, <0 = error */

/* BlockDecodingStrategy (frame_decoder.rs:96-100) */
#define B200Z_STRATEGY_ALL 0
#define B200Z_STRATEGY_UPTO_BLOCKS 1
#define B200Z_STRATEGY_UPTO_BYTES 2
#define B200Z_DEFAULT_MAX_WINDOW_SIZE (1024ull * 1024ull * 128ull) /* frame_decoder.rs:25 */

typedef struct b200z_frame_decoder b200z_frame_decoder;
int b200z_frame_decoder_new(b200z_ctx *ctx, b200z_frame_decoder **out);                    /* FrameDecoder::new :158 */
void b200z_frame_decoder_free(b200z_frame_decoder *d);
void b200z_frame_decoder_set_max_window_size(b200z_frame_decoder *d, uint64_t n);          /* :175 */
uint64_t b200z_frame_decoder_max_window_size(const b200z_frame_decoder *d);                /* :180 */
int b200z_frame_decoder_init(b200z_frame_decoder *d, b200z_read_fn read_cb, void *user);   /* init :190 */
int b200z_frame_decoder_reset(b200z_frame_decoder *d, b200z_read_fn read_cb, void *user);  /* reset :200 */
/* on B200Z_ERR_SKIP_FRAME from init/reset: the SkipFrame{length} payload (frame.rs:15-23) */
uint32_t b200z_frame_decoder_skip_frame_length(const b200z_frame_decoder *d);
int b200z_frame_decoder_add_dict(b200z_frame_decoder *d, const uint8_t *raw, size_t len);  /* decode_dict + add_dict :224 */
int b200z_frame_decoder_add_raw_content_dict(b200z_frame_decoder *d, uint32_t id, const uint8_t *content, size_t len); /* EXTENSION */
int b200z_frame_decoder_force_dict(b200z_frame_decoder *d, uint32_t dict_id);              /* :229 */
int b200z_frame_decoder_decode_blocks(b200z_frame_decoder *d, b200z_read_fn read_cb, void *user, int strategy,
                                      size_t n, int *finished);                            /* :309 */
long b200z_frame_decoder_read(b200z_frame_decoder *d, uint8_t *buf, size_t len);           /* impl Read :615 */
long b200z_frame_decoder_collect_to_writer(b200z_frame_decoder *d, b200z_write_fn write_cb, void *user); /* :393 */
size_t b200z_frame_decoder_can_collect(const b200z_frame_decoder *d);                      /* :409 */
int b200z_frame_decoder_is_finished(const b200z_frame_decoder *d);                         /* :284 */
size_t b200z_frame_decoder_blocks_decoded(const b200z_frame_decoder *d);                   /* :297 */
uint64_t b200z_frame_decoder_bytes_read_from_source(const b200z_frame_decoder *d);         /* :273 */
uint64_t b200z_frame_decoder_content_size(const b200z_frame_decoder *d);                   /* :246 */
int b200z_frame_decoder_get_checksum_from_data(const b200z_frame_decoder *d, uint32_t *out);  /* :254; 1 = Some */
int b200z_frame_decoder_get_calculated_checksum(const b200z_frame_decoder *d, uint32_t *out); /* :262; 1 = Some */
int b200z_frame_decoder_decode_from_to(b200z_frame_decoder *d, const uint8_t *src, size_t src_len, uint8_t *dst,
                                       size_t dst_len, size_t *read, size_t *written);     /* :439 */
int b200z_frame_decoder_decode_all(b200z_frame_decoder *d, const uint8_t *input, size_t input_len, uint8_t *output,
                                   size_t output_cap, size_t *written);                    /* :541 */
int b200z_frame_decoder_last_stage(const b200z_frame_decoder *d);
const char *b200z_frame_decoder_last_error_message(const b200z_frame_decoder *d);

/* ------------------------------------------------------------------------------------------------------------
 * Mirror of ruzstd's StreamingDecoder (decoding/streaming_decoder.rs:45-156): owns a source callback and a
 * frame decoder (its own, or a borrowed one = new_with_decoder).
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct b200z_streaming_decoder b200z_streaming_decoder;
int b200z_streaming_decoder_new(b200z_ctx *ctx, b200z_read_fn read_cb, void *user, b200z_streaming_decoder **out); /* :61 */
int b200z_streaming_decoder_new_with_decoder(b200z_read_fn read_cb, void *user, b200z_frame_decoder *dec,
                                             b200z_streaming_decoder **out);               /* :51 */
int b200z_streaming_decoder_new_with_max_window_size(b200z_ctx *ctx, b200z_read_fn read_cb, void *user,
                                                     uint64_t max_window_size, b200z_streaming_decoder **out); /* :72 */
long b200z_streaming_decoder_read(b200z_streaming_decoder *s, uint8_t *buf, size_t len, int *error); /* impl Read :118 */
b200z_frame_decoder *b200z_streaming_decoder_frame_decoder(b200z_streaming_decoder *s);    /* get at .decoder :46 */
/* into_frame_decoder :113 -- destroys the wrapper, returns the decoder (caller frees it unless it was borrowed) */
b200z_frame_decoder *b200z_streaming_decoder_into_frame_decoder(b200z_streaming_decoder *s);
void b200z_streaming_decoder_free(b200z_streaming_decoder *s);

/* ------------------------------------------------------------------------------------------------------------
 * Compression -- ruzstd's encoding module (encoding/mod.rs, frame_compressor.rs:131-224) on the GPU.  Every 128 KiB block of
 * every frame is compressed at once (the reference's Fastest matcher never looks outside the current block,
 * match_generator.rs:28-53).  Frames: magic, no dictionary, not single-segment, Window_Descriptor 128 KiB
 * (FrameHeader::serialize, frame_header.rs), blocks of at most 128 KiB, the last one empty when the input is a multiple of
 * 128 KiB (frame_compressor.rs:141-186).  A frame's bytes depend only on its plaintext, the level and the flags.
 * ---------------------------------------------------------------------------------------------------------- */
/* CompressionLevel (encoding/mod.rs:47-68) */
#define B200Z_LEVEL_UNCOMPRESSED 0   /* Raw blocks only: byte-identical to the reference                                  */
#define B200Z_LEVEL_FASTEST 1        /* RLE / Compressed / Raw per block, as levels/fastest.rs decides                    */
#define B200Z_LEVEL_DEFAULT 2        /* unimplemented!() in the reference (frame_compressor.rs:202-204):                 */
#define B200Z_LEVEL_BETTER 3         /*   -> B200Z_ERR_REFERENCE_WOULD_PANIC                                              */
#define B200Z_LEVEL_BEST 4
#define B200Z_COMPRESS_CHECKSUM 1u     /* Content_Checksum (the reference's default, feature "hash")                       */
#define B200Z_COMPRESS_CONTENT_SIZE 2u /* EXTENSION: write Frame_Content_Size (the reference writes none); the field is the
                                          smallest of 2 / 4 / 8 bytes that holds it (the 1-byte field needs Single_Segment) */

typedef struct b200z_compress_result {
    uint64_t out_size;       /* compressed bytes written at out_off                                               */
    int32_t status;          /* 0 or B200Z_ERR_TARGET_TOO_SMALL (out_cap, or the output buffer, is too short)    */
    int32_t stage;
    uint32_t num_blocks, raw_blocks, rle_blocks, compressed_blocks;
    uint32_t checksum;       /* low 32 bits of XXH64(seed 0) of the plaintext, written when flagged             */
    uint32_t reserved;
} b200z_compress_result;

/* largest frame b200z_compress_frames_batch writes for src_size bytes: header with Frame_Content_Size, 3 bytes per block,
 * the plaintext (every block Raw) and the checksum */
size_t b200z_compress_bound(size_t src_size);
/* Many independent frames: frames[i] = {src_off, src_size, out_off, out_cap} (src = plaintext inside `input`, out = where
 * the frame goes inside `output`); host or device memory on either side (B200Z_MEM_*).  Only results[i].out_size bytes at
 * each successful frame's out_off are written; the rest of `output` is left as it was.  Returns 0 when the submission ran
 * (per-frame outcome in results[i]), B200Z_ERR_REFERENCE_WOULD_PANIC for levels Default / Better / Best, or another
 * b200z_error for a submission-level failure.
 * Device memory: the whole submission is in flight at once, with a fixed worst-case scratch of about 570 KB per 128 KiB block
 * at the Fastest level (about 4.4 x the plaintext), plus a device copy of host input and of host output.  There is no
 * chunking: a submission that does not fit fails with B200Z_ERR_OUT_OF_MEMORY, and the caller splits it into several. */
int b200z_compress_frames_batch(b200z_ctx *ctx, const uint8_t *input, size_t input_len, int input_mem, const b200z_frame_io *frames,
                                size_t nframes, int level, uint32_t flags, uint8_t *output, size_t output_cap, int output_mem,
                                b200z_compress_result *results);
/* encoding::compress(source, target, level) (mod.rs:24-30): reads `read_cb` to EOF, writes one frame to `write_cb`
 * (one submission: the device-memory limit above applies to the whole stream) */
int b200z_compress(b200z_ctx *ctx, b200z_read_fn read_cb, void *ruser, b200z_write_fn write_cb, void *wuser, int level, uint32_t flags);

/* XXH64(seed 0) of a host buffer -- the content-checksum hash the reference feeds on drain
 * (decode_buffer.rs:42,225,290,301); exposed so bindings can verify checksums like tests/decode_corpus.rs:61-74 */
uint64_t b200z_xxh64(const uint8_t *data, size_t len);

#ifdef __cplusplus
}
#endif
#endif /* B200ZSTD_H */
