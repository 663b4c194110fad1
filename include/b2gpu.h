/* b2gpu.h — C ABI of the B200-native BZip2 block encoder that stands behind Zip-Ada's
 * `BZip2.Encoding.Encode` (reference: zip_lib/bzip2-encoding.ads:38-56).
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types.  The Ada body of
 * `BZip2.Encoding` binds these entry points with `pragma Import (C, ...)` over Interfaces.C
 * (the binding is shown in INTEGRATION.md and zip-ada_b200/ada/bzip2-encoding.adb); the C++ and
 * Python hosts in this repository use the same symbols.
 *
 * Every function returns 0 on success and a non-zero B2_ERR_* otherwise; b2_last_error() gives a
 * human-readable message for the calling thread.  There is NO CPU fallback: if no CUDA device is
 * usable, b2_create fails.
 *
 * Threading: one host thread per handle at a time; handles are independent (no global mutable
 * state), matching the reference's "can be used ad libitum in parallel processing"
 * (doc/zipada.txt:26).
 */
#ifndef B2GPU_H
#define B2GPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Only the entry points below are exported by libb2gpu.so. */
#if defined(__GNUC__)
#define B2_API __attribute__((visibility("default")))
#else
#define B2_API
#endif

#define B2_OK 0
#define B2_ERR_ARGUMENT 1
#define B2_ERR_OUTPUT_TOO_SMALL 2
#define B2_ERR_ALLOC 3
#define B2_ERR_CUDA 10
#define B2_ERR_INTERNAL 11
#define B2_ERR_ABORTED 12          /* the progress callback asked to stop: Zip.User_abort (zip-compress.ads:149) */
#define B2_ERR_DUPLICATE_NAME 20   /* Zip.Create.Duplicate_name (zip-create.ads, zip-create.adb:138-147) */

/* Compression_Option (bzip2-encoding.ads:40-43): block_100k / block_400k / block_900k.
 * Zip.Compress.BZip2_E maps BZip2_1/2/3 to them (zip-compress-bzip2_e.adb:122-126). */
#define B2_BLOCK_100K 1
#define B2_BLOCK_400K 4
#define B2_BLOCK_900K 9

/* Stream_Size_Type / unknown_size (bzip2-encoding.ads:45-47). */
#define B2_UNKNOWN_SIZE (-1)

typedef struct b2_encoder b2_encoder;

/* Creates an encoder bound to CUDA device `device` (0-based).  `level` is one of B2_BLOCK_*.
 * Replaces: the per-call heap allocations of Encode (bzip2-encoding.adb:162, :263, :272, :372,
 * :1157) — the handle owns all device workspaces and reuses them across calls. */
B2_API int b2_create(int level, int device, b2_encoder **out);

/* Releases everything the handle owns.  Mirrors the exception-path clean-up of
 * bzip2-encoding.adb:1128-1133, :1351-1357, :1377-1381: the Ada body calls it from a handler. */
B2_API void b2_destroy(b2_encoder *enc);

/* Upper bound of the encoded size for `n` input bytes (for sizing `out`). */
B2_API uint64_t b2_bound(uint64_t n);

/* Whole-stream encode, host buffers: produces exactly the bytes that
 * `Encode (option, size_hint)` sends through Write_Byte for the bytes that Read_Byte/More_Bytes
 * deliver (bzip2-encoding.adb:1413-1431): "BZh<level>", blocks, footer.
 * `size_hint` is the reference's size_hint (B2_UNKNOWN_SIZE = -1): it changes the cutting of the
 * last two chunks (bzip2-encoding.adb:1416-1424).  Copies in -> device and device -> out. */
B2_API int b2_encode_stream(b2_encoder *enc, const uint8_t *in, uint64_t n, int64_t size_hint,
                     uint8_t *out, uint64_t out_cap, uint64_t *out_len);

/* Same, with input and output already in device memory of the handle's device (no PCIe traffic;
 * used to measure the kernels alone).  `d_in` needs 64 readable bytes of slack after `n`;
 * `d_out` must be 4-byte aligned. */
B2_API int b2_encode_stream_device(b2_encoder *enc, const uint8_t *d_in, uint64_t n, int64_t size_hint,
                            uint8_t *d_out, uint64_t out_cap, uint64_t *out_len);

/* Many independent streams in one call (archive entries: every entry of a Zip archive written with
 * BZip2_1..3 is its own stream; Zip.Create.Add_Stream calls Compress_Data once per entry,
 * zip-create.adb:253-265, which is serial per entry).  Entry i is the `sizes[i]` bytes at
 * `in + in_offsets[i]`, encoded exactly as `Encode (option, size_hints[i])` would (size_hints may be
 * NULL = unknown_size for all).  The streams are written back to back, each 8-byte aligned, into
 * `out`; out_offsets[i] / out_lens[i] locate stream i.  Chunks of all entries share the device
 * batches, so 100 000 small entries are as efficient as one large stream. */
B2_API int b2_encode_batch(b2_encoder *enc, uint32_t n_entries, const uint8_t *in, const uint64_t *in_offsets,
                    const uint64_t *sizes, const int64_t *size_hints, uint8_t *out, uint64_t out_cap,
                    uint64_t *out_offsets, uint64_t *out_lens);

/* ---- One stream over several devices (SURVEY.md 8e; north star: "the input stream is sharded block-wise
 * across the 8 GPUs of one box with per-device streams and pinned host buffers, no collective") -------------
 * The reference's own parallelism is four tasks sharing one chunk (bzip2-encoding.adb:1226-1303); chunks
 * themselves are independent once their start is known.  A stream is split into contiguous byte ranges, one
 * per shard (handle = device); a shard owns the chunks that START in its range.  What crosses shards is
 * scalars only:
 *   - the cutting is a chain (Data_Acquisition, :1160-1208): shard r learns where its first chunk starts from
 *     shard r-1 (`entry` / `handoff`);
 *   - the winner of a chunk depends on the incoming bit offset mod 8 (:1319-1325) and the combined CRC is
 *     folded block by block (:990): each shard reports, for each of the 8 possible incoming offsets, the bits
 *     it appends and its CRC fold (b2_shard_link); b2_shard_resolve composes them in shard order.
 * Call order per shard: b2_shard_open (upload + scans, asynchronous) -> b2_shard_cut (needs the previous
 * shard's handoff) -> b2_shard_encode -> [exchange links, b2_shard_resolve] -> b2_shard_finish.
 * b2_encode_stream_multi does all of it for the handles of one process (one host thread per handle); under
 * one-process-per-GPU launchers the two exchanges are a point-to-point send of 8 bytes and an all-gather of
 * 128 bytes per rank (bench.py). */
typedef struct b2_shard_link {
  uint64_t total_bits[8];   /* bits appended when the shard's first chunk starts at bit offset k mod 8 */
  uint32_t crc_rot[8];      /* combined CRC: crc_out = rotl (crc_in, crc_rot[k]) xor crc_fold[k] */
  uint32_t crc_fold[8];
} b2_shard_link;

/* Bytes a shard needs beyond the end of its range (a chunk is at most 10 x capacity raw bytes, :1156). */
B2_API uint64_t b2_shard_margin(int level);
/* Range bounds[r] .. bounds[r+1] of every shard (bounds has n_shards + 1 entries, 4096-byte aligned inside).
 * Later shards start later (the cutting is serial), so their shares shrink by stagger_permille / 1000 per shard
 * (-1: default / env B2GPU_SHARD_STAGGER). */
B2_API int b2_shard_plan(uint64_t n, int n_shards, int level, int stagger_permille, uint64_t *bounds);
/* `in` (host, or device memory of the handle's device) holds the stream bytes [base, base + n_local): from
 * the start of the shard's range to min (stream_size, own_end + b2_shard_margin).  own_end = bounds[r + 1]. */
B2_API int b2_shard_open(b2_encoder *enc, const uint8_t *in, int in_is_device, uint64_t base, uint64_t n_local,
                         uint64_t stream_size, int64_t size_hint, uint64_t own_end);
/* entry: stream offset where this shard's first chunk starts (0 for the first shard; the previous shard's
 * handoff otherwise).  handoff: where the next shard's first chunk starts. */
B2_API int b2_shard_cut(b2_encoder *enc, uint64_t entry, uint64_t *handoff);
B2_API int b2_shard_encode(b2_encoder *enc, b2_shard_link *link);
/* bit_offsets[r] = bit offset in the stream of shard r's first block (bit_offsets[0] = 32, behind "BZh9"),
 * crcs[r] = combined CRC before it; both arrays have n_shards + 1 entries; the stream has
 * (bit_offsets[n_shards] + 80 + 7) / 8 bytes. */
B2_API int b2_shard_resolve(const b2_shard_link *links, int n_shards, uint64_t *bit_offsets, uint32_t *crcs);
/* Writes the shard's piece of the stream to `out`: stream bytes [*out_byte_offset, + *out_len).  The first and
 * the last byte may be shared with the neighbouring pieces (each piece holds only its own bits there: OR them);
 * their values are also returned separately.  The first shard writes the stream header, the last the footer. */
B2_API int b2_shard_finish(b2_encoder *enc, uint64_t bit_offset, uint32_t crc_in, uint8_t *out, int out_is_device,
                           uint64_t out_cap, uint64_t *out_byte_offset, uint64_t *out_len, uint8_t *first_byte,
                           uint8_t *last_byte);
/* Encode (option, size_hint) of one stream on the devices of `encs` (host buffers; pinned memory makes the
 * copies asynchronous).  Byte-identical to b2_encode_stream on one handle. */
B2_API int b2_encode_stream_multi(b2_encoder **encs, int n_encs, const uint8_t *in, uint64_t n, int64_t size_hint,
                                  uint8_t *out, uint64_t out_cap, uint64_t *out_len);

/* ---- One stream fed in pieces (the streaming shape of Encode: Read_Byte / More_Bytes / Write_Byte) ------------
 * Incremental Encode (option, size_hint): input in pieces, finished output in pieces.
 * The concatenation of every out of b2_stream_write and b2_stream_end is byte-identical to what
 * b2_encode_stream gives for the concatenated input and the same size_hint.
 *   - One open stream per handle.  While it is open, every other call that uses the handle's device buffers
 *     (encode, batch, zip, shard, verify, zip_crc32, dbg) returns B2_ERR_ARGUMENT; b2_stream_*, b2_set_*,
 *     b2_get_*, b2_reset_stats and b2_destroy are allowed.
 *   - The handle holds the bytes not yet encoded on the device, from the start of the next chunk.  When
 *     window_bytes + b2_shard_margin (level) of them are held, it encodes the chunks that start in the first
 *     window_bytes (a shard of the stream whose bit offset and CRC are known) and keeps the rest.  Device input
 *     memory is at most 2 x (window_bytes + b2_shard_margin + 256) bytes, whatever the stream length and write sizes.
 *     window_bytes: 0 = 512 MiB; below 1 MiB is B2_ERR_ARGUMENT.
 *   - `in` is host memory (pinned memory lets the upload run under the encode of the window before); the caller
 *     may reuse it as soon as the write returns.  `out` receives every byte that is final; the last partial byte
 *     is held back until the next window's bits or the footer complete it.
 *   - out_cap < b2_stream_bound (enc, n) returns B2_ERR_OUTPUT_TOO_SMALL before any input is taken: the stream is
 *     unchanged and the call can be repeated.  Any other error, B2_ERR_ABORTED included, closes the stream; the
 *     handle stays usable.
 *   - b2_set_progress fires after every device batch with the stream bytes encoded so far and size_hint (or, when
 *     it is unknown, that plus the bytes held); a non-zero return ends the write with B2_ERR_ABORTED.
 *   - b2_stats counts one stream; b2_get_trace after b2_stream_end gives every chunk with stream offsets. */
B2_API int b2_stream_begin(b2_encoder *enc, int64_t size_hint, uint64_t window_bytes);
/* An out_cap that always suffices for a write of n bytes (b2_stream_end: n = 0) in the stream's current state. */
B2_API uint64_t b2_stream_bound(b2_encoder *enc, uint64_t n);
B2_API int b2_stream_write(b2_encoder *enc, const uint8_t *in, uint64_t n,
                           uint8_t *out, uint64_t out_cap, uint64_t *out_len);
/* Encodes what is held as the last window and writes the footer ("BZh<level>" and the footer alone for an empty
 * stream); closes the stream. */
B2_API int b2_stream_end(b2_encoder *enc, uint8_t *out, uint64_t out_cap, uint64_t *out_len);
/* Closes the open stream, if any, discarding what it holds. */
B2_API int b2_stream_abort(b2_encoder *enc);

/* ---- Archive side: batched Zip.Create for BZip2 entries ------------------------------------------
 * One call = Create_Archive, Add_Stream for every entry, Finish (zip-create.adb:194-297, :645-756)
 * with Compress_Method = BZip2_1/2/3 (the level of `enc`), no password.  The bytes written to `out`
 * are the archive the reference leaves in its output Zipstream:
 *   per entry  local header PK\3\4 (zip-headers.adb:243-277) with needed_extract_version 10, the
 *              entry name with '\\' turned into '/' (Unixify, zip-create.adb:180-192), the short Zip64
 *              extension when the size or the offset needs it (:233-251, :279-292), then the payload:
 *              the BZip2 stream of the entry (method 12, size_hint = size), or the bytes themselves
 *              (method 0) when the stream is not smaller than the input (Compression_inefficient,
 *              zip-compress.adb:468-490 -> Store, :224-237);
 *   then       central headers PK\1\2 (made_by_version 23, zip-create.adb:122-131,
 *              zip-headers.adb:167-192), Zip64 end record + locator when needed (:727-749), end
 *              record PK\5\6.
 * The Zip CRC-32 of every entry (zip-crc_crypto.adb:31-61; the reference updates it per byte in the
 * Read_Byte callback, zip-compress-bzip2_e.adb:70-98) is computed on the device.
 * names: all entry names back to back; name i = names[name_offsets[i] .. name_offsets[i+1]).
 * dos_times: Zip_Streams.Time values as stored in the headers (NULL = Zip_Streams.default_time).
 * flags: B2_ZIP_* bits per entry (NULL = 0).  duplicates: Duplicate_name_policy.
 * info (may be NULL) receives crc, final method (Final_Method), compressed size (Compressed_Size)
 * and header offset of every entry.  Encryption, comments and Preselection are outside this path. */
#define B2_ZIP_UNICODE_NAME 1u        /* Zip_Streams.Is_Unicode_Name -> Language_Encoding_Flag_Bit */
#define B2_ZIP_READ_ONLY 2u           /* Stream.Is_Read_Only -> external_attributes bit 0 */
#define B2_ZIP_ADMIT_DUPLICATES 0
#define B2_ZIP_ERROR_ON_DUPLICATE 1
typedef struct b2_zip_entry_info {
  uint32_t crc32;
  uint16_t zip_type;                  /* 12 = bzip2_code, 0 = store_code */
  uint16_t reserved;
  uint64_t compressed_size;
  uint64_t local_header_offset;
} b2_zip_entry_info;
B2_API uint64_t b2_zip_bound(uint32_t n_entries, uint64_t total_name_bytes, uint64_t total_input_bytes);
B2_API int b2_zip_create(b2_encoder *enc, uint32_t n_entries, const uint8_t *in, const uint64_t *in_offsets,
                  const uint64_t *sizes, const char *names, const uint32_t *name_offsets,
                  const uint32_t *dos_times, const uint32_t *flags, int duplicates,
                  uint8_t *out, uint64_t out_cap, uint64_t *out_len, b2_zip_entry_info *info);

/* Zip CRC-32 of a host buffer, computed on the device (zip-crc_crypto.adb:31-61: Init, Update, Final). */
B2_API int b2_zip_crc32(b2_encoder *enc, const uint8_t *in, uint64_t n, uint32_t *crc);

/* ---- Decode / verify on the device (SURVEY.md 8f row 4) ---------------------------------------------------
 * The reference decodes a method-12 entry with BZip2.Decoding.Decompress (bzip2-decoding.adb:34-640, hooked at
 * unzip-decompress.adb:1898-1915), one block after the other, checking every block CRC and the combined CRC.
 * b2_verify_stream decodes ALL blocks of a stream at the same time (the block starts are found by their 48-bit
 * magic at any bit offset and validated by following the chain of block ends), checks the same CRCs and,
 * when `expect` is given, compares the decoded bytes with it.  Accepts any BZip2 stream without randomised
 * blocks (e.g. libbz2's), not only this encoder's. */
typedef struct b2_verify_result {
  uint64_t blocks;               /* blocks decoded on the chain from the header to the footer */
  uint64_t decoded_bytes;
  uint64_t mismatch_at;          /* first decoded byte that differs from `expect` (or a length difference); ~0 = none */
  uint64_t candidates;           /* occurrences of the block / footer magics in the stream (>= blocks + 1) */
  uint32_t level;                /* '1'..'9' of the stream header */
  uint32_t stored_stream_crc, computed_stream_crc;
  int32_t ok;                    /* 1: header, every block CRC, the combined CRC, the end of the stream and `expect` all agree */
  int32_t first_bad_block;       /* index of the first block that failed, -1 = none */
  uint32_t first_bad_status;     /* 1 bad header; 2 randomised block; 3-13 malformed block; 20 no block where one must start;
                                    21 bytes behind the footer; 22 no footer; 30 block CRC mismatch */
  double ms;                     /* CUDA-event time of the call */
} b2_verify_result;
B2_API int b2_verify_stream(b2_encoder *enc, const uint8_t *stream, int stream_is_device, uint64_t n,
                            const uint8_t *expect, int expect_is_device, uint64_t expect_n, b2_verify_result *result);

/* Feedback and abort (zip.ads:301-306 Feedback_Proc; zip-compress-bzip2_e.adb:78-96 fires it from Read_Byte and
 * raises User_abort).  The batched calls read no bytes through callbacks, so the hook moves here: `fn` is called
 * on the CALLING thread (never from a library thread) after every device batch of b2_encode_stream* /
 * b2_encode_batch / b2_zip_create with the uncompressed bytes done so far and the total; a non-zero result
 * stops the remaining batches and the call returns B2_ERR_ABORTED (the Ada body raises User_abort).  NULL = off. */
typedef int (*b2_progress_fn)(void *user, uint64_t done_bytes, uint64_t total_bytes);
B2_API int b2_set_progress(b2_encoder *enc, b2_progress_fn fn, void *user);

/* Last error message of the calling thread (never NULL). */
B2_API const char *b2_last_error(void);

/* ---------------------------------------------------------------------------------------------
 * Measurement taps (bench.py).  Times are CUDA-event times on the handle's stream. */
typedef struct b2_stats {
  uint64_t streams;              /* b2_encode_stream* calls since the last reset */
  uint64_t input_bytes;
  uint64_t chunks;               /* Read_and_Split_Block calls (bzip2-encoding.adb:1144) */
  uint64_t blocks;               /* Encode_Block calls after de-duplication (:148) */
  uint64_t block_bytes;          /* post-RLE1 bytes sorted (sum of N over blocks) */
  uint64_t kernel_launches;      /* kernels launched */
  uint64_t sort_rounds;          /* doubling rounds, summed over batches */
  uint64_t sort_elems_round0;    /* suffixes entering round 0 */
  uint64_t sort_elems_later;     /* sum over later rounds of suffixes re-sorted */
  uint64_t scatter_launches;     /* radix scatter launches */
  uint64_t scatter_elems;        /* elements moved by them */
  double scatter_ms;             /* their summed duration (only with b2_set_timing(enc, 1)) */
  double stage_ms[8];            /* cut+segment, rle1, sort, mtf, entropy, pack, concat, copies (timing level 2) */
  double call_ms;                /* CUDA-event time of the encode calls, first to last operation on the stream (timing >= 1) */
  double sort_ms;                /* CUDA-event time of the BWT sort stage (all its kernels), summed over batches (timing >= 1) */
} b2_stats;

/* level 0: off; 1: events around every encode call and every radix scatter launch (no extra
 * synchronisation); 2: also per-stage timers (adds stream synchronisations, diagnostic only). */
B2_API int b2_set_timing(b2_encoder *enc, int level);
B2_API int b2_get_stats(b2_encoder *enc, b2_stats *out);
B2_API int b2_reset_stats(b2_encoder *enc);

/* ---------------------------------------------------------------------------------------------
 * Parity taps (tests only): the intermediates the reference prints at verbosity `detailed` /
 * `super_detailed` (bzip2-encoding.adb:109-140, :205-209, :282-289, :337, :956-960). */
typedef struct b2_block_info {
  uint32_t n_rle, origin, crc, n_mtf, eob, n_used, n_sel, ec_count, max_len, sample_width, cost, pad;
  uint64_t bits;
} b2_block_info;

/* One Encode_Block (bzip2-encoding.adb:148) on the device.  Any output pointer may be NULL.
 * rle_out/bwt_out: >= len*5/4+64 bytes; mtf_out: >= len*5/4+64 uint16; sel_out: >= 18002;
 * lens_out: 6*258 bytes; bits_out: the block's bitstream from bit 0. */
B2_API int b2_dbg_block(b2_encoder *enc, const uint8_t *raw, uint32_t len,
                 uint8_t *rle_out, uint8_t *bwt_out, uint16_t *mtf_out, uint8_t *sel_out,
                 uint8_t *lens_out, uint8_t *bits_out, uint64_t bits_cap, b2_block_info *info);

typedef struct b2_chunk_trace {
  uint64_t start;
  uint32_t len, dyn_capacity;
  int32_t winner;                /* 0 single, 1 parts_4, 2 segmented_1, 3 segmented_2 (:1217) */
  uint32_t n_seg1, n_seg2, pad;
  uint64_t bytes[4];             /* destination_index of each tactic (:1319-1325) */
  uint64_t bits[4];
} b2_chunk_trace;

/* Trace of the last b2_encode_stream* call: one record per chunk. */
B2_API int b2_get_trace(b2_encoder *enc, b2_chunk_trace *out, uint64_t cap, uint64_t *n);

/* Segment_by_Entropy cut list of one chunk of the last call (profile 0 = segmented_1, 1 = segmented_2). */
B2_API int b2_get_segments(b2_encoder *enc, uint64_t chunk, int profile, uint32_t *cuts, uint32_t cap, uint32_t *n);

#ifdef __cplusplus
}
#endif
#endif
