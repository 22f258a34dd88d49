/*
 * b200z.h -- C ABI of libb200z.so: B200 (sm_100a) DEFLATE / BZip2 block codecs behind the
 * Dart `archive` package's codec classes.
 *
 * The reference (brendan-duncan/archive 4.2.0) is pure Dart and has no FFI of its own; the
 * entry points below are what a `dart:ffi` binding for its codec hot path binds (see
 * INTEGRATION.md and dart/lib/src/b200z_ffi.dart).  Each entry point cites the reference
 * interface it replaces (paths relative to /root/reference/).
 *
 * Conventions
 *   - plain pointers + sizes, no C++ / torch types; every call is blocking.
 *   - one process drives ONE GPU (b200z_init(device)); multi-GPU = one process per GPU,
 *     units sharded by the caller (bench.py / torchrun), see DESIGN.md "Multi-GPU".
 *   - return value: 0 (B200Z_OK) or a negative B200Z_E_* code.  The reference's error
 *     convention on this path is "stop, keep partial output, never throw"
 *     (inflate.dart:150-151,166-168; bzip2_decoder.dart:32-78): data errors therefore still
 *     produce the partial output the reference would have produced, and the per-stream
 *     status says why decoding stopped.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     B200Z_E_NODEVICE.
 */
#ifndef B200Z_H
#define B200Z_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes -------------------------------------------------------------------- */
#define B200Z_OK 0
#define B200Z_E_NODEVICE (-1) /* no CUDA device / b200z_init not called / CUDA runtime error   */
#define B200Z_E_ARG (-2)      /* invalid argument (Deflate._init returning false, deflate.dart:107-118) */
#define B200Z_E_NOSPC (-3)    /* out_cap too small; *out_len = bytes needed when known          */
#define B200Z_E_DATA (-4)     /* decodeStream() returned false (bad header / adler / crc)       */
#define B200Z_E_THROW (-5)    /* the Dart code would have thrown (RangeError: distance > output,
                                 output_memory_stream.dart:83-86; code-length overrun inflate.dart:359) */
#define B200Z_E_INTERNAL (-6)

/* per-unit status written by the batch decoders (int32) */
#define B200Z_U_DONE 0       /* BFINAL block decoded (inflate.dart:155)                          */
#define B200Z_U_EOS 1        /* input exhausted before a final block (inflate.dart:111 loop end)  */
#define B200Z_U_STOP (-1)    /* _parseBlock returned false: bad block type / code / short read    */
#define B200Z_U_NOSPC (-2)   /* unit output would exceed out_cap                                  */
#define B200Z_U_RANGE (-3)   /* back-reference before start of output (Dart RangeError)           */
#define B200Z_U_BADCODE (-4) /* over-subscribed or unusable Huffman code set (reference would
                                decode garbage / never terminate; see DESIGN.md "Divergences")    */
#define B200Z_U_THROW (-5)   /* code-length run overruns HLIT+HDIST (Dart RangeError)             */
#define B200Z_U_TOKCAP (-6)  /* internal token buffer too small (library retries)                 */

/* ---- lifetime ------------------------------------------------------------------------ */
int b200z_init(int device, uint32_t flags); /* selects the GPU for this process; idempotent  */
void b200z_shutdown(void);
const char *b200z_last_error(void); /* thread-local, never NULL                      */
int b200z_device_count(void);       /* 0 when no CUDA device is visible              */
const char *b200z_version(void);

/* pinned host memory for callers that want full-speed PCIe copies (Dart: Pointer<Uint8>) */
void *b200z_host_alloc(size_t bytes);
void b200z_host_free(void *p);

/* ---- single stream, reference class semantics ---------------------------------------- */
/* Inflate(bytes).getBytes()  -- inflate.dart:23-28,102.  Raw DEFLATE.  *in_consumed is where
 * the reference leaves the input stream (inflate.dart:337-340).  *unit_status = B200Z_U_*.  */
int b200z_inflate_raw(const uint8_t *in, size_t in_len, uint8_t *out, size_t out_cap,
                      size_t *out_len, size_t *in_consumed, int32_t *unit_status);

/* GZipDecoderWeb().decodeBytes -- _gzip_decoder_web.dart:19-58 (member loop, header skip,
 * CRC/ISIZE read and ignored, zlib fallback when there is no gzip header).  The members share
 * one output stream, as in the reference (:38): a member's back-references may reach into the
 * members decoded before it.  A stream that ends inside a block: B200Z_E_THROW (the reference's
 * trailer read runs past the end), with the bytes decoded so far in `out`.                  */
#define B200Z_GZIP_VERIFY 1 /* bits of `verify`: verify, and the `raw` the reference hands on to the zlib decoder when */
#define B200Z_GZIP_RAW 2    /* the input has no gzip header (_gzip_decoder_web.dart:31-37)                            */
int b200z_gzip_decode(const uint8_t *in, size_t in_len, int verify, uint8_t *out, size_t out_cap,
                      size_t *out_len);
/* ZLibDecoderWeb().decodeBytes -- _zlib_decoder_web.dart:21-107 (stream loop, Adler-32 when
 * verify, raw = no wrapper).  Every stream has an output of its own and reaches `out` only once
 * the next stream's header has been accepted, or at the end (:82-84, :101-103).            */
int b200z_zlib_decode(const uint8_t *in, size_t in_len, int verify, int raw, uint8_t *out,
                      size_t out_cap, size_t *out_len);
/* Upper bound for the output of b200z_gzip_decode / b200z_zlib_decode, from the framing's own
 * size fields where present (ISIZE), else 0 = unknown (call with a guess, retry on E_NOSPC). */
size_t b200z_gzip_bound(const uint8_t *in, size_t in_len);

/* Deflate(bytes, level:, windowBits:).getBytes() and .crc32 -- deflate.dart:39-48,72-75,31.  Raw DEFLATE, byte-identical
 * to the reference at the same level and windowBits (9..15).  Levels 4-9 are data parallel inside a stream; 1-3
 * (deflate_fast, whose hash chains depend on the parse) are one warp per stream with all state in shared memory -- their
 * parallel axis is the batch (b200z_deflate_batch); 0 is stored.  Invalid level / windowBits
 * (Deflate._init returning false, :107-118) -> B200Z_E_ARG.                                                          */
int b200z_deflate_raw(const uint8_t *in, size_t in_len, int level, int window_bits, uint8_t *out, size_t out_cap,
                      size_t *out_len, uint32_t *crc32_of_input);
size_t b200z_deflate_bound(size_t in_len); /* output capacity that always suffices (+18 for gzip, +6 for zlib) */
/* n_units independent Deflate(bytes, level:, windowBits:) streams in one call -- what ZipEncoder does member by member
 * (zip_encoder.dart:185-259, platformZLibEncoder.encodeStream(raw: true) :244-249).  Unit u reads
 * in_base[in_off[u] .. +in_len[u]) and writes out_base[out_off[u] .. +out_cap[u]); out_len[u] = its compressed size,
 * crc32[u] (may be NULL) = CRC-32 of its input, status[u] = B200Z_OK or B200Z_U_NOSPC (out_len[u] = bytes needed).  All
 * inputs are staged at once and up to 8 members (B200Z_DEFLATE_LANES) are in flight on separate CUDA streams; at levels
 * 1-3 the match finding of ALL members runs first, as one launch with a warp per member.  Every stream is byte-identical
 * to b200z_deflate_raw of the same input.                                                                            */
int b200z_deflate_batch(const uint8_t *in_base, const uint64_t *in_off, const uint64_t *in_len, size_t n_units, int level,
                        int window_bits, uint8_t *out_base, const uint64_t *out_off, const uint64_t *out_cap,
                        uint64_t *out_len, uint32_t *crc32, int32_t *status);
/* ZLibEncoderWeb().encodeBytes -- _zlib_encoder_web.dart:17-73 (header 78 01 at every level, Adler-32 trailer)      */
int b200z_zlib_encode(const uint8_t *in, size_t in_len, int level, int window_bits, int raw, uint8_t *out,
                      size_t out_cap, size_t *out_len);
/* GZipEncoderWeb().encodeBytes -- _gzip_encoder_web.dart:17-100 (MTIME is "now" in the reference: a parameter here) */
int b200z_gzip_encode(const uint8_t *in, size_t in_len, int level, uint32_t mtime, uint8_t *out, size_t out_cap,
                      size_t *out_len);

/* BZip2Decoder().decodeBytes(data, verify:) -- bzip2_decoder.dart:13-88.  Stops after the first end-of-stream
 * block; CRCs are compared only when verify; B200Z_E_DATA == decodeStream returning false (the blocks decoded
 * before the failure are kept, as in the reference).                                                    */
int b200z_bzip2_decode(const uint8_t *in, size_t in_len, int verify, uint8_t *out, size_t out_cap,
                       size_t *out_len);
/* One rank's share of a BZip2 stream (SURVEY.md 8e: blocks are independent once the bit-level magic scan has found
 * them; only the combined CRC and the output offsets chain across blocks).  Rank `rank` of `world` decodes the block
 * candidates [n*rank/world, n*(rank+1)/world) into `out`, back to back, and reports EVERY candidate of its share plus
 * the end-of-stream candidates: the caller merges the reports of all ranks, walks the chain as decodeStream does
 * (bzip2_decoder.dart:46-87: a block must start where the previous one ended), checks the CRCs and derives the output
 * offsets (archive_b200/shard.py: bzip2_decode_sharded).                                                         */
typedef struct {
  uint64_t start_bit, end_bit; /* position of the 48-bit magic; first bit after the block's last symbol */
  uint64_t out_bytes;          /* decoded size (0 when the block could not be decoded)                  */
  uint32_t crc_calc, crc_stored;
  int32_t status;              /* 0 ok, -1 data error, -2 read past the end of the input               */
  uint32_t flags;              /* B200Z_BZ2_*                                                           */
} b200z_bz2_block;
#define B200Z_BZ2_EOS 1u            /* an end-of-stream magic (crc_stored = the combined CRC) */
#define B200Z_BZ2_RANDOMISED 2u     /* (unused: randomised blocks are decoded)                */
#define B200Z_BZ2_CORRUPT_CYCLE 4u  /* inverse BWT is not one cycle: not decoded              */
#define B200Z_BZ2_OVERRUN 8u        /* the run-length walk overran the block (bzip2_decoder.dart:497-499, 628-631):
                                     * its bytes ARE written, then decodeStream returns false */
int b200z_bzip2_decode_shard(const uint8_t *in, size_t in_len, uint32_t rank, uint32_t world, uint8_t *out,
                             size_t out_cap, size_t *out_len, b200z_bz2_block *blocks, size_t blocks_cap,
                             size_t *n_blocks);
/* BZip2Encoder().encodeBytes(data) -- bzip2_encoder.dart:15-81: always "BZh9", never randomised, the pending RLE1
 * run is closed at every block end (which is where the bytes differ from libbzip2 on multi-block inputs).
 * Inputs of 4 GiB and more: B200Z_E_ARG.                                                                       */
int b200z_bzip2_encode(const uint8_t *in, size_t in_len, uint8_t *out, size_t out_cap, size_t *out_len);
size_t b200z_bzip2_bound(size_t in_len); /* output capacity that always suffices */

/* getCrc32(bytes) -- crc32.dart:6-27 (CRC-32, reflected 0xEDB88320) of a host buffer, computed on the device (tile CRCs
 * folded with x^(8n) mod P): what ZipEncoder stores for members it does not deflate (zip_encoder.dart:113-134).   */
int b200z_crc32(const uint8_t *in, size_t in_len, uint32_t *crc);

/* ---- ZIP container: ZipDecoder / ZipDirectory / ZipFileHeader / ZipFile ------------------------------------
 * b200z_zip_list   = ZipDirectory.read (zip_directory.dart:25-183) + ZipFileHeader.read (zip_file_header.dart:28-111)
 *                    + ZipFile.read (zip_file.dart:73-149), host only: no device is needed.
 * b200z_zip_extract = ZipFile.getStream / decompress (zip_file.dart:164-249) for ALL listed members at once: the deflate
 *                    members are one batch of the inflate kernels, stored members are copies, bzip2 members are
 *                    decoded one after the other.  Names are byte ranges of the archive (decoding them is the host
 *                    language's business).  Encrypted members (ZipCrypto / AES) are reported, not decoded.        */
typedef struct {
  uint64_t local_header_off; /* ZipFileHeader.localHeaderOffset (zip64 applied)                               */
  uint64_t data_off;         /* first byte of the member's data; valid when has_data                          */
  uint64_t comp_size;        /* bytes of member data (central directory value, clipped to the archive)        */
  uint64_t uncomp_size;      /* ZipFile.uncompressedSize: central directory value, or the data descriptor's   */
  uint64_t hint_uncomp_size; /* the central directory value (a size hint only: the data decide)               */
  uint64_t name_off, cd_name_off; /* file name in the local header (what ZipFile.filename is) / in the directory */
  uint32_t name_len, cd_name_len;
  uint32_t crc32, method, flags; /* from the local header (CRC from the data descriptor when flag bit 3 is set) */
  uint32_t mod_time, mod_date, ext_attr, version_made_by;
  uint32_t has_data;         /* 0: no local header signature at local_header_off -> empty content              */
} b200z_zip_entry;
int b200z_zip_list(const uint8_t *zip, size_t zip_len, b200z_zip_entry *entries, size_t cap, size_t *n_entries);
/* ZipDirectory.zipFileComment: byte range of the archive comment inside `zip` (host only). */
int b200z_zip_comment(const uint8_t *zip, size_t zip_len, uint64_t *off, uint32_t *len);
#define B200Z_ZIP_WEB_EOS 1u      /* flags: pure-Dart Inflate end-of-stream behaviour (SURVEY Q1) instead of dart:io's  */
#define B200Z_ZIP_NO_SPLIT 2u     /* flags: do not look for full-flush points inside members                        */
#define B200Z_ZIP_ENCRYPTED (-20)  /* status: encrypted member, not decoded                                      */
#define B200Z_ZIP_TOO_LARGE (-21)  /* status: member of 4 GiB or more                                            */
/* Member i is written to out[out_off[i] .. +out_room[i]); out_len[i] = bytes it produced (may exceed the room:
 * status B200Z_U_NOSPC), status[i] = B200Z_U_* / B200Z_ZIP_*.                                                    */
int b200z_zip_extract(const uint8_t *zip, size_t zip_len, const b200z_zip_entry *entries, size_t n, uint8_t *out,
                      size_t out_cap, const uint64_t *out_off, const uint64_t *out_room, uint64_t *out_len,
                      int32_t *status, uint32_t flags);

/* ---- file streams: InputFileStream -> codec -> OutputFileStream -------------------------------------------------
 * decodeStream / encodeStream with an InputFileStream and an OutputFileStream (input_file_stream.dart:11-221,
 * output_file_stream.dart:11-235; callers: extractFileToDisk, io/extract_archive_to_disk.dart:160-267, and the *_test.dart
 * stream tests).  The reference pulls the file through a FileBuffer cache (file_buffer.dart:10, 1 KiB by default) one
 * readByte() at a time; here the binding passes the PATHS and byte ranges and the library moves the data itself: page-locked
 * segment buffers kept for the life of the library, filled and drained by threads with large pread()/pwrite() calls, so
 * that reading segment k+1, decoding segment k and writing segment k-1 overlap.  GZip members with size hints are cut into
 * segments at member boundaries (B200Z_FILE_SEG_KB, default 256 MiB of compressed bytes); every other case is one segment.
 *
 * Reads in_path[in_off .. in_off+in_len) (clamped to the file, as readBytes does) and writes the result to out_path from
 * byte out_off on (the file is created if needed and NOT truncated: OutputFileStream has done that when it opened it).
 * *in_used = bytes consumed (the streams are read to their end), *out_len = bytes written.  Return codes as for the memory
 * entry points; on B200Z_E_DATA / B200Z_E_THROW the bytes produced before the error are in the file, as in the reference.
 *   op                        a0       a1           a2
 *   B200Z_FILE_GZIP_DECODE    verify   -            -        GZipDecoderWeb.decodeStream  (_gzip_decoder_web.dart:27-58)
 *   B200Z_FILE_ZLIB_DECODE    verify   raw          -        ZLibDecoderWeb.decodeStream  (_zlib_decoder_web.dart:31-107)
 *   B200Z_FILE_BZIP2_DECODE   verify   -            -        BZip2Decoder.decodeStream    (bzip2_decoder.dart:21-88)
 *   B200Z_FILE_ZLIB_ENCODE    level    window_bits  raw      ZLibEncoderWeb.encodeStream  (_zlib_encoder_web.dart:30-73)
 *   B200Z_FILE_GZIP_ENCODE    level    -            mtime    GZipEncoderWeb.encodeStream  (_gzip_encoder_web.dart:30-100)
 *   B200Z_FILE_BZIP2_ENCODE   -        -            -        BZip2Encoder.encodeStream    (bzip2_encoder.dart:25-81)     */
#define B200Z_FILE_GZIP_DECODE 1
#define B200Z_FILE_ZLIB_DECODE 2
#define B200Z_FILE_BZIP2_DECODE 3
#define B200Z_FILE_ZLIB_ENCODE 4
#define B200Z_FILE_GZIP_ENCODE 5
#define B200Z_FILE_BZIP2_ENCODE 6
int b200z_file_codec(int op, const char *in_path, uint64_t in_off, uint64_t in_len, const char *out_path, uint64_t out_off,
                     int32_t a0, int32_t a1, uint32_t a2, uint64_t *in_used, uint64_t *out_len);
/* How the last b200z_file_codec call of this process went: segments decoded through the member-boundary pipeline, and
 * ranges handed to a memory entry point in one piece (tests, tuning of B200Z_FILE_SEG_KB).                          */
void b200z_file_last_stats(uint32_t *n_segments, uint32_t *n_whole);

/* ---- batched independent units (what the kernels run) --------------------------------- */
/* n_units raw DEFLATE streams: unit u reads in_base[in_off[u] .. +in_len[u]) and writes
 * out_base[out_off[u] .. +out_cap[u]).  Per unit: out_len, status (B200Z_U_*), in_used.
 * Host-pointer variant: copies in, runs, copies out (the end-to-end path).  Only the units'
 * slots are copied out: bytes of out_base between slots are left as the caller had them.    */
int b200z_inflate_batch(const uint8_t *in_base, size_t in_bytes, const uint64_t *in_off,
                        const uint32_t *in_len, uint8_t *out_base, size_t out_bytes,
                        const uint64_t *out_off, const uint32_t *out_cap, uint32_t *out_len,
                        int32_t *status, uint32_t *in_used, size_t n_units);
/* Device-pointer variant: every pointer is device memory on the b200z_init device; work is
 * enqueued on `cuda_stream` (a cudaStream_t, NULL = the library's stream) and NOT synchronised.
 * `workspace` must hold b200z_inflate_workspace_bytes(...) bytes.  Its third argument is the
 * EXTENT of the output layout, max over u of out_off[u] + out_cap[u] -- not the sum of the caps:
 * the workspace mirrors the output layout, gaps included.
 * Test and diagnostic mode: with B200Z_FAST=2 in the environment (read at every call) only the
 * shared-memory kernel runs.  A unit it does not finish keeps the out_len / status / in_used
 * values the caller put there, and its output slot is not written.  B200Z_FAST=0 runs only the
 * exact kernels; the default (1) runs both, the exact ones on what the first leaves.         */
size_t b200z_inflate_workspace_bytes(size_t n_units, size_t total_in_bytes, size_t out_extent);
int b200z_inflate_batch_device(const uint8_t *d_in_base, const uint64_t *d_in_off,
                               const uint32_t *d_in_len, uint8_t *d_out_base,
                               const uint64_t *d_out_off, const uint32_t *d_out_cap,
                               uint32_t *d_out_len, int32_t *d_status, uint32_t *d_in_used,
                               size_t n_units, void *d_workspace, size_t workspace_bytes,
                               void *cuda_stream);

/* ---- several GPUs of one box driven by ONE process (SURVEY.md 8b: device_mask / n_gpus; 8e) ----------------
 * The reference decodes the members of a gzip stream in one loop and returns one buffer
 * (_gzip_decoder_web.dart:27-38).  Here the members -- or the units of a batch -- are cut into one contiguous range
 * per GPU (balanced by compressed bytes); every GPU receives its range over its own link, decodes it, and its part of
 * the output stream goes straight to its place in the caller's buffer.  B200Z_MULTI_GATHER: the shards are also
 * exchanged over NVLink (NCCL, communicators owned by the library, looked up at run time) so that EVERY device then
 * holds the whole stream in block order (b200z_multi_device_output) -- BASELINE north_star's all-gather.
 * b200z_multi_init(mask): bit d = CUDA device d; also runs b200z_init on the first device of the mask, which serves
 * whatever cannot be dealt (members without size hints, hints that lie, the zlib fall-back).                       */
#define B200Z_MULTI_GATHER 1u
int b200z_multi_init(uint32_t device_mask, uint32_t flags);
void b200z_multi_shutdown(void);
int b200z_multi_device_count(void);
int b200z_gzip_decode_multi(const uint8_t *in, size_t in_len, int verify, uint8_t *out, size_t out_cap,
                            size_t *out_len, uint32_t flags);
int b200z_inflate_batch_multi(const uint8_t *in_base, size_t in_bytes, const uint64_t *in_off,
                              const uint32_t *in_len, uint8_t *out_base, size_t out_bytes,
                              const uint64_t *out_off, const uint32_t *out_cap, uint32_t *out_len,
                              int32_t *status, uint32_t *in_used, size_t n_units, uint32_t flags);
/* after a B200Z_MULTI_GATHER call: device `slot` (0 .. b200z_multi_device_count()-1) holds *bytes of output at the
 * returned device pointer; NULL when the last call did not gather.                                             */
const void *b200z_multi_device_output(int slot, size_t *bytes);

/* Number of kernel launches issued by this library since b200z_init (bench.py gpu_launches). */
uint64_t b200z_launch_count(void);
/* Optional per-kernel timing with CUDA events on the launching stream: enable, run batches, then read
 * the summed durations (ms) of the three inflate kernels (k_inflate_fast, then the exact pair k_inflate_decode /
 * k_inflate_expand over the units the first one left) and the number of batches timed.                        */
void b200z_profile_enable(int on);
int b200z_profile_read(double *fast_ms, double *decode_ms, double *expand_ms, uint64_t *n_batches);

#ifdef __cplusplus
}
#endif
#endif /* B200Z_H */
