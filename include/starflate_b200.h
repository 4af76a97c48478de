/* starflate_b200 — C ABI of the B200-native raw-DEFLATE decompressor.
 *
 * This is the drop-in boundary for the one hot path of garymm/starflate:
 *   starflate::decompress(std::span<const std::byte>, std::span<std::byte>) -> DecompressStatus
 *   (reference: src/decompress.hpp:63-64, src/decompress.cpp:402-461)
 * The reference has no FFI/plugin registry; its C++ free function *is* the interface.  The
 * C++23 mirror of that interface lives in starflate_b200/cpp/ (g++), and reaches the CUDA
 * kernels (nvcc, C++20) only through the functions declared here — plain pointers and sizes,
 * no C++ or torch types.  INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Two kinds of result:
 *   - the return value of every function is an *infrastructure* code (sfb200_rc): 0 on success,
 *     non-zero for CUDA / argument failures.  There is no CPU fallback: without a usable CUDA
 *     device every entry point fails with SFB200_RC_NO_DEVICE.
 *   - per-stream results are starflate::DecompressStatus values (src/decompress.hpp:13-23),
 *     one uint8_t per stream, bit-identical to what the reference returns for that stream, plus
 *     `written` (bytes produced) — an extension the reference cannot report.
 */
#ifndef STARFLATE_B200_H
#define STARFLATE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SFB200_ABI_VERSION 6

/* starflate::DecompressStatus, numeric values preserved (src/decompress.hpp:13-23). */
enum sfb200_status {
  SFB200_SUCCESS = 0,
  SFB200_ERROR = 1, /* never produced by the reference; used here only for streams that
                       violate the batch preconditions (sizes >= 4 GiB, see below) */
  SFB200_INVALID_BLOCK_HEADER = 2,
  SFB200_NO_COMPRESSION_LEN_MISMATCH = 3,
  SFB200_DST_TOO_SMALL = 4,
  SFB200_SRC_TOO_SMALL = 5,
  SFB200_INVALID_LIT_OR_LEN = 6,
  SFB200_INVALID_DISTANCE = 7
};

/* infrastructure return codes */
enum sfb200_rc {
  SFB200_RC_OK = 0,
  SFB200_RC_NO_DEVICE = 1,    /* no CUDA device / driver: the product has no CPU path */
  SFB200_RC_BAD_ARGUMENT = 2,
  SFB200_RC_CUDA_ERROR = 3,   /* see sfb200_last_error() */
  SFB200_RC_OUT_OF_MEMORY = 4
};

typedef struct sfb200_ctx sfb200_ctx;

/* Create / destroy a context bound to one CUDA device (one per process-rank; streams of a
 * batch are independent, so multi-GPU use is one context per GPU with no communication). */
int sfb200_create(int device, sfb200_ctx** out);
void sfb200_destroy(sfb200_ctx* ctx);
const char* sfb200_last_error(const sfb200_ctx* ctx);
int sfb200_abi_version(void);

/* Batched decompress, everything resident in device memory (the metric's path).
 *
 * Stream i reads  src_base[src_off[i] .. src_off[i]+src_len[i])  and writes
 *                 dst_base[dst_off[i] .. dst_off[i]+dst_cap[i]);
 * `dst_bytes` is the size of the buffer at dst_base (every dst_off[i]+dst_cap[i] <= dst_bytes);
 * it sizes the scratch the decoder needs (kept in the context): one bit per dst byte, and for a
 * call with n == 1 — the single-stream route, which decodes the blocks of the stream side by side
 * and resolves back-references over the whole output at once — about 4.5 bytes per dst byte more.
 * status[i] receives the DecompressStatus, written[i] (may be NULL) the bytes produced.
 * All six arrays are DEVICE pointers; regions of different streams must not overlap.
 * Replaces one reference call per stream: decompress(src_i, dst_i) (src/decompress.cpp:402).
 * Semantics preserved per stream: first error wins, bytes already produced stay in dst,
 * dst beyond `written` is never touched, trailing src bytes after the final block are ignored.
 * Precondition: src_len[i], dst_cap[i] < 2^32 - 256 (else status[i] = SFB200_ERROR).
 * Memory touched: src is read in aligned 16-byte blocks, never past a stream's last byte and at
 * most 15 bytes before its first (inside the same 16-byte block); dst is read and written in
 * aligned words, only words that hold at least one byte of a stream's region, and only the
 * region's own bytes are ever modified.
 * Threading: a context serves one call at a time (it owns scratch buffers and streams); use one
 * context per thread (the C++ layer does) or serialise calls.  Every entry point leaves the calling
 * thread's current CUDA device as it found it.
 * `cuda_stream` is a cudaStream_t (NULL = default stream); the call is asynchronous. */
int sfb200_decompress_batch_device(sfb200_ctx* ctx, const uint8_t* src_base,
                                   const uint64_t* src_off, const uint64_t* src_len,
                                   uint8_t* dst_base, uint64_t dst_bytes, const uint64_t* dst_off,
                                   const uint64_t* dst_cap, uint8_t* status,
                                   uint64_t* written, uint64_t n, void* cuda_stream);

/* Same batch, HOST buffers, in bounded device memory.  The batch is cut into sub-batches of
 * consecutive streams that flow through a ring of three staging slots on the device
 * (SFB200_HOST_STAGING_MB, default 3456 MiB in all; a single stream larger than a slot makes the
 * slots grow to hold it): the upload of one sub-batch, the kernels of the one before and the
 * download of the one before that overlap, so a batch of any size — larger than the GPU's memory
 * included — decodes at the speed of the slower PCIe direction.  `src_bytes` / `dst_bytes` are the
 * sizes of the two flat buffers.  dst is NOT uploaded and only bytes the decoder produced are
 * copied back, so everything else in the caller's buffer keeps its value (reference contract:
 * dst beyond what was written is never touched).  Synchronous.  Pinned host buffers
 * (cudaHostAlloc / cudaHostRegister) make the copies asynchronous; pageable ones work, slower. */
int sfb200_decompress_batch_host(sfb200_ctx* ctx, const uint8_t* src, uint64_t src_bytes,
                                 const uint64_t* src_off, const uint64_t* src_len,
                                 uint8_t* dst, uint64_t dst_bytes, const uint64_t* dst_off,
                                 const uint64_t* dst_cap, uint8_t* status, uint64_t* written,
                                 uint64_t n);

/* One batch, several GPUs of one box (BASELINE.json configs[2]: "sharded across 2/4/8 B200";
 * SURVEY.md §8e).  `ctxs` are n_ctx contexts, normally one per device: the streams are cut into
 * n_ctx contiguous shards balanced by sum(src_len + dst_cap) (sfb200_partition_streams) and every
 * context decodes its shard with sfb200_decompress_batch_host on a host thread of its own.  The
 * streams are independent: there is no communication between the devices.  Results land in the
 * same arrays as the single-device call would have put them. */
int sfb200_decompress_batch_host_multi(sfb200_ctx* const* ctxs, int n_ctx, const uint8_t* src, uint64_t src_bytes,
                                       const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst,
                                       uint64_t dst_bytes, const uint64_t* dst_off, const uint64_t* dst_cap,
                                       uint8_t* status, uint64_t* written, uint64_t n);
/* cut[0] = 0 <= cut[1] <= ... <= cut[parts] = n: shard k is streams [cut[k], cut[k+1]). */
void sfb200_partition_streams(const uint64_t* src_len, const uint64_t* dst_cap, uint64_t n, int parts,
                              uint64_t* cut);

/* Device memory the host-buffer entry points hold for staging right now (the three slots). */
uint64_t sfb200_staging_bytes(const sfb200_ctx* ctx);

/* Single stream, host buffers: the exact shape of the reference entry point
 * decompress(span src, span dst) (src/decompress.hpp:63-64).  *status receives the
 * DecompressStatus; *written (may be NULL) the bytes produced. */
int sfb200_decompress(sfb200_ctx* ctx, const uint8_t* src, size_t src_len, uint8_t* dst,
                      size_t dst_cap, uint8_t* status, uint64_t* written);

/* Chunked input for ONE stream (extension; SURVEY.md §8 f3 — the reference anticipates it at
 * src/decompress.cpp:214): the compressed bytes arrive in pieces, the output leaves in pieces, and
 * neither has to fit device (or host) memory as a whole.  The unit of progress is the deflate
 * BLOCK: a call decodes every block that is complete in the input fed so far and that fits `dst`,
 * and carries to the next call the bytes from the next block header on, the bit offset of that
 * header and the last 32 KiB of output (the LZ77 window) — all on the device.
 *   feed(src, src_len, last, dst, dst_cap):  `src` = the next src_len bytes of the stream (host
 *   memory; 0 is fine: decode more of what is buffered), `last` != 0 = no input comes after these.
 *   *written = bytes put into dst by this call (they follow what earlier calls returned);
 *   *finished != 0: the stream has ended and *status is its DecompressStatus — Success after the
 *   final block, else exactly the status one sfb200_decompress call over the whole input would
 *   return (with `last` set, input that stops short is an error as it is there; the bytes decoded
 *   before it are returned).  Running out of room never ends the stream: while *finished == 0,
 *   *status is SFB200_SUCCESS, or SFB200_DST_TOO_SMALL with *written == 0 when dst cannot hold even
 *   the next block: nothing is lost, call again with more room (zlib's blocks are tens to hundreds of KiB of output; a block of
 *   back-to-back maximum-length matches can reach a few MiB).  An error inside a block that is not
 *   the last chunk cannot be told from input that merely stops short, so it is reported once `last`
 *   is set.  Synchronous; a stream belongs to the context it was created on (one call at a time). */
typedef struct sfb200_inflate_stream sfb200_inflate_stream;
int sfb200_inflate_stream_create(sfb200_ctx* ctx, sfb200_inflate_stream** out);
void sfb200_inflate_stream_destroy(sfb200_inflate_stream* s);
int sfb200_inflate_stream_feed(sfb200_inflate_stream* s, const uint8_t* src, size_t src_len, int last, uint8_t* dst,
                               size_t dst_cap, uint64_t* written, uint8_t* status, int* finished);

/* Batched COMPRESSION to raw DEFLATE (extension; SURVEY.md §8 f4 — the direction the reference's
 * README names as not built yet, README.md:5-7; it only has the Huffman-table construction,
 * huffman/src/table.hpp:246-298).  Stream i = src_base[src_off[i] .. +src_len[i]) is written as one
 * RFC 1951 stream to dst_base[dst_off[i] .. +dst_cap[i]): LZ77 by hashing (4-byte minimum match,
 * 32 KiB window, greedy) and ONE Huffman block — dynamic (code lengths derived on the device from
 * the stream's own symbol counts) where that is smaller, else fixed — or stored blocks where
 * neither beats the input.
 * status[i] = SFB200_SUCCESS with written[i] bytes, or SFB200_DST_TOO_SMALL (written[i] = 0: neither
 * form fits; sfb200_compress_bound(src_len) always does), or SFB200_ERROR for src_len[i] >= 2^32 -
 * 256.  Bytes of the dst region past written[i] may have been used as scratch.  The output decodes
 * with sfb200_decompress_*, with zlib and with the reference's decompress().  All arrays are
 * DEVICE pointers; asynchronous on `cuda_stream`. */
uint64_t sfb200_compress_bound(uint64_t src_len);
int sfb200_compress_batch_device(sfb200_ctx* ctx, const uint8_t* src_base, const uint64_t* src_off,
                                 const uint64_t* src_len, uint8_t* dst_base, const uint64_t* dst_off,
                                 const uint64_t* dst_cap, uint8_t* status, uint64_t* written, uint64_t n,
                                 void* cuda_stream);
/* One stream in host memory.  It is compressed by ONE warp (about 10 MB/s); a large buffer goes
 * through sfb200_compress_parallel* instead, which writes one stream at batch speed. */
int sfb200_compress(sfb200_ctx* ctx, const uint8_t* src, size_t src_len, uint8_t* dst, size_t dst_cap,
                    uint8_t* status, uint64_t* written);

/* Size discovery (extension; SURVEY.md §8 f2).  The reference's decompress() returns no size and
 * requires the caller to bring a dst that is large enough (src/decompress.hpp:57-64).  This runs
 * the Huffman layer of every stream without storing anything: size[i] receives the number of bytes
 * decompress(src_i, dst) would produce into a dst without a limit, status[i] the status it would
 * return (Success, or the error that ends the stream; size[i] is then the bytes produced before
 * it).  No dst, no scratch.  All arrays are DEVICE pointers; asynchronous on `cuda_stream`.
 * Precondition: src_len[i] < 2^32 - 256, decompressed size < 2^32 - 528 (else SFB200_ERROR or
 * SFB200_DST_TOO_SMALL respectively). */
int sfb200_decompressed_size_batch_device(sfb200_ctx* ctx, const uint8_t* src_base,
                                          const uint64_t* src_off, const uint64_t* src_len,
                                          uint8_t* status, uint64_t* size, uint64_t n,
                                          void* cuda_stream);

/* The same for one stream in host memory (what dst.size() a caller of sfb200_decompress needs). */
int sfb200_decompressed_size(sfb200_ctx* ctx, const uint8_t* src, size_t src_len, uint8_t* status,
                             uint64_t* size);

/* zlib (RFC 1950) and gzip (RFC 1952) containers (extension; SURVEY.md §8 f1 — the reference is
 * raw-DEFLATE only).  Same arguments as sfb200_decompress_batch_device, each stream being a whole
 * container: the header is parsed and the trailer's Adler-32 / CRC-32 (and gzip's ISIZE) verified
 * against the produced bytes, all on the device.  `container`: SFB200_CONTAINER_*; AUTO decides
 * per stream (gzip magic, else a valid zlib header, else raw).  status[i] is the DecompressStatus
 * of the DEFLATE payload, or one of the values below.  One member per stream, no trailing bytes,
 * no preset dictionary. */
enum sfb200_container {
  SFB200_CONTAINER_RAW = 0,
  SFB200_CONTAINER_ZLIB = 1,
  SFB200_CONTAINER_GZIP = 2,
  SFB200_CONTAINER_AUTO = 3
};
enum sfb200_container_status {
  SFB200_BAD_CONTAINER = 8,      /* malformed or unsupported header (nothing is written) */
  SFB200_CHECKSUM_MISMATCH = 9,  /* the payload decoded, its Adler-32 / CRC-32 is not the trailer's */
  SFB200_SIZE_MISMATCH = 10      /* gzip: ISIZE is not the decoded size modulo 2^32 */
};
int sfb200_decompress_container_batch_device(sfb200_ctx* ctx, int container, const uint8_t* src_base,
                                             const uint64_t* src_off, const uint64_t* src_len,
                                             uint8_t* dst_base, uint64_t dst_bytes,
                                             const uint64_t* dst_off, const uint64_t* dst_cap,
                                             uint8_t* status, uint64_t* written, uint64_t n,
                                             void* cuda_stream);
/* One container in host memory (the shape of sfb200_decompress). */
int sfb200_decompress_container(sfb200_ctx* ctx, int container, const uint8_t* src, size_t src_len,
                                uint8_t* dst, size_t dst_cap, uint8_t* status, uint64_t* written);

/* gzip FILES: a series of gzip members (RFC 1952 §2.2), as gzip(1), zlib's gunzip and Python's
 * gzip.decompress accept them — `cat a.gz b.gz`, and BGZF (BAM, bgzip / tabix .vcf.gz, .fastq.gz),
 * whose members carry their compressed size in the header (extra subfield 'B','C').  The members
 * are found on the device (BGZF members without any serial walk) and decoded side by side through
 * the container batch path; a member without the BGZF field costs one extra decode of its payload
 * to find where it ends.  Member k's output follows member k-1's in dst.
 *   *status   Success; or the status of the FIRST failing member in file order (the DEFLATE status
 *             of its payload, SFB200_CHECKSUM_MISMATCH, SFB200_SIZE_MISMATCH — also when a member's
 *             payload produces more than its ISIZE while dst still had room (for a member without
 *             the BGZF field: room for its whole payload, as its ISIZE is read only after it) —,
 *             SFB200_DST_TOO_SMALL
 *             when dst ends inside a member: every byte that fits is produced); SFB200_BAD_CONTAINER
 *             for bytes behind the last member that are neither zero padding (ignored) nor a gzip
 *             member, for a file that does not start with a member, and for a file that ends inside
 *             a header or trailer.  An empty file is Success with 0 bytes.
 *   *written  (may be NULL) bytes of dst that hold the file's output: on failure, that member's dst
 *             offset plus what it produced.  On Success dst past *written is untouched; after a
 *             failure the bytes past *written are unspecified (later members may have been decoded).
 *   *members  (may be NULL) members found.
 * `src` and `dst` are DEVICE pointers, the three results HOST pointers.  Synchronous on
 * `cuda_stream` (the member count sizes the launches).  Members must be < 4 GiB compressed and
 * decompressed (BGZF members are <= 64 KiB).  Memory touched: the member scan reads src in aligned
 * 16-byte blocks, up to 15 bytes before its first and after its last byte.  More than 2^32 - 2
 * BGZF header candidates (only a file of > 8 GiB of header-like bytes) is SFB200_RC_BAD_ARGUMENT. */
int sfb200_decompress_gzip_file_device(sfb200_ctx* ctx, const uint8_t* src, uint64_t src_len, uint8_t* dst,
                                       uint64_t dst_cap, uint8_t* status, uint64_t* written, uint64_t* members,
                                       void* cuda_stream);
/* The same with HOST buffers.  The whole file and its output must fit in device memory (it is staged
 * there whole); only the bytes produced are copied back. */
int sfb200_decompress_gzip_file(sfb200_ctx* ctx, const uint8_t* src, size_t src_len, uint8_t* dst, size_t dst_cap,
                                uint8_t* status, uint64_t* written, uint64_t* members);
/* Discovery only (HOST buffer): *size = the sum of ISIZE over the members the walk reaches,
 * *members (may be NULL) their number; *complete (may be NULL) = 1 when they cover the file (zero
 * padding aside).  A member without the BGZF field, or anything else that is not a BGZF member,
 * ends the walk with *complete = 0.  BGZF callers size dst with it exactly. */
int sfb200_gzip_file_size(sfb200_ctx* ctx, const uint8_t* src, size_t src_len, uint64_t* size, uint64_t* members,
                          int* complete);

/* ZIP ARCHIVES (PKWARE APPNOTE 6.3 as Python's zipfile reads them: ZIP64, prepended bytes, data
 * descriptors).  The entry table is the interface: list it, optionally filter or reorder its rows,
 * then extract them.  Deflated (method 8) entries are decoded side by side by the batch path, stored
 * (method 0) ones copied; the CRC-32 of every entry's output is checked against the central
 * directory, all on the device.  Sizes and CRC come from the central directory; data descriptors
 * are skipped, not read.  Other methods, encryption and split archives are not supported. */
typedef struct sfb200_zip_entry {  /* 64 bytes */
  uint64_t name_off;   /* file name bytes: src[name_off .. + name_len) (central directory) */
  uint64_t data_off;   /* stored / compressed bytes: src[data_off .. + comp_size) */
  uint64_t comp_size;
  uint64_t size;       /* uncompressed size (central directory) */
  uint64_t dst_off;    /* where extract writes the entry; list fills it packed in directory order */
  uint64_t written;    /* extract: bytes produced */
  uint32_t crc32;
  uint16_t method, flags;
  uint16_t name_len;
  uint8_t status;      /* list: Success, or SFB200_BAD_CONTAINER for a row that cannot be extracted
                        * (bad local header, data outside the file, a method other than 0 / 8,
                        * encryption); extract: the entry's result (below) */
  uint8_t pad[5];
} sfb200_zip_entry;
/* *status: Success, or SFB200_BAD_CONTAINER for the archive as a whole (no end-of-central-directory
 * record, a split archive, a central directory whose chain of records does not hold exactly the
 * record's count).  *count = entries in the archive (0 when it is rejected); only the first
 * min(count, cap) rows are written (cap 0 sizes the table).  *total_size = sum of `size` = the dst_cap
 * a packed extract needs.  src and entries are DEVICE pointers, the three results HOST pointers;
 * synchronous on cuda_stream.  Memory touched: aligned 16-byte loads inside the blocks that hold the
 * archive's bytes. */
int sfb200_zip_list_device(sfb200_ctx* ctx, const uint8_t* src, uint64_t src_len, sfb200_zip_entry* entries,
                           uint64_t cap, uint8_t* status, uint64_t* count, uint64_t* total_size, void* cuda_stream);
/* The same with HOST buffers (the archive is staged on the device whole). */
int sfb200_zip_list(sfb200_ctx* ctx, const uint8_t* src, size_t src_len, sfb200_zip_entry* entries, uint64_t cap,
                    uint8_t* status, uint64_t* count, uint64_t* total_size);
/* Decodes rows [0, n) of `entries` (any subset or order of a list's rows) into
 * dst[dst_off .. + size) and writes status / written into the rows.  Regions must not overlap.
 * Per-row status: the DEFLATE status of the payload; SFB200_CHECKSUM_MISMATCH (the output's CRC-32 is
 * not the central directory's); SFB200_SIZE_MISMATCH (the output size is not `size`, a stored entry
 * whose comp_size is not its size, or a payload that produces more than `size` while dst had room);
 * SFB200_DST_TOO_SMALL (dst ends inside the entry's region: every byte that fits is produced);
 * SFB200_BAD_CONTAINER (a row list marked so, data outside src, an unsupported method or
 * encryption); SFB200_ERROR (a deflated entry of >= 2^32 - 256 bytes, compressed or not; stored
 * entries have no size limit).  src, entries and dst are DEVICE pointers; synchronous on cuda_stream. */
int sfb200_zip_extract_device(sfb200_ctx* ctx, const uint8_t* src, uint64_t src_len, sfb200_zip_entry* entries,
                              uint64_t n, uint8_t* dst, uint64_t dst_cap, void* cuda_stream);
/* The same with HOST buffers: only the bytes produced are copied back (dst keeps its other bytes). */
int sfb200_zip_extract(sfb200_ctx* ctx, const uint8_t* src, size_t src_len, sfb200_zip_entry* entries, uint64_t n,
                       uint8_t* dst, size_t dst_cap);

/* COMPRESSION to zlib (RFC 1950) and gzip (RFC 1952): sfb200_compress_batch_device's streams with
 * header and trailer, the Adler-32 / CRC-32 (and ISIZE) of each stream's SOURCE bytes computed on the
 * device.  zlib: 78 9c, payload, Adler-32 big endian.  gzip: 1f 8b 08 00, MTIME 0, XFL 0, OS 255
 * (the first 10 bytes Python's gzip.GzipFile writes at level 6 with mtime=0), payload, CRC-32 and ISIZE little
 * endian.  The payload is what sfb200_compress_batch_device writes for the stream.  `container`:
 * RAW (exactly sfb200_compress_batch_device), ZLIB or GZIP; AUTO is SFB200_RC_BAD_ARGUMENT.
 * Statuses as there: SFB200_DST_TOO_SMALL with written[i] = 0 when the framed stream does not fit
 * dst_cap[i] (sfb200_compress_container_bound(container, src_len) always does), SFB200_ERROR for
 * src_len[i] >= 2^32 - 256.  Bytes of the dst region past written[i] may have been used as scratch.
 * src is read twice (the compressor, then the checksum: 16-byte loads inside the same aligned 16-byte
 * blocks as the stream's bytes).  The context keeps 16 bytes per stream of scratch.  All arrays are
 * DEVICE pointers; asynchronous on `cuda_stream`. */
uint64_t sfb200_compress_container_bound(int container, uint64_t src_len);
int sfb200_compress_container_batch_device(sfb200_ctx* ctx, int container, const uint8_t* src_base,
                                           const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst_base,
                                           const uint64_t* dst_off, const uint64_t* dst_cap, uint8_t* status,
                                           uint64_t* written, uint64_t n, void* cuda_stream);
/* One stream in host memory, compressed by one warp: for a large buffer see sfb200_compress_parallel*. */
int sfb200_compress_container(sfb200_ctx* ctx, int container, const uint8_t* src, size_t src_len, uint8_t* dst,
                              size_t dst_cap, uint8_t* status, uint64_t* written);

/* COMPRESSION of one buffer to a BGZF file: the input is cut into pieces of 65 280 bytes (bgzip's), every
 * piece compressed by the batch compressor as one BGZF member (header 1f 8b 08 04, MTIME 0, XFL 0,
 * OS 255, XLEN 6, subfield 'B' 'C' SLEN 2 BSIZE = member length - 1; payload; CRC-32 and ISIZE),
 * the pieces side by side, then the 28-byte EOF marker of the SAM/BAM specification.  The output
 * decodes with gzip(1), Python's gzip, htslib and sfb200_decompress_gzip_file*.  Any src_len,
 * 4 GiB and more included.
 *   *status   Success; SFB200_DST_TOO_SMALL when the file does not fit dst_cap (never with dst_cap >=
 *             sfb200_compress_bgzf_bound(src_len)): *written = 0, no byte past dst_cap is touched and
 *             the bytes before it are unspecified.
 *   *written  (may be NULL) the file's size.   *members  (may be NULL) members written, the EOF marker
 *             included (what sfb200_decompress_gzip_file* reports for the file); 0 on failure.
 * `src` and `dst` are DEVICE pointers, the three results HOST pointers; synchronous on `cuda_stream`.
 * Scratch kept in the context: 64 KiB + 41 bytes per piece of a round.  A round holds at most
 * SFB200_BGZF_SCRATCH_MB (default 8192) MiB of pieces' scratch; larger inputs take several rounds,
 * with a constant number of kernel launches each and no host round trip between them.  src is read
 * twice (the compressor, then the CRC-32), in 16-byte loads inside the aligned 16-byte blocks that
 * hold its bytes; dst is written once. */
uint64_t sfb200_compress_bgzf_bound(uint64_t src_len);
int sfb200_compress_bgzf_device(sfb200_ctx* ctx, const uint8_t* src, uint64_t src_len, uint8_t* dst, uint64_t dst_cap,
                                uint8_t* status, uint64_t* written, uint64_t* members, void* cuda_stream);
/* The same with HOST buffers: input and output are staged on the device whole; only the bytes written
 * are copied back. */
int sfb200_compress_bgzf(sfb200_ctx* ctx, const uint8_t* src, size_t src_len, uint8_t* dst, size_t dst_cap,
                         uint8_t* status, uint64_t* written, uint64_t* members);

/* COMPRESSION of one buffer to ONE raw-DEFLATE, zlib or gzip stream at batch speed (what PNG IDAT, PDF
 * FlateDecode, HTTP deflate, zip entries and single-member .gz files hold).  The input is cut into
 * BGZF's pieces of 65 280 bytes; piece k is compressed by the batch compressor as one self-contained
 * block (dynamic or fixed Huffman, or stored where neither is smaller than the piece + 5 bytes), BFINAL
 * set only on the last piece, and the blocks follow one another at BIT granularity, with no gap and no
 * empty stored block between them.  The last byte is padded with zero bits.  Header and trailer are
 * byte-identical to sfb200_compress_container's (zlib 78 9c .. Adler-32; gzip 1f 8b 08 00, MTIME 0,
 * XFL 0, OS 255 .. CRC-32, ISIZE = src_len mod 2^32), the checksum over the whole source computed on
 * the device.  For src_len <= 65 280 the output is exactly sfb200_compress_container's.  The stream is
 * one dynamic block per piece, which sfb200_decompress* decodes block by block side by side.
 * `container`: RAW, ZLIB or GZIP; AUTO (or anything else) is SFB200_RC_BAD_ARGUMENT.  Any src_len,
 * 4 GiB and more included.
 *   *status   Success; SFB200_DST_TOO_SMALL when the stream does not fit dst_cap (never with dst_cap >=
 *             sfb200_compress_parallel_bound(container, src_len) = header + trailer + src_len +
 *             6 x max(1, ceil(src_len / 65 280))): *written = 0, no byte past dst_cap is touched and the
 *             bytes before it are unspecified.
 *   *written  (may be NULL) the stream's size.
 * `src` and `dst` are DEVICE pointers, the results HOST pointers; synchronous on `cuda_stream`.
 * Scratch and rounds are those of sfb200_compress_bgzf_device (SFB200_BGZF_SCRATCH_MB), with five kernel
 * launches per round and no host round trip between them.  src is read twice (the compressor, then the
 * checksum and the bytes of stored pieces); dst is written once. */
uint64_t sfb200_compress_parallel_bound(int container, uint64_t src_len);
int sfb200_compress_parallel_device(sfb200_ctx* ctx, int container, const uint8_t* src, uint64_t src_len,
                                    uint8_t* dst, uint64_t dst_cap, uint8_t* status, uint64_t* written,
                                    void* cuda_stream);
/* The same with HOST buffers: input and output are staged on the device whole; only the bytes written
 * are copied back. */
int sfb200_compress_parallel(sfb200_ctx* ctx, int container, const uint8_t* src, size_t src_len,
                             uint8_t* dst, size_t dst_cap, uint8_t* status, uint64_t* written);

/* Position-weighted 64-bit checksum of each stream's output region [0, len[i]) computed on the
 * device (used by tests/bench to verify multi-GiB outputs without a device->host copy):
 *   sum_j (byte_j + 1) * (0x9E3779B97F4A7C15 * (j + 1) | 1)   mod 2^64. */
int sfb200_checksum_batch_device(sfb200_ctx* ctx, const uint8_t* base, const uint64_t* off,
                                 const uint64_t* len, uint64_t* out, uint64_t n,
                                 void* cuda_stream);

/* Tuning / introspection (bench harness only; not part of the reference surface). */
typedef struct sfb200_launch_info {
  int sm_count;
  /* pass 1, huff_lanes_kernel (one lane per stream) */
  int warps_per_cta;
  int ctas_per_sm;
  int smem_bytes_per_cta;
  int regs_per_thread;
  /* pass 1 with the small table geometry (tried first; 0 CTAs per SM = unavailable) */
  int small_warps_per_cta;
  int small_ctas_per_sm;
  int small_regs_per_thread;
  /* pass 1 in single-stream mode, huff_stream_kernel (one warp per stream; few, large streams) */
  int stream_ctas_per_sm;
  int stream_regs_per_thread;
  /* pass 2, lz_window_kernel (one warp per stream) */
  int lz_threads_per_cta;
  int lz_ctas_per_sm;
  int lz_regs_per_thread;
  uint64_t kernel_launches; /* kernels launched by this context so far */
} sfb200_launch_info;
int sfb200_get_launch_info(sfb200_ctx* ctx, sfb200_launch_info* out);

/* Device time of the most recent sfb200_decompress_batch_device call on this context, from CUDA
 * events recorded on its stream inside that call (waits for the call to finish), milliseconds:
 *   out3[0] scratch clearing and batch preparation,
 *   out3[1] pass 1, the Huffman layer (huff_lanes_kernel; one stream or a few large ones:
 *           find / verify candidates, huff_stream_kernel counting and writing, the chain),
 *   out3[2] pass 2, the LZ77 back-references (lz_window_kernel; single-stream route: lz_jump_*).
 * (With SFB200_OVERLAP=1 — the experimental wave form — the passes overlap: out3[1] then runs to
 * the end of the last wave of pass 1 and out3[2] is what remains of pass 2 after that.) */
int sfb200_last_pass_ms(sfb200_ctx* ctx, float* out3);

#ifdef __cplusplus
}
#endif
#endif /* STARFLATE_B200_H */
