// starflate_b200 — drop-in C++23 interface of the reference's decompress path
// (garymm/starflate src/decompress.hpp:13-71): same namespace, names, enumerator values and
// call shapes, so a caller of the reference compiles against this header unchanged.
// The work is done by the CUDA library behind the C ABI in include/starflate_b200.h
// (nvcc cannot parse C++23, hence the seam).  There is no CPU decode path: without a usable
// CUDA device decompress() terminates the process with a diagnostic.
#pragma once

#include "huffman/huffman.hpp"

#include <cstddef>
#include <cstdint>
#include <expected>
#include <ranges>
#include <optional>
#include <span>
#include <vector>

namespace starflate {

// numeric values are part of the contract (they cross the C ABI as uint8_t)
enum class DecompressStatus : std::uint8_t
{
  Success,
  Error,
  InvalidBlockHeader,
  NoCompressionLenMismatch,
  DstTooSmall,
  SrcTooSmall,
  InvalidLitOrLen,
  InvalidDistance,
};

namespace detail {

enum class BlockType : std::uint8_t
{
  NoCompression,
  FixedHuffman,
  DynamicHuffman,
};

struct BlockHeader
{
  bool final;
  BlockType type;
};

/// 3-bit block header (BFINAL, BTYPE); consumes it on success (reference :370-385).
auto read_header(huffman::bit_span& compressed_bits) -> std::expected<BlockHeader, DecompressStatus>;

/// Copies n bytes from (dst - distance) to dst, repeating when the ranges overlap
/// (reference :388-398).  @pre dst - distance is valid.
void copy_from_before(std::uint16_t distance, std::span<std::byte>::iterator dst, std::uint16_t n);

}  // namespace detail

/// Decompresses one raw-DEFLATE stream (reference :402-461), on the GPU.
auto decompress(std::span<const std::byte> src, std::span<std::byte> dst) -> DecompressStatus;

template <std::ranges::contiguous_range R>
  requires std::same_as<std::ranges::range_value_t<R>, std::byte>
auto decompress(const R& src, std::span<std::byte> dst)
{
  return decompress(std::span<const std::byte>{src.data(), src.size()}, dst);
}

// ---- extension: size discovery --------------------------------------------------------------
/// The number of bytes decompress(src, dst) produces into a dst that is large enough — which the
/// reference leaves to the caller to know — or the status that ends the stream.  Nothing is
/// stored; one H2D copy of src, one kernel.
auto decompressed_size(std::span<const std::byte> src) -> std::expected<std::size_t, DecompressStatus>;

// ---- extension: zlib (RFC 1950) / gzip (RFC 1952) containers ----------------------------------
enum class Container : std::uint8_t { Raw = 0, Zlib = 1, Gzip = 2, Auto = 3 };
/// DecompressStatus (same values) plus what only a container can get wrong.
enum class ContainerStatus : std::uint8_t
{
  Success = 0,
  Error,
  InvalidBlockHeader,
  NoCompressionLenMismatch,
  DstTooSmall,
  SrcTooSmall,
  InvalidLitOrLen,
  InvalidDistance,
  BadContainer,      // malformed or unsupported header
  ChecksumMismatch,  // Adler-32 / CRC-32 of the output is not the trailer's
  SizeMismatch,      // gzip ISIZE
};
/// decompress() for a whole zlib / gzip container: header, DEFLATE payload, trailer checksum
/// (verified on the device).  `written`, if given, receives the number of bytes produced.
auto decompress_container(std::span<const std::byte> src, std::span<std::byte> dst, Container container,
                          std::size_t* written = nullptr) -> ContainerStatus;
/// A gzip FILE: any number of members (BGZF, `cat a.gz b.gz`; RFC 1952 §2.2), their outputs one
/// behind the other in dst.  Success, or the status of the first failing member in file order
/// (BadContainer: bytes behind the last member that are neither zero padding nor a member).
/// `written` receives the bytes of dst that hold output, `members` the members found.
auto decompress_gzip_file(std::span<const std::byte> src, std::span<std::byte> dst, std::size_t* written = nullptr,
                          std::size_t* members = nullptr) -> ContainerStatus;
/// The sum of ISIZE over the BGZF members of src — the dst.size() decompress_gzip_file needs — or
/// nothing when they do not cover the file (a member without the BGZF field, trailing bytes).
auto gzip_file_size(std::span<const std::byte> src) -> std::optional<std::size_t>;

// ---- extension: zip archives -----------------------------------------------------------------
/// One entry of a zip archive (the C ABI's sfb200_zip_entry): where its name and data lie in the
/// archive, its sizes and CRC-32 from the central directory, where zip_extract writes it and what that
/// produced.  `status`: ContainerStatus values.
struct ZipEntry
{
  std::uint64_t name_off, data_off, comp_size, size, dst_off, written;
  std::uint32_t crc32;
  std::uint16_t method, flags, name_len;
  std::uint8_t status;
  std::uint8_t pad[5];
};
static_assert(sizeof(ZipEntry) == 64);
/// The entry table of a zip archive (dst_off packed in directory order), or BadContainer (or the
/// infrastructure failure) for an archive this cannot read.
auto zip_list(std::span<const std::byte> src) -> std::expected<std::vector<ZipEntry>, ContainerStatus>;
/// Extracts the given rows (any subset or order of zip_list's) into dst[dst_off .. + size), checking
/// every entry's CRC-32; status / written are written into the rows.  False on an infrastructure failure.
auto zip_extract(std::span<const std::byte> src, std::span<ZipEntry> entries, std::span<std::byte> dst) -> bool;

// ---- extension: compression to raw DEFLATE, zlib, gzip and BGZF ---------------------------------
/// Compresses src into dst as one raw-DEFLATE, zlib or gzip stream (Auto is Error), the checksum of
/// src computed on the device.  Success, or DstTooSmall (nothing written) when it does not fit;
/// dst.size() >= compress_bound(container, src.size()) always fits.  `written` receives the size.
auto compress_container(std::span<const std::byte> src, std::span<std::byte> dst, Container container,
                        std::size_t* written = nullptr) -> ContainerStatus;
/// Compresses src into dst as a BGZF file (pieces of 65 280 bytes compressed side by side, then the
/// EOF marker); it decodes with decompress_gzip_file, gzip(1) and htslib.  `members` receives the
/// members written, the EOF marker included.
auto compress_bgzf(std::span<const std::byte> src, std::span<std::byte> dst, std::size_t* written = nullptr,
                   std::size_t* members = nullptr) -> ContainerStatus;
/// Compresses src into dst as ONE raw-DEFLATE, zlib or gzip stream at batch speed (Auto is Error): pieces
/// of 65 280 bytes compressed side by side as self-contained blocks, joined bit-exactly.  For inputs up
/// to one piece the output is compress_container's.  Success, or DstTooSmall (nothing written);
/// dst.size() >= compress_parallel_bound(container, src.size()) always fits.
auto compress_parallel(std::span<const std::byte> src, std::span<std::byte> dst, Container container,
                       std::size_t* written = nullptr) -> ContainerStatus;
/// The dst.size() that always holds the output (0 for Auto).
auto compress_bound(Container container, std::size_t src_size) -> std::size_t;
auto compress_bgzf_bound(std::size_t src_size) -> std::size_t;
auto compress_parallel_bound(Container container, std::size_t src_size) -> std::size_t;

// ---- extension: the batched form the GPU is built for ------------------------------------------
/// Stream i reads src[i] and writes dst[i] (host memory); status[i] / written[i] receive its
/// result.  One call = one H2D copy, two kernels, one D2H copy.  Returns false on an
/// infrastructure (CUDA) failure, which is distinct from any per-stream DecompressStatus.
auto decompress_batch(std::span<const std::span<const std::byte>> src,
                      std::span<const std::span<std::byte>> dst, std::span<DecompressStatus> status,
                      std::span<std::size_t> written) -> bool;

}  // namespace starflate
