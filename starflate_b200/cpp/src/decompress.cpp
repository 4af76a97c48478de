// C++23 host side of the drop-in interface: forwards to the CUDA library through the C ABI.
#include "src/decompress.hpp"

#include "starflate_b200.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <mutex>
#include <vector>

namespace starflate {
namespace {

// The reference's decompress() is re-entrant: callers run it on as many threads as they like
// (one stream per core).  A CUDA context object serves one call at a time, so the mirror keeps a
// small POOL of them — created on first use, at most STARFLATE_B200_CONTEXTS (default 4), spread
// round-robin over the devices named in STARFLATE_B200_DEVICES ("0,1,..."; default: device
// STARFLATE_B200_DEVICE or 0) — and a call borrows one for its duration.  More threads than
// contexts wait their turn; the GPU is shared by all of them either way.
class ContextPool {
 public:
  class Lease {
   public:
    Lease(ContextPool& p, sfb200_ctx* c) : pool_(p), ctx_(c) {}
    Lease(const Lease&) = delete;
    auto operator=(const Lease&) -> Lease& = delete;
    ~Lease() { pool_.give_back(ctx_); }
    auto get() const -> sfb200_ctx* { return ctx_; }

   private:
    ContextPool& pool_;
    sfb200_ctx* ctx_;
  };

  auto borrow() -> Lease
  {
    std::unique_lock lock{m_};
    for (;;) {
      if (!free_.empty()) {
        sfb200_ctx* c = free_.back();
        free_.pop_back();
        return Lease{*this, c};
      }
      if (created_ < limit()) {
        const int device = next_device();
        ++created_;
        lock.unlock();
        sfb200_ctx* c = nullptr;
        const int rc = sfb200_create(device, &c);
        if (rc != SFB200_RC_OK) {
          std::fprintf(stderr,
                       "starflate_b200: cannot create a CUDA context on device %d (rc=%d). "
                       "This library has no CPU decode path.\n",
                       device, rc);
          std::abort();
        }
        return Lease{*this, c};
      }
      cv_.wait(lock);
    }
  }

 private:
  void give_back(sfb200_ctx* c)
  {
    {
      const std::lock_guard lock{m_};
      free_.push_back(c);
    }
    cv_.notify_one();
  }
  static auto limit() -> int
  {
    static const int n = [] {
      const char* e = std::getenv("STARFLATE_B200_CONTEXTS");
      const int v = e ? std::atoi(e) : 4;
      return v > 0 ? v : 1;
    }();
    return n;
  }
  auto next_device() -> int
  {
    static const std::vector<int> devices = [] {
      std::vector<int> d;
      if (const char* e = std::getenv("STARFLATE_B200_DEVICES")) {
        for (const char* p = e; *p;) {
          char* end = nullptr;
          const long v = std::strtol(p, &end, 10);
          if (end == p) break;
          d.push_back(static_cast<int>(v));
          p = *end == ',' ? end + 1 : end;
        }
      }
      if (d.empty()) {
        const char* e = std::getenv("STARFLATE_B200_DEVICE");
        d.push_back(e ? std::atoi(e) : 0);
      }
      return d;
    }();
    return devices[static_cast<std::size_t>(created_) % devices.size()];
  }

  std::mutex m_;
  std::condition_variable cv_;
  std::vector<sfb200_ctx*> free_;  // (contexts live as long as the process: the reference has no teardown either)
  int created_ = 0;
};

auto pool() -> ContextPool&
{
  static ContextPool p;
  return p;
}

// An infrastructure failure has no DecompressStatus of its own.  Running out of device memory is
// reported as the reference's catch-all, DecompressStatus::Error (the caller can retry with less
// in flight); anything else — a lost device, a driver error — ends the process, loudly: there is no
// CPU path to fall back to.
auto infra(const char* what, int rc, sfb200_ctx* ctx) -> DecompressStatus
{
  if (rc == SFB200_RC_OUT_OF_MEMORY) return DecompressStatus::Error;
  std::fprintf(stderr, "starflate_b200: %s failed (rc=%d): %s\n", what, rc, sfb200_last_error(ctx));
  std::abort();
}

}  // namespace

namespace detail {

auto read_header(huffman::bit_span& compressed_bits) -> std::expected<BlockHeader, DecompressStatus>
{
  if (std::ranges::size(compressed_bits) < 3) return std::unexpected{DecompressStatus::InvalidBlockHeader};
  auto it = compressed_bits.begin();
  const bool final_block = static_cast<bool>(*it++);
  unsigned type = static_cast<bool>(*it++) ? 1u : 0u;
  type |= static_cast<bool>(*it++) ? 2u : 0u;
  if (type > 2) return std::unexpected{DecompressStatus::InvalidBlockHeader};
  compressed_bits.consume(3);
  return BlockHeader{final_block, static_cast<BlockType>(type)};
}

void copy_from_before(std::uint16_t distance, std::span<std::byte>::iterator dst, std::uint16_t n)
{
  // byte-serial forward copy: by definition what the LZ77 reference string means (RFC 1951
  // §3.2.3); the device does the same with a period-`distance` gather (csrc/lz_warp.cuh)
  for (std::uint16_t i = 0; i < n; ++i, ++dst) *dst = *(dst - distance);
}

}  // namespace detail

auto decompress(std::span<const std::byte> src, std::span<std::byte> dst) -> DecompressStatus
{
  std::uint8_t status = 0;
  const auto lease = pool().borrow();
  const int rc = sfb200_decompress(lease.get(), reinterpret_cast<const std::uint8_t*>(src.data()), src.size(),
                                   reinterpret_cast<std::uint8_t*>(dst.data()), dst.size(), &status, nullptr);
  if (rc != SFB200_RC_OK) return infra("sfb200_decompress", rc, lease.get());
  return static_cast<DecompressStatus>(status);
}

auto decompressed_size(std::span<const std::byte> src) -> std::expected<std::size_t, DecompressStatus>
{
  std::uint8_t status = 0;
  std::uint64_t size = 0;
  const auto lease = pool().borrow();
  const int rc = sfb200_decompressed_size(lease.get(), reinterpret_cast<const std::uint8_t*>(src.data()), src.size(),
                                          &status, &size);
  if (rc != SFB200_RC_OK) return std::unexpected{infra("sfb200_decompressed_size", rc, lease.get())};
  if (status != 0) return std::unexpected{static_cast<DecompressStatus>(status)};
  return static_cast<std::size_t>(size);
}

auto decompress_container(std::span<const std::byte> src, std::span<std::byte> dst, Container container,
                          std::size_t* written) -> ContainerStatus
{
  std::uint8_t status = 0;
  std::uint64_t wr = 0;
  const auto lease = pool().borrow();
  const int rc = sfb200_decompress_container(lease.get(), static_cast<int>(container),
                                             reinterpret_cast<const std::uint8_t*>(src.data()), src.size(),
                                             reinterpret_cast<std::uint8_t*>(dst.data()), dst.size(), &status, &wr);
  if (rc != SFB200_RC_OK) return static_cast<ContainerStatus>(infra("sfb200_decompress_container", rc, lease.get()));
  if (written) *written = static_cast<std::size_t>(wr);
  return static_cast<ContainerStatus>(status);
}

auto decompress_gzip_file(std::span<const std::byte> src, std::span<std::byte> dst, std::size_t* written,
                          std::size_t* members) -> ContainerStatus
{
  std::uint8_t status = 0;
  std::uint64_t wr = 0, nm = 0;
  const auto lease = pool().borrow();
  const int rc = sfb200_decompress_gzip_file(lease.get(), reinterpret_cast<const std::uint8_t*>(src.data()), src.size(),
                                             reinterpret_cast<std::uint8_t*>(dst.data()), dst.size(), &status, &wr, &nm);
  if (rc != SFB200_RC_OK) return static_cast<ContainerStatus>(infra("sfb200_decompress_gzip_file", rc, lease.get()));
  if (written) *written = static_cast<std::size_t>(wr);
  if (members) *members = static_cast<std::size_t>(nm);
  return static_cast<ContainerStatus>(status);
}

auto gzip_file_size(std::span<const std::byte> src) -> std::optional<std::size_t>
{
  std::uint64_t size = 0;
  int complete = 0;
  const auto lease = pool().borrow();
  const int rc = sfb200_gzip_file_size(lease.get(), reinterpret_cast<const std::uint8_t*>(src.data()), src.size(), &size,
                                       nullptr, &complete);
  if (rc != SFB200_RC_OK) {
    infra("sfb200_gzip_file_size", rc, lease.get());
    return std::nullopt;
  }
  if (!complete) return std::nullopt;
  return static_cast<std::size_t>(size);
}

auto zip_list(std::span<const std::byte> src) -> std::expected<std::vector<ZipEntry>, ContainerStatus>
{
  static_assert(sizeof(ZipEntry) == sizeof(sfb200_zip_entry));
  std::uint8_t status = 0;
  std::uint64_t count = 0;
  const auto lease = pool().borrow();
  const auto* s = reinterpret_cast<const std::uint8_t*>(src.data());
  int rc = sfb200_zip_list(lease.get(), s, src.size(), nullptr, 0, &status, &count, nullptr);
  std::vector<ZipEntry> rows;
  if (rc == SFB200_RC_OK && status == 0 && count) {
    rows.resize(count);
    rc = sfb200_zip_list(lease.get(), s, src.size(), reinterpret_cast<sfb200_zip_entry*>(rows.data()), count, &status,
                         &count, nullptr);
  }
  if (rc != SFB200_RC_OK) return std::unexpected{static_cast<ContainerStatus>(infra("sfb200_zip_list", rc, lease.get()))};
  if (status != 0) return std::unexpected{static_cast<ContainerStatus>(status)};
  return rows;
}

auto zip_extract(std::span<const std::byte> src, std::span<ZipEntry> entries, std::span<std::byte> dst) -> bool
{
  const auto lease = pool().borrow();
  const int rc = sfb200_zip_extract(lease.get(), reinterpret_cast<const std::uint8_t*>(src.data()), src.size(),
                                    reinterpret_cast<sfb200_zip_entry*>(entries.data()), entries.size(),
                                    reinterpret_cast<std::uint8_t*>(dst.data()), dst.size());
  if (rc != SFB200_RC_OK) {
    infra("sfb200_zip_extract", rc, lease.get());
    return false;
  }
  return true;
}

auto compress_container(std::span<const std::byte> src, std::span<std::byte> dst, Container container,
                        std::size_t* written) -> ContainerStatus
{
  if (container == Container::Auto) return ContainerStatus::Error;
  std::uint8_t status = 0;
  std::uint64_t wr = 0;
  const auto lease = pool().borrow();
  const int rc = sfb200_compress_container(lease.get(), static_cast<int>(container),
                                           reinterpret_cast<const std::uint8_t*>(src.data()), src.size(),
                                           reinterpret_cast<std::uint8_t*>(dst.data()), dst.size(), &status, &wr);
  if (rc != SFB200_RC_OK) return static_cast<ContainerStatus>(infra("sfb200_compress_container", rc, lease.get()));
  if (written) *written = static_cast<std::size_t>(wr);
  return static_cast<ContainerStatus>(status);
}

auto compress_bgzf(std::span<const std::byte> src, std::span<std::byte> dst, std::size_t* written,
                   std::size_t* members) -> ContainerStatus
{
  std::uint8_t status = 0;
  std::uint64_t wr = 0, nm = 0;
  const auto lease = pool().borrow();
  const int rc = sfb200_compress_bgzf(lease.get(), reinterpret_cast<const std::uint8_t*>(src.data()), src.size(),
                                      reinterpret_cast<std::uint8_t*>(dst.data()), dst.size(), &status, &wr, &nm);
  if (rc != SFB200_RC_OK) return static_cast<ContainerStatus>(infra("sfb200_compress_bgzf", rc, lease.get()));
  if (written) *written = static_cast<std::size_t>(wr);
  if (members) *members = static_cast<std::size_t>(nm);
  return static_cast<ContainerStatus>(status);
}

auto compress_parallel(std::span<const std::byte> src, std::span<std::byte> dst, Container container,
                       std::size_t* written) -> ContainerStatus
{
  if (container == Container::Auto) return ContainerStatus::Error;
  std::uint8_t status = 0;
  std::uint64_t wr = 0;
  const auto lease = pool().borrow();
  const int rc = sfb200_compress_parallel(lease.get(), static_cast<int>(container),
                                          reinterpret_cast<const std::uint8_t*>(src.data()), src.size(),
                                          reinterpret_cast<std::uint8_t*>(dst.data()), dst.size(), &status, &wr);
  if (rc != SFB200_RC_OK) return static_cast<ContainerStatus>(infra("sfb200_compress_parallel", rc, lease.get()));
  if (written) *written = static_cast<std::size_t>(wr);
  return static_cast<ContainerStatus>(status);
}

auto compress_bound(Container container, std::size_t src_size) -> std::size_t
{
  return static_cast<std::size_t>(sfb200_compress_container_bound(static_cast<int>(container), src_size));
}

auto compress_bgzf_bound(std::size_t src_size) -> std::size_t
{
  return static_cast<std::size_t>(sfb200_compress_bgzf_bound(src_size));
}

auto compress_parallel_bound(Container container, std::size_t src_size) -> std::size_t
{
  return static_cast<std::size_t>(sfb200_compress_parallel_bound(static_cast<int>(container), src_size));
}

auto decompress_batch(std::span<const std::span<const std::byte>> src,
                      std::span<const std::span<std::byte>> dst, std::span<DecompressStatus> status,
                      std::span<std::size_t> written) -> bool
{
  const std::size_t n = src.size();
  if (dst.size() != n || status.size() != n || (!written.empty() && written.size() != n)) return false;
  if (n == 0) return true;
  // pack into the flat layout of the C ABI (16-byte aligned regions)
  std::vector<std::uint64_t> so(n), sl(n), dof(n), dc(n), wr(n);
  std::uint64_t stot = 0, dtot = 0;
  for (std::size_t i = 0; i < n; ++i) {
    so[i] = stot;
    sl[i] = src[i].size();
    stot += (sl[i] + 15) & ~std::uint64_t{15};
    dof[i] = dtot;
    dc[i] = dst[i].size();
    dtot += (dc[i] + 31) & ~std::uint64_t{31};
  }
  std::vector<std::uint8_t> sbuf(stot + 16), dbuf(dtot + 32), st(n);
  for (std::size_t i = 0; i < n; ++i) {
    if (sl[i]) std::memcpy(sbuf.data() + so[i], src[i].data(), sl[i]);
    if (dc[i]) std::memcpy(dbuf.data() + dof[i], dst[i].data(), dc[i]);
  }
  const auto lease = pool().borrow();
  const int rc = sfb200_decompress_batch_host(lease.get(), sbuf.data(), sbuf.size(), so.data(), sl.data(),
                                              dbuf.data(), dbuf.size(), dof.data(), dc.data(), st.data(),
                                              wr.data(), n);
  if (rc != SFB200_RC_OK) return false;
  for (std::size_t i = 0; i < n; ++i) {
    if (dc[i]) std::memcpy(dst[i].data(), dbuf.data() + dof[i], dc[i]);
    status[i] = static_cast<DecompressStatus>(st[i]);
    if (!written.empty()) written[i] = static_cast<std::size_t>(wr[i]);
  }
  return true;
}

}  // namespace starflate
