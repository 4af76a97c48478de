// starflate::zip_list / starflate::zip_extract (C++23 mirror) on one archive:
//   zip_test FILE  ->  "status count status:crc32-of-output(hex) ..." (one pair per entry)
// tests/test_gpu_zip.py compares the line with what the C ABI returns through Python.
#include "src/decompress.hpp"

#include <cstdint>
#include <cstdio>
#include <fstream>
#include <iterator>
#include <vector>

int main(int argc, char** argv)
{
  if (argc != 2) return 2;
  std::ifstream in(argv[1], std::ios::binary);
  const std::vector<char> raw((std::istreambuf_iterator<char>(in)), std::istreambuf_iterator<char>());
  std::vector<std::byte> src(raw.size());
  for (std::size_t i = 0; i < raw.size(); ++i) src[i] = static_cast<std::byte>(raw[i]);
  auto rows = starflate::zip_list(src);
  if (!rows) {
    std::printf("%d 0\n", static_cast<int>(rows.error()));
    return 0;
  }
  std::size_t total = 0;
  for (const auto& r : *rows) total += r.size;
  std::vector<std::byte> dst(total);
  if (!starflate::zip_extract(src, *rows, dst)) return 1;
  std::printf("0 %zu", rows->size());
  for (const auto& r : *rows) {
    std::uint32_t crc = 0xffffffffu;
    for (std::size_t i = r.dst_off; i < r.dst_off + r.written; ++i) {
      crc ^= static_cast<std::uint32_t>(dst[i]);
      for (int k = 0; k < 8; ++k) crc = (crc & 1u) ? (crc >> 1) ^ 0xedb88320u : crc >> 1;
    }
    std::printf(" %d:%08x", static_cast<int>(r.status), ~crc);
  }
  std::printf("\n");
  return 0;
}
