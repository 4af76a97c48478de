// starflate::decompress_gzip_file / starflate::gzip_file_size (C++23 mirror) on one file:
//   gzip_file_test FILE DST_CAP  ->  "status written members size|none crc32-of-output(hex)"
// tests/test_gpu_gzip_file.py compares the line with what the C ABI returns through Python.
#include "src/decompress.hpp"

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iterator>
#include <vector>

int main(int argc, char** argv)
{
  if (argc != 3) return 2;
  std::ifstream in(argv[1], std::ios::binary);
  const std::vector<char> raw((std::istreambuf_iterator<char>(in)), std::istreambuf_iterator<char>());
  std::vector<std::byte> src(raw.size());
  for (std::size_t i = 0; i < raw.size(); ++i) src[i] = static_cast<std::byte>(raw[i]);
  std::vector<std::byte> dst(std::strtoull(argv[2], nullptr, 10));
  std::size_t written = 0, members = 0;
  const auto st = starflate::decompress_gzip_file(src, dst, &written, &members);
  const auto size = starflate::gzip_file_size(src);
  std::uint32_t crc = 0xffffffffu;
  for (std::size_t i = 0; i < written; ++i) {
    crc ^= static_cast<std::uint32_t>(dst[i]);
    for (int k = 0; k < 8; ++k) crc = (crc & 1u) ? (crc >> 1) ^ 0xedb88320u : crc >> 1;
  }
  crc = ~crc;
  if (size) std::printf("%d %zu %zu %zu %08x\n", static_cast<int>(st), written, members, *size, crc);
  else std::printf("%d %zu %zu none %08x\n", static_cast<int>(st), written, members, crc);
  return 0;
}
