// starflate::compress_parallel (C++23 mirror) on one file:
//   compress_parallel_test IN raw|zlib|gzip OUT  ->  OUT holds the stream; prints "status written bound"
// tests/test_gpu_compress_parallel.py compares OUT with what the C ABI writes through Python.
#include "src/decompress.hpp"

#include <cstdint>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iterator>
#include <vector>

int main(int argc, char** argv)
{
  if (argc != 4) return 2;
  std::ifstream in(argv[1], std::ios::binary);
  const std::vector<char> raw((std::istreambuf_iterator<char>(in)), std::istreambuf_iterator<char>());
  std::vector<std::byte> src(raw.size());
  for (std::size_t i = 0; i < raw.size(); ++i) src[i] = static_cast<std::byte>(raw[i]);
  const auto container = std::strcmp(argv[2], "zlib") == 0   ? starflate::Container::Zlib
                         : std::strcmp(argv[2], "gzip") == 0 ? starflate::Container::Gzip
                                                             : starflate::Container::Raw;
  const std::size_t bound = starflate::compress_parallel_bound(container, src.size());
  std::vector<std::byte> dst(bound);
  std::size_t written = 0;
  const auto st = starflate::compress_parallel(src, dst, container, &written);
  std::ofstream out(argv[3], std::ios::binary);
  out.write(reinterpret_cast<const char*>(dst.data()), static_cast<std::streamsize>(written));
  std::printf("%d %zu %zu\n", static_cast<int>(st), written, bound);
  return 0;
}
