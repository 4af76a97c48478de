// starflate::compress_container / starflate::compress_bgzf (C++23 mirror) on one file:
//   compress_test IN raw|zlib|gzip|bgzf OUT  ->  OUT holds the output; prints "status written members"
// tests/test_gpu_compress_container.py compares OUT with what the C ABI writes through Python.
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
  const bool bgzf = std::strcmp(argv[2], "bgzf") == 0;
  const auto container = std::strcmp(argv[2], "zlib") == 0   ? starflate::Container::Zlib
                         : std::strcmp(argv[2], "gzip") == 0 ? starflate::Container::Gzip
                                                             : starflate::Container::Raw;
  std::vector<std::byte> dst(bgzf ? starflate::compress_bgzf_bound(src.size())
                                  : starflate::compress_bound(container, src.size()));
  std::size_t written = 0, members = 0;
  const auto st = bgzf ? starflate::compress_bgzf(src, dst, &written, &members)
                       : starflate::compress_container(src, dst, container, &written);
  std::ofstream out(argv[3], std::ios::binary);
  out.write(reinterpret_cast<const char*>(dst.data()), static_cast<std::streamsize>(written));
  std::printf("%d %zu %zu\n", static_cast<int>(st), written, members);
  return 0;
}
