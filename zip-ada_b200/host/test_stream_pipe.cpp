// stdin -> stdout through Encode_Streamed on a pooled handle: a BZip2 stream of a pipe, written while it is read.
// Usage: test_stream_pipe <size_hint> [window_bytes]
//        test_stream_pipe --throw-after <n> <size_hint> [window_bytes]
//   The second form reads all of stdin, encodes it once with Write_Byte throwing after n bytes, then encodes it again
//   on the same pooled handle to stdout, and prints "created=<handles created> thrown=<k>" on stderr.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "bzip2_encoding.hpp"

struct Stop {};

int main(int argc, char **argv) {
  int a = 1;
  long long throw_after = -1;
  if (argc > 2 && std::strcmp(argv[1], "--throw-after") == 0) { throw_after = std::atoll(argv[2]); a = 3; }
  if (argc <= a) return 2;
  const int64_t hint = std::atoll(argv[a]);
  const uint64_t window = argc > a + 1 ? std::strtoull(argv[a + 1], nullptr, 10) : 0;
  std::vector<uint8_t> obuf;
  auto put = [&](uint8_t b) {
    obuf.push_back(b);
    if (obuf.size() == (1u << 20)) { std::fwrite(obuf.data(), 1, obuf.size(), stdout); obuf.clear(); }
  };
  if (throw_after < 0) {
    std::vector<uint8_t> ibuf(1u << 20);
    size_t have = 0, pos = 0;
    auto more = [&]() {
      if (pos < have) return true;
      have = std::fread(ibuf.data(), 1, ibuf.size(), stdin); pos = 0;
      return have > 0;
    };
    bzip2_encoding::Encode_Streamed([&]() { return ibuf[pos++]; }, more, put, bzip2_encoding::block_900k, hint, 0, window);
  } else {
    std::vector<uint8_t> in;
    std::vector<uint8_t> chunk(1u << 20);
    for (size_t k; (k = std::fread(chunk.data(), 1, chunk.size(), stdin)) > 0;) in.insert(in.end(), chunk.begin(), chunk.begin() + k);
    size_t pos = 0;
    long long written = 0;
    int thrown = 0;
    try {
      bzip2_encoding::Encode_Streamed([&]() { return in[pos++]; }, [&]() { return pos < in.size(); },
                                      [&](uint8_t) { if (++written > throw_after) throw Stop(); }, bzip2_encoding::block_900k, hint, 0,
                                      window);
    } catch (const Stop &) {
      thrown++;
    }
    pos = 0;
    bzip2_encoding::Encode_Streamed([&]() { return in[pos++]; }, [&]() { return pos < in.size(); }, put, bzip2_encoding::block_900k,
                                    hint, 0, window);
    std::fprintf(stderr, "created=%llu thrown=%d\n", (unsigned long long)bzip2_encoding::Handle_Pool::instance().created(), thrown);
  }
  std::fwrite(obuf.data(), 1, obuf.size(), stdout);
  return 0;
}
