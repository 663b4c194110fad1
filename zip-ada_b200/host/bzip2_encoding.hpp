// C++ mirror of the reference's generic `BZip2.Encoding.Encode` (zip_lib/bzip2-encoding.ads:47-56)
// above the C ABI of include/b2gpu.h.  Same shape as the Ada generic: three callbacks for the
// bytes, `option` and `size_hint` as arguments; exceptions thrown by the callbacks propagate and
// the handle goes back to the pool on every path (cf. bzip2-encoding.adb:1377-1381).  No CPU fallback.
//
// Handles are pooled per (block size, device): Zip.Create calls Encode once per archive entry
// (zip-create.adb:253-265) and creating a handle (CUDA streams, tables, workspaces) per entry would
// dominate small entries.  Concurrent callers each take their own handle (doc/zipada.txt:26).
#pragma once
#include <cstdint>
#include <map>
#include <mutex>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../../include/b2gpu.h"

namespace bzip2_encoding {

enum Compression_Option { block_100k = B2_BLOCK_100K, block_400k = B2_BLOCK_400K, block_900k = B2_BLOCK_900K };
using Stream_Size_Type = int64_t;
constexpr Stream_Size_Type unknown_size = B2_UNKNOWN_SIZE;

struct b2gpu_error : std::runtime_error { using std::runtime_error::runtime_error; };

class Handle_Pool {
 public:
  static Handle_Pool &instance() { static Handle_Pool p; return p; }
  b2_encoder *take(int level, int device) {
    {
      std::lock_guard<std::mutex> lk(mu_);
      auto &v = idle_[{level, device}];
      if (!v.empty()) { b2_encoder *e = v.back(); v.pop_back(); return e; }
    }
    b2_encoder *e = nullptr;
    if (b2_create(level, device, &e) != B2_OK) throw b2gpu_error(std::string("b2_create: ") + b2_last_error());
    created_++;
    return e;
  }
  void give(int level, int device, b2_encoder *e) {
    std::lock_guard<std::mutex> lk(mu_);
    idle_[{level, device}].push_back(e);
  }
  uint64_t created() const { return created_; }
  void clear() {
    std::lock_guard<std::mutex> lk(mu_);
    for (auto &kv : idle_) for (b2_encoder *e : kv.second) b2_destroy(e);
    idle_.clear();
  }
  ~Handle_Pool() { clear(); }
 private:
  std::mutex mu_;
  std::map<std::pair<int, int>, std::vector<b2_encoder *>> idle_;
  uint64_t created_ = 0;
};

// generic
//   with function Read_Byte return Byte; with function More_Bytes return Boolean;
//   with procedure Write_Byte (b : Byte);
// procedure Encode (option := block_900k; size_hint := unknown_size);
template <class ReadByte, class MoreBytes, class WriteByte>
void Encode(ReadByte Read_Byte, MoreBytes More_Bytes, WriteByte Write_Byte,
            Compression_Option option = block_900k, Stream_Size_Type size_hint = unknown_size, int device = 0) {
  std::vector<uint8_t> in;
  while (More_Bytes()) in.push_back(Read_Byte());          // may throw (User_abort): nothing to release yet
  std::vector<uint8_t> out(b2_bound(in.size()) + 1024 * (in.size() / 40000 + 16));
  uint64_t out_len = 0;
  {
    b2_encoder *enc = Handle_Pool::instance().take((int)option, device);
    struct Guard { int l, d; b2_encoder *e; ~Guard() { Handle_Pool::instance().give(l, d, e); } } guard{(int)option, device, enc};
    if (b2_encode_stream(enc, in.data(), in.size(), size_hint, out.data(), out.size(), &out_len) != B2_OK)
      throw b2gpu_error(std::string("b2_encode_stream: ") + b2_last_error());
  }
  for (uint64_t i = 0; i < out_len; i++) Write_Byte(out[i]);  // may throw (Compression_inefficient): the handle is back in the pool
}

// The same Encode, streaming: bytes are read into a 16 MiB staging buffer and handed to the device a buffer at a
// time (b2_stream_write), and the bytes that are final go out through Write_Byte after every buffer, so memory does not
// grow with the input.  Byte-identical to Encode.  An exception out of a callback aborts the handle's stream
// (b2_stream_abort) before it propagates; the handle goes back to the pool.  window_bytes: see b2_stream_begin.
template <class ReadByte, class MoreBytes, class WriteByte>
void Encode_Streamed(ReadByte Read_Byte, MoreBytes More_Bytes, WriteByte Write_Byte,
                     Compression_Option option = block_900k, Stream_Size_Type size_hint = unknown_size, int device = 0,
                     uint64_t window_bytes = 0) {
  b2_encoder *enc = Handle_Pool::instance().take((int)option, device);
  struct Guard { int l, d; b2_encoder *e; ~Guard() { b2_stream_abort(e); Handle_Pool::instance().give(l, d, e); } } guard{(int)option, device, enc};
  if (b2_stream_begin(enc, size_hint, window_bytes) != B2_OK) throw b2gpu_error(std::string("b2_stream_begin: ") + b2_last_error());
  std::vector<uint8_t> in(16u << 20), out;
  uint64_t out_len = 0;
  for (bool more = true; more;) {
    size_t n = 0;
    while (n < in.size() && (more = More_Bytes())) in[n++] = Read_Byte();
    out.resize(b2_stream_bound(enc, n));
    if (b2_stream_write(enc, in.data(), n, out.data(), out.size(), &out_len) != B2_OK)
      throw b2gpu_error(std::string("b2_stream_write: ") + b2_last_error());
    for (uint64_t i = 0; i < out_len; i++) Write_Byte(out[i]);
  }
  out.resize(b2_stream_bound(enc, 0));
  if (b2_stream_end(enc, out.data(), out.size(), &out_len) != B2_OK) throw b2gpu_error(std::string("b2_stream_end: ") + b2_last_error());
  for (uint64_t i = 0; i < out_len; i++) Write_Byte(out[i]);
}

}  // namespace bzip2_encoding
