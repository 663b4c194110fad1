// The Zip records of an archive written by Zip.Create with BZip2 entries, host only: local headers
// (zip-create.adb:194-297, zip-headers.adb:243-277), central headers (zip-headers.adb:167-192), the Zip64
// end record and locator and the end record (zip-create.adb:645-756), and Check_Size (:161-179).
// b2_zip_create lays out a whole catalogue in one go; the b2_zip_* writer lays it out one group of entries
// after the other.  Both use ZipLayout, so the bytes of an archive do not depend on how it was cut into groups.
// Plain C++17 (tests/zip_layout_check.cpp compiles it with g++).
#pragma once
#include <cstdint>
#include <string>
#include <vector>

namespace b2zip {

struct ByteSink {                                   // little-endian fields (zip-headers.adb:54-70)
  std::vector<uint8_t> b;
  void u16le(uint32_t v) { b.push_back((uint8_t)v); b.push_back((uint8_t)(v >> 8)); }
  void u32le(uint64_t v) { for (int k = 0; k < 4; k++) b.push_back((uint8_t)(v >> (8 * k))); }
  void u64le(uint64_t v) { for (int k = 0; k < 8; k++) b.push_back((uint8_t)(v >> (8 * k))); }
  void sig(uint8_t c1, uint8_t c2) { b.push_back(0x50); b.push_back(0x4B); b.push_back(c1); b.push_back(c2); }
  void str(const std::string &s) { b.insert(b.end(), s.begin(), s.end()); }
};

// Entry names: back slashes become forward slashes (Unixify, zip-create.adb:180-192).
inline std::string unixify(const char *p, size_t n) {
  std::string s(p, p + n);
  for (char &c : s) if (c == '\\') c = '/';
  return s;
}

struct ZipEntryRecord {
  std::string name;
  uint64_t usize, csize, offset;
  uint32_t crc, time, ext_attr;
  uint16_t flag, method;
};

// What Add_Stream and Finish leave in the output stream.  Per entry: open_entry before the entry is compressed
// (Check_Size on its size, its offset, the length of its local header), close_entry once its CRC, method and
// compressed size are known.  Then finish.
class ZipLayout {
 public:
  static constexpr uint64_t four_gib = 1ull << 32, max_size = 0x1FFFFFFFFFFFFFFFull;
  static constexpr uint64_t check_margin = 22 + 56 + 20 + 65536 + 10;     // Check_Size (:161-179)
  static constexpr uint32_t default_time = 16789u * 65536u;               // Zip_Streams.default_time
  static constexpr uint32_t unicode_name = 1u, read_only = 2u;             // B2_ZIP_UNICODE_NAME / B2_ZIP_READ_ONLY

  uint64_t pos = 0;                                 // archive bytes laid out so far
  bool zip64 = false;
  std::vector<ZipEntryRecord> cat;

  // The local header's Zip64 extension is decided BEFORE compression, with compressed size = size (:233-243).
  static bool local_ext(uint64_t usize, uint64_t offset) { return usize >= 0xFFFFFFFFull || offset >= 0xFFFFFFFFull; }
  static uint64_t local_header_bytes(size_t name_len, bool ext) { return 30 + name_len + (ext ? 20 : 0); }
  // Central header with the Zip64 extension, the largest it can be.
  static uint64_t central_header_max(size_t name_len) { return 46 + name_len + 28; }
  static constexpr uint64_t end_records_max = 56 + 20 + 22;

  // false: Zip_Capacity_Exceeded.
  bool open_entry(uint64_t usize, size_t name_len, uint64_t *offset, uint64_t *header_bytes) {
    if (check_size(usize)) return false;
    *offset = pos;
    *header_bytes = local_header_bytes(name_len, local_ext(usize, pos));
    return true;
  }

  // The local header of the entry opened last (written to `hdr`, which is replaced); the entry's payload of `csize`
  // bytes follows it.  method: 12 = BZip2, 0 = Store.
  void close_entry(const std::string &name, uint64_t usize, uint64_t csize, uint32_t crc, uint32_t time, uint32_t flags,
                   uint16_t method, std::vector<uint8_t> &hdr) {
    ZipEntryRecord c;
    c.name = name; c.usize = usize; c.csize = csize; c.offset = pos; c.crc = crc; c.time = time; c.method = method;
    c.flag = (flags & unicode_name) ? 0x0800 : 0;                          // Language_Encoding_Flag_Bit (:222-224)
    c.ext_attr = (flags & read_only) ? 1u : 0u;                            // (:228-230)
    const bool ext = local_ext(usize, c.offset);
    ByteSink h;
    h.sig(3, 4);
    h.u16le(10); h.u16le(c.flag); h.u16le(c.method); h.u32le(c.time); h.u32le(c.crc);
    if (ext) { h.u32le(0xFFFFFFFFu); h.u32le(0xFFFFFFFFu); } else { h.u32le(c.csize); h.u32le(c.usize); }
    h.u16le((uint32_t)name.size()); h.u16le(ext ? 20 : 0);
    h.str(name);
    if (ext) { h.u16le(1); h.u16le(16); h.u64le(c.usize); h.u64le(c.csize); }
    pos += h.b.size() + csize;
    hdr.swap(h.b);
    cat.push_back(std::move(c));
  }

  // Finish: central directory, Zip64 end record and locator when needed, end record.  false: Zip_Capacity_Exceeded.
  bool finish(std::vector<uint8_t> &out) {
    ByteSink d;
    const uint64_t n_entries = cat.size();
    const uint64_t cd_offset = pos;
    uint64_t cd_size = 0;
    if (!zip64 && n_entries >= 65535u) zip64 = true;                       // too many entries for Zip_32 (:680-685)
    for (const ZipEntryRecord &c : cat) {
      const bool ext = c.csize >= 0xFFFFFFFFull || c.usize >= 0xFFFFFFFFull || c.offset >= 0xFFFFFFFFull;
      if (ext) zip64 = true;
      d.sig(1, 2);
      d.u16le(23); d.u16le(10); d.u16le(c.flag); d.u16le(c.method); d.u32le(c.time); d.u32le(c.crc);
      d.u32le(ext ? 0xFFFFFFFFull : c.csize); d.u32le(ext ? 0xFFFFFFFFull : c.usize);
      d.u16le((uint32_t)c.name.size()); d.u16le(ext ? 28 : 0);
      d.u16le(0); d.u16le(0); d.u16le(0); d.u32le(c.ext_attr);
      d.u32le(ext ? 0xFFFFFFFFull : c.offset);
      d.str(c.name);
      if (ext) { d.u16le(1); d.u16le(24); d.u64le(c.usize); d.u64le(c.csize); d.u64le(c.offset); }
      cd_size += 46 + c.name.size() + (ext ? 28 : 0);
    }
    if (n_entries && check_size(cd_offset + cd_size + 1)) return false;
    uint64_t tot = n_entries, dtot = n_entries, cds = cd_size, cdo = cd_offset;
    if (zip64) {
      d.sig(6, 6);
      d.u64le(44); d.u16le(0x2D); d.u16le(0x2D); d.u32le(0); d.u32le(0); d.u64le(n_entries); d.u64le(n_entries); d.u64le(cd_size); d.u64le(cd_offset);
      d.sig(6, 7);
      d.u32le(0); d.u64le(cd_offset + cd_size); d.u32le(1);
      tot = dtot = 0xFFFF; cds = 0xFFFFFFFFull; cdo = 0xFFFFFFFFull;
    }
    d.sig(5, 6);
    d.u16le(0); d.u16le(0); d.u16le((uint32_t)dtot); d.u16le((uint32_t)tot); d.u32le(cds); d.u32le(cdo); d.u16le(0);
    pos += d.b.size();
    out.swap(d.b);
    return true;
  }

 private:
  int check_size(uint64_t value) {
    if (!zip64 && value >= four_gib - check_margin) {
      zip64 = true;
      if (value >= max_size - check_margin) return 1;
    }
    return 0;
  }
};

// ---- Zip CRC-32 of a concatenation from the CRCs of its parts (GF(2) polynomial arithmetic, reflected
// polynomial 0xEDB88320).  crc32_combine (crc (A), crc (B), |B|) = crc (A & B), crc being Init + Update + Final
// (zip-crc_crypto.adb:31-61).

// a * b mod P; bit 31 is x^0.
inline uint32_t crc_multmodp(uint32_t a, uint32_t b) {
  uint32_t m = 1u << 31, p = 0;
  for (;;) {
    if (a & m) {
      p ^= b;
      if ((a & (m - 1)) == 0) break;
    }
    m >>= 1;
    b = (b & 1) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
  }
  return p;
}

// x^(8 n) mod P
inline uint32_t crc_xpow8n(uint64_t n) {
  uint32_t sq = 1u << 30;                           // x^1, squared up to x^(2^k)
  for (int k = 0; k < 3; k++) sq = crc_multmodp(sq, sq);
  uint32_t p = 1u << 31;
  for (; n; n >>= 1) {
    if (n & 1) p = crc_multmodp(sq, p);
    sq = crc_multmodp(sq, sq);
  }
  return p;
}

inline uint32_t crc32_combine(uint32_t crc1, uint32_t crc2, uint64_t len2) {
  return crc_multmodp(crc_xpow8n(len2), crc1) ^ crc2;
}

}  // namespace b2zip
