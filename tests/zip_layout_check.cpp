// Host checks of zip-ada_b200/csrc/b2_zip_layout.h, driven by tests/test_zip_writer_layout.py.
//
//   zip_layout_check layout FILE   FILE: lines "name usize csize"; usize / csize are synthetic (no data), csize >= usize
//                                  means Store; entry k has CRC 0x12345678 + k, the default time and flags k mod 4.
//                                  Prints every local header and the central directory with the end records as
//                                  "archive offset hex" lines.
//   zip_layout_check crc FILE k1 k2 ...   Zip CRC-32 of FILE from the CRCs of the parts [0, k1), [k1, k2), ... and
//                                  crc32_combine; prints it in decimal.
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <sstream>
#include <string>
#include <vector>

#include "../zip-ada_b200/csrc/b2_zip_layout.h"

static void hex_line(uint64_t off, const std::vector<uint8_t> &b) {
  std::printf("%llu ", (unsigned long long)off);
  for (uint8_t c : b) std::printf("%02x", c);
  std::printf("\n");
}

static uint32_t crc_plain(const uint8_t *p, uint64_t n) {        // Init, Update, Final (zip-crc_crypto.adb:31-61)
  static uint32_t tab[256];
  if (!tab[1]) for (uint32_t i = 0; i < 256; i++) { uint32_t c = i; for (int k = 0; k < 8; k++) c = (c & 1) ? (c >> 1) ^ 0xEDB88320u : c >> 1; tab[i] = c; }
  uint32_t c = 0xFFFFFFFFu;
  for (uint64_t i = 0; i < n; i++) c = tab[(c ^ p[i]) & 0xFF] ^ (c >> 8);
  return ~c;
}

int main(int argc, char **argv) {
  if (argc < 3) return 2;
  const std::string mode = argv[1];
  if (mode == "crc") {
    std::ifstream f(argv[2], std::ios::binary);
    std::vector<uint8_t> d((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    std::vector<uint64_t> cuts;
    for (int i = 3; i < argc; i++) cuts.push_back(std::strtoull(argv[i], nullptr, 10));
    cuts.push_back(d.size());
    uint32_t crc = 0;
    uint64_t at = 0;
    for (uint64_t k : cuts) {
      crc = b2zip::crc32_combine(crc, crc_plain(d.data() + at, k - at), k - at);
      at = k;
    }
    std::printf("%u\n", crc);
    return 0;
  }
  if (mode != "layout") return 2;
  struct Ent { std::string name; uint64_t usize, csize; };
  std::vector<Ent> ents;
  std::ifstream f(argv[2]);
  for (std::string line; std::getline(f, line);) {
    std::istringstream is(line);
    Ent e;
    if (is >> e.name >> e.usize >> e.csize) ents.push_back(e);
  }
  b2zip::ZipLayout L;
  std::vector<uint8_t> hdr;
  for (size_t k = 0; k < ents.size(); k++) {
    uint64_t off = 0, hb = 0;
    if (!L.open_entry(ents[k].usize, ents[k].name.size(), &off, &hb)) { std::puts("capacity"); return 1; }
    const bool stored = ents[k].csize >= ents[k].usize;
    L.close_entry(ents[k].name, ents[k].usize, stored ? ents[k].usize : ents[k].csize, 0x12345678u + (uint32_t)k,
                  b2zip::ZipLayout::default_time, (uint32_t)(k % 4), stored ? 0 : 12, hdr);
    if (hdr.size() != hb) { std::puts("header length changed"); return 1; }
    hex_line(off, hdr);
  }
  const uint64_t at = L.pos;
  if (!L.finish(hdr)) { std::puts("capacity"); return 1; }
  hex_line(at, hdr);
  return 0;
}
