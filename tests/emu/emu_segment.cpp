// Host emulation of k_segment (zip-ada_b200/csrc/b2_segment.cuh): runs the kernel, unchanged, as one CTA over one chunk
// with its test taps on and writes what it computed for tests/test_emu_segment.py to compare with the oracle.
// Test infrastructure; usage: emu_segment <chunk file> <output prefix>
//   <prefix>.series  float64, the sum after every step (len - 16 000 values; none when len <= 20 000)
//   <prefix>.cuts    uint32: n0, n1, then the n0 cuts of profile 0 and the n1 cuts of profile 1
//   <prefix>.paths   uint32[4]: batches started on one binade, on two binades, restarts, batches of the literal chain
#include "cuda_emu.h"
#define B2_EMU 1
#include "../../zip-ada_b200/csrc/b2_segment.cuh"

#include <cmath>
#include <cstdio>
#include <string>

void b2_set_error(const char *, int, const char *) {}

static bool write_file(const std::string &path, const void *p, size_t bytes) {
  FILE *f = fopen(path.c_str(), "wb");
  if (!f) return false;
  const bool ok = fwrite(p, 1, bytes, f) == bytes;
  return fclose(f) == 0 && ok;
}

int main(int argc, char **argv) {
  if (argc != 3) { fprintf(stderr, "usage: emu_segment <chunk file> <output prefix>\n"); return 2; }
  FILE *f = fopen(argv[1], "rb");
  if (!f) { perror(argv[1]); return 2; }
  std::vector<u8> in;
  for (int ch; (ch = fgetc(f)) != EOF;) in.push_back((u8)ch);
  fclose(f);
  const u32 len = (u32)in.size();
  if (len == 0 || len > 9000000) { fprintf(stderr, "chunk of %u bytes\n", len); return 2; }
  in.resize((size_t)len + 256, 0);
  // the table of b2_create (b2_api.cu): T[c] = -(p * Log (p)), p = c / 16 000
  std::vector<double> T(16002, 0.0);
  const double inv = 1.0 / 16000.0;
  for (int c = 1; c <= 16001; c++) { const double p = (double)c * inv; T[c] = -(p * std::log(p)); }
  const B2Chunk chunk{0, len, 0, 0, 0};
  std::vector<u32> seg(2 * B2_MAX_SEG, 0xEEEEEEEEu), nseg(2, 0xEEEEEEEEu), paths(4, 0);
  const size_t steps = len > 20000 ? len - 16000 : 0;
  std::vector<double> series(steps + 1, std::nan(""));
  emu_launch(1, SG_THREADS, sizeof(SegSmem), 1, [&]() {
    k_segment<true>(in.data(), &chunk, 1, T.data(), seg.data(), nseg.data(), nullptr, series.data(), paths.data());
  });
  if (nseg[0] > B2_MAX_SEG || nseg[1] > B2_MAX_SEG) { fprintf(stderr, "segment counts %u %u\n", nseg[0], nseg[1]); return 1; }
  std::vector<u32> cuts(nseg.begin(), nseg.end());
  for (int p = 0; p < 2; p++) cuts.insert(cuts.end(), seg.begin() + (size_t)p * B2_MAX_SEG, seg.begin() + (size_t)p * B2_MAX_SEG + nseg[p]);
  const std::string out = argv[2];
  if (!write_file(out + ".series", series.data(), steps * sizeof(double)) || !write_file(out + ".cuts", cuts.data(), cuts.size() * sizeof(u32)) ||
      !write_file(out + ".paths", paths.data(), paths.size() * sizeof(u32))) { perror(argv[2]); return 2; }
  printf("OK\n");
  return 0;
}
