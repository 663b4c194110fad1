// Host emulation of stage A7 (zip-ada_b200/csrc/b2_mtf.cuh): runs k_mtf_masks, k_mtf_seqg<8>, k_mtf_seqg<16>, k_mtf_seq
// and k_rle2, unchanged, on a batch of given last columns and writes what they computed for tests/test_emu_mtf.py to
// compare with the oracle.  The batch is laid out and planned as b2_dbg_mtf does it (256-aligned slots of
// min (n * 5/4 + 8, 900 064) positions, 4096-position tiles, 32 768-position segments by kernel class); `window` CTAs
// of a launch run at a time.  The slot padding behind every column, the masks, the index bytes and the symbols are
// poisoned first.  Test infrastructure; usage: emu_mtf <batch file> <output prefix> <window>
//   batch file: uint32 count, uint32 n[count], then the columns one after the other
//   <prefix>.idx   the n index bytes of every block, one block after the other
//   <prefix>.mtf   the n_mtf uint16 symbols of every block, one block after the other
//   <prefix>.info  uint32 n_mtf, n_groups per block
#include "cuda_emu.h"
#define B2_EMU 1
#include "../../zip-ada_b200/csrc/b2_mtf.cuh"

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
  if (argc != 4) { fprintf(stderr, "usage: emu_mtf <batch file> <output prefix> <window>\n"); return 2; }
  FILE *f = fopen(argv[1], "rb");
  if (!f) { perror(argv[1]); return 2; }
  std::vector<u8> in;
  for (int ch; (ch = fgetc(f)) != EOF;) in.push_back((u8)ch);
  fclose(f);
  const unsigned window = (unsigned)atoi(argv[3]);
  u32 J = 0;
  if (in.size() < 4 || window == 0) { fprintf(stderr, "bad arguments\n"); return 2; }
  memcpy(&J, in.data(), 4);
  if (in.size() < 4 + 4 * (size_t)J) { fprintf(stderr, "short batch file\n"); return 2; }
  std::vector<B2Job> jobs(J);
  std::vector<u32> ns(J);
  memcpy(ns.data(), in.data() + 4, 4 * (size_t)J);
  size_t src = 4 + 4 * (size_t)J;
  u64 pos = 0, mpos = 0;
  for (u32 j = 0; j < J; j++) {
    B2Job &b = jobs[j];
    memset(&b, 0, sizeof b);
    if (ns[j] > 900000) { fprintf(stderr, "block %u: %u positions\n", j, ns[j]); return 2; }
    b.n = b.raw_len = ns[j];
    u64 cap = std::min<u64>((u64)b.n * 5 / 4 + 8, 900064);
    cap = (cap + 255) & ~255ull;
    b.pos_off = (u32)pos; b.cap = (u32)cap; pos += cap;
    b.mtf_off = (u32)mpos; mpos += (cap + 2 + 7) & ~7ull;
  }
  std::vector<u8> bwt(pos + 64, 0xA5), idx(pos + 64, 0xA5);
  std::vector<u32> m16((pos / 16 + 8) * 8, 0u), m256((pos / 256 + 8) * 8, 0u);   // an unwritten mask reads as "no byte here"
  std::vector<u16> mtf(mpos + 64, 0xA5A5);
  std::vector<B2SortTile> tiles, segs[3];
  for (u32 j = 0; j < J; j++) {
    B2Job &b = jobs[j];
    if (src + b.n > in.size()) { fprintf(stderr, "short batch file\n"); return 2; }
    memcpy(bwt.data() + b.pos_off, in.data() + src, b.n);
    for (u32 i = 0; i < b.n; i++) b.in_use[in[src + i] >> 5] |= 1u << (in[src + i] & 31);
    src += b.n;
    for (int q = 0; q < 8; q++) b.n_used += __builtin_popcount(b.in_use[q]);
    b.tile0 = (u32)tiles.size();
    for (u32 s = 0; s < b.n; s += B2_MTF_TILE) tiles.push_back(B2SortTile{j, s});
    for (u32 s = 0; s < b.n; s += B2_MTF_SEG) segs[b.n_used <= 64 ? 0 : b.n_used <= 128 ? 1 : 2].push_back(B2SortTile{j, s});
  }
  std::vector<u32> tilemask((tiles.size() + 1) * 8, 0u);
  const size_t smem = 16384;
  if (!tiles.empty()) {
    emu_launch((u32)tiles.size(), MI_THREADS, smem, window, [&]() { k_mtf_masks(tiles.data(), jobs.data(), bwt.data(), m16.data(), m256.data(), tilemask.data()); });
    const u32 n0 = (u32)segs[0].size(), n1 = (u32)segs[1].size(), n2 = (u32)segs[2].size();
    if (n0) emu_launch((n0 + 4 * MS_WARPS - 1) / (4 * MS_WARPS), 32 * MS_WARPS, smem, window, [&]() { k_mtf_seqg<8>(segs[0].data(), n0, jobs.data(), bwt.data(), m16.data(), m256.data(), idx.data()); });
    if (n1) emu_launch((n1 + 2 * MS_WARPS - 1) / (2 * MS_WARPS), 32 * MS_WARPS, smem, window, [&]() { k_mtf_seqg<16>(segs[1].data(), n1, jobs.data(), bwt.data(), m16.data(), m256.data(), idx.data()); });
    if (n2) emu_launch((n2 + MS_WARPS - 1) / MS_WARPS, 32 * MS_WARPS, smem, window, [&]() { k_mtf_seq(segs[2].data(), n2, jobs.data(), bwt.data(), m16.data(), m256.data(), idx.data()); });
  }
  if (J) emu_launch(J, R2_THREADS, smem, window, [&]() { k_rle2(jobs.data(), idx.data(), mtf.data()); });
  std::vector<u8> idx_out;
  std::vector<u16> mtf_out;
  std::vector<u32> info;
  for (const B2Job &b : jobs) {
    if (b.n_mtf > b.cap + 2) { fprintf(stderr, "n_mtf %u above the slot of %u\n", b.n_mtf, b.cap); return 1; }
    idx_out.insert(idx_out.end(), idx.begin() + b.pos_off, idx.begin() + b.pos_off + b.n);
    mtf_out.insert(mtf_out.end(), mtf.begin() + b.mtf_off, mtf.begin() + b.mtf_off + b.n_mtf);
    info.push_back(b.n_mtf); info.push_back(b.n_groups);
  }
  const std::string out = argv[2];
  if (!write_file(out + ".idx", idx_out.data(), idx_out.size()) || !write_file(out + ".mtf", mtf_out.data(), mtf_out.size() * 2) ||
      !write_file(out + ".info", info.data(), info.size() * 4)) { perror(argv[2]); return 2; }
  printf("OK\n");
  return 0;
}
