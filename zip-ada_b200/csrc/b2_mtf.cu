// Stage A7: move-to-front + zero-run coding (RLE2).  The kernels are in b2_mtf.cuh (shared with the host emulation
// of tests/emu); this unit launches them.
#include "b2_mtf.cuh"

int b2k_mtf(cudaStream_t st, B2Job *d_jobs, u32 n_jobs, const B2SortTile *d_tiles, u32 n_tiles,
            const B2SortTile *d_segs, u32 n_segs_small, u32 n_segs_mid, u32 n_segs, const u8 *d_bwt, u32 *d_m16, u32 *d_m256,
            u32 *d_tilemask, u8 *d_idx, u16 *d_mtf) {
  // d_segs[0 .. n_segs_small) belong to blocks with <= 64 distinct bytes, the next n_segs_mid to blocks with
  // <= 128, the rest to the others
  if (n_tiles) {
    k_mtf_masks<<<n_tiles, MI_THREADS, 0, st>>>(d_tiles, d_jobs, d_bwt, d_m16, d_m256, d_tilemask);
    if (n_segs_small)
      k_mtf_seqg<8><<<(n_segs_small + 4 * MS_WARPS - 1) / (4 * MS_WARPS), 32 * MS_WARPS, 0, st>>>(d_segs, n_segs_small, d_jobs, d_bwt, d_m16, d_m256, d_idx);
    if (n_segs_mid)
      k_mtf_seqg<16><<<(n_segs_mid + 2 * MS_WARPS - 1) / (2 * MS_WARPS), 32 * MS_WARPS, 0, st>>>(d_segs + n_segs_small, n_segs_mid, d_jobs, d_bwt, d_m16, d_m256, d_idx);
    const u32 rest = n_segs - n_segs_small - n_segs_mid;
    if (rest)
      k_mtf_seq<<<(rest + MS_WARPS - 1) / MS_WARPS, 32 * MS_WARPS, 0, st>>>(d_segs + n_segs_small + n_segs_mid, rest, d_jobs, d_bwt, d_m16, d_m256, d_idx);
  }
  if (n_jobs) k_rle2<<<n_jobs, R2_THREADS, 0, st>>>(d_jobs, d_idx, d_mtf);
  B2_CUDA_CHECK(cudaGetLastError());
  return 0;
}
