// Stage A3: entropy segmentation (Segment_by_Entropy) on the device: the launcher of k_segment (b2_segment.cuh).
#include "b2_segment.cuh"

int b2k_segment(cudaStream_t st, const u8 *d_in, const B2Chunk *d_chunks, u32 n_chunks, const double *d_T,
                u32 *d_seg, u32 *d_nseg, const u32 *d_progress, double *d_dbg_series, u32 *d_dbg_paths) {
  if (n_chunks == 0) return 0;
  if (d_dbg_series || d_dbg_paths)
    k_segment<true><<<n_chunks, SG_THREADS, 0, st>>>(d_in, d_chunks, n_chunks, d_T, d_seg, d_nseg, d_progress, d_dbg_series, d_dbg_paths);
  else
    k_segment<false><<<n_chunks, SG_THREADS, 0, st>>>(d_in, d_chunks, n_chunks, d_T, d_seg, d_nseg, d_progress, nullptr, nullptr);
  B2_CUDA_CHECK(cudaGetLastError());
  return 0;
}
