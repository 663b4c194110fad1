// Host-callable launchers of the b2gpu kernels (internal; the public boundary is include/b2gpu.h).
#pragma once
#include "b2_common.cuh"

struct B2Chunk { u64 start; u32 len; u32 cap; u32 pad; u32 pad2; };

struct B2CrcTables {
  u32 byte_tab[256];      // bzip2.adb:34-100 table
  u32 xp_thread[1024];    // x^(8*16*(1023-t)) mod P
  u32 x_tile;             // x^(8*16384)
  u32 xinv_a[1024];       // x^(-128*a)
  u32 xinv_b[16];         // x^(-8*b)
  u32 pw2[32];            // x^(8*2^k)
};

struct B2SortTile { u32 job; u32 start; };
struct B2SortTileRR { u32 job; u32 start; u32 prev; u32 pad; };   // scatter order: prev = place of the block's tile before this one

// statistics of the BWT sort for the roofline report (see DESIGN.md §Measurement)
struct B2SortStats {
  u64 scatter_launches;        // radix scatter launches
  u64 scatter_elems;           // elements moved by them (sum over launches)
  double scatter_ms;           // CUDA-event time of those launches (only when timing enabled)
  u64 rounds;                  // doubling rounds executed (sum over batches)
  u64 sorted_elems_round0;     // suffixes entering round 0
  u64 sorted_elems_later;      // sum over later rounds of active suffixes
  double sort_ms;              // all sort kernels
  u64 launches;                // kernels launched by the sort driver
};

// b2_chunks.cu  (per 2048-byte tile work arrays of the chunk cutter)
struct B2CutWork { u32 *firstchg, *lastchg, *tsum; u64 *carry_r, *tincl; u8 *gs; u16 *gm; };   // gs / gm: per 16-byte granule
int b2k_cut(cudaStream_t st, const u8 *d_in, u64 n, i64 size_hint, int level, i64 win_lo, i64 win_hi,
            B2Chunk *d_chunks, u32 *d_n_chunks, u32 max_chunks, B2CutWork *w, u32 *d_progress, cudaEvent_t ev_chain_starts);
int b2k_cut_scans(cudaStream_t st, const u8 *d_in, u64 n, B2CutWork *w);
int b2k_cut_chain(cudaStream_t st, const u8 *d_in, u64 n, i64 size_hint, int level, i64 win_lo, i64 win_hi,
                  B2Chunk *d_chunks, u32 *d_n_chunks, u32 max_chunks, B2CutWork *w, u32 *d_progress, cudaEvent_t ev_chain_starts,
                  u64 gbase, u64 pos0, u64 stop);
// b2_segment.cu
#define B2_SEG_GAVE_UP 0xFFFFFFFDu     // a CTA following the chunk chain never saw its chunk (time-sliced GPU): segment again afterwards
#define B2_SEG_PENDING 0xFEFEFEFEu
int b2k_segment(cudaStream_t st, const u8 *d_in, const B2Chunk *d_chunks, u32 n_chunks, const double *d_T,
                u32 *d_seg, u32 *d_nseg, const u32 *d_progress, double *d_dbg_series, u32 *d_dbg_paths);   // taps: b2_segment.cuh
// b2_rle1.cu
void b2k_make_crc_tables(B2CrcTables *t);
int b2k_rle1(cudaStream_t st, const u8 *d_in, B2Job *d_jobs, u32 n_jobs, u8 *d_text, const B2CrcTables *d_ct);

struct B2SortJob { u32 job, tile0, ntiles, pad; };
struct B2ConcatItem { u64 src_word; u64 nbits; u64 dst_bit; };
struct B2StreamEnd { u64 out_off; u64 end_bit; u32 crc; u32 pad; };   // per stream: region start (bytes), bits written so far
struct B2PackItem { u64 src_off; u64 dst_off; u64 len; };           // bytes

struct B2SortCtx {
  u64 *keysA, *keysB;
  u32 *valsA, *valsB, *rank, *grp;
  u32 *slotA, *slotB, *sa_full, *d_tile_cnt;
  B2SortTile *d_tiles;
  B2SortJob *d_sj;
  u32 *d_hist, *d_digit_base;    // look-back tile states [tile][256]; digit bases [block][8 passes][256]
  B2SortTileRR *d_tiles_rr;
  u32 *d_ticket;                 // error flag of the look-back
  const B2Job *h_jobs;           // host copy of the batch's blocks (pos_off), indexed by block id
  u32 max_used;                  // the largest alphabet (bytes in use) of the batch
  int sym_bits;                  // bits per character of the round-0 keys (ceil log2 of the largest alphabet of the batch)
  i32 *d_tile_head, *d_carry;
  u32 *d_unsorted, *h_unsorted;
  size_t max_tiles, max_jobs;
  bool timing;
  B2SortStats stats;
};

#define LL_MAXCODE 20

#ifdef __cplusplus
#include <vector>
// b2_bwt.cu
int b2k_bwt_batch(B2SortCtx *cx, cudaStream_t st, B2Job *d_jobs, const std::vector<u32> &job_ids,
                  const std::vector<u32> &job_n, const u8 *d_text, u8 *d_bwt);
#endif
// b2_mtf.cu  (tiles of 4096 positions, segments of 256 and 16)
#define B2_MTF_TILE 4096
#define B2_SORT_TILE 2048
#define B2_MTF_SEG 32768
int b2k_mtf(cudaStream_t st, B2Job *d_jobs, u32 n_jobs, const B2SortTile *d_tiles, u32 n_tiles,
            const B2SortTile *d_segs, u32 n_segs_small, u32 n_segs_mid, u32 n_segs, const u8 *d_bwt, u32 *d_m16, u32 *d_m256,
            u32 *d_tilemask, u8 *d_idx, u16 *d_mtf);
// b2_entropy.cu
int b2k_entropy(cudaStream_t st, B2Job *d_jobs, u32 n_jobs, u32 max_groups_per_job, u32 total_groups,
                const u16 *d_mtf, u16 *d_ghist, u8 *d_gdist, u32 *d_rank3, u32 *d_rank4, u8 *d_sel, u8 *d_selprev,
                u32 *d_gpack, u16 *d_gselcost,
                u32 *d_hist, u32 *d_leaves, u32 *d_wl, u8 *d_lens, u32 *d_stat, u32 *d_selcost, u32 *d_cost, u32 *d_low,
                int level, u32 max_alpha, u32 *d_activated, u64 *launches);
// b2_pack.cu
int b2k_bits_layout(cudaStream_t st, B2Job *d_jobs, u32 n_jobs, u64 *d_total_words);
int b2k_pack(cudaStream_t st, const B2Job *d_jobs, u32 n_jobs, const u16 *d_mtf, const u8 *d_sel, const u8 *d_lens,
             u8 *d_selpos, u32 *d_bits, int level, u32 total_groups);
int b2k_concat(cudaStream_t st, const B2ConcatItem *d_items, u32 n_items, const u32 *d_bits, u32 *d_out);
int b2k_stream_ends(cudaStream_t st, const B2StreamEnd *d_ends, u32 n, int level, u32 *d_out);
int b2k_pack_streams(cudaStream_t st, const B2PackItem *d_items, u32 n, const u8 *d_src, u8 *d_dst);

// ---- archive side (b2_zip.cu) --------------------------------------------------------------------
#define B2_ZIP_TILE 65536
struct B2ZipCrcTables {
  u32 byte_tab[256];      // MSB-first table of 0x04C11DB7 (fed with bit-reversed bytes)
  u32 xp_thread[1024];    // x^(8*64*(1023-t))
  u32 pw2[48];            // x^(8*2^k)
};
struct B2ZipTile { u64 begin; u64 end; };               // bytes [max(begin, end-65536), end) of the input arena
struct B2ZipEntry { u64 len; u32 tile0; u32 n_tiles; };
struct B2ZipCopy { u64 src_off; u64 dst_off; u32 len; u32 which; };
void b2k_make_zipcrc_tables(B2ZipCrcTables *t);
int b2k_zipcrc(cudaStream_t st, const u8 *d_in, const B2ZipTile *d_tiles, u32 n_tiles, const B2ZipEntry *d_ents, u32 n_entries,
               const B2ZipCrcTables *d_zt, u32 *d_partial, u32 *d_crc);
int b2k_zip_gather(cudaStream_t st, const B2ZipCopy *d_items, u32 n, const u8 *d_src0, const u8 *d_src1, u8 *d_dst);

// ---- decode / verify (b2_verify.cu) -----------------------------------------------------------------------
struct B2VBlock {
  u64 start_bit;      // position of the block's 48-bit magic in the stream
  u64 end_bit;        // (out) first bit behind the block
  u64 raw_len;        // (out) raw bytes of the block (after RLE1 decoding)
  u64 raw_off;        // (in, for the comparison) where the block's raw bytes start in the decoded stream
  u32 stored_crc, computed_crc, n_rle, orig_ptr, status, pad;
};
int b2k_verify_find(cudaStream_t st, const u8 *d_stream, u64 n_bytes, u64 *d_cand, u32 *d_n_cand, u32 cap);
int b2k_verify_decode(cudaStream_t st, const u8 *d_stream, u64 n_bytes, B2VBlock *d_blocks, u32 n_blocks, u32 max_n, u32 *d_link, u8 *d_lcol,
                      u8 *d_rle, u8 *d_sel, const u32 *d_crc_tab);
int b2k_verify_compare(cudaStream_t st, const B2VBlock *d_blocks, const u32 *d_chain, u32 n_chain, u32 max_n, const u8 *d_rle,
                       const u8 *d_expect, u64 expect_n, unsigned long long *d_first_bad);
