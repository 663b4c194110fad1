// Host orchestration + the C ABI of include/b2gpu.h.
//
// Mirrors the stream level of the reference, zip_lib/bzip2-encoding.adb:1136-1431:
//   Write_Stream_Header (:1384-1391) -> { Read_and_Split_Block (:1144) }* -> Write_Stream_Footer (:1395-1407)
// with Block_Split_Parallel's four tactics (:1214-1359) expanded into a de-duplicated list of
// blocks ("jobs") that are encoded in batches on the device.  The only serial cross-chunk data are
// scalars — incoming bit offset, winner, combined CRC — replayed here in O(#chunks) (SURVEY §8e).
//
// Flow of one call: chunk cutting (tile scans + one warp walking the chunk chain) -> entropy
// segmentation (for a single large stream on a second CUDA stream, following the chain chunk by chunk)
// -> the calling thread plans batches of whole chunks as their cut lists arrive and hands them to the
// worker thread(s); each of W workspaces (default 1) owns a CUDA stream and a worker that runs
// RLE1 -> BWT sort -> MTF/RLE2 -> entropy search -> bit packing for its batch and then resolves the
// winners of its chunks strictly in chunk order (shift-concatenation into the output stream).
// b2_zip_create adds the archive side around the same machinery (Zip CRC-32, headers, Store fallback).
#include "b2_common.cuh"
#include "b2_kernels.h"
#include "b2_zip_layout.h"
#include "../../include/b2gpu.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <chrono>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>
#include <unordered_set>

static thread_local std::string g_last_error = "";
void b2_set_error(const char *file, int line, const char *msg) {
  char buf[512];
  snprintf(buf, sizeof buf, "%s:%d: %s", file, line, msg);
  g_last_error = buf;
}
#define B2_FAIL(code, msg) do { b2_set_error(__FILE__, __LINE__, msg); return code; } while (0)
#define B2_TRY(x) do { int rc_ = (x); if (rc_) return rc_; } while (0)
// calls that use the handle's device buffers are refused while b2_stream_* or b2_zip_begin .. finish own them
#define B2_NO_STREAM(e) do { if ((e)->stream.open) B2_FAIL(B2_ERR_ARGUMENT, "a stream is open on this handle (b2_stream_begin)"); \
                             if ((e)->zip.open) B2_FAIL(B2_ERR_ARGUMENT, "an archive is open on this handle (b2_zip_begin)"); } while (0)

namespace {

template <class T> struct DevBuf {
  T *p = nullptr; size_t cap = 0;
  int ensure(size_t n) {
    if (n <= cap) return 0;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = n + n / 8 + 256;
    cudaError_t e = cudaMalloc((void **)&p, want * sizeof(T));
    if (e != cudaSuccess) { b2_set_error(__FILE__, __LINE__, cudaGetErrorString(e)); return B2_ERR_ALLOC; }
    cap = want;
    return 0;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct ChunkPlan {
  u64 start; u32 len; u32 cap;
  std::vector<u32> tactic_jobs[4];   // job ids inside the chunk's batch, in stream order
  u32 n_seg[2];
  int n_tactics;
};

struct Batch {
  u32 c0, c1;                        // chunk range [c0, c1)
  std::vector<B2Job> jobs;
};

// Everything one in-flight batch needs on the device.
struct Workspace {
  cudaStream_t st = nullptr;
  cudaEvent_t ev[2] = {nullptr, nullptr};
  cudaEvent_t ev_sort[2] = {nullptr, nullptr};
  double sort_ms = 0;
  DevBuf<u32> d_scalars;
  DevBuf<B2Job> d_jobs;
  DevBuf<u8> d_text, d_bwt, d_idx;
  DevBuf<u32> d_m16, d_m256, d_tilemask;
  DevBuf<u64> d_keysA, d_keysB;
  DevBuf<u32> d_valsA, d_valsB, d_rank, d_grp, d_slotA, d_slotB, d_sa, d_tile_cnt;
  DevBuf<B2SortTile> d_tiles, d_mtiles, d_msegs;
  DevBuf<B2SortTileRR> d_tiles_rr;
  DevBuf<B2SortJob> d_sj;
  DevBuf<u32> d_hist, d_digit_base;
  DevBuf<i32> d_tile_head, d_carry;
  DevBuf<u32> d_unsorted;
  DevBuf<u16> d_mtf, d_ghist;
  DevBuf<u8> d_gdist;
  DevBuf<u32> d_rank3, d_rank4;
  DevBuf<u8> d_sel, d_selprev, d_selpos, d_lens;
  DevBuf<u32> d_ehist, d_leaves, d_wl, d_estat, d_selcost;
  DevBuf<u32> d_gpack;
  DevBuf<u16> d_gselcost;
  DevBuf<u32> d_cost, d_low;
  DevBuf<u32> d_bits;
  DevBuf<B2ConcatItem> d_items;
  u32 *h_unsorted = nullptr; size_t h_unsorted_cap = 0;
  std::vector<B2Job> batch_jobs;      // jobs of the current batch, as read back
  u32 total_groups = 0;
  // accumulated by this workspace during one encode call
  B2SortStats sort_stats;
  u64 launches = 0, blocks = 0, block_bytes = 0;
  double stage_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};

  void release() {
    d_scalars.release(); d_jobs.release(); d_text.release(); d_bwt.release(); d_idx.release(); d_m16.release();
    d_m256.release(); d_tilemask.release(); d_keysA.release(); d_keysB.release(); d_valsA.release(); d_valsB.release();
    d_rank.release(); d_grp.release(); d_slotA.release(); d_slotB.release(); d_sa.release(); d_tile_cnt.release(); d_tiles.release(); d_tiles_rr.release(); d_mtiles.release(); d_msegs.release(); d_sj.release(); d_hist.release();
    d_digit_base.release(); d_tile_head.release(); d_carry.release(); d_unsorted.release(); d_mtf.release(); d_ghist.release(); d_gdist.release();
    d_rank3.release(); d_rank4.release(); d_sel.release(); d_selprev.release(); d_selpos.release(); d_lens.release();
    d_ehist.release(); d_leaves.release(); d_wl.release(); d_estat.release(); d_selcost.release(); d_gpack.release(); d_gselcost.release(); d_cost.release();
    d_low.release(); d_bits.release(); d_items.release();
    if (h_unsorted) cudaFreeHost(h_unsorted);
    h_unsorted = nullptr; h_unsorted_cap = 0;
    if (ev[0]) cudaEventDestroy(ev[0]);
    if (ev[1]) cudaEventDestroy(ev[1]);
    if (ev_sort[0]) cudaEventDestroy(ev_sort[0]);
    if (ev_sort[1]) cudaEventDestroy(ev_sort[1]);
    ev_sort[0] = ev_sort[1] = nullptr;
    if (st) cudaStreamDestroy(st);
    st = nullptr; ev[0] = ev[1] = nullptr;
  }
};

}  // namespace

// One stream spread over several handles (b2_shard_*), or one window of a stream fed in pieces (b2_stream_*):
// what this handle keeps between the calls.
struct ShardCand { u32 arena; u32 blocks; u64 word_off; u64 nbits; u32 fold; u32 kept; };
struct ShardState {
  bool open = false, cut = false, encoded = false;
  bool last = false;                   // the shard ends the stream: its chain walks to the end of its bytes, it writes the footer
  const u8 *d_in = nullptr;            // the shard's bytes on the device: stream bytes [base, base + n_local)
  u64 base = 0, n_local = 0, own_end = 0, entry = 0, handoff = 0;
  i64 hint = -1;
  std::vector<DevBuf<u32> *> arenas;   // candidate bitstreams that may still win, one arena per batch (kept across calls)
  std::vector<ShardCand> cands;        // [chunk][tactic]
  std::vector<int> n_tactics;
};

// One stream fed in pieces (b2_stream_*).  Every window is a shard of the stream on this handle (DESIGN.md §6b).
struct StreamState {
  bool open = false;
  i64 hint = -1;
  u64 window = 0, margin = 0;          // W, and M = b2_shard_margin (level)
  u8 *buf[2] = {nullptr, nullptr};     // two window buffers of W + M + 256 bytes (kept across streams of the same W)
  u64 buf_bytes = 0;
  int cur = 0;                         // buf[cur] holds the stream bytes [base, base + held), not encoded yet
  u64 base = 0, held = 0;
  u64 bit = 32;                        // stream bit offset where the next window's first block starts
  u32 crc = 0;                         // combined CRC before it
  u64 out_end = 0;                     // stream bytes whose final value has been written to an `out`
  u8 tail = 0;                         // the bits of byte out_end so far (the partial byte held back)
  std::vector<b2_chunk_trace> trace;   // every chunk of the stream so far, stream offsets
};

// One archive written entry by entry (b2_zip_*, DESIGN.md §7c).  Small entries are queued in stream.buf[0]; an entry
// above the window goes through the windows of b2_stream_* (the StreamState) with its own size as size_hint.
struct ZipQueued { std::string name; u64 off, n; u32 time, flags; };
struct ZipState {
  bool open = false;
  int duplicates = 0;
  b2zip::ZipLayout layout;               // pos = archive bytes written to an `out` so far
  std::unordered_set<std::string> names; // with B2_ZIP_ERROR_ON_DUPLICATE
  std::vector<ZipQueued> queue;          // entries uploaded, not encoded yet
  u64 q_end = 0, q_bytes = 0;            // staging bytes in use (16-byte aligned placement), input bytes queued
  u64 q_bound = 0;                       // archive bytes the queue can become
  u64 cd_bound = 0;                      // central directory bytes, at most, of every entry added
  u64 done = 0, added = 0;               // uncompressed bytes encoded, added
};

struct b2_encoder {
  int level = 9, device = 0;
  ShardState shard;
  StreamState stream;
  ZipState zip;
  cudaStream_t cst = nullptr;           // uploads of b2_stream_write, overlapping the encode of the window before
  cudaEvent_t ev_up = nullptr;          // recorded on cst after every upload
  b2_progress_fn progress = nullptr;    // called on the calling thread between batches; non-zero return aborts
  void *progress_user = nullptr;
  cudaStream_t st = nullptr;            // stream of the stream-level work (cut, segment, copies, footer)
  cudaStream_t st2 = nullptr;           // segmentation following the chunk chain
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  int timing = 0;                       // 0 off, 1 scatter + call events, 2 also per-stage timers (adds syncs, no pipelining)
  // constants
  DevBuf<B2CrcTables> d_ct;
  DevBuf<double> d_T;
  // stream-level
  DevBuf<u8> d_in;
  DevBuf<u32> d_out;
  DevBuf<B2Chunk> d_chunks;
  DevBuf<u32> d_scalars;
  DevBuf<u32> d_seg, d_nseg;
  DevBuf<B2StreamEnd> d_ends;
  DevBuf<B2PackItem> d_packitems;
  DevBuf<u8> d_packed;
  DevBuf<u32> d_cut_first, d_cut_last, d_cut_tsum;
  DevBuf<u64> d_cut_carry, d_cut_tincl;
  DevBuf<u8> d_cut_gs;
  DevBuf<u16> d_cut_gm;
  // archive side (b2_zip_create)
  DevBuf<B2ZipCrcTables> d_zt;
  DevBuf<B2ZipTile> d_ztiles;
  DevBuf<B2ZipEntry> d_zents;
  DevBuf<B2ZipCopy> d_zcopies;
  DevBuf<u32> d_zpartial, d_zcrc;
  // decode / verify (b2_verify_stream)
  DevBuf<u8> d_vstream, d_vlcol, d_vrle, d_vsel;
  DevBuf<u32> d_vlink, d_vchain, d_vscal;
  DevBuf<u64> d_vcand;
  DevBuf<B2VBlock> d_vblocks;
  std::vector<Workspace *> ws;
  // host state of the last call
  std::vector<B2Chunk> chunks;
  std::vector<u32> nseg;
  std::vector<std::vector<u32>> seg;     // cut lists of (chunk, profile); empty when the list is just [len]
  std::vector<b2_chunk_trace> trace;
  b2_stats stats;
  B2SortStats sort_stats;
  bool batch_positions_fixed = false;   // B2GPU_BATCH_POSITIONS was given: the adaptive single-batch rule below is off
  size_t batch_positions = 1536ull << 20;  // positions per batch (env B2GPU_BATCH_POSITIONS); big batches amortise the latency-bound kernels (about 45 B of device memory per position)
  size_t first_batch_positions = ~(size_t)0;     // optional smaller first batch of a single large stream (env B2GPU_FIRST_BATCH_POSITIONS; measured: not a gain)
  size_t batch_jobs_max = 65535;        // blocks per batch    (env B2GPU_BATCH_JOBS)
  int n_workspaces = 1;                 // batches in flight   (env B2GPU_PIPELINE)
  u64 launches_other = 0;
  cudaEvent_t ev[2] = {nullptr, nullptr};
  cudaEvent_t ev_call[2] = {nullptr, nullptr};
};

namespace {

struct StageTimer {
  cudaStream_t st; cudaEvent_t *ev; double *acc; bool on;
  StageTimer(b2_encoder *e, cudaStream_t st_, cudaEvent_t *ev_, double *acc_) : st(st_), ev(ev_), acc(acc_), on(e->timing >= 2) {
    if (on) cudaEventRecord(ev[0], st);
  }
  ~StageTimer() {
    if (on) {
      cudaEventRecord(ev[1], st);
      cudaEventSynchronize(ev[1]);
      float ms = 0; cudaEventElapsedTime(&ms, ev[0], ev[1]);
      *acc += ms;
    }
  }
};

void balance_window(int level, i64 &lo, i64 &hi) {
  // Float (stream_rest) in Float (block_capacity) * (1.0 + 0.05) .. Float (block_capacity) * (1.0 + 0.30)
  // evaluated in IEEE single precision (bzip2-encoding.adb:1410-1418).
  volatile float fcap = (float)(100000 * level);
  volatile float flo = fcap * 1.05f, fhi = fcap * 1.30f;
  lo = -1; hi = -2;
  i64 base = 100000ll * level;
  for (i64 v = base; v <= 2 * base; v++) {
    volatile float f = (float)v;
    if (f >= flo && f <= fhi) { if (lo < 0) lo = v; hi = v; }
  }
}

int ensure_batch_workspace(Workspace *w, size_t T, size_t J) {
  const size_t max_tiles = T / B2_SORT_TILE + J + 8;
  const size_t max_mtiles = T / B2_MTF_TILE + J + 8;
  const size_t GT = T / B2_GROUP_SIZE + 20 * J + 32;
  B2_TRY(w->d_scalars.ensure(16));
  B2_TRY(w->d_jobs.ensure(J));
  B2_TRY(w->d_text.ensure(T + 64)); B2_TRY(w->d_bwt.ensure(T + 64)); B2_TRY(w->d_idx.ensure(T + 64));
  B2_TRY(w->d_m16.ensure((T / 16 + 8 * J + 8) * 8)); B2_TRY(w->d_m256.ensure((T / 256 + 2 * J + 8) * 8));
  B2_TRY(w->d_keysA.ensure(T)); B2_TRY(w->d_keysB.ensure(T));
  B2_TRY(w->d_valsA.ensure(T)); B2_TRY(w->d_valsB.ensure(T));
  B2_TRY(w->d_rank.ensure(T)); B2_TRY(w->d_grp.ensure(T));
  B2_TRY(w->d_slotA.ensure(T)); B2_TRY(w->d_slotB.ensure(T)); B2_TRY(w->d_sa.ensure(T)); B2_TRY(w->d_tile_cnt.ensure(max_tiles));
  B2_TRY(w->d_tiles.ensure(max_tiles)); B2_TRY(w->d_tiles_rr.ensure(max_tiles)); B2_TRY(w->d_mtiles.ensure(max_mtiles));
  B2_TRY(w->d_tilemask.ensure(max_mtiles * 8)); B2_TRY(w->d_msegs.ensure(T / B2_MTF_SEG + J + 8));
  B2_TRY(w->d_sj.ensure(J));
  B2_TRY(w->d_hist.ensure(max_tiles * 256)); B2_TRY(w->d_digit_base.ensure(J * 8 * 256 + 256));
  B2_TRY(w->d_tile_head.ensure(max_tiles)); B2_TRY(w->d_carry.ensure(max_tiles));
  B2_TRY(w->d_unsorted.ensure(J));
  B2_TRY(w->d_mtf.ensure(T + 16 * J + 64)); B2_TRY(w->d_ghist.ensure(T + 16 * J + 64));
  B2_TRY(w->d_rank3.ensure(GT)); B2_TRY(w->d_rank4.ensure(GT)); B2_TRY(w->d_gdist.ensure(GT));
  B2_TRY(w->d_sel.ensure(GT * B2_N_TRIPLES + 64)); B2_TRY(w->d_selprev.ensure(GT * B2_N_TRIPLES + 64));
  B2_TRY(w->d_selpos.ensure(GT));
  B2_TRY(w->d_gpack.ensure(GT * B2_N_TRIPLES + 64)); B2_TRY(w->d_gselcost.ensure(GT * B2_N_TRIPLES + 64));
  B2_TRY(w->d_ehist.ensure(J * B2_N_TRIPLES * B2_MAX_CODERS * 260));
  B2_TRY(w->d_leaves.ensure((J * B2_N_TRIPLES * B2_MAX_CODERS + 64) * 260)); B2_TRY(w->d_wl.ensure(J * B2_N_TRIPLES * (B2_MAX_CODERS + 3) + J / 32 + 512));
  B2_TRY(w->d_estat.ensure(J * B2_N_TRIPLES * 2)); B2_TRY(w->d_selcost.ensure(J * B2_N_TRIPLES));
  B2_TRY(w->d_lens.ensure(J * B2_N_TRIPLES * B2_MAX_CODERS * B2_MAX_ALPHA));
  B2_TRY(w->d_cost.ensure(J * B2_N_TRIPLES)); B2_TRY(w->d_low.ensure(J * B2_N_TRIPLES));
  B2_TRY(w->d_items.ensure(J));
  if (J > w->h_unsorted_cap) {
    if (w->h_unsorted) cudaFreeHost(w->h_unsorted);
    B2_CUDA_CHECK(cudaMallocHost((void **)&w->h_unsorted, (J + 64) * sizeof(u32)));
    w->h_unsorted_cap = J + 64;
  }
  return 0;
}

// Assigns arena offsets to jobs (host); returns the number of positions.
u64 layout_jobs(std::vector<B2Job> &jobs, int level) {
  u64 pos = 0, mpos = 0;
  for (auto &j : jobs) {
    u64 cap = std::min<u64>((u64)j.raw_len * 5 / 4 + 8, (u64)level * 100000 + 64);
    cap = (cap + 255) & ~255ull;     // 256-aligned slots: the MTF segment masks are addressed by pos_off >> 4 / >> 8
    j.pos_off = (u32)pos; j.cap = (u32)cap;
    pos += cap;
    j.mtf_off = (u32)mpos;
    mpos += (cap + 2 + 7) & ~7ull;
  }
  return pos;
}

// The MTF stage's plan (host; needs n and n_used of every block): the 4096-position tiles of k_mtf_masks (b.tile0 = a
// block's first) and the segments of B2_MTF_SEG positions, blocks with <= 64 bytes in use first, then <= 128, then
// the others (the kernel classes of b2k_mtf).
struct MtfPlan {
  std::vector<B2SortTile> tiles, segs;
  u32 n_small = 0, n_mid = 0;
};

void plan_mtf(std::vector<B2Job> &jobs, MtfPlan &P) {
  std::vector<B2SortTile> mid, big;
  P.tiles.clear(); P.segs.clear();
  for (u32 j = 0; j < (u32)jobs.size(); j++) {
    B2Job &b = jobs[j];
    b.tile0 = (u32)P.tiles.size();
    for (u32 s = 0; s < b.n; s += B2_MTF_TILE) P.tiles.push_back(B2SortTile{j, s});
    for (u32 s = 0; s < b.n; s += B2_MTF_SEG) (b.n_used <= 64 ? P.segs : b.n_used <= 128 ? mid : big).push_back(B2SortTile{j, s});
  }
  P.n_small = (u32)P.segs.size(); P.n_mid = (u32)mid.size();
  P.segs.insert(P.segs.end(), mid.begin(), mid.end());
  P.segs.insert(P.segs.end(), big.begin(), big.end());
}

// Uploads the plan and launches the stage on w's stream: w->d_bwt (the last columns) -> w->d_idx, w->d_mtf and
// n_mtf / n_groups of w->d_jobs.
int launch_mtf(Workspace *w, u32 J, const MtfPlan &P) {
  cudaStream_t st = w->st;
  if (!P.tiles.empty())
    B2_CUDA_CHECK(cudaMemcpyAsync(w->d_mtiles.p, P.tiles.data(), P.tiles.size() * sizeof(B2SortTile), cudaMemcpyHostToDevice, st));
  if (!P.segs.empty())
    B2_CUDA_CHECK(cudaMemcpyAsync(w->d_msegs.p, P.segs.data(), P.segs.size() * sizeof(B2SortTile), cudaMemcpyHostToDevice, st));
  B2_TRY(b2k_mtf(st, w->d_jobs.p, J, w->d_mtiles.p, (u32)P.tiles.size(), w->d_msegs.p, P.n_small, P.n_mid, (u32)P.segs.size(), w->d_bwt.p,
                 w->d_m16.p, w->d_m256.p, w->d_tilemask.p, w->d_idx.p, w->d_mtf.p));
  w->launches += 4;
  return 0;
}

// Runs one batch through RLE1 -> BWT -> MTF/RLE2 -> entropy search -> bit packing on workspace w.
// On return w->batch_jobs holds the device's view of the jobs (n, crc, origin, nbits, bits_off ...).
int run_batch(b2_encoder *e, Workspace *w, const u8 *d_in, std::vector<B2Job> &jobs) {
  const u32 J = (u32)jobs.size();
  if (J == 0) return 0;
  const u64 T = layout_jobs(jobs, e->level);
  if (T >= (1ull << 32) - (1ull << 20)) B2_FAIL(B2_ERR_INTERNAL, "batch too large for 32-bit arena offsets (lower B2GPU_BATCH_POSITIONS)");
  B2_TRY(ensure_batch_workspace(w, (size_t)T + 64, J));
  cudaStream_t st = w->st;
  B2_CUDA_CHECK(cudaMemcpyAsync(w->d_jobs.p, jobs.data(), J * sizeof(B2Job), cudaMemcpyHostToDevice, st));
  {
    StageTimer tm(e, st, w->ev, &w->stage_ms[1]);
    B2_TRY(b2k_rle1(st, d_in, w->d_jobs.p, J, w->d_text.p, e->d_ct.p));
    w->launches += 1;
  }
  w->batch_jobs.resize(J);
  B2_CUDA_CHECK(cudaMemcpyAsync(w->batch_jobs.data(), w->d_jobs.p, J * sizeof(B2Job), cudaMemcpyDeviceToHost, st));
  B2_CUDA_CHECK(cudaStreamSynchronize(st));
  // group arena offsets need n (M <= n + 1)
  u32 gpos = 0, max_g = 1;
  std::vector<u32> ids(J), ns(J);
  for (u32 j = 0; j < J; j++) {
    B2Job &b = w->batch_jobs[j];
    if (b.n > b.cap) B2_FAIL(B2_ERR_INTERNAL, "RLE1 output exceeds its slot");
    u32 gmax = (b.n / B2_GROUP_SIZE + 2 + 15) & ~15u;     // multiple of 16: vector loads in k_ent_sweep / k_ent_selcost
    b.grp_off = gpos; gpos += gmax;
    max_g = std::max(max_g, gmax);
    ids[j] = j; ns[j] = b.n;
    b.na = b.n;
    w->block_bytes += b.n;
  }
  MtfPlan mplan;
  plan_mtf(w->batch_jobs, mplan);
  w->blocks += J;
  w->total_groups = gpos;
  // write grp_off / tile0 / na back (the only fields changed on the host)
  B2_CUDA_CHECK(cudaMemcpyAsync(w->d_jobs.p, w->batch_jobs.data(), J * sizeof(B2Job), cudaMemcpyHostToDevice, st));
  {
    StageTimer tm(e, st, w->ev, &w->stage_ms[2]);
    B2SortCtx cx;
    cx.keysA = w->d_keysA.p; cx.keysB = w->d_keysB.p; cx.valsA = w->d_valsA.p; cx.valsB = w->d_valsB.p;
    cx.rank = w->d_rank.p; cx.grp = w->d_grp.p; cx.d_tiles = w->d_tiles.p; cx.d_sj = w->d_sj.p;
    cx.slotA = w->d_slotA.p; cx.slotB = w->d_slotB.p; cx.sa_full = w->d_sa.p; cx.d_tile_cnt = w->d_tile_cnt.p;
    cx.d_hist = w->d_hist.p; cx.d_digit_base = w->d_digit_base.p; cx.d_tiles_rr = w->d_tiles_rr.p; cx.d_ticket = w->d_digit_base.p + w->d_digit_base.cap - 256; cx.d_tile_head = w->d_tile_head.p; cx.d_carry = w->d_carry.p;
    cx.d_unsorted = w->d_unsorted.p; cx.h_unsorted = w->h_unsorted;
    cx.max_tiles = w->d_tiles.cap; cx.max_jobs = w->d_sj.cap; cx.timing = e->timing >= 1;
    cx.stats = w->sort_stats;
    {
      u32 max_used = 1;
      for (u32 j = 0; j < J; j++) max_used = std::max(max_used, w->batch_jobs[j].n_used);
      cx.sym_bits = 1;
      while ((1u << cx.sym_bits) < max_used) cx.sym_bits++;
      cx.max_used = max_used;
      cx.h_jobs = w->batch_jobs.data();
    }
    if (e->timing >= 1) cudaEventRecord(w->ev_sort[0], st);
    int rc = b2k_bwt_batch(&cx, st, w->d_jobs.p, ids, ns, w->d_text.p, w->d_bwt.p);
    if (e->timing >= 1) cudaEventRecord(w->ev_sort[1], st);
    w->sort_stats = cx.stats;
    if (rc) return rc;
  }
  {
    StageTimer tm(e, st, w->ev, &w->stage_ms[3]);
    B2_TRY(launch_mtf(w, J, mplan));
  }
  // exact group counts: the ranking heap sorts size their shared memory by the largest block
  B2_CUDA_CHECK(cudaMemcpyAsync(w->batch_jobs.data(), w->d_jobs.p, J * sizeof(B2Job), cudaMemcpyDeviceToHost, st));
  B2_CUDA_CHECK(cudaStreamSynchronize(st));
  max_g = 1;
  u32 max_alpha = 2;
  for (u32 j = 0; j < J; j++) {
    max_g = std::max(max_g, w->batch_jobs[j].n_groups);
    max_alpha = std::max(max_alpha, w->batch_jobs[j].n_used + 2);
  }
  {
    StageTimer tm(e, st, w->ev, &w->stage_ms[4]);
    B2_TRY(b2k_entropy(st, w->d_jobs.p, J, max_g, gpos, w->d_mtf.p, w->d_ghist.p, w->d_gdist.p, w->d_rank3.p, w->d_rank4.p, w->d_sel.p,
                       w->d_selprev.p, w->d_gpack.p, w->d_gselcost.p, w->d_ehist.p, w->d_leaves.p, w->d_wl.p, w->d_lens.p, w->d_estat.p, w->d_selcost.p,
                       w->d_cost.p, w->d_low.p, e->level, max_alpha, w->d_scalars.p + 8, &w->launches));
  }
  {
    StageTimer tm(e, st, w->ev, &w->stage_ms[5]);
    u64 *d_total = (u64 *)(w->d_scalars.p + 2);
    B2_TRY(b2k_bits_layout(st, w->d_jobs.p, J, d_total));
    u64 total_words = 0;
    B2_CUDA_CHECK(cudaMemcpyAsync(&total_words, d_total, sizeof(u64), cudaMemcpyDeviceToHost, st));
    B2_CUDA_CHECK(cudaStreamSynchronize(st));
    B2_TRY(w->d_bits.ensure(total_words + 64));
    B2_CUDA_CHECK(cudaMemsetAsync(w->d_bits.p, 0, (total_words + 8) * sizeof(u32), st));
    B2_TRY(b2k_pack(st, w->d_jobs.p, J, w->d_mtf.p, w->d_sel.p, w->d_lens.p, w->d_selpos.p, w->d_bits.p, e->level, gpos));
    w->launches += 2;
  }
  B2_CUDA_CHECK(cudaMemcpyAsync(w->batch_jobs.data(), w->d_jobs.p, J * sizeof(B2Job), cudaMemcpyDeviceToHost, st));
  B2_CUDA_CHECK(cudaStreamSynchronize(st));
  if (e->timing >= 1) { float ms = 0; if (cudaEventElapsedTime(&ms, w->ev_sort[0], w->ev_sort[1]) == cudaSuccess) w->sort_ms += ms; }
  return 0;
}

inline u32 rotl1(u32 x) { return (x << 1) | (x >> 31); }

// Slices of one chunk per tactic -> de-duplicated jobs (SURVEY §9 R3); ids start at first_id.
int plan_chunk(b2_encoder *e, u32 c, ChunkPlan &P, std::vector<B2Job> &add, size_t first_id, u64 &addpos) {
  const int level = e->level;
  std::vector<std::pair<u32, u32>> slices[4];       // (start, len) relative to the chunk
  int nt = 1;
  slices[0].push_back({0, P.len});                                   // single (:1236, slices = 1)
  if (level == 9) {
    nt = 4;
    u32 size = P.len / 4, stop = 0;                                  // parts_4 (:1238-1254)
    for (u32 count = 1; count <= 4; count++) {
      u32 start = stop;
      stop = (count == 4) ? P.len : count * size;
      slices[1].push_back({start, stop - start});
    }
    for (int k = 0; k < 2; k++) {                                    // segmented_1/2 (:1266-1291)
      u32 ns = e->nseg[2 * c + k];
      P.n_seg[k] = ns;
      if (ns == 0) slices[2 + k].push_back({0, 0});                  // seg.Is_Empty -> one empty block (:1283-1284)
      else if (ns == 1) slices[2 + k].push_back({0, P.len});         // trivial segmentation = [len] (:102-104)
      else {
        const std::vector<u32> &cuts = e->seg[2 * c + k];
        u32 index_start = 0;
        for (u32 s = 0; s < ns; s++) { slices[2 + k].push_back({index_start, cuts[s] - index_start}); index_start = cuts[s]; }
      }
    }
  }
  std::map<std::pair<u32, u32>, u32> seen;
  add.clear(); addpos = 0;
  for (int t = 0; t < nt; t++) {
    P.tactic_jobs[t].clear();
    for (auto &sl : slices[t]) {
      auto it = seen.find(sl);
      u32 id;
      if (it == seen.end()) {
        id = (u32)(first_id + add.size());
        seen[sl] = id;
        B2Job j; memset(&j, 0, sizeof j);
        j.raw_off = P.start + sl.first; j.raw_len = sl.second;
        add.push_back(j);
        addpos += std::min<u64>((u64)sl.second * 5 / 4 + 264, (u64)level * 100000 + 320);
      } else id = it->second;
      P.tactic_jobs[t].push_back(id);
    }
  }
  P.n_tactics = nt;
  return 0;
}

// One BZip2 stream of a batch call: `n` bytes at d_in + off, reference size_hint `hint`.
// Filled by encode_streams: where its bytes start in e->d_out and how many there are.
struct StreamDesc {
  u64 off, n; i64 hint;
  u64 out_off, out_len;        // bytes
  u32 chunk0, n_chunks;
};

// Encodes streams[*] (all resident in d_in) into disjoint regions of e->d_out.  Every stream is what
// one `Encode (option, size_hint)` call writes (bzip2-encoding.adb:1413-1431); chunks of all streams
// share the batches, so many small entries fill the device as well as one large stream.
void reset_workspace_stats(b2_encoder *e) {
  for (auto *w : e->ws) {
    memset(&w->sort_stats, 0, sizeof w->sort_stats);
    w->launches = 0; w->blocks = 0; w->block_bytes = 0; w->sort_ms = 0;
    for (int i = 0; i < 8; i++) w->stage_ms[i] = 0;
  }
}

void merge_workspace_stats(b2_encoder *e) {
  for (auto *w : e->ws) {
    e->sort_stats.scatter_launches += w->sort_stats.scatter_launches;
    e->sort_stats.scatter_elems += w->sort_stats.scatter_elems;
    e->sort_stats.scatter_ms += w->sort_stats.scatter_ms;
    e->sort_stats.rounds += w->sort_stats.rounds;
    e->sort_stats.sorted_elems_round0 += w->sort_stats.sorted_elems_round0;
    e->sort_stats.sorted_elems_later += w->sort_stats.sorted_elems_later;
    e->sort_stats.launches += w->sort_stats.launches;
    e->launches_other += w->launches;
    e->stats.blocks += w->blocks; e->stats.block_bytes += w->block_bytes; e->stats.sort_ms += w->sort_ms;
    for (int i = 1; i < 8; i++) e->stats.stage_ms[i] += w->stage_ms[i];
  }
  e->stats.sort_rounds = e->sort_stats.rounds;
  e->stats.sort_elems_round0 = e->sort_stats.sorted_elems_round0;
  e->stats.sort_elems_later = e->sort_stats.sorted_elems_later;
  e->stats.scatter_launches = e->sort_stats.scatter_launches;
  e->stats.scatter_elems = e->sort_stats.scatter_elems;
  e->stats.scatter_ms = e->sort_stats.scatter_ms;
  e->stats.kernel_launches = e->launches_other + e->sort_stats.launches;
}

int encode_chunks(b2_encoder *e, const u8 *d_in, std::vector<StreamDesc> &streams, std::vector<u32> &chunk_stream, bool followed,
                  ShardState *sh);

int encode_streams(b2_encoder *e, const u8 *d_in, std::vector<StreamDesc> &streams) {
  cudaStream_t st = e->st;
  const int level = e->level;
  B2_CUDA_CHECK(cudaStreamSynchronize(e->st2));     // nothing of an earlier (failed) call may still be following a chain
  e->shard.open = e->shard.cut = e->shard.encoded = false;
  e->trace.clear(); e->chunks.clear(); e->nseg.clear(); e->seg.clear();
  i64 win_lo, win_hi;
  balance_window(level, win_lo, win_hi);
  const i64 full_cap = (i64)level * 100000;
  // ---- A1 chunk cutting --------------------------------------------------------------------------
  std::vector<u32> chunk_stream;          // stream of every chunk
  bool followed = false;                  // the segmentation already ran, following the chunk chain
  {
    StageTimer tm(e, st, e->ev, &e->stats.stage_ms[0]);
    // a stream whose RLE1 output cannot reach the smallest possible capacity is a single chunk
    const u64 small_limit = (u64)((win_lo / 2 - 16) * 4 / 5);
    for (size_t si = 0; si < streams.size(); si++) {
      StreamDesc &S = streams[si];
      e->stats.streams++; e->stats.input_bytes += S.n;
      S.chunk0 = (u32)e->chunks.size();
      if (S.n <= small_limit) {
        const i64 rest = S.hint < 0 ? -1 : S.hint;                        // stream_rest before the first read
        const i64 cap = (rest >= win_lo && rest <= win_hi) ? rest / 2 : full_cap;   // (:1416-1424)
        e->chunks.push_back(B2Chunk{S.off, (u32)S.n, (u32)cap, 0, 0});
      } else {
        const u32 max_chunks = (u32)(S.n / (40000ull * level) + 16);
        B2_TRY(e->d_chunks.ensure(max_chunks));
        const size_t ct = (size_t)(S.n / 2048 + 2);
        B2_TRY(e->d_cut_first.ensure(ct)); B2_TRY(e->d_cut_last.ensure(ct)); B2_TRY(e->d_cut_tsum.ensure(ct));
        B2_TRY(e->d_cut_carry.ensure(ct)); B2_TRY(e->d_cut_tincl.ensure(ct));
        B2_TRY(e->d_cut_gs.ensure(ct * 128)); B2_TRY(e->d_cut_gm.ensure(ct * 128));
        B2CutWork cw{e->d_cut_first.p, e->d_cut_last.p, e->d_cut_tsum.p, e->d_cut_carry.p, e->d_cut_tincl.p, e->d_cut_gs.p, e->d_cut_gm.p};
        // A single large stream: the segmentation of a chunk starts as soon as the chain has cut it
        // (k_segment on a second stream follows the chain's progress counter) instead of after the
        // whole chain, which is one warp walking from chunk to chunk.
        const bool follow = level == 9 && streams.size() == 1 && e->timing < 2;
        if (follow) {
          B2_TRY(e->d_seg.ensure((size_t)max_chunks * 2 * B2_MAX_SEG));
          B2_TRY(e->d_nseg.ensure((size_t)max_chunks * 2));
          B2_CUDA_CHECK(cudaMemsetAsync(e->d_nseg.p, 0xFE, (size_t)max_chunks * 2 * sizeof(u32), st));   // "not there yet"
        }
        B2_TRY(b2k_cut(st, d_in + S.off, S.n, S.hint, level, win_lo, win_hi, e->d_chunks.p, e->d_scalars.p, max_chunks, &cw,
                       follow ? e->d_scalars.p + 12 : nullptr, follow ? e->ev_fork : nullptr));
        e->launches_other += 5;
        if (follow) {
          B2_CUDA_CHECK(cudaStreamWaitEvent(e->st2, e->ev_fork, 0));
          B2_TRY(b2k_segment(e->st2, d_in + S.off, e->d_chunks.p, max_chunks, e->d_T.p, e->d_seg.p, e->d_nseg.p, e->d_scalars.p + 12, nullptr, nullptr));
          B2_CUDA_CHECK(cudaEventRecord(e->ev_join, e->st2));
          e->launches_other += 1;
          followed = true;
        }
        u32 nc = 0;
        B2_CUDA_CHECK(cudaMemcpyAsync(&nc, e->d_scalars.p, sizeof(u32), cudaMemcpyDeviceToHost, st));
        B2_CUDA_CHECK(cudaStreamSynchronize(st));
        if (nc > max_chunks) B2_FAIL(B2_ERR_INTERNAL, "chunk table overflow");
        const size_t base = e->chunks.size();
        e->chunks.resize(base + nc);
        B2_CUDA_CHECK(cudaMemcpyAsync(e->chunks.data() + base, e->d_chunks.p, nc * sizeof(B2Chunk), cudaMemcpyDeviceToHost, st));
        B2_CUDA_CHECK(cudaStreamSynchronize(st));
        for (size_t c = base; c < e->chunks.size(); c++) e->chunks[c].start += S.off;
      }
      S.n_chunks = (u32)e->chunks.size() - S.chunk0;
      for (u32 c = 0; c < S.n_chunks; c++) chunk_stream.push_back((u32)si);
    }
  }
  return encode_chunks(e, d_in, streams, chunk_stream, followed, nullptr);
}

// Everything after the cutting: e->chunks holds the chunks (offsets into d_in), chunk_stream their streams.
// sh != nullptr: the chunks are one shard of a stream (b2_shard_encode) — the candidates that can still win are
// kept for b2_shard_finish instead of being concatenated, and no header / footer is written.
int encode_chunks(b2_encoder *e, const u8 *d_in, std::vector<StreamDesc> &streams, std::vector<u32> &chunk_stream, bool followed,
                  ShardState *sh) {
  cudaStream_t st = e->st;
  const int level = e->level;
  const u32 n_chunks = (u32)e->chunks.size();
  e->stats.chunks += n_chunks;
  e->trace.resize(n_chunks);
  if (sh) { sh->cands.assign((size_t)n_chunks * 4, ShardCand{0, 0, 0, 0, 0, 0}); sh->n_tactics.assign(n_chunks, 0); }
  // ---- A3 segmentation of every chunk --------------------------------------------------------------
  {
    StageTimer tm(e, st, e->ev, &e->stats.stage_ms[0]);
    if (!followed) {
      B2_TRY(e->d_chunks.ensure(n_chunks));
      B2_CUDA_CHECK(cudaMemcpyAsync(e->d_chunks.p, e->chunks.data(), n_chunks * sizeof(B2Chunk), cudaMemcpyHostToDevice, st));
    }
    if (level == 9) {
      e->nseg.assign((size_t)n_chunks * 2, 0);
      e->seg.assign((size_t)n_chunks * 2, std::vector<u32>());
      if (!followed) {
        B2_TRY(e->d_seg.ensure((size_t)n_chunks * 2 * B2_MAX_SEG));
        B2_TRY(e->d_nseg.ensure((size_t)n_chunks * 2));
        B2_TRY(b2k_segment(st, d_in, e->d_chunks.p, n_chunks, e->d_T.p, e->d_seg.p, e->d_nseg.p, nullptr, nullptr, nullptr));
        e->launches_other += 1;
      }
    }
    B2_CUDA_CHECK(cudaStreamSynchronize(st));
  }
  // Cut lists of the chunks below `upto`, brought to the host.  When the segmentation is still following
  // the chunk chain on the other stream, this waits for exactly those chunks, so that the first batches
  // start while later chunks are still being segmented.
  u32 seg_have = 0;
  auto fetch_seg = [&](u32 upto) -> int {
    if (level != 9 || upto <= seg_have) return 0;
    upto = std::min(n_chunks, std::max(upto, seg_have + 64));
    for (u32 tries = 0;; tries++) {
      B2_CUDA_CHECK(cudaMemcpyAsync(e->nseg.data() + 2 * (size_t)seg_have, e->d_nseg.p + 2 * (size_t)seg_have,
                                    2 * (size_t)(upto - seg_have) * sizeof(u32), cudaMemcpyDeviceToHost, st));
      B2_CUDA_CHECK(cudaStreamSynchronize(st));
      bool all = true, gave_up = false;
      for (u32 k = 2 * seg_have; k < 2 * upto; k++) {
        if (e->nseg[k] == B2_SEG_PENDING) { all = false; break; }
        if (e->nseg[k] == B2_SEG_GAVE_UP) gave_up = true;
      }
      if (all && gave_up) {
        // a CTA following the chain never saw its chunk (the chain kernel was not co-scheduled: time-sliced GPU):
        // segment every chunk again now that the chain is complete
        B2_CUDA_CHECK(cudaStreamSynchronize(e->st2));
        B2_CUDA_CHECK(cudaMemcpyAsync(e->d_chunks.p, e->chunks.data(), n_chunks * sizeof(B2Chunk), cudaMemcpyHostToDevice, st));
        B2_TRY(b2k_segment(st, d_in, e->d_chunks.p, n_chunks, e->d_T.p, e->d_seg.p, e->d_nseg.p, nullptr, nullptr, nullptr));
        e->launches_other += 1;
        followed = false;
        continue;
      }
      if (all) break;
      if (!followed || tries > 2000000u) B2_FAIL(B2_ERR_INTERNAL, "segmentation results missing");
      std::this_thread::sleep_for(std::chrono::microseconds(50));
    }
    // only chunks with a real segmentation need their cut lists (a trivial one is just [len])
    for (u32 k = 2 * seg_have; k < 2 * upto; k++) {
      const u32 ns = e->nseg[k];
      if (ns > B2_MAX_SEG) B2_FAIL(B2_ERR_INTERNAL, "segment table overflow");
      if (ns > 1) {
        e->seg[k].resize(ns);
        B2_CUDA_CHECK(cudaMemcpyAsync(e->seg[k].data(), e->d_seg.p + (size_t)k * B2_MAX_SEG, ns * sizeof(u32), cudaMemcpyDeviceToHost, st));
      }
    }
    B2_CUDA_CHECK(cudaStreamSynchronize(st));
    seg_have = upto;
    return 0;
  };
  // ---- output regions ------------------------------------------------------------------------------
  u64 out_total = 0;
  for (auto &S : streams) {
    S.out_off = out_total;
    out_total += (b2_bound(S.n) + 1024ull * S.n_chunks + 71) & ~7ull;
  }
  if (!sh) {
    B2_TRY(e->d_out.ensure(out_total / 4 + 16));
    B2_CUDA_CHECK(cudaMemsetAsync(e->d_out.p, 0, (out_total / 4 + 8) * sizeof(u32), st));
    B2_CUDA_CHECK(cudaStreamSynchronize(st));           // output zeroed before any concat
  }
  // ---- batches of whole chunks: planned by this thread, run by the workers as they appear -----------
  std::vector<ChunkPlan> plans(n_chunks);
  std::deque<Batch> batches;                          // grows while the workers run (references stay valid)
  std::mutex bmu;
  std::condition_variable bcv;
  bool planned_all = false;                           // guarded by bmu
  // ---- pipelined batches ---------------------------------------------------------------------
  // serial state carried from chunk to chunk inside a stream (:1305-1345)
  std::vector<B2StreamEnd> ends(streams.size());
  for (size_t si = 0; si < streams.size(); si++) { ends[si].out_off = streams[si].out_off; ends[si].end_bit = 32; ends[si].crc = 0; ends[si].pad = 0; }
  u64 out_words_needed = 0;
  const int W = (e->timing >= 2) ? 1 : std::max<int>(1, (int)e->ws.size());
  reset_workspace_stats(e);
  std::atomic<u32> next{0};
  std::mutex mu;
  std::condition_variable cv;
  u32 turn = 0;                 // next batch to resolve (guarded by mu)
  u32 planned_total = 0xFFFFFFFFu;   // number of batches, known once the planning is complete (guarded by mu)
  int err = 0;
  std::string err_msg;
  auto worker = [&](int wi) {
    cudaSetDevice(e->device);
    Workspace *w = e->ws[wi];
    for (;;) {
      const u32 b = next.fetch_add(1);
      Batch *B = nullptr;
      {
        std::unique_lock<std::mutex> lk(bmu);
        bcv.wait(lk, [&] { return b < batches.size() || planned_all; });
        if (b < batches.size()) B = &batches[b];
      }
      if (!B) break;
      int rc = 0;
      {
        std::lock_guard<std::mutex> lk(mu);
        if (err) rc = err;
      }
      if (!rc) rc = run_batch(e, w, d_in, B->jobs);
      std::unique_lock<std::mutex> lk(mu);
      cv.wait(lk, [&] { return turn == b; });
      if (!rc && !err && sh) {
        // one shard of a stream: the bit offset its first chunk lands on is not known yet.  A candidate can
        // only win if it is the best for one of the eight incoming offsets (:1319-1325 compares flushed
        // bytes); those are copied, each from a 64-bit boundary, into an arena that outlives the batch.
        std::vector<B2ConcatItem> items;
        u64 cursor = 0;
        for (u32 c = B->c0; c < B->c1; c++) {
          ChunkPlan &P = plans[c];
          u64 bits[4] = {0, 0, 0, 0};
          for (int t = 0; t < P.n_tactics; t++) for (u32 id : P.tactic_jobs[t]) bits[t] += w->batch_jobs[id].nbits;
          u32 keep = 0;
          for (u32 phase = 0; phase < 8; phase++) {
            int best = 0;
            for (int t = 0; t < P.n_tactics; t++) if (((phase + bits[t]) >> 3) < ((phase + bits[best]) >> 3)) best = t;
            keep |= 1u << best;
          }
          sh->n_tactics[c] = P.n_tactics;
          b2_chunk_trace tr; memset(&tr, 0, sizeof tr);
          tr.start = sh->base + P.start; tr.len = P.len; tr.dyn_capacity = P.cap; tr.n_seg1 = P.n_seg[0]; tr.n_seg2 = P.n_seg[1];
          tr.winner = -1;
          for (int t = 0; t < P.n_tactics; t++) {
            tr.bits[t] = bits[t];
            ShardCand &cd = sh->cands[(size_t)c * 4 + t];
            cd.arena = b; cd.nbits = bits[t]; cd.kept = (keep >> t) & 1u; cd.blocks = (u32)P.tactic_jobs[t].size(); cd.fold = 0;
            for (u32 id : P.tactic_jobs[t]) cd.fold = rotl1(cd.fold) ^ w->batch_jobs[id].crc;      // (:990) from a zero CRC
            if (!cd.kept) continue;
            cursor = (cursor + 63) & ~63ull;
            cd.word_off = cursor >> 5;
            for (u32 id : P.tactic_jobs[t]) {
              const B2Job &jb = w->batch_jobs[id];
              items.push_back(B2ConcatItem{jb.bits_off, jb.nbits, cursor});
              cursor += jb.nbits;
            }
          }
          e->trace[c] = tr;
        }
        while (sh->arenas.size() <= b) sh->arenas.push_back(new DevBuf<u32>());
        DevBuf<u32> *ar = sh->arenas[b];
        rc = ar->ensure((cursor >> 5) + 8);
        if (!rc && cudaMemsetAsync(ar->p, 0, ((cursor >> 5) + 8) * sizeof(u32), w->st) != cudaSuccess) rc = B2_ERR_CUDA;
        if (!rc) rc = w->d_items.ensure(items.size() + 1);
        if (!rc && !items.empty() && cudaMemcpyAsync(w->d_items.p, items.data(), items.size() * sizeof(B2ConcatItem), cudaMemcpyHostToDevice, w->st) != cudaSuccess) rc = B2_ERR_CUDA;
        for (size_t i0 = 0; !rc && i0 < items.size(); i0 += 65535) {
          rc = b2k_concat(w->st, w->d_items.p + i0, (u32)std::min<size_t>(65535, items.size() - i0), w->d_bits.p, ar->p);
          w->launches += 1;
        }
        if (!rc && cudaStreamSynchronize(w->st) != cudaSuccess) { rc = B2_ERR_CUDA; b2_set_error(__FILE__, __LINE__, cudaGetErrorString(cudaGetLastError())); }
      } else if (!rc && !err) {
        // winners of the chunks of this batch, in order
        std::vector<B2ConcatItem> items;
        for (u32 c = B->c0; c < B->c1; c++) {
          ChunkPlan &P = plans[c];
          B2StreamEnd &E = ends[chunk_stream[c]];
          b2_chunk_trace tr; memset(&tr, 0, sizeof tr);
          tr.start = P.start - streams[chunk_stream[c]].off; tr.len = P.len; tr.dyn_capacity = P.cap;
          tr.n_seg1 = P.n_seg[0]; tr.n_seg2 = P.n_seg[1];
          int best = 0;
          const u32 in_bits = (u32)(E.end_bit & 7);
          for (int t = 0; t < P.n_tactics; t++) {
            u64 bits = 0;
            for (u32 id : P.tactic_jobs[t]) bits += w->batch_jobs[id].nbits;
            tr.bits[t] = bits;
            tr.bytes[t] = (in_bits + bits) >> 3;      // destination_index: whole bytes flushed
          }
          for (int t = 0; t < P.n_tactics; t++) if (tr.bytes[t] < tr.bytes[best]) best = t;
          tr.winner = best;
          for (u32 id : P.tactic_jobs[best]) {
            const B2Job &jb = w->batch_jobs[id];
            items.push_back(B2ConcatItem{jb.bits_off, jb.nbits, E.out_off * 8 + E.end_bit});
            E.end_bit += jb.nbits;
            E.crc = rotl1(E.crc) ^ jb.crc;             // (:990)
          }
          e->trace[c] = tr;
          const StreamDesc &S = streams[chunk_stream[c]];
          const u64 region = (b2_bound(S.n) + 1024ull * S.n_chunks + 71) & ~7ull;
          if ((E.end_bit + 128) / 8 > region) { rc = B2_ERR_INTERNAL; b2_set_error(__FILE__, __LINE__, "output bound exceeded"); break; }
        }
        if (!rc) {
          StageTimer tm(e, w->st, w->ev, &w->stage_ms[6]);
          rc = w->d_items.ensure(items.size());
          if (!rc && cudaMemcpyAsync(w->d_items.p, items.data(), items.size() * sizeof(B2ConcatItem), cudaMemcpyHostToDevice, w->st) != cudaSuccess) rc = B2_ERR_CUDA;
          for (size_t i0 = 0; !rc && i0 < items.size(); i0 += 65535)
            rc = b2k_concat(w->st, w->d_items.p + i0, (u32)std::min<size_t>(65535, items.size() - i0), w->d_bits.p, e->d_out.p);
          if (!rc && cudaStreamSynchronize(w->st) != cudaSuccess) { rc = B2_ERR_CUDA; b2_set_error(__FILE__, __LINE__, cudaGetErrorString(cudaGetLastError())); }
          w->launches += 1;
        }
      }
      if (rc && !err) { err = rc; err_msg = g_last_error; }
      turn = b + 1;
      lk.unlock();
      cv.notify_all();
    }
  };
  // One batch instead of two is worth 4 % on a 1 GiB text stream (the latency-bound kernels run once over all the
  // blocks; profiles/r02c_variants.jsonl).  When the whole call is expected to fit - about 2.8 positions per input byte,
  // 52 bytes of workspace per position including the slack of the buffers - into what the workspace already holds
  // plus the device memory that is free right now (less a margin for the caller), the batch limit is raised to that.
  // An estimate that turns out too low just starts a second batch.
  size_t batch_limit = e->batch_positions;
  if (!e->batch_positions_fixed && W == 1) {
    u64 total_len = 0;
    for (u32 c = 0; c < n_chunks; c++) total_len += e->chunks[c].len;
    const u64 est = (u64)((double)total_len * 2.8) + (u64)n_chunks * 4096;
    size_t free_b = 0, total_b = 0;
    if (est > batch_limit && cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
      const size_t have = e->ws[0]->d_keysA.cap;                       // positions the workspace holds already
      const size_t margin = (size_t)12 << 30;
      size_t can = have + (free_b > margin ? (size_t)((double)(free_b - margin) / 52.0) : 0);
      can = std::min<size_t>(can, 4200000000ull);                      // 32-bit arena offsets: below 2^32 less one chunk's worst case
      if (est <= can) batch_limit = can;
    }
  }
  std::vector<std::thread> th;
  for (int i = 0; i < W; i++) th.emplace_back(worker, i);
  int plan_rc = 0;
  std::string plan_msg;
  {
    u32 published = 0;
    auto publish = [&](Batch &&bt) {
      { std::lock_guard<std::mutex> lk(bmu); batches.push_back(std::move(bt)); }
      bcv.notify_all();
      published++;
    };
    Batch cur; cur.c0 = 0;
    u64 positions = 0;
    std::vector<B2Job> add;
    for (u32 c = 0; c < n_chunks && !plan_rc; c++) {
      ChunkPlan &P = plans[c];
      P.start = e->chunks[c].start; P.len = e->chunks[c].len; P.cap = e->chunks[c].cap;
      P.n_seg[0] = P.n_seg[1] = 0;
      u64 addpos = 0;
      if ((plan_rc = fetch_seg(c + 1))) break;                 // may wait for the segmentation of this chunk
      if ((plan_rc = plan_chunk(e, c, P, add, cur.jobs.size(), addpos))) break;
      // While the segmentation is still following the chunk chain the device has nothing else to do: the
      // first batch is kept small so that it starts as soon as its few chunks are cut and segmented.
      const size_t limit = (followed && published == 0) ? std::min(e->first_batch_positions, batch_limit) : batch_limit;
      if (!cur.jobs.empty() && (positions + addpos > limit || cur.jobs.size() + add.size() > e->batch_jobs_max)) {
        cur.c1 = c;
        publish(std::move(cur));
        cur = Batch(); cur.c0 = c; positions = 0;
        if ((plan_rc = plan_chunk(e, c, P, add, 0, addpos))) break;      // job ids restart in the new batch
      }
      cur.jobs.insert(cur.jobs.end(), add.begin(), add.end());
      positions += addpos;
    }
    if (!plan_rc && n_chunks) { cur.c1 = n_chunks; publish(std::move(cur)); }
    if (plan_rc) {
      plan_msg = g_last_error;
      std::lock_guard<std::mutex> lk(mu);
      if (!err) { err = plan_rc; err_msg = plan_msg; }
    }
    size_t nb_total = 0;
    { std::lock_guard<std::mutex> lk(bmu); planned_all = true; nb_total = batches.size(); }
    bcv.notify_all();
    { std::lock_guard<std::mutex> lk(mu); planned_total = (u32)nb_total; }
    cv.notify_all();
  }
  if (e->progress) {
    // Feedback / User_abort (zip.ads:301-306, zip-compress-bzip2_e.adb:78-96): the callback runs on the calling
    // thread (never on a worker) after every batch; a non-zero result stops the remaining batches
    u64 total_bytes = 0;
    for (u32 c = 0; c < n_chunks; c++) total_bytes += e->chunks[c].len;
    std::unique_lock<std::mutex> lk(mu);
    u32 seen = 0;
    for (;;) {
      cv.wait(lk, [&] { return turn > seen || err || (planned_total != 0xFFFFFFFFu && turn >= planned_total); });
      if (turn > seen) {
        seen = turn;
        u64 done_bytes = 0;
        { std::lock_guard<std::mutex> lb(bmu); for (u32 b = 0; b < seen && b < batches.size(); b++) for (u32 c = batches[b].c0; c < batches[b].c1; c++) done_bytes += e->chunks[c].len; }
        lk.unlock();
        const int stop = e->progress(e->progress_user, done_bytes, total_bytes);
        lk.lock();
        if (stop && !err) { err = B2_ERR_ABORTED; err_msg = "aborted by the progress callback (User_abort)"; }
      }
      if (err || (planned_total != 0xFFFFFFFFu && turn >= planned_total)) break;
    }
  }
  for (auto &t : th) t.join();
  if (followed) B2_CUDA_CHECK(cudaStreamSynchronize(e->st2));
  (void)out_words_needed;
  if (err) { g_last_error = err_msg; return err; }
  // ---- stream headers and footers (:1384-1407) on the device ----------------------------------------
  if (!sh) {
    B2_TRY(e->d_ends.ensure(ends.size()));
    B2_CUDA_CHECK(cudaMemcpyAsync(e->d_ends.p, ends.data(), ends.size() * sizeof(B2StreamEnd), cudaMemcpyHostToDevice, st));
    B2_TRY(b2k_stream_ends(st, e->d_ends.p, (u32)ends.size(), level, e->d_out.p));
    e->launches_other += 1;
    B2_CUDA_CHECK(cudaStreamSynchronize(st));
    for (size_t si = 0; si < streams.size(); si++) streams[si].out_len = (ends[si].end_bit + 80 + 7) >> 3;
  }
  merge_workspace_stats(e);
  return 0;
}

// The whole stream, input resident on the device.  Output bytes land at the start of e->d_out.
int encode_device(b2_encoder *e, const u8 *d_in, u64 n, i64 size_hint, u64 *out_len) {
  std::vector<StreamDesc> streams(1);
  streams[0] = StreamDesc{0, n, size_hint, 0, 0, 0, 0};
  B2_TRY(encode_streams(e, d_in, streams));
  *out_len = streams[0].out_len;
  return 0;
}

}  // namespace

// =============================================================================================
// ---- archive side -----------------------------------------------------------------------------------
namespace {
int zip_crc_device(b2_encoder *e, const u8 *d_in, u32 n_entries, const u64 *offs, const u64 *sizes) {
  // Zip CRC-32 of every entry (zip-crc_crypto.adb:31-61), results in e->d_zcrc
  if (!e->d_zt.p) {
    B2ZipCrcTables *zt = new B2ZipCrcTables();
    b2k_make_zipcrc_tables(zt);
    int rc = e->d_zt.ensure(1);
    if (!rc && cudaMemcpy(e->d_zt.p, zt, sizeof(B2ZipCrcTables), cudaMemcpyHostToDevice) != cudaSuccess) rc = B2_ERR_CUDA;
    delete zt;
    if (rc) B2_FAIL(rc, "zip crc tables");
  }
  std::vector<B2ZipTile> tiles;
  std::vector<B2ZipEntry> ents(n_entries);
  for (u32 i = 0; i < n_entries; i++) {
    const u64 nt = (sizes[i] + B2_ZIP_TILE - 1) / B2_ZIP_TILE;
    ents[i] = B2ZipEntry{sizes[i], (u32)tiles.size(), (u32)nt};
    for (u64 k = 0; k < nt; k++) tiles.push_back(B2ZipTile{offs[i], offs[i] + sizes[i] - (nt - 1 - k) * (u64)B2_ZIP_TILE});
  }
  if (tiles.size() >= (1ull << 31)) B2_FAIL(B2_ERR_ARGUMENT, "too much input for one archive call");
  B2_TRY(e->d_ztiles.ensure(tiles.size() + 1));
  B2_TRY(e->d_zents.ensure(n_entries + 1));
  B2_TRY(e->d_zpartial.ensure(tiles.size() + 1));
  B2_TRY(e->d_zcrc.ensure(n_entries + 1));
  if (!tiles.empty()) B2_CUDA_CHECK(cudaMemcpyAsync(e->d_ztiles.p, tiles.data(), tiles.size() * sizeof(B2ZipTile), cudaMemcpyHostToDevice, e->st));
  if (n_entries) B2_CUDA_CHECK(cudaMemcpyAsync(e->d_zents.p, ents.data(), n_entries * sizeof(B2ZipEntry), cudaMemcpyHostToDevice, e->st));
  B2_TRY(b2k_zipcrc(e->st, d_in, e->d_ztiles.p, (u32)tiles.size(), e->d_zents.p, n_entries, e->d_zt.p, e->d_zpartial.p, e->d_zcrc.p));
  e->launches_other += 2;
  B2_CUDA_CHECK(cudaStreamSynchronize(e->st));     // the host vectors above go out of scope
  return 0;
}

struct HeaderSpan { u64 dst; std::vector<u8> bytes; };
}  // namespace


extern "C" {

const char *b2_last_error(void) { return g_last_error.c_str(); }

uint64_t b2_bound(uint64_t n) { return n + n / 50 + 4096; }

int b2_create(int level, int device, b2_encoder **out) {
  if (!out) B2_FAIL(B2_ERR_ARGUMENT, "out is NULL");
  *out = nullptr;
  if (level != 1 && level != 4 && level != 9) B2_FAIL(B2_ERR_ARGUMENT, "level must be 1, 4 or 9");
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev == 0) B2_FAIL(B2_ERR_CUDA, "no CUDA device available (b2gpu has no CPU fallback)");
  if (device < 0 || device >= ndev) B2_FAIL(B2_ERR_ARGUMENT, "bad device index");
  B2_CUDA_CHECK(cudaSetDevice(device));
  b2_encoder *e = new b2_encoder();
  e->level = level; e->device = device;
  memset(&e->stats, 0, sizeof e->stats);
  memset(&e->sort_stats, 0, sizeof e->sort_stats);
  // arena offsets are 32-bit: a batch plus one more chunk's worth of blocks must stay below 2^32 positions
  if (const char *s = getenv("B2GPU_BATCH_POSITIONS")) { long long v = atoll(s); if (v >= (1 << 20)) { e->batch_positions = (size_t)std::min<long long>(v, 3ll << 30); e->batch_positions_fixed = true; } }
  if (const char *s = getenv("B2GPU_FIRST_BATCH_POSITIONS")) { long long v = atoll(s); if (v >= (1 << 20)) e->first_batch_positions = (size_t)v; }
  if (const char *s = getenv("B2GPU_BATCH_JOBS")) { long long v = atoll(s); if (v >= 8) e->batch_jobs_max = (size_t)std::min<long long>(v, 65535); }   // grid.y of the per-(triple, block) kernels
  if (const char *s = getenv("B2GPU_PIPELINE")) { int v = atoi(s); if (v >= 1 && v <= 8) e->n_workspaces = v; }
  auto init = [&]() -> int {
    B2_CUDA_CHECK(cudaStreamCreateWithFlags(&e->st, cudaStreamNonBlocking));
    B2_CUDA_CHECK(cudaStreamCreateWithFlags(&e->st2, cudaStreamNonBlocking));
    B2_CUDA_CHECK(cudaStreamCreateWithFlags(&e->cst, cudaStreamNonBlocking));
    B2_CUDA_CHECK(cudaEventCreateWithFlags(&e->ev_up, cudaEventDisableTiming));
    B2_CUDA_CHECK(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
    B2_CUDA_CHECK(cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming));
    B2_CUDA_CHECK(cudaEventCreate(&e->ev[0])); B2_CUDA_CHECK(cudaEventCreate(&e->ev[1]));
    B2_CUDA_CHECK(cudaEventCreate(&e->ev_call[0])); B2_CUDA_CHECK(cudaEventCreate(&e->ev_call[1]));
    for (int i = 0; i < e->n_workspaces; i++) {
      Workspace *w = new Workspace();
      e->ws.push_back(w);
      B2_CUDA_CHECK(cudaStreamCreateWithFlags(&w->st, cudaStreamNonBlocking));
      B2_CUDA_CHECK(cudaEventCreate(&w->ev[0])); B2_CUDA_CHECK(cudaEventCreate(&w->ev[1]));
      B2_CUDA_CHECK(cudaEventCreate(&w->ev_sort[0])); B2_CUDA_CHECK(cudaEventCreate(&w->ev_sort[1]));
    }
    // constant tables
    {
      std::vector<B2CrcTables> ct(1);
      b2k_make_crc_tables(ct.data());
      B2_TRY(e->d_ct.ensure(1));
      B2_CUDA_CHECK(cudaMemcpy(e->d_ct.p, ct.data(), sizeof(B2CrcTables), cudaMemcpyHostToDevice));
    }
    // T[c] = -(p * Log (p)), p = Real (c) * inv_window_size, window 16_000 (data_segmentation.adb:44-50)
    std::vector<double> T(16002, 0.0);
    const double inv = 1.0 / 16000.0;
    for (int c = 1; c <= 16001; c++) { double p = (double)c * inv; T[c] = -(p * std::log(p)); }
    B2_TRY(e->d_T.ensure(T.size()));
    B2_CUDA_CHECK(cudaMemcpy(e->d_T.p, T.data(), T.size() * sizeof(double), cudaMemcpyHostToDevice));
    B2_TRY(e->d_scalars.ensure(16));
    return 0;
  };
  const int rc = init();
  if (rc) { const std::string msg = g_last_error; b2_destroy(e); g_last_error = msg; return rc; }
  *out = e;
  return 0;
}

void b2_destroy(b2_encoder *e) {
  if (!e) return;
  cudaSetDevice(e->device);
  if (e->st) cudaStreamSynchronize(e->st);
  if (e->cst) { cudaStreamSynchronize(e->cst); cudaStreamDestroy(e->cst); }
  if (e->ev_up) cudaEventDestroy(e->ev_up);
  for (int i = 0; i < 2; i++) if (e->stream.buf[i]) cudaFree(e->stream.buf[i]);
  for (auto *w : e->ws) { if (w->st) cudaStreamSynchronize(w->st); w->release(); delete w; }
  e->ws.clear();
  e->d_ct.release(); e->d_T.release(); e->d_in.release(); e->d_out.release(); e->d_chunks.release();
  e->d_scalars.release(); e->d_seg.release(); e->d_nseg.release(); e->d_ends.release(); e->d_packitems.release(); e->d_packed.release(); e->d_cut_first.release(); e->d_cut_last.release();
  e->d_cut_tsum.release(); e->d_cut_carry.release(); e->d_cut_tincl.release(); e->d_cut_gs.release(); e->d_cut_gm.release();
  e->d_vstream.release(); e->d_vlcol.release(); e->d_vrle.release(); e->d_vsel.release(); e->d_vlink.release(); e->d_vchain.release();
  e->d_vscal.release(); e->d_vcand.release(); e->d_vblocks.release();
  e->d_zt.release(); e->d_ztiles.release(); e->d_zents.release(); e->d_zcopies.release(); e->d_zpartial.release(); e->d_zcrc.release();
  if (e->ev[0]) cudaEventDestroy(e->ev[0]);
  if (e->ev[1]) cudaEventDestroy(e->ev[1]);
  if (e->ev_call[0]) cudaEventDestroy(e->ev_call[0]);
  if (e->ev_call[1]) cudaEventDestroy(e->ev_call[1]);
  if (e->st2) { cudaStreamSynchronize(e->st2); cudaStreamDestroy(e->st2); }
  if (e->ev_fork) cudaEventDestroy(e->ev_fork);
  if (e->ev_join) cudaEventDestroy(e->ev_join);
  if (e->st) cudaStreamDestroy(e->st);
  delete e;
}

int b2_encode_stream_device(b2_encoder *e, const uint8_t *d_in, uint64_t n, int64_t size_hint,
                            uint8_t *d_out, uint64_t out_cap, uint64_t *out_len) {
  if (!e || !out_len || (n && !d_in)) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  B2_NO_STREAM(e);
  B2_CUDA_CHECK(cudaSetDevice(e->device));
  u64 len = 0;
  if (e->timing) cudaEventRecord(e->ev_call[0], e->st);
  B2_TRY(encode_device(e, d_in, n, size_hint, &len));
  *out_len = len;
  if (len > out_cap) B2_FAIL(B2_ERR_OUTPUT_TOO_SMALL, "output buffer too small");
  if (d_out) B2_CUDA_CHECK(cudaMemcpyAsync(d_out, e->d_out.p, len, cudaMemcpyDeviceToDevice, e->st));
  if (e->timing) cudaEventRecord(e->ev_call[1], e->st);
  B2_CUDA_CHECK(cudaStreamSynchronize(e->st));
  if (e->timing) { float ms = 0; cudaEventElapsedTime(&ms, e->ev_call[0], e->ev_call[1]); e->stats.call_ms += ms; }
  return 0;
}

int b2_encode_stream(b2_encoder *e, const uint8_t *in, uint64_t n, int64_t size_hint,
                     uint8_t *out, uint64_t out_cap, uint64_t *out_len) {
  if (!e || !out_len || (n && !in)) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  B2_NO_STREAM(e);
  B2_CUDA_CHECK(cudaSetDevice(e->device));
  B2_TRY(e->d_in.ensure(n + 256));
  if (e->timing) cudaEventRecord(e->ev_call[0], e->st);
  {
    StageTimer tm(e, e->st, e->ev, &e->stats.stage_ms[7]);
    if (n) B2_CUDA_CHECK(cudaMemcpyAsync(e->d_in.p, in, n, cudaMemcpyHostToDevice, e->st));
    B2_CUDA_CHECK(cudaMemsetAsync(e->d_in.p + n, 0, 128, e->st));
  }
  u64 len = 0;
  B2_TRY(encode_device(e, e->d_in.p, n, size_hint, &len));
  *out_len = len;
  if (len > out_cap) B2_FAIL(B2_ERR_OUTPUT_TOO_SMALL, "output buffer too small");
  {
    StageTimer tm(e, e->st, e->ev, &e->stats.stage_ms[7]);
    if (out) B2_CUDA_CHECK(cudaMemcpyAsync(out, e->d_out.p, len, cudaMemcpyDeviceToHost, e->st));
    if (e->timing) cudaEventRecord(e->ev_call[1], e->st);
    B2_CUDA_CHECK(cudaStreamSynchronize(e->st));
  }
  if (e->timing) { float ms = 0; cudaEventElapsedTime(&ms, e->ev_call[0], e->ev_call[1]); e->stats.call_ms += ms; }
  return 0;
}

int b2_encode_batch(b2_encoder *e, uint32_t n_entries, const uint8_t *in, const uint64_t *in_offsets,
                    const uint64_t *sizes, const int64_t *size_hints, uint8_t *out, uint64_t out_cap,
                    uint64_t *out_offsets, uint64_t *out_lens) {
  if (!e || (n_entries && (!in_offsets || !sizes || !out_offsets || !out_lens))) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  B2_NO_STREAM(e);
  B2_CUDA_CHECK(cudaSetDevice(e->device));
  u64 total_in = 0;
  for (u32 i = 0; i < n_entries; i++) total_in = std::max<u64>(total_in, in_offsets[i] + sizes[i]);
  if (total_in && !in) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  B2_TRY(e->d_in.ensure(total_in + 256));
  if (e->timing) cudaEventRecord(e->ev_call[0], e->st);
  if (total_in) B2_CUDA_CHECK(cudaMemcpyAsync(e->d_in.p, in, total_in, cudaMemcpyHostToDevice, e->st));
  B2_CUDA_CHECK(cudaMemsetAsync(e->d_in.p + total_in, 0, 128, e->st));
  std::vector<StreamDesc> streams(n_entries);
  for (u32 i = 0; i < n_entries; i++) streams[i] = StreamDesc{in_offsets[i], sizes[i], size_hints ? size_hints[i] : -1, 0, 0, 0, 0};
  B2_TRY(encode_streams(e, e->d_in.p, streams));
  // pack the streams back to back (8-byte aligned) and bring them to the host
  std::vector<B2PackItem> items(n_entries);
  u64 pos = 0;
  for (u32 i = 0; i < n_entries; i++) {
    items[i] = B2PackItem{streams[i].out_off, pos, streams[i].out_len};
    out_offsets[i] = pos; out_lens[i] = streams[i].out_len;
    pos += (streams[i].out_len + 7) & ~7ull;
  }
  if (pos > out_cap) B2_FAIL(B2_ERR_OUTPUT_TOO_SMALL, "output buffer too small");
  if (n_entries) {
    B2_TRY(e->d_packitems.ensure(n_entries));
    B2_TRY(e->d_packed.ensure(pos + 64));
    B2_CUDA_CHECK(cudaMemcpyAsync(e->d_packitems.p, items.data(), n_entries * sizeof(B2PackItem), cudaMemcpyHostToDevice, e->st));
    B2_TRY(b2k_pack_streams(e->st, e->d_packitems.p, n_entries, (const u8 *)e->d_out.p, e->d_packed.p));
    if (out && pos) B2_CUDA_CHECK(cudaMemcpyAsync(out, e->d_packed.p, pos, cudaMemcpyDeviceToHost, e->st));
  }
  if (e->timing) cudaEventRecord(e->ev_call[1], e->st);
  B2_CUDA_CHECK(cudaStreamSynchronize(e->st));
  if (e->timing) { float ms = 0; cudaEventElapsedTime(&ms, e->ev_call[0], e->ev_call[1]); e->stats.call_ms += ms; }
  return 0;
}

// ---- one stream over several handles (devices / processes): SURVEY.md §8e ----------------------------
// Chunks are independent given where they start; the only data that cross shards are scalars: the start of
// the next shard's first chunk (the cutting is a chain, bzip2-encoding.adb:1160-1208), and per shard, for
// each of the 8 possible incoming bit offsets, the bits it appends and how it folds the combined CRC
// (:990, :1319-1345).  No bulk data moves between devices.
uint64_t b2_shard_margin(int level) { return 10ull * 100000ull * (u64)level + 4096; }

int b2_shard_plan(uint64_t n, int n_shards, int level, int stagger_permille, uint64_t *bounds) {
  if (!bounds || n_shards < 1) return B2_ERR_ARGUMENT;
  (void)level;
  // Shard r can only start once shard r-1 has cut its chunks, so its share is smaller by the factor
  // (1 - stagger): all shards then finish together (stagger = encode rate / cutting rate of one device).
  if (stagger_permille < 0) {
    stagger_permille = 12;
    if (const char *sv = getenv("B2GPU_SHARD_STAGGER")) { int v = atoi(sv); if (v >= 0 && v < 500) stagger_permille = v; }
  }
  const double q = 1.0 - stagger_permille / 1000.0;
  double tot = 0, w = 1;
  for (int r = 0; r < n_shards; r++) { tot += w; w *= q; }
  double acc = 0; w = 1;
  bounds[0] = 0;
  for (int r = 0; r < n_shards; r++) {
    acc += w; w *= q;
    u64 b = (u64)((double)n * (acc / tot));
    b &= ~4095ull;                                    // device pointers of the slices stay aligned for vector loads
    if (b < bounds[r]) b = bounds[r];
    bounds[r + 1] = r + 1 == n_shards ? n : std::min<u64>(b, n);
  }
  return 0;
}

}  // extern "C"

namespace {
// What a shard does to the bit offset and the combined CRC, given the incoming ones (:990, :1319-1345).
void link_step(const b2_shard_link &l, u64 &bit, u32 &crc) {
  const u32 ph = (u32)(bit & 7);
  const u32 k = l.crc_rot[ph] & 31u;
  crc = (k ? ((crc << k) | (crc >> (32 - k))) : crc) ^ l.crc_fold[ph];
  bit += l.total_bits[ph];
}

// The four steps of a shard on this handle, for b2_shard_* and for the windows of b2_stream_*.
// d_in: the stream bytes [base, base + n_local) on the device, followed by 128 zero bytes.
int shard_load(b2_encoder *e, const u8 *d_in, u64 base, u64 n_local, u64 own_end, bool last, i64 size_hint) {
  B2_CUDA_CHECK(cudaStreamSynchronize(e->st2));
  ShardState &sh = e->shard;
  sh.open = sh.cut = sh.encoded = false;
  sh.d_in = d_in; sh.base = base; sh.n_local = n_local; sh.own_end = own_end; sh.last = last; sh.hint = size_hint;
  // the scans of the cutting do not depend on where the first chunk starts: they run while the shards
  // before this one are still cutting
  const size_t ct = (size_t)(n_local / 2048 + 2);
  B2_TRY(e->d_cut_first.ensure(ct)); B2_TRY(e->d_cut_last.ensure(ct)); B2_TRY(e->d_cut_tsum.ensure(ct));
  B2_TRY(e->d_cut_carry.ensure(ct)); B2_TRY(e->d_cut_tincl.ensure(ct));
  B2_TRY(e->d_cut_gs.ensure(ct * 128)); B2_TRY(e->d_cut_gm.ensure(ct * 128));
  B2CutWork cw{e->d_cut_first.p, e->d_cut_last.p, e->d_cut_tsum.p, e->d_cut_carry.p, e->d_cut_tincl.p, e->d_cut_gs.p, e->d_cut_gm.p};
  B2_TRY(b2k_cut_scans(e->st, sh.d_in, n_local, &cw));
  e->launches_other += 4;
  sh.open = true;
  return 0;
}

int shard_cut(b2_encoder *e, u64 entry, u64 *handoff) {
  ShardState &sh = e->shard;
  cudaStream_t st = e->st;
  const int level = e->level;
  e->trace.clear(); e->chunks.clear(); e->nseg.clear(); e->seg.clear();
  i64 win_lo, win_hi;
  balance_window(level, win_lo, win_hi);
  const u64 own = sh.own_end > entry ? sh.own_end - entry : 0;
  const u32 max_chunks = (u32)(own / (40000ull * level) + 16);
  B2_TRY(e->d_chunks.ensure(max_chunks));
  B2CutWork cw{e->d_cut_first.p, e->d_cut_last.p, e->d_cut_tsum.p, e->d_cut_carry.p, e->d_cut_tincl.p, e->d_cut_gs.p, e->d_cut_gm.p};
  const bool follow = level == 9 && e->timing < 2;
  if (level == 9) {
    B2_TRY(e->d_seg.ensure((size_t)max_chunks * 2 * B2_MAX_SEG));
    B2_TRY(e->d_nseg.ensure((size_t)max_chunks * 2));
    B2_CUDA_CHECK(cudaMemsetAsync(e->d_nseg.p, 0xFE, (size_t)max_chunks * 2 * sizeof(u32), st));
  }
  // the last shard walks to the end of the stream; the others stop at the first chunk that belongs to the next one
  const u64 stop = sh.last ? sh.n_local : sh.own_end - sh.base;
  B2_TRY(b2k_cut_chain(st, sh.d_in, sh.n_local, sh.hint, level, win_lo, win_hi, e->d_chunks.p, e->d_scalars.p, max_chunks, &cw,
                       follow ? e->d_scalars.p + 12 : nullptr, follow ? e->ev_fork : nullptr, sh.base, entry - sh.base, stop));
  e->launches_other += 1;
  if (follow) {
    B2_CUDA_CHECK(cudaStreamWaitEvent(e->st2, e->ev_fork, 0));
    B2_TRY(b2k_segment(e->st2, sh.d_in, e->d_chunks.p, max_chunks, e->d_T.p, e->d_seg.p, e->d_nseg.p, e->d_scalars.p + 12, nullptr, nullptr));
    B2_CUDA_CHECK(cudaEventRecord(e->ev_join, e->st2));
    e->launches_other += 1;
  }
  u32 sc[4] = {0, 0, 0, 0};
  B2_CUDA_CHECK(cudaMemcpyAsync(sc, e->d_scalars.p, sizeof sc, cudaMemcpyDeviceToHost, st));
  B2_CUDA_CHECK(cudaStreamSynchronize(st));
  const u32 nc = sc[0];
  if (nc > max_chunks) B2_FAIL(B2_ERR_INTERNAL, "chunk table overflow");
  e->chunks.resize(nc);
  if (nc) B2_CUDA_CHECK(cudaMemcpy(e->chunks.data(), e->d_chunks.p, nc * sizeof(B2Chunk), cudaMemcpyDeviceToHost));
  sh.entry = entry;
  sh.handoff = sh.base + ((u64)sc[2] | ((u64)sc[3] << 32));
  *handoff = sh.handoff;
  sh.cut = true;
  // followed: the segmentation is running behind the chain on the other stream
  return 0;
}

int shard_encode(b2_encoder *e, b2_shard_link *link) {
  ShardState &sh = e->shard;
  const u32 nc = (u32)e->chunks.size();
  std::vector<StreamDesc> streams(1);
  streams[0] = StreamDesc{0, sh.n_local, sh.hint, 0, 0, 0, nc};
  std::vector<u32> chunk_stream(nc, 0u);
  const bool followed = e->level == 9 && e->timing < 2;
  B2_TRY(encode_chunks(e, sh.d_in, streams, chunk_stream, followed, &sh));
  // what the shard does to the bit offset and to the combined CRC, for every incoming offset mod 8
  for (u32 phase0 = 0; phase0 < 8; phase0++) {
    u64 total = 0; u32 rot = 0, fold = 0, ph = phase0;
    for (u32 c = 0; c < nc; c++) {
      const ShardCand *cd = &sh.cands[(size_t)c * 4];
      int best = 0;
      for (int t = 0; t < sh.n_tactics[c]; t++) if (((ph + cd[t].nbits) >> 3) < ((ph + cd[best].nbits) >> 3)) best = t;
      total += cd[best].nbits; ph = (u32)((ph + cd[best].nbits) & 7);
      const u32 k = cd[best].blocks & 31u;
      fold = (k ? ((fold << k) | (fold >> (32 - k))) : fold) ^ cd[best].fold;
      rot = (rot + cd[best].blocks) & 31u;
    }
    link->total_bits[phase0] = total; link->crc_rot[phase0] = rot; link->crc_fold[phase0] = fold;
  }
  sh.encoded = true;
  return 0;
}

int shard_finish(b2_encoder *e, u64 bit_offset, u32 crc_in, u8 *out, int out_is_device, u64 out_cap,
                 u64 *out_byte_offset, u64 *out_len, u8 *first_byte, u8 *last_byte) {
  ShardState &sh = e->shard;
  cudaStream_t st = e->st;
  const bool first = sh.base == 0 && sh.entry == 0, last = sh.last;
  if (first && bit_offset != 32) B2_FAIL(B2_ERR_ARGUMENT, "the first shard starts behind the 32-bit stream header");
  const u64 byte0 = first ? 0 : bit_offset >> 3;         // first byte of the stream this shard touches
  const u64 lbit0 = bit_offset - 8 * byte0;              // its bits start here in its piece
  const u32 nc = (u32)e->chunks.size();
  // winners, in order (:1305-1345), now that the incoming offset is known
  std::vector<std::vector<B2ConcatItem>> items(sh.arenas.size());
  u64 lbit = lbit0;
  u32 crc = crc_in;
  for (u32 c = 0; c < nc; c++) {
    const ShardCand *cd = &sh.cands[(size_t)c * 4];
    const u32 in_bits = (u32)(lbit & 7);
    int best = 0;
    b2_chunk_trace &tr = e->trace[c];
    for (int t = 0; t < sh.n_tactics[c]; t++) tr.bytes[t] = (in_bits + cd[t].nbits) >> 3;
    for (int t = 0; t < sh.n_tactics[c]; t++) if (tr.bytes[t] < tr.bytes[best]) best = t;
    tr.winner = best;
    if (!cd[best].kept) B2_FAIL(B2_ERR_INTERNAL, "the winning candidate was not kept");
    if (cd[best].arena >= items.size()) B2_FAIL(B2_ERR_INTERNAL, "candidate arena missing");
    items[cd[best].arena].push_back(B2ConcatItem{cd[best].word_off, cd[best].nbits, lbit});
    lbit += cd[best].nbits;
    const u32 k = cd[best].blocks & 31u;
    crc = (k ? ((crc << k) | (crc >> (32 - k))) : crc) ^ cd[best].fold;
  }
  const u64 end_bit = lbit + (last ? 80 : 0);
  const u64 len = (end_bit + 7) >> 3;
  *out_len = len; *out_byte_offset = byte0;
  if (len > out_cap) B2_FAIL(B2_ERR_OUTPUT_TOO_SMALL, "output buffer too small");
  B2_TRY(e->d_out.ensure(len / 4 + 16));
  B2_CUDA_CHECK(cudaMemsetAsync(e->d_out.p, 0, (len / 4 + 8) * sizeof(u32), st));
  Workspace *w = e->ws[0];
  for (size_t a = 0; a < items.size(); a++) {
    if (items[a].empty()) continue;
    B2_TRY(w->d_items.ensure(items[a].size()));
    B2_CUDA_CHECK(cudaMemcpyAsync(w->d_items.p, items[a].data(), items[a].size() * sizeof(B2ConcatItem), cudaMemcpyHostToDevice, st));
    for (size_t i0 = 0; i0 < items[a].size(); i0 += 65535) {
      B2_TRY(b2k_concat(st, w->d_items.p + i0, (u32)std::min<size_t>(65535, items[a].size() - i0), sh.arenas[a]->p, e->d_out.p));
      e->launches_other += 1;
    }
    B2_CUDA_CHECK(cudaStreamSynchronize(st));          // d_items is reused by the next arena
  }
  if (first || last) {
    B2StreamEnd E{0, lbit, crc, (first ? 0u : 1u) | (last ? 0u : 2u)};
    B2_TRY(e->d_ends.ensure(1));
    B2_CUDA_CHECK(cudaMemcpyAsync(e->d_ends.p, &E, sizeof E, cudaMemcpyHostToDevice, st));
    B2_TRY(b2k_stream_ends(st, e->d_ends.p, 1, e->level, e->d_out.p));
    e->launches_other += 1;
  }
  if (out && len) B2_CUDA_CHECK(cudaMemcpyAsync(out, e->d_out.p, len, out_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
  u8 fb[2] = {0, 0};
  if (len) {
    B2_CUDA_CHECK(cudaMemcpyAsync(&fb[0], e->d_out.p, 1, cudaMemcpyDeviceToHost, st));
    B2_CUDA_CHECK(cudaMemcpyAsync(&fb[1], (const u8 *)e->d_out.p + (len - 1), 1, cudaMemcpyDeviceToHost, st));
  }
  if (e->timing) cudaEventRecord(e->ev_call[1], st);
  B2_CUDA_CHECK(cudaStreamSynchronize(st));
  if (first_byte) *first_byte = fb[0];
  if (last_byte) *last_byte = fb[1];
  if (e->timing) { float ms = 0; cudaEventElapsedTime(&ms, e->ev_call[0], e->ev_call[1]); e->stats.call_ms += ms; }
  sh.encoded = false; sh.cut = false; sh.open = false;
  return 0;
}
}  // namespace

extern "C" {

int b2_shard_resolve(const b2_shard_link *links, int n_shards, uint64_t *bit_offsets, uint32_t *crcs) {
  if (!links || !bit_offsets || !crcs || n_shards < 1) return B2_ERR_ARGUMENT;
  bit_offsets[0] = 32; crcs[0] = 0;                  // behind "BZh<level>" (:1384-1391)
  for (int r = 0; r < n_shards; r++) {
    u64 bit = bit_offsets[r]; u32 crc = crcs[r];
    link_step(links[r], bit, crc);
    bit_offsets[r + 1] = bit; crcs[r + 1] = crc;
  }
  return 0;
}

int b2_shard_open(b2_encoder *e, const uint8_t *in, int in_is_device, uint64_t base, uint64_t n_local,
                  uint64_t stream_size, int64_t size_hint, uint64_t own_end) {
  if (!e || (n_local && !in) || base + n_local > stream_size || own_end > stream_size || own_end < base) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  B2_NO_STREAM(e);
  B2_CUDA_CHECK(cudaSetDevice(e->device));
  B2_CUDA_CHECK(cudaStreamSynchronize(e->st2));
  e->shard.open = e->shard.cut = e->shard.encoded = false;
  if (e->timing) cudaEventRecord(e->ev_call[0], e->st);
  const u8 *d_in = in;
  if (!in_is_device) {
    B2_TRY(e->d_in.ensure(n_local + 256));
    if (n_local) B2_CUDA_CHECK(cudaMemcpyAsync(e->d_in.p, in, n_local, cudaMemcpyHostToDevice, e->st));
    B2_CUDA_CHECK(cudaMemsetAsync(e->d_in.p + n_local, 0, 128, e->st));
    d_in = e->d_in.p;
  }
  return shard_load(e, d_in, base, n_local, own_end, own_end >= stream_size, size_hint);
}

int b2_shard_cut(b2_encoder *e, uint64_t entry, uint64_t *handoff) {
  if (!e || !handoff) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  B2_NO_STREAM(e);
  ShardState &sh = e->shard;
  if (!sh.open) B2_FAIL(B2_ERR_ARGUMENT, "b2_shard_cut without b2_shard_open");
  if (entry < sh.base || entry > sh.base + sh.n_local) B2_FAIL(B2_ERR_ARGUMENT, "entry outside the shard's bytes");
  B2_CUDA_CHECK(cudaSetDevice(e->device));
  return shard_cut(e, entry, handoff);
}

int b2_shard_encode(b2_encoder *e, b2_shard_link *link) {
  if (!e || !link) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  B2_NO_STREAM(e);
  ShardState &sh = e->shard;
  if (!sh.cut) B2_FAIL(B2_ERR_ARGUMENT, "b2_shard_encode without b2_shard_cut");
  B2_CUDA_CHECK(cudaSetDevice(e->device));
  e->stats.streams++; e->stats.input_bytes += sh.handoff - sh.entry;
  return shard_encode(e, link);
}

int b2_shard_finish(b2_encoder *e, uint64_t bit_offset, uint32_t crc_in, uint8_t *out, int out_is_device, uint64_t out_cap,
                    uint64_t *out_byte_offset, uint64_t *out_len, uint8_t *first_byte, uint8_t *last_byte) {
  if (!e || !out_len || !out_byte_offset) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  B2_NO_STREAM(e);
  if (!e->shard.encoded) B2_FAIL(B2_ERR_ARGUMENT, "b2_shard_finish without b2_shard_encode");
  B2_CUDA_CHECK(cudaSetDevice(e->device));
  return shard_finish(e, bit_offset, crc_in, out, out_is_device, out_cap, out_byte_offset, out_len, first_byte, last_byte);
}

}  // extern "C"

// ---- one stream fed in pieces (b2_stream_*, DESIGN.md §6b) ---------------------------------------------------------
// Every window is a shard of the stream on this handle whose incoming bit offset and CRC are already known: it owns
// the chunks that start before base + W, and a chunk that starts there ends before base + W + M, so it sees the bytes
// of a one-shot encode.  The bytes from the next chunk start on move to the head of the other window buffer.
namespace {
struct ProgressShim { b2_progress_fn fn; void *user; u64 done0, total; };
int progress_shim(void *u, u64 done, u64 total) {
  (void)total;
  const ProgressShim *p = (const ProgressShim *)u;
  return p->fn(p->user, p->done0 + done, p->total);
}

void stream_close(b2_encoder *e) {
  cudaStreamSynchronize(e->cst);                       // no upload may read the caller's `in` after the call returns
  e->stream.open = false;
  e->shard.open = e->shard.cut = e->shard.encoded = false;
}

int stream_upload(b2_encoder *e, int b, u64 at, const u8 *in, u64 k) {
  if (!k) return 0;
  B2_CUDA_CHECK(cudaMemcpyAsync(e->stream.buf[b] + at, in, k, cudaMemcpyHostToDevice, e->cst));
  B2_CUDA_CHECK(cudaEventRecord(e->ev_up, e->cst));
  return 0;
}

// Encodes the held bytes as one window and writes its finished bytes to out[stream byte - out0].  A window that is
// not the last moves the bytes behind it to the other buffer and, before its blocks are encoded, enqueues the upload
// of what follows them from in[*taken, n), so that the copy runs under the encode.
int stream_window(b2_encoder *e, bool last, const u8 *in, u64 n, u64 *taken, u8 *out, u64 out_cap, u64 out0) {
  StreamState &S = e->stream;
  cudaStream_t st = e->st;
  u8 *d = S.buf[S.cur];
  if (e->timing) cudaEventRecord(e->ev_call[0], st);
  B2_CUDA_CHECK(cudaStreamWaitEvent(st, e->ev_up, 0));
  B2_CUDA_CHECK(cudaMemsetAsync(d + S.held, 0, 256, st));
  B2_TRY(shard_load(e, d, S.base, S.held, last ? S.base + S.held : S.base + S.window, last, S.hint));
  u64 handoff = 0;
  B2_TRY(shard_cut(e, S.base, &handoff));
  const int nxt = S.cur ^ 1;
  u64 next_held = 0;
  if (!last) {
    const u64 carry = S.base + S.held - handoff;
    B2_CUDA_CHECK(cudaMemcpyAsync(S.buf[nxt], d + (handoff - S.base), carry, cudaMemcpyDeviceToDevice, e->cst));
    const u64 k = std::min<u64>(S.window + S.margin - carry, n - *taken);
    B2_CUDA_CHECK(cudaEventRecord(e->ev_up, e->cst));
    B2_TRY(stream_upload(e, nxt, carry, in + *taken, k));
    *taken += k;
    next_held = carry + k;
  }
  b2_shard_link link;
  {
    ProgressShim ps{e->progress, e->progress_user, S.base, S.hint >= 0 ? (u64)S.hint : S.base + S.held};
    if (ps.fn) { e->progress = progress_shim; e->progress_user = &ps; }
    const int rc = shard_encode(e, &link);
    e->progress = ps.fn; e->progress_user = ps.user;
    B2_TRY(rc);
  }
  u64 bit = S.bit;
  u32 crc = S.crc;
  link_step(link, bit, crc);
  const u64 piece = S.base == 0 ? 0 : S.bit >> 3;      // where the window's bytes start in the stream
  u64 off = 0, len = 0;
  B2_TRY(shard_finish(e, S.bit, S.crc, out + (piece - out0), 0, out_cap - (piece - out0), &off, &len, nullptr, nullptr));
  if (off != piece) B2_FAIL(B2_ERR_INTERNAL, "window piece misplaced");
  if (len) out[piece - out0] |= S.tail;                // the byte held back from the window before
  S.trace.insert(S.trace.end(), e->trace.begin(), e->trace.end());
  e->stats.input_bytes += (last ? S.base + S.held : handoff) - S.base;
  S.bit = bit; S.crc = crc;
  if (last) { S.out_end = piece + len; S.tail = 0; S.held = 0; return 0; }
  S.out_end = bit >> 3;
  S.tail = (bit & 7) ? out[S.out_end - out0] : 0;
  S.cur = nxt; S.base = handoff; S.held = next_held;
  return 0;
}
// The two window buffers of W + M + 256 bytes (kept across streams and archives of the same W).
int stream_buffers(b2_encoder *e, u64 window_bytes) {
  StreamState &S = e->stream;
  const u64 W = window_bytes ? window_bytes : 512ull << 20;
  if (W < (1ull << 20)) B2_FAIL(B2_ERR_ARGUMENT, "window_bytes below 1 MiB");
  if (W > (1ull << 40)) B2_FAIL(B2_ERR_ARGUMENT, "window_bytes above 1 TiB");
  const u64 M = b2_shard_margin(e->level);
  const u64 bytes = W + M + 256;
  if (S.buf_bytes != bytes) {
    for (int i = 0; i < 2; i++) { if (S.buf[i]) cudaFree(S.buf[i]); S.buf[i] = nullptr; }
    S.buf_bytes = 0;
    for (int i = 0; i < 2; i++) {
      const cudaError_t ce = cudaMalloc((void **)&S.buf[i], bytes);
      if (ce != cudaSuccess) {
        for (int j = 0; j < 2; j++) { if (S.buf[j]) cudaFree(S.buf[j]); S.buf[j] = nullptr; }
        B2_FAIL(B2_ERR_ALLOC, cudaGetErrorString(ce));
      }
    }
    S.buf_bytes = bytes;
  }
  S.window = W; S.margin = M;
  return 0;
}

// A new stream of the window size of the buffers: nothing held, the first block behind "BZh<level>".
void stream_reset(b2_encoder *e, i64 size_hint) {
  StreamState &S = e->stream;
  S.hint = size_hint;
  S.cur = 0; S.base = 0; S.held = 0; S.bit = 32; S.crc = 0; S.out_end = 0; S.tail = 0;
  S.trace.clear();
}
}  // namespace

extern "C" {

uint64_t b2_stream_bound(b2_encoder *e, uint64_t n) {
  const u64 m = n + (e && e->stream.open ? e->stream.held : 0);
  return b2_bound(m) + 1024ull * (m / 40000 + 16) + 16;
}

int b2_stream_begin(b2_encoder *e, int64_t size_hint, uint64_t window_bytes) {
  if (!e) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  StreamState &S = e->stream;
  if (S.open) B2_FAIL(B2_ERR_ARGUMENT, "a stream is already open on this handle");
  if (e->zip.open) B2_FAIL(B2_ERR_ARGUMENT, "an archive is open on this handle (b2_zip_begin)");
  B2_CUDA_CHECK(cudaSetDevice(e->device));
  B2_TRY(stream_buffers(e, window_bytes));
  stream_reset(e, size_hint);
  e->stats.streams++;
  S.open = true;
  return 0;
}

int b2_stream_write(b2_encoder *e, const uint8_t *in, uint64_t n, uint8_t *out, uint64_t out_cap, uint64_t *out_len) {
  if (!e || !out_len || (n && !in) || !out) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  StreamState &S = e->stream;
  if (!S.open) B2_FAIL(B2_ERR_ARGUMENT, "b2_stream_write without b2_stream_begin");
  *out_len = 0;
  if (out_cap < b2_stream_bound(e, n)) B2_FAIL(B2_ERR_OUTPUT_TOO_SMALL, "output buffer below b2_stream_bound");
  const u64 out0 = S.out_end;
  auto run = [&]() -> int {
    B2_CUDA_CHECK(cudaSetDevice(e->device));
    const u64 full = S.window + S.margin;
    u64 taken = 0;
    for (;;) {
      const u64 k = std::min<u64>(full - S.held, n - taken);
      B2_TRY(stream_upload(e, S.cur, S.held, in + taken, k));
      S.held += k; taken += k;
      if (S.held < full) return 0;
      B2_TRY(stream_window(e, false, in, n, &taken, out, out_cap, out0));
    }
  };
  const int rc = run();
  if (rc) { const std::string msg = g_last_error; stream_close(e); g_last_error = msg; return rc; }
  B2_CUDA_CHECK(cudaStreamSynchronize(e->cst));          // the caller may reuse `in` once this returns
  *out_len = S.out_end - out0;
  return 0;
}

int b2_stream_end(b2_encoder *e, uint8_t *out, uint64_t out_cap, uint64_t *out_len) {
  if (!e || !out_len || !out) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  StreamState &S = e->stream;
  if (!S.open) B2_FAIL(B2_ERR_ARGUMENT, "b2_stream_end without b2_stream_begin");
  *out_len = 0;
  if (out_cap < b2_stream_bound(e, 0)) B2_FAIL(B2_ERR_OUTPUT_TOO_SMALL, "output buffer below b2_stream_bound");
  const u64 out0 = S.out_end;
  u64 taken = 0;
  int rc = cudaSetDevice(e->device) == cudaSuccess ? 0 : B2_ERR_CUDA;
  if (rc) b2_set_error(__FILE__, __LINE__, "cudaSetDevice");
  if (!rc) rc = stream_window(e, true, nullptr, 0, &taken, out, out_cap, out0);
  const std::string msg = g_last_error;
  stream_close(e);
  if (rc) { g_last_error = msg; return rc; }
  e->trace.swap(S.trace);
  S.trace.clear();
  *out_len = S.out_end - out0;
  return 0;
}

int b2_stream_abort(b2_encoder *e) {
  if (!e) return B2_ERR_ARGUMENT;
  if (e->stream.open) stream_close(e);
  return 0;
}

// One stream over the devices of several handles of this process: the north star's block-wise sharding
// (per-device streams, pinned host buffers, no collective).  One host thread per handle.
int b2_encode_stream_multi(b2_encoder **encs, int n_encs, const uint8_t *in, uint64_t n, int64_t size_hint,
                           uint8_t *out, uint64_t out_cap, uint64_t *out_len) {
  if (!encs || n_encs < 1 || !out_len || (n && !in)) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  for (int i = 0; i < n_encs; i++) if (!encs[i] || encs[i]->level != encs[0]->level) B2_FAIL(B2_ERR_ARGUMENT, "handles must share the block size");
  for (int i = 0; i < n_encs; i++) B2_NO_STREAM(encs[i]);
  const int level = encs[0]->level;
  u64 min_share = 64ull << 20;
  if (const char *sv = getenv("B2GPU_SHARD_MIN_BYTES")) { long long v = atoll(sv); if (v >= 65536) min_share = (u64)v; }
  const int ns = (int)std::max<u64>(1, std::min<u64>((u64)n_encs, n / min_share));
  if (ns == 1) return b2_encode_stream(encs[0], in, n, size_hint, out, out_cap, out_len);
  std::vector<u64> bounds(ns + 1);
  B2_TRY(b2_shard_plan(n, ns, level, -1, bounds.data()));
  const u64 margin = b2_shard_margin(level);
  std::vector<b2_shard_link> links(ns);
  std::vector<u64> entry(ns + 1, 0), bit_off(ns + 1, 0), piece_off(ns, 0), piece_len(ns, 0);
  std::vector<u32> crcs(ns + 1, 0);
  std::vector<u8> fb(ns, 0), lb(ns, 0);
  std::vector<int> rcs(ns, 0);
  std::vector<std::string> msgs(ns);
  std::mutex mu;
  std::condition_variable cv;
  int cut_done = 0, enc_done = 0;           // shards that have cut / encoded (guarded by mu)
  bool failed = false, resolved = false;
  auto run = [&](int r) {
    b2_encoder *e = encs[r];
    int rc = 0;
    auto fail = [&](int code) {
      rc = code; msgs[r] = g_last_error;
      { std::lock_guard<std::mutex> lk(mu); failed = true; }
      cv.notify_all();
    };
    const u64 lo = bounds[r], hi = std::min<u64>(n, bounds[r + 1] + (r + 1 < ns ? margin : 0));
    if ((rc = b2_shard_open(e, in + lo, 0, lo, hi - lo, n, size_hint, bounds[r + 1]))) { fail(rc); rcs[r] = rc; return; }
    {
      std::unique_lock<std::mutex> lk(mu);
      cv.wait(lk, [&] { return cut_done == r || failed; });
      if (failed) { rcs[r] = B2_ERR_INTERNAL; return; }
    }
    u64 ho = 0;
    if ((rc = b2_shard_cut(e, entry[r], &ho))) { fail(rc); rcs[r] = rc; return; }
    { std::lock_guard<std::mutex> lk(mu); entry[r + 1] = ho; cut_done = r + 1; }
    cv.notify_all();
    if ((rc = b2_shard_encode(e, &links[r]))) { fail(rc); rcs[r] = rc; return; }
    {
      std::unique_lock<std::mutex> lk(mu);
      enc_done++;
      if (enc_done == ns) {
        b2_shard_resolve(links.data(), ns, bit_off.data(), crcs.data());
        resolved = true;
        cv.notify_all();
      }
      cv.wait(lk, [&] { return resolved || failed; });
      if (failed) { rcs[r] = B2_ERR_INTERNAL; return; }
    }
    const u64 total = (bit_off[ns] + 80 + 7) >> 3;
    if (total > out_cap) { b2_set_error(__FILE__, __LINE__, "output buffer too small"); fail(B2_ERR_OUTPUT_TOO_SMALL); rcs[r] = B2_ERR_OUTPUT_TOO_SMALL; return; }
    const u64 b0 = r == 0 ? 0 : bit_off[r] >> 3;
    if ((rc = b2_shard_finish(e, bit_off[r], crcs[r], out + b0, 0, out_cap - b0, &piece_off[r], &piece_len[r], &fb[r], &lb[r]))) { fail(rc); rcs[r] = rc; return; }
  };
  std::vector<std::thread> th;
  for (int r = 0; r < ns; r++) th.emplace_back(run, r);
  for (auto &t : th) t.join();
  for (int r = 0; r < ns; r++) if (rcs[r] && !msgs[r].empty()) { g_last_error = msgs[r]; return rcs[r]; }
  for (int r = 0; r < ns; r++) if (rcs[r]) return rcs[r];
  // neighbouring pieces share a byte when the boundary is not on a byte: every piece wrote only its own bits
  // there, whichever copy landed last; the byte is the OR of all contributions
  std::map<u64, u8> edge;
  for (int r = 0; r < ns; r++) {
    if (!piece_len[r]) continue;
    edge[piece_off[r]] |= fb[r];
    edge[piece_off[r] + piece_len[r] - 1] |= lb[r];
  }
  for (auto &kv : edge) out[kv.first] = kv.second;
  *out_len = (bit_off[ns] + 80 + 7) >> 3;
  return 0;
}

// ---- decode / verify on the device (SURVEY.md §8f row 4) ---------------------------------------------------------
int b2_verify_stream(b2_encoder *e, const uint8_t *stream, int stream_is_device, uint64_t n, const uint8_t *expect,
                     int expect_is_device, uint64_t expect_n, b2_verify_result *res) {
  if (!e || !res || (n && !stream)) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  B2_NO_STREAM(e);
  memset(res, 0, sizeof *res);
  res->first_bad_block = -1; res->mismatch_at = ~0ull;
  B2_CUDA_CHECK(cudaSetDevice(e->device));
  cudaStream_t st = e->st;
  if (n < 14) { res->first_bad_status = 1; return 0; }                      // "BZh9" + footer is the shortest stream
  B2_TRY(e->d_vstream.ensure(n + 128));
  B2_CUDA_CHECK(cudaEventRecord(e->ev[0], st));
  B2_CUDA_CHECK(cudaMemcpyAsync(e->d_vstream.p, stream, n, stream_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
  B2_CUDA_CHECK(cudaMemsetAsync(e->d_vstream.p + n, 0, 128, st));
  u8 head[4];
  B2_CUDA_CHECK(cudaMemcpyAsync(head, e->d_vstream.p, 4, cudaMemcpyDeviceToHost, st));
  B2_CUDA_CHECK(cudaStreamSynchronize(st));
  if (head[0] != 'B' || head[1] != 'Z' || head[2] != 'h' || head[3] < '1' || head[3] > '9') { res->first_bad_status = 1; return 0; }
  const u32 level = head[3] - '0';
  res->level = level;
  const u32 max_n = level * 100000u;
  // candidates: every occurrence of the two magics, at any bit offset
  const u32 cap = (u32)std::min<u64>(n / 32 + 4096, 1u << 26);
  B2_TRY(e->d_vcand.ensure(cap));
  B2_TRY(e->d_vscal.ensure(8));
  B2_CUDA_CHECK(cudaMemsetAsync(e->d_vscal.p, 0, 8 * sizeof(u32), st));
  B2_TRY(b2k_verify_find(st, e->d_vstream.p, n, e->d_vcand.p, e->d_vscal.p, cap));
  u32 n_cand = 0;
  B2_CUDA_CHECK(cudaMemcpyAsync(&n_cand, e->d_vscal.p, sizeof(u32), cudaMemcpyDeviceToHost, st));
  B2_CUDA_CHECK(cudaStreamSynchronize(st));
  if (n_cand > cap) B2_FAIL(B2_ERR_INTERNAL, "too many block-magic candidates");
  std::vector<u64> cand(n_cand);
  if (n_cand) B2_CUDA_CHECK(cudaMemcpy(cand.data(), e->d_vcand.p, n_cand * sizeof(u64), cudaMemcpyDeviceToHost));
  std::sort(cand.begin(), cand.end());
  res->candidates = n_cand;
  // device copy of the expected bytes
  const u8 *d_expect = nullptr;
  if (expect) {
    if (expect_is_device) d_expect = expect;
    else {
      B2_TRY(e->d_in.ensure(expect_n + 256));
      if (expect_n) B2_CUDA_CHECK(cudaMemcpyAsync(e->d_in.p, expect, expect_n, cudaMemcpyHostToDevice, st));
      d_expect = e->d_in.p;
    }
    const unsigned long long none = ~0ull;
    B2_CUDA_CHECK(cudaMemcpyAsync(e->d_vscal.p + 2, &none, sizeof none, cudaMemcpyHostToDevice, st));
  }
  // waves of candidates in stream order; the chain "next block starts where this one ended" is followed as the
  // results arrive
  size_t wave = 2048;
  if (const char *sv = getenv("B2GPU_VERIFY_WAVE")) { long v = atol(sv); if (v >= 1) wave = (size_t)v; }
  u64 cur = 32, raw_total = 0;
  u32 combined = 0;
  bool done = false, failed = false;
  u64 n_chain = 0;
  std::vector<B2VBlock> blk;
  std::vector<u32> chain;
  for (size_t c0 = 0; c0 < cand.size() && !done && !failed;) {
    // skip candidates the chain has already passed (magic look-alikes inside a block)
    while (c0 < cand.size() && (cand[c0] >> 1) < cur) c0++;
    if (c0 >= cand.size()) break;
    const size_t c1 = std::min(cand.size(), c0 + wave);
    const u32 nb = (u32)(c1 - c0);
    blk.assign(nb, B2VBlock{});
    for (u32 k = 0; k < nb; k++) { blk[k].start_bit = cand[c0 + k] >> 1; blk[k].status = (cand[c0 + k] & 1) ? 0xFFu : 0u; }
    B2_TRY(e->d_vblocks.ensure(nb));
    B2_TRY(e->d_vlink.ensure((size_t)nb * (max_n + 32)));
    B2_TRY(e->d_vlcol.ensure((size_t)nb * (max_n + 32)));
    B2_TRY(e->d_vrle.ensure((size_t)nb * (max_n + 32)));
    B2_TRY(e->d_vsel.ensure((size_t)nb * 18016));
    B2_CUDA_CHECK(cudaMemcpyAsync(e->d_vblocks.p, blk.data(), nb * sizeof(B2VBlock), cudaMemcpyHostToDevice, st));
    B2_TRY(b2k_verify_decode(st, e->d_vstream.p, n, e->d_vblocks.p, nb, max_n, e->d_vlink.p, e->d_vlcol.p, e->d_vrle.p, e->d_vsel.p,
                             e->d_ct.p->byte_tab));
    e->launches_other += 1;
    B2_CUDA_CHECK(cudaMemcpyAsync(blk.data(), e->d_vblocks.p, nb * sizeof(B2VBlock), cudaMemcpyDeviceToHost, st));
    B2_CUDA_CHECK(cudaStreamSynchronize(st));
    chain.clear();
    size_t k = 0;
    while (k < nb) {
      if (blk[k].start_bit < cur) { k++; continue; }
      if (blk[k].start_bit > cur) { failed = true; res->first_bad_block = (int32_t)n_chain; res->first_bad_status = 20; break; }   // a gap: no block where one must start
      if (cand[c0 + k] & 1) {                        // the stream footer (:1395-1407): 48-bit magic, combined CRC
        u8 f[12];
        B2_CUDA_CHECK(cudaMemcpy(f, e->d_vstream.p + ((cur + 48) >> 3), 8, cudaMemcpyDeviceToHost));
        const u32 sh = (u32)((cur + 48) & 7);
        u64 w = 0;
        for (int q = 0; q < 8; q++) w = (w << 8) | f[q];
        res->stored_stream_crc = (u32)((w << sh) >> 32);
        res->computed_stream_crc = combined;
        const u64 end_bytes = (cur + 80 + 7) >> 3;
        done = true;
        if (end_bytes != n) { failed = true; res->first_bad_status = 21; }          // bytes behind the footer
        break;
      }
      const B2VBlock &b = blk[k];
      if (b.status != 0 || b.computed_crc != b.stored_crc) {
        failed = true; res->first_bad_block = (int32_t)n_chain; res->first_bad_status = b.status ? b.status : 30;
        break;
      }
      blk[k].raw_off = raw_total;
      raw_total += b.raw_len;
      combined = rotl1(combined) ^ b.stored_crc;
      cur = b.end_bit;
      chain.push_back((u32)k);
      n_chain++;
      k++;
    }
    if (d_expect && !chain.empty()) {
      B2_TRY(e->d_vchain.ensure(chain.size()));
      B2_CUDA_CHECK(cudaMemcpyAsync(e->d_vblocks.p, blk.data(), nb * sizeof(B2VBlock), cudaMemcpyHostToDevice, st));
      B2_CUDA_CHECK(cudaMemcpyAsync(e->d_vchain.p, chain.data(), chain.size() * sizeof(u32), cudaMemcpyHostToDevice, st));
      B2_TRY(b2k_verify_compare(st, e->d_vblocks.p, e->d_vchain.p, (u32)chain.size(), max_n, e->d_vrle.p, d_expect, expect_n,
                                (unsigned long long *)(e->d_vscal.p + 2)));
      e->launches_other += 1;
      B2_CUDA_CHECK(cudaStreamSynchronize(st));
    }
    c0 = c1;
  }
  if (!done && !failed) { failed = true; res->first_bad_block = (int32_t)n_chain; res->first_bad_status = 22; }   // no footer
  res->blocks = n_chain;
  res->decoded_bytes = raw_total;
  if (d_expect) {
    unsigned long long bad = ~0ull;
    B2_CUDA_CHECK(cudaMemcpy(&bad, e->d_vscal.p + 2, sizeof bad, cudaMemcpyDeviceToHost));
    res->mismatch_at = bad;
    if (bad == ~0ull && !failed && raw_total != expect_n) res->mismatch_at = std::min<u64>(raw_total, expect_n);
  }
  B2_CUDA_CHECK(cudaEventRecord(e->ev[1], st));
  B2_CUDA_CHECK(cudaStreamSynchronize(st));
  { float ms = 0; cudaEventElapsedTime(&ms, e->ev[0], e->ev[1]); res->ms = ms; }
  res->ok = (!failed && done && res->stored_stream_crc == res->computed_stream_crc && (!d_expect || res->mismatch_at == ~0ull)) ? 1 : 0;
  return 0;
}

// ---- archive side: Zip.Create for BZip2 entries (SURVEY.md §8f 1-3) ----
uint64_t b2_zip_bound(uint32_t n_entries, uint64_t total_name_bytes, uint64_t total_input_bytes) {
  // per entry: local header 30 + name + 20 (Zip64 extension), payload <= input (store fallback);
  // central header 46 + name + 28; end records 56 + 20 + 22
  return (u64)n_entries * (30 + 20 + 46 + 28) + 2 * total_name_bytes + total_input_bytes + 56 + 20 + 22;
}

int b2_zip_crc32(b2_encoder *e, const uint8_t *in, uint64_t n, uint32_t *crc) {
  if (!e || !crc || (n && !in)) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  B2_NO_STREAM(e);
  B2_CUDA_CHECK(cudaSetDevice(e->device));
  B2_TRY(e->d_in.ensure(n + 256));
  if (n) B2_CUDA_CHECK(cudaMemcpyAsync(e->d_in.p, in, n, cudaMemcpyHostToDevice, e->st));
  const u64 off = 0;
  B2_TRY(zip_crc_device(e, e->d_in.p, 1, &off, &n));
  B2_CUDA_CHECK(cudaMemcpy(crc, e->d_zcrc.p, sizeof(u32), cudaMemcpyDeviceToHost));
  return 0;
}

int b2_zip_create(b2_encoder *e, uint32_t n_entries, const uint8_t *in, const uint64_t *in_offsets, const uint64_t *sizes,
                  const char *names, const uint32_t *name_offsets, const uint32_t *dos_times, const uint32_t *flags,
                  int duplicates, uint8_t *out, uint64_t out_cap, uint64_t *out_len, b2_zip_entry_info *info) {
  if (!e || !out_len || (n_entries && (!in_offsets || !sizes || !names || !name_offsets))) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  B2_NO_STREAM(e);
  B2_CUDA_CHECK(cudaSetDevice(e->device));
  // entry names: back slashes become forward slashes (Unixify, zip-create.adb:180-192)
  std::vector<std::string> nm(n_entries);
  {
    std::unordered_set<std::string> seen;
    for (u32 i = 0; i < n_entries; i++) {
      if (name_offsets[i + 1] < name_offsets[i] || name_offsets[i + 1] - name_offsets[i] > 65535u) B2_FAIL(B2_ERR_ARGUMENT, "bad entry name length");
      nm[i] = b2zip::unixify(names + name_offsets[i], name_offsets[i + 1] - name_offsets[i]);
      if (duplicates == B2_ZIP_ERROR_ON_DUPLICATE && !seen.insert(nm[i]).second) {   // Duplicate_name (zip-create.adb:138-147)
        g_last_error = "Duplicate_name: Entry name = " + nm[i];
        return B2_ERR_DUPLICATE_NAME;
      }
    }
  }
  u64 total_in = 0;
  for (u32 i = 0; i < n_entries; i++) total_in = std::max<u64>(total_in, in_offsets[i] + sizes[i]);
  if (total_in && !in) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  B2_TRY(e->d_in.ensure(total_in + 256));
  if (e->timing) cudaEventRecord(e->ev_call[0], e->st);
  if (total_in) B2_CUDA_CHECK(cudaMemcpyAsync(e->d_in.p, in, total_in, cudaMemcpyHostToDevice, e->st));
  B2_CUDA_CHECK(cudaMemsetAsync(e->d_in.p + total_in, 0, 128, e->st));
  B2_TRY(zip_crc_device(e, e->d_in.p, n_entries, in_offsets, sizes));
  std::vector<u32> crc(n_entries);
  if (n_entries) B2_CUDA_CHECK(cudaMemcpyAsync(crc.data(), e->d_zcrc.p, n_entries * sizeof(u32), cudaMemcpyDeviceToHost, e->st));
  // every entry is one Encode call with the size known (zip-compress-bzip2_e.adb:122-129)
  std::vector<StreamDesc> streams(n_entries);
  for (u32 i = 0; i < n_entries; i++) streams[i] = StreamDesc{in_offsets[i], sizes[i], (i64)sizes[i], 0, 0, 0, 0};
  B2_TRY(encode_streams(e, e->d_in.p, streams));
  B2_CUDA_CHECK(cudaStreamSynchronize(e->st));

  // ---- layout: what Add_Stream (zip-create.adb:194-297) and Finish (:645-756) leave in the stream ----
  b2zip::ZipLayout L;
  std::vector<HeaderSpan> spans;
  std::vector<B2ZipCopy> copies;
  for (u32 i = 0; i < n_entries; i++) {
    u64 offset = 0, hbytes = 0;
    if (!L.open_entry(sizes[i], nm[i].size(), &offset, &hbytes)) B2_FAIL(B2_ERR_ARGUMENT, "Zip_Capacity_Exceeded: archive too large");
    // Compression_inefficient <=> the stream is not smaller than the input (zip-compress.adb:468-490) -> Store (:224-237)
    const bool stored = streams[i].out_len >= sizes[i];
    const u64 csize = stored ? sizes[i] : streams[i].out_len;
    HeaderSpan h{offset, {}};
    L.close_entry(nm[i], sizes[i], csize, crc[i], dos_times ? dos_times[i] : b2zip::ZipLayout::default_time, flags ? flags[i] : 0,
                  stored ? 0 : 12, h.bytes);
    const u64 payload = offset + hbytes;
    spans.push_back(std::move(h));
    const u64 src = stored ? in_offsets[i] : streams[i].out_off;
    for (u64 o = 0; o < csize; o += 65536) copies.push_back(B2ZipCopy{src + o, payload + o, (u32)std::min<u64>(65536, csize - o), stored ? 1u : 0u});
    if (info) { info[i].crc32 = crc[i]; info[i].zip_type = stored ? 0 : 12; info[i].reserved = 0; info[i].compressed_size = csize; info[i].local_header_offset = offset; }
  }
  {
    HeaderSpan d{L.pos, {}};
    if (!L.finish(d.bytes)) B2_FAIL(B2_ERR_ARGUMENT, "Zip_Capacity_Exceeded: archive too large");
    spans.push_back(std::move(d));
  }
  const u64 pos = L.pos;
  *out_len = pos;
  if (pos > out_cap) B2_FAIL(B2_ERR_OUTPUT_TOO_SMALL, "output buffer too small");
  if (!out) B2_FAIL(B2_ERR_ARGUMENT, "out is NULL");
  // payloads: gathered into the archive image on the device, one copy back; headers written by the host
  if (!copies.empty()) {
    if (copies.size() >= (1ull << 31)) B2_FAIL(B2_ERR_ARGUMENT, "too much output for one archive call");
    B2_TRY(e->d_zcopies.ensure(copies.size()));
    B2_TRY(e->d_packed.ensure(pos + 64));
    B2_CUDA_CHECK(cudaMemcpyAsync(e->d_zcopies.p, copies.data(), copies.size() * sizeof(B2ZipCopy), cudaMemcpyHostToDevice, e->st));
    B2_TRY(b2k_zip_gather(e->st, e->d_zcopies.p, (u32)copies.size(), (const u8 *)e->d_out.p, e->d_in.p, e->d_packed.p));
    e->launches_other += 1;
    const u64 first = copies.front().dst_off, last = copies.back().dst_off + copies.back().len;
    B2_CUDA_CHECK(cudaMemcpyAsync(out + first, e->d_packed.p + first, last - first, cudaMemcpyDeviceToHost, e->st));
  }
  if (e->timing) cudaEventRecord(e->ev_call[1], e->st);
  B2_CUDA_CHECK(cudaStreamSynchronize(e->st));
  for (const HeaderSpan &sp : spans) memcpy(out + sp.dst, sp.bytes.data(), sp.bytes.size());
  if (e->timing) { float ms = 0; cudaEventElapsedTime(&ms, e->ev_call[0], e->ev_call[1]); e->stats.call_ms += ms; }
  return 0;
}

}  // extern "C"

// ---- one archive written entry by entry (b2_zip_begin / add / finish, DESIGN.md §7c) ------------------------------------
// Entries of at most W bytes are queued in stream.buf[0] and encoded together as one batch of b2_zip_create when the
// next one would not fit.  A larger entry is one stream through the windows of b2_stream_* (size_hint = its size),
// written behind its local header, whose length is known before compression; its Zip CRC-32 is folded window by window.
namespace {
// Progress of the archive: `done` counts on from the archive's bytes encoded before the call, the total is what was added.
struct ProgressScope {
  b2_encoder *e;
  ProgressShim ps;
  ProgressScope(b2_encoder *e_, u64 done0, u64 total) : e(e_), ps{e_->progress, e_->progress_user, done0, total} {
    if (ps.fn) { e->progress = progress_shim; e->progress_user = &ps; }
  }
  ~ProgressScope() { e->progress = ps.fn; e->progress_user = ps.user; }
};

// Entries per batch of the queue.  Every queued entry costs device memory whatever its size: its chunk's two cut lists
// (18 KiB at level 9), its output region (at least 5 KiB) and up to six blocks of batch workspace (about 330 KiB each,
// DESIGN.md §3).  One entry per 32 KiB of W keeps that part of a batch below 64 bytes per byte of W.
u64 zip_queue_max(u64 window) { return std::max<u64>(32, window >> 15); }

void zip_close(b2_encoder *e) {
  cudaStreamSynchronize(e->cst);                       // no upload may read the caller's `in` after the call returns
  ZipState &Z = e->zip;
  Z.open = false;
  Z.layout = b2zip::ZipLayout();
  Z.names.clear(); Z.queue.clear();
  e->shard.open = e->shard.cut = e->shard.encoded = false;
}

// Encodes the queued entries as one batch and writes their archive bytes (local headers and payloads) to out[0 ..).
int zip_flush(b2_encoder *e, u8 *out) {
  ZipState &Z = e->zip;
  const u32 nq = (u32)Z.queue.size();
  if (!nq) return 0;
  cudaStream_t st = e->st;
  u8 *d = e->stream.buf[0];
  B2_CUDA_CHECK(cudaStreamWaitEvent(st, e->ev_up, 0));
  B2_CUDA_CHECK(cudaMemsetAsync(d + Z.q_end, 0, 128, st));
  std::vector<u64> offs(nq), sizes(nq);
  for (u32 i = 0; i < nq; i++) { offs[i] = Z.queue[i].off; sizes[i] = Z.queue[i].n; }
  B2_TRY(zip_crc_device(e, d, nq, offs.data(), sizes.data()));
  std::vector<u32> crc(nq);
  B2_CUDA_CHECK(cudaMemcpyAsync(crc.data(), e->d_zcrc.p, nq * sizeof(u32), cudaMemcpyDeviceToHost, st));
  std::vector<StreamDesc> streams(nq);
  for (u32 i = 0; i < nq; i++) streams[i] = StreamDesc{offs[i], sizes[i], (i64)sizes[i], 0, 0, 0, 0};
  {
    ProgressScope ps(e, Z.done, Z.added);
    B2_TRY(encode_streams(e, d, streams));
  }
  B2_CUDA_CHECK(cudaStreamSynchronize(st));
  b2zip::ZipLayout &L = Z.layout;
  const u64 base = L.pos;
  std::vector<HeaderSpan> spans;
  std::vector<B2ZipCopy> copies;
  for (u32 i = 0; i < nq; i++) {
    const ZipQueued &q = Z.queue[i];
    u64 offset = 0, hbytes = 0;
    if (!L.open_entry(q.n, q.name.size(), &offset, &hbytes)) B2_FAIL(B2_ERR_ARGUMENT, "Zip_Capacity_Exceeded: archive too large");
    const bool stored = streams[i].out_len >= q.n;       // Store fallback, as in b2_zip_create
    const u64 csize = stored ? q.n : streams[i].out_len;
    HeaderSpan h{offset - base, {}};
    L.close_entry(q.name, q.n, csize, crc[i], q.time, q.flags, stored ? 0 : 12, h.bytes);
    const u64 payload = offset - base + hbytes;
    spans.push_back(std::move(h));
    const u64 src = stored ? q.off : streams[i].out_off;
    for (u64 o = 0; o < csize; o += 65536) copies.push_back(B2ZipCopy{src + o, payload + o, (u32)std::min<u64>(65536, csize - o), stored ? 1u : 0u});
  }
  if (!copies.empty()) {
    B2_TRY(e->d_zcopies.ensure(copies.size()));
    B2_TRY(e->d_packed.ensure(L.pos - base + 64));
    B2_CUDA_CHECK(cudaMemcpyAsync(e->d_zcopies.p, copies.data(), copies.size() * sizeof(B2ZipCopy), cudaMemcpyHostToDevice, st));
    B2_TRY(b2k_zip_gather(st, e->d_zcopies.p, (u32)copies.size(), (const u8 *)e->d_out.p, d, e->d_packed.p));
    e->launches_other += 1;
    const u64 first = copies.front().dst_off, last = copies.back().dst_off + copies.back().len;
    B2_CUDA_CHECK(cudaMemcpyAsync(out + first, e->d_packed.p + first, last - first, cudaMemcpyDeviceToHost, st));
  }
  B2_CUDA_CHECK(cudaStreamSynchronize(st));
  for (const HeaderSpan &sp : spans) memcpy(out + sp.dst, sp.bytes.data(), sp.bytes.size());
  Z.done += Z.q_bytes;
  Z.queue.clear();
  Z.q_end = Z.q_bytes = Z.q_bound = 0;
  return 0;
}

// One entry above W: its local header and payload to out[0 ..), the stream written through the windows of b2_stream_*.
int zip_add_windowed(b2_encoder *e, const std::string &name, u32 time, u32 flags, const u8 *in, u64 n, u8 *out, u64 out_cap) {
  ZipState &Z = e->zip;
  StreamState &S = e->stream;
  b2zip::ZipLayout &L = Z.layout;
  u64 offset = 0, hbytes = 0;
  if (!L.open_entry(n, name.size(), &offset, &hbytes)) B2_FAIL(B2_ERR_ARGUMENT, "Zip_Capacity_Exceeded: archive too large");
  u8 *payload = out + hbytes;
  const u64 cap = out_cap - hbytes;
  stream_reset(e, (i64)n);
  u32 crc = 0;
  u64 crc_done = 0;                                    // entry bytes folded into crc
  auto crc_window = [&]() -> int {                     // the window's bytes that no window before it held
    const u64 k = S.base + S.held - crc_done;
    if (!k) return 0;
    B2_CUDA_CHECK(cudaStreamWaitEvent(e->st, e->ev_up, 0));
    const u64 at = crc_done - S.base;                  // an offset, not a pointer: k_zipcrc_tiles's vector loads need an aligned base
    B2_TRY(zip_crc_device(e, S.buf[S.cur], 1, &at, &k));
    u32 c = 0;
    B2_CUDA_CHECK(cudaMemcpy(&c, e->d_zcrc.p, sizeof c, cudaMemcpyDeviceToHost));
    crc = b2zip::crc32_combine(crc, c, k);
    crc_done += k;
    return 0;
  };
  ProgressScope ps(e, Z.done, Z.added);
  const u64 full = S.window + S.margin;
  u64 taken = 0;
  for (;;) {                                           // b2_stream_write of the whole entry
    const u64 k = std::min<u64>(full - S.held, n - taken);
    B2_TRY(stream_upload(e, S.cur, S.held, in + taken, k));
    S.held += k; taken += k;
    if (S.held < full) break;
    B2_TRY(crc_window());
    B2_TRY(stream_window(e, false, in, n, &taken, payload, cap, 0));
  }
  B2_TRY(crc_window());
  B2_TRY(stream_window(e, true, nullptr, 0, &taken, payload, cap, 0));   // b2_stream_end
  if (taken != n || crc_done != n) B2_FAIL(B2_ERR_INTERNAL, "entry not taken whole");
  const bool stored = S.out_end >= n;                  // Store fallback: the bytes from the caller's `in`
  if (stored && n) memcpy(payload, in, n);
  std::vector<u8> hdr;
  L.close_entry(name, n, stored ? n : S.out_end, crc, time, flags, stored ? 0 : 12, hdr);
  if (hdr.size() != hbytes) B2_FAIL(B2_ERR_INTERNAL, "local header length changed");
  memcpy(out, hdr.data(), hbytes);
  Z.done += n;
  return 0;
}
}  // namespace

extern "C" {

int b2_zip_begin(b2_encoder *e, int duplicates, uint64_t window_bytes) {
  if (!e) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  ZipState &Z = e->zip;
  if (Z.open) B2_FAIL(B2_ERR_ARGUMENT, "an archive is already open on this handle");
  if (e->stream.open) B2_FAIL(B2_ERR_ARGUMENT, "a stream is open on this handle (b2_stream_begin)");
  if (duplicates != B2_ZIP_ADMIT_DUPLICATES && duplicates != B2_ZIP_ERROR_ON_DUPLICATE) B2_FAIL(B2_ERR_ARGUMENT, "bad duplicate policy");
  B2_CUDA_CHECK(cudaSetDevice(e->device));
  B2_TRY(stream_buffers(e, window_bytes));
  Z.layout = b2zip::ZipLayout();
  Z.names.clear(); Z.queue.clear();
  Z.q_end = Z.q_bytes = Z.q_bound = Z.cd_bound = Z.done = Z.added = 0;
  Z.duplicates = duplicates;
  Z.open = true;
  return 0;
}

uint64_t b2_zip_add_bound(b2_encoder *e, uint64_t n, uint32_t name_bytes) {
  const bool queued = e && e->zip.open && n <= e->stream.window;
  const u64 q = e && e->zip.open ? e->zip.q_bound : 0;
  return q + b2zip::ZipLayout::local_header_bytes(name_bytes, true) + (queued ? n : b2_stream_bound(nullptr, n));
}

uint64_t b2_zip_finish_bound(b2_encoder *e) {
  if (!e || !e->zip.open) return b2zip::ZipLayout::end_records_max;
  return e->zip.q_bound + e->zip.cd_bound + b2zip::ZipLayout::end_records_max;
}

int b2_zip_add(b2_encoder *e, const char *name, uint32_t name_bytes, uint32_t dos_time, uint32_t flags,
               const uint8_t *in, uint64_t n, uint8_t *out, uint64_t out_cap, uint64_t *out_len) {
  if (!e || !out_len || (n && !in) || (name_bytes && !name) || !out) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  ZipState &Z = e->zip;
  if (!Z.open) B2_FAIL(B2_ERR_ARGUMENT, "b2_zip_add without b2_zip_begin");
  *out_len = 0;
  if (name_bytes > 65535u) B2_FAIL(B2_ERR_ARGUMENT, "bad entry name length");
  if (out_cap < b2_zip_add_bound(e, n, name_bytes)) B2_FAIL(B2_ERR_OUTPUT_TOO_SMALL, "output buffer below b2_zip_add_bound");
  const std::string nm = b2zip::unixify(name, name_bytes);
  if (Z.duplicates == B2_ZIP_ERROR_ON_DUPLICATE && Z.names.count(nm)) {   // Duplicate_name (zip-create.adb:138-147)
    g_last_error = "Duplicate_name: Entry name = " + nm;
    return B2_ERR_DUPLICATE_NAME;
  }
  const u64 out0 = Z.layout.pos;
  auto run = [&]() -> int {
    B2_CUDA_CHECK(cudaSetDevice(e->device));
    if (Z.duplicates == B2_ZIP_ERROR_ON_DUPLICATE) Z.names.insert(nm);
    Z.added += n;
    Z.cd_bound += b2zip::ZipLayout::central_header_max(nm.size());
    const StreamState &S = e->stream;
    if (n > S.window) {
      B2_TRY(zip_flush(e, out));
      const u64 at = Z.layout.pos - out0;
      return zip_add_windowed(e, nm, dos_time, flags, in, n, out + at, out_cap - at);
    }
    u64 at = (Z.q_end + 15) & ~15ull;
    if (!Z.queue.empty() && (Z.q_bytes + n > S.window || at + n + 128 > S.buf_bytes || Z.queue.size() >= zip_queue_max(S.window))) {
      B2_TRY(zip_flush(e, out));
      at = 0;
    }
    B2_TRY(stream_upload(e, 0, at, in, n));
    Z.queue.push_back(ZipQueued{nm, at, n, dos_time, flags});
    Z.q_end = at + n; Z.q_bytes += n;
    Z.q_bound += b2zip::ZipLayout::local_header_bytes(nm.size(), true) + n;
    return 0;
  };
  const int rc = run();
  if (rc) { const std::string msg = g_last_error; zip_close(e); g_last_error = msg; return rc; }
  B2_CUDA_CHECK(cudaStreamSynchronize(e->cst));          // the caller may reuse `in` once this returns
  *out_len = Z.layout.pos - out0;
  return 0;
}

int b2_zip_finish(b2_encoder *e, uint8_t *out, uint64_t out_cap, uint64_t *out_len, b2_zip_entry_info *info, uint64_t info_cap,
                  uint64_t *n_entries) {
  if (!e || !out_len || !out || (info_cap && !info)) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  ZipState &Z = e->zip;
  if (!Z.open) B2_FAIL(B2_ERR_ARGUMENT, "b2_zip_finish without b2_zip_begin");
  *out_len = 0;
  if (n_entries) *n_entries = 0;
  if (out_cap < b2_zip_finish_bound(e)) B2_FAIL(B2_ERR_OUTPUT_TOO_SMALL, "output buffer below b2_zip_finish_bound");
  b2zip::ZipLayout &L = Z.layout;
  const u64 out0 = L.pos;
  auto run = [&]() -> int {
    B2_CUDA_CHECK(cudaSetDevice(e->device));
    B2_TRY(zip_flush(e, out));
    std::vector<u8> tail;
    const u64 at = L.pos - out0;
    if (!L.finish(tail)) B2_FAIL(B2_ERR_ARGUMENT, "Zip_Capacity_Exceeded: archive too large");
    memcpy(out + at, tail.data(), tail.size());
    return 0;
  };
  const int rc = run();
  if (rc) { const std::string msg = g_last_error; zip_close(e); g_last_error = msg; return rc; }
  for (size_t i = 0; i < L.cat.size() && i < info_cap; i++) {
    const b2zip::ZipEntryRecord &c = L.cat[i];
    info[i].crc32 = c.crc; info[i].zip_type = c.method; info[i].reserved = 0; info[i].compressed_size = c.csize;
    info[i].local_header_offset = c.offset;
  }
  if (n_entries) *n_entries = L.cat.size();
  *out_len = L.pos - out0;
  zip_close(e);
  return 0;
}

int b2_zip_abort(b2_encoder *e) {
  if (!e) return B2_ERR_ARGUMENT;
  if (e->zip.open) zip_close(e);
  return 0;
}

int b2_set_timing(b2_encoder *e, int on) { if (!e) return B2_ERR_ARGUMENT; e->timing = on; return 0; }
int b2_get_stats(b2_encoder *e, b2_stats *out) { if (!e || !out) return B2_ERR_ARGUMENT; *out = e->stats; return 0; }
int b2_reset_stats(b2_encoder *e) {
  if (!e) return B2_ERR_ARGUMENT;
  memset(&e->stats, 0, sizeof e->stats); memset(&e->sort_stats, 0, sizeof e->sort_stats);
  e->launches_other = 0;
  return 0;
}

int b2_set_progress(b2_encoder *e, b2_progress_fn fn, void *user) {
  if (!e) return B2_ERR_ARGUMENT;
  e->progress = fn; e->progress_user = user;
  return 0;
}

int b2_get_trace(b2_encoder *e, b2_chunk_trace *out, uint64_t cap, uint64_t *n) {
  if (!e || !n || (cap && !out)) return B2_ERR_ARGUMENT;
  *n = e->trace.size();
  for (size_t i = 0; i < e->trace.size() && i < cap; i++) out[i] = e->trace[i];
  return 0;
}

int b2_get_segments(b2_encoder *e, uint64_t chunk, int profile, uint32_t *cuts, uint32_t cap, uint32_t *n) {
  if (!e || !n || profile < 0 || profile > 1) return B2_ERR_ARGUMENT;
  const size_t k = chunk * 2 + profile;
  if (k >= e->nseg.size()) { *n = 0; return B2_ERR_ARGUMENT; }
  const u32 ns = e->nseg[k];
  *n = ns;
  if (ns == 1 && cap >= 1) cuts[0] = e->chunks[chunk].len;
  else for (u32 i = 0; i < ns && i < cap; i++) cuts[i] = e->seg[k][i];
  return 0;
}

int b2_dbg_block(b2_encoder *e, const uint8_t *raw, uint32_t len, uint8_t *rle_out, uint8_t *bwt_out,
                 uint16_t *mtf_out, uint8_t *sel_out, uint8_t *lens_out, uint8_t *bits_out, uint64_t bits_cap,
                 b2_block_info *info) {
  if (!e || (len && !raw)) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  B2_NO_STREAM(e);
  B2_CUDA_CHECK(cudaSetDevice(e->device));
  Workspace *w = e->ws[0];
  cudaStream_t st = w->st;
  B2_TRY(e->d_in.ensure((size_t)len + 256));
  if (len) B2_CUDA_CHECK(cudaMemcpyAsync(e->d_in.p, raw, len, cudaMemcpyHostToDevice, st));
  B2_CUDA_CHECK(cudaMemsetAsync(e->d_in.p + len, 0, 128, st));
  std::vector<B2Job> jobs(1);
  memset(&jobs[0], 0, sizeof(B2Job));
  jobs[0].raw_off = 0; jobs[0].raw_len = len;
  reset_workspace_stats(e);
  memset(&e->sort_stats, 0, sizeof e->sort_stats);
  e->launches_other = 0;
  B2_TRY(run_batch(e, w, e->d_in.p, jobs));
  merge_workspace_stats(e);
  const B2Job &b = w->batch_jobs[0];
  if (rle_out && b.n) B2_CUDA_CHECK(cudaMemcpyAsync(rle_out, w->d_text.p + b.pos_off, b.n, cudaMemcpyDeviceToHost, st));
  if (bwt_out && b.n) B2_CUDA_CHECK(cudaMemcpyAsync(bwt_out, w->d_bwt.p + b.pos_off, b.n, cudaMemcpyDeviceToHost, st));
  if (mtf_out) B2_CUDA_CHECK(cudaMemcpyAsync(mtf_out, w->d_mtf.p + b.mtf_off, (size_t)b.n_mtf * 2, cudaMemcpyDeviceToHost, st));
  const u32 total_groups = w->total_groups;
  if (sel_out) B2_CUDA_CHECK(cudaMemcpyAsync(sel_out, w->d_sel.p + (size_t)b.best * total_groups + b.grp_off, b.n_groups, cudaMemcpyDeviceToHost, st));
  if (lens_out) B2_CUDA_CHECK(cudaMemcpyAsync(lens_out, w->d_lens.p + (size_t)b.best * (B2_MAX_CODERS * B2_MAX_ALPHA), B2_MAX_CODERS * B2_MAX_ALPHA, cudaMemcpyDeviceToHost, st));
  u64 nbytes = (b.nbits + 7) >> 3;
  if (bits_out) {
    if (nbytes > bits_cap) B2_FAIL(B2_ERR_OUTPUT_TOO_SMALL, "bits_out too small");
    B2_CUDA_CHECK(cudaMemcpyAsync(bits_out, (u8 *)(w->d_bits.p + b.bits_off), nbytes, cudaMemcpyDeviceToHost, st));
  }
  B2_CUDA_CHECK(cudaStreamSynchronize(st));
  if (info) {
    int max_len, sw, ec;
    b2_triple(e->level, (int)b.best, max_len, sw, ec);
    info->n_rle = b.n; info->origin = b.origin; info->crc = b.crc; info->n_mtf = b.n_mtf; info->eob = b.n_used + 1;
    info->n_used = b.n_used; info->n_sel = b.n_groups; info->ec_count = (u32)ec; info->max_len = (u32)max_len;
    info->sample_width = (u32)sw; info->cost = b.best_cost; info->pad = 0; info->bits = b.nbits;
  }
  return 0;
}

int b2_dbg_mtf(b2_encoder *e, const uint8_t *cols, const uint64_t *col_offs, const uint32_t *lens, uint32_t n_cols,
               uint8_t *idx_out, uint16_t *mtf_out, uint64_t mtf_cap, uint32_t *n_mtf, uint32_t *n_groups) {
  if (!e || n_cols == 0 || n_cols > e->batch_jobs_max || !col_offs || !lens || !idx_out || !mtf_out || !n_mtf || !n_groups)
    B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  u64 need = 0;
  for (u32 j = 0; j < n_cols; j++) {
    if (lens[j] > (u32)e->level * 100000u) B2_FAIL(B2_ERR_ARGUMENT, "column longer than a block of this level");
    if (lens[j] && !cols) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
    need += (u64)lens[j] + 2;
  }
  if (mtf_cap < need) B2_FAIL(B2_ERR_OUTPUT_TOO_SMALL, "mtf_out too small");
  B2_NO_STREAM(e);
  B2_CUDA_CHECK(cudaSetDevice(e->device));
  Workspace *w = e->ws[0];
  cudaStream_t st = w->st;
  std::vector<B2Job> jobs(n_cols);
  for (u32 j = 0; j < n_cols; j++) {
    B2Job &b = jobs[j];
    memset(&b, 0, sizeof b);
    b.raw_len = b.n = lens[j];
    const uint8_t *c = cols + col_offs[j];
    for (u32 i = 0; i < b.n; i++) b.in_use[c[i] >> 5] |= 1u << (c[i] & 31);
    for (int q = 0; q < 8; q++) b.n_used += (u32)__builtin_popcount(b.in_use[q]);
  }
  const u64 T = layout_jobs(jobs, e->level);
  B2_TRY(ensure_batch_workspace(w, (size_t)T + 64, n_cols));
  // Poison: slot padding and index bytes 0xA5, symbols 0xA5A5, masks 0 (an unwritten mask reads as "no byte here", so
  // the list rebuild misses bytes).  A read of anything not written, or an output not written, shows as a difference.
  B2_CUDA_CHECK(cudaMemsetAsync(w->d_bwt.p, 0xA5, w->d_bwt.cap, st));
  B2_CUDA_CHECK(cudaMemsetAsync(w->d_idx.p, 0xA5, w->d_idx.cap, st));
  B2_CUDA_CHECK(cudaMemsetAsync(w->d_m16.p, 0, w->d_m16.cap * sizeof(u32), st));
  B2_CUDA_CHECK(cudaMemsetAsync(w->d_m256.p, 0, w->d_m256.cap * sizeof(u32), st));
  B2_CUDA_CHECK(cudaMemsetAsync(w->d_mtf.p, 0xA5, w->d_mtf.cap * sizeof(u16), st));
  for (u32 j = 0; j < n_cols; j++)
    if (jobs[j].n) B2_CUDA_CHECK(cudaMemcpyAsync(w->d_bwt.p + jobs[j].pos_off, cols + col_offs[j], jobs[j].n, cudaMemcpyHostToDevice, st));
  MtfPlan P;
  plan_mtf(jobs, P);
  B2_CUDA_CHECK(cudaMemcpyAsync(w->d_jobs.p, jobs.data(), n_cols * sizeof(B2Job), cudaMemcpyHostToDevice, st));
  B2_TRY(launch_mtf(w, n_cols, P));
  B2_CUDA_CHECK(cudaMemcpyAsync(jobs.data(), w->d_jobs.p, n_cols * sizeof(B2Job), cudaMemcpyDeviceToHost, st));
  B2_CUDA_CHECK(cudaStreamSynchronize(st));
  u64 mo = 0;
  for (u32 j = 0; j < n_cols; j++) {
    const B2Job &b = jobs[j];
    if (b.n_mtf > b.n + 2) B2_FAIL(B2_ERR_INTERNAL, "more symbols than positions");
    if (b.n) B2_CUDA_CHECK(cudaMemcpyAsync(idx_out + col_offs[j], w->d_idx.p + b.pos_off, b.n, cudaMemcpyDeviceToHost, st));
    B2_CUDA_CHECK(cudaMemcpyAsync(mtf_out + mo, w->d_mtf.p + b.mtf_off, (size_t)b.n_mtf * sizeof(u16), cudaMemcpyDeviceToHost, st));
    n_mtf[j] = b.n_mtf; n_groups[j] = b.n_groups;
    mo += b.n_mtf;
  }
  B2_CUDA_CHECK(cudaStreamSynchronize(st));
  return 0;
}

int b2_dbg_segment(b2_encoder *e, const uint8_t *raw, uint64_t len, uint32_t *cuts0, uint32_t *n0, uint32_t *cuts1,
                   uint32_t *n1, uint32_t cap, double *series, uint64_t series_cap, uint32_t *paths) {
  if (!e || !raw || len == 0 || len > 9000000 || !n0 || !n1 || (cap && (!cuts0 || !cuts1))) B2_FAIL(B2_ERR_ARGUMENT, "bad argument");
  const u64 steps = len > 20000 ? len - 16000 : 0;      // window 16 000; no step below window + 4 000 (b2_segment.cuh)
  if (series && series_cap < steps) B2_FAIL(B2_ERR_OUTPUT_TOO_SMALL, "series too small");
  B2_NO_STREAM(e);
  B2_CUDA_CHECK(cudaSetDevice(e->device));
  cudaStream_t st = e->st;
  struct Taps { DevBuf<double> series; DevBuf<u32> paths; ~Taps() { series.release(); paths.release(); } } taps;
  B2_TRY(e->d_in.ensure((size_t)len + 256));
  B2_CUDA_CHECK(cudaMemcpyAsync(e->d_in.p, raw, len, cudaMemcpyHostToDevice, st));
  B2_CUDA_CHECK(cudaMemsetAsync(e->d_in.p + len, 0, 128, st));
  const B2Chunk chunk{0, (u32)len, 0, 0, 0};
  B2_TRY(e->d_chunks.ensure(1));
  B2_CUDA_CHECK(cudaMemcpyAsync(e->d_chunks.p, &chunk, sizeof chunk, cudaMemcpyHostToDevice, st));
  B2_TRY(e->d_seg.ensure(2 * B2_MAX_SEG));
  B2_TRY(e->d_nseg.ensure(2));
  if (series && steps) B2_TRY(taps.series.ensure(steps));
  if (paths) {
    B2_TRY(taps.paths.ensure(4));
    B2_CUDA_CHECK(cudaMemsetAsync(taps.paths.p, 0, 4 * sizeof(u32), st));
  }
  B2_TRY(b2k_segment(st, e->d_in.p, e->d_chunks.p, 1, e->d_T.p, e->d_seg.p, e->d_nseg.p, nullptr,
                     series && steps ? taps.series.p : nullptr, paths ? taps.paths.p : nullptr));
  u32 ns[2] = {0, 0};
  B2_CUDA_CHECK(cudaMemcpyAsync(ns, e->d_nseg.p, sizeof ns, cudaMemcpyDeviceToHost, st));
  if (series && steps) B2_CUDA_CHECK(cudaMemcpyAsync(series, taps.series.p, steps * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (paths) B2_CUDA_CHECK(cudaMemcpyAsync(paths, taps.paths.p, 4 * sizeof(u32), cudaMemcpyDeviceToHost, st));
  B2_CUDA_CHECK(cudaStreamSynchronize(st));
  uint32_t *cuts[2] = {cuts0, cuts1};
  for (int p = 0; p < 2; p++) {
    if (ns[p] > B2_MAX_SEG) B2_FAIL(B2_ERR_INTERNAL, "segment table overflow");
    const u32 k = std::min(ns[p], cap);
    if (k) B2_CUDA_CHECK(cudaMemcpy(cuts[p], e->d_seg.p + (size_t)p * B2_MAX_SEG, k * sizeof(u32), cudaMemcpyDeviceToHost));
  }
  *n0 = ns[0]; *n1 = ns[1];
  return 0;
}

}  // extern "C"
