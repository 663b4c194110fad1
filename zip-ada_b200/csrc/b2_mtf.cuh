// Stage A7: move-to-front + zero-run coding (RUN_A/RUN_B), parallel over positions.
//
// Reference: zip_lib/bzip2-encoding.adb:318-413.  The reference keeps a 256-entry list, finds the
// symbol by linear search and shifts (:384-396).  The MTF index of position i equals the number of
// DISTINCT symbols seen since the previous occurrence of the same symbol; if there is none, it is
// (rank of the symbol among the used bytes) + (number of distinct symbols seen so far that are
// larger), because the list starts in increasing order (:374-376, :320-328).  That is a pure
// function of the data before i, so a block can be cut into segments that are processed
// independently once the list at the segment start is known (k_mtf_seq).
//
// To keep the backward search short, k_mtf_masks first records which byte values occur in every
// 16-position segment (256-bit mask), every 256-position segment and every 4096-position tile; a
// search that leaves its own 16-segment skips whole segments / tiles by OR-ing their masks until it
// meets one that contains the symbol, descends, and only then walks bytes again.  Worst case per
// position: 2*15 byte steps + 4*15 segment masks + (tiles of the block) tile masks.
//
// The zero-run coding (:348-363, :400-410) is a max-scan (last non-zero position) plus an add-scan
// (output offsets) per block (k_rle2).
//
// Included by b2_mtf.cu; also compiled for the host by tests/emu (a thread-per-lane emulation of CTAs that checks the
// index bytes and the symbols of designed last columns against the oracle's literal MTF - `-m "not gpu"`), hence the
// B2_EMU switches: the emulator's __shared__ is empty, so a plain array would be per thread; there the shared arrays
// come from the emulator's per-CTA memory, which it poisons.
#pragma once
#include "b2_common.cuh"
#include "b2_kernels.h"

#define MI_THREADS 256
#define MI_ITEMS (B2_MTF_TILE / MI_THREADS)

struct Mask256 { u32 w[8]; };

__device__ __forceinline__ void mask_or(u32 *seen, const u32 *__restrict__ m) {
  const uint4 a = *reinterpret_cast<const uint4 *>(m), b = *reinterpret_cast<const uint4 *>(m + 4);
  seen[0] |= a.x; seen[1] |= a.y; seen[2] |= a.z; seen[3] |= a.w;
  seen[4] |= b.x; seen[5] |= b.y; seen[6] |= b.z; seen[7] |= b.w;
}
__device__ __forceinline__ void seen_set(u32 *seen, u32 x) {
  const u32 bit = 1u << (x & 31), wsel = x >> 5;
#pragma unroll
  for (int w = 0; w < 8; w++) seen[w] |= (w == (int)wsel) ? bit : 0u;
}

// One CTA per 4096-position tile; thread t owns the 16 positions [16t, 16t+16) of the tile:
// 256 masks of 16 positions, 16 masks of 256 positions, 1 tile mask.
__global__ void __launch_bounds__(MI_THREADS)
k_mtf_masks(const B2SortTile *__restrict__ tiles, const B2Job *__restrict__ jobs, const u8 *__restrict__ bwt,
            u32 *__restrict__ m16, u32 *__restrict__ m256, u32 *__restrict__ tilemask) {
#ifndef B2_EMU
  __shared__ u32 tm[8];
#else
  auto &tm = emu_shared<u32[8]>();
#endif
  const B2SortTile tl = tiles[blockIdx.x];
  const B2Job &job = jobs[tl.job];
  const u32 n = job.n, off = job.pos_off;
  const u8 *d = bwt + off;
  const u32 tid = threadIdx.x, l = lane_id();
  if (tid < 8) tm[tid] = 0;
  __syncthreads();
  const u32 p0 = tl.start + tid * 16;
  u32 mk[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (p0 < n) {
    const uint4 v = *reinterpret_cast<const uint4 *>(d + p0);      // pos_off is a multiple of 64
    const u32 w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 16; k++) {
      if (p0 + k < n) seen_set(mk, (w[k >> 2] >> (8 * (k & 3))) & 255u);
    }
    u32 *o = m16 + ((size_t)(off >> 4) + (p0 >> 4)) * 8;
    *reinterpret_cast<uint4 *>(o) = make_uint4(mk[0], mk[1], mk[2], mk[3]);
    *reinterpret_cast<uint4 *>(o + 4) = make_uint4(mk[4], mk[5], mk[6], mk[7]);
  }
  // 256-position masks: OR over the 16 threads of a half warp
  const u32 hm = (l < 16) ? 0x0000FFFFu : 0xFFFF0000u;
  u32 r[8];
#pragma unroll
  for (int q = 0; q < 8; q++) r[q] = __reduce_or_sync(hm, mk[q]);
  if ((l & 15) == 0 && p0 < n) {
    u32 *o = m256 + ((size_t)(off >> 8) + (p0 >> 8)) * 8;
#pragma unroll
    for (int q = 0; q < 8; q++) { o[q] = r[q]; if (r[q]) atomicOr(&tm[q], r[q]); }
  }
  __syncthreads();
  if (tid < 8) tilemask[(size_t)blockIdx.x * 8 + tid] = tm[tid];
}

// ---------------------------------------------------------------------------------------------
// k_mtf_seq: one warp per segment of B2_MTF_SEG positions.
//  1. The list at the segment start is rebuilt from the data before it: walking backwards, the
//     symbols appear in the order of their last occurrence, which IS the list order; whole
//     16- / 256-position segments that hold no symbol not yet seen are skipped through their masks;
//     symbols never seen keep the initial increasing order (:374-376) behind the seen ones.
//  2. The segment is then processed in order.  Not the list is kept but its inverse, the PLACE of every
//     byte (as a dense code) in the list, eight places per lane as bytes of two registers: a byte with
//     place r is coded as r, every place below r moves up by one (a per-byte compare-and-add on the
//     packed registers), its own place becomes 0 (:384-396 without the search and without the shift).
// ---------------------------------------------------------------------------------------------
#define MS_WARPS 4

__device__ __forceinline__ bool mask_has_new(const u32 *m, const u32 *seen) {
  u32 r = 0;
#pragma unroll
  for (int q = 0; q < 8; q++) r |= m[q] & ~seen[q];
  return r != 0;
}
__device__ __forceinline__ void load_mask(const u32 *__restrict__ p, u32 *m) {
  const uint4 a = *reinterpret_cast<const uint4 *>(p), c = *reinterpret_cast<const uint4 *>(p + 4);
  m[0] = a.x; m[1] = a.y; m[2] = a.z; m[3] = a.w; m[4] = c.x; m[5] = c.y; m[6] = c.z; m[7] = c.w;
}
__device__ __forceinline__ bool seen_has(const u32 *seen, u32 x) {
  u32 w = seen[0];
#pragma unroll
  for (int q = 1; q < 8; q++) w = ((x >> 5) == (u32)q) ? seen[q] : w;
  return (w >> (x & 31)) & 1u;
}

// Phase 1 of k_mtf_seq*: the MTF list at position p0 of a block, rebuilt by one warp into lst[0..255]
// (places >= n_used are padded with zeros).
__device__ void mtf_build_list(const B2Job &job, const u8 *__restrict__ d, const u32 *__restrict__ s16,
                               const u32 *__restrict__ s256, u32 p0, u8 *lst) {
  const u32 l = lane_id(), lt = (1u << l) - 1u;
  const u32 n_used = job.n_used;
  // ---- 1. list at p0 ---------------------------------------------------------------------------
  u32 seen[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  u32 count = 0;
  u32 q = p0;                                   // everything at positions >= q has been examined
  while (count < n_used && q > 0) {
    // a) bytes of the 16-segment that ends at q (those below q), most recent first
    {
      const u32 sbeg = (q - 1) & ~15u;
      const u32 pos = q - 1 - l;
      const bool valid = l < 16 && q >= 1 + l && pos >= sbeg;
      const u32 x = valid ? d[pos] : (256u + l);
      const bool fresh = valid && !seen_has(seen, x);
      const u32 peers = __match_any_sync(0xffffffffu, x);
      const bool first = fresh && ((peers & lt) == 0);         // most recent occurrence within these 16
      const u32 bm = __ballot_sync(0xffffffffu, first);
      if (first) lst[count + __popc(bm & lt)] = (u8)x;
      count += __popc(bm);
      u32 mine[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      if (first) seen_set(mine, x);
#pragma unroll
      for (int w = 0; w < 8; w++) seen[w] |= __reduce_or_sync(0xffffffffu, mine[w]);
      q = sbeg;
    }
    if (count >= n_used || q == 0) break;
    // b) remaining 16-segments of the current 256-segment
    bool located = false;
    if (q & 255u) {
      const i32 from = (i32)(q >> 4) - 1, lo = (i32)((q >> 8) << 4);
      const i32 sidx = from - (i32)l;
      bool has = false;
      if (sidx >= lo) { u32 m[8]; load_mask(s16 + (size_t)sidx * 8, m); has = mask_has_new(m, seen); }
      const u32 hm = __ballot_sync(0xffffffffu, has);
      if (hm) { q = (u32)(from - (__ffs(hm) - 1) + 1) << 4; located = true; }
      else q = (q >> 8) << 8;
    }
    // c) whole 256-segments, 32 per step
    while (!located && q > 0) {
      const i32 from = (i32)(q >> 8) - 1;
      const i32 sidx = from - (i32)l;
      bool has = false;
      if (sidx >= 0) { u32 m[8]; load_mask(s256 + (size_t)sidx * 8, m); has = mask_has_new(m, seen); }
      const u32 hm = __ballot_sync(0xffffffffu, has);
      if (hm) {
        const i32 hit = from - (__ffs(hm) - 1);                // nearest 256-segment with a new symbol
        // its 16-segments, from the last one down
        const i32 f16 = (hit << 4) + 15;
        u32 m[8]; load_mask(s16 + (size_t)(f16 - (i32)(l & 15)) * 8, m);
        const u32 h16 = __ballot_sync(0xffffffffu, l < 16 && mask_has_new(m, seen));
        q = (u32)(f16 - (__ffs(h16) - 1) + 1) << 4;
        located = true;
      } else {
        q = (from >= 31) ? (u32)(from - 31) << 8 : 0u;
      }
    }
  }
  __syncwarp();
  // symbols never seen: increasing order behind the others
  if (count < n_used) {
    for (u32 base = 0; base < 256; base += 32) {
      const u32 x = base + l;
      const bool add = ((job.in_use[x >> 5] >> (x & 31)) & 1u) && !seen_has(seen, x);
      const u32 bm = __ballot_sync(0xffffffffu, add);
      if (add) lst[count + __popc(bm & lt)] = (u8)x;
      count += __popc(bm);
    }
  }
  for (u32 i = count + l; i < 256; i += 32) lst[i] = 0;          // unused places (never matched: see `live`)
  __syncwarp();
}

__global__ void __launch_bounds__(32 * MS_WARPS)
k_mtf_seq(const B2SortTile *__restrict__ segs, u32 n_segs, const B2Job *__restrict__ jobs, const u8 *__restrict__ bwt,
          const u32 *__restrict__ m16, const u32 *__restrict__ m256, u8 *__restrict__ idx_out) {
  // One warp per segment; lane g holds the places of the codes 8g .. 8g+7 in the list as bytes of two
  // registers (see k_mtf_seq8 for the scheme: no list shifting, no search).
#ifndef B2_EMU
  __shared__ u8 lists[MS_WARPS][256];
  __shared__ u8 ctab[MS_WARPS][256];
  __shared__ __align__(8) u8 place0[MS_WARPS][256];
#else
  auto &lists = emu_shared<u8[MS_WARPS][256]>();
  auto &ctab = emu_shared<u8[MS_WARPS][256]>();
  auto &place0 = emu_shared<u8[MS_WARPS][256]>();
#endif
  const u32 unit = blockIdx.x * MS_WARPS + warp_id();
  if (unit >= n_segs) return;
  const u32 l = lane_id();
  const B2SortTile sg = segs[unit];
  const B2Job &job = jobs[sg.job];
  const u32 n = job.n, off = job.pos_off;
  const u8 *d = bwt + off;
  u8 *lst = lists[warp_id()], *ct = ctab[warp_id()], *pl = place0[warp_id()];
  const u32 p0 = sg.start, p1 = min(n, sg.start + B2_MTF_SEG);
  const u32 n_used = job.n_used;
  mtf_build_list(job, d, m16 + (size_t)(off >> 4) * 8, m256 + (size_t)(off >> 8) * 8, p0, lst);
  {
    u32 pre = 0;                                     // bytes in use below 32 * (my word)
    for (u32 q = 0; q < 8; q++) {
      const u32 wv = job.in_use[q];
      ct[32 * q + l] = (u8)(pre + __popc(wv & ((1u << l) - 1u)));
      pre += __popc(wv);
      pl[32 * q + l] = 255;                          // codes not in use never move (a place is at most 255 and
    }                                                // "< r" with r <= 255 is false for them)
    __syncwarp();
    for (u32 pos = l; pos < n_used; pos += 32) pl[ct[lst[pos]]] = (u8)pos;
  }
  __syncwarp();
  // ---- 2. the segment, in order ------------------------------------------------------------------
  u32 R0 = *reinterpret_cast<const u32 *>(pl + 8 * l), R1 = *reinterpret_cast<const u32 *>(pl + 8 * l + 4);
  // With 256 bytes in use the place 255 is a real one; slots of unused codes only exist when n_used < 256,
  // and then no real place reaches 255, so the two never meet.
  u32 prevb = p0 > 0 ? d[p0 - 1] : 256u;
  for (u32 b0 = p0; b0 < p1; b0 += 32) {
    const u32 pi = b0 + l;
    const u32 mybyte = pi < p1 ? d[pi] : 0u;
    const u32 mycode = ct[mybyte];
    u32 myidx = 0;
    // positions whose byte differs from the one before them; the others continue a run (index 0)
    u32 before = __shfl_up_sync(0xffffffffu, mybyte, 1);
    if (l == 0) before = prevb;
    u32 todo = __ballot_sync(0xffffffffu, pi < p1 && mybyte != before);
    const u32 steps = min(32u, p1 - b0);
    prevb = __shfl_sync(0xffffffffu, mybyte, steps - 1);
    while (todo) {
      const u32 k = (u32)(__ffs(todo) - 1);
      todo &= todo - 1;
      const u32 c = __shfl_sync(0xffffffffu, mycode, k);
      const u32 sh = 8 * (c & 3u);
      const u32 mine = (((c & 4u) ? R1 : R0) >> sh) & 255u;      // its place, if I am the lane that holds it
      const u32 r = __shfl_sync(0xffffffffu, mine, c >> 3);
      const u32 m = r * 0x01010101u;
      R0 += __vcmpltu4(R0, m) & 0x01010101u;                     // places below r move up
      R1 += __vcmpltu4(R1, m) & 0x01010101u;
      if (l == (c >> 3)) { if (c & 4u) R1 &= ~(0xFFu << sh); else R0 &= ~(0xFFu << sh); }   // the byte goes to the front
      if (l == k) myidx = r;
    }
    if (pi < p1) idx_out[off + pi] = (u8)myidx;
  }
}

// ---------------------------------------------------------------------------------------------
// k_mtf_seqg<LG>: the same for blocks with at most 8 * LG distinct bytes (LG = 8: plain text, LG = 16: text
// with capitals, digits and punctuation).  The list then fits the registers of LG lanes, so one warp advances
// 32 / LG segments at a time, one per group of LG lanes.
// ---------------------------------------------------------------------------------------------
template <int LG>
__global__ void __launch_bounds__(32 * MS_WARPS)
k_mtf_seqg(const B2SortTile *__restrict__ segs, u32 n_segs, const B2Job *__restrict__ jobs, const u8 *__restrict__ bwt,
           const u32 *__restrict__ m16, const u32 *__restrict__ m256, u8 *__restrict__ idx_out) {
  // Per unit: the list at the segment start (bytes in list order), the dense code of every byte (its
  // rank among the bytes in use) and, from both, the PLACE of every code in the list.  Phase 2 keeps the
  // places, not the list: lane g of a group holds the places of codes 8g .. 8g+7 as bytes of two
  // registers.  A byte b with place r is coded as r; then every place below r moves up by one (a per-byte
  // compare and add on the packed registers) and b's place becomes 0.  No list shifting, no search.
  constexpr int NU = 32 / LG;                      // units (segments) per warp
  constexpr int PPL = 32 / LG;                     // positions per lane and step (32 positions per group and step)
  constexpr u32 CMASK = 8 * LG - 1;
#ifndef B2_EMU
  __shared__ u8 lists[MS_WARPS][NU][256];
  __shared__ u8 ctab[MS_WARPS][NU][256];
  __shared__ __align__(8) u8 place0[MS_WARPS][NU][8 * LG];
#else
  auto &lists = emu_shared<u8[MS_WARPS][NU][256]>();
  auto &ctab = emu_shared<u8[MS_WARPS][NU][256]>();
  auto &place0 = emu_shared<u8[MS_WARPS][NU][8 * LG]>();
#endif
  const u32 l = lane_id(), gl = l & (LG - 1), grp = l / LG;
  const u32 unit0 = (blockIdx.x * MS_WARPS + warp_id()) * NU;
  if (unit0 >= n_segs) return;
  // phase 1, one unit after the other with the whole warp
  for (u32 u = 0; u < (u32)NU; u++) {
    if (unit0 + u < n_segs) {
      const B2SortTile sg = segs[unit0 + u];
      const B2Job &job = jobs[sg.job];
      const u32 off = job.pos_off;
      u8 *lst = lists[warp_id()][u], *ct = ctab[warp_id()][u], *pl = place0[warp_id()][u];
      mtf_build_list(job, bwt + off, m16 + (size_t)(off >> 4) * 8, m256 + (size_t)(off >> 8) * 8, sg.start, lst);
      u32 pre = 0;                                   // bytes in use below 32 * (my word)
      for (u32 q = 0; q < 8; q++) {
        const u32 wv = job.in_use[q];
        ct[32 * q + l] = (u8)(pre + __popc(wv & ((1u << l) - 1u)));
        pre += __popc(wv);
      }
      for (u32 i = l; i < 8 * LG; i += 32) pl[i] = 255;   // codes not in use never move
      __syncwarp();
      for (u32 pos = l; pos < job.n_used; pos += 32) pl[ct[lst[pos]]] = (u8)pos;
    }
  }
  __syncwarp();
  // phase 2, NU units side by side
  const bool have = unit0 + grp < n_segs;
  const B2SortTile sg = segs[have ? unit0 + grp : unit0];
  const B2Job &job = jobs[sg.job];
  const u32 n = job.n, off = job.pos_off;
  const u8 *d = bwt + off;
  const u8 *ct = ctab[warp_id()][have ? grp : 0];
  const u32 p0 = sg.start, p1 = have ? min(n, sg.start + B2_MTF_SEG) : sg.start;
  u32 R0 = *reinterpret_cast<const u32 *>(place0[warp_id()][have ? grp : 0] + 8 * gl);
  u32 R1 = *reinterpret_cast<const u32 *>(place0[warp_id()][have ? grp : 0] + 8 * gl + 4);
  const u32 gbase = grp * LG;                      // first lane of my group
  u32 prevb = (have && p0 > 0) ? d[p0 - 1] : 256u;
  const u32 nb = (B2_MTF_SEG / 32);
  for (u32 it = 0; it < nb; it++) {
    const u32 b0 = p0 + it * 32;
    if (!__any_sync(0xffffffffu, b0 < p1)) break;
    const u32 pi = b0 + PPL * gl;                  // my positions
    u32 word = 0;                                  // slots are 256-aligned and padded
    if (b0 < p1) word = PPL == 4 ? *reinterpret_cast<const u32 *>(d + pi) : (u32)*reinterpret_cast<const u16 *>(d + pi);
    u32 cword = 0;                                 // the codes of my bytes
#pragma unroll
    for (int j = 0; j < PPL; j++) cword |= (u32)ct[(word >> (8 * j)) & 255u] << (8 * j);
    // bits of my positions whose byte differs from the byte before it
    u32 before = __shfl_up_sync(0xffffffffu, (word >> (8 * (PPL - 1))) & 255u, 1, LG);
    if (gl == 0) before = prevb;
    const u32 shifted = (word << 8) | (before & 255u);
    u32 nib = 0;
#pragma unroll
    for (int j = 0; j < PPL; j++) {
      const bool differs = ((word >> (8 * j)) & 255u) != ((shifted >> (8 * j)) & 255u) || (j == 0 && gl == 0 && before > 255u);
      if (differs && pi + j < p1) nib |= 1u << j;
    }
    u32 todo = nib << (PPL * gl);
#pragma unroll
    for (int o = 1; o < LG; o <<= 1) todo |= __shfl_xor_sync(0xffffffffu, todo, o);
    {
      // (warp-wide shuffle: executed by every lane, also by groups that have run out of work)
      const u32 lastpos = (b0 < p1) ? min(31u, p1 - b0 - 1) : 0u;
      const u32 lw = __shfl_sync(0xffffffffu, word, gbase + lastpos / PPL);
      if (b0 < p1) prevb = (lw >> (8 * (lastpos % PPL))) & 255u;
    }
    u32 myidx = 0;
    while (__any_sync(0xffffffffu, todo != 0)) {
      const bool act = todo != 0;
      const u32 k = act ? (u32)(__ffs(todo) - 1) : 0u;
      todo &= todo - 1;
      const u32 ck = __shfl_sync(0xffffffffu, cword, gbase + k / PPL);
      const u32 c = (ck >> (8 * (k % PPL))) & CMASK;             // code of the byte at position k (< 8 * LG here)
      const u32 sh = 8 * (c & 3u);
      const u32 mine = (((c & 4u) ? R1 : R0) >> sh) & 255u;      // its place, if I am the lane that holds it
      const u32 r = __shfl_sync(0xffffffffu, mine, gbase + (c >> 3));
      if (act) {
        const u32 m = r * 0x01010101u;
        R0 += __vcmpltu4(R0, m) & 0x01010101u;                   // places below r move up
        R1 += __vcmpltu4(R1, m) & 0x01010101u;
        if (gl == (c >> 3)) { if (c & 4u) R1 &= ~(0xFFu << sh); else R0 &= ~(0xFFu << sh); }   // the byte goes to the front
        if (gl == k / PPL) myidx |= r << (8 * (k % PPL));
      }
    }
    if (b0 < p1) {
      // PPL index bytes per lane; positions beyond p1 inside the last word are never read
      if (PPL == 4) *reinterpret_cast<u32 *>(idx_out + off + pi) = myidx;
      else *reinterpret_cast<u16 *>(idx_out + off + pi) = (u16)myidx;
    }
  }
}

#define R2_THREADS 1024
#define R2_ITEMS 4
#define R2_TILE (R2_THREADS * R2_ITEMS)

__global__ void __launch_bounds__(R2_THREADS, 1)
k_rle2(B2Job *jobs, const u8 *__restrict__ idx_in, u16 *__restrict__ mtf) {
#ifndef B2_EMU
  __shared__ i32 sm_i[40];
  __shared__ u32 sm_u[40];
#else
  auto &sm_i = emu_shared<i32[40]>();
  auto &sm_u = emu_shared<u32[40]>();
#endif
  B2Job &job = jobs[blockIdx.x];
  const u32 n = job.n, off = job.pos_off;
  const u8 *ix = idx_in + off;
  u16 *out = mtf + job.mtf_off;
  const u32 tid = threadIdx.x;
  i32 carry_nz = -1;
  u32 out_base = 0;
  for (u32 t0 = 0; t0 < n; t0 += R2_TILE) {
    const u32 a = t0 + tid * R2_ITEMS;
    u32 v[R2_ITEMS];
    i32 lnz = -1;
#pragma unroll
    for (int k = 0; k < R2_ITEMS; k++) {
      v[k] = (a + k < n) ? ix[a + k] : 0;
      if (a + k < n && v[k]) lnz = (i32)(a + k);
    }
    i32 tot_nz;
    i32 prev_nz = block_excl_max(lnz, -1, sm_i, &tot_nz);
    prev_nz = max(prev_nz, carry_nz);
    u32 cnt = 0;
    {
      i32 p = prev_nz;
#pragma unroll
      for (int k = 0; k < R2_ITEMS; k++) {
        if (a + k < n && v[k]) {
          u32 run = (u32)((i32)(a + k) - 1 - p);
          cnt += 1 + (run ? (31 - __clz(run + 1)) : 0);
          p = (i32)(a + k);
        }
      }
    }
    u32 tile_total;
    u32 base = block_excl_add(cnt, sm_u, &tile_total);
    {
      u32 o = out_base + base;
      i32 p = prev_nz;
#pragma unroll
      for (int k = 0; k < R2_ITEMS; k++) {
        if (a + k < n && v[k]) {
          u32 run = (u32)((i32)(a + k) - 1 - p);
          if (run) {
            u32 rc = run + 1;                      // bijective base 2, RUN_A = 0, RUN_B = 1 (:348-363)
            do { out[o++] = (u16)(rc & 1); rc >>= 1; } while (rc >= 2);
          }
          out[o++] = (u16)(1 + v[k]);              // (:404)
          p = (i32)(a + k);
        }
      }
    }
    out_base += tile_total;
    carry_nz = max(carry_nz, tot_nz);
    __syncthreads();
  }
  if (tid == 0) {
    u32 o = out_base;
    u32 run = (u32)((i32)n - 1 - carry_nz);        // trailing zero run (:409)
    if (run) {
      u32 rc = run + 1;
      do { out[o++] = (u16)(rc & 1); rc >>= 1; } while (rc >= 2);
    }
    out[o++] = (u16)(job.n_used + 1);              // EOB (:330-335, :410)
    job.n_mtf = o;
    job.n_groups = 1 + (o - 1) / B2_GROUP_SIZE;    // selector_count (:968)
  }
}
