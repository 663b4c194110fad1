// b2gpu — B200-native BZip2 block encoder behind Zip-Ada's BZip2.Encoding interface.
// Common device/host declarations.  sm_100a only.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cuda_runtime.h>

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;
typedef int32_t i32;
typedef int64_t i64;

// ---- format constants (reference: zip_lib/bzip2.ads:77-122) ----------------
#define B2_GROUP_SIZE 50
#define B2_MAX_CODERS 6
#define B2_MAX_ALPHA 258
#define B2_N_TRIPLES 20          // 2 max_code_len x 2 sample_width x 5 coder counts (bzip2-encoding.adb:901-921)
#define B2_MAX_SEG 2304          // > 9_000_000 / 4_000 segments per (chunk, profile)

// One BWT block to encode = one reference `Encode_Block` call (bzip2-encoding.adb:148).
struct B2Job {
  u64 raw_off;      // offset of the raw slice in the input arena
  u32 raw_len;      // raw bytes
  u32 pos_off;      // offset into the per-position arenas (text/bwt/sa/rank...)
  u32 cap;          // positions reserved
  u32 n;            // post-RLE1 size                 (written by k_rle1)
  u32 crc;          // block CRC, finalised           (written by k_rle1)
  u32 origin;       // BWT origin pointer             (written by k_bwt_out)
  u32 in_use[8];    // 256-bit byte usage map         (written by k_rle1)
  u32 n_used;       // popcount(in_use)
  u32 mtf_off;      // offset (u16 units) into the MTF arena
  u32 n_mtf;        // M                              (written by k_mtf)
  u32 grp_off;      // offset into per-group arenas
  u32 n_groups;     // G = 1 + (M-1)/50
  u32 best;         // winning triple index           (written by k_choose)
  u32 best_cost;
  u32 unsorted;     // sort bookkeeping: rows not yet alone in their class after the current round
  u32 na;           // sort bookkeeping: rows in the compact (active) list of the current round
  u32 pad1;
  u32 tile0;        // index of the block's first 4096-tile in the MTF tile table
  u64 nbits;        // exact size of the block's bitstream (written by k_choose)
  u64 bits_off;     // u32-word offset in the bit arena (written by k_bits_layout)
};

// triple index t in 0..19 <-> (max_code_len, sample_width, coders) in the reference's loop order
// (bzip2-encoding.adb:930-935): max_len in (15,17) outer, sample_width in (3,4), coders 6 down to 2.
__host__ __device__ inline void b2_triple(int level, int t, int &max_len, int &sw, int &ec) {
  int a = t / 10, b = (t / 5) % 2, c = t % 5;
  if (level == 9) { max_len = a ? 17 : 15; sw = b ? 4 : 3; }
  else { max_len = 16; sw = 4; }
  ec = 6 - c;
}

#define B2_CUDA_CHECK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { b2_set_error(__FILE__, __LINE__, cudaGetErrorString(e_)); return 10; } } while (0)
void b2_set_error(const char *file, int line, const char *msg);

// Device helpers; the host emulation of tests/emu compiles them too, against its restated intrinsics (cuda_emu.h defines
// B2_EMU_DEVICE_HELPERS).
#if defined(__CUDACC__) || defined(B2_EMU_DEVICE_HELPERS)
__device__ __forceinline__ u32 lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ u32 warp_id() { return threadIdx.x >> 5; }

// Inclusive warp scans
__device__ __forceinline__ u32 warp_incl_add(u32 v) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { u32 t = __shfl_up_sync(0xffffffffu, v, o); if (lane_id() >= (u32)o) v += t; }
  return v;
}
__device__ __forceinline__ i32 warp_incl_max(i32 v) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { i32 t = __shfl_up_sync(0xffffffffu, v, o); if (lane_id() >= (u32)o) v = max(v, t); }
  return v;
}
// Block exclusive add-scan; `sm` needs 33 u32.  Returns exclusive prefix; *total = block sum.
// All threads must call.  blockDim.x multiple of 32, <= 1024.
__device__ __forceinline__ u32 block_excl_add(u32 v, u32 *sm, u32 *total) {
  u32 inc = warp_incl_add(v);
  u32 w = warp_id(), l = lane_id(), nw = blockDim.x >> 5;
  __syncthreads();
  if (l == 31) sm[w] = inc;
  __syncthreads();
  if (w == 0) {
    u32 x = l < nw ? sm[l] : 0;
    u32 xi = warp_incl_add(x);
    sm[l] = xi - x;
    if (l == 31) sm[32] = xi;
  }
  __syncthreads();
  u32 r = sm[w] + inc - v;
  if (total) *total = sm[32];
  return r;
}
// Block exclusive max-scan over i32 (identity = INT_MIN passed by caller as `ident`).
__device__ __forceinline__ i32 block_excl_max(i32 v, i32 ident, i32 *sm, i32 *total) {
  i32 inc = warp_incl_max(v);
  u32 w = warp_id(), l = lane_id(), nw = blockDim.x >> 5;
  __syncthreads();
  if (l == 31) sm[w] = inc;
  __syncthreads();
  if (w == 0) {
    i32 x = l < nw ? sm[l] : ident;
    i32 xi = warp_incl_max(x);
    i32 ex = __shfl_up_sync(0xffffffffu, xi, 1);
    if (l == 0) ex = ident;
    sm[l] = ex;
    if (l == 31) sm[32] = xi;
  }
  __syncthreads();
  i32 prev = __shfl_up_sync(0xffffffffu, inc, 1);
  if (l == 0) prev = ident;
  i32 r = max(sm[w], prev);
  if (total) *total = sm[32];
  return r;
}
// ---- GF(2) polynomial arithmetic for the CRCs (bzip2.adb:34-118; zip-crc_crypto.adb:31-61) ------
#define CRC_POLY 0x04C11DB7u
__device__ __forceinline__ u32 gf_mulmod(u32 a, u32 b) {
  // (a * b) mod P over GF(2); bit i = coefficient of x^i
  u32 r = 0;
#pragma unroll 4
  for (int i = 31; i >= 0; i--) {
    r = (r << 1) ^ ((r & 0x80000000u) ? CRC_POLY : 0u);
    if ((b >> i) & 1u) r ^= a;
  }
  return r;
}
#endif
