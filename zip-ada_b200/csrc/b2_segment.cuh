// Stage A3: entropy segmentation (Segment_by_Entropy) on the device.
//
// Reference: zip_lib/data_segmentation.adb:39-105, instantiated with the two profiles of
// zip_lib/bzip2-encoding.adb:1262-1281.
//
// One CTA per chunk replays the running FP64 entropy sum.  Both profiles share window_size =
// 16_000, hence the same entropy series; they differ in thresholds and marks only.
// T[c] = -(c/16000)*ln(c/16000) is built on the host with glibc `log` (SURVEY §9 R7).
//
// The sum is order dependent (four roundings per input byte, :75-90).  It is replayed 256 steps
// at a time:
//  * the window counts met by the incoming / outgoing byte of every step are derived in parallel
//    (integer, exact): counts at the batch start + occurrences earlier in the batch (no atomics: inside
//    a warp equal bytes are found with match.any, across warps by a 256-column prefix);
//  * the sum is followed as an integer k' in units of u' = the ulp of a binade B, over the two binades
//    [2^B, 2^(B+2)): a round-to-nearest-even add of a term d lands on the grid u' (result in binade B) or
//    2u' (result in binade B+1); which one is predicted from the sum at the batch start plus the step's
//    own terms and verified afterwards.  Given the grid, fl (k' u' + d) is a map on k' that only looks at
//    k' mod 4 (where exact ties go depends on the parity of k' or of k'/2): "k' -> k' + a[k' mod 4]".
//    Such maps compose associatively, so the 4 x 256 roundings of a batch are a prefix scan over the CTA.
//    Ties are frequent (d / u' has few fractional bits), hence the care;
//  * the first step whose prediction fails (the sum drifted across 2^(B+1), or left the two binades) is
//    done with its four literal adds and the scan restarts behind it; sums below 2^-12 (windows that are
//    nearly one byte value) and batches with many restarts are replayed by one warp with the literal
//    chain of adds.
//
// Included by b2_segment.cu; also compiled for the host by tests/emu (a thread-per-lane emulation of one CTA that
// checks the sum after every step against the oracle's literal chain - `-m "not gpu"`), hence the B2_EMU switch.
#pragma once
#include "b2_common.cuh"
#include "b2_kernels.h"

#define SEG_WINDOW 16000
#define SG_THREADS 256
#define SG_WARPS (SG_THREADS / 32)

typedef long long i64s;

__device__ __forceinline__ double pow2d(int e) { return __longlong_as_double((long long)(e + 1023) << 52); }   // 2^e, -1022 <= e <= 1023

// k -> k + a[k mod N], N = 2 (one binade: only the parity of k matters) or 4 (two binades)
template <int N> struct PF { i64s a[N]; };

template <int N> __device__ __forceinline__ i64s pf_pick(const PF<N> &g, i64s idx) {
  const int r = (int)(idx & (N - 1));
  if (N == 2) return r ? g.a[1] : g.a[0];
  const i64s lo = (r & 1) ? g.a[1] : g.a[0];
  const i64s hi = (r & 1) ? g.a[N - 1] : g.a[N - 2];
  return (r & 2) ? hi : lo;
}
template <int N> __device__ __forceinline__ PF<N> pf_compose(const PF<N> &f, const PF<N> &g) {   // first f, then g
  PF<N> r;
#pragma unroll
  for (int i = 0; i < N; i++) r.a[i] = f.a[i] + pf_pick<N>(g, (i64s)i + f.a[i]);
  return r;
}
// One add applied to a known k: the same rounding as pf_term below, without the table.
__device__ __forceinline__ i64s pf_apply(i64s k, double x, bool coarse) {
  const double fl = floor(x);
  const i64s X = (i64s)fl;
  const double fr = x - fl;
  if (!coarse) {
    const i64s m = X + (fr > 0.5 ? 1 : 0);
    return k + m + (((fr == 0.5) && ((k + m) & 1)) ? 1 : 0);
  }
  const i64s Y = X + (k & 1);
  const bool odd = (Y & 1) != 0;
  const i64s q = (k >> 1) + (Y >> 1) + ((odd && fr > 0.0) ? 1 : 0);
  return 2 * (q + ((odd && fr == 0.0 && (q & 1)) ? 1 : 0));
}
// The add of a term x (in units of u', any real) whose result lies on the grid u' (coarse = false) or
// 2u' (coarse = true, N = 4 only), round to nearest, ties to even.
template <int N> __device__ __forceinline__ PF<N> pf_term(double x, bool coarse) {
  const double fl = floor(x);
  const i64s X = (i64s)fl;
  const double fr = x - fl;                         // exact: x has at most 53 significant bits
  PF<N> f;
  if (N == 2 || !coarse) {
    const i64s m = X + (fr > 0.5 ? 1 : 0);
    const bool tie = fr == 0.5;
#pragma unroll
    for (int r = 0; r < N; r++) f.a[r] = m + ((tie && ((r + m) & 1)) ? 1 : 0);
  } else {
    // k' = 2q + b: (k' + x) / 2 = q + (X + b) / 2 + fr / 2
#pragma unroll
    for (int b = 0; b < 2; b++) {
      const i64s Y = X + b;
      const bool odd = (Y & 1) != 0;
      const i64s m = (Y >> 1) + ((odd && fr > 0.0) ? 1 : 0);
      const bool tie = odd && fr == 0.0;
#pragma unroll
      for (int qp = 0; qp < 2; qp++) f.a[(2 * qp + b) & (N - 1)] = 2 * (m + ((tie && ((qp + m) & 1)) ? 1 : 0)) - b;
    }
  }
  return f;
}

struct SegSmem {
  u32 F[256];                      // window counts at the batch start
  u32 Hn[SG_WARPS][256];           // occurrences of each byte among the incoming bytes of a warp
  u32 Ho[SG_WARPS][256];           // ... among the outgoing bytes
  u16 Pn[SG_WARPS][256];           // the same, summed over the warps before
  u16 Po[SG_WARPS][256];
  double terms[SG_THREADS * 4];    // serial replay: the four table terms of every step
  double series[SG_THREADS];       // serial replay: the sum after every step
  i64s wtot[SG_WARPS][4];
  double cutval[2];
  double restartE;
  u32 first[2];
  u32 firstbad;
  u8 bn[SG_THREADS], bo[SG_THREADS];
  u32 pm_lt[8][32], pm_le[8][32];
  double entropy;
};

// One attempt at the steps of a batch from the sum E: every participating thread gets the sum before
// (kb) and after (k) its step in units of u' = 1 / scale, and whether its step broke an assumption.
template <int N> __device__ __forceinline__ void seg_scan(SegSmem &S, double E, double scale, double split, bool part,
                                                          const double (&d)[4], i64s &kb, i64s &k, bool &mybad) {
  const u32 l = lane_id(), w = warp_id();
  const i64s K0 = (i64s)(E * scale);                      // exact, in [2^52, 2^53) (N = 2) or [2^52, 2^54)
  // predicted grid of each of my four results: from E and my own terms (the drift of the sum over
  // the steps before me is small; a wrong guess is caught below)
  u32 coarse = 0;
  PF<N> inc, mine_f;
  {
    double v = E;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      v += d[j];
      const bool cj = N == 4 && part && v >= split;
      coarse |= (u32)cj << j;
      const PF<N> fj = pf_term<N>(part ? d[j] * scale : 0.0, cj);
      inc = j == 0 ? fj : pf_compose<N>(inc, fj);
    }
    mine_f = inc;
  }
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    PF<N> nb;
#pragma unroll
    for (int r = 0; r < N; r++) nb.a[r] = __shfl_up_sync(0xffffffffu, inc.a[r], o);
    if (l >= (u32)o) inc = pf_compose<N>(nb, inc);
  }
  if (l == 31) {
#pragma unroll
    for (int r = 0; r < N; r++) S.wtot[w][r] = inc.a[r];
  }
  PF<N> excl;                                              // lanes before me in my warp
#pragma unroll
  for (int r = 0; r < N; r++) { excl.a[r] = __shfl_up_sync(0xffffffffu, inc.a[r], 1); if (l == 0) excl.a[r] = 0; }
  __syncthreads();
  PF<N> pre;                                               // warps before mine
#pragma unroll
  for (int r = 0; r < N; r++) pre.a[r] = 0;
  for (u32 ww = 0; ww < w; ww++) {
    PF<N> g;
#pragma unroll
    for (int r = 0; r < N; r++) g.a[r] = S.wtot[ww][r];
    pre = pf_compose<N>(pre, g);
  }
  pre = pf_compose<N>(pre, excl);
  kb = K0 + pf_pick<N>(pre, K0);                           // the sum before my step, in units of u'
  if (N == 2) {
    // One binade is only chosen when E is at least 0.75 away from both ends of its binade: a term is at
    // most 1/e = 0.368 and the sum moves by less than 256 * 2 * ln (16000) / 16000 = 0.31 over a batch, so
    // no intermediate sum can leave the binade and nothing has to be checked.
    k = K0 + pf_pick<N>(pf_compose<N>(pre, mine_f), K0);
    mybad = false;
    return;
  }
  k = kb;
  const i64s lo = 1ll << 52, mid = 1ll << 53, hi = N == 2 ? mid : (1ll << 54);
  mybad = false;
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const bool cj = ((coarse >> j) & 1u) != 0;
    k = pf_apply(k, d[j] * scale, cj);
    mybad = mybad || k < lo || k >= hi || (N == 4 && ((k >= mid) != cj));
  }
  mybad = mybad && part;
}

// Test taps, compiled in only for TAPS = true (b2_dbg_segment and tests/emu; every production launch passes nullptr and
// runs the TAPS = false instantiation, which is the kernel without them):
//  dbg_series: the sum after every step of the chunk, at step index - SEG_WINDOW (data_segmentation.adb:91);
//  dbg_paths:  per CTA, batches that start on one binade / on two binades, failed predictions (restarts),
//              batches finished by the literal warp chain.
#define SEG_PATH_ONE 0
#define SEG_PATH_TWO 1
#define SEG_PATH_RESTART 2
#define SEG_PATH_LITERAL 3
template <bool TAPS>
__global__ void __launch_bounds__(SG_THREADS, 3)
k_segment(const u8 *__restrict__ in, const B2Chunk *chunks, u32 n_chunks,
          const double *__restrict__ T, u32 *__restrict__ seg, u32 *__restrict__ nseg, const u32 *progress,
          double *dbg_series, u32 *dbg_paths) {
#ifdef B2_EMU
  SegSmem &S = *reinterpret_cast<SegSmem *>(emu_dynamic_smem());   // poisoned for every CTA
#else
  __shared__ SegSmem S;
#endif
  const u32 c = blockIdx.x;
  if (c >= n_chunks) return;
  const u32 tid = threadIdx.x, l = lane_id(), w = warp_id();
  if (progress) {
    // following the chunk chain (k_cut_chain on another stream): wait until my chunk is there.  CTAs
    // are dispatched in chunk order, so the resident ones are always the next chunks to appear; the
    // CTAs of the unused tail of the table leave when the chain reports the end.
    if (tid == 0) {
      u32 state = 2;                                    // 0 no such chunk, 1 ready, 2 gave up
      for (u32 spins = 0; spins < 8000000u; spins++) {
        const u32 done = ((const volatile u32 *)progress)[1];
        const u32 ready = ((const volatile u32 *)progress)[0];
        if (ready > c) { state = 1; break; }
        if (done) { state = 0; break; }
        __nanosleep(400);
      }
      S.first[0] = state;
      if (state == 2) { nseg[2 * c] = B2_SEG_GAVE_UP; nseg[2 * c + 1] = B2_SEG_GAVE_UP; }   // the host segments again after the chain
    }
    __syncthreads();
    const u32 state = S.first[0];
    __syncthreads();
    if (state != 1) return;
    __threadfence();
  }
  const u32 lt = (1u << l) - 1u;
  // (the table may be written by the chain kernel while this kernel runs: no read-only cache path)
  const u8 *buf = in + __ldcg(&chunks[c].start);
  const i32 len = (i32)__ldcg(&chunks[c].len);
  const double thr[2] = {(double)0.6f, (double)0.4f};    // Float generic formal widened (data_segmentation.ads:43)
  const i32 ithr[2] = {4000, 8000};
  i32 index_mark[2] = {1, 1};
  double mark[2] = {0.0, 0.0};
  u32 cnt[2] = {0, 0};
  u32 *out[2] = {seg + (size_t)(2 * c) * B2_MAX_SEG, seg + (size_t)(2 * c + 1) * B2_MAX_SEG};
  const bool act[2] = {len > SEG_WINDOW + ithr[0], len > SEG_WINDOW + ithr[1]};
  if (act[0] || act[1]) {
    S.F[tid] = 0;
    for (int i = tid; i < SG_WARPS * 256; i += SG_THREADS) { (&S.Hn[0][0])[i] = 0; (&S.Ho[0][0])[i] = 0; }
    __syncthreads();
    for (i32 i = tid; i < SEG_WINDOW; i += SG_THREADS) atomicAdd(&S.F[buf[i]], 1u);
    __syncthreads();
    // initial entropy, b = 0 .. 255 in order (data_segmentation.adb:63-72), by warp 0
    if (w == 0) {
      double e = 0.0;
      for (int g = 0; g < 8; g++) {
        const u32 f = S.F[g * 32 + l];
        const double tv = T[f];
        for (int k = 0; k < 32; k++) {
          const u32 fk = __shfl_sync(0xffffffffu, f, k);
          const double tk = __shfl_sync(0xffffffffu, tv, k);
          if (fk > 0) e = __dadd_rn(e, tk);
        }
      }
      if (l == 0) S.entropy = e;
    }
    __syncthreads();
    double entropy = S.entropy;
    mark[0] = entropy; mark[1] = entropy;
    // byte-prefix masks for "count bytes j < l" / "j <= l" over a 32-byte row held as 8 words
    // (kept in shared memory, one column per lane, to spare 16 registers)
    if (w == 0) {
#pragma unroll
      for (int q = 0; q < 8; q++) {
        const int lo = 4 * q;
        const int a_lt = (int)l - lo, a_le = (int)l + 1 - lo;
        S.pm_lt[q][l] = a_lt >= 4 ? 0xFFFFFFFFu : (a_lt <= 0 ? 0u : ((1u << (8 * a_lt)) - 1u));
        S.pm_le[q][l] = a_le >= 4 ? 0xFFFFFFFFu : (a_le <= 0 ? 0u : ((1u << (8 * a_le)) - 1u));
      }
    }
    __syncthreads();
    const u32 *rown = reinterpret_cast<const u32 *>(S.bn + 32 * w);
    const u32 *rowo = reinterpret_cast<const u32 *>(S.bo + 32 * w);
    // bytes are loaded one batch ahead of their use
    u32 pre_n = (SEG_WINDOW + (i32)tid < len) ? buf[SEG_WINDOW + tid] : 0u;
    u32 pre_o = (SEG_WINDOW + (i32)tid < len) ? buf[tid] : 0u;
    for (i32 i0 = SEG_WINDOW; i0 < len; i0 += SG_THREADS) {   // 0-based step index; reference i = index + 1
      const i32 i = i0 + (i32)tid;
      const bool valid = i < len;
      const u32 bn = pre_n, bo = pre_o;                       // incoming / outgoing byte of my step
      {
        const i32 i2 = i + SG_THREADS;
        const bool v2 = i2 < len;
        pre_n = v2 ? buf[i2] : 0u;
        pre_o = v2 ? buf[i2 - SEG_WINDOW] : 0u;
      }
      const int steps = min(SG_THREADS, len - i0);
      S.bn[tid] = (u8)bn; S.bo[tid] = (u8)bo;
      if (tid < 2) S.first[tid] = 0xFFFFFFFFu;
      // occurrences in my own warp: the first lane of every distinct byte records the count
      const u32 key_n = valid ? bn : (256u + l), key_o = valid ? bo : (512u + l);
      const u32 peers_n = __match_any_sync(0xffffffffu, key_n), peers_o = __match_any_sync(0xffffffffu, key_o);
      const u32 c_nn = __popc(peers_n & lt);                  // #{j<k : bn_j = bn_k}
      const u32 c_oo = __popc(peers_o & lt);                  // #{j<k : bo_j = bo_k}
      const bool lead_n = valid && c_nn == 0, lead_o = valid && c_oo == 0;
      if (lead_n) S.Hn[w][bn] = __popc(peers_n);
      if (lead_o) S.Ho[w][bo] = __popc(peers_o);
      __syncthreads();
      i32 dF;                                                 // change of the window count of byte value `tid` over the batch
      {                                                       // per byte value: occurrences in the warps before
        u32 rn = 0, ro = 0;
#pragma unroll
        for (int ww = 0; ww < SG_WARPS; ww++) {
          S.Pn[ww][tid] = (u16)rn; S.Po[ww][tid] = (u16)ro;
          rn += S.Hn[ww][tid]; ro += S.Ho[ww][tid];
        }
        dF = (i32)rn - (i32)ro;
      }
      __syncthreads();
      const u32 sp_n = bn * 0x01010101u, sp_o = bo * 0x01010101u;
      u32 c_on = 0, c_no = 0;
#pragma unroll
      for (int q = 0; q < 8; q++) {
        c_on += __popc(__vcmpeq4(rowo[q], sp_n) & S.pm_lt[q][l]);   // #{j<k  : bo_j = bn_k}
        c_no += __popc(__vcmpeq4(rown[q], sp_o) & S.pm_le[q][l]);   // #{j<=k : bn_j = bo_k}
      }
      c_on >>= 3; c_no >>= 3;
      // invalid lanes hold byte 0 in the rows: they are the LAST lanes of the last warp, so they are
      // never counted by a valid lane (prefix masks), and their own results are discarded
      u32 fnb = 0, fob = 1;
      if (valid) {
        fnb = S.F[bn] + (S.Pn[w][bn] + c_nn) - (S.Po[w][bn] + c_on);        // count met by the incoming byte
        fob = S.F[bo] + (S.Pn[w][bo] + c_no) - (S.Po[w][bo] + c_oo);        // count met by the outgoing byte
      }
      const double c1 = T[fnb], c2 = T[fnb + 1], c3 = T[fob], c4 = T[fob - 1];   // T[0] = 0 covers "p = 0" (:84-89)
      // Replay of the steps of this batch.  `start` = first step not yet replayed, E = the sum before it.
      double mine = 0.0;
      u32 start = 0;
      double E = entropy;
      int attempts = 0;
      bool finished = false;
      while (!finished) {
        if (E >= 0x1p-12 && E < 8.0 && attempts < 12) {
          // one binade when no add of this batch can leave the binade of E (every term is below 0.37 and
          // the sum moves by less than 0.3 over a batch), else the two binades [2^B, 2^(B+2)) around E: the
          // one below when E sits in the lower half of its own
          const int eb = (int)((__double_as_longlong(E) >> 52) & 0x7FF) - 1023;       // E is normal and positive here
          const double blo = pow2d(eb);
          const bool one = (E - blo >= 0.75) && (2.0 * blo - E > 0.75);
          const int B = one ? eb : ((E < 1.5 * blo) ? eb - 1 : eb);
          const double scale = pow2d(52 - B), inv = pow2d(B - 52);
          const bool part = valid && tid >= start;
          if (tid == 0) S.firstbad = 0xFFFFFFFFu;
          const double d[4] = {-c1, c2, -c3, c4};
          i64s kb, k;
          bool mybad;
          if (one) seg_scan<2>(S, E, scale, pow2d(B + 1), part, d, kb, k, mybad);
          else seg_scan<4>(S, E, scale, pow2d(B + 1), part, d, kb, k, mybad);
          if (TAPS && dbg_paths && tid == 0 && attempts == 0) dbg_paths[4 * c + (one ? SEG_PATH_ONE : SEG_PATH_TWO)]++;
          if (__syncthreads_or(mybad) == 0) {
            if (part) mine = (double)k * inv;
            if ((int)tid == steps - 1) S.entropy = mine;
            finished = true;
          } else {
            // everything before the first failing step stands; that step is done with the four literal
            // adds, and the scan restarts behind it
            if (TAPS && dbg_paths && tid == 0) dbg_paths[4 * c + SEG_PATH_RESTART]++;
            if (mybad) atomicMin(&S.firstbad, tid);
            __syncthreads();
            const u32 fb = S.firstbad;
            if (part && tid < fb) mine = (double)k * inv;
            if (tid == fb) {
              double ee = (double)kb * inv;
              ee = __dsub_rn(ee, c1);                             // data_segmentation.adb:75-90
              ee = __dadd_rn(ee, c2);
              ee = __dsub_rn(ee, c3);
              ee = __dadd_rn(ee, c4);
              mine = ee;
              S.restartE = ee;
              if ((int)tid == steps - 1) S.entropy = ee;
            }
            __syncthreads();
            E = S.restartE;
            start = fb + 1;
            attempts++;
            if ((int)start >= steps) finished = true;
          }
        } else {
          // outside the range of the integer replay (sum near zero, or too many restarts in one
          // batch): the literal sequential chain for the remaining steps, by one warp
          if (TAPS && dbg_paths && tid == 0) dbg_paths[4 * c + SEG_PATH_LITERAL]++;
          S.terms[tid * 4 + 0] = c1; S.terms[tid * 4 + 1] = c2; S.terms[tid * 4 + 2] = c3; S.terms[tid * 4 + 3] = c4;
          __syncthreads();
          if (w == 0) {
            double e = E;
            for (int k = (int)start; k < steps; k++) {
              const double2 ab = *reinterpret_cast<const double2 *>(&S.terms[k * 4]);
              const double2 cd = *reinterpret_cast<const double2 *>(&S.terms[k * 4 + 2]);
              e = __dsub_rn(e, ab.x);                           // data_segmentation.adb:75-90
              e = __dadd_rn(e, ab.y);
              e = __dsub_rn(e, cd.x);
              e = __dadd_rn(e, cd.y);
              if (l == 0) S.series[k] = e;
            }
            if (l == 0) S.entropy = e;
          }
          __syncthreads();
          if (tid >= start) mine = S.series[tid];
          finished = true;
        }
      }
      if (TAPS && dbg_series && valid) dbg_series[i - SEG_WINDOW] = mine;
      // threshold tests for the 256 steps at once (:91-97).  A cut moves index_mark to within 256 of
      // every later step of the batch, so at most one cut per profile can happen in a batch.
      const i32 sp = i + 1 - SEG_WINDOW;
      bool maybe[2];
#pragma unroll
      for (int p = 0; p < 2; p++) {
        maybe[p] = act[p] && (i0 + steps - SEG_WINDOW - index_mark[p] > ithr[p]);
        if (maybe[p] && valid && fabs(__dsub_rn(mine, mark[p])) > thr[p] && (sp - index_mark[p] > ithr[p])) atomicMin(&S.first[p], tid);
      }
      // clear my histogram entries for the next batch
      if (lead_n) S.Hn[w][bn] = 0;
      if (lead_o) S.Ho[w][bo] = 0;
      __syncthreads();
      S.F[tid] = (u32)((i32)S.F[tid] + dF);                   // window counts at the start of the next batch
#pragma unroll
      for (int p = 0; p < 2; p++) if (maybe[p] && S.first[p] == tid) S.cutval[p] = mine;
      __syncthreads();
      entropy = S.entropy;
#pragma unroll
      for (int p = 0; p < 2; p++) {
        if (maybe[p] && S.first[p] != 0xFFFFFFFFu) {
          const i32 seg_point = i0 + (i32)S.first[p] + 1 - SEG_WINDOW;
          if (tid == 0 && cnt[p] < B2_MAX_SEG - 1) out[p][cnt[p]] = (u32)seg_point;
          cnt[p]++;
          index_mark[p] = seg_point;
          mark[p] = S.cutval[p];
        }
      }
      __syncthreads();
    }
  }
  if (tid == 0) {
    for (int k = 0; k < 2; k++) {
      if (len > 0) { if (cnt[k] < B2_MAX_SEG) out[k][cnt[k]] = (u32)len; cnt[k]++; }   // :102-104
    }
    __threadfence();                                   // the cut lists are complete before their counts show
    nseg[2 * c] = cnt[0]; nseg[2 * c + 1] = cnt[1];
  }
}
