// ORACLE — TEST INFRASTRUCTURE ONLY.  Not part of the product path.
//
// CPU restatement (C++17, single thread, no CUDA) of Zip-Ada's BZip2 stream
// encoder `BZip2.Encoding.Encode` (reference v.62).  Only tests/,
// __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
// may load this library.  The CUDA product (zip-ada_b200/csrc) never calls it.
//
// PARITY STATUS: **parity unpinned**.  The reference cannot be compiled here (no
// GNAT) and its own tests hold no golden encoder bytes (SURVEY.md §0.5, §8c).
// What pins this oracle: (i) every stream it writes is decoded by the
// independent decoders in this image (libbz2 1.0.8 through Python `bz2` and
// /usr/bin/bzip2) back to the input; (ii) the steps whose result is a unique
// function of the input (RLE1, BWT+origin, MTF/RLE2, CRCs, canonical codes,
// bit layout) are checked against a second, literal restatement (`faithful`
// BWT = the reference's heap sort + rotation comparator); (iii) the
// length-limited code lengths are checked for optimality against an
// independent package-merge.  Two steps depend on code that is NOT under
// /root/reference: GNAT's Ada.Containers.Generic_Constrained_Array_Sort
// (libgnat a-cgcaso.adb, no pinned version; restated below from its published
// algorithm: heap sort "adapted from GNAT.Heap_Sort_G") and libm `log`.
//
// Every function cites the reference file:line it follows
// (paths relative to /root/reference/zip_lib/).
//
// Build flags mirror zipada.gpr "Fast" mode (:91-108): -O2, no -march, no
// -ffast-math, so double/float arithmetic is plain IEEE SSE2.

#include <cstdint>
#include <cstring>
#include <cstdlib>
#include <cmath>
#include <vector>
#include <algorithm>
#include <numeric>
#include <atomic>
#include <thread>

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;
typedef int32_t i32;
typedef int64_t i64;

namespace {

// ---------------------------------------------------------------------------
// bzip2.ads:77-122 — format constants
// ---------------------------------------------------------------------------
const int run_a = 0;                 // bzip2.ads:83
const int run_b = 1;                 // bzip2.ads:84
const int max_alphabet_size = 258;   // bzip2.ads:92
const int min_entropy_coders = 2;    // bzip2.ads:109
const int max_entropy_coders = 6;    // bzip2.ads:110
const int group_size = 50;           // bzip2.ads:111
const i32 sub_block_size = 100000;   // bzip2.ads:116

// ---------------------------------------------------------------------------
// bzip2.adb:34-118 — CRC-32, MSB first, polynomial 0x04C11DB7
// (table generated instead of typed in; identical values)
// ---------------------------------------------------------------------------
u32 crc_table[256];
bool crc_table_ready = false;
void crc_make_table() {
  if (crc_table_ready) return;
  for (u32 i = 0; i < 256; i++) {
    u32 c = i << 24;
    for (int k = 0; k < 8; k++) c = (c & 0x80000000u) ? (c << 1) ^ 0x04C11DB7u : (c << 1);
    crc_table[i] = c;
  }
  crc_table_ready = true;
}
inline void crc_init(u32 &c) { c = 0xFFFFFFFFu; }                       // bzip2.adb:110-113
inline u32 crc_final(u32 c) { return ~c; }                               // bzip2.adb:115-118
inline void crc_update(u32 &c, u8 v) {                                   // bzip2.adb:102-108
  c = crc_table[0xFF & ((c >> 24) ^ (u32)v)] ^ (c << 8);
}

// ---------------------------------------------------------------------------
// bzip2-buffers.ads:19-36, .adb:9-43 — MSB-first bit writer
// State mirrors Bit_Buffer_Type: `buffer` (partial byte), `bit_index`
// (7 = empty .. 0), destination bytes; destination_index == dest.size().
// ---------------------------------------------------------------------------
struct BitBuffer {
  u8 buffer = 0;
  int bit_index = 7;
  std::vector<u8> dest;
  void attach_new() { dest.clear(); }                                    // bzip2-buffers.adb:3-7
  void flush() {                                                         // bzip2-buffers.adb:9-16
    dest.push_back(buffer);
    buffer = 0;
    bit_index = 7;
  }
  void put_bits(u32 data, int amount) {                                  // bzip2-buffers.adb:18-31
    for (int count = amount; count >= 1; count--) {
      if (data & (1u << (count - 1))) buffer |= (u8)(1u << bit_index);
      if (bit_index == 0) flush(); else bit_index--;
    }
  }
  void put_bool(bool b) { put_bits(b ? 1 : 0, 1); }                      // bzip2-buffers.adb:33-36
  void put_string(const char *s, int n) {                                // bzip2-buffers.adb:38-43
    for (int i = 0; i < n; i++) put_bits((u8)s[i], 8);
  }
  u64 total_bits() const { return (u64)dest.size() * 8 + (u64)(7 - bit_index); }
};

// ---------------------------------------------------------------------------
// GNAT runtime: Ada.Containers.Generic_Constrained_Array_Sort (a-cgcaso.adb).
// NOT under /root/reference; restated from the published FSF GNAT algorithm
// (in-place heap sort adapted from GNAT.Heap_Sort_G, Floyd's variant: sift the
// hole down to a leaf, then climb).  1-based indices.  `lt` is the generic "<".
// Used by bzip2-encoding.adb:257-261 (BWT, total order: any sort gives the same
// result) and :564-568/:619 (Ranking_Sort, key-only order: tie order depends
// on exactly this algorithm).  Isolated here on purpose (SURVEY §7.3 #1).
// ---------------------------------------------------------------------------
template <class T, class Less>
void gnat_constrained_array_sort(T *a1 /* a1[1..n] valid */, i64 n, Less lt) {
  i64 max = n;
  T temp;
  auto sift = [&](i64 s) {
    i64 c = s;
    for (;;) {
      i64 son = 2 * c;
      if (son > max) break;
      if (son < max && lt(a1[son], a1[son + 1])) son = son + 1;
      a1[c] = a1[son];
      c = son;
    }
    while (c != s) {
      i64 father = c / 2;
      if (lt(a1[father], temp)) {
        a1[c] = a1[father];
        c = father;
      } else break;
    }
    a1[c] = temp;
  };
  for (i64 j = max / 2; j >= 1; j--) {
    temp = a1[j];
    sift(j);
  }
  while (max > 1) {
    temp = a1[max];
    a1[max] = a1[1];
    max = max - 1;
    sift(1);
  }
}

// ---------------------------------------------------------------------------
// huffman-encoding-length_limited_coding.adb:46-280 — boundary package-merge,
// literal restatement including the in-tree unstable Quick_sort (:191-223)
// whose tie order decides which equal-weight symbols get the longer codes.
// counts[0..n-1] -> lens[0..n-1], max_bits = length limit.
// ---------------------------------------------------------------------------
struct LLHC {
  struct Node { i64 weight; i64 count; i32 tail; bool in_use; };         // :56-61
  struct Leaf { i64 weight; int symbol; };                               // :63-66
  static const i32 null_index = 0x7FFFFFFF;                              // :52
  int max_bits;
  std::vector<Node> pool;                                                // :69
  i32 pool_next = 0;                                                     // :70
  i32 lists[32][2];                                                      // :72-73
  std::vector<Leaf> leaves;                                              // :75-76
  i64 num_symbols = 0;                                                   // :78

  void init_node(i64 weight, i64 count, i32 tail, i32 idx) {             // :87-93
    pool[idx].weight = weight; pool[idx].count = count; pool[idx].tail = tail; pool[idx].in_use = true;
  }
  i32 get_free_node(bool use_lists) {                                    // :98-122
    i32 pool_last = (i32)pool.size() - 1;
    for (;;) {
      if (pool_next > pool_last) {
        for (auto &p : pool) p.in_use = false;
        if (use_lists) {
          for (int i = 0; i <= max_bits * 2 - 1; i++) {
            i32 node_idx = lists[i / 2][i % 2];
            while (node_idx != null_index) {
              pool[node_idx].in_use = true;
              node_idx = pool[node_idx].tail;
            }
          }
        }
        pool_next = 0;
      }
      if (!pool[pool_next].in_use) break;
      pool_next++;
    }
    pool_next++;
    return pool_next - 1;
  }
  void boundary_pm(int index, bool final) {                              // :131-163
    i64 lastcount = pool[lists[index][1]].count;
    if (index == 0 && lastcount >= num_symbols) return;
    i32 newchain = get_free_node(true);
    i32 oldchain = lists[index][1];
    lists[index][0] = oldchain; lists[index][1] = newchain;
    if (index == 0) {
      init_node(leaves[lastcount].weight, lastcount + 1, null_index, newchain);
    } else {
      i64 sum = pool[lists[index - 1][0]].weight + pool[lists[index - 1][1]].weight;
      if (lastcount < num_symbols && sum > leaves[lastcount].weight) {
        init_node(leaves[lastcount].weight, lastcount + 1, pool[oldchain].tail, newchain);
      } else {
        init_node(sum, lastcount, lists[index - 1][1], newchain);
        if (!final) {
          boundary_pm(index - 1, false);
          boundary_pm(index - 1, false);
        }
      }
    }
  }
  static void quick_sort(Leaf *a, i64 n) {                               // :191-223
    if (n < 2) return;
    Leaf p = a[n / 2];
    i64 i = 0, j = n - 1;
    for (;;) {
      while (a[i].weight < p.weight) i++;
      while (p.weight < a[j].weight) j--;
      if (i >= j) break;
      Leaf t = a[i]; a[i] = a[j]; a[j] = t;
      i++; j--;
    }
    quick_sort(a, i);
    quick_sort(a + i, n - i);
  }
  void run(const u32 *freq, int n, int max_bits_, u32 *bit_lengths) {    // :227-280
    max_bits = max_bits_;
    pool.assign((size_t)(2 * max_bits * (max_bits + 1)), Node{0, 0, null_index, false});
    pool_next = 0;
    leaves.assign((size_t)n, Leaf{0, 0});
    num_symbols = 0;
    for (int a = 0; a < n; a++) bit_lengths[a] = 0;
    for (int a = 0; a < n; a++)
      if (freq[a] > 0) { leaves[num_symbols].weight = freq[a]; leaves[num_symbols].symbol = a; num_symbols++; }
    if (num_symbols == 0) return;
    if (num_symbols == 1) { bit_lengths[leaves[0].symbol] = 1; return; }
    quick_sort(leaves.data(), num_symbols);
    // Init_Lists :167-174
    i32 node0 = get_free_node(false);
    i32 node1 = get_free_node(false);
    init_node(leaves[0].weight, 1, null_index, node0);
    init_node(leaves[1].weight, 2, null_index, node1);
    for (int i = 0; i < max_bits; i++) { lists[i][0] = node0; lists[i][1] = node1; }
    i64 runs = 2 * num_symbols - 4;                                      // :259
    for (i64 i = 1; i <= runs; i++) boundary_pm(max_bits - 1, i == runs);
    // Extract_Bit_Lengths :180-189
    i32 node_idx = lists[max_bits - 1][1];
    while (node_idx != null_index) {
      for (i64 i = 0; i <= pool[node_idx].count - 1; i++) bit_lengths[leaves[i].symbol]++;
      node_idx = pool[node_idx].tail;
    }
  }
};

// ---------------------------------------------------------------------------
// huffman-encoding.adb:45-80 — canonical codes from lengths (RFC 1951 3.2.2),
// invert_bit_order = False as called at bzip2-encoding.adb:511-512.
// ---------------------------------------------------------------------------
void prepare_codes(const u32 *len, u32 *code, int n, int max_huffman_bits) {
  std::vector<u32> bl_count(max_huffman_bits + 1, 0), next_code(max_huffman_bits + 1, 0);
  for (int i = 0; i < n; i++) bl_count[len[i]]++;
  u32 c = 0;
  for (int bits = 1; bits <= max_huffman_bits; bits++) {
    c = (c + bl_count[bits - 1]) * 2;
    next_code[bits] = c;
  }
  for (int i = 0; i < n; i++) {
    u32 bl = len[i];
    if (bl > 0) { code[i] = next_code[bl]; next_code[bl]++; } else code[i] = 0;
  }
}

// ---------------------------------------------------------------------------
// data_segmentation.adb:39-105 — entropy change-point detector, FP64, libm log.
// threshold is a Float (single precision) generic formal, widened (ads:43).
// Returns ascending 1-based end indices; last = len (if len > 0).
// series (optional): the running sum after the initial window (i = window_size) and after every
// later step, at the point where it is tested against the threshold (tests/test_emu_segment.py).
// ---------------------------------------------------------------------------
void segment_by_entropy(const u8 *buffer /*0-based*/, i32 len, float discrepancy_threshold,
                        i32 index_threshold, i32 window_size, std::vector<i32> &seg,
                        std::vector<double> *series = nullptr) {
  typedef double Real;                                                   // :41 digits 15
  const Real inv_window_size = 1.0 / (Real)window_size;                  // :44
  i32 freq[256]; Real elem[256];
  for (int i = 0; i < 256; i++) { freq[i] = 0; elem[i] = 0.0; }
  volatile Real entropy = 0.0;  // volatile: forbid any re-association / excess precision
  Real entropy_mark = 0.0;
  i32 index_mark = 1;                                                    // :53
  seg.clear();
  if (len > window_size + index_threshold) {                             // :58
    for (i32 i = 1; i <= len; i++) {
      int bt = buffer[i - 1];
      freq[bt]++;
      if (i == window_size) {                                            // :63-72
        for (int b = 0; b < 256; b++) {
          Real p = (Real)freq[b] * inv_window_size;
          if (p > 0.0) {
            elem[b] = -(p * std::log(p));
            entropy = entropy + elem[b];
          }
        }
        entropy_mark = entropy;
        if (series) series->push_back((Real)entropy);
      } else if (i > window_size) {                                      // :73-98
        entropy = entropy - elem[bt];
        Real p = (Real)freq[bt] * inv_window_size;
        elem[bt] = -(p * std::log(p));
        entropy = entropy + elem[bt];
        bt = buffer[i - window_size - 1];
        entropy = entropy - elem[bt];
        freq[bt]--;
        p = (Real)freq[bt] * inv_window_size;
        if (p > 0.0) {
          elem[bt] = -(p * std::log(p));
          entropy = entropy + elem[bt];
        } else {
          elem[bt] = 0.0;
        }
        if (series) series->push_back((Real)entropy);
        if (std::fabs(entropy - entropy_mark) > (Real)discrepancy_threshold) {
          i32 seg_point = i - window_size;
          if (seg_point - index_mark > index_threshold) {
            seg.push_back(seg_point);
            index_mark = seg_point;
            entropy_mark = entropy;
          }
        }
      }
    }
  }
  if (len > 0) seg.push_back(len);                                       // :102-104
}

// ---------------------------------------------------------------------------
// BWT.  bzip2-encoding.adb:219-296.
// `bwt_faithful` is the literal restatement (GNAT heap sort over offsets with
// the rotation comparator :229-255).  `bwt_fast` computes the same unique
// result (comparator is a total order, SURVEY §9 R1) by cyclic prefix doubling;
// it exists so that the oracle finishes 900k blocks and pathological repeats
// in seconds.  tests/ check fast == faithful on small inputs.
// ---------------------------------------------------------------------------
void bwt_faithful(const u8 *d /*0-based, n bytes*/, i32 n, u8 *out, u32 &bwt_index) {
  bwt_index = 0;
  if (n == 0) return;
  std::vector<i32> offset((size_t)n + 1);
  for (i32 i = 0; i < n; i++) offset[i + 1] = i;                         // :266-268
  auto smaller = [&](i32 left, i32 right) -> bool {                      // :229-255
    i32 il = 1 + (left == 0 ? 0 : n - left);
    i32 ir = 1 + (right == 0 ? 0 : n - right);
    for (i32 i = 0; i < n; i++) {
      u8 l = d[il - 1], r = d[ir - 1];
      if (l < r) return true;
      if (l > r) return false;
      il++; if (il > n) il = 1;
      ir++; if (ir > n) ir = 1;
    }
    return left < right;
  };
  gnat_constrained_array_sort(offset.data(), (i64)n, smaller);           // :270
  for (i32 i = 0; i < n; i++) {                                          // :273-280
    i32 off = offset[i + 1];
    out[i] = d[(((i64)n - 1 - off) % n + n) % n];
    if (off == 0) bwt_index = (u32)i;
  }
}

void bwt_fast(const u8 *d, i32 n, u8 *out, u32 &bwt_index) {
  bwt_index = 0;
  if (n == 0) return;
  if (n == 1) { out[0] = d[0]; return; }
  // sa[] holds rotation START positions; rank[i] = index of the first row of the
  // class of rotation i (equal prefixes share a rank).  Cyclic: successor (i+h) mod n.
  std::vector<i32> sa(n), rank(n);
  std::vector<std::pair<i32, i32>> groups, next_groups;
  {
    // initial order by the first 4 bytes (cyclic) — LSD radix, 4 passes of 8 bits
    std::vector<u32> key(n), key2(n);
    std::vector<i32> sa2(n);
    for (i32 i = 0; i < n; i++) {
      u32 k = 0;
      for (int j = 0; j < 4; j++) k = (k << 8) | d[(i + j) % n];
      key[i] = k; sa[i] = i;
    }
    for (int pass = 0; pass < 4; pass++) {
      u32 cnt[257] = {0};
      int sh = pass * 8;
      for (i32 i = 0; i < n; i++) cnt[((key[i] >> sh) & 255) + 1]++;
      for (int c = 0; c < 256; c++) cnt[c + 1] += cnt[c];
      for (i32 i = 0; i < n; i++) { u32 p = cnt[(key[i] >> sh) & 255]++; key2[p] = key[i]; sa2[p] = sa[i]; }
      key.swap(key2); sa.swap(sa2);
    }
    i32 head = 0;
    for (i32 p = 0; p < n; p++) {
      if (p > 0 && key[p] != key[p - 1]) { if (p - head > 1) groups.push_back({head, p}); head = p; }
      rank[sa[p]] = head;
    }
    if (n - head > 1) groups.push_back({head, n});
  }
  std::vector<std::pair<i32, i32>> ks;      // (key, rotation)
  std::vector<std::pair<i32, i32>> pending; // (rotation, new rank)
  for (i64 h = 4; !groups.empty() && h < n; h *= 2) {
    next_groups.clear(); pending.clear();
    for (auto &g : groups) {
      i32 s = g.first, e = g.second;
      ks.clear();
      for (i32 p = s; p < e; p++) ks.push_back({rank[(i32)(((i64)sa[p] + h) % n)], sa[p]});
      std::sort(ks.begin(), ks.end());
      i32 head = s;
      for (i32 p = s; p < e; p++) {
        sa[p] = ks[p - s].second;
        if (p > s && ks[p - s].first != ks[p - s - 1].first) { if (p - head > 1) next_groups.push_back({head, p}); head = p; }
        pending.push_back({sa[p], head});
      }
      if (e - head > 1) next_groups.push_back({head, e});
    }
    for (auto &u : pending) rank[u.first] = u.second;
    groups.swap(next_groups);
  }
  // Rows of equal rotations (periodic block): content identical, so the last
  // column is identical too; the row of the original message is the FIRST row
  // of its class (offset 0 sorts first, :254) = rank of rotation 0.
  for (i32 i = 0; i < n; i++) out[i] = d[(sa[i] + n - 1) % n];
  bwt_index = (u32)rank[0];
}

// ---------------------------------------------------------------------------
// Taps: every intermediate of one Encode_Block, for the parity harness.
// ---------------------------------------------------------------------------
struct BlockTaps {
  std::vector<u8> rle1, bwt;
  std::vector<u16> mtf;
  std::vector<u8> selector;            // 1-based coder per group
  u32 lens[6][258];
  u32 origin = 0, crc = 0, eob = 0, n_used = 0;
  int ec_count = 0, max_len = 0, sample_width = 0;
  u32 best_cost = 0;
  u64 bits = 0;                         // bits written by this block
  int constructs = 0;                   // number of Construct calls in the search
};

struct EncoderConfig {
  int level;        // 1, 4, 9
  int bwt_mode;     // 0 = fast, 1 = faithful
};

// ---------------------------------------------------------------------------
// bzip2-encoding.adb:148-1134 — Encode_Block
// ---------------------------------------------------------------------------
struct BlockEncoder {
  const EncoderConfig &cfg;
  i32 block_capacity;
  // RLE_1 state
  std::vector<u8> rle_1_data;
  bool in_use[256];
  u32 block_crc;
  // BWT
  std::vector<u8> bwt_data;
  u32 bwt_index = 0;
  // MTF
  std::vector<u16> mtf_data;            // 0-based storage of mtf_data(1..mtf_last)
  i32 mtf_last = 0;
  int normal_symbols_in_use = 0, last_symbol_in_use = 0, EOB = 0;
  // entropy
  u32 descr_len[7][258];                // [1..6][symbol]
  u32 descr_code[7][258];
  int entropy_coder_count = 2;
  i32 selector_count = 0;
  std::vector<u8> selector;             // 1-based index -> coder (1..6); selector[0] unused
  int max_code_len = 0;
  bool low_cluster_usage = false;
  int defector_groups = 0;
  int constructs = 0;
  LLHC llhc;

  explicit BlockEncoder(const EncoderConfig &c) : cfg(c) { block_capacity = sub_block_size * c.level; }

  // :165-210
  void RLE_1(const u8 *raw, i64 len) {
    rle_1_data.clear();
    rle_1_data.reserve((size_t)len + len / 4 + 8);
    for (int i = 0; i < 256; i++) in_use[i] = false;
    u8 b_prev = 0;
    int run = 0;
    auto store = [&](u8 x) { rle_1_data.push_back(x); in_use[x] = true; };
    auto store_run = [&]() {
      for (int count = 1; count <= std::min(4, run); count++) store(b_prev);
      if (run >= 4) store((u8)(run - 4));
      run = 1;
    };
    bool start = true;
    crc_init(block_crc);
    for (i64 k = 0; k < len; k++) {
      u8 b = raw[k];
      crc_update(block_crc, b);
      if (start || b != b_prev) { store_run(); start = false; }
      else if (run == 259) store_run();
      else run++;
      b_prev = b;
    }
    store_run();
  }

  // :219-296
  void BWT() {
    i32 n = (i32)rle_1_data.size();
    bwt_data.assign((size_t)n, 0);
    if (cfg.bwt_mode == 1) bwt_faithful(rle_1_data.data(), n, bwt_data.data(), bwt_index);
    else bwt_fast(rle_1_data.data(), n, bwt_data.data(), bwt_index);
  }

  // :318-413.  idx_out (may be null): the MTF index of every position of bwt_data (the search result of :384-392).
  void MTF_and_RLE_2(u8 *idx_out = nullptr) {
    u8 unseq_to_seq[256];
    normal_symbols_in_use = 0;                                           // :320-328
    for (int i = 0; i < 256; i++)
      if (in_use[i]) { unseq_to_seq[i] = (u8)normal_symbols_in_use; normal_symbols_in_use++; }
    last_symbol_in_use = normal_symbols_in_use + 3 - 1 - 1;              // :330
    EOB = last_symbol_in_use;                                            // :335
    mtf_data.clear();
    mtf_data.reserve(bwt_data.size() + 2);
    i64 run = 0;
    auto store = [&](int a) { mtf_data.push_back((u16)a); };
    auto store_run = [&]() {                                             // :348-363
      if (run > 0) {
        u32 rc = (u32)(run + 1);
        for (;;) {
          store((int)(rc & 1));
          rc >>= 1;
          if (rc < 2) break;
        }
        run = 0;
      }
    };
    u8 mtf_symbol[256];
    for (int i = 0; i < 256; i++) mtf_symbol[i] = (u8)i;
    for (size_t k = 0; k < bwt_data.size(); k++) {                       // :378-407
      u8 bt_seq = unseq_to_seq[bwt_data[k]];
      int idx = 0;
      for (int search = 0; search < 256; search++)
        if (mtf_symbol[search] == bt_seq) { idx = search; break; }
      if (idx_out) idx_out[k] = (u8)idx;
      for (int i = idx; i >= 1; i--) mtf_symbol[i] = mtf_symbol[i - 1];
      mtf_symbol[0] = bt_seq;
      if (idx == 0) run++;
      else { store_run(); store(1 + idx); }
    }
    store_run();                                                         // :409
    store(EOB);                                                          // :410
    mtf_last = (i32)mtf_data.size();
  }

  // :439-462
  void Avoid_Zeros(u32 *freq, int n) {
    int zeroes = 0;
    for (int i = 0; i < n; i++) if (freq[i] == 0) zeroes++;
    if (zeroes == 0) return;
    if (zeroes <= 100) { for (int i = 0; i < n; i++) freq[i] = std::max<u32>(1, freq[i]); }
    else { for (int i = 0; i < n; i++) freq[i] = (freq[i] == 0 ? 1 : freq[i] * 2); }
  }

  // :495-513
  void Define_Descriptor(u32 *freq, int des) {
    int n = last_symbol_in_use + 1;
    Avoid_Zeros(freq, n);
    llhc.run(freq, n, max_code_len, descr_len[des]);
    prepare_codes(descr_len[des], descr_code[des], n, max_code_len);
  }

  // :551-633
  void Initial_Clustering_Ranking_Method(int sample_width) {
    struct Pair { i32 key; i32 index; };
    std::vector<Pair> ranking((size_t)selector_count + 2);               // 1-based
    int pos_countdown = group_size;
    i32 sel_idx = 1;
    i32 key = 0;
    const int last_symbol_sampled = std::min(EOB - 1, run_a + sample_width - 1);   // :593
    for (i32 mtf_idx = 1; mtf_idx <= mtf_last; mtf_idx++) {              // :598-610
      int symbol = mtf_data[mtf_idx - 1];
      if (symbol >= run_a && symbol <= last_symbol_sampled) key++;
      pos_countdown--;
      if (pos_countdown == 0) {
        ranking[sel_idx] = Pair{key, sel_idx};
        pos_countdown = group_size;
        sel_idx++;
        key = 0;
      }
    }
    if (pos_countdown < group_size) ranking[sel_idx] = Pair{key, sel_idx};   // :611-614
    gnat_constrained_array_sort(ranking.data(), (i64)selector_count,     // :619
                                [](const Pair &l, const Pair &r) { return l.key < r.key; });
    static const int attr2[] = {2, 1}, attr3[] = {3, 1, 2}, attr4[] = {4, 2, 1, 3},
                     attr5[] = {5, 3, 1, 2, 4}, attr6[] = {6, 4, 2, 1, 3, 5};       // :625-631
    const int *attr = nullptr;
    switch (entropy_coder_count) {
      case 2: attr = attr2; break; case 3: attr = attr3; break; case 4: attr = attr4; break;
      case 5: attr = attr5; break; default: attr = attr6; break;
    }
    i64 na = entropy_coder_count, ns = selector_count;                   // :572-588
    i64 low = 1;
    for (i64 a32 = 1; a32 <= na; a32++) {
      i64 high = a32 * ns / na;
      for (i64 i = low; i <= high; i++) selector[ranking[i].index] = (u8)attr[a32 - 1];
      low = 1 + high;
    }
  }

  // :635-657
  void Define_Descriptors() {
    int n = last_symbol_in_use + 1;
    static thread_local std::vector<u32> freq_cluster;
    freq_cluster.assign((size_t)7 * 258, 0);
    int pos_countdown = group_size;
    i32 selector_idx = 1;
    int cluster = selector[1];
    for (i32 mtf_idx = 1; mtf_idx <= mtf_last; mtf_idx++) {
      int symbol = mtf_data[mtf_idx - 1];
      freq_cluster[cluster * 258 + symbol]++;
      pos_countdown--;
      if (pos_countdown == 0 && mtf_idx < mtf_last) {
        pos_countdown = group_size;
        selector_idx++;
        cluster = selector[selector_idx];
      }
    }
    (void)n;
    for (int cl = 1; cl <= entropy_coder_count; cl++) Define_Descriptor(&freq_cluster[cl * 258], cl);
  }

  // :661-753
  void Simulate_Entropy_Coding_Variants_and_Reclassify() {
    int pos_countdown = group_size;
    i32 selector_idx = 1;
    int cluster = selector[1];
    u32 bit_count[7] = {0, 0, 0, 0, 0, 0, 0};
    int mtf_cluster_value[7];
    int mtf_cluster_index = 1;
    auto optimize_group = [&]() {                                        // :672-718
      u32 min_bits = 0x7FFFFFFFu;
      int best = cluster;
      for (int cl = 1; cl <= entropy_coder_count; cl++) {
        u32 cost = bit_count[cl];
        for (int search = 1; search <= entropy_coder_count; search++)
          if (mtf_cluster_value[search] == cl) { mtf_cluster_index = search; break; }
        cost += (u32)mtf_cluster_index;
        if (cost < min_bits) { min_bits = cost; best = cl; }
      }
      if (best != cluster) { selector[selector_idx] = (u8)best; defector_groups++; }
      for (int search = 1; search <= entropy_coder_count; search++)
        if (mtf_cluster_value[search] == selector[selector_idx]) { mtf_cluster_index = search; break; }
      for (int j = mtf_cluster_index; j >= 2; j--) mtf_cluster_value[j] = mtf_cluster_value[j - 1];
      mtf_cluster_value[1] = selector[selector_idx];
    };
    for (int w = 1; w <= entropy_coder_count; w++) mtf_cluster_value[w] = w;
    defector_groups = 0;
    pos_countdown = group_size;
    for (i32 mtf_idx = 1; mtf_idx <= mtf_last; mtf_idx++) {              // :731-748
      int symbol = mtf_data[mtf_idx - 1];
      for (int cl = 1; cl <= entropy_coder_count; cl++) bit_count[cl] += descr_len[cl][symbol];
      pos_countdown--;
      if (pos_countdown == 0) {
        optimize_group();
        pos_countdown = group_size;
        if (mtf_idx < mtf_last) {
          for (int cl = 1; cl <= 6; cl++) bit_count[cl] = 0;
          selector_idx++;
          cluster = selector[selector_idx];
        }
      }
    }
    if (pos_countdown < group_size) optimize_group();                    // :749-752
  }

  // :757-778
  void Cluster_Statistics() {
    i32 stat_cluster[7] = {0, 0, 0, 0, 0, 0, 0};
    const i32 uniform_usage = selector_count / (i32)entropy_coder_count;
    low_cluster_usage = false;
    for (i32 i = 1; i <= selector_count; i++) stat_cluster[selector[i]]++;
    for (int c = 1; c <= entropy_coder_count; c++)
      if (stat_cluster[c] < uniform_usage / 2) low_cluster_usage = true;
  }

  // :780-809
  void Construct(int sample_width) {
    constructs++;
    Initial_Clustering_Ranking_Method(sample_width);
    for (int iteration = 1; iteration <= 10; iteration++) {
      Cluster_Statistics();
      Define_Descriptors();
      Simulate_Entropy_Coding_Variants_and_Reclassify();
      if (defector_groups == 0) break;
    }
    if (defector_groups > 0) Define_Descriptors();
    Cluster_Statistics();
  }

  // :811-887
  u32 Compute_Total_Entropy_Cost() {
    // selectors :815-837
    u32 sel_bits = 0;
    {
      int v[7]; int idx = 1;
      for (int w = 1; w <= entropy_coder_count; w++) v[w] = w;
      for (i32 i = 1; i <= selector_count; i++) {
        for (int search = 1; search <= entropy_coder_count; search++)
          if (v[search] == selector[i]) { idx = search; break; }
        for (int j = idx; j >= 2; j--) v[j] = v[j - 1];
        v[1] = selector[i];
        sel_bits += (u32)idx;
      }
    }
    // bit lengths :839-865
    u32 len_bits = 0;
    for (int coder = 1; coder <= entropy_coder_count; coder++) {
      u32 cur = descr_len[coder][0];
      len_bits += 5;
      for (int i = 0; i <= last_symbol_in_use; i++) {
        u32 nw = descr_len[coder][i];
        for (;;) {
          if (cur == nw) { len_bits += 1; break; }
          len_bits += 2;
          if (cur < nw) cur++; else cur--;
        }
      }
    }
    // data :867-881
    u32 bits = 0;
    int pos_countdown = group_size;
    i32 selector_idx = 1;
    int cluster = selector[1];
    for (i32 mtf_idx = 1; mtf_idx <= mtf_last; mtf_idx++) {
      bits += descr_len[cluster][mtf_data[mtf_idx - 1]];
      pos_countdown--;
      if (pos_countdown == 0 && mtf_idx < mtf_last) {
        pos_countdown = group_size;
        selector_idx++;
        cluster = selector[selector_idx];
      }
    }
    return bits + sel_bits + len_bits;
  }

  int best_ec_count = 0, best_max_code_len = 0, best_sample_width = 0;
  u32 best_cost = 0x7FFFFFFFu;

  // :541-962
  void Multiple_Entropy_Coders() {
    std::vector<int> max_code_len_choices, coder_choices, sample_width_choices;   // :901-921
    if (cfg.level == 9) {
      max_code_len_choices = {15, 17};
      if (mtf_last <= 5000) coder_choices = {2, 3, 6};
      else if (mtf_last <= 10000) coder_choices = {3, 4, 6};
      else coder_choices = {3, 4, 5, 6};
      sample_width_choices = {3, 4};
    } else {
      max_code_len_choices = {16};
      coder_choices = {4, 6};
      sample_width_choices = {4};
    }
    best_cost = 0x7FFFFFFFu;
    low_cluster_usage = false;                                           // :755
    for (int max_code_len_test : max_code_len_choices) {                 // :930-952
      max_code_len = max_code_len_test;
      for (int sample_width_test : sample_width_choices) {
        for (int ec_test = max_entropy_coders; ec_test >= min_entropy_coders; ec_test--) {
          bool in_choices = std::find(coder_choices.begin(), coder_choices.end(), ec_test) != coder_choices.end();
          if (low_cluster_usage || in_choices) {
            entropy_coder_count = ec_test;
            Construct(sample_width_test);
            u32 cost = Compute_Total_Entropy_Cost();
            if (cost < best_cost) {
              best_cost = cost;
              best_ec_count = ec_test;
              best_max_code_len = max_code_len;
              best_sample_width = sample_width_test;
            }
          }
        }
      }
    }
    max_code_len = best_max_code_len;                                    // :954-961
    entropy_coder_count = best_ec_count;
    Construct(best_sample_width);
  }

  // :433-978
  void Entropy_Calculations() {
    selector_count = 1 + (mtf_last - 1) / group_size;                    // :968
    selector.assign((size_t)selector_count + 2, 0);
    Multiple_Entropy_Coders();
  }

  // :984-994
  void Put_Block_Header(BitBuffer &out, u32 &combined_crc) {
    out.put_string("1AY&SY", 6);                                         // bzip2.ads:122
    block_crc = crc_final(block_crc);
    out.put_bits(block_crc, 32);
    combined_crc = ((combined_crc << 1) | (combined_crc >> 31)) ^ block_crc;   // :990
    out.put_bits(0, 1);
    out.put_bits(bwt_index, 24);
  }

  // :996-1086
  void Put_Block_Trees_Descriptors(BitBuffer &out) {
    bool in_use_16[16];                                                  // :998-1021
    for (int i = 0; i < 16; i++) {
      in_use_16[i] = false;
      for (int j = 0; j < 16; j++) if (in_use[i * 16 + j]) in_use_16[i] = true;
    }
    for (int i = 0; i < 16; i++) out.put_bool(in_use_16[i]);
    for (int i = 0; i < 16; i++)
      if (in_use_16[i]) for (int j = 0; j < 16; j++) out.put_bool(in_use[i * 16 + j]);
    out.put_bits((u32)entropy_coder_count, 3);                           // :1083
    out.put_bits((u32)selector_count, 15);                               // :1027
    {
      int v[7]; int idx = 1;
      for (int w = 1; w <= entropy_coder_count; w++) v[w] = w;
      for (i32 i = 1; i <= selector_count; i++) {                        // :1032-1050
        for (int search = 1; search <= entropy_coder_count; search++)
          if (v[search] == selector[i]) { idx = search; break; }
        for (int j = idx; j >= 2; j--) v[j] = v[j - 1];
        v[1] = selector[i];
        for (int bar = 1; bar <= idx - 1; bar++) out.put_bits(1, 1);
        out.put_bits(0, 1);
      }
    }
    for (int coder = 1; coder <= entropy_coder_count; coder++) {         // :1053-1079
      u32 cur = descr_len[coder][0];
      out.put_bits(cur, 5);
      for (int i = 0; i <= last_symbol_in_use; i++) {
        u32 nw = descr_len[coder][i];
        for (;;) {
          if (cur == nw) { out.put_bits(0, 1); break; }
          out.put_bits(1, 1);
          if (cur < nw) { cur++; out.put_bits(0, 1); }
          else { cur--; out.put_bits(1, 1); }
        }
      }
    }
  }

  // :1088-1112
  void Entropy_Output(BitBuffer &out) {
    int pos_countdown = group_size;
    i32 selector_idx = 1;
    int cluster = selector[1];
    for (i32 mtf_idx = 1; mtf_idx <= mtf_last; mtf_idx++) {
      int symbol = mtf_data[mtf_idx - 1];
      out.put_bits(descr_code[cluster][symbol], (int)descr_len[cluster][symbol]);
      pos_countdown--;
      if (pos_countdown == 0 && mtf_idx < mtf_last) {
        pos_countdown = group_size;
        selector_idx++;
        cluster = selector[selector_idx];
      }
    }
  }

  // :1114-1126
  void Encode_Block(const u8 *raw, i64 len, BitBuffer &out, u32 &combined_crc, BlockTaps *taps) {
    u64 bits_before = out.total_bits();
    constructs = 0;
    RLE_1(raw, len);
    BWT();
    MTF_and_RLE_2();
    Entropy_Calculations();
    Put_Block_Header(out, combined_crc);
    Put_Block_Trees_Descriptors(out);
    Entropy_Output(out);
    if (taps) {
      taps->rle1 = rle_1_data;
      taps->bwt = bwt_data;
      taps->origin = bwt_index;
      taps->mtf = mtf_data;
      taps->crc = block_crc;
      taps->eob = (u32)EOB;
      taps->n_used = (u32)normal_symbols_in_use;
      taps->ec_count = entropy_coder_count;
      taps->max_len = max_code_len;
      taps->sample_width = best_sample_width;
      taps->best_cost = best_cost;
      taps->selector.assign(selector.begin() + 1, selector.begin() + 1 + selector_count);
      memset(taps->lens, 0, sizeof(taps->lens));
      for (int c = 1; c <= entropy_coder_count; c++)
        for (int s = 0; s <= last_symbol_in_use; s++) taps->lens[c - 1][s] = descr_len[c][s];
      taps->bits = out.total_bits() - bits_before;
      taps->constructs = constructs;
    }
  }
};

// ---------------------------------------------------------------------------
// Stream level.  bzip2-encoding.adb:1136-1431
// ---------------------------------------------------------------------------
struct ChunkTrace {
  u64 start; u32 len; u32 dyn_capacity;
  int winner;                    // 0 single, 1 parts_4, 2 segmented_1, 3 segmented_2
  u64 bytes[4];                  // destination_index per tactic
  u64 bits[4];                   // bits appended per tactic (excluding incoming partial byte)
  u32 n_seg[2];
};

struct StreamEncoder {
  EncoderConfig cfg;
  const u8 *in; u64 n; u64 pos = 0;
  i64 stream_rest;
  u32 combined_crc = 0;
  std::vector<u8> &out;
  std::vector<ChunkTrace> *trace;
  i32 block_capacity;

  StreamEncoder(EncoderConfig c, const u8 *in_, u64 n_, i64 size_hint, std::vector<u8> &out_, std::vector<ChunkTrace> *tr)
      : cfg(c), in(in_), n(n_), stream_rest(size_hint), out(out_), trace(tr) {
    block_capacity = sub_block_size * c.level;
  }
  bool More_Bytes() const { return pos < n; }

  // :1160-1208 — returns raw length of the chunk starting at `pos`
  u32 Data_Acquisition(i32 dyn_block_capacity) {
    i64 rle_1_block_size = 0;
    u8 b_prev = 0;
    int run = 0;
    bool start = true;
    i64 raw_buf_index = 0;
    const i64 raw_buf_last = 10 * (i64)dyn_block_capacity;                // :1156-1157
    auto simulate_store_run = [&]() {                                    // :1171-1179
      rle_1_block_size += std::min(4, run);
      if (run >= 4) rle_1_block_size += 1;
      run = 1;
    };
    while (More_Bytes() && rle_1_block_size + 5 < dyn_block_capacity && raw_buf_index < raw_buf_last) {
      u8 b = in[pos++];
      raw_buf_index++;
      if (stream_rest != -1) stream_rest--;                              // :1192-1194
      if (start || b != b_prev) { simulate_store_run(); start = false; }
      else if (run == 259) simulate_store_run();
      else run++;
      b_prev = b;
    }
    simulate_store_run();
    return (u32)raw_buf_index;
  }

  // The four candidate encodings of one chunk (:1223-1299), each continuing a clone of the running bit
  // buffer (buffer, bit_index) and of the combined CRC.
  void Encode_Variants(const u8 *raw, u32 len, u8 in_buffer, int in_bit_index, u32 in_crc,
                       BitBuffer variant[4], u32 crc_variant[4], u32 n_seg[2]) {
      for (int t = 0; t < 4; t++) {
        variant[t].buffer = in_buffer; variant[t].bit_index = in_bit_index;               // :1223
        variant[t].attach_new();                                                          // :1309-1311
        crc_variant[t] = in_crc;                                                          // :1224
      }
      for (int tactic = 0; tactic < 2; tactic++) {                       // :1238-1254
        i64 slices = tactic == 0 ? 1 : 4;
        i64 size = (i64)len / slices;
        i64 stop = 0, startk;
        BlockEncoder be(cfg);
        for (i64 count = 1; count <= slices; count++) {
          startk = stop + 1;
          if (count == slices) stop = len; else stop = count * size;
          be.Encode_Block(raw + (startk - 1), stop - startk + 1, variant[tactic], crc_variant[tactic], nullptr);
        }
      }
      for (int tactic = 2; tactic < 4; tactic++) {                       // :1262-1299
        std::vector<i32> seg;
        if (tactic == 2) segment_by_entropy(raw, (i32)len, 0.6f, 4000, 16000, seg);
        else segment_by_entropy(raw, (i32)len, 0.4f, 8000, 16000, seg);
        n_seg[tactic - 2] = (u32)seg.size();
        BlockEncoder be(cfg);
        if (seg.empty()) {
          be.Encode_Block(raw, 0, variant[tactic], crc_variant[tactic], nullptr);
        } else {
          i64 index_start = 1;
          for (i32 s : seg) {
            be.Encode_Block(raw + (index_start - 1), s - index_start + 1, variant[tactic], crc_variant[tactic], nullptr);
            index_start = (i64)s + 1;
          }
        }
      }
  }

  // :1144-1382
  void Read_and_Split_Block(BitBuffer &main_buf, i32 dyn_block_capacity) {
    u64 start = pos;
    u32 len = Data_Acquisition(dyn_block_capacity);
    const u8 *raw = in + start;
    ChunkTrace ct{};
    ct.start = start; ct.len = len; ct.dyn_capacity = (u32)dyn_block_capacity;
    if (cfg.level != 9) {                                                // :1364-1370
      main_buf.attach_new();
      BlockEncoder be(cfg);
      u64 b0 = main_buf.total_bits();
      be.Encode_Block(raw, len, main_buf, combined_crc, nullptr);
      ct.winner = 0; ct.bytes[0] = main_buf.dest.size(); ct.bits[0] = main_buf.total_bits() - b0;
      out.insert(out.end(), main_buf.dest.begin(), main_buf.dest.end());
      main_buf.dest.clear();
    } else {
      // Block_Split_Parallel :1214-1359 (the four tasks run one after another here;
      // they only touch private state, so the result is the same)
      BitBuffer variant[4];
      u32 crc_variant[4];
      u64 bits0 = (u64)(7 - main_buf.bit_index);
      Encode_Variants(raw, len, main_buf.buffer, main_buf.bit_index, combined_crc, variant, crc_variant, ct.n_seg);
      int best = 0;                                                      // :1305, 1319-1325
      for (int t = 0; t < 4; t++)
        if (variant[t].dest.size() < variant[best].dest.size()) best = t;
      for (int t = 0; t < 4; t++) { ct.bytes[t] = variant[t].dest.size(); ct.bits[t] = variant[t].total_bits() - bits0; }
      ct.winner = best;
      out.insert(out.end(), variant[best].dest.begin(), variant[best].dest.end());   // :1335-1337
      main_buf.bit_index = variant[best].bit_index;                      // :1339-1343
      main_buf.buffer = variant[best].buffer;
      main_buf.dest.clear();
      combined_crc = crc_variant[best];                                  // :1345
    }
    if (trace) trace->push_back(ct);
  }

  // The chunk loop of Encode (:1413-1429) with the cutting only: (start, len, capacity) of every chunk.
  void Cut_Only(std::vector<ChunkTrace> &chunks, u64 stop = ~0ull, bool at_least_one = true) {
    volatile float fcap = (float)block_capacity;
    volatile float flo = fcap * 1.05f;
    volatile float fhi = fcap * 1.30f;
    for (;;) {
      if (pos >= stop && !(at_least_one && chunks.empty())) break;      // (a shard ends with the first chunk of the next one)
      volatile float frest = (float)stream_rest;
      const i32 cap = (frest >= flo && frest <= fhi) ? (i32)stream_rest / 2 : block_capacity;
      ChunkTrace ct{};
      ct.start = pos; ct.dyn_capacity = (u32)cap;
      ct.len = Data_Acquisition(cap);
      chunks.push_back(ct);
      if (!More_Bytes()) break;
    }
  }

  // :1413-1431
  void Encode() {
    const char magic[4] = {'B', 'Z', 'h', (char)('0' + cfg.level)};      // :1384-1391
    for (int i = 0; i < 4; i++) out.push_back((u8)magic[i]);
    BitBuffer main_bit_buffer;
    // Float (block_capacity) * (1.0 + small_block_prop_min/max), single precision (:1416-1418)
    volatile float fcap = (float)block_capacity;
    volatile float flo = fcap * 1.05f;
    volatile float fhi = fcap * 1.30f;
    for (;;) {
      volatile float frest = (float)stream_rest;
      if (frest >= flo && frest <= fhi)
        Read_and_Split_Block(main_bit_buffer, (i32)stream_rest / 2);     // :1424
      else
        Read_and_Split_Block(main_bit_buffer, block_capacity);           // :1426
      if (!More_Bytes()) break;                                          // :1428
    }
    // Write_Stream_Footer :1395-1407
    main_bit_buffer.attach_new();
    static const u8 footer[6] = {0x17, 0x72, 0x45, 0x38, 0x50, 0x90};    // bzip2.ads:118-119
    for (int i = 0; i < 6; i++) main_bit_buffer.put_bits(footer[i], 8);
    main_bit_buffer.put_bits(combined_crc, 32);
    if (main_bit_buffer.bit_index < 7) main_bit_buffer.flush();
    out.insert(out.end(), main_bit_buffer.dest.begin(), main_bit_buffer.dest.end());
  }
};

}  // namespace

// ===========================================================================
// C API (ctypes-friendly).  All functions return 0 on success.
// ===========================================================================
extern "C" {

struct orc_block_info {
  u32 n_rle, origin, crc, n_mtf, eob, n_used, n_sel, ec_count, max_len, sample_width, cost, constructs;
  u64 bits;
};

struct orc_chunk_trace {
  u64 start;
  u32 len, dyn_capacity;
  i32 winner;
  u32 n_seg1, n_seg2, pad;
  u64 bytes[4];
  u64 bits[4];
};

int orc_version() { return 63; }

// Whole stream: what `Encode (option, size_hint)` writes through Write_Byte.
int orc_encode_stream(const u8 *in, u64 n, int level, i64 size_hint, int bwt_mode,
                      u8 *out, u64 out_cap, u64 *out_len,
                      orc_chunk_trace *trace, u64 trace_cap, u64 *n_trace) {
  crc_make_table();
  if (level != 1 && level != 4 && level != 9) return 1;
  std::vector<u8> o;
  o.reserve((size_t)(n + n / 50 + 4096));
  std::vector<ChunkTrace> tr;
  EncoderConfig cfg{level, bwt_mode};
  StreamEncoder se(cfg, in, n, size_hint, o, &tr);
  se.Encode();
  if (out_len) *out_len = o.size();
  if (n_trace) *n_trace = tr.size();
  if (trace) {
    for (size_t i = 0; i < tr.size() && i < trace_cap; i++) {
      orc_chunk_trace &t = trace[i];
      t.start = tr[i].start; t.len = tr[i].len; t.dyn_capacity = tr[i].dyn_capacity; t.winner = tr[i].winner;
      t.n_seg1 = tr[i].n_seg[0]; t.n_seg2 = tr[i].n_seg[1]; t.pad = 0;
      for (int k = 0; k < 4; k++) { t.bytes[k] = tr[i].bytes[k]; t.bits[k] = tr[i].bits[k]; }
    }
  }
  if (o.size() > out_cap) return 2;
  if (out) memcpy(out, o.data(), o.size());
  return 0;
}

// The same stream with the chunks encoded on `threads` host threads (golden scripts and CPU baselines
// over large inputs).  A candidate's bits do not depend on the incoming bit offset — only the winner test
// does (it compares flushed bytes, :1319-1325) — and the combined CRC is folded by c -> rotl (c, 1) xor
// block_crc (:990), which is affine: every chunk is encoded from an empty bit buffer and a zero CRC, then
// one serial pass picks the winners in order, appends their bits at the running offset and composes the
// folds.  tests/test_oracle.py checks it against orc_encode_stream.
int orc_encode_stream_mt(const u8 *in, u64 n, int level, i64 size_hint, int bwt_mode, int threads,
                         u8 *out, u64 out_cap, u64 *out_len,
                         orc_chunk_trace *trace, u64 trace_cap, u64 *n_trace) {
  crc_make_table();
  if (level != 1 && level != 4 && level != 9) return 1;
  EncoderConfig cfg{level, bwt_mode};
  std::vector<u8> dummy;
  std::vector<ChunkTrace> chunks;
  {
    StreamEncoder se(cfg, in, n, size_hint, dummy, nullptr);
    se.Cut_Only(chunks);
  }
  const size_t nc = chunks.size();
  const int nt = level == 9 ? 4 : 1;
  struct Cand { std::vector<u8> bytes; u64 bits; u32 fold; u32 blocks; };
  const size_t window = 256;                 // chunks encoded in parallel before the serial pass takes them (bounds memory)
  std::vector<Cand> cand(window * 4);
  size_t w0 = 0;
  std::atomic<size_t> next{0};
  auto work = [&]() {
    for (;;) {
      const size_t c = next.fetch_add(1);
      if (c >= std::min(nc, w0 + window)) break;
      StreamEncoder se(cfg, in, n, size_hint, dummy, nullptr);
      BitBuffer variant[4];
      u32 crcv[4] = {0, 0, 0, 0};
      const u8 *raw = in + chunks[c].start;
      if (level == 9) {
        se.Encode_Variants(raw, chunks[c].len, 0, 7, 0, variant, crcv, chunks[c].n_seg);
      } else {
        variant[0].attach_new();
        BlockEncoder be(cfg);
        be.Encode_Block(raw, chunks[c].len, variant[0], crcv[0], nullptr);
      }
      for (int t = 0; t < nt; t++) {
        Cand &cd = cand[(c - w0) * 4 + t];
        cd.bits = variant[t].total_bits();
        cd.bytes = std::move(variant[t].dest);
        if (variant[t].bit_index != 7) cd.bytes.push_back(variant[t].buffer);
        cd.fold = crcv[t];
        cd.blocks = t == 0 ? 1u : t == 1 ? 4u : std::max<u32>(1u, chunks[c].n_seg[t - 2]);
      }
    }
  };
  std::vector<u8> o;
  o.reserve((size_t)(n + n / 50 + 4096));
  const char magic[4] = {'B', 'Z', 'h', (char)('0' + level)};
  for (int i = 0; i < 4; i++) o.push_back((u8)magic[i]);
  u64 total_bits = 32;                       // bits written so far; o holds ceil (total_bits / 8) bytes
  u32 combined = 0;
  auto append = [&](const std::vector<u8> &src, u64 nbits) {
    const u32 sh = (u32)(total_bits & 7);
    const u64 nbytes = (nbits + 7) >> 3;
    if (sh == 0) o.insert(o.end(), src.begin(), src.begin() + nbytes);
    else {
      for (u64 i = 0; i < nbytes; i++) {
        o.back() |= (u8)(src[i] >> sh);
        o.push_back((u8)(src[i] << (8 - sh)));
      }
    }
    total_bits += nbits;
    o.resize((size_t)((total_bits + 7) >> 3));
  };
  for (w0 = 0; w0 < nc; w0 += window) {
    next = w0;
    {
      std::vector<std::thread> th;
      for (int i = 0; i < std::max(1, threads); i++) th.emplace_back(work);
      for (auto &t : th) t.join();
    }
    for (size_t c = w0; c < std::min(nc, w0 + window); c++) {
      ChunkTrace &ct = chunks[c];
      const u64 in_bits = total_bits & 7;
      int best = 0;
      for (int t = 0; t < nt; t++) { ct.bits[t] = cand[(c - w0) * 4 + t].bits; ct.bytes[t] = (in_bits + ct.bits[t]) >> 3; }
      for (int t = 0; t < nt; t++) if (ct.bytes[t] < ct.bytes[best]) best = t;
      ct.winner = best;
      Cand &w = cand[(c - w0) * 4 + best];
      append(w.bytes, w.bits);
      const u32 k = w.blocks & 31u;
      combined = (k ? ((combined << k) | (combined >> (32 - k))) : combined) ^ w.fold;
      for (int t = 0; t < nt; t++) std::vector<u8>().swap(cand[(c - w0) * 4 + t].bytes);
    }
  }
  {
    static const u8 footer[6] = {0x17, 0x72, 0x45, 0x38, 0x50, 0x90};
    std::vector<u8> f(footer, footer + 6);
    for (int k = 3; k >= 0; k--) f.push_back((u8)(combined >> (8 * k)));
    append(f, 80);
  }
  if (out_len) *out_len = o.size();
  if (n_trace) *n_trace = nc;
  if (trace) {
    for (size_t i = 0; i < nc && i < trace_cap; i++) {
      orc_chunk_trace &t = trace[i];
      t.start = chunks[i].start; t.len = chunks[i].len; t.dyn_capacity = chunks[i].dyn_capacity; t.winner = chunks[i].winner;
      t.n_seg1 = chunks[i].n_seg[0]; t.n_seg2 = chunks[i].n_seg[1]; t.pad = 0;
      for (int k = 0; k < 4; k++) { t.bytes[k] = chunks[i].bytes[k]; t.bits[k] = chunks[i].bits[k]; }
    }
  }
  if (o.size() > out_cap) return 2;
  if (out) memcpy(out, o.data(), o.size());
  return 0;
}

// ---- one shard of a stream (mirror of b2_shard_* in include/b2gpu.h, for the CPU tests of the protocol) ----
// `in_local` holds the stream bytes [base, base + n_local).  Chunks that start in [entry, own_end) are cut
// and encoded from an empty bit buffer; link = bits appended and CRC fold for each incoming bit offset mod 8.
struct orc_shard_link { u64 total_bits[8]; u32 crc_rot[8]; u32 crc_fold[8]; };
struct OrcShard {
  struct Cand { std::vector<u8> bytes; u64 bits; u32 fold; u32 blocks; };
  std::vector<ChunkTrace> chunks;
  std::vector<Cand> cand;
  int level, nt;
  bool first, last;
};
static inline u32 rotl32(u32 c, u32 k) { k &= 31u; return k ? ((c << k) | (c >> (32 - k))) : c; }

void *orc_shard_encode(const u8 *in_local, u64 base, u64 n_local, u64 stream_n, int level, i64 size_hint, int bwt_mode,
                       int threads, u64 entry, u64 own_end, u64 *handoff, orc_shard_link *link) {
  crc_make_table();
  EncoderConfig cfg{level, bwt_mode};
  std::vector<u8> dummy;
  OrcShard *S = new OrcShard();
  S->level = level; S->nt = level == 9 ? 4 : 1;
  S->first = base == 0 && entry == 0; S->last = own_end >= stream_n;
  const u8 *in = in_local - base;                    // indexed with stream offsets
  {
    StreamEncoder se(cfg, in, base + n_local, size_hint, dummy, nullptr);
    se.pos = entry;
    se.stream_rest = size_hint < 0 ? -1 : ((i64)entry <= size_hint ? size_hint - (i64)entry : -1);   // :1192-1194
    se.Cut_Only(S->chunks, S->last ? ~0ull : own_end, S->first && stream_n == 0);
    if (S->last && entry >= stream_n && !(S->first && stream_n == 0)) S->chunks.clear();
    *handoff = se.pos;
  }
  const size_t nc = S->chunks.size();
  S->cand.resize(nc * 4);
  std::atomic<size_t> next{0};
  auto work = [&]() {
    for (;;) {
      const size_t c = next.fetch_add(1);
      if (c >= nc) break;
      StreamEncoder se(cfg, in, base + n_local, size_hint, dummy, nullptr);
      BitBuffer variant[4];
      u32 crcv[4] = {0, 0, 0, 0};
      const u8 *raw = in + S->chunks[c].start;
      if (level == 9) se.Encode_Variants(raw, S->chunks[c].len, 0, 7, 0, variant, crcv, S->chunks[c].n_seg);
      else { variant[0].attach_new(); BlockEncoder be(cfg); be.Encode_Block(raw, S->chunks[c].len, variant[0], crcv[0], nullptr); }
      for (int t = 0; t < S->nt; t++) {
        OrcShard::Cand &cd = S->cand[c * 4 + t];
        cd.bits = variant[t].total_bits();
        cd.bytes = std::move(variant[t].dest);
        if (variant[t].bit_index != 7) cd.bytes.push_back(variant[t].buffer);
        cd.fold = crcv[t];
        cd.blocks = t == 0 ? 1u : t == 1 ? 4u : std::max<u32>(1u, S->chunks[c].n_seg[t - 2]);
      }
    }
  };
  {
    std::vector<std::thread> th;
    for (int i = 0; i < std::max(1, threads); i++) th.emplace_back(work);
    for (auto &t : th) t.join();
  }
  for (u32 p0 = 0; p0 < 8; p0++) {
    u64 total = 0; u32 rot = 0, fold = 0, ph = p0;
    for (size_t c = 0; c < nc; c++) {
      int best = 0;
      for (int t = 0; t < S->nt; t++) if (((ph + S->cand[c * 4 + t].bits) >> 3) < ((ph + S->cand[c * 4 + best].bits) >> 3)) best = t;
      const OrcShard::Cand &w = S->cand[c * 4 + best];
      total += w.bits; ph = (u32)((ph + w.bits) & 7);
      fold = rotl32(fold, w.blocks) ^ w.fold; rot = (rot + w.blocks) & 31u;
    }
    link->total_bits[p0] = total; link->crc_rot[p0] = rot; link->crc_fold[p0] = fold;
  }
  return S;
}

int orc_shard_finish(void *h, u64 bit_offset, u32 crc_in, u8 *out, u64 out_cap, u64 *byte_offset, u64 *out_len) {
  OrcShard *S = (OrcShard *)h;
  const u64 byte0 = S->first ? 0 : bit_offset >> 3;
  std::vector<u8> o;
  u64 total_bits = bit_offset - 8 * byte0;            // bits of the piece in place so far
  if (S->first) { const char magic[4] = {'B', 'Z', 'h', (char)('0' + S->level)}; for (int i = 0; i < 4; i++) o.push_back((u8)magic[i]); }
  else if (total_bits) o.push_back(0);
  auto append = [&](const std::vector<u8> &src, u64 nbits) {
    const u32 sh = (u32)(total_bits & 7);
    const u64 nbytes = (nbits + 7) >> 3;
    if (sh == 0) o.insert(o.end(), src.begin(), src.begin() + nbytes);
    else for (u64 i = 0; i < nbytes; i++) { o.back() |= (u8)(src[i] >> sh); o.push_back((u8)(src[i] << (8 - sh))); }
    total_bits += nbits;
    o.resize((size_t)((total_bits + 7) >> 3));
  };
  u32 crc = crc_in;
  for (size_t c = 0; c < S->chunks.size(); c++) {
    const u64 in_bits = total_bits & 7;
    int best = 0;
    for (int t = 0; t < S->nt; t++) if (((in_bits + S->cand[c * 4 + t].bits) >> 3) < ((in_bits + S->cand[c * 4 + best].bits) >> 3)) best = t;
    const OrcShard::Cand &w = S->cand[c * 4 + best];
    append(w.bytes, w.bits);
    crc = rotl32(crc, w.blocks) ^ w.fold;
  }
  if (S->last) {
    static const u8 footer[6] = {0x17, 0x72, 0x45, 0x38, 0x50, 0x90};
    std::vector<u8> f(footer, footer + 6);
    for (int k = 3; k >= 0; k--) f.push_back((u8)(crc >> (8 * k)));
    append(f, 80);
  }
  *byte_offset = byte0; *out_len = o.size();
  if (o.size() > out_cap) return 2;
  if (out && !o.empty()) memcpy(out, o.data(), o.size());
  return 0;
}

void orc_shard_free(void *h) { delete (OrcShard *)h; }

// One Encode_Block with every intermediate.  Buffers may be NULL.
// rle_out: >= len*5/4+8; bwt_out same; mtf_out: >= len*5/4+10 u16; sel_out >= 18002;
// lens_out: 6*258 bytes; bits_out: the block's bits starting at bit 0 of byte 0.
int orc_encode_block(const u8 *raw, u32 len, int level, int bwt_mode,
                     u8 *rle_out, u8 *bwt_out, u16 *mtf_out, u8 *sel_out, u8 *lens_out,
                     u8 *bits_out, u64 bits_cap_bytes, orc_block_info *info) {
  crc_make_table();
  EncoderConfig cfg{level, bwt_mode};
  BlockEncoder be(cfg);
  BitBuffer bb;
  u32 ccrc = 0;
  BlockTaps t;
  be.Encode_Block(raw, len, bb, ccrc, &t);
  if (bb.bit_index < 7) bb.flush();
  if (rle_out) memcpy(rle_out, t.rle1.data(), t.rle1.size());
  if (bwt_out) memcpy(bwt_out, t.bwt.data(), t.bwt.size());
  if (mtf_out) memcpy(mtf_out, t.mtf.data(), t.mtf.size() * 2);
  if (sel_out) memcpy(sel_out, t.selector.data(), t.selector.size());
  if (lens_out) for (int c = 0; c < 6; c++) for (int s = 0; s < 258; s++) lens_out[c * 258 + s] = (u8)t.lens[c][s];
  if (bits_out) { if (bb.dest.size() > bits_cap_bytes) return 2; memcpy(bits_out, bb.dest.data(), bb.dest.size()); }
  if (info) {
    info->n_rle = (u32)t.rle1.size(); info->origin = t.origin; info->crc = t.crc; info->n_mtf = (u32)t.mtf.size();
    info->eob = t.eob; info->n_used = t.n_used; info->n_sel = (u32)t.selector.size(); info->ec_count = (u32)t.ec_count;
    info->max_len = (u32)t.max_len; info->sample_width = (u32)t.sample_width; info->cost = t.best_cost;
    info->constructs = (u32)t.constructs; info->bits = t.bits;
  }
  return 0;
}

// MTF_and_RLE_2 of a given last column col[0..n) (in_use = the bytes of col): the symbols mtf_data(1..mtf_last) into
// mtf_out (>= n + 2 u16) and the MTF index of every position into idx_out (may be null).
int orc_mtf_rle2(const u8 *col, u32 n, u16 *mtf_out, u32 *n_mtf, u8 *idx_out) {
  EncoderConfig cfg{9, 0};
  BlockEncoder be(cfg);
  for (int i = 0; i < 256; i++) be.in_use[i] = false;
  for (u32 i = 0; i < n; i++) be.in_use[col[i]] = true;
  be.bwt_data.assign(col, col + n);
  be.MTF_and_RLE_2(idx_out);
  memcpy(mtf_out, be.mtf_data.data(), be.mtf_data.size() * 2);
  *n_mtf = (u32)be.mtf_last;
  return 0;
}

int orc_bwt(const u8 *d, u32 n, int mode, u8 *out, u32 *origin) {
  u32 o = 0;
  if (mode == 1) bwt_faithful(d, (i32)n, out, o); else bwt_fast(d, (i32)n, out, o);
  *origin = o;
  return 0;
}

int orc_segment(const u8 *raw, u32 len, int profile, u32 *cuts, u32 cap, u32 *n_cuts) {
  std::vector<i32> seg;
  if (profile == 0) segment_by_entropy(raw, (i32)len, 0.6f, 4000, 16000, seg);
  else segment_by_entropy(raw, (i32)len, 0.4f, 8000, 16000, seg);
  *n_cuts = (u32)seg.size();
  for (size_t i = 0; i < seg.size() && i < cap; i++) cuts[i] = (u32)seg[i];
  return seg.size() > cap ? 2 : 0;
}

// The running entropy sum of Segment_by_Entropy (window 16_000; both profiles share it): *init after the
// first window, series[k] after step k (reference i = 16_001 + k).  Empty when len <= 20_000: the loop
// of the reference does not run (data_segmentation.adb:58).  Returns 2 when cap is too small.
int orc_entropy_series(const u8 *raw, u32 len, double *init, double *series, u64 cap, u64 *n) {
  std::vector<i32> seg;
  std::vector<double> all;
  segment_by_entropy(raw, (i32)len, 0.6f, 4000, 16000, seg, &all);
  *init = all.empty() ? 0.0 : all[0];
  *n = all.empty() ? 0 : all.size() - 1;
  for (u64 k = 0; k < *n && k < cap; k++) series[k] = all[k + 1];
  return *n > cap ? 2 : 0;
}

int orc_llhc(const u32 *freq, int n, int max_bits, u32 *lens) {
  LLHC l;
  l.run(freq, n, max_bits, lens);
  return 0;
}

int orc_prepare_codes(const u32 *lens, int n, int max_bits, u32 *codes) {
  prepare_codes(lens, codes, n, max_bits);
  return 0;
}

// Ranking_Sort tie order: sorts (key,index) pairs by key only with the GNAT heap sort.
int orc_gnat_sort_pairs(i32 *keys, i32 *index, u32 n) {
  struct Pair { i32 key; i32 index; };
  std::vector<Pair> a((size_t)n + 2);
  for (u32 i = 0; i < n; i++) a[i + 1] = Pair{keys[i], index[i]};
  gnat_constrained_array_sort(a.data(), (i64)n, [](const Pair &l, const Pair &r) { return l.key < r.key; });
  for (u32 i = 0; i < n; i++) { keys[i] = a[i + 1].key; index[i] = a[i + 1].index; }
  return 0;
}

u32 orc_crc32(const u8 *d, u64 n) {
  crc_make_table();
  u32 c; crc_init(c);
  for (u64 i = 0; i < n; i++) crc_update(c, d[i]);
  return crc_final(c);
}

// -1 terminated list of the float32 balancing window for a level (A0), for tests.
void orc_balance_window(int level, i64 *lo, i64 *hi) {
  volatile float fcap = (float)(sub_block_size * level);
  volatile float flo = fcap * 1.05f, fhi = fcap * 1.30f;
  i64 l = -1, h = -1;
  for (i64 v = (i64)(sub_block_size * level); v <= (i64)(sub_block_size * level) * 2; v++) {
    volatile float f = (float)v;
    if (f >= flo && f <= fhi) { if (l < 0) l = v; h = v; }
  }
  *lo = l; *hi = h;
}

}  // extern "C"
