// ORACLE — TEST INFRASTRUCTURE ONLY (see the header of b2_oracle.cpp; same rules: only tests/,
// __graft_entry__.smoke() and bench.py's CPU legs may load this library).
//
// CPU restatement of the archive side of the path (SURVEY.md §8f rows 1-3): what
// Zip.Create.Create_Archive / Add_Stream / Finish leave in the output Zipstream when every entry is
// compressed with BZip2_1..3 and there is no password.  The flow is the reference's own: a seekable
// output stream, a local header written with incomplete information, the payload, a seek back to
// rewrite the header (zip-create.adb:194-297), then the central directory (:645-756).
// PARITY STATUS: parity unpinned, as for the encoder.  What pins this part: Python's `zipfile`
// (an independent reader) opens every archive written here, `testzip ()` passes and the entries
// read back equal the inputs; the CRC is compared with zlib's.
//
// Paths below are relative to /root/reference/zip_lib/.
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;
typedef int64_t i64;

extern "C" int orc_encode_stream(const u8 *in, u64 n, int level, i64 size_hint, int bwt_mode, u8 *out, u64 out_cap,
                                 u64 *out_len, void *trace, u64 trace_cap, u64 *n_trace);

namespace {

// ---- Zip.CRC_Crypto (zip-crc_crypto.adb:28-77) ----------------------------------------------------
u32 crc32_table[256];
bool table_empty = true;

void Prepare_table() {                                  // :30-46
  const u32 Seed = 0xEDB88320u;
  for (u32 i = 0; i < 256; i++) {
    u32 l = i;
    for (int bit = 0; bit <= 7; bit++) l = (l & 1) == 0 ? (l >> 1) : ((l >> 1) ^ Seed);
    crc32_table[i] = l;
  }
}
void Init(u32 &crc) {                                   // :63-70
  if (table_empty) { Prepare_table(); table_empty = false; }
  crc = 0xFFFFFFFFu;
}
void Update(u32 &crc, const u8 *buf, u64 n) {           // :48-59
  u32 local = crc;
  for (u64 i = 0; i < n; i++) local = crc32_table[0xFF & (local ^ buf[i])] ^ (local >> 8);
  crc = local;
}
u32 Final(u32 crc) { return ~crc; }                     // :72-75

// ---- a memory Zipstream with Index / Set_Index (1-based, zip_streams.ads) ---------------------------
struct MemStream {
  std::vector<u8> data;
  u64 index = 1;
  void Write(const u8 *p, u64 n) {
    if (index - 1 + n > data.size()) data.resize(index - 1 + n);
    if (n) memcpy(data.data() + index - 1, p, n);
    index += n;
  }
};

// ---- Zip.Headers (zip-headers.adb:54-70: Intel_bf) -------------------------------------------------
struct Buf {
  std::vector<u8> b;
  void bf16(u32 v) { for (int i = 0; i < 2; i++) { b.push_back((u8)(v & 255)); v /= 256; } }
  void bf32(u64 v) { for (int i = 0; i < 4; i++) { b.push_back((u8)(v & 255)); v /= 256; } }
  void bf64(u64 v) { for (int i = 0; i < 8; i++) { b.push_back((u8)(v & 255)); v /= 256; } }
  void PK(u8 c1, u8 c2) { b.push_back(0x50); b.push_back(0x4B); b.push_back(c1); b.push_back(c2); }   // :85-88
};

struct Local_File_Header {                              // zip-headers.ads:139-147
  u16 needed_extract_version = 0, bit_flag = 0, zip_type = 0;
  u32 file_timedate = 0;
  u32 crc_32 = 0;
  u64 compressed_size = 0, uncompressed_size = 0;
  u16 filename_length = 0, extra_field_length = 0;
};
struct Central_File_Header {                            // zip-headers.ads:222-238
  u16 made_by_version = 0;
  Local_File_Header short_info;
  u16 comment_length = 0, disk_number_start = 0, internal_attributes = 0;
  u32 external_attributes = 0;
  u64 local_header_offset = 0;
};
enum Extra_Field_Policy_Kind { from_header, force_empty, force_zip_64 };
const u32 local_header_extension_length = 28, local_header_extension_short_length = 20;

bool Needs_Local_Zip_64_Header_Extension(const Local_File_Header &h, u64 offset) {   // zip-headers.adb:194-207
  return h.compressed_size >= 0xFFFFFFFFull || h.uncompressed_size >= 0xFFFFFFFFull || offset >= 0xFFFFFFFFull;
}

void Write_Local(MemStream &s, const Local_File_Header &h, Extra_Field_Policy_Kind pol) {   // zip-headers.adb:243-277
  Buf lhb;
  lhb.PK(3, 4);
  lhb.bf16(h.needed_extract_version); lhb.bf16(h.bit_flag); lhb.bf16(h.zip_type);
  lhb.bf32(h.file_timedate);
  lhb.bf32(h.crc_32);
  if (pol == force_zip_64) { lhb.bf32(0xFFFFFFFFu); lhb.bf32(0xFFFFFFFFu); }
  else { lhb.bf32((u32)h.compressed_size); lhb.bf32((u32)h.uncompressed_size); }
  lhb.bf16(h.filename_length);
  u16 extra_length = 0;
  switch (pol) {
    case from_header: extra_length = h.extra_field_length; break;
    case force_empty: extra_length = 0; break;
    case force_zip_64: extra_length = (u16)local_header_extension_short_length; break;
  }
  lhb.bf16(extra_length);
  s.Write(lhb.b.data(), lhb.b.size());
}

struct Local_File_Header_Extension { u16 tag = 0, size = 0; u64 value_64[3] = {0, 0, 0}; };
void Write_Ext(MemStream &s, const Local_File_Header_Extension &h, bool is_short) {   // zip-headers.adb:336-355
  Buf lhb;
  lhb.bf16(h.tag); lhb.bf16(h.size);
  lhb.bf64(h.value_64[0]); lhb.bf64(h.value_64[1]); lhb.bf64(h.value_64[2]);
  s.Write(lhb.b.data(), is_short ? local_header_extension_short_length : local_header_extension_length);
}

void Write_Central(MemStream &s, const Central_File_Header &h) {   // zip-headers.adb:167-192
  Buf chb;
  chb.PK(1, 2);
  chb.bf16(h.made_by_version);
  chb.bf16(h.short_info.needed_extract_version); chb.bf16(h.short_info.bit_flag); chb.bf16(h.short_info.zip_type);
  chb.bf32(h.short_info.file_timedate);
  chb.bf32(h.short_info.crc_32);
  chb.bf32((u32)h.short_info.compressed_size); chb.bf32((u32)h.short_info.uncompressed_size);
  chb.bf16(h.short_info.filename_length); chb.bf16(h.short_info.extra_field_length);
  chb.bf16(h.comment_length); chb.bf16(h.disk_number_start); chb.bf16(h.internal_attributes);
  chb.bf32(h.external_attributes);
  chb.bf32((u32)h.local_header_offset);
  s.Write(chb.b.data(), chb.b.size());
}

struct Entry { Central_File_Header head; std::string name; };

struct Zip_Create_Info {
  MemStream stream;
  int level = 9;                                       // BZip2_1 / _2 / _3 <-> 1 / 4 / 9
  bool zip_64 = false;
  std::vector<Entry> contains;
};

const u64 four_GiB = 1ull << 32, max_size = 0x1FFFFFFFFFFFFFFFull;   // zip-create.adb:157, zip-create.ads:224

int Check_Size(Zip_Create_Info &info, u64 value) {      // zip-create.adb:161-179
  const u64 margin = 22 + 56 + 20 + 65536 + 10;
  if (!info.zip_64 && value >= four_GiB - margin) {
    info.zip_64 = true;
    if (value >= max_size - margin) return 1;           // Zip_Capacity_Exceeded
  }
  return 0;
}

// Where Compress_Data takes the BZip2 stream of an entry from: encoded here (stream == nullptr), or given by the
// caller (orc_zip_create_given), e.g. a stream the oracle cannot afford to encode in a test.
struct Stream_Source { const u8 *stream = nullptr; u64 stream_len = 0; };

// Zip.Compress.Compress_Data for a BZip2 single method (zip-compress.adb:60-237), input size known.
void Compress_Data(Zip_Create_Info &info, const u8 *in, u64 input_size, const Stream_Source &src, u32 &CRC, u64 &output_size,
                   u16 &zip_type) {
  const u64 idx_out = info.stream.index;                // :84
  Init(CRC);                                            // :150
  // BZip2_E (zip-compress-bzip2_e.adb:110-135): the CRC is updated by Read_Byte for every byte read
  // (:70-98); the encoder reads the whole input before the inefficiency test can fire on a flush.
  std::vector<u8> comp;
  const u8 *comp_data = src.stream;
  u64 comp_len = src.stream_len;
  if (!comp_data) {
    comp.resize((size_t)(input_size + input_size / 50 + 4096));
    orc_encode_stream(in, input_size, info.level, (i64)input_size, 0, comp.data(), comp.size(), &comp_len, nullptr, 0, nullptr);
    comp_data = comp.data();
  }
  Update(CRC, in, input_size);
  // Write_Block raises Compression_inefficient as soon as output_size >= input_size (zip-compress.adb:468-490);
  // the running total reaches its maximum at the final flush, so the test is on the whole stream.
  bool compression_ok = !(comp_len >= input_size);
  if (compression_ok) {
    info.stream.Write(comp_data, comp_len);
    output_size = comp_len;
    zip_type = 12;                                      // Compression_format_code.bzip2_code (:209)
  }
  CRC = Final(CRC);                                     // :218
  if (!compression_ok) {                                // :224-235: go back and just store the data
    info.stream.index = idx_out;
    Init(CRC);
    zip_type = 0;                                       // Store_data (:105)
    Update(CRC, in, input_size);
    info.stream.Write(in, input_size);
    output_size = input_size;
    CRC = Final(CRC);
  }
}

int Add_Stream(Zip_Create_Info &info, const std::string &stream_name, const u8 *data, u64 size, const Stream_Source &src, u32 time,
               bool unicode, bool read_only) {                        // zip-create.adb:194-297
  std::string entry_name = stream_name;                 // Unixify (:180-192)
  for (char &c : entry_name) if (c == '\\') c = '/';
  info.contains.emplace_back();                         // Add_catalogue_entry (:103-134)
  Central_File_Header &cfh = info.contains.back().head;
  cfh.made_by_version = 23;
  cfh.comment_length = 0; cfh.disk_number_start = 0; cfh.internal_attributes = 0; cfh.external_attributes = 0;
  cfh.short_info.needed_extract_version = 10;
  cfh.short_info.bit_flag = 0;
  Local_File_Header &shi = cfh.short_info;
  if (unicode) shi.bit_flag |= 1u << 11;                // Language_Encoding_Flag_Bit (:222-224)
  if (read_only) cfh.external_attributes |= 1;          // :228-230
  info.contains.back().name = entry_name;
  if (Check_Size(info, size)) return 1;
  shi.file_timedate = time;
  shi.uncompressed_size = size;
  shi.compressed_size = shi.uncompressed_size;
  shi.filename_length = (u16)entry_name.size();
  shi.extra_field_length = 0;
  const u64 mem1 = info.stream.index;
  cfh.local_header_offset = mem1 - 1;
  const Extra_Field_Policy_Kind pol = Needs_Local_Zip_64_Header_Extension(shi, cfh.local_header_offset) ? force_zip_64 : force_empty;
  Write_Local(info.stream, shi, pol);                   // incomplete informations (:244-245)
  info.stream.Write((const u8 *)entry_name.data(), entry_name.size());
  Local_File_Header_Extension fh_extra;
  if (pol == force_zip_64) {
    fh_extra.tag = 1; fh_extra.size = (u16)(local_header_extension_short_length - 4);
    Write_Ext(info.stream, fh_extra, true);
  }
  Compress_Data(info, data, size, src, shi.crc_32, shi.compressed_size, shi.zip_type);
  const u64 mem2 = info.stream.index;
  info.stream.index = mem1;                             // rewrite with complete informations (:279-292)
  Write_Local(info.stream, shi, pol);
  if (pol == force_zip_64) {
    info.stream.Write((const u8 *)entry_name.data(), entry_name.size());
    fh_extra.value_64[0] = shi.uncompressed_size; fh_extra.value_64[1] = shi.compressed_size; fh_extra.value_64[2] = cfh.local_header_offset;
    Write_Ext(info.stream, fh_extra, true);
  }
  info.stream.index = mem2;
  return 0;
}

int Finish(Zip_Create_Info &info) {                     // zip-create.adb:645-756
  u64 current_index = info.stream.index;
  u64 central_dir_offset = current_index - 1, total_entries = 0, central_dir_size = 0;
  if (!info.zip_64 && info.contains.size() >= 65535) info.zip_64 = true;
  for (Entry &cat : info.contains) {
    total_entries++;
    const bool needs = Needs_Local_Zip_64_Header_Extension(cat.head.short_info, cat.head.local_header_offset);
    Local_File_Header_Extension fh_extra;
    if (needs) {
      cat.head.short_info.extra_field_length = (u16)local_header_extension_length;
      fh_extra.tag = 1; fh_extra.size = (u16)(local_header_extension_length - 4);
      fh_extra.value_64[0] = cat.head.short_info.uncompressed_size;
      fh_extra.value_64[1] = cat.head.short_info.compressed_size;
      fh_extra.value_64[2] = cat.head.local_header_offset;
      cat.head.short_info.uncompressed_size = 0xFFFFFFFFull;
      cat.head.short_info.compressed_size = 0xFFFFFFFFull;
      cat.head.local_header_offset = 0xFFFFFFFFull;
      info.zip_64 = true;
    } else {
      cat.head.short_info.extra_field_length = 0;
    }
    Write_Central(info.stream, cat.head);
    info.stream.Write((const u8 *)cat.name.data(), cat.name.size());
    if (needs) Write_Ext(info.stream, fh_extra, false);
    central_dir_size += 46 + cat.head.short_info.filename_length + cat.head.short_info.extra_field_length;
    current_index = info.stream.index;
  }
  if (!info.contains.empty() && Check_Size(info, current_index)) return 1;
  u64 disk_total_entries = total_entries;
  if (info.zip_64) {
    Buf eb;                                             // zip-headers.adb:522-538
    eb.PK(6, 6);
    eb.bf64(44); eb.bf16(0x2D); eb.bf16(0x2D); eb.bf32(0); eb.bf32(0);
    eb.bf64(disk_total_entries); eb.bf64(total_entries); eb.bf64(central_dir_size); eb.bf64(central_dir_offset);
    const u64 rel = info.stream.index - 1;
    info.stream.Write(eb.b.data(), eb.b.size());
    Buf el;                                             // :556-567
    el.PK(6, 7);
    el.bf32(0); el.bf64(rel); el.bf32(1);
    info.stream.Write(el.b.data(), el.b.size());
    disk_total_entries = 0xFFFF; total_entries = 0xFFFF; central_dir_size = 0xFFFFFFFFull; central_dir_offset = 0xFFFFFFFFull;
  }
  Buf ed;                                               // :477-494
  ed.PK(5, 6);
  ed.bf16(0); ed.bf16(0); ed.bf16((u32)disk_total_entries); ed.bf16((u32)total_entries);
  ed.bf32(central_dir_size); ed.bf32(central_dir_offset); ed.bf16(0);
  info.stream.Write(ed.b.data(), ed.b.size());
  return 0;
}

int zip_create(int level, u32 n_entries, const u8 *in, const u64 *in_offsets, const u64 *sizes, const char *names,
               const u32 *name_offsets, const u32 *dos_times, const u32 *flags, const u8 *streams, const u64 *stream_offsets,
               const u64 *stream_lens, u8 *out, u64 out_cap, u64 *out_len, u16 *methods) {
  Zip_Create_Info info;
  info.level = level;
  for (u32 i = 0; i < n_entries; i++) {
    const std::string nm(names + name_offsets[i], names + name_offsets[i + 1]);
    const u32 fl = flags ? flags[i] : 0;
    Stream_Source src;
    if (streams) { src.stream = streams + stream_offsets[i]; src.stream_len = stream_lens[i]; }
    if (Add_Stream(info, nm, in + in_offsets[i], sizes[i], src, dos_times ? dos_times[i] : 16789u * 65536u, fl & 1u, fl & 2u)) return 3;
    if (methods) methods[i] = info.contains.back().head.short_info.zip_type;
  }
  if (Finish(info)) return 3;
  if (out_len) *out_len = info.stream.data.size();
  if (info.stream.data.size() > out_cap) return 2;
  if (out) memcpy(out, info.stream.data.data(), info.stream.data.size());
  return 0;
}

}  // namespace

extern "C" {

u32 orc_zip_crc32(const u8 *in, u64 n) {
  u32 c;
  Init(c);
  Update(c, in, n);
  return Final(c);
}

// methods[i] (may be NULL) receives the final zip_type of entry i.
int orc_zip_create(int level, u32 n_entries, const u8 *in, const u64 *in_offsets, const u64 *sizes, const char *names,
                   const u32 *name_offsets, const u32 *dos_times, const u32 *flags, u8 *out, u64 out_cap, u64 *out_len,
                   u16 *methods) {
  return zip_create(level, n_entries, in, in_offsets, sizes, names, name_offsets, dos_times, flags, nullptr, nullptr, nullptr,
                    out, out_cap, out_len, methods);
}

// The same archive with the BZip2 stream of entry i given as streams[stream_offsets[i] ..][0 .. stream_lens[i]) instead
// of encoded here.  An entry with stream_lens[i] >= sizes[i] is stored, and its stream bytes are not read.
int orc_zip_create_given(int level, u32 n_entries, const u8 *in, const u64 *in_offsets, const u64 *sizes, const char *names,
                         const u32 *name_offsets, const u32 *dos_times, const u32 *flags, u8 *out, u64 out_cap, u64 *out_len,
                         u16 *methods, const u8 *streams, const u64 *stream_offsets, const u64 *stream_lens) {
  return zip_create(level, n_entries, in, in_offsets, sizes, names, name_offsets, dos_times, flags, streams, stream_offsets,
                    stream_lens, out, out_cap, out_len, methods);
}

}  // extern "C"
