// C++ mirror of the part of Zip.Create (zip_lib/zip-create.ads:60-279) that leads to the BZip2 encoder:
// Create_Archive, Set, Add_String, Add_File, Add_Stream (from memory), Add_Empty_Folder, Finish — above
// the C ABI of include/b2gpu.h.  The reference compresses an entry inside every Add_* call
// (zip-create.adb:253-265, serial per entry); here the Add_* calls only queue the entry and Finish
// sends the whole catalogue through ONE b2_zip_create call, so that the blocks of all entries share
// the device batches (SURVEY.md §8f row 1, "Add_Streams-style front end").  Zip_Writer below keeps the
// reference's shape instead: every Add_* goes to the device at once (b2_zip_add) and the archive file grows as
// entries complete, so memory does not grow with the archive.  The archive bytes are the ones the reference
// writes.  No CPU fallback: without the CUDA library every call throws.
#pragma once
#include <cstdint>
#include <cstdio>
#include <fcntl.h>
#include <fstream>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/b2gpu.h"

namespace zip_create {

// Zip.Compress.Compression_Method, the BZip2 members only (zip-compress.ads)
enum Compression_Method { BZip2_1 = B2_BLOCK_100K, BZip2_2 = B2_BLOCK_400K, BZip2_3 = B2_BLOCK_900K };
enum Duplicate_name_policy { admit_duplicates = B2_ZIP_ADMIT_DUPLICATES, error_on_duplicate = B2_ZIP_ERROR_ON_DUPLICATE };
using Time = uint32_t;                                        // Zip_Streams.Time (DOS date-time)
constexpr Time default_creation_time = 16789u * 65536u;       // Zip_Streams.default_time (zip_streams.ads:223)

struct Zip_error : std::runtime_error { using std::runtime_error::runtime_error; };
struct Duplicate_name : Zip_error { using Zip_error::Zip_error; };

class Zip_Create_Info {
 public:
  // Create_Archive (zip-create.ads:72-77); the archive goes to memory (Zip_Memory_Stream) or to a file
  void Create_Archive(const std::string &Archive_Name, Compression_Method Compress_Method = BZip2_3,
                      Duplicate_name_policy Duplicates = admit_duplicates, int device = 0) {
    name_ = Archive_Name; method_ = Compress_Method; duplicates_ = Duplicates; device_ = device;
    created_ = true;
    data_.clear(); offs_.clear(); sizes_.clear(); names_.clear(); name_offs_.assign(1, 0); times_.clear(); flags_.clear();
  }
  bool Is_Created() const { return created_; }
  const std::string &Name() const { return name_; }
  // Set (zip-create.ads:85-86).  One method per archive here: the entries are compressed together.
  void Set(Compression_Method New_Method) {
    if (!sizes_.empty() && New_Method != method_) throw Zip_error("Set: all queued entries share one BZip2 method");
    method_ = New_Method;
  }
  // Add_String (zip-create.ads:139-146)
  void Add_String(const std::string &Contents, const std::string &Name_in_archive, bool Name_UTF_8_encoded = false,
                  Time Creation_time = default_creation_time) {
    Add_Stream(reinterpret_cast<const uint8_t *>(Contents.data()), Contents.size(), Name_in_archive, Creation_time,
               Name_UTF_8_encoded, false);
  }
  // Add_Stream (zip-create.ads:94-103), the stream being a memory buffer with its name, time and attributes
  void Add_Stream(const uint8_t *bytes, uint64_t size, const std::string &Name, Time Modification_time = default_creation_time,
                  bool Is_Unicode_Name = false, bool Is_Read_Only = false) {
    require_created();
    offs_.push_back(data_.size());
    sizes_.push_back(size);
    data_.insert(data_.end(), bytes, bytes + size);
    data_.resize((data_.size() + 15) & ~size_t(15));
    names_ += Name;
    name_offs_.push_back((uint32_t)names_.size());
    times_.push_back(Modification_time);
    flags_.push_back((Is_Unicode_Name ? B2_ZIP_UNICODE_NAME : 0u) | (Is_Read_Only ? B2_ZIP_READ_ONLY : 0u));
  }
  // Add_File (zip-create.ads:124-135)
  void Add_File(const std::string &File_Name, const std::string &Name_in_archive = "", bool Delete_file_after = false,
                bool Name_UTF_8_encoded = false, Time Modification_time = default_creation_time, bool Is_read_only = false) {
    std::ifstream f(File_Name, std::ios::binary);
    if (!f) throw Zip_error("Add_File: cannot open " + File_Name);
    std::vector<uint8_t> buf((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    Add_Stream(buf.data(), buf.size(), Name_in_archive.empty() ? File_Name : Name_in_archive, Modification_time,
               Name_UTF_8_encoded, Is_read_only);
    if (Delete_file_after) std::remove(File_Name.c_str());
  }
  // Add_Empty_Folder (zip-create.ads:157-161): an empty entry whose name ends with '/'
  void Add_Empty_Folder(const std::string &Folder_Name, bool Name_UTF_8_encoded = false) {
    std::string n = Folder_Name;
    if (n.empty() || (n.back() != '/' && n.back() != '\\')) n += '/';
    Add_Stream(nullptr, 0, n, default_creation_time, Name_UTF_8_encoded, false);
  }
  // Finish (zip-create.ads:265): compresses the queued entries on the device, writes local headers,
  // payloads, central directory and end records; to the file Archive_Name unless it is empty.
  const std::vector<uint8_t> &Finish() {
    require_created();
    b2_encoder *enc = nullptr;
    if (b2_create((int)method_, device_, &enc) != B2_OK) throw Zip_error(std::string("b2_create: ") + b2_last_error());
    struct Guard { b2_encoder *e; ~Guard() { b2_destroy(e); } } guard{enc};
    const uint32_t n = (uint32_t)sizes_.size();
    archive_.resize(b2_zip_bound(n, names_.size(), data_.size()));
    info_.resize(n);
    uint64_t len = 0;
    const int rc = b2_zip_create(enc, n, data_.data(), offs_.data(), sizes_.data(), names_.data(), name_offs_.data(),
                                 times_.data(), flags_.data(), (int)duplicates_, archive_.data(), archive_.size(), &len,
                                 info_.data());
    if (rc == B2_ERR_DUPLICATE_NAME) throw Duplicate_name(b2_last_error());
    if (rc != B2_OK) throw Zip_error(std::string("b2_zip_create: ") + b2_last_error());
    archive_.resize(len);
    if (!name_.empty()) {
      std::ofstream f(name_, std::ios::binary);
      f.write(reinterpret_cast<const char *>(archive_.data()), (std::streamsize)archive_.size());
      if (!f) throw Zip_error("Finish: cannot write " + name_);
    }
    created_ = false;
    return archive_;
  }
  // Compressed_Size / Final_Method of every entry (the out parameters of Add_Stream, zip-create.ads:98-103)
  const std::vector<b2_zip_entry_info> &Entries() const { return info_; }

 private:
  void require_created() const { if (!created_) throw Zip_error("archive not created"); }
  bool created_ = false;
  std::string name_;
  Compression_Method method_ = BZip2_3;
  Duplicate_name_policy duplicates_ = admit_duplicates;
  int device_ = 0;
  std::vector<uint8_t> data_, archive_;
  std::vector<uint64_t> offs_, sizes_;
  std::string names_;
  std::vector<uint32_t> name_offs_{0}, times_, flags_;
  std::vector<b2_zip_entry_info> info_;
};

// Zip.Create as the reference runs it (zip-create.adb:194-297): every Add_* compresses its entry at once, through
// b2_zip_add, and the archive file is written as entries complete.  Host memory holds one entry's input and its
// output; device memory is bounded by the window (include/b2gpu.h, b2_zip_begin).  The bytes are those of
// Zip_Create_Info for the same calls.
class Zip_Writer {
 public:
  Zip_Writer() = default;
  Zip_Writer(const Zip_Writer &) = delete;
  Zip_Writer &operator=(const Zip_Writer &) = delete;
  ~Zip_Writer() {
    if (enc_) { b2_zip_abort(enc_); b2_destroy(enc_); }
  }
  // Create_Archive (zip-create.ads:72-77).  window_bytes: see b2_zip_begin (0 = 512 MiB).
  void Create_Archive(const std::string &Archive_Name, Compression_Method Compress_Method = BZip2_3,
                      Duplicate_name_policy Duplicates = admit_duplicates, int device = 0, uint64_t window_bytes = 0) {
    if (enc_ && (method_ != Compress_Method || device_ != device)) { b2_zip_abort(enc_); b2_destroy(enc_); enc_ = nullptr; }
    if (!enc_ && b2_create((int)Compress_Method, device, &enc_) != B2_OK) throw Zip_error(std::string("b2_create: ") + b2_last_error());
    method_ = Compress_Method; device_ = device;
    b2_zip_abort(enc_);
    if (b2_zip_begin(enc_, (int)Duplicates, window_bytes) != B2_OK) throw Zip_error(std::string("b2_zip_begin: ") + b2_last_error());
    file_.close();
    file_.open(Archive_Name, std::ios::binary | std::ios::trunc);
    if (!file_) { b2_zip_abort(enc_); throw Zip_error("Create_Archive: cannot write " + Archive_Name); }
    n_ = 0;
    info_.clear();
    created_ = true;
  }
  bool Is_Created() const { return created_; }
  // Add_String (zip-create.ads:139-146)
  void Add_String(const std::string &Contents, const std::string &Name_in_archive, bool Name_UTF_8_encoded = false,
                  Time Creation_time = default_creation_time) {
    Add_Stream(reinterpret_cast<const uint8_t *>(Contents.data()), Contents.size(), Name_in_archive, Creation_time,
               Name_UTF_8_encoded, false);
  }
  // Add_Stream (zip-create.ads:94-103), the stream being a memory buffer: compressed and written before it returns.
  void Add_Stream(const uint8_t *bytes, uint64_t size, const std::string &Name, Time Modification_time = default_creation_time,
                  bool Is_Unicode_Name = false, bool Is_Read_Only = false) {
    require_created();
    out_.resize(b2_zip_add_bound(enc_, size, (uint32_t)Name.size()));
    uint64_t len = 0;
    const uint32_t fl = (Is_Unicode_Name ? B2_ZIP_UNICODE_NAME : 0u) | (Is_Read_Only ? B2_ZIP_READ_ONLY : 0u);
    const int rc = b2_zip_add(enc_, Name.data(), (uint32_t)Name.size(), Modification_time, fl, bytes, size, out_.data(),
                              out_.size(), &len);
    if (rc == B2_ERR_DUPLICATE_NAME) throw Duplicate_name(b2_last_error());     // the archive stays open
    if (rc != B2_OK) { created_ = false; throw Zip_error(std::string("b2_zip_add: ") + b2_last_error()); }
    n_++;
    write(len);
  }
  // Add_File (zip-create.ads:124-135): the file is mapped, one file at a time.
  void Add_File(const std::string &File_Name, const std::string &Name_in_archive = "", bool Delete_file_after = false,
                bool Name_UTF_8_encoded = false, Time Modification_time = default_creation_time, bool Is_read_only = false) {
    require_created();
    const int fd = open(File_Name.c_str(), O_RDONLY);
    if (fd < 0) throw Zip_error("Add_File: cannot open " + File_Name);
    struct stat st;
    if (fstat(fd, &st) != 0) { close(fd); throw Zip_error("Add_File: cannot stat " + File_Name); }
    const uint64_t size = (uint64_t)st.st_size;
    void *map = nullptr;
    if (size) {
      map = mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
      if (map == MAP_FAILED) { close(fd); throw Zip_error("Add_File: cannot map " + File_Name); }
    }
    close(fd);
    struct Unmap { void *p; uint64_t n; ~Unmap() { if (p) munmap(p, n); } } unmap{map, size};
    Add_Stream(static_cast<const uint8_t *>(map), size, Name_in_archive.empty() ? File_Name : Name_in_archive,
               Modification_time, Name_UTF_8_encoded, Is_read_only);
    if (Delete_file_after) std::remove(File_Name.c_str());
  }
  // Add_Empty_Folder (zip-create.ads:157-161): an empty entry whose name ends with '/'
  void Add_Empty_Folder(const std::string &Folder_Name, bool Name_UTF_8_encoded = false) {
    std::string n = Folder_Name;
    if (n.empty() || (n.back() != '/' && n.back() != '\\')) n += '/';
    Add_Stream(nullptr, 0, n, default_creation_time, Name_UTF_8_encoded, false);
  }
  // Finish (zip-create.ads:265): the queued entries, central directory and end records; closes the file.
  void Finish() {
    require_created();
    created_ = false;
    out_.resize(b2_zip_finish_bound(enc_));
    info_.resize(n_);
    uint64_t len = 0, n = 0;
    if (b2_zip_finish(enc_, out_.data(), out_.size(), &len, info_.data(), info_.size(), &n) != B2_OK)
      throw Zip_error(std::string("b2_zip_finish: ") + b2_last_error());
    write(len);
    file_.close();
    if (!file_) throw Zip_error("Finish: cannot write the archive");
  }
  // Compressed_Size / Final_Method of every entry, after Finish
  const std::vector<b2_zip_entry_info> &Entries() const { return info_; }

 private:
  void require_created() const { if (!created_) throw Zip_error("archive not created"); }
  void write(uint64_t len) {
    file_.write(reinterpret_cast<const char *>(out_.data()), (std::streamsize)len);
    if (!file_) { b2_zip_abort(enc_); created_ = false; throw Zip_error("cannot write the archive"); }
  }
  b2_encoder *enc_ = nullptr;
  Compression_Method method_ = BZip2_3;
  int device_ = 0;
  bool created_ = false;
  std::ofstream file_;
  std::vector<uint8_t> out_;
  uint64_t n_ = 0;
  std::vector<b2_zip_entry_info> info_;
};

}  // namespace zip_create
