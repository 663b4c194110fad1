// Writes the files named on the command line into a Zip archive with zip_create::Zip_Writer (one entry per file,
// compressed and written as it is added).
//   test_zip_writer [--level 1|4|9] [--window BYTES] [--error-on-duplicate] ARCHIVE FILE...
// Prints "entries=N" on success; exit 1 with the message on an error, 3 on Duplicate_name.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "zip_create.hpp"

int main(int argc, char **argv) {
  int level = 9, i = 1;
  uint64_t window = 0;
  zip_create::Duplicate_name_policy dup = zip_create::admit_duplicates;
  for (; i < argc && argv[i][0] == '-' && argv[i][1] == '-'; i++) {
    if (!strcmp(argv[i], "--level") && i + 1 < argc) level = atoi(argv[++i]);
    else if (!strcmp(argv[i], "--window") && i + 1 < argc) window = strtoull(argv[++i], nullptr, 10);
    else if (!strcmp(argv[i], "--error-on-duplicate")) dup = zip_create::error_on_duplicate;
    else { fprintf(stderr, "unknown option %s\n", argv[i]); return 2; }
  }
  if (i >= argc) { fprintf(stderr, "usage: test_zip_writer [--level L] [--window W] [--error-on-duplicate] ARCHIVE FILE...\n"); return 2; }
  try {
    zip_create::Zip_Writer z;
    z.Create_Archive(argv[i], (zip_create::Compression_Method)level, dup, 0, window);
    for (int k = i + 1; k < argc; k++) z.Add_File(argv[k]);
    z.Finish();
    printf("entries=%zu\n", z.Entries().size());
  } catch (const zip_create::Duplicate_name &e) {
    fprintf(stderr, "%s\n", e.what());
    return 3;
  } catch (const std::exception &e) {
    fprintf(stderr, "%s\n", e.what());
    return 1;
  }
  return 0;
}
