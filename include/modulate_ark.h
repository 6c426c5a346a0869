/*
 * modulate_ark.h -- C binding of the archive-level facade (CArk / CDtaFile), for callers that cannot
 * link C++ classes (scripting languages, bench.py's end-to-end repack workload).
 *
 * Each function is one of the reference's command bodies run on the facade classes of
 * modulate_b200/csrc/ (which forward the data-parallel half to the kernels behind
 * modulate_b200.h):
 *   mod_ark_unpack   Unpack   (reference Modulate.cpp:291-317: CArk::Load + CArk::ExtractFiles)
 *   mod_ark_find     search every entry for a byte pattern (CArk::Load + CArk::FindInFiles; no
 *                    reference counterpart)
 *   mod_ark_find_set the same for a set of patterns in one pass (CArk::FindSetInFiles)
 *   mod_ark_find_masked / mod_ark_find_set_nocase  wildcard and case-insensitive forms of the two
 *   mod_ark_pack     Pack     (reference Modulate.cpp:380-450: song list from the DTA configs unless
 *                              pack_all, CArk::Load of the reference header, ConstructFromDirectory,
 *                              BuildArk, SaveArk)
 *   mod_dta_set_int  the host-side DTA patch of a repack: CDtaFile::Load, replace the integer that
 *                    follows the symbol `key`, CDtaFile::Save
 * They return the reference's eError codes (0 = eError_NoError, reference Error.h:5-20) and print
 * the reference's messages to stdout.  Like the reference they go through the process-wide CSettings
 * switches, so they are not re-entrant.  `body_key` != 0 ciphers every entry body with that key,
 * stream restarting per entry (extension: the reference never ciphers ARK bodies).
 */
#ifndef MODULATE_ARK_H
#define MODULATE_ARK_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* `header_path`: the .hdr file; `part_dir`: directory of the .ark parts ("" = current directory);
 * `target_dir`: where the files go (created as needed; must end in '/'). */
int mod_ark_unpack(const char* header_path, const char* part_dir, const char* target_dir, int32_t body_key);

/* CArk::Load + CArk::FindInFiles: every position at which an entry's deciphered bytes (entry keys all
 * `body_key`) hold the `len`-byte pattern (1..64).  *out_total gets the exact number of matches;
 * out_file / out_offset (capacity max_matches each; may be NULL when max_matches is 0) get the first
 * min(total, max_matches) of them, (file table index, offset in the entry), sorted -- see CArk.h for
 * when a truncated list is not the first ones.  Returns an eError (0 = success). */
int mod_ark_find(const char* header_path, const char* part_dir, const uint8_t* pattern, uint32_t len, int32_t body_key,
                 uint64_t max_matches, uint32_t* out_file, uint32_t* out_offset, uint64_t* out_total);

/* CArk::Load + CArk::FindSetInFiles: mod_ark_find for the `n` patterns (1..256, distinct, 1..64 bytes each) given
 * as `lens` bytes each of `bytes`, concatenated in list order, searched in one pass.  out_file / out_offset /
 * out_pattern (capacity max_matches each; may be NULL when max_matches is 0) get the first min(total, max_matches)
 * matches sorted by (file, offset, pattern); out_pattern_counts (n entries, may be NULL) the exact matches per
 * pattern.  Returns an eError (0 = success). */
int mod_ark_find_set(const char* header_path, const char* part_dir, const uint8_t* bytes, const uint32_t* lens, uint32_t n,
                     int32_t body_key, uint64_t max_matches, uint32_t* out_file, uint32_t* out_offset, uint32_t* out_pattern,
                     uint64_t* out_total, uint64_t* out_pattern_counts);

/* mod_ark_find with a mask byte per pattern byte (CArk::FindMaskedInFiles): an entry byte t matches pattern byte k
 * when ((t ^ pattern[k]) & mask[k]) == 0 -- 0x00 is any byte, 0xDF on an upper-case letter either case.  A null or
 * all-zero mask is eError_InvalidParameter. */
int mod_ark_find_masked(const char* header_path, const char* part_dir, const uint8_t* pattern, const uint8_t* mask, uint32_t len,
                        int32_t body_key, uint64_t max_matches, uint32_t* out_file, uint32_t* out_offset, uint64_t* out_total);

/* mod_ark_find_set ignoring ASCII case (mod_pattern_set_create_nocase): the patterns must differ ignoring case. */
int mod_ark_find_set_nocase(const char* header_path, const char* part_dir, const uint8_t* bytes, const uint32_t* lens, uint32_t n,
                            int32_t body_key, uint64_t max_matches, uint32_t* out_file, uint32_t* out_offset,
                            uint32_t* out_pattern, uint64_t* out_total, uint64_t* out_pattern_counts);

/* `input_dir` and `output_dir` must end in '/'; the header is written to output_dir + header_name. */
int mod_ark_pack(const char* reference_header_path, const char* input_dir, const char* output_dir,
                 const char* header_name, int ps4, int pack_all, int ignore_new_files, int32_t body_key);

int mod_dta_set_int(const char* dta_path, const char* key, int32_t value);

#ifdef __cplusplus
}
#endif

#endif /* MODULATE_ARK_H */
