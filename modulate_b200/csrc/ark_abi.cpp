// ark_abi.cpp -- the C binding declared in include/modulate_ark.h: the reference's Unpack / Pack
// command bodies (Modulate.cpp:291-317, :380-450) and the archive search on the facade classes.
#include "../../include/modulate_ark.h"

#include <algorithm>
#include <exception>
#include <iostream>
#include <string>
#include <vector>

#include "CArk.h"
#include "CDtaFile.h"
#include "Error.h"
#include "Settings.h"

namespace {

// No C++ exception may cross the extern "C" boundary.
template <class F>
int Guarded(F lBody)
{
    try {
        return (int)lBody();
    } catch (const std::exception& lError) {
        std::cout << "ERROR: " << lError.what() << "\n";
        return (int)eError_InvalidData;
    } catch (...) {
        return (int)eError_InvalidData;
    }
}

}  // namespace

extern "C" {

int mod_ark_unpack(const char* header_path, const char* part_dir, const char* target_dir, int32_t body_key)
{
    return Guarded([&]() -> eError {
        if (!header_path || !target_dir)
            return eError_InvalidParameter;
        CArk lArkHeader;
        lArkHeader.SetUniformEntryKey(body_key);
        lArkHeader.SetPartDirectory(part_dir ? part_dir : "");
        eError leError = lArkHeader.Load(header_path);
        SHOW_ERROR_AND_RETURN;
        leError = lArkHeader.ExtractFiles(0, lArkHeader.GetNumFiles(), target_dir);
        SHOW_ERROR_AND_RETURN;
        return eError_NoError;
    });
}

// The body of mod_ark_find and mod_ark_find_masked (mask null: the exact search).
static int ArkFind(const char* header_path, const char* part_dir, const uint8_t* pattern, const uint8_t* mask, uint32_t len,
                   int32_t body_key, uint64_t max_matches, uint32_t* out_file, uint32_t* out_offset, uint64_t* out_total)
{
    return Guarded([&]() -> eError {
        if (!header_path || !pattern || !out_total || (max_matches && (!out_file || !out_offset)))
            return eError_InvalidParameter;
        CArk lArkHeader;
        lArkHeader.SetUniformEntryKey(body_key);
        lArkHeader.SetPartDirectory(part_dir ? part_dir : "");
        eError leError = lArkHeader.Load(header_path);
        SHOW_ERROR_AND_RETURN;
        std::vector<SFileMatch> laMatches;
        leError = mask ? lArkHeader.FindMaskedInFiles(pattern, mask, len, max_matches, laMatches, out_total)
                       : lArkHeader.FindInFiles(pattern, len, max_matches, laMatches, out_total);
        SHOW_ERROR_AND_RETURN;
        for (size_t ii = 0; ii < laMatches.size(); ++ii) {
            out_file[ii] = (uint32_t)laMatches[ii].file;
            out_offset[ii] = laMatches[ii].offset;
        }
        return eError_NoError;
    });
}

int mod_ark_find(const char* header_path, const char* part_dir, const uint8_t* pattern, uint32_t len, int32_t body_key,
                 uint64_t max_matches, uint32_t* out_file, uint32_t* out_offset, uint64_t* out_total)
{
    return ArkFind(header_path, part_dir, pattern, nullptr, len, body_key, max_matches, out_file, out_offset, out_total);
}

int mod_ark_find_masked(const char* header_path, const char* part_dir, const uint8_t* pattern, const uint8_t* mask, uint32_t len,
                        int32_t body_key, uint64_t max_matches, uint32_t* out_file, uint32_t* out_offset, uint64_t* out_total)
{
    if (!mask)
        return eError_InvalidParameter;
    return ArkFind(header_path, part_dir, pattern, mask, len, body_key, max_matches, out_file, out_offset, out_total);
}

// The body of mod_ark_find_set and mod_ark_find_set_nocase.
static int ArkFindSet(const char* header_path, const char* part_dir, const uint8_t* bytes, const uint32_t* lens, uint32_t n,
                      int32_t body_key, uint64_t max_matches, uint32_t* out_file, uint32_t* out_offset, uint32_t* out_pattern,
                      uint64_t* out_total, uint64_t* out_pattern_counts, bool ignore_case)
{
    return Guarded([&]() -> eError {
        if (!header_path || !bytes || !lens || !out_total || (max_matches && (!out_file || !out_offset || !out_pattern)))
            return eError_InvalidParameter;
        std::vector<std::string> laPatterns;
        uint64_t luAt = 0;
        for (uint32_t jj = 0; jj < n; ++jj) {
            laPatterns.emplace_back((const char*)bytes + luAt, lens[jj]);
            luAt += lens[jj];
        }
        CArk lArkHeader;
        lArkHeader.SetUniformEntryKey(body_key);
        lArkHeader.SetPartDirectory(part_dir ? part_dir : "");
        eError leError = lArkHeader.Load(header_path);
        SHOW_ERROR_AND_RETURN;
        std::vector<SFileSetMatch> laMatches;
        std::vector<uint64_t> laPatternCounts;
        leError = lArkHeader.FindSetInFiles(laPatterns, max_matches, laMatches, out_total, nullptr, &laPatternCounts, ignore_case);
        SHOW_ERROR_AND_RETURN;
        for (size_t ii = 0; ii < laMatches.size(); ++ii) {
            out_file[ii] = (uint32_t)laMatches[ii].file;
            out_offset[ii] = laMatches[ii].offset;
            out_pattern[ii] = laMatches[ii].pattern;
        }
        if (out_pattern_counts)
            std::copy(laPatternCounts.begin(), laPatternCounts.end(), out_pattern_counts);
        return eError_NoError;
    });
}

int mod_ark_find_set(const char* header_path, const char* part_dir, const uint8_t* bytes, const uint32_t* lens, uint32_t n,
                     int32_t body_key, uint64_t max_matches, uint32_t* out_file, uint32_t* out_offset, uint32_t* out_pattern,
                     uint64_t* out_total, uint64_t* out_pattern_counts)
{
    return ArkFindSet(header_path, part_dir, bytes, lens, n, body_key, max_matches, out_file, out_offset, out_pattern, out_total,
                      out_pattern_counts, false);
}

int mod_ark_find_set_nocase(const char* header_path, const char* part_dir, const uint8_t* bytes, const uint32_t* lens, uint32_t n,
                            int32_t body_key, uint64_t max_matches, uint32_t* out_file, uint32_t* out_offset,
                            uint32_t* out_pattern, uint64_t* out_total, uint64_t* out_pattern_counts)
{
    return ArkFindSet(header_path, part_dir, bytes, lens, n, body_key, max_matches, out_file, out_offset, out_pattern, out_total,
                      out_pattern_counts, true);
}

int mod_ark_pack(const char* reference_header_path, const char* input_dir, const char* output_dir, const char* header_name,
                 int ps4, int pack_all, int ignore_new_files, int32_t body_key)
{
    return Guarded([&]() -> eError {
        if (!reference_header_path || !input_dir || !output_dir || !header_name)
            return eError_InvalidParameter;
        CSettings::mbPS4 = ps4 != 0;
        CSettings::msPlatform = ps4 ? "ps4" : "ps3";
        CSettings::mbPackAllFiles = pack_all != 0;
        CSettings::mbIgnoreNewFiles = ignore_new_files != 0;
        const std::string lInputPath = input_dir, lPlatform = CSettings::msPlatform;

        eError leError = eError_NoError;
        std::vector<SSongConfig> lSongs;
        if (!CSettings::mbPackAllFiles) {
            CDtaFile lAmpConfig;
            leError = lAmpConfig.Load((lInputPath + lPlatform + "/config/amp_config.dta_dta_" + lPlatform).c_str());
            SHOW_ERROR_AND_RETURN;
            lSongs = lAmpConfig.GetSongs();
            CDtaFile lSongsConfig;
            leError = lSongsConfig.Load((lInputPath + lPlatform + "/config/amp_songs_config.dta_dta_" + lPlatform).c_str());
            SHOW_ERROR_AND_RETURN;
            lSongsConfig.GetSongData(lSongs);
        }
        CArk lReferenceArkHeader;
        leError = lReferenceArkHeader.Load(reference_header_path);
        SHOW_ERROR_AND_RETURN;
        CArk lArkHeader;
        lArkHeader.SetUniformEntryKey(body_key);
        leError = lArkHeader.ConstructFromDirectory(input_dir, lReferenceArkHeader, lSongs);
        SHOW_ERROR_AND_RETURN;
        leError = lArkHeader.BuildArk(input_dir, lSongs);
        SHOW_ERROR_AND_RETURN;
        leError = lArkHeader.SaveArk(output_dir, header_name);
        SHOW_ERROR_AND_RETURN;
        return eError_NoError;
    });
}

int mod_dta_set_int(const char* dta_path, const char* key, int32_t value)
{
    return Guarded([&]() -> eError {
        if (!dta_path || !key)
            return eError_InvalidParameter;
        CDtaFile lDta;
        eError leError = lDta.Load(dta_path);
        ERROR_RETURN;
        if (!lDta.SetIntAfter(key, value))
            return eError_InvalidParameter;
        return lDta.Save(dta_path);
    });
}

}  // extern "C"
