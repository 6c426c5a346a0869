// CArk.h -- drop-in for the archive-container class of the reference (/root/reference/Modulate/
// CArk.h:10-90): same public method names, argument meaning and eError convention, portable
// C++17 (the reference is Win32/MSVC-only), with the data-parallel half moved to the GPU:
//
//   Load                  reads the .hdr, deciphers it on the GPU (mod_cycle; reference call site
//                         CArk.cpp:338-339) and parses it on the host (ArkHeader.cpp)
//   LoadArkData           concatenates the .ark parts into one PINNED host image (CArk.cpp:723-758)
//   ExtractFiles          turns the file table into ONE descriptor plan (mod_plan_create) and gathers
//                         the entries through the batched kernel group by group (mod_plan_run_window;
//                         CArk.cpp:494) in the reader -> GPU -> writer slot-ring pipeline of
//                         ArkPipeline.h, over every visible GPU: nothing is ever waited for on the
//                         thread that enqueues
//   FindInFiles           searches every entry for a byte pattern through the same pipeline, reading
//                         the parts like ExtractFiles and keeping only the match lists (mod_plan_find_window)
//   BuildArk              assigns byte-packed offsets and part sizes from the file sizes (CArk.cpp:760-828)
//   SaveArk               serialises + enciphers the header (CArk.cpp:1135-1136) and STREAMS the payload
//                         from the input files into the part files through the same pipeline (entries
//                         that carry a key are ciphered on the GPU on the way)
//
// The reference never ciphers ARK bodies (SURVEY.md Finding 2): all entry keys default to 0, the
// identity keystream, so the bytes produced are the reference's.  SetEntryKeys / SetUniformEntryKey
// are extensions used by the synthetic per-entry-key configurations of BASELINE.json.
#pragma once

#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "ArkHeader.h"
#include "CDtaFile.h"  // SSongConfig, like the reference (CArk.h:6)
#include "Error.h"

namespace arkpipe {
struct Group;
struct Stage;
}

// One match of CArk::FindInFiles: entry `file` (index into the file table) holds the pattern at `offset`.
struct SFileMatch {
    int file;
    uint32_t offset;
};

// One match of CArk::FindSetInFiles: entry `file` holds pattern `pattern` (its index in the list) at `offset`.
struct SFileSetMatch {
    int file;
    uint32_t offset;
    uint32_t pattern;
};

class CArk
{
public:
    CArk();
    ~CArk();
    CArk(const CArk&) = delete;
    CArk& operator=(const CArk&) = delete;

    eError ConstructFromDirectory(const char* lpInputDirectory, const CArk& lReferenceHeader,
                                  std::vector<SSongConfig> laSongs);
    eError BuildArk(const char* lpInputDirectory, std::vector<SSongConfig> laSongs);
    eError SaveArk(const char* lpOutputDirectory, const char* lpHeaderFilename) const;

    eError Load(const char* lpHeaderFilename);
    eError ExtractFiles(int liFirstFileIndex, int liNumFiles, const char* lpTargetDirectory);
    bool FileExists(const char* lpFilename) const;

    int GetNumFiles() const;

    eError LoadArkData();

    // ---- extensions (not in the reference) ----
    void SetUniformEntryKey(int liKey);                  // every entry ciphered with liKey, stream restarting per entry
    void SetEntryKeys(const std::vector<int>& laKeys);   // one key per entry, in table order
    void SetPartDirectory(const char* lpDirectory);      // where LoadArkData looks for the part files ("" = cwd)
    // Every position at which an entry's deciphered bytes hold the luLen-byte pattern (1..64), overlapping
    // ones included, found on the GPU in one pass over the part files that writes nothing.  Entries that
    // share a name are each searched and reported (ExtractFiles keeps only one of them).  *lpTotal gets the
    // exact number of matches and lpFileCounts, when given, the exact number per entry in table order;
    // laMatches gets min(total, luMaxMatches) of them sorted by (file, offset) -- all of them, and so the
    // first luMaxMatches, unless more than luMaxMatches fall into one pipeline group (MOD_IO_GROUP_MIB of the
    // image), in which case which ones that group keeps is unspecified.
    eError FindInFiles(const unsigned char* lpPattern, uint32_t luLen, uint64_t luMaxMatches, std::vector<SFileMatch>& laMatches,
                       uint64_t* lpTotal, std::vector<uint64_t>* lpFileCounts = nullptr);
    // FindInFiles for a set of 1 to 256 distinct patterns of 1 to 64 bytes each, lengths mixed, in one pass: every
    // (pattern, position) at which an entry holds a pattern, overlapping matches and matches of different patterns
    // at one position included.  laMatches is sorted by (file, offset, pattern) and truncated like FindInFiles';
    // lpFileCounts gets the exact matches per entry and lpPatternCounts the exact matches per pattern, in list order.
    eError FindSetInFiles(const std::vector<std::string>& laPatterns, uint64_t luMaxMatches, std::vector<SFileSetMatch>& laMatches,
                          uint64_t* lpTotal, std::vector<uint64_t>* lpFileCounts = nullptr,
                          std::vector<uint64_t>* lpPatternCounts = nullptr, bool lbIgnoreCase = false);
    // lbIgnoreCase: ASCII letters match either case (mod_pattern_set_create_nocase), and patterns equal ignoring case
    // are refused.
    // FindInFiles with a mask byte per pattern byte: an entry byte t matches pattern byte k when
    // ((t ^ lpPattern[k]) & lpMask[k]) == 0 (0x00 any byte, 0xDF on a letter either case; mod_plan_find_masked).  An
    // all-zero mask is eError_InvalidParameter.
    eError FindMaskedInFiles(const unsigned char* lpPattern, const unsigned char* lpMask, uint32_t luLen, uint64_t luMaxMatches,
                             std::vector<SFileMatch>& laMatches, uint64_t* lpTotal, std::vector<uint64_t>* lpFileCounts = nullptr);
    const modark::HeaderImage& Header() const { return mHeader; }

private:
    int EntryKey(size_t liIndex) const;
    eError AllocateArkData();
    eError ReadParts();
    bool ReadImageRange(std::vector<int>& laFds, uint64_t luOffset, uint64_t luSize, unsigned char* lpDst) const;
    arkpipe::Stage ReadGroupsStage(const std::vector<arkpipe::Group>& laGroups, std::vector<int>& laPartFds) const;
    eError CheckEntriesInImage(uint64_t luImageSize) const;
    struct SearchSlot;
    struct SearchPass;
    // FindInFiles (lpMask null) and FindMaskedInFiles.
    eError FindOneInFiles(const unsigned char* lpPattern, const unsigned char* lpMask, uint32_t luLen, uint64_t luMaxMatches,
                          std::vector<SFileMatch>& laMatches, uint64_t* lpTotal, std::vector<uint64_t>* lpFileCounts);
    eError SearchParts(const SearchPass& lPass, std::vector<uint64_t>& laFileCounts, std::vector<uint64_t>& laPatternCounts);
    struct PartTarget {
        int miFd = -1;             // part file open for writing
        unsigned char* mpMap = nullptr;  // its mapping, when it could be mapped
        uint64_t muImageStart = 0; // first image byte it receives
        uint64_t muSize = 0;
    };
    eError StreamBuiltImage(const std::vector<PartTarget>& laTargets) const;
    bool ShouldPackFile(const std::vector<SSongConfig>& laSongs, const char* lpFilename) const;
    void ReleaseArkData();

    modark::HeaderImage mHeader;
    bool mbLoaded = false;

    unsigned char* mpArkData = nullptr;  // pinned host memory (mod_host_alloc), LoadArkData only
    uint64_t muArkDataSize = 0;

    bool mbBuilt = false;                // BuildArk has laid the image out; SaveArk streams it
    std::string mBuildInputDirectory;
    uint64_t muBuiltImageSize = 0;

    std::vector<int> maEntryKeys;
    int miUniformKey = 0;
    std::string mPartDirectory;
};
