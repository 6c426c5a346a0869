#include "CArk.h"

#include <dirent.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/types.h>
#include <unistd.h>

#include <algorithm>
#include <cctype>
#include <mutex>
#include <unordered_map>
#include <unordered_set>
#include <cstdio>
#include <cstring>
#include <functional>
#include <iostream>

#include "../../include/modulate_b200.h"
#include "ArkPipeline.h"
#include "CEncryptionCycler.h"
#include "Settings.h"

// The search entry points are an addition to version 2 of the C ABI: they are referenced weakly, so the
// facade still links against an implementation of the ABI that predates them, and FindInFiles /
// FindSetInFiles report that the library lacks the search instead of the program failing to load.
#pragma weak mod_plan_find_window
#pragma weak mod_plan_find_set_window
#pragma weak mod_pattern_set_create
#pragma weak mod_pattern_set_destroy
#pragma weak mod_plan_find_masked_window
#pragma weak mod_pattern_set_create_nocase

namespace {

bool ReadWholeFile(const std::string& lPath, std::vector<unsigned char>& lOut)
{
    FILE* lpFile = std::fopen(lPath.c_str(), "rb");
    if (!lpFile)
        return false;
    std::fseek(lpFile, 0, SEEK_END);
    const long liSize = std::ftell(lpFile);
    std::fseek(lpFile, 0, SEEK_SET);
    lOut.resize(liSize > 0 ? (size_t)liSize : 0);
    const size_t liRead = lOut.empty() ? 0 : std::fread(lOut.data(), 1, lOut.size(), lpFile);
    std::fclose(lpFile);
    return liRead == lOut.size();
}

long FileSize(const std::string& lPath)
{
    struct stat lInfo;
    if (stat(lPath.c_str(), &lInfo) != 0 || !S_ISREG(lInfo.st_mode))
        return -1;
    return (long)lInfo.st_size;
}

bool IsDirectory(const std::string& lPath)
{
    struct stat lInfo;
    return stat(lPath.c_str(), &lInfo) == 0 && S_ISDIR(lInfo.st_mode);
}

// mkdir -p for every directory component of lFilePath (the part before the last '/').
bool MakeParentDirectories(const std::string& lFilePath)
{
    for (size_t liSlash = lFilePath.find('/'); liSlash != std::string::npos; liSlash = lFilePath.find('/', liSlash + 1)) {
        if (liSlash == 0)
            continue;
        const std::string lDir = lFilePath.substr(0, liSlash);
        mkdir(lDir.c_str(), 0777);
        if (!IsDirectory(lDir))
            return false;
    }
    return true;
}

// An entry name may not climb out of the target directory ("..": the reference would follow it).
bool EscapesTarget(const std::string& lName)
{
    size_t liStart = 0;
    for (;;) {
        const size_t liSlash = lName.find('/', liStart);
        const std::string lPart = lName.substr(liStart, liSlash == std::string::npos ? std::string::npos : liSlash - liStart);
        if (lPart == "..")
            return true;
        if (liSlash == std::string::npos)
            return false;
        liStart = liSlash + 1;
    }
}

// Existing non-empty output is kept only when overwriting is disabled (reference CArk.cpp:439-454).
bool KeepExistingOutput(const std::string& lPath)
{
    if (CSettings::mbOverwriteOutputFiles)
        return false;
    return FileSize(lPath) > 0;
}

// Relative names of every regular file under lRoot (which ends in '/'), files of a directory first,
// then its sub-directories, each level in the order NTFS keeps its directory index in: by UPPER-CASED
// name (the reference walks with FindFirstFileA, Utils.cpp:5-70, and takes whatever order the file
// system returns; '_' therefore sorts after the letters, not before them).
void ListFiles(const std::string& lRoot, const std::string& lRelative, std::vector<std::string>& laOut)
{
    DIR* lpDir = opendir((lRoot + lRelative).c_str());
    if (!lpDir)
        return;
    std::vector<std::string> laFiles, laDirs;
    while (dirent* lpEntry = readdir(lpDir)) {
        const std::string lName = lpEntry->d_name;
        if (lName == "." || lName == "..")
            continue;
        // the directory entry usually says what it is; stat only when it does not (or for symlinks)
        bool lbDirectory = lpEntry->d_type == DT_DIR, lbFile = lpEntry->d_type == DT_REG;
        if (!lbDirectory && !lbFile) {
            const std::string lFull = lRoot + lRelative + lName;
            lbDirectory = IsDirectory(lFull);
            lbFile = !lbDirectory && FileSize(lFull) >= 0;
        }
        if (lbDirectory)
            laDirs.push_back(lName);
        else if (lbFile)
            laFiles.push_back(lName);
    }
    closedir(lpDir);
    // names that differ only in case cannot coexist on NTFS; on a case-sensitive file system they are
    // ordered by their bytes so that the walk is deterministic
    auto lLess = [](const std::string& lA, const std::string& lB) {
        const auto lUpperLess = [](char a, char b) { return std::toupper((unsigned char)a) < std::toupper((unsigned char)b); };
        if (std::lexicographical_compare(lA.begin(), lA.end(), lB.begin(), lB.end(), lUpperLess))
            return true;
        if (std::lexicographical_compare(lB.begin(), lB.end(), lA.begin(), lA.end(), lUpperLess))
            return false;
        return lA < lB;
    };
    std::sort(laFiles.begin(), laFiles.end(), lLess);
    std::sort(laDirs.begin(), laDirs.end(), lLess);
    for (const std::string& lName : laFiles)
        laOut.push_back(lRelative + lName);
    for (const std::string& lName : laDirs)
        ListFiles(lRoot, lRelative + lName + "/", laOut);
}

// mkdir -p with a per-thread memo of directories already known to exist (thousands of entries share
// a handful of folders; the reference re-runs _mkdir + stat for every component of every file,
// CArk.cpp:463-483).
bool MakeParentDirectoriesCached(const std::string& lFilePath, std::unordered_set<std::string>& lKnown)
{
    const size_t liLast = lFilePath.rfind('/');
    if (liLast == std::string::npos || liLast == 0)
        return true;
    if (lKnown.count(lFilePath.substr(0, liLast)))
        return true;
    if (!MakeParentDirectories(lFilePath))
        return false;
    lKnown.insert(lFilePath.substr(0, liLast));
    return true;
}

// pread / pwrite the whole range (short transfers are retried; a short FILE reads as zeros).
bool ReadFully(int liFd, unsigned char* lpDst, uint64_t luSize, uint64_t luOffset)
{
    while (luSize) {
        const ssize_t liGot = pread(liFd, lpDst, (size_t)std::min<uint64_t>(luSize, 1u << 30), (off_t)luOffset);
        if (liGot < 0)
            return false;
        if (liGot == 0) {
            std::memset(lpDst, 0, (size_t)luSize);
            return true;
        }
        lpDst += liGot;
        luOffset += (uint64_t)liGot;
        luSize -= (uint64_t)liGot;
    }
    return true;
}

bool WriteFully(int liFd, const unsigned char* lpSrc, uint64_t luSize, uint64_t luOffset)
{
    while (luSize) {
        const ssize_t liPut = pwrite(liFd, lpSrc, (size_t)std::min<uint64_t>(luSize, 1u << 30), (off_t)luOffset);
        if (liPut <= 0)
            return false;
        lpSrc += liPut;
        luOffset += (uint64_t)liPut;
        luSize -= (uint64_t)liPut;
    }
    return true;
}

}  // namespace

CArk::CArk() {}

CArk::~CArk() { ReleaseArkData(); }

void CArk::ReleaseArkData()
{
    if (mpArkData)
        mod_host_free(mpArkData);
    mpArkData = nullptr;
    muArkDataSize = 0;
}

void CArk::SetUniformEntryKey(int liKey)
{
    miUniformKey = liKey;
    maEntryKeys.clear();
}

void CArk::SetEntryKeys(const std::vector<int>& laKeys) { maEntryKeys = laKeys; }

void CArk::SetPartDirectory(const char* lpDirectory)
{
    mPartDirectory = lpDirectory ? lpDirectory : "";
    if (!mPartDirectory.empty() && mPartDirectory.back() != '/')
        mPartDirectory += '/';
}

int CArk::EntryKey(size_t liIndex) const { return liIndex < maEntryKeys.size() ? maEntryKeys[liIndex] : miUniformKey; }

int CArk::GetNumFiles() const { return (int)mHeader.maFiles.size(); }

bool CArk::FileExists(const char* lpFilename) const
{
    for (const modark::FileDef& lFile : mHeader.maFiles)
        if (lFile.mName == lpFilename)
            return true;
    return false;
}

// ---- read side ---------------------------------------------------------------------------------------

eError CArk::Load(const char* lpHeaderFilename)
{
    if (mbLoaded)
        return eError_AlreadyLoaded;  // reference CArk.cpp:303-306

    VERBOSE_OUT("Loading header file " << lpHeaderFilename);
    std::vector<unsigned char> lData;
    if (!ReadWholeFile(lpHeaderFilename, lData))
        return eError_FailedToOpenFile;
    VERBOSE_OUT("\nLoaded header (" << lData.size() << ") bytes\n");
    if (lData.size() < sizeof(uint32_t))
        return eError_UnknownVersionNumber;

    uint32_t luVersion = 0;
    std::memcpy(&luVersion, lData.data(), sizeof(luVersion));
    if (luVersion != CSettings::kuEncryptedVersionPS3 && luVersion != CSettings::kuEncryptedVersionPS4)
        return eError_UnknownVersionNumber;
    const unsigned int kuInitialKey =
        (luVersion == CSettings::kuEncryptedVersionPS3) ? CSettings::kuEncryptedPS3Key : CSettings::kuEncryptedPS4Key;

    // the magic stays in clear; everything after it is one Cycle() -- on the GPU
    CEncryptionCycler lDecrypt;
    lDecrypt.Cycle(lData.data() + sizeof(uint32_t), (unsigned int)(lData.size() - sizeof(uint32_t)), (int)kuInitialKey);

    eError leError = modark::ParseHeader(lData.data(), lData.size(), mHeader);
    SHOW_ERROR_AND_RETURN;
    mbLoaded = true;
    return eError_NoError;
}

// Read the parts back to back into the pinned image (reference CArk.cpp:741-755).
eError CArk::ReadParts()
{
    std::vector<int> laFds;
    const bool lbOk = ReadImageRange(laFds, 0, muArkDataSize, mpArkData);
    for (int liFd : laFds)
        if (liFd >= 0)
            close(liFd);
    return lbOk ? eError_NoError : eError_FailedToOpenFile;
}

eError CArk::AllocateArkData()
{
    ReleaseArkData();
    uint64_t luTotalArkSize = 0;
    for (const modark::PartDef& lPart : mHeader.maParts)
        luTotalArkSize += lPart.muSize;
    mpArkData = (unsigned char*)mod_host_alloc(luTotalArkSize ? luTotalArkSize : 1);
    if (!mpArkData) {
        std::cout << "Failed to allocate pinned memory for the archive: " << mod_last_error() << "\n";
        return eError_NoData;
    }
    muArkDataSize = luTotalArkSize;
    return eError_NoError;
}

// The reference's whole-image load (CArk.cpp:723-758), kept for callers that want the flat image;
// ExtractFiles does not need it any more (it streams ranges through a slot ring).
eError CArk::LoadArkData()
{
    eError leError = AllocateArkData();
    ERROR_RETURN;
    leError = ReadParts();
    SHOW_ERROR_AND_RETURN;
    return eError_NoError;
}

// Copy bytes [luOffset, luOffset + luSize) of the concatenated part files into lpDst with pread (safe
// from several threads at once), opening each part on first use (laFds caches the descriptors; it
// must be sized and guarded by the caller when shared).  Bytes a short part file lacks read as zero.
bool CArk::ReadImageRange(std::vector<int>& laFds, uint64_t luOffset, uint64_t luSize, unsigned char* lpDst) const
{
    static std::mutex lOpenMutex;
    {
        std::lock_guard<std::mutex> lLock(lOpenMutex);
        if (laFds.size() < mHeader.maParts.size())
            laFds.resize(mHeader.maParts.size(), -1);
    }
    uint64_t luPartStart = 0;
    for (size_t ii = 0; ii < mHeader.maParts.size() && luSize; ++ii) {
        const uint64_t luPartSize = mHeader.maParts[ii].muSize;
        const uint64_t luPartEnd = luPartStart + luPartSize;
        if (luOffset < luPartEnd) {
            int liFd;
            {
                std::lock_guard<std::mutex> lLock(lOpenMutex);
                if (laFds[ii] < 0)
                    laFds[ii] = open((mPartDirectory + mHeader.maParts[ii].mPath).c_str(), O_RDONLY);
                liFd = laFds[ii];
            }
            if (liFd < 0)
                return false;
            const uint64_t luTake = std::min(luSize, luPartEnd - luOffset);
            if (!ReadFully(liFd, lpDst, luTake, luOffset - luPartStart))
                return false;
            lpDst += luTake;
            luOffset += luTake;
            luSize -= luTake;
        }
        luPartStart = luPartEnd;
    }
    return luSize == 0;
}

// Fill stage of the pipelines that read the archive: the image range of a group, 8 MiB per task (laPartFds
// caches the part files' descriptors; the caller closes them).
arkpipe::Stage CArk::ReadGroupsStage(const std::vector<arkpipe::Group>& laGroups, std::vector<int>& laPartFds) const
{
    const uint64_t kuReadPiece = 8ull << 20;
    return arkpipe::Stage{
        [&laGroups, kuReadPiece](size_t gg) {
            return (int)std::max<uint64_t>(1, (laGroups[gg].srcHi - laGroups[gg].srcLo + kuReadPiece - 1) / kuReadPiece);
        },
        [this, &laGroups, &laPartFds, kuReadPiece](size_t gg, int tt, unsigned char* lpRange) {
            arkpipe::SlowOp lTimer("ExtractFiles read of an 8 MiB image piece");
            const arkpipe::Group& lGroup = laGroups[gg];
            const uint64_t luLo = (uint64_t)tt * kuReadPiece, luHi = std::min(lGroup.srcHi - lGroup.srcLo, luLo + kuReadPiece);
            if (luHi > luLo && !ReadImageRange(laPartFds, lGroup.srcLo + luLo, luHi - luLo, lpRange + luLo))
                return eError_FailedToOpenFile;
            return eError_NoError;
        }};
}

// Entries that lie (partly) outside the image of luImageSize bytes are refused, whatever reads the archive.
eError CArk::CheckEntriesInImage(uint64_t luImageSize) const
{
    for (const modark::FileDef& lFile : mHeader.maFiles) {
        if ((uint64_t)lFile.mi64Offset > luImageSize || (uint64_t)lFile.miSize > luImageSize - (uint64_t)lFile.mi64Offset) {
            std::cout << "Entry " << lFile.mName.c_str() << " lies outside the archive data\n";
            eError leError = eError_InvalidData;
            SHOW_ERROR_AND_RETURN;
        }
    }
    return eError_NoError;
}

// Extraction streams the archive through the slot-ring pipeline (ArkPipeline.h) instead of the
// reference's one archive-sized buffer (CArk.cpp:431, :738) and its serial one-file-at-a-time writes
// (:435-501): the entries, ordered by image offset, are packed back to back into a staging space, and
// the batched kernel gathers and deciphers each group of them there.  Entries that share an output name
// are resolved up front to the one whose bytes the reference's in-order loop would leave on disk.
eError CArk::ExtractFiles(int liFirstFileIndex, int liNumFiles, const char* lpTargetDirectory)
{
    (void)liFirstFileIndex;  // the reference ignores both and walks the whole table (CArk.cpp:435)
    (void)liNumFiles;
    if (mHeader.maFiles.empty())
        return eError_NoData;
    const std::string lTarget = lpTargetDirectory;

    uint64_t luImageSize = 0;
    for (const modark::PartDef& lPart : mHeader.maParts)
        luImageSize += lPart.muSize;

    const size_t liCount = mHeader.maFiles.size();
    eError leError = CheckEntriesInImage(luImageSize);
    ERROR_RETURN;

    // Duplicate output names.  The reference writes in table order, one file at a time (CArk.cpp:435-501):
    // with overwriting on (the default) the LAST entry of a name is what stays on disk; with it off a
    // file is only rewritten while it is still empty, so the FIRST non-empty entry stays.  Resolve that
    // here so that exactly one entry per name is extracted, whatever order the pipeline writes in.
    std::vector<uint32_t> laWinners;
    {
        std::unordered_map<std::string, uint32_t> lByName;  // name -> position in laWinners
        laWinners.reserve(liCount);
        for (size_t ii = 0; ii < liCount; ++ii) {
            const modark::FileDef& lFile = mHeader.maFiles[ii];
            const auto lFound = lByName.find(lFile.mName);
            if (lFound == lByName.end()) {
                lByName.emplace(lFile.mName, (uint32_t)laWinners.size());
                laWinners.push_back((uint32_t)ii);
                continue;
            }
            uint32_t& luWinner = laWinners[lFound->second];
            if (CSettings::mbOverwriteOutputFiles || mHeader.maFiles[luWinner].miSize == 0)
                luWinner = (uint32_t)ii;
            VERBOSE_OUT("Duplicate entry " << lFile.mName.c_str() << "\n");
        }
    }

    // order by where the entries sit in the image
    std::vector<uint32_t> laOrder = laWinners;
    std::stable_sort(laOrder.begin(), laOrder.end(), [&](uint32_t a, uint32_t b) {
        return mHeader.maFiles[a].mi64Offset < mHeader.maFiles[b].mi64Offset;
    });
    const uint64_t kuGroupBytes = arkpipe::GroupBytes();
    std::vector<arkpipe::Piece> laPieces;
    std::vector<mod_desc> laDescs;
    laPieces.reserve(laOrder.size());
    laDescs.reserve(laOrder.size());
    uint64_t luStaged = 0;
    for (uint32_t luFile : laOrder) {
        const modark::FileDef& lFile = mHeader.maFiles[luFile];
        arkpipe::CutEntry(luFile, (uint64_t)lFile.miSize, (uint64_t)lFile.mi64Offset, luStaged, EntryKey(luFile), kuGroupBytes, 0,
                          laPieces, laDescs);
        luStaged += (uint64_t)lFile.miSize;
    }
    const std::vector<arkpipe::Group> laGroups = arkpipe::GroupPieces(laDescs, kuGroupBytes);
    auto lInPieces = [&](const arkpipe::Piece& lPiece) { return lPiece.size != (uint32_t)mHeader.maFiles[lPiece.file].miSize; };

    // files that arrive in several pieces are created (and emptied) up front, so that the pieces -- written by
    // whichever threads get them, in any order -- only ever pwrite into an existing file
    std::vector<uint8_t> laSkipFile(liCount, 0);
    for (const arkpipe::Piece& lPiece : laPieces) {
        if (!lInPieces(lPiece) || lPiece.fileOffset != 0)
            continue;
        const modark::FileDef& lFile = mHeader.maFiles[lPiece.file];
        const std::string lOutputPath = lTarget + lFile.mName;
        laSkipFile[lPiece.file] = 1;
        if (EscapesTarget(lFile.mName)) {
            std::cout << "Refusing to write outside the target directory: " << lFile.mName.c_str() << "\n";
        } else if (KeepExistingOutput(lOutputPath)) {
            VERBOSE_OUT("Output file already exists, skipping: " << lOutputPath.c_str() << "\n");
        } else if (!MakeParentDirectories(lOutputPath)) {
            eError leError = eError_FailedToCreateDirectory;
            SHOW_ERROR_AND_RETURN;
        } else {
            const int liFd = open(lOutputPath.c_str(), O_WRONLY | O_CREAT | O_TRUNC, 0666);
            if (liFd < 0) {
                std::cout << "Failed to create " << lOutputPath.c_str() << "\n";
            } else {
                close(liFd);
                laSkipFile[lPiece.file] = 0;
            }
        }
    }

    std::vector<int> laPartFds(mHeader.maParts.size(), -1);
    const arkpipe::Stage lRead = ReadGroupsStage(laGroups, laPartFds);

    // drain: the files of a group, 48 per task
    const size_t kiFilesPerTask = 48;
    const arkpipe::Stage lWrite{
        [&](size_t gg) { return (int)((laGroups[gg].last - laGroups[gg].first + kiFilesPerTask - 1) / kiFilesPerTask); },
        [&](size_t gg, int tt, unsigned char* lpStaged) {
            thread_local std::unordered_set<std::string> lKnownDirectories;
            arkpipe::SlowOp lTimer("ExtractFiles writer task (up to 48 files)");
            const arkpipe::Group& lGroup = laGroups[gg];
            const size_t liFrom = lGroup.first + (size_t)tt * kiFilesPerTask, liTo = std::min(lGroup.last, liFrom + kiFilesPerTask);
            for (size_t ii = liFrom; ii < liTo; ++ii) {
                const arkpipe::Piece& lPiece = laPieces[ii];
                const modark::FileDef& lFile = mHeader.maFiles[lPiece.file];
                const std::string lOutputPath = lTarget + lFile.mName;
                const unsigned char* lpBytes = lpStaged + (laDescs[ii].dst_off - lGroup.dstLo);
                if (lInPieces(lPiece)) {  // one piece of a big file that was created up front
                    if (laSkipFile[lPiece.file])
                        continue;
                    const int liFd = open(lOutputPath.c_str(), O_WRONLY);
                    const bool lbOk = liFd >= 0 && WriteFully(liFd, lpBytes, lPiece.size, lPiece.fileOffset);
                    if (liFd >= 0)
                        close(liFd);
                    if (!lbOk)
                        return eError_FailedToWriteData;
                    continue;
                }
                if (EscapesTarget(lFile.mName)) {
                    std::cout << "Refusing to write outside the target directory: " << lFile.mName.c_str() << "\n";
                    continue;
                }
                if (KeepExistingOutput(lOutputPath)) {
                    VERBOSE_OUT("Output file already exists, skipping: " << lOutputPath.c_str() << "\n");
                    continue;
                }
                if (!MakeParentDirectoriesCached(lOutputPath, lKnownDirectories))
                    return eError_FailedToCreateDirectory;
                const int liFd = open(lOutputPath.c_str(), O_WRONLY | O_CREAT | O_TRUNC, 0666);
                if (liFd < 0) {
                    std::cout << "Failed to create " << lOutputPath.c_str() << "\n";  // the reference carries on too (CArk.cpp:488-491)
                    continue;
                }
                const bool lbOk = lFile.miSize == 0 || WriteFully(liFd, lpBytes, (uint64_t)lFile.miSize, 0);
                close(liFd);
                if (!lbOk)
                    return eError_FailedToWriteData;
            }
            return eError_NoError;
        }};

    const int liCores = arkpipe::HostThreads();
    leError = arkpipe::RunPipeline("extract", laDescs, laGroups, luImageSize, luStaged, true, std::max(2, std::min(8, liCores / 4)),
                                          std::max(4, std::min(16, liCores / 2)), lRead, arkpipe::CipherStep(), lWrite);
    for (int liFd : laPartFds)
        if (liFd >= 0)
            close(liFd);
    if (leError == eError_NoData)  // the GPU could not be set up; RunPipeline has said why
        return leError;
    SHOW_ERROR_AND_RETURN;
    return eError_NoError;
}

// What a search launch gets for one group: the slot's plan, stream and device buffers, the group's tiles and
// source window, and the device's result arrays.
struct CArk::SearchSlot {
    size_t miDeviceIndex;
    mod_plan* mpPlan;
    uint64_t muTile0, muTile1;
    const void* mpDevIn;       // the group's source range
    uint64_t muSrcLo, muRange;
    uint32_t* mpCounts;        // per descriptor
    const uint32_t* mpOwned;   // per descriptor: starts the piece owns
    uint64_t* mpPatternCounts;
    void* mpList;              // muCap records
    uint64_t muCap;
    uint64_t* mpTotal;
    void* mpStream;
};

// One search over the parts: pieces of big entries overlap by muOverlap bytes; each group's list holds records of
// muRecordBytes, the first 8 bytes {descriptor, position}; mLaunch enqueues the kernel for one group.
struct CArk::SearchPass {
    uint32_t muOverlap;
    size_t miPatterns;  // per-pattern counts kept (0: none)
    uint64_t muMaxMatches;
    uint64_t muRecordBytes;
    std::function<bool(const SearchSlot&)> mLaunch;
    std::function<void(uint32_t luFile, uint32_t luOffset, const unsigned char* lpRecord)> mCollect;  // under a lock
};

// The search reads the parts like ExtractFiles, but the GPU step deciphers and matches instead of storing: only
// each group's short match list comes back over PCIe, and nothing is written.  Entries are searched in image
// order, pieces of big entries overlapping by Lmax - 1 bytes (CutEntry), and every entry is searched, also
// when another one has the same name.  Each piece but an entry's last owns the starts before the next piece's
// first byte (the owned-start bounds): a pattern shorter than Lmax that starts in the overlap is the next piece's.
eError CArk::SearchParts(const SearchPass& lPass, std::vector<uint64_t>& laFileCounts, std::vector<uint64_t>& laPatternCounts)
{
    if (mHeader.maFiles.empty())
        return eError_NoData;
    uint64_t luImageSize = 0;
    for (const modark::PartDef& lPart : mHeader.maParts)
        luImageSize += lPart.muSize;
    eError leError = CheckEntriesInImage(luImageSize);
    ERROR_RETURN;

    const size_t liCount = mHeader.maFiles.size();
    std::vector<uint32_t> laOrder(liCount);
    for (size_t ii = 0; ii < liCount; ++ii)
        laOrder[ii] = (uint32_t)ii;
    std::stable_sort(laOrder.begin(), laOrder.end(), [&](uint32_t a, uint32_t b) {
        return mHeader.maFiles[a].mi64Offset < mHeader.maFiles[b].mi64Offset;
    });
    const uint64_t kuGroupBytes = arkpipe::GroupBytes();
    std::vector<arkpipe::Piece> laPieces;
    std::vector<mod_desc> laDescs;  // dst_off == src_off: the plan's chunk grid lies on the image
    for (uint32_t luFile : laOrder) {
        const modark::FileDef& lFile = mHeader.maFiles[luFile];
        arkpipe::CutEntry(luFile, (uint64_t)lFile.miSize, (uint64_t)lFile.mi64Offset, (uint64_t)lFile.mi64Offset, EntryKey(luFile),
                          kuGroupBytes, lPass.muOverlap, laPieces, laDescs);
    }
    const std::vector<arkpipe::Group> laGroups = arkpipe::GroupPieces(laDescs, kuGroupBytes);
    uint64_t luCap = 0;  // list slots per group: a group cannot hold more matches than it has bytes
    for (const arkpipe::Group& lGroup : laGroups)
        luCap = std::max(luCap, std::min<uint64_t>(lPass.muMaxMatches, lGroup.dstHi - lGroup.dstLo));
    const uint64_t luListBytes = 16 + lPass.muRecordBytes * luCap;  // total (8 bytes), 8 spare, the list

    // Per device, one array of [counts per descriptor | owned starts per descriptor | counts per pattern], set up on
    // the device's first group from laInit.
    const size_t liDescs = laDescs.size();
    std::vector<uint32_t> laInit(2 * liDescs + 2 * lPass.miPatterns, 0);
    for (size_t ii = 0; ii < liDescs; ++ii) {
        const bool lbNext = ii + 1 < liDescs && laPieces[ii + 1].file == laPieces[ii].file && laPieces[ii + 1].fileOffset != 0;
        laInit[liDescs + ii] = lbNext ? (uint32_t)(laPieces[ii + 1].fileOffset - laPieces[ii].fileOffset) : laPieces[ii].size;
    }
    struct DeviceCounts {
        int miDevice = -1;
        uint32_t* mpCounts = nullptr;
    };
    std::vector<DeviceCounts> laCounts(64);
    arkpipe::GpuStep lFind;
    lFind.muOutBytes = luListBytes;
    lFind.mEnqueue = [&](const arkpipe::Group& lGroup, const arkpipe::SlotView& lSlot) {
        DeviceCounts& lCounts = laCounts[lSlot.miDeviceIndex];
        if (!lCounts.mpCounts) {
            lCounts.miDevice = mod_current_device();
            lCounts.mpCounts = (uint32_t*)mod_device_alloc(4 * laInit.size());
            if (!lCounts.mpCounts || mod_memcpy_h2d(lCounts.mpCounts, laInit.data(), 4 * laInit.size(), lSlot.mpStream) != MOD_OK ||
                mod_stream_sync(lSlot.mpStream) != MOD_OK)
                return false;
        }
        const uint64_t luRange = lGroup.srcHi - lGroup.srcLo;
        unsigned char* lpDevIn = (unsigned char*)lSlot.mpDevIn + (lGroup.srcLo & 15u);
        unsigned char* lpList = lSlot.mpHostOut + (lGroup.dstLo & 15u);
        std::memset(lpList, 0, 16);
        SearchSlot lSearch{lSlot.miDeviceIndex, lSlot.mpPlan, 0, 0, lpDevIn, lGroup.srcLo, luRange, lCounts.mpCounts,
                           lCounts.mpCounts + liDescs, (uint64_t*)(lCounts.mpCounts + 2 * liDescs),
                           (unsigned char*)lSlot.mpDevOut + 16, luCap, (uint64_t*)lSlot.mpDevOut, lSlot.mpStream};
        return mod_plan_tile_range(lSlot.mpPlan, lGroup.first, lGroup.last, &lSearch.muTile0, &lSearch.muTile1) == MOD_OK &&
               mod_memcpy_h2d(lSlot.mpDevOut, lpList, 16, lSlot.mpStream) == MOD_OK &&
               mod_memcpy_h2d(lpDevIn, lSlot.mpHostIn + (lGroup.srcLo & 15u), luRange, lSlot.mpStream) == MOD_OK &&
               lPass.mLaunch(lSearch) && mod_memcpy_d2h(lpList, lSlot.mpDevOut, luListBytes, lSlot.mpStream) == MOD_OK;
    };

    // drain: the group's list, as (file, offset in the entry)
    std::mutex lMutex;
    const arkpipe::Stage lCollect{
        [&](size_t gg) { return laGroups[gg].dstHi > laGroups[gg].dstLo ? 1 : 0; },
        [&](size_t, int, unsigned char* lpList) {
            uint64_t luTotal = 0;
            std::memcpy(&luTotal, lpList, 8);
            const uint64_t luKept = std::min(luTotal, luCap);
            std::lock_guard<std::mutex> lLock(lMutex);
            for (uint64_t kk = 0; kk < luKept; ++kk) {
                const unsigned char* lpRecord = lpList + 16 + lPass.muRecordBytes * kk;
                mod_match lMatch;
                std::memcpy(&lMatch, lpRecord, sizeof(lMatch));
                const arkpipe::Piece& lPiece = laPieces[lMatch.desc];
                lPass.mCollect(lPiece.file, (uint32_t)(lPiece.fileOffset + lMatch.pos), lpRecord);
            }
            return eError_NoError;
        }};

    std::vector<int> laPartFds(mHeader.maParts.size(), -1);
    const int liOriginalDevice = mod_current_device();
    const int liCores = arkpipe::HostThreads();
    leError = arkpipe::RunPipeline("find", laDescs, laGroups, luImageSize, luImageSize, true, std::max(2, std::min(8, liCores / 4)), 2,
                                   ReadGroupsStage(laGroups, laPartFds), lFind, lCollect);
    for (int liFd : laPartFds)
        if (liFd >= 0)
            close(liFd);

    // exact counts: the devices' arrays, summed per entry and per pattern
    laFileCounts.assign(liCount, 0);
    laPatternCounts.assign(lPass.miPatterns, 0);
    std::vector<uint32_t> laDescCounts(liDescs);
    std::vector<uint64_t> laDevicePatternCounts(lPass.miPatterns);
    for (DeviceCounts& lCounts : laCounts) {
        if (!lCounts.mpCounts)
            continue;
        if (leError == eError_NoError &&
            (mod_init(lCounts.miDevice) != MOD_OK || mod_memcpy_d2h(laDescCounts.data(), lCounts.mpCounts, 4 * liDescs, nullptr) != MOD_OK ||
             mod_memcpy_d2h(laDevicePatternCounts.data(), lCounts.mpCounts + 2 * liDescs, 8 * lPass.miPatterns, nullptr) != MOD_OK ||
             mod_stream_sync(nullptr) != MOD_OK)) {
            std::cout << "GPU find failed: " << mod_last_error() << "\n";
            leError = eError_InvalidData;
        }
        for (size_t ii = 0; ii < liDescs && leError == eError_NoError; ++ii)
            laFileCounts[laPieces[ii].file] += laDescCounts[ii];
        for (size_t jj = 0; jj < lPass.miPatterns && leError == eError_NoError; ++jj)
            laPatternCounts[jj] += laDevicePatternCounts[jj];
        mod_device_free(lCounts.mpCounts);
    }
    if (liOriginalDevice >= 0)
        mod_init(liOriginalDevice);
    if (leError == eError_NoData)  // the GPU could not be set up; RunPipeline has said why
        return leError;
    SHOW_ERROR_AND_RETURN;
    return eError_NoError;
}

eError CArk::FindInFiles(const unsigned char* lpPattern, uint32_t luLen, uint64_t luMaxMatches, std::vector<SFileMatch>& laMatches,
                         uint64_t* lpTotal, std::vector<uint64_t>* lpFileCounts)
{
    return FindOneInFiles(lpPattern, nullptr, luLen, luMaxMatches, laMatches, lpTotal, lpFileCounts);
}

eError CArk::FindMaskedInFiles(const unsigned char* lpPattern, const unsigned char* lpMask, uint32_t luLen, uint64_t luMaxMatches,
                               std::vector<SFileMatch>& laMatches, uint64_t* lpTotal, std::vector<uint64_t>* lpFileCounts)
{
    laMatches.clear();
    if (!lpMask || std::all_of(lpMask, lpMask + std::min<uint32_t>(luLen, 64), [](unsigned char c) { return c == 0; }))
        return eError_InvalidParameter;
    return FindOneInFiles(lpPattern, lpMask, luLen, luMaxMatches, laMatches, lpTotal, lpFileCounts);
}

eError CArk::FindOneInFiles(const unsigned char* lpPattern, const unsigned char* lpMask, uint32_t luLen, uint64_t luMaxMatches,
                            std::vector<SFileMatch>& laMatches, uint64_t* lpTotal, std::vector<uint64_t>* lpFileCounts)
{
    laMatches.clear();
    if (!lpPattern || luLen == 0 || luLen > 64 || !lpTotal)
        return eError_InvalidParameter;
    *lpTotal = 0;
    if (!mod_plan_find_window) {
        std::cout << "The GPU library in use has no search (mod_plan_find_window)\n";
        return eError_NoData;
    }
    if (lpMask && !mod_plan_find_masked_window) {
        std::cout << "The GPU library in use has no masked search (mod_plan_find_masked_window)\n";
        return eError_NoData;
    }
    SearchPass lPass;
    lPass.muOverlap = luLen - 1;
    lPass.miPatterns = 0;
    lPass.muMaxMatches = luMaxMatches;
    lPass.muRecordBytes = sizeof(mod_match);
    lPass.mLaunch = [&](const SearchSlot& lSlot) {
        if (lpMask)
            return mod_plan_find_masked_window(lSlot.mpPlan, lSlot.muTile0, lSlot.muTile1, lSlot.mpDevIn, lSlot.muSrcLo, lSlot.muRange,
                                               lpPattern, lpMask, luLen, lSlot.mpCounts, (mod_match*)lSlot.mpList, lSlot.muCap,
                                               lSlot.mpTotal, lSlot.mpStream) == MOD_OK;
        return mod_plan_find_window(lSlot.mpPlan, lSlot.muTile0, lSlot.muTile1, lSlot.mpDevIn, lSlot.muSrcLo, lSlot.muRange, lpPattern,
                                    luLen, lSlot.mpCounts, (mod_match*)lSlot.mpList, lSlot.muCap, lSlot.mpTotal, lSlot.mpStream) == MOD_OK;
    };
    lPass.mCollect = [&](uint32_t luFile, uint32_t luOffset, const unsigned char*) {
        laMatches.push_back(SFileMatch{(int)luFile, luOffset});
    };
    std::vector<uint64_t> laFileCounts, laPatternCounts;
    const eError leError = SearchParts(lPass, laFileCounts, laPatternCounts);
    if (leError != eError_NoError)
        return leError;
    for (uint64_t luCount : laFileCounts)
        *lpTotal += luCount;
    std::sort(laMatches.begin(), laMatches.end(),
              [](const SFileMatch& a, const SFileMatch& b) { return a.file != b.file ? a.file < b.file : a.offset < b.offset; });
    if (laMatches.size() > luMaxMatches)
        laMatches.resize((size_t)luMaxMatches);
    if (lpFileCounts)
        *lpFileCounts = std::move(laFileCounts);
    return eError_NoError;
}

eError CArk::FindSetInFiles(const std::vector<std::string>& laPatterns, uint64_t luMaxMatches, std::vector<SFileSetMatch>& laMatches,
                            uint64_t* lpTotal, std::vector<uint64_t>* lpFileCounts, std::vector<uint64_t>* lpPatternCounts,
                            bool lbIgnoreCase)
{
    laMatches.clear();
    if (laPatterns.empty() || laPatterns.size() > 256 || !lpTotal)
        return eError_InvalidParameter;
    std::string lBytes;
    std::vector<uint32_t> laLens;
    uint32_t luMax = 0;
    for (const std::string& lPattern : laPatterns) {
        if (lPattern.empty() || lPattern.size() > 64)
            return eError_InvalidParameter;
        lBytes += lPattern;
        laLens.push_back((uint32_t)lPattern.size());
        luMax = std::max(luMax, (uint32_t)lPattern.size());
    }
    std::unordered_set<std::string> lDistinct;
    for (std::string lPattern : laPatterns) {
        if (lbIgnoreCase)
            for (char& c : lPattern)
                c = (char)(c >= 'a' && c <= 'z' ? c - 0x20 : c);
        lDistinct.insert(std::move(lPattern));
    }
    if (lDistinct.size() != laPatterns.size())
        return eError_InvalidParameter;
    *lpTotal = 0;
    if (!mod_plan_find_set_window || !mod_pattern_set_create || !mod_pattern_set_destroy) {
        std::cout << "The GPU library in use has no set search (mod_plan_find_set_window)\n";
        return eError_NoData;
    }
    if (lbIgnoreCase && !mod_pattern_set_create_nocase) {
        std::cout << "The GPU library in use has no case-insensitive set search (mod_pattern_set_create_nocase)\n";
        return eError_NoData;
    }
    const auto lCreate = lbIgnoreCase ? mod_pattern_set_create_nocase : mod_pattern_set_create;
    std::vector<mod_pattern_set*> laSets(64, nullptr);  // one per device, created on its first group
    SearchPass lPass;
    lPass.muOverlap = luMax - 1;
    lPass.miPatterns = laPatterns.size();
    lPass.muMaxMatches = luMaxMatches;
    lPass.muRecordBytes = sizeof(mod_set_match);
    lPass.mLaunch = [&](const SearchSlot& lSlot) {
        mod_pattern_set*& lpSet = laSets[lSlot.miDeviceIndex];
        if (!lpSet && lCreate((const uint8_t*)lBytes.data(), laLens.data(), (uint32_t)laLens.size(), &lpSet) != MOD_OK)
            return false;
        return mod_plan_find_set_window(lSlot.mpPlan, lSlot.muTile0, lSlot.muTile1, lSlot.mpDevIn, lSlot.muSrcLo, lSlot.muRange, lpSet,
                                        lSlot.mpOwned, lSlot.mpCounts, lSlot.mpPatternCounts, (mod_set_match*)lSlot.mpList, lSlot.muCap,
                                        lSlot.mpTotal, lSlot.mpStream) == MOD_OK;
    };
    lPass.mCollect = [&](uint32_t luFile, uint32_t luOffset, const unsigned char* lpRecord) {
        mod_set_match lMatch;
        std::memcpy(&lMatch, lpRecord, sizeof(lMatch));
        laMatches.push_back(SFileSetMatch{(int)luFile, luOffset, lMatch.pattern});
    };
    std::vector<uint64_t> laFileCounts, laPatternCounts;
    const eError leError = SearchParts(lPass, laFileCounts, laPatternCounts);
    for (mod_pattern_set* lpSet : laSets)
        mod_pattern_set_destroy(lpSet);
    if (leError != eError_NoError)
        return leError;
    for (uint64_t luCount : laFileCounts)
        *lpTotal += luCount;
    std::sort(laMatches.begin(), laMatches.end(), [](const SFileSetMatch& a, const SFileSetMatch& b) {
        return a.file != b.file ? a.file < b.file : a.offset != b.offset ? a.offset < b.offset : a.pattern < b.pattern;
    });
    if (laMatches.size() > luMaxMatches)
        laMatches.resize((size_t)luMaxMatches);
    if (lpFileCounts)
        *lpFileCounts = std::move(laFileCounts);
    if (lpPatternCounts)
        *lpPatternCounts = std::move(laPatternCounts);
    return eError_NoError;
}

// ---- write side --------------------------------------------------------------------------------------

bool CArk::ShouldPackFile(const std::vector<SSongConfig>& laSongs, const char* lpFilename) const
{
    // Files under ".../songs/<name>/" are packed only when <name> occurs in some configured song
    // path; everything else always is (policy of the reference, CArk.cpp:58-92).
    const char* lpSongs = std::strstr(lpFilename, "/songs/");
    if (!lpSongs)
        return true;
    const char* lpEnd = lpSongs + std::strlen("/songs/");
    while (*lpEnd && *lpEnd != '/')
        ++lpEnd;
    if (!*lpEnd)
        return false;
    std::string lSongName(lpSongs, lpEnd - lpSongs);
    std::transform(lSongName.begin(), lSongName.end(), lSongName.begin(), [](unsigned char c) { return (char)std::tolower(c); });
    for (const SSongConfig& lSong : laSongs)
        if (lSong.mPath.find(lSongName) != std::string::npos)
            return true;
    return false;
}

eError CArk::ConstructFromDirectory(const char* lpInputDirectory, const CArk& lReferenceHeader, std::vector<SSongConfig> laSongs)
{
    for (const char* lpAlways : {"/songs/credits", "/songs/tut0", "/songs/tut1", "/songs/tutc"}) {
        SSongConfig lSong;
        lSong.mPath = lpAlways;
        laSongs.push_back(lSong);
    }

    std::string lRoot = lpInputDirectory;
    if (!lRoot.empty() && lRoot.back() != '/')
        lRoot += '/';
    std::vector<std::string> laFilenames;
    ListFiles(lRoot, "", laFilenames);
    if (laFilenames.empty()) {
        eError leError = eError_NoData;
        SHOW_ERROR_AND_RETURN;
    }
    VERBOSE_OUT("Found " << laFilenames.size() << " files\n");

    mHeader = modark::HeaderImage();
    mHeader.mbPS4 = CSettings::mbPS4;
    uint64_t luTotalFileSize = 0;
    // name -> FIRST entry of that name in the reference header (the reference scans linearly for the first
    // match of the name hash, CArk.cpp:1194-1209)
    std::unordered_map<std::string, const modark::FileDef*> lReferenceByName;
    lReferenceByName.reserve(lReferenceHeader.mHeader.maFiles.size());
    for (const modark::FileDef& lCandidate : lReferenceHeader.mHeader.maFiles)
        lReferenceByName.emplace(lCandidate.mName, &lCandidate);
    for (const std::string& lFilename : laFilenames) {
        const auto lFound = lReferenceByName.find(lFilename);
        const modark::FileDef* lpReference = lFound == lReferenceByName.end() ? nullptr : lFound->second;
        if (!lpReference && CSettings::mbIgnoreNewFiles)
            continue;  // only files the reference header knows are repacked (-pack); -pack_add lifts this
        if (!CSettings::mbPackAllFiles && !ShouldPackFile(laSongs, lFilename.c_str()))
            continue;
        const long liSize = FileSize(lRoot + lFilename);
        if (liSize < 0) {
            std::cout << "Unable to open file: " << lFilename.c_str() << "\n";
            continue;
        }
        modark::FileDef lFile = lpReference ? *lpReference : modark::FileDef();
        lFile.mName = lFilename;
        lFile.miSize = (int)liSize;
        luTotalFileSize += (uint64_t)liSize;
        mHeader.maFiles.push_back(lFile);
    }
    if (mHeader.maFiles.empty()) {
        eError leError = eError_NoData;
        SHOW_ERROR_AND_RETURN;
    }

    // part plan: the reference header's part list, each part allowed an equal share of what is left
    mHeader.maParts = lReferenceHeader.mHeader.maParts;
    uint64_t luSizeRemaining = luTotalFileSize;
    const size_t liNumArks = mHeader.maParts.size();
    for (size_t ii = 0; ii < liNumArks; ++ii) {
        mHeader.maParts[ii].muSize = (unsigned int)(luSizeRemaining / (liNumArks - ii));
        luSizeRemaining -= mHeader.maParts[ii].muSize;
    }
    mbLoaded = true;
    return eError_NoError;
}

// BuildArk assigns every entry its byte-packed offset and closes the parts (reference CArk.cpp:760-828)
// from the SIZES alone; the payload itself is never gathered into one archive-sized buffer
// (CArk.cpp:769-811 does): SaveArk streams it from the input files straight into the part files.
eError CArk::BuildArk(const char* lpInputDirectory, std::vector<SSongConfig> laSongs)
{
    (void)laSongs;  // the reference appends its four defaults and never reads them here (CArk.cpp:762-765)
    VERBOSE_OUT("Building ark\n");
    if (mHeader.maParts.empty())
        return eError_NoData;
    ReleaseArkData();
    mBuildInputDirectory = lpInputDirectory;

    size_t liArkIndex = 0;
    int64_t li64Allowed = mHeader.maParts[0].muSize;
    uint64_t luPtr = 0, luPartStart = 0;
    for (size_t ii = 0; ii < mHeader.maFiles.size(); ++ii) {
        modark::FileDef& lFile = mHeader.maFiles[ii];
        if (lFile.miSize == 0) {
            lFile.mi64Offset = 0;
            continue;
        }
        // the reference opens (and reads) the file here and gives up on the first one it cannot open
        if (access((mBuildInputDirectory + lFile.mName).c_str(), R_OK) != 0) {
            eError leError = eError_FailedToOpenFile;
            SHOW_ERROR_AND_RETURN;
        }
        // scatter: the file lands at the running, byte-packed offset
        lFile.mi64Offset = (int64_t)luPtr;
        luPtr += (uint64_t)lFile.miSize;

        // a part closes once it EXCEEDS its allowance; the overshoot shortens the next allowance
        if ((int64_t)(luPtr - luPartStart) > li64Allowed) {
            const unsigned int liArkSize = (unsigned int)(luPtr - luPartStart);
            mHeader.maParts[liArkIndex].muSize = liArkSize;
            if (liArkIndex + 1 >= mHeader.maParts.size()) {
                // the reference would index past mpArks here (CArk.cpp:817-818); grow a part instead
                modark::PartDef lExtra = mHeader.maParts[liArkIndex];
                lExtra.mPath += ".extra";
                lExtra.muSize = 0;
                mHeader.maParts.push_back(lExtra);
            }
            ++liArkIndex;
            li64Allowed += (int64_t)mHeader.maParts[liArkIndex].muSize - (int64_t)liArkSize;
            luPartStart = luPtr;
        }
    }
    mHeader.maParts[liArkIndex].muSize = (unsigned int)(luPtr - luPartStart);
    muBuiltImageSize = luPtr;
    mbBuilt = true;
    VERBOSE_OUT("Ark built\n");
    return eError_NoError;
}

// Stream the image BuildArk laid out into the part files through the slot-ring pipeline (ArkPipeline.h):
// reader threads load the input files of a ~32 MiB group, entries that carry a key are ciphered on the
// GPU, writer threads pwrite the group's byte range into the part file(s) it falls in.  With all keys 0
// (the reference never ciphers ARK bodies) the GPU is not involved and the bytes go from the read buffer
// straight to the part files.
eError CArk::StreamBuiltImage(const std::vector<PartTarget>& laTargets) const
{
    // non-empty entries in table order == image order, which is also where they go: destination == source
    const uint64_t kuGroupBytes = arkpipe::GroupBytes();
    std::vector<arkpipe::Piece> laPieces;
    std::vector<mod_desc> laDescs;
    bool lbAnyKey = false;
    for (size_t ii = 0; ii < mHeader.maFiles.size(); ++ii) {
        const modark::FileDef& lFile = mHeader.maFiles[ii];
        if (lFile.miSize == 0)
            continue;
        const int liKey = EntryKey(ii);
        lbAnyKey = lbAnyKey || (liKey % 0x7FFFFFFF) != 0;
        arkpipe::CutEntry((uint32_t)ii, (uint64_t)lFile.miSize, (uint64_t)lFile.mi64Offset, (uint64_t)lFile.mi64Offset, liKey,
                          kuGroupBytes, 0, laPieces, laDescs);
    }
    if (laPieces.empty())
        return eError_NoError;
    const std::vector<arkpipe::Group> laGroups = arkpipe::GroupPieces(laDescs, kuGroupBytes);

    // each group's range, cut into 4 MiB writes (several writer threads share a group) per part file that
    // receives it; none when every part the group falls in was skipped (existing output kept)
    struct Range {
        size_t target;
        uint64_t lo, hi;
    };
    std::vector<std::vector<Range>> laRanges(laGroups.size());
    const uint64_t kuWritePiece = 4ull << 20;
    for (size_t gg = 0; gg < laGroups.size(); ++gg)
        for (size_t tt = 0; tt < laTargets.size(); ++tt) {
            const uint64_t luLo = std::max(laGroups[gg].dstLo, laTargets[tt].muImageStart);
            const uint64_t luHi = std::min(laGroups[gg].dstHi, laTargets[tt].muImageStart + laTargets[tt].muSize);
            if (laTargets[tt].miFd < 0)
                continue;
            for (uint64_t luAt = luLo; luAt < luHi; luAt += kuWritePiece)
                laRanges[gg].push_back(Range{tt, luAt, std::min(luHi, luAt + kuWritePiece)});
        }

    // fill: the input files of a group, 48 per task (the reference's one fread per file, CArk.cpp:796-811 --
    // thousands of small files are latency-bound on any file system)
    const size_t kiFilesPerTask = 48;
    const arkpipe::Stage lRead{
        [&](size_t gg) { return (int)((laGroups[gg].last - laGroups[gg].first + kiFilesPerTask - 1) / kiFilesPerTask); },
        [&](size_t gg, int tt, unsigned char* lpRange) {
            arkpipe::SlowOp lTimer("SaveArk reader task (up to 48 input files)");
            const arkpipe::Group& lGroup = laGroups[gg];
            const size_t liFrom = lGroup.first + (size_t)tt * kiFilesPerTask, liTo = std::min(lGroup.last, liFrom + kiFilesPerTask);
            for (size_t ii = liFrom; ii < liTo; ++ii) {
                const arkpipe::Piece& lPiece = laPieces[ii];
                const int liFd = open((mBuildInputDirectory + mHeader.maFiles[lPiece.file].mName).c_str(), O_RDONLY);
                if (liFd < 0)
                    return eError_FailedToOpenFile;
                unsigned char* lpDst = lpRange + (laDescs[ii].src_off - lGroup.srcLo);
                const bool lbOk = ReadFully(liFd, lpDst, lPiece.size, lPiece.fileOffset);  // a file that shrank reads as zeros
                close(liFd);
                if (!lbOk)
                    return eError_FailedToOpenFile;
            }
            return eError_NoError;
        }};

    // drain: one 4 MiB range into its part file
    const arkpipe::Stage lWrite{
        [&](size_t gg) { return (int)laRanges[gg].size(); },
        [&](size_t gg, int tt, unsigned char* lpImage) {
            arkpipe::SlowOp lTimer("SaveArk writer task (a 4 MiB range)");
            const Range& lRange = laRanges[gg][tt];
            const PartTarget& lPart = laTargets[lRange.target];
            const unsigned char* lpBytes = lpImage + (lRange.lo - laGroups[gg].dstLo);
            if (lPart.mpMap) {  // pages of a mapped file are faulted in and filled by many threads at once
                std::memcpy(lPart.mpMap + (lRange.lo - lPart.muImageStart), lpBytes, (size_t)(lRange.hi - lRange.lo));
                return eError_NoError;
            }
            return WriteFully(lPart.miFd, lpBytes, lRange.hi - lRange.lo, lRange.lo - lPart.muImageStart) ? eError_NoError
                                                                                                      : eError_FailedToWriteData;
        }};

    const int liThreads = std::max(2, std::min(12, arkpipe::HostThreads() / 2));
    return arkpipe::RunPipeline("build", laDescs, laGroups, muBuiltImageSize, muBuiltImageSize, lbAnyKey, liThreads, liThreads, lRead,
                                arkpipe::CipherStep(), lWrite);
}

eError CArk::SaveArk(const char* lpOutputDirectory, const char* lpHeaderFilename) const
{
    // header: serialise on the host, encipher everything after the magic on the GPU, write
    std::vector<unsigned char> lImage = modark::SerialiseHeader(mHeader);
    CEncryptionCycler lEncrypt;
    lEncrypt.Cycle(lImage.data() + sizeof(uint32_t), (unsigned int)(lImage.size() - sizeof(uint32_t)),
                   (int)(mHeader.mbPS4 ? CSettings::kuEncryptedPS4Key : CSettings::kuEncryptedPS3Key));

    const std::string lHeaderPath = std::string(lpOutputDirectory) + lpHeaderFilename;
    if (KeepExistingOutput(lHeaderPath)) {
        VERBOSE_OUT("Output file already exists, skipping: " << lHeaderPath.c_str() << "\n");
    } else {
        MakeParentDirectories(lHeaderPath);
        VERBOSE_OUT("Writing " << lHeaderPath.c_str() << "\n");
        FILE* lpOutputFile = std::fopen(lHeaderPath.c_str(), "wb");
        if (lpOutputFile) {
            const size_t liWritten = std::fwrite(lImage.data(), 1, lImage.size(), lpOutputFile);
            std::fclose(lpOutputFile);
            if (liWritten != lImage.size()) {
                eError leError = eError_FailedToWriteData;
                SHOW_ERROR_AND_RETURN;
            }
        } else {
            std::cout << "Failed to open file for writing: " << lHeaderPath.c_str() << "\n";
        }
    }

    // parts: consecutive slices of the image.  Like the reference, the image cursor does not advance
    // past a part that is skipped because its output already exists (CArk.cpp:863-868) or cannot be
    // created (:880-897).
    std::vector<PartTarget> laTargets;
    uint64_t luCursor = 0;
    for (const modark::PartDef& lPart : mHeader.maParts) {
        const std::string lFilename = std::string(lpOutputDirectory) + lPart.mPath;
        if (KeepExistingOutput(lFilename)) {
            std::cout << "Output file already exists: " << lFilename.c_str() << "\n";
            continue;
        }
        std::cout << "Writing " << lFilename.c_str() << "\n";
        MakeParentDirectories(lFilename);
        PartTarget lTarget;
        lTarget.miFd = open(lFilename.c_str(), O_RDWR | O_CREAT | O_TRUNC, 0666);
        if (lTarget.miFd < 0) {
            std::cout << "Failed to open file for writing: " << lFilename.c_str() << "\n";
            continue;
        }
        lTarget.muImageStart = luCursor;
        lTarget.muSize = lPart.muSize;
        // size the file up front and map it: writer threads then fill disjoint ranges concurrently (write()
        // calls on one file serialise on its inode lock); if the mapping fails they fall back to pwrite
        if (mbBuilt && lPart.muSize && ftruncate(lTarget.miFd, (off_t)lPart.muSize) == 0) {
            void* lpMap = mmap(nullptr, lPart.muSize, PROT_READ | PROT_WRITE, MAP_SHARED, lTarget.miFd, 0);
            if (lpMap != MAP_FAILED)
                lTarget.mpMap = (unsigned char*)lpMap;
        }
        laTargets.push_back(lTarget);
        luCursor += lPart.muSize;
    }

    eError leError = eError_NoError;
    if (mbBuilt) {
        leError = StreamBuiltImage(laTargets);
    } else if (mpArkData) {  // a loaded image (Load + LoadArkData) saved again
        for (const PartTarget& lTarget : laTargets) {
            const uint64_t luTake = lTarget.muImageStart < muArkDataSize ? std::min<uint64_t>(lTarget.muSize, muArkDataSize - lTarget.muImageStart) : 0;
            if (luTake != lTarget.muSize || !WriteFully(lTarget.miFd, mpArkData + lTarget.muImageStart, luTake, 0))
                leError = eError_FailedToWriteData;
        }
    } else {
        for (const PartTarget& lTarget : laTargets)
            if (lTarget.muSize)
                leError = eError_FailedToWriteData;  // nothing to write the parts from
    }
    for (const PartTarget& lTarget : laTargets) {
        if (lTarget.mpMap)
            munmap(lTarget.mpMap, lTarget.muSize);
        close(lTarget.miFd);
    }
    SHOW_ERROR_AND_RETURN;
    return eError_NoError;
}
