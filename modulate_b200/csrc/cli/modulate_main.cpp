// modulate_main.cpp -- portable command line over the facade: the reference's archive commands
// (-ps3 -verbose -force -packall -unpack -pack -pack_add -decode; Modulate.cpp:45-70, :291-317,
// :380-502, :895-972) with the same left-to-right command deque and exit convention.  -pack reads
// the song list from the DTA configs like the reference; the song-list EDITING commands of the
// reference are host-side tooling outside the hot path and are not provided.
//
// Extensions: -bodykey K (cipher every entry body with key K, stream restarting per entry -- the
// synthetic per-entry-key configurations), -device N (bind GPU N), -find TEXT / -findhex HEX (which
// entries hold a byte pattern, searched on the GPU without unpacking), -findlist FILE / -findhexlist FILE
// (the same for a list of patterns, all found in one pass), -findi TEXT / -findilist FILE (ignoring ASCII
// case) and -findwild HEX (hex with '?' nibbles that match anything).
#include <algorithm>
#include <cctype>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <fstream>
#include <functional>
#include <iostream>
#include <string>
#include <strings.h>
#include <unordered_map>
#include <vector>

#include "../../../include/modulate_b200.h"
#include "../CArk.h"
#include "../CDtaFile.h"
#include "../CEncryptionCycler.h"
#include "../Error.h"
#include "../Settings.h"

namespace {

int giBodyKey = 0;

std::string HeaderName() { return std::string("main_") + CSettings::msPlatform + ".hdr"; }

void WithSlash(std::string& lPath)
{
    if (lPath.empty() || (lPath.back() != '/' && lPath.back() != '\\'))
        lPath += "/";
}

eError PS3(std::deque<std::string>&)
{
    CSettings::mbPS4 = false;
    CSettings::msPlatform = "ps3";
    return eError_NoError;
}

eError EnableVerbose(std::deque<std::string>&)
{
    CSettings::mbVerbose = true;
    return eError_NoError;
}

eError EnableForceWrite(std::deque<std::string>&)
{
    CSettings::mbOverwriteOutputFiles = true;
    return eError_NoError;
}

eError EnablePackAll(std::deque<std::string>&)
{
    CSettings::mbPackAllFiles = true;
    return eError_NoError;
}

eError BodyKey(std::deque<std::string>& laParams)
{
    if (laParams.empty())
        return eError_InvalidParameter;
    giBodyKey = (int)std::strtoll(laParams.front().c_str(), nullptr, 0);
    laParams.pop_front();
    return eError_NoError;
}

eError Device(std::deque<std::string>& laParams)
{
    if (laParams.empty())
        return eError_InvalidParameter;
    const int liDevice = std::atoi(laParams.front().c_str());
    laParams.pop_front();
    if (mod_init(liDevice) != MOD_OK) {
        std::cout << mod_last_error() << "\n";
        return eError_InvalidParameter;
    }
    return eError_NoError;
}

eError Unpack(std::deque<std::string>& laParams)
{
    std::cout << "Unpacking " << HeaderName() << " to ";
    if (laParams.empty())
        return eError_InvalidParameter;
    std::string lOutputDirectory = laParams.front();
    laParams.pop_front();
    std::cout << lOutputDirectory << "\n";
    WithSlash(lOutputDirectory);

    const bool lbTrace = std::getenv("MOD_TRACE") != nullptr;
    const auto lNow = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double ldStart = lNow();
    CArk lArkHeader;
    lArkHeader.SetUniformEntryKey(giBodyKey);
    eError leError = lArkHeader.Load(HeaderName().c_str());
    SHOW_ERROR_AND_RETURN;
    const double ldLoaded = lNow();
    leError = lArkHeader.ExtractFiles(0, lArkHeader.GetNumFiles(), lOutputDirectory.c_str());
    SHOW_ERROR_AND_RETURN;
    if (lbTrace)
        std::fprintf(stderr, "[mod] Unpack: Load (CUDA init + header Cycle + parse) %.3f s, ExtractFiles %.3f s\n",
                     ldLoaded - ldStart, lNow() - ldLoaded);
    return eError_NoError;
}

// -find / -findhex / -findi / -findwild: one line "<name>\t<offset>" per match in table order, then by offset, at
// most kiMaxLines of them, and always the exact "<total> matches in <files> files".  lpMask (one byte per pattern
// byte, see CArk::FindMaskedInFiles) or null for the exact search; lpHow is added to the header line.
eError FindPattern(const std::string& lPattern, const std::string* lpMask = nullptr, const char* lpHow = "")
{
    constexpr uint64_t kiMaxLines = 10000;
    if (lPattern.empty() || lPattern.size() > 64) {
        std::cout << "The pattern must be 1 to 64 bytes long\n";
        return eError_InvalidParameter;
    }
    std::cout << "Searching " << HeaderName() << " for " << lPattern.size() << " bytes" << lpHow << "\n";
    CArk lArkHeader;
    lArkHeader.SetUniformEntryKey(giBodyKey);
    eError leError = lArkHeader.Load(HeaderName().c_str());
    SHOW_ERROR_AND_RETURN;
    std::vector<SFileMatch> laMatches;
    std::vector<uint64_t> laFileCounts;
    uint64_t luTotal = 0;
    if (lpMask)
        leError = lArkHeader.FindMaskedInFiles((const unsigned char*)lPattern.data(), (const unsigned char*)lpMask->data(),
                                               (uint32_t)lPattern.size(), kiMaxLines, laMatches, &luTotal, &laFileCounts);
    else
        leError = lArkHeader.FindInFiles((const unsigned char*)lPattern.data(), (uint32_t)lPattern.size(), kiMaxLines, laMatches,
                                         &luTotal, &laFileCounts);
    SHOW_ERROR_AND_RETURN;
    for (const SFileMatch& lMatch : laMatches)
        std::cout << lArkHeader.Header().maFiles[(size_t)lMatch.file].mName << "\t" << lMatch.offset << "\n";
    if (luTotal > laMatches.size())
        std::cout << "... " << luTotal - laMatches.size() << " more\n";
    const size_t liFiles = (size_t)std::count_if(laFileCounts.begin(), laFileCounts.end(), [](uint64_t n) { return n != 0; });
    std::cout << luTotal << " matches in " << liFiles << " files\n";
    return eError_NoError;
}

eError Find(std::deque<std::string>& laParams)
{
    if (laParams.empty())
        return eError_InvalidParameter;
    const std::string lText = laParams.front();
    laParams.pop_front();
    return FindPattern(lText);
}

// ASCII upper case: the folded form of a case-insensitive pattern ('a'..'z' -> 'A'..'Z', every other byte itself).
std::string Folded(std::string lText)
{
    for (char& c : lText)
        if (c >= 'a' && c <= 'z')
            c = (char)(c - 0x20);
    return lText;
}

// -findi: -find with every letter matching either case (pattern byte upper-cased, mask 0xDF; 0xFF elsewhere).
eError FindIgnoreCase(std::deque<std::string>& laParams)
{
    if (laParams.empty())
        return eError_InvalidParameter;
    const std::string lText = Folded(laParams.front());
    laParams.pop_front();
    std::string lMask(lText.size(), (char)0xFF);
    for (size_t ii = 0; ii < lText.size(); ++ii)
        if (lText[ii] >= 'A' && lText[ii] <= 'Z')
            lMask[ii] = (char)0xDF;
    return FindPattern(lText, &lMask, ", ignoring case");
}

// -findwild: pairs of hex digits, whitespace ignored, in which any digit may be '?' (any nibble; "??" any byte).
eError FindWild(std::deque<std::string>& laParams)
{
    if (laParams.empty())
        return eError_InvalidParameter;
    std::string lDigits;
    for (char c : laParams.front())
        if (!std::isspace((unsigned char)c))
            lDigits += (char)std::tolower((unsigned char)c);
    laParams.pop_front();
    if (lDigits.size() % 2 != 0 || lDigits.find_first_not_of("0123456789abcdef?") != std::string::npos) {
        std::cout << "-findwild takes pairs of hex digits, any of them ?\n";
        return eError_InvalidParameter;
    }
    if (lDigits.empty() || lDigits.size() > 128) {
        std::cout << "The pattern must be 1 to 64 bytes long\n";
        return eError_InvalidParameter;
    }
    if (lDigits.find_first_not_of('?') == std::string::npos) {
        std::cout << "-findwild: the pattern has no hex digit that is not ?\n";
        return eError_InvalidParameter;
    }
    std::string lBytes, lMask;
    for (size_t ii = 0; ii < lDigits.size(); ii += 2) {
        uint32_t luValue = 0, luMask = 0;
        for (size_t kk = 0; kk < 2; ++kk) {
            const char c = lDigits[ii + kk];
            luValue <<= 4;
            luMask <<= 4;
            if (c != '?') {
                luValue |= (uint32_t)std::stoi(std::string(1, c), nullptr, 16);
                luMask |= 0xFu;
            }
        }
        lBytes += (char)luValue;
        lMask += (char)luMask;
    }
    return FindPattern(lBytes, &lMask);
}

// Hex digit pairs, whitespace ignored (the -findhex syntax) -> lBytes; lpShown, when given, gets the digits
// lowercased and without spaces.
bool ParseHex(const std::string& lText, std::string& lBytes, std::string* lpShown)
{
    std::string lDigits;
    for (char c : lText)
        if (!std::isspace((unsigned char)c))
            lDigits += (char)std::tolower((unsigned char)c);
    if (lDigits.size() % 2 != 0 || lDigits.find_first_not_of("0123456789abcdef") != std::string::npos)
        return false;
    lBytes.clear();
    for (size_t ii = 0; ii < lDigits.size(); ii += 2)
        lBytes += (char)std::stoi(lDigits.substr(ii, 2), nullptr, 16);
    if (lpShown)
        *lpShown = lDigits;
    return true;
}

eError FindHex(std::deque<std::string>& laParams)
{
    if (laParams.empty())
        return eError_InvalidParameter;
    std::string lBytes;
    const bool lbHex = ParseHex(laParams.front(), lBytes, nullptr);
    laParams.pop_front();
    if (!lbHex) {
        std::cout << "-findhex takes pairs of hex digits\n";
        return eError_InvalidParameter;
    }
    return FindPattern(lBytes);
}

// -findlist / -findhexlist: one pattern per line (a trailing '\r' stripped, empty lines skipped), all searched in one
// pass.  One line "<name>\t<offset>\t<pattern>" per match in table order, then by offset, then list order, at most
// kiMaxLines of them; then "<count>\t<pattern>" per pattern in list order, and the "<total> matches in <files>
// files" of -find.  A hex pattern is shown as given, lowercased and without spaces.  lbFold (-findilist): text
// patterns whose letters match either case; two lines equal ignoring case are refused.
eError FindList(std::deque<std::string>& laParams, bool lbHex, bool lbFold = false)
{
    constexpr uint64_t kiMaxLines = 10000;
    const char* lpWhat = lbFold ? "-findilist" : lbHex ? "-findhexlist" : "-findlist";
    if (laParams.empty())
        return eError_InvalidParameter;
    const std::string lListPath = laParams.front();
    laParams.pop_front();
    std::ifstream lList(lListPath, std::ios::binary);
    if (!lList) {
        std::cout << lpWhat << ": cannot read " << lListPath << "\n";
        return eError_FailedToOpenFile;
    }
    std::vector<std::string> laPatterns, laShown;
    std::unordered_map<std::string, size_t> lLineOf;
    std::string lLine;
    for (size_t liLine = 1; std::getline(lList, lLine); ++liLine) {
        if (!lLine.empty() && lLine.back() == '\r')
            lLine.pop_back();
        if (lLine.empty())
            continue;
        std::string lBytes = lLine, lShown = lLine;
        if (lbHex && !ParseHex(lLine, lBytes, &lShown)) {
            std::cout << lpWhat << ": line " << liLine << " is not pairs of hex digits\n";
            return eError_InvalidParameter;
        }
        if (lBytes.empty() || lBytes.size() > 64) {
            std::cout << lpWhat << ": line " << liLine << ": the pattern must be 1 to 64 bytes long\n";
            return eError_InvalidParameter;
        }
        const auto lSeen = lLineOf.emplace(lbFold ? Folded(lBytes) : lBytes, liLine);
        if (!lSeen.second) {
            std::cout << lpWhat << ": line " << liLine << " repeats the pattern of line " << lSeen.first->second
                      << (lbFold ? " ignoring case" : "") << "\n";
            return eError_InvalidParameter;
        }
        if (laPatterns.size() == 256) {
            std::cout << lpWhat << ": line " << liLine << ": a list holds at most 256 patterns\n";
            return eError_InvalidParameter;
        }
        laPatterns.push_back(lBytes);
        laShown.push_back(lShown);
    }
    if (laPatterns.empty()) {
        std::cout << lpWhat << ": " << lListPath << " holds no pattern\n";
        return eError_InvalidParameter;
    }
    std::cout << "Searching " << HeaderName() << " for " << laPatterns.size() << " patterns" << (lbFold ? ", ignoring case" : "")
              << "\n";
    CArk lArkHeader;
    lArkHeader.SetUniformEntryKey(giBodyKey);
    eError leError = lArkHeader.Load(HeaderName().c_str());
    SHOW_ERROR_AND_RETURN;
    std::vector<SFileSetMatch> laMatches;
    std::vector<uint64_t> laFileCounts, laPatternCounts;
    uint64_t luTotal = 0;
    leError = lArkHeader.FindSetInFiles(laPatterns, kiMaxLines, laMatches, &luTotal, &laFileCounts, &laPatternCounts, lbFold);
    SHOW_ERROR_AND_RETURN;
    for (const SFileSetMatch& lMatch : laMatches)
        std::cout << lArkHeader.Header().maFiles[(size_t)lMatch.file].mName << "\t" << lMatch.offset << "\t" << laShown[lMatch.pattern]
                  << "\n";
    if (luTotal > laMatches.size())
        std::cout << "... " << luTotal - laMatches.size() << " more\n";
    for (size_t jj = 0; jj < laPatterns.size(); ++jj)
        std::cout << laPatternCounts[jj] << "\t" << laShown[jj] << "\n";
    const size_t liFiles = (size_t)std::count_if(laFileCounts.begin(), laFileCounts.end(), [](uint64_t n) { return n != 0; });
    std::cout << luTotal << " matches in " << liFiles << " files\n";
    return eError_NoError;
}

eError FindListText(std::deque<std::string>& laParams) { return FindList(laParams, false); }
eError FindListHex(std::deque<std::string>& laParams) { return FindList(laParams, true); }
eError FindListIgnoreCase(std::deque<std::string>& laParams) { return FindList(laParams, false, true); }

eError PackImpl(std::deque<std::string>& laParams)
{
    std::cout << "Packing " << HeaderName() << " from ";
    if (laParams.empty())
        return eError_InvalidParameter;
    std::string lInputPath = laParams.front();
    laParams.pop_front();
    std::cout << lInputPath << " to ";
    if (laParams.empty())
        return eError_InvalidParameter;
    std::string lOutputPath = laParams.front();
    laParams.pop_front();
    std::cout << lOutputPath << "\n";
    WithSlash(lInputPath);
    WithSlash(lOutputPath);

    // Unless -packall is given the song list comes from the two DTA configs inside the input tree,
    // like the reference (Modulate.cpp:410-432): it decides which /songs/<name>/ folders are packed.
    eError leError = eError_NoError;
    std::vector<SSongConfig> lSongs;
    if (!CSettings::mbPackAllFiles) {
        const std::string lPlatform = CSettings::msPlatform;
        const std::string lAmpConfigPath = lInputPath + lPlatform + "/config/amp_config.dta_dta_" + lPlatform;
        std::cout << "Loading " << lAmpConfigPath << "\n";
        CDtaFile lAmpConfig;
        leError = lAmpConfig.Load(lAmpConfigPath.c_str());
        SHOW_ERROR_AND_RETURN;
        lSongs = lAmpConfig.GetSongs();
        CDtaFile lSongsConfig;
        const std::string lAmpSongsConfigPath = lInputPath + lPlatform + "/config/amp_songs_config.dta_dta_" + lPlatform;
        leError = lSongsConfig.Load(lAmpSongsConfigPath.c_str());
        SHOW_ERROR_AND_RETURN;
        lSongsConfig.GetSongData(lSongs);
    }

    CArk lReferenceArkHeader;
    leError = lReferenceArkHeader.Load(HeaderName().c_str());
    SHOW_ERROR_AND_RETURN;

    CArk lArkHeader;
    lArkHeader.SetUniformEntryKey(giBodyKey);
    leError = lArkHeader.ConstructFromDirectory(lInputPath.c_str(), lReferenceArkHeader, lSongs);
    SHOW_ERROR_AND_RETURN;
    leError = lArkHeader.BuildArk(lInputPath.c_str(), lSongs);
    SHOW_ERROR_AND_RETURN;
    leError = lArkHeader.SaveArk(lOutputPath.c_str(), HeaderName().c_str());
    SHOW_ERROR_AND_RETURN;
    return eError_NoError;
}

eError Pack(std::deque<std::string>& laParams) { return PackImpl(laParams); }

eError AddPack(std::deque<std::string>& laParams)
{
    CSettings::mbIgnoreNewFiles = false;  // reference Modulate.cpp:580-586
    return PackImpl(laParams);
}

eError Decode(std::deque<std::string>&)
{
    const std::string lHeaderFilename = HeaderName();
    FILE* lpHeaderFile = std::fopen(lHeaderFilename.c_str(), "rb");
    if (!lpHeaderFile)
        return eError_FailedToOpenFile;
    std::fseek(lpHeaderFile, 0, SEEK_END);
    const long liHeaderSize = std::ftell(lpHeaderFile);
    std::fseek(lpHeaderFile, 0, SEEK_SET);
    std::vector<unsigned char> lData((size_t)std::max(0l, liHeaderSize));
    const size_t liRead = lData.empty() ? 0 : std::fread(lData.data(), 1, lData.size(), lpHeaderFile);
    std::fclose(lpHeaderFile);
    if (liRead != lData.size() || lData.size() < 4)
        return eError_UnknownVersionNumber;

    unsigned int luVersion = 0;
    std::memcpy(&luVersion, lData.data(), 4);
    if (luVersion != CSettings::kuEncryptedVersionPS3 && luVersion != CSettings::kuEncryptedVersionPS4)
        return eError_UnknownVersionNumber;
    const unsigned int kuInitialKey =
        (luVersion == CSettings::kuEncryptedVersionPS3) ? CSettings::kuEncryptedPS3Key : CSettings::kuEncryptedPS4Key;
    CEncryptionCycler lDecrypt;
    lDecrypt.Cycle(lData.data() + 4, (unsigned int)(lData.size() - 4), (int)kuInitialKey);

    const std::string lOut = lHeaderFilename + ".dec";
    FILE* lpOut = std::fopen(lOut.c_str(), "wb");
    if (!lpOut)
        return eError_FailedToCreateFile;
    const size_t liWritten = std::fwrite(lData.data(), 1, lData.size(), lpOut);
    std::fclose(lpOut);
    return liWritten == lData.size() ? eError_NoError : eError_FailedToWriteData;
}

// -listsongs <dir>: the reference's read-only song listing (Modulate.cpp:504-547), same output format.
eError ListSongs(std::deque<std::string>& laParams)
{
    std::cout << "Loading ";
    if (laParams.empty())
        return eError_InvalidParameter;
    std::string lBasePath = laParams.front();
    laParams.pop_front();
    WithSlash(lBasePath);
    const std::string lPlatform = CSettings::msPlatform;
    const std::string lAmpConfigPath = lBasePath + lPlatform + "/config/amp_config.dta_dta_" + lPlatform;
    std::cout << lAmpConfigPath << "\n";
    CDtaFile lAmpConfig;
    eError leError = lAmpConfig.Load(lAmpConfigPath.c_str());
    SHOW_ERROR_AND_RETURN;
    const std::string lAmpSongsConfigPath = lBasePath + lPlatform + "/config/amp_songs_config.dta_dta_" + lPlatform;
    std::cout << "Loading " << lAmpSongsConfigPath << "\n";
    CDtaFile lSongsConfig;
    leError = lSongsConfig.Load(lAmpSongsConfigPath.c_str());
    SHOW_ERROR_AND_RETURN;
    std::cout << "\n";
    int ii = 1;
    std::vector<SSongConfig> lSongs = lAmpConfig.GetSongs();
    lSongsConfig.GetSongData(lSongs);
    for (const SSongConfig& lSong : lSongs) {
        std::cout << "Song " << ii << "\t  " << lSong.mId << " - " << lSong.mName << " - " << lSong.mType << "\n\t  "
                  << lSong.mPath << "\n\t  Unlocked by " << lSong.mUnlockMethod << " " << lSong.miUnlockCount << "\n"
                  << "\t  Arena: " << lSong.mArena << "\n\n";
        ++ii;
    }
    return eError_NoError;
}

// -dtaset <file> <key> <value>: load a binary DTA file, replace the value that follows the symbol
// <key> (integer or string, whichever is there) and save it back -- the host-side patch step of a
// repack.  -dtacopy <in> <out>: load + save (codec round trip).
eError DtaSet(std::deque<std::string>& laParams)
{
    if (laParams.size() < 3)
        return eError_InvalidParameter;
    const std::string lFile = laParams[0], lKey = laParams[1], lValue = laParams[2];
    laParams.erase(laParams.begin(), laParams.begin() + 3);
    CDtaFile lDta;
    eError leError = lDta.Load(lFile.c_str());
    ERROR_RETURN;
    char* lpEnd = nullptr;
    const long liValue = std::strtol(lValue.c_str(), &lpEnd, 0);
    const bool lbNumeric = lpEnd && *lpEnd == 0 && !lValue.empty();
    if (!((lbNumeric && lDta.SetIntAfter(lKey, (int32_t)liValue)) || lDta.SetStringAfter(lKey, lValue))) {
        std::cout << "No value of a matching type follows " << lKey << "\n";
        return eError_InvalidParameter;
    }
    return lDta.Save(lFile.c_str());
}

eError DtaCopy(std::deque<std::string>& laParams)
{
    if (laParams.size() < 2)
        return eError_InvalidParameter;
    const std::string lIn = laParams[0], lOut = laParams[1];
    laParams.erase(laParams.begin(), laParams.begin() + 2);
    CDtaFile lDta;
    eError leError = lDta.Load(lIn.c_str());
    ERROR_RETURN;
    return lDta.Save(lOut.c_str());
}

void PrintUsage()
{
    std::cout << "Usage: modulate <options> <command>\n\n"
              << "Options:\n"
              << "  -verbose        Show additional information during operation\n"
              << "  -ps3            Switch to PS3 mode (default PS4)\n"
              << "  -force          Overwrite existing output files\n"
              << "  -packall        Pack every file found, bypassing the /songs/ filter\n"
              << "  -bodykey <k>    Cipher entry bodies with key k (extension; default 0 = plain, like the game)\n"
              << "  -device <n>     Run on GPU n\n\n"
              << "Commands:\n"
              << "  -unpack <out_dir>           Unpack main_<platform>.hdr (+ .ark parts) from the current directory\n"
              << "  -pack <in_dir> <out_dir>    Repack the files the reference header knows\n"
              << "  -pack_add <in_dir> <out_dir> Repack, also adding new files\n"
              << "  -decode                     Write the deciphered header to main_<platform>.hdr.dec\n"
              << "  -find <text>                List the entries (and offsets) whose bytes contain <text>\n"
              << "  -findhex <hex>              Same for a pattern given as hex bytes, e.g. 00ff1a\n"
              << "  -findlist <file>            Same for every pattern of <file> (one per line, up to 256), in one pass\n"
              << "  -findhexlist <file>         Same for a file of hex patterns, one per line\n"
              << "  -findi <text>               -find ignoring the case of ASCII letters\n"
              << "  -findilist <file>           -findlist ignoring the case of ASCII letters\n"
              << "  -findwild <hex>             -findhex where any hex digit may be ?, e.g. 0a??00?f\n"
              << "  -listsongs <dir>            List the songs the DTA configs under <dir> define\n"
              << "  -dtaset <file> <key> <val>  Patch the value following symbol <key> in a binary DTA file\n"
              << "  -dtacopy <in> <out>         Load and re-save a binary DTA file\n";
}

}  // namespace

// MOD_TRACE=1: wall-clock stamps of the process phases (a cold start is dominated by CUDA context creation and
// page-locking, not by the archive work; tools/cli_timing.sh reads these).
static void TraceStamp(const char* lpWhat)
{
    const char* lpTrace = std::getenv("MOD_TRACE");
    if (!lpTrace || !*lpTrace || *lpTrace == '0')
        return;
    const double ldNow = std::chrono::duration<double>(std::chrono::system_clock::now().time_since_epoch()).count();
    std::fprintf(stderr, "[mod] cli %s at %.3f\n", lpWhat, ldNow);
}

int main(int argc, char* argv[])
{
    TraceStamp("main entered");
    struct sCommandPair {
        const char* mpCommandName;
        std::function<eError(std::deque<std::string>&)> mFunction;
    };
    const sCommandPair kaCommands[] = {
        {"-ps3", PS3},       {"-verbose", EnableVerbose}, {"-force", EnableForceWrite}, {"-packall", EnablePackAll},
        {"-bodykey", BodyKey}, {"-device", Device},       {"-unpack", Unpack},          {"-pack", Pack},
        {"-pack_add", AddPack}, {"-decode", Decode},   {"-dtaset", DtaSet},          {"-dtacopy", DtaCopy},
        {"-listsongs", ListSongs}, {"-find", Find},     {"-findhex", FindHex},
        {"-findlist", FindListText}, {"-findhexlist", FindListHex},
        {"-findi", FindIgnoreCase}, {"-findilist", FindListIgnoreCase}, {"-findwild", FindWild},
    };

    std::deque<std::string> laParams;
    for (int ii = 1; ii < argc; ++ii)
        laParams.push_back(argv[ii]);
    if (laParams.empty()) {
        PrintUsage();
        return 0;
    }
    while (!laParams.empty()) {
        bool lbMatched = false;
        for (const sCommandPair& lCommand : kaCommands) {
            if (strcasecmp(laParams.front().c_str(), lCommand.mpCommandName) != 0)
                continue;
            lbMatched = true;
            laParams.pop_front();
            TraceStamp(lCommand.mpCommandName);
            const eError leError = lCommand.mFunction(laParams);
            if (leError != eError_NoError) {
                ShowError(leError);
                return -1;
            }
            std::cout << "\n";
            break;
        }
        if (!lbMatched) {
            std::cout << "Unkown parameter: " << laParams.front() << "\nAborting\n\n";
            PrintUsage();
            return -1;
        }
    }
    std::cout << "Complete!\n";
    TraceStamp("main returns");
    return 0;
}
