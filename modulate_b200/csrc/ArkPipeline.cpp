#include "ArkPipeline.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <deque>
#include <iostream>
#include <mutex>
#include <string>
#include <thread>

namespace arkpipe {

namespace {

double NowSeconds()
{
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

bool TraceEnabled()
{
    const char* lpValue = std::getenv("MOD_TRACE");
    return lpValue && *lpValue && *lpValue != '0';
}

// A few worker threads draining a queue of closures: the reader and writer stages of the pipeline.
class TaskPool
{
public:
    explicit TaskPool(int liThreads)
    {
        for (int ii = 0; ii < liThreads; ++ii)
            maThreads.emplace_back([this]() { Loop(); });
    }
    ~TaskPool() { Finish(); }
    void Push(std::function<void()> lTask)
    {
        {
            std::lock_guard<std::mutex> lLock(mMutex);
            maTasks.push_back(std::move(lTask));
        }
        mSignal.notify_one();
    }
    void Finish()  // run what is queued, then stop
    {
        {
            std::lock_guard<std::mutex> lLock(mMutex);
            mbClosed = true;
        }
        mSignal.notify_all();
        for (std::thread& lThread : maThreads)
            if (lThread.joinable())
                lThread.join();
    }

private:
    void Loop()
    {
        for (;;) {
            std::function<void()> lTask;
            {
                std::unique_lock<std::mutex> lLock(mMutex);
                mSignal.wait(lLock, [this]() { return !maTasks.empty() || mbClosed; });
                if (maTasks.empty())
                    return;
                lTask = std::move(maTasks.front());
                maTasks.pop_front();
            }
            lTask();
        }
    }
    std::mutex mMutex;
    std::condition_variable mSignal;
    std::deque<std::function<void()>> maTasks;
    std::vector<std::thread> maThreads;
    bool mbClosed = false;
};

// Tuning aid: MOD_IO_<NAME>=<n> overrides a pipeline's thread / slot count (tools/unpack_timing.py sweeps them).
int Tunable(const char* lpName, int liDefault)
{
    const char* lpValue = std::getenv(lpName);
    const int liValue = lpValue && *lpValue ? std::atoi(lpValue) : 0;
    return liValue > 0 ? liValue : liDefault;
}

// GPUs the facade spreads an archive over: every visible device (MOD_DEVICES = bit mask restricts
// them) once the archive is large enough to be worth it, else only the calling thread's device.
std::vector<int> FacadeDevices(uint64_t luBytes)
{
    std::vector<int> laDevices;
    const int liCurrent = std::max(0, mod_current_device());
    const int liCount = mod_device_count();
    const char* lpMask = std::getenv("MOD_DEVICES");
    const uint64_t luMask = lpMask && *lpMask ? std::strtoull(lpMask, nullptr, 0) : 0;
    const uint64_t kuMultiGpuThreshold = 256ull << 20;
    if (liCount > 1 && luBytes >= kuMultiGpuThreshold)
        for (int ii = 0; ii < liCount && ii < 64; ++ii)
            if (luMask == 0 || ((luMask >> ii) & 1ull))
                laDevices.push_back(ii);
    if (laDevices.empty())
        laDevices.push_back(liCurrent);
    return laDevices;
}

// One stage buffer set of the pipeline: pinned host memory either side of the GPU, the two HBM
// windows the batched kernel works on, and the stream that orders upload -> kernel -> download.
struct Slot {
    enum eState { eFree, eFilling, eFilled, eDraining };
    int miDevice = 0;
    unsigned char* mpHostIn = nullptr;   // what the readers fill (image range / input files)
    unsigned char* mpHostOut = nullptr;  // what the writers drain (extracted files / ciphered image range)
    void* mpDevIn = nullptr;
    void* mpDevOut = nullptr;
    void* mpStream = nullptr;
    eState meState = eFree;
    int miTasksLeft = 0;  // of the fill or drain stage under way
    bool mbUsedGpu = false;
    uint64_t muInCapacity = 0, muOutCapacity = 0;
};

// Slots handed back by a finished pipeline, kept for the next one: page-locking memory costs more than
// moving the data does (0.3-1 ms per MiB), and a repack runs an extract and a build back to back.  At
// most kiMaxCached slots are kept; the cache is never destroyed (the CUDA context may be gone by the
// time static destructors run), the OS reclaims it with the process.
struct SlotCache {
    std::mutex mMutex;
    std::vector<Slot> maSlots;
    static constexpr size_t kiMaxCached = 24;
    static SlotCache& Get()
    {
        static SlotCache* lpCache = new SlotCache();
        return *lpCache;
    }
    bool Take(int liDevice, uint64_t luIn, uint64_t luOut, bool lbNeedGpu, Slot& lOut)
    {
        std::lock_guard<std::mutex> lLock(mMutex);
        for (size_t ii = 0; ii < maSlots.size(); ++ii) {
            Slot& lSlot = maSlots[ii];
            if (lSlot.muInCapacity >= luIn && lSlot.muOutCapacity >= luOut && (!lbNeedGpu || (lSlot.mpStream && lSlot.miDevice == liDevice))) {
                lOut = lSlot;
                maSlots.erase(maSlots.begin() + (long)ii);
                return true;
            }
        }
        return false;
    }
    bool Give(const Slot& lSlot)
    {
        std::lock_guard<std::mutex> lLock(mMutex);
        if (maSlots.size() >= kiMaxCached)
            return false;
        maSlots.push_back(lSlot);
        return true;
    }
};

struct SlotRing {
    std::vector<Slot> maSlots;
    std::mutex mMutex;
    std::condition_variable mSignal;
    std::atomic<int> miError{(int)eError_NoError};

    void Fail(eError leWhat)
    {
        int liExpected = (int)eError_NoError;
        miError.compare_exchange_strong(liExpected, (int)leWhat);
        mSignal.notify_all();
    }
    bool Failed() const { return miError.load() != (int)eError_NoError; }
    // the slot's group starts liTasks units of work in state leBusy (eFilling / eDraining); with none it
    // moves on at once
    void Start(Slot& lSlot, Slot::eState leBusy, int liTasks)
    {
        {
            std::lock_guard<std::mutex> lLock(mMutex);
            lSlot.meState = liTasks ? leBusy : Next(leBusy);
            lSlot.miTasksLeft = liTasks;
        }
        mSignal.notify_all();
    }
    // one unit of fill / drain work done; the last one flips the slot's state
    void TaskDone(Slot& lSlot)
    {
        bool lbLast = false;
        {
            std::lock_guard<std::mutex> lLock(mMutex);
            lbLast = --lSlot.miTasksLeft == 0;
            if (lbLast)
                lSlot.meState = Next(lSlot.meState);
        }
        if (lbLast)
            mSignal.notify_all();
    }
    static Slot::eState Next(Slot::eState leBusy) { return leBusy == Slot::eFilling ? Slot::eFilled : Slot::eFree; }
    // Allocate liPerDevice slots on each device: pinned buffers of luInBytes / luOutBytes, HBM windows
    // of the same sizes (+ slack for the 16-byte phase), one stream each.
    bool Allocate(const std::vector<int>& laDevices, int liPerDevice, size_t liGroups, uint64_t luInBytes, uint64_t luOutBytes,
                  bool lbNeedGpu)
    {
        const size_t liWanted = std::min(liGroups, (size_t)liPerDevice * laDevices.size());
        maSlots.resize(std::max<size_t>(1, liWanted));
        std::vector<size_t> laFresh;  // slots the cache could not supply
        for (size_t ii = 0; ii < maSlots.size(); ++ii) {
            Slot& lSlot = maSlots[ii];
            const int liDevice = laDevices[ii % laDevices.size()];
            if (SlotCache::Get().Take(liDevice, luInBytes + 32, luOutBytes + 32, lbNeedGpu, lSlot)) {
                lSlot.meState = Slot::eFree;
                lSlot.mbUsedGpu = false;
                continue;
            }
            lSlot.miDevice = liDevice;
            lSlot.muInCapacity = luInBytes + 32;
            lSlot.muOutCapacity = luOutBytes + 32;
            laFresh.push_back(ii);
        }
        // Page-locking dominates a cold start (0.3-1 ms per MiB, i.e. more than the whole pipeline of a 1 GiB
        // archive): the fresh slots are therefore set up side by side, one thread each.
        std::atomic<bool> lbOk{true};
        auto lSetUp = [&](size_t ii) {
            Slot& lSlot = maSlots[ii];
            lSlot.mpHostIn = (unsigned char*)mod_host_alloc(lSlot.muInCapacity);
            lSlot.mpHostOut = (unsigned char*)mod_host_alloc(lSlot.muOutCapacity);
            bool lbGood = lSlot.mpHostIn && lSlot.mpHostOut;
            if (lbGood && lbNeedGpu) {
                lbGood = mod_init(lSlot.miDevice) == MOD_OK;
                if (lbGood) {
                    lSlot.mpDevIn = mod_device_alloc(lSlot.muInCapacity);
                    lSlot.mpDevOut = mod_device_alloc(lSlot.muOutCapacity);
                    lSlot.mpStream = mod_stream_create();
                    lbGood = lSlot.mpDevIn && lSlot.mpDevOut && lSlot.mpStream;
                }
            }
            if (!lbGood)
                lbOk.store(false);
        };
        if (laFresh.size() <= 1 || Tunable("MOD_IO_SERIAL_SETUP", 0)) {
            for (size_t ii : laFresh)
                lSetUp(ii);
        } else {
            std::vector<std::thread> laThreads;
            for (size_t ii : laFresh)
                laThreads.emplace_back(lSetUp, ii);
            for (std::thread& lThread : laThreads)
                lThread.join();
        }
        return lbOk.load();
    }
    void Release()
    {
        for (Slot& lSlot : maSlots) {
            if (lSlot.mpStream)
                mod_stream_sync(lSlot.mpStream);
            if (lSlot.mpHostIn && lSlot.mpHostOut && SlotCache::Get().Give(lSlot))
                continue;
            if (lSlot.mpStream)
                mod_stream_destroy(lSlot.mpStream);
            mod_device_free(lSlot.mpDevIn);
            mod_device_free(lSlot.mpDevOut);
            mod_host_free(lSlot.mpHostIn);
            mod_host_free(lSlot.mpHostOut);
        }
        maSlots.clear();
    }
};

}  // namespace

SlowOp::SlowOp(const char* lpWhat) : mpWhat(lpWhat), mdStart(TraceEnabled() ? NowSeconds() : 0.0) {}

SlowOp::~SlowOp()
{
    if (mdStart > 0.0 && NowSeconds() - mdStart > 0.05)
        std::fprintf(stderr, "[mod] slow: %s took %.3f s\n", mpWhat, NowSeconds() - mdStart);
}

int HostThreads()
{
    const unsigned int luCores = std::thread::hardware_concurrency();
    return luCores ? (int)luCores : 4;
}

uint64_t GroupBytes() { return (uint64_t)Tunable("MOD_IO_GROUP_MIB", 32) << 20; }

void CutEntry(uint32_t luFile, uint64_t luSize, uint64_t luSrc, uint64_t luDst, int32_t liKey, uint64_t luGroupBytes,
              std::vector<Piece>& laPieces, std::vector<mod_desc>& laDescs)
{
    uint64_t luAt = 0;
    do {
        uint64_t luTake = luSize <= luGroupBytes + luGroupBytes / 2 ? luSize : std::min(luGroupBytes, luSize - luAt);
        if (luSize - luAt - luTake < luGroupBytes / 2)
            luTake = luSize - luAt;  // no short tail piece
        laPieces.push_back(Piece{luFile, luAt, (uint32_t)luTake});
        laDescs.push_back(mod_desc{luSrc + luAt, luDst + luAt, (uint32_t)luTake, luAt ? mod_key_jump(liKey, luAt) : liKey});
        luAt += luTake;
    } while (luAt < luSize);
}

std::vector<Group> GroupPieces(const std::vector<mod_desc>& laDescs, uint64_t luGroupBytes)
{
    std::vector<Group> laGroups;
    for (size_t liFirst = 0; liFirst < laDescs.size();) {
        Group lGroup{liFirst, liFirst, UINT64_MAX, 0, laDescs[liFirst].dst_off, laDescs[liFirst].dst_off};
        while (lGroup.last < laDescs.size() && (lGroup.dstHi - lGroup.dstLo < luGroupBytes || lGroup.last == liFirst)) {
            const mod_desc& lDesc = laDescs[lGroup.last++];
            if (lDesc.len) {
                lGroup.srcLo = std::min(lGroup.srcLo, lDesc.src_off);
                lGroup.srcHi = std::max(lGroup.srcHi, lDesc.src_off + lDesc.len);
            }
            lGroup.dstHi = std::max(lGroup.dstHi, lDesc.dst_off + lDesc.len);
        }
        if (lGroup.srcLo == UINT64_MAX)
            lGroup.srcLo = lGroup.srcHi = 0;
        laGroups.push_back(lGroup);
        liFirst = lGroup.last;
    }
    return laGroups;
}

eError RunPipeline(const char* lpName, const std::vector<mod_desc>& laDescs, const std::vector<Group>& laGroups,
                   uint64_t luSrcBytes, uint64_t luDstBytes, bool lbUseGpu, int liReaders, int liWriters, const Stage& lFill,
                   const Stage& lDrain)
{
    const double ldStart = NowSeconds();
    uint64_t luMaxRange = 1, luMaxPayload = 1;
    for (const Group& lGroup : laGroups) {
        luMaxRange = std::max(luMaxRange, lGroup.srcHi - lGroup.srcLo);
        luMaxPayload = std::max(luMaxPayload, lGroup.dstHi - lGroup.dstLo);
    }

    // slots on every GPU in use, and the plan on each of them
    const int liOriginalDevice = lbUseGpu ? mod_current_device() : -1;
    const std::vector<int> laDevices = lbUseGpu ? FacadeDevices(luDstBytes) : std::vector<int>{0};
    SlotRing lRing;
    std::vector<mod_plan*> laPlans(laDevices.size(), nullptr);
    const int liSlotsPerDevice = Tunable("MOD_IO_SLOTS", std::max(3, 6 / (int)laDevices.size()));
    bool lbReady = lRing.Allocate(laDevices, liSlotsPerDevice, laGroups.size(), luMaxRange, lbUseGpu ? luMaxPayload : 0, lbUseGpu);
    for (size_t dd = 0; dd < laDevices.size() && lbReady && lbUseGpu; ++dd)
        lbReady = mod_init(laDevices[dd]) == MOD_OK &&
                  mod_plan_create(laDescs.data(), laDescs.size(), luSrcBytes, luDstBytes, 0, &laPlans[dd]) == MOD_OK;
    const double ldReady = NowSeconds();
    double ldEnqueued = ldReady, ldDrained = ldReady;
    const size_t liSlots = lRing.maSlots.size();
    if (!lbReady) {
        std::cout << "GPU " << lpName << " could not be set up: " << mod_last_error() << "\n";
    } else {
        TaskPool lReaders(Tunable("MOD_IO_READERS", liReaders));
        TaskPool lWriters(Tunable("MOD_IO_WRITERS", liWriters));
        const std::string lSyncWhat = std::string(lpName) + " stream sync", lEnqueueWhat = std::string(lpName) + " GPU enqueue of a group";
        auto lSlotOf = [&](size_t gg) -> Slot& { return lRing.maSlots[gg % liSlots]; };
        // the tasks of group gg's fill or drain stage, queued on the readers / writers; a drain waits for the
        // slot's stream first, and a task is skipped once the pipeline has failed
        auto lStart = [&](bool lbDrain, size_t gg, unsigned char* lpBytes) {
            Slot* lpSlot = &lSlotOf(gg);
            const int liTasks = (lbDrain ? lDrain : lFill).mTasks(gg);
            const bool lbSync = lbDrain && lpSlot->mbUsedGpu;
            lRing.Start(*lpSlot, lbDrain ? Slot::eDraining : Slot::eFilling, liTasks);
            for (int tt = 0; tt < liTasks; ++tt) {
                (lbDrain ? lWriters : lReaders).Push([&, lbDrain, gg, tt, lpBytes, lpSlot, lbSync]() {
                    if (lbSync && !lRing.Failed() &&
                        [&]() { SlowOp lSync(lSyncWhat.c_str()); return mod_stream_sync(lpSlot->mpStream); }() != MOD_OK) {
                        std::cout << "GPU " << lpName << " failed: " << mod_last_error() << "\n";
                        lRing.Fail(eError_InvalidData);
                    }
                    const eError leError = lRing.Failed() ? eError_NoError : (lbDrain ? lDrain : lFill).mRun(gg, tt, lpBytes);
                    if (leError != eError_NoError)
                        lRing.Fail(leError);
                    lRing.TaskDone(*lpSlot);
                });
            }
        };
        // upload -> kernel over the group's tiles -> download on the slot's stream, on the slot's device
        auto lEnqueue = [&](const Group& lGroup, Slot& lSlot) {
            const uint64_t luRange = lGroup.srcHi - lGroup.srcLo, luPayload = lGroup.dstHi - lGroup.dstLo;
            const size_t liDeviceIndex = (size_t)(std::find(laDevices.begin(), laDevices.end(), lSlot.miDevice) - laDevices.begin());
            uint64_t luTile0 = 0, luTile1 = 0;
            SlowOp lTimer(lEnqueueWhat.c_str());
            unsigned char* lpDevIn = (unsigned char*)lSlot.mpDevIn + (lGroup.srcLo & 15u);
            unsigned char* lpDevOut = (unsigned char*)lSlot.mpDevOut + (lGroup.dstLo & 15u);
            return mod_init(lSlot.miDevice) == MOD_OK &&
                   mod_plan_tile_range(laPlans[liDeviceIndex], lGroup.first, lGroup.last, &luTile0, &luTile1) == MOD_OK &&
                   mod_memcpy_h2d(lpDevIn, lSlot.mpHostIn + (lGroup.srcLo & 15u), luRange, lSlot.mpStream) == MOD_OK &&
                   mod_plan_run_window(laPlans[liDeviceIndex], luTile0, luTile1, lpDevIn, lGroup.srcLo, luRange, lpDevOut,
                                       lGroup.dstLo, luPayload, lSlot.mpStream) == MOD_OK &&
                   mod_memcpy_d2h(lSlot.mpHostOut + (lGroup.dstLo & 15u), lpDevOut, luPayload, lSlot.mpStream) == MOD_OK;
        };

        // this thread: start fills while slots are free, enqueue each filled group in turn, never waiting for the GPU
        size_t liNextFill = 0, liNextGpu = 0;
        auto lCanFill = [&]() {
            return liNextFill < laGroups.size() && liNextFill < liNextGpu + liSlots && lSlotOf(liNextFill).meState == Slot::eFree;
        };
        auto lCanRun = [&]() { return liNextGpu < liNextFill && lSlotOf(liNextGpu).meState == Slot::eFilled; };
        while (liNextGpu < laGroups.size() && !lRing.Failed()) {
            {
                std::unique_lock<std::mutex> lLock(lRing.mMutex);
                lRing.mSignal.wait(lLock, [&]() { return lCanFill() || lCanRun() || lRing.Failed(); });
            }
            if (lRing.Failed())
                break;
            while (lCanFill()) {
                const size_t gg = liNextFill++;
                lStart(false, gg, lSlotOf(gg).mpHostIn + (laGroups[gg].srcLo & 15u));
            }
            while (lCanRun()) {
                const size_t gg = liNextGpu++;
                const Group& lGroup = laGroups[gg];
                Slot& lSlot = lSlotOf(gg);
                lSlot.mbUsedGpu = lbUseGpu && lGroup.dstHi > lGroup.dstLo;
                if (lSlot.mbUsedGpu && !lEnqueue(lGroup, lSlot)) {
                    std::cout << "GPU " << lpName << " failed: " << mod_last_error() << "\n";
                    lRing.Fail(eError_InvalidData);
                    break;
                }
                // without the GPU the bytes read are the bytes to write (the source and destination layouts agree)
                lStart(true, gg, lSlot.mbUsedGpu ? lSlot.mpHostOut + (lGroup.dstLo & 15u) : lSlot.mpHostIn + (lGroup.srcLo & 15u));
            }
        }
        ldEnqueued = NowSeconds();
        lReaders.Finish();
        lWriters.Finish();
        ldDrained = NowSeconds();
    }

    lRing.Release();
    for (mod_plan* lpPlan : laPlans)
        mod_plan_destroy(lpPlan);
    if (liOriginalDevice >= 0)
        mod_init(liOriginalDevice);
    if (TraceEnabled())
        std::fprintf(stderr, "[mod] %s pipeline: %zu groups on %zu GPU(s), %zu slots; setup %.3f s, pipeline %.3f s, drain %.3f s, free %.3f s\n",
                     lpName, laGroups.size(), lbUseGpu ? laDevices.size() : 0, liSlots, ldReady - ldStart, ldEnqueued - ldReady,
                     ldDrained - ldEnqueued, NowSeconds() - ldDrained);
    return lbReady ? (eError)lRing.miError.load() : eError_NoData;
}

}  // namespace arkpipe
