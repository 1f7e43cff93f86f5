// Host engine behind the C ABI (include/megaverse_b200.h): owns the HBM state, the host level generators and their
// worker pool, and launches the two kernels of a step on one CUDA stream.
//
//   mv_step  =  [H2D actions] -> stepKernel (physics + scenario + in-kernel reset + instance lists)
//                             -> viewKernel (geometry + raster + shading in shared memory -> obs tensor)
//                             -> [D2H obs/rewards/dones] -> schedule next-level generation
//
// There is no host synchronisation between physics, episode reset and rendering (the reference resets finished envs
// serially on the caller thread between the two, vector_env.cpp:94-105): every env always has its NEXT level pre-staged
// in HBM (no RNG draw happens during an episode, so the next level only depends on the env's RNG state after the
// previous generation), and the step kernel flips to it by itself when the episode ends.
#include <cuda_runtime.h>

#include <atomic>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <functional>
#include <mutex>
#include <queue>
#include <string>
#include <thread>
#include <vector>

#include "../../include/megaverse_b200.h"
#include "hostmath.hpp"
#include "levelgen.hpp"
#include "raster_view.cuh"
#include "step_kernel.cuh"

namespace {

// every entry point runs on the engine's device and leaves the calling thread's current device as it found it
struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        ok = (prev == dev) || cudaSetDevice(dev) == cudaSuccess;
        if (prev == dev) prev = -1;  // nothing to restore
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

thread_local std::string g_createError;

#define MV_CUDA(call)                                                                                             \
    do {                                                                                                          \
        cudaError_t err__ = (call);                                                                               \
        if (err__ != cudaSuccess) {                                                                               \
            setError(std::string(#call) + ": " + cudaGetErrorString(err__));                                      \
            return MV_ERR_CUDA;                                                                                   \
        }                                                                                                         \
    } while (0)

class WorkerPool {
public:
    explicit WorkerPool(int n) {
        for (int i = 0; i < n; ++i)
            threads_.emplace_back([this] {
                for (;;) {
                    std::function<void()> job;
                    {
                        std::unique_lock<std::mutex> lk(m_);
                        cv_.wait(lk, [this] { return stop_ || !q_.empty(); });
                        if (stop_ && q_.empty()) return;
                        job = std::move(q_.front());
                        q_.pop();
                    }
                    job();
                    {
                        std::lock_guard<std::mutex> lk(m_);
                        --pending_;
                    }
                    done_.notify_all();
                }
            });
    }
    ~WorkerPool() {
        { std::lock_guard<std::mutex> lk(m_); stop_ = true; }
        cv_.notify_all();
        for (auto &t : threads_) t.join();
    }
    void submit(std::function<void()> f) {
        { std::lock_guard<std::mutex> lk(m_); q_.push(std::move(f)); ++pending_; }
        cv_.notify_one();
    }
    void waitAll() {
        std::unique_lock<std::mutex> lk(m_);
        done_.wait(lk, [this] { return pending_ == 0; });
    }

private:
    std::vector<std::thread> threads_;
    std::queue<std::function<void()>> q_;
    std::mutex m_;
    std::condition_variable cv_, done_;
    int pending_ = 0;
    bool stop_ = false;
};

template <typename T> struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    cudaError_t alloc(size_t count) { n = count; return cudaMalloc(reinterpret_cast<void **>(&p), sizeof(T) * (count ? count : 1)); }
    void free() { if (p) cudaFree(p); p = nullptr; }
};
template <typename T> struct PinBuf {
    T *p = nullptr;
    size_t n = 0;
    cudaError_t alloc(size_t count) { n = count; return cudaMallocHost(reinterpret_cast<void **>(&p), sizeof(T) * (count ? count : 1)); }
    void free() { if (p) cudaFreeHost(p); p = nullptr; }
};

}  // namespace

struct MvConsts;
static void fillConstsFor(MvConsts &k, int W, int H);

struct mv_engine {
    std::string error;
    void setError(const std::string &e) { error = e; }

    std::string scenarioName;
    int scenario = 0, W = 0, H = 0, E = 0, A = 0, N = 0, threads = 1, device = 0;
    mv::FloatParams params;
    std::vector<std::vector<std::pair<std::string, float>>> shaping;  // per agent view: ordered key list (std::map order)
    std::vector<mv::LevelGenerator> gens;
    std::mt19937 master{std::random_device{}()};
    std::unique_ptr<WorkerPool> pool;

    int gridCells = 0, gridWords = 0;
    int triCap = 368;              // triangle-list capacity of one raster CTA (shared memory); larger views are drawn in several batches
    std::atomic<int> maxObjSeen{0};
    bool wantDepth = false, obsToHost = true, didReset = false, fastShading = true;
    bool hostStepPending = false;  // between mv_step_begin and mv_step_end
    bool skipUnfitLevels = false;  // option "skip_unfit_levels": replace a level that exceeds a fixed capacity by the stream's next one
    std::atomic<int> levelsSkipped{0};
    // host delivery of the obs tensor (host-facing steps).  zero copy (default): the raster kernel stores the rows straight into pinned
    // host memory, the PCIe writes overlap the drawing (measured best from 9 MB to 151 MB per step: 40 GB/s effective at Collect 1024 x 4).
    // Otherwise: rasterise into HBM in host_slices launches, each slice's download on the copy engine while the next is drawn.
    int zeroCopyOpt = 1, hostSlicesOpt = 0;
    bool rasterToHost = false;
    bool deviceObsFresh = false;   // the HBM obs tensor holds the last step's frames (false after a zero-copy host-facing step)
    int sliceCount = 1;            // this launch: > 1 = sliced download on copyStream
    // progressive delivery (option "host_progressive" = slices): ONE raster launch into HBM; the rasteriser counts finished work items per slice
    // of whole envs (d_sliceDone, never reset: the host keeps the running targets), the copy stream waits on each counter in turn
    // (cuStreamWaitValue32) and downloads that slice with the copy engine while the rest of the batch is still being drawn
    int progSlicesOpt = 0, progSlices = 0;
    DevBuf<uint32_t> d_sliceDone;
    uint32_t sliceTarget[16] = {};
    typedef int (*WaitValue32Fn)(cudaStream_t, unsigned long long, unsigned int, unsigned int);
    WaitValue32Fn waitValue32 = nullptr;
    cudaStream_t copyStream = nullptr;
    std::vector<cudaEvent_t> sliceEv;
    int numSMs = 148;
    MvConsts consts{};

    cudaStream_t stream = nullptr;
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
    float lastMs[2] = {0, 0};
    int64_t launches = 0;

    DevBuf<MvLevel> d_levels;
    DevBuf<MvBox> d_statics;       // [E][2][staticCap]
    DevBuf<float> d_staticRot;     // [E][2][staticCap][2]
    int staticCap = MV_INITIAL_STATIC_CAP;  // grows when a generated level has more static boxes (growStatics)
    DevBuf<uint32_t> d_solid;
    DevBuf<uint8_t> d_objGrid;
    DevBuf<MvEnvState> d_envs;
    DevBuf<MvAgent> d_agents;
    DevBuf<MvObject> d_objects;
    DevBuf<MvInstance> d_inst;
    DevBuf<int32_t> d_instCounts;
    DevBuf<float> d_views;
    DevBuf<int32_t> d_actions;
    DevBuf<float> d_rtable;
    DevBuf<float> d_rewards;
    DevBuf<uint8_t> d_dones;
    DevBuf<float> d_trueObj;
    DevBuf<uint8_t> d_obs;
    DevBuf<float> d_depth;
    uint8_t *obsOut = nullptr;     // where the rasteriser writes in HBM: d_obs, or the caller's tensor slice (mv_set_obs_buffer)
    float *depthOut = nullptr;
    DevBuf<int32_t> d_faults;
    // rasteriser (raster_view.cuh): a persistent grid of CTAs pulling (view, band) items from a never-reset counter
    DevBuf<uint32_t> d_workCounter;
    uint32_t counterBase = 0;          // what the counter read before the next launch's first claim
    DevBuf<unsigned long long> d_spill;  // [rasterGrid][spillStride]
    DevBuf<unsigned long long> d_rasterStats;  // mv_debug_raster_stats only
    DevBuf<uint32_t> d_viewCost;       // cost-ordered work queue: [N * H / 4] cost per work item of the current raster launch (N * bands used), [E] env order for the next one, exit counter
    size_t costItems() const { return size_t(N) * size_t(H / 4); }
    int rasterGridCap = 0;             // option "raster_grid": upper bound of the raster grid (0: all CTAs the GPU holds) -- for several engines sharing one GPU
    int rasterSched = 1;               // option "raster_sched": 0 natural order, 1 cost-ordered when the launch has several items per CTA, 2 always
    int rasterGrid = 0, rasterCtasPerSM = 0, spillStride = 0, rasterBands = 1;
    size_t rasterSmem = 0;
    // hi-res pass (draw_hires): its own output buffers, allocated on first use
    struct Hires {
        int W = 0, H = 0;
        DevBuf<uint8_t> d_obs; PinBuf<uint8_t> h_obs;
        DevBuf<unsigned long long> spill;
        void free() { d_obs.free(); h_obs.free(); spill.free(); W = H = 0; }
    } hires;
    DevBuf<MvDeco> d_deco;
    PinBuf<MvDeco> h_deco;
    int decoCap = 1, instCap = MV_DYN_INSTANCES + MV_INITIAL_STATIC_CAP + 1;

    PinBuf<MvLevel> h_levels;      // [E][2] staging mirror
    PinBuf<MvBox> h_statics;       // [E][2][staticCap]
    PinBuf<float> h_staticRot;
    // levels with more static boxes than the arrays hold: parked here by the workers until flushUploads has grown the arrays
    std::vector<std::pair<int, mv::LevelOut>> oversize;
    int wantStaticCap = 0;
    PinBuf<uint32_t> h_solid;      // [E][2][gridWords]
    PinBuf<int32_t> h_actions;
    PinBuf<float> h_rtable;
    PinBuf<float> h_rewards;
    PinBuf<uint8_t> h_dones;
    PinBuf<float> h_trueObj;
    PinBuf<uint8_t> h_obs;
    PinBuf<float> h_depth;
    PinBuf<int32_t> h_faults;
    PinBuf<int32_t> h_faultWord;   // OR of all fault bits raised so far, written by the step kernel (system-scope atomic)

    // mv_step_device pipeline: results of step k are consumed by the host while steps k+1, k+2 already run
    struct Pending { bool valid = false; uint64_t step = 0; cudaEvent_t ev = nullptr; PinBuf<float> rewards, trueObj; PinBuf<uint8_t> dones; };
    std::vector<int64_t> lastAsyncDone;  // [E] asynchronous step index of the env's previous episode end
    bool asyncContractBroken = false;
    Pending ring[3];
    DevBuf<uint32_t> d_prof;  // mv_debug_step_profile only
    DevBuf<uint32_t> d_ready; // per-env step completion stamps (step kernel -> geometry kernel)
    uint32_t readyStamp = 0;
    bool overlap = true;      // geometry kernel launched as a programmatic dependent of the step kernel
    uint64_t asyncSteps = 0;

    std::vector<int> hostSlot, hostEpisode;   // mirrors of the device's live slot / episode index
    std::vector<int> levelWords;              // [E*2] words of the bit planes a staged level uses
    std::vector<int> pendingUpload;           // env ids whose freshly generated next level waits for H2D
    std::vector<std::string> genErrors;
    std::mutex genMutex;
    bool rtableDirty = true;

    // ------------------------------------------------------------------ level generation scheduling
    // generate the level for episode `serial` of env e into staging slot s (worker thread)
    void scheduleGen(int e, int s, int serial) {
        pool->submit([this, e, s, serial] {
            mv::LevelOut out;
            try {
                if (skipUnfitLevels) {
                    const int skipped = gens[size_t(e)].generateFitting(out, serial, gridCells);
                    if (skipped) levelsSkipped.fetch_add(skipped);
                } else {
                    gens[size_t(e)].generate(out, serial, gridCells);
                }
            } catch (const std::exception &ex) {
                std::lock_guard<std::mutex> lk(genMutex);
                genErrors.push_back(ex.what());
                return;
            }
            {
                int curO = maxObjSeen.load();
                while (out.level.n_obj > curO && !maxObjSeen.compare_exchange_weak(curO, out.level.n_obj)) {}
            }
            if (int(out.statics.size()) > staticCap) {  // the arrays are grown on the caller's thread (flushUploads), then the level goes in
                std::lock_guard<std::mutex> lk(genMutex);
                wantStaticCap = std::max(wantStaticCap, int(out.statics.size()));
                oversize.emplace_back(e * 2 + s, std::move(out));
                return;
            }
            stageLevel(e * 2 + s, out);
        });
    }
    // worker thread (or flushUploads for parked levels): copy a generated level into the pinned staging mirrors and queue its upload
    void stageLevel(int id, const mv::LevelOut &out) {
        {
            std::memcpy(&h_levels.p[size_t(id)], &out.level, sizeof(MvLevel));
            if (!out.statics.empty()) {
                std::memcpy(h_statics.p + size_t(id) * size_t(staticCap), out.statics.data(), sizeof(MvBox) * out.statics.size());
                std::memcpy(h_staticRot.p + size_t(id) * size_t(staticCap) * 2, out.staticRot.data(), sizeof(float) * out.staticRot.size());
            }
            const int e = id >> 1, s = id & 1;
            if (!out.deco.empty()) std::memcpy(&h_deco.p[(size_t(e) * 2 + s) * size_t(decoCap)], out.deco.data(), sizeof(MvDeco) * out.deco.size());
            uint32_t *dst = h_solid.p + (size_t(e) * 2 + s) * 3 * gridWords;  // planes: solid, exit, lava
            const size_t nw = std::min(out.solid.size(), size_t(gridWords));
            std::memcpy(dst, out.solid.data(), sizeof(uint32_t) * nw);
            std::memcpy(dst + gridWords, out.exitBits.data(), sizeof(uint32_t) * nw);
            std::memcpy(dst + 2 * size_t(gridWords), out.lavaBits.data(), sizeof(uint32_t) * nw);
            levelWords[size_t(e) * 2 + s] = int(nw);
            std::lock_guard<std::mutex> lk(genMutex);
            pendingUpload.push_back(e * 2 + s);
        }
    }
    // more static boxes per level: re-pitch every array that is laid out by staticCap (level statics, instance lists), device and host
    int growStatics(int need) {
        const int newCap = std::max(staticCap * 2, ((need + 255) / 256) * 256);
        const int newInstCap = MV_DYN_INSTANCES + newCap + decoCap;
        if (newInstCap > mvr::kMaxInstancesPerEnv) { setError("a level needs more drawables than the draw-order key can number"); return MV_ERR_CAPACITY; }
        MV_CUDA(cudaStreamSynchronize(stream));
        DevBuf<MvBox> nStat; DevBuf<float> nRot; DevBuf<MvInstance> nInst; PinBuf<MvBox> hStat; PinBuf<float> hRot;
        const size_t rows = size_t(E) * 2;
        if (nStat.alloc(rows * newCap) != cudaSuccess || nRot.alloc(rows * newCap * 2) != cudaSuccess || nInst.alloc(size_t(E) * newInstCap) != cudaSuccess ||
            hStat.alloc(rows * newCap) != cudaSuccess || hRot.alloc(rows * newCap * 2) != cudaSuccess) {
            nStat.free(); nRot.free(); nInst.free(); hStat.free(); hRot.free();
            setError("growing the static-box arrays: allocation failed");
            return MV_ERR_CUDA;
        }
        MV_CUDA(cudaMemcpy2D(nStat.p, sizeof(MvBox) * newCap, d_statics.p, sizeof(MvBox) * staticCap, sizeof(MvBox) * staticCap, rows, cudaMemcpyDeviceToDevice));
        MV_CUDA(cudaMemcpy2D(nRot.p, sizeof(float) * 2 * newCap, d_staticRot.p, sizeof(float) * 2 * staticCap, sizeof(float) * 2 * staticCap, rows, cudaMemcpyDeviceToDevice));
        MV_CUDA(cudaMemcpy2D(nInst.p, sizeof(MvInstance) * newInstCap, d_inst.p, sizeof(MvInstance) * instCap, sizeof(MvInstance) * instCap, size_t(E), cudaMemcpyDeviceToDevice));
        for (size_t r = 0; r < rows; ++r) {
            std::memcpy(hStat.p + r * newCap, h_statics.p + r * staticCap, sizeof(MvBox) * staticCap);
            std::memcpy(hRot.p + r * newCap * 2, h_staticRot.p + r * staticCap * 2, sizeof(float) * 2 * staticCap);
        }
        d_statics.free(); d_staticRot.free(); d_inst.free(); h_statics.free(); h_staticRot.free();
        d_statics = nStat; d_staticRot = nRot; d_inst = nInst; h_statics = hStat; h_staticRot = hRot;
        staticCap = newCap; instCap = newInstCap;
        return MV_OK;
    }
    int flushUploads() {
        pool->waitAll();
        std::vector<int> todo;
        {
            std::lock_guard<std::mutex> lk(genMutex);
            // sticky: the env whose level could not be generated would otherwise flip to a stale level later; only mv_close recovers
            if (!genErrors.empty()) { setError("level generation failed: " + genErrors.front()); return MV_ERR_CAPACITY; }
        }
        if (!oversize.empty()) {  // workers are idle (waitAll above): grow, then stage what they parked
            const int rc = growStatics(wantStaticCap);
            if (rc) return rc;
            for (auto &po : oversize) stageLevel(po.first, po.second);
            oversize.clear();
            wantStaticCap = 0;
        }
        {
            std::lock_guard<std::mutex> lk(genMutex);
            todo.swap(pendingUpload);
        }
        for (int id : todo) {
            MV_CUDA(cudaMemcpyAsync(&d_levels.p[id], &h_levels.p[id], sizeof(MvLevel), cudaMemcpyHostToDevice, stream));
            if (const int nst = h_levels.p[id].n_static) {
                MV_CUDA(cudaMemcpyAsync(d_statics.p + size_t(id) * size_t(staticCap), h_statics.p + size_t(id) * size_t(staticCap), sizeof(MvBox) * size_t(nst), cudaMemcpyHostToDevice, stream));
                MV_CUDA(cudaMemcpyAsync(d_staticRot.p + size_t(id) * size_t(staticCap) * 2, h_staticRot.p + size_t(id) * size_t(staticCap) * 2, sizeof(float) * 2 * size_t(nst), cudaMemcpyHostToDevice, stream));
            }
            if (h_levels.p[id].n_deco > 0)
                MV_CUDA(cudaMemcpyAsync(&d_deco.p[size_t(id) * size_t(decoCap)], &h_deco.p[size_t(id) * size_t(decoCap)], sizeof(MvDeco) * size_t(h_levels.p[id].n_deco), cudaMemcpyHostToDevice, stream));
            const size_t nw = size_t(levelWords[size_t(id)]);  // only the words this level's grid uses
            for (int plane = 0; plane < ((scenario == MV_SCENARIO_TOWER || scenario == MV_SCENARIO_REARRANGE) ? 1 : 3); ++plane)
                MV_CUDA(cudaMemcpyAsync(d_solid.p + (size_t(id) * 3 + plane) * gridWords, h_solid.p + (size_t(id) * 3 + plane) * gridWords, sizeof(uint32_t) * nw, cudaMemcpyHostToDevice, stream));
        }
        return MV_OK;
    }

    void fillRtableRow(int view) {
        float *row = h_rtable.p + size_t(view) * MV_R_COUNT;
        for (int i = 0; i < MV_R_COUNT; ++i) row[i] = 0.0f;
        for (auto &kv : shaping[size_t(view)]) {
            const int slot = mv::rewardSlot(scenario, kv.first);
            if (slot >= 0) row[slot] = kv.second;
        }
    }

    int launchStep(const int32_t *dActions, bool forceReset, Pending *mirror = nullptr) {
        mvk::StepParams sp;
        sp.hostRewards = mirror ? mirror->rewards.p : nullptr; sp.hostTrueObjectives = mirror ? mirror->trueObj.p : nullptr;
        sp.hostDones = mirror ? mirror->dones.p : nullptr;
        sp.hostFaults = h_faultWord.p;
        sp.levels = d_levels.p; sp.statics = d_statics.p; sp.staticRot = d_staticRot.p; sp.staticCap = staticCap; sp.solid = d_solid.p; sp.objGrid = d_objGrid.p; sp.envs = d_envs.p; sp.agents = d_agents.p;
        sp.objects = d_objects.p; sp.instances = d_inst.p; sp.instCounts = d_instCounts.p; sp.views = d_views.p;
        sp.actions = dActions; sp.rtable = d_rtable.p; sp.rewards = d_rewards.p; sp.dones = d_dones.p; sp.trueObjectives = d_trueObj.p;
        sp.prof = d_prof.p;
        sp.deco = d_deco.p; sp.decoCap = decoCap; sp.instStride = instCap;
        sp.ready = d_ready.p; sp.readyStamp = ++readyStamp;
        sp.envOrder = rasterSched ? d_viewCost.p + costItems() : nullptr;  // a permutation at all times (identity until a cost-ordered raster launch has sorted it)
        sp.maxObj = std::min(int(MV_MAX_OBJECTS), maxObjSeen.load());
        sp.E = E; sp.A = A; sp.gridCells = gridCells; sp.gridWords = gridWords; sp.forceReset = forceReset ? 1 : 0;
        sp.k = consts;
        const int warpsPerBlock = 2;
        const int blocks = (E + warpsPerBlock - 1) / warpsPerBlock;
        const size_t smem = sizeof(mvk::WarpShared) * warpsPerBlock;
        const bool timing = !(mirror && overlap);  // the asynchronous fast path carries no timing events
        if (timing) MV_CUDA(cudaEventRecord(ev[0], stream));
        mvk::stepKernel<<<blocks, warpsPerBlock * 32, smem, stream>>>(sp);
        MV_CUDA(cudaGetLastError());
        if (!overlap) MV_CUDA(cudaEventRecord(ev[1], stream));  // an event between the two kernels would serialise them
        launches += 1;
        int rc = launchRaster();
        if (rc) return rc;
        if (timing) MV_CUDA(cudaEventRecord(ev[2], stream));
        return MV_OK;
    }
    // One persistent launch over all (view, band) items.  Every CTA makes exactly one failing claim when the queue is empty, so the
    // work counter advances by items + grid per launch and the host keeps the base instead of resetting the counter (no memset node
    // between the step kernel and its programmatic dependent).
    int launchView(mvr::ViewParams &vp, int grid, bool dependent) {
        if ((vp.W / 32) * (vp.bandRows / 4) > mvr::kMaxBandTiles) { setError("raster band has more tiles than the bins hold"); return MV_ERR_ARG; }
        vp.workCounter = d_workCounter.p; vp.counterBase = counterBase;
        counterBase += uint32_t(vp.N) * uint32_t(vp.bands) + uint32_t(grid);
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(unsigned(grid)); cfg.blockDim = dim3(mvr::kThreads); cfg.dynamicSmemBytes = rasterSmem; cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = dependent ? 1 : 0;
        if (fastShading) MV_CUDA(cudaLaunchKernelEx(&cfg, mvr::viewKernel<true>, vp));
        else MV_CUDA(cudaLaunchKernelEx(&cfg, mvr::viewKernel<false>, vp));
        launches += 1;
        return MV_OK;
    }
    // the cost-ordered queue starts in natural order
    cudaError_t resetViewOrder() {
        std::vector<uint32_t> init(costItems() + size_t(E) + 1, 0u);  // item costs, env order, exit counter
        for (int e = 0; e < E; ++e) init[costItems() + size_t(e)] = uint32_t(e);
        return cudaMemcpy(d_viewCost.p, init.data(), sizeof(uint32_t) * init.size(), cudaMemcpyHostToDevice);
    }
    int launchRaster() {
        mvr::ViewParams vp = {};
        vp.instances = d_inst.p; vp.instCounts = d_instCounts.p; vp.views = d_views.p; vp.instStride = instCap;
        // pinned allocations are mapped into the device address space (UVA), so the kernel can store through the host pointer
        vp.obs = rasterToHost ? h_obs.p : obsOut; vp.depth = wantDepth ? (rasterToHost ? h_depth.p : depthOut) : nullptr;
        vp.spill = d_spill.p; vp.spillStride = spillStride; vp.consumed = nullptr; vp.stats = d_rasterStats.p;
        vp.A = A; vp.W = W; vp.H = H; vp.bands = rasterBands; vp.bandRows = ((H / 4 + rasterBands - 1) / rasterBands) * 4; vp.triCap = triCap;
        vp.p00 = consts.p00; vp.p11 = consts.p11; vp.p22 = consts.p22; vp.p32 = consts.p32;
        // programmatic dependent launch: the grid may start before the step kernel has drained; a CTA waits for its env's stamp
        vp.ready = overlap ? d_ready.p : nullptr; vp.readyStamp = overlap ? readyStamp : 0;
        deviceObsFresh = !rasterToHost;
        if (sliceCount <= 1) {
            vp.viewBase = 0; vp.N = N;
            const int grid = std::min(rasterGridCap > 0 ? std::min(rasterGrid, rasterGridCap) : rasterGrid, N * rasterBands);
            if (rasterSched == 2 || (rasterSched == 1 && N * rasterBands > grid)) {  // more work items than CTAs: their order matters
                vp.viewCost = d_viewCost.p; vp.order = d_viewCost.p + costItems(); vp.exitCounter = d_viewCost.p + costItems() + size_t(E);
            }
            if (progSlices > 0) { vp.sliceDone = d_sliceDone.p; vp.envsPerSlice = (E + progSlices - 1) / progSlices; }
            const int rcl = launchView(vp, grid, overlap);
            if (rcl || progSlices <= 0) return rcl;
            // downloads: slice k as soon as all of its work items are drawn (cyclic >= comparison on the device counter)
            const size_t px = size_t(W) * H;
            for (int k = 0, e0 = 0; e0 < E; ++k, e0 += vp.envsPerSlice) {
                const int envs = std::min(vp.envsPerSlice, E - e0);
                sliceTarget[k] += uint32_t(envs) * uint32_t(A) * uint32_t(rasterBands);
                if (waitValue32(copyStream, (unsigned long long)(uintptr_t)(d_sliceDone.p + k), sliceTarget[k], 1u /* CU_STREAM_WAIT_VALUE_GEQ */) != 0) {
                    setError("cuStreamWaitValue32 failed");
                    return MV_ERR_CUDA;
                }
                const size_t v0 = size_t(e0) * A, cnt = size_t(envs) * A;
                MV_CUDA(cudaMemcpyAsync(h_obs.p + v0 * px * 4, obsOut + v0 * px * 4, cnt * px * 4, cudaMemcpyDeviceToHost, copyStream));
                if (wantDepth) MV_CUDA(cudaMemcpyAsync(h_depth.p + v0 * px, depthOut + v0 * px, sizeof(float) * cnt * px, cudaMemcpyDeviceToHost, copyStream));
            }
            return MV_OK;
        }
        // sliced download: whole envs per slice; slice s is copied down by the copy engine while slice s+1 is rasterised
        const size_t px = size_t(W) * H;
        const int perSlice = ((E + sliceCount - 1) / sliceCount) * A;
        for (int base = 0, si = 0; base < N; base += perSlice, ++si) {
            const int cnt = std::min(perSlice, N - base);
            vp.viewBase = base; vp.N = cnt;
            const int rc = launchView(vp, std::min(rasterGrid, cnt * rasterBands), overlap && si == 0);
            if (rc) return rc;
            while (int(sliceEv.size()) <= si) { cudaEvent_t e2; MV_CUDA(cudaEventCreateWithFlags(&e2, cudaEventDisableTiming)); sliceEv.push_back(e2); }
            MV_CUDA(cudaEventRecord(sliceEv[size_t(si)], stream));
            MV_CUDA(cudaStreamWaitEvent(copyStream, sliceEv[size_t(si)], 0));
            MV_CUDA(cudaMemcpyAsync(h_obs.p + size_t(base) * px * 4, obsOut + size_t(base) * px * 4, size_t(cnt) * px * 4, cudaMemcpyDeviceToHost, copyStream));
            if (wantDepth) MV_CUDA(cudaMemcpyAsync(h_depth.p + size_t(base) * px, depthOut + size_t(base) * px, sizeof(float) * size_t(cnt) * px, cudaMemcpyDeviceToHost, copyStream));
        }
        return MV_OK;
    }
    // decide how this host-facing launch delivers its frames
    void chooseDelivery(bool copyObs) {
        progSlices = 0;
        if (copyObs && progSlicesOpt > 0 && waitValue32 && d_sliceDone.p) { rasterToHost = false; sliceCount = 1; progSlices = std::min({progSlicesOpt, E, 16}); return; }
        const int d = copyObs ? hostDelivery() : 1;
        rasterToHost = copyObs && d == 0; sliceCount = std::max(1, d);
    }
    // how a host-facing step delivers its obs: returns the slice count (0 = zero-copy stores, 1 = one copy after the raster)
    int hostDelivery() const {
        const size_t bytes = size_t(N) * W * H * (wantDepth ? 8 : 4);
        const bool zc = zeroCopyOpt != 0;
        if (zc) return 0;
        if (hostSlicesOpt > 0) return std::min(hostSlicesOpt, E);
        return int(std::max<size_t>(1, std::min<size_t>({size_t(2), size_t(E), bytes / (size_t(32) << 20)})));  // two slices measured best at 151 MB
    }
    // draw_hires (megaverse.cpp:154-177): every agent view once more, at (w, h), from the instance lists and camera matrices of
    // the last step -- the same kernel over row bands of the large frame.  Result in hires.h_obs, uint8[N][h][w][4].
    int drawHires(int w, int hgt) {
        if (!didReset) { setError("mv_draw_hires before mv_reset"); return MV_ERR_STATE; }
        if (w < 32 || hgt < 4 || (w % 32) || (hgt % 4) || w > 4096 || hgt > 4096) { setError("hi-res size must be a multiple of 32 x 4"); return MV_ERR_ARG; }
        int rc = drain();
        if (rc) return rc;
        // bands of about a hundred 32x4 tiles each
        const int tilesX = w / 32, tileRows = hgt / 4;
        const int rowsPerBand = std::max(1, 96 / tilesX) * 4;
        const int bands = (hgt + rowsPerBand - 1) / rowsPerBand;
        const int stride = w * rowsPerBand;
        (void)tileRows;
        if (hires.W != w || hires.H != hgt) {
            hires.free();
            const size_t px = size_t(N) * w * hgt * 4;
            if (hires.d_obs.alloc(px) != cudaSuccess || hires.h_obs.alloc(px) != cudaSuccess || hires.spill.alloc(size_t(rasterGrid) * size_t(stride)) != cudaSuccess) {
                hires.free();
                setError("hi-res buffers: allocation failed");
                return MV_ERR_CUDA;
            }
            hires.W = w; hires.H = hgt;
        }
        MvConsts k;
        fillConstsFor(k, w, hgt);
        mvr::ViewParams vp = {};
        vp.instances = d_inst.p; vp.instCounts = d_instCounts.p; vp.views = d_views.p; vp.instStride = instCap;
        vp.obs = hires.d_obs.p; vp.depth = nullptr; vp.spill = hires.spill.p; vp.spillStride = stride; vp.consumed = nullptr;
        vp.viewBase = 0; vp.N = N; vp.A = A; vp.W = w; vp.H = hgt; vp.bands = bands; vp.bandRows = rowsPerBand; vp.triCap = triCap;
        vp.p00 = k.p00; vp.p11 = k.p11; vp.p22 = k.p22; vp.p32 = k.p32;
        vp.ready = nullptr; vp.readyStamp = 0;
        rc = launchView(vp, std::min(rasterGrid, N * bands), false);
        if (rc) return rc;
        MV_CUDA(cudaMemcpyAsync(hires.h_obs.p, hires.d_obs.p, size_t(N) * w * hgt * 4, cudaMemcpyDeviceToHost, stream));
        MV_CUDA(cudaStreamSynchronize(stream));
        return MV_OK;
    }
    // shared-memory carve-up, occupancy and the per-CTA spill slabs for the current triangle-list capacity / band count
    int configureRaster() {
        if (stream) cudaStreamSynchronize(stream);
        rasterSmem = mvr::smemLayout(triCap).total;
        int maxOptin = 0;
        MV_CUDA(cudaDeviceGetAttribute(&maxOptin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
        if (int(rasterSmem) > maxOptin) { setError("tri_cap needs more shared memory than an SM has"); return MV_ERR_ARG; }
        for (int fast = 0; fast < 2; ++fast) {
            const void *fn = fast ? reinterpret_cast<const void *>(mvr::viewKernel<true>) : reinterpret_cast<const void *>(mvr::viewKernel<false>);
            MV_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, maxOptin));  // per function, not per engine: allow the device maximum
            int perSM = 0;
            MV_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, fn, mvr::kThreads, rasterSmem));
            if (perSM < 1) { setError("raster kernel does not fit on an SM with this tri_cap"); return MV_ERR_CUDA; }
            rasterCtasPerSM = fast ? std::min(rasterCtasPerSM, perSM) : perSM;
        }
        rasterGrid = numSMs * rasterCtasPerSM;
        const int bandRows = ((H / 4 + rasterBands - 1) / rasterBands) * 4;
        spillStride = W * bandRows;
        d_spill.free();
        if (d_spill.alloc(size_t(rasterGrid) * size_t(spillStride)) != cudaSuccess) { setError("raster spill slab allocation failed"); return MV_ERR_CUDA; }
        hires.free();  // its spill slab is sized by the grid
        return MV_OK;
    }

    // after a step (or forced reset): flip host mirrors for finished envs and start generating the level after next
    void afterFlip(const uint8_t *flipped) {
        for (int e = 0; e < E; ++e) {
            if (!flipped || flipped[e]) {
                hostSlot[size_t(e)] ^= 1;
                hostEpisode[size_t(e)] += 1;
                scheduleGen(e, hostSlot[size_t(e)] ^ 1, hostEpisode[size_t(e)] + 1);
            }
        }
    }

    // per-kernel times exist only when the kernels run back to back (overlap off); with the dependent launch the step and
    // geometry kernels overlap and only their union is meaningful: {-1, whole step}
    void readKernelTimes() {
        if (cudaEventQuery(ev[2]) != cudaSuccess) return;
        if (overlap) { lastMs[0] = -1.0f; cudaEventElapsedTime(&lastMs[1], ev[0], ev[2]); }
        else { cudaEventElapsedTime(&lastMs[0], ev[0], ev[1]); cudaEventElapsedTime(&lastMs[1], ev[1], ev[2]); }
    }

    int finishStep(bool copyObs, bool wait = true) {
        MV_CUDA(cudaMemcpyAsync(h_rewards.p, d_rewards.p, sizeof(float) * N, cudaMemcpyDeviceToHost, stream));
        MV_CUDA(cudaMemcpyAsync(h_dones.p, d_dones.p, E, cudaMemcpyDeviceToHost, stream));
        MV_CUDA(cudaMemcpyAsync(h_trueObj.p, d_trueObj.p, sizeof(float) * N, cudaMemcpyDeviceToHost, stream));
        if (copyObs && !rasterToHost && sliceCount <= 1 && progSlices <= 0) {
            MV_CUDA(cudaMemcpyAsync(h_obs.p, obsOut, size_t(N) * W * H * 4, cudaMemcpyDeviceToHost, stream));
            if (wantDepth) MV_CUDA(cudaMemcpyAsync(h_depth.p, depthOut, sizeof(float) * size_t(N) * W * H, cudaMemcpyDeviceToHost, stream));
        }
        if (!wait) return MV_OK;
        MV_CUDA(cudaStreamSynchronize(stream));
        if (sliceCount > 1 || progSlices > 0) MV_CUDA(cudaStreamSynchronize(copyStream));
        readKernelTimes();
        return MV_OK;
    }

    // consume one finished asynchronous step: publish its host copies, flip mirrors, schedule level generation
    int retire(Pending &p) {
        if (!p.valid) return MV_OK;
        MV_CUDA(cudaEventSynchronize(p.ev));
        std::memcpy(h_rewards.p, p.rewards.p, sizeof(float) * N);
        std::memcpy(h_dones.p, p.dones.p, E);
        std::memcpy(h_trueObj.p, p.trueObj.p, sizeof(float) * N);
        p.valid = false;
        // the pre-staged next level of an env is delivered three calls after its episode ended: an env that finishes again sooner
        // flipped to a stale level on the device (MV_FAULT_LEVEL_NOT_READY is latched there as well) -- refuse to go on
        if (lastAsyncDone.empty()) lastAsyncDone.assign(size_t(E), -1000);
        for (int e = 0; e < E; ++e)
            if (h_dones.p[e]) {
                if (int64_t(p.step) - lastAsyncDone[size_t(e)] < 3) asyncContractBroken = true;
                lastAsyncDone[size_t(e)] = int64_t(p.step);
            }
        afterFlip(h_dones.p);
        if (asyncContractBroken) { setError("mv_step_device: an episode lasted fewer than 3 steps -- outside the asynchronous call's contract; use mv_step"); return MV_ERR_STATE; }
        return MV_OK;
    }
    int drain() {
        for (int k = 0; k < 3; ++k) {  // oldest first
            const int rc = retire(ring[(asyncSteps + k) % 3]);
            if (rc) return rc;
        }
        return MV_OK;
    }
    // asynchronous device-resident step: returns after enqueueing.  Episode bookkeeping lags two steps, which is safe
    // because an env cannot finish twice within four steps (doneWithTimer leaves 0.3 s = 4.5 steps, scenario.hpp:114-117)
    int stepAsync(const int32_t *dActions) {
        if (!didReset) { setError("mv_step_device before mv_reset"); return MV_ERR_STATE; }
        if (hostStepPending) { const int rcp = stepEnd(); if (rcp) return rcp; }
        if (asyncContractBroken) { setError("mv_step_device: an episode lasted fewer than 3 steps -- outside the asynchronous call's contract; use mv_step"); return MV_ERR_STATE; }
        Pending &slotP = ring[asyncSteps % 3];
        // levels generated since the previous call go up first (done at step k-3 -> retired at call k-1 -> uploaded ahead
        // of kernel k; that env cannot flip again before step k+1), then step k-2 is retired and its regeneration jobs
        // run on the worker pool while this call's kernels are enqueued
        int rc = flushUploads();
        if (rc) return rc;
        rc = retire(ring[(asyncSteps + 1) % 3]);
        if (rc) return rc;
        rc = retire(slotP);  // only if the ring wrapped without retiring
        if (rc) return rc;
        if (rtableDirty) {
            MV_CUDA(cudaMemcpyAsync(d_rtable.p, h_rtable.p, sizeof(float) * N * MV_R_COUNT, cudaMemcpyHostToDevice, stream));
            rtableDirty = false;
        }
        rasterToHost = false; sliceCount = 1; progSlices = 0;
        rc = launchStep(dActions, false, &slotP);  // rewards / dones / true objectives land in the ring slot straight from the kernel
        if (rc) return rc;
        MV_CUDA(cudaEventRecord(slotP.ev, stream));
        slotP.valid = true;
        slotP.step = asyncSteps;
        ++asyncSteps;
        return MV_OK;
    }

    int stepCommon(const int32_t *dActions, bool copyObs, bool split = false) {
        if (!didReset) { setError("mv_step before mv_reset"); return MV_ERR_STATE; }
        if (hostStepPending) { setError("mv_step_begin is outstanding: call mv_step_end first"); return MV_ERR_STATE; }
        int rc = drain();
        if (rc) return rc;
        rc = flushUploads();
        if (rc) return rc;
        if (rtableDirty) {
            MV_CUDA(cudaMemcpyAsync(d_rtable.p, h_rtable.p, sizeof(float) * N * MV_R_COUNT, cudaMemcpyHostToDevice, stream));
            rtableDirty = false;
        }
        chooseDelivery(copyObs);
        rc = launchStep(dActions, false);
        if (rc) return rc;
        rc = finishStep(copyObs, !split);
        if (rc) return rc;
        if (split) { hostStepPending = true; return MV_OK; }
        afterFlip(h_dones.p);
        return MV_OK;
    }
    // second half of a split host-facing step (mv_step_begin / mv_step_end): wait for the copies enqueued by stepCommon(split)
    int stepEnd() {
        if (!hostStepPending) { setError("mv_step_end without mv_step_begin"); return MV_ERR_STATE; }
        MV_CUDA(cudaStreamSynchronize(stream));
        if (sliceCount > 1 || progSlices > 0) MV_CUDA(cudaStreamSynchronize(copyStream));
        readKernelTimes();
        hostStepPending = false;
        std::memset(h_actions.p, 0, sizeof(int32_t) * N);  // env.cpp:140-142: actions are cleared after every step
        afterFlip(h_dones.p);
        return MV_OK;
    }

    void freeAll() {
        if (pool) { pool->waitAll(); pool.reset(); }
        d_levels.free(); d_statics.free(); d_staticRot.free(); h_statics.free(); h_staticRot.free(); d_solid.free(); d_objGrid.free(); d_envs.free(); d_agents.free(); d_objects.free(); d_inst.free(); d_instCounts.free();
        d_views.free(); d_actions.free(); d_rtable.free(); d_rewards.free(); d_dones.free(); d_trueObj.free(); d_obs.free(); d_depth.free(); d_faults.free();
        hires.free(); d_deco.free(); h_deco.free(); d_prof.free(); d_ready.free(); d_workCounter.free(); d_spill.free(); d_rasterStats.free(); d_viewCost.free(); d_sliceDone.free();
        h_levels.free(); h_solid.free(); h_actions.free(); h_rtable.free(); h_rewards.free(); h_dones.free(); h_trueObj.free(); h_obs.free(); h_depth.free();
        h_faults.free(); h_faultWord.free();
        for (auto &e : ev) if (e) { cudaEventDestroy(e); e = nullptr; }
        for (auto &p : ring) { if (p.ev) { cudaEventDestroy(p.ev); p.ev = nullptr; } p.rewards.free(); p.trueObj.free(); p.dones.free(); }
        for (auto &e2 : sliceEv) if (e2) cudaEventDestroy(e2);
        sliceEv.clear();
        if (copyStream) { cudaStreamDestroy(copyStream); copyStream = nullptr; }
        if (stream) { cudaStreamDestroy(stream); stream = nullptr; }
    }
};

namespace {

const uint32_t kPaletteRgb[22] = {0xffdd3c, 0x3bb372, 0x50c878, 0x2eb5d0, 0xadd8e6, 0x3a7fa6, 0x2c3e50, 0xffb400, 0xb3b3b3, 0x555555, 0x222222,
                                  0xffffff, 0xff0000, 0xffa770, 0xd468ee, 0xffe6e6, 0xffffe6, 0xccffcc, 0xe6ecff, 0xd9d9d9, 0xf2e6ff, 0xffebcc};

int uploadPalette(mv_engine *h) {
    float pal[22][3];
    for (int i = 0; i < 22; ++i) {  // toRgbf: byte / 255 (util/magnum.hpp:25-32)
        pal[i][0] = float((kPaletteRgb[i] >> 16) & 255) / 255.0f;
        pal[i][1] = float((kPaletteRgb[i] >> 8) & 255) / 255.0f;
        pal[i][2] = float(kPaletteRgb[i] & 255) / 255.0f;
    }
    cudaError_t err = cudaMemcpyToSymbol(mvr::c_palette, pal, sizeof(pal));
    if (err != cudaSuccess) { h->setError(std::string("palette upload: ") + cudaGetErrorString(err)); return MV_ERR_CUDA; }
    return MV_OK;
}

void fillConsts(MvConsts &k, int W, int H) {
    k.dt = 1.0f / 15.0f;                              // env.hpp:160-161
    mvh::yawBasis(3.5f * k.dt, k.look_left);          // agent.cpp:100-108,128-133
    mvh::yawBasis(-3.5f * k.dt, k.look_right);
    k.max_slope_cos = mvh::crcos(45.0f * (3.14159265358979323846f / 180.0f));
    const float aspect = float(W) / float(H);
    const float halfTan = mvh::crtan((100.0f * 0.01745329251994329576923690768489f) / 2.0f);
    const float nearZ = 0.01f, farZ = 120.0f;
    k.p00 = 1.0f / halfTan;
    k.p11 = -aspect / halfTan;
    k.p22 = farZ / (nearZ - farZ);
    k.p32 = farZ * nearZ / (nearZ - farZ);
}

}  // namespace
static void fillConstsFor(MvConsts &k, int W, int H) { fillConsts(k, W, H); }
namespace {

int setKernelAttrs(mv_engine *h) {
    cudaError_t err = cudaFuncSetAttribute(mvk::stepKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(mvk::WarpShared) * 4));
    if (err != cudaSuccess) { h->setError(std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(err)); return MV_ERR_CUDA; }
    return MV_OK;
}

}  // namespace

extern "C" {

const char *mv_last_error(mv_handle h) { return h ? h->error.c_str() : g_createError.c_str(); }

int mv_create(const char *scenario, int w, int h, int num_envs, int num_agents, int num_threads, int device, const char *const *keys, const float *vals,
              int nparams, mv_handle *out) {
    if (!out) return MV_ERR_ARG;
    *out = nullptr;
    const int sc = scenario ? mv::scenarioFromName(scenario) : -1;
    if (sc < 0) { g_createError = std::string("unknown scenario ") + (scenario ? scenario : "(null)"); return MV_ERR_ARG; }
    if (w <= 0 || h <= 0 || w % 32 != 0 || h % 4 != 0 || (w / 32) * (h / 4) > mvr::kMaxBandTiles) { g_createError = "render size must be a multiple of 32x4 with at most 128 tiles"; return MV_ERR_ARG; }
    if (num_envs <= 0 || num_agents <= 0 || num_agents > MV_MAX_AGENTS) { g_createError = "bad num_envs / num_agents_per_env"; return MV_ERR_ARG; }
    for (int i = 0; i < nparams; ++i) {
        if (!keys || !keys[i] || !vals) { g_createError = "null parameter key / value array"; return MV_ERR_ARG; }
        // the interactive viewer's reward-indicator HUD (scenario_default.hpp:144-160, set by viewer_app.cpp:147 only) adds drawables this
        // engine does not draw: refuse instead of rendering frames that differ from the reference's
        if (std::string(keys[i]) == "useUIRewardIndicators" && vals[i] > 0.0f) {
            g_createError = "useUIRewardIndicators > 0 (the viewer's reward-indicator HUD) is not supported";
            return MV_ERR_ARG;
        }
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { g_createError = "no CUDA device: megaverse_b200 has no CPU fallback"; return MV_ERR_CUDA; }
    if (device < 0 || device >= ndev) { g_createError = "bad CUDA device ordinal"; return MV_ERR_ARG; }
    auto *e = new mv_engine;
    auto fail = [&](int code) { g_createError = e->error; e->freeAll(); delete e; return code; };
    DeviceGuard dg__(device);
    if (!dg__.ok) { e->setError("cudaSetDevice failed"); return fail(MV_ERR_CUDA); }
    e->scenario = sc; e->W = w; e->H = h; e->E = num_envs; e->A = num_agents; e->N = num_envs * num_agents; e->device = device;
    e->threads = num_threads < 1 ? 1 : num_threads;
    e->scenarioName = scenario;
    e->params = mv::defaultFloatParams(e->scenarioName);
    for (int i = 0; i < nparams; ++i) e->params[keys[i]] = vals[i];
    {
        auto def = mv::defaultRewardShaping(e->scenarioName);
        std::map<std::string, float> m{{"teamSpirit", 0.0f}};
        for (auto &kv : def) m[kv.first] = kv.second;
        std::vector<std::pair<std::string, float>> ordered(m.begin(), m.end());
        e->shaping.assign(size_t(e->N), ordered);
    }
    try {
        for (int i = 0; i < e->E; ++i) e->gens.emplace_back(e->scenarioName, e->A, e->params);
    } catch (const std::exception &ex) {  // e.g. Sokoban without a Boxoban dataset (the reference exit()s here, scenario_sokoban.cpp:76-78)
        e->setError(ex.what());
        return fail(MV_ERR_ARG);
    }
    e->levelWords.assign(size_t(e->E) * 2, 0);
    e->pool.reset(new WorkerPool(e->threads));
    e->gridCells = mv::gridCapacity(sc);
    e->decoCap = mv::decoCapacity(sc);
    e->instCap = MV_DYN_INSTANCES + e->staticCap + e->decoCap;
    e->gridWords = e->gridCells / 32;
    fillConsts(e->consts, w, h);

    auto ck = [&](cudaError_t err, const char *what) { if (err != cudaSuccess) { e->setError(std::string(what) + ": " + cudaGetErrorString(err)); return false; } return true; };
    const size_t E = size_t(e->E), N = size_t(e->N), px = size_t(w) * h;
    bool ok = ck(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking), "stream") && ck(cudaStreamCreateWithFlags(&e->copyStream, cudaStreamNonBlocking), "copy stream");
    for (auto &evx : e->ev) ok = ok && ck(cudaEventCreate(&evx), "event");
    ok = ok && ck(e->d_levels.alloc(E * 2), "levels") && ck(e->d_statics.alloc(E * 2 * size_t(e->staticCap)), "statics") && ck(e->d_staticRot.alloc(E * 2 * size_t(e->staticCap) * 2), "staticRot") &&
         ck(e->h_statics.alloc(E * 2 * size_t(e->staticCap)), "h_statics") && ck(e->h_staticRot.alloc(E * 2 * size_t(e->staticCap) * 2), "h_staticRot") && ck(e->d_solid.alloc(E * 2 * 3 * e->gridWords), "solid") && ck(e->d_objGrid.alloc(E * e->gridCells), "objGrid") &&
         ck(e->d_envs.alloc(E), "envs") && ck(e->d_agents.alloc(N), "agents") && ck(e->d_objects.alloc(E * MV_MAX_OBJECTS), "objects") &&
         ck(e->d_inst.alloc(E * size_t(e->instCap)), "instances") && ck(e->d_deco.alloc(E * 2 * size_t(e->decoCap)), "deco") && ck(e->h_deco.alloc(E * 2 * size_t(e->decoCap)), "h_deco") && ck(e->d_instCounts.alloc(E * 8), "instCounts") && ck(e->d_views.alloc(N * 16), "views") &&
         ck(e->d_actions.alloc(N), "actions") && ck(e->d_rtable.alloc(N * MV_R_COUNT), "rtable") && ck(e->d_rewards.alloc(N), "rewards") &&
         ck(e->d_dones.alloc(E), "dones") && ck(e->d_trueObj.alloc(N), "trueObj") && ck(e->d_obs.alloc(N * px * 4), "obs") && ck(e->d_faults.alloc(E), "faults") &&
         ck(e->d_workCounter.alloc(4), "workCounter") && ck(cudaMemset(e->d_workCounter.p, 0, 16), "workCounter") &&
         ck(e->d_sliceDone.alloc(16), "sliceDone") && ck(cudaMemset(e->d_sliceDone.p, 0, 64), "sliceDone") &&
         ck(e->d_viewCost.alloc(e->costItems() + size_t(E) + 1), "viewCost") && ck(e->resetViewOrder(), "viewOrder") && ck(e->d_ready.alloc(E), "ready") &&
         ck(cudaMemset(e->d_ready.p, 0, sizeof(uint32_t) * size_t(E)), "ready");
    { cudaDeviceProp prop; if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) e->numSMs = prop.multiProcessorCount; }
    {   // stream memory operation of the driver API (no link dependency on libcuda): the copy stream of the progressive delivery waits on it
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &fn, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess && fn)
            e->waitValue32 = reinterpret_cast<mv_engine::WaitValue32Fn>(fn);
        else
            (void)cudaGetLastError();
    }
    if (e->instCap > mvr::kMaxInstancesPerEnv) { e->setError("instance capacity exceeds the draw-order key range"); return fail(MV_ERR_CAPACITY); }
    // few views: split every view into row bands so that the persistent grid (2 CTAs per SM) has something to balance.  With the
    // cost-ordered queue finer items pay up to about two views per CTA (measured: 256 views 3 bands 0.128 ms per step, 2 bands 0.144, 6 bands
    // 0.144; 512 views 2 bands 0.169, 1 band 0.188; 1024 views 1 band 0.241, 2 bands 0.273 -- every band repeats the view's geometry)
    e->rasterBands = N <= 320 ? 3 : (N <= 640 ? 2 : 1);
    while (e->rasterBands > 1 && (h / 4) % e->rasterBands) --e->rasterBands;
    if (ok && e->configureRaster() != MV_OK) return fail(MV_ERR_CUDA);
    ok = ok && ck(e->h_levels.alloc(E * 2), "h_levels") && ck(e->h_solid.alloc(E * 2 * 3 * e->gridWords), "h_solid") && ck(e->h_actions.alloc(N), "h_actions") &&
         ck(e->h_rtable.alloc(N * MV_R_COUNT), "h_rtable") && ck(e->h_rewards.alloc(N), "h_rewards") && ck(e->h_dones.alloc(E), "h_dones") &&
         ck(e->h_trueObj.alloc(N), "h_trueObj") && ck(e->h_obs.alloc(N * px * 4), "h_obs") && ck(e->h_faults.alloc(E), "h_faults") && ck(e->h_faultWord.alloc(1), "h_faultWord");
    for (auto &p : e->ring) ok = ok && ck(cudaEventCreateWithFlags(&p.ev, cudaEventDisableTiming), "event") && ck(p.rewards.alloc(N), "ring") && ck(p.trueObj.alloc(N), "ring") && ck(p.dones.alloc(E), "ring");
    if (!ok) return fail(MV_ERR_CUDA);
    std::memset(e->h_actions.p, 0, sizeof(int32_t) * N);
    e->h_faultWord.p[0] = 0;
    std::memset(e->h_rewards.p, 0, sizeof(float) * N);
    std::memset(e->h_dones.p, 0, E);
    std::memset(e->h_trueObj.p, 0, sizeof(float) * N);
    std::memset(e->h_obs.p, 0, N * px * 4);
    for (size_t v = 0; v < N; ++v) e->fillRtableRow(int(v));
    ok = ck(cudaMemset(e->d_trueObj.p, 0, sizeof(float) * N), "memset") && ck(cudaMemset(e->d_faults.p, 0, sizeof(int32_t) * E), "memset") &&
         ck(cudaMemset(e->d_actions.p, 0, sizeof(int32_t) * N), "memset") && ck(cudaMemset(e->d_agents.p, 0, sizeof(MvAgent) * N), "memset") &&
         ck(cudaMemset(e->d_objects.p, 0, sizeof(MvObject) * E * MV_MAX_OBJECTS), "memset");
    if (!ok) return fail(MV_ERR_CUDA);
    e->obsOut = e->d_obs.p;
    if (uploadPalette(e) != MV_OK) return fail(MV_ERR_CUDA);
    if (setKernelAttrs(e) != MV_OK) return fail(MV_ERR_CUDA);
    *out = e;
    return MV_OK;
}

int mv_set_option(mv_handle h, const char *key, int value) {
    if (!h || !key) return MV_ERR_ARG;
    const std::string k = key;
    if (k == "depth") {
        if (h->didReset) { h->setError("option depth must be set before the first reset"); return MV_ERR_STATE; }
        h->wantDepth = value != 0;
        if (h->wantDepth && !h->d_depth.p) {
            const size_t cnt = size_t(h->N) * h->W * h->H;
            if (h->d_depth.alloc(cnt) != cudaSuccess || h->h_depth.alloc(cnt) != cudaSuccess) { h->setError("depth allocation failed"); return MV_ERR_CUDA; }
            if (!h->depthOut) h->depthOut = h->d_depth.p;
        }
        return MV_OK;
    }
    if (k == "tri_cap") {  // triangles a raster CTA keeps in shared memory; views with more are drawn in several batches
        if (value < 32 || value > mvr::kMaxTriCap) { h->setError("tri_cap out of range [32,1022]"); return MV_ERR_ARG; }
        const int old = h->triCap;
        h->triCap = value;
        const int rc = h->configureRaster();
        if (rc) { h->triCap = old; h->configureRaster(); }
        return rc;
    }
    if (k == "static_cap") {  // initial size of the per-level static-box arrays (they grow on demand; tests start small to exercise that)
        if (h->didReset) { h->setError("option static_cap must be set before the first reset"); return MV_ERR_STATE; }
        if (value < 1 || value > (1 << 20)) return MV_ERR_ARG;
        const size_t rows = size_t(h->E) * 2;
        h->d_statics.free(); h->d_staticRot.free(); h->h_statics.free(); h->h_staticRot.free(); h->d_inst.free();
        h->staticCap = value;
        h->instCap = MV_DYN_INSTANCES + h->staticCap + h->decoCap;
        if (h->d_statics.alloc(rows * value) != cudaSuccess || h->d_staticRot.alloc(rows * value * 2) != cudaSuccess || h->h_statics.alloc(rows * value) != cudaSuccess ||
            h->h_staticRot.alloc(rows * value * 2) != cudaSuccess || h->d_inst.alloc(size_t(h->E) * size_t(h->instCap)) != cudaSuccess) {
            h->setError("static_cap: allocation failed");
            return MV_ERR_CUDA;
        }
        return MV_OK;
    }
    if (k == "raster_bands") {  // row bands per view (each band is one work item of the persistent raster grid)
        if (value < 1 || value > h->H / 4 || (h->H / 4) % value) { h->setError("raster_bands must divide the number of 4-pixel tile rows"); return MV_ERR_ARG; }
        h->rasterBands = value;
        return h->configureRaster();
    }
    if (k == "raster_sched") {  // work order of the persistent raster grid: 0 natural, 1 cost-ordered for launches with several views per CTA, 2 always
        if (value < 0 || value > 2) return MV_ERR_ARG;
        cudaStreamSynchronize(h->stream);
        h->rasterSched = value;
        return h->resetViewOrder() == cudaSuccess ? MV_OK : MV_ERR_CUDA;
    }
    if (k == "raster_grid") {  // CTAs of the persistent raster grid (0 = as many as the GPU holds): engines that share a GPU take a share each
        if (value < 0) return MV_ERR_ARG;
        cudaStreamSynchronize(h->stream);
        h->rasterGridCap = value;
        return MV_OK;
    }
    if (k == "host_progressive") {  // slices of the progressive host delivery (0 = off): one raster launch, the copy engine follows it slice by slice
        if (value < 0 || value > 16) return MV_ERR_ARG;
        if (value > 0 && !h->waitValue32) { h->setError("host_progressive: cuStreamWaitValue32 is not available"); return MV_ERR_STATE; }
        h->progSlicesOpt = value;
        return MV_OK;
    }
    if (k == "obs_to_host") { h->obsToHost = value != 0; return MV_OK; }
    if (k == "zero_copy") { h->zeroCopyOpt = value != 0; return MV_OK; }
    if (k == "host_slices") { if (value < 0 || value > 64) return MV_ERR_ARG; h->hostSlicesOpt = value; return MV_OK; }
    if (k == "skip_unfit_levels") { h->skipUnfitLevels = value != 0; return MV_OK; }
    if (k == "fast_shading") { h->fastShading = value != 0; return MV_OK; }
    if (k == "overlap") { cudaStreamSynchronize(h->stream); h->overlap = value != 0; return MV_OK; }
    h->setError("unknown option " + k);
    return MV_ERR_ARG;
}

static void regenerateNext(mv_handle h) {
    // (re)build every env's pre-staged next level from its current RNG state
    for (int e = 0; e < h->E; ++e) h->scheduleGen(e, h->hostSlot[size_t(e)] ^ 1, h->hostEpisode[size_t(e)] + 1);
}

static void ensureMirrors(mv_handle h) {
    if (h->hostSlot.empty()) {
        h->hostSlot.assign(size_t(h->E), 1);      // first flip lands on slot 0
        h->hostEpisode.assign(size_t(h->E), -1);  // ... as episode 0
    }
}

int mv_seed(mv_handle h, int seed) {
    if (!h) return MV_ERR_ARG;
    h->pool->waitAll();
    h->master.seed((unsigned long)seed);
    for (int e = 0; e < h->E; ++e) h->gens[size_t(e)].seed((unsigned long)std::uniform_int_distribution<>{0, (1 << 30) - 1}(h->master));
    if (h->didReset) {  // the staged next levels were drawn from the old streams: redo them
        { std::lock_guard<std::mutex> lk(h->genMutex); h->pendingUpload.clear(); }
        regenerateNext(h);
    }
    return MV_OK;
}

int mv_seed_env(mv_handle h, int env, int seed) {
    if (!h || env < 0 || env >= h->E) return MV_ERR_ARG;
    h->pool->waitAll();
    h->gens[size_t(env)].seed((unsigned long)seed);
    if (h->didReset) h->scheduleGen(env, h->hostSlot[size_t(env)] ^ 1, h->hostEpisode[size_t(env)] + 1);
    return MV_OK;
}

int mv_reset(mv_handle h) {
    if (!h) return MV_ERR_ARG;
    DeviceGuard dg__(h->device);
    if (!dg__.ok) { h->setError("cudaSetDevice failed"); return MV_ERR_CUDA; }
    ensureMirrors(h);
    if (h->hostStepPending) { const int rcp = h->stepEnd(); if (rcp) return rcp; }
    if (h->didReset) { const int rcd = h->drain(); if (rcd) return rcd; }
    if (!h->didReset) {
        // initial device state: slot 1 / episode -1 so that the forced flip lands on (slot 0, episode 0)
        std::vector<MvEnvState> init(size_t(h->E));
        std::memset(init.data(), 0, sizeof(MvEnvState) * init.size());
        for (auto &s : init) { s.slot = 1; s.episode_idx = -1; mvBzInit(s); }
        if (cudaMemcpy(h->d_envs.p, init.data(), sizeof(MvEnvState) * init.size(), cudaMemcpyHostToDevice) != cudaSuccess) { h->setError("env init upload failed"); return MV_ERR_CUDA; }
        regenerateNext(h);
        h->didReset = true;
    }
    int rc = h->flushUploads();
    if (rc) return rc;
    if (h->rtableDirty) {
        if (cudaMemcpyAsync(h->d_rtable.p, h->h_rtable.p, sizeof(float) * h->N * MV_R_COUNT, cudaMemcpyHostToDevice, h->stream) != cudaSuccess) { h->setError("rtable upload failed"); return MV_ERR_CUDA; }
        h->rtableDirty = false;
    }
    h->chooseDelivery(h->obsToHost);
    rc = h->launchStep(h->d_actions.p, true);
    if (rc) return rc;
    rc = h->finishStep(h->obsToHost);
    if (rc) return rc;
    h->afterFlip(nullptr);
    return MV_OK;
}

int32_t mv_encode_action(const int32_t *heads6) {  // megaverse.cpp:100-116 with Env::actionSpaceSizes {3,3,3,2,2,3}
    static const int sizes[6] = {3, 3, 3, 2, 2, 3};
    int idx = 0, mask = 0;
    for (int i = 0; i < 6; ++i) {
        if (heads6[i] > 0) mask |= 1 << (idx + heads6[i]);
        idx += sizes[i] - 1;
    }
    return mask;
}

int mv_set_actions(mv_handle h, const int32_t *masks) {
    if (!h || !masks) return MV_ERR_ARG;
    std::memcpy(h->h_actions.p, masks, sizeof(int32_t) * h->N);
    return MV_OK;
}

int mv_step(mv_handle h) {
    if (!h) return MV_ERR_ARG;
    DeviceGuard dg__(h->device);
    if (!dg__.ok) { h->setError("cudaSetDevice failed"); return MV_ERR_CUDA; }
    if (!h->didReset) { h->setError("mv_step before mv_reset"); return MV_ERR_STATE; }
    if (h->hostStepPending) { h->setError("mv_step_begin is outstanding: call mv_step_end first"); return MV_ERR_STATE; }
    if (cudaMemcpyAsync(h->d_actions.p, h->h_actions.p, sizeof(int32_t) * h->N, cudaMemcpyHostToDevice, h->stream) != cudaSuccess) { h->setError("actions upload failed"); return MV_ERR_CUDA; }
    const int rc = h->stepCommon(h->d_actions.p, h->obsToHost);
    if (rc) cudaStreamSynchronize(h->stream);  // the upload may still be reading the pinned masks
    std::memset(h->h_actions.p, 0, sizeof(int32_t) * h->N);  // env.cpp:140-142: actions are cleared after every step
    return rc;
}

int mv_step_begin(mv_handle h) {
    if (!h) return MV_ERR_ARG;
    DeviceGuard dg__(h->device);
    if (!dg__.ok) { h->setError("cudaSetDevice failed"); return MV_ERR_CUDA; }
    if (cudaMemcpyAsync(h->d_actions.p, h->h_actions.p, sizeof(int32_t) * h->N, cudaMemcpyHostToDevice, h->stream) != cudaSuccess) { h->setError("actions upload failed"); return MV_ERR_CUDA; }
    return h->stepCommon(h->d_actions.p, h->obsToHost, true);
}

int mv_step_end(mv_handle h) {
    if (!h) return MV_ERR_ARG;
    DeviceGuard dg__(h->device);
    if (!dg__.ok) { h->setError("cudaSetDevice failed"); return MV_ERR_CUDA; }
    return h->stepEnd();
}

int mv_step_device(mv_handle h, const int32_t *d_masks) {
    if (!h) return MV_ERR_ARG;
    DeviceGuard dg__(h->device);
    if (!dg__.ok) { h->setError("cudaSetDevice failed"); return MV_ERR_CUDA; }
    return h->stepAsync(d_masks ? d_masks : h->d_actions.p);
}

// host-only: the colour tables of the level generators followed by the rasteriser's palette (float bit patterns), in the layout of
// the oracle's / reference shim's *_color_tables
int mv_debug_color_tables(uint32_t *out, int cap) {
    std::vector<uint32_t> o = mv::colorTables();
    for (int i = 0; i < 22; ++i)
        for (float f : {float((kPaletteRgb[i] >> 16) & 255) / 255.0f, float((kPaletteRgb[i] >> 8) & 255) / 255.0f, float(kPaletteRgb[i] & 255) / 255.0f}) {
            uint32_t u; std::memcpy(&u, &f, 4); o.push_back(u);
        }
    if (int(o.size()) > cap) return -int(o.size());
    std::copy(o.begin(), o.end(), out);
    return int(o.size());
}

// host-only: a scenario's default reward shaping (as mv_create builds it) and default float parameters, as text
// "R key=bits\n" / "P key=bits\n" lines in key order, float values as 8 hex digits
int mv_debug_defaults(const char *scenario, char *out, int cap) {
    if (!scenario || mv::scenarioFromName(scenario) < 0) return MV_ERR_ARG;
    std::map<std::string, float> m{{"teamSpirit", 0.0f}};
    for (auto &kv : mv::defaultRewardShaping(scenario)) m[kv.first] = kv.second;
    std::string text;
    char line[160];
    auto put = [&](char tag, const std::string &k, float v) {
        uint32_t u; std::memcpy(&u, &v, 4);
        std::snprintf(line, sizeof(line), "%c %s=%08x\n", tag, k.c_str(), u);
        text += line;
    };
    for (auto &kv : m) put('R', kv.first, kv.second);
    for (auto &kv : mv::defaultFloatParams(scenario)) put('P', kv.first, kv.second);
    if (int(text.size()) + 1 > cap) return -int(text.size()) - 1;
    std::memcpy(out, text.c_str(), text.size() + 1);
    return int(text.size());
}

// host-only: how many levels of the env stream (seed env_seed) up to and including `episode` generateFitting had to skip, or < 0
int mv_debug_count_unfit_levels(const char *scenario, int num_agents, int env_seed, int episodes, const char *const *keys, const float *vals, int nparams) {
    if (!scenario || mv::scenarioFromName(scenario) < 0 || num_agents < 1 || num_agents > MV_MAX_AGENTS) return MV_ERR_ARG;
    try {
        mv::FloatParams params = mv::defaultFloatParams(scenario);
        for (int i = 0; i < nparams; ++i) params[keys[i]] = vals[i];
        mv::LevelGenerator gen(scenario, num_agents, params);
        gen.seed((unsigned long)env_seed);
        mv::LevelOut lo;
        int skipped = 0;
        for (int ep = 0; ep < episodes; ++ep) skipped += gen.generateFitting(lo, ep, 1 << 30);
        return skipped;
    } catch (const std::exception &ex) { g_createError = ex.what(); return MV_ERR_CAPACITY; }
}

int mv_levels_skipped(mv_handle h) { return h ? h->levelsSkipped.load() : MV_ERR_ARG; }

int mv_draw_hires(mv_handle h, int w, int hgt, const uint8_t **out) {
    if (!h) return MV_ERR_ARG;
    DeviceGuard dg__(h->device);
    if (!dg__.ok) { h->setError("cudaSetDevice failed"); return MV_ERR_CUDA; }
    const int rc = h->drawHires(w, hgt);
    if (rc) return rc;
    if (out) *out = h->hires.h_obs.p;
    return MV_OK;
}

int mv_fetch_obs(mv_handle h) {
    if (!h) return MV_ERR_ARG;
    DeviceGuard dg__(h->device);
    if (!dg__.ok) { h->setError("cudaSetDevice failed"); return MV_ERR_CUDA; }
    if (h->hostStepPending) { const int rcp = h->stepEnd(); if (rcp) return rcp; }
    const int rc = h->drain();
    if (rc) return rc;
    if (!h->deviceObsFresh) return MV_OK;  // the last step stored its frames straight into the host buffer: that copy is the newer one
    const size_t px = size_t(h->N) * h->W * h->H;
    if (cudaMemcpyAsync(h->h_obs.p, h->obsOut, px * 4, cudaMemcpyDeviceToHost, h->stream) != cudaSuccess) { h->setError("obs download failed"); return MV_ERR_CUDA; }
    if (h->wantDepth && cudaMemcpyAsync(h->h_depth.p, h->depthOut, px * sizeof(float), cudaMemcpyDeviceToHost, h->stream) != cudaSuccess) { h->setError("depth download failed"); return MV_ERR_CUDA; }
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) { h->setError("stream sync failed"); return MV_ERR_CUDA; }
    return MV_OK;
}

int mv_debug_step_profile(mv_handle h, uint32_t *out, int enable) {
    if (!h) return MV_ERR_ARG;
    DeviceGuard dg__(h->device);
    if (!dg__.ok) return MV_ERR_CUDA;
    cudaStreamSynchronize(h->stream);
    if (enable && !h->d_prof.p) {
        if (h->d_prof.alloc(size_t(h->E) * 16) != cudaSuccess) { h->setError("profile buffer allocation failed"); return MV_ERR_CUDA; }
        cudaMemset(h->d_prof.p, 0, sizeof(uint32_t) * size_t(h->E) * 16);
    }
    if (out && h->d_prof.p && cudaMemcpy(out, h->d_prof.p, sizeof(uint32_t) * size_t(h->E) * 16, cudaMemcpyDeviceToHost) != cudaSuccess) return MV_ERR_CUDA;
    if (!enable) h->d_prof.free();
    return MV_OK;
}

int mv_sync(mv_handle h) {
    if (!h) return MV_ERR_ARG;
    DeviceGuard dg__(h->device);
    if (!dg__.ok) { h->setError("cudaSetDevice failed"); return MV_ERR_CUDA; }
    const int rc = h->drain();
    if (rc) return rc;
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) { h->setError("stream sync failed"); return MV_ERR_CUDA; }
    h->readKernelTimes();
    return MV_OK;
}

int mv_obs_host(mv_handle h, const uint8_t **out) { if (!h || !out) return MV_ERR_ARG; *out = h->h_obs.p; return MV_OK; }
int mv_depth_host(mv_handle h, const float **out) { if (!h || !out || !h->wantDepth) return MV_ERR_ARG; *out = h->h_depth.p; return MV_OK; }
int mv_rewards(mv_handle h, const float **out) { if (!h || !out) return MV_ERR_ARG; *out = h->h_rewards.p; return MV_OK; }
int mv_dones(mv_handle h, const uint8_t **out) { if (!h || !out) return MV_ERR_ARG; *out = h->h_dones.p; return MV_OK; }
int mv_true_objectives(mv_handle h, const float **out) { if (!h || !out) return MV_ERR_ARG; *out = h->h_trueObj.p; return MV_OK; }
int mv_set_obs_buffer(mv_handle h, uint8_t *d_obs, float *d_depth) {
    if (!h) return MV_ERR_ARG;
    DeviceGuard dg__(h->device);
    if (!dg__.ok) { h->setError("cudaSetDevice failed"); return MV_ERR_CUDA; }
    // the pointer is a launch parameter: steps already enqueued keep writing the previous buffer, the next step writes the new one.  No
    // synchronisation here (a consumer that double-buffers its tensor switches every step); mv_sync before freeing a buffer.
    h->obsOut = d_obs ? d_obs : h->d_obs.p;
    h->depthOut = d_depth ? d_depth : h->d_depth.p;
    return MV_OK;
}
int mv_actions_device(mv_handle h, int32_t **p) { if (!h || !p) return MV_ERR_ARG; *p = h->d_actions.p; return MV_OK; }
int mv_obs_device(mv_handle h, uint8_t **p) {
    if (!h || !p) return MV_ERR_ARG;
    if (h->didReset && !h->deviceObsFresh) { h->setError("the last step delivered its frames to the host buffer only (zero-copy): the HBM tensor is stale; use mv_step_device or option zero_copy=0"); return MV_ERR_STATE; }
    *p = h->obsOut;
    return MV_OK;
}
int mv_depth_device(mv_handle h, float **p) {
    if (!h || !p || !h->wantDepth) return MV_ERR_ARG;
    if (h->didReset && !h->deviceObsFresh) { h->setError("the last step delivered its frames to the host buffer only (zero-copy): the HBM tensor is stale"); return MV_ERR_STATE; }
    *p = h->depthOut;
    return MV_OK;
}
int mv_rewards_device(mv_handle h, float **p) { if (!h || !p) return MV_ERR_ARG; *p = h->d_rewards.p; return MV_OK; }
int mv_dones_device(mv_handle h, uint8_t **p) { if (!h || !p) return MV_ERR_ARG; *p = h->d_dones.p; return MV_OK; }
int mv_stream(mv_handle h, void **s) { if (!h || !s) return MV_ERR_ARG; *s = h->stream; return MV_OK; }

int mv_get_reward_shaping(mv_handle h, int env, int agent, const char **keys, float *vals, int cap, int *n) {
    if (!h || env < 0 || env >= h->E || agent < 0 || agent >= h->A || !n) return MV_ERR_ARG;
    auto &rs = h->shaping[size_t(env) * h->A + agent];
    *n = int(rs.size());
    for (int i = 0; i < int(rs.size()) && i < cap; ++i) { keys[i] = rs[size_t(i)].first.c_str(); vals[i] = rs[size_t(i)].second; }
    return MV_OK;
}

int mv_set_reward_shaping(mv_handle h, int env, int agent, const char *const *keys, const float *vals, int n) {
    if (!h || env < 0 || env >= h->E || agent < 0 || agent >= h->A) return MV_ERR_ARG;
    // Scenario::setRewardShaping replaces the whole map (scenario.hpp:215); a scheme lacking a key the scenario reads
    // makes the reference throw std::out_of_range at the next reward event (scenario.hpp:253) -> reject it up front
    std::map<std::string, float> m;
    for (int i = 0; i < n; ++i) m[keys[i]] = vals[i];
    for (auto &kv : mv::defaultRewardShaping(h->scenarioName))
        if (!m.count(kv.first)) { h->setError("reward shaping lacks key " + kv.first); return MV_ERR_ARG; }
    const size_t view = size_t(env) * h->A + agent;
    h->shaping[view].assign(m.begin(), m.end());
    h->fillRtableRow(int(view));
    h->rtableDirty = true;
    return MV_OK;
}

int mv_faults(mv_handle h, int32_t *out) {
    if (!h || !out) return MV_ERR_ARG;
    if (h->stream) cudaStreamSynchronize(h->stream);
    std::vector<MvEnvState> st(size_t(h->E));
    if (cudaMemcpy(st.data(), h->d_envs.p, sizeof(MvEnvState) * st.size(), cudaMemcpyDeviceToHost) != cudaSuccess) return MV_ERR_CUDA;
    if (cudaMemcpy(h->h_faults.p, h->d_faults.p, sizeof(int32_t) * h->E, cudaMemcpyDeviceToHost) != cudaSuccess) return MV_ERR_CUDA;
    int32_t f = 0;
    for (int e = 0; e < h->E; ++e) f |= st[size_t(e)].faults | h->h_faults.p[e];
    *out = f;
    return MV_OK;
}
// totals since enable: {work items, instances read, instances with visible items, items, clipped items, triangles, batches, item
// sub-passes, six thread-0 cycle counts, (tile, triangle) pairs kept by the binning, pairs in the triangles' pixel boxes}
int mv_debug_raster_stats(mv_handle h, unsigned long long *out16, int enable) {
    if (!h) return MV_ERR_ARG;
    DeviceGuard dg__(h->device);
    if (!dg__.ok) return MV_ERR_CUDA;
    cudaStreamSynchronize(h->stream);
    if (out16 && h->d_rasterStats.p && cudaMemcpy(out16, h->d_rasterStats.p, 128, cudaMemcpyDeviceToHost) != cudaSuccess) return MV_ERR_CUDA;
    if (enable && !h->d_rasterStats.p) {
        if (h->d_rasterStats.alloc(16) != cudaSuccess) { h->setError("raster stats allocation failed"); return MV_ERR_CUDA; }
    }
    if (enable) cudaMemset(h->d_rasterStats.p, 0, 128);
    else h->d_rasterStats.free();
    return MV_OK;
}
int mv_debug_static_cap(mv_handle h) { return h ? h->staticCap : MV_ERR_ARG; }  // current size of the per-level static-box arrays
int mv_debug_raster_config(mv_handle h, int32_t *out4) {  // {persistent grid, CTAs per SM, dynamic shared memory bytes, row bands per view}
    if (!h || !out4) return MV_ERR_ARG;
    out4[0] = h->rasterGrid; out4[1] = h->rasterCtasPerSM; out4[2] = int32_t(h->rasterSmem); out4[3] = h->rasterBands;
    return MV_OK;
}
int mv_fault_word(mv_handle h, int32_t *out) {  // no device round trip: the step kernel ORs raised bits into pinned host memory
    if (!h || !out) return MV_ERR_ARG;
    *out = *const_cast<volatile int32_t *>(h->h_faultWord.p);
    return MV_OK;
}
int mv_kernel_launches(mv_handle h, int64_t *out) { if (!h || !out) return MV_ERR_ARG; *out = h->launches; return MV_OK; }
int mv_last_kernel_ms(mv_handle h, float *out2) { if (!h || !out2) return MV_ERR_ARG; out2[0] = h->lastMs[0]; out2[1] = h->lastMs[1]; return MV_OK; }

int mv_close(mv_handle h) {
    if (!h) return MV_ERR_ARG;
    DeviceGuard dg__(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    h->freeAll();
    delete h;
    return MV_OK;
}

// ------------------------------------------------------------------------------------------------ introspection (tests)
// reward-object voxels; for the hexagonal mazes the free-standing colliders instead (bit patterns of centre, half extents, orientation)
static void dumpLevelExtras(const MvLevel &L, const MvBox *statics, const float *staticRot, std::vector<int32_t> &o) {
    const bool hex = L.scenario == MV_SCENARIO_HEX_EXPLORE || L.scenario == MV_SCENARIO_HEX_MEMORY || L.scenario == MV_SCENARIO_EMPTY;
    o.push_back(hex ? 0 : L.n_reward);
    for (int i = 0; i < L.n_reward && !hex; ++i) for (int a = 0; a < 3; ++a) o.push_back(L.reward_voxel[i][a]);
    if (!hex) return;
    o.push_back(L.n_static);
    for (int i = 0; i < L.n_static; ++i) {
        const MvBox &b = statics[i];
        const float rot[2] = {(b.flags & MV_ROTATED) ? staticRot[i * 2] : 1.0f, (b.flags & MV_ROTATED) ? staticRot[i * 2 + 1] : 0.0f};
        int32_t w[8];
        std::memcpy(w, b.c, 12); std::memcpy(w + 3, b.h, 12); std::memcpy(w + 6, rot, 8);
        for (int k = 0; k < 8; ++k) o.push_back(w[k]);
    }
}

int mv_debug_get_level(mv_handle h, int env, int32_t *out, int cap) {
    if (!h || env < 0 || env >= h->E || !h->didReset) return MV_ERR_ARG;
    const size_t lid = size_t(env) * 2 + h->hostSlot[size_t(env)];
    const MvLevel &L = h->h_levels.p[lid];
    const MvBox *statics = h->h_statics.p + lid * size_t(h->staticCap);
    const float *staticRot = h->h_staticRot.p + lid * size_t(h->staticCap) * 2;
    std::vector<int32_t> o;
    o.push_back(L.n_grid_static); o.push_back(L.n_terrain); o.push_back(L.n_obj);
    for (int a = 0; a < 3; ++a) o.push_back(L.bz_min[a]);
    for (int a = 0; a < 3; ++a) o.push_back(L.bz_max[a]);
    static const uint32_t pal[22] = {0xffdd3c, 0x3bb372, 0x50c878, 0x2eb5d0, 0xadd8e6, 0x3a7fa6, 0x2c3e50, 0xffb400, 0xb3b3b3, 0x555555, 0x222222,
                                     0xffffff, 0xff0000, 0xffa770, 0xd468ee, 0xffe6e6, 0xffffe6, 0xccffcc, 0xe6ecff, 0xd9d9d9, 0xf2e6ff, 0xffebcc};
    for (int i = 0; i < L.n_grid_static; ++i) {
        const MvBox &b = statics[i];
        // invert centre/half back to inclusive voxel bounds: min = c - h, max = c + h - 1
        const float vs = L.scenario == MV_SCENARIO_SOKOBAN ? 2.0f : 1.0f;  // voxel size of the scenario's grid
        for (int a = 0; a < 3; ++a) o.push_back(int(lroundf((b.c[a] - b.h[a]) / vs)));
        for (int a = 0; a < 3; ++a) o.push_back(int(lroundf((b.c[a] + b.h[a]) / vs)) - 1);
        o.push_back(b.flags & 255); o.push_back(int(pal[b.color]));
    }
    for (int i = 0; i < L.n_terrain; ++i) {
        o.push_back(L.terrain[i].type);
        for (int a = 0; a < 6; ++a) o.push_back(L.terrain[i].bb[a]);
    }
    for (int i = 0; i < L.n_obj; ++i) for (int a = 0; a < 3; ++a) o.push_back(L.obj_init[i].voxel[a]);
    for (int i = 0; i < h->A; ++i) for (int a = 0; a < 3; ++a) o.push_back(int(L.init_pos[i][a]));
    if (L.scenario != MV_SCENARIO_TOWER) {
        o.push_back(L.n_movable);  // numPlatforms
        dumpLevelExtras(L, statics, staticRot, o);
    }
    if (int(o.size()) > cap) return -int(o.size());
    std::memcpy(out, o.data(), o.size() * sizeof(int32_t));
    return int(o.size());
}

int mv_debug_get_state(mv_handle h, int env, float *out, int cap) {
    if (!h || env < 0 || env >= h->E || !h->didReset) return MV_ERR_ARG;
    MvEnvState es;
    std::vector<MvAgent> ag(size_t(h->A));
    std::vector<MvObject> ob(MV_MAX_OBJECTS);
    cudaStreamSynchronize(h->stream);
    if (cudaMemcpy(&es, &h->d_envs.p[env], sizeof es, cudaMemcpyDeviceToHost) != cudaSuccess) return MV_ERR_CUDA;
    if (cudaMemcpy(ag.data(), &h->d_agents.p[size_t(env) * h->A], sizeof(MvAgent) * h->A, cudaMemcpyDeviceToHost) != cudaSuccess) return MV_ERR_CUDA;
    if (cudaMemcpy(ob.data(), &h->d_objects.p[size_t(env) * MV_MAX_OBJECTS], sizeof(MvObject) * MV_MAX_OBJECTS, cudaMemcpyDeviceToHost) != cudaSuccess) return MV_ERR_CUDA;
    const MvLevel &L = h->h_levels.p[size_t(env) * 2 + es.slot];
    std::vector<float> o;
    int ncol = h->A + L.n_obj;
    const MvBox *statics = h->h_statics.p + (size_t(env) * 2 + es.slot) * size_t(h->staticCap);
    for (int i = 0; i < L.n_static; ++i) ncol += (statics[i].flags & MV_SOLID) ? 1 : 0;
    const float len = L.episode_len;
    o.push_back(es.episode_sec); o.push_back(len); o.push_back(float(es.num_frames)); o.push_back(float(es.highest_tower));
    o.push_back(es.bz_reward); o.push_back(float(L.n_obj)); o.push_back(float(ncol)); o.push_back(0.f);
    for (int i = 0; i < h->A; ++i) {
        const MvAgent &a = ag[size_t(i)];
        for (int k = 0; k < 3; ++k) o.push_back(a.pos[k]);
        for (int k = 0; k < 9; ++k) o.push_back(a.basis[k]);
        for (int k = 0; k < 3; ++k) o.push_back(a.hvel[k]);
        for (float x : {a.vvel, a.voff, a.step_off, a.was_on_ground ? 1.f : 0.f, a.was_jumping ? 1.f : 0.f, a.jump_speed, a.cur_x, float(a.carrying), a.total_reward,
                        h->h_rewards.p[size_t(env) * h->A + i], 0.f})
            o.push_back(x);
    }
    for (int i = 0; i < L.n_obj; ++i) {
        const MvObject &b = ob[size_t(i)];
        float t[3] = {b.t[0], b.t[1], b.t[2]};
        if (b.parent >= 0) {  // absolute translation of a carried object: ((agent*camera)*pickup)*local, as the oracle reports it
            const MvAgent &a = ag[size_t(b.parent)];
            mvh::M4 objT, cam;
            std::memcpy(&objT.c[0][0], a.object_t, 64); std::memcpy(&cam.c[0][0], a.cam_local, 64);
            const mvh::M4 pick = mvh::mul(mvh::translation(0.0f, -0.44f, -1.0f), mvh::identity());
            const mvh::M4 local = mvh::mul(mvh::translation(b.t[0], b.t[1], b.t[2]), mvh::mul(mvh::scaling(b.s[0], b.s[1], b.s[2]), mvh::identity()));
            const mvh::M4 abs = mvh::mul(mvh::mul(mvh::mul(objT, cam), pick), local);
            t[0] = abs.c[3][0]; t[1] = abs.c[3][1]; t[2] = abs.c[3][2];
        }
        for (float x : {t[0], t[1], t[2], b.s[0], b.s[1], b.s[2], float(b.parent), b.enabled ? 1.f : 0.f, 0.f}) o.push_back(x);
    }
    if (L.scenario != MV_SCENARIO_TOWER) {
        o.push_back(float(es.solved)); o.push_back(float(L.scenario == MV_SCENARIO_HEX_MEMORY ? uint32_t(es.positive_collected) : es.reached_exit));
        for (int w = 0; w < 3; ++w) o.push_back(float(es.reward_alive[w] & 0xffffffu)), o.push_back(float(es.reward_alive[w] >> 24));
    }
    if (int(o.size()) > cap) return -int(o.size());
    std::memcpy(out, o.data(), o.size() * sizeof(float));
    return int(o.size());
}

int mv_debug_get_voxels(mv_handle h, int env, int32_t *out, int cap) {
    if (!h || env < 0 || env >= h->E || !h->didReset) return MV_ERR_ARG;
    MvEnvState es;
    cudaStreamSynchronize(h->stream);
    if (cudaMemcpy(&es, &h->d_envs.p[env], sizeof es, cudaMemcpyDeviceToHost) != cudaSuccess) return MV_ERR_CUDA;
    const MvLevel &L = h->h_levels.p[size_t(env) * 2 + es.slot];
    const uint32_t *sol = h->h_solid.p + (size_t(env) * 2 + es.slot) * 3 * h->gridWords;
    const MvBox *statics = h->h_statics.p + (size_t(env) * 2 + es.slot) * size_t(h->staticCap);
    std::vector<uint8_t> og(size_t(h->gridCells));
    if (cudaMemcpy(og.data(), h->d_objGrid.p + size_t(env) * h->gridCells, og.size(), cudaMemcpyDeviceToHost) != cudaSuccess) return MV_ERR_CUDA;
    // opacity is a property of the box a solid voxel belongs to
    std::vector<std::array<int32_t, 4>> v;
    for (int x = 0; x < L.grid_dim[0]; ++x)
        for (int y = 0; y < L.grid_dim[1]; ++y)
            for (int z = 0; z < L.grid_dim[2]; ++z) {
                const int idx = (x * L.grid_dim[1] + y) * L.grid_dim[2] + z;
                int flags = 0;
                if ((sol[idx >> 5] >> (idx & 31)) & 1u) {
                    flags |= 1;
                    const float vs = L.scenario == MV_SCENARIO_SOKOBAN ? 2.0f : 1.0f;
                    const float cx = (x + L.grid_org[0] + 0.5f) * vs, cy = (y + L.grid_org[1] + 0.5f) * vs, cz = (z + L.grid_org[2] + 0.5f) * vs;
                    for (int i = 0; i < L.n_grid_static; ++i) {
                        const MvBox &b = statics[i];
                        if (fabsf(cx - b.c[0]) < b.h[0] && fabsf(cy - b.c[1]) < b.h[1] && fabsf(cz - b.c[2]) < b.h[2]) { flags |= (b.flags & MV_OPAQUE); break; }
                    }
                }
                if (og[size_t(idx)] != MV_NO_OBJECT) flags |= 4;
                if ((sol[size_t(h->gridWords) + (idx >> 5)] >> (idx & 31)) & 1u) flags |= 1 << 8;
                if ((sol[2 * size_t(h->gridWords) + (idx >> 5)] >> (idx & 31)) & 1u) flags |= 2 << 8;
                if (flags) v.push_back({x + L.grid_org[0], y + L.grid_org[1], z + L.grid_org[2], flags});
            }
    std::sort(v.begin(), v.end());
    if (int(v.size()) * 4 > cap) return -int(v.size()) * 4;
    for (size_t i = 0; i < v.size(); ++i) std::memcpy(out + i * 4, v[i].data(), 16);
    return int(v.size()) * 4;
}

int mv_debug_get_instances(mv_handle h, int env, float *out, int cap) {
    if (!h || env < 0 || env >= h->E || !h->didReset) return MV_ERR_ARG;
    int32_t cnt[8];
    cudaStreamSynchronize(h->stream);
    if (cudaMemcpy(cnt, h->d_instCounts.p + size_t(env) * 8, 32, cudaMemcpyDeviceToHost) != cudaSuccess) return MV_ERR_CUDA;
    std::vector<MvInstance> inst(static_cast<size_t>(cnt[1] > 0 ? cnt[1] : 1));
    if (cudaMemcpy(inst.data(), h->d_inst.p + size_t(env) * size_t(h->instCap), sizeof(MvInstance) * inst.size(), cudaMemcpyDeviceToHost) != cudaSuccess) return MV_ERR_CUDA;
    if (cnt[1] * 18 > cap) return -cnt[1] * 18;
    for (int i = 0; i < cnt[1]; ++i) {
        out[i * 18] = float(inst[size_t(i)].mesh); out[i * 18 + 1] = float(inst[size_t(i)].color);
        std::memcpy(out + i * 18 + 2, inst[size_t(i)].model, 64);
    }
    return cnt[1] * 18;
}

int mv_debug_get_view(mv_handle h, int env, int agent, float *out16) {
    if (!h || env < 0 || env >= h->E || agent < 0 || agent >= h->A || !h->didReset) return MV_ERR_ARG;
    cudaStreamSynchronize(h->stream);
    if (cudaMemcpy(out16, h->d_views.p + (size_t(env) * h->A + agent) * 16, 64, cudaMemcpyDeviceToHost) != cudaSuccess) return MV_ERR_CUDA;
    return MV_OK;
}

int mv_debug_render_instances(const float *view16, const float *inst18, int n, int w, int h, uint8_t *rgba, float *depth) {
    if (!view16 || !inst18 || n < 0 || n > 4096 || w % 32 || h % 4 || (w / 32) * (h / 4) > mvr::kMaxBandTiles) return MV_ERR_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return MV_ERR_CUDA;
    // instances must arrive boxes-first (draw order); count the leading boxes
    std::vector<MvInstance> inst(size_t(n ? n : 1));
    int nBox = 0;
    for (int i = 0; i < n; ++i) {
        inst[size_t(i)].mesh = int(inst18[i * 18]); inst[size_t(i)].color = int(inst18[i * 18 + 1]);
        std::memcpy(inst[size_t(i)].model, inst18 + i * 18 + 2, 64);
        if (inst[size_t(i)].mesh == 0) { if (nBox != i) return MV_ERR_ARG; ++nBox; }
    }
    mv_engine tmp;  // only for the constants / palette
    MvConsts k;
    fillConsts(k, w, h);
    if (uploadPalette(&tmp) != MV_OK) return MV_ERR_CUDA;
    int32_t cnt[8] = {nBox, n, 0, 0, 0, 0, 0, 0};
    {   // instances must be sorted by mesh type (draw order)
        int last = 0;
        for (int i = 0; i < n; ++i) {
            const int m = inst[size_t(i)].mesh;
            if (m < last || m > 4) return MV_ERR_ARG;
            last = m;
            if (m >= 1) cnt[1 + m] += 1;
        }
    }
    // a small triangle list on purpose: scenes of a few hundred triangles exercise the multi-batch path
    const int triCap = 96;
    const size_t smem = mvr::smemLayout(triCap).total;
    MvInstance *dInst = nullptr; int32_t *dCnt = nullptr; float *dView = nullptr, *dDepth = nullptr; uint8_t *dObs = nullptr;
    uint32_t *dCtr = nullptr; unsigned long long *dSpill = nullptr;
    const int bands = (h / 4) % 2 == 0 ? 2 : 1, bandRows = (h / 4 / bands) * 4;
    bool ok = cudaMalloc(&dInst, sizeof(MvInstance) * inst.size()) == cudaSuccess && cudaMalloc(&dCnt, 32) == cudaSuccess &&
              cudaMalloc(&dView, 64) == cudaSuccess && cudaMalloc(&dObs, size_t(w) * h * 4) == cudaSuccess && cudaMalloc(&dDepth, size_t(w) * h * 4) == cudaSuccess &&
              cudaMalloc(&dCtr, 16) == cudaSuccess && cudaMalloc(&dSpill, sizeof(unsigned long long) * size_t(bands) * size_t(w) * bandRows) == cudaSuccess &&
              cudaFuncSetAttribute(mvr::viewKernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)) == cudaSuccess;
    if (ok) {
        cudaMemcpy(dInst, inst.data(), sizeof(MvInstance) * inst.size(), cudaMemcpyHostToDevice);
        cudaMemcpy(dCnt, cnt, 32, cudaMemcpyHostToDevice);
        cudaMemcpy(dView, view16, 64, cudaMemcpyHostToDevice);
        cudaMemset(dCtr, 0, 16);
        mvr::ViewParams vp = {};
        vp.instances = dInst; vp.instCounts = dCnt; vp.views = dView; vp.instStride = int(inst.size()); vp.obs = dObs; vp.depth = depth ? dDepth : nullptr;
        vp.workCounter = dCtr; vp.counterBase = 0; vp.ready = nullptr; vp.readyStamp = 0; vp.consumed = nullptr; vp.spill = dSpill; vp.spillStride = w * bandRows;
        vp.viewBase = 0; vp.N = 1; vp.A = 1; vp.W = w; vp.H = h; vp.bands = bands; vp.bandRows = bandRows; vp.triCap = triCap;
        vp.p00 = k.p00; vp.p11 = k.p11; vp.p22 = k.p22; vp.p32 = k.p32;
        mvr::viewKernel<false><<<bands, mvr::kThreads, smem>>>(vp);
        ok = cudaDeviceSynchronize() == cudaSuccess;
        if (ok) {
            cudaMemcpy(rgba, dObs, size_t(w) * h * 4, cudaMemcpyDeviceToHost);
            if (depth) cudaMemcpy(depth, dDepth, size_t(w) * h * 4, cudaMemcpyDeviceToHost);
        }
    }
    cudaFree(dCtr); cudaFree(dSpill); cudaFree(dInst); cudaFree(dCnt); cudaFree(dView); cudaFree(dObs); cudaFree(dDepth);
    return ok ? MV_OK : MV_ERR_CUDA;
}

// host-only (no CUDA): run the product's level generator for env stream `env_seed` and dump episode `episode`'s level in
// the mv_debug_get_level layout.  Lets the CPU test-suite compare level generation with the oracle without a GPU.
int mv_debug_generate_level(const char *scenario, int num_agents, int env_seed, int episode, const char *const *keys, const float *vals, int nparams,
                            int32_t *out, int cap) {
    const int sc = scenario ? mv::scenarioFromName(scenario) : -1;
    if (sc < 0 || num_agents < 1 || num_agents > MV_MAX_AGENTS || episode < 0) return MV_ERR_ARG;
    mv::FloatParams params = mv::defaultFloatParams(scenario);
    for (int i = 0; i < nparams; ++i) params[keys[i]] = vals[i];
    mv::LevelGenerator gen(scenario, num_agents, params);
    gen.seed((unsigned long)env_seed);
    mv::LevelOut lo;
    try {
        for (int ep = 0; ep <= episode; ++ep) gen.generate(lo, ep, 1 << 30);
    } catch (const std::exception &ex) { g_createError = ex.what(); return MV_ERR_CAPACITY; }  // mv_last_error(NULL) tells why
    const MvLevel &L = lo.level;
    std::vector<int32_t> o;
    o.push_back(L.n_grid_static); o.push_back(L.n_terrain); o.push_back(L.n_obj);
    for (int a = 0; a < 3; ++a) o.push_back(L.bz_min[a]);
    for (int a = 0; a < 3; ++a) o.push_back(L.bz_max[a]);
    for (int i = 0; i < L.n_grid_static; ++i) {
        const MvBox &b = lo.statics[size_t(i)];
        const float vs = L.scenario == MV_SCENARIO_SOKOBAN ? 2.0f : 1.0f;  // voxel size of the scenario's grid
        for (int a = 0; a < 3; ++a) o.push_back(int(lroundf((b.c[a] - b.h[a]) / vs)));
        for (int a = 0; a < 3; ++a) o.push_back(int(lroundf((b.c[a] + b.h[a]) / vs)) - 1);
        o.push_back(b.flags & 255); o.push_back(int(kPaletteRgb[b.color]));
    }
    for (int i = 0; i < L.n_terrain; ++i) {
        o.push_back(L.terrain[i].type);
        for (int a = 0; a < 6; ++a) o.push_back(L.terrain[i].bb[a]);
    }
    for (int i = 0; i < L.n_obj; ++i) for (int a = 0; a < 3; ++a) o.push_back(L.obj_init[i].voxel[a]);
    for (int i = 0; i < num_agents; ++i) for (int a = 0; a < 3; ++a) o.push_back(int(L.init_pos[i][a]));
    if (L.scenario != MV_SCENARIO_TOWER) {
        o.push_back(L.n_movable);  // numPlatforms
        dumpLevelExtras(L, lo.statics.data(), lo.staticRot.data(), o);
    }
    // spawn yaw basis bits, so the float side of spawnAgents is pinned too
    for (int i = 0; i < num_agents; ++i) for (int k = 0; k < 9; ++k) { int32_t u; std::memcpy(&u, &L.spawn_basis[i][k], 4); o.push_back(u); }
    if (int(o.size()) > cap) return -int(o.size());
    std::memcpy(out, o.data(), o.size() * sizeof(int32_t));
    return int(o.size());
}

int mv_debug_bzset(const int32_t *ops, int nops, int32_t *out_xyz, int cap) {
    MvEnvState s;
    std::memset(&s, 0, sizeof s);
    mvBzInit(s);
    for (int i = 0; i < nops; ++i) {
        const int32_t *o = ops + i * 4;
        if (o[0] == 0) mvBzInsert(s, o[1], o[2], o[3]);
        else if (o[0] == 1) mvBzErase(s, o[1], o[2], o[3]);
        else mvBzClear(s);
    }
    if (s.bz_count * 3 > cap) return -s.bz_count;
    for (int i = 0; i < s.bz_count; ++i) for (int a = 0; a < 3; ++a) out_xyz[i * 3 + a] = s.bz_items[i][a];
    return s.bz_count;
}

}  // extern "C"
