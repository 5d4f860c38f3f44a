// Internals of the host engine shared by its translation units (engine.cu: the C ABI; engine_setup.cu: per-pair preprocessing,
// device layout, DT build, Initialize; engine_search.cu: the three schedulers of GoICP::Register).
#pragma once
#include <cuda_runtime.h>
#include <cmath>
#include <stdlib.h>
#include <atomic>
#include <chrono>
#include <memory>
#include <mutex>
#include <thread>
#include <map>
#include <unordered_map>
#include <unordered_set>
#include "host_search.h"   // with the C library, <algorithm>, <string> and <vector>, goicp_b200.h and goicp_dev.h
#include "launch.h"
#include "search_dev.h"


using clk = std::chrono::steady_clock;
inline double secs_since(clk::time_point t0) { return std::chrono::duration<double>(clk::now() - t0).count(); }

extern std::string g_create_error;

struct DevBuf {
    void* p = nullptr; size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { e = cudaMalloc(&p, bytes); want = bytes; }
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() { return reinterpret_cast<T*>(p); }
};
struct PinBuf {
    void* p = nullptr; size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = bytes * 2 + 256;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template <class T> T* as() { return reinterpret_cast<T*>(p); }
};

// pinned host memory mapped into the device address space: kernels read requests / write results directly over the bus,
// so a wave is one launch + one wait (no copies, no memset)
struct MapBuf {
    void* h = nullptr; void* d = nullptr; size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (h) cudaFreeHost(h);
        h = d = nullptr; cap = 0;
        size_t want = bytes * 2 + 4096;
        cudaError_t e = cudaHostAlloc(&h, want, cudaHostAllocMapped | cudaHostAllocPortable);
        if (e != cudaSuccess) return e;
        if ((e = cudaHostGetDevicePointer(&d, h, 0)) != cudaSuccess) return e;
        cap = want;
        return cudaSuccess;
    }
    void release() { if (h) cudaFreeHost(h); h = d = nullptr; cap = 0; }
};

struct Problem {
    // ---- inputs ----
    int Nm = 0, NdAll = 0, Nd = 0, ncolours = 1;
    std::vector<float> mxyz, dxyz;       // host copies of a single registration's clouds (goicp_set_model / goicp_set_data), AoS as
    std::vector<int> mc, dc;             // given; a batch keeps none
    std::vector<float> mf, df;           // N x 41 or empty
    // ---- the clouds in the input arena (upload_clouds) ----
    bool uploaded = false;               // the arena holds the current clouds: K1 can run again from it
    bool hasF = false;                   // ... with both clouds' c-FPFH rows
    int *mcol = nullptr, *dcol = nullptr;        // colour codes, 0 where none were given
    float *mfpfh = nullptr, *dfpfh = nullptr;    // descriptor rows or NULL
    int* cell_col = nullptr;             // K1: colour of each cell, -1 if mixed (CELL.c, what goicp_dt_download reports)
    // ---- grid ----
    goicp_dt_info info{};
    bool prepared = false, dt_built = false, initialized = false;
    // ---- device ----
    PairDev dev{};
    size_t inBytes = 0, workBytes = 0, inOff = 0, workOff = 0;
    // ---- outputs ----
    SearchResult res;
    double t_dt = 0, t_reg = 0;
};

// host-side parallel loop (staging of a batch's clouds and descriptors)
template <class F> static void parallel_for(int n, F fn) {
    const int nt = (int)std::min<unsigned>(std::max(1u, std::thread::hardware_concurrency()), (unsigned)std::max(1, n / 16));
    if (nt <= 1) { for (int i = 0; i < n; i++) fn(i); return; }
    std::atomic<int> next(0);
    std::vector<std::thread> th;
    for (int t = 0; t < nt; t++) th.emplace_back([&]() { for (;;) { const int i = next.fetch_add(1); if (i >= n) break; fn(i); } });
    for (auto& t : th) t.join();
}


// Everything one stream of waves needs: a worker thread of a batch owns one, the handle's own stream has `main`.
struct WaveCtx {
    cudaStream_t stream = nullptr; bool ownStream = false;
    DevBuf dCounter, dHeaps, dBnbScratch, dIcp, dMemo;
    MapBuf mProbs, mOuts, mIcp;
    bool counterReady = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, evDone = nullptr;
    float ms[5] = {0, 0, 0, 0, 0}; long long launches[5] = {0, 0, 0, 0, 0};
    long long waves = 0, callsLaunched = 0;
    double tLogic = 0, tInnerEnq = 0, tInnerWait = 0;   // host seconds
    int heapCap = 1 << 14;
    int ctaCap = 0;   // 0: numSM x occupancy
    goicp_status init(bool own, cudaStream_t st) {
        ownStream = own; stream = st;
        if (own && cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking) != cudaSuccess) return GOICP_ERR_CUDA;
        if (cudaEventCreate(&ev0) != cudaSuccess || cudaEventCreate(&ev1) != cudaSuccess ||
            cudaEventCreateWithFlags(&evDone, cudaEventBlockingSync | cudaEventDisableTiming) != cudaSuccess) return GOICP_ERR_CUDA;
        return GOICP_OK;
    }
    // waits without spinning a host core (worker threads outnumber cores)
    cudaError_t sync() {
        cudaError_t e = cudaEventRecord(evDone, stream); if (e != cudaSuccess) return e;
        return cudaEventSynchronize(evDone);
    }
    void reset_timing() {
        memset(ms, 0, sizeof ms); memset(launches, 0, sizeof launches); waves = callsLaunched = 0;
        tLogic = tInnerEnq = tInnerWait = 0;
    }
    void release() {
        DevBuf* bufs[] = {&dCounter, &dHeaps, &dBnbScratch, &dIcp, &dMemo};
        for (DevBuf* b : bufs) b->release();
        mProbs.release(); mOuts.release(); mIcp.release();
        if (ev0) cudaEventDestroy(ev0); if (ev1) cudaEventDestroy(ev1); if (evDone) cudaEventDestroy(evDone);
        ev0 = ev1 = evDone = nullptr;
        if (ownStream && stream) cudaStreamDestroy(stream);
        stream = nullptr;
    }
};

// the 16 doubles of goicp_get_stats, in the order include/goicp_b200.h documents
struct SearchStats {
    double waves = 0, callsExecuted = 0, callsUsed = 0, hostThreads = 0, hostSeconds = 0;
    double tRequests = 0, tEnqueue = 0, tWait = 0;   // wave scheduler: host seconds
    double calls = 0, pops = 0, callCycles = 0, cornerMisses = 0, idleCycles = 0, ctas = 0, rerunPairs = 0, ctaCycles = 0;   // device-resident search
};
static_assert(sizeof(SearchStats) == 16 * sizeof(double), "");

struct goicp_handle_s {
    int device = 0; cudaStream_t stream = nullptr; bool ownStream = false; int numSM = 148;
    goicp_params params; bool haveParams = false;
    int exact_sums = 1, spec_width = 32, use_dt_replay = 1;
    int groups = 0, slots = 0;   // 0 = auto
    int batch_spec_width = 4;    // wave scheduler: speculation width inside a batch (pairs already fill the GPU)
    bool dtUploaded = false;   // the DT came from goicp_dt_upload (test hook): no 16-bit distance codes
    int bnb_threads = goicp_bnb_default_threads(); bool bnb_threads_set = false;   // threads per InnerBnB CTA (64..512): more threads = shorter pops, fewer resident calls   // batch: worker streams (0 = auto) and pairs advanced in lock-step per stream
    std::vector<Problem> probs;
    DevBuf arenaIn, arenaWork, dPairs, dTmp, dTmp2, dTmp3, dSepBits, dSepNx, dSepNxy, dSepCid;
    PinBuf hStage, hPairs;
    DevBuf dRaw, dPrep; PinBuf hPrep;   // K1: staged host clouds; PrepPair array, summaries and scratch; their host side
    std::vector<PrepPair> prep;         // per problem, filled by upload_clouds
    long long packElems = 0;            // > 0: the clouds of the last upload_clouds still wait for the pack kernel
    WaveCtx main;
    DevBuf qHeaps, qScratch, qMemo, devCounters;   // per-CTA slabs of the device-resident search: translation queues, staging arrays (large Nd), corner memo; DevCounters
    DevBuf sCtl, sHdrs, sSlots, sStates, sRq, sIcp, sOuts; PinBuf hOuts;   // device-resident search (k_search.cu)
    int spec_groups = SR_NGROUP - 4;   // device-resident search: most rotation-queue nodes with speculative calls per owner CTA (0: never speculate)
    int shardRank = 0, shardN = 1; goicp_allgather_fn allgather = nullptr; void* allgatherUser = nullptr;   // frontier sharding
    std::vector<InnerOut> xSend, xRecv;
    int relaxed = 0, wave_nodes = 64;   // single registrations: 1 = relaxed-order wave search (goicp_set_search_mode), wave_nodes rotation nodes per wave
    int resident = 1;            // 1: device-resident search (k_search.cu) whenever the clouds allow it; 0: wave scheduler (one launch per wave, host-side OuterBnB)
    std::vector<std::unique_ptr<WaveCtx>> workers;
    std::mutex errMutex;
    std::string err, trace;
    SearchStats stats;
};


typedef goicp_handle_s Eng;

inline goicp_status fail(Eng* h, goicp_status s, const char* fmt, ...) {
    char buf[512]; va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    if (h) { std::lock_guard<std::mutex> lk(h->errMutex); h->err = buf; } else g_create_error = buf;
    return s;
}
#define CU(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return fail(h, GOICP_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); } while (0)

inline size_t al256(size_t b) { return (b + 255) & ~(size_t)255; }

struct EvTimer {   // CUDA-event time of a kernel group on a wave context's stream
    WaveCtx& c; int slot;
    EvTimer(WaveCtx& c_, int slot_) : c(c_), slot(slot_) { cudaEventRecord(c.ev0, c.stream); }
    void stop(int nlaunch) { cudaEventRecord(c.ev1, c.stream); cudaEventSynchronize(c.ev1); float ms = 0; cudaEventElapsedTime(&ms, c.ev0, c.ev1); c.ms[slot] += ms; c.launches[slot] += nlaunch; }
};

// keys of the trimmed-ICP bitonic sort (icp_device.cuh): next power of two >= n, at least 32
inline size_t sort_cap(int n) { size_t c = 32; while (c < (size_t)n) c <<= 1; return c; }
struct BnbCfg { int NdP, NdQ; size_t smemFloats, smemBytes; int useSmem, perSM, threads, gridOff, S3p, ct; };

// engine_setup.cu
goicp_status upload_clouds(Eng* h, const goicp_pair_desc* src, bool onDevice);
goicp_status upload_pairdevs(Eng* h);
goicp_status build_dt_all(Eng* h, bool replay);
goicp_status initialize_all(Eng* h);
BnbCfg bnb_config(Eng* h);
goicp_status prepare_all(Eng* h);
void set_cloud(std::vector<float>& xyz, std::vector<int>& c, std::vector<float>& f, const float* pxyz, const int32_t* pc, const float* pf, int n);
// engine_search.cu
goicp_status run_inner(Eng* h, WaveCtx& c, const BnbCfg& cfg, std::vector<InnerProb>& reqs, std::vector<InnerOut>& outs);
goicp_status run_icp(Eng* h, WaveCtx& c, std::vector<IcpState>& states);
IcpState make_icp_state(int pair, IcpMode mode, const double* R, const double* t);
goicp_status register_all(Eng* h);
void fill_result(Eng* h, const Problem& P, goicp_result* out);
