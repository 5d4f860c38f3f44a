// Host engine + C ABI of libgoicp_b200.so (include/goicp_b200.h).
//
// GoICP::Register runs on the device: by default the whole batch in one launch of the device-resident search (k_search.cu),
// otherwise by one of the host wave schedulers of engine_search.cu.  DESIGN.md section 5 says which runs when.
//
// There is no CPU fallback anywhere in this file: every numeric result comes from a kernel.
#include <cuda.h>   // types of the driver range query (no link dependency)
#include "engine_internal.h"

std::string g_create_error;

namespace {
static goicp_status ensure_single(Eng* h) {
    if (h->probs.size() != 1) return fail(h, GOICP_ERR_ARG, "no single registration problem set (call goicp_set_model/goicp_set_data)");
    return GOICP_OK;
}

// Validation of caller buffers in device memory.  cudaPointerGetAttributes says whether a pointer is device or managed
// memory of which device; the driver's range query (reached through the runtime, so the library does not link libcuda)
// gives the whole allocation, so that the buffers of a packed batch cost one query per allocation, not one per pair.
struct DevRanges {
    std::vector<std::pair<uintptr_t, uintptr_t>> ok;   // validated allocations [begin, end)
    // NULL if [ptr, ptr + bytes) lies in one device or managed allocation of `device`, else the reason
    const char* check(int device, const void* ptr, size_t bytes) {
        const uintptr_t b = (uintptr_t)ptr, e = b + bytes;
        for (auto& r : ok) if (b >= r.first && e <= r.second) return nullptr;
        cudaPointerAttributes a;
        if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) { cudaGetLastError(); return "is not memory"; }
        if ((a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != device) return "is not device or managed memory";
        typedef CUresult (*RangeFn)(CUdeviceptr*, size_t*, CUdeviceptr);
        static RangeFn range = nullptr;
        if (!range) {
            void* fn = nullptr; cudaDriverEntryPointQueryResult q;
            if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !fn) return "cannot be checked (no driver range query)";
            range = (RangeFn)fn;
        }
        CUdeviceptr base = 0; size_t size = 0;
        if (a.type == cudaMemoryTypeManaged) { base = (CUdeviceptr)b; size = bytes; }   // managed: no range query; this buffer only
        else if (range(&base, &size, (CUdeviceptr)b) != CUDA_SUCCESS) return "is not in a device allocation";
        if (b < base || e > base + size) return "extends past its allocation";
        ok.emplace_back((uintptr_t)base, (uintptr_t)(base + size));
        return nullptr;
    }
};
}  // namespace

// =====================================================================================================================
extern "C" {

const char* goicp_version(void) { return "goicp-b200 0.1 (sm_100a)"; }
const char* goicp_last_error(goicp_handle h) { return h ? h->err.c_str() : g_create_error.c_str(); }

void goicp_params_default(goicp_params* p) {   // shipped config.txt:4-53
    p->MSEThresh = 0.01f;
    p->rotMinX = p->rotMinY = p->rotMinZ = -3.1416f; p->rotWidth = 6.2832f;
    p->transMinX = p->transMinY = p->transMinZ = -0.5f; p->transWidth = 1.0f;
    p->trimFraction = 0.0f;
    p->regularization = 0.0005f; p->regularizationNeighbors = 0.0f; p->regularizationFPFH = 0.0f;
    p->cfpfh = 0; p->norm = 2; p->ponderation = 1;
    p->distTransSize = 20; p->distTransExpandFactor = 2.0;
}

goicp_status goicp_create(goicp_handle* out, int device, void* stream_or_null) {
    if (!out) return GOICP_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0) return fail(nullptr, GOICP_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    if (device < 0 || device >= ndev) return fail(nullptr, GOICP_ERR_ARG, "device %d out of range (0..%d)", device, ndev - 1);
    if ((e = cudaSetDevice(device)) != cudaSuccess) return fail(nullptr, GOICP_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return fail(nullptr, GOICP_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major < 10) return fail(nullptr, GOICP_ERR_CUDA, "device %s is sm_%d%d; this library is built for sm_100a only", prop.name, prop.major, prop.minor);
    Eng* h = new Eng();
    h->device = device; h->numSM = prop.multiProcessorCount;
    if (stream_or_null) { h->stream = (cudaStream_t)stream_or_null; h->ownStream = false; }
    else { if ((e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) { delete h; return fail(nullptr, GOICP_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); } h->ownStream = true; }
    if ((e = goicp_preload_bnb()) != cudaSuccess || (e = goicp_preload_dt()) != cudaSuccess || (e = goicp_preload_icp()) != cudaSuccess || (e = goicp_preload_misc()) != cudaSuccess || (e = goicp_preload_search()) != cudaSuccess ||
        (e = goicp_preload_prep()) != cudaSuccess) {
        delete h; return fail(nullptr, GOICP_ERR_CUDA, "kernel preload failed: %s (library built for sm_100a only)", cudaGetErrorString(e));
    }
    if (h->devCounters.ensure(sizeof(DevCounters)) != cudaSuccess || cudaMemset(h->devCounters.p, 0, sizeof(DevCounters)) != cudaSuccess) { delete h; return fail(nullptr, GOICP_ERR_CUDA, "device allocation failed"); }
    if (h->main.init(false, h->stream) != GOICP_OK || cudaEventCreateWithFlags(&h->evPairs, cudaEventDisableTiming) != cudaSuccess) {
        goicp_destroy(h); return fail(nullptr, GOICP_ERR_CUDA, "event creation failed");
    }
    goicp_params_default(&h->params); h->haveParams = true;
    *out = h;
    return GOICP_OK;
}

void goicp_destroy(goicp_handle h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    DevBuf* bufs[] = {&h->arenaIn, &h->arenaWork, &h->dPairs, &h->dTmp, &h->dTmp2, &h->dTmp3, &h->dSepBits, &h->dSepNx, &h->dSepNxy, &h->dSepCid, &h->dRaw, &h->dPrep, &h->sCtl, &h->sHdrs, &h->sSlots, &h->sStates, &h->sRq, &h->sIcp, &h->sOuts, &h->dCutoff};
    for (DevBuf* b : bufs) b->release();
    h->hStage.release(); h->hPairs.release(); h->hPrep.release(); h->hOuts.release(); h->hCutoff.release(); h->qHeaps.release(); h->qScratch.release(); h->qMemo.release(); h->devCounters.release();
    h->main.release();
    for (auto& w : h->workers) w->release();
    if (h->evPairs) cudaEventDestroy(h->evPairs);
    if (h->ownStream) cudaStreamDestroy(h->stream);
    delete h;
}

goicp_status goicp_set_model(goicp_handle h, const float* xyz, const int32_t* c, const float* fpfh41, int32_t Nm) {
    if (!h || !xyz || Nm < 1) return h ? fail(h, GOICP_ERR_ARG, "set_model: bad arguments") : GOICP_ERR_ARG;
    if (h->probs.size() != 1) { h->probs.clear(); h->probs.resize(1); }
    Problem& P = h->probs[0];
    set_cloud(P.mxyz, P.mc, P.mf, xyz, c, fpfh41, Nm); P.Nm = Nm;
    P.uploaded = P.prepared = P.dt_built = P.initialized = false;
    return GOICP_OK;
}
goicp_status goicp_set_data(goicp_handle h, const float* xyz, const int32_t* c, const float* fpfh41, int32_t Nd) {
    if (!h || !xyz || Nd < 1) return h ? fail(h, GOICP_ERR_ARG, "set_data: bad arguments") : GOICP_ERR_ARG;
    if (h->probs.size() != 1) { h->probs.clear(); h->probs.resize(1); }
    Problem& P = h->probs[0];
    set_cloud(P.dxyz, P.dc, P.df, xyz, c, fpfh41, Nd); P.NdAll = Nd; P.Nd = Nd;
    P.uploaded = P.prepared = P.dt_built = P.initialized = false;
    return GOICP_OK;
}
goicp_status goicp_set_params(goicp_handle h, const goicp_params* p) {
    if (!h || !p) return GOICP_ERR_ARG;
    const bool gridChanged = !h->haveParams || p->distTransSize != h->params.distTransSize || p->distTransExpandFactor != h->params.distTransExpandFactor ||
                             (p->trimFraction < 0.001) != (h->params.trimFraction < 0.001) ||
                             p->cfpfh != h->params.cfpfh || p->regularizationFPFH != h->params.regularizationFPFH ||
                             (p->regularizationNeighbors > 0) != (h->params.regularizationNeighbors > 0);   // every key K1 or the arena layout depends on
    h->params = *p; h->haveParams = true; h->pairsDirty = true;
    for (auto& P : h->probs) { P.initialized = false; if (gridChanged) P.prepared = P.dt_built = false; }
    return GOICP_OK;
}
goicp_status goicp_set_options(goicp_handle h, int32_t exact_sums, int32_t spec_width, int32_t use_dt_replay) {
    if (!h) return GOICP_ERR_ARG;
    if (exact_sums >= 0) h->exact_sums = exact_sums ? 1 : 0;
    if (spec_width >= 0) h->spec_width = spec_width;
    if (use_dt_replay >= 0) h->use_dt_replay = use_dt_replay ? 1 : 0;
    return GOICP_OK;
}

static goicp_status build_dt_impl(goicp_handle h, goicp_dt_info* out, bool replay) {
    goicp_status s;
    if ((s = ensure_single(h))) return s;
    Problem& P = h->probs[0];
    if (P.Nm < 1 || P.NdAll < 1) return fail(h, GOICP_ERR_ARG, "build_dt: model and data clouds must be set first");
    cudaSetDevice(h->device);
    if ((s = prepare_all(h))) return s;
    if ((s = build_dt_all(h, replay, true))) return s;
    h->dtUploaded = false;
    if (out) *out = P.info;
    return GOICP_OK;
}
goicp_status goicp_build_dt(goicp_handle h, goicp_dt_info* out) {
    if (!h) return GOICP_ERR_ARG;
    return build_dt_impl(h, out, h->use_dt_replay && h->params.distTransSize <= 32);
}
goicp_status goicp_build_dt_replay(goicp_handle h, goicp_dt_info* out) { if (!h) return GOICP_ERR_ARG; return build_dt_impl(h, out, true); }

goicp_status goicp_dt_upload(goicp_handle h, const float* dist, const int32_t* nearest_xyz) {
    if (!h) return GOICP_ERR_ARG;
    goicp_status s; if ((s = ensure_single(h))) return s;
    Problem& P = h->probs[0];
    if (!P.dt_built) return fail(h, GOICP_ERR_ARG, "dt_upload before build_dt");
    cudaSetDevice(h->device);
    const int S = P.info.size; const size_t S3 = (size_t)S * S * S;
    if (dist) { CU(cudaMemcpyAsync(P.dev.g.dist, dist, sizeof(float) * S3, cudaMemcpyHostToDevice, h->stream)); h->dtUploaded = true; }
    if (nearest_xyz) {
        std::vector<int> vn(S3);
        for (size_t i = 0; i < S3; i++) vn[i] = (nearest_xyz[3 * i + 2] * S + nearest_xyz[3 * i + 1]) * S + nearest_xyz[3 * i];
        CU(cudaMemcpyAsync(P.dev.g.vnear, vn.data(), sizeof(int) * S3, cudaMemcpyHostToDevice, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        CU(goicp_launch_dt_vcell(P.dev.g, h->numSM, h->stream));
    }
    CU(cudaStreamSynchronize(h->stream));
    P.initialized = false;
    return GOICP_OK;
}
goicp_status goicp_dt_download(goicp_handle h, float* dist, int32_t* nearest, int32_t* cellc) {
    if (!h) return GOICP_ERR_ARG;
    goicp_status s; if ((s = ensure_single(h))) return s;
    Problem& P = h->probs[0];
    if (!P.dt_built) return fail(h, GOICP_ERR_ARG, "dt_download before build_dt");
    cudaSetDevice(h->device);
    const int S = P.info.size; const size_t S3 = (size_t)S * S * S;
    if (dist) CU(cudaMemcpyAsync(dist, P.dev.g.dist, sizeof(float) * S3, cudaMemcpyDeviceToHost, h->stream));
    std::vector<int> vn, cv, cc;
    if (nearest) { vn.resize(S3); CU(cudaMemcpyAsync(vn.data(), P.dev.g.vnear, sizeof(int) * S3, cudaMemcpyDeviceToHost, h->stream)); }
    const int nc = P.info.ncells;
    if (cellc && nc > 0) {
        cv.resize(nc); cc.resize(nc);
        CU(cudaMemcpyAsync(cv.data(), P.dev.g.cell_vox, sizeof(int) * nc, cudaMemcpyDeviceToHost, h->stream));
        CU(cudaMemcpyAsync(cc.data(), P.cell_col, sizeof(int) * nc, cudaMemcpyDeviceToHost, h->stream));
    }
    CU(cudaStreamSynchronize(h->stream));
    if (nearest) for (size_t i = 0; i < S3; i++) { int v = vn[i]; nearest[3 * i] = v % S; nearest[3 * i + 1] = (v / S) % S; nearest[3 * i + 2] = v / (S * S); }
    if (cellc) {
        for (size_t i = 0; i < S3; i++) cellc[i] = -2;
        for (int c = 0; c < nc; c++) cellc[cv[c]] = cc[c];
    }
    return GOICP_OK;
}
goicp_status goicp_dt_distance(goicp_handle h, const double* xyz, int32_t n, float* dist, int32_t* cell) {
    if (!h || !xyz || !dist || n < 0) return GOICP_ERR_ARG;
    goicp_status s; if ((s = ensure_single(h))) return s;
    if (!h->probs[0].dt_built) return fail(h, GOICP_ERR_ARG, "dt_distance before build_dt");
    if (n == 0) return GOICP_OK;
    cudaSetDevice(h->device);
    CU(h->dTmp.ensure(sizeof(double) * 3 * (size_t)n)); CU(h->dTmp2.ensure(sizeof(float) * (size_t)n)); CU(h->dTmp3.ensure(sizeof(int) * 3 * (size_t)n));
    CU(cudaMemcpyAsync(h->dTmp.p, xyz, sizeof(double) * 3 * (size_t)n, cudaMemcpyHostToDevice, h->stream));
    CU(goicp_launch_dt_distance(h->dPairs.as<PairDev>(), 0, h->dTmp.as<double>(), n, h->dTmp2.as<float>(), h->dTmp3.as<int>(), h->stream));
    CU(cudaMemcpyAsync(dist, h->dTmp2.p, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    if (cell) CU(cudaMemcpyAsync(cell, h->dTmp3.p, sizeof(int) * 3 * (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return GOICP_OK;
}
goicp_status goicp_set_nd(goicp_handle h, int32_t nd) {
    if (!h) return GOICP_ERR_ARG;
    goicp_status s; if ((s = ensure_single(h))) return s;
    Problem& P = h->probs[0];
    if (nd < 1 || nd > P.NdAll) return fail(h, GOICP_ERR_ARG, "set_nd: %d outside [1,%d]", nd, P.NdAll);
    P.Nd = nd; P.initialized = false; h->pairsDirty = true;
    return GOICP_OK;
}
goicp_status goicp_initialize(goicp_handle h) {
    if (!h) return GOICP_ERR_ARG;
    goicp_status s; if ((s = ensure_single(h))) return s;
    cudaSetDevice(h->device);
    if ((s = initialize_all(h))) return s;
    h->main.collect(1);
    return GOICP_OK;
}
goicp_status goicp_get_weights(goicp_handle h, float* w) {
    if (!h || !w) return GOICP_ERR_ARG;
    goicp_status s; if ((s = ensure_single(h))) return s;
    Problem& P = h->probs[0]; if (!P.initialized) return fail(h, GOICP_ERR_ARG, "not initialized");
    CU(cudaMemcpyAsync(w, P.dev.weights, sizeof(float) * P.Nd, cudaMemcpyDeviceToHost, h->stream)); CU(cudaStreamSynchronize(h->stream));
    return GOICP_OK;
}
goicp_status goicp_get_maxrotdis(goicp_handle h, float* out) {
    if (!h || !out) return GOICP_ERR_ARG;
    goicp_status s; if ((s = ensure_single(h))) return s;
    Problem& P = h->probs[0]; if (!P.initialized) return fail(h, GOICP_ERR_ARG, "not initialized");
    CU(cudaMemcpyAsync(out, P.dev.maxRotDis, sizeof(float) * GOICP_MAXROTLEVEL * P.Nd, cudaMemcpyDeviceToHost, h->stream)); CU(cudaStreamSynchronize(h->stream));
    return GOICP_OK;
}
goicp_status goicp_get_thresholds(goicp_handle h, float* sse, int32_t* inlier) {
    if (!h) return GOICP_ERR_ARG;
    goicp_status s; if ((s = ensure_single(h))) return s;
    Problem& P = h->probs[0]; if (!P.initialized) return fail(h, GOICP_ERR_ARG, "not initialized");
    if (sse) *sse = P.dev.SSEThresh; if (inlier) *inlier = P.dev.inlierNum;
    return GOICP_OK;
}

goicp_status goicp_eval_bounds(goicp_handle h, const float* R, const int32_t* level, int32_t nr, const float* tcube, const int32_t* rot_of,
                               int32_t nt, float* ub, float* lb, int32_t* incomp_minmax, int32_t* fpfh_minmax) {
    if (!h || !R || !level || !tcube || !ub || !lb || nr < 1 || nt < 0) return GOICP_ERR_ARG;
    goicp_status s; if ((s = ensure_single(h))) return s;
    Problem& P = h->probs[0]; if (!P.initialized) return fail(h, GOICP_ERR_ARG, "eval_bounds before initialize");
    if (nt == 0) return GOICP_OK;
    cudaSetDevice(h->device);
    std::vector<WaveCube> cubes(nt);
    for (int k = 0; k < nt; k++) { cubes[k].x = tcube[4 * k]; cubes[k].y = tcube[4 * k + 1]; cubes[k].z = tcube[4 * k + 2]; cubes[k].w = tcube[4 * k + 3]; cubes[k].rot = rot_of ? rot_of[k] : 0;
        if (cubes[k].rot < 0 || cubes[k].rot >= nr) return fail(h, GOICP_ERR_ARG, "rot_of[%d]=%d out of range", k, cubes[k].rot); }
    const int nwarps = std::min(nt, h->numSM * 8 * 8);
    const size_t bR = al256(sizeof(float) * 9 * nr), bL = al256(sizeof(int) * nr), bC = al256(sizeof(WaveCube) * nt), bF = al256(sizeof(float) * nt), bI = al256(sizeof(int) * 2 * nt);
    CU(h->dTmp.ensure(bR + bL + bC + 2 * bF + 2 * bI));
    CU(h->dTmp2.ensure(sizeof(float) * (size_t)nwarps * P.Nd));
    char* d = h->dTmp.as<char>();
    float* dR = (float*)d; int* dL = (int*)(d + bR); WaveCube* dC = (WaveCube*)(d + bR + bL); float* dU = (float*)(d + bR + bL + bC); float* dLb = (float*)(d + bR + bL + bC + bF);
    int* dI = (int*)(d + bR + bL + bC + 2 * bF); int* dFm = (int*)(d + bR + bL + bC + 2 * bF + bI);
    CU(cudaMemcpyAsync(dR, R, sizeof(float) * 9 * nr, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(dL, level, sizeof(int) * nr, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(dC, cubes.data(), sizeof(WaveCube) * nt, cudaMemcpyHostToDevice, h->stream));
    { EvTimer tm(h->main, 2);
      CU(goicp_launch_eval_bounds(h->dPairs.as<PairDev>(), 0, dR, dL, dC, nt, dU, dLb, dI, dFm, h->dTmp2.as<float>(), nwarps, h->stream));
      tm.stop(1); }
    CU(cudaMemcpyAsync(ub, dU, sizeof(float) * nt, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(lb, dLb, sizeof(float) * nt, cudaMemcpyDeviceToHost, h->stream));
    if (incomp_minmax) CU(cudaMemcpyAsync(incomp_minmax, dI, sizeof(int) * 2 * nt, cudaMemcpyDeviceToHost, h->stream));
    if (fpfh_minmax) CU(cudaMemcpyAsync(fpfh_minmax, dFm, sizeof(int) * 2 * nt, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    h->main.collect(2);
    return GOICP_OK;
}

goicp_status goicp_eval_inclusion(goicp_handle h, const float* R, int32_t level, const float* tcube, int32_t nt, uint8_t* mask, float* resid) {
    if (!h || !R || !tcube || !mask || nt < 0) return GOICP_ERR_ARG;
    goicp_status s; if ((s = ensure_single(h))) return s;
    Problem& P = h->probs[0]; if (!P.initialized) return fail(h, GOICP_ERR_ARG, "eval_inclusion before initialize");
    if (level >= GOICP_MAXROTLEVEL) return fail(h, GOICP_ERR_ARG, "level %d >= MAXROTLEVEL", level);
    if (nt == 0) return GOICP_OK;
    cudaSetDevice(h->device);
    std::vector<WaveCube> cubes(nt);
    for (int k = 0; k < nt; k++) { cubes[k].x = tcube[4 * k]; cubes[k].y = tcube[4 * k + 1]; cubes[k].z = tcube[4 * k + 2]; cubes[k].w = tcube[4 * k + 3]; cubes[k].rot = 0; }
    const size_t bR = al256(sizeof(float) * 9), bC = al256(sizeof(WaveCube) * nt), bF = al256(sizeof(float) * (size_t)nt * P.Nd), bM = al256((size_t)nt * P.Nd);
    CU(h->dTmp.ensure(bR + bC + bF + bM));
    char* d = h->dTmp.as<char>();
    float* dR = (float*)d; WaveCube* dC = (WaveCube*)(d + bR); float* dF = (float*)(d + bR + bC); uint8_t* dM = (uint8_t*)(d + bR + bC + bF);
    CU(cudaMemcpyAsync(dR, R, sizeof(float) * 9, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(dC, cubes.data(), sizeof(WaveCube) * nt, cudaMemcpyHostToDevice, h->stream));
    CU(goicp_launch_eval_inclusion(h->dPairs.as<PairDev>(), 0, dR, level, dC, nt, dF, dM, std::min(nt, h->numSM * 64), h->stream)); h->main.launches[2]++;
    CU(cudaMemcpyAsync(mask, dM, (size_t)nt * P.Nd, cudaMemcpyDeviceToHost, h->stream));
    if (resid) CU(cudaMemcpyAsync(resid, dF, sizeof(float) * (size_t)nt * P.Nd, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return GOICP_OK;
}

goicp_status goicp_inner_bnb(goicp_handle h, const float* R, const int32_t* level, const float* opt_error, int32_t n, float* err,
                             float* tnode, int64_t* pops_subcubes) {
    if (!h || !R || !level || !opt_error || !err || n < 0) return GOICP_ERR_ARG;
    goicp_status s; if ((s = ensure_single(h))) return s;
    Problem& P = h->probs[0]; if (!P.initialized) return fail(h, GOICP_ERR_ARG, "inner_bnb before initialize");
    cudaSetDevice(h->device);
    std::vector<InnerProb> reqs(n); std::vector<InnerOut> outs;
    for (int k = 0; k < n; k++) {
        if (level[k] >= GOICP_MAXROTLEVEL) return fail(h, GOICP_ERR_ARG, "level %d >= MAXROTLEVEL", level[k]);
        reqs[k].pair = 0; reqs[k].level = level[k]; reqs[k].optError = opt_error[k]; memcpy(reqs[k].R, R + 9 * k, sizeof(float) * 9);
    }
    const BnbCfg cfg = bnb_config(h);
    h->main.ctaCap = 0;
    if ((s = run_inner(h, h->main, cfg, reqs, outs))) return s;
    for (int k = 0; k < n; k++) {
        err[k] = outs[k].err;
        if (tnode) memcpy(tnode + 4 * k, outs[k].node, sizeof(float) * 4);
        if (pops_subcubes) { pops_subcubes[2 * k] = outs[k].pops; pops_subcubes[2 * k + 1] = outs[k].subcubes; }
    }
    return GOICP_OK;
}

goicp_status goicp_icp(goicp_handle h, double* R, double* t, float* err, int32_t* corr) {
    if (!h || !R || !t || !err) return GOICP_ERR_ARG;
    goicp_status s; if ((s = ensure_single(h))) return s;
    Problem& P = h->probs[0]; if (!P.initialized) return fail(h, GOICP_ERR_ARG, "icp before initialize");
    cudaSetDevice(h->device);
    std::vector<IcpState> st{make_icp_state(0, ICP_REFINE, R, t)};
    if ((s = run_icp(h, h->main, st))) return s;
    memcpy(R, st[0].R, sizeof(double) * 9); memcpy(t, st[0].t, sizeof(double) * 3); *err = st[0].error;
    if (corr) {
        std::vector<unsigned long long> nn(P.Nd);
        CU(cudaMemcpyAsync(nn.data(), P.dev.nn, sizeof(unsigned long long) * P.Nd, cudaMemcpyDeviceToHost, h->stream)); CU(cudaStreamSynchronize(h->stream));
        for (int i = 0; i < P.Nd; i++) corr[i] = (int)(nn[i] & 0xFFFFFFFFu);
    }
    return GOICP_OK;
}

goicp_status goicp_register(goicp_handle h, goicp_result* out) {
    if (!h || !out) return GOICP_ERR_ARG;
    goicp_status s; if ((s = ensure_single(h))) return s;
    cudaSetDevice(h->device);
    Problem& P = h->probs[0];
    h->main.reset_timing();
    if (!P.dt_built) { const int nd = P.Nd; if ((s = goicp_build_dt(h, nullptr))) return s; P.Nd = nd; }
    if ((s = register_all(h))) return s;
    h->trace = P.res.trace;
    fill_result(h, P, out);
    return GOICP_OK;
}
goicp_status goicp_outer_bnb(goicp_handle h, goicp_result* out) {
    if (!h || !out) return GOICP_ERR_ARG;
    goicp_status s; if ((s = ensure_single(h))) return s;
    Problem& P = h->probs[0];
    if (!P.initialized) return fail(h, GOICP_ERR_ARG, "outer_bnb before initialize");
    return goicp_register(h, out);   // (Initialize is idempotent: the search starts from the same prepared state)
}
const char* goicp_last_trace(goicp_handle h) { return h ? h->trace.c_str() : ""; }

// ---- batch -----------------------------------------------------------------------------------------------------------
static goicp_status batch_upload_impl(goicp_handle h, const goicp_params* p, int32_t npairs, const goicp_pair_desc* pairs, bool onDevice) {
    if (!h || !p || npairs < 1 || !pairs) return GOICP_ERR_ARG;
    cudaSetDevice(h->device);
    for (int i = 0; i < npairs; i++) {
        const goicp_pair_desc& d = pairs[i];
        if (!d.model_xyz || !d.data_xyz || d.Nm < 1 || d.NdAll < 1) return fail(h, GOICP_ERR_ARG, "pair %d: empty cloud", i);
    }
    if (onDevice) {   // every buffer must lie inside one allocation of device or managed memory of this handle's device
        const bool wantF = p->cfpfh != 0;
        DevRanges ok;
        for (int i = 0; i < npairs; i++) {
            const goicp_pair_desc& d = pairs[i];
            const size_t m = d.Nm, n = d.NdAll, F = sizeof(float) * GOICP_NBINS;
            const struct { const void* ptr; size_t bytes; const char* name; } bufs[6] = {
                {d.model_xyz, 12 * m, "model_xyz"}, {d.model_c, 4 * m, "model_c"}, {wantF ? d.model_fpfh : nullptr, F * m, "model_fpfh"},
                {d.data_xyz, 12 * n, "data_xyz"}, {d.data_c, 4 * n, "data_c"}, {wantF ? d.data_fpfh : nullptr, F * n, "data_fpfh"}};
            for (const auto& b : bufs) {
                if (!b.ptr) continue;
                const char* why = ok.check(h->device, b.ptr, b.bytes);
                if (why) return fail(h, GOICP_ERR_ARG, "pair %d: %s %s of device %d", i, b.name, why, h->device);
            }
        }
    }
    h->params = *p; h->haveParams = true;
    h->probs.clear(); h->probs.resize(npairs);
    for (int i = 0; i < npairs; i++) {
        const goicp_pair_desc& d = pairs[i]; Problem& P = h->probs[i];
        P.Nm = d.Nm; P.NdAll = d.NdAll; P.Nd = (d.Nd > 0 && d.Nd <= d.NdAll) ? d.Nd : d.NdAll;
    }
    goicp_status s;
    if ((s = upload_clouds(h, pairs, onDevice))) return s;
    if ((s = prepare_all(h))) return s;
    CU(cudaStreamSynchronize(h->stream));
    return GOICP_OK;
}
goicp_status goicp_batch_upload(goicp_handle h, const goicp_params* p, int32_t npairs, const goicp_pair_desc* pairs) {
    return batch_upload_impl(h, p, npairs, pairs, false);
}
goicp_status goicp_batch_upload_dev(goicp_handle h, const goicp_params* p, int32_t npairs, const goicp_pair_desc* pairs) {
    return batch_upload_impl(h, p, npairs, pairs, true);
}
goicp_status goicp_get_cells(goicp_handle h, int32_t pair, int32_t* cell_vox, int32_t* cell_start, int32_t* cell_pts, uint32_t* cmask,
                             uint8_t* mprop, uint8_t* dprop, goicp_dt_info* info) {
    if (!h) return GOICP_ERR_ARG;
    if (pair < 0 || pair >= (int)h->probs.size()) return fail(h, GOICP_ERR_ARG, "get_cells: pair %d out of range", pair);
    Problem& P = h->probs[pair];
    if (!P.prepared) return fail(h, GOICP_ERR_ARG, "get_cells before the grid is prepared (batch upload or build_dt)");
    cudaSetDevice(h->device);
    const int nc = P.info.ncells;
    std::vector<int> start(nc + 1);
    CU(cudaMemcpyAsync(start.data(), P.dev.cell_start, sizeof(int) * (nc + 1), cudaMemcpyDeviceToHost, h->stream));
    if (cell_vox && nc) CU(cudaMemcpyAsync(cell_vox, P.dev.g.cell_vox, sizeof(int) * nc, cudaMemcpyDeviceToHost, h->stream));
    if (cmask) CU(cudaMemcpyAsync(cmask, P.dev.g.cmask, sizeof(uint32_t) * (nc + 1), cudaMemcpyDeviceToHost, h->stream));
    if (mprop) CU(cudaMemcpyAsync(mprop, P.dev.mprop, P.Nm, cudaMemcpyDeviceToHost, h->stream));
    if (dprop) CU(cudaMemcpyAsync(dprop, P.dev.dprop, P.NdAll, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (cell_start) memcpy(cell_start, start.data(), sizeof(int) * (nc + 1));
    if (cell_pts && start[nc] > 0) {
        CU(cudaMemcpyAsync(cell_pts, P.dev.cell_pts, sizeof(int) * start[nc], cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
    }
    if (info) *info = P.info;
    return GOICP_OK;
}
goicp_status goicp_batch_run(goicp_handle h, goicp_result* results) {
    if (!h || !results) return GOICP_ERR_ARG;
    if (h->probs.empty() || !h->probs[0].prepared) return fail(h, GOICP_ERR_ARG, "batch_run before a successful batch_upload");
    cudaSetDevice(h->device);
    h->main.reset_timing();
    goicp_status s;
    // DT, Initialize and the search are enqueued back to back; the host waits once, for the search
    if ((s = build_dt_all(h, h->use_dt_replay && h->params.distTransSize <= 32, false))) return s;
    if ((s = register_all(h))) return s;
    for (size_t i = 0; i < h->probs.size(); i++) fill_result(h, h->probs[i], results + i);
    h->trace = h->probs[0].res.trace;
    return GOICP_OK;
}
goicp_status goicp_register_batch(goicp_handle h, const goicp_params* p, int32_t npairs, const goicp_pair_desc* pairs, goicp_result* results) {
    goicp_status s;
    if ((s = goicp_batch_upload(h, p, npairs, pairs))) return s;
    return goicp_batch_run(h, results);
}
goicp_status goicp_set_frontier_sharding(goicp_handle h, int32_t rank, int32_t nranks, goicp_allgather_fn allgather, void* user) {
    if (!h || nranks < 1 || rank < 0 || rank >= nranks || (nranks > 1 && !allgather)) return h ? fail(h, GOICP_ERR_ARG, "set_frontier_sharding: bad arguments") : GOICP_ERR_ARG;
    h->shardRank = rank; h->shardN = nranks; h->allgather = allgather; h->allgatherUser = user;
    return GOICP_OK;
}
goicp_status goicp_test_exchange(goicp_handle h, const void* send, void* recv, int64_t bytes_per_rank) {
    if (!h || !send || !recv || bytes_per_rank < 1 || !h->allgather) return GOICP_ERR_ARG;
    return h->allgather(send, recv, bytes_per_rank, h->allgatherUser) == 0 ? GOICP_OK : fail(h, GOICP_ERR_ARG, "all-gather callback failed");
}
goicp_status goicp_set_search_mode(goicp_handle h, int32_t relaxed_order, int32_t wave_nodes) {
    if (!h) return GOICP_ERR_ARG;
    if (relaxed_order >= 0) h->relaxed = relaxed_order ? 1 : 0;
    if (wave_nodes >= 1) h->wave_nodes = wave_nodes;
    return GOICP_OK;
}
goicp_status goicp_set_error_cutoff(goicp_handle h, const float* cutoff_or_null, int32_t n) {
    if (!h) return GOICP_ERR_ARG;
    if (h->probs.empty()) return fail(h, GOICP_ERR_ARG, "set_error_cutoff before any problem is set (set_model / set_data or a batch upload)");
    if (n != (int32_t)h->probs.size()) return fail(h, GOICP_ERR_ARG, "set_error_cutoff: %d values for %d problems", n, (int)h->probs.size());
    if (cutoff_or_null)
        for (int i = 0; i < n; i++) if (std::isnan(cutoff_or_null[i])) return fail(h, GOICP_ERR_ARG, "set_error_cutoff: the cutoff of problem %d is NaN", i);
    for (int i = 0; i < n; i++) h->probs[i].cutoff = cutoff_or_null ? cutoff_or_null[i] : INFINITY;
    h->pairsDirty = true;
    return GOICP_OK;
}
goicp_status goicp_get_search_ends(goicp_handle h, int32_t* kind, float* lb) {
    if (!h || !kind || !lb) return GOICP_ERR_ARG;
    if (h->probs.empty() || h->probs[0].res.endKind == 0) return fail(h, GOICP_ERR_ARG, "get_search_ends before a register or batch run");
    for (size_t i = 0; i < h->probs.size(); i++) { kind[i] = h->probs[i].res.endKind; lb[i] = h->probs[i].res.endLb; }
    return GOICP_OK;
}
goicp_status goicp_set_batch_options(goicp_handle h, int32_t groups, int32_t slots) {
    if (!h) return GOICP_ERR_ARG;
    if (groups >= 0) h->groups = groups;
    if (slots >= 0) h->slots = slots;
    { const char* e = getenv("GOICP_BATCH_SPEC"); if (e && atoi(e) >= 0) h->batch_spec_width = atoi(e); }
    { const char* e = getenv("GOICP_BNB_THREADS"); if (e) { int t = atoi(e); if (t >= 64 && t <= goicp_bnb_default_threads() && t % 32 == 0) { h->bnb_threads = t; h->bnb_threads_set = true; } } }
    return GOICP_OK;
}
goicp_status goicp_get_stats(goicp_handle h, double* out16) {
    if (!h || !out16) return GOICP_ERR_ARG;
    memcpy(out16, &h->stats, sizeof h->stats);
    return GOICP_OK;
}
goicp_status goicp_test_pairdev_uploads(goicp_handle h, int64_t* count) {
    if (!h || !count) return GOICP_ERR_ARG;
    *count = h->pairUploads;
    return GOICP_OK;
}
goicp_status goicp_get_timings(goicp_handle h, float* ms5, int64_t* launches5) {
    if (!h) return GOICP_ERR_ARG;
    for (int k = 0; k < 5; k++) { if (ms5) ms5[k] = h->main.ms[k]; if (launches5) launches5[k] = h->main.launches[k]; }
    return GOICP_OK;
}

// ---- Transformation ----------------------------------------------------------------------------------------------------
goicp_status goicp_normalize_cloud(goicp_handle h, double* xyz, int32_t n, double* mean3, double* max_norm) {
    if (!h || !xyz || n < 1) return GOICP_ERR_ARG;
    cudaSetDevice(h->device);
    CU(h->dTmp.ensure(sizeof(double) * 3 * (size_t)n)); CU(h->dTmp2.ensure(sizeof(double) * 4));
    CU(cudaMemcpyAsync(h->dTmp.p, xyz, sizeof(double) * 3 * (size_t)n, cudaMemcpyHostToDevice, h->stream));
    CU(goicp_launch_normalize(h->dTmp.as<double>(), n, h->dTmp2.as<double>(), h->stream)); h->main.launches[4]++;
    double out4[4];
    CU(cudaMemcpyAsync(xyz, h->dTmp.p, sizeof(double) * 3 * (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(out4, h->dTmp2.p, sizeof out4, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (mean3) { mean3[0] = out4[0]; mean3[1] = out4[1]; mean3[2] = out4[2]; }
    if (max_norm) *max_norm = out4[3];
    return GOICP_OK;
}
goicp_status goicp_scale_cloud(goicp_handle h, double* xyz, int32_t n, double scale) {
    if (!h || !xyz || n < 1) return GOICP_ERR_ARG;
    cudaSetDevice(h->device);
    CU(h->dTmp.ensure(sizeof(double) * 3 * (size_t)n));
    CU(cudaMemcpyAsync(h->dTmp.p, xyz, sizeof(double) * 3 * (size_t)n, cudaMemcpyHostToDevice, h->stream));
    CU(goicp_launch_scale(h->dTmp.as<double>(), n, scale, h->stream)); h->main.launches[4]++;
    CU(cudaMemcpyAsync(xyz, h->dTmp.p, sizeof(double) * 3 * (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return GOICP_OK;
}
goicp_status goicp_apply_rigid(goicp_handle h, const double* xyz, int32_t n, const double* R, const double* t, double* out) {
    if (!h || !xyz || !R || !t || !out || n < 1) return GOICP_ERR_ARG;
    cudaSetDevice(h->device);
    CU(h->dTmp.ensure(sizeof(double) * 3 * (size_t)n)); CU(h->dTmp2.ensure(sizeof(double) * 3 * (size_t)n)); CU(h->dTmp3.ensure(sizeof(double) * 12));
    double Rt[12]; memcpy(Rt, R, sizeof(double) * 9); memcpy(Rt + 9, t, sizeof(double) * 3);
    CU(cudaMemcpyAsync(h->dTmp.p, xyz, sizeof(double) * 3 * (size_t)n, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->dTmp3.p, Rt, sizeof Rt, cudaMemcpyHostToDevice, h->stream));
    CU(goicp_launch_apply_rigid(h->dTmp.as<double>(), n, h->dTmp3.as<double>(), h->dTmp2.as<double>(), h->stream)); h->main.launches[4]++;
    CU(cudaMemcpyAsync(out, h->dTmp2.p, sizeof(double) * 3 * (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return GOICP_OK;
}
goicp_status goicp_rescale_translation(goicp_handle h, double scale, const double* meanT, const double* meanS, const double* R, const double* t, double* out3) {
    if (!h || !meanT || !meanS || !R || !t || !out3) return GOICP_ERR_ARG;
    cudaSetDevice(h->device);
    double in[19]; in[0] = scale; memcpy(in + 1, meanT, 24); memcpy(in + 4, meanS, 24); memcpy(in + 7, R, 72); memcpy(in + 16, t, 24);
    CU(h->dTmp.ensure(sizeof(double) * 24));
    CU(cudaMemcpyAsync(h->dTmp.p, in, sizeof in, cudaMemcpyHostToDevice, h->stream));
    CU(goicp_launch_rescale(h->dTmp.as<double>(), h->dTmp.as<double>() + 19, h->stream)); h->main.launches[4]++;
    CU(cudaMemcpyAsync(out3, h->dTmp.as<double>() + 19, sizeof(double) * 3, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return GOICP_OK;
}
goicp_status goicp_rmsd(goicp_handle h, const double* a, const double* b, int32_t n, float* rmsd) {
    if (!h || !a || !b || !rmsd || n < 1) return GOICP_ERR_ARG;
    cudaSetDevice(h->device);
    CU(h->dTmp.ensure(sizeof(double) * 3 * (size_t)n)); CU(h->dTmp2.ensure(sizeof(double) * 3 * (size_t)n)); CU(h->dTmp3.ensure(sizeof(double) * (size_t)n + 64));
    CU(cudaMemcpyAsync(h->dTmp.p, a, sizeof(double) * 3 * (size_t)n, cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->dTmp2.p, b, sizeof(double) * 3 * (size_t)n, cudaMemcpyHostToDevice, h->stream));
    float* dOut = reinterpret_cast<float*>(h->dTmp3.as<char>() + sizeof(double) * (size_t)n);
    CU(goicp_launch_rmsd(h->dTmp.as<double>(), h->dTmp2.as<double>(), n, h->dTmp3.as<double>(), dOut, h->stream)); h->main.launches[4]++;
    CU(cudaMemcpyAsync(rmsd, dOut, sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return GOICP_OK;
}

}  // extern "C"
