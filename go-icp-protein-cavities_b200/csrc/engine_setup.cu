// Host engine, part 1: the device layout of a batch, the per-pair preprocessing K1 (bounding cube, seeding, cell lists,
// colour masks; kernels in k_prep.cu), the DT build and GoICP::Initialize launches.
#include "engine_internal.h"

// ---- the clouds in the input arena ------------------------------------------------------------------------------------
// Lays out every pair's block of the input arena and queues the packing of `src` (one descriptor per problem) into it.
// Host clouds are staged in pinned memory and copied in one cudaMemcpyAsync; device clouds are read in place by the pack
// kernel, which prepare_all launches ahead of K1.  The block keeps the clouds (SoA), their colour codes and, when the
// configuration uses them, their c-FPFH rows, so that K1 can run again from it when the grid keys change.
goicp_status upload_clouds(Eng* h, const goicp_pair_desc* src, bool onDevice) {
    const bool wantF = h->params.cfpfh != 0;   // descriptors are only copied when the configuration uses them
    const int n = (int)h->probs.size();
    size_t inTot = 0, rawTot = 0;
    long long maxElems = 1;
    std::vector<size_t> rawOff(n);
    for (int i = 0; i < n; i++) {
        Problem& P = h->probs[i]; const goicp_pair_desc& d = src[i];
        P.hasF = wantF && d.model_fpfh && d.data_fpfh;
        const size_t Nm = P.Nm, Nd = P.NdAll;
        size_t in = 3 * al256(sizeof(float) * Nd) + 3 * al256(sizeof(float) * Nm) + 2 * al256(Nd) + al256(Nm);
        if (P.hasF) in += al256(sizeof(float) * GOICP_NBINS * Nd) + al256(sizeof(float) * GOICP_NBINS * Nm);
        in += al256(sizeof(int) * Nm) + 2 * al256(sizeof(int) * (Nm + 1)) + al256(sizeof(int) * Nm);   // cells: ncells <= Nm
        in += al256(sizeof(int) * Nd) + 2 * al256(sizeof(int) * Nm);                                    // colour codes, cell colours
        P.inBytes = in; P.inOff = inTot; inTot += in;
        maxElems = std::max(maxElems, (long long)std::max(Nm, Nd) * (P.hasF ? GOICP_NBINS : 1));
        rawOff[i] = rawTot;
        if (!onDevice) rawTot += al256(12 * Nm) + al256(12 * Nd) + (d.model_c ? al256(4 * Nm) : 0) + (d.data_c ? al256(4 * Nd) : 0) +
                                 (P.hasF ? al256(4 * GOICP_NBINS * Nm) + al256(4 * GOICP_NBINS * Nd) : 0);
    }
    CU(h->arenaIn.ensure(inTot));
    if (!onDevice) { CU(h->dRaw.ensure(rawTot)); CU(h->hStage.ensure(rawTot)); }
    h->prep.assign(n, PrepPair{});
    char* dIn = h->arenaIn.as<char>();
    parallel_for(n, [&](int i) {
        Problem& P = h->probs[i]; const goicp_pair_desc& d = src[i];
        PairDev& D = P.dev; PrepPair& Q = h->prep[i];
        memset(&D, 0, sizeof D);
        size_t o = P.inOff;
        auto take = [&](size_t bytes) { char* p = dIn + o; o += al256(bytes); return p; };
        D.dx = (float*)take(sizeof(float) * P.NdAll); D.dy = (float*)take(sizeof(float) * P.NdAll); D.dz = (float*)take(sizeof(float) * P.NdAll);
        D.mx = (float*)take(sizeof(float) * P.Nm); D.my = (float*)take(sizeof(float) * P.Nm); D.mz = (float*)take(sizeof(float) * P.Nm);
        D.dprop = (uint8_t*)take(P.NdAll); D.dknown = (uint8_t*)take(P.NdAll); D.mprop = (uint8_t*)take(P.Nm);
        P.dfpfh = P.hasF ? (float*)take(sizeof(float) * GOICP_NBINS * P.NdAll) : nullptr;
        P.mfpfh = P.hasF ? (float*)take(sizeof(float) * GOICP_NBINS * P.Nm) : nullptr;
        D.g.cell_vox = (int*)take(sizeof(int) * P.Nm);
        D.g.cmask = (uint32_t*)take(sizeof(uint32_t) * (P.Nm + 1));
        D.cell_start = (int*)take(sizeof(int) * (P.Nm + 1));
        D.cell_pts = (int*)take(sizeof(int) * P.Nm);
        P.dcol = (int*)take(sizeof(int) * P.NdAll); P.mcol = (int*)take(sizeof(int) * P.Nm);
        P.cell_col = (int*)take(sizeof(int) * P.Nm);
        D.Nm = P.Nm; D.Nd = P.Nd; D.NdAll = P.NdAll;
        Q.Nm = P.Nm; Q.NdAll = P.NdAll;
        Q.mx = D.mx; Q.my = D.my; Q.mz = D.mz; Q.dx = D.dx; Q.dy = D.dy; Q.dz = D.dz;
        Q.mcol = P.mcol; Q.dcol = P.dcol; Q.mfpfh = P.mfpfh; Q.dfpfh = P.dfpfh;
        Q.mprop = D.mprop; Q.dprop = D.dprop; Q.dknown = D.dknown;
        Q.cell_vox = D.g.cell_vox; Q.cell_start = D.cell_start; Q.cell_pts = D.cell_pts; Q.cell_col = P.cell_col; Q.cmask = D.g.cmask;
        Q.rmxyz = d.model_xyz; Q.rdxyz = d.data_xyz; Q.rmc = d.model_c; Q.rdc = d.data_c;
        Q.rmf = P.hasF ? d.model_fpfh : nullptr; Q.rdf = P.hasF ? d.data_fpfh : nullptr;
        if (onDevice) return;
        size_t r = rawOff[i];
        auto stage = [&](const void* from, size_t bytes) { memcpy(h->hStage.as<char>() + r, from, bytes); const void* to = h->dRaw.as<char>() + r; r += al256(bytes); return to; };
        Q.rmxyz = (const float*)stage(d.model_xyz, 12 * (size_t)P.Nm);
        Q.rdxyz = (const float*)stage(d.data_xyz, 12 * (size_t)P.NdAll);
        if (d.model_c) Q.rmc = (const int*)stage(d.model_c, 4 * (size_t)P.Nm);
        if (d.data_c) Q.rdc = (const int*)stage(d.data_c, 4 * (size_t)P.NdAll);
        if (P.hasF) { Q.rmf = (const float*)stage(d.model_fpfh, 4 * GOICP_NBINS * (size_t)P.Nm); Q.rdf = (const float*)stage(d.data_fpfh, 4 * GOICP_NBINS * (size_t)P.NdAll); }
    });
    if (!onDevice) CU(cudaMemcpyAsync(h->dRaw.p, h->hStage.p, rawTot, cudaMemcpyHostToDevice, h->stream));
    h->packElems = maxElems;
    h->pairsDirty = true;
    for (auto& P : h->probs) { P.uploaded = true; P.prepared = P.dt_built = P.initialized = false; }
    return GOICP_OK;
}

// ---- work arena layout: every pair's grid and search workspaces, with `nc` cells per pair ---------------------------------
static goicp_status layout_work(Eng* h, bool ncellsBound) {
    const goicp_params& p = h->params;
    const int S = p.distTransSize; const size_t S3 = (size_t)S * S * S;
    const bool useF = p.cfpfh != 0;
    size_t workTot = 0;
    for (auto& P : h->probs) {
        const int nc = ncellsBound ? P.Nm : P.info.ncells;
        size_t w = 0;
        w += al256(sizeof(float) * S3) + al256(sizeof(int) * S3) + 2 * al256(sizeof(int) * S3) + al256(S3 + 16) + al256(sizeof(double) * GOICP_OVN)
             + (S <= 32 ? al256(2 * (S3 + 16)) + al256(sizeof(float) * (3 * (size_t)(S - 1) * (S - 1) + 6)) : 0);
        w += 2 * al256(sizeof(float) * P.NdAll) + al256(sizeof(float) * GOICP_MAXROTLEVEL * (size_t)P.NdAll);
        if (useF && p.regularizationFPFH > 0) w += al256(sizeof(float) * P.NdAll * (nc + 1));
        if (p.regularizationNeighbors > 0) w += al256(sizeof(int) * P.NdAll) + al256(sizeof(int) * P.Nm);
        w += al256(sizeof(unsigned long long) * P.NdAll) + al256(sizeof(int) * P.NdAll) + al256(sizeof(float) * 8 * (size_t)std::max(P.NdAll, 1));
        if (!(p.trimFraction < 0.001)) w += al256(sizeof(unsigned long long) * sort_cap(P.NdAll));
        P.workBytes = w; P.workOff = workTot; workTot += w;
    }
    CU(h->arenaWork.ensure(workTot));
    char* dWork = h->arenaWork.as<char>();
    for (auto& P : h->probs) {
        const int nc = ncellsBound ? P.Nm : P.info.ncells;
        PairDev& D = P.dev;
        size_t w = P.workOff;
        auto take = [&](size_t bytes) { char* q = dWork + w; w += al256(bytes); return q; };
        D.g.dist = (float*)take(sizeof(float) * S3);
        D.g.vnear = (int*)take(sizeof(int) * S3);
        D.g.vcell = (int*)take(sizeof(int) * S3); D.g.vmask = (uint32_t*)take(sizeof(int) * S3); D.g.vmask8 = (uint8_t*)take(S3 + 16);
        D.g.ovl = (double*)take(sizeof(double) * GOICP_OVN);
        D.g.dcode = nullptr; D.g.dlut = nullptr; D.g.nlut = 0;
        if (S <= 32) {
            D.g.dcode = (uint16_t*)take(2 * (S3 + 16));
            D.g.dlut = (float*)take(sizeof(float) * (3 * (size_t)(S - 1) * (S - 1) + 6));
            D.g.nlut = 3 * (S - 1) * (S - 1) + 2;
        }
        D.normData = (float*)take(sizeof(float) * P.NdAll);
        D.weights = (float*)take(sizeof(float) * P.NdAll);
        D.maxRotDis = (float*)take(sizeof(float) * GOICP_MAXROTLEVEL * (size_t)P.NdAll);
        D.fpfhD = (useF && p.regularizationFPFH > 0) ? (float*)take(sizeof(float) * P.NdAll * (nc + 1)) : nullptr;
        D.nbD = D.nbM = nullptr;
        if (p.regularizationNeighbors > 0) { D.nbD = (int*)take(sizeof(int) * P.NdAll); D.nbM = (int*)take(sizeof(int) * P.Nm); }
        D.nn = (unsigned long long*)take(sizeof(unsigned long long) * P.NdAll);
        D.order = (int*)take(sizeof(int) * P.NdAll);
        D.scratch = (float*)take(sizeof(float) * 8 * (size_t)std::max(P.NdAll, 1));
        D.sortKeys = !(p.trimFraction < 0.001) ? (unsigned long long*)take(sizeof(unsigned long long) * sort_cap(P.NdAll)) : nullptr;
        D.dfpfh = useF ? P.dfpfh : nullptr; D.mfpfh = useF ? P.mfpfh : nullptr;
        D.g.S = S; D.g.ncells = nc; D.g.xMin = P.info.xMin; D.g.yMin = P.info.yMin; D.g.zMin = P.info.zMin; D.g.scale = P.info.scale;
        D.Nm = P.Nm; D.Nd = P.Nd; D.NdAll = P.NdAll;
    }
    h->pairsDirty = true;
    return GOICP_OK;
}

// fills the parameter-derived fields of every PairDev (GoICP::Initialize :180-267 scalars) and uploads the array, with the
// cutoffs; nothing to do unless something they derive from changed since the last upload (Eng::pairsDirty).  The copies are
// stream-ordered before every kernel that reads them; the host only waits for the previous copy before it rewrites the pinned
// staging buffers.
goicp_status upload_pairdevs(Eng* h) {
    if (!h->pairsDirty) return GOICP_OK;
    const goicp_params& p = h->params;
    const bool doTrim = !(p.trimFraction < 0.001);   // GoICP() :54 sets true; readConfig clears it (jly_main.cpp:259)
    for (auto& P : h->probs) {
        PairDev& D = P.dev;
        D.Nd = P.Nd;
        D.doTrim = doTrim ? 1 : 0;
        D.inlierNum = doTrim ? (int)(P.Nd * (1 - p.trimFraction)) : P.Nd;           // :244-252
        D.norm = p.norm; D.cfpfh = p.cfpfh; D.ponderation = p.ponderation;
        D.fpfh_b = 0; D.fpfh_e = 0;
        if (p.cfpfh == 1) D.fpfh_e = 41; else if (p.cfpfh == 2) D.fpfh_e = 33; else if (p.cfpfh == 3) { D.fpfh_b = 33; D.fpfh_e = 41; }
        D.use_reg = p.regularization > 0 ? 1 : 0;
        D.use_fpfh = (p.regularizationFPFH > 0 && p.cfpfh != 0) ? 1 : 0;
        D.use_nb = p.regularizationNeighbors > 0 ? 1 : 0;
        D.reg = p.regularization; D.regF = p.regularizationFPFH; D.regN = p.regularizationNeighbors;
        D.MSEThresh = p.MSEThresh; D.trimFraction = p.trimFraction;
        D.SSEThresh = p.MSEThresh * D.inlierNum;                                     // :266
        D.tMinX = p.transMinX; D.tMinY = p.transMinY; D.tMinZ = p.transMinZ; D.tWidth = p.transWidth;
        {   // FP32 fast path of the voxel index (goicp_dev.h: GridDev.vf*): fraction bits kept and the ambiguity zone around
            // each rounding boundary, from a bound on the float evaluation error of (v - min) * scale + 0.5 inside the grid
            GridDev& g = D.g;
            const int S = g.S;
            int lg = 0; while ((1 << lg) < S + GOICP_OVLIM + 2) lg++;
            const int f = std::min(16, 22 - lg);
            const double ulp = std::ldexp(1.0, -f);
            const double ext = (double)(S + GOICP_OVLIM + 1) / g.scale, lo = (double)(GOICP_OVLIM + 1) / g.scale;
            const double A = std::max({std::fabs(g.xMin - lo), std::fabs(g.xMin + ext), std::fabs(g.yMin - lo), std::fabs(g.yMin + ext), std::fabs(g.zMin - lo), std::fabs(g.zMin + ext)});
            const double T = std::max({std::fabs((double)p.transMinX), std::fabs((double)p.transMinX + p.transWidth), std::fabs((double)p.transMinY), std::fabs((double)p.transMinY + p.transWidth),
                                       std::fabs((double)p.transMinZ), std::fabs((double)p.transMinZ + p.transWidth)});
            // |v| <= A for a voxel at most GOICP_OVLIM outside the grid, |p| = |v - trans| <= A + T; terms: float rounding of v = p + trans, of the scale, of C and of the fma
            const double err = g.scale * std::ldexp(1.0, -24) * (2 * A + T) * 1.25 + ulp + 1e-9;
            const int E = (int)std::ceil(err / ulp) + 1;
            g.vfScale = (float)g.scale; g.vfShift = f; g.vfMask = (1u << f) - 1u;
            const float magic = (float)std::ldexp(1.5, 23 - f);
            unsigned mb; memcpy(&mb, &magic, 4);
            g.vfBias = mb >> f;
            g.vfMagic = (double)magic + 0.5 + E * ulp;
            g.vfZone = (f >= 8 && (2 * E + 1) * 64 < (1 << f) && std::isfinite(err)) ? (unsigned)(2 * E + 1) : 0xFFFFFFFFu;
            if (getenv("GOICP_NO_VOXFAST")) g.vfZone = 0xFFFFFFFFu;
        }
        for (int l = 0; l < GOICP_MAXROTLEVEL; l++) {                                // :195-204, host libm as the reference
            float sigma = (float)(p.rotWidth / pow(2.0, l) / 2.0);
            float maxAngle = (float)(GOICP_SQRT3 * sigma);
            if (maxAngle > GOICP_PI) maxAngle = (float)GOICP_PI;
            D.s2[l] = 2 * sinf(maxAngle / 2);
        }
    }
    const size_t n = h->probs.size();
    CU(cudaEventSynchronize(h->evPairs));   // (returns at once when the previous copy is done, or there was none)
    CU(h->dPairs.ensure(sizeof(PairDev) * n));
    CU(h->hPairs.ensure(sizeof(PairDev) * n));
    PairDev* st = h->hPairs.as<PairDev>();
    for (size_t i = 0; i < n; i++) st[i] = h->probs[i].dev;
    CU(cudaMemcpyAsync(h->dPairs.p, st, sizeof(PairDev) * n, cudaMemcpyHostToDevice, h->stream));
    h->cutoffOn = std::any_of(h->probs.begin(), h->probs.end(), [](const Problem& P) { return P.cutoff != INFINITY; });
    if (h->cutoffOn) {   // (the search kernel reads no cutoffs when every pair has none)
        CU(h->dCutoff.ensure(sizeof(float) * n));
        CU(h->hCutoff.ensure(sizeof(float) * n));
        for (size_t i = 0; i < n; i++) h->hCutoff.as<float>()[i] = h->probs[i].cutoff;
        CU(cudaMemcpyAsync(h->dCutoff.p, h->hCutoff.p, sizeof(float) * n, cudaMemcpyHostToDevice, h->stream));
    }
    CU(cudaEventRecord(h->evPairs, h->stream));
    h->pairsDirty = false; h->pairUploads++;
    return GOICP_OK;
}

goicp_status build_dt_all(Eng* h, bool replay, bool wait) {
    const int S = h->params.distTransSize;
    auto t0 = clk::now();
    goicp_status s = upload_pairdevs(h);
    if (s) return s;
    EvTimer tm(h->main, 0);
    int nl = 0;
    if (replay) {
        if (S > 32) return fail(h, GOICP_ERR_UNSUPPORTED, "the 8SED replay builder supports distTransSize <= 32 (got %d)", S);
        CU(goicp_launch_dt_replay(h->dPairs.as<PairDev>(), 0, (int)h->probs.size(), S, h->stream)); nl = 1;
    } else {
        const int SW = (S + 31) / 32; const size_t S3 = (size_t)S * S * S;
        CU(h->dSepBits.ensure((size_t)S * S * SW * sizeof(unsigned)));
        CU(h->dSepNx.ensure(S3 * sizeof(unsigned short)));
        CU(h->dSepNxy.ensure(S3 * sizeof(unsigned)));
        CU(h->dSepCid.ensure(S3 * sizeof(int)));
        for (auto& P : h->probs) { CU(goicp_launch_dt_separable(P.dev.g, h->dSepBits.as<unsigned>(), h->dSepNx.as<unsigned short>(), h->dSepNxy.as<unsigned>(), h->dSepCid.as<int>(), h->numSM, h->stream)); nl += 4; }
    }
    tm.stop(nl);
    CU(cudaGetLastError());
    if (wait) h->main.collect(0);
    const double dt = secs_since(t0) / std::max<size_t>(1, h->probs.size());
    for (auto& P : h->probs) { P.dt_built = true; P.t_dt = dt; }
    return GOICP_OK;
}

goicp_status initialize_all(Eng* h) {
    const goicp_params& p = h->params;
    for (auto& P : h->probs) {
        if (!P.dt_built) return fail(h, GOICP_ERR_ARG, "initialize before build_dt");
        if (p.ponderation == 1 && P.Nd < 20) return fail(h, GOICP_ERR_UNSUPPORTED, "ponderation=1 needs Nd >= 20 (neighborsWeights never terminates below; Nd=%d)", P.Nd);
        if (p.norm != 1 && p.norm != 2) return fail(h, GOICP_ERR_UNSUPPORTED, "norm must be 1 or 2");
    }
    goicp_status s = upload_pairdevs(h);
    if (s) return s;
    EvTimer tm(h->main, 1);
    int nl = 1;
    CU(goicp_launch_initialize(h->dPairs.as<PairDev>(), 0, (int)h->probs.size(), h->stream));
    if (p.regularizationFPFH > 0 && p.cfpfh != 0) { CU(goicp_launch_fpfh_table(h->dPairs.as<PairDev>(), 0, (int)h->probs.size(), 32, h->stream)); nl++; }
    if (p.regularizationNeighbors > 0) {   // assignNeighbors (BuildDT :94); both clouds, every source point
        int maxN = 1; for (auto& P : h->probs) maxN = std::max(maxN, P.NdAll + P.Nm);
        CU(goicp_launch_assign_neighbors(h->dPairs.as<PairDev>(), 0, (int)h->probs.size(), std::min(64, (maxN + 255) / 256), h->stream)); nl++;
    }
    tm.stop(nl);
    CU(cudaGetLastError());
    for (auto& P : h->probs) P.initialized = true;
    return GOICP_OK;
}

BnbCfg bnb_config(Eng* h) {
    int maxNd = 1, maxCol = 1; bool anyTrim = false, anyF = false, anyNb = false;
    for (auto& P : h->probs) { maxNd = std::max(maxNd, P.Nd); anyTrim |= P.dev.doTrim != 0; anyF |= P.dev.use_fpfh != 0; anyNb |= P.dev.use_nb != 0; maxCol = std::max(maxCol, P.ncolours); }
    BnbCfg c;
    c.ct = (anyF || anyNb) ? 1 : 0;
    c.NdP = (maxNd + 31) & ~31; c.NdQ = c.NdP + 4;   // row stride = 4 mod 32: the chain lanes' float4 reads of the 8 rows hit 8 different bank quads
    const bool needMd = h->exact_sums || anyTrim, needFp = h->exact_sums && anyF;
    c.smemFloats = goicp_bnb_smem_floats(c.NdP, c.NdQ, h->exact_sums != 0, needMd, needFp);
    c.smemBytes = c.smemFloats * sizeof(float);
    c.useSmem = c.smemBytes <= 180 * 1024;   // + ~32 KB static in the resident kernel
    c.gridOff = 0; c.S3p = 0;
    // small volumes (cavity grids, 20^3): distances + one colour-mask byte per voxel are staged in shared memory per call
    const int S = h->params.distTransSize; const size_t S3 = (size_t)S * S * S;
    const size_t S3p = (S3 + 15) & ~(size_t)15;
    const size_t nlutP = ((size_t)3 * (S - 1) * (S - 1) + 2 + 3) & ~(size_t)3;
    if (c.useSmem && S <= 32 && maxCol <= 8 && !h->dtUploaded && !getenv("GOICP_NO_GRID_SMEM") && ((c.smemFloats + 3) & ~(size_t)3) * 4 + nlutP * 4 + S3p * 3 <= 100 * 1024) {
        c.gridOff = (int)((c.smemFloats + 3) & ~(size_t)3); c.S3p = (int)S3p;
        c.smemBytes = (size_t)c.gridOff * 4 + nlutP * 4 + S3p * 3;   // distance table + 16-bit distance codes + colour-mask bytes
        c.useSmem = 2;
    }
    // batches on shared-memory volumes: 192-thread CTAs, four per SM (measured +5 % over 256 x 3; a single registration keeps
    // the shorter pops of 256-thread CTAs)
    c.threads = (h->bnb_threads_set || !(c.useSmem == 2 && h->probs.size() > 1)) ? h->bnb_threads : std::min(192, h->bnb_threads);
    c.perSM = goicp_inner_bnb_occupancy(c.smemBytes, h->exact_sums, c.threads, c.useSmem, c.ct);
    return c;
}
// K1 for every problem on the device (k_prep.cu), from the clouds in the input arena; one readback of the per-pair
// summaries, then the work arena is laid out with the real cell counts.
goicp_status prepare_all(Eng* h) {
    if (!h->haveParams) return fail(h, GOICP_ERR_ARG, "goicp_set_params not called");
    const goicp_params& p = h->params;
    const int S = p.distTransSize, n = (int)h->probs.size();
    if (S < 2 || S > 1024) return fail(h, GOICP_ERR_UNSUPPORTED, "distTransSize %d outside [2,1024]", S);
    const bool useF = p.cfpfh != 0;
    bool fromHost = false;   // single registrations keep host copies; a new cloud or newly needed descriptors re-upload them
    for (auto& P : h->probs) {
        if (P.Nm < 1 || P.NdAll < 1) return fail(h, GOICP_ERR_ARG, "empty cloud (Nm=%d Nd=%d)", P.Nm, P.NdAll);
        fromHost |= !P.uploaded || (useF && !P.hasF && !P.mxyz.empty());
    }
    goicp_status s;
    if (fromHost) {
        std::vector<goicp_pair_desc> src(n);
        for (int i = 0; i < n; i++) {
            Problem& P = h->probs[i];
            if (P.mxyz.empty() || P.dxyz.empty()) return fail(h, GOICP_ERR_ARG, "pair %d: clouds not uploaded", i);
            src[i] = goicp_pair_desc{P.mxyz.data(), P.mc.data(), P.mf.empty() ? nullptr : P.mf.data(), P.Nm,
                                     P.dxyz.data(), P.dc.data(), P.df.empty() ? nullptr : P.df.data(), P.NdAll, P.Nd};
        }
        if ((s = upload_clouds(h, src.data(), false))) return s;
    }
    for (auto& P : h->probs) if (useF && !P.hasF) return fail(h, GOICP_ERR_ARG, "cfpfh=%d needs c-FPFH descriptors for both clouds", p.cfpfh);
    // K1 uses the pair's vnear / vcell grids as scratch: lay out the work arena with room for one cell per model point
    if ((s = layout_work(h, true))) return s;
    const int nb = goicp_prep_nblocks(S);
    int maxNm = 1; size_t sumNm = 0;
    for (auto& P : h->probs) { maxNm = std::max(maxNm, P.Nm); sumNm += P.Nm; }
    const size_t bPairs = al256(sizeof(PrepPair) * n), bSums = al256(sizeof(PrepSummary) * n), bBlk = al256(sizeof(long long) * nb * (size_t)n);
    CU(h->dPrep.ensure(bPairs + bSums + bBlk + sizeof(int) * sumNm));
    CU(h->hPrep.ensure(bPairs + bSums));
    PrepPair* hq = h->hPrep.as<PrepPair>();
    PrepSummary* hs = reinterpret_cast<PrepSummary*>(h->hPrep.as<char>() + bPairs);
    char* dp = h->dPrep.as<char>();
    int* tmp = reinterpret_cast<int*>(dp + bPairs + bSums + bBlk);
    for (int i = 0; i < n; i++) {
        Problem& P = h->probs[i];
        PrepPair& Q = h->prep[i];
        Q.vcount = P.dev.g.vnear; Q.vcid = P.dev.g.vcell; Q.tmp = tmp; tmp += P.Nm;
        hq[i] = Q;
    }
    const PrepPair* dq = reinterpret_cast<const PrepPair*>(dp);
    PrepSummary* ds = reinterpret_cast<PrepSummary*>(dp + bPairs);
    CU(cudaMemcpyAsync(dp, hq, sizeof(PrepPair) * n, cudaMemcpyHostToDevice, h->stream));
    if (h->packElems) { CU(goicp_launch_prep_pack(dq, n, h->packElems, h->stream)); h->packElems = 0; }
    CU(goicp_launch_prep(dq, ds, reinterpret_cast<long long*>(dp + bPairs + bSums), n, maxNm, S, p.distTransExpandFactor, h->stream));
    CU(cudaMemcpyAsync(hs, ds, sizeof(PrepSummary) * n, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < n; i++) {
        Problem& P = h->probs[i]; const PrepSummary& r = hs[i];
        P.info.xMin = r.xMin; P.info.xMax = r.xMax; P.info.yMin = r.yMin; P.info.yMax = r.yMax; P.info.zMin = r.zMin; P.info.zMax = r.zMax;
        P.info.scale = r.scale; P.info.size = S; P.info.ncells = r.ncells;
        P.ncolours = r.ncolours;
        if (r.status == PREP_DEGENERATE) return fail(h, GOICP_ERR_ARG, "degenerate model bounding box");
        if (r.status == PREP_COLOURS) return fail(h, GOICP_ERR_UNSUPPORTED, "more than 32 distinct colour codes in one pair (pair %d)", i);
    }
    if ((s = layout_work(h, false))) return s;
    for (auto& P : h->probs) { P.prepared = true; P.dt_built = false; P.initialized = false; }
    return GOICP_OK;
}
void set_cloud(std::vector<float>& xyz, std::vector<int>& c, std::vector<float>& f, const float* pxyz, const int32_t* pc, const float* pf, int n) {
    xyz.assign(pxyz, pxyz + 3 * (size_t)n);
    if (pc) c.assign(pc, pc + n); else c.assign(n, 0);
    if (pf) f.assign(pf, pf + 41 * (size_t)n); else f.clear();
}

