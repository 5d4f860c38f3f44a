// Host engine, part 1: per-pair preprocessing (bounding cube, seeding, cell lists, colour masks), the device layout of a batch,
// the DT build and GoICP::Initialize launches.
#include "engine_internal.h"

// ---- host preprocessing of one pair: bbox/scale (jly_3ddt.cpp:899-931), seeding (:976-995), cell lists and colour
//      masks (assignCellColor jly_goicp.cpp:951-969, checkProperty :1068-1092) -----------------------------------------
goicp_status prepare_problem(Eng* h, Problem& P) {
    const goicp_params& p = h->params;
    const int S = p.distTransSize, num = P.Nm;
    if (S < 2 || S > 1024) return fail(h, GOICP_ERR_UNSUPPORTED, "distTransSize %d outside [2,1024]", S);
    if (num < 1 || P.NdAll < 1) return fail(h, GOICP_ERR_ARG, "empty cloud (Nm=%d Nd=%d)", num, P.NdAll);
    const float* m = P.mxyz.data();
    double xMin = m[0], xMax = m[0], yMin = m[1], yMax = m[1], zMin = m[2], zMax = m[2];
    for (int i = 1; i < num; i++) {
        double x = m[3 * i], y = m[3 * i + 1], z = m[3 * i + 2];
        if (xMin > x) xMin = x; if (xMax < x) xMax = x;
        if (yMin > y) yMin = y; if (yMax < y) yMax = y;
        if (zMin > z) zMin = z; if (zMax < z) zMax = z;
    }
    const double ef = p.distTransExpandFactor;
    const double xC = (xMin + xMax) / 2, yC = (yMin + yMax) / 2, zC = (zMin + zMax) / 2;
    xMin = xC - ef * (xMax - xC); xMax = xC + ef * (xMax - xC);
    yMin = yC - ef * (yMax - yC); yMax = yC + ef * (yMax - yC);
    zMin = zC - ef * (zMax - zC); zMax = zC + ef * (zMax - zC);
    double mx = xMax - xMin > yMax - yMin ? xMax - xMin : yMax - yMin;
    mx = mx > zMax - zMin ? mx : zMax - zMin;
    xMin = xC - mx / 2; xMax = xC + mx / 2; yMin = yC - mx / 2; yMax = yC + mx / 2; zMin = zC - mx / 2; zMax = zC + mx / 2;
    P.info.xMin = xMin; P.info.xMax = xMax; P.info.yMin = yMin; P.info.yMax = yMax; P.info.zMin = zMin; P.info.zMax = zMax;
    P.info.scale = S / mx; P.info.size = S;
    const double scale = P.info.scale;
    if (!(mx > 0)) return fail(h, GOICP_ERR_ARG, "degenerate model bounding box");

    // colour dictionary (<= 32 distinct colours over both clouds)
    std::map<int, int> dict;
    for (int i = 0; i < num; i++) dict.emplace(P.mc.empty() ? 0 : P.mc[i], 0);
    for (int i = 0; i < P.NdAll; i++) dict.emplace(P.dc.empty() ? 0 : P.dc[i], 0);
    if (dict.size() > 32) return fail(h, GOICP_ERR_UNSUPPORTED, "more than 32 distinct colour codes in one pair (%zu)", dict.size());
    { int k = 0; for (auto& kv : dict) kv.second = k++; }
    P.ncolours = (int)dict.size();
    P.mprop.resize(num); P.dprop.resize(P.NdAll); P.dknown.resize(P.NdAll);
    for (int i = 0; i < num; i++) P.mprop[i] = (uint8_t)dict[P.mc.empty() ? 0 : P.mc[i]];
    for (int i = 0; i < P.NdAll; i++) { int c = P.dc.empty() ? 0 : P.dc[i]; P.dprop[i] = (uint8_t)dict[c]; P.dknown[i] = known_prop(c) ? 1 : 0; }

    // seeding: voxel of every model point, cells = occupied voxels in ascending voxel order, points in index order
    std::vector<std::pair<int, int>> vp; vp.reserve(num);
    for (int i = 0; i < num; i++) {
        int x = ROUND_HOST(((double)m[3 * i] - xMin) * scale), y = ROUND_HOST(((double)m[3 * i + 1] - yMin) * scale), z = ROUND_HOST(((double)m[3 * i + 2] - zMin) * scale);
        if (x < 0 || x >= S || y < 0 || y >= S || z < 0 || z >= S) continue;   // :989 (only reachable for expandFactor <= 1)
        vp.emplace_back((z * S + y) * S + x, i);
    }
    std::sort(vp.begin(), vp.end());
    P.cell_vox.clear(); P.cell_start.clear(); P.cell_pts.clear(); P.cell_colour.clear(); P.cmask.clear();
    for (size_t k = 0; k < vp.size(); k++) {
        if (k == 0 || vp[k].first != vp[k - 1].first) { P.cell_vox.push_back(vp[k].first); P.cell_start.push_back((int)k); }
        P.cell_pts.push_back(vp[k].second);
    }
    P.cell_start.push_back((int)vp.size());
    const int nc = (int)P.cell_vox.size();
    P.info.ncells = nc;
    P.cell_colour.resize(nc); P.cmask.assign(nc + 1, 0u);
    for (int c = 0; c < nc; c++) {
        const int b = P.cell_start[c], e = P.cell_start[c + 1];
        auto col = [&](int k) { return P.mc.empty() ? 0 : P.mc[P.cell_pts[k]]; };
        int prop = col(b); bool mixed = false; uint32_t orbits = 0;
        for (int k = b; k < e; k++) { if (col(k) != prop) mixed = true; orbits |= 1u << dict[col(k)]; }
        P.cell_colour[c] = mixed ? -1 : prop;
        P.cmask[c] = mixed ? orbits : (known_prop(prop) ? (1u << dict[prop]) : 0u);   // checkProperty :1068-1092
    }
    P.prepared = true; P.dt_built = false; P.initialized = false;
    return GOICP_OK;
}

// ---- device layout + upload of all problems ----------------------------------------------------------------------
goicp_status upload_problems(Eng* h) {
    const goicp_params& p = h->params;
    const int S = p.distTransSize; const size_t S3 = (size_t)S * S * S;
    const bool useF = p.cfpfh != 0;
    const bool wantVcell = true;
    size_t inTot = 0, workTot = 0;
    for (auto& P : h->probs) {
        if (useF && (P.mf.empty() || P.df.empty())) return fail(h, GOICP_ERR_ARG, "cfpfh=%d needs c-FPFH descriptors for both clouds", p.cfpfh);
        const int nc = P.info.ncells;
        size_t in = 0;
        in += 3 * al256(sizeof(float) * P.NdAll) + 3 * al256(sizeof(float) * P.Nm);
        in += 2 * al256(P.NdAll) + al256(P.Nm);
        if (useF) in += al256(sizeof(float) * 41 * (size_t)P.NdAll) + al256(sizeof(float) * 41 * (size_t)P.Nm);
        in += al256(sizeof(int) * std::max(nc, 1)) + al256(sizeof(uint32_t) * (nc + 1)) + al256(sizeof(int) * (nc + 1)) + al256(sizeof(int) * P.Nm);
        P.inBytes = in; P.inOff = inTot; inTot += in;
        size_t w = 0;
        w += al256(sizeof(float) * S3) + al256(sizeof(int) * S3) + (wantVcell ? 2 * al256(sizeof(int) * S3) + al256(S3 + 16) : 0) + al256(sizeof(double) * GOICP_OVN)
             + (S <= 32 ? al256(2 * (S3 + 16)) + al256(sizeof(float) * (3 * (size_t)(S - 1) * (S - 1) + 6)) : 0);
        w += 2 * al256(sizeof(float) * P.NdAll) + al256(sizeof(float) * GOICP_MAXROTLEVEL * (size_t)P.NdAll);
        if (useF && p.regularizationFPFH > 0) w += al256(sizeof(float) * (size_t)P.NdAll * (nc + 1));
        if (p.regularizationNeighbors > 0) w += al256(sizeof(int) * P.NdAll) + al256(sizeof(int) * P.Nm);
        w += al256(sizeof(unsigned long long) * P.NdAll) + al256(sizeof(int) * P.NdAll) + al256(sizeof(float) * 8 * (size_t)std::max(P.NdAll, 1));
        if (!(p.trimFraction < 0.001)) w += al256(sizeof(unsigned long long) * sort_cap(P.NdAll));
        P.workBytes = w; P.workOff = workTot; workTot += w;
    }
    CU(h->arenaIn.ensure(inTot));
    CU(h->arenaWork.ensure(workTot));
    CU(h->hStage.ensure(inTot));
    char* stage = h->hStage.as<char>();
    char* dIn = h->arenaIn.as<char>(); char* dWork = h->arenaWork.as<char>();
    parallel_for((int)h->probs.size(), [&](int pi) {
        Problem& P = h->probs[pi];
        const int nc = P.info.ncells;
        size_t o = P.inOff;
        PairDev& D = P.dev;
        memset(&D, 0, sizeof D);
        auto putf = [&](float*& dptr, size_t count, auto fill) { dptr = reinterpret_cast<float*>(dIn + o); fill(reinterpret_cast<float*>(stage + o)); o += al256(sizeof(float) * count); };
        putf(D.dx, P.NdAll, [&](float* s) { for (int i = 0; i < P.NdAll; i++) s[i] = P.dxyz[3 * i]; });
        putf(D.dy, P.NdAll, [&](float* s) { for (int i = 0; i < P.NdAll; i++) s[i] = P.dxyz[3 * i + 1]; });
        putf(D.dz, P.NdAll, [&](float* s) { for (int i = 0; i < P.NdAll; i++) s[i] = P.dxyz[3 * i + 2]; });
        putf(D.mx, P.Nm, [&](float* s) { for (int i = 0; i < P.Nm; i++) s[i] = P.mxyz[3 * i]; });
        putf(D.my, P.Nm, [&](float* s) { for (int i = 0; i < P.Nm; i++) s[i] = P.mxyz[3 * i + 1]; });
        putf(D.mz, P.Nm, [&](float* s) { for (int i = 0; i < P.Nm; i++) s[i] = P.mxyz[3 * i + 2]; });
        D.dprop = reinterpret_cast<uint8_t*>(dIn + o); memcpy(stage + o, P.dprop.data(), P.NdAll); o += al256(P.NdAll);
        D.dknown = reinterpret_cast<uint8_t*>(dIn + o); memcpy(stage + o, P.dknown.data(), P.NdAll); o += al256(P.NdAll);
        D.mprop = reinterpret_cast<uint8_t*>(dIn + o); memcpy(stage + o, P.mprop.data(), P.Nm); o += al256(P.Nm);
        if (useF) {
            D.dfpfh = reinterpret_cast<float*>(dIn + o); memcpy(stage + o, P.df.data(), sizeof(float) * 41 * (size_t)P.NdAll); o += al256(sizeof(float) * 41 * (size_t)P.NdAll);
            D.mfpfh = reinterpret_cast<float*>(dIn + o); memcpy(stage + o, P.mf.data(), sizeof(float) * 41 * (size_t)P.Nm); o += al256(sizeof(float) * 41 * (size_t)P.Nm);
        }
        D.g.cell_vox = reinterpret_cast<int*>(dIn + o); memcpy(stage + o, P.cell_vox.data(), sizeof(int) * nc); o += al256(sizeof(int) * std::max(nc, 1));
        D.g.cmask = reinterpret_cast<uint32_t*>(dIn + o); memcpy(stage + o, P.cmask.data(), sizeof(uint32_t) * (nc + 1)); o += al256(sizeof(uint32_t) * (nc + 1));
        D.cell_start = reinterpret_cast<int*>(dIn + o); memcpy(stage + o, P.cell_start.data(), sizeof(int) * (nc + 1)); o += al256(sizeof(int) * (nc + 1));
        D.cell_pts = reinterpret_cast<int*>(dIn + o); memcpy(stage + o, P.cell_pts.data(), sizeof(int) * P.cell_pts.size()); o += al256(sizeof(int) * P.Nm);
        size_t w = P.workOff;
        D.g.dist = reinterpret_cast<float*>(dWork + w); w += al256(sizeof(float) * S3);
        D.g.vnear = reinterpret_cast<int*>(dWork + w); w += al256(sizeof(int) * S3);
        if (wantVcell) { D.g.vcell = reinterpret_cast<int*>(dWork + w); w += al256(sizeof(int) * S3); D.g.vmask = reinterpret_cast<uint32_t*>(dWork + w); w += al256(sizeof(int) * S3); D.g.vmask8 = reinterpret_cast<uint8_t*>(dWork + w); w += al256(S3 + 16); }
        D.g.ovl = reinterpret_cast<double*>(dWork + w); w += al256(sizeof(double) * GOICP_OVN);
        if (S <= 32) {
            D.g.dcode = reinterpret_cast<uint16_t*>(dWork + w); w += al256(2 * (S3 + 16));
            D.g.dlut = reinterpret_cast<float*>(dWork + w); w += al256(sizeof(float) * (3 * (size_t)(S - 1) * (S - 1) + 6));
            D.g.nlut = 3 * (S - 1) * (S - 1) + 2;
        }
        D.normData = reinterpret_cast<float*>(dWork + w); w += al256(sizeof(float) * P.NdAll);
        D.weights = reinterpret_cast<float*>(dWork + w); w += al256(sizeof(float) * P.NdAll);
        D.maxRotDis = reinterpret_cast<float*>(dWork + w); w += al256(sizeof(float) * GOICP_MAXROTLEVEL * (size_t)P.NdAll);
        if (useF && p.regularizationFPFH > 0) { D.fpfhD = reinterpret_cast<float*>(dWork + w); w += al256(sizeof(float) * (size_t)P.NdAll * (nc + 1)); }
        if (p.regularizationNeighbors > 0) { D.nbD = reinterpret_cast<int*>(dWork + w); w += al256(sizeof(int) * P.NdAll); D.nbM = reinterpret_cast<int*>(dWork + w); w += al256(sizeof(int) * P.Nm); }
        D.nn = reinterpret_cast<unsigned long long*>(dWork + w); w += al256(sizeof(unsigned long long) * P.NdAll);
        D.order = reinterpret_cast<int*>(dWork + w); w += al256(sizeof(int) * P.NdAll);
        D.scratch = reinterpret_cast<float*>(dWork + w); w += al256(sizeof(float) * 8 * (size_t)std::max(P.NdAll, 1));
        if (!(p.trimFraction < 0.001)) { D.sortKeys = reinterpret_cast<unsigned long long*>(dWork + w); w += al256(sizeof(unsigned long long) * sort_cap(P.NdAll)); }
        D.g.S = S; D.g.ncells = nc; D.g.xMin = P.info.xMin; D.g.yMin = P.info.yMin; D.g.zMin = P.info.zMin; D.g.scale = P.info.scale;
        D.Nm = P.Nm; D.Nd = P.Nd; D.NdAll = P.NdAll;
    });
    CU(cudaMemcpyAsync(dIn, stage, inTot, cudaMemcpyHostToDevice, h->stream));
    return GOICP_OK;
}

// fills the parameter-derived fields of every PairDev (GoICP::Initialize :180-267 scalars) and uploads the array
goicp_status upload_pairdevs(Eng* h) {
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
    CU(h->dPairs.ensure(sizeof(PairDev) * n));
    CU(h->hPairs.ensure(sizeof(PairDev) * n));
    PairDev* st = h->hPairs.as<PairDev>();
    for (size_t i = 0; i < n; i++) st[i] = h->probs[i].dev;
    CU(cudaMemcpyAsync(h->dPairs.p, st, sizeof(PairDev) * n, cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return GOICP_OK;
}

goicp_status build_dt_all(Eng* h, bool replay) {
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
goicp_status prepare_all(Eng* h) {
    if (!h->haveParams) return fail(h, GOICP_ERR_ARG, "goicp_set_params not called");
    goicp_status s;
    std::atomic<int> bad(0);
    parallel_for((int)h->probs.size(), [&](int i) { goicp_status r = prepare_problem(h, h->probs[i]); if (r) bad.store((int)r); });
    if (bad.load()) return (goicp_status)bad.load();
    if ((s = upload_problems(h))) return s;
    return GOICP_OK;
}
void set_cloud(std::vector<float>& xyz, std::vector<int>& c, std::vector<float>& f, const float* pxyz, const int32_t* pc, const float* pf, int n) {
    xyz.assign(pxyz, pxyz + 3 * (size_t)n);
    if (pc) c.assign(pc, pc + n); else c.assign(n, 0);
    if (pf) f.assign(pf, pf + 41 * (size_t)n); else f.clear();
}

