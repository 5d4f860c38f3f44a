// Device-side ICP (GoICP::ICP jly_goicp.cpp:102-178 -> ICP3D<float>::Run jly_icp3d.hpp:197-311), shared by the ICP kernels
// (k_icp.cu) and by the resident batch kernel (k_bnb.cu), which serves ICP requests between InnerBnB calls.
#pragma once
#include "dev_common.cuh"

namespace {

constexpr int NN_THREADS = 128;
constexpr int NN_TILE = 512;

// ---- begin: reset workspaces, optional updateCompatibilities at the entry pose (jly_goicp.cpp:933-946) ------------
__device__ __forceinline__ void icp_begin_part(const PairDev& P, IcpState& st) {
    const int Nd = P.Nd;
    __shared__ int s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    int bad = 0;
    for (int i = threadIdx.x; i < Nd; i += blockDim.x) {
        if (st.mode == ICP_REFINE) { P.nn[i] = GOICP_NN_EMPTY; P.order[i] = i; }   // ICP_INIT_ERROR / ICP_COMPAT may share a launch with an ICP_REFINE state of the same pair
        if (st.mode == ICP_COMPAT) {
            const double x0 = P.dx[i], y0 = P.dy[i], z0 = P.dz[i];
            const float x = (float)(st.R[0] * x0 + st.R[1] * y0 + st.R[2] * z0 + st.t[0]);
            const float y = (float)(st.R[3] * x0 + st.R[4] * y0 + st.R[5] * z0 + st.t[1]);
            const float z = (float)(st.R[6] * x0 + st.R[7] * y0 + st.R[8] * z0 + st.t[2]);
            const int cell = clamp_cell(P.g, x, y, z);
            bad += ((P.g.cmask[cell] >> P.dprop[i]) & 1u) ? 0 : 1;
        }
    }
    if (st.mode == ICP_COMPAT) {
        bad = warp_sum_i(bad);
        if ((threadIdx.x & 31) == 0) atomicAdd(&s_cnt, bad);
        __syncthreads();
        if (threadIdx.x == 0) { st.compat_pose = s_cnt; st.done = 1; }
    }
}


// one-sided Jacobi SVD of a 3x3 (double), H = U diag(W) V^T
__device__ void svd3(const double H[9], double U[9], double W[3], double V[9]) {
    double A[9];
    for (int i = 0; i < 9; i++) { A[i] = H[i]; V[i] = (i % 4 == 0) ? 1.0 : 0.0; }
    for (int sweep = 0; sweep < 60; sweep++) {
        double off = 0;
        for (int p = 0; p < 2; p++) for (int q = p + 1; q < 3; q++) {
            double al = 0, be = 0, ga = 0;
            for (int k = 0; k < 3; k++) { al += A[3 * k + p] * A[3 * k + p]; be += A[3 * k + q] * A[3 * k + q]; ga += A[3 * k + p] * A[3 * k + q]; }
            if (ga == 0) continue;
            if (fabs(ga) > off * 0 + 1e-300) { double r = fabs(ga) / sqrt(al * be + 1e-300); if (r > off) off = r; }
            const double zeta = (be - al) / (2 * ga);
            const double t = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1 + zeta * zeta));
            const double cs = 1 / sqrt(1 + t * t), sn = cs * t;
            for (int k = 0; k < 3; k++) {
                const double ap = A[3 * k + p], aq = A[3 * k + q]; A[3 * k + p] = cs * ap - sn * aq; A[3 * k + q] = sn * ap + cs * aq;
                const double vp = V[3 * k + p], vq = V[3 * k + q]; V[3 * k + p] = cs * vp - sn * vq; V[3 * k + q] = sn * vp + cs * vq;
            }
        }
        if (off < 1e-15) break;
    }
    for (int j = 0; j < 3; j++) {
        const double n = sqrt(A[j] * A[j] + A[3 + j] * A[3 + j] + A[6 + j] * A[6 + j]);
        W[j] = n;
        for (int k = 0; k < 3; k++) U[3 * k + j] = n > 0 ? A[3 * k + j] / n : 0;
    }
    // order the singular triplets by descending singular value, as Matrix::svd does (matrix.cpp:770-800): the float `det`
    // of jly_icp3d.hpp:291-297 then scales the same (smallest) direction as in the reference
    for (int a = 0; a < 2; a++) for (int b = a + 1; b < 3; b++) if (W[b] > W[a]) {
        double tw = W[a]; W[a] = W[b]; W[b] = tw;
        for (int k = 0; k < 3; k++) { double tu = U[3 * k + a]; U[3 * k + a] = U[3 * k + b]; U[3 * k + b] = tu; double tv = V[3 * k + a]; V[3 * k + a] = V[3 * k + b]; V[3 * k + b] = tv; }
    }
    for (int j = 0; j < 3; j++) if (W[j] <= 1e-300) {   // rank-deficient column: complete U to an orthonormal basis
        const int a = (j + 1) % 3, b = (j + 2) % 3;
        U[j] = U[3 + a] * U[6 + b] - U[6 + a] * U[3 + b];
        U[3 + j] = U[6 + a] * U[b] - U[a] * U[6 + b];
        U[6 + j] = U[a] * U[3 + b] - U[3 + a] * U[b];
    }
}

// ---- per-iteration update: [trim sort], centroids, err, H, SVD, compose (jly_icp3d.hpp:252-308) ---------------------
// returns true (uniformly) when the call has finished (converged / maxIter / error)
// `sT`/`sCap`: shared-memory staging (16-byte aligned, sCap floats, at least 18*32).  The order-sensitive sums of the reference are
// sequential chains; everything that is NOT on a chain (gathers, float->double conversions, the centred products of H) is produced by
// the whole CTA into `sT`, chunk by chunk, so that a chain step is one shared-memory load and one add.
__device__ __forceinline__ bool icp_update_part(const PairDev& P, IcpState& st, float* sT, int sCap) {
    const int n = P.Nd, num = P.inlierNum, tid = threadIdx.x;
    const int iter0 = st.iter;   // st.iter is only written by thread 0 after the last barrier below
    __shared__ double s_mu[6];
    __shared__ double s_H[9];
    __shared__ float s_err;
    __shared__ int s_done;
    double* D = reinterpret_cast<double*>(sT);
    const int C = min(num > 0 ? num : 1, sCap / 18);   // positions of `order` per chunk: 9 double rows (pass 2) = 18 floats per position

    if (P.doTrim) {   // qsort of POINTREF by dis (:252-255); ties keep index order.  Bitonic sort in the pair's global scratch
        unsigned long long* keys = P.sortKeys;   // next power of two >= Nd keys (engine_setup.cu)
        if (keys == nullptr) { if (tid == 0) { st.status = 3; st.done = 1; } return true; }
        int cap = 32; while (cap < n) cap <<= 1;
        for (int i = tid; i < cap; i += blockDim.x)
            keys[i] = (i < n) ? (((P.nn[i] >> 32) << 32) | (unsigned)i) : GOICP_NN_EMPTY;
        __syncthreads();
        for (int k = 2; k <= cap; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int i = tid; i < cap; i += blockDim.x) {
                    const int ixj = i ^ j;
                    if (ixj > i) {
                        const unsigned long long a = keys[i], b = keys[ixj];
                        const bool up = (i & k) == 0;
                        if ((a > b) == up) { keys[i] = b; keys[ixj] = a; }
                    }
                }
                __syncthreads();
            }
        for (int i = tid; i < n; i += blockDim.x) P.order[i] = (int)(keys[i] & 0xFFFFFFFFu);
        __syncthreads();
    }
    const float r00 = (float)st.R[0], r01 = (float)st.R[1], r02 = (float)st.R[2], r10 = (float)st.R[3], r11 = (float)st.R[4],
                r12 = (float)st.R[5], r20 = (float)st.R[6], r21 = (float)st.R[7], r22 = (float)st.R[8];
    const float t0 = (float)st.t[0], t1 = (float)st.t[1], t2 = (float)st.t[2];
    // pass 1 (:257-271): rows 0-2 = p_m xyz, 3-5 = p_d xyz as doubles, then the float row of squared distances.
    // Seven sequential chains: mu_m, mu_d (double, never reset: Q4) on six lanes of warp 0, err_new on warp 1 (its own warp, so the
    // two loops run side by side instead of as two divergent halves of one warp).
    // err_new: the reference accumulates `float += double(float)`, i.e. (float)((double)e + (double)r).  The double sum of two floats
    // rounded to float equals the float sum (53 >= 2*24+2 bits: double rounding is innocuous for +), so one FADD per element, same bits
    {
        float* E = reinterpret_cast<float*>(D + (size_t)6 * C);
        double acc = 0; float e = 0.f;
        if (tid < 6) acc = (tid < 3) ? st.mu_m[tid] : st.mu_d[tid - 3];
        for (int base = 0; base < num; base += C) {
            const int cnt = min(C, num - base);
            if (base > 0) __syncthreads();
            for (int j = tid; j < cnt; j += blockDim.x) {
                const int id = P.order[base + j];
                const unsigned long long k = P.nn[id];
                const int m = (int)(k & 0xFFFFFFFFu);
                const float x = P.dx[id], y = P.dy[id], z = P.dz[id];
                D[j] = (double)P.mx[m]; D[C + j] = (double)P.my[m]; D[2 * C + j] = (double)P.mz[m];
                D[3 * C + j] = (double)(r00 * x + r01 * y + r02 * z + t0);
                D[4 * C + j] = (double)(r10 * x + r11 * y + r12 * z + t1);
                D[5 * C + j] = (double)(r20 * x + r21 * y + r22 * z + t2);
                E[j] = __uint_as_float((unsigned)(k >> 32));
            }
            __syncthreads();
            if (tid < 6) {
                const double* row = D + (size_t)tid * C;
#pragma unroll 8
                for (int i = 0; i < cnt; ++i) acc = acc + row[i];
            } else if (tid == 32) {
#pragma unroll 8
                for (int i = 0; i < cnt; ++i) e = __fadd_rn(e, E[i]);
            }
        }
        if (tid < 6) s_mu[tid] = acc; else if (tid == 32) s_err = e;
    }
    __syncthreads();
    if (tid == 0) {
        const float err_new = s_err;
        const float err_diff = P.MSEThresh / 10000;                                  // jly_goicp.cpp:232
        int done = 0;
        if (st.err > 0 && st.err - err_new < err_diff * (float)num) done = 1;        // :273
        else {
            st.err = err_new;
            for (int k = 0; k < 6; ++k) s_mu[k] = s_mu[k] / (double)(float)n;        // :278-279: /n, not /num
        }
        for (int k = 0; k < 3; ++k) { st.mu_m[k] = s_mu[k]; st.mu_d[k] = s_mu[3 + k]; }
        s_done = done;
        if (done) st.done = 1;
    }
    __syncthreads();
    if (s_done) return true;
    {   // H = ~q_t * q_m (:284), Matrix operator* accumulates over k in order: nine chains on nine lanes; the centred products
        // (p_d[a] - mu_d[a]) * (p_m[b] - mu_m[b]) are not on the chains and come from the whole CTA
        double s_ = 0;
        const double mm0 = s_mu[0], mm1 = s_mu[1], mm2 = s_mu[2], md0 = s_mu[3], md1 = s_mu[4], md2 = s_mu[5];
        for (int base = 0; base < num; base += C) {
            const int cnt = min(C, num - base);
            __syncthreads();
            for (int j = tid; j < cnt; j += blockDim.x) {
                const int id = P.order[base + j];
                const int m = (int)(P.nn[id] & 0xFFFFFFFFu);
                const float x = P.dx[id], y = P.dy[id], z = P.dz[id];
                const double pm0 = (double)P.mx[m] - mm0, pm1 = (double)P.my[m] - mm1, pm2 = (double)P.mz[m] - mm2;
                const double pd0 = (double)(r00 * x + r01 * y + r02 * z + t0) - md0, pd1 = (double)(r10 * x + r11 * y + r12 * z + t1) - md1,
                             pd2 = (double)(r20 * x + r21 * y + r22 * z + t2) - md2;
                D[j] = pd0 * pm0; D[C + j] = pd0 * pm1; D[2 * C + j] = pd0 * pm2;
                D[3 * C + j] = pd1 * pm0; D[4 * C + j] = pd1 * pm1; D[5 * C + j] = pd1 * pm2;
                D[6 * C + j] = pd2 * pm0; D[7 * C + j] = pd2 * pm1; D[8 * C + j] = pd2 * pm2;
            }
            __syncthreads();
            if (tid < 9) {
                const double* row = D + (size_t)tid * C;
#pragma unroll 8
                for (int k = 0; k < cnt; ++k) s_ = s_ + row[k];
            }
        }
        if (tid < 9) s_H[tid] = s_;
    }
    __syncthreads();
    if (tid == 0) {
        double H[9], U[9], W[3], V[9], R_[9], Rn[9], tn[3], t_[3];
        for (int k = 0; k < 9; ++k) H[k] = s_H[k];
        svd3(H, U, W, V);
        for (int a = 0; a < 3; a++) for (int b = 0; b < 3; b++) { double s = 0; for (int k = 0; k < 3; k++) s += V[3 * a + k] * U[3 * b + k]; R_[3 * a + b] = s; }   // V*~U :287
        const float da = (float)(R_[0] * (R_[4] * R_[8] - R_[5] * R_[7])), db = (float)(-R_[1] * (R_[3] * R_[8] - R_[5] * R_[6])),
                    dc = (float)(R_[2] * (R_[3] * R_[7] - R_[4] * R_[6]));
        const float det = da + db + dc;                                              // T = float :291-297
        for (int a = 0; a < 3; a++) for (int b = 0; b < 3; b++) { double s = 0; for (int k = 0; k < 3; k++) s += V[3 * a + k] * (k == 2 ? (double)det : 1.0) * U[3 * b + k]; R_[3 * a + b] = s; }   // :299-302
        for (int a = 0; a < 3; a++) t_[a] = s_mu[a] - (R_[3 * a] * s_mu[3] + R_[3 * a + 1] * s_mu[4] + R_[3 * a + 2] * s_mu[5]);   // :304
        for (int a = 0; a < 3; a++) {
            for (int b = 0; b < 3; b++) { double s = 0; for (int k = 0; k < 3; k++) s += R_[3 * a + k] * st.R[3 * k + b]; Rn[3 * a + b] = s; }
            tn[a] = R_[3 * a] * st.t[0] + R_[3 * a + 1] * st.t[1] + R_[3 * a + 2] * st.t[2] + t_[a];   // :307-308
        }
        for (int k = 0; k < 9; ++k) st.R[k] = Rn[k];
        for (int k = 0; k < 3; ++k) st.t[k] = tn[k];
        st.iter++;
        if (st.iter >= 10000) st.done = 1;   // maxIter :148
    }
    if (iter0 + 1 < 10000)   // reset for the next nearest-neighbour pass (kept after the last iteration: `points`)
        for (int i = tid; i < n; i += blockDim.x) P.nn[i] = GOICP_NN_EMPTY;
    return iter0 + 1 >= 10000;
}


// ---- scoring: initial error at identity (jly_goicp.cpp:601-627) or the DT re-score of GoICP::ICP (:117-175) ---------
__device__ __forceinline__ void icp_score_part(const PairDev& P, IcpState& st) {
    const int Nd = P.Nd, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float* val = P.scratch + (st.mode == ICP_INIT_ERROR ? 7 * Nd : 0);   // Nd: per data index; ICP_INIT_ERROR may run beside an ICP_REFINE state whose update uses [0, 7 Nd)
    float* fd = P.scratch + Nd;        // Nd: per position of `order`
    __shared__ int s_bad, s_nb;
    __shared__ float s_geom, s_fpfh, s_trim;
    if (tid == 0) { s_bad = 0; s_nb = 0; s_geom = 0.f; s_fpfh = 0.f; s_trim = 0.f; }
    __syncthreads();
    int bad = 0, nb = 0;
    for (int i = tid; i < Nd; i += blockDim.x) {
        float x, y, z;
        if (st.mode == ICP_INIT_ERROR) { x = P.dx[i]; y = P.dy[i]; z = P.dz[i]; }
        else {
            const double x0 = P.dx[i], y0 = P.dy[i], z0 = P.dz[i];
            x = (float)(st.R[0] * x0 + st.R[1] * y0 + st.R[2] * z0 + st.t[0]);       // double expr -> float store :120-122
            y = (float)(st.R[3] * x0 + st.R[4] * y0 + st.R[5] * z0 + st.t[1]);
            z = (float)(st.R[6] * x0 + st.R[7] * y0 + st.R[8] * z0 + st.t[2]);
        }
        const float dt = dt_distance(P.g, P.g.dist, x, y, z);
        val[i] = (st.mode == ICP_REFINE && P.doTrim) ? dt : P.weights[i] * dt;                // :135: no weight when trimming
        if (st.mode == ICP_REFINE) {
            const int idd = P.order[i];
            const int idm = (int)(P.nn[idd] & 0xFFFFFFFFu);
            if (P.cfpfh != 0) {   // computeFPFHDifference(true, i) :1625-1641
                float d = 0.f;
                for (int k = P.fpfh_b; k < P.fpfh_e; ++k) d = d + fabsf(P.dfpfh[(size_t)idd * GOICP_NBINS + k] - P.mfpfh[(size_t)idm * GOICP_NBINS + k]);
                fd[i] = d;
            }
            bad += (P.dknown[idd] && P.dprop[idd] == P.mprop[idm]) ? 0 : 1;   // countCompatibilities :890-914
            if (P.use_nb) nb += abs(P.nbD[idd] - P.nbM[idm]);                  // compareNeighbors(true) :1250-1288
        }
    }
    if (st.mode == ICP_REFINE) { bad = warp_sum_i(bad); nb = warp_sum_i(nb); if (lane == 0) { atomicAdd(&s_bad, bad); atomicAdd(&s_nb, nb); } }
    __syncthreads();
    if (!P.doTrim) {
        if (tid == 0) {   // sequential float sum in index order
            float e = 0.f;
            if (P.norm == 2) { for (int i = 0; i < Nd; ++i) e = e + val[i] * val[i]; }
            else { for (int i = 0; i < Nd; ++i) e = e + val[i]; }
            s_geom = e;
        }
    } else if (warp == 0) {
        float su, sl;
        warp_trimmed_sums(val, Nd, P.inlierNum, lane, (st.mode == ICP_REFINE) ? 2 : P.norm, 0.f, &su, &sl);   // :171-174 always squares
        if (lane == 0) s_trim = su;
    }
    if (st.mode == ICP_REFINE && P.cfpfh != 0 && tid == 32) {
        float f = 0.f;
        for (int i = 0; i < Nd; ++i) f = f + fd[i];
        s_fpfh = f / (float)Nd;                                                      // :147
    }
    __syncthreads();
    if (tid == 0) {
        float error = s_geom;
        if (st.mode == ICP_REFINE) {
            if (P.use_nb) error = error + P.regN * (float)(s_nb * s_nb);              // :149-153
            if (P.use_reg) error = error + P.reg * (float)(s_bad * s_bad);            // :154-159
            if (P.regF > 0.f) error = error + P.regF * (s_fpfh * s_fpfh);             // :160-163
        }
        if (P.doTrim) error = error + s_trim;
        st.error = error; st.incomp = s_bad; st.fpfh = s_fpfh;
        st.done = 1;
    }
}

// ---- small problems: the whole GoICP::ICP call (begin, every ICP3D::Run iteration, DT re-score) in ONE launch, one CTA per
//      request; the model cloud is tiled through shared memory for the exact nearest-neighbour pass ---------------------
// Runs on one CTA (any multiple of 32 threads).  `gstate` may live in mapped host memory: the request is staged in shared memory and
// written back once at the end.
__device__ __forceinline__ void icp_fused_body(const PairDev* __restrict__ pairs, IcpState* gstate, float* tile /* shared, >= 3*NN_TILE floats */, int tileCap /* floats */) {
    __shared__ IcpState st;
    const int tid = threadIdx.x, nthr = blockDim.x;
    __syncthreads();
    // the request lives in mapped host memory and the same address is reused by every ICP request of the pair: read it with
    // volatile loads, a plain load may be served from an L1 line this SM kept from the pair's previous request
    { const volatile unsigned* src = reinterpret_cast<const volatile unsigned*>(gstate); unsigned* dst = reinterpret_cast<unsigned*>(&st);
      for (int k = tid; k < (int)(sizeof(IcpState) / 4); k += nthr) dst[k] = src[k]; }
    __syncthreads();
    const PairDev& P = pairs[st.pair];
    const int Nd = P.Nd, Nm = P.Nm;
    float* sx = tile; float* sy = tile + NN_TILE; float* sz = tile + 2 * NN_TILE;
    icp_begin_part(P, st);
    __syncthreads();
    // the state goes back to (possibly mapped host) memory; the system fence orders it before the completion record that thread 0
    // writes afterwards -- a host that sees the record must see the results
    if (st.mode == ICP_COMPAT) { if (tid == 0) { *gstate = st; __threadfence_system(); } return; }
    if (st.mode == ICP_REFINE) {
        for (;;) {
            const float r00 = (float)st.R[0], r01 = (float)st.R[1], r02 = (float)st.R[2], r10 = (float)st.R[3], r11 = (float)st.R[4],
                        r12 = (float)st.R[5], r20 = (float)st.R[6], r21 = (float)st.R[7], r22 = (float)st.R[8];
            const float t0 = (float)st.t[0], t1 = (float)st.t[1], t2 = (float)st.t[2];
            for (int i0 = 0; i0 < Nd; i0 += nthr) {   // uniform trip count: every thread takes part in the tile loads
                const int i = i0 + tid;
                float q0 = 0.f, q1 = 0.f, q2 = 0.f;
                if (i < Nd) {
                    const float x = P.dx[i], y = P.dy[i], z = P.dz[i];
                    q0 = r00 * x + r01 * y + r02 * z + t0;
                    q1 = r10 * x + r11 * y + r12 * z + t1;
                    q2 = r20 * x + r21 * y + r22 * z + t2;
                }
                float best = __int_as_float(0x7f800000); int bi = 0;
                for (int base = 0; base < Nm; base += NN_TILE) {
                    const int cnt = min(NN_TILE, Nm - base);
                    __syncthreads();
                    for (int k = tid; k < cnt; k += nthr) { sx[k] = P.mx[base + k]; sy[k] = P.my[base + k]; sz[k] = P.mz[base + k]; }
                    __syncthreads();
#pragma unroll 4
                    for (int k = 0; k < cnt; ++k) {
                        const float d0 = q0 - sx[k], d1 = q1 - sy[k], d2 = q2 - sz[k];
                        float d = d0 * d0; d = d + d1 * d1; d = d + d2 * d2;
                        if (d < best) { best = d; bi = base + k; }
                    }
                }
                if (i < Nd) P.nn[i] = ((unsigned long long)__float_as_uint(best) << 32) | (unsigned)bi;
            }
            __syncthreads();
            const bool done = icp_update_part(P, st, tile, tileCap);   // (the model tile is idle during the update)
            __syncthreads();
            if (done) break;
        }
        if (st.status != 0) { if (tid == 0) { *gstate = st; __threadfence_system(); } return; }
    }
    icp_score_part(P, st);
    __syncthreads();
    if (tid == 0) { *gstate = st; __threadfence_system(); }
}


}  // namespace
