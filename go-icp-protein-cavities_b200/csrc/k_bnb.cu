// Branch-and-bound bound evaluation kernels (north_star (b)).
//
//  inner_bnb_kernel   one CTA serves one request: a whole GoICP::InnerBnB call (jly_goicp.cpp:286-579) or the upper- and the
//                     lower-bound call of one rotation cube.  The rotated cloud, weights and rotation-uncertainty radii are
//                     staged in shared memory once; for cavity-sized grids the DT volume is staged too (TMA: 16-bit
//                     squared-distance codes + distance table + colour-mask bytes).  Each pop of the translation queue
//                     evaluates 8 child cubes x Nd points (work item = 32-point chunk x 4 cubes: FP32 magic-number voxel
//                     index with exact FP64 fallback, gather, x weight, - radius, clamp) plus the lattice corners of the
//                     fork's incompatibility / c-FPFH / neighbour-count terms the per-call memo does not hold.
//                     EXACT=true reproduces the reference's sequential float sums bit for bit (16 independent FADD
//                     chains on 16 lanes of one warp), EXACT=false uses warp-shuffle tree sums.
//                     One launch per wave of calls (the wave schedulers of engine_search.cu); the device-resident search (k_search.cu)
//                     runs the same call code (bnb_device.cuh) inside its own kernel.
//  eval_bounds_kernel flat wave: one warp per (rotation cube, translation sub-cube), leaf-level (ub, lb) only.
//
// The translation priority queue (8-byte keys + payload slots, top in shared memory, rest in a per-CTA global slab) follows
// libstdc++'s push_heap/pop_heap step for step so that ties between equal (lb, w) keys pop in the reference's order.
// The structure of one pop and what was measured on the way is in DESIGN.md section 4 and profiles/README.md.
#include "bnb_device.cuh"

namespace {

// Per pop of the translation queue (three CTA barriers):
//   phase A1 (all warps)  work items (32-point chunk, 4 child cubes): a lane loads its point once and evaluates the four
//                         cubes as independent chains (translate -> voxel -> DT gather -> weight, radius, clamp); warp 0 then
//                         files the corner-memo look-ups it issued at the end of the previous pop;
//   phase A2              warp 0 lanes 0..15: the sixteen sequential (ub, lb) sums [EXACT] or the fixed-order combine of the
//                         per-chunk partial sums; all other warps (then warp 0 too): the corners the memo missed, work items
//                         (32-point chunk, 4 corners); trimmed sums: one warp per child;
//   phase C (warp 0)      c-FPFH corner sums, memo update, per-child corner min/max on 8 lanes, the eight decisions as a warp
//                         prefix-min, then lane 0: pushes and the next pop; lanes 0..14 derive the next node's voxel constants
//                         and lanes 0..26 issue its memo look-ups.
// The calls are probs[0..nprob), claimed through counter[0] (one launch per wave).
// GS=true (needs SMEM): the call's DT volume (float distances + one colour-mask byte per voxel) is staged in shared memory by
// TMA as 16-bit squared-distance codes + a distance table + one colour-mask byte per voxel (S^3 * 3 bytes + the table at
// dynamic-smem offset gridOff), so the per-point gathers are LDS instead of L1/L2 sector gathers.
// CT=false: no c-FPFH / neighbour-count corner terms in any pair of the launch (their code and registers drop out).
template <bool EXACT, bool SMEM, bool GS, bool CT>
__global__ void __launch_bounds__(BNB_MAX_THREADS, GOICP_BNB_MIN_CTAS)
inner_bnb_kernel(const PairDev* __restrict__ pairs, const InnerProb* probs, InnerOut* outs,
                 int nprob, int* __restrict__ counter, HeapEnt* __restrict__ heaps, int heapCap,
                 float* gscratch, size_t gstride, int NdP, int NdQ, int useSmem,
                 uint4* memoAll, int memoCap, DevCounters* ctr, int gridOff, int S3p) {
    extern __shared__ float4 dyn_smem4[];
    __shared__ InnerProb s_pr;
    __shared__ InnerOut s_out;
    __shared__ unsigned long long s_gbar;   // mbarrier of the DT staging copies
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    __shared__ struct { int prob; } shk;
    float* icpTile;   // model tile of an ICP request: aliases the staging arrays (the dynamic region holds >= 3*NN_TILE floats)
    if constexpr (SMEM) icpTile = reinterpret_cast<float*>(dyn_smem4); else { __shared__ float s_tile[3 * NN_TILE]; icpTile = s_tile; }
    CallCtx cx;
    __shared__ CancelSh s_cancel;   // unused here (CANCEL = false)
    if (GS) { if (tid == 0) mbar_init(&s_gbar, 1); __syncthreads(); }

    for (;;) {
        __syncthreads();
        {
            if (tid == 0) shk.prob = atomicAdd(counter, 1);
            __syncthreads();
            if (shk.prob >= nprob) {   // the last CTA to leave re-arms the counters, so the host never has to memset them
                if (tid == 0) { __threadfence(); if (atomicAdd(counter + 1, 1) == (int)gridDim.x - 1) { counter[0] = 0; counter[1] = 0; } }
                return;
            }
            if (tid < (int)(sizeof(InnerProb) / 4)) reinterpret_cast<int*>(&s_pr)[tid] = reinterpret_cast<const volatile int*>(probs + shk.prob)[tid];
        }
        __syncthreads();
        const int p = shk.prob;
        const InnerProb& pr = s_pr;   // (stays in shared memory: R is only read while staging)
        inner_call<EXACT, SMEM, GS, CT, false>(pairs, pr, s_out, s_gbar, cx, s_cancel, heaps, heapCap, gscratch, gstride, NdP, NdQ, useSmem, memoAll, memoCap, ctr, gridOff, S3p);
        if (warp == 0) {   // the record leaves the SM as ONE coalesced 64-byte store (it may live in mapped host memory)
            __syncwarp();
            InnerOut* dst = outs + p;
            if (lane < 16) reinterpret_cast<unsigned*>(dst)[lane] = reinterpret_cast<const unsigned*>(&s_out)[lane];
        }
    }
}

// Flat wave: every (rotation cube, translation sub-cube) of a frontier in one launch, one warp per sub-cube.
// Leaf-level bounds (pure functions, SURVEY.md H4) incl. the corner terms; tree sums.
__global__ void __launch_bounds__(256)
eval_bounds_kernel(const PairDev* __restrict__ pairs, int pair, const float* __restrict__ Rs, const int* __restrict__ levels,
                   const WaveCube* __restrict__ cubes, int nt, float* __restrict__ ub_out, float* __restrict__ lb_out,
                   int* __restrict__ incomp_mm, int* __restrict__ fpfh_mm, float* __restrict__ scratch) {
    const int lane = threadIdx.x & 31;
    const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nw = (gridDim.x * blockDim.x) >> 5;
    const PairDev& P = pairs[pair];
    const GridDev& g = P.g;
    const int Nd = P.Nd;
    const int ncp1 = g.ncells + 1;
    const float* __restrict__ dist = g.dist;
    float* md = scratch + (size_t)wid * Nd;   // per-warp residual buffer (trimmed case only)
    for (int k = wid; k < nt; k += nw) {
        const WaveCube cb = cubes[k];
        const float* R = Rs + 9 * cb.rot;
        const int level = levels[cb.rot];
        const float r0 = R[0], r1 = R[1], r2 = R[2], r3 = R[3], r4 = R[4], r5 = R[5], r6 = R[6], r7 = R[7], r8 = R[8];
        const float half = cb.w / 2;
        const float transX = cb.x + half, transY = cb.y + half, transZ = cb.z + half;
        const float mtd = (float)(GOICP_SQRT3 / 2.0 * cb.w);
        float su = 0.f, sl = 0.f;
        int bad[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        int nbs[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        float fs[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int i = lane; i < Nd; i += 32) {
            const float x = P.dx[i], y = P.dy[i], z = P.dz[i];
            const float px = r0 * x + r1 * y + r2 * z, py = r3 * x + r4 * y + r5 * z, pz = r6 * x + r7 * y + r8 * z;
            float d = P.weights[i] * dt_distance(g, dist, px + transX, py + transY, pz + transZ);
            if (level >= 0) d = d - P.maxRotDis[(size_t)level * Nd + i];
            if (d < 0.f) d = 0.f;
            if (P.doTrim) md[i] = d;
            else {
                su += (P.norm == 2) ? d * d : d;
                const float dis = d - mtd;
                if (dis > 0.f) sl += (P.norm == 2) ? dis * dis : dis;
            }
            if (P.use_reg || P.use_fpfh || P.use_nb) {
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const float cx = cb.x + (float)(c & 1) * cb.w, cy = cb.y + (float)((c >> 1) & 1) * cb.w, cz = cb.z + (float)((c >> 2) & 1) * cb.w;
                    const int cell = clamp_cell(g, px + cx, py + cy, pz + cz);
                    if (P.use_reg) bad[c] += ((__ldg(g.cmask + cell) >> P.dprop[i]) & 1u) ? 0 : 1;
                    if (P.use_fpfh) fs[c] += __ldg(P.fpfhD + (size_t)i * ncp1 + cell);
                    if (P.use_nb) nbs[c] += nb_diff(P, cell, i, px + cx, py + cy, pz + cz);
                }
            }
        }
        if (P.doTrim) { __syncwarp(); warp_trimmed_sums(md, Nd, P.inlierNum, lane, P.norm, mtd, &su, &sl); __syncwarp(); }
        else { su = warp_sum(su); sl = warp_sum(sl); }
        int minI = 0, maxI = 0, minN = 0, maxN = 0; float minF = 0.f, maxF = 0.f;
        if (P.use_reg || P.use_fpfh || P.use_nb) {
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                if (P.use_fpfh) { const float f = (float)(int)(warp_sum(fs[c]) / (float)Nd); if (c == 0) { minF = maxF = f; } else { maxF = fmaxf(maxF, f); minF = fminf(minF, f); } }
                if (P.use_reg) { const int n = warp_sum_i(bad[c]); if (c == 0) { minI = maxI = n; } else { maxI = max(maxI, n); minI = min(minI, n); } }
                if (P.use_nb) { const int n = warp_sum_i(nbs[c]); if (c == 0) { minN = maxN = n; } else { maxN = max(maxN, n); minN = min(minN, n); } }
            }
            if (P.use_reg) { su = su + P.reg * (float)(maxI * maxI); sl = sl + P.reg * (float)(minI * minI); }
            if (P.use_nb) { su = su + P.regN * (float)(maxN * maxN); sl = sl + P.regN * (float)(minN * minN); }
            if (P.use_fpfh) { su = su + P.regF * (maxF * maxF); sl = sl + P.regF * (minF * minF); }
        }
        if (lane == 0) {
            ub_out[k] = su; lb_out[k] = sl;
            if (incomp_mm) { incomp_mm[2 * k] = minI; incomp_mm[2 * k + 1] = maxI; }
            if (fpfh_mm) { fpfh_mm[2 * k] = (int)minF; fpfh_mm[2 * k + 1] = (int)maxF; }
        }
    }
}

// Per-cube point-inclusion masks of the trimmed error (north_star: "per-cube point-inclusion masks bit-exact"): one warp per
// child translation cube computes the residual row exactly as the search kernels do (jly_goicp.cpp:343-382) and runs the same
// radix select + membership rule as their trimmed sums (warp_trimmed_sums).  resid / mask: nt x Nd.
__global__ void __launch_bounds__(256)
eval_inclusion_kernel(const PairDev* __restrict__ pairs, int pair, const float* __restrict__ R, int level, const WaveCube* __restrict__ cubes, int nt,
                      float* __restrict__ resid, uint8_t* __restrict__ mask) {
    const int lane = threadIdx.x & 31;
    const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nw = (gridDim.x * blockDim.x) >> 5;
    const PairDev& P = pairs[pair];
    const GridDev& g = P.g;
    const int Nd = P.Nd;
    const float r0 = R[0], r1 = R[1], r2 = R[2], r3 = R[3], r4 = R[4], r5 = R[5], r6 = R[6], r7 = R[7], r8 = R[8];
    for (int k = wid; k < nt; k += nw) {
        const WaveCube cb = cubes[k];
        const float half = cb.w / 2;
        const float transX = cb.x + half, transY = cb.y + half, transZ = cb.z + half;
        float* md = resid + (size_t)k * Nd;
        uint8_t* mk = mask + (size_t)k * Nd;
        for (int i = lane; i < Nd; i += 32) {
            const float x = P.dx[i], y = P.dy[i], z = P.dz[i];
            const float px = r0 * x + r1 * y + r2 * z, py = r3 * x + r4 * y + r5 * z, pz = r6 * x + r7 * y + r8 * z;
            float d = P.weights[i] * dt_distance(g, g.dist, px + transX, py + transY, pz + transZ);
            if (level >= 0) d = d - P.maxRotDis[(size_t)level * Nd + i];
            if (d < 0.f) d = 0.f;
            md[i] = d;
            if (!P.doTrim) mk[i] = 1;
        }
        __syncwarp();
        if (P.doTrim) { float su, sl; warp_trimmed_sums(md, Nd, P.inlierNum, lane, P.norm, 0.f, &su, &sl, mk); }
        __syncwarp();
    }
}

}  // namespace

// ---- launchers ---------------------------------------------------------------------------------------------
int goicp_bnb_default_threads() { return BNB_MAX_THREADS; }
size_t goicp_bnb_smem_floats(int NdP, int NdQ, bool exact, bool needMd, bool needFp) {
    const size_t n = (size_t)5 * NdP + (size_t)(NdP >> 2) + (exact ? 0 : (size_t)((43 * (NdP >> 5) + 3) & ~3)) + (needMd ? (size_t)8 * NdQ : 0) + (needFp ? (size_t)27 * NdQ : 0);
    return n > 3 * 512 ? n : 3 * 512;   // an ICP request tiles the model cloud through the same region (icp_device.cuh NN_TILE)
}

typedef void (*bnb_kernel_t)(const PairDev*, const InnerProb*, InnerOut*, int, int*, HeapEnt*, int, float*, size_t, int, int, int, uint4*, int, DevCounters*, int, int);
template <bool SMEM, bool GS, bool CT>
static bnb_kernel_t bnb_kernel_sel(int exact) { return exact ? inner_bnb_kernel<true, SMEM, GS, CT> : inner_bnb_kernel<false, SMEM, GS, CT>; }
// smem: 0 staging arrays in a global slab, 1 in shared memory, 2 shared memory incl. the DT volume; ct: generic corner terms
static bnb_kernel_t bnb_kernel(int exact, int smem, int ct) {
    if (smem == 2) return ct ? bnb_kernel_sel<true, true, true>(exact) : bnb_kernel_sel<true, true, false>(exact);
    if (smem == 1) return ct ? bnb_kernel_sel<true, false, true>(exact) : bnb_kernel_sel<true, false, false>(exact);
    return ct ? bnb_kernel_sel<false, false, true>(exact) : bnb_kernel_sel<false, false, false>(exact);
}
static int g_bnb_attr_set[16] = {0};
static cudaError_t bnb_attr(int exact, int smem, int ct) {
    const int k = (exact ? 1 : 0) + 2 * smem + 8 * (ct ? 1 : 0);
    if (g_bnb_attr_set[k]) return cudaSuccess;
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, bnb_kernel(exact, smem, ct));
    if (e != cudaSuccess) return e;
    const int maxDyn = 227 * 1024 - (int)fa.sharedSizeBytes - 1024;   // static (queue top, ICP tiles) + dynamic <= 227 KB per CTA
    e = cudaFuncSetAttribute(bnb_kernel(exact, smem, ct), cudaFuncAttributeMaxDynamicSharedMemorySize, maxDyn);
    if (e == cudaSuccess) g_bnb_attr_set[k] = 1;
    return e;
}

cudaError_t goicp_launch_inner_bnb(const PairDev* pairs, const InnerProb* probs, InnerOut* outs, int nprob, int* counter,
                                   HeapEnt* heaps, int heapCap, int maxCtas, float* gscratch, size_t gstride,
                                   int NdP, int NdQ, size_t smemBytes, int useSmem, int gridOff, int S3p, int exact, int ct, int threads, void* memo, int memoCap, DevCounters* ctr, cudaStream_t st, int* ctasLaunched) {
    if (nprob <= 0) { if (ctasLaunched) *ctasLaunched = 0; return cudaSuccess; }
    const size_t smem = useSmem ? smemBytes : 0;
    cudaError_t e = bnb_attr(exact, useSmem, ct);
    if (e != cudaSuccess) return e;
    int grid = nprob < maxCtas ? nprob : maxCtas;
    if (ctasLaunched) *ctasLaunched = grid;
    bnb_kernel(exact, useSmem, ct)<<<grid, threads, smem, st>>>(pairs, probs, outs, nprob, counter, heaps, heapCap, gscratch, gstride, NdP, NdQ, useSmem, (uint4*)memo, memoCap, ctr, gridOff, S3p);
    return cudaGetLastError();
}

int goicp_inner_bnb_occupancy(size_t smemBytes, int exact, int threads, int useSmem, int ct) {
    if (bnb_attr(exact, useSmem, ct) != cudaSuccess) return 1;
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, bnb_kernel(exact, useSmem, ct), threads, useSmem ? smemBytes : 0) != cudaSuccess || n < 1) n = 1;
    return n;
}

cudaError_t goicp_launch_eval_bounds(const PairDev* pairs, int pair, const float* Rs, const int* levels, const WaveCube* cubes,
                                     int nt, float* ub, float* lb, int* incomp_mm, int* fpfh_mm, float* scratch, int nwarps,
                                     cudaStream_t st) {
    if (nt <= 0) return cudaSuccess;
    const int blocks = (nwarps + 7) / 8;
    eval_bounds_kernel<<<blocks, 256, 0, st>>>(pairs, pair, Rs, levels, cubes, nt, ub, lb, incomp_mm, fpfh_mm, scratch);
    return cudaGetLastError();
}

cudaError_t goicp_launch_eval_inclusion(const PairDev* pairs, int pair, const float* R, int level, const WaveCube* cubes, int nt, float* resid, uint8_t* mask, int nwarps, cudaStream_t st) {
    if (nt <= 0) return cudaSuccess;
    eval_inclusion_kernel<<<(nwarps + 7) / 8, 256, 0, st>>>(pairs, pair, R, level, cubes, nt, resid, mask);
    return cudaGetLastError();
}

// forces the (lazily loaded) kernels of this file into the context: a first launch while a resident kernel is spinning
// would otherwise wait for that kernel (CUDA lazy module loading)
cudaError_t goicp_preload_bnb() {
    cudaFuncAttributes a; cudaError_t e;
    for (int exact = 0; exact < 2; exact++) for (int smem = 0; smem < 3; smem++) for (int ct = 0; ct < 2; ct++)
        if ((e = cudaFuncGetAttributes(&a, bnb_kernel(exact, smem, ct))) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, eval_bounds_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, eval_inclusion_kernel)) != cudaSuccess) return e;
    return cudaSuccess;
}
