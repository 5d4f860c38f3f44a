// ICP refinement kernels (north_star (c)): GoICP::ICP (jly_goicp.cpp:102-178) -> ICP3D<float>::Run
// (jly_icp3d.hpp:197-311).  The nanoflann kd-tree is replaced by an exact brute-force nearest-neighbour kernel
// (model cloud tiled through shared memory, same float distance expression as L2_Simple_Adaptor, lowest model index
// wins ties = the tree's first-found rule is order-dependent, exact NN distance is not), the Matrix::svd call by a
// closed-form one-sided Jacobi 3x3 SVD in double (only V*diag(1,1,det)*U^T is consumed, unique for full-rank H).
// All order-sensitive sums of the reference (centroids, err, H, the DT re-score) are done as sequential chains on
// separate lanes so that R, t and the error reproduce the CPU arithmetic.
#include <cstdlib>
#include "icp_device.cuh"
#include "launch.h"

namespace {

__global__ void __launch_bounds__(256)
icp_begin_kernel(const PairDev* __restrict__ pairs, IcpState* __restrict__ states) {
    IcpState& st = states[blockIdx.x];
    icp_begin_part(pairs[st.pair], st);
}

// ---- exact nearest neighbours (replaces nanoflann knnSearch, jly_icp3d.hpp:234-250) --------------------------------
__global__ void __launch_bounds__(NN_THREADS)
icp_nn_kernel(const PairDev* __restrict__ pairs, IcpState* __restrict__ states, int nchunks, int flaggedOnly) {
    const IcpState& st = states[blockIdx.z];
    if (st.done || st.mode != ICP_REFINE) return;
    const PairDev& P = pairs[st.pair];
    const int Nd = P.Nd, Nm = P.Nm;
    if ((int)(blockIdx.x * NN_THREADS) >= Nd) return;
    const int chunk = (Nm + nchunks - 1) / nchunks;
    const int m0 = blockIdx.y * chunk, m1 = min(Nm, m0 + chunk);
    if (m0 >= m1) return;
    __shared__ float sx[NN_TILE], sy[NN_TILE], sz[NN_TILE];
    const int i = blockIdx.x * NN_THREADS + threadIdx.x;
    // flaggedOnly: the grid kernel has answered every point it could; only the flagged ones are left
    const bool mine = i < Nd && (!flaggedOnly || reinterpret_cast<const int*>(P.scratch + 7 * (size_t)Nd)[i] != 0);
    if (!__syncthreads_or(mine ? 1 : 0)) return;
    float q0 = 0.f, q1 = 0.f, q2 = 0.f;
    if (i < Nd) {
        const float r00 = (float)st.R[0], r01 = (float)st.R[1], r02 = (float)st.R[2], r10 = (float)st.R[3], r11 = (float)st.R[4],
                    r12 = (float)st.R[5], r20 = (float)st.R[6], r21 = (float)st.R[7], r22 = (float)st.R[8];
        const float t0 = (float)st.t[0], t1 = (float)st.t[1], t2 = (float)st.t[2];
        const float x = P.dx[i], y = P.dy[i], z = P.dz[i];
        q0 = r00 * x + r01 * y + r02 * z + t0;
        q1 = r10 * x + r11 * y + r12 * z + t1;
        q2 = r20 * x + r21 * y + r22 * z + t2;
    }
    float best = __int_as_float(0x7f800000); int bi = 0;
    for (int base = m0; base < m1; base += NN_TILE) {
        const int cnt = min(NN_TILE, m1 - base);
        __syncthreads();
        for (int k = threadIdx.x; k < cnt; k += NN_THREADS) { sx[k] = P.mx[base + k]; sy[k] = P.my[base + k]; sz[k] = P.mz[base + k]; }
        __syncthreads();
#pragma unroll 4
        for (int k = 0; k < cnt; ++k) {
            const float d0 = q0 - sx[k], d1 = q1 - sy[k], d2 = q2 - sz[k];
            float d = d0 * d0; d = d + d1 * d1; d = d + d2 * d2;
            if (d < best) { best = d; bi = base + k; }
        }
    }
    if (mine) {
        const unsigned long long key = ((unsigned long long)__float_as_uint(best) << 32) | (unsigned)bi;
        atomicMin(P.nn + i, key);
    }
}

// ---- exact nearest neighbours through the DT grid (north_star (c): "a DT/grid-cell NN gather kernel") ------------------------------
// One WARP per data point.  The voxel of the transformed point names its closest occupied cell (GridDev.vcell, the index map the DT
// build emits); the nearest point of that cell bounds the answer, and the occupied voxels of the cube that encloses the bounding
// sphere are then searched through the CSR cell lists, 32 voxels per step.  Same float distance expression and the same tie rule
// (lowest model index: the minimum of the packed (distance bits, index) keys) as the exhaustive kernel, so both give bit-identical
// correspondences.  A point whose cube would exceed `cubeMax` voxels (far from the model: the first iterations of a badly aligned
// start) is flagged instead and left to the tiled exhaustive kernel, which then only works on flagged points.
__global__ void __launch_bounds__(128)
icp_nn_grid_kernel(const PairDev* __restrict__ pairs, IcpState* __restrict__ states, int cubeMax) {
    const IcpState& st = states[blockIdx.y];
    if (st.done || st.mode != ICP_REFINE) return;
    const PairDev& P = pairs[st.pair];
    const GridDev& g = P.g;
    const int Nd = P.Nd, S = g.S, lane = threadIdx.x & 31;
    const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (i >= Nd) return;
    int* far = reinterpret_cast<int*>(P.scratch + 7 * (size_t)Nd);   // row 7 of the scratch: 1 = left to the exhaustive kernel
    const float r00 = (float)st.R[0], r01 = (float)st.R[1], r02 = (float)st.R[2], r10 = (float)st.R[3], r11 = (float)st.R[4],
                r12 = (float)st.R[5], r20 = (float)st.R[6], r21 = (float)st.R[7], r22 = (float)st.R[8];
    const float t0 = (float)st.t[0], t1 = (float)st.t[1], t2 = (float)st.t[2];
    const float x = P.dx[i], y = P.dy[i], z = P.dz[i];
    const float q0 = r00 * x + r01 * y + r02 * z + t0, q1 = r10 * x + r11 * y + r12 * z + t1, q2 = r20 * x + r21 * y + r22 * z + t2;
    const float sc = (float)g.scale;
    const int ix = (int)floorf((q0 - (float)g.xMin) * sc + 0.5f), iy = (int)floorf((q1 - (float)g.yMin) * sc + 0.5f), iz = (int)floorf((q2 - (float)g.zMin) * sc + 0.5f);
    unsigned long long best = GOICP_NN_EMPTY;
    auto visit = [&](int k) {
        const float d0 = q0 - __ldg(P.mx + k), d1 = q1 - __ldg(P.my + k), d2 = q2 - __ldg(P.mz + k);
        float d = d0 * d0; d = d + d1 * d1; d = d + d2 * d2;
        const unsigned long long key = ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)k;
        best = key < best ? key : best;
    };
    auto reduce = [&]() {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { const unsigned long long v = __shfl_xor_sync(GOICP_FULL, best, o); best = v < best ? v : best; }
    };
    const int cx = min(max(ix, 0), S - 1), cy = min(max(iy, 0), S - 1), cz = min(max(iz, 0), S - 1);
    const int cell0 = g.ncells > 0 ? __ldg(g.vcell + ((size_t)cz * S + cy) * S + cx) : g.ncells;
    bool isFar = cell0 >= g.ncells;
    int lx = 0, ly = 0, lz = 0, nx = 0, ny = 0, nz = 0;
    if (!isFar) {
        for (int k = __ldg(P.cell_start + cell0) + lane, e = __ldg(P.cell_start + cell0 + 1); k < e; k += 32) visit(__ldg(P.cell_pts + k));
        reduce();
        const int rv = (int)ceilf(sqrtf(__uint_as_float((unsigned)(best >> 32))) * sc) + 2;   // voxels: the sphere through the best point so far, plus rounding slack
        lx = max(ix - rv, 0); ly = max(iy - rv, 0); lz = max(iz - rv, 0);
        nx = min(ix + rv, S - 1) - lx + 1; ny = min(iy + rv, S - 1) - ly + 1; nz = min(iz + rv, S - 1) - lz + 1;
        if (nx <= 0 || ny <= 0 || nz <= 0 || (long long)nx * ny * nz > cubeMax) isFar = true;
    }
    if (isFar) { if (lane == 0) far[i] = 1; return; }   // (P.nn[i] stays GOICP_NN_EMPTY)
    const int vol = nx * ny * nz;
    for (int c = lane; c < vol; c += 32) {
        const int vx = lx + c % nx, vy = ly + (c / nx) % ny, vz = lz + c / (nx * ny);
        const size_t v = ((size_t)vz * S + vy) * S + vx;
        if (__ldg(g.vnear + v) != (int)v) continue;   // not an occupied voxel
        const int cell = __ldg(g.vcell + v);
        for (int k = __ldg(P.cell_start + cell), e = __ldg(P.cell_start + cell + 1); k < e; ++k) visit(__ldg(P.cell_pts + k));
    }
    reduce();
    if (lane == 0) { P.nn[i] = best; far[i] = 0; }
}

__global__ void __launch_bounds__(256)
icp_update_kernel(const PairDev* __restrict__ pairs, IcpState* __restrict__ states, int rowCap) {
    IcpState& st = states[blockIdx.x];
    if (st.done || st.mode != ICP_REFINE) return;
    extern __shared__ __align__(16) float s_rows[];
    icp_update_part(pairs[st.pair], st, s_rows, rowCap);
}
__global__ void __launch_bounds__(256)
icp_score_kernel(const PairDev* __restrict__ pairs, IcpState* __restrict__ states) {
    IcpState& st = states[blockIdx.x];
    if (st.mode == ICP_COMPAT || (st.mode == ICP_REFINE && (!st.done || st.status != 0))) return;
    icp_score_part(pairs[st.pair], st);
}

__global__ void __launch_bounds__(256, 4)
icp_fused_kernel(const PairDev* __restrict__ pairs, IcpState* states) { __shared__ __align__(16) float s_tile[18 * 512]; icp_fused_body(pairs, states + blockIdx.x, s_tile, 18 * 512); }

}  // namespace

cudaError_t goicp_launch_icp_begin(const PairDev* pairs, IcpState* states, int n, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    icp_begin_kernel<<<n, 256, 0, st>>>(pairs, states);
    return cudaGetLastError();
}
cudaError_t goicp_launch_icp_iter(const PairDev* pairs, IcpState* states, int n, int maxNd, int maxNm, int numSM, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    const int gx = (maxNd + NN_THREADS - 1) / NN_THREADS;
    int gy = (numSM * 4) / (gx * n > 0 ? gx * n : 1);
    if (gy < 1) gy = 1;
    const int maxChunks = (maxNm + NN_TILE - 1) / NN_TILE;
    if (gy > maxChunks) gy = maxChunks;
    if (gy > 65535) gy = 65535;
    // The tiled exhaustive kernel is the default: measured on B200 the grid kernel only pays for clouds far larger than the fork's
    // (bunny 39.5 vs 65.5 ms of ICP per Register, 100k-point model 1247 vs 1195 ms; both bit-identical).  GOICP_ICP_NN_GRID=1 selects it.
    const char* genv = getenv("GOICP_ICP_NN_GRID");   // (read per call: the tests switch it); value = largest bounding radius in voxels (default 6)
    const bool brute = genv == nullptr;
    int rmax = genv ? atoi(genv) : 0; if (rmax < 2) rmax = 6; if (rmax > 40) rmax = 40;
    const int cubeMax = (2 * rmax + 1) * (2 * rmax + 1) * (2 * rmax + 1);
    if (brute) icp_nn_kernel<<<dim3(gx, gy, n), NN_THREADS, 0, st>>>(pairs, states, gy, 0);
    else {
        icp_nn_grid_kernel<<<dim3((maxNd + 3) / 4, n), 128, 0, st>>>(pairs, states, cubeMax);
        icp_nn_kernel<<<dim3(gx, gy, n), NN_THREADS, 0, st>>>(pairs, states, gy, 1);
    }
    // staging for the update's chains: 72 bytes per position, at most 2048 positions (144 KB) at a time
    const size_t rowBytes = (size_t)72 * (maxNd < 2048 ? (maxNd < 32 ? 32 : maxNd) : 2048);
    if (rowBytes > 48 * 1024) { cudaError_t e = cudaFuncSetAttribute(icp_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 72 * 2048); if (e != cudaSuccess) return e; }
    icp_update_kernel<<<n, 256, rowBytes, st>>>(pairs, states, (int)(rowBytes / sizeof(float)));
    return cudaGetLastError();
}
cudaError_t goicp_launch_icp_fused(const PairDev* pairs, IcpState* states, int n, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    icp_fused_kernel<<<n, 256, 0, st>>>(pairs, states);
    return cudaGetLastError();
}
cudaError_t goicp_launch_icp_score(const PairDev* pairs, IcpState* states, int n, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    icp_score_kernel<<<n, 256, 0, st>>>(pairs, states);
    return cudaGetLastError();
}

// forces the (lazily loaded) kernels of this file into the context: a first launch while a resident kernel is spinning
// would otherwise wait for that kernel (CUDA lazy module loading)
cudaError_t goicp_preload_icp() {
    cudaFuncAttributes a; cudaError_t e;
    if ((e = cudaFuncGetAttributes(&a, icp_begin_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, icp_nn_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, icp_nn_grid_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, icp_update_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, icp_score_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, icp_fused_kernel)) != cudaSuccess) return e;
    return cudaSuccess;
}
