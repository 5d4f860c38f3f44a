// K1, the per-pair preprocessing before the distance transform, for a whole batch on the device: packing of the raw
// clouds into the input arena, the bounding cube (jly_3ddt.cpp:899-931), the colour dictionary, voxel seeding (:976-995),
// the CSR cell lists and the per-cell colour masks (assignCellColor jly_goicp.cpp:951-969, checkProperty :1068-1092).
// Every stage is one launch for the whole batch; the grid size S is shared by all pairs.
#include <limits.h>
#include <algorithm>
#include "launch.h"

namespace {

constexpr int PREP_THREADS = 256;
constexpr int PREP_VPT = PREP_BLOCK_VOXELS / PREP_THREADS;   // consecutive voxels per thread in the scan stages
static_assert(PREP_VPT * PREP_THREADS == PREP_BLOCK_VOXELS, "");

// colour codes of the `properties` enum (transformation.hpp:36) that are keys of the identity compatibility map
// (jly_goicp.cpp:66-73); C = 1 is not a key.
__constant__ int c_known_props[8] = {8204959, 30894, 15219528, 15231913, 4646984, 16741671, 7566712, 0};
__device__ __forceinline__ bool known_prop(int c) {
    bool k = false;
#pragma unroll
    for (int j = 0; j < 8; j++) k |= c_known_props[j] == c;
    return k;
}

// ROUND of jly_3ddt.cpp:30: (int)(x + 0.5), a C cast that truncates toward zero (so -0.7 lands in voxel 0)
__device__ __forceinline__ int voxel_of(const PrepPair& Q, const PrepSummary& s, int S, int i) {
    const int x = (int)(((double)Q.mx[i] - s.xMin) * s.scale + 0.5);
    const int y = (int)(((double)Q.my[i] - s.yMin) * s.scale + 0.5);
    const int z = (int)(((double)Q.mz[i] - s.zMin) * s.scale + 0.5);
    if (x < 0 || x >= S || y < 0 || y >= S || z < 0 || z >= S) return -1;   // :989 (only reachable for expandFactor <= 1)
    return (z * S + y) * S + x;
}

template <int T> __device__ long long block_min(long long v) {
    __shared__ long long w[T / 32];
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) w[threadIdx.x >> 5] = v;
    __syncthreads();
    v = w[0];
    for (int k = 1; k < T / 32; k++) v = min(v, w[k]);
    __syncthreads();
    return v;
}

// exclusive prefix sum over the CTA; *total = the sum of all threads' values
template <int T> __device__ long long block_excl_scan(long long v, long long* total) {
    __shared__ long long w[T / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long x = v;
    for (int o = 1; o < 32; o <<= 1) { const long long y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) w[warp] = x;
    __syncthreads();
    if (warp == 0) {
        long long s = lane < T / 32 ? w[lane] : 0;
        for (int o = 1; o < 32; o <<= 1) { const long long y = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += y; }
        if (lane < T / 32) w[lane] = s;
    }
    __syncthreads();
    const long long pre = (warp ? w[warp - 1] : 0) + x - v;
    *total = w[T / 32 - 1];
    __syncthreads();
    return pre;
}

// raw clouds (AoS xyz, optional colour codes and c-FPFH rows) -> the input arena (SoA xyz, colour codes, descriptor rows)
__global__ void __launch_bounds__(PREP_THREADS) prep_pack_kernel(const PrepPair* __restrict__ pairs, int npairs) {
    for (int p = blockIdx.y; p < npairs; p += gridDim.y) {
        const PrepPair& Q = pairs[p];
        const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
        if (j < Q.Nm) {
            Q.mx[j] = Q.rmxyz[3 * j]; Q.my[j] = Q.rmxyz[3 * j + 1]; Q.mz[j] = Q.rmxyz[3 * j + 2];
            Q.mcol[j] = Q.rmc ? Q.rmc[j] : 0;
        }
        if (j < Q.NdAll) {
            Q.dx[j] = Q.rdxyz[3 * j]; Q.dy[j] = Q.rdxyz[3 * j + 1]; Q.dz[j] = Q.rdxyz[3 * j + 2];
            Q.dcol[j] = Q.rdc ? Q.rdc[j] : 0;
        }
        if (Q.mfpfh && j < (long long)GOICP_NBINS * Q.Nm) Q.mfpfh[j] = Q.rmf[j];
        if (Q.dfpfh && j < (long long)GOICP_NBINS * Q.NdAll) Q.dfpfh[j] = Q.rdf[j];
    }
}

// One CTA per pair: the bounding cube, the colour dictionary and every point's colour index.
__global__ void __launch_bounds__(PREP_THREADS) prep_cube_kernel(const PrepPair* __restrict__ pairs, PrepSummary* __restrict__ sums, int S, double ef) {
    const PrepPair& Q = pairs[blockIdx.x];
    PrepSummary& out = sums[blockIdx.x];
    const int tid = threadIdx.x;
    __shared__ double s_box[6];
    __shared__ int s_dict[33];
    __shared__ int s_n;
    // bounds: min / max of the float coordinates (exact in any order)
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = tid; i < Q.Nm; i += PREP_THREADS) {
        const float v[3] = {Q.mx[i], Q.my[i], Q.mz[i]};
        for (int a = 0; a < 3; a++) { lo[a] = fminf(lo[a], v[a]); hi[a] = fmaxf(hi[a], v[a]); }
    }
    for (int a = 0; a < 3; a++) {   // order-preserving integer keys of the floats: min of keys = min of values
        const int kl = __float_as_int(lo[a]), kh = __float_as_int(hi[a]);
        const long long ml = block_min<PREP_THREADS>(kl < 0 ? (long long)(kl ^ 0x7fffffff) : (long long)kl);
        const long long mh = -block_min<PREP_THREADS>(-(kh < 0 ? (long long)(kh ^ 0x7fffffff) : (long long)kh));
        if (tid == 0) {
            const int bl = (int)ml, bh = (int)mh;
            s_box[2 * a] = (double)__int_as_float(bl < 0 ? bl ^ 0x7fffffff : bl);
            s_box[2 * a + 1] = (double)__int_as_float(bh < 0 ? bh ^ 0x7fffffff : bh);
        }
    }
    if (tid == 0) {   // jly_3ddt.cpp:899-931, every double operation separately rounded (-fmad=false)
        double xMin = s_box[0], xMax = s_box[1], yMin = s_box[2], yMax = s_box[3], zMin = s_box[4], zMax = s_box[5];
        const double xC = (xMin + xMax) / 2, yC = (yMin + yMax) / 2, zC = (zMin + zMax) / 2;
        xMin = xC - ef * (xMax - xC); xMax = xC + ef * (xMax - xC);
        yMin = yC - ef * (yMax - yC); yMax = yC + ef * (yMax - yC);
        zMin = zC - ef * (zMax - zC); zMax = zC + ef * (zMax - zC);
        double mx = xMax - xMin > yMax - yMin ? xMax - xMin : yMax - yMin;
        mx = mx > zMax - zMin ? mx : zMax - zMin;
        out.xMin = xC - mx / 2; out.xMax = xC + mx / 2; out.yMin = yC - mx / 2; out.yMax = yC + mx / 2; out.zMin = zC - mx / 2; out.zMax = zC + mx / 2;
        out.scale = S / mx;
        out.status = (mx > 0) ? PREP_OK : PREP_DEGENERATE;
        out.ncells = 0;
    }
    // colour dictionary: the distinct codes of both clouds in ascending signed order (std::map<int,int>), by repeated
    // extraction of the smallest code above the last one; a 33rd code ends the search
    int n = 0;
    long long last = LLONG_MIN;
    for (; n < 33; n++) {
        long long m = LLONG_MAX;
        for (int i = tid; i < Q.Nm; i += PREP_THREADS) { const long long c = Q.mcol[i]; if (c > last && c < m) m = c; }
        for (int i = tid; i < Q.NdAll; i += PREP_THREADS) { const long long c = Q.dcol[i]; if (c > last && c < m) m = c; }
        m = block_min<PREP_THREADS>(m);
        if (m == LLONG_MAX) break;
        if (tid == 0) s_dict[n] = (int)m;
        last = m;
    }
    if (tid == 0) { s_n = n; out.ncolours = n; if (n > 32 && out.status == PREP_OK) out.status = PREP_COLOURS; }
    __syncthreads();
    if (s_n > 32) return;
    auto index_of = [&](int c) { int lo = 0, hi = s_n - 1; while (lo < hi) { const int mid = (lo + hi) >> 1; if (s_dict[mid] < c) lo = mid + 1; else hi = mid; } return lo; };
    for (int i = tid; i < Q.Nm; i += PREP_THREADS) Q.mprop[i] = (uint8_t)index_of(Q.mcol[i]);
    for (int i = tid; i < Q.NdAll; i += PREP_THREADS) { const int c = Q.dcol[i]; Q.dprop[i] = (uint8_t)index_of(c); Q.dknown[i] = known_prop(c) ? 1 : 0; }
}

__global__ void __launch_bounds__(PREP_THREADS) prep_zero_kernel(const PrepPair* __restrict__ pairs, const PrepSummary* __restrict__ sums, int npairs, long long S3) {
    for (int p = blockIdx.y; p < npairs; p += gridDim.y) {
        if (sums[p].status != PREP_OK) continue;
        int* cnt = pairs[p].vcount;
        for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < S3; v += (long long)gridDim.x * blockDim.x) cnt[v] = 0;
    }
}

// points per voxel
__global__ void __launch_bounds__(PREP_THREADS) prep_count_kernel(const PrepPair* __restrict__ pairs, const PrepSummary* __restrict__ sums, int npairs, int S) {
    for (int p = blockIdx.y; p < npairs; p += gridDim.y) {
        const PrepSummary& s = sums[p];
        const PrepPair& Q = pairs[p];
        const int i = blockIdx.x * blockDim.x + threadIdx.x;
        if (s.status != PREP_OK || i >= Q.Nm) continue;
        const int v = voxel_of(Q, s, S, i);
        if (v >= 0) atomicAdd(Q.vcount + v, 1);
    }
}

// per block of PREP_BLOCK_VOXELS voxels: (occupied voxels << 32) + points
__global__ void __launch_bounds__(PREP_THREADS) prep_block_sums_kernel(const PrepPair* __restrict__ pairs, const PrepSummary* __restrict__ sums, long long* __restrict__ bsum,
                                                                    int npairs, int nb, long long S3) {
    for (int p = blockIdx.y; p < npairs; p += gridDim.y) {
        if (sums[p].status != PREP_OK) continue;
        const int* cnt = pairs[p].vcount;
        const long long v0 = (long long)blockIdx.x * PREP_BLOCK_VOXELS + threadIdx.x * PREP_VPT;
        long long acc = 0;
        for (int k = 0; k < PREP_VPT; k++) if (v0 + k < S3) { const int c = cnt[v0 + k]; acc += c ? (1ll << 32) + c : 0; }
        long long tot;
        block_excl_scan<PREP_THREADS>(acc, &tot);
        if (threadIdx.x == 0) bsum[(size_t)p * nb + blockIdx.x] = tot;
    }
}

// one CTA per pair: exclusive scan of the block sums; ncells, the CSR sentinel and the sentinel cell's empty mask
__global__ void __launch_bounds__(1024) prep_scan_blocks_kernel(const PrepPair* __restrict__ pairs, PrepSummary* __restrict__ sums, long long* __restrict__ bsum, int nb) {
    const int p = blockIdx.x;
    if (sums[p].status != PREP_OK) return;
    long long* b = bsum + (size_t)p * nb;
    long long carry = 0;
    for (int base = 0; base < nb; base += 1024) {
        const int k = base + threadIdx.x;
        const long long v = k < nb ? b[k] : 0;
        long long tot;
        const long long pre = block_excl_scan<1024>(v, &tot);
        if (k < nb) b[k] = carry + pre;
        carry += tot;
    }
    if (threadIdx.x == 0) {
        const PrepPair& Q = pairs[p];
        const int nc = (int)(carry >> 32), npts = (int)(carry & 0xffffffffll);
        sums[p].ncells = nc;
        Q.cell_start[nc] = npts;
        Q.cmask[nc] = 0u;
    }
}

// occupied voxels in ascending order -> cell ids, cell_vox, cell_start; each voxel's count becomes its scatter cursor
__global__ void __launch_bounds__(PREP_THREADS) prep_cells_kernel(const PrepPair* __restrict__ pairs, const PrepSummary* __restrict__ sums, const long long* __restrict__ bsum,
                                                               int npairs, int nb, long long S3) {
    for (int p = blockIdx.y; p < npairs; p += gridDim.y) {
        if (sums[p].status != PREP_OK) continue;
        const PrepPair& Q = pairs[p];
        const long long v0 = (long long)blockIdx.x * PREP_BLOCK_VOXELS + threadIdx.x * PREP_VPT;
        int c[PREP_VPT];
        long long acc = 0;
        for (int k = 0; k < PREP_VPT; k++) { c[k] = v0 + k < S3 ? Q.vcount[v0 + k] : 0; acc += c[k] ? (1ll << 32) + c[k] : 0; }
        long long tot;
        long long off = bsum[(size_t)p * nb + blockIdx.x] + block_excl_scan<PREP_THREADS>(acc, &tot);
        for (int k = 0; k < PREP_VPT; k++) {
            if (!c[k]) continue;
            const int cell = (int)(off >> 32), start = (int)(off & 0xffffffffll);
            const int v = (int)(v0 + k);
            Q.cell_vox[cell] = v; Q.cell_start[cell] = start;
            Q.vcount[v] = start; Q.vcid[v] = cell;
            off += (1ll << 32) + c[k];
        }
    }
}

// every seeded point into its cell, in arrival order
__global__ void __launch_bounds__(PREP_THREADS) prep_scatter_kernel(const PrepPair* __restrict__ pairs, const PrepSummary* __restrict__ sums, int npairs, int S) {
    for (int p = blockIdx.y; p < npairs; p += gridDim.y) {
        const PrepSummary& s = sums[p];
        const PrepPair& Q = pairs[p];
        const int i = blockIdx.x * blockDim.x + threadIdx.x;
        if (s.status != PREP_OK || i >= Q.Nm) continue;
        const int v = voxel_of(Q, s, S, i);
        if (v >= 0) Q.tmp[atomicAdd(Q.vcount + v, 1)] = i;
    }
}

// each point's place in its cell is its rank by index among the cell's points (cells hold a handful of points); the
// cell's first point also writes the cell's colour and mask (assignCellColor :951-969, checkProperty :1068-1092)
__global__ void __launch_bounds__(PREP_THREADS) prep_order_kernel(const PrepPair* __restrict__ pairs, const PrepSummary* __restrict__ sums, int npairs, int S) {
    for (int p = blockIdx.y; p < npairs; p += gridDim.y) {
        const PrepSummary& s = sums[p];
        const PrepPair& Q = pairs[p];
        const int i = blockIdx.x * blockDim.x + threadIdx.x;
        if (s.status != PREP_OK || i >= Q.Nm) continue;
        const int v = voxel_of(Q, s, S, i);
        if (v < 0) continue;
        const int cell = Q.vcid[v], b = Q.cell_start[cell], e = Q.cell_start[cell + 1];
        int rank = 0;
        for (int k = b; k < e; k++) rank += Q.tmp[k] < i;
        Q.cell_pts[b + rank] = i;
        if (rank) continue;
        const int prop = Q.mcol[i];
        bool mixed = false;
        uint32_t orbits = 0;
        for (int k = b; k < e; k++) { const int j = Q.tmp[k]; mixed |= Q.mcol[j] != prop; orbits |= 1u << Q.mprop[j]; }
        Q.cell_col[cell] = mixed ? -1 : prop;
        Q.cmask[cell] = mixed ? orbits : (known_prop(prop) ? 1u << Q.mprop[i] : 0u);
    }
}

inline dim3 pair_grid(long long x, int npairs) { return dim3((unsigned)std::max(1ll, x), (unsigned)std::min(npairs, 65535)); }

}  // namespace

cudaError_t goicp_launch_prep_pack(const PrepPair* pairs, int npairs, long long maxElems, cudaStream_t st) {
    prep_pack_kernel<<<pair_grid((maxElems + PREP_THREADS - 1) / PREP_THREADS, npairs), PREP_THREADS, 0, st>>>(pairs, npairs);
    return cudaGetLastError();
}

cudaError_t goicp_launch_prep(const PrepPair* pairs, PrepSummary* sums, long long* bsum, int npairs, int maxNm, int S, double ef, cudaStream_t st) {
    const long long S3 = (long long)S * S * S;
    const int nb = goicp_prep_nblocks(S);
    const long long ptBlocks = (maxNm + PREP_THREADS - 1) / PREP_THREADS;
    prep_cube_kernel<<<npairs, PREP_THREADS, 0, st>>>(pairs, sums, S, ef);
    prep_zero_kernel<<<pair_grid(std::min<long long>((S3 + PREP_THREADS - 1) / PREP_THREADS, 4096), npairs), PREP_THREADS, 0, st>>>(pairs, sums, npairs, S3);
    prep_count_kernel<<<pair_grid(ptBlocks, npairs), PREP_THREADS, 0, st>>>(pairs, sums, npairs, S);
    prep_block_sums_kernel<<<pair_grid(nb, npairs), PREP_THREADS, 0, st>>>(pairs, sums, bsum, npairs, nb, S3);
    prep_scan_blocks_kernel<<<npairs, 1024, 0, st>>>(pairs, sums, bsum, nb);
    prep_cells_kernel<<<pair_grid(nb, npairs), PREP_THREADS, 0, st>>>(pairs, sums, bsum, npairs, nb, S3);
    prep_scatter_kernel<<<pair_grid(ptBlocks, npairs), PREP_THREADS, 0, st>>>(pairs, sums, npairs, S);
    prep_order_kernel<<<pair_grid(ptBlocks, npairs), PREP_THREADS, 0, st>>>(pairs, sums, npairs, S);
    return cudaGetLastError();
}

cudaError_t goicp_preload_prep() {
    cudaFuncAttributes a; cudaError_t e;
    if ((e = cudaFuncGetAttributes(&a, prep_pack_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, prep_cube_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, prep_zero_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, prep_count_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, prep_block_sums_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, prep_scan_blocks_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, prep_cells_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&a, prep_scatter_kernel)) != cudaSuccess) return e;
    return cudaFuncGetAttributes(&a, prep_order_kernel);
}
