// Kernel launchers (defined next to their kernels in k_*.cu, called by engine.cu).  All asynchronous on `st`.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include "goicp_dev.h"

// k_bnb.cu
int goicp_bnb_default_threads();   // CTA size the kernel is compiled for (launch bounds)
size_t goicp_bnb_smem_floats(int NdP, int NdQ, bool exact, bool needMd, bool needFp);
// useSmem: 0 staging arrays in a global scratch slab, 1 in shared memory, 2 shared memory incl. the DT volume (TMA-staged per call)
int goicp_inner_bnb_occupancy(size_t smemBytes, int exact, int threads, int useSmem, int ct);
cudaError_t goicp_launch_inner_bnb(const PairDev* pairs, const InnerProb* probs, InnerOut* outs, int nprob, int* counter,
                                   HeapEnt* heaps, int heapCap, int maxCtas, float* gscratch, size_t gstride,
                                   int NdP, int NdQ, size_t smemBytes, int useSmem, int gridOff, int S3p, int exact, int ct, int threads, void* memo, int memoCap, DevCounters* ctr, cudaStream_t st, int* ctasLaunched);
cudaError_t goicp_launch_eval_bounds(const PairDev* pairs, int pair, const float* Rs, const int* levels, const WaveCube* cubes,
                                     int nt, float* ub, float* lb, int* incomp_mm, int* fpfh_mm, float* scratch, int nwarps,
                                     cudaStream_t st);
cudaError_t goicp_launch_eval_inclusion(const PairDev* pairs, int pair, const float* R, int level, const WaveCube* cubes, int nt, float* resid, uint8_t* mask, int nwarps, cudaStream_t st);
// k_dt.cu
cudaError_t goicp_launch_dt_replay(PairDev* pairs, int first, int count, int S, cudaStream_t st);
cudaError_t goicp_launch_dt_separable(const GridDev& g, unsigned* bits, unsigned short* nx, unsigned* nxy, int* cid, int numSM, cudaStream_t st);
cudaError_t goicp_launch_dt_vcell(const GridDev& g, int numSM, cudaStream_t st);
cudaError_t goicp_launch_dt_distance(const PairDev* pairs, int pair, const double* xyz, int n, float* out, int* cell, cudaStream_t st);
// k_icp.cu
cudaError_t goicp_launch_icp_begin(const PairDev* pairs, IcpState* states, int n, cudaStream_t st);
cudaError_t goicp_launch_icp_iter(const PairDev* pairs, IcpState* states, int n, int maxNd, int maxNm, int numSM, cudaStream_t st);
cudaError_t goicp_launch_icp_fused(const PairDev* pairs, IcpState* states, int n, cudaStream_t st);
cudaError_t goicp_launch_icp_score(const PairDev* pairs, IcpState* states, int n, cudaStream_t st);
// k_misc.cu
cudaError_t goicp_launch_initialize(PairDev* pairs, int first, int count, cudaStream_t st);
cudaError_t goicp_launch_fpfh_table(PairDev* pairs, int first, int count, int blocksPerPair, cudaStream_t st);
cudaError_t goicp_launch_assign_neighbors(PairDev* pairs, int first, int count, int blocksPerPair, cudaStream_t st);
cudaError_t goicp_launch_normalize(double* xyz, int n, double* out4, cudaStream_t st);
cudaError_t goicp_launch_scale(double* xyz, int n, double scale, cudaStream_t st);
cudaError_t goicp_launch_apply_rigid(const double* xyz, int n, const double* Rt, double* out, cudaStream_t st);
cudaError_t goicp_launch_rescale(const double* in19, double* out3, cudaStream_t st);
cudaError_t goicp_launch_rmsd(const double* a, const double* b, int n, double* terms, float* out, cudaStream_t st);
// k_prep.cu: K1 (packing of the raw clouds, bounding cube, colour dictionary, seeding, cell lists, colour masks)
enum { PREP_OK = 0, PREP_DEGENERATE = 1, PREP_COLOURS = 2 };
struct PrepSummary {          // what the host reads back after K1, per pair
    int status;               // PREP_*
    int ncells, ncolours, pad;
    double xMin, xMax, yMin, yMax, zMin, zMax, scale;
};
struct PrepPair {
    const float *rmxyz, *rdxyz;          // raw clouds: AoS xyz, colour codes or NULL, c-FPFH rows or NULL (read by the pack only)
    const int *rmc, *rdc;
    const float *rmf, *rdf;
    int Nm, NdAll;
    float *mx, *my, *mz, *dx, *dy, *dz;  // input arena: SoA clouds
    int *mcol, *dcol;                    // colour codes (0 where none were given)
    float *mfpfh, *dfpfh;                // descriptor rows, NULL when not kept
    uint8_t *mprop, *dprop, *dknown;     // K1 outputs (PairDev fields of the same names)
    int *cell_vox, *cell_start, *cell_pts, *cell_col;
    uint32_t* cmask;
    int *vcount, *vcid;                  // S^3 scratch (the pair's vnear / vcell of the work arena): points per voxel, then
                                         // the scatter cursor; cell id of each occupied voxel
    int* tmp;                            // Nm: cell members in arrival order
};
#define PREP_BLOCK_VOXELS 4096
inline int goicp_prep_nblocks(int S) { return (int)(((long long)S * S * S + PREP_BLOCK_VOXELS - 1) / PREP_BLOCK_VOXELS); }
// maxElems: the largest per-pair element count of any raw array (41 x points when descriptors are packed)
cudaError_t goicp_launch_prep_pack(const PrepPair* pairs, int npairs, long long maxElems, cudaStream_t st);
// bsum: npairs x goicp_prep_nblocks(S) scratch
cudaError_t goicp_launch_prep(const PrepPair* pairs, PrepSummary* sums, long long* bsum, int npairs, int maxNm, int S, double ef, cudaStream_t st);
// lazy-loading guards (see k_*.cu)
cudaError_t goicp_preload_prep();
cudaError_t goicp_preload_bnb();
cudaError_t goicp_preload_dt();
cudaError_t goicp_preload_icp();
cudaError_t goicp_preload_misc();
