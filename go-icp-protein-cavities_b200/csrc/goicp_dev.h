// Device-side data layout of one registration problem ("pair") resident in HBM, shared by all kernels.
// Host code (engine.cu) fills these; kernels only read them (except the marked workspaces).
// All file:line citations are relative to the reference checkout (guillaumebaldi/Go-ICP-protein-cavities).
#pragma once
#include <stddef.h>
#include <stdint.h>

#define GOICP_MAXROTLEVEL 20               // jly_goicp.h:95
#define GOICP_NBINS 41                     // c-FPFH descriptor length (jly_main.cpp:306)
#define GOICP_FPFH_SENTINEL 1000000000.0f  // jly_goicp.cpp:1656
#define GOICP_PI 3.1415926536              // jly_goicp.h:44
#define GOICP_SQRT3 1.732050808            // jly_goicp.h:45
#define GOICP_NN_EMPTY 0xFFFFFFFFFFFFFFFFull
#define GOICP_OVLIM 24                      // voxels outside the grid served by the overshoot table GridDev.ovl
#define GOICP_OVN (3 * GOICP_OVLIM * GOICP_OVLIM + 1)
#define GOICP_REQ_BOTH 0x100               // InnerProb.level = GOICP_REQ_BOTH + level: upper-bound call, then the lower-bound call at `level`

// DT3D (jly_3ddt.h:123-139) as laid out in HBM: structure-of-arrays, voxel index (z*S+y)*S+x.
struct GridDev {
    int S;
    int ncells;              // occupied voxels ("cells", jly_3ddt.h:112); id ncells = the empty sentinel cell
    double xMin, yMin, zMin, scale;
    float* dist;             // S^3   DEucl3D.distance / scale   (the 4 B per cube.point bound eval)
    int* vnear;              // S^3   linear voxel index of the nearest occupied voxel (EMPTYCELL); self if none
    int* vcell;              // S^3   compact id of that cell (ncells if the voxel points at an empty cell)
    int* cell_vox;           // ncells   voxel of each occupied cell, ascending
    uint32_t* cmask;         // ncells+1   bit k set <=> a source point of colour index k is compatible (checkProperty)
    uint32_t* vmask;         // S^3   cmask of the voxel's closest cell (one gather for the incompatibility term)
    uint16_t* dcode;         // S^3 (padded to 16) squared voxel distance q of each voxel (nlut-1: no seed), or NULL (S > 32);
    float* dlut;             // nlut  dist as a function of q: the 16-bit form of `dist` that is staged in shared memory
    int nlut;                // 3 (S-1)^2 + 2
    uint8_t* vmask8;         // S^3 (padded to 16)   low byte of vmask: the form staged in shared memory when a pair has <= 8 colours
    double* ovl;             // GOICP_OVN   (double)sqrtf(s) / scale for a squared voxel overshoot s (DT3D::Distance outside the grid)
    // FP32 fast path of ROUND((v-min)*scale) (dev_common.cuh:vox_fast): t = fma(p, vfScale, C) + magic keeps vfShift
    // fractional bits of the voxel coordinate in the float's mantissa; a coordinate closer than the float error bound to a
    // rounding boundary (fraction bits < vfZone) or outside the grid takes the exact FP64 path instead.
    double vfMagic;          // 1.5*2^(23-vfShift) + 0.5 + E*2^-vfShift
    float vfScale;
    int vfShift;
    unsigned vfBias, vfMask, vfZone;   // vfZone = 0xFFFFFFFF disables the fast path
};

// GoICP state after Initialize (jly_goicp.cpp:180-267) for one pair.
struct PairDev {
    GridDev g;
    int Nd, Nm;
    int NdAll;               // every source point given (Nd = the first Nd of them, READMEGo-ICP.md:50)
    int inlierNum;
    int norm;                // 1 or 2
    int doTrim;
    int cfpfh;               // config key; 0 = descriptors unused
    int fpfh_b, fpfh_e;      // c-FPFH bin range selected by `cfpfh` (jly_goicp.cpp:1660-1674)
    int use_reg, use_fpfh;   // regularization > 0 ; regularizationFPFH > 0 && cfpfh != 0 (corner terms, :436)
    int use_nb;              // regularizationNeighbors > 0 (neighbour-count term, :462-466,:489-493,:542-545)
    int ponderation;
    float reg, regF, regN;
    float SSEThresh, MSEThresh, trimFraction;
    float tMinX, tMinY, tMinZ, tWidth;   // initNodeTrans
    float s2[GOICP_MAXROTLEVEL];         // 2*sinf(maxAngle/2) per rotation level, computed on the host (glibc sinf)
    float *dx, *dy, *dz;                 // data (source) cloud, SoA
    float *mx, *my, *mz;                 // model (target) cloud, SoA
    float* normData;                     // Nd
    float* weights;                      // Nd
    float* maxRotDis;                    // [20][Nd]
    uint8_t* dprop;                      // Nd colour index of each data point (0..31)
    uint8_t* mprop;                      // Nm
    uint8_t* dknown;                     // Nd: 1 if the colour is a key of the compatibility map (jly_goicp.cpp:66-73)
    float* dfpfh;                        // Nd x 41
    float* mfpfh;                        // Nm x 41
    int* cell_start;                     // ncells+1 CSR of cellPoints[].points (insertion = index order)
    int* cell_pts;                       // Nm
    float* fpfhD;                        // Nd x (ncells+1): min over the cell's points of the L1 descriptor distance
    int* nbD;                            // NdAll: POINT3D.neighbors of the data points (assignNeighbors :1213-1248); NULL unless use_nb
    int* nbM;                            // Nm
    // ICP workspace (written by the ICP kernels)
    unsigned long long* nn;              // Nd packed (float bits of squared distance << 32 | model index)
    int* order;                          // Nd: id_data of points[i] (identity unless trimmed, jly_icp3d.hpp:252)
    float* scratch;                      // 8*Nd floats
    unsigned long long* sortKeys;        // next power of two >= NdAll (at least 32) keys for the trimmed-ICP sort (NULL unless trimming)
};

struct InnerProb {          // one GoICP::InnerBnB call (jly_goicp.cpp:286)
    int pair;
    int level;              // -1: upper bound (maxRotDisL == NULL)
    float optError;
    float R[9];
};
struct alignas(64) InnerOut {   // one 64-byte record: it leaves the SM as a single coalesced warp store
    unsigned seq0;          // (unused)
    float err;              // optErrorT
    float node[4];          // best translation node x,y,z,w
    int improved;
    int pops;
    int subcubes;
    int status;             // 0 ok, 4 heap overflow
    float err2;             // GOICP_REQ_BOTH: optErrorT, pops and sub-cubes of the lower-bound call; ran2 = 0 if the upper-bound
    int pops2, subcubes2;   // call improved the incumbent (the lower-bound call is then not made)
    int ran2;
    int pad;
    unsigned seq1;
};

struct alignas(16) HeapEnt { float lb, w, x, y, z, pad0, pad1, pad2; };   // TRANSNODE without ub (never read, jly_goicp.h:75-87)

enum IcpMode { ICP_REFINE = 0, ICP_INIT_ERROR = 1, ICP_COMPAT = 2 };   // ICP + re-score (:102), error at the identity (:601-627), updateCompatibilities (:933)
struct IcpState {           // one GoICP::ICP call (jly_goicp.cpp:102) in flight
    int pair;
    int mode;               // IcpMode
    double R[9], t[3];
    double mu_m[3], mu_d[3];  // never reset between iterations (jly_icp3d.hpp:221-222, SURVEY Q4)
    float err;              // previous err (-1 at start)
    int iter;
    int done;
    int status;
    // outputs of the final DT re-score (jly_goicp.cpp:117-175)
    float error;
    int incomp;             // countCompatibilities over the correspondences
    float fpfh;
    int compat_pose;        // checkCompatibility count at the pose (ICP_COMPAT)
};

struct WaveCube { float x, y, z, w; int rot; };   // a child translation cube to evaluate under rotation `rot`

// Counters of one handle's kernels: the corner memo's generation word, then statistics the host reads and clears after each search
struct DevCounters {
    unsigned gen;   // bumped per call: tags the call's entries in the corner memo
    unsigned long long callCycles, pops, cornerMisses, calls;   // all calls: CTA cycles inside calls, translation-queue pops, corner evaluations the memo missed, calls
    unsigned long long idleCycles, unused, icpRequests, ctaCycles;   // search kernel: CTA cycles scheduling / waiting / idle, (none), ICP requests, CTA cycles in total
    unsigned long long phaseCycles[12];   // per-phase cycles of a pop (built with -DGOICP_PHASE_TIMING)
};
static_assert(offsetof(DevCounters, gen) == 0, "");
static_assert(offsetof(DevCounters, callCycles) == 8, "");
static_assert(offsetof(DevCounters, pops) == 16, "");
static_assert(offsetof(DevCounters, cornerMisses) == 24, "");
static_assert(offsetof(DevCounters, calls) == 32, "");
static_assert(offsetof(DevCounters, idleCycles) == 40, "");
static_assert(offsetof(DevCounters, unused) == 48, "");
static_assert(offsetof(DevCounters, icpRequests) == 56, "");
static_assert(offsetof(DevCounters, ctaCycles) == 64, "");
static_assert(offsetof(DevCounters, phaseCycles) == 72 && sizeof(DevCounters) == 168, "");
