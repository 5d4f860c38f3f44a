/* goicp_b200.h -- C ABI of the B200-native Go-ICP registration engine (libgoicp_b200.so).
 *
 * This is the drop-in boundary for the hot path of guillaumebaldi/Go-ICP-protein-cavities.  The reference has
 * no FFI: its boundary is the C++ class surface of jly_goicp.h / jly_3ddt.h / transformation.hpp.  Each entry
 * point below names the reference interface it replaces (file:line under the reference checkout); the C++
 * drop-in classes with the reference's names (GoICP, DT3D, Transformation; goicp_dropin.hpp) are thin
 * wrappers over these calls, and INTEGRATION.md shows the binding a maintainer adds on the reference side.
 *
 * Conventions: plain pointers and sizes only; every pointer is HOST memory unless the name ends in _dev;
 * all calls return goicp_status (0 = ok) and never throw; a handle owns all of its device memory and one
 * CUDA stream, and is not thread-safe (the reference is single-threaded and non-re-entrant too).
 * There is NO CPU fallback: if no CUDA device is usable every call fails with GOICP_ERR_CUDA.
 */
#ifndef GOICP_B200_H
#define GOICP_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef enum goicp_status {
    GOICP_OK = 0,
    GOICP_ERR_CUDA = 1,        /* no device / CUDA runtime error (see goicp_last_error) */
    GOICP_ERR_ARG = 2,         /* bad argument / call order */
    GOICP_ERR_UNSUPPORTED = 3, /* configuration outside the implemented range */
    GOICP_ERR_OVERFLOW = 4     /* a device-side queue overflowed its scratch capacity */
} goicp_status;

/* config.txt keys, exactly the 18 read by readConfig (jly_main.cpp:231-270).  trimFraction < 0.001 means
 * "no trimming" (jly_main.cpp:259).  Defaults of the shipped config.txt: goicp_params_default(). */
typedef struct goicp_params {
    float MSEThresh;
    float rotMinX, rotMinY, rotMinZ, rotWidth;
    float transMinX, transMinY, transMinZ, transWidth;
    float trimFraction;
    float regularization, regularizationNeighbors, regularizationFPFH;
    int32_t cfpfh, norm, ponderation;
    int32_t distTransSize;
    double distTransExpandFactor;
} goicp_params;

/* DT3D public geometry (jly_3ddt.h:126-128). */
typedef struct goicp_dt_info {
    double xMin, xMax, yMin, yMax, zMin, zMax, scale;
    int32_t size;
    int32_t ncells; /* occupied voxels */
} goicp_dt_info;

/* What jly_main.cpp:131-141 writes per pair, plus search statistics. */
typedef struct goicp_result {
    double R[9];          /* optR, row-major */
    double t[3];          /* optT */
    float optError;
    int32_t optComp;      /* incompatibility count; "Compatibilities" = Nd - optComp */
    int64_t counters[8];  /* 0 InnerBnB calls, 1 translation pops, 2 translation sub-cubes, 3 rotation pops,
                             4 rotation cubes, 5 ICP calls, 6 device launches, 7 speculative InnerBnB re-runs */
    double seconds_dt, seconds_register; /* host wall clock */
    float gpu_ms_dt, gpu_ms_bnb, gpu_ms_icp; /* CUDA-event time of the kernels on the handle's stream */
    int32_t status;       /* goicp_status of this pair */
} goicp_result;

/* One cavity pair of a batch (bo1_GoICP.py:40-54 runs one ./GoICP process per such pair). */
typedef struct goicp_pair_desc {
    const float* model_xyz;  /* Nm x 3, target cloud (already normalised, jly_main.cpp:72-104) */
    const int32_t* model_c;  /* Nm colour codes (transformation.hpp:36) or NULL */
    const float* model_fpfh; /* Nm x 41 or NULL */
    int32_t Nm;
    const float* data_xyz;   /* NdAll x 3, source cloud */
    const int32_t* data_c;
    const float* data_fpfh;
    int32_t NdAll;
    int32_t Nd;              /* NdDownsampled: first Nd points are registered (jly_main.cpp:114-117); 0 = all */
} goicp_pair_desc;

typedef struct goicp_handle_s* goicp_handle;

const char* goicp_version(void);
const char* goicp_last_error(goicp_handle h); /* h may be NULL: error of the last failed goicp_create */
void goicp_params_default(goicp_params* p);   /* shipped config.txt:4-53 */

/* GoICP::GoICP() (jly_goicp.cpp:43).  stream_or_null: an existing cudaStream_t to run on (e.g. torch's
 * current stream) or NULL for a private non-blocking stream. */
goicp_status goicp_create(goicp_handle* out, int device, void* stream_or_null);
void goicp_destroy(goicp_handle h);

/* ---- single registration (the GoICP object of jly_main.cpp:61-123) ---------------------------------- */
/* goicp.pModel/Nm, goicp.pData/Nd assignments (jly_main.cpp:99-104) */
goicp_status goicp_set_model(goicp_handle h, const float* xyz, const int32_t* c, const float* fpfh41, int32_t Nm);
goicp_status goicp_set_data(goicp_handle h, const float* xyz, const int32_t* c, const float* fpfh41, int32_t Nd);
/* readConfig (jly_main.cpp:231) */
goicp_status goicp_set_params(goicp_handle h, const goicp_params* p);
/* GoICP::BuildDT (jly_goicp.cpp:79) = DT3D::Build (jly_3ddt.cpp:897) + assignCellColor (jly_goicp.cpp:951):
 * parallel separable exact EDT + nearest-occupied-cell index map + per-cell colour masks (+ c-FPFH table). */
goicp_status goicp_build_dt(goicp_handle h, goicp_dt_info* out_or_null);
/* Bit-exact replay of the reference's sequential 8SED propagation (jly_3ddt.cpp:716-750) and its
 * emptyCells tie choices (:999-1136); supported for distTransSize <= 32 (SURVEY.md H1). */
goicp_status goicp_build_dt_replay(goicp_handle h, goicp_dt_info* out_or_null);
/* test hook: overwrite the grid with externally produced values (S^3 floats, S^3 x 3 nearest-cell coords) */
goicp_status goicp_dt_upload(goicp_handle h, const float* dist_or_null, const int32_t* nearest_xyz_or_null);
/* DT3D internals for parity: dist[S^3] (index (z*S+y)*S+x), nearest[S^3*3] = emptyCells (cx,cy,cz),
 * cellc[S^3] = CELL.c after assignCellColor (-2 empty, -1 mixed, else the uniform colour). NULL skips. */
goicp_status goicp_dt_download(goicp_handle h, float* dist, int32_t* nearest, int32_t* cellc);
/* DT3D::Distance (jly_3ddt.cpp:1139), batched: xyz n x 3 doubles -> dist[n], cell[n x 3] (unclamped voxel) */
goicp_status goicp_dt_distance(goicp_handle h, const double* xyz, int32_t n, float* dist, int32_t* cell_or_null);
/* `goicp.Nd = NdDownsampled` (jly_main.cpp:114-117) */
goicp_status goicp_set_nd(goicp_handle h, int32_t nd);
/* GoICP::Initialize (jly_goicp.cpp:180): normData, maxRotDis[20][Nd], weights (neighborsWeights :1453),
 * inlierNum, SSEThresh. */
goicp_status goicp_initialize(goicp_handle h);
goicp_status goicp_get_weights(goicp_handle h, float* w /*Nd*/);
goicp_status goicp_get_maxrotdis(goicp_handle h, float* out /*20*Nd*/);
goicp_status goicp_get_thresholds(goicp_handle h, float* sse_thresh, int32_t* inlier_num);

/* The bound evaluation of InnerBnB's inner loop (jly_goicp.cpp:331-550) for nt CHILD translation cubes
 * tcube[nt x 4] = (x,y,z,w), cube k evaluated under rotation R[rot_of[k]] (R: nr x 9 floats, row-major) at
 * rotation level level[rot] (-1: no rotation-uncertainty radius = upper-bound mode, jly_goicp.cpp:375).
 * ub/lb include the corner terms; incomp_minmax / fpfh_minmax (nt x 2, may be NULL) are the (min,max) over the
 * cube's 8 corners.  One launch evaluates every rotation cube x translation sub-cube x point. */
goicp_status goicp_eval_bounds(goicp_handle h, const float* R, const int32_t* level, int32_t nr,
                               const float* tcube, const int32_t* rot_of, int32_t nt,
                               float* ub, float* lb, int32_t* incomp_minmax, int32_t* fpfh_minmax);
/* The trimmed-error selection of InnerBnB (intro_select, jly_sorting.hpp:229-313, called at jly_goicp.cpp:384-390) for nt
 * CHILD translation cubes under one rotation R (9 floats) at `level` (-1: upper-bound mode): mask[nt x Nd] = 1 for the points
 * whose residual is among the inlierNum smallest (the per-cube point-inclusion mask; points tied with the inlierNum-th
 * smallest value are taken in ascending index order), resid[nt x Nd] (may be NULL) = the residual rows themselves
 * (jly_goicp.cpp:343-382).  Without trimming every point is included. */
goicp_status goicp_eval_inclusion(goicp_handle h, const float* R, int32_t level, const float* tcube, int32_t nt,
                                  uint8_t* mask, float* resid_or_null);
/* GoICP::InnerBnB (jly_goicp.cpp:286) for n independent calls made as OuterBnB makes them (:750-768,:861):
 * call k rotates the data by R[k] (9 floats), searches translations best-first on the device and returns
 * err[k] (= optErrorT) and, when tnode != NULL, the best translation node (x,y,z,w). level[k] = -1 for the
 * upper bound, else the rotation level whose uncertainty radii are subtracted. */
goicp_status goicp_inner_bnb(goicp_handle h, const float* R, const int32_t* level, const float* opt_error, int32_t n,
                             float* err, float* tnode_or_null, int64_t* pops_subcubes_or_null /* n x 2 */);
/* GoICP::ICP (jly_goicp.cpp:102) -> ICP3D::Run (jly_icp3d.hpp:197): exact nearest neighbours + closed-form
 * Kabsch update until convergence, then the DT re-score with the fork's terms.  R,t in/out. */
goicp_status goicp_icp(goicp_handle h, double* R /*9*/, double* t /*3*/, float* err, int32_t* corr_or_null /*Nd*/);
/* GoICP::Register (jly_goicp.cpp:878) = Initialize + OuterBnB + Clear; builds the DT if needed. */
goicp_status goicp_register(goicp_handle h, goicp_result* out);
/* GoICP::OuterBnB (jly_goicp.cpp:582-876) alone: the search on a problem that goicp_initialize has prepared (Register = Initialize +
 * OuterBnB + Clear, :878-885). */
goicp_status goicp_outer_bnb(goicp_handle h, goicp_result* out);
/* the "Error*:" improvement trace of the last goicp_register (what OuterBnB prints, jly_goicp.cpp:627-839) */
const char* goicp_last_trace(goicp_handle h);
/* search options: exact_sums=1 (default) reproduces the reference's sequential float sums bit for bit;
 * 0 uses warp-shuffle tree sums (bounds equal to ~1e-6 relative).  spec_width = rotation nodes evaluated
 * speculatively per device launch (results are used only when the reference's order reaches them). */
goicp_status goicp_set_options(goicp_handle h, int32_t exact_sums, int32_t spec_width, int32_t use_dt_replay);

/* Search order of SINGLE registrations.  relaxed_order = 0 (default): the reference's visitation order is reproduced exactly (same
 * node counters and improvement trace).  relaxed_order = 1: frontier waves -- every wave pops the `wave_nodes` (default 64) best
 * rotation nodes, evaluates all their child cubes in one launch and applies the results together (SURVEY H4: visitation order may
 * differ, the certificate optError - min lower bound <= SSEThresh is the reference's, jly_goicp.cpp:685).  -1 leaves a value as is. */
goicp_status goicp_set_search_mode(goicp_handle h, int32_t relaxed_order, int32_t wave_nodes);

/* ---- one deep registration sharded over several GPUs (SURVEY 8(e), second shard) -------------------------------
 * Every rank holds the same clouds / DT and runs the same (deterministic) rotation queue; each wave's InnerBnB calls are
 * dealt round-robin to the ranks and the results are exchanged with ONE all-gather per wave, so every rank sees every
 * bound (the best upper bound per wave is the min over the gathered results) and the search stays identical to the
 * single-GPU one.  `allgather(send, recv, bytes_per_rank, user)` must fill recv[rank * bytes_per_rank ...] for all ranks
 * (host buffers); the python binding implements it with torch.distributed (NCCL on GPUs, gloo in the CPU tests). */
typedef int (*goicp_allgather_fn)(const void* send, void* recv, int64_t bytes_per_rank, void* user);
goicp_status goicp_set_frontier_sharding(goicp_handle h, int32_t rank, int32_t nranks, goicp_allgather_fn allgather, void* user);
/* test hook: runs the exchange on `bytes_per_rank` bytes (no device needed once the handle exists) */
goicp_status goicp_test_exchange(goicp_handle h, const void* send, void* recv, int64_t bytes_per_rank);

/* ---- batch of independent pairs (the dataset sweep of bo1_GoICP.py, one GPU) ------------------------- */
/* BuildDT + Register for npairs pairs with shared params: one DT-build launch, one Initialize launch and ONE search launch for
 * the whole batch (the rotation BnB of every pair runs on the device; CTAs claim pairs from a counter). */
goicp_status goicp_register_batch(goicp_handle h, const goicp_params* p, int32_t npairs,
                                  const goicp_pair_desc* pairs, goicp_result* results);
/* Same, split so that inputs can be made resident first (bench.py "value" leg): upload copies host->device,
 * run does DT build + Initialize + search entirely from HBM, results come back in goicp_batch_run. */
goicp_status goicp_batch_upload(goicp_handle h, const goicp_params* p, int32_t npairs, const goicp_pair_desc* pairs);
goicp_status goicp_batch_run(goicp_handle h, goicp_result* results);
/* goicp_batch_upload with the six cloud pointers of every descriptor in DEVICE memory (device or managed memory of the
 * handle's device), e.g. the storage of CUDA tensors; the descriptor array and its sizes are host memory.  The buffers are
 * read by kernels on the handle's stream, so they are read after work already queued on that stream, and they are not read
 * after the call returns.  A pointer that is not device or managed memory of the handle's device, or a buffer that runs
 * past its allocation, fails with GOICP_ERR_ARG before any launch.  goicp_batch_run follows as after goicp_batch_upload. */
goicp_status goicp_batch_upload_dev(goicp_handle h, const goicp_params* p, int32_t npairs, const goicp_pair_desc* pairs);
/* test hook: the cell lists and colour masks of pair `pair` (0 for a single registration) once its grid is prepared
 * (batch upload or build_dt) -- cell_vox[ncells] ascending voxel indices (z*S+y)*S+x of the occupied voxels,
 * cell_start[ncells+1] CSR offsets into cell_pts[cell_start[ncells]] (<= Nm model point indices, ascending within a cell),
 * cmask[ncells+1] per-cell colour masks (checkProperty, jly_goicp.cpp:1068-1092; the last entry is 0), mprop[Nm] and
 * dprop[NdAll] the colour-dictionary index of every point, info the grid geometry.  NULL skips an output. */
goicp_status goicp_get_cells(goicp_handle h, int32_t pair, int32_t* cell_vox, int32_t* cell_start, int32_t* cell_pts, uint32_t* cmask,
                             uint8_t* mprop, uint8_t* dprop, goicp_dt_info* info);
/* Error cutoff for screening: cutoff[i] ends problem i's search at the first rotation pop whose lower bound lb is >= cutoff[i]
 * while the reference's own end test (optError - lb <= SSEThresh, jly_goicp.cpp:685) does not hold.  Best-first order makes lb a
 * lower bound on the optimum there, so the pair is certified above its cutoff; it returns the incumbent, counters and "Error*:"
 * events it held at that pop and the end line "Cutoff reached\nError*: %g, LB: %g, cutoff: %g".  A pair that is not cut returns
 * exactly what it returns without a cutoff; +inf is no cutoff.  n must equal the number of problems the handle holds (1 after
 * goicp_set_model / goicp_set_data, npairs after a batch upload); NULL clears every cutoff; a NaN or another n fails with
 * GOICP_ERR_ARG.  The batch uploads and goicp_register_batch clear the cutoffs: upload, set the cutoffs, then goicp_batch_run. */
goicp_status goicp_set_error_cutoff(goicp_handle h, const float* cutoff_or_null, int32_t n);
/* how the search of every problem of the last register / batch run ended: kind[i] 1 rotation queue empty, 2 threshold reached
 * (jly_goicp.cpp:685), 3 cutoff reached (goicp_set_error_cutoff); lb[i] the lower bound of its end line (kinds 2 and 3: the
 * lower bound of the node popped last, a certified lower bound on the pair's optimum).  One entry per problem. */
goicp_status goicp_get_search_ends(goicp_handle h, int32_t* kind, float* lb);
/* device-event timings (ms) and launch counts of the last batch_run / register:
 * out[0] dt build, [1] initialize, [2] inner-BnB kernels, [3] ICP kernels, [4] other; launches[0..4] likewise */
goicp_status goicp_get_timings(goicp_handle h, float* ms5, int64_t* launches5);
/* test hook: how many times the handle has copied its per-pair parameter records to the device.  A register or batch run copies
 * them only when something they derive from changed since the last copy (parameters, Nd, clouds, error cutoffs). */
goicp_status goicp_test_pairdev_uploads(goicp_handle h, int64_t* count);
/* wave scheduler only (large clouds, frontier sharding, GOICP_PERSISTENT=0): `groups` worker streams (0 = auto), each advancing
 * `slots` pairs (0 = auto) in lock-step waves and pulling the next pair from a shared counter when one finishes.  The default
 * device-resident search needs no host threads (bo1_GoICP.py:40-54 is one serial process per pair). */
goicp_status goicp_set_batch_options(goicp_handle h, int32_t groups, int32_t slots);
/* search statistics of the last register / batch_run (16 doubles): [0] waves (wave scheduler), [1] InnerBnB calls executed (incl.
 * look-ahead calls that were abandoned), [2] InnerBnB calls the reference order consumed, [3] host worker threads (0: device-resident
 * search), [4] host seconds of the search, [5..7] wave scheduler: host seconds building requests, enqueueing, waiting;
 * device-resident search: [8] calls, [9] translation-queue pops, [10] CTA cycles inside calls, [11] corner evaluations the memo
 * missed, [12] CTA cycles scheduling / waiting / idle, [13] CTAs, [14] pairs re-run by the wave scheduler because a queue outgrew
 * its slab, [15] CTA cycles in total */
goicp_status goicp_get_stats(goicp_handle h, double* out16);

/* ---- Transformation (transformation.cpp), per-pair pre/post-processing -------------------------------- */
/* normalizeMolCloud (:311): centre in place (n x 3 doubles), returns mean[3] and the max norm. */
goicp_status goicp_normalize_cloud(goicp_handle h, double* xyz, int32_t n, double* mean3, double* max_norm);
/* scaleCloud (:355) */
goicp_status goicp_scale_cloud(goicp_handle h, double* xyz, int32_t n, double scale);
/* rescaleCloud (:403-412): t' = -R*meanS + scale*t + meanT */
goicp_status goicp_rescale_translation(goicp_handle h, double scale, const double* meanT, const double* meanS,
                                       const double* R, const double* t, double* out3);
/* applyTransformationProtein (:485-497): out = R*x + t for n atoms */
goicp_status goicp_apply_rigid(goicp_handle h, const double* xyz, int32_t n, const double* R, const double* t, double* out);
/* computeRMSD (:453-464) over n matched atoms */
goicp_status goicp_rmsd(goicp_handle h, const double* a, const double* b, int32_t n, float* rmsd);

#ifdef __cplusplus
}
#endif
#endif
