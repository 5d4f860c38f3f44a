// Data shared by the device-resident search kernel (k_search.cu) and the host engine.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "goicp_dev.h"

#define SR_NGROUP 40                 // slot groups per owner CTA; one group = the calls of the 8 children of one rotation node
#define SR_NSLOT (8 * SR_NGROUP)
#define SR_MAXEV 60                  // improvement events kept per pair (pair 2 of the reference's dataset has 10)
#define GOICP_SR_UNSUPPORTED 3       // = GOICP_ERR_UNSUPPORTED
#define GOICP_SR_OVERFLOW 4          // = GOICP_ERR_OVERFLOW: a queue / event list outgrew its slab; the host re-runs the pair with growing slabs

// One InnerBnB request + its result; its state word lives in SearchArgs.states (contiguous per owner, so that a helper reads all
// of an owner's states in one round trip).  state: 0 free, 1 queued (any CTA may claim it), 2 running, 3 done, 4 skip (child cube outside
// the pi-ball).  Only the owner moves a slot to free / queued / skip; a claim is a compare-and-swap queued -> running; the CTA that
// ran the call stores the result, fences and sets done.
struct alignas(128) SearchSlot {
    unsigned gen;        // the owner's generation when the request was made
    int pad0[3];
    InnerProb pr;        // 48 bytes
    InnerOut out;        // 64 bytes
};
struct alignas(128) OwnerHdr {
    int pair;            // pair this CTA searches (-1: none)
    unsigned gen;        // bumped whenever the pair's incumbent error improves and when the pair ends
    unsigned nQueued;    // slots in state queued (a hint for helpers; may be transiently off by the calls being claimed)
    unsigned pad;
};
// SearchCtl::diag: CTA cycles and event counts, by index rather than field name because the kernel picks some of them at run time
enum SearchDiag {
    DIAG_OWNER_CYCLES, DIAG_PUBLISH_CYCLES, DIAG_HELP_SCAN_CYCLES, DIAG_IDLE_CYCLES, DIAG_OWNER_WAIT_CYCLES,   // CTA cycles: OuterBnB state machine, publishing speculative calls, looking for calls to help with, idle (no pair), owner waiting for a helper's result
    DIAG_HELPER_CALLS, DIAG_HELPER_ABANDONED, DIAG_ICP_CYCLES,   // calls run for another owner, of which abandoned; CTA cycles in ICP
    DIAG_PAIRS_OUT_LAST_NS, DIAG_PAIRS_OUT_FIRST_NS,   // ns after the start when the last / the first CTA found the pair counter run out
    DIAG_PRUNE_CYCLES, DIAG_POP_CYCLES,   // CTA cycles: queue pruning after improvements, rotation-queue pops
    DIAG_POPS_AHEAD, DIAG_POPS_NOT_AHEAD, DIAG_CHILD_READY, DIAG_CHILD_WAITED,   // rotation nodes popped with / without calls made ahead; children whose result was there when the search reached them / waited for
    DIAG_N
};
struct SearchCtl {
    int nextPair, pairsDone, owners, pad;
    unsigned long long diag[DIAG_N];   // diagnostics (GOICP_DEBUG), indexed by SearchDiag
    unsigned long long t0ns;
    int finishHist[256], helpHist[256];
    unsigned wantHelp[32];           // bit per CTA: it has published calls nobody has claimed yet (a hint)
};

struct PairOut {         // GoICP::Register's outputs for one pair
    double R[9], t[3];
    float optError; int optComp;
    long long cnt[6];    // InnerBnB calls, translation pops, translation sub-cubes, rotation pops, rotation cubes, ICP calls
    int status;          // 0, GOICP_SR_*
    int endKind;         // 1 "Rotation Queue Empty", 2 "Threshold reached"
    float endLb;
    int nEvents;
    float tStartMs, tEndMs;   // diagnostics: when the pair was claimed / finished, relative to the kernel's start
    struct { int kind; float v; } ev[SR_MAXEV];   // the "Error*:" trace: kind 0 Init, 1 ICP, 2 BNB
};

struct SearchArgs {
    const PairDev* pairs; int npairs; int nCtas;
    float rotMinX, rotMinY, rotMinZ, rotWidth;   // initNodeRot (jly_main.cpp:241-244)
    int fma;             // which build of sinf / cosf the host libm runs (libm_exact.h)
    int specMax;         // most slot groups attached to rotation-queue nodes (0: never speculate)
    int quietRamp;       // 1: after an improvement the look-ahead restarts at 1 node and doubles per rotation pop
    int walkEvery;       // a full look-ahead walk of the queue front every walkEvery-th rotation pop (in between: incremental)
    int managerRatio;    // an owner stops running calls itself (and only manages) once helpers >= managerRatio x owners (0: never)
    int deepCalls;       // a pair asks for help while unclaimed pairs remain once it has consumed this many InnerBnB calls (one more group per multiple)
    SearchCtl* ctl; OwnerHdr* hdrs; SearchSlot* slots; unsigned* states; void* rq; int rqCap; IcpState* icp; PairOut* outs;
    // inner_call
    HeapEnt* heaps; int heapCap; float* gscratch; size_t gstride; int NdP, NdQ, useSmem; uint4* memo; int memoCap; DevCounters* ctr; int gridOff, S3p;
};

size_t goicp_search_slot_bytes();
size_t goicp_search_hdr_bytes();
size_t goicp_search_rnode_bytes();
int goicp_search_occupancy(size_t smemBytes, int exact, int threads, int useSmem, int ct);
cudaError_t goicp_launch_search(const SearchArgs& A, int ctas, int threads, size_t smemBytes, int exact, int ct, cudaStream_t st);
cudaError_t goicp_preload_search();
