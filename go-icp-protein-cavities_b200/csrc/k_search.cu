// Device-resident registration: GoICP::Register (jly_goicp.cpp:878) = OuterBnB (:582-876) + every InnerBnB call (:286-579) + every
// ICP refinement (:102-178) of a whole BATCH of pairs in ONE kernel launch, with no host round trip.
//
//  * The kernel is launched with (SMs x occupancy) CTAs.  A CTA claims a pair from a device counter and becomes its OWNER: warp 0
//    runs the rotation branch-and-bound as a small state machine (rotation queue = a binary heap in the CTA's global slab that
//    follows libstdc++'s push_heap / pop_heap step for step, so equal (lb, w) keys pop in the reference's order; rotation matrices
//    from libm_exact.h = the host libm's own operation sequence), and the whole CTA executes what that needs: InnerBnB calls
//    (bnb_device.cuh:inner_call -- the upper- and lower-bound call of one rotation cube as one request) and GoICP::ICP calls
//    (icp_device.cuh).  While unclaimed pairs remain, every CTA works on its own pair strictly in the reference's order: nothing
//    speculative is ever computed and nothing is polled.
//  * When the pair counter runs out, CTAs without a pair become HELPERS.  An owner then publishes, in the order the reference
//    would make them if the incumbent error does not change, the calls of its current node's remaining children and of the next
//    rotation-queue nodes into its slot array in global memory; helpers scan the owners' slot arrays, claim a slot with a
//    compare-and-swap, run the call and store the result in the slot.  The owner consumes a result only when the reference's order
//    reaches that call (with the same incumbent), so the search stays semantically sequential: optimum, node counters and the
//    improvement trace are those of the reference.  An improvement bumps the owner's generation word; speculative calls made
//    under the old incumbent see it at their next queue pop and stop.
//  * Results (R, t, optError, optComp, counters, improvement events) are written to one record per pair; the host reads the
//    array back once after the kernel.
#include "bnb_device.cuh"
#include "libm_exact.h"
#include "search_dev.h"

namespace {

enum { SL_FREE = 0, SL_QUEUED = 1, SL_RUNNING = 2, SL_DONE = 3, SL_SKIP = 4 };
enum { OW_NONE = 0, OW_START, OW_AFTER_INIT, OW_POP, OW_CHILD, OW_AFTER_IMPROVE };
enum { ACT_NONE = 0, ACT_CALL, ACT_ICP, ACT_EXIT };
enum { RQ_ACTION = 0, RQ_SPAWN, RQ_FINDWORK, RQ_AGAIN, RQ_WAIT };

struct alignas(16) RNodeD { float lb; int l; int group; float ub; float a, b, c, w; };   // ROTNODE (jly_goicp.h:59-73) + the slot group that holds its children's calls

struct OwnerSh {
    int pair, phase;
    float optError, SSE;
    double optR[9], optT[3];
    int optComp;
    long long cnt[6];
    RNodeD par; int j, needLbOnly; float ubChild, lastLb;
    int heapN, nEvents, status;
    int grpUse[SR_NGROUP];       // 0 free, 1 holds the calls of a node (the current one or a queue node), 2 draining (abandoned calls may still run)
    alignas(16) unsigned grpKey[SR_NGROUP][4];   // the node a group belongs to: level and the bits of (a, b, c)
    unsigned grpStamp[SR_NGROUP];                // last look-ahead walk that found the node among the next ones to pop
    unsigned walkStamp;
    int specGroups;              // (diagnostic) groups attached during the last walk
    int action, actOwner, actSlot, actCancel;
    int noMorePairs, lastSpawnJ, manager;
    int waited;
    // incremental look-ahead: a full walk of the queue's front is made every SearchArgs.walkEvery pops; in between only the nodes pushed since
    // the last call are attached, if their lower bound lies inside the window the last walk covered
    int walkLeft, lastTarget, nNew; float winLb; float newLb[8]; alignas(16) unsigned newKey[8][4]; float newW[8];
    int waitPolls;               // manager mode: polls spent waiting for a helper to take the call the search needs next
    int quiet;                   // rotation nodes popped since the incumbent last improved: look-ahead grows 1, 3, 7, ... with it (calls made under an incumbent that is about to improve are wasted)
    // results of the current node's children as last fetched by the warp (a slot that was done then stays done until the owner frees it)
    unsigned pfState[8]; float pfOpt[8]; alignas(64) unsigned pfOut[8][16];   // (rows are read as InnerOut records)
    unsigned short cand[64]; unsigned candKey[64]; int ncand;   // frontier of the look-ahead walk: heap positions and their 32-bit keys (lb bits, low 6 bits clear)
};

__device__ __forceinline__ unsigned ld_vol(const unsigned* p) { return *reinterpret_cast<const volatile unsigned*>(p); }
__device__ __forceinline__ int ld_voli(const int* p) { return *reinterpret_cast<const volatile int*>(p); }
__device__ __forceinline__ void st_vol(unsigned* p, unsigned v) { *reinterpret_cast<volatile unsigned*>(p) = v; }

__device__ __forceinline__ bool rnode_less(const RNodeD& n1, const RNodeD& n2) {   // ROTNODE operator< (jly_goicp.h:64-71)
    if (n1.lb != n2.lb) return n1.lb > n2.lb;
    return n1.w < n2.w;
}
__device__ __forceinline__ RNodeD ld_node(const RNodeD* p) { const float4* q = reinterpret_cast<const float4*>(p); const float4 a = q[0], b = q[1]; RNodeD n; n.lb = a.x; n.l = __float_as_int(a.y); n.group = __float_as_int(a.z); n.ub = a.w; n.a = b.x; n.b = b.y; n.c = b.z; n.w = b.w; return n; }
__device__ __forceinline__ void st_node(RNodeD* p, const RNodeD& n) { float4* q = reinterpret_cast<float4*>(p); q[0] = make_float4(n.lb, __int_as_float(n.l), __int_as_float(n.group), n.ub); q[1] = make_float4(n.a, n.b, n.c, n.w); }
// std::priority_queue<ROTNODE>::push / pop as libstdc++ implements them (__push_heap, __adjust_heap); one lane
__device__ void rq_push(RNodeD* h, int& n, const RNodeD& val) {
    int hole = n++;
    while (hole > 0) {
        const int parent = (hole - 1) / 2;
        const RNodeD pe = ld_node(h + parent);
        if (!rnode_less(pe, val)) break;
        st_node(h + hole, pe); hole = parent;
    }
    st_node(h + hole, val);
}
__device__ RNodeD rq_pop(RNodeD* h, int& n) {
    const RNodeD top = ld_node(h);
    const int len = --n;
    if (len > 0) {
        const RNodeD val = ld_node(h + len);
        int hole = 0, child = 0;
        while (child < (len - 1) / 2) {
            child = 2 * (child + 1);
            RNodeD c1 = ld_node(h + child); const RNodeD c0 = ld_node(h + child - 1);
            if (rnode_less(c1, c0)) { child--; c1 = c0; }
            st_node(h + hole, c1); hole = child;
        }
        if ((len & 1) == 0 && child == (len - 2) / 2) { child = 2 * (child + 1); st_node(h + hole, ld_node(h + child - 1)); hole = child - 1; }
        while (hole > 0) {
            const int parent = (hole - 1) / 2;
            const RNodeD pe = ld_node(h + parent);
            if (!rnode_less(pe, val)) break;
            st_node(h + hole, pe); hole = parent;
        }
        st_node(h + hole, val);
    }
    return top;
}

// child cube j of a rotation node (jly_goicp.cpp:707-712) and its rotation matrix (:716-747); false: the cube lies outside the pi-ball (:723)
__device__ __forceinline__ RNodeD child_of(const RNodeD& par, int j) {
    RNodeD nr; nr.w = par.w / 2; nr.l = par.l + 1; nr.group = -1; nr.ub = 0.f; nr.lb = 0.f;
    nr.a = par.a + (float)(j & 1) * nr.w; nr.b = par.b + (float)((j >> 1) & 1) * nr.w; nr.c = par.c + (float)((j >> 2) & 1) * nr.w;
    return nr;
}
__device__ bool child_rotation(bool fma, const RNodeD& nr, float* R) {
    float v1 = nr.a + nr.w / 2, v2 = nr.b + nr.w / 2, v3 = nr.c + nr.w / 2;
    const float t = __fsqrt_rn(v1 * v1 + v2 * v2 + v3 * v3);
    if ((double)t - GOICP_SQRT3 * (double)nr.w / 2 > GOICP_PI) return false;
    if (t > 0) {
        v1 = __fdiv_rn(v1, t); v2 = __fdiv_rn(v2, t); v3 = __fdiv_rn(v3, t);
        const float ct = libm_exact::cosf_glibc(fma, t), ct2 = 1 - ct, st = libm_exact::sinf_glibc(fma, t);
        const float tmp121 = v1 * v2 * ct2, tmp122 = v3 * st, tmp131 = v1 * v3 * ct2, tmp132 = v2 * st, tmp231 = v2 * v3 * ct2, tmp232 = v1 * st;
        R[0] = ct + v1 * v1 * ct2; R[1] = tmp121 - tmp122; R[2] = tmp131 + tmp132;
        R[3] = tmp121 + tmp122; R[4] = ct + v2 * v2 * ct2; R[5] = tmp231 - tmp232;
        R[6] = tmp131 - tmp132; R[7] = tmp231 + tmp232; R[8] = ct + v3 * v3 * ct2;
    } else {
        for (int k = 0; k < 9; k++) R[k] = (k % 4 == 0) ? 1.f : 0.f;
    }
    return true;
}

struct Cta {   // what every routine of this file needs about the CTA's place in the world
    const SearchArgs& A;
    OwnerSh& os;
    SearchSlot* slots;       // this CTA's own slots ...
    unsigned* st;            // ... and their state words: SL_* in the low byte, queued calls carry their priority above it
    OwnerHdr* hdr;           // this CTA's header
    RNodeD* rq;              // this CTA's rotation queue
    IcpState* icp;           // this CTA's two ICP states
    int me, lane;
    float* scr;              // >= 4 KB of shared memory that is idle while the scheduler runs (the staging region of the calls)
};
__device__ __forceinline__ unsigned st_of(unsigned w) { return w & 0xFFu; }
__device__ __forceinline__ unsigned queued_word(unsigned prio) { return SL_QUEUED | (prio & 0xFFFFFF00u); }   // prio: float bits of the node's lb (>= 0: bit order = value order)

__device__ __forceinline__ void add_event(Cta& c, int kind, float v) {
    OwnerSh& os = c.os;
    if (os.nEvents < SR_MAXEV) { PairOut& o = c.A.outs[os.pair]; o.ev[os.nEvents].kind = kind; o.ev[os.nEvents].v = v; }
    else os.status = GOICP_SR_OVERFLOW;
    os.nEvents++;
}

// a request for child `ch` (rotation R) of the current incumbent into slot s; the state word is set by the caller
__device__ __forceinline__ void fill_request(Cta& c, SearchSlot* s, const RNodeD& ch, const float* R, bool lbOnly) {
    const int lbLevel = min(ch.l, GOICP_MAXROTLEVEL - 1);   // Q2: the reference indexes maxRotDis[level] without a bound check; clamped
    s->pr.pair = c.os.pair; s->pr.level = lbOnly ? lbLevel : GOICP_REQ_BOTH + lbLevel; s->pr.optError = c.os.optError;
#pragma unroll
    for (int k = 0; k < 9; k++) s->pr.R[k] = R[k];
    s->gen = ld_vol(&c.hdr->gen);
}
// withdraws a queued call; false if a helper has just claimed it
__device__ __forceinline__ bool withdraw(Cta& c, int s, unsigned w) {
    if (atomicCAS(c.st + s, w, (unsigned)SL_FREE) == w) { atomicSub(&c.hdr->nQueued, 1u); return true; }
    return false;
}

// the incumbent changed (or the pair ended): every speculative call is void.  Unclaimed ones are withdrawn, running ones are left to
// finish (they notice the new generation at their next pop); their groups drain.  Called by all lanes of warp 0.
__device__ void invalidate_spec(Cta& c) {
    OwnerSh& os = c.os;
    if (c.lane == 0) { st_vol(&c.hdr->gen, ld_vol(&c.hdr->gen) + 1u); __threadfence(); }
    __syncwarp();
    for (int s = c.lane; s < SR_NSLOT; s += 32) {
        if (os.grpUse[s >> 3] == 0) continue;
        const unsigned w = ld_vol(c.st + s);
        if (st_of(w) == SL_QUEUED) withdraw(c, s, w);
        else if (st_of(w) == SL_DONE || st_of(w) == SL_SKIP) st_vol(c.st + s, SL_FREE);
    }
    __syncwarp();
    if (c.lane == 0) { for (int g = 0; g < SR_NGROUP; g++) if (os.grpUse[g] != 0) os.grpUse[g] = 2; os.specGroups = 0; }
    if (c.lane < 8) os.pfState[c.lane] = SL_FREE;
    __syncwarp();
}
__device__ __forceinline__ uint4 node_key(const RNodeD& n) { return make_uint4((unsigned)n.l, __float_as_uint(n.a), __float_as_uint(n.b), __float_as_uint(n.c)); }
// the group that holds the calls of node `key`, or -1.  Lane 0 (serial form, used at a pop).
__device__ int lookup_group(Cta& c, const uint4 key) {
    OwnerSh& os = c.os;
    for (int g = 0; g < SR_NGROUP; g++) {
        if (os.grpUse[g] != 1) continue;
        const uint4 k = *reinterpret_cast<const uint4*>(os.grpKey[g]);
        if (k.x == key.x && k.y == key.y && k.z == key.z && k.w == key.w) return g;
    }
    return -1;
}
// the same by all lanes
__device__ __forceinline__ int lookup_group_w(Cta& c, const uint4 key) {
    OwnerSh& os = c.os;
    int f = -1;
    for (int g = c.lane; g < SR_NGROUP; g += 32) {
        if (os.grpUse[g] != 1) continue;
        const uint4 k = *reinterpret_cast<const uint4*>(os.grpKey[g]);
        if (k.x == key.x && k.y == key.y && k.z == key.z && k.w == key.w) f = g;
    }
    return __reduce_max_sync(GOICP_FULL, f);
}
// empties group g: unclaimed calls are withdrawn, finished ones dropped; false if a call is still running somewhere (the group
// then drains: grpUse = 2)
__device__ bool clear_group(Cta& c, int g) {
    bool busy = false;
    for (int k = 0; k < 8; k++) {
        const unsigned w = ld_vol(c.st + 8 * g + k);
        unsigned st = st_of(w);
        if (st == SL_QUEUED) st = withdraw(c, 8 * g + k, w) ? SL_FREE : SL_RUNNING;
        if (st == SL_RUNNING) busy = true; else if (st != SL_FREE) st_vol(c.st + 8 * g + k, SL_FREE);
    }
    c.os.grpUse[g] = busy ? 2 : 0;
    return !busy;
}
// A group for a node: a free one, a drained one, or -- when every group is taken -- the one whose node has been longest out of
// the look-ahead window (its node sank in the queue; speculation follows the front).  -1: nothing available right now.  Lane 0.
__device__ int alloc_group(Cta& c, int keep) {
    OwnerSh& os = c.os;
    for (int g = 0; g < SR_NGROUP; g++) {
        if (os.grpUse[g] == 2) clear_group(c, g);
        if (os.grpUse[g] == 0) { os.grpUse[g] = 1; return g; }
    }
    for (int tries = 0; tries < 4; tries++) {
        int victim = -1; unsigned oldest = 0;
        for (int g = 0; g < SR_NGROUP; g++) {
            if (os.grpUse[g] != 1 || g == keep || os.grpStamp[g] == os.walkStamp) continue;
            const unsigned age = os.walkStamp - os.grpStamp[g];
            if (victim < 0 || age > oldest) { victim = g; oldest = age; }
        }
        if (victim < 0) return -1;
        if (clear_group(c, victim)) { os.grpUse[victim] = 1; return victim; }
    }
    return -1;
}

__device__ void finish_pair(Cta& c, int endKind) {   // lane 0
    OwnerSh& os = c.os;
    PairOut& o = c.A.outs[os.pair];
    for (int k = 0; k < 9; k++) o.R[k] = os.optR[k];
    for (int k = 0; k < 3; k++) o.t[k] = os.optT[k];
    o.optError = os.optError; o.optComp = os.optComp;
    for (int k = 0; k < 6; k++) o.cnt[k] = os.cnt[k];
    { unsigned long long now; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now)); o.tEndMs = (float)((now - c.A.ctl->t0ns) * 1e-6); }
    o.status = os.status; o.endKind = endKind; o.endLb = endKind == 2 ? os.par.lb : os.lastLb; o.nEvents = min(os.nEvents, SR_MAXEV);
}

// The state words of the current node's 8 children in one load, then the result records of the finished ones (two round trips to
// L2 for the whole node instead of a dozen dependent ones per child).  All lanes of warp 0.
__device__ __forceinline__ void prefetch_group(Cta& c) {
    OwnerSh& os = c.os;
    const int g = os.par.group, lane = c.lane;
    unsigned w = SL_FREE;
    if (lane < 8) w = ld_vol(c.st + 8 * g + lane);
    const unsigned doneMask = __ballot_sync(GOICP_FULL, lane < 8 && st_of(w) == SL_DONE && os.pfState[lane & 7] != SL_DONE);
    __threadfence();
    if (doneMask) {
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int k = (lane + 32 * q) >> 4, word = (lane + 32 * q) & 15;
            if ((doneMask >> k) & 1u) os.pfOut[k][word] = reinterpret_cast<const volatile unsigned*>(&c.slots[8 * g + k].out)[word];
        }
        if (lane < 8 && ((doneMask >> lane) & 1u)) os.pfOpt[lane] = *reinterpret_cast<const volatile float*>(&c.slots[8 * g + lane].pr.optError);
    }
    if (lane < 8 && os.pfState[lane] != SL_DONE) os.pfState[lane] = st_of(w);
    __syncwarp();
}

__device__ __forceinline__ void note_pushed(OwnerSh& os, const RNodeD& n) {   // lane 0
    if (os.nNew < 8) { const int q = os.nNew++; os.newLb[q] = n.lb; os.newW[q] = n.w; os.newKey[q][0] = (unsigned)n.l; os.newKey[q][1] = __float_as_uint(n.a); os.newKey[q][2] = __float_as_uint(n.b); os.newKey[q][3] = __float_as_uint(n.c); }
    else os.walkLeft = 0;
}
// ---- the OuterBnB state machine, lane 0 of the owner's warp 0.  Returns what it needs next. --------------------------------------
__device__ __forceinline__ int owner_serial(Cta& c) {
    OwnerSh& os = c.os;
    const SearchArgs& A = c.A;
    for (;;) {
        switch (os.phase) {
        case OW_START: {   // initial error (:601-627) and ICP from the identity (:634)
            const PairDev& P = A.pairs[os.pair];
            { unsigned long long now; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now)); A.outs[os.pair].tStartMs = (float)((now - A.ctl->t0ns) * 1e-6); }
            os.quiet = 0; os.walkLeft = 0; os.lastTarget = -1; os.nNew = 0; os.winLb = 0.f;
            os.SSE = P.SSEThresh; os.optComp = 0; os.status = 0; os.nEvents = 0; os.heapN = 0; os.lastLb = 0.f; os.needLbOnly = 0;
            for (int k = 0; k < 6; k++) os.cnt[k] = 0;
            for (int k = 0; k < 9; k++) os.optR[k] = (k % 4 == 0) ? 1.0 : 0.0;
            os.optT[0] = os.optT[1] = os.optT[2] = 0.0;
            for (int q = 0; q < 2; q++) {
                IcpState& s = c.icp[q];
                s.pair = os.pair; s.mode = q == 0 ? ICP_INIT_ERROR : ICP_REFINE;
                for (int k = 0; k < 9; k++) s.R[k] = (k % 4 == 0) ? 1.0 : 0.0;
                for (int k = 0; k < 3; k++) { s.t[k] = 0.0; s.mu_m[k] = 0.0; s.mu_d[k] = 0.0; }
                s.err = -1.f; s.iter = 0; s.done = 0; s.status = 0; s.error = 0.f; s.incomp = 0; s.fpfh = 0.f; s.compat_pose = 0;
            }
            __threadfence();
            os.phase = OW_AFTER_INIT; os.action = ACT_ICP;
            return RQ_ACTION;
        }
        case OW_AFTER_INIT: {   // :623-661
            const PairDev& P = A.pairs[os.pair];
            const volatile IcpState* s0 = c.icp; const volatile IcpState* s1 = c.icp + 1;
            if (s0->status != 0 || s1->status != 0) { os.status = GOICP_SR_UNSUPPORTED; finish_pair(c, 0); os.phase = OW_NONE; break; }
            float optError = s0->error;
            if (P.reg > 0) optError += P.reg * (float)(P.Nd * P.Nd);                       // :623
            if (P.regF > 0) optError += P.regF * (float)(100 * 8 * 100 * 8);               // :624
            if (P.regN > 0) optError += P.regN * (float)(P.Nd * 6 * P.Nd * 6);             // :625
            os.optError = optError;
            add_event(c, 0, optError);
            os.cnt[5]++;
            const float icpErr = s1->error;
            if (icpErr < os.optError) {                                                    // :636-661
                os.optError = icpErr;
                for (int k = 0; k < 9; k++) os.optR[k] = s1->R[k];
                for (int k = 0; k < 3; k++) os.optT[k] = s1->t[k];
                os.optComp = s1->incomp;
                add_event(c, 1, icpErr);
            }
            RNodeD root; root.a = A.rotMinX; root.b = A.rotMinY; root.c = A.rotMinZ; root.w = A.rotWidth; root.l = 0; root.lb = 0.f; root.ub = 0.f; root.group = -1;
            rq_push(c.rq, os.heapN, root);
            os.phase = OW_POP;
            break;
        }
        case OW_POP: {
            if (os.status != 0) { finish_pair(c, 0); os.phase = OW_NONE; break; }
            if (os.heapN == 0) { finish_pair(c, 1); os.phase = OW_NONE; break; }                   // :670-677
            os.quiet++;
            { const long long tp0 = clock64(); os.par = rq_pop(c.rq, os.heapN); atomicAdd(&A.ctl->diag[DIAG_POP_CYCLES], (unsigned long long)(clock64() - tp0)); } os.cnt[3]++;
            if ((os.optError - os.par.lb) <= os.SSE) { finish_pair(c, 2); os.phase = OW_NONE; break; }   // :685
            {
                const uint4 key = node_key(os.par);
                int g = lookup_group(c, key);   // calls made ahead of time for this node?
                atomicAdd(&A.ctl->diag[g >= 0 ? DIAG_POPS_AHEAD : DIAG_POPS_NOT_AHEAD], 1ull);
                if (g < 0) {
                    // (no victim: every group has calls running -- they stop at their next pop if abandoned -- or carries the current
                    //  walk stamp, which the pops between two full walks do not advance: age them; the next look-ahead is a full walk)
                    while ((g = alloc_group(c, -1)) < 0) { os.walkStamp++; os.walkLeft = 0; __nanosleep(200); }
                    *reinterpret_cast<uint4*>(os.grpKey[g]) = key;
                }
                os.grpStamp[g] = os.walkStamp + 1u;   // the walk that follows must not take it away
                os.par.group = g;
            }
            for (int k = 0; k < 8; k++) os.pfState[k] = SL_FREE;
            os.j = 0; os.needLbOnly = 0; os.phase = OW_CHILD; os.lastSpawnJ = 0;
            return RQ_SPAWN;
        }
        case OW_CHILD: {
            if (os.j >= 8) {
                for (int k = 0; k < 8; k++) st_vol(c.st + 8 * os.par.group + k, SL_FREE);
                os.grpUse[os.par.group] = 0;
                os.phase = OW_POP; break;
            }
            const int sidx = 8 * os.par.group + os.j;
            SearchSlot* sl = c.slots + sidx;
            if (os.pfState[os.j] == SL_DONE) { atomicAdd(&A.ctl->diag[os.waited ? DIAG_CHILD_WAITED : DIAG_CHILD_READY], 1ull); os.waited = 0; os.waitPolls = 0; } else os.waited = 1;
            if (os.pfState[os.j] != SL_DONE) {   // not finished when the warp last looked: what is it doing now?
                const unsigned w = ld_vol(c.st + sidx);
                const unsigned st = st_of(w);
                if (st == SL_DONE) return RQ_AGAIN;   // finished meanwhile: fetch its record
                if (st == SL_SKIP) { os.j++; break; }
                if (st == SL_FREE) {
                    if (A.specMax > 0 && os.lastSpawnJ != os.j && os.cnt[0] >= 16) { os.lastSpawnJ = os.j; os.walkLeft = 0; return RQ_SPAWN; }   // helpers may have appeared since the last pop
                    const RNodeD ch = child_of(os.par, os.j);
                    float R[9];
                    if (!child_rotation(A.fma != 0, ch, R)) { os.j++; break; }
                    fill_request(c, sl, ch, R, os.needLbOnly != 0);
                    if (os.manager) {   // plenty of helpers: the owner only manages; a helper runs the call
                        __threadfence(); st_vol(c.st + sidx, queued_word(0u)); atomicAdd(&c.hdr->nQueued, 1u); atomicOr(&A.ctl->wantHelp[c.me >> 5], 1u << (c.me & 31));
                        return RQ_WAIT;
                    }
                    st_vol(c.st + sidx, SL_RUNNING);
                    os.action = ACT_CALL; os.actOwner = c.me; os.actSlot = sidx; os.actCancel = 0;
                    return RQ_ACTION;
                }
                if (st == SL_QUEUED) {
                    if (os.manager && ++os.waitPolls < 400) { atomicOr(&A.ctl->wantHelp[c.me >> 5], 1u << (c.me & 31)); return RQ_WAIT; }   // (a helper that found nothing a moment ago may have cleared the hint; after ~50 us without a taker the owner runs the call itself)
                    if (atomicCAS(c.st + sidx, w, (unsigned)SL_RUNNING) == w) {
                        atomicSub(&c.hdr->nQueued, 1u);
                        __threadfence();
                        os.action = ACT_CALL; os.actOwner = c.me; os.actSlot = sidx; os.actCancel = 0;
                        return RQ_ACTION;
                    }
                    break;   // a helper took it this instant
                }
                return os.manager ? RQ_WAIT : RQ_FINDWORK;   // running on a helper: do something useful meanwhile
            }
            // done: consume in the reference's order (the record was fetched by prefetch_group)
            const InnerOut& o = *reinterpret_cast<const InnerOut*>(os.pfOut[os.j]);
            os.pfState[os.j] = SL_FREE;
            if (o.status == 7) { st_vol(c.st + sidx, SL_FREE); break; }   // abandoned under an older generation (cannot be the call we wait for, but harmless): redo
            if (o.status != 0) { os.status = GOICP_SR_OVERFLOW; finish_pair(c, 0); os.phase = OW_NONE; break; }
            if (os.pfOpt[os.j] != os.optError) { st_vol(c.st + sidx, SL_FREE); break; }     // made under another incumbent: redo (defensive; invalidation withdraws these)
            if (!os.needLbOnly) {
                os.cnt[4]++; os.cnt[0]++; os.cnt[1] += o.pops; os.cnt[2] += o.subcubes;     // :768
                os.ubChild = o.err;
                if (o.err < os.optError) {                                                  // :771-790
                    os.optError = o.err;
                    for (int k = 0; k < 9; k++) os.optR[k] = (double)*reinterpret_cast<const volatile float*>(&sl->pr.R[k]);
                    const float n0 = o.node[0], n1 = o.node[1], n2 = o.node[2], nw = o.node[3];
                    os.optT[0] = (double)(n0 + nw / 2); os.optT[1] = (double)(n1 + nw / 2); os.optT[2] = (double)(n2 + nw / 2);
                    for (int q = 0; q < 2; q++) {   // updateCompatibilities (:791) + ICP(R, t) (:810) at the new incumbent
                        IcpState& s = c.icp[q];
                        s.pair = os.pair; s.mode = q == 0 ? ICP_COMPAT : ICP_REFINE;
                        for (int k = 0; k < 9; k++) s.R[k] = os.optR[k];
                        for (int k = 0; k < 3; k++) { s.t[k] = os.optT[k]; s.mu_m[k] = 0.0; s.mu_d[k] = 0.0; }
                        s.err = -1.f; s.iter = 0; s.done = 0; s.status = 0; s.error = 0.f; s.incomp = 0; s.fpfh = 0.f; s.compat_pose = 0;
                    }
                    __threadfence();
                    st_vol(c.st + sidx, SL_FREE);
                    os.quiet = 0;
                    os.needLbOnly = 1; os.phase = OW_AFTER_IMPROVE; os.action = ACT_ICP;
                    return RQ_ACTION;
                }
                if (!o.ran2) { st_vol(c.st + sidx, SL_FREE); os.needLbOnly = 1; break; }     // (cannot happen: the second call is skipped only on improvement)
                os.cnt[0]++; os.cnt[1] += o.pops2; os.cnt[2] += o.subcubes2;                 // :861
                os.lastLb = o.err2;
                if (!(o.err2 >= os.optError)) {                                             // :863-871
                    RNodeD nr = child_of(os.par, os.j); nr.ub = os.ubChild; nr.lb = o.err2;
                    if (os.heapN >= A.rqCap) { os.status = GOICP_SR_OVERFLOW; finish_pair(c, 0); os.phase = OW_NONE; break; }
                    rq_push(c.rq, os.heapN, nr); note_pushed(os, nr);
                }
            } else {
                os.cnt[0]++; os.cnt[1] += o.pops; os.cnt[2] += o.subcubes;
                os.lastLb = o.err;
                if (!(o.err >= os.optError)) {
                    RNodeD nr = child_of(os.par, os.j); nr.ub = os.ubChild; nr.lb = o.err;
                    if (os.heapN >= A.rqCap) { os.status = GOICP_SR_OVERFLOW; finish_pair(c, 0); os.phase = OW_NONE; break; }
                    rq_push(c.rq, os.heapN, nr); note_pushed(os, nr);
                }
                os.needLbOnly = 0;
            }
            st_vol(c.st + sidx, SL_FREE);
            os.j++;
            break;
        }
        case OW_AFTER_IMPROVE: {   // :791-854 (the speculative calls were invalidated by the caller)
            const volatile IcpState* s0 = c.icp; const volatile IcpState* s1 = c.icp + 1;
            if (s0->status != 0 || s1->status != 0) { os.status = GOICP_SR_UNSUPPORTED; finish_pair(c, 0); os.phase = OW_NONE; break; }
            os.optComp = s0->compat_pose;                                                   // :791
            add_event(c, 2, os.optError);
            os.cnt[5]++;
            const float icpErr = s1->error;
            if (icpErr < os.optError) {                                                     // :813-840
                os.optError = icpErr;
                for (int k = 0; k < 9; k++) os.optR[k] = s1->R[k];
                for (int k = 0; k < 3; k++) os.optT[k] = s1->t[k];
                os.optComp = s1->incomp;
                add_event(c, 1, icpErr);
            }
            // :843-853: pop in order into a new queue until the first node with lb >= optError.  Pushing in pop order never sifts
            // (no parent is "less" than a later key), so the new heap array is the popped prefix itself.
            {
                const long long tp0 = clock64();
                RNodeD* tmp = c.rq + A.rqCap;   // second half of the slab
                int n = os.heapN, m = 0;
                while (n > 0) { RNodeD nd = rq_pop(c.rq, n); if (nd.lb < os.optError) { st_node(tmp + m, nd); m++; } else break; }
                for (int k = 0; k < m; k++) st_node(c.rq + k, ld_node(tmp + k));
                os.heapN = m;
                atomicAdd(&A.ctl->diag[DIAG_PRUNE_CYCLES], (unsigned long long)(clock64() - tp0));
            }
            { int g; while ((g = alloc_group(c, -1)) < 0) { os.walkStamp++; __nanosleep(200); } os.par.group = g; *reinterpret_cast<uint4*>(os.grpKey[g]) = node_key(os.par); os.grpStamp[g] = os.walkStamp + 1u; }   // the old group drains (calls of the previous incumbent)
            for (int k = 0; k < 8; k++) os.pfState[k] = SL_FREE;
            os.lastSpawnJ = os.j; os.walkLeft = 0;
            os.phase = OW_CHILD;
            return RQ_SPAWN;
        }
        default: return RQ_ACTION;   // OW_NONE: handled by the scheduler
        }
        if (os.phase == OW_NONE) { os.action = ACT_NONE; return RQ_ACTION; }
    }
}

// How many slot groups the owner should keep attached to queue nodes: none while unclaimed pairs remain (idle CTAs take pairs) unless
// the pair is already deep; afterwards the helpers are shared among the owners.  All lanes (warp-uniform result).
__device__ __forceinline__ int spec_target(Cta& c) {
    const SearchArgs& A = c.A;
    int t = 0;
    if (c.lane == 0 && A.specMax > 0) {
        // a pair that has already consumed many calls is likely one of the few deep ones that decide when the batch ends: it
        // asks for help early (CTAs look for such calls before they claim their next pair), the more the deeper it gets
        const long long calls = c.os.cnt[0];
        int manager = 0;
        // (the bar sinks as the pair list runs out: a deep pair that is claimed late has little time left to show its depth)
        const int next = ld_voli(&A.ctl->nextPair);
        const long long bar = max(16ll, (long long)A.deepCalls * max(0, A.npairs - next) / max(1, A.npairs));
        if (calls >= bar) t = (int)min((long long)A.specMax, calls / bar);
        if (next >= A.npairs) {
            const int owners = max(1, ld_voli(&A.ctl->owners));
            const int helpers = max(0, A.nCtas - owners);
            const int tasks = (helpers + owners - 1) / owners;     // calls in flight per owner that keep every helper busy
            if (tasks > 0) t = A.specMax;   // helpers outnumber what one node can feed: look as far ahead as the slots allow (a node that is popped without
                                            // results costs a whole call of latency, so the hit rate matters more than the abandoned work)
            manager = A.managerRatio > 0 && helpers >= A.managerRatio * owners;
        }
        c.os.manager = manager;
        if (A.quietRamp && next < A.npairs && c.os.quiet < 6) t = min(t, (1 << c.os.quiet) - 1);   // (helpers are scarce only while pairs are still being claimed)
    }
    return __shfl_sync(GOICP_FULL, t, 0);
}

// Publish speculative calls: the remaining children of the current node, then the children of the next queue nodes in pop order.
// All lanes of warp 0.
__device__ __forceinline__ void spawn_spec(Cta& c) {
    OwnerSh& os = c.os;
    const SearchArgs& A = c.A;
    const int target = spec_target(c);
    if (target <= 0 || os.phase != OW_CHILD) return;
    const int lane = c.lane;
    int published = 0;
    // children after the current one (the current one is the owner's own next call)
    if (lane < 8 && lane > os.j) {
        const int sidx = 8 * os.par.group + lane;
        if (st_of(ld_vol(c.st + sidx)) == SL_FREE) {
            const RNodeD ch = child_of(os.par, lane);
            float R[9];
            if (!child_rotation(A.fma != 0, ch, R)) st_vol(c.st + sidx, SL_SKIP);
            else { fill_request(c, c.slots + sidx, ch, R, false); __threadfence(); st_vol(c.st + sidx, queued_word(0u)); published++; }
        }
    }
    // The next nodes in pop order: the queue is a binary heap, so they are reached from the root through a frontier of candidate
    // positions whose keys sit in shared memory and are compared by all lanes at once.  The walk is only made when several groups
    // are missing (one walk then attaches them all).
    // (the decision and the count come from lane 0 through shuffles: lane 0 rewrites both words below, and lanes of a warp do not
    //  run in lock-step -- a lane that read them late would take the other branch and the warp-wide operations would never meet)
    int fast = 0, nNewL = 0;
    if (lane == 0) { fast = (os.walkLeft > 0 && target == os.lastTarget) ? 1 : 0; nNewL = os.nNew; }
    fast = __shfl_sync(GOICP_FULL, fast, 0);
    if (fast) {
        // fast path: the window of the last full walk still stands; only the nodes pushed since then can have entered it
        const int nNew = __shfl_sync(GOICP_FULL, nNewL, 0);
        const float winLb = os.winLb, optE = os.optError, sse = os.SSE;
        __syncwarp();
        bool ok = true;
        for (int q = 0; q < nNew && ok; q++) {
            const float lb = os.newLb[q];
            if (lb > winLb || (optE - lb) <= sse) continue;
            const uint4 key = *reinterpret_cast<const uint4*>(os.newKey[q]);
            int g = lookup_group_w(c, key);
            if (g >= 0) continue;
            if (lane == 0) g = alloc_group(c, os.par.group);
            g = __shfl_sync(GOICP_FULL, g, 0);
            if (g < 0) { ok = false; break; }   // the groups of nodes that fell out of the window are only recognised by a full walk
            if (lane == 0) { *reinterpret_cast<uint4*>(os.grpKey[g]) = key; os.grpStamp[g] = os.walkStamp; os.specGroups++; }
            if (lane < 8) {
                RNodeD nd; nd.l = (int)key.x; nd.a = __uint_as_float(key.y); nd.b = __uint_as_float(key.z); nd.c = __uint_as_float(key.w); nd.w = os.newW[q]; nd.lb = lb; nd.ub = 0.f; nd.group = -1;
                const int sidx = 8 * g + lane;
                const RNodeD ch = child_of(nd, lane);
                float R[9];
                if (!child_rotation(A.fma != 0, ch, R)) st_vol(c.st + sidx, SL_SKIP);
                else { fill_request(c, c.slots + sidx, ch, R, false); __threadfence(); st_vol(c.st + sidx, queued_word(__float_as_uint(lb) | 0x100u)); published++; }
            }
            __syncwarp();
        }
        __syncwarp();
        if (ok) {
            if (lane == 0) { os.nNew = 0; os.walkLeft--; }
            published = __reduce_add_sync(GOICP_FULL, published);
            if (lane == 0 && published) { atomicAdd(&c.hdr->nQueued, (unsigned)published); atomicOr(&A.ctl->wantHelp[c.me >> 5], 1u << (c.me & 31)); }
            __syncwarp();
            return;
        }
    }
    if (lane == 0) { os.nNew = 0; os.walkLeft = A.walkEvery - 1; os.lastTarget = target; os.winLb = 0.f; }
    __syncwarp();
    // The top of the heap (first TOPN positions: where nearly every node of the walk and its children sit) is copied to shared memory
    // with all lanes' loads in flight at once; the walk then pays one global round trip instead of two per node.
    constexpr int TOPN = 127;
    RNodeD* top = reinterpret_cast<RNodeD*>(c.scr);
    const int topN = target > 0 ? min(os.heapN, TOPN) : 0;
    for (int k = lane; k < topN; k += 32) top[k] = ld_node(c.rq + k);
    __syncwarp();
    auto node_at = [&](int pos) -> RNodeD { return pos < topN ? top[pos] : ld_node(c.rq + pos); };
    if (lane == 0) { os.walkStamp++; os.grpStamp[os.par.group] = os.walkStamp; os.specGroups = 0; os.ncand = 0; if (os.heapN > 0) { os.cand[0] = 0; os.candKey[0] = __float_as_uint(node_at(0).lb) & ~63u; os.ncand = 1; } }
    __syncwarp();
    for (int it = 0; it < target; it++) {
        const int nc = os.ncand;
        if (nc == 0) { if (lane == 0) os.winLb = 3.0e38f; break; }   // the whole queue is inside the window
        // (the order of the walk only decides which calls are made ahead of time, never a result: lb truncated to 26 bits, ties in
        //  frontier order, so that the minimum is one warp reduction)
        unsigned best = ~0u;
        for (int k = lane; k < nc; k += 32) { const unsigned key = os.candKey[k] | (unsigned)k; best = key < best ? key : best; }
        best = __reduce_min_sync(GOICP_FULL, best);
        const int k = (int)(best & 63u);
        const int pos = os.cand[k];
        __syncwarp();
        if (lane < 2) {   // the node leaves the frontier, its two heap children enter
            const int cp = 2 * pos + 1 + lane;
            unsigned key = 0; const bool have = cp < os.heapN;
            if (have) key = __float_as_uint(node_at(cp).lb) & ~63u;
            const unsigned hm = __ballot_sync(0x3u, have);
            int n2 = nc - 1;
            if (lane == 0) { os.cand[k] = os.cand[n2]; os.candKey[k] = os.candKey[n2]; }
            __syncwarp(0x3u);
            const int slot = n2 + __popc(hm & ((1u << lane) - 1u));
            if (have && slot < 62) { os.cand[slot] = cp; os.candKey[slot] = key; }
            if (lane == 0) os.ncand = min(62, n2 + __popc(hm));
        }
        __syncwarp();
        const RNodeD nd = node_at(pos);
        if ((os.optError - nd.lb) <= os.SSE) break;   // the search ends when this node is popped (:685)
        const uint4 key = node_key(nd);
        int g = lookup_group_w(c, key);
        if (g >= 0) { if (lane == 0) { os.grpStamp[g] = os.walkStamp; os.winLb = nd.lb; } __syncwarp(); continue; }   // its calls are already out
        if (lane == 0) g = alloc_group(c, os.par.group);
        g = __shfl_sync(GOICP_FULL, g, 0);
        if (g < 0) break;
        if (lane == 0) { *reinterpret_cast<uint4*>(os.grpKey[g]) = key; os.grpStamp[g] = os.walkStamp; os.specGroups++; os.winLb = nd.lb; }   // (winLb: the window reaches this far)
        if (lane < 8) {
            const int sidx = 8 * g + lane;
            const RNodeD ch = child_of(nd, lane);
            float R[9];
            if (!child_rotation(A.fma != 0, ch, R)) st_vol(c.st + sidx, SL_SKIP);
            else { fill_request(c, c.slots + sidx, ch, R, false); __threadfence(); st_vol(c.st + sidx, queued_word(__float_as_uint(nd.lb) | 0x100u)); published++; }
        }
        __syncwarp();
    }
    published = __reduce_add_sync(GOICP_FULL, published);
    if (lane == 0 && published) { atomicAdd(&c.hdr->nQueued, (unsigned)published); atomicOr(&A.ctl->wantHelp[c.me >> 5], 1u << (c.me & 31)); }
    __syncwarp();
}

// Claims an unclaimed call of owner `o`.  While pairs are still being claimed helpers are scarce and take the most urgent call (the
// smallest priority); afterwards hundreds of helpers look at the same owner at once, so each takes a different one (the r-th in slot
// order, r derived from the CTA index).  All lanes; returns the slot, -1 if nothing is queued, -2 if other helpers were faster.
__device__ int claim_from(Cta& c, int o, bool urgent) {
    unsigned* st = c.A.states + (size_t)o * SR_NSLOT;
    for (int tries = 0; tries < 3; tries++) {
        unsigned w[SR_NSLOT / 32];
#pragma unroll
        for (int q = 0; q < SR_NSLOT / 32; q++) w[q] = ld_vol(st + 32 * q + c.lane);   // one round trip: the state words are contiguous
        int s = -1; unsigned word = 0;
        if (urgent) {
            unsigned long long best = ~0ull;
#pragma unroll
            for (int q = 0; q < SR_NSLOT / 32; q++) if (st_of(w[q]) == SL_QUEUED) { const unsigned long long key = ((unsigned long long)w[q] << 16) | (unsigned)(32 * q + c.lane); best = key < best ? key : best; }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) { const unsigned long long v = __shfl_xor_sync(GOICP_FULL, best, off); best = v < best ? v : best; }
            if (best == ~0ull) return -1;
            s = (int)(best & 0xFFFFu); word = (unsigned)(best >> 16);
        } else {
            unsigned masks[SR_NSLOT / 32]; int total = 0;
#pragma unroll
            for (int q = 0; q < SR_NSLOT / 32; q++) { masks[q] = __ballot_sync(GOICP_FULL, st_of(w[q]) == SL_QUEUED); total += __popc(masks[q]); }
            if (total == 0) return -1;
            int r = (int)(((unsigned)c.me * 2654435761u + (unsigned)tries * 40503u) >> 8) % total;
#pragma unroll
            for (int q = 0; q < SR_NSLOT / 32; q++) {
                const int n = __popc(masks[q]);
                if (s < 0) { if (r < n) { unsigned m = masks[q]; for (int k = 0; k < r; k++) m &= m - 1; const int ln = __ffs(m) - 1; s = 32 * q + ln; word = __shfl_sync(GOICP_FULL, w[q], ln); } else r -= n; }
            }
        }
        int ok = 0;
        if (c.lane == 0) { ok = atomicCAS(st + s, word, (unsigned)SL_RUNNING) == word; if (ok) { atomicSub(&c.A.hdrs[o].nQueued, 1u); __threadfence(); } }
        ok = __shfl_sync(GOICP_FULL, ok, 0);
        if (ok) return s;
    }
    return -2;
}
// an owner that has published calls nobody has claimed yet (a hint bitmap: owners set their bit when they publish, a helper that
// finds nothing queued there clears it); claims one of its calls.  All lanes; returns the owner (slot in *slot) or -1.
__device__ int find_help(Cta& c, int* slot) {
    const SearchArgs& A = c.A;
    const int nw = (A.nCtas + 31) >> 5;
    bool urgent = false;
    if (c.lane == 0) urgent = ld_voli(&A.ctl->nextPair) < A.npairs;
    urgent = __shfl_sync(GOICP_FULL, urgent ? 1 : 0, 0) != 0;
    for (int tries = 0; tries < 3; tries++) {
        unsigned m = 0;
        if (c.lane < nw) m = ld_vol(&A.ctl->wantHelp[c.lane]);
        if (c.lane == (c.me >> 5)) m &= ~(1u << (c.me & 31));
        const unsigned any = __ballot_sync(GOICP_FULL, m != 0u);
        if (!any) return -1;
        // start from a word / bit that depends on the CTA so that helpers spread over the owners
        const int rot = (c.me * 5 + tries * 3) % nw;
        const unsigned anyRot = (rot == 0) ? any : ((any >> rot) | (any << (32 - rot)));
        const int wsel = (__ffs(anyRot) - 1 + rot) % 32;
        const unsigned word = __shfl_sync(GOICP_FULL, m, wsel);
        const int brot = (c.me + 7 * tries) & 31;
        const unsigned wr = (brot == 0) ? word : ((word >> brot) | (word << (32 - brot)));
        const int o = 32 * wsel + (__ffs(wr) - 1 + brot) % 32;
        const int s = claim_from(c, o, urgent);
        if (s >= 0) { *slot = s; return o; }
        if (s == -1 && c.lane == 0) atomicAnd(&A.ctl->wantHelp[o >> 5], ~(1u << (o & 31)));   // (the owner sets it again with its next call)
        __syncwarp();
    }
    return -1;
}

// warp 0: decide what the CTA does next
__device__ __forceinline__ void schedule(Cta& c) {
    OwnerSh& os = c.os;
    const SearchArgs& A = c.A;
    const int lane = c.lane;
    for (;;) {
        // ---- no pair: first see whether a deep pair asks for help, then claim the next pair ----
        if (os.pair < 0 && !os.noMorePairs) {
            if (A.specMax > 0) {
                int s = -1;
                const int o = find_help(c, &s);
                if (o >= 0) { if (lane == 0) { os.action = ACT_CALL; os.actOwner = o; os.actSlot = s; os.actCancel = 1; atomicAdd(&A.ctl->diag[DIAG_HELPER_CALLS], 1ull); } __syncwarp(); return; }
            }
            int i = 0;
            if (lane == 0) i = atomicAdd(&A.ctl->nextPair, 1);
            i = __shfl_sync(GOICP_FULL, i, 0);
            if (lane == 0) {
                if (i < A.npairs) { os.pair = i; os.phase = OW_START; os.manager = 0; st_vol(reinterpret_cast<unsigned*>(&c.hdr->pair), (unsigned)i); atomicAdd(&A.ctl->owners, 1); }
                else { os.noMorePairs = 1; unsigned long long now; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now)); atomicMax(&A.ctl->diag[DIAG_PAIRS_OUT_LAST_NS], now - A.ctl->t0ns); atomicCAS(&A.ctl->diag[DIAG_PAIRS_OUT_FIRST_NS], 0ull, now - A.ctl->t0ns); }
            }
            __syncwarp();
        }
        // ---- own pair: advance the search ----
        if (os.pair >= 0) {
            int rq = 0;
            const long long tq0 = clock64();
            // (decided by lane 0 and broadcast: lane 0 rewrites phase and j in owner_serial below, and a lane that evaluated the condition
            //  late would walk into prefetch_group's warp-wide operations alone)
            { int pf = (os.phase == OW_CHILD && os.j < 8) ? 1 : 0; pf = __shfl_sync(GOICP_FULL, pf, 0); if (pf) prefetch_group(c); }
            if (lane == 0) { rq = owner_serial(c); atomicAdd(&A.ctl->diag[DIAG_OWNER_CYCLES], (unsigned long long)(clock64() - tq0)); }
            rq = __shfl_sync(GOICP_FULL, rq, 0);
            __syncwarp();
            if (rq == RQ_AGAIN) continue;
            if (rq == RQ_SPAWN) { const long long ts0 = clock64(); spawn_spec(c); if (lane == 0) atomicAdd(&A.ctl->diag[DIAG_PUBLISH_CYCLES], (unsigned long long)(clock64() - ts0)); continue; }
            if (rq == RQ_ACTION) {
                if (os.phase == OW_AFTER_IMPROVE && os.action == ACT_ICP) invalidate_spec(c);   // the incumbent just improved
                if (os.phase == OW_NONE) {   // the pair is finished
                    if (lane == 0) { unsigned long long now; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now)); atomicAdd(&A.ctl->finishHist[min(255ull, (now - A.ctl->t0ns) / 4000000ull)], 1); }
                    invalidate_spec(c);
                    if (lane == 0) { os.pair = -1; st_vol(reinterpret_cast<unsigned*>(&c.hdr->pair), 0xFFFFFFFFu); atomicSub(&A.ctl->owners, 1); __threadfence(); atomicAdd(&A.ctl->pairsDone, 1); }
                    __syncwarp();
                    continue;
                }
                if (os.action != ACT_NONE) return;
                continue;
            }
            if (rq == RQ_WAIT) {   // manager: a helper runs the call the search waits for
                const long long tw0 = clock64();
                __nanosleep(100);
                if (lane == 0) atomicAdd(&A.ctl->diag[DIAG_OWNER_WAIT_CYCLES], (unsigned long long)(clock64() - tw0));
                continue;
            }
            // RQ_FINDWORK: the call the search waits for runs on a helper; take the next unclaimed call of this pair instead
            const int s = claim_from(c, c.me, true);
            if (s >= 0) { if (lane == 0) { os.action = ACT_CALL; os.actOwner = c.me; os.actSlot = s; os.actCancel = 1; } __syncwarp(); return; }
        }
        // ---- nothing of its own to run: help another owner ----
        const long long th0 = clock64();
        {
            int s = -1;
            const int o = find_help(c, &s);
            if (o >= 0) {
                if (lane == 0) { os.action = ACT_CALL; os.actOwner = o; os.actSlot = s; os.actCancel = 1; atomicAdd(&A.ctl->diag[DIAG_HELP_SCAN_CYCLES], (unsigned long long)(clock64() - th0)); atomicAdd(&A.ctl->diag[DIAG_HELPER_CALLS], 1ull);
                                 unsigned long long now; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now)); atomicAdd(&A.ctl->helpHist[min(255ull, (now - A.ctl->t0ns) / 4000000ull)], 1); }
                __syncwarp();
                return;
            }
        }
        // ---- idle ----
        if (os.pair < 0) {
            int done = 0;
            if (lane == 0) done = ld_voli(&A.ctl->pairsDone) >= A.npairs;
            done = __shfl_sync(GOICP_FULL, done, 0);
            if (done) { if (lane == 0) os.action = ACT_EXIT; __syncwarp(); return; }
        }
        __nanosleep(os.pair >= 0 ? 200 : 500);
        if (lane == 0) atomicAdd(&A.ctl->diag[os.pair >= 0 ? DIAG_OWNER_WAIT_CYCLES : DIAG_IDLE_CYCLES], (unsigned long long)(clock64() - th0));
        __syncwarp();
    }
}

template <bool EXACT, bool SMEM, bool GS, bool CT>
__global__ void __launch_bounds__(BNB_MAX_THREADS, GOICP_BNB_MIN_CTAS)
search_kernel(const SearchArgs A) {
    extern __shared__ float4 dyn_smem4[];
    __shared__ InnerProb s_pr;
    __shared__ InnerOut s_out;
    __shared__ unsigned long long s_gbar;
    __shared__ OwnerSh os;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float* icpTile; int icpCap = 3 * NN_TILE;   // the call staging region is idle while an ICP request runs
    if constexpr (SMEM) { icpTile = reinterpret_cast<float*>(dyn_smem4); icpCap = (int)A.gstride; } else { __shared__ __align__(16) float s_tile[3 * NN_TILE]; icpTile = s_tile; }
    CallCtx cx;
    __shared__ CancelSh s_cancel;
    __shared__ long long s_tStart, s_tIdle;
    if (tid == 0) {
        os.pair = -1; os.phase = OW_NONE; os.noMorePairs = 0; os.lastSpawnJ = -1; os.manager = 0; os.waitPolls = 0; os.walkStamp = 1u; for (int k = 0; k < 8; k++) os.pfState[k] = SL_FREE; os.specGroups = 0; os.action = ACT_NONE;
        for (int g = 0; g < SR_NGROUP; g++) os.grpUse[g] = 0;
        if (GS) mbar_init(&s_gbar, 1);
        unsigned long long now; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now)); atomicCAS(&A.ctl->t0ns, 0ull, now);
    }
    __syncthreads();
    if (tid == 0) { s_tStart = clock64(); s_tIdle = 0; }

    for (;;) {
        __syncthreads();
        if (warp == 0) {
            Cta c{A, os, A.slots + (size_t)blockIdx.x * SR_NSLOT, A.states + (size_t)blockIdx.x * SR_NSLOT, A.hdrs + blockIdx.x, reinterpret_cast<RNodeD*>(A.rq) + (size_t)blockIdx.x * 2 * A.rqCap, A.icp + 2 * (size_t)blockIdx.x, (int)blockIdx.x, lane, icpTile};
            const long long t0 = clock64(); schedule(c); if (lane == 0) s_tIdle += clock64() - t0;
        }
        __syncthreads();
        const int act = os.action;
        if (act == ACT_EXIT) break;
        if (act == ACT_ICP) {
            IcpState* icp = A.icp + 2 * (size_t)blockIdx.x;
            const long long ti0 = clock64();
            icp_fused_body(A.pairs, icp, icpTile, icpCap);
            __syncthreads();
            icp_fused_body(A.pairs, icp + 1, icpTile, icpCap);
            if (tid == 0) { atomicAdd(&A.ctr->icpRequests, 2ull); atomicAdd(&A.ctl->diag[DIAG_ICP_CYCLES], (unsigned long long)(clock64() - ti0)); }
            continue;
        }
        // ACT_CALL: one request out of slot (actOwner, actSlot)
        {
            SearchSlot* sl = A.slots + (size_t)os.actOwner * SR_NSLOT + os.actSlot;
            if (tid < (int)(sizeof(InnerProb) / 4)) reinterpret_cast<unsigned*>(&s_pr)[tid] = reinterpret_cast<const volatile unsigned*>(&sl->pr)[tid];
            if (tid == 32) { s_cancel.word = os.actCancel ? &A.hdrs[os.actOwner].gen : nullptr; s_cancel.gen = os.actCancel ? ld_vol(&sl->gen) : 0u; s_cancel.flag = 0; }
        }
        inner_call<EXACT, SMEM, GS, CT, true>(A.pairs, s_pr, s_out, s_gbar, cx, s_cancel, A.heaps, A.heapCap, A.gscratch, A.gstride, A.NdP, A.NdQ, A.useSmem, A.memo, A.memoCap, A.ctr, A.gridOff, A.S3p);
        if (warp == 0) {
            SearchSlot* sl = A.slots + (size_t)os.actOwner * SR_NSLOT + os.actSlot;
            __syncwarp();
            if (lane < 16) reinterpret_cast<volatile unsigned*>(&sl->out)[lane] = reinterpret_cast<const unsigned*>(&s_out)[lane];
            __threadfence();
            __syncwarp();
            if (lane == 0) { st_vol(A.states + (size_t)os.actOwner * SR_NSLOT + os.actSlot, SL_DONE); if (os.actCancel && s_out.status == 7) atomicAdd(&A.ctl->diag[DIAG_HELPER_ABANDONED], 1ull); }
        }
    }
    if (tid == 0) { atomicAdd(&A.ctr->idleCycles, (unsigned long long)s_tIdle); atomicAdd(&A.ctr->ctaCycles, (unsigned long long)(clock64() - s_tStart)); }
}

typedef void (*search_kernel_t)(const SearchArgs);
template <bool SMEM, bool GS>
search_kernel_t search_sel(int exact, int ct) {
    if (exact) return ct ? search_kernel<true, SMEM, GS, true> : search_kernel<true, SMEM, GS, false>;
    return ct ? search_kernel<false, SMEM, GS, true> : search_kernel<false, SMEM, GS, false>;
}
search_kernel_t search_fn(int exact, int smem, int ct) {
    if (smem == 2) return search_sel<true, true>(exact, ct);
    if (smem == 1) return search_sel<true, false>(exact, ct);
    return search_sel<false, false>(exact, ct);
}
int g_search_attr[16] = {0};
cudaError_t search_attr(int exact, int smem, int ct) {
    const int k = (exact ? 1 : 0) + 2 * smem + 8 * (ct ? 1 : 0);
    if (g_search_attr[k]) return cudaSuccess;
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, search_fn(exact, smem, ct));
    if (e != cudaSuccess) return e;
    const int maxDyn = 227 * 1024 - (int)fa.sharedSizeBytes - 1024;
    e = cudaFuncSetAttribute(search_fn(exact, smem, ct), cudaFuncAttributeMaxDynamicSharedMemorySize, maxDyn);
    if (e == cudaSuccess) g_search_attr[k] = 1;
    return e;
}

}  // namespace

size_t goicp_search_slot_bytes() { return sizeof(SearchSlot); }
size_t goicp_search_hdr_bytes() { return sizeof(OwnerHdr); }
size_t goicp_search_rnode_bytes() { return sizeof(RNodeD); }

int goicp_search_occupancy(size_t smemBytes, int exact, int threads, int useSmem, int ct) {
    if (search_attr(exact, useSmem, ct) != cudaSuccess) return 1;
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, search_fn(exact, useSmem, ct), threads, useSmem ? smemBytes : 0) != cudaSuccess || n < 1) n = 1;
    return n;
}
cudaError_t goicp_launch_search(const SearchArgs& A, int ctas, int threads, size_t smemBytes, int exact, int ct, cudaStream_t st) {
    cudaError_t e = search_attr(exact, A.useSmem & 3, ct);
    if (e != cudaSuccess) return e;
    // CTAs wait for one another (an owner for its helpers' results), so all of them must be resident at once: a cooperative launch
    // guarantees that or fails (the grid is sized from the occupancy query)
    void* args[] = {const_cast<SearchArgs*>(&A)};
    e = cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(search_fn(exact, A.useSmem & 3, ct)), dim3(ctas), dim3(threads), args, (A.useSmem & 3) ? smemBytes : 0, st);
    if (e != cudaSuccess) return e;
    return cudaGetLastError();
}
cudaError_t goicp_preload_search() {
    cudaFuncAttributes a; cudaError_t e;
    for (int exact = 0; exact < 2; exact++) for (int smem = 0; smem < 3; smem++) for (int ct = 0; ct < 2; ct++)
        if ((e = cudaFuncGetAttributes(&a, search_fn(exact, smem, ct))) != cudaSuccess) return e;
    return cudaSuccess;
}
