// GoICP::OuterBnB's bookkeeping as the host schedulers of engine_search.cu run it: the rotation queue, the child cubes, and one
// function per rule of the reference for the incumbent and the trace.  Plain C++ (no CUDA), so tests compile it with g++ alone.
#pragma once
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <algorithm>
#include <string>
#include <vector>
#include "../../include/goicp_b200.h"
#include "goicp_dev.h"

inline void tracef(std::string& s, const char* fmt, ...) {
    char buf[256]; va_list ap; va_start(ap, fmt); int n = vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    if (n > 0) s.append(buf, std::min(n, (int)sizeof buf - 1));
}

// ROTNODE (jly_goicp.h:59-73) + a unique id for the speculation cache
struct RNode { float a, b, c, w, ub, lb; int l; int id; };
inline bool rnode_less(const RNode& n1, const RNode& n2) {   // operator< :64-71
    if (n1.lb != n2.lb) return n1.lb > n2.lb;
    return n1.w < n2.w;
}
// std::priority_queue<ROTNODE> as libstdc++ implements it; spelled out so that equal keys pop in the reference's order
// independently of the standard library this file is compiled against.
inline void rheap_push(std::vector<RNode>& h, const RNode& val) {
    h.push_back(val);
    int hole = (int)h.size() - 1, parent = (hole - 1) / 2;
    while (hole > 0 && rnode_less(h[parent], val)) { h[hole] = h[parent]; hole = parent; parent = (hole - 1) / 2; }
    h[hole] = val;
}
inline RNode rheap_pop(std::vector<RNode>& h) {
    RNode top = h[0];
    const int len = (int)h.size() - 1;
    if (len > 0) {
        RNode val = h[len];
        int hole = 0, child = 0;
        while (child < (len - 1) / 2) {
            child = 2 * (child + 1);
            if (rnode_less(h[child], h[child - 1])) child--;
            h[hole] = h[child]; hole = child;
        }
        if ((len & 1) == 0 && child == (len - 2) / 2) { child = 2 * (child + 1); h[hole] = h[child - 1]; hole = child - 1; }
        int parent = (hole - 1) / 2;
        while (hole > 0 && rnode_less(h[parent], val)) { h[hole] = h[parent]; hole = parent; parent = (hole - 1) / 2; }
        h[hole] = val;
    }
    h.pop_back();
    return top;
}

// Queue pruning after an improvement (jly_goicp.cpp:843-853).  Both keep the nodes with lb < optError but leave different heaps.
// Exact order: the reference's loop (pop in order, keep the popped prefix), so later ties pop as in the reference.
inline void prune_in_pop_order(std::vector<RNode>& q, float optError) {
    std::vector<RNode> qn;
    while (!q.empty()) { RNode n = rheap_pop(q); if (n.lb < optError) rheap_push(qn, n); else break; }
    q.swap(qn);
}
// Relaxed order: filter the array and re-push; its heap decides how later ties pop, so replacing it would change relaxed results.
inline void prune_any_order(std::vector<RNode>& q, float optError) {
    std::vector<RNode> qn;
    for (const RNode& n : q) if (n.lb < optError) rheap_push(qn, n);
    q.swap(qn);
}

// rotation of a child cube (jly_goicp.cpp:716-747): false if the cube lies outside the pi-ball
inline bool child_rotation(const RNode& nr, float* R) {
    float v1 = nr.a + nr.w / 2, v2 = nr.b + nr.w / 2, v3 = nr.c + nr.w / 2;
    if ((double)sqrtf(v1 * v1 + v2 * v2 + v3 * v3) - GOICP_SQRT3 * nr.w / 2 > GOICP_PI) return false;   // :723
    float t = sqrtf(v1 * v1 + v2 * v2 + v3 * v3);                                                    // :729
    if (t > 0) {
        v1 /= t; v2 /= t; v3 /= t;
        float ct = cosf(t), ct2 = 1 - ct, st = sinf(t);
        float tmp121 = v1 * v2 * ct2, tmp122 = v3 * st, tmp131 = v1 * v3 * ct2, tmp132 = v2 * st, tmp231 = v2 * v3 * ct2, tmp232 = v1 * st;
        R[0] = ct + v1 * v1 * ct2; R[1] = tmp121 - tmp122; R[2] = tmp131 + tmp132;
        R[3] = tmp121 + tmp122; R[4] = ct + v2 * v2 * ct2; R[5] = tmp231 - tmp232;
        R[6] = tmp131 - tmp132; R[7] = tmp231 + tmp232; R[8] = ct + v3 * v3 * ct2;
    } else {
        for (int k = 0; k < 9; k++) R[k] = (k % 4 == 0) ? 1.f : 0.f;   // :759-762 copies the cloud unrotated
    }
    return true;
}
inline RNode child_of(const RNode& par, int j) {
    RNode nr{}; nr.w = par.w / 2; nr.l = par.l + 1;
    nr.a = par.a + (j & 1) * nr.w; nr.b = par.b + ((j >> 1) & 1) * nr.w; nr.c = par.c + ((j >> 2) & 1) * nr.w;   // :710-712
    return nr;
}

// What GoICP::Register leaves behind for one pair (GoICP::Initialize :240-241 resets optR / optT).
struct SearchResult {
    float optError = 0; double optR[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, optT[3] = {0, 0, 0}; int optComp = 0;
    long long cnt[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // goicp_result.counters
    std::string trace;
};

enum TraceKind { TRACE_INIT = 0, TRACE_ICP = 1, TRACE_BNB = 2 };   // also PairOut.ev[].kind
inline void trace_event(std::string& s, int kind, float err) {
    static const char* kinds[3] = {"Init", "ICP", "BNB"};
    tracef(s, "Error*: %g (%s)\n", err, kinds[kind % 3]);
}
// the end of OuterBnB: queue empty (:670-677) or the certificate optError - lb <= SSEThresh (:685)
inline void trace_end(std::string& s, bool queueEmpty, float optError, float lb, float sse) {
    if (queueEmpty) tracef(s, "Rotation Queue Empty\nError*: %g, LB: %g\n", optError, lb);
    else tracef(s, "Threshold reached\nError*: %g, LB: %g, epsilon: %g\n", optError, lb, sse);
}

// the initial error at the identity plus the regularisation terms (:601-627)
inline void init_incumbent(SearchResult& r, float initErr, const goicp_params& p, int Nd) {
    r.optError = initErr;
    if (p.regularization > 0) r.optError += p.regularization * (Nd * Nd);                      // :623
    if (p.regularizationFPFH > 0) r.optError += p.regularizationFPFH * (100 * 8 * 100 * 8);    // :624
    if (p.regularizationNeighbors > 0) r.optError += p.regularizationNeighbors * (Nd * 6 * Nd * 6);
    trace_event(r.trace, TRACE_INIT, r.optError);
    r.cnt[5]++;
}
// an InnerBnB upper bound below the incumbent: the cube's rotation and the centre of the best translation node (:771-790)
inline void take_bnb(SearchResult& r, float err, const float* R, const float* tnode) {
    r.optError = err;
    for (int k = 0; k < 9; k++) r.optR[k] = R[k];
    r.optT[0] = tnode[0] + tnode[3] / 2; r.optT[1] = tnode[1] + tnode[3] / 2; r.optT[2] = tnode[2] + tnode[3] / 2;   // float expr -> double
}
// the result of ICP(R, t) with its re-score (jly_goicp.cpp:102-175) replaces the incumbent if it is lower (:636-661, :813-840)
inline void take_icp(SearchResult& r, const IcpState& icp) {
    if (!(icp.error < r.optError)) return;
    r.optError = icp.error;
    memcpy(r.optR, icp.R, sizeof r.optR); memcpy(r.optT, icp.t, sizeof r.optT);
    r.optComp = icp.incomp;
    trace_event(r.trace, TRACE_ICP, icp.error);
}
// after an improvement: the compatibility count at the new pose (:791), the BnB's trace line, then ICP(R, t) (:813-840)
inline void after_bnb(SearchResult& r, const IcpState& compat, const IcpState& icp) {
    r.optComp = compat.compat_pose;
    trace_event(r.trace, TRACE_BNB, r.optError);
    r.cnt[5]++;
    take_icp(r, icp);
}
