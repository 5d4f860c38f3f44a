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

enum TraceKind { TRACE_INIT = 0, TRACE_ICP = 1, TRACE_BNB = 2 };   // also PairOut.ev[].kind
// How OuterBnB ended (also PairOut.endKind and goicp_get_search_ends): the queue ran empty (:670-677), the certificate
// optError - lb <= SSEThresh held at a pop (:685), or a pop that :685 did not end had lb >= the pair's error cutoff.  Best-first
// order makes lb a lower bound on every alignment not yet ruled out, and the ruled-out ones lie above the incumbent, so the
// optimum is >= lb >= cutoff: the pair is certified above the cutoff.
enum SearchEnd { END_QUEUE_EMPTY = 1, END_THRESHOLD = 2, END_CUTOFF = 3 };

// The "Error*:" trace OuterBnB prints (jly_goicp.cpp:627-839, :670-685), kept as the values it is printed from: the improvement
// events in order and the end record.  A batch records every pair's trace but reads at most one, so the text is only built by
// str() / c_str(), when it is read.
struct TraceEvent { int kind; float v; };   // TraceKind, the new incumbent
struct Trace {
    std::vector<TraceEvent> events;
    int endKind = 0; float endErr = 0, endLb = 0, endSse = 0, endCutoff = 0;   // SearchEnd (0: no end line yet) and what it prints
    mutable std::string text;   // the last str()
    const std::string& str() const {
        static const char* kinds[3] = {"Init", "ICP", "BNB"};
        text.clear();
        for (const TraceEvent& e : events) tracef(text, "Error*: %g (%s)\n", e.v, kinds[e.kind % 3]);
        if (endKind == END_QUEUE_EMPTY) tracef(text, "Rotation Queue Empty\nError*: %g, LB: %g\n", endErr, endLb);
        else if (endKind == END_THRESHOLD) tracef(text, "Threshold reached\nError*: %g, LB: %g, epsilon: %g\n", endErr, endLb, endSse);
        else if (endKind != 0) tracef(text, "Cutoff reached\nError*: %g, LB: %g, cutoff: %g\n", endErr, endLb, endCutoff);
        return text;
    }
    const char* c_str() const { return str().c_str(); }
};

// What GoICP::Register leaves behind for one pair (GoICP::Initialize :240-241 resets optR / optT).
struct SearchResult {
    float optError = 0; double optR[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, optT[3] = {0, 0, 0}; int optComp = 0;
    long long cnt[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // goicp_result.counters
    Trace trace;
    int endKind = 0; float endLb = 0;   // how the search ended (SearchEnd; 0: it has not run) and the lower bound of its end line
};

inline void trace_event(Trace& t, int kind, float err) { t.events.push_back(TraceEvent{kind, err}); }
inline void trace_end(SearchResult& r, int kind, float lb, float sse, float cutoff) {
    r.endKind = kind; r.endLb = lb;
    Trace& t = r.trace;
    t.endKind = kind; t.endErr = r.optError; t.endLb = lb; t.endSse = sse; t.endCutoff = cutoff;
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
