// Host engine, part 2: GoICP::Register.  Three schedulers:
//  * device-resident (k_search.cu): the whole batch -- OuterBnB, every InnerBnB call, every ICP -- in one cooperative launch;
//    the host uploads, launches, and reads one result record per pair;
//  * wave scheduler: GoICP::OuterBnB (jly_goicp.cpp:582-876) as a host priority queue that follows the reference's pop order
//    exactly, InnerBnB calls launched in waves (one CTA per call, k_bnb.cu) with the calls the reference would make next
//    evaluated speculatively; used for large clouds (multi-kernel ICP), frontier sharding and re-runs with growing queue slabs;
//  * relaxed-order waves (goicp_set_search_mode): many rotation nodes per wave, the reference's certificate, not its order.
// The incumbent and trace rules all three share are in host_search.h.
#include "engine_internal.h"

// ---- one launch of InnerBnB calls (handles heap overflow by re-running the overflowed calls with larger heaps) -------
static goicp_status run_inner_local(Eng* h, WaveCtx& c, const BnbCfg& cfg, std::vector<InnerProb>& reqs, std::vector<InnerOut>& outs) {
    const int n = (int)reqs.size();
    outs.resize(n);
    if (n == 0) return GOICP_OK;
    int maxCtas = h->numSM * cfg.perSM;
    if (c.ctaCap > 0) maxCtas = std::min(maxCtas, c.ctaCap);
    int heapCap = c.heapCap;
    CU(c.mProbs.ensure(sizeof(InnerProb) * (size_t)n));
    CU(c.mOuts.ensure(sizeof(InnerOut) * (size_t)n));
    if (!c.counterReady) { CU(c.dCounter.ensure(2 * sizeof(int))); CU(cudaMemsetAsync(c.dCounter.p, 0, 2 * sizeof(int), c.stream)); c.counterReady = true; }
    std::vector<int> todo(n); for (int i = 0; i < n; i++) todo[i] = i;
    for (int attempt = 0; attempt < 12 && !todo.empty(); attempt++) {
        const int m = (int)todo.size();
        InnerProb* hp = reinterpret_cast<InnerProb*>(c.mProbs.h);
        for (int i = 0; i < m; i++) hp[i] = reqs[todo[i]];
        const int ctas = std::min(m, maxCtas);
        CU(c.dHeaps.ensure(sizeof(HeapEnt) * (size_t)ctas * heapCap));
        if (!cfg.useSmem) CU(c.dBnbScratch.ensure(sizeof(float) * cfg.smemFloats * (size_t)ctas));
        const int memoCap = 4096;
        if (c.dMemo.cap < (size_t)32 * memoCap * ctas) { CU(c.dMemo.ensure((size_t)32 * memoCap * ctas)); CU(cudaMemsetAsync(c.dMemo.p, 0, c.dMemo.cap, c.stream)); }
        auto tq = clk::now();
        cudaEventRecord(c.ev0, c.stream);
        int launched = 0;
        CU(goicp_launch_inner_bnb(h->dPairs.as<PairDev>(), reinterpret_cast<const InnerProb*>(c.mProbs.d), reinterpret_cast<InnerOut*>(c.mOuts.d), m, c.dCounter.as<int>(),
                                  c.dHeaps.as<HeapEnt>(), heapCap, ctas, c.dBnbScratch.as<float>(), cfg.smemFloats, cfg.NdP, cfg.NdQ, cfg.smemBytes, cfg.useSmem, cfg.gridOff, cfg.S3p,
                                  h->exact_sums, cfg.ct, cfg.threads, c.dMemo.p, memoCap, h->devCounters.as<DevCounters>(), c.stream, &launched));
        cudaEventRecord(c.ev1, c.stream);
        c.tInnerEnq += secs_since(tq); tq = clk::now();
        CU(c.sync());
        c.tInnerWait += secs_since(tq);
        float ms = 0; cudaEventElapsedTime(&ms, c.ev0, c.ev1); c.ms[2] += ms; c.launches[2] += 1;
        const InnerOut* ho = reinterpret_cast<const InnerOut*>(c.mOuts.h);
        std::vector<int> again;
        for (int i = 0; i < m; i++) {
            if (ho[i].status == 4) again.push_back(todo[i]);   // the translation queue outgrew its slab: re-run with a larger one
            else if (ho[i].status != 0) return fail(h, GOICP_ERR_CUDA, "InnerBnB call %d of pair %d ended with internal status %d", todo[i], reqs[todo[i]].pair, ho[i].status);
            else outs[todo[i]] = ho[i];
        }
        todo.swap(again);
        if (!todo.empty()) { heapCap *= 4; const size_t fit = ((size_t)4 << 30) / sizeof(HeapEnt) / (size_t)heapCap; maxCtas = (int)std::max<size_t>(1, std::min<size_t>((size_t)maxCtas, fit)); }
    }
    if (!todo.empty()) return fail(h, GOICP_ERR_OVERFLOW, "translation queue exceeded %d entries", heapCap);
    c.callsLaunched += n;
    return GOICP_OK;
}
// One wave of InnerBnB calls.  With frontier sharding the calls are dealt round-robin to the ranks, evaluated locally and
// exchanged with one all-gather, so every rank continues with the complete, identical result set.
goicp_status run_inner(Eng* h, WaveCtx& c, const BnbCfg& cfg, std::vector<InnerProb>& reqs, std::vector<InnerOut>& outs) {
    const int n = (int)reqs.size();
    if (h->shardN <= 1 || !h->allgather) return run_inner_local(h, c, cfg, reqs, outs);
    outs.resize(n);
    const int N = h->shardN, r = h->shardRank, per = (n + N - 1) / N;
    std::vector<InnerProb> mine; std::vector<InnerOut> mineOut;
    for (int k = r; k < n; k += N) mine.push_back(reqs[k]);
    goicp_status s = run_inner_local(h, c, cfg, mine, mineOut);
    if (s) return s;
    h->xSend.assign(std::max(per, 1), InnerOut{}); h->xRecv.assign((size_t)std::max(per, 1) * N, InnerOut{});
    for (size_t k = 0; k < mineOut.size(); k++) h->xSend[k] = mineOut[k];
    if (h->allgather(h->xSend.data(), h->xRecv.data(), (int64_t)sizeof(InnerOut) * std::max(per, 1), h->allgatherUser) != 0)
        return fail(h, GOICP_ERR_ARG, "frontier sharding: the all-gather callback failed");
    for (int k = 0; k < n; k++) outs[k] = h->xRecv[(size_t)(k % N) * std::max(per, 1) + k / N];
    return GOICP_OK;
}

// ---- ICP / scoring pipeline for a set of states ----------------------------------------------------------------------
goicp_status run_icp(Eng* h, WaveCtx& c, std::vector<IcpState>& states) {
    const int n = (int)states.size();
    if (n == 0) return GOICP_OK;
    int maxNd = 1, maxNm = 1; bool anyIcp = false; bool small = true;
    for (auto& s : states) {
        const Problem& P = h->probs[s.pair]; maxNd = std::max(maxNd, P.Nd); maxNm = std::max(maxNm, P.Nm); anyIcp |= s.mode == ICP_REFINE;
        if ((size_t)P.Nd * P.Nm > ((size_t)1 << 21) || (P.dev.doTrim && P.Nd > 2048)) small = false;
    }
    CU(c.mIcp.ensure(sizeof(IcpState) * n));   // small: the fused kernel works in this mapped host memory; otherwise it stages a device copy
    if (!small) CU(c.dIcp.ensure(sizeof(IcpState) * n));
    IcpState* hs = reinterpret_cast<IcpState*>(c.mIcp.h);
    for (int i = 0; i < n; i++) hs[i] = states[i];
    cudaEventRecord(c.ev0, c.stream);
    int nl = 0;
    if (small) {   // whole ICP (begin, every iteration, re-score) in one launch, one CTA per request
        CU(goicp_launch_icp_fused(h->dPairs.as<PairDev>(), reinterpret_cast<IcpState*>(c.mIcp.d), n, c.stream)); nl++;
    } else {
        CU(cudaMemcpyAsync(c.dIcp.p, hs, sizeof(IcpState) * n, cudaMemcpyHostToDevice, c.stream));
        CU(goicp_launch_icp_begin(h->dPairs.as<PairDev>(), c.dIcp.as<IcpState>(), n, c.stream)); nl++;
        if (anyIcp) {
            int burst = 4;
            for (int it = 0; it < 10000;) {
                for (int b = 0; b < burst; b++) { CU(goicp_launch_icp_iter(h->dPairs.as<PairDev>(), c.dIcp.as<IcpState>(), n, maxNd, maxNm, h->numSM, c.stream)); nl += 2; }
                it += burst;
                CU(cudaMemcpyAsync(hs, c.dIcp.p, sizeof(IcpState) * n, cudaMemcpyDeviceToHost, c.stream));
                CU(c.sync());
                bool all = true;
                for (int i = 0; i < n; i++) if (hs[i].mode == ICP_REFINE && !hs[i].done) all = false;
                if (all) break;
                if (burst < 16) burst *= 2;
            }
        }
        CU(goicp_launch_icp_score(h->dPairs.as<PairDev>(), c.dIcp.as<IcpState>(), n, c.stream)); nl++;
    }
    cudaEventRecord(c.ev1, c.stream);
    if (!small) CU(cudaMemcpyAsync(hs, c.dIcp.p, sizeof(IcpState) * n, cudaMemcpyDeviceToHost, c.stream));
    CU(c.sync());
    float ms = 0; cudaEventElapsedTime(&ms, c.ev0, c.ev1); c.ms[3] += ms; c.launches[3] += nl;
    for (int i = 0; i < n; i++) states[i] = hs[i];
    for (int i = 0; i < n; i++) if (states[i].status != 0) return fail(h, GOICP_ERR_ARG, "trimmed ICP without its sort workspace (trimFraction changed after the clouds were set?)");
    return GOICP_OK;
}

IcpState make_icp_state(int pair, IcpMode mode, const double* R, const double* t) {
    IcpState s; memset(&s, 0, sizeof s);
    s.pair = pair; s.mode = mode;
    memcpy(s.R, R, sizeof s.R); memcpy(s.t, t, sizeof s.t);
    s.err = -1.f;
    return s;
}

static inline unsigned long long call_key(int nodeId, int j, int kind) { return ((unsigned long long)(unsigned)nodeId << 4) | (unsigned)(j << 1) | (unsigned)kind; }

struct CallRes { float entryOpt; InnerOut out; };

enum Phase { PH_WAIT_INIT, PH_POP, PH_CHILD_UB, PH_WAIT_ICP, PH_CHILD_LB, PH_DONE };

// A host scheduler's state of one pair's OuterBnB while it runs; the incumbent and the counters are the pair's Problem::res.
struct HostSearch {
    int pair;
    Phase phase = PH_WAIT_INIT;
    std::vector<RNode> q;
    RNode par{}, child{}; int j = 0; float R[9]; float ubChild = 0; float lastLb = 0;
    std::unordered_map<unsigned long long, CallRes> cache;   // InnerBnB results by call_key, valid under the incumbent `entryOpt`
    int nextId = 1, quiet = 0;
};

struct ReqTag { int search; unsigned long long key; float entryOpt; };   // search: index into register_group's `active`

// the two ICP requests that start a search (error at the identity, ICP from it) or follow an improvement (compatibility count, ICP)
static void push_icps(std::vector<IcpState>& icps, int pair, IcpMode first, const SearchResult& r) {
    icps.push_back(make_icp_state(pair, first, r.optR, r.optT)); icps.push_back(make_icp_state(pair, ICP_REFINE, r.optR, r.optT));
}
// initial error, first ICP and the root node (:601-664)
static void start_search(Eng* h, HostSearch& S, const IcpState& init, const IcpState& icp) {
    const goicp_params& p = h->params;
    Problem& P = h->probs[S.pair];
    init_incumbent(P.res, init.error, p, P.Nd);
    take_icp(P.res, icp);
    RNode root{}; root.a = p.rotMinX; root.b = p.rotMinY; root.c = p.rotMinZ; root.w = p.rotWidth; root.l = 0; root.lb = 0; root.id = 0;
    rheap_push(S.q, root);
    S.phase = PH_POP;
}

// Advance one pair's OuterBnB as far as cached results allow; on return S.phase tells what it waits for.
static void advance(Eng* h, HostSearch& S) {
    SearchResult& r = h->probs[S.pair].res;
    const float SSE = h->probs[S.pair].dev.SSEThresh, cutoff = h->probs[S.pair].cutoff;
    for (;;) {
        switch (S.phase) {
        case PH_WAIT_INIT: case PH_WAIT_ICP: case PH_DONE: return;
        case PH_POP: {
            if (S.q.empty()) { trace_end(r, END_QUEUE_EMPTY, S.lastLb, SSE, cutoff); S.phase = PH_DONE; return; }   // :670-677
            S.par = rheap_pop(S.q); r.cnt[3]++;
            if ((r.optError - S.par.lb) <= SSE) { trace_end(r, END_THRESHOLD, S.par.lb, SSE, cutoff); S.phase = PH_DONE; return; }   // :685
            if (S.par.lb >= cutoff) { trace_end(r, END_CUTOFF, S.par.lb, SSE, cutoff); S.phase = PH_DONE; return; }
            S.j = 0; S.phase = PH_CHILD_UB;
            break;
        }
        case PH_CHILD_UB: {
            if (S.j >= 8) { S.phase = PH_POP; break; }
            S.child = child_of(S.par, S.j);
            if (!child_rotation(S.child, S.R)) { S.j++; break; }
            auto it = S.cache.find(call_key(S.par.id, S.j, 0));
            if (it == S.cache.end() || it->second.entryOpt != r.optError) return;   // blocked
            const InnerOut c = it->second.out; S.cache.erase(it);
            r.cnt[4]++; r.cnt[0]++; r.cnt[1] += c.pops; r.cnt[2] += c.subcubes;
            S.ubChild = c.err;
            if (c.err < r.optError) {   // :771-790, then updateCompatibilities + ICP at the new incumbent
                take_bnb(r, c.err, S.R, c.node);
                S.cache.clear(); S.quiet = 0;
                S.phase = PH_WAIT_ICP;
                return;
            }
            S.phase = PH_CHILD_LB;
            break;
        }
        case PH_CHILD_LB: {
            auto it = S.cache.find(call_key(S.par.id, S.j, 1));
            if (it == S.cache.end() || it->second.entryOpt != r.optError) return;   // blocked
            const InnerOut c = it->second.out; S.cache.erase(it);
            r.cnt[0]++; r.cnt[1] += c.pops; r.cnt[2] += c.subcubes;
            S.lastLb = c.err;
            if (!(c.err >= r.optError)) {   // :863-871
                RNode nr = S.child; nr.ub = S.ubChild; nr.lb = c.err; nr.id = S.nextId++;
                rheap_push(S.q, nr);
            }
            S.j++; S.phase = PH_CHILD_UB;
            break;
        }
        }
    }
}

// Requests of one blocked pair: the blocking call first, then speculation in the reference's expected order.
static void gather_requests(Eng* h, HostSearch& S, int search, std::vector<InnerProb>& reqs, std::vector<ReqTag>& tags) {
    const Problem& P = h->probs[S.pair];
    const float SSE = P.dev.SSEThresh, optError = P.res.optError, cutoff = P.cutoff;
    std::unordered_set<unsigned long long> seen;
    // a call that is cached under the current incumbent or already in flight needs no request (and no rotation matrix)
    auto known = [&](const RNode& par, int j, int kind) {
        auto it = S.cache.find(call_key(par.id, j, kind));
        return it != S.cache.end() && it->second.entryOpt == optError;
    };
    auto want = [&](const RNode& par, int j, int kind, const RNode& ch, const float* R) {
        const unsigned long long key = call_key(par.id, j, kind);
        if (known(par, j, kind) || !seen.insert(key).second) return;
        // Q2: the reference indexes maxRotDis[level] without a bound check (undefined beyond level 19); we clamp.
        const int lbLevel = std::min(ch.l, GOICP_MAXROTLEVEL - 1);
        InnerProb ip; ip.pair = S.pair; ip.level = kind ? lbLevel : -1; ip.optError = optError;
        memcpy(ip.R, R, sizeof ip.R);
        reqs.push_back(ip); tags.push_back(ReqTag{search, key, optError});
    };
    auto want_children = [&](const RNode& nd, int j0, bool skipUb0) {   // both calls of children j0..7 (no upper bound of j0 if skipUb0)
        for (int j = j0; j < 8; j++) {
            const bool skipUb = skipUb0 && j == j0;
            if ((skipUb || known(nd, j, 0)) && known(nd, j, 1)) continue;
            RNode ch = child_of(nd, j); float R[9];
            if (!child_rotation(ch, R)) continue;
            if (!skipUb) want(nd, j, 0, ch, R);
            want(nd, j, 1, ch, R);
        }
    };
    want_children(S.par, S.j, S.phase == PH_CHILD_LB);   // current parent, from the blocking call on
    // the next queue nodes in pop order; width grows while the incumbent stays unchanged
    // inside a batch the pairs themselves fill the GPU
    const int specw = h->probs.size() > 1 ? std::min(h->spec_width, h->batch_spec_width) : h->spec_width;
    int width = std::min(specw, S.quiet < 30 ? (1 << std::min(S.quiet, 20)) - 1 : specw);
    if (width > 0 && !S.q.empty()) {
        // the `width` best nodes of the rotation queue: S.q is a binary heap, so they are reached from the root through a
        // frontier of candidate positions (no copy, no sort of the whole queue)
        const int n = (int)S.q.size(), k = std::min(width, n);
        int cand[80]; int nc = 0; cand[nc++] = 0;
        for (int i = 0; i < k && nc > 0; i++) {
            int b = 0;
            for (int c = 1; c < nc; c++) if (rnode_less(S.q[cand[b]], S.q[cand[c]])) b = c;
            const int pos = cand[b]; cand[b] = cand[--nc];
            if (2 * pos + 1 < n && nc < 78) cand[nc++] = 2 * pos + 1;
            if (2 * pos + 2 < n && nc < 78) cand[nc++] = 2 * pos + 2;
            const RNode& nd = S.q[pos];
            if ((optError - nd.lb) <= SSE || nd.lb >= cutoff) break;   // the search ends when this node is popped
            want_children(nd, 0, false);
        }
    }
    S.quiet++;
}

// a search's two ICP requests have returned: start of OuterBnB (:601-664) or post-improvement (:791-854)
static void after_icp(Eng* h, HostSearch& S, const IcpState& first, const IcpState& icp) {
    if (S.phase == PH_WAIT_INIT) return start_search(h, S, first, icp);
    SearchResult& r = h->probs[S.pair].res;
    after_bnb(r, first, icp);
    prune_in_pop_order(S.q, r.optError);
    S.cache.clear();
    S.phase = PH_CHILD_LB;
}

// One stream of lock-step waves over up to `slots` pairs at a time; finished pairs are replaced from the shared
// counter `next` (so a deep pair never stalls more than its own stream).  GoICP::OuterBnB (jly_goicp.cpp:582) per pair.
static goicp_status register_group(Eng* h, WaveCtx& c, const BnbCfg& cfg, std::atomic<int>& next, int slots, const std::vector<int>* subset = nullptr) {
    const int np = subset ? (int)subset->size() : (int)h->probs.size();
    std::vector<HostSearch> active;
    std::vector<InnerProb> reqs; std::vector<ReqTag> tags; std::vector<InnerOut> outs; std::vector<IcpState> icps; std::vector<int> icpOwner;   // one owner per two requests
    goicp_status s;
    auto tl = clk::now();
    for (;;) {
        active.erase(std::remove_if(active.begin(), active.end(), [](const HostSearch& S) { return S.phase == PH_DONE; }), active.end());
        reqs.clear(); tags.clear(); icps.clear(); icpOwner.clear();
        while ((int)active.size() < slots) {   // initial error (:601-627) and ICP from the identity (:634)
            const int k = next.fetch_add(1); if (k >= np) break;
            const int i = subset ? (*subset)[k] : k;
            h->probs[i].res = SearchResult(); active.push_back(HostSearch{i});
            push_icps(icps, i, ICP_INIT_ERROR, h->probs[i].res); icpOwner.push_back((int)active.size() - 1);
        }
        if (active.empty()) break;
        for (int a = 0; a < (int)active.size(); a++) {
            HostSearch& S = active[a];
            advance(h, S);
            if (S.phase == PH_WAIT_ICP) { push_icps(icps, S.pair, ICP_COMPAT, h->probs[S.pair].res); icpOwner.push_back(a); }   // :791, :810
            else if (S.phase != PH_DONE && S.phase != PH_WAIT_INIT) gather_requests(h, S, a, reqs, tags);
        }
        if (reqs.empty() && icps.empty()) continue;
        c.waves++;
        c.tLogic += secs_since(tl);
        if ((s = run_inner(h, c, cfg, reqs, outs))) return s;
        if ((s = run_icp(h, c, icps))) return s;
        tl = clk::now();
        for (size_t k = 0; k < tags.size(); k++) active[tags[k].search].cache[tags[k].key] = CallRes{tags[k].entryOpt, outs[k]};
        for (size_t k = 0; k < icpOwner.size(); k++) after_icp(h, active[icpOwner[k]], icps[2 * k], icps[2 * k + 1]);
    }
    return GOICP_OK;
}

// ---- relaxed-order wave search of ONE registration (north_star (b): "the host priority queue expands frontier waves"; SURVEY H4) ----
// The exact-order schedulers reproduce the reference's visitation order, so a single deep registration advances one rotation node at
// a time along its dependency chain.  Here every wave pops the `wave_nodes` best rotation nodes at once, evaluates ALL their children
// (upper- and lower-bound InnerBnB call of each cube as one request) in one launch under the incumbent error of the wave's start,
// and then applies the results together: the best improving upper bound becomes the incumbent (followed by updateCompatibilities +
// ICP as in jly_goicp.cpp:791-840 and the queue pruning of :843-853), children whose lower bound stays below it are pushed.  Node
// visitation order differs from the reference; the certificate is the reference's own: the search ends when the queue is empty or
// optError - (smallest lower bound in the queue) <= SSEThresh (:685).  With frontier sharding (goicp_set_frontier_sharding) the
// requests of a wave are dealt to the ranks and their results exchanged once per wave (run_inner), so every rank applies the same
// results and holds the same queue and incumbent: the minimum over the wave's upper bounds is the per-wave "allreduce(min)".
// An error cutoff is checked once per wave, before its pops, and only when no lower-bound call is carried over: a carried cube is
// in no queue, so the queue's front bounds the optimum only once every cube of the domain is either queued or discarded.
static goicp_status register_relaxed(Eng* h, WaveCtx& c, const BnbCfg& cfg, int pi) {
    Problem& P = h->probs[pi];
    SearchResult& r = P.res = SearchResult();
    HostSearch S{pi};
    goicp_status s;
    std::vector<IcpState> icps;
    push_icps(icps, pi, ICP_INIT_ERROR, r);
    if ((s = run_icp(h, c, icps))) return s;
    start_search(h, S, icps[0], icps[1]);
    const float SSE = P.dev.SSEThresh, cutoff = P.cutoff;
    struct Item { RNode node; float R[9]; bool lbOnly; float ub; };
    std::vector<Item> items, carry;   // carry: cubes whose upper bound improved the incumbent of their wave: their lower-bound call is still due (:856-861)
    std::vector<InnerProb> reqs; std::vector<InnerOut> outs;
    const int W = std::max(1, h->wave_nodes);
    for (;;) {
        items.clear(); items.swap(carry);
        if (items.empty() && !S.q.empty() && (r.optError - S.q.front().lb) > SSE && S.q.front().lb >= cutoff) {
            trace_end(r, END_CUTOFF, S.q.front().lb, SSE, cutoff);
            r.cnt[3]++;   // the pop that meets the cutoff counts, as in the exact order
            break;
        }
        int popped = 0;
        while (!S.q.empty() && popped < W && (r.optError - S.q.front().lb) > SSE) {
            const RNode par = rheap_pop(S.q); r.cnt[3]++; popped++;
            for (int j = 0; j < 8; j++) {
                Item it{child_of(par, j), {}, false, 0.f};
                if (child_rotation(it.node, it.R)) items.push_back(it);
            }
        }
        if (items.empty()) {
            const bool empty = S.q.empty();
            trace_end(r, empty ? END_QUEUE_EMPTY : END_THRESHOLD, empty ? S.lastLb : S.q.front().lb, SSE, cutoff);
            if (!empty) r.cnt[3]++;   // the pop that meets the certificate counts, as in the exact order
            break;
        }
        reqs.resize(items.size());
        for (size_t k = 0; k < items.size(); k++) {
            const int lbLevel = std::min(items[k].node.l, GOICP_MAXROTLEVEL - 1);
            reqs[k].pair = pi; reqs[k].level = items[k].lbOnly ? lbLevel : GOICP_REQ_BOTH + lbLevel; reqs[k].optError = r.optError;
            memcpy(reqs[k].R, items[k].R, sizeof reqs[k].R);
        }
        c.waves++;
        if ((s = run_inner(h, c, cfg, reqs, outs))) return s;
        int best = -1;
        for (size_t k = 0; k < items.size(); k++) {
            const InnerOut& o = outs[k];
            r.cnt[0]++; r.cnt[1] += o.pops; r.cnt[2] += o.subcubes;
            if (items[k].lbOnly) continue;
            r.cnt[4]++;
            items[k].ub = o.err;
            if (o.err < r.optError && (best < 0 || o.err < outs[best].err)) best = (int)k;
        }
        if (best >= 0) {   // :771-840 for the wave's best cube
            take_bnb(r, outs[best].err, items[best].R, outs[best].node);
            icps.clear();
            push_icps(icps, pi, ICP_COMPAT, r);
            if ((s = run_icp(h, c, icps))) return s;
            after_bnb(r, icps[0], icps[1]);
        }
        for (size_t k = 0; k < items.size(); k++) {   // lower bounds (:856-871)
            const InnerOut& o = outs[k];
            float lb;
            if (items[k].lbOnly) lb = o.err;
            else if (o.ran2) { r.cnt[0]++; r.cnt[1] += o.pops2; r.cnt[2] += o.subcubes2; lb = o.err2; }
            else { Item it = items[k]; it.lbOnly = true; carry.push_back(it); continue; }   // its upper bound improved on the wave's incumbent: lower bound in the next wave
            S.lastLb = lb;
            if (!(lb >= r.optError)) { RNode nr = items[k].node; nr.ub = items[k].ub; nr.lb = lb; nr.id = S.nextId++; rheap_push(S.q, nr); }
        }
        if (best >= 0) prune_any_order(S.q, r.optError);   // :843-853
    }
    return GOICP_OK;
}

// ---- device-resident search (k_search.cu): the whole batch in one launch, results read back once --------------------------------
static bool host_libm_uses_fma() {   // glibc's ifunc rule for sinf / cosf on x86-64 (sysdeps/x86_64/fpu/multiarch/ifunc-fma.h)
#if defined(__x86_64__)
    __builtin_cpu_init();
    return __builtin_cpu_supports("fma") && __builtin_cpu_supports("avx2");
#else
    return true;
#endif
}
// GOICP_DEBUG=1: where the device-resident search spent its CTA cycles (SearchCtl, DevCounters) and which pairs ended last
static void print_search_debug(Eng* h, int ctas, const DevCounters& dc, const PairOut* outs, int np) {
    SearchCtl ctl; cudaMemcpy(&ctl, h->sCtl.p, sizeof ctl, cudaMemcpyDeviceToHost);
    const unsigned long long* d = ctl.diag;
    fprintf(stderr, "[search] CTA cycles: OuterBnB state machine %.3g, publishing %.3g, help scan %.3g, idle (no pair) %.3g, owner waiting %.3g, ICP(2nd) %.3g; helper calls %llu (abandoned %llu); pair counter ran out at %.1f..%.1f ms\n",
            (double)d[DIAG_OWNER_CYCLES], (double)d[DIAG_PUBLISH_CYCLES], (double)d[DIAG_HELP_SCAN_CYCLES], (double)d[DIAG_IDLE_CYCLES], (double)d[DIAG_OWNER_WAIT_CYCLES], (double)d[DIAG_ICP_CYCLES], d[DIAG_HELPER_CALLS], d[DIAG_HELPER_ABANDONED], d[DIAG_PAIRS_OUT_FIRST_NS] * 1e-6, d[DIAG_PAIRS_OUT_LAST_NS] * 1e-6);
    fprintf(stderr, "[search] CTA cycles: queue pruning after improvements %.3g, rotation-queue pops %.3g; rotation nodes popped with calls made ahead %llu / without %llu; children whose result was there when the search reached them %llu / waited for %llu\n", (double)d[DIAG_PRUNE_CYCLES], (double)d[DIAG_POP_CYCLES], d[DIAG_POPS_AHEAD], d[DIAG_POPS_NOT_AHEAD], d[DIAG_CHILD_READY], d[DIAG_CHILD_WAITED]);
    std::vector<int> idx(np); for (int i = 0; i < np; i++) idx[i] = i;
    for (const char* what : {"late", "deep"}) {   // the 12 pairs that finished last, then the 12 with the most calls
        std::sort(idx.begin(), idx.end(), [&](int x, int y) { return what[0] == 'l' ? outs[x].tEndMs > outs[y].tEndMs : outs[x].cnt[0] > outs[y].cnt[0]; });
        for (int k = 0; k < std::min(np, 12); k++) { const PairOut& o = outs[idx[k]]; fprintf(stderr, "[search] %s pair %d: claimed %.1f ms, finished %.1f ms, %lld calls, %lld rotation pops, %d events\n", what, idx[k], o.tStartMs, o.tEndMs, o.cnt[0], o.cnt[3], o.nEvents); }
    }
    std::string a = "[search] pairs finished per 4 ms:", b = "[search] helper calls per 4 ms:  ";
    int last = 0; for (int k = 0; k < 256; k++) if (ctl.finishHist[k] || ctl.helpHist[k]) last = k;
    for (int k = 0; k <= last; k++) { char t[32]; snprintf(t, sizeof t, " %d", ctl.finishHist[k]); a += t; snprintf(t, sizeof t, " %d", ctl.helpHist[k]); b += t; }
    fprintf(stderr, "%s\n%s\n", a.c_str(), b.c_str());
    fprintf(stderr, "[search] ctas %d calls %llu pops %llu busy-cycles/pop %.0f corner-misses/pop %.2f; CTA cycles: total %.4g in calls %.4g scheduling+idle %.4g; icp requests %llu\n", ctas, dc.calls, dc.pops,
            (double)dc.callCycles / std::max<double>(1, dc.pops), (double)dc.cornerMisses / std::max<double>(1, dc.pops), (double)dc.ctaCycles, (double)dc.callCycles, (double)dc.idleCycles, dc.icpRequests);
    if (dc.phaseCycles[0]) fprintf(stderr, "[phases] cycles per pop: stage(per call) %.0f  A1 %.0f  A2 %.0f (chain on warp 0: %.0f)  C %.0f\n", (double)dc.phaseCycles[0] / std::max<double>(1, dc.calls), (double)dc.phaseCycles[1] / std::max<double>(1, dc.pops), (double)dc.phaseCycles[2] / std::max<double>(1, dc.pops), (double)dc.phaseCycles[4] / std::max<double>(1, dc.pops), (double)dc.phaseCycles[3] / std::max<double>(1, dc.pops));
}
static goicp_status register_resident(Eng* h, const BnbCfg& cfg) {
    const goicp_params& p = h->params;
    const int np = (int)h->probs.size();
    int perSM = goicp_search_occupancy(cfg.smemBytes, h->exact_sums, cfg.threads, cfg.useSmem, cfg.ct);
    { const char* e = getenv("GOICP_CTAS_PER_SM"); if (e && atoi(e) >= 1) perSM = std::min(perSM, atoi(e)); }
    int ctas = h->numSM * perSM;
    { const char* e = getenv("GOICP_CTAS"); if (e && atoi(e) >= 1) ctas = std::min(ctas, atoi(e)); }
    // per-CTA slabs: translation queue (32 B per entry) and rotation queue (2 x 32 B per node); a pair that outgrows either is re-run by
    // the wave scheduler with growing slabs -- slow, so the slabs are generous (4 MB + 1 MB per CTA)
    int heapCap = 1 << 17;
    { const char* e = getenv("GOICP_HEAPCAP"); if (e && atoi(e) >= 129) heapCap = atoi(e); }   // test hook: force the overflow re-run
    const int rqCap = 1 << 14;
    const int memoCap = 8192;
    CU(h->sCtl.ensure(sizeof(SearchCtl)));
    CU(h->sHdrs.ensure(goicp_search_hdr_bytes() * (size_t)ctas));
    CU(h->sSlots.ensure(goicp_search_slot_bytes() * (size_t)ctas * SR_NSLOT));
    CU(h->sStates.ensure(sizeof(unsigned) * (size_t)ctas * SR_NSLOT));
    CU(h->sRq.ensure(goicp_search_rnode_bytes() * (size_t)ctas * 2 * rqCap));
    CU(h->sIcp.ensure(sizeof(IcpState) * 2 * (size_t)ctas));
    CU(h->sOuts.ensure(sizeof(PairOut) * (size_t)np));
    CU(h->hOuts.ensure(sizeof(PairOut) * (size_t)np));
    CU(h->qHeaps.ensure(sizeof(HeapEnt) * (size_t)ctas * heapCap));
    if (!cfg.useSmem) CU(h->qScratch.ensure(sizeof(float) * cfg.smemFloats * (size_t)ctas));
    if (h->qMemo.cap < (size_t)32 * memoCap * ctas) { CU(h->qMemo.ensure((size_t)32 * memoCap * ctas)); CU(cudaMemsetAsync(h->qMemo.p, 0, h->qMemo.cap, h->stream)); }
    CU(cudaMemsetAsync(h->sCtl.p, 0, sizeof(SearchCtl), h->stream));
    CU(cudaMemsetAsync(h->sHdrs.p, 0, goicp_search_hdr_bytes() * (size_t)ctas, h->stream));
    CU(cudaMemsetAsync(h->sStates.p, 0, sizeof(unsigned) * (size_t)ctas * SR_NSLOT, h->stream));
    SearchArgs A{};
    A.pairs = h->dPairs.as<PairDev>(); A.npairs = np; A.nCtas = ctas;
    A.rotMinX = p.rotMinX; A.rotMinY = p.rotMinY; A.rotMinZ = p.rotMinZ; A.rotWidth = p.rotWidth;
    A.fma = host_libm_uses_fma() ? 1 : 0;
    { const char* e = getenv("GOICP_LIBM_FMA"); if (e) A.fma = atoi(e) != 0; }
    A.specMax = std::max(0, std::min(h->spec_groups, SR_NGROUP - 4));
    { const char* e = getenv("GOICP_SPEC_GROUPS"); if (e) A.specMax = std::max(0, std::min(atoi(e), SR_NGROUP - 4)); }
    A.quietRamp = 1;
    A.walkEvery = np > 1 ? 16 : 8;   // measured: batch step 500 / 496 / 488 / 477 ms and pair 2 alone 86 / 71 / 66 / 71 ms at 1 / 4 / 8 / 16
    { const char* e = getenv("GOICP_WALK_EVERY"); if (e) A.walkEvery = std::max(1, atoi(e)); }
    { const char* e = getenv("GOICP_QUIET_RAMP"); if (e) A.quietRamp = atoi(e) != 0; }
    A.managerRatio = 8;
    { const char* e = getenv("GOICP_MANAGER_RATIO"); if (e && atoi(e) >= 0) A.managerRatio = atoi(e); }
    // help during the bulk takes CTAs away from unclaimed pairs; measured on 4096 BO1 pairs (B200, 1000 W), ms per step:
    // 471 / 462 / 452 / 448 at 1024 / 2048 / 4096 / 16384.  A single registration never meets the bar (no pair is left unclaimed).
    A.deepCalls = 16384;
    { const char* e = getenv("GOICP_DEEP_CALLS"); if (e && atoi(e) >= 1) A.deepCalls = atoi(e); }
    A.ctl = h->sCtl.as<SearchCtl>(); A.hdrs = h->sHdrs.as<OwnerHdr>(); A.slots = h->sSlots.as<SearchSlot>(); A.states = h->sStates.as<unsigned>(); A.rq = h->sRq.p; A.rqCap = rqCap;
    A.icp = h->sIcp.as<IcpState>(); A.outs = h->sOuts.as<PairOut>();
    A.heaps = h->qHeaps.as<HeapEnt>(); A.heapCap = heapCap; A.gscratch = h->qScratch.as<float>(); A.gstride = cfg.smemFloats; A.NdP = cfg.NdP; A.NdQ = cfg.NdQ; A.useSmem = cfg.useSmem;
    A.memo = reinterpret_cast<uint4*>(h->qMemo.p); A.memoCap = memoCap; A.ctr = h->devCounters.as<DevCounters>(); A.gridOff = cfg.gridOff; A.S3p = cfg.S3p;
    A.cutoff = h->cutoffOn ? h->dCutoff.as<float>() : nullptr;
    cudaEventRecord(h->main.ev0, h->stream);
    CU(goicp_launch_search(A, ctas, cfg.threads, cfg.smemBytes, h->exact_sums, cfg.ct, h->stream));
    cudaEventRecord(h->main.ev1, h->stream);
    CU(cudaMemcpyAsync(h->hOuts.p, h->sOuts.p, sizeof(PairOut) * (size_t)np, cudaMemcpyDeviceToHost, h->stream));
    const cudaError_t e = h->main.sync();
    if (e != cudaSuccess) return fail(h, GOICP_ERR_CUDA, "device-resident search kernel: %s", cudaGetErrorString(e));
    float ms = 0; cudaEventElapsedTime(&ms, h->main.ev0, h->main.ev1); h->main.ms[2] += ms; h->main.launches[2] += 1;
    const PairOut* outs = h->hOuts.as<PairOut>();
    std::vector<int> redo;
    for (int i = 0; i < np; i++) {
        const PairOut& o = outs[i];
        if (o.status == GOICP_SR_UNSUPPORTED) return fail(h, GOICP_ERR_ARG, "trimmed ICP without its sort workspace (trimFraction changed after the clouds were set?)");
        if (o.status != 0) { redo.push_back(i); continue; }
        SearchResult& r = h->probs[i].res = SearchResult();
        memcpy(r.optR, o.R, sizeof r.optR); memcpy(r.optT, o.t, sizeof r.optT);
        r.optError = o.optError; r.optComp = o.optComp;
        for (int k = 0; k < 6; k++) r.cnt[k] = o.cnt[k];
        r.trace.events.resize(o.nEvents);
        for (int k = 0; k < o.nEvents; k++) r.trace.events[k] = TraceEvent{o.ev[k].kind, o.ev[k].v};
        trace_end(r, o.endKind, o.endLb, h->probs[i].dev.SSEThresh, h->probs[i].cutoff);
    }
    h->stats.rerunPairs = (int)redo.size();
    if (!redo.empty()) {   // a queue outgrew its per-CTA slab: re-run those pairs with the wave scheduler, which grows the slabs on demand
        std::atomic<int> nx(0);
        h->main.ctaCap = 0;
        if (goicp_status s2 = register_group(h, h->main, cfg, nx, std::min<int>(64, (int)redo.size()), &redo)) return s2;
    }
    DevCounters dc;   // read, then cleared for the next search; the memo's generation word keeps counting
    cudaMemcpy(&dc, h->devCounters.p, sizeof dc, cudaMemcpyDeviceToHost);
    cudaMemset(h->devCounters.as<char>() + offsetof(DevCounters, callCycles), 0, sizeof dc - offsetof(DevCounters, callCycles));
    SearchStats& st = h->stats;
    st.calls = dc.calls; st.pops = dc.pops; st.callCycles = dc.callCycles; st.cornerMisses = dc.cornerMisses; st.idleCycles = dc.idleCycles;
    st.ctas = ctas; st.ctaCycles = dc.ctaCycles;
    h->main.callsLaunched += (long long)dc.calls;
    if (getenv("GOICP_DEBUG")) print_search_debug(h, ctas, dc, outs, np);
    return GOICP_OK;
}

// GoICP::Register (jly_goicp.cpp:878) for every problem of the handle.  One problem: waves on the handle's stream.
// A batch: `groups` worker threads, each with its own stream, pull pairs from a shared counter.
goicp_status register_all(Eng* h) {
    auto t0 = clk::now();
    goicp_status s;
    if ((s = initialize_all(h))) return s;
    const int np = (int)h->probs.size();
    const BnbCfg cfg = bnb_config(h);
    h->stats = SearchStats();
    std::atomic<int> next(0);
    int groups = 1, slots = 1;
    if (np > 1) {
        unsigned cores = std::max(1u, std::thread::hardware_concurrency());
        { const char* e = getenv("LOCAL_WORLD_SIZE"); const int lws = e ? atoi(e) : 1; if (lws > 1) cores = std::max(2u, cores / (unsigned)lws); }   // one process per GPU (torchrun): share the host cores
        groups = h->groups > 0 ? h->groups : (int)std::min<unsigned>(32u, std::max(cores >= 4u ? 4u : 2u, cores));
        slots = h->slots > 0 ? h->slots : std::min(128, std::max(8, (np + groups - 1) / groups));
        groups = std::min(groups, (np + slots - 1) / slots);
    }
    { const char* e = getenv("GOICP_PERSISTENT"); if (e) h->resident = atoi(e) != 0; }   // 0: wave scheduler (one launch per wave, OuterBnB on the host)
    bool allSmall = true;
    for (auto& P : h->probs) if ((size_t)P.Nd * P.Nm > ((size_t)1 << 21) || (P.dev.doTrim && P.Nd > 2048)) allSmall = false;
    const bool resident = h->resident && allSmall && h->shardN <= 1 && !(h->relaxed && np == 1);
    if (h->relaxed && np == 1) {
        h->main.ctaCap = 0;
        if ((s = register_relaxed(h, h->main, cfg, 0))) return s;
    } else if (resident) {
        groups = 0;
        if ((s = register_resident(h, cfg))) return s;
    } else if (groups <= 1) {
        h->main.ctaCap = 0;
        if ((s = register_group(h, h->main, cfg, next, slots))) return s;
    } else {
        while ((int)h->workers.size() < groups) {
            std::unique_ptr<WaveCtx> w(new WaveCtx());
            if (w->init(true, nullptr) != GOICP_OK) return fail(h, GOICP_ERR_CUDA, "worker stream creation failed");
            h->workers.push_back(std::move(w));
        }
        CU(cudaStreamSynchronize(h->stream));   // inputs / DT / Initialize were enqueued on the handle's stream
        std::vector<goicp_status> st(groups, GOICP_OK);
        std::vector<std::thread> th;
        for (int g = 0; g < groups; g++) {
            WaveCtx* w = h->workers[g].get();
            w->ctaCap = std::max(64, 2 * h->numSM * cfg.perSM / groups);
            w->reset_timing();
            th.emplace_back([h, w, &cfg, &next, &st, g, slots]() { cudaSetDevice(h->device); st[g] = register_group(h, *w, cfg, next, slots); });
        }
        for (auto& t : th) t.join();
        for (int g = 0; g < groups; g++) if (st[g]) return st[g];
        for (int g = 0; g < groups; g++) {
            WaveCtx* w = h->workers[g].get();
            for (int k = 0; k < 5; k++) { h->main.ms[k] += w->ms[k]; h->main.launches[k] += w->launches[k]; }
            h->main.waves += w->waves; h->main.callsLaunched += w->callsLaunched;
            h->main.tLogic += w->tLogic; h->main.tInnerEnq += w->tInnerEnq; h->main.tInnerWait += w->tInnerWait;
        }
    }
    h->main.collect();   // the DT / Initialize timers (every scheduler has synchronised the handle's stream past them)
    const double dt = secs_since(t0);
    for (auto& P : h->probs) P.t_reg = dt / std::max(1, np);
    SearchStats& st = h->stats;
    st.waves = h->main.waves; st.callsExecuted = h->main.callsLaunched; st.hostThreads = groups; st.hostSeconds = dt;
    for (auto& P : h->probs) st.callsUsed += P.res.cnt[0];
    if (!resident) { st.tRequests = h->main.tLogic; st.tEnqueue = h->main.tInnerEnq; st.tWait = h->main.tInnerWait; }
    return GOICP_OK;
}

void fill_result(Eng* h, const Problem& P, goicp_result* out) {
    const SearchResult& r = P.res;
    memset(out, 0, sizeof *out);
    memcpy(out->R, r.optR, sizeof out->R); memcpy(out->t, r.optT, sizeof out->t);
    out->optError = r.optError; out->optComp = r.optComp;
    for (int k = 0; k < 8; k++) out->counters[k] = r.cnt[k];
    out->counters[6] = h->main.launches[0] + h->main.launches[1] + h->main.launches[2] + h->main.launches[3] + h->main.launches[4];
    out->counters[7] = (long long)h->stats.callsExecuted - (long long)h->stats.callsUsed;
    out->seconds_dt = P.t_dt; out->seconds_register = P.t_reg;
    out->gpu_ms_dt = h->main.ms[0]; out->gpu_ms_bnb = h->main.ms[2]; out->gpu_ms_icp = h->main.ms[3];
}

