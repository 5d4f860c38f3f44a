// host check of csrc/host_search.h against std::priority_queue over the reference's ROTNODE (tests/test_host_search.py)
#include <cstdio>
#include <cstdlib>
#include <queue>
#include <random>
#include <vector>
#include "host_search.h"

// jly_goicp.h:59-73; `a` carries a unique id here
typedef struct _ROTNODE {
    float a, b, c, w;
    float ub, lb;
    int l;
    friend bool operator<(const struct _ROTNODE& n1, const struct _ROTNODE& n2) {
        if (n1.lb != n2.lb) return n1.lb > n2.lb;
        else return n1.w < n2.w;
    }
} ROTNODE;

struct Pair { std::priority_queue<ROTNODE> ref; std::vector<RNode> mine; };

static void push(Pair& p, int id, float lb, float w) {
    ROTNODE r{}; r.a = (float)id; r.lb = lb; r.w = w; p.ref.push(r);
    RNode n{}; n.id = id; n.lb = lb; n.w = w; rheap_push(p.mine, n);
}
// pops both until empty; true if the ids come out in the same order
static bool same_pops(Pair& p) {
    while (!p.ref.empty()) {
        const int a = (int)p.ref.top().a; p.ref.pop();
        if (p.mine.empty() || rheap_pop(p.mine).id != a) return false;
    }
    return p.mine.empty();
}

int main(int argc, char** argv) {
    const int cases = argc > 1 ? atoi(argv[1]) : 2000;
    std::mt19937 rng(12345);
    const float lbs[4] = {0.5f, 1.f, 1.5f, 2.f}, ws[3] = {1.f, 0.5f, 0.25f};   // few distinct keys: many ties
    long heapBad = 0, popOrderBad = 0, anyOrderBad = 0;
    for (int c = 0; c < cases; c++) {
        // (a) interleaved pushes and pops
        Pair p; int id = 0;
        const int ops = 1 + (int)(rng() % 400);
        for (int k = 0; k < ops; k++) {
            if (!p.ref.empty() && rng() % 3 == 0) {
                const int a = (int)p.ref.top().a; p.ref.pop();
                if (rheap_pop(p.mine).id != a) { heapBad++; break; }
            } else push(p, id++, lbs[rng() % 4], ws[rng() % 3]);
        }
        if (!same_pops(p)) heapBad++;
        // (b) the queue pruning of jly_goicp.cpp:843-853, then every remaining pop
        Pair q; id = 0;
        const int n = 1 + (int)(rng() % 300);
        for (int k = 0; k < n; k++) { push(q, id++, lbs[rng() % 4], ws[rng() % 3]); if (rng() % 5 == 0) { q.ref.pop(); rheap_pop(q.mine); } }
        const float optError = lbs[rng() % 4];
        std::vector<RNode> any = q.mine;
        std::priority_queue<ROTNODE> queueRotNew;
        while (!q.ref.empty()) {
            ROTNODE node = q.ref.top();
            q.ref.pop();
            if (node.lb < optError) queueRotNew.push(node);
            else break;
        }
        q.ref = queueRotNew;
        Pair r{q.ref, any};
        prune_in_pop_order(q.mine, optError);
        if (!same_pops(q)) popOrderBad++;
        prune_any_order(r.mine, optError);
        if (!same_pops(r)) anyOrderBad++;
    }
    printf("cases %d heap_mismatches %ld prune_in_pop_order_mismatches %ld prune_any_order_mismatches %ld\n", cases, heapBad, popOrderBad, anyOrderBad);
    return heapBad || popOrderBad ? 1 : 0;
}
