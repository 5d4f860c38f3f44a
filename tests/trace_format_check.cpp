// The "Error*:" trace of csrc/host_search.h is recorded as values and formatted when read (Trace::str).  This check holds the
// formatter to the text the rules used to write as they ran: the eager functions below are that code, kept verbatim.  Random
// traces (every event kind, every end kind, values from denormals to infinities and NaN) must give the same bytes both ways.
//   usage: trace_format_check <cases>      prints "cases N mismatches M"
#include <random>
#include "host_search.h"

namespace eager {
inline void trace_event(std::string& s, int kind, float err) {
    static const char* kinds[3] = {"Init", "ICP", "BNB"};
    tracef(s, "Error*: %g (%s)\n", err, kinds[kind % 3]);
}
inline void trace_end(std::string& s, float optError, int kind, float lb, float sse, float cutoff) {
    if (kind == END_QUEUE_EMPTY) tracef(s, "Rotation Queue Empty\nError*: %g, LB: %g\n", optError, lb);
    else if (kind == END_THRESHOLD) tracef(s, "Threshold reached\nError*: %g, LB: %g, epsilon: %g\n", optError, lb, sse);
    else tracef(s, "Cutoff reached\nError*: %g, LB: %g, cutoff: %g\n", optError, lb, cutoff);
}
}  // namespace eager

static float any_float(std::mt19937_64& rng) {
    static const float special[] = {0.f, -0.f, 1.f, 8.45388f, 1e-45f, 1.17549435e-38f, 3.4028235e38f, 1e30f, 123456789.f, 0.1f, -2.5f,
                                    INFINITY, -INFINITY, NAN};
    switch (rng() % 4) {
    case 0: return special[rng() % (sizeof special / sizeof special[0])];
    case 1: { uint32_t u = (uint32_t)rng(); float f; memcpy(&f, &u, 4); return f; }   // any bit pattern
    default: return std::ldexp((float)(rng() % 1000000) / 1e5f, (int)(rng() % 40) - 20);
    }
}

int main(int argc, char** argv) {
    const int cases = argc > 1 ? atoi(argv[1]) : 1000;
    std::mt19937_64 rng(20261022);
    int bad = 0;
    for (int c = 0; c < cases; c++) {
        SearchResult r;
        std::string want;
        // the schedulers' rules: init_incumbent, take_icp, after_bnb append events; trace_end closes the trace
        init_incumbent(r, any_float(rng), goicp_params{}, 1 + (int)(rng() % 300));
        eager::trace_event(want, TRACE_INIT, r.optError);
        const int n = (int)(rng() % 12);
        for (int k = 0; k < n; k++) {
            const int kind = (int)(rng() % 3);
            const float v = any_float(rng);
            trace_event(r.trace, kind, v); eager::trace_event(want, kind, v);
            r.optError = v;
        }
        const bool ended = c % 7 != 0;   // a trace read before its end line (no end record yet)
        if (ended) {
            const int kind = 1 + c % 3;
            const float lb = any_float(rng), sse = any_float(rng), cutoff = any_float(rng);
            trace_end(r, kind, lb, sse, cutoff); eager::trace_end(want, r.optError, kind, lb, sse, cutoff);
        }
        const std::string got = r.trace.str();
        if (got != want || std::string(r.trace.c_str()) != want || r.trace.str() != want) {
            if (bad < 3) printf("case %d differs:\n--- eager\n%s--- on read\n%s", c, want.c_str(), got.c_str());
            bad++;
        }
    }
    printf("cases %d mismatches %d\n", cases, bad);
    return bad != 0;
}
