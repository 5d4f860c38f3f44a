// Device side of one GoICP::InnerBnB call (jly_goicp.cpp:286-579) -- shared by the wave kernel (k_bnb.cu) and by the
// device-resident search kernel (k_search.cu).  See k_bnb.cu for the structure of one translation-queue pop.
#pragma once
#include <cstdlib>
#include "icp_device.cuh"
#include "launch.h"

namespace {

#ifndef GOICP_BNB_THREADS
#define GOICP_BNB_THREADS 256
#endif
#ifndef GOICP_BNB_MIN_CTAS
#define GOICP_BNB_MIN_CTAS 3
#endif
constexpr int BNB_MAX_THREADS = GOICP_BNB_THREADS;

// ---- 1-D TMA (cp.async.bulk) global -> shared with mbarrier completion: the S<=~26 DT volume of a call is staged in shared
//      memory by the copy engine while the CTA rotates the cloud ----------------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
// plain shared-memory atomics (nvcc wraps atomicAdd in ~30 instructions of warp-aggregation code; the callers below already
// elect one lane)
__device__ __forceinline__ int smem_fetch_add(int* p, int v) {
    int old; asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(smem_u32(p)), "r"(v) : "memory"); return old;
}
__device__ __forceinline__ void smem_red_add(int* p, int v) { asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory"); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile("{\n .reg .pred p;\n WAIT_LOOP:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n @p bra.uni WAIT_DONE;\n bra.uni WAIT_LOOP;\n WAIT_DONE:\n}"
                 ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

// The translation queue.  A node is a 64-bit key {lb, (level << 26) | slot} plus a payload slot {x, y, z}: only the keys move
// when the heap is sifted.  The node width is tWidth / 2^level exactly (every level halves it, jly_goicp.cpp:322), so
// TRANSNODE operator< (jly_goicp.h:79-86: larger lb is "less"; equal lb: smaller w is "less") compares levels instead of
// widths.  Keys [0, HK_SMEM) and payload slots [0, HP_SMEM) live in shared memory, the rest in the CTA's global slab.
// Only lane 0 of warp 0 touches the queue; it follows libstdc++'s push_heap / pop_heap step for step, so ties between equal
// (lb, w) keys pop in the reference's order.
constexpr int HK_SMEM = 512;
constexpr int HP_SMEM = 128;
constexpr int HF_SMEM = 128;
constexpr int MAX_TLEVEL = 64;
__device__ __forceinline__ bool key_less(const uint2 a, const uint2 b) {
    const float la = __uint_as_float(a.x), lb = __uint_as_float(b.x);
    if (la != lb) return la > lb;
    return (a.y >> 26) > (b.y >> 26);
}
// corner-memo hash: the coordinates are dyadic floats (long runs of trailing zero bits), so mix with rotations and take the
// HIGH bits of a multiplicative hash
__device__ __forceinline__ unsigned memo_hash(unsigned kx, unsigned ky, unsigned kz) {
    unsigned h = kx * 0x9E3779B1u;
    h = __funnelshift_l(h, h, 13) ^ (ky * 0x85EBCA77u);
    h = __funnelshift_l(h, h, 11) ^ (kz * 0xC2B2AE3Du);
    h ^= h >> 16; h *= 0x7FEB352Du; h ^= h >> 15;
    return h * 0x846CA68Bu;
}
__device__ __forceinline__ unsigned memo_slot(unsigned h, int shift) { return h >> shift; }
struct Heap {
    uint2* ks;       // shared keys
    uint2* kg;       // global keys (slab)
    float4* ps;      // shared payload slots
    float4* pg;      // global payload slots
    __device__ __forceinline__ uint2 key(int i) const { return (i < HK_SMEM) ? ks[i] : kg[i]; }
    __device__ __forceinline__ void setkey(int i, const uint2 k) const { if (i < HK_SMEM) ks[i] = k; else kg[i] = k; }
    __device__ __forceinline__ float4 pay(int sl) const { return (sl < HP_SMEM) ? ps[sl] : pg[sl]; }
    __device__ __forceinline__ void setpay(int sl, const float4 v) const { if (sl < HP_SMEM) ps[sl] = v; else pg[sl] = v; }
};
// shared-memory-only, warp-cooperative forms (queue shorter than HK_SMEM: the common case).  Called by all 32 lanes.
// __push_heap from position `hole` with value `val`: lane l reads the l-th ancestor; val stops below the first ancestor that is
// not "less" than it; the ancestors it passes each move down one step.  Same final layout as the sequential loop.
__device__ __forceinline__ void heap_siftup_w(uint2* ks, int hole, const uint2 val, int lane) {
    const int anc = ((hole + 1) >> min(lane + 1, 31)) - 1;           // parent^(lane+1)(hole); -1 above the root
    const uint2 pe = ks[max(anc, 0)];
    const unsigned m = __ballot_sync(GOICP_FULL, anc >= 0 && key_less(pe, val));
    const int moves = __ffs(~m) - 1;                                 // leading ancestors that are "less" than val
    if (lane < moves) ks[lane == 0 ? hole : ((hole + 1) >> lane) - 1] = pe;
    if (lane == 0) ks[moves == 0 ? hole : ((hole + 1) >> moves) - 1] = val;
    __syncwarp();
}
// std::pop_heap: __adjust_heap walks the hole to the bottom along the "not less" children (every lane follows the same path,
// lane 0 stores), then the former last element is sifted up from there.  n = size before the pop; returns the former top.
__device__ __forceinline__ uint2 heap_pop_w(uint2* ks, int n, int lane) {
    const uint2 top = ks[0];
    const int len = n - 1;
    if (len > 0) {
        const uint2 val = ks[len];
        int hole = 0, child = 0;
        while (child < (len - 1) / 2) {
            child = 2 * (child + 1);
            uint2 c1 = ks[child]; const uint2 c0 = ks[child - 1];
            if (key_less(c1, c0)) { child--; c1 = c0; }
            if (lane == 0) ks[hole] = c1;
            hole = child;
        }
        if ((len & 1) == 0 && child == (len - 2) / 2) {
            child = 2 * (child + 1);
            if (lane == 0) ks[hole] = ks[child - 1];
            hole = child - 1;
        }
        __syncwarp();
        heap_siftup_w(ks, hole, val, lane);
    }
    return top;
}
// std::push_heap (__push_heap) on h[0..n) + val
__device__ __forceinline__ void heap_push(const Heap& h, int& n, const uint2 val) {
    int hole = n++;
    while (hole > 0) {
        const int parent = (hole - 1) >> 1;
        const uint2 pe = h.key(parent);
        if (!key_less(pe, val)) break;
        h.setkey(hole, pe);
        hole = parent;
    }
    h.setkey(hole, val);
}
// std::pop_heap (__adjust_heap to the bottom, then __push_heap of the former last element); returns the former top
__device__ __forceinline__ uint2 heap_pop(const Heap& h, int& n) {
    const uint2 top = h.key(0);
    const int len = --n;
    if (len > 0) {
        const uint2 val = h.key(len);
        int hole = 0, child = 0;
        while (child < (len - 1) / 2) {
            child = 2 * (child + 1);
            uint2 c1 = h.key(child); const uint2 c0 = h.key(child - 1);
            if (key_less(c1, c0)) { child--; c1 = c0; }
            h.setkey(hole, c1); hole = child;
        }
        if ((len & 1) == 0 && child == (len - 2) / 2) {
            child = 2 * (child + 1);
            h.setkey(hole, h.key(child - 1)); hole = child - 1;
        }
        while (hole > 0) {
            const int parent = (hole - 1) >> 1;
            const uint2 pe = h.key(parent);
            if (!key_less(pe, val)) break;
            h.setkey(hole, pe);
            hole = parent;
        }
        h.setkey(hole, val);
    }
    return top;
}

struct BnbShared {
    float ub[8], lb[8];
    int cnt[27];
    int cntN[27];                  // neighbour-count term per lattice corner (compareNeighbors :1250-1288)
    float cf[27];
    float X[9];                    // corner lattice of the popped node: X[0..2] x, X[3..5] y, X[6..8] z (child origins = the first two of each)
    float CX[9];                   // vox_fast constants of the lattice coordinates (corner terms), same layout
    float HX[6];                   // child-centre translations X[k] + w/2 (:331-333): [0..1] x, [2..3] y, [4..5] z ...
    float DX[6];                   // ... and their vox_fast constants
    float wtab[MAX_TLEVEL];        // node width per level: tWidth halved level times (:322)
    float wc, mtd;
    float optErrorT;
    int level;                     // level of the children being evaluated
    int running, prob, status;
    int pops, subcubes, improved;
    float best[4];
    int missList[27];
    unsigned mSlot[27], mChk[27];  // memo slot and key checksum of the missed corners
    int cntNM[27];                 // neighbour-count terms of the missed corners, in missList order
    int cntM[27];                  // incompatibility counts of the missed corners, in missList order
    float mC[81];                  // vox_fast constants of the missed corners: [m] x, [27+m] y, [54+m] z
    int nmiss, workCtr, workA;
    unsigned gen;
    long long t0; int missTot;
#ifdef GOICP_PHASE_TIMING
    long long tp[12]; long long tmark;
#endif
};

// Per pop of the translation queue (three CTA barriers):
//   phase A1 (all warps)  work items (32-point chunk, 4 child cubes): a lane loads its point once and evaluates the four
//                         cubes as independent chains (translate -> voxel -> DT gather -> weight, radius, clamp); warp 0 then
//                         files the corner-memo look-ups it issued at the end of the previous pop;
//   phase A2              warp 0 lanes 0..15: the sixteen sequential (ub, lb) sums [EXACT] or the fixed-order combine of the
//                         per-chunk partial sums; all other warps (then warp 0 too): the corners the memo missed, work items
//                         (32-point chunk, 4 corners); trimmed sums: one warp per child;
//   phase C (warp 0)      c-FPFH corner sums, memo update, per-child corner min/max on 8 lanes, the eight decisions as a warp
//                         prefix-min, then lane 0: pushes and the next pop; lanes 0..14 derive the next node's voxel constants
//                         and lanes 0..26 issue its memo look-ups.
// (k_bnb.cu: the calls of a wave are claimed through a counter; k_search.cu: the device-resident search hands them out itself.)
// GS=true (needs SMEM): the call's DT volume (float distances + one colour-mask byte per voxel) is staged in shared memory by
// TMA as 16-bit squared-distance codes + a distance table + one colour-mask byte per voxel (S^3 * 3 bytes + the table at
// dynamic-smem offset gridOff), so the per-point gathers are LDS instead of L1/L2 sector gathers.

// state a CTA carries from one call to the next
struct CallCtx {
    unsigned gphase = 0;                       // parity of the DT-staging mbarrier
    int gpair = -1;                            // pair whose DT volume sits in shared memory
};
// CANCEL (speculative calls of the device-resident search): lives in shared memory; the call is abandoned (status 7) once
// *word != gen.  One lane of the last warp polls the word while the corners are evaluated; warp 0 only reads the flag.
struct CancelSh { const volatile unsigned* word; unsigned gen; int flag; };

// One request = one InnerBnB call, or (level >= GOICP_REQ_BOTH) the upper- and the lower-bound call of one rotation cube.
// Called by every thread of the CTA; `pr` and `s_out` live in shared memory; the result is left in `s_out` (thread 0 wrote it;
// a __syncthreads / __syncwarp of warp 0 is needed before other threads read it).  `s_gbar` is an mbarrier initialised once by the
// kernel (GS only).  `ctr` collects the device counters.
template <bool EXACT, bool SMEM, bool GS, bool CT, bool CANCEL>
__device__ __forceinline__ void inner_call(const PairDev* __restrict__ pairs, const InnerProb& pr, InnerOut& s_out, unsigned long long& s_gbar, CallCtx& cx, CancelSh& cs,
                                           HeapEnt* __restrict__ heaps, int heapCap, float* gscratch, size_t gstride, int NdP, int NdQ, int useSmem,
                                           uint4* memoAll, int memoCap, DevCounters* ctr, int gridOff, int S3p) {
    extern __shared__ float4 dyn_smem4[];
    __shared__ BnbShared sh;
    __shared__ uint2 s_hkey[HK_SMEM];
    __shared__ float4 s_hpay[HP_SMEM];
    __shared__ int s_free[HF_SMEM];   // recycled payload slots (stack)
    __shared__ uint2 s_pk[8];         // keys of the children being pushed
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthreads = blockDim.x, nwarps = blockDim.x >> 5;
    float* base = SMEM ? reinterpret_cast<float*>(dyn_smem4) : gscratch + (size_t)blockIdx.x * gstride;   // SMEM: address space known -> LDS/STS
    float* tx = base; float* ty = tx + NdP; float* tz = ty + NdP; float* wgt = tz + NdP; float* mrd = wgt + NdP;
    uint8_t* dprop_s = reinterpret_cast<uint8_t*>(mrd + NdP);   // [NdP] colour index of each data point
    float* part = mrd + NdP + (NdP >> 2);                       // [8][nchunks][2] + [27][nchunks] per-chunk partial sums (tree-sum mode)
    float* md = part + (EXACT ? 0 : ((43 * (NdP >> 5) + 3) & ~3));   // [8][NdQ] clamped residuals d of the 8 child cubes (EXACT / trimmed); rows 16-byte aligned
    float* fp = md + 8 * NdQ;                                   // [27][NdQ]  (EXACT with the c-FPFH term)
    Heap heap;
    {
        char* slab = reinterpret_cast<char*>(heaps + (size_t)blockIdx.x * heapCap);      // 32 bytes per queue entry: 8 key + 16 payload used
        heap.ks = s_hkey; heap.kg = reinterpret_cast<uint2*>(slab);
        heap.ps = s_hpay; heap.pg = reinterpret_cast<float4*>(slab + (size_t)heapCap * 8);
    }
    uint4* memo = memoAll + 2 * (size_t)blockIdx.x * memoCap;
    const int memoShift = 32 - (31 - __clz(memoCap));   // this CTA's corner memo: direct-mapped, 32 B entries, tagged with the call's generation
    // GS: the pair's volume in shared memory as [nlutP] distance table, [S3p] 16-bit squared-distance codes, [S3p] colour-mask bytes
    float* slut = reinterpret_cast<float*>(dyn_smem4) + gridOff;
    const int chainWarp = nwarps > 1 ? 1 : 0;
    unsigned& gphase = cx.gphase; int& gpair = cx.gpair;
    __syncthreads();   // the previous call of this CTA has left the shared arrays
    {
        const PairDev& P = pairs[pr.pair];
        const GridDev& g = P.g;
        const bool gload = GS && (gpair != pr.pair || (useSmem & 16));   // bit 4 of useSmem: debugging switch, restage for every request   // (the __syncthreads at the top of the loop ordered the last reads of the old volume)
        const int nlutP = (g.nlut + 3) & ~3;
        const uint16_t* scode = reinterpret_cast<const uint16_t*>(slut + nlutP);
        const uint8_t* svm = reinterpret_cast<const uint8_t*>(scode + S3p);
        if (gload && tid == 0) {
            mbar_expect_tx(&s_gbar, (unsigned)nlutP * 4u + (unsigned)S3p * 3u);
            tma_bulk_g2s(slut, g.dlut, (unsigned)nlutP * 4u, &s_gbar);
            tma_bulk_g2s(const_cast<uint16_t*>(scode), g.dcode, (unsigned)S3p * 2u, &s_gbar);
            tma_bulk_g2s(const_cast<uint8_t*>(svm), g.vmask8, (unsigned)S3p, &s_gbar);
        }
        // per-problem constants in registers (the PairDev lives in global memory)
        const int Nd = P.Nd;
        const int nchunks = (Nd + 31) >> 5;
        const bool doTrim = P.doTrim != 0;
        const bool useMd = EXACT || doTrim;
        const int ncp1 = g.ncells + 1;
        const int norm = P.norm;
        const int inlierNum = P.inlierNum;
        const int S = g.S;
        const bool use_reg = P.use_reg != 0, use_fpfh = CT && P.use_fpfh != 0, use_nb = CT && P.use_nb != 0;
        const bool corners = use_reg || use_fpfh || use_nb;
        const VoxFast vf = vox_fast_of(g);

        // A request may ask for both InnerBnB calls OuterBnB makes for one rotation cube (jly_goicp.cpp:768 and :856): the upper-
        // bound call (no rotation radii) and, unless that one improves the incumbent, the lower-bound call at the cube's level.
        // The two searches share the staged cloud, the DT volume and the corner memo (corner terms do not depend on the level).
        const bool both = pr.level >= GOICP_REQ_BOTH;
        const int nparts = both ? 2 : 1;
        for (int cpart = 0; cpart < nparts; ++cpart) {
        const int level = both ? (cpart == 0 ? -1 : pr.level - GOICP_REQ_BOTH) : pr.level;
        if (cpart == 1) {
            __syncthreads();
            if (s_out.err < pr.optError || s_out.status != 0) break;   // the upper bound improved: OuterBnB runs ICP before the next call (:771-840)
        }
        // ---- stage the rotated cloud (jly_goicp.cpp:750-756), weights and rotation radii ---------------------
        for (int i = tid; i < Nd; i += nthreads) {
            if (cpart == 0) {
                const float x = P.dx[i], y = P.dy[i], z = P.dz[i];
                tx[i] = pr.R[0] * x + pr.R[1] * y + pr.R[2] * z;
                ty[i] = pr.R[3] * x + pr.R[4] * y + pr.R[5] * z;
                tz[i] = pr.R[6] * x + pr.R[7] * y + pr.R[8] * z;
                wgt[i] = P.weights[i];
                dprop_s[i] = P.dprop[i];
            }
            mrd[i] = level >= 0 ? P.maxRotDis[(size_t)level * Nd + i] : 0.f;   // d - 0 == d
        }
        if (tid < 27) sh.cnt[tid] = 0;
        if (tid == 0) {
            sh.status = 0; sh.pops = 1; sh.subcubes = 0; sh.improved = 0;
            if (cpart == 0) { sh.gen = atomicAdd(&ctr->gen, 1u) + 1u; sh.t0 = clock64(); sh.missTot = 0; }
            sh.nmiss = 0; sh.workCtr = 0; sh.workA = 0;
#ifdef GOICP_PHASE_TIMING
            if (cpart == 0) for (int k = 0; k < 12; k++) sh.tp[k] = 0;
            sh.tmark = clock64();
#endif
            sh.optErrorT = pr.optError;                                              // :297
            sh.best[0] = sh.best[1] = sh.best[2] = sh.best[3] = 0.f;
            { float w = P.tWidth; for (int l = 0; l < MAX_TLEVEL; l++) { sh.wtab[l] = w; w = w / 2; } }   // :322
            // the first pop is always the initial node (:300,:314) with lb = 0
            if (pr.optError - 0.f < P.SSEThresh) sh.running = 0;                     // :317
            else {
                sh.running = 1;
                const float wc = P.tWidth / 2;
                sh.wc = wc; sh.mtd = (float)(GOICP_SQRT3 / 2.0 * wc); sh.level = 1;
                sh.X[0] = P.tMinX; sh.X[1] = P.tMinX + wc; sh.X[2] = sh.X[1] + wc;
                sh.X[3 + (0)] = P.tMinY; sh.X[3 + (1)] = P.tMinY + wc; sh.X[3 + (2)] = sh.X[3 + (1)] + wc;
                sh.X[6 + (0)] = P.tMinZ; sh.X[6 + (1)] = P.tMinZ + wc; sh.X[6 + (2)] = sh.X[6 + (1)] + wc;
            }
        }
        __syncthreads();
        // voxel-index constants of the first node (lanes 0..14 of warp 0, as after every later pop)
        if (warp == 0 && sh.running) {
            const float half = sh.wc / 2;
            if (lane < 9) { const int a = lane / 3; sh.CX[lane] = vox_fast_c(g.vfMagic, sh.X[lane], a == 0 ? g.xMin : a == 1 ? g.yMin : g.zMin, g.scale); }
            else if (lane < 15) { const int a = (lane - 9) >> 1, k = (lane - 9) & 1; const float t = sh.X[3 * a + k] + half;   // :331-333
                                  sh.HX[2 * a + k] = t; sh.DX[2 * a + k] = vox_fast_c(g.vfMagic, t, a == 0 ? g.xMin : a == 1 ? g.yMin : g.zMin, g.scale); }
        }
        uint4 me0 = make_uint4(0u, 0u, 0u, 0u), me1 = make_uint4(0u, 0u, 0u, 0u);   // warp 0, lanes 0..26: this pop's memo look-ups (gen 0 never matches)
        if (cpart == 1 && corners && warp == 0 && lane < 27 && sh.running) {   // the root lattice was evaluated by the upper-bound call
            const int cz_ = lane / 9, cy_ = (lane - 9 * cz_) / 3, cx_ = lane - 9 * cz_ - 3 * cy_;
            const unsigned hsh = memo_hash(__float_as_uint(sh.X[cx_]), __float_as_uint(sh.X[3 + cy_]), __float_as_uint(sh.X[6 + cz_]));
            const uint4* e = memo + 2 * (size_t)memo_slot(hsh, memoShift);
            me0 = e[0]; me1 = e[1];
        }
        // search state of the call, warp-uniform registers of warp 0 (the only warp that runs phase C)
        float optT = pr.optError;                                                    // :297
        int heapN = 0, freeTop = 0, bump = 0, sh_pops = 1, sh_subcubes = 0;
        int dNpush = 0, dPop = 0, predSlot = -1, intErr = 0;                        // queue update deferred past barrier 1
        const float SSE = P.SSEThresh, regW = P.reg, regFW = P.regF, regNW = P.regN;
        if (gload && cpart == 0) { mbar_wait(&s_gbar, gphase); gphase ^= 1u; gpair = pr.pair; }

        for (;;) {
            __syncthreads();                                                         // (1) the popped node and its constants are visible
#ifdef GOICP_PHASE_TIMING
            if (tid == 0) { const long long n_ = clock64(); sh.tp[sh_subcubes == 0 ? 0 : 3] += n_ - sh.tmark; sh.tmark = n_; }
#endif
            if (!sh.running) break;
            const float mtd = sh.mtd;

            // ---- phase A1: the cube.point bound evals (:343-382).  Item = (chunk of 32 points, 4 child cubes), dealt dynamically ----
            for (;;) {
                int it = 0;
                if (lane == 0) it = smem_fetch_add(&sh.workA, 1);
                it = __shfl_sync(GOICP_FULL, it, 0);
                if (it >= 2 * nchunks) break;
                const int ch = it >> 1, q4 = (it & 1) * 4;
                const int i = ch * 32 + lane;
                const bool valid = i < Nd;
                const float px = valid ? tx[i] : 0.f, py = valid ? ty[i] : 0.f, pz = valid ? tz[i] : 0.f;
                const float w_i = valid ? wgt[i] : 0.f, r_i = valid ? mrd[i] : 0.f;
                const float dzc = sh.DX[4 + (q4 >> 2)], hz = sh.HX[4 + (q4 >> 2)];
                float dres[4]; int vox[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) vox[k] = vox_fast(vf, S, px, py, pz, sh.DX[k & 1], sh.DX[2 + (k >> 1)], dzc);
                unsigned flags = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) { dres[k] = GS ? slut[scode[max(vox[k], 0)]] : __ldg(g.dist + max(vox[k], 0)); flags |= (vox[k] < 0 ? 1u : 0u) << k; }
                unsigned any = __reduce_or_sync(GOICP_FULL, flags);
                while (any) {   // some lane is outside the grid or on a rounding boundary (rare): overshoot table, else the exact form
                    const int k = __ffs(any) - 1; any &= any - 1;
                    if (flags & (1u << k)) {
                        int idx, s2;
                        if (vox_near(vf, S, px, py, pz, sh.DX[k & 1], sh.DX[2 + ((k >> 1) & 1)], dzc, &idx, &s2)) {
                            const float d0 = __ldg(g.dist + idx);
                            const float dn = (s2 == 0) ? d0 : (float)(__ldg(g.ovl + s2) + (double)d0);
                            if (k == 0) dres[0] = dn; else if (k == 1) dres[1] = dn; else if (k == 2) dres[2] = dn; else dres[3] = dn;
                        } else {
                            const float dn = dt_distance_v<true>(S, g.xMin, g.yMin, g.zMin, g.scale, g.dist, px + sh.HX[k & 1], py + sh.HX[2 + ((k >> 1) & 1)], pz + hz);
                            if (k == 0) dres[0] = dn; else if (k == 1) dres[1] = dn; else if (k == 2) dres[2] = dn; else dres[3] = dn;
                        }
                    }
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    float d = w_i * dres[k];
                    d = d - r_i;
                    if (d < 0.f) d = 0.f;
                    dres[k] = d;
                }
                if (useMd) {
                    if (valid) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) md[(q4 + k) * NdQ + i] = dres[k];
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const float d = valid ? dres[k] : 0.f;
                        float su = (norm == 2) ? d * d : d;
                        const float dis = d - mtd;
                        float sl = (dis > 0.f) ? ((norm == 2) ? dis * dis : dis) : 0.f;
                        su = warp_sum(su); sl = warp_sum(sl);
                        if (lane == 0) { part[2 * ((q4 + k) * nchunks + ch)] = su; part[2 * ((q4 + k) * nchunks + ch) + 1] = sl; }
                    }
                }
            }
            // warp 0 files the memo look-ups issued at the end of the previous pop (the reference memoises corner terms per
            // InnerBnB call too, :304-305)
            if (corners && warp == 0) {
                bool miss = false;
                unsigned mkx = 0, mky = 0, mkz = 0;
                if (lane < 27) {
                    const int cz_ = lane / 9, cy_ = (lane - 9 * cz_) / 3, cx_ = lane - 9 * cz_ - 3 * cy_;
                    const unsigned kx = __float_as_uint(sh.X[cx_]), ky = __float_as_uint(sh.X[3 + (cy_)]), kz = __float_as_uint(sh.X[6 + (cz_)]);
                    mkx = kx; mky = ky; mkz = kz;
                    if (me0.x == kx && me0.y == ky && me0.z == kz && me0.w == sh.gen && me1.z == (kx ^ __funnelshift_l(ky, ky, 11) ^ __funnelshift_l(kz, kz, 22))) { sh.cnt[lane] = (int)me1.x; sh.cf[lane] = __uint_as_float(me1.y); sh.cntN[lane] = (int)me1.w; }
                    else { miss = true; sh.cnt[lane] = 0; }
                }
                const unsigned mm = __ballot_sync(GOICP_FULL, miss);
                if (miss) {   // compact list of the corners to evaluate, with their voxel constants
                    const int m = __popc(mm & ((1u << lane) - 1u));
                    const int cz_ = lane / 9, cy_ = (lane - 9 * cz_) / 3, cx_ = lane - 9 * cz_ - 3 * cy_;
                    sh.missList[m] = lane;
                    const unsigned slot = memo_slot(memo_hash(mkx, mky, mkz), memoShift);   // the entry's key half is written now, its value half after phase A2
                    memo[2 * (size_t)slot] = make_uint4(mkx, mky, mkz, sh.gen);
                    sh.mSlot[m] = slot; sh.mChk[m] = mkx ^ __funnelshift_l(mky, mky, 11) ^ __funnelshift_l(mkz, mkz, 22);
                    sh.mC[m] = sh.CX[cx_]; sh.mC[27 + m] = sh.CX[3 + cy_]; sh.mC[54 + m] = sh.CX[6 + cz_];
                }
                if (lane < 27) { sh.cntM[lane] = 0; sh.cntNM[lane] = 0; }
                if (lane == 0) { sh.nmiss = __popc(mm); sh.workCtr = 0; sh.missTot += __popc(mm); }
            }
            __syncthreads();                                                         // (2)
#ifdef GOICP_PHASE_TIMING
            if (tid == 0) { const long long n_ = clock64(); sh.tp[1] += n_ - sh.tmark; sh.tmark = n_; }
#endif
            // warp 0 brings the queue up to date (the pushes and the pop decided at the end of the previous pop) while warp 1 sums
            // the residuals and the other warps start on the corners
            if (warp == 0 && dPop) {
                uint2 top = make_uint2(0u, 0u);
                if (heapN + dNpush <= HK_SMEM) {
                    for (int r2 = 0; r2 < dNpush; ++r2) heap_siftup_w(s_hkey, heapN + r2, s_pk[r2], lane);
                    top = heap_pop_w(s_hkey, heapN + dNpush, lane);
                } else if (lane == 0) {
                    int n2 = heapN;
                    for (int r2 = 0; r2 < dNpush; ++r2) heap_push(heap, n2, s_pk[r2]);
                    top = heap_pop(heap, n2);
                }
                heapN += dNpush - 1;
                const int sl = (int)(__shfl_sync(GOICP_FULL, top.y, 0) & 0x3FFFFFFu);
                if (sl != predSlot) intErr = 1;                                      // cannot happen (see phase C)
                if (freeTop < HF_SMEM) { if (lane == 0) s_free[freeTop] = sl; freeTop++; }   // (a full stack leaks the slot: `bump` then runs into heapCap and the call is re-run)
                dPop = 0; dNpush = 0;
#ifdef GOICP_PHASE_TIMING
                if (lane == 0) sh.tp[5] += ((heapN > HK_SMEM) ? (1ll << 38) : 0ll) + (heapN >> 4);
                if (tid == 0) sh.tp[10] += clock64() - sh.tmark;
#endif
            }
            if (CANCEL && warp == nwarps - 1 && lane == 0 && cs.word != nullptr && *cs.word != cs.gen) cs.flag = 1;
            // ---- phase A2: warp 0 sums the residuals while the other warps evaluate the corners the memo missed -----------
            if (doTrim) {   // radix select replaces intro_select (:384-390); one warp per child
                for (int c = warp; c < 8; c += nwarps) {
                    float su, sl;
                    warp_trimmed_sums(md + c * NdQ, Nd, inlierNum, lane, norm, mtd, &su, &sl);
                    if (lane == 0) { sh.ub[c] = su; sh.lb[c] = sl; }
                }
            } else if (warp == chainWarp && lane < 16) {
                const int c = lane >> 1;
                float acc = 0.f;
                if (EXACT) {   // sequential float sums in index order (:393-415): lane = (child, ub|lb); 16 independent chains
                    const float sub = (lane & 1) ? mtd : 0.f;   // d - 0 == d and max(d, 0) == d: one code path for both sums
                    const float* m = md + c * NdQ;
                    const float4* m4 = reinterpret_cast<const float4*>(m);
                    const int n4 = inlierNum >> 2;
                    float4 cur = m4[0];
                    for (int k = 0; k < n4; ++k) {
                        const float4 nxt = m4[k + 1];   // rows are padded: the read-ahead stays inside the row
                        float t;
                        t = fmaxf(cur.x - sub, 0.f); acc = acc + ((norm == 2) ? t * t : t);
                        t = fmaxf(cur.y - sub, 0.f); acc = acc + ((norm == 2) ? t * t : t);
                        t = fmaxf(cur.z - sub, 0.f); acc = acc + ((norm == 2) ? t * t : t);
                        t = fmaxf(cur.w - sub, 0.f); acc = acc + ((norm == 2) ? t * t : t);
                        cur = nxt;
                    }
                    for (int i = n4 * 4; i < inlierNum; ++i) { const float t = fmaxf(m[i] - sub, 0.f); acc = acc + ((norm == 2) ? t * t : t); }
                } else {
                    const float* qd = part + 2 * c * nchunks + (lane & 1);
                    for (int k = 0; k < nchunks; ++k) acc = acc + qd[2 * k];
                }
                if (lane & 1) sh.lb[c] = acc; else sh.ub[c] = acc;
#ifdef GOICP_PHASE_TIMING
                if (lane == 0) sh.tp[4] += clock64() - sh.tmark;
#endif
            }
            if (corners) {   // corner terms (:431-550, checkCompatibilities :919, sumFPFH :1689): item = (chunk, half of the missed corners)
                const int nmiss = sh.nmiss;
                const int ngrp = (nmiss + 3) >> 2, ghalf = (ngrp + 1) >> 1;
                for (;;) {
                    int it = 0;
                    if (lane == 0) it = smem_fetch_add(&sh.workCtr, 1);
                    it = __shfl_sync(GOICP_FULL, it, 0);
                    if (it >= 2 * nchunks) break;
                    const int ch = it >> 1;
                    const int g0 = (it & 1) * ghalf, g1 = min(ngrp, g0 + ghalf);
                    const int i = ch * 32 + lane;
                    const bool valid = i < Nd;
                    const float px = valid ? tx[i] : 0.f, py = valid ? ty[i] : 0.f, pz = valid ? tz[i] : 0.f;
                    const unsigned dp = valid ? dprop_s[i] : 0u;
                    for (int gq = g0; gq < g1; ++gq) {
                        // four missed corners per step as independent chains: voxel of the point at each corner ...
                        int vox[4];
                        unsigned flags = 0;
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const int m = min(gq * 4 + k, nmiss - 1);
                            vox[k] = vox_fast(vf, S, px, py, pz, sh.mC[m], sh.mC[27 + m], sh.mC[54 + m]);
                            flags |= (vox[k] < 0 ? 1u : 0u) << k;
                        }
                        unsigned any = __reduce_or_sync(GOICP_FULL, flags);
                        while (any) {   // clamped INTO the grid (checkCompatibility :976-984): near table, else the exact form
                            const int k = __ffs(any) - 1; any &= any - 1;
                            if (flags & (1u << k)) {
                                const int m = min(gq * 4 + k, nmiss - 1);
                                const int c = sh.missList[m];
                                const int cz_ = c / 9, cy_ = (c - 9 * cz_) / 3, cx_ = c - 9 * cz_ - 3 * cy_;
                                int idx, s2;
                                if (!vox_near(vf, S, px, py, pz, sh.mC[m], sh.mC[27 + m], sh.mC[54 + m], &idx, &s2))
                                    idx = clamp_vox_v(S, g.xMin, g.yMin, g.zMin, g.scale, px + sh.X[cx_], py + sh.X[3 + cy_], pz + sh.X[6 + cz_]);
                                if (k == 0) vox[0] = idx; else if (k == 1) vox[1] = idx; else if (k == 2) vox[2] = idx; else vox[3] = idx;
                            }
                        }
                        // ... incompatibility counts (:919-928): one packed warp reduction for the four corners
                        if (use_reg) {
                            unsigned packed = 0;
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                const unsigned mk = GS ? (unsigned)svm[vox[k]] : __ldg(g.vmask + vox[k]);   // per-voxel mask of the closest cell: one gather
                                packed |= (((mk >> dp) & 1u) ^ 1u) << (8 * k);
                            }
                            packed = __reduce_add_sync(GOICP_FULL, valid ? packed : 0u);   // <= 32 per byte field
                            if (lane < 4 && gq * 4 + lane < nmiss) {
                                const unsigned bad = (packed >> (8 * lane)) & 0xFFu;
                                if (bad) smem_red_add(&sh.cntM[gq * 4 + lane], (int)bad);
                            }
                        }
                        if (use_fpfh || use_nb) {   // (CT) terms that need the closest cell itself
                            int cell[4];
#pragma unroll
                            for (int k = 0; k < 4; ++k) cell[k] = __ldg(g.vcell + vox[k]);
                            if (use_fpfh) {   // sumFPFH :1689: per point the min descriptor distance to the cell, tabulated per pair
                                float fv[4];
#pragma unroll
                                for (int k = 0; k < 4; ++k) fv[k] = valid ? __ldg(P.fpfhD + (size_t)i * ncp1 + cell[k]) : 0.f;
#pragma unroll
                                for (int k = 0; k < 4; ++k) {
                                    const int m = gq * 4 + k;
                                    if (m < nmiss) {
                                        if (EXACT) { if (valid) fp[m * NdQ + i] = fv[k]; }
                                        else { const float fs = warp_sum(fv[k]); if (lane == 0) part[16 * nchunks + m * nchunks + ch] = fs; }
                                    }
                                }
                            }
                            if (use_nb) {   // nearestNeighbor inside the closest cell + compareNeighbors (:1200-1211, :1250-1288)
                                for (int k = 0; k < 4; ++k) {
                                    const int m = gq * 4 + k;
                                    if (m >= nmiss) break;
                                    const int c = sh.missList[m];
                                    const int cz_ = c / 9, cy_ = (c - 9 * cz_) / 3, cx_ = c - 9 * cz_ - 3 * cy_;
                                    const int cl = k == 0 ? cell[0] : k == 1 ? cell[1] : k == 2 ? cell[2] : cell[3];
                                    int dn = valid ? nb_diff(P, cl, i, px + sh.X[cx_], py + sh.X[3 + cy_], pz + sh.X[6 + cz_]) : 0;
                                    dn = warp_sum_i(dn);
                                    if (lane == 0 && dn) smem_red_add(&sh.cntNM[m], dn);
                                }
                            }
                        }
                    }
                }
            }
            __syncthreads();                                                         // (3)
#ifdef GOICP_PHASE_TIMING
            if (tid == 0) { const long long n_ = clock64(); sh.tp[2] += n_ - sh.tmark; sh.tmark = n_; }
#endif
            if (warp == 1 && use_fpfh) {   // c-FPFH sums of the missed corners, one chain per lane
                if (lane < sh.nmiss) {
                    float s_ = 0.f;
                    if (EXACT) {   // sumFPFH :1692-1695, sequential in index order
                        const float* f = fp + lane * NdQ; const float4* f4 = reinterpret_cast<const float4*>(f);
                        const int n4 = Nd >> 2;
                        float4 cur = f4[0];
                        for (int k = 0; k < n4; ++k) { const float4 nxt = f4[k + 1]; s_ = s_ + cur.x; s_ = s_ + cur.y; s_ = s_ + cur.z; s_ = s_ + cur.w; cur = nxt; }
                        for (int i = n4 * 4; i < Nd; ++i) s_ = s_ + f[i];
                    }
                    else { const float* f = part + 16 * nchunks + lane * nchunks; for (int k = 0; k < nchunks; ++k) s_ = s_ + f[k]; }
                    sh.cf[sh.missList[lane]] = (float)(int)(s_ / (float)Nd);          // :1696, int truncation :468,:495 (H7)
                }
                __syncwarp();
                asm volatile("bar.sync 1, 64;" ::: "memory");
            }
            if (warp != 0) continue;
            __syncwarp();
            if (use_fpfh) asm volatile("bar.sync 1, 64;" ::: "memory");
            __syncwarp();
            if (corners && lane < sh.nmiss) {   // scatter the fresh counts to their lattice corners and complete their memo entries
                const int c = sh.missList[lane];
                const int n = sh.cntM[lane];
                const int nn = sh.cntNM[lane];
                sh.cnt[c] = n; sh.cntN[c] = nn;
                memo[2 * (size_t)sh.mSlot[lane] + 1] = make_uint4((unsigned)n, use_fpfh ? __float_as_uint(sh.cf[c]) : 0u, sh.mChk[lane], (unsigned)nn);
            }
            __syncwarp();
            // ---- phase C: corner min/max per child on 8 lanes (:431-550), the eight decisions (:554-572) as a prefix-min ----
            const float INF = __int_as_float(0x7f800000);
            const int jx = lane & 1, jy = (lane >> 1) & 1, jz = (lane >> 2) & 1;
            float ubj = INF, lbj = INF;
            if (lane < 8) {
                float ub = sh.ub[lane], lb = sh.lb[lane];
                if (corners) {
                    int minI = 0, maxI = 0, minN = 0, maxN = 0; float minF = 0.f, maxF = 0.f;
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const int c = (jx + (k & 1)) + 3 * (jy + ((k >> 1) & 1)) + 9 * (jz + ((k >> 2) & 1));
                        if (use_nb) { const int n = sh.cntN[c]; if (k == 0) { minN = maxN = n; } else { if (n > maxN) maxN = n; if (n < minN) minN = n; } }
                        if (use_fpfh) { const float f = sh.cf[c]; if (k == 0) { minF = maxF = f; } else { if (f > maxF) maxF = f; if (f < minF) minF = f; } }
                        if (use_reg) { const int n = sh.cnt[c]; if (k == 0) { minI = maxI = n; } else { if (n > maxI) maxI = n; if (n < minI) minI = n; } }
                    }
                    if (use_reg) { ub = ub + regW * (float)(maxI * maxI); lb = lb + regW * (float)(minI * minI); }      // :536-538
                    if (use_nb) { ub = ub + regNW * (float)(maxN * maxN); lb = lb + regNW * (float)(minN * minN); }      // :542-545
                    if (use_fpfh) { ub = ub + regFW * (maxF * maxF); lb = lb + regFW * (minF * minF); }                  // :546-549
                }
                ubj = ub; lbj = lb;
            }
            // optErrorT after child j = min(optErrorT, ub_0..ub_j) (:554-566 takes a strictly smaller ub); child j is pushed
            // unless lb_j >= that value (:568-572)
            float run = ubj;
#pragma unroll
            for (int o = 1; o < 8; o <<= 1) { const float v = __shfl_up_sync(GOICP_FULL, run, o); if (lane >= o) run = fminf(run, v); }
            const float optj = fminf(optT, run);
            float optPrev = __shfl_up_sync(GOICP_FULL, optj, 1); if (lane == 0) optPrev = optT;
            const unsigned impMask = __ballot_sync(GOICP_FULL, lane < 8 && ubj < optPrev);
            const unsigned pushMask = __ballot_sync(GOICP_FULL, lane < 8 && !(lbj >= optj));
            optT = __shfl_sync(GOICP_FULL, optj, 7);
#ifdef GOICP_PHASE_TIMING
            if (tid == 0) sh.tp[8] += clock64() - sh.tmark;
#endif
            // the node's own lattice origin and width (lane j < 8: origin of child j)
            const float ox = sh.X[jx], oy = sh.X[3 + (jy)], oz = sh.X[6 + (jz)];
            const float wc = sh.wc;
            const int lvl = sh.level;
            if (impMask) {   // the last child that lowered optErrorT holds the final value
                const int jb = 31 - __clz(impMask);
                if (lane == jb) { sh.improved = 1; sh.best[0] = ox; sh.best[1] = oy; sh.best[2] = oz; sh.best[3] = wc; }
            }
            // every pushed child takes a payload slot and stages its key.  The queue itself is updated later (after barrier 1,
            // while the other warps already evaluate the next node): the node popped next is known without touching the queue.
            // It is the queue's top T unless a pushed child is strictly better than T, and then the first such child with the
            // smallest lb: __push_heap moves a key up only past strictly worse ancestors, so equal keys stay below older ones.
            const int npush = __popc(pushMask);
            int status = 0, running = 1;
            sh_subcubes += 8;
#ifdef GOICP_PHASE_TIMING
            if (tid == 0) sh.tp[9] += clock64() - sh.tmark;
#endif
            if (heapN + npush > heapCap || bump + npush > heapCap) { status = 4; running = 0; }
            else {
                const bool pushed = (pushMask >> lane) & 1u;
                const int r = __popc(pushMask & ((1u << lane) - 1u));
                int mySlot = 0;
                if (pushed) {
                    mySlot = (r < freeTop) ? s_free[freeTop - 1 - r] : bump + (r - freeTop);
                    heap.setpay(mySlot, make_float4(ox, oy, oz, 0.f));
                    s_pk[r] = make_uint2(__float_as_uint(lbj), ((unsigned)lvl << 26) | (unsigned)mySlot);
                }
                const int fromFree = min(npush, freeTop);
                freeTop -= fromFree; bump += npush - fromFree;
                const unsigned minBits = __reduce_min_sync(GOICP_FULL, pushed ? __float_as_uint(lbj) : 0xFFFFFFFFu);   // lb >= +0: bit order = value order
                const uint2 T = s_hkey[0];
                const bool childBetter = npush > 0 && (heapN == 0 || key_less(T, make_uint2(minBits, (unsigned)lvl << 26)));
                if (!childBetter && heapN == 0) running = 0;                         // queue empty (:314)
                else {
                    float nlb, nx, ny, nz; int plev;
                    if (childBetter) {
                        const int a = __ffs(__ballot_sync(GOICP_FULL, pushed && __float_as_uint(lbj) == minBits)) - 1;
                        nlb = __uint_as_float(minBits); plev = lvl;
                        nx = __shfl_sync(GOICP_FULL, ox, a); ny = __shfl_sync(GOICP_FULL, oy, a); nz = __shfl_sync(GOICP_FULL, oz, a);
                        predSlot = __shfl_sync(GOICP_FULL, mySlot, a);
                    } else {
                        nlb = __uint_as_float(T.x); plev = min((int)(T.y >> 26), MAX_TLEVEL - 1);
                        predSlot = (int)(T.y & 0x3FFFFFFu);
                        const float4 pp = heap.pay(predSlot);
                        nx = pp.x; ny = pp.y; nz = pp.z;
                    }
                    sh_pops++;
                    dNpush = npush; dPop = 1;
                    if (optT - nlb < SSE) running = 0;   // :317
                    else {
                        const float w2 = sh.wtab[plev] / 2;                          // :322
                        // child / corner lattice, voxel-index constants: lane = 3 * axis + k (9 lanes), child-centre forms on lanes 9..14
                        const int a = lane < 9 ? lane / 3 : (lane - 9) >> 1, k = lane < 9 ? lane - 3 * a : (lane - 9) & 1;
                        const float o = a == 0 ? nx : a == 1 ? ny : nz;
                        const double mn = a == 0 ? g.xMin : a == 1 ? g.yMin : g.zMin;
                        float t = o; if (k >= 1) t = o + w2; if (k == 2) t = t + w2;   // X[1] = x + w, X[2] = X[1] + w
                        if (lane < 9) {
                            sh.X[3 * a + k] = t;                                     // X, Y, Z are contiguous
                            sh.CX[3 * a + k] = vox_fast_c(g.vfMagic, t, mn, g.scale);
                        } else if (lane < 15) {
                            const float th = t + w2 / 2;                             // :331-333
                            sh.HX[2 * a + k] = th;
                            sh.DX[2 * a + k] = vox_fast_c(g.vfMagic, th, mn, g.scale);
                        } else if (lane == 15) {
                            sh.wc = w2; sh.level = min(plev + 1, MAX_TLEVEL - 1);
                            sh.mtd = (float)(GOICP_SQRT3 / 2.0 * w2);                // :323
                            sh.workA = 0;
                        }
                        if (corners && lane < 27) {   // corner-memo look-ups of the next node, consumed after its phase A1
                            const int cz_ = lane / 9, cy_ = (lane - 9 * cz_) / 3, cx_ = lane - 9 * cz_ - 3 * cy_;
                            float cxv = nx; if (cx_ >= 1) cxv = nx + w2; if (cx_ == 2) cxv = cxv + w2;
                            float cyv = ny; if (cy_ >= 1) cyv = ny + w2; if (cy_ == 2) cyv = cyv + w2;
                            float czv = nz; if (cz_ >= 1) czv = nz + w2; if (cz_ == 2) czv = czv + w2;
                            const unsigned hsh = memo_hash(__float_as_uint(cxv), __float_as_uint(cyv), __float_as_uint(czv));
                            const uint4* e = memo + 2 * (size_t)memo_slot(hsh, memoShift);
                            me0 = e[0]; me1 = e[1];
                        }
                    }
                }
            }
            if (CANCEL && running && *reinterpret_cast<volatile int*>(&cs.flag)) { running = 0; status = 7; }   // the owner of this (speculative) call has moved on
            if (lane == 0) { sh.running = running; sh.status = status; }
        }
        if (tid == 0) {
            if (intErr) sh.status = 6;
            if (cpart == 0) {
                InnerOut o;
                o.err = optT; o.node[0] = sh.best[0]; o.node[1] = sh.best[1]; o.node[2] = sh.best[2]; o.node[3] = sh.best[3];
                o.improved = sh.improved; o.pops = sh_pops; o.subcubes = sh_subcubes; o.status = sh.status;
                o.seq0 = o.seq1 = 1u; o.err2 = 0.f; o.pops2 = 0; o.subcubes2 = 0; o.ran2 = 0; o.pad = 0;
                s_out = o;
            } else {
                s_out.err2 = optT; s_out.pops2 = sh_pops; s_out.subcubes2 = sh_subcubes; s_out.ran2 = 1; s_out.status = sh.status;
            }
            atomicAdd(&ctr->pops, (unsigned long long)sh_pops); atomicAdd(&ctr->calls, 1ull);
        }
        }   // cpart
        if (tid == 0) {
            atomicAdd(&ctr->callCycles, (unsigned long long)(clock64() - sh.t0)); atomicAdd(&ctr->cornerMisses, (unsigned long long)sh.missTot);
#ifdef GOICP_PHASE_TIMING
            for (int k = 0; k < 12; k++) atomicAdd(&ctr->phaseCycles[k], (unsigned long long)sh.tp[k]);
#endif
        }
    }
}

}  // namespace
