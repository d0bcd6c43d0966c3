// Pipelined scheme of the "octant" formulation of the fused FactMixer core: ONE persistent launch per direction
// (reference factorizer/factorizer.py:41-50: reshape -> ReLU -> NMF -> inverse reshape, and its adjoint).
//
// The three passes of fz_swnmf_octant.cuh (pass 1: per-octant sums of every tile; pass 2: per-window 8-vector
// recursion; pass 3: per-voxel output) need the volume twice.  As three launches the second read comes from HBM
// again (1.55x / 1.70x the compulsory traffic forward / backward).  Here the passes run as a self-timed pipeline over
// PLANE-GROUPS of tiles (PipeGeom in fz_swnmf_octant.cuh): a shifted window only reaches into the tile planes
// t0 - 1 and t0, so pass 3 of a plane can follow pass 1 at a distance of a few planes, and finds its tiles in L2.
//
// Three global queues, each claimed in order with atomicAdd:
//   pass 1 queue   tiles of plane-group 0, 1, 2, ...                       (claimed by the producers)
//   pass 3 queue   tiles of plane-group 1, 2, ..., and each gang's first-read plane last   (claimed by the producers)
//   pass 2 queue   per plane-group: its unshifted windows, and the shifted window plane it completes  (solver warps)
// and per plane-group completion counters for each of them.  Inside a CTA (12 warps, fixed roles):
//   producer   one warp.  Feeds a ring of tile slots in shared memory: claims pass 1 / pass 3 positions, and issues an
//              item only when it can run to completion -- pass 3 when the solve steps it needs are complete, pass 1 when
//              it is at most `lead` plane-groups ahead of the completed pass 3 (that bound is what keeps the tiles in
//              L2) -- with one TMA box for the tile and small bulk copies for the window records the item needs.
//   consumers  take the slots in ring order, wait for the slot's mbarrier, compute from shared memory, release the slot.
//              They never wait for anything else, so a slot cannot be held by an item that depends on a later one.
//   solvers    run pass 2 items (4 windows x 8 lanes); few registers (setmaxnreg), latency hidden by their number.
//   watcher    one thread: polls the completion counters (acquire, gpu scope) and republishes "every step below k is
//              complete" in shared memory (release, cta scope), so a dependency test is one shared-memory load.
// Every dependency points to an EARLIER position of a queue and positions are claimed in order by warps that are
// running, so the earliest unfinished item can always proceed: no deadlock, no co-residency requirement.
// Completion is published with red.release.gpu after a __syncwarp (the item's stores are ordered before it); readers
// fetch what it guards from L2 only (bulk copies / ld.global.cg).
#include "fz_swnmf_octant.cuh"

namespace fz {
using namespace oct;
namespace {

constexpr int kThreads = 384;         // three warpgroups
constexpr int kFwdSlots = 13;
constexpr int kFwdSide = 9 * kFacF;                    // floats per slot beside the tile: the nine windows' factors
constexpr int kFwdSlotFloats = 4096;
constexpr int kBwdSlots = 6;
constexpr int kBwdSide = 9 * kMbF;                     // the nine windows' records (pass 3) / their u_T (pass 1)
constexpr int kBwdSlotFloats = 8192;

__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void red_release_gpu(int* p, int v) {
    asm volatile("red.release.gpu.global.add.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void red_relaxed_gpu(int* p, int v) {
    asm volatile("red.relaxed.gpu.global.add.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// known[] (shared memory): the watcher's "every step below k is complete" for pass 1, pass 2, pass 3.  A look is a
// relaxed load; whoever finds its step complete passes an acquire fence (cta scope: cheap) before relying on it.
__device__ __forceinline__ int peek_known(const int* p) {
    int v;
    asm volatile("ld.relaxed.cta.shared::cta.s32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
    return v;
}
__device__ __forceinline__ void acquire_cta() { asm volatile("fence.acq_rel.cta;" ::: "memory"); }
__device__ __forceinline__ void st_known(int* p, int v) {
    asm volatile("st.release.cta.shared::cta.s32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory");
}
// blocking: one lane polls (sleeping in between: the shared-memory pipe belongs to the consumers)
__device__ __forceinline__ void wait_known(const int* p, int need, int lane) {
    if (lane == 0) {
        while (peek_known(p) < need) __nanosleep(200);
        acquire_cta();
    }
    __syncwarp();
}
// L2 eviction priorities (createpolicy): pass 1 reads a tile that pass 3 will want again, pass 3 reads it for the last time
__device__ __forceinline__ uint64_t policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}

#ifdef FZ_TUNING
__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// item log of CTA 0 (experiment builds): 4 timestamps + kind per item, solver warp at [0, 256), consumer 0 at [256, 512)
#define FZ_LOG(G, base, idx, a, b, c, d, kind)                                                             \
    do {                                                                                                   \
        if ((G).trace && blockIdx.x == 0 && lane == 0 && (idx) < 50) {                                     \
            unsigned long long* L = (G).trace + 3 * ((G).NP + 1) + ((base) + (idx)) * 5;                   \
            L[0] = a; L[1] = b; L[2] = c; L[3] = d; L[4] = kind;                                           \
        }                                                                                                  \
    } while (0)
#else
#define FZ_LOG(G, base, idx, a, b, c, d, kind) do {} while (0)
__device__ __forceinline__ unsigned long long gtime() { return 0; }
#endif

// ---- queue decoding -------------------------------------------------------------------------------------
// tile `idx` of plane-group (gang, pos)
__device__ __forceinline__ void plane_tile(const PhaseParams& P, int gang, int pos, int idx, TileCoord& c) {
    const PipeGeom& G = P.pipe;
    int svg, t1, t2;
    if (P.pow2) {
        t2 = idx & (P.G2 - 1); idx >>= P.s2;
        t1 = idx & (P.G1 - 1); svg = idx >> P.s1;
    } else {
        svg = idx / G.per_plane;
        const int rem = idx - svg * G.per_plane;
        t1 = rem / P.G2; t2 = rem - t1 * P.G2;
    }
    const int sv = (gang << G.gs_shift) + svg;
    if (P.pow2) { c.b = sv >> P.sh; c.h = sv & (P.heads - 1); }
    else { c.b = sv / P.heads; c.h = sv - c.b * P.heads; }
    c.t0 = pos == 0 ? P.G0 - 1 : pos - 1;
    c.t1 = t1; c.t2 = t2;
}

// What a slot holds.  kind: 0 = pass 1 tile, 1 = pass 3 tile, 3 = end of the stream; pos = place of the plane in its gang
struct alignas(16) Desc { int kind, J, b, h, t0, t1, t2, pos; };

// Position q of the pass 1 queue (is_c = 0: plane-group J = q / nA, tile q % nA) or of the pass 3 queue (is_c = 1:
// step Jc = 1 + q / nA; a step with pos 0 is the first-read plane of the PREVIOUS gang).  False past the end.
__device__ __forceinline__ bool decode_position(const PhaseParams& P, int q, int is_c, int step_shift, Desc& d) {
    const PipeGeom& G = P.pipe;
    if (q >= G.NP * G.nA) return false;
    int K, idx;
    if (step_shift >= 0) { K = q >> step_shift; idx = q & ((1 << step_shift) - 1); }
    else { K = q / G.nA; idx = q - K * G.nA; }
    const int J = is_c ? K + 1 : K;
    int gang, pos;
    if (P.pow2) { gang = J >> P.s0; pos = J & (P.G0 - 1); }
    else { gang = J / P.G0; pos = J - gang * P.G0; }
    if (is_c && pos == 0) gang -= 1;
    TileCoord c;
    plane_tile(P, gang, pos, idx, c);
    d.kind = is_c; d.J = J; d.b = c.b; d.h = c.h; d.t0 = c.t0; d.t1 = c.t1; d.t2 = c.t2; d.pos = pos;
    return true;
}

// pass 3 step Jc needs solve steps Jc and Jc + 1 (its own windows and the shifted plane above)
__device__ __forceinline__ int need_b_for_apply(const PipeGeom& G, int Jc) { return (Jc + 1 < G.NP ? Jc + 1 : G.NP) + 1; }
// pass 1 of plane-group J overwrites the record slot last used `ring` (for a gang's first-read plane: one gang) earlier
__device__ __forceinline__ int need_b_for_gram(const PhaseParams& P, int J, int pos) {
    return pos == 0 ? J - P.G0 + 1 : J - P.pipe.ring + 2;
}

// queue positions in chunks: one atomicAdd per kChunk positions, the next chunk's claim in flight meanwhile
constexpr int kChunk = 4;
struct Claimer {
    int* ctr;
    int claimed, base, left, lane;
    __device__ __forceinline__ void start(int* c, int l, bool used = true) {
        ctr = c; lane = l; left = 0; base = 0; claimed = 0;
        if (lane == 0 && used) claimed = atomicAdd(ctr, kChunk);
    }
    __device__ __forceinline__ int next() {
        if (left == 0) {
            base = __shfl_sync(0xffffffffu, claimed, 0);
            left = kChunk;
            if (lane == 0) claimed = atomicAdd(ctr, kChunk);
        }
        --left;
        return base++;
    }
};

// ---- the watcher: one thread per CTA ----------------------------------------------------------------------
// ctr layout: [0] pass 1 queue head | [1] pass 2 queue head | [2] pass 3 queue head | [3] pad |
//             done_a[NP] | done_b[NP + 1] | done_c[NP + 1] (index = step Jc, 1 .. NP)
__device__ __forceinline__ int* done_a_of(const PipeGeom& G) { return G.ctr + 4; }
__device__ __forceinline__ int* done_b_of(const PipeGeom& G) { return G.ctr + 4 + G.NP; }
__device__ __forceinline__ int* done_c_of(const PipeGeom& G) { return G.ctr + 4 + 2 * G.NP + 1; }

// One warp: lanes 0-7 look at the next eight pass 1 counters, 8-15 at the next eight pass 2 counters, 16-23 at pass 3,
// all with one acquire load each, so every round (one L2 round trip) can advance each prefix by up to eight steps.
__device__ __forceinline__ void watch(const PhaseParams& P, int* known, int lane) {
    const PipeGeom& G = P.pipe;
    const int *done_a = done_a_of(G), *done_b = done_b_of(G), *done_c = done_c_of(G);
    int ka = 0, kb = 0, kc = 0;          // complete: pass 1 steps < ka, pass 2 steps < kb, pass 3 steps <= kc
    const int which = lane >> 3, ofs = lane & 7;
    while (ka < G.NP || kb <= G.NP || kc < G.NP) {
        bool complete = false;
        if (which == 0) {
            const int k = ka + ofs;
            if (k < G.NP) complete = ld_acquire_gpu(done_a + k) >= G.nA;
        } else if (which == 1) {
            const int k = kb + ofs;
            if (k <= G.NP) complete = ld_acquire_gpu(done_b + k) >= G.nBset * ((k < G.NP ? 1 : 0) + (k >= 1 ? 1 : 0));
        } else if (which == 2) {
            const int k = kc + ofs;
            if (k < G.NP) complete = ld_acquire_gpu(done_c + k + 1) >= G.nA;
        }
        const unsigned m = __ballot_sync(0xffffffffu, complete);
        // leading run of complete steps in each group of eight lanes
        const int na = __ffs(~(m & 0xffu)) - 1, nb = __ffs(~((m >> 8) & 0xffu)) - 1, nc = __ffs(~((m >> 16) & 0xffu)) - 1;
        if (lane == 0) {
            if (na > 0) st_known(&known[0], ka + na);
            if (nb > 0) st_known(&known[1], kb + nb);
            if (nc > 0) st_known(&known[2], kc + nc);
#ifdef FZ_TUNING
            if (G.trace && blockIdx.x == 0) {       // when CTA 0 saw each prefix advance (ns, globaltimer)
                unsigned long long t;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
                for (int q = 0; q < na; ++q) G.trace[ka + q] = t;
                for (int q = 0; q < nb; ++q) G.trace[G.NP + 1 + kb + q] = t;
                for (int q = 0; q < nc; ++q) G.trace[2 * (G.NP + 1) + kc + q] = t;
            }
#endif
        }
        ka += na; kb += nb; kc += nc;
        if (na + nb + nc == 0) __nanosleep(64);
    }
}

// ---- solver warps: pass 2 items ------------------------------------------------------------------------------
// Solve step Jb: set 0 = the unshifted windows of plane-group Jb; set 1 = the shifted window plane that plane-group Jb
// completes (for the first-read plane of a gang: the wrap-around plane of the PREVIOUS gang).  Returns false past the end.
struct SItem { int valid, Jb, set, gang, pos, batch; };
__device__ __forceinline__ bool decode_solve_item(const PhaseParams& P, int q, SItem& it) {
    const PipeGeom& G = P.pipe;
    if (q >= G.solve_items) return false;
    const int per = 2 * G.nBset;
    it.Jb = q / per;
    const int r = q - it.Jb * per;
    it.set = r >= G.nBset ? 1 : 0;
    it.batch = r - it.set * G.nBset;
    it.gang = it.Jb / P.G0;
    it.pos = it.Jb - it.gang * P.G0;
    it.valid = it.set ? (it.Jb >= 1) : (it.Jb < G.NP);
    if (it.set && it.pos == 0) it.gang -= 1;
    return true;
}
// canonical window index of window `wl` of the item's plane, or -1
__device__ __forceinline__ long long solve_window(const PhaseParams& P, const SItem& it, int wl) {
    if (!it.valid || wl >= P.pipe.nA) return -1;
    TileCoord c;
    plane_tile(P, it.gang, it.pos, wl, c);
    return (long long)it.set * P.tiles + tile_index(P, c);
}

template <bool BWD>
__device__ __forceinline__ void solve_loop(const PhaseParams& P, float* scratch, const int* known, float b1, int lane, int log_items = -1) {
    const PipeGeom& G = P.pipe;
    int* done_b = done_b_of(G);
    int claimed = 0;
    if (lane == 0) claimed = atomicAdd(G.ctr + 1, 1);
    for (;;) {
        const int q = __shfl_sync(0xffffffffu, claimed, 0);
        SItem it;
        if (!decode_solve_item(P, q, it)) break;
        if (lane == 0) claimed = atomicAdd(G.ctr + 1, 1);       // the next item's position arrives while this one runs
        if (!it.valid) continue;
        const unsigned long long t0 = gtime();
        wait_known(&known[0], it.Jb + 1 < G.NP ? it.Jb + 1 : G.NP, lane);
        const unsigned long long t1 = gtime();
        long long gwin = solve_window(P, it, it.batch * 4 + (lane >> 3));
        const bool active = gwin >= 0;
        if (!active) gwin = solve_window(P, it, it.batch * 4);       // the batch's first window always exists
        if (BWD) bwd_solve_window(P, reinterpret_cast<float(*)[kBwdOct]>(scratch + (lane >> 3) * 8 * kBwdOct), gwin, it.set, lane, active);
        else fwd_solve_window(P, scratch + (lane >> 3) * 64, gwin, it.set, lane, active, b1);
        __syncwarp();
        const unsigned long long t2 = gtime();
        if (lane == 0) red_release_gpu(done_b + it.Jb, 1);
        if (log_items >= 0) { FZ_LOG(G, 0, log_items, t0, t1, t2, gtime(), it.Jb); ++log_items; }
    }
}

// ---- the producer warp ---------------------------------------------------------------------------------------
// SLOTS ring slots of SLOT_FLOATS floats (tile[s]) + SIDE floats (window records); BWD: the tile is X | dY.
template <bool BWD, int SLOTS, int SLOT_FLOATS, int SIDE, int CONSUMERS>
__device__ __forceinline__ void produce(const PhaseParams& P, float* tiles, float* side, Desc* descs, uint64_t* full,
                                        uint64_t* empty, const int* known, int lane, int role) {
    const PipeGeom& G = P.pipe;
    int step_shift = -1;
    if ((G.nA & (G.nA - 1)) == 0) { step_shift = 0; while ((1 << step_shift) < G.nA) ++step_shift; }
    const uint64_t pol_keep = policy_evict_last(), pol_last = policy_evict_first();
    Claimer qa, qc;
    qa.start(G.ctr, lane, role == 0);
    qc.start(G.ctr + 2, lane, role == 1);
    Desc da, dc;
    bool have_a = false, have_c = false, end_a = false, end_c = false;
    if (role == 0) end_c = true; else end_a = true;       // this CTA's pass only (cta_role)
    int seq = 0;
    bool prefer_c = false;
    for (;;) {
        if (!have_a && !end_a) { have_a = decode_position(P, qa.next(), 0, step_shift, da); end_a = !have_a; }
        if (!have_c && !end_c) { have_c = decode_position(P, qc.next(), 1, step_shift, dc); end_c = !have_c; }
        if (!have_a && !have_c) break;
        // an item goes into the ring only when it can run to completion
        const int kb = peek_known(&known[1]), kc = peek_known(&known[2]);
        const bool c_ok = have_c && kb >= need_b_for_apply(G, dc.J);
        const bool a_ok = have_a && kc >= da.J - G.lead && kb >= need_b_for_gram(P, da.J, da.pos);
        if (!c_ok && !a_ok) { __nanosleep(64); continue; }
        acquire_cta();
        const bool take_c = c_ok && (prefer_c || !a_ok);
        prefer_c = !take_c;
        const Desc d = take_c ? dc : da;
        if (take_c) have_c = false; else have_a = false;

        const int slot = seq % SLOTS;
        mbar_wait(&empty[slot], ((seq / SLOTS) & 1) ^ 1);
        ++seq;
        float* tile = tiles + (size_t)slot * SLOT_FLOATS;
        float* sd = side + (size_t)slot * SIDE;
        TileCoord c;
        c.b = d.b; c.h = d.h; c.t0 = d.t0; c.t1 = d.t1; c.t2 = d.t2;
        const int tid = tile_index(P, c);
        // which small records ride along: forward pass 3 -> the nine windows' factors; backward pass 1 -> their u_T;
        // backward pass 3 -> their pass 2 records.  Lane w (0 .. 8) copies window w's.
        const float* src = nullptr;
        uint32_t rec_bytes = 0;
        if (lane < 9) {
            const long long wid = lane == 0 ? (long long)tid : (long long)P.tiles + shifted_window_of(P, c, lane - 1);
            if (!BWD) {
                if (d.kind == 1) { src = P.fac + wid * kFacF; rec_bytes = kFacF * 4; }
            } else if (d.kind == 0) {
                src = P.saved + wid * P.rec_floats + 8 * (P.T - 1); rec_bytes = 32;
            } else {
                src = P.mb + wid * kMbF; rec_bytes = kMbF * 4;
            }
        }
        if (lane == 0) {
            *reinterpret_cast<int4*>(&descs[slot]) = make_int4(d.kind, d.J, d.b, d.h);
            *(reinterpret_cast<int4*>(&descs[slot]) + 1) = make_int4(d.t0, d.t1, d.t2, d.pos);
            const uint32_t tile_bytes = (BWD ? 2 : 1) * kTileBytes;
            const uint32_t side_bytes = BWD ? 9u * (d.kind == 0 ? 32u : kMbF * 4u) : (d.kind == 1 ? 9u * kFacF * 4u : 0u);
            mbar_arrive_expect_tx(&full[slot], tile_bytes + side_bytes);
            // a gang's first-read plane is not needed again before the gang ends: no point asking L2 to keep it
            const bool keep = d.kind == 0 && d.pos != 0 && (G.flags & 1), last = d.kind == 1 && (G.flags & 2);
            if (keep || last) {
                const uint64_t pol = keep ? pol_keep : pol_last;
                tma_load_tile_hint(tile, &P.tm_x, &full[slot], c.t2 * 8, c.t1 * 8, c.t0 * 8, c.h * 8, c.b, pol);
                if (BWD) tma_load_tile_hint(tile + 4096, &P.tm_g, &full[slot], c.t2 * 8, c.t1 * 8, c.t0 * 8, c.h * 8, c.b, pol);
            } else {
                tma_load_tile(tile, &P.tm_x, &full[slot], c.t2 * 8, c.t1 * 8, c.t0 * 8, c.h * 8, c.b);
                if (BWD) tma_load_tile(tile + 4096, &P.tm_g, &full[slot], c.t2 * 8, c.t1 * 8, c.t0 * 8, c.h * 8, c.b);
            }
        }
        __syncwarp();
        if (rec_bytes) bulk_copy(sd + lane * (rec_bytes / 4), src, rec_bytes, &full[slot]);
    }
    // one end-of-stream marker per consumer
    for (int k = 0; k < CONSUMERS; ++k) {
        const int slot = seq % SLOTS;
        mbar_wait(&empty[slot], ((seq / SLOTS) & 1) ^ 1);
        ++seq;
        if (lane == 0) {
            *reinterpret_cast<int4*>(&descs[slot]) = make_int4(3, 0, 0, 0);
            mbar_arrive(&full[slot]);
        }
        __syncwarp();
    }
}

// ---- CTA roles -----------------------------------------------------------------------------------------------------
// An SM's instruction cache is 32 KiB and the three tile / window routines together are several times that, so every CTA
// runs ONE of them (its role, from blockIdx): pass 1 CTAs and pass 3 CTAs are a producer warp, a watcher warp and eight
// consumer warps around a ring of tile slots; solver CTAs are a watcher and eleven solver warps.
enum { kRoleGram = 0, kRoleApply = 1, kRoleSolve = 2 };
__device__ __forceinline__ int cta_role(const PipeGeom& G) {
    const int r = (int)blockIdx.x % G.role_period;
    return r < G.role_solve ? kRoleSolve : (r < G.role_solve + G.role_gram ? kRoleGram : kRoleApply);
}
constexpr int kConsumers = 8;         // warps 4-11 of a pass 1 / pass 3 CTA
// A consumer may only wait for the current or the previous phase of a slot's mbarrier, so the consumers -- who take
// consecutive sequence numbers -- must be fewer than the slots: the backward (6 slots of 32 KiB) runs 5 of them.
constexpr int kBwdActive = 5;
static_assert(kConsumers < kFwdSlots && kBwdActive < kBwdSlots, "consumers must not lap the ring");

struct RingShared {
    uint64_t full[kFwdSlots], empty[kFwdSlots];
    Desc descs[kFwdSlots];
    int known[4];
    int next_seq;
};
__device__ __forceinline__ void ring_init(RingShared& R, int slots) {
    R.known[0] = R.known[1] = R.known[2] = 0;
    R.next_seq = 0;
    for (int s = 0; s < slots; ++s) { mbar_init(&R.full[s], 1); mbar_init(&R.empty[s], 1); }
    fence_mbarrier_init();
}
// next slot of the ring for a consumer warp: its sequence number's slot, once the producer's data has landed; false at
// the end of the stream
template <int SLOTS>
__device__ __forceinline__ bool ring_next(RingShared& R, int lane, int& slot, int4& d0, int4& d1) {
    int n = 0;
    if (lane == 0) n = atomicAdd(&R.next_seq, 1);
    n = __shfl_sync(0xffffffffu, n, 0);
    slot = n % SLOTS;
    mbar_wait(&R.full[slot], (n / SLOTS) & 1);
    d0 = *reinterpret_cast<const int4*>(&R.descs[slot]);
    if (d0.x == 3) return false;
    d1 = *(reinterpret_cast<const int4*>(&R.descs[slot]) + 1);
    return true;
}

// ---- forward --------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 1) pipe_fwd(const __grid_constant__ PhaseParams P) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(16) float v0s[512];
    __shared__ __align__(16) float side[kFwdSlots * kFwdSide];
    __shared__ RingShared R;
    __shared__ float b1s;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const PipeGeom& G = P.pipe;
    const int role = cta_role(G);
    float* tiles = reinterpret_cast<float*>(smem_raw);

    for (int j = threadIdx.x; j < 512; j += blockDim.x) v0s[j] = P.v0[j];
    if (threadIdx.x == 0) ring_init(R, kFwdSlots);
    __syncthreads();

    if (role == kRoleSolve) {
        if (warp == 0) { watch(P, R.known, lane); return; }
        // b_1 = v_0 . v_0 is the same for every window
        float sq = 0.f;
        for (int j = lane; j < 512; j += 32) sq = fmaf(v0s[j], v0s[j], sq);
        sq = warp_sum_f(sq);
        // the window sums live where the other roles keep their tile ring
        solve_loop<false>(P, tiles + (size_t)(warp - 1) * 4 * 64, R.known, sq, lane, warp == 1 ? 0 : -1);
        return;
    }
    if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 88;");
        if (warp == 0) produce<false, kFwdSlots, kFwdSlotFloats, kFwdSide, kConsumers>(P, tiles, side, R.descs, R.full, R.empty, R.known, lane, role);
        else if (warp == 1) watch(P, R.known, lane);
        return;
    }
    // registers move within the CTA only: 88 + 2 x 208 = 3 x 168, the launch allocation of the three warpgroups
    asm volatile("setmaxnreg.inc.sync.aligned.u32 208;");
    int slot;
    int4 d0, d1;
    if (role == kRoleGram) {
        int* done_a = done_a_of(G);
        int dst[15];
        gram_destinations(lane, dst);
        while (ring_next<kFwdSlots>(R, lane, slot, d0, d1)) {
            TileCoord c;
            c.b = d0.z; c.h = d0.w; c.t0 = d1.x; c.t1 = d1.y; c.t2 = d1.z;
            fwd_tile_gram(tiles + (size_t)slot * kFwdSlotFloats, v0s, dst, lane, P.oct + (size_t)rec_slot(P, c) * kTileRec);
            __syncwarp();
            if (lane == 0) { mbar_arrive(&R.empty[slot]); red_release_gpu(done_a + d0.y, 1); }
        }
    } else {
        int* done_c = done_c_of(G);
        const int oct = lane >> 2;
        while (ring_next<kFwdSlots>(R, lane, slot, d0, d1)) {
            TileCoord c;
            c.b = d0.z; c.h = d0.w; c.t0 = d1.x; c.t1 = d1.y; c.t2 = d1.z;
            const float* sd = side + slot * kFwdSide;
            Fac f0, f1;
            {
                const float4* a = reinterpret_cast<const float4*>(sd);
                const float4* b = reinterpret_cast<const float4*>(sd + (1 + oct) * kFacF);
                const float4 a0 = a[0], a1 = a[1], a2 = a[2], b0 = b[0], b1 = b[1], b2 = b[2];
                f0.u[0] = a0.x; f0.u[1] = a0.y; f0.u[2] = a0.z; f0.u[3] = a0.w; f0.u[4] = a1.x; f0.u[5] = a1.y; f0.u[6] = a1.z; f0.u[7] = a1.w; f0.rd = a2.x;
                f1.u[0] = b0.x; f1.u[1] = b0.y; f1.u[2] = b0.z; f1.u[3] = b0.w; f1.u[4] = b1.x; f1.u[5] = b1.y; f1.u[6] = b1.z; f1.u[7] = b1.w; f1.rd = b2.x;
            }
            fwd_tile_apply<true, true>(P, tiles + (size_t)slot * kFwdSlotFloats, f0, f1, c, lane);
            __syncwarp();
            if (lane == 0) { mbar_arrive(&R.empty[slot]); red_relaxed_gpu(done_c + d0.y, 1); }
        }
    }
}

// ---- backward -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 1) pipe_bwd(const __grid_constant__ PhaseParams P) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(16) float v0s[512];
    __shared__ __align__(16) float side[kBwdSlots * kBwdSide];
    __shared__ RingShared R;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const PipeGeom& G = P.pipe;
    const int role = cta_role(G);
    float* tiles = reinterpret_cast<float*>(smem_raw);

    for (int j = threadIdx.x; j < 512; j += blockDim.x) v0s[j] = P.v0[j];
    if (threadIdx.x == 0) ring_init(R, kBwdSlots);
    __syncthreads();

    if (role == kRoleSolve) {
        if (warp == 0) { watch(P, R.known, lane); return; }
        solve_loop<true>(P, tiles + (size_t)(warp - 1) * 4 * 8 * kBwdOct, R.known, 0.f, lane, warp == 1 ? 0 : -1);
        return;
    }
    if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
        if (warp == 0) produce<true, kBwdSlots, kBwdSlotFloats, kBwdSide, kBwdActive>(P, tiles, side, R.descs, R.full, R.empty, R.known, lane, role);
        else if (warp == 1) watch(P, R.known, lane);
        return;
    }
    asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");      // 56 + 2 x 224 = 3 x 168
    if (warp - 4 >= kBwdActive) return;
    int slot;
    int4 d0, d1;
    if (role == kRoleGram) {
        int* done_a = done_a_of(G);
        const int oct = lane >> 2;
        while (ring_next<kBwdSlots>(R, lane, slot, d0, d1)) {
            TileCoord c;
            c.b = d0.z; c.h = d0.w; c.t0 = d1.x; c.t1 = d1.y; c.t2 = d1.z;
            const float* sd = side + slot * kBwdSide;
            UT f0, f1;
            {
                const float4* a = reinterpret_cast<const float4*>(sd);
                const float4* b = reinterpret_cast<const float4*>(sd + (1 + oct) * 8);
                const float4 a0 = a[0], a1 = a[1], b0 = b[0], b1 = b[1];
                f0.u[0] = a0.x; f0.u[1] = a0.y; f0.u[2] = a0.z; f0.u[3] = a0.w; f0.u[4] = a1.x; f0.u[5] = a1.y; f0.u[6] = a1.z; f0.u[7] = a1.w;
                f1.u[0] = b0.x; f1.u[1] = b0.y; f1.u[2] = b0.z; f1.u[3] = b0.w; f1.u[4] = b1.x; f1.u[5] = b1.y; f1.u[6] = b1.z; f1.u[7] = b1.w;
                // rd_T with the instruction sequence of load_ut (bit-equal to the three-launch scheme)
                float d = f0.u[0] * f0.u[0], e = f1.u[0] * f1.u[0];
#pragma unroll
                for (int j = 1; j < 8; ++j) { d = fmaf(f0.u[j], f0.u[j], d); e = fmaf(f1.u[j], f1.u[j], e); }
                f0.rd = rcp_nr(d + P.eps);
                f1.rd = rcp_nr(e + P.eps);
            }
            bwd_tile_reduce(P, tiles + (size_t)slot * kBwdSlotFloats, f0, f1, lane, P.oct + (size_t)rec_slot(P, c) * kBwdTileRec);
            __syncwarp();
            if (lane == 0) { mbar_arrive(&R.empty[slot]); red_release_gpu(done_a + d0.y, 1); }
        }
    } else {
        int* done_c = done_c_of(G);
        while (ring_next<kBwdSlots>(R, lane, slot, d0, d1)) {
            TileCoord c;
            c.b = d0.z; c.h = d0.w; c.t0 = d1.x; c.t1 = d1.y; c.t2 = d1.z;
            bwd_tile_apply<true>(P, tiles + (size_t)slot * kBwdSlotFloats, side + slot * kBwdSide, v0s, c, lane);
            __syncwarp();
            if (lane == 0) { mbar_arrive(&R.empty[slot]); red_relaxed_gpu(done_c + d0.y, 1); }
        }
    }
}

// ---- host ----------------------------------------------------------------------------------------------------
struct Plan { PipeGeom g; size_t off_oct, off_fac, off_mb, off_trace, ctr_bytes, total; };

Plan make_plan(const DevGeom& G) {
    Plan pl;
    memset(&pl, 0, sizeof(pl));
    PipeGeom& g = pl.g;
    const int svs = G.B * G.heads, per_plane = G.g[1] * G.g[2];
    int group_tiles = 256, lead_tiles = 3072, flags = 7;
#ifdef FZ_TUNING            // experiment builds only (bench_probes/); the shipped library has no environment knobs
    if (const char* e = getenv("FZ_PIPE_GROUP")) group_tiles = atoi(e);
    if (const char* e = getenv("FZ_PIPE_LEAD")) lead_tiles = atoi(e);
    if (const char* e = getenv("FZ_PIPE_FLAGS")) flags = atoi(e);
    if (const char* e = getenv("FZ_PIPE_ROLES")) sscanf(e, "%d,%d,%d", &g.role_period, &g.role_solve, &g.role_gram);
#endif
    // a gang: the largest power-of-two divisor of the sub-volume count that keeps a plane-group at or below group_tiles
    int gs = 1;
    while (svs % (2 * gs) == 0 && 2 * gs * per_plane <= group_tiles) gs *= 2;
    g.enabled = 1;
    g.gs = gs; g.gs_shift = 0;
    while ((1 << g.gs_shift) < gs) ++g.gs_shift;
    g.per_plane = per_plane;
    g.nA = gs * per_plane;
    g.nBset = (g.nA + 3) / 4;
    g.NP = (svs / gs) * G.g[0];
    // pass 1 may run this many plane-groups ahead of the completed pass 3: lead_tiles tiles = 16 KiB each of X (and of
    // dY) that have to stay in L2, and at least 3 so that the pipeline can fill
    int lead = (lead_tiles + g.nA - 1) / g.nA;
    if (lead < 3) lead = 3;
    g.lead = lead;
    g.ring = 4;
    while (g.ring < lead + 3) g.ring *= 2;
    g.flags = flags;
    // of every role_period consecutive CTAs: role_solve run pass 2, role_gram pass 1, the rest pass 3
    if (g.role_period <= 0) { g.role_period = 10; g.role_solve = 1; g.role_gram = 4; }
    g.solve_items = (g.NP + 1) * 2 * g.nBset;
    pl.ctr_bytes = align_up((size_t)(4 + 3 * g.NP + 2) * sizeof(int), 256);
    pl.off_oct = pl.ctr_bytes;
    const size_t oct_bytes = (size_t)(g.ring + 2) * g.nA * kTileRec * sizeof(float);     // forward records (the backward's are smaller)
    pl.off_fac = pl.off_oct + align_up(oct_bytes, 256);
    pl.off_mb = pl.off_fac + align_up((size_t)2 * G.mats_per_shift * kFacF * sizeof(float), 256);
    pl.off_trace = pl.off_mb + align_up((size_t)2 * G.mats_per_shift * kMbF * sizeof(float), 256);
    pl.total = pl.off_trace;
#ifdef FZ_TUNING
    pl.total += align_up((size_t)(3 * (g.NP + 1) + 5 * 100) * sizeof(unsigned long long) + 64, 256);
#endif
    return pl;
}

void fill(PhaseParams& P, const Plan& pl, const DevGeom& G, const fz_solver& s, int K, void* workspace) {
    fill_common(P, G, s, K);
    char* ws = static_cast<char*>(workspace);
    P.pipe = pl.g;
    P.pipe.ctr = reinterpret_cast<int*>(ws);
    P.oct = reinterpret_cast<float*>(ws + pl.off_oct);
    P.fac = reinterpret_cast<float*>(ws + pl.off_fac);
    P.mb = reinterpret_cast<float*>(ws + pl.off_mb);
#ifdef FZ_TUNING
    P.pipe.trace = getenv("FZ_PIPE_TRACE") ? reinterpret_cast<unsigned long long*>(ws + pl.off_trace) : nullptr;
    if (P.pipe.trace) fprintf(stderr, "[fz] pipe plan: NP=%d nA=%d lead=%d ring=%d trace at byte %zu\n", pl.g.NP, pl.g.nA, pl.g.lead, pl.g.ring, pl.off_trace);
#endif
    P.t_begin = 0; P.t_count = P.tiles;
}

constexpr size_t kFwdSmem = (size_t)kFwdSlots * kFwdSlotFloats * sizeof(float);
constexpr size_t kBwdSmem = (size_t)kBwdSlots * kBwdSlotFloats * sizeof(float);

}  // namespace

// Measured on B200 at config 2 (profiles/r02_pipeline.md): correct (bit-equal to the three-launch scheme) but slower --
// 310-380 us forward against 183 us -- because the dependency chain pass 1 -> pass 2 -> pass 3 -> (lead bound) -> pass 1
// takes tens of microseconds per plane-group while the tiles of a plane-group are worth 1.6 us of HBM time.  It is
// therefore only taken on request (fz_geom.path = FZ_PATH_OCTANT_PIPELINE); FZ_PATH_AUTO keeps the three-launch scheme.
bool pipe_supported(const DevGeom& G, const fz_solver& s, int relu, int force) {
    if (force <= 0 || G.dtype != FZ_DTYPE_F32) return false;
    if (!phase_supported(G, s, relu)) return false;
    return G.mats_per_shift < (1LL << 24);
}

size_t pipe_workspace_bytes(const DevGeom& G, const fz_solver& s) {
    (void)s;
    return make_plan(G).total;
}

int pipe_forward(const float* x, const float* v0, float* y, void* saved, void* workspace,
                 const DevGeom& G, const fz_solver& s, cudaStream_t st) {
    if (!workspace) return fail(FZ_ERR_INVALID, "fz_swnmf_forward: workspace of %zu bytes required", pipe_workspace_bytes(G, s));
    if (reinterpret_cast<uintptr_t>(y) & 15) return fail(FZ_ERR_INVALID, "output pointer %p is not 16-byte aligned", (void*)y);
    const Plan pl = make_plan(G);
    static thread_local PhaseParams P;
    fill(P, pl, G, s, 0, workspace);
    if (int e = make_tile_map(&P.tm_x, x, G)) return e;
    P.x = x; P.out = y; P.v0 = v0; P.saved = static_cast<float*>(saved);
    static SmemConfig cfg;
    FZ_CUDA_CHECK(cfg.ensure(pipe_fwd, kFwdSmem));
    FZ_CUDA_CHECK(cudaMemsetAsync(workspace, 0, pl.ctr_bytes, st));
    pipe_fwd<<<num_sms(), kThreads, kFwdSmem, st>>>(P);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

int pipe_backward(const float* x, const float* gy, const float* v0, const void* saved, float* gx,
                  void* workspace, const DevGeom& G, const fz_solver& s, int K, cudaStream_t st) {
    if (!workspace) return fail(FZ_ERR_INVALID, "fz_swnmf_backward: workspace of %zu bytes required", pipe_workspace_bytes(G, s));
    if (!saved) return fail(FZ_ERR_INVALID, "fz_swnmf_backward: the `saved` buffer written by fz_swnmf_forward is required");
    if (reinterpret_cast<uintptr_t>(gx) & 15) return fail(FZ_ERR_INVALID, "output pointer %p is not 16-byte aligned", (void*)gx);
    const Plan pl = make_plan(G);
    static thread_local PhaseParams P;
    fill(P, pl, G, s, K, workspace);
    if (int e = make_tile_map(&P.tm_x, x, G)) return e;
    if (int e = make_tile_map(&P.tm_g, gy, G)) return e;
    P.x = x; P.gy = gy; P.out = gx; P.v0 = v0;
    P.saved = const_cast<float*>(static_cast<const float*>(saved));
    static SmemConfig cfg;
    FZ_CUDA_CHECK(cfg.ensure(pipe_bwd, kBwdSmem));
    FZ_CUDA_CHECK(cudaMemsetAsync(workspace, 0, pl.ctr_bytes, st));
    pipe_bwd<<<num_sms(), kThreads, kBwdSmem, st>>>(P);
    FZ_LAUNCH_CHECK();
    return FZ_OK;
}

}  // namespace fz
