// mpp_astar.cuh -- exact emulation of the reference's two A* connectors by one LANE GROUP per search.
//
//   variant 0: AStarSolver.solve  (astar.py:33-101)  -- closed set seeded from nodes_to_avoid minus
//              {start,target}, relax from the popped g, in-place decrease-key.
//   variant 2: DijkstraSolver.solve (dijkstra.py:32-97) -- variant 0 with a zero heuristic (key (g, r, c)).
//   variant 1: MPA._a_star        (MPA.py:106-151)   -- no closed set, avoid-set filters neighbours only,
//              relax from g_score[current], keys of nodes already in the open set are left stale,
//              nodes not in the open set (incl. already expanded ones) are re-pushed.
//
// Both are fully described by "extract-min over the total order (f, g, r, c)" + their relax rules
// (SURVEY 8(a) A1/A2, validated 0/1500 mismatches against the unmodified reference); heap internals do
// not matter.  A search is a dependent chain of expansions; the lanes of its group relax the 8 neighbours in
// parallel, push them together (one shared-memory atomic each) and scan / reduce the priority queue.  Every
// warp-level primitive is issued under the group's lane mask, so the group width MPP_GL is a build option:
// 32 (default) = one search per warp.  Measured on B200, config 3 (4096 individuals x 6 searches, 512x512):
// MPP_GL = 32: 0.86 s, 16: 1.27 s, 8: 2.09 s per population -- four searches per warp do NOT share an instruction
// stream (every expansion branches on its own data: ring or heap, stale entry, bucket scan length), so the narrow
// groups only serialise four chains inside one warp and leave fewer warps to hide memory latency
// (profiles/r02_astar_summary.md).  Decrease-key is done by lazy deletion (variant 0: the fresher entry always
// sorts first, the stale one is dropped when popped because its cell is closed), which keeps the pop sequence
// identical to the reference's.
#pragma once
#include "mpp_common.cuh"

#define MPP_INF_BITS 0x7ff0000000000000ll
#define MPP_ASTAR_SQRT2 1.4142135623730951

// neighbour order helper.py:30-36 == MPA.py:71-77: (0,1),(0,-1),(1,0),(-1,0),(1,1),(1,-1),(-1,1),(-1,-1)
// (delta+1) packed two bits per move
#define MPP_NB_R 0x0A25u  // r+1: 1,1,2,0,2,2,0,0
#define MPP_NB_C 0x2252u  // c+1: 2,0,1,1,2,0,2,0

// ---------------------------------------------------------------------------------------------
// lane groups
// ---------------------------------------------------------------------------------------------
#ifndef MPP_GL
#define MPP_GL 32                                  // lanes per search (8, 16 or 32)
#endif
#define MPP_GROUPS_PER_WARP (32 / MPP_GL)
#define MPP_GL_MASK (MPP_GL == 32 ? 0xffffffffu : ((1u << (MPP_GL & 31)) - 1u))   // MPP_GL low bits
struct LaneGroup {
    uint32_t mask;                                 // the group's lanes inside the warp
    int base, gl;                                  // first lane of the group, this lane's index inside it
};
__device__ __forceinline__ LaneGroup lane_group() {
    LaneGroup L;
    const int lane = threadIdx.x & 31;
    L.base = lane & ~(MPP_GL - 1);
    L.gl = lane & (MPP_GL - 1);
    L.mask = MPP_GL_MASK << L.base;
    return L;
}
__device__ __forceinline__ uint32_t grp_ballot(const LaneGroup &L, bool p) {
    return (__ballot_sync(L.mask, p) >> L.base) & MPP_GL_MASK;
}
template <typename T>
__device__ __forceinline__ T grp_shfl(const LaneGroup &L, T v, int src) { return __shfl_sync(L.mask, v, src, MPP_GL); }
__device__ __forceinline__ void grp_sync(const LaneGroup &L) { __syncwarp(L.mask); }

struct AStarGrid {
    const uint32_t *occ;  // padded occupancy bits (shared or global)
    int pitch, R, C;
    int allow_diag, restrict_corner;
};

// ---------------------------------------------------------------------------------------------
// Priority queue = exact extract-min over (f, g, cell), built for one lane group:
//   * a ring of MPP_PQ_NB buckets keyed by floor((f - f0) * MPP_PQ_SCALE), MPP_PQ_CAP (= MPP_GL, one per lane)
//     entries each, bucket fill counts (bytes) in shared memory.  push = one shared-memory atomic on the count + one
//     store, all neighbours of an expansion at once; pop = one load of the lowest non-empty bucket + a group arg-min
//     (bucket index is monotone in f, so the global minimum lives in the lowest non-empty bucket);
//   * an overflow MPP_GL-ary min-heap in HBM for entries outside the ring window or landing in a full bucket;
//     its root key is cached in registers and compared with the ring minimum on every pop.
// Either structure alone is exact; together they keep the common case at one memory round trip per pop.
// ---------------------------------------------------------------------------------------------
#define MPP_PQ_NB 2048
#define MPP_PQ_CAP MPP_GL
#define MPP_PQ_SCALE 256.0

struct __align__(16) AStarRec { double g; uint32_t meta; uint32_t pad; };  // meta: [31:8] stamp, bit4 closed, bit3 in_open, [2:0] parent move

// per-group scratch slot (HBM)
struct AStarSlot {
    AStarRec *rec;
    double *bf, *bg;   // ring buckets
    int32_t *bc;
    double *hf, *hg;   // overflow heap
    int32_t *hc;
    uint32_t *hdr;     // hdr[0] = stamp counter
    uint8_t *cnt;      // shared memory: MPP_PQ_NB bucket fill counts of this group
    int heap_cap;
};

// Occupancy staging of the connector, fitness and MPA kernels (the <true> instantiations): a map of up to
// MPP_OCC_STAGE_MAX bytes of packed occupancy is copied into dynamic shared memory by every block, a larger one is read
// through L2 by the <false> instantiation.  The kernels also declare ~16 KB of static shared memory (the bucket
// counts), so a staged launch needs the kernel's dynamic limit raised as soon as static + dynamic exceeds the default
// 48 KB -- a map of exactly 32 KB (510x510) already does.  One MppStaging per staged kernel caches its static size and,
// per device, the limit raised so far (the attribute only grows; the call is slow).
#define MPP_OCC_STAGE_MAX (40 * 1024)
struct MppStaging {
    int static_bytes;       // -1: not read yet
    int raised[64];         // dynamic limit set on device d & 63 (0: the default)
};
// *stage = whether `kernel` (a <true> instantiation) stages `occ_bytes`; if it does, the launch may use that much.
int mpp_occ_staging(const void *kernel, MppStaging &st, int device, size_t occ_bytes, bool *stage);

__host__ __device__ __forceinline__ size_t astar_align256(size_t b) { return (b + 255) & ~(size_t)255; }
__host__ __device__ __forceinline__ size_t astar_slot_bytes(int rc, int heap_cap) {
    size_t b = 256;                                                    // header
    b += astar_align256((size_t)rc * sizeof(AStarRec));
    b += 2 * astar_align256((size_t)MPP_PQ_NB * MPP_PQ_CAP * 8) + astar_align256((size_t)MPP_PQ_NB * MPP_PQ_CAP * 4);
    const size_t hs = (size_t)heap_cap + 64;                           // heap storage index = node + MPP_GL - 1, padded
    b += 2 * astar_align256(hs * 8) + astar_align256(hs * 4);
    return b;
}
__device__ __forceinline__ AStarSlot astar_slot_at(char *base, int rc, int heap_cap, uint8_t *cnt_smem) {
    AStarSlot s;
    s.hdr = (uint32_t *)base; base += 256;
    s.rec = (AStarRec *)base; base += astar_align256((size_t)rc * sizeof(AStarRec));
    s.bf = (double *)base; base += astar_align256((size_t)MPP_PQ_NB * MPP_PQ_CAP * 8);
    s.bg = (double *)base; base += astar_align256((size_t)MPP_PQ_NB * MPP_PQ_CAP * 8);
    s.bc = (int32_t *)base; base += astar_align256((size_t)MPP_PQ_NB * MPP_PQ_CAP * 4);
    const size_t hs = (size_t)heap_cap + 64;
    s.hf = (double *)base; base += astar_align256(hs * 8);
    s.hg = (double *)base; base += astar_align256(hs * 8);
    s.hc = (int32_t *)base;
    s.cnt = cnt_smem;
    s.heap_cap = heap_cap;
    return s;
}

__device__ __forceinline__ bool occ_bit(const AStarGrid &G, int r, int c) {  // true = blocked (incl. out of bounds)
    const int pb = c + 1;
    return (G.occ[(r + 1) * G.pitch + (pb >> 5)] >> (pb & 31)) & 1u;
}
__device__ __forceinline__ double hdist_dev(int r0, int c0, int r1, int c1) {  // helper.py:8-12
    const long long dr = r0 - r1, dc = c0 - c1;
    return sqrt((double)(dr * dr + dc * dc));                                 // IEEE correctly rounded
}

// lexicographic (f, g, cell) "a < b"
__device__ __forceinline__ bool key_less(double fa, double ga, int ca, double fb, double gb, int cb) {
    if (fa != fb) return fa < fb;
    if (ga != gb) return ga < gb;
    return ca < cb;
}

// group arg-min over lanes of (f, g, cell); lanes with f = +inf are empty.  All lanes get the winner's index in the group.
__device__ __forceinline__ int grp_argmin_key(const LaneGroup &L, double f, double g, int cell) {
    // non-negative doubles: unsigned bit order == numeric order (+inf sorts last)
    const unsigned long long kf = (unsigned long long)__double_as_longlong(f);
    uint32_t hi = (uint32_t)(kf >> 32), lo = (uint32_t)kf;
    uint32_t mh = __reduce_min_sync(L.mask, hi);
    uint32_t ml = __reduce_min_sync(L.mask, hi == mh ? lo : 0xffffffffu);
    uint32_t m = grp_ballot(L, hi == mh && lo == ml);
    if (__popc(m) > 1) {
        const unsigned long long kg = (unsigned long long)__double_as_longlong(g);
        const bool in = (m >> L.gl) & 1u;
        hi = in ? (uint32_t)(kg >> 32) : 0xffffffffu;
        lo = (uint32_t)kg;
        mh = __reduce_min_sync(L.mask, hi);
        ml = __reduce_min_sync(L.mask, (in && hi == mh) ? lo : 0xffffffffu);
        m = grp_ballot(L, in && hi == mh && lo == ml);
        if (__popc(m) > 1) {
            const bool in2 = (m >> L.gl) & 1u;
            const uint32_t mc = __reduce_min_sync(L.mask, in2 ? (uint32_t)cell : 0xffffffffu);
            m = grp_ballot(L, in2 && (uint32_t)cell == mc);
        }
    }
    return __ffs(m) - 1;
}

#define HIDX(k) ((k) + MPP_GL - 1)  // node k -> storage index; children of k = nodes GL*k+1..GL*k+GL (storage aligned to GL)

// Overflow heap push (f,g,cell) -- group-uniform arguments.  Returns false on overflow.
__device__ __forceinline__ bool heap_push(const LaneGroup &L, AStarSlot &S, int &n, double f, double g, int cell) {
    if (n >= S.heap_cap) return false;
    int k = n++;
    while (k > 0) {
        const int p = (k - 1) / MPP_GL;
        const double pf = S.hf[HIDX(p)], pg = S.hg[HIDX(p)];
        const int pc = S.hc[HIDX(p)];
        if (!key_less(f, g, cell, pf, pg, pc)) break;
        if (L.gl == 0) { S.hf[HIDX(k)] = pf; S.hg[HIDX(k)] = pg; S.hc[HIDX(k)] = pc; }
        k = p;
    }
    if (L.gl == 0) { S.hf[HIDX(k)] = f; S.hg[HIDX(k)] = g; S.hc[HIDX(k)] = cell; }
    grp_sync(L);
    return true;
}

// Overflow heap pop -- returns the minimum in (f,g,cell) (group-uniform).  n > 0 required.
__device__ __forceinline__ void heap_pop(const LaneGroup &L, AStarSlot &S, int &n, double &f, double &g, int &cell) {
    f = S.hf[HIDX(0)]; g = S.hg[HIDX(0)]; cell = S.hc[HIDX(0)];
    --n;
    if (n == 0) return;
    const double xf = S.hf[HIDX(n)], xg = S.hg[HIDX(n)];
    const int xc = S.hc[HIDX(n)];
    grp_sync(L);
    int k = 0;
    for (;;) {
        const int c0 = MPP_GL * k + 1;
        if (c0 >= n) break;
        const int ci = c0 + L.gl;
        double cf = __longlong_as_double(MPP_INF_BITS), cg = 0.0;
        int cc = 0x7fffffff;
        if (ci < n) { cf = S.hf[HIDX(ci)]; cg = S.hg[HIDX(ci)]; cc = S.hc[HIDX(ci)]; }
        const int w = grp_argmin_key(L, cf, cg, cc);
        const double mf = grp_shfl(L, cf, w), mg = grp_shfl(L, cg, w);
        const int mc = grp_shfl(L, cc, w);
        if (!key_less(mf, mg, mc, xf, xg, xc)) break;
        if (L.gl == 0) { S.hf[HIDX(k)] = mf; S.hg[HIDX(k)] = mg; S.hc[HIDX(k)] = mc; }
        k = c0 + w;
    }
    if (L.gl == 0) { S.hf[HIDX(k)] = xf; S.hg[HIDX(k)] = xg; S.hc[HIDX(k)] = xc; }
    grp_sync(L);
}

struct AStarPQ {
    int qlo;         // every ring entry has bucket index >= qlo
    int n_ring, hn;  // entries in the ring / in the overflow heap
    double f0;       // bucket origin (f of the start node; f never drops below it except by rounding)
    double rf, rg;   // cached overflow-heap root key (valid when hn > 0)
    int rc;
    uint32_t ring_pushes, heap_pushes;
};

// bucket index of a key (monotone in f)
__device__ __forceinline__ int pq_bucket(const AStarPQ &Q, double f) {
    const double x = (f - Q.f0) * MPP_PQ_SCALE;
    return (x >= 0.0) ? (x < 2.0e9 ? (int)x : 0x7ffffff0) : -1;
}

// Push the entries of all lanes with `want` at once: (f, g, cell, q = pq_bucket(f)) are per lane.
// `cell` is the packed node id (row << 16 | col): same (r, c) lexicographic order as the reference's tuples.
__device__ __forceinline__ bool pq_push_many(const LaneGroup &L, AStarSlot &S, AStarPQ &Q, bool want, double f, double g,
                                             int cell, int q) {
    if (Q.n_ring == 0) {                                         // empty ring: re-centre the window on the lowest new key
        const uint32_t lo = __reduce_min_sync(L.mask, (want && q >= 0) ? (uint32_t)q : 0x7fffffffu);
        if (lo != 0x7fffffffu) Q.qlo = (int)lo;
    }
    bool ok = false;
    if (want && q >= Q.qlo && q - Q.qlo < MPP_PQ_NB) {
        const int b = q & (MPP_PQ_NB - 1);
        uint32_t *w = (uint32_t *)S.cnt + (b >> 2);
        const uint32_t sh = 8u * (uint32_t)(b & 3);
        const uint32_t c = (atomicAdd(w, 1u << sh) >> sh) & 0xFFu;           // shared-memory atomic on the byte's word
        if (c < MPP_PQ_CAP) {
            const int i = b * MPP_PQ_CAP + (int)c;
            S.bf[i] = f; S.bg[i] = g; S.bc[i] = cell;
            ok = true;
        } else {
            atomicSub(w, 1u << sh);                                          // the bucket is full: the entry goes to the heap
        }
    }
    const uint32_t done = grp_ballot(L, ok);
    Q.n_ring += __popc(done);
    Q.ring_pushes += __popc(done);
    uint32_t rest = grp_ballot(L, want && !ok);
    grp_sync(L);
    while (rest) {
        const int l = __ffs(rest) - 1;
        rest &= rest - 1;
        const double hf = grp_shfl(L, f, l), hg = grp_shfl(L, g, l);
        const int hc = grp_shfl(L, cell, l);
        const bool was_empty = Q.hn == 0;
        if (!heap_push(L, S, Q.hn, hf, hg, hc)) return false;
        if (was_empty || key_less(hf, hg, hc, Q.rf, Q.rg, Q.rc)) { Q.rf = hf; Q.rg = hg; Q.rc = hc; }
        ++Q.heap_pushes;
    }
    return true;
}

// extract-min (requires n_ring + hn > 0)
__device__ __forceinline__ void pq_pop(const LaneGroup &L, AStarSlot &S, AStarPQ &Q, double &f, double &g, int &cell) {
    double cf = __longlong_as_double(MPP_INF_BITS), cg = 0.0, mf = cf, mg = 0.0;
    int cc = 0x7fffffff, mc = 0x7fffffff, w = 0, b = 0, c = 0;
    if (Q.n_ring > 0) {
        // lowest non-empty bucket: each lane looks at four count bytes (one word) per round, starting at qlo's word
        int wbase = Q.qlo >> 2;
        uint32_t first_mask = 0xFFFFFFFFu << (8u * (uint32_t)(Q.qlo & 3));   // buckets below qlo in the first word belong
        for (;;) {                                                          // to the far end of the window
            uint32_t wv = ((const uint32_t *)S.cnt)[(wbase + L.gl) & (MPP_PQ_NB / 4 - 1)];
            if (L.gl == 0) wv &= first_mask;
            const uint32_t m = grp_ballot(L, wv != 0u);
            if (m) {
                const int src = __ffs(m) - 1;
                const uint32_t sv = grp_shfl(L, wv, src);
                Q.qlo = ((wbase + src) << 2) + ((__ffs(sv) - 1) >> 3);
                break;
            }
            wbase += MPP_GL;
            first_mask = 0xFFFFFFFFu;
#ifdef MPP_ASTAR_DEBUG
            if (wbase - (Q.qlo >> 2) > MPP_PQ_NB) { if (L.gl == 0) printf("scan loop: n_ring=%d qlo=%d\n", Q.n_ring, Q.qlo); __trap(); }
#endif
        }
        b = Q.qlo & (MPP_PQ_NB - 1);
        c = S.cnt[b];
        if (L.gl < c) { const int i = b * MPP_PQ_CAP + L.gl; cf = S.bf[i]; cg = S.bg[i]; cc = S.bc[i]; }
        w = (c == 1) ? 0 : grp_argmin_key(L, cf, cg, cc);
        mf = grp_shfl(L, cf, w); mg = grp_shfl(L, cg, w); mc = grp_shfl(L, cc, w);
    }
    if (Q.hn > 0 && (Q.n_ring == 0 || key_less(Q.rf, Q.rg, Q.rc, mf, mg, mc))) {
        heap_pop(L, S, Q.hn, f, g, cell);
        if (Q.hn > 0) { Q.rf = S.hf[HIDX(0)]; Q.rg = S.hg[HIDX(0)]; Q.rc = S.hc[HIDX(0)]; }
        return;
    }
    f = mf; g = mg; cell = mc;
    const int last = c - 1;
    if (w != last) {                                            // fill the hole with the bucket's last entry
        const double lf = grp_shfl(L, cf, last), lg = grp_shfl(L, cg, last);
        const int lc = grp_shfl(L, cc, last);
        if (L.gl == 0) { const int i = b * MPP_PQ_CAP + w; S.bf[i] = lf; S.bg[i] = lg; S.bc[i] = lc; }
    }
    if (L.gl == 0) S.cnt[b] = (uint8_t)last;
    grp_sync(L);
    --Q.n_ring;
}

// One search by one lane group.  Returns number of path cells written to out[0..) in forward order
// (0 = no path / invalid endpoints, -1 = heap overflow).  avoid: bitmap over cells or nullptr.
// *g_out = g of the popped target entry (+inf when no path).  counters: [0] expansions, [1] relaxations,
// [2] ring pushes, [3] overflow-heap pushes (nullable).
static __device__ int astar_search(const LaneGroup &L, const AStarGrid &G, AStarSlot &S, int variant, int src, int dst,
                            const uint32_t *avoid, int32_t *out, int out_cap, double *g_out,
                            unsigned long long *counters) {
    const int lane = L.gl;
    const int C = G.C;
    const int sr = src / C, sc = src % C, tr = dst / C, tc = dst % C;
    const double INF = __longlong_as_double(MPP_INF_BITS);
    if (g_out) *g_out = INF;
    if (variant == 1 && src == dst) { if (lane == 0 && out_cap > 0) out[0] = src; if (g_out) *g_out = 0.0; grp_sync(L); return 1; }  // MPA.py:107-108
    if (occ_bit(G, sr, sc) || occ_bit(G, tr, tc)) return 0;        // astar.py:37-39 / MPA.py:109-111
    if (variant != 1 && src == dst) { if (lane == 0 && out_cap > 0) out[0] = src; if (g_out) *g_out = 0.0; grp_sync(L); return 1; }  // astar.py:41-42
    const bool dijkstra = (variant == 2);                          // dijkstra.py:44,59,88: the key is (g, node)
    if (dijkstra) variant = 0;
    // new stamp for this search (records of older searches become invalid without clearing)
    uint32_t stamp = S.hdr[0] + 1;
    if (stamp >= (1u << 24)) {  // wrap: clear the records once every 16M searches
        for (int i = lane; i < G.R * C; i += MPP_GL) S.rec[i].meta = 0;
        stamp = 1;
    }
    grp_sync(L);
    if (lane == 0) S.hdr[0] = stamp;
    const uint32_t stamp_hi = stamp << 8;
    for (int i = lane; i < MPP_PQ_NB / 4; i += MPP_GL) ((uint32_t *)S.cnt)[i] = 0u;
    if (lane == 0) { AStarRec r0; r0.g = 0.0; r0.meta = stamp_hi | 8u; r0.pad = 0u; S.rec[src] = r0; }
    grp_sync(L);
    AStarPQ Q;
    Q.qlo = 0; Q.n_ring = 0; Q.hn = 0; Q.rf = 0.0; Q.rg = 0.0; Q.rc = 0; Q.ring_pushes = 0; Q.heap_pushes = 0;
    Q.f0 = dijkstra ? 0.0 : hdist_dev(sr, sc, tr, tc);
    const int dst_rc = (tr << 16) | tc;
    pq_push_many(L, S, Q, lane == 0, Q.f0, 0.0, (sr << 16) | sc, 0);         // astar.py:45 / MPA.py:113
    const uint32_t max_steps = (uint32_t)G.R * (uint32_t)C * (variant == 0 ? 3u : 2u);   // astar.py:58 / MPA.py:118 (R*C < 2^30)
    uint32_t steps = 0, exps = 0, rels = 0;
    // per-lane neighbour deltas
    const bool nb_lane = lane < (G.allow_diag ? 8 : 4);
    const int dr = (int)((MPP_NB_R >> (2 * (lane & 7))) & 3u) - 1, dc = (int)((MPP_NB_C >> (2 * (lane & 7))) & 3u) - 1;
    const double step_cost = (lane & 7) >= 4 ? MPP_ASTAR_SQRT2 : 1.0;  // distance_euclidean: sqrt(1)=1, sqrt(2)
    int found = 0;
    double cur_g = 0.0;
    while (Q.n_ring + Q.hn > 0 && steps < max_steps) {
        double cf;
        int cur_rc;
        pq_pop(L, S, Q, cf, cur_g, cur_rc);
        if (cur_rc == dst_rc) { found = 1; ++steps; break; }                  // astar.py:64 / MPA.py:123
        // ---- one round of loads: the popped node's record and, per lane, a neighbour's record + avoid word ----
        const int cr = cur_rc >> 16, cc = cur_rc & 0xffff;
        const int cur = cr * C + cc;
        const uint4 vcur = *reinterpret_cast<const uint4 *>(&S.rec[cur]);
        bool open_nb = false;
        int j = 0, nr = 0, nc = 0;
        uint4 vj = make_uint4(0u, 0u, 0u, 0u);
        uint32_t aw = 0u;
        if (nb_lane) {
            nr = cr + dr; nc = cc + dc;
            bool blocked = occ_bit(G, nr, nc);
            if (!blocked && ((lane & 7) >= 4) && G.restrict_corner)                  // helper.py:45-49 / MPA.py:86-96
                blocked = occ_bit(G, cr + dr, cc) || occ_bit(G, cr, cc + dc);
            if (!blocked) {
                open_nb = true;
                j = nr * C + nc;
                vj = *reinterpret_cast<const uint4 *>(&S.rec[j]);
                if (avoid) aw = avoid[j >> 5];
            }
        }
        if (lane >= MPP_GL - 4) {
            // warm L2 for the records two rows away (the neighbours of this node's neighbours): a search mostly
            // continues next to where it just was, and first touches of a record are otherwise DRAM-latency misses
            const int pr = cr + ((lane & 1) ? 2 : -2);
            const int pc = cc + ((lane & 2) ? 2 : -2);
            if (pr >= 0 && pr < G.R) {
                const int pcc = pc < 0 ? 0 : (pc >= C ? C - 1 : pc);
                asm volatile("prefetch.global.L2 [%0];" ::"l"(&S.rec[pr * C + pcc]));
            }
        }
        // heuristic of the neighbour, in parallel across lanes while the loads are in flight (astar.py:90)
        const double hj = (open_nb && !dijkstra) ? hdist_dev(nr, nc, tr, tc) : 0.0;
        // every lane has its copy of the popped node's record before lane 0 changes it: the lanes of a group are not
        // guaranteed to run in lock step (independent thread scheduling), and a lane that read the record AFTER the
        // closed bit was set would take the "stale entry" branch alone
        grp_sync(L);
        const uint32_t mcur = vcur.z;
        if (variant == 0) {
            if (mcur & 16u) continue;                                         // stale (lazily deleted) entry
            ++steps;
            if (lane == 0) S.rec[cur].meta = mcur | 16u;                       // closed_set.add astar.py:74
        } else {
            ++steps;
            if (lane == 0) S.rec[cur].meta = mcur & ~8u;                       // left the open set
        }
        ++exps;
        const double gcur = __longlong_as_double((long long)(((unsigned long long)vcur.y << 32) | vcur.x));
        const double gbase = (variant == 0) ? cur_g : gcur;                    // astar.py:85 vs MPA.py:135
        // ---- relax the neighbours, one per lane ----
        bool push = false;
        double tg = 0.0, pf = 0.0;
        int pq = 0;
        if (open_nb) {
            const bool av = (aw >> (j & 31)) & 1u;
            uint32_t mj = vj.z;
            const bool seen = (mj & 0xffffff00u) == stamp_hi;
            if (!seen) mj = 0;
            bool excluded;
            if (variant == 0) excluded = (av && j != src && j != dst) || (mj & 16u);   // closed set astar.py:51-56,80
            else excluded = av;                                                       // MPA.py:132
            if (!excluded) {
                tg = gbase + step_cost;
                const double gj = seen ? __longlong_as_double((long long)(((unsigned long long)vj.y << 32) | vj.x)) : INF;
                if (tg < gj) {                                                 // astar.py:87 / MPA.py:137
                    // parent = the move taken cur -> j; variant 1 keeps a stale key if already in open
                    push = (variant == 0) ? true : !(mj & 8u);
                    AStarRec nrc; nrc.g = tg; nrc.meta = stamp_hi | (mj & 16u) | 8u | (uint32_t)(lane & 7); nrc.pad = 0u;
                    S.rec[j] = nrc;
                    pf = tg + hj;                                              // astar.py:90 / MPA.py:140
                    pq = pq_bucket(Q, pf);
                    ++rels;
                }
            }
        }
        grp_sync(L);
        if (!pq_push_many(L, S, Q, push, pf, tg, (nr << 16) | nc, pq)) return -1;   // all neighbours at once
    }
    rels = __reduce_add_sync(L.mask, rels);
    if (lane == 0 && counters) {
        atomicAdd(counters, (unsigned long long)exps);
        atomicAdd(counters + 1, (unsigned long long)rels);
        atomicAdd(counters + 2, (unsigned long long)Q.ring_pushes);
        atomicAdd(counters + 3, (unsigned long long)Q.heap_pushes);
    }
    if (!found) return 0;
    if (g_out) *g_out = cur_g;
    // ---- rebuild: follow parent moves target -> start (astar.py:65-69 / MPA.py:124-130) ----
    int len = 0;
    if (lane == 0) {
        int t = dst;
        while (true) {
            if (len < out_cap) out[len] = t;
            ++len;
#ifdef MPP_ASTAR_DEBUG
            if (len > G.R * C) { printf("rebuild loop: src=%d dst=%d t=%d variant=%d\n", src, dst, t, variant); __trap(); }
#endif
            if (t == src) break;
            const uint32_t mv = S.rec[t].meta & 7u;
            const int pdr = (int)((MPP_NB_R >> (2 * mv)) & 3u) - 1, pdc = (int)((MPP_NB_C >> (2 * mv)) & 3u) - 1;
            t -= pdr * C + pdc;
        }
    }
    len = grp_shfl(L, len, 0);
    grp_sync(L);
    const int m = len < out_cap ? len : out_cap;  // (if truncated the caller sees len > cap)
    for (int i = lane; i < m / 2; i += MPP_GL) {   // reverse in place
        const int32_t a = out[i], b = out[m - 1 - i];
        out[i] = b; out[m - 1 - i] = a;
    }
    grp_sync(L);
    return len;
}
