// mpp_stats.cuh -- lane-group path statistics shared by the fitness and MPA kernels (one path per lane group, mpp_astar.cuh).
#pragma once
#include "mpp_astar.cuh"

// ---------------------------------------------------------------------------------------------
// K7: path statistics by one lane group (helper.py:98-113 / MPA.py:215-229)
// out[5] = length, turns, safety penalty, diagonal penalty, fitness
// ---------------------------------------------------------------------------------------------
struct StatsCtx {
    const uint32_t *occ;
    int pitch, R, C;
    const uint16_t *cls;    // safety classes (may be null when mode == 1 or spf table not needed)
    const double *lut;
    mpp_policy pol;
};

// X for the maps of a batch (mpp_astar.cu): their occupancy, the policy and -- mode 0 on a batch with obstacles -- the
// batch's safety tables (mpp_map_batch_safety_table).  A kernel offsets occ / cls to the map a path lies on.
int mpp_stats_ctx(mpp_map_batch *maps, const mpp_policy *pol, void *stream, StatsCtx *X);

// the statistics weights of a map's per-map parameters (mpp_pop_params) in place of the policy's
static __device__ __forceinline__ void mpp_pop_weights(mpp_policy &pol, const mpp_pop_params &p) {
    pol.turn_penalty_factor = p.turn_penalty_factor;
    pol.safety_penalty_factor = p.safety_penalty_factor;
    pol.diagonal_obstacle_penalty_value = p.diagonal_obstacle_penalty_value;
}

static __device__ void path_stats_warp(const LaneGroup &L, const StatsCtx &X, const int32_t *cells, int n, double *out) {
    const int lane = L.gl;
    const double INF = __longlong_as_double(MPP_INF_BITS);
    if (n <= 0) {                                                        // helper.py:104-105
        if (lane == 0) { out[0] = INF; out[1] = 0.0; out[2] = 0.0; out[3] = 0.0; out[4] = INF; }
        return;
    }
    const int C = X.C;
    double f = 0.0, comp = 0.0, saf = 0.0;
    int turns = 0, ndiag = 0;
    const bool want_safety = (X.pol.mode == 0) && X.cls != nullptr;
    for (int base = 0; base < n; base += MPP_GL) {
        const int i = base + lane;
        const int c0 = i < n ? cells[i] : 0;
        const int c1 = (i + 1) < n ? cells[i + 1] : c0;
        const int c2 = (i + 2) < n ? cells[i + 2] : c1;
        const int r0 = c0 / C, q0 = c0 % C, r1 = c1 / C, q1 = c1 % C, r2 = c2 / C, q2 = c2 % C;
        const int dr1 = r1 - r0, dc1 = q1 - q0, dr2 = r2 - r1, dc2 = q2 - q1;
        double x = 0.0;
        if (i + 1 < n) x = hdist_dev(r0, q0, r1, q1);                   // helper.py:106
        const bool is_turn = (i + 2 < n) && (dr1 != dr2 || dc1 != dc2);  // helper.py:58-65
        bool is_diag_cut = false;                                       // helper.py:82-96
        if (i + 1 < n && (dr1 == 1 || dr1 == -1) && (dc1 == 1 || dc1 == -1)) {
            const int pb0 = q0 + 1, pb1 = q1 + 1;
            const bool b1 = (X.occ[(r1 + 1) * X.pitch + (pb0 >> 5)] >> (pb0 & 31)) & 1u;   // (next_r, curr_c)
            const bool b2 = (X.occ[(r0 + 1) * X.pitch + (pb1 >> 5)] >> (pb1 & 31)) & 1u;   // (curr_r, next_c)
            is_diag_cut = b1 || b2;
        }
        double pen = 0.0;
        if (want_safety && i < n) pen = X.lut[X.cls[c0]];               // helper.py:70-79
        turns += __popc(grp_ballot(L, is_turn));
        ndiag += __popc(grp_ballot(L, is_diag_cut));
        // sequential folds in path order (fp64 addition is not associative)
        const int cnt = (n - base) < MPP_GL ? (n - base) : MPP_GL;
        for (int l = 0; l < cnt; ++l) {
            const double xl = grp_shfl(L, x, l);
            const double pl = grp_shfl(L, pen, l);
            const int gi = base + l;
            if (gi + 1 < n) {
                if (gi == 0) f = xl;                                    // 0 + x0 leaves CPython's int fast path
                else {                                                  // Neumaier step (CPython 3.12 sum())
                    const double t = f + xl;
                    if (fabs(f) >= fabs(xl)) comp += (f - t) + xl; else comp += (xl - t) + f;
                    f = t;
                }
            }
            saf += pl;                                                  // + 0.0 is exact
        }
    }
    if (comp != 0.0 && comp == comp && fabs(comp) != INF) f += comp;
    const double length = (n > 1) ? f : 0.0;
    const double safety = want_safety ? saf / (double)n : 0.0;          // helper.py:80 ; MPA.py:173 -> 0.0
    double diag = 0.0;
    if (n >= 2 && X.pol.restrict_policy)
        for (int k = 0; k < ndiag; ++k) diag += X.pol.diagonal_obstacle_penalty_value;
    if (lane == 0) {
        out[0] = length; out[1] = (double)turns; out[2] = safety; out[3] = diag;
        out[4] = length + X.pol.turn_penalty_factor * (double)turns + X.pol.safety_penalty_factor * safety + diag;
    }
}

