/* dijkstra_field_oracle.c -- TEST INFRASTRUCTURE: the C oracle's Dijkstra (orc_astar variant 2) run until its heap is
 * empty, recording the popped g and the parent move of every cell.  It includes the oracle's source, so the heap, the
 * (g, cell) order and the neighbour / corner rules (cell_ok, NB_R / NB_C) are the oracle's own.  Built by
 * field_oracle.py into a temporary directory. */
#include "../oracle/mpp_oracle.c"

/* g_out[R*C] = popped g (+inf: never popped), parent_out[R*C] = move parent -> cell in NB_R / NB_C order (0xFF: none).
 * A source outside the map or on an obstacle leaves everything at (+inf, 0xFF). */
ORC_API void orc_dijkstra_field(astar_ctx *x, int src, double *g_out, uint8_t *parent_out) {
    const int R = x->R, C = x->C;
    const size_t n = (size_t)R * C;
    for (size_t i = 0; i < n; ++i) { g_out[i] = INFINITY; parent_out[i] = 0xFF; }
    if (src < 0 || (size_t)src >= n || !cell_ok(x, src / C, src % C)) return;
    memset(x->seen, 0, n); memset(x->closed, 0, n);
    for (size_t i = 0; i < n; ++i) x->pos[i] = -1;
    heap_t H = { x->heap, 0, x->pos, C };
    x->g[src] = 0.0; x->seen[src] = 1; x->parent[src] = -1;
    hent e0 = { 0.0, 0.0, src };
    H.h[0] = e0; H.pos[src] = 0; H.n = 1;
    while (H.n > 0) {                                   /* orc_astar's loop without the target test */
        hent cur = hpop(&H);
        if (x->closed[cur.cell]) continue;
        x->closed[cur.cell] = 1;
        int cr = cur.cell / C, cc = cur.cell % C;
        g_out[cur.cell] = cur.g;
        if (x->parent[cur.cell] >= 0) {
            int p = x->parent[cur.cell], dr = cr - p / C, dc = cc - p % C;
            for (int m = 0; m < 8; ++m)
                if (NB_R[m] == dr && NB_C[m] == dc) parent_out[cur.cell] = (uint8_t)m;
        }
        int nmv = x->allow_diag ? 8 : 4;
        for (int m = 0; m < nmv; ++m) {
            int nr = cr + NB_R[m], nc = cc + NB_C[m];
            if (!cell_ok(x, nr, nc)) continue;
            int j = nr * C + nc;
            if (x->closed[j]) continue;
            if (m >= 4 && x->restrict_corner) {
                if (!cell_ok(x, cr + NB_R[m], cc) || !cell_ok(x, cr, cc + NB_C[m])) continue;
            }
            double tg = cur.g + (m >= 4 ? sqrt(2.0) : 1.0);
            if (!x->seen[j] || tg < x->g[j]) {
                x->parent[j] = cur.cell; x->g[j] = tg; x->seen[j] = 1;
                hent e = { tg, tg, j };
                if (H.pos[j] < 0) { int i = H.n++; H.h[i] = e; H.pos[j] = i; hup(&H, i); }
                else { int i = H.pos[j]; H.h[i] = e; hup(&H, i); hdown(&H, H.pos[j]); }
            }
        }
    }
}
