/*
 * edge_pin_oracle.c — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * The oracle's SSD with genes and regulatory edges pinned: the CPU restatement that tests/test_gpu_edge_pins.py compares
 * pbn_ssd_pinned_edges against.  It is compiled together with oracle/pbn_oracle.c (same translation unit, see
 * tests/edge_pin_oracle.py) so that it uses the oracle's own Philox streams, node updates and geometric gaps, byte per node,
 * and shares nothing with the product.  Rules 1-3 are those of orc_ssd_pinned (tests/pinned_oracle.c), which
 * tests/test_oracle_edge_pins.py checks this function against when no edge is pinned.
 */
#include "pbn_oracle.c"

/* orc_ssd with a pin set and edge pins, env = NULL, PHILOX draws (pbn_ssd_pinned_edges, one variant per call): pin[i] = 0 or
   1 holds node i at that value, any other value leaves it free; edges[0..E) are entries dst | src << 12 | c << 24
   (0xFFFFFFFF = empty, c = bit 24).
     1. before the first iteration every pinned node is set to its value;
     2. an update that picks a pinned node consumes its draws (node index, predictor or table draw) and the node keeps its value;
     3. a perturbation event on a pinned node is drawn and not applied;
     4. when the update of a node dst reads its input src and an entry pins (src, dst, c), it reads c (the first such entry
        of the row): restated on the gather side, the update reads a copy of the state with each pinned source replaced.
        src, and every other node that reads it, keep the real value.  An entry whose dst is not below n, or whose src dst
        never reads, changes nothing.
   Chain e draws from the streams of global id env0 + e, as in orc_ssd.  Returns 1 for a misaligned env0, 2 for replay draws. */
int orc_ssd_pinned_edges(const OrcNet *net, uint8_t *state, int64_t chains, int64_t env0, int64_t iters, double p,
                         const int8_t *pin, const uint32_t *edges, int E, const int32_t *tgt_nodes, int g, uint64_t *hist,
                         const OrcDraws *dr) {
    const int n = net->n;
    const int64_t nb = (int64_t)1 << g;
    const float inv = orc_geom_inv(p);
    const int flips = !(inv > 0);
    const uint32_t W = (uint32_t)n * 32u, NONE = 0xFFFFFFFFu;
    if (dr->mode != ORC_PHILOX) return 2;
    if (flips && (env0 & 31)) return 1;
    for (int64_t e = 0; e < chains; e++)
        for (int i = 0; i < n; i++)
            if (pin[i] == 0 || pin[i] == 1) state[e * n + i] = (uint8_t)pin[i];
    int nthreads = 1;
#ifdef _OPENMP
    extern int omp_get_max_threads(void); extern int omp_get_thread_num(void);
    nthreads = omp_get_max_threads();
#endif
    uint64_t *priv = (uint64_t *)calloc((size_t)(nthreads * nb), sizeof(uint64_t));
    const int64_t groups = (chains + 31) / 32;
#pragma omp parallel for schedule(static) if (chains >= 256)
    for (int64_t gi = 0; gi < groups; gi++) {
        int tid = 0;
#ifdef _OPENMP
        tid = omp_get_thread_num();
#endif
        uint64_t *h = priv + (int64_t)tid * nb;
        uint8_t *seen = (uint8_t *)malloc((size_t)n); /* rule 4: the state as the update of dst reads it */
        const int64_t gb = gi * 32;
        Dr d[32], dp[32];
        uint32_t ev[64], last_p1 = 0;
        for (int l = 0; l < 32; l++) {
            dr_init(&d[l], dr, gb + l < chains ? gb + l : 0, env0 + gb + l);
            dp[l] = d[l];
            dp[l].ctr[0] = 0x80000000u;
            ev[2 * l] = ev[2 * l + 1] = NONE;
        }
        for (int64_t t = 0; t < iters; t++) {
            for (int l = 0; l < 32 && gb + l < chains; l++) {
                const uint8_t *st = state + (gb + l) * n;
                int64_t b = 0;
                for (int k = 0; k < g; k++) b = (b << 1) | st[tgt_nodes[k]];
                h[b]++;
            }
            if (flips) {
                for (;;) {
                    for (int k = 0; k < 64; k++)
                        if (ev[k] < W) {
                            uint32_t tl = ev[k] & 31u, bit = ev[k] >> 5;
                            if (gb + tl < chains && pin[bit] != 0 && pin[bit] != 1) state[(gb + tl) * n + bit] ^= 1; /* rule 3 */
                            ev[k] = NONE;
                        }
                    if (last_p1 > W) break;
                    uint32_t pre = 0;
                    for (int k = 0; k < 64; k++) { pre += 1u + orc_geom(dr_u32(&dp[k >> 1]), inv); ev[k] = last_p1 - 1u + pre; }
                    last_p1 = ev[63] + 1u;
                }
                for (int k = 0; k < 64; k++) if (ev[k] != NONE) ev[k] -= W;
                last_p1 -= W;
            }
            for (int l = 0; l < 32 && gb + l < chains; l++) {
                uint8_t *st = state + (gb + l) * n;
                const int i = dr_randint(&d[l], net->first, n - net->first);
                const uint8_t *in = st;
                for (int k = E - 1; k >= 0; k--) /* last to first: the first entry of an edge is the one that stays */
                    if (edges[k] != 0xFFFFFFFFu && (int)(edges[k] & 0xFFFu) == i && (int)((edges[k] >> 12) & 0xFFFu) < n) {
                        if (in == st) { memcpy(seen, st, (size_t)n); in = seen; }
                        seen[(edges[k] >> 12) & 0xFFFu] = (uint8_t)((edges[k] >> 24) & 1u);
                    }
                const int v = net->kind == ORC_TT ? tt_next_value(net, in, i, &d[l]) : pred_next_value(net, in, i, &d[l]);
                st[i] = (uint8_t)(pin[i] == 0 || pin[i] == 1 ? pin[i] : v); /* rule 2 */
            }
        }
        free(seen);
    }
    for (int t = 0; t < nthreads; t++) for (int64_t b = 0; b < nb; b++) hist[b] += priv[t * nb + b];
    free(priv);
    return 0;
}
