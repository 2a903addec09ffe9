/*
 * pinned_oracle.c — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * The oracle's SSD with genes pinned: the CPU restatement that tests/test_gpu_pinned_ssd.py compares pbn_ssd_pinned
 * against.  It is compiled together with oracle/pbn_oracle.c (same translation unit, see tests/pinned_oracle.py) so that it
 * uses the oracle's own Philox streams, node updates and geometric gaps, byte per node, and shares nothing with the product.
 */
#include "pbn_oracle.c"

/* orc_ssd with a pin set, env = NULL, PHILOX draws (pbn_ssd_pinned, one variant per call): pin[i] = 0 or 1 holds node i at
   that value, any other value leaves it free.
     1. before the first iteration every pinned node is set to its value;
     2. an update that picks a pinned node consumes its draws (node index, predictor or table draw) and the node keeps its value;
     3. a perturbation event on a pinned node is drawn and not applied.
   Chain e draws from the streams of global id env0 + e, as in orc_ssd.  Returns 1 for a misaligned env0, 2 for replay draws. */
int orc_ssd_pinned(const OrcNet *net, uint8_t *state, int64_t chains, int64_t env0, int64_t iters, double p, const int8_t *pin,
                   const int32_t *tgt_nodes, int g, uint64_t *hist, const OrcDraws *dr) {
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
                const int v = net->kind == ORC_TT ? tt_next_value(net, st, i, &d[l]) : pred_next_value(net, st, i, &d[l]);
                st[i] = (uint8_t)(pin[i] == 0 || pin[i] == 1 ? pin[i] : v); /* rule 2 */
            }
        }
    }
    for (int t = 0; t < nthreads; t++) for (int64_t b = 0; b < nb; b++) hist[b] += priv[t * nb + b];
    free(priv);
    return 0;
}
