/*
 * passage_oracle.c — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * The oracle's first-passage loop: the CPU restatement that tests/test_gpu_passage.py compares pbn_first_passage against.
 * It is compiled together with oracle/pbn_oracle.c (same translation unit, see tests/passage_oracle.py) so that it uses
 * the oracle's own Philox streams, node updates and geometric gaps, byte per node, and shares nothing with the product.
 * The loop is orc_ssd_pinned_edges's (tests/edge_pin_oracle.c, rules 1-4 there) with the histogram count replaced by a
 * membership test of the current bucket in a list of goal buckets; tests/test_oracle_passage.py checks it against
 * orc_ssd_pinned_edges run for t iterations.
 */
#include "pbn_oracle.c"

/* One variant per call (pin[i] = 0 or 1 pins node i, edges[0..E) as in orc_ssd_pinned_edges), PHILOX draws, env = NULL.
   t_hit[e] >= 0 on entry: chain e has arrived; its entry and its state are left as they are.  Any other chain e runs
   `iters` iterations; at iteration t, before the perturbation, a bucket found in goal[0..ngoal) sets t_hit[e] = t0 + t the
   first time.  Every chain runs through all iterations (the kernel stops a warp whose chains have all arrived, so the state
   of a chain that arrived is not compared).  Chain e draws from the streams of global id env0 + e.  Returns 1 for a
   misaligned env0, 2 for replay draws. */
int orc_first_passage(const OrcNet *net, uint8_t *state, int64_t chains, int64_t env0, int64_t iters, int64_t t0, double p,
                      const int8_t *pin, const uint32_t *edges, int E, const int32_t *tgt_nodes, int g, const int64_t *goal,
                      int ngoal, int64_t *t_hit, const OrcDraws *dr) {
    const int n = net->n;
    const float inv = orc_geom_inv(p);
    const int flips = !(inv > 0);
    const uint32_t W = (uint32_t)n * 32u, NONE = 0xFFFFFFFFu;
    if (dr->mode != ORC_PHILOX) return 2;
    if (flips && (env0 & 31)) return 1;
    uint8_t *keep = (uint8_t *)malloc((size_t)(chains * n + 1)), *arrived = (uint8_t *)malloc((size_t)(chains + 1));
    memcpy(keep, state, (size_t)(chains * n));
    for (int64_t e = 0; e < chains; e++) arrived[e] = t_hit[e] >= 0;
    for (int64_t e = 0; e < chains; e++)
        for (int i = 0; i < n; i++)
            if (pin[i] == 0 || pin[i] == 1) state[e * n + i] = (uint8_t)pin[i];
    const int64_t groups = (chains + 31) / 32;
#pragma omp parallel for schedule(static) if (chains >= 256)
    for (int64_t gi = 0; gi < groups; gi++) {
        uint8_t *seen = (uint8_t *)malloc((size_t)n);
        const int64_t gb = gi * 32;
        int live[32];
        Dr d[32], dp[32];
        uint32_t ev[64], last_p1 = 0;
        for (int l = 0; l < 32; l++) {
            live[l] = gb + l < chains && !arrived[gb + l];
            dr_init(&d[l], dr, gb + l < chains ? gb + l : 0, env0 + gb + l);
            dp[l] = d[l];
            dp[l].ctr[0] = 0x80000000u;
            ev[2 * l] = ev[2 * l + 1] = NONE;
        }
        for (int64_t t = 0; t < iters; t++) {
            for (int l = 0; l < 32 && gb + l < chains; l++) {
                if (!live[l]) continue;
                const uint8_t *st = state + (gb + l) * n;
                int64_t b = 0;
                for (int k = 0; k < g; k++) b = (b << 1) | st[tgt_nodes[k]];
                for (int k = 0; k < ngoal; k++)
                    if (goal[k] == b) {
                        t_hit[gb + l] = t0 + t;
                        live[l] = 0;
                        break;
                    }
            }
            if (flips) {
                for (;;) {
                    for (int k = 0; k < 64; k++)
                        if (ev[k] < W) {
                            uint32_t tl = ev[k] & 31u, bit = ev[k] >> 5;
                            if (gb + tl < chains && pin[bit] != 0 && pin[bit] != 1) state[(gb + tl) * n + bit] ^= 1;
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
                for (int k = E - 1; k >= 0; k--)
                    if (edges[k] != 0xFFFFFFFFu && (int)(edges[k] & 0xFFFu) == i && (int)((edges[k] >> 12) & 0xFFFu) < n) {
                        if (in == st) { memcpy(seen, st, (size_t)n); in = seen; }
                        seen[(edges[k] >> 12) & 0xFFFu] = (uint8_t)((edges[k] >> 24) & 1u);
                    }
                const int v = net->kind == ORC_TT ? tt_next_value(net, in, i, &d[l]) : pred_next_value(net, in, i, &d[l]);
                st[i] = (uint8_t)(pin[i] == 0 || pin[i] == 1 ? pin[i] : v);
            }
        }
        free(seen);
    }
    for (int64_t e = 0; e < chains; e++) /* arrived before this call: state untouched */
        if (arrived[e]) memcpy(state + e * n, keep + e * n, (size_t)n);
    free(keep);
    free(arrived);
    return 0;
}
