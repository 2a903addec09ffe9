// pbn_coop.cuh — group-cooperative runner of the step-until-attractor loop (predictor networks, Philox draws).
//
//   while not is_attracting_state(state): graph.step()      pbn_target.py:270-271, pbn_target_multi.py:135-146
//
// The loop is strictly serial per env and heavy-tailed (1 .. 40 000 updates, SURVEY.md §0.9); a launch lasts as long as its
// slowest env, so what matters for that env is the LATENCY of one update.  An asynchronous update has two halves:
//   * the DRAW half depends only on the env's Philox stream: node index, predictor choice (threshold row compare), the
//     predictor's record (four input positions + LUT).  No state input.
//   * the STATE half: four bit extracts, one LUT bit, one bit insert — and the attractor test of the new state.
// A group of g lanes (g = 4, 8, 16 or 32; 32/g groups per warp, each on its own env) splits them: in phase A every lane
// computes TWO Philox blocks of the env's update stream and turns their four updates into four 32-byte ENTRIES in a per-warp
// staging buffer, everything pre-digested (rotate amounts that drop input j's bit on bit 3-j of the LUT index, the LUT
// doubled and pre-rotated so that ONE rotate by the index lands the wanted bit on the node's position, the node's bit mask,
// shared-memory addresses for multi-word states).  In phase B all lanes of the group apply the 4g entries in order,
// redundantly, on the same state: five dependent ALU instructions per update for a one-word network (SHF, LOP3, LOP3, SHF,
// LOP3), plus one shared-memory round trip for larger ones.  The attractor test is OFF that chain: the lanes share out the
// cubes, each records the first entry at which one of its cubes matched, and the updates run on speculatively to the end of
// the batch; a group minimum then gives the stop entry (first match or the inner-step cap) and the group replays the
// batch's first entries from a checkpoint to land on the exact stopping state.  The words consumed are the ones the
// one-lane loop takes (update t of the stream uses words 2t, 2t+1), so the result is bit-identical to it and to the oracle.
#pragma once

#define PBN_COOP_NB 2            // Philox blocks per lane and batch (two chains in flight: the latency of one)
#define PBN_COOP_ENTRIES (32 * 2 * PBN_COOP_NB)  // per warp: two per Philox block
#define PBN_COOP_ENTRY_BYTES 32  // {g0, g1, g2, g3} {Lrot, mask, word address, cube word offset}
// per-warp staging bytes: the entries (+ 16 bytes of padding per group: the groups of a warp read the same entry index at the
// same time, and regions a multiple of 128 bytes apart would put all those 16-byte reads on the same four banks) + one
// checkpoint column (w32 words) for each of up to 16 groups
#define PBN_COOP_GROUPS_MAX 16   // groups of two lanes: the throughput end of the trade (resume passes with long lists)
#define PBN_COOP_ENT_BYTES (PBN_COOP_ENTRIES * PBN_COOP_ENTRY_BYTES + PBN_COOP_GROUPS_MAX * 16)
__host__ __device__ inline int coop_warp_bytes(int w32) { return PBN_COOP_ENT_BYTES + ((PBN_COOP_GROUPS_MAX * w32 * 4 + 15) & ~15); }

__device__ __forceinline__ uint4 lds_v4(u32 a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint2 lds_v2(u32 a) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts_v4(u32 a, const uint4 v) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" :: "r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ u32 rotr32(u32 x, u32 s) { return __funnelshift_r(x, x, s); }  // by s & 31
// (a & c) | (b & ~c) as ONE LOP3 the compiler cannot re-associate: the merges below are a two-level tree, not a chain
__device__ __forceinline__ u32 bitsel(u32 a, u32 b, u32 c) {
    u32 d;
    asm("lop3.b32 %0, %1, %2, %3, 0xE4;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// #{k : t[k] <= r} for an ascending quad of thresholds (cumulative COD rows are ascending, so the predicates are monotone
// and a select chain replaces the sum)
__device__ __forceinline__ u32 count_le(const uint4 t, u32 r) {
    u32 j;
    asm("{ .reg .pred p0, p1, p2, p3;\n\t"
        "setp.le.u32 p0, %1, %5; setp.le.u32 p1, %2, %5; setp.le.u32 p2, %3, %5; setp.le.u32 p3, %4, %5;\n\t"
        "selp.u32 %0, 1, 0, p0; selp.u32 %0, 2, %0, p1; selp.u32 %0, 3, %0, p2; selp.u32 %0, 4, %0, p3; }"
        : "=r"(j) : "r"(t.x), "r"(t.y), "r"(t.z), "r"(t.w), "r"(r));
    return j;
}
// index of the predictor selected by the 31-bit draw r (bittner/base.py:94-97): first k with r < cum_k, else the last
template <int TQ>
__device__ __forceinline__ u32 pred_pick(const NetView &nv, const unsigned char *blob, u32 i, u32 r) {
    const uint4 *thr = reinterpret_cast<const uint4 *>(blob + nv.off_thr) + i * nv.tsq_stride;
    const int nq = TQ > 0 ? TQ : (nv.ts >> 2);
    if (nq == 1) return count_le(thr[0], r);
    if (nq <= 4) {  // leading quad = last threshold of each quad (pbn_device.cuh: pred_next)
        u32 q = count_le(thr[0], r);
        q = q < (u32)(nq - 1) ? q : (u32)(nq - 1);
        return 4u * q + count_le(thr[1 + q], r);
    }
    u32 j = 0;
    for (int q = 0; q < nq; q++) j += count_le(thr[q], r);
    return j;
}

// DRAW half of one update -> one entry.  wa picks the node, wb the predictor (words 2t, 2t+1 of the update stream).
// `on` = false writes a zero bit mask and points the entry's read-modify-write at its own pad word: it is applied like any
// other entry and touches no state (an idle group must not write back a stale word of a column another group is updating).
template <int TQ, bool W1>
__device__ __forceinline__ void coop_entry(const NetView &nv, const unsigned char *blob, u32 col, u32 wa, u32 wb, u32 dst, bool on,
                                           uint4 &a, uint4 &b) {
    const u32 i = (u32)nv.first + __umulhi(wa, (u32)(nv.n - nv.first));
    const u32 j = pred_pick<TQ>(nv, blob, i, wb >> 1);
    const uint2 rec = reinterpret_cast<const uint2 *>(blob + nv.off_rec)[i * nv.fmax + j];
    const u32 p0 = rec.x & 0xFFu, p1 = (rec.x >> 8) & 0xFFu, p2 = (rec.x >> 16) & 0xFFu, p3 = rec.x >> 24;
    const u32 l32 = (rec.y & 0xFFFFu) * 0x10001u;  // the LUT twice: bit 4 of the index may be garbage
    if constexpr (W1) {  // rotate right by p + k - 3 (mod 32) drops bit p on bit 3 - k; the funnel shift reads 5 bits
        a.x = p0 + 29u; a.y = p1 + 30u; a.z = p2 + 31u; a.w = p3;
    } else {             // bits 31..8: shared address of the input's state word, bits 4..0: rotate amount
        a.x = ((col + ((p0 >> 5) << 10)) << 8) | ((p0 + 29u) & 31u);
        a.y = ((col + ((p1 >> 5) << 10)) << 8) | ((p1 + 30u) & 31u);
        a.z = ((col + ((p2 >> 5) << 10)) << 8) | ((p2 + 31u) & 31u);
        a.w = ((col + ((p3 >> 5) << 10)) << 8) | (p3 & 31u);
    }
    b.x = __funnelshift_l(l32, l32, i);  // rotl by i & 31: rotr(b.x, idx) has LUT bit idx on bit i & 31
    b.y = on ? (1u << (i & 31u)) : 0u;
    b.z = on ? col + ((i >> 5) << 10) : dst + 28u;
    b.w = on ? (i >> 5) * 8u : 0u;       // byte offset of the node's (care, value) pair inside a cube
}

// STATE half: LUT index from four rotated words (two-level merge), one rotate of the prepared LUT, one masked merge
__device__ __forceinline__ u32 coop_merge(u32 r0, u32 r1, u32 r2, u32 r3, u32 lrot, u32 m, u32 old) {
    const u32 idx = bitsel(bitsel(r0, r1, 8u), bitsel(r2, r3, 2u), 12u);
    return bitsel(rotr32(lrot, idx), old, m);
}

// Per-lane attractor test of a multi-word state, kept incrementally: mm = number of cared positions at which the state
// differs from this lane's cube; an update changes at most one position, so mm moves by -1, 0 or +1 and the state matches
// iff mm == 0.  Lanes without a cube start from a count no batch can bring to zero.
struct CoopCube {
    u32 addr, addr1;  // shared addresses of the lane's two cubes: (care, value) word pairs
    int mm, mm1;
};

// One batch entry after the other: test the state BEFORE the entry (off the dependent chain), then apply it.  Every lane
// tests its cube `sub` (TWO: and cube sub + g; EXTRA: more than 2g cubes, the surplus is tested directly).  Returns the first
// entry whose before-state matched.  The next entry is fetched one trip ahead at a constant offset — past the last entry that
// reads the neighbouring group's first entry or the checkpoint area, never used.
template <bool W1, bool TWO, bool EXTRA>
__device__ __forceinline__ int coop_phase_b(u32 ebuf, int E, u32 &st, u32 col, u32 care0, u32 val0, u32 care1, u32 val1, CoopCube &cc,
                                            const u32 *cubes, int n_cubes, int w32, int g, u32 sub) {
    int first = E;
    uint4 ea = lds_v4(ebuf), eb = lds_v4(ebuf + 16u);
    for (int e0 = 0; e0 < E; e0 += 4) {
        const u32 eb0 = ebuf + (u32)e0 * PBN_COOP_ENTRY_BYTES;
        u32 m4 = 0u;  // bit k: the state before entry e0 + k matched
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint4 na = lds_v4(eb0 + (k + 1) * PBN_COOP_ENTRY_BYTES), nb = lds_v4(eb0 + (k + 1) * PBN_COOP_ENTRY_BYTES + 16u);
            if constexpr (W1) {
                bool hit = (st & care0) == val0;
                if constexpr (TWO) hit |= (st & care1) == val1;
                if constexpr (EXTRA)
                    for (int c = (int)sub + 2 * g; c < n_cubes; c += g) hit |= (st & cubes[2 * c]) == cubes[2 * c + 1];
                if (hit) m4 |= 1u << k;
                st = coop_merge(rotr32(st, ea.x), rotr32(st, ea.y), rotr32(st, ea.z), rotr32(st, ea.w), eb.x, eb.y, st);
            } else {
                bool hit = cc.mm == 0;
                if constexpr (TWO) hit |= cc.mm1 == 0;
                if constexpr (EXTRA)
                    for (int c = (int)sub + 2 * g; c < n_cubes; c += g) {
                        const u32 *pc = cubes + (size_t)c * w32 * 2;
                        bool ok = true;
                        for (int w = 0; w < w32; w++) ok &= (lds_u32(col + 1024u * w) & pc[2 * w]) == pc[2 * w + 1];
                        hit |= ok;
                    }
                if (hit) m4 |= 1u << k;
                const uint2 cw = lds_v2(cc.addr + eb.w);  // (care, value) of the word the entry writes
                const u32 w0 = lds_u32(ea.x >> 8), w1 = lds_u32(ea.y >> 8), w2 = lds_u32(ea.z >> 8), w3 = lds_u32(ea.w >> 8);
                const u32 old = lds_u32(eb.z);
                const u32 nw = coop_merge(rotr32(w0, ea.x), rotr32(w1, ea.y), rotr32(w2, ea.z), rotr32(w3, ea.w), eb.x, eb.y, old);
                sts_u32(eb.z, nw);
                const u32 flip = old ^ nw;                     // the written bit, if it changed
                cc.mm += (flip & cw.x) ? (((nw ^ cw.y) & eb.y) ? 1 : -1) : 0;  // the cube cares: one mismatch more or one fewer
                if constexpr (TWO) {
                    const uint2 cv = lds_v2(cc.addr1 + eb.w);
                    cc.mm1 += (flip & cv.x) ? (((nw ^ cv.y) & eb.y) ? 1 : -1) : 0;
                }
            }
            ea = na; eb = nb;
        }
        if (m4 != 0u && first == E) first = e0 + __ffs((int)m4) - 1;
    }
    return first;
}

// Runs the loop for 32/g envs at once, group r (lanes r*g .. r*g+g-1) on the env whose column is col_ptr (group-uniform,
// like env_id, in, stop_in, pos_base and active).  pos_base = updates the env's stream had served before this env.step
// began: update number `in` of the step takes words 2*(pos_base + in), +1.  A group stops at the first attracting state or
// when its count reaches stop_in (the inner-step cap, or less under a budget).  Returns the group's update count.  The call returns when
// `exit_at` groups have stopped since it began (1: at the first, so the caller can re-form wider groups) or none is left.
// wbuf: coop_warp_bytes(w32) bytes of shared memory owned by this warp, 16-byte aligned.
template <int TQ, bool W1>
__device__ __forceinline__ int coop_steps(const NetView &nv, const EnvView &ev, const DrawView &dv, const unsigned char *blob,
                                          const int *att_off, const u32 *cubes, u32 *col_ptr, long long env_id, int in,
                                          int stop_in, bool active, int g, u32 pos_base, unsigned char *wbuf, int exit_at) {
    const u32 lane = threadIdx.x & 31u;
    const u32 sub = lane & (u32)(g - 1), gbase = lane & ~(u32)(g - 1);
    const u32 gmask = (g == 32 ? 0xFFFFFFFFu : ((1u << g) - 1u)) << gbase;
    const int w32 = nv.w32;
    const int E = 2 * PBN_COOP_NB * g;
    const u32 lane_ent = (2u * PBN_COOP_NB) * PBN_COOP_ENTRY_BYTES;  // bytes of entries per lane
    const u32 grp_idx = gbase >> (__ffs(g) - 1);
    const u32 ebuf = smem_addr(wbuf) + gbase * lane_ent + grp_idx * 16u;
    const u32 ckp = smem_addr(wbuf) + PBN_COOP_ENT_BYTES + grp_idx * (u32)w32 * 4u;
    const u32 col = smem_addr(col_ptr);
    const int n_cubes = att_off[ev.n_att];
    const bool has_cube = (int)sub < n_cubes, has_cube1 = (int)sub + g < n_cubes;
    // one-word networks: this lane's two cubes in registers (care 0 / value 1 never matches)
    u32 care0 = 0u, val0 = 1u, care1 = 0u, val1 = 1u;
    if (W1 && has_cube) { care0 = cubes[2 * sub]; val0 = cubes[2 * sub + 1]; }
    if (W1 && has_cube1) { care1 = cubes[2 * (sub + g)]; val1 = cubes[2 * (sub + g) + 1]; }
    // larger ones: mismatch counts of the entry state; from here on they follow the updates (a lane without a cube reads
    // cube 0 and counts from a value no launch brings to zero)
    const u32 c0 = has_cube ? sub : 0u, c1 = has_cube1 ? sub + (u32)g : 0u;
    CoopCube cc{smem_addr(cubes) + c0 * (u32)w32 * 8u, smem_addr(cubes) + c1 * (u32)w32 * 8u, 1 << 24, 1 << 24};
    u32 st = W1 ? *col_ptr : 0u;
    if constexpr (!W1) {
        int mm = 0, mm1 = 0;
        for (int w = 0; w < w32; w++) {
            const u32 sw = col_ptr[w * PBN_BLOCK];
            mm += __popc((sw ^ cubes[(c0 * w32 + w) * 2 + 1]) & cubes[(c0 * w32 + w) * 2]);
            mm1 += __popc((sw ^ cubes[(c1 * w32 + w) * 2 + 1]) & cubes[(c1 * w32 + w) * 2]);
        }
        if (has_cube) cc.mm = mm;
        if (has_cube1) cc.mm1 = mm1;
    }
    bool running = active;
    int n_stopped = 0;
    unsigned live = __ballot_sync(0xFFFFFFFFu, running);
    for (;;) {
        // ---- phase A: 4g updates' worth of the stream, from the even update at or before position p
        const u32 p = pos_base + (u32)in, u0 = p & 1u;
        {
            u32 x[PBN_COOP_NB][4];
#pragma unroll
            for (int k = 0; k < PBN_COOP_NB; k++)
                philox4x32_10_rk((p >> 1) + sub * PBN_COOP_NB + k, dv.epoch, (u32)env_id, (u32)((u64)env_id >> 32), dv, x[k][0], x[k][1],
                                 x[k][2], x[k][3]);
            // the entries are computed first and stored together: the stores (volatile asm) would otherwise fence the table
            // loads of the next entry behind them and serialise four chains that can run side by side
            uint4 ea[2 * PBN_COOP_NB], eb[2 * PBN_COOP_NB];
            const u32 dst = ebuf + sub * lane_ent;
#pragma unroll
            for (int k = 0; k < PBN_COOP_NB; k++) {
                coop_entry<TQ, W1>(nv, blob, col, x[k][0], x[k][1], dst + (2 * k) * PBN_COOP_ENTRY_BYTES,
                                   running && !(k == 0 && sub == 0u && u0 != 0u), ea[2 * k], eb[2 * k]);
                coop_entry<TQ, W1>(nv, blob, col, x[k][2], x[k][3], dst + (2 * k + 1) * PBN_COOP_ENTRY_BYTES, running, ea[2 * k + 1],
                                   eb[2 * k + 1]);
            }
#pragma unroll
            for (int k = 0; k < 2 * PBN_COOP_NB; k++) {
                sts_v4(dst + k * PBN_COOP_ENTRY_BYTES, ea[k]);
                sts_v4(dst + k * PBN_COOP_ENTRY_BYTES + 16u, eb[k]);
            }
        }
        const u32 ck = st;  // checkpoint of the state the batch starts from
        if constexpr (!W1)
            for (int w = (int)sub; w < w32; w += g) sts_u32(ckp + 4u * w, lds_u32(col + 1024u * w));
        __syncwarp();
        // ---- phase B
        int first;
        if (n_cubes <= g) first = coop_phase_b<W1, false, false>(ebuf, E, st, col, care0, val0, care1, val1, cc, cubes, n_cubes, w32, g, sub);
        else if (n_cubes <= 2 * g) first = coop_phase_b<W1, true, false>(ebuf, E, st, col, care0, val0, care1, val1, cc, cubes, n_cubes, w32, g, sub);
        else first = coop_phase_b<W1, true, true>(ebuf, E, st, col, care0, val0, care1, val1, cc, cubes, n_cubes, w32, g, sub);
        // ---- stop entry: first match of any lane's cubes, or the entry at which the cap is reached
        int cap = stop_in - in;
        cap = (cap < 0 ? 0 : cap) + (int)u0;
        first = first < cap ? first : cap;
        if (g == 32) first = __reduce_min_sync(0xFFFFFFFFu, first);
        else
            for (int o = 1; o < g; o <<= 1) {  // a group-masked REDUX runs once per distinct mask: butterflies are cheaper
                const int other = __shfl_xor_sync(0xFFFFFFFFu, first, o);
                first = other < first ? other : first;
            }
        const bool stop = running && first < E;
        if (stop) {  // replay entries [0, ks) from the checkpoint (entry 0 is a no-op when the batch began at an odd update)
            const int ks = first < (int)u0 ? (int)u0 : first;
            if constexpr (W1) {
                st = ck;
                for (int e = 0; e < ks; e++) {
                    const u32 ex = ebuf + (u32)e * PBN_COOP_ENTRY_BYTES;
                    const uint4 ea = lds_v4(ex), eb = lds_v4(ex + 16u);
                    st = coop_merge(rotr32(st, ea.x), rotr32(st, ea.y), rotr32(st, ea.z), rotr32(st, ea.w), eb.x, eb.y, st);
                }
            } else {
                for (int w = (int)sub; w < w32; w += g) sts_u32(col + 1024u * w, lds_u32(ckp + 4u * w));
                __syncwarp(gmask);
                for (int e = 0; e < ks; e++) {
                    const u32 ex = ebuf + (u32)e * PBN_COOP_ENTRY_BYTES;
                    const uint4 ea = lds_v4(ex), eb = lds_v4(ex + 16u);
                    const u32 w0 = lds_u32(ea.x >> 8), w1 = lds_u32(ea.y >> 8), w2 = lds_u32(ea.z >> 8), w3 = lds_u32(ea.w >> 8);
                    const u32 old = lds_u32(eb.z);
                    sts_u32(eb.z, coop_merge(rotr32(w0, ea.x), rotr32(w1, ea.y), rotr32(w2, ea.z), rotr32(w3, ea.w), eb.x, eb.y, old));
                }
            }
            in += ks - (int)u0;
            running = false;
        } else if (running) {
            in += E - (int)u0;
        }
        const unsigned now = __ballot_sync(0xFFFFFFFFu, running);
        n_stopped += __popc(live & ~now) >> (__ffs(g) - 1);  // whole groups leave together
        live = now;
        __syncwarp();  // every read of the batch's entries precedes the next batch's writes
        if (live == 0u || n_stopped >= exit_at) break;
    }
    if (W1 && active) *col_ptr = st;  // every lane of the group holds the same word
    return in;
}

// Hands the envs of the lanes in `hv` (a ballot of the warp) to lane groups, all at once: k groups of 32/k lanes, k the least
// power of two >= the number of envs, group r on the env of the r-th lane of hv.  Every lane passes its own env's id, update count `in`, stream base
// (coop_steps: pos_base) and stop_in; the owners' values are used.  sst: the block's state columns (lane l's at sst + l within
// its warp), coop_buf: the block's staging, coop_warp_bytes(w32) per warp.  Returns the owner's new update count, and `in`
// to every other lane.
template <int TQ, bool W1>
__device__ __forceinline__ int coop_take_over(unsigned hv, const NetView &nv, const EnvView &ev, const DrawView &dv,
                                              const unsigned char *blob, const int *att_off, const u32 *cubes, u32 *sst,
                                              unsigned char *coop_buf, long long id, int in, u32 base, int stop_in, int exit_at) {
    const u32 lane = threadIdx.x & 31u;
    const int nl = __popc(hv);
    int k = 1;
    while (k < nl) k <<= 1;
    const int g = 32 / k;  // lanes per group
    const int grp = (int)lane / g;
    const bool on = grp < nl;
    const int owner = on ? (int)__fns(hv, 0u, grp + 1) : 0;  // the grp-th lane of hv
    const long long idL = __shfl_sync(0xFFFFFFFFu, id, owner);
    const int inL = __shfl_sync(0xFFFFFFFFu, in, owner);
    const u32 baseL = __shfl_sync(0xFFFFFFFFu, base, owner);
    const int stopL = __shfl_sync(0xFFFFFFFFu, stop_in, owner);
    u32 *colL = sst + (threadIdx.x & ~31u) + (u32)owner;
    unsigned char *wb = coop_buf + (threadIdx.x >> 5) * coop_warp_bytes(nv.w32);
    const int fin = coop_steps<TQ, W1>(nv, ev, dv, blob, att_off, cubes, colL, idL, inL, stopL, on, g, baseL, wb, exit_at);
    __syncwarp();
    int out = in;
#pragma unroll 1  // (unrolled, its __fns calls add ~4 % to the kernel's code)
    for (int r = 0; r < nl; r++) {  // each group's count back to the lane that owns the env
        const int v = __shfl_sync(0xFFFFFFFFu, fin, r * g);
        if ((int)lane == (int)__fns(hv, 0u, r + 1)) out = v;
    }
    __syncwarp();
    return out;
}
