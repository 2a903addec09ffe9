// pbn_b200.cu — sm_100a kernels and the C-ABI of libpbn_b200.so (see include/pbn_b200.h).
//
// Thread-per-env kernels; the packed network image and the cube tables are staged once per block into
// shared memory, each env's bit-packed state lives in a shared-memory column for the whole launch, so a
// rollout / SSD launch touches HBM only for 2*W32 words per env plus the histogram.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "pbn_device.cuh"

// ----------------------------------------------------------------------------------------------- errors
static thread_local std::string g_err;
static int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
// A failed runtime call also stays the thread's last error; it is consumed here, so that it cannot surface as the failure of a
// later call's cudaGetLastError().
#define CK(call)                                                                                     \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess) {                                                                     \
            cudaGetLastError();                                                                      \
            return fail(PBN_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));           \
        }                                                                                            \
    } while (0)

int pbn_fail_(int code, const std::string &msg) { return fail(code, msg); }  // for the other translation units
extern "C" const char *pbn_last_error(void) { return g_err.c_str(); }
extern "C" const char *pbn_version(void) { return "pbn_b200 0.1 (sm_100a)"; }

#ifndef PBN_REC16_MAX
#define PBN_REC16_MAX (32 * 1024)  // predictor networks get the 16-byte fast-path records when they fit this many bytes
#endif
#ifndef PBN_TT_THR_SMEM_MAX
#define PBN_TT_THR_SMEM_MAX (16 * 1024)
#endif

// ----------------------------------------------------------------------------------------------- handles
struct PbnNet {
    NetView v;
    std::vector<void *> owned;
    u32 tt_const;  // TT: index (in the threshold table) of two constant entries, 0 (never 1) and 2^31 (always 1)
};
struct PbnEnv {
    EnvView v;
    const PbnNet *net;
    std::vector<void *> owned;
    bool has_small_att;  // some attractor has at most 10 states: the PBN family's reset loop terminates
};

template <class T>
static int upload(std::vector<void *> &owned, const T *host, size_t count, const T **dev) {
    void *p = nullptr;
    size_t bytes = (count ? count : 1) * sizeof(T);
    CK(cudaMalloc(&p, bytes));
    owned.push_back(p);
    if (count) CK(cudaMemcpy(p, host, count * sizeof(T), cudaMemcpyHostToDevice));
    *dev = static_cast<const T *>(p);
    return PBN_OK;
}

static inline u32 thr31(double p) {  // smallest T with (r31 < T) <=> (r31 / 2^31 < p)
    double t = std::ceil(p * 2147483648.0);
    if (!(t > 0)) return 0;
    if (t > 2147483648.0) t = 2147483648.0;
    return (u32)t;
}

// Network compiler back end (host): reference-form tables -> packed image.
extern "C" int pbn_net_create(const PbnNetDesc *d, PbnNet **out) {
    if (!d || !out) return fail(PBN_ERR_ARG, "null argument");
    const int n = d->n_nodes;
    if (n < 1) return fail(PBN_ERR_ARG, "n_nodes < 1");
    if (d->first_updatable < 0 || d->first_updatable >= n) return fail(PBN_ERR_ARG, "first_updatable out of range");
    PbnNet *net = new PbnNet();
    NetView &v = net->v;
    memset(&v, 0, sizeof v);
    v.kind = d->kind; v.n = n; v.first = d->first_updatable; v.w32 = (n + 31) / 32;
    std::vector<unsigned char> blob;
    int rc = PBN_OK;
    if (d->kind == PBN_NET_PRED) {
        if (n > 256) { delete net; return fail(PBN_ERR_UNSUPPORTED, "predictor networks support at most 256 nodes"); }
        int fmax = 0;
        for (int i = 0; i < n; i++) {
            int f = d->pr_off[i + 1] - d->pr_off[i];
            if (f < 1) { delete net; return fail(PBN_ERR_ARG, "node without predictors"); }
            fmax = f > fmax ? f : fmax;
        }
        const int ts = ((fmax - 1 + 3) / 4) * 4 > 0 ? ((fmax - 1 + 3) / 4) * 4 : 4;
        v.fmax = fmax; v.ts = ts;
        // one quad (up to 5 predictors): the row IS the quad.  More: the row starts with a quad holding the LAST threshold
        // of each threshold quad, so that the search is two 16-byte loads (which quad, then where in it) however many
        // predictors a node has — divergent 16-byte loads cost four shared-memory wavefronts each
        const int lead = (ts > 4 && ts <= 16) ? 1 : 0;
        v.tsq_stride = (lead + ts / 4) | 1;  // odd number of quads per row (bank-conflict padding)
        const int row = v.tsq_stride * 4;
        v.off_thr = 0;
        v.off_rec = n * row * 4;
        blob.resize((size_t)v.off_rec + (size_t)n * fmax * 8);
        u32 *thr = reinterpret_cast<u32 *>(blob.data());
        uint2 *rec = reinterpret_cast<uint2 *>(blob.data() + v.off_rec);
        for (int i = 0; i < n; i++) {
            const int q0 = d->pr_off[i], f = d->pr_off[i + 1] - q0;
            for (int k = 0; k < row; k++) thr[i * row + k] = 0x80000000u;
            for (int k = 1; k < f; k++)  // the threshold search (count / select chain) relies on ascending rows
                if (!(d->pr_cum[q0 + k] >= d->pr_cum[q0 + k - 1])) { delete net; return fail(PBN_ERR_ARG, "cumulative COD must be non-decreasing (negative COD?)"); }
            for (int k = 0; k < ts; k++) {
                const u32 t = (k < f - 1) ? thr31(d->pr_cum[q0 + k] / d->pr_codsum[i]) : 0x80000000u;
                thr[i * row + lead * 4 + k] = t;
                if (lead && (k & 3) == 3) thr[i * row + (k >> 2)] = t;
            }
            for (int k = 0; k < fmax; k++) {
                const int q = q0 + (k < f ? k : f - 1);
                u32 packed = 0;
                for (int j = 0; j < 4; j++) {
                    int idx = d->pr_in[4 * q + j];
                    if (idx < 0 || idx >= n) { delete net; return fail(PBN_ERR_ARG, "predictor input out of range"); }
                    packed |= (u32)idx << (8 * j);
                }
                rec[i * fmax + k] = make_uint2(packed, d->pr_lut[q]);
            }
        }
        if ((size_t)n * fmax * 16 <= PBN_REC16_MAX) {
            // 16-byte records of the fast asynchronous paths (ssd_fast_update), appended to the image and staged only by
            // them: x = f0 | f1 << 16, y = f2 | f3 << 16 with f_j = (word of input j) << 10 | rotate amount that brings the
            // input's bit to position 3 - j; z = the 16-bit LUT in both halves (the index may carry garbage in bit 4); w = 0
            v.off_rec16 = (int)((blob.size() + 15) & ~(size_t)15);
            blob.resize((size_t)v.off_rec16 + (size_t)n * fmax * 16);
            uint4 *r16 = reinterpret_cast<uint4 *>(blob.data() + v.off_rec16);
            const uint2 *r8 = reinterpret_cast<const uint2 *>(blob.data() + v.off_rec);
            for (int q = 0; q < n * fmax; q++) {
                u32 fld[4];
                for (int j = 0; j < 4; j++) {
                    const u32 pj = (r8[q].x >> (8 * j)) & 0xFFu;
                    fld[j] = ((pj >> 5) << 10) | (((pj & 31u) - (3u - (u32)j)) & 31u);
                }
                const u32 lut = r8[q].y & 0xFFFFu;
                r16[q] = make_uint4(fld[0] | (fld[1] << 16), fld[2] | (fld[3] << 16), lut | (lut << 16), 0u);
            }
        }
        if (fmax <= 5) {  // mask table of the bit-sliced synchronous kernel
            const int lrow = fmax * 16 + 4;  // +16 B per node: consecutive nodes (lanes) start in different bank groups
            std::vector<u32> lm((size_t)n * lrow, 0u);
            for (int i = 0; i < n; i++) {
                const int q0 = d->pr_off[i], f = d->pr_off[i + 1] - q0;
                for (int k = 0; k < fmax; k++) {
                    const int q = q0 + (k < f ? k : f - 1);
                    for (int b = 0; b < 16; b++) lm[(size_t)i * lrow + k * 16 + b] = ((d->pr_lut[q] >> b) & 1) ? 0xFFFFFFFFu : 0u;
                }
            }
            rc |= upload(net->owned, lm.data(), lm.size(), &v.lutmask);
        }
        const int np = d->pr_off[n];
        rc |= upload(net->owned, d->pr_off, (size_t)n + 1, &v.pr_off);
        rc |= upload(net->owned, d->pr_cum, (size_t)np, &v.pr_cum);
        rc |= upload(net->owned, d->pr_codsum, (size_t)n, &v.pr_codsum);
    } else if (d->kind == PBN_NET_TT) {
        if (n > 65536) { delete net; return fail(PBN_ERR_UNSUPPORTED, "truth-table networks support at most 65536 nodes"); }
        const int nin = d->tt_in_off[n], ntab = d->tt_tab_off[n];
        if (nin > 65535) { delete net; return fail(PBN_ERR_UNSUPPORTED, "too many inputs in total"); }
        v.off_node = 0;
        v.off_in = n * 8;
        v.off_thr = (v.off_in + nin * 2 + 15) & ~15;
        blob.resize((size_t)v.off_thr + (size_t)ntab * 4);
        uint2 *node = reinterpret_cast<uint2 *>(blob.data());
        unsigned short *in = reinterpret_cast<unsigned short *>(blob.data() + v.off_in);
        u32 *thr = reinterpret_cast<u32 *>(blob.data() + v.off_thr);
        for (int i = 0; i < n; i++) {
            const int k = d->tt_in_off[i + 1] - d->tt_in_off[i];
            if (k < 0 || k > 16 || d->tt_tab_off[i + 1] - d->tt_tab_off[i] != (1 << k)) {
                delete net;
                return fail(PBN_ERR_ARG, "truth table size does not match its input count (k <= 16)");
            }
            node[i] = make_uint2((u32)d->tt_tab_off[i], (u32)d->tt_in_off[i] | ((u32)k << 16));
        }
        for (int q = 0; q < nin; q++) {
            if (d->tt_in[q] < 0 || d->tt_in[q] >= n) { delete net; return fail(PBN_ERR_ARG, "input index out of range"); }
            in[q] = (unsigned short)d->tt_in[q];
        }
        for (int q = 0; q < ntab; q++) thr[q] = thr31(d->tt_prob[q]);
        rc |= upload(net->owned, d->tt_prob, (size_t)ntab, &v.tt_prob);
    } else {
        delete net;
        return fail(PBN_ERR_ARG, "unknown network kind");
    }
    blob.resize((blob.size() + 15) & ~(size_t)15);
    v.blob_bytes = v.blob_fast_bytes = (int)blob.size();
    if (v.off_rec16) v.blob_bytes = v.off_rec16;  // everything but the fast paths stages the image without the 16-byte records
    if (d->kind == PBN_NET_TT) {
        // behind the image (not staged by the existing kernels): the constant entries that pbn_ssd_pinned points the node
        // records of pinned nodes at
        net->tt_const = (u32)(blob.size() - v.off_thr) / 4u;
        blob.resize(blob.size() + 16, 0);
        reinterpret_cast<u32 *>(blob.data() + v.blob_bytes)[1] = 0x80000000u;
    }
    rc |= upload(net->owned, blob.data(), blob.size(), &v.blob);
    if (rc) { pbn_net_destroy(net); return PBN_ERR_CUDA; }
    v.thr_dev = nullptr;
    if (d->kind == PBN_NET_TT && v.blob_bytes - v.off_thr > PBN_TT_THR_SMEM_MAX) {
        // Large truth-table networks: the threshold table (4 B per table entry, the last section of the image) stays in
        // global memory and is read through the L1 (one load per update); only node records and input lists are staged.
        // With the 32-word state columns of a 1024-node network the image would otherwise limit an SM to two blocks.
        v.thr_dev = reinterpret_cast<const u32 *>(v.blob + v.off_thr);
        v.blob_bytes = v.blob_fast_bytes = v.off_thr;
    }
    if (v.blob_bytes > 160 * 1024) { pbn_net_destroy(net); return fail(PBN_ERR_UNSUPPORTED, "network image exceeds shared memory"); }
    *out = net;
    return PBN_OK;
}

extern "C" int pbn_net_destroy(PbnNet *net) {
    if (!net) return PBN_OK;
    for (void *p : net->owned) cudaFree(p);
    delete net;
    return PBN_OK;
}
extern "C" int pbn_net_words(const PbnNet *net) { return net ? net->v.w32 : 0; }

extern "C" int pbn_env_create(const PbnNet *net, const PbnEnvDesc *d, PbnEnv **out) {
    if (!net || !d || !out) return fail(PBN_ERR_ARG, "null argument");
    if (d->kind < PBN_ENV_PBN || d->kind > PBN_ENV_PBCN_ST) return fail(PBN_ERR_ARG, "unknown env kind");
    const bool self_trig = d->kind == PBN_ENV_PBN_ST || d->kind == PBN_ENV_PBCN_ST;
    if (self_trig && (!d->gamma_pow || d->n_gamma < 1 || d->max_interval < 0))
        return fail(PBN_ERR_ARG, "self-triggering envs need the gamma**i table and T >= 0");
    const int n = net->v.n, w32 = net->v.w32;
    // control="write" stores the control vector into nodes 0..M-1 of the env's own state column: M > N would write past it
    if (d->n_control < 0 || d->n_control > n) return fail(PBN_ERR_ARG, "n_control must be in 0..n_nodes");
    PbnEnv *env = new PbnEnv();
    env->net = net;
    EnvView &v = env->v;
    memset(&v, 0, sizeof v);
    v.kind = d->kind; v.horizon = d->horizon; v.max_inner = d->max_inner > 0 ? d->max_inner : 1;
    v.force = d->force; v.dedup = d->dedup; v.control_write = d->control_write; v.n_control = d->n_control;
    v.successful_reward = d->successful_reward; v.wrong_attractor_cost = d->wrong_attractor_cost;
    v.n_att = d->n_att; v.tgt_first = d->tgt_first; v.n_tgt = d->n_tgt;
    env->has_small_att = false;  // PBNEnv.reset redraws until it holds an attractor of at most 10 states (pbn_env.py:196-199)
    for (int a = 0; a < d->n_att; a++) env->has_small_att |= d->att_off[a + 1] - d->att_off[a] <= 10;
    const int n_att_cubes = d->n_att > 0 ? d->att_off[d->n_att] : 0;
    v.n_cubes = n_att_cubes > d->tgt_first + d->n_tgt ? n_att_cubes : d->tgt_first + d->n_tgt;
    if (d->n_tgt == 0) v.n_cubes = n_att_cubes;
    v.off_cubes = ((d->n_att + 1) * 4 + 15) & ~15;
    std::vector<unsigned char> img((size_t)v.off_cubes + (size_t)v.n_cubes * w32 * 8 + 16, 0);
    int *off = reinterpret_cast<int *>(img.data());
    for (int a = 0; a <= d->n_att; a++) off[a] = d->n_att > 0 ? d->att_off[a] : 0;
    u32 *cw = reinterpret_cast<u32 *>(img.data() + v.off_cubes);
    for (int c = 0; c < v.n_cubes; c++)
        for (int i = 0; i < n; i++) {
            int8_t x = d->cube[(size_t)c * n + i];
            if (x == 0 || x == 1) {
                cw[((size_t)c * w32 + (i >> 5)) * 2] |= 1u << (i & 31);
                if (x) cw[((size_t)c * w32 + (i >> 5)) * 2 + 1] |= 1u << (i & 31);
            } else if (x != 2) {
                delete env;
                return fail(PBN_ERR_ARG, "cube entries must be 0, 1 or 2 ('*')");
            }
        }
    img.resize((img.size() + 15) & ~(size_t)15);
    v.img_bytes = (int)img.size();
    if (v.img_bytes + net->v.blob_bytes > 190 * 1024) { delete env; return fail(PBN_ERR_UNSUPPORTED, "cube tables exceed shared memory"); }
    if (upload(env->owned, img.data(), img.size(), &v.img)) { pbn_env_destroy(env); return PBN_ERR_CUDA; }
    if (self_trig) {
        v.n_gamma = d->n_gamma; v.max_interval = d->max_interval;
        if (upload(env->owned, d->gamma_pow, (size_t)d->n_gamma, &v.gamma_pow)) { pbn_env_destroy(env); return PBN_ERR_CUDA; }
    }
    *out = env;
    return PBN_OK;
}
extern "C" int pbn_env_destroy(PbnEnv *env) {
    if (!env) return PBN_OK;
    for (void *p : env->owned) cudaFree(p);
    delete env;
    return PBN_OK;
}

// ----------------------------------------------------------------------------------------------- kernel helpers
extern __shared__ __align__(16) unsigned char smem_raw[];

__device__ __forceinline__ void stage(unsigned char *dst, const unsigned char *src, int bytes) {
    const uint4 *s = reinterpret_cast<const uint4 *>(src);
    uint4 *d = reinterpret_cast<uint4 *>(dst);
    for (int i = threadIdx.x; i < (bytes >> 4); i += blockDim.x) d[i] = s[i];
}
__device__ __forceinline__ void load_state(const Col &c, const u32 *g, long long B, long long e, int w32) {
    for (int w = 0; w < w32; w++) c.set_word(w, g[(long long)w * B + e]);
}
__device__ __forceinline__ void store_state(const Col &c, u32 *g, long long B, long long e, int w32) {
    for (int w = 0; w < w32; w++) g[(long long)w * B + e] = c.word(w);
}

// the launch's epoch when it lives (partly) in device memory: epoch + *epoch_ptr
__device__ __forceinline__ void resolve_epoch(DrawView &dv) {
    if (dv.epoch_ptr) dv.epoch += *dv.epoch_ptr;
}

// An intervention on node `pos`; an index outside the network (a policy network can emit anything) is ignored and counted —
// it must not flip a bit of a neighbouring env's column or of the staged network image.  Returns 1 iff the flip was applied:
// an ignored intervention costs nothing either (the env.step equals one with action 0).
__device__ __forceinline__ int flip_node(const Col &st, int pos, int n, int &bad) {
    if (pos >= 0 && pos < n) { st.flip((u32)pos); return 1; }
    bad++;
    return 0;
}

// ---- shared-memory accesses by 32-bit shared-window address (the hot SSD loop keeps its base addresses in registers;
// through generic pointers ptxas re-derives them from the CTA id in every iteration)
__device__ __forceinline__ u32 smem_addr(const void *p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ u32 lds_u32(u32 a) { u32 v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void sts_u32(u32 a, u32 v) { asm volatile("st.shared.u32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void red_xor_u32(u32 a, u32 v) { asm volatile("red.shared.xor.b32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void red_add_u32(u32 a, u32 v) { asm volatile("red.shared.add.u32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ uint4 ldc_v4(u32 a) {  // read-only image data: free to schedule
    uint4 v; asm("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a)); return v;
}
__device__ __forceinline__ u32 ldc_u32(u32 a) { u32 v; asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint2 ldc_v2(u32 a) { uint2 v; asm("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a)); return v; }
__device__ __forceinline__ u32 keep(u32 x) { asm volatile("" : "+r"(x)); return x; }  // pins a loop invariant in a register

// State columns of networks up to 256 nodes start on a power-of-two boundary >= w32 KB of the shared window, so that
// "column address + word offset" is an OR and folds into the LOP3 that masks the offset (fast paths below).
__host__ __device__ inline unsigned col_align_bytes(int w32) {
    if (w32 > 8) return 0u;
    unsigned a = 1024u;
    while (a < (unsigned)w32 * 1024u) a <<= 1;
    return a;
}
__device__ __forceinline__ u32 *align_cols(u32 *p, int w32) {
    const u32 al = col_align_bytes(w32);
    if (!al) return p;
    const u32 a = smem_addr(p);
    return reinterpret_cast<u32 *>(reinterpret_cast<char *>(p) + ((al - (a & (al - 1u))) & (al - 1u)));
}

// Loop invariants of the predictor-network SSD loop, as registers.
struct SsdFast {
    u32 col;        // shared address of this thread's state column (word w at col + w*1024)
    u32 warp_cols;  // shared address of lane 0's column of this warp
    u32 thr, rec;   // shared addresses of the threshold rows / 16-byte predictor records
    u32 thr_stride, rec_stride;  // bytes per node
    u32 shist;      // shared address of the block histogram
    u32 n, W;
    u32 b_off, b_sh, b_up;  // bucket field: word offset, right shift, left shift (32 - g)
    float inv, gdelta;  // gdelta: 0.5 - margin of the gap shortcut
};

// 16 * #{k : t[k] <= r} for an ascending quad of thresholds (cumulative COD rows are ascending, so the predicates are
// monotone and a select chain replaces the sum): 4 compares + 4 selects
__device__ __forceinline__ u32 count_le_x16(const uint4 t, u32 r) {
    u32 j8;
    asm("{ .reg .pred p0, p1, p2, p3;\n\t"
        "setp.le.u32 p0, %1, %5; setp.le.u32 p1, %2, %5; setp.le.u32 p2, %3, %5; setp.le.u32 p3, %4, %5;\n\t"
        "selp.u32 %0, 16, 0, p0; selp.u32 %0, 32, %0, p1; selp.u32 %0, 48, %0, p2; selp.u32 %0, 64, %0, p3; }"
        : "=r"(j8) : "r"(t.x), "r"(t.y), "r"(t.z), "r"(t.w), "r"(r));
    return j8;
}

// one asynchronous update of a predictor network from two words of the update stream (bittner/base.py:89-119,306-312), in two
// halves: the DRAW half (node, predictor pick, the predictor's record) depends only on the stream and can be issued ahead of
// whatever still changes the state; the STATE half gathers the four input bits, looks the LUT bit up and writes it
struct FastDraw {
    u32 i, rx, ry, rz;
};
template <int TQ>
__device__ __forceinline__ FastDraw ssd_fast_draw(const SsdFast &f, u32 wa, u32 wb) {
    const u32 i = __umulhi(wa, f.n);  // Graph.step picks i in [0, N)
    const u32 r = wb >> 1;
    u32 j16;  // 16 * (index of the selected predictor)
    if constexpr (TQ == 1) {
        j16 = count_le_x16(ldc_v4(f.thr + i * f.thr_stride), r);
    } else {  // leading quad = last threshold of each quad (at most four quads when TQ is known)
        const uint4 m = ldc_v4(f.thr + i * f.thr_stride);
        u32 q = (m.x <= r) + (m.y <= r) + (m.z <= r) + (m.w <= r);
        q = q < (u32)TQ - 1u ? q : (u32)TQ - 1u;
        j16 = 64u * q + count_le_x16(ldc_v4(f.thr + i * f.thr_stride + 16u + q * 16u), r);
    }
    const uint4 rec = ldc_v4(f.rec + i * f.rec_stride + j16);
    return FastDraw{i, rec.x, rec.y, rec.z};
}
__device__ __forceinline__ void ssd_fast_apply_update(const SsdFast &f, const FastDraw &d) {
    const u32 f1 = d.rx >> 16, f3 = d.ry >> 16;
    // columns are aligned (align_cols): column address | word offset; a rotate brings input j's bit to position 3 - j
    const u32 w0 = lds_u32(f.col | (d.rx & 0x1C00u));
    const u32 w1 = lds_u32(f.col | (f1 & 0x1C00u));
    const u32 w2 = lds_u32(f.col | (d.ry & 0x1C00u));
    const u32 w3 = lds_u32(f.col | (f3 & 0x1C00u));
    u32 idx = (__funnelshift_r(w0, w0, d.rx) & 8u) | (__funnelshift_r(w1, w1, f1) & ~8u);
    idx = (idx & 0xCu) | (__funnelshift_r(w2, w2, d.ry) & ~0xCu);
    idx = (idx & 0xEu) | (__funnelshift_r(w3, w3, f3) & ~0xEu);  // bits 3..0: LUT index; above: garbage (shifts wrap, LUT doubled)
    const u32 v = __funnelshift_r(d.rz, 0u, idx);
    const u32 wa_addr = f.col | ((d.i & ~31u) << 5);
    const u32 m = __funnelshift_l(0u, 1u, d.i);  // 1 << (i & 31)
    const u32 old = lds_u32(wa_addr);
    sts_u32(wa_addr, (old & ~m) | (__funnelshift_l(0u, v, d.i) & m));  // bit i <- LUT bit idx
}
template <int TQ>
__device__ __forceinline__ void ssd_fast_update(const SsdFast &f, u32 wa, u32 wb) {
    ssd_fast_apply_update(f, ssd_fast_draw<TQ>(f, wa, wb));
}

#include "pbn_coop.cuh"
#include "pbn_smem.cuh"

// the state half of an update, predicated (`on`) and reporting the old and the new word — for callers that track the state
// incrementally (the lockstep first pass of the step-until-attractor envs keeps per-cube mismatch counts)
__device__ __forceinline__ void fast_apply_io(const SsdFast &f, const FastDraw &d, bool on, u32 &old, u32 &nw) {
    const u32 f1 = d.rx >> 16, f3 = d.ry >> 16;
    const u32 w0 = lds_u32(f.col | (d.rx & 0x1C00u));
    const u32 w1 = lds_u32(f.col | (f1 & 0x1C00u));
    const u32 w2 = lds_u32(f.col | (d.ry & 0x1C00u));
    const u32 w3 = lds_u32(f.col | (f3 & 0x1C00u));
    u32 idx = (__funnelshift_r(w0, w0, d.rx) & 8u) | (__funnelshift_r(w1, w1, f1) & ~8u);
    idx = (idx & 0xCu) | (__funnelshift_r(w2, w2, d.ry) & ~0xCu);
    idx = (idx & 0xEu) | (__funnelshift_r(w3, w3, f3) & ~0xEu);
    const u32 v = __funnelshift_r(d.rz, 0u, idx);
    const u32 wa_addr = f.col | ((d.i & ~31u) << 5);
    const u32 m = __funnelshift_l(0u, 1u, d.i);
    old = lds_u32(wa_addr);
    nw = on ? (old & ~m) | (__funnelshift_l(0u, v, d.i) & m) : old;
    sts_u32(wa_addr, nw);
}

static DrawView make_draws(const PbnDraws *d) {
    DrawView v;
    v.mode = d->mode; v.epoch = d->epoch;
    v.seed_lo = (u32)d->seed; v.seed_hi = (u32)(d->seed >> 32);
    v.ints = d->ints; v.dbls = d->dbls;
    v.int_stride = d->int_stride; v.dbl_stride = d->dbl_stride;
    for (int r = 0; r < 10; r++) {
        v.rk[2 * r] = v.seed_lo + (u32)r * 0x9E3779B9u;
        v.rk[2 * r + 1] = v.seed_hi + (u32)r * 0xBB67AE85u;
    }
    v.used = (long long *)d->used;
    v.epoch_ptr = d->epoch_dev;
    return v;
}

// ----------------------------------------------------------------------------------------------- K1 rollout
template <int NET, int MODE, int TQ>
__global__ void __launch_bounds__(PBN_BLOCK) k_rollout(NetView nv, DrawView dv, u32 *state, long long B, long long env0,
                                                       long long steps, int sync) {
    unsigned char *blob = smem_raw;
    const RolloutSmem L = rollout_smem(nv, sync);
    u32 *sst = align_cols(reinterpret_cast<u32 *>(smem_raw + L.cols), nv.w32);
    stage(blob, nv.blob, L.image);
    const long long e = (long long)blockIdx.x * PBN_BLOCK + threadIdx.x;
    Col st{sst + threadIdx.x};
    Col tmp{sst + nv.w32 * PBN_BLOCK + threadIdx.x};
    if (e < B) load_state(st, state, B, e, nv.w32);
    __syncthreads();
    if (e >= B) return;
    Draw<MODE> d;
    d.init(dv, e, env0 + e);
    if (sync) {
        long long t = 0;
        if constexpr (MODE == PBN_DRAW_PHILOX) {
            if ((nv.n & 3) == 0) {
                u32 ublk = 0;
                for (; t < steps; t++) sync_step_x4<NET, TQ>(nv, dv, blob, st, tmp, d, ublk);
                d.blk = ublk;
                d.have = 0;
            }
        }
        for (; t < steps; t++) sync_step<NET, MODE, TQ>(nv, blob, st, tmp, d);
    } else {
        long long t = 0;
        if constexpr (MODE == PBN_DRAW_PHILOX) {
            // an update takes exactly two words of the env's stream: one Philox block per two updates, no buffer bookkeeping
            u32 ublk = 0;
            if constexpr (NET == PBN_NET_PRED && TQ > 0) {
              if (nv.off_rec16) {
                SsdFast f;
                f.col = keep(smem_addr(st.s));
                f.thr = keep(smem_addr(blob + nv.off_thr));
                f.rec = keep(smem_addr(blob + nv.off_rec16));
                f.thr_stride = keep((u32)nv.tsq_stride * 16u);
                f.rec_stride = keep((u32)nv.fmax * 16u);
                f.n = keep((u32)nv.n);
                for (; t + 1 < steps; t += 2) {
                    u32 x0, x1, x2, x3;
                    philox4x32_10_rk(ublk++, d.c1, d.c2, d.c3, dv, x0, x1, x2, x3);
                    ssd_fast_update<TQ>(f, x0, x1);
                    ssd_fast_update<TQ>(f, x2, x3);
                }
              }
            }
            {
                for (; t + 1 < steps; t += 2) {
                    u32 x0, x1, x2, x3;
                    philox4x32_10_rk(ublk++, d.c1, d.c2, d.c3, dv, x0, x1, x2, x3);
                    micro_step_words<NET, TQ>(nv, blob, st, x0, x1, d);
                    micro_step_words<NET, TQ>(nv, blob, st, x2, x3, d);
                }
            }
            d.blk = ublk;
            d.have = 0;
        }
        for (; t < steps; t++) micro_step<NET, MODE, TQ>(nv, blob, st, d);
    }
    store_state(st, state, B, e, nv.w32);
    d.done(dv, e);
}

// ----------------------------------------------------------------------------------------------- reset
// One env's reset, on global memory (used by k_env_reset and by the fused vector step).
//   TARGET: pbn_target.py:328-352 — sample(all_attractors, 2), a cube of each, '*' -> randint(0,1) position by position
//   MULTI : pbn_target_multi.py:227-259 — first attractor -> last attractor (Q14)
//   PBN family: pbn_env.py:190-213 — an attractor with <= 10 states, a uniform state of it, state[0] = 0 (common/pbn.py:77)
// Curriculum of PBNTargetMultiEnv (pbn_target_multi.py:159-181, 232-235), one probability row per env — a vector env is B
// independent env objects of the reference, each with its own table.
struct CurView {
    double *prob;    // [B][n_att] or null
    int *pair;       // [B][2] sampled (state attractor id, target attractor id)
    int sample_pair; // 1: the sampled ids choose the attractors; 0: first -> last as the reference does (Q14), ids only recorded
};
// np.random.choice(range(A), size=2, replace=False, p=prob) from three uniforms (numpy legacy RandomState.choice: searchsorted
// on the normalised cumulative sum, first occurrences kept, the found id's mass zeroed before the redraw)
__device__ __forceinline__ void sample_pair_dev(const double *prob, int A, const double *u, int &a, int &b) {
    double p[64], cdf[64];
    auto draw = [&](double x) {
        int k = 0;
        while (k < A && cdf[k] <= x) k++;
        return k < A ? k : A - 1;
    };
    auto build = [&]() {
        double acc = 0.0;
        for (int k = 0; k < A; k++) { acc += p[k]; cdf[k] = acc; }
        for (int k = 0; k < A; k++) cdf[k] /= acc;
    };
    for (int k = 0; k < A; k++) p[k] = prob[k];
    build();
    a = draw(u[0]);
    b = draw(u[1]);
    if (a == b) {
        p[a] = 0.0;
        build();
        b = draw(u[2]);
    }
}
// rework_probas(episode_len) on one row
__device__ __forceinline__ void rework_probas_dev(double *prob, int A, int s, int t, int len) {
    const double eps = 1.0 * 1.0 / A, lo = 0.01 * 1.0 / A, hi = 0.5;
    if (len < 20) {
        prob[s] -= eps; prob[t] -= eps;
        prob[s] = prob[s] > lo ? prob[s] : lo;
        prob[t] = prob[t] > lo ? prob[t] : lo;
    }
    if (len >= 99) {
        prob[s] += eps; prob[t] += eps;
        prob[s] = prob[s] < hi ? prob[s] : hi;
        prob[t] = prob[t] < hi ? prob[t] : hi;
    }
    for (int k = 0; k < A; k++) prob[k] = lo > prob[k] ? lo : prob[k];
    // `s = sum(self.probabilities)`: CPython >= 3.12 sums floats with Neumaier compensation (bltinmodule.c: cs_add)
    double sum = 0.0, comp = 0.0;
    for (int k = 0; k < A; k++) {
        const double x = prob[k], t = sum + x;
        comp += fabs(sum) >= fabs(x) ? (sum - t) + x : (x - t) + sum;
        sum = t;
    }
    if (comp != 0.0 && isfinite(comp)) sum += comp;
    for (int k = 0; k < A; k++) prob[k] /= sum;
}

template <int MODE>
__device__ __forceinline__ void reset_env(const NetView &nv, const EnvView &ev, const DrawView &dv, u32 *state, int *n_steps,
                                          int *target_att, u32 *target_state, long long B, long long e, long long env0,
                                          const CurView cv = CurView{nullptr, nullptr, 0}) {
    const int *att_off = reinterpret_cast<const int *>(ev.img);
    const u32 *cubes = reinterpret_cast<const u32 *>(ev.img + ev.off_cubes);
    const int n = nv.n, w32 = nv.w32;
    Draw<MODE> d;
    d.init(dv, e, env0 + e);
    if (ev.kind == PBN_ENV_TARGET || ev.kind == PBN_ENV_MULTI) {
        const int A = ev.n_att;
        int a, b;
        if (ev.kind == PBN_ENV_TARGET) {  // random.sample(all_attractors, 2), pbn_target.py:333
            if constexpr (MODE == PBN_DRAW_REPLAY) { a = d.randint(0, A); b = d.randint(0, A); }
            else { a = d.randint(0, A); b = d.randint(0, A - 1); if (b >= a) b++; }
        } else {
            a = 0; b = A - 1;  // first -> last (pbn_target_multi.py:237-238)
            if constexpr (MODE == PBN_DRAW_PHILOX) {
                if (cv.prob && A >= 2 && A <= 64) {  // the pair drawn from this env's table (:232-235), three words, always
                    double u[3];
                    for (int k = 0; k < 3; k++) u[k] = ((double)d.next() + 0.5) * (1.0 / 4294967296.0);
                    int sa, sb;
                    sample_pair_dev(cv.prob + e * A, A, u, sa, sb);
                    cv.pair[2 * e] = sa; cv.pair[2 * e + 1] = sb;
                    if (cv.sample_pair) { a = sa; b = sb; }
                }
            }
        }
        const int cs = att_off[a] + d.randint(0, att_off[a + 1] - att_off[a]);
        const int ct = att_off[b] + d.randint(0, att_off[b + 1] - att_off[b]);
        const u32 *ps = cubes + (size_t)cs * w32 * 2, *pt = cubes + (size_t)ct * w32 * 2;
        // '*' -> randint(0,1), state then target, position by position (:336-340).  Replay: one recorded draw per '*'.
        // Philox: the wildcards take the BITS of the stream's words in that same order, most significant first (32 per word
        // instead of one word each: a 199-node reset with 120-wildcard cubes is 8 words, not 240), and only positions that
        // have a wildcard are visited.
        u32 bitbuf = 0;
        int nbits = 0;
        auto wild = [&]() -> u32 {
            if constexpr (MODE == PBN_DRAW_PHILOX) {
                if (nbits == 0) { bitbuf = d.next(); nbits = 32; }
                nbits--;
                const u32 v = bitbuf >> 31;
                bitbuf <<= 1;
                return v;
            } else {
                return (u32)d.randint(0, 2);
            }
        };
        for (int w = 0; w < w32; w++) {
            const u32 valid = (w == w32 - 1 && (n & 31)) ? ((1u << (n & 31)) - 1u) : 0xFFFFFFFFu;
            const u32 sc = ps[2 * w], tc = pt[2 * w];
            u32 sw = ps[2 * w + 1] & sc, tw = pt[2 * w + 1] & tc;
            for (u32 m = (~sc | ~tc) & valid; m != 0u; m &= m - 1u) {
                const u32 bit = m & (0u - m);
                if (!(sc & bit)) sw |= wild() ? bit : 0u;
                if (!(tc & bit)) tw |= wild() ? bit : 0u;
            }
            state[(long long)w * B + e] = sw;
            if (target_state) target_state[(long long)w * B + e] = tw;
        }
        target_att[e] = b;
        n_steps[e] = 0;
    } else {
        int a;
        do { a = d.randint(0, ev.n_att); } while (att_off[a + 1] - att_off[a] > 10);
        const int c = att_off[a] + d.randint(0, att_off[a + 1] - att_off[a]);
        const u32 *p = cubes + (size_t)c * w32 * 2;
        for (int w = 0; w < w32; w++) state[(long long)w * B + e] = (w == 0) ? (p[1] & ~1u) : p[2 * w + 1];
        if (n_steps) n_steps[e] = 0;
    }
    d.done(dv, e);
}

template <int MODE>
__global__ void __launch_bounds__(PBN_BLOCK) k_env_reset(NetView nv, EnvView ev, DrawView dv, u32 *state, int *n_steps,
                                                         int *target_att, u32 *target_state, const unsigned char *mask,
                                                         long long B, long long env0, CurView cv) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B || (mask && !mask[e])) return;
    resolve_epoch(dv);
    reset_env<MODE>(nv, ev, dv, state, n_steps, target_att, target_state, B, e, env0, cv);
}

// Vector-env epilogue of one finished env.step (fused into the step kernels): episode bookkeeping, block-aggregated
// statistics, and — when the episode ended and autoreset is on — the reset, drawn from its own epoch so that the
// fused launch is bit-identical to "step launch, then masked reset launch".
struct VecView {
    int enabled, autoreset;
    long long *ep_return;
    int *ep_len;
    unsigned long long *stats;  // [8] episodes, return sum, length sum, successes, cap hits, env steps, ignored interventions, -
    u32 *final_obs, *target_state;
    DrawView rdv;
    CurView cur;
    double *ep_return_f64, *return_sum_f64;  // self-triggering envs: float64 discounted returns (per env; sum over finished episodes)
};
template <int MODE>
__device__ __forceinline__ void vec_finish(const NetView &nv, const EnvView &ev, const VecView &vx, unsigned long long *s_stats,
                                           u32 *state, int *n_steps, int *target_att, u32 *obs_state, long long B,
                                           long long e, long long env0, int rew, int tm, int tr, int in, double rew_f64 = 0.0) {
    const bool f64 = vx.ep_return_f64 != nullptr;  // self-triggering envs keep float64 returns (self_triggering.py:76,178)
    const long long ret = f64 ? 0 : vx.ep_return[e] + rew;
    const double ret_d = f64 ? vx.ep_return_f64[e] + rew_f64 : 0.0;
    const int len = vx.ep_len[e] + 1;
    atomicAdd(&s_stats[5], 1ULL);
    if (tm) atomicAdd(&s_stats[3], 1ULL);
    if ((ev.kind == PBN_ENV_TARGET || ev.kind == PBN_ENV_MULTI) && in >= ev.max_inner) atomicAdd(&s_stats[4], 1ULL);
    if (vx.final_obs)
        for (int w = 0; w < nv.w32; w++) vx.final_obs[(long long)w * B + e] = obs_state[(long long)w * B + e];
    if (tm | tr) {
        atomicAdd(&s_stats[0], 1ULL);
        if (f64) { atomicAdd(vx.return_sum_f64, ret_d); vx.ep_return_f64[e] = 0.0; }
        else {
            atomicAdd(&s_stats[1], (unsigned long long)ret);  // two's complement: sums of negative returns wrap correctly
            vx.ep_return[e] = 0;
        }
        atomicAdd(&s_stats[2], (unsigned long long)len);
        vx.ep_len[e] = 0;
        if (vx.cur.prob && ev.kind == PBN_ENV_MULTI && ev.n_att >= 2)  // env.rework_probas(episode_len), then the reset draws from it
            rework_probas_dev(vx.cur.prob + e * ev.n_att, ev.n_att, vx.cur.pair[2 * e], vx.cur.pair[2 * e + 1], len);
        if (vx.autoreset) {
            reset_env<MODE>(nv, ev, vx.rdv, state, n_steps, target_att, vx.target_state, B, e, env0, vx.cur);
            for (int w = 0; w < nv.w32; w++) obs_state[(long long)w * B + e] = state[(long long)w * B + e];  // reset envs observe their new state
        }
    } else {
        if (f64) vx.ep_return_f64[e] = ret_d;
        else vx.ep_return[e] = ret;
        vx.ep_len[e] = len;
    }
}
__device__ __forceinline__ void vec_flush_stats(const VecView &vx, unsigned long long *s_stats) {
    __syncthreads();
    if (vx.enabled && threadIdx.x < 8 && s_stats[threadIdx.x]) atomicAdd(&vx.stats[threadIdx.x], s_stats[threadIdx.x]);
}

// ----------------------------------------------------------------------------------------------- K1 sync, bit-sliced
// 32x32 bit-matrix transpose across a warp: afterwards lane i's bit j is what lane j's bit i was.
__device__ __forceinline__ u32 warp_transpose32(u32 x, u32 lane) {
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const u32 m = s == 16 ? 0x0000FFFFu : s == 8 ? 0x00FF00FFu : s == 4 ? 0x0F0F0F0Fu : s == 2 ? 0x33333333u : 0x55555555u;
        const u32 y = __shfl_xor_sync(0xFFFFFFFFu, x, s);
        x = (lane & s) ? (((y & ~m) >> s) | (x & ~m)) : ((x & m) | ((y & m) << s));
    }
    return x;
}

// Graph.synch_step (base.py:300-303) for 32 envs at a time: a WARP owns a group of 32 consecutive envs, the state is
// held TRANSPOSED in shared memory (one 32-bit word per node, bit b = env b of the group), lane l computes the nodes
// i = l, l+32, ...  The predictor choice of the 32 envs is one bit-serial comparison of 32 uniforms with the node's
// thresholds (a fresh random word per bit level, levels stop when every env is decided: ~10 words instead of 32 draws),
// every predictor is evaluated on all 32 envs with a 15-instruction mux tree over precomputed LUT masks.
// Semantics restated in oracle/pbn_oracle.c: orc_rollout_sync_sliced.
__global__ void __launch_bounds__(PBN_BLOCK) k_sync_sliced(NetView nv, DrawView dv, u32 *state, long long B, long long env0, int steps) {
    const int n = nv.n, fmax = nv.fmax, w32 = nv.w32;
    const int npad = w32 * 32;
    unsigned char *blob = smem_raw;
    const SlicedSmem L = sliced_smem(nv);
    u32 *lm = reinterpret_cast<u32 *>(smem_raw + L.lm);
    const int lrow = fmax * 16 + 4;
    u32 *words = reinterpret_cast<u32 *>(smem_raw + L.words);  // [8 warps][2][npad]
    stage(blob, nv.blob, L.image);
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(nv.lutmask);
        uint4 *dst = reinterpret_cast<uint4 *>(lm);
        for (int i = threadIdx.x; i < n * lrow / 4; i += PBN_BLOCK) dst[i] = src[i];
    }
    const u32 lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const long long e0 = ((long long)blockIdx.x * (PBN_BLOCK / 32) + warp) * 32;  // first env of this warp's group
    u32 *cur = words + warp * 2 * npad, *nxt = cur + npad;
    const bool live = e0 < B;
    if (live) {
        const long long e = e0 + lane;
        for (int w = 0; w < w32; w++) {
            const u32 x = e < B ? state[(long long)w * B + e] : 0u;
            cur[w * 32 + lane] = warp_transpose32(x, lane);
        }
    }
    __syncthreads();
    if (!live) return;
    const u32 G = (u32)((unsigned long long)(env0 + e0) >> 5);
    const uint4 *thr = reinterpret_cast<const uint4 *>(blob + nv.off_thr);
    const uint2 *rec = reinterpret_cast<const uint2 *>(blob + nv.off_rec);
    for (int t = 0; t < steps; t++) {
        for (int base = 0; base < n; base += 32) {
            const int i = base + (int)lane;
            const bool valid = i < n;
            const int ii = valid ? i : 0;
            const uint4 T = thr[ii * nv.tsq_stride];
            u32 T0 = T.x, T1 = T.y, T2 = T.z, T3 = T.w;
            // a threshold of 2^31 (p = 1, and the padding of absent predictors) is "always below": decided at once
            u32 lt0 = T0 >> 31 ? ~0u : 0u, lt1 = T1 >> 31 ? ~0u : 0u, lt2 = T2 >> 31 ? ~0u : 0u, lt3 = T3 >> 31 ? ~0u : 0u;
            u32 u0 = ~lt0, u1 = ~lt1, u2 = ~lt2, u3 = ~lt3;
            if (!valid) u0 = u1 = u2 = u3 = 0;
            T0 <<= 1; T1 <<= 1; T2 <<= 1; T3 <<= 1;  // bit 30 -> sign position
            u32 b0 = 0, b1 = 0, b2 = 0, b3 = 0;
            for (int l = 0; l < 31; l++) {
                if (!__any_sync(0xFFFFFFFFu, (u0 | u1 | u2 | u3) != 0u)) break;
                if ((l & 3) == 0) philox4x32_10((u32)(l >> 2), dv.epoch, G, ((u32)t << 12) | (u32)ii, dv.seed_lo, dv.seed_hi, b0, b1, b2, b3);
                const u32 R = b0;
                b0 = b1; b1 = b2; b2 = b3;
                const u32 s0 = (u32)((int)T0 >> 31), s1 = (u32)((int)T1 >> 31), s2 = (u32)((int)T2 >> 31), s3 = (u32)((int)T3 >> 31);
                lt0 |= u0 & ~R & s0; u0 &= ~(R ^ s0);
                lt1 |= u1 & ~R & s1; u1 &= ~(R ^ s1);
                lt2 |= u2 & ~R & s2; u2 &= ~(R ^ s2);
                lt3 |= u3 & ~R & s3; u3 &= ~(R ^ s3);
                T0 <<= 1; T1 <<= 1; T2 <<= 1; T3 <<= 1;
            }
            if (valid) {
                // predictor j is chosen where r >= T_{j-1} and r < T_j (absent thresholds are "always below")
                const u32 c0 = lt0, c1 = lt1 & ~lt0, c2 = lt2 & ~lt1, c3 = lt3 & ~lt2, c4 = ~lt3;
                u32 out = 0;
                for (int j = 0; j < fmax; j++) {
                    const u32 chosen = j == 0 ? c0 : j == 1 ? c1 : j == 2 ? c2 : j == 3 ? c3 : c4;
                    const uint2 r = rec[i * fmax + j];
                    const u32 x0 = cur[r.x & 0xFF], x1 = cur[(r.x >> 8) & 0xFF], x2 = cur[(r.x >> 16) & 0xFF], x3 = cur[r.x >> 24];
                    const uint4 *M = reinterpret_cast<const uint4 *>(lm + (size_t)i * lrow + j * 16);
                    const uint4 m0 = M[0], m1 = M[1], m2 = M[2], m3 = M[3];
                    // 16 -> 8 on x3 (index bit 0), 8 -> 4 on x2, 4 -> 2 on x1, 2 -> 1 on x0
                    const u32 a0 = (x3 & m0.y) | (~x3 & m0.x), a1 = (x3 & m0.w) | (~x3 & m0.z);
                    const u32 a2 = (x3 & m1.y) | (~x3 & m1.x), a3 = (x3 & m1.w) | (~x3 & m1.z);
                    const u32 a4 = (x3 & m2.y) | (~x3 & m2.x), a5 = (x3 & m2.w) | (~x3 & m2.z);
                    const u32 a6 = (x3 & m3.y) | (~x3 & m3.x), a7 = (x3 & m3.w) | (~x3 & m3.z);
                    const u32 d0 = (x2 & a1) | (~x2 & a0), d1 = (x2 & a3) | (~x2 & a2);
                    const u32 d2 = (x2 & a5) | (~x2 & a4), d3 = (x2 & a7) | (~x2 & a6);
                    const u32 g0 = (x1 & d1) | (~x1 & d0), g1 = (x1 & d3) | (~x1 & d2);
                    out |= chosen & ((x0 & g1) | (~x0 & g0));
                }
                nxt[i] = out;
            }
        }
        __syncwarp();
        u32 *tmp = cur; cur = nxt; nxt = tmp;
    }
    {
        const long long e = e0 + lane;
        for (int w = 0; w < w32; w++) {
            u32 x = cur[w * 32 + lane];
            if (w * 32 + (int)lane >= n) x = 0;
            x = warp_transpose32(x, lane);
            if (e < B) state[(long long)w * B + e] = x;
        }
    }
}

// ----------------------------------------------------------------------------------------------- K2 env step
__device__ __forceinline__ bool is_attracting(const EnvView &ev, const int *att_off, const u32 *cubes, const Col &st, int w32) {
    if (ev.n_att == 0) return true;
    return match_range(cubes, 0, att_off[ev.n_att], st, w32);
}
__device__ __forceinline__ int pbcn_reward(const EnvView &ev, const int *att_off, const u32 *cubes, const Col &st, int w32,
                                           int &term) {
    if (match_range(cubes, ev.tgt_first, ev.tgt_first + ev.n_tgt, st, w32)) { term = 1; return ev.successful_reward; }
    int m = 0;
    for (int a = 0; a < ev.n_att; a++) m += match_range(cubes, att_off[a], att_off[a + 1], st, w32) ? 1 : 0;
    term = 0;
    return -ev.wrong_attractor_cost * m;
}

// The same tests through 32-bit shared-window addresses held in registers.  Through generic pointers ptxas re-derives the
// window base (S2R SR_CgaCtaId, LEA) inside the cube loops — 46 instructions per attractor where 12 do — and k_env_step runs
// these loops after EVERY update of a sampled-data / self-triggering macro step.
struct CubeView {
    u32 cubes, att_off, col;  // shared addresses: cube table, attractor offsets, this thread's state column
    int w32;
};
__device__ __forceinline__ bool cube_match_sa(const CubeView &cv, int c) {
    const u32 pa = cv.cubes + (u32)c * (u32)cv.w32 * 8u;
    for (int w = 0; w < cv.w32; w++) {  // early exit per word: a many-care cube fails in its first words
        const uint2 cw = ldc_v2(pa + 8u * (u32)w);
        if ((lds_u32(cv.col + 1024u * (u32)w) & cw.x) != cw.y) return false;
    }
    return true;
}
__device__ __forceinline__ bool match_range_sa(const CubeView &cv, int c0, int c1) {
    for (int c = c0; c < c1; c++)
        if (cube_match_sa(cv, c)) return true;
    return false;
}
__device__ __forceinline__ int pbcn_reward_sa(const EnvView &ev, const CubeView &cv, int &term) {
    if (match_range_sa(cv, ev.tgt_first, ev.tgt_first + ev.n_tgt)) { term = 1; return ev.successful_reward; }
    int m = 0;
    int c0 = (int)lds_u32(cv.att_off);
    for (int a = 0; a < ev.n_att; a++) {
        const int c1 = (int)lds_u32(cv.att_off + 4u * (u32)(a + 1));
        m += match_range_sa(cv, c0, c1) ? 1 : 0;
        c0 = c1;
    }
    term = 0;
    return -ev.wrong_attractor_cost * m;
}

// One asynchronous update of a truth-table network (Node.compute_next_value common/node.py:31-38, PBN.step common/pbn.py:88-92,
// PBCN.step common/pbcn.py:59-61) through shared-window addresses held in registers; same words, same result as micro_step.
struct TtView {
    u32 node, in, thr, col;  // shared addresses: node records, input lists, threshold table (unused with thr_dev), state column
    const u32 *thr_dev;
    u32 first, span;         // the updated node is first + mulhi(word, span)
};
__device__ __forceinline__ void tt_micro_step_words_sa(const TtView &tv, u32 wa, u32 wb);
__device__ __forceinline__ void tt_micro_step_sa(const TtView &tv, Draw<PBN_DRAW_PHILOX> &d) {
    const u32 wa = d.next(), wb = d.next();
    tt_micro_step_words_sa(tv, wa, wb);
}
// the same update from two given words of the env's update stream (wa picks the node, wb decides)
__device__ __forceinline__ void tt_micro_step_words_sa(const TtView &tv, u32 wa, u32 wb) {
    const u32 i = tv.first + __umulhi(wa, tv.span);
    const uint2 nr = ldc_v2(tv.node + 8u * i);  // (table offset, input offset | k << 16)
    const u32 k = nr.y >> 16;
    u32 ia = tv.in + 2u * (nr.y & 0xFFFFu);
    u32 idx = 0;
    for (u32 q = 0; q < k; q++, ia += 2u) {
        u32 pos;
        asm("ld.shared.u16 %0, [%1];" : "=r"(pos) : "r"(ia));
        const u32 w = lds_u32(tv.col + ((pos & ~31u) << 5));
        idx = (idx << 1) | ((w >> (pos & 31u)) & 1u);
    }
    const u32 thr = tv.thr_dev ? __ldg(tv.thr_dev + nr.x + idx) : lds_u32(tv.thr + 4u * (nr.x + idx));
    const u32 v = ((wb >> 1) < thr) ? 1u : 0u;
    const u32 wd = tv.col + ((i & ~31u) << 5);
    const u32 m = 1u << (i & 31u);
    const u32 old = lds_u32(wd);
    sts_u32(wd, v ? (old | m) : (old & ~m));
}

// control="write" (the PBCN envs of sampled_data.py and self_triggering.py): the control vector goes into nodes 0..M-1 before
// every update.  For M <= 32 that is one masked store into the first state word, of bits gathered once per env.step, instead
// of M single-bit writes fed by M global loads per update.  `ctl` = the env.step's actions from index 1 on (pbcn: the env
// has a control vector there).
struct CtlWrite {
    const int *ctl;
    u32 bits, mask;
    __device__ __forceinline__ CtlWrite(const EnvView &ev, const int *c, bool pbcn)
        : ctl(c), bits(0u), mask(ev.n_control >= 32 ? 0xFFFFFFFFu : ((1u << ev.n_control) - 1u)) {
        if (pbcn && ev.control_write && ev.n_control <= 32)
            for (int k = 0; k < ev.n_control; k++) bits |= (ctl[k] != 0 ? 1u : 0u) << k;
    }
    __device__ __forceinline__ void apply(const EnvView &ev, const Col &st) const {
        if (!ev.control_write) return;
        if (ev.n_control <= 32) st.set_word(0, (st.word(0) & ~mask) | bits);
        else
            for (int k = 0; k < ev.n_control; k++) st.put(k, ctl[k] != 0);
    }
};

template <int NET, int MODE>
__global__ void __launch_bounds__(PBN_BLOCK, 4) k_env_step(NetView nv, EnvView ev, DrawView dv, u32 *state, int *n_steps,
                                                        const int *target_att, const int *actions, int K, u32 *obs_state,
                                                        int *reward, unsigned char *terminated, unsigned char *truncated,
                                                        int *inner_steps, long long B, long long env0, VecView vx, double *rew_f64) {
    resolve_epoch(dv);
    resolve_epoch(vx.rdv);
    unsigned char *blob = smem_raw;
    const EnvSmem L = env_smem(nv, ev, 1, false, false);
    unsigned char *img = smem_raw + L.img;
    u32 *sst = reinterpret_cast<u32 *>(smem_raw + L.cols);
    __shared__ unsigned long long s_stats[8];
    stage(blob, nv.blob, L.image);
    stage(img, ev.img, ev.img_bytes);
    if (threadIdx.x < 8) s_stats[threadIdx.x] = 0;
    const int *att_off = reinterpret_cast<const int *>(img);
    const u32 *cubes = reinterpret_cast<const u32 *>(img + ev.off_cubes);
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int w32 = nv.w32;
    Col st{sst + threadIdx.x};
    if (e < B) load_state(st, state, B, e, w32);
    __syncthreads();
    if (e < B) {
    const CubeView cv{keep(smem_addr(cubes)), keep(smem_addr(att_off)), keep(smem_addr(st.s)), w32};
    const TtView tv{keep(smem_addr(blob + nv.off_node)), keep(smem_addr(blob + nv.off_in)), keep(smem_addr(blob + nv.off_thr)), cv.col,
                    nv.thr_dev, (u32)nv.first, (u32)(nv.n - nv.first)};
    Draw<MODE> d;
    d.init(dv, e, env0 + e);
    auto update = [&]() {
        if constexpr (NET == PBN_NET_TT && MODE == PBN_DRAW_PHILOX) tt_micro_step_sa(tv, d);
        else micro_step<NET, MODE>(nv, blob, st, d);
    };
    const int *act = actions + e * K;
    int rew = 0, tm = 0, tr = 0, in = 0, bad = 0;
    double rew_d = 0.0;
    switch (ev.kind) {
    case PBN_ENV_PBN: {  // pbn_env.py:141-154, reward :171-183
        int a = act[0];
        const int cost = a != 0 ? flip_node(st, a, nv.n, bad) : 0;  // flips index `action` itself (Q3)
        update(); in = 1;
        if (match_range_sa(cv, ev.tgt_first, ev.tgt_first + ev.n_tgt)) { rew = 20; tm = 1; }
        else rew = -4 - cost;
    } break;
    case PBN_ENV_PBCN: {  // pbcn_env.py:67-80
        int a = act[0];
        if (a != 0) flip_node(st, a, nv.n, bad);
        update(); in = 1;
        rew = pbcn_reward_sa(ev, cv, tm);
    } break;
    case PBN_ENV_PBN_SD: {  // sampled_data.py:52-88
        int a = act[0], interval = act[1];
        for (int i = 0; i < interval; i++) {
            const int cost = a != 0 ? flip_node(st, a - 1, nv.n, bad) : 0;
            update(); in++;
            if (match_range_sa(cv, ev.tgt_first, ev.tgt_first + ev.n_tgt)) { rew += 20; tm = 1; }
            else { rew += -4 - cost; tm = 0; }
        }
    } break;
    case PBN_ENV_PBCN_SD: {  // sampled_data.py:139-189
        int interval = act[0], tstep = -1;
        const CtlWrite cw(ev, act + 1, true);
        auto one = [&](int i, auto &&step) {
            cw.apply(ev, st);
            step(); in++;
            int r = pbcn_reward_sa(ev, cv, tm) - 1;  // time_step_cost = 1
            if (tstep >= 0) r -= ev.successful_reward;                // overshoot penalty
            else if (tm) tstep = i;
            rew += r;
        };
        if constexpr (NET == PBN_NET_TT && MODE == PBN_DRAW_PHILOX) {
            // an update takes exactly two words of the env's stream: one Philox block per two updates, no buffer bookkeeping
            u32 blk = d.blk;  // (0: the stream starts with this step)
            int i = 0;
            for (; i + 1 < interval; i += 2) {
                u32 x0, x1, x2, x3;
                philox4x32_10_rk(blk++, d.c1, d.c2, d.c3, dv, x0, x1, x2, x3);
                one(i, [&]() { tt_micro_step_words_sa(tv, x0, x1); });
                one(i + 1, [&]() { tt_micro_step_words_sa(tv, x2, x3); });
            }
            d.blk = blk;
            d.have = 0;
            if (i < interval) one(i, [&]() { tt_micro_step_sa(tv, d); });  // odd tail: the stream object takes over
        } else {
            for (int i = 0; i < interval; i++) one(i, update);
        }
    } break;
    case PBN_ENV_PBN_ST:     // self_triggering.py:56-93: (action, prob 1..10)
    case PBN_ENV_PBCN_ST: {  // self_triggering.py:146-197: (prob 1..10, control bits...)
        const bool pbcn = ev.kind == PBN_ENV_PBCN_ST;
        const int a = pbcn ? 0 : act[0];
        int pv = act[pbcn ? 0 : 1];                            // MultiDiscrete value 1..10 (self_triggering.py:29,120)
        if (pv < 1 || pv > 10) { bad++; pv = pv < 1 ? 1 : 10; }  // a stop probability of 0 would never end the macro step
        const double prob = (double)pv / 10.0;                 // convert value in [1,10] to [0.1 .. 1]
        const u32 stop_thr = (u32)ceil(prob * 2147483648.0);   // Philox: stop iff r31 < ceil(prob * 2^31)
        const CtlWrite cw(ev, act + 1, pbcn);
        double total = 0.0;
        int i = 0;
        bool end = false;
        while (!end) {
            int r;
            if (!pbcn) {
                const int cost = a != 0 ? flip_node(st, a - 1, nv.n, bad) : 0;
                update();
                if (match_range_sa(cv, ev.tgt_first, ev.tgt_first + ev.n_tgt)) { r = 20; tm = 1; }
                else { r = -4 - cost; tm = 0; }
            } else {
                cw.apply(ev, st);
                update();
                r = pbcn_reward_sa(ev, cv, tm) - 1;  // time step cost
            }
            total += ev.gamma_pow[i < ev.n_gamma ? i : ev.n_gamma - 1] * (double)r;  // total_reward += gamma**i * reward
            i++;
            bool stop;
            if constexpr (MODE == PBN_DRAW_PHILOX) stop = (d.next() >> 1) < stop_thr;
            else stop = d.dbl() <= prob;  // random.uniform(0, 1) <= prob
            end = stop || i == ev.max_interval;
        }
        in = i;
        rew = (int)total;
        rew_d = total;
        if (rew_f64) rew_f64[e] = total;
    } break;
    default: break;
    }
    store_state(st, state, B, e, w32);
    if (obs_state) store_state(st, obs_state, B, e, w32);
    reward[e] = rew;
    terminated[e] = (unsigned char)tm;
    truncated[e] = (unsigned char)tr;
    if (inner_steps) inner_steps[e] = in;
    if (bad && vx.enabled) atomicAdd(&s_stats[6], 1ULL);  // env.steps whose intervention was out of range (ignored)
    d.done(dv, e);
    if (vx.enabled) vec_finish<MODE>(nv, ev, vx, s_stats, state, n_steps, nullptr, obs_state, B, e, env0, rew, tm, tr, in, rew_d);
    }
    vec_flush_stats(vx, s_stats);
}

// K2 for the two step-until-attractor envs (PBNTargetEnv, PBNTargetMultiEnv).  The inner loop is unbounded in the
// reference and heavy-tailed in practice (1 .. 40 000 updates per env.step, SURVEY.md §0.9): with one env per thread a
// warp, and then its whole block, lives as long as its slowest env.  So the kernel is PERSISTENT: each block owns a
// contiguous range of envs and its threads pull the next env from a block-local counter the moment they finish one, in a
// flat loop whose every trip is "one attractor test + at most one update" for every lane — lanes never wait at the end
// of an inner loop.  An env's result does not depend on which thread ran it (its Philox stream is keyed by its id).
// Straggler mode of the step-until-attractor kernel (predictor networks, Philox draws): when a block's queue is empty and
// only a few lanes of a warp still hold an env, the warp stops running them as lone lanes (a lone lane's update is a
// ~1 500-cycle dependent chain) and splits into 1, 2, 4 or 8 groups of 32/k lanes, each finishing one env with the draw
// half of the updates spread over its lanes and the state half pipelined (pbn_coop.cuh: coop_steps).  The env's words are
// the ones the ordinary loop would have used (update k takes words 2k, 2k+1), so results are identical.
#ifndef PBN_COOP_MAX
#define PBN_COOP_MAX 8   // live envs per warp at which straggler mode takes over (groups of 32 / 8 = 4 lanes)
#endif
#ifndef PBN_COOP_EXIT_AT
#define PBN_COOP_EXIT_AT 2  // group mode, queue not empty: stopped groups at which a call returns to finalize / refill
#endif
#ifndef PBN_COOP_WIDE_FACTOR
#define PBN_COOP_WIDE_FACTOR 1  // a resume list longer than this many times 8 envs per warp runs 16 envs per warp
#endif

// is_attracting without early exits (the lockstep first pass: a warp's lanes test together, a branch per cube only diverges)
__device__ __forceinline__ bool is_attracting_flat(const EnvView &ev, const int *att_off, const u32 *cubes, const Col &st, int w32) {
    if (ev.n_att == 0) return true;
    const int n_cubes = att_off[ev.n_att];
    bool hit = false;
    if (w32 == 1) {
        const u32 sw = st.word(0);
        const uint2 *cv = reinterpret_cast<const uint2 *>(cubes);
#pragma unroll 4
        for (int c = 0; c < n_cubes; c++) hit |= (sw & cv[c].x) == cv[c].y;
        return hit;
    }
    for (int c = 0; c < n_cubes; c++) {
        const uint2 *cv = reinterpret_cast<const uint2 *>(cubes) + (size_t)c * w32;
        bool ok = true;
        for (int w = 0; w < w32; w++) ok &= (st.word(w) & cv[w].x) == cv[w].y;
        hit |= ok;
    }
    return hit;
}

// ---- pieces of one env.step of the step-until-attractor envs, shared by the kernels below
// the intervention: pbn_target.py:261-269 (one node) / pbn_target_multi.py:120-134 (a set of nodes, the observation captured
// BEFORE the first update).  An env.step with an out-of-range node is counted here, once, whichever pass finishes it.
// Returns the pending action cost (MULTI: -len(actions), the ignored slots left out).
__device__ __forceinline__ int att_begin(const NetView &nv, const EnvView &ev, const VecView &vx, unsigned long long *s_stats,
                                         const Col &st, const Col &ob, const int *act, int K) {
    int bad = 0, cnt = 0;
    if (ev.kind != PBN_ENV_MULTI) {
        const int a = act[0];
        if (a != 0) flip_node(st, a - 1, nv.n, bad);
    } else {
        for (int k = 0; k < K; k++) {
            const int a = act[k];
            if (a < 0) continue;
            if (ev.dedup) {
                bool dup = false;
                for (int j = 0; j < k; j++) dup |= (act[j] == a);
                if (dup) continue;
            }
            cnt += a != 0 ? flip_node(st, a - 1, nv.n, bad) : 1;  // an ignored slot is not an action: it costs nothing
        }
        for (int w = 0; w < nv.w32; w++) ob.set_word(w, st.word(w));  // observation captured BEFORE the update (:133)
    }
    if (bad && vx.enabled) atomicAdd(&s_stats[6], 1ULL);  // env.steps whose intervention was out of range (ignored)
    return -cnt;  // reward -= len(actions)
}
// reward and flags of a finished env.step; `ob` = the observation the loop ended on (MULTI), st = the state
__device__ __forceinline__ void att_result(const EnvView &ev, const int *att_off, const u32 *cubes, const Col &st, const Col &ob,
                                           int w32, int ta, int pend, int &rew, int &tm) {
    tm = 0;
    if (ev.kind != PBN_ENV_MULTI) {  // PBNTargetEnv._get_reward, pbn_target.py:303-326: any cube of the target attractor
        if (match_range(cubes, att_off[ta], att_off[ta + 1], st, w32)) { rew = 20; tm = 1; } else rew = -5;
    } else {  // in_target returns at the first mismatch of the FIRST cube (Q12), pbn_target_multi.py:190-225
        rew = pend;
        if (att_off[ta] < att_off[ta + 1] && cube_match(cubes, att_off[ta], ob, w32)) { rew += 1000; tm = 1; }
    }
}

// Budgeted / resumable execution (include/pbn_b200.h: PbnStepPlan).  Lists are {count, queue head, -, -, env ids...}.
struct PlanView {
    int budget, resume;
    unsigned char *running;
    int *list_in, *list_out;
};

// out of budget: park the env for a resume pass, which goes on from its state, update count and pending cost
__device__ __forceinline__ void att_park(const PlanView &pl, const Col &st, u32 *state, int *inner_steps, int *reward, long long B,
                                         long long e, int w32, int in, int pend) {
    store_state(st, state, B, e, w32);
    inner_steps[e] = in;
    reward[e] = pend;
    pl.running[e] = 1;
    pl.list_out[4 + atomicAdd(&pl.list_out[0], 1)] = (int)e;
}
// a finished env.step: results, flags and the vector-env epilogue.  `fo` = the column the observation is (MULTI: the state
// observed last), used_a / used_b = the draws record (Draw::tell); pl.running is null without a plan.
template <int MODE>
__device__ __forceinline__ void att_finish(const NetView &nv, const EnvView &ev, const DrawView &dv, const PlanView &pl, const VecView &vx,
                                           unsigned long long *s_stats, const int *att_off, const u32 *cubes, const Col &st,
                                           const Col &fo, u32 *state, int *n_steps, int *target_att, u32 *obs_state, int *reward,
                                           unsigned char *terminated, unsigned char *truncated, int *inner_steps, long long B,
                                           long long e, long long env0, int in, int pend, u32 used_a, u32 used_b) {
    const int w32 = nv.w32;
    int rew, tm;
    att_result(ev, att_off, cubes, st, fo, w32, target_att[e], pend, rew, tm);
    store_state(st, state, B, e, w32);
    if (obs_state) store_state(fo, obs_state, B, e, w32);
    reward[e] = rew;
    terminated[e] = (unsigned char)tm;
    const int tr = (n_steps[e] == ev.horizon);
    truncated[e] = (unsigned char)tr;
    if (inner_steps) inner_steps[e] = in;
    if (pl.running) pl.running[e] = 0;
    if (dv.used) { dv.used[2 * e] = used_a; dv.used[2 * e + 1] = used_b; }
    if (vx.enabled) vec_finish<MODE>(nv, ev, vx, s_stats, state, n_steps, target_att, obs_state, B, e, env0, rew, tm, tr, in);
}

// W1: one-word networks (N <= 32) — the group runner keeps the state in a register; a separate instantiation, because both
// runners inlined in one kernel made it 120 KB of SASS and instruction fetch its top stall (ncu: no_inst 21 %)
template <int NET, int MODE, int TQ, bool W1>
__global__ void __launch_bounds__(PBN_BLOCK, 2) k_env_step_att(NetView nv, EnvView ev, DrawView dv, u32 *state, int *n_steps,
                                                            const int *target_att, const int *actions, int K, u32 *obs_state,
                                                            int *reward, unsigned char *terminated, unsigned char *truncated,
                                                            int *inner_steps, long long B, long long env0, long long per_block,
                                                            int coop_on, int grp_mode, PlanView pl, VecView vx) {
    resolve_epoch(dv);
    resolve_epoch(vx.rdv);
    unsigned char *blob = smem_raw;
    const EnvSmem L = env_smem(nv, ev, 2, false, coop_on);
    unsigned char *img = smem_raw + L.img;
    u32 *sst = reinterpret_cast<u32 *>(smem_raw + L.cols);
    const int w32 = nv.w32;
    unsigned char *coop_buf = reinterpret_cast<unsigned char *>(sst + L.coop);  // straggler-mode staging, per warp
    __shared__ int s_next;
    __shared__ unsigned long long s_stats[8];
    stage(blob, nv.blob, L.image);
    stage(img, ev.img, ev.img_bytes);
    if (threadIdx.x < 8) s_stats[threadIdx.x] = 0;
    const int *att_off = reinterpret_cast<const int *>(img);
    const u32 *cubes = reinterpret_cast<const u32 *>(img + ev.off_cubes);
    // work queue: a fresh step hands every block a contiguous range of envs, taken through a block-local counter; a resume
    // pass takes the parked envs of the previous launch from one global queue, so the few long-running envs spread over the
    // whole GPU whatever block first ran them
    const bool resume = pl.resume != 0;
    const long long lo = resume ? 0 : (long long)blockIdx.x * per_block;
    const long long hi = resume ? (long long)pl.list_in[0] : (lo + per_block < B ? lo + per_block : B);
    // GROUP mode (predictor networks, Philox draws, real attractors): only every fourth lane owns an env — 64 per block at a
    // time — and every env is run from its second update on by a group of 4 .. 32 lanes (pbn_coop.cuh), 8 envs per warp side
    // by side: an update costs ~100 cycles there against ~2 500 for a lane running alone in the loop below, which then only
    // starts and finishes env.steps.  Otherwise every lane owns an env and groups only take over a warp's last few.
    const bool grp = MODE == PBN_DRAW_PHILOX && NET == PBN_NET_PRED && grp_mode != 0;
    const int slots = grp ? PBN_BLOCK / 4 : PBN_BLOCK;
    if (threadIdx.x == 0) s_next = slots;  // the first envs of the range are taken statically
    __syncthreads();
    const bool multi = ev.kind == PBN_ENV_MULTI;
    const int coop_min_in = multi ? 2 : 1;  // MULTI tests the pre-update observation first; from its second test on, the state
    Col st{sst + threadIdx.x}, ob{sst + w32 * PBN_BLOCK + threadIdx.x};
    Draw<MODE> d;
    bool have = false;
    // a resume pass sizes its groups to the list: narrow groups carry more envs per instruction (an entry costs the warp the
    // same ~16 ALU-pipe slots whether it serves 8 envs or one), wide ones finish an env sooner (130 against 50 cycles per
    // update), and an SM whose 16 warps all run groups is bound by its ALU pipes, not by latency.  So a list that fits is
    // dealt out STATICALLY (a racing queue hands the first blocks to arrive everything and leaves other SMs idle): over 4 of a
    // block's 8 warps — one per scheduler — when that gives at most 8 envs per warp, else over all 8; what a longer list
    // has left goes through the queue.
    int quota = 8;
    long long static_n = 0, per_slot = 0;  // list positions dealt out statically (resume passes), in rounds of per_slot
    bool warp_on = true;
    // owners sit on every fourth lane (8 envs per warp, groups of >= 4 lanes) — or, in a resume pass whose list would keep every
    // warp queueing, on every second lane: 16 envs per warp in groups of two lanes.  An entry costs the warp the same
    // instructions whatever the group width, so narrow groups double the envs served per instruction; their update takes
    // longer (the draw half of a batch is amortised over 8 entries instead of 16), which only pays while the pass is bound by
    // throughput, and every lane then tests up to two cubes itself, so only for envs with at most four cubes.
    int osh = 2;
    if (resume) {
        const long long nb = gridDim.x;
        const int A = hi <= nb * 4 * 8 ? 4 : 8;
        if (grp && A == 8 && hi > nb * 8 * 8 * PBN_COOP_WIDE_FACTOR && ev.n_att > 0 && att_off[ev.n_att] <= 4) osh = 1;
        const int qmax = 32 >> osh;
        const long long q = (hi + nb * A - 1) / (nb * A);
        quota = q < 1 ? 1 : (q > qmax ? qmax : (int)q);
        per_slot = nb * A;
        static_n = quota * per_slot;
        warp_on = (int)(threadIdx.x >> 5) < A;
    }
    const bool owner_lane = !grp || ((threadIdx.x & ((1u << osh) - 1u)) == 0 && (int)((threadIdx.x & 31) >> osh) < quota);
    long long e = 0, nxt = hi;
    if (owner_lane) {
        if (!resume) nxt = lo + (grp ? threadIdx.x >> 2 : threadIdx.x);
        else if (!grp) nxt = (long long)atomicAdd(&pl.list_in[1], 1);  // (lane mode: every lane pulls)
        else if (warp_on)  // consecutive positions go to different blocks, i.e. SMs, first
            nxt = (long long)((threadIdx.x & 31) >> osh) * per_slot + (long long)(threadIdx.x >> 5) * gridDim.x + blockIdx.x;
    }
    if (resume && !grp) static_n = 0;
    int used = 0;  // updates made for the current env in this launch (budget)
    int in = 0, pend = 0;
    for (;;) {
        if (!have && nxt < hi && resume) {  // a parked env goes on from its saved state, update count and pending cost
            e = pl.list_in[4 + nxt];
            load_state(st, state, B, e, w32);
            in = inner_steps[e];
            pend = reward[e];
            d.seek(dv, e, env0 + e, 2u * (u32)in, 0u);
            if (multi)
                for (int w = 0; w < w32; w++) ob.set_word(w, st.word(w));
            used = 0;
            have = true;
        } else if (!have && nxt < hi) {
            e = nxt;
            load_state(st, state, B, e, w32);
            d.init(dv, e, env0 + e);
            n_steps[e] += 1;
            pend = att_begin(nv, ev, vx, s_stats, st, ob, actions + e * K, K);
            micro_step<NET, MODE, TQ>(nv, blob, st, d);
            in = 1;
            used = 1;
            have = true;
        }
        // warp-uniform exit.  The full-mask vote is also where the lanes of the warp RE-CONVERGE every trip: without it,
        // lanes that once took the finalize branch keep running as separate sub-warps (ncu: 2.9 active threads per
        // instruction), because a loop with per-lane exits only reconverges at its end.
        if (!__any_sync(0xFFFFFFFFu, have)) break;
        if (have) {
            // while not force and not is_attracting_state(state): graph.step()                  (pbn_target.py:270-271)
            // while not is_attracting_state(observation): observation = graph.step()            (pbn_target_multi.py:135-146)
            const bool done = (!multi && ev.force) || in >= ev.max_inner || is_attracting(ev, att_off, cubes, multi ? ob : st, w32);
            if (!done && pl.budget > 0 && used >= pl.budget) {
                att_park(pl, st, state, inner_steps, reward, B, e, w32, in, pend);
                have = false;
                nxt = resume ? static_n + (long long)atomicAdd(&pl.list_in[1], 1) : lo + atomicAdd(&s_next, 1);
            } else if (!done) {
                micro_step<NET, MODE, TQ>(nv, blob, st, d);
                if (multi)
                    for (int w = 0; w < w32; w++) ob.set_word(w, st.word(w));
                in++;
                used++;
            } else {
                u32 ua, ub;
                d.tell(ua, ub);
                att_finish<MODE>(nv, ev, dv, pl, vx, s_stats, att_off, cubes, st, multi ? ob : st, state, n_steps,
                                 const_cast<int *>(target_att), obs_state, reward, terminated, truncated, inner_steps, B, e, env0,
                                 in, pend, ua, ub);
                have = false;
                nxt = resume ? static_n + (long long)atomicAdd(&pl.list_in[1], 1) : lo + atomicAdd(&s_next, 1);
            }
        }
        if constexpr (MODE == PBN_DRAW_PHILOX && NET == PBN_NET_PRED) {
            // straggler mode: few lanes left, nothing more to pull (pbn_coop.cuh)
            const unsigned hv = (ev.n_att > 0 && !ev.force) ? __ballot_sync(0xFFFFFFFFu, have && in >= coop_min_in) : 0u;
            const unsigned live = __ballot_sync(0xFFFFFFFFu, have);
            const u32 lane = threadIdx.x & 31u;
            // the queue position is read by one lane and broadcast: the branch below runs full-mask collectives
            int qn = 0;
            if (lane == 0u) qn = resume ? *reinterpret_cast<volatile int *>(&pl.list_in[1]) : *reinterpret_cast<volatile int *>(&s_next);
            qn = __shfl_sync(0xFFFFFFFFu, qn, 0);
            const bool drained = (resume ? static_n : lo) + qn >= hi;
            if (coop_on && hv != 0u && (grp || (__popc(live) <= PBN_COOP_MAX && drained))) {
                // the group stops at the cap or when the launch's budget for the env is used up, whichever comes first
                int stop_in = ev.max_inner;
                if (pl.budget > 0 && in - used + pl.budget < stop_in) stop_in = in - used + pl.budget;
                // the call returns when `exit_at` groups have stopped: their owners finalize on the next trip (and, while the
                // block's queue lasts, start the next env), the other envs come back here — in wider groups once the queue
                // is empty, which is why the first stop ends the call then
                const int exit_at = drained ? 1 : (__popc(hv) > 8 ? 2 * PBN_COOP_EXIT_AT : PBN_COOP_EXIT_AT);
                const int v = coop_take_over<TQ, W1>(hv, nv, ev, dv, blob, att_off, cubes, sst, coop_buf, env0 + e, in, 0u, stop_in, exit_at);
                if (v != in) {
                    used += v - in;
                    in = v;
                    d.seek(dv, e, env0 + e, 2u * (u32)v, 0u);
                    if (multi)
                        for (int w = 0; w < w32; w++) ob.set_word(w, st.word(w));
                }
            }
        }
    }
    vec_flush_stats(vx, s_stats);
}


// First pass of a planned env.step (predictor networks, Philox draws): every thread owns one env, all envs start together and
// make at most pl.budget updates, so the whole launch is in lockstep on the update index — the Philox block of the update
// stream (one per two updates) is computed by all lanes at once, nobody pulls work, nothing diverges but the predicate "still
// running".  Most envs reach an attractor within a few updates and are finished here (coalesced result stores after the loop);
// the rest are parked for the resume pass (k_env_step_att, groups of lanes).  Same words, same result as any other split.
// FAST (networks with the 16-byte fast-path records, at most 8 state words, at most two attractor cubes or one state word):
// the update of the asynchronous rollout kernel (ssd_fast_update: one LOP3 per gather address, rotate-merge LUT index) and
// an INCREMENTAL attractor test — a mismatch count per cube that moves by -1, 0 or +1 with the one bit an update writes,
// instead of comparing every state word with every cube after every update.
#ifndef PBN_FIRST_MIN_BLOCKS
#define PBN_FIRST_MIN_BLOCKS 3
#endif
template <int TQ, bool FAST>
__global__ void __launch_bounds__(PBN_BLOCK, PBN_FIRST_MIN_BLOCKS) k_env_step_first(NetView nv, EnvView ev, DrawView dv, u32 *state, int *n_steps,
                                                              int *target_att, const int *actions, int K, u32 *obs_state,
                                                              int *reward, unsigned char *terminated, unsigned char *truncated,
                                                              int *inner_steps, long long B, long long env0, PlanView pl, VecView vx) {
    resolve_epoch(dv);
    resolve_epoch(vx.rdv);
    unsigned char *blob = smem_raw;
    const EnvSmem L = env_smem(nv, ev, 2, FAST, false);
    unsigned char *img = smem_raw + L.img;
    const int w32 = nv.w32;
    u32 *sst = reinterpret_cast<u32 *>(smem_raw + L.cols);
    if (FAST) sst = align_cols(sst, w32);
    __shared__ unsigned long long s_stats[8];
    stage(blob, nv.blob, L.image);
    stage(img, ev.img, ev.img_bytes);
    if (threadIdx.x < 8) s_stats[threadIdx.x] = 0;
    const int *att_off = reinterpret_cast<const int *>(img);
    const u32 *cubes = reinterpret_cast<const u32 *>(img + ev.off_cubes);
    const long long e = (long long)blockIdx.x * PBN_BLOCK + threadIdx.x;
    const bool valid = e < B;
    const bool multi = ev.kind == PBN_ENV_MULTI;
    Col st{sst + threadIdx.x}, ob{sst + w32 * PBN_BLOCK + threadIdx.x};
    int pend = 0;
    if (valid) {
        load_state(st, state, B, e, w32);
        n_steps[e] += 1;
    }
    __syncthreads();  // the images are staged and s_stats is zeroed before att_begin counts into it
    if (valid) pend = att_begin(nv, ev, vx, s_stats, st, ob, actions + e * K, K);
    Draw<PBN_DRAW_PHILOX> dummy;
    const u32 c2 = (u32)(env0 + e), c3 = (u32)((u64)(env0 + e) >> 32);
    u32 x0 = 0, x1 = 0, x2 = 0, x3 = 0;
    int in = 0;
    bool run = valid;
    // FAST: loop invariants of the update, and the mismatch counts of this env's state against (up to) two cubes
    SsdFast f;
    const int n_cubes = ev.n_att > 0 ? att_off[ev.n_att] : 0;
    const bool inc = FAST && w32 > 1 && n_cubes >= 1 && n_cubes <= 2;  // one-word states are tested directly: two instructions per cube
    int mm0 = 1, mm1 = 1;
    bool hit_s0 = false;  // MULTI: the observation captured before the first update, which is what its first test looks at
    if constexpr (FAST) {
        f.col = keep(smem_addr(st.s));
        f.thr = keep(smem_addr(blob + nv.off_thr));
        f.rec = keep(smem_addr(blob + nv.off_rec16));
        f.thr_stride = keep((u32)nv.tsq_stride * 16u);
        f.rec_stride = keep((u32)nv.fmax * 16u);
        f.n = keep((u32)nv.n);
        if (inc && valid) {
            mm0 = mm1 = 0;
            for (int w = 0; w < w32; w++) {
                const u32 sw = st.word(w);
                mm0 += __popc((sw ^ cubes[2 * w + 1]) & cubes[2 * w]);
                if (n_cubes > 1) mm1 += __popc((sw ^ cubes[2 * (w32 + w) + 1]) & cubes[2 * (w32 + w)]);
            }
            if (n_cubes < 2) mm1 = 1;
            hit_s0 = mm0 == 0 || mm1 == 0;
        }
    }
    // One round = the attractor test of every running env, then one update.  The DRAW half of an update (node, predictor pick,
    // record, and the cube words the incremental test needs) depends only on the stream: both rounds of a Philox block are drawn
    // at once, ahead of the state halves, so that their dependent shared-memory loads are over when the state half starts.
    auto test = [&](int t) {
        if (t > 0 && run) {
            // while not is_attracting_state(...): graph.step()  (pbn_target.py:270-271, pbn_target_multi.py:135-146; MULTI's
            // first test looks at the observation captured before the first update)
            bool hit;
            if (inc) hit = (multi && in == 1) ? hit_s0 : (mm0 == 0 || mm1 == 0);
            else hit = is_attracting_flat(ev, att_off, cubes, (multi && in == 1) ? ob : st, w32);
            const bool done = (!multi && ev.force) || in >= ev.max_inner || hit || ev.n_att == 0;
            run = !done;
        }
        return t == pl.budget || !__any_sync(0xFFFFFFFFu, run);
    };
    auto round = [&](u32 wa, u32 wb, const FastDraw &dr) {
        if constexpr (FAST) {
            u32 old, nw;
            fast_apply_io(f, dr, run, old, nw);
            if (inc) {
                const u32 i = dr.i;
                const u32 flip = old ^ nw;  // the written bit, if it changed
                const uint2 c0 = reinterpret_cast<const uint2 *>(cubes)[i >> 5];
                mm0 += (flip & c0.x) ? (((nw ^ c0.y) & flip) ? 1 : -1) : 0;
                if (n_cubes > 1) {
                    const uint2 c1 = reinterpret_cast<const uint2 *>(cubes)[w32 + (i >> 5)];
                    mm1 += (flip & c1.x) ? (((nw ^ c1.y) & flip) ? 1 : -1) : 0;
                }
            }
            in += run ? 1 : 0;
        } else if (run) {
            micro_step_words<PBN_NET_PRED, TQ>(nv, blob, st, wa, wb, dummy);
            in++;
        }
    };
    for (int t = 0;; t += 2) {  // t updates made so far by every running env
        if (test(t)) break;
        philox4x32_10_rk((u32)(t >> 1), dv.epoch, c2, c3, dv, x0, x1, x2, x3);
        FastDraw da{}, db{};
        if constexpr (FAST) {
            da = ssd_fast_draw<TQ>(f, x0, x1);
            db = ssd_fast_draw<TQ>(f, x2, x3);
        }
        round(x0, x1, da);
        if (test(t + 1)) break;
        round(x2, x3, db);
    }
    if (valid && run) {
        att_park(pl, st, state, inner_steps, reward, B, e, w32, in, pend);
    } else if (valid) {  // MULTI: the observation is the state from the second update on; an update takes two stream words
        att_finish<PBN_DRAW_PHILOX>(nv, ev, dv, pl, vx, s_stats, att_off, cubes, st, (multi && in == 1) ? ob : st, state, n_steps,
                                    target_att, obs_state, reward, terminated, truncated, inner_steps, B, e, env0, in, pend,
                                    2u * (u32)in, 0u);
    }
    vec_flush_stats(vx, s_stats);
}

template <int MODE>
__global__ void __launch_bounds__(PBN_BLOCK) k_rand_state(NetView nv, DrawView dv, u32 *state, long long B, long long env0) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B) return;
    Draw<MODE> d;
    d.init(dv, e, env0 + e);
    u32 acc = 0;
    for (int i = 0; i < nv.n; i++) {  // Graph.genRandState base.py:368-370
        acc |= (u32)d.randint(0, 2) << (i & 31);
        if ((i & 31) == 31 || i == nv.n - 1) { state[(long long)(i >> 5) * B + e] = acc; acc = 0; }
    }
    d.done(dv, e);
}

// Index of the first attractor with a cube containing each env's state, -1 if none: is_attracting_state (pbn_target.py:562-574)
// as an index.  The cube image is staged into shared memory when it is small (staged = 1), else read from global memory.
__global__ void __launch_bounds__(PBN_BLOCK) k_attractor_index(EnvView ev, int w32, const u32 *state, long long B, int *att_out,
                                                               int staged) {
    const unsigned char *img = staged ? smem_raw : ev.img;
    u32 *sst = reinterpret_cast<u32 *>(smem_raw + index_smem(ev, w32, staged).cols);
    if (staged) stage(smem_raw, ev.img, ev.img_bytes);
    const int *att_off = reinterpret_cast<const int *>(img);
    const u32 *cubes = reinterpret_cast<const u32 *>(img + ev.off_cubes);
    const long long e = (long long)blockIdx.x * PBN_BLOCK + threadIdx.x;
    Col st{sst + threadIdx.x};
    if (e < B) load_state(st, state, B, e, w32);
    __syncthreads();
    if (e >= B) return;
    int idx = -1;
    for (int a = 0; a < ev.n_att && idx < 0; a++)
        if (match_range(cubes, att_off[a], att_off[a + 1], st, w32)) idx = a;
    att_out[e] = idx;
}

// ----------------------------------------------------------------------------------------------- K3 SSD
// bucket = target-node bits, first target = most significant (pbn_target.py:383-391)
__device__ __forceinline__ int ssd_bucket(const SsdParams &sp, const u32 *s_tgt, const Col &st) {
    if (sp.fast_t0 >= 0) {
        u32 field = (*st.wp((u32)sp.fast_t0) >> (sp.fast_t0 & 31)) << (32 - sp.g);
        return (int)__brev(field);
    }
    int b = 0;
    for (int k = 0; k < sp.g; k++) b = (b << 1) | (int)st.bit(s_tgt[k]);
    return b;
}

struct SsdLoopArgs {
    const NetView &nv;
    const EnvView &ev;
    const SsdParams &sp;
    const DrawView &dv;
    const unsigned char *blob;
    const int *att_off;
    const u32 *cubes;
    const u32 *s_tgt;
    u32 *shist;
    unsigned long long *hist;
    u32 *sst;
    int iters;
    u32 nvalid;
    u32 *flipbuf;  // per block: [warps][win][w32][32] words, or nullptr (no windowed path)
    int win;
    long long chain_id;  // global id of this thread's chain (Philox counter words 2, 3)
    unsigned char *coop_buf;  // per block: [warps][coop_warp_bytes(w32)] straggler-mode staging (windowed path only)
};

// inclusive warp prefix sum; shfl.up's predicate output says whether the source lane exists, so each step is two
// instructions (SHFL + predicated add)
__device__ __forceinline__ u32 warp_scan_add(u32 v) {
#pragma unroll
    for (int off = 1; off < 32; off <<= 1)
        asm volatile("{ .reg .pred p; .reg .u32 t; shfl.sync.up.b32 t|p, %0, %1, 0, 0xffffffff; @p add.u32 %0, %0, t; }"
                     : "+r"(v) : "r"(off));
    return v;
}

// The SSD iteration loop of one warp.  FULL = every lane owns a chain (all warps but possibly the last of the job).
// PHILOX perturbation: ONE Bernoulli(p) renewal process per group of 32 consecutive chains over the interleaved index
// c = node*32 + lane (window = 32*n positions per iteration).  Each ROUND every lane draws TWO geometric gaps from
// consecutive words of its own PERTURBATION stream (block indices from 2^31 on); the round's 64 events are ordered
// lane-major (lane l holds events 2l and 2l+1), one warp prefix sum over the lanes' (gap + 1) pairs turns them into 64 event
// positions, and an event inside the current window flips bit (c>>5) of chain (c&31) with a shared-memory atomic.  Same law
// as n independent Bernoulli(p) per chain per iteration (eval.py:92-95), ~1 draw per chain per iteration, no divergence,
// and at p*n = 1 a round (mean span: two windows) is due every second iteration.  A round is drawn only when the previous
// one lies wholly inside the current window, so two event slots per lane are enough.
// The UPDATE stream is then consumed at exactly two words per update, so when every iteration is one update (no
// attractor loop) a Philox block serves two iterations with no buffer bookkeeping (STATIC path below).
struct SsdPerturb {
    u32 e0, e1;   // this lane's pending events, relative to the window start (0xFFFFFFFF = none)
    u32 last_p1;  // (position of the last generated event) + 1, relative to the window start
};

// gap draw of the generic paths: the verified shortcut when the launch carries a margin (hmd = 0.5 - margin > 0)
__device__ __forceinline__ u32 ssd_gap(u32 word, float inv, float hmd) {
    bool ok;
    u32 gap = geom_gap_approx(word, inv, hmd, &ok);
    if (!ok) gap = geom_gap(word, inv);
    return gap;
}

// positions of a round's events from this lane's two gaps
__device__ __forceinline__ void ssd_round(SsdPerturb &ps, u32 g0, u32 g1) {
    const u32 incl = warp_scan_add(g0 + g1 + 2u);
    ps.e1 = ps.last_p1 - 1u + incl;
    ps.e0 = ps.e1 - 1u - g1;
    ps.last_p1 = __shfl_sync(0xFFFFFFFFu, ps.e1, 31) + 1u;
}

// PIN (k_ssd_pinned): an event on a node outside the free mask s_free (word w = nodes 32w..32w+31) is drawn and not applied
template <bool FULL, bool PIN = false>
__device__ __forceinline__ void ssd_perturb(SsdPerturb &ps, Draw<PBN_DRAW_PHILOX> &dp, char *warp_cols, u32 W, float inv, float hmd, u32 nvalid,
                                            const u32 *s_free = nullptr) {
    auto apply = [&](u32 &e) {
        if (e < W) {
            const u32 tl = e & 31u;
            // word (node>>5) of column tl: byte offset = tl*4 + (node>>5)*1024, node = e>>5.  Two statements rather than a
            // masked bit formed ahead: that form reschedules (changes the SASS of) the unpinned k_ssd instantiations
            if constexpr (PIN) {
                if (FULL || tl < nvalid)
                    atomicXor(reinterpret_cast<u32 *>(warp_cols + tl * 4u + ((e >> 10) << 10)), (1u << ((e >> 5) & 31u)) & s_free[e >> 10]);
            } else {
                if (FULL || tl < nvalid) atomicXor(reinterpret_cast<u32 *>(warp_cols + tl * 4u + ((e >> 10) << 10)), 1u << ((e >> 5) & 31u));
            }
            e = 0xFFFFFFFFu;
        }
    };
    for (;;) {
        apply(ps.e0);
        apply(ps.e1);
        if (ps.last_p1 > W) break;  // the last generated event lies beyond this window
        const u32 g0 = ssd_gap(dp.next(), inv, hmd);
        const u32 g1 = ssd_gap(dp.next(), inv, hmd);
        ssd_round(ps, g0, g1);
    }
    if (ps.e0 != 0xFFFFFFFFu) ps.e0 -= W;
    if (ps.e1 != 0xFFFFFFFFu) ps.e1 -= W;
    ps.last_p1 -= W;
    __syncwarp();
}

// The same renewal process, with the events of one iteration recorded in a flip mask [w32][32] (word w of chain tl at
// buf[w*32 + tl]) instead of being applied: the windowed loop below draws the masks of several iterations ahead.
template <bool FULL>
__device__ __forceinline__ void ssd_perturb_buf(SsdPerturb &ps, Draw<PBN_DRAW_PHILOX> &dp, u32 *buf, u32 W, float inv, float hmd, u32 nvalid) {
    auto apply = [&](u32 &e) {
        if (e < W) {
            const u32 tl = e & 31u;
            if (FULL || tl < nvalid) atomicXor(buf + ((e >> 10) << 5) + tl, 1u << ((e >> 5) & 31u));
            e = 0xFFFFFFFFu;
        }
    };
    for (;;) {
        apply(ps.e0);
        apply(ps.e1);
        if (ps.last_p1 > W) break;
        const u32 g0 = ssd_gap(dp.next(), inv, hmd);
        const u32 g1 = ssd_gap(dp.next(), inv, hmd);
        ssd_round(ps, g0, g1);
    }
    if (ps.e0 != 0xFFFFFFFFu) ps.e0 -= W;
    if (ps.e1 != 0xFFFFFFFFu) ps.e1 -= W;
    ps.last_p1 -= W;
}

struct SsdCount {
    int cur;
    u32 run;
};
__device__ __forceinline__ void ssd_count(SsdCount &c, const SsdLoopArgs &a, const Col &st) {
    const int b = ssd_bucket(a.sp, a.s_tgt, st);
    if (b != c.cur) {  // run-length aggregated histogram update (a chain rarely changes bucket)
        if (a.sp.smem_hist) atomicAdd(&a.shist[c.cur], c.run);
        else atomicAdd(&a.hist[c.cur], (unsigned long long)c.run);
        c.cur = b; c.run = 0;
    }
    c.run++;
}

// GOAL (k_passage): the count of an iteration becomes a goal test.  Bit b of the goal mask (staged where the histogram
// would sit, a.shist) says whether bucket b lies in the goal; hit = the first iteration whose bucket does, ~0u while none
// has (iterations ascend, so the first hit is the least)
__device__ __forceinline__ void ssd_goal(u32 &hit, const SsdLoopArgs &a, const Col &st, u32 it) {
    const int b = ssd_bucket(a.sp, a.s_tgt, st);
    hit = min(hit, (a.shist[b >> 5] >> (b & 31)) & 1u ? it : ~0u);
}

// Perturbation state of the static loop.  Each event is resolved once, when its round is drawn: the iteration it is due in,
// the shared address of the word it flips and the bit.  Checking a slot in an iteration is then a compare, a select and one
// shared-memory XOR.  An applied event stays in its slot until the next round overwrites it: its iteration has passed, and
// the iteration counter never meets it again.  The lane's perturbation stream is held as "next block index + the unused
// half of the last block" (a round takes two words, so every second round computes a block).
struct SsdFastPerturb {
    u32 t0, t1;   // iteration each slot's event is due in
    u32 a0, a1;   // shared address of the word it flips
    u32 m0, m1;   // the bit it flips
    u32 next;     // iteration of the last generated event: the next round is drawn in it
    u32 last_p1;  // (position of the last generated event) + 1, relative to the window of iteration `next`
    u32 blk, half, sx, sy;
};

// XOR the slot's bit in if its event is due in iteration `it`, else XOR 0: every lane issues the atomic (a predicated
// atomic becomes a branch with reconvergence code)
__device__ __forceinline__ void ssd_fast_apply(u32 t_due, u32 a, u32 m, u32 it) { red_xor_u32(a, t_due == it ? m : 0u); }

// the slot of an event at position e relative to the window of iteration `it`: window e / W (ssd_window_div), and in it
// bit (c>>5) of chain (c&31), i.e. word (c>>10) of column (c&31) at byte offset (c&31)*4 + (c>>10)*1024.  PIN: the bit is
// masked with word (c>>10) of the free mask at shared address `free` (an event on a pinned node XORs 0)
template <bool PIN = false>
__device__ __forceinline__ void ssd_fast_slot(const SsdFast &f, const SsdParams &sp, u32 e, u32 it, u32 &t_due, u32 &a, u32 &m,
                                              u32 free = 0u) {
    const u32 q = __umulhi(e >> 4, sp.wq_mul) >> sp.wq_sh;
    const u32 c = e - q * f.W;
    t_due = it + q;
    a = f.warp_cols | ((c << 2) & 0x7Cu) | (c & 0xFFFFFC00u);
    m = 1u << ((c >> 5) & 31u);
    if constexpr (PIN) m &= ldc_u32(free + ((c >> 8) & ~3u));
}

__device__ __forceinline__ u32 ssd_fast_gap(const SsdFast &f, u32 word, bool &ok) { return geom_gap_approx(word, f.inv, f.gdelta, &ok); }

// iteration `it` of the perturbation process: apply the events due in it, and draw rounds while the last generated event
// lies inside its window (a round is drawn only when every pending event is due in this iteration, so two slots suffice)
template <bool PIN = false>
__device__ __forceinline__ void ssd_fast_perturb(const SsdFast &f, const SsdParams &sp, SsdFastPerturb &ps, const Draw<PBN_DRAW_PHILOX> &dp,
                                                 const DrawView &dv, u32 it, u32 free = 0u) {
    ssd_fast_apply(ps.t0, ps.a0, ps.m0, it);
    ssd_fast_apply(ps.t1, ps.a1, ps.m1, it);
    if (ps.next == it) {
        // last_p1 comes out of a warp reduction: the compiler knows it is the same in every lane and branches on it without
        // reconvergence code
        u32 last_p1 = ps.last_p1;
        do {
            u32 wa, wb;
            if (ps.half == 0u) {  // a round takes two words: every second one computes a block
                u32 x2, x3;
                philox4x32_10_rk(ps.blk, dp.c1, dp.c2, dp.c3, dv, wa, wb, x2, x3);
                ps.blk++;
                ps.sx = x2; ps.sy = x3;
                ps.half = 1u;
            } else {
                wa = ps.sx; wb = ps.sy;
                ps.half = 0u;
            }
            bool ok0, ok1;
            u32 g0 = ssd_fast_gap(f, wa, ok0), g1 = ssd_fast_gap(f, wb, ok1);
            if (!(ok0 && ok1)) {  // within the margin of an integer (or shortcut off): the defining polynomial
                if (!ok0) g0 = geom_gap(wa, f.inv);
                if (!ok1) g1 = geom_gap(wb, f.inv);
            }
            const u32 incl = warp_scan_add(g0 + g1 + 2u);
            const u32 e1 = last_p1 - 1u + incl;
            const u32 e0 = e1 - 1u - g1;
            last_p1 = __reduce_max_sync(0xFFFFFFFFu, e1) + 1u;  // lane 31's: positions ascend with the lane
            ssd_fast_slot<PIN>(f, sp, e0, it, ps.t0, ps.a0, ps.m0, free);
            ssd_fast_slot<PIN>(f, sp, e1, it, ps.t1, ps.a1, ps.m1, free);
            ssd_fast_apply(ps.t0, ps.a0, ps.m0, it);
            ssd_fast_apply(ps.t1, ps.a1, ps.m1, it);
        } while (last_p1 <= f.W);
        const u32 q = __umulhi((last_p1 - 1u) >> 4, sp.wq_mul) >> sp.wq_sh;  // >= 1: the window of the last event
        ps.next = it + q;
        ps.last_p1 = last_p1 - q * f.W;
    }
    __syncwarp();
}

// STATIC path of predictor networks, full warps, no attractor loop, shared histogram, targets inside one state word:
// the configuration the headline number is measured in.  Returns the number of iterations done (even), or -1 when (GOAL)
// the warp left because every lane's chain has arrived: then nothing is handed back, as no iteration follows.
template <int TQ, bool PIN = false, bool GOAL = false>
__device__ __forceinline__ int ssd_loop_pred_static(const SsdLoopArgs &a, const Col &st, Draw<PBN_DRAW_PHILOX> &d,
                                                    Draw<PBN_DRAW_PHILOX> &dp, SsdPerturb &ps0, SsdCount &cnt, const u32 *s_free = nullptr,
                                                    u32 *hit = nullptr) {
    if (a.iters < 2) return 0;
    const NetView &nv = a.nv;
    SsdFast f;
    f.col = keep(smem_addr(st.s));
    f.warp_cols = keep(smem_addr(a.sst + (threadIdx.x & ~31u)));
    f.thr = keep(smem_addr(a.blob + nv.off_thr));
    f.rec = keep(smem_addr(a.blob + nv.off_rec16));
    f.thr_stride = keep((u32)nv.tsq_stride * 16u);
    f.rec_stride = keep((u32)nv.fmax * 16u);
    f.shist = keep(smem_addr(a.shist));
    f.n = keep((u32)nv.n);
    f.W = keep((u32)nv.n * 32u);
    f.b_off = keep(((u32)a.sp.fast_t0 >> 5) << 10);
    f.b_sh = keep((u32)a.sp.fast_t0 & 31u);
    f.b_up = keep(32u - (u32)a.sp.g);
    f.inv = a.sp.inv;
    f.gdelta = 0.5f - a.sp.gdelta;  // the shortcut compares against 0.5 - margin (negative: never taken)
    u32 free = 0u;
    if constexpr (PIN) free = keep(smem_addr(s_free));
    // entered at the start of the loop: no pending events, the first round due in iteration 0, no buffered words in dp
    // (the empty slots still hold a valid address: every lane XORs through both slots in every iteration)
    SsdFastPerturb ps{~0u, ~0u, f.warp_cols, f.warp_cols, 0u, 0u, 0u, ps0.last_p1, dp.blk, 0u, 0u, 0u};
    u32 ublk = 0;
    int t = 0;
    u32 cur = (u32)cnt.cur, run = cnt.run;
    u32 h = 0u, c2 = d.c2, c3 = d.c3;
    if constexpr (GOAL) {
        h = *hit;
        // the chain-id words of the update stream held in registers: left to ptxas, the goal loop recomputes them from
        // the block and thread index in every trip (10 instructions)
        c2 = keep(c2);
        c3 = keep(c3);
    }
    auto count = [&](u32 it) {
        const u32 b = __brev((lds_u32(f.col + f.b_off) >> f.b_sh) << f.b_up);
        if constexpr (GOAL) {  // the goal word of bucket b, a bit test, the hit iteration selected: no atomics
            const u32 w = lds_u32(f.shist + ((b >> 5) << 2));
            h = min(h, (w >> (b & 31u)) & 1u ? it : ~0u);
        } else {
            u32 r0;  // run-length aggregation, predicated: flush the run when the bucket changes
            asm volatile("{ .reg .pred p; setp.ne.u32 p, %1, %2; @p red.shared.add.u32 [%3], %4; selp.u32 %0, 0, %4, p; }"
                         : "=r"(r0) : "r"(b), "r"(cur), "r"(f.shist + cur * 4u), "r"(run) : "memory");
            cur = b;
            run = r0 + 1u;
        }
    };
    for (int left = a.iters >> 1; left > 0; left--, t += 2) {  // (a count-down: the bound is not re-read from the parameter bank)
        if constexpr (GOAL) {
            if (__all_sync(0xFFFFFFFFu, h != ~0u)) {  // no live lane: leave without handing anything back
                *hit = h;
                return -1;
            }
        }
        u32 x0, x1, x2, x3;
        philox4x32_10_rk(ublk, d.c1, c2, c3, a.dv, x0, x1, x2, x3);
        ublk++;
        // the draw half of an update does not depend on the state: issued ahead of the perturbation, its two dependent
        // shared-memory loads are over when the state half needs them
        const FastDraw da = ssd_fast_draw<TQ>(f, x0, x1);
        count((u32)t);
        ssd_fast_perturb<PIN>(f, a.sp, ps, dp, a.dv, (u32)t, free);
        ssd_fast_apply_update(f, da);
        __syncwarp();
        const FastDraw db = ssd_fast_draw<TQ>(f, x2, x3);
        count((u32)t + 1u);
        ssd_fast_perturb<PIN>(f, a.sp, ps, dp, a.dv, (u32)t + 1u, free);
        ssd_fast_apply_update(f, db);
        __syncwarp();
    }
    d.blk = ublk;
    d.have = 0;
    // hand the perturbation stream and the pending events back to the generic loop (an odd last iteration), as positions
    // relative to the window of iteration t; the loop drew a round in iteration 0, so both slots hold events
    dp.blk = ps.blk;
    dp.have = ps.half ? 2 : 0;
    dp.b0 = ps.sx; dp.b1 = ps.sy;
    const u32 tu = (u32)t;
    auto position = [&](u32 t_due, u32 addr, u32 m) {
        if (t_due < tu) return 0xFFFFFFFFu;  // applied
        if constexpr (PIN) {
            if (m == 0u) return 0xFFFFFFFFu;  // on a pinned node: never applied
        }
        const u32 x = addr ^ f.warp_cols;   // (word << 10) | (chain << 2)
        return (t_due - tu) * f.W + ((x & 0xFFFFFC00u) | ((31u - __clz(m)) << 5) | ((x >> 2) & 31u));
    };
    ps0.e0 = position(ps.t0, ps.a0, ps.m0);
    ps0.e1 = position(ps.t1, ps.a1, ps.m1);
    ps0.last_p1 = (ps.next - tu) * f.W + ps.last_p1;
    cnt.cur = (int)cur; cnt.run = run;
    if constexpr (GOAL) *hit = h;
    return t;
}

// PIN (k_ssd_pinned, k_passage): perturbation events are masked with the free-node mask s_free of the block's variant.
// GOAL (k_passage): each count is a goal test recording this lane's first hit in *hit (ssd_goal), and the warp leaves the
// loop when no lane is live (*hit != ~0u in every lane): checked once per two-iteration trip on the static paths, once per
// iteration in the tail.
template <int NET, int MODE, int TQ, bool HAS_ENV, bool FULL, bool PIN = false, bool GOAL = false>
__device__ __forceinline__ void ssd_loop(const SsdLoopArgs &a, const Col &st, Draw<MODE> &d, Draw<MODE> &dp, const u32 *s_free = nullptr,
                                         u32 *hit = nullptr) {
    const NetView &nv = a.nv;
    const SsdParams &sp = a.sp;
    const u32 lane = threadIdx.x & 31u;
    const bool active = FULL || lane < a.nvalid;
    const u32 n = (u32)nv.n, W = n * 32u;
    const float inv = sp.inv;
    const float hmd = 0.5f - sp.gdelta;  // gap shortcut: 0.5 - margin (negative: never taken)
    const bool flips = inv <= 0.f;
    SsdPerturb ps{0xFFFFFFFFu, 0xFFFFFFFFu, 0u};
    char *warp_cols = reinterpret_cast<char *>(a.sst + (threadIdx.x & ~31u));
    SsdCount cnt{active ? ssd_bucket(sp, a.s_tgt, st) : 0, 0u};
    int t = 0;
    if constexpr (MODE == PBN_DRAW_PHILOX && !HAS_ENV && FULL && NET == PBN_NET_PRED && TQ > 0) {
        if (flips && sp.smem_hist && sp.fast_t0 >= 0 && nv.off_rec16) t = ssd_loop_pred_static<TQ, PIN, GOAL>(a, st, d, dp, ps, cnt, s_free, hit);
        if constexpr (GOAL) {
            if (t < 0) return;  // the warp left early: d, dp and ps were not handed back, and nothing follows
        }
    }
    if constexpr (MODE == PBN_DRAW_PHILOX && !HAS_ENV && FULL) {
        // STATIC path: one Philox block of the update stream per two iterations, words used in stream order
        u32 ublk = d.blk;
        for (; t + 1 < a.iters; t += 2) {
            if constexpr (GOAL) {
                if (__all_sync(0xFFFFFFFFu, *hit != ~0u)) {
                    t = a.iters;
                    break;
                }
            }
            u32 x0, x1, x2, x3;
            philox4x32_10(ublk, d.c1, d.c2, d.c3, d.k0, d.k1, x0, x1, x2, x3);
            ublk++;
            if constexpr (GOAL) ssd_goal(*hit, a, st, (u32)t);
            else ssd_count(cnt, a, st);
            if (flips) ssd_perturb<true, PIN>(ps, dp, warp_cols, W, inv, hmd, 32u, s_free);
            micro_step_words<NET, TQ>(nv, a.blob, st, x0, x1, d);
            __syncwarp();  // updates land before the next iteration's cross-lane flips
            if constexpr (GOAL) ssd_goal(*hit, a, st, (u32)t + 1u);
            else ssd_count(cnt, a, st);
            if (flips) ssd_perturb<true, PIN>(ps, dp, warp_cols, W, inv, hmd, 32u, s_free);
            micro_step_words<NET, TQ>(nv, a.blob, st, x2, x3, d);
            __syncwarp();
        }
        d.blk = ublk;  // the stream object takes over where the static part stopped (block boundary)
        d.have = 0;
    }
    if constexpr (MODE == PBN_DRAW_PHILOX && HAS_ENV) {
        // WINDOWED path (step-until-attractor inside every iteration): the number of updates per iteration is heavy-tailed,
        // and iteration by iteration a warp would wait for its slowest chain every time.  The perturbation stream does not
        // depend on the states, so the flip masks of the next `win` iterations are drawn first (warp-cooperatively, as
        // always); then every chain runs through those iterations at its own pace in a flat loop whose trip is "start an
        // iteration" or "one attractor test + at most one update", and the warp only waits once per window.
        if (a.flipbuf != nullptr && !a.ev.force) {
            const int w32 = nv.w32;
            u32 *fb = a.flipbuf + (size_t)(threadIdx.x >> 5) * a.win * w32 * 32;
            u32 pos = 0;  // updates this chain's stream has served so far in this launch
            while (t < a.iters) {
                const int kk = a.iters - t < a.win ? a.iters - t : a.win;
                for (int k = 0; k < kk; k++) {
                    for (int w = 0; w < w32; w++) fb[(k * w32 + w) * 32 + lane] = 0u;
                    __syncwarp();
                    if (flips) ssd_perturb_buf<FULL>(ps, dp, fb + k * w32 * 32, W, inv, hmd, a.nvalid);
                }
                __syncwarp();
                int k = 0, in = 0;
                bool start = true;
                for (;;) {
                    const bool live = active && k < kk;
                    if (!__any_sync(0xFFFFFFFFu, live)) break;
                    if (live) {
                        if (start) {
                            ssd_count(cnt, a, st);
                            for (int w = 0; w < w32; w++) st.set_word(w, st.word(w) ^ fb[(k * w32 + w) * 32 + lane]);
                            micro_step<NET, MODE, TQ>(nv, a.blob, st, d);  // env.step(0): pbn_target.py:269-271
                            in = 1;
                            pos++;
                            start = false;
                        } else if (in >= a.ev.max_inner || is_attracting(a.ev, a.att_off, a.cubes, st, w32)) {
                            k++;
                            start = true;
                        } else {
                            micro_step<NET, MODE, TQ>(nv, a.blob, st, d);
                            in++;
                            pos++;
                        }
                    }
                    if constexpr (NET == PBN_NET_PRED) {
                        // straggler mode (as in k_env_step_att): the last chains of the warp inside their attractor loops are
                        // finished by groups of lanes, all groups at once
                        const unsigned hv = __ballot_sync(0xFFFFFFFFu, live && !start && k < kk);
                        if (hv != 0u && __popc(__ballot_sync(0xFFFFFFFFu, active && k < kk)) <= PBN_COOP_MAX) {
                            const u32 base = pos - (u32)in;
                            const int v = w32 == 1 ? coop_take_over<TQ, true>(hv, nv, a.ev, a.dv, a.blob, a.att_off, a.cubes, a.sst, a.coop_buf,
                                                                              a.chain_id, in, base, a.ev.max_inner, 32)
                                                   : coop_take_over<TQ, false>(hv, nv, a.ev, a.dv, a.blob, a.att_off, a.cubes, a.sst, a.coop_buf,
                                                                               a.chain_id, in, base, a.ev.max_inner, 32);
                            if (v != in) {
                                pos += (u32)(v - in);
                                in = v;
                                d.seek(a.dv, 0, a.chain_id, 2u * pos, 0u);  // later iterations go on drawing from this stream
                            }
                        }
                    }
                }
                __syncwarp();
                t += kk;
            }
        }
    }
    for (; t < a.iters; t++) {
        if constexpr (GOAL) {
            if (__all_sync(0xFFFFFFFFu, *hit != ~0u)) break;
            if (active) ssd_goal(*hit, a, st, (u32)t);
        } else {
            if (active) ssd_count(cnt, a, st);
        }
        if constexpr (MODE == PBN_DRAW_REPLAY) {
            if (active)
                for (u32 j = 0; j < n; j++)
                    if (d.dbl() < sp.p) st.flip(j);  // np.random.rand(N) < p ; flipNode(j)  (eval.py:92-95)
        } else {
            if (flips) ssd_perturb<FULL, PIN>(ps, dp, warp_cols, W, inv, hmd, a.nvalid, s_free);
        }
        if (active) {
            micro_step<NET, MODE, TQ>(nv, a.blob, st, d);  // env.step(0): pbn_target.py:269-271
            if constexpr (HAS_ENV) {
                if (!a.ev.force) {
                    int in = 1;
                    while (in < a.ev.max_inner && !is_attracting(a.ev, a.att_off, a.cubes, st, nv.w32)) {
                        micro_step<NET, MODE, TQ>(nv, a.blob, st, d);
                        in++;
                    }
                }
            }
        }
        if constexpr (MODE == PBN_DRAW_PHILOX) __syncwarp();  // updates land before the next iteration's cross-lane flips
    }
    if constexpr (!GOAL) {
        if (active && cnt.run) {
            if (sp.smem_hist) atomicAdd(&a.shist[cnt.cur], cnt.run);
            else atomicAdd(&a.hist[cnt.cur], (unsigned long long)cnt.run);
        }
    }
}

#ifndef PBN_SSD_MIN_BLOCKS
#define PBN_SSD_MIN_BLOCKS 4
#endif
template <int NET, int MODE, int TQ, bool HAS_ENV>
__global__ void __launch_bounds__(PBN_BLOCK, HAS_ENV ? 3 : PBN_SSD_MIN_BLOCKS) k_ssd(NetView nv, EnvView ev, DrawView dv, SsdParams sp, u32 *state,
                                                   long long chains, long long env0, int iters,
                                                   unsigned long long *hist) {
    unsigned char *blob = smem_raw;
    const SsdSmem L = ssd_smem(nv, ev, sp, HAS_ENV);
    unsigned char *img = smem_raw + L.img;
    u32 *s_tgt = reinterpret_cast<u32 *>(smem_raw + L.tgt);
    u32 *shist = reinterpret_cast<u32 *>(smem_raw + L.hist);
    const int nb = 1 << sp.g;
    // the columns (L.cols) addressed from the histogram: from smem_raw + L.cols, ptxas allocates the SSD loops' registers
    // differently (other register counts and spill sizes in several instantiations)
    u32 *sst = align_cols(shist + (sp.smem_hist ? nb : 0), nv.w32);
    stage(blob, nv.blob, L.image);
    if (HAS_ENV) stage(img, ev.img, ev.img_bytes);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < 24; k++) s_tgt[k] = (u32)sp.tgt[k];  // static indices: read straight from the parameter bank
    }
    if (sp.smem_hist)
        for (int b = threadIdx.x; b < nb; b += PBN_BLOCK) shist[b] = 0;
    const int *att_off = reinterpret_cast<const int *>(img);
    const u32 *cubes = reinterpret_cast<const u32 *>(img + ev.off_cubes);
    const long long e = (long long)blockIdx.x * PBN_BLOCK + threadIdx.x;
    const int w32 = nv.w32;
    Col st{sst + threadIdx.x};
    const int win = sp.win;
    u32 *flipbuf = (HAS_ENV && win > 0) ? sst + L.flip : nullptr;
    unsigned char *coop_buf = flipbuf ? reinterpret_cast<unsigned char *>(flipbuf + L.coop) : nullptr;
    const bool active = e < chains;
    if (active) load_state(st, state, chains, e, w32);
    __syncthreads();
    // a warp runs as long as its first chain exists; its missing lanes (tail of the job) still take part in the
    // warp-cooperative perturbation stream but own no state
    const long long warp_left = chains - (e - (threadIdx.x & 31));
    if (warp_left > 0) {
        Draw<MODE> d, dp;
        d.init(dv, e, env0 + e);
        dp.init_perturb(dv, e, env0 + e);
        const u32 nvalid = warp_left >= 32 ? 32u : (u32)warp_left;  // lanes of this warp that own a chain
        SsdLoopArgs a{nv, ev, sp, dv, blob, att_off, cubes, s_tgt, shist, hist, sst, iters, nvalid, flipbuf, win, env0 + e, coop_buf};
        if (nvalid == 32u) ssd_loop<NET, MODE, TQ, HAS_ENV, true>(a, st, d, dp);   // every lane owns a chain: no predication
        else ssd_loop<NET, MODE, TQ, HAS_ENV, false>(a, st, d, dp);
        if (active) {
            store_state(st, state, chains, e, w32);
            d.done(dv, e);
        }
    }
    if (sp.smem_hist) {
        __syncthreads();
        for (int b = threadIdx.x; b < nb; b += PBN_BLOCK)
            if (shist[b]) atomicAdd(&hist[b], (unsigned long long)shist[b]);
    }
}

// A 16-bit predictor LUT (or its doubled 32-bit form) whose index bit b reads the constant c: every entry takes the value of
// its partner with bit b = c.  M = the indices with bit b clear, s = the distance to their partners.
__device__ __forceinline__ u32 lut_fold(u32 lut, u32 b, u32 c) {
    const u32 M = b == 0 ? 0x55555555u : (b == 1 ? 0x33333333u : (b == 2 ? 0x0F0F0F0Fu : 0x00FF00FFu));
    const u32 s = 1u << b;
    return c ? (lut & ~M) | ((lut & ~M) >> s) : (lut & M) | ((lut & M) << s);
}

// Edge pin (src -> dst, c) on the block's copy of the image: node dst's function reads c in place of node src; src not an
// input of dst: nothing changes.  A second pin of the same edge changes nothing either (it folds a bit the function no
// longer depends on), so the first entry of a row applies.  Called, not inlined, with the image fields by value: inlined,
// or given the kernel's NetView, it changes how ptxas schedules the SSD loop of k_ssd_pinned behind the patch.
//   Predictor networks fold LUT bit 3 - j of each of dst's fmax records (padding records too) whose input byte j is src,
//   in the 8-byte records and, when present, both halves of the doubled LUT of the 16-byte ones.
//   Truth-table networks (threshold table staged) fold index bit k - 1 - j of dst's 2^k thresholds where its input j is
//   src, in place: an entry the fold reads is never written by it.
struct FoldImage { unsigned char *blob; int off_rec, off_rec16, fmax, off_node, off_in, off_thr; };
template <int NET>
__device__ __noinline__ void fold_edge(FoldImage im, u32 dst, u32 src, u32 c) {
    if constexpr (NET == PBN_NET_PRED) {
        uint2 *rec = reinterpret_cast<uint2 *>(im.blob + im.off_rec) + dst * im.fmax;
        uint4 *r16 = reinterpret_cast<uint4 *>(im.blob + im.off_rec16) + dst * im.fmax;
        for (int k = 0; k < im.fmax; k++)
            for (u32 j = 0; j < 4; j++) {
                if (((rec[k].x >> (8 * j)) & 0xFFu) != src) continue;
                rec[k].y = lut_fold(rec[k].y, 3u - j, c);
                if (im.off_rec16) r16[k].z = lut_fold(r16[k].z, 3u - j, c);
            }
    } else {
        const uint2 nr = reinterpret_cast<const uint2 *>(im.blob + im.off_node)[dst];
        const unsigned short *in = reinterpret_cast<const unsigned short *>(im.blob + im.off_in) + (nr.y & 0xFFFFu);
        u32 *thr = reinterpret_cast<u32 *>(im.blob + im.off_thr) + nr.x;
        const u32 k = nr.y >> 16;
        for (u32 j = 0; j < k; j++) {
            if (in[j] != src) continue;
            const u32 s = 1u << (k - 1u - j);
            for (u32 idx = 0; idx < (1u << k); idx++)
                if (!(idx & s)) {
                    if (c) thr[idx] = thr[idx | s];
                    else thr[idx | s] = thr[idx];
                }
        }
    }
}

// Word w of a variant's care mask: bits at or above N are ignored
__device__ __forceinline__ u32 pin_care_word(int n, int w32, const u32 *care, int w) {
    return (w == w32 - 1 && (n & 31)) ? care[w] & ((1u << (n & 31)) - 1u) : care[w];
}

// The pins of variant blockIdx.y (k_ssd_pinned, k_passage) on the block's copy of the image, called when the image has been
// staged: the free-node mask s_free (read by the SSD loop behind a later barrier), the caller's other shared words
// (`stage_rest`), then behind a block barrier the pinned edges of the free nodes folded and the records of the pinned nodes
// patched.  `edges` is the variant's row of E edge entries.  Inlined, in this order: ptxas schedules the static SSD loop
// of k_ssd_pinned behind it differently otherwise (109.5 instructions per iteration as a call taking the image fields by
// value, as fold_edge does; 103, or longer perturbation rounds, when the barrier or s_free move).
// (edge entry dst | src << 12 | c << 24, 0xFFFFFFFF = empty: 12 bits hold every node index that gets here, as predictor
// networks have at most 256 nodes and a staged threshold table at most 4096 entries, one or more per node)
template <int NET, class F>
__device__ __forceinline__ void pin_patch(const NetView &nv, unsigned char *blob, u32 *s_free, const u32 *care, const u32 *value,
                                          u32 tt_const, const u32 *edges, int E, F &&stage_rest) {
    for (int w = threadIdx.x; w < nv.w32; w += PBN_BLOCK) s_free[w] = ~pin_care_word(nv.n, nv.w32, care, w);
    stage_rest();
    __syncthreads();
    for (int i = threadIdx.x; i < nv.n; i += PBN_BLOCK) {
        if (!((care[i >> 5] >> (i & 31)) & 1u)) {
            for (int k = 0; k < E; k++) {
                const u32 x = edges[k];
                if (x != 0xFFFFFFFFu && (x & 0xFFFu) == (u32)i)
                    fold_edge<NET>(FoldImage{blob, nv.off_rec, nv.off_rec16, nv.fmax, nv.off_node, nv.off_in, nv.off_thr}, (u32)i,
                                   (x >> 12) & 0xFFFu, (x >> 24) & 1u);
            }
            continue;
        }
        const u32 v = (value[i >> 5] >> (i & 31)) & 1u;
        if constexpr (NET == PBN_NET_PRED) {  // every predictor's LUT all zeros or all ones
            uint2 *rec = reinterpret_cast<uint2 *>(blob + nv.off_rec) + i * nv.fmax;
            for (int k = 0; k < nv.fmax; k++) rec[k].y = v ? 0xFFFFu : 0u;
            if (nv.off_rec16) {  // the doubled LUT field of the 16-byte records
                uint4 *r16 = reinterpret_cast<uint4 *>(blob + nv.off_rec16) + i * nv.fmax;
                for (int k = 0; k < nv.fmax; k++) r16[k].z = v ? 0xFFFFFFFFu : 0u;
            }
        } else {  // no inputs, table entry tt_const + v (staged behind the image, or read through thr_dev)
            reinterpret_cast<uint2 *>(blob + nv.off_node)[i] = make_uint2(tt_const + v, 0u);
        }
    }
}

// A chain's start state under its variant's pins: every pinned node set to its value
__device__ __forceinline__ void pin_state(const NetView &nv, const Col &st, const u32 *care, const u32 *value) {
    for (int w = 0; w < nv.w32; w++) {
        const u32 c = pin_care_word(nv.n, nv.w32, care, w);
        st.set_word(w, (st.word(w) & ~c) | (value[w] & c));
    }
}

// k_ssd (no env, Philox draws) under K pin sets (pbn_ssd_pinned_edges): variant k owns blocks (x, k), its chain c is state
// column k * chains + c and draws from the streams of chain id env0 + c, as in k_ssd.  A pin acts through the block's copy of
// the network image, where the pinned node's function becomes the constant (an update that picks it draws as usual) and an
// edge pin folds the input it pins out of its target's function, and through the perturbation events, whose bit is masked
// with the variant's free nodes where it is formed (pin_patch).
template <int NET, int TQ>
__global__ void __launch_bounds__(PBN_BLOCK, PBN_SSD_MIN_BLOCKS) k_ssd_pinned(NetView nv, DrawView dv, SsdParams sp, u32 *state,
                                                                              long long chains, long long env0, int iters,
                                                                              unsigned long long *hist, const u32 *pin_care,
                                                                              const u32 *pin_value, u32 tt_const,
                                                                              const u32 *pin_edges, int E) {
    EnvView ev;
    memset(&ev, 0, sizeof ev);
    unsigned char *blob = smem_raw;
    const SsdSmem L = ssd_smem(nv, ev, sp, false, true);
    u32 *s_free = reinterpret_cast<u32 *>(smem_raw + L.pin);
    u32 *s_tgt = reinterpret_cast<u32 *>(smem_raw + L.tgt);
    u32 *shist = reinterpret_cast<u32 *>(smem_raw + L.hist);
    const int nb = 1 << sp.g;
    u32 *sst = align_cols(shist + (sp.smem_hist ? nb : 0), nv.w32);
    const int w32 = nv.w32;
    const u32 *care = pin_care + (size_t)blockIdx.y * w32, *value = pin_value + (size_t)blockIdx.y * w32;
    stage(blob, nv.blob, L.image);
    pin_patch<NET>(nv, blob, s_free, care, value, tt_const, pin_edges + (size_t)blockIdx.y * E, E, [&] {
        if (threadIdx.x == 0) {
#pragma unroll
            for (int k = 0; k < 24; k++) s_tgt[k] = (u32)sp.tgt[k];
        }
        if (sp.smem_hist)
            for (int b = threadIdx.x; b < nb; b += PBN_BLOCK) shist[b] = 0;
    });
    const long long e = (long long)blockIdx.x * PBN_BLOCK + threadIdx.x;
    const long long B = (long long)gridDim.y * chains, col = (long long)blockIdx.y * chains + e;
    Col st{sst + threadIdx.x};
    const bool active = e < chains;
    if (active) {
        load_state(st, state, B, col, w32);
        pin_state(nv, st, care, value);
    }
    __syncthreads();
    unsigned long long *vhist = hist + ((size_t)blockIdx.y << sp.g);
    const long long warp_left = chains - (e - (threadIdx.x & 31));
    if (warp_left > 0) {
        Draw<PBN_DRAW_PHILOX> d, dp;
        d.init(dv, e, env0 + e);
        dp.init_perturb(dv, e, env0 + e);
        const u32 nvalid = warp_left >= 32 ? 32u : (u32)warp_left;
        SsdLoopArgs a{nv, ev, sp, dv, blob, nullptr, nullptr, s_tgt, shist, vhist, sst, iters, nvalid, nullptr, 0, env0 + e, nullptr};
        if (nvalid == 32u) ssd_loop<NET, PBN_DRAW_PHILOX, TQ, false, true, true>(a, st, d, dp, s_free);
        else ssd_loop<NET, PBN_DRAW_PHILOX, TQ, false, false, true>(a, st, d, dp, s_free);
        if (active) store_state(st, state, B, col, w32);
    }
    if (sp.smem_hist) {
        __syncthreads();
        for (int b = threadIdx.x; b < nb; b += PBN_BLOCK)
            if (shist[b]) atomicAdd(&vhist[b], (unsigned long long)shist[b]);
    }
}

// The goal of k_passage: bit b (bit b & 31 of word b >> 5) = bucket b lies in the goal, 2^g <= 4096 buckets.  A parameter
// of its own rather than a field of SsdParams, whose size sets the parameter offsets of every k_ssd instantiation.
struct GoalMask { u32 w[128]; };

// First passage into the goal (pbn_first_passage): k_ssd_pinned's chains, variants and draws, with the count of each
// iteration replaced by a goal test (ssd_loop's GOAL).  The goal mask is staged where k_ssd_pinned keeps its histogram.
// t_hit [K][chains] (index = state column): a chain whose entry is >= 0 has arrived and is neither run nor written (its lane
// still draws the warp's perturbation stream); any other gets t0 + its first hit, or keeps -1 and has its state stored.
template <int NET, int TQ>
__global__ void __launch_bounds__(PBN_BLOCK, PBN_SSD_MIN_BLOCKS) k_passage(NetView nv, DrawView dv, SsdParams sp, u32 *state,
                                                                           long long chains, long long env0, int iters,
                                                                           long long t0, long long *t_hit, const u32 *pin_care,
                                                                           const u32 *pin_value, u32 tt_const,
                                                                           const u32 *pin_edges, int E, GoalMask goal) {
    EnvView ev;
    memset(&ev, 0, sizeof ev);
    unsigned char *blob = smem_raw;
    const SsdSmem L = ssd_smem(nv, ev, sp, false, true);  // sp.smem_hist: g <= 12
    u32 *s_free = reinterpret_cast<u32 *>(smem_raw + L.pin);
    u32 *s_tgt = reinterpret_cast<u32 *>(smem_raw + L.tgt);
    u32 *s_goal = reinterpret_cast<u32 *>(smem_raw + L.hist);
    const int nb = 1 << sp.g;
    u32 *sst = align_cols(s_goal + nb, nv.w32);
    const int w32 = nv.w32;
    const u32 *care = pin_care + (size_t)blockIdx.y * w32, *value = pin_value + (size_t)blockIdx.y * w32;
    stage(blob, nv.blob, L.image);
    pin_patch<NET>(nv, blob, s_free, care, value, tt_const, pin_edges + (size_t)blockIdx.y * E, E, [&] {
        if (threadIdx.x == 0) {
#pragma unroll
            for (int k = 0; k < 24; k++) s_tgt[k] = (u32)sp.tgt[k];
#pragma unroll
            for (int k = 0; k < 128; k++)  // static indices: read straight from the parameter bank
                if (k < ((nb + 31) >> 5)) s_goal[k] = goal.w[k];
        }
    });
    const long long e = (long long)blockIdx.x * PBN_BLOCK + threadIdx.x;
    const long long B = (long long)gridDim.y * chains, col = (long long)blockIdx.y * chains + e;
    Col st{sst + threadIdx.x};
    const bool active = e < chains;
    const bool run = active && t_hit[col] < 0;
    if (run) {
        load_state(st, state, B, col, w32);
        pin_state(nv, st, care, value);
    }
    __syncthreads();
    const long long warp_left = chains - (e - (threadIdx.x & 31));
    if (warp_left > 0) {
        Draw<PBN_DRAW_PHILOX> d, dp;
        d.init(dv, e, env0 + e);
        dp.init_perturb(dv, e, env0 + e);
        const u32 nvalid = warp_left >= 32 ? 32u : (u32)warp_left;
        u32 hit = run ? ~0u : 0u;  // a lane without a chain to run is never live
        SsdLoopArgs a{nv, ev, sp, dv, blob, nullptr, nullptr, s_tgt, s_goal, nullptr, sst, iters, nvalid, nullptr, 0, env0 + e, nullptr};
        if (nvalid == 32u) ssd_loop<NET, PBN_DRAW_PHILOX, TQ, false, true, true, true>(a, st, d, dp, s_free, &hit);
        else ssd_loop<NET, PBN_DRAW_PHILOX, TQ, false, false, true, true>(a, st, d, dp, s_free, &hit);
        if (run) {
            if (hit != ~0u) t_hit[col] = t0 + (long long)hit;
            else store_state(st, state, B, col, w32);
        }
    }
}

// ----------------------------------------------------------------------------------------------- pack / unpack
__global__ void k_unpack(const u32 *state, long long B, int n, unsigned char *out) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= B * n) return;
    const long long e = idx / n;
    const int i = (int)(idx - e * n);
    out[idx] = (unsigned char)((state[(long long)(i >> 5) * B + e] >> (i & 31)) & 1u);
}
__global__ void k_pack(const unsigned char *in, long long B, int n, int w32, u32 *state) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= B * w32) return;
    const long long e = idx % B;
    const int w = (int)(idx / B);
    u32 acc = 0;
    for (int b = 0; b < 32 && w * 32 + b < n; b++) acc |= (u32)(in[e * n + w * 32 + b] != 0) << b;
    state[(long long)w * B + e] = acc;
}

// ----------------------------------------------------------------------------------------------- issue-peak microbenchmarks
__global__ void __launch_bounds__(256) k_peak_alu(long long iters, u32 *sink) {
    u32 a0 = threadIdx.x, a1 = a0 * 3 + 1, a2 = a0 * 5 + 2, a3 = a0 * 7 + 3, a4 = a0 ^ 0x55, a5 = a0 + 9, a6 = ~a0, a7 = a0 << 3;
    const u32 k = blockIdx.x | 1;
    for (long long t = 0; t < iters; t++) {
#pragma unroll
        for (int u = 0; u < 8; u++) {  // 8 independent chains x 2 ops (LOP3 + IADD3) x 8 = 128 ops / iteration
            a0 = (a0 ^ k) + a1; a1 = (a1 ^ k) + a2; a2 = (a2 ^ k) + a3; a3 = (a3 ^ k) + a4;
            a4 = (a4 ^ k) + a5; a5 = (a5 ^ k) + a6; a6 = (a6 ^ k) + a7; a7 = (a7 ^ k) + a0;
        }
    }
    if ((a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7) == 0x12345678u) sink[0] = a0;
}
// single-opcode variants (inline PTX so that ptxas cannot trade one opcode for another): which pipe an opcode class issues on,
// and at what rate, decides how far a given instruction MIX can get towards one instruction per cycle per scheduler
template <int OP>  // 0 = LOP3, 1 = SHF (funnel shift), 2 = IMAD (mad.lo), 3 = IADD3
__global__ void __launch_bounds__(256) k_peak_op(long long iters, u32 *sink) {
    u32 a[8];
#pragma unroll
    for (int i = 0; i < 8; i++) a[i] = threadIdx.x * (2 * i + 3) + i;
    const u32 k = blockIdx.x | 1, k2 = (blockIdx.x << 3) | 5;
    for (long long t = 0; t < iters; t++) {
#pragma unroll
        for (int u = 0; u < 16; u++) {  // 8 independent chains x 16 = 128 ops / iteration
#pragma unroll
            for (int i = 0; i < 8; i++) {
                if (OP == 0) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(a[i]) : "r"(k), "r"(k2));
                else if (OP == 1) asm volatile("shf.r.wrap.b32 %0, %0, %1, %2;" : "+r"(a[i]) : "r"(k), "r"(k2));
                else if (OP == 2) asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(a[i]) : "r"(k), "r"(k2));
                else asm volatile("add.u32 %0, %0, %1;" : "+r"(a[i]) : "r"(k));
            }
        }
    }
    u32 x = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) x ^= a[i];
    if (x == 0x12345678u) sink[0] = x;
}
__global__ void __launch_bounds__(256) k_peak_philox(long long iters, u32 *sink) {
    u32 acc = 0, o0, o1, o2, o3;
    const u32 tid = blockIdx.x * blockDim.x + threadIdx.x;
    for (long long t = 0; t < iters; t++) {
        philox4x32_10((u32)t, 0, tid, 0, 1234u, 5678u, o0, o1, o2, o3);
        acc ^= o0 ^ o1 ^ o2 ^ o3;
    }
    if (acc == 0x12345678u) sink[0] = acc;
}

extern "C" int pbn_issue_peak(int32_t kind, int64_t iters, float *ms_out, double *ops_out) {
    int dev = 0, sms = 0;
    CK(cudaGetDevice(&dev));
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    u32 *sink = nullptr;
    CK(cudaMalloc(&sink, 4));
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a));
    CK(cudaEventCreate(&b));
    const int grid = sms * 8, block = 256;
    for (int rep = 0; rep < 2; rep++) {  // first pass warms up
        CK(cudaEventRecord(a));
        if (kind == 0) k_peak_alu<<<grid, block>>>(iters, sink);
        else if (kind == 1) k_peak_philox<<<grid, block>>>(iters, sink);
        else if (kind == 2) k_peak_op<0><<<grid, block>>>(iters, sink);
        else if (kind == 3) k_peak_op<1><<<grid, block>>>(iters, sink);
        else if (kind == 4) k_peak_op<2><<<grid, block>>>(iters, sink);
        else if (kind == 5) k_peak_op<3><<<grid, block>>>(iters, sink);
        else return fail(PBN_ERR_ARG, "pbn_issue_peak: kind must be 0..5");
        CK(cudaEventRecord(b));
        CK(cudaEventSynchronize(b));
    }
    CK(cudaGetLastError());
    CK(cudaEventElapsedTime(ms_out, a, b));
    *ops_out = (double)grid * block * (double)iters * (kind == 1 ? 1.0 : 128.0);
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    cudaFree(sink);
    return PBN_OK;
}

// ----------------------------------------------------------------------------------------------- launch glue
// A launch's dynamic shared memory (its layout's bytes) against what a block of `kernel` may have: the device's opt-in maximum
// less the kernel's static shared memory.  A layout that does not fit is refused and nothing is launched.
template <class K>
static int fit_smem(K kernel, const char *name, size_t bytes) {
    int dev = 0, optin = 0;
    cudaFuncAttributes fa;
    CK(cudaGetDevice(&dev));
    CK(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    CK(cudaFuncGetAttributes(&fa, kernel));
    const size_t avail = (size_t)optin - fa.sharedSizeBytes;
    if (bytes > avail)
        return fail(PBN_ERR_UNSUPPORTED, std::string(name) + " needs " + std::to_string(bytes) +
                                             " bytes of shared memory per block; the device allows " + std::to_string(avail));
    // static + dynamic shared memory above 48 KB needs the opt-in
    if (fa.sharedSizeBytes + bytes > 48 * 1024) CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return PBN_OK;
}

// Kernels are instantiated per (network kind, draw source, threshold quads TQ); TQ = 1 covers predictor sets with up to 5
// predictors per node (every shipped *_5_* set), TQ = 4 up to 17 (the 28_15 set), TQ = 0 reads the count at run time.
// f(NK, MD, TQ) gets the three as std::integral_constant, usable as template arguments.
template <int V>
using Ic = std::integral_constant<int, V>;
template <class F>
static int dispatch(int kind, int mode, int ts, F &&f) {
    if (kind == PBN_NET_PRED && mode == PBN_DRAW_PHILOX) {
        if (ts == 4) return f(Ic<PBN_NET_PRED>(), Ic<PBN_DRAW_PHILOX>(), Ic<1>());
        if (ts == 16) return f(Ic<PBN_NET_PRED>(), Ic<PBN_DRAW_PHILOX>(), Ic<4>());
        return f(Ic<PBN_NET_PRED>(), Ic<PBN_DRAW_PHILOX>(), Ic<0>());
    }
    if (kind == PBN_NET_PRED) return f(Ic<PBN_NET_PRED>(), Ic<PBN_DRAW_REPLAY>(), Ic<0>());
    if (mode == PBN_DRAW_PHILOX) return f(Ic<PBN_NET_TT>(), Ic<PBN_DRAW_PHILOX>(), Ic<0>());
    return f(Ic<PBN_NET_TT>(), Ic<PBN_DRAW_REPLAY>(), Ic<0>());
}

static int check_draws(const PbnDraws *d) {
    if (!d) return fail(PBN_ERR_ARG, "draws is null");
    if (d->mode != PBN_DRAW_PHILOX && d->mode != PBN_DRAW_REPLAY) return fail(PBN_ERR_ARG, "unknown draw mode");
    if (d->mode == PBN_DRAW_REPLAY && (!d->ints || !d->dbls)) return fail(PBN_ERR_ARG, "replay draws need ints and dbls");
    return PBN_OK;
}

extern "C" int pbn_rollout(const PbnNet *net, uint32_t *state, int64_t B, int64_t env0, int64_t steps, int32_t sync,
                           const PbnDraws *draws, void *stream) {
    if (!net || !state || B < 0 || steps < 0) return fail(PBN_ERR_ARG, "bad argument");
    if (int rc = check_draws(draws)) return rc;
    if (B == 0 || steps == 0) return PBN_OK;
    const NetView &nv = net->v;
    const DrawView dv = make_draws(draws);
    cudaStream_t s = (cudaStream_t)stream;
    if (sync == 2) {  // bit-sliced synchronous mode
        if (nv.kind != PBN_NET_PRED || !nv.lutmask || nv.ts != 4)
            return fail(PBN_ERR_UNSUPPORTED, "bit-sliced synchronous mode needs a predictor network with at most 5 predictors per node");
        if (dv.mode != PBN_DRAW_PHILOX) return fail(PBN_ERR_UNSUPPORTED, "bit-sliced synchronous mode has no replay source (use sync=1)");
        if (env0 & 31) return fail(PBN_ERR_ARG, "env0 must be a multiple of 32: a group of 32 consecutive env ids shares the random words");
        if (steps >= (1 << 20)) return fail(PBN_ERR_ARG, "at most 2^20 steps per launch");
        const size_t sm = sliced_smem(nv).bytes;
        if (sm > 200 * 1024) return fail(PBN_ERR_UNSUPPORTED, "network too large for the bit-sliced tables");
        if (int rc = fit_smem(k_sync_sliced, "k_sync_sliced", sm)) return rc;
        const long long groups = (B + 31) / 32;
        const unsigned g2 = (unsigned)((groups + PBN_BLOCK / 32 - 1) / (PBN_BLOCK / 32));
        k_sync_sliced<<<g2, PBN_BLOCK, sm, s>>>(nv, dv, state, B, env0, (int)steps);
        CK(cudaGetLastError());
        return PBN_OK;
    }
    const unsigned grid = (unsigned)((B + PBN_BLOCK - 1) / PBN_BLOCK);
    const size_t smem = rollout_smem(nv, sync).bytes;
    return dispatch(nv.kind, dv.mode, nv.ts, [&](auto NK, auto MD, auto TQ) {
        if (int rc = fit_smem(k_rollout<NK, MD, TQ>, "k_rollout", smem)) return rc;
        k_rollout<NK, MD, TQ><<<grid, PBN_BLOCK, smem, s>>>(nv, dv, state, B, env0, steps, sync);
        CK(cudaGetLastError());
        return PBN_OK;
    });
}

// Persistent grid of k_env_step_att: as many blocks as stay resident, each owning a contiguous range of envs (group mode: one
// env per four lanes).  A resume pass learns its env count on the device; B only bounds it.
static int att_grid(const void *kernel, size_t smem, long long B, bool grp_mode, long long &grid, long long &per_block) {
    int dev = 0, sms = 0, bps = 0;
    CK(cudaGetDevice(&dev));
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kernel, PBN_BLOCK, smem));
    const int envs_per_block = grp_mode ? PBN_BLOCK / 4 : PBN_BLOCK;
    grid = (long long)sms * (bps > 0 ? bps : 1);
    if (grid > (B + envs_per_block - 1) / envs_per_block) grid = (B + envs_per_block - 1) / envs_per_block;
    per_block = (B + grid - 1) / grid;
    grid = (B + per_block - 1) / per_block;
    return PBN_OK;
}

static int env_step_impl(const PbnEnv *env, uint32_t *state, int32_t *n_steps, const int32_t *target_att,
                         const int32_t *actions, int32_t K, uint32_t *obs_state, int32_t *reward, uint8_t *terminated,
                         uint8_t *truncated, int32_t *inner_steps, int64_t B, int64_t env0, const PbnDraws *draws,
                         const PbnVecState *vec, void *stream, double *reward_f64 = nullptr, const PbnStepPlan *plan = nullptr) {
    if (!env || !state || !actions || !reward || !terminated || !truncated || B < 0 || K < 1) return fail(PBN_ERR_ARG, "bad argument");
    if (!reward_f64 && vec && vec->reward_f64) reward_f64 = vec->reward_f64;
    const EnvView &ev = env->v;
    const bool att = ev.kind == PBN_ENV_TARGET || ev.kind == PBN_ENV_MULTI;
    const bool st_kind = ev.kind == PBN_ENV_PBN_ST || ev.kind == PBN_ENV_PBCN_ST;
    if (st_kind && !reward_f64) return fail(PBN_ERR_ARG, "self-triggering envs return a float64 reward: call pbn_env_step_f64");
    if (((ev.kind == PBN_ENV_PBN_ST || ev.kind == PBN_ENV_PBN_SD) && K != 2) ||
        ((ev.kind == PBN_ENV_PBCN_ST || ev.kind == PBN_ENV_PBCN_SD) && K != 1 + ev.n_control))
        return fail(PBN_ERR_ARG, "wrong action width for this env kind");
    if (att && (!n_steps || !target_att)) return fail(PBN_ERR_ARG, "target envs need n_steps and target_att");
    if (int rc = check_draws(draws)) return rc;
    if (B == 0) return PBN_OK;
    const NetView &nv = env->net->v;
    const DrawView dv = make_draws(draws);
    VecView vx;
    memset(&vx, 0, sizeof vx);
    if (vec) {
        if (st_kind && (!vec->ep_return_f64 || !vec->return_sum_f64))
            return fail(PBN_ERR_ARG, "the vector step of a self-triggering env needs ep_return_f64 and return_sum_f64");
        if ((!st_kind && !vec->ep_return) || !vec->ep_len || !vec->stats || !obs_state) return fail(PBN_ERR_ARG, "vector step needs ep_return, ep_len, stats and obs_state");
        if (vec->autoreset) {
            if (int rc = check_draws(&vec->reset_draws)) return rc;
            if (ev.n_att < (ev.kind == PBN_ENV_TARGET ? 2 : 1)) return fail(PBN_ERR_ARG, "autoreset needs attractors");
            if (!att && !env->has_small_att) return fail(PBN_ERR_ARG, "autoreset needs an attractor with at most 10 states (pbn_env.py:196-199)");
            if (att && !vec->target_state) return fail(PBN_ERR_ARG, "autoreset of target envs needs target_state");
            vx.rdv = make_draws(&vec->reset_draws);
        }
        vx.enabled = 1; vx.autoreset = vec->autoreset;
        vx.ep_return = (long long *)vec->ep_return; vx.ep_len = vec->ep_len; vx.stats = (unsigned long long *)vec->stats;
        vx.final_obs = vec->final_obs; vx.target_state = vec->target_state;
        if (st_kind) { vx.ep_return_f64 = vec->ep_return_f64; vx.return_sum_f64 = vec->return_sum_f64; }
        if (vec->probabilities) {
            if (ev.kind != PBN_ENV_MULTI || !vec->pair_ids || ev.n_att < 2 || ev.n_att > 64)
                return fail(PBN_ERR_ARG, "a probability table needs a MULTI env with 2..64 attractors and pair_ids");
            if (dv.mode != PBN_DRAW_PHILOX) return fail(PBN_ERR_UNSUPPORTED, "the curriculum draws its pairs from Philox words");
            vx.cur.prob = vec->probabilities; vx.cur.pair = vec->pair_ids; vx.cur.sample_pair = vec->sample_pair != 0;
        }
    }
    const unsigned grid = (unsigned)((B + PBN_BLOCK - 1) / PBN_BLOCK);
    cudaStream_t s = (cudaStream_t)stream;
    PlanView pl;
    memset(&pl, 0, sizeof pl);
    if (plan) {
        if (!att) return fail(PBN_ERR_UNSUPPORTED, "a step plan applies to the step-until-attractor envs (TARGET, MULTI)");
        if (dv.mode != PBN_DRAW_PHILOX) return fail(PBN_ERR_UNSUPPORTED, "a step plan needs Philox draws (a resumed env re-enters its stream by position)");
        if (!plan->running || !plan->work || !inner_steps) return fail(PBN_ERR_ARG, "a step plan needs running, work and inner_steps");
        if (plan->budget < 0 || (plan->phase != 0 && plan->phase != 1)) return fail(PBN_ERR_ARG, "bad step plan");
        if (ev.kind == PBN_ENV_MULTI && plan->budget == 1) return fail(PBN_ERR_ARG, "MULTI envs need a budget of at least 2 updates");
        pl.budget = plan->budget; pl.resume = plan->resume != 0;
        pl.running = plan->running;
        pl.list_out = plan->work + (size_t)plan->phase * (size_t)(B + 4);
        pl.list_in = plan->work + (size_t)(plan->phase ^ 1) * (size_t)(B + 4);
        CK(cudaMemsetAsync(pl.list_out, 0, 16, s));
    }
    // a budgeted first pass has no tail to cut (every lane owns an env, nobody runs past the budget); images that leave no
    // room run without the group machinery (the per-warp staging of the straggler mode) as well
    const bool first_pass = plan && !pl.resume && pl.budget > 0;
    const int coop_on = att && env_smem(nv, ev, 2, false, true).bytes <= 200 * 1024 && !first_pass;
    // group mode pays when env.steps can be long; under a small cap a lane per env (4x the envs in flight) is faster
    const int grp_mode = coop_on && nv.kind == PBN_NET_PRED && dv.mode == PBN_DRAW_PHILOX && ev.n_att > 0 && !ev.force &&
                         (ev.max_inner > 64 || pl.resume);
    // the lockstep first pass of predictor networks takes the fast-path update where the records and the state width allow it
    const bool fast = nv.off_rec16 != 0 && nv.w32 <= 8 && (nv.ts == 4 || nv.ts == 16);

    // one launch function per kernel; the instantiation is picked below
    auto launch_first = [&](auto kernel, bool fst) -> int {
        const size_t sm = env_smem(nv, ev, 2, fst, false).bytes;
        if (int rc = fit_smem(kernel, "k_env_step_first", sm)) return rc;
        kernel<<<grid, PBN_BLOCK, sm, s>>>(nv, ev, dv, state, n_steps, const_cast<int32_t *>(target_att), actions, K, obs_state,
                                           reward, terminated, truncated, inner_steps, B, env0, pl, vx);
        return PBN_OK;
    };
    auto launch_att = [&](auto kernel) -> int {
        const size_t sm = env_smem(nv, ev, 2, false, coop_on).bytes;
        if (int rc = fit_smem(kernel, "k_env_step_att", sm)) return rc;
        long long pgrid = 0, per_block = 0;
        if (int rc = att_grid((const void *)kernel, sm, B, grp_mode, pgrid, per_block)) return rc;
        kernel<<<(unsigned)pgrid, PBN_BLOCK, sm, s>>>(nv, ev, dv, state, n_steps, target_att, actions, K, obs_state, reward,
                                                     terminated, truncated, inner_steps, B, env0, per_block, coop_on, grp_mode, pl, vx);
        return PBN_OK;
    };
    auto launch_step = [&](auto kernel) -> int {
        const size_t sm = env_smem(nv, ev, 1, false, false).bytes;
        if (int rc = fit_smem(kernel, "k_env_step", sm)) return rc;
        kernel<<<grid, PBN_BLOCK, sm, s>>>(nv, ev, dv, state, n_steps, target_att, actions, K, obs_state, reward, terminated,
                                           truncated, inner_steps, B, env0, vx, reward_f64);
        return PBN_OK;
    };
    const int rc = dispatch(nv.kind, dv.mode, att ? nv.ts : 0, [&](auto NK, auto MD, auto TQ) -> int {
        if (!att) return launch_step(k_env_step<NK, MD>);
        if constexpr (NK == PBN_NET_PRED && MD == PBN_DRAW_PHILOX) {
            if (first_pass) {  // lockstep first pass (Philox: checked above)
                if constexpr (TQ > 0) {
                    if (fast) return launch_first(k_env_step_first<TQ, true>, true);
                }
                return launch_first(k_env_step_first<TQ, false>, false);
            }
        }
        if (NK == PBN_NET_PRED && MD == PBN_DRAW_PHILOX && nv.w32 == 1) return launch_att(k_env_step_att<NK, MD, TQ, true>);
        return launch_att(k_env_step_att<NK, MD, TQ, false>);
    });
    if (rc) return rc;
    CK(cudaGetLastError());
    return PBN_OK;
}

extern "C" int pbn_env_step(const PbnEnv *env, uint32_t *state, int32_t *n_steps, const int32_t *target_att,
                            const int32_t *actions, int32_t K, uint32_t *obs_state, int32_t *reward, uint8_t *terminated,
                            uint8_t *truncated, int32_t *inner_steps, int64_t B, int64_t env0, const PbnDraws *draws,
                            void *stream) {
    return env_step_impl(env, state, n_steps, target_att, actions, K, obs_state, reward, terminated, truncated, inner_steps, B,
                         env0, draws, nullptr, stream);
}

extern "C" int pbn_env_step_f64(const PbnEnv *env, uint32_t *state, int32_t *n_steps, const int32_t *target_att,
                                const int32_t *actions, int32_t K, uint32_t *obs_state, int32_t *reward, double *reward_f64,
                                uint8_t *terminated, uint8_t *truncated, int32_t *inner_steps, int64_t B, int64_t env0,
                                const PbnDraws *draws, void *stream) {
    if (!reward_f64) return fail(PBN_ERR_ARG, "reward_f64 is null");
    return env_step_impl(env, state, n_steps, target_att, actions, K, obs_state, reward, terminated, truncated, inner_steps, B,
                         env0, draws, nullptr, stream, reward_f64);
}

extern "C" int pbn_vec_step(const PbnEnv *env, uint32_t *state, int32_t *n_steps, int32_t *target_att, const int32_t *actions,
                            int32_t K, uint32_t *obs_state, int32_t *reward, uint8_t *terminated, uint8_t *truncated,
                            int32_t *inner_steps, const PbnVecState *vec, int64_t B, int64_t env0, const PbnDraws *draws,
                            void *stream) {
    if (!vec) return fail(PBN_ERR_ARG, "vec is null");
    return env_step_impl(env, state, n_steps, target_att, actions, K, obs_state, reward, terminated, truncated, inner_steps, B,
                         env0, draws, vec, stream);
}

extern "C" int pbn_env_step_plan(const PbnEnv *env, uint32_t *state, int32_t *n_steps, int32_t *target_att, const int32_t *actions,
                                 int32_t K, uint32_t *obs_state, int32_t *reward, uint8_t *terminated, uint8_t *truncated,
                                 int32_t *inner_steps, const PbnVecState *vec, const PbnStepPlan *plan, int64_t B, int64_t env0,
                                 const PbnDraws *draws, void *stream) {
    if (!plan) return fail(PBN_ERR_ARG, "plan is null");
    return env_step_impl(env, state, n_steps, target_att, actions, K, obs_state, reward, terminated, truncated, inner_steps, B,
                         env0, draws, vec, stream, nullptr, plan);
}

static int env_reset_impl(const PbnEnv *env, uint32_t *state, int32_t *n_steps, int32_t *target_att, uint32_t *target_state,
                          const uint8_t *mask, int64_t B, int64_t env0, const PbnDraws *draws, void *stream, CurView cv);
extern "C" int pbn_env_reset(const PbnEnv *env, uint32_t *state, int32_t *n_steps, int32_t *target_att, uint32_t *target_state,
                             const uint8_t *mask, int64_t B, int64_t env0, const PbnDraws *draws, void *stream) {
    return env_reset_impl(env, state, n_steps, target_att, target_state, mask, B, env0, draws, stream, CurView{nullptr, nullptr, 0});
}
extern "C" int pbn_env_reset_cur(const PbnEnv *env, uint32_t *state, int32_t *n_steps, int32_t *target_att, uint32_t *target_state,
                                 const uint8_t *mask, double *probabilities, int32_t *pair_ids, int32_t sample_pair, int64_t B,
                                 int64_t env0, const PbnDraws *draws, void *stream) {
    if (!env || !probabilities || !pair_ids) return fail(PBN_ERR_ARG, "bad argument");
    if (env->v.kind != PBN_ENV_MULTI || env->v.n_att < 2 || env->v.n_att > 64)
        return fail(PBN_ERR_ARG, "a probability table needs a MULTI env with 2..64 attractors");
    if (!draws || draws->mode != PBN_DRAW_PHILOX) return fail(PBN_ERR_UNSUPPORTED, "the curriculum draws its pairs from Philox words");
    return env_reset_impl(env, state, n_steps, target_att, target_state, mask, B, env0, draws, stream,
                          CurView{probabilities, pair_ids, sample_pair != 0});
}
static int env_reset_impl(const PbnEnv *env, uint32_t *state, int32_t *n_steps, int32_t *target_att, uint32_t *target_state,
                          const uint8_t *mask, int64_t B, int64_t env0, const PbnDraws *draws, void *stream, CurView cv) {
    if (!env || !state || B < 0) return fail(PBN_ERR_ARG, "bad argument");
    const EnvView &ev = env->v;
    if (ev.kind == PBN_ENV_TARGET || ev.kind == PBN_ENV_MULTI) {
        if (!n_steps || !target_att) return fail(PBN_ERR_ARG, "target envs need n_steps and target_att");
        if (ev.n_att < (ev.kind == PBN_ENV_TARGET ? 2 : 1)) return fail(PBN_ERR_ARG, "reset needs attractors (sample of 2, pbn_target.py:333)");
    } else {
        if (ev.n_att < 1) return fail(PBN_ERR_ARG, "reset needs attractors");
        // pbn_env.py:196-199 redraws an attractor until one has at most 10 states; in Python that loop can be interrupted, on
        // the device it would hang the GPU
        if (!env->has_small_att) return fail(PBN_ERR_ARG, "reset needs an attractor with at most 10 states (pbn_env.py:196-199 would loop forever)");
    }
    if (int rc = check_draws(draws)) return rc;
    if (B == 0) return PBN_OK;
    const DrawView dv = make_draws(draws);
    const unsigned grid = (unsigned)((B + PBN_BLOCK - 1) / PBN_BLOCK);
    cudaStream_t s = (cudaStream_t)stream;
    if (dv.mode == PBN_DRAW_PHILOX)
        k_env_reset<PBN_DRAW_PHILOX><<<grid, PBN_BLOCK, 0, s>>>(env->net->v, ev, dv, state, n_steps, target_att, target_state, mask, B, env0, cv);
    else
        k_env_reset<PBN_DRAW_REPLAY><<<grid, PBN_BLOCK, 0, s>>>(env->net->v, ev, dv, state, n_steps, target_att, target_state, mask, B, env0, cv);
    CK(cudaGetLastError());
    return PBN_OK;
}

extern "C" int pbn_rand_state(const PbnNet *net, uint32_t *state, int64_t B, int64_t env0, const PbnDraws *draws, void *stream) {
    if (!net || !state || B < 0) return fail(PBN_ERR_ARG, "bad argument");
    if (int rc = check_draws(draws)) return rc;
    if (B == 0) return PBN_OK;
    const DrawView dv = make_draws(draws);
    const unsigned grid = (unsigned)((B + PBN_BLOCK - 1) / PBN_BLOCK);
    cudaStream_t s = (cudaStream_t)stream;
    if (dv.mode == PBN_DRAW_PHILOX) k_rand_state<PBN_DRAW_PHILOX><<<grid, PBN_BLOCK, 0, s>>>(net->v, dv, state, B, env0);
    else k_rand_state<PBN_DRAW_REPLAY><<<grid, PBN_BLOCK, 0, s>>>(net->v, dv, state, B, env0);
    CK(cudaGetLastError());
    return PBN_OK;
}

extern "C" int pbn_env_attractor_index(const PbnEnv *env, const uint32_t *state, int64_t B, int32_t *att_out, void *stream) {
    if (!env || !state || !att_out || B < 0) return fail(PBN_ERR_ARG, "bad argument");
    const EnvView &ev = env->v;
    if (ev.n_att < 1) return fail(PBN_ERR_ARG, "the env has no attractor list");
    if (B == 0) return PBN_OK;
    const int w32 = env->net->v.w32;
    const unsigned grid = (unsigned)((B + PBN_BLOCK - 1) / PBN_BLOCK);
    // staged only while three blocks stay resident per SM: the kernel is one pass over the states, and a large cube list
    // read by every thread of a block is served from L1 as well
    const int staged = index_smem(ev, w32, true).bytes <= 64 * 1024;
    const size_t smem = index_smem(ev, w32, staged).bytes;
    if (int rc = fit_smem(k_attractor_index, "k_attractor_index", smem)) return rc;
    k_attractor_index<<<grid, PBN_BLOCK, smem, (cudaStream_t)stream>>>(ev, w32, state, B, att_out, staged);
    CK(cudaGetLastError());
    return PBN_OK;
}

// Exhaustive check of the gap shortcut for one value of inv: the gap depends on the top 23 bits of the draw only.
__global__ void __launch_bounds__(256) k_geom_verify(float inv, float dlt, unsigned int *bad, unsigned int *taken) {
    const u32 r = ((u32)blockIdx.x * 256u + threadIdx.x) << 9;
    bool ok;
    const u32 a = geom_gap_approx(r, inv, 0.5f - dlt, &ok);
    if (ok) {
        if (a != geom_gap(r, inv)) atomicAdd(bad, 1u);
    } else {
        atomicAdd(taken, 1u);  // inputs that take the polynomial anyway
    }
}
// Margin for inv, or 1.0 (shortcut off) when it would not pay or the exhaustive comparison finds a disagreement.  Verified once
// per value of inv and device (blocking, ~0.1 ms); during stream capture an unverified value runs without the shortcut.
static float geom_shortcut_delta(float inv, cudaStream_t s) {
    static std::mutex mu;
    static std::map<std::pair<int, u32>, float> cache;
    if (!(inv < 0.f)) return 1.0f;
    // |lg2.approx - log2| <= 2^-22 * max(1, |log2 u|) (documented), |log2 u| <= 24; the polynomial is within 2e-7 of log2 on
    // the reduced interval; twice the sum, scaled by |inv|
    const float dlt = -inv * 2.0f * (24.0f * 2.3841858e-7f + 2e-7f);
    if (!(dlt < 0.05f)) return 1.0f;  // more than ~10 % of the draws would fall back: not worth it
    int dev = 0;
    cudaGetDevice(&dev);
    u32 bits;
    memcpy(&bits, &inv, 4);
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find({dev, bits});
    if (it != cache.end()) return it->second;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(s, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone) return 1.0f;
    unsigned int *d = nullptr, h[2] = {1u, 0u};
    float res = 1.0f;
    if (cudaMalloc(&d, 8) == cudaSuccess) {
        if (cudaMemsetAsync(d, 0, 8, s) == cudaSuccess) {
            k_geom_verify<<<(1u << 23) / 256u, 256, 0, s>>>(inv, dlt, d, d + 1);
            if (cudaMemcpyAsync(h, d, 8, cudaMemcpyDeviceToHost, s) == cudaSuccess && cudaStreamSynchronize(s) == cudaSuccess &&
                h[0] == 0u)
                res = dlt;
        }
        cudaFree(d);
    }
    cache[{dev, bits}] = res;
    return res;
}

extern "C" int pbn_geom_shortcut_check(double p, float *delta, uint32_t *disagree, uint32_t *fallback) {
    if (!(p > 0.0 && p < 1.0) || !delta || !disagree || !fallback) return fail(PBN_ERR_ARG, "bad argument");
    const float inv = (float)(1.0 / std::log2(1.0 - p));
    *delta = geom_shortcut_delta(inv, nullptr);
    const float dlt = -inv * 2.0f * (24.0f * 2.3841858e-7f + 2e-7f);  // the margin the shortcut would use
    unsigned int *d = nullptr, h[2] = {0u, 0u};
    CK(cudaMalloc(&d, 8));
    cudaMemset(d, 0, 8);
    k_geom_verify<<<(1u << 23) / 256u, 256>>>(inv, dlt < 0.5f ? dlt : 0.5f, d, d + 1);
    cudaError_t e = cudaMemcpy(h, d, 8, cudaMemcpyDeviceToHost);
    cudaFree(d);
    CK(e);
    *disagree = h[0];
    *fallback = h[1];
    return PBN_OK;
}

// The static SSD loop finds the window (iteration) of a perturbation position e without a divide: e / W, W = 32 n, is
// umulhi(e >> 4, wq_mul) >> wq_sh.  Exact for every position the loop forms: those are below 2^31 + 2^14 (a round starts
// at most W <= 8192 into its window and spans 64 gaps of at most 2^25 + 1), so y = e >> 4 < 2^28 and e / W = y / d with
// d = 2n >= 2.  With sh = ceil(log2 d) - 1 and mul = ceil(2^(32+sh) / d) = (2^(32+sh) + r) / d, 0 <= r < d <= 2^(sh+1):
// y mul / 2^(32+sh) = y / d + y r / (d 2^(32+sh)) and y r < 2^28 2^(sh+1) < 2^(32+sh), so the excess is below 1/d and
// cannot reach the next integer.  mul < 2^32 because d > 2^sh.
static void ssd_window_div(int n, SsdParams &sp) {
    const unsigned long long d = 2ull * (unsigned)n;
    sp.wq_sh = 63 - __builtin_clzll(d - 1);
    sp.wq_mul = (unsigned)(((1ull << (32 + sp.wq_sh)) + d - 1) / d);
}

// Argument checks and launch parameters shared by pbn_ssd and pbn_ssd_pinned (sp.win is left to the caller).  *run = false:
// nothing to launch (no chains or no iterations).
static int ssd_prepare(const NetView &nv, int64_t chains, int64_t env0, int64_t iters, double p, const int32_t *tgt, int32_t g,
                       const PbnDraws *draws, cudaStream_t s, SsdParams &sp, bool *run) {
    *run = false;
    if (g < 1 || g > 24) return fail(PBN_ERR_ARG, "1 <= g <= 24 target nodes");
    if (!(p >= 0.0 && p <= 1.0)) return fail(PBN_ERR_ARG, "Invalid Bit Flip Probability value.");  // eval.py:31-33
    if (int rc = check_draws(draws)) return rc;
    if (chains == 0 || iters == 0) return PBN_OK;
    if (draws->mode == PBN_DRAW_PHILOX && p > 0 && (env0 & 31))
        return fail(PBN_ERR_ARG, "env0 must be a multiple of 32: the perturbation stream is shared by groups of 32 consecutive chain ids");
    if (p > 0 && p < 1e-6) return fail(PBN_ERR_UNSUPPORTED, "bit_flip_prob below 1e-6 is not supported (gap law is truncated at 2^25)");
    sp.g = g; sp.p = p; sp.smem_hist = g <= 12;
    sp.inv = p <= 0 ? 1.0f : (p >= 1 ? 0.0f : (float)(1.0 / std::log2(1.0 - p)));
    sp.gdelta = 1.0f;
    sp.win = 0;
    ssd_window_div(nv.n, sp);
    memset(sp.tgt, 0, sizeof sp.tgt);
    for (int k = 0; k < g; k++) {
        if (tgt[k] < 0 || tgt[k] >= nv.n) return fail(PBN_ERR_ARG, "target node out of range");
        if (tgt[k] > 32767) return fail(PBN_ERR_UNSUPPORTED, "target node indices above 32767 are not supported");
        sp.tgt[k] = (short)tgt[k];
    }
    // fast bucket path: targets are consecutive ascending nodes inside one 32-bit state word
    sp.fast_t0 = tgt[0];
    for (int k = 1; k < g; k++)
        if (tgt[k] != tgt[0] + k) sp.fast_t0 = -1;
    if (sp.fast_t0 >= 0 && (tgt[0] >> 5) != ((tgt[0] + g - 1) >> 5)) sp.fast_t0 = -1;
    if (iters >= (1LL << 31) || (sp.smem_hist && (double)iters * PBN_BLOCK >= 4294967296.0))
        return fail(PBN_ERR_ARG, "iters too large for one launch; split the estimate");
    if (draws->mode == PBN_DRAW_PHILOX) sp.gdelta = geom_shortcut_delta(sp.inv, s);  // gaps are drawn with the verified shortcut
    *run = true;
    return PBN_OK;
}

extern "C" int pbn_ssd(const PbnNet *net, const PbnEnv *env, uint32_t *state, int64_t chains, int64_t env0, int64_t iters,
                       double p, const int32_t *tgt, int32_t g, uint64_t *hist, const PbnDraws *draws, void *stream) {
    if (!net || !state || !tgt || !hist || chains < 0 || iters < 0) return fail(PBN_ERR_ARG, "bad argument");
    if (env && env->net != net) return fail(PBN_ERR_ARG, "env belongs to another network");
    const NetView &nv = net->v;
    cudaStream_t s = (cudaStream_t)stream;
    SsdParams sp;
    bool run;
    if (int rc = ssd_prepare(nv, chains, env0, iters, p, tgt, g, draws, s, sp, &run)) return rc;
    if (!run) return PBN_OK;
    const DrawView dv = make_draws(draws);
    const unsigned grid = (unsigned)((chains + PBN_BLOCK - 1) / PBN_BLOCK);
    EnvView ev;
    memset(&ev, 0, sizeof ev);
    if (env) ev = env->v;
    // windowed step-until-attractor path: flip masks of `win` iterations per warp, 2 KB per warp (networks up to 256 nodes)
    sp.win = (env && draws->mode == PBN_DRAW_PHILOX && !ev.force && nv.w32 <= 8) ? (16 / nv.w32 > 2 ? 16 / nv.w32 : 2) : 0;
    const size_t smem = ssd_smem(nv, ev, sp, env != nullptr).bytes;
    auto launch = [&](auto kernel) -> int {
        if (int rc = fit_smem(kernel, "k_ssd", smem)) return rc;
        kernel<<<grid, PBN_BLOCK, smem, s>>>(nv, ev, dv, sp, state, chains, env0, (int)iters, (unsigned long long *)hist);
        CK(cudaGetLastError());
        return PBN_OK;
    };
    return dispatch(nv.kind, dv.mode, nv.ts, [&](auto NK, auto MD, auto TQ) {
        return env ? launch(k_ssd<NK, MD, TQ, true>) : launch(k_ssd<NK, MD, TQ, false>);
    });
}

// Argument checks and launch set-up shared by pbn_ssd_pinned_edges and pbn_first_passage.  *run = false: nothing to launch.
struct PinnedLaunch {
    SsdParams sp;
    NetView nv;
    DrawView dv;
    size_t smem;
    dim3 grid;
};
static int pinned_prepare(const PbnNet *net, const uint32_t *state, int64_t chains, int64_t env0, int64_t iters, double p,
                          const uint32_t *pin_care, const uint32_t *pin_value, int32_t K, const uint32_t *pin_edges, int32_t E,
                          const int32_t *tgt, int32_t g, const PbnDraws *draws, cudaStream_t s, PinnedLaunch &P, bool *run) {
    *run = false;
    if (!net || !state || !pin_care || !pin_value || !tgt || chains < 0 || iters < 0) return fail(PBN_ERR_ARG, "bad argument");
    if (K < 1 || K > 65535) return fail(PBN_ERR_ARG, "1 <= K <= 65535 pin sets");
    if (E < 0 || E > 64) return fail(PBN_ERR_ARG, "0 <= E <= 64 edge slots per pin set");
    if (E > 0 && !pin_edges) return fail(PBN_ERR_ARG, "E > 0 edge slots need pin_edges");
    if (draws && draws->mode == PBN_DRAW_REPLAY) return fail(PBN_ERR_UNSUPPORTED, "pinned SSD estimates draw from Philox streams only");
    // folding an edge rewrites the node's thresholds, which a table read through thr_dev would need a per-variant copy of
    if (E > 0 && net->v.thr_dev) return fail(PBN_ERR_UNSUPPORTED, "edge pins need the threshold table in shared memory (at most PBN_TT_THR_SMEM_MAX bytes)");
    if (int rc = ssd_prepare(net->v, chains, env0, iters, p, tgt, g, draws, s, P.sp, run)) return rc;
    if (!*run) return PBN_OK;
    P.nv = net->v;
    // a truth-table network whose threshold table is staged also stages the two constant entries behind it
    if (P.nv.kind == PBN_NET_TT && !P.nv.thr_dev) P.nv.blob_bytes = P.nv.blob_fast_bytes = P.nv.blob_bytes + 16;
    P.dv = make_draws(draws);
    EnvView ev;
    memset(&ev, 0, sizeof ev);
    P.smem = ssd_smem(P.nv, ev, P.sp, false, true).bytes;
    P.grid = dim3((unsigned)((chains + PBN_BLOCK - 1) / PBN_BLOCK), (unsigned)K);
    return PBN_OK;
}

extern "C" int pbn_ssd_pinned_edges(const PbnNet *net, uint32_t *state, int64_t chains, int64_t env0, int64_t iters, double p,
                                    const uint32_t *pin_care, const uint32_t *pin_value, int32_t K, const uint32_t *pin_edges,
                                    int32_t E, const int32_t *tgt, int32_t g, uint64_t *hist, const PbnDraws *draws, void *stream) {
    if (!hist) return fail(PBN_ERR_ARG, "bad argument");
    cudaStream_t s = (cudaStream_t)stream;
    PinnedLaunch P;
    bool run;
    if (int rc = pinned_prepare(net, state, chains, env0, iters, p, pin_care, pin_value, K, pin_edges, E, tgt, g, draws, s, P, &run))
        return rc;
    if (!run) return PBN_OK;
    auto launch = [&](auto kernel) -> int {
        if (int rc = fit_smem(kernel, "k_ssd_pinned", P.smem)) return rc;
        kernel<<<P.grid, PBN_BLOCK, P.smem, s>>>(P.nv, P.dv, P.sp, state, chains, env0, (int)iters, (unsigned long long *)hist,
                                                 pin_care, pin_value, net->tt_const, pin_edges, (int)E);
        CK(cudaGetLastError());
        return PBN_OK;
    };
    return dispatch(P.nv.kind, P.dv.mode, P.nv.ts, [&](auto NK, auto, auto TQ) { return launch(k_ssd_pinned<NK, TQ>); });
}

extern "C" int pbn_first_passage(const PbnNet *net, uint32_t *state, int64_t chains, int64_t env0, int64_t iters, int64_t t0,
                                 double p, const uint32_t *pin_care, const uint32_t *pin_value, int32_t K,
                                 const uint32_t *pin_edges, int32_t E, const int32_t *tgt, int32_t g, const uint32_t *goal_host,
                                 int64_t *t_hit, const PbnDraws *draws, void *stream) {
    if (!goal_host || !t_hit || t0 < 0) return fail(PBN_ERR_ARG, "bad argument");
    if (g < 1 || g > 12) return fail(PBN_ERR_ARG, "1 <= g <= 12 target nodes: the goal mask sits where the block histogram would");
    cudaStream_t s = (cudaStream_t)stream;
    PinnedLaunch P;
    bool run;
    if (int rc = pinned_prepare(net, state, chains, env0, iters, p, pin_care, pin_value, K, pin_edges, E, tgt, g, draws, s, P, &run))
        return rc;
    if (!run) return PBN_OK;
    GoalMask goal;
    memset(&goal, 0, sizeof goal);
    memcpy(goal.w, goal_host, (g >= 5 ? (size_t)1 << (g - 5) : 1) * 4);
    auto launch = [&](auto kernel) -> int {
        if (int rc = fit_smem(kernel, "k_passage", P.smem)) return rc;
        kernel<<<P.grid, PBN_BLOCK, P.smem, s>>>(P.nv, P.dv, P.sp, state, chains, env0, (int)iters, (long long)t0,
                                                 (long long *)t_hit, pin_care, pin_value, net->tt_const, pin_edges, (int)E, goal);
        CK(cudaGetLastError());
        return PBN_OK;
    };
    return dispatch(P.nv.kind, P.dv.mode, P.nv.ts, [&](auto NK, auto, auto TQ) { return launch(k_passage<NK, TQ>); });
}

extern "C" int pbn_ssd_pinned(const PbnNet *net, uint32_t *state, int64_t chains, int64_t env0, int64_t iters, double p,
                              const uint32_t *pin_care, const uint32_t *pin_value, int32_t K, const int32_t *tgt, int32_t g,
                              uint64_t *hist, const PbnDraws *draws, void *stream) {
    return pbn_ssd_pinned_edges(net, state, chains, env0, iters, p, pin_care, pin_value, K, nullptr, 0, tgt, g, hist, draws, stream);
}

struct HistParams { int g; short tgt[24]; };
__global__ void __launch_bounds__(256) k_bucket_hist(const u32 *state, long long B, HistParams hp, unsigned long long *hist) {
    extern __shared__ u32 sh[];
    const int nb = 1 << hp.g;
    const bool smem = hp.g <= 12;
    if (smem)
        for (int b = threadIdx.x; b < nb; b += blockDim.x) sh[b] = 0;
    __syncthreads();
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < B; e += (long long)gridDim.x * blockDim.x) {
        int b = 0;
#pragma unroll
        for (int k = 0; k < 24; k++)
            if (k < hp.g) b = (b << 1) | (int)((state[(long long)(hp.tgt[k] >> 5) * B + e] >> (hp.tgt[k] & 31)) & 1u);
        if (smem) atomicAdd(&sh[b], 1u);
        else atomicAdd(&hist[b], 1ULL);
    }
    if (smem) {
        __syncthreads();
        for (int b = threadIdx.x; b < nb; b += blockDim.x)
            if (sh[b]) atomicAdd(&hist[b], (unsigned long long)sh[b]);
    }
}
extern "C" int pbn_bucket_hist(const uint32_t *state, int64_t B, int32_t n_nodes, const int32_t *tgt, int32_t g, uint64_t *hist,
                               void *stream) {
    if (!state || !tgt || !hist || B < 0 || n_nodes < 1) return fail(PBN_ERR_ARG, "bad argument");
    if (g < 1 || g > 24) return fail(PBN_ERR_ARG, "1 <= g <= 24 target nodes");
    if (B == 0) return PBN_OK;
    HistParams hp;
    memset(&hp, 0, sizeof hp);
    hp.g = g;
    for (int k = 0; k < g; k++) {
        if (tgt[k] < 0 || tgt[k] >= n_nodes) return fail(PBN_ERR_ARG, "target node out of range");
        hp.tgt[k] = (short)tgt[k];
    }
    long long blocks = (B + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    k_bucket_hist<<<(unsigned)blocks, 256, g <= 12 ? ((size_t)4 << g) : 0, (cudaStream_t)stream>>>(state, B, hp, (unsigned long long *)hist);
    CK(cudaGetLastError());
    return PBN_OK;
}

extern "C" int pbn_ssd_host(const PbnNet *net, const PbnEnv *env, int64_t chains, int64_t env0, int64_t iters, double p,
                            const int32_t *tgt, int32_t g, uint64_t seed, uint32_t epoch, uint64_t *hist_host) {
    if (!net || !hist_host || chains < 1) return fail(PBN_ERR_ARG, "bad argument");
    if (g < 1 || g > 24) return fail(PBN_ERR_ARG, "1 <= g <= 24 target nodes");
    u32 *state = nullptr;
    uint64_t *hist = nullptr;
    CK(cudaMalloc(&state, (size_t)net->v.w32 * chains * 4));
    CK(cudaMalloc(&hist, (size_t)8 << g));
    CK(cudaMemsetAsync(hist, 0, (size_t)8 << g, 0));
    PbnDraws d;
    memset(&d, 0, sizeof d);
    d.mode = PBN_DRAW_PHILOX; d.seed = seed; d.epoch = epoch;
    int rc = pbn_rand_state(net, state, chains, env0, &d, nullptr);
    d.epoch = epoch + 1;
    if (!rc) rc = pbn_ssd(net, env, state, chains, env0, iters, p, tgt, g, hist, &d, nullptr);
    if (!rc) {
        cudaError_t e = cudaMemcpy(hist_host, hist, (size_t)8 << g, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) rc = fail(PBN_ERR_CUDA, cudaGetErrorString(e));
    }
    cudaFree(state);
    cudaFree(hist);
    return rc;
}

// ----------------------------------------------------------------------------------------------- exhaustive STG
// masks[s] bit i = node i can change value in state s.  Reads the packed image straight from global memory (one pass
// over 2^N states, not a hot loop); probabilities are compared as float64 exactly like common/pbn.py:186-197.
__global__ void __launch_bounds__(256) k_change_masks(NetView nv, u32 *masks) {
    const unsigned long long total = 1ULL << nv.n;
    for (unsigned long long s = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; s < total;
         s += (unsigned long long)gridDim.x * blockDim.x) {
        const u32 st = (u32)s;
        u32 m = 0;
        if (nv.kind == PBN_NET_TT) {
            const uint2 *node = reinterpret_cast<const uint2 *>(nv.blob + nv.off_node);
            const unsigned short *in = reinterpret_cast<const unsigned short *>(nv.blob + nv.off_in);
            for (int i = 0; i < nv.n; i++) {
                const uint2 nr = node[i];
                const int k = (int)(nr.y >> 16);
                u32 idx = 0;
                for (int q = 0; q < k; q++) idx = (idx << 1) | ((st >> in[(nr.y & 0xFFFF) + q]) & 1u);
                const double p = nv.tt_prob[nr.x + idx];
                const u32 cur = (st >> i) & 1u;
                if ((cur == 0 && p > 0.0) || (cur == 1 && p < 1.0)) m |= 1u << i;
            }
        } else {
            const uint2 *rec = reinterpret_cast<const uint2 *>(nv.blob + nv.off_rec);
            for (int i = 0; i < nv.n; i++) {
                const int q0 = nv.pr_off[i], f = nv.pr_off[i + 1] - q0;
                const u32 cur = (st >> i) & 1u;
                bool can = false;
                double prev = 0.0;
                for (int j = 0; j < f; j++) {
                    const double c = nv.pr_cum[q0 + j];
                    if (c > prev) {  // predictor j has positive COD weight: it can be drawn (base.py:94-97)
                        const uint2 r = rec[i * nv.fmax + j];
                        const u32 idx = (((st >> (r.x & 0xFF)) & 1u) << 3) | (((st >> ((r.x >> 8) & 0xFF)) & 1u) << 2) |
                                        (((st >> ((r.x >> 16) & 0xFF)) & 1u) << 1) | ((st >> (r.x >> 24)) & 1u);
                        can |= (((r.y >> idx) & 1u) != cur);
                    }
                    prev = c;
                }
                if (can) m |= 1u << i;
            }
        }
        masks[s] = m;
    }
}

__global__ void __launch_bounds__(256) k_stg_expand(const u32 *masks, int n, const u32 *frontier, const u32 *visited,
                                                    const u32 *within, u32 *next, int direction) {
    const unsigned long long words = (1ULL << n) >> 5 ? (1ULL << n) >> 5 : 1ULL;
    for (unsigned long long w = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; w < words;
         w += (unsigned long long)gridDim.x * blockDim.x) {
        u32 fw = frontier[w];
        while (fw) {
            const int b = __ffs(fw) - 1;
            fw &= fw - 1;
            const u32 s = (u32)(w << 5) | (u32)b;
            if (direction == 0) {  // successors: s ^ (1<<i) for every changeable node i
                u32 m = masks[s];
                while (m) {
                    const int i = __ffs(m) - 1;
                    m &= m - 1;
                    const u32 t = s ^ (1u << i), tw = t >> 5, tb = 1u << (t & 31);
                    if (!(visited[tw] & tb) && (!within || (within[tw] & tb))) atomicOr(&next[tw], tb);
                }
            } else {  // predecessors: t = s ^ (1<<i) with node i changeable in t
                for (int i = 0; i < n; i++) {
                    const u32 t = s ^ (1u << i), tw = t >> 5, tb = 1u << (t & 31);
                    if (!(visited[tw] & tb) && (!within || (within[tw] & tb)) && ((masks[t] >> i) & 1u)) atomicOr(&next[tw], tb);
                }
            }
        }
    }
}

__global__ void k_stg_walk(const u32 *masks, int n, u32 start, long long steps, u32 k0, u32 k1, u32 *out) {
    u32 s = start, o0, o1, o2, o3;
    for (long long t = 0; t < steps; t++) {
        const u32 m = masks[s];
        if (!m) break;  // fixed point
        philox4x32_10((u32)t, (u32)(t >> 32), 0x57a1u, 0, k0, k1, o0, o1, o2, o3);
        int pick = (int)__umulhi(o0, (u32)__popc(m));
        u32 mm = m;
        while (pick--) mm &= mm - 1;
        s ^= 1u << (__ffs(mm) - 1);
    }
    *out = s;
}

extern "C" int pbn_stg_change_masks(const PbnNet *net, uint32_t *masks, void *stream) {
    if (!net || !masks) return fail(PBN_ERR_ARG, "bad argument");
    if (net->v.n > 32) return fail(PBN_ERR_UNSUPPORTED, "the exhaustive state-transition graph supports at most 32 nodes");
    const unsigned long long total = 1ULL << net->v.n;
    unsigned long long blocks = (total + 255) / 256;
    if (blocks > 148ULL * 32) blocks = 148ULL * 32;
    k_change_masks<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(net->v, masks);
    CK(cudaGetLastError());
    return PBN_OK;
}
extern "C" int pbn_stg_expand(const uint32_t *masks, int32_t n, const uint32_t *frontier, const uint32_t *visited,
                              const uint32_t *within, uint32_t *next, int32_t direction, void *stream) {
    if (!masks || !frontier || !visited || !next || n < 1 || n > 32) return fail(PBN_ERR_ARG, "bad argument");
    const unsigned long long words = ((1ULL << n) + 31) >> 5;
    unsigned long long blocks = (words + 255) / 256;
    if (blocks > 148ULL * 32) blocks = 148ULL * 32;
    k_stg_expand<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(masks, n, frontier, visited, within, next, direction);
    CK(cudaGetLastError());
    return PBN_OK;
}
extern "C" int pbn_stg_walk(const uint32_t *masks, int32_t n, uint32_t start, int64_t steps, uint64_t seed, uint32_t *out,
                            void *stream) {
    if (!masks || !out || n < 1 || n > 32 || steps < 0) return fail(PBN_ERR_ARG, "bad argument");
    k_stg_walk<<<1, 1, 0, (cudaStream_t)stream>>>(masks, n, start, steps, (u32)seed, (u32)(seed >> 32), out);
    CK(cudaGetLastError());
    return PBN_OK;
}

extern "C" int pbn_upload(void *dst_dev, const void *src_host, int64_t nbytes, void *stream) {
    if (!dst_dev || !src_host || nbytes < 0) return fail(PBN_ERR_ARG, "bad argument");
    CK(cudaMemcpyAsync(dst_dev, src_host, (size_t)nbytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return PBN_OK;
}
extern "C" int pbn_fetch_host(const void *const *src_dev, const int64_t *nbytes, int32_t n, void *dst_host, void *stream) {
    if (!src_dev || !nbytes || !dst_host || n < 0) return fail(PBN_ERR_ARG, "bad argument");
    char *dst = static_cast<char *>(dst_host);
    for (int i = 0; i < n; i++) {  // one cudaMemcpyAsync per buffer (no batched-copy API)
        CK(cudaMemcpyAsync(dst, src_dev[i], (size_t)nbytes[i], cudaMemcpyDeviceToHost, (cudaStream_t)stream));
        dst += nbytes[i];
    }
    CK(cudaStreamSynchronize((cudaStream_t)stream));
    return PBN_OK;
}

__global__ void k_gather_step(const int *reward, const unsigned char *terminated, const unsigned char *truncated, const int *inner,
                              const u32 *state, const u32 *obs, int w32, long long B, long long e, u32 *out) {
    const int t = threadIdx.x;
    if (t == 0) {
        out[0] = (u32)reward[e];
        out[1] = inner ? (u32)inner[e] : 0u;
        out[2] = (u32)terminated[e] | ((u32)truncated[e] << 8);
    }
    for (int w = t; w < w32; w += blockDim.x) {
        out[3 + w] = state[(long long)w * B + e];
        out[3 + w32 + w] = obs ? obs[(long long)w * B + e] : 0u;
    }
}
extern "C" int pbn_fetch_step_host(const int32_t *reward, const uint8_t *terminated, const uint8_t *truncated, const int32_t *inner,
                                   const uint32_t *state, const uint32_t *obs_state, int32_t w32, int64_t B, int64_t e,
                                   void *scratch_dev, void *dst_host, void *stream) {
    if (!reward || !terminated || !truncated || !state || !scratch_dev || !dst_host || w32 < 1 || e < 0 || e >= B)
        return fail(PBN_ERR_ARG, "bad argument");
    cudaStream_t s = (cudaStream_t)stream;
    k_gather_step<<<1, 32, 0, s>>>(reward, terminated, truncated, inner, state, obs_state, w32, B, e, (u32 *)scratch_dev);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(dst_host, scratch_dev, (size_t)(12 + 8 * w32), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return PBN_OK;
}

extern "C" int pbn_unpack_state(const uint32_t *state, int64_t B, int32_t n, uint8_t *out, void *stream) {
    if (!state || !out || B < 0 || n < 1) return fail(PBN_ERR_ARG, "bad argument");
    if (B == 0) return PBN_OK;
    const long long total = (long long)B * n;
    k_unpack<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(state, B, n, out);
    CK(cudaGetLastError());
    return PBN_OK;
}
extern "C" int pbn_pack_state(const uint8_t *in, int64_t B, int32_t n, uint32_t *state, void *stream) {
    if (!state || !in || B < 0 || n < 1) return fail(PBN_ERR_ARG, "bad argument");
    if (B == 0) return PBN_OK;
    const int w32 = (n + 31) / 32;
    const long long total = (long long)B * w32;
    k_pack<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(in, B, n, w32, state);
    CK(cudaGetLastError());
    return PBN_OK;
}
