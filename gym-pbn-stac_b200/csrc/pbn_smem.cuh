// pbn_smem.cuh — dynamic shared-memory layouts of the kernels of pbn_b200.cu (included there after col_align_bytes and
// pbn_coop.cuh, whose coop_warp_bytes they use), and the SSD launch parameters that the SSD layout reads.
#pragma once

struct SsdParams {
    int g;
    int smem_hist;  // 1: per-block shared histogram (g <= 12), 0: global atomics
    int fast_t0;    // >= 0: the targets are nodes t0, t0+1, .. t0+g-1 inside one state word (bucket = bit-reversed field)
    int win;        // iterations per window of the step-until-attractor path (0 = iteration by iteration)
    float inv;      // 1/log2(1-p) <= 0; a value > 0 means flips disabled (p == 0)
    float gdelta;   // margin of the lg2.approx shortcut of the gap draw (geom_gap_approx); >= 0.5: shortcut off
    unsigned wq_mul;  // window of a perturbation position e: e / (32 n) = umulhi(e >> 4, wq_mul) >> wq_sh (ssd_window_div)
    int wq_sh;
    double p;
    short tgt[24];
};

// One layout per kernel family, computed from the kernel's arguments by the kernel (to carve smem_raw) and by its launch
// (for the byte count).  Regions follow each other in the order they are added, the network image at offset 0.  A column
// region that align_cols aligns starts with a reserve of col_align_bytes(w32): where in it the columns begin depends on the
// shared address, known only in the kernel.  So the regions behind the state columns are given as distances in words from
// the region before them (also where a sum from smem_raw would work: ptxas then allocates the kernels' registers differently).
struct Smem {
    size_t image = 0, bytes = 0;  // bytes of the network image, of the whole layout
    __host__ __device__ size_t add(size_t n) { const size_t at = bytes; bytes += n; return at; }
};
// k_rollout: image (asynchronous rollouts also stage the 16-byte records), two aligned columns per env
struct RolloutSmem : Smem { size_t cols; };
__host__ __device__ inline RolloutSmem rollout_smem(const NetView &nv, bool sync) {
    RolloutSmem L;
    L.bytes = L.image = sync ? nv.blob_bytes : nv.blob_fast_bytes;
    L.cols = L.add(col_align_bytes(nv.w32) + (size_t)2 * nv.w32 * PBN_BLOCK * 4);
    return L;
}
// k_sync_sliced: image, LUT masks (a row of fmax * 16 + 4 words per node), two transposed state groups per warp
struct SlicedSmem : Smem { size_t lm, words; };
__host__ __device__ inline SlicedSmem sliced_smem(const NetView &nv) {
    SlicedSmem L;
    L.bytes = L.image = nv.blob_bytes;
    L.lm = L.add((size_t)nv.n * (nv.fmax * 16 + 4) * 4);
    L.words = L.add((size_t)(PBN_BLOCK / 32) * 2 * nv.w32 * 32 * 4);
    return L;
}
// k_env_step (ncols 1), k_env_step_first and k_env_step_att (ncols 2): image, cube image, the state columns; FAST (lockstep
// first pass) stages the 16-byte records and aligns the columns; `coop` appends the straggler-mode staging of every warp,
// L.coop words behind the start of the columns
struct EnvSmem : Smem {
    size_t img, cols;
    int coop;
};
__host__ __device__ inline EnvSmem env_smem(const NetView &nv, const EnvView &ev, int ncols, bool fast, bool coop) {
    EnvSmem L;
    L.bytes = L.image = fast ? nv.blob_fast_bytes : nv.blob_bytes;
    L.img = L.add(ev.img_bytes);
    L.coop = ncols * nv.w32 * PBN_BLOCK;
    L.cols = L.add((fast ? col_align_bytes(nv.w32) : 0) + (size_t)L.coop * 4);
    L.add(coop ? (size_t)(PBN_BLOCK / 32) * coop_warp_bytes(nv.w32) : 0);
    return L;
}
// k_attractor_index: the cube image when staged, one column per env
struct IndexSmem : Smem { size_t cols; };
__host__ __device__ inline IndexSmem index_smem(const EnvView &ev, int w32, bool staged) {
    IndexSmem L;
    L.add(staged ? ev.img_bytes : 0);
    L.cols = L.add((size_t)w32 * PBN_BLOCK * 4);
    return L;
}
// k_ssd: image (without an env also the 16-byte records), cube image, 32 target words, the block histogram (smem_hist), one
// aligned column per chain; the windowed path (sp.win) adds win flip masks per warp and the straggler-mode staging behind
// the aligned columns: flip and coop are their distances in words from the region before them.  k_ssd_pinned (pin) adds
// the free-node mask of the block's variant (w32 words) in front of the target words.
struct SsdSmem : Smem {
    size_t img, pin, tgt, hist, cols;
    int flip, coop;
};
__host__ __device__ inline SsdSmem ssd_smem(const NetView &nv, const EnvView &ev, const SsdParams &sp, bool env, bool pin = false) {
    SsdSmem L;
    L.bytes = L.image = env ? nv.blob_bytes : nv.blob_fast_bytes;
    L.img = L.add(env ? ev.img_bytes : 0);
    L.pin = L.add(pin ? (size_t)nv.w32 * 4 : 0);
    L.tgt = L.add(32 * 4);
    L.hist = L.add((size_t)(sp.smem_hist ? 1 << sp.g : 0) * 4);
    L.flip = nv.w32 * PBN_BLOCK;
    L.coop = (PBN_BLOCK / 32) * sp.win * nv.w32 * 32;
    const size_t coop = sp.win ? (size_t)(PBN_BLOCK / 32) * coop_warp_bytes(nv.w32) : 0;
    L.cols = L.add(col_align_bytes(nv.w32) + ((size_t)L.flip + L.coop) * 4 + coop);
    return L;
}
