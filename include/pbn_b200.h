/*
 * pbn_b200.h — C-ABI of the B200-native PB(C)N simulator (libpbn_b200.so).
 *
 * The reference (jakub-zarzycki2022/gym-PBN-stac) is pure Python and has no FFI; this ABI sits
 * *below* the drop-in gymnasium classes (gym_PBN.envs.*) and is what they call through ctypes.
 * Every entry point cites the reference interface it replaces.  Plain pointers and sizes only:
 * no torch types.  Unless a name ends in `_host`, every data pointer is a DEVICE pointer and the
 * call only enqueues work on `stream` (a cudaStream_t passed as void*; NULL = default stream).
 *
 * All functions return 0 on success or a PBN_ERR_* code; nothing throws across the boundary.
 * pbn_last_error() returns a thread-local message for the last failure.
 *
 * Layouts
 *   state      uint32 planes [W32][B], W32 = ceil(N/32); node i of env e = bit (i&31) of state[(i>>5)*B + e]
 *   actions    int32 [B][K] row-major
 *   histogram  uint64 [2^g], bucket = target-node bits MSB-first (pbn_target.py:383-391)
 */
#ifndef PBN_B200_H
#define PBN_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PBN_OK 0
#define PBN_ERR_ARG 1         /* bad argument / unsupported size */
#define PBN_ERR_CUDA 2        /* CUDA runtime error (message in pbn_last_error) */
#define PBN_ERR_UNSUPPORTED 3

/* network kinds */
#define PBN_NET_TT 0   /* truth-table PBN / PBCN: gym_PBN/envs/common/{node,pbn,pbcn}.py */
#define PBN_NET_PRED 1 /* Bittner predictor graph: gym_PBN/envs/bittner/base.py Node/Graph */

/* Host-side description handed to the network compiler (arrays are HOST pointers, copied once). */
typedef struct {
    int32_t kind;
    int32_t n_nodes;
    int32_t first_updatable; /* randint lower bound: 1 = PBN.step (common/pbn.py:90), 0 = Graph.step (base.py:308) */
    /* PBN_NET_TT: node i reads tt_in[tt_in_off[i]..tt_in_off[i+1]) (ascending node index, first = MSB of the
       table index, common/node.py:31-32); P(next=1) = tt_prob[tt_tab_off[i] + idx] */
    const int32_t *tt_in_off;  /* [N+1] */
    const int32_t *tt_in;
    const int32_t *tt_tab_off; /* [N+1] */
    const double *tt_prob;
    /* PBN_NET_PRED: node i owns predictors pr_off[i]..pr_off[i+1); predictor q reads nodes pr_in[4q..4q+3]
       (3 inputs, then the node itself: base.py:100-104); pr_lut[q] bit (x0<<3|x1<<2|x2<<1|x3) = [X.A >= 0]
       tabulated on the host with the reference's float expression (base.py:110-118); pr_cum = cumulative COD
       (base.py:30-45); pr_codsum[i] = CODsum */
    const int32_t *pr_off; /* [N+1] */
    const int32_t *pr_in;
    const uint16_t *pr_lut;
    const double *pr_cum;
    const double *pr_codsum; /* [N] */
} PbnNetDesc;

typedef struct PbnNet PbnNet; /* opaque; immutable after creation, shareable across streams */

/* Network compiler back end: lowers the description into the packed device image (gather indices, 16-bit LUTs,
   31-bit integer thresholds) that kernels stage into shared memory.  Replaces PBN.__init__ / Node.__init__
   (common/pbn.py:16-46, common/node.py:6-26) and Node.add_predictors (base.py:30-45). */
int pbn_net_create(const PbnNetDesc *desc, PbnNet **out);
int pbn_net_destroy(PbnNet *net);
int pbn_net_words(const PbnNet *net); /* W32 */

/* Environment kinds: one per reference env class on the hot path. */
#define PBN_ENV_PBN 0     /* PBNEnv             pbn_env.py:125-188 */
#define PBN_ENV_PBCN 1    /* PBCNEnv            pbcn_env.py:52-80 */
#define PBN_ENV_TARGET 2  /* PBNTargetEnv       pbn_target.py:241-326 (+ Bittner7.is_attracting_state :562-574) */
#define PBN_ENV_MULTI 3   /* PBNTargetMultiEnv  pbn_target_multi.py:119-225 */
#define PBN_ENV_PBN_SD 4  /* PBNSampledDataEnv  sampled_data.py:52-88 */
#define PBN_ENV_PBCN_SD 5 /* PBCNSampledDataEnv sampled_data.py:139-189 */
#define PBN_ENV_PBN_ST 6  /* PBNSelfTriggeringEnv  self_triggering.py:56-93 */
#define PBN_ENV_PBCN_ST 7 /* PBCNSelfTriggeringEnv self_triggering.py:146-197 */

typedef struct {
    int32_t kind;
    int32_t horizon;   /* truncated = (n_steps == horizon), pbn_target.py:325 */
    int32_t max_inner; /* cap on updates per env.step (the reference loop is unbounded, pbn_target.py:270-271) */
    int32_t force;     /* PBNTargetEnv.step(force=True): exactly one update */
    int32_t dedup;     /* multi: 1 = tensor actions (unique()'d), 0 = python list, pbn_target_multi.py:120-121 */
    int32_t control_write; /* PBCN sampled-data: 0 = reference (control never reaches the dynamics), 1 = state[0:M] <- control */
    int32_t n_control;
    int32_t successful_reward, wrong_attractor_cost; /* PBCNEnv._get_reward pbcn_env.py:52-65 */
    /* attractor a owns cubes att_off[a]..att_off[a+1); cube c = cube[c*N..(c+1)*N), values 0/1/2 ('*').
       n_att == 0 means every state is attracting.  HOST pointers, copied once. */
    int32_t n_att;
    const int32_t *att_off;
    const int8_t *cube;
    int32_t tgt_first, n_tgt; /* PBN family: the target set = cubes tgt_first .. tgt_first+n_tgt (full states) */
    /* self-triggering envs: gamma_pow[i] = gamma**i as the HOST computes it (Python float pow; the device only multiplies
       and adds), i < n_gamma (later steps reuse the last entry); max_interval = T, 0 = no cap (self_triggering.py:75-80) */
    const double *gamma_pow;
    int32_t n_gamma;
    int32_t max_interval;
} PbnEnvDesc;

typedef struct PbnEnv PbnEnv;
int pbn_env_create(const PbnNet *net, const PbnEnvDesc *desc, PbnEnv **out);
int pbn_env_destroy(PbnEnv *env);

/* Draw source.  PHILOX: Philox4x32-10, key = seed, counter = (block, epoch, env_lo, env_hi); env e consumes
   its own stream sequentially, so results do not depend on how envs are split over launches or GPUs.
   REPLAY: recorded draws of the reference's RNGs (SURVEY.md §3.5), row e = ints + e*int_stride etc. */
#define PBN_DRAW_PHILOX 0
#define PBN_DRAW_REPLAY 1
typedef struct {
    int32_t mode;
    uint32_t epoch;
    uint64_t seed;
    const int32_t *ints; /* device */
    const double *dbls;  /* device */
    int64_t int_stride, dbl_stride;
    int64_t *used; /* device, optional [B][2]: draws consumed per env */
    const uint32_t *epoch_dev; /* device, optional: the launch uses epoch + *epoch_dev.  Lets a captured CUDA graph of an
                                  env.step advance its Philox epoch from device memory between replays (honoured by the env
                                  step / reset entry points: pbn_env_step*, pbn_vec_step, pbn_env_step_plan, pbn_env_reset*) */
} PbnDraws;

/* K1 — `steps` updates of B envs in one launch, state resident on chip.
   sync=0: PBN.step (common/pbn.py:88-92) / Graph.step (base.py:306-312); sync=1: Graph.synch_step (base.py:300-303);
   sync=2: the same synchronous law, bit-sliced over groups of 32 consecutive env ids (predictor networks with at most
   5 predictors per node, Philox draws, env0 % 32 == 0). */
int pbn_rollout(const PbnNet *net, uint32_t *state, int64_t B, int64_t env0, int64_t steps, int32_t sync,
                const PbnDraws *draws, void *stream);

/* K2 — one env.step for B envs: intervention -> update(s) until attracting (cap) -> reward/terminated/truncated.
   actions [B][K]: PBN/PBCN/TARGET K=1; MULTI K slots (<0 = absent); PBN_SD (action, interval);
   PBCN_SD (interval, control bits...); PBN_ST / PBCN_ST need pbn_env_step_f64.  obs_state (optional) receives the packed observation planes (differs from
   `state` only for MULTI's pre-update capture, pbn_target_multi.py:133-135). */
int pbn_env_step(const PbnEnv *env, uint32_t *state, int32_t *n_steps, const int32_t *target_att,
                 const int32_t *actions, int32_t K, uint32_t *obs_state, int32_t *reward, uint8_t *terminated,
                 uint8_t *truncated, int32_t *inner_steps, int64_t B, int64_t env0, const PbnDraws *draws, void *stream);

/* The same call for the self-triggering envs (PBN_ENV_PBN_ST / PBN_ENV_PBCN_ST), whose reward is the discounted sum of the
   inner rewards, a float64 (self_triggering.py:76,178): actions (action, prob 1..10) resp. (prob 1..10, control bits...);
   after every primitive step the macro action stops w.p. prob/10 or at T; reward_f64 [B] receives the sum, `reward` its
   truncation to int, inner_steps the interval.  Draws per primitive step: node index, node value, stop. */
int pbn_env_step_f64(const PbnEnv *env, uint32_t *state, int32_t *n_steps, const int32_t *target_att,
                     const int32_t *actions, int32_t K, uint32_t *obs_state, int32_t *reward, double *reward_f64,
                     uint8_t *terminated, uint8_t *truncated, int32_t *inner_steps, int64_t B, int64_t env0,
                     const PbnDraws *draws, void *stream);

/* Vector-env step: K2 plus, in the same launch, the bookkeeping a batched env needs — running episode return/length,
   block-aggregated statistics (episodes, return sum, length sum, successes, inner-cap hits, env steps, env steps whose
   intervention was out of range and therefore ignored, reserved; accumulated into stats[8]), the step's observation copied to final_obs, and for finished envs the reset (reset_draws, its own epoch), after
   which obs_state holds the NEW state of those envs.  Bit-identical to pbn_env_step followed by a masked pbn_env_reset.
   The reference has no vector env (SURVEY.md §2.1); this serves gym_PBN.b200.vector_env.PBNVectorEnv.step. */
typedef struct {
    int64_t *ep_return;     /* [B] */
    int32_t *ep_len;        /* [B] */
    int64_t *stats;         /* [8] */
    uint32_t *final_obs;    /* planes [W32][B], optional */
    uint32_t *target_state; /* planes [W32][B], written on reset (target envs) */
    int32_t autoreset;
    PbnDraws reset_draws;
    /* curriculum of PBNTargetMultiEnv (pbn_target_multi.py:159-181, 232-235), optional: one probability row per env (a vector
       env is B independent env objects of the reference).  When an episode ends the launch applies rework_probas(episode
       length) to the env's row, and the reset draws the (state attractor, target attractor) ids from it like
       np.random.choice(range(A), size=2, replace=False, p=row) (three Philox words, u = (word + 0.5) / 2^32).  sample_pair = 0
       keeps first -> last for the attractors themselves, as the reference does (SURVEY.md Q14); 1 uses the sampled ids. */
    double *probabilities;  /* [B][n_att], NULL = no curriculum */
    int32_t *pair_ids;      /* [B][2] */
    int32_t sample_pair;
    /* self-triggering envs (PBN_ENV_PBN_ST / PBN_ENV_PBCN_ST; self_triggering.py:56-93,146-197): the macro step's discounted
       float64 reward, the running float64 episode return (instead of ep_return) and the sum of finished episodes' returns
       (instead of stats[1]); with these pbn_vec_step serves them like the other kinds: macro step + bookkeeping + reset in
       one launch */
    double *reward_f64;      /* [B] */
    double *ep_return_f64;   /* [B] */
    double *return_sum_f64;  /* [1] */
} PbnVecState;
int pbn_vec_step(const PbnEnv *env, uint32_t *state, int32_t *n_steps, int32_t *target_att, const int32_t *actions,
                 int32_t K, uint32_t *obs_state, int32_t *reward, uint8_t *terminated, uint8_t *truncated,
                 int32_t *inner_steps, const PbnVecState *vec, int64_t B, int64_t env0, const PbnDraws *draws, void *stream);

/* Budgeted / resumable env.step of the step-until-attractor envs (PBN_ENV_TARGET, PBN_ENV_MULTI; Philox draws).  The
   reference's inner loop `while not is_attracting_state(state): graph.step()` (pbn_target.py:270-271,
   pbn_target_multi.py:135-146) is unbounded and heavy-tailed, and a launch lasts as long as its slowest env; with a plan, a
   launch makes at most `budget` updates per env and PARKS the envs that are still outside every attractor: their state,
   update count (inner_steps) and pending action cost (reward) stay in the caller's arrays, running[e] = 1, and their ids are
   appended to a list in `work`.  A later call with resume = 1 continues exactly those envs from where they stopped (update
   t of an env.step always takes words 2t, 2t+1 of the env's stream: pass the SAME draws as the call that began the step), so
   a step split over k launches is bit-identical to the one-launch result.  This is also how the library itself runs a full
   step fast: a first pass with a small budget in which every lane owns an env (most envs finish within a few updates), then
   a resume pass without budget in which the few long-running envs are spread over the whole GPU, each run by a group of
   lanes (gym_PBN.b200.engine.Simulator.env_step).
     running  uint8 [B]: out, 1 = step unfinished
     work     int32 [2 * (B + 4)]: two parking lists {count, queue head, -, -, env ids...}; list `phase` is written,
              list `phase ^ 1` is read when resume = 1.  The call clears the header of the list it writes.
     budget   updates per env in this launch, 0 = until every env is done (then no env is parked)
     resume   0: every env begins a new env.step (actions applied);  1: the envs of list `phase ^ 1` continue
   vec may be NULL (= pbn_env_step semantics) or the vector-env epilogue of pbn_vec_step, which runs when an env finishes. */
typedef struct {
    uint8_t *running;
    int32_t *work;
    int32_t budget, resume, phase;
} PbnStepPlan;
int pbn_env_step_plan(const PbnEnv *env, uint32_t *state, int32_t *n_steps, int32_t *target_att, const int32_t *actions,
                      int32_t K, uint32_t *obs_state, int32_t *reward, uint8_t *terminated, uint8_t *truncated,
                      int32_t *inner_steps, const PbnVecState *vec_or_null, const PbnStepPlan *plan, int64_t B, int64_t env0,
                      const PbnDraws *draws, void *stream);

/* reset of the envs selected by mask (NULL = all): PBNTargetEnv.reset pbn_target.py:328-352,
   PBNTargetMultiEnv.reset pbn_target_multi.py:227-259, PBNEnv.reset pbn_env.py:190-213 (+ PBN.reset common/pbn.py:55-78). */
int pbn_env_reset(const PbnEnv *env, uint32_t *state, int32_t *n_steps, int32_t *target_att, uint32_t *target_state,
                  const uint8_t *mask, int64_t B, int64_t env0, const PbnDraws *draws, void *stream);

/* pbn_env_reset for PBNTargetMultiEnv with the curriculum table of PbnVecState (same draws: the three pair words come first). */
int pbn_env_reset_cur(const PbnEnv *env, uint32_t *state, int32_t *n_steps, int32_t *target_att, uint32_t *target_state,
                      const uint8_t *mask, double *probabilities, int32_t *pair_ids, int32_t sample_pair, int64_t B,
                      int64_t env0, const PbnDraws *draws, void *stream);

/* att_out[e] = index of the first attractor that has a cube containing state e, -1 if none (pbn_target.py:562-574,
   is_attracting_state, as an index).  state: planes [W32][B].  PBN_ERR_ARG when the env has no attractor list. */
int pbn_env_attractor_index(const PbnEnv *env, const uint32_t *state, int64_t B, int32_t *att_out, void *stream);

/* Graph.genRandState base.py:368-370 */
int pbn_rand_state(const PbnNet *net, uint32_t *state, int64_t B, int64_t env0, const PbnDraws *draws, void *stream);

/* K3 — utils/eval.py:76-103 _ssd_run for `chains` chains x `iters` iterations (model=None), histogram summed over
   chains into hist[2^g] (uint64, accumulated: caller zeroes).  env may be NULL (= one update per iteration).
   bit_flip_prob is 0 (no perturbation) or in [1e-6, 1]: with Philox draws the flips of eval.py:92-95 are drawn as geometric
   gaps (capped at 2^25 positions, which a smaller probability would reach), PBN_ERR_UNSUPPORTED below that; Philox-mode
   shards must start at a multiple of 32 chain ids (env0 % 32 == 0: one perturbation process per 32 consecutive chains). */
int pbn_ssd(const PbnNet *net, const PbnEnv *env, uint32_t *state, int64_t chains, int64_t env0, int64_t iters,
            double bit_flip_prob, const int32_t *tgt_nodes_host, int32_t g, uint64_t *hist, const PbnDraws *draws,
            void *stream);

/* hist[bucket(state_e)] += 1 for every env e — the first two lines of an _ssd_run iteration (utils/eval.py:88-89) as a
   stand-alone kernel, for estimates whose actions come from a policy between steps (eval.py:97-101). */
int pbn_bucket_hist(const uint32_t *state, int64_t B, int32_t n_nodes, const int32_t *tgt_nodes_host, int32_t g,
                    uint64_t *hist, void *stream);

/* Same estimate with HOST buffers: uploads nothing but the description, draws random start states on device
   (genRandState), runs K3 and copies the histogram back; blocks until done.  The call compute_ssd_hist maps to. */
int pbn_ssd_host(const PbnNet *net, const PbnEnv *env, int64_t chains, int64_t env0, int64_t iters,
                 double bit_flip_prob, const int32_t *tgt_nodes_host, int32_t g, uint64_t seed, uint32_t epoch,
                 uint64_t *hist_host);

/* layout helpers: packed planes <-> uint8 [B][N] (what env.render()/get_state() hand out, pbn_target.py:354-355) */
int pbn_unpack_state(const uint32_t *state, int64_t B, int32_t n_nodes, uint8_t *out, void *stream);
int pbn_pack_state(const uint8_t *in, int64_t B, int32_t n_nodes, uint32_t *state, void *stream);

/* Exhaustive asynchronous state-transition graph on the device (networks up to 32 nodes; state s = bit i is node i).
   Replaces the O(2^N) host loops behind PBNEnv.compute_attractors (pbn_env.py:238-244 -> PBN.print_STG /
   _compute_next_states common/pbn.py:132-197) and Graph.genSTG / getNextStates / findAttractors
   (bittner/base.py:199-242,398-399); the attractors are the terminal strongly connected components.
     pbn_stg_change_masks  masks[s] bit i = node i can change value in state s (edge s -> s ^ (1<<i)):
                           truth tables: P(next=1) > 0 from 0, < 1 from 1 (common/pbn.py:186-197, float64 tables);
                           predictor graphs: some predictor with positive COD weight outputs the other value.
     pbn_stg_expand        one BFS level over bitsets of 2^N bits: next |= neighbours(frontier) & ~visited (& within).
                           direction 0 = successors, 1 = predecessors.  `within` may be NULL.
     pbn_stg_walk          `steps` uniformly random forward moves from `start` (a cheap way to land in a terminal SCC). */
int pbn_stg_change_masks(const PbnNet *net, uint32_t *masks, void *stream);
int pbn_stg_expand(const uint32_t *masks, int32_t n_nodes, const uint32_t *frontier, const uint32_t *visited,
                   const uint32_t *within, uint32_t *next, int32_t direction, void *stream);
int pbn_stg_walk(const uint32_t *masks, int32_t n_nodes, uint32_t start, int64_t steps, uint64_t seed, uint32_t *out,
                 void *stream);

/* Network inference — the COD scan of the Bittner predictor-set fitter (gym_PBN/envs/bittner/gen/predictor_sets.py:
   _gen_predictor_sets_gene :41-78, add_to_buff :80-102, gen_COD :105-124).  For every target gene the reference fits
   every triple of other genes (every product of their duplicate rows, every target row) by least squares, rounds the
   fitted values and keeps the n_predictors best coefficients of determination.  Rows are binary over <= 32 samples, so
   a row is one 32-bit mask and the device solves each 4x4 fit in exact integer arithmetic (csrc/pbn_fit.cuh).
     rows      [R] bit s = binarised expression of sample s; gene i owns rows row_off[i]..row_off[i+1]
     cod_rank  [R][S+1] class of the COD a target row gets for k misclassified samples (0 = highest COD), tabulated on
               the host with the reference's float expressions; classes are comparable across the rows of one gene
   Keys (smaller = better): rank<<52 | a<<40 | b<<28 | c<<16 | y<<12 | sc with a<b<c indices into the gene list with
   the target removed, y the target row, sc the index of the input-row product — the reference's visiting order, so ties
   in COD resolve as its strict `<` does.  Per gene g only candidates with key > key_gt[g] and visiting order < arr_lt[g]
   are considered (NULL = no filter).  top_keys receives the [G][top_l] winners in ascending key order (all-ones = empty).
   Candidates whose rounded fit is decided by a fitted value of exactly one half (the reference's outcome then depends on
   float noise) never enter top_keys; when tie_rank_le is given, those whose best case ranks <= tie_rank_le[g] are
   written to tie_keys as (key with the best-case rank, gene) pairs, *n_ties = how many there were (may exceed tie_cap).
   All pointers are HOST pointers; the call blocks.  kernel_ms (optional) = device time of the scan. */
typedef struct {
    int32_t n_genes;
    int32_t n_samples;
    const int32_t *row_off;   /* [G+1] */
    const uint32_t *rows;     /* [R] */
    const uint16_t *cod_rank; /* [R][S+1], values < 1024 */
} PbnFitDesc;
int pbn_fit_scan_host(const PbnFitDesc *desc, int32_t top_l, const uint64_t *key_gt, const uint64_t *arr_lt,
                      const uint16_t *tie_rank_le, uint64_t *top_keys, uint64_t *tie_keys, int64_t tie_cap,
                      int64_t *n_ties, float *kernel_ms);
/* The per-candidate solver run on the HOST for n candidates (masks4 = [n][4]: inputs a, b, c and the target row):
   squared-error counts for both roundings.  A test hook for the exact arithmetic; the product never calls it. */
int pbn_fit_eval_host(const uint32_t *masks4, int64_t n, int32_t n_samples, int32_t *k_lo, int32_t *k_hi);

/* Small-transfer helpers for the single-env drop-in classes (one env.step = one launch + one read-back):
   pbn_upload enqueues a host->device copy on `stream`; pbn_fetch_host enqueues n device->host copies into one host
   buffer (concatenated in order) and waits for the stream — the reference hands back host values (NumPy arrays, ints,
   bools: pbn_env.py:150-154), so a synchronisation per step is part of its contract. */
int pbn_upload(void *dst_dev, const void *src_host, int64_t nbytes, void *stream);
int pbn_fetch_host(const void *const *src_dev, const int64_t *nbytes, int32_t n, void *dst_host, void *stream);
/* Read-back of ONE env's step result (env index e of a batch of B): packs {reward int32, inner int32, terminated u8,
   truncated u8, pad u16, state words [W32], obs words [W32]} into `scratch_dev` (>= 12 + 8*W32 bytes) with a 1-block
   kernel, copies it to dst_host in a single transfer and waits for the stream. */
int pbn_fetch_step_host(const int32_t *reward, const uint8_t *terminated, const uint8_t *truncated, const int32_t *inner,
                        const uint32_t *state, const uint32_t *obs_state, int32_t w32, int64_t B, int64_t e,
                        void *scratch_dev, void *dst_host, void *stream);

/* instruction-issue microbenchmarks used by bench.py for the roofline denominator (SURVEY.md §8d):
   kind 0 = dependent-free LOP3/IADD3 chain, kind 1 = Philox4x32-10 blocks, kinds 2..5 = one opcode only (LOP3, SHF, IMAD,
   IADD) to see the issue rate of each class.  Writes elapsed ms and the number of thread-level operations executed. */
int pbn_issue_peak(int32_t kind, int64_t iters, float *ms_out, double *ops_out);

/* Test hook of the SSD kernel's gap draw (utils/eval.py:92-95 flips each node with probability p; the kernels draw the
   geometric gaps between flips instead).  The gap is DEFINED by a fixed single-precision polynomial for log2 (the oracle's
   orc_geom); the fast path takes the hardware lg2.approx when the result lies further than `delta` from an integer.  This
   call runs both on all 2^23 possible inputs for flip probability p and reports the margin in use (1.0 = shortcut off),
   how many inputs disagreed where the shortcut would have been taken (must be 0), and how many inputs fall back. */
int pbn_geom_shortcut_check(double p, float *delta, uint32_t *disagree, uint32_t *fallback);

const char *pbn_last_error(void);
const char *pbn_version(void);

#ifdef __cplusplus
}
#endif
#endif
