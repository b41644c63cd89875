/*
 * acsolver_b200.h -- C ABI of libacsolver_b200.so, the B200 (sm_100a) implementation of
 * AC-Solver's AC-move transition function and of the BFS / greedy searches built on it.
 *
 * The reference (shehper/AC-Solver) has no FFI: its seam is a Python function API on
 * host numpy arrays.  Every entry point below names the reference function it replaces
 * (paths relative to the reference root).  Two flavours exist for the batched ops:
 *   *_host : plain HOST pointers in and out -- what a reference-side binding (ctypes,
 *            see INTEGRATION.md) calls; host<->device copies happen inside the call,
 *            pipelined in chunks over several CUDA streams;
 *   no suffix : DEVICE pointers + a cudaStream_t (as void*) for GPU-resident callers
 *            (PPO rollouts with the policy in torch); asynchronous, nothing is copied.
 *
 * Conventions
 *   - A presentation is 2*mrl int8 letters: relator 0 then relator 1, letters in
 *     {+1,-1,+2,-2} = {x, x^-1, y, y^-1}, zero-padded on the right (envs/utils.py:4-7).
 *     Rows of a batch are contiguous with stride 2*mrl bytes.  1 <= mrl <= 64 for the
 *     packed kernels, <= 127 for the generic byte kernels.
 *   - Every function returns ACS_OK (0) or a negative ACS_ERR_* code; nothing throws
 *     across the ABI.  acs_last_error() returns a thread-local message.
 *   - Per-row `status` bytes report what the reference would have raised for that row:
 *     ACS_ROW_OK, ACS_ROW_ASSERT (AssertionError, envs/utils.py:261-263) or
 *     ACS_ROW_INDEX (IndexError, envs/ac_moves.py:119).  Such rows are left unchanged.
 *   - The caller owns every buffer it passes.  The library owns only what *_create
 *     returns.  No global mutable state.  The *_host calls of one context share its streams and
 *     scratch buffers and are serialised by a mutex inside the context: they are thread-safe but do
 *     not overlap; use one context per thread for concurrency.
 *   - The batched packed kernels require rows that are zero right-padded over the
 *     alphabet {+-1,+-2} (check once with acs_validate_batch); words need not be reduced
 *     and relators may be empty.  The generic kernels accept any int8 letters.
 */
#ifndef ACSOLVER_B200_H
#define ACSOLVER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ACS_OK 0
#define ACS_ERR_INVALID (-1)     /* bad argument                                   */
#define ACS_ERR_CUDA (-2)        /* CUDA runtime error, see acs_last_error()       */
#define ACS_ERR_UNSUPPORTED (-3) /* e.g. mrl out of range for the packed kernels   */
#define ACS_ERR_NOMEM (-4)       /* device or host allocation failed               */
#define ACS_ERR_NO_DEVICE (-5)   /* no CUDA device: there is NO CPU fallback       */

#define ACS_ROW_OK 0
#define ACS_ROW_ASSERT 1
#define ACS_ROW_INDEX 2

/* generic ops (acs_generic_*): which reference function is evaluated */
#define ACS_OP_ACMOVE 0                /* envs/ac_moves.py:159-231 ACMove               */
#define ACS_OP_CONCAT_RAW 1            /* envs/ac_moves.py:4-76   concatenate_relators  */
#define ACS_OP_CONJ_RAW 2              /* envs/ac_moves.py:79-156 conjugate             */
#define ACS_OP_SIMPLIFY_RELATOR 3      /* envs/utils.py:175-240   simplify_relator      */
#define ACS_OP_SIMPLIFY_PRESENTATION 4 /* envs/utils.py:243-280   simplify_presentation */

typedef struct acs_ctx acs_ctx;

int acs_version(void);
const char *acs_last_error(void);
/* number of visible CUDA devices (0 if none / driver missing) */
int acs_device_count(void);

/* A context binds a device and owns the streams / scratch used by the *_host calls. */
int acs_ctx_create(int device, acs_ctx **out);
void acs_ctx_destroy(acs_ctx *ctx);

/* ---- ACMove, batched (envs/ac_moves.py:159-231) --------------------------------- */
/* out may alias in.  lens [n,2] (recomputed lengths), status [n], err (two uint64:
 * number of non-OK rows, smallest such row; must be initialised to {0, ~0}) may be NULL.
 * flags: ACS_FLAG_CYCLICAL = ACMove's `cyclical` argument; ACS_FLAG_NORMALIZED = the caller
 * guarantees every input word is already a normal form for that cyclical flag (freely
 * reduced, and cyclically reduced if cyclical) -- true for any state this library produced
 * with the same flag -- which lets the kernel skip re-validating the untouched relator. */
#define ACS_FLAG_CYCLICAL 1
#define ACS_FLAG_NORMALIZED 2
/* ACS_FLAG_LENS_VALID (only with ACS_FLAG_NORMALIZED and a non-NULL lens array): lens[n,2] holds
 * the current relator lengths ON ENTRY, exactly as ACEnv keeps `self.lengths` beside `self.state`
 * (envs/ac_env.py:84-92); the kernel then reads them instead of recounting the letters and
 * writes the new lengths back.  lens written by a previous call on the same states qualify. */
#define ACS_FLAG_LENS_VALID 4
int acs_moves_batch(const int8_t *d_in, const uint8_t *d_action, int8_t *d_out, uint8_t *d_lens,
                    uint8_t *d_status, uint64_t *d_err, int64_t n, int mrl, int flags, void *stream);
int acs_moves_batch_host(acs_ctx *ctx, const int8_t *h_in, const uint8_t *h_action, int8_t *h_out,
                         uint8_t *h_lens, uint8_t *h_status, int64_t n, int mrl, int flags);

/* ---- ACEnv.step, batched (envs/ac_env.py:95-113) --------------------------------- */
/* n independent environments; state [n,2*mrl] updated in place (cyclical=True as in the
 * reference); reward = horizon*mrl*2 if done else -(len0+len1); step_count += 1;
 * truncated = step_count >= horizon.  d_lens / d_status / d_err may be NULL.
 * flags: ACS_FLAG_NORMALIZED as above (every state after an environment's first step is
 * normalized; pass it unless a reset just planted caller-supplied states). */
int acs_env_step_batch(int8_t *d_state, const uint8_t *d_action, int32_t *d_reward, uint8_t *d_done,
                       uint8_t *d_truncated, int32_t *d_step_count, uint8_t *d_lens, uint8_t *d_status,
                       uint64_t *d_err, int64_t n, int mrl, int horizon, int flags, void *stream);
/* Same step with the environment state RESIDENT on the device (d_state, d_step_count
 * owned by the caller) and host actions in / host observations, rewards and flags out:
 * the vector-env call of agents/training.py:154-156.  h_obs may be NULL (observations
 * stay on the device).  *n_bad receives the number of rows whose move raised. */
int acs_env_step_host(acs_ctx *ctx, int8_t *d_state, int32_t *d_step_count, const uint8_t *h_action,
                      int8_t *h_obs, int32_t *h_reward, uint8_t *h_done, uint8_t *h_truncated,
                      int64_t n, int mrl, int horizon, int flags, int64_t *n_bad);

/* Vector-environment step for GPU-resident rollouts: acs_env_step_batch followed, in the same
 * stream and with no host involvement, by the auto-reset of gymnasium's SyncVectorEnv as the
 * reference uses it (agents/environment.py:60-127): environments with done|truncated copy their
 * observation to d_final_obs and their episode length to d_final_steps (either may be NULL) and
 * return to d_initial_state with zeroed counters.
 * d_action_log [n, log_stride] (may be NULL) receives each action at the pre-step counter, i.e.
 * ACEnv.actions (envs/ac_env.py:96).  Capturable in a CUDA graph (no allocation, no sync). */
int acs_vecenv_step(int8_t *d_state, const int8_t *d_initial_state, const uint8_t *d_action, int32_t *d_reward,
                    uint8_t *d_done, uint8_t *d_truncated, int32_t *d_step_count, uint8_t *d_lens,
                    const uint8_t *d_initial_lens, uint8_t *d_action_log, int log_stride, int8_t *d_final_obs,
                    int32_t *d_final_steps, uint64_t *d_err, int64_t n, int mrl, int horizon, int flags,
                    void *stream);

/* ---- reward wrappers and curriculum of the PPO rollout, on the device ---------------------------- */
/* gymnasium 0.28.1 NormalizeReward per environment (agents/environment.py:45-46) followed by the
 * TransformReward clip (environment.py:48-52).  d_stats: [4][n] doubles (returns, mean, var, count;
 * initialise to 0, 0, 1, 1e-4).  d_out: float rewards as PPO consumes them. */
int acs_reward_transform(const int32_t *d_reward, const uint8_t *d_done, double *d_stats, float *d_out, int64_t n,
                         double gamma, double eps, int normalize, int clip, double lo, double hi, void *stream);
/* One vector-env step with the reference's curriculum reset (agents/training.py:169-224) on the
 * device: finished environments record their result (solved set, shortest action sequence per
 * initial state -- success_record / ACMoves_hist) and continue with another initial state of the
 * pool: the unprocessed ones in order first, then an unsolved one with probability
 * 1 - repeat_solved_prob (or while nothing is solved), else a solved one.  No host involvement;
 * capturable in a CUDA graph.  counters: {next unprocessed state, number solved, draws, episodes}. */
typedef struct {
    int8_t *state;             /* [n, 2*mrl] */
    const int8_t *pool;        /* [n_states, 2*mrl] initial states */
    const uint8_t *pool_lens;  /* [n_states, 2] */
    uint8_t *lens;             /* [n, 2] */
    const uint8_t *action;     /* [n] */
    int32_t *reward;
    uint8_t *done, *truncated;
    int32_t *step_count;
    int32_t *cur_state;        /* [n] pool index of each environment's current episode */
    uint8_t *solved;           /* [n_states rounded up to 4] */
    int32_t *solved_list;      /* [n_states] */
    uint64_t *best;            /* [n_states] (length << 32 | env) of the shortest solving episode, ~0 = none */
    uint8_t *best_actions;     /* [n_states, log_stride] */
    uint8_t *action_log;       /* [n, log_stride] */
    int8_t *final_obs;         /* [n, 2*mrl] or NULL */
    int32_t *final_steps;      /* [n] or NULL */
    int64_t *counters;         /* [4] */
    uint64_t *err;             /* {count, min row} or NULL */
    int64_t n;
    int32_t n_states, mrl, horizon, log_stride, flags;
    float repeat_solved_prob;
    uint64_t seed;
} acs_curriculum_args;
int acs_vecenv_curriculum_step(const acs_curriculum_args *a, void *stream);

/* ---- boundary validation (envs/utils.py:13-54) ------------------------------------ */
/* flags[row]: bit0 is_array_valid_presentation, bit1 letters in {0,+-1,+-2},
 * bit2 zeros only on the right of each half. */
int acs_validate_batch(const int8_t *d_in, uint8_t *d_flags, int64_t n, int mrl, void *stream);
int acs_validate_batch_host(acs_ctx *ctx, const int8_t *h_in, uint8_t *h_flags, int64_t n, int mrl);

/* ---- generic byte-domain ops, any int8 alphabet ----------------------------------- */
/* width = letters per row (2*mrl; the relator width for SIMPLIFY_RELATOR).
 * aux: ACMOVE / SIMPLIFY_PRESENTATION -> int32 [n,2] lengths; *_RAW -> int32 [n] new
 * length of r_i, -1 rejected (row unchanged), -2 IndexError; SIMPLIFY_RELATOR -> [n]. */
int acs_generic_batch(int op, const int8_t *d_in, const uint8_t *d_action, int8_t *d_out, int32_t *d_aux,
                      uint8_t *d_status, int64_t n, int width, int i, int j, int sign, int cyclical,
                      void *stream);
int acs_generic_host(acs_ctx *ctx, int op, const int8_t *h_in, const uint8_t *h_action, int8_t *h_out,
                     int32_t *h_aux, uint8_t *h_status, int64_t n, int width, int i, int j, int sign,
                     int cyclical);

/* ---- searches (search/breadth_first.py:15-97, search/greedy.py:15-121) ------------ */
typedef struct {
    int32_t solved;        /* a child of total length 2 was generated                   */
    int32_t status;        /* ACS_ROW_* of the move that raised in reference order, or 0 */
    int32_t budget_hit;    /* the reference would print "Exiting search as ..."          */
    int32_t path_len;      /* (action,length) pairs written to path                      */
    int64_t n_visited;     /* len(tree_nodes) at return                                  */
    int64_t n_expanded;    /* nodes whose 12 children were generated                     */
    int64_t n_moves;       /* ACMove evaluations the reference would have made           */
    int64_t frontier_left; /* len(to_explore) at return                                  */
    int32_t n_levels;      /* BFS levels / greedy rounds executed on the device          */
    int32_t n_minlen;      /* entries of minlen_log                                      */
    int32_t minlen_log[128]; /* successive "New minimal length found" values (verbose)   */
    double seconds_device; /* CUDA-event time of the search proper                       */
} acs_search_result;

typedef struct acs_bfs acs_bfs;
/* max_nodes: node budget; device capacity is derived from it (16 B/node keys for mrl <= 29,
 * 32 B for mrl <= 61, + 8 B parent link + 16 B of hash table).  ctx may be NULL. */
int acs_bfs_create(acs_ctx *ctx, int device, int mrl, int64_t max_nodes, int cyclical, acs_bfs **out);
/* Runs the whole search on the device.  path: int32 pairs, capacity path_cap pairs. */
int acs_bfs_run(acs_bfs *b, const int8_t *h_presentation, int32_t *h_path, int path_cap,
                acs_search_result *res);
/* visited states in insertion (FIFO) order as int8 rows; returns rows written via *n_out */
int acs_bfs_visited(acs_bfs *b, int8_t *h_out, int64_t cap_rows, int64_t *n_out);
void acs_bfs_destroy(acs_bfs *b);

/* Batched breadth-first search: n_search independent searches of the same mrl and cyclical flag,
 * one budget each, advanced together through the same kernel launches on one GPU (csrc/mbfs.cu).
 * Every search's result, path, counters and visited array equal acs_bfs_run on its row.
 * acs_bfs_batch_bytes: device bytes an engine for these arguments allocates (for planning batches).
 * chunk_parents <= 0: default chunk size.  h_presentations [n_search, 2*mrl]; h_paths
 * [n_search, path_cap, 2] int32 (action, total_length) pairs; results [n_search].  A row the
 * reference raises on has results[s].status != 0.  A path longer than path_cap makes the run
 * return ACS_ERR_INVALID with every other result filled (results[s].path_len holds the needed
 * length); acs_bfs_batch_paths then fetches the paths of that run into a larger buffer without
 * searching again.  path_cap may be 0 (with h_paths NULL) when no search can solve.
 * chunk_parents caps the parents expanded per chunk after the first, which expands every root. */
typedef struct acs_bfs_batch acs_bfs_batch;
int acs_bfs_batch_bytes(int n_search, int mrl, const int64_t *max_nodes, int64_t chunk_parents, int64_t *bytes_out);
int acs_bfs_batch_create(int device, int n_search, int mrl, const int64_t *max_nodes /* [n_search] */,
                         int cyclical, int64_t chunk_parents, acs_bfs_batch **out);
int acs_bfs_batch_run(acs_bfs_batch *b, const int8_t *h_presentations, int32_t *h_paths, int path_cap,
                      acs_search_result *results /* [n_search] */);
int acs_bfs_batch_paths(acs_bfs_batch *b, int32_t *h_paths, int path_cap);
/* visited states of search `search` of the last run, insertion (FIFO) order, int8 rows */
int acs_bfs_batch_visited(acs_bfs_batch *b, int search, int8_t *h_out, int64_t cap_rows, int64_t *n_out);
void acs_bfs_batch_destroy(acs_bfs_batch *b);

/* Goal sets (csrc/goalset.cu): device-resident sets of states keyed by the state alone, for the goal
 * test of the batched search.  An entry holds a state, a parent link and a root index; when a state
 * occurs more than once the smallest entry index represents it.
 * acs_goalset_from_rows: rows [n, 2*mrl] int8; each row must be a state a search can generate (both
 * relators non-empty, right-padded, freely reduced, and cyclically reduced when cyclical), else
 * ACS_ERR_INVALID before any device work.  Entry i is row i, its own root.
 * acs_goalset_from_bfs_batch: every committed node of every search of b's last run, in (search, FIFO
 * id) order; roots are search indices.  b's memory goes to the set or is freed: b can only be destroyed.
 * acs_goalset_path: (-1, L_root), (action, total_length), ... from the entry's root to the entry; a
 * path longer than path_cap is ACS_ERR_INVALID with *path_len the needed length. */
typedef struct acs_goalset acs_goalset;
int acs_goalset_from_rows(int device, int mrl, int cyclical, const int8_t *h_rows, int64_t n, acs_goalset **out);
int acs_goalset_from_bfs_batch(acs_bfs_batch *b, acs_goalset **out);
int acs_goalset_size(const acs_goalset *g, int64_t *n_entries, int64_t *n_states, int64_t *bytes);
int acs_goalset_path(const acs_goalset *g, int64_t entry, int *root, int32_t *h_path, int path_cap, int *path_len);
void acs_goalset_destroy(acs_goalset *g);
/* Options of the next runs of b.  g (may be NULL; must outlive those runs): a search stops at the first
 * generated child in g, tested after the length-2 test and before the visited test, exactly as a solve
 * stops it (solved = 1; the path ends with (action, total length of the goal state)); a root in g is a
 * hit at depth 0.  stop_at_trivial = 0 turns the length-2 rule off, so searches run until a goal,
 * their budget or exhaustion.  g's mrl, cyclical flag and device must be b's.  With g NULL and
 * stop_at_trivial = 1 the engine runs exactly as without this call.
 * acs_bfs_batch_goal_hits: per search of the last run, the goal entry it stopped at, or -1. */
int acs_bfs_batch_set_goals(acs_bfs_batch *b, const acs_goalset *g, int stop_at_trivial);
int acs_bfs_batch_goal_hits(acs_bfs_batch *b, int64_t *h_entry /* [n_search] */);

/* Presentation symmetries (csrc/ac_sym.cuh): the group G of order 16 generated by the signed permutations
 * of the generators and the swap of the relators acts on the AC' graph by automorphisms.  Element
 * g = 8r + 4s + 2a + b: swap x <-> y (s), then invert x (a), then invert y (b), then swap the relators (r).
 * acs_canonical_form: h_out [n, 2*mrl] the canonical form of each row (the smallest of its 16 images in the
 * order of ac_sym.cuh) and h_elem [n] the smallest g with h_out = g.row.  Rows must be right-padded with
 * letters in {+-1, +-2}, else ACS_ERR_INVALID.
 * acs_bfs_batch_set_symmetric: symmetric != 0 makes the next runs of b orbit searches: breadth-first
 * search over canonical states, the root stored canonical, a child new when its canonical form is unseen.
 * Distances to the trivial presentations are exact; paths are moves of the input row, in the format of
 * acs_bfs_batch_run; visited arrays hold the canonical states in insertion order.  Goal sets must be
 * symmetric (ACS_ERR_INVALID otherwise); acs_goalset_from_bfs_batch of such an engine makes a symmetric set. */
int acs_canonical_form(int device, int mrl, const int8_t *h_rows, int64_t n, int8_t *h_out, uint8_t *h_elem);
int acs_bfs_batch_set_symmetric(acs_bfs_batch *b, int symmetric);

/* Batched greedy search (search/greedy.py:15-121): n_search independent presentations of the
 * same mrl, one warp each, one launch.  h_presentations [n_search, 2*mrl]; h_paths
 * [n_search, path_cap, 2] int32 (action, total_length) pairs; results [n_search].  On failure
 * the path is the reference's `path + [(11, len)]` of the last popped node.  max_nodes < 2^24.
 * Device memory: n_search * (max_nodes+16) * (16|32 + 8 + 4 + 8) B + the tables. */
typedef struct acs_greedy acs_greedy;
int acs_greedy_create(int device, int n_search, int mrl, int64_t max_nodes, int cyclical, int path_cap,
                      acs_greedy **out);
int acs_greedy_run(acs_greedy *g, const int8_t *h_presentations, int32_t *h_paths, acs_search_result *results);
int acs_greedy_visited(acs_greedy *g, int search, int8_t *h_out, int64_t cap_rows, int64_t *n_out);
void acs_greedy_destroy(acs_greedy *g);
/* Goal set of the next runs of g (may be NULL; must outlive those runs): a search stops at the first
 * generated child in gs, tested after the length-2 test and before the visited test, exactly as a solve
 * stops it (solved = 1; the path ends with (action, total length of the goal state); the solve wins on
 * the same child); a root in gs is a hit at depth 0 with the path [(-1, L0)].  gs's mrl, cyclical flag
 * and device must be g's, else ACS_ERR_INVALID.  NULL restores the plain engine exactly.
 * acs_greedy_goal_hits: per search of the last run, the goal entry it stopped at, or -1. */
int acs_greedy_set_goals(acs_greedy *g, const acs_goalset *gs);
int acs_greedy_goal_hits(acs_greedy *g, int64_t *h_entry /* [n_search] */);
/* Symmetric goal sets hold canonical forms and answer "is any image of this state in the set?"; exact
 * and orbit searches (bfs_batch, greedy) can stop at them.  An orbit search needs a symmetric set.
 * acs_goalset_from_rows_symmetric: acs_goalset_from_rows storing each row's canonical form.
 * acs_goalset_from_bfs_batch of an orbit-search engine makes a symmetric set.
 * acs_goalset_path_frame: acs_goalset_path (moves of the root's row, also for symmetric sets) and *frame =
 * the element H with (end state of that path) = H.(the entry's stored state); 0 for exact sets.
 * acs_bfs_batch_goal_hit_elements / acs_greedy_goal_hit_elements: per search of the last run, the element u
 * with u.(end state of the returned path) = the state of the entry it stopped at (0 for an exact set), or
 * -1 when it did not stop at a goal. */
int acs_goalset_from_rows_symmetric(int device, int mrl, int cyclical, const int8_t *h_rows, int64_t n,
                                    acs_goalset **out);
int acs_goalset_is_symmetric(const acs_goalset *g, int *symmetric);
int acs_goalset_path_frame(const acs_goalset *g, int64_t entry, int *root, int32_t *h_path, int path_cap,
                           int *path_len, int *frame);
int acs_bfs_batch_goal_hit_elements(acs_bfs_batch *b, int32_t *h_elem /* [n_search] */);
int acs_greedy_goal_hit_elements(acs_greedy *g, int32_t *h_elem /* [n_search] */);

/* Batched beam search (csrc/beam.cu): n_search independent searches of the same mrl and cyclical flag, one
 * node budget each, advanced together level by level through the same kernel launches on one GPU.  A search
 * keeps a visited list V = [root] and a beam = [root].  At each level the candidates c = 12*i + m (move m of
 * beam node i) are walked in increasing c: the first that raises (results[s].status), has total length 2 or
 * is in the goal set ends the search and nothing of that level is kept.  Otherwise the children whose state
 * is not in V, each at its smallest c, are ordered by (total length, c) and the first
 * min(beam_width, max_nodes[s] - |V|) become the next beam, appended to V in that order.  A search stops
 * after a level whose next beam is empty, that brought |V| to max_nodes[s] (budget_hit), or the
 * max_depth-th level.  Counters and paths are those of acs_bfs_batch_run: n_moves counts candidates up to
 * and including the one that ended the search, n_expanded the beam nodes expanded, frontier_left the beam
 * nodes left, n_levels the levels kept, minlen_log every new minimal total length in (level, c) order.
 * Orbit (symmetric) search is not offered by this engine; symmetric goal sets are.
 * acs_beam_bytes: device bytes an engine for these arguments allocates (for planning batches).
 * acs_beam_create: 1 <= beam_width <= 2^24, every max_nodes[s] >= 1, max_depth >= 1 or 0 for no limit,
 * 1 <= mrl <= 61; anything else is ACS_ERR_INVALID / ACS_ERR_UNSUPPORTED before any device work.
 * acs_beam_run: h_presentations [n_search, 2*mrl] (a row that is not right-padded or has an empty relator
 * gets status ACS_ROW_ASSERT and is not searched); h_paths [n_search, path_cap, 2] int32 (action,
 * total_length) pairs; results [n_search].  A path longer than path_cap makes the run return
 * ACS_ERR_INVALID with every other result filled (results[s].path_len holds the needed length);
 * acs_beam_paths then fetches the paths of that run into a larger buffer without searching again.
 * acs_beam_visited: V of search `search` of the last run, in order, as int8 rows.
 * acs_beam_set_goals: goal set of the next runs (may be NULL; must outlive those runs), exact or symmetric;
 * its mrl, cyclical flag and device must be b's, else ACS_ERR_INVALID.  A root in the set is a hit at depth
 * 0 with the path [(-1, L0)].  acs_beam_goal_hits / acs_beam_goal_hit_elements: as for acs_bfs_batch. */
typedef struct acs_beam acs_beam;
int acs_beam_bytes(int n_search, int mrl, int64_t beam_width, const int64_t *max_nodes, int max_depth,
                   int64_t *bytes_out);
int acs_beam_create(int device, int n_search, int mrl, int64_t beam_width, const int64_t *max_nodes /* [n_search] */,
                    int max_depth, int cyclical, acs_beam **out);
int acs_beam_set_goals(acs_beam *b, const acs_goalset *g);
int acs_beam_run(acs_beam *b, const int8_t *h_presentations, int32_t *h_paths, int path_cap,
                 acs_search_result *results /* [n_search] */);
int acs_beam_paths(acs_beam *b, int32_t *h_paths, int path_cap);
int acs_beam_visited(acs_beam *b, int search, int8_t *h_out, int64_t cap_rows, int64_t *n_out);
int acs_beam_goal_hits(acs_beam *b, int64_t *h_entry /* [n_search] */);
int acs_beam_goal_hit_elements(acs_beam *b, int32_t *h_elem /* [n_search] */);
void acs_beam_destroy(acs_beam *b);

/* ---- hash-partitioned multi-GPU BFS: per-rank device kernels --------------------------------- */
/* The host loop (ac_solver_b200/search/sharded.py, one process per GPU, torch.distributed/NCCL
 * for the all-to-all and the small all-reduces) drives these on caller-allocated device buffers.
 * Same sequential contract as acs_bfs_run for every world size.  All pointers are DEVICE
 * pointers; every call is asynchronous on `stream`. */
typedef struct {
    uint64_t *keys;      /* [cap][2W] owned nodes, increasing global id                     */
    int64_t *parent;     /* [cap] (parent global id << 4 | action), root -1                 */
    int64_t *gid;        /* [cap] global id of each owned node                              */
    uint64_t *table;     /* [tmask+1] visited table of this rank (zero-initialised)         */
    uint64_t tmask;
    int64_t n_local;     /* owned nodes committed so far                                    */
    int64_t l0, l1;      /* local index range of this chunk's parents                       */
    int64_t head;        /* global id of the chunk's first parent                           */
    int64_t nparents;    /* parents in the chunk, all ranks together                        */
    int64_t n_nodes;     /* global node count at chunk start                                */
    int64_t budget;
    int64_t limit;       /* commit: chunk-local candidate ids below this are appended       */
    int32_t mrl, cyclical, trusted, world, rank, min_len, W, pad_;
    unsigned long long *dest_count;  /* [world] records per destination (phase 0)           */
    unsigned long long *dest_cursor; /* [world] running write offsets (phase 1)             */
    uint64_t *send_keys; /* [n_send][2W]                                                    */
    uint32_t *send_c;    /* [n_send] chunk-local candidate id                               */
    unsigned long long *ctrl; /* [130] min-reduced: solving id, error id<<2|status, first_len[128] */
    const uint64_t *recv_keys;
    const uint32_t *recv_c;
    int64_t n_recv;
    uint32_t *rec_slot;  /* [n_recv] scratch                                                */
    uint32_t *bitmap_local, *bitmap_global; /* [ceil(12*nparents/32)] winner bits           */
    uint32_t *prefix_local, *prefix_global; /* [words+1] exclusive popcount prefixes        */
    unsigned long long *cut; /* [1] min chunk-local parent at which the budget is reached   */
} acs_sbfs_args;

int acs_sbfs_pack_root(const int8_t *h_presentation, int mrl, uint64_t *key_out4, uint64_t *hash_out,
                       int *total_len, int *valid);
int acs_sbfs_owner(uint64_t hash, int world);
int acs_sbfs_expand(const acs_sbfs_args *a, int phase, void *stream);
int acs_sbfs_insert_mark(const acs_sbfs_args *a, void *stream);
/* d_prefix: nwords+1 prefixes (the last is the total) followed by ceil(nwords/2048)+1 words of scratch */
int acs_sbfs_scan(const uint32_t *d_bitmap, uint32_t *d_prefix, int64_t nwords, void *stream);
int acs_sbfs_cut(const acs_sbfs_args *a, void *stream);
int acs_sbfs_rank_at(const acs_sbfs_args *a, uint64_t *d_out2, void *stream);
int acs_sbfs_commit(const acs_sbfs_args *a, void *stream);
int acs_sbfs_lower_bound(const int64_t *d_gid, int64_t n, int64_t value, int64_t *d_out, void *stream);
int acs_sbfs_lookup(const acs_sbfs_args *a, int64_t gid, int64_t *d_out4, void *stream);
int acs_sbfs_unpack(const uint64_t *d_keys, int8_t *d_out, int64_t n, int mrl, void *stream);

/* ---- hash-partitioned BFS, native driver (csrc/pbfs.cu) ------------------------------------------
 * Replaces search/breadth_first.py:15-97 for one GPU (world 1) and for a hash-partitioned search over
 * the GPUs of one node (one process per GPU).  The chunk loop runs on the device streams with no host
 * synchronisation; newly generated states go straight into the owner rank's inbox by peer stores over
 * NVLink (the exchange arena is shared through cudaIpc handles), synchronised by release/acquire
 * epoch flags in peer memory.  Same sequential contract and bit-identical results for every world
 * size.  Usage, on every rank: create -> export -> (all-gather the 64-byte handles with any host
 * channel, e.g. torch.distributed) -> connect -> run (same arguments on every rank) -> lookup /
 * visited -> destroy.  For tests all ranks may live in one process: create world shards, then
 * acs_pbfs_connect_local. */
typedef struct acs_pbfs acs_pbfs;
/* chunk_parents <= 0 picks the default (world * 4 Mi parents per chunk). */
int acs_pbfs_create(int device, int rank, int world, int mrl, int64_t max_nodes, int cyclical,
                    int64_t chunk_parents, acs_pbfs **out);
int acs_pbfs_export(acs_pbfs *b, void *handle64);
int acs_pbfs_connect(acs_pbfs *b, const void *handles /* world x 64 bytes, rank order */);
int acs_pbfs_connect_local(acs_pbfs **shards, int n);
/* shards: this process's one rank, or all ranks of a single-process world.  h_path (int32 pairs,
 * capacity path_cap) is filled only when all ranks are local; otherwise use acs_pbfs_lookup. */
int acs_pbfs_run(acs_pbfs **shards, int n_local, const int8_t *h_presentation, int32_t *h_path, int path_cap,
                 acs_search_result *res);
/* out4 = {found on this rank, parent global id (-1 root), action (-1 root), total length} */
int acs_pbfs_lookup(acs_pbfs *b, int64_t gid, int64_t *out4);
/* this rank's visited states and their global ids (= FIFO positions of the reference's tree_nodes) */
int acs_pbfs_visited(acs_pbfs *b, int64_t *h_gid, int8_t *h_rows, int64_t cap_rows, int64_t *n_out);
/* {n_local, chunks, records sent, records received, chunk_cap, record-log capacity per source, arena bytes, table slots} */
int acs_pbfs_stats(acs_pbfs *b, int64_t *out8);
int acs_pbfs_set_timeout(acs_pbfs *b, double seconds);
void acs_pbfs_destroy(acs_pbfs *b);

/* ---- barcode_analysis state model (SURVEY 8f-3): unordered relator pairs, full free reduction ----
 * Replaces the BFS of barcode_analysis/5_steps_neibourhoods/neibourhoods.cpp:18-54 (size of the
 * radius-r ball: radius >= 0, size_cap 0) and of barcode_analysis/simplex_data_generation/<prime|classic>_moves/
 * ac_bfs.cpp:36-91 (all states of total length <= size_cap, radius < 0, with the 0/1-simplices and
 * their filtration values).  h_letters: relator 1 then relator 2 as letters +-1, +-2 (no padding).
 * classic != 0: the 14 classic moves, else the 12 prime moves (AC_UTILS_no_hash.cpp:153-211).
 * Nodes are numbered in the reference's FIFO discovery order.  h_sizes / h_levels (capacity cap_nodes),
 * h_edges ((cn, cc, filtration) uint32 triples, capacity cap_edges) may be NULL. */
int acs_ball_explore(int device, const int8_t *h_letters, int len1, int len2, int radius, int size_cap, int classic,
                     int64_t max_nodes, int64_t *n_nodes_out, uint16_t *h_sizes, uint8_t *h_levels, int64_t cap_nodes,
                     uint32_t *h_edges, int64_t cap_edges, int64_t *n_edges_out);
/* neibourhoods.cpp read_do_and_write (:58-103) for a whole input file at once: the radius-`radius` ball sizes of
 * n_roots presentations in ONE exploration (every node carries the index of its start presentation and the
 * visited set is keyed by (root, state), so the balls are independent but share every kernel launch).
 * Root r = letters [h_off[2r], h_off[2r+1]) and [h_off[2r+1], h_off[2r+2]) of h_letters; h_counts[n_roots].
 * max_nodes bounds the SUM of the ball sizes (ACS_ERR_NOMEM if exceeded: split the batch). */
int acs_ball_sizes(int device, const int8_t *h_letters, const int64_t *h_off, int n_roots, int radius, int classic,
                   int64_t max_nodes, int64_t *h_counts);

/* ---- PPO update path (SURVEY 8f-4): the non-GEMM part, fused --------------------------------------
 * acs_gae replaces the generalised-advantage-estimation loop of ac_solver/agents/training.py:230-250:
 * rewards / values / dones are [T, N] fp32 (time major, as the rollout stores them), next_value / next_done [N];
 * advantages and returns [T, N] out.  Same fp32 operation order as the reference's elementwise torch ops
 * (bit-identical results).  All pointers are device pointers; the work is enqueued on `stream`. */
int acs_gae(const float *d_rewards, const float *d_values, const float *d_dones, const float *d_next_value,
            const float *d_next_done, float *d_advantages, float *d_returns, int T, int64_t N, double gamma,
            double gae_lambda, void *stream);
/* acs_ppo_loss replaces the loss arithmetic of training.py:262-318 for one minibatch of B samples and ALSO
 * returns its gradient: d_logits [B, n_actions] actor outputs, d_newvalue [B] critic outputs, d_action [B] int64,
 * d_old_logprob / d_adv (raw advantages; normalised here when norm_adv) / d_returns / d_old_value [B].
 * d_out8 = {loss, pg_loss, v_loss, entropy, approx_kl, clipfrac, 0, 0}; d_dlogits [B, n_actions] and d_dvalue [B] =
 * d loss / d logits, d loss / d newvalue (feed them to the backward pass of the two networks).  loss_clip: the
 * clipped surrogate, else the KL-penalised one with the device scalar *d_beta.  d_workspace: at least
 * acs_ppo_loss_workspace_bytes() bytes of device memory. */
int acs_ppo_loss_workspace_bytes(void);
int acs_ppo_loss(const float *d_logits, const float *d_newvalue, const int64_t *d_action, const float *d_old_logprob,
                 const float *d_adv, const float *d_returns, const float *d_old_value, const float *d_beta,
                 float *d_dlogits, float *d_dvalue, float *d_out8, void *d_workspace, int64_t B, int n_actions,
                 int norm_adv, int loss_clip, int clip_vloss, double clip_coef, double ent_coef, double vf_coef,
                 void *stream);

/* Rollout bookkeeping of the PPO loop (agents/training.py:139-228 of the reference), two launches per vector step.
 * d_ctr2 = device int64[2] {time index t, draw counter}; the caller resets t per update and adds 1 to both after every
 * step (torch: ctr.add_(1)), so one captured CUDA graph serves every step.
 * acs_rollout_sample_record: action ~ Categorical(logits) (Gumbel-max, counter-based generator keyed by seed, draw
 *   counter, row), log-probability of the action, and obs[t] = state, dones[t] = next_done, values[t], actions[t],
 *   logprobs[t]; d_action_u8 [N] feeds acs_vecenv_step.  1 <= n_actions <= 16.
 * acs_rollout_finish (after the environment step and acs_reward_transform): rewards[t] = reward, next_done = done,
 *   episodic return / length accumulation, and for finished episodes (done | truncated) an entry in the ring of the
 *   last `ring` episodes (the reference's deque(maxlen=100)); d_counters[0] counts finished episodes. */
int acs_rollout_sample_record(const int8_t *d_state, const float *d_next_done, const float *d_logits, const float *d_value,
                              const int64_t *d_ctr2, int8_t *d_obs_buf, float *d_dones_buf, float *d_values_buf,
                              float *d_logprobs_buf, int64_t *d_actions_buf, uint8_t *d_action_u8, int64_t N, int64_t T,
                              int width, int n_actions, uint64_t seed, void *stream);
int acs_rollout_finish(const float *d_reward, const uint8_t *d_done, const uint8_t *d_truncated, const int64_t *d_ctr2,
                       float *d_rewards_buf, float *d_next_done, float *d_ep_return, float *d_ep_length, float *d_ring_ret,
                       float *d_ring_len, uint64_t *d_counters, int64_t N, int64_t T, int ring, void *stream);

#ifdef __cplusplus
}
#endif
#endif
