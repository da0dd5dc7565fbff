/*
 * hironaka_b200.h — C-ABI of the B200-native batched Hironaka game engine.
 *
 * This is the drop-in boundary for the reference's env-step path.  The reference
 * (honglu2875/hironaka) has one C-ABI precedent,
 *     extern "C" void getNewtonPolytope_approx(long* points, int batchNum, int m, int n, long* newPoints)
 *     (hironaka/cpp/cppUtil.cpp:58-63, bound with ctypes in hironaka/src/_np_ops.py:6-15),
 * and this header keeps its conventions (caller-owned contiguous row-major [B, N, d]
 * buffers, plain pointers and sizes, ctypes-loadable) and extends them with an `int`
 * status return, a CUDA stream and a mode bitfield, so that one library serves the three
 * de-facto seams of the reference (SURVEY.md section 8b):
 *   (1) TensorPoints / hironaka.src._torch_ops   (hironaka/core/tensor_points.py:11-126,
 *                                                 hironaka/src/_torch_ops.py:8-146)
 *   (2) the functional JAX step API              (hironaka/jax/util.py:22-214,
 *                                                 hironaka/src/_jax_ops.py:15-123)
 *   (3) the per-op signatures op(points, ..., inplace, padding_value).
 *
 * Device entry points (hk_*) take RAW DEVICE POINTERS into caller-owned contiguous
 * buffers and a cudaStream_t (passed as void*); they never allocate, never synchronise
 * and keep no global state, so they are re-entrant and CUDA-graph capturable.
 * Host entry points (hk_session_*) own device buffers for one shard of games and take
 * HOST pointers; they are what a ctypes/numpy caller (the style of _np_ops.py) binds.
 *
 * No torch types appear here.  All functions return HK_OK (0), a negative HK_ERR_* code
 * for argument errors, or a positive cudaError_t.
 */
#ifndef HIRONAKA_B200_H
#define HIRONAKA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HK_VERSION 106 /* major*100 + minor */

/* ---- status codes ---------------------------------------------------------------- */
#define HK_OK 0
#define HK_ERR_BAD_ARG (-1)     /* null pointer, non-positive size, bad flag combination   */
#define HK_ERR_UNSUPPORTED (-2) /* shape outside HK_MAX_* or op not defined for the dtype   */
#define HK_ERR_ALIGN (-3)       /* state pointer not 4-byte aligned                         */

/* ---- limits ------------------------------------------------------------------------ */
#define HK_MAX_DIM 10          /* reference caps dimension at _MAX_DIM-1 = 10
                                  (hironaka/jax/host_action_preprocess.py:27,62)            */
#define HK_MAX_POINTS 1024     /* max_num_points per game                                   */
#define HK_MAX_GAME_WORDS 4096 /* N*d 32-bit words per game (16 KiB of shared memory)       */

/* ---- element type of the point tensor ---------------------------------------------- */
#define HK_DTYPE_I32 0 /* int32 state, padding is the integer -1 (the engine's native form) */
#define HK_DTYPE_F32 1 /* float32 state, the reference's storage (TensorPoints default)     */

/* ---- ops; a step executes the selected ones in THIS order ----------------------------
 * shift -> reposition -> newton -> rescale is get_take_actions (hironaka/jax/util.py:117-123);
 * shift -> newton -> rescale is FusedGame.agent_move (hironaka/trainer/fused_game.py:150-162). */
#define HK_OP_SHIFT (1u << 0)      /* x_a <- sum_{j in S} x_j       (_torch_ops.py:46-110, _jax_ops.py:76-90)   */
#define HK_OP_REPOSITION (1u << 1) /* per coord subtract min over live rows (_torch_ops.py:113-133, _jax_ops.py:114-123) */
#define HK_OP_NEWTON (1u << 2)     /* dedupe + dominance filter     (_fn.py:192-213, _torch_ops.py:8-39, _jax_ops.py:32-73) */
#define HK_OP_RESCALE (1u << 3)    /* divide live entries by the game max; F32 state only (_torch_ops.py:136-146, _jax_ops.py:93-111) */
#define HK_OP_DEDUPE (1u << 4)     /* remove_repeated alone: later copies of identical rows become padding (_fn.py:192-213,
                                      _jax_ops.py:32-40); runs after reposition, before newton (which subsumes it) */

/* ---- semantics flags ---------------------------------------------------------------- */
#define HK_F_NOOP_INVALID (1u << 0)   /* torch: axis not in S  => state unchanged (_torch_ops.py:90-91). Unset = JAX: applied anyway */
#define HK_F_FREEZE_ENDED (1u << 1)   /* torch ignore_ended_games: <2 live points => no shift (_torch_ops.py:92-93) */
#define HK_F_ACT_DISCRETE (1u << 2)   /* host_action[] holds discrete ids 0..2^d-d-2 (HostActionEncoder, _fn.py:241-325;
                                         decode_table, host_action_preprocess.py:8-24). Unset = coordinate bitmask, bit k <=> coordinate k */
#define HK_F_ROLE_AGENT (1u << 3)     /* reward = -(done & !prev_done) (util.py:142-144); unset = host role (+) */
#define HK_F_OBS_RESCALE (1u << 4)    /* observation features are rescaled (scale_observation, util.py:183) */
#define HK_F_OBS_SORT_COORD0 (1u << 5)/* rows sorted by coordinate 0, descending, stable (TensorPoints.get_features, tensor_points.py:72-74) */
#define HK_F_OBS_SORT_LEX (1u << 6)   /* rows sorted descending lexicographically, LAST coordinate primary, stable (util.py:195) */
#define HK_F_ACT_U8 (1u << 7)         /* host_action[] / axis[] / obs_coord[] are uint8 arrays instead of int32 (ids < 256, i.e.
                                         discrete ids up to d = 8 or bitmasks up to d = 8): 2 instead of 8 action bytes per game-step */

/* Fixed players evaluated inside the kernel (zero host round-trips in validation rollouts).  With a
 * host flag set host_action may be NULL, with an agent flag set axis may be NULL. */
#define HK_F_HOST_ALL_COORD (1u << 8)  /* host picks every coordinate (all_coord_host_fn, hironaka/jax/players.py:42-52;
                                          AllCoordHostModule, trainer/player_modules/modules.py:68-79) */
#define HK_F_HOST_ZEILLINGER (1u << 9) /* Zeillinger's host (zeillinger_fn, players.py:55-105) on the state before the step */
#define HK_F_AGENT_FIRST (1u << 10)    /* agent picks the first chosen coordinate (choose_first_agent_fn, players.py:156-183) */
#define HK_F_AGENT_LAST (1u << 11)     /* agent picks the last chosen coordinate (choose_last_agent_fn, players.py:186-212) */

#define HK_F_OBS_SORT_LEX_FIRST (1u << 12) /* rows sorted descending lexicographically, coordinate 0 primary: the order of
                                              ListPoints (Python sorted(points, reverse=True), hironaka/src/_list_ops.py:25) */
#define HK_F_STORE_ALL (1u << 13) /* in-place calls (out == in) write back only the games that changed; set this to
                                     rewrite every game (the results are identical; for measurements) */
#define HK_F_ACT_PACKED (1u << 14) /* host_action[] is a uint8 array holding BOTH players' actions, one byte per game(-step):
                                      the host action (coordinate bitmask or discrete id, < 32) in the low 5 bits, the agent's
                                      axis (< 8) in the high 3 bits; axis[] is ignored.  Halves the bytes of an action stream
                                      again (1 instead of 2 per game-step).  Needs d <= 5; not with the fixed players. */

#define HK_F_RESCALE_EPS (1u << 15) /* rescale (the op and the rescaled observation) leaves a game whose maximum is <= 1e-8
                                       unchanged: calculate_rescale of the JAX flavour (hironaka/src/_jax_ops.py:93-98).
                                       Unset = rescale_torch: only a maximum of exactly 0 is replaced by 1 (_torch_ops.py:139) */

#define HK_F_ACT_NIBBLE (1u << 16) /* host_action[] is a uint8 array holding the actions of TWO games per byte (game 2i in the low
                                      nibble, 2i+1 in the high one); a nibble is the discrete host id (< 4) | axis (< 4) << 2.
                                      Half a byte of action stream per game-step; d <= 3 with HK_F_ACT_DISCRETE only; axis[] ignored. */

/* Random players drawn inside the kernel (hk_rollout_seeded / hk_step_seeded), so that a random-play rollout needs no
 * [T,B] action streams in memory.  Philox4x32-10 with counter (game index low, high, step, 0) and key (seed low,
 * high): every (game, step) owns its random words whatever the launch geometry, the number of GPUs, or how the
 * rollout is cut into calls.  Not jax.random's bits — the same distribution (RNG contract in DESIGN.md). */
#define HK_F_HOST_RANDOM (1u << 17)  /* host: a discrete action id uniform over the 2^d - d - 1 coordinate sets,
                                        floor(word0 * n / 2^32) (random_host_fn, hironaka/jax/players.py:28-39) */
#define HK_F_AGENT_RANDOM (1u << 18) /* agent: an axis uniform over ALL d axes, floor(word1 * d / 2^32)
                                        (random_agent_fn, players.py:142-153) */

/* ---- introspection ------------------------------------------------------------------ */
int hk_version(void);
const char* hk_error_string(int code);
/* 1 if (N,d) runs on the register-resident thread-per-game kernel, 0 if on the generic
 * warp-per-game kernel, <0 if unsupported. */
int hk_kernel_class(int N, int d);
/* Test hook: when on != 0, shapes of the thread-per-game class are routed through the generic
 * warp-per-game kernel too (so both kernel families are parity-tested on every shape). */
int hk_debug_force_generic(int on);
/* Tuning hook: programmatic dependent launch (cudaLaunchAttributeProgrammaticStreamSerialization) of
 * the thread-per-game kernel, off by default (measured: no gain); results do not depend on it. */
int hk_debug_set_pdl(int on);
/* Test / tuning hook: hk_session_rollout_ex replays a repeated call (same arguments) as a CUDA graph; 0 turns that off. */
int hk_debug_set_session_graphs(int on);

/* ---- the fused step ------------------------------------------------------------------
 * One launch = one game-step for B independent games:
 *   prev_done -> [shift] -> [reposition] -> [dedupe] -> [newton] -> [rescale] -> done / reward / num_points
 *   -> [observation features]
 * Replaces shift_torch + get_newton_polytope_torch + rescale_torch + ended_batch_in_tensor +
 * FusedGame._default_reward (fused_game.py:150-182) and take_actions + get_dones + reward_fn +
 * feature_fn (util.py:34-35,82-149,172-214).
 *
 *   state_in / state_out  [B,N,d] dtype; may be the same pointer (in place = the reference's
 *                         inplace=True) or disjoint (inplace=False).  Dead rows are negative in
 *                         coordinate 0 and are rewritten with padding_value.  In place, only the games
 *                         the step changed are written back (same result, fewer bytes; HK_F_STORE_ALL
 *                         rewrites every game).
 *   host_action [B] int32 coordinate bitmask or discrete id (HK_F_ACT_DISCRETE); required with HK_OP_SHIFT
 *   axis        [B] int32 agent's coordinate; required with HK_OP_SHIFT
 *   done        [B] uint8  (#live rows <= 1 after the step), nullable        (util.py:34-35)
 *   reward      [B] float  +-(done & !prev_done), nullable                   (util.py:136-144)
 *   num_points  [B] int32  live rows after the step, nullable                (tensor_points.py:65-70)
 *   obs         [B, N*d (+d if obs_coord)] float, nullable: features of the new state
 *   obs_coord   [B] int32  coordinate set appended to obs as d floats 0/1 (make_agent_obs, util.py:22-31), nullable
 *   exceed_flag [1] int32  set to 1 if any live entry >= value_threshold (TensorPoints.exceed_threshold,
 *                         tensor_points.py:57-63), nullable; never cleared by the library
 */
int hk_step(const void* state_in, void* state_out, const int32_t* host_action, const int32_t* axis,
            uint8_t* done, float* reward, int32_t* num_points, float* obs, const int32_t* obs_coord,
            int32_t* exceed_flag, int64_t B, int32_t N, int32_t d, int32_t dtype, uint32_t ops,
            uint32_t flags, float padding_value, float value_threshold, void* stream);

/* ---- the in-place step with a census ------------------------------------------------------
 * The same step as hk_step with state_out == state_in, plus `census`: one byte per game that the library
 * writes after every step and reads before the next one, so that a rollout's work follows the games still in
 * play instead of the batch size.  A game at rest (no live row, or a lone point at the origin: the fixed point
 * every ended game of a reposition rollout reaches, hironaka/src/_jax_ops.py:76-90,114-123; or any ended game
 * under HK_F_FREEZE_ENDED without reposition / rescale, _torch_ops.py:92-93) is NOT READ: its done = 1,
 * reward = 0 and num_points come from its census byte.  Games in play are ordered by their live-row count
 * before they are processed (thread-per-game shapes), so that the 32 games a warp steps together are alike.
 * Results are identical to hk_step's, bit for bit.
 *   census [hk_census_bytes(B, N, d)] uint8, in/out.  Byte g describes game g: 0 = unknown (the game is read and
 *          counted): zero-fill the first B bytes before the first call and ZERO THE BYTE OF ANY GAME YOU REWRITE
 *          between calls.  Other values belong to the library (1..127: live rows of a game in play;
 *          0x80 | rows | 2 * at_rest: ended game, dead rows normalised).  For large padded shapes with N <= 64 and
 *          2 <= d <= 5 the buffer continues, 8-byte aligned after the B bytes, with one 64-bit live mask per game
 *          (bit i <=> row i alive, meaningful while the byte is non-zero): games down to at most 8 live rows are
 *          then stepped thread-per-game on their live rows alone (hk_rows_kernel), the others warp-per-game.
 *   done_bits [ceil(B/32)] uint32, nullable: the done flags as a bit mask (bit g % 32 of word g / 32), every word
 *          written — one eighth of the bytes of `done` for a host that reads the flags back every step.
 *   done_count [1] int32, nullable: incremented by the number of finished games after the step.
 * Not available with a fused observation, the in-kernel players, out-of-place states or ops == 0
 * (HK_ERR_UNSUPPORTED). */
int64_t hk_census_bytes(int64_t B, int32_t N, int32_t d);
int hk_step_census(void* state, const int32_t* host_action, const int32_t* axis, uint8_t* done, uint32_t* done_bits,
                   float* reward, int32_t* num_points, uint8_t* census, int32_t* done_count, int32_t* exceed_flag, int64_t B, int32_t N,
                   int32_t d, int32_t dtype, uint32_t ops, uint32_t flags, float padding_value, float value_threshold,
                   void* stream);

/* hk_step_census with the fused observation of the new state (obs [B, N*d (+d if obs_coord)] float, as hk_step's):
 * thread-per-game shapes and the sorted observation modes only (HK_ERR_UNSUPPORTED otherwise).  A game at rest has a
 * constant observation — its lone point, at the origin, sorts first; the rest is padding (get_feature_fn,
 * hironaka/jax/util.py:186-196; TensorPoints.get_features tensor_points.py:72-74) — so it is written from the
 * census byte and only the games in play run the feature code. */
int hk_step_census_obs(void* state, const int32_t* host_action, const int32_t* axis, uint8_t* done, uint32_t* done_bits,
                       float* reward, int32_t* num_points, float* obs, const int32_t* obs_coord, uint8_t* census,
                       int32_t* done_count, int32_t* exceed_flag, int64_t B, int32_t N, int32_t d, int32_t dtype,
                       uint32_t ops, uint32_t flags, float padding_value, float value_threshold, void* stream);

/* ---- per-op entry points (the reference's hironaka.src op surface) ---------------------
 * Each is one launch of the same kernel family with a single op selected. */
int hk_shift(const void* state_in, void* state_out, const int32_t* host_action, const int32_t* axis,
             int64_t B, int32_t N, int32_t d, int32_t dtype, uint32_t flags, float padding_value,
             void* stream);
int hk_reposition(const void* state_in, void* state_out, int64_t B, int32_t N, int32_t d,
                  int32_t dtype, float padding_value, void* stream);
int hk_newton_polytope(const void* state_in, void* state_out, int64_t B, int32_t N, int32_t d,
                       int32_t dtype, float padding_value, void* stream);
int hk_rescale(const void* state_in, void* state_out, int64_t B, int32_t N, int32_t d, int32_t dtype,
               float padding_value, void* stream); /* F32 only */
int hk_features(const void* state_in, float* obs, const int32_t* obs_coord, int64_t B, int32_t N,
                int32_t d, int32_t dtype, uint32_t flags, float padding_value, void* stream);
int hk_dones(const void* state_in, uint8_t* done, int32_t* num_points, int64_t B, int32_t N, int32_t d,
             int32_t dtype, void* stream);

/* The coordinate set a FIXED HOST would choose on each game, as a bitmask (bit k <=> coordinate k),
 * without moving anything: flags = HK_F_HOST_ALL_COORD (AllCoordHost, hironaka/host.py:44-47;
 * all_coord_host_fn, hironaka/jax/players.py:42-52) or HK_F_HOST_ZEILLINGER (Zeillinger,
 * hironaka/host.py:50-92; zeillinger_fn, players.py:55-105: pairs of live rows in slot order, so a
 * state kept in ListPoints order reproduces host.py).  A game without live rows gets 0.  This is what
 * a host-side environment returns to the agent as `coords` (HironakaHostEnv.step,
 * hironaka/gym_env/hironaka_host_env.py:62-66). */
int hk_host_policy(const void* state_in, int32_t* coord_mask, int64_t B, int32_t N, int32_t d, int32_t dtype,
                   uint32_t flags, float padding_value, void* stream);

/* ---- game-tree search of a fixed host ------------------------------------------------------
 * How long can an adversarial agent make the game last against a fixed host?  The batched, level-by-level form of
 * search_depth (hironaka/util/search.py): every agent reply is explored, every limit is explicit.
 * For each root b of roots [B,N,d] (int32 state, taken as given: filter it first if you want filtered roots):
 *   - a node is a state; it is ENDED when it has <= 1 live row (hk_step's done rule);
 *   - a node at level k that has not ended is expanded: S = hk_host_policy(node) with flags (exactly one of
 *     HK_F_HOST_ZEILLINGER, HK_F_HOST_ALL_COORD), and each axis a in S, in increasing order, gives one child at level
 *     k + 1: hk_step of the node with coordinate bitmask S and axis a, ops (HK_OP_SHIFT | HK_OP_NEWTON, optionally
 *     HK_OP_REPOSITION) and the JAX flags (0); padding -1;
 *   - equal states are not merged and cycles are not detected: a state reached twice is counted twice.
 * Outputs per root:
 *   depth  [B] int32: height of the explored tree, 0 for an ended root; for a cut root a lower bound (its deepest level)
 *   nodes  [B] int64: states in the explored tree, the root and the ended leaves included, cut levels not
 *   status [B] int8 HK_SEARCH_*: RESOLVED; MAX_DEPTH (nodes at level max_depth have not ended); MAX_NODES (adding the
 *          next level would take the root past max_nodes; the level is not added); CAPACITY (the next level of all
 *          roots does not fit in `capacity` nodes: the roots are dropped from the highest index down until it fits);
 *          INT32_BOUND (a node to expand has a live entry >= floor(2^30 / d): its children would not be exact).
 *          At one level the checks apply in the order INT32_BOUND, MAX_NODES, CAPACITY.  A cut root has no later levels.
 * The results do not depend on the launch geometry or on the other roots of the batch, except through CAPACITY.
 * workspace: hk_search_workspace_bytes(B, N, d, capacity) bytes of device memory owned by the caller: two frontiers of
 * `capacity` nodes (N*d*4 bytes each) and O(B + capacity) words of bookkeeping; the call allocates nothing.
 * The call is SYNCHRONOUS: after every level it reads two counters back to the host (to size the next level's launches
 * and to stop when no node is left), so it is not graph-capturable.
 * Errors: float32 state HK_ERR_UNSUPPORTED; other flags, ops without HK_OP_SHIFT | HK_OP_NEWTON or with
 * HK_OP_RESCALE / HK_OP_DEDUPE, max_depth < 1, max_nodes < 1, capacity < 1: HK_ERR_BAD_ARG. */
#define HK_SEARCH_RESOLVED 0
#define HK_SEARCH_MAX_DEPTH 1
#define HK_SEARCH_MAX_NODES 2
#define HK_SEARCH_CAPACITY 3
#define HK_SEARCH_INT32_BOUND 4
int64_t hk_search_workspace_bytes(int64_t B, int32_t N, int32_t d, int64_t capacity);
int hk_search_depth(const void* roots, int32_t* depth, int64_t* nodes, int8_t* status, int64_t B, int32_t N, int32_t d,
                    int32_t dtype, uint32_t ops, uint32_t flags, int32_t max_depth, int64_t max_nodes, int64_t capacity,
                    void* workspace, void* stream);

/* ---- game value: minimax over the host's choices -----------------------------------------------
 * How few moves does the best host need to end the game, whatever the agent replies?  For each root b of roots [B,N,d]
 * (int32 state, taken as given, 2 <= d <= 6), level by level with the limits of hk_search_depth:
 *   - a node with <= 1 live row has ENDED; its value is 0;
 *   - an open node is expanded into one child per (S, axis): S over every coordinate set with |S| >= 2 in increasing
 *     bitmask order, the axis over the members of S in increasing order; the child is hk_step of the node with bitmask S
 *     and that axis, ops as for hk_search_depth, the JAX flags (0), padding -1.  The children of one S form a GROUP.
 *     d*2^(d-1) - d children: 2, 9, 28, 75 or 186;
 *   - after level L is built (round L): every ended node of level L is solved; a group is won when all its children
 *     are solved; a node is solved when its first group is won, up to the root in the same round.  A node of level l
 *     solved in round L has value L - l (the rounds go in level order, so this first value is the minimum);
 *   - a node is expanded only if it is open, not solved and has no solved ancestor;
 *   - limits: max_depth, max_nodes per root, `capacity` nodes per level of the whole batch, the int32 bound
 *     (floor(2^30 / d)), and `history`: the nodes of every level of the whole batch, roots included, which the search
 *     keeps to walk up from solved nodes.  At one level the cuts apply in the order INT32_BOUND, MAX_NODES, CAPACITY,
 *     HISTORY; the last two drop roots from the highest index down.
 * Outputs per root:
 *   value     [B] int32: the game value when status is RESOLVED; otherwise the last level whose round was done for the
 *             root, and the value is strictly larger
 *   best_mask [B] int32: the smallest S among the root's groups won in the round that solved it, 0 for a root that has
 *             ended, -1 when not RESOLVED
 *   nodes     [B] int64: states in the explored tree, the root included (as hk_search_depth)
 *   status    [B] int8 HK_SEARCH_*: RESOLVED, MAX_DEPTH, MAX_NODES, CAPACITY, INT32_BOUND as for hk_search_depth, or
 *             HISTORY (the next level would take the batch's history past `history` nodes; it is not added).
 * The results do not depend on the launch geometry or on the other roots of the batch, except through CAPACITY and
 * HISTORY.  workspace: hk_search_value_workspace_bytes(B, N, d, capacity, history) bytes of device memory owned by
 * the caller: two frontiers of `capacity` nodes (N*d*4 bytes each), 14 bytes per history node and O(B + capacity)
 * words of bookkeeping; it returns 0 for arguments hk_search_value refuses.  SYNCHRONOUS, as hk_search_depth.
 * Errors: float32 state, d outside 2..6: HK_ERR_UNSUPPORTED; ops as for hk_search_depth, max_depth < 1,
 * max_nodes < 1, capacity < 1, history < max(B, 1) or history > 2^31 - 1: HK_ERR_BAD_ARG. */
#define HK_SEARCH_HISTORY 5
int64_t hk_search_value_workspace_bytes(int64_t B, int32_t N, int32_t d, int64_t capacity, int64_t history);
int hk_search_value(const void* roots, int32_t* value, int32_t* best_mask, int64_t* nodes, int8_t* status, int64_t B,
                    int32_t N, int32_t d, int32_t dtype, uint32_t ops, int32_t max_depth, int64_t max_nodes,
                    int64_t capacity, int64_t history, void* workspace, void* stream);

/* ---- lines of play from the searches ---------------------------------------------------------
 * A line is a sequence of moves (host coordinate bitmask S, agent axis), each the JAX step of the searches (shift,
 * reposition if HK_OP_REPOSITION, Newton polytope, flags 0, padding -1).  line_mask and line_axis are [B, max_depth]
 * int32; entries past a root's line length hold mask 0 and axis -1.
 *
 * hk_search_depth_line: hk_search_depth with the WORST LINE against the fixed host.  Its length is depth[b]; every mask
 * is hk_host_policy (same flags) of the state it is played on; the axes are the lexicographically smallest sequence
 * among the lines that reach level depth[b] of the explored tree.  For a RESOLVED root it is the smallest of the
 * longest games and ends at an ended state; for a cut root it is the smallest line to its deepest explored level,
 * which need not have ended.  The search keeps a history of every state of the batch (the parent's entry, int32, and
 * the set, 16 bits, and the axis, one byte: 7 bytes per state), so `history` is one more limit: the states of all levels of the
 * batch, roots included.  The cuts apply in the order INT32_BOUND, MAX_NODES, CAPACITY, HISTORY, the last two dropping
 * roots from the highest index down, as in hk_search_value; a root cut by the history gets HK_SEARCH_HISTORY.  With a
 * history large enough for the whole search, depth, nodes and status equal hk_search_depth's.
 * workspace: hk_search_depth_line_workspace_bytes(B, N, d, capacity, history) bytes (hk_search_depth's, 7 bytes per
 * history state and 12 per root); it returns 0 for arguments hk_search_depth_line refuses.
 * Errors: those of hk_search_depth; history < max(B, 1) or > 2^31 - 1, null line outputs: HK_ERR_BAD_ARG.
 *
 * hk_search_value_line: hk_search_value with an OPTIMAL LINE for each RESOLVED root of value v > 0, of length v.  From a
 * state of value u > 0 the host plays the smallest S whose children all have value <= u - 1 (at the root, best_mask),
 * and the agent the smallest axis of S whose child has value exactly u - 1; the line ends at an ended state.  Roots
 * that ended on entry and roots whose status is not RESOLVED get an empty line.  Every state of the line is solved in
 * the root's round, so these are read from the search's own history: no extra memory, the workspace of
 * hk_search_value.  value, best_mask, nodes and status equal hk_search_value's.
 * Errors: those of hk_search_value; null line outputs: HK_ERR_BAD_ARG.  Both calls are SYNCHRONOUS. */
int64_t hk_search_depth_line_workspace_bytes(int64_t B, int32_t N, int32_t d, int64_t capacity, int64_t history);
int hk_search_depth_line(const void* roots, int32_t* depth, int64_t* nodes, int8_t* status, int32_t* line_mask,
                         int32_t* line_axis, int64_t B, int32_t N, int32_t d, int32_t dtype, uint32_t ops,
                         uint32_t flags, int32_t max_depth, int64_t max_nodes, int64_t capacity, int64_t history,
                         void* workspace, void* stream);
int hk_search_value_line(const void* roots, int32_t* value, int32_t* best_mask, int64_t* nodes, int8_t* status,
                         int32_t* line_mask, int32_t* line_axis, int64_t B, int32_t N, int32_t d, int32_t dtype,
                         uint32_t ops, int32_t max_depth, int64_t max_nodes, int64_t capacity, int64_t history,
                         void* workspace, void* stream);

/* ---- value labels from the game-value search ---------------------------------------------------
 * hk_search_value_labels: hk_search_value, then every state of its history that was SOLVED with value >= 1, whatever
 * its root's status.  A state of level l solved in round R has the exact value R - l (no state below a solved state is
 * solved in a later round), and its OPTIMAL host moves are exactly its groups whose children are all solved (a group
 * with an unsolved child has a value above R - l).  value, best_mask, nodes and status equal hk_search_value's.
 * Outputs:
 *   *label_count   HOST int64: the number of labels, also when it exceeds max_labels
 *   the first min(count, max_labels) labels in history order (level non-decreasing, within a level root
 *   non-decreasing); entries past them are not written:
 *   label_root     [max_labels] int32: the root the state lies under
 *   label_level    [max_labels] int32: its level, the moves from the root
 *   label_value    [max_labels] int32: its value
 *   label_optimal  [max_labels] uint64: bit g is set when the host move with action id g (the sets with |S| >= 2 in
 *                  increasing bitmask order: 57 at d = 6) is optimal
 *   label_mask, label_axis [max_labels, max_depth] int32: the moves from the root to the state; mask 0 and axis -1
 *                  past the label's level, as the lines.
 * Equal states reached by different paths are separate labels.  max_labels == 0 counts only; the label pointers may
 * then be null.  workspace: hk_search_value_labels_workspace_bytes(B, N, d, capacity, history) bytes: hk_search_value's
 * and 12 bytes per 256 history states; it returns 0 for arguments hk_search_value refuses.  SYNCHRONOUS.
 * Errors: those of hk_search_value; max_labels < 0, a null label_count, a null label output with max_labels > 0:
 * HK_ERR_BAD_ARG. */
int64_t hk_search_value_labels_workspace_bytes(int64_t B, int32_t N, int32_t d, int64_t capacity, int64_t history);
int hk_search_value_labels(const void* roots, int32_t* value, int32_t* best_mask, int64_t* nodes, int8_t* status,
                           int64_t max_labels, int64_t* label_count, int32_t* label_root, int32_t* label_level,
                           int32_t* label_value, uint64_t* label_optimal, int32_t* label_mask, int32_t* label_axis,
                           int64_t B, int32_t N, int32_t d, int32_t dtype, uint32_t ops, int32_t max_depth,
                           int64_t max_nodes, int64_t capacity, int64_t history, void* workspace, void* stream);

/* ---- multi-step rollout ------------------------------------------------------------------
 * T consecutive steps with the state held on chip between steps: one read and one write of
 * the state per T steps.  Action streams are [T,B].  Outputs per step are optional:
 *   done_t [T,B] uint8, reward_t [T,B] float; done_count [T] int32 is incremented atomically
 *   (number of finished games after each step, the quantity compute_rho reads every step,
 *   hironaka/jax/jax_trainer.py:533-534); length [B] int32 = first step index (1-based) after
 *   which the game was done, 0 if done at entry, T+1 if never. All nullable. */
int hk_rollout(const void* state_in, void* state_out, const int32_t* host_action_t, const int32_t* axis_t,
               uint8_t* done_t, float* reward_t, int32_t* done_count, int32_t* length, int64_t B,
               int32_t N, int32_t d, int32_t T, int32_t dtype, uint32_t ops, uint32_t flags,
               float padding_value, void* stream);

/* hk_rollout / hk_step with the in-kernel random players: flags carry HK_F_HOST_RANDOM and / or HK_F_AGENT_RANDOM, the
 * action array of a random player may be NULL, `seed` is the Philox key and step t of the call draws the words
 * of step step_offset + t (so per-step calls and one fused call play the same game).  hk_random_actions writes
 * the same streams out, [T,B] int32 each (either pointer nullable), for callers that want to see them. */
int hk_rollout_seeded(const void* state_in, void* state_out, const int32_t* host_action_t, const int32_t* axis_t,
                      uint8_t* done_t, float* reward_t, int32_t* done_count, int32_t* length, int64_t B, int32_t N,
                      int32_t d, int32_t T, int32_t dtype, uint32_t ops, uint32_t flags, float padding_value,
                      uint64_t seed, int32_t step_offset, void* stream);
int hk_random_actions(int32_t* host_action_t, int32_t* axis_t, int64_t B, int32_t d, int32_t T, uint64_t seed,
                      int32_t step_offset, void* stream);

/* ---- recorded rollout -----------------------------------------------------------------------
 * hk_rollout / hk_rollout_seeded that also writes the trajectory, for training data: what the players saw before
 * every step and what they played.  seed / step_offset are read only with HK_F_HOST_RANDOM / HK_F_AGENT_RANDOM.
 * Every output is nullable; with obs_t, host_mask_t and axis_played_t all null the call is hk_rollout(_seeded).
 *   obs_t         [T,B,OW] float: row t = the features of the state BEFORE step t, as hk_features computes them with the
 *                 same flags (sort mode, HK_F_OBS_RESCALE, HK_F_RESCALE_EPS), bit for bit; row 0 = hk_features(state_in),
 *                 and hk_features(state_out) is the observation after the last step.  OW = N*d, or N*d + d with
 *                 agent_obs != 0: the host's coordinate set of step t appended as d floats 0/1 (make_agent_obs,
 *                 hironaka/jax/util.py:22-31).  agent_obs without obs_t is HK_ERR_BAD_ARG.
 *   host_mask_t   [T,B] int32: the coordinate bitmask step t's shift used (discrete ids decoded, packed and nibble
 *                 streams unpacked, the choices of fixed and random players as made; a fixed host on a game without
 *                 live rows records 0, as hk_host_policy does)
 *   axis_played_t [T,B] int32: the axis step t's shift used
 * Both are 0 without HK_OP_SHIFT.  Fed back to hk_rollout as bitmask / int32 streams (HK_F_ACT_DISCRETE cleared, the
 * player flags removed) they replay the rollout bit for bit.  The other outputs are hk_rollout's. */
int hk_rollout_record(const void* state_in, void* state_out, const int32_t* host_action_t, const int32_t* axis_t,
                      float* obs_t, int32_t agent_obs, int32_t* host_mask_t, int32_t* axis_played_t, uint8_t* done_t,
                      float* reward_t, int32_t* done_count, int32_t* length, int64_t B, int32_t N, int32_t d, int32_t T,
                      int32_t dtype, uint32_t ops, uint32_t flags, float padding_value, uint64_t seed, int32_t step_offset,
                      void* stream);

/* ---- rollout with a value threshold ---------------------------------------------------------
 * hk_rollout_record that also follows every game against a value threshold (TensorPoints.value_threshold and
 * exceed_threshold, the gym environments' stop_at_threshold), inside the one launch.  A game has crossed when a live
 * entry is >= value_threshold (non-strict, compared as float32 like hk_overflow with strict = 0; for integer states a
 * strict threshold v is v + 1).
 *   over_step [B] int32, nullable, laid out like length: 0 if the input state has already crossed, t + 1 for the first
 *             step t after which it has, T + 1 if it never does.
 *   stop_at_threshold != 0: a game that has crossed (on entry or after step t) is not stepped again in this call.  Its
 *             state stays as it was after the crossing step (on entry: as read, dead rows padded), done_t repeats its
 *             done flag and done_count counts it by that flag, reward_t is 0.0 (-0.0 with HK_F_ROLE_AGENT), length
 *             stays T + 1 unless it was already done; obs_t rows are the features of the frozen state, host_mask_t 0
 *             and axis_played_t -1 for the steps it sits out.  The in-kernel random players stay keyed by
 *             (game, step): every other game plays as without the stop.  Since a stopped game enters the next call
 *             over the threshold, it stays stopped across calls.  Replayed as streams through this call with the same
 *             threshold and stop flag, the recorded actions give the rollout back bit for bit.
 *   Without the stop, games play on after they cross; over_step says from which step a game's int32 results can no
 *   longer be trusted (int32 results are exact below 2^30).
 * value_threshold: NaN is HK_ERR_BAD_ARG; with int32 state a finite threshold must be <= floor(2^30 / d)
 * (HK_ERR_BAD_ARG otherwise): live inputs below it give shift sums below 2^30, so with the stop every state the kernel
 * holds or writes is exact (1e8, the reference's default, passes for every d <= 10).  +inf never crosses; with +inf
 * and over_step null the call is hk_rollout_record (same kernels, same results). */
int hk_rollout_threshold(const void* state_in, void* state_out, const int32_t* host_action_t, const int32_t* axis_t,
                         float* obs_t, int32_t agent_obs, int32_t* host_mask_t, int32_t* axis_played_t, uint8_t* done_t,
                         float* reward_t, int32_t* done_count, int32_t* length, int64_t B, int32_t N, int32_t d, int32_t T,
                         int32_t dtype, uint32_t ops, uint32_t flags, float padding_value, uint64_t seed, int32_t step_offset,
                         float value_threshold, int32_t stop_at_threshold, int32_t* over_step, void* stream);

/* ---- experience writer (SURVEY 8f rank 2) --------------------------------------------------------
 * Appends the rows with skip[b] == 0, IN BATCH ORDER, to circular replay buffers at
 * (pos + rank) mod capacity and advances the DEVICE-resident pos / full — the no-sync form of
 * FusedGame.step's `[~done]` filtering (hironaka/trainer/fused_game.py:82-99) followed by
 * ReplayBuffer.add (hironaka/trainer/replay_buffer.py:63-127).  Any source/buffer pair may be NULL.
 *   obs/next_obs [B, obs_width] float, coords/next_coords [B, coord_width] float (agent dict obs),
 *   action [B] int32, reward [B] float, done [B] uint8; buffers have `capacity` rows of the same widths;
 *   pos [1] int64 and full [1] int32 live on the device; appended [1] int32 (nullable) gets the count;
 *   scratch: hk_experience_scratch_words(B) int32 words of device memory owned by the caller. */
int64_t hk_experience_scratch_words(int64_t B);
int hk_experience_append(const uint8_t* skip, const float* obs, const float* next_obs, int32_t obs_width,
                         const float* coords, const float* next_coords, int32_t coord_width,
                         const int32_t* action, const float* reward, const uint8_t* done, float* buf_obs,
                         float* buf_next_obs, float* buf_coords, float* buf_next_coords, int32_t* buf_action,
                         float* buf_reward, uint8_t* buf_done, int64_t capacity, int64_t* pos, int32_t* full,
                         int32_t* appended, int32_t* scratch, int64_t B, void* stream);

/* ---- rollout value targets (SURVEY 8f rank 3) --------------------------------------------------
 * calculate_value_using_reward_fn (hironaka/jax/util.py:261-284) behind JAXTrainer.rollout_postprocess
 * (hironaka/jax/jax_trainer.py:558-592).  Give either obs [B,T,W] (points per step are recovered as
 * #(entries >= 0) / dimension - offset, :584) or num_points [B,T].  value [B,T] out; num_points_out
 * nullable.  est_sign: +1 host / -1 agent (get_value_est_fn util.py:152-169); reward_sign: +1 host /
 * -1 agent reward function; unified != 0 flips the discount sign every step (unified MC tree). */
int hk_value_targets(const float* obs, const int32_t* num_points, int32_t* num_points_out, float* value, int64_t B,
                     int32_t T, int32_t W, int32_t dimension, int32_t offset, float discount, int32_t est_sign,
                     int32_t reward_sign, int32_t unified, void* stream);

/* ---- per-game overflow flags ------------------------------------------------------------------
 * overflow [B] uint8: 1 iff some entry of the game reaches value_threshold (>=, or > when strict != 0): the per-game
 * form of TensorPoints.exceed_threshold (hironaka/core/tensor_points.py:57-63) and the rule the gym environments
 * stop on (ListPoints.exceed_threshold, strict; hironaka/gym_env/hironaka_host_env.py:57-58). */
int hk_overflow(const void* state, uint8_t* overflow, int64_t B, int32_t N, int32_t d, int32_t dtype, float value_threshold,
                int32_t strict, void* stream);

/* ---- host action packing ----------------------------------------------------------------------
 * Multi-binary coordinate vectors coords[B, d] (what HostActionEncoder.decode_tensor and
 * get_batch_decode return, hironaka/src/_fn.py:313-325, hironaka/jax/host_action_preprocess.py:58-65)
 * -> int32 bitmasks mask[B] for hk_step.  src_dtype: 0 int32, 1 float32, 2 int64, 3 uint8/bool. */
int hk_pack_coords(const void* coords, int32_t src_dtype, int32_t* mask, int64_t B, int32_t d, void* stream);

/* ---- host-buffer sessions (numpy / ctypes callers; the _np_ops.py calling style) -------
 * A session owns the device state of one shard of B games on one GPU plus staging buffers
 * and a stream.  All pointers below are HOST pointers (pinned or pageable). */
typedef struct hk_session hk_session;

int hk_session_create(hk_session** out, int device, int64_t B, int32_t N, int32_t d, int32_t dtype,
                      float padding_value);
int hk_session_destroy(hk_session* s);
int hk_session_set_state(hk_session* s, const void* state_host);   /* H2D of [B,N,d]            */
int hk_session_get_state(hk_session* s, void* state_host);         /* D2H of [B,N,d], blocking   */
/* One step: H2D(host_action, axis) -> hk_step -> D2H(done, reward, done_count), blocking.
 * done_host / reward_host / done_count_host are nullable; done_count_host receives the
 * number of finished games after the step (a single int32). */
int hk_session_step(hk_session* s, const int32_t* host_action_host, const int32_t* axis_host,
                    uint8_t* done_host, float* reward_host, int32_t* done_count_host, uint32_t ops,
                    uint32_t flags);
/* T steps driven from host action streams [T,B] (int32, or uint8 with HK_F_ACT_U8; pinned memory
 * recommended): step t+1's actions are copied on a second stream while step t runs; after every
 * step the number of finished games is copied to done_count_host[t] (the per-step read of
 * compute_rho, hironaka/jax/jax_trainer.py:533-534).  One synchronisation at the end. */
int hk_session_rollout(hk_session* s, const void* host_action_host, const void* axis_host, int32_t T,
                       int32_t* done_count_host, uint32_t ops, uint32_t flags);
/* The same with the per-game results of every step: done_host [T,B] uint8 (pinned recommended; nullable) receives
 * each step's done flags, read back on a third stream while the next steps run.  From the second call with the
 * same arguments on, the whole schedule (uploads, steps, read-backs) is one CUDA-graph launch.  The session keeps a census
 * of its resident state (hk_step_census), so the steps of a long rollout cost what the games still in play cost. */
int hk_session_rollout_ex(hk_session* s, const void* host_action_host, const void* axis_host, int32_t T,
                          int32_t* done_count_host, uint8_t* done_host, uint32_t ops, uint32_t flags);
/* The same with the done flags of every step as bit masks: done_bits_host [T, ceil(B/32)] uint32 (pinned
 * recommended): 1 bit instead of 1 byte per game-step comes back over PCIe. */
int hk_session_rollout_bits(hk_session* s, const void* host_action_host, const void* axis_host, int32_t T,
                            int32_t* done_count_host, uint32_t* done_bits_host, uint32_t ops, uint32_t flags);
void* hk_session_state_ptr(hk_session* s); /* device pointer of the resident state (zero-copy interop) */
void* hk_session_stream(hk_session* s);

#ifdef __cplusplus
}
#endif
#endif /* HIRONAKA_B200_H */
