/* hexb.h - C ABI of the B200-native batched Hex simulator (libhexb.so).
 *
 * This is the drop-in boundary for the hot path of MBPrdctns/hex_gym_env. The reference has no FFI: its
 * boundary is the Python class API (HexGame / HexEnv / SelfPlayEnv), consumed by stable-baselines3 through
 * gymnasium. Each entry point below names the reference call(s) it replaces (file:line relative to the
 * reference root); the Python classes in hex_gym_env_b200/ bind these symbols with ctypes and keep the
 * reference's names, arguments and return conventions (see INTEGRATION.md).
 *
 * Conventions
 *   - Plain C, no C++/torch types. Every pointer is a DEVICE pointer unless the name ends in _host.
 *   - obs / term_obs buffers are void*: int8 or float32 elements as hexb_config.obs_dtype says.
 *   - All calls are asynchronous on `stream` (a cudaStream_t passed as void*), except the *_host call and
 *     hexb_create/hexb_destroy. No hidden synchronisation, no host reads of device data.
 *   - Return value: 0 = HEXB_OK, negative = error (hexb_strerror). Illegal GAME moves are data (ret 3 /
 *     done), never errors. Nothing throws across this boundary.
 *   - The caller owns every buffer, including the packed state (hexb_state_bytes tells its size); the
 *     handle only remembers pointers. One handle per device, not re-entrant.
 *   - G games = one shard. Game i of the shard is global game game_offset + i; the random stream of a
 *     game depends only on (seed, global index), so results do not depend on how games are sharded.
 */
#ifndef HEXB_H
#define HEXB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HEXB_OK 0
#define HEXB_ERR_ARG (-1)     /* bad argument / unsupported configuration */
#define HEXB_ERR_CUDA (-2)    /* a CUDA call failed; hexb_last_cuda_error() has the code */
#define HEXB_ERR_STATE (-3)   /* state buffer too small or misaligned */
#define HEXB_ERR_NOGPU (-4)   /* no usable CUDA device */

#define HEXB_VARIANT_A 0 /* minihex/HexGame.py: board 0/1/2 in true coordinates, opponent inside step() */
#define HEXB_VARIANT_B 1 /* minihex/HexSingleGame.py + SelfplayWrapper.py: board -1/+1/0 in the mover's view */

#define HEXB_AGENT_BLACK 0
#define HEXB_AGENT_WHITE 1
#define HEXB_AGENT_RANDOM 2 /* agent_player_num=None: random.randint(0,1) once per game (SelfplayWrapper.py:72-73) */

#define HEXB_OBS_I8 0  /* observations as int8 (what the kernels compute in) */
#define HEXB_OBS_F32 1 /* observations as float32: the reference's board is a float array (HexSingleGame.py:175, HexGame.py:174)
                          and stable-baselines3 feeds its policies float32 */

#define HEXB_MIN_BOARD 3
#define HEXB_MAX_BOARD 19

typedef struct hexb_env hexb_env;

typedef struct hexb_config {
    int32_t board_size;     /* N, 3..19 */
    int32_t variant;        /* HEXB_VARIANT_A | HEXB_VARIANT_B */
    int64_t num_games;      /* G, games in this shard */
    int64_t game_offset;    /* global index of game 0 of this shard */
    uint64_t seed;          /* key of the per-game Philox4x32-10 streams */
    int32_t agent_mode;     /* variant B: HEXB_AGENT_*; variant A: must be HEXB_AGENT_BLACK (player_color=WHITE is
                               corrupt in the reference, HexGame.py:245-248, and is rejected) */
    int32_t opponent_first; /* variant A: ctor current_player_num=WHITE, the opponent opens (HexGame.py:224-230) */
    int32_t auto_reset;     /* 1: finished games restart inside step (DummyVecEnv semantics) */
    int32_t eval_state;     /* variant B: SelfPlayEnv.set_eval(True): setup_opponents draws nothing (SelfplayWrapper.py:92-96) */
    int32_t raw;            /* 1: bare HexGame batch for hexb_ply (no opponent, no draws) */
    int32_t device;         /* CUDA device ordinal */
    int32_t manual_opponent;/* 1: the opponent is the caller's policy (OpponentPolicy, SelfplayWrapper.py:26-35): use
                               hexb_half_step instead of hexb_step; resets leave the opening move to the caller */
    int32_t pool_size;      /* opponent pool size for the index drawn in setup_opponents (SelfplayWrapper.py:97-103); 0 = none */
    int32_t obs_dtype;      /* HEXB_OBS_I8 | HEXB_OBS_F32: element type of every obs / term_obs buffer handed to hexb_reset,
                               hexb_step, hexb_rollout, hexb_half_step, hexb_encode and hexb_step_host (observation_space of
                               HexEnv: Box(..., (N,N)), HexGame.py:189, HexSingleGame.py:192; the values are the same integers) */
} hexb_config;

/* Library / ABI version (major << 16 | minor). */
int32_t hexb_version(void);
const char *hexb_strerror(int32_t code);
int32_t hexb_last_cuda_error(void);

/* Bytes of packed device state for `cfg` (0 on a bad config). Layout (chunk-major): per chunk of 32 games the label bytes
 * u8[32][N*N] followed by the record words u32[R][32] (occupancy bitboard, counters, flags, draw index); then striped
 * int64[128][8] statistics. */
size_t hexb_state_bytes(const hexb_config *cfg);

/* Create a handle over caller-allocated, 256-byte-aligned device memory and zero it on `stream`.
 * Replaces HexEnv.__init__ (HexGame.py:152-197, HexSingleGame.py:163-196) and SelfPlayEnv.__init__
 * (SelfplayWrapper.py:39-67). Games are not playable until hexb_reset. */
int32_t hexb_create(const hexb_config *cfg, void *state, size_t state_bytes, void *stream, hexb_env **out);
int32_t hexb_destroy(hexb_env *env);
/* The configuration the handle was created with (the attribute reads .board_size etc. of the reference's env objects); bindings
 * use it to validate the sizes of the buffers they are handed. */
int32_t hexb_get_config(const hexb_env *env, hexb_config *out);

/* reset(): HexGame.__init__ on an empty board (HexGame.py:21-68, HexSingleGame.py:26-71), HexEnv.reset
 * (HexGame.py:206-242, HexSingleGame.py:208-231), SelfPlayEnv.reset + setup_opponents + opening continue_game
 * (SelfplayWrapper.py:69-104). reset_mask u8[G] (null = all games); open_u f64[G] (null = per-game stream)
 * replaces the opponent's opening draw. Emits obs i8[G,N,N] and mask u8[G,N*N] (either may be null). */
int32_t hexb_reset(hexb_env *env, const uint8_t *reset_mask, const double *open_u, void *obs, uint8_t *mask, void *stream);

/* step(): one env step for every game = agent ply + random-opponent reply, fused with the win check, reward,
 * done, auto-reset, observation and legal-action mask.
 *   variant B: SelfPlayEnv.step (SelfplayWrapper.py:174-199) -> HexEnv.step (HexSingleGame.py:233-263) ->
 *              fast_move / flood_fill (:88-153), continue_game + BaseRandomPolicy.choose_action (:146-172, :17-22),
 *              legal_actions (:205-206), invert_board (:265-271)
 *   variant A: HexEnv.step (HexGame.py:244-295), opponent_move (:332-349), random_policy (minihex/__init__.py:8-12),
 *              fast_move / flood_fill (:85-142), get_action_mask (:203-204)
 * actions i32[G] in the agent's view (null: the agent is the random policy too and draws from the game's stream);
 * opp_u f64[G,2] (null: stream) = [reply draw, opening draw after an auto-reset];
 * outputs (each may be null): obs i8[G,N,N], mask u8[G,N*N], reward f32[G], done u8[G],
 * term_obs i8[G,N,N] (written only for games that finished in this call: the observation step() returned before
 * the auto-reset, i.e. SB3's info["terminal_observation"]), actions_out i32[G] (the agent action played). */
int32_t hexb_step(hexb_env *env, const int32_t *actions, const double *opp_u, void *obs, uint8_t *mask, float *reward,
                  uint8_t *done, void *term_obs, int32_t *actions_out, void *stream);

/* How hexb_step / hexb_rollout spread a chunk of 32 games over warps: 0 (default) = chosen by the depth of the launch, 1 = one
 * warp per chunk (the form for deep, bandwidth-bound launches), 4 = a CTA of 4 warps per chunk (sub-wave launches, where a step
 * costs one warp's instruction latency: the warps split the relabel sweeps of flood_fill, HexGame.py:124-142 /
 * HexSingleGame.py:135-153, the observation + mask encode and the games of the thread-per-game phase). Any other value returns
 * HEXB_ERR_ARG. Results do not depend on the form; the call lets tests run each form on batch sizes where the depth rule would
 * pick the other. */
int32_t hexb_set_launch_form(hexb_env *env, int32_t warps_per_chunk);

/* T env steps in ONE launch with the fused random agent (the reference's random-vs-random rollout loop,
 *   for t in range(T): a = BaseRandomPolicy().choose_action(obs); obs, r, done, _, _ = env.step(a); reset on done,
 * i.e. hexb_step(actions = null) called T times) with the packed state staying on chip between steps: a warp keeps its 32 games
 * in shared memory and registers and the state crosses HBM once per launch instead of once per step. Bit-identical to T calls
 * of hexb_step. Every output gets a leading step dimension: obs i8[T,G,N,N], mask u8[T,G,N*N], reward f32[T,G], done u8[T,G],
 * term_obs i8[T,G,N,N], actions_out i32[T,G] (each nullable) - the layout of a rollout buffer. */
int32_t hexb_rollout(hexb_env *env, int32_t num_steps, void *obs, uint8_t *mask, float *reward, uint8_t *done, void *term_obs,
                     int32_t *actions_out, void *stream);

/* Optional per-game outputs of every following hexb_step (null = off): what the reference returns in the info dict of variant-A
 * HexEnv.step (HexGame.py:281-286) - last_move_opponent i32[G] (the opponent's move of this step as HexEnv reports it: variant A
 * the true cell, variant B the cell in the opponent's own view; -1 if it did not move) and winner i8[G] (env.winner: -1 None,
 * 0 BLACK, 1 WHITE, 3 illegal move). info["last_move_player"] is hexb_step's actions_out. */
int32_t hexb_set_info_buffers(hexb_env *env, int32_t *last_move_opponent, int8_t *winner);

/* The same step with HOST buffers (pinned memory recommended): copies actions_host to the device, steps, copies
 * obs/mask/reward/done back and waits for them. This is the call a host-side (CPU policy) user of the reference
 * API makes; it needs hexb_host_workspace_bytes(cfg) bytes of device scratch passed at every call. */
size_t hexb_host_workspace_bytes(const hexb_config *cfg);
int32_t hexb_step_host(hexb_env *env, void *workspace, const int32_t *actions_host, void *obs_host, uint8_t *mask_host,
                       float *reward_host, uint8_t *done_host, void *stream);

/* Transport of the observation + mask bytes inside hexb_step_host (they are 2*N*N of the 2*N*N + 5 bytes per game): by default
 * the games of a step are split between plain DMA copies and a 2-bit-per-cell transport that host threads expand into the same
 * arrays while the DMA runs (see hexb_step_host_packed); the split is searched during the first 22 calls (five coarse splits and
 * two neighbours of the best, three timed calls each - which mix is fastest depends on how many GPUs share the host's memory
 * system) and then kept. The bytes that arrive do not depend on it. dma_fraction in [0,1] pins the share of games copied as plain bytes (1 = no host threads,
 * plain DMA only, the behaviour of library version 1.2), a negative value selects the adaptive default again. Environment:
 * HEXB_HOST_DMA_FRACTION, HEXB_HOST_THREADS. Applies when obs_host and mask_host are both given, obs_dtype is HEXB_OBS_I8
 * and the shard has at least 4,096 games. */
int32_t hexb_set_host_transport(hexb_env *env, double dma_fraction);
int32_t hexb_get_host_transport(const hexb_env *env, double *dma_fraction);

/* The same call split in two, so that a host-side policy can work while the step and its copies are in flight:
 * hexb_step_host_begin enqueues H2D + step + D2H on `stream` and returns at once; hexb_step_host_end waits until the results
 * are in the host buffers (the host threads of the packed part of the transport work inside _end). One step may be pending per
 * handle (a second _begin before _end is HEXB_ERR_ARG). */
int32_t hexb_step_host_begin(hexb_env *env, void *workspace, const int32_t *actions_host, void *obs_host, uint8_t *mask_host,
                             float *reward_host, uint8_t *done_host, void *stream);
int32_t hexb_step_host_end(hexb_env *env);

/* hexb_step_host with ONLY the bit-packed transport (hexb_step_host itself mixes both): the step's observations cross PCIe as 2 bits per cell (the legal-action mask is
 * implied: legal == empty, HexSingleGame.py:205-206 / HexGame.py:203-204) and a pool of host threads (HEXB_HOST_THREADS, default:
 * the calling thread's CPU affinity count) expands them into the same int8 obs_host[G,N,N] and uint8 mask_host[G,N*N] arrays
 * hexb_step_host fills - bit-identical results, 8x fewer bytes on the device->host path, host cores doing the writes instead of
 * the DMA engine. packed_host: hexb_host_packed_bytes(cfg) bytes of (pinned) host staging. obs_dtype must be HEXB_OBS_I8 and
 * obs_host / mask_host must both be given. hexb_host_threads() = size of the pool. */
size_t hexb_host_packed_bytes(const hexb_config *cfg);
int32_t hexb_step_host_packed(hexb_env *env, void *workspace, void *packed_host, const int32_t *actions_host, int8_t *obs_host,
                              uint8_t *mask_host, float *reward_host, uint8_t *done_host, void *stream);
int32_t hexb_host_threads(void);

/* Device memory for the packed state and the step's large outputs, optionally COMPRESSIBLE (cuMemCreate with
 * CU_MEM_ALLOCATION_COMP_GENERIC: the L2's inline compression then shrinks what these buffers move over HBM; ordinary
 * allocations always travel uncompressed). The buffers hold what the reference keeps in numpy arrays (board and region planes:
 * HexGame.py:23,38-45, HexSingleGame.py:27,42-49; the observation and mask a step returns); their contents and every result are
 * unchanged, only the bytes that cross HBM are fewer: measured on B200, 1 Mi games, us per step ordinary / compressible: 19x19
 * 244 / 187-209, 11x11 88.1 / 86.5 (profiles/r2v_*). bytes is rounded up to the allocation granularity (2 MiB); *ptr is aligned to
 * it. compressible != 0 asks for compression; *granted (nullable) says whether the allocation really is compressible (the
 * driver may refuse, then ordinary memory is returned). Free with hexb_mem_free only. Not asynchronous, not graph-capturable:
 * allocate before the step loop. */
int32_t hexb_mem_alloc(int32_t device, size_t bytes, int32_t compressible, void **ptr, int32_t *granted);
int32_t hexb_mem_free(void *ptr);

/* Batched HexGame.make_move (fast_move: HexGame.py:85-111, HexSingleGame.py:88-122) on a raw=1 handle.
 * actions i32[G]: variant A true row-major cell, variant B the mover's-view cell as HexEnv.step passes it.
 * ret i8[G]: -1 = None, 0 = BLACK won, 1 = WHITE won, 3 = illegal (state untouched). */
int32_t hexb_ply(hexb_env *env, const int32_t *actions, int8_t *ret, void *stream);

/* Observation + mask of the current state without stepping (get_action_mask HexGame.py:203-204, legal_actions
 * HexSingleGame.py:205-206, the live simulator.board). view 0 = the agent's (what step/reset return), view 1 = the
 * side to move's (variant-B HexEnv one-ply loop: board after invert_board, HexSingleGame.py:259-262; variant A: the transposed,
 * colour-swapped board HexEnv.opponent_move hands its policy when the opponent is to move, HexGame.py:333-334). */
int32_t hexb_encode(hexb_env *env, int32_t view, void *obs, uint8_t *mask, void *stream);

/* k-th-empty-cell sampler, standalone (BaseRandomPolicy.choose_action SelfplayWrapper.py:17-22; random_policy
 * minihex/__init__.py:8-12): actions_out[g] = int(u[g] * n_empty)-th empty cell of game g in row-major order of the
 * chosen view (see hexb_encode). u f64[G] must be given. */
int32_t hexb_sample_actions(hexb_env *env, int32_t view, const double *u, int32_t *actions_out, void *stream);

/* Reference-layout dump for parity checks and checkpoints (attribute reads .board/.regions/.region_counter/...):
 * board f64[G,N,N] (live simulator.board), regions f64[G,2,N+2,N+2] incl. borders, region_counter f64[G,2],
 * cur i8[G] (simulator.current_player_num), done u8[G], winner i8[G] (-1 none), agent i8[G] (true colour),
 * draws u32[G] (stream position). Any pointer may be null. */
int32_t hexb_export_state(hexb_env *env, double *board, double *regions, double *region_counter, int8_t *cur, uint8_t *done,
                          int8_t *winner, int8_t *agent, uint32_t *draws, void *stream);

/* HexGame.__init__ with a preset board and connected_stones=None (HexGame.py:53-61, HexSingleGame.py:57-65): stones are
 * inserted in raster order through flood_fill. board_true i8[G,N,N] in {0 BLACK, 1 WHITE, 2 EMPTY}, true coordinates and
 * colours; to_move i8[G] (true colour to move, null = BLACK); import_mask u8[G] (null = every game). On a raw=1 handle this is
 * the constructor; on an env handle (after hexb_reset) it is HexEnv.reset with sample_board=True (HexSingleGame.py:217-222,
 * random_board :300-331): the game keeps its agent colour and stream position. If the opponent is then to move, call
 * hexb_half_step(side 1, actions) with the caller's opponent, or with actions = null for the built-in random opponent
 * (SelfPlayEnv.reset -> continue_game, SelfplayWrapper.py:79-80); env handles used this way are manual_opponent=1 ones, whose
 * resets leave the opening move to that call. */
int32_t hexb_import_boards(hexb_env *env, const int8_t *board_true, const int8_t *to_move, const uint8_t *import_mask, void *stream);

/* HexGame.__init__ with connected_stones given (HexGame.py:46-51, HexSingleGame.py:50-55): the region-label planes are adopted as
 * they are and region_counter = max(plane) + 1 - what HexEnv.reset does from its second call on with the planes cached at the
 * first (HexGame.py:214-220, HexSingleGame.py:226-231), and with a user-supplied `regions=`. board_true as in hexb_import_boards;
 * regions u8[G,2,N+2,N+2] in the reference's layout (plane 0 BLACK, plane 1 WHITE, true coordinates, borders included; every
 * stone must carry its label, labels < 128). */
int32_t hexb_import_labels(hexb_env *env, const int8_t *board_true, const uint8_t *regions, const int8_t *to_move,
                           const uint8_t *import_mask, void *stream);

/* Tree-search primitives (library version 1.5).
 *
 * copy.deepcopy(env.simulator) for many games at once (the HexGame.__init__ state, HexGame.py:21-68, HexSingleGame.py:26-71: board,
 * regions, region_counter, current_player_num, done, winner). dst game dst_index[i] becomes a bare HexGame holding the position of
 * src game src_index[i], for i < count. dst must be a raw=1 handle; src may be any handle of the same board_size and variant on the
 * same device (else HEXB_ERR_ARG before any launch; obs_dtype, seed, num_games and game_offset may differ). src_index / dst_index
 * are device i64[count]; null = the identity 0..count-1. Broadcasting one root into many children is the main use
 * (src_index = roots.repeat_interleave(C)). The copy is exact: hexb_export_state gives the same regions, region_counter (the
 * counters themselves, not max(plane) + 1 as hexb_import_labels sets them), cur, done and winner for both games, and the next
 * hexb_ply on the copy does what the reference's make_move (HexGame.py:85-111, HexSingleGame.py:88-122) does on the copied
 * simulator. An env game whose agent is WHITE is converted from its agent's orientation into true coordinates. Entries of dst_index
 * must be distinct and, when dst == src, disjoint from the src games read; otherwise the result is undefined. A pair with an
 * out-of-range index writes nothing; dst games not named in dst_index are untouched. */
int32_t hexb_copy_games(hexb_env *dst, const hexb_env *src, const int64_t *src_index, const int64_t *dst_index, int64_t count,
                        void *stream);

/* Random playouts: playout p of global game g starts from the game's current position with simulator.current_player_num to move,
 * colours alternating; ply k plays the int(u * n_empty)-th empty cell in true row-major order (random_policy,
 * minihex/__init__.py:8-12) with u built like every other draw (CPython's random.random() recipe) from Philox4x32-10 at counter
 * (k, g_lo, g_hi, p + 1) under the handle's seed (c3 = p + 1: the env streams use c3 = 0, so the two never overlap). The playout's
 * winner is the colour whose edges connect on the filled board (BLACK rows 0 and N-1, WHITE columns 0 and N-1; the reference's
 * neighbourhood, HexGame.py:124-142); a full Hex board has exactly one. p runs over [first_playout, first_playout + num_playouts):
 * calls with different first_playout give independent samples. first_playout >= 0, num_playouts >= 1 and
 * first_playout + num_playouts < 2^32. wins i32[G] = playouts won by the side to move, or -1 for a finished game, a game never
 * reset and a game with game_mask[i] == 0 (u8[G], null = every game). Any handle: raw, variant A or variant B env. */
int32_t hexb_playouts(hexb_env *env, int32_t num_playouts, int64_t first_playout, const uint8_t *game_mask, int32_t *wins,
                      void *stream);

/* Playout policies. Both play the same plies with the same draws u; they differ only in the cell a ply takes.
 * HEXB_PLAYOUT_RANDOM: the playout above (hexb_playouts).
 * HEXB_PLAYOUT_BRIDGE: save bridges. D = ((-1,0), (-1,1), (0,1), (1,0), (1,-1), (0,-1)) lists the six neighbours (dy, dx) of a
 *   cell in cyclic order; the common neighbours of c and c + D[i] are c + D[i-1] and c + D[i+1] (indices mod 6). A point is
 *   colour m's if it is on the board and holds a stone of m, or if it is off the board on m's side: BLACK owns the points with
 *   y < 0 or y >= N and 0 <= x < N, WHITE the points with x < 0 or x >= N and 0 <= y < N; no one owns the other off-board points
 *   (so a stone on the second row with both cells to its edge empty is bridged to the edge). At ply k with mover m and prev the
 *   cell of ply k-1, the reply set R is every cell e = prev + D[i] that is on the board and empty and whose prev + D[i-1] and
 *   prev + D[i+1] are both m's. If R is not empty, ply k plays the choice_of(u, |R|) = int(u * |R|)-th cell of R in true
 *   row-major order; otherwise the int(u * n_empty)-th empty cell, as the random policy does. A ply with an empty R therefore
 *   plays the cell the random policy would play on the same board. Ply 0 has no prev in hexb_playouts_policy (R is empty); in
 *   hexb_mcts_search_policy a leaf at depth >= 1 uses the move into it (the path's last cell) and node 0 has none.
 * Any other policy value: HEXB_ERR_ARG before any launch. */
#define HEXB_PLAYOUT_RANDOM 0
#define HEXB_PLAYOUT_BRIDGE 1
/* hexb_playouts with playouts of `policy`; hexb_playouts is policy HEXB_PLAYOUT_RANDOM. */
int32_t hexb_playouts_policy(hexb_env *env, int32_t num_playouts, int64_t first_playout, int32_t policy, const uint8_t *game_mask,
                             int32_t *wins, void *stream);

/* Batched Monte-Carlo tree search (PUCT), one tree per game g of `env` (any handle: raw, variant A or B env), in a device buffer
 * of hexb_mcts_tree_bytes(env, max_nodes) bytes (16-byte aligned; layout: csrc/hexb_mcts.cuh). Every call is asynchronous on
 * `stream`, allocates nothing and reads nothing on the host (CUDA-graph capturable). Bad max_nodes (1..2^24), num_simulations
 * (>= 1), playouts_per_leaf (1..65536), c_puct / fpu (NaN) or first_playout (0..2^32-1): HEXB_ERR_ARG; a null or misaligned
 * tree, or one smaller than hexb_mcts_tree_bytes: HEXB_ERR_STATE. A buffer that holds no tree of this handle (init never ran on
 * it, other board size or game count) is left alone by search / select / expand / root / advance.
 *
 * init: each root's current position is read in true orientation. A root is inactive (nothing is ever done for it) if its game
 *   is finished, was never reset or has root_mask[g] == 0 (u8[G], null = all); an active root gets node 0, unexpanded, and
 *   s = 0 simulations. c_puct, fpu (as float32) and first_playout are kept in the tree.
 * Nodes are numbered in creation order, at most max_nodes per root; a node's side to move is the root's, alternating with depth.
 *   An expanded node has one edge per cell: child (-1 none), N (i32), W, P (f32); every node has Nn (simulations whose path
 *   contained it) and a terminal flag.
 * One simulation:
 *   1 select: from node 0, at an expanded non-terminal node take the empty cell with the largest Q + U, Q = W / N if N > 0 else
 *     fpu, U = c_puct * P * sqrt(Nn) / (1 + N), in float32 with every operation rounded once (no FMA; exactly
 *     ((c_puct * P) * sqrt(Nn)) / (1 + N), then Q + U), ties to the lowest true row-major cell; -0 and +0 tie. A NaN Q + U
 *     ranks below every number: such a cell is taken only when every empty cell's Q + U is NaN, and then the lowest such cell
 *     wins. (A NaN can come from infinite or NaN values, c_puct = inf with a zero prior, or fpu = -inf against an infinite U.
 *     Which NaN bit pattern W, q and value then hold is not part of this definition.) An expanded child: descend; a
 *     terminal child is the leaf; no child: the new position is the leaf. Node 0 before its first simulation, and a node with no
 *     empty cell, is itself the leaf.
 *   2 value v for the leaf's side to move: if the move into a new leaf connects the mover's edges the leaf is terminal and
 *     v = -1 (so is a terminal child's). Otherwise, in hexb_mcts_search, P playouts exactly as hexb_playouts with playout index
 *     p = first_playout + s * P + j (mod 2^32) of the root's global game index, v = (2 * wins - P) / P, priors 1 / n_empty on
 *     the empty cells; in the split form v and the priors come from hexb_mcts_expand (cells not empty are ignored, nothing is
 *     renormalised).
 *   3 store: if fewer than max_nodes nodes exist, a new leaf becomes a node (expanded with the priors: children -1, N = W = 0;
 *     or terminal); node 0 is expanded in place. A full pool stores nothing; the value is still backed up.
 *   4 back up: Nn += 1 on every node of the path (leaf included: a new node starts at 1); every edge of the path gets N += 1 and
 *     W += the value for the player who made that move (-v into the leaf, sign alternating upwards); the root sums v as seen by
 *     its side to move; s += 1.
 * Per-cell arrays (visits, q, priors, leaf_obs, leaf_mask) use hexb_ply's action convention of a raw handle of the same variant
 * for the side to move at that node: variant A true cells, variant B the mover's view (transposed for WHITE). For an env root at
 * the agent's turn that is the agent's action space. */
int32_t hexb_mcts_tree_bytes(const hexb_env *env, int32_t max_nodes, size_t *bytes);
int32_t hexb_mcts_init(const hexb_env *env, void *tree, size_t tree_bytes, int32_t max_nodes, double c_puct, double fpu,
                       int64_t first_playout, const uint8_t *root_mask, void *stream);
/* The fused form: num_simulations simulations with playout evaluation for every active root, in one launch. search(a) followed
 * by search(b) equals search(a + b). */
int32_t hexb_mcts_search(const hexb_env *env, void *tree, size_t tree_bytes, int32_t num_simulations, int32_t playouts_per_leaf,
                         void *stream);
/* hexb_mcts_search with leaf playouts of `policy` (HEXB_PLAYOUT_*; hexb_mcts_search is HEXB_PLAYOUT_RANDOM). The policy is an
 * argument of the call, not state of the tree: search(a) followed by search(b) equals search(a + b) under one policy. */
int32_t hexb_mcts_search_policy(const hexb_env *env, void *tree, size_t tree_bytes, int32_t num_simulations, int32_t playouts_per_leaf,
                                int32_t policy, void *stream);
/* The split form, one simulation per select / expand pair (results are defined only when they alternate). select: step 1 for
 * every active root. A leaf that needs an evaluation gets leaf_obs[g] (obs_dtype [G,N,N]) and leaf_mask[g] (u8 [G,C]) - what
 * hexb_encode(view 1) returns for a raw game of the same variant holding the leaf - and pending[g] = 1 (u8 [G]); a terminal
 * leaf is backed up at once and, like an inactive root, gets pending[g] = 0 and no leaf row. expand: steps 2-4 for the pending
 * roots with priors f32[G,C] and values f32[G] (rows of the others are ignored). Root Dirichlet noise is the caller's: add it
 * to the priors of the first expand, whose leaf is the root. */
int32_t hexb_mcts_select(const hexb_env *env, void *tree, size_t tree_bytes, void *leaf_obs, uint8_t *leaf_mask, uint8_t *pending,
                         void *stream);
int32_t hexb_mcts_expand(const hexb_env *env, void *tree, size_t tree_bytes, const float *priors, const float *values, void *stream);
/* The root's edges: visits i32[G,C], q f32[G,C] (W / N, 0 where N = 0), value f32[G] (the root's value sum / its Nn, 0 before
 * the first simulation), nodes_used i32[G] (0 = inactive root). Every output is nullable. */
int32_t hexb_mcts_root(const hexb_env *env, const void *tree, size_t tree_bytes, int32_t *visits, float *q, float *value,
                       int32_t *nodes_used, void *stream);
/* Tree reuse across moves: re-root every root's tree on the position its game has reached. For each root g:
 *   1 a root whose game is finished, was never reset or has root_mask[g] == 0 (u8[G], null = all) becomes inactive, as in init.
 *   2 the game's position P' (true orientation, side to move t') is compared with the root's position P (side to move t0): every
 *     stone of P must still be in P' with the same colour; A = the stones P' adds. |A| = 0 and t' = t0: the tree is kept as it
 *     is. |A| = 1, a stone of t0 and t' = t0 ^ 1: the path is (c1). |A| = 2, one stone of each colour and t' = t0: the path is
 *     (c1 = t0's stone, c2 = the other). Anything else, or a root that was inactive: a fresh tree, exactly as init leaves it.
 *   3 the path is walked from node 0: every node on it must be expanded, its child at the path cell a stored node
 *     (0 <= child < nodes used), and the node r reached expanded; otherwise the root gets a fresh tree (a move never visited, a
 *     pool that was full when the child would have been stored, node 0 before its first simulation).
 *   4 the kept nodes are r and every node reachable from it through child pointers, renumbered in increasing old number (r
 *     becomes node 0); each keeps its flag, Nn and edges (child pointers renumbered). Nodes used = the kept count, the root's
 *     position = P' with t' to move, s and node 0's Nn = N of the edge into r, the root's value sum = -W of that edge (an exact
 *     float32 sign flip). Usually that N equals Nn(r); they differ only when r was stored after its edge had been visited (a
 *     pool that was full, then freed by an earlier advance). A pending split-form leaf is cleared.
 *   5 first_playout (0..2^32-1) replaces the tree's: later fused simulations use playout index first_playout + s * P + j with
 *     the root's new s. c_puct, fpu and max_nodes are unchanged.
 * So after a one-move advance the root's visits are the old edge's N and its value is -(the old root's q at the played cell).
 * Stones are matched, not moves: ply() on a raw handle adds one stone, an env step the agent's move and the opponent's reply, and
 * an episode end or auto-reset gives a fresh or inactive root. A select / expand pair must not straddle an advance. Argument
 * checks as above; asynchronous, no allocation, no host read. */
int32_t hexb_mcts_advance(const hexb_env *env, void *tree, size_t tree_bytes, int64_t first_playout, const uint8_t *root_mask,
                          void *stream);

/* Episode statistics accumulated by hexb_step since creation, int64[8] on the device:
 * [0] episodes finished, [1] BLACK wins, [2] WHITE wins, [3] agent wins, [4] plies of finished episodes,
 * [5] episodes ended by an illegal agent move, [6] env steps, [7] plies. Copies them to out8 (device). The multi-GPU
 * layer all-reduces this vector with NCCL; nothing else ever crosses GPUs. */
int32_t hexb_stats(hexb_env *env, int64_t *out8, void *stream);

/* Split step for a learned opponent (SURVEY.md section 8f row 2). On a manual_opponent=1 handle one env step is
 *   hexb_half_step(side 0, agent actions)  ->  hexb_encode(view 1) for the games with to_move == 1  ->  opponent network  ->
 *   hexb_half_step(side 1, opponent actions)  [twice: a game the opponent just won restarts, and if the opponent also opens the
 *   new episode it needs the opening move]
 * (hexb_half_step(side 1, actions = null) lets the built-in random opponent move instead of the caller's.)
 * hexb_half_step plays ONE ply of `side` (0 agent, 1 opponent) in every live, unfinished game whose turn it is: the agent's half
 * of SelfPlayEnv.step (SelfplayWrapper.py:174-176, HexSingleGame.py:233-263) or continue_game (:146-172) with the action supplied
 * by the caller in the mover's own perspective (exactly what OpponentPolicy.choose_action returns). Other games are untouched.
 * reward f32[G]: this ply's reward for the AGENT (+1 agent won, -1 opponent won, 0; variant A: -100 illegal agent move); done u8[G];
 * term_obs as in hexb_step (each nullable). Finished games auto-reset if configured; a restarted game whose opponent opens
 * waits for the caller. hexb_set_opponent_buffers registers two optional per-game outputs written by every reset and half step:
 * opp_index i32[G] (the opponent setup_opponents chose: -1 best model, k pool entry) and to_move u8[G] (0 agent, 1 opponent,
 * 2 finished). */
int32_t hexb_set_opponent_buffers(hexb_env *env, int32_t *opp_index, uint8_t *to_move);

/* SelfPlayEnv.set_eval(eval_state) (SelfplayWrapper.py:117-120; what SelfPlayCallback calls around its evaluation,
 * EvaluationCallback.py:31-33) at run time: hexb_config.eval_state from now on. While it is set, a reset draws nothing for the
 * opponent choice, and - when both opp_index (hexb_set_opponent_buffers) and eval_episode i32[G] (device, nullable, registered by
 * this call and zeroed on `stream`, as set_eval zeroes self.eval_episode) are there - episode k of a game since this call meets
 * pool entry k: opp_index = k while k <= pool_size - 1, later episodes keep the opponent they have (setup_opponents :92-96).
 * The running episode is not touched. Variant B handles only. */
int32_t hexb_set_eval(hexb_env *env, int32_t eval_state, int32_t *eval_episode, void *stream);

/* Variant-A HexEnv(opponent_policy="opponent_predict", opponent_model=..., eps=...) (HexGame.py:165-167,180,354-359; what
 * scripts/selfplay.py:38-44 creates through gym.make("hex-v0", ...)) for a manual_opponent=1 variant-A handle: from now on every
 * opponent ply of hexb_half_step(side 1, actions) first takes one draw rv from the game's stream (random.uniform(0,1)); with
 * rv < eps random_policy moves (one more draw, minihex/__init__.py:8-12), otherwise the caller's action - the model's prediction on
 * the view hexb_encode(view 1) shows - is played. eps < 0 switches the mix off again (the caller's action always, no draw). */
int32_t hexb_set_opponent_eps(hexb_env *env, double eps);
int32_t hexb_half_step(hexb_env *env, int32_t side, const int32_t *actions, float *reward, uint8_t *done, void *term_obs,
                       void *stream);

/* Masked categorical sampling for a batch of policy outputs (the rollout feed of SURVEY.md section 8f, row 1). Replaces what
 * sb3_contrib's MaskableCategoricalDistribution does between MaskablePPO's policy network and env.step in the reference's
 * training scripts (scripts/experiments/ *.py:40-47): illegal cells get probability 0, an action is drawn by inverse CDF from
 * the caller's uniforms and its log-probability is returned. No env handle: logits f32[G,C] row-major, mask u8[G,C]
 * (1 = legal, as hexb_step writes it), u f64[G] in [0,1); out: actions i32[G], logp f32[G] (either may be null),
 * entropy f32[G] (nullable). A row without a legal cell yields action -1, logp 0. */
int32_t hexb_masked_sample(const float *logits, const uint8_t *mask, const double *u, int64_t num_games, int32_t num_cells,
                           int32_t *actions, float *logp, float *entropy, int32_t device, void *stream);

/* Generalised advantage estimation over a [T,G] rollout collected with hexb_step (the rollout feed of SURVEY.md section 8f, row
 * 1): what stable-baselines3's RolloutBuffer.compute_returns_and_advantage does after MaskablePPO.collect_rollouts in the
 * reference's training scripts (scripts/experiments/ *.py:40-47; gamma 0.99, gae_lambda 0.95 in the saved models). No env handle.
 * rewards f32[T,G], values f32[T+1,G] (row T = the value of the observation after the last step), dones u8[T,G] (hexb_step's
 * done output: the episode ended in step t, which cuts bootstrap and trace);  out: advantages f32[T,G], returns f32[T,G] (nullable)
 *   delta_t = r_t + gamma * V_{t+1} * (1 - done_t) - V_t;  A_t = delta_t + gamma * lambda * (1 - done_t) * A_{t+1};  R_t = A_t + V_t
 * in float32, operation for operation like the eager loop it replaces. One thread per game, backward over t. */
int32_t hexb_gae(const float *rewards, const float *values, const uint8_t *dones, int32_t num_steps, int64_t num_games, double gamma,
                 double gae_lambda, float *advantages, float *returns, int32_t device, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* HEXB_H */
