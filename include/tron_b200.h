/*
 * tron_b200.h -- C ABI of the B200-native batched 2-player TRON environment and GPU replay ring.
 *
 * This is the drop-in boundary for the one hot path of ckawoalt/Deep-Q-Learning_TRON
 * (reference paths below are relative to Deep-Q-learning_TRON/ in that repository):
 *
 *   tron/game.py:70-91     Game.__init__            -> tron_reset
 *   tron/game.py:149-252   Game.next_frame          -> tron_step   (move, collision, trail/head writes)
 *   tron/game.py:254-277   Game.step (winner/draw)  -> tron_step   (done / winner resolution)
 *   tron/map.py:67-84      Map.color / state_for_player -> tron_step / tron_observe (TRON_ENC_LUT1)
 *   tron/util.py:11-37     pop_up                   -> tron_step / tron_observe (TRON_ENC_POPUP3)
 *   tron/util.py:38-45     prob_map                 -> TRON_ENC_POPUP3_CONST (4th constant plane)
 *   tron/util.py:46-84     make_game (spawn rule)   -> tron_reset / auto-reset inside tron_step
 *   tron/util.py:87-94, DQN.py:224-241, DDQN.py:289-305   reward policies -> tron_reward_t
 *   tron/game.py:137-139   Game.get_multy ([degree, weight]) -> tron_step_args.extra
 *   ACKTR.py:285-317       vector-env auto-reset contract -> tron_step(auto_reset=1)
 *   DDQN.py:90-110, DQN.py:63-64   epsilon-greedy   -> tron_select_actions
 *   DQN.py:81-132          ReplayMemory             -> replay_push / replay_gather / replay_sample_indices / replay_sample_gather
 *   DDQN.py:167-203        ReplayBuffer             -> replay_push / replay_gather / replay_sample_indices / replay_sample_gather
 *   DDQN.py:264-308, DQN.py:198-252   per-transition replay fill of the training loops -> replay_frames (the tick kernel writes
 *                          observations, rewards and done flags straight into the ring; replay_frames_sample_gather reads them back)
 *                          or replay_states (the ring keeps each tick's env state and actions; replay_states_sample_gather re-runs
 *                          the sampled ticks and renders both frames)
 *
 * Conventions
 *   - Every entry point is extern "C", returns 0 (TRON_OK) or a negative tron_status, never throws.
 *   - Every pointer documented "device" is a CUDA device pointer owned by the caller (torch allocates,
 *     the library owns no device memory except inside the opaque tron_host_env used for host buffers).
 *   - Device entry points are asynchronous w.r.t. the host and run on the cudaStream_t passed as
 *     `stream` (typed void* here so that C / cgo / ctypes callers need no CUDA headers).
 *   - The CUDA device is the caller's current device.
 *   - There is NO CPU fallback: without a usable CUDA device every compute call returns TRON_ERR_CUDA.
 *
 * Geometry (tron/map.py:43-48,86-92): a game of width W, height H stores (W+2) x (H+2) cells row-major,
 * `position = [p0, p1]` lives in cell (p0+1)*(H+2) + (p1+1); the border ring is WALL.  C := (W+2)*(H+2).
 * Actions (tron/player.py:107-132): 0=UP (p0-1) 1=RIGHT (p1+1) 2=DOWN (p0+1) 3=LEFT (p1-1).
 */
#ifndef TRON_B200_H
#define TRON_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TRON_B200_ABI_VERSION 4

typedef void* tron_stream_t; /* cudaStream_t */

typedef enum tron_status {
    TRON_OK = 0,
    TRON_ERR_INVALID = -1,     /* bad argument (null pointer, size, enum) */
    TRON_ERR_UNSUPPORTED = -2, /* valid but not implemented for this geometry/layout */
    TRON_ERR_CUDA = -3,        /* CUDA runtime error (no device, launch failure) */
    TRON_ERR_ALIGN = -4        /* pointer not aligned as documented */
} tron_status;

/* Cell codes, verbatim Tile.value (tron/map.py:9-17). */
enum {
    TRON_TILE_WALL = -1,
    TRON_TILE_EMPTY = 0,
    TRON_TILE_P1_BODY = 1,
    TRON_TILE_P1_HEAD = 2,
    TRON_TILE_P2_BODY = 3,
    TRON_TILE_P2_HEAD = 4,
    TRON_TILE_P1_SLIDE = 5,
    TRON_TILE_P2_SLIDE = 6
};

/* dtypes */
enum { TRON_U8 = 0, TRON_I32 = 1, TRON_I64 = 2, TRON_BF16 = 3, TRON_F32 = 4, TRON_I8 = 5 };

/* observation encodings */
enum {
    TRON_ENC_NONE = 0,        /* pure step, no observation written */
    TRON_ENC_LUT1 = 1,        /* 1 plane: Map.state_for_player (tron/map.py:67-84) */
    TRON_ENC_POPUP3 = 2,      /* 3 planes [wall, my, enemy]: pop_up (tron/util.py:11-37) */
    TRON_ENC_POPUP3_CONST = 3 /* pop_up + 4th constant plane (prob_map, tron/util.py:38-45) */
};

/* state layouts */
enum {
    TRON_LAYOUT_TILE8 = 0, /* int8 Tile.value per cell (any grid size, all modes) + 8-byte meta + 8-byte dirty boxes per env */
    TRON_LAYOUT_BITS10 = 1, /* 10x10 grids only, no slide modes: two 128-bit planes (trail occupancy, trail owner) over the
                              100 interior cells = 32 bytes per game; walls implicit, heads in the meta.  4.5x less state traffic. */
    TRON_LAYOUT_TRAIL = 2, /* any grid, all modes: per game a 16-byte header + the list of trail cells both players left behind
                              (capacity W*H each, 2 bytes per cell).  The header and the first 12 list entries of every game (64
                              bytes, "hot") are stored as four dense uint4 arrays [4][N] so that a tick streams them fully
                              coalesced; the rest of each list lives in a per-game cold area touched only by long episodes,
                              next to an occupancy bitmap of the cells those cold entries name (one probe per lookup).
                              Observations are rendered without materialising a grid: template rows in shared memory, patched
                              and bulk-stored by the TMA engine.  The fastest layout for fused observations from 12x12 up and
                              for pure ticks on large grids. */
    TRON_LAYOUT_BITS = 3   /* grids with W*H <= 128, all modes (incl. ice/temper): three 128-bit planes over the interior cells
                              (trail occupancy, trail owner, slide tile), stored as three dense uint4 arrays [3][N] = 48 bytes per
                              game; walls implicit, heads in the meta.  The bit-plane path for config.py's GAME_MODE="temper". */
};

/* RNG spawn rules of make_game (tron/util.py:46-84) */
enum {
    TRON_SPAWN_UNIFORM = 0, /* both heads uniform over the grid, (x1,y1) re-drawn while equal (util.py:64-78) */
    TRON_SPAWN_FAIR = 1     /* P1 in the clipped 3x3 box around a random point, P2 in the point-mirrored box (util.py:48-62) */
};

/* built-in synthetic policies for benchmark action streams (actions == NULL) */
enum {
    TRON_POLICY_UNIFORM = 0,  /* iid uniform{0..3} ("random policy") */
    TRON_POLICY_FREE_EPS = 1  /* epsilon-greedy proxy: with probability epsilon uniform{0..3}, else a uniformly random FREE
                                 neighbour cell of the own head if one exists, else uniform (SURVEY section 8d) */
};

/* slide ("ice"/"temper") modes, tron/game.py:163-178 */
enum {
    TRON_SLIDE_NONE = 0,
    TRON_SLIDE_TAPE = 1, /* explicit Bernoulli outcomes slide_tape[N,2] (1 = slide if eligible) */
    TRON_SLIDE_ICE = 2,  /* on-device RNG, constant rate (config.py:32 slide) */
    TRON_SLIDE_TEMPER = 3 /* on-device RNG, per-game rate from slide_params[N,4] = {degree, weight1, weight2, 0} */
};

/* Per-env metadata, 8 bytes, stored after the grids inside the state blob. */
typedef struct tron_meta {
    int8_t r1, c1, r2, c2; /* head positions [p0,p1] of player 1 and 2; range -1..W / -1..H */
    uint8_t flags;         /* bit0 P1 alive, bit1 P2 alive, bit2 done, bits3-4 winner (0 none,1,2), bit5 dirty boxes valid */
    uint8_t reserved;
    uint16_t ep_len;       /* ticks played in the current episode (len(game.history)-1) */
} tron_meta;

#define TRON_FLAG_ALIVE1 0x01u
#define TRON_FLAG_ALIVE2 0x02u
#define TRON_FLAG_DONE 0x04u
#define TRON_FLAG_WINNER_SHIFT 3

/* Reward policy.  Non-terminal step: step_base + step_per_tick * k, k = ticks already played in the
 * episode (DQN.py:224-225 `reward = historyStep`).  Terminal: (win, lose) or (draw, draw).
 *   DQN.py:224-241 survivor as coded : {0, 1, 100, -25, 0}     README.md:97-111 survivor : {1, 0, 100, -25, 0}
 *   README.md:47 basic (no code in the reference) : {0, 0, 100, -25, 0}
 *   DDQN.py:289-305 : {-1, 0, 100, -100, 0}     ACKTR.py:316 + config.py:37 : {-1, 0, 10, -10, 0} */
typedef struct tron_reward {
    float step_base, step_per_tick, win, lose, draw;
} tron_reward_t;

/* On-device statistics: TRON_STATS_SLOTS stripes of TRON_STATS_FIELDS uint64 counters; sum the stripes. */
#define TRON_STATS_SLOTS 64
#define TRON_STATS_FIELDS 8
enum {
    TRON_STAT_EPISODES = 0,
    TRON_STAT_P1_WINS = 1,
    TRON_STAT_P2_WINS = 2,
    TRON_STAT_DRAWS = 3,
    TRON_STAT_EP_TICKS = 4,   /* sum of finished-episode lengths */
    TRON_STAT_BAD_ACTION = 5, /* env-ticks skipped because an action was outside 0..3 */
    TRON_STAT_ENV_STEPS = 6   /* env-ticks actually advanced */
};

/* Arguments of tron_step / tron_observe / tron_step_many.  Zero-initialise, set struct_size. */
typedef struct tron_step_args {
    uint32_t struct_size; /* sizeof(tron_step_args) */
    int32_t n_envs;       /* N */
    int32_t width, height;
    int32_t layout;       /* TRON_LAYOUT_TILE8 | TRON_LAYOUT_BITS10 | TRON_LAYOUT_TRAIL */
    void* state;          /* device, tron_state_bytes() bytes, 256-byte aligned */

    const void* actions;  /* device [N,2] (P1,P2) values 0..3, or NULL -> built-in synthetic policy (see `policy`) from (seed,counter) */
    int32_t action_dtype; /* TRON_U8 | TRON_I32 | TRON_I64 */

    void* obs;            /* device [N,2,P,W+2,H+2], 16-byte aligned, or NULL when obs_enc == TRON_ENC_NONE */
    int32_t obs_dtype;    /* TRON_BF16 | TRON_F32 | TRON_I8 */
    int32_t obs_enc;      /* TRON_ENC_* */
    int8_t lut[6];        /* {empty, wall, own body, enemy body, own head, enemy head}; all zero -> {1,-1,-2,-3,10,-10} */
    int8_t pad0[2];
    float const_plane;    /* value of the 4th plane for TRON_ENC_POPUP3_CONST */

    float* reward;        /* device [N,2] or NULL */
    tron_reward_t reward_table;
    uint8_t* done;        /* device [N] or NULL */
    uint8_t* winner;      /* device [N] (0 none/draw, 1, 2) or NULL */
    int32_t* ep_len_out;  /* device [N]: length of the episode that just finished, else 0; or NULL */

    int32_t auto_reset;   /* 1: a finished game is replaced by a fresh one in the same call (ACKTR.py:296-310) */
    const int8_t* spawn;  /* device [N,4] = {x1,y1,x2,y2} used by envs that reset in this call; NULL -> RNG spawn (util.py:70-78) */
    int32_t spawn_mode;   /* RNG spawn rule: TRON_SPAWN_UNIFORM (make_game default) | TRON_SPAWN_FAIR (make_game mode="fair", util.py:48-62) */

    uint64_t seed;        /* Philox key */
    uint64_t counter;     /* Philox counter low word: the caller advances it once per tick */
    uint64_t env_id_base; /* global id of env 0 of this shard (results independent of the sharding) */
    const uint64_t* counter_dev; /* optional device u64 added to `counter` when the kernel runs: lets a captured CUDA graph
                                    advance the RNG counter between replays (tron_advance_counter), NULL -> unused */

    int32_t slide_mode;   /* TRON_SLIDE_* */
    float slide_rate;     /* TRON_SLIDE_ICE */
    const uint8_t* slide_tape;  /* device [N,2] for TRON_SLIDE_TAPE */
    int8_t* slide_params;       /* device [N,4] {degree, weight1, weight2, 0}: the per-game parameters Game.__init__ draws for every
                                   game in every mode (tron/game.py:83,87).  Whenever given they are re-drawn for each game that is
                                   reset (tron_reset_ex, auto-reset); TRON_SLIDE_TEMPER needs them (slip rate), `extra` reports them. */

    uint64_t* stats;      /* device [TRON_STATS_SLOTS*TRON_STATS_FIELDS] or NULL */

    int32_t policy;       /* used when actions == NULL: TRON_POLICY_UNIFORM | TRON_POLICY_FREE_EPS */
    float policy_epsilon; /* TRON_POLICY_FREE_EPS: probability of a uniform move */

    /* tron_step_many only */
    int32_t n_ticks;      /* T */
    int32_t obs_every_tick; /* 1: obs is [T,N,2,P,W+2,H+2]; 0: obs (if any) holds the last tick only */
    /* with n_ticks>1: actions is [T,N,2] (or NULL -> RNG), spawn is [T,N,4] (or NULL -> RNG),
     * reward [T,N,2], done [T,N], winner [T,N], ep_len_out [T,N] (each may be NULL) */

    /* ---- added in ABI version 2 ---- */
    void* obs_terminal;   /* optional device buffer shaped and typed like `obs`: the rows of games that FINISHED in this call and were
                             auto-reset receive the observation of the finished game's last frame -- what DDQN.py:270-308 stores as
                             next_state of a terminal transition, while `obs` already shows the fresh game (ACKTR.py:309-310).  Rows
                             of other games are left untouched.  tron_step only.  Every layout; on TRAIL the observation rows of a group of
                             games must fit the bulk-store kernel's shared-memory budget (200 KB; TRON_ERR_UNSUPPORTED otherwise, e.g.
                             126x126 f32 with 4 planes).  NULL -> not written. */
    float* extra;         /* optional device [N,2,2] f32: per player {degree, weight_p} of the game `obs` shows (Game.get_multy,
                             tron/game.py:137-139) taken from slide_params; needs slide_params.  Written by tron_step,
                             tron_step_many (last tick), tron_observe and tron_reset_ex. */

    /* ---- added in ABI version 3 ---- */
    int32_t obs_prev;     /* tron_step only, a hint: 1 promises that, for every game, `obs` already holds the observation of the game's
                             state before this call, as the previous call left it, in the same encoding, dtype and lut.  A kernel may
                             then skip the 32-byte units of a row that this tick does not change (the 10x10 bit-plane layouts with bf16
                             or f32 observations do); every other kernel writes full rows.  obs_terminal rows are written in full. */
    int32_t pad1;
} tron_step_args;

/* ---- library ---- */
int tron_abi_version(void);
const char* tron_status_string(int status);
/* Number of CUDA devices visible, or a negative tron_status. */
int tron_device_count(void);

/* ---- geometry helpers (host only, no CUDA call) ---- */
/* Bytes of the state blob for N envs; cells per env; planes for an encoding; element size of a dtype. */
int tron_state_bytes(int n_envs, int width, int height, int layout, size_t* total_bytes);
int tron_state_offsets(int n_envs, int width, int height, int layout, size_t* grid_off, size_t* meta_off,
                       size_t* boxes_off);
/* Tuning knobs (process-wide).  TRON_OPT_SPARSE_MIN_CELLS: pure ticks (TRON_ENC_NONE) of games with at least this
 * many cells run thread-per-game on HBM with dirty-box resets instead of staging whole grids (default 1024). */
enum {
    TRON_OPT_SPARSE_MIN_CELLS = 1,
    TRON_OPT_TILE_BYTES = 2, /* shared-memory budget of one tile of games in the generic-size fused kernel (default 18432) */
    TRON_OPT_ENCODE_VARIANT = 3, /* experiments (bit mask, 0 = default): 8 = per-plane observation store schedule on 10x10 boards instead of
                                     the linear one; 32 = element-store observation kernel on the trail layout instead of the bulk-store one;
                                     64 = full observation rows even when tron_step_args.obs_prev is set */
    TRON_OPT_BITS_CTAS_PER_SM = 4, /* resident CTAs per SM of the fused bit-plane kernels (capped by padding the dynamic shared memory).
                                     0 = default: 4 for the two-plane kernels, 5 with the slide plane -- these kernels are write
                                     streams and FEWER concurrent streams per SM than the register limit of 8 run faster on B200
                                     (0.95 -> 0.99 of the measured HBM peak, profiles/r2_cta_cap_sweep.jsonl); 32 = no cap */
    TRON_OPT_TILE_CTAS_PER_SM = 5 /* the same cap for the fused int8 tile kernels (0 = their default, 32 = no cap) */
};
int tron_set_option(int option, int64_t value);
int tron_cells_per_env(int width, int height);
int tron_enc_planes(int obs_enc);
int tron_dtype_size(int dtype);
/* Expand a 6-entry LUT + encoding into the per-player plane tables tab[2][planes][8] indexed by Tile.value+1. */
int tron_build_plane_tables(const int8_t lut6[6], int obs_enc, int8_t* tab /* [2*planes*8] */);

/* ---- environment (device pointers) ---- */
/* Fresh games (Game.__init__, tron/game.py:70-91): grid border WALL, interior EMPTY, heads written.
 * spawn: device [N,4] {x1,y1,x2,y2} or NULL -> RNG spawn with make_game's re-draw rule (util.py:70-78).
 * env_mask: device [N] u8, only envs with mask != 0 are reset; NULL -> all. */
int tron_reset(void* state, int n_envs, int width, int height, int layout, const int8_t* spawn, int spawn_mode,
               const uint8_t* env_mask, uint64_t seed, uint64_t counter, uint64_t env_id_base,
               tron_stream_t stream);
/* tron_reset with the full argument block: additionally draws the per-game parameters (slide_params[N,4] = {degree, weight1,
 * weight2, 0}, Game.__init__ tron/game.py:83,87) for every env it resets when slide_params is given, and fills `extra`.
 * Uses state, geometry, layout, spawn, spawn_mode, seed, counter, env_id_base, slide_mode, slide_params, extra. */
int tron_reset_ex(const tron_step_args* args, const uint8_t* env_mask, tron_stream_t stream);
/* One tick of every env, fused with observation encoding, rewards, done/winner and auto-reset. */
int tron_step(const tron_step_args* args, tron_stream_t stream);
/* Observation of the current state only (no tick): uses state, obs, obs_dtype, obs_enc, lut, const_plane. */
int tron_observe(const tron_step_args* args, tron_stream_t stream);
/* n_ticks ticks in one launch (grids stay in shared memory between ticks). */
int tron_step_many(const tron_step_args* args, tron_stream_t stream);
/* Copy out Tile.value grids [N,C] int8, heads [N,4] int8, alive [N,2] u8, done [N] u8, winner [N] u8,
 * ep_len [N] i32 (each may be NULL).  For history / drop-in shims / tests. */
int tron_export_grid(const void* state, int n_envs, int width, int height, int layout, int8_t* tiles,
                     int8_t* heads, uint8_t* alive, uint8_t* done, uint8_t* winner, int32_t* ep_len,
                     tron_stream_t stream);
/* Overwrite state from Tile.value grids + heads + alive (inverse of tron_export_grid; Map.__setitem__ shim).  Every array may be
 * NULL (= keep).  The bit-plane and trail layouts keep heads outside the cell data: with tiles given and heads == NULL they take the
 * head positions from the P1_HEAD / P2_HEAD tiles of the grid (a grid showing only P2's head is the shared-cell head-on state);
 * a grid with several head tiles of one player, or slide tiles on TRON_LAYOUT_BITS10, is representable on TRON_LAYOUT_TILE8 only. */
int tron_import_grid(void* state, int n_envs, int width, int height, int layout, const int8_t* tiles,
                     const int8_t* heads, const uint8_t* alive, const uint8_t* done,
                     const uint8_t* winner, const int32_t* ep_len, tron_stream_t stream);

/* ---- policies ---- */
/* Uniform random actions [n,2] u8 from Philox(seed; counter, env) -- same draws tron_step uses when actions==NULL. */
int tron_random_actions(uint8_t* actions, int n_envs, uint64_t seed, uint64_t counter, const uint64_t* counter_dev,
                        uint64_t env_id_base, tron_stream_t stream);
/* epsilon-greedy (DDQN.py:90-110): q device [n_rows,4] (TRON_F32|TRON_BF16); explore iff u <= epsilon.
 * Row i uses Philox stream row_id_base+i.  actions: device [n_rows] u8. */
int tron_select_actions(const void* q, int q_dtype, int n_rows, float epsilon, uint8_t* actions,
                        uint64_t seed, uint64_t counter, const uint64_t* counter_dev, uint64_t row_id_base,
                        tron_stream_t stream);
/* *counter_dev += delta on the stream (one thread); put it after the calls that read counter_dev inside a CUDA graph. */
int tron_advance_counter(uint64_t* counter_dev, uint64_t delta, tron_stream_t stream);

/* Scripted opponent: the action (0..3) MinimaxPlayer(2, voronoi) (tron/minimax.py:58-310) would take for `player` (1|2) in every
 * game.  tiles: device [N, (W+2)(H+2)] Tile.value grids (the TRON_LAYOUT_TILE8 state itself, or tron_export_grid output);
 * grids of at most 256 cells.  tie_mode 0: first best move / UP when boxed in; 1: Philox-uniform (random.choice / randint).
 * values: optional device [N,4] int32 minimax value of each root move (INT32_MIN = move not expanded).
 * child_ties: optional device [N,4] int32, per root move what the reference's depth-1 node draws from the global RNG when it
 * finishes (minimax.py:233-234,266-267): -1 = move not expanded (no draw), 0 = the enemy is boxed in (one random.randint(1,4)),
 * L in 1..4 = one random.choice over the L enemy moves that attain the minimum.  Lets a drop-in consume Python's global RNG
 * exactly like the reference (tron/minimax.py of this package). */
int tron_minimax_actions(const int8_t* tiles, int n_envs, int width, int height, int player, int tie_mode, uint64_t seed,
                         uint64_t counter, const uint64_t* counter_dev, uint64_t env_id_base, uint8_t* actions,
                         int32_t* values, int32_t* child_ties, tron_stream_t stream);

/* pop_up on observations that are already encoded (reference tron/util.py:11-37): obs device [n_maps, cells]
 * (TRON_I8|TRON_I32|TRON_I64|TRON_BF16|TRON_F32) -> planes device [n_maps, 3, cells] = {wall, my, enemy}
 * (TRON_F32|TRON_BF16|TRON_I8).  The fused path (TRON_ENC_POPUP3) never materialises the 1-plane form. */
int tron_pop_up(const void* obs, int obs_dtype, int64_t n_maps, int cells, void* planes, int out_dtype,
                tron_stream_t stream);

/* ---- replay ring (DQN.py:81-132 ReplayMemory, DDQN.py:167-203 ReplayBuffer) ---- */
typedef struct replay_ring {
    uint32_t struct_size;
    int32_t frame_elems; /* P*(W+2)*(H+2) */
    int32_t frame_dtype; /* TRON_BF16 | TRON_F32 | TRON_I8 */
    int32_t pad0;
    int64_t capacity;    /* transitions */
    void* state;         /* device [capacity, frame_elems]  (old_state / state) */
    void* next_state;    /* device [capacity, frame_elems]  (new_state / next_state) */
    uint8_t* action;     /* device [capacity] */
    float* reward;       /* device [capacity] */
    uint8_t* done;       /* device [capacity]  (terminal) */
} replay_ring;

/* Append n transitions at ring position `cursor % capacity` (wrapping; oldest overwritten, like
 * ReplayMemory.push DQN.py:92-96 and deque(maxlen) DDQN.py:182-189).  done_stride: 1 -> done[i] per
 * transition, 2 -> done[i/2] (one flag per env, two transitions per env).  n <= capacity. */
int replay_push(const replay_ring* ring, uint64_t cursor, const void* state, const void* next_state,
                const uint8_t* action, const float* reward, const uint8_t* done, int done_stride,
                int64_t n, tron_stream_t stream);
/* Gather k transitions by ring slot (ReplayBuffer.sample DDQN.py:191-200 output types):
 * out_state/out_next [k, frame_elems] in out_dtype (TRON_F32|TRON_BF16), out_action [k] i64,
 * out_reward [k] f32, out_done [k] f32. */
int replay_gather(const replay_ring* ring, const int64_t* idx, int64_t k, void* out_state,
                  void* out_next, int out_dtype, int64_t* out_action, float* out_reward,
                  float* out_done, tron_stream_t stream);
/* k distinct slots uniform in [0,size) (random.sample without replacement, DDQN.py:193, DQN.py:111-112): idx[i] = pi(i) where pi
 * is a keyed pseudo-random PERMUTATION of [0,size) (6-round Feistel network on ceil(log2 size) bits, round keys from
 * Philox(seed; counter), cycle-walking back into range).  Every index is computed independently, so any k <= size works and the
 * same function runs inside replay_sample_gather / replay_frames_sample_gather without a separate launch. */
int replay_sample_indices(int64_t size, int64_t k, uint64_t seed, uint64_t counter, int64_t* idx,
                          tron_stream_t stream);
/* replay_sample_indices + replay_gather in ONE launch: row i of the outputs is transition pi(i) of the `size` valid ring slots
 * [0,size).  out_idx: optional device [k] receiving the sampled slots. */
int replay_sample_gather(const replay_ring* ring, int64_t size, int64_t k, uint64_t seed, uint64_t counter, void* out_state,
                         void* out_next, int out_dtype, int64_t* out_action, float* out_reward, float* out_done,
                         int64_t* out_idx, tron_stream_t stream);

/* ---- frame-sharing replay ring (the batched training loops, DDQN.py:264-308 / DQN.py:198-252) ----
 * A ring of S time slots; slot (t % S) holds, for all `rows` = 2N (env, player) pairs, the observation the policy saw at tick t,
 * the action it took, the reward it got and the env's done flag.  next_state of transition (t, row) is the frame in slot
 * (t+1) % S -- the same memory the next tick's state lives in -- unless the env finished at tick t: then it is the row of
 * `terminal` the tick kernel filled through tron_step_args.obs_terminal.  The caller points tron_step's obs / reward / done /
 * obs_terminal and tron_select_actions' output at the slot, so "push" moves no data at all. */
typedef struct replay_frames {
    uint32_t struct_size;
    int32_t frame_elems; /* P*(W+2)*(H+2) */
    int32_t frame_dtype; /* TRON_BF16 | TRON_F32 | TRON_I8 */
    int32_t n_slots;     /* S >= 2 */
    int64_t rows;        /* 2N: row = 2*env + player */
    void* frames;        /* device [S, rows, frame_elems] */
    void* terminal;      /* device [S, rows, frame_elems] or NULL (then next_state of a terminal transition is the reset frame) */
    uint8_t* action;     /* device [S, rows] */
    float* reward;       /* device [S, rows] */
    uint8_t* done;       /* device [S, rows/2]: one flag per env */
} replay_frames;
/* Sample k distinct transitions uniformly among ticks [first_tick, first_tick + n_ticks) x rows (all of whose next frames must
 * already be in the ring: n_ticks <= S-1) and gather them, one launch.  Outputs as replay_gather; out_idx (optional) receives
 * tick * rows + row of each sample. */
int replay_frames_sample_gather(const replay_frames* fr, int64_t first_tick, int64_t n_ticks, int64_t k, uint64_t seed,
                                uint64_t counter, void* out_state, void* out_next, int out_dtype, int64_t* out_action,
                                float* out_reward, float* out_done, int64_t* out_idx, tron_stream_t stream);

/* ---- state replay ring (ABI 4): the same transitions from 42 bytes per game-tick (TRON_LAYOUT_BITS10) ----
 * Slot (t % S) holds the env's state blob BEFORE tick t (its first slot_bytes bytes: the bit planes and the tron_meta array, i.e.
 * meta_off + 8*N of tron_state_offsets, rounded up to 16), the two actions of tick t and, when the tick draws slide numbers, the
 * RNG counter it ran with and the temper mode's per-game parameters.  A transition (s, a, r, s', d) is a function of those: the
 * sampler re-runs the tick (tron_step's rules, no auto-reset), so s' of a game that finished is its last frame, as with
 * replay_frames.terminal.  Bit-plane layouts only (TRON_LAYOUT_BITS10, TRON_LAYOUT_BITS), every slide mode but TRON_SLIDE_TAPE. */
typedef struct replay_states {
    uint32_t struct_size;
    int32_t n_slots;        /* S >= 1 */
    int64_t slot_bytes;     /* >= meta_off + 8*N, a multiple of 16 */
    void* states;           /* device [S, slot_bytes], 16-byte aligned */
    uint8_t* action;        /* device [S, N, 2] */
    uint64_t* counter;      /* device [S]: the counter tick t ran with (tron_step_args.counter + *counter_dev); needed for ICE / TEMPER */
    int8_t* slide_params;   /* device [S, N, 4]: {degree, weight1, weight2, 0} of each game during tick t; needed for TEMPER */
} replay_states;
/* Sample k distinct transitions uniformly among ticks [first_tick, first_tick + n_ticks) x 2N rows (n_ticks <= S: s' is
 * recomputed, no slot holds it) and render them, one launch.  The same (seed, counter) picks the same (tick, row) as
 * replay_frames_sample_gather over the same window.  `env` is the argument block of the env the ring records: it supplies the
 * geometry, layout, encoding, obs dtype, lut, const plane, reward table, slide mode and rate, seed and env_id_base, and is
 * validated like a tron_step call (its obs, actions and output pointers are not used; its state pointer is not read).  Every output
 * element is what tron_step would have stored in the env's obs dtype, converted to out_dtype (TRON_F32 | TRON_BF16) as
 * replay_frames_sample_gather converts; outputs, alignment and out_idx (tick * 2N + row) as there.  TRON_ERR_UNSUPPORTED for
 * the other layouts and for TRON_SLIDE_TAPE. */
int replay_states_sample_gather(const replay_states* rs, const tron_step_args* env, int64_t first_tick, int64_t n_ticks, int64_t k,
                                uint64_t seed, uint64_t counter, void* out_state, void* out_next, int out_dtype, int64_t* out_action,
                                float* out_reward, float* out_done, int64_t* out_idx, tron_stream_t stream);

/* ---- host-buffer front end (what a Game.step caller with numpy arrays binds to) ---- */
typedef struct tron_host_env tron_host_env;
/* Owns device state for n_envs games plus staging streams; obs/reward policy fixed at creation. */
int tron_host_env_create(tron_host_env** out, const tron_step_args* proto /* geometry, obs, lut, reward, seed, auto_reset */,
                         int n_chunks);
int tron_host_env_destroy(tron_host_env* env);
/* spawn_host [N,4] or NULL (RNG); obs_host receives the initial observations (may be NULL). */
int tron_host_env_reset(tron_host_env* env, const int8_t* spawn_host, void* obs_host);
/* Host in: actions_host [N,2] u8, spawn_host [N,4] or NULL.  Host out (each may be NULL): obs, reward [N,2],
 * done [N], winner [N].  One H2D copy of the inputs, the tick kernels chunk by chunk, the observation D2H copies chunk by chunk
 * behind them on a dedicated copy stream and one D2H copy per scalar array; returns after all outputs landed. */
int tron_host_env_step(tron_host_env* env, const uint8_t* actions_host, const int8_t* spawn_host,
                       void* obs_host, float* reward_host, uint8_t* done_host, uint8_t* winner_host);
/* The same step split in two so that consecutive steps pipeline: _begin enqueues everything and returns at once (the
 * host buffers belong to the library until the matching _wait); _wait blocks until the OLDEST outstanding step has landed.
 * At most two steps may be outstanding (device observations are double-buffered: tick t+1 runs while tick t drains over PCIe). */
int tron_host_env_step_begin(tron_host_env* env, const uint8_t* actions_host, const int8_t* spawn_host,
                             void* obs_host, float* reward_host, uint8_t* done_host, uint8_t* winner_host);
int tron_host_env_step_wait(tron_host_env* env);
/* Device state pointer of a host env (for tron_export_grid). */
void* tron_host_env_state(tron_host_env* env);
/* Pinned host memory for the buffers above (plain malloc'd memory also works, slower).  Pages are placed on the NUMA node of
 * the current CUDA device (the calling thread is moved onto the device's local CPUs while the pages are allocated). */
int tron_host_alloc(void** ptr, size_t bytes);
int tron_host_free(void* ptr);
/* Measured PCIe ceiling of this process's device: `repeats` back-to-back cudaMemcpyAsync of `bytes` between tron_host_alloc
 * memory and device memory (direction 0 = host->device, 1 = device->host), timed with CUDA events -> GB/s. */
int tron_host_copy_bandwidth(size_t bytes, int direction, int repeats, double* gb_per_s);

/* ---- debug build (libtron_b200_debug.so, -DTRON_DEBUG; tests only) ----
 * Every computed cell index, trail-list position, ring slot and env ownership is range-checked on the device; a violation is
 * counted (and the access skipped) instead of corrupting memory.  Release builds return TRON_ERR_UNSUPPORTED. */
int tron_debug_violations(uint64_t* count, int32_t* first_code);

#ifdef __cplusplus
}
#endif
#endif /* TRON_B200_H */
