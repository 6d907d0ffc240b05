/*
 * agarcl_b200.h — C-ABI of the B200-native batched AgarCL simulator.
 *
 * This is the drop-in boundary for ONE hot path of machado-research/AgarCL:
 *   N lockstep instances of  BaseEnvironment::step  (environment/envs/BaseEnvironment.hpp:89-122)
 *     = ticks_per_step x Engine::tick (agario/engine/Engine.hpp:208-240), built-in bots
 *       (agario/bots/ headers), regen/respawn, rewards, dones,
 *   + GridObservation::add_frame (environment/envs/GridEnvironment.hpp:91-123).
 *
 * Every entry point below replaces what the reference's pybind11 module `agarcl`
 * (environment/bindings.cpp:94-135) binds for that path; the cited line is the
 * reference interface it stands in for.  Plain pointers and sizes only: no C++
 * or torch types cross this boundary.  All functions return 0 on success and a
 * negative agarcl_status on failure; agarcl_last_error() gives the text.
 *
 * The same header also fixes the per-instance STATE BLOB layout that is shared by
 *   - the CUDA library (device state = N blobs, `stride` bytes apart),
 *   - oracle/oracle.c (CPU restatement, test infrastructure only),
 *   - oracle/ref_harness.cpp (the compiled reference, dumps into the same blob),
 *   - tests/draw_oracle.c (CPU restatement of the pictures of agarcl_batch_draw, test infrastructure only),
 *   - tests/bot_oracle.c (oracle_bot_decide: oracle.c's bot code as the spec of agarcl_batch_bot_actions, test infrastructure only).
 */
#ifndef AGARCL_B200_H
#define AGARCL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---------------------------------------------------------------- constants
 * agario/core/settings.hpp, agario/core/Entities.hpp (SURVEY Appendix B).     */
#define AGARCL_CELL_MIN_SIZE 25u
#define AGARCL_CELL_SPLIT_MINIMUM 50u
#define AGARCL_PLAYER_CELL_LIMIT 14
#define AGARCL_FOOD_MASS 10u
#define AGARCL_PELLET_MASS 1u
#define AGARCL_VIRUS_INITIAL_MASS 100u
#define AGARCL_MAX_MASS_IN_THE_GAME 22500u
#define AGARCL_NEW_MASS_IF_NO_SPLIT 22000u
#define AGARCL_RECOMBINE_TICKS 300u /* RECOMBINE_TIMER_SEC(10) * 30 ticks/s, sim-time (DESIGN.md Q1) */

#define AGARCL_MAX_CELLS 32   /* cell slots per player (reference limit 14, Engine.hpp:592-601 can overshoot) */
#define AGARCL_VET_CAP 16     /* remembered virus_eaten_ticks per player (Player.hpp:31) */
#define AGARCL_MAX_PLAYERS 64 /* agents + bots per instance */
#define AGARCL_LUT_SIZE 65536 /* integer-mass lookup tables (radius, max_speed, split_speed) */

/* hdr.flags bits: set by the simulator when a fixed capacity was hit or a
 * non-replayable reference path was taken.  Parity is only claimed while 0.  */
#define AGARCL_FLAG_FOOD_OVERFLOW 0x001u
#define AGARCL_FLAG_VIRUS_OVERFLOW 0x002u
#define AGARCL_FLAG_CELL_OVERFLOW 0x004u
#define AGARCL_FLAG_VET_OVERFLOW 0x008u
#define AGARCL_FLAG_EATER_OVERFLOW 0x010u
#define AGARCL_FLAG_REPLAY_EXHAUSTED 0x020u
#define AGARCL_FLAG_PCD_TIE 0x040u     /* (round 1: >16 cells in one PCD strip with equal y.  No longer raised: libstdc++'s std::sort is restated exactly, ties included) */
#define AGARCL_FLAG_RAND_SITE 0x080u   /* a libc rand() site was reached (Bot.hpp:93-96,121-126) */
#define AGARCL_FLAG_MASS_LUT 0x100u    /* a cell mass exceeded AGARCL_LUT_SIZE */
#define AGARCL_FLAG_REMOVE_OVERFLOW 0x200u

typedef enum agarcl_status {
  AGARCL_OK = 0,
  AGARCL_ERR_INVALID = -1,   /* bad argument / config (EnvironmentException in the reference) */
  AGARCL_ERR_CUDA = -2,      /* CUDA runtime failure */
  AGARCL_ERR_NOMEM = -3,
  AGARCL_ERR_STATE = -4      /* call order (e.g. step before reset) */
} agarcl_status;

typedef enum agarcl_rng_mode {
  AGARCL_RNG_PHILOX = 0,  /* counter-based per-instance Philox4x32-10 on device */
  AGARCL_RNG_REPLAY = 1,  /* draws come from a per-instance stream uploaded with agarcl_batch_set_replay */
  AGARCL_RNG_MT19937 = 2  /* the host keeps one std::mt19937_64 per instance -- seeded by agarcl_batch_seed exactly as
                             Engine::seed does (Engine.hpp:242-245), from std::random_device when never seeded
                             (GameState.hpp:59) -- and feeds its uniform_real_distribution<float> draws
                             (random_location, Engine.hpp:143-148) to the device through a ring that it refills
                             ahead of every instance's cursor: the stream never runs out */
} agarcl_rng_mode;

typedef enum agarcl_obs_dtype { AGARCL_OBS_I32 = 0, AGARCL_OBS_I16 = 1 } agarcl_obs_dtype;

/* ------------------------------------------------------------------- config
 * Fields 2..11 are the positional arguments of agarcl.GridEnvironment
 * (environment/bindings.cpp:102, BaseEnvironment.hpp:39-51); fields 12..17 are
 * the keys of configure_observation (bindings.cpp:104-114).                   */
typedef struct agarcl_cfg {
  int32_t n_instances;
  int32_t num_agents, ticks_per_step, arena_size, pellet_regen, num_pellets, num_viruses, num_bots;
  int32_t reward_type, c_death, mode_number;
  int32_t num_frames, grid_size, observe_cells, observe_others, observe_viruses, observe_pellets;
  int32_t obs_dtype;        /* agarcl_obs_dtype; int32 is the reference's */
  int32_t strict_reference; /* 1: keep quirk Q11 (frame index) exactly, and quirk Q3: the player order of the episode that follows the
                               k-th unmasked agarcl_batch_reset is the one the reference has after its k-th reset (its player map and pid
                               counter outlive a reset, Engine.hpp:72,98-101); 0: always render the last frame(s), every episode in the
                               player order of a fresh engine */
  int32_t rng_mode;         /* agarcl_rng_mode */
  int32_t cap_viruses, cap_foods, cap_replay; /* 0 = defaults */
  int32_t device;           /* CUDA device ordinal */
  int32_t instance_base;    /* global index of local instance 0 (multi-GPU sharding; keys the RNG) */
  int32_t ram_obs;          /* 1: every step also produces the structured observation (agarcl_batch_ram); 2: ONLY that one
                               (agario-ram-v0: the grid frame is not rendered, agarcl_batch_obs stays zero) */
  int32_t task_modes;       /* 0: every instance plays mode_number.  Otherwise a MIXED-TASK batch: bit m set = mode m may run in it
                               (see "mixed-task batches" below); mode_number's bit must be set, it is every instance's first task */
  int32_t pixel_obs;        /* 0: off.  S, a multiple of 16 in [16, 2048]: the PIXEL OBSERVATION -- every step and reset produce one
                               RGB picture per agent (agarcl_batch_pixels) instead of the grid frame, which is not rendered
                               (agarcl_batch_obs stays zero, as under ram_obs = 2).  Needs num_frames = 1 (frame stacking is the
                               caller's: info reset_mask says which stacks to clear), strict_reference = 0 and ram_obs != 2 */
} agarcl_cfg;

/* ------------------------------------------------------------- state records */
typedef struct agarcl_cell { /* 48 B; agario/core/Entities.hpp:118-212 */
  float x, y, vx, vy;
  float svx, svy;        /* splitting_velocity */
  uint32_t mass;
  uint32_t id;           /* creation order inside the instance (Ball.hpp:15,18; only relative order is used) */
  uint32_t recomb_tick;  /* engine tick from which can_recombine() holds (Entities.hpp:183-193, sim-time) */
  uint32_t pad[3];
} agarcl_cell;

typedef struct agarcl_virus { /* 32 B; Entities.hpp:82-114 */
  float x, y;
  uint32_t mass;
  int32_t hits;          /* _num_food_hits */
  float vx, vy;
  uint32_t pad[2];
} agarcl_virus;

typedef struct agarcl_food { float x, y, vx, vy; } agarcl_food; /* 16 B; Entities.hpp:41-55 */
typedef struct agarcl_pellet { float x, y; } agarcl_pellet;     /* 8 B;  Entities.hpp:22-38 */

typedef struct agarcl_player { /* 128 B; agario/core/Player.hpp:25-41,211-215 */
  int32_t n_cells;
  float target_x, target_y;
  int32_t action;          /* 0 none, 1 feed, 2 split (core/types.hpp:59-61) */
  int32_t split_cd, feed_cd;
  float anti_team_decay;
  int32_t elapsed_ticks, last_decay_tick;
  int32_t bot_type;        /* -1 agent; 0 Hungry, 1 HungryShy, 2 Aggressive, 3 AggressiveShy */
  uint32_t min_mass_cell;
  int32_t food_eaten;
  uint32_t highest_mass;
  int32_t cells_eaten, viruses_eaten;
  int32_t vet_count;       /* virus_eaten_ticks.size() */
  int32_t vet_ticks[AGARCL_VET_CAP];
} agarcl_player;

typedef struct agarcl_inst_hdr { /* 64 B */
  uint32_t tick;           /* GameState::ticks */
  uint32_t next_cell_id;
  int32_t n_pellets, n_viruses, n_foods;
  uint32_t rng_cursor;     /* uniform draws consumed so far */
  uint32_t flags;          /* AGARCL_FLAG_* */
  uint32_t seed_lo, seed_hi;
  uint32_t done_sticky;    /* mode 3 sticky done (BaseEnvironment.hpp:132-135) */
  uint32_t respawned_lo, respawned_hi; /* players respawned at the end of the last step: the step's
                             observation is taken BEFORE repsawn_all_players (BaseEnvironment.hpp:96-101) */
  uint32_t pad[4];
} agarcl_inst_hdr;

/* Byte offsets of one instance's arrays inside its blob. */
typedef struct agarcl_layout {
  int32_t P, A;            /* players (agents + bots), agents */
  int32_t cap_cells, cap_pellets, cap_viruses, cap_foods, cap_replay;
  uint32_t off_hdr, off_players, off_cells, off_viruses, off_foods, off_pellets;
  uint32_t stride;         /* bytes per instance, multiple of 128 */
  /* engine mode flags, Engine::set_mode (Engine.hpp:367-416) */
  int32_t mass_decay, squared_pellets, regen, agent_mass;
  int32_t obs_channels;    /* per frame: 1 + cells + 2*others + 2*viruses + 2*pellets (GridEnvironment.hpp:188-195) */
  int32_t order[AGARCL_MAX_PLAYERS];    /* player index processed k-th (libstdc++ unordered_map order, SURVEY App. C) */
  int32_t bot_type[AGARCL_MAX_PLAYERS];
} agarcl_layout;

/* Fills `L` from `c` (host side; uses the same libstdc++ unordered_map the reference
 * iterates, GameState.hpp:44).  Returns AGARCL_ERR_INVALID on a bad config.  */
int agarcl_make_layout(const agarcl_cfg* c, agarcl_layout* L);

/* ---------------------------------------------------------------- batch API */
typedef struct agarcl_batch agarcl_batch;

/* GridEnvironment ctor + configure_observation (bindings.cpp:102-114). Allocates all device memory. */
int agarcl_batch_create(const agarcl_cfg* cfg, agarcl_batch** out);
int agarcl_batch_destroy(agarcl_batch* b);
int agarcl_batch_get_layout(const agarcl_batch* b, agarcl_layout* out);

/* BaseEnvironment::seed (BaseEnvironment.hpp:211): seeds[i] for instance i (host pointer, N entries). */
int agarcl_batch_seed(agarcl_batch* b, const uint64_t* seeds);
/* BaseEnvironment::reset (BaseEnvironment.hpp:179-204) for instances with mask[i]!=0 (NULL = all).  Like the reference's,
 * a reset does not reseed: the instance's draw stream goes on where the last episode left it (successive episodes
 * differ); only agarcl_batch_seed / agarcl_batch_set_replay / a snapshot load restart it at its first draw. */
int agarcl_batch_reset(agarcl_batch* b, const uint8_t* mask, void* stream);
/* (strict_reference: an unmasked reset changes layout.order -- fetch it again with agarcl_batch_get_layout) */
/* BaseEnvironment::take_actions (BaseEnvironment.hpp:141-176): dxdy[N*A*2], act[N*A].
 * on_device!=0: device pointers, read by the next step without a copy. */
int agarcl_batch_set_actions(agarcl_batch* b, const float* dxdy, const int32_t* act, int on_device, void* stream);
/* BaseEnvironment::step + GridObservation::add_frame for every agent, enqueued on `stream` (cudaStream_t). */
int agarcl_batch_step(agarcl_batch* b, void* stream);
/* get_state (bindings.cpp:67-91) without the copy: device pointer to obs [N*A, C*num_frames, G, G]. */
int agarcl_batch_obs(agarcl_batch* b, void** dev_ptr, int64_t shape[4], int32_t* dtype);
int agarcl_batch_rewards(agarcl_batch* b, double** dev_ptr); /* step() return value, f64[N*A] */
int agarcl_batch_dones(agarcl_batch* b, uint8_t** dev_ptr);  /* dones(), u8[N*A] */
/* The reference-facing call with HOST buffers: copies actions in, steps, copies obs/rewards/dones
 * out (any of the out pointers may be NULL) and synchronises.  This is what `e2e` in bench.py times. */
int agarcl_batch_step_host(agarcl_batch* b, const float* dxdy, const int32_t* act,
                           void* obs_out, double* rewards_out, uint8_t* dones_out);

/* ---------------------------------------------------- vector environment: auto-reset on the device
 * What gym_agario's AgarioEnv.step (AgarioEnv.py:77-112) adds around the step, for every instance, without the host reading
 * anything back, so the host can queue step t+1 while step t runs:
 *   done_out[i*A+a] = dones[i*A+a] | (max_steps > 0 && steps[i] >= max_steps)   (checked before the increment)
 *   reset_mask[i]   = any agent of i done;  steps[i] += 1;  then the instances in reset_mask are reset (same step: the
 *                     observation of a reset instance is the first of its new episode; rewards and done_out are the finished step's)
 * Episode statistics: per agent the f64 sum of the rewards since the instance's last reset, per instance its steps; where
 * reset_mask is set they are written to final_return / final_length and restart at 0.  Every reset, agarcl_batch_reset
 * included, restarts the counters of the instances it resets.
 *   agarcl_batch_reset_device   agarcl_batch_reset with mask[N] in DEVICE memory (NULL = all): no copy, no host loop, no wait.
 *   agarcl_batch_set_autoreset  enables the bookkeeping and allocates its buffers (synchronises the device; every instance's
 *                               counters start at 0).  max_steps 0: no step limit (continuing task).  keep_final_obs != 0: before
 *                               the reset, the observation images of the reset instances are copied to final_obs
 *                               [N*A, frames*C, G, G] (not with ram_obs = 2) and their ram records to final_ram [N, P,
 *                               AGARCL_RAM_RECORD] (cfg.ram_obs) -- as much memory again as the observation.  reset = 0:
 *                               bookkeeping only -- done_out and steps as above, nothing is reset, reset_mask stays 0 (requires
 *                               keep_final_obs = 0).  May be called again to change the settings.
 *   agarcl_batch_step_autoreset step, bookkeeping, final copy, masked reset, all enqueued on `stream`; AGARCL_ERR_STATE before
 *                               agarcl_batch_set_autoreset.  Under AGARCL_RNG_MT19937 the host reads the draw cursors back
 *                               now and then to refill the draw ring, as after any step or reset: the one wait that remains.
 *   agarcl_batch_episode        device pointers of the buffers below; each step_autoreset overwrites them.  The final_* entries
 *                               hold the last finished episode of each instance: read them where reset_mask is set.   */
typedef struct agarcl_episode {
  uint8_t* done_out;       /* u8 [N*A] */
  uint8_t* reset_mask;     /* u8 [N] */
  int64_t* steps;          /* [N] steps since the instance's last reset */
  double* final_return;    /* f64 [N*A] */
  int64_t* final_length;   /* [N] */
  void* final_obs;         /* observation dtype [N*A, frames*C, G, G]; NULL unless keep_final_obs and a grid observation */
  float* final_ram;        /* [N, P, AGARCL_RAM_RECORD]; NULL unless keep_final_obs and cfg.ram_obs */
} agarcl_episode;
int agarcl_batch_reset_device(agarcl_batch* b, const uint8_t* d_mask, void* stream);
int agarcl_batch_set_autoreset(agarcl_batch* b, int32_t max_steps, int32_t keep_final_obs, int32_t reset);
int agarcl_batch_step_autoreset(agarcl_batch* b, void* stream);
int agarcl_batch_episode(agarcl_batch* b, agarcl_episode* out);

/* ---------------------------------------------------- mixed-task batches: a game mode and an episode limit per instance
 * The mini-games of AgarCL differ in mode_number only (bench/tasks_configs: modes 1..10 at the same arena, pellets, viruses).
 * With cfg.task_modes != 0 every instance plays its own mode of that set and its own step limit, and changes them at its next
 * reset without the host waiting -- one batch for a multi-task policy or a curriculum instead of one batch per mode.
 * Layout: P = A + the most bots of any mode of the set (bots(0) = num_bots, bots(1..6) = 0, bots(7..10) = 1); cap_pellets the most
 * of any mode (the squared-pellet modes 1, 2 and 5 need 4 * (arena_size / 2)).  layout.mass_decay .. agent_mass and bot_type stay
 * those of mode_number: the kernels of a mixed batch derive the rules of each instance from its current mode.
 * ABSENT players: an instance of mode m plays P_m = A + bots(m) players; players P_m .. P-1 are never spawned, drawn for, ticked,
 * observed or counted -- from the reset on they are dead records (n_cells 0).  A reset draws 2 P_m spawn points and starts cell ids
 * at 1 + P_m, so an instance of mode m is bit-identical to the same instance (seed, global index, actions) of a batch of mode m alone.
 * Refused (AGARCL_ERR_INVALID) by agarcl_make_layout / agarcl_batch_create: strict_reference; a mode outside 0..10; mode_number not
 * in the set; mode 0 with a mode of another bot count (mode 0 respawns every dead player, absent ones included); a set where the
 * batch's player order, restricted to players < P_m, is not the order of a batch of mode m alone (cannot happen for one agent).
 * Task state, library-owned device arrays of N int32 (agarcl_batch_tasks):
 *   mode, max_steps             the current episode's task
 *   next_mode, next_max_steps   what the instance's next reset plays
 * Initially mode_number and -1.  A step limit of -1 means agarcl_batch_set_autoreset's max_steps, 0 no limit, > 0 that many
 * steps.  EVERY reset (agarcl_batch_reset, _reset_device, the reset inside _step_autoreset) copies next -> current for the
 * instances it resets before it spawns them: a running episode never changes its rules.
 *   agarcl_batch_set_tasks  d_mode[N] (device; -1 keeps the pending mode) and d_max_steps[N] (device, may be NULL: every pending
 *                           limit is kept) become the pending task.  Checked on the device; *d_result (may be NULL) receives the
 *                           library-owned u8 [N] result, overwritten by the next call: 0 nothing set, 1 set, 2 rejected (the mode
 *                           is not in task_modes or the limit is < -1: that instance's pending task is not touched).  Stream-
 *                           ordered, no host wait.  AGARCL_ERR_STATE on a batch without task_modes.
 *   agarcl_batch_tasks      the four device pointers; AGARCL_ERR_STATE on a batch without task_modes.
 * Snapshot pools store the source's current mode and max_steps (agarcl_snapshot_hdr.task_mode / task_max_steps); a restore makes
 * them the destination's current task (its pending task is untouched) and rejects a slot whose mode is not in the destination's
 * set.  agarcl_batch_save_env_state writes the instance's current mode as "mode_number"; agarcl_batch_load_env_state accepts any
 * mode of the set and makes it the instance's current task.                                                                    */
typedef struct agarcl_tasks {
  int32_t* mode;            /* [N] */
  int32_t* max_steps;       /* [N] */
  int32_t* next_mode;       /* [N] */
  int32_t* next_max_steps;  /* [N] */
} agarcl_tasks;
int agarcl_batch_set_tasks(agarcl_batch* b, const int32_t* d_mode, const int32_t* d_max_steps, uint8_t** d_result, void* stream);
int agarcl_batch_tasks(agarcl_batch* b, agarcl_tasks* out);
/* Game sizes per instance (mixed-task batch): three more task values with the lifecycle of mode / max_steps.
 *   bots      bot players of a mode-0 episode (modes 1..10 keep their own roster: none, or the one custom bot of 7..10)
 *   pellets   pellets spawned at the reset and the target of pellet regen (ignored by the squared-pellet modes 1, 2 and 5)
 *   viruses   viruses spawned at the reset and the target of virus regen (every mode)
 * cfg.num_bots, num_pellets and num_viruses are the MAXIMA: the layout is sized from them (P, cap_pellets, cap_viruses) as without
 * sizes, and current and pending sizes start at them, so a batch that never sets sizes plays exactly as before.  An instance with
 * current (mode, bots, pellets, viruses) is bit-identical to the same instance (seed, global index, actions) of a batch created with
 * mode_number = mode, num_bots = bots, num_pellets = pellets, num_viruses = viruses and the same cap_viruses.  A mode-0 instance
 * plays A + bots players; players A + bots .. P-1 are absent (never spawned, respawned, drawn for or ticked).
 * Allowed bot counts: 0 .. num_bots, every one of them when mode 0 is not in task_modes (the count then means nothing, and num_bots
 * may exceed the players of the layout); when mode 0 is in task_modes only those whose A + bots players keep the player-order check
 * above (the batch's order restricted to players < A + bots is the order of a batch of A + bots players alone).  Not every count
 * passes, even for one agent: with 1 agent and 25 bots the counts 1 .. 12 fail (the unordered_map rehashes between 13 and 26
 * players), and 0 and 13 .. 25 pass.
 *   agarcl_batch_set_task_sizes  d_bots, d_pellets, d_viruses: device int32 [N] each, or NULL to keep every pending value; an entry
 *                                of -1 keeps that value.  Checked on the device; *d_result (may be NULL) receives the library-owned
 *                                u8 [N] result, overwritten by the next call: 0 nothing set, 1 set, 2 rejected (a value outside
 *                                [0, maximum] or a bot count that is not allowed: none of that instance's pending sizes is touched).
 *                                Stream-ordered, no host wait.  AGARCL_ERR_STATE on a batch without task_modes.
 *   agarcl_batch_task_sizes      the six device pointers; AGARCL_ERR_STATE on a batch without task_modes.
 * Every reset copies the pending sizes to the current ones together with the mode.  Snapshot slots of a mixed batch carry the
 * source's current sizes (agarcl_snapshot_hdr.sizes_marker = AGARCL_SNAPSHOT_SIZES_MARKER, task_bots / task_pellets /
 * task_viruses); a restore or a start-state reset makes them current, and rejects (result 2) a slot whose sizes exceed the
 * destination's maxima or whose bot count the destination does not allow.  A slot without the marker restores with the maxima.
 * agarcl_batch_save_env_state writes the instance's current num_bots / num_pellets / num_viruses; agarcl_batch_load_env_state
 * accepts any within the maxima (and an allowed bot count) and makes them current; the num_bots of a file whose mode_number is not 0
 * is not checked, and the instance's bot count becomes the maximum. */
typedef struct agarcl_task_sizes {
  int32_t* bots;          /* [N] */
  int32_t* pellets;       /* [N] */
  int32_t* viruses;       /* [N] */
  int32_t* next_bots;     /* [N] */
  int32_t* next_pellets;  /* [N] */
  int32_t* next_viruses;  /* [N] */
} agarcl_task_sizes;
int agarcl_batch_set_task_sizes(agarcl_batch* b, const int32_t* d_bots, const int32_t* d_pellets, const int32_t* d_viruses,
                                uint8_t** d_result, void* stream);
int agarcl_batch_task_sizes(agarcl_batch* b, agarcl_task_sizes* out);

/* ---------------------------------------------------- snapshot pools: save and restore game states on the device
 * The batched counterpart of agarcl_batch_save_env_state / load_env_state: chosen instances are copied into slots of a
 * caller-owned POOL in device memory and slots back into chosen instances, stream-ordered, driven by index arrays in device
 * memory, without the host waiting.  A pool is pool_slots slots of agarcl_snapshot_slot_bytes bytes (16-byte aligned device
 * memory of cfg.device).  A slot holds no pointer: a pool may be copied to the host, stored, moved to another device and
 * restored into any batch of the same configuration -- n_instances, device, instance_base and cap_replay may differ.
 * Slot layout, every segment 16-byte aligned (S = layout.stride, A agents, P players, esz 4 for int32 and 2 for int16):
 *   [0, 64)               agarcl_snapshot_hdr below
 *   [64, 64 + S)          the state blob: it includes hdr.rng_cursor, the seed, the tick, done_sticky and the respawn mask
 *   off_ep  = 64 + S      episode record, E = align16(8 + 8 A) bytes: int64 steps, then f64 return[A] since the instance's last
 *                         reset (agarcl_batch_set_autoreset); zeros when the bookkeeping was off at the save, and written on a
 *                         restore only when it is on
 *   off_ram = off_ep + E  cfg.ram_obs: the ram records [P][AGARCL_RAM_RECORD] f32, R = P * 4 * AGARCL_RAM_RECORD bytes (copied, not
 *                         re-rendered: a player with nothing in view keeps its previous record), else R = 0
 *   off_obs = off_ram + R num_frames > 1 and a grid observation: the instance's images [A][frames*C][G][G], O = align16(A * frames *
 *                         C * G * G * esz) bytes (the earlier frames are history the blob does not hold), else O = 0
 *   slot bytes            align128(off_obs + O)
 * A one-frame grid observation is not stored: the restore ends with k_obs on the restored instances, showing players respawned at
 * the end of the last step as still dead -- the frame the step that produced the state showed (after a reset: the reset's).  A
 * state saved right after agarcl_batch_render therefore comes back with the step's frame, not render()'s.
 *   agarcl_batch_save_states     for k < n: slot d_slot[k] (d_slot NULL: slot k) <- instance d_src[k].  Slots out of
 *                                [0, pool_slots) are skipped; a source out of [0, N) writes a header with magic 0, which a restore
 *                                rejects.  The slots of one call must be distinct.
 *   agarcl_batch_restore_states  for every instance i with d_slot_of[i] >= 0 (N entries): instance i <- that slot.  *d_result (may
 *                                be NULL) receives the library-owned u8 [N] result, overwritten by the next restore:
 *                                0 not requested, 1 restored, 2 rejected (slot out of [0, pool_slots), or magic, version,
 *                                fingerprint or slot bytes differ): a rejected or unrequested instance is not touched, bit for bit.
 *                                A restored instance's rewards and dones are zeroed, like after a reset; the reset_mask and done_out
 *                                of the last agarcl_batch_step_autoreset are left as they are.  As after a reset, call
 *                                agarcl_batch_sync_mirror before the next agarcl_batch_step_mirror.
 * Fork = save once, then restore with several instances naming the same slot.
 * Draw stream: the restore writes the instance's seed from the restored blob and marks the stream as not fresh, so its next reset
 * continues the restored stream.  Under AGARCL_RNG_PHILOX the stream is keyed by (seed, global instance index, cursor): a state
 * restored into an instance whose instance_base + i equals the source's global index reproduces the source's future exactly;
 * restored anywhere else it continues on the destination's key and diverges from the source at its first draw (pellet regen,
 * respawn) -- forked children that receive identical actions still differ where the game draws.
 * Refused with an error before anything is enqueued (the games do not move): strict_reference (the player order belongs to the
 * batch and changes with every unmasked reset), AGARCL_RNG_MT19937 (its generators live on the host), a call before the first
 * reset, a NULL / misaligned pool or one that is not device memory of cfg.device, pool_slots < 1, n < 0, a NULL index array.
 * The fingerprint is FNV-1a 64 over agarcl_layout without cap_replay and the agarcl_cfg fields num_agents .. ram_obs except
 * cap_viruses, cap_foods, cap_replay, device and instance_base (those two caps are part of the layout), then task_modes when it
 * is not 0.  A mixed-task batch: the header also carries the source's task, and a slot whose task_mode is not in the
 * destination's task_modes is rejected. */
#define AGARCL_SNAPSHOT_MAGIC 0x4E534741u /* "AGSN" */
#define AGARCL_SNAPSHOT_VERSION 1u
typedef struct agarcl_snapshot_hdr { /* 64 B */
  uint32_t magic;          /* AGARCL_SNAPSHOT_MAGIC; 0: the slot holds no state */
  uint32_t version;        /* AGARCL_SNAPSHOT_VERSION */
  uint64_t fingerprint;    /* of the configuration the slot was saved from */
  uint64_t slot_bytes;
  int32_t source;          /* global index (instance_base + i) of the instance saved */
  int32_t task_mode;       /* mixed-task batch (cfg.task_modes != 0): the source's current mode; 0 otherwise */
  int32_t task_max_steps;  /* mixed-task batch: the source's current step limit (-1 default, 0 none); 0 otherwise */
  uint32_t sizes_marker;   /* mixed-task batch: AGARCL_SNAPSHOT_SIZES_MARKER when the three sizes below are stored; 0 otherwise */
  int32_t task_bots;       /* mixed-task batch: the source's current game sizes (agarcl_batch_set_task_sizes); 0 otherwise */
  int32_t task_pellets;
  int32_t task_viruses;
  uint32_t pad[3];
} agarcl_snapshot_hdr;
#define AGARCL_SNAPSHOT_SIZES_MARKER 0x5A534741u /* "AGSZ" */
/* bytes of one snapshot slot of configuration c: a multiple of 128; no device needed */
int agarcl_snapshot_slot_bytes(const agarcl_cfg* c, int64_t* out);
/* pool slot d_slot[k] <- instance d_src[k], k < n (device int32 arrays; d_slot NULL = slots 0..n-1); enqueued on stream */
int agarcl_batch_save_states(agarcl_batch* b, void* pool, int64_t pool_slots, const int32_t* d_src, const int32_t* d_slot,
                             int32_t n, void* stream);
/* instance i <- pool slot d_slot_of[i] where >= 0; *d_result = the library-owned u8 [N] result above; enqueued on stream */
int agarcl_batch_restore_states(agarcl_batch* b, const void* pool, int64_t pool_slots, const int32_t* d_slot_of,
                                uint8_t** d_result, void* stream);
/* Start states: episodes that begin in saved games (a Go-Explore return, start-state curricula, evaluation on fixed start
 * positions, continual runs that begin mid-game).  A batch may hold a START-STATE TABLE: a pool and a start slot per instance.
 * EVERY reset (agarcl_batch_reset, _reset_device, the reset inside _step_autoreset) of an instance whose start slot is >= 0 is a
 * reset whose spawn is replaced by the slot's game:
 *   game          the instance's blob becomes the slot's blob (tick, cells, timers, flags, done_sticky, player records)
 *   draw stream   it goes on where a spawn would have drawn first: hdr.seed = the instance's seed, hdr.rng_cursor = 0 when the
 *                 stream is fresh (seeded since its last reset), else the instance's cursor before the reset; the stream is then
 *                 no longer fresh.  Successive episodes from one slot, and instances started from one slot, differ where the game
 *                 draws; a slot's own stream is never reused.  hdr.respawned_lo / respawned_hi are cleared, as by a reset.
 *   around it     exactly what a reset does: dones zeroed (rewards are not: step_autoreset returns the finished step's), episode
 *                 counters restarted, ram records cleared, a grid observation cleared and rendered (pre_respawn 0) or the
 *                 pictures drawn; with keep_final_obs the final observation is copied before the reset, as always.
 *   ignored       the slot's episode record, ram records, observation history and source.
 *   mixed tasks   the slot's task_mode becomes the current mode (the game belongs to it); the current step limit is the PENDING
 *                 one (next_max_steps: the limit belongs to the episode); the pending mode is left as it is.
 * A slot is checked as agarcl_batch_restore_states checks it (range, magic, version, fingerprint, slot bytes, a mode of the set);
 * an instance whose slot fails is spawned exactly as without a table, and reported.  Instances with start slot -1 (any negative
 * value), and every reset of a batch without a table, are untouched: game, stream, observation and counters bit for bit those of
 * a spawn.  A reset with a table is one more launch (k_start_states, one CTA per instance) in front of k_reset.
 *   agarcl_batch_set_start_states  pool NULL: no table (every reset spawns).  d_start_slot: device int32 [N], copied on `stream`
 *                                  into a library-owned array (the caller may reuse its buffer).  The pool pointer is kept: it
 *                                  must stay allocated while it is set, and slots saved into it later are read as they are when
 *                                  a reset runs (stream order).  May be called before the first reset.  Refused with an error,
 *                                  the table left as it was: strict_reference, AGARCL_RNG_MT19937, a misaligned pool or one that
 *                                  is not device memory of cfg.device, pool_slots < 1, a NULL d_start_slot with a pool.
 *   agarcl_batch_start_result      the library-owned u8 [N] result of the latest reset with a table: 0 not reset or spawned with
 *                                  slot -1, 1 started from its slot, 2 slot rejected -> spawned fresh.  The restore result is
 *                                  not touched by resets. */
int agarcl_batch_set_start_states(agarcl_batch* b, const void* pool, int64_t pool_slots, const int32_t* d_start_slot, void* stream);
int agarcl_batch_start_result(agarcl_batch* b, uint8_t** d_result);

/* Go-Explore cell archive: every agarcl_batch_step_autoreset files each game under its CELL and keeps, per cell, the best game
 * seen in a snapshot slot; with select = 1 every reset returns to a chosen cell.  A Go-Explore loop is then step_autoreset in a
 * loop: the host never waits and writes no archive code.
 *   agarcl_batch_set_archive  attaches an archive of K = pool_slots entries to the batch; entry e is slot e of `pool` (caller-
 *                             owned, the slot format above, kept while attached).  Attaching clears the archive (nothing is read
 *                             from the pool); it allocates and synchronises the device.  pool NULL detaches it.
 *   agarcl_batch_archive      device pointers of the arrays below; nothing of the archive is ever read back by the host.
 * CELL of instance i after a step, for agent a = cfg.agent: none (-1) if the agent has no cells.  Otherwise m = the u32 total
 * mass of its cells and (cx, cy) its centroid exactly as the agent view of agarcl_batch_draw defines it (fp32, cell order);
 * bx = clamp((int)(cx * (float)n / W), 0, n - 1), by the same with cy (each operation one rounded fp32 operation, no FMA, the
 * conversion truncates); mb = 31 - clz(m); key = (mb * n + by) * n + bx in [0, 32 n^2).
 * CANDIDATES: instance i is one when it has a cell and no agent of it is done by the game in this step (agarcl_batch_dones,
 * before the step limit: an instance truncated by the limit is still a candidate).  Its trajectory score is s_i =
 * base_score[i] + (return[a] + reward[a]) (f64: the agent's episode return including this step's reward), its trajectory
 * length l_i = base_length[i] + (steps + 1) (i64).  Every candidate adds 1 to visits[key].
 * UPDATE, once per step_autoreset, behind the step and in front of the episode bookkeeping (it sees the games before any reset):
 *   winner     per key with candidates: the highest s, then the lowest l, then the lowest instance index
 *   new key    gets the next entry if fewer than K are in use; the entries created in one step are numbered after those in
 *              use, in ascending order of their winner's instance.  When the archive is full the discovery is counted in
 *              `dropped` and nothing is stored (its visits still count)
 *   known key  its entry is replaced when s > score, or s == score and l < length; each replacement counts in `improved`
 *   stored     a new or replaced entry takes (key, s, l), and the winner's game is saved into slot e exactly as
 *              agarcl_batch_save_states would save it at that moment (header, blob, ram records, observation history; the
 *              episode record holds the counters before this step's bookkeeping, and start states ignore it)
 *   cell_of[i] the key, or -1: what a count-based exploration bonus reads (visits[cell_of])
 * SELECTION (select = 1): the archive owns the start-state table (agarcl_batch_set_start_states returns AGARCL_ERR_STATE), and at
 * every reset (agarcl_batch_reset, _reset_device, the reset inside _step_autoreset) each reset instance i draws an entry:
 *   weight     w_e = floor(2^20 / (1 + isqrt(chosen_e))) for the entries in use (Go-Explore's 1 / sqrt(C + 1) in integers), from
 *              the counts before this reset; W = sum of w_e (u64)
 *   draw       Philox4x32-10 (the spawn generator) with key = (seed low, seed high word) and counter = (c_i, 0x41524348,
 *              instance_base + i, 0), c_i = the draws instance i made before; x = word 0 | word 1 << 32; the pick is the first e
 *              in entry order whose inclusive prefix sum of weights exceeds x mod W.  After the picks of the reset every
 *              chosen_e grows by the instances that picked it.  With an empty archive the instance spawns (no draw).
 *   start      the instance starts from slot e as start states define it (agarcl_batch_start_result reports it)
 * With select = 0 the start-state table stays the caller's (a caller may fill it from the read-out).
 * TRAJECTORY BASE: a reset instance that starts from a slot of the archive's pool (result 1, the slot an entry in use) gets
 * base = (score_e, length_e) as they are at that reset; any other reset instance -- spawned, rejected, started from another pool --
 * and every instance agarcl_batch_restore_states restores gets (0, 0).  Every launch is stream-ordered; no host wait.
 * Refused with an error before anything is enqueued, the archive left as it was: strict_reference, AGARCL_RNG_MT19937, a
 * mixed-task batch (task_modes != 0: a reset would need one selection per pending mode; not supported), a call before
 * agarcl_batch_set_autoreset or with its reset = 0 (agarcl_batch_set_autoreset(reset = 0) is refused while one is attached),
 * cells_per_side outside [1, 256], agent outside [0, A), select not 0 or 1, a pool that is misaligned or not device memory of
 * cfg.device, pool_slots < 1 or > 65536 (the selection scans the weights in one CTA).
 * A batch without an archive launches nothing new.  With one, step_autoreset adds k_archive_cells, k_archive_commit and the save
 * (k_snapshot, one CTA per instance: those of the non-winners exit at once), every reset k_archive_base, and with select = 1
 * k_archive_select (one CTA; it exits at once when nothing resets) and k_start_states. */
typedef struct agarcl_archive_cfg {
  int32_t cells_per_side;  /* n, 1..256 */
  int32_t agent;           /* whose cell it is, 0..A-1 */
  int32_t select;          /* 1: the archive chooses the start slot of every reset; 0: the caller's start-state table */
  int32_t pad;
  uint64_t seed;           /* Philox key of the selection */
} agarcl_archive_cfg;
typedef struct agarcl_archive {
  int32_t* cell_of;        /* [N] key of the instance's cell after the last step, -1: none */
  double* base_score;      /* [N] trajectory base of the running episode */
  int64_t* base_length;    /* [N] */
  int32_t* key_entry;      /* [32 n^2] entry of a key, -1: none */
  uint32_t* visits;        /* [32 n^2] candidates seen in the key */
  int32_t* entry_key;      /* [K] key of entry e (entries [0, used) are in use) */
  double* entry_score;     /* [K] best trajectory score of the cell */
  int64_t* entry_length;   /* [K] its trajectory length */
  uint32_t* entry_chosen;  /* [K] selections of the entry */
  uint64_t* counters;      /* [3] used, dropped, improved */
  int64_t keys, entries;   /* 32 n^2, K */
} agarcl_archive;
int agarcl_batch_set_archive(agarcl_batch* b, void* pool, int64_t pool_slots, const agarcl_archive_cfg* cfg);
int agarcl_batch_archive(agarcl_batch* b, agarcl_archive* out);

/* ---------------------------------------------------- pictures of game states, for people (render() and videos)
 * A picture is uint8 [S][S][3], RGB, row-major (HWC): row r is world y, column c world x, row 0 the smallest y.  S is a multiple of
 * 16 in [16, 2048].  It is drawn from the state blob as it is at the call: players respawned at the end of the last step are drawn
 * at their new cells.  It is not a training observation and claims no likeness to the reference's OpenGL frames; this spec is
 * what it means, and tests/draw_oracle.c (oracle_draw) restates it.  The training observation is cfg.pixel_obs below.
 * Views (every operation one rounded fp32 operation, no FMA, C order of evaluation):
 *   AGARCL_DRAW_ARENA  the arena [0, W)^2, W = (float)arena_size: pixel centre x = ((float)c + 0.5f) * W / (float)S, y the same
 *                      with r; pixel width px = W / (float)S.
 *   AGARCL_DRAW_AGENT  the window of the agent's grid observation: its centroid (cx, cy) as k_obs computes it (sum over its cells in
 *                      cell order of x * (float)mass, over (float)(total mass)), view = clamp(2 * total mass, 100, 300);
 *                      x = cx + ((float)c - (float)(S / 2.0)) * view / (float)S (GridObservation's _grid_to_world: corners), y the
 *                      same with r; px = view / (float)S.  With S = G the out-of-arena pixels are exactly the -1 elements of
 *                      observation channel 0, transposed.  A dead agent (no cells: NaN centroid) is all out-of-arena colour.
 * Colour of a pixel at (x, y):
 *   !(0 <= x < W && 0 <= y < W)  AGARCL_DRAW_RGB_OUT
 *   otherwise                    the colour of the TOPMOST entity whose disc contains it, else AGARCL_DRAW_RGB_BACKGROUND.
 *   disc test: dx = x - ex, dy = y - ey, dx * dx + dy * dy <= R * R; drawn radius R = max(radius(mass), px), radius(m) =
 *   (float)sqrt((double)m / M_PI) (radius_conversion); pellets have mass AGARCL_PELLET_MASS, foods AGARCL_FOOD_MASS.  Cells and
 *   viruses show their border colour where d2 > (0.85f * R) * (0.85f * R).
 * Draw order, bottom to top: pellets in array order, foods in array order, then cells and viruses together by the key (mass, kind
 * [virus 0, cell 1], cell id or virus index) ascending.  Counts are taken from the header and player records, limited to the
 * layout's capacities (cap_pellets, cap_foods, cap_viruses, cap_cells); dead and absent players have no cells and draw nothing.
 * Cell colours: player p < A (an agent) AGARCL_DRAW_RGB_AGENTS[p % 8]; a bot AGARCL_DRAW_RGB_BOTS[bot_type & 3] (the player
 * record's bot_type); border = each channel * 3 / 4 (integer).  A picture whose source is out of range is all zeros.
 *   agarcl_batch_draw  n pictures [n][size][size][3] into d_out (caller-owned, 16-byte aligned device memory of cfg.device),
 *                      enqueued on stream, no host wait, the state only read.  d_src[k] (device int32): arena view an instance in
 *                      [0, N); agent view an image instance * A + agent in [0, N * A), the observation's numbering.  d_src NULL:
 *                      picture k shows source k (n = N, or N * A, draws them all).  Refused before anything is enqueued, nothing
 *                      written: a call before the first reset (AGARCL_ERR_STATE), an unknown view, a size that is not a multiple
 *                      of 16 in [16, 2048], n < 0, a NULL or misaligned d_out or one that is not device memory of cfg.device. */
#define AGARCL_DRAW_ARENA 0
#define AGARCL_DRAW_AGENT 1

/* ---------------------------------------------------- the pixel observation (cfg.pixel_obs = S): pictures for training
 * A batch created with pixel_obs = S renders, after every step, reset and restore, the picture of every agent uint8
 * [N*A, S, S, 3] (image instance * A + agent) in library-owned device memory, in place of the grid frame.  Picture j is what
 * agarcl_batch_draw(AGARCL_DRAW_AGENT, S) would draw, with one difference: players respawned at the end of the step that
 * produced the state are drawn as still dead (no cells), and an agent that was respawned is therefore a dead agent whose
 * every pixel is AGARCL_DRAW_RGB_OUT.  The picture shows the same moment as the grid observation the step would have
 * produced.  Equivalently: oracle_draw(AGARCL_DRAW_AGENT, S) on the instance's blob after setting n_cells = 0 for the players
 * in hdr.respawned_lo / respawned_hi (a reset clears that mask; a restore keeps the saved one).
 *   reset          the pictures of the instances it resets (masked: only those); the others are not touched
 *   restore        the pictures of the restored instances; snapshot slots hold no pictures (they are re-rendered, never
 *                  stored), so slot bytes and fingerprints are those of the same configuration without pixel_obs, and a pool
 *                  moves between a pixel batch and a grid batch of the same game both ways
 *   step_autoreset with keep_final_obs, the pictures of the instances it resets are first copied to final_pixels, as final_obs
 * agarcl_batch_pixels: device pointers of the pictures and of the final pictures (NULL unless keep_final_obs) and their shape
 * {N*A, S, S, 3}; AGARCL_ERR_STATE on a batch without pixel_obs.  The host paths of the grid observation
 * (agarcl_batch_step_host, _step_mirror, _step_lists, _sync_mirror) refuse a pixel batch with AGARCL_ERR_STATE. */
int agarcl_batch_pixels(agarcl_batch* b, uint8_t** d_pixels, uint8_t** d_final_pixels, int64_t shape[4]);
#define AGARCL_DRAW_RGB_OUT 0x2B2B33u
#define AGARCL_DRAW_RGB_BACKGROUND 0xF4F6F8u
#define AGARCL_DRAW_RGB_PELLET 0x8CCB5Eu
#define AGARCL_DRAW_RGB_FOOD 0xE8A33Du
#define AGARCL_DRAW_RGB_VIRUS 0x3DBB4Fu
#define AGARCL_DRAW_RGB_VIRUS_BORDER 0x1E7A2Cu
#define AGARCL_DRAW_RGB_AGENTS {0x2F6FDEu, 0xD9413Bu, 0x8E44ADu, 0x16A3A3u, 0xE67E22u, 0xC0398Eu, 0x5D6D7Eu, 0x9C7A1Eu}
#define AGARCL_DRAW_RGB_BOTS {0x7F8C8Du, 0xA3B1C2u, 0x8B5A3Cu, 0xB86F8Fu}
int agarcl_batch_draw(agarcl_batch* b, int32_t view, int32_t size, const int32_t* d_src, int32_t n, uint8_t* d_out, void* stream);

/* ---------------------------------------------------- built-in bot policies for agents: scripted actions on the device
 * The four bots of the reference (agario/bots/HungryBot.hpp, HungryShyBot.hpp, AggressiveBot.hpp, AggressiveShyBot.hpp) as a
 * policy for the agents: for baselines, expert actions for imitation, and scripted partners or opponents of a learner.
 * For every agent j = i * A + a with d_type[j] in 0..3, what Bot::take_action of that bot type would leave in agent a's player
 * record (target_x, target_y, action), on instance i's state as it is at the call: exactly oracle.c's bot_take_action run on
 * player a with bot_type = d_type[j], and so:
 *   - Hungry: action 0, the nearest pellet.  HungryShy: action 0; flee from the first player (other than a) in the order below
 *     whose centre lies at distance < 25, whatever its mass (the template compares against a mass of 0, see oracle.c's bot_flee),
 *     target = loc - (other - loc); else the nearest pellet.  Aggressive: chase the first player in the order at distance <= 20
 *     that has a cell the agent's largest cell can eat (Cell::can_eat), target = loc + 3 * (mass-weighted centre of those cells
 *     - loc), the action left as it is; else action 0 and the nearest pellet.  AggressiveShy: flee (action left as it is), else
 *     chase, else action 0 and the nearest pellet.
 *   - players are visited in the batch's current layout.order (strict_reference: the order after the latest unmasked reset).
 *     A dead player, and an absent player of a mixed-task batch, has no cells: its location is NaN and fails every test.
 *   - the nearest pellet is the first strict minimum in array order of sqrtf(dx * dx + dy * dy) among the pellets with
 *     (double)d > 0.01; (0, 0) when no pellet qualifies.
 *   - locations are Player::x / y: fp32 sums of x * (float)mass in cell order over (float)(total mass).
 * Nothing of the state is written: no target, no action, no flag.  Outputs, caller-owned device memory of cfg.device:
 *   d_dxdy    f32 [N*A][2]  (target - loc) / 10 in fp32, the inverse of agarcl_batch_set_actions' target = loc + 10 * dxdy.  Not
 *                           clamped to [-1, 1] (a pellet 60 units away gives 6): the step accepts it, and clamping would change
 *                           the speed, which is 3 * (target - cell) capped at max_speed.
 *   d_act     i32 [N*A]
 *   d_target  f32 [N*A][2]  the world target (may be NULL)
 *   d_status  u8  [N*A]     (may be NULL) AGARCL_BOT_*:
 *     SKIPPED    0  d_type[j] == -1: nothing but the status is written for j (fill only the scripted agents of an action
 *                   buffer that a policy already wrote)
 *     DECIDED    1
 *     NO_PELLET  2  the nearest pellet was needed and there is none (the reference would call std::rand(), Bot.hpp:93-97):
 *                   dxdy 0, target = loc, act 0; no state flag is raised
 *     DEAD       3  the agent has no cells: dxdy 0, act 0, target (0, 0) (takes precedence over NO_PELLET)
 *     BAD_TYPE   4  d_type[j] outside -1..3: nothing but the status is written for j
 * Stream-ordered, no host wait, can be captured in a CUDA graph (the player order is taken at the call).  Refused before anything
 * is enqueued: a call before the first reset (AGARCL_ERR_STATE); a NULL d_type, d_dxdy or d_act; an array that is not device
 * memory of cfg.device; d_dxdy or d_target not 8-byte aligned.                                                                  */
#define AGARCL_BOT_HUNGRY 0
#define AGARCL_BOT_HUNGRY_SHY 1
#define AGARCL_BOT_AGGRESSIVE 2
#define AGARCL_BOT_AGGRESSIVE_SHY 3
#define AGARCL_BOT_SKIPPED 0
#define AGARCL_BOT_DECIDED 1
#define AGARCL_BOT_NO_PELLET 2
#define AGARCL_BOT_DEAD 3
#define AGARCL_BOT_BAD_TYPE 4
int agarcl_batch_bot_actions(agarcl_batch* b, const int32_t* d_type, float* d_dxdy, int32_t* d_act, float* d_target,
                             uint8_t* d_status, void* stream);

/* ---------------------------------------------------- host-resident observation mirror
 * get_state (bindings.cpp:67-91) hands every agent's frame to HOST memory; for a batch that is 512 KB per agent
 * per step, and the dense copy above is bound by PCIe.  The mirror is a library-owned, pinned host tensor
 * [N*A, C*num_frames, G, G] of the observation dtype that the library keeps IDENTICAL to the device observation
 * while moving only what a grid observation really contains: per frame the row/column bit masks of the
 * out-of-bounds channel (GridEnvironment.hpp:235-248) and the (offset, value) list of the few hundred non-zero
 * elements of the other channels (:212-232).  Host threads undo the previous step's list, patch the mask rows /
 * columns that changed and store the new list.  Images that do not fit the scheme are copied densely, so the
 * result never depends on it.  The caller reads the mirror and must not write to it.
 *   agarcl_batch_mirror       creates the mirror on first use, syncs it, returns the host pointer (stable).
 *   agarcl_batch_sync_mirror  brings it up to date with the current device observation (after a reset, a
 *                             render, or agarcl_batch_step); synchronises `stream`.
 *   agarcl_batch_step_mirror  = take_actions (host) + step + sync_mirror + rewards/dones to host: the
 *                             reference-facing call `e2e` in bench.py times.  When the step is the single fused
 *                             kernel (int32, one frame) that kernel lists what it scatters itself and flags
 *                             finished chunks of instances in host-mapped memory, so the host fetches and
 *                             expands chunk k while the device still steps chunk k+1.
 *   agarcl_batch_mirror_stats out[0] entries moved by the last sync, [1] images copied densely, [2] bytes copied
 *                             device->host, [3] host threads.                                                  */
int agarcl_batch_mirror(agarcl_batch* b, void** host_ptr, int64_t shape[4], int32_t* dtype);
int agarcl_batch_sync_mirror(agarcl_batch* b, void* stream);
int agarcl_batch_step_mirror(agarcl_batch* b, const float* dxdy, const int32_t* act, double* rewards_out, uint8_t* dones_out);
int agarcl_batch_mirror_stats(const agarcl_batch* b, uint64_t out[4]);
/* last agarcl_batch_step_mirror, microseconds: out[0] the calling thread waiting for the device (chunk flags, list
 * copies), out[1] first wait to mirror complete, out[2] action staging + kernel launch, out[3] the whole call. */
int agarcl_batch_mirror_timing(const agarcl_batch* b, uint64_t out[4]);

/* ---------------------------------------------------- the observation as LISTS (zero-copy, no dense host tensor)
 * A grid observation is almost entirely structure: per frame the out-of-bounds channel is a row mask and a column mask
 * (GridEnvironment.hpp:235-248) and the other channels hold a few dozen non-zero elements (:212-232).  The step kernel
 * writes exactly that -- per image a record and a list of integer operations -- straight into pinned host memory while it
 * runs; the dense mirror above is those lists replayed by host threads, which is what stops scaling when 8 GPUs feed one
 * host (DESIGN.md 3b).  agarcl_batch_step_lists hands the lists themselves to the caller: take_actions (host) + step +
 * rewards / dones to host, observation left in library-owned pinned memory as described by agarcl_obs_lists, valid until
 * the next step call on the batch.  A learner expands them where it trains (one scatter per image) or consumes them as
 * they are; agarcl_batch_lists_expand is the reference decoder for one image.  Requires the configuration whose step is
 * the single fused kernel (one frame, strict_reference = 0); AGARCL_ERR_STATE otherwise.
 *   chunk c                = chunks + c * chunk_words                     (32-bit words)
 *   slot s (of n_images)   : chunk s / images_per_chunk, index li = s % images_per_chunk inside it; slot_of[image] = s
 *   record of the slot     = chunk + off_rec + li * rec_words :
 *        [0] entries (0xFFFFFFFF: the image overflowed entries_per_image -> read it from agarcl_batch_obs)
 *        [1] index of its first entry in the chunk's entry array   [2] the image (instance * agents + agent)
 *        [3 ..] per frame: mask_words words of ROW bits (bit i: row i of channel 0 is -1), then mask_words of COLUMN bits
 *        [rec_words-3, -2] the agent's reward (f64)   [rec_words-1] its done flag
 *   entries of the chunk   = (uint32 pairs) chunk + off_entries : (op << 29 | element offset inside the image, operand), applied in
 *        order onto a zero frame: op 0 x = v, 1 x += v, 2 x = (x != 0 && x < v) ? x : v, 3 x = max(x, v); int16 saturates at 32767 */
typedef struct agarcl_obs_lists {
  int32_t n_images, n_chunks, images_per_chunk, frames, channels, grid, obs_dtype;
  int32_t mask_words, rec_words, entries_per_image;
  uint32_t off_rec, off_entries, chunk_words;
  const uint32_t* chunks;   /* pinned host memory */
  const uint32_t* slot_of;  /* [n_images] */
} agarcl_obs_lists;
int agarcl_batch_step_lists(agarcl_batch* b, const float* dxdy, const int32_t* act, double* rewards_out, uint8_t* dones_out,
                            agarcl_obs_lists* out);
/* Decodes image `image` of the lists of the last agarcl_batch_step_lists into dense_out ([frames*C, G, G] of the observation
 * dtype, host memory); an image that overflowed its slot is copied from the device tensor instead. */
int agarcl_batch_lists_expand(agarcl_batch* b, int32_t image, void* dense_out);

/* ---------------------------------------------------- structured ("ram") observation
 * GoBiggerObservation::add_frame (environment/envs/GoBiggerEnvironment.hpp:515-548, _store_entities
 * 446-513): for EVERY player of the instance, the in-view viruses, pellets ("food"), ejected foods
 * ("spores") and the player's own cells ("clones"), player-relative, in entity index order — what
 * agarcl.GoBiggerEnvironment.get_state() (environment/bindings.cpp:28-47,323-374) hands out as
 * PlayerState objects.  Here one player is one fixed-size float32 record, zero padded:
 *   hdr   [8]      n_food, n_virus, n_spore, n_clone (true in-view counts), score (= player mass),
 *                  player x, player y, overflow mask (bit0 food, bit1 virus, bit2 spore, bit3 clone)
 *   food  [KP][4]  dx, dy, radius, score            (FoodInfo)
 *   virus [KV][4]  dx, dy, radius, score            (VirusInfo; its velocity is the constant (0,0))
 *   spore [KS][4]  dx, dy, radius, score            (SporeInfo; velocity (0,0), owner = this player)
 *   clone [KC][8]  dx, dy, radius, score, vx, vy, direction, owner   (CloneInfo; teamId is always 0)
 * A player with nothing in view (a dead one) keeps its previous record, like the reference, whose
 * PlayerState is only committed when an entity lands inside the grid (:495-509).  reset() clears.   */
#define AGARCL_RAM_HDR 8
#define AGARCL_RAM_KP 192
#define AGARCL_RAM_KV 16
#define AGARCL_RAM_KS 32
#define AGARCL_RAM_KC 32
#define AGARCL_RAM_OFF_FOOD AGARCL_RAM_HDR
#define AGARCL_RAM_OFF_VIRUS (AGARCL_RAM_OFF_FOOD + 4 * AGARCL_RAM_KP)
#define AGARCL_RAM_OFF_SPORE (AGARCL_RAM_OFF_VIRUS + 4 * AGARCL_RAM_KV)
#define AGARCL_RAM_OFF_CLONE (AGARCL_RAM_OFF_SPORE + 4 * AGARCL_RAM_KS)
#define AGARCL_RAM_RECORD (AGARCL_RAM_OFF_CLONE + 8 * AGARCL_RAM_KC) /* 1224 floats per player */
/* Device pointer to the records [N, P, AGARCL_RAM_RECORD] float32 (cfg.ram_obs must be 1). */
int agarcl_batch_ram(agarcl_batch* b, float** dev_ptr, int64_t shape[3]);
/* get_state() of agarcl.GoBiggerEnvironment (bindings.cpp:28-47) with a HOST buffer: all records [N, P, AGARCL_RAM_RECORD]
 * copied out (synchronises the device). */
int agarcl_batch_ram_host(agarcl_batch* b, float* out);
/* Run only the structured-observation kernel on the current state (tests). */
int agarcl_batch_render_ram(agarcl_batch* b, void* stream);

/* Parity / snapshot transport: one instance's blob (layout.stride bytes) to / from host memory. */
int agarcl_batch_download_state(agarcl_batch* b, int32_t instance, void* blob);
int agarcl_batch_upload_state(agarcl_batch* b, int32_t instance, const void* blob);
/* BaseEnvironment::save_env_state / load_env_state (environment/envs/BaseEnvironment.hpp:213-343,
 * agario/engine/Engine.hpp:247-348; bound at bindings.cpp:135,170,374): one instance to / from the
 * reference's JSON snapshot.  The reference format is lossy (no splitting velocity, recombine timers, virus
 * food hits, tick): those travel as extra keys the reference ignores and are restored with lossless != 0.
 * After a load the instance's draw stream restarts from the snapshot's seed, like Engine::seed there.   */
int agarcl_batch_save_env_state(agarcl_batch* b, int32_t instance, const char* path);
int agarcl_batch_load_env_state(agarcl_batch* b, int32_t instance, const char* path, int lossless);
/* The same on a host blob of `L->stride` bytes (no device needed): what the two calls above run. */
int agarcl_snapshot_write(const agarcl_cfg* c, const agarcl_layout* L, const void* blob, const char* path);
int agarcl_snapshot_read(const agarcl_cfg* c, const agarcl_layout* L, void* blob, const char* path, int lossless);
/* Recorded uniform draws in [0,1) for instance i (replay of the reference's mt19937_64, SURVEY 8c). */
int agarcl_batch_set_replay(agarcl_batch* b, int32_t instance, const float* draws, int32_t n);
/* Run only the observation kernel on the current state (tests; add_frame on a cleared buffer). */
int agarcl_batch_render(agarcl_batch* b, void* stream);
/* Per-kernel device timing (bench.py roofline): when enabled, every agarcl_batch_step brackets the
 * engine-tick kernel and the observation kernel with CUDA events on the launching stream.
 * agarcl_batch_get_timing synchronises, returns the accumulated milliseconds and step count since the
 * last call, and resets the accumulators. */
int agarcl_batch_set_timing(agarcl_batch* b, int enable);
int agarcl_batch_get_timing(agarcl_batch* b, double* sim_ms, double* obs_ms, int32_t* steps);
/* Number of kernel launches issued by the last agarcl_batch_step. */
int agarcl_batch_launches_per_step(const agarcl_batch* b);
/* hdr.flags of the whole batch, reduced on the device: *or_all = OR over all instances, counts[bit] = instances with
 * AGARCL_FLAG bit `bit` set (either pointer may be NULL).  Synchronises `stream`.  The reference has no counterpart: its
 * containers grow without bound where this library has fixed capacities (BaseEnvironment.hpp / Engine.hpp vectors). */
int agarcl_batch_flags(agarcl_batch* b, void* stream, uint32_t* or_all, uint32_t counts[32]);
/* Diagnostics of the schedule: cycles every instance worked in the last step (what the cost-sorted schedule orders the next step by;
 * waiting at the alignment barriers excluded).  out: HOST array of N entries.  Synchronises `stream`.  No reference counterpart. */
int agarcl_batch_costs(agarcl_batch* b, void* stream, uint32_t* out);
/* Self-test of the device's restatement of libstdc++'s std::sort (k_step's strip_std_sort; the reference sorts the strips of
 * PrecisionCollisionDetection::solve with it, agario/utils/collision_detection.hpp:29-31): sorts the indices 0..n-1 by the HOST keys
 * ys[n] on the current device and writes the resulting order to order_out[n].  n <= 65535.  tests/test_gpu_std_sort.py compares it
 * with the oracle's restatement, which is pinned against the real std::sort. */
int agarcl_selftest_std_sort(const float* ys, int32_t n, uint16_t* order_out);
/* Host helper: first n canonical floats of std::mt19937_64(seed) as uniform_real_distribution<float>
 * draws them (random.hpp:6-20). */
int agarcl_mt19937_draws(uint64_t seed, float* out, int32_t n);

const char* agarcl_last_error(void);
const char* agarcl_version(void);

#ifdef __cplusplus
}
#endif
#endif /* AGARCL_B200_H */
