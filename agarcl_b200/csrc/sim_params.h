// sim_params.h — kernel parameter blocks shared by the host API (batch.cu) and the kernels.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "../../include/agarcl_b200.h"
#include "device_math.cuh"
#include "mode_rules.h"

namespace ag {

constexpr int kMaxWarpsPerCta = 16;   // one warp owns one game instance; ONE persistent CTA per SM of as many independent warps as the
                                      // shared memory holds (16 x 13.9 KB at 1000 pellets) and the register file allows (4 per SM
                                      // sub-partition x 128 registers per thread)
constexpr int kPremCap = 192;         // pellets_to_remove entries per tick (Engine.hpp:212)
constexpr int kVremCap = 32;          // viruses_to_remove entries per tick (Engine.hpp:213)
constexpr int kCandCap = 32;          // pellet candidates resolved in registers per cell
constexpr int kLaneCand = 8;          // pellet candidates a single lane resolves in the lane-per-player phase
constexpr int kZeroTileBytes = 2560;  // CTA-shared all-zero tile, source of the TMA bulk stores that clear the observation
constexpr int kColdCtxBytes = 96;    // per-warp slot of ColdCtx (sim_kernel.cu) + 16 B of the solver pool's counters
constexpr int kSnapCap = 96;          // cells staged in shared memory by the players_collision pre-test (12 bytes each: x, y, mass | player << 24)
constexpr int kPairCap = 48;          // (eater, eaten) pairs per tick in players_collision
constexpr int kCellRefCap = 256;      // total live cells per instance handled by players_collision

// byte offsets of one warp's shared-memory arrays (sim_shared.cuh)
struct SmemOff {
  uint32_t hcnt, htmp, hsorted, spel, mbar, cellref, rows, strip, hitq, snap, vcache, psum, pcell, pairs, reskeys, resorder, cand, prem, vrem, lprem, cold;
  uint32_t sweep_in_hash;  // the exact collision sweep's scratch lies over hsorted: running it invalidates the pellet hash
};

// Transfer lists of the host-resident observation mirror (mirror.cu), produced on the device either by the fused
// observation finish of k_step (no second pass over the dense tensor) or by k_pack.  The agent images are grouped
// into CHUNKS of `ipc` consecutive images; one chunk = one contiguous block of 32-bit words
//   [0] entries used in the chunk (k_pack only)   [1..3] pad
//   rec[ipc][rec_words]   per slot: count (entries of the image, or 0xFFFFFFFF: does not fit the scheme, copy the
//                         image densely), base (its first entry in the chunk's entry array), the index of the image
//                         the slot describes (k_step fills the slots in the order of its schedule, so that the chunks
//                         complete one after the other while it runs; k_pack: slot = image), then per frame the row
//                         bit mask and the column bit mask of the out-of-bounds channel (bit i: row i out of bounds),
//                         then the agent's reward (f64, two words) and done flag of the step (k_step only)
//   entries[cap_chunk]    uint2 (op << 29 | element offset inside the image, operand): the integer operation the
//                         host replays on its copy of the element (kPkSet .. kPkMax)
// k_step writes its blocks STRAIGHT INTO PINNED HOST MEMORY (`chunks` is then the device address of a host-mapped
// buffer): every image owns the fixed slot [li * slot, (li + 1) * slot) of its chunk's entry array -- slack costs
// nothing because only the bytes written cross PCIe -- and the warp writes its entries as coalesced 16-byte
// stores while it scatters.  The warp that finishes the last instance of a chunk raises the chunk's flag in
// host-mapped memory, so the host expands chunk k while the kernel is still stepping the instances of chunk k+1
// and nothing is left to copy when the kernel ends.  k_pack writes compact blocks in device memory (one cursor per
// chunk), which the host fetches with one copy per chunk.
struct PackOut {
  uint32_t* chunks;          // nullptr: no lists wanted
  uint32_t* cursor;          // [n_chunks] running entry count (k_pack; self-rewinding)
  uint32_t* done;            // [n_chunks] images finished (self-rewinding)
  volatile uint32_t* flags;  // [n_chunks] host-mapped: last step sequence number whose chunk is complete; may be nullptr
  uint32_t chunk_words;      // words between consecutive chunk blocks
  uint32_t ipc;              // slots (images) per chunk (a multiple of the agents per instance)
  uint32_t rec_words;        // 3 + frames * 2 * MW + 3
  uint32_t cap_chunk;        // entry capacity of a chunk
  uint32_t slot;             // k_step: entries per image slot (even; ipc * slot <= cap_chunk)
  uint32_t n_img;
  uint32_t seq;
  int32_t MW;                // 32-bit words per row (or column) mask
};
constexpr uint32_t kPackDense = 0xFFFFFFFFu;
// entry operations: x = v | x += v | x = x ? min(x, v) : v | x = max(x, v)   (GridObservation's at_least_ / total_mass_ /
// min / max channel rules, environment/envs/GridEnvironment.hpp:212-232); k_pack lists final values as kPkSet
constexpr uint32_t kPkSet = 0u, kPkAdd = 1u, kPkMinNz = 2u, kPkMax = 3u;
constexpr uint32_t kPkOffMask = 0x1FFFFFFFu;
__host__ __device__ inline uint32_t pk_off_rec(const PackOut&) { return 4u; }
__host__ __device__ inline uint32_t pk_off_entries(const PackOut& k) { return (4u + k.ipc * k.rec_words + 3u) & ~3u; }

struct SimParams {
  agarcl_layout L;
  Luts T;
  uint8_t* state;          // N blobs, L.stride apart
  const float* dxdy;       // [N*A*2] actions for this step
  const int32_t* act;      // [N*A]
  double* rewards;         // [N*A]
  uint8_t* dones;          // [N*A]
  float* before;           // [N*A] masses<float>() at step begin (BaseEnvironment.hpp:92)
  const float* replay;     // [N*cap_replay] or nullptr
  uint32_t* tickets;       // [2] persistent-grid work counter: next instance, warps that have left (k_step without alignment)
  uint32_t* cost;          // [N] cycles every instance worked in this step (nullptr: not wanted)
  const uint32_t* perm;    // [N] cost-sorted instance order of the previous step (nullptr: identity)
  uint32_t* sched;         // [2] or nullptr: [0] schedule of this launch (1: aligned as tick_barrier says, 0: free-running), set by k_order
                           // from [1], the instances that held a multi-cell player at the end of the previous launch
  int32_t N;
  int32_t instance_base;
  int32_t n_ticks;         // ticks to run in this launch
  int32_t do_begin;        // apply actions + record `before`
  int32_t do_end;          // respawn / dones / rewards
  int32_t mode, reward_type, rng_mode;
  const int32_t* task_mode;  // [N] mixed-task batch (cfg.task_modes): each instance's current mode, read once per launch into ColdCtx;
                             // nullptr: every instance plays `mode` with the flags of L
  int32_t num_bots;          // cfg.num_bots (mode_rules, mixed-task batch)
  int32_t target_pellets, target_viruses;
  // mixed-task batch: each instance's current game sizes (agarcl_batch_set_task_sizes), read from global memory at the regen tick
  // (the regen targets) and at the mode-0 respawn (players >= A + bots are absent); nullptr: target_* and L.P for all
  const int32_t *task_bots, *task_pellets, *task_viruses;
  int32_t HG;              // spatial hash is HG x HG over the arena
  float W;                 // arena width == height
  float hash_scale;        // HG / W
  float r_pellet;          // radius_conversion(PELLET_MASS = 1), the table's entry (core/utils.hpp:8-11)
  int32_t gw_pellet;       // reference pellet bucket grid width (bucket 510, Engine.hpp:962-965)
  int32_t gw_virus;        // reference virus bucket grid width (bucket 25, Engine.hpp:1207-1211)
  uint32_t smem_per_warp;  // bytes
  uint32_t tiles_bytes;    // CTA-wide tiles in front of the warps' carve-ups: the zero tile, then the all-ones tile (fused finish only)
  SmemOff so;
  // fused observation clear: the engine-tick kernel streams the zeros of channels 1..C-1 of every
  // agent frame (state independent, 7/8 of all bytes of the step) while it computes; k_obs then only
  // writes channel 0 and scatters the entities.  zero_vec_per_agent == 0 disables it.
  void* obs;                    // frame slot of agent 0 of instance 0
  uint32_t zero_vec_per_agent;  // 16-byte vectors to clear per agent frame
  uint32_t zero_skip_vec;       // vectors of channel 0 in front of them
  uint32_t agent_stride_vec;    // vectors between consecutive agents' frame slots
  // fused observation finish (one frame): after the last tick each warp also writes channel 0
  // and scatters the entities of its instance, so the step is ONE kernel.  obs_finish == 0: k_obs does it; 1: int32; 2: int16.
  int32_t obs_finish, obs_G, obs_C;
  int32_t zero_chunks;          // > 0: the clear is queued in this many pieces (4 per tick); 0: spread over the ticks
  int32_t observe_cells, observe_others, observe_viruses, observe_pellets;
  int32_t tick_barrier;         // instruction-fetch alignment (step_instance), bit mask of the CTA barriers of a tick: 1 tick start, 2 around the
                                // pooled pair solver, 4 before players_collision, 8 before move_foods, 16 before apply_removals; 0: free-running warps
  int32_t dyn_stripes;          // aligned schedule: 1 = stripes handed out by the ticket counter (default), 0 = the static round-robin pairing
  int32_t align_group;          // warps per alignment group (a divisor-free choice: the last group of a CTA may be smaller)
  PackOut pk;                   // with obs_finish only
  int32_t inst_first;           // this launch steps instances [inst_first, inst_first + N) of the batch
};

// How k_step is launched on one device: found by setup_step when a batch is created there and kept by the batch, because
// function attributes belong to the device's context and a process may hold batches on several devices
struct StepLaunch {
  int sms;         // k_step's persistent grid has at most one CTA per SM
  int smem_optin;  // opt-in shared memory per block: the dynamic shared memory k_step (and k_ram) may use on this device
  int max_warps;   // warps per CTA at most: kMaxWarpsPerCta, or fewer when capped (AGARCL_WARPS)
};
// On the current device: fills S and opts k_step in to S.smem_optin bytes of dynamic shared memory.  warps_cap > 0 caps S.max_warps.
cudaError_t setup_step(int warps_cap, StepLaunch& S);
// One CTA per SM, as many warps (= concurrent instances) as the shared memory holds, at most S.max_warps.
cudaError_t launch_step(const SimParams& P, const StepLaunch& S, cudaStream_t stream);
cudaError_t launch_order(const uint32_t* cost, uint32_t* perm, int N, uint32_t* sched, cudaStream_t stream);
cudaError_t selftest_std_sort(const float* ys, int n, uint16_t* order_out);

struct ResetParams {
  agarcl_layout L;
  Luts T;
  uint8_t* state;
  const uint8_t* mask;     // [N] or nullptr (all)
  const uint64_t* seeds;   // [N]
  const float* replay;
  uint8_t* fresh;          // [N] != 0: the instance was (re)seeded since its last reset -> its draw stream starts at 0; otherwise the
                           // stream goes on where the last episode left it, like the reference's engine RNG across reset()
                           // (BaseEnvironment.hpp:179-204 does not reseed); cleared by the kernel
  uint8_t* dones;
  // mixed-task batch (cfg.task_modes; nullptr otherwise): every reset instance takes its pending task (next_*) as its current one
  // and is spawned by the rules of that mode, with players P_m .. P-1 absent
  int32_t *task_mode, *task_max_steps;
  const int32_t *next_mode, *next_max_steps;
  agarcl_task_sizes sizes;   // the same for the game sizes: next_* become the current ones and are what the reset spawns
  int32_t N, instance_base, rng_mode, num_pellets, num_viruses;
  float W;
};
cudaError_t launch_reset(const ResetParams& P, cudaStream_t stream);
cudaError_t launch_flags(const uint8_t* state, const agarcl_layout& L, int N, uint32_t* out33, cudaStream_t stream);

struct ObsParams {
  agarcl_layout L;
  const uint8_t* state;
  void* obs;               // [N*A][frames*C][G][G] int32 or int16
  int32_t N, G, C, frames, frame;  // frame: which frame slot this launch fills
  int32_t observe_cells, observe_others, observe_viruses, observe_pellets;
  int32_t obs_dtype;
  int32_t pre_respawn;     // 1: show players respawned at the end of the step as still dead
  int32_t skip_zero;       // 1: channels 1..C-1 were already cleared by the engine-tick kernel
  const uint8_t* mask;     // [N] or nullptr: render only the instances with mask != 0 (masked reset)
  float W;
};
cudaError_t launch_obs(const ObsParams& P, cudaStream_t stream);

struct RamParams {
  agarcl_layout L;
  Luts T;
  const uint8_t* state;
  float* ram;              // [N][P][AGARCL_RAM_RECORD]
  int32_t N, G;
  int32_t pre_respawn;     // 1: players respawned at the end of the step are still dead (BaseEnvironment.hpp:96-101)
  int32_t pid_base;        // CloneInfo::owner is the player's pid: index + pid of player 0 (non-zero only in later episodes of strict_reference, Q3)
};
// On the current device: opts k_ram in to the dynamic shared memory it needs for layout L (up to smem_optin bytes)
cudaError_t setup_ram(const agarcl_layout& L, int smem_optin);
cudaError_t launch_ram(const RamParams& P, cudaStream_t stream);

constexpr int kMaskedThreads = 512;  // threads of k_masked_bytes, one CTA per instance

// Episode bookkeeping of agarcl_batch_step_autoreset (episode_kernel.cu, k_episode)
struct EpisodeParams {
  const uint8_t* dones;      // [N*A] of the step that just ran
  const double* rewards;     // [N*A]
  uint8_t* done_out;         // [N*A] dones with the step limit folded in
  uint8_t* reset_mask;       // [N]
  int64_t* steps;            // [N] steps since the instance's last reset
  double* ret;               // [N*A] rewards summed since the instance's last reset
  double* final_ret;         // [N*A] ret of the episode that finished last
  int64_t* final_len;        // [N] steps of the episode that finished last
  const uint8_t* clear_mask; // clear mode: the instances being reset, nullptr = all
  const int32_t* task_max_steps;  // [N] mixed-task batch: the instance's step limit (-1: max_steps, 0: none); nullptr: max_steps for all
  int32_t N, A, max_steps;
  int32_t reset;             // 1: finished instances are reset by this step (auto-reset); 0: bookkeeping only
  int32_t clear;             // 1: a reset restarts the counters of clear_mask's instances (no step)
};
cudaError_t launch_episode(const EpisodeParams& P, cudaStream_t stream);
// agarcl_batch_set_tasks: pending task of instance i <- (mode[i], max_steps[i]) where given and valid; result[i] 0 / 1 / 2
struct SetTasksParams {
  const int32_t* mode;       // [N], -1 keeps the pending mode
  const int32_t* max_steps;  // [N] or nullptr (every pending limit kept)
  int32_t *next_mode, *next_max_steps;
  uint8_t* result;
  int32_t N, task_modes;
};
cudaError_t launch_set_tasks(const SetTasksParams& P, cudaStream_t stream);
// The maxima and allowed bot counts of a mixed-task batch's game sizes (agarcl_batch_set_task_sizes)
struct SizeLimits {
  int32_t bots, pellets, viruses;  // cfg.num_bots, num_pellets, num_viruses
  int32_t bots_any;                // 1: mode 0 is not in task_modes, the bot count means nothing and every one of 0 .. bots is allowed
  uint64_t bots_allowed;           // otherwise bit b: b bots pass the player-order check (layout.cpp, task_bot_counts; bots < 64)
};
__host__ __device__ inline bool sizes_allowed(const SizeLimits& M, int32_t bots, int32_t pellets, int32_t viruses) {
  return bots >= 0 && bots <= M.bots && (M.bots_any || ((M.bots_allowed >> bots) & 1u)) && pellets >= 0 && pellets <= M.pellets &&
         viruses >= 0 && viruses <= M.viruses;
}
// agarcl_batch_set_task_sizes: pending sizes of instance i <- the given entries (-1 or a nullptr array: kept) when all are valid
struct SetTaskSizesParams {
  const int32_t *bots, *pellets, *viruses;  // [N] or nullptr
  int32_t *next_bots, *next_pellets, *next_viruses;
  uint8_t* result;
  SizeLimits lim;
  int32_t N;
};
cudaError_t launch_set_task_sizes(const SetTaskSizesParams& P, cudaStream_t stream);
// dst = src (nullptr: zeros) in the `per`-byte slices of the instances with mask != 0
cudaError_t launch_masked_bytes(void* dst, const void* src, size_t per, const uint8_t* mask, int N, cudaStream_t stream);

// Snapshot pools (snapshot_kernel.cu, k_snapshot): the slot layout of include/agarcl_b200.h, agarcl_snapshot_hdr
struct SnapLayout {
  uint64_t off_blob, off_ep, off_ram, off_obs;  // segment offsets inside a slot (16-byte aligned)
  uint64_t ep_bytes, ram_bytes, obs_bytes;      // segment sizes; ram_bytes / obs_bytes 0 when the segment is not stored
  uint64_t slot_bytes;                          // a multiple of 128
};
constexpr int kSnapThreads = 512;  // threads of k_snapshot and k_start_states, one CTA per saved entry / restored or reset instance
struct SnapParams {
  uint8_t* pool;             // pool_slots slots of slot_bytes
  int64_t pool_slots;
  SnapLayout S;
  uint64_t fingerprint;
  uint8_t* state;            // the batch's N blobs, L.stride apart
  uint32_t stride, off_hdr;  // L.stride, L.off_hdr
  int64_t* steps;            // [N] episode bookkeeping, nullptr when it is off
  double* ret;               // [N*A]
  uint8_t* ram;              // [N] records of S.ram_bytes (when stored)
  uint8_t* obs;              // [N] observation images of S.obs_bytes (when stored)
  // save: pool slot (slot ? slot[k] : k) <- instance src[k], k < n
  const int32_t* src;
  const int32_t* slot;
  // restore: instance i <- pool slot slot_of[i] where >= 0
  const int32_t* slot_of;
  uint64_t* seeds;           // [N] the reset kernel's per-instance seed
  uint8_t* fresh;            // [N] ResetParams::fresh
  double* rewards;           // [N*A]
  uint8_t* dones;            // [N*A]
  uint8_t* result;           // [N] 0 not requested, 1 restored, 2 rejected
  uint8_t* restored;         // [N] 1 where restored: the mask of the k_obs launch behind
  int32_t* task_mode;        // [N] mixed-task batch: the current task, stored in the slot header and restored from it; else nullptr
  int32_t* task_max_steps;   // [N]
  int32_t task_modes;        // cfg.task_modes: a restored slot's mode must be in it
  agarcl_task_sizes sizes;   // mixed-task batch: the slot's game sizes become the current ones (maxima without the marker)
  SizeLimits lim;            //   and must be within these
  int32_t N, A, instance_base;
  // start states (agarcl_batch_set_start_states, k_start_states): in front of k_reset, instance i in `mask` (nullptr: all) <-
  // slot slot_of[i] where >= 0, with the instance's draw stream; result is the start result, not the restore's
  const uint8_t* mask;       // [N] the reset mask, or nullptr
  uint8_t* spawn;            // [N] out: the mask k_reset spawns (reset and not started from a slot)
  const int32_t* next_max_steps;  // [N] mixed-task batch: the pending step limit, which becomes the current one
};
cudaError_t launch_snapshot_save(const SnapParams& P, int n, cudaStream_t stream);
cudaError_t launch_snapshot_restore(const SnapParams& P, cudaStream_t stream);
cudaError_t launch_snapshot_start(const SnapParams& P, cudaStream_t stream);

// Go-Explore cell archive (archive_kernel.cu): the spec of include/agarcl_b200.h, agarcl_batch_set_archive
constexpr int kArchiveThreads = 1024;         // threads of the one-CTA kernels k_archive_commit and k_archive_select
constexpr int64_t kArchiveMaxSlots = 65536;   // entries of an archive at most: k_archive_select scans their weights in one CTA
struct ArchiveParams {
  agarcl_layout L;
  const uint8_t* state;      // N blobs, L.stride apart
  const uint8_t* dones;      // [N*A] of the step, before the step limit is folded in
  const double* rewards;     // [N*A]
  const double* ret;         // [N*A] episode return before this step (episode bookkeeping)
  const int64_t* steps;      // [N] episode steps before this step
  int32_t N, A, agent, n, K, instance_base;
  float W;
  uint64_t seed;
  // per instance
  int32_t* cell_of;          // key of the instance's cell, -1: none
  double* base_score;        // trajectory base of the running episode
  int64_t* base_length;
  int32_t* cand_key;         // this step: the key of a candidate, -1 otherwise
  double* cand_s;            // this step: a candidate's trajectory score and length
  int64_t* cand_l;
  int32_t* save_slot;        // this step: the slot instance i is saved into, -1 none (k_snapshot<true>'s slot list)
  uint32_t* draws;           // selection draws made so far
  // per key [32 n^2]
  int32_t* key_entry;
  uint32_t* visits;
  uint64_t* best_s;          // winner scratch, neutral 0: max of ordered_bits(score)
  uint64_t* best_li;         // winner scratch, neutral ~0: min of (min(length, 2^32 - 1) << 32 | instance)
  // per entry [K]
  int32_t* entry_key;
  double* entry_score;
  int64_t* entry_length;
  uint32_t* entry_chosen;
  uint64_t* prefix;          // k_archive_select scratch: inclusive prefix sums of the weights
  uint64_t* counters;        // [3] used, dropped, improved
  // resets
  const uint8_t* mask;       // [N] the instances reset (or restored), nullptr: all
  int32_t* start_slot;       // [N] the batch's start-state table
  const uint8_t* start_result;  // k_archive_base: the start result when the table is the archive's pool, else nullptr
};
cudaError_t launch_archive_update(const ArchiveParams& P, cudaStream_t stream);  // k_archive_cells + k_archive_commit
cudaError_t launch_archive_select(const ArchiveParams& P, cudaStream_t stream);
cudaError_t launch_archive_base(const ArchiveParams& P, cudaStream_t stream);

// Pictures of game states (draw_kernel.cu): the spec of include/agarcl_b200.h, agarcl_batch_draw.  k_draw draws arena views,
// k_draw_views agent views and the pixel observation (cfg.pixel_obs)
struct DrawParams {
  agarcl_layout L;
  const float* radius;     // Luts::radius
  const uint8_t* state;    // N blobs, L.stride apart
  uint8_t* out;            // [n][S][S][3]
  const int32_t* src;      // [n] or nullptr (picture k shows source k)
  int32_t n, S, view, N;
  float W;
  int32_t pre_respawn;     // k_draw_views: 1 draws players respawned at the end of the last step as still dead (the observation)
  const uint8_t* mask;     // k_draw_views: [N] or nullptr: only the pictures of instances with mask != 0 are written
};
cudaError_t launch_draw(const DrawParams& P, cudaStream_t stream);
// On the current device: opts k_draw_views in to the dynamic shared memory of its largest picture
cudaError_t setup_draw_views();
cudaError_t launch_draw_views(const DrawParams& P, cudaStream_t stream);

// Built-in bot policies for agents (bot_kernel.cu, k_bot_actions): the spec of include/agarcl_b200.h, agarcl_batch_bot_actions
struct BotParams {
  agarcl_layout L;         // with the batch's current player order
  const uint8_t* state;    // N blobs, L.stride apart
  const int32_t* type;     // [N*A] bot type per agent, -1: not requested
  float* dxdy;             // [N*A][2]
  int32_t* act;            // [N*A]
  float* target;           // [N*A][2] or nullptr
  uint8_t* status;         // [N*A] or nullptr
  int32_t N;
};
cudaError_t launch_bot_actions(const BotParams& P, cudaStream_t stream);

}  // namespace ag
