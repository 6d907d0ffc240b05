// batch.cu — host side of the C ABI (include/agarcl_b200.h): owns the device memory of a batch of
// N lockstep instances and enqueues the kernels.  Mirrors, for the batched path, what
// environment/bindings.cpp:99-135 binds on agario::env::GridEnvironment (ctor, seed,
// configure_observation, take_actions, step, get_state, dones, reset).
//
// There is NO CPU fallback: every entry point that computes needs a CUDA device and fails with
// AGARCL_ERR_CUDA otherwise.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <memory>
#include <new>
#include <random>
#include <unordered_map>
#include <vector>

#include "host_util.h"
#include "mirror.h"
#include "sim_params.h"
#include "sim_shared.cuh"

// Device memory owned by a batch: freed with it.
template <typename T>
class DevBuf {
 public:
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { cudaFree(p_); }
  cudaError_t alloc(size_t bytes) { return cudaMalloc((void**)&p_, bytes); }
  T* get() const { return p_; }
  operator T*() const { return p_; }

 private:
  T* p_ = nullptr;
};

// The Go-Explore cell archive of a batch (agarcl_batch_set_archive): its settings and device arrays (ArchiveParams)
struct Archive {
  const void* pool = nullptr;
  int64_t K = 0;
  agarcl_archive_cfg cfg;
  int64_t keys = 0;  // 32 n^2
  DevBuf<int32_t> cell_of, cand_key, save_slot, src, key_entry, entry_key;
  DevBuf<double> base_score, cand_s, entry_score;
  DevBuf<int64_t> base_length, cand_l, entry_length;
  DevBuf<uint32_t> draws, visits, entry_chosen;
  DevBuf<uint64_t> best_s, best_li, prefix, counters;
};

// The A/B knobs of the step (names, defaults and effects: DESIGN.md section 8), read from the environment when a batch is created
struct Knobs {
  int fuse_clear = 2, sort_schedule = 1, auto_schedule = 1, tick_barrier = 6, dyn_stripes = 1, zero_chunks = 0;
  int warps = 0;  // > 0: at most this many warps per k_step CTA
  double hash_per_cell = 3.0;
};

static Knobs read_knobs() {
  Knobs k;
  auto env_int = [](const char* name, int& v) { if (const char* e = std::getenv(name)) v = std::atoi(e); };
  env_int("AGARCL_FUSE_CLEAR", k.fuse_clear);
  env_int("AGARCL_SORT_SCHEDULE", k.sort_schedule);
  env_int("AGARCL_AUTO_SCHEDULE", k.auto_schedule);
  env_int("AGARCL_TICK_BARRIER", k.tick_barrier);
  env_int("AGARCL_DYNAMIC_STRIPES", k.dyn_stripes);
  env_int("AGARCL_ZERO_CHUNKS", k.zero_chunks);
  env_int("AGARCL_WARPS", k.warps);
  if (const char* e = std::getenv("AGARCL_HASH_PER_CELL")) k.hash_per_cell = std::atof(e);
  return k;
}

struct agarcl_batch {
  agarcl_cfg cfg;
  agarcl_layout L;
  // strict_reference, quirk Q3: the reference's player map and pid counter outlive a reset (GameState::clear keeps the bucket
  // array, Engine::reset does not rewind next_pid), so the iteration order of the players depends on how many times the
  // environment has been reset.  The same container, fed the same insert sequence, reset after reset.
  std::unordered_map<unsigned short, int> pmap;
  unsigned short next_pid = 0;
  int32_t pid_base = 0;  // pid of player index 0 in the current episode
  int N, A, G, C, frames;
  size_t obs_elems, obs_bytes;
  Knobs knobs;
  ag::StepLaunch step_launch;
  DevBuf<uint8_t> d_state;
  DevBuf<void> d_obs;
  DevBuf<float> d_ram;  // structured observation records [N][P][AGARCL_RAM_RECORD], only with cfg.ram_obs
  DevBuf<double> d_rewards;
  DevBuf<uint8_t> d_dones;
  DevBuf<float> d_before;
  DevBuf<float> d_dxdy;
  DevBuf<int32_t> d_act;
  const float* cur_dxdy = nullptr;  // what the next step reads (own buffers or caller's device pointers)
  const int32_t* cur_act = nullptr;
  DevBuf<float> d_replay;
  DevBuf<uint64_t> d_seeds;
  DevBuf<uint8_t> d_mask;
  DevBuf<uint32_t> d_tickets;  // k_step's ticket counter pair (self-rewinding)
  DevBuf<uint32_t> d_sched;    // [2] schedule selector of k_step (SimParams::sched)
  DevBuf<uint32_t> d_cost, d_perm;  // per-instance cost of the last step and the cost-sorted schedule made from it (k_order)
  bool perm_valid = false;
  DevBuf<float> d_lut_radius, d_lut_speed, d_lut_split;
  std::vector<uint64_t> seeds;
  // AGARCL_RNG_MT19937: the reference's generator per instance (GameState::rng, GameState.hpp:51), kept on the host; its
  // uniform_real_distribution<float> draws are fed to the device through d_replay used as a RING that refill_replay keeps
  // filled ahead of every instance's draw cursor (filled[i] = draws generated so far; the ring holds [filled - cap, filled))
  std::vector<std::mt19937_64> gens;
  std::vector<uint64_t> filled;
  int64_t draw_budget = 0;      // draws every instance is known to have ahead of its cursor
  int64_t max_draws_per_step = 0;
  DevBuf<uint8_t> d_fresh;      // [N] instance (re)seeded since its last reset (ResetParams::fresh)
  DevBuf<uint32_t> d_flagbuf;   // [33] agarcl_batch_flags scratch
  ag::Luts T;
  int HG;
  uint32_t smem_per_warp;
  ag::SmemOff so;
  bool was_reset = false;
  int launches_last_step = 0;
  // vector-env episode bookkeeping (agarcl_batch_set_autoreset); buffers allocated on first use
  bool autoreset = false, autoreset_reset = true, keep_final = false;
  int32_t max_steps = 0;
  DevBuf<uint8_t> d_done_out, d_reset_mask;
  DevBuf<int64_t> d_steps, d_final_len;
  DevBuf<double> d_ret, d_final_ret;
  DevBuf<void> d_final_obs;          // [N*A, frames*C, G, G], only with keep_final_obs and a grid observation
  DevBuf<float> d_final_ram;         // [N, P, AGARCL_RAM_RECORD], only with keep_final_obs and cfg.ram_obs
  // pixel observation (cfg.pixel_obs = S): every agent's picture [N*A, S, S, 3] after every step and reset, and the finishing ones
  DevBuf<uint8_t> d_pixels, d_final_pixels;  // (d_final_pixels only with keep_final_obs)
  size_t pixel_bytes = 0;
  // snapshot pools (agarcl_batch_save_states / _restore_states): the slot layout, the configuration's fingerprint, the
  // library-owned result of the last restore and the mask of the instances it restored
  ag::SnapLayout snap;
  uint64_t fingerprint = 0;
  DevBuf<uint8_t> d_snap_result, d_snap_restored;
  // start states of resets (agarcl_batch_set_start_states): the pool (nullptr: every reset spawns), a start slot per instance,
  // the result of the latest reset with a table and the mask of the instances that reset spawns
  const void* start_pool = nullptr;
  int64_t start_pool_slots = 0;
  DevBuf<int32_t> d_start_slot;
  DevBuf<uint8_t> d_start_result, d_spawn;
  std::unique_ptr<Archive> archive;  // Go-Explore cell archive (agarcl_batch_set_archive), nullptr: none
  // mixed-task batch (cfg.task_modes != 0, include/agarcl_b200.h): current and pending task per instance, result of the last set_tasks
  DevBuf<int32_t> d_task_mode, d_task_max_steps, d_next_mode, d_next_max_steps;
  DevBuf<uint8_t> d_task_result;
  // and its game sizes (agarcl_batch_set_task_sizes): current and pending bots, pellets, viruses, their limits, the last result
  DevBuf<int32_t> d_bots, d_pellets, d_viruses, d_next_bots, d_next_pellets, d_next_viruses;
  DevBuf<uint8_t> d_size_result;
  ag::SizeLimits size_lim = {};
  ag::HostMirror* mirror = nullptr;  // host-resident observation mirror (mirror.cu), created on first use
  ag::HostMirror* lists = nullptr;   // the lists-only twin behind agarcl_batch_step_lists (no dense tensor, no worker threads)
  uint64_t mirror_launch_us = 0, mirror_call_us = 0;  // last agarcl_batch_step_mirror: staging + launch, whole call
  // optional per-kernel timing: (start, after sim, after obs) event triples of steps not yet collected
  bool timing = false;
  std::vector<cudaEvent_t> ev;
  size_t ev_used = 0;
  double acc_sim_ms = 0.0, acc_obs_ms = 0.0;
  int acc_steps = 0;

  ~agarcl_batch() {
    ag::mirror_destroy(mirror);
    ag::mirror_destroy(lists);
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
  }
};

static cudaEvent_t next_event(agarcl_batch* b) {
  if (b->ev_used == b->ev.size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    b->ev.push_back(e);
  }
  return b->ev[b->ev_used++];
}
static void collect_timing(agarcl_batch* b) {
  if (!b->ev_used) return;
  cudaEventSynchronize(b->ev[b->ev_used - 1]);
  for (size_t i = 0; i + 2 < b->ev_used; i += 3) {
    float a = 0.f, c = 0.f;
    cudaEventElapsedTime(&a, b->ev[i], b->ev[i + 1]);
    cudaEventElapsedTime(&c, b->ev[i + 1], b->ev[i + 2]);
    b->acc_sim_ms += a;
    b->acc_obs_ms += c;
    b->acc_steps++;
  }
  b->ev_used = 0;
}

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      return agarcl_set_error(AGARCL_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e__));   \
  } while (0)

// Allocates `bytes` of device memory for `buf` unless it holds some already, and fills them with the byte `fill` (-1: left as is).
template <typename T>
static int alloc(DevBuf<T>& buf, size_t bytes, int fill = -1) {
  if (buf) return AGARCL_OK;
  const cudaError_t e = buf.alloc(bytes);
  if (e != cudaSuccess) return agarcl_set_error(AGARCL_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
  if (fill >= 0) CK(cudaMemset(buf, fill, bytes));
  return AGARCL_OK;
}

// The six game-size arrays of a mixed-task batch (all nullptr otherwise)
static agarcl_task_sizes task_sizes_of(const agarcl_batch* b) {
  agarcl_task_sizes z;
  z.bots = b->d_bots; z.pellets = b->d_pellets; z.viruses = b->d_viruses;
  z.next_bots = b->d_next_bots; z.next_pellets = b->d_next_pellets; z.next_viruses = b->d_next_viruses;
  return z;
}

static void fill_sim_params(const agarcl_batch* b, ag::SimParams& P) {
  P.L = b->L;
  P.T = b->T;
  P.state = b->d_state;
  P.dxdy = b->cur_dxdy;
  P.act = b->cur_act;
  P.rewards = b->d_rewards;
  P.dones = b->d_dones;
  P.before = b->d_before;
  P.replay = b->d_replay;
  P.tickets = b->d_tickets;
  P.cost = nullptr;
  P.perm = nullptr;
  P.sched = nullptr;
  P.N = b->N;
  P.instance_base = b->cfg.instance_base;
  P.mode = b->cfg.mode_number;
  P.task_mode = b->d_task_mode;
  P.num_bots = b->cfg.num_bots;
  P.reward_type = b->cfg.reward_type;
  P.rng_mode = b->cfg.rng_mode;
  P.target_pellets = b->cfg.num_pellets;
  P.target_viruses = b->cfg.num_viruses;
  P.task_bots = b->d_bots; P.task_pellets = b->d_pellets; P.task_viruses = b->d_viruses;
  P.HG = b->HG;
  P.W = (float)b->cfg.arena_size;
  P.hash_scale = (float)b->HG / (float)b->cfg.arena_size;
  P.r_pellet = (float)std::sqrt((double)AGARCL_PELLET_MASS / 1.0 / M_PI);
  // initialize_pellet_grid / initialize_virus_grid: int((W + size - 1) / size) in fp32 (Engine.hpp:962-965,1207-1211)
  P.gw_pellet = (int)(((float)b->cfg.arena_size + 510.0f - 1.0f) / 510.0f);
  P.gw_virus = (int)(((float)b->cfg.arena_size + 25.0f - 1.0f) / 25.0f);
  P.smem_per_warp = b->smem_per_warp;
  P.tiles_bytes = ag::kZeroTileBytes;  // (+ the all-ones tile when the kernel also finishes the observation, fuse_obs_clear)
  P.so = b->so;
  P.obs = nullptr;
  P.zero_vec_per_agent = 0; P.zero_skip_vec = 0; P.agent_stride_vec = 0;
  P.obs_finish = 0; P.obs_G = b->G; P.obs_C = b->C;
  P.zero_chunks = b->knobs.zero_chunks;
  P.dyn_stripes = b->knobs.dyn_stripes;
  P.tick_barrier = b->knobs.tick_barrier;
  P.align_group = ag::kMaxWarpsPerCta;  // the whole CTA (groups of 8 / 4 / 2 warps were slower: 1.78 / 1.97 / 2.16 vs 1.70 ms)
  P.observe_cells = b->cfg.observe_cells; P.observe_others = b->cfg.observe_others;
  P.observe_viruses = b->cfg.observe_viruses; P.observe_pellets = b->cfg.observe_pellets;
  std::memset(&P.pk, 0, sizeof(P.pk));
  P.inst_first = 0;
}

// Whether the batch renders a grid frame: not under the structured observation only (agario-ram-v0), not with pixels
static bool renders_grid(const agarcl_batch* b) { return b->cfg.ram_obs != 2 && !b->cfg.pixel_obs; }

// Whether the engine-tick kernel writes the whole observation frame itself (SimParams::obs_finish): 0 no (k_obs renders
// it), 1 int32, 2 int16.  Needs the fused clear, rows of whole 16-byte vectors, one row of channel 0 = one bulk store from
// the ones tile, and the row of y masks in the collision scratch.
static int obs_finish_kind(const agarcl_batch* b) {
  const size_t esz = b->cfg.obs_dtype == AGARCL_OBS_I16 ? 2 : 4;
  const size_t row = (size_t)b->G * esz;
  if ((row * b->G) % 16 != 0 || b->C < 2 || b->knobs.fuse_clear < 2) return 0;
  if (row % 16 != 0 || row > (size_t)ag::kZeroTileBytes || row > (size_t)(b->so.vcache - b->so.cellref)) return 0;
  return esz == 2 ? 2 : 1;
}

// Lets the engine-tick kernel clear channels 1..C-1 of frame slot `frame` (see SimParams); false when
// the planes are not 16-byte multiples.
static bool fuse_obs_clear(const agarcl_batch* b, ag::SimParams& P, int frame) {
  const size_t esz = b->cfg.obs_dtype == AGARCL_OBS_I16 ? 2 : 4;
  const size_t plane = (size_t)b->G * b->G * esz;
  if (plane % 16 != 0 || b->C < 2 || b->knobs.fuse_clear == 0) return false;
  P.obs = (uint8_t*)b->d_obs.get() + (size_t)frame * b->C * plane;
  P.zero_skip_vec = (uint32_t)(plane / 16);
  P.zero_vec_per_agent = (uint32_t)((size_t)(b->C - 1) * plane / 16);
  P.agent_stride_vec = (uint32_t)((size_t)b->frames * b->C * plane / 16);
  P.obs_finish = obs_finish_kind(b);
  if (P.obs_finish) P.tiles_bytes = ag::kZeroTileBytes + (((uint32_t)b->G * (uint32_t)esz + 127u) & ~127u);
  return true;
}

// Whether the one-frame step's k_step also writes the host lists of every image (agarcl_batch_step_mirror / _step_lists):
// it finishes the observation itself, and an image's record (count, base, image, row and column masks, reward, done) is
// one store of a warp's 32 lanes.
static bool kernel_writes_lists(const agarcl_batch* b) {
  return b->frames == 1 && !b->cfg.strict_reference && renders_grid(b) && obs_finish_kind(b) != 0 &&
         6 + 2 * ((b->G + 31) / 32) <= 32;
}

static void fill_obs_params(const agarcl_batch* b, ag::ObsParams& P, int frame, int pre_respawn, int skip_zero = 0) {
  P.pre_respawn = pre_respawn;
  P.skip_zero = skip_zero;
  P.mask = nullptr;
  P.L = b->L;
  P.state = b->d_state;
  P.obs = b->d_obs;
  P.N = b->N;
  P.G = b->G;
  P.C = b->C;
  P.frames = b->frames;
  P.frame = frame;
  P.observe_cells = b->cfg.observe_cells;
  P.observe_others = b->cfg.observe_others;
  P.observe_viruses = b->cfg.observe_viruses;
  P.observe_pellets = b->cfg.observe_pellets;
  P.obs_dtype = b->cfg.obs_dtype;
  P.W = (float)b->cfg.arena_size;
}

// ---- AGARCL_RNG_MT19937 stream plumbing
static inline float mt_next(std::mt19937_64& g) {  // exactly what agarcl_mt19937_draws / Engine::random<float> draw (random.hpp:6-20)
  std::uniform_real_distribution<float> d(0.0f, 1.0f);
  return d(g);
}
// Generates draws [filled, upto) of instance i and stores them at their ring positions on the device.
static int mt_extend(agarcl_batch* b, int i, uint64_t upto) {
  const uint64_t cap = (uint64_t)b->L.cap_replay;
  if (upto <= b->filled[i]) return AGARCL_OK;
  uint64_t from = b->filled[i];
  if (upto - from > cap) {  // (only the last `cap` draws can live in the ring)
    for (uint64_t k = from; k < upto - cap; k++) (void)mt_next(b->gens[i]);
    from = upto - cap;
  }
  std::vector<float> buf((size_t)(upto - from));
  for (auto& v : buf) v = mt_next(b->gens[i]);
  float* row = b->d_replay + (size_t)i * cap;
  uint64_t k = from;
  while (k < upto) {
    const uint64_t pos = k % cap, n = std::min<uint64_t>(upto - k, cap - pos);
    if (cudaMemcpy(row + pos, buf.data() + (k - from), (size_t)n * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess)
      return agarcl_set_error(AGARCL_ERR_CUDA, "replay ring upload failed");
    k += n;
  }
  b->filled[i] = upto;
  return AGARCL_OK;
}
// (Re)starts instance i's stream at draw index `at` from `seed` (Engine::seed, Engine.hpp:242-245) and fills the ring ahead of it.
static int mt_restart(agarcl_batch* b, int i, uint64_t seed, uint64_t at) {
  b->gens[i].seed((unsigned)seed);  // BaseEnvironment::seed(int) -> Engine::seed(unsigned)
  b->filled[i] = 0;
  for (uint64_t k = 0; k < at; k++) (void)mt_next(b->gens[i]);
  b->filled[i] = at;
  return mt_extend(b, i, at + (uint64_t)b->L.cap_replay);
}
// Called behind every launch that may draw (step, reset): when the instances may have come within one step's worth of
// draws of the end of what the ring holds, read the cursors back and fill the ring ahead of them again.
static int refill_replay(agarcl_batch* b, cudaStream_t s) {
  if (b->cfg.rng_mode != AGARCL_RNG_MT19937) return AGARCL_OK;
  b->draw_budget -= b->max_draws_per_step;
  if (b->draw_budget >= b->max_draws_per_step) return AGARCL_OK;
  std::vector<uint32_t> cur((size_t)b->N);
  if (cudaMemcpy2DAsync(cur.data(), sizeof(uint32_t), b->d_state + b->L.off_hdr + offsetof(agarcl_inst_hdr, rng_cursor), b->L.stride,
                        sizeof(uint32_t), (size_t)b->N, cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess)
    return agarcl_set_error(AGARCL_ERR_CUDA, "draw cursor read-back failed: %s", cudaGetErrorString(cudaGetLastError()));
  int64_t budget = b->L.cap_replay;
  for (int i = 0; i < b->N; i++) {
    // the 32-bit device cursor counts modulo 2^32; the stream position is the one nearest below `filled`
    uint64_t c = (b->filled[i] & ~0xffffffffull) | cur[i];
    if (c > b->filled[i]) c -= 0x100000000ull;
    const uint64_t ahead = b->filled[i] - c;
    if ((int64_t)ahead < (int64_t)b->L.cap_replay / 2 || (int64_t)ahead < 2 * b->max_draws_per_step) {
      int rc = mt_extend(b, i, c + (uint64_t)b->L.cap_replay);
      if (rc) return rc;
    }
    budget = std::min<int64_t>(budget, (int64_t)(b->filled[i] - c));
  }
  b->draw_budget = budget;
  return AGARCL_OK;
}

// ---- snapshot pools: the slot layout of include/agarcl_b200.h (agarcl_snapshot_hdr) and the configuration fingerprint
static uint64_t align_to(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

static void snapshot_layout(const agarcl_cfg& c, const agarcl_layout& L, ag::SnapLayout& S) {
  const uint64_t esz = c.obs_dtype == AGARCL_OBS_I16 ? 2 : 4;
  S.off_blob = sizeof(agarcl_snapshot_hdr);
  S.off_ep = S.off_blob + L.stride;
  S.ep_bytes = align_to(8 + 8 * (uint64_t)L.A, 16);
  S.off_ram = S.off_ep + S.ep_bytes;
  S.ram_bytes = c.ram_obs ? (uint64_t)L.P * AGARCL_RAM_RECORD * sizeof(float) : 0;
  S.off_obs = S.off_ram + S.ram_bytes;
  S.obs_bytes = (c.num_frames > 1 && c.ram_obs != 2)
                    ? (uint64_t)L.A * c.num_frames * L.obs_channels * c.grid_size * c.grid_size * esz : 0;
  S.slot_bytes = align_to(S.off_obs + align_to(S.obs_bytes, 16), 128);
}

// FNV-1a 64 over the layout without cap_replay and the configuration fields that shape a game state (not n_instances, the caps
// of the layout, device or instance_base: a pool moves between batch sizes, shards and devices)
static uint64_t config_fingerprint(const agarcl_cfg& c, const agarcl_layout& L) {
  uint64_t h = 0xcbf29ce484222325ull;
  auto mix = [&h](const void* p, size_t n) {
    for (size_t k = 0; k < n; k++) { h ^= ((const uint8_t*)p)[k]; h *= 0x100000001b3ull; }
  };
  agarcl_layout l = L;
  l.cap_replay = 0;
  mix(&l, sizeof(l));
  const int32_t f[] = {c.num_agents, c.ticks_per_step, c.arena_size, c.pellet_regen, c.num_pellets, c.num_viruses, c.num_bots,
                       c.reward_type, c.c_death, c.mode_number, c.num_frames, c.grid_size, c.observe_cells, c.observe_others,
                       c.observe_viruses, c.observe_pellets, c.obs_dtype, c.strict_reference, c.rng_mode, c.ram_obs};
  mix(f, sizeof(f));
  if (c.task_modes) mix(&c.task_modes, sizeof(c.task_modes));  // (pools of batches without tasks keep their fingerprint)
  return h;
}

extern "C" int agarcl_snapshot_slot_bytes(const agarcl_cfg* c, int64_t* out) {
  if (!c || !out) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  agarcl_layout L;
  int rc = agarcl_make_layout(c, &L);
  if (rc != AGARCL_OK) return rc;
  ag::SnapLayout S;
  snapshot_layout(*c, L, S);
  *out = (int64_t)S.slot_bytes;
  return AGARCL_OK;
}

extern "C" int agarcl_batch_destroy(agarcl_batch* b) {
  delete b;
  return AGARCL_OK;
}

extern "C" int agarcl_batch_create(const agarcl_cfg* cfg, agarcl_batch** out) {
  if (!cfg || !out) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  *out = nullptr;
  if (cfg->n_instances < 1) return agarcl_set_error(AGARCL_ERR_INVALID, "n_instances must be >= 1");
  agarcl_layout L;
  int rc = agarcl_make_layout(cfg, &L);
  if (rc != AGARCL_OK) return rc;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return agarcl_set_error(AGARCL_ERR_CUDA, "no CUDA device: agarcl_b200 has no CPU path (%s)", cudaGetErrorString(e));
  if (cfg->device < 0 || cfg->device >= ndev) return agarcl_set_error(AGARCL_ERR_INVALID, "device %d out of range", cfg->device);
  CK(cudaSetDevice(cfg->device));
  std::unique_ptr<agarcl_batch> b(new (std::nothrow) agarcl_batch());  // (frees whatever was made when a step below fails)
  if (!b) return agarcl_set_error(AGARCL_ERR_NOMEM, "out of host memory");
  b->cfg = *cfg;
  b->L = L;
  b->N = cfg->n_instances;
  b->A = L.A;
  b->G = cfg->grid_size;
  b->C = L.obs_channels;
  b->frames = cfg->num_frames;
  b->knobs = read_knobs();
  snapshot_layout(*cfg, L, b->snap);
  b->fingerprint = config_fingerprint(*cfg, L);
  CK(ag::setup_step(b->knobs.warps, b->step_launch));
  if (cfg->ram_obs) CK(ag::setup_ram(L, b->step_launch.smem_optin));
  CK(ag::setup_draw_views());
  b->obs_elems = (size_t)b->N * b->A * b->frames * b->C * b->G * b->G;
  b->obs_bytes = b->obs_elems * (cfg->obs_dtype == AGARCL_OBS_I16 ? 2 : 4);
  // spatial hash resolution: about 3 pellets per hash cell, 4..64 cells per side
  int hg = (int)std::floor(std::sqrt((double)L.cap_pellets / b->knobs.hash_per_cell));
  b->HG = hg < 4 ? 4 : (hg > 64 ? 64 : hg);
  b->smem_per_warp = ag::make_smem_offsets(L, b->HG, b->so);
  if ((size_t)b->smem_per_warp + 2 * ag::kZeroTileBytes > (size_t)b->step_launch.smem_optin)  // (room for one warp with both tiles at full size)
    return agarcl_set_error(AGARCL_ERR_INVALID, "configuration needs %u B of shared memory per instance (too many pellets/viruses)", b->smem_per_warp);
  const size_t NA = (size_t)b->N * b->A, lut_bytes = AGARCL_LUT_SIZE * sizeof(float);
  if ((rc = alloc(b->d_state, (size_t)b->N * L.stride, 0)) || (rc = alloc(b->d_obs, b->obs_bytes, 0)) ||
      (rc = alloc(b->d_rewards, NA * sizeof(double), 0)) || (rc = alloc(b->d_dones, NA, 0)) || (rc = alloc(b->d_before, NA * sizeof(float))) ||
      (rc = alloc(b->d_dxdy, NA * 2 * sizeof(float), 0)) || (rc = alloc(b->d_act, NA * sizeof(int32_t), 0)) ||
      (rc = alloc(b->d_seeds, (size_t)b->N * sizeof(uint64_t))) || (rc = alloc(b->d_mask, (size_t)b->N)) ||
      (rc = alloc(b->d_tickets, 2 * sizeof(uint32_t), 0)) || (rc = alloc(b->d_cost, (size_t)b->N * sizeof(uint32_t))) ||
      (rc = alloc(b->d_perm, (size_t)b->N * sizeof(uint32_t))) || (rc = alloc(b->d_sched, 2 * sizeof(uint32_t))) ||
      (rc = alloc(b->d_fresh, (size_t)b->N, 1)) || (rc = alloc(b->d_flagbuf, 33 * sizeof(uint32_t))) ||
      (rc = alloc(b->d_snap_result, (size_t)b->N, 0)) || (rc = alloc(b->d_snap_restored, (size_t)b->N, 0)) ||
      (rc = alloc(b->d_start_slot, (size_t)b->N * sizeof(int32_t))) || (rc = alloc(b->d_start_result, (size_t)b->N, 0)) ||
      (rc = alloc(b->d_spawn, (size_t)b->N)) ||
      (L.cap_replay > 0 && (rc = alloc(b->d_replay, (size_t)b->N * L.cap_replay * sizeof(float), 0))) ||
      (cfg->ram_obs && (rc = alloc(b->d_ram, (size_t)b->N * L.P * AGARCL_RAM_RECORD * sizeof(float), 0))) ||
      (cfg->pixel_obs && (rc = alloc(b->d_pixels, b->pixel_bytes = NA * cfg->pixel_obs * cfg->pixel_obs * 3, 0))) ||
      (rc = alloc(b->d_lut_radius, lut_bytes)) || (rc = alloc(b->d_lut_speed, lut_bytes)) || (rc = alloc(b->d_lut_split, lut_bytes)))
    return rc;
  { const uint32_t init[2] = {1u, 0u}; CK(cudaMemcpy(b->d_sched, init, sizeof(init), cudaMemcpyHostToDevice)); }
  if (cfg->task_modes) {  // every instance starts on mode_number with the batch's step limit
    const size_t bytes = (size_t)b->N * sizeof(int32_t);
    if ((rc = alloc(b->d_task_mode, bytes)) || (rc = alloc(b->d_task_max_steps, bytes)) || (rc = alloc(b->d_next_mode, bytes)) ||
        (rc = alloc(b->d_next_max_steps, bytes)) || (rc = alloc(b->d_task_result, (size_t)b->N, 0)))
      return rc;
    const std::vector<int32_t> modes((size_t)b->N, cfg->mode_number), limits((size_t)b->N, -1);
    CK(cudaMemcpy(b->d_task_mode, modes.data(), bytes, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(b->d_next_mode, modes.data(), bytes, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(b->d_task_max_steps, limits.data(), bytes, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(b->d_next_max_steps, limits.data(), bytes, cudaMemcpyHostToDevice));
    // game sizes: the configured counts are the maxima, which every instance plays until it is given others
    b->size_lim = {cfg->num_bots, cfg->num_pellets, cfg->num_viruses, !(cfg->task_modes & 1), task_bot_counts(cfg, &L)};
    DevBuf<int32_t>* bufs[6] = {&b->d_bots, &b->d_pellets, &b->d_viruses, &b->d_next_bots, &b->d_next_pellets, &b->d_next_viruses};
    for (int k = 0; k < 6; k++) {
      if ((rc = alloc(*bufs[k], bytes))) return rc;
      const std::vector<int32_t> v((size_t)b->N, k % 3 == 0 ? cfg->num_bots : k % 3 == 1 ? cfg->num_pellets : cfg->num_viruses);
      CK(cudaMemcpy(*bufs[k], v.data(), bytes, cudaMemcpyHostToDevice));
    }
    if ((rc = alloc(b->d_size_result, (size_t)b->N, 0))) return rc;
  }
  b->cur_dxdy = b->d_dxdy;
  b->cur_act = b->d_act;
  // lookup tables of functions of an integer mass, computed with the host libm the reference uses
  {
    std::vector<float> rad(AGARCL_LUT_SIZE), spd(AGARCL_LUT_SIZE), spl(AGARCL_LUT_SIZE);
    for (uint32_t m = 0; m < AGARCL_LUT_SIZE; m++) {
      rad[m] = (float)std::sqrt((double)m / 1.0 / M_PI);                  // radius_conversion, core/utils.hpp:8-11
      spd[m] = (float)(300 / std::pow((double)m, 0.439));                 // max_speed, Engine.hpp:1300-1302
      double v = 3 * std::pow((double)spd[m], 1.2);                       // split_speed, Engine.hpp:1296-1298
      v = (130.0 < v) ? 130.0 : v;
      v = (v < 20.0) ? 20.0 : v;
      spl[m] = (float)v;
    }
    CK(cudaMemcpy(b->d_lut_radius, rad.data(), lut_bytes, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(b->d_lut_speed, spd.data(), lut_bytes, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(b->d_lut_split, spl.data(), lut_bytes, cudaMemcpyHostToDevice));
    b->T.radius = b->d_lut_radius;
    b->T.max_speed = b->d_lut_speed;
    b->T.split_speed = b->d_lut_split;
    b->T.anti_team[0] = 1.0f;
    for (int n = 1; n <= AGARCL_VET_CAP; n++) b->T.anti_team[n] = (float)std::pow(1.1, (double)(n - 1));  // Engine.hpp:567
  }
  b->seeds.resize(b->N);
  for (int i = 0; i < b->N; i++) b->seeds[i] = (uint64_t)(cfg->instance_base + i);
  b->max_draws_per_step = 2 * ((int64_t)L.cap_pellets + L.cap_viruses + L.P);  // regen deficits + respawns of one step; a whole reset
  if (cfg->rng_mode == AGARCL_RNG_MT19937) {
    // an UNSEEDED reference environment draws from std::random_device (GameState.hpp:59): so does an unseeded batch
    if ((int64_t)L.cap_replay <= b->max_draws_per_step)
      return agarcl_set_error(AGARCL_ERR_INVALID, "cap_replay %d cannot hold the draws of one step (%lld): raise cfg.cap_replay", L.cap_replay,
                              (long long)b->max_draws_per_step);
    b->gens.resize(b->N);
    b->filled.assign(b->N, 0);
    std::random_device rd;
    for (int i = 0; i < b->N; i++) {
      uint64_t s0;
      try { s0 = rd(); } catch (...) { s0 = (uint64_t)(cfg->instance_base + i) * 0x9E3779B97F4A7C15ull + 1u; }
      b->seeds[i] = s0 & 0xffffffffull;
      if ((rc = mt_restart(b.get(), i, b->seeds[i], 0))) return rc;
    }
    b->draw_budget = L.cap_replay;
  }
  CK(cudaMemcpy(b->d_seeds, b->seeds.data(), b->N * sizeof(uint64_t), cudaMemcpyHostToDevice));
  CK(cudaDeviceSynchronize());
  *out = b.release();
  return AGARCL_OK;
}

extern "C" int agarcl_batch_get_layout(const agarcl_batch* b, agarcl_layout* out) {
  if (!b || !out) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  *out = b->L;
  return AGARCL_OK;
}

extern "C" int agarcl_batch_seed(agarcl_batch* b, const uint64_t* seeds) {
  if (!b || !seeds) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  CK(cudaSetDevice(b->cfg.device));
  for (int i = 0; i < b->N; i++) b->seeds[i] = seeds[i];
  CK(cudaMemcpy(b->d_seeds, b->seeds.data(), b->N * sizeof(uint64_t), cudaMemcpyHostToDevice));
  if (b->cfg.rng_mode == AGARCL_RNG_MT19937) {
    CK(cudaDeviceSynchronize());
    for (int i = 0; i < b->N; i++) {
      int rc = mt_restart(b, i, seeds[i], 0);
      if (rc) return rc;
    }
    b->draw_budget = b->L.cap_replay;
  }
  CK(cudaMemset(b->d_fresh, 1, (size_t)b->N));  // seed() restarts the stream: the next reset draws from index 0
  return AGARCL_OK;
}

extern "C" int agarcl_batch_set_replay(agarcl_batch* b, int32_t instance, const float* draws, int32_t n) {
  if (!b || !draws) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  if (instance < 0 || instance >= b->N) return agarcl_set_error(AGARCL_ERR_INVALID, "instance out of range");
  if (!b->d_replay) return agarcl_set_error(AGARCL_ERR_STATE, "batch was not created with a replay rng_mode");
  if (n > b->L.cap_replay) n = b->L.cap_replay;
  CK(cudaSetDevice(b->cfg.device));
  CK(cudaMemcpy(b->d_replay + (size_t)instance * b->L.cap_replay, draws, (size_t)n * sizeof(float), cudaMemcpyHostToDevice));
  CK(cudaMemset(b->d_fresh + instance, 1, 1));  // a new stream starts at its first draw
  return AGARCL_OK;
}

static int render_frame(agarcl_batch* b, int frame, cudaStream_t s, int pre_respawn, int skip_zero = 0,
                        const uint8_t* d_mask = nullptr) {
  ag::ObsParams P;
  fill_obs_params(b, P, frame, pre_respawn, skip_zero);
  P.mask = d_mask;
  CK(ag::launch_obs(P, s));
  return AGARCL_OK;
}

static int render_ram(agarcl_batch* b, cudaStream_t s, int pre_respawn) {
  ag::RamParams P;
  P.L = b->L;
  P.T = b->T;
  P.state = b->d_state;
  P.ram = b->d_ram;
  P.N = b->N;
  P.G = b->G;
  P.pre_respawn = pre_respawn;
  P.pid_base = b->pid_base;
  CK(ag::launch_ram(P, s));
  return AGARCL_OK;
}

static ag::DrawParams draw_params(const agarcl_batch* b, int view, int size, const int32_t* d_src, int n, uint8_t* d_out) {
  ag::DrawParams P;
  P.L = b->L;
  P.radius = b->T.radius;
  P.state = b->d_state;
  P.out = d_out;
  P.src = d_src;
  P.n = n;
  P.S = size;
  P.view = view;
  P.N = b->N;
  P.W = (float)b->cfg.arena_size;
  P.pre_respawn = 0;
  P.mask = nullptr;
  return P;
}

// The pixel observation of the instances with d_mask != 0 (nullptr: all); pre_respawn 1 shows the step's moment, as k_obs does
static int render_pixels(agarcl_batch* b, cudaStream_t s, int pre_respawn, const uint8_t* d_mask) {
  ag::DrawParams P = draw_params(b, AGARCL_DRAW_AGENT, b->cfg.pixel_obs, nullptr, b->N * b->A, b->d_pixels);
  P.pre_respawn = pre_respawn;
  P.mask = d_mask;
  CK(ag::launch_draw_views(P, s));
  return AGARCL_OK;
}

extern "C" int agarcl_batch_pixels(agarcl_batch* b, uint8_t** d_pixels, uint8_t** d_final_pixels, int64_t shape[4]) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  if (!b->cfg.pixel_obs) return agarcl_set_error(AGARCL_ERR_STATE, "batch was created without cfg.pixel_obs");
  if (d_pixels) *d_pixels = b->d_pixels;
  if (d_final_pixels) *d_final_pixels = b->keep_final ? b->d_final_pixels.get() : nullptr;
  if (shape) { shape[0] = (int64_t)b->N * b->A; shape[1] = shape[2] = b->cfg.pixel_obs; shape[3] = 3; }
  return AGARCL_OK;
}

extern "C" int agarcl_batch_ram(agarcl_batch* b, float** dev_ptr, int64_t shape[3]) {
  if (!b || !dev_ptr) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  if (!b->d_ram) return agarcl_set_error(AGARCL_ERR_STATE, "batch was created without cfg.ram_obs");
  *dev_ptr = b->d_ram;
  if (shape) { shape[0] = b->N; shape[1] = b->L.P; shape[2] = AGARCL_RAM_RECORD; }
  return AGARCL_OK;
}

extern "C" int agarcl_batch_ram_host(agarcl_batch* b, float* out) {
  if (!b || !out) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  if (!b->d_ram) return agarcl_set_error(AGARCL_ERR_STATE, "batch was created without cfg.ram_obs");
  CK(cudaSetDevice(b->cfg.device));
  CK(cudaMemcpy(out, b->d_ram, (size_t)b->N * b->L.P * AGARCL_RAM_RECORD * sizeof(float), cudaMemcpyDeviceToHost));
  return AGARCL_OK;
}

extern "C" int agarcl_batch_render_ram(agarcl_batch* b, void* stream) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  if (!b->d_ram) return agarcl_set_error(AGARCL_ERR_STATE, "batch was created without cfg.ram_obs");
  CK(cudaSetDevice(b->cfg.device));
  return render_ram(b, (cudaStream_t)stream, 0);
}

extern "C" int agarcl_batch_render(agarcl_batch* b, void* stream) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  CK(cudaSetDevice(b->cfg.device));
  return render_frame(b, b->frames - 1, (cudaStream_t)stream, 0);
}

static ag::EpisodeParams episode_params(const agarcl_batch* b) {
  ag::EpisodeParams E;
  E.dones = b->d_dones; E.rewards = b->d_rewards;
  E.done_out = b->d_done_out; E.reset_mask = b->d_reset_mask; E.steps = b->d_steps;
  E.ret = b->d_ret; E.final_ret = b->d_final_ret; E.final_len = b->d_final_len;
  E.clear_mask = nullptr;
  E.task_max_steps = b->d_task_max_steps;
  E.N = b->N; E.A = b->A; E.max_steps = b->max_steps;
  E.reset = b->autoreset_reset ? 1 : 0;
  E.clear = 0;
  return E;
}

static ag::SnapParams snapshot_params(const agarcl_batch* b, const void* pool, int64_t pool_slots);

static ag::ArchiveParams archive_params(const agarcl_batch* b, const uint8_t* mask) {
  const Archive& a = *b->archive;
  ag::ArchiveParams P;
  P.L = b->L;
  P.state = b->d_state;
  P.dones = b->d_dones;
  P.rewards = b->d_rewards;
  P.ret = b->d_ret;
  P.steps = b->d_steps;
  P.N = b->N; P.A = b->A; P.agent = a.cfg.agent; P.n = a.cfg.cells_per_side; P.K = (int32_t)a.K;
  P.instance_base = b->cfg.instance_base;
  P.W = (float)b->cfg.arena_size;
  P.seed = a.cfg.seed;
  P.cell_of = a.cell_of; P.base_score = a.base_score; P.base_length = a.base_length;
  P.cand_key = a.cand_key; P.cand_s = a.cand_s; P.cand_l = a.cand_l; P.save_slot = a.save_slot; P.draws = a.draws;
  P.key_entry = a.key_entry; P.visits = a.visits; P.best_s = a.best_s; P.best_li = a.best_li;
  P.entry_key = a.entry_key; P.entry_score = a.entry_score; P.entry_length = a.entry_length; P.entry_chosen = a.entry_chosen;
  P.prefix = a.prefix; P.counters = a.counters;
  P.mask = mask;
  P.start_slot = b->d_start_slot;
  P.start_result = (b->start_pool && b->start_pool == a.pool) ? b->d_start_result.get() : nullptr;
  return P;
}

// The masked reset: instances with d_mask[i] != 0 (device memory; nullptr = all).  Everything is enqueued on `s`; the
// host neither reads the mask nor waits, except for refill_replay's draw cursor read-back under AGARCL_RNG_MT19937.
// clear_episode: restart the episode counters of the reset instances (agarcl_batch_step_autoreset has done so already).
// With start states, k_snapshot first loads the slots of the instances that have one and k_reset spawns the others; every
// launch behind it treats both alike (mask dm).
static int reset_impl(agarcl_batch* b, const uint8_t* dm, cudaStream_t s, bool clear_episode) {
  CK(cudaSetDevice(b->cfg.device));
  const uint8_t* spawn = dm;
  if (b->archive && b->archive->cfg.select) CK(ag::launch_archive_select(archive_params(b, dm), s));  // (the archive owns the table)
  if (b->start_pool) {
    ag::SnapParams S = snapshot_params(b, b->start_pool, b->start_pool_slots);
    S.slot_of = b->d_start_slot;
    S.result = b->d_start_result;
    S.mask = dm;
    S.spawn = b->d_spawn;
    S.next_max_steps = b->d_next_max_steps;
    CK(ag::launch_snapshot_start(S, s));
    spawn = b->d_spawn;
  }
  if (b->archive) CK(ag::launch_archive_base(archive_params(b, dm), s));
  ag::ResetParams P;
  P.L = b->L;
  P.T = b->T;
  P.state = b->d_state;
  P.mask = spawn;
  P.seeds = b->d_seeds;
  P.replay = b->d_replay;
  P.fresh = b->d_fresh;
  P.dones = b->d_dones;
  P.N = b->N;
  P.instance_base = b->cfg.instance_base;
  P.rng_mode = b->cfg.rng_mode;
  P.num_pellets = b->cfg.num_pellets;
  P.num_viruses = b->cfg.num_viruses;
  P.task_mode = b->d_task_mode;
  P.task_max_steps = b->d_task_max_steps;
  P.next_mode = b->d_next_mode;
  P.next_max_steps = b->d_next_max_steps;
  P.sizes = task_sizes_of(b);
  P.W = (float)b->cfg.arena_size;
  if (b->cfg.strict_reference && !dm) {
    // BaseEnvironment::reset of every instance (BaseEnvironment.hpp:179-197): players.clear(), then add_player for the agents and
    // the bots with the pids that follow the last episode's; a masked reset (one instance of a vector env) keeps the batch's order
    b->pmap.clear();
    b->pid_base = (int32_t)b->next_pid;
    for (int p = 0; p < b->L.P; p++) b->pmap.insert(std::make_pair(b->next_pid++, p));
    int k = 0;
    for (auto& kv : b->pmap) b->L.order[k++] = kv.second;
    P.L = b->L;
  }
  CK(ag::launch_reset(P, s));
  b->was_reset = true;
  if (clear_episode && b->autoreset) {
    ag::EpisodeParams E = episode_params(b);
    E.clear = 1;
    E.clear_mask = dm;
    CK(ag::launch_episode(E, s));
  }
  { int rc = refill_replay(b, s); if (rc) return rc; }
  // (a masked reset touches only the records and observations of the instances it resets)
  auto clear = [&](void* buf, size_t bytes) -> cudaError_t {
    if (!dm) return cudaMemsetAsync(buf, 0, bytes, s);
    return ag::launch_masked_bytes(buf, nullptr, bytes / (size_t)b->N, dm, b->N, s);
  };
  if (b->d_ram)  // GoBiggerEnvironment::reset ends with observation.clear() (GoBiggerEnvironment.hpp:698-702)
    CK(clear(b->d_ram, (size_t)b->N * b->L.P * AGARCL_RAM_RECORD * sizeof(float)));
  // the reference ends reset() with _partial_observation (BaseEnvironment.hpp:202-203)
  if (b->cfg.pixel_obs) return render_pixels(b, s, 0, dm);
  if (!renders_grid(b)) return AGARCL_OK;  // no grid observation in this mode
  if (b->cfg.strict_reference) {
    CK(clear(b->d_obs, b->obs_bytes));
    int frame = 0 - (b->cfg.ticks_per_step - b->frames);
    if (frame >= 0) return render_frame(b, frame, s, 0, 0, dm);
    return AGARCL_OK;
  }
  if (b->frames > 1) CK(clear(b->d_obs, b->obs_bytes));
  return render_frame(b, b->frames - 1, s, 0, 0, dm);
}

extern "C" int agarcl_batch_reset(agarcl_batch* b, const uint8_t* mask, void* stream) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  CK(cudaSetDevice(b->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  if (mask) CK(cudaMemcpyAsync(b->d_mask, mask, b->N, cudaMemcpyHostToDevice, s));
  return reset_impl(b, mask ? b->d_mask.get() : nullptr, s, true);
}

extern "C" int agarcl_batch_reset_device(agarcl_batch* b, const uint8_t* d_mask, void* stream) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  return reset_impl(b, d_mask, (cudaStream_t)stream, true);
}

extern "C" int agarcl_batch_set_actions(agarcl_batch* b, const float* dxdy, const int32_t* act, int on_device, void* stream) {
  if (!b || !dxdy || !act) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  CK(cudaSetDevice(b->cfg.device));
  const size_t NA = (size_t)b->N * b->A;
  if (on_device) {
    b->cur_dxdy = dxdy;
    b->cur_act = act;
  } else {
    cudaStream_t s = (cudaStream_t)stream;
    CK(cudaMemcpyAsync(b->d_dxdy, dxdy, NA * 2 * sizeof(float), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(b->d_act, act, NA * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    b->cur_dxdy = b->d_dxdy;
    b->cur_act = b->d_act;
  }
  return AGARCL_OK;
}

// One env-step of every instance.  `lists_to`: when the step is the single fused kernel, it also leaves the transfer lists of
// that HostMirror in host memory (*lists_made = true); nullptr: no lists.
static int step_impl(agarcl_batch* b, cudaStream_t s, ag::HostMirror* lists_to, bool* lists_made) {
  if (lists_made) *lists_made = false;
  if (!b->was_reset) return agarcl_set_error(AGARCL_ERR_STATE, "step() before reset()");
  CK(cudaSetDevice(b->cfg.device));
  ag::SimParams P;
  fill_sim_params(b, P);
  const int tps = b->cfg.ticks_per_step;
  int launches = 0;
  if (b->cfg.strict_reference) {
    // quirk Q11: one _partial_observation(agent, 0) after all ticks, frame_index = -(tps - num_frames)
    P.n_ticks = tps; P.do_begin = 1; P.do_end = 1;
    CK(cudaMemsetAsync(b->d_obs, 0, b->obs_bytes, s));  // _step_hook: clear_data
    CK(ag::launch_step(P, b->step_launch, s)); launches++;
    int frame = 0 - (tps - b->frames);
    if (frame >= 0) { int rc = render_frame(b, frame, s, 1); if (rc) return rc; launches++; }
  } else if (!renders_grid(b) || b->frames == 1) {
    // one k_step runs every tick of the step; a grid frame (none with the structured observation only, agario-ram-v0, or with
    // pixels) is finished by k_step itself or by k_obs behind it
    const bool grid = renders_grid(b);
    P.n_ticks = tps; P.do_begin = 1; P.do_end = 1;
    const int fused = grid && fuse_obs_clear(b, P, 0) ? 1 : 0;
    if (lists_to && kernel_writes_lists(b)) {
      P.pk = ag::mirror_pack_out(lists_to);
      *lists_made = true;
    }
    const bool sorted = P.tick_barrier && b->knobs.sort_schedule;
    if (sorted) { P.cost = b->d_cost; P.perm = b->perm_valid ? b->d_perm.get() : nullptr; P.sched = b->knobs.auto_schedule ? b->d_sched.get() : nullptr; }
    if (b->timing) { if (b->ev_used >= 3 * 2048) collect_timing(b); CK(cudaEventRecord(next_event(b), s)); }
    CK(ag::launch_step(P, b->step_launch, s)); launches++;
    if (b->timing) CK(cudaEventRecord(next_event(b), s));
    if (sorted) { CK(ag::launch_order(b->d_cost, b->d_perm, b->N, P.sched, s)); b->perm_valid = true; launches++; }
    if (grid) {
      if (!P.obs_finish) { int rc = render_frame(b, 0, s, 1, fused); if (rc) return rc; launches++; }
      if (b->timing) CK(cudaEventRecord(next_event(b), s));
    }
  } else {
    // the last num_frames ticks of the step each contribute one frame (the documented intent of
    // GridEnvironment::_partial_observation, GridEnvironment.hpp:413-433)
    if (b->frames > tps) CK(cudaMemsetAsync(b->d_obs, 0, b->obs_bytes, s));
    for (int t = 0; t < tps; t++) {
      P.n_ticks = 1; P.do_begin = (t == 0); P.do_end = 0;
      CK(ag::launch_step(P, b->step_launch, s)); launches++;
      int frame = t - (tps - b->frames);
      if (frame >= 0) { int rc = render_frame(b, frame, s, 1); if (rc) return rc; launches++; }
    }
    P.n_ticks = 0; P.do_begin = 0; P.do_end = 1;
    CK(ag::launch_step(P, b->step_launch, s)); launches++;
  }
  if (b->d_ram) {
    int rc = render_ram(b, s, 1); if (rc) return rc; launches++;
    if (b->timing && b->cfg.ram_obs == 2) CK(cudaEventRecord(next_event(b), s));  // (k_ram is this mode's observation kernel)
  }
  if (b->cfg.pixel_obs) {
    int rc = render_pixels(b, s, 1, nullptr); if (rc) return rc; launches++;
    if (b->timing) CK(cudaEventRecord(next_event(b), s));
  }
  b->launches_last_step = launches;
  return refill_replay(b, s);
}

extern "C" int agarcl_batch_step(agarcl_batch* b, void* stream) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  return step_impl(b, (cudaStream_t)stream, nullptr, nullptr);
}

extern "C" int agarcl_batch_set_autoreset(agarcl_batch* b, int32_t max_steps, int32_t keep_final_obs, int32_t reset) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  if (max_steps < 0) return agarcl_set_error(AGARCL_ERR_INVALID, "max_steps must be >= 0 (0: no step limit)");
  if (keep_final_obs && !reset) return agarcl_set_error(AGARCL_ERR_INVALID, "keep_final_obs needs reset: nothing is overwritten without one");
  if (!reset && b->archive) return agarcl_set_error(AGARCL_ERR_STATE, "an attached archive needs reset: detach it first");
  CK(cudaSetDevice(b->cfg.device));
  const size_t NA = (size_t)b->N * b->A;
  int rc;
  if ((rc = alloc(b->d_done_out, NA, 0)) || (rc = alloc(b->d_reset_mask, (size_t)b->N, 0)) ||
      (rc = alloc(b->d_steps, (size_t)b->N * sizeof(int64_t), 0)) || (rc = alloc(b->d_final_len, (size_t)b->N * sizeof(int64_t), 0)) ||
      (rc = alloc(b->d_ret, NA * sizeof(double), 0)) || (rc = alloc(b->d_final_ret, NA * sizeof(double), 0)))
    return rc;
  if (keep_final_obs) {
    if (renders_grid(b) && (rc = alloc(b->d_final_obs, b->obs_bytes, 0))) return rc;
    if (b->cfg.pixel_obs && (rc = alloc(b->d_final_pixels, b->pixel_bytes, 0))) return rc;
    if (b->d_ram && (rc = alloc(b->d_final_ram, (size_t)b->N * b->L.P * AGARCL_RAM_RECORD * sizeof(float), 0))) return rc;
  }
  // every instance starts counting here
  CK(cudaMemset(b->d_steps, 0, (size_t)b->N * sizeof(int64_t)));
  CK(cudaMemset(b->d_ret, 0, NA * sizeof(double)));
  CK(cudaDeviceSynchronize());  // (the zeroing is done before a step on any stream can read the counters)
  b->autoreset = true;
  b->autoreset_reset = reset != 0;
  b->keep_final = keep_final_obs != 0;
  b->max_steps = max_steps;
  return AGARCL_OK;
}

extern "C" int agarcl_batch_step_autoreset(agarcl_batch* b, void* stream) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  if (!b->autoreset) return agarcl_set_error(AGARCL_ERR_STATE, "agarcl_batch_step_autoreset before agarcl_batch_set_autoreset");
  cudaStream_t s = (cudaStream_t)stream;
  int rc = step_impl(b, s, nullptr, nullptr);
  if (rc) return rc;
  if (b->archive) {  // the archive sees the step's games and counters before the bookkeeping and the reset
    const Archive& a = *b->archive;
    CK(ag::launch_archive_update(archive_params(b, nullptr), s));
    ag::SnapParams S = snapshot_params(b, a.pool, a.K);
    S.src = a.src;
    S.slot = a.save_slot;
    CK(ag::launch_snapshot_save(S, b->N, s));
  }
  CK(ag::launch_episode(episode_params(b), s));
  if (!b->autoreset_reset) return AGARCL_OK;
  if (b->keep_final) {  // the observation the finished episode ended on, before the reset overwrites it
    if (b->d_final_obs) CK(ag::launch_masked_bytes(b->d_final_obs, b->d_obs, b->obs_bytes / (size_t)b->N, b->d_reset_mask, b->N, s));
    if (b->d_final_pixels)
      CK(ag::launch_masked_bytes(b->d_final_pixels, b->d_pixels, b->pixel_bytes / (size_t)b->N, b->d_reset_mask, b->N, s));
    if (b->d_final_ram)
      CK(ag::launch_masked_bytes(b->d_final_ram, b->d_ram, (size_t)b->L.P * AGARCL_RAM_RECORD * sizeof(float), b->d_reset_mask, b->N, s));
  }
  return reset_impl(b, b->d_reset_mask, s, false);
}

extern "C" int agarcl_batch_episode(agarcl_batch* b, agarcl_episode* out) {
  if (!b || !out) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  if (!b->autoreset) return agarcl_set_error(AGARCL_ERR_STATE, "no episode bookkeeping: call agarcl_batch_set_autoreset first");
  out->done_out = b->d_done_out;
  out->reset_mask = b->d_reset_mask;
  out->steps = b->d_steps;
  out->final_return = b->d_final_ret;
  out->final_length = b->d_final_len;
  out->final_obs = b->keep_final ? b->d_final_obs.get() : nullptr;
  out->final_ram = b->keep_final ? b->d_final_ram.get() : nullptr;
  return AGARCL_OK;
}

extern "C" int agarcl_batch_set_timing(agarcl_batch* b, int enable) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  collect_timing(b);
  b->timing = enable != 0;
  b->acc_sim_ms = b->acc_obs_ms = 0.0;
  b->acc_steps = 0;
  return AGARCL_OK;
}
extern "C" int agarcl_batch_get_timing(agarcl_batch* b, double* sim_ms, double* obs_ms, int32_t* steps) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  collect_timing(b);
  if (sim_ms) *sim_ms = b->acc_sim_ms;
  if (obs_ms) *obs_ms = b->acc_obs_ms;
  if (steps) *steps = b->acc_steps;
  b->acc_sim_ms = b->acc_obs_ms = 0.0;
  b->acc_steps = 0;
  return AGARCL_OK;
}

extern "C" int agarcl_batch_launches_per_step(const agarcl_batch* b) { return b ? b->launches_last_step : 0; }

extern "C" int agarcl_batch_costs(agarcl_batch* b, void* stream, uint32_t* out) {
  if (!b || !out) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  if (!b->d_cost) return agarcl_set_error(AGARCL_ERR_STATE, "this batch keeps no per-instance costs");
  CK(cudaSetDevice(b->cfg.device));
  CK(cudaMemcpyAsync(out, b->d_cost, sizeof(uint32_t) * (size_t)b->N, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  CK(cudaStreamSynchronize((cudaStream_t)stream));
  return AGARCL_OK;
}

extern "C" int agarcl_selftest_std_sort(const float* ys, int32_t n, uint16_t* order_out) {
  if (n < 0 || n > 65535 || (n > 0 && (!ys || !order_out))) return agarcl_set_error(AGARCL_ERR_INVALID, "bad keys / count");
  CK(ag::selftest_std_sort(ys, n, order_out));
  return AGARCL_OK;
}

extern "C" int agarcl_batch_flags(agarcl_batch* b, void* stream, uint32_t* or_all, uint32_t counts[32]) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  CK(cudaSetDevice(b->cfg.device));
  cudaStream_t s = (cudaStream_t)stream;
  CK(ag::launch_flags(b->d_state, b->L, b->N, b->d_flagbuf, s));
  uint32_t h[33];
  CK(cudaMemcpyAsync(h, b->d_flagbuf, sizeof(h), cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  if (or_all) *or_all = h[32];
  if (counts) std::memcpy(counts, h, 32 * sizeof(uint32_t));
  return AGARCL_OK;
}

extern "C" int agarcl_batch_obs(agarcl_batch* b, void** dev_ptr, int64_t shape[4], int32_t* dtype) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  if (dev_ptr) *dev_ptr = b->d_obs;
  if (shape) { shape[0] = (int64_t)b->N * b->A; shape[1] = (int64_t)b->frames * b->C; shape[2] = b->G; shape[3] = b->G; }
  if (dtype) *dtype = b->cfg.obs_dtype;
  return AGARCL_OK;
}
extern "C" int agarcl_batch_rewards(agarcl_batch* b, double** dev_ptr) {
  if (!b || !dev_ptr) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  *dev_ptr = b->d_rewards;
  return AGARCL_OK;
}
extern "C" int agarcl_batch_dones(agarcl_batch* b, uint8_t** dev_ptr) {
  if (!b || !dev_ptr) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  *dev_ptr = b->d_dones;
  return AGARCL_OK;
}

// The host paths of the grid observation: refused for a pixel batch, which renders no grid frame
static int refuse_pixels(const agarcl_batch* b, const char* what) {
  if (b->cfg.pixel_obs) return agarcl_set_error(AGARCL_ERR_STATE, "%s serves the grid observation: a pixel batch (cfg.pixel_obs) has none", what);
  return AGARCL_OK;
}

extern "C" int agarcl_batch_step_host(agarcl_batch* b, const float* dxdy, const int32_t* act, void* obs_out,
                                      double* rewards_out, uint8_t* dones_out) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  if (int rc = refuse_pixels(b, "agarcl_batch_step_host")) return rc;
  int rc = agarcl_batch_set_actions(b, dxdy, act, 0, nullptr);
  if (rc) return rc;
  rc = agarcl_batch_step(b, nullptr);
  if (rc) return rc;
  const size_t NA = (size_t)b->N * b->A;
  if (obs_out) CK(cudaMemcpyAsync(obs_out, b->d_obs, b->obs_bytes, cudaMemcpyDeviceToHost, nullptr));
  if (rewards_out) CK(cudaMemcpyAsync(rewards_out, b->d_rewards, NA * sizeof(double), cudaMemcpyDeviceToHost, nullptr));
  if (dones_out) CK(cudaMemcpyAsync(dones_out, b->d_dones, NA, cudaMemcpyDeviceToHost, nullptr));
  CK(cudaStreamSynchronize(nullptr));
  return AGARCL_OK;
}

// ---- host-resident observation mirror (mirror.cu): b->mirror, or its lists-only twin b->lists, created on first use
static int ensure_mirror(agarcl_batch* b, bool lists_only = false) {
  ag::HostMirror*& m = lists_only ? b->lists : b->mirror;
  if (m) return AGARCL_OK;
  CK(cudaSetDevice(b->cfg.device));
  m = ag::mirror_create(b->N * b->A, b->A, b->frames * b->C, b->C, b->G, b->cfg.obs_dtype, lists_only);
  return m ? AGARCL_OK : AGARCL_ERR_NOMEM;
}

extern "C" int agarcl_batch_sync_mirror(agarcl_batch* b, void* stream) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  if (int rc = refuse_pixels(b, "agarcl_batch_sync_mirror")) return rc;
  int rc = ensure_mirror(b);
  if (rc) return rc;
  CK(cudaSetDevice(b->cfg.device));
  return ag::mirror_sync(b->mirror, b->d_obs, (cudaStream_t)stream);
}

extern "C" int agarcl_batch_mirror(agarcl_batch* b, void** host_ptr, int64_t shape[4], int32_t* dtype) {
  if (!b || !host_ptr) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  const bool fresh = b->mirror == nullptr;
  int rc = ensure_mirror(b);
  if (rc) return rc;
  if (fresh) {
    rc = ag::mirror_sync(b->mirror, b->d_obs, nullptr);
    if (rc) return rc;
  }
  *host_ptr = ag::mirror_ptr(b->mirror);
  if (shape) { shape[0] = (int64_t)b->N * b->A; shape[1] = (int64_t)b->frames * b->C; shape[2] = b->G; shape[3] = b->G; }
  if (dtype) *dtype = b->cfg.obs_dtype;
  return AGARCL_OK;
}

// One step of agarcl_batch_step_mirror (lists_only = false) or agarcl_batch_step_lists: the kernel reads the actions straight
// from the host-mapped staging of b->mirror or b->lists (no H2D copy in front of the launch) and, when the step is the single
// fused kernel, writes that HostMirror's lists (*lists_made).  A step that cannot write them is refused for the lists-only
// twin, before anything is enqueued: the games do not move.
static int staged_step(agarcl_batch* b, bool lists_only, const float* dxdy, const int32_t* act, bool* lists_made) {
  if (!b || !dxdy || !act) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  if (int rc = refuse_pixels(b, lists_only ? "agarcl_batch_step_lists" : "agarcl_batch_step_mirror")) return rc;
  if (lists_only && (b->frames != 1 || b->cfg.strict_reference || b->cfg.ram_obs == 2))
    return agarcl_set_error(AGARCL_ERR_STATE, "observation lists need the single fused step kernel (one frame, strict_reference = 0, a grid observation)");
  if (lists_only && !kernel_writes_lists(b))
    return agarcl_set_error(AGARCL_ERR_STATE, "this observation configuration is not finished by the step kernel: no lists");
  if (int rc = ensure_mirror(b, lists_only)) return rc;
  ag::HostMirror* m = lists_only ? b->lists : b->mirror;
  ag::mirror_stage_actions(m, dxdy, act, &b->cur_dxdy, &b->cur_act);
  return step_impl(b, nullptr, m, lists_made);
}

extern "C" int agarcl_batch_step_mirror(agarcl_batch* b, const float* dxdy, const int32_t* act, double* rewards_out,
                                        uint8_t* dones_out) {
  const auto t0 = std::chrono::steady_clock::now();
  bool lists_made = false;
  int rc = staged_step(b, false, dxdy, act, &lists_made);
  if (rc) return rc;
  b->mirror_launch_us = (uint64_t)(std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() * 1e6);
  if (lists_made) {  // k_step lists what it scatters (and reward / done) into pinned host memory while it runs
    rc = ag::mirror_collect(b->mirror, b->d_obs, nullptr, rewards_out, dones_out);
    b->mirror_call_us = (uint64_t)(std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() * 1e6);
    return rc;
  }
  const size_t NA = (size_t)b->N * b->A;
  if (rewards_out) CK(cudaMemcpyAsync(rewards_out, b->d_rewards, NA * sizeof(double), cudaMemcpyDeviceToHost, nullptr));
  if (dones_out) CK(cudaMemcpyAsync(dones_out, b->d_dones, NA, cudaMemcpyDeviceToHost, nullptr));
  rc = ag::mirror_sync(b->mirror, b->d_obs, nullptr);
  b->launches_last_step += 1;  // k_pack
  b->mirror_call_us = (uint64_t)(std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() * 1e6);
  return rc;
}

extern "C" int agarcl_batch_step_lists(agarcl_batch* b, const float* dxdy, const int32_t* act, double* rewards_out, uint8_t* dones_out,
                                       agarcl_obs_lists* out) {
  if (!out) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  bool lists_made = false;
  int rc = staged_step(b, true, dxdy, act, &lists_made);
  if (rc) return rc;
  if (!lists_made) {  // (staged_step refuses a step that would not write them)
    CK(cudaStreamSynchronize(nullptr));
    return agarcl_set_error(AGARCL_ERR_STATE, "the step kernel did not write the observation lists");
  }
  rc = ag::mirror_collect_lists(b->lists, nullptr, rewards_out, dones_out);
  if (rc) return rc;
  ag::mirror_lists_view(b->lists, out);
  return AGARCL_OK;
}

extern "C" int agarcl_batch_lists_expand(agarcl_batch* b, int32_t image, void* dense_out) {
  if (!b || !dense_out) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  if (!b->lists) return agarcl_set_error(AGARCL_ERR_STATE, "no lists yet (agarcl_batch_step_lists)");
  if (image < 0 || image >= b->N * b->A) return agarcl_set_error(AGARCL_ERR_INVALID, "image out of range");
  if (ag::mirror_lists_expand(b->lists, image, dense_out) == 1) {  // overflowed its slot: the dense frame is on the device
    CK(cudaSetDevice(b->cfg.device));
    const size_t bytes = b->obs_bytes / ((size_t)b->N * b->A);
    CK(cudaMemcpy(dense_out, (const uint8_t*)b->d_obs.get() + bytes * (size_t)image, bytes, cudaMemcpyDeviceToHost));
  }
  return AGARCL_OK;
}

extern "C" int agarcl_batch_mirror_stats(const agarcl_batch* b, uint64_t out[4]) {
  if (!b || !out) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  if (!b->mirror) return agarcl_set_error(AGARCL_ERR_STATE, "no host mirror yet (agarcl_batch_mirror)");
  ag::MirrorStats st;
  ag::mirror_stats(b->mirror, &st);
  out[0] = st.entries; out[1] = st.dense_images; out[2] = st.d2h_bytes; out[3] = st.host_threads;
  return AGARCL_OK;
}

extern "C" int agarcl_batch_mirror_timing(const agarcl_batch* b, uint64_t out[4]) {
  if (!b || !out) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  if (!b->mirror) return agarcl_set_error(AGARCL_ERR_STATE, "no host mirror yet (agarcl_batch_mirror)");
  ag::MirrorStats st;
  ag::mirror_stats(b->mirror, &st);
  out[0] = st.wait_us; out[1] = st.total_us; out[2] = b->mirror_launch_us; out[3] = b->mirror_call_us;
  return AGARCL_OK;
}

// Copies the L.stride bytes of one instance's game between the device and `host` (kind: cudaMemcpyDeviceToHost or
// cudaMemcpyHostToDevice) once the device has finished everything enqueued.
static int copy_instance(agarcl_batch* b, int32_t instance, void* host, cudaMemcpyKind kind) {
  if (instance < 0 || instance >= b->N) return agarcl_set_error(AGARCL_ERR_INVALID, "instance out of range");
  CK(cudaSetDevice(b->cfg.device));
  CK(cudaDeviceSynchronize());
  uint8_t* dev = b->d_state + (size_t)instance * b->L.stride;
  if (kind == cudaMemcpyHostToDevice) CK(cudaMemcpy(dev, host, b->L.stride, kind));
  else CK(cudaMemcpy(host, dev, b->L.stride, kind));
  return AGARCL_OK;
}

extern "C" int agarcl_batch_save_env_state(agarcl_batch* b, int32_t instance, const char* path) {
  if (!b || !path) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  std::vector<uint8_t> blob(b->L.stride);
  int rc = copy_instance(b, instance, blob.data(), cudaMemcpyDeviceToHost);
  if (rc) return rc;
  if (!b->cfg.task_modes) return agarcl_snapshot_write(&b->cfg, &b->L, blob.data(), path);
  // mixed-task batch: the instance as a batch of its current task sees it (its players, its mode_number and sizes)
  agarcl_cfg c = b->cfg;
  CK(cudaMemcpy(&c.mode_number, b->d_task_mode + instance, sizeof(int32_t), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(&c.num_bots, b->d_bots + instance, sizeof(int32_t), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(&c.num_pellets, b->d_pellets + instance, sizeof(int32_t), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(&c.num_viruses, b->d_viruses + instance, sizeof(int32_t), cudaMemcpyDeviceToHost));
  agarcl_layout L;
  task_layout(&b->cfg, &b->L, c.mode_number, c.num_bots, &L);
  return agarcl_snapshot_write(&c, &L, blob.data(), path);
}

extern "C" int agarcl_batch_load_env_state(agarcl_batch* b, int32_t instance, const char* path, int lossless) {
  if (!b || !path) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  std::vector<uint8_t> blob(b->L.stride);
  int rc = copy_instance(b, instance, blob.data(), cudaMemcpyDeviceToHost);
  if (rc) return rc;
  if (!b->was_reset) return agarcl_set_error(AGARCL_ERR_STATE, "load_env_state() before reset()");
  agarcl_cfg c = b->cfg;
  agarcl_layout L = b->L;
  if (b->cfg.task_modes) {  // mixed-task batch: any mode of the set and sizes within the maxima, which become the instance's current task
    rc = snapshot_file_task(path, &c);
    if (rc) return rc;
    if (c.mode_number < 0 || c.mode_number > 10 || !((b->cfg.task_modes >> c.mode_number) & 1))
      return agarcl_set_error(AGARCL_ERR_INVALID, "snapshot mode_number %d is not in the batch's task_modes 0x%x", c.mode_number, b->cfg.task_modes);
    if (c.mode_number != 0) c.num_bots = b->cfg.num_bots;  // (the bot count means something in mode 0 only: the file's is not checked)
    if (!ag::sizes_allowed(b->size_lim, c.num_bots, c.num_pellets, c.num_viruses))
      return agarcl_set_error(AGARCL_ERR_INVALID, "snapshot sizes (num_bots %d, num_pellets %d, num_viruses %d) are not allowed in the batch",
                              c.num_bots, c.num_pellets, c.num_viruses);
    task_layout(&b->cfg, &b->L, c.mode_number, c.num_bots, &L);
  }
  rc = agarcl_snapshot_read(&c, &L, blob.data(), path, lossless);
  if (rc) return rc;
  if (b->cfg.task_modes) {
    agarcl_player* pls = reinterpret_cast<agarcl_player*>(blob.data() + b->L.off_players);
    for (int p = L.P; p < b->L.P; p++) {  // the mode's absent players, as a reset leaves them
      std::memset(&pls[p], 0, sizeof(agarcl_player));
      pls[p].bot_type = ag::mode_bot_type(c.mode_number, p, b->L.A);
    }
    CK(cudaMemcpy(b->d_task_mode + instance, &c.mode_number, sizeof(int32_t), cudaMemcpyHostToDevice));  // (its step limit stays)
    CK(cudaMemcpy(b->d_bots + instance, &c.num_bots, sizeof(int32_t), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(b->d_pellets + instance, &c.num_pellets, sizeof(int32_t), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(b->d_viruses + instance, &c.num_viruses, sizeof(int32_t), cudaMemcpyHostToDevice));
  }
  const agarcl_inst_hdr* hdr = reinterpret_cast<const agarcl_inst_hdr*>(blob.data() + b->L.off_hdr);
  b->seeds[instance] = (uint64_t)hdr->seed_lo | ((uint64_t)hdr->seed_hi << 32);
  CK(cudaMemcpy(b->d_seeds + instance, &b->seeds[instance], sizeof(uint64_t), cudaMemcpyHostToDevice));
  if (b->cfg.rng_mode == AGARCL_RNG_MT19937) {  // Engine::seed(agarcl_data["seed"]): the mt19937_64 stream restarts (at the saved cursor when lossless)
    rc = mt_restart(b, instance, hdr->seed_lo, hdr->rng_cursor);
    if (rc) return rc;
  }
  return copy_instance(b, instance, blob.data(), cudaMemcpyHostToDevice);
}

extern "C" int agarcl_batch_download_state(agarcl_batch* b, int32_t instance, void* blob) {
  if (!b || !blob) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  return copy_instance(b, instance, blob, cudaMemcpyDeviceToHost);
}
extern "C" int agarcl_batch_upload_state(agarcl_batch* b, int32_t instance, const void* blob) {
  if (!b || !blob) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  const int rc = copy_instance(b, instance, const_cast<void*>(blob), cudaMemcpyHostToDevice);
  if (rc) return rc;
  b->was_reset = true;
  return AGARCL_OK;
}

// Refuses a caller's array that is not device memory of the batch's device; `what` names it in the message ("the pool").
static int check_device_array(const agarcl_batch* b, const void* p, const char* what) {
  cudaPointerAttributes a;
  const cudaError_t e = cudaPointerGetAttributes(&a, p);  // (does not synchronise)
  if (e != cudaSuccess) {
    cudaGetLastError();  // (clears the error, which would otherwise be reported by the next CUDA call)
    return agarcl_set_error(AGARCL_ERR_INVALID, "%s is not device memory: %s", what, cudaGetErrorString(e));
  }
  if (a.type != cudaMemoryTypeDevice || a.device != b->cfg.device)
    return agarcl_set_error(AGARCL_ERR_INVALID, "%s must be device memory of device %d", what, b->cfg.device);
  return AGARCL_OK;
}

// ---- snapshot pools (include/agarcl_b200.h): refusals are decided here, before anything is enqueued
// need_reset: refused before the first reset (save and restore read or write a game; start states only name a pool)
static int snapshot_check(agarcl_batch* b, const void* pool, int64_t pool_slots, bool need_reset = true) {
  if (b->cfg.strict_reference)
    return agarcl_set_error(AGARCL_ERR_INVALID, "snapshot pools are refused under strict_reference: the player order belongs to the batch");
  if (b->cfg.rng_mode == AGARCL_RNG_MT19937)
    return agarcl_set_error(AGARCL_ERR_INVALID, "snapshot pools are refused under AGARCL_RNG_MT19937: its generators live on the host");
  if (need_reset && !b->was_reset) return agarcl_set_error(AGARCL_ERR_STATE, "save / restore of states before reset()");
  if (!pool) return agarcl_set_error(AGARCL_ERR_INVALID, "null pool");
  if ((uintptr_t)pool & 15u) return agarcl_set_error(AGARCL_ERR_INVALID, "the pool must be 16-byte aligned");
  if (pool_slots < 1) return agarcl_set_error(AGARCL_ERR_INVALID, "pool_slots must be >= 1");
  CK(cudaSetDevice(b->cfg.device));
  return check_device_array(b, pool, "the pool");
}

static ag::SnapParams snapshot_params(const agarcl_batch* b, const void* pool, int64_t pool_slots) {
  ag::SnapParams P = {};
  P.pool = (uint8_t*)pool;
  P.pool_slots = pool_slots;
  P.S = b->snap;
  P.fingerprint = b->fingerprint;
  P.state = b->d_state;
  P.stride = b->L.stride;
  P.off_hdr = b->L.off_hdr;
  P.steps = b->autoreset ? b->d_steps.get() : nullptr;
  P.ret = b->autoreset ? b->d_ret.get() : nullptr;
  P.ram = (uint8_t*)b->d_ram.get();
  P.obs = (uint8_t*)b->d_obs.get();
  P.seeds = b->d_seeds;
  P.fresh = b->d_fresh;
  P.rewards = b->d_rewards;
  P.dones = b->d_dones;
  P.result = b->d_snap_result;
  P.restored = b->d_snap_restored;
  P.task_mode = b->d_task_mode;
  P.task_max_steps = b->d_task_max_steps;
  P.task_modes = b->cfg.task_modes;
  P.sizes = task_sizes_of(b);
  P.lim = b->size_lim;
  P.N = b->N;
  P.A = b->A;
  P.instance_base = b->cfg.instance_base;
  return P;
}

extern "C" int agarcl_batch_set_start_states(agarcl_batch* b, const void* pool, int64_t pool_slots, const int32_t* d_start_slot,
                                             void* stream) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  if (b->archive && b->archive->cfg.select)
    return agarcl_set_error(AGARCL_ERR_STATE, "the attached archive (select = 1) owns the start-state table");
  if (!pool) {  // every reset spawns again
    b->start_pool = nullptr;
    b->start_pool_slots = 0;
    return AGARCL_OK;
  }
  if (!d_start_slot) return agarcl_set_error(AGARCL_ERR_INVALID, "null start slot array");
  int rc = snapshot_check(b, pool, pool_slots, false);
  if (rc) return rc;
  CK(cudaMemcpyAsync(b->d_start_slot, d_start_slot, (size_t)b->N * sizeof(int32_t), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  b->start_pool = pool;
  b->start_pool_slots = pool_slots;
  return AGARCL_OK;
}

extern "C" int agarcl_batch_start_result(agarcl_batch* b, uint8_t** d_result) {
  if (!b || !d_result) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  *d_result = b->d_start_result;
  return AGARCL_OK;
}

extern "C" int agarcl_batch_set_archive(agarcl_batch* b, void* pool, int64_t pool_slots, const agarcl_archive_cfg* cfg) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  if (!pool) {  // detach; an archive that selected gives the start-state table back (no table)
    if (b->archive && b->archive->cfg.select) { b->start_pool = nullptr; b->start_pool_slots = 0; }
    b->archive.reset();
    return AGARCL_OK;
  }
  if (!cfg) return agarcl_set_error(AGARCL_ERR_INVALID, "null archive configuration");
  if (b->cfg.task_modes)
    return agarcl_set_error(AGARCL_ERR_INVALID, "archives are refused in mixed-task batches: a reset would need one selection per pending mode");
  int rc = snapshot_check(b, pool, pool_slots, false);
  if (rc) return rc;
  if (!b->autoreset || !b->autoreset_reset)
    return agarcl_set_error(AGARCL_ERR_STATE, "an archive needs agarcl_batch_set_autoreset with reset = 1 first");
  if (cfg->cells_per_side < 1 || cfg->cells_per_side > 256) return agarcl_set_error(AGARCL_ERR_INVALID, "cells_per_side must be in [1, 256]");
  if (cfg->agent < 0 || cfg->agent >= b->A) return agarcl_set_error(AGARCL_ERR_INVALID, "agent %d out of [0, %d)", cfg->agent, b->A);
  if (cfg->select != 0 && cfg->select != 1) return agarcl_set_error(AGARCL_ERR_INVALID, "select must be 0 or 1");
  if (pool_slots > ag::kArchiveMaxSlots)
    return agarcl_set_error(AGARCL_ERR_INVALID, "an archive holds at most %lld entries", (long long)ag::kArchiveMaxSlots);
  std::unique_ptr<Archive> a(new (std::nothrow) Archive());
  if (!a) return agarcl_set_error(AGARCL_ERR_NOMEM, "out of host memory");
  a->pool = pool;
  a->K = pool_slots;
  a->cfg = *cfg;
  a->keys = 32ll * cfg->cells_per_side * cfg->cells_per_side;
  const size_t N = (size_t)b->N, K = (size_t)pool_slots, keys = (size_t)a->keys;
  if ((rc = alloc(a->cell_of, N * 4, 0xFF)) || (rc = alloc(a->cand_key, N * 4, 0xFF)) || (rc = alloc(a->save_slot, N * 4, 0xFF)) ||
      (rc = alloc(a->src, N * 4)) || (rc = alloc(a->base_score, N * 8, 0)) || (rc = alloc(a->base_length, N * 8, 0)) ||
      (rc = alloc(a->cand_s, N * 8, 0)) || (rc = alloc(a->cand_l, N * 8, 0)) || (rc = alloc(a->draws, N * 4, 0)) ||
      (rc = alloc(a->key_entry, keys * 4, 0xFF)) || (rc = alloc(a->visits, keys * 4, 0)) || (rc = alloc(a->best_s, keys * 8, 0)) ||
      (rc = alloc(a->best_li, keys * 8, 0xFF)) || (rc = alloc(a->entry_key, K * 4, 0xFF)) || (rc = alloc(a->entry_score, K * 8, 0)) ||
      (rc = alloc(a->entry_length, K * 8, 0)) || (rc = alloc(a->entry_chosen, K * 4, 0)) || (rc = alloc(a->prefix, K * 8, 0)) ||
      (rc = alloc(a->counters, 3 * 8, 0)))
    return rc;
  std::vector<int32_t> iota(N);
  for (size_t i = 0; i < N; i++) iota[i] = (int32_t)i;
  CK(cudaMemcpy(a->src, iota.data(), N * 4, cudaMemcpyHostToDevice));
  if (cfg->select) CK(cudaMemset(b->d_start_slot, 0xFF, N * 4));
  CK(cudaDeviceSynchronize());
  if (b->archive && b->archive->cfg.select && !cfg->select) { b->start_pool = nullptr; b->start_pool_slots = 0; }
  if (cfg->select) { b->start_pool = pool; b->start_pool_slots = pool_slots; }
  b->archive = std::move(a);
  return AGARCL_OK;
}

extern "C" int agarcl_batch_archive(agarcl_batch* b, agarcl_archive* out) {
  if (!b || !out) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  if (!b->archive) return agarcl_set_error(AGARCL_ERR_STATE, "no archive attached (agarcl_batch_set_archive)");
  Archive& a = *b->archive;
  out->cell_of = a.cell_of; out->base_score = a.base_score; out->base_length = a.base_length;
  out->key_entry = a.key_entry; out->visits = a.visits;
  out->entry_key = a.entry_key; out->entry_score = a.entry_score; out->entry_length = a.entry_length; out->entry_chosen = a.entry_chosen;
  out->counters = a.counters;
  out->keys = a.keys;
  out->entries = a.K;
  return AGARCL_OK;
}

extern "C" int agarcl_batch_save_states(agarcl_batch* b, void* pool, int64_t pool_slots, const int32_t* d_src, const int32_t* d_slot,
                                        int32_t n, void* stream) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  if (n < 0) return agarcl_set_error(AGARCL_ERR_INVALID, "n must be >= 0");
  if (n > 0 && !d_src) return agarcl_set_error(AGARCL_ERR_INVALID, "null source index array");
  int rc = snapshot_check(b, pool, pool_slots);
  if (rc) return rc;
  if (n == 0) return AGARCL_OK;
  ag::SnapParams P = snapshot_params(b, pool, pool_slots);
  P.src = d_src;
  P.slot = d_slot;
  CK(ag::launch_snapshot_save(P, n, (cudaStream_t)stream));
  return AGARCL_OK;
}

extern "C" int agarcl_batch_restore_states(agarcl_batch* b, const void* pool, int64_t pool_slots, const int32_t* d_slot_of,
                                           uint8_t** d_result, void* stream) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  if (!d_slot_of) return agarcl_set_error(AGARCL_ERR_INVALID, "null slot index array");
  int rc = snapshot_check(b, pool, pool_slots);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  ag::SnapParams P = snapshot_params(b, pool, pool_slots);
  P.slot_of = d_slot_of;
  CK(ag::launch_snapshot_restore(P, s));
  if (b->archive) {  // a restored game is no trajectory of the archive's: its base restarts at (0, 0)
    ag::ArchiveParams A = archive_params(b, b->d_snap_restored);
    A.start_result = nullptr;
    CK(ag::launch_archive_base(A, s));
  }
  // a one-frame grid observation is re-rendered, as the step that produced the state showed it (respawned players still dead)
  if (renders_grid(b) && b->frames == 1 && (rc = render_frame(b, 0, s, 1, 0, b->d_snap_restored))) return rc;
  if (b->cfg.pixel_obs && (rc = render_pixels(b, s, 1, b->d_snap_restored))) return rc;
  if (d_result) *d_result = b->d_snap_result;
  return AGARCL_OK;
}

// ---- pictures of game states (include/agarcl_b200.h): refusals are decided here, before anything is enqueued
extern "C" int agarcl_batch_draw(agarcl_batch* b, int32_t view, int32_t size, const int32_t* d_src, int32_t n, uint8_t* d_out,
                                 void* stream) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  if (!b->was_reset) return agarcl_set_error(AGARCL_ERR_STATE, "draw before reset()");
  if (view != AGARCL_DRAW_ARENA && view != AGARCL_DRAW_AGENT)
    return agarcl_set_error(AGARCL_ERR_INVALID, "unknown view %d (AGARCL_DRAW_ARENA 0, AGARCL_DRAW_AGENT 1)", view);
  if (size < 16 || size > 2048 || size % 16)
    return agarcl_set_error(AGARCL_ERR_INVALID, "picture size %d must be a multiple of 16 in [16, 2048]", size);
  if (n < 0) return agarcl_set_error(AGARCL_ERR_INVALID, "n must be >= 0");
  if (!d_out) return agarcl_set_error(AGARCL_ERR_INVALID, "null output");
  if ((uintptr_t)d_out & 15u) return agarcl_set_error(AGARCL_ERR_INVALID, "the output must be 16-byte aligned");
  CK(cudaSetDevice(b->cfg.device));
  const int rc = check_device_array(b, d_out, "the output");
  if (rc || n == 0) return rc;
  const ag::DrawParams P = draw_params(b, view, size, d_src, n, d_out);
  if (view == AGARCL_DRAW_AGENT) CK(ag::launch_draw_views(P, (cudaStream_t)stream));
  else CK(ag::launch_draw(P, (cudaStream_t)stream));
  return AGARCL_OK;
}

// ---- built-in bot policies for agents (include/agarcl_b200.h): refusals are decided here, before anything is enqueued
extern "C" int agarcl_batch_bot_actions(agarcl_batch* b, const int32_t* d_type, float* d_dxdy, int32_t* d_act, float* d_target,
                                        uint8_t* d_status, void* stream) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  if (!b->was_reset) return agarcl_set_error(AGARCL_ERR_STATE, "bot actions before reset()");
  if (!d_type || !d_dxdy || !d_act) return agarcl_set_error(AGARCL_ERR_INVALID, "null type, dxdy or act array");
  if (((uintptr_t)d_dxdy | (uintptr_t)d_target) & 7u)
    return agarcl_set_error(AGARCL_ERR_INVALID, "dxdy and target must be 8-byte aligned");
  CK(cudaSetDevice(b->cfg.device));
  const std::pair<const void*, const char*> arrays[] = {{d_type, "the type array"}, {d_dxdy, "the dxdy array"}, {d_act, "the act array"},
                                                        {d_target, "the target array"}, {d_status, "the status array"}};
  for (const auto& p : arrays) {
    const int rc = p.first ? check_device_array(b, p.first, p.second) : AGARCL_OK;
    if (rc) return rc;
  }
  ag::BotParams P;
  P.L = b->L;
  P.state = b->d_state;
  P.type = d_type;
  P.dxdy = d_dxdy;
  P.act = d_act;
  P.target = d_target;
  P.status = d_status;
  P.N = b->N;
  CK(ag::launch_bot_actions(P, (cudaStream_t)stream));
  return AGARCL_OK;
}

// ---- mixed-task batches (include/agarcl_b200.h)
extern "C" int agarcl_batch_set_tasks(agarcl_batch* b, const int32_t* d_mode, const int32_t* d_max_steps, uint8_t** d_result, void* stream) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  if (!b->cfg.task_modes) return agarcl_set_error(AGARCL_ERR_STATE, "the batch was created without task_modes");
  if (!d_mode) return agarcl_set_error(AGARCL_ERR_INVALID, "null mode array");
  CK(cudaSetDevice(b->cfg.device));
  ag::SetTasksParams P;
  P.mode = d_mode;
  P.max_steps = d_max_steps;
  P.next_mode = b->d_next_mode;
  P.next_max_steps = b->d_next_max_steps;
  P.result = b->d_task_result;
  P.N = b->N;
  P.task_modes = b->cfg.task_modes;
  CK(ag::launch_set_tasks(P, (cudaStream_t)stream));
  if (d_result) *d_result = b->d_task_result;
  return AGARCL_OK;
}

extern "C" int agarcl_batch_tasks(agarcl_batch* b, agarcl_tasks* out) {
  if (!b || !out) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  if (!b->cfg.task_modes) return agarcl_set_error(AGARCL_ERR_STATE, "the batch was created without task_modes");
  out->mode = b->d_task_mode;
  out->max_steps = b->d_task_max_steps;
  out->next_mode = b->d_next_mode;
  out->next_max_steps = b->d_next_max_steps;
  return AGARCL_OK;
}

extern "C" int agarcl_batch_set_task_sizes(agarcl_batch* b, const int32_t* d_bots, const int32_t* d_pellets, const int32_t* d_viruses,
                                           uint8_t** d_result, void* stream) {
  if (!b) return agarcl_set_error(AGARCL_ERR_INVALID, "null batch");
  if (!b->cfg.task_modes) return agarcl_set_error(AGARCL_ERR_STATE, "the batch was created without task_modes");
  CK(cudaSetDevice(b->cfg.device));
  ag::SetTaskSizesParams P;
  P.bots = d_bots; P.pellets = d_pellets; P.viruses = d_viruses;
  P.next_bots = b->d_next_bots; P.next_pellets = b->d_next_pellets; P.next_viruses = b->d_next_viruses;
  P.result = b->d_size_result;
  P.lim = b->size_lim;
  P.N = b->N;
  CK(ag::launch_set_task_sizes(P, (cudaStream_t)stream));
  if (d_result) *d_result = b->d_size_result;
  return AGARCL_OK;
}

extern "C" int agarcl_batch_task_sizes(agarcl_batch* b, agarcl_task_sizes* out) {
  if (!b || !out) return agarcl_set_error(AGARCL_ERR_INVALID, "null argument");
  if (!b->cfg.task_modes) return agarcl_set_error(AGARCL_ERR_STATE, "the batch was created without task_modes");
  *out = task_sizes_of(b);
  return AGARCL_OK;
}
