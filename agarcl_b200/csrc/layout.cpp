// layout.cpp — host-side derivation of the per-instance state layout and of everything that is a
// pure function of the environment configuration (mode flags and bot roster from mode_rules.h, player iteration order).
//
// Reference behaviour restated here:
//   create_squared_pellets (count only)  agario/engine/Engine.hpp:426-475
//   GridObservation::channels_per_frame  environment/envs/GridEnvironment.hpp:188-195
//   GameState::PlayerMap iteration       agario/engine/GameState.hpp:44  (std::unordered_map<pid, ...>)
#include <algorithm>
#include <cstring>
#include <random>
#include <unordered_map>

#include "../../include/agarcl_b200.h"
#include "host_util.h"
#include "mode_rules.h"

static uint32_t align_up(uint32_t x, uint32_t a) { return (x + a - 1) / a * a; }

// player iteration order: the same container the reference iterates, fed the same insert sequence
static void player_order(int P, int32_t* order) {
  std::unordered_map<unsigned short, int> m;
  for (int p = 0; p < P; p++) m.insert(std::make_pair((unsigned short)p, p));
  int k = 0;
  for (auto& kv : m) order[k++] = kv.second;
}

// whether the order of L's players, restricted to players < Pm, is the order of a batch of Pm players alone
static bool order_restricts(const agarcl_layout* L, int Pm) {
  int alone[AGARCL_MAX_PLAYERS];
  player_order(Pm, alone);
  int k = 0;
  for (int j = 0; j < L->P; j++)
    if (L->order[j] < Pm && L->order[j] != alone[k++]) return false;
  return true;
}

uint64_t task_bot_counts(const agarcl_cfg* c, const agarcl_layout* L) {
  uint64_t bits = 0;
  if (!(c->task_modes & 1)) return bits;
  for (int b = 0; b <= c->num_bots; b++)  // (mode 0 in the set: P = A + num_bots <= 64, so b < 64)
    if (order_restricts(L, L->A + b)) bits |= 1ull << b;
  return bits;
}

void task_layout(const agarcl_cfg* c, const agarcl_layout* L, int mode, int bots, agarcl_layout* out) {
  *out = *L;
  const ag::ModeRules R = ag::mode_rules(mode, bots);
  out->P = L->A + R.bots;
  out->mass_decay = R.mass_decay;
  out->squared_pellets = R.squared_pellets;
  out->regen = R.regen;
  out->agent_mass = R.agent_mass;
  for (int p = 0; p < AGARCL_MAX_PLAYERS; p++) out->bot_type[p] = p < out->P ? ag::mode_bot_type(mode, p, L->A) : 0;
  player_order(out->P, out->order);
  for (int p = out->P; p < AGARCL_MAX_PLAYERS; p++) out->order[p] = 0;
}

extern "C" int agarcl_make_layout(const agarcl_cfg* c, agarcl_layout* L) {
  if (!c || !L) return agarcl_set_error(AGARCL_ERR_INVALID, "null cfg/layout");
  std::memset(L, 0, sizeof(*L));
  if (c->num_agents < 1) return agarcl_set_error(AGARCL_ERR_INVALID, "num_agents must be >= 1");
  if (c->ticks_per_step < 1) return agarcl_set_error(AGARCL_ERR_INVALID, "ticks_per_step must be a positive integer");
  if (c->arena_size < 8 || c->arena_size > 16384) return agarcl_set_error(AGARCL_ERR_INVALID, "arena_size out of range [8,16384]");
  if (c->num_pellets < 0 || c->num_pellets > 65000) return agarcl_set_error(AGARCL_ERR_INVALID, "num_pellets out of range [0,65000]");
  if (c->num_viruses < 0 || c->num_viruses > 4096) return agarcl_set_error(AGARCL_ERR_INVALID, "num_viruses out of range");
  if (c->num_bots < 0) return agarcl_set_error(AGARCL_ERR_INVALID, "num_bots must be >= 0");
  if (c->mode_number < 0 || c->mode_number > 10) return agarcl_set_error(AGARCL_ERR_INVALID, "Invalid mode number");
  if (c->grid_size < 1 || c->grid_size > 1024) return agarcl_set_error(AGARCL_ERR_INVALID, "grid_size out of range");
  if (c->num_frames < 1) return agarcl_set_error(AGARCL_ERR_INVALID, "num_frames must be >= 1");
  if (c->pixel_obs) {  // the pixel observation (include/agarcl_b200.h, agarcl_cfg.pixel_obs)
    if (c->pixel_obs < 16 || c->pixel_obs > 2048 || c->pixel_obs % 16)
      return agarcl_set_error(AGARCL_ERR_INVALID, "pixel_obs %d must be 0 or a multiple of 16 in [16, 2048]", c->pixel_obs);
    if (c->num_frames != 1)
      return agarcl_set_error(AGARCL_ERR_INVALID, "pixel_obs needs num_frames = 1: frame stacking of pictures is the caller's");
    if (c->strict_reference) return agarcl_set_error(AGARCL_ERR_INVALID, "pixel_obs is refused under strict_reference");
    if (c->ram_obs == 2) return agarcl_set_error(AGARCL_ERR_INVALID, "pixel_obs is refused with ram_obs = 2 (one observation or the other)");
  }

  const int mode = c->mode_number;
  const int task_modes = c->task_modes;
  if (task_modes) {  // a mixed-task batch: every mode of the set can run in it (include/agarcl_b200.h, agarcl_cfg.task_modes)
    if (task_modes & ~0x7FF) return agarcl_set_error(AGARCL_ERR_INVALID, "task_modes holds a mode outside 0..10");
    if (!((task_modes >> mode) & 1)) return agarcl_set_error(AGARCL_ERR_INVALID, "task_modes must contain mode_number %d", mode);
    if (c->strict_reference)
      return agarcl_set_error(AGARCL_ERR_INVALID, "task_modes is refused under strict_reference: the player order belongs to the batch");
  }
  const ag::ModeRules R = ag::mode_rules(mode, c->num_bots);
  L->mass_decay = R.mass_decay;
  L->squared_pellets = R.squared_pellets;
  L->regen = R.regen;
  L->agent_mass = R.agent_mass;

  // players: the agents, then the bots of the mode with the most of them
  int bots = R.bots;
  for (int m = 0; m <= 10; m++)
    if ((task_modes >> m) & 1) bots = std::max(bots, ag::mode_rules(m, c->num_bots).bots);
  if (((task_modes >> 0) & 1) && task_modes != 1) {
    // mode 0 respawns every dead player, an absent one included: it may only share a batch with modes of its bot count
    for (int m = 1; m <= 10; m++)
      if (((task_modes >> m) & 1) && ag::mode_rules(m, c->num_bots).bots != c->num_bots)
        return agarcl_set_error(AGARCL_ERR_INVALID, "task_modes: mode 0 (%d bots) cannot share a batch with mode %d (%d bots)", c->num_bots, m,
                                ag::mode_rules(m, c->num_bots).bots);
  }
  L->A = c->num_agents;
  L->P = c->num_agents + bots;
  if (L->P > AGARCL_MAX_PLAYERS) return agarcl_set_error(AGARCL_ERR_INVALID, "too many players per instance (agents + bots > 64)");
  for (int p = 0; p < L->P; p++) L->bot_type[p] = ag::mode_bot_type(mode, p, L->A);
  player_order(L->P, L->order);
  for (int m = 0; m <= 10; m++) {
    if (!((task_modes >> m) & 1)) continue;
    // an instance of mode m plays players 0 .. P_m - 1 in the batch's order: it must be the order of a batch of mode m alone
    const int Pm = L->A + ag::mode_rules(m, c->num_bots).bots;
    if (!order_restricts(L, Pm))
      return agarcl_set_error(AGARCL_ERR_INVALID, "task_modes: the player order of mode %d differs from the batch's (%d agents, %d players)", m,
                                L->A, L->P);
  }

  L->cap_cells = AGARCL_MAX_CELLS;
  int cap_p = c->num_pellets;
  for (int m = 0; m <= 10; m++) {
    if (m != mode && !((task_modes >> m) & 1)) continue;
    if (ag::mode_rules(m, c->num_bots).squared_pellets) {
      int sq = 4 * (c->arena_size / 2);  // 4 sides x int(min(W,H)/2 / spacing 1)
      if (sq > cap_p) cap_p = sq;
    }
  }
  if (cap_p < 1) cap_p = 1;
  if (cap_p > 65000) return agarcl_set_error(AGARCL_ERR_INVALID, "pellet capacity exceeds 65000");
  L->cap_pellets = cap_p;
  L->cap_viruses = c->cap_viruses > 0 ? c->cap_viruses : c->num_viruses + 32;
  if (L->cap_viruses < c->num_viruses) return agarcl_set_error(AGARCL_ERR_INVALID, "cap_viruses < num_viruses");
  L->cap_foods = c->cap_foods > 0 ? c->cap_foods : 256;
  L->cap_replay = c->cap_replay > 0 ? c->cap_replay : ((c->rng_mode == AGARCL_RNG_PHILOX) ? 0 : 16384);
  L->obs_channels = 1 + (c->observe_cells != 0) + 2 * (c->observe_others != 0) + 2 * (c->observe_viruses != 0) +
                    2 * (c->observe_pellets != 0);

  uint32_t off = 0;
  L->off_hdr = off;      off += (uint32_t)sizeof(agarcl_inst_hdr);
  L->off_players = off;  off += (uint32_t)sizeof(agarcl_player) * (uint32_t)L->P;
  L->off_cells = off;    off += (uint32_t)sizeof(agarcl_cell) * (uint32_t)L->P * (uint32_t)L->cap_cells;
  L->off_viruses = off;  off += (uint32_t)sizeof(agarcl_virus) * (uint32_t)L->cap_viruses;
  L->off_foods = off;    off += (uint32_t)sizeof(agarcl_food) * (uint32_t)L->cap_foods;
  off = align_up(off, 16);
  L->off_pellets = off;  off += (uint32_t)sizeof(agarcl_pellet) * (uint32_t)L->cap_pellets;
  L->stride = align_up(off, 128);
  return AGARCL_OK;
}

// std::mt19937_64 + std::uniform_real_distribution<float>: the generator the reference seeds in
// Engine::seed (Engine.hpp:242-245) and draws from in random_location (Engine.hpp:143-148,1304-1311).
extern "C" int agarcl_mt19937_draws(uint64_t seed, float* out, int32_t n) {
  if (!out || n < 0) return agarcl_set_error(AGARCL_ERR_INVALID, "bad draws buffer");
  std::mt19937_64 rng((unsigned)seed);  // BaseEnvironment::seed(int) -> Engine::seed(unsigned)
  for (int i = 0; i < n; i++) {
    std::uniform_real_distribution<float> d(0.0f, 1.0f);
    out[i] = d(rng);
  }
  return AGARCL_OK;
}
