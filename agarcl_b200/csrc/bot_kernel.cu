// bot_kernel.cu — the built-in bot policies for agents (agarcl_batch_bot_actions; the spec is include/agarcl_b200.h), for sm_100a.
//
// One warp decides for one agent j = i * A + a: what Bot::take_action of bot type type[j] would leave in agent a's player record,
// on instance i's state as it is at the call (oracle.c's bot_take_action, agario/bots/*.hpp).  The kernel only reads the state.
//   location        Player::x / y / mass: fp32 sums in cell order, then one division; every lane computes the same numbers from
//                   the same (broadcast) loads
//   flee, chase     lane k tests player layout.order[k] (a second round when P > 32); the lowest bit of the ballot is the first
//                   player in the order that meets the condition.  A dead or absent player has a NaN location: it fails every test
//   nearest pellet  lanes stride over the pellets in ascending index and keep their first strict minimum; a reduction on
//                   (distance, index) then gives the first minimum of the sequential scan
#include <cuda_runtime.h>

#include <climits>

#include "sim_params.h"

namespace ag {

constexpr int kBotThreads = 256;

struct PlayerLoc {
  float x, y;
  uint32_t mass;
};

// Player::x / y / mass (Player.hpp:102-126); 0 / 0 = NaN for a player without cells (quirk Q20)
__device__ __forceinline__ PlayerLoc player_loc(const agarcl_cell* c, int n) {
  float xs = 0.0f, ys = 0.0f;
  uint32_t m = 0;
  for (int i = 0; i < n; i++) {
    const float2 p = *reinterpret_cast<const float2*>(&c[i].x);
    const uint32_t mi = c[i].mass;
    xs = xs + p.x * (float)mi;
    ys = ys + p.y * (float)mi;
    m += mi;
  }
  return {xs / (float)m, ys / (float)m, m};
}

// Coordinate::distance_to (types.hpp:101-103), as oracle.c's dist_to
__device__ __forceinline__ float dist_to(float ax, float ay, float bx, float by) { return sqrtf(sqr_dist(bx, by, ax, ay)); }

// the first k < P in layout.order for which test(order[k]) holds, or -1; every lane of the warp returns the same k
template <class Test>
__device__ __forceinline__ int first_in_order(const agarcl_layout& L, int lane, Test test) {
  for (int base = 0; base < L.P; base += 32) {
    const int k = base + lane;
    const unsigned bal = __ballot_sync(AG_FULL, k < L.P && test(L.order[k]));
    if (bal) return base + __ffs(bal) - 1;
  }
  return -1;
}

__global__ void __launch_bounds__(kBotThreads) k_bot_actions(const __grid_constant__ BotParams P) {
  const int lane = threadIdx.x & 31;
  const int64_t j = (int64_t)blockIdx.x * (kBotThreads / 32) + (threadIdx.x >> 5);
  if (j >= (int64_t)P.N * P.L.A) return;
  const int type = P.type[j];
  if (type < 0 || type > 3) {  // not requested, or not a bot type: only the status is written
    if (lane == 0 && P.status) P.status[j] = type == -1 ? AGARCL_BOT_SKIPPED : AGARCL_BOT_BAD_TYPE;
    return;
  }
  const agarcl_layout& L = P.L;
  const int a = (int)(j % L.A);
  const uint8_t* blob = P.state + (size_t)(j / L.A) * L.stride;
  const agarcl_inst_hdr* hdr = reinterpret_cast<const agarcl_inst_hdr*>(blob + L.off_hdr);
  const agarcl_player* players = reinterpret_cast<const agarcl_player*>(blob + L.off_players);
  const agarcl_cell* cells = reinterpret_cast<const agarcl_cell*>(blob + L.off_cells);
  auto n_cells = [&](int p) { return min(max(players[p].n_cells, 0), L.cap_cells); };
  auto pcells = [&](int p) { return cells + (size_t)p * L.cap_cells; };

  const int n = n_cells(a);
  const PlayerLoc me = player_loc(pcells(a), n);
  float tx = 0.0f, ty = 0.0f, dx = 0.0f, dy = 0.0f;
  int status = AGARCL_BOT_DEAD;
  bool keep_action = false;  // flee and chase leave the agent's action as it is, except HungryShyBot's flee
  if (n > 0) {
    status = AGARCL_BOT_DECIDED;
    bool decided = false;
    if (type == AGARCL_BOT_HUNGRY_SHY || type == AGARCL_BOT_AGGRESSIVE_SHY) {
      // HungryShyBot.hpp:26-40, AggressiveShyBot.hpp:30-43: `other.mass() > mass()` compares against 0 (oracle.c's bot_flee)
      const int k = first_in_order(L, lane, [&](int o) {
        if (o == a) return false;
        const PlayerLoc q = player_loc(pcells(o), n_cells(o));
        return dist_to(q.x, q.y, me.x, me.y) < 25.0f && q.mass > 0u;
      });
      if (k >= 0) {
        const PlayerLoc q = player_loc(pcells(L.order[k]), n_cells(L.order[k]));
        tx = me.x - (q.x - me.x);
        ty = me.y - (q.y - me.y);
        decided = true;
        keep_action = type == AGARCL_BOT_AGGRESSIVE_SHY;
      }
    }
    if (!decided && (type == AGARCL_BOT_AGGRESSIVE || type == AGARCL_BOT_AGGRESSIVE_SHY)) {
      // AggressiveBot.hpp:28-49, AggressiveShyBot.hpp:45-64; Bot::largest_cell, Bot.hpp:70-79 (the first of the largest)
      const agarcl_cell* mc = pcells(a);
      uint32_t big = mc[0].mass;
      for (int i = 1; i < n; i++) big = mc[i].mass > big ? mc[i].mass : big;
      const int k = first_in_order(L, lane, [&](int o) {
        if (o == a) return false;
        const int no = n_cells(o);
        const PlayerLoc q = player_loc(pcells(o), no);
        if (!(dist_to(q.x, q.y, me.x, me.y) <= 20.0f)) return false;
        uint32_t edible = 0;  // Bot::edible_mass, Bot.hpp:81-88
        for (int i = 0; i < no; i++) {
          const uint32_t m = pcells(o)[i].mass;
          if (cell_can_eat_cell(big, m)) edible += m;
        }
        return edible > 0u;
      });
      if (k >= 0) {
        // Bot::target_player, Bot.hpp:55-67: three times the way to the mass-weighted centre of the edible cells
        const int o = L.order[k], no = n_cells(o);
        const agarcl_cell* oc = pcells(o);
        float sx = 0.0f, sy = 0.0f;
        uint32_t m = 0;
        for (int i = 0; i < no; i++) {
          if (cell_can_eat_cell(big, oc[i].mass)) {
            sx = sx + oc[i].x * (float)oc[i].mass;
            sy = sy + oc[i].y * (float)oc[i].mass;
            m += oc[i].mass;
          }
        }
        const float dsx = sx / (float)m - me.x, dsy = sy / (float)m - me.y;
        tx = me.x + dsx * 3.0f;
        ty = me.y + dsy * 3.0f;
        decided = true;
        keep_action = true;
      }
    }
    if (!decided) {
      const int np = min(max(hdr->n_pellets, 0), L.cap_pellets);
      if (np == 0) {
        // Bot::nearest_pellet would call std::rand() (Bot.hpp:93-97): reported, nothing flagged
        status = AGARCL_BOT_NO_PELLET;
        tx = me.x;
        ty = me.y;
      } else {
        // Bot::nearest_pellet, Bot.hpp:92-129: the first strict minimum with (double)d > 0.01, target (0, 0) if there is none
        const float2* pel = reinterpret_cast<const float2*>(blob + L.off_pellets);
        float best = 3.402823466e+38f;
        int bi = INT_MAX;
        for (int i = lane; i < np; i += 32) {
          const float2 p = pel[i];
          const float d = dist_to(p.x, p.y, me.x, me.y);
          if (d < best && (double)d > 0.01) {
            best = d;
            bi = i;
          }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
          const float ob = __shfl_xor_sync(AG_FULL, best, off);
          const int oi = __shfl_xor_sync(AG_FULL, bi, off);
          if (ob < best || (ob == best && oi < bi)) {
            best = ob;
            bi = oi;
          }
        }
        if (bi != INT_MAX) {
          const float2 p = pel[bi];
          tx = p.x;
          ty = p.y;
        }
      }
    }
    if (status == AGARCL_BOT_DECIDED) {  // the inverse of BaseEnvironment::take_action's target = loc + dxdy * 10
      dx = (tx - me.x) / 10.0f;
      dy = (ty - me.y) / 10.0f;
    }
  }
  if (lane == 0) {
    reinterpret_cast<float2*>(P.dxdy)[j] = make_float2(dx, dy);
    P.act[j] = keep_action ? players[a].action : 0;
    if (P.target) reinterpret_cast<float2*>(P.target)[j] = make_float2(tx, ty);
    if (P.status) P.status[j] = (uint8_t)status;
  }
}

cudaError_t launch_bot_actions(const BotParams& P, cudaStream_t stream) {
  const int64_t warps = (int64_t)P.N * P.L.A;
  const int64_t grid = (warps + kBotThreads / 32 - 1) / (kBotThreads / 32);
  if (grid > 0) k_bot_actions<<<(unsigned)grid, kBotThreads, 0, stream>>>(P);
  return cudaGetLastError();
}

}  // namespace ag
