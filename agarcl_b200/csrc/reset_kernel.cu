// reset_kernel.cu — BaseEnvironment::reset on a fresh Engine, one warp per (masked) instance.
//
// Reference: BaseEnvironment::reset (environment/envs/BaseEnvironment.hpp:179-204), Engine::reset /
// initialize_game (agario/engine/Engine.hpp:98-117), add_pellets / add_viruses (418-424,480-485),
// create_squared_pellets (426-475), add_player -> respawn (71-83,119-137), Player::kill
// (agario/core/Player.hpp:75-86).  Draw order is the reference's: pellets (x then y each), viruses,
// then one spawn point per player in pid order; with a counter-based stream every lane computes its
// own draw index, so the whole reset is lane-parallel.
#include <cuda_runtime.h>

#include "sim_params.h"

namespace ag {

struct ResetCtx {
  const ResetParams& P;
  uint32_t seed_lo, seed_hi, inst_global, flags;
  int inst_local;
  __device__ ResetCtx(const ResetParams& p) : P(p) {}
};

__device__ __forceinline__ float rdraw(ResetCtx& c, uint32_t k) {
  if (c.P.rng_mode == AGARCL_RNG_PHILOX) return philox_uniform(c.seed_lo, c.seed_hi, c.inst_global, k);
  // the host keeps the mt19937_64 stream filled ahead of the cursor in a ring (batch.cu, refill_replay)
  if (c.P.rng_mode == AGARCL_RNG_MT19937 && c.P.replay) return c.P.replay[(size_t)c.inst_local * c.P.L.cap_replay + k % (uint32_t)c.P.L.cap_replay];
  if ((int)k < c.P.L.cap_replay && c.P.replay) return c.P.replay[(size_t)c.inst_local * c.P.L.cap_replay + k];
  c.flags |= AGARCL_FLAG_REPLAY_EXHAUSTED;
  return 0.5f;
}
__device__ __forceinline__ void rloc(ResetCtx& c, uint32_t k, float radius, float& x, float& y) {
  float span = c.P.W - 2.0f * radius;
  x = (rdraw(c, k) * span + 0.0f) + radius;
  y = (rdraw(c, k + 1) * span + 0.0f) + radius;
}

__global__ void __launch_bounds__(128) k_reset(const __grid_constant__ ResetParams P) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int inst = blockIdx.x * 4 + warp;
  if (inst >= P.N) return;
  if (P.mask && !P.mask[inst]) return;
  ResetCtx c(P);
  c.inst_local = inst;
  c.inst_global = (uint32_t)(P.instance_base + inst);
  c.seed_lo = (uint32_t)(P.seeds[inst] & 0xffffffffull);
  c.seed_hi = (uint32_t)(P.seeds[inst] >> 32);
  c.flags = 0;
  uint8_t* blob = P.state + (size_t)inst * P.L.stride;
  agarcl_inst_hdr* hdr = reinterpret_cast<agarcl_inst_hdr*>(blob + P.L.off_hdr);
  agarcl_player* players = reinterpret_cast<agarcl_player*>(blob + P.L.off_players);
  agarcl_cell* cells = reinterpret_cast<agarcl_cell*>(blob + P.L.off_cells);
  agarcl_virus* vir = reinterpret_cast<agarcl_virus*>(blob + P.L.off_viruses);
  float2* pel = reinterpret_cast<float2*>(blob + P.L.off_pellets);
  const float W = P.W;
  // the rules this episode plays: mode_number's (the layout's flags), or in a mixed-task batch the instance's pending task,
  // which becomes its current one here
  int squared = P.L.squared_pellets, agent_mass = P.L.agent_mass, Pm = P.L.P, mode = 0;
  int num_pellets = P.num_pellets, num_viruses = P.num_viruses;
  if (P.task_mode) {
    mode = P.next_mode[inst];
    const int32_t ms = P.next_max_steps[inst], bots = P.sizes.next_bots[inst];
    num_pellets = P.sizes.next_pellets[inst];
    num_viruses = P.sizes.next_viruses[inst];
    const ModeRules R = mode_rules(mode, bots);
    squared = R.squared_pellets;
    agent_mass = R.agent_mass;
    Pm = P.L.A + R.bots;
    if (lane == 0) {
      P.task_mode[inst] = mode; P.task_max_steps[inst] = ms;
      P.sizes.bots[inst] = bots; P.sizes.pellets[inst] = num_pellets; P.sizes.viruses[inst] = num_viruses;
    }
  }
  // Engine::reset does not touch the RNG (Engine.hpp:98-117): a second episode goes on in the stream; only seed() restarts it
  uint32_t cursor = (P.fresh && !P.fresh[inst]) ? hdr->rng_cursor : 0u;
  __syncwarp();
  int n_pellets = 0;

  if (squared) {
    // create_squared_pellets: four sides of a centred square, one pellet per unit, kept if inside
    float square = W / 2.0f, spacing = 1.0f;
    int pps = (int)(square / spacing);
    float cx = W / 2.0f, cy = W / 2.0f, half = square / 2.0f;
    for (int base = 0; base < 4 * pps; base += 32) {
      int t = base + lane;
      bool ok = false;
      float x = 0.f, y = 0.f;
      if (t < 4 * pps) {
        int side = t / pps;
        float fi = (float)(t % pps);
        if (side == 0) { x = cx - half + fi * spacing; y = cy - half; }
        else if (side == 1) { x = cx + half; y = cy - half + fi * spacing; }
        else if (side == 2) { x = cx + half - fi * spacing; y = cy + half; }
        else { x = cx - half; y = cy + half - fi * spacing; }
        ok = x >= 0 && x <= W && y >= 0 && y <= W;
      }
      unsigned m = __ballot_sync(AG_FULL, ok);
      int pos = n_pellets + __popc(m & ((1u << lane) - 1u));
      if (ok && pos < P.L.cap_pellets) pel[pos] = make_float2(x, y);
      n_pellets = min(n_pellets + __popc(m), P.L.cap_pellets);
    }
  } else {
    float r = radius_of(P.T, AGARCL_PELLET_MASS);
    for (int k = lane; k < num_pellets; k += 32) {
      float x, y;
      rloc(c, cursor + 2u * (uint32_t)k, r, x, y);
      if (k < P.L.cap_pellets) pel[k] = make_float2(x, y);
    }
    cursor += 2u * (uint32_t)num_pellets;
    n_pellets = min(num_pellets, P.L.cap_pellets);
  }
  {
    float r = radius_of(P.T, AGARCL_VIRUS_INITIAL_MASS);
    for (int k = lane; k < num_viruses; k += 32) {
      float x, y;
      rloc(c, cursor + 2u * (uint32_t)k, r, x, y);
      float4* v = reinterpret_cast<float4*>(vir + k);
      v[0] = make_float4(x, y, __uint_as_float(AGARCL_VIRUS_INITIAL_MASS), __int_as_float(0));
      v[1] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    cursor += 2u * (uint32_t)num_viruses;
  }
  __syncwarp();
  // players: Player ctor defaults + respawn (Player.hpp:25-41; Engine.hpp:119-137)
  const uint32_t mass = (uint32_t)(agent_mass > 25 ? agent_mass : 25);
  const float r25 = radius_of(P.T, AGARCL_CELL_MIN_SIZE);
  const bool anchored = squared && n_pellets > 0;
  for (int p = Pm + lane; p < P.L.P; p += 32) {  // absent players (mixed-task batch): dead records, no draw
    uint4* pr = reinterpret_cast<uint4*>(players + p);
    for (int q = 0; q < 8; q++) pr[q] = make_uint4(0u, 0u, 0u, 0u);
    players[p].bot_type = mode_bot_type(mode, p, P.L.A);
  }
  for (int p = lane; p < Pm; p += 32) {
    float x, y;
    if (anchored) {
      float2 p0 = pel[0];
      x = fmin_std(p0.x + 2.0f * r25, W - r25);
      y = fmin_std(p0.y + 2.0f * r25, W - r25);
    } else {
      rloc(c, cursor + 2u * (uint32_t)p, r25, x, y);
    }
    uint4* pr = reinterpret_cast<uint4*>(players + p);
    for (int q = 0; q < 8; q++) pr[q] = make_uint4(0u, 0u, 0u, 0u);
    agarcl_player* pl = players + p;
    pl->n_cells = 1;
    pl->anti_team_decay = 1.0f;
    pl->bot_type = P.task_mode ? mode_bot_type(mode, p, P.L.A) : P.L.bot_type[p];
    pl->min_mass_cell = AGARCL_CELL_MIN_SIZE;
    pl->highest_mass = AGARCL_CELL_MIN_SIZE;
    float4* cp = reinterpret_cast<float4*>(cells + (size_t)p * AGARCL_MAX_CELLS);
    cp[0] = make_float4(x, y, 0.f, 0.f);
    cp[1] = make_float4(0.f, 0.f, __uint_as_float(mass > AGARCL_CELL_MIN_SIZE ? mass : AGARCL_CELL_MIN_SIZE),
                        __uint_as_float(1u + (uint32_t)p));
    reinterpret_cast<uint4*>(cp)[2] = make_uint4(0u, 0u, 0u, 0u);  // recomb_tick = tick 0
  }
  if (!anchored) cursor += 2u * (uint32_t)Pm;
  c.flags = __reduce_or_sync(AG_FULL, c.flags);
  for (int a = lane; a < P.L.A; a += 32) P.dones[(size_t)inst * P.L.A + a] = 0;
  if (lane == 0) {
    if (P.fresh) P.fresh[inst] = 0;
    hdr->tick = 0;
    hdr->next_cell_id = 1u + (uint32_t)Pm;
    hdr->n_pellets = n_pellets;
    hdr->n_viruses = min(num_viruses, P.L.cap_viruses);
    hdr->n_foods = 0;
    hdr->rng_cursor = cursor;
    hdr->flags = c.flags;
    hdr->seed_lo = c.seed_lo; hdr->seed_hi = c.seed_hi;
    hdr->done_sticky = 0;
    hdr->respawned_lo = 0; hdr->respawned_hi = 0;
    for (int q = 0; q < 4; q++) hdr->pad[q] = 0;
  }
}

// agarcl_batch_flags: OR and per-bit instance counts of hdr.flags over the whole batch (out[0..31] counts, out[32] OR)
__global__ void __launch_bounds__(256) k_flags(const uint8_t* __restrict__ state, uint32_t off_hdr, uint32_t stride, int N, uint32_t* __restrict__ out) {
  __shared__ uint32_t cnt[33];
  if (threadIdx.x < 33) cnt[threadIdx.x] = 0u;
  __syncthreads();
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
    uint32_t f = reinterpret_cast<const agarcl_inst_hdr*>(state + (size_t)i * stride + off_hdr)->flags;
    if (f) atomicOr(&cnt[32], f);
    while (f) { const int bit = __ffs(f) - 1; f &= f - 1u; atomicAdd(&cnt[bit], 1u); }
  }
  __syncthreads();
  if (threadIdx.x < 32 && cnt[threadIdx.x]) atomicAdd(&out[threadIdx.x], cnt[threadIdx.x]);
  if (threadIdx.x == 32 && cnt[32]) atomicOr(&out[32], cnt[32]);
}
cudaError_t launch_flags(const uint8_t* state, const agarcl_layout& L, int N, uint32_t* out33, cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(out33, 0, 33 * sizeof(uint32_t), stream);
  if (e != cudaSuccess) return e;
  int ctas = (N + 255) / 256;
  if (ctas > 148) ctas = 148;
  k_flags<<<ctas, 256, 0, stream>>>(state, L.off_hdr, L.stride, N, out33);
  return cudaGetLastError();
}

cudaError_t launch_reset(const ResetParams& P, cudaStream_t stream) {
  int ctas = (P.N + 3) / 4;
  k_reset<<<ctas, 128, 0, stream>>>(P);
  return cudaGetLastError();
}

}  // namespace ag
