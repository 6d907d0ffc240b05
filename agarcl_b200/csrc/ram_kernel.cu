// ram_kernel.cu — the structured ("ram" / GoBigger-style) observation for sm_100a.
//
// Reference: environment/envs/GoBiggerEnvironment.hpp — GoBiggerObservation::add_frame 515-548,
// _store_entities 446-513, _view_size 425-427, _world_to_grid 429-438, _inside_grid 335-338; record
// layout in include/agarcl_b200.h.  For EVERY player: in-view viruses, pellets, ejected foods and own
// cells, player-relative, in entity index order.
//
// One CTA per instance: the pellet array is staged once in shared memory (it is scanned by every
// player), then each warp takes players round-robin: centroid in cell order (Player::x / y), view,
// and four ordered compactions (ballot + prefix popcount keep the reference's index order).  The
// pellets -- 1000 per player, of which a few dozen are in view -- first go through a cheap bounding-box
// filter into a per-warp candidate list (ascending index); the exact in-view test with its two IEEE
// divisions per pellet then runs over the candidates only (r01: every pellet twice).  A record
// is written whole — used entries then zero padding — with coalesced 16-byte stores; a player with
// nothing in view keeps its previous record (the reference only commits a PlayerState when an entity
// lands inside the grid).  HBM-write bound: P * 4896 B per instance.
#include <cuda_runtime.h>

#include "sim_params.h"

namespace ag {

constexpr int kRamWarps = 8;

__global__ void __launch_bounds__(kRamWarps * 32) k_ram(const __grid_constant__ RamParams P) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  float2* s_pel = reinterpret_cast<float2*>(smem_raw);  // [cap_pellets]
  const int inst = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cand_cap = (P.L.cap_pellets + 7) & ~7;
  uint16_t* s_cand = reinterpret_cast<uint16_t*>(smem_raw + (size_t)cand_cap * sizeof(float2)) + (size_t)warp * cand_cap;  // this warp's candidates
  const uint8_t* blob = P.state + (size_t)inst * P.L.stride;
  const agarcl_inst_hdr* hdr = reinterpret_cast<const agarcl_inst_hdr*>(blob + P.L.off_hdr);
  const agarcl_player* players = reinterpret_cast<const agarcl_player*>(blob + P.L.off_players);
  const agarcl_cell* cells = reinterpret_cast<const agarcl_cell*>(blob + P.L.off_cells);
  const agarcl_virus* vir = reinterpret_cast<const agarcl_virus*>(blob + P.L.off_viruses);
  const float4* food = reinterpret_cast<const float4*>(blob + P.L.off_foods);
  const float2* pel = reinterpret_cast<const float2*>(blob + P.L.off_pellets);
  const int np = hdr->n_pellets, nv = hdr->n_viruses, nf = hdr->n_foods;
  for (int i = threadIdx.x; i < np; i += kRamWarps * 32) s_pel[i] = pel[i];
  __syncthreads();
  const unsigned long long resp = P.pre_respawn ? ((unsigned long long)hdr->respawned_hi << 32 | hdr->respawned_lo) : 0ull;
  const int G = P.G;
  const float centering = (float)G / 2.0f;
  const float r_pellet = radius_of(P.T, AGARCL_PELLET_MASS), r_food = radius_of(P.T, AGARCL_FOOD_MASS);

  for (int p = warp; p < P.L.P; p += kRamWarps) {
    const int n = ((resp >> p) & 1ull) ? 0 : players[p].n_cells;
    if (n == 0) continue;  // dead: Player::x() is NaN, nothing is inside the grid, the record stays as it was
    const agarcl_cell* pc = cells + (size_t)p * AGARCL_MAX_CELLS;
    // own cells, one per lane
    float cx = 0.f, cy = 0.f, cvx = 0.f, cvy = 0.f;
    uint32_t cm = 0;
    if (lane < n) {
      float4 a = reinterpret_cast<const float4*>(pc + lane)[0];
      cx = a.x; cy = a.y; cvx = a.z; cvy = a.w;
      cm = pc[lane].mass;
    }
    // Player::x / y / mass (Player.hpp:102-126): sequential fp32 accumulation in cell order
    float xs = 0.0f, ys = 0.0f;
    uint32_t tot = 0;
    for (int i = 0; i < n; i++) {
      float x = __shfl_sync(AG_FULL, cx, i), y = __shfl_sync(AG_FULL, cy, i);
      uint32_t m = __shfl_sync(AG_FULL, cm, i);
      xs += x * (float)m;
      ys += y * (float)m;
      tot += m;
    }
    const float px = xs / (float)tot, py = ys / (float)tot;
    const float view = clamp_std((float)(2u * tot), 100.0f, 300.0f);
    auto inside = [&](float x, float y) -> bool {
      int gx = to_int_x86((float)G * (x - px) / view + centering);
      int gy = to_int_x86((float)G * (y - py) / view + centering);
      return 0 <= gx && gx < G && 0 <= gy && gy < G;
    };
    float* rec = P.ram + ((size_t)inst * P.L.P + p) * AGARCL_RAM_RECORD;
    float4* food4 = reinterpret_cast<float4*>(rec + AGARCL_RAM_OFF_FOOD);
    float4* virus4 = reinterpret_cast<float4*>(rec + AGARCL_RAM_OFF_VIRUS);
    float4* spore4 = reinterpret_cast<float4*>(rec + AGARCL_RAM_OFF_SPORE);
    float4* clone4 = reinterpret_cast<float4*>(rec + AGARCL_RAM_OFF_CLONE);
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);

    // ---- pass 0: pellets that can be in view at all (the exact test truncates towards zero, so column 0 reaches one grid
    //      cell beyond -view/2; one more world unit of slack on top), in index order
    int nc = 0;
    {
      const float h = 0.5f * view + view / (float)G + 1.0f;
      for (int b = 0; b < np; b += 32) {
        const int i = b + lane;
        bool near = false;
        if (i < np) { const float2 q = s_pel[i]; near = fabsf(q.x - px) <= h && fabsf(q.y - py) <= h; }
        const unsigned m = __ballot_sync(AG_FULL, near);
        if (near) s_cand[nc + __popc(m & ((1u << lane) - 1u))] = (uint16_t)i;
        nc += __popc(m);
      }
      __syncwarp();
    }
    // ---- pass 1: counts only (nothing may be written when nothing is in view)
    int n_food = 0, n_virus = 0, n_spore = 0, n_clone = 0;
    for (int b = 0; b < nc; b += 32) {
      const int k = b + lane;
      bool in = false;
      if (k < nc) { const float2 q = s_pel[s_cand[k]]; in = inside(q.x, q.y); }
      n_food += __popc(__ballot_sync(AG_FULL, in));
    }
    for (int b = 0; b < nv; b += 32) {
      int i = b + lane;
      bool in = i < nv && inside(vir[i].x, vir[i].y);
      n_virus += __popc(__ballot_sync(AG_FULL, in));
    }
    for (int b = 0; b < nf; b += 32) {
      int i = b + lane;
      bool in = false;
      if (i < nf) { float4 f = food[i]; in = inside(f.x, f.y); }
      n_spore += __popc(__ballot_sync(AG_FULL, in));
    }
    const bool clone_in = lane < n && inside(cx, cy);
    const unsigned clone_mask = __ballot_sync(AG_FULL, clone_in);
    n_clone = __popc(clone_mask);
    if (n_food + n_virus + n_spore + n_clone == 0) { __syncwarp(); continue; }

    // ---- pass 2: ordered compaction + zero padding
    int w = 0;
    for (int b = 0; b < nc; b += 32) {
      const int k = b + lane;
      const float2 q = k < nc ? s_pel[s_cand[k]] : make_float2(0.f, 0.f);
      const bool in = k < nc && inside(q.x, q.y);
      unsigned m = __ballot_sync(AG_FULL, in);
      int pos = w + __popc(m & ((1u << lane) - 1u));
      if (in && pos < AGARCL_RAM_KP) food4[pos] = make_float4(q.x - px, q.y - py, r_pellet, (float)AGARCL_PELLET_MASS);
      w += __popc(m);
    }
    for (int k = min(w, AGARCL_RAM_KP) + lane; k < AGARCL_RAM_KP; k += 32) food4[k] = zero;
    w = 0;
    for (int b = 0; b < nv; b += 32) {
      int i = b + lane;
      float vx = 0.f, vy = 0.f;
      uint32_t vm = 0;
      if (i < nv) { vx = vir[i].x; vy = vir[i].y; vm = vir[i].mass; }
      bool in = i < nv && inside(vx, vy);
      unsigned m = __ballot_sync(AG_FULL, in);
      int pos = w + __popc(m & ((1u << lane) - 1u));
      if (in && pos < AGARCL_RAM_KV) virus4[pos] = make_float4(vx - px, vy - py, radius_of(P.T, vm), (float)vm);
      w += __popc(m);
    }
    for (int k = min(w, AGARCL_RAM_KV) + lane; k < AGARCL_RAM_KV; k += 32) virus4[k] = zero;
    w = 0;
    for (int b = 0; b < nf; b += 32) {
      int i = b + lane;
      float4 f = i < nf ? food[i] : zero;
      bool in = i < nf && inside(f.x, f.y);
      unsigned m = __ballot_sync(AG_FULL, in);
      int pos = w + __popc(m & ((1u << lane) - 1u));
      if (in && pos < AGARCL_RAM_KS) spore4[pos] = make_float4(f.x - px, f.y - py, r_food, (float)AGARCL_FOOD_MASS);
      w += __popc(m);
    }
    for (int k = min(w, AGARCL_RAM_KS) + lane; k < AGARCL_RAM_KS; k += 32) spore4[k] = zero;
    {
      int pos = __popc(clone_mask & ((1u << lane) - 1u));
      if (clone_in && pos < AGARCL_RAM_KC) {
        clone4[2 * pos] = make_float4(cx - px, cy - py, radius_of(P.T, cm), (float)cm);
        clone4[2 * pos + 1] = make_float4(cvx, cvy, vel_direction(cvx, cvy), (float)(p + P.pid_base));
      }
      for (int k = 2 * min(n_clone, AGARCL_RAM_KC) + lane; k < 2 * AGARCL_RAM_KC; k += 32) clone4[k] = zero;
    }
    if (lane == 0) {
      int ovf = (n_food > AGARCL_RAM_KP ? 1 : 0) | (n_virus > AGARCL_RAM_KV ? 2 : 0) | (n_spore > AGARCL_RAM_KS ? 4 : 0) |
                (n_clone > AGARCL_RAM_KC ? 8 : 0);
      reinterpret_cast<float4*>(rec)[0] = make_float4((float)n_food, (float)n_virus, (float)n_spore, (float)n_clone);
      reinterpret_cast<float4*>(rec)[1] = make_float4((float)tot, px, py, (float)ovf);
    }
    __syncwarp();  // (the candidate list is reused for the warp's next player)
  }
}

// pellets + one candidate list per warp
static size_t ram_smem(const agarcl_layout& L) {
  const size_t cand_cap = ((size_t)L.cap_pellets + 7) & ~(size_t)7;
  return cand_cap * sizeof(float2) + (size_t)kRamWarps * cand_cap * sizeof(uint16_t);
}

cudaError_t setup_ram(const agarcl_layout& L, int smem_optin) {
  const size_t smem = ram_smem(L);
  if (smem > (size_t)smem_optin) return cudaErrorInvalidValue;
  // (the device's whole opt-in, so that the batches of other layouts on this device keep what they were set up with)
  if (smem > 48 * 1024) return cudaFuncSetAttribute(k_ram, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin);
  return cudaSuccess;
}

cudaError_t launch_ram(const RamParams& P, cudaStream_t stream) {
  k_ram<<<P.N, kRamWarps * 32, ram_smem(P.L), stream>>>(P);
  return cudaGetLastError();
}

}  // namespace ag
