// sim_kernel.cu — the engine tick for N lockstep instances, hand-written for sm_100a.
//
// Mapping: ONE WARP OWNS ONE GAME INSTANCE for a whole env-step (ticks_per_step ticks); a CTA is up to
// kMaxWarpsPerCta such warps.  Inside an instance only __syncwarp / shuffles / ballots; the warps of a CTA meet at
// alignment barriers inside every tick (instruction-fetch sharing, step_instance) and share the pair solver's
// batches through shared-memory mailboxes (premove_players).
//   * a player's cells live in REGISTERS, one cell per lane (<= 32 cells), for the whole of its
//     Engine::tick_player; order-dependent reference semantics (Gauss-Seidel self-collision,
//     swap-pop recombine, eat order) are replayed with ballots + shuffles instead of loops over memory;
//   * uniform-grid spatial hash of the pellets built by a warp-level counting sort in shared memory
//     (count -> warp scan -> scatter) and patched on removals, used to FIND pellet candidates; hits are then
//     re-ordered and applied in the reference's order (510-unit buckets, ascending index,
//     Engine.hpp:976-1000) so that events are bit-exact;
//   * everything of an instance is one contiguous blob in HBM (include/agarcl_b200.h), read with
//     16-byte vector loads / one TMA bulk load (pellets); it stays shared-memory / L2 resident for the step;
//   * the grid observation is written by the same kernel: TMA bulk stores of zeros during the ticks,
//     channel 0 rows and the entity scatter after the last tick (obs_finish_warp).
// Control flow is warp-uniform everywhere a shuffle/ballot is issued.
//
// Reference functions restated here (agario/engine/Engine.hpp unless noted): tick 208-240,
// tick_player 495-542, move_player 609-630, check_player_self_collisions 763-794, prevent_overlap
// 857-888, elastic_collision_between_balls 893-938, avoid_static_overlap 701-749, separate_cells
// 803-848, optimized_check_virus_collisions 1223-1252, disrupt 1263-1294,
// get_pellets_to_remove_and_increment_cells 976-1000, remove_pellets 1002-1009, remove_viruses
// 1253-1260, may_be_auto_split 592-601, cell_split 1067-1093, eat_food 1011-1025, emit_foods
// 1027-1044, maybe_split/player_split 1056-1107, recombine_cells 1160-1179,
// maybe_activate_anti_team/mass_decay 550-584, players_collision 150-200 with
// PrecisionCollisionDetection::solve (agario/utils/collision_detection.hpp:11-64), move_foods /
// maybe_hit_virus 632-687, add_pellets/add_viruses 418-424,480-485, respawn 119-137; bots
// (agario/bots/Bot.hpp:31-129, HungryBot.hpp:19-22, HungryShyBot.hpp:23-44, AggressiveBot.hpp:28-52,
// AggressiveShyBot.hpp:28-68); BaseEnvironment::step / take_action (environment/envs/
// BaseEnvironment.hpp:89-122,164-176).
#ifdef AGARCL_PHASE_TIMING
#include <cstdio>
#endif
#include <cuda_runtime.h>

#include <cstdlib>
#include <vector>

#include "sim_params.h"
#include "sim_shared.cuh"

namespace ag {

// ------------------------------------------------------------------------------------------------
// per-lane cell (registers) and shuffles
// ------------------------------------------------------------------------------------------------
struct Cell {
  float x, y, vx, vy, svx, svy;
  uint32_t mass, id, rec;
};

__device__ __forceinline__ Cell cell_load(const agarcl_cell* g) {
  const float4* p = reinterpret_cast<const float4*>(g);
  float4 a = ldg_keep(p);
  float4 b = ldg_keep(p + 1);
  Cell c;
  c.x = a.x; c.y = a.y; c.vx = a.z; c.vy = a.w;
  c.svx = b.x; c.svy = b.y;
  c.mass = __float_as_uint(b.z); c.id = __float_as_uint(b.w);
  c.rec = ldg_keep(reinterpret_cast<const uint32_t*>(g) + 8);
  return c;
}
constexpr int kEatUnknown = 0xff;    // premove_batch did not resolve the cell's pellets (no pellets / too many candidates for a lane)
constexpr int kPremoveShadow = 16;  // cell slot of a premoved player's first result cell (players of up to 16 cells are premoved)
// a premoved player's cell: position and velocities from the result slot, mass / id / recombine tick from the live cell
__device__ __forceinline__ Cell cell_load_premoved(const agarcl_cell* g) {
  const float4* r = reinterpret_cast<const float4*>(g + kPremoveShadow);
  const float4* p = reinterpret_cast<const float4*>(g);
  float4 a = ldg_keep(r);
  float4 b = ldg_keep(r + 1);
  float4 o = ldg_keep(p + 1);
  Cell c;
  c.x = a.x; c.y = a.y; c.vx = a.z; c.vy = a.w;
  c.svx = b.x; c.svy = b.y;
  c.mass = __float_as_uint(o.z); c.id = __float_as_uint(o.w);
  c.rec = ldg_keep(reinterpret_cast<const uint32_t*>(g) + 8);
  return c;
}
__device__ __forceinline__ void cell_store(agarcl_cell* g, const Cell& c) {
  float4* p = reinterpret_cast<float4*>(g);
  stg_keep(p, make_float4(c.x, c.y, c.vx, c.vy));
  stg_keep(p + 1, make_float4(c.svx, c.svy, __uint_as_float(c.mass), __uint_as_float(c.id)));
  stg_keep(p + 2, make_float4(__uint_as_float(c.rec), 0.f, 0.f, 0.f));
}
__device__ __forceinline__ Cell cell_bcast(const Cell& c, int src) {
  Cell r;
  r.x = __shfl_sync(AG_FULL, c.x, src); r.y = __shfl_sync(AG_FULL, c.y, src);
  r.vx = __shfl_sync(AG_FULL, c.vx, src); r.vy = __shfl_sync(AG_FULL, c.vy, src);
  r.svx = __shfl_sync(AG_FULL, c.svx, src); r.svy = __shfl_sync(AG_FULL, c.svy, src);
  r.mass = __shfl_sync(AG_FULL, c.mass, src); r.id = __shfl_sync(AG_FULL, c.id, src);
  r.rec = __shfl_sync(AG_FULL, c.rec, src);
  return r;
}
// warp reductions: one REDUX instruction each (sm_80+) instead of five shuffle/op pairs -- less latency and, as
// they are inlined at dozens of sites, a good deal less code for the 32 KB instruction cache
__device__ __forceinline__ uint32_t warp_sum_u32(uint32_t v) { return __reduce_add_sync(AG_FULL, v); }
__device__ __forceinline__ uint32_t warp_min_u32(uint32_t v) { return __reduce_min_sync(AG_FULL, v); }
__device__ __forceinline__ uint32_t warp_max_u32(uint32_t v) { return __reduce_max_sync(AG_FULL, v); }
// Alignment barrier of the warp's group (step_instance): `ag` consecutive warps of the CTA, barrier 1 + group.
__device__ __forceinline__ void align_barrier(int ag) {
  const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5, g = warp / ag;
  const int members = min(ag, nw - g * ag);
  asm volatile("barrier.sync %0, %1;" :: "r"(1 + g), "r"(members * 32) : "memory");
}
__device__ __forceinline__ uint32_t lanemask_lt(int lane) { return (1u << lane) - 1u; }
constexpr int kHashDead = 0xffff;  // hash entry of a pellet removed since the hash was built

// ------------------------------------------------------------------------------------------------
// per-warp context: uniform registers + pointers
// ------------------------------------------------------------------------------------------------
// The warp-uniform state of the instance that is touched a few times per tick at most.  It lives in the warp's shared memory:
// as members of Ctx these values were spilled to local memory around every solver loop (32 copies of each, one per lane, in
// an L1 of ~24 KB next to 227 KB of shared memory: 69 % of the spill reloads missed, profiles/r02_experiments), here they are
// one 4-byte broadcast load away.  Every lane stores the same value (warp-uniform code only), so no lane election is needed.
struct ColdCtx {
  long long work, t_mark;   // cycles this instance has worked (waiting at the alignment barriers excluded) / start of the current stretch
  uint32_t zagent, zoff, zchunk;  // fused observation clear: cursor (agent, vector) and vectors per chunk
  uint32_t next_id, cursor, done_sticky;  // header fields
  uint32_t min_vmass;   // smallest virus mass this tick (0xffffffff without viruses)
  uint32_t pre_lo, pre_hi;  // players whose move + self-collisions of this tick are already done (premove_players)
  uint32_t sorted_lo, sorted_hi;  // players whose cells are known to be in ascending id order (sort_player_cells can be skipped)
  int emitted;          // foods appended by the last tick_player (Engine::emit_foods)
  int inst_local;
  int pos;              // position of the instance in this launch's schedule (the host mirror's lists are laid out by position)
  int tb;               // the alignment barriers of this launch (P.tick_barrier, or 0 when the launch runs the free-running schedule)
  int mode;             // the instance's current mode (P.task_mode[inst] in a mixed-task batch, else P.mode)
};
static_assert(sizeof(ColdCtx) <= kColdCtxBytes - 16, "ColdCtx outgrew its shared-memory slot");

#ifdef AGARCL_PHASE_TIMING
// experiment builds only (tools/build_variant.sh with EXTRA=-DAGARCL_PHASE_TIMING): cycles per phase summed over all instance warps,
// printed (running totals) by the first thread of every launch
__device__ unsigned long long g_phase[32];
__device__ unsigned int g_cta_cycles[256];  // lifetime of every CTA of the last launch (cycles / 1024)
#define AG_PH(c, i) do { const long long t_ = clock64(); if ((c).lane == 0) atomicAdd(&g_phase[i], (unsigned long long)(t_ - (c).ph_t)); (c).ph_t = t_; } while (0)
#else
#define AG_PH(c, i) do { } while (0)
#endif

struct Ctx {
  const SimParams& P;
  int lane;
#ifdef AGARCL_PHASE_TIMING
  long long ph_t;
#endif
  uint8_t* blob;  // this instance's state; the arrays are blob + constant-bank offsets, formed where used
  WarpSmem sm;
  __device__ __forceinline__ agarcl_player* players_() const { return reinterpret_cast<agarcl_player*>(blob + P.L.off_players); }
  __device__ __forceinline__ agarcl_cell* cells_() const { return reinterpret_cast<agarcl_cell*>(blob + P.L.off_cells); }
  __device__ __forceinline__ agarcl_virus* vir_() const { return reinterpret_cast<agarcl_virus*>(blob + P.L.off_viruses); }
  __device__ __forceinline__ agarcl_food* food_() const { return reinterpret_cast<agarcl_food*>(blob + P.L.off_foods); }
  __device__ __forceinline__ agarcl_pellet* pel_() const { return reinterpret_cast<agarcl_pellet*>(blob + P.L.off_pellets); }
  __device__ __forceinline__ ColdCtx& cold() const { return *reinterpret_cast<ColdCtx*>(sm.base + P.so.cold); }
  // header, kept in registers for the whole launch
  uint32_t tick, flags;
  int n_pellets, n_viruses, n_foods;
  int nprem, nvrem;
  bool hash_valid;      // the pellet hash in shared memory matches the pellet array
  bool pel_dirty;       // the pellet array in shared memory differs from the blob's (written back when the warp leaves the instance)
  bool vc_valid;        // the virus cache in shared memory matches the virus array
  bool lanes_dirty;     // players_collision changed players: lanes must reload their registers
  float W;
  static constexpr float dt = (float)(1.0 / 30.0);
  __device__ Ctx(const SimParams& p) : P(p) {}
  __device__ __forceinline__ agarcl_cell* pcells(int p) const { return cells_() + (size_t)p * AGARCL_MAX_CELLS; }
  // the rules of the instance's mode: the launch parameters' unless the batch mixes tasks (mode_rules.h)
  __device__ __forceinline__ ModeRules rules() const { return mode_rules(cold().mode, P.num_bots); }
  __device__ __forceinline__ bool mass_decay() const { return P.task_mode ? rules().mass_decay != 0 : P.L.mass_decay != 0; }
  __device__ __forceinline__ bool regen() const { return P.task_mode ? rules().regen != 0 : P.L.regen != 0; }
  __device__ __forceinline__ bool squared_pellets() const { return P.task_mode ? rules().squared_pellets != 0 : P.L.squared_pellets != 0; }
  __device__ __forceinline__ int agent_mass() const { return P.task_mode ? rules().agent_mass : P.L.agent_mass; }
  __device__ __forceinline__ int bot_type(int p) const { return P.task_mode ? mode_bot_type(cold().mode, p, P.L.A) : P.L.bot_type[p]; }
};

// one uniform draw in [0,1): k-th draw of this instance (Engine::random<T>, Engine.hpp:1304-1311)
__device__ __forceinline__ float draw_at(Ctx& c, uint32_t k) {
  if (c.P.rng_mode == AGARCL_RNG_PHILOX) {  // seed lives in the header: draws are rare (regen, respawn)
    const agarcl_inst_hdr* hdr = reinterpret_cast<const agarcl_inst_hdr*>(c.blob + c.P.L.off_hdr);
    return philox_uniform(hdr->seed_lo, hdr->seed_hi, (uint32_t)(c.P.instance_base + c.cold().inst_local), k);
  }
  // the host keeps the mt19937_64 stream filled ahead of the cursor in a ring (batch.cu, refill_replay)
  if (c.P.rng_mode == AGARCL_RNG_MT19937 && c.P.replay) return c.P.replay[(size_t)c.cold().inst_local * c.P.L.cap_replay + k % (uint32_t)c.P.L.cap_replay];
  if ((int)k < c.P.L.cap_replay && c.P.replay) return c.P.replay[(size_t)c.cold().inst_local * c.P.L.cap_replay + k];
  c.flags |= AGARCL_FLAG_REPLAY_EXHAUSTED;
  return 0.5f;
}
// Engine::random_location(radius), Engine.hpp:143-148, for the draw pair starting at k
__device__ __forceinline__ void random_location_at(Ctx& c, uint32_t k, float radius, float& x, float& y) {
  float span = c.W - 2.0f * radius;
  float ux = draw_at(c, k);
  x = (ux * span + 0.0f) + radius;
  float uy = draw_at(c, k + 1);
  y = (uy * span + 0.0f) + radius;
}

// Ball::touches, Ball.hpp:36-43
__device__ __forceinline__ bool touches(const Luts& T, float ax, float ay, uint32_t am, float bx, float by, uint32_t bm) {
  float s = radius_of(T, am) + radius_of(T, bm);
  return s * s >= sqr_dist(ax, ay, bx, by) + 0.0f;
}
__device__ __forceinline__ void bound_cell(const Ctx& c, Cell& k) {
  float r = radius_of(c.P.T, k.mass);
  k.x = bound_axis(k.x, r, c.W);
  k.y = bound_axis(k.y, r, c.W);
}
__device__ __forceinline__ void cell_move(Cell& k, float dt) {  // Cell::move, Entities.hpp:161-164
  k.x += (k.vx + k.svx) * dt;
  k.y += (k.vy + k.svy) * dt;
}

// ------------------------------------------------------------------------------------------------
// pair routines of the self-collision solver; operate on broadcast copies (uniform within the lane group
// that owns the player).  The radii come in as arguments: the masses do not change in this phase, so every
// lane computes the radius of its cell once (radius_of is a table load) instead of once per use.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool touches_r(float ax, float ay, float ar, float bx, float by, float br) {  // Ball::touches, Ball.hpp:36-43
  float s = ar + br;
  return s * s >= sqr_dist(ax, ay, bx, by) + 0.0f;
}
__device__ __forceinline__ void bound_cell_r(float W, Cell& k, float r) {
  k.x = bound_axis(k.x, r, W);
  k.y = bound_axis(k.y, r, W);
}

__device__ __forceinline__ void avoid_static_overlap(float W, Cell& a, Cell& b, float ra, float rb) {  // Engine.hpp:701-749
  float dx = b.x - a.x, dy = b.y - a.y;
  float dist = sqrtf(dx * dx + dy * dy);
  float target = ra + rb;
  if (dist > target) return;
  float xr = dx / (fabsf(dx) + fabsf(dy));
  float yr = dy / (fabsf(dx) + fabsf(dy));
  float depth = target - dist;
  float arx = 0.5f, ary = 0.5f, brx = 0.5f, bry = 0.5f;
  if (a.x == ra || a.x == W - ra) { arx = 1.0f; a.vx = 0.0f; }
  if (a.y == ra || a.y == W - ra) { ary = 1.0f; a.vy = 0.0f; }
  if (b.x == rb || b.x == W - rb) { brx = 1.0f; b.vx = 0.0f; }
  if (b.y == rb || b.y == W - rb) { bry = 1.0f; b.vy = 0.0f; }
  a.x -= xr * depth * arx;
  a.y -= yr * depth * ary;
  b.x += xr * depth * brx;
  b.y += yr * depth * bry;
  bound_cell_r(W, a, ra);
  bound_cell_r(W, b, rb);
}

__device__ __forceinline__ void separate_cells(Cell& a, Cell& b, float ra, float rb, float tx, float ty) {  // Engine.hpp:803-848
  float dx = b.x - a.x, dy = b.y - a.y;
  float dist = sqrtf(dx * dx + dy * dy);
  float target = ra + rb;
  if (dist > target) return;
  float xr = dx / (fabsf(dx) + fabsf(dy));
  float yr = dy / (fabsf(dx) + fabsf(dy));
  float diff_a = sqr_dist(tx, ty, a.x, a.y);
  float diff_b = sqr_dist(tx, ty, b.x, b.y);
  float depth = target - dist;
  int s1 = (a.mass < b.mass) ? 1 : -1;
  int s2 = (diff_a >= diff_b) ? 1 : -1;
  float fs = (float)((s1 == s2) ? s2 : 0);
  bool move_a = a.mass < b.mass;
  float tx_ = move_a ? a.x : b.x, ty_ = move_a ? a.y : b.y;
  if (dx >= 0) {
    tx_ -= xr * depth * fs;
    if (dy >= 0) ty_ -= yr * depth * fs; else ty_ += yr * depth * fs;
  } else {
    tx_ += xr * depth * fs;
    if (dy >= 0) ty_ -= yr * depth * fs; else ty_ += yr * depth * fs;
  }
  if (move_a) { a.x = tx_; a.y = ty_; } else { b.x = tx_; b.y = ty_; }
}

__device__ __forceinline__ void elastic(Cell& a, Cell& b, float dx, float dy, float dist) {  // Engine.hpp:893-938
  float nx = dx / dist, ny = dy / dist;
  float tx = -ny, ty = nx;
  float dpn1 = a.vx * nx + a.vy * ny;
  float dpn2 = b.vx * nx + b.vy * ny;
  float dpt1 = a.vx * tx + a.vy * ty;
  float dpt2 = b.vx * tx + b.vy * ty;
  int m1 = (int)a.mass, m2 = (int)b.mass;
  float v1 = (dpn1 * (float)(m1 - m2) + 2.0f * (float)m2 * dpn2) / (float)(m1 + m2);
  float v2 = (dpn2 * (float)(m2 - m1) + 2.0f * (float)m1 * dpn1) / (float)(m1 + m2);
  if (a.mass < b.mass) {
    a.vx = tx * dpt1 + nx * v1; a.vy = ty * dpt1 + ny * v1;
  } else if (a.mass > b.mass) {
    b.vx = tx * dpt2 + nx * v2; b.vy = ty * dpt2 + ny * v2;
  } else {
    a.vx = tx * dpt1 + nx * v1; a.vy = ty * dpt1 + ny * v1;
    b.vx = tx * dpt2 + nx * v2; b.vy = ty * dpt2 + ny * v2;
  }
}

__device__ __forceinline__ void prevent_overlap(float W, Cell& a, Cell& b, float ra, float rb, float tx, float ty) {  // Engine.hpp:857-888
  float dx = b.x - a.x, dy = b.y - a.y;
  float dist = sqrtf(dx * dx + dy * dy);
  float target = ra + rb;
  if (dist > target) return;
  const float dt = Ctx::dt;
  a.x -= (a.vx + a.svx) * dt;
  a.y -= (a.vy + a.svy) * dt;
  b.x -= (b.vx + b.svx) * dt;
  b.y -= (b.vy + b.svy) * dt;
  elastic(a, b, dx, dy, dist);
  cell_move(a, dt);
  cell_move(b, dt);
  if (touches_r(a.x, a.y, ra, b.x, b.y, rb)) {
    int diff = (int)(a.mass - b.mass);
    if (abs(diff) <= 10) avoid_static_overlap(W, a, b, ra, rb);
    else separate_cells(a, b, ra, rb, tx, ty);
  }
  bound_cell_r(W, a, ra);
  bound_cell_r(W, b, rb);
}

// Engine::check_player_self_collisions, Engine.hpp:763-794, for up to 32 / gw players at once: the warp is cut
// into groups of `gw` lanes (8, 16 or 32), every group owns one player with one cell per lane (gl = lane in the
// group, gbase = first lane of the group, n = the group's cell count, 0 for an idle group).  The reference walks
// the pairs (a < b) of a player in index order and resolves the touching ones, which is inherently sequential
// PER PLAYER; the groups run that sequence side by side under one control flow (a group without a pair at the
// current step is predicated off), so a tick costs the longest player's pair sequence instead of the sum.
// For a fixed `a`, one ballot finds the next touching b, the pair is resolved on group-broadcast copies, and the
// ballot is re-issued against the moved a.  static_pass: avoid_static_overlap instead of prevent_overlap.
__device__ __forceinline__ bool self_pass(float W, Cell& me, float myr, int n, bool on, float tx, float ty,
                                         int gbase, int gl, unsigned gmask, bool static_pass) {
  bool overlap = false;
  const int nmax = (int)warp_max_u32(on ? (uint32_t)n : 0u);
  // what a pair routine reads (position, both velocities, mass) / writes (position, velocity)
  auto bcast = [&](int src) {
    Cell r;
    r.x = __shfl_sync(AG_FULL, me.x, src); r.y = __shfl_sync(AG_FULL, me.y, src);
    r.vx = __shfl_sync(AG_FULL, me.vx, src); r.vy = __shfl_sync(AG_FULL, me.vy, src);
    r.svx = __shfl_sync(AG_FULL, me.svx, src); r.svy = __shfl_sync(AG_FULL, me.svy, src);
    r.mass = __shfl_sync(AG_FULL, me.mass, src); r.id = 0u; r.rec = 0u;
    return r;
  };
  for (int a = 0; a + 1 < nmax; a++) {
    const bool mine_a = on && a + 1 < n;
    bool ga = mine_a;
    int b_last = a;
    // cell `a` stays in the group-uniform copy A for all its pairs and returns to its lane afterwards
    // (an idle group reads a foreign lane here: never used, never written back)
    Cell A = bcast(gbase + a);
    const float ar = __shfl_sync(AG_FULL, myr, gbase + a);
    while (true) {
      const bool t = ga && gl > b_last && gl < n && touches_r(A.x, A.y, ar, me.x, me.y, myr);
      const unsigned mg = (__ballot_sync(AG_FULL, t) & gmask) >> gbase;
      const bool has = mg != 0u;
      if (!__any_sync(AG_FULL, has)) break;
      const int b = has ? __ffs(mg) - 1 : 0;
      Cell B = bcast(gbase + b);
      const float rb = __shfl_sync(AG_FULL, myr, gbase + b);
      if (has) {
        if (static_pass) avoid_static_overlap(W, A, B, ar, rb);
        else prevent_overlap(W, A, B, ar, rb, tx, ty);
        if (gl == b) { me.x = B.x; me.y = B.y; me.vx = B.vx; me.vy = B.vy; }
        overlap = true;
        b_last = b;
      } else {
        ga = false;  // this group is through with `a`
      }
    }
    if (mine_a && gl == a) { me.x = A.x; me.y = A.y; me.vx = A.vx; me.vy = A.vy; }
  }
  return overlap;
}
// ONE out-of-line copy for both callers (premove_players and tick_player): the pair loop is the hottest code of
// mature games and the instruction cache holds 32 KB; arguments and result by value, so nothing of the callers'
// state is forced into local memory.
__device__ __noinline__ Cell self_collisions_fn(Cell me, float myr, int n, float tx, float ty, int gbase, int gl, int gw, float W) {
  const unsigned gmask = (gw >= 32 ? 0xffffffffu : ((1u << gw) - 1u)) << gbase;
  bool on = n >= 2;
  int passes = 0;  // passes 0..4: prevent_overlap while the previous one found an overlap; pass 5: the static pass after five overlapping ones
  while (__any_sync(AG_FULL, on)) {
    const bool overlap = self_pass(W, me, myr, n, on, tx, ty, gbase, gl, gmask, passes == 5);
    on = on && overlap && passes < 5;  // "if (!overlap) break" of the group's player
    passes++;
  }
  return me;
}
__device__ __forceinline__ void self_collisions(const Ctx& c, Cell& me, int n, float tx, float ty, int gbase, int gl, int gw) {
  me = self_collisions_fn(me, radius_of(c.P.T, me.mass), n, tx, ty, gbase, gl, gw, c.W);
}

// Player::x / y / mass (Player.hpp:102-126): sequential fp32 accumulation in cell order
__device__ __forceinline__ float4 centroid_of(const Cell& me, int n) {
  float xs = 0.0f, ys = 0.0f;
  uint32_t tot = 0;
  for (int i = 0; i < n; i++) {
    float x = __shfl_sync(AG_FULL, me.x, i), y = __shfl_sync(AG_FULL, me.y, i);
    uint32_t m = __shfl_sync(AG_FULL, me.mass, i);
    xs += x * (float)m;
    ys += y * (float)m;
    tot += m;
  }
  float fm = (float)tot;
  return make_float4(xs / fm, ys / fm, __uint_as_float(tot), __int_as_float(n));
}
// same thing straight from global memory, by one lane (divergent trip counts allowed: no shuffles)
__device__ float4 centroid_from_global(const agarcl_cell* g, int n) {
  float xs = 0.0f, ys = 0.0f;
  uint32_t tot = 0;
  for (int i = 0; i < n; i++) {
    float4 a = ldg_keep(reinterpret_cast<const float4*>(g + i));
    uint32_t m = __float_as_uint(ldg_keep(reinterpret_cast<const float4*>(g + i) + 1).z);
    xs += a.x * (float)m;
    ys += a.y * (float)m;
    tot += m;
  }
  float fm = (float)tot;
  return make_float4(xs / fm, ys / fm, __uint_as_float(tot), __int_as_float(n));
}

// ------------------------------------------------------------------------------------------------
// bots
// ------------------------------------------------------------------------------------------------
// Bot::nearest_pellet, Bot.hpp:92-129: first index attaining the minimum of sqrtf(d^2) among d > 0.01
__device__ void lane_nearest_pellet(const Ctx& c, float lx, float ly, float& tx, float& ty);
__device__ bool lane_eat_pellets(const Ctx& c, float cx, float cy, uint32_t& mass, int& ne, uint16_t* out);
__device__ void nearest_pellet(Ctx& c, float lx, float ly, float& tx, float& ty) {
  if (c.n_pellets == 0) {  // std::rand() % arena: not replayable (flagged), same stand-in as the oracle
    c.flags |= AGARCL_FLAG_RAND_SITE;
    tx = 0.0f; ty = 0.0f;
    return;
  }
  if (c.hash_valid) {  // one lane walks the hash rings in shared memory instead of 32 dependent trips over the pellet array
    if (c.lane == 0) lane_nearest_pellet(c, lx, ly, tx, ty);
    tx = __shfl_sync(AG_FULL, tx, 0);
    ty = __shfl_sync(AG_FULL, ty, 0);
    return;
  }
  float best = 3.402823466e+38f;
  uint32_t best_i = 0xffffffffu;
  for (int i = c.lane; i < c.n_pellets; i += 32) {
    float2 p = c.sm.spel()[i];
    float d = sqrtf(sqr_dist(lx, ly, p.x, p.y));  // (other - this).norm()
    if (d < best && (double)d > 0.01) { best = d; best_i = (uint32_t)i; }
  }
  // global first-min: smallest distance, then smallest index
  float gbest = best;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) gbest = fminf(gbest, __shfl_xor_sync(AG_FULL, gbest, o));
  uint32_t cand = (best == gbest && best_i != 0xffffffffu) ? best_i : 0xffffffffu;
  cand = warp_min_u32(cand);
  if (cand == 0xffffffffu) { tx = 0.0f; ty = 0.0f; return; }  // nothing qualified: Location() default
  float2 p = c.sm.spel()[cand];
  tx = p.x; ty = p.y;
}

// flee loop of HungryShyBot.hpp:26-40 / AggressiveShyBot.hpp:30-43.  `other.mass() > mass()` compares
// against the TYPE agario::mass value-initialised to 0 (core/types.hpp:52), i.e. "other is alive".
__device__ bool bot_flee(Ctx& c, int p, float lx, float ly, float& tx, float& ty) {
  const int P = c.P.L.P;
  for (int base = 0; base < P; base += 32) {
    int k = base + c.lane;
    bool cond = false;
    float ox = 0.f, oy = 0.f;
    if (k < P) {
      int o = c.P.L.order[k];
      float4 s = c.sm.psum()[o];
      ox = s.x; oy = s.y;
      float d = sqrtf(sqr_dist(ox, oy, lx, ly));
      cond = (o != p) && (d < 25.0f) && (__float_as_uint(s.z) > 0u);
    }
    unsigned m = __ballot_sync(AG_FULL, cond);
    if (m) {
      int src = __ffs(m) - 1;
      ox = __shfl_sync(AG_FULL, ox, src);
      oy = __shfl_sync(AG_FULL, oy, src);
      tx = lx - (ox - lx);
      ty = ly - (oy - ly);
      return true;
    }
  }
  return false;
}

// chase loop of AggressiveBot.hpp:33-49 / AggressiveShyBot.hpp:47-64 with Bot::edible_mass and
// Bot::target_player (Bot.hpp:55-88)
__device__ bool bot_chase(Ctx& c, int p, const Cell& me, int n, float lx, float ly, float& tx, float& ty) {
  // Bot::largest_cell: first maximum
  uint32_t mymass = c.lane < n ? me.mass : 0u;
  uint32_t big = warp_max_u32(mymass);
  const int P = c.P.L.P;
  for (int base = 0; base < P; base += 32) {
    int k = base + c.lane;
    bool near = false;
    if (k < P) {
      int o = c.P.L.order[k];
      float4 s = c.sm.psum()[o];
      float d = sqrtf(sqr_dist(s.x, s.y, lx, ly));
      near = (o != p) && (d <= 20.0f);
    }
    unsigned m = __ballot_sync(AG_FULL, near);
    while (m) {
      int src = __ffs(m) - 1;
      m &= m - 1;
      int o = c.P.L.order[base + src];
      int on = __float_as_int(c.sm.psum()[o].w);
      Cell oc;
      oc.mass = 0; oc.x = 0.f; oc.y = 0.f;
      if (c.lane < on) {
        const agarcl_cell* g = c.pcells(o) + c.lane;
        float4 a = reinterpret_cast<const float4*>(g)[0];
        oc.x = a.x; oc.y = a.y; oc.mass = g->mass;
      }
      bool edible = c.lane < on && cell_can_eat_cell(big, oc.mass);
      unsigned em = __ballot_sync(AG_FULL, edible);
      if (em) {
        float sx = 0.0f, sy = 0.0f;
        uint32_t sm = 0;
        for (int i = 0; i < on; i++) {
          float x = __shfl_sync(AG_FULL, oc.x, i), y = __shfl_sync(AG_FULL, oc.y, i);
          uint32_t mm = __shfl_sync(AG_FULL, oc.mass, i);
          if (em & (1u << i)) { sx += x * (float)mm; sy += y * (float)mm; sm += mm; }
        }
        float dsx = sx / (float)sm - lx, dsy = sy / (float)sm - ly;
        tx = lx + dsx * 3.0f;
        ty = ly + dsy * 3.0f;
        return true;
      }
    }
  }
  return false;
}

// ------------------------------------------------------------------------------------------------
// per-tick builds: pellet spatial hash (warp counting sort in shared memory) and virus cache
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int hash_coord(const Ctx& c, float v) {
  int h = (int)(v * c.P.hash_scale);
  return min(max(h, 0), c.P.HG - 1);
}
__device__ void build_pellet_hash(Ctx& c) {
  const int HG = c.P.HG, nc = HG * HG;
  uint32_t* cnt = c.sm.htmp();  // 32-bit counters for the shared-memory atomics (scratch that is dead at the start of a tick)
  for (int i = c.lane; i < nc; i += 32) cnt[i] = 0u;
  __syncwarp();
  const float2* pel = c.sm.spel();
  for (int i = c.lane; i < c.n_pellets; i += 32) {
    float2 p = pel[i];
    atomicAdd(&cnt[hash_coord(c, p.y) * HG + hash_coord(c, p.x)], 1u);
  }
  __syncwarp();
  // exclusive scan over nc counters, 32 at a time
  uint32_t carry = 0;
  for (int base = 0; base < nc; base += 32) {
    int i = base + c.lane;
    uint32_t v = i < nc ? cnt[i] : 0u;
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t t = __shfl_up_sync(AG_FULL, incl, o);
      if (c.lane >= o) incl += t;
    }
    if (i < nc) cnt[i] = carry + incl - v;
    carry += __shfl_sync(AG_FULL, incl, 31);
  }
  __syncwarp();
  for (int i = c.lane; i < c.n_pellets; i += 32) {
    float2 p = pel[i];
    uint32_t pos = atomicAdd(&cnt[hash_coord(c, p.y) * HG + hash_coord(c, p.x)], 1u);
    c.sm.hsorted()[pos] = (uint16_t)i;
  }
  __syncwarp();
  // now cnt[k] = end of cell k; kept as 16-bit: start of cell k = (k ? hcnt[k-1] : 0)
  for (int i = c.lane; i < nc; i += 32) c.sm.hcnt()[i] = (uint16_t)cnt[i];
  __syncwarp();
}
__device__ void build_virus_cache(Ctx& c) {
  uint32_t mn = 0xffffffffu;
  for (int v = c.lane; v < c.n_viruses; v += 32) {
    const float4 a = ldg_keep(reinterpret_cast<const float4*>(c.vir_() + v));  // x, y, mass, hits
    uint32_t vm = __float_as_uint(a.z);
    mn = min(mn, vm);
    c.sm.vcache()[v] = make_float4(a.x, a.y, radius_of(c.P.T, vm), a.z);
  }
  c.cold().min_vmass = warp_min_u32(mn);
  __syncwarp();
}

// ------------------------------------------------------------------------------------------------
// Engine::tick_player
// ------------------------------------------------------------------------------------------------
// Engine::move_player for one cell (Engine.hpp:609-630)
__device__ __forceinline__ void move_cell(const SimParams& P, uint32_t& flags, Cell& me, float tx, float ty) {
  me.vx = 3.0f * (tx - me.x);
  me.vy = 3.0f * (ty - me.y);
  float limit = max_speed_of(P.T, me.mass, flags);
  if (vmag(me.vx, me.vy) > limit) {  // Velocity::clamp_speed + set_speed (quirk Q8)
    me.vx *= limit / vmag(me.vx, me.vy);
    me.vy *= limit / vmag(me.vx, me.vy);
  }
  cell_move(me, Ctx::dt);
  decelerate(me.svx, me.svy, 80.0f, Ctx::dt);
  bound_cell_r(P.W, me, radius_of(P.T, me.mass));
}

// Engine::move_player + check_player_self_collisions of the multi-cell players, BEFORE the ordered player loop.
// Both depend only on the player's own cells and its target, i.e. on nothing another player does in the same
// tick (pellets, viruses and foods are touched by the later phases of tick_player; cells of other players only by
// players_collision after the loop), so they can leave the serial order: four players of up to 8 cells (then two
// of up to 16) are moved and resolved side by side in lane groups -- in mature games the pair sequences of split
// and popped players are most of the work of a tick.  Not on bot-decision ticks (every 10th): there a target may
// come out of the ordered loop itself.  The results go back to the cell arrays; tick_player skips what is done.
// One batch of the pair solver: up to 32 >> gshift players of one instance (state blob `blob`), one lane group each.
// desc: w0 = gshift | players << 8, w1 / w2 = (player | cells << 8) of the groups, 16 bits each.  Returns the
// players done as a bit mask (lo, hi) and ORs state flags into `flags`; everything else goes back to the cell arrays.
__device__ void premove_batch(const SimParams& P, uint8_t* blob, uint8_t* owner_smem, bool eat, uint32_t w0, uint32_t w1, uint32_t w2, int lane,
                              uint32_t& done_lo, uint32_t& done_hi, uint32_t& flags) {
  const int gshift = (int)(w0 & 0xffu), count = (int)(w0 >> 8), gw = 1 << gshift;
  const int g = lane >> gshift, gl = lane & (gw - 1), gbase = g << gshift;
  const bool have = g < count;
  const uint32_t pn = ((g < 2 ? w1 : w2) >> ((g & 1) * 16)) & 0xffffu;
  const int gp = (int)(pn & 0xffu), gn = have ? (int)(pn >> 8) : 0;
  agarcl_cell* cells = reinterpret_cast<agarcl_cell*>(blob + P.L.off_cells) + (size_t)gp * AGARCL_MAX_CELLS;
  Cell me;
  me.x = me.y = me.vx = me.vy = me.svx = me.svy = 0.0f;
  me.mass = 0; me.id = 0; me.rec = 0;
  float tx = 0.0f, ty = 0.0f;
  const bool valid = have && gl < gn;
  if (have) {
    const agarcl_player* pl = reinterpret_cast<const agarcl_player*>(blob + P.L.off_players) + gp;
    tx = pl->target_x; ty = pl->target_y;
  }
  if (valid) {
    me = cell_load(cells + gl);
    move_cell(P, flags, me, tx, ty);
  }
  me = self_collisions_fn(me, radius_of(P.T, me.mass), gn, tx, ty, gbase, gl, gw, P.W);
  // the results go to the UPPER half of the player's cell slots (kPremoveShadow): the live cells stay as they were until the
  // player's own turn, which is what a looking bot earlier in the order must see on a decision tick (bot_chase reads cells)
  // ... and so does what the cell eats: get_pellets_to_remove_and_increment_cells (Engine.hpp:976-1000) sees the pellets of the
  // tick's start whoever is ticked before (they are removed behind the player loop, :221) and the cell where the solver left it,
  // unless a virus gets in between (tick_player then scans again).  The scan runs against the OWNER's hash and pellet array in
  // shared memory; the new mass, the count and up to kLaneCand indices travel in the unused words of the result slot.
  uint32_t eat_mass = me.mass;
  int eat_n = kEatUnknown;
  uint16_t eat_idx[kLaneCand];
#pragma unroll
  for (int k = 0; k < kLaneCand; k++) eat_idx[k] = 0;
  if (valid && eat) {
    Ctx oc(P);  // (only P and the shared-memory carve-up of the owner are read)
    oc.sm.base = owner_smem;
    oc.sm.o = &P.so;
    oc.lane = lane;
    if (!lane_eat_pellets(oc, me.x, me.y, eat_mass, eat_n, eat_idx)) { eat_n = kEatUnknown; eat_mass = me.mass; }
  }
  if (valid) {
    float4* r = reinterpret_cast<float4*>(cells + kPremoveShadow + gl);
    stg_keep(r, make_float4(me.x, me.y, me.vx, me.vy));
    stg_keep(r + 1, make_float4(me.svx, me.svy, __uint_as_float(eat_mass), __int_as_float(eat_n)));
    static_assert(kLaneCand == 8, "eight 16-bit indices in the slot's last four words");
    stg_keep(reinterpret_cast<int4*>(r + 2), make_int4((int)(eat_idx[0] | (uint32_t)eat_idx[1] << 16), (int)(eat_idx[2] | (uint32_t)eat_idx[3] << 16),
                                                       (int)(eat_idx[4] | (uint32_t)eat_idx[5] << 16), (int)(eat_idx[6] | (uint32_t)eat_idx[7] << 16)));
  }
  const bool mark = have && gl == 0;
  done_lo |= __reduce_or_sync(AG_FULL, (mark && gp < 32) ? 1u << gp : 0u);
  done_hi |= __reduce_or_sync(AG_FULL, (mark && gp >= 32) ? 1u << (gp - 32) : 0u);
}

// The warp's mailbox for the pooled pair solver (scratch that is dead before the player loop):
// [0] batches  [1] [2] players done (lo, hi)  [3] state flags  [4] instance  [5] cycles spent on its batches  [6] pellet eating may be
// resolved against this warp's hash  [8 + 4k ..] batch k
constexpr int kMailHdr = 8, kMailBatches = 40;
static_assert((kMailHdr + 4 * kMailBatches) * 4 <= kCandCap * 8 + (kPremCap * 2 + 15) / 16 * 16 + (kVremCap * 2 + 15) / 16 * 16,
              "the mailbox must fit into cand + prem + vrem: the lanes' speculation (lprem) may run before the pool's barrier");
// What must outlive the mailbox (scratch that the owner's player loop overwrites): [0] batches listed  [1] handed out  [2] completed.
__device__ __forceinline__ volatile uint32_t* pool_slot(const SimParams& P, uint8_t* smem_raw, int warp) {
  return reinterpret_cast<volatile uint32_t*>(smem_raw + P.tiles_bytes + (size_t)warp * P.smem_per_warp + P.so.cold + kColdCtxBytes - 16);
}
__device__ __forceinline__ volatile uint32_t* mailbox(const SimParams& P, uint8_t* smem_raw, int warp) {
  return reinterpret_cast<volatile uint32_t*>(smem_raw + P.tiles_bytes + (size_t)warp * P.smem_per_warp + P.so.cand);
}

// Engine::move_player + check_player_self_collisions of the multi-cell players, BEFORE the ordered player loop.
// Both depend only on the player's own cells and its target, i.e. on nothing another player does in the same
// tick (pellets, viruses and foods are touched by the later phases of tick_player; cells of other players only by
// players_collision after the loop), so they can leave the serial order: four players of up to 8 cells (or two
// of up to 16) are moved and resolved side by side in lane groups -- in mature games the pair sequences of split
// and popped players are most of the work of a tick.  Not on bot-decision ticks (every 10th): there a target may
// come out of the ordered loop itself.  The results go back to the cell arrays; tick_player skips what is done.
//
// POOLED over the CTA (c == nullptr: a warp without an instance in this round only helps): every warp lists the
// batches of its instance in its mailbox and publishes it, and ANY warp takes the next batch of ANY published
// instance of the CTA -- the solver needs nothing but the state blob -- so the instance with three popped players
// no longer keeps fifteen warps waiting at the barrier behind the solver, and a warp that arrives late finds its
// own batches already being worked on.
__device__ void premove_players(const SimParams& P, uint8_t* smem_raw, Ctx* c, int warp, int lane, int tb) {
  const int nw = blockDim.x >> 5;
  volatile uint32_t* mine = mailbox(P, smem_raw, warp);
  uint32_t nb = 0;
  __syncwarp();  // the mailbox lies over scratch the lanes read until the end of the previous tick (collision snapshot, removal lists)
  if (c) {
    const int Pn = P.L.P;
    const bool deciding = c->tick % 10u == 0u;  // bots decide on this tick (Engine.hpp:498-499)
    for (int base = 0; base < Pn; base += 32) {
      const int k = base + lane;
      const int p = k < Pn ? P.L.order[k] : 0;
      int np = k < Pn ? __float_as_int(c->sm.psum()[p].w) : 0;
      if (deciding) {
        // A target that comes out of the ordered loop cannot be premoved -- but HungryBot's does not: it is the pellet nearest
        // to the bot's location at the START of the tick (HungryBot.hpp:19-22, Bot::nearest_pellet Bot.hpp:92-129; pellets
        // only disappear behind the loop), so the multi-cell HungryBots decide HERE, every one on its own lane, and join the
        // pool; agents keep the target of their action.  The bots that look at other players (types 1..3) stay in the loop.
        const int bt = k < Pn ? c->bot_type(p) : 0;
        if (np >= 2 && np <= 16 && bt == 0 && c->n_pellets > 0 && c->hash_valid) {
          const float4 sp = c->sm.psum()[p];
          float tx = 0.0f, ty = 0.0f;
          lane_nearest_pellet(*c, sp.x, sp.y, tx, ty);
          agarcl_player* pl = c->players_() + p;
          pl->target_x = tx; pl->target_y = ty;
          pl->action = 0;
        } else if (bt >= 0) {
          np = 0;  // (decides in the loop: not premoved)
        }
      }
#pragma unroll 1
      for (int wide = 1; wide >= 0; wide--) {  // the long pair sequences (players of 9..16 cells) first
        const int gshift = wide ? 4 : 3, per = 32 >> gshift;
        unsigned todo = __ballot_sync(AG_FULL, wide ? (np > 8 && np <= 16) : (np >= 2 && np <= 8));
        while (todo) {
          uint32_t w1 = 0u, w2 = 0u;  // (two scalars: an array indexed by g lives in local memory)
          int count = 0;
          for (int g = 0; g < per && todo; g++) {
            // the player with the most cells that is left: a batch costs its longest pair sequence, so the long ones go together
            const int src = (int)(warp_max_u32(((todo >> lane) & 1u) ? ((uint32_t)np << 8 | (uint32_t)(31 - lane)) : 0u) & 0xffu) ^ 31;
            todo &= ~(1u << src);
            const uint32_t pn = ((uint32_t)__shfl_sync(AG_FULL, p, src) | ((uint32_t)__shfl_sync(AG_FULL, np, src) << 8)) << ((g & 1) * 16);
            if (g < 2) w1 |= pn; else w2 |= pn;
            count++;
          }
          if (nb < (uint32_t)kMailBatches) {
            if (lane == 0) {
              mine[kMailHdr + 4 * nb] = (uint32_t)gshift | ((uint32_t)count << 8);
              mine[kMailHdr + 4 * nb + 1] = w1;
              mine[kMailHdr + 4 * nb + 2] = w2;
            }
            nb++;
          }  // (more batches than the mailbox holds: tick_player does those players itself)
        }
      }
    }
  }
  // publish: header, then (fenced) this warp's publication counter -- it lives in the spare half of the warp's mbarrier
  // slot, because the mailbox itself is scratch that the rest of the tick overwrites
  volatile uint32_t* pub = reinterpret_cast<volatile uint32_t*>(smem_raw + P.tiles_bytes + (size_t)warp * P.smem_per_warp + P.so.mbar + 8);
  uint32_t epoch = 0u;  // the same in every warp: all of them come here once per tick of a round
  if (lane == 0) epoch = *pub + 1u;
  epoch = __shfl_sync(AG_FULL, epoch, 0);
  if (lane == 0) {
    mine[0] = nb; mine[1] = 0u; mine[2] = 0u; mine[3] = 0u; mine[5] = 0u; mine[7] = 0u;
    volatile uint32_t* ps = pool_slot(P, smem_raw, warp);
    ps[0] = nb; ps[1] = 0u; ps[2] = 0u;
    mine[4] = c ? (uint32_t)c->cold().inst_local : 0u;
    mine[6] = (c && c->n_pellets > 0 && c->hash_valid) ? 1u : 0u;  // the batches may resolve pellet eating against this warp's hash
    __threadfence_block();
    *pub = epoch;
  }
  __syncwarp();
  if (c) c->cold().work += clock64() - c->cold().t_mark;
  // No barrier in front of the pool: a warp that gets here early starts on whatever has been published (its own
  // batches included) instead of waiting for the slowest instance of the CTA to arrive.  It takes the next batch of
  // the mailbox that has handed out the fewest so far (the mailboxes list their long batches first: roughly
  // longest-processing-time order) and leaves when every warp has published and nothing is left to take.
  for (;;) {
    const bool pubd = lane < nw &&
        *reinterpret_cast<volatile uint32_t*>(smem_raw + P.tiles_bytes + (size_t)lane * P.smem_per_warp + P.so.mbar + 8) == epoch;
    volatile uint32_t* ml = pool_slot(P, smem_raw, lane < nw ? lane : 0);
    const uint32_t cnt = pubd ? ml[0] : 0u, tk = pubd ? ml[1] : 0u;
    const bool open = pubd && tk < cnt;
    const unsigned om = __ballot_sync(AG_FULL, open), pm = __ballot_sync(AG_FULL, pubd);
    if (om == 0u) {
      if (__popc(pm) == nw) break;
      __nanosleep(100);
      continue;
    }
    const int owner = (int)(warp_min_u32(open ? (tk << 8 | (uint32_t)lane) : 0xffffffffu) & 0xffu);
    volatile uint32_t* mb = mailbox(P, smem_raw, owner);
    uint32_t idx = 0;
    volatile uint32_t* os = pool_slot(P, smem_raw, owner);
    if (lane == 0) idx = atomicAdd(const_cast<uint32_t*>(os + 1), 1u);
    idx = __shfl_sync(AG_FULL, idx, 0);
    if (idx >= __shfl_sync(AG_FULL, cnt, owner)) continue;  // (another warp was quicker)
    const long long t0 = clock64();
    uint32_t lo = 0u, hi = 0u, fl = 0u;
    premove_batch(P, P.state + (size_t)mb[4] * P.L.stride, smem_raw + P.tiles_bytes + (size_t)owner * P.smem_per_warp, mb[6] != 0u,
                  mb[kMailHdr + 4 * idx], mb[kMailHdr + 4 * idx + 1], mb[kMailHdr + 4 * idx + 2], lane, lo, hi, fl);
    fl = __reduce_or_sync(AG_FULL, fl);
    if (lane == 0) {
      atomicOr(const_cast<uint32_t*>(mb + 1), lo);
      atomicOr(const_cast<uint32_t*>(mb + 2), hi);
      if (fl) atomicOr(const_cast<uint32_t*>(mb + 3), fl);
      atomicAdd(const_cast<uint32_t*>(mb + 5), (uint32_t)(clock64() - t0));
      __threadfence_block();  // the batch's cells and the words above, then the completion count
      atomicAdd(const_cast<uint32_t*>(os + 2), 1u);
    }
  }
  if (tb & 64) {  // the caller finishes the pool (premove_finish) behind the work that does not need its results
    if (c) c->cold().t_mark = clock64();
    return;
  }
  if (tb & 32) {
    // no CTA barrier behind the pool: a warp goes on as soon as ITS batches are done (other warps may still be solving theirs;
    // the barrier in front of players_collision takes up the skew).  Nothing touches a mailbox once its last batch is completed:
    // the hand-out and completion counters live outside the scratch, and a warp cannot list the next tick's batches before every
    // warp of the CTA has left this pool (they all meet at the barrier in front of players_collision first).
    if (lane == 0) {
      volatile uint32_t* ps = pool_slot(P, smem_raw, warp);
      while (ps[2] < nb) __nanosleep(40);
      __threadfence_block();
    }
    __syncwarp();
  } else {
    __threadfence_block();
    if (c) AG_PH(*c, 2);
    align_barrier(nw);  // every batch is done: the cells are back in the cell arrays, the mailboxes say which players
  }
  if (c) {
    c->cold().pre_lo = mine[1]; c->cold().pre_hi = mine[2];
    c->flags |= mine[3];
    c->cold().work += (long long)mine[5];
    c->cold().t_mark = clock64();
  }
  __syncwarp();
}

// The end of the pool when premove_players left it open (tick_barrier bit 64): the CTA barrier, then the results.
__device__ __forceinline__ void premove_finish(const SimParams& P, uint8_t* smem_raw, Ctx* c, int warp) {
  if (c) c->cold().work += clock64() - c->cold().t_mark;
  __threadfence_block();
  align_barrier(blockDim.x >> 5);
  if (c) {
    volatile uint32_t* mine = mailbox(P, smem_raw, warp);
    c->cold().pre_lo = mine[1]; c->cold().pre_hi = mine[2];
    c->flags |= mine[3];
    c->cold().work += (long long)mine[5];
    c->cold().t_mark = clock64();
  }
  __syncwarp();
}

__device__ void tick_player(Ctx& c, int p) {
  const Luts& T = c.P.T;
  agarcl_player* pl = c.players_() + p;
  int n = __float_as_int(c.sm.psum()[p].w);  // == pl->n_cells, without the trip to memory in front of the cell loads
  c.cold().emitted = 0;
  if (n == 0) return;  // dead players are not ticked (Engine.hpp:216)
  const int lane = c.lane;
  AG_PH(c, 22);  // (lane-path time since the last mark)
  // the first 64 bytes of the player record in ONE round trip, next to the cell loads below (every later field access would
  // otherwise be its own dependent trip to L1 / L2 behind the stores in between): w0 n_cells, target x / y, action |
  // w1 split_cd, feed_cd, anti_team_decay, elapsed_ticks | w2 last_decay_tick, bot_type, min_mass_cell, food_eaten |
  // w3 highest_mass, cells_eaten, viruses_eaten, vet_count
  int4 w0, w1, w2, w3;
  {
    const int4* rec = reinterpret_cast<const int4*>(pl);
    w0 = ldg_keep(rec); w1 = ldg_keep(rec + 1); w2 = ldg_keep(rec + 2); w3 = ldg_keep(rec + 3);
  }
  float tx = __int_as_float(w0.y), ty = __int_as_float(w0.z);
  int action = w0.w;
  const int bot_type = w2.y;
  int elapsed = w1.w + 1;

  // Engine::move_player + check_player_self_collisions may have run ahead in the pooled pair solver (premove_players)
  const bool premoved = ((p < 32 ? c.cold().pre_lo >> p : c.cold().pre_hi >> (p - 32)) & 1u) != 0u;
  Cell me;
  me.x = me.y = me.vx = me.vy = me.svx = me.svy = 0.0f;
  me.mass = 0; me.id = 0; me.rec = 0;
  if (lane < n) me = premoved ? cell_load_premoved(c.pcells(p) + lane) : cell_load(c.pcells(p) + lane);

  AG_PH(c, 12);
  // ---- bots decide every 10th tick (Engine.hpp:498-499); a premoved bot has decided already (premove_players)
  if (c.tick % 10u == 0u && bot_type >= 0 && !premoved) {
    float4 s = c.sm.psum()[p];
    float lx = s.x, ly = s.y;
    bool decided = false;
    if (bot_type == 1 || bot_type == 3) {
      if (bot_type == 1) action = 0;
      decided = bot_flee(c, p, lx, ly, tx, ty);
    }
    if (!decided && (bot_type == 2 || bot_type == 3)) decided = bot_chase(c, p, me, n, lx, ly, tx, ty);
    if (!decided) {
      action = 0;
      nearest_pellet(c, lx, ly, tx, ty);
    }
  }

  AG_PH(c, 13);
  // ---- Engine::move_player + check_player_self_collisions (unless premove_players has done them for this tick)
  uint32_t smallest = 0xffffffffu;
  if (lane < n) {
    smallest = me.mass;
    if (!premoved) move_cell(c.P, c.flags, me, tx, ty);
  }
  smallest = warp_min_u32(smallest);
  c.flags = __reduce_or_sync(AG_FULL, c.flags);
  if (n >= 2 && !premoved) self_collisions(c, me, n, tx, ty, 0, lane, 32);

  // ---- created cells accumulate in lanes [n, n+created) (they are inactive until add_cells)
  int created = 0;
  int create_limit = AGARCL_PLAYER_CELL_LIMIT - n;
  const bool can_eat_virus = n >= AGARCL_PLAYER_CELL_LIMIT;
  int viruses_eaten_inc = 0;
  int vet_count = w3.w;

  AG_PH(c, 14);
  // ---- optimized_check_virus_collisions: first hit in (cell, dx, dy, virus index) order
  if (c.n_viruses > 0) {
    // only cells that could eat the smallest virus can touch one at all (mass > 1.1 * virus mass): the 25-mass
    // fragments of a popped player are skipped wholesale
    unsigned vcells = __ballot_sync(AG_FULL, lane < n && can_eat_mass(me.mass, c.cold().min_vmass));
    while (vcells) {
      const int i = __ffs(vcells) - 1;
      vcells &= vcells - 1u;
      float cx = __shfl_sync(AG_FULL, me.x, i), cy = __shfl_sync(AG_FULL, me.y, i);
      uint32_t cm = __shfl_sync(AG_FULL, me.mass, i);
      float cr = radius_of(T, cm);
      int gx = (int)cx / 25, gy = (int)cy / 25;
      uint32_t bestkey = 0xffffffffu;
      for (int base = 0; base < c.n_viruses; base += 32) {
        int v = base + lane;
        uint32_t key = 0xffffffffu;
        if (v < c.n_viruses) {
          float4 vc = c.sm.vcache()[v];
          int vgx = (int)vc.x / 25, vgy = (int)vc.y / 25;
          int ddx = vgx - gx, ddy = vgy - gy;
          uint32_t vm = __float_as_uint(vc.w);
          bool ok = ddx >= -1 && ddx <= 1 && ddy >= -1 && ddy <= 1 && vgx < c.P.gw_virus && vgy < c.P.gw_virus &&
                    can_eat_mass(cm, vm) && collides(cx, cy, cr, vc.x, vc.y, vc.z);
          if (ok) key = ((uint32_t)((ddx + 1) * 3 + (ddy + 1)) << 16) | (uint32_t)v;
        }
        bestkey = min(bestkey, warp_min_u32(key));
      }
      if (bestkey != 0xffffffffu) {
        int v = (int)(bestkey & 0xffffu);
        float4 vc = c.sm.vcache()[v];
        uint32_t vm = __float_as_uint(vc.w);
        if (can_eat_virus) {
          if (lane == i) me.mass = floor_mass(me.mass + vm);
        } else {
          // Engine::disrupt
          Cell par = cell_bcast(me, i);
          uint32_t total = par.mass;
          uint32_t m2 = floor_mass((uint32_t)((float)par.mass / 2.0f));
          m2 = floor_mass(m2 + (total - m2) % 25u);
          uint32_t pop = total - m2;
          int num = (int)((pop + 24u) / 25u);
          if (create_limit < num) num = create_limit;
          if (num < 0) num = 0;
          if (n + num > 32) { num = 32 - n; c.flags |= AGARCL_FLAG_CELL_OVERFLOW; }
          float theta = vel_direction(par.vx, par.vy);
          float sp = max_speed_of(T, 25u, c.flags);
          int ci = lane - n;
          const uint32_t nid = c.cold().next_id;
          if (ci >= 0 && ci < num) {
            float dvel = theta + (float)(2 * AG_PI * ci / num);
            float ang = theta + dvel;
            me.x = vc.x; me.y = vc.y;
            me.vx = par.vx; me.vy = par.vy;
            me.svx = sp * g_sincosf(ang, 1); me.svy = sp * g_sincosf(ang, 0);  // Velocity(angle, speed), core/types.hpp:158-159
            me.mass = 25u;
            me.id = nid + (uint32_t)ci;
            me.rec = c.tick + AGARCL_RECOMBINE_TICKS;
          }
          if (lane == i) { me.mass = m2; me.rec = c.tick + AGARCL_RECOMBINE_TICKS; }
          created += num;
          __syncwarp();
          c.cold().next_id = nid + (uint32_t)num;
        }
        if (c.nvrem < kVremCap) { if (lane == 0) c.sm.vrem()[c.nvrem] = (uint16_t)v; c.nvrem++; }
        else c.flags |= AGARCL_FLAG_REMOVE_OVERFLOW;
        if (vet_count < AGARCL_VET_CAP) { if (lane == 0) pl->vet_ticks[vet_count] = elapsed; vet_count++; }
        else c.flags |= AGARCL_FLAG_VET_OVERFLOW;
        viruses_eaten_inc = 1;
        break;  // only collide once (Engine.hpp:1244)
      }
    }
  }

  AG_PH(c, 15);
  // ---- get_pellets_to_remove_and_increment_cells
  int pellets_eaten = 0;
  bool pellets_done = c.n_pellets == 0;
  if (!pellets_done && n >= 2) {
    // The cells of a player eat independently of each other within a tick (pellets only disappear after the
    // player loop, Engine.hpp:221), so every lane resolves its own cell with the exact single-lane scan; the
    // eaten indices then go to pellets_to_remove in cell order.  Any cell with too many candidates for the
    // lane scan sends the whole player through the cell-by-cell warp scan below.
    uint16_t mine[kLaneCand];
    int ne = 0;
    uint32_t nm = me.mass;
    bool ok = true;
    bool pooled = false;
    if (premoved && viruses_eaten_inc == 0) {
      // the pool has resolved this already (premove_batch), on the cells as the solver left them and the masses of the tick's
      // start -- which is what they still are without a virus contact
      int4 idx = make_int4(0, 0, 0, 0);
      int pne = 0;
      uint32_t pm = me.mass;
      if (lane < n) {
        const float4* r = reinterpret_cast<const float4*>(c.pcells(p) + kPremoveShadow + lane);
        const float4 b = ldg_keep(r + 1);
        idx = ldg_keep(reinterpret_cast<const int4*>(r + 2));
        pm = __float_as_uint(b.z);
        pne = __float_as_int(b.w);
      }
      if (__all_sync(AG_FULL, pne != kEatUnknown)) {
        pooled = true;
        ne = pne;
        nm = pm;
        mine[0] = (uint16_t)idx.x; mine[1] = (uint16_t)((uint32_t)idx.x >> 16); mine[2] = (uint16_t)idx.y; mine[3] = (uint16_t)((uint32_t)idx.y >> 16);
        mine[4] = (uint16_t)idx.z; mine[5] = (uint16_t)((uint32_t)idx.z >> 16); mine[6] = (uint16_t)idx.w; mine[7] = (uint16_t)((uint32_t)idx.w >> 16);
      }
    }
    if (!pooled && lane < n) ok = lane_eat_pellets(c, me.x, me.y, nm, ne, mine);
    if (__all_sync(AG_FULL, ok)) {
      int incl = ne;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(AG_FULL, incl, o);
        if (lane >= o) incl += t;
      }
      const int total = __shfl_sync(AG_FULL, incl, 31);
      if (total > 0) {
        const int off = c.nprem + incl - ne;
        for (int e = 0; e < ne; e++) {
          if (off + e < kPremCap) c.sm.prem()[off + e] = mine[e];
          else c.flags |= AGARCL_FLAG_REMOVE_OVERFLOW;
        }
        c.nprem = min(c.nprem + total, kPremCap);
        c.flags = __reduce_or_sync(AG_FULL, c.flags);
        me.mass = nm;
        pellets_eaten = total;
        __syncwarp();
      }
      pellets_done = true;
    }
  }
  if (!pellets_done) {
    const int HG = c.P.HG;
    const float rp = radius_of(T, 1u);
    for (int i = 0; i < n; i++) {
      float cx = __shfl_sync(AG_FULL, me.x, i), cy = __shfl_sync(AG_FULL, me.y, i);
      uint32_t cm = __shfl_sync(AG_FULL, me.mass, i);
      const int gx = (int)cx / 510, gy = (int)cy / 510;
      float Rc = fmax_std(radius_of(T, cm + (uint32_t)kCandCap), rp);
      float Rc2 = Rc * Rc;
      int hx0 = hash_coord(c, cx - Rc), hx1 = hash_coord(c, cx + Rc);
      int hy0 = hash_coord(c, cy - Rc), hy1 = hash_coord(c, cy + Rc);
      int ncand = 0;
      for (int hy = hy0; hy <= hy1; hy++) {
        int k0 = hy * HG + hx0, k1 = hy * HG + hx1;
        int s = k0 ? (int)c.sm.hcnt()[k0 - 1] : 0, e = (int)c.sm.hcnt()[k1];
        for (int jb = s; jb < e; jb += 32) {
          int j = jb + lane;
          bool cand = false;
          uint32_t key = 0;
          float d2 = 0.f;
          if (j < e) {
            int idx = c.sm.hsorted()[j];
            if (idx != kHashDead) {
              float2 q = c.sm.spel()[idx];
              d2 = sqr_dist(cx, cy, q.x, q.y);
              int bx = (int)q.x / 510 - gx, by = (int)q.y / 510 - gy;
              cand = d2 <= Rc2 && bx >= -1 && bx <= 1 && by >= -1 && by <= 1;
              key = ((uint32_t)((bx + 1) * 3 + (by + 1)) << 16) | (uint32_t)idx;
            }
          }
          unsigned m = __ballot_sync(AG_FULL, cand);
          if (cand) {
            int pos = ncand + __popc(m & lanemask_lt(lane));
            if (pos < kCandCap) c.sm.cand()[pos] = make_uint2(key, __float_as_uint(d2));
          }
          ncand += __popc(m);
        }
      }
      if (ncand == 0) continue;
      __syncwarp();
      uint32_t newmass = cm;
      if (ncand <= kCandCap) {
        // replay the candidates in reference order with the growing mass
        uint2 mine = lane < ncand ? c.sm.cand()[lane] : make_uint2(0xffffffffu, 0u);
        for (int it = 0; it < ncand; it++) {
          uint32_t kmin = warp_min_u32(mine.x);
          unsigned wm = __ballot_sync(AG_FULL, mine.x == kmin);
          int w = __ffs(wm) - 1;
          float d2 = __uint_as_float(__shfl_sync(AG_FULL, mine.y, w));
          float r = fmax_std(radius_of(T, newmass), rp);
          if (r * r >= d2) {  // Ball::collides_with; can_eat(pellet) always holds for mass >= 25
            if (c.nprem < kPremCap) { if (lane == 0) c.sm.prem()[c.nprem] = (uint16_t)(kmin & 0xffffu); c.nprem++; }
            else c.flags |= AGARCL_FLAG_REMOVE_OVERFLOW;
            newmass = floor_mass(newmass + 1u);
            pellets_eaten++;
          }
          if (lane == w) mine.x = 0xffffffffu;
        }
      } else {
        // dense case (giant cell): ordered scan of ALL pellets in the reference's own order
        float Rf = fmax_std(radius_of(T, cm + (uint32_t)c.n_pellets), rp);
        float Rf2 = Rf * Rf;
        for (int dxb = -1; dxb <= 1; dxb++)
          for (int dyb = -1; dyb <= 1; dyb++) {
            int nx = gx + dxb, ny = gy + dyb;
            if (!(nx >= 0 && nx < c.P.gw_pellet && ny >= 0 && ny < c.P.gw_pellet)) continue;
            for (int base = 0; base < c.n_pellets; base += 32) {
              int idx = base + lane;
              bool cand = false;
              float d2 = 0.f;
              if (idx < c.n_pellets) {
                float2 q = c.sm.spel()[idx];
                d2 = sqr_dist(cx, cy, q.x, q.y);
                cand = ((int)q.x / 510 == nx) && ((int)q.y / 510 == ny) && d2 <= Rf2;
              }
              unsigned m = __ballot_sync(AG_FULL, cand);
              while (m) {
                int w = __ffs(m) - 1;
                m &= m - 1;
                float dd = __shfl_sync(AG_FULL, d2, w);
                float r = fmax_std(radius_of(T, newmass), rp);
                if (r * r >= dd) {
                  if (c.nprem < kPremCap) { if (lane == 0) c.sm.prem()[c.nprem] = (uint16_t)(base + w); c.nprem++; }
                  else c.flags |= AGARCL_FLAG_REMOVE_OVERFLOW;
                  newmass = floor_mass(newmass + 1u);
                  pellets_eaten++;
                }
              }
            }
          }
      }
      if (lane == i) me.mass = newmass;
      __syncwarp();
    }
  }
  int food_eaten = w2.w + pellets_eaten;
  uint32_t total_mass = warp_sum_u32(lane < n ? me.mass : 0u);
  uint32_t highest = max((uint32_t)w3.x, total_mass);

  AG_PH(c, 16);
  // ---- may_be_auto_split for every cell (children keep cell order), then eat_food cell by cell
  {
    bool big = lane < n && me.mass >= AGARCL_MAX_MASS_IN_THE_GAME;
    unsigned bm = __ballot_sync(AG_FULL, big);
    if (bm) {
      if (n < AGARCL_PLAYER_CELL_LIMIT) {
        // Engine::cell_split on the parent lanes
        float chx = 0.f, chy = 0.f, chvx = 0.f, chvy = 0.f;
        uint32_t chm = 0;
        if (big) {
          uint32_t split_mass = me.mass / 2u, remaining = me.mass - split_mass;
          me.mass = floor_mass(remaining);
          float ddx = tx - me.x, ddy = ty - me.y;
          float norm = sqrtf(fabsf(ddx) * fabsf(ddx) + fabsf(ddy) * fabsf(ddy));
          float dirx = ddx / norm, diry = ddy / norm;
          float r = radius_of(T, me.mass);
          chx = bound_axis(me.x + dirx * r, r, c.W);
          chy = bound_axis(me.y + diry * r, r, c.W);
          float sp = split_speed_of(T, split_mass, c.flags);
          chvx = dirx * sp; chvy = diry * sp;
          chm = split_mass;
          me.rec = c.tick + AGARCL_RECOMBINE_TICKS;
        }
        int cnt = __popc(bm);
        if (n + created + cnt > 32) c.flags |= AGARCL_FLAG_CELL_OVERFLOW;
        int r = lane - (n + created);
        int src = (r >= 0 && r < cnt) ? (int)__fns(bm, 0, r + 1) : lane;
        float gx_ = __shfl_sync(AG_FULL, chx, src), gy_ = __shfl_sync(AG_FULL, chy, src);
        float gvx = __shfl_sync(AG_FULL, chvx, src), gvy = __shfl_sync(AG_FULL, chvy, src);
        uint32_t gm = __shfl_sync(AG_FULL, chm, src);
        const uint32_t nid = c.cold().next_id;
        if (r >= 0 && r < cnt) {
          me.x = gx_; me.y = gy_; me.vx = gvx; me.vy = gvy; me.svx = gvx; me.svy = gvy;
          me.mass = floor_mass(gm);
          me.id = nid + (uint32_t)r;
          me.rec = c.tick + AGARCL_RECOMBINE_TICKS;
        }
        created += cnt;
        __syncwarp();
        c.cold().next_id = nid + (uint32_t)cnt;
      } else if (big) {
        me.mass = AGARCL_NEW_MASS_IF_NO_SPLIT;
      }
    }
  }
  if (c.n_foods > 0) {
    const float rf = radius_of(T, AGARCL_FOOD_MASS);
    for (int i = 0; i < n; i++) {
      float cx = __shfl_sync(AG_FULL, me.x, i), cy = __shfl_sync(AG_FULL, me.y, i);
      uint32_t cm = __shfl_sync(AG_FULL, me.mass, i);
      float cr = radius_of(T, cm);
      bool eater = can_eat_mass(cm, AGARCL_FOOD_MASS);
      int w = 0;
      const int nf = c.n_foods;
      for (int base = 0; base < nf; base += 32) {
        int j = base + lane;
        float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
        bool keep = false;
        if (j < nf) {
          f = reinterpret_cast<const float4*>(c.food_())[j];
          keep = !(eater && collides(cx, cy, cr, f.x, f.y, rf));
        }
        unsigned km = __ballot_sync(AG_FULL, keep);
        int dst = w + __popc(km & lanemask_lt(lane));
        if (keep && dst != j) reinterpret_cast<float4*>(c.food_())[dst] = f;
        w += __popc(km);
        __syncwarp();
      }
      int num = nf - w;
      if (num) {
        c.n_foods = w;
        if (lane == i) me.mass = floor_mass(me.mass + (uint32_t)num * AGARCL_FOOD_MASS);
        food_eaten += num;
      }
    }
  }
  create_limit -= created;

  AG_PH(c, 17);
  // ---- maybe_emit_food / emit_foods
  int feed_cd = w1.y, split_cd = w1.x;
  if (feed_cd > 0) feed_cd -= 1;
  if (action == 1 && feed_cd == 0) {
    bool emit = lane < n && me.mass >= AGARCL_CELL_MIN_SIZE + AGARCL_FOOD_MASS;
    unsigned em = __ballot_sync(AG_FULL, emit);
    if (emit) {
      float ddx = tx - me.x, ddy = ty - me.y;
      float norm = sqrtf(fabsf(ddx) * fabsf(ddx) + fabsf(ddy) * fabsf(ddy));
      float dirx = ddx / norm, diry = ddy / norm;
      float r = radius_of(T, me.mass);
      int slot = c.n_foods + __popc(em & lanemask_lt(lane));
      if (slot < c.P.L.cap_foods)
        reinterpret_cast<float4*>(c.food_())[slot] = make_float4(me.x + dirx * r, me.y + diry * r, dirx * 100.0f, diry * 100.0f);
      me.mass = floor_mass(me.mass - AGARCL_FOOD_MASS);
    }
    int add = __popc(em);
    if (c.n_foods + add > c.P.L.cap_foods) { c.flags |= AGARCL_FLAG_FOOD_OVERFLOW; add = c.P.L.cap_foods - c.n_foods; }
    c.n_foods += add;
    c.cold().emitted = add;
    feed_cd = 10;
    __syncwarp();
  }

  // ---- maybe_split / player_split
  if (split_cd > 0) split_cd -= 1;
  if (action == 2 && split_cd == 0) {
    if (create_limit != 0) {
      bool elig = lane < n && !(me.mass < AGARCL_CELL_SPLIT_MINIMUM || me.mass < 2u * AGARCL_CELL_MIN_SIZE);
      unsigned eligm = __ballot_sync(AG_FULL, elig);
      int rank = __popc(eligm & lanemask_lt(lane));
      bool split = elig && (create_limit < 0 || rank < create_limit);
      unsigned sm_ = __ballot_sync(AG_FULL, split);
      float chx = 0.f, chy = 0.f, chvx = 0.f, chvy = 0.f;
      uint32_t chm = 0;
      if (split) {
        uint32_t split_mass = me.mass / 2u, remaining = me.mass - split_mass;
        me.mass = floor_mass(remaining);
        float ddx = tx - me.x, ddy = ty - me.y;
        float norm = sqrtf(fabsf(ddx) * fabsf(ddx) + fabsf(ddy) * fabsf(ddy));
        float dirx = ddx / norm, diry = ddy / norm;  // NaN when the target is the cell itself (quirk Q19)
        float r = radius_of(T, me.mass);
        chx = bound_axis(me.x + dirx * r, r, c.W);
        chy = bound_axis(me.y + diry * r, r, c.W);
        float sp = split_speed_of(T, split_mass, c.flags);
        chvx = dirx * sp; chvy = diry * sp;
        chm = split_mass;
        me.rec = c.tick + AGARCL_RECOMBINE_TICKS;
      }
      int cnt = __popc(sm_);
      if (n + created + cnt > 32) c.flags |= AGARCL_FLAG_CELL_OVERFLOW;
      int r = lane - (n + created);
      int src = (r >= 0 && r < cnt) ? (int)__fns(sm_, 0, r + 1) : lane;
      float gx_ = __shfl_sync(AG_FULL, chx, src), gy_ = __shfl_sync(AG_FULL, chy, src);
      float gvx = __shfl_sync(AG_FULL, chvx, src), gvy = __shfl_sync(AG_FULL, chvy, src);
      uint32_t gm = __shfl_sync(AG_FULL, chm, src);
      const uint32_t nid = c.cold().next_id;
      if (r >= 0 && r < cnt) {
        me.x = gx_; me.y = gy_; me.vx = gvx; me.vy = gvy; me.svx = gvx; me.svy = gvy;
        me.mass = floor_mass(gm);
        me.id = nid + (uint32_t)r;
        me.rec = c.tick + AGARCL_RECOMBINE_TICKS;
      }
      created += cnt;
      __syncwarp();
      c.cold().next_id = nid + (uint32_t)cnt;
    }
    split_cd = 30;
  }
  c.flags = __reduce_or_sync(AG_FULL, c.flags);

  // ---- Player::add_cells
  n = min(n + created, 32);

  AG_PH(c, 18);
  // ---- recombine_cells (swap-with-back semantics)
  bool merged = false;  // (a merge moves the last cell into the hole: the only thing that breaks the ascending id order)
  // (a pair merges only if BOTH cells' timers have expired: with fewer than two such cells the pair loop cannot do anything)
  if (n >= 2 && __popc(__ballot_sync(AG_FULL, lane < n && c.tick >= me.rec)) >= 2) {
    for (int a = 0; a < n; a++) {
      uint32_t arec = __shfl_sync(AG_FULL, me.rec, a);
      if (!(c.tick >= arec)) continue;
      int b_cur = a + 1;
      while (true) {
        float ax = __shfl_sync(AG_FULL, me.x, a), ay = __shfl_sync(AG_FULL, me.y, a);
        uint32_t am = __shfl_sync(AG_FULL, me.mass, a);
        bool t = lane >= b_cur && lane < n && c.tick >= me.rec && touches(T, ax, ay, am, me.x, me.y, me.mass);
        unsigned m = __ballot_sync(AG_FULL, t);
        if (!m) break;
        int b = __ffs(m) - 1;
        uint32_t bmass = __shfl_sync(AG_FULL, me.mass, b);
        Cell last = cell_bcast(me, n - 1);
        if (lane == a) me.mass = floor_mass(me.mass + bmass);
        if (lane == b) me = last;
        n--;
        b_cur = b;
        merged = true;
      }
    }
  }

  AG_PH(c, 19);
  // ---- once per 60 player-ticks: anti-team + decay
  float atd = __int_as_float(w1.z);
  int last_decay = w2.x;
  if (c.mass_decay() && elapsed % 60 == 0) {
    int fall_off = elapsed - 60 * 60;
    __syncwarp();
    int t = (lane < vet_count) ? pl->vet_ticks[lane] : 0;
    __syncwarp();
    bool keep = lane < vet_count && !(t < fall_off);
    unsigned km = __ballot_sync(AG_FULL, keep);
    if (keep) pl->vet_ticks[__popc(km & lanemask_lt(lane))] = t;
    vet_count = __popc(km);
    if (vet_count > 0) atd = T.anti_team[vet_count];
    if (elapsed - last_decay >= 60) {
      if (lane < n) {
        uint32_t nm = (uint32_t)((double)me.mass * (1 - 0.002 * (double)atd));
        me.mass = nm > AGARCL_CELL_MIN_SIZE ? nm : AGARCL_CELL_MIN_SIZE;
      }
      last_decay = elapsed;
    }
    __syncwarp();
  }

  if (merged) { if (p < 32) c.cold().sorted_lo &= ~(1u << p); else c.cold().sorted_hi &= ~(1u << (p - 32)); }
  AG_PH(c, 20);
  // ---- publish: centroid for later readers this tick, cells and player record back to the blob
  float4 s = centroid_of(me, n);
  if (lane < n) cell_store(c.pcells(p) + lane, me);
  if (lane == 0) {
    c.sm.psum()[p] = s;
    c.sm.pcell()[p].w = -1.0f;  // not lane-ticked: the collision snapshot reads this player from memory
    int4* rec = reinterpret_cast<int4*>(pl);  // (cells_eaten, w3.y, is players_collision's: carried over)
    stg_keep(rec, make_int4(n, __float_as_int(tx), __float_as_int(ty), action));
    stg_keep(rec + 1, make_int4(split_cd, feed_cd, __float_as_int(atd), elapsed));
    stg_keep(rec + 2, make_int4(last_decay, bot_type, (int)smallest, food_eaten));
    stg_keep(rec + 3, make_int4((int)highest, w3.y, w3.z + viruses_eaten_inc, vet_count));
  }
  __syncwarp();
  AG_PH(c, 21);
}

// ------------------------------------------------------------------------------------------------
// lane-per-player phase.  Inside Engine::tick's player loop (Engine.hpp:214-218) two players only
// interact through (a) the foods list (eat_food / emit_foods) and (b) bots that read the other
// players when they decide (HungryShy / Aggressive / AggressiveShy, every 10th tick); pellets and
// viruses are not removed until the loop is over (:221-222).  A single-cell player that does
// nothing structural this tick (no virus contact, no split / eject, no food in reach, <= kLaneCand
// pellet candidates) is therefore ticked by ONE LANE, up to 32 players at a time, speculatively in
// registers; results are then committed in the reference's player order, and every player that
// does not qualify is ticked by the whole warp (tick_player) at its place in that order.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void hash_range(const Ctx& c, int k0, int k1, int& s, int& e) {
  s = k0 ? (int)c.sm.hcnt()[k0 - 1] : 0;
  e = (int)c.sm.hcnt()[k1];
}

// Visits the hash entries of ring `r` (Chebyshev distance r in hash cells) around cell (hx, hy).
template <typename F>
__device__ __forceinline__ void ring_visit(const Ctx& c, int hx, int hy, int r, F&& f) {
  const int HG = c.P.HG;
  const int x0 = hx - r, x1 = hx + r, y0 = hy - r, y1 = hy + r;
  const int cx0 = max(x0, 0), cx1 = min(x1, HG - 1);
#pragma unroll 1
  for (int yy = max(y0, 0); yy <= min(y1, HG - 1); yy++) {
    const bool edge = (yy == y0) || (yy == y1);
#pragma unroll 1
    for (int side = 0; side < 2; side++) {
      int a, b;
      if (edge) { if (side) break; a = cx0; b = cx1; }
      else if (side == 0) { if (x0 < 0) continue; a = b = x0; }
      else { if (x1 >= HG) continue; a = b = x1; }
      int s, e;
      hash_range(c, yy * HG + a, yy * HG + b, s, e);
#pragma unroll 1
      for (int j = s; j < e; j++) f(j);
    }
  }
}

// Bot::nearest_pellet (Bot.hpp:92-129) by one lane: walks rings of hash cells around the bot until no
// pellet outside the searched block can be nearer than the best one found, evaluating every entry with
// the reference's own comparison on the exact fp32 position (shared memory).  First index among equal
// sqrtf(d^2); d <= 0.01 is skipped as in the reference.
__device__ void lane_nearest_pellet(const Ctx& c, float lx, float ly, float& tx, float& ty) {
  const int HG = c.P.HG;
  const float cw = c.W / (float)HG;
  const float2* pel = c.sm.spel();
  const int hx = hash_coord(c, lx), hy = hash_coord(c, ly);
  const float INF = 3.402823466e+38f;
  float best = INF;
  uint32_t best_i = 0xffffffffu;
#pragma unroll 1
  for (int r = 0; r < HG; r++) {
    ring_visit(c, hx, hy, r, [&](int j) {
      uint32_t idx = c.sm.hsorted()[j];
      if (idx == (uint32_t)kHashDead) return;
      float2 q = pel[idx];
      float d = sqrtf(sqr_dist(lx, ly, q.x, q.y));  // (other - this).norm()
      if ((d < best || (d == best && idx < best_i)) && (double)d > 0.01) { best = d; best_i = idx; }
    });
    // every pellet outside the block lies beyond one of its sides (0.01 covers all fp32 rounding)
    const int x0 = hx - r, x1 = hx + r, y0 = hy - r, y1 = hy + r;
    float bound = INF;
    if (x0 > 0) bound = fminf(bound, lx - (float)x0 * cw);
    if (x1 < HG - 1) bound = fminf(bound, (float)(x1 + 1) * cw - lx);
    if (y0 > 0) bound = fminf(bound, ly - (float)y0 * cw);
    if (y1 < HG - 1) bound = fminf(bound, (float)(y1 + 1) * cw - ly);
    if (bound == INF || best < bound - 0.01f) break;
  }
  if (best_i == 0xffffffffu) { tx = 0.0f; ty = 0.0f; return; }  // nothing qualified: Location() default
  float2 q = pel[best_i];
  tx = q.x; ty = q.y;
}

// get_pellets_to_remove_and_increment_cells (Engine.hpp:976-1000) for one cell by one lane: the
// candidates (same superset as the warp-wide path) are collected by ONE scan of the hash, put into the
// reference's order (bucket offset, then index) and then tested one after the other against the growing
// cell.  false: too many candidates for a lane.
__device__ bool lane_eat_pellets(const Ctx& c, float cx, float cy, uint32_t& mass, int& ne, uint16_t* out) {
  const Luts& T = c.P.T;
  const int HG = c.P.HG;
  const float2* pel = c.sm.spel();
  const float rp = c.P.r_pellet;  // radius_of(T, 1)
  const int gx = (int)cx / 510, gy = (int)cy / 510;
  // candidate radius: any upper bound of the radius the cell can reach in this scan, radius(mass + kCandCap), will do (every
  // candidate is tested with its exact radius below) -- computed, not looked up: most scans find nothing and then never
  // touch the table at all
  const float Rc = fmax_std(__fsqrt_ru(__fmul_ru((float)(mass + (uint32_t)kCandCap), 0.31830990f)) * 1.00001f, rp);
  const float Rc2 = Rc * Rc;
  const int hx0 = hash_coord(c, cx - Rc), hx1 = hash_coord(c, cx + Rc);
  const int hy0 = hash_coord(c, cy - Rc), hy1 = hash_coord(c, cy + Rc);
  // the reference's order key of a pellet: 510-unit bucket offset (dx major, dy minor), then the index
  auto key_of = [&](uint32_t idx) -> uint32_t {
    const float2 q = pel[idx];
    const int bx = (int)q.x / 510 - gx, by = (int)q.y / 510 - gy;
    return ((uint32_t)((bx + 1) * 3 + (by + 1)) << 16) | idx;
  };
  // ONE scan of the hash: the candidates' indices go to `out` (which the eaten ones overwrite from the front afterwards)
  int cnt = 0;
  ne = 0;
#pragma unroll 1
  for (int hy = hy0; hy <= hy1; hy++) {
    int s, e;
    hash_range(c, hy * HG + hx0, hy * HG + hx1, s, e);
#pragma unroll 1
    for (int j = s; j < e; j++) {
      const uint32_t idx = c.sm.hsorted()[j];
      if (idx == (uint32_t)kHashDead) continue;
      const float2 q = pel[idx];
      if (!(sqr_dist(cx, cy, q.x, q.y) <= Rc2)) continue;
      const int bx = (int)q.x / 510 - gx, by = (int)q.y / 510 - gy;
      if (bx >= -1 && bx <= 1 && by >= -1 && by <= 1) {
        if (cnt < kLaneCand) out[cnt] = (uint16_t)idx;
        cnt++;
      }
    }
  }
  if (cnt > kLaneCand) return false;
  if (cnt == 0) return true;
  // ascending key (insertion sort of at most kLaneCand entries; the keys are distinct: they carry the index)
  for (int i = 1; i < cnt; i++) {
    const uint16_t v = out[i];
    const uint32_t kv = key_of(v);
    int j = i - 1;
    while (j >= 0 && key_of(out[j]) > kv) { out[j + 1] = out[j]; j--; }
    out[j + 1] = v;
  }
  uint32_t newmass = mass;
  for (int i = 0; i < cnt; i++) {
    const uint16_t idx = out[i];
    const float2 q = pel[idx];
    const float d2 = sqr_dist(cx, cy, q.x, q.y);
    const float r = fmax_std(radius_of(T, newmass), rp);
    if (r * r >= d2) {  // Ball::collides_with; can_eat(pellet) always holds for mass >= 25
      out[ne++] = idx;
      newmass = floor_mass(newmass + 1u);
    }
  }
  mass = newmass;
  return true;
}

// Lane versions of the scans of the bots that look at other players (HungryShyBot.hpp:26-40,
// AggressiveBot.hpp:33-49, AggressiveShyBot.hpp:30-64 with Bot::edible_mass / target_player, Bot.hpp:55-88):
// same player order, same arithmetic as bot_flee / bot_chase above, run by the bot's own lane.
__device__ bool lane_bot_flee(const Ctx& c, int p, float lx, float ly, float& tx, float& ty) {
  const int P = c.P.L.P;
#pragma unroll 1
  for (int k = 0; k < P; k++) {
    const int o = c.P.L.order[k];
    const float4 s = c.sm.psum()[o];
    const float d = sqrtf(sqr_dist(s.x, s.y, lx, ly));
    if (o != p && d < 25.0f && __float_as_uint(s.z) > 0u) {
      tx = lx - (s.x - lx);
      ty = ly - (s.y - ly);
      return true;
    }
  }
  return false;
}
__device__ bool lane_bot_chase(const Ctx& c, int p, uint32_t big, float lx, float ly, float& tx, float& ty) {
  const int P = c.P.L.P;
#pragma unroll 1
  for (int k = 0; k < P; k++) {
    const int o = c.P.L.order[k];
    const float4 s = c.sm.psum()[o];
    const float d = sqrtf(sqr_dist(s.x, s.y, lx, ly));
    if (o == p || !(d <= 20.0f)) continue;
    const int on = __float_as_int(s.w);
    const agarcl_cell* g = c.pcells(o);
    float sx = 0.0f, sy = 0.0f;
    uint32_t sm = 0;
    bool any = false;
#pragma unroll 1
    for (int i = 0; i < on; i++) {
      const float4 a = reinterpret_cast<const float4*>(g + i)[0];
      const uint32_t mm = g[i].mass;
      if (cell_can_eat_cell(big, mm)) { sx += a.x * (float)mm; sy += a.y * (float)mm; sm += mm; any = true; }
    }
    if (any) {
      const float dsx = sx / (float)sm - lx, dsy = sy / (float)sm - ly;
      tx = lx + dsx * 3.0f;
      ty = ly + dsy * 3.0f;
      return true;
    }
  }
  return false;
}

// What a lane keeps in registers about its player between the ticks of a launch.
struct LaneState {
  Cell me;
  int4 w0, w1, w2, w3;  // first 64 B of the player record
  bool fresh;           // registers == global memory (the lane committed this player itself)
};

__device__ __forceinline__ void tick_players_block(Ctx& c, int base, LaneState& ls, bool pool_open) {
  const Luts& T = c.P.T;
  const int lane = c.lane;
  const int k = base + lane;
  const bool valid = k < c.P.L.P;
  const int p = valid ? c.P.L.order[k] : 0;
  agarcl_player* pl = c.players_() + p;
  Cell& me = ls.me;
  int4 &w0 = ls.w0, &w1 = ls.w1, &w2 = ls.w2, &w3 = ls.w3;
  // the cell count comes from the summary table (== the record's n_cells); only a lane that ticks its player itself (one cell)
  // needs the record and the cell in registers -- the lanes of multi-cell and dead players no longer send the whole warp to
  // memory at the start of every tick
  const int n = valid ? __float_as_int(c.sm.psum()[p].w) : 0;
  if (n == 1 && !ls.fresh) {  // record and cell in ONE round trip
    const int4* rec = reinterpret_cast<const int4*>(pl);
    w0 = ldg_keep(rec); w1 = ldg_keep(rec + 1); w2 = ldg_keep(rec + 2); w3 = ldg_keep(rec + 3);
    me = cell_load(c.pcells(p));
    ls.fresh = true;
  }
  // lane states: a looking bot that decides this tick must see the players before it in the order as already
  // committed, so it is speculated LATE, alone, when the ordered commit reaches it
  enum { kIdle = 0, kPending = 1, kLate = 2, kReady = 3, kSerial = 4 };
  int st = n >= 2 ? kSerial : (n == 1 ? kPending : kIdle);  // dead players are not ticked (Engine.hpp:216)
  if (st == kPending && c.tick % 10u == 0u && c.bot_type(p) > 0) st = kLate;
  float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
  uint32_t food_mass = 0;  // mass at the time of eat_food (after pellets, before decay)
  int ne = 0;
  uint16_t* myeat = c.sm.lprem() + lane * kLaneCand;
  int pos = 0;

 while (true) {
  if (st == kPending || (st == kLate && lane == pos)) do {
    st = kSerial;  // until the speculation reaches its end
    float tx = __int_as_float(w0.y), ty = __int_as_float(w0.z);
    int action = w0.w;
    int split_cd = w1.x, feed_cd = w1.y;
    const float atd = __int_as_float(w1.z);
    const int elapsed = w1.w + 1;
    int last_decay = w2.x;
    const int bot_type = w2.y;
    const int vet_count = w3.w;

    // ---- bots decide every 10th tick (Engine.hpp:498-499; HungryBot.hpp:19-22, HungryShyBot.hpp:23-44,
    //      AggressiveBot.hpp:28-52, AggressiveShyBot.hpp:28-68)
    if (c.tick % 10u == 0u && bot_type >= 0) {
      const float4 s = c.sm.psum()[p];
      bool decided = false;
      if (bot_type == 1 || bot_type == 3) {
        if (bot_type == 1) action = 0;
        decided = lane_bot_flee(c, p, s.x, s.y, tx, ty);
      }
      if (!decided && (bot_type == 2 || bot_type == 3)) decided = lane_bot_chase(c, p, me.mass, s.x, s.y, tx, ty);
      if (!decided) {
        if (c.n_pellets == 0) break;  // libc rand() site: the whole-warp path flags it
        action = 0;
        lane_nearest_pellet(c, s.x, s.y, tx, ty);
      }
    }

    // ---- Engine::move_player (no self-collisions with one cell)
    const uint32_t smallest = me.mass;
    me.vx = 3.0f * (tx - me.x);
    me.vy = 3.0f * (ty - me.y);
    {
      float limit = max_speed_of(T, me.mass, c.flags);
      if (vmag(me.vx, me.vy) > limit) {  // Velocity::clamp_speed + set_speed (quirk Q8)
        me.vx *= limit / vmag(me.vx, me.vy);
        me.vy *= limit / vmag(me.vx, me.vy);
      }
    }
    cell_move(me, c.dt);
    decelerate(me.svx, me.svy, 80.0f, c.dt);
    bound_cell(c, me);

    // ---- optimized_check_virus_collisions: any contact (eat or disrupt) is structural -> serial
    if (c.n_viruses > 0 && can_eat_mass(me.mass, c.cold().min_vmass)) {
      const float cr = radius_of(T, me.mass);
      const int gx = (int)me.x / 25, gy = (int)me.y / 25;
      bool hit = false;
      for (int v = 0; v < c.n_viruses; v++) {
        float4 vc = c.sm.vcache()[v];
        if (collides(me.x, me.y, cr, vc.x, vc.y, vc.z)) {
          int vgx = (int)vc.x / 25, vgy = (int)vc.y / 25;
          int ddx = vgx - gx, ddy = vgy - gy;
          if (ddx >= -1 && ddx <= 1 && ddy >= -1 && ddy <= 1 && vgx < c.P.gw_virus && vgy < c.P.gw_virus &&
              can_eat_mass(me.mass, __float_as_uint(vc.w)))
            hit = true;
        }
      }
      if (hit) break;
    }

    // ---- pellets
    if (c.n_pellets > 0 && !lane_eat_pellets(c, me.x, me.y, me.mass, ne, myeat)) break;
    const int food_eaten = w2.w + ne;
    const uint32_t highest = max((uint32_t)w3.x, me.mass);

    // ---- may_be_auto_split / eat_food / emit / split: anything that happens goes serial
    if (me.mass >= AGARCL_MAX_MASS_IN_THE_GAME) break;
    food_mass = me.mass;
    if (c.n_foods > 0 && can_eat_mass(me.mass, AGARCL_FOOD_MASS)) {
      const float cr = radius_of(T, me.mass), rf = radius_of(T, AGARCL_FOOD_MASS);
      bool hit = false;
      for (int j = 0; j < c.n_foods; j++) {
        float4 f = reinterpret_cast<const float4*>(c.food_())[j];
        if (collides(me.x, me.y, cr, f.x, f.y, rf)) hit = true;
      }
      if (hit) break;
    }
    if (feed_cd > 0) feed_cd -= 1;
    if (action == 1 && feed_cd == 0) {
      if (me.mass >= AGARCL_CELL_MIN_SIZE + AGARCL_FOOD_MASS) break;
      feed_cd = 10;
    }
    if (split_cd > 0) split_cd -= 1;
    if (action == 2 && split_cd == 0) {
      if (!(me.mass < AGARCL_CELL_SPLIT_MINIMUM || me.mass < 2u * AGARCL_CELL_MIN_SIZE)) break;
      split_cd = 30;
    }

    // ---- once per 60 player-ticks: anti-team (only with remembered virus hits -> serial) + decay
    if (c.mass_decay() && elapsed % 60 == 0) {
      if (vet_count > 0) break;
      if (elapsed - last_decay >= 60) {
        uint32_t nm = (uint32_t)((double)me.mass * (1 - 0.002 * (double)atd));
        me.mass = nm > AGARCL_CELL_MIN_SIZE ? nm : AGARCL_CELL_MIN_SIZE;
        last_decay = elapsed;
      }
    }

    // ---- results (Player::x / y / mass with one cell: same fp32 expression as centroid_of)
    float fm = (float)me.mass;
    sum = make_float4((0.0f + me.x * fm) / fm, (0.0f + me.y * fm) / fm, __uint_as_float(me.mass), __int_as_float(1));
    w0.y = __float_as_int(tx); w0.z = __float_as_int(ty); w0.w = action;
    w1.x = split_cd; w1.y = feed_cd; w1.w = elapsed;
    w2.x = last_decay; w2.z = (int)smallest; w2.w = food_eaten;
    w3.x = (int)highest;
    st = kReady;
  } while (0);

  AG_PH(c, 23);
  if (st == kSerial) ls.fresh = false;  // ticked by the whole warp below: registers are stale afterwards
  if (pool_open) {
    // the one-cell players have been speculated on the state of the tick's start; everything from here on (tick_player of the
    // premoved players) needs the pool's results.  A warp that ran out of batches early has done its speculation meanwhile.
    extern __shared__ __align__(128) uint8_t smem_raw[];
    premove_finish(c.P, smem_raw, &c, (int)(threadIdx.x >> 5));
    pool_open = false;
  }
  // ---- ordered commit: the run of speculated players up to the next barrier (a whole-warp player or a late lane)
  {
    const unsigned serm = __ballot_sync(AG_FULL, st == kSerial);
    const unsigned rest = (serm | __ballot_sync(AG_FULL, st == kLate)) & ~lanemask_lt(pos);
    const int nxt = rest ? __ffs(rest) - 1 : 32;
    const bool mine = st == kReady && lane >= pos && lane < nxt;
    if (__ballot_sync(AG_FULL, mine && ne > 0)) {
      // pellets_to_remove keeps the player order (Engine.hpp:212,221)
      int v = mine ? ne : 0, incl = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(AG_FULL, incl, o);
        if (lane >= o) incl += t;
      }
      int off = c.nprem + incl - v;
      for (int e = 0; e < v; e++) {
        if (off + e < kPremCap) c.sm.prem()[off + e] = myeat[e];
        else c.flags |= AGARCL_FLAG_REMOVE_OVERFLOW;
      }
      c.nprem = min(c.nprem + __shfl_sync(AG_FULL, incl, 31), kPremCap);
    }
    if (mine) {
      cell_store(c.pcells(p), me);
      int4* rec = reinterpret_cast<int4*>(pl);
      stg_keep(rec, w0); stg_keep(rec + 1, w1); stg_keep(rec + 2, w2); stg_keep(rec + 3, w3);
      c.sm.psum()[p] = sum;
      c.sm.pcell()[p] = make_float4(me.x, me.y, __uint_as_float(me.mass), 1.0f);
      st = kIdle;
    }
    __syncwarp();
    AG_PH(c, 24);
    if (nxt >= 32) break;
    if (!((serm >> nxt) & 1u)) { pos = nxt; continue; }  // a late lane: it speculates now, on what has been committed
    tick_player(c, c.P.L.order[base + nxt]);
    if (lane == nxt) st = kIdle;
    if (c.cold().emitted > 0) {
      // foods emitted by this player can be eaten by later players in the same tick (Engine.hpp:1011-1025)
      bool hit = false;
      if (st == kReady && lane > nxt && can_eat_mass(food_mass, AGARCL_FOOD_MASS)) {
        const float cr = radius_of(T, food_mass), rf = radius_of(T, AGARCL_FOOD_MASS);
        for (int j = c.n_foods - c.cold().emitted; j < c.n_foods; j++) {
          float4 f = reinterpret_cast<const float4*>(c.food_())[j];
          if (collides(me.x, me.y, cr, f.x, f.y, rf)) hit = true;
        }
      }
      if (hit) { st = kSerial; ls.fresh = false; }
    }
    pos = nxt + 1;
    if (pos >= 32) break;
  }
 }
  c.flags = __reduce_or_sync(AG_FULL, c.flags);
}

// ------------------------------------------------------------------------------------------------
// after the player loop: removals, players_collision, foods, regen
// ------------------------------------------------------------------------------------------------
// the pellet hash is kept across ticks: rename entry `from` of the hash cell containing `pos`
__device__ __forceinline__ void hash_patch(Ctx& c, uint32_t from, uint32_t to, float2 pos) {
  int k = hash_coord(c, pos.y) * c.P.HG + hash_coord(c, pos.x);
  int s = k ? (int)c.sm.hcnt()[k - 1] : 0, e = (int)c.sm.hcnt()[k];
  for (int j = s; j < e; j++)
    if (c.sm.hsorted()[j] == from) { c.sm.hsorted()[j] = (uint16_t)to; break; }
}

__device__ void apply_removals(Ctx& c) {  // Engine.hpp:1002-1009,1253-1260 incl. stale/duplicate indices (Q4/Q5)
  if (c.nprem == 0 && c.nvrem == 0) return;
  if (c.lane == 0) {
    float2* pel = c.sm.spel();
    for (int k = 0; k < c.nprem; k++) {
      uint32_t idx = c.sm.prem()[k], size = (uint32_t)c.n_pellets;
      if (size == 0u) continue;
      uint32_t last = size - 1u;
      if (idx < last) {  // swap-with-back: the pellet at `idx` disappears, the last one takes its index
        float2 pi = pel[idx], pl_ = pel[last];
        if (c.hash_valid) { hash_patch(c, idx, kHashDead, pi); hash_patch(c, last, idx, pl_); }
        pel[idx] = pl_;
      } else if (c.hash_valid) {  // idx == last, or a stale index (Q4): the last pellet is popped
        hash_patch(c, last, kHashDead, pel[last]);
      }
      c.n_pellets--;
    }
    for (int k = 0; k < c.nvrem; k++) {
      uint32_t idx = c.sm.vrem()[k], size = (uint32_t)c.n_viruses;
      if (idx < size - 1u && size > 1u) {
        reinterpret_cast<float4*>(c.vir_() + idx)[0] = reinterpret_cast<float4*>(c.vir_() + size - 1u)[0];
        reinterpret_cast<float4*>(c.vir_() + idx)[1] = reinterpret_cast<float4*>(c.vir_() + size - 1u)[1];
      }
      if (size >= 1u) c.n_viruses--;
    }
  }
  c.n_pellets = __shfl_sync(AG_FULL, c.n_pellets, 0);
  c.n_viruses = __shfl_sync(AG_FULL, c.n_viruses, 0);
  if (c.nvrem > 0) c.vc_valid = false;
  if (c.nprem > 0) c.pel_dirty = true;
  c.nprem = 0;
  c.nvrem = 0;
  __syncwarp();
}

// sort(player.cells) by id (Engine.hpp:157): every tick, for every player, even without collisions
__device__ void sort_player_cells(Ctx& c, int p, int n) {
  Cell me;
  me.x = me.y = me.vx = me.vy = me.svx = me.svy = 0.f; me.mass = 0; me.id = 0xffffffffu; me.rec = 0;
  if (c.lane < n) me = cell_load(c.pcells(p) + c.lane);
  uint32_t prev = __shfl_up_sync(AG_FULL, me.id, 1);
  bool bad = c.lane > 0 && c.lane < n && prev > me.id;
  if (!__ballot_sync(AG_FULL, bad)) return;
  int rank = 0;
  for (int j = 0; j < n; j++) {
    uint32_t oid = __shfl_sync(AG_FULL, me.id, j);
    rank += (oid < me.id) ? 1 : 0;
  }
  if (c.lane < n) cell_store(c.pcells(p) + rank, me);
  __syncwarp();
  Cell s;
  s.x = s.y = s.vx = s.vy = s.svx = s.svy = 0.f; s.mass = 0; s.id = 0; s.rec = 0;
  if (c.lane < n) s = cell_load(c.pcells(p) + c.lane);
  float4 sum = centroid_of(s, n);  // summation order changed
  if (c.lane == 0) c.sm.psum()[p] = sum;
  __syncwarp();
}

__device__ __forceinline__ int get_row(float x, float W) { return (int)(x / W * 100.0f); }  // collision_detection.hpp:17-19

// libstdc++ unordered_map<int,...> insertion-order model (SURVEY Appendix C): place `key` in `list`
__device__ void umap_place(uint16_t* list, int& n, int nb, int key) {
  int b = key % nb, pos = -1;
  for (int i = 0; i < n; i++)
    if (list[i] % nb == b) { pos = i; break; }
  if (pos < 0) pos = 0;
  for (int i = n; i > pos; i--) list[i] = list[i - 1];
  list[pos] = (uint16_t)key;
  n++;
}

struct PairRec { uint16_t q, g; uint32_t eaten_mass, eater_id, eaten_id; };  // 16 B

// exact PrecisionCollisionDetection::solve + application (rare path: only for the query cells the all-pairs
// pre-test flagged; everything the strip sweep can return is in that set).  The strip search is run by the whole
// warp -- the members of a strip are gathered with ballots, ranked by (y, snapshot index) (what the reference's
// std::sort == insertion sort does for <= 16 elements), and the scan from the lower bound to the first own cell is
// one ballot -- because every other warp of the CTA waits at the next barrier while this one is busy here.  Strips
// of more than 32 cells, the results map and the application of the results stay with one lane.
// the pre-test snapshot in shared memory: x[kSnapCap], y[kSnapCap], (mass | player << 24)[kSnapCap] (12 bytes per cell)
__device__ __forceinline__ float* snap_x(const Ctx& c) { return reinterpret_cast<float*>(c.sm.snap()); }
__device__ __forceinline__ float* snap_y(const Ctx& c) { return reinterpret_cast<float*>(c.sm.snap()) + kSnapCap; }
__device__ __forceinline__ uint32_t* snap_mp(const Ctx& c) { return reinterpret_cast<uint32_t*>(c.sm.snap()) + 2 * kSnapCap; }

// The y key of a strip member for strip_std_sort: from the staged snapshot (shared memory) or from the cell itself.  Raw pointers
// only, passed by value: nothing of Ctx may have its address taken (it would move to local memory for the whole kernel).
struct StripKey {
  const float* sy;
  const uint16_t* ref;
  const agarcl_cell* cells;
  __device__ __forceinline__ float operator()(int g) const {
    return sy ? sy[g] : (cells + (size_t)(ref[g] >> 8) * AGARCL_MAX_CELLS + (ref[g] & 0xff))->y;
  }
};

// std::sort as the reference's toolchain implements it (GCC 13 libstdc++, bits/stl_algo.h: __introsort_loop with the median of
// (first + 1, mid, last - 1) moved to first, __unguarded_partition, depth limit 2 * lg(n) with the heap-sort fallback of
// bits/stl_heap.h, then __final_insertion_sort with threshold 16), on the members of one PrecisionCollisionDetection strip
// (collision_detection.hpp:29-31: comparator a.second < b.second), run by ONE lane.  std::sort is not stable: for more than 16
// elements the place of two cells with the SAME y depends on this very sequence of swaps, and that place decides where the scan
// of the strip stops (quirk Q7) -- so it is restated operation for operation, like oracle.c's se_std_sort, which
// tests/test_std_sort.py pins against the real std::sort.  The two halves of a partition are independent, so the recursion is
// an explicit stack (the order in which they are finished does not matter).
__device__ __noinline__ void strip_std_sort(uint16_t* a, int n, StripKey key) {
  if (n <= 0) return;
  auto swp = [&](int i, int j) { const uint16_t t = a[i]; a[i] = a[j]; a[j] = t; };
  auto unguarded_linear_insert = [&](int last) {
    const uint16_t val = a[last];
    const float vy = key(val);
    int next = last - 1;
    while (vy < key(a[next])) { a[last] = a[next]; last = next; --next; }
    a[last] = val;
  };
  auto insertion_sort = [&](int first, int last) {
    if (first == last) return;
    for (int i = first + 1; i != last; ++i) {
      if (key(a[i]) < key(a[first])) {
        const uint16_t val = a[i];
        for (int j = i; j > first; --j) a[j] = a[j - 1];  // move_backward(first, i, i + 1)
        a[first] = val;
      } else {
        unguarded_linear_insert(i);
      }
    }
  };
  // heap routines on a[base .. base + len)
  auto adjust_heap = [&](int base, int hole, int len, uint16_t value) {
    const int top = hole;
    const float vy = key(value);
    int child = hole;
    while (child < (len - 1) / 2) {
      child = 2 * (child + 1);
      if (key(a[base + child]) < key(a[base + child - 1])) child--;
      a[base + hole] = a[base + child];
      hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
      child = 2 * (child + 1);
      a[base + hole] = a[base + child - 1];
      hole = child - 1;
    }
    int parent = (hole - 1) / 2;  // __push_heap
    while (hole > top && key(a[base + parent]) < vy) { a[base + hole] = a[base + parent]; hole = parent; parent = (hole - 1) / 2; }
    a[base + hole] = value;
  };
  auto heap_sort = [&](int first, int last) {  // __partial_sort(first, last, last)
    const int len = last - first;
    if (len >= 2) {
      int parent = (len - 2) / 2;
      for (;;) {
        adjust_heap(first, parent, len, a[first + parent]);
        if (parent == 0) break;
        parent--;
      }
    }
    while (last - first > 1) {
      --last;
      const uint16_t value = a[last];
      a[last] = a[first];
      adjust_heap(first, 0, last - first, value);
    }
  };
  constexpr int kStack = 40;  // one entry per partitioning level: at most 2 * lg(n) + 1 <= 33
  int sf[kStack], sl[kStack], sd[kStack], sp = 0;
  sf[0] = 0; sl[0] = n; sd[0] = 2 * (31 - __clz(n)); sp = 1;
  while (sp > 0) {
    --sp;
    int first = sf[sp], last = sl[sp], depth = sd[sp];
    while (last - first > 16) {
      if (depth == 0) { heap_sort(first, last); break; }
      --depth;
      {  // __move_median_to_first(first, first + 1, mid, last - 1)
        const int A = first + 1, B = first + (last - first) / 2, C = last - 1;
        const float ya = key(a[A]), yb = key(a[B]), yc = key(a[C]);
        int m;
        if (ya < yb) m = (yb < yc) ? B : ((ya < yc) ? C : A);
        else m = (ya < yc) ? A : ((yb < yc) ? C : B);
        swp(first, m);
      }
      const float yp = key(a[first]);
      int lo = first + 1, hi = last;  // __unguarded_partition(first + 1, last, pivot = first)
      for (;;) {
        while (key(a[lo]) < yp) ++lo;
        --hi;
        while (yp < key(a[hi])) --hi;
        if (!(lo < hi)) break;
        swp(lo, hi);
        ++lo;
      }
      if (sp < kStack) { sf[sp] = lo; sl[sp] = last; sd[sp] = depth; sp++; }  // __introsort_loop(cut, last, depth_limit)
      last = lo;
    }
  }
  if (n > 16) {  // __final_insertion_sort
    insertion_sort(0, 16);
    for (int i = 16; i != n; ++i) unguarded_linear_insert(i);
  } else {
    insertion_sort(0, n);
  }
}

__device__ void players_collision_exact(Ctx& c, int total, int nhit, bool staged) {
  const Luts& T = c.P.T;
  const int lane = c.lane;
  const uint16_t* ref = c.sm.cellref();  // (player << 8 | cell) in snapshot order
  const int16_t* rows = c.sm.rows();     // strip id of every snapshot cell (filled by the caller)
  uint16_t* strip = c.sm.strip();        // one strip, sorted by y (stable)
  PairRec* pairs = reinterpret_cast<PairRec*>(c.sm.pairs());
  uint16_t* rkeys = c.sm.reskeys();      // query ids with results, first-insert order
  uint16_t* rorder = c.sm.resorder();    // iteration order of the results map
  auto cellp = [&](int g) -> const agarcl_cell* { return c.pcells(ref[g] >> 8) + (ref[g] & 0xff); };
  // the sweep reads the pre-application snapshot (Engine.hpp:153-166): shared-memory copy when staged
  auto gy_of = [&](int g) -> float { return staged ? snap_y(c)[g] : cellp(g)->y; };
  auto gx_of = [&](int g) -> float { return staged ? snap_x(c)[g] : cellp(g)->x; };
  auto gm_of = [&](int g) -> uint32_t { return staged ? (snap_mp(c)[g] & 0xffffffu) : cellp(g)->mass; };
  int npairs = 0, nres = 0;  // warp-uniform
  for (int hq = 0; hq < nhit; hq++) {
    int q = c.sm.hitq()[hq];
    int qp = ref[q] >> 8;
    const agarcl_cell* qc = cellp(q);
    float qx = gx_of(q), qy = gy_of(q);
    uint32_t qm = gm_of(q);
    float qr = radius_of(T, qm);
    float left = qx - qr, right = qx + qr;
    int top = get_row(left, c.W), bottom = get_row(right, c.W);
    bool opened = false;
    for (int row = top; row <= bottom; row++) {
      // members of the strip, in snapshot order
      int l = 0;
      for (int g0 = 0; g0 < total; g0 += 32) {
        const int g = g0 + lane;
        const bool mem = g < total && rows[g] == row;
        const unsigned bm = __ballot_sync(AG_FULL, mem);
        if (mem) strip[l + __popc(bm & lanemask_lt(lane))] = (uint16_t)g;
        l += __popc(bm);
      }
      if (l == 0) continue;
      __syncwarp();
      const StripKey skey{staged ? snap_y(c) : nullptr, ref, c.cells_()};
      if (l > 32) {  // long strip: one lane, literally
        if (lane == 0) {
          strip_std_sort(strip, l, skey);
          int start_pos = 0;
          for (int j = 10; j >= 0; j--)
            if (start_pos + (1 << j) < l && gy_of(strip[start_pos + (1 << j)]) < left) start_pos += (1 << j);
          for (int j = start_pos; j < l; j++) {
            int g = strip[j];
            int gp = ref[g] >> 8;
            if (gp == qp) break;  // quirk Q7: the scan stops at the first own cell
            uint32_t gm = gm_of(g);
            if (collides(qx, qy, qr, gx_of(g), gy_of(g), radius_of(T, gm)) && cell_can_eat_cell(qm, gm)) {
              const agarcl_cell* gc = cellp(g);
              if (npairs < kPairCap) {
                if (!opened) { rkeys[nres++] = (uint16_t)q; opened = true; }
                pairs[npairs].q = (uint16_t)q; pairs[npairs].g = (uint16_t)g;
                pairs[npairs].eaten_mass = gm; pairs[npairs].eater_id = qc->id; pairs[npairs].eaten_id = gc->id;
                npairs++;
              } else c.flags |= AGARCL_FLAG_EATER_OVERFLOW;
            }
          }
        }
        npairs = __shfl_sync(AG_FULL, npairs, 0);
        nres = __shfl_sync(AG_FULL, nres, 0);
        opened = __shfl_sync(AG_FULL, (int)opened, 0) != 0;
        __syncwarp();
        continue;
      }
      // stable rank by y: lane i holds member i
      const int myg = lane < l ? (int)strip[lane] : 0;
      const float myy = lane < l ? gy_of(myg) : 0.0f;
      int rank = 0;
      for (int j = 0; j < l; j++) {
        const float yj = __shfl_sync(AG_FULL, myy, j);
        rank += (yj < myy || (yj == myy && j < lane)) ? 1 : 0;
      }
      __syncwarp();
      if (lane < l) strip[rank] = (uint16_t)myg;
      __syncwarp();
      int sg = lane < l ? (int)strip[lane] : 0;  // lane j holds position j of the sorted strip
      float sy = lane < l ? gy_of(sg) : 0.0f;
      {
        // more than 16 members AND equal keys: where std::sort leaves the equal ones is up to its unstable part -- one lane redoes
        // the strip from the snapshot order with the reference's own algorithm (rare: cells pressed against a wall)
        const float prev = __shfl_up_sync(AG_FULL, sy, 1);
        if (l > 16 && __ballot_sync(AG_FULL, lane >= 1 && lane < l && sy == prev)) {
          __syncwarp();
          if (lane < l) strip[lane] = (uint16_t)myg;
          __syncwarp();
          if (lane == 0) strip_std_sort(strip, l, skey);
          __syncwarp();
          sg = lane < l ? (int)strip[lane] : 0;
          sy = lane < l ? gy_of(sg) : 0.0f;
        }
      }
      // the reference's lower-bound stepping on a sorted strip: the last position >= 1 whose y is left of the query, else 0
      const unsigned lt = __ballot_sync(AG_FULL, lane >= 1 && lane < l && sy < left);
      const int start_pos = lt ? 31 - __clz(lt) : 0;
      const int gp = lane < l ? (int)(ref[sg] >> 8) : -1;
      const unsigned own = __ballot_sync(AG_FULL, lane >= start_pos && lane < l && gp == qp);
      const int stop = own ? __ffs(own) - 1 : l;  // quirk Q7: the scan stops at the first own cell
      const bool inr = lane >= start_pos && lane < stop;
      const uint32_t gm = inr ? gm_of(sg) : 0u;
      const bool hit = inr && collides(qx, qy, qr, gx_of(sg), sy, radius_of(T, gm)) && cell_can_eat_cell(qm, gm);
      const unsigned hm = __ballot_sync(AG_FULL, hit);
      if (hm) {
        const int pos = npairs + __popc(hm & lanemask_lt(lane));
        const bool fits = hit && pos < kPairCap;
        const unsigned fm = __ballot_sync(AG_FULL, fits);
        if (fm && !opened) {
          if (lane == 0) rkeys[nres] = (uint16_t)q;
          nres++;
          opened = true;
        }
        if (fits) {
          pairs[pos].q = (uint16_t)q; pairs[pos].g = (uint16_t)sg;
          pairs[pos].eaten_mass = gm; pairs[pos].eater_id = qc->id; pairs[pos].eaten_id = cellp(sg)->id;
        }
        if (fm != hm) c.flags |= AGARCL_FLAG_EATER_OVERFLOW;
        npairs += __popc(fm);
      }
      __syncwarp();
    }
  }
  c.flags = __reduce_or_sync(AG_FULL, c.flags);
  __syncwarp();
  if (npairs == 0 || lane != 0) return;
  // iteration order of std::unordered_map<int, vector<...>> results (Engine.hpp:168)
  int cnt = 0, nb = 1, next_resize = 0;
  for (int k = 0; k < nres; k++) {
    if (cnt + 1 > next_resize) {
      int floor_min = (cnt + 1 > (next_resize ? 0 : 11)) ? cnt + 1 : (next_resize ? 0 : 11);
      if (floor_min >= nb) {
        int want = floor_min + 1;
        if (nb * 2 > want) want = nb * 2;
        int nnb = want <= 13 ? 13 : want <= 29 ? 29 : want <= 59 ? 59 : want <= 127 ? 127 : want <= 257 ? 257 : 541;
        next_resize = nnb;
        uint16_t* tmp = strip;  // strip scratch is free now
        for (int i = 0; i < cnt; i++) tmp[i] = rorder[i];
        int m = 0;
        for (int i = 0; i < cnt; i++) umap_place(rorder, m, nnb, tmp[i]);
        nb = nnb;
      } else next_resize = nb;
    }
    umap_place(rorder, cnt, nb, rkeys[k]);
  }
  // apply (Engine.hpp:168-194): eater found by lower_bound on its CURRENT cell list, eaten erased
  for (int oi = 0; oi < cnt; oi++) {
    int q = rorder[oi];
    for (int k = 0; k < npairs; k++) {
      if (pairs[k].q != q) continue;
      int g = pairs[k].g;
      int pp = ref[q] >> 8, ep = ref[g] >> 8;
      agarcl_player* ppl = c.players_() + pp;
      agarcl_player* epl = c.players_() + ep;
      agarcl_cell* pc = c.pcells(pp);
      int pn = ppl->n_cells, it = 0;
      while (it < pn && pc[it].id < pairs[k].eater_id) it++;
      if (it != pn) {
        pc[it].mass = floor_mass(pc[it].mass + pairs[k].eaten_mass);
        ppl->cells_eaten++;
      }
      agarcl_cell* ec = c.pcells(ep);
      int en = epl->n_cells, eit = 0;
      while (eit < en && ec[eit].id < pairs[k].eaten_id) eit++;
      if (eit != en) {
        for (int m = eit; m + 1 < en; m++) {
          reinterpret_cast<uint4*>(ec + m)[0] = reinterpret_cast<uint4*>(ec + m + 1)[0];
          reinterpret_cast<uint4*>(ec + m)[1] = reinterpret_cast<uint4*>(ec + m + 1)[1];
          reinterpret_cast<uint4*>(ec + m)[2] = reinterpret_cast<uint4*>(ec + m + 1)[2];
        }
        epl->n_cells = en - 1;
      }
    }
  }
}

__device__ void players_collision(Ctx& c) {
  const int P = c.P.L.P;
  const int lane = c.lane;
  // 1. sort multi-cell players by id; snapshot enumeration (map order, then cell order)
  int total = 0;
  for (int base = 0; base < P; base += 32) {
    const int k = base + lane;
    const int p = k < P ? c.P.L.order[k] : 0;
    const int n = k < P ? __float_as_int(c.sm.psum()[p].w) : 0;
    unsigned multi = __ballot_sync(AG_FULL, n >= 2);
    while (multi) {
      int src = __ffs(multi) - 1;
      multi &= multi - 1;
      const int sp = __shfl_sync(AG_FULL, p, src);
      // new cells get ascending ids and are appended, erased cells close the gap: a player that was in order stays in order
      // until a merge (tick_player) -- no need to load its cells just to find that out
      if ((sp < 32 ? c.cold().sorted_lo >> sp : c.cold().sorted_hi >> (sp - 32)) & 1u) continue;
      sort_player_cells(c, sp, __shfl_sync(AG_FULL, n, src));
      if (sp < 32) c.cold().sorted_lo |= 1u << sp; else c.cold().sorted_hi |= 1u << (sp - 32);
    }
    int incl = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(AG_FULL, incl, o);
      if (lane >= o) incl += t;
    }
    const int off = total + incl - n;
    for (int i = 0; i < n; i++)
      if (off + i < kCellRefCap) c.sm.cellref()[off + i] = (uint16_t)((p << 8) | i);
    total += __shfl_sync(AG_FULL, incl, 31);
  }
  if (total > kCellRefCap) { c.flags |= AGARCL_FLAG_EATER_OVERFLOW; total = kCellRefCap; }
  __syncwarp();
  // 2. all-pairs pre-test (superset of what the strip sweep can return); hit queries in ascending order.
  //    q can only eat g if mass_q > mass_g, so max(r_q, r_g) = r_q in Ball::collides_with.
  bool staged = total <= kSnapCap;
  if (staged) {
    for (int g = lane; g < total; g += 32) {
      int r = c.sm.cellref()[g];
      float4 pc = c.sm.pcell()[r >> 8];
      float sx, sy;
      uint32_t smass;
      if (pc.w >= 0.0f) {  // lane-ticked single-cell player: its cell is already in shared memory
        sx = pc.x; sy = pc.y; smass = __float_as_uint(pc.z);
      } else {
        const agarcl_cell* gc = c.pcells(r >> 8) + (r & 0xff);
        float4 a = reinterpret_cast<const float4*>(gc)[0];
        sx = a.x; sy = a.y; smass = gc->mass;
      }
      snap_x(c)[g] = sx; snap_y(c)[g] = sy;
      snap_mp(c)[g] = (smass & 0xffffffu) | ((uint32_t)(r >> 8) << 24);
    }
    __syncwarp();
  }
  int nhit = 0;
  for (int qb = 0; qb < total; qb += 32) {
    int q = qb + lane;
    float qx = 0.f, qy = 0.f, qr2 = 0.f;
    uint32_t qm = 0;
    int qp = -1;
    if (q < total) {
      if (staged) {
        const uint32_t mp = snap_mp(c)[q];
        qx = snap_x(c)[q]; qy = snap_y(c)[q]; qm = mp & 0xffffffu; qp = (int)(mp >> 24);
      } else {
        int r = c.sm.cellref()[q];
        qp = r >> 8;
        const agarcl_cell* g = c.pcells(qp) + (r & 0xff);
        float4 a = reinterpret_cast<const float4*>(g)[0];
        qx = a.x; qy = a.y; qm = g->mass;
      }
      float qr = radius_of(c.P.T, qm);
      qr2 = qr * qr;
    }
    bool hungry = qm > 25u;
    if (!__ballot_sync(AG_FULL, hungry)) continue;
    bool hit = false;
    if (staged) {
      for (int g = 0; g < total; g++) {
        const uint32_t mp = snap_mp(c)[g];
        if (qr2 >= sqr_dist(qx, qy, snap_x(c)[g], snap_y(c)[g]) && hungry && (int)(mp >> 24) != qp && can_eat_mass(qm, mp & 0xffffffu))
          hit = true;
      }
    } else {
      for (int g = 0; g < total; g++) {
        int r = c.sm.cellref()[g];
        int gp = r >> 8;
        const agarcl_cell* gc = c.pcells(gp) + (r & 0xff);
        float4 a = reinterpret_cast<const float4*>(gc)[0];
        uint32_t gm = gc->mass;
        if (hungry && gp != qp && qr2 >= sqr_dist(qx, qy, a.x, a.y) && can_eat_mass(qm, gm)) hit = true;
      }
    }
    unsigned hm = __ballot_sync(AG_FULL, hit);
    if (hit) {
      int pos = nhit + __popc(hm & lanemask_lt(lane));
      if (pos < kPairCap) c.sm.hitq()[pos] = (uint16_t)q;
    }
    nhit += __popc(hm);
  }
  if (nhit == 0) return;
  if (nhit > kPairCap) { c.flags |= AGARCL_FLAG_EATER_OVERFLOW; nhit = kPairCap; }
  __syncwarp();
  // 3. exact path: strip ids of the snapshot cells by all lanes, then the serial sweep by one
  for (int g = lane; g < total; g += 32) {
    float x;
    if (staged) x = snap_x(c)[g];
    else { int r = c.sm.cellref()[g]; x = (c.pcells(r >> 8) + (r & 0xff))->x; }
    c.sm.rows()[g] = (int16_t)get_row(x, c.W);
  }
  __syncwarp();
  if (c.P.so.sweep_in_hash) c.hash_valid = false;  // the sweep's scratch (rows above included) lies over the hash's index array
  players_collision_exact(c, total, nhit, staged);
  __syncwarp();
  c.flags = __shfl_sync(AG_FULL, c.flags, 0);
  c.lanes_dirty = true;  // masses / cell lists changed under the lanes' registers
  // 4. refresh summaries (masses / counts changed)
  for (int base = 0; base < P; base += 32) {
    int p = base + lane;
    if (p < P) {
      c.sm.psum()[p] = centroid_from_global(c.pcells(p), c.players_()[p].n_cells);
      c.sm.pcell()[p].w = -1.0f;
    }
  }
  __syncwarp();
}

// Engine::move_foods + maybe_hit_virus, literal and serial (one lane); used when a food may hit a virus
__device__ void move_foods_serial(Ctx& c) {
  const Luts& T = c.P.T;
  const float rf = radius_of(T, AGARCL_FOOD_MASS);
  const float dt = c.dt;
  int nf = c.n_foods, nv = c.n_viruses;
  for (int i = 0; i < nf;) {
    agarcl_food f = c.food_()[i];
    if (vmag(f.vx, f.vy) == 0.0f) { i++; continue; }
    float fvx = f.vx, fvy = f.vy;
    decelerate(f.vx, f.vy, 80.0f, dt);
    f.x += f.vx * dt;
    f.y += f.vy * dt;
    f.x = bound_axis(f.x, rf, c.W);
    f.y = bound_axis(f.y, rf, c.W);
    c.food_()[i] = f;
    bool hit = false;
    for (int v = 0; v < nv; v++) {
      agarcl_virus* vr = c.vir_() + v;
      if (collides(f.x, f.y, rf, vr->x, vr->y, radius_of(T, vr->mass))) {
        if (vr->hits >= 7) {
          vr->hits = 0;
          vr->mass = AGARCL_VIRUS_INITIAL_MASS;
          float dt10 = (float)((1.0 / 30.0) * 10);
          float rv = radius_of(T, AGARCL_VIRUS_INITIAL_MASS);
          float nx = bound_axis(vr->x + fvx * dt10, rv, c.W);
          float ny = bound_axis(vr->y + fvy * dt10, rv, c.W);
          if (nv < c.P.L.cap_viruses) {
            agarcl_virus* nw = c.vir_() + nv;
            nw->x = nx; nw->y = ny; nw->mass = AGARCL_VIRUS_INITIAL_MASS; nw->hits = 0; nw->vx = fvx; nw->vy = fvy;
            nw->pad[0] = 0; nw->pad[1] = 0;
            nv++;
          } else c.flags |= AGARCL_FLAG_VIRUS_OVERFLOW;
        } else {
          vr->hits += 1;
          vr->mass += AGARCL_FOOD_MASS;
        }
        hit = true;
        break;
      }
    }
    if (hit) {
      if (nf > 1) c.food_()[i] = c.food_()[nf - 1];
      nf--;
    } else i++;
  }
  c.n_foods = nf;
  c.n_viruses = nv;
}

__device__ void move_foods(Ctx& c) {
  if (c.n_foods == 0) return;
  const Luts& T = c.P.T;
  const float rf = radius_of(T, AGARCL_FOOD_MASS);
  // pass 1 (pure): would any moving food end inside any virus, even one grown by 70 mass this tick?
  bool danger = false;
  for (int base = 0; base < c.n_foods; base += 32) {
    int j = base + c.lane;
    if (j < c.n_foods) {
      float4 f = reinterpret_cast<const float4*>(c.food_())[j];
      if (vmag(f.z, f.w) != 0.0f) {
        decelerate(f.z, f.w, 80.0f, c.dt);
        f.x = bound_axis(f.x + f.z * c.dt, rf, c.W);
        f.y = bound_axis(f.y + f.w * c.dt, rf, c.W);
        for (int v = 0; v < c.n_viruses; v++) {
          float r = fmax_std(radius_of(T, max(c.vir_()[v].mass, 180u) + 10u), rf);  // a fed virus never exceeds 100 + 7*10
          if (r * r >= sqr_dist(f.x, f.y, c.vir_()[v].x, c.vir_()[v].y)) danger = true;
        }
      }
    }
  }
  if (__ballot_sync(AG_FULL, danger)) {
    c.vc_valid = false;  // a virus may be fed / reset / shot
    if (c.lane == 0) move_foods_serial(c);
    __syncwarp();
    c.n_foods = __shfl_sync(AG_FULL, c.n_foods, 0);
    c.n_viruses = __shfl_sync(AG_FULL, c.n_viruses, 0);
    c.flags = __shfl_sync(AG_FULL, c.flags, 0);
    return;
  }
  // pass 2: no virus can be hit -> foods move independently
  for (int base = 0; base < c.n_foods; base += 32) {
    int j = base + c.lane;
    if (j < c.n_foods) {
      float4 f = reinterpret_cast<const float4*>(c.food_())[j];
      if (vmag(f.z, f.w) != 0.0f) {
        decelerate(f.z, f.w, 80.0f, c.dt);
        f.x += f.z * c.dt;
        f.y += f.w * c.dt;
        f.x = bound_axis(f.x, rf, c.W);
        f.y = bound_axis(f.y, rf, c.W);
        reinterpret_cast<float4*>(c.food_())[j] = f;
      }
    }
  }
  __syncwarp();
}

// add_pellets / add_viruses for the regen tick (Engine.hpp:230-237)
__device__ void regen(Ctx& c) {
  const int inst = c.cold().inst_local;  // (a mixed-task batch tops up to the instance's own sizes)
  int dp = (c.P.task_pellets ? c.P.task_pellets[inst] : c.P.target_pellets) - c.n_pellets;
  if (dp > 0) {
    float r = radius_of(c.P.T, AGARCL_PELLET_MASS);
    const uint32_t cur = c.cold().cursor;
    for (int k = c.lane; k < dp; k += 32) {
      float x, y;
      random_location_at(c, cur + 2u * (uint32_t)k, r, x, y);
      if (c.n_pellets + k < c.P.L.cap_pellets) c.sm.spel()[c.n_pellets + k] = make_float2(x, y);
    }
    __syncwarp();
    c.cold().cursor = cur + 2u * (uint32_t)dp;
    c.n_pellets = min(c.n_pellets + dp, c.P.L.cap_pellets);
    c.hash_valid = false;
    c.pel_dirty = true;
  }
  int dv = (c.P.task_viruses ? c.P.task_viruses[inst] : c.P.target_viruses) - c.n_viruses;
  if (dv > 0) {
    float r = radius_of(c.P.T, AGARCL_VIRUS_INITIAL_MASS);
    int room = c.P.L.cap_viruses - c.n_viruses;
    const uint32_t cur = c.cold().cursor;
    for (int k = c.lane; k < dv; k += 32) {
      float x, y;
      random_location_at(c, cur + 2u * (uint32_t)k, r, x, y);
      if (k < room) {
        float4* v = reinterpret_cast<float4*>(c.vir_() + c.n_viruses + k);
        v[0] = make_float4(x, y, __uint_as_float(AGARCL_VIRUS_INITIAL_MASS), __int_as_float(0));
        v[1] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    __syncwarp();
    c.cold().cursor = cur + 2u * (uint32_t)dv;
    if (dv > room) { c.flags |= AGARCL_FLAG_VIRUS_OVERFLOW; dv = room; }
    c.n_viruses += dv;
    c.vc_valid = false;
  }
  c.flags = __reduce_or_sync(AG_FULL, c.flags);
  __syncwarp();
}

// Fused observation clear: queue the next `nvec` zero vectors of this instance's agent frames as TMA
// bulk stores (cp.async.bulk shared -> global) from the CTA's all-zero tile.  One lane issues one
// instruction per kZeroTileBytes; the copy engine streams them to HBM while the warp goes on ticking,
// so the 7/8 of the observation bytes that do not depend on the state cost no issue slots and never
// stall the tick (the warp only waits for the tile READS to finish before it exits).
__device__ __forceinline__ void zero_chunk(Ctx& c, uint32_t nvec) {
  const uint32_t per = c.P.zero_vec_per_agent;
  if (per == 0u) return;
  ColdCtx& cc = c.cold();
  uint32_t zagent = cc.zagent, zoff = cc.zoff;
  if (zagent >= (uint32_t)c.P.L.A) return;
  const uint32_t inst_local = (uint32_t)cc.inst_local;
  __syncwarp();  // (every lane has read the cursor before any lane moves it)
  while (nvec > 0u && zagent < (uint32_t)c.P.L.A) {
    const uint32_t n = min(nvec, per - zoff);
    if (c.lane == 0) {
      extern __shared__ __align__(128) uint8_t smem_raw[];
      const uint32_t zero_tile = (uint32_t)__cvta_generic_to_shared(smem_raw);
      uint64_t zpolicy;  // L2 evict-first: the observation stream must not push the game state out of L2
      asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(zpolicy));
      uint8_t* dst = reinterpret_cast<uint8_t*>(c.P.obs) +
                     16ull * (((size_t)inst_local * c.P.L.A + zagent) * c.P.agent_stride_vec + c.P.zero_skip_vec + zoff);
      uint32_t bytes = n * 16u;
      while (bytes > 0u) {
        const uint32_t b = min(bytes, (uint32_t)kZeroTileBytes);
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                     :: "l"(dst), "r"(zero_tile), "r"(b), "l"(zpolicy) : "memory");
        dst += b;
        bytes -= b;
      }
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
    nvec -= n;
    zoff += n;
    if (zoff == per) { zoff = 0u; zagent++; }
  }
  cc.zagent = zagent; cc.zoff = zoff;
}

// ------------------------------------------------------------------------------------------------
// GridObservation::add_frame by the warp that owns the instance (environment/envs/GridEnvironment.hpp:
// add_frame 91-123, _store_entities 212-232, _mark_out_of_bounds 235-248, _view_size 251-254,
// _world_to_grid 257-267, _grid_to_world 270-279).  Channels 1..C-1 were cleared by this warp's own
// TMA bulk stores during the ticks; here channel 0 (separable out-of-bounds mask) is streamed and
// the in-view entities are scattered with L2 atomics.  Runs BEFORE repsawn_all_players, like the
// reference (BaseEnvironment.hpp:96-101).  Same arithmetic as k_obs (obs_kernel.cu), int32 only.
// ------------------------------------------------------------------------------------------------
// Element updates of the scatter.  int32 (the reference's dtype): L2 reductions / atomics.  int16 (opt-in, half the bytes):
// there are no 16-bit global atomics, so every update is a CAS on the containing 32-bit word (two grid cells share it),
// saturating at 32767 like k_obs (obs_kernel.cu ObsOps<int16_t>); sums only grow and min / max / set are idempotent, so the
// result does not depend on the order of the updates.
template <typename T> struct FinOps;
template <> struct FinOps<int32_t> {
  static __device__ __forceinline__ void set_stream(int32_t* p, int v) { __stcs(p, v); }
  static __device__ __forceinline__ void add_stream(int32_t* p, int v) { red_add_stream(p, v); }
  static __device__ __forceinline__ void add(int32_t* p, int v) { atomicAdd(p, v); }
  static __device__ __forceinline__ void set(int32_t* p, int v) { *p = v; }
  static __device__ __forceinline__ void min_nz(int32_t* p, int v) {  // empty cell: take the mass; otherwise minimum (masses are > 0)
    const int old = atomicCAS(p, 0, v);
    if (old != 0) atomicMin(p, v);
  }
  static __device__ __forceinline__ void maxs(int32_t* p, int v) { atomicMax(p, v); }
};
template <> struct FinOps<int16_t> {
  template <typename F> static __device__ __forceinline__ void rmw(int16_t* p, F f) {
    unsigned* w = reinterpret_cast<unsigned*>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)3);
    const int sh = (reinterpret_cast<uintptr_t>(p) & 2) ? 16 : 0;
    unsigned old = *reinterpret_cast<volatile unsigned*>(w), assumed;
    do {
      assumed = old;
      const int16_t cur = (int16_t)((assumed >> sh) & 0xffffu);
      const int16_t nv = f(cur);
      if (nv == cur) break;
      old = atomicCAS(w, assumed, (assumed & ~(0xffffu << sh)) | (((unsigned)(uint16_t)nv) << sh));
    } while (old != assumed);
  }
  static __device__ __forceinline__ int16_t sat(int v) { return (int16_t)(v > 32767 ? 32767 : v); }
  static __device__ __forceinline__ void set_stream(int16_t* p, int v) { set(p, v); }
  static __device__ __forceinline__ void add_stream(int16_t* p, int v) { add(p, v); }
  static __device__ __forceinline__ void add(int16_t* p, int v) { rmw(p, [v](int16_t c) { return sat((int)c + v); }); }
  static __device__ __forceinline__ void set(int16_t* p, int v) { const int16_t s = sat(v); rmw(p, [s](int16_t) { return s; }); }
  static __device__ __forceinline__ void min_nz(int16_t* p, int v) { const int16_t s = sat(v); rmw(p, [s](int16_t c) { return (c != 0 && c < s) ? c : s; }); }
  static __device__ __forceinline__ void maxs(int16_t* p, int v) { const int16_t s = sat(v); rmw(p, [s](int16_t c) { return c > s ? c : s; }); }
};

template <typename T>
__device__ void obs_finish_warp(Ctx& c) {
  const SimParams& P = c.P;
  const int G = P.obs_G, lane = c.lane, A = P.L.A, Pn = P.L.P;
  const size_t plane = (size_t)G * G;
  T* yrow = reinterpret_cast<T*>(c.sm.cellref());  // [G]: the collision scratch is free now
  if (!c.vc_valid && P.observe_viruses) { build_virus_cache(c); c.vc_valid = true; }
  // the zero vectors of this instance must have landed before anything is scattered onto them
  if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  __syncwarp();
  __threadfence();
  const float W = c.W;
  const float centering = (float)(G / 2.0);
  const float2* pel = c.sm.spel();
  extern __shared__ __align__(128) uint8_t smem_raw[];
  const uint32_t ones_tile = (uint32_t)__cvta_generic_to_shared(smem_raw + kZeroTileBytes);  // (present with obs_finish)
  const uint32_t yrow_s = (uint32_t)__cvta_generic_to_shared(yrow);
  for (int a = 0; a < A; a++) {
    T* out = reinterpret_cast<T*>(P.obs) + ((size_t)c.cold().inst_local * A + a) * ((size_t)P.agent_stride_vec * (16u / sizeof(T)));
    const float4 s = c.sm.psum()[a];
    const float px = s.x, py = s.y;  // Player::x / y: NaN for a dead agent (quirk Q20)
    const uint32_t tot = __float_as_uint(s.z);
    const int n = __float_as_int(s.w);
    const float view = clamp_std((float)(2u * tot), 100.0f, 300.0f);
    // Channel 0 (_mark_out_of_bounds) is separable: cell (i, j) = xmask[i] | ymask[j] (_grid_to_world + _in_bounds).
    // Row i is therefore either all -1 (x out of bounds) or THE row of y masks: the row lives in shared
    // memory and every lane queues its rows as TMA bulk stores, from it or from the CTA's all-ones tile.
    if (a > 0) {  // the previous agent's stores may still be reading the row
      asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      __syncwarp();
    }
    for (int j = lane; j < G; j += 32) {
      float wy = py + ((float)j - centering) * view / (float)G;
      yrow[j] = (0 <= wy && wy < W) ? (T)0 : (T)-1;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    {
      uint64_t zpolicy;
      asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(zpolicy));
      const uint32_t row_bytes = (uint32_t)G * (uint32_t)sizeof(T);
      for (int i = lane; i < G; i += 32) {
        float wx = px + ((float)i - centering) * view / (float)G;
        const uint32_t src = (0 <= wx && wx < W) ? yrow_s : ones_tile;
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                     :: "l"(out + (size_t)i * G), "r"(src), "r"(row_bytes), "l"(zpolicy) : "memory");
      }
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
    // host-mirror lists (PackOut, sim_params.h): this image's record and entry slot in pinned host memory
    bool emit = P.pk.chunks != nullptr;
    uint32_t* pk_rec = nullptr;
    uint4* pk_ent = nullptr;     // the image's slot, two entries per 16-byte store
    uint32_t pk_mine = 0u;       // lane l holds word l of the record: count, base, image, row masks, column masks
    uint32_t wq = 0u;            // entries listed so far (warp-uniform, even)
    if (emit) {
      const uint32_t slot = (uint32_t)c.cold().pos * (uint32_t)A + (uint32_t)a;  // the image's place in this launch's schedule
      const uint32_t chunk = slot / P.pk.ipc, li = slot - chunk * P.pk.ipc;
      uint32_t* blk = P.pk.chunks + (size_t)chunk * P.pk.chunk_words;
      pk_rec = blk + pk_off_rec(P.pk) + (size_t)li * P.pk.rec_words;
      pk_ent = reinterpret_cast<uint4*>(blk + pk_off_entries(P.pk)) + (size_t)li * (P.pk.slot / 2u);
      if (lane == 1) pk_mine = li * P.pk.slot;
      if (lane == 2) pk_mine = (uint32_t)c.cold().inst_local * (uint32_t)A + (uint32_t)a;  // which image this is
      const int MW = P.pk.MW;
      for (int i0 = 0, w = 0; i0 < G; i0 += 32, w++) {  // the row / column bit masks of channel 0 from the predicates above
        const int i = i0 + lane;
        const float wx = px + ((float)i - centering) * view / (float)G;
        const float wy = py + ((float)i - centering) * view / (float)G;
        const unsigned rb = __ballot_sync(AG_FULL, i < G && !(0 <= wx && wx < W));
        const unsigned cb = __ballot_sync(AG_FULL, i < G && !(0 <= wy && wy < W));
        if (lane == 3 + w) pk_mine = rb;
        if (lane == 3 + MW + w) pk_mine = cb;
      }
    }
    auto grid_of = [&](float x, float y, int& gx, int& gy) -> bool {
      gx = to_int_x86((float)G * (x - px) / view + centering);
      gy = to_int_x86((float)G * (y - py) / view + centering);
      return 0 <= gx && gx < G && 0 <= gy && gy < G;
    };
    // Appends two entries for every lane with `hit` (warp-uniform call): the hit lanes' entries are consecutive, so
    // the warp's stores coalesce into a few PCIe writes.  Entry = (op << 29 | element offset, operand).
    auto list2 = [&](bool hit, uint32_t op0, uint32_t off0, uint32_t v0, uint32_t op1, uint32_t off1, uint32_t v1) {
      if (!emit) return;
      const unsigned m = __ballot_sync(AG_FULL, hit);
      if (m == 0u) return;
      const uint32_t k = wq + 2u * (uint32_t)__popc(m & lanemask_lt(lane));
      wq += 2u * (uint32_t)__popc(m);
      if (hit && k + 2u <= P.pk.slot) pk_ent[k >> 1] = make_uint4(op0 << 29 | off0, v0, op1 << 29 | off1, v1);
    };
    if (n > 0) {  // (a dead agent: nothing lands inside the grid)
      int channel = 0;
      if (P.observe_pellets) {
        const uint32_t o1 = (uint32_t)((channel + 1) * plane), o2 = (uint32_t)((channel + 2) * plane);
        auto put_pellet = [&](bool valid, float2 pq) {
          int gx = 0, gy = 0;
          const bool hit = valid && grid_of(pq.x, pq.y, gx, gy);
          const uint32_t o = (uint32_t)gx * G + gy;
          if (hit) {
            FinOps<T>::set_stream(out + o1 + o, 1);  // at_least_: data = mass (1)
            FinOps<T>::add_stream(out + o2 + o, 1);  // total_mass_
          }
          list2(hit, kPkSet, o1 + o, 1u, kPkAdd, o2 + o, 1u);
        };
        if (c.hash_valid) {
          // only the hash cells under the view: grid_of truncates towards zero, so column 0 reaches one grid
          // cell beyond -view/2; one more world unit of slack on top (grid_of itself is the exact test)
          const int HG = P.HG;
          const float h = 0.5f * view + view / (float)G + 1.0f;
          const int hx0 = hash_coord(c, px - h), hx1 = hash_coord(c, px + h);
          const int hy0 = hash_coord(c, py - h), hy1 = hash_coord(c, py + h);
          for (int hy = hy0; hy <= hy1; hy++) {
            int s0, e0;
            hash_range(c, hy * HG + hx0, hy * HG + hx1, s0, e0);
            for (int j0 = s0; j0 < e0; j0 += 32) {
              const int j = j0 + lane;
              const uint32_t idx = j < e0 ? (uint32_t)c.sm.hsorted()[j] : (uint32_t)kHashDead;
              const bool valid = idx != (uint32_t)kHashDead;
              put_pellet(valid, valid ? pel[idx] : make_float2(0.f, 0.f));
            }
          }
        } else {
          for (int k0 = 0; k0 < c.n_pellets; k0 += 32) {
            const int k = k0 + lane;
            put_pellet(k < c.n_pellets, k < c.n_pellets ? pel[k] : make_float2(0.f, 0.f));
          }
        }
        channel += 2;
      }
      if (P.observe_viruses) {
        const uint32_t o3 = (uint32_t)((channel + 1) * plane), o4 = (uint32_t)((channel + 2) * plane);
        const int nv = c.n_viruses;
        const float4* vc = c.sm.vcache();  // x, y, radius, mass bits: valid (rebuilt above if a virus changed in the last tick)
        for (int k0 = 0; k0 < nv; k0 += 32) {
          const int k = k0 + lane;
          int gx = 0, gy = 0;
          const float4 vk = k < nv ? vc[k] : make_float4(0.f, 0.f, 0.f, 0.f);
          const bool hit = k < nv && grid_of(vk.x, vk.y, gx, gy);
          const uint32_t o = (uint32_t)gx * G + gy;
          const uint32_t vm = __float_as_uint(vk.w);
          bool last = true;
          if (hit) {
            FinOps<T>::add(out + o4 + o, (int)vm);
            // at_least_ keeps the LAST writer in index order: write only if no later virus shares the cell
            for (int k2 = k + 1; k2 < nv; k2++) {
              int hx, hy;
              if (grid_of(vc[k2].x, vc[k2].y, hx, hy) && hx == gx && hy == gy) { last = false; break; }
            }
            if (last) FinOps<T>::set(out + o3 + o, (int)vm);
          }
          list2(hit, kPkAdd, o4 + o, vm, last ? kPkSet : kPkAdd, last ? o3 + o : o4 + o, last ? vm : 0u);  // (not last: a no-op)
        }
        channel += 2;
      }
      if (P.observe_cells) {
        const uint32_t o5 = (uint32_t)((channel + 1) * plane);
        auto put_own = [&](bool valid, float x, float y, uint32_t m) {
          int gx = 0, gy = 0;
          const bool hit = valid && grid_of(x, y, gx, gy);
          const uint32_t o = (uint32_t)gx * G + gy;
          if (hit) FinOps<T>::add(out + o5 + o, (int)m);
          list2(hit, kPkAdd, o5 + o, m, kPkAdd, o5 + o, 0u);  // (entries come in pairs: the second is a no-op)
        };
        const float4 pcv = c.sm.pcell()[a];
        if (n == 1 && pcv.w >= 0.0f) {  // lane-ticked one-cell agent: its cell is in shared memory
          put_own(lane == 0, pcv.x, pcv.y, __float_as_uint(pcv.z));
        } else {
          const agarcl_cell* pc = c.pcells(a);
          for (int k0 = 0; k0 < n; k0 += 32) {
            const int k = k0 + lane;
            const bool v = k < n;
            put_own(v, v ? pc[k].x : 0.f, v ? pc[k].y : 0.f, v ? pc[k].mass : 0u);
          }
        }
        channel += 1;
      }
      if (P.observe_others) {
        const uint32_t o6 = (uint32_t)((channel + 1) * plane);  // min over non-empty
        const uint32_t o7 = (uint32_t)((channel + 2) * plane);  // max
        auto put = [&](bool valid, float x, float y, uint32_t m) {
          int gx = 0, gy = 0;
          const bool hit = valid && grid_of(x, y, gx, gy);
          const uint32_t o = (uint32_t)gx * G + gy;
          if (hit) {
            FinOps<T>::min_nz(out + o6 + o, (int)m);
            FinOps<T>::maxs(out + o7 + o, (int)m);
          }
          list2(hit, kPkMinNz, o6 + o, m, kPkMax, o7 + o, m);
        };
        for (int base = 0; base < Pn; base += 32) {
          const int p = base + lane;
          const int np = p < Pn ? __float_as_int(c.sm.psum()[p].w) : 0;
          {  // first cells: one player per lane
            const bool v = p != a && np >= 1;
            float x = 0.f, y = 0.f;
            uint32_t m = 0u;
            if (v) {
              const float4 pcv = c.sm.pcell()[p];
              if (pcv.w >= 0.0f) { x = pcv.x; y = pcv.y; m = __float_as_uint(pcv.z); }
              else { const agarcl_cell* oc = c.pcells(p); x = oc->x; y = oc->y; m = oc->mass; }
            }
            put(v, x, y, m);
          }
          unsigned multi = __ballot_sync(AG_FULL, p != a && np >= 2);
          while (multi) {  // further cells of split players: one cell per lane
            const int src = __ffs(multi) - 1;
            multi &= multi - 1;
            const int mp = base + src, mn = __shfl_sync(AG_FULL, np, src);
            const agarcl_cell* oc = c.pcells(mp);
            const bool v = lane + 1 < mn;
            put(v, v ? oc[lane + 1].x : 0.f, v ? oc[lane + 1].y : 0.f, v ? oc[lane + 1].mass : 0u);
          }
        }
      }
    }
    if (emit) {  // the image's record in one store: count (or "copy me densely"), base, masks
      if (lane == 0) pk_mine = wq <= P.pk.slot ? wq : kPackDense;
      if (lane < (int)P.pk.rec_words - 3) pk_rec[lane] = pk_mine;  // (the last three words: reward and done, at the end of the step)
    }
  }
}

// Engine::tick
__device__ __forceinline__ void engine_tick(Ctx& c, LaneState& ls) {
  AG_PH(c, 9);
  if (!c.hash_valid) { build_pellet_hash(c); c.hash_valid = true; }
  if (!c.vc_valid) { build_virus_cache(c); c.vc_valid = true; }
  zero_chunk(c, c.cold().zchunk);
  AG_PH(c, 1);
  c.nprem = 0;
  c.nvrem = 0;
  const int P = c.P.L.P;
  if (c.lanes_dirty) { ls.fresh = false; c.lanes_dirty = false; }
  if (c.cold().tb & 2) {  // the pair solver, pooled over the CTA; the warps enter the player loop together behind it
    extern __shared__ __align__(128) uint8_t smem_raw[];
    premove_players(c.P, smem_raw, &c, (int)(threadIdx.x >> 5), c.lane, c.cold().tb);
  } else {
    c.cold().pre_lo = 0u; c.cold().pre_hi = 0u;  // (no alignment barriers: tick_player moves and resolves every player itself)
  }
  AG_PH(c, 3);
  // ONE call site, so that the body is inlined once (two sites made the compiler duplicate ~30 % of the kernel, or -- when it
  // declined -- call it with Ctx in local memory): with more than 32 players every block starts from global memory, which is
  // current because a lane commits its player before it leaves tick_players_block
  for (int base = 0; base < P; base += 32) {
    if (P > 32) ls.fresh = false;
    tick_players_block(c, base, ls, base == 0 && (c.cold().tb & 66) == 66);
  }
  if (P > 32) ls.fresh = false;
  AG_PH(c, 4);
  zero_chunk(c, c.cold().zchunk);
  if (c.cold().tb & 16) { c.cold().work += clock64() - c.cold().t_mark; align_barrier(c.P.align_group); c.cold().t_mark = clock64(); }
  apply_removals(c);
  zero_chunk(c, c.cold().zchunk);
  AG_PH(c, 5);
  if (c.cold().tb & 4) { c.cold().work += clock64() - c.cold().t_mark; align_barrier(c.P.align_group); c.cold().t_mark = clock64(); }  // ... and the cross-player sweep
  AG_PH(c, 6);
  players_collision(c);
  zero_chunk(c, c.cold().zchunk);
  AG_PH(c, 7);
  if (c.cold().tb & 8) { c.cold().work += clock64() - c.cold().t_mark; align_barrier(c.P.align_group); c.cold().t_mark = clock64(); }
  move_foods(c);
  if (c.regen() && c.tick % 120u == 0u) regen(c);
  c.tick++;
  AG_PH(c, 8);
}

// Player::kill + Engine::respawn for a dead player, spawn point from draw pair `k` (Engine.hpp:119-137)
__device__ void respawn_player(Ctx& c, int p, uint32_t k) {
  agarcl_player* pl = c.players_() + p;
  const int agent_mass = c.agent_mass();
  uint32_t mass = (uint32_t)(agent_mass > 25 ? agent_mass : 25);
  float r25 = radius_of(c.P.T, AGARCL_CELL_MIN_SIZE);
  float x, y;
  if (c.n_pellets > 0 && c.squared_pellets()) {
    float2 p0 = c.sm.spel()[0];
    x = fmin_std(p0.x + 2.0f * r25, c.W - r25);
    y = fmin_std(p0.y + 2.0f * r25, c.W - r25);
  } else {
    random_location_at(c, k, r25, x, y);
  }
  Cell n;
  n.x = x; n.y = y; n.vx = n.vy = n.svx = n.svy = 0.0f;
  n.mass = floor_mass(mass);
  n.id = 0;  // assigned by the caller (needs the ordered rank)
  n.rec = c.tick;
  cell_store(c.pcells(p), n);
  pl->n_cells = 1;
  pl->min_mass_cell = AGARCL_CELL_MIN_SIZE;
  pl->split_cd = 0; pl->feed_cd = 0;
  pl->anti_team_decay = 1.0f;
  pl->elapsed_ticks = 0; pl->last_decay_tick = 0;
  pl->vet_count = 0;
}

// ------------------------------------------------------------------------------------------------
// kernel: BaseEnvironment::step for one instance per warp
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void step_instance(const SimParams& P, uint8_t* smem_raw, const int inst, const int pos, const int warp,
                                              const int lane, uint32_t& mbar_phase, const int tb) {
  Ctx c(P);
  c.lane = lane;
#ifdef AGARCL_PHASE_TIMING
  c.ph_t = clock64();
#endif
  c.blob = P.state + (size_t)inst * P.L.stride;
  c.sm.base = smem_raw + P.tiles_bytes + (size_t)warp * P.smem_per_warp;
  c.sm.o = &P.so;
  __syncwarp();  // (the previous instance of this warp is done with the slot)
  c.cold().tb = tb;
  c.cold().pos = pos;
  c.cold().work = 0; c.cold().t_mark = clock64();
  c.cold().inst_local = inst;
  int mode = P.mode;  // (the instance's mode is requested below with the rest of the step's first round trip)
  // the pellet array comes in by one TMA bulk load (whole capacity: the count is not known yet); everything
  // below that does not touch pellets overlaps with it, build_pellet_hash is its first consumer
  const uint32_t pel_bytes = ((uint32_t)P.L.cap_pellets * 8u + 15u) & ~15u;  // pellets are the blob's last array: the pad is inside its stride
  if (lane == 0) {
    const uint32_t mb = (uint32_t)__cvta_generic_to_shared(c.sm.mbar());
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(c.sm.spel());
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(mb), "r"(pel_bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 :: "r"(dst), "l"(c.pel_()), "r"(pel_bytes), "r"(mb), "l"(l2_evict_last()) : "memory");
  }
  agarcl_inst_hdr* hdr = reinterpret_cast<agarcl_inst_hdr*>(c.blob + P.L.off_hdr);
  const int Pn = P.L.P, A = P.L.A;
  // ---- ONE round trip to memory for everything else the step starts from.  Under the observation's store
  // stream a trip to HBM costs microseconds, so nothing here may depend on the value of another load: the
  // header, this lane's player record + first cell (block 0 of the player order), two virus records per
  // lane and the agents' actions are all requested before the first of them is used.
  LaneState ls;
  uint32_t done_sticky;  // lives in ColdCtx across the ticks
  const int k0 = lane;
  const bool valid0 = k0 < Pn;
  const int p0 = valid0 ? P.L.order[k0] : 0;
  {
    const int4* rec = reinterpret_cast<const int4*>(c.players_() + p0);
    ls.w0 = ldg_keep(rec); ls.w1 = ldg_keep(rec + 1); ls.w2 = ldg_keep(rec + 2); ls.w3 = ldg_keep(rec + 3);
    ls.me = cell_load(c.pcells(p0));
    ls.fresh = valid0;
  }
  if (P.task_mode) mode = P.task_mode[inst];
  float4 vpre[2];
#pragma unroll
  for (int j = 0; j < 2; j++) {
    const int v = lane + 32 * j;
    vpre[j] = v < P.L.cap_viruses ? ldg_keep(reinterpret_cast<const float4*>(c.vir_() + v)) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  // actions: for agent `lane` (take_actions below) and for the agent this lane holds in registers
  float adx = 0.f, ady = 0.f, hdx = 0.f, hdy = 0.f;
  int aact = 0, hact = 0;
  if (P.do_begin) {
    if (lane < A) {
      const size_t gi = (size_t)inst * A + lane;
      adx = P.dxdy[2 * gi]; ady = P.dxdy[2 * gi + 1]; aact = P.act[gi];
    }
    if (valid0 && p0 < A) {
      const size_t gi = (size_t)inst * A + p0;
      hdx = P.dxdy[2 * gi]; hdy = P.dxdy[2 * gi + 1]; hact = P.act[gi];
    }
  }
  {
    const int4 h0 = ldg_keep(reinterpret_cast<const int4*>(hdr));
    const int4 h1 = ldg_keep(reinterpret_cast<const int4*>(hdr) + 1);
    const int4 h2 = ldg_keep(reinterpret_cast<const int4*>(hdr) + 2);
    c.tick = (uint32_t)h0.x; c.cold().next_id = (uint32_t)h0.y; c.n_pellets = h0.z; c.n_viruses = h0.w;
    c.n_foods = h1.x; c.cold().cursor = (uint32_t)h1.y; c.flags = (uint32_t)h1.z; done_sticky = (uint32_t)h2.y;
  }
  c.nprem = 0; c.nvrem = 0;
  c.cold().mode = mode;
  c.cold().emitted = 0; c.hash_valid = false; c.vc_valid = false; c.lanes_dirty = false; c.cold().min_vmass = 0xffffffffu;
  c.pel_dirty = false;
  c.cold().sorted_lo = 0u; c.cold().sorted_hi = 0u;
  c.W = P.W;

  // player summaries (centroid, mass, count): from the registers for a one-cell player
  if (valid0) {
    const int n = ls.w0.x;
    float4 sum;
    if (n == 1) {
      const float fm = (float)ls.me.mass;
      sum = make_float4((0.0f + ls.me.x * fm) / fm, (0.0f + ls.me.y * fm) / fm, __uint_as_float(ls.me.mass), __int_as_float(1));
    } else {
      sum = centroid_from_global(c.pcells(p0), n);
    }
    c.sm.psum()[p0] = sum;
    c.sm.pcell()[p0] = make_float4(0.f, 0.f, 0.f, -1.0f);
  }
  for (int base = 32; base < Pn; base += 32) {
    const int k = base + lane;
    if (k < Pn) {
      const int p = P.L.order[k];
      c.sm.psum()[p] = centroid_from_global(c.pcells(p), c.players_()[p].n_cells);
      c.sm.pcell()[p] = make_float4(0.f, 0.f, 0.f, -1.0f);
    }
  }
  // virus cache straight from the prefetched records (build_virus_cache redoes it whenever a virus changes)
  if (c.n_viruses <= 64) {
    uint32_t mn = 0xffffffffu;
#pragma unroll
    for (int j = 0; j < 2; j++) {
      const int v = lane + 32 * j;
      if (v < c.n_viruses) {
        const uint32_t vm = __float_as_uint(vpre[j].z);
        mn = min(mn, vm);
        c.sm.vcache()[v] = make_float4(vpre[j].x, vpre[j].y, radius_of(P.T, vm), vpre[j].z);
      }
    }
    c.cold().min_vmass = warp_min_u32(mn);
    c.vc_valid = true;
  }
  __syncwarp();

  if (P.do_begin) {
    if (lane == 0) { hdr->respawned_lo = 0u; hdr->respawned_hi = 0u; }
    // BaseEnvironment::take_actions + `before = masses<float>()`
    for (int a = lane; a < A; a += 32) {
      float4 s = c.sm.psum()[a];
      uint32_t m = __float_as_uint(s.z);
      size_t gi = (size_t)inst * A + a;
      P.before[gi] = (float)m;
      if (__float_as_int(s.w) > 0) {
        agarcl_player* pl = c.players_() + a;
        if (a >= 32) { adx = P.dxdy[2 * gi]; ady = P.dxdy[2 * gi + 1]; aact = P.act[gi]; }
        pl->target_x = s.x + adx * 10.0f;
        pl->target_y = s.y + ady * 10.0f;
        pl->action = aact;
      }
      if (c.cold().mode == 3 && m >= 23000u) done_sticky = 1u;
    }
    // the lane that holds an agent's record in registers applies the same action to its copy
    if (valid0 && p0 < A && ls.w0.x > 0) {
      const float4 s = c.sm.psum()[p0];
      ls.w0.y = __float_as_int(s.x + hdx * 10.0f);
      ls.w0.z = __float_as_int(s.y + hdy * 10.0f);
      ls.w0.w = hact;
    }
    done_sticky = __reduce_or_sync(AG_FULL, done_sticky);
    __syncwarp();
  }
  c.cold().done_sticky = done_sticky;

  c.cold().zagent = 0u; c.cold().zoff = 0u;
  {
    const uint32_t total = P.zero_vec_per_agent * (uint32_t)A;
    // spread evenly over all ticks: bursts of stores slow the ticks' own loads down more than the
    // last pieces cost the finish in waiting (measured, tools/exp_chunks.sh)
    const uint32_t chunks = P.zero_chunks > 0 ? (uint32_t)P.zero_chunks : (uint32_t)(4 * (P.n_ticks > 0 ? P.n_ticks : 1));
    c.cold().zchunk = (total + chunks - 1u) / chunks;
  }
  {  // the pellets have arrived (all lanes observe the phase flip: their later reads are ordered behind it)
    const uint32_t mb = (uint32_t)__cvta_generic_to_shared(c.sm.mbar());
    uint32_t ok = 0;
    while (!ok) {
      asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                   : "=r"(ok) : "r"(mb), "r"(mbar_phase) : "memory");
    }
    mbar_phase ^= 1u;
  }
  for (int t = 0; t < P.n_ticks; t++) {
    // INSTRUCTION-FETCH ALIGNMENT.  k_step is ~440 KB of code against a 32 KB instruction cache per SM, and 16 warps
    // at unrelated places of it made the kernel instruction-fetch bound (65 % of the stall cycles of steady-state games
    // were no_instruction, profiles/r01l_*).  The warps of the CTA therefore meet inside every tick -- around the pooled
    // pair solver (premove_players, tick_barrier bit 2) and in front of players_collision (bit 4); bits 1 / 8 / 16 are
    // further places kept for A/B timing -- so that they run the same code at about the same time and one fetch serves
    // all of them: no_instruction fell from 10 to 0.5 stall cycles per issued instruction.  Every instance runs the same
    // number of barriers, so the warps move through their instances in rounds (k_step: cost-sorted stripes); what a
    // warp waits for the slowest one is far less than what the shared fetch saves (2.22 -> 1.41 ms per steady-state
    // step with the sorted schedule).  Finer alignment (per solver batch, more phases) loses more than it gains.
    if (c.cold().tb & 1) { c.cold().work += clock64() - c.cold().t_mark; align_barrier(P.align_group); c.cold().t_mark = clock64(); }
    engine_tick(c, ls);
  }
  zero_chunk(c, 0xffffffffu);  // whatever is left (n_ticks == 0, rounding)

  done_sticky = c.cold().done_sticky;
  if (P.do_end) {
    if (P.obs_finish == 1) obs_finish_warp<int32_t>(c);
    else if (P.obs_finish == 2) obs_finish_warp<int16_t>(c);
    const int mode_now = c.cold().mode;
    if (mode_now == 0) {
      // repsawn_all_players in map order: the r-th dead player takes draw pair r.  Players >= Pm are absent (a mixed-task batch's
      // instance of fewer bots): not respawned, ranked or reported
      const int Pm = P.task_bots ? A + P.task_bots[inst] : Pn;
      uint32_t rank_base = 0;
      uint32_t resp_lo = 0, resp_hi = 0;
      for (int base = 0; base < Pn; base += 32) {
        int k = base + lane;
        int p = k < Pn ? P.L.order[k] : 0;
        bool dead = k < Pn && p < Pm && __float_as_int(c.sm.psum()[p].w) == 0;
        unsigned dm = __ballot_sync(AG_FULL, dead);
        if (dead) {
          uint32_t r = rank_base + (uint32_t)__popc(dm & lanemask_lt(lane));
          respawn_player(c, p, c.cold().cursor + 2u * r);
          c.pcells(p)->id = c.cold().next_id + r;
          c.sm.psum()[p] = centroid_from_global(c.pcells(p), 1);
        }
        rank_base += (uint32_t)__popc(dm);
        // dead players in map-order slots -> bit per PLAYER index
        unsigned long long bit = dead ? (1ull << p) : 0ull;
        resp_lo |= __reduce_or_sync(AG_FULL, (uint32_t)(bit & 0xffffffffull));
        resp_hi |= __reduce_or_sync(AG_FULL, (uint32_t)(bit >> 32));
      }
      if (lane == 0) { hdr->respawned_lo = resp_lo; hdr->respawned_hi = resp_hi; }
      c.cold().next_id += rank_base;
      if (!(c.squared_pellets() && c.n_pellets > 0)) c.cold().cursor += 2u * rank_base;
      c.flags = __reduce_or_sync(AG_FULL, c.flags);
      __syncwarp();
    } else if (mode_now > 6) {
      bool dead = false;
      for (int p = lane; p < Pn; p += 32) dead |= __float_as_int(c.sm.psum()[p].w) == 0;
      done_sticky = __ballot_sync(AG_FULL, dead) ? 1u : 0u;  // dones_[0] rewritten every step (BaseEnvironment.hpp:103-114)
    }
    for (int a = lane; a < A; a += 32) {
      uint32_t m = __float_as_uint(c.sm.psum()[a].z);
      if (mode_now == 3 && m >= 23000u) done_sticky = 1u;
    }
    done_sticky = __reduce_or_sync(AG_FULL, done_sticky);
    for (int a = lane; a < A; a += 32) {
      size_t gi = (size_t)inst * A + a;
      uint32_t m = __float_as_uint(c.sm.psum()[a].z);
      double r = (double)m;
      if (P.reward_type) r -= (double)(P.before[gi] - 0.0f);
      P.rewards[gi] = r;
      const uint8_t dn = (a == 0) ? (uint8_t)(done_sticky != 0u) : (uint8_t)0;
      P.dones[gi] = dn;
      if (P.pk.chunks != nullptr && P.obs_finish) {  // host mirror: reward and done travel in the image's record
        const uint32_t slot = (uint32_t)c.cold().pos * (uint32_t)A + (uint32_t)a, chunk = slot / P.pk.ipc, li = slot - chunk * P.pk.ipc;
        uint32_t* tail = P.pk.chunks + (size_t)chunk * P.pk.chunk_words + pk_off_rec(P.pk) + (size_t)li * P.pk.rec_words + (P.pk.rec_words - 3u);
        const unsigned long long rb = (unsigned long long)__double_as_longlong(r);
        tail[0] = (uint32_t)rb; tail[1] = (uint32_t)(rb >> 32); tail[2] = (uint32_t)dn;
      }
    }
  }

  c.flags = __reduce_or_sync(AG_FULL, c.flags);
  if (c.pel_dirty) {  // pellets eaten / spawned: the shared-memory array is the truth, one bulk store puts it back
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane == 0) {
      const uint32_t src = (uint32_t)__cvta_generic_to_shared(c.sm.spel());
      const uint32_t bytes = min(((uint32_t)c.n_pellets * 8u + 15u) & ~15u, pel_bytes);
      if (bytes > 0u) {
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;"
                     :: "l"(c.pel_()), "r"(src), "r"(bytes), "l"(l2_evict_last()) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    }
  }
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // the source tiles / rows / pellets outlive their readers
  if (lane == 0) {
    hdr->tick = c.tick; hdr->next_cell_id = c.cold().next_id;
    hdr->n_pellets = c.n_pellets; hdr->n_viruses = c.n_viruses; hdr->n_foods = c.n_foods;
    hdr->rng_cursor = c.cold().cursor; hdr->flags = c.flags; hdr->done_sticky = done_sticky;
  }
  AG_PH(c, 10);
  if (P.sched) {  // instances that hold a multi-cell player when the launch ends: k_order picks the next launch's schedule from the count
    bool multi = false;
    for (int p = lane; p < Pn; p += 32) multi |= __float_as_int(c.sm.psum()[p].w) >= 2;
    if (__ballot_sync(AG_FULL, multi) && lane == 0) atomicAdd(P.sched + 1, 1u);
  }
  if (P.cost && lane == 0) {  // what the instance cost this step: next step's schedule puts equals together (k_order)
    const long long w = c.cold().work + (clock64() - c.cold().t_mark);
    P.cost[inst] = (uint32_t)(w < 0xffffffffll ? w : 0xffffffffll);
  }
  if (P.pk.chunks != nullptr && P.do_end && P.obs_finish) {
    // host mirror: the warp that finishes the last instance of a chunk rewinds the chunk's counter for the next
    // launch and raises the flag the host polls; the system-scope fences order every warp's list stores (pinned
    // host memory) before the flag (PackOut, sim_params.h)
    __threadfence_system();
    __syncwarp();
    if (lane == 0) {
      const uint32_t chunk = ((uint32_t)pos * (uint32_t)A) / P.pk.ipc;
      const uint32_t in_chunk = min(P.pk.ipc, P.pk.n_img - chunk * P.pk.ipc);
      if (atomicAdd(P.pk.done + chunk, (uint32_t)A) + (uint32_t)A == in_chunk) {
        P.pk.done[chunk] = 0u;
        __threadfence_system();
        P.pk.flags[chunk] = P.pk.seq;
      }
    }
  }
  __syncwarp();
}

// PERSISTENT grid: one CTA per SM (launch_step) of as many warps as the shared memory holds; every warp owns one
// instance at a time and the CTA walks through the batch.  Two schedules:
//   * aligned (tick_barrier != 0, the default): the warps of a CTA meet at barriers inside every tick (step_instance)
//     and therefore move through their instances in rounds; a CTA takes stripes of the cost-sorted order `perm`.
//   * free-running (tick_barrier == 0): every warp draws the next instance from a global ticket counter
//     (tickets[0] = next instance, tickets[1] = warps that have left; the last warp to leave rewinds both, so the next
//     launch on the stream starts from zero again without a memset).
__global__ void __launch_bounds__(kMaxWarpsPerCta * 32, 1) k_step(const __grid_constant__ SimParams P) {
  extern __shared__ __align__(128) uint8_t smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#ifdef AGARCL_PHASE_TIMING
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    printf("PHASES");
    for (int i = 0; i < 28; i++) printf(" %llu", g_phase[i]);
    printf("\n");
    printf("CTAS");
    for (int i = 0; i < (int)gridDim.x && i < 256; i++) printf(" %u", g_cta_cycles[i]);
    printf("\n");
  }
  const long long t_kernel0 = clock64();
#endif
  // the CTA's all-zero tile (first kZeroTileBytes of shared memory), made visible to the async proxy
  // ... and its all-ones (-1) tile right behind it, source of the out-of-bounds rows of channel 0
  for (int i = threadIdx.x; i < (int)P.tiles_bytes / 16; i += blockDim.x)
    reinterpret_cast<int4*>(smem_raw)[i] = i < kZeroTileBytes / 16 ? make_int4(0, 0, 0, 0) : make_int4(-1, -1, -1, -1);
  if (lane == 0) {  // this warp's mbarrier (one arrival: the lane that queues the pellet load)
    const uint32_t mb = (uint32_t)__cvta_generic_to_shared(smem_raw + P.tiles_bytes + (size_t)warp * P.smem_per_warp + P.so.mbar);
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(mb) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // this warp's publication counter of the pooled pair solver (spare half of its mbarrier slot)
  if (lane == 0) *reinterpret_cast<volatile uint32_t*>(smem_raw + P.tiles_bytes + (size_t)warp * P.smem_per_warp + P.so.mbar + 8) = 0u;
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncthreads();
  uint32_t mbar_phase = 0u;
  // The schedule of this launch.  Aligned warps pay for the slowest instance of their CTA at every barrier; that buys the
  // shared instruction fetch mature games need, but young games (every player one cell: short, uniform ticks) run ~10 %
  // faster free.  k_order decides for the NEXT launch from what this one counts: the aligned schedule as soon as 5 % of the
  // instances hold a multi-cell player (P.sched[0]; nullptr: always what tick_barrier says).
  const int tb = (P.sched && *reinterpret_cast<volatile const uint32_t*>(P.sched) == 0u) ? 0 : P.tick_barrier;
  if (tb) {
    // Aligned warps move through their instances in rounds (every instance runs the same number of barriers), so the
    // schedule is static: in round r this CTA takes the r-th stripe of consecutive positions of the cost-sorted order
    // `perm` (k_order: most expensive first, so the instances of one round of one CTA cost about the same and nobody
    // waits long at the barriers), odd rounds in reverse CTA order (the CTAs with the expensive stripes of round r get
    // the cheap ones of round r+1).  The last, partial round is cut into narrower stripes so that it still uses every
    // SM (12 instances on each of 148 SMs run faster than 16 on each of 108).  A warp without an instance in a round
    // arrives at the round's barriers all the same.
    const uint32_t nw = blockDim.x >> 5, per_round = gridDim.x * nw;
    const uint32_t full = (uint32_t)P.N / per_round, rem = (uint32_t)P.N - full * per_round;
    const uint32_t wl = (rem + gridDim.x - 1u) / gridDim.x;  // stripe width of the last round
    const int bars_rest = __popc((unsigned)tb & 28u);  // barriers of a tick behind the pair solver
    // DYNAMIC STRIPES (default).  What a round costs a CTA cannot be predicted well enough from the last step (a rare collision
    // sweep or a popped looking bot on a decision tick makes one CTA's round 50 % longer): with the static pairing the slowest
    // CTA ran 20-35 % longer than the average one and the other SMs idled behind it.  So the stripes of 16 consecutive
    // positions of the cost-sorted order are handed out by a ticket counter, most expensive first: a CTA that comes out of a
    // round early takes the most expensive stripe that is left, one that was held up finds nothing left to take -- list
    // scheduling on the ACTUAL round times.  (s_stripe lives in the spare word of warp 0's pool slot.)
    const uint32_t n_stripes = ((uint32_t)P.N + nw - 1u) / nw;
    volatile uint32_t* s_stripe = pool_slot(P, smem_raw, 0) + 3;
#ifdef AGARCL_PHASE_TIMING
    int rounds_done = 0;
#endif
    for (uint32_t r = 0; P.dyn_stripes || r <= full; r++) {
      uint32_t k = (r & 1u) ? gridDim.x - 1u - blockIdx.x : blockIdx.x;
      uint32_t width = r < full ? nw : wl;
      uint32_t t = r * per_round + k * width + (uint32_t)warp;
      if (P.dyn_stripes) {
        if (threadIdx.x == 0) *s_stripe = atomicAdd(P.tickets, 1u);
        __syncthreads();
        const uint32_t stripe = *s_stripe;
        __syncthreads();  // (everybody has read it before thread 0 draws the next one)
        if (stripe >= n_stripes) break;
#ifdef AGARCL_PHASE_TIMING
        rounds_done++;
#endif
        width = nw;
        t = stripe * nw + (uint32_t)warp;
      }
      if ((uint32_t)warp < width && t < (uint32_t)P.N) {
        const uint32_t inst = P.perm ? P.perm[t] : t;
        step_instance(P, smem_raw, P.inst_first + (int)inst, (int)t, warp, lane, mbar_phase, tb);
      } else {  // no instance in this round: arrive at its barriers, and help with the pooled pair solver
#ifdef AGARCL_PHASE_TIMING
        const long long t_idle0 = clock64();
#endif
        for (int tk = 0; tk < P.n_ticks; tk++) {
          if (tb & 1) align_barrier(P.align_group);
          if (tb & 2) { premove_players(P, smem_raw, nullptr, warp, lane, tb); if (tb & 64) premove_finish(P, smem_raw, nullptr, warp); }
          for (int b = 0; b < bars_rest; b++) align_barrier(P.align_group);
        }
#ifdef AGARCL_PHASE_TIMING
        if (lane == 0) atomicAdd(&g_phase[11], (unsigned long long)(clock64() - t_idle0));
#endif
      }
    }
#ifdef AGARCL_PHASE_TIMING
    if (lane == 0) atomicAdd(&g_phase[0], (unsigned long long)(clock64() - t_kernel0));  // whole kernel, per warp
    if (threadIdx.x == 0 && blockIdx.x < 256) g_cta_cycles[blockIdx.x] = (unsigned int)((clock64() - t_kernel0) >> 10) | ((unsigned int)rounds_done << 28);
#endif
    if (P.dyn_stripes && threadIdx.x == 0) {  // the last CTA to leave rewinds the ticket counter for the next launch
      const uint32_t left = atomicAdd(P.tickets + 1, 1u);
      if (left == gridDim.x - 1u) { P.tickets[0] = 0u; P.tickets[1] = 0u; }
    }
    return;
  }
  while (true) {
    uint32_t t = 0;
    if (lane == 0) t = atomicAdd(P.tickets, 1u);
    t = __shfl_sync(AG_FULL, t, 0);
    if (t >= (uint32_t)P.N) break;
    step_instance(P, smem_raw, P.inst_first + (int)t, (int)t, warp, lane, mbar_phase, 0);
  }
  if (lane == 0) {
    const uint32_t left = atomicAdd(P.tickets + 1, 1u);
    if (left == gridDim.x * (blockDim.x >> 5) - 1u) { P.tickets[0] = 0u; P.tickets[1] = 0u; }
  }
}

// Cost-sorted schedule for the next step (one CTA): perm = instance indices ordered by the cycles they worked in this
// step, most expensive first -- a 256-bucket counting sort on the cost relative to the maximum is all the precision
// the schedule needs (the order inside a bucket is arbitrary; it only moves instances between warps, never results).
__global__ void __launch_bounds__(1024) k_order(const uint32_t* __restrict__ cost, uint32_t* __restrict__ perm, int N, uint32_t* sched) {
  __shared__ uint32_t s_max, cnt[256];
  const int tid = threadIdx.x;
  if (sched && tid == 0) {  // aligned schedule from 5 % multi-cell instances on (k_step), free-running below
    sched[0] = (sched[1] * 20u >= (uint32_t)N) ? 1u : 0u;
    sched[1] = 0u;
  }
  if (tid == 0) s_max = 1u;
  if (tid < 256) cnt[tid] = 0u;
  __syncthreads();
  uint32_t mx = 0u;
  for (int i = tid; i < N; i += 1024) mx = max(mx, cost[i]);
  mx = __reduce_max_sync(AG_FULL, mx);
  if ((tid & 31) == 0) atomicMax(&s_max, mx);
  __syncthreads();
  const float scale = 255.0f / (float)s_max;
  auto bucket = [&](uint32_t c) { return 255 - min(255, (int)((float)c * scale)); };
  for (int i = tid; i < N; i += 1024) atomicAdd(&cnt[bucket(cost[i])], 1u);
  __syncthreads();
  if (tid < 32) {  // exclusive scan of the 256 counters by one warp
    uint32_t carry = 0u;
    for (int b0 = 0; b0 < 256; b0 += 32) {
      const uint32_t v = cnt[b0 + tid];
      uint32_t incl = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(AG_FULL, incl, o);
        if (tid >= o) incl += t;
      }
      cnt[b0 + tid] = carry + incl - v;
      carry += __shfl_sync(AG_FULL, incl, 31);
    }
  }
  __syncthreads();
  for (int i = tid; i < N; i += 1024) perm[atomicAdd(&cnt[bucket(cost[i])], 1u)] = (uint32_t)i;
}
cudaError_t launch_order(const uint32_t* cost, uint32_t* perm, int N, uint32_t* sched, cudaStream_t stream) {
  k_order<<<1, 1024, 0, stream>>>(cost, perm, N, sched);
  return cudaGetLastError();
}

// agarcl_selftest_std_sort (include/agarcl_b200.h): strip_std_sort on keys in global memory, one thread
__global__ void k_selftest_sort(const float* ys, uint16_t* idx, int n) {
  if (threadIdx.x == 0 && blockIdx.x == 0) strip_std_sort(idx, n, StripKey{ys, nullptr, nullptr});
}
cudaError_t selftest_std_sort(const float* ys, int n, uint16_t* order_out) {
  float* d_y = nullptr;
  uint16_t* d_i = nullptr;
  std::vector<uint16_t> init((size_t)n);
  for (int i = 0; i < n; i++) init[(size_t)i] = (uint16_t)i;
  cudaError_t e = cudaMalloc(&d_y, sizeof(float) * (size_t)(n > 0 ? n : 1));
  if (e == cudaSuccess) e = cudaMalloc(&d_i, sizeof(uint16_t) * (size_t)(n > 0 ? n : 1));
  if (e == cudaSuccess && n > 0) e = cudaMemcpy(d_y, ys, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice);
  if (e == cudaSuccess && n > 0) e = cudaMemcpy(d_i, init.data(), sizeof(uint16_t) * (size_t)n, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) { k_selftest_sort<<<1, 32>>>(d_y, d_i, n); e = cudaGetLastError(); }
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e == cudaSuccess && n > 0) e = cudaMemcpy(order_out, d_i, sizeof(uint16_t) * (size_t)n, cudaMemcpyDeviceToHost);
  cudaFree(d_y);
  cudaFree(d_i);
  return e;
}

cudaError_t setup_step(int warps_cap, StepLaunch& S) {
  int dev = 0;
  cudaError_t e;
  if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
  if ((e = cudaDeviceGetAttribute(&S.sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
  if ((e = cudaDeviceGetAttribute(&S.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)) != cudaSuccess) return e;
  S.max_warps = warps_cap > 0 && warps_cap < kMaxWarpsPerCta ? warps_cap : kMaxWarpsPerCta;
  return cudaFuncSetAttribute(k_step, cudaFuncAttributeMaxDynamicSharedMemorySize, S.smem_optin);
}

cudaError_t launch_step(const SimParams& P, const StepLaunch& S, cudaStream_t stream) {
  int warps = (int)(((size_t)S.smem_optin - P.tiles_bytes) / P.smem_per_warp);
  if (warps > S.max_warps) warps = S.max_warps;
  if (warps < 1) return cudaErrorInvalidConfiguration;
  const size_t smem = (size_t)P.tiles_bytes + (size_t)P.smem_per_warp * warps;
  int ctas = (P.N + warps - 1) / warps;
  if (ctas > S.sms) ctas = S.sms;
  k_step<<<ctas, warps * 32, smem, stream>>>(P);
  return cudaGetLastError();
}

}  // namespace ag
