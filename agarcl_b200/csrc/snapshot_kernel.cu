// snapshot_kernel.cu — batched save / restore of game states into a caller-owned pool of slots
// (agarcl_batch_save_states / agarcl_batch_restore_states; slot layout: include/agarcl_b200.h, agarcl_snapshot_hdr), and the
// start states of resets (agarcl_batch_set_start_states, k_start_states).
// A slot is the instance's state blob plus what the blob does not hold: the episode record of the vector environment,
// the ram records (a player with nothing in view keeps its previous one) and, with several frames, the observation
// history.  One CTA per entry; nothing is read back by the host.
#include <cuda_runtime.h>

#include "block_copy.cuh"
#include "sim_params.h"

namespace ag {

// Copies n bytes with every thread of the CTA.  Segments of the state, the ram records and the slot share their alignment
// modulo 16; an observation image of an odd grid may not (its instance offset is not a multiple of 16 while its slot
// offset is), and is then copied byte by byte.
__device__ __forceinline__ void copy_segment(uint8_t* __restrict__ d, const uint8_t* __restrict__ s, size_t n) {
  if ((((uintptr_t)d ^ (uintptr_t)s) & 15u) == 0) {
    block_copy<true>(d, s, n);
    return;
  }
  for (size_t k = threadIdx.x; k < n; k += blockDim.x) d[k] = s[k];
}

// The game sizes (bots, pellets, viruses) a slot of a mixed-task batch carries: its own with the marker, else the maxima (a slot
// saved before sizes were stored)
__device__ __forceinline__ int3 slot_sizes(const SnapParams& P, const agarcl_snapshot_hdr* h) {
  return h->sizes_marker == AGARCL_SNAPSHOT_SIZES_MARKER ? make_int3(h->task_bots, h->task_pellets, h->task_viruses)
                                                         : make_int3(P.lim.bots, P.lim.pellets, P.lim.viruses);
}
// A mixed-task slot's task is one this batch may play: a mode of the set, sizes within the maxima and an allowed bot count
__device__ __forceinline__ bool slot_task_valid(const SnapParams& P, const agarcl_snapshot_hdr* h) {
  const int3 z = slot_sizes(P, h);
  return h->task_mode >= 0 && h->task_mode <= 10 && ((P.task_modes >> h->task_mode) & 1) && sizes_allowed(P.lim, z.x, z.y, z.z);
}
// The slot's task becomes instance i's current one (its step limit is the caller's: the slot's or the pending one)
__device__ __forceinline__ void take_slot_task(const SnapParams& P, const agarcl_snapshot_hdr* h, int i, int32_t max_steps) {
  const int3 z = slot_sizes(P, h);
  P.task_mode[i] = h->task_mode;
  P.task_max_steps[i] = max_steps;
  P.sizes.bots[i] = z.x;
  P.sizes.pellets[i] = z.y;
  P.sizes.viruses[i] = z.z;
}

// Whether slot `slot` (at sl) holds a state this batch may load: in range, saved from this configuration, a task of the batch
// (the restore below makes the same checks)
__device__ __forceinline__ bool slot_valid(const SnapParams& P, int32_t slot, const uint8_t* sl) {
  bool valid = slot < P.pool_slots;
  if (valid) {
    const agarcl_snapshot_hdr* h = reinterpret_cast<const agarcl_snapshot_hdr*>(sl);
    valid = h->magic == AGARCL_SNAPSHOT_MAGIC && h->version == AGARCL_SNAPSHOT_VERSION && h->fingerprint == P.fingerprint &&
            h->slot_bytes == P.S.slot_bytes;
    if (valid && P.task_mode) valid = slot_task_valid(P, h);
  }
  return valid;
}

// The start states of a reset (agarcl_batch_set_start_states), launched in front of k_reset: the game of the slot in place of a
// spawn, on the instance's own draw stream, which goes on where the spawn would have drawn first.  Everything else about the
// reset (episode counters, ram records, observation) is done by the launches behind k_reset with the reset mask, as for a
// spawned instance.  A kernel of its own beside k_snapshot's two directions, whose code stays as it was.
__global__ void __launch_bounds__(kSnapThreads) k_start_states(const __grid_constant__ SnapParams P) {
  const int i = blockIdx.x, t = threadIdx.x, A = P.A;
  const uint8_t reset = P.mask ? P.mask[i] : (uint8_t)1;
  const int32_t slot = reset ? P.slot_of[i] : -1;
  if (slot < 0) {  // not reset, or spawned
    if (t == 0) { P.spawn[i] = reset; P.result[i] = 0; }
    return;
  }
  const uint8_t* sl = P.pool + (uint64_t)slot * P.S.slot_bytes;
  if (!slot_valid(P, slot, sl)) {  // rejected: spawned, as without a start state
    if (t == 0) { P.spawn[i] = 1; P.result[i] = 2; }
    return;
  }
  uint8_t* blob = P.state + (size_t)i * P.stride;
  __shared__ uint32_t cursor;  // (in shared memory: nothing stays live in registers across the copy)
  if (t == 0) cursor = P.fresh[i] ? 0u : reinterpret_cast<const agarcl_inst_hdr*>(blob + P.off_hdr)->rng_cursor;  // where k_reset would draw first
  __syncthreads();  // the cursor is read before the blob is overwritten
  copy_segment(blob, sl + P.S.off_blob, P.stride);
  for (int a = t; a < A; a += blockDim.x) P.dones[(size_t)i * A + a] = 0;
  __syncthreads();  // the slot's header is in place before it is patched
  if (t == 0) {
    agarcl_inst_hdr* hdr = reinterpret_cast<agarcl_inst_hdr*>(P.state + (size_t)i * P.stride + P.off_hdr);
    const uint64_t seed = P.seeds[i];
    hdr->seed_lo = (uint32_t)seed;
    hdr->seed_hi = (uint32_t)(seed >> 32);
    hdr->rng_cursor = cursor;
    hdr->respawned_lo = 0; hdr->respawned_hi = 0;
    if (P.task_mode)  // the game's mode and sizes become the current ones; the step limit belongs to the episode: the pending one
      take_slot_task(P, reinterpret_cast<const agarcl_snapshot_hdr*>(sl), i, P.next_max_steps[i]);
    P.fresh[i] = 0;
    P.spawn[i] = 0;
    P.result[i] = 1;
  }
}

template <bool kSave>
__global__ void __launch_bounds__(kSnapThreads) k_snapshot(const __grid_constant__ SnapParams P) {
  const int t = threadIdx.x, nt = blockDim.x, A = P.A;
  if (kSave) {
    const int k = blockIdx.x;
    const int64_t slot = P.slot ? (int64_t)P.slot[k] : (int64_t)k;
    if (slot < 0 || slot >= P.pool_slots) return;  // skipped
    uint8_t* sl = P.pool + (uint64_t)slot * P.S.slot_bytes;
    const int src = P.src[k];
    const bool ok = src >= 0 && src < P.N;
    if (ok) {
      copy_segment(sl + P.S.off_blob, P.state + (size_t)src * P.stride, P.stride);
      // episode record: steps, then the per-agent return (zeros without bookkeeping), then zero padding
      uint64_t* ep = reinterpret_cast<uint64_t*>(sl + P.S.off_ep);
      for (int w = t; w < (int)(P.S.ep_bytes / 8); w += nt) {
        uint64_t v = 0;
        if (P.steps && w == 0) v = (uint64_t)P.steps[src];
        else if (P.steps && w <= A) v = (uint64_t)__double_as_longlong(P.ret[(size_t)src * A + (w - 1)]);
        ep[w] = v;
      }
      if (P.S.ram_bytes) copy_segment(sl + P.S.off_ram, P.ram + (size_t)src * P.S.ram_bytes, P.S.ram_bytes);
      if (P.S.obs_bytes) copy_segment(sl + P.S.off_obs, P.obs + (size_t)src * P.S.obs_bytes, P.S.obs_bytes);
    }
    __syncthreads();  // the header goes last; a source out of range leaves magic 0, which a restore rejects
    if (t == 0) {  // agarcl_snapshot_hdr: magic, version, fingerprint, slot_bytes, source, task and sizes (mixed-task batch), zero padding
      const uint4 z = make_uint4(0u, 0u, 0u, 0u);
      uint4* hv = reinterpret_cast<uint4*>(sl);
      const bool task = ok && P.task_mode;
      hv[0] = ok ? make_uint4(AGARCL_SNAPSHOT_MAGIC, AGARCL_SNAPSHOT_VERSION, (uint32_t)P.fingerprint, (uint32_t)(P.fingerprint >> 32)) : z;
      hv[1] = ok ? make_uint4((uint32_t)P.S.slot_bytes, (uint32_t)(P.S.slot_bytes >> 32), (uint32_t)(P.instance_base + src),
                              task ? (uint32_t)P.task_mode[src] : 0u) : z;
      hv[2] = task ? make_uint4((uint32_t)P.task_max_steps[src], AGARCL_SNAPSHOT_SIZES_MARKER, (uint32_t)P.sizes.bots[src],
                                (uint32_t)P.sizes.pellets[src]) : z;
      hv[3] = make_uint4(task ? (uint32_t)P.sizes.viruses[src] : 0u, 0u, 0u, 0u);
    }
    return;
  }
  const int i = blockIdx.x;
  const int32_t slot = P.slot_of[i];
  if (slot < 0) {  // not requested: the instance is not touched
    if (t == 0) { P.result[i] = 0; P.restored[i] = 0; }
    return;
  }
  const uint8_t* sl = P.pool + (uint64_t)slot * P.S.slot_bytes;
  bool valid = slot < P.pool_slots;  // (slot_valid, written out: this code predates it and keeps its SASS)
  if (valid) {
    const agarcl_snapshot_hdr* h = reinterpret_cast<const agarcl_snapshot_hdr*>(sl);
    valid = h->magic == AGARCL_SNAPSHOT_MAGIC && h->version == AGARCL_SNAPSHOT_VERSION && h->fingerprint == P.fingerprint &&
            h->slot_bytes == P.S.slot_bytes;
    if (valid && P.task_mode) valid = slot_task_valid(P, h);
  }
  if (!valid) {  // rejected: the instance is not touched
    if (t == 0) { P.result[i] = 2; P.restored[i] = 0; }
    return;
  }
  copy_segment(P.state + (size_t)i * P.stride, sl + P.S.off_blob, P.stride);
  if (P.steps) {
    const uint64_t* ep = reinterpret_cast<const uint64_t*>(sl + P.S.off_ep);
    for (int w = t; w <= A; w += nt) {
      if (w == 0) P.steps[i] = (int64_t)ep[0];
      else P.ret[(size_t)i * A + (w - 1)] = __longlong_as_double((long long)ep[w]);
    }
  }
  if (P.S.ram_bytes) copy_segment(P.ram + (size_t)i * P.S.ram_bytes, sl + P.S.off_ram, P.S.ram_bytes);
  if (P.S.obs_bytes) copy_segment(P.obs + (size_t)i * P.S.obs_bytes, sl + P.S.off_obs, P.S.obs_bytes);
  for (int a = t; a < A; a += nt) {  // like after a reset
    P.rewards[(size_t)i * A + a] = 0.0;
    P.dones[(size_t)i * A + a] = 0;
  }
  if (t == 0) {
    // the next reset of the instance continues the restored draw stream (ResetParams::fresh == 0 -> from hdr.rng_cursor)
    const agarcl_inst_hdr* ih = reinterpret_cast<const agarcl_inst_hdr*>(sl + P.S.off_blob + P.off_hdr);
    P.seeds[i] = (uint64_t)ih->seed_lo | ((uint64_t)ih->seed_hi << 32);
    if (P.task_mode) {  // the slot's task becomes the current one; the pending task is left alone
      const agarcl_snapshot_hdr* h = reinterpret_cast<const agarcl_snapshot_hdr*>(sl);
      take_slot_task(P, h, i, h->task_max_steps);
    }
    P.fresh[i] = 0;
    P.result[i] = 1;
    P.restored[i] = 1;
  }
}

cudaError_t launch_snapshot_save(const SnapParams& P, int n, cudaStream_t stream) {
  k_snapshot<true><<<n, kSnapThreads, 0, stream>>>(P);
  return cudaGetLastError();
}

cudaError_t launch_snapshot_restore(const SnapParams& P, cudaStream_t stream) {
  k_snapshot<false><<<P.N, kSnapThreads, 0, stream>>>(P);
  return cudaGetLastError();
}

cudaError_t launch_snapshot_start(const SnapParams& P, cudaStream_t stream) {
  k_start_states<<<P.N, kSnapThreads, 0, stream>>>(P);
  return cudaGetLastError();
}

}  // namespace ag
