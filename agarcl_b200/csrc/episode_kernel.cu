// episode_kernel.cu — what a vector environment with auto-reset does around the step, on the device: the episode
// bookkeeping of agarcl_batch_step_autoreset (done flags with the step limit folded in, the reset mask, step counters,
// returns), the pending tasks of a mixed-task batch (agarcl_batch_set_tasks) and the masked per-instance byte copy / clear used by a masked reset and by the final-observation copy.
// Neither needs the host to look at the step's dones, so the step, the bookkeeping and the reset queue back to back.
#include <cuda_runtime.h>

#include "block_copy.cuh"
#include "sim_params.h"

namespace ag {

// One thread per instance.
//   clear == 0, after a step: done_out = dones | (max_steps > 0 && steps >= max_steps), checked before the increment like
//     gym_agario's AgarioEnv.step; steps += 1; ret += rewards.  With `reset`, an instance with any done agent gets
//     reset_mask = 1, its return and length go to final_ret / final_len, and its steps and ret restart at 0.  Must run
//     before k_reset, which zeroes the dones of the instances it resets.
//   clear == 1, a reset of the instances in clear_mask (nullptr: all): their steps and ret restart at 0.
__global__ void __launch_bounds__(256) k_episode(const __grid_constant__ EpisodeParams P) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.N) return;
  const int A = P.A;
  if (P.clear) {
    if (P.clear_mask && !P.clear_mask[i]) return;
    P.steps[i] = 0;
    for (int a = 0; a < A; a++) P.ret[(size_t)i * A + a] = 0.0;
    return;
  }
  int64_t s = P.steps[i];
  int32_t max_steps = P.max_steps;
  if (P.task_max_steps && P.task_max_steps[i] >= 0) max_steps = P.task_max_steps[i];  // (-1: the batch's limit)
  const bool limit = max_steps > 0 && s >= (int64_t)max_steps;
  bool any = false;
  for (int a = 0; a < A; a++) {
    const size_t k = (size_t)i * A + a;
    const bool d = P.dones[k] != 0 || limit;
    P.done_out[k] = d ? 1 : 0;
    any |= d;
  }
  s += 1;
  const bool reset = P.reset && any;
  for (int a = 0; a < A; a++) {
    const size_t k = (size_t)i * A + a;
    const double r = P.ret[k] + P.rewards[k];
    if (reset) P.final_ret[k] = r;
    P.ret[k] = reset ? 0.0 : r;
  }
  if (reset) P.final_len[i] = s;
  P.steps[i] = reset ? 0 : s;
  P.reset_mask[i] = reset ? 1 : 0;
}

// One thread per instance: agarcl_batch_set_tasks.  A rejected entry leaves the instance's pending task as it is.
__global__ void __launch_bounds__(256) k_set_tasks(const __grid_constant__ SetTasksParams P) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.N) return;
  const int32_t m = P.mode[i];
  const bool set_mode = m != -1, set_limit = P.max_steps != nullptr;
  const int32_t ms = set_limit ? P.max_steps[i] : -1;
  const bool bad_mode = set_mode && (m < 0 || m > 10 || !((P.task_modes >> m) & 1));
  if (bad_mode || ms < -1) { P.result[i] = 2; return; }
  if (set_mode) P.next_mode[i] = m;
  if (set_limit) P.next_max_steps[i] = ms;
  P.result[i] = (set_mode || set_limit) ? 1 : 0;
}

// One thread per instance: agarcl_batch_set_task_sizes.  The entries given (not -1, array not nullptr) replace the pending sizes
// only when the resulting sizes are all valid; a rejected instance keeps all three.
__global__ void __launch_bounds__(256) k_set_task_sizes(const __grid_constant__ SetTaskSizesParams P) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.N) return;
  const int32_t b = P.bots ? P.bots[i] : -1, p = P.pellets ? P.pellets[i] : -1, v = P.viruses ? P.viruses[i] : -1;
  if (b == -1 && p == -1 && v == -1) { P.result[i] = 0; return; }
  const int32_t nb = b == -1 ? P.next_bots[i] : b, np = p == -1 ? P.next_pellets[i] : p, nv = v == -1 ? P.next_viruses[i] : v;
  if (!sizes_allowed(P.lim, nb, np, nv)) { P.result[i] = 2; return; }
  P.next_bots[i] = nb;
  P.next_pellets[i] = np;
  P.next_viruses[i] = nv;
  P.result[i] = 1;
}

// One CTA per instance: bytes [i * per, (i + 1) * per) of dst get those of src (kCopy) or zeros, for the instances with
// mask[i] != 0; the CTAs of the others exit at once.  dst and src are allocations of the same alignment, so the slices
// of one instance share their alignment modulo 16 (block_copy).
template <bool kCopy>
__global__ void __launch_bounds__(kMaskedThreads) k_masked_bytes(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src,
                                                                 size_t per, const uint8_t* __restrict__ mask) {
  const int inst = blockIdx.x;
  if (!mask[inst]) return;
  block_copy<kCopy>(dst + (size_t)inst * per, kCopy ? src + (size_t)inst * per : nullptr, per);
}

cudaError_t launch_episode(const EpisodeParams& P, cudaStream_t stream) {
  k_episode<<<(P.N + 255) / 256, 256, 0, stream>>>(P);
  return cudaGetLastError();
}

cudaError_t launch_set_tasks(const SetTasksParams& P, cudaStream_t stream) {
  k_set_tasks<<<(P.N + 255) / 256, 256, 0, stream>>>(P);
  return cudaGetLastError();
}

cudaError_t launch_set_task_sizes(const SetTaskSizesParams& P, cudaStream_t stream) {
  k_set_task_sizes<<<(P.N + 255) / 256, 256, 0, stream>>>(P);
  return cudaGetLastError();
}

cudaError_t launch_masked_bytes(void* dst, const void* src, size_t per, const uint8_t* mask, int N, cudaStream_t stream) {
  if (src) k_masked_bytes<true><<<N, kMaskedThreads, 0, stream>>>((uint8_t*)dst, (const uint8_t*)src, per, mask);
  else k_masked_bytes<false><<<N, kMaskedThreads, 0, stream>>>((uint8_t*)dst, nullptr, per, mask);
  return cudaGetLastError();
}

}  // namespace ag
