// archive_kernel.cu — the Go-Explore cell archive of a batch (agarcl_batch_set_archive; spec: include/agarcl_b200.h): the cell
// of every instance after a step, the winner of every cell, the entries it creates or improves, the choice of an entry at
// every reset and the trajectory base of the instances that start from one.  Nothing is read back by the host.
//   behind the step:    k_archive_cells (a warp per instance), k_archive_commit (one CTA), then k_snapshot<true> saves the
//                       winners with the (instance, slot) list k_archive_commit wrote (slot -1: not saved)
//   in front of reset:  k_archive_select (one CTA, select = 1) writes the start slots of the reset instances
//   behind k_start_states / a restore: k_archive_base sets the trajectory base of the reset or restored instances
// The winner of a key is decided without sorting: atomicMax of the order-preserving bits of the score, then, among the
// candidates that hold the maximum, atomicMin of (length, instance).  The winners put the per-key scratch back to its neutral
// values, so no pass over the 32 n^2 keys is needed.
#include <cuda_runtime.h>

#include "sim_params.h"

namespace ag {

// f64 -> u64 with the order of the doubles (for all but NaN): the sign bit flipped for positives, every bit for negatives
__device__ __forceinline__ uint64_t ordered_bits(double s) {
  const uint64_t u = (uint64_t)__double_as_longlong(s);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

// One warp per instance: the key of the archive agent's cell, and for a candidate its trajectory score and length, a visit of
// its key and the first round of the winner (the key's best score).
__global__ void __launch_bounds__(256) k_archive_cells(const __grid_constant__ ArchiveParams P) {
  const int i = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (i >= P.N) return;
  const uint8_t* blob = P.state + (size_t)i * P.L.stride;
  const agarcl_player* pl = reinterpret_cast<const agarcl_player*>(blob + P.L.off_players) + P.agent;
  const agarcl_cell* cells = reinterpret_cast<const agarcl_cell*>(blob + P.L.off_cells) + (size_t)P.agent * P.L.cap_cells;
  const int nc = min(max(pl->n_cells, 0), P.L.cap_cells);
  // the centroid of agarcl_batch_draw's agent view: sums in cell order, one rounded fp32 operation each; the lanes form the
  // products and every lane adds them up in order
  float sx = 0.f, sy = 0.f;
  uint32_t m = 0;
  for (int c0 = 0; c0 < nc; c0 += 32) {
    float px = 0.f, py = 0.f;
    uint32_t cm = 0;
    if (c0 + lane < nc) {
      const agarcl_cell& c = cells[c0 + lane];
      cm = c.mass;
      px = __fmul_rn(c.x, (float)cm);
      py = __fmul_rn(c.y, (float)cm);
    }
    const int cnt = min(32, nc - c0);
    for (int k = 0; k < cnt; k++) {
      sx = __fadd_rn(sx, __shfl_sync(AG_FULL, px, k));
      sy = __fadd_rn(sy, __shfl_sync(AG_FULL, py, k));
      m += __shfl_sync(AG_FULL, cm, k);
    }
  }
  if (lane) return;
  int32_t key = -1;
  if (nc > 0 && m > 0) {
    const float fn = (float)P.n;
    const float cx = __fdiv_rn(sx, (float)m), cy = __fdiv_rn(sy, (float)m);
    const int bx = min(max(__float2int_rz(__fdiv_rn(__fmul_rn(cx, fn), P.W)), 0), P.n - 1);
    const int by = min(max(__float2int_rz(__fdiv_rn(__fmul_rn(cy, fn), P.W)), 0), P.n - 1);
    const int mb = 31 - __clz((int)m);
    key = (mb * P.n + by) * P.n + bx;
  }
  P.cell_of[i] = key;
  bool done = false;
  for (int a = 0; a < P.A; a++) done |= P.dones[(size_t)i * P.A + a] != 0;
  int32_t ck = -1;
  if (key >= 0 && !done) {
    const size_t k = (size_t)i * P.A + P.agent;
    const double s = __dadd_rn(P.base_score[i], __dadd_rn(P.ret[k], P.rewards[k]));
    const int64_t l = P.base_length[i] + P.steps[i] + 1;
    P.cand_s[i] = s;
    P.cand_l[i] = l;
    atomicAdd(&P.visits[key], 1u);
    atomicMax(reinterpret_cast<unsigned long long*>(&P.best_s[key]), (unsigned long long)ordered_bits(s));
    ck = key;
  }
  P.cand_key[i] = ck;
}

// Exclusive prefix count of `flag` over the CTA's threads in thread order; *total receives the count of the whole CTA.
// `warp_sums` is shared scratch of blockDim.x / 32 words.  Every thread of the CTA must call it.
__device__ __forceinline__ uint32_t cta_rank(bool flag, uint32_t* warp_sums, uint32_t* total) {
  const int t = threadIdx.x, lane = t & 31, w = t >> 5, nw = blockDim.x >> 5;
  const uint32_t bal = __ballot_sync(AG_FULL, flag);
  __syncthreads();  // (warp_sums of the previous call have been read)
  if (lane == 0) warp_sums[w] = __popc(bal);
  __syncthreads();
  uint32_t before = 0, all = 0;
  for (int k = 0; k < nw; k++) {
    const uint32_t v = warp_sums[k];
    before += k < w ? v : 0u;
    all += v;
  }
  *total = all;
  return before + __popc(bal & ((1u << lane) - 1u));
}

// One CTA: the second round of the winners, then, in instance order, the entries they create or replace, the save list and the
// counters.  Entries created in one step are numbered in ascending order of their winner's instance.
__global__ void __launch_bounds__(kArchiveThreads) k_archive_commit(const __grid_constant__ ArchiveParams P) {
  __shared__ uint32_t warp_sums[kArchiveThreads / 32];
  __shared__ uint32_t s_improved, s_dropped;
  const int t = threadIdx.x;
  if (t == 0) { s_improved = 0; s_dropped = 0; }
  for (int i = t; i < P.N; i += blockDim.x) {
    const int32_t key = P.cand_key[i];
    if (key >= 0 && ordered_bits(P.cand_s[i]) == __ldcg(&P.best_s[key])) {
      const uint64_t l = (uint64_t)min(P.cand_l[i], (int64_t)0xFFFFFFFF);
      atomicMin(reinterpret_cast<unsigned long long*>(&P.best_li[key]), (unsigned long long)(l << 32 | (uint32_t)i));
    }
  }
  __syncthreads();  // (the atomics of the CTA are done: __ldcg below reads them from L2)
  uint64_t used = P.counters[0];
  for (int i0 = 0; i0 < P.N; i0 += blockDim.x) {
    const int i = i0 + t;
    const int32_t key = i < P.N ? P.cand_key[i] : -1;
    const bool win = key >= 0 && (uint32_t)__ldcg(&P.best_li[key]) == (uint32_t)i;
    int32_t e = -1;
    bool fresh = false;
    double s = 0.0;
    int64_t l = 0;
    if (win) {
      s = P.cand_s[i];
      l = P.cand_l[i];
      e = P.key_entry[key];
      if (e < 0) {
        fresh = true;
      } else if (s > P.entry_score[e] || (s == P.entry_score[e] && l < P.entry_length[e])) {
        atomicAdd(&s_improved, 1u);
      } else {
        e = -1;
      }
      P.best_s[key] = 0ull;  // the neutral values of both rounds (a loser reading ~0 does not match its index)
      P.best_li[key] = ~0ull;
    }
    uint32_t n_fresh;
    const uint32_t rank = cta_rank(fresh, warp_sums, &n_fresh);
    if (fresh) {
      if (used + rank < (uint64_t)P.K) {
        e = (int32_t)(used + rank);
        P.key_entry[key] = e;
        P.entry_key[e] = key;
      } else {
        atomicAdd(&s_dropped, 1u);
      }
    }
    used = min(used + n_fresh, (uint64_t)P.K);
    if (e >= 0) {
      P.entry_score[e] = s;
      P.entry_length[e] = l;
    }
    if (i < P.N) P.save_slot[i] = e;
  }
  __syncthreads();
  if (t == 0) {
    P.counters[0] = used;
    P.counters[1] += s_dropped;
    P.counters[2] += s_improved;
  }
}

// One CTA, in front of k_start_states (select = 1): every reset instance draws an entry with weight
// floor(2^20 / (1 + isqrt(chosen))) and takes its slot as start slot (-1 with an empty archive); then the counts grow.
__global__ void __launch_bounds__(kArchiveThreads) k_archive_select(const __grid_constant__ ArchiveParams P) {
  __shared__ uint32_t warp_sums[kArchiveThreads / 32];
  const int t = threadIdx.x;
  bool any = false;
  for (int i = t; i < P.N; i += blockDim.x) any |= !P.mask || P.mask[i];
  if (!__syncthreads_or(any)) return;  // (most steps: nothing resets)
  const uint32_t used = (uint32_t)P.counters[0];
  // inclusive prefix sums of the weights, in chunks of the CTA's threads (a chunk's sum fits 32 bits: 1024 * 2^20)
  uint64_t carry = 0;
  for (uint32_t e0 = 0; e0 < used; e0 += blockDim.x) {
    const uint32_t e = e0 + t;
    const uint32_t w = e < used ? (1u << 20) / (1u + (uint32_t)__dsqrt_rn((double)P.entry_chosen[e])) : 0u;
    // warp inclusive scan, then the warps' totals
    uint32_t v = w;
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t o = __shfl_up_sync(AG_FULL, v, d);
      if ((t & 31) >= d) v += o;
    }
    __syncthreads();
    if ((t & 31) == 31) warp_sums[t >> 5] = v;
    __syncthreads();
    uint32_t before = 0, all = 0;
    for (int k = 0; k < (int)(blockDim.x >> 5); k++) {
      const uint32_t x = warp_sums[k];
      before += k < (t >> 5) ? x : 0u;
      all += x;
    }
    if (e < used) P.prefix[e] = carry + before + v;
    carry += all;
  }
  __syncthreads();  // (the prefix sums and the counts are read below; the counts grow after every pick is made)
  const uint64_t W = carry;
  for (int i = t; i < P.N; i += blockDim.x) {
    if (P.mask && !P.mask[i]) continue;
    if (used == 0) {
      P.start_slot[i] = -1;
      continue;
    }
    const uint32_t c = P.draws[i];
    const uint4 r = philox4x32_10(make_uint4(c, 0x41524348u, (uint32_t)(P.instance_base + i), 0u),
                                  make_uint2((uint32_t)P.seed, (uint32_t)(P.seed >> 32)));
    const uint64_t x = ((uint64_t)r.y << 32 | r.x) % W;
    uint32_t lo = 0, hi = used - 1;  // the first entry whose inclusive prefix sum exceeds x
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      if (P.prefix[mid] > x) hi = mid; else lo = mid + 1;
    }
    P.start_slot[i] = (int32_t)lo;
    P.draws[i] = c + 1;
  }
  __syncthreads();
  for (int i = t; i < P.N; i += blockDim.x)
    if ((!P.mask || P.mask[i]) && used) atomicAdd(&P.entry_chosen[P.start_slot[i]], 1u);
}

// One thread per instance in `mask` (nullptr: all): the trajectory base.  An instance started from an archive slot (start
// result 1, P.start_result set when the start table is the archive's pool) takes the entry's score and length; every other
// one (spawned, rejected, restored) starts at (0, 0).
__global__ void __launch_bounds__(256) k_archive_base(const __grid_constant__ ArchiveParams P) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.N || (P.mask && !P.mask[i])) return;
  double s = 0.0;
  int64_t l = 0;
  if (P.start_result && P.start_result[i] == 1) {
    const int32_t e = P.start_slot[i];
    if (e >= 0 && (uint64_t)e < P.counters[0]) {
      s = P.entry_score[e];
      l = P.entry_length[e];
    }
  }
  P.base_score[i] = s;
  P.base_length[i] = l;
}

cudaError_t launch_archive_update(const ArchiveParams& P, cudaStream_t stream) {
  k_archive_cells<<<(P.N + 7) / 8, 256, 0, stream>>>(P);
  k_archive_commit<<<1, kArchiveThreads, 0, stream>>>(P);
  return cudaGetLastError();
}

cudaError_t launch_archive_select(const ArchiveParams& P, cudaStream_t stream) {
  k_archive_select<<<1, kArchiveThreads, 0, stream>>>(P);
  return cudaGetLastError();
}

cudaError_t launch_archive_base(const ArchiveParams& P, cudaStream_t stream) {
  k_archive_base<<<(P.N + 255) / 256, 256, 0, stream>>>(P);
  return cudaGetLastError();
}

}  // namespace ag
