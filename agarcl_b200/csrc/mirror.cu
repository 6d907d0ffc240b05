// mirror.cu — host-resident observation mirror: the reference-facing hand-off of GridObservation frames to
// HOST memory (get_state, environment/bindings.cpp:67-91, copies 512 KB per agent per step) without moving
// the dense tensor over PCIe.
//
// A grid observation is almost entirely structure: channel 0 of every frame is the out-of-bounds mask, which
// is the union of whole rows and whole columns (GridObservation::_mark_out_of_bounds,
// environment/envs/GridEnvironment.hpp:235-248: a grid point is marked iff its x or its y leaves the arena),
// and the other channels hold a few hundred non-zero elements (one per in-view entity,
// _store_entities :212-232).  So per step
//   1. the device produces, per image, the row/column bit masks of every mask channel and the (offset, value)
//      list of all other non-zeros, grouped into chunks of consecutive images (PackOut, sim_params.h):
//      - agarcl_batch_step_mirror: the fused observation finish of k_step lists what it scatters while it
//        scatters it (sim_kernel.cu, obs_finish_warp) -- the dense tensor is never read back;
//      - agarcl_batch_sync_mirror (after a reset / render, or a configuration k_step does not finish itself):
//        k_pack, one CTA per image, reads the dense device observation once;
//   2. every finished chunk (a few hundred KB instead of 2.1 GB at configs[1]) is copied to pinned host memory
//      by ONE copy -- in the fused path as soon as the kernel flags the chunk in host-mapped memory, while it is
//      still stepping the instances of the next chunks;
//   3. a pool of host threads brings the library-owned dense mirror [N*A, frames*C, G, G] up to date in place,
//      chunk by chunk as they arrive: zero the previous step's entries, rewrite only the mask rows/columns that
//      changed, store the new entries.
// An image that does not fit the scheme (entry capacity exceeded, or a mask channel that is not a row/column
// union) is copied densely instead, so the mirror is ALWAYS identical to the device tensor — the parity test
// tests/test_gpu_mirror.py compares them element for element after every step.
#include "mirror.h"

#include <sys/mman.h>

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

#include "host_util.h"

namespace ag {

constexpr int kPackThreads = 256;

struct PackParams {
  const void* obs;
  int32_t CH, C, G;
  uint32_t cap_img;  // entries staged in shared memory per image
  PackOut pk;
};

template <typename T> struct Vec;
template <> struct Vec<int32_t> {
  static constexpr int kN = 4;
  static __device__ __forceinline__ void unpack(const int4& q, int (&e)[4]) { e[0] = q.x; e[1] = q.y; e[2] = q.z; e[3] = q.w; }
};
template <> struct Vec<int16_t> {
  static constexpr int kN = 8;
  static __device__ __forceinline__ void unpack(const int4& q, int (&e)[8]) {
    const int w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int k = 0; k < 4; k++) {
      e[2 * k] = (int)(int16_t)(w[k] & 0xFFFF);
      e[2 * k + 1] = w[k] >> 16;
    }
  }
};

// One CTA per agent image.  HBM-bound: reads every element of the dense observation exactly once from DRAM
// (the mask channels a second time from L2); algorithmic bytes = sizeof(obs) in, lists out.
template <typename T>
__global__ void __launch_bounds__(kPackThreads) k_pack(const PackParams P) {
  constexpr int VE = Vec<T>::kN;
  extern __shared__ __align__(16) uint8_t smem[];
  uint2* s_ent = reinterpret_cast<uint2*>(smem);
  uint8_t* row_any = smem + (size_t)P.cap_img * sizeof(uint2);  // row i holds an in-bounds (zero) element
  uint8_t* col_any = row_any + P.G;
  __shared__ uint32_t s_cnt, s_bad, s_base;
  const uint32_t tid = threadIdx.x, img = blockIdx.x;
  const uint32_t G = (uint32_t)P.G, plane = G * G, pv = plane / VE;
  const uint32_t MW = (uint32_t)P.pk.MW;
  const uint32_t chunk = img / P.pk.ipc, li = img - chunk * P.pk.ipc;
  uint32_t* blk = P.pk.chunks + (size_t)chunk * P.pk.chunk_words;
  const T* base = reinterpret_cast<const T*>(P.obs) + (size_t)img * P.CH * plane;
  if (tid == 0) { s_cnt = 0; s_bad = 0; }
  for (uint32_t i = tid; i < 2 * G; i += kPackThreads) row_any[i] = 0;
  __syncthreads();
  const int frames = P.CH / P.C;
  for (int f = 0; f < frames; f++) {
    const int4* p = reinterpret_cast<const int4*>(base + (size_t)f * P.C * plane);
    for (uint32_t v = tid; v < pv; v += kPackThreads) {
      int e[VE];
      Vec<T>::unpack(__ldg(p + v), e);
#pragma unroll
      for (int k = 0; k < VE; k++)
        if (e[k] == 0) {
          const uint32_t idx = v * VE + k;
          row_any[idx / G] = 1;
          col_any[idx % G] = 1;
        }
    }
    __syncthreads();
    bool bad = false;
    for (uint32_t v = tid; v < pv; v += kPackThreads) {
      int e[VE];
      Vec<T>::unpack(__ldg(p + v), e);
#pragma unroll
      for (int k = 0; k < VE; k++) {
        const uint32_t idx = v * VE + k;
        const int expect = (row_any[idx / G] & col_any[idx % G]) ? 0 : -1;
        bad |= (e[k] != expect);
      }
    }
    if (bad) s_bad = 1;
    uint32_t* mk = blk + pk_off_rec(P.pk) + (size_t)li * P.pk.rec_words + 3 + (size_t)f * 2 * MW;
    for (uint32_t w = tid; w < 2u * MW; w += kPackThreads) {
      const uint8_t* any = w < MW ? row_any : col_any;
      const uint32_t w0 = (w % MW) * 32;
      uint32_t bits = 0;
      for (uint32_t b = 0; b < 32 && w0 + b < G; b++)
        if (!any[w0 + b]) bits |= 1u << b;
      mk[w] = bits;
    }
    __syncthreads();
    for (uint32_t i = tid; i < 2 * G; i += kPackThreads) row_any[i] = 0;
    __syncthreads();
  }
  // every other channel: non-zero elements are rare, four 16-byte loads in flight per thread
  for (int c = 0; c < P.CH; c++) {
    if (c % P.C == 0) continue;
    const int4* p = reinterpret_cast<const int4*>(base + (size_t)c * plane);
    for (uint32_t v0 = tid; v0 < pv; v0 += 4 * kPackThreads) {
      int4 q[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const uint32_t v = v0 + u * kPackThreads;
        q[u] = v < pv ? __ldcs(p + v) : make_int4(0, 0, 0, 0);
      }
#pragma unroll
      for (int u = 0; u < 4; u++) {
        if ((q[u].x | q[u].y | q[u].z | q[u].w) == 0) continue;
        int e[VE];
        Vec<T>::unpack(q[u], e);
#pragma unroll
        for (int k = 0; k < VE; k++)
          if (e[k] != 0) {
            const uint32_t slot = atomicAdd(&s_cnt, 1u);
            if (slot < P.cap_img) s_ent[slot] = make_uint2((uint32_t)c * plane + (v0 + u * kPackThreads) * VE + k, (uint32_t)e[k]);
          }
      }
    }
  }
  __syncthreads();
  if (tid == 0) {
    uint32_t cnt = s_cnt, b0 = 0;
    if (s_bad || cnt > P.cap_img) cnt = kPackDense;
    else if (cnt) {
      b0 = atomicAdd(P.pk.cursor + chunk, cnt);
      if (b0 + cnt > P.pk.cap_chunk) cnt = kPackDense;
    }
    uint32_t* rec = blk + pk_off_rec(P.pk) + (size_t)li * P.pk.rec_words;
    rec[0] = cnt;
    rec[1] = b0;
    rec[2] = img;  // slot = image on this path
    s_cnt = cnt;
    s_base = b0;
  }
  __syncthreads();
  const uint32_t cnt = s_cnt;
  if (cnt != kPackDense) {
    uint2* ent = reinterpret_cast<uint2*>(blk + pk_off_entries(P.pk));
    for (uint32_t k = tid; k < cnt; k += kPackThreads) ent[s_base + k] = s_ent[k];
  }
  // the CTA that finishes the last image of the chunk publishes the entry count and rewinds the counters
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    const uint32_t in_chunk = min(P.pk.ipc, P.pk.n_img - chunk * P.pk.ipc);
    if (atomicAdd(P.pk.done + chunk, 1u) + 1u == in_chunk) {
      __threadfence();
      blk[0] = atomicExch(P.pk.cursor + chunk, 0u);
      P.pk.done[chunk] = 0u;
      if (P.pk.flags) {
        __threadfence_system();
        P.pk.flags[chunk] = P.pk.seq;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ host pool
static inline void cpu_relax() {
#if defined(__x86_64__) || defined(__i386__)
  __builtin_ia32_pause();
#else
  std::this_thread::yield();
#endif
}

// Every worker (and, from join() on, the caller) runs the same job, which pulls work from atomic counters.
// Workers sleep on a condition variable between jobs; the END of a job is awaited by spinning on an atomic
// (a futex wake-up of the caller would add tens of microseconds to every step).
class Pool {
 public:
  explicit Pool(int workers) {
    for (int i = 0; i < workers; i++) th_.emplace_back([this] { loop(); });
  }
  ~Pool() {
    {
      std::lock_guard<std::mutex> g(mu_);
      stop_ = true;
    }
    cv_start_.notify_all();
    for (auto& t : th_) t.join();
  }
  int threads() const { return (int)th_.size() + 1; }
  void start(const std::function<void()>& job) {  // wakes the workers; the job object must live until join() returns
    {
      std::lock_guard<std::mutex> g(mu_);
      job_ = &job;
      pending_.store((int)th_.size(), std::memory_order_relaxed);
      gen_++;
    }
    cv_start_.notify_all();
  }
  void join() {  // the caller works too, then waits for the workers
    (*job_)();
    while (pending_.load(std::memory_order_acquire) != 0) cpu_relax();
    job_ = nullptr;
  }
  void run(const std::function<void()>& job) {
    start(job);
    join();
  }

 private:
  void loop() {
    uint64_t seen = 0;
    for (;;) {
      const std::function<void()>* job;
      {
        std::unique_lock<std::mutex> g(mu_);
        cv_start_.wait(g, [&] { return stop_ || gen_ != seen; });
        if (stop_) return;
        seen = gen_;
        job = job_;
      }
      (*job)();
      pending_.fetch_sub(1, std::memory_order_release);
    }
  }
  std::vector<std::thread> th_;
  std::mutex mu_;
  std::condition_variable cv_start_;
  const std::function<void()>* job_ = nullptr;
  uint64_t gen_ = 0;
  std::atomic<int> pending_{0};
  bool stop_ = false;
};

struct HostMirror {
  int n_img = 0, CH = 0, C = 0, G = 0, frames = 0, MW = 0, dtype = 0;
  size_t esz = 4, img_elems = 0, img_bytes = 0;
  uint32_t cap_img = 0;
  int n_chunks = 1;
  PackOut pk{};                   // device side of the chunk blocks (flags / seq filled per use)
  size_t meta_words = 0;          // words of a chunk block in front of its entries
  void* h_obs = nullptr;          // pinned [n_img][CH][G][G]
  bool obs_malloced = false, obs_registered = false;
  uint32_t* d_chunks = nullptr;
  uint32_t* d_counters = nullptr; // [2][n_chunks] cursor, done
  uint32_t* h_chunks[2] = {nullptr, nullptr};  // pinned + host-mapped, same block layout; [cur] = this step's lists, [cur^1] = the previous step's
  uint32_t* dh_chunks[2] = {nullptr, nullptr}; // their device addresses (k_step writes its lists straight into them)
  float* h_dxdy = nullptr;                     // host-mapped action staging [n_img][2], [n_img]: k_step reads the step's
  int32_t* h_act = nullptr;                    // actions straight from host memory
  float* d_dxdy = nullptr;
  int32_t* d_act = nullptr;
  volatile uint32_t* h_flags = nullptr;        // host-mapped [n_chunks]
  uint32_t* d_flags = nullptr;                 // its device address
  uint32_t seq = 0;
  int cur = 0;
  std::vector<uint32_t> slot_of[2];  // per staging buffer: the slot that describes image i
  std::vector<size_t> guess;      // per chunk: entries fetched together with the meta words (the remainder, if any, in a second copy)
  Pool* pool = nullptr;
  bool lists_only = false;        // no dense mirror: the lists themselves are the product (agarcl_batch_step_lists)
  MirrorStats stats{};
  uint32_t* blk(int w, int chunk) const { return h_chunks[w] + (size_t)chunk * pk.chunk_words; }
  // the record of list slot `slot` in staging buffer `w`, and the entries it counts
  const uint32_t* rec(int w, uint32_t slot) const { return blk(w, (int)(slot / pk.ipc)) + pk_off_rec(pk) + (size_t)(slot % pk.ipc) * pk.rec_words; }
  const uint2* entries(int w, uint32_t slot) const {
    return reinterpret_cast<const uint2*>(blk(w, (int)(slot / pk.ipc)) + pk_off_entries(pk)) + rec(w, slot)[1];
  }
};

static inline bool bit(const uint32_t* m, int i) { return (m[i >> 5] >> (i & 31)) & 1u; }

// Channel 0 of one frame: element (i, j) is -1 iff row i or column j is out of bounds.
template <typename T>
static void apply_mask_delta(T* p, const uint32_t* om, const uint32_t* nm, int G, int MW) {
  const uint32_t *orow = om, *ocol = om + MW, *nrow = nm, *ncol = nm + MW;
  const bool col_changed = std::memcmp(ocol, ncol, (size_t)MW * 4) != 0;
  for (int i = 0; i < G; i++) {
    const bool ro = bit(orow, i), rn = bit(nrow, i);
    T* r = p + (size_t)i * G;
    if (rn) {
      if (!ro) std::memset(r, 0xFF, (size_t)G * sizeof(T));
      continue;
    }
    if (ro) {
      for (int j = 0; j < G; j++) r[j] = bit(ncol, j) ? (T)-1 : (T)0;
      continue;
    }
    if (col_changed)
      for (int w = 0; w < MW; w++)
        for (uint32_t d = ocol[w] ^ ncol[w]; d; d &= d - 1) {
          const int j = w * 32 + __builtin_ctz(d);
          r[j] = bit(ncol, j) ? (T)-1 : (T)0;
        }
  }
}

// Replays one image's lists over its dense frames `p`, which hold the previous step's masks and no entries: the mask delta of
// every frame from `om` (the previous masks; nullptr: nothing out of bounds), then the entries.  The library's one replay of
// the list format: it must stay bit-identical to batch.py ObsLists.decode.  Forced inline: the mirror's host threads spend
// their time in this loop.
static const uint32_t kZeroMasks[2 * 128] = {};  // (G <= 4096, mirror_create)
template <typename T>
static __forceinline__ void replay_image(const HostMirror* m, T* p, const uint32_t* om, const uint32_t* nm, const uint2* ne, uint32_t n) {
  const size_t mw2 = 2 * (size_t)m->MW, plane = (size_t)m->G * m->G;
  for (int f = 0; f < m->frames; f++) {
    const uint32_t* o = om ? om + f * mw2 : kZeroMasks;
    if (std::memcmp(o, nm + f * mw2, mw2 * 4) != 0) apply_mask_delta<T>(p + (size_t)f * m->C * plane, o, nm + f * mw2, m->G, m->MW);
  }
  // (operands are masses / counts >= 0; the 16-bit dtype saturates exactly like the device's updates, sim_kernel.cu FinOps<int16_t>)
  constexpr int32_t kTop = sizeof(T) == 2 ? 32767 : 2147483647;
  for (uint32_t e = 0; e < n; e++) {
    T& x = p[ne[e].x & kPkOffMask];
    const int32_t v32 = (int32_t)ne[e].y;
    const T v = (T)(v32 > kTop ? kTop : v32);
    switch (ne[e].x >> 29) {
      case kPkSet: x = v; break;
      case kPkAdd: { const int64_t t = (int64_t)x + v32; x = (T)(t > kTop ? kTop : t); break; }
      case kPkMinNz: x = (x != 0 && x < v) ? x : v; break;
      default: x = x > v ? x : v; break;
    }
  }
}

// The elements an image's two lists touch are scattered over its 512 KB: ask for their cache lines (for writing)
// one slot ahead, so that the misses of the next image overlap the read-modify-writes of this one.
template <typename T>
static void prefetch_slot(const HostMirror* m, int slot) {
  const int cur = m->cur, prev = cur ^ 1;
  const uint32_t* crec = m->rec(cur, (uint32_t)slot);
  const uint32_t img = crec[2];
  if (img >= (uint32_t)m->n_img) return;
  const T* p = reinterpret_cast<const T*>(m->h_obs) + (size_t)img * m->img_elems;
  if (crec[0] != kPackDense) {
    const uint2* e = m->entries(cur, (uint32_t)slot);
    for (uint32_t i = 0; i < crec[0]; i++) __builtin_prefetch(p + (e[i].x & kPkOffMask), 1, 1);
  }
  const uint32_t ps = m->slot_of[prev][img];
  const uint32_t* prec = m->rec(prev, ps);
  if (prec[0] != kPackDense) {
    const uint2* e = m->entries(prev, ps);
    for (uint32_t i = 0; i < prec[0]; i++) __builtin_prefetch(p + (e[i].x & kPkOffMask), 1, 1);
  }
}

// Slots [lo, hi) of the current lists: every slot names its image; the image's previous lists are found through slot_of.
template <typename T>
static void expand_range(HostMirror* m, int lo, int hi) {
  const int cur = m->cur, prev = cur ^ 1;
  static const int ahead = [] { const char* e = std::getenv("AGARCL_MIRROR_PREFETCH"); return e ? std::atoi(e) : 1; }();
  for (int a = 0; a < ahead && lo + a < hi; a++) prefetch_slot<T>(m, lo + a);
  for (int slot = lo; slot < hi; slot++) {
    if (slot + ahead < hi) prefetch_slot<T>(m, slot + ahead);
    const uint32_t* crec = m->rec(cur, (uint32_t)slot);
    const uint32_t img = crec[2];
    if (img >= (uint32_t)m->n_img) continue;  // (cannot happen with lists the kernels wrote)
    const uint32_t cnt = crec[0];
    if (cnt == kPackDense) continue;  // the dense copy of this image is made by the calling thread
    const uint32_t ps = m->slot_of[prev][img];
    const uint32_t* prec = m->rec(prev, ps);
    T* p = reinterpret_cast<T*>(m->h_obs) + (size_t)img * m->img_elems;
    const uint32_t pcnt = prec[0];
    if (pcnt == kPackDense) {
      std::memset(p, 0, m->img_bytes);
    } else {
      const uint2* pe = m->entries(prev, ps);
      for (uint32_t e = 0; e < pcnt; e++) p[pe[e].x & kPkOffMask] = 0;
    }
    replay_image<T>(m, p, pcnt == kPackDense ? nullptr : prec + 3, crec + 3, m->entries(cur, (uint32_t)slot), cnt);
  }
}

// The records of chunk `c` of this step's lists: checks the image each names and points slot_of at its slot, adds the chunk's
// entries to *entries and its dense images to *dense, and copies the step's reward and done flag out of the records (k_step
// writes them there; rewards_out / dones_out may be null).
static int read_records(HostMirror* m, int c, uint64_t* entries, std::vector<int>* dense, double* rewards_out, uint8_t* dones_out) {
  const PackOut& k = m->pk;
  const int lo = c * (int)k.ipc, hi = lo + (int)k.ipc < m->n_img ? lo + (int)k.ipc : m->n_img;
  for (int i = lo; i < hi; i++) {
    const uint32_t* rec = m->rec(m->cur, (uint32_t)i);
    const uint32_t img = rec[2];
    if (img >= (uint32_t)m->n_img) return agarcl_set_error(AGARCL_ERR_STATE, "list slot %d names image %u of %d", i, img, m->n_img);
    m->slot_of[m->cur][img] = (uint32_t)i;
    if (rec[0] == kPackDense) dense->push_back((int)img);
    else *entries += rec[0];
    if (rewards_out) std::memcpy(rewards_out + img, rec + k.rec_words - 3, sizeof(double));
    if (dones_out) dones_out[img] = (uint8_t)rec[k.rec_words - 1];
  }
  return AGARCL_OK;
}

// What k_step writes over PCIe for one step's lists: every record, every chunk flag and the entries.
static uint64_t lists_d2h_bytes(const HostMirror* m, uint64_t entries) {
  return (uint64_t)m->n_img * m->pk.rec_words * 4 + (uint64_t)m->n_chunks * 4 + entries * 8;
}

// Waits for the kernel launched on `s` with mirror_pack_out() to flag every chunk of this step in host-mapped memory, and calls
// on_chunk(c) for each as its flag arrives (in any order); an error on_chunk returns ends the wait.  Between polls the thread
// runs idle(), which returns whether it did a piece of other work (counted as 64 spins, a pause as one).  Every `query_spins`
// spins the stream is queried, so that a failed launch cannot hang the caller.
template <typename OnChunk, typename Idle>
static int wait_chunks(HostMirror* m, cudaStream_t s, uint32_t query_spins, OnChunk&& on_chunk, Idle&& idle) {
  const int K = m->n_chunks;
  std::vector<uint8_t> seen((size_t)K, 0);
  int left = K;
  bool finished = false;  // the stream is complete: a chunk not flagged at the next poll never will be
  for (uint32_t spins = 0; left > 0;) {
    bool any = false;
    for (int c = 0; c < K; c++)
      if (!seen[(size_t)c] && m->h_flags[c] == m->seq) {
        seen[(size_t)c] = 1; left--; any = true;
        if (const int rc = on_chunk(c)) return rc;
      }
    if (any) continue;
    if (finished) return agarcl_set_error(AGARCL_ERR_STATE, "step kernel finished without completing every list chunk");
    if (idle()) spins += 64u;
    else { cpu_relax(); spins += 1u; }
    if (spins >= query_spins) {
      spins = 0u;
      const cudaError_t q = cudaStreamQuery(s);
      if (q == cudaSuccess) finished = true;
      else if (q != cudaErrorNotReady) return agarcl_set_error(AGARCL_ERR_CUDA, "cudaStreamQuery failed: %s", cudaGetErrorString(q));
    }
  }
  return AGARCL_OK;
}

// ---- the lists as the observation (agarcl_batch_step_lists): wait for every chunk flag of the launch that was handed
// mirror_pack_out(); nothing is expanded.  rewards / dones come from the records.
int mirror_collect_lists(HostMirror* m, cudaStream_t s, double* rewards_out, uint8_t* dones_out) {
  m->cur ^= 1;
  uint64_t entries = 0;
  std::vector<int> dense;
  const int rc = wait_chunks(m, s, 4096u, [&](int c) { return read_records(m, c, &entries, &dense, rewards_out, dones_out); },
                             [] { return false; });
  if (rc) return rc;
  m->stats.entries = entries;
  m->stats.dense_images = dense.size();
  m->stats.d2h_bytes = lists_d2h_bytes(m, entries);
  return AGARCL_OK;
}

void mirror_lists_view(const HostMirror* m, agarcl_obs_lists* out) {
  const PackOut& k = m->pk;
  out->n_images = m->n_img; out->n_chunks = m->n_chunks; out->images_per_chunk = (int32_t)k.ipc;
  out->frames = m->frames; out->channels = m->C; out->grid = m->G; out->obs_dtype = m->dtype;
  out->mask_words = m->MW; out->rec_words = (int32_t)k.rec_words; out->entries_per_image = (int32_t)k.slot;
  out->off_rec = pk_off_rec(k); out->off_entries = pk_off_entries(k); out->chunk_words = k.chunk_words;
  out->chunks = m->h_chunks[m->cur];
  out->slot_of = m->slot_of[m->cur].data();
}

// Decodes image `img` of the current lists into a dense [CH][G][G] frame of the mirror's dtype.  Returns 1 when the image did
// not fit its slot (the caller takes it from the device tensor), 0 otherwise.
template <typename T>
static int lists_expand_t(const HostMirror* m, int img, T* p) {
  const uint32_t slot = m->slot_of[m->cur][(size_t)img];
  const uint32_t* rec = m->rec(m->cur, slot);
  if (rec[0] == kPackDense) return 1;
  std::memset(p, 0, m->img_bytes);
  replay_image<T>(m, p, nullptr, rec + 3, m->entries(m->cur, slot), rec[0]);
  return 0;
}
int mirror_lists_expand(const HostMirror* m, int img, void* dense_out) {
  return m->dtype == AGARCL_OBS_I16 ? lists_expand_t<int16_t>(m, img, static_cast<int16_t*>(dense_out))
                                    : lists_expand_t<int32_t>(m, img, static_cast<int32_t*>(dense_out));
}

void mirror_destroy(HostMirror* m) {
  if (!m) return;
  delete m->pool;
  cudaFree(m->d_chunks);
  cudaFree(m->d_counters);
  for (int w = 0; w < 2; w++) cudaFreeHost(m->h_chunks[w]);
  cudaFreeHost((void*)m->h_flags);
  cudaFreeHost(m->h_dxdy);
  cudaFreeHost(m->h_act);
  if (m->obs_malloced) {
    if (m->obs_registered) cudaHostUnregister(m->h_obs);
    std::free(m->h_obs);
  } else {
    cudaFreeHost(m->h_obs);
  }
  delete m;
}

HostMirror* mirror_create(int n_img, int agents, int CH, int C, int G, int dtype, bool lists_only) {
  const size_t esz = dtype == AGARCL_OBS_I16 ? 2 : 4;
  if (((size_t)G * G * esz) % 16 != 0 || G > 4096 || (uint64_t)CH * G * G > kPkOffMask) {
    agarcl_set_error(AGARCL_ERR_INVALID, "the host mirror needs grid planes that are multiples of 16 bytes (grid_size %d)", G);
    return nullptr;
  }
  HostMirror* m = new (std::nothrow) HostMirror();
  if (!m) {
    agarcl_set_error(AGARCL_ERR_NOMEM, "out of host memory");
    return nullptr;
  }
  m->n_img = n_img; m->CH = CH; m->C = C; m->G = G; m->frames = CH / C; m->MW = (G + 31) / 32; m->dtype = dtype;
  m->esz = esz;
  m->img_elems = (size_t)CH * G * G;
  m->img_bytes = m->img_elems * esz;
  m->cap_img = 2048;
  if (const char* e = std::getenv("AGARCL_MIRROR_CAP_IMG")) m->cap_img = (uint32_t)std::atoi(e);
  // chunks: whole instances, about 32 per batch but not smaller than 64 images
  if (agents < 1) agents = 1;
  int want = 32;
  if (const char* e = std::getenv("AGARCL_MIRROR_CHUNKS")) want = std::atoi(e);
  if (want < 1) want = 1;
  const int inst = n_img / agents;
  int ipc_inst = (inst + want - 1) / want;
  if (ipc_inst * agents < 64) ipc_inst = (64 + agents - 1) / agents;
  if (ipc_inst < 1) ipc_inst = 1;
  PackOut& k = m->pk;
  k.ipc = (uint32_t)ipc_inst * (uint32_t)agents;
  m->n_chunks = (n_img + (int)k.ipc - 1) / (int)k.ipc;
  k.rec_words = (uint32_t)(3 + m->frames * 2 * m->MW + 3);
  k.MW = m->MW;
  k.n_img = (uint32_t)n_img;
  uint32_t per_img = (m->cap_img < 1024 ? m->cap_img : 1024) & ~1u;  // entries per image (k_step: the image's slot)
  if (per_img < 2) per_img = 2;
  k.slot = per_img;
  k.cap_chunk = k.ipc * per_img;
  m->meta_words = pk_off_entries(k);
  k.chunk_words = (uint32_t)(m->meta_words + 2 * (size_t)k.cap_chunk);
  const size_t all_words = (size_t)m->n_chunks * k.chunk_words;
  // the mirror itself: 2 MB-aligned, transparent huge pages requested (random element updates over gigabytes are
  // TLB-bound with 4 KB pages), then page-locked; plain cudaHostAlloc if that does not work
  bool ok = true;
  m->lists_only = lists_only;
  if (!lists_only) {
    const size_t bytes = (size_t)n_img * m->img_bytes, two_mb = (size_t)2 << 20;
    void* p = nullptr;
    if (!std::getenv("AGARCL_MIRROR_NO_THP") && posix_memalign(&p, two_mb, (bytes + two_mb - 1) / two_mb * two_mb) == 0 && p) {
#ifdef MADV_HUGEPAGE
      madvise(p, (bytes + two_mb - 1) / two_mb * two_mb, MADV_HUGEPAGE);
#endif
      m->h_obs = p;
      m->obs_registered = false;  // registered after the first touch below
      m->obs_malloced = true;
    } else {
      ok = cudaHostAlloc(&m->h_obs, bytes, cudaHostAllocDefault) == cudaSuccess;
    }
  }
  ok = ok && cudaMalloc((void**)&m->d_chunks, all_words * 4) == cudaSuccess;
  ok = ok && cudaMalloc((void**)&m->d_counters, 2 * (size_t)m->n_chunks * 4) == cudaSuccess;
  ok = ok && cudaMemset(m->d_counters, 0, 2 * (size_t)m->n_chunks * 4) == cudaSuccess;
  ok = ok && cudaHostAlloc((void**)&m->h_flags, (size_t)m->n_chunks * 4, cudaHostAllocMapped) == cudaSuccess;
  ok = ok && cudaHostGetDevicePointer((void**)&m->d_flags, (void*)m->h_flags, 0) == cudaSuccess;
  ok = ok && cudaHostAlloc((void**)&m->h_dxdy, (size_t)n_img * 2 * sizeof(float), cudaHostAllocMapped) == cudaSuccess;
  ok = ok && cudaHostGetDevicePointer((void**)&m->d_dxdy, m->h_dxdy, 0) == cudaSuccess;
  ok = ok && cudaHostAlloc((void**)&m->h_act, (size_t)n_img * sizeof(int32_t), cudaHostAllocMapped) == cudaSuccess;
  ok = ok && cudaHostGetDevicePointer((void**)&m->d_act, m->h_act, 0) == cudaSuccess;
  for (int w = 0; w < 2 && ok; w++) {
    ok = ok && cudaHostAlloc((void**)&m->h_chunks[w], all_words * 4, cudaHostAllocMapped) == cudaSuccess;
    ok = ok && cudaHostGetDevicePointer((void**)&m->dh_chunks[w], m->h_chunks[w], 0) == cudaSuccess;
    if (ok)  // no entries, nothing out of bounds == the all-zero mirror
      for (int c = 0; c < m->n_chunks; c++) std::memset(m->blk(w, c), 0, m->meta_words * 4);
  }
  if (!ok) {
    agarcl_set_error(AGARCL_ERR_NOMEM, "host mirror allocation failed (%zu B pinned): %s", (size_t)n_img * m->img_bytes,
                     cudaGetErrorString(cudaGetLastError()));
    mirror_destroy(m);
    return nullptr;
  }
  for (int c = 0; c < m->n_chunks; c++) m->h_flags[c] = 0u;
  k.chunks = m->d_chunks;
  k.cursor = m->d_counters;
  k.done = m->d_counters + m->n_chunks;
  k.flags = nullptr;
  k.seq = 0;
  int nt = (int)std::thread::hardware_concurrency();
  if (const char* e = std::getenv("AGARCL_HOST_THREADS")) nt = std::atoi(e);
  nt = nt < 1 ? 1 : (nt > 64 ? 64 : nt);
  if (nt > n_img) nt = n_img;
  if (lists_only) nt = 1;  // (nobody expands anything: the caller reads the lists)
  m->pool = new Pool(nt - 1);
  m->stats.host_threads = (uint64_t)nt;
  m->guess.assign((size_t)m->n_chunks, (size_t)k.ipc * 64);
  for (int w = 0; w < 2; w++) {
    m->slot_of[w].resize((size_t)n_img);
    for (int i = 0; i < n_img; i++) m->slot_of[w][(size_t)i] = (uint32_t)i;
  }
  // first touch of the mirror by the threads that will write it
  if (!lists_only) {
    std::atomic<int> next{0};
    m->pool->run([&] {
      for (int i; (i = next.fetch_add(8)) < n_img;) {
        const int hi = i + 8 < n_img ? i + 8 : n_img;
        std::memset((uint8_t*)m->h_obs + (size_t)i * m->img_bytes, 0, (size_t)(hi - i) * m->img_bytes);
      }
    });
  }
  if (m->obs_malloced && !lists_only) {  // page-lock it (dense fallback copies land here; callers may copy it to a device)
    if (cudaHostRegister(m->h_obs, (size_t)n_img * m->img_bytes, cudaHostRegisterDefault) == cudaSuccess) m->obs_registered = true;
    else cudaGetLastError();  // stays pageable: only the rare dense copies get slower
  }
  return m;
}

void* mirror_ptr(HostMirror* m) { return m->h_obs; }
void mirror_stats(const HostMirror* m, MirrorStats* out) { *out = m->stats; }

void mirror_stage_actions(HostMirror* m, const float* dxdy, const int32_t* act, const float** d_dxdy, const int32_t** d_act) {
  std::memcpy(m->h_dxdy, dxdy, (size_t)m->n_img * 2 * sizeof(float));
  std::memcpy(m->h_act, act, (size_t)m->n_img * sizeof(int32_t));
  *d_dxdy = m->d_dxdy;
  *d_act = m->d_act;
}

PackOut mirror_pack_out(HostMirror* m) {
  PackOut k = m->pk;
  k.chunks = m->dh_chunks[m->cur ^ 1];  // mirror_collect flips `cur`: the kernel writes what the host then reads as [cur]
  k.flags = m->d_flags;
  k.seq = ++m->seq;
  return k;
}

#define MCK(call)                                                                                  \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      return agarcl_set_error(AGARCL_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e__));   \
  } while (0)

// Fetches the chunks as they become complete and expands them into the mirror.  `flagged`: a kernel launched on
// `s` with mirror_pack_out() raises the flags (the chunks are fetched on the copy stream while it runs);
// otherwise everything on `s` is complete already.
static int collect(HostMirror* m, const void* d_obs, cudaStream_t s, bool flagged, double* rewards_out = nullptr,
                   uint8_t* dones_out = nullptr) {
  using clk = std::chrono::steady_clock;
  const auto t0 = clk::now();
  m->cur ^= 1;
  const int cur = m->cur, K = m->n_chunks;
  const PackOut& k = m->pk;
  // Chunks become ready in ANY order (under the cost-sorted schedule the first positions are the most expensive
  // instances and finish late): the calling thread appends them to `ready`, the workers take tasks (a chunk's slots in
  // pieces of `grab`) in that order.
  const int grab = 8, tpc = ((int)k.ipc + grab - 1) / grab;  // tasks per chunk
  std::vector<int> ready((size_t)K, 0);
  std::atomic<int> next{0}, n_ready{0};
  std::atomic<bool> abort{false};
  // one task, if there is one: 1 done, 0 nothing ready yet, -1 all tasks taken (or aborted)
  auto try_one = [&]() -> int {
    int i = next.load(std::memory_order_relaxed);
    if (i >= K * tpc || abort.load(std::memory_order_relaxed)) return -1;
    if (i >= n_ready.load(std::memory_order_acquire) * tpc) return 0;
    if (!next.compare_exchange_weak(i, i + 1, std::memory_order_relaxed)) return 1;
    const int c = ready[(size_t)(i / tpc)];
    const int base = c * (int)k.ipc, end = base + (int)k.ipc < m->n_img ? base + (int)k.ipc : m->n_img;
    const int lo = base + (i % tpc) * grab, hi = lo + grab < end ? lo + grab : end;
    if (lo < hi) {
      if (m->dtype == AGARCL_OBS_I16) expand_range<int16_t>(m, lo, hi);
      else expand_range<int32_t>(m, lo, hi);
    }
    return 1;
  };
  const std::function<void()> job = [&] {
    uint32_t idle = 0;
    for (;;) {
      const int r = try_one();
      if (r < 0) break;
      if (r == 1) { idle = 0; continue; }
      cpu_relax();
      if (++idle >= 4096u) { idle = 0; std::this_thread::yield(); }  // (a fully subscribed box: let the threads that have work run)
    }
  };
  m->pool->start(job);
  static const bool trace_env = std::getenv("AGARCL_MIRROR_TRACE") != nullptr;
  const bool trace = trace_env && flagged && (m->seq % 16u == 0u);
  uint64_t d2h = 0, entries = 0;
  std::vector<int> dense_imgs;
  double wait_s = 0.0;
  int rc = AGARCL_OK;
  auto fail = [&](cudaError_t e, const char* what) {
    rc = agarcl_set_error(AGARCL_ERR_CUDA, "%s failed: %s", what, cudaGetErrorString(e));
  };
  // one chunk has arrived in host memory: its records (dense fallbacks, rewards, dones), then hand it to the workers
  auto publish = [&](int c) -> int {
    if (const int r = read_records(m, c, &entries, &dense_imgs, rewards_out, dones_out)) return r;
    const int r = n_ready.load(std::memory_order_relaxed);
    ready[(size_t)r] = c;
    n_ready.store(r + 1, std::memory_order_release);
    if (trace) std::fprintf(stderr, "chunk %d ready at %.0f us, workers at task %d of %d\n", c,
                            std::chrono::duration<double>(clk::now() - t0).count() * 1e6, next.load(), K * tpc);
    return AGARCL_OK;
  };
  if (flagged) {
    // the kernel flags finished chunks in host-mapped memory; the calling thread patches too while it waits for the next flag
    const auto w0 = clk::now();
    rc = wait_chunks(m, s, 1024u, publish, [&] { return try_one() == 1; });
    wait_s = std::chrono::duration<double>(clk::now() - w0).count();
    d2h = lists_d2h_bytes(m, entries);
  } else {
    for (int c = 0; c < K && rc == AGARCL_OK; c++) {  // k_pack left compact blocks in device memory: one copy each (a second one if the guess was short)
      const auto w0 = clk::now();
      uint32_t* hb = m->blk(cur, c);
      const uint32_t* db = m->d_chunks + (size_t)c * k.chunk_words;
      size_t got = m->guess[c] < k.cap_chunk ? m->guess[c] : k.cap_chunk;
      cudaError_t e = cudaMemcpyAsync(hb, db, (m->meta_words + 2 * got) * 4, cudaMemcpyDeviceToHost, s);
      if (e == cudaSuccess) e = cudaStreamSynchronize(s);
      if (e != cudaSuccess) { fail(e, "chunk copy"); break; }
      d2h += (m->meta_words + 2 * got) * 4;
      size_t total = hb[0];
      if (total > k.cap_chunk) total = k.cap_chunk;
      if (total > got) {
        e = cudaMemcpyAsync(hb + m->meta_words + 2 * got, db + m->meta_words + 2 * got, (total - got) * 8, cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) { fail(e, "chunk copy (remainder)"); break; }
        d2h += (total - got) * 8;
      }
      m->guess[c] = total + total / 8 + 1024;
      wait_s += std::chrono::duration<double>(clk::now() - w0).count();
      rc = publish(c);
    }
  }
  // images that do not fit the scheme: dense copies into the pinned mirror (the workers skip them); in the fused
  // path the frames are only known to be complete in device memory once the kernel has ended
  if (rc == AGARCL_OK && !dense_imgs.empty()) {
    cudaError_t e = flagged ? cudaStreamSynchronize(s) : cudaSuccess;
    for (size_t j = 0; j < dense_imgs.size() && e == cudaSuccess; j++) {
      const size_t i = (size_t)dense_imgs[j];
      e = cudaMemcpyAsync((uint8_t*)m->h_obs + i * m->img_bytes, (const uint8_t*)d_obs + i * m->img_bytes, m->img_bytes,
                          cudaMemcpyDeviceToHost, s);
    }
    if (e != cudaSuccess) fail(e, "dense image copy");
  }
  const uint64_t dense = dense_imgs.size();
  if (rc != AGARCL_OK) abort.store(true);
  m->pool->join();
  if (trace) std::fprintf(stderr, "join done at %.0f us\n", std::chrono::duration<double>(clk::now() - t0).count() * 1e6);
  // Every chunk flag is up: all instances have been stepped and everything the caller reads is in host memory.  The
  // kernel's last warps may still be leaving; whatever is enqueued on `s` next is ordered behind them, so only the
  // dense copies (if any) need the stream.
  if (rc == AGARCL_OK && dense) {
    const cudaError_t e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) fail(e, "cudaStreamSynchronize");
  }
  m->stats.entries = entries;
  m->stats.dense_images = dense;
  m->stats.d2h_bytes = d2h + dense * m->img_bytes;
  m->stats.wait_us = (uint64_t)(wait_s * 1e6);
  m->stats.total_us = (uint64_t)(std::chrono::duration<double>(clk::now() - t0).count() * 1e6);
  return rc;
}

int mirror_collect(HostMirror* m, const void* d_obs, cudaStream_t s, double* rewards_out, uint8_t* dones_out) {
  return collect(m, d_obs, s, true, rewards_out, dones_out);
}

int mirror_sync(HostMirror* m, const void* d_obs, cudaStream_t s) {
  PackParams P;
  P.obs = d_obs;
  P.CH = m->CH; P.C = m->C; P.G = m->G;
  P.cap_img = m->cap_img;
  P.pk = m->pk;  // no flags: the host waits for the stream
  const size_t smem = (size_t)m->cap_img * sizeof(uint2) + 2 * (size_t)m->G + 16;
  if (m->dtype == AGARCL_OBS_I16) {
    if (smem > 48 * 1024) MCK(cudaFuncSetAttribute(k_pack<int16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_pack<int16_t><<<m->n_img, kPackThreads, smem, s>>>(P);
  } else {
    if (smem > 48 * 1024) MCK(cudaFuncSetAttribute(k_pack<int32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_pack<int32_t><<<m->n_img, kPackThreads, smem, s>>>(P);
  }
  MCK(cudaGetLastError());
  MCK(cudaStreamSynchronize(s));
  return collect(m, d_obs, s, false);
}

}  // namespace ag
