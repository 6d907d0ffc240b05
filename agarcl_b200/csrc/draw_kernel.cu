// draw_kernel.cu — pictures of game states for people (agarcl_batch_draw; the spec is include/agarcl_b200.h), for sm_100a.
//
// k_draw: arena views.  One CTA draws one tile of one picture (1024 pixels, 256 at S = 16 * odd), and loops over (picture, tile)
// pairs.  (Agent views: k_draw_views below.)
//   1. the world rectangle of the tile;
//   2. the cells and viruses whose drawn disc can reach that rectangle are culled into shared memory with their order key
//      (mass, kind, id, slot) and rank-sorted there; every pixel scans them from the top down and stops at its first hit;
//   3. pixels no cell or virus covers scan the culled pellets and foods, kept in descending array order by warp-ballot
//      compaction, from the top down;
//   4. the tile's RGB bytes, staged in shared memory, leave with one 16-byte store each.
// A culled list that outgrows its shared-memory capacity is resolved in passes: every pixel keeps the key of its best hit,
// so a later pass of cells and viruses only replaces it with a higher key, and a pixel a pellet or food already covered in
// an earlier (higher-index) pass of that list is done.  Nothing is dropped.  The kernel only reads the state.
#include <cuda_runtime.h>

#include "sim_params.h"

namespace ag {

constexpr int kDrawThreads = 256;
constexpr int kDrawTop = 512;    // cells and viruses per pass
constexpr int kDrawLow = 1024;   // pellets and foods per pass
constexpr int kDrawPix = 4;      // pixels per thread at most (1024-pixel tiles)

__constant__ uint32_t c_agent_rgb[8] = AGARCL_DRAW_RGB_AGENTS;
__constant__ uint32_t c_bot_rgb[4] = AGARCL_DRAW_RGB_BOTS;

struct DrawShared {
  float4 top[kDrawTop];                 // x, y, R * R, (0.85 R)^2
  unsigned long long top_k1[kDrawTop];  // mass << 1 | kind (virus 0, cell 1)
  unsigned long long top_k2[kDrawTop];  // id (virus index) << 32 | slot: equal ids (which the game never makes) by slot
  uint32_t top_rgb[kDrawTop], top_border[kDrawTop];
  uint16_t perm[kDrawTop];              // perm[rank] = entry
  float4 low[kDrawLow];                 // x, y, R * R, colour bits; descending array index
  __align__(16) uint8_t pix[1024 * 3];
  uint32_t wcnt[kDrawThreads / 32];
};

__device__ __forceinline__ uint32_t border_rgb(uint32_t c) {
  return ((((c >> 16) & 255u) * 3u / 4u) << 16) | ((((c >> 8) & 255u) * 3u / 4u) << 8) | ((c & 255u) * 3u / 4u);
}
__device__ __forceinline__ float draw_radius(const float* lut, uint32_t m, float px) {
  const float r = m < AGARCL_LUT_SIZE ? lut[m] : radius_exact(m);
  return fmax_std(r, px);
}
__device__ __forceinline__ float disc_d2(float x, float y, float ex, float ey) {
  const float dx = __fsub_rn(x, ex), dy = __fsub_rn(y, ey);
  return __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
}
__device__ __forceinline__ bool key_less(unsigned long long a1, unsigned long long a2, unsigned long long b1, unsigned long long b2) {
  return a1 < b1 || (a1 == b1 && a2 < b2);
}

__global__ void __launch_bounds__(kDrawThreads) k_draw(const __grid_constant__ DrawParams P) {
  __shared__ DrawShared sh;
  const int S = P.S, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int TW = (S % 64 == 0) ? 64 : (S % 32 == 0) ? 32 : 16;
  const int TH = (TW == 16) ? 16 : 1024 / TW;
  const int npix = TW * TH, tiles_x = S / TW, tiles = tiles_x * (S / TH);
  const int64_t n_src = P.N;
  const float W = P.W, fS = (float)S;
  const unsigned lt_mask = (1u << lane) - 1u;
  const int64_t total = (int64_t)P.n * tiles;

  for (int64_t t = blockIdx.x; t < total; t += gridDim.x) {
    const int img = (int)(t / tiles), tile = (int)(t % tiles);
    const int c0 = (tile % tiles_x) * TW, r0 = (tile / tiles_x) * TH;
    const int src = P.src ? P.src[img] : img;
    const bool valid = src >= 0 && src < n_src;
    const int inst = valid ? src : 0;
    const uint8_t* blob = P.state + (size_t)inst * P.L.stride;
    const agarcl_inst_hdr* hdr = reinterpret_cast<const agarcl_inst_hdr*>(blob + P.L.off_hdr);
    const agarcl_player* players = reinterpret_cast<const agarcl_player*>(blob + P.L.off_players);
    const agarcl_cell* cells = reinterpret_cast<const agarcl_cell*>(blob + P.L.off_cells);
    __syncthreads();  // the previous tile is done with the shared memory
    // world coordinate of pixel column (row) i: monotone in i
    auto coord = [&](int i) -> float { return __fdiv_rn(__fmul_rn(__fadd_rn((float)i, 0.5f), W), fS); };
    const float px = __fdiv_rn(W, fS);
    const float x0 = coord(c0), x1 = coord(c0 + TW - 1), y0 = coord(r0), y1 = coord(r0 + TH - 1);

    // per pixel: world position, state (0 open, 1 cell / virus, 2 pellet / food, 3 final), colour, key of the best hit
    const int ppt = npix / kDrawThreads;
    float pxw[kDrawPix], pyw[kDrawPix];
    int res[kDrawPix];
    uint32_t rgb[kDrawPix];
    unsigned long long bk1[kDrawPix], bk2[kDrawPix];
#pragma unroll
    for (int j = 0; j < kDrawPix; j++) {
      res[j] = 3;
      rgb[j] = 0u;
      bk1[j] = bk2[j] = 0ull;
      pxw[j] = pyw[j] = 0.f;
      if (j < ppt && valid) {
        const int p = tid + j * kDrawThreads;
        pxw[j] = coord(c0 + p % TW);
        pyw[j] = coord(r0 + p / TW);
        const bool in = 0 <= pxw[j] && pxw[j] < W && 0 <= pyw[j] && pyw[j] < W;
        res[j] = in ? 0 : 3;
        rgb[j] = in ? AGARCL_DRAW_RGB_BACKGROUND : AGARCL_DRAW_RGB_OUT;
      }
    }
    // a tile entirely outside the arena needs no entity
    const bool any_in = valid && x1 >= 0 && x0 < W && y1 >= 0 && y0 < W;
    if (any_in) {
      // conservative reach of a drawn disc into the tile's rectangle: the margin covers the rounding of the disc test
      const float mag = fabsf(x0) + fabsf(x1) + fabsf(y0) + fabsf(y1);
      auto reaches = [&](float ex, float ey, float R) -> bool {
        const float rr = R + R * 1e-3f + (fabsf(ex) + fabsf(ey) + mag) * 1e-5f;
        return ex + rr >= x0 && ex - rr <= x1 && ey + rr >= y0 && ey - rr <= y1;
      };
      // ---- cells and viruses
      auto resolve_top = [&](int cnt) {
        __syncthreads();
        for (int i = tid; i < cnt; i += kDrawThreads) {
          const unsigned long long a1 = sh.top_k1[i], a2 = sh.top_k2[i];
          int rank = 0;
          for (int k = 0; k < cnt; k++) rank += key_less(sh.top_k1[k], sh.top_k2[k], a1, a2);
          sh.perm[rank] = (uint16_t)i;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < kDrawPix; j++) {
          if (j >= ppt || res[j] == 3) continue;
          for (int k = cnt - 1; k >= 0; k--) {
            const int e = sh.perm[k];
            const unsigned long long e1 = sh.top_k1[e], e2 = sh.top_k2[e];
            if (res[j] == 1 && key_less(e1, e2, bk1[j], bk2[j])) break;  // below the hit of an earlier pass
            const float4 d = sh.top[e];
            const float d2 = disc_d2(pxw[j], pyw[j], d.x, d.y);
            if (d2 <= d.z) {
              res[j] = 1;
              bk1[j] = e1;
              bk2[j] = e2;
              rgb[j] = d2 > d.w ? sh.top_border[e] : sh.top_rgb[e];
              break;
            }
          }
        }
        __syncthreads();
      };
      const int cap_c = P.L.cap_cells;
      const int n_cell_slots = P.L.P * cap_c;
      const int nv = min(max(hdr->n_viruses, 0), P.L.cap_viruses);
      const int ntop = n_cell_slots + nv;
      const agarcl_virus* vir = reinterpret_cast<const agarcl_virus*>(blob + P.L.off_viruses);
      int cnt = 0;
      for (int base = 0; base < ntop; base += kDrawThreads) {
        const int k = base + tid;
        bool keep = false;
        float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
        unsigned long long k1 = 0, k2 = 0;
        uint32_t col = 0, bcol = 0;
        if (k < n_cell_slots) {
          const int p = k / cap_c, i = k - p * cap_c;
          if (i < players[p].n_cells) {
            const agarcl_cell c = cells[k];
            const float R = draw_radius(P.radius, c.mass, px);
            keep = reaches(c.x, c.y, R);
            const float b = __fmul_rn(0.85f, R);
            d = make_float4(c.x, c.y, __fmul_rn(R, R), __fmul_rn(b, b));
            k1 = (unsigned long long)c.mass << 1 | 1ull;
            k2 = (unsigned long long)c.id << 32 | (unsigned)k;
            col = p < P.L.A ? c_agent_rgb[p % 8] : c_bot_rgb[(unsigned)players[p].bot_type & 3u];
            bcol = border_rgb(col);
          }
        } else if (k < ntop) {
          const int v = k - n_cell_slots;
          const agarcl_virus vv = vir[v];
          const float R = draw_radius(P.radius, vv.mass, px);
          keep = reaches(vv.x, vv.y, R);
          const float b = __fmul_rn(0.85f, R);
          d = make_float4(vv.x, vv.y, __fmul_rn(R, R), __fmul_rn(b, b));
          k1 = (unsigned long long)vv.mass << 1;
          k2 = (unsigned long long)(unsigned)v << 32 | (unsigned)v;
          col = AGARCL_DRAW_RGB_VIRUS;
          bcol = AGARCL_DRAW_RGB_VIRUS_BORDER;
        }
        const unsigned bal = __ballot_sync(AG_FULL, keep);
        if (lane == 0) sh.wcnt[warp] = __popc(bal);
        __syncthreads();
        int before = 0, blk = 0;
        for (int w = 0; w < kDrawThreads / 32; w++) {
          const int c = sh.wcnt[w];
          before += w < warp ? c : 0;
          blk += c;
        }
        if (cnt + blk > kDrawTop) {
          resolve_top(cnt);
          cnt = 0;
        }
        if (keep) {
          const int pos = cnt + before + __popc(bal & lt_mask);
          sh.top[pos] = d;
          sh.top_k1[pos] = k1;
          sh.top_k2[pos] = k2;
          sh.top_rgb[pos] = col;
          sh.top_border[pos] = bcol;
        }
        cnt += blk;
        __syncthreads();
      }
      if (cnt) resolve_top(cnt);

      // ---- pellets and foods, only for pixels no cell or virus covers
      int open = 0;
#pragma unroll
      for (int j = 0; j < kDrawPix; j++) open |= (j < ppt && res[j] == 0);
      if (__syncthreads_or(open)) {
        auto resolve_low = [&](int cnt) {
          __syncthreads();
#pragma unroll
          for (int j = 0; j < kDrawPix; j++) {
            if (j >= ppt || res[j] != 0) continue;
            for (int k = 0; k < cnt; k++) {
              const float4 d = sh.low[k];
              if (disc_d2(pxw[j], pyw[j], d.x, d.y) <= d.z) {
                res[j] = 2;
                rgb[j] = __float_as_uint(d.w);
                break;
              }
            }
          }
          __syncthreads();
        };
        const int np = min(max(hdr->n_pellets, 0), P.L.cap_pellets);
        const int nf = min(max(hdr->n_foods, 0), P.L.cap_foods);
        const int nlow = np + nf;
        const float2* pel = reinterpret_cast<const float2*>(blob + P.L.off_pellets);
        const agarcl_food* food = reinterpret_cast<const agarcl_food*>(blob + P.L.off_foods);
        const float Rp = draw_radius(P.radius, AGARCL_PELLET_MASS, px), Rf = draw_radius(P.radius, AGARCL_FOOD_MASS, px);
        const float Rp2 = __fmul_rn(Rp, Rp), Rf2 = __fmul_rn(Rf, Rf);
        cnt = 0;
        for (int base = 0; base < nlow; base += kDrawThreads) {
          const int q = nlow - 1 - (base + tid);  // descending: the top of the list first
          bool keep = false;
          float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
          if (q >= np) {
            const agarcl_food f = food[q - np];
            keep = reaches(f.x, f.y, Rf);
            d = make_float4(f.x, f.y, Rf2, __uint_as_float(AGARCL_DRAW_RGB_FOOD));
          } else if (q >= 0) {
            const float2 e = pel[q];
            keep = reaches(e.x, e.y, Rp);
            d = make_float4(e.x, e.y, Rp2, __uint_as_float(AGARCL_DRAW_RGB_PELLET));
          }
          const unsigned bal = __ballot_sync(AG_FULL, keep);
          if (lane == 0) sh.wcnt[warp] = __popc(bal);
          __syncthreads();
          int before = 0, blk = 0;
          for (int w = 0; w < kDrawThreads / 32; w++) {
            const int c = sh.wcnt[w];
            before += w < warp ? c : 0;
            blk += c;
          }
          if (cnt + blk > kDrawLow) {
            resolve_low(cnt);
            cnt = 0;
          }
          if (keep) sh.low[cnt + before + __popc(bal & lt_mask)] = d;
          cnt += blk;
          __syncthreads();
        }
        if (cnt) resolve_low(cnt);
      }
    }

    // ---- stage the tile's bytes, then one 16-byte store per vector (a tile row is TW * 3 bytes, a multiple of 48)
#pragma unroll
    for (int j = 0; j < kDrawPix; j++) {
      if (j >= ppt) continue;
      uint8_t* o = sh.pix + (tid + j * kDrawThreads) * 3;
      o[0] = (uint8_t)(rgb[j] >> 16);
      o[1] = (uint8_t)(rgb[j] >> 8);
      o[2] = (uint8_t)rgb[j];
    }
    __syncthreads();
    const int row_vec = TW * 3 / 16, nvec = npix * 3 / 16;
    uint8_t* dst = P.out + ((size_t)img * S * S + (size_t)r0 * S + c0) * 3;
    for (int v = tid; v < nvec; v += kDrawThreads) {
      const int rr = v / row_vec, cv = v - rr * row_vec;
      __stcs(reinterpret_cast<int4*>(dst + (size_t)rr * S * 3) + cv, reinterpret_cast<const int4*>(sh.pix)[v]);
    }
  }
}

cudaError_t launch_draw(const DrawParams& P, cudaStream_t stream) {
  const int TW = (P.S % 64 == 0) ? 64 : (P.S % 32 == 0) ? 32 : 16;
  const int TH = (TW == 16) ? 16 : 1024 / TW;
  const int64_t total = (int64_t)P.n * (P.S / TW) * (P.S / TH);
  const int grid = (int)(total < (1 << 20) ? total : (1 << 20));
  if (grid > 0) k_draw<<<grid, kDrawThreads, 0, stream>>>(P);
  return cudaGetLastError();
}

// ---- k_draw_views: agent views, one CTA per picture (and the pixel observation, cfg.pixel_obs)
//   1. the camera of the picture and the world coordinate of every pixel column and row (xs, ys);
//   2. the cells and viruses, then the pellets and foods, whose drawn disc can reach the picture's window are culled ONCE into
//      shared lists, each entry with its pixel bounding box and its place in the draw order (pellet q: q + 1, food f: np + f + 1,
//      cell or virus: np + nf + 1 + its rank by (mass, kind, id, slot) among every cell and virus of the instance);
//   3. the picture is rasterised in bands of rows: every entry paints the pixels of its box inside the band that pass the exact
//      disc test with atomicMax of (order << 32 | colour) into a per-pixel word, so the topmost entity wins whatever the order
//      of the painting; a band's colours are staged as bytes and leave with 16-byte stores.
// A culled list that outgrows its capacity is painted and refilled in passes (painting commutes), and then every band culls
// again; nothing is dropped.  The kernel only reads the state.
constexpr int kViewThreads = 256;
constexpr int kViewPix = 4096;  // pixels of one band
constexpr int kViewTop = 256;   // cells and viruses per pass (>= kViewThreads)
constexpr int kViewLow = 512;   // pellets and foods per pass (>= kViewThreads)

struct ViewTop {
  float x, y, r2, b2;  // centre, R * R, (0.85 R)^2
  uint32_t col, bcol;
  uint32_t order;      // slot (cell slot, or P * cap_cells + virus index) until ranked, then the draw order
  uint16_t c0, c1, r0, r1;  // pixel bounding box, inclusive
};
struct ViewLow {
  float x, y, r2;
  uint32_t order;
  uint16_t c0, c1, r0, r1;
};

static size_t views_smem(int S) {
  return (size_t)kViewPix * 8 + (size_t)kViewPix * 3 + sizeof(ViewTop) * kViewTop + sizeof(ViewLow) * kViewLow + 2 * (size_t)S * 4;
}

__device__ __forceinline__ int first_ge(const float* a, int n, float v) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int m = (lo + hi) >> 1;
    if (a[m] < v) lo = m + 1; else hi = m;
  }
  return lo;
}
__device__ __forceinline__ int first_gt(const float* a, int n, float v) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int m = (lo + hi) >> 1;
    if (a[m] <= v) lo = m + 1; else hi = m;
  }
  return lo;
}

__global__ void __launch_bounds__(kViewThreads) k_draw_views(const __grid_constant__ DrawParams P) {
  extern __shared__ __align__(16) unsigned char vsm[];
  unsigned long long* pix = reinterpret_cast<unsigned long long*>(vsm);
  uint8_t* stage = vsm + (size_t)kViewPix * 8;
  ViewTop* top = reinterpret_cast<ViewTop*>(stage + (size_t)kViewPix * 3);
  ViewLow* low = reinterpret_cast<ViewLow*>(top + kViewTop);
  float* xs = reinterpret_cast<float*>(low + kViewLow);
  float* ys = xs + P.S;
  __shared__ uint32_t wcnt[kViewThreads / 32];
  __shared__ float s_cx, s_cy, s_view;
  const int S = P.S, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int A = P.L.A, cap_c = P.L.cap_cells, n_cell_slots = P.L.P * cap_c;
  const int64_t n_src = (int64_t)P.N * A;
  const int band_rows = kViewPix / S < S ? kViewPix / S : S;
  const float W = P.W, fS = (float)S, half = (float)(S / 2.0);
  const unsigned lt_mask = (1u << lane) - 1u;

  for (int64_t img = blockIdx.x; img < P.n; img += gridDim.x) {
    const int src = P.src ? P.src[img] : (int)img;
    const bool valid = src >= 0 && src < n_src;
    const int inst = valid ? src / A : 0;
    if (valid && P.mask && !P.mask[inst]) continue;  // (uniform over the CTA)
    const uint8_t* blob = P.state + (size_t)inst * P.L.stride;
    const agarcl_inst_hdr* hdr = reinterpret_cast<const agarcl_inst_hdr*>(blob + P.L.off_hdr);
    const agarcl_player* players = reinterpret_cast<const agarcl_player*>(blob + P.L.off_players);
    const agarcl_cell* cells = reinterpret_cast<const agarcl_cell*>(blob + P.L.off_cells);
    const agarcl_virus* vir = reinterpret_cast<const agarcl_virus*>(blob + P.L.off_viruses);
    // pre_respawn: players respawned at the end of the last step are drawn as still dead (no cells)
    const unsigned long long resp = (valid && P.pre_respawn) ? ((unsigned long long)hdr->respawned_hi << 32 | hdr->respawned_lo) : 0ull;
    auto ncells = [&](int p) -> int { return ((resp >> p) & 1ull) ? 0 : min(max(players[p].n_cells, 0), cap_c); };
    __syncthreads();  // the previous picture is done with the shared memory
    if (tid == 0) {
      // the centroid and window of k_obs (Player::x/y/mass in cell order, _view_size = clamp(2 * mass, 100, 300))
      const int a = valid ? src % A : 0;
      const agarcl_cell* pc = cells + (size_t)a * cap_c;
      const int n = valid ? ncells(a) : 0;
      float sx = 0.f, sy = 0.f;
      uint32_t tot = 0;
      for (int i = 0; i < n; i++) {
        sx = __fadd_rn(sx, __fmul_rn(pc[i].x, (float)pc[i].mass));
        sy = __fadd_rn(sy, __fmul_rn(pc[i].y, (float)pc[i].mass));
        tot += pc[i].mass;
      }
      s_cx = __fdiv_rn(sx, (float)tot);
      s_cy = __fdiv_rn(sy, (float)tot);
      s_view = clamp_std((float)(2u * tot), 100.0f, 300.0f);
    }
    __syncthreads();
    const float cx = s_cx, cy = s_cy, view = s_view;
    for (int i = tid; i < S; i += kViewThreads) {
      const float d = __fdiv_rn(__fmul_rn(__fsub_rn((float)i, half), view), fS);
      xs[i] = __fadd_rn(cx, d);
      ys[i] = __fadd_rn(cy, d);
    }
    __syncthreads();
    const float px = __fdiv_rn(view, fS);
    const float x0 = xs[0], x1 = xs[S - 1], y0 = ys[0], y1 = ys[S - 1];
    // a picture entirely outside the arena (or of a dead agent: NaN camera) needs no entity
    const bool any_in = valid && x1 >= 0 && x0 < W && y1 >= 0 && y0 < W;
    const float mag = fabsf(x0) + fabsf(x1) + fabsf(y0) + fabsf(y1);
    // conservative reach of a drawn disc into the window and its pixel box; false when no pixel centre is near enough
    auto box = [&](float ex, float ey, float R, uint16_t& bc0, uint16_t& bc1, uint16_t& br0, uint16_t& br1) -> bool {
      const float rr = R + R * 1e-3f + (fabsf(ex) + fabsf(ey) + mag) * 1e-5f;
      if (!(ex + rr >= x0 && ex - rr <= x1 && ey + rr >= y0 && ey - rr <= y1)) return false;
      const int c0 = first_ge(xs, S, ex - rr), c1 = first_gt(xs, S, ex + rr) - 1;
      const int r0 = first_ge(ys, S, ey - rr), r1 = first_gt(ys, S, ey + rr) - 1;
      bc0 = (uint16_t)c0; bc1 = (uint16_t)max(c1, 0); br0 = (uint16_t)r0; br1 = (uint16_t)max(r1, 0);
      return c0 <= c1 && r0 <= r1;
    };
    const int nv = min(max(hdr->n_viruses, 0), P.L.cap_viruses);
    const int ntop = n_cell_slots + nv;
    const int np = min(max(hdr->n_pellets, 0), P.L.cap_pellets);
    const int nf = min(max(hdr->n_foods, 0), P.L.cap_foods);
    const int nlow = np + nf;
    const float2* pel = reinterpret_cast<const float2*>(blob + P.L.off_pellets);
    const agarcl_food* food = reinterpret_cast<const agarcl_food*>(blob + P.L.off_foods);
    const float Rp = draw_radius(P.radius, AGARCL_PELLET_MASS, px), Rf = draw_radius(P.radius, AGARCL_FOOD_MASS, px);
    const float Rp2 = __fmul_rn(Rp, Rp), Rf2 = __fmul_rn(Rf, Rf);
    // the order key of cell or virus slot k (key_less order; equal ids, which the game never makes, by slot)
    auto top_key = [&](int k, unsigned long long& k1, unsigned long long& k2) {
      if (k < n_cell_slots) {
        k1 = (unsigned long long)cells[k].mass << 1 | 1ull;
        k2 = (unsigned long long)cells[k].id << 32 | (unsigned)k;
      } else {
        const int v = k - n_cell_slots;
        k1 = (unsigned long long)vir[v].mass << 1;
        k2 = (unsigned long long)(unsigned)v << 32 | (unsigned)v;
      }
    };
    // one warp paints one entry's box inside band rows [rb0, rb1)
    auto paint = [&](float ex, float ey, float r2, float b2, unsigned long long vf, unsigned long long vb, int c0, int c1, int r0, int r1,
                     int rb0, int rb1) {
      const int ra = max(r0, rb0), rz = min(r1, rb1 - 1);
      if (ra > rz) return;
      const int w = c1 - c0 + 1, n = w * (rz - ra + 1);
      for (int q = lane; q < n; q += 32) {
        const int rq = q / w, r = ra + rq, c = c0 + q - rq * w;
        const float d2 = disc_d2(xs[c], ys[r], ex, ey);
        if (d2 <= r2) atomicMax(&pix[(r - rb0) * S + c], d2 > b2 ? vb : vf);
      }
    };
    auto paint_top = [&](int cnt, int rb0, int rb1) {
      for (int e = warp; e < cnt; e += kViewThreads / 32) {
        const ViewTop t = top[e];
        const unsigned long long o = (unsigned long long)t.order << 32;
        paint(t.x, t.y, t.r2, t.b2, o | t.col, o | t.bcol, t.c0, t.c1, t.r0, t.r1, rb0, rb1);
      }
    };
    auto paint_low = [&](int cnt, int rb0, int rb1) {
      for (int e = warp; e < cnt; e += kViewThreads / 32) {
        const ViewLow l = low[e];
        const unsigned long long v = (unsigned long long)l.order << 32 | ((int)l.order <= np ? AGARCL_DRAW_RGB_PELLET : AGARCL_DRAW_RGB_FOOD);
        paint(l.x, l.y, l.r2, -1.f, v, v, l.c0, l.c1, l.r0, l.r1, rb0, rb1);
      }
    };
    // ranks the first cnt entries of the top list among every cell and virus of the instance, then paints them
    auto flush_top = [&](int cnt, int rb0, int rb1) {
      __syncthreads();
      for (int e = tid; e < cnt; e += kViewThreads) {
        unsigned long long a1, a2, b1, b2;
        top_key((int)top[e].order, a1, a2);
        uint32_t rank = 0;
        for (int p = 0; p < P.L.P; p++) {
          const int n = min(max(players[p].n_cells, 0), cap_c);
          for (int i = 0; i < n; i++) {
            top_key(p * cap_c + i, b1, b2);
            rank += key_less(b1, b2, a1, a2);
          }
        }
        for (int v = 0; v < nv; v++) {
          top_key(n_cell_slots + v, b1, b2);
          rank += key_less(b1, b2, a1, a2);
        }
        top[e].order = (uint32_t)nlow + 1u + rank;
      }
      __syncthreads();
      paint_top(cnt, rb0, rb1);
      __syncthreads();
    };
    auto flush_low = [&](int cnt, int rb0, int rb1) {
      __syncthreads();
      paint_low(cnt, rb0, rb1);
      __syncthreads();
    };
    // block-wide compaction of the kept entries of one round of kViewThreads candidates: (position before this thread, total)
    auto compact = [&](bool keep, int& before, int& blk) {
      const unsigned bal = __ballot_sync(AG_FULL, keep);
      if (lane == 0) wcnt[warp] = __popc(bal);
      __syncthreads();
      before = __popc(bal & lt_mask);
      blk = 0;
      for (int w = 0; w < kViewThreads / 32; w++) {
        const int c = wcnt[w];
        before += w < warp ? c : 0;
        blk += c;
      }
    };

    int n_top = 0, n_low = 0;
    bool fits = false;  // the lists hold everything culled: later bands paint them again without culling
    for (int rb0 = 0; rb0 < S; rb0 += band_rows) {
      const int rb1 = min(S, rb0 + band_rows), npx = (rb1 - rb0) * S;
      for (int i = tid; i < npx; i += kViewThreads) pix[i] = 0ull;
      __syncthreads();
      if (any_in && fits) {
        paint_top(n_top, rb0, rb1);
        paint_low(n_low, rb0, rb1);
      } else if (any_in) {
        bool passes = false;
        // ---- cells and viruses
        int cnt = 0;
        for (int base = 0; base < ntop; base += kViewThreads) {
          const int k = base + tid;
          bool keep = false;
          ViewTop t;
          if (k < n_cell_slots) {
            const int p = k / cap_c, i = k - p * cap_c;
            if (i < ncells(p)) {
              const agarcl_cell c = cells[k];
              const float R = draw_radius(P.radius, c.mass, px), b = __fmul_rn(0.85f, R);
              keep = box(c.x, c.y, R, t.c0, t.c1, t.r0, t.r1);
              t.x = c.x; t.y = c.y; t.r2 = __fmul_rn(R, R); t.b2 = __fmul_rn(b, b);
              t.col = p < A ? c_agent_rgb[p % 8] : c_bot_rgb[(unsigned)players[p].bot_type & 3u];
              t.bcol = border_rgb(t.col);
              t.order = (uint32_t)k;
            }
          } else if (k < ntop) {
            const agarcl_virus v = vir[k - n_cell_slots];
            const float R = draw_radius(P.radius, v.mass, px), b = __fmul_rn(0.85f, R);
            keep = box(v.x, v.y, R, t.c0, t.c1, t.r0, t.r1);
            t.x = v.x; t.y = v.y; t.r2 = __fmul_rn(R, R); t.b2 = __fmul_rn(b, b);
            t.col = AGARCL_DRAW_RGB_VIRUS;
            t.bcol = AGARCL_DRAW_RGB_VIRUS_BORDER;
            t.order = (uint32_t)k;
          }
          int before, blk;
          compact(keep, before, blk);
          if (cnt + blk > kViewTop) {
            flush_top(cnt, rb0, rb1);
            cnt = 0;
            passes = true;
          }
          if (keep) top[cnt + before] = t;
          cnt += blk;
          __syncthreads();
        }
        if (cnt) flush_top(cnt, rb0, rb1);
        n_top = cnt;
        // ---- pellets and foods
        cnt = 0;
        for (int base = 0; base < nlow; base += kViewThreads) {
          const int q = base + tid;
          bool keep = false;
          ViewLow l;
          if (q < np) {
            const float2 e = pel[q];
            keep = box(e.x, e.y, Rp, l.c0, l.c1, l.r0, l.r1);
            l.x = e.x; l.y = e.y; l.r2 = Rp2;
            l.order = (uint32_t)q + 1u;
          } else if (q < nlow) {
            const agarcl_food f = food[q - np];
            keep = box(f.x, f.y, Rf, l.c0, l.c1, l.r0, l.r1);
            l.x = f.x; l.y = f.y; l.r2 = Rf2;
            l.order = (uint32_t)q + 1u;
          }
          int before, blk;
          compact(keep, before, blk);
          if (cnt + blk > kViewLow) {
            flush_low(cnt, rb0, rb1);
            cnt = 0;
            passes = true;
          }
          if (keep) low[cnt + before] = l;
          cnt += blk;
          __syncthreads();
        }
        if (cnt) flush_low(cnt, rb0, rb1);
        n_low = cnt;
        fits = !passes;
      }
      __syncthreads();
      // ---- the band's colours: out of the arena, the topmost painted entity, or the background; all zero for a bad source
      for (int p = tid; p < npx; p += kViewThreads) {
        const int r = rb0 + p / S, c = p % S;
        uint32_t rgb = 0u;
        if (valid) {
          const float x = xs[c], y = ys[r];
          const unsigned long long v = pix[p];
          rgb = !(0 <= x && x < W && 0 <= y && y < W) ? AGARCL_DRAW_RGB_OUT : v ? (uint32_t)v : AGARCL_DRAW_RGB_BACKGROUND;
        }
        stage[3 * p] = (uint8_t)(rgb >> 16);
        stage[3 * p + 1] = (uint8_t)(rgb >> 8);
        stage[3 * p + 2] = (uint8_t)rgb;
      }
      __syncthreads();
      int4* dst = reinterpret_cast<int4*>(P.out + ((size_t)img * S * S + (size_t)rb0 * S) * 3);
      for (int v = tid; v < npx * 3 / 16; v += kViewThreads) __stcs(dst + v, reinterpret_cast<const int4*>(stage)[v]);
      __syncthreads();
    }
  }
}

cudaError_t setup_draw_views() {
  return cudaFuncSetAttribute(k_draw_views, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)views_smem(2048));
}

cudaError_t launch_draw_views(const DrawParams& P, cudaStream_t stream) {
  const int grid = P.n < (1 << 20) ? P.n : (1 << 20);
  if (grid > 0) k_draw_views<<<grid, kViewThreads, views_smem(P.S), stream>>>(P);
  return cudaGetLastError();
}

}  // namespace ag
