/*
 * draw_oracle.c — TEST INFRASTRUCTURE ONLY.  CPU restatement of the pictures of game states (agarcl_batch_draw), from the spec
 * in include/agarcl_b200.h, on the state blob of that header.  tests/test_draw_oracle.py compiles it into a temporary directory
 * (gcc -ffp-contract=off: every fp32 operation rounded on its own, like the device built with -fmad=false) and holds both the spec
 * and the device kernel (tests/test_gpu_draw.py) to it.  The product never links or falls back to it.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#include "../include/agarcl_b200.h"

#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif

/* radius_conversion, core/utils.hpp:8-11 */
static float radius_of(uint32_t mass) { return (float)sqrt((double)mass / 1.0 / M_PI); }
/* std::min / std::max / agario::clamp on floats, the libstdc++ way */
static float fmin_std(float a, float b) { return (b < a) ? b : a; }
static float fmax_std(float a, float b) { return (a < b) ? b : a; }
static float clampf_std(float x, float lo, float hi) { return fmax_std(fmin_std(x, hi), lo); }
static int clamp_count(int n, int cap) { return n < 0 ? 0 : (n > cap ? cap : n); }

/* ------------------------------------------------------------------------------------------------
 * Pictures for people: agarcl_batch_draw, restated from its spec in include/agarcl_b200.h.  The device resolves each pixel
 * from the top down; this paints every entity bottom to top over the pixels its disc covers (the last painter is the
 * topmost), so the two share the spec and nothing else.
 * out: uint8 [size][size][3].  agent: the agent index for AGARCL_DRAW_AGENT (ignored for the arena view).
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  uint64_t k1, k2; /* (mass << 1 | kind [virus 0, cell 1], id or virus index << 32 | slot) */
  float x, y;
  uint32_t mass, rgb, border;
} draw_ent;

static int cmp_draw_ent(const void* a, const void* b) {
  const draw_ent *p = (const draw_ent*)a, *q = (const draw_ent*)b;
  if (p->k1 != q->k1) return p->k1 < q->k1 ? -1 : 1;
  if (p->k2 != q->k2) return p->k2 < q->k2 ? -1 : 1;
  return 0;
}
static uint32_t draw_border_rgb(uint32_t c) {
  return ((((c >> 16) & 255u) * 3u / 4u) << 16) | ((((c >> 8) & 255u) * 3u / 4u) << 8) | ((c & 255u) * 3u / 4u);
}
static float draw_coord(int view, int i, float c, float span, float W, int S) {
  if (view == AGARCL_DRAW_AGENT) return c + ((float)i - (float)(S / 2.0)) * span / (float)S; /* _grid_to_world */
  return ((float)i + 0.5f) * W / (float)S;
}
/* the pixel indices whose coordinate may lie within r of e (coord is monotone in i; the exact test decides) */
static int draw_range(float e, float r, float a, float pw, int S, int* lo, int* hi) {
  double l = floor(((double)e - r - a) / pw) - 2.0, h = ceil(((double)e + r - a) / pw) + 2.0;
  if (!(l <= h) || h < 0 || l > S - 1) return 0;
  *lo = l < 0 ? 0 : (int)l;
  *hi = h > S - 1 ? S - 1 : (int)h;
  return 1;
}

void oracle_draw(const agarcl_cfg* c, const agarcl_layout* L, void* blob, int view, int agent, int size, uint8_t* out) {
  uint8_t* b = (uint8_t*)blob;
  const agarcl_inst_hdr* hdr = (const agarcl_inst_hdr*)(b + L->off_hdr);
  const agarcl_player* pl = (const agarcl_player*)(b + L->off_players);
  const agarcl_cell* cells = (const agarcl_cell*)(b + L->off_cells); /* [P][cap_cells] */
  const agarcl_virus* vir = (const agarcl_virus*)(b + L->off_viruses);
  const agarcl_food* food = (const agarcl_food*)(b + L->off_foods);
  const agarcl_pellet* pel = (const agarcl_pellet*)(b + L->off_pellets);
  const int S = size;
  const float W = (float)c->arena_size;
  float cx = 0.f, cy = 0.f, span = 0.f;
  if (view == AGARCL_DRAW_AGENT) { /* the centroid and window of the grid observation (Player::x/y/mass in cell order) */
    const agarcl_cell* pc = cells + (size_t)agent * L->cap_cells;
    const int n = clamp_count(pl[agent].n_cells, L->cap_cells);
    float xs = 0.0f, ys = 0.0f;
    uint32_t tot = 0;
    for (int i = 0; i < n; i++) { xs += pc[i].x * (float)pc[i].mass; ys += pc[i].y * (float)pc[i].mass; tot += pc[i].mass; }
    cx = xs / (float)tot; /* 0/0 = NaN for a dead agent: every pixel out of the arena */
    cy = ys / (float)tot;
    span = clampf_std((float)(2u * tot), 100.0f, 300.0f);
  }
  const float px = view == AGARCL_DRAW_AGENT ? span / (float)S : W / (float)S;
  const float ax = draw_coord(view, 0, cx, span, W, S), ay = draw_coord(view, 0, cy, span, W, S);
  float* xs = (float*)malloc(sizeof(float) * S);
  float* ys = (float*)malloc(sizeof(float) * S);
  uint32_t* pix = (uint32_t*)malloc(sizeof(uint32_t) * (size_t)S * S);
  for (int i = 0; i < S; i++) { xs[i] = draw_coord(view, i, cx, span, W, S); ys[i] = draw_coord(view, i, cy, span, W, S); }
  for (size_t k = 0; k < (size_t)S * S; k++) pix[k] = AGARCL_DRAW_RGB_BACKGROUND;

  /* paints colour rgb (border where d2 > b2, when b2 >= 0) over the pixels the disc (ex, ey, R) contains */
#define DRAW_PAINT(ex, ey, R, b2, rgb, border)                                                          \
  do {                                                                                                  \
    int c_lo, c_hi, r_lo, r_hi;                                                                         \
    float R2_ = (R) * (R);                                                                              \
    if (draw_range((ex), (R), ax, px, S, &c_lo, &c_hi) && draw_range((ey), (R), ay, px, S, &r_lo, &r_hi)) \
      for (int r = r_lo; r <= r_hi; r++)                                                                \
        for (int q = c_lo; q <= c_hi; q++) {                                                            \
          float dx = xs[q] - (ex), dy = ys[r] - (ey);                                                   \
          float d2 = dx * dx + dy * dy;                                                                 \
          if (d2 <= R2_) pix[(size_t)r * S + q] = ((b2) >= 0.0f && d2 > (b2)) ? (border) : (rgb);       \
        }                                                                                               \
  } while (0)

  const float radius_pel = fmax_std(radius_of(AGARCL_PELLET_MASS), px), radius_food = fmax_std(radius_of(AGARCL_FOOD_MASS), px);
  const int np = clamp_count(hdr->n_pellets, L->cap_pellets), nf = clamp_count(hdr->n_foods, L->cap_foods);
  const int nv = clamp_count(hdr->n_viruses, L->cap_viruses);
  for (int i = 0; i < np; i++) DRAW_PAINT(pel[i].x, pel[i].y, radius_pel, -1.0f, AGARCL_DRAW_RGB_PELLET, 0u);
  for (int i = 0; i < nf; i++) DRAW_PAINT(food[i].x, food[i].y, radius_food, -1.0f, AGARCL_DRAW_RGB_FOOD, 0u);

  static const uint32_t agent_rgb[8] = AGARCL_DRAW_RGB_AGENTS, bot_rgb[4] = AGARCL_DRAW_RGB_BOTS;
  draw_ent* ents = (draw_ent*)malloc(sizeof(draw_ent) * ((size_t)L->P * L->cap_cells + nv + 1));
  int ne = 0;
  for (int p = 0; p < L->P; p++) {
    const int n = clamp_count(pl[p].n_cells, L->cap_cells);
    uint32_t rgb = p < L->A ? agent_rgb[p % 8] : bot_rgb[(uint32_t)pl[p].bot_type & 3u];
    for (int i = 0; i < n; i++) {
      const agarcl_cell* cl = cells + (size_t)p * L->cap_cells + i;
      draw_ent e = {(uint64_t)cl->mass << 1 | 1u, (uint64_t)cl->id << 32 | (uint32_t)(p * L->cap_cells + i), cl->x, cl->y, cl->mass,
                    rgb, draw_border_rgb(rgb)};
      ents[ne++] = e;
    }
  }
  for (int v = 0; v < nv; v++) {
    draw_ent e = {(uint64_t)vir[v].mass << 1, (uint64_t)(uint32_t)v << 32 | (uint32_t)v, vir[v].x, vir[v].y, vir[v].mass,
                  AGARCL_DRAW_RGB_VIRUS, AGARCL_DRAW_RGB_VIRUS_BORDER};
    ents[ne++] = e;
  }
  qsort(ents, ne, sizeof(draw_ent), cmp_draw_ent);
  for (int k = 0; k < ne; k++) {
    float R = fmax_std(radius_of(ents[k].mass), px);
    float b = 0.85f * R;
    DRAW_PAINT(ents[k].x, ents[k].y, R, b * b, ents[k].rgb, ents[k].border);
  }
#undef DRAW_PAINT
  for (int r = 0; r < S; r++)
    for (int q = 0; q < S; q++) {
      uint32_t v = (0 <= xs[q] && xs[q] < W && 0 <= ys[r] && ys[r] < W) ? pix[(size_t)r * S + q] : AGARCL_DRAW_RGB_OUT;
      uint8_t* o = out + ((size_t)r * S + q) * 3;
      o[0] = (uint8_t)(v >> 16);
      o[1] = (uint8_t)(v >> 8);
      o[2] = (uint8_t)v;
    }
  free(ents);
  free(pix);
  free(xs);
  free(ys);
}
