// snapshot.cpp — the reference's JSON environment snapshot for one instance blob (host only).
//
// Writes what BaseEnvironment::save_env_state writes (environment/envs/BaseEnvironment.hpp:213-318: config,
// players with cooldowns / statistics / cells, pellets, viruses, foods) and reads it back the way
// Engine::load_env_state does (agario/engine/Engine.hpp:247-348: bot type from the player name, cell
// (id, x, y, mass, velocity), ticks = 0, rng re-seeded).  The reference format is LOSSY (no splitting
// velocity, recombine timers, virus food hits); those are written as extra keys the reference ignores
// ("split_velocity_*", "recombine_tick", "food_hits", "ticks", "action", "min_mass_cell", "rng_cursor",
// "next_cell_id") and are restored only when `lossless` is set on load.
// Difference from the reference: players keep the "pid" recorded in the file (the reference renumbers
// them in file order, which permutes agents and bots after a reload).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "host_util.h"

namespace {

// ---------------------------------------------------------------- minimal JSON value + parser
struct JV {
  enum T { NUL, BOOL, NUM, STR, ARR, OBJ } t = NUL;
  double num = 0;
  bool b = false;
  std::string str;
  std::vector<JV> arr;
  std::vector<std::pair<std::string, JV>> obj;
  const JV* get(const char* k) const {
    for (auto& kv : obj)
      if (kv.first == k) return &kv.second;
    return nullptr;
  }
  double n(const char* k, double dflt = 0) const {
    const JV* v = get(k);
    if (!v) return dflt;
    if (v->t == BOOL) return v->b ? 1 : 0;
    return v->t == NUM ? v->num : dflt;
  }
};

struct Parser {
  const char* p;
  const char* end;
  bool ok = true;
  void ws() { while (p < end && (*p == ' ' || *p == '\n' || *p == '\t' || *p == '\r')) p++; }
  bool lit(const char* s) {
    size_t n = strlen(s);
    if ((size_t)(end - p) >= n && !strncmp(p, s, n)) { p += n; return true; }
    return false;
  }
  std::string string() {
    std::string out;
    p++;  // opening quote
    while (p < end && *p != '"') {
      if (*p == '\\' && p + 1 < end) {
        p++;
        switch (*p) {
          case 'n': out += '\n'; break;
          case 't': out += '\t'; break;
          case 'u': p += 4; out += '?'; break;
          default: out += *p;
        }
        p++;
      } else out += *p++;
    }
    if (p < end) p++; else ok = false;
    return out;
  }
  JV value() {
    JV v;
    ws();
    if (p >= end) { ok = false; return v; }
    if (*p == '{') {
      v.t = JV::OBJ;
      p++;
      ws();
      if (p < end && *p == '}') { p++; return v; }
      while (ok) {
        ws();
        if (p >= end || *p != '"') { ok = false; break; }
        std::string k = string();
        ws();
        if (p >= end || *p != ':') { ok = false; break; }
        p++;
        v.obj.emplace_back(std::move(k), value());
        ws();
        if (p < end && *p == ',') { p++; continue; }
        if (p < end && *p == '}') { p++; break; }
        ok = false;
      }
    } else if (*p == '[') {
      v.t = JV::ARR;
      p++;
      ws();
      if (p < end && *p == ']') { p++; return v; }
      while (ok) {
        v.arr.push_back(value());
        ws();
        if (p < end && *p == ',') { p++; continue; }
        if (p < end && *p == ']') { p++; break; }
        ok = false;
      }
    } else if (*p == '"') {
      v.t = JV::STR;
      v.str = string();
    } else if (lit("true")) { v.t = JV::BOOL; v.b = true; }
    else if (lit("false")) { v.t = JV::BOOL; v.b = false; }
    else if (lit("null")) { v.t = JV::NUL; }
    else {
      char* e = nullptr;
      v.num = strtod(p, &e);
      if (e == p) ok = false; else { v.t = JV::NUM; p = e; }
    }
    return v;
  }
};

const char* kBotNames[4] = {"HungryBot", "HungryShyBot", "AggressiveBot", "AggressiveShyBot"};

// the whole file parsed; AGARCL_ERR_INVALID when it cannot be read or is not a JSON object
int parse_file(const char* path, JV& root) {
  FILE* f = fopen(path, "r");
  if (!f) return agarcl_set_error(AGARCL_ERR_INVALID, "Failed to open %s for reading", path);
  std::string text;
  char buf[1 << 16];
  size_t n;
  while ((n = fread(buf, 1, sizeof buf, f)) > 0) text.append(buf, n);
  fclose(f);
  Parser ps{text.data(), text.data() + text.size()};
  root = ps.value();
  if (!ps.ok || root.t != JV::OBJ) return agarcl_set_error(AGARCL_ERR_INVALID, "%s is not a JSON environment snapshot", path);
  return AGARCL_OK;
}

}  // namespace

int snapshot_file_task(const char* path, agarcl_cfg* c) {
  JV root;
  int rc = parse_file(path, root);
  if (rc) return rc;
  if (!root.get("mode_number")) return agarcl_set_error(AGARCL_ERR_INVALID, "snapshot %s has no mode_number", path);
  c->mode_number = (int)root.n("mode_number");
  c->num_bots = (int)root.n("num_bots", c->num_bots);
  c->num_pellets = (int)root.n("num_pellets", c->num_pellets);
  c->num_viruses = (int)root.n("num_viruses", c->num_viruses);
  return AGARCL_OK;
}

// blob -> file.  `cfg` supplies what the blob does not carry (BaseEnvironment's own members).
// Players are written in pid order: Engine::load_env_state re-adds them in file order with fresh pids
// (Engine.hpp:270-284), so this is the order in which a reload by the reference keeps every pid.
extern "C" int agarcl_snapshot_write(const agarcl_cfg* c, const agarcl_layout* L, const void* blob_, const char* path) {
  const uint8_t* blob = static_cast<const uint8_t*>(blob_);
  const auto* hdr = reinterpret_cast<const agarcl_inst_hdr*>(blob + L->off_hdr);
  const auto* pls = reinterpret_cast<const agarcl_player*>(blob + L->off_players);
  const auto* cells = reinterpret_cast<const agarcl_cell*>(blob + L->off_cells);
  const auto* vir = reinterpret_cast<const agarcl_virus*>(blob + L->off_viruses);
  const auto* food = reinterpret_cast<const agarcl_food*>(blob + L->off_foods);
  const auto* pel = reinterpret_cast<const agarcl_pellet*>(blob + L->off_pellets);
  FILE* f = fopen(path, "w");
  if (!f) return agarcl_set_error(AGARCL_ERR_INVALID, "Failed to open %s for writing", path);
  fprintf(f, "{\n");
  fprintf(f, "    \"arena_size\": %d,\n    \"c_death\": %d,\n    \"mode_number\": %d,\n    \"num_agents\": %d,\n    \"num_bots\": %d,\n",
          c->arena_size, c->c_death, c->mode_number, c->num_agents, c->num_bots);
  fprintf(f, "    \"pellet_count\": %d,\n    \"pellet_regen\": %s,\n    \"reward_type\": %d,\n    \"ticks_per_step\": %d,\n",
          hdr->n_pellets, c->pellet_regen ? "true" : "false", c->reward_type, c->ticks_per_step);
  if (c->task_modes)  // a mixed-task batch's instance: its game sizes (agarcl_batch_set_task_sizes)
    fprintf(f, "    \"num_pellets\": %d,\n    \"num_viruses\": %d,\n", c->num_pellets, c->num_viruses);
  // "seed" is what the reference reads back (Engine.hpp:346, 32 bits); the upper half of a 64-bit Philox key travels as an extra key
  fprintf(f, "    \"seed\": %u,\n    \"seed_hi\": %u,\n    \"ticks\": %u,\n    \"rng_cursor\": %u,\n    \"next_cell_id\": %u,\n", hdr->seed_lo,
          hdr->seed_hi, hdr->tick, hdr->rng_cursor, hdr->next_cell_id);
  fprintf(f, "    \"players\": [");
  for (int k = 0; k < L->P; k++) {
    const int p = k;
    const agarcl_player& pl = pls[p];
    const int bt = L->bot_type[p];
    char name[32];
    if (bt >= 0 && bt < 4) snprintf(name, sizeof name, "%s", kBotNames[bt]);
    else snprintf(name, sizeof name, "agent%d", p);
    fprintf(f, "%s\n        {\n", k ? "," : "");
    fprintf(f, "            \"pid\": %d,\n            \"name\": \"%s\",\n            \"is_bot\": %s,\n            \"dead\": %s,\n", p, name,
            bt >= 0 ? "true" : "false", pl.n_cells == 0 ? "true" : "false");
    fprintf(f, "            \"target_x\": %.9g,\n            \"target_y\": %.9g,\n            \"action\": %d,\n", pl.target_x, pl.target_y, pl.action);
    fprintf(f, "            \"split_cooldown\": %d,\n            \"feed_cooldown\": %d,\n            \"anti_team_decay\": %.9g,\n", pl.split_cd,
            pl.feed_cd, pl.anti_team_decay);
    fprintf(f, "            \"elapsed_ticks\": %d,\n            \"last_decay_tick\": %d,\n            \"food_eaten\": %d,\n", pl.elapsed_ticks,
            pl.last_decay_tick, pl.food_eaten);
    fprintf(f, "            \"highest_mass\": %u,\n            \"cells_eaten\": %d,\n            \"viruses_eaten\": %d,\n            \"top_position\": 0,\n",
            pl.highest_mass, pl.cells_eaten, pl.viruses_eaten);
    fprintf(f, "            \"min_mass_cell\": %u,\n            \"virus_eaten_ticks\": [", pl.min_mass_cell);
    for (int i = 0; i < pl.vet_count && i < AGARCL_VET_CAP; i++) fprintf(f, "%s%d", i ? ", " : "", pl.vet_ticks[i]);
    fprintf(f, "],\n            \"cells\": [");
    for (int i = 0; i < pl.n_cells && i < L->cap_cells; i++) {
      const agarcl_cell& cl = cells[(size_t)p * L->cap_cells + i];
      fprintf(f, "%s\n                {\"id\": %u, \"x\": %.9g, \"y\": %.9g, \"mass\": %u, \"velocity_x\": %.9g, \"velocity_y\": %.9g, \"color\": 0, "
                 "\"split_velocity_x\": %.9g, \"split_velocity_y\": %.9g, \"recombine_tick\": %u}",
              i ? "," : "", cl.id, cl.x, cl.y, cl.mass, cl.vx, cl.vy, cl.svx, cl.svy, cl.recomb_tick);
    }
    fprintf(f, "%s]\n        }", pl.n_cells ? "\n            " : "");
  }
  fprintf(f, "\n    ],\n    \"pellets\": [");
  for (int i = 0; i < hdr->n_pellets; i++) fprintf(f, "%s\n        {\"x\": %.9g, \"y\": %.9g}", i ? "," : "", pel[i].x, pel[i].y);
  fprintf(f, "\n    ],\n    \"viruses\": [");
  for (int i = 0; i < hdr->n_viruses; i++)
    fprintf(f, "%s\n        {\"x\": %.9g, \"y\": %.9g, \"velocity_x\": %.9g, \"velocity_y\": %.9g, \"mass\": %.1f, \"food_hits\": %d}", i ? "," : "",
            vir[i].x, vir[i].y, vir[i].vx, vir[i].vy, (double)vir[i].mass, vir[i].hits);
  fprintf(f, "\n    ],\n    \"foods\": [");
  for (int i = 0; i < hdr->n_foods; i++)
    fprintf(f, "%s\n        {\"x\": %.9g, \"y\": %.9g, \"velocity_x\": %.9g, \"velocity_y\": %.9g}", i ? "," : "", food[i].x, food[i].y, food[i].vx,
            food[i].vy);
  fprintf(f, "\n    ]\n}\n");
  if (fclose(f) != 0) return agarcl_set_error(AGARCL_ERR_INVALID, "write to %s failed", path);
  return AGARCL_OK;
}

// file -> blob (Engine::load_env_state).  `blob` must be an initialised blob of this layout (its header seed/flags are kept unless the file has them).
extern "C" int agarcl_snapshot_read(const agarcl_cfg* c, const agarcl_layout* L, void* blob_, const char* path, int lossless) {
  JV root;
  int rc = parse_file(path, root);
  if (rc) return rc;
  if ((int)root.n("mode_number", c->mode_number) != c->mode_number)
    return agarcl_set_error(AGARCL_ERR_INVALID, "snapshot mode_number %d does not match the environment's %d", (int)root.n("mode_number"), c->mode_number);
  const JV* players = root.get("players");
  const JV* pellets = root.get("pellets");
  const JV* viruses = root.get("viruses");
  const JV* foods = root.get("foods");
  if (!players || players->t != JV::ARR || !pellets || !viruses || !foods)
    return agarcl_set_error(AGARCL_ERR_INVALID, "snapshot lacks players / pellets / viruses / foods");
  if ((int)players->arr.size() != L->P)
    return agarcl_set_error(AGARCL_ERR_INVALID, "snapshot has %d players, the environment %d", (int)players->arr.size(), L->P);
  if ((int)pellets->arr.size() > L->cap_pellets || (int)viruses->arr.size() > L->cap_viruses || (int)foods->arr.size() > L->cap_foods)
    return agarcl_set_error(AGARCL_ERR_INVALID, "snapshot exceeds a capacity of the environment (pellets %d, viruses %d, foods %d)",
                            (int)pellets->arr.size(), (int)viruses->arr.size(), (int)foods->arr.size());
  uint8_t* blob = static_cast<uint8_t*>(blob_);
  auto* hdr = reinterpret_cast<agarcl_inst_hdr*>(blob + L->off_hdr);
  auto* pls = reinterpret_cast<agarcl_player*>(blob + L->off_players);
  auto* cells = reinterpret_cast<agarcl_cell*>(blob + L->off_cells);
  auto* vir = reinterpret_cast<agarcl_virus*>(blob + L->off_viruses);
  auto* food = reinterpret_cast<agarcl_food*>(blob + L->off_foods);
  auto* pel = reinterpret_cast<agarcl_pellet*>(blob + L->off_pellets);
  std::vector<char> seen(L->P, 0);
  uint32_t max_id = 0;
  const uint32_t tick = lossless ? (uint32_t)root.n("ticks", 0) : 0u;  // state.ticks = 0 (Engine.hpp:345)
  for (size_t k = 0; k < players->arr.size(); k++) {
    const JV& pd = players->arr[k];
    int p = (int)pd.n("pid", (double)k);
    if (p < 0 || p >= L->P || seen[p]) return agarcl_set_error(AGARCL_ERR_INVALID, "snapshot player pid %d is out of range or repeated", p);
    seen[p] = 1;
    const JV* nm = pd.get("name");
    int bt = -1;
    for (int i = 0; i < 4; i++)
      if (nm && nm->str == kBotNames[i]) bt = i;
    if (bt != L->bot_type[p])
      return agarcl_set_error(AGARCL_ERR_INVALID, "snapshot player %d is \"%s\" but the environment's roster has bot type %d there", p,
                              nm ? nm->str.c_str() : "?", L->bot_type[p]);
    agarcl_player& pl = pls[p];
    memset(&pl, 0, sizeof pl);
    pl.bot_type = bt;
    pl.target_x = (float)pd.n("target_x");
    pl.target_y = (float)pd.n("target_y");
    pl.action = lossless ? (int)pd.n("action", 0) : 0;
    pl.split_cd = (int)pd.n("split_cooldown");
    pl.feed_cd = (int)pd.n("feed_cooldown");
    pl.anti_team_decay = (float)pd.n("anti_team_decay", 1.0);
    pl.elapsed_ticks = (int)pd.n("elapsed_ticks");
    pl.last_decay_tick = (int)pd.n("last_decay_tick");
    pl.food_eaten = (int)pd.n("food_eaten");
    pl.highest_mass = (uint32_t)pd.n("highest_mass");
    pl.cells_eaten = (int)pd.n("cells_eaten");
    pl.viruses_eaten = (int)pd.n("viruses_eaten");
    pl.min_mass_cell = lossless ? (uint32_t)pd.n("min_mass_cell", AGARCL_CELL_MIN_SIZE) : AGARCL_CELL_MIN_SIZE;
    if (const JV* vt = pd.get("virus_eaten_ticks"))
      for (size_t i = 0; i < vt->arr.size() && i < AGARCL_VET_CAP; i++) pl.vet_ticks[pl.vet_count++] = (int)vt->arr[i].num;
    const JV* cs = pd.get("cells");
    if (cs && (int)cs->arr.size() > L->cap_cells) return agarcl_set_error(AGARCL_ERR_INVALID, "snapshot player %d has too many cells", p);
    for (size_t i = 0; cs && i < cs->arr.size(); i++) {
      const JV& cd = cs->arr[i];
      agarcl_cell& cl = cells[(size_t)p * L->cap_cells + i];
      memset(&cl, 0, sizeof cl);
      cl.x = (float)cd.n("x"); cl.y = (float)cd.n("y");
      cl.vx = (float)cd.n("velocity_x"); cl.vy = (float)cd.n("velocity_y");
      uint32_t m = (uint32_t)(float)cd.n("mass");
      cl.mass = m > AGARCL_CELL_MIN_SIZE ? m : AGARCL_CELL_MIN_SIZE;  // Cell::set_mass
      cl.id = (uint32_t)cd.n("id");
      cl.recomb_tick = tick;  // _recombine_timer = now(): may recombine at once (Entities.hpp:124-128)
      if (lossless) {
        cl.svx = (float)cd.n("split_velocity_x"); cl.svy = (float)cd.n("split_velocity_y");
        cl.recomb_tick = (uint32_t)cd.n("recombine_tick", tick);
      }
      if (cl.id > max_id) max_id = cl.id;
      pl.n_cells++;
    }
  }
  hdr->n_pellets = (int)pellets->arr.size();
  for (int i = 0; i < hdr->n_pellets; i++) { pel[i].x = (float)pellets->arr[i].n("x"); pel[i].y = (float)pellets->arr[i].n("y"); }
  hdr->n_viruses = (int)viruses->arr.size();
  for (int i = 0; i < hdr->n_viruses; i++) {
    const JV& v = viruses->arr[i];
    memset(&vir[i], 0, sizeof vir[i]);
    vir[i].x = (float)v.n("x"); vir[i].y = (float)v.n("y");
    vir[i].vx = (float)v.n("velocity_x"); vir[i].vy = (float)v.n("velocity_y");
    vir[i].mass = (uint32_t)(float)v.n("mass", AGARCL_VIRUS_INITIAL_MASS);
    vir[i].hits = lossless ? (int)v.n("food_hits", 0) : 0;
  }
  hdr->n_foods = (int)foods->arr.size();
  for (int i = 0; i < hdr->n_foods; i++) {
    const JV& v = foods->arr[i];
    food[i].x = (float)v.n("x"); food[i].y = (float)v.n("y");
    food[i].vx = (float)v.n("velocity_x"); food[i].vy = (float)v.n("velocity_y");
  }
  hdr->tick = tick;
  hdr->next_cell_id = lossless && root.get("next_cell_id") ? (uint32_t)root.n("next_cell_id") : max_id + 1u;
  hdr->rng_cursor = lossless ? (uint32_t)root.n("rng_cursor", 0) : 0u;  // seed(agarcl_data["seed"]) restarts the stream (Engine.hpp:346)
  if (root.get("seed")) {  // (a file without a seed leaves the instance's key alone)
    hdr->seed_lo = (uint32_t)root.n("seed", hdr->seed_lo);
    hdr->seed_hi = (uint32_t)root.n("seed_hi", 0);  // absent in files written by the reference: its seeds are 32 bits
  }
  hdr->flags = 0;
  hdr->done_sticky = 0;
  hdr->respawned_lo = hdr->respawned_hi = 0;
  return AGARCL_OK;
}
