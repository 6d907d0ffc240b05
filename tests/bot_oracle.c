/*
 * bot_oracle.c — TEST INFRASTRUCTURE ONLY.  oracle_bot_decide: the spec of agarcl_batch_bot_actions (include/agarcl_b200.h) as
 * oracle/oracle.c's own bot code.  It includes oracle.c unchanged, so the static bot_take_action that the compiled-reference
 * lockstep tests pin is the very code it runs.  tests/test_bot_actions_oracle.py compiles it into a temporary directory with the
 * oracle's flags (gcc -ffp-contract=off) and holds the device kernel (tests/test_gpu_bot_actions.py) to it.  The product never
 * links or falls back to it.
 */
#include "../oracle/oracle.c"

/* What Bot::take_action of bot type `type` would leave in agent `agent`'s player record, on a private copy of the blob (the blob
 * is not touched).  out_dxdy = (target - loc) / 10 in fp32, out_status AGARCL_BOT_*; type outside 0..3: status BAD_TYPE and
 * nothing else written (-1: SKIPPED, likewise). */
void oracle_bot_decide(const agarcl_cfg* c, const agarcl_layout* L, const void* blob, int agent, int type, float* out_dxdy,
                       float* out_target, int32_t* out_act, uint8_t* out_status) {
  if (type == -1) { *out_status = AGARCL_BOT_SKIPPED; return; }
  if (type < 0 || type > 3) { *out_status = AGARCL_BOT_BAD_TYPE; return; }
  void* copy = malloc(L->stride);
  memcpy(copy, blob, L->stride);
  inst S, *s = &S;
  bind(s, c, L, copy, NULL, 0);
  agarcl_player* pl = &s->pl[agent];
  if (pl->n_cells == 0) {
    *out_status = AGARCL_BOT_DEAD;
    out_dxdy[0] = out_dxdy[1] = 0.0f;
    out_target[0] = out_target[1] = 0.0f;
    *out_act = 0;
    free(copy);
    return;
  }
  float lx, ly;
  player_loc(s, agent, &lx, &ly);
  s->hdr->flags &= ~AGARCL_FLAG_RAND_SITE;
  pl->bot_type = type;
  bot_take_action(s, agent);
  if (s->hdr->flags & AGARCL_FLAG_RAND_SITE) {
    *out_status = AGARCL_BOT_NO_PELLET;
    out_dxdy[0] = out_dxdy[1] = 0.0f;
    out_target[0] = lx;
    out_target[1] = ly;
    *out_act = 0;
  } else {
    *out_status = AGARCL_BOT_DECIDED;
    out_dxdy[0] = (pl->target_x - lx) / 10.0f;
    out_dxdy[1] = (pl->target_y - ly) / 10.0f;
    out_target[0] = pl->target_x;
    out_target[1] = pl->target_y;
    *out_act = pl->action;
  }
  free(copy);
}
