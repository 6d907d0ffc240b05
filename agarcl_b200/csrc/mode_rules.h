// mode_rules.h — what a mode_number means for the game, as one function of the mode shared by the host layout
// (layout.cpp) and the kernels (a mixed-task batch derives the rules of every instance from its current mode).
//
// Reference behaviour restated here:
//   Engine::set_mode                     agario/engine/Engine.hpp:367-416
//   BaseEnvironment::reset / add_bots    environment/envs/BaseEnvironment.hpp:179-204,374-425
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define AG_HD __host__ __device__ __forceinline__
#else
#define AG_HD inline
#endif

namespace ag {

struct ModeRules {
  int32_t mass_decay, squared_pellets, regen, agent_mass;
  int32_t bots;  // bot players that follow the agents
};

// Engine::set_mode, and the bot count of BaseEnvironment::reset: num_bots of them in mode 0, exactly one in modes 7..10
AG_HD ModeRules mode_rules(int mode, int num_bots) {
  int base = mode;
  if (mode == 5) base = 2;
  if (mode >= 6) base = 4;
  ModeRules r;
  r.mass_decay = (base == 0 || base == 2 || base == 4);
  r.squared_pellets = (base == 1 || base == 2);
  r.regen = (base == 0 || base == 3 || base == 4);
  r.agent_mass = (mode == 5 || mode == 6) ? 1000 : 25;
  r.bots = mode == 0 ? num_bots : (mode > 6 ? 1 : 0);
  return r;
}

// bot type of player p (A agents): -1 for an agent; add_bots in mode 0 (switch (i % num_bots_) with i < num_bots_, quirk Q14),
// custom_add_bot (type mode - 7) otherwise
AG_HD int32_t mode_bot_type(int mode, int p, int A) {
  if (p < A) return -1;
  if (mode == 0) {
    const int i = p - A;
    return i < 4 ? i : 0;
  }
  const int idx = mode - 7;
  return (idx >= 0 && idx < 4) ? idx : 0;
}

}  // namespace ag
