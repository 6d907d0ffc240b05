// host_util.h — error plumbing shared by the host translation units of libagarcl_b200.so.
// The reference raises C++ exceptions (EnvironmentException, BaseEnvironment.hpp:19); nothing may
// unwind across the C ABI, so every entry point records a message and returns a status instead.
#pragma once
#include "../../include/agarcl_b200.h"

int agarcl_set_error(int status, const char* fmt, ...);

// snapshot.cpp: the reference's JSON environment snapshot to / from one instance blob (host memory)
extern "C" int agarcl_snapshot_write(const agarcl_cfg* c, const agarcl_layout* L, const void* blob, const char* path);
extern "C" int agarcl_snapshot_read(const agarcl_cfg* c, const agarcl_layout* L, void* blob, const char* path, int lossless);
// snapshot.cpp: the task a JSON snapshot was written in: mode_number, and num_bots / num_pellets / num_viruses where the file has
// them (c's values are kept otherwise)
int snapshot_file_task(const char* path, agarcl_cfg* c);

// layout.cpp, mixed-task batches (cfg.task_modes): the layout of the batch as an instance of `mode` with `bots` bots in mode 0
// sees it -- P = A + its bots, its mode flags and bot types, and the player order a batch of that mode alone uses
// (agarcl_make_layout checks that it is the order of the batch's players < P)
void task_layout(const agarcl_cfg* c, const agarcl_layout* L, int mode, int bots, agarcl_layout* out);
// layout.cpp, a batch of c and L with mode 0 in task_modes: bit b set = a mode-0 instance of b bots (0 .. num_bots) may play in it
// (agarcl_batch_set_task_sizes): its A + b players keep the player-order check.  0 when mode 0 is not in the set.
uint64_t task_bot_counts(const agarcl_cfg* c, const agarcl_layout* L);
