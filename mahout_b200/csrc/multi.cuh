// multi.cuh -- the one-process multi-GPU handle (mb200_create_multi, csrc/job.cu) and the host helpers shared by
// the calls that drive it: the item-similarity job (job.cu) and the replicated sized bank (sized_multi.cu).
#pragma once

#include <chrono>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"

struct mb200_multi {
  int n = 0;
  std::vector<int> devices;
  std::vector<mb200_ctx*> ctx;
  std::string err;
  std::mutex mu;  // one call at a time per handle
};

static inline double multi_now_s() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

static inline int multi_fail(mb200_multi* m, int code, const std::string& msg) {
  if (m) m->err = msg;
  mb200_set_global_error(msg.c_str());
  return code;
}
