// One per-episode condition (aom_condition): the common value, and while per-environment values are in force their
// device array [E] and its host copy (both null otherwise).  Host readers take at(e); kernels take dev or common.
// The context keeps the only store of them, EnvCond cond[aom_condition][layer] (layer 0 for those of the sensor and the
// controller), which the atmosphere and the controller read through a pointer.
#pragma once

struct EnvCond {
  float common;
  float* dev;
  float* host;
  float at(int e) const { return host ? host[e] : common; }
};
