// le_td3_api.h — entry points of le_td3.cu used by le_api.cu
#pragma once
#include "le_inner_loop.cuh"

namespace le {
// shapes of the maxima configuration tc: slot floats, minibatch rows and parameter counts (the init / final row strides)
struct Td3Plan { int grid, bmax, rowf, p_actor, p_critic; int64_t slot_floats; };
int td3_plan(const le_td3_cfg* tc, int n_lanes, int ring_cap, int sms, Td3Plan* tp);
// lane i runs cfg_dev[n_cfg == 1 ? 0 : i]; tp.grid resident lanes; null init pointers: device init from P_TD3_INIT
cudaError_t td3_launch(const le_td3_cfg* cfg_dev, int n_cfg, const le_td3_cfg* cfg_host0, const RunParams& rp, float* slots, const Td3Plan& tp,
                       const float* actor_init, const float* c1_init, const float* c2_init, int per_lane_init, float* actor_final, cudaStream_t st);
}  // namespace le
