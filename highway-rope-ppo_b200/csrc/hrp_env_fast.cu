// hrp_env_fast.cu -- the highway-fast-v0 step kernels (hrp_cfg.ego_collisions_only = 1; DESIGN.md Appendix C).
//
// hrp_env.cu compiled a second time, as its own translation unit, with the ego-only collision pass of simulate_frame
// switched on: the eight step kernels (fp32 / fp64 x with and without final_obs x Kinematics / OccupancyGrid) and
// hrp_launch_step_ego.  Reset, observe and embed have no collisions and stay in hrp_env.cu.
#define HRP_ENV_FAST_TU
#include "hrp_env.cu"
