// macm_kernels_huge.cu -- the step kernels of sims that asked for more than 240 touching contacts per env
// (macm_params.max_touching > 240, macm_buffers.touch_scratch): macm_kernels.cu compiled a second time with the
// global-memory solver stage in (GmemStage, dense_solve_velocity_huge / dense_solve_position_huge).  A translation
// unit of its own so that ptxas allocates the default kernels' registers exactly as without it: their 72-register,
// zero-spill allocation does not survive ANY call added to their body, not even one under `if constexpr` in a sibling
// instantiation (measured; each spilled variant cost 2 % of the headline).  Exports macm_launch_step_huge /
// macm_prepare_kernels_huge.
#define MACM_HUGE_TU 1
#include "macm_kernels.cu"
