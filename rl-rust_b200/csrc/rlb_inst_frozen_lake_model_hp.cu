// rlb_inst_frozen_lake_model_hp.cu — k_run_hp with the Dyna model attached (per-agent hyper-parameter sets, per-set planning counts) for RLB_ENV_FROZEN_LAKE (see rlb_launch.h).
#include "rlb_launch_impl.cuh"
namespace rlb { RLB_INSTANTIATE_ENV_MODEL_HP(RLB_ENV_FROZEN_LAKE) }
