// rlb_inst_blackjack_hp.cu — k_run_hp and the _hp step kernels (per-agent hyper-parameter sets) for RLB_ENV_BLACKJACK (see rlb_launch.h).
#include "rlb_launch_impl.cuh"
namespace rlb { RLB_INSTANTIATE_ENV_HP(RLB_ENV_BLACKJACK) }
