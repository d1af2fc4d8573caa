// K4 instantiation for the "pack" sample-side form that ppo_loss_pair.cu does not take (see ppo_loss.cuh).
#include "ppo_loss.cuh"

namespace srl {
namespace loss {
// One lane per thread and the general configuration only: with a pack, the four-lane conditions (n % 4 == 0, row strides
// % 4 == 0, 16-byte aligned policy-side tensors and lane_idx) imply the pair kernel's (even n and strides, 8-byte
// alignment), so every pack call that could run four lanes per thread runs ppo_loss_pair_kernel instead.
int launch_loss_pack(LossBatch& b, int n_problems, cudaStream_t st) {
  return LossLauncher<1, kPack, RuntimeCfg>::launch(b, n_problems, st);
}
}  // namespace loss
}  // namespace srl
