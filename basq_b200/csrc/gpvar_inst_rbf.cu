// gpvar_fused_kernel instantiations: rbf (see gpvar.cuh)
#include "gpvar.cuh"
namespace basq {
int launch_gpvar_fused_rbf(basq_ctx* ctx, const KParams& kp, const GpfDev& dev) {
  return launch_gpvar_fused_family<BASQ_RBF>(ctx, kp, dev);
}
}  // namespace basq
