// gpvar_fused_kernel instantiations: m25 (see gpvar.cuh)
#include "gpvar.cuh"
namespace basq {
int launch_gpvar_fused_m25(basq_ctx* ctx, const KParams& kp, const GpfDev& dev) {
  return launch_gpvar_fused_family<BASQ_MATERN25>(ctx, kp, dev);
}
}  // namespace basq
