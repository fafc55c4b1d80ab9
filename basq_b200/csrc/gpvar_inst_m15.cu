// gpvar_fused_kernel instantiations: m15 (see gpvar.cuh)
#include "gpvar.cuh"
namespace basq {
int launch_gpvar_fused_m15(basq_ctx* ctx, const KParams& kp, const GpfDev& dev) {
  return launch_gpvar_fused_family<BASQ_MATERN15>(ctx, kp, dev);
}
}  // namespace basq
