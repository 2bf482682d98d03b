// Split-residual instantiations (runs/71081, V3g), element type float: the V3c kernels (per-input norms + lambdas) that also
// write x0t = nrm(t) and x0b = C'_n (the run-time-flag kernel, which the fp32 V3c launch runs: kModeSplitResidualRT), and
// whose recompute backward takes their gradients (kModeSplitResidual).  Widths 512 and 1024 columns, as for bf16.
#include "mot_embed_kernels.cuh"
namespace mot {
int dispatch_fwd_resid_f32(const EmbedParams& p, cudaStream_t s) {
  using T = float;
  if (p.Do == 512) return launch_fwd<T, 2, kModeSplitResidualRT>(p, s);
  if (p.Do == 1024) return launch_fwd<T, 4, kModeSplitResidualRT>(p, s);
  return MOT_ERR_UNSUPPORTED;
}
int dispatch_bwd_resid_f32(const EmbedParams& p, cudaStream_t s) {
  using T = float;
  if (p.Do == 512) return launch_bwd<T, 4, kModeSplitResidual>(p, s);
  if (p.Do == 1024) return launch_bwd<T, 8, kModeSplitResidual>(p, s);
  return MOT_ERR_UNSUPPORTED;
}
}  // namespace mot
