// Split-residual instantiations (runs/71081, V3g), element type __nv_bfloat16: the V3c kernels (per-input norms + lambdas) that also
// write x0t = nrm(t) and x0b = C'_n, and whose recompute backward takes their gradients (kModeSplitResidual).  Widths of
// the V3c fast path: 512 and 1024 columns.
#include "mot_embed_kernels.cuh"
namespace mot {
int dispatch_fwd_resid_bf16(const EmbedParams& p, cudaStream_t s) {
  using T = __nv_bfloat16;
  if (p.Do == 512) return launch_fwd<T, 2, kModeSplitResidual>(p, s);
  if (p.Do == 1024) return launch_fwd<T, 4, kModeSplitResidual>(p, s);
  return MOT_ERR_UNSUPPORTED;
}
int dispatch_bwd_resid_bf16(const EmbedParams& p, cudaStream_t s) {
  using T = __nv_bfloat16;
  if (p.Do == 512) return launch_bwd<T, 4, kModeSplitResidual>(p, s);
  if (p.Do == 1024) return launch_bwd<T, 8, kModeSplitResidual>(p, s);
  return MOT_ERR_UNSUPPORTED;
}
}  // namespace mot
