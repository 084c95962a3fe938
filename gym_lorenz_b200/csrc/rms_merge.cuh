// Chan et al. parallel update of one (mean, var) component of a running mean / variance with one batch's
// shifted sums -- SB3 RunningMeanStd.update_from_moments (stable_baselines3/common/running_mean_std.py), the
// same operations in the same order.  cl_rms_update (tu_rl_ops.cu) and the training-mode fused collector
// (tu_policy.cu) both merge with it, so the collector's statistics are bit-identical to DeviceVecNormalize's;
// both translation units are built with -fmad=false.
//   acc1 = sum(x - mean), acc2 = sum((x - mean)^2) over the batch's n rows; cnt = the running count before it
#pragma once

__device__ __forceinline__ void rms_merge(double& mean, double& var, const double cnt, const double n,
                                          const double& acc1, const double& acc2) {
  const double tot = cnt + n;
  const double d1 = acc1 / n;                     // batch_mean - mean
  const double batch_var = acc2 / n - d1 * d1;
  const double batch_mean = mean + d1;
  const double delta = batch_mean - mean;
  const double new_mean = mean + delta * n / tot;
  const double m2 = var * cnt + batch_var * n + delta * delta * cnt * n / tot;
  mean = new_mean;
  var = m2 / tot;
}
