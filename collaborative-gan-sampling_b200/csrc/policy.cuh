// sampling/policy.py:26-64 as device functions shared by the standalone policy kernel and the fused 2-D refiner.
// Every operation is rounded separately (no FMA contraction) and constants are rounded to FP32 from the python
// doubles exactly where numpy would, so that given identical inputs the update is bit-identical to the reference.
#pragma once
#include "cgs.h"

namespace cgs {

struct PolicyConsts {
  int method;
  float step;       // lambda_
  float alpha;      // alpha_
  float b1, b1c;    // beta1_, (1. - beta1_)
  float b2, b2c;
  float b3, b3c;
  float eps;
};

inline PolicyConsts make_policy_consts(const cgs_policy_cfg& c) {
  PolicyConsts k;
  k.method = c.method;
  k.step = (float)c.step_size;
  k.alpha = (float)c.alpha;
  k.b1 = (float)c.beta1;  k.b1c = (float)(1.0 - c.beta1);
  k.b2 = (float)c.beta2;  k.b2c = (float)(1.0 - c.beta2);
  k.b3 = (float)c.beta3;  k.b3c = (float)(1.0 - c.beta3);
  k.eps = (float)c.eps;
  return k;
}

// policy.py:27-29
__device__ __forceinline__ float sgd_update(const PolicyConsts& c, float theta, float g) {
  return __fsub_rn(theta, __fmul_rn(c.step, g));
}
// policy.py:31-37
__device__ __forceinline__ float momentum_update(const PolicyConsts& c, float theta, float g, float& m, int first) {
  m = first ? __fmul_rn(c.step, g) : __fadd_rn(__fmul_rn(c.alpha, m), __fmul_rn(c.step, g));
  return __fsub_rn(theta, m);
}
// policy.py:47-50
__device__ __forceinline__ float ladam_loss_avg(const PolicyConsts& c, float avg, float loss, int first) {
  return first ? loss : __fadd_rn(__fmul_rn(c.b3, avg), __fmul_rn(c.b3c, loss));
}
// policy.py:39-46 and :61 (numpy branch; clip_hi adds the 1e4 bound of the TF branch :56)
__device__ __forceinline__ float ladam_update(const PolicyConsts& c, float theta, float g, float& m, float& v,
                                              float loss_avg, int first, int clip_hi) {
  const float g2 = __fmul_rn(g, g);
  m = first ? g : __fadd_rn(__fmul_rn(c.b1, m), __fmul_rn(c.b1c, g));
  v = first ? g2 : __fadd_rn(__fmul_rn(c.b2, v), __fmul_rn(c.b2c, g2));
  float r = fmaxf(__fadd_rn(loss_avg, 0.5f), 0.0f);
  if (clip_hi) r = fminf(r, 10000.0f);
  const float r2 = __fmul_rn(r, r);                                        // ** degree_ (= 2)
  const float dx = __fdiv_rn(__fmul_rn(c.step, m), __fadd_rn(__fsqrt_rn(v), c.eps));
  return __fsub_rn(theta, __fmul_rn(dx, r2));
}

// the discriminator's score (synthetic/GAN.py:108), shared by every form of the 2-D refiner so they agree bit for bit
__device__ __forceinline__ float sigmoid_f32(float l) { return 1.f / (1.f + expf(-l)); }

}  // namespace cgs
