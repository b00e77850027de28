// The sampler update of one mel bin, shared by k_ddpm_update / k_plms_update (fp32 path), k_tc_head and k_tc_stack.  Written
// in the reference's fp32 operation order with __f*_rn (no FMA contraction): that order keeps the fp32 path bit-exact to the
// reference and the tensor-core paths inside their bounds.  Loads, noise draws and stores stay with the callers.
#pragma once
#include "dsx_internal.h"

namespace dsx {

// p_sample after the network (usr/diff/shallow_diffusion_tts.py:134-166): x_recon = A*x - Bc*eps; clamp;
// mean = c1*x_recon + c2*x; + sigma*z
__device__ __forceinline__ float ddpm_step(const DdpmCoef& c, float x, float eps, float z) {
  float xr = __fsub_rn(__fmul_rn(c.A, x), __fmul_rn(c.Bc, eps));
  xr = fminf(fmaxf(xr, -1.f), 1.f);
  const float mean = __fadd_rn(__fmul_rn(c.c1, xr), __fmul_rn(c.c2, x));
  return __fadd_rn(mean, __fmul_rn(c.sigma, z));
}

// PLMS (shallow_diffusion_tts.py:174-199): eps' = (w0*eps + w1*h1 + w2*h2 + w3*h3) / denom, left to right over the history
// terms that are present (u1..u3); get_x_pred: x + a_diff * (kx*x - ke*eps')
__device__ __forceinline__ float plms_step(const PlmsCoef& c, float x, float eps, float h1, float h2, float h3, bool u1, bool u2,
                                           bool u3) {
  float comb = __fmul_rn(c.w0, eps);
  if (u1) comb = __fadd_rn(comb, __fmul_rn(c.w1, h1));
  if (u2) comb = __fadd_rn(comb, __fmul_rn(c.w2, h2));
  if (u3) comb = __fadd_rn(comb, __fmul_rn(c.w3, h3));
  const float ep = __fdiv_rn(comb, c.denom);
  const float inner = __fsub_rn(__fmul_rn(c.kx, x), __fmul_rn(c.ke, ep));
  return __fadd_rn(x, __fmul_rn(c.a_diff, inner));
}

}  // namespace dsx
