// The per-timestep head formulas of the objective: DiagGauss and Categorical surrogate / KL / entropy and their
// gradients, the squared error of the value head, and the Fisher metric of each head (trpo.py:37-63,
// ppo.py:35-49, core.py:339-365,402-438,613-617).  Every kernel path that runs layers >= 2 computes its head with
// these functions, so the numerics of the objective are written once:
//   - per-element terms, used by the register chains of mlp_chain.cu in the mma fragment layout;
//   - row functions over the tile layout ([feature][MRL_LDT], one thread per timestep), used by mid_* (mlp_mid.cu)
//     and the layer-by-layer heads (mlp_layers.cu).
#pragma once
#include "common.cuh"

#define MRL_LOG_2PIE 2.8378770664093453f   // log(2 pi e): DiagGauss entropy = sum log sigma + d/2 log(2 pi e)
#define MRL_MAX_DOUT 64                    // outputs of a net (mrl_net_create rejects more)

// ---- per-element terms (one action dimension / one class of one timestep)
// DiagGauss logp - oldlogp, term by term
__device__ __forceinline__ float gauss_logratio(float mu, float ac, float m0, float s0, float sg) {
  const float t = (ac - mu) / sg, t0 = (ac - m0) / s0;
  return -0.5f * (t - t0) * (t + t0) - log1pf((sg - s0) / s0);   // log1pf(..) = log(sigma / sigma0)
}
// DiagGauss KL(old || new) (reverse_kl: KL(new || old), ppo.py:40-41):
// log(s1/s0) + (s0^2 + dm^2)/(2 s1^2) - 1/2, with the s0 ~ s1 cancellation taken analytically
// = g(u) + u^2/2 + dm^2/(2 s1^2), u = (s0-s1)/s1   (reverse: roles of s0, s1 swapped)
__device__ __forceinline__ float gauss_kl(float mu, float m0, float s0, float sg, int reverse_kl) {
  const float dm = m0 - mu;
  const float den = reverse_kl ? s0 : sg;
  const float u = (reverse_kl ? (sg - s0) : (s0 - sg)) / den;
  return u_minus_log1p(u) + 0.5f * (u * u + (dm / den) * (dm / den));
}
// DiagGauss gradient of  w * ratio + ck * kl  (w = -ratio * adv * cs): d_mu = d/dmu, d_ls = d/dlogstd.  iv = 1/sigma^2
__device__ __forceinline__ void gauss_grad(float mu, float ac, float m0, float s0, float sg, float iv, float w, float ck,
                                           int reverse_kl, float& d_mu, float& d_ls) {
  const float t2 = (ac - mu) * (ac - mu) * iv;
  float dkl_dmu, dkl_dls;
  if (!reverse_kl) {
    dkl_dmu = (mu - m0) * iv;
    dkl_dls = ((sg - s0) * (sg + s0) - (m0 - mu) * (m0 - mu)) * iv;   // 1 - (s0^2+dm^2)/s1^2
  } else {
    const float i0 = 1.f / (s0 * s0);
    dkl_dmu = (mu - m0) * i0;
    dkl_dls = (sg - s0) * (sg + s0) * i0;                              // -1 + s1^2/s0^2
  }
  d_mu = w * (ac - mu) * iv + ck * dkl_dmu;
  d_ls = w * (t2 - 1.f) + ck * dkl_dls;
}
// Categorical KL term of one class, p = new, p0 = old probability:
// q log(q/w) = q g(v) - (w - q), v = (w-q)/q : no cancellation between the terms of the sum
__device__ __forceinline__ float cat_kl(float p, float p0, int reverse_kl) {
  const float q = reverse_kl ? p : p0, w = reverse_kl ? p0 : p;
  return q * u_minus_log1p((w - q) / q) - (w - q);
}
// Categorical dL/dlogit of one class: w = -(pa / p0a) * adv * cs, hot = the class is the action taken,
// klrow = sum_j p log(p / p0) of the row (reverse KL only)
__device__ __forceinline__ float cat_grad(float p, float p0, float w, float ck, float klrow, bool hot, int reverse_kl) {
  const float dk = reverse_kl ? p * (logf(p / p0) - klrow) : (p - p0);
  return w * ((hot ? 1.f : 0.f) - p) + ck * dk;
}
// PPO clipped surrogate of one row, r = pi / pi_old (the ratio the surrogate forms above): the row's share of the
// objective min(r A, clip(r, 1 - eps, 1 + eps) A).  eps = +inf: r A.
__device__ __forceinline__ float clip_objective(float r, float adv, float eps) {
  return fminf(r * adv, fminf(fmaxf(r, 1.f - eps), 1.f + eps) * adv);
}
// the row's gradient is cut off where the clipped branch is the smaller one, outside the inclusive clip range (the
// derivative torch autograd takes of torch.minimum(r A, torch.clamp(r, 1 - eps, 1 + eps) A); a tie passes it).
// Ungated rows carry the surrogate's gradient, weight w = -r A, with no KL term.
__device__ __forceinline__ bool clip_gated(float r, float adv, float eps) {
  return (adv > 0.f && r > 1.f + eps) || (adv < 0.f && r < 1.f - eps);
}
// the row counts towards clipfrac: r outside [1 - eps, 1 + eps]
__device__ __forceinline__ bool clip_outside(float r, float eps) { return r < 1.f - eps || r > 1.f + eps; }
// a valid row of the clipped objective: its term added to the surrogate sum, counted in s_clip when outside the range
__device__ __forceinline__ void clip_row(float r, float adv, float eps, double& s_surr, double& s_clip) {
  s_surr += (double)clip_objective(r, adv, eps);
  s_clip += clip_outside(r, eps) ? 1.0 : 0.0;
}

// value head: squared error against the target y, and its derivative d/dpred
__device__ __forceinline__ double value_sqerr(float y, float pred) {
  const float df = y - pred;
  return (double)df * (double)df;
}
__device__ __forceinline__ float value_dpred(float pred, float y) { return 2.f * (pred - y); }

// ---- row functions: timestep r of a tile.  H / E = the head rows [dL][MRL_LDT] of the tile; aux = the side-input
// rows at timestep r (adv | actions | old mean | old std, or adv | action | old probs, or the value target), nullptr
// when there are no losses; valid = r is a timestep of the batch, not padding.  sig, logsig, ivar = sigma, log sigma
// and 1/sigma^2 per dimension (DiagGauss).

// Forward: the Categorical probabilities rewritten in place of the logits; the row's surr / kl / ent added to the sums.
// CLIP: surr takes the clipped objective of the row (clip range eps) and s_clip counts the rows outside the range.
template <int HEAD, bool CLIP = false>
__device__ __forceinline__ void head_fwd_row(float* H, const float* aux, int r, int dL, bool valid, int reverse_kl,
                                             const float* sig, const float* logsig, double& s_surr, double& s_kl,
                                             double& s_ent, float eps, double& s_clip) {
  if (HEAD == MRL_HEAD_GAUSS) {
    if (aux) {
      const float adv = aux[0];
      float dl = 0.f, kl = 0.f, sls = 0.f;
      for (int j = 0; j < dL; ++j) {
        const float mu = H[j * MRL_LDT + r];
        const float ac = aux[(1 + j) * MRL_LDT];
        const float m0 = aux[(1 + dL + j) * MRL_LDT];
        const float s0 = aux[(1 + 2 * dL + j) * MRL_LDT];
        const float sg = sig[j];
        dl += gauss_logratio(mu, ac, m0, s0, sg);
        kl += gauss_kl(mu, m0, s0, sg, reverse_kl);
        sls += logsig[j];
      }
      if (valid) {
        if constexpr (CLIP) clip_row(expf(dl), adv, eps, s_surr, s_clip);
        else s_surr += (double)(expf(dl) * adv);
        s_kl += (double)kl;
        s_ent += (double)(sls + 0.5f * MRL_LOG_2PIE * dL);
      }
    }
  } else if (HEAD == MRL_HEAD_CAT) {
    float m = -INFINITY;
    for (int j = 0; j < dL; ++j) m = fmaxf(m, H[j * MRL_LDT + r]);
    float s = 0.f;
    for (int j = 0; j < dL; ++j) {
      const float e = expf(H[j * MRL_LDT + r] - m);
      H[j * MRL_LDT + r] = e;
      s += e;
    }
    const float inv = 1.f / s;
    float kl = 0.f, ent = 0.f, pa = 1.f, p0a = 1.f;
    const int ai = aux ? (int)aux[1 * MRL_LDT] : 0;
    for (int j = 0; j < dL; ++j) {
      const float p = H[j * MRL_LDT + r] * inv;
      H[j * MRL_LDT + r] = p;
      if (aux) {
        const float p0 = aux[(2 + j) * MRL_LDT];
        kl += cat_kl(p, p0, reverse_kl);
        ent -= p * logf(p);
        if (j == ai) { pa = p; p0a = p0; }
      }
    }
    if (aux && valid) {
      if constexpr (CLIP) clip_row(pa / p0a, aux[0], eps, s_surr, s_clip);
      else s_surr += (double)((pa / p0a) * aux[0]);
      s_kl += (double)kl;
      s_ent += (double)ent;
    }
  } else if (aux && valid) {
    s_surr += value_sqerr(aux[0], H[r]);
  }
}

// Backward, E holding the head's input rows.  Gradient mode: E = delta_L (un-normalised; 1/N is applied by the slab
// reduce) and, DiagGauss, the logstd partial added to GL[j * MRL_TILE + r]; cs, ck = the coefficients of the surrogate
// and the KL.  Clipped-gradient mode: the same for the clipped objective (clip range eps), zeros for a gated row.
// Fvp mode: E = Rz_L, replaced by the Fisher metric applied to it.  Padded timesteps give zeros.
template <int HEAD, int MODE>
__device__ __forceinline__ void head_bwd_row(const float* H, float* E, float* GL, const float* aux, int r, int dL,
                                             bool valid, int reverse_kl, float cs, float ck, const float* sig,
                                             const float* ivar, float eps = 0.f) {
  if (MODE == MRL_MODE_FVP) {
    if (HEAD == MRL_HEAD_GAUSS) {          // M = diag(1/sigma^2) on the mean block
      for (int j = 0; j < dL; ++j) E[j * MRL_LDT + r] = valid ? E[j * MRL_LDT + r] * ivar[j] : 0.f;
    } else if (HEAD == MRL_HEAD_CAT) {     // M = diag(p) - p p^T
      float s = 0.f;
      for (int j = 0; j < dL; ++j) s += H[j * MRL_LDT + r] * E[j * MRL_LDT + r];
      for (int j = 0; j < dL; ++j) {
        const float p = H[j * MRL_LDT + r];
        E[j * MRL_LDT + r] = valid ? p * (E[j * MRL_LDT + r] - s) : 0.f;
      }
    } else {
      for (int j = 0; j < dL; ++j)
        if (!valid) E[j * MRL_LDT + r] = 0.f;
    }
  } else if (!valid) {
    for (int j = 0; j < dL; ++j) E[j * MRL_LDT + r] = 0.f;
  } else if (HEAD == MRL_HEAD_GAUSS) {
    const float adv = aux[0];
    float dl = 0.f;
    for (int j = 0; j < dL; ++j) {
      const float mu = H[j * MRL_LDT + r];
      const float ac = aux[(1 + j) * MRL_LDT];
      const float m0 = aux[(1 + dL + j) * MRL_LDT];
      const float s0 = aux[(1 + 2 * dL + j) * MRL_LDT];
      dl += gauss_logratio(mu, ac, m0, s0, sig[j]);
    }
    if constexpr (MODE == MRL_MODE_GRAD_CLIP) {
      const float rt = expf(dl);
      if (clip_gated(rt, adv, eps)) {
        for (int j = 0; j < dL; ++j) E[j * MRL_LDT + r] = 0.f;
        return;
      }
      cs = 1.f;
      ck = 0.f;
    }
    const float w = -expf(dl) * adv * cs;
    for (int j = 0; j < dL; ++j) {
      const float mu = H[j * MRL_LDT + r];
      const float ac = aux[(1 + j) * MRL_LDT];
      const float m0 = aux[(1 + dL + j) * MRL_LDT];
      const float s0 = aux[(1 + 2 * dL + j) * MRL_LDT];
      float d_mu, d_ls;
      gauss_grad(mu, ac, m0, s0, sig[j], ivar[j], w, ck, reverse_kl, d_mu, d_ls);
      E[j * MRL_LDT + r] = d_mu;
      GL[j * MRL_TILE + r] += d_ls;
    }
  } else if (HEAD == MRL_HEAD_CAT) {
    const float adv = aux[0];
    const int ai = (int)aux[1 * MRL_LDT];
    const float pa = H[ai * MRL_LDT + r], p0a = aux[(2 + ai) * MRL_LDT];
    if constexpr (MODE == MRL_MODE_GRAD_CLIP) {
      if (clip_gated(pa / p0a, adv, eps)) {
        for (int j = 0; j < dL; ++j) E[j * MRL_LDT + r] = 0.f;
        return;
      }
      cs = 1.f;
      ck = 0.f;
      reverse_kl = 0;
    }
    const float w = -(pa / p0a) * adv * cs;
    float klrow = 0.f;
    if (reverse_kl)
      for (int j = 0; j < dL; ++j) {
        const float p = H[j * MRL_LDT + r];
        klrow += p * logf(p / aux[(2 + j) * MRL_LDT]);
      }
    for (int j = 0; j < dL; ++j)
      E[j * MRL_LDT + r] = cat_grad(H[j * MRL_LDT + r], aux[(2 + j) * MRL_LDT], w, ck, klrow, j == ai, reverse_kl);
  } else {
    E[r] = value_dpred(H[r], aux[0]);
  }
}
