// K4: fused dense optimizer update + L2 over the whole parameter arena in one launch (sm_100a, HBM-bound).
//
// Replaces (reference, DRecPy/): Recommender/recommender_abc.py:328-334 (one optimizer.apply_gradients per
// variable => the step counter advances once per variable, SURVEY.md Q2), the dense update of the Keras optimizer
// (recommender_abc.py:153, Adam by default; the per-kind rules are restated in update1 below and in oracle/optim.py), and
// the L2 terms of Recommender/cdae.py:81-82 (reg/B * l2_loss) / Keras regularizers.l2 (dmf.py:47), whose gradient is
// folded into g here and whose value (at the pre-update weights) is reduced into reg_part for the reported loss.
// One body, instantiated per update rule: the segment walk, the L2 fold, the row_mask skip, the reg_part reduction and
// the fused loss finalisation are shared; only the per-element rule and the state arrays it reads differ.
#include "kernels.h"

#include <cmath>

namespace {

constexpr int kAdamThreads = 256;

// state arrays an update rule reads and writes: m = a.m, v = a.v, x = e.x (the third arena)
__host__ __device__ constexpr bool uses_m(int k) { return k != OPT_SGD; }
__host__ __device__ constexpr bool uses_v(int k) {
  return k == OPT_ADAM || k == OPT_RMSPROP_CENTERED || k == OPT_RMSPROP_MOMENTUM || k == OPT_RMSPROP_CENTERED_MOMENTUM ||
         k == OPT_ADAMAX || k == OPT_AMSGRAD;
}
__host__ __device__ constexpr bool uses_x(int k) { return k == OPT_RMSPROP_CENTERED_MOMENTUM || k == OPT_AMSGRAD; }

// One element of every rule but Adam (whose statements stay inline in k_update, as they always were).  g already holds
// the L2 term; alpha is the segment's host-computed step size (lr_t, or lr_t / (1 - beta1^t) for Adamax, alpha_t for
// AMSGrad).  Keras-2 / TF 2.0-2.3 OptimizerV2 dense kernels, fp32.
template <int K>
__device__ __forceinline__ void update1(const AdamArgs& a, const OptimExtra& e, float alpha, float g, float& w, float& m,
                                        float& v, float& x) {
  if (K == OPT_SGD) {                               // ResourceApplyGradientDescent
    w -= alpha * g;
  } else if (K == OPT_SGD_MOMENTUM) {               // ResourceApplyKerasMomentum: m = accumulator
    m = m * e.momentum - alpha * g;
    w += e.nesterov ? m * e.momentum - alpha * g : m;
  } else if (K == OPT_RMSPROP || K == OPT_RMSPROP_CENTERED) {   // RMSprop._resource_apply_dense, momentum == 0
    m = e.rho * m + (1.0f - e.rho) * (g * g);       // m = ms, v = mg
    float d = m;
    if (K == OPT_RMSPROP_CENTERED) {
      v = e.rho * v + (1.0f - e.rho) * g;
      d = m - v * v;
    }
    w -= alpha * g / (sqrtf(d) + a.eps);
  } else if (K == OPT_RMSPROP_MOMENTUM || K == OPT_RMSPROP_CENTERED_MOMENTUM) {   // (Centered)ApplyRMSProp: eps in the sqrt
    m += (g * g - m) * (1.0f - e.rho);              // m = ms, v = mom (plain) / mg (centered, mom in x)
    float d = m + a.eps;
    float& mom = K == OPT_RMSPROP_CENTERED_MOMENTUM ? x : v;
    if (K == OPT_RMSPROP_CENTERED_MOMENTUM) {
      v += (g - v) * (1.0f - e.rho);
      d = m - v * v + a.eps;
    }
    mom = mom * e.momentum + alpha * g / sqrtf(d);
    w -= mom;
  } else if (K == OPT_ADAGRAD) {                    // ResourceApplyAdagradV2: m = accumulator
    m += g * g;
    w -= alpha * g / (sqrtf(m) + a.eps);
  } else if (K == OPT_ADAMAX) {                     // ResourceApplyAdaMax: m, v = u
    m += (g - m) * (1.0f - a.beta1);
    v = fmaxf(a.beta2 * v, fabsf(g));
    w -= alpha * (m / (v + a.eps));
  } else if (K == OPT_AMSGRAD) {                    // ResourceApplyAdamWithAmsgrad: m, v, x = vhat
    m += (g - m) * (1.0f - a.beta1);
    v += (g * g - v) * (1.0f - a.beta2);
    x = fmaxf(x, v);
    w -= m * alpha / (sqrtf(x) + a.eps);
  }
}

__device__ __forceinline__ OptimExtra optim_extra() { return OptimExtra{}; }
__device__ __forceinline__ OptimExtra optim_extra(const OptimExtra& e) { return e; }

// K4 for update rule K.  Adam's instantiation takes no OptimExtra argument: its kernel keeps the (AdamArgs, total4)
// signature and, statement for statement, the body it always had (its SASS is that of the former k_adam).  The
// profiler names are k_adam and k_optim_<rule> (optim_kernel_name).
template <int K, typename... Extra>
__global__ void __launch_bounds__(kAdamThreads) k_update(AdamArgs a, int64_t total4, Extra... extra) {
  const OptimExtra e = optim_extra(extra...);
  __shared__ float sred[kAdamThreads];
  float reg = 0.f;
  const float omb1 = 1.0f - a.beta1, omb2 = 1.0f - a.beta2;
  for (int64_t i = a.seg[0].off4 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4;
       i += (int64_t)gridDim.x * blockDim.x) {
    int s = 0;
#pragma unroll 1
    while (s + 1 < a.nseg && i >= a.seg[s + 1].off4) s++;
    if (i >= a.seg[s].off4 + a.seg[s].n4) continue;  // alignment gap between segments
    const float alpha = a.alpha_dev ? __ldg(a.alpha_dev + a.seg[s].alpha_idx) : a.seg[s].alpha;
    const float l2 = a.seg[s].l2, regw = a.seg[s].regw;
    float4 w = reinterpret_cast<float4*>(a.w)[i];
    float4 m = make_float4(0.f, 0.f, 0.f, 0.f), v = m, x = m;
    if (uses_m(K)) m = reinterpret_cast<float4*>(a.m)[i];
    if (uses_v(K)) v = reinterpret_cast<float4*>(a.v)[i];
    if (uses_x(K)) x = reinterpret_cast<float4*>(e.x)[i];
    float4 g0 = make_float4(0.f, 0.f, 0.f, 0.f);
    bool read_g = true;
    if (s == a.row_seg) {          // rows of this table without a gradient this step hold zeros: do not read them
      const uint32_t row = (uint32_t)(i - a.seg[s].off4) / (uint32_t)a.row_len4;
      read_g = (__ldg(a.row_mask + (row >> 5)) >> (row & 31)) & 1u;
    }
    if (read_g) g0 = __ldg(reinterpret_cast<const float4*>(a.g) + i);
    reg += regw * (w.x * w.x + w.y * w.y + w.z * w.z + w.w * w.w);
    if (K == OPT_ADAM) {
#define DRB_ADAM1(c)                                           \
    {                                                          \
      const float g = g0.c + l2 * w.c;                         \
      m.c += (g - m.c) * omb1;                                 \
      v.c += (g * g - v.c) * omb2;                             \
      w.c -= alpha * m.c / (sqrtf(v.c) + a.eps);               \
    }
      DRB_ADAM1(x) DRB_ADAM1(y) DRB_ADAM1(z) DRB_ADAM1(w)
#undef DRB_ADAM1
    } else {
      update1<K>(a, e, alpha, g0.x + l2 * w.x, w.x, m.x, v.x, x.x);
      update1<K>(a, e, alpha, g0.y + l2 * w.y, w.y, m.y, v.y, x.y);
      update1<K>(a, e, alpha, g0.z + l2 * w.z, w.z, m.z, v.z, x.z);
      update1<K>(a, e, alpha, g0.w + l2 * w.w, w.w, m.w, v.w, x.w);
    }
    reinterpret_cast<float4*>(a.w)[i] = w;
    if (uses_m(K)) reinterpret_cast<float4*>(a.m)[i] = m;
    if (uses_v(K)) reinterpret_cast<float4*>(a.v)[i] = v;
    if (uses_x(K)) reinterpret_cast<float4*>(e.x)[i] = x;
  }
  sred[threadIdx.x] = reg;
  __syncthreads();
  for (int s = kAdamThreads / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) sred[threadIdx.x] += sred[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) a.reg_part[blockIdx.x] = sred[0];
  if (!a.fin_loss_out) return;
  // fused loss finalisation: the last block to get here sums the loss terms and the regularisation partials
  __shared__ bool last;
  __shared__ double sa[kAdamThreads], sb[kAdamThreads];
  if (threadIdx.x == 0) {
    __threadfence();
    last = atomicInc(a.fin_ticket, gridDim.x - 1) == gridDim.x - 1;      // wraps to 0: ready for the next launch
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  const int n_reg = a.fin_n_reg > 0 ? a.fin_n_reg : (int)gridDim.x;
  double la = 0.0, lb = 0.0;
  for (int i = threadIdx.x; i < a.fin_n_loss; i += kAdamThreads) la += (double)__ldcg(a.fin_loss_part + i);
  const float* regs = a.fin_reg_part ? a.fin_reg_part : a.reg_part;
  for (int i = threadIdx.x; i < n_reg; i += kAdamThreads) lb += (double)__ldcg(regs + i);
  sa[threadIdx.x] = la;
  sb[threadIdx.x] = lb;
  __syncthreads();
  for (int s = kAdamThreads / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      sa[threadIdx.x] += sa[threadIdx.x + s];
      sb[threadIdx.x] += sb[threadIdx.x + s];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    a.fin_loss_out[0] = (float)(sa[0] * (double)a.fin_scale) + (float)sb[0];
    a.fin_loss_out[1] = (float)(sa[0] * (double)a.fin_scale);
  }
}

__global__ void __launch_bounds__(256) k_finalize_loss(const float* __restrict__ loss_part, int n_loss, float scale,
                                                       const float* __restrict__ reg_part, int n_reg,
                                                       float* __restrict__ loss_out) {
  __shared__ double sa[256], sb[256];
  double la = 0.0, lb = 0.0;
  for (int i = threadIdx.x; i < n_loss; i += 256) la += (double)loss_part[i];
  for (int i = threadIdx.x; i < n_reg; i += 256) lb += (double)reg_part[i];
  sa[threadIdx.x] = la;
  sb[threadIdx.x] = lb;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      sa[threadIdx.x] += sa[threadIdx.x + s];
      sb[threadIdx.x] += sb[threadIdx.x + s];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    loss_out[0] = (float)(sa[0] * (double)scale) + (float)sb[0];   // reported loss: batch term + regularisation
    loss_out[1] = (float)(sa[0] * (double)scale);                  // batch term alone (summed over ranks when data parallel)
  }
}

struct Scalars8 { float v[8]; };
__global__ void k_set_scalars(float* __restrict__ dst, Scalars8 s, int n) {
  if ((int)threadIdx.x < n) dst[threadIdx.x] = s.v[threadIdx.x];
}

}  // namespace

int launch_set_scalars(drb_ctx* ctx, float* dst, const float* vals, int n) {
  if (n < 0 || n > 8) return drb_fail(DRB_E_INVALID, "launch_set_scalars: n must be in [0, 8]");
  Scalars8 s{};
  for (int i = 0; i < n; i++) s.v[i] = vals[i];
  k_set_scalars<<<1, 32, 0, ctx->stream>>>(dst, s, n);
  DRB_LAUNCH_CHECK(ctx, "k_set_scalars");
  return DRB_OK;
}

float drb_adam_alpha(float lr, float beta1, float beta2, int t) {
  // Keras computes this in fp32: lr * sqrt(1 - beta2^t) / (1 - beta1^t)
  const float b1p = powf(beta1, (float)t), b2p = powf(beta2, (float)t);
  return lr * sqrtf(1.0f - b2p) / (1.0f - b1p);
}

int launch_adam(drb_ctx* ctx, const AdamArgs& a, int* n_blocks_out, const OptimExtra& e) {
  if (a.nseg < 1 || a.nseg > DRB_MAX_SEGS) return drb_fail(DRB_E_INVALID, "adam: bad segment count");
  if (e.kind < 0 || e.kind >= OPT_N_KINDS) return drb_fail(DRB_E_INVALID, "optimizer update: bad kind %d", e.kind);
  const int64_t total4 = a.seg[a.nseg - 1].off4 + a.seg[a.nseg - 1].n4;      // the launch covers [seg[0].off4, total4)
  int64_t want = (total4 - a.seg[0].off4 + kAdamThreads - 1) / kAdamThreads;
  // 16 float4 per thread in flight across the grid keeps HBM busy; grid is a multiple of the SM count
  int blocks = (int)std::min<int64_t>(want, (int64_t)ctx->sm_count * 16);
  if (blocks < 1) blocks = 1;
  *n_blocks_out = blocks;
  using Kern = void (*)(AdamArgs, int64_t, OptimExtra);
  static const Kern kern[OPT_N_KINDS] = {
      nullptr, k_update<OPT_SGD, OptimExtra>, k_update<OPT_SGD_MOMENTUM, OptimExtra>, k_update<OPT_RMSPROP, OptimExtra>,
      k_update<OPT_RMSPROP_CENTERED, OptimExtra>, k_update<OPT_RMSPROP_MOMENTUM, OptimExtra>,
      k_update<OPT_RMSPROP_CENTERED_MOMENTUM, OptimExtra>, k_update<OPT_ADAGRAD, OptimExtra>,
      k_update<OPT_ADAMAX, OptimExtra>, k_update<OPT_AMSGRAD, OptimExtra>};
  const char* name = optim_kernel_name(e.kind);
  drb_prof_scope prof_(ctx, name);
  if (e.kind == OPT_ADAM)
    k_update<OPT_ADAM><<<blocks, kAdamThreads, 0, ctx->stream>>>(a, total4);
  else
    kern[e.kind]<<<blocks, kAdamThreads, 0, ctx->stream>>>(a, total4, e);
  DRB_LAUNCH_CHECK(ctx, name);
  return DRB_OK;
}

const char* optim_kernel_name(int kind) {
  static const char* const names[OPT_N_KINDS] = {
      "k_adam", "k_optim_sgd", "k_optim_sgd_momentum", "k_optim_rmsprop", "k_optim_rmsprop_centered",
      "k_optim_rmsprop_momentum", "k_optim_rmsprop_centered_momentum", "k_optim_adagrad", "k_optim_adamax",
      "k_optim_amsgrad"};
  return kind >= 0 && kind < OPT_N_KINDS ? names[kind] : "k_optim_invalid";
}

float drb_optim_step_size(const drb_optim_desc& o, float lr, int t) {
  // Keras-2 decay (OptimizerV2._decayed_lr): lr_t = lr / (1 + decay * iterations), iterations = t - 1, in fp32
  const float lr_t = o.decay != 0.f ? lr / (1.0f + o.decay * (float)(t - 1)) : lr;
  switch (o.kind) {
    case DRB_OPT_ADAM:
      return drb_adam_alpha(lr_t, o.beta1, o.beta2, t);       // alpha_t (AMSGrad too)
    case DRB_OPT_ADAMAX:
      return lr_t / (1.0f - powf(o.beta1, (float)t));          // ResourceApplyAdaMax: lr / (1 - beta1_power)
    default:
      return lr_t;
  }
}

int optim_update_kind(const drb_optim_desc& o) {
  switch (o.kind) {
    case DRB_OPT_ADAM: return o.amsgrad ? OPT_AMSGRAD : OPT_ADAM;
    case DRB_OPT_SGD: return o.momentum > 0.f ? OPT_SGD_MOMENTUM : OPT_SGD;
    case DRB_OPT_RMSPROP:
      if (o.momentum > 0.f) return o.centered ? OPT_RMSPROP_CENTERED_MOMENTUM : OPT_RMSPROP_MOMENTUM;
      return o.centered ? OPT_RMSPROP_CENTERED : OPT_RMSPROP;
    case DRB_OPT_ADAGRAD: return OPT_ADAGRAD;
    case DRB_OPT_ADAMAX: return OPT_ADAMAX;
    default: return -1;
  }
}

void optim_fill_args(const drb_optim_desc& o, AdamArgs& a, OptimExtra& e) {
  a.beta1 = o.beta1; a.beta2 = o.beta2; a.eps = o.epsilon;
  e.kind = optim_update_kind(o);
  e.momentum = o.momentum; e.rho = o.rho; e.nesterov = o.nesterov;
  e.x = o.third_state;
}

int optim_check(const drb_optim_desc* o, const char* who) {
  if (!o) return drb_fail(DRB_E_INVALID, "%s: NULL optimizer descriptor", who);
  if (optim_update_kind(*o) < 0)
    return drb_fail(DRB_E_INVALID, "%s: unknown optimizer kind %d (supported: DRB_OPT_ADAM, DRB_OPT_SGD, DRB_OPT_RMSPROP, "
                    "DRB_OPT_ADAGRAD, DRB_OPT_ADAMAX)", who, o->kind);
  if ((o->nesterov != 0 && o->nesterov != 1) || (o->centered != 0 && o->centered != 1) || (o->amsgrad != 0 && o->amsgrad != 1))
    return drb_fail(DRB_E_INVALID, "%s: nesterov, centered and amsgrad must be 0 or 1", who);
  if (!(o->decay >= 0.f) || !std::isfinite(o->decay)) return drb_fail(DRB_E_INVALID, "%s: decay must be >= 0", who);
  if ((o->kind == DRB_OPT_SGD || o->kind == DRB_OPT_RMSPROP) && !(o->momentum >= 0.f && o->momentum <= 1.f))
    return drb_fail(DRB_E_INVALID, "%s: momentum must be in [0, 1]", who);
  if (o->kind == DRB_OPT_RMSPROP && !(o->rho >= 0.f && o->rho <= 1.f))
    return drb_fail(DRB_E_INVALID, "%s: rho must be in [0, 1]", who);
  if ((o->kind == DRB_OPT_ADAM || o->kind == DRB_OPT_ADAMAX) &&
      !(o->beta1 >= 0.f && o->beta1 < 1.f && o->beta2 >= 0.f && o->beta2 < 1.f))
    return drb_fail(DRB_E_INVALID, "%s: beta1 and beta2 must be in [0, 1)", who);
  if (o->kind != DRB_OPT_SGD && !(o->epsilon >= 0.f && std::isfinite(o->epsilon)))
    return drb_fail(DRB_E_INVALID, "%s: epsilon must be finite and >= 0", who);
  if (o->kind != DRB_OPT_SGD && o->kind != DRB_OPT_ADAM && !(o->epsilon > 0.f))
    return drb_fail(DRB_E_INVALID, "%s: epsilon must be > 0 (zero-padded arena entries would divide 0 by 0)", who);
  const int k = optim_update_kind(*o);
  if (k == OPT_AMSGRAD || k == OPT_RMSPROP_CENTERED_MOMENTUM) {
    if (!o->third_state)
      return drb_fail(DRB_E_INVALID, "%s: AMSGrad and centered RMSprop with momentum need third_state (an arena-sized "
                      "device buffer)", who);
    if ((uintptr_t)o->third_state & 15) return drb_fail(DRB_E_INVALID, "%s: third_state must be 16-byte aligned", who);
  }
  return DRB_OK;
}

int launch_finalize_loss(drb_ctx* ctx, const float* loss_part, int n_loss, float scale, const float* reg_part,
                         int n_reg, float* loss_out) {
  drb_prof_scope prof_(ctx, "k_finalize_loss");
  k_finalize_loss<<<1, 256, 0, ctx->stream>>>(loss_part, n_loss, scale, reg_part, n_reg, loss_out);
  DRB_LAUNCH_CHECK(ctx, "k_finalize_loss");
  return DRB_OK;
}
