// adam.cu -- Adam / AdamW over ONE flat fp32 parameter buffer, and the global gradient norm
// (sm_100a).
//
// The reference optimises with torch.optim.Adam over ~100 small tensors
// (train_Votenet_FSB.py:176-181); PyTorch's fused implementation needs three multi-tensor launches
// (~60 us for 0.96 M parameters) at the very end of the step's critical path.  With parameters,
// gradients and both moments in flat buffers (dist_utils.FlatGradBucket already packs the gradients
// for the NCCL all-reduce) the update is one streaming pass: 16 B read + 12 B written per
// parameter, ~27 MB, a few microseconds.  Same arithmetic as torch.optim.Adam(amsgrad=False,
// maximize=False): m = b1*m + (1-b1)*g; v = b2*v + (1-b2)*g*g;
// p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps), with optional L2 weight decay g += wd*p,
// or (decoupled, torch.optim.AdamW) p *= 1 - lr*wd before the moments.
// The step counter lives on the device so the launch can be replayed from a CUDA graph.
//
// One kernel, two instances: b2r_adam_flat_step passes one lr / weight decay by value (baked into
// a captured graph); b2r_adam_flat_step_groups reads per-group lr / weight decay from a device
// table, so a learning-rate schedule written into that table between replays takes effect, and
// optionally scales the gradient by the clip coefficient b2r_flat_grad_norm wrote.
//
// The norm (clip_grad_norm_ with norm_type 2) is a fixed-grid fp64 partial sum per block followed
// by one block that adds the partials in a fixed order: no atomics, so identical gradients give a
// bit-identical norm on every replay, and no host synchronisation.
#include "common.cuh"

namespace b2r {
namespace {

struct AdamState {     // device-resident: { t, 1/(1-b1^t), 1/sqrt(1-b2^t) }
  float t, inv_bc1, inv_sqrt_bc2, pad;
};

__global__ void adam_tick_kernel(AdamState *st, float b1, float b2) {
  const float t = st->t + 1.0f;
  st->t = t;
  st->inv_bc1 = (float)(1.0 / (1.0 - pow((double)b1, (double)t)));
  st->inv_sqrt_bc2 = (float)(1.0 / sqrt(1.0 - pow((double)b2, (double)t)));
}

struct AdamArgs {
  float *p;
  const float *g;
  float *m, *v;
  long long n4, n;
  const AdamState *st;
  const b2r_adam_group *groups;  // kTable: device table of n_groups entries
  int n_groups;
  float lr, wd;                  // !kTable: the one group [0, n), by value
  float b1, b2, eps, gscale;
  int decoupled;                 // kTable only
  const float *clip;             // kTable only; NULL: no clipping
};

// kTable = false: b2r_adam_flat_step (one group, hyperparameters by value, L2 decay, no clip).
template <bool kTable>
__global__ void __launch_bounds__(256) adam_flat_kernel(const AdamArgs a) {
  __shared__ b2r_adam_group tab[kTable ? B2R_ADAM_MAX_GROUPS : 1];
  if (kTable) {
    for (int i = threadIdx.x; i < a.n_groups; i += blockDim.x) tab[i] = a.groups[i];
    __syncthreads();
  }
  const float b1 = a.b1, b2 = a.b2, eps = a.eps, isb2 = a.st->inv_sqrt_bc2;
  const float inv_bc1 = a.st->inv_bc1;
  // the clip coefficient multiplies the gradient after grad_scale, as clip_grad_norm_ multiplies
  // the averaged gradient
  const float coef = (kTable && a.clip) ? *a.clip : 1.f;
  // current group of this thread: [lo, hi) in elements.  A thread's indices only increase, so the
  // group index only moves forward.
  int gi = kTable ? -1 : 0;
  long long lo = 0, hi = kTable ? 0 : a.n;
  float wd = a.wd, step_size = a.lr * inv_bc1, decay = 1.f;
  auto in_group = [&](long long e) -> bool {
    if (kTable) {
      while (e >= hi && gi + 1 < a.n_groups) {
        ++gi;
        lo = tab[gi].start; hi = tab[gi].end;
        const float lr = tab[gi].lr;
        wd = tab[gi].weight_decay;
        step_size = lr * inv_bc1;
        decay = 1.f - lr * wd;
      }
    }
    return e >= lo && e < hi;
  };
  auto upd = [&](float &pp, float gg, float &mm, float &vv) {
    gg *= a.gscale;
    if (kTable && a.clip) gg *= coef;
    if (wd != 0.f) {
      if (kTable && a.decoupled) pp *= decay;
      else gg = fmaf(wd, pp, gg);
    }
    mm = fmaf(b1, mm, (1.f - b1) * gg);
    vv = fmaf(b2, vv, (1.f - b2) * gg * gg);
    pp -= step_size * mm / (sqrtf(vv) * isb2 + eps);
  };
  float *__restrict__ p = a.p, *__restrict__ m = a.m, *__restrict__ v = a.v;
  const float *__restrict__ g = a.g;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n4; i += stride) {
    if (!in_group(i * 4)) continue;   // group bounds are multiples of 4 (or n): whole vectors
    float4 pp = reinterpret_cast<float4 *>(p)[i], mm = reinterpret_cast<float4 *>(m)[i],
           vv = reinterpret_cast<float4 *>(v)[i];
    const float4 gg = reinterpret_cast<const float4 *>(g)[i];
    upd(pp.x, gg.x, mm.x, vv.x); upd(pp.y, gg.y, mm.y, vv.y);
    upd(pp.z, gg.z, mm.z, vv.z); upd(pp.w, gg.w, mm.w, vv.w);
    reinterpret_cast<float4 *>(p)[i] = pp;
    reinterpret_cast<float4 *>(m)[i] = mm;
    reinterpret_cast<float4 *>(v)[i] = vv;
  }
  for (long long i = a.n4 * 4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += stride)
    if (in_group(i)) upd(p[i], g[i], m[i], v[i]);
}

int launch_adam(const AdamArgs &a, bool table, cudaStream_t st) {
  adam_tick_kernel<<<1, 1, 0, st>>>(const_cast<AdamState *>(a.st), a.b1, a.b2);
  B2R_CHECK_LAUNCH();
  long long blocks = (a.n4 + 255) / 256;
  if (blocks > 4LL * kNumSMs) blocks = 4LL * kNumSMs;
  if (blocks < 1) blocks = 1;
  if (table)
    adam_flat_kernel<true><<<(unsigned)blocks, 256, 0, st>>>(a);
  else
    adam_flat_kernel<false><<<(unsigned)blocks, 256, 0, st>>>(a);
  B2R_CHECK_LAUNCH();
  return B2R_OK;
}

// ---- global L2 norm -------------------------------------------------------------------------
constexpr int kNormThreads = 256;

// grid size: a function of n only, so the partials (and their sum) are always formed the same way
long long norm_blocks(long long n) {
  long long b = (n / 4 + kNormThreads - 1) / kNormThreads;
  if (b > 4LL * kNumSMs) b = 4LL * kNumSMs;
  return b < 1 ? 1 : b;
}

__device__ __forceinline__ double block_sum(double s, double *red) {
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
  return t;   // valid in thread 0
}

__global__ void __launch_bounds__(kNormThreads)
    grad_sumsq_partial_kernel(const float *__restrict__ g, long long n4, long long n, float gscale,
                              double *__restrict__ partial) {
  __shared__ double red[kNormThreads / 32];
  double s = 0.0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const int4 r = ldg_stream_v4(reinterpret_cast<const int4 *>(g) + i);
    const float x = __int_as_float(r.x) * gscale, y = __int_as_float(r.y) * gscale,
                z = __int_as_float(r.z) * gscale, w = __int_as_float(r.w) * gscale;
    s += (double)x * x + (double)y * y + (double)z * z + (double)w * w;
  }
  for (long long i = n4 * 4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float x = g[i] * gscale;
    s += (double)x * x;
  }
  const double t = block_sum(s, red);
  if (threadIdx.x == 0) partial[blockIdx.x] = t;
}

__global__ void __launch_bounds__(kNormThreads)
    grad_norm_final_kernel(const double *__restrict__ partial, int nparts, float max_norm,
                           float *__restrict__ norm_out, float *__restrict__ coef_out) {
  __shared__ double red[kNormThreads / 32];
  double s = 0.0;
  for (int i = threadIdx.x; i < nparts; i += blockDim.x) s += partial[i];
  const double t = block_sum(s, red);
  if (threadIdx.x == 0) {
    const float norm = (float)sqrt(t);
    *norm_out = norm;
    // torch: clip_coef = max_norm / (total_norm + 1e-6); clamp(clip_coef, max=1.0), in fp32.
    // A scalar divided by a tensor is reciprocal() * scalar in torch (Tensor.__rtruediv__): same
    // roundings here.  A NaN norm gives a NaN coefficient, an infinite one 0
    // (error_if_nonfinite=False).
    const float c = __fmul_rn(__frcp_rn(__fadd_rn(norm, 1e-6f)), max_norm);
    *coef_out = c > 1.f ? 1.f : c;
  }
}

}  // namespace
}  // namespace b2r

extern "C" int b2r_adam_state_bytes(void) { return (int)sizeof(b2r::AdamState); }

extern "C" int b2r_adam_flat_step(float *params, const float *grads, float *exp_avg, float *exp_avg_sq,
                                  long long n, void *state, float lr, float beta1, float beta2,
                                  float eps, float weight_decay, float grad_scale, void *stream) {
  B2R_REQUIRE(n >= 0, "b2r_adam_flat_step: negative size");
  if (n == 0) return B2R_OK;
  B2R_REQUIRE(params && grads && exp_avg && exp_avg_sq && state, "b2r_adam_flat_step: null pointer");
  B2R_REQUIRE(((reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(grads) |
                reinterpret_cast<uintptr_t>(exp_avg) | reinterpret_cast<uintptr_t>(exp_avg_sq)) & 15) == 0,
              "b2r_adam_flat_step: buffers must be 16-byte aligned");
  b2r::AdamArgs a{};
  a.p = params; a.g = grads; a.m = exp_avg; a.v = exp_avg_sq;
  a.n4 = n / 4; a.n = n;
  a.st = static_cast<const b2r::AdamState *>(state);
  a.lr = lr; a.wd = weight_decay;
  a.b1 = beta1; a.b2 = beta2; a.eps = eps; a.gscale = grad_scale;
  return b2r::launch_adam(a, false, static_cast<cudaStream_t>(stream));
}

extern "C" int b2r_adam_flat_step_groups(const b2r_adam_desc *d, void *stream) {
  B2R_REQUIRE(d != nullptr, "b2r_adam_flat_step_groups: null descriptor");
  B2R_REQUIRE(d->n >= 0, "b2r_adam_flat_step_groups: negative size");
  B2R_REQUIRE(d->n_groups >= 1 && d->n_groups <= B2R_ADAM_MAX_GROUPS,
              "b2r_adam_flat_step_groups: n_groups = %d outside [1, %d]", d->n_groups,
              B2R_ADAM_MAX_GROUPS);
  if (d->n == 0) return B2R_OK;
  B2R_REQUIRE(d->params && d->grads && d->exp_avg && d->exp_avg_sq && d->state && d->groups,
              "b2r_adam_flat_step_groups: null pointer");
  B2R_REQUIRE(((reinterpret_cast<uintptr_t>(d->params) | reinterpret_cast<uintptr_t>(d->grads) |
                reinterpret_cast<uintptr_t>(d->exp_avg) | reinterpret_cast<uintptr_t>(d->exp_avg_sq)) &
               15) == 0,
              "b2r_adam_flat_step_groups: buffers must be 16-byte aligned");
  b2r::AdamArgs a{};
  a.p = d->params; a.g = d->grads; a.m = d->exp_avg; a.v = d->exp_avg_sq;
  a.n4 = d->n / 4; a.n = d->n;
  a.st = static_cast<const b2r::AdamState *>(d->state);
  a.groups = d->groups; a.n_groups = d->n_groups;
  a.b1 = d->beta1; a.b2 = d->beta2; a.eps = d->eps; a.gscale = d->grad_scale;
  a.decoupled = d->decoupled != 0;
  a.clip = d->clip_coef;
  return b2r::launch_adam(a, true, static_cast<cudaStream_t>(stream));
}

extern "C" long long b2r_flat_grad_norm_workspace_bytes(long long n) {
  if (n < 0) return -1;
  return b2r::norm_blocks(n) * (long long)sizeof(double);
}

extern "C" int b2r_flat_grad_norm(const float *grads, long long n, float grad_scale, float max_norm,
                                  void *workspace, float *norm_out, float *coef_out, void *stream) {
  B2R_REQUIRE(n >= 0, "b2r_flat_grad_norm: negative size");
  B2R_REQUIRE((grads || n == 0) && workspace && norm_out && coef_out, "b2r_flat_grad_norm: null pointer");
  B2R_REQUIRE(((reinterpret_cast<uintptr_t>(grads) | reinterpret_cast<uintptr_t>(workspace)) & 15) == 0,
              "b2r_flat_grad_norm: grads and workspace must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long blocks = b2r::norm_blocks(n);
  auto *part = static_cast<double *>(workspace);
  b2r::grad_sumsq_partial_kernel<<<(unsigned)blocks, b2r::kNormThreads, 0, st>>>(grads, n / 4, n,
                                                                                 grad_scale, part);
  B2R_CHECK_LAUNCH();
  b2r::grad_norm_final_kernel<<<1, b2r::kNormThreads, 0, st>>>(part, (int)blocks, max_norm, norm_out,
                                                               coef_out);
  B2R_CHECK_LAUNCH();
  return B2R_OK;
}
