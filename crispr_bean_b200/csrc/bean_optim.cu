// bean_optim.cu -- pyro.optim.ClippedAdam (bean/model/run.py:368-373; SURVEY App. A.6) for the models whose ELBO is
// assembled by torch autograd around the likelihood kernel (tiling, survival, covariates): ONE launch updates every
// parameter tensor of the model.  The step index and the per-step step size (lr_t * sqrt(1 - beta2^t) / (1 - beta1^t),
// lr_t = lr * lrd^t) are read from device memory, so the launch can sit inside a captured CUDA graph.
// (The fused sorting step has its own in-kernel copy of the update, bean_svi.cu:clipped_adam.)
#include "bean_common.cuh"

namespace bean {

constexpr int ADAM_THREADS = 256;

template <typename real>
struct AdamTensor {
  real* theta;
  const real* grad;
  real* m;
  real* v;
  long long n;
};

template <typename real>
struct AdamParams {
  AdamTensor<real> t[BEAN_ADAM_MAX_TENSORS];
  const double* step_sizes;
  const long long* step;
  long long n_steps;
  real beta1, beta2, eps, clip;
  const double* loss;   // loss[*step] or NULL
  int* nonfinite;       // first non-finite step or NULL (BeanAdamArgs.nonfinite_step)
};

template <typename real>
__global__ void __launch_bounds__(ADAM_THREADS) clipped_adam_kernel(const AdamParams<real> p) {
  const AdamTensor<real> t = p.t[blockIdx.y];
  long long s = *p.step;
  s = s < 0 ? 0 : (s >= p.n_steps ? p.n_steps - 1 : s);
  const real step_size = real(p.step_sizes[s]);
  real probe = real(0);  // NaN once a gradient was NaN / inf (g * 0): no predicate in the loop
  for (long long i = (long long)blockIdx.x * ADAM_THREADS + threadIdx.x; i < t.n; i += (long long)gridDim.x * ADAM_THREADS) {
    real g = t.grad[i];
    probe += g * real(0);
    g = g < -p.clip ? -p.clip : (g > p.clip ? p.clip : g);  // elementwise clamp, not a norm clip
    const real m = p.beta1 * t.m[i] + (real(1) - p.beta1) * g;
    const real v = p.beta2 * t.v[i] + (real(1) - p.beta2) * g * g;
    t.m[i] = m;
    t.v[i] = v;
    t.theta[i] -= step_size * m / (sqrt(v) + p.eps);
  }
  if (p.nonfinite) {  // launch-uniform
    bool bad = probe != probe;
    if (p.loss && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) bad |= !isfinite(p.loss[s]);
    const unsigned any = __ballot_sync(0xffffffffu, bad);
    if (any != 0u && (int)(threadIdx.x & 31u) == __ffs(any) - 1 && *(volatile int*)p.nonfinite > (int)s) atomicMin(p.nonfinite, (int)s);
  }
}

template <typename real>
static int launch_adam(const BeanAdamArgs* a, void* stream) {
  BEAN_REQUIRE(a != nullptr, BEAN_EINVAL, "args is NULL");
  BEAN_REQUIRE(a->n_tensors >= 1 && a->n_tensors <= BEAN_ADAM_MAX_TENSORS, BEAN_EINVAL, "n_tensors %d out of range [1, %d]",
               a->n_tensors, BEAN_ADAM_MAX_TENSORS);
  BEAN_REQUIRE(a->step_sizes && a->step && a->n_steps >= 1, BEAN_EINVAL, "step_sizes / step must be non-NULL, n_steps >= 1");
  BEAN_REQUIRE(a->clip > 0 && a->beta1 >= 0 && a->beta1 < 1 && a->beta2 >= 0 && a->beta2 < 1, BEAN_EINVAL, "bad optimiser constants");
  AdamParams<real> p{};
  long long n_max = 0;
  for (int i = 0; i < a->n_tensors; ++i) {
    const BeanAdamTensor& s = a->tensors[i];
    BEAN_REQUIRE(s.n >= 0, BEAN_EINVAL, "tensor %d: negative size", i);
    BEAN_REQUIRE(s.n == 0 || (s.theta && s.grad && s.m && s.v), BEAN_EINVAL, "tensor %d: theta / grad / m / v must be non-NULL", i);
    p.t[i].theta = static_cast<real*>(s.theta);
    p.t[i].grad = static_cast<const real*>(s.grad);
    p.t[i].m = static_cast<real*>(s.m);
    p.t[i].v = static_cast<real*>(s.v);
    p.t[i].n = s.n;
    n_max = s.n > n_max ? s.n : n_max;
  }
  if (n_max == 0) return BEAN_OK;
  p.step_sizes = a->step_sizes;
  p.step = reinterpret_cast<const long long*>(a->step);
  p.n_steps = a->n_steps;
  p.beta1 = real(a->beta1); p.beta2 = real(a->beta2); p.eps = real(a->eps); p.clip = real(a->clip);
  p.loss = a->loss;
  p.nonfinite = a->nonfinite_step;
  long long blocks = (n_max + ADAM_THREADS - 1) / ADAM_THREADS;
  if (blocks > 148 * 8) blocks = 148 * 8;  // grid-stride beyond one wave of 8 CTAs per SM
  const dim3 grid((unsigned)blocks, (unsigned)a->n_tensors);
  clipped_adam_kernel<real><<<grid, ADAM_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(p);
  BEAN_CUDA(cudaPeekAtLastError());
  return BEAN_OK;
}

}  // namespace bean

extern "C" {
int bean_clipped_adam_f32(const BeanAdamArgs* a, void* stream) { return bean::launch_adam<float>(a, stream); }
int bean_clipped_adam_f64(const BeanAdamArgs* a, void* stream) { return bean::launch_adam<double>(a, stream); }
}
