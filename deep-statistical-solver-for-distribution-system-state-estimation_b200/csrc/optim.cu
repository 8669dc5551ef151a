// Adjacent row (SURVEY.md 8f-2): flat-buffer Adamax, torch.optim.Adamax defaults (dss2_run.py:91-92,143).
// The reference steps ~180 tiny tensors through torch's foreach path; here all parameters live in one flat
// fp32 buffer and one launch updates them.  The step counter lives in device memory so that a captured
// CUDA graph advances its own bias correction on every replay.
#include "common.cuh"

namespace {

__global__ void k_adamax(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ u,
                         int64_t n, float lr, float beta1, float beta2, float eps, float gscale, const uint64_t* step_state) {
  __shared__ float s_clr;
  if (threadIdx.x == 0) {
    const double step = (double)(step_state[1] + 1);
    s_clr = (float)((double)lr / (1.0 - pow((double)beta1, step)));
  }
  __syncthreads();
  const float clr = s_clr;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float grad = g[i] * gscale;
    float mi = m[i];
    mi = mi + (1.0f - beta1) * (grad - mi);              // exp_avg.lerp_(grad, 1 - beta1)
    const float ui = fmaxf(u[i] * beta2, fabsf(grad) + eps);   // exp_inf = max(exp_inf * beta2, |grad| + eps)
    m[i] = mi;
    u[i] = ui;
    p[i] = p[i] - clr * (mi / ui);                       // param.addcdiv_(exp_avg, exp_inf, value=-clr)
  }
}
__global__ void k_bump(uint64_t* step_state) { step_state[1] += 1; }

}  // namespace

extern "C" int dss2_adamax_step(float* param, const float* grad, float* exp_avg, float* exp_inf, int64_t count, float lr,
                                float beta1, float beta2, float eps, float grad_scale, uint64_t* step_state, int bump,
                                void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DSS2_CHECK_ARG(param && grad && exp_avg && exp_inf && step_state && count >= 0, "dss2_adamax_step: bad argument");
  if (count > 0) {
    int grid = (int)max((int64_t)1, min((int64_t)148 * 4, (count + 255) / 256));
    k_adamax<<<grid, 256, 0, stream>>>(param, grad, exp_avg, exp_inf, count, lr, beta1, beta2, eps, grad_scale, step_state);
    DSS2_LAUNCH_CHECK();
  }
  if (bump) {
    k_bump<<<1, 1, 0, stream>>>(step_state);
    DSS2_LAUNCH_CHECK();
  }
  return 0;
}

// The clock of a forward-only stream (the captured evaluator): one increment per forward keeps its dropout draws and tile-mark
// sequence numbers fresh on every replay.
extern "C" int dss2_step_advance(uint64_t* step_state, void* stream_) {
  DSS2_CHECK_ARG(step_state, "dss2_step_advance: null argument");
  k_bump<<<1, 1, 0, (cudaStream_t)stream_>>>(step_state);
  DSS2_LAUNCH_CHECK();
  return 0;
}
