// hsb_grad_harness.cpp -- drives the HSBGrad OpKernels of this project's TF plugin (polee_b200/tf/hsb_ops_b200.cpp)
// through the stub TF API, as oracle/tf_stub/ref_hsb_harness.cpp drives the other three ops.  The reference's op file
// has no HSBGrad (hsb_ops.cpp:123-125), so this harness only ever links with the shim.  TEST INFRASTRUCTURE ONLY:
// tests/test_gpu_hsb_grad.py compiles it with hsb_ops_b200.cpp into a library of its own.
#include <cstring>
#include <memory>
#include "tf_stub_core.h"

using namespace tensorflow;

// device "CPU": host tensors, the output copied back.  device "GPU": data tensors and the output are device memory the
// caller owns, the kernel writes the output in place and enqueues on `stream`.
static int run_hsb_grad(int64_t B, int64_t n, const float* x_grad, const float* y_logit, const int32_t* left,
                        const int32_t* right, const int32_t* leaf, float* y_logit_grad, const char* device, void* stream) {
  auto& reg = OpRegistryStub::Global();
  const bool gpu = std::string(device) == "GPU";
  auto it = reg.kernels.find(std::string("HSBGrad/") + device);
  if (it == reg.kernels.end()) return -1;
  const int64_t N = 2 * n - 1;
  Tensor xg(DT_FLOAT, TensorShape({B, n}), (void*)x_grad), yl(DT_FLOAT, TensorShape({B, n - 1}), (void*)y_logit),
      l(DT_INT32, TensorShape({B, N}), (void*)left), r(DT_INT32, TensorShape({B, N}), (void*)right),
      f(DT_INT32, TensorShape({B, N}), (void*)leaf);
  OpKernelConstruction c;
  std::unique_ptr<OpKernel> k(it->second(&c));
  OpKernelContext ctx;
  ctx.inputs = {&xg, &yl, &l, &r, &f};
  ctx.output_types = {DT_FLOAT};
  ctx.dev.w_.num_threads = 1;
  ctx.dev.w_.workers = nullptr;
  if (gpu) {
    ctx.output_prealloc = {y_logit_grad};
    ctx.gpu_stream = stream;
  }
  k->Compute(&ctx);
  if (!ctx.status.ok()) return -2;
  if (!gpu) std::memcpy(y_logit_grad, ctx.outputs[0]->raw(), (size_t)(B * (n - 1)) * 4);
  return 0;
}

extern "C" {

int shim_hsb_grad(int64_t B, int64_t n, const float* x_grad, const float* y_logit, const int32_t* left,
                  const int32_t* right, const int32_t* leaf, float* y_logit_grad) {
  return run_hsb_grad(B, n, x_grad, y_logit, left, right, leaf, y_logit_grad, "CPU", nullptr);
}

int shim_hsb_grad_gpu(int64_t B, int64_t n, const float* d_x_grad, const float* d_y_logit, const int32_t* left,
                      const int32_t* right, const int32_t* leaf, float* d_y_logit_grad, void* stream) {
  return run_hsb_grad(B, n, d_x_grad, d_y_logit, left, right, leaf, d_y_logit_grad, "GPU", stream);
}
}
