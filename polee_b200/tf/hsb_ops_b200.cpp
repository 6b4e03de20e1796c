// hsb_ops_b200.cpp -- drop-in replacement for the reference's src/tensorflow_ext/hsb_ops.cpp: the same three
// ops (names, inputs, outputs, dtypes, shape functions: hsb_ops.cpp:17-38, 128-150, 252-278) whose Compute()
// forwards to libpolee_b200.so.  Python keeps doing `tf.load_op_library(...)` and calling `hsb`, `inv_hsb`,
// `inv_hsb_grad` (src/polee_approx_likelihood.py:13-28, 50, 408) unchanged.  A fourth op, HSBGrad, is the gradient
// of HSB that the reference leaves as a TODO (hsb_ops.cpp:123-125); INTEGRATION.md §3 registers it for `hsb`.
//
// Build (mirrors src/tensorflow_ext/mkfile and PoleeModel.jl:53-64):
//   g++ -std=c++14 -shared -fPIC -O2 hsb_ops_b200.cpp -o hsb_ops.so $TF_CFLAGS $TF_LFLAGS
//       -I<repo>/include -L<repo>/polee_b200 -lpolee_b200 -Wl,-rpath,<repo>/polee_b200
// TensorFlow is not installed in the build image; `make -C tests/tf_shim check` compiles this file against a stub
// of the TF op API (the same stub that builds the reference's own op file) and the GPU tests drive it that way.
//
// Every op is registered twice.  DEVICE_CPU (what the reference registers, hsb_ops.cpp:120, 249, 402): TF hands over
// host tensors and the library does its own transfers (polee_*_with_plan).  DEVICE_GPU: the data tensors are device
// memory and are consumed and produced in place on the op's CUDA stream (polee_*_device; no copy, no allocation per
// call); only the three index tensors are pinned to host memory (HostMemory), because the tree plan is built from them
// on the host once and cached.
#include "tensorflow/core/framework/op.h"
#include "tensorflow/core/framework/op_kernel.h"
#include "tensorflow/core/framework/shape_inference.h"

#include <cstdint>
#include <cstring>
#include <map>
#include <mutex>

#include "polee_b200.h"

#ifdef POLEE_TF_STUB_CORE_H
// the stand-in API of the test build carries the stream in the context
static void* polee_tf_stream(tensorflow::OpKernelContext* c) { return c->gpu_stream; }
#else
// real TensorFlow (build with the CUDA toolkit's headers on the include path): the op's compute stream
#define EIGEN_USE_GPU
#include "tensorflow/core/framework/tensor.h"
#include "unsupported/Eigen/CXX11/Tensor"
static void* polee_tf_stream(tensorflow::OpKernelContext* c) {
    return (void*)c->eigen_device<Eigen::GpuDevice>().stream();
}
#endif

using namespace tensorflow;

namespace {

// Index tensors are constants of the model (src/estimate.jl:357-376), so the validated + scheduled trees are
// cached on the device, keyed by shape and a 64-bit FNV-1a hash of the three index arrays.
struct PlanKey {
    int64_t n, idx_batch;
    uint64_t hash;
    bool operator<(const PlanKey& o) const {
        if (n != o.n) return n < o.n;
        if (idx_batch != o.idx_batch) return idx_batch < o.idx_batch;
        return hash < o.hash;
    }
};

uint64_t fnv1a(const void* p, size_t bytes, uint64_t h) {
    const unsigned char* c = static_cast<const unsigned char*>(p);
    for (size_t i = 0; i < bytes; ++i) { h ^= c[i]; h *= 1099511628211ull; }
    return h;
}

std::mutex g_mu;
std::map<PlanKey, polee_hsb_plan*> g_plans;

int device_ordinal() {
    const char* e = std::getenv("POLEE_B200_DEVICE");
    return e ? std::atoi(e) : 0;
}

// all rows share one tree when every row of the index tensors is identical (the reference requires [B, 2n-1])
polee_hsb_plan* plan_for(int64_t B, int64_t n, const int32* left, const int32* right, const int32* leaf, std::string* err) {
    const int64_t N = 2 * n - 1;
    bool shared = true;
    for (int64_t b = 1; b < B && shared; ++b)
        shared = !std::memcmp(left, left + b * N, N * 4) && !std::memcmp(right, right + b * N, N * 4) &&
                 !std::memcmp(leaf, leaf + b * N, N * 4);
    const int64_t ib = shared ? 1 : B;
    uint64_t h = 1469598103934665603ull;
    h = fnv1a(left, (size_t)ib * N * 4, h);
    h = fnv1a(right, (size_t)ib * N * 4, h);
    h = fnv1a(leaf, (size_t)ib * N * 4, h);
    PlanKey key{n, ib, h};
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = g_plans.find(key);
    if (it != g_plans.end()) return it->second;
    polee_hsb_plan* p = nullptr;
    if (polee_hsb_plan_create(&p, device_ordinal(), n, ib, left, right, leaf) != POLEE_OK) {
        *err = polee_hsb_last_error();
        return nullptr;
    }
    g_plans[key] = p;
    return p;
}

Status fail(const std::string& msg) { return Status("polee_b200: " + msg); }

}  // namespace

REGISTER_OP("HSB")
    .Input("y_logit: float32")
    .Input("left_index: int32")
    .Input("right_index: int32")
    .Input("leaf_index: int32")
    .Output("x: float32")
    .SetShapeFn([](shape_inference::InferenceContext* c) {
        shape_inference::ShapeHandle y_logit, unused;
        TF_RETURN_IF_ERROR(c->WithRank(c->input(0), 2, &y_logit));
        TF_RETURN_IF_ERROR(c->WithRank(c->input(1), 2, &unused));
        TF_RETURN_IF_ERROR(c->WithRank(c->input(2), 2, &unused));
        TF_RETURN_IF_ERROR(c->WithRank(c->input(3), 2, &unused));
        shape_inference::DimensionHandle m = c->Dim(y_logit, 0);
        shape_inference::DimensionHandle n = c->MakeDim(c->Value(c->Dim(y_logit, 1)) + 1);
        c->set_output(0, c->MakeShape({m, n}));
        return Status::OK();
    });

template <bool ON_DEVICE>
class HSBOpB200 : public OpKernel {
   public:
    explicit HSBOpB200(OpKernelConstruction* context) : OpKernel(context) {}
    void Compute(OpKernelContext* context) override {
        const Tensor& y_logit = context->input(0);
        const int64 B = y_logit.dim_size(0), n = y_logit.dim_size(1) + 1;
        Tensor* x = nullptr;
        OP_REQUIRES_OK(context, context->allocate_output(0, TensorShape({B, n}), &x));
        std::string err;
        polee_hsb_plan* p = plan_for(B, n, &context->input(1).flat_inner_dims<int32>()(0, 0),
                                     &context->input(2).flat_inner_dims<int32>()(0, 0),
                                     &context->input(3).flat_inner_dims<int32>()(0, 0), &err);
        if (!p) OP_REQUIRES_OK(context, fail(err));
        const float* in = &y_logit.flat_inner_dims<float>()(0, 0);
        float* out = &x->flat_inner_dims<float>()(0, 0);
        const int rc = ON_DEVICE ? polee_hsb_device(p, B, in, out, polee_tf_stream(context)) : polee_hsb_with_plan(p, B, in, out);
        if (rc != POLEE_OK) OP_REQUIRES_OK(context, fail(polee_hsb_last_error()));
    }
};
REGISTER_KERNEL_BUILDER(Name("HSB").Device(DEVICE_CPU), HSBOpB200<false>);
REGISTER_KERNEL_BUILDER(Name("HSB").Device(DEVICE_GPU).HostMemory("left_index").HostMemory("right_index").HostMemory("leaf_index"),
                        HSBOpB200<true>);

REGISTER_OP("InvHSB")
    .Input("x: float32")
    .Input("left_index: int32")
    .Input("right_index: int32")
    .Input("leaf_index: int32")
    .Output("y: float64")
    .Output("ladj: float32")
    .SetShapeFn([](shape_inference::InferenceContext* c) {
        shape_inference::ShapeHandle x, unused;
        TF_RETURN_IF_ERROR(c->WithRank(c->input(0), 2, &x));
        TF_RETURN_IF_ERROR(c->WithRank(c->input(1), 2, &unused));
        TF_RETURN_IF_ERROR(c->WithRank(c->input(2), 2, &unused));
        TF_RETURN_IF_ERROR(c->WithRank(c->input(3), 2, &unused));
        shape_inference::DimensionHandle m = c->Dim(x, 0);
        shape_inference::DimensionHandle nm1 = c->MakeDim(c->Value(c->Dim(x, 1)) - 1);
        c->set_output(0, c->MakeShape({m, nm1}));
        c->set_output(1, c->MakeShape({m, 1}));
        return Status::OK();
    });

template <bool ON_DEVICE>
class InvHSBOpB200 : public OpKernel {
   public:
    explicit InvHSBOpB200(OpKernelConstruction* context) : OpKernel(context) {}
    void Compute(OpKernelContext* context) override {
        const Tensor& x = context->input(0);
        const int64 B = x.dim_size(0), n = x.dim_size(1);
        Tensor *y = nullptr, *ladj = nullptr;
        OP_REQUIRES_OK(context, context->allocate_output(0, TensorShape({B, n - 1}), &y));
        OP_REQUIRES_OK(context, context->allocate_output(1, TensorShape({B, 1}), &ladj));
        std::string err;
        polee_hsb_plan* p = plan_for(B, n, &context->input(1).flat_inner_dims<int32>()(0, 0),
                                     &context->input(2).flat_inner_dims<int32>()(0, 0),
                                     &context->input(3).flat_inner_dims<int32>()(0, 0), &err);
        if (!p) OP_REQUIRES_OK(context, fail(err));
        const float* in = &x.flat_inner_dims<float>()(0, 0);
        double* yo = &y->flat_inner_dims<double>()(0, 0);
        float* lo = &ladj->flat_inner_dims<float>()(0, 0);
        const int rc = ON_DEVICE ? polee_inv_hsb_device(p, B, in, yo, lo, polee_tf_stream(context)) : polee_inv_hsb_with_plan(p, B, in, yo, lo);
        if (rc != POLEE_OK) OP_REQUIRES_OK(context, fail(polee_hsb_last_error()));
    }
};
REGISTER_KERNEL_BUILDER(Name("InvHSB").Device(DEVICE_CPU), InvHSBOpB200<false>);
REGISTER_KERNEL_BUILDER(Name("InvHSB").Device(DEVICE_GPU).HostMemory("left_index").HostMemory("right_index").HostMemory("leaf_index"),
                        InvHSBOpB200<true>);

REGISTER_OP("InvHSBGrad")
    .Input("y_grad: float64")
    .Input("ladj_grad: float32")
    .Input("y: float64")
    .Input("ladj: float32")
    .Input("left_index: int32")
    .Input("right_index: int32")
    .Input("leaf_index: int32")
    .Output("backprops: float32")
    .SetShapeFn([](shape_inference::InferenceContext* c) {
        shape_inference::ShapeHandle y, unused;
        TF_RETURN_IF_ERROR(c->WithRank(c->input(0), 2, &y));
        TF_RETURN_IF_ERROR(c->WithRank(c->input(1), 2, &unused));
        TF_RETURN_IF_ERROR(c->WithRank(c->input(2), 2, &unused));
        TF_RETURN_IF_ERROR(c->WithRank(c->input(3), 2, &unused));
        TF_RETURN_IF_ERROR(c->WithRank(c->input(4), 2, &unused));
        shape_inference::DimensionHandle m = c->Dim(y, 0);
        shape_inference::DimensionHandle n = c->MakeDim(c->Value(c->Dim(y, 1)) + 1);
        c->set_output(0, c->MakeShape({m, n}));
        return Status::OK();
    });

template <bool ON_DEVICE>
class InvHSBGradOpB200 : public OpKernel {
   public:
    explicit InvHSBGradOpB200(OpKernelConstruction* context) : OpKernel(context) {}
    void Compute(OpKernelContext* context) override {
        const Tensor& y_grad = context->input(0);
        const Tensor& ladj_grad = context->input(1);
        const Tensor& y = context->input(2);
        const int64 B = y.dim_size(0), n = y.dim_size(1) + 1;
        Tensor* bp = nullptr;
        OP_REQUIRES_OK(context, context->allocate_output(0, TensorShape({B, n}), &bp));
        std::string err;
        polee_hsb_plan* p = plan_for(B, n, &context->input(4).flat_inner_dims<int32>()(0, 0),
                                     &context->input(5).flat_inner_dims<int32>()(0, 0),
                                     &context->input(6).flat_inner_dims<int32>()(0, 0), &err);
        if (!p) OP_REQUIRES_OK(context, fail(err));
        const double* yg = &y_grad.flat_inner_dims<double>()(0, 0);
        const float* lg = &ladj_grad.flat_inner_dims<float>()(0, 0);
        const double* yv = &y.flat_inner_dims<double>()(0, 0);
        float* out = &bp->flat_inner_dims<float>()(0, 0);
        const int rc = ON_DEVICE ? polee_inv_hsb_grad_device(p, B, yg, lg, yv, out, polee_tf_stream(context))
                                 : polee_inv_hsb_grad_with_plan(p, B, yg, lg, yv, out);
        if (rc != POLEE_OK) OP_REQUIRES_OK(context, fail(polee_hsb_last_error()));
    }
};
REGISTER_KERNEL_BUILDER(Name("InvHSBGrad").Device(DEVICE_CPU), InvHSBGradOpB200<false>);
REGISTER_KERNEL_BUILDER(Name("InvHSBGrad").Device(DEVICE_GPU).HostMemory("left_index").HostMemory("right_index").HostMemory("leaf_index"),
                        InvHSBGradOpB200<true>);

REGISTER_OP("HSBGrad")
    .Input("x_grad: float32")
    .Input("y_logit: float32")
    .Input("left_index: int32")
    .Input("right_index: int32")
    .Input("leaf_index: int32")
    .Output("y_logit_grad: float32")
    .SetShapeFn([](shape_inference::InferenceContext* c) {
        shape_inference::ShapeHandle y_logit, unused;
        TF_RETURN_IF_ERROR(c->WithRank(c->input(0), 2, &unused));
        TF_RETURN_IF_ERROR(c->WithRank(c->input(1), 2, &y_logit));
        TF_RETURN_IF_ERROR(c->WithRank(c->input(2), 2, &unused));
        TF_RETURN_IF_ERROR(c->WithRank(c->input(3), 2, &unused));
        TF_RETURN_IF_ERROR(c->WithRank(c->input(4), 2, &unused));
        c->set_output(0, y_logit);
        return Status::OK();
    });

template <bool ON_DEVICE>
class HSBGradOpB200 : public OpKernel {
   public:
    explicit HSBGradOpB200(OpKernelConstruction* context) : OpKernel(context) {}
    void Compute(OpKernelContext* context) override {
        const Tensor& x_grad = context->input(0);
        const Tensor& y_logit = context->input(1);
        const int64 B = y_logit.dim_size(0), n = y_logit.dim_size(1) + 1;
        Tensor* out = nullptr;
        OP_REQUIRES_OK(context, context->allocate_output(0, TensorShape({B, n - 1}), &out));
        std::string err;
        polee_hsb_plan* p = plan_for(B, n, &context->input(2).flat_inner_dims<int32>()(0, 0),
                                     &context->input(3).flat_inner_dims<int32>()(0, 0),
                                     &context->input(4).flat_inner_dims<int32>()(0, 0), &err);
        if (!p) OP_REQUIRES_OK(context, fail(err));
        const float* xg = &x_grad.flat_inner_dims<float>()(0, 0);
        const float* yl = &y_logit.flat_inner_dims<float>()(0, 0);
        float* o = &out->flat_inner_dims<float>()(0, 0);
        const int rc = ON_DEVICE ? polee_hsb_grad_device(p, B, xg, yl, o, polee_tf_stream(context))
                                 : polee_hsb_grad_with_plan(p, B, xg, yl, o);
        if (rc != POLEE_OK) OP_REQUIRES_OK(context, fail(polee_hsb_last_error()));
    }
};
REGISTER_KERNEL_BUILDER(Name("HSBGrad").Device(DEVICE_CPU), HSBGradOpB200<false>);
REGISTER_KERNEL_BUILDER(Name("HSBGrad").Device(DEVICE_GPU).HostMemory("left_index").HostMemory("right_index").HostMemory("leaf_index"),
                        HSBGradOpB200<true>);
