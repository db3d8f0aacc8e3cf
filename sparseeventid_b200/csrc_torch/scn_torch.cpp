// Thin PyTorch C++ layer over the C ABI (include/scn_b200.h): the autograd functions of the hot modules
// (convolutions, BatchNormalization(+leaky), AddTable+LeakyReLU, LeakyReLU) as torch::autograd::Function, so that a
// module forward/backward costs one native call instead of a Python autograd.Function round trip.  No arithmetic
// here: torch supplies device memory, the current stream and the autograd tape; every kernel is in libscn_b200.so.
// Required: the modules (scn/modules.py::_native) run these outside ops.Profiler and for contiguous fp32 parameters;
// scn/functional.py holds the per-kernel functions for the rest.  SCN counterpart: the pybind11 module
// `sparseconvnet.SCN` (SURVEY.md 8b).
#include <c10/cuda/CUDAStream.h>
#include <torch/extension.h>

#include <unordered_map>

#include "../../include/scn_b200.h"

namespace {

using torch::autograd::AutogradContext;
using torch::autograd::variable_list;

inline void* cur_stream() { return (void*)c10::cuda::getCurrentCUDAStream().stream(); }
inline int dcode(const at::Tensor& t) {
  if (t.scalar_type() == at::kFloat) return SCN_F32;
  TORCH_CHECK(t.scalar_type() == at::kBFloat16, "scn_b200: feature dtype must be float32 or bfloat16");
  return SCN_BF16;
}
inline void check(int rc, const char* what) {
  TORCH_CHECK(rc == 0, what, ": ", rc > 0 ? "CUDA error " : "SCN error ", rc);
}
inline bool has(const at::Tensor& t) { return t.defined() && t.numel() > 0; }
inline void* optr(const at::Tensor& t) { return has(t) ? t.data_ptr() : nullptr; }

// fp64 [2*C] scratch of the column reductions: one buffer per device, shared by every layer (stream-ordered)
at::Tensor& stats_scratch(const at::Device& dev, int64_t c) {
  static std::unordered_map<int, at::Tensor> table;
  at::Tensor& t = table[dev.index()];
  if (!t.defined() || t.numel() < 2 * c)
    t = at::empty({std::max<int64_t>(2 * c, 2048)}, at::TensorOptions().dtype(at::kDouble).device(dev));
  return t;
}

// gradient buffer to accumulate into in place (trainer.FlatGradArena), or an undefined tensor
at::Tensor direct_grad(const at::Tensor& p, bool direct) {
  if (!direct || !has(p)) return at::Tensor();
  const at::Tensor& g = p.grad();
  if (!g.defined() || g.scalar_type() != at::kFloat || !g.is_contiguous() || g.device() != p.device()) return at::Tensor();
  return g;
}

// optional Python callable(param): "the gradient of this parameter is complete" (distributed bucketed all-reduce);
// heap-allocated and never destroyed so no Python object is released after interpreter shutdown
py::object* g_ready_cb = nullptr;
void grad_ready(const at::Tensor& p) {
  if (g_ready_cb == nullptr) return;
  py::gil_scoped_acquire gil;
  if (!g_ready_cb->is_none()) (*g_ready_cb)(p);
}

// Column sums of the dx a BatchNorm backward just wrote (scn_bn_backward_colsum).  When that dx is the grad_output of a
// convolution with a bias -- conv -> BatchNorm, every convolution of the reference's blocks
// (src/networks/sparse_building_blocks.py:29-39) -- they ARE its bias gradient, and the convolution's backward skips its
// own column-sum pass.  The dx tensor is kept alive with them, so a matching data pointer cannot be a recycled address.
struct BnColsum {
  at::Tensor dx, colsum;
};
BnColsum& last_bn_colsum() {
  static BnColsum* v = new BnColsum();      // never destroyed: no CUDA free after the context is gone
  return *v;
}

struct ConvFn : public torch::autograd::Function<ConvFn> {
  static at::Tensor forward(AutogradContext* ctx, at::Tensor x, at::Tensor weight, at::Tensor bias, at::Tensor nbr_fwd,
                            at::Tensor nbr_bwd, int64_t n_out_rows, bool mirror, int64_t prec, int64_t out_code,
                            at::Tensor wimg, at::Tensor wimg_t, bool skip_prep, bool direct_w, bool direct_b) {
    x = x.contiguous();
    const int64_t K = weight.size(0), cin = weight.size(-2), cout = weight.size(-1);
    at::Tensor out = at::empty({n_out_rows, cout}, x.options().dtype(out_code == SCN_F32 ? at::kFloat : at::kBFloat16));
    check(scn_conv_module_forward(x.data_ptr(), dcode(x), x.size(0), nbr_fwd.data_ptr<int32_t>(), (int)K, n_out_rows,
                                  nbr_fwd.size(1), (int)cin, (int)cout, weight.data_ptr<float>(),
                                  has(bias) ? bias.data_ptr<float>() : nullptr, (int)prec, wimg.data_ptr(),
                                  skip_prep ? 1 : 0, out.data_ptr(), (int)out_code, cur_stream()),
          "scn_conv_module_forward");
    ctx->save_for_backward({x, weight, bias, nbr_fwd, nbr_bwd, wimg_t});
    ctx->saved_data["n_out_rows"] = n_out_rows;
    ctx->saved_data["mirror"] = mirror;
    ctx->saved_data["prec"] = prec;
    ctx->saved_data["direct_w"] = direct_w;
    ctx->saved_data["direct_b"] = direct_b;
    ctx->saved_data["skip_prep"] = skip_prep;
    ctx->saved_data["wver"] = (int64_t)weight._version();
    return out;
  }

  static variable_list backward(AutogradContext* ctx, variable_list grads) {
    auto saved = ctx->get_saved_variables();
    at::Tensor x = saved[0], weight = saved[1], bias = saved[2], nbr_fwd = saved[3], nbr_bwd = saved[4], wimg_t = saved[5];
    at::Tensor dout = grads[0].contiguous();
    const int64_t K = weight.size(0), cin = weight.size(-2), cout = weight.size(-1);
    const bool need_dx = ctx->needs_input_grad(0), need_dw = ctx->needs_input_grad(1);
    const bool need_db = has(bias) && ctx->needs_input_grad(2);
    at::Tensor gw = need_dw ? direct_grad(weight, ctx->saved_data["direct_w"].toBool()) : at::Tensor();
    at::Tensor gb = need_db ? direct_grad(bias, ctx->saved_data["direct_b"].toBool()) : at::Tensor();
    at::Tensor dx, dw, db;
    if (need_dx) dx = at::empty({x.size(0), cin}, x.options());
    if (need_dw && !gw.defined()) dw = at::empty(weight.sizes(), weight.options().dtype(at::kFloat));
    if (need_db && !gb.defined()) db = at::empty(bias.sizes(), bias.options().dtype(at::kFloat));
    at::Tensor* wtarget = gw.defined() ? &gw : &dw;
    at::Tensor* btarget = gb.defined() ? &gb : &db;
    // bias gradient already summed by the BatchNorm backward that produced this grad_output?
    BnColsum& bc = last_bn_colsum();
    at::Tensor colsum;
    if (need_db && bc.dx.defined() && bc.dx.data_ptr() == dout.data_ptr() && bc.dx.sizes() == dout.sizes() &&
        bc.colsum.numel() == cout)
      colsum = bc.colsum;
    bc.dx = at::Tensor();
    bc.colsum = at::Tensor();
    double* ws = need_db ? stats_scratch(x.device(), cout).data_ptr<double>() : nullptr;
    TORCH_CHECK(!need_dx || has(wimg_t), "scn_b200: dgrad needs the transposed weight-image workspace");
    check(scn_conv_module_backward_colsum(x.data_ptr(), dcode(x), x.size(0), dout.data_ptr(), dcode(dout),
                                   ctx->saved_data["n_out_rows"].toInt(), nbr_fwd.data_ptr<int32_t>(), nbr_fwd.size(1),
                                   nbr_bwd.data_ptr<int32_t>(), nbr_bwd.size(1), (int)K, (int)cin, (int)cout,
                                   weight.data_ptr<float>(), ctx->saved_data["mirror"].toBool() ? 1 : 0,
                                   (int)ctx->saved_data["prec"].toInt(), optr(wimg_t), ctx->saved_data["skip_prep"].toBool() ? 1 : 0, optr(dx),
                                   wtarget->defined() ? wtarget->data_ptr<float>() : nullptr, gw.defined() ? 0 : 1,
                                   btarget->defined() ? btarget->data_ptr<float>() : nullptr, gb.defined() ? 1 : 0,
                                   colsum.defined() ? colsum.data_ptr<float>() : nullptr, ws, cur_stream()),
          "scn_conv_module_backward_colsum");
    if (gw.defined()) grad_ready(weight);
    if (gb.defined()) grad_ready(bias);
    return {dx, dw, db, at::Tensor(), at::Tensor(), at::Tensor(), at::Tensor(), at::Tensor(), at::Tensor(),
            at::Tensor(), at::Tensor(), at::Tensor(), at::Tensor(), at::Tensor()};
  }
};

struct BatchNormFn : public torch::autograd::Function<BatchNormFn> {
  static at::Tensor forward(AutogradContext* ctx, at::Tensor x, at::Tensor weight, at::Tensor bias, at::Tensor rm,
                            at::Tensor rv, bool training, double eps, double momentum, double leak, bool direct) {
    x = x.contiguous();
    const int64_t n = x.size(0), c = x.size(1);
    at::Tensor stats = at::empty({2, c}, x.options().dtype(at::kFloat));
    at::Tensor out = at::empty_like(x);
    float* sp = stats.data_ptr<float>();
    check(scn_bn_forward(x.data_ptr(), dcode(x), n, (int)c, has(weight) ? weight.data_ptr<float>() : nullptr,
                         has(bias) ? bias.data_ptr<float>() : nullptr, rm.data_ptr<float>(), rv.data_ptr<float>(),
                         training ? 1 : 0, (float)eps, (float)momentum, (float)leak, sp, sp + c,
                         stats_scratch(x.device(), c).data_ptr<double>(), out.data_ptr(), cur_stream()),
          "scn_bn_forward");
    ctx->save_for_backward({x, weight, bias, stats});
    ctx->saved_data["training"] = training;
    ctx->saved_data["leak"] = leak;
    ctx->saved_data["direct"] = direct;
    return out;
  }

  static variable_list backward(AutogradContext* ctx, variable_list grads) {
    auto saved = ctx->get_saved_variables();
    at::Tensor x = saved[0], weight = saved[1], bias = saved[2], stats = saved[3];
    at::Tensor dout = grads[0].contiguous();
    const int64_t n = x.size(0), c = x.size(1);
    const bool affine = has(weight);
    const bool direct = ctx->saved_data["direct"].toBool() && affine && ctx->needs_input_grad(1) && ctx->needs_input_grad(2);
    at::Tensor gw = direct_grad(weight, direct), gb = direct_grad(bias, direct);
    const bool acc = gw.defined() && gb.defined();
    at::Tensor both, dg, db;
    if (!acc) {
      both = at::empty({2, c}, x.options().dtype(at::kFloat));
      dg = both[0];
      db = both[1];
    }
    at::Tensor dx = at::empty_like(x);
    float* sp = stats.data_ptr<float>();
    const bool training = ctx->saved_data["training"].toBool();
    // training mode: the column sums of dx come out of the same pass (the bias gradient of a convolution in front)
    at::Tensor colsum = (training && n > 0) ? at::empty({c}, x.options().dtype(at::kFloat)) : at::Tensor();
    check(scn_bn_backward_colsum(x.data_ptr(), dout.data_ptr(), dcode(x), n, (int)c,
                                 affine ? weight.data_ptr<float>() : nullptr, affine ? bias.data_ptr<float>() : nullptr, sp,
                                 sp + c, training ? 1 : 0, (float)ctx->saved_data["leak"].toDouble(),
                                 stats_scratch(x.device(), c).data_ptr<double>(), dx.data_ptr(),
                                 acc ? gw.data_ptr<float>() : dg.data_ptr<float>(), acc ? gb.data_ptr<float>() : db.data_ptr<float>(),
                                 acc ? 1 : 0, colsum.defined() ? colsum.data_ptr<float>() : nullptr, cur_stream()),
          "scn_bn_backward_colsum");
    BnColsum& bc = last_bn_colsum();
    bc.dx = colsum.defined() ? dx : at::Tensor();
    bc.colsum = colsum;
    if (acc) {
      grad_ready(weight);
      grad_ready(bias);
      dg = at::Tensor();
      db = at::Tensor();
    }
    if (!affine) {
      dg = at::Tensor();
      db = at::Tensor();
    }
    return {dx, dg, db, at::Tensor(), at::Tensor(), at::Tensor(), at::Tensor(), at::Tensor(), at::Tensor(), at::Tensor()};
  }
};

struct AddLeakyFn : public torch::autograd::Function<AddLeakyFn> {
  static at::Tensor forward(AutogradContext* ctx, at::Tensor a, at::Tensor b, double leak) {
    a = a.contiguous();
    b = b.contiguous();
    at::Tensor out = at::empty_like(a);
    check(scn_add_forward(a.data_ptr(), b.data_ptr(), dcode(a), a.numel(), (float)leak, out.data_ptr(), cur_stream()),
          "scn_add_forward");
    if (leak != 1.0) ctx->save_for_backward({out});
    ctx->saved_data["leak"] = leak;
    return out;
  }
  static variable_list backward(AutogradContext* ctx, variable_list grads) {
    const double leak = ctx->saved_data["leak"].toDouble();
    if (leak == 1.0) return {grads[0], grads[0], at::Tensor()};
    at::Tensor out = ctx->get_saved_variables()[0];
    at::Tensor dout = grads[0].contiguous();
    at::Tensor d = at::empty_like(out);
    // sign(out) == sign(a + b) for leak > 0; for leak == 0 (ReLU) out > 0 <=> a + b > 0 as well
    check(scn_leaky_backward(out.data_ptr(), dout.data_ptr(), dcode(out), out.numel(), (float)leak, d.data_ptr(), cur_stream()),
          "scn_leaky_backward");
    return {d, d, at::Tensor()};
  }
};

struct LeakyFn : public torch::autograd::Function<LeakyFn> {
  static at::Tensor forward(AutogradContext* ctx, at::Tensor x, double leak) {
    x = x.contiguous();
    at::Tensor out = at::empty_like(x);
    check(scn_leaky_forward(x.data_ptr(), dcode(x), x.numel(), (float)leak, out.data_ptr(), cur_stream()), "scn_leaky_forward");
    ctx->save_for_backward({x});
    ctx->saved_data["leak"] = leak;
    return out;
  }
  static variable_list backward(AutogradContext* ctx, variable_list grads) {
    at::Tensor x = ctx->get_saved_variables()[0];
    at::Tensor dout = grads[0].contiguous();
    at::Tensor dx = at::empty_like(x);
    check(scn_leaky_backward(x.data_ptr(), dout.data_ptr(), dcode(x), x.numel(), (float)ctx->saved_data["leak"].toDouble(),
                             dx.data_ptr(), cur_stream()),
          "scn_leaky_backward");
    return {dx, at::Tensor()};
  }
};

// Function::apply wants defined tensors: an absent optional becomes an EMPTY fp32 tensor on x's device
at::Tensor opt(const c10::optional<at::Tensor>& t, const at::Tensor& like) {
  return t.has_value() ? *t : at::empty({0}, like.options().dtype(at::kFloat));
}

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "torch autograd functions of the sparse modules over libscn_b200.so";
  m.def("conv", [](at::Tensor x, at::Tensor weight, c10::optional<at::Tensor> bias, at::Tensor nbr_fwd, at::Tensor nbr_bwd,
                   int64_t n_out_rows, bool mirror, int64_t prec, int64_t out_code, at::Tensor wimg,
                   c10::optional<at::Tensor> wimg_t, bool skip_prep, bool direct_w, bool direct_b) {
    return ConvFn::apply(x, weight, opt(bias, x), nbr_fwd, nbr_bwd, n_out_rows, mirror, prec, out_code, wimg, opt(wimg_t, x),
                         skip_prep, direct_w, direct_b);
  });
  m.def("batch_norm", [](at::Tensor x, c10::optional<at::Tensor> weight, c10::optional<at::Tensor> bias, at::Tensor rm,
                         at::Tensor rv, bool training, double eps, double momentum, double leak, bool direct) {
    return BatchNormFn::apply(x, opt(weight, x), opt(bias, x), rm, rv, training, eps, momentum, leak, direct);
  });
  m.def("add_leaky", [](at::Tensor a, at::Tensor b, double leak) { return AddLeakyFn::apply(a, b, leak); });
  m.def("leaky", [](at::Tensor x, double leak) { return LeakyFn::apply(x, leak); });
  m.def("set_grad_ready_callback", [](py::object cb) {
    if (g_ready_cb == nullptr) g_ready_cb = new py::object();
    *g_ready_cb = cb;
  });
}
