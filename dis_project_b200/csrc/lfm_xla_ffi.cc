// XLA FFI custom-call handlers over the C-ABI of include/lfm_b200.h: the route by which the reference's
// `jax.value_and_grad(self.loss)` (src/trainer.py:126), `CustomConjMLL.step` (src/objectives.py:64-78),
// `ExactLFM.latent_predict / multi_gene_predict / cross_covariance` (src/model.py:372-514) reach the sm_100a kernels
// from inside jit / grad / lax.scan (north_star: "a thin C-ABI registered as JAX FFI custom calls").
//
// OPTIONAL translation unit: it needs `xla/ffi/api/ffi.h`, which ships with jaxlib (`jax.ffi.include_dir()`, JAX >= 0.4.31;
// the reference pins 0.4.28, which predates the public FFI module).  The build image has neither JAX nor the header, so
// `make xla_ffi` builds liblfm_xla_ffi.so only where the header is found (XLA_FFI_INCLUDE=... or an importable jax);
// tests/test_host.py compiles this file against a structural mock of the header so that the handler signatures stay in
// step with the bindings.  dis_project_b200/jax_ffi.py registers the targets and wraps the objective in jax.custom_vjp.
//
// Contract of every handler = contract of the C-ABI: XLA owns every buffer and the stream; nothing here allocates,
// synchronises or throws; scratch is an extra RESULT buffer sized by the *_workspace_bytes queries at trace time;
// a numerical failure (Sigma not positive definite) is reported through the `info` result and NaN outputs, like JAX's
// own Cholesky; an lfm_status error becomes an ffi::Error.
#include <cuda_runtime_api.h>

#include <cstdint>

#include "xla/ffi/api/ffi.h"

#include "../../include/lfm_b200.h"

namespace ffi = xla::ffi;

namespace {

using F64 = ffi::Buffer<ffi::F64>;
using RF64 = ffi::ResultBuffer<ffi::F64>;
using RS32 = ffi::ResultBuffer<ffi::S32>;
using RU8 = ffi::ResultBuffer<ffi::U8>;

inline ffi::Error status(int st) {
  return st == LFM_OK ? ffi::Error::Success() : ffi::Error(ffi::ErrorCode::kInternal, lfm_status_string(st));
}
inline int64_t rows(const F64& x) { return x.dimensions().size() ? (int64_t)x.dimensions()[0] : 0; }
// `variances` is an optional operand: an empty (0-element) array selects the homoscedastic objective
inline const double* optional(const F64& v) { return v.element_count() ? v.typed_data() : nullptr; }

// CustomConjMLL(negative=True)(model, Dataset(X, y))            src/objectives.py:21-78   -> out[1]
ffi::Error Nlml(cudaStream_t stream, F64 X, F64 y, F64 variances, F64 theta, double jitter, int64_t G, int64_t time_grid,
                RF64 out, RS32 info, RU8 ws) {
  return status(lfm_nlml_het_tg(stream, rows(X), (int)G, X.typed_data(), y.typed_data(), optional(variances),
                                theta.typed_data(), jitter, time_grid, ws->typed_data(), ws->element_count(),
                                out->typed_data(), info->typed_data()));
}
// value and gradient w.r.t. the CONSTRAINED theta                                           -> out[1 + P]
ffi::Error NlmlGrad(cudaStream_t stream, F64 X, F64 y, F64 variances, F64 theta, double jitter, int64_t G,
                    int64_t time_grid, RF64 out, RS32 info, RU8 ws) {
  return status(lfm_nlml_grad_het_tg(stream, rows(X), (int)G, X.typed_data(), y.typed_data(), optional(variances),
                                     theta.typed_data(), jitter, time_grid, ws->typed_data(), ws->element_count(),
                                     out->typed_data(), info->typed_data()));
}
// jax.value_and_grad(JaxTrainer.loss) w.r.t. the UNCONSTRAINED leaves   src/trainer.py:86-103,126   -> out[1 + P]
ffi::Error NlmlGradUnc(cudaStream_t stream, F64 X, F64 y, F64 variances, F64 theta_unc, double jitter, int64_t G,
                       int64_t time_grid, RF64 out, RS32 info, RU8 ws) {
  return status(lfm_nlml_grad_unc_het_tg(stream, rows(X), (int)G, X.typed_data(), y.typed_data(), optional(variances),
                                         theta_unc.typed_data(), jitter, time_grid, ws->typed_data(),
                                         ws->element_count(), out->typed_data(), info->typed_data()));
}
// ExactLFM.cross_covariance(kernel, x, y) / gram                          src/model.py:372-414        -> out[N, M]
ffi::Error CrossCovariance(cudaStream_t stream, F64 X, F64 Y, F64 theta, int64_t G, RF64 out) {
  const int64_t M = rows(Y);
  return status(lfm_cross_covariance(stream, rows(X), M, X.typed_data(), Y.typed_data(), (int)G, theta.typed_data(),
                                     out->typed_data(), M));
}
// ExactLFM.mean_function(x)                                               src/model.py:124-149        -> out[N]
ffi::Error MeanFunction(cudaStream_t stream, F64 X, F64 theta, int64_t G, RF64 out) {
  return status(lfm_mean_function(stream, rows(X), X.typed_data(), (int)G, theta.typed_data(), out->typed_data()));
}
// ExactLFM.latent_predict(test_inputs, train_data)                        src/model.py:420-463        -> mean, var [T*]
ffi::Error LatentPosterior(cudaStream_t stream, F64 X, F64 y, F64 variances, F64 theta, F64 Xstar, double jitter,
                           int64_t G, RF64 mean, RF64 var, RS32 info, RU8 ws) {
  return status(lfm_latent_posterior(stream, rows(X), (int)G, X.typed_data(), y.typed_data(), variances.typed_data(),
                                     theta.typed_data(), jitter, rows(Xstar), Xstar.typed_data(), ws->typed_data(),
                                     ws->element_count(), mean->typed_data(), var->typed_data(), info->typed_data()));
}
// ExactLFM.multi_gene_predict(test_inputs, train_data)                    src/model.py:465-514        -> mean, cov, var
ffi::Error GenePosterior(cudaStream_t stream, F64 X, F64 y, F64 variances, F64 theta, F64 Xstar, double jitter,
                         int64_t G, RF64 mean, RF64 cov, RF64 var, RS32 info, RU8 ws) {
  return status(lfm_gene_posterior(stream, rows(X), (int)G, X.typed_data(), y.typed_data(), variances.typed_data(),
                                   theta.typed_data(), jitter, rows(Xstar), Xstar.typed_data(), ws->typed_data(),
                                   ws->element_count(), mean->typed_data(), cov->typed_data(), var->typed_data(),
                                   info->typed_data()));
}
// B independent JaxTrainer.fit loops                                      src/trainer.py:162-228
// theta_unc (B x P) and adam (B x 2P) are operands that XLA aliases to the results of the same name
// (input_output_aliases in the ffi_call), so the kernel updates them in place.
ffi::Error BatchedFit(cudaStream_t stream, F64 X, F64 y, F64 theta_unc_in, F64 adam_in, double jitter, double lr, double b1,
                      double b2, double eps, int64_t G, int64_t steps, int64_t fix_params, int64_t steps_per_epoch,
                      int64_t unique_rows, int64_t time_grid, RF64 theta_unc, RF64 adam, RF64 hist, RF64 theta,
                      RS32 info) {
  const int64_t B = theta_unc_in.dimensions().size() ? (int64_t)theta_unc_in.dimensions()[0] : 0;
  const int64_t N = rows(X);
  const size_t P = 3 * (size_t)G + 2;
  if (theta_unc->typed_data() != theta_unc_in.typed_data()) {   // not aliased by the caller: carry the state over
    if (cudaMemcpyAsync(theta_unc->typed_data(), theta_unc_in.typed_data(), (size_t)B * P * 8, cudaMemcpyDeviceToDevice,
                        stream) != cudaSuccess)
      return status(LFM_ERR_CUDA);
  }
  if (adam->typed_data() != adam_in.typed_data()) {
    if (cudaMemcpyAsync(adam->typed_data(), adam_in.typed_data(), (size_t)B * 2 * P * 8, cudaMemcpyDeviceToDevice,
                        stream) != cudaSuccess)
      return status(LFM_ERR_CUDA);
  }
  // y is (N,) -- every LFM fits the same observations -- or (B, N): one row per LFM
  const int64_t y_stride = y.dimensions().size() == 2 ? N : 0;
  return status(lfm_batched_fit_het(stream, B, N, (int)G, X.typed_data(), y.typed_data(), y_stride, nullptr, 0,
                                    theta_unc->typed_data(), adam->typed_data(), jitter, lr, b1, b2, eps, 0, (int)steps,
                                    (int)steps, (int)fix_params, (int)steps_per_epoch, (int)unique_rows, (int)time_grid,
                                    hist->typed_data(), steps, theta->typed_data(), info->typed_data(), nullptr,
                                    nullptr, nullptr, 0, nullptr, 0));
}

}  // namespace

#define LFM_STREAM Ctx<ffi::PlatformStream<cudaStream_t>>()

XLA_FFI_DEFINE_HANDLER_SYMBOL(LfmNlml, Nlml,
                              ffi::Ffi::Bind().LFM_STREAM.Arg<F64>().Arg<F64>().Arg<F64>().Arg<F64>()
                                  .Attr<double>("jitter").Attr<int64_t>("G").Attr<int64_t>("time_grid")
                                  .Ret<F64>().Ret<ffi::Buffer<ffi::S32>>().Ret<ffi::Buffer<ffi::U8>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(LfmNlmlGrad, NlmlGrad,
                              ffi::Ffi::Bind().LFM_STREAM.Arg<F64>().Arg<F64>().Arg<F64>().Arg<F64>()
                                  .Attr<double>("jitter").Attr<int64_t>("G").Attr<int64_t>("time_grid")
                                  .Ret<F64>().Ret<ffi::Buffer<ffi::S32>>().Ret<ffi::Buffer<ffi::U8>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(LfmNlmlGradUnc, NlmlGradUnc,
                              ffi::Ffi::Bind().LFM_STREAM.Arg<F64>().Arg<F64>().Arg<F64>().Arg<F64>()
                                  .Attr<double>("jitter").Attr<int64_t>("G").Attr<int64_t>("time_grid")
                                  .Ret<F64>().Ret<ffi::Buffer<ffi::S32>>().Ret<ffi::Buffer<ffi::U8>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(LfmCrossCovariance, CrossCovariance,
                              ffi::Ffi::Bind().LFM_STREAM.Arg<F64>().Arg<F64>().Arg<F64>().Attr<int64_t>("G").Ret<F64>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(LfmMeanFunction, MeanFunction,
                              ffi::Ffi::Bind().LFM_STREAM.Arg<F64>().Arg<F64>().Attr<int64_t>("G").Ret<F64>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(LfmLatentPosterior, LatentPosterior,
                              ffi::Ffi::Bind().LFM_STREAM.Arg<F64>().Arg<F64>().Arg<F64>().Arg<F64>().Arg<F64>()
                                  .Attr<double>("jitter").Attr<int64_t>("G")
                                  .Ret<F64>().Ret<F64>().Ret<ffi::Buffer<ffi::S32>>().Ret<ffi::Buffer<ffi::U8>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(LfmGenePosterior, GenePosterior,
                              ffi::Ffi::Bind().LFM_STREAM.Arg<F64>().Arg<F64>().Arg<F64>().Arg<F64>().Arg<F64>()
                                  .Attr<double>("jitter").Attr<int64_t>("G")
                                  .Ret<F64>().Ret<F64>().Ret<F64>().Ret<ffi::Buffer<ffi::S32>>().Ret<ffi::Buffer<ffi::U8>>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(LfmBatchedFit, BatchedFit,
                              ffi::Ffi::Bind().LFM_STREAM.Arg<F64>().Arg<F64>().Arg<F64>().Arg<F64>()
                                  .Attr<double>("jitter").Attr<double>("lr").Attr<double>("b1").Attr<double>("b2")
                                  .Attr<double>("eps").Attr<int64_t>("G").Attr<int64_t>("steps")
                                  .Attr<int64_t>("fix_params").Attr<int64_t>("steps_per_epoch")
                                  .Attr<int64_t>("unique_rows").Attr<int64_t>("time_grid")
                                  .Ret<F64>().Ret<F64>().Ret<F64>().Ret<F64>().Ret<ffi::Buffer<ffi::S32>>());
