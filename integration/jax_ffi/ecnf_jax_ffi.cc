// XLA typed-FFI handlers over the C-ABI of libecnf_b200.so: the `jax.ffi` custom calls BASELINE.json's north_star asks for.
//
// NOT BUILT IN THIS REPOSITORY'S IMAGE: it needs jaxlib's headers (xla/ffi/api/ffi.h), and neither JAX nor XLA is
// installed here (DESIGN.md section 1).  With JAX present:
//
//   g++ -O2 -std=c++17 -fPIC -shared ecnf_jax_ffi.cc -o libecnf_jax_ffi.so \
//       -I$(python -c "import jax.ffi; print(jax.ffi.include_dir())") -I../../include -I/usr/local/cuda/include \
//       -L../../ecnf_b200 -lecnf_b200 -Wl,-rpath,'$ORIGIN/../../ecnf_b200'
//
// One handler per entry point of include/ecnf_b200.h.  Conventions:
//   * `model` (int64 attribute) is the address of a TEMPLATE handle made once on the host with ecnf_model_create (it
//     carries the hyper-parameters, the engine choice and the training chunk size); the parameters arrive per call as a
//     buffer, and every handler binds them with ecnf_model_clone -> launch -> ecnf_model_destroy (host-side, no device
//     work; kernel arguments are copied at launch), so handlers are re-entrant across streams and threads;
//   * ecnf_solve_ctrl travels as scalar attributes (fixed, step_size, rtol, atol, dtmin, max_steps, err_scale);
//   * the workspace is an operand sized by the Python side with ecnf_*_workspace_bytes (the library never allocates);
//   * a non-zero return code becomes ffi::Error::Internal(ecnf_last_error()).
#include <cstdint>
#include <vector>

#include <cuda_runtime_api.h>

#include "ecnf_b200.h"
#include "xla/ffi/api/ffi.h"

namespace ffi = xla::ffi;

namespace {

struct Bound {      // the template handle bound to this call's parameter buffer
  ecnf_model* m = nullptr;
  Bound(int64_t model, const float* params) { ecnf_model_clone(reinterpret_cast<const ecnf_model*>(model), params, &m); }
  ~Bound() { if (m) ecnf_model_destroy(m); }
  Bound(const Bound&) = delete;
  Bound& operator=(const Bound&) = delete;
};

ffi::Error Status(int rc) { return rc == 0 ? ffi::Error::Success() : ffi::Error::Internal(ecnf_last_error()); }

ecnf_solve_ctrl Ctrl(int32_t fixed, float step_size, float rtol, float atol, float dtmin, int32_t max_steps, float err_scale) {
  return ecnf_solve_ctrl{fixed, step_size, rtol, atol, dtmin, max_steps, 0.9f, 0.2f, 10.f, 5.f, err_scale};
}

// cnf.apply(params, x, t, features)  (build_cnf.py:68-93)
ffi::Error VfForwardImpl(cudaStream_t stream, int64_t model, ffi::Buffer<ffi::F32> params, ffi::Buffer<ffi::F32> x,
                         ffi::Buffer<ffi::F32> t, ffi::Buffer<ffi::S32> feat, ffi::Buffer<ffi::U8> ws,
                         ffi::ResultBuffer<ffi::F32> out_f) {
  Bound b(model, params.typed_data());
  const int64_t B = x.dimensions()[0];
  return Status(ecnf_vf_forward(b.m, x.typed_data(), t.typed_data(), feat.typed_data(), B, out_f->typed_data(),
                                ws.untyped_data(), (int64_t)ws.size_bytes(), stream));
}

// joint_vector_field with the exact trace  (sample_and_log_prob.py:58-67)
ffi::Error VfForwardDivImpl(cudaStream_t stream, int64_t model, ffi::Buffer<ffi::F32> params, ffi::Buffer<ffi::F32> x,
                            ffi::Buffer<ffi::F32> t, ffi::Buffer<ffi::S32> feat, ffi::Buffer<ffi::U8> ws,
                            ffi::ResultBuffer<ffi::F32> out_f, ffi::ResultBuffer<ffi::F32> out_div) {
  Bound b(model, params.typed_data());
  const int64_t B = x.dimensions()[0];
  return Status(ecnf_vf_forward_div(b.m, x.typed_data(), t.typed_data(), feat.typed_data(), B, out_f->typed_data(),
                                    out_div->typed_data(), ws.untyped_data(), (int64_t)ws.size_bytes(), stream));
}

// joint_vector_field with the Hutchinson estimate  (sample_and_log_prob.py:69-78)
ffi::Error VfForwardHutchinsonImpl(cudaStream_t stream, int64_t model, ffi::Buffer<ffi::F32> params, ffi::Buffer<ffi::F32> x,
                                   ffi::Buffer<ffi::F32> t, ffi::Buffer<ffi::S32> feat, ffi::Buffer<ffi::F32> eps,
                                   ffi::Buffer<ffi::U8> ws, ffi::ResultBuffer<ffi::F32> out_f,
                                   ffi::ResultBuffer<ffi::F32> out_div) {
  Bound b(model, params.typed_data());
  const int64_t B = x.dimensions()[0];
  return Status(ecnf_vf_forward_hutchinson(b.m, x.typed_data(), t.typed_data(), feat.typed_data(), eps.typed_data(), B,
                                           out_f->typed_data(), out_div->typed_data(), ws.untyped_data(),
                                           (int64_t)ws.size_bytes(), stream));
}

// diffeqsolve call sites of sample_cnf / get_log_prob / sample_and_log_prob_cnf  (sample_and_log_prob.py:33-37,85-89,140-144)
ffi::Error SolveImpl(cudaStream_t stream, int64_t model, int32_t mode, int32_t fixed, float step_size, float rtol, float atol,
                     float dtmin, int32_t max_steps, float err_scale, ffi::Buffer<ffi::F32> params,
                     ffi::Buffer<ffi::F32> x_init, ffi::Buffer<ffi::S32> feat, ffi::Buffer<ffi::U8> ws,
                     ffi::ResultBuffer<ffi::F32> out_x, ffi::ResultBuffer<ffi::F32> out_logs,
                     ffi::ResultBuffer<ffi::S32> out_stats) {
  Bound b(model, params.typed_data());
  const int64_t B = x_init.dimensions()[0];
  const ecnf_solve_ctrl ctrl = Ctrl(fixed, step_size, rtol, atol, dtmin, max_steps, err_scale);
  return Status(ecnf_solve(b.m, mode, x_init.typed_data(), feat.typed_data(), B, &ctrl, out_x->typed_data(),
                           out_logs->typed_data(), out_stats->typed_data(), ws.untyped_data(), (int64_t)ws.size_bytes(),
                           stream));
}

// the approx=True branches: one probe per trajectory, fixed for the whole solve  (sample_and_log_prob.py:69-78,123-133)
ffi::Error SolveHutchinsonImpl(cudaStream_t stream, int64_t model, int32_t mode, int32_t fixed, float step_size, float rtol,
                               float atol, float dtmin, int32_t max_steps, float err_scale, ffi::Buffer<ffi::F32> params,
                               ffi::Buffer<ffi::F32> x_init, ffi::Buffer<ffi::S32> feat, ffi::Buffer<ffi::F32> eps,
                               ffi::Buffer<ffi::U8> ws, ffi::ResultBuffer<ffi::F32> out_x,
                               ffi::ResultBuffer<ffi::F32> out_logs, ffi::ResultBuffer<ffi::S32> out_stats) {
  Bound b(model, params.typed_data());
  const int64_t B = x_init.dimensions()[0];
  const ecnf_solve_ctrl ctrl = Ctrl(fixed, step_size, rtol, atol, dtmin, max_steps, err_scale);
  return Status(ecnf_solve_hutchinson(b.m, mode, x_init.typed_data(), feat.typed_data(), eps.typed_data(), B, &ctrl,
                                      out_x->typed_data(), out_logs->typed_data(), out_stats->typed_data(),
                                      ws.untyped_data(), (int64_t)ws.size_bytes(), stream));
}

// jaxlib decodes an array attribute into a host ffi::Span<const T>.  The minimal header stand-in the syntax test compiles
// against (tests/mock_xla) has no Span; there a vector, which has the same begin() / end(), takes its place.
#ifdef XLA_FFI_API_FFI_H_
using F32Array = ffi::Span<const float>;
#else
using F32Array = std::vector<float>;
#endif

// diffeqsolve(..., saveat=SaveAt(ts=ts)): the solve + the path at the times of the array attribute `ts`, which the library
// copies into the workspace before returning (eps: the Hutchinson probes, or a zero-size operand for the exact trace;
// out_traj_delta: a zero-size result in SAMPLE mode)
ffi::Error SolveSaveatImpl(cudaStream_t stream, int64_t model, int32_t mode, int32_t fixed, float step_size, float rtol,
                           float atol, float dtmin, int32_t max_steps, float err_scale, F32Array ts,
                           ffi::Buffer<ffi::F32> params, ffi::Buffer<ffi::F32> x_init, ffi::Buffer<ffi::S32> feat,
                           ffi::Buffer<ffi::F32> eps, ffi::Buffer<ffi::U8> ws, ffi::ResultBuffer<ffi::F32> out_x,
                           ffi::ResultBuffer<ffi::F32> out_logs, ffi::ResultBuffer<ffi::S32> out_stats,
                           ffi::ResultBuffer<ffi::F32> out_traj, ffi::ResultBuffer<ffi::F32> out_traj_delta) {
  Bound b(model, params.typed_data());
  const int64_t B = x_init.dimensions()[0];
  const ecnf_solve_ctrl ctrl = Ctrl(fixed, step_size, rtol, atol, dtmin, max_steps, err_scale);
  const std::vector<float> t(ts.begin(), ts.end());
  return Status(ecnf_solve_saveat(b.m, mode, x_init.typed_data(), feat.typed_data(),
                                  eps.element_count() ? eps.typed_data() : nullptr, B, &ctrl, (int)t.size(), t.data(),
                                  out_x->typed_data(), out_logs->typed_data(), out_stats->typed_data(),
                                  out_traj->typed_data(), out_traj_delta->typed_data(), ws.untyped_data(),
                                  (int64_t)ws.size_bytes(), stream));
}

// x0 = base_scale * remove_mean(eps) with eps = jax.random.normal(key, ...) drawn on the JAX side  (zero_com_base.py:44-47)
ffi::Error BaseSampleFromNoiseImpl(cudaStream_t stream, int64_t model, ffi::Buffer<ffi::F32> eps,
                                   ffi::ResultBuffer<ffi::F32> out_x0) {
  return Status(ecnf_base_sample_from_noise(reinterpret_cast<const ecnf_model*>(model), eps.typed_data(),
                                            eps.dimensions()[0], out_x0->typed_data(), stream));
}

// cnf.log_prob_base  (build_cnf.py:49-55, zero_com_base.py:64-84)
ffi::Error BaseLogProbImpl(cudaStream_t stream, int64_t model, ffi::Buffer<ffi::F32> x, ffi::ResultBuffer<ffi::F32> out) {
  return Status(ecnf_base_log_prob(reinterpret_cast<const ecnf_model*>(model), x.typed_data(), x.dimensions()[0],
                                   out->typed_data(), stream));
}

// flow_matching_loss_fn + jax.grad  (loss.py:10-32, gradient_step.py:31-37); x0 and t are drawn on the JAX side
ffi::Error FmLossGradImpl(cudaStream_t stream, int64_t model, float loss_denominator, ffi::Buffer<ffi::F32> params,
                          ffi::Buffer<ffi::F32> x_data, ffi::Buffer<ffi::F32> x0, ffi::Buffer<ffi::F32> t,
                          ffi::Buffer<ffi::S32> feat, ffi::Buffer<ffi::U8> ws, ffi::ResultBuffer<ffi::F32> out_loss,
                          ffi::ResultBuffer<ffi::F32> out_grad) {
  Bound b(model, params.typed_data());
  const int64_t B = x_data.dimensions()[0];
  return Status(ecnf_fm_loss_grad(b.m, x_data.typed_data(), x0.typed_data(), t.typed_data(), feat.typed_data(), B,
                                  loss_denominator, out_loss->typed_data(), out_grad->typed_data(), ws.untyped_data(),
                                  (int64_t)ws.size_bytes(), stream));
}

// optax.adam + EMA + norms  (gradient_step.py:39-50).  The four state buffers are updated in place: the Python side passes
// input_output_aliases {params: 0, mu: 1, nu: 2, ema: 3}, so each result buffer IS the corresponding operand.
ffi::Error AdamStepImpl(cudaStream_t stream, int64_t count, int64_t step, float lr, float b1, float b2, float eps,
                        float ema_beta, ffi::Buffer<ffi::F32> params, ffi::Buffer<ffi::F32> grad, ffi::Buffer<ffi::F32> mu,
                        ffi::Buffer<ffi::F32> nu, ffi::Buffer<ffi::F32> ema, ffi::ResultBuffer<ffi::F32> params_out,
                        ffi::ResultBuffer<ffi::F32> mu_out, ffi::ResultBuffer<ffi::F32> nu_out,
                        ffi::ResultBuffer<ffi::F32> ema_out, ffi::ResultBuffer<ffi::F32> out_norms) {
  if (params_out->typed_data() != params.typed_data() || mu_out->typed_data() != mu.typed_data() ||
      nu_out->typed_data() != nu.typed_data() || ema_out->typed_data() != ema.typed_data())
    return ffi::Error::InvalidArgument("ecnf_adam_step: pass input_output_aliases for params, mu, nu and ema");
  return Status(ecnf_adam_step(params_out->typed_data(), grad.typed_data(), mu_out->typed_data(), nu_out->typed_data(),
                               ema_out->typed_data(), count, step, lr, b1, b2, eps, ema_beta, out_norms->typed_data(),
                               stream));
}

// sufficient statistics of the reverse / forward ESS  (setup_training.py:175-182, utils/evaluation.py:10-22)
ffi::Error EssStatsImpl(cudaStream_t stream, ffi::Buffer<ffi::F32> log_w, ffi::ResultBuffer<ffi::F32> out5) {
  return Status(ecnf_ess_stats(log_w.typed_data(), (int64_t)log_w.element_count(), out5->typed_data(), stream));
}

// log p = -E of the LJ / DW targets  (leonard_jones.py:10-27, double_well.py:9-19)
ffi::Error TargetLogProbImpl(cudaStream_t stream, int32_t kind, int32_t n_frames, int32_t dim, ffi::Buffer<ffi::F32> x,
                             ffi::ResultBuffer<ffi::F32> out) {
  return Status(ecnf_target_log_prob(kind, x.typed_data(), x.dimensions()[0], n_frames, dim, out->typed_data(), stream));
}

using Stream = ffi::PlatformStream<cudaStream_t>;
using F32 = ffi::Buffer<ffi::F32>;
using S32 = ffi::Buffer<ffi::S32>;
using U8 = ffi::Buffer<ffi::U8>;

}  // namespace

XLA_FFI_DEFINE_HANDLER_SYMBOL(EcnfVfForward, VfForwardImpl,
                              ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("model").Arg<F32>().Arg<F32>().Arg<F32>().Arg<S32>()
                                  .Arg<U8>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(EcnfVfForwardDiv, VfForwardDivImpl,
                              ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("model").Arg<F32>().Arg<F32>().Arg<F32>().Arg<S32>()
                                  .Arg<U8>().Ret<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(EcnfVfForwardHutchinson, VfForwardHutchinsonImpl,
                              ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("model").Arg<F32>().Arg<F32>().Arg<F32>().Arg<S32>()
                                  .Arg<F32>().Arg<U8>().Ret<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(EcnfSolve, SolveImpl,
                              ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("model").Attr<int32_t>("mode").Attr<int32_t>("fixed")
                                  .Attr<float>("step_size").Attr<float>("rtol").Attr<float>("atol").Attr<float>("dtmin")
                                  .Attr<int32_t>("max_steps").Attr<float>("err_scale").Arg<F32>().Arg<F32>().Arg<S32>().Arg<U8>()
                                  .Ret<F32>().Ret<F32>().Ret<S32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(EcnfSolveHutchinson, SolveHutchinsonImpl,
                              ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("model").Attr<int32_t>("mode").Attr<int32_t>("fixed")
                                  .Attr<float>("step_size").Attr<float>("rtol").Attr<float>("atol").Attr<float>("dtmin")
                                  .Attr<int32_t>("max_steps").Attr<float>("err_scale").Arg<F32>().Arg<F32>().Arg<S32>().Arg<F32>()
                                  .Arg<U8>().Ret<F32>().Ret<F32>().Ret<S32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(EcnfSolveSaveat, SolveSaveatImpl,
                              ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("model").Attr<int32_t>("mode").Attr<int32_t>("fixed")
                                  .Attr<float>("step_size").Attr<float>("rtol").Attr<float>("atol").Attr<float>("dtmin")
                                  .Attr<int32_t>("max_steps").Attr<float>("err_scale").Attr<F32Array>("ts").Arg<F32>()
                                  .Arg<F32>().Arg<S32>().Arg<F32>().Arg<U8>().Ret<F32>().Ret<F32>().Ret<S32>().Ret<F32>()
                                  .Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(EcnfBaseSampleFromNoise, BaseSampleFromNoiseImpl,
                              ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("model").Arg<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(EcnfBaseLogProb, BaseLogProbImpl,
                              ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("model").Arg<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(EcnfFmLossGrad, FmLossGradImpl,
                              ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("model").Attr<float>("loss_denominator").Arg<F32>()
                                  .Arg<F32>().Arg<F32>().Arg<F32>().Arg<S32>().Arg<U8>().Ret<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(EcnfAdamStep, AdamStepImpl,
                              ffi::Ffi::Bind().Ctx<Stream>().Attr<int64_t>("count").Attr<int64_t>("step").Attr<float>("lr")
                                  .Attr<float>("b1").Attr<float>("b2").Attr<float>("eps").Attr<float>("ema_beta").Arg<F32>()
                                  .Arg<F32>().Arg<F32>().Arg<F32>().Arg<F32>().Ret<F32>().Ret<F32>().Ret<F32>().Ret<F32>()
                                  .Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(EcnfEssStats, EssStatsImpl, ffi::Ffi::Bind().Ctx<Stream>().Arg<F32>().Ret<F32>());
XLA_FFI_DEFINE_HANDLER_SYMBOL(EcnfTargetLogProb, TargetLogProbImpl,
                              ffi::Ffi::Bind().Ctx<Stream>().Attr<int32_t>("kind").Attr<int32_t>("n_frames").Attr<int32_t>("dim")
                                  .Arg<F32>().Ret<F32>());
