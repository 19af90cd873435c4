// C-ABI entry points of engine A (dispatch over the compiled (U, H) instantiations).
// Kernel: ecnf_solve_impl.cuh; instantiations: ecnf_solve_inst_*.cu (one translation unit each so they build in parallel).
#include <vector>

#include "ecnf_solve_decl.cuh"

using namespace ecnf_solve_detail;

namespace {

template <bool DIV, bool SAVE>
int launch_uh(const ecnf_model* mdl, KernelArgs& a, int grid, cudaStream_t st) {
  const int U = mdl->cfg.mlp_units, H = mdl->cfg.n_hidden;
  if (U == 128 && H == 64) return launch_t<128, 64, DIV, SAVE>(mdl, a, grid, st);
  if (U == 256 && H == 32) return launch_t<256, 32, DIV, SAVE>(mdl, a, grid, st);
  if (U == 64 && H == 32) return launch_t<64, 32, DIV, SAVE>(mdl, a, grid, st);
  ecnf_set_error("unsupported (mlp_units=%d, n_hidden=%d): compiled pairs are (128,64), (256,32), (64,32)", U, H);
  return ECNF_ERR_UNSUPPORTED;
}

template <bool DIV>
int simt_check_uh(const ecnf_model* mdl) {
  const int U = mdl->cfg.mlp_units, H = mdl->cfg.n_hidden;
  if (U == 128 && H == 64) return simt_check<128, 64, DIV>(mdl);
  if (U == 256 && H == 32) return simt_check<256, 32, DIV>(mdl);
  if (U == 64 && H == 32) return simt_check<64, 32, DIV>(mdl);
  ecnf_set_error("unsupported (mlp_units=%d, n_hidden=%d): compiled pairs are (128,64), (256,32), (64,32)", U, H);
  return ECNF_ERR_UNSUPPORTED;
}

int grid_for(const ecnf_model* m, int64_t B) {
  int64_t g = m->num_sms;
  if (B < g) g = B;
  if (g < 1) g = 1;
  return (int)g;
}

bool use_tc(const ecnf_model* m, bool div) {   // m->engine: 0 = auto (tensor cores where eligible), 1 = fp32 SIMT
  return m->engine == 0 && tc_eligible(m, div);
}

int64_t scratch_stride_of(const ecnf_model* m, bool div) {
  return (scratch_floats(m->cfg.n_frames, m->cfg.dim, m->cfg.n_hidden, m->cfg.mlp_units, div) + 63) & ~63LL;
}

bool mode_div(int mode) { return mode == ECNF_MODE_VF_DIV || mode == ECNF_MODE_SAMPLE_LOGQ || mode == ECNF_MODE_LOGPROB; }

int64_t round256(int64_t v) { return (v + 255) & ~255LL; }

// SaveAt(ts) of one solve call: the internal save times already in the workspace, and where the path goes
struct SaveArgs {
  const float* ts = nullptr;
  int n_save = 0;
  float* out_traj = nullptr;
  float* out_traj_delta = nullptr;
};

int run(const ecnf_model* m, int mode, const float* x, const float* t, const int32_t* feat, const float* eps, int64_t B,
        const ecnf_solve_ctrl* ctrl, float* out_x, float* out_logs, int32_t* out_stats, void* ws, int64_t ws_bytes,
        void* stream, const SaveArgs& sv = SaveArgs()) {
  if (!m || !x || !feat || !out_x || B < 0) {
    ecnf_set_error("ecnf_solve: null argument");
    return ECNF_ERR_INVALID;
  }
  if (B == 0) return ECNF_OK;
  const int64_t need = ecnf_solve_workspace_bytes(m, mode, B);
  if (!ws || ws_bytes < need) {
    ecnf_set_error("workspace too small: need %lld bytes, got %lld", (long long)need, (long long)ws_bytes);
    return ECNF_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const bool div = mode_div(mode);
  const bool tc = use_tc(m, div);           // (Hutchinson probes: the tensor-core engine carries one tangent direction)
  const int grid = grid_for(m, B);
  KernelArgs a;
  a.m = ecnf_make_dev(m, m->d_params);
  a.mode = mode;
  a.B = B;
  a.x_init = x;
  a.t_in = t;
  a.feat = feat;
  a.eps = div ? eps : nullptr;
  if (ctrl) a.ctrl = *ctrl;
  else a.ctrl = ecnf_solve_ctrl{0, 0.05f, 1e-5f, 1e-5f, 1e-5f, 4096, 0.9f, 0.2f, 10.f, 5.f, 1.f};
  if (!(a.ctrl.err_scale > 0.f)) a.ctrl.err_scale = 1.f;
  a.out_x = out_x;
  a.out_logs = out_logs;
  a.out_stats = out_stats;
  a.counter = reinterpret_cast<unsigned int*>(ws);
  a.scratch = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + 256);
  a.scratch_stride = scratch_stride_of(m, div);
  a.img.base = nullptr;
  a.ts = sv.ts;
  a.n_save = sv.n_save;
  a.out_traj = sv.out_traj;
  a.out_traj_delta = sv.out_traj_delta;
  const bool save = sv.n_save > 0;
  ECNF_CHECK_CUDA(cudaMemsetAsync(ws, 0, 256, st));
  if (tc) {
    void* image_ws = reinterpret_cast<char*>(ws) + 256 + (int64_t)grid * a.scratch_stride * (int64_t)sizeof(float);
    return launch_tc(m, a, grid, image_ws, div, save, st);
  }
  if (save) return div ? launch_uh<true, true>(m, a, grid, st) : launch_uh<false, true>(m, a, grid, st);
  return div ? launch_uh<true, false>(m, a, grid, st) : launch_uh<false, false>(m, a, grid, st);
}

// checks shared by ecnf_solve_hutchinson and ecnf_solve_saveat
int check_solve_args(int mode, const float* out_logs, const ecnf_solve_ctrl* ctrl) {
  if (mode != ECNF_MODE_SAMPLE && mode != ECNF_MODE_SAMPLE_LOGQ && mode != ECNF_MODE_LOGPROB) {
    ecnf_set_error("ecnf_solve: bad mode %d", mode);
    return ECNF_ERR_INVALID;
  }
  if (mode != ECNF_MODE_SAMPLE && !out_logs) {
    ecnf_set_error("ecnf_solve: out_logs is required for log-density modes");
    return ECNF_ERR_INVALID;
  }
  if (ctrl && !ctrl->fixed && !(ctrl->rtol > 0.f || ctrl->atol > 0.f)) {
    ecnf_set_error("ecnf_solve: adaptive stepping needs rtol or atol > 0");
    return ECNF_ERR_INVALID;
  }
  return ECNF_OK;
}

}  // namespace

extern "C" {

int64_t ecnf_solve_workspace_bytes(const ecnf_model* m, int mode, int64_t B) {
  if (!m) return 0;
  const bool div = mode_div(mode);
  const int64_t stride = scratch_stride_of(m, div);
  return 256 + (int64_t)grid_for(m, B < 1 ? 1 : B) * stride * (int64_t)sizeof(float) + (tc_eligible(m, div) ? tc_image_bytes(m) : 0);
}

int64_t ecnf_solve_tensor_flops_per_eval(const ecnf_model* m) {
  if (!m || !use_tc(m, true)) return 0;
  return tc_flops_per_eval(m);
}

int ecnf_solve_engine_for(const ecnf_model* m, int mode) {
  if (!m || mode < ECNF_MODE_VF || mode > ECNF_MODE_LOGPROB) {
    ecnf_set_error("ecnf_solve_engine_for: null model or bad mode %d", mode);
    return ECNF_ERR_INVALID;
  }
  const bool div = mode_div(mode);
  if (use_tc(m, div)) return 0;
  const int rc = div ? simt_check_uh<true>(m) : simt_check_uh<false>(m);
  return rc == ECNF_OK ? 1 : rc;
}

int ecnf_solve_tc_tile_table(const ecnf_model* m, int kind, uint32_t* out_host, int64_t cap_words) {
  if (!m || !tc_eligible(m, true)) return 0;
  return tc_tile_table(m, kind, out_host, cap_words);
}

int ecnf_model_set_engine(ecnf_model* m, int engine) {
  if (!m || (engine != 0 && engine != 1)) { ecnf_set_error("ecnf_model_set_engine: 0 = auto, 1 = fp32 SIMT"); return ECNF_ERR_INVALID; }
  m->engine = engine;
  return ECNF_OK;
}

int ecnf_vf_forward(const ecnf_model* m, const float* x, const float* t, const int32_t* feat, int64_t B, float* out_f,
                    void* ws, int64_t ws_bytes, void* stream) {
  if (B == 0) return ECNF_OK;
  if (!t) { ecnf_set_error("ecnf_vf_forward: t is null"); return ECNF_ERR_INVALID; }
  return run(m, ECNF_MODE_VF, x, t, feat, nullptr, B, nullptr, out_f, nullptr, nullptr, ws, ws_bytes, stream);
}

int ecnf_vf_forward_div(const ecnf_model* m, const float* x, const float* t, const int32_t* feat, int64_t B,
                        float* out_f, float* out_div, void* ws, int64_t ws_bytes, void* stream) {
  if (B == 0) return ECNF_OK;
  if (!t || !out_div) { ecnf_set_error("ecnf_vf_forward_div: null argument"); return ECNF_ERR_INVALID; }
  return run(m, ECNF_MODE_VF_DIV, x, t, feat, nullptr, B, nullptr, out_f, out_div, nullptr, ws, ws_bytes, stream);
}

int ecnf_vf_forward_hutchinson(const ecnf_model* m, const float* x, const float* t, const int32_t* feat, const float* eps,
                               int64_t B, float* out_f, float* out_div, void* ws, int64_t ws_bytes, void* stream) {
  if (B == 0) return ECNF_OK;
  if (!t || !out_div || !eps) { ecnf_set_error("ecnf_vf_forward_hutchinson: null argument"); return ECNF_ERR_INVALID; }
  return run(m, ECNF_MODE_VF_DIV, x, t, feat, eps, B, nullptr, out_f, out_div, nullptr, ws, ws_bytes, stream);
}

int ecnf_solve(const ecnf_model* m, int mode, const float* x_init, const int32_t* feat, int64_t B,
               const ecnf_solve_ctrl* ctrl, float* out_x, float* out_logs, int32_t* out_stats, void* ws,
               int64_t ws_bytes, void* stream) {
  return ecnf_solve_hutchinson(m, mode, x_init, feat, nullptr, B, ctrl, out_x, out_logs, out_stats, ws, ws_bytes, stream);
}

int ecnf_solve_hutchinson(const ecnf_model* m, int mode, const float* x_init, const int32_t* feat, const float* eps,
                          int64_t B, const ecnf_solve_ctrl* ctrl, float* out_x, float* out_logs, int32_t* out_stats,
                          void* ws, int64_t ws_bytes, void* stream) {
  if (mode != ECNF_MODE_SAMPLE && mode != ECNF_MODE_SAMPLE_LOGQ && mode != ECNF_MODE_LOGPROB) {
    ecnf_set_error("ecnf_solve: bad mode %d", mode);
    return ECNF_ERR_INVALID;
  }
  if (B == 0) return ECNF_OK;
  const int rc = check_solve_args(mode, out_logs, ctrl);
  if (rc != ECNF_OK) return rc;
  return run(m, mode, x_init, nullptr, feat, eps, B, ctrl, out_x, out_logs, out_stats, ws, ws_bytes, stream);
}

int64_t ecnf_solve_saveat_workspace_bytes(const ecnf_model* m, int mode, int64_t B, int n_save) {
  const int64_t base = ecnf_solve_workspace_bytes(m, mode, B);
  if (!m || n_save <= 0) return base;
  return round256(base) + round256((int64_t)n_save * (int64_t)sizeof(float));
}

int ecnf_solve_saveat(const ecnf_model* m, int mode, const float* x_init, const int32_t* feat, const float* eps,
                      int64_t B, const ecnf_solve_ctrl* ctrl, int n_save, const float* ts_host, float* out_x,
                      float* out_logs, int32_t* out_stats, float* out_traj, float* out_traj_delta, void* ws,
                      int64_t ws_bytes, void* stream) {
  if (n_save < 0 || n_save > ECNF_MAX_SAVE_TIMES) {
    ecnf_set_error("ecnf_solve_saveat: n_save = %d outside [0, %d]", n_save, ECNF_MAX_SAVE_TIMES);
    return ECNF_ERR_INVALID;
  }
  if (n_save == 0)
    return ecnf_solve_hutchinson(m, mode, x_init, feat, eps, B, ctrl, out_x, out_logs, out_stats, ws, ws_bytes, stream);
  const int rc = check_solve_args(mode, out_logs, ctrl);
  if (rc != ECNF_OK) return rc;
  if (!ts_host || !out_traj) {
    ecnf_set_error("ecnf_solve_saveat: ts_host and out_traj are required when n_save > 0");
    return ECNF_ERR_INVALID;
  }
  if (mode != ECNF_MODE_SAMPLE && !out_traj_delta) {
    ecnf_set_error("ecnf_solve_saveat: out_traj_delta is required for log-density modes");
    return ECNF_ERR_INVALID;
  }
  // internal time runs forward: tau = t (SAMPLE, SAMPLE_LOGQ: 0 -> 1), tau = -t (LOGPROB: 1 -> 0)
  const float dir = mode == ECNF_MODE_LOGPROB ? -1.f : 1.f;
  std::vector<float> tau((size_t)n_save);
  for (int k = 0; k < n_save; ++k) {
    const float tk = ts_host[k];
    if (!(tk >= 0.f && tk <= 1.f)) {
      ecnf_set_error("ecnf_solve_saveat: ts[%d] = %g is outside [0, 1]", k, (double)tk);
      return ECNF_ERR_INVALID;
    }
    tau[k] = dir * tk;
    if (k > 0 && !(tau[k] > tau[k - 1])) {
      ecnf_set_error("ecnf_solve_saveat: ts must be strictly %s in mode %d (ts[%d] = %g after %g)",
                     dir > 0.f ? "increasing" : "decreasing", mode, k, (double)tk, (double)ts_host[k - 1]);
      return ECNF_ERR_INVALID;
    }
  }
  if (B == 0) return ECNF_OK;
  if (!m) {
    ecnf_set_error("ecnf_solve: null argument");
    return ECNF_ERR_INVALID;
  }
  const int64_t need = ecnf_solve_saveat_workspace_bytes(m, mode, B, n_save);
  if (!ws || ws_bytes < need) {
    ecnf_set_error("workspace too small: need %lld bytes, got %lld", (long long)need, (long long)ws_bytes);
    return ECNF_ERR_WORKSPACE;
  }
  // the save-time table sits at the tail of the workspace; the copy from pageable memory is staged before it returns
  float* d_tau = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + round256(ecnf_solve_workspace_bytes(m, mode, B)));
  ECNF_CHECK_CUDA(cudaMemcpyAsync(d_tau, tau.data(), (size_t)n_save * sizeof(float), cudaMemcpyHostToDevice,
                                  (cudaStream_t)stream));
  SaveArgs sv;
  sv.ts = d_tau;
  sv.n_save = n_save;
  sv.out_traj = out_traj;
  sv.out_traj_delta = mode == ECNF_MODE_SAMPLE ? nullptr : out_traj_delta;
  return run(m, mode, x_init, nullptr, feat, eps, B, ctrl, out_x, out_logs, out_stats, ws, ws_bytes, stream, sv);
}

}  // extern "C"
