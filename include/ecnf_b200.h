/* ecnf_b200 -- C-ABI of the B200-native (sm_100a) implementation of the ecnf hot path.
 *
 * The reference (Kalyan0821/ecnf-baseline-neurips-2023) has no FFI: its boundary is the Python function API in
 * ecnf/cnf/{core,build_cnf,sample_and_log_prob,loss,gradient_step}.py and ecnf/nets/egnn.py.  Each entry
 * point below names the reference function (file:line under the reference root) it replaces.  The signatures
 * are XLA-FFI shaped on purpose: device buffers in, device buffers out, scalar attributes, a stream, no hidden
 * state except the opaque model handle (config + parameter pointer + engine choice, read at launch time; one handle
 * per concurrent caller) -- so a jax.ffi handler is a thin shim (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer named d_* / x / t / feat / out_* / ws is a DEVICE pointer owned by the caller;
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on it;
 *   - the library never allocates device memory: scratch comes from the caller's workspace (query the size
 *     with the matching *_workspace_bytes function);
 *   - return value: 0 = OK, negative = error (ecnf_last_error() gives the text, thread-local);
 *   - all floating point is fp32 (the reference runs jax with x64 off); node features are int32;
 *   - positions are flat [B, n_frames*dim], node-major / coordinate-minor (build_cnf.py:77).
 */
#ifndef ECNF_B200_H
#define ECNF_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ECNF_OK 0
#define ECNF_ERR_INVALID (-1)
#define ECNF_ERR_CUDA (-2)
#define ECNF_ERR_UNSUPPORTED (-3)
#define ECNF_ERR_WORKSPACE (-4)

typedef struct ecnf_model ecnf_model;

/* Arguments of build_cnf (ecnf/cnf/build_cnf.py:34-44) + EGNN defaults (ecnf/nets/egnn.py:117-128). */
typedef struct ecnf_config {
  int32_t n_frames;      /* nodes per graph, 2..32 */
  int32_t dim;           /* 2 or 3 */
  int32_t n_blocks;      /* n_blocks_egnn, 1..8 */
  int32_t n_layers;      /* len(mlp_units), 1..6 */
  int32_t mlp_units;     /* width U of every entry of mlp_units: 64, 128 or 256 (all shipped configs are uniform) */
  int32_t n_hidden;      /* n_invariant_feat_hidden H: 32 or 64 */
  int32_t time_dim;      /* time_embedding_dim T: even, 4..16 */
  int32_t n_features;    /* rows of the nn.Embed table */
  float sigma_min;       /* core.py:35 */
  float base_scale;      /* build_cnf.py:48 */
  float normalization_constant; /* egnn.py:127 (1.0) */
  float freqs[8];        /* fp32 table exp(-k*log(1e4)/(T/2-1)), k<T/2 (build_cnf.py:25-27), computed by the host */
} ecnf_config;

const char* ecnf_last_error(void);
int ecnf_version(void);

/* ---- model handle: hyper-parameters + a flat fp32 parameter buffer in the library's aligned layout.
 * Replaces the flax variable dict produced by FlatEgnn.init (build_cnf.py:65-97; SURVEY Appendix D).       */
int ecnf_model_create(const ecnf_config* cfg, const float* d_params, ecnf_model** out);
void ecnf_model_destroy(ecnf_model* m);
int ecnf_model_set_params(ecnf_model* m, const float* d_params);
/* A second handle with the same hyper-parameters and per-handle attributes (engine choice, training chunk size) bound to
 * another parameter buffer (NULL: the same one).  Host-side and cheap (no device work, no allocation on the device): the
 * way to pass the parameters PER CALL -- an XLA FFI handler clones the template handle with the call's parameter buffer,
 * launches, and destroys the clone (kernel arguments are copied at launch), so concurrent calls never share mutable state. */
int ecnf_model_clone(const ecnf_model* m, const float* d_params, ecnf_model** out);
int64_t ecnf_model_param_count(const ecnf_model* m);   /* floats, incl. alignment padding */
int ecnf_model_num_tensors(const ecnf_model* m);
/* idx-th tensor: flax path ("EGNN_0/0/phi_e/Dense_0/kernel"), float offset, shape (cols==0 => vector/scalar). */
int ecnf_model_param_layout(const ecnf_model* m, int idx, char* name, int name_cap, int64_t* offset,
                            int64_t* rows, int64_t* cols);

/* ---- vector field: cnf.apply(params, x, t, features)  (build_cnf.py:68-93 -> egnn.py:131-190, :49-114)  */
#define ECNF_MODE_VF 0          /* one evaluation, no divergence            */
#define ECNF_MODE_VF_DIV 1      /* one evaluation + exact Jacobian trace    */
#define ECNF_MODE_SAMPLE 2      /* sample_cnf                (sample_and_log_prob.py:11-38)   */
#define ECNF_MODE_SAMPLE_LOGQ 3 /* sample_and_log_prob_cnf   (sample_and_log_prob.py:97-149)  */
#define ECNF_MODE_LOGPROB 4     /* get_log_prob              (sample_and_log_prob.py:41-94)   */

int64_t ecnf_solve_workspace_bytes(const ecnf_model* m, int mode, int64_t B);
/* Engine selection of ONE model handle (solve / vector-field / training entry points): 0 = automatic (tcgen05
 * tensor-core engine where the shape is eligible, fp32 SIMT otherwise), 1 = always fp32 SIMT (the accuracy
 * reference).  A handle is the triple (config, parameter pointer, engine); every call reads it at launch time, so
 * concurrent callers (threads / streams) use one handle each -- there is no process-wide state.             */
int ecnf_model_set_engine(ecnf_model* m, int engine);
/* tcgen05 flops the tensor-core engine issues per vector-field evaluation with exact divergence (3 bf16 passes over
 * every 128-lane x N-column tile-layer), 0 when the shape runs on the fp32 SIMT engine.  For roofline reports.   */
int64_t ecnf_solve_tensor_flops_per_eval(const ecnf_model* m);
/* Which engine a solve / vector-field call of `mode` (ECNF_MODE_*; VF_DIV covers the Hutchinson entry points too) runs on
 * with this handle's current engine choice: 0 = tcgen05 tensor cores, 1 = fp32 SIMT; negative = that call would fail
 * (ECNF_ERR_UNSUPPORTED: the shape exceeds the SIMT engine's limits, ecnf_last_error() says which; ECNF_ERR_INVALID: null
 * handle or bad mode).  No device work.                                                                             */
int ecnf_solve_engine_for(const ecnf_model* m, int mode);
/* Host copy of the tensor-core engine's tile table of one kind (0 node/primal-only, 1 node, 2 first-block edges,
 * 3 middle-block edges, 4 last-block edges, 5 edges/primal-only; kind + 8: the one-tangent (Hutchinson) variant, used for
 * kinds 1 and 3): 48 uint32 per tile = 32 chunk words (2 sub-tiles x 16 chunks of 8 columns: bit31 valid, [0,10) group,
 * [10,18) slot of the chunk's column 1 (0: dense chunk of 8 primal rows), [18,22) valid columns, bit22 last chunk of its
 * thread group in a run, bit23 owner of the group's primal row, bit24 run end) + 16 header words (MMA N, flush, message
 * window, chunks per (sub-tile, half), first/last receiver, chunk count, accumulator rows, run-end mask).
 * Returns the number of tiles (writes at most cap_words), 0 when the shape is not eligible.  Test / debug aid.      */
int ecnf_solve_tc_tile_table(const ecnf_model* m, int kind, uint32_t* out_host, int64_t cap_words);

int ecnf_vf_forward(const ecnf_model* m, const float* x, const float* t, const int32_t* feat, int64_t B,
                    float* out_f, void* ws, int64_t ws_bytes, void* stream);
/* + exact divergence tr(df/dx) over the flattened, un-centred input (sample_and_log_prob.py:58-67), computed
 * with forward-mode tangents fused into the layer kernel instead of the reference's D reverse passes.      */
int ecnf_vf_forward_div(const ecnf_model* m, const float* x, const float* t, const int32_t* feat, int64_t B,
                        float* out_f, float* out_div, void* ws, int64_t ws_bytes, void* stream);
/* Hutchinson estimate eps^T (df/dx) eps of the divergence with one caller-supplied probe eps [B, n_frames*dim] per
 * sample: the reference's `approx=True` branch (sample_and_log_prob.py:69-78, :123-133).  One forward-mode tangent
 * instead of n_frames*dim.                                                                                       */
int ecnf_vf_forward_hutchinson(const ecnf_model* m, const float* x, const float* t, const int32_t* feat, const float* eps,
                               int64_t B, float* out_f, float* out_div, void* ws, int64_t ws_bytes, void* stream);

/* ---- ODE solve: diffrax.diffeqsolve(ODETerm, Dopri5, PIDController | ConstantStepSize) as one persistent
 * on-device loop per trajectory (call sites sample_and_log_prob.py:33-37,85-89,140-144).                   */
typedef struct ecnf_solve_ctrl {
  int32_t fixed;      /* use_fixed_step_size */
  float step_size;    /* 0.05 */
  float rtol, atol;   /* 1e-5, 1e-5 */
  float dtmin;        /* 1e-5 */
  int32_t max_steps;  /* diffrax default 4096 */
  float safety, factormin, factormax, error_order; /* PIDController defaults 0.9, 0.2, 10, 5 */
  float err_scale;    /* multiplies the embedded error estimate sum_i (b - b_hat)_i k_i: 1 = diffrax / torchdiffeq's b_hat
                         (the default; <= 0 is read as 1), 1.5 = the classic Hairer-Wanner b_hat (SURVEY Appendix B: a
                         mismatch with the installed diffrax is a configuration change, not a rebuild)              */
} ecnf_solve_ctrl;

/* mode SAMPLE:       x_init = x0 ~ base;   out_x = x(1);          out_logs unused (may be NULL)
 * mode SAMPLE_LOGQ:  x_init = x0 ~ base;   out_x = x(1);          out_logs[b] = {log_q, log_p0(x0), delta}
 * mode LOGPROB:      x_init = data x;      out_x = x(0);          out_logs[b] = {log_p, log_p0(x(0)), delta}
 * out_stats[b] = {n_steps, n_accepted, n_evals, status(0 ok, 1 max_steps reached)}                         */
int ecnf_solve(const ecnf_model* m, int mode, const float* x_init, const int32_t* feat, int64_t B,
               const ecnf_solve_ctrl* ctrl, float* out_x, float* out_logs, int32_t* out_stats, void* ws,
               int64_t ws_bytes, void* stream);
/* ecnf_solve with the Hutchinson estimate in place of the exact trace (modes SAMPLE_LOGQ / LOGPROB); the probe of a
 * trajectory is fixed for the whole solve, as in the reference (eps == NULL: identical to ecnf_solve).           */
int ecnf_solve_hutchinson(const ecnf_model* m, int mode, const float* x_init, const int32_t* feat, const float* eps,
                          int64_t B, const ecnf_solve_ctrl* ctrl, float* out_x, float* out_logs, int32_t* out_stats,
                          void* ws, int64_t ws_bytes, void* stream);

/* ---- ODE solve that also reports the path: diffeqsolve(..., saveat=SaveAt(ts=ts)) at the same call sites
 * (sample_and_log_prob.py:33-37,85-89,140-144).  ts_host is a HOST array of n_save (<= ECNF_MAX_SAVE_TIMES) fp32 times in
 * [0, 1], strictly increasing for SAMPLE / SAMPLE_LOGQ and strictly decreasing for LOGPROB (the direction of integration);
 * it is copied before the call returns.  Row k of the path is the joint state at ts[k]:
 *   out_traj[b, k, :]    = x(ts[k])                                            [B, n_save, D] (vmap of a per-trajectory solve)
 *   out_traj_delta[b, k] = the divergence integral accumulated from the start time to ts[k]   [B, n_save], log modes only
 * so along a sample path log q_t(x_t) = log p0(x0) - out_traj_delta[b, k].  A time equal to the start time gives x_init and
 * 0; a time equal to the end time gives out_x and out_logs[b, 2] bit for bit; an interior time comes from the Dopri5
 * 4th-order dense output of the accepted step that contains it.  Saving does not change the step sequence: out_x,
 * out_logs and out_stats are those of ecnf_solve_hutchinson.  A trajectory stopped on max_steps (status 1) has NaN in the
 * rows it never reached.  n_save = 0: exactly ecnf_solve_hutchinson (ts_host / out_traj* unused).
 * The workspace is ecnf_solve_saveat_workspace_bytes: ecnf_solve_workspace_bytes + the save-time table, rounded up to
 * 256 B (the same value when n_save = 0).                                                                        */
#define ECNF_MAX_SAVE_TIMES 1024
int64_t ecnf_solve_saveat_workspace_bytes(const ecnf_model* m, int mode, int64_t B, int n_save);
int ecnf_solve_saveat(const ecnf_model* m, int mode, const float* x_init, const int32_t* feat, const float* eps,
                      int64_t B, const ecnf_solve_ctrl* ctrl, int n_save, const float* ts_host,
                      float* out_x, float* out_logs, int32_t* out_stats,
                      float* out_traj, float* out_traj_delta,
                      void* ws, int64_t ws_bytes, void* stream);

/* ---- base distribution (build_cnf.py:46-61, zero_com_base.py:44-47,64-93)                                */
/* x0 = base_scale * remove_mean(eps); eps from a counter-based Philox4x32-10 stream keyed by
 * (seed, global sample index) so a sharded run reproduces the single-GPU draw.                             */
int ecnf_base_sample(const ecnf_model* m, uint64_t seed, int64_t global_offset, int64_t B, float* out_x0,
                     void* stream);
/* N(0,1) draws [B, n_frames*dim] from the same counter-based stream as ecnf_base_sample: value = f(seed, global sample
 * index goff + b, element, substream).  substream 0 reproduces the raw noise underneath ecnf_base_sample (the reference
 * reuses the base-sample key for the Hutchinson probe, sample_and_log_prob.py:130,137); use another for independent
 * draws (jax.random.normal(key, x.shape) in get_log_prob, sample_and_log_prob.py:55).                              */
int ecnf_normal_noise(const ecnf_model* m, uint64_t seed, int64_t goff, int64_t B, uint32_t substream, float* out, void* stream);
int ecnf_base_sample_from_noise(const ecnf_model* m, const float* eps, int64_t B, float* out_x0, void* stream);
int ecnf_base_log_prob(const ecnf_model* m, const float* x, int64_t B, float* out, void* stream);

/* ---- flow-matching loss and gradient (loss.py:10-32 + jax.grad in gradient_step.py:31-37).
 * x_t = (1-(1-sigma)t) x0 + t x_data, u = x_data - (1-sigma) x0 (core.py:35-39); loss = mean((v-u)^2).
 * out_loss: 1 float; out_grad: param_count floats in the parameter layout (sum over the B rows given,
 * already divided by `loss_denominator` = global_B * D so that shards add up under an all-reduce).         */
int64_t ecnf_fm_workspace_bytes(const ecnf_model* m, int64_t B);
/* A minibatch is processed in chunks of `graphs` graphs whose gradients accumulate (0, the default = the whole minibatch
 * in one pass).  A per-handle attribute like the engine choice; changes the workspace size.  The result is the same sum
 * over rows in a different order (loss.py:25-31 is a mean over the batch).                                           */
int ecnf_model_set_fm_chunk(ecnf_model* m, int64_t graphs);
int ecnf_fm_loss_grad(const ecnf_model* m, const float* x_data, const float* x0, const float* t,
                      const int32_t* feat, int64_t B, float loss_denominator, float* out_loss, float* out_grad,
                      void* ws, int64_t ws_bytes, void* stream);
/* t ~ U[0,1) and x0 ~ base from the same Philox stream (substream 1 / 0), keyed by global row index.       */
int ecnf_fm_draw_noise(const ecnf_model* m, uint64_t seed, int64_t global_offset, int64_t B, float* out_x0,
                       float* out_t, void* stream);

/* ---- optimiser: optax.adam(lr) with warmup_cosine_decay_schedule (setup_training.py:96-109), update/grad
 * global norms and optional EMA (gradient_step.py:39-50).  `lr` is the schedule value for this step;
 * `step` is the 0-based count before the update.  out_norms = {grad_norm, update_norm}.                    */
int ecnf_adam_step(float* params, const float* grad, float* mu, float* nu, float* ema_or_null, int64_t count,
                   int64_t step, float lr, float b1, float b2, float eps, float ema_beta, float* out_norms,
                   void* stream);
float ecnf_warmup_cosine_lr(int64_t step, float init_value, float peak_value, int64_t warmup_steps,
                            int64_t decay_steps, float end_value);

/* ---- importance-weight statistics (setup_training.py:175-182, utils/evaluation.py:10-22).
 * out5 = {max(log_w), sum exp(w-max), sum exp(2(w-max)), max(-log_w), sum exp(-w-max(-w))}: sufficient
 * statistics that merge across ranks; the host turns them into reverse / forward ESS.                      */
int ecnf_ess_stats(const float* log_w, int64_t N, float* out5, void* stream);

/* ---- target energies (targets/target_energy/leonard_jones.py:10-27, double_well.py:9-19): log p = -E    */
#define ECNF_TARGET_LJ 0
#define ECNF_TARGET_DW 1
int ecnf_target_log_prob(int kind, const float* x, int64_t B, int n_frames, int dim, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ECNF_B200_H */
