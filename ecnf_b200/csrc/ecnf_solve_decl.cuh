// Declarations shared by the engine-A dispatch (ecnf_solve.cu) and its per-(U,H) instantiation units.
#pragma once
#include "ecnf_common.cuh"

namespace ecnf_solve_detail {

// per-CTA global scratch (floats): h (current), h_in, P_s, P_r, aggregated messages, P_h (tensor-core engine only)
__host__ __device__ inline int64_t scratch_floats(int n, int dim, int H, int U, bool div) {
  const int64_t ND = div ? 1 + n * dim : 1;
  return n * ND * (2 * (int64_t)H + 4 * (int64_t)U) + 2 * (int64_t)U;   // + one all-zero row after P_s and after P_r (tensor-core engine)
}

// byte offsets of the bf16 (hi, lo) weight images used by the tensor-core engine (ecnf_solve_tc.cuh)
struct TcImgBlock {
  int Wd, We0, We[ECNF_MAX_LAYERS], Wx[ECNF_MAX_LAYERS], Wh0m, Wh0h, Wh[ECNF_MAX_LAYERS], WhL;
};
struct TcImages {
  const unsigned char* base;
  TcImgBlock blk[ECNF_MAX_BLOCKS];
};

// shared-memory carve-up of the tensor-core engine (byte offsets), computed on the host
struct TcSmemLayout {
  int bop, macc, xt, xtacc, dacc, xs, xs0, xacc, mu, tau, cvec, ode, red, colsd, colmrow, chw, hdr, pdot, pdh, wA, wB, cdbuf,
      egv, bars, prof, total_bytes;
  int mrows;   // rows of the message accumulator (one window of receivers x slots)
};

// tile tables of the tensor-core engine: which (group, slot) rows sit in which 8-column chunk (ecnf_solve_tc.cuh)
// *1: primal rows only (no divergence); *_S: TT_NODE / TT_MID with the s shape-space tangents of the middle blocks
enum { TT_NODE1 = 0, TT_NODE, TT_FIRST, TT_MID, TT_LAST, TT_EDGE1, TT_NODE_S, TT_MID_S, TT_COUNT };
constexpr int TC_TILE_WORDS = 48;    // 32 chunk words (2 sub-tiles x 16 chunks) + 16 header words
struct TcTabs {
  const uint32_t* base;
  int off[TT_COUNT];   // first tile of each kind
  int cnt[TT_COUNT];   // tiles per kind
};

struct KernelArgs {
  EcnfModelDev m;
  int mode;
  long long B;
  const float* x_init;   // [B, D]
  const float* t_in;     // [B] (VF modes)
  const int32_t* feat;   // [B, n]
  const float* eps;      // [B, D] Hutchinson probes, or null for the exact trace
  ecnf_solve_ctrl ctrl;
  float* out_x;          // [B, D]   (VF modes: f)
  float* out_logs;       // [B, 3]   (VF_DIV: out_div [B])
  int32_t* out_stats;    // [B, 4]
  float* scratch;        // per-CTA global scratch
  long long scratch_stride;
  unsigned int* counter;
  TcImages img;
  TcSmemLayout lay;
  TcTabs tabs;
  // SaveAt(ts) (kernels instantiated with SAVE only)
  const float* ts;        // [n_save] internal (direction-multiplied) save times, increasing, in the workspace
  int n_save;
  float* out_traj;        // [B, n_save, D]
  float* out_traj_delta;  // [B, n_save] (log-density modes)
};
static_assert(sizeof(KernelArgs) <= 4096, "KernelArgs is a by-value kernel parameter (4 KB limit)");

// fp32 SIMT engine: its shape limits (ECNF_OK, or ECNF_ERR_UNSUPPORTED with the reason set), launch
template <int U, int H, bool DIV>
int simt_check(const ecnf_model* mdl);
template <int U, int H, bool DIV, bool SAVE = false>
int launch_t(const ecnf_model* mdl, KernelArgs& a, int grid, cudaStream_t st);

// tensor-core engine ((U, H) = (128, 64) and (64, 32)): eligibility, extra workspace, launch
bool tc_eligible(const ecnf_model* mdl, bool div);
int64_t tc_image_bytes(const ecnf_model* mdl);
int64_t tc_flops_per_eval(const ecnf_model* mdl);
int tc_tile_table(const ecnf_model* mdl, int kind, uint32_t* out, int64_t cap_words);
int launch_tc(const ecnf_model* mdl, KernelArgs& a, int grid, void* image_ws, bool div, bool save, cudaStream_t st);

}  // namespace ecnf_solve_detail
