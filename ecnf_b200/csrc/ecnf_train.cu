// Engine B: flow-matching loss, forward and hand-written backward, layer by layer over the whole minibatch.
//
// Replaces  flow_matching_loss_fn (ecnf/cnf/loss.py:10-32) under jax.grad (ecnf/cnf/gradient_step.py:31-37):
//   x_t, u_t = OT path (core.py:35-39);  v = cnf.apply(params, x_t, t, features);  loss = mean((v - u_t)^2)
// and produces d loss / d params in the library's flat parameter layout.
//
// Layout in HBM: every Dense layer is one row-major [rows x width] fp32 matrix over the whole batch, rows =
// B*n node rows or B*n*(n-1) edge rows (receiver-major inside a graph, utils/graph.py:6-14).  The forward keeps
// the pre-activations z of every layer; the backward overwrites them in place with dz.  The square GEMMs and weight
// gradients over the edge rows run on the tensor cores (ecnf_train_tc.cuh); every other GEMM, and all of them when the
// handle selects the SIMT engine, uses the register-tiled fp32 building block of engine A (ecnf_tile.cuh).
#include <algorithm>

#include "ecnf_tile.cuh"
#include "ecnf_train_tc.cuh"

namespace {
using ecnf_tile::ColT;
using ecnf_tile::NTHREADS;
using ecnf_tile::tile_gemm;
using ecnf_tile::WCHUNK;
using ecnf_train_tc::GemmArgs;

// What every launch of one ecnf_fm_loss_grad call needs from the model handle and the caller
struct LaunchCtx {
  int num_sms;
  bool use_tc;   // the handle's engine choice: tensor cores where eligible (engine 0), or fp32 SIMT everywhere
  cudaStream_t st;
};

// Shapes with a tensor-core kernel (ecnf_train_tc.cuh)
constexpr bool tc_shape(int K, int N) { return K == N && (K == 128 || K == 256); }
// The big square GEMMs over the edge rows go to the tensor cores.  `plain`: dense leading dimensions, no second operand
// and no per-graph row vector, which only the SIMT kernels support.
bool use_tc(const LaunchCtx& lc, int K, int N, int M, bool plain) {
  return lc.use_tc && plain && tc_shape(K, N) && M >= 8192;
}

__device__ __forceinline__ float silu_f(float z) { return z * ecnf_sigmoid(z); }
__device__ __forceinline__ float dsilu_f(float z) {
  const float s = ecnf_sigmoid(z);
  return s * (1.f + z * (1.f - s));
}

// ------------------------------------------------------------------------------------------------
// C[M,N] = epilogue( op(A)[M,K] W[K,N] (+ A2[M,K2] W2[K2,N]) )   (GemmArgs)
// ------------------------------------------------------------------------------------------------
template <int K, int N>
struct GemmGeo {
  static constexpr int TR = (K == 256 || N == 256) ? 64 : 128;
  static constexpr int LD = K + 4;
};

template <int K, int N, int K2>
__global__ void __launch_bounds__(NTHREADS, 1) gemm_rows_kernel(const __grid_constant__ GemmArgs g) {
  constexpr int TR = GemmGeo<K, N>::TR, LD = K + 4, LD2 = (K2 > 0 ? K2 : 4) + 4, RT = TR / 16, CT = ColT<N>::CT,
                NSEG = CT / 4;
  extern __shared__ __align__(16) float smem[];
  float* X = smem;
  float* X2 = X + TR * LD;
  float* Wb = X2 + (K2 > 0 ? TR * LD2 : 0);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, warp = tid >> 5;
  const int ntiles = (g.M + TR - 1) / TR;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int r0 = tile * TR, nrows = min(TR, g.M - r0);
    __syncthreads();
    for (int idx = tid; idx < nrows * (K / 4); idx += NTHREADS) {
      const int row = idx / (K / 4), c4 = idx % (K / 4);
      float4 v = *reinterpret_cast<const float4*>(g.A + (size_t)(r0 + row) * K + c4 * 4);
      if (g.a_op) { v.x = silu_f(v.x); v.y = silu_f(v.y); v.z = silu_f(v.z); v.w = silu_f(v.w); }
      *reinterpret_cast<float4*>(X + row * LD + c4 * 4) = v;
    }
    if (K2 > 0 && g.A2) {
      for (int idx = tid; idx < nrows * (K2 / 4); idx += NTHREADS) {
        const int row = idx / (K2 / 4), c4 = idx % (K2 / 4);
        *reinterpret_cast<float4*>(X2 + row * LD2 + c4 * 4) =
            *reinterpret_cast<const float4*>(g.A2 + (size_t)(r0 + row) * K2 + c4 * 4);
      }
    }
    __syncthreads();
    float acc[RT][CT];
    tile_gemm<K, N, TR, LD, true>(X, g.W, Wb, acc, nrows);
    if (K2 > 0 && g.A2) tile_gemm<(K2 > 0 ? K2 : 32), N, TR, LD2, false>(X2, g.W2, Wb, acc, nrows);
    const bool active = (2 * RT * warp < nrows) && (tx * 4 < N);
    if (active) {
      const int row0 = 2 * RT * warp + (ty & 1);
#pragma unroll
      for (int rr = 0; rr < RT; ++rr) {
        const int row = row0 + 2 * rr;
        if (row >= nrows) continue;
        const size_t grow = (size_t)(r0 + row);
#pragma unroll
        for (int sg = 0; sg < NSEG; ++sg) {
          const int col = sg * 64 + tx * 4;
          float v[4] = {acc[rr][4 * sg], acc[rr][4 * sg + 1], acc[rr][4 * sg + 2], acc[rr][4 * sg + 3]};
          if (g.bias) {
            const float4 b = *reinterpret_cast<const float4*>(g.bias + col);
            v[0] += b.x; v[1] += b.y; v[2] += b.z; v[3] += b.w;
          }
          if (g.rowvec) {
            const float4 b = *reinterpret_cast<const float4*>(g.rowvec + (grow / g.rows_per_vec) * N + col);
            v[0] += b.x; v[1] += b.y; v[2] += b.z; v[3] += b.w;
          }
          if (g.resid) {
            const float4 b = *reinterpret_cast<const float4*>(g.resid + grow * N + col);
            v[0] += b.x; v[1] += b.y; v[2] += b.z; v[3] += b.w;
          }
          if (g.add) {
            const float4 b = *reinterpret_cast<const float4*>(g.add + grow * N + col);
            v[0] += b.x; v[1] += b.y; v[2] += b.z; v[3] += b.w;
          }
          if (g.mulz) {
            const float4 z = *reinterpret_cast<const float4*>(g.mulz + grow * N + col);
            v[0] *= dsilu_f(z.x); v[1] *= dsilu_f(z.y); v[2] *= dsilu_f(z.z); v[3] *= dsilu_f(z.w);
          }
          *reinterpret_cast<float4*>(g.C + grow * N + col) = make_float4(v[0], v[1], v[2], v[3]);
        }
      }
    }
  }
}

template <int K, int N, int K2>
int launch_gemm(const LaunchCtx& lc, const GemmArgs& g) {
  if constexpr (tc_shape(K, N)) {
    if (use_tc(lc, K, N, g.M, !g.A2 && !g.rowvec)) {
      ECNF_CHECK_CUDA((ecnf_train_tc::launch<K, N>(g, lc.num_sms, lc.st)));
      return ECNF_OK;
    }
  }
  constexpr int TR = GemmGeo<K, N>::TR;
  const size_t smem = (size_t)(TR * (K + 4) + (K2 > 0 ? TR * (K2 + 4) : 0) + 2 * WCHUNK) * sizeof(float);
  auto kern = gemm_rows_kernel<K, N, K2>;
  static bool configured = false;  // per instantiation
  if (!configured) {
    ECNF_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  const int ntiles = (g.M + TR - 1) / TR;
  const int grid = std::min(ntiles, lc.num_sms * 8);
  kern<<<grid, NTHREADS, smem, lc.st>>>(g);
  ECNF_CHECK_CUDA(cudaGetLastError());
  return ECNF_OK;
}

// ------------------------------------------------------------------------------------------------
// dW[K,N] += op(A)[M,K]^T dZ[M,N]      (split over row slabs, atomics into the gradient buffer)
// block (BK x BN) per CTA, thread tile (BK/16) x (BN/16)
// ------------------------------------------------------------------------------------------------
template <int BK, int BN>
__global__ void __launch_bounds__(NTHREADS) dw_kernel(const float* __restrict__ A, int lda, int a_op,
                                                      const float* __restrict__ dZ, int ldz, float* __restrict__ dW,
                                                      int ldw, int M, int rows_per_cta) {
  constexpr int RC = 32, TK = BK / 16, TN = BN / 16, LA = BK + 4, LZ = BN + 4;
  constexpr int A4 = RC * BK / 4 / NTHREADS > 0 ? RC * BK / 4 / NTHREADS : 1;  // float4 per thread per chunk
  constexpr int Z4 = RC * BN / 4 / NTHREADS > 0 ? RC * BN / 4 / NTHREADS : 1;
  __shared__ __align__(16) float As[RC * LA];
  __shared__ __align__(16) float Zs[RC * LZ];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int k0 = blockIdx.y * BK, n0 = blockIdx.z * BN;
  const int m_begin = blockIdx.x * rows_per_cta, m_end = min(M, m_begin + rows_per_cta);
  float acc[TK][TN];
#pragma unroll
  for (int i = 0; i < TK; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;
  float4 pa[A4], pz[Z4];
  auto fetch = [&](int m0) {
#pragma unroll
    for (int q = 0; q < A4; ++q) {
      const int idx = tid + q * NTHREADS;
      const int row = idx / (BK / 4), c4 = idx % (BK / 4);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (idx < RC * BK / 4 && m0 + row < m_end) {
        v = *reinterpret_cast<const float4*>(A + (size_t)(m0 + row) * lda + k0 + c4 * 4);
        if (a_op) { v.x = silu_f(v.x); v.y = silu_f(v.y); v.z = silu_f(v.z); v.w = silu_f(v.w); }
      }
      pa[q] = v;
    }
#pragma unroll
    for (int q = 0; q < Z4; ++q) {
      const int idx = tid + q * NTHREADS;
      const int row = idx / (BN / 4), c4 = idx % (BN / 4);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (idx < RC * BN / 4 && m0 + row < m_end) v = *reinterpret_cast<const float4*>(dZ + (size_t)(m0 + row) * ldz + n0 + c4 * 4);
      pz[q] = v;
    }
  };
  auto stash = [&]() {
#pragma unroll
    for (int q = 0; q < A4; ++q) {
      const int idx = tid + q * NTHREADS;
      if (idx < RC * BK / 4) *reinterpret_cast<float4*>(As + (idx / (BK / 4)) * LA + (idx % (BK / 4)) * 4) = pa[q];
    }
#pragma unroll
    for (int q = 0; q < Z4; ++q) {
      const int idx = tid + q * NTHREADS;
      if (idx < RC * BN / 4) *reinterpret_cast<float4*>(Zs + (idx / (BN / 4)) * LZ + (idx % (BN / 4)) * 4) = pz[q];
    }
  };
  if (m_begin < m_end) fetch(m_begin);
  for (int m0 = m_begin; m0 < m_end; m0 += RC) {
    __syncthreads();
    stash();
    __syncthreads();
    if (m0 + RC < m_end) fetch(m0 + RC);
#pragma unroll 4
    for (int r = 0; r < RC; ++r) {
      float a[TK], z[TN];
#pragma unroll
      for (int i = 0; i < TK; ++i) a[i] = As[r * LA + ty * TK + i];
#pragma unroll
      for (int j = 0; j < TN; ++j) z[j] = Zs[r * LZ + (TN >= 4 ? (j >> 2) * 64 + tx * 4 + (j & 3) : tx * TN + j)];
#pragma unroll
      for (int i = 0; i < TK; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], z[j], acc[i][j]);
    }
  }
#pragma unroll
  for (int i = 0; i < TK; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int col = TN >= 4 ? (j >> 2) * 64 + tx * 4 + (j & 3) : tx * TN + j;
      atomicAdd(dW + (size_t)(k0 + ty * TK + i) * ldw + n0 + col, acc[i][j]);
    }
}

__global__ void colsum_kernel(const float* __restrict__ Z, int M, int N, float* __restrict__ out, int rows_per_cta);
// out[N] += column sums of Z[M,N].  Rows per CTA: >= 4 CTAs per SM for the big (edge-row) matrices, enough CTAs to cover
// the latency for the node-row ones (9 728 rows in 38 CTAs took 27 us per launch)
void launch_colsum(const LaunchCtx& lc, const float* Z, int M, int N, float* out) {
  const int rows = M >= 65536 ? 256 : 32;
  colsum_kernel<<<(unsigned)((M + rows - 1) / rows), NTHREADS, 0, lc.st>>>(Z, M, N, out, rows);
}

// dW += op(A)^T dZ; bias_grad (optional) += column sums of dZ (fused into the tensor-core kernel, else a second launch)
int launch_dw(const LaunchCtx& lc, const float* A, int lda, int a_op, const float* dZ, int ldz, float* dW, int K, int N,
              int M, float* bias_grad = nullptr) {
  if (use_tc(lc, K, N, M, lda == K && ldz == N)) {
    if (K == 256) ECNF_CHECK_CUDA((ecnf_train_tc::launch_dw<256, 256>(A, a_op, dZ, dW, bias_grad, M, lc.num_sms, lc.st)));
    else ECNF_CHECK_CUDA((ecnf_train_tc::launch_dw<128, 128>(A, a_op, dZ, dW, bias_grad, M, lc.num_sms, lc.st)));
    return ECNF_OK;
  }
  if (bias_grad) launch_colsum(lc, dZ, M, N, bias_grad);
  // block shape: 128 where the dimension allows, else 64 / 32
  auto pick = [](int d) { return d % 128 == 0 ? 128 : (d % 64 == 0 ? 64 : 32); };
  const int BK = pick(K), BN = pick(N);
  const int nb = (K / BK) * (N / BN);
  int nslabs = std::max(1, (lc.num_sms * 2) / nb);
  int rows_per_cta = ((M + nslabs - 1) / nslabs + 31) / 32 * 32;
  nslabs = (M + rows_per_cta - 1) / rows_per_cta;
  dim3 grid(nslabs, K / BK, N / BN);
#define DW_CASE(bk, bn)                                                                             \
  if (BK == bk && BN == bn) {                                                                       \
    dw_kernel<bk, bn><<<grid, NTHREADS, 0, lc.st>>>(A, lda, a_op, dZ, ldz, dW, N, M, rows_per_cta); \
    ECNF_CHECK_CUDA(cudaGetLastError());                                                            \
    return ECNF_OK;                                                                                 \
  }
  DW_CASE(128, 128) DW_CASE(128, 64) DW_CASE(64, 128) DW_CASE(64, 64) DW_CASE(32, 128) DW_CASE(128, 32) DW_CASE(32, 64)
  DW_CASE(64, 32) DW_CASE(32, 32)
#undef DW_CASE
  ecnf_set_error("dw: unsupported block (%d,%d)", BK, BN);
  return ECNF_ERR_UNSUPPORTED;
}

// out[N] += column sums of Z[M,N]   (N <= 256)
__global__ void colsum_kernel(const float* __restrict__ Z, int M, int N, float* __restrict__ out, int rows_per_cta) {
  __shared__ float red[NTHREADS];
  const int tid = threadIdx.x, col = tid % N, lane_r = tid / N, nr = NTHREADS / N;
  const int m0 = blockIdx.x * rows_per_cta, m1 = min(M, m0 + rows_per_cta);
  // four independent partial sums keep four loads in flight per thread (the kernel is HBM bound)
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  int r = m0 + lane_r;
  for (; r + 3 * nr < m1; r += 4 * nr) {
    s0 += Z[(size_t)r * N + col];
    s1 += Z[(size_t)(r + nr) * N + col];
    s2 += Z[(size_t)(r + 2 * nr) * N + col];
    s3 += Z[(size_t)(r + 3 * nr) * N + col];
  }
  for (; r < m1; r += nr) s0 += Z[(size_t)r * N + col];
  float s = (s0 + s1) + (s2 + s3);
  red[tid] = s;
  __syncthreads();
  if (lane_r == 0) {
    for (int q = 1; q < nr; ++q) s += red[q * N + col];
    atomicAdd(out + col, s);
  }
}

// all weight transposes of a step in ONE launch: blockIdx.y = matrix, blockIdx.x strides over its 32 x 32 tiles
struct TrItem {
  const float* src;
  float* dst;
  int R, C;
};
struct TrList {
  int n;
  TrItem it[112];
};
__global__ void transpose_all_kernel(const __grid_constant__ TrList list) {
  __shared__ float tile[32][33];
  const TrItem it = list.it[blockIdx.y];
  const int tx = (it.C + 31) / 32, ty = (it.R + 31) / 32;
  for (int t = blockIdx.x; t < tx * ty; t += gridDim.x) {
    const int bx = (t % tx) * 32, by = (t / tx) * 32;
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
      const int r = by + i, c = bx + threadIdx.x;
      if (r < it.R && c < it.C) tile[i][threadIdx.x] = it.src[(size_t)r * it.C + c];
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
      const int c = bx + i, r = by + threadIdx.x;
      if (r < it.R && c < it.C) it.dst[(size_t)c * it.R + r] = tile[threadIdx.x][i];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// per-graph / per-edge / per-node kernels
// ------------------------------------------------------------------------------------------------
struct Dims {
  int B, n, dim, D, E, H, U, T, L, nfeat;
  float C, sigma_min;
  float freqs[8];   // fp32 timestep frequencies (build_cnf.py:25-27), from the model handle
};

// x_t, u_t (core.py:35-39), centring, time embedding (build_cnf.py:18-32), embedding lookup (build_cnf.py:79)
__global__ void fm_prep_kernel(Dims d, const float* __restrict__ x_data, const float* __restrict__ x0,
                               const float* __restrict__ t, const int32_t* __restrict__ feat,
                               const float* __restrict__ embed, float* __restrict__ ut,
                               float* __restrict__ mu, float* __restrict__ xs0, float* __restrict__ tau,
                               float* __restrict__ h0) {
  const int g = blockIdx.x, tid = threadIdx.x;
  __shared__ float xt[ECNF_MAX_NODES * 3];
  __shared__ float m[4];
  const float tt = t[g];
  for (int i = tid; i < d.D; i += blockDim.x) {
    const float a = x0[(size_t)g * d.D + i], b = x_data[(size_t)g * d.D + i];
    xt[i] = (1.f - (1.f - d.sigma_min) * tt) * a + tt * b;
    ut[(size_t)g * d.D + i] = b - (1.f - d.sigma_min) * a;
  }
  __syncthreads();
  if (tid < d.dim) {
    float s = 0.f;
    for (int i = 0; i < d.n; ++i) s += xt[i * d.dim + tid];
    m[tid] = s / (float)d.n;
    mu[(size_t)g * 4 + tid] = m[tid];
  }
  if (tid >= 32 && tid < 32 + d.T / 2) {
    const int k = tid - 32;
    const float arg = (tt * 1000.f) * d.freqs[k];
    tau[(size_t)g * d.T + k] = sinf(arg);
    tau[(size_t)g * d.T + k + d.T / 2] = cosf(arg);
  }
  __syncthreads();
  for (int i = tid; i < d.D; i += blockDim.x) xs0[(size_t)g * d.D + i] = xt[i] - m[i % d.dim];
  for (int idx = tid; idx < d.n * d.H; idx += blockDim.x) {
    const int node = idx / d.H, col = idx - node * d.H;
    int f = feat[(size_t)g * d.n + node];
    f = max(0, min(d.nfeat - 1, f));
    h0[((size_t)g * d.n + node) * d.H + col] = embed[f * d.H + col];
  }
}

// cvec[g][col] = bd[col] + sum_k tau[g][k] Wd[H + k][col]      (egnn.py:166-167, the tau part)
__global__ void tau_proj_kernel(Dims d, const float* __restrict__ tau, const float* __restrict__ Wd,
                                const float* __restrict__ bd, float* __restrict__ cvec) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= d.B * d.H) return;
  const int g = idx / d.H, col = idx - g * d.H;
  float a = bd[col];
  for (int k = 0; k < d.T; ++k) a = fmaf(tau[(size_t)g * d.T + k], Wd[(d.H + k) * d.H + col], a);
  cvec[idx] = a;
}

__device__ __forceinline__ void edge_nodes(int e_in_graph, int n, int& i, int& j) {
  i = e_in_graph / (n - 1);
  j = i + 1 + (e_in_graph - i * (n - 1));
  if (j >= n) j -= n;
}

// z_e0[e] = P_s[send] + P_r[recv] + |v|^2 w_d     (egnn.py:73-76 + first Dense of phi_e; bias folded into P_r)
__global__ void edge_gather_kernel(Dims d, const float* __restrict__ xs, const float* __restrict__ Ps,
                                   const float* __restrict__ Pr, const float* __restrict__ wd, float* __restrict__ Z) {
  const int U4 = d.U / 4;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)d.B * d.E * U4) return;
  const size_t erow = idx / U4;
  const int c4 = (int)(idx - erow * U4);
  const int g = (int)(erow / d.E);
  int i, j;
  edge_nodes((int)(erow - (size_t)g * d.E), d.n, i, j);
  float s = 0.f;
  for (int c = 0; c < d.dim; ++c) {
    const float v = xs[(size_t)g * d.D + i * d.dim + c] - xs[(size_t)g * d.D + j * d.dim + c];
    s = fmaf(v, v, s);
  }
  if (s == 0.f) s = 1.f;
  const float4 a = *reinterpret_cast<const float4*>(Ps + ((size_t)g * d.n + j) * d.U + c4 * 4);
  const float4 b = *reinterpret_cast<const float4*>(Pr + ((size_t)g * d.n + i) * d.U + c4 * 4);
  const float4 w = *reinterpret_cast<const float4*>(wd + c4 * 4);
  *reinterpret_cast<float4*>(Z + erow * d.U + c4 * 4) =
      make_float4(a.x + b.x + s * w.x, a.y + b.y + s * w.y, a.z + b.z + s * w.z, a.w + b.w + s * w.w);
}

// Lane l owns the VW = min(4, U/32) consecutive columns (32 v + l) VW .. of every group v < NV of 32 VW columns, so
// every access is one 8- or 16-byte vector and a warp covers 32 VW contiguous floats; all loads of a row are issued before
// the first use, and the elementwise SiLU uses ex2 / rcp (as in ecnf_train_tc.cuh).
template <int VW> struct VecT;
template <> struct VecT<2> { using T = float2; };
template <> struct VecT<4> { using T = float4; };
template <int VW>
__device__ __forceinline__ void ldv(const float* p, float (&o)[VW]) {
  const typename VecT<VW>::T v = *reinterpret_cast<const typename VecT<VW>::T*>(p);
  const float* f = reinterpret_cast<const float*>(&v);
#pragma unroll
  for (int i = 0; i < VW; ++i) o[i] = f[i];
}
template <int VW>
__device__ __forceinline__ void stv(float* p, const float (&o)[VW]) {
  typename VecT<VW>::T v;
  float* f = reinterpret_cast<float*>(&v);
#pragma unroll
  for (int i = 0; i < VW; ++i) f[i] = o[i];
  *reinterpret_cast<typename VecT<VW>::T*>(p) = v;
}

// per edge row (one warp): attention gate e = sigmoid(m.wa + ba), head p = y.wp + bp   (egnn.py:83-85, 99-101)
template <int U>
__global__ void edge_heads_kernel(Dims d, const float* __restrict__ Ze, const float* __restrict__ Zx,
                                  const float* __restrict__ wa, const float* __restrict__ ba,
                                  const float* __restrict__ wp, const float* __restrict__ bp, float* __restrict__ eatt,
                                  float* __restrict__ pout) {
  constexpr int Q = U / 32, VW = Q < 4 ? Q : 4, NV = Q / VW;
  using ecnf_train_tc::sigm;
  const int lane = threadIdx.x & 31;
  const size_t row = (size_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= (size_t)d.B * d.E) return;
  float sa = 0.f, sp = 0.f;
  float ze[NV][VW], zx[NV][VW], wav[NV][VW], wpv[NV][VW];
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int col = (32 * v + lane) * VW;
    ldv<VW>(Ze + row * U + col, ze[v]);
    ldv<VW>(Zx + row * U + col, zx[v]);
    ldv<VW>(wa + col, wav[v]);
    ldv<VW>(wp + col, wpv[v]);
  }
#pragma unroll
  for (int v = 0; v < NV; ++v)
#pragma unroll
    for (int k = 0; k < VW; ++k) {
      sa = fmaf(ze[v][k] * sigm(ze[v][k]), wav[v][k], sa);
      sp = fmaf(zx[v][k] * sigm(zx[v][k]), wpv[v][k], sp);
    }
  for (int o = 16; o > 0; o >>= 1) {
    sa += __shfl_xor_sync(0xffffffffu, sa, o);
    sp += __shfl_xor_sync(0xffffffffu, sp, o);
  }
  if (lane == 0) {
    eatt[row] = ecnf_sigmoid(sa + ba[0]);
    pout[row] = sp + bp[0];
  }
}

// per (graph, node): M_i = sum_j m_ij e_ij / sqrt(n-1);  x_i += sum_j p_ij v_ij / (C + |v_ij|) / (n-1)
__global__ void node_aggregate_kernel(Dims d, const float* __restrict__ xs, const float* __restrict__ Ze,
                                      const float* __restrict__ eatt, const float* __restrict__ p,
                                      float* __restrict__ Mout, float* __restrict__ xs_next, int want_m) {
  const int gi = blockIdx.x, g = gi / d.n, i = gi - g * d.n, tid = threadIdx.x;
  const size_t row0 = (size_t)g * d.E + (size_t)i * (d.n - 1);
  if (want_m) {
    using ecnf_train_tc::sigm;
    const float sc = rsqrtf((float)(d.n - 1));
    for (int c4 = tid; c4 < d.U / 4; c4 += blockDim.x) {
      float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 6
      for (int jj = 0; jj < d.n - 1; ++jj) {
        const float4 z = *reinterpret_cast<const float4*>(Ze + (row0 + jj) * d.U + 4 * c4);
        const float e = eatt[row0 + jj];
        s.x = fmaf(z.x * sigm(z.x), e, s.x); s.y = fmaf(z.y * sigm(z.y), e, s.y);
        s.z = fmaf(z.z * sigm(z.z), e, s.z); s.w = fmaf(z.w * sigm(z.w), e, s.w);
      }
      *reinterpret_cast<float4*>(Mout + (size_t)gi * d.U + 4 * c4) = make_float4(s.x * sc, s.y * sc, s.z * sc, s.w * sc);
    }
  }
  if (tid < d.dim) {
    const float* xg = xs + (size_t)g * d.D;
    float acc = 0.f;
    for (int jj = 0; jj < d.n - 1; ++jj) {
      int j = i + 1 + jj; if (j >= d.n) j -= d.n;
      float s = 0.f;
      for (int c = 0; c < d.dim; ++c) { const float v = xg[i * d.dim + c] - xg[j * d.dim + c]; s = fmaf(v, v, s); }
      const float len = sqrtf(s == 0.f ? 1.f : s);
      acc = fmaf(p[row0 + jj] * (xg[i * d.dim + tid] - xg[j * d.dim + tid]), 1.f / (d.C + len), acc);
    }
    xs_next[(size_t)g * d.D + i * d.dim + tid] = xg[i * d.dim + tid] + acc / (float)(d.n - 1);
  }
}

// v = (x_L - x_0 - mu) fs; loss = sum (v-u)^2 / denom; d x_L = 2 (v-u) fs / denom; d fs
__global__ void loss_kernel(Dims d, const float* __restrict__ xsL, const float* __restrict__ xs0,
                            const float* __restrict__ mu, const float* __restrict__ ut, const float* __restrict__ fs,
                            float denom, float* __restrict__ loss, float* __restrict__ dxs, float* __restrict__ dfs) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  float l = 0.f, df = 0.f;
  if (idx < (size_t)d.B * d.D) {
    const int g = (int)(idx / d.D), k = (int)(idx - (size_t)g * d.D);
    const float raw = xsL[idx] - xs0[idx] - mu[(size_t)g * 4 + k % d.dim];
    const float f = fs[0];
    const float diff = raw * f - ut[idx];
    l = diff * diff / denom;
    const float dv = 2.f * diff / denom;
    dxs[idx] = dv * f;
    df = dv * raw;
  }
  for (int o = 16; o > 0; o >>= 1) {
    l += __shfl_xor_sync(0xffffffffu, l, o);
    df += __shfl_xor_sync(0xffffffffu, df, o);
  }
  __shared__ float sl[32], sd[32];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { sl[w] = l; sd[w] = df; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int q = 1; q < (blockDim.x >> 5); ++q) { l += sl[q]; df += sd[q]; }
    atomicAdd(loss, l);
    atomicAdd(dfs, df);
  }
}

// backward of attention / message / head / coordinate update, one warp per edge row.
// In:  dM [B*n, U] (grad wrt aggregated message, null in the last block), dxs_next [B, D]
// Out: DM [EB, U] = grad wrt m from the message path (0 if last); Zx <- d z_x[L-1] (in place);
//      dvgeo [EB, 4] = grad wrt v_ij from the coordinate path; accumulates d wa, d ba, d wp, d bp.
template <int U>
__global__ void __launch_bounds__(256) heads_bwd_kernel(Dims d, const float* __restrict__ xs, const float* __restrict__ Ze,
                                 float* __restrict__ Zx, const float* __restrict__ eatt, const float* __restrict__ p,
                                 const float* __restrict__ dM, const float* __restrict__ dxs_next,
                                 const float* __restrict__ wa, const float* __restrict__ wp, float* __restrict__ DM,
                                 float* __restrict__ dvgeo, float* __restrict__ g_wa, float* __restrict__ g_ba,
                                 float* __restrict__ g_wp, float* __restrict__ g_bp, int rows_per_warp) {
  constexpr int Q = U / 32, VW = Q < 4 ? Q : 4, NV = Q / VW;
  using ecnf_train_tc::sigm;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const size_t EB = (size_t)d.B * d.E;
  const size_t r_begin = ((size_t)blockIdx.x * nw + warp) * rows_per_warp;
  const size_t r_end = min(EB, r_begin + rows_per_warp);
  float awa[NV][VW], awp[NV][VW], aba = 0.f, abp = 0.f, wav[NV][VW], wpv[NV][VW];
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    ldv<VW>(wa + (32 * v + lane) * VW, wav[v]);
    ldv<VW>(wp + (32 * v + lane) * VW, wpv[v]);
#pragma unroll
    for (int i = 0; i < VW; ++i) { awa[v][i] = 0.f; awp[v][i] = 0.f; }
  }
  const float inv_sqrt = rsqrtf((float)(d.n - 1)), inv_nb = 1.f / (float)(d.n - 1);
#pragma unroll 2
  for (size_t row = r_begin; row < r_end; ++row) {
    const int g = (int)(row / d.E);
    int i, j;
    edge_nodes((int)(row - (size_t)g * d.E), d.n, i, j);
    float ze[NV][VW], zx[NV][VW], dmr[NV][VW];
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int col = (32 * v + lane) * VW;
      ldv<VW>(Ze + row * U + col, ze[v]);
      ldv<VW>(Zx + row * U + col, zx[v]);
      if (dM) ldv<VW>(dM + ((size_t)g * d.n + i) * U + col, dmr[v]);
    }
    const float* xg = xs + (size_t)g * d.D;
    float v3[3] = {0.f, 0.f, 0.f}, s = 0.f, dcv = 0.f, dc[3] = {0.f, 0.f, 0.f};
    for (int c = 0; c < d.dim; ++c) {
      v3[c] = xg[i * d.dim + c] - xg[j * d.dim + c];
      s = fmaf(v3[c], v3[c], s);
      dc[c] = dxs_next[(size_t)g * d.D + i * d.dim + c] * inv_nb;
      dcv = fmaf(dc[c], v3[c], dcv);
    }
    const bool isz = (s == 0.f);
    const float len = sqrtf(isz ? 1.f : s), inv = 1.f / (d.C + len);
    const float pv = p[row], e = eatt[row];
    const float dp = dcv * inv;
    float de = 0.f;
#pragma unroll
    for (int v = 0; v < NV; ++v)
#pragma unroll
      for (int k = 0; k < VW; ++k) {
        ze[v][k] *= sigm(ze[v][k]);                       // m = silu(z_e)
        if (dM) { dmr[v][k] *= inv_sqrt; de = fmaf(dmr[v][k], ze[v][k], de); }
      }
    for (int o = 16; o > 0; o >>= 1) de += __shfl_xor_sync(0xffffffffu, de, o);
    const float dlogit = de * e * (1.f - e);
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int col = (32 * v + lane) * VW;
      float dm[VW], dzx[VW];
#pragma unroll
      for (int k = 0; k < VW; ++k) {
        dm[k] = 0.f;
        if (dM) {
          dm[k] = fmaf(dmr[v][k], e, dlogit * wav[v][k]);
          awa[v][k] = fmaf(dlogit, ze[v][k], awa[v][k]);
        }
        const float z = zx[v][k], sg = sigm(z);
        awp[v][k] = fmaf(dp, z * sg, awp[v][k]);
        dzx[k] = dp * wpv[v][k] * (sg * (1.f + z * (1.f - sg)));
      }
      stv<VW>(DM + row * U + col, dm);
      stv<VW>(Zx + row * U + col, dzx);
    }
    aba += dlogit;
    abp += dp;
    if (lane < d.dim) {
      float gv = dc[lane] * pv * inv;
      if (!isz) gv -= pv * dcv * inv * inv * v3[lane] / len;
      dvgeo[row * 4 + lane] = gv;
    }
  }
  // block reduction of the vector accumulators
  __shared__ float red[8][2 * 256 + 2];
#pragma unroll
  for (int v = 0; v < NV; ++v)
#pragma unroll
    for (int k = 0; k < VW; ++k) {
      red[warp][(32 * v + lane) * VW + k] = awa[v][k];
      red[warp][U + (32 * v + lane) * VW + k] = awp[v][k];
    }
  if (lane == 0) { red[warp][2 * U] = aba; red[warp][2 * U + 1] = abp; }
  __syncthreads();
  for (int idx = threadIdx.x; idx < 2 * U + 2; idx += blockDim.x) {
    float sacc = 0.f;
    for (int w = 0; w < nw; ++w) sacc += red[w][idx];
    if (idx < U) { if (dM) atomicAdd(g_wa + idx, sacc); }
    else if (idx < 2 * U) atomicAdd(g_wp + (idx - U), sacc);
    else if (idx == 2 * U) { if (dM) atomicAdd(g_ba, sacc); }
    else atomicAdd(g_bp, sacc);
  }
}

// per edge row: d|v|^2 = dz_e0 . w_d  ->  dvgeo += 2 d|v|^2 v ;  d w_d += |v|^2 dz_e0
template <int U>
__global__ void __launch_bounds__(256) gather_bwd_edge_kernel(Dims d, const float* __restrict__ xs, const float* __restrict__ dZ,
                                       const float* __restrict__ wd, float* __restrict__ dvgeo, float* __restrict__ g_wd,
                                       float* __restrict__ g_be, int rows_per_warp) {
  constexpr int Q = U / 32, VW = Q < 4 ? Q : 4, NV = Q / VW;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const size_t EB = (size_t)d.B * d.E;
  const size_t r_begin = ((size_t)blockIdx.x * nw + warp) * rows_per_warp;
  const size_t r_end = min(EB, r_begin + rows_per_warp);
  float awd[NV][VW], abe[NV][VW], wdv[NV][VW];      // d w_d, d b_e0 (column sums of dZ), w_d
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    ldv<VW>(wd + (32 * v + lane) * VW, wdv[v]);
#pragma unroll
    for (int k = 0; k < VW; ++k) { awd[v][k] = 0.f; abe[v][k] = 0.f; }
  }
#pragma unroll 2
  for (size_t row = r_begin; row < r_end; ++row) {
    float z[NV][VW];
#pragma unroll
    for (int v = 0; v < NV; ++v) ldv<VW>(dZ + row * U + (32 * v + lane) * VW, z[v]);
    const int g = (int)(row / d.E);
    int i, j;
    edge_nodes((int)(row - (size_t)g * d.E), d.n, i, j);
    const float* xg = xs + (size_t)g * d.D;
    float v3[3] = {0.f, 0.f, 0.f}, s = 0.f;
    for (int c = 0; c < d.dim; ++c) { v3[c] = xg[i * d.dim + c] - xg[j * d.dim + c]; s = fmaf(v3[c], v3[c], s); }
    const bool isz = (s == 0.f);
    const float s1 = isz ? 1.f : s;
    float ds = 0.f;
#pragma unroll
    for (int v = 0; v < NV; ++v)
#pragma unroll
      for (int k = 0; k < VW; ++k) {
        ds = fmaf(z[v][k], wdv[v][k], ds);
        awd[v][k] = fmaf(s1, z[v][k], awd[v][k]);
        abe[v][k] += z[v][k];
      }
    for (int o = 16; o > 0; o >>= 1) ds += __shfl_xor_sync(0xffffffffu, ds, o);
    if (lane < d.dim && !isz) dvgeo[row * 4 + lane] += 2.f * ds * v3[lane];
  }
  __shared__ float red[8][2 * 256];
#pragma unroll
  for (int v = 0; v < NV; ++v)
#pragma unroll
    for (int k = 0; k < VW; ++k) {
      red[warp][(32 * v + lane) * VW + k] = awd[v][k];
      red[warp][U + (32 * v + lane) * VW + k] = abe[v][k];
    }
  __syncthreads();
  for (int idx = threadIdx.x; idx < 2 * U; idx += blockDim.x) {
    float sacc = 0.f;
    for (int w = 0; w < nw; ++w) sacc += red[w][idx];
    atomicAdd((idx < U ? g_wd : g_be - U) + idx, sacc);
  }
}

// per (graph, node a): dP_r[a] = sum over edges received by a; dP_s[a] = sum over edges sent by a;
// d x_a = d x_a(next) + sum_recv dv - sum_send dv
__global__ void gather_bwd_node_kernel(Dims d, const float* __restrict__ dZ, const float* __restrict__ dvgeo,
                                       const float* __restrict__ dxs_next, float* __restrict__ dPs,
                                       float* __restrict__ dPr, float* __restrict__ dxs) {
  const int ga = blockIdx.x, g = ga / d.n, a = ga - g * d.n, tid = threadIdx.x;
  const size_t e0 = (size_t)g * d.E;
  // one float4 column group per thread; the loads of the unrolled edge loops are independent (HBM / L2 bound)
  for (int c4 = tid; c4 < d.U / 4; c4 += blockDim.x) {
    float4 sr = make_float4(0.f, 0.f, 0.f, 0.f), ss = sr;
    const float* base = dZ + e0 * d.U + 4 * c4;
#pragma unroll 6
    for (int jj = 0; jj < d.n - 1; ++jj) {
      const float4 z = *reinterpret_cast<const float4*>(base + ((size_t)a * (d.n - 1) + jj) * d.U);
      sr.x += z.x; sr.y += z.y; sr.z += z.z; sr.w += z.w;
    }
#pragma unroll 6
    for (int k = 1; k < d.n; ++k) {            // senders i = a + k (mod n): their edge to a is slot jj = n - 1 - k
      int i = a + k; if (i >= d.n) i -= d.n;
      const float4 z = *reinterpret_cast<const float4*>(base + ((size_t)i * (d.n - 1) + (d.n - 1 - k)) * d.U);
      ss.x += z.x; ss.y += z.y; ss.z += z.z; ss.w += z.w;
    }
    *reinterpret_cast<float4*>(dPr + (size_t)ga * d.U + 4 * c4) = sr;
    *reinterpret_cast<float4*>(dPs + (size_t)ga * d.U + 4 * c4) = ss;
  }
  if (dxs && tid < d.dim) {
    float acc = dxs_next[(size_t)g * d.D + a * d.dim + tid];
    for (int jj = 0; jj < d.n - 1; ++jj) acc += dvgeo[(e0 + (size_t)a * (d.n - 1) + jj) * 4 + tid];
    for (int i = 0; i < d.n; ++i) {
      if (i == a) continue;
      int jj = a - i - 1; if (jj < 0) jj += d.n;
      acc -= dvgeo[(e0 + (size_t)i * (d.n - 1) + jj) * 4 + tid];
    }
    dxs[(size_t)g * d.D + a * d.dim + tid] = acc;
  }
}

// d Wd[H + k][col] += sum_g tau[g][k] * sum_i dhin[g, i][col]
__global__ void tau_grad_kernel(Dims d, const float* __restrict__ tau, const float* __restrict__ dhin,
                                float* __restrict__ g_Wd_tau, int graphs_per_cta) {
  const int col = threadIdx.x % d.H, k = threadIdx.x / d.H;  // blockDim = H * T
  const int g0 = blockIdx.x * graphs_per_cta, g1 = min(d.B, g0 + graphs_per_cta);
  float acc = 0.f;
  for (int g = g0; g < g1; ++g) {
    float s = 0.f;
    for (int i = 0; i < d.n; ++i) s += dhin[((size_t)g * d.n + i) * d.H + col];
    acc = fmaf(tau[(size_t)g * d.T + k], s, acc);
  }
  atomicAdd(g_Wd_tau + k * d.H + col, acc);
}

__global__ void embed_bwd_kernel(Dims d, const int32_t* __restrict__ feat, const float* __restrict__ dh,
                                 float* __restrict__ g_embed) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)d.B * d.n * d.H) return;
  const size_t node = idx / d.H;
  const int col = (int)(idx - node * d.H);
  int f = feat[node];
  f = max(0, min(d.nfeat - 1, f));
  atomicAdd(g_embed + f * d.H + col, dh[idx]);
}

// ------------------------------------------------------------------------------------------------
// host orchestration
// ------------------------------------------------------------------------------------------------
// Graphs per chunk of a minibatch (ecnf_model_set_fm_chunk; 0 = the whole minibatch in one pass); the gradients of the
// chunks accumulate
int64_t fm_chunk_graphs(const ecnf_model* m, int64_t B) { return m->fm_chunk > 0 && m->fm_chunk < B ? m->fm_chunk : B; }

// Every buffer of the workspace of one chunk
struct FmWorkspace {
  float *ut, *mu, *tau, *xs[ECNF_MAX_BLOCKS + 1], *dxs[2], *cvec;
  float *hprev[ECNF_MAX_BLOCKS + 1], *hin[ECNF_MAX_BLOCKS];
  float *Ps, *Pr;   // also dPs, dPr
  float *Mb[ECNF_MAX_BLOCKS], *Zh[ECNF_MAX_BLOCKS][ECNF_MAX_LAYERS];
  float *Ze[ECNF_MAX_BLOCKS][ECNF_MAX_LAYERS], *Zx[ECNF_MAX_BLOCKS][ECNF_MAX_LAYERS];
  float *pb[ECNF_MAX_BLOCKS], *eb[ECNF_MAX_BLOCKS];
  float *DM, *dvgeo, *dM, *dhin, *dh[2];
  float* Wt;   // transposed weights, at the offsets of the parameter layout
};

// Lays out the buffers of a chunk of `Bws` graphs from `base` into `w` (256-byte aligned) and returns the bytes they
// take.  With a null base it only counts: ecnf_fm_workspace_bytes sizes the workspace with it.
size_t fm_layout(const ecnf_model* m, int64_t Bws, void* base, FmWorkspace& w) {
  const ecnf_config& c = m->cfg;
  const size_t n = c.n_frames, D = n * c.dim, H = c.n_hidden, U = c.mlp_units, T = c.time_dim;
  const size_t B = (size_t)Bws, NB = B * n, EB = B * n * (n - 1);
  const int nb = c.n_blocks, L = c.n_layers;
  size_t off = 256;
  auto take = [&](size_t nfloats) {
    float* p = base ? reinterpret_cast<float*>(static_cast<char*>(base) + off) : nullptr;
    off += (nfloats * sizeof(float) + 255) & ~(size_t)255;
    return p;
  };
  w.ut = take(B * D);
  w.mu = take(B * 4);
  w.tau = take(B * T);
  for (int b = 0; b <= nb; ++b) w.xs[b] = take(B * D);
  for (float*& p : w.dxs) p = take(B * D);
  w.cvec = take(B * H);
  for (int b = 0; b <= nb; ++b) w.hprev[b] = take(NB * H);
  for (int b = 0; b < nb; ++b) w.hin[b] = take(NB * H);
  w.Ps = take(NB * U);
  w.Pr = take(NB * U);
  for (int b = 0; b < nb; ++b) w.Mb[b] = take(NB * U);
  for (int b = 0; b < nb; ++b)
    for (int l = 0; l < L; ++l) w.Zh[b][l] = take(NB * U);
  for (int b = 0; b < nb; ++b)
    for (int l = 0; l < L; ++l) { w.Ze[b][l] = take(EB * U); w.Zx[b][l] = take(EB * U); }
  for (int b = 0; b < nb; ++b) { w.pb[b] = take(EB); w.eb[b] = take(EB); }
  w.DM = take(EB * U);
  w.dvgeo = take(EB * 4);
  w.dM = take(NB * U);
  w.dhin = take(NB * H);
  for (float*& p : w.dh) p = take(NB * H);
  w.Wt = take((size_t)m->param_count);
  return off;
}

// One chunk of `B` graphs (rows [0, B) of the pointers given) through forward + backward.  The workspace is laid out for
// `Bws` >= B graphs; every gradient (and the loss) is ACCUMULATED, so the chunks of a minibatch add up.  `first`: clear the
// gradient / loss and transpose the weights (once per minibatch).
template <int U, int H>
int fm_run(const ecnf_model* m, const float* x_data, const float* x0, const float* t, const int32_t* feat, int64_t B,
           int64_t Bws, bool first, float denom, float* out_loss, float* out_grad, void* ws, const LaunchCtx& lc) {
  const ecnf_config& c = m->cfg;
  const EcnfModelDev md = ecnf_make_dev(m, m->d_params);
  const EcnfModelDev gd = ecnf_make_dev(m, out_grad);  // same layout, pointing into the gradient buffer
  Dims d;
  d.B = (int)B; d.n = c.n_frames; d.dim = c.dim; d.D = d.n * d.dim; d.E = d.n * (d.n - 1); d.H = H; d.U = U;
  d.T = c.time_dim; d.L = c.n_layers; d.nfeat = c.n_features; d.C = c.normalization_constant; d.sigma_min = c.sigma_min;
  for (int k = 0; k < 8; ++k) d.freqs[k] = c.freqs[k];
  const int nb = c.n_blocks, L = c.n_layers;
  const size_t NB = (size_t)B * d.n, EB = (size_t)B * d.E;
  const cudaStream_t st = lc.st;
  FmWorkspace w;
  fm_layout(m, Bws, ws, w);
  const EcnfModelDev td = ecnf_make_dev(m, w.Wt);  // transposed weights live at the same offsets

  if (first) {
    ECNF_CHECK_CUDA(cudaMemsetAsync(out_grad, 0, (size_t)m->param_count * sizeof(float), st));
    ECNF_CHECK_CUDA(cudaMemsetAsync(out_loss, 0, sizeof(float), st));
  }

  TrList trl;
  trl.n = 0;
  auto transpose_flush = [&]() {
    if (trl.n > 0) transpose_all_kernel<<<dim3(16, trl.n), dim3(32, 8), 0, st>>>(trl);
    trl.n = 0;
  };
  auto transpose = [&](const float* W, const float* Wt_c, int R, int Cc) {
    if (trl.n == 112) transpose_flush();
    trl.it[trl.n++] = TrItem{W, const_cast<float*>(Wt_c), R, Cc};
  };
  for (int b = 0; first && b < nb; ++b) {
    const EcnfBlockParams &p = md.blk[b], &q = td.blk[b];
    transpose(p.Wd, q.Wd, H, H);
    transpose(p.We[0], q.We[0], H, U);
    transpose(p.We[0] + (size_t)H * U, q.We[0] + (size_t)H * U, H, U);
    for (int l = 1; l < L; ++l) transpose(p.We[l], q.We[l], U, U);
    for (int l = 0; l < L; ++l) transpose(p.Wx[l], q.Wx[l], U, U);
    if (b + 1 < nb) {
      transpose(p.Wh[0], q.Wh[0], U, U);
      transpose(p.Wh[0] + (size_t)U * U, q.Wh[0] + (size_t)U * U, H, U);
      for (int l = 1; l < L; ++l) transpose(p.Wh[l], q.Wh[l], U, U);
      transpose(p.Wh[L], q.Wh[L], U, H);
    }
  }
  transpose_flush();
  ECNF_CHECK_CUDA(cudaGetLastError());

  auto gemm_args = [](const float* A, const float* W, float* C, int M) {
    GemmArgs g{};
    g.A = A; g.W = W; g.C = C; g.M = M; g.rows_per_vec = 1;
    return g;
  };
  const int ew_threads = 256;
  const int rows_per_warp = 8;
  const int heads_grid = (int)((EB + 8 * rows_per_warp - 1) / (8 * rows_per_warp));
  int rc;

  // ------------------------------ forward ------------------------------
  fm_prep_kernel<<<(unsigned)B, 128, 0, st>>>(d, x_data, x0, t, feat, md.embed, w.ut, w.mu, w.xs[0], w.tau, w.hprev[0]);
  for (int b = 0; b < nb; ++b) {
    const EcnfBlockParams& p = md.blk[b];
    const bool last = (b == nb - 1);
    tau_proj_kernel<<<(unsigned)((B * H + 255) / 256), 256, 0, st>>>(d, w.tau, p.Wd, p.bd, w.cvec);
    {
      GemmArgs g = gemm_args(w.hprev[b], p.Wd, w.hin[b], (int)NB);
      g.rowvec = w.cvec; g.rows_per_vec = d.n;
      if ((rc = launch_gemm<H, H, 0>(lc, g))) return rc;
    }
    {
      GemmArgs g = gemm_args(w.hin[b], p.We[0], w.Ps, (int)NB);
      if ((rc = launch_gemm<H, U, 0>(lc, g))) return rc;
      g = gemm_args(w.hin[b], p.We[0] + (size_t)H * U, w.Pr, (int)NB);
      g.bias = p.be[0];
      if ((rc = launch_gemm<H, U, 0>(lc, g))) return rc;
    }
    edge_gather_kernel<<<(unsigned)((EB * (U / 4) + ew_threads - 1) / ew_threads), ew_threads, 0, st>>>(
        d, w.xs[b], w.Ps, w.Pr, p.We[0] + (size_t)2 * H * U, w.Ze[b][0]);
    for (int l = 1; l < L; ++l) {
      GemmArgs g = gemm_args(w.Ze[b][l - 1], p.We[l], w.Ze[b][l], (int)EB);
      g.a_op = 1; g.bias = p.be[l];
      if ((rc = launch_gemm<U, U, H>(lc, g))) return rc;
    }
    for (int l = 0; l < L; ++l) {
      GemmArgs g = gemm_args(l == 0 ? w.Ze[b][L - 1] : w.Zx[b][l - 1], p.Wx[l], w.Zx[b][l], (int)EB);
      g.a_op = 1; g.bias = p.bx[l];
      if ((rc = launch_gemm<U, U, H>(lc, g))) return rc;
    }
    edge_heads_kernel<U><<<(unsigned)((EB + 7) / 8), 256, 0, st>>>(d, w.Ze[b][L - 1], w.Zx[b][L - 1], p.wa, p.ba, p.wp, p.bp,
                                                                 w.eb[b], w.pb[b]);
    node_aggregate_kernel<<<(unsigned)NB, U / 4 < 32 ? 32 : U / 4, 0, st>>>(d, w.xs[b], w.Ze[b][L - 1], w.eb[b], w.pb[b], w.Mb[b], w.xs[b + 1], !last);
    if (!last) {
      GemmArgs g = gemm_args(w.Mb[b], p.Wh[0], w.Zh[b][0], (int)NB);
      g.A2 = w.hin[b]; g.W2 = p.Wh[0] + (size_t)U * U; g.bias = p.bh[0];
      if ((rc = launch_gemm<U, U, H>(lc, g))) return rc;
      for (int l = 1; l < L; ++l) {
        g = gemm_args(w.Zh[b][l - 1], p.Wh[l], w.Zh[b][l], (int)NB);
        g.a_op = 1; g.bias = p.bh[l];
        if ((rc = launch_gemm<U, U, H>(lc, g))) return rc;
      }
      g = gemm_args(w.Zh[b][L - 1], p.Wh[L], w.hprev[b + 1], (int)NB);
      g.a_op = 1; g.bias = p.bh[L]; g.resid = w.hin[b];
      if ((rc = launch_gemm<U, H, 0>(lc, g))) return rc;
    }
  }
  loss_kernel<<<(unsigned)((B * d.D + 255) / 256), 256, 0, st>>>(d, w.xs[nb], w.xs[0], w.mu, w.ut, md.final_scaling, denom, out_loss,
                                                               w.dxs[0], const_cast<float*>(gd.final_scaling));
  ECNF_CHECK_CUDA(cudaGetLastError());

  // ------------------------------ backward ------------------------------
  int cur = 0;        // dxs[cur] = grad wrt coordinates leaving block b
  int hcur = 0;       // dh[hcur] = grad wrt h leaving block b (valid for b < nb-1)
  for (int b = nb - 1; b >= 0; --b) {
    const EcnfBlockParams &p = md.blk[b], &q = td.blk[b], &gp = gd.blk[b];
    const bool last = (b == nb - 1);
    bool dhin_valid = false;
    if (!last) {
      // h_out = phi_h([M | h_in]) + h_in
      const float* dho = w.dh[hcur];
      if ((rc = launch_dw(lc, w.Zh[b][L - 1], U, 1, dho, H, const_cast<float*>(gp.Wh[L]), U, H, (int)NB))) return rc;
      launch_colsum(lc, dho, (int)NB, H, const_cast<float*>(gp.bh[L]));
      GemmArgs g = gemm_args(dho, q.Wh[L], w.Zh[b][L - 1], (int)NB);   // [NB,H] x [H,U]
      g.mulz = w.Zh[b][L - 1];
      if ((rc = launch_gemm<H, U, 0>(lc, g))) return rc;
      for (int l = L - 1; l >= 1; --l) {
        if ((rc = launch_dw(lc, w.Zh[b][l - 1], U, 1, w.Zh[b][l], U, const_cast<float*>(gp.Wh[l]), U, U, (int)NB))) return rc;
        launch_colsum(lc, w.Zh[b][l], (int)NB, U, const_cast<float*>(gp.bh[l]));
        g = gemm_args(w.Zh[b][l], q.Wh[l], w.Zh[b][l - 1], (int)NB);
        g.mulz = w.Zh[b][l - 1];
        if ((rc = launch_gemm<U, U, H>(lc, g))) return rc;
      }
      if ((rc = launch_dw(lc, w.Mb[b], U, 0, w.Zh[b][0], U, const_cast<float*>(gp.Wh[0]), U, U, (int)NB))) return rc;
      if ((rc = launch_dw(lc, w.hin[b], H, 0, w.Zh[b][0], U, const_cast<float*>(gp.Wh[0]) + (size_t)U * U, H, U, (int)NB))) return rc;
      launch_colsum(lc, w.Zh[b][0], (int)NB, U, const_cast<float*>(gp.bh[0]));
      g = gemm_args(w.Zh[b][0], q.Wh[0], w.dM, (int)NB);
      if ((rc = launch_gemm<U, U, H>(lc, g))) return rc;
      g = gemm_args(w.Zh[b][0], q.Wh[0] + (size_t)U * U, w.dhin, (int)NB);   // [NB,U] x [U,H]
      g.resid = dho;
      if ((rc = launch_gemm<U, H, 0>(lc, g))) return rc;
      dhin_valid = true;
    }
    // attention / head / coordinate update
    heads_bwd_kernel<U><<<heads_grid, 256, 0, st>>>(d, w.xs[b], w.Ze[b][L - 1], w.Zx[b][L - 1], w.eb[b], w.pb[b], last ? nullptr : w.dM,
                                                   w.dxs[cur], p.wa, p.wp, w.DM, w.dvgeo, const_cast<float*>(gp.wa),
                                                   const_cast<float*>(gp.ba), const_cast<float*>(gp.wp),
                                                   const_cast<float*>(gp.bp), rows_per_warp);
    // phi_x chain
    for (int l = L - 1; l >= 0; --l) {
      const float* Ain = (l == 0) ? w.Ze[b][L - 1] : w.Zx[b][l - 1];
      if ((rc = launch_dw(lc, Ain, U, 1, w.Zx[b][l], U, const_cast<float*>(gp.Wx[l]), U, U, (int)EB,
                          const_cast<float*>(gp.bx[l])))) return rc;
      GemmArgs g = gemm_args(w.Zx[b][l], q.Wx[l], l == 0 ? w.Ze[b][L - 1] : w.Zx[b][l - 1], (int)EB);
      g.mulz = (l == 0) ? w.Ze[b][L - 1] : w.Zx[b][l - 1];
      if (l == 0) g.add = w.DM;
      if ((rc = launch_gemm<U, U, H>(lc, g))) return rc;
    }
    // phi_e chain
    for (int l = L - 1; l >= 1; --l) {
      if ((rc = launch_dw(lc, w.Ze[b][l - 1], U, 1, w.Ze[b][l], U, const_cast<float*>(gp.We[l]), U, U, (int)EB,
                          const_cast<float*>(gp.be[l])))) return rc;
      GemmArgs g = gemm_args(w.Ze[b][l], q.We[l], w.Ze[b][l - 1], (int)EB);
      g.mulz = w.Ze[b][l - 1];
      if ((rc = launch_gemm<U, U, H>(lc, g))) return rc;
    }
    // first phi_e layer: gather backward
    // first phi_e layer: d|v|^2 -> dvgeo, d w_d and the bias gradient (column sums of dZ_e0) in one pass over dZ_e0
    gather_bwd_edge_kernel<U><<<heads_grid, 256, 0, st>>>(d, w.xs[b], w.Ze[b][0], p.We[0] + (size_t)2 * H * U, w.dvgeo,
                                                         const_cast<float*>(gp.We[0]) + (size_t)2 * H * U,
                                                         const_cast<float*>(gp.be[0]), rows_per_warp);
    gather_bwd_node_kernel<<<(unsigned)NB, U / 4 < 32 ? 32 : U / 4, 0, st>>>(d, w.Ze[b][0], w.dvgeo, w.dxs[cur], w.Ps, w.Pr, b > 0 ? w.dxs[cur ^ 1] : nullptr);
    if ((rc = launch_dw(lc, w.hin[b], H, 0, w.Ps, U, const_cast<float*>(gp.We[0]), H, U, (int)NB))) return rc;
    if ((rc = launch_dw(lc, w.hin[b], H, 0, w.Pr, U, const_cast<float*>(gp.We[0]) + (size_t)H * U, H, U, (int)NB))) return rc;
    {
      GemmArgs g = gemm_args(w.Ps, q.We[0], w.dhin, (int)NB);   // [NB,U] x [U,H]
      if (dhin_valid) g.resid = w.dhin;
      if ((rc = launch_gemm<U, H, 0>(lc, g))) return rc;
      g = gemm_args(w.Pr, q.We[0] + (size_t)H * U, w.dhin, (int)NB);
      g.resid = w.dhin;
      if ((rc = launch_gemm<U, H, 0>(lc, g))) return rc;
    }
    // h_in = [h | tau] Wd + bd
    if ((rc = launch_dw(lc, w.hprev[b], H, 0, w.dhin, H, const_cast<float*>(gp.Wd), H, H, (int)NB))) return rc;
    launch_colsum(lc, w.dhin, (int)NB, H, const_cast<float*>(gp.bd));
    tau_grad_kernel<<<(unsigned)((B + 15) / 16), H * d.T, 0, st>>>(d, w.tau, w.dhin, const_cast<float*>(gp.Wd) + (size_t)H * H, 16);
    {
      GemmArgs g = gemm_args(w.dhin, q.Wd, w.dh[hcur ^ 1], (int)NB);
      if ((rc = launch_gemm<H, H, 0>(lc, g))) return rc;
      hcur ^= 1;
    }
    cur ^= 1;
  }
  embed_bwd_kernel<<<(unsigned)((NB * H + 255) / 256), 256, 0, st>>>(d, feat, w.dh[hcur], const_cast<float*>(gd.embed));
  ECNF_CHECK_CUDA(cudaGetLastError());
  return ECNF_OK;
}

}  // namespace

extern "C" {

int64_t ecnf_fm_workspace_bytes(const ecnf_model* m, int64_t B) {
  if (!m || B <= 0) return 256;
  FmWorkspace w;
  return (int64_t)fm_layout(m, fm_chunk_graphs(m, B), nullptr, w);
}

int ecnf_fm_loss_grad(const ecnf_model* m, const float* x_data, const float* x0, const float* t, const int32_t* feat,
                      int64_t B, float loss_denominator, float* out_loss, float* out_grad, void* ws, int64_t ws_bytes,
                      void* stream) {
  if (!m || !x_data || !x0 || !t || !feat || !out_loss || !out_grad || B <= 0 || !(loss_denominator > 0.f)) {
    ecnf_set_error("ecnf_fm_loss_grad: bad argument");
    return ECNF_ERR_INVALID;
  }
  if (B * (int64_t)m->cfg.n_frames * (m->cfg.n_frames - 1) > 0x7fffffffLL / 4) {
    ecnf_set_error("ecnf_fm_loss_grad: batch too large for 32-bit row indices");
    return ECNF_ERR_UNSUPPORTED;
  }
  const int64_t need = ecnf_fm_workspace_bytes(m, B);
  if (!ws || ws_bytes < need) {
    ecnf_set_error("workspace too small: need %lld bytes, got %lld", (long long)need, (long long)ws_bytes);
    return ECNF_ERR_WORKSPACE;
  }
  const LaunchCtx lc{m->num_sms, m->engine == 0, (cudaStream_t)stream};
  const int U = m->cfg.mlp_units, H = m->cfg.n_hidden;
  if (!((U == 128 && H == 64) || (U == 256 && H == 32) || (U == 64 && H == 32))) {
    ecnf_set_error("unsupported (mlp_units=%d, n_hidden=%d): compiled pairs are (128,64), (256,32), (64,32)", U, H);
    return ECNF_ERR_UNSUPPORTED;
  }
  const int64_t Bc = fm_chunk_graphs(m, B), D = (int64_t)m->cfg.n_frames * m->cfg.dim, n = m->cfg.n_frames;
  for (int64_t b0 = 0; b0 < B; b0 += Bc) {
    const int64_t bn = B - b0 < Bc ? B - b0 : Bc;
    const float *xd = x_data + b0 * D, *xz = x0 + b0 * D, *tt = t + b0;
    const int32_t* ft = feat + b0 * n;
    int rc;
    if (U == 128) rc = fm_run<128, 64>(m, xd, xz, tt, ft, bn, Bc, b0 == 0, loss_denominator, out_loss, out_grad, ws, lc);
    else if (U == 256) rc = fm_run<256, 32>(m, xd, xz, tt, ft, bn, Bc, b0 == 0, loss_denominator, out_loss, out_grad, ws, lc);
    else rc = fm_run<64, 32>(m, xd, xz, tt, ft, bn, Bc, b0 == 0, loss_denominator, out_loss, out_grad, ws, lc);
    if (rc != ECNF_OK) return rc;
  }
  return ECNF_OK;
}

int ecnf_model_set_fm_chunk(ecnf_model* m, int64_t graphs) {
  if (!m || graphs < 0) { ecnf_set_error("ecnf_model_set_fm_chunk: bad argument"); return ECNF_ERR_INVALID; }
  m->fm_chunk = graphs;
  return ECNF_OK;
}

}  // extern "C"
