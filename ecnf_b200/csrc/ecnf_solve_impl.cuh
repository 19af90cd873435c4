// Engine A: persistent per-trajectory kernel = EGNN vector field (+ exact divergence by fused forward-mode
// tangents) inside an on-device Dopri5 loop.
//
// Replaces, for a whole batch of independent trajectories,
//   cnf.apply                      ecnf/cnf/build_cnf.py:68-93 -> ecnf/nets/egnn.py:131-190, :49-114
//   joint_vector_field (exact)     ecnf/cnf/sample_and_log_prob.py:58-67, :112-121
//   diffeqsolve(Dopri5, PID|const) ecnf/cnf/sample_and_log_prob.py:33-37, :85-89, :140-144   (diffrax, not in tree)
//
// One CTA (256 threads) owns one trajectory at a time, pulled from a global work queue, and runs the entire
// solve on device: particle coordinates, their D x D tangent matrix and all ODE state live in shared memory;
// the wide per-node / per-edge feature rows are processed as [TR x U] row tiles that go through the whole
// phi_e -> {attention, phi_x} chain in shared memory, weights streamed from L2 with cp.async.  A "row" is
// (edge or node, slot) where slot 0 is the primal value and slot 1+k the tangent in input direction k.
//
// Exact divergence (DESIGN.md "tangent rows"): block 0 carries only the 2*dim directions that touch an edge,
// the last block only the dim directions of the receiver (only the Jacobian diagonal is needed), middle
// blocks all D.  phi_e layer 0 is split into two node-level GEMMs plus a rank-1 |v|^2 term.
#pragma once
#include <cstdio>

#include "ecnf_solve_decl.cuh"
#include "ecnf_tile.cuh"

namespace ecnf_solve_detail {

using ecnf_tile::NTHREADS;
using ecnf_tile::WCHUNK;
using ecnf_tile::ColT;
using ecnf_tile::tile_gemm;

enum { KIND_FIRST = 0, KIND_MID = 1, KIND_LAST = 2 };

static __constant__ float c_A[7][6] = {
    {0, 0, 0, 0, 0, 0},
    {(float)(1.0 / 5), 0, 0, 0, 0, 0},
    {(float)(3.0 / 40), (float)(9.0 / 40), 0, 0, 0, 0},
    {(float)(44.0 / 45), (float)(-56.0 / 15), (float)(32.0 / 9), 0, 0, 0},
    {(float)(19372.0 / 6561), (float)(-25360.0 / 2187), (float)(64448.0 / 6561), (float)(-212.0 / 729), 0, 0},
    {(float)(9017.0 / 3168), (float)(-355.0 / 33), (float)(46732.0 / 5247), (float)(49.0 / 176),
     (float)(-5103.0 / 18656), 0},
    {(float)(35.0 / 384), 0, (float)(500.0 / 1113), (float)(125.0 / 192), (float)(-2187.0 / 6784),
     (float)(11.0 / 84)}};
static __constant__ float c_C[7] = {0.f, 0.2f, 0.3f, 0.8f, (float)(8.0 / 9), 1.f, 1.f};
// b - b_hat with diffrax/torchdiffeq's embedded weights (see oracle/ecnf_oracle.py DP_BERR).
static __constant__ float c_BERR[7] = {(float)(35.0 / 384 - 1951.0 / 21600),
                                0.f,
                                (float)(500.0 / 1113 - 22642.0 / 50085),
                                (float)(125.0 / 192 - 451.0 / 720),
                                (float)(-2187.0 / 6784 + 12231.0 / 42400),
                                (float)(11.0 / 84 - 649.0 / 6300),
                                (float)(-1.0 / 60)};
// Dense output: y(t_mid) - y0 = sum_i c_MID[i] k_i, the midpoint weights of the Dopri5 4th-order interpolant as torchdiffeq and
// diffrax carry them.  Recalled, like the b_hat above, not read from diffrax (DESIGN.md 3.1d).
static __constant__ float c_MID[7] = {(float)(6025192743.0 / 30085553152.0 / 2),
                               0.f,
                               (float)(51252292925.0 / 65400821598.0 / 2),
                               (float)(-2691868925.0 / 45128329728.0 / 2),
                               (float)(187940372067.0 / 1594534317056.0 / 2),
                               (float)(-1776094331.0 / 19743644256.0 / 2),
                               (float)(11237099.0 / 235043384.0 / 2)};

template <int U_, int H_>
struct Geo {
  static constexpr int U = U_, H = H_;
  static constexpr int TR = (U_ == 256) ? 64 : 128;  // rows per tile (64 KB of fp32 per tile buffer)
  static constexpr int LD = U_ + 4;                  // padded row stride (floats)
  static constexpr int RT = TR / 16;                 // rows per thread
  static constexpr int GMAX = TR / 3 + 1;            // max groups per tile when tangent rows exist
};

// ------------------------------------------------------------------------------------------------
// shared-memory carve-up (same function on host and device)
// ------------------------------------------------------------------------------------------------
struct SmemLayout {
  int X1, X2, Wb, G, xt, xtacc, dacc, xs, xs0, xacc, mu, rowdot, rowsd, gv, gs1, glen, ginv, ge, tau, cvec,
      ode, red, rowslot, rowgrp, gi, gj, giz, epsv, total_floats;
};

template <int U, int H>
__host__ __device__ inline SmemLayout make_layout(int n, int dim, bool div) {
  using G_ = Geo<U, H>;
  const int D = n * dim, S = D + 1;
  SmemLayout L;
  int o = 0;
  auto take = [&](int nfl) { int r = o; o += (nfl + 3) & ~3; return r; };
  L.X1 = take(G_::TR * G_::LD);
  L.X2 = take(G_::TR * G_::LD);
  L.Wb = take(2 * WCHUNK);
  L.G = take(div ? G_::GMAX * U : 4);
  L.xt = take(div ? D * D : 4);
  L.xtacc = take(div ? D * D : 4);
  L.dacc = take(D);
  L.xs = take(D);
  L.xs0 = take(D);
  L.xacc = take(D);
  L.mu = take(4);
  L.rowdot = take(G_::TR);
  L.rowsd = take(G_::TR);
  L.gv = take(G_::TR * 3);
  L.gs1 = take(G_::TR);
  L.glen = take(G_::TR);
  L.ginv = take(G_::TR);
  L.ge = take(G_::TR);
  L.tau = take(ECNF_MAX_T);
  L.cvec = take(64);
  L.ode = take(11 * S);
  L.red = take(S + 16);
  L.rowslot = take(G_::TR);
  L.rowgrp = take(G_::TR);
  L.gi = take(G_::TR);
  L.gj = take(G_::TR);
  L.giz = take(G_::TR);
  L.epsv = take(D);
  L.total_floats = o;
  return L;
}

// bias + SiLU on primal rows, silu'(z_primal) * z_tangent on tangent rows.  dst may alias the GEMM input.
template <int N, int TR, int LD>
__device__ __forceinline__ void epi_act(float (&acc)[TR / 16][ColT<N>::CT], const float* __restrict__ bias,
                                        float* dst, int nrows, int r, const int* rowgrp, float* G, bool has_tan) {
  constexpr int RT = TR / 16, CT = ColT<N>::CT, NSEG = CT / 4;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, warp = tid >> 5;
  const bool active = (2 * RT * warp < nrows) && (tx * 4 < N);
  const int row0 = 2 * RT * warp + (ty & 1);
  if (active) {
#pragma unroll
    for (int rr = 0; rr < RT; ++rr) {
      const int row = row0 + 2 * rr;
      if (row >= nrows) continue;
      const int g = rowgrp[row];
      if (row != g * r) continue;
#pragma unroll
      for (int sg = 0; sg < NSEG; ++sg) {
        const int col = sg * 64 + tx * 4;
        const float4 b = *reinterpret_cast<const float4*>(bias + col);
        const float bb[4] = {b.x, b.y, b.z, b.w};
        float a[4], gg[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float z = acc[rr][4 * sg + q] + bb[q];
          const float s = ecnf_sigmoid(z);
          a[q] = z * s;
          gg[q] = s * (1.f + z * (1.f - s));
        }
        *reinterpret_cast<float4*>(dst + row * LD + col) = make_float4(a[0], a[1], a[2], a[3]);
        if (has_tan) *reinterpret_cast<float4*>(G + g * N + col) = make_float4(gg[0], gg[1], gg[2], gg[3]);
      }
    }
  }
  if (has_tan) {
    __syncthreads();
    if (active) {
#pragma unroll
      for (int rr = 0; rr < RT; ++rr) {
        const int row = row0 + 2 * rr;
        if (row >= nrows) continue;
        const int g = rowgrp[row];
        if (row == g * r) continue;
#pragma unroll
        for (int sg = 0; sg < NSEG; ++sg) {
          const int col = sg * 64 + tx * 4;
          const float4 gg = *reinterpret_cast<const float4*>(G + g * N + col);
          *reinterpret_cast<float4*>(dst + row * LD + col) =
              make_float4(acc[rr][4 * sg] * gg.x, acc[rr][4 * sg + 1] * gg.y, acc[rr][4 * sg + 2] * gg.z,
                          acc[rr][4 * sg + 3] * gg.w);
        }
      }
    }
  }
  __syncthreads();
}

// dst = acc (+ bias on primal rows) (+ resid tile)
template <int N, int TR, int LD>
__device__ __forceinline__ void epi_linear(float (&acc)[TR / 16][ColT<N>::CT], const float* bias, float* dst,
                                           int nrows, int r, const int* rowgrp, const float* resid) {
  constexpr int RT = TR / 16, CT = ColT<N>::CT, NSEG = CT / 4;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, warp = tid >> 5;
  const bool active = (2 * RT * warp < nrows) && (tx * 4 < N);
  const int row0 = 2 * RT * warp + (ty & 1);
  if (active) {
#pragma unroll
    for (int rr = 0; rr < RT; ++rr) {
      const int row = row0 + 2 * rr;
      if (row >= nrows) continue;
      const bool primal = (row == rowgrp[row] * r);
#pragma unroll
      for (int sg = 0; sg < NSEG; ++sg) {
        const int col = sg * 64 + tx * 4;
        float v[4] = {acc[rr][4 * sg], acc[rr][4 * sg + 1], acc[rr][4 * sg + 2], acc[rr][4 * sg + 3]};
        if (bias != nullptr && primal) {
#pragma unroll
          for (int q = 0; q < 4; ++q) v[q] += bias[col + q];
        }
        if (resid != nullptr) {
          const float4 rv = *reinterpret_cast<const float4*>(resid + row * LD + col);
          v[0] += rv.x; v[1] += rv.y; v[2] += rv.z; v[3] += rv.w;
        }
        *reinterpret_cast<float4*>(dst + row * LD + col) = make_float4(v[0], v[1], v[2], v[3]);
      }
    }
  }
  __syncthreads();
}

__device__ __forceinline__ int dirmap(int kind, int qq, int i, int j, int dim) {
  if (kind == KIND_MID) return qq;
  if (kind == KIND_LAST) return i * dim + qq;
  return (qq < dim) ? i * dim + qq : j * dim + (qq - dim);
}


// ------------------------------------------------------------------------------------------------
template <int U, int H, bool DIV>
struct Engine {
  using G_ = Geo<U, H>;
  static constexpr int TR = G_::TR, LD = G_::LD, RT = G_::RT;
  static constexpr int NT = NTHREADS;
  const EcnfModelDev& m;
  // ntan = tangent directions carried: D (exact trace: the basis), 1 (Hutchinson: the probe eps), 0 (no divergence)
  const bool hutch;
  const int n, dim, D, ntan, ND, E;
  const int tid;
  const float* eps_g;   // Hutchinson probe of the current trajectory (global, D floats)
  float *X1, *X2, *Wb, *G, *xt, *xtacc, *dacc, *xs, *xs0, *xacc, *mu, *rowdot, *rowsd, *gv, *gs1, *glen, *ginv,
      *ge, *tau, *cvec, *ode, *red, *epsv;
  int *rowslot, *rowgrp, *gi, *gj, *giz;
  float *hA, *hB, *Ps, *Pr, *Mg;  // global scratch (this CTA's), NOT read through the non-coherent path

  __device__ Engine(const EcnfModelDev& m_, float* smem, float* scratch, bool hutch_)
      : m(m_), hutch(DIV && hutch_), n(m_.n), dim(m_.dim), D(m_.n * m_.dim),
        ntan(DIV ? (hutch_ ? 1 : m_.n * m_.dim) : 0), ND(1 + ntan), E(m_.n * (m_.n - 1)), tid(threadIdx.x), eps_g(nullptr) {
    const SmemLayout L = make_layout<U, H>(n, dim, DIV);
    X1 = smem + L.X1; X2 = smem + L.X2; Wb = smem + L.Wb; G = smem + L.G; xt = smem + L.xt;
    xtacc = smem + L.xtacc; dacc = smem + L.dacc; xs = smem + L.xs; xs0 = smem + L.xs0; xacc = smem + L.xacc;
    mu = smem + L.mu; rowdot = smem + L.rowdot; rowsd = smem + L.rowsd; gv = smem + L.gv; gs1 = smem + L.gs1;
    glen = smem + L.glen; ginv = smem + L.ginv; ge = smem + L.ge; tau = smem + L.tau; cvec = smem + L.cvec;
    ode = smem + L.ode; red = smem + L.red; epsv = smem + L.epsv;
    rowslot = reinterpret_cast<int*>(smem + L.rowslot); rowgrp = reinterpret_cast<int*>(smem + L.rowgrp);
    gi = reinterpret_cast<int*>(smem + L.gi); gj = reinterpret_cast<int*>(smem + L.gj);
    giz = reinterpret_cast<int*>(smem + L.giz);
    hA = scratch; hB = hA + (size_t)n * ND * H; Ps = hB + (size_t)n * ND * H; Pr = Ps + (size_t)n * ND * U;
    Mg = Pr + (size_t)n * ND * U;
  }

  __device__ __forceinline__ void set_eps(const float* e) { eps_g = e; }
  __device__ __forceinline__ float* ode_ptr() const { return ode; }
  __device__ __forceinline__ float* red_ptr() const { return red; }

  // rowdot[row] = sum_col X[row][col] * vec[col]   (one warp per row)
  __device__ void rowdot_tile(const float* X, const float* __restrict__ vec, int nrows) {
    const int warp = tid >> 5, lane = tid & 31;
    float v[U / 32];
#pragma unroll
    for (int j = 0; j < U / 32; ++j) v[j] = vec[lane + 32 * j];
    for (int row = warp; row < nrows; row += NTHREADS / 32) {
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < U / 32; ++j) s = fmaf(X[row * LD + lane + 32 * j], v[j], s);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) rowdot[row] = s;
    }
    __syncthreads();
  }

  // copy tile rows (width W floats) from smem tile to global rows: dst[(node*ND + slot)*W + col]
  template <int W>
  __device__ void store_node_tile(const float* X, float* dst, int node0, int nrows, int r) {
    for (int idx = tid; idx < nrows * (W / 4); idx += NTHREADS) {
      const int row = idx / (W / 4), c4 = idx % (W / 4);
      const int g = row / r, q = row - g * r;
      *reinterpret_cast<float4*>(dst + ((size_t)(node0 + g) * ND + q) * W + c4 * 4) =
          *reinterpret_cast<const float4*>(X + row * LD + c4 * 4);
    }
  }
  template <int W>
  __device__ void load_node_tile(float* X, const float* src, int node0, int nrows, int r, bool tan_valid) {
    for (int idx = tid; idx < nrows * (W / 4); idx += NTHREADS) {
      const int row = idx / (W / 4), c4 = idx % (W / 4);
      const int g = row / r, q = row - g * r;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (q == 0 || tan_valid) v = *reinterpret_cast<const float4*>(src + ((size_t)(node0 + g) * ND + q) * W + c4 * 4);
      *reinterpret_cast<float4*>(X + row * LD + c4 * 4) = v;
    }
  }
  __device__ void set_rowgrp(int nrows, int r) {
    for (int row = tid; row < nrows; row += NTHREADS) rowgrp[row] = row / r;
  }

  // ---- node phase 1: h_in = [h | tau] Wd + bd ; P_s = h_in We0[0:H] ; P_r = h_in We0[H:2H] + be0 ----
  __device__ void node_pre(int b, bool htan) {
    const EcnfBlockParams& bp = m.blk[b];
    if (tid < H) {
      float a = bp.bd[tid];
      for (int k = 0; k < m.T; ++k) a = fmaf(tau[k], bp.Wd[(H + k) * H + tid], a);
      cvec[tid] = a;
    }
    const int r = htan ? ND : 1;
    const int gpt = TR / r;
    for (int node0 = 0; node0 < n; node0 += gpt) {
      const int nn = min(gpt, n - node0), nrows = nn * r;
      __syncthreads();
      load_node_tile<H>(X1, hA, node0, nrows, r, true);
      set_rowgrp(nrows, r);
      __syncthreads();
      {
        float acc[RT][ColT<H>::CT];
        tile_gemm<H, H, TR, LD, true>(X1, bp.Wd, Wb, acc, nrows);
        epi_linear<H, TR, LD>(acc, cvec, X2, nrows, r, rowgrp, nullptr);
      }
      store_node_tile<H>(X2, hB, node0, nrows, r);
      {
        float acc[RT][ColT<U>::CT];
        tile_gemm<H, U, TR, LD, true>(X2, bp.We[0], Wb, acc, nrows);
        epi_linear<U, TR, LD>(acc, nullptr, X1, nrows, r, rowgrp, nullptr);
        store_node_tile<U>(X1, Ps, node0, nrows, r);
        tile_gemm<H, U, TR, LD, true>(X2, bp.We[0] + (size_t)H * U, Wb, acc, nrows);
        epi_linear<U, TR, LD>(acc, bp.be[0], X1, nrows, r, rowgrp, nullptr);
        store_node_tile<U>(X1, Pr, node0, nrows, r);
      }
    }
    __syncthreads();
  }

  // ---- node phase 2: h <- phi_h([M | h_in]) + h_in ----
  __device__ void node_post(int b, bool htan) {
    const EcnfBlockParams& bp = m.blk[b];
    const int r = ND;  // aggregated-message tangents are dense in every non-last block
    const int gpt = TR / r;
    for (int node0 = 0; node0 < n; node0 += gpt) {
      const int nn = min(gpt, n - node0), nrows = nn * r;
      __syncthreads();
      load_node_tile<U>(X1, Mg, node0, nrows, r, true);
      load_node_tile<H>(X2, hB, node0, nrows, r, htan);
      set_rowgrp(nrows, r);
      __syncthreads();
      {
        float acc[RT][ColT<U>::CT];
        tile_gemm<U, U, TR, LD, true>(X1, bp.Wh[0], Wb, acc, nrows);
        tile_gemm<H, U, TR, LD, false>(X2, bp.Wh[0] + (size_t)U * U, Wb, acc, nrows);
        epi_act<U, TR, LD>(acc, bp.bh[0], X1, nrows, r, rowgrp, G, DIV);
        for (int l = 1; l < m.L; ++l) {
          tile_gemm<U, U, TR, LD, true>(X1, bp.Wh[l], Wb, acc, nrows);
          epi_act<U, TR, LD>(acc, bp.bh[l], X1, nrows, r, rowgrp, G, DIV);
        }
      }
      {
        float acc[RT][ColT<H>::CT];
        tile_gemm<U, H, TR, LD, true>(X1, bp.Wh[m.L], Wb, acc, nrows);
        epi_linear<H, TR, LD>(acc, bp.bh[m.L], X1, nrows, r, rowgrp, X2);
      }
      store_node_tile<H>(X1, hA, node0, nrows, r);
    }
    __syncthreads();
  }

  // ---- edge phase of block b ----
  // lastb: last block (no messages / phi_h).  kind: tangent-row structure; with a Hutchinson probe every block is "MID"
  // (one dense direction), also the last one, whose full coordinate tangent is then needed.
  __device__ void edge_phase(int b, int kind, bool htan, bool lastb) {
    const EcnfBlockParams& bp = m.blk[b];
    const int nact = !DIV ? 0 : (kind == KIND_MID ? ntan : kind == KIND_LAST ? dim : 2 * dim);
    const int r = 1 + nact;
    const int gpt = DIV ? min(TR / r, n - 1) : TR;
    const float inv_sqrt_nb = rsqrtf((float)(n - 1));
    const float* wd = bp.We[0] + (size_t)2 * H * U;
    const float bpv = bp.bp[0];
    const float bav = bp.ba[0];
    // zero the accumulators of this block
    for (int i = tid; i < D; i += NTHREADS) { xacc[i] = 0.f; dacc[i] = 0.f; }
    if (DIV && kind != KIND_LAST)
      for (int i = tid; i < D * ntan; i += NTHREADS) xtacc[i] = 0.f;
    if (!lastb)
      for (int i = tid; i < n * ND * U; i += NTHREADS) Mg[i] = 0.f;
    __syncthreads();

    int e0 = 0;
    while (e0 < E) {
      int ng;
      if (DIV) {
        const int i = e0 / (n - 1);
        ng = min(gpt, (i + 1) * (n - 1) - e0);
      } else {
        ng = min(TR, E - e0);
      }
      const int nrows = ng * r;
      // -- A: per-edge geometry
      if (tid < ng) {
        const int e = e0 + tid, i = e / (n - 1), jj = e - i * (n - 1);
        int j = i + 1 + jj; if (j >= n) j -= n;
        float s = 0.f;
        for (int c = 0; c < dim; ++c) {
          const float v = xs[i * dim + c] - xs[j * dim + c];
          gv[tid * 3 + c] = v;
          s = fmaf(v, v, s);
        }
        const int isz = (s == 0.f);
        const float s1 = isz ? 1.f : s;
        const float len = sqrtf(s1);
        gi[tid] = i; gj[tid] = j; giz[tid] = isz; gs1[tid] = s1; glen[tid] = len; ginv[tid] = 1.f / (m.C + len);
      }
      __syncthreads();
      // -- B: per-row metadata (slot, d|v|^2)
      for (int row = tid; row < nrows; row += NTHREADS) {
        const int g = row / r, q = row - g * r;
        rowgrp[row] = g;
        if (q == 0) {
          rowslot[row] = 0;
          rowsd[row] = gs1[g];
        } else {
          const int i = gi[g], j = gj[g];
          const int k = dirmap(kind, q - 1, i, j, dim);
          float sd = 0.f;
          for (int c = 0; c < dim; ++c)
            sd = fmaf(gv[g * 3 + c], xt[(i * dim + c) * ntan + k] - xt[(j * dim + c) * ntan + k], sd);
          rowslot[row] = 1 + k;
          rowsd[row] = giz[g] ? 0.f : 2.f * sd;
        }
      }
      __syncthreads();
      // -- C: phi_e layer 0 by gather: z0 = P_s[j] + P_r[i] + (|v|^2 or its tangent) * w_d ; then SiLU / tangent
      {
        const int col = tid % U;
        const float wdc = wd[col];
        for (int g = tid / U; g < ng; g += NTHREADS / U) {
          const int row = g * r;
          const float z = Ps[((size_t)gj[g] * ND) * U + col] + Pr[((size_t)gi[g] * ND) * U + col] + rowsd[row] * wdc;
          const float s = ecnf_sigmoid(z);
          X1[row * LD + col] = z * s;
          if (DIV) G[g * U + col] = s * (1.f + z * (1.f - s));
        }
        if (DIV) {
          __syncthreads();
          for (int row = tid / U; row < nrows; row += NTHREADS / U) {
            const int g = rowgrp[row];
            if (row == g * r) continue;
            float z = rowsd[row] * wdc;
            if (htan) {
              const int slot = rowslot[row];
              z += Ps[((size_t)gj[g] * ND + slot) * U + col] + Pr[((size_t)gi[g] * ND + slot) * U + col];
            }
            X1[row * LD + col] = z * G[g * U + col];
          }
        }
      }
      __syncthreads();
      {
        float acc[RT][ColT<U>::CT];
        for (int l = 1; l < m.L; ++l) {
          tile_gemm<U, U, TR, LD, true>(X1, bp.We[l], Wb, acc, nrows);
          epi_act<U, TR, LD>(acc, bp.be[l], X1, nrows, r, rowgrp, G, DIV);
        }
        if (!lastb) {
          // attention gate + message aggregation (egnn.py:99-104)
          rowdot_tile(X1, bp.wa, nrows);
          if (tid < ng) ge[tid] = ecnf_sigmoid(rowdot[tid * r] + bav);
          __syncthreads();
          for (int idx = tid; idx < nrows * U; idx += NTHREADS) {
            const int row = idx / U, col = idx - row * U;
            const int g = rowgrp[row];
            const float e = ge[g];
            float v = X1[row * LD + col] * e;
            if (row != g * r) v = fmaf(X1[g * r * LD + col], e * (1.f - e) * rowdot[row], v);
            X2[row * LD + col] = v;
          }
          __syncthreads();
          if (DIV) {
            const int i = gi[0];
            for (int idx = tid; idx < r * U; idx += NTHREADS) {
              const int q = idx / U, col = idx - q * U;
              const bool shared_q = (q == 0) || kind == KIND_MID || (q - 1 < dim);
              if (shared_q) {
                const int slot = (q == 0) ? 0 : 1 + dirmap(kind, q - 1, i, 0, dim);
                float s = 0.f;
                for (int g = 0; g < ng; ++g) s += X2[(g * r + q) * LD + col];
                Mg[((size_t)i * ND + slot) * U + col] += s * inv_sqrt_nb;
              } else {
                for (int g = 0; g < ng; ++g) {
                  const int slot = 1 + gj[g] * dim + (q - 1 - dim);
                  Mg[((size_t)i * ND + slot) * U + col] += X2[(g * r + q) * LD + col] * inv_sqrt_nb;
                }
              }
            }
          } else {
            const int i_first = e0 / (n - 1), i_last = (e0 + ng - 1) / (n - 1);
            for (int idx = tid; idx < (i_last - i_first + 1) * U; idx += NTHREADS) {
              const int ri = idx / U, col = idx - ri * U, i = i_first + ri;
              const int ga = max(e0, i * (n - 1)) - e0, gb = min(e0 + ng, (i + 1) * (n - 1)) - e0;
              float s = 0.f;
              for (int g = ga; g < gb; ++g) s += X2[g * LD + col];
              Mg[(size_t)i * U + col] += s * inv_sqrt_nb;
            }
          }
          // no barrier needed here: the phi_x GEMM below starts with barriers before X1 is overwritten,
          // and X2 / Mg are not touched again until the next tile's barriers.
        }
        // phi_x torso + head (egnn.py:82-85)
        for (int l = 0; l < m.L; ++l) {
          tile_gemm<U, U, TR, LD, true>(X1, bp.Wx[l], Wb, acc, nrows);
          epi_act<U, TR, LD>(acc, bp.bx[l], X1, nrows, r, rowgrp, G, DIV);
        }
      }
      rowdot_tile(X1, bp.wp, nrows);
      // coordinate update (egnn.py:87-95): shift_i += p * v / (C + len)
      {
        const int i_first = e0 / (n - 1), i_last = (e0 + ng - 1) / (n - 1);
        const int nprim = (i_last - i_first + 1) * dim;
        const int nwork_tan = DIV ? (r - 1) * dim : 0;
        for (int idx = tid; idx < nprim + nwork_tan; idx += NTHREADS) {
          if (idx < nprim) {
            const int ri = idx / dim, c = idx - ri * dim, i = i_first + ri;
            const int ga = max(e0, i * (n - 1)) - e0, gb = min(e0 + ng, (i + 1) * (n - 1)) - e0;
            float s = 0.f;
            for (int g = ga; g < gb; ++g) s = fmaf((rowdot[g * r] + bpv) * gv[g * 3 + c], ginv[g], s);
            xacc[i * dim + c] += s;
          } else {
            const int t2 = idx - nprim;
            const int q = 1 + t2 / dim, c = t2 % dim;
            const int i = gi[0];
            for (int g = 0; g < ng; ++g) {
              const int j = gj[g];
              const int k = dirmap(kind, q - 1, i, j, dim);
              if (kind == KIND_LAST && k != i * dim + c) continue;
              const float pg = rowdot[g * r] + bpv, pd = rowdot[g * r + q];
              const float vc = gv[g * 3 + c], inv = ginv[g];
              const float vd = xt[(i * dim + c) * ntan + k] - xt[(j * dim + c) * ntan + k];
              const float ld = giz[g] ? 0.f : rowsd[g * r + q] / (2.f * glen[g]);
              const float cd = (pd * vc + pg * vd) * inv - pg * vc * ld * inv * inv;
              if (kind == KIND_LAST) dacc[i * dim + c] += cd;
              else xtacc[(i * dim + c) * ntan + k] += cd;
            }
          }
        }
      }
      __syncthreads();
      e0 += ng;
    }
  }

  // ---- one evaluation of the vector field at time t for the positions in xin (smem, D floats) ----
  // fout[0..D) = f, fout[D] = divergence (DIV only)
  __device__ void eval(float t, const float* xin, const int32_t* feat, float* fout) {
    // centre, tangent init, embeddings, time embedding
    if (tid < dim) {
      float s = 0.f;
      for (int i = 0; i < n; ++i) s += xin[i * dim + tid];
      mu[tid] = s / (float)n;
    }
    if (tid >= 32 && tid < 32 + m.T / 2) {
      const int k = tid - 32;
      const float arg = (t * 1000.f) * m.freqs[k];
      tau[k] = sinf(arg);
      tau[k + m.T / 2] = cosf(arg);
    }
    __syncthreads();
    for (int i = tid; i < D; i += NTHREADS) {
      const float v = xin[i] - mu[i % dim];
      xs[i] = v;
      xs0[i] = v;
    }
    if (DIV && !hutch) {
      const float invn = 1.f / (float)n;
      for (int idx = tid; idx < D * D; idx += NTHREADS) {
        const int a = idx / D, k = idx - a * D;
        const int ia = a / dim, ca = a - ia * dim, ik = k / dim, ck = k - ik * dim;
        xt[idx] = (ca == ck) ? ((ia == ik ? 1.f : 0.f) - invn) : 0.f;
      }
    }
    if (hutch) {
      // tangent of the centred positions in the probe direction: eps - mean_nodes(eps)
      for (int i = tid; i < D; i += NTHREADS) epsv[i] = eps_g[i];
      __syncthreads();
      for (int i = tid; i < D; i += NTHREADS) {
        float mean = 0.f;
        for (int node = 0; node < n; ++node) mean += epsv[node * dim + i % dim];
        xt[i] = epsv[i] - mean / (float)n;
      }
    }
    for (int idx = tid; idx < n * H; idx += NTHREADS) {
      const int node = idx / H, col = idx - node * H;
      int f = feat[node];
      f = max(0, min(m.nfeat - 1, f));
      hA[(size_t)node * ND * H + col] = m.embed[f * H + col];
    }
    __syncthreads();
    for (int b = 0; b < m.nblocks; ++b) {
      const bool last = (b == m.nblocks - 1);
      const int kind = hutch ? KIND_MID : (last ? KIND_LAST : (b == 0 ? KIND_FIRST : KIND_MID));
      const bool htan = DIV && b > 0;
      node_pre(b, htan);
      edge_phase(b, kind, htan, last);
      if (!last) node_post(b, htan);
      const float invnb = 1.f / (float)(n - 1);
      for (int i = tid; i < D; i += NTHREADS) xs[i] += xacc[i] * invnb;
      if (DIV && (!last || hutch))
        for (int i = tid; i < D * ntan; i += NTHREADS) xt[i] += xtacc[i] * invnb;
      __syncthreads();
    }
    const float fs = m.final_scaling[0];
    for (int i = tid; i < D; i += NTHREADS) fout[i] = (xs[i] - xs0[i] - mu[i % dim]) * fs;
    if (DIV && tid == 0) {
      float s = 0.f;
      if (hutch) {
        // eps . (J eps): the output tangent is fs (x_L-dot - x0-dot - mean(eps)) = fs (xt - eps)   (egnn.py:183-188)
        for (int d = 0; d < D; ++d) s = fmaf(epsv[d], xt[d] - epsv[d], s);
        fout[D] = fs * s;
      } else {
        const float invnb = 1.f / (float)(n - 1);
        for (int d = 0; d < D; ++d) s += xt[d * D + d] + dacc[d] * invnb;
        fout[D] = fs * (s - (float)D);
      }
    }
    __syncthreads();
  }
};

__device__ __forceinline__ float clip_to_end(float tprev, float tnext, float T1, bool keep) {
  if (tnext > T1 - 1e-6f) return keep ? T1 : tprev + 0.5f * (T1 - tprev);
  return tnext;
}

// The ODE driver (diffrax.diffeqsolve restated), generic over the engine that evaluates the vector field.
// Written as a state machine around ONE call site of eng.eval so that the (large) evaluation code is inlined exactly
// once and the engine's state stays in registers.
// SAVE: also write the path at the caller's times a.ts (diffrax SaveAt(ts)) from the Dopri5 dense output of each accepted
// step.  A template parameter, so that the kernels without it keep their registers and spills.
template <class Eng, bool DIV, bool SAVE>
__device__ __forceinline__ void solve_body(const KernelArgs& a, Eng& eng, long long& s_traj, float* s_ctl) {
  const int tid = threadIdx.x;
  const int D = eng.D, S = DIV ? D + 1 : D;
  float* y = eng.ode_ptr();    // [S]
  float* ys = y + S;           // [S] stage input
  float* f0 = ys + S;          // [S] FSAL derivative (direction applied)
  float* fo = f0 + S;          // [S] eval output
  float* kk = fo + S;          // [7][S]
  float* red = eng.red_ptr();
  const ecnf_solve_ctrl& c = a.ctrl;
  const bool vf_mode = (a.mode == ECNF_MODE_VF || a.mode == ECNF_MODE_VF_DIV);
  const bool reverse = (a.mode == ECNF_MODE_LOGPROB);
  const float dir = reverse ? -1.f : 1.f;
  const float T0 = reverse ? -1.f : 0.f, T1 = reverse ? 0.f : 1.f;  // internal (direction-multiplied) times
  enum { PH_VF = 0, PH_F0 = 1, PH_F1 = 2, PH_STAGE = 3 };

  auto rms_of_red = [&]() -> float {  // sqrt(mean(red[0..S)^2)), result broadcast to all threads
    __syncthreads();
    if (tid == 0) {
      float s = 0.f;
      for (int i = 0; i < S; ++i) s = fmaf(red[i], red[i], s);
      s_ctl[0] = sqrtf(s / (float)S);
    }
    __syncthreads();
    const float r = s_ctl[0];
    __syncthreads();
    return r;
  };
  // log p0 of the D positions in v (zero_com_base.py:44-47,64-84 + ildj), computed by thread 0, broadcast
  auto base_logp = [&](const float* v) -> float {
    __syncthreads();
    if (tid == 0) {
      float s = 0.f;
      for (int cdim = 0; cdim < eng.dim; ++cdim) {
        float mean = 0.f;
        for (int i = 0; i < eng.n; ++i) mean += v[i * eng.dim + cdim] / a.m.base_scale;
        mean /= (float)eng.n;
        for (int i = 0; i < eng.n; ++i) {
          const float z = v[i * eng.dim + cdim] / a.m.base_scale - mean;
          s = fmaf(z, z, s);
        }
      }
      const float dof = (float)((eng.n - 1) * eng.dim);
      s_ctl[1] = -0.5f * s - 0.5f * dof * 1.8378770664093453f - dof * logf(a.m.base_scale);
    }
    __syncthreads();
    const float r = s_ctl[1];
    __syncthreads();
    return r;
  };

  for (;;) {
    if (tid == 0) s_traj = (long long)atomicAdd(a.counter, 1u);
    __syncthreads();
    const long long b = s_traj;
    __syncthreads();
    if (b >= a.B) break;
    const int32_t* feat = a.feat + b * eng.n;
    const float* xin = a.x_init + b * D;
    eng.set_eps(a.eps ? a.eps + b * D : nullptr);
    // save row k, component i < S: positions to out_traj [B, n_save, D], the divergence integral to out_traj_delta [B, n_save]
    auto put = [&](int k, int i, float v) {
      if (i < D) a.out_traj[(b * a.n_save + k) * D + i] = v;
      else a.out_traj_delta[b * a.n_save + k] = v;
    };
    int next_save = 0;   // first save time not yet written

    int phase, stage = 0, n_steps = 0, n_acc = 0, n_evals = 0, status = 0;
    float tprev = T0, tnext = T0, dt = 0.f, h0 = 0.f, d1 = 0.f, t_eval, lp0_start = 0.f;
    bool at_dtmin = false;
    const float* ein;
    if (vf_mode) {
      for (int i = tid; i < D; i += Eng::NT) ys[i] = xin[i];
      phase = PH_VF;
      t_eval = a.t_in[b];
      ein = ys;
    } else {
      for (int i = tid; i < S; i += Eng::NT) y[i] = (i < D) ? xin[i] : 0.f;
      phase = PH_F0;
      t_eval = dir * T0;
      ein = y;
    }
    __syncthreads();
    if constexpr (SAVE) {   // a save time at the start time: the initial state, divergence integral 0
      for (; next_save < a.n_save && a.ts[next_save] <= T0; ++next_save)
        for (int i = tid; i < S; i += Eng::NT) put(next_save, i, y[i]);
    }
    if (DIV && !vf_mode && !reverse) lp0_start = base_logp(y);   // log p0(x0), sample_and_log_prob.py:147

    bool running = true;
    while (running) {
      eng.eval(t_eval, ein, feat, fo);      // fo[0..D) = f, fo[D] = div f  -- the single evaluation site
      ++n_evals;
      bool begin_step = false;
      if (phase == PH_VF) {
        for (int i = tid; i < D; i += Eng::NT) a.out_x[b * D + i] = fo[i];
        if (DIV && tid == 0) a.out_logs[b] = fo[D];
        running = false;
      } else if (phase == PH_F0) {
        // F(tau, y) = dir * f(dir * tau, y); FSAL initialisation
        for (int i = tid; i < S; i += Eng::NT) f0[i] = dir * fo[i];
        __syncthreads();
        if (c.fixed) {
          tnext = clip_to_end(tprev, tprev + fabsf(c.step_size), T1, true);
          begin_step = true;
        } else {
          // Hairer-Wanner initial step (diffrax _select_initial_step)
          for (int i = tid; i < S; i += Eng::NT) red[i] = y[i] / (c.atol + fabsf(y[i]) * c.rtol);
          const float d0 = rms_of_red();
          for (int i = tid; i < S; i += Eng::NT) red[i] = f0[i] / (c.atol + fabsf(y[i]) * c.rtol);
          d1 = rms_of_red();
          const bool cond = (d0 < 1e-5f) || (d1 < 1e-5f);
          h0 = cond ? 1e-6f : 0.01f * d0 / d1;
          for (int i = tid; i < S; i += Eng::NT) ys[i] = y[i] + h0 * f0[i];
          __syncthreads();
          t_eval = dir * (tprev + h0);
          ein = ys;
          phase = PH_F1;
        }
      } else if (phase == PH_F1) {
        for (int i = tid; i < S; i += Eng::NT) red[i] = (dir * fo[i] - f0[i]) / (c.atol + fabsf(y[i]) * c.rtol);
        const float d2 = rms_of_red() / h0;
        const float md = fmaxf(d1, d2);
        const float h1 = (md <= 1e-15f) ? fmaxf(1e-6f, h0 * 1e-3f) : powf(0.01f / md, 1.f / c.error_order);
        const float dt0 = fmaxf(fminf(100.f * h0, h1), c.dtmin);
        tnext = clip_to_end(tprev, tprev + dt0, T1, true);
        begin_step = true;
      } else {  // PH_STAGE: stage `stage` (1..6) of the current step has just been evaluated at ys
        for (int i = tid; i < S; i += Eng::NT) kk[stage * S + i] = (dir * fo[i]) * dt;
        __syncthreads();
        if (stage < 6) {
          ++stage;
        } else {
          // ys holds the 5th-order solution y1; dir * fo = F(t + dt, y1) is next step's first stage (FSAL)
          bool keep = true;
          float new_prev, new_next;
          if (c.fixed) {
            new_prev = tnext;
            new_next = tnext + dt;
          } else {
            for (int i = tid; i < S; i += Eng::NT) {
              float e = 0.f;
              for (int j = 0; j < 7; ++j) {
                const float bj = c_BERR[j];
                if (bj != 0.f) e = e + bj * kk[j * S + i];
              }
              red[i] = (c.err_scale * e) / (c.atol + fmaxf(fabsf(y[i]), fabsf(ys[i])) * c.rtol);
            }
            const float err = rms_of_red();
            keep = (err < 1.f) || at_dtmin;
            const float inv = (err == 0.f) ? INFINITY : 1.f / err;
            float factor = c.safety * powf(inv, 1.f / c.error_order);
            const float fmin_ = keep ? 1.f : c.factormin;
            factor = fminf(fmaxf(factor, fmin_), c.factormax);
            float ndt = dt * factor;
            at_dtmin = ndt <= c.dtmin;
            ndt = fmaxf(ndt, c.dtmin);
            new_prev = keep ? tnext : tprev;
            new_next = new_prev + ndt;
          }
          new_prev = fminf(new_prev, T1);
          new_next = clip_to_end(new_prev, new_next, T1, keep);
          if constexpr (SAVE) {
            // every pending save time in (tprev, tnext] of this accepted step, from y0 = y, y1 = ys and k_0..k_6 (k_6 = dt F(tnext,
            // y1), the FSAL stage): the Dopri5 4th-order interpolant (torchdiffeq _interp_fit), y1 itself at tnext.  Each thread
            // reads the components of y it overwrites below, so no barrier is needed in between.
            for (; keep && next_save < a.n_save && a.ts[next_save] <= tnext; ++next_save) {
              const float tau_s = a.ts[next_save];
              const bool at_end = !(tau_s < tnext);
              const float sx = (tau_s - tprev) / dt;
              for (int i = tid; i < S; i += Eng::NT) {
                const float y0 = y[i], y1 = ys[i];
                float v = y1;
                if (!at_end) {
                  const float k0 = kk[i], k6 = kk[6 * S + i];
                  float ym = y0;
                  for (int j = 0; j < 7; ++j) {
                    const float cj = c_MID[j];
                    if (cj != 0.f) ym = ym + cj * kk[j * S + i];
                  }
                  const float pa = 2.f * (k6 - k0) - 8.f * (y1 + y0) + 16.f * ym;
                  const float pb = 5.f * k0 - 3.f * k6 + 18.f * y0 + 14.f * y1 - 32.f * ym;
                  const float pc = k6 - 4.f * k0 - 11.f * y0 - 5.f * y1 + 16.f * ym;
                  v = (((pa * sx + pb) * sx + pc) * sx + k0) * sx + y0;
                }
                put(next_save, i, v);
              }
            }
          }
          if (keep) {
            for (int i = tid; i < S; i += Eng::NT) { y[i] = ys[i]; f0[i] = dir * fo[i]; }
            ++n_acc;
          }
          __syncthreads();
          tprev = new_prev;
          tnext = new_next;
          ++n_steps;
          if (!(tprev < T1)) running = false;
          else if (n_steps >= c.max_steps) { status = 1; running = false; }
          else begin_step = true;
        }
      }
      if (begin_step) {
        dt = tnext - tprev;
        for (int i = tid; i < S; i += Eng::NT) kk[i] = f0[i] * dt;
        __syncthreads();
        stage = 1;
        phase = PH_STAGE;
        if (c.max_steps <= 0) { status = 1; running = false; }
      }
      if (running && phase == PH_STAGE) {
        // stage input: ys = y + sum_j a[stage][j] k_j ; time tprev + c[stage] dt
        for (int i = tid; i < S; i += Eng::NT) {
          float v = y[i];
          for (int j = 0; j < stage; ++j) {
            const float aj = c_A[stage][j];
            if (aj != 0.f) v = v + aj * kk[j * S + i];
          }
          ys[i] = v;
        }
        __syncthreads();
        t_eval = dir * (tprev + c_C[stage] * dt);
        ein = ys;
      }
    }
    if (vf_mode) { __syncthreads(); continue; }
    if constexpr (SAVE) {   // stopped on max_steps: NaN in the rows never reached
      const int left = a.n_save - next_save;
      for (int idx = tid; idx < left * S; idx += Eng::NT) put(next_save + idx / S, idx % S, __int_as_float(0x7fffffff));
    }

    for (int i = tid; i < D; i += Eng::NT) a.out_x[b * D + i] = y[i];
    float lpb_end = 0.f;
    if (DIV && reverse) lpb_end = base_logp(y);
    if (tid == 0) {
      if (a.out_stats) {
        a.out_stats[b * 4 + 0] = n_steps; a.out_stats[b * 4 + 1] = n_acc;
        a.out_stats[b * 4 + 2] = n_evals; a.out_stats[b * 4 + 3] = status;
      }
      if (DIV && a.out_logs) {
        const float delta = y[D];
        if (!reverse) {
          a.out_logs[b * 3 + 0] = lp0_start - delta;
          a.out_logs[b * 3 + 1] = lp0_start;
          a.out_logs[b * 3 + 2] = delta;
        } else {
          a.out_logs[b * 3 + 0] = lpb_end + delta;
          a.out_logs[b * 3 + 1] = lpb_end;
          a.out_logs[b * 3 + 2] = delta;
        }
      }
    }
    __syncthreads();
  }
}

template <int U, int H, bool DIV, bool SAVE>
__global__ void __launch_bounds__(NTHREADS, 1) ecnf_solve_kernel(const __grid_constant__ KernelArgs a) {
  extern __shared__ __align__(16) float smem[];
  __shared__ long long s_traj;
  __shared__ float s_ctl[8];
  Engine<U, H, DIV> eng(a.m, smem, a.scratch + (size_t)blockIdx.x * a.scratch_stride, a.eps != nullptr);
  solve_body<Engine<U, H, DIV>, DIV, SAVE>(a, eng, s_traj, s_ctl);
}

template <int U, int H, bool DIV>
int simt_check(const ecnf_model* mdl) {
  const SmemLayout L = make_layout<U, H>(mdl->cfg.n_frames, mdl->cfg.dim, DIV);
  const size_t smem = (size_t)L.total_floats * sizeof(float);
  if (smem > 227 * 1024) {
    ecnf_set_error("shared memory need %zu B exceeds 227 KB (n_frames=%d dim=%d U=%d)", smem, mdl->cfg.n_frames,
                   mdl->cfg.dim, U);
    return ECNF_ERR_UNSUPPORTED;
  }
  if (DIV && 1 + mdl->cfg.n_frames * mdl->cfg.dim > Geo<U, H>::TR) {
    ecnf_set_error("1 + n_frames*dim = %d tangent slots exceed the %d-row tile of U=%d", 1 + mdl->cfg.n_frames * mdl->cfg.dim,
                   Geo<U, H>::TR, U);
    return ECNF_ERR_UNSUPPORTED;
  }
  return ECNF_OK;
}

template <int U, int H, bool DIV, bool SAVE>
int launch_t(const ecnf_model* mdl, KernelArgs& a, int grid, cudaStream_t st) {
  const int rc = simt_check<U, H, DIV>(mdl);
  if (rc != ECNF_OK) return rc;
  const size_t smem = (size_t)make_layout<U, H>(mdl->cfg.n_frames, mdl->cfg.dim, DIV).total_floats * sizeof(float);
  auto kern = ecnf_solve_kernel<U, H, DIV, SAVE>;
  ECNF_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, NTHREADS, smem, st>>>(a);
  ECNF_CHECK_CUDA(cudaGetLastError());
  return ECNF_OK;
}


}  // namespace ecnf_solve_detail
