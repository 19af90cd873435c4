// Engine B on the tensor cores: the GEMMs over the edge rows of the flow-matching step, M = B*n*(n-1) rows (175 k for
// QM9 at batch 512), K = N = mlp_units = 128 or 256, as tcgen05.mma with the same 3-pass bf16 split as engine A
// (hi*hi + lo*hi + hi*lo, fp32 accumulate in TMEM, ~4e-6 relative error):
//
//   * gemm_rows_tcT_kernel: C[M, N] = epilogue( op(A)[M, K] x W[K, N] ), the forward Dense layers and, with the
//     pre-transposed weights, the backward-data GEMMs dA = dZ W^T; epilogue + bias, + residual, + add, x silu'(z);
//   * dw_tc_kernel: dW[K, N] += op(A)[M, K]^T dZ[M, N], the weight gradients, with the bias gradient (the column sums of
//     dZ) accumulated on the way.
//
// The launchers in ecnf_train.cu send a GEMM here only for these shapes; everything else runs on their fp32 SIMT kernels.
#pragma once
#include "ecnf_tc.cuh"

namespace ecnf_train_tc {

using namespace ecnf_tc;

// One row GEMM  C[M, N] = epilogue( op(A)[M, K] W[K, N] (+ A2[M, K2] W2[K2, N]) ), for the SIMT kernel of ecnf_train.cu
// and for gemm_rows_tcT_kernel, which supports neither A2 nor rowvec (the caller keeps such GEMMs on the SIMT kernel).
struct GemmArgs {
  const float* A;
  const float* A2;
  const float* W;
  const float* W2;
  const float* bias;    // [N]
  const float* rowvec;  // [M / rows_per_vec, N]
  int rows_per_vec;
  const float* resid;   // [M,N], added
  const float* add;     // [M,N], added before the multiplication
  const float* mulz;    // [M,N], multiply by silu'(mulz)
  float* C;
  int M;
  int a_op;  // 1: silu on A while loading
};

// ex2 / rcp based sigmoid (~1e-6 relative, well inside the 3-pass GEMM error): these elementwise ops run on 45 M elements
// per layer and would otherwise dominate the kernels
__device__ __forceinline__ float sigm(float z) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(z * -1.4426950408889634f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.f + e));      // e = inf -> 0, e = 0 -> 1
  return r;
}
__device__ __forceinline__ float silu(float z) { return z * sigm(z); }
__device__ __forceinline__ float dsilu(float z) {
  const float s = sigm(z);
  return s * (1.f + z * (1.f - s));
}

// =====================================================================================================================
// C = epilogue( op(A) W ), transposed and warp-specialised:
//
//     C^T[n (TMEM lane), m (column)] = W^T[n][k] (A operand, TENSOR MEMORY) x op(A)^T[k][m] (B operand, shared memory)
//
//   * the 128 output features of this CTA's column half are the TMEM lanes, so a warp of epilogue threads reads /
//     writes 32 consecutive floats of one row of C, z, add ... : every global access of the epilogue is a coalesced
//     128-byte line and the bias is a per-thread constant -- no shared-memory staging of C;
//   * the B operand is "MN-major" (8 rows of one k = one 16-byte vector, as in engine A): a producer thread loads the
//     same k of 8 consecutive rows (a warp load = 128 contiguous bytes of a row), applies op, splits to bf16 (hi, lo)
//     and stores 16 bytes; a warp stores 512 contiguous bytes -- no shared-memory staging of A either;
//   * W^T (hi | lo) is written to tensor memory once per CTA; the MMA reads only B from shared memory;
//   * warps 0-7: epilogue, warps 8-23: producers (global -> registers one chunk ahead -> ring of 64-k chunks),
//     warp 24: MMA issue; hand-over by mbarriers only (full / empty per ring slot, full / empty per accumulator), so the
//     loads, the conversion, the MMAs and the epilogue of consecutive tiles overlap freely.
// =====================================================================================================================
constexpr int T_NT = 800;       // warps 0-7: epilogue, 8-23: producers, 24: MMA issue
constexpr int T_KC = 64;                        // k per ring slot
constexpr int T_IMG = 128 * T_KC * 2;           // one (hi or lo) image of a chunk: [16 row groups][64 k][8 rows] bf16
constexpr int T_SLOT = 2 * T_IMG;
constexpr int T_NS = 6;                         // ring slots (192 KB)
constexpr uint32_t T_LBO = 128, T_SBO = T_KC * 16;
constexpr uint32_t T_WCOL = 256;                // W^T operand: TMEM columns [256, 256 + K); accumulators [0, 128), [128, 256)

// 32 consecutive rows of one output column: C = ((acc + bias) + resid + add) * silu'(z); the pointers advance by one row
// (N floats) per step, i.e. by compile-time immediates.  RS / AD / MZ say which operands exist (checked once, uniformly,
// by the caller), so the loads of a batch are unconditional and issued back to back before the first use.
template <int N, bool RS, bool AD, bool MZ, bool FULL>
__device__ __forceinline__ void epi_rows(const GemmArgs& g, const uint32_t (&x)[32], size_t o0, float bias, int nrows) {
  const float* rsp = g.resid + o0;
  const float* adp = g.add + o0;
  const float* mzp = g.mulz + o0;
  float* cp = g.C + o0;
  constexpr int BT = (RS || AD) ? 8 : 16;      // loads in flight per operand
#pragma unroll
  for (int j0 = 0; j0 < 32; j0 += BT) {
    float ad[BT], rs[BT], mz[BT];
#pragma unroll
    for (int j = 0; j < BT; ++j) {
      const bool ok = FULL || j0 + j < nrows;
      if (RS) rs[j] = ok ? rsp[(j0 + j) * N] : 0.f;
      if (AD) ad[j] = ok ? adp[(j0 + j) * N] : 0.f;
      if (MZ) mz[j] = ok ? mzp[(j0 + j) * N] : 0.f;
    }
#pragma unroll
    for (int j = 0; j < BT; ++j) {
      float v = __uint_as_float(x[j0 + j]) + bias;
      if (RS) v += rs[j];
      if (AD) v += ad[j];
      if (MZ) v *= dsilu(mz[j]);
      if (FULL || j0 + j < nrows) cp[(j0 + j) * N] = v;
    }
  }
}
template <int N, bool RS, bool AD, bool MZ>
__device__ __forceinline__ void epi_rows_any(const GemmArgs& g, const uint32_t (&x)[32], size_t o0, float bias, int nrows) {
  if (nrows >= 32) epi_rows<N, RS, AD, MZ, true>(g, x, o0, bias, 32);
  else epi_rows<N, RS, AD, MZ, false>(g, x, o0, bias, nrows);
}

template <int K, int N>
__global__ void __launch_bounds__(T_NT, 1) gemm_rows_tcT_kernel(const __grid_constant__ GemmArgs g) {
  static_assert((K == 128 || K == 256) && (N == 128 || N == 256), "shapes");
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ uint32_t tmem_slot;
  __shared__ __align__(8) uint64_t bar_full[T_NS], bar_empty[T_NS], bar_accfull[2], bar_accempty[2];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (warp == 0) tmem_alloc(&tmem_slot, 512);
  if (tid == 32) {
    for (int i = 0; i < T_NS; ++i) { mbar_init(&bar_full[i], 512); mbar_init(&bar_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_accfull[i], 1); mbar_init(&bar_accempty[i], 256); }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  constexpr int NH = N / 128, NCH = K / T_KC;
  const int nh = blockIdx.x % NH, tile0 = blockIdx.x / NH, tile_step = gridDim.x / NH;
  const int ntiles = (g.M + 127) / 128;

  if (warp < 8) {
    // ================================ epilogue warps ================================
    const int n = 32 * (warp & 3) + lane, hh = warp >> 2;
    const uint32_t lane_addr = (uint32_t)(32 * (warp & 3)) << 16;
    const int col = 128 * nh + n;
    {
      // W[:, col] -> bf16 (hi, lo) pairs of consecutive k -> TMEM; this thread covers k in [hh K/2, (hh+1) K/2)
      const float* wsrc = g.W + col;
#pragma unroll 1
      for (int q = 0; q < K / 64; ++q) {
        uint32_t h[16], l[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int k = hh * (K / 2) + 32 * q + 2 * j;
          split_pack(wsrc[(size_t)k * N], wsrc[(size_t)(k + 1) * N], h[j], l[j]);
        }
        const uint32_t c0 = T_WCOL + (uint32_t)(hh * (K / 4) + 16 * q);
        tmem_st16(tmem + lane_addr + c0, h);
        tmem_st16(tmem + lane_addr + c0 + K / 2, l);
      }
      tmem_wait_st();
      tc_fence_before();
      named_bar_sync(1, 288);
    }
    const float bias = g.bias ? g.bias[col] : 0.f;
    // rows [16 warp, +16) of the tile's blocks of z / add / resid -> L2, one tile ahead of their use
    auto prefetch_tile = [&](int tile_) {
      const int row = tile_ * 128 + 16 * warp;
      if (lane == 0 && tile_ < ntiles && row < g.M) {
        const uint32_t bytes = (uint32_t)min(16, g.M - row) * N * 4u;
        if (g.mulz) prefetch_l2_bulk(g.mulz + (size_t)row * N, bytes);
        if (g.add) prefetch_l2_bulk(g.add + (size_t)row * N, bytes);
        if (g.resid) prefetch_l2_bulk(g.resid + (size_t)row * N, bytes);
      }
    };
    prefetch_tile(tile0);
    int t = 0;
    for (int tile = tile0; tile < ntiles; tile += tile_step, ++t) {
      const int a = t & 1;
      prefetch_tile(tile + tile_step);
      mbar_wait_parked(&bar_accfull[a], (uint32_t)(t >> 1) & 1u, 2000u);
      tc_fence_after();
      const int r0 = tile * 128 + 64 * hh;
#pragma unroll 1
      for (int b = 0; b < 2; ++b) {
        uint32_t x[32];
        tmem_ld32(tmem + 128u * a + lane_addr + (uint32_t)(64 * hh + 32 * b), x);
        tmem_wait_ld();
        if (b == 1) {      // the accumulator is in registers: the MMAs of tile t + 2 may overwrite it
          tc_fence_before();
          mbar_arrive(&bar_accempty[a]);
        }
        const int rb = r0 + 32 * b;
        const size_t o0 = (size_t)rb * N + col;
        const int nrows = g.M - rb;
        const int ops = (g.resid ? 4 : 0) | (g.add ? 2 : 0) | (g.mulz ? 1 : 0);
        switch (ops) {
          case 0: epi_rows_any<N, false, false, false>(g, x, o0, bias, nrows); break;
          case 1: epi_rows_any<N, false, false, true>(g, x, o0, bias, nrows); break;
          case 2: epi_rows_any<N, false, true, false>(g, x, o0, bias, nrows); break;
          case 3: epi_rows_any<N, false, true, true>(g, x, o0, bias, nrows); break;
          case 4: epi_rows_any<N, true, false, false>(g, x, o0, bias, nrows); break;
          case 5: epi_rows_any<N, true, false, true>(g, x, o0, bias, nrows); break;
          case 6: epi_rows_any<N, true, true, false>(g, x, o0, bias, nrows); break;
          default: epi_rows_any<N, true, true, true>(g, x, o0, bias, nrows); break;
        }
      }
    }
  } else if (warp < 24) {
    // ================================ producer warps ================================
    // warp pw owns row group pw (8 rows) of every chunk: lane l loads k = l and k = 32 + l of its 8 rows
    const int pw = warp - 8;
    float nx[16];
    auto fetch = [&](int tile_, int c_) {
      const int rbase = tile_ * 128 + 8 * pw;
      const float* src = g.A + (size_t)rbase * K + c_ * T_KC + lane;
      if (rbase + 8 <= g.M && tile_ < ntiles) {      // all 8 rows exist: immediate offsets, no predicates
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
          for (int r = 0; r < 8; ++r) nx[8 * u + r] = src[r * K + 32 * u];
      } else {
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
          for (int r = 0; r < 8; ++r)
            nx[8 * u + r] = (tile_ < ntiles && rbase + r < g.M) ? src[r * K + 32 * u] : 0.f;
      }
    };
    // my rows of a tile's block of A -> L2, two tiles ahead of the register loads
    auto prefetch_tile = [&](int tile_) {
      const int row = tile_ * 128 + 8 * pw;
      if (lane == 0 && tile_ < ntiles && row < g.M)
        prefetch_l2_bulk(g.A + (size_t)row * K, (uint32_t)min(8, g.M - row) * K * 4u);
    };
    prefetch_tile(tile0 + tile_step);
    // register loads run two chunks ahead of the conversion (nx0: next chunk, nx: the one after)
    float nx0[16];
    fetch(tile0, 0);
#pragma unroll
    for (int i = 0; i < 16; ++i) nx0[i] = nx[i];
    if (NCH > 1) fetch(tile0, 1); else fetch(tile0 + tile_step, 0);
    int gch = 0;
    for (int tile = tile0; tile < ntiles; tile += tile_step) {
      prefetch_tile(tile + 2 * tile_step);
#pragma unroll 1
      for (int c = 0; c < NCH; ++c, ++gch) {
        float cur[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) { cur[i] = nx0[i]; nx0[i] = nx[i]; }
        if (c + 2 < NCH) fetch(tile, c + 2);
        else fetch(tile + tile_step, c + 2 - NCH);
        if (g.a_op) {
#pragma unroll
          for (int i = 0; i < 16; ++i) cur[i] = silu(cur[i]);
        }
        uint32_t h[2][4], l[2][4];
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
          for (int p = 0; p < 4; ++p) split_pack(cur[8 * u + 2 * p], cur[8 * u + 2 * p + 1], h[u][p], l[u][p]);
        const int slot = gch % T_NS, use = gch / T_NS;
        if (use > 0) mbar_wait_parked(&bar_empty[slot], (uint32_t)(use - 1) & 1u, 1000u);
        unsigned char* d = smem + slot * T_SLOT + pw * (int)T_SBO + lane * 16;
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          *reinterpret_cast<uint4*>(d + u * 512) = make_uint4(h[u][0], h[u][1], h[u][2], h[u][3]);
          *reinterpret_cast<uint4*>(d + u * 512 + T_IMG) = make_uint4(l[u][0], l[u][1], l[u][2], l[u][3]);
        }
        fence_proxy_async();
        mbar_arrive(&bar_full[slot]);
      }
    }
  } else {
    // ================================ MMA issue warp ================================
    named_bar_sync(1, 288);      // W^T is in tensor memory
    tc_fence_after();
    if (lane == 0) {
      const uint32_t idesc = make_idesc_bf16(128, 128) | IDESC_B_MN;
      const uint32_t sbase = smem_u32(smem);
      int gch = 0, t = 0;
      for (int tile = tile0; tile < ntiles; tile += tile_step, ++t) {
        const int a = t & 1;
        if (t >= 2) { while (!mbar_try_wait(&bar_accempty[a], (uint32_t)((t >> 1) - 1) & 1u)) __nanosleep(64); tc_fence_after(); }
        const uint32_t acc = tmem + 128u * a;
#pragma unroll 1
        for (int c = 0; c < NCH; ++c, ++gch) {
          const int slot = gch % T_NS, use = gch / T_NS;
          while (!mbar_try_wait(&bar_full[slot], (uint32_t)use & 1u)) __nanosleep(32);
          tc_fence_after();
          const uint32_t bsm = sbase + (uint32_t)slot * T_SLOT;
#pragma unroll
          for (int ks = 0; ks < T_KC / 16; ++ks) {
            const uint64_t bh = make_sdesc(bsm + ks * 2 * T_LBO, T_LBO, T_SBO);
            const uint64_t bl = make_sdesc(bsm + T_IMG + ks * 2 * T_LBO, T_LBO, T_SBO);
            const uint32_t a_hi = tmem + T_WCOL + (uint32_t)(c * (T_KC / 2) + ks * 8), a_lo = a_hi + K / 2;
            mma_ts(acc, a_hi, bh, idesc, (c | ks) ? 1u : 0u);
            mma_ts(acc, a_lo, bh, idesc, 1u);
            mma_ts(acc, a_hi, bl, idesc, 1u);
          }
          mma_commit(&bar_empty[slot]);
        }
        mma_commit(&bar_accfull[a]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

template <int K, int N>
cudaError_t launch(const GemmArgs& g, int num_sms, cudaStream_t st) {
  const int ntiles = (g.M + 127) / 128;
  constexpr int NH = N / 128;
  int groups = num_sms / NH;
  if (groups > ntiles) groups = ntiles;
  const size_t smem = (size_t)T_NS * T_SLOT;
  auto kern = gemm_rows_tcT_kernel<K, N>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  kern<<<groups * NH, T_NT, smem, st>>>(g);
  return cudaGetLastError();
}

// =====================================================================================================================
// dW[K, N] += op(A)[M, K]^T dZ[M, N]   (weight gradients: the reduction runs over the M = 175 k edge rows)
//
//   D[k (TMEM lane), n (column)] += A'[k][m] B'[m][n]  with K' = m: both operands are the row-major fp32 matrices
//   themselves, which is exactly the MN-major canonical layout once 8 consecutive columns of a row are packed into one
//   16-byte bf16 vector:  offset(col, m) = (m/8) LBO + (col/8) 128 + (m%8) 16 + (col%8) 2.  A CTA walks its slab of rows
//   in 32-row chunks: coalesced loads -> op -> bf16 (hi, lo) -> shared memory (conflict-free 512-byte warp stores), two
//   stages, the MMAs of chunk c (3 passes x 2 row steps x K/128 lane halves, N = 256 columns each) run while chunk c+1 is
//   converted.  The fp32 accumulators fill tensor memory (K/128 x N columns); at the end every CTA adds its partial to
//   dW with 16-byte vector reductions.
// =====================================================================================================================
constexpr uint32_t IDESC_A_MN = 1u << 15;
constexpr int DW_NT = 512;
constexpr int DW_PF = 3;        // L2 prefetch distance in 32-row chunks
constexpr int DW_NS = 3;        // ring stages (64 KB each for K = N = 256)

// Rows [r0, r0 + 32) of a row-major [M x C] matrix -> the (hi, lo) images at dst (C * 64 B each), in two steps so that
// the loads of the next chunk are in flight while this one is converted: load_chunk (coalesced 2 x 16 B per thread and
// (row group, column block) combination) and convert_chunk (op, bf16 split, conflict-free 16-byte stores); csum
// (optional) accumulates this thread's share of the column sums (the bias gradient) on the way
// 256-bit global load (sm_100): 8 consecutive floats, 32-byte aligned
__device__ __forceinline__ void ldg256(const float* p, float4& a, float4& b) {
  asm volatile("ld.global.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
               : "l"(p));
}
template <int C>
__device__ __forceinline__ void load_chunk(const float* __restrict__ src, int M, int r0, int tid,
                                           float4 (&v)[4 * (C / 32) / (512 / 32)][2]) {
  constexpr int XB = C / 32, NW = 512 / 32, NJ = 4 * XB / NW;
  static_assert(NJ >= 1, "warps");
  const int warp = tid >> 5, lane = tid & 31;
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    const int combo = warp + NW * j, mg = combo & 3, x = combo >> 2;
    const int m = 8 * mg + (lane & 7), cg = 4 * x + (lane >> 3);
    v[j][0] = make_float4(0.f, 0.f, 0.f, 0.f);
    v[j][1] = v[j][0];
    if (r0 + m < M) {
      const float* p = src + (size_t)(r0 + m) * C + 8 * cg;
      ldg256(p, v[j][0], v[j][1]);      // one request per 32-byte sector: a warp load = 8 rows x one full 128-byte line
    }
  }
}
template <int C, bool SUM>
__device__ __forceinline__ void convert_chunk(const float4 (&v)[4 * (C / 32) / (512 / 32)][2], int op, unsigned char* dst_hi,
                                              unsigned char* dst_lo, int tid, float (&csum)[4 * (C / 32) / (512 / 32)][8]) {
  constexpr int XB = C / 32;                  // blocks of 4 column groups (32 columns) per row
  constexpr int NW = DW_NT / 32;
  constexpr int NJ = 4 * XB / NW;             // (row group, block) combinations per warp
  const int warp = tid >> 5, lane = tid & 31;
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    const int combo = warp + NW * j, mg = combo & 3, x = combo >> 2;
    const int m = 8 * mg + (lane & 7), cg = 4 * x + (lane >> 3);
    float4 a = v[j][0], b = v[j][1];
    if (op) {
      a.x = silu(a.x); a.y = silu(a.y); a.z = silu(a.z); a.w = silu(a.w);
      b.x = silu(b.x); b.y = silu(b.y); b.z = silu(b.z); b.w = silu(b.w);
    }
    if (SUM) {
      csum[j][0] += a.x; csum[j][1] += a.y; csum[j][2] += a.z; csum[j][3] += a.w;
      csum[j][4] += b.x; csum[j][5] += b.y; csum[j][6] += b.z; csum[j][7] += b.w;
    }
    uint32_t h[4], l[4];
    split_pack(a.x, a.y, h[0], l[0]); split_pack(a.z, a.w, h[1], l[1]);
    split_pack(b.x, b.y, h[2], l[2]); split_pack(b.z, b.w, h[3], l[3]);
    const int off = mg * (C * 16) + cg * 128 + (m & 7) * 16;
    *reinterpret_cast<uint4*>(dst_hi + off) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(dst_lo + off) = make_uint4(l[0], l[1], l[2], l[3]);
  }
}

template <int K, int N>
__global__ void __launch_bounds__(DW_NT + 32, 1) dw_tc_kernel(const float* __restrict__ A, int a_op, const float* __restrict__ dZ,
                                                            float* __restrict__ dW, float* __restrict__ colsum, int M,
                                                            int rows_per_cta) {
  static_assert((K == 128 || K == 256) && (N == 128 || N == 256) && (K / 128) * N <= 512, "shapes");
  constexpr int A_IMG = 32 * K * 2, B_IMG = 32 * N * 2;           // bytes of one (hi or lo) image of a 32-row chunk
  constexpr int STAGE = 2 * A_IMG + 2 * B_IMG;
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ uint32_t tmem_slot;
  __shared__ __align__(8) uint64_t bar_full[DW_NS], bar_empty[DW_NS], bar_done;
  const int tid = threadIdx.x, warp = tid >> 5;
  if (warp == 0) tmem_alloc(&tmem_slot, 512);
  if (tid == 32) {
    for (int i = 0; i < DW_NS; ++i) { mbar_init(&bar_full[i], DW_NT); mbar_init(&bar_empty[i], 1); }
    mbar_init(&bar_done, 1);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  const int m_begin = blockIdx.x * rows_per_cta, m_end = min(M, m_begin + rows_per_cta);
  const int nchunks = (m_end - m_begin + 31) / 32;
  constexpr int NJA = 4 * (K / 32) / (DW_NT / 32), NJB = 4 * (N / 32) / (DW_NT / 32);
  float asum[NJA][8], bsum[NJB][8];      // asum is never used (SUM = false); bsum: column sums of dZ = the bias gradient
#pragma unroll
  for (int j = 0; j < NJB; ++j)
#pragma unroll
    for (int i = 0; i < 8; ++i) bsum[j][i] = 0.f;
  if (warp == DW_NT / 32) {
    // ---- MMA issue warp: chunk c of the ring -> 3 passes x 2 row steps x K/128 lane halves into the accumulators ----
    if ((tid & 31) == 0) {
      const uint32_t idesc = make_idesc_bf16(128, N) | IDESC_A_MN | IDESC_B_MN;
      constexpr uint32_t LBO_A = K * 16, LBO_B = N * 16;
      for (int c = 0; c < nchunks; ++c) {
        const int s = c % DW_NS, use = c / DW_NS;
        while (!mbar_try_wait(&bar_full[s], (uint32_t)use & 1u)) __nanosleep(32);
        tc_fence_after();
        const uint32_t a_hi = smem_u32(smem + s * STAGE), a_lo = a_hi + A_IMG, b_hi = a_hi + 2 * A_IMG, b_lo = b_hi + B_IMG;
#pragma unroll
        for (int h = 0; h < K / 128; ++h) {
#pragma unroll
          for (int ms = 0; ms < 2; ++ms) {
            const uint64_t ah = make_sdesc(a_hi + h * 2048 + ms * 2 * LBO_A, LBO_A, 128);
            const uint64_t al = make_sdesc(a_lo + h * 2048 + ms * 2 * LBO_A, LBO_A, 128);
            const uint64_t bh = make_sdesc(b_hi + ms * 2 * LBO_B, LBO_B, 128);
            const uint64_t bl = make_sdesc(b_lo + ms * 2 * LBO_B, LBO_B, 128);
            const uint32_t acc = tmem + (uint32_t)(h * N);
            mma_ss(acc, ah, bh, idesc, (c > 0 || ms > 0) ? 1u : 0u);
            mma_ss(acc, al, bh, idesc, 1u);
            mma_ss(acc, ah, bl, idesc, 1u);
          }
        }
        mma_commit(&bar_empty[s]);
      }
      mma_commit(&bar_done);
    }
  } else {
    // ---- conversion warps: every warp runs ahead on its own (no CTA barrier), bounded by the ring ----
    float4 na[NJA][2], nb[NJB][2];         // the next chunk, loaded one iteration ahead
    if (nchunks > 0) { load_chunk<K>(A, m_end, m_begin, tid, na); load_chunk<N>(dZ, m_end, m_begin, tid, nb); }
    if (tid < 2 && nchunks > 1) {               // the first DW_PF - 1 chunks after chunk 0 -> L2
      const int r = m_begin + 32;
      const uint32_t rows = (uint32_t)min(32 * (DW_PF - 1), m_end - r);
      if (tid == 0) prefetch_l2_bulk(A + (size_t)r * K, rows * K * 4u);
      else prefetch_l2_bulk(dZ + (size_t)r * N, rows * N * 4u);
    }
    for (int c = 0; c < nchunks; ++c) {
      const int s = c % DW_NS, use = c / DW_NS;
      float4 ca[NJA][2], cb[NJB][2];
#pragma unroll
      for (int j = 0; j < NJA; ++j) { ca[j][0] = na[j][0]; ca[j][1] = na[j][1]; }
#pragma unroll
      for (int j = 0; j < NJB; ++j) { cb[j][0] = nb[j][0]; cb[j][1] = nb[j][1]; }
      if (c + 1 < nchunks) {
        load_chunk<K>(A, m_end, m_begin + 32 * (c + 1), tid, na);
        load_chunk<N>(dZ, m_end, m_begin + 32 * (c + 1), tid, nb);
      }
      if (tid < 2 && c + DW_PF < nchunks) {      // chunk c + DW_PF of A / dZ (contiguous 32 rows) -> L2
        const int r = m_begin + 32 * (c + DW_PF);
        const uint32_t rows = (uint32_t)min(32, m_end - r);
        if (tid == 0) prefetch_l2_bulk(A + (size_t)r * K, rows * K * 4u);
        else prefetch_l2_bulk(dZ + (size_t)r * N, rows * N * 4u);
      }
      if (use > 0) mbar_wait_parked(&bar_empty[s], (uint32_t)(use - 1) & 1u, 500u);   // the MMAs of chunk c - DW_NS have left stage s
      unsigned char* st = smem + s * STAGE;
      convert_chunk<K, false>(ca, a_op, st, st + A_IMG, tid, asum);
      if (colsum) convert_chunk<N, true>(cb, 0, st + 2 * A_IMG, st + 2 * A_IMG + B_IMG, tid, bsum);
      else convert_chunk<N, false>(cb, 0, st + 2 * A_IMG, st + 2 * A_IMG + B_IMG, tid, bsum);
      fence_proxy_async();
      mbar_arrive(&bar_full[s]);
    }
  }
  if (warp < DW_NT / 32) {
  if (colsum) {
    // my partial column sums: lanes that differ in the row (lane & 7) hold the same columns
    const int lane = tid & 31;
#pragma unroll
    for (int j = 0; j < NJB; ++j) {
      const int combo = warp + (DW_NT / 32) * j, x = combo >> 2, cg = 4 * x + (lane >> 3);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float v = bsum[j][i];
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        v += __shfl_xor_sync(0xffffffffu, v, 4);
        if ((lane & 7) == 0) atomicAdd(colsum + 8 * cg + i, v);
      }
    }
  }
  // bar_done: every MMA has completed
  if (nchunks > 0) {
    mbar_wait_parked(&bar_done, 0u, 1000u);
    tc_fence_after();
    const uint32_t lane_addr = (uint32_t)(32 * (warp & 3)) << 16;
    const int lane_k = tid & 127, ch = tid >> 7;          // my lane (k within the half) and my quarter of the N columns
#pragma unroll 1
    for (int h = 0; h < K / 128; ++h) {
#pragma unroll 1
      for (int q = 0; q < N / 128; ++q) {
        uint32_t v[32];
        const int col = ch * (N / 4) + 32 * q;
        tmem_ld32(tmem + (uint32_t)(h * N) + lane_addr + (uint32_t)col, v);
        tmem_wait_ld();
        float* dst = dW + (size_t)(128 * h + lane_k) * N + col;
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4)
          asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + 4 * c4), "f"(__uint_as_float(v[4 * c4])),
                       "f"(__uint_as_float(v[4 * c4 + 1])), "f"(__uint_as_float(v[4 * c4 + 2])), "f"(__uint_as_float(v[4 * c4 + 3]))
                       : "memory");
      }
    }
  }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

template <int K, int N>
cudaError_t launch_dw(const float* A, int a_op, const float* dZ, float* dW, float* colsum, int M, int num_sms, cudaStream_t st) {
  constexpr int STAGE = 2 * (32 * K * 2) + 2 * (32 * N * 2);
  const size_t smem = (size_t)DW_NS * STAGE;
  auto kern = dw_tc_kernel<K, N>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  int rows_per_cta = ((M + num_sms - 1) / num_sms + 31) / 32 * 32;
  const int grid = (M + rows_per_cta - 1) / rows_per_cta;
  kern<<<grid, DW_NT + 32, smem, st>>>(A, a_op, dZ, dW, colsum, M, rows_per_cta);
  return cudaGetLastError();
}

}  // namespace ecnf_train_tc
