// Engine A on the 5th-generation tensor cores (tcgen05 + TMEM): (mlp_units, n_invariant_feat_hidden) = (128, 64)
// (DW4 / LJ13) and (64, 32) (ALDP), with or without the exact divergence.
//
// Same algorithm and tangent-row scheme as the fp32 SIMT engine (ecnf_solve_impl.cuh); the formulation is transposed
// ("feature on lane") so that everything the tangent rule needs is thread-local:
//
//     D^T[out feature (TMEM lane), row (TMEM column)] = W^T (A operand, TMEM) x Act^T (B operand, shared memory)
//
//   * a row tile is 128 accumulator COLUMNS = 16 chunks of 8 columns; a chunk is "one primal row of an edge / node and
//     up to 7 of its tangent rows" (a group with more tangents takes several chunks, each repeating the primal column),
//     so the activation rule  a = silu(z + b) / a-dot = silu'(z_primal) z-dot  is the same straight-line code for every
//     chunk: column 0 of a chunk is a static register and silu' a per-chunk scalar;
//   * thread (f, hh) of the 256 epilogue threads owns TMEM lane f and the 64 columns [64 hh, +64) -- the natural
//     tcgen05.ld 32x32b ownership.  With U = 128 lane = feature; with U = 64 two SUB-TILES are stacked on the lanes
//     (lanes [0, 64) sub-tile 0, [64, 128) sub-tile 1) and the weights are block-diagonal, so all 128 lanes, all epilogue
//     threads and the same K = 128 pipeline are used for the narrow network too;
//   * activations: accumulator (TMEM, fp32) -> registers -> rule -> bf16 (hi, lo) split -> B operand in shared memory,
//     MN-major no-swizzle canonical layout (8 rows of one feature = one 16-byte store, a warp stores 512 contiguous B);
//   * phi_e layer 0 (the sender / receiver gather) is an MMA too: node phase 1 leaves h_in as pre-split bf16 (hi | lo)
//     rows in the CTA's scratch (L2), and the B operand [h_in[sender] | h_in[receiver]] (K-major) of a tile is assembled
//     by 16-byte cp.async copies -- no register staging, no split, no L2 latency on the epilogue threads;
//   * weights: pre-split bf16 (hi, lo) images, loaded from L2 straight into TENSOR MEMORY (tcgen05.st) by the epilogue
//     threads, double buffered, so the MMA reads only B from shared memory;
//   * every Dense layer is 3 x (K/16) tcgen05.mma (hi*hi + lo*hi + hi*lo, fp32 accumulate: ~2^-17 relative per
//     product, measured 4e-6 by tools/probe_tc2.cu) -- single-pass bf16/tf32 misses the 1e-4 tolerance on log q;
//   * warp roles (384 threads): warps 0-7 epilogue (the MLP chain, the two Dense(1) head dot products, the message
//     aggregation), warps 8-10 "side" warps, a thread per tile column (per-column metadata, the layer-0 gather, the
//     coordinate update and its tangents), warp 11 issues the MMAs.  Two tiles are in flight (two accumulators, two B
//     buffers); all hand-over is by mbarriers:  side -built-> MMA -done-> epilogue -ready-> MMA ... epilogue -heads-> side;
//   * message aggregation: the chunks of one (receiver, slot group) are consecutive, so their gated messages are summed in
//     registers and added once per run to a shared-memory accumulator (one copy per thread group: fixed order, run-to-run
//     deterministic);
//   * tile composition (which (group, slot) sits in which chunk) is precomputed per (n, dim, kind) into a table.
#pragma once
#include "ecnf_solve_impl.cuh"
#include "ecnf_tc.cuh"

namespace ecnf_solve_detail {

using namespace ecnf_tc;

constexpr int TC_NT = 384;          // 8 epilogue warps + 3 side warps + 1 MMA-issue warp (12 warps: 168 registers each)
constexpr int TC_EPI = 256, TC_SIDE = 96;
#ifndef TC_WPREFETCH
#define TC_WPREFETCH 0   // 1: 2 KB of spills at 168 registers (measured: slower)
#endif
constexpr int TC_BOP = 65536;       // one B-operand buffer: hi image [K = 128][N = 128] + lo image
constexpr uint32_t TC_LBO = 128, TC_SBO = 2048;       // MN-major B (activations written by the epilogue threads)
constexpr uint32_t TC_LBO_K = 2048, TC_SBO_K = 128;   // K-major B (the gathered layer-0 operand)
constexpr int TC_WCOL = 256;        // first TMEM column of the weight buffers (accumulators: [0, 128) and [128, 256))

// chunk word of a tile table
constexpr uint32_t CH_VALID = 1u << 31, CH_GRPEND = 1u << 22, CH_OWNER = 1u << 23, CH_RUNEND = 1u << 24;
__host__ __device__ __forceinline__ int ch_gid(uint32_t w) { return (int)(w & 1023u); }
__host__ __device__ __forceinline__ int ch_qb(uint32_t w) { return (int)((w >> 10) & 255u); }    // slot of column 1 (0: dense chunk)
__host__ __device__ __forceinline__ int ch_cnt(uint32_t w) { return (int)((w >> 18) & 15u); }     // valid columns, 1..8
// header words (from word 32 of a tile)
enum { TH_N = 0, TH_FLUSH, TH_WIN_I, TH_WIN_NR, TH_WIN_S, TH_WIN_NS, TH_NCH /* +sub*2+hh */, TH_IFIRST = 10, TH_ILAST, TH_P, TH_MR, TH_RUNMASK };

// sigmoid from ex2.approx / rcp.approx (5 instructions, ~1e-7 absolute: well inside the 3-pass GEMM error)
__device__ __forceinline__ float fast_sigmoid(float z) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(z * -1.4426950408889634f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.f + e));
  return r;
}
// the same on a pair (the two multiplies and adds packed, ex2 / rcp per lane)
__device__ __forceinline__ float2 fast_sigmoid2(float2 z) {
  const float2 t = mul2(z, splat2(-1.4426950408889634f));
  float2 e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.x) : "f"(t.x));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.y) : "f"(t.y));
  const float2 d = add2(splat2(1.f), e);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r.x) : "f"(d.x));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r.y) : "f"(d.y));
  return r;
}
// columns (c, c + 1) of a thread's 64 accumulator values as a pair (c even)
__device__ __forceinline__ float2 col2(const float (&v)[64], int c) { return make_float2(v[c], v[c + 1]); }
__device__ __forceinline__ void set_col2(float (&v)[64], int c, float2 p) { v[c] = p.x; v[c + 1] = p.y; }

// ntan = tangent directions carried: n * dim (exact trace: the basis) or 1 (Hutchinson: the probe; tables TT_NODE and TT_MID)
__host__ __device__ inline int tc_rows_of_kind(int kind, int n, int dim, int ntan) {
  const int ND = 1 + ntan;
  return (kind == TT_NODE1 || kind == TT_EDGE1) ? 1 : kind == TT_NODE ? ND : kind == TT_FIRST ? 1 + 2 * dim : kind == TT_MID ? ND : 1 + dim;
}

// Packs the groups (nodes or edges) of one table kind into tiles of 16 * SUB chunks; returns the tile count, writes them
// when out != null.  Chunk p of a tile sits in sub-tile p % SUB, column half (p / SUB) % 2, chunk position p / (2 SUB)
// (both halves and both sub-tiles fill evenly).  MR = rows of the message accumulator: tiles of the message-passing kinds
// never span two windows (a window = some receivers x a slot range whose aggregate fits MR rows).
// stage: optional TC_TILE_WORDS-word scratch the current tile is assembled in (the device builder passes shared memory: the
// packing is a chain of read-modify-writes that costs ~1 ms per launch straight on global memory); it is copied out on close.
__host__ __device__ inline int tc_pack(int kind, int n, int dim, int SUB, int MR, uint32_t* out, int ntan, uint32_t* stage = nullptr) {
  const int ND = 1 + ntan, nb = n - 1;
  const bool edge = kind >= TT_FIRST;
  const int ngroups = edge ? n * nb : n;
  const int r = tc_rows_of_kind(kind, n, dim, ntan);
  const bool dense = (r == 1);
  const int CAP = 16 * SUB;
  int tile = 0, p = 0;
  int win_i = 0, win_nr = 0, win_s = 0, win_ns = 0, i_first = 0, i_last = 0;
  int run_start = 0;     // first chunk (index in the tile) of the current run
  auto tp = [&](int t) { return stage ? stage : out + (size_t)t * TC_TILE_WORDS; };
  auto word_index = [&](int q) { return (q % SUB) * 16 + ((q / SUB) % 2) * 8 + q / (2 * SUB); };
  // chunks [run_start, p) form a run (the chunks whose coordinate contributions are summed): mark its end (CH_RUNEND) and the
  // last chunk of every thread group (CH_GRPEND: where the epilogue threads flush their message partial sums); each_chunk:
  // every chunk flushes on its own (first block: the per-sender tangent rows)
  auto end_run = [&](bool each_chunk = false) {
    if (out && p > run_start) {
      tp(tile)[word_index(p - 1)] |= CH_RUNEND;
      for (int q = run_start; q < p; ++q)
        if (each_chunk || q + 2 * SUB >= p) tp(tile)[word_index(q)] |= CH_GRPEND;
    }
    run_start = p;
  };
  auto close = [&](int flush) {
    if (p == 0) return;
    end_run();
    if (out) {
      uint32_t* h = tp(tile) + 32;
      int nmax0 = 0, nmax1 = 0;
      for (int sb = 0; sb < SUB; ++sb)
        for (int hh = 0; hh < 2; ++hh) {
          // chunks q = sb + SUB * hh + 2 SUB * pos < p
          const int first = sb + SUB * hh;
          const int cntp = p > first ? (p - first + 2 * SUB - 1) / (2 * SUB) : 0;
          h[TH_NCH + sb * 2 + hh] = (uint32_t)cntp;
          if (hh == 0 && cntp > nmax0) nmax0 = cntp;
          if (hh == 1 && cntp > nmax1) nmax1 = cntp;
        }
      int N = nmax1 > 0 ? 64 + 8 * nmax1 : 8 * nmax0;
      N = (N + 15) & ~15;
      h[TH_N] = (uint32_t)(N < 16 ? 16 : N);
      h[TH_FLUSH] = (uint32_t)flush;
      h[TH_WIN_I] = (uint32_t)win_i; h[TH_WIN_NR] = (uint32_t)win_nr; h[TH_WIN_S] = (uint32_t)win_s; h[TH_WIN_NS] = (uint32_t)win_ns;
      h[TH_IFIRST] = (uint32_t)i_first; h[TH_ILAST] = (uint32_t)i_last; h[TH_P] = (uint32_t)p; h[TH_MR] = (uint32_t)MR;
      uint32_t rm = 0u;      // bit q: chunk q (sequence index) ends a run
      for (int q = 0; q < p; ++q)
        if (tp(tile)[word_index(q)] & CH_RUNEND) rm |= 1u << q;
      h[TH_RUNMASK] = rm;
      if (stage)
        for (int k = 0; k < TC_TILE_WORDS; ++k) out[(size_t)tile * TC_TILE_WORDS + k] = stage[k];
    }
    ++tile;
    p = 0; run_start = 0;
  };
  auto put = [&](int gid, int qb, int cnt, bool owner) {
    if (p == CAP) close(0);
    if (p == 0 && out)
      for (int k = 0; k < TC_TILE_WORDS; ++k) tp(tile)[k] = 0;
    const int i = edge ? gid / nb : gid;
    if (p == 0) i_first = i;
    i_last = edge ? (gid + (dense ? cnt - 1 : 0)) / nb : gid + (dense ? cnt - 1 : 0);
    if (out)
      tp(tile)[word_index(p)] = CH_VALID | (uint32_t)gid | ((uint32_t)qb << 10) | ((uint32_t)cnt << 18) | (owner ? CH_OWNER : 0u);
    ++p;
  };
  if (dense) {                       // TT_NODE1 / TT_EDGE1: 8 consecutive groups per chunk, every column a primal row
    win_i = 0; win_nr = n; win_s = 0; win_ns = 1;
    for (int g = 0; g < ngroups; g += 8) {
      put(g, 0, ngroups - g < 8 ? ngroups - g : 8, true);
      end_run();
    }
    close(kind == TT_EDGE1 ? 1 : 0);
    return tile;
  }
  if (kind == TT_NODE) {             // (node, slot group) chunks, no windows
    for (int g = 0; g < n; ++g)
      for (int qb = 1; qb < r; qb += 7) { put(g, qb, 1 + (r - qb < 7 ? r - qb : 7), qb == 1); end_run(); }
    close(0);
    return tile;
  }
  if (kind == TT_LAST) {             // one chunk per edge; a run = the edges of one receiver (coordinate sums)
    for (int i = 0; i < n; ++i) {
      for (int e = i * nb; e < (i + 1) * nb; ++e) {
        if (p == CAP) close(0);
        put(e, 1, r, true);
      }
      end_run();
    }
    close(0);
    return tile;
  }
  if (kind == TT_FIRST) {            // one chunk per edge; accumulator rows: (receiver, {primal, its own dim directions})
    const int rows_per = 1 + dim;
    int W = MR / rows_per; if (W < 1) W = 1; if (W > n) W = n;
    for (int i0 = 0; i0 < n; i0 += W) {
      win_i = i0; win_nr = (n - i0 < W) ? n - i0 : W; win_s = 0; win_ns = rows_per;
      for (int i = i0; i < i0 + win_nr; ++i) {
        for (int e = i * nb; e < (i + 1) * nb; ++e) {
          if (p == CAP) { end_run(true); close(0); }
          put(e, 1, r, true);
        }
        end_run(true);               // a run = the edges of one receiver; the message partial sums flush per chunk
      }
      close(1);
    }
    return tile;
  }
  // TT_MID: windows of whole receivers when ND <= MR, else one receiver x a slot range made of whole chunks
  if (ND <= MR) {
    int W = MR / ND; if (W > n) W = n;
    for (int i0 = 0; i0 < n; i0 += W) {
      win_i = i0; win_nr = (n - i0 < W) ? n - i0 : W; win_s = 0; win_ns = ND;
      for (int i = i0; i < i0 + win_nr; ++i)
        for (int qb = 1; qb < r; qb += 7) {
          for (int e = i * nb; e < (i + 1) * nb; ++e) {
            if (p == CAP) close(0);
            put(e, qb, 1 + (r - qb < 7 ? r - qb : 7), qb == 1);
          }
          end_run();
        }
      close(1);
    }
  } else {
    const int cpw = (MR - 1) / 7 > 0 ? (MR - 1) / 7 : 1;       // chunks (slot groups) per window
    for (int i = 0; i < n; ++i)
      for (int qw = 1; qw < r; qw += 7 * cpw) {
        const int q_end = (qw + 7 * cpw < r) ? qw + 7 * cpw : r;
        win_i = i; win_nr = 1; win_s = (qw == 1) ? 0 : qw; win_ns = q_end - win_s;
        for (int qb = qw; qb < q_end; qb += 7) {
          for (int e = i * nb; e < (i + 1) * nb; ++e) {
            if (p == CAP) close(0);
            put(e, qb, 1 + (r - qb < 7 ? r - qb : 7), qb == 1);
          }
          end_run();
        }
        close(1);
      }
  }
  return tile;
}

// shared-memory carve-up; MR (rows of the message accumulator) is the largest 1 + 7k (<= ND) that fits in 227 KB
template <int U, int H>
__host__ __device__ inline TcSmemLayout make_tc_layout(int n, int dim, int MR) {
  constexpr int SUB = 128 / U;
  const int D = n * dim, S = D + 1, E = n * (n - 1);
  TcSmemLayout L;
  int o = 0;
  auto take = [&](int bytes) { int r = o; o += (bytes + 127) & ~127; return r; };
  L.bop = take(2 * TC_BOP);
  L.mrows = MR;
  L.macc = take(2 * SUB * (MR + 1) * U * 4);   // one copy per (column half, sub-tile) thread group, + a dump row each
  L.xt = take(D * D * 4);
  L.xtacc = take(D * D * 4);
  L.dacc = take(D * 4);
  L.xs = take(D * 4);
  L.xs0 = take(D * 4);
  L.xacc = take(D * 4);
  L.mu = take(16);
  L.tau = take(ECNF_MAX_T * 4);
  L.cvec = take(64 * 4);
  L.ode = take(11 * S * 4);
  L.red = take((S + 16) * 4);
  // per-tile tables: one buffer per (slot, tile parity) so that the side warps prepare a tile two tiles ahead of its use
  L.colsd = take(4 * SUB * 128 * 4);
  L.colmrow = take(4 * SUB * 128 * 4);     // node phases: row offset of a column (coloffR)
  L.chw = take(4 * 32 * 4);
  L.hdr = take(4 * 16 * 4);
  L.pdot = take(2 * 8 * 64 * 4);           // attention-logit partials (consumed by the epilogue threads themselves)
  L.pdh = take(4 * 8 * 64 * 4);            // coordinate-head partials per (slot, tile parity), consumed by the side warps
  L.wA = take(8 * 64 * 4);
  L.wB = take(8 * 64 * 4);
  L.cdbuf = take(SUB * 128 * 3 * 4);
  L.egv = take(E * 4 * 4);     // per edge: v = x_i - x_j (3 floats) and the packed node pair (i | j << 8)
  L.bars = take(128);
  L.prof = take(32 * 8);
  L.total_bytes = o;
  return L;
}
template <int U, int H>
__host__ inline int tc_pick_mrows(int n, int dim, bool div) {
  const int ND = div ? 1 + n * dim : 1;
  if (!div) return n;                                   // primal-only edge tiles aggregate over all receivers at once
  int best = 0;
  const int cap = ND > 40 ? ND : 40;                    // whole receivers per window where they are small
  for (int mr = 8; mr <= cap; ++mr) {
    if (mr < ND && (mr - 1) % 7 != 0) continue;
    if (make_tc_layout<U, H>(n, dim, mr).total_bytes + 1024 <= 227 * 1024) best = mr;
  }
  return best;
}

extern __shared__ __align__(1024) unsigned char smem_tc[];

// Every buffer is addressed as (shared-memory base + offset from the kernel parameters): the offsets are constant-bank
// loads, so no pointer has to be kept alive in (or spilled from) registers across the very large inlined body.
#define TCF(field) (reinterpret_cast<float*>(smem_tc + a.lay.field))
#define TCI(field) (reinterpret_cast<int*>(smem_tc + a.lay.field))
#define TCW(field) (reinterpret_cast<uint32_t*>(smem_tc + a.lay.field))

// DIV = false: sample_cnf without a divergence -- primal rows only (tile kinds TT_NODE1 / TT_EDGE1, no tangent state)
template <int U_, int H_, bool DIV>
struct EngineTC {
  static constexpr int U = U_, H = H_, SUB = 128 / U_;
  static constexpr int NT = TC_NT;
  static constexpr int KN = SUB * H;      // K of the node-level layers (h rows of both sub-tiles)
  static constexpr int ROWB = 4 * H;      // bytes of one pre-split h_in row: H bf16 hi | H bf16 lo
  const KernelArgs& a;     // the __grid_constant__ kernel parameter
  const EcnfModelDev& m;
  const TcImages& img;
  const bool hutch;        // Hutchinson estimate: ONE tangent direction (the probe eps), every block of kind TT_MID
  const int n, dim, D, ntan, ND, E;
  const float* eps_g;      // probe of the current trajectory (global, D floats)
  const int tid, f, hh, warp, lane, sub, fu;
  const bool is_epi, is_side;
  uint32_t tmem;         // TMEM base address
  uint32_t lane_addr;    // (32 * (warp & 3)) << 16
  uint32_t par;          // phase parities of the mbarriers this thread waits on: bit (kind * 2 + slot)

  enum { B_READY = 0, B_DONE = 1, B_BUILT = 2, B_HEADS = 3, B_BFREE = 4 };
  enum { P_NODE_PRE, P_EDGE, P_NODE_POST, P_WAIT, P_EPI, P_MSG, P_HEAD, P_WLOAD, P_SIDE_WAIT, P_SIDE_GATHER, P_SIDE_COORD,
         P_SIDE_META, P_SIDE_CPWAIT, P_NBUILD, P_NCOUNT };
#ifdef ECNF_TC_PROFILE
  long long prof_t0, prof_t1;
  __device__ __forceinline__ long long* prof_s() const { return reinterpret_cast<long long*>(smem_tc + a.lay.prof); }
  __device__ __forceinline__ void pbeg() { prof_t0 = clock64(); }
  __device__ __forceinline__ void pend(int k) { const long long t1 = clock64(); if (tid == 0) prof_s()[k] += t1 - prof_t0; prof_t0 = t1; }
  __device__ __forceinline__ void qbeg() { prof_t1 = clock64(); }
  __device__ __forceinline__ void qend(int k) { const long long t1 = clock64(); if (tid == 0 || tid == TC_EPI) prof_s()[k] += t1 - prof_t1; prof_t1 = t1; }
#else
  __device__ __forceinline__ void pbeg() {}
  __device__ __forceinline__ void pend(int) {}
  __device__ __forceinline__ void qbeg() {}
  __device__ __forceinline__ void qend(int) {}
#endif

  __device__ __forceinline__ void set_eps(const float* e) { eps_g = e; }
  __device__ __forceinline__ float* ode_ptr() const { return TCF(ode); }
  __device__ __forceinline__ float* red_ptr() const { return TCF(red); }
  __device__ __forceinline__ uint64_t* bar(int kind, int s) const { return reinterpret_cast<uint64_t*>(smem_tc + a.lay.bars) + kind * 2 + s; }
  __device__ __forceinline__ uint32_t* tmem_slot() const { return reinterpret_cast<uint32_t*>(smem_tc + a.lay.bars + 96); }
  // per-CTA global scratch (L2 resident): h, h_in [n][ND][H] fp32; aggregated messages, P_h [n][ND][U] fp32;
  // h_in as pre-split bf16 rows [n * ND + 1][hi H | lo H] (the last row is all zero)
  __device__ __forceinline__ float* hA() const { return a.scratch + (size_t)blockIdx.x * a.scratch_stride; }
  __device__ __forceinline__ float* hB() const { return hA() + (size_t)n * ND * H; }
  __device__ __forceinline__ float* Mg() const { return hB() + (size_t)n * ND * H; }
  __device__ __forceinline__ float* Ph() const { return Mg() + (size_t)n * ND * U; }
  __device__ __forceinline__ unsigned char* Himg() const { return reinterpret_cast<unsigned char*>(Ph() + (size_t)n * ND * U); }

  __device__ __forceinline__ EngineTC(const KernelArgs& a_)
      : a(a_), m(a_.m), img(a_.img), hutch(DIV && a_.eps != nullptr), n(a_.m.n), dim(a_.m.dim), D(a_.m.n * a_.m.dim),
        ntan(DIV ? (a_.eps != nullptr ? 1 : a_.m.n * a_.m.dim) : 0), ND(1 + (DIV ? (a_.eps != nullptr ? 1 : a_.m.n * a_.m.dim) : 0)),
        E(a_.m.n * (a_.m.n - 1)), eps_g(nullptr), tid(threadIdx.x), f(threadIdx.x & 127), hh((threadIdx.x >> 7) & 1), warp(threadIdx.x >> 5),
        lane(threadIdx.x & 31), sub((threadIdx.x & 127) / U_), fu((threadIdx.x & 127) % U_), is_epi(threadIdx.x < TC_EPI),
        is_side(threadIdx.x >= TC_EPI && threadIdx.x < TC_EPI + TC_SIDE) {
    if (tid == 0) {
      mbar_init(bar(B_READY, 0), TC_EPI); mbar_init(bar(B_READY, 1), TC_EPI);
      mbar_init(bar(B_DONE, 0), 1); mbar_init(bar(B_DONE, 1), 1);
      mbar_init(bar(B_BUILT, 0), TC_SIDE); mbar_init(bar(B_BUILT, 1), TC_SIDE);
      mbar_init(bar(B_HEADS, 0), TC_EPI); mbar_init(bar(B_HEADS, 1), TC_EPI);
      mbar_init(bar(B_BFREE, 0), 1); mbar_init(bar(B_BFREE, 1), 1);
#ifdef ECNF_TC_PROFILE
      for (int k = 0; k < P_NCOUNT; ++k) prof_s()[k] = 0;
#endif
    }
    __syncwarp();
    if (warp == 0) tmem_alloc(tmem_slot(), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    tmem = *tmem_slot();
    lane_addr = (uint32_t)(32 * (warp & 3)) << 16;
    par = 0;
    if (is_epi) {   // accumulators start finite (columns beyond a tile's N are read but never used)
      uint32_t z[32];
#pragma unroll
      for (int c = 0; c < 32; ++c) z[c] = 0u;
#pragma unroll
      for (int q = 0; q < 4; ++q) tmem_st32(tmem + lane_addr + 128u * hh + 32u * q, z);
      tmem_wait_st();
    }
    if (is_side)    // the all-zero row of the pre-split h_in image
      for (int k = tid - TC_EPI; k < ROWB / 4; k += TC_SIDE) reinterpret_cast<uint32_t*>(Himg() + (size_t)n * ND * ROWB)[k] = 0u;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
  }
  __device__ __forceinline__ void finish(long long* out) {
#ifdef ECNF_TC_PROFILE
    if (out && tid == 0 && blockIdx.x == 0)
      for (int k = 0; k < P_NCOUNT; ++k) out[k] = prof_s()[k];
#endif
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
  }

  // ---- hand-over between the thread groups ----------------------------------------------------------------------------
  __device__ __forceinline__ void epi_bar() const { named_bar_sync(1, TC_EPI); }
  // the four warps that own one column half (their partial dot products are summed by each of them)
  __device__ __forceinline__ void half_bar() const { named_bar_sync(2 + hh, TC_EPI / 2); }
  __device__ __forceinline__ void side_bar() const { named_bar_sync(4, TC_SIDE); }
  __device__ __forceinline__ void phase_bar() const { named_bar_sync(5, TC_EPI + TC_SIDE); }   // epilogue + side threads
  __device__ __forceinline__ void wait_bar(int kind, int s) {
    const uint32_t bit = 1u << (kind * 2 + s);
    mbar_wait_parked(bar(kind, s), (par & bit) ? 1u : 0u, 20000u);
    par ^= bit;
    tc_fence_after();
  }
  __device__ __forceinline__ void wait_done(int s) { qbeg(); wait_bar(B_DONE, s); qend(P_WAIT); }
  // my part of slot s's next operands (B in shared memory, weights / drained accumulator in TMEM) is complete
  __device__ __forceinline__ void arrive(int kind, int s) {
    fence_proxy_async();
    tc_fence_before();
    mbar_arrive(bar(kind, s));
  }
  // issue warp: wait for the producers, then acc[s] = W^T (TMEM columns a_col: hi [0, K/2), lo [K/2, K)) x B[s]
  // (K x N), 3-pass split; commit -> done[s].  kmajor: B is the gathered layer-0 operand.
  // tb: table buffer of the tile (slot * 2 + tile parity).  free_b: these are the last MMAs of the tile that read B[s] -- a
  // second commit tells the side warps that the buffer can take the next tile's gathered operand.
  // drained: additionally wait until the epilogue threads have read the previous tile's last accumulator out of acc[s].
  __device__ __forceinline__ void issue_mma(int s, int tb, int wait_kind, uint32_t a_col, int K, bool kmajor, bool free_b,
                                            bool drained = false) {
    if (lane == 0) {
      if (drained) wait_bar(B_READY, s);
      wait_bar(wait_kind, s);
      const int N = hdr(tb, TH_N);
      const uint32_t idesc = make_idesc_bf16(128, N) | (kmajor ? 0u : IDESC_B_MN);
      const uint32_t bsm = smem_u32(smem_tc + a.lay.bop) + (uint32_t)s * TC_BOP;
      const uint32_t lbo = kmajor ? TC_LBO_K : TC_LBO, sbo = kmajor ? TC_SBO_K : TC_SBO;
      uint64_t bh = make_sdesc(bsm, lbo, sbo);
      uint64_t bl = make_sdesc(bsm + 32768u, lbo, sbo);
      const uint32_t acc = tmem + 128u * s;
      uint32_t a_hi = tmem + a_col, a_lo = tmem + a_col + (uint32_t)(K >> 1);
      const int nk = K >> 4;
      mma_ts(acc, a_hi, bh, idesc, 0u);
      mma_ts(acc, a_lo, bh, idesc, 1u);
      mma_ts(acc, a_hi, bl, idesc, 1u);
      for (int ks = 1; ks < nk; ++ks) {
        bh += (2u * lbo) >> 4; bl += (2u * lbo) >> 4; a_hi += 8; a_lo += 8;
        mma_ts(acc, a_hi, bh, idesc, 1u);
        mma_ts(acc, a_lo, bh, idesc, 1u);
        mma_ts(acc, a_hi, bl, idesc, 1u);
      }
      mma_commit(bar(B_DONE, s));
      if (free_b) mma_commit(bar(B_BFREE, s));
    }
  }

  // ---- per-thread column helpers (thread (f, hh): TMEM lane f, columns [64 hh, +64) of slot s) ------------------------
  __device__ __forceinline__ uint32_t my_acc(int s) const { return tmem + 128u * s + lane_addr + 64u * hh; }
  __device__ __forceinline__ void ld_acc(int s, float (&v)[64]) {
    uint32_t x[32], y[32];
    const uint32_t addr = my_acc(s);
    tmem_ld32(addr, x);
    tmem_ld32(addr + 32u, y);
    tmem_wait_ld();
#pragma unroll
    for (int c = 0; c < 32; ++c) { v[c] = __uint_as_float(x[c]); v[32 + c] = __uint_as_float(y[c]); }
  }
  // B operand of slot s (MN-major) <- v at K row `krow`, bf16 hi / lo
  __device__ __forceinline__ void write_B(int s, const float (&v)[64], int krow) {
    unsigned char* base = smem_tc + a.lay.bop + s * TC_BOP + (8 * hh) * (int)TC_SBO + krow * 16;
#pragma unroll
    for (int g8 = 0; g8 < 8; ++g8) {
      uint32_t h[4], l[4];
#pragma unroll
      for (int p = 0; p < 4; ++p) split_pack(v[8 * g8 + 2 * p], v[8 * g8 + 2 * p + 1], h[p], l[p]);
      *reinterpret_cast<uint4*>(base + g8 * (int)TC_SBO) = make_uint4(h[0], h[1], h[2], h[3]);
      *reinterpret_cast<uint4*>(base + 32768 + g8 * (int)TC_SBO) = make_uint4(l[0], l[1], l[2], l[3]);
    }
  }
  // The same three steps on one 32-column half (chunks [4 hf, 4 hf + 4)) at a time, so that the TMEM load of the second half is
  // in flight while the first half goes through the rule, the split and the stores.
  __device__ __forceinline__ void ld_half_issue(int s, int hf, uint32_t (&x)[32]) { tmem_ld32(my_acc(s) + 32u * hf, x); }
  template <bool L0>
  __device__ __forceinline__ void act_half(float (&v)[64], int hf, float bias, int tb, float wdf) {
    const float* sdp = TCF(colsd) + (tb * SUB + sub) * 128 + 64 * hh;
#pragma unroll
    for (int c4 = 0; c4 < 4; ++c4) act_chunk<L0>(v, 4 * hf + c4, bias, sdp, wdf);
  }
  __device__ __forceinline__ void write_half(int s, const float (&v)[64], int hf, int krow) {
    unsigned char* base = smem_tc + a.lay.bop + s * TC_BOP + (8 * hh + 4 * hf) * (int)TC_SBO + krow * 16;
#pragma unroll
    for (int g8 = 0; g8 < 4; ++g8) {
      uint32_t h[4], l[4];
#pragma unroll
      for (int p = 0; p < 4; ++p) split_pack(v[32 * hf + 8 * g8 + 2 * p], v[32 * hf + 8 * g8 + 2 * p + 1], h[p], l[p]);
      *reinterpret_cast<uint4*>(base + g8 * (int)TC_SBO) = make_uint4(h[0], h[1], h[2], h[3]);
      *reinterpret_cast<uint4*>(base + 32768 + g8 * (int)TC_SBO) = make_uint4(l[0], l[1], l[2], l[3]);
    }
  }
  // tile tables live in one buffer per (slot, tile parity):  tb = slot * 2 + ((tile >> 1) & 1)
  __device__ __forceinline__ static int tb_of(int s, int tile) { return s * 2 + ((tile >> 1) & 1); }
  __device__ __forceinline__ int hdr(int tb, int k) const { return TCI(hdr)[tb * 16 + k]; }
  __device__ __forceinline__ int my_nch(int tb) const { return hdr(tb, TH_NCH + sub * 2 + hh); }   // chunks in use in my 64 columns
  __device__ __forceinline__ uint32_t my_chw(int tb, int ch) const { return TCW(chw)[tb * 32 + sub * 16 + 8 * hh + ch]; }
  // Activation rule: a = silu(z + bias) on the primal column of every chunk, a-dot = silu'(z_primal) z-dot on the 7 tangent
  // columns behind it.  L0: z gets the rank-1 |v|^2 term of phi_e layer 0 first (sd = the tile's per-column table, wdf =
  // my feature's entry of w_d).  Branch-free over all 8 chunks: columns beyond the used ones hold finite stale values that
  // no table refers to.
  template <bool L0>
  __device__ __forceinline__ void act_rule(float (&v)[64], float bias, int tb, float wdf) {
    const float* sdp = TCF(colsd) + (tb * SUB + sub) * 128 + 64 * hh;
#pragma unroll
    for (int ch = 0; ch < 8; ++ch) act_chunk<L0>(v, ch, bias, sdp, wdf);
  }
  // the rule on chunk ch, on column pairs (every lane of a pair is the scalar operation of that column):
  // the primal column's z * sigmoid(z) shares its multiply with column 1's tangent scaling
  template <bool L0>
  __device__ __forceinline__ static void act_chunk(float (&v)[64], int ch, float bias, const float* sdp, float wdf) {
    const int c0 = 8 * ch;
    if constexpr (L0) {      // z += |v|^2 w_d
      const float4 s0 = reinterpret_cast<const float4*>(sdp)[2 * ch], s1 = reinterpret_cast<const float4*>(sdp)[2 * ch + 1];
      const float2 w2 = splat2(wdf);
      set_col2(v, c0, fma2(make_float2(s0.x, s0.y), w2, col2(v, c0)));
      set_col2(v, c0 + 2, fma2(make_float2(s0.z, s0.w), w2, col2(v, c0 + 2)));
      set_col2(v, c0 + 4, fma2(make_float2(s1.x, s1.y), w2, col2(v, c0 + 4)));
      set_col2(v, c0 + 6, fma2(make_float2(s1.z, s1.w), w2, col2(v, c0 + 6)));
    }
    if constexpr (!DIV) {      // every column is a primal row
#pragma unroll
      for (int u = 0; u < 8; u += 2) {
        const float2 z = add2(col2(v, c0 + u), splat2(bias));
        set_col2(v, c0 + u, mul2(z, fast_sigmoid2(z)));
      }
    } else {
      const float z = v[c0] + bias;
      const float sg = fast_sigmoid(z);
      const float cur = sg * (1.f + z * (1.f - sg));
      set_col2(v, c0, mul2(make_float2(z, v[c0 + 1]), make_float2(sg, cur)));
#pragma unroll
      for (int u = 2; u < 8; u += 2) set_col2(v, c0 + u, mul2(col2(v, c0 + u), splat2(cur)));
    }
  }
  template <int W>   // 2W partial sums -> W, exchanging with lane ^ (W/2)
  __device__ __forceinline__ void bfly_round(float (&x)[32]) const {
    const bool b = (lane & (W >> 1)) != 0;
#pragma unroll
    for (int i = 0; i < W; ++i) {
      const float keep = b ? x[W + i] : x[i], send = b ? x[i] : x[W + i];
      x[i] = keep + __shfl_xor_sync(0xffffffffu, send, W >> 1);
    }
  }
  // column sums over the 32 lanes of this warp of v[c] * wf (transposing butterfly): lane l ends with the columns
  // 2l and 2l+1 of its half, stored to pd[2l], pd[2l+1]
  __device__ __forceinline__ void warp_dot(const float (&v)[64], float wf, float* pd) {
    float x[32];
    {
      const bool b = (lane & 16) != 0;
      const float2 w2 = splat2(wf);
#pragma unroll
      for (int i = 0; i < 32; i += 2) {
        const float2 lo2 = mul2(col2(v, i), w2), hi2 = mul2(col2(v, 32 + i), w2);
        const float lo[2] = {lo2.x, lo2.y}, hi[2] = {hi2.x, hi2.y};
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const float keep = b ? hi[j] : lo[j], send = b ? lo[j] : hi[j];
          x[i + j] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
      }
    }
    bfly_round<16>(x);
    bfly_round<8>(x);
    bfly_round<4>(x);
    bfly_round<2>(x);
    *reinterpret_cast<float2*>(pd + 2 * lane) = make_float2(x[0], x[1]);
  }
  // complete dot product of column c (0..63 of half h2) of sub-tile sb from the 8 x 64 per-warp partials at pd
  __device__ __forceinline__ float full_dot(const float* pd, int h2, int sb, int c) const {
    const float* p4 = pd + (4 * h2) * 64 + c;
    if constexpr (SUB == 1) return (p4[0] + p4[64]) + (p4[128] + p4[192]);
    else return p4[(2 * sb) * 64] + p4[(2 * sb + 1) * 64];
  }
  // weight image (hi | lo, K x 128 lanes) -> registers -> TMEM columns [col, col + K)
  template <int K>
  __device__ __forceinline__ void fetch_w(int img_off, uint32_t (&wv)[2][K / 4]) {
    constexpr int NC = K / 16;     // uint4 chunks per thread and part
    const uint4* src = reinterpret_cast<const uint4*>(img.base + img_off);
#pragma unroll
    for (int p = 0; p < 2; ++p)
#pragma unroll
      for (int j = 0; j < NC; ++j) {
        const uint4 q = __ldg(src + (size_t)(p * (K / 8) + hh * NC + j) * 128 + f);
        wv[p][4 * j] = q.x; wv[p][4 * j + 1] = q.y; wv[p][4 * j + 2] = q.z; wv[p][4 * j + 3] = q.w;
      }
  }
  template <int K>
  __device__ __forceinline__ void store_w(const uint32_t (&wv)[2][K / 4], uint32_t col) {
#pragma unroll
    for (int p = 0; p < 2; ++p) {
      const uint32_t addr = tmem + col + lane_addr + (uint32_t)(p * (K / 2) + hh * (K / 4));
      if constexpr (K == 128) tmem_st32(addr, wv[p]);
      else tmem_st16(addr, wv[p]);
    }
    tmem_wait_st();
  }
  template <int K>
  __device__ __forceinline__ void load_w(int img_off, uint32_t col) {
    constexpr int NC = K / 16;     // uint4 chunks per thread and part
    uint32_t wv[2][K / 4];
    const uint4* src = reinterpret_cast<const uint4*>(img.base + img_off);
#pragma unroll
    for (int p = 0; p < 2; ++p)
#pragma unroll
      for (int j = 0; j < NC; ++j) {
        const uint4 q = __ldg(src + (size_t)(p * (K / 8) + hh * NC + j) * 128 + f);
        wv[p][4 * j] = q.x; wv[p][4 * j + 1] = q.y; wv[p][4 * j + 2] = q.z; wv[p][4 * j + 3] = q.w;
      }
#pragma unroll
    for (int p = 0; p < 2; ++p) {
      const uint32_t addr = tmem + col + lane_addr + (uint32_t)(p * (K / 2) + hh * (K / 4));
      if constexpr (K == 128) tmem_st32(addr, wv[p]);
      else tmem_st16(addr, wv[p]);
    }
    tmem_wait_st();
  }

  // ---- tile tables ---------------------------------------------------------------------------------------------------
  __device__ __forceinline__ const uint32_t* tile_ptr(int kind, int tile) const {
    return a.tabs.base + (size_t)(a.tabs.off[kind] + tile) * TC_TILE_WORDS;
  }
  // (valid, group id, slot q) of column c (0..127) given its chunk word
  __device__ __forceinline__ bool col_of(uint32_t cw, int c, int& gid, int& q) const {
    const int u = c & 7;
    const bool valid = (cw & CH_VALID) && u < ch_cnt(cw);
    const int qb = ch_qb(cw);
    if (qb == 0) { gid = ch_gid(cw) + u; q = 0; }       // dense chunk: 8 consecutive groups, primal rows
    else { gid = ch_gid(cw); q = (u == 0) ? 0 : qb + u - 1; }
    return valid;
  }

  // =============================================================================================================
  // The software pipeline shared by the three phases.  P provides
  //   ntiles, NL (layers per tile), kind (tile table), stream (weights streamed layer by layer through two buffers),
  //   side_build (the side warpgroup builds the first operand of every tile and consumes its last accumulator)
  //   prologue()                  before the first tile (epilogue threads; edge phase: epilogue + side threads)
  //   build(s, tile)              epilogue threads: first B operand of the tile            (!side_build)
  //   side_first(s, tile), side_gather(s, tile), side_coords(s, tile), side_meta(s, tile)  (side_build)
  //   epi(s, tile, w)             epilogue threads: consume the accumulator of layer w (and write the next B operand)
  //   wimg(w)                     image offset of the weights of layer w (stream only)
  //   a_col(q, w), K(w)           MMA operand position / depth for layer w at stream position q
  // =============================================================================================================
  template <class P>
  __device__ __forceinline__ void run_phase(P& p) {
    const int ntiles = p.ntiles, NL = p.NL;
    const int npairs = (ntiles + 1) >> 1;
    const int total_q = npairs * NL;
    if (is_epi || (P::side_build && is_side)) p.prologue();
    if (is_epi && p.stream) {
      load_w<128>(p.wimg(0), TC_WCOL);
      if (total_q > 1) load_w<128>(p.wimg(1 % NL), TC_WCOL + 128);
    }
    if constexpr (P::side_build) {
      if (is_epi || is_side) phase_bar();     // per-edge geometry and the cleared accumulators are visible
    }
    if (is_side) {
      if constexpr (P::side_build) {
        // tables run two tiles (per slot) ahead of their use; the gather of tile t + 2 starts as soon as the tensor core
        // has finished reading B[s] for tile t; the coordinate update of tile t fills the time in between
#pragma unroll 1
        for (int t0 = 0; t0 < 2 && t0 < ntiles; ++t0) {
          p.side_meta(tb_of(t0, t0), t0);
          p.side_gather(t0, t0);
          cp_async_wait<0>();
          arrive(B_BUILT, t0);
        }
#pragma unroll 1
        for (int t0 = 2; t0 < 4 && t0 < ntiles; ++t0) p.side_meta(tb_of(t0 & 1, t0), t0);
#pragma unroll 1
        for (int pr = 0; pr < npairs; ++pr) {
          qbeg();
#pragma unroll 1
          for (int s = 0; s < 2; ++s) {        // the operands the epilogue threads will wait for come first
            const int tile = 2 * pr + s, ntile = tile + 2;
            if (tile >= ntiles) continue;
            if (ntile < ntiles) {
              wait_bar(B_BFREE, s);
              qend(P_SIDE_WAIT);
              p.side_gather(s, ntile);
              qend(P_SIDE_GATHER);
              cp_async_wait<0>();
              qend(P_SIDE_CPWAIT);
            }
            // heads[s] of this tile is consumed BEFORE the next tile of the slot is released: the epilogue threads can
            // then never complete a second phase of the barrier (tile + 2) before this wait (an mbarrier parity wait cannot
            // tell phase k from phase k + 2)
            wait_bar(B_HEADS, s);
            qend(P_SIDE_WAIT);
            if (ntile < ntiles) arrive(B_BUILT, s);
          }
#pragma unroll 1
          for (int s = 0; s < 2; ++s) {
            const int tile = 2 * pr + s;
            if (tile >= ntiles) continue;
            p.side_coords(tb_of(s, tile), tile);
            qend(P_SIDE_COORD);
            if (tile + 4 < ntiles) p.side_meta(tb_of(s, tile + 4), tile + 4);      // = this tile's table buffer, free now
            qend(P_SIDE_META);
          }
        }
      }
      return;
    }
    const int first_kind = P::side_build ? B_BUILT : B_READY;
#pragma unroll 1
    for (int s = 0; s < 2; ++s) {
      if (s >= ntiles) continue;
      if (is_epi) {
        if constexpr (!P::side_build) { p.build(s, tb_of(s, s), s); arrive(B_READY, s); }
      } else {
        issue_mma(s, tb_of(s, s), first_kind, p.a_col(0, 0), p.K(0), P::side_build, false);
      }
    }
    int q = 0;
#pragma unroll 1
    for (int pr = 0; pr < npairs; ++pr) {
#pragma unroll 1
      for (int w = 0; w < NL; ++w, ++q) {
#pragma unroll 1
        for (int s = 0; s < 2; ++s) {
          const int tile = 2 * pr + s;
          if (tile >= ntiles) continue;
          const bool last_slot = (s == 1) || (tile + 1 >= ntiles);
          const int ntile = tile + 2;
          const int tb = tb_of(s, tile);
          if (is_epi) {
            // the weights two layers ahead go into the buffer that layer q's MMAs (complete once done[last slot]
            // fires) have been reading
            const bool do_w = p.stream && last_slot && q + 2 < total_q;
#if TC_WPREFETCH
            // fetched into registers before the wait (the L2 latency hides behind it), stored to TMEM after it
            uint32_t wv[2][32];
            if (do_w) fetch_w<128>(p.wimg((w + 2) % NL), wv);
            wait_done(s);
            if (do_w) { qbeg(); store_w<128>(wv, TC_WCOL + 128 * (q & 1)); qend(P_WLOAD); }
#else
            wait_done(s);
            if (do_w) { qbeg(); load_w<128>(p.wimg((w + 2) % NL), TC_WCOL + 128 * (q & 1)); qend(P_WLOAD); }
#endif
            p.epi(s, tb, tile, w);
            if (w < NL - 1) arrive(B_READY, s);
            else if constexpr (P::side_build) arrive(B_HEADS, s);
            else if (ntile < ntiles) { p.build(s, tb_of(s, ntile), ntile); arrive(B_READY, s); }
          } else {
            // the MMAs of layer NL - 1 are the last readers of B[s] for this tile
            // (one B_BFREE commit per tile that has a successor in its slot: the side warps wait for exactly those)
            if (w < NL - 1)
              issue_mma(s, tb, B_READY, p.a_col(q + 1, w + 1), p.K(w + 1), false, P::side_build && w + 1 == NL - 1 && ntile < ntiles);
            else if (ntile < ntiles)
              issue_mma(s, tb_of(s, ntile), first_kind, p.a_col(q + 1, 0), p.K(0), P::side_build, false, P::side_build);
          }
        }
      }
    }
  }

  // column metadata of a node tile (kinds TT_NODE1 / TT_NODE): row offset (node * ND + slot) or -1, chunk words, header
  __device__ __forceinline__ void node_meta(int tb, int kind, int tile) {
    epi_bar();     // every thread is done with the previous contents of this table buffer
    const uint32_t* tp = tile_ptr(kind, tile);
    if (tid < 128) {
#pragma unroll
      for (int sb = 0; sb < SUB; ++sb) {
        const uint32_t cw = __ldg(tp + sb * 16 + (tid >> 3));
        int g, q;
        const bool valid = col_of(cw, tid, g, q);
        TCI(colmrow)[(tb * SUB + sb) * 128 + tid] = valid ? g * ND + q : -1;
      }
    } else if (tid < 128 + 48) {
      const uint32_t w = __ldg(tp + (tid - 128));
      if (tid < 128 + 32) TCW(chw)[tb * 32 + (tid - 128)] = w;
      else TCW(hdr)[tb * 16 + (tid - 160)] = w;
    }
    epi_bar();
  }

  // =============================================================================================================
  // node phase 1: h_in = [h | tau] Wd + bd  (fp32 to hB, pre-split bf16 rows to Himg) ; P_h = h_in Wh0[U:U+H] + bh0
  // =============================================================================================================
  struct NodePre {
    EngineTC& e;
    int b, ntiles, NL, kind;
    static constexpr bool stream = false;
    static constexpr bool side_build = false;
    __device__ __forceinline__ uint32_t a_col(int, int w) const { return TC_WCOL + 64u * w; }
    __device__ __forceinline__ int K(int) const { return KN; }
    __device__ __forceinline__ int wimg(int) const { return 0; }
    __device__ __forceinline__ void prologue() {
      const KernelArgs& a = e.a;
      const EcnfBlockParams& bp = e.m.blk[b];
      const TcImgBlock& ib = e.img.blk[b];
      if (e.tid < H) {
        float cv = bp.bd[e.tid];
        for (int k = 0; k < e.m.T; ++k) cv = fmaf(TCF(tau)[k], bp.Wd[(H + k) * H + e.tid], cv);
        TCF(cvec)[e.tid] = cv;
      }
      e.template load_w<KN>(ib.Wd, TC_WCOL);
      if (NL > 1) e.template load_w<KN>(ib.Wh0h, TC_WCOL + 64);
    }
    __device__ __forceinline__ void build(int s, int tb, int tile) {
      const KernelArgs& a = e.a;
      e.qbeg();
      e.node_meta(tb, kind, tile);
      if (e.fu < H) {
        float v[64];
        const float* src = e.hA() + e.fu;
        const int* ro_ = TCI(colmrow) + (tb * SUB + e.sub) * 128 + 64 * e.hh;
#pragma unroll
        for (int c = 0; c < 64; ++c) {
          const int ro = ro_[c];
          const float x = src[(size_t)(ro >= 0 ? ro : 0) * H];
          v[c] = ro >= 0 ? x : 0.f;
        }
        e.write_B(s, v, e.sub * H + e.fu);
      }
      e.qend(P_NBUILD);
    }
    __device__ __forceinline__ void epi(int s, int tb, int, int w) {
      const KernelArgs& a = e.a;
      const EcnfBlockParams& bp = e.m.blk[b];
      float v[64];
      e.ld_acc(s, v);
      const int* ro_ = TCI(colmrow) + (tb * SUB + e.sub) * 128 + 64 * e.hh;
      if (w == 0) {
        if (e.fu >= H) return;      // lanes beyond the H outputs of h_in
        const float bias = TCF(cvec)[e.fu];
        float* dst = e.hB() + e.fu;
        unsigned char* himg = e.Himg() + 2 * e.fu;
        const bool dense = (kind == TT_NODE1);              // every column a primal row (first block / no divergence)
#pragma unroll
        for (int c = 0; c < 64; ++c) {
          const bool pr = dense || (c & 7) == 0;            // bias on primal columns only
          v[c] += pr ? bias : 0.f;
          const int ro = ro_[c];
          if (ro >= 0) {       // a repeated primal column rewrites the same values
            dst[(size_t)ro * H] = v[c];
            const __nv_bfloat16 hi = __float2bfloat16_rn(v[c]);
            const __nv_bfloat16 lo = __float2bfloat16_rn(v[c] - __bfloat162float(hi));
            *reinterpret_cast<__nv_bfloat16*>(himg + (size_t)ro * ROWB) = hi;
            *reinterpret_cast<__nv_bfloat16*>(himg + (size_t)ro * ROWB + 2 * H) = lo;
          }
        }
        if (NL > 1) e.write_B(s, v, e.sub * H + e.fu);
      } else {
        const float bias = bp.bh[0][e.fu];
        float* dst = e.Ph() + e.fu;
        const bool dense = (kind == TT_NODE1);
#pragma unroll
        for (int c = 0; c < 64; ++c) {
          const bool pr = dense || (c & 7) == 0;
          const int ro = ro_[c];
          if (ro >= 0) dst[(size_t)ro * U] = v[c] + (pr ? bias : 0.f);
        }
      }
    }
  };

  // =============================================================================================================
  // node phase 2: h <- phi_h([M | h_in]) + h_in        (the h_in part of layer 0 is P_h from phase 1)
  // =============================================================================================================
  struct NodePost {
    EngineTC& e;
    int b, ntiles, NL, kind;
    bool htan;
    static constexpr bool stream = true;
    static constexpr bool side_build = false;
    __device__ __forceinline__ uint32_t a_col(int q, int) const { return TC_WCOL + 128u * (q & 1); }
    __device__ __forceinline__ int K(int) const { return 128; }
    __device__ __forceinline__ void prologue() {}
    __device__ __forceinline__ int wimg(int w) const {
      const TcImgBlock& ib = e.img.blk[b];
      const int L = e.m.L;
      return w == 0 ? ib.Wh0m : (w < L ? ib.Wh[w] : ib.WhL);
    }
    __device__ __forceinline__ void build(int s, int tb, int tile) {
      const KernelArgs& a = e.a;
      e.qbeg();
      e.node_meta(tb, kind, tile);
      float v[64];
      const float* src = e.Mg() + e.fu;
      const int* ro_ = TCI(colmrow) + (tb * SUB + e.sub) * 128 + 64 * e.hh;
#pragma unroll
      for (int cb = 0; cb < 64; cb += 16) {
#pragma unroll
        for (int u = 0; u < 16; ++u) {
          const int ro = ro_[cb + u];
          const float x = src[(size_t)(ro >= 0 ? ro : 0) * U];
          v[cb + u] = ro >= 0 ? x : 0.f;
        }
      }
      e.write_B(s, v, e.f);
      e.qend(P_NBUILD);
    }
    __device__ __forceinline__ void epi(int s, int tb, int, int w) {
      const KernelArgs& a = e.a;
      const EcnfBlockParams& bp = e.m.blk[b];
      const int L = e.m.L;
      const int* ro_ = TCI(colmrow) + (tb * SUB + e.sub) * 128 + 64 * e.hh;
      float v[64];
      if (w == 0) {
        const float* ph = e.Ph() + e.fu;
        // + P_h (primal always; tangent columns where h_in carries tangents)
        e.ld_acc(s, v);
#pragma unroll
        for (int cb = 0; cb < 64; cb += 16) {
          float pv[16];
#pragma unroll
          for (int u = 0; u < 16; ++u) {
            const int c = cb + u;
            const bool pr = DIV ? ((c & 7) == 0) : true;
            const int ro = ro_[c];
            const bool use = ro >= 0 && (pr || htan);
            const float x = ph[(size_t)(use ? ro : 0) * U];
            pv[u] = use ? x : 0.f;
          }
#pragma unroll
          for (int u = 0; u < 16; ++u) v[cb + u] += pv[u];
        }
        e.template act_rule<false>(v, 0.f, tb, 0.f);
        e.write_B(s, v, e.f);
      } else if (w < L) {
        const float bias = bp.bh[w][e.fu];
        e.ld_acc(s, v);
        e.template act_rule<false>(v, bias, tb, 0.f);
        e.write_B(s, v, e.f);
      } else {
        if (e.fu >= H) return;
        const float bias = bp.bh[L][e.fu];
        const float* hin = e.hB() + e.fu;
        float* dst = e.hA() + e.fu;
        e.ld_acc(s, v);
#pragma unroll
        for (int cb = 0; cb < 64; cb += 16) {
          float hv[16];
#pragma unroll
          for (int u = 0; u < 16; ++u) {
            const int c = cb + u;
            const bool pr = DIV ? ((c & 7) == 0) : true;
            const int ro = ro_[c];
            const bool use = ro >= 0 && (pr || htan);
            const float x = hin[(size_t)(use ? ro : 0) * H];
            hv[u] = (use ? x : 0.f) + (pr ? bias : 0.f);
          }
#pragma unroll
          for (int u = 0; u < 16; ++u) {
            const int ro = ro_[cb + u];
            if (ro >= 0) dst[(size_t)ro * H] = v[cb + u] + hv[u];
          }
        }
      }
    }
  };

  // =============================================================================================================
  // edge phase: phi_e (layer 0 = MMA on the gathered h_in rows) -> {attention gate + message aggregation,
  //             phi_x -> coordinate update}
  // =============================================================================================================
  struct EdgePh {
    EngineTC& e;
    int b, ntiles, NL, kind;   // kind = tile table (TT_FIRST / TT_MID / TT_LAST / TT_EDGE1)
    bool htan, want_msg;       // want_msg: the aggregated messages feed phi_h (every block but the last)
    float wdf, waf, wpf;       // my feature's entry of w_d (|v|^2 column of phi_e layer 0), attention and head weights
    static constexpr bool stream = true;
    static constexpr bool side_build = true;
    __device__ __forceinline__ uint32_t a_col(int q, int) const { return TC_WCOL + 128u * (q & 1); }
    __device__ __forceinline__ int K(int) const { return 128; }
    __device__ __forceinline__ int ekind() const { return kind == TT_FIRST ? KIND_FIRST : kind == TT_MID ? KIND_MID : KIND_LAST; }   // TT_EDGE1 has no tangent columns: the value is never used
    __device__ __forceinline__ int wimg(int w) const {
      const TcImgBlock& ib = e.img.blk[b];
      const int L = e.m.L;
      return w == 0 ? ib.We0 : (w < L ? ib.We[w] : ib.Wx[w - L]);
    }
    __device__ __forceinline__ void prologue() {      // epilogue + side threads (384)
      const KernelArgs& a = e.a;
      const EcnfBlockParams& bp = e.m.blk[b];
      const int n = e.n, dim = e.dim, D = e.D;
      constexpr int NTH = TC_EPI + TC_SIDE;
      if (e.is_epi) {
        wdf = bp.We[0][(size_t)2 * H * U + e.fu];
        waf = bp.wa[e.fu];
        wpf = bp.wp[e.fu];
      }
      for (int i = e.tid; i < D; i += NTH) { TCF(xacc)[i] = 0.f; TCF(dacc)[i] = 0.f; }
      if (DIV && kind != TT_LAST)
        for (int i = e.tid; i < D * e.ntan; i += NTH) TCF(xtacc)[i] = 0.f;
      if (want_msg)
        for (int i = e.tid; i < 2 * SUB * (a.lay.mrows + 1) * U; i += NTH) TCF(macc)[i] = 0.f;
      // per-edge geometry (egnn.py:73)
      for (int ed = e.tid; ed < e.E; ed += NTH) {
        const int i = ed / (n - 1), jj = ed - i * (n - 1);
        int j = i + 1 + jj; if (j >= n) j -= n;
        float vv[3];
        for (int c = 0; c < 3; ++c) vv[c] = c < dim ? TCF(xs)[i * dim + c] - TCF(xs)[j * dim + c] : 0.f;
        reinterpret_cast<float4*>(TCF(egv))[ed] = make_float4(vv[0], vv[1], vv[2], __int_as_float(i | (j << 8)));
      }
    }
    // (i, j) of an edge, its squared length with the safe rule (numerical.py:7-10)
    __device__ __forceinline__ float4 edge_geo(int ed, int& i, int& j, float& sq) const {
      const KernelArgs& a = e.a;
      const float4 g = reinterpret_cast<const float4*>(TCF(egv))[ed];
      const int ij = __float_as_int(g.w);
      i = ij & 255; j = ij >> 8;
      sq = fmaf(g.z, g.z, fmaf(g.y, g.y, g.x * g.x));
      return g;
    }

    // ---- side warpgroup: one thread per tile column (x SUB sub-tiles) ---------------------------------------------------
    // B operand of phi_e layer 0 for `tile`: [h_in[sender] | h_in[receiver]] rows, K-major, by 16-byte cp.async copies
    __device__ __forceinline__ void side_gather(int s, int tile) {
      const KernelArgs& a = e.a;
      const int n = e.n, ND = e.ND;
      const uint32_t* tp = e.tile_ptr(kind, tile);
      const unsigned char* himg = e.Himg();
#pragma unroll 1
      for (int item = e.tid - TC_EPI; item < SUB * 128; item += TC_SIDE) {
        const int sb = item >> 7, c = item & 127;
        unsigned char* bbase = smem_tc + a.lay.bop + s * TC_BOP + (c >> 3) * (int)TC_SBO_K + (c & 7) * 16;
        const uint32_t cw = __ldg(tp + sb * 16 + (c >> 3));
        int ed, q;
        const bool valid = e.col_of(cw, c, ed, q);
        int rs = n * ND, rr = n * ND;        // the all-zero row
        if (valid && (q == 0 || htan)) {
          const int ij = __float_as_int(TCF(egv)[ed * 4 + 3]);
          const int i = ij & 255, j = ij >> 8;
          const int slot = q == 0 ? 0 : 1 + dirmap(ekind(), q - 1, i, j, e.dim);
          rs = j * ND + slot; rr = i * ND + slot;
        }
        const unsigned char* src_s = himg + (size_t)rs * ROWB;
        const unsigned char* src_r = himg + (size_t)rr * ROWB;
        // K rows of this sub-tile: [sb * 2H, +H) sender features, [sb * 2H + H, +H) receiver features
        unsigned char* d0 = bbase + ((sb * 2 * H) >> 3) * (int)TC_LBO_K;
#pragma unroll
        for (int g = 0; g < H / 8; ++g) {
          cp_async16(d0 + g * (int)TC_LBO_K, src_s + 16 * g);                                   // hi, sender
          cp_async16(d0 + 32768 + g * (int)TC_LBO_K, src_s + 2 * H + 16 * g);                   // lo, sender
          cp_async16(d0 + (H / 8 + g) * (int)TC_LBO_K, src_r + 16 * g);                         // hi, receiver
          cp_async16(d0 + 32768 + (H / 8 + g) * (int)TC_LBO_K, src_r + 2 * H + 16 * g);         // lo, receiver
        }
      }
      cp_async_commit();
    }
    // per-column tables of `tile` for the epilogue threads: |v|^2 (or its tangent), message-accumulator row
    __device__ __forceinline__ void side_meta(int tb, int tile) {
      const KernelArgs& a = e.a;
      const int sc = e.tid - TC_EPI, n = e.n, dim = e.dim, D = e.D, ND = e.ND;
      const uint32_t* tp = e.tile_ptr(kind, tile);
      const int win_i = (int)__ldg(tp + 32 + TH_WIN_I), win_s = (int)__ldg(tp + 32 + TH_WIN_S), win_ns = (int)__ldg(tp + 32 + TH_WIN_NS);
      const int dump = a.lay.mrows * U;
#pragma unroll 1
      for (int item = sc; item < SUB * 128; item += TC_SIDE) {
        const int sb = item >> 7, c = item & 127;
        const uint32_t cw = __ldg(tp + sb * 16 + (c >> 3));
        int ed, q;
        const bool valid = e.col_of(cw, c, ed, q);
        float sd = 0.f;
        int mr = dump;
        if (valid) {
          int i, j; float sq;
          const float4 g = edge_geo(ed, i, j, sq);
          const float gv[3] = {g.x, g.y, g.z};
          const bool isz = (sq == 0.f);
          int gslot = 0;
          if (q == 0) {
            sd = isz ? 1.f : sq;
          } else {
            const int k = dirmap(ekind(), q - 1, i, j, dim);
            gslot = 1 + k;
            float acc = 0.f;
#pragma unroll
            for (int cc = 0; cc < 3; ++cc)
              if (cc < dim) acc = fmaf(gv[cc], TCF(xt)[(i * dim + cc) * e.ntan + k] - TCF(xt)[(j * dim + cc) * e.ntan + k], acc);
            sd = isz ? 0.f : 2.f * acc;
          }
          if (want_msg && !((c & 7) == 0 && DIV && !(cw & CH_OWNER))) {      // a repeated primal column contributes nothing
            if (kind == TT_FIRST) {
              const int u = c & 7;
              if (u <= dim) mr = ((i - win_i) * (1 + dim) + u) * U;
              else mr = -(1 + (i * ND + gslot));                              // per-sender direction: written straight to M
            } else if (kind == TT_EDGE1) {
              mr = i * U;
            } else {
              mr = ((i - win_i) * win_ns + (gslot - win_s)) * U;
            }
          }
        }
        TCF(colsd)[(tb * SUB + sb) * 128 + c] = sd;
        TCI(colmrow)[(tb * SUB + sb) * 128 + c] = mr;
      }
      if (sc < 48) {
        const uint32_t w = __ldg(tp + sc);
        if (sc < 32) TCW(chw)[tb * 32 + sc] = w;
        else TCW(hdr)[tb * 16 + (sc - 32)] = w;
      }
    }
    // coordinate head + coordinate update (egnn.py:82-95) and its tangents, from the head dot products of the tile
    __device__ __forceinline__ void side_coords(int tb, int tile) {
      const KernelArgs& a = e.a;
      const EcnfBlockParams& bp = e.m.blk[b];
      const int sc = e.tid - TC_EPI, n = e.n, dim = e.dim, D = e.D;
      const int ek = ekind();
      const float bpv = bp.bp[0];
      float* cd = TCF(cdbuf);
      const float* pd = TCF(pdh) + tb * 512;
      // stage 1: the contribution of a column to each coordinate of its receiver
#pragma unroll 1
      for (int item = sc; item < SUB * 128; item += TC_SIDE) {
        const int sb = item >> 7, c = item & 127;
        const uint32_t cw = TCW(chw)[tb * 32 + sb * 16 + (c >> 3)];
        int ed, q;
        const bool valid = e.col_of(cw, c, ed, q);
        float val[3] = {0.f, 0.f, 0.f};
        if (valid) {
          int i, j; float sq;
          const float4 g = edge_geo(ed, i, j, sq);
          const float gv[3] = {g.x, g.y, g.z};
          const bool isz = (sq == 0.f);
          const float len = sqrtf(isz ? 1.f : sq), inv = 1.f / (e.m.C + len);
          const int h2 = c >> 6, cl = c & 63;
          if (q == 0) {
            const float pg = e.full_dot(pd, h2, sb, cl) + bpv;
#pragma unroll
            for (int cc = 0; cc < 3; ++cc) val[cc] = pg * gv[cc] * inv;
          } else {
            const int k = dirmap(ek, q - 1, i, j, dim);
            const float pg = e.full_dot(pd, h2, sb, cl & ~7) + bpv, pdv = e.full_dot(pd, h2, sb, cl);
            const float ld = isz ? 0.f : TCF(colsd)[(tb * SUB + sb) * 128 + c] / (2.f * len);
#pragma unroll
            for (int cc = 0; cc < 3; ++cc) {
              if (cc < dim) {
                const float vc = gv[cc];
                const float vd = TCF(xt)[(i * dim + cc) * e.ntan + k] - TCF(xt)[(j * dim + cc) * e.ntan + k];
                val[cc] = (pdv * vc + pg * vd) * inv - pg * vc * ld * inv * inv;
              }
            }
          }
        }
        cd[(sb * 128 + c) * 3] = val[0]; cd[(sb * 128 + c) * 3 + 1] = val[1]; cd[(sb * 128 + c) * 3 + 2] = val[2];
      }
      e.side_bar();
      // stage 2: fixed-order sums over the chunks of a run (the edges of one receiver)
      const int P = e.hdr(tb, TH_P);
      if constexpr (!DIV) {
        const int i_first = e.hdr(tb, TH_IFIRST), i_last = e.hdr(tb, TH_ILAST);
        const int g0 = ch_gid(TCW(chw)[tb * 32]);      // first edge of the tile (dense chunks, chunk p = 8 consecutive edges)
        for (int idx = sc; idx < (i_last - i_first + 1) * dim; idx += TC_SIDE) {
          const int i = i_first + idx / dim, cc = idx % dim;
          const int ea = max(g0, i * (n - 1)), eb = min(g0 + 8 * P, min((i + 1) * (n - 1), e.E));
          float acc = 0.f;
          for (int ed = ea; ed < eb; ++ed) {
            const int lg = ed - g0, pch = lg >> 3;
            const int sb = pch % SUB, col = ((pch / SUB) & 1) * 64 + (pch / (2 * SUB)) * 8 + (lg & 7);
            acc += cd[(sb * 128 + col) * 3 + cc];
          }
          TCF(xacc)[i * dim + cc] += acc;
        }
      } else {
        auto widx = [](int q) { return (q % SUB) * 16 + ((q / SUB) & 1) * 8 + q / (2 * SUB); };
        const int per = 8 * dim;
        if (ek == KIND_FIRST) {      // per-sender directions: one entry per (edge, direction, coordinate), no sum
          const int pp = dim * dim;
#pragma unroll 1
          for (int item = sc; item < P * pp; item += TC_SIDE) {
            const int pch = item / pp, rem = item - pch * pp, u = 1 + dim + rem / dim, cc = rem % dim;
            const uint32_t cw = TCW(chw)[tb * 32 + widx(pch)];
            const int ij = __float_as_int(TCF(egv)[ch_gid(cw) * 4 + 3]);
            const int i = ij & 255, j = ij >> 8;
            const int col = (pch % SUB) * 128 + ((pch / SUB) & 1) * 64 + (pch / (2 * SUB)) * 8 + u;
            TCF(xtacc)[(i * dim + cc) * D + j * dim + (u - 1 - dim)] += cd[col * 3 + cc];
          }
        }
        // one work item per (chunk that ends a run, column position u, coordinate cc): walks back over the run's chunks
        const uint32_t runmask = (uint32_t)e.hdr(tb, TH_RUNMASK);
        const int nruns = __popc(runmask);
#pragma unroll 1
        for (int item = sc; item < nruns * per; item += TC_SIDE) {
          const int ri = item / per, rem = item - ri * per, u = rem / dim, cc = rem - u * dim;
          const int pch = __fns(runmask, 0, ri + 1);
          auto colof = [&](int q) { return (q % SUB) * 128 + ((q / SUB) & 1) * 64 + (q / (2 * SUB)) * 8 + u; };
          const uint32_t cw = TCW(chw)[tb * 32 + widx(pch)];
          if (u >= ch_cnt(cw)) continue;
          const int i = __float_as_int(TCF(egv)[ch_gid(cw) * 4 + 3]) & 255;
          if (ek == KIND_FIRST && u > dim) continue;
          if (u == 0 && !(cw & CH_OWNER)) continue;              // repeated primal columns
          if (ek == KIND_LAST && u > 0 && u - 1 != cc) continue;   // only the Jacobian diagonal is needed in the last block
          float acc = 0.f;
          int q = pch;
          do {
            acc += cd[colof(q) * 3 + cc];
            --q;
          } while (q >= 0 && !(TCW(chw)[tb * 32 + widx(q)] & CH_RUNEND));
          if (u == 0) TCF(xacc)[i * dim + cc] += acc;
          else if (ek == KIND_LAST) TCF(dacc)[i * dim + cc] += acc;
          else TCF(xtacc)[(i * dim + cc) * e.ntan + (ek == KIND_MID ? ch_qb(cw) + u - 2 : i * dim + (u - 1))] += acc;
        }
      }
      e.side_bar();      // cdbuf is rewritten by the next tile
    }

    // ---- epilogue threads ------------------------------------------------------------------------------------------------
    __device__ __forceinline__ void epi(int s, int tb, int tile, int w) {
      const KernelArgs& a = e.a;
      const EcnfBlockParams& bp = e.m.blk[b];
      const int L = e.m.L;
      float v[64];
      e.qbeg();
      if (w == 0) e.wait_bar(B_BUILT, s);      // the side warps' per-column tables of this tile are visible to me
      const float bias = w < L ? bp.be[w][e.fu] : bp.bx[w - L][e.fu];
      {
        uint32_t x[32], y[32];
        e.ld_half_issue(s, 0, x);
        tmem_wait_ld();
        e.ld_half_issue(s, 1, y);         // in flight while the first half is processed
#pragma unroll
        for (int c = 0; c < 32; ++c) v[c] = __uint_as_float(x[c]);
        if (w == 0) e.template act_half<true>(v, 0, bias, tb, wdf);
        else e.template act_half<false>(v, 0, bias, tb, 0.f);
        if (w < NL - 1) e.write_half(s, v, 0, e.f);
        tmem_wait_ld();
#pragma unroll
        for (int c = 0; c < 32; ++c) v[32 + c] = __uint_as_float(y[c]);
      }
      // last layer: acc[s] is drained -- the next tile of this slot (its operand may already be gathered) can start
      if (w == NL - 1 && tile + 2 < ntiles) e.arrive(B_READY, s);
      if (w == 0) e.template act_half<true>(v, 1, bias, tb, wdf);
      else e.template act_half<false>(v, 1, bias, tb, 0.f);
      if (w < NL - 1) {
        e.write_half(s, v, 1, e.f);
        e.qend(P_EPI);
        if (w == L - 1 && want_msg) { messages(s, tb, v); e.qend(P_MSG); }
      } else {
        e.qend(P_EPI);
        e.warp_dot(v, wpf, TCF(pdh) + tb * 512 + e.warp * 64);      // coordinate head partials for the side warps
        e.qend(P_HEAD);
      }
    }
    // attention gate + message aggregation (egnn.py:99-104) from the fp32 phi_e outputs in v
    __device__ __forceinline__ void messages(int s, int tb, const float (&v)[64]) {
      const KernelArgs& a = e.a;
      const EcnfBlockParams& bp = e.m.blk[b];
      const int hh = e.hh, lane = e.lane, warp = e.warp, sub = e.sub;
      const float* pd = TCF(pdot) + s * 512;
      e.warp_dot(v, waf, TCF(pdot) + s * 512 + warp * 64);
      e.half_bar();
      {
        // msg = m e,  msg-dot = m-dot e + m e (1 - e) (m-dot . wa): per column the coefficient of its own value (wA) and of
        // its chunk's primal value (wB); columns that contribute nothing (repeated primal, padding) get zeros
        const float bav = bp.ba[0];
        float aco[2], bco[2];
        const uint32_t cw = e.my_chw(tb, lane >> 2);
        const float raw[2] = {e.full_dot(pd, hh, sub, 2 * lane), e.full_dot(pd, hh, sub, 2 * lane + 1)};
        float eg[2];
        if constexpr (DIV) {      // the gate of the chunk's edge comes from its primal column = first column of lane & ~3
          const float rawp = __shfl_sync(0xffffffffu, raw[0], lane & ~3);
          eg[0] = eg[1] = fast_sigmoid(rawp + bav);
        } else {
          eg[0] = fast_sigmoid(raw[0] + bav);
          eg[1] = fast_sigmoid(raw[1] + bav);
        }
#pragma unroll
        for (int u2 = 0; u2 < 2; ++u2) {
          const int u = (2 * lane + u2) & 7;
          const bool valid = (cw & CH_VALID) && u < ch_cnt(cw);
          const bool prim = !DIV || u == 0;
          aco[u2] = !valid ? 0.f : (prim ? ((!DIV || (cw & CH_OWNER)) ? eg[u2] : 0.f) : eg[u2]);
          bco[u2] = (!valid || prim) ? 0.f : eg[u2] * (1.f - eg[u2]) * raw[u2];
        }
        *reinterpret_cast<float2*>(TCF(wA) + warp * 64 + 2 * lane) = make_float2(aco[0], aco[1]);
        *reinterpret_cast<float2*>(TCF(wB) + warp * 64 + 2 * lane) = make_float2(bco[0], bco[1]);
      }
      __syncwarp();
      const int nc = e.my_nch(tb);
      float* mac = TCF(macc) + (size_t)(hh * SUB + sub) * (a.lay.mrows + 1) * U + e.fu;
      const float* wa_ = TCF(wA) + warp * 64;
      const int* mr_ = TCI(colmrow) + (tb * SUB + sub) * 128 + 64 * hh;
      if constexpr (!DIV) {
        // msg = m e per edge column; the columns of one receiver are consecutive, so a running sum is added to the
        // receiver's accumulator row whenever the row changes (padding columns go to the dump row)
        int cur = mr_[0];
        float acc = 0.f;
#pragma unroll
        for (int c = 0; c < 64; ++c) {
          if (c < 8 * nc) {
            const int mr = mr_[c];
            if (mr != cur) { mac[cur] += acc; acc = 0.f; cur = mr; }
            acc = fmaf(v[c], wa_[c], acc);
          }
        }
        mac[cur] += acc;
      } else {
        const float* wb_ = TCF(wB) + warp * 64;
        const float inv_sqrt_nb = rsqrtf((float)(e.n - 1));
        float2 acc2[4];      // columns (2k, 2k + 1) of the chunk: acc = v wa + (curm wb + acc), per lane as fmaf(v, wa, fmaf(curm, wb, acc))
#pragma unroll
        for (int k = 0; k < 4; ++k) acc2[k] = make_float2(0.f, 0.f);
#pragma unroll
        for (int ch = 0; ch < 8; ++ch) {
          if (ch < nc) {
            const float2 curm = splat2(v[8 * ch]);
            const float4 wa0 = reinterpret_cast<const float4*>(wa_)[2 * ch], wa1 = reinterpret_cast<const float4*>(wa_)[2 * ch + 1];
            const float4 wb0 = reinterpret_cast<const float4*>(wb_)[2 * ch], wb1 = reinterpret_cast<const float4*>(wb_)[2 * ch + 1];
            const float2 wav[4] = {make_float2(wa0.x, wa0.y), make_float2(wa0.z, wa0.w), make_float2(wa1.x, wa1.y), make_float2(wa1.z, wa1.w)};
            const float2 wbv[4] = {make_float2(wb0.x, wb0.y), make_float2(wb0.z, wb0.w), make_float2(wb1.x, wb1.y), make_float2(wb1.z, wb1.w)};
#pragma unroll
            for (int k = 0; k < 4; ++k) acc2[k] = fma2(col2(v, 8 * ch + 2 * k), wav[k], fma2(curm, wbv[k], acc2[k]));
            if (e.my_chw(tb, ch) & CH_GRPEND) {
              // my last chunk of this run: add the run's partial sums to the accumulator rows of its columns (distinct rows;
              // padding shares the dump row); a negative entry is a per-sender row of the first block, stored straight to M
              const int4 ma = reinterpret_cast<const int4*>(mr_)[2 * ch], mb = reinterpret_cast<const int4*>(mr_)[2 * ch + 1];
              const int mr[8] = {ma.x, ma.y, ma.z, ma.w, mb.x, mb.y, mb.z, mb.w};
              float old[8];
#pragma unroll
              for (int u = 0; u < 8; ++u) old[u] = mac[mr[u] >= 0 ? mr[u] : a.lay.mrows * U];
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const float acc[2] = {acc2[k].x, acc2[k].y};
                const float2 sum = add2(make_float2(old[2 * k], old[2 * k + 1]), acc2[k]);
                const float s[2] = {sum.x, sum.y};
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                  const int u = 2 * k + j;
                  if (mr[u] >= 0) mac[mr[u]] = s[j];
                  else e.Mg()[(size_t)(-1 - mr[u]) * U + e.fu] = acc[j] * inv_sqrt_nb;
                }
                acc2[k] = make_float2(0.f, 0.f);
              }
            }
          }
        }
      }
      if (e.hdr(tb, TH_FLUSH)) {
        // the window is complete: write its aggregate to global (coalesced) and clear the accumulators
        e.epi_bar();
        const int win_i = e.hdr(tb, TH_WIN_I), win_nr = e.hdr(tb, TH_WIN_NR), win_s = e.hdr(tb, TH_WIN_S), win_ns = e.hdr(tb, TH_WIN_NS);
        const float inv_sqrt_nb = rsqrtf((float)(e.n - 1));
        const size_t cstride = (size_t)(a.lay.mrows + 1) * U;
        float* m0p = TCF(macc) + e.fu;
        constexpr int RG = TC_EPI / U;       // row groups handled in parallel
        for (int wi = 0; wi < win_nr; ++wi) {
          const int i = win_i + wi;
          for (int ws = e.tid / U; ws < win_ns; ws += RG) {
            const int rr = wi * win_ns + ws;
            const int gslot = (kind == TT_FIRST) ? (ws == 0 ? 0 : 1 + i * e.dim + (ws - 1)) : win_s + ws;
            float sum = 0.f;
#pragma unroll
            for (int cp = 0; cp < 2 * SUB; ++cp) { sum += m0p[cp * cstride + rr * U]; m0p[cp * cstride + rr * U] = 0.f; }
            e.Mg()[((size_t)i * e.ND + gslot) * U + e.fu] = sum * inv_sqrt_nb;
          }
        }
        e.epi_bar();
      }
    }
  };

  // ---- one evaluation of (f, div f) at time t for the positions in xin (shared memory, D floats) ----
  __device__ __forceinline__ void eval(float t, const float* xin, const int32_t* feat, float* fout) {
    if (is_epi) {
      if (tid < dim) {
        float s = 0.f;
        for (int i = 0; i < n; ++i) s += xin[i * dim + tid];
        TCF(mu)[tid] = s / (float)n;
      }
      if (tid >= 32 && tid < 32 + m.T / 2) {
        const int k = tid - 32;
        const float arg = (t * 1000.f) * m.freqs[k];
        TCF(tau)[k] = sinf(arg);
        TCF(tau)[k + m.T / 2] = cosf(arg);
      }
      epi_bar();
      for (int i = tid; i < D; i += TC_EPI) {
        const float v = xin[i] - TCF(mu)[i % dim];
        TCF(xs)[i] = v;
        TCF(xs0)[i] = v;
      }
      const float invn = 1.f / (float)n;
      if constexpr (DIV) {
        if (hutch) {
          // tangent of the centred positions in the probe direction: eps - mean_nodes(eps)
          for (int i = tid; i < D; i += TC_EPI) {
            float mean = 0.f;
            for (int node = 0; node < n; ++node) mean += eps_g[node * dim + i % dim];
            TCF(xt)[i] = eps_g[i] - mean * invn;
          }
        } else {
          for (int idx = tid; idx < D * D; idx += TC_EPI) {
            const int ra = idx / D, k = idx - ra * D;
            const int ia = ra / dim, ca = ra - ia * dim, ik = k / dim, ck = k - ik * dim;
            TCF(xt)[idx] = (ca == ck) ? ((ia == ik ? 1.f : 0.f) - invn) : 0.f;
          }
        }
      }
      float* h0 = hA();
      for (int idx = tid; idx < n * H; idx += TC_EPI) {
        const int node = idx / H, col = idx - node * H;
        int ft = feat[node];
        ft = max(0, min(m.nfeat - 1, ft));
        h0[(size_t)node * ND * H + col] = m.embed[ft * H + col];
      }
      epi_bar();
    }
#pragma unroll 1
    for (int b = 0; b < m.nblocks; ++b) {
      const bool last = (b == m.nblocks - 1);
      const bool htan = DIV && b > 0;
      const int ekind = !DIV ? TT_EDGE1 : hutch ? TT_MID : last ? TT_LAST : (b == 0 ? TT_FIRST : TT_MID);
      const int nkind = DIV ? TT_NODE : TT_NODE1;
      pbeg();
      if (!is_side) {
        const int kind = htan ? TT_NODE : TT_NODE1;
        NodePre p{*this, b, a.tabs.cnt[kind], last ? 1 : 2, kind};
        run_phase(p);
      }
      if (is_epi || is_side) phase_bar();     // h_in (fp32 and pre-split rows) / P_h of every node are in global memory
      pend(P_NODE_PRE);
      {
        EdgePh p{*this, b, a.tabs.cnt[ekind], 2 * m.L, ekind, htan, !last, 0.f, 0.f, 0.f};
        run_phase(p);
      }
      if (is_epi || is_side) phase_bar();     // coordinate accumulators and aggregated messages complete
      pend(P_EDGE);
      if (!last && !is_side) {
        NodePost p{*this, b, a.tabs.cnt[nkind], m.L + 1, nkind, htan};
        run_phase(p);
      }
      if (is_epi) {
        epi_bar();
        const float invnb = 1.f / (float)(n - 1);
        for (int i = tid; i < D; i += TC_EPI) TCF(xs)[i] += TCF(xacc)[i] * invnb;
        if (DIV && (!last || hutch))
          for (int i = tid; i < D * ntan; i += TC_EPI) TCF(xt)[i] += TCF(xtacc)[i] * invnb;
      }
      if (is_epi || is_side) phase_bar();
      pend(P_NODE_POST);
    }
    if (is_epi) {
      const float fs = m.final_scaling[0];
      for (int i = tid; i < D; i += TC_EPI) fout[i] = (TCF(xs)[i] - TCF(xs0)[i] - TCF(mu)[i % dim]) * fs;
      if (DIV && tid == 0) {
        float s = 0.f;
        if (hutch) {
          // eps . (J eps): the output tangent is fs (x_L-dot - x0-dot - mean(eps)) = fs (xt - eps)   (egnn.py:183-188)
          for (int d = 0; d < D; ++d) s = fmaf(eps_g[d], TCF(xt)[d] - eps_g[d], s);
          fout[D] = fs * s;
        } else {
          const float invnb = 1.f / (float)(n - 1);
          for (int d = 0; d < D; ++d) s += TCF(xt)[d * D + d] + TCF(dacc)[d] * invnb;
          fout[D] = fs * (s - (float)D);
        }
      }
    }
    __syncthreads();
  }
};

template <int U, int H, bool DIV, bool SAVE>
__global__ void __launch_bounds__(TC_NT, 1) ecnf_solve_tc_kernel(const __grid_constant__ KernelArgs a) {
  __shared__ long long s_traj;
  __shared__ float s_ctl[8];
  EngineTC<U, H, DIV> eng(a);
  solve_body<EngineTC<U, H, DIV>, DIV, SAVE>(a, eng, s_traj, s_ctl);
  eng.finish(reinterpret_cast<long long*>(reinterpret_cast<char*>(a.counter) + 64));
}

// ---- weight images: fp32 [K][N] (flax kernel) -> bf16 hi | lo over 128 TMEM lanes, block-diagonal over `nsub` sub-tiles
// (lane = sub * lane_stride + out feature, k = sub * ksub + in feature; zero elsewhere), two consecutive k per 32-bit
// word, 4 words per 16-byte chunk:  uint4 index = (part * K/8 + chunk) * 128 + lane,  K = nsub * ksub ---------------------
struct TcPrepItem {
  int src_off;   // floats, into the parameter buffer
  int dst_off;   // bytes, into the image buffer
  int ksub, N;   // rows / columns of the source matrix
  int nsub, lane_stride;
};
constexpr int TC_PREP_MAX = 64;   // items per tc_prep_kernel launch (the list is a by-value kernel parameter)
struct TcPrepList {
  int count;
  TcPrepItem item[TC_PREP_MAX];
};

__global__ void tc_prep_kernel(const float* __restrict__ params, unsigned char* __restrict__ image, const TcPrepList list) {
  const TcPrepItem it = list.item[blockIdx.y];
  uint32_t* dst = reinterpret_cast<uint32_t*>(image + it.dst_off);
  const int K = it.nsub * it.ksub;
  const int words = K / 2;                 // per lane and part
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < 128 * words; idx += gridDim.x * blockDim.x) {
    const int wd = idx / 128, lane = idx - wd * 128;
    const int sl = lane / it.lane_stride, o = lane - sl * it.lane_stride;
    const int k0 = 2 * wd, sk = k0 / it.ksub, kk = k0 - sk * it.ksub;      // ksub is even: both k of a word share a sub-tile
    float x0 = 0.f, x1 = 0.f;
    if (sl == sk && sl < it.nsub && o < it.N) {
      x0 = params[it.src_off + (size_t)kk * it.N + o];
      x1 = params[it.src_off + (size_t)(kk + 1) * it.N + o];
    }
    uint32_t h, l;
    split_pack(x0, x1, h, l);
    const size_t oo = ((size_t)(wd >> 2) * 128 + lane) * 4 + (wd & 3);
    dst[oo] = h;
    dst[(size_t)(K / 8) * 128 * 4 + oo] = l;
  }
}

// one CTA per table kind (a single thread packs: the work is sequential), the current tile staged in shared memory
__global__ void tc_tables_kernel(uint32_t* __restrict__ out, int n, int dim, int SUB, int MR, int ntan, TcTabs tabs) {
  __shared__ uint32_t stage[TC_TILE_WORDS];
  const int k = blockIdx.x;
  if (threadIdx.x == 0 && k < TT_COUNT) tc_pack(k, n, dim, SUB, MR, out + (size_t)tabs.off[k] * TC_TILE_WORDS, ntan, stage);
}

#undef TCF
#undef TCI
#undef TCW

}  // namespace ecnf_solve_detail
