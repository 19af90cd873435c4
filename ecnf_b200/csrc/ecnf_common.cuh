// Shared declarations for the ecnf_b200 CUDA library (sm_100a).
//
// The library replaces the reference's Python/JAX hot path (ecnf/cnf/*.py, ecnf/nets/egnn.py) -- see
// include/ecnf_b200.h for the C-ABI and DESIGN.md for the kernel map.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/ecnf_b200.h"

#define ECNF_MAX_BLOCKS 8
#define ECNF_MAX_LAYERS 6
#define ECNF_MAX_T 16
#define ECNF_MAX_NODES 32

// Device view of one EGCL block's parameters (ecnf/nets/egnn.py:38-47,83-85,99,166-167).
struct EcnfBlockParams {
  const float *Wd, *bd;                                          // Dense_b   [(H+T) x H], [H]
  const float *We[ECNF_MAX_LAYERS], *be[ECNF_MAX_LAYERS];        // phi_e     l=0: [(2H+1) x U]
  const float *Wx[ECNF_MAX_LAYERS], *bx[ECNF_MAX_LAYERS];        // phi_x_torso
  const float *Wh[ECNF_MAX_LAYERS + 1], *bh[ECNF_MAX_LAYERS + 1];  // phi_h     l=0: [(U+H) x U], last [U x H]
  const float *wp, *bp, *wa, *ba;                                // phi_x head (Dense_0), attention (Dense_1)
};

// Passed by value to kernels (< 4 KB).
struct EcnfModelDev {
  int n, dim, H, T, U, L, nblocks, nfeat;
  float C;           // normalization_constant (egnn.py:127)
  float base_scale;  // build_cnf.py:48
  float sigma_min;   // core.py:35-39
  float freqs[ECNF_MAX_T / 2];  // fp32 timestep frequencies (build_cnf.py:25-27), computed on the host
  const float* embed;           // [nfeat x H]
  const float* final_scaling;   // []
  EcnfBlockParams blk[ECNF_MAX_BLOCKS];
};

// Offsets (in floats) of every tensor inside the flat, 16-byte-aligned parameter buffer.
struct EcnfBlockOffsets {
  int64_t Wd, bd, We[ECNF_MAX_LAYERS], be[ECNF_MAX_LAYERS], Wx[ECNF_MAX_LAYERS], bx[ECNF_MAX_LAYERS],
      Wh[ECNF_MAX_LAYERS + 1], bh[ECNF_MAX_LAYERS + 1], wp, bp, wa, ba;
};

struct ecnf_model {
  ecnf_config cfg;
  int64_t param_count;  // floats, padding included
  int64_t embed_off, final_scaling_off;
  EcnfBlockOffsets off[ECNF_MAX_BLOCKS];
  const float* d_params;
  int num_sms;
  int device;
  int engine;   // ecnf_model_set_engine: 0 = tensor cores where eligible, 1 = fp32 SIMT everywhere
  int64_t fm_chunk;   // ecnf_model_set_fm_chunk: graphs per chunk of a training minibatch, 0 = the whole minibatch
};

EcnfModelDev ecnf_make_dev(const ecnf_model* m, const float* d_params);
void ecnf_set_error(const char* fmt, ...);

#define ECNF_CHECK_CUDA(expr)                                                              \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      ecnf_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return ECNF_ERR_CUDA;                                                                \
    }                                                                                      \
  } while (0)

__device__ __forceinline__ float ecnf_sigmoid(float z) { return 1.0f / (1.0f + expf(-z)); }

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}
