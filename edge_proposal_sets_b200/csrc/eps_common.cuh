// Shared helpers for libeps_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/eps.h"

namespace eps {

void set_error(const char *fmt, ...);
int sm_count();

#define EPS_CHECK_ARG(cond, msg)                      \
  do {                                                \
    if (!(cond)) {                                    \
      eps::set_error("%s: %s", __func__, msg);        \
      return EPS_ERR_INVALID;                         \
    }                                                 \
  } while (0)

#define EPS_CUDA(call)                                                              \
  do {                                                                              \
    cudaError_t e__ = (call);                                                       \
    if (e__ != cudaSuccess) {                                                       \
      eps::set_error("%s: %s -> %s", __func__, #call, cudaGetErrorString(e__));     \
      return EPS_ERR_CUDA;                                                          \
    }                                                                               \
  } while (0)

#define EPS_LAUNCH_CHECK()                                                          \
  do {                                                                              \
    cudaError_t e__ = cudaGetLastError();                                           \
    if (e__ != cudaSuccess) {                                                       \
      eps::set_error("%s: launch failed -> %s", __func__, cudaGetErrorString(e__)); \
      return EPS_ERR_CUDA;                                                          \
    }                                                                               \
  } while (0)

constexpr unsigned FULL = 0xffffffffu;

constexpr int EPS_MAX_MLP_LAYERS = 8;
struct MlpParams {  // device pointers, passed to kernels by value
  const float *W[EPS_MAX_MLP_LAYERS];
  const float *b[EPS_MAX_MLP_LAYERS];
};
int linkpred_fp32_launch(const float *h, int H, const int *pu, const int *pv, long long M,
                         const MlpParams &prm, int L, int apply_sigmoid, float *score,
                         cudaStream_t stream);
int linkpred_tc_launch(const float *h, int n, int H, const int *pu, const int *pv, long long M,
                       const MlpParams &prm, int L, int apply_sigmoid, float *score, void *workspace,
                       size_t workspace_bytes, bool prepared, cudaStream_t stream);
size_t linkpred_tc_workspace_bytes(int n, int H, int L, long long M);
bool linkpred_tc_uses_table(int n, long long M);

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ float sigmoidf_ref(float x) {
  // torch.sigmoid in fp32: 1 / (1 + exp(-x))
  return __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-x)));
}

// ---- exact pair-score accumulation (K3 and the fused K6+K3 kernel) ----
// A term t (fp32) becomes the signed 64-bit integer RN(t * 2^EPS_FX_FRAC_BITS); sums of terms are
// integer sums (order-independent, usable with atomics) and the score is the correctly rounded fp32
// value of that sum.  Terms with |t| >= 2^-15 are represented exactly (fp32 ulp >= 2^-38), smaller
// ones carry <= 2^-39 absolute error each; |sum| must stay below 2^25 (n < 2^24 ids, AA terms <= 1.45).
constexpr int EPS_FX_FRAC_BITS = 38;
__device__ __forceinline__ unsigned long long to_fixed(float t) {
  return (unsigned long long)__float2ll_rn(t * 274877906944.0f /* 2^38, exact scaling */);
}
__device__ __forceinline__ float from_fixed(unsigned long long s) {
  return __ll2float_rn((long long)s) * 3.637978807091713e-12f /* 2^-38 */;
}

// ---- degree-normalised similarity scores (include/eps.h, EPS_SCORE_*) ----
__host__ __device__ constexpr int score_kind(int flags) { return (flags & EPS_SCORE_KIND_MASK) >> EPS_SCORE_KIND_SHIFT; }
constexpr int SK_JACCARD = score_kind(EPS_SCORE_JACCARD), SK_SORENSEN = score_kind(EPS_SCORE_SORENSEN),
              SK_SALTON = score_kind(EPS_SCORE_SALTON), SK_HUB_PROMOTED = score_kind(EPS_SCORE_HUB_PROMOTED),
              SK_LHN = score_kind(EPS_SCORE_LHN), SK_PREF_ATTACH = score_kind(EPS_SCORE_PREF_ATTACH);

// KIND = score_kind(flags), 1..7 (0 = the kernel's own CN / AA / RA score, which never reaches here).
// c = exact common-neighbour count, a = deg u, b = deg v.  a + b < 2^24 (host check), so every integer below is exact in
// fp32 and the fp32 divisions are the correctly rounded quotients.  A zero denominator gives 0.
template <int KIND>
__device__ __forceinline__ float similarity_score(int c, int a, int b) {
  if (KIND == SK_PREF_ATTACH) return __ll2float_rn((long long)a * (long long)b);
  if (KIND == SK_SALTON || KIND == SK_LHN) {
    const double ab = (double)a * (double)b;                   // exact: < 2^48
    if (ab == 0.0) return 0.f;
    return (float)((double)c / (KIND == SK_SALTON ? sqrt(ab) : ab));
  }
  int num = c, den;
  if (KIND == SK_JACCARD) den = a + b - c;
  else if (KIND == SK_SORENSEN) { num = 2 * c; den = a + b; }
  else if (KIND == SK_HUB_PROMOTED) den = min(a, b);
  else den = max(a, b);                                         // EPS_SCORE_HUB_DEPRESSED
  return den == 0 ? 0.f : __fdiv_rn((float)num, (float)den);
}

// streaming (read-once) loads that do not pollute L1
__device__ __forceinline__ int ld_stream_s32(const int *p) {
  int r;
  asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(r) : "l"(p));
  return r;
}

}  // namespace eps
