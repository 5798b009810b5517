// K3 — Common-Neighbour / Adamic-Adar / Resource-Allocation pair scoring on sorted CSR.
//
// Replaces /root/reference/models.py:536-554 (index_select + sparse*sparse mul + sparse sum)
// and /root/reference/adamic_utils.py:20-23 (scipy row-index, csr_elmul_csr, row sum).
//
// Two kernels, identical results.  Every per-neighbour term t_k (an fp32 value: w_k, or
// a_u * (a_v * w_k) on weighted graphs) is converted to 64-bit fixed point with EPS_FX_FRAC_BITS
// fractional bits and the terms of a pair are added as INTEGERS, so a score is the correctly
// rounded fp32 value of the exact sum  RN_fp32(sum_k t_k)  — a function of (graph, u, v) alone,
// never of summation order, batch composition, grid size or GPU count, and bit-identical to the
// fused enumeration+scoring kernel (twohop_score.cu), which reaches the same sums through atomics.
// (terms >= 2^-16 are exact in fixed point; smaller ones carry <= 2^-40 absolute error each):
//
//  cn_grouped_kernel   the filter hot path.  Candidates arrive in the reference's column-major
//                      order (filter.py:96-109), i.e. long runs of equal v.  One CTA owns a tile
//                      of consecutive pairs; for every run it turns N(v) into a bitmap in shared
//                      memory once, then its warps stream the N(u) lists of 32 candidates at a
//                      time as ONE flattened, fully coalesced sequence (degree skew inside the
//                      32 lists costs nothing) and probe the bitmap: one 4-byte read of `col`
//                      and one shared-memory bit test per neighbour.
//  cn_pairs_kernel     arbitrary pair lists and weighted graphs (collab): an 8-lane group per
//                      pair walks the shorter list and binary-searches the longer one.
#include "eps_common.cuh"

namespace eps {

constexpr int CN_THREADS = 512;
constexpr int CN_TILE_PAIRS = 1024;
constexpr size_t CN_MAX_BITMAP_BYTES = 200 * 1024;

// One warp scores 32 candidates (u_lane, v) against the bitmap of N(v).
//  phase A  every list with >= CN_LONG neighbours is streamed by the whole warp, aligned to the
//           list start, four 128-byte loads in flight per lane: one LDG + one shared-memory bit test
//           + ballot/popc per 32 neighbours;
//  phase B  the remaining short lists are walked as ONE flattened sequence (lane -> owner list by a
//           shuffle binary search over the inclusive length prefix), so 32 lists of 3 neighbours cost
//           3 iterations, not 32.
// In both phases the weighted terms of a pair are added as 64-bit fixed-point integers: the score
// never depends on which phase handled the list or in which order the terms arrived.
constexpr int CN_LONG = 64;

// KIND != 0: a similarity score (EPS_SCORE_*) of the exact count, deg u (= len) and deg v (= *dv, in shared memory: a
// register live across the walk spills) replaces the CN score.
template <bool HAS_W, int KIND>
__device__ __forceinline__ void grouped_batch(const int *__restrict__ rowptr,
                                              const int *__restrict__ col,
                                              const float *__restrict__ wtable,
                                              const uint32_t *bitmap, const int *__restrict__ pu,
                                              long long base, int cnt, int flags, const int *dv,
                                              float *__restrict__ score, int *__restrict__ count) {
  const int lane = lane_id();
  const bool valid = lane < cnt;
  int s = 0, len = 0;
  if (valid) {
    const int u = pu[base + lane];
    s = __ldg(rowptr + u);
    len = __ldg(rowptr + u + 1) - s;
  }
  int c_acc = 0;
  unsigned long long a_acc = 0ull;
  // ---------------- phase A: long lists, one at a time, warp-wide ----------------
  unsigned longmask = __ballot_sync(FULL, len >= CN_LONG);
  while (longmask) {
    const int b = __ffs(longmask) - 1;
    longmask &= longmask - 1;
    const int sb = __shfl_sync(FULL, s, b);
    const int lb = __shfl_sync(FULL, len, b);
    const int *__restrict__ lp = col + sb;
    int c = 0;
    unsigned long long a = 0ull;      // this lane's share of the list's fixed-point sum
    for (int off = 0; off < lb; off += 128) {
      int k[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int p = off + q * 32 + lane;
        k[q] = p < lb ? __ldg(lp + p) : -1;
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const bool hit = k[q] >= 0 && ((bitmap[k[q] >> 5] >> (k[q] & 31)) & 1u);
        unsigned hm = __ballot_sync(FULL, hit);
        c += __popc(hm);
        if (HAS_W && hit) a += to_fixed(__ldg(wtable + k[q]));
      }
    }
    if (HAS_W) {
#pragma unroll
      for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(FULL, a, o);   // exact: integer adds commute
    }
    if (lane == b) { c_acc = c; a_acc = a; }
  }
  // ---------------- phase B: short lists, flattened ----------------
  const int slen = len >= CN_LONG ? 0 : len;
  int pin = slen;  // inclusive prefix of the short-list lengths
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    int t = __shfl_up_sync(FULL, pin, d);
    if (lane >= d) pin += t;
  }
  const int pex = pin - slen;
  const int total = __shfl_sync(FULL, pin, 31);
  for (int j = 0; j < total; j += 32) {
    const int p = j + lane;
    // owner slot of flattened position p = #lists that end at or before p
    int lo = 0;
#pragma unroll
    for (int step = 16; step >= 1; step >>= 1) {
      int t = __shfl_sync(FULL, pin, lo + step - 1);
      if (t <= p) lo += step;
    }
    const int s_t = __shfl_sync(FULL, s, lo);
    const int pe_t = __shfl_sync(FULL, pex, lo);
    const bool in = p < total;
    int k = 0;
    if (in) k = __ldg(col + s_t + (p - pe_t));
    const bool hit = in && ((bitmap[k >> 5] >> (k & 31)) & 1u);
    const unsigned hm = __ballot_sync(FULL, hit);
    if (hm == 0) continue;  // warp-uniform
    // bits of this chunk that belong to the list owned by this lane
    const int lo_b = min(max(pex - j, 0), 32);
    const int hi_b = min(max(pin - j, 0), 32);
    unsigned segmask = 0;
    if (hi_b > lo_b) {
      const unsigned hi_m = hi_b >= 32 ? 0xffffffffu : ((1u << hi_b) - 1u);
      segmask = hi_m & ~((1u << lo_b) - 1u);
    }
    unsigned m = hm & segmask;
    c_acc += __popc(m);
    if (HAS_W) {
      const unsigned long long w = hit ? to_fixed(__ldg(wtable + k)) : 0ull;
      while (__any_sync(FULL, m != 0)) {
        const int b = m ? (__ffs(m) - 1) : 0;
        const unsigned long long t = __shfl_sync(FULL, w, b);
        if (m) {
          a_acc += t;
          m &= m - 1;
        }
      }
    }
  }
  if (valid) {
    if (count) count[base + lane] = c_acc;
    if (score) {
      float sc;
      if (KIND) {
        sc = similarity_score<KIND>(c_acc, len, *dv);
      } else {
        sc = HAS_W ? from_fixed(a_acc) : (float)c_acc;
        if (flags & EPS_CN_SIGMOID) sc = sigmoidf_ref(sc);
      }
      score[base + lane] = sc;
    }
  }
}

template <bool HAS_W, int KIND = 0>
__global__ void __launch_bounds__(CN_THREADS)
cn_grouped_kernel(const int *__restrict__ rowptr, const int *__restrict__ col,
                  const float *__restrict__ wtable, int n, const int *__restrict__ pu,
                  const int *__restrict__ pv, long long M, int flags, float *__restrict__ score,
                  int *__restrict__ count, unsigned long long *tile_counter) {
  extern __shared__ uint32_t bitmap[];
  __shared__ long long s_tile;
  __shared__ long long s_end;
  __shared__ int s_dv;               // deg v of the current run (similarity kinds)
  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int nwarps = CN_THREADS / 32;
  const int words = (n + 31) >> 5;
  for (int w = tid; w < words; w += CN_THREADS) bitmap[w] = 0;
  const long long ntiles = (M + CN_TILE_PAIRS - 1) / CN_TILE_PAIRS;
  for (;;) {
    __syncthreads();  // bitmap zeroed / previous tile fully done
    if (tid == 0) s_tile = (long long)atomicAdd(tile_counter, 1ull);
    __syncthreads();
    const long long tile = s_tile;
    if (tile >= ntiles) break;
    const long long i1 = min(M, (tile + 1) * CN_TILE_PAIRS);
    long long i = tile * CN_TILE_PAIRS;
    while (i < i1) {
      const int v = pv[i];
      // end of the run of equal v (robust to any input order)
      long long j = i + 1;
      for (;;) {
        if (j >= i1) { j = i1; break; }
        if (tid == 0) s_end = i1;
        __syncthreads();
        const long long idx = j + tid;
        if (idx < i1 && pv[idx] != v) atomicMin((unsigned long long *)&s_end, (unsigned long long)idx);
        __syncthreads();
        const long long e = s_end;
        __syncthreads();
        if (e < i1 || j + CN_THREADS >= i1) { j = e; break; }
        j += CN_THREADS;
      }
      const int vs = __ldg(rowptr + v), ve = __ldg(rowptr + v + 1);
      if (KIND && tid == 0) s_dv = ve - vs;            // read after the barrier below
      for (int p = vs + tid; p < ve; p += CN_THREADS) {
        const int k = __ldg(col + p);
        atomicOr(&bitmap[k >> 5], 1u << (k & 31));
      }
      __syncthreads();
      for (long long base = i + (long long)warp * 32; base < j; base += (long long)nwarps * 32) {
        const int cnt = (int)min((long long)32, j - base);
        grouped_batch<HAS_W, KIND>(rowptr, col, wtable, bitmap, pu, base, cnt, flags, &s_dv, score, count);
      }
      __syncthreads();
      for (int p = vs + tid; p < ve; p += CN_THREADS) bitmap[__ldg(col + p) >> 5] = 0;
      __syncthreads();
      i = j;
    }
  }
}

constexpr int PAIR_G = 8;

template <bool HAS_VAL, bool HAS_W, int KIND = 0>
__global__ void __launch_bounds__(256)
cn_pairs_kernel(const int *__restrict__ rowptr, const int *__restrict__ col,
                const float *__restrict__ val, const float *__restrict__ wtable,
                const int *__restrict__ pu, const int *__restrict__ pv, long long M, int flags,
                float *__restrict__ score, int *__restrict__ count) {
  const int gl = threadIdx.x % PAIR_G;
  const int lane = lane_id();
  const unsigned gmask = ((1u << PAIR_G) - 1u) << ((lane / PAIR_G) * PAIR_G);
  const int gbase = (lane / PAIR_G) * PAIR_G;
  const long long ngroups = (long long)gridDim.x * (blockDim.x / PAIR_G);
  for (long long pair = (long long)blockIdx.x * (blockDim.x / PAIR_G) + threadIdx.x / PAIR_G;
       pair < M; pair += ngroups) {
    const int u = pu[pair], v = pv[pair];
    const int su = __ldg(rowptr + u), lu = __ldg(rowptr + u + 1) - su;
    const int sv = __ldg(rowptr + v), lv = __ldg(rowptr + v + 1) - sv;
    const bool swp = lv < lu;  // walk the shorter list, search the longer one
    const int sa = swp ? sv : su, la = swp ? lv : lu;
    const int sb = swp ? su : sv, lb = swp ? lu : lv;
    int c_acc = 0;
    unsigned long long a_acc = 0ull;
    int hint = 0;
    for (int j = 0; j < la; j += PAIR_G) {
      const int p = j + gl;
      const bool in = p < la;
      int lo = lb;
      int ka = 0;
      if (in) {
        ka = __ldg(col + sa + p);
        lo = hint;
        int hi = lb;
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (__ldg(col + sb + mid) < ka) lo = mid + 1; else hi = mid;
        }
      }
      const bool hit = in && lo < lb && __ldg(col + sb + lo) == ka;
      const unsigned hm = __ballot_sync(gmask, hit) & gmask;
      hint = __shfl_sync(gmask, lo, gbase + PAIR_G - 1);
      c_acc += __popc(hm);
      if (HAS_VAL || HAS_W) {
        float term = 0.f;
        if (hit) {
          const float w = HAS_W ? __ldg(wtable + ka) : 1.f;
          if (HAS_VAL) {
            const float xa = __ldg(val + sa + p), xb = __ldg(val + sb + lo);
            const float a_u = swp ? xb : xa, a_v = swp ? xa : xb;
            term = HAS_W ? __fmul_rn(a_u, __fmul_rn(a_v, w)) : __fmul_rn(a_u, a_v);
          } else {
            term = w;
          }
        }
        unsigned long long fx = hit ? to_fixed(term) : 0ull;
        if (hm) {  // uniform inside the 8-lane group; exact integer sum of the group's terms
#pragma unroll
          for (int o = PAIR_G / 2; o; o >>= 1) fx += __shfl_xor_sync(gmask, fx, o);
          a_acc += fx;
        }
      }
    }
    if (gl == 0) {
      if (count) count[pair] = c_acc;
      if (score) {
        float sc;
        if (KIND) {
          sc = similarity_score<KIND>(c_acc, lu, lv);
        } else {
          sc = (HAS_VAL || HAS_W) ? from_fixed(a_acc) : (float)c_acc;
          if (flags & EPS_CN_SIGMOID) sc = sigmoidf_ref(sc);
        }
        score[pair] = sc;
      }
    }
  }
}

using GroupedKernel = void (*)(const int *, const int *, const float *, int, const int *, const int *, long long, int,
                               float *, int *, unsigned long long *);
using PairsKernel = void (*)(const int *, const int *, const float *, const float *, const int *, const int *,
                             long long, int, float *, int *);
// index = similarity kind (EPS_SCORE_* >> EPS_SCORE_KIND_SHIFT); entry 0 is never used
static const GroupedKernel kGroupedKinds[8] = {
    cn_grouped_kernel<false, 0>, cn_grouped_kernel<false, 1>, cn_grouped_kernel<false, 2>, cn_grouped_kernel<false, 3>,
    cn_grouped_kernel<false, 4>, cn_grouped_kernel<false, 5>, cn_grouped_kernel<false, 6>, cn_grouped_kernel<false, 7>};
static const PairsKernel kPairsKinds[8] = {
    cn_pairs_kernel<false, false, 0>, cn_pairs_kernel<false, false, 1>, cn_pairs_kernel<false, false, 2>,
    cn_pairs_kernel<false, false, 3>, cn_pairs_kernel<false, false, 4>, cn_pairs_kernel<false, false, 5>,
    cn_pairs_kernel<false, false, 6>, cn_pairs_kernel<false, false, 7>};

}  // namespace eps

extern "C" size_t eps_cn_aa_workspace_bytes(void) { return 256; }

extern "C" int eps_cn_aa(const int32_t *rowptr, const int32_t *col, const float *val,
                         const float *wtable, int32_t n, const int32_t *pair_u,
                         const int32_t *pair_v, int64_t M, int flags, float *score,
                         int32_t *count, void *workspace, size_t workspace_bytes, void *stream_) {
  using namespace eps;
  cudaStream_t stream = (cudaStream_t)stream_;
  EPS_CHECK_ARG(n > 0 && M >= 0, "bad n or M");
  EPS_CHECK_ARG(!(flags & ~(EPS_CN_SIGMOID | EPS_CN_GROUPED_BY_V | EPS_SCORE_KIND_MASK)), "unknown flag bits");
  const int kind = score_kind(flags);
  EPS_CHECK_ARG(!kind || (!wtable && !val && !(flags & EPS_CN_SIGMOID)),
                "a similarity kind (EPS_SCORE_*) needs wtable == NULL, val == NULL and no EPS_CN_SIGMOID");
  if (M == 0) return EPS_OK;  // empty pair list: nothing to read or write
  EPS_CHECK_ARG(rowptr && col && pair_u && pair_v, "null graph or pair pointer");
  EPS_CHECK_ARG(score || count, "score and count both NULL");
  const int sms = sm_count();
  if (sms <= 0) { set_error("eps_cn_aa: no CUDA device"); return EPS_ERR_CUDA; }
  const size_t bitmap_bytes = (size_t)((n + 31) / 32) * 4;
  const bool grouped = (flags & EPS_CN_GROUPED_BY_V) && val == nullptr &&
                       bitmap_bytes <= CN_MAX_BITMAP_BYTES;
  if (grouped) {
    if (!workspace || workspace_bytes < eps_cn_aa_workspace_bytes()) {
      set_error("eps_cn_aa: workspace too small");
      return EPS_ERR_WORKSPACE;
    }
    EPS_CUDA(cudaMemsetAsync(workspace, 0, 8, stream));
    GroupedKernel kern = kind ? kGroupedKinds[kind] : wtable ? cn_grouped_kernel<true> : cn_grouped_kernel<false>;
    EPS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)bitmap_bytes));
    int occ = 0;
    EPS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, CN_THREADS, bitmap_bytes));
    if (occ < 1) occ = 1;
    const long long ntiles = (M + CN_TILE_PAIRS - 1) / CN_TILE_PAIRS;
    const int grid = (int)std::min<long long>(ntiles, (long long)sms * occ);
    kern<<<grid, CN_THREADS, bitmap_bytes, stream>>>(rowptr, col, wtable, n, pair_u, pair_v,
                                                     (long long)M, flags, score, count,
                                                     (unsigned long long *)workspace);
    EPS_LAUNCH_CHECK();
    return EPS_OK;
  }
  const long long groups_per_block = 256 / PAIR_G;
  const long long want = (M + groups_per_block - 1) / groups_per_block;
  const int grid = (int)std::min<long long>(want, (long long)sms * 8 * 4);
#define EPS_LAUNCH_PAIRS(HV, HW)                                                             \
  cn_pairs_kernel<HV, HW><<<grid, 256, 0, stream>>>(rowptr, col, val, wtable, pair_u, pair_v, \
                                                    (long long)M, flags, score, count)
  if (kind) kPairsKinds[kind]<<<grid, 256, 0, stream>>>(rowptr, col, val, wtable, pair_u, pair_v, (long long)M, flags,
                                                       score, count);
  else if (val && wtable) EPS_LAUNCH_PAIRS(true, true);
  else if (val) EPS_LAUNCH_PAIRS(true, false);
  else if (wtable) EPS_LAUNCH_PAIRS(false, true);
  else EPS_LAUNCH_PAIRS(false, false);
#undef EPS_LAUNCH_PAIRS
  EPS_LAUNCH_CHECK();
  return EPS_OK;
}
